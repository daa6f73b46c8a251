"""The per-round SAM record of -bam / -trf (mirge3.0_b200/csrc/sam_format.cuh: QNAME, RNAME, POS, SEQ / QUAL of the
round's query window, XA / MD / NM over the library text) compiled for the host and held byte for byte against
oracle/pyoracle.py::sam_line on seeded adversarial cases: keys with N, lower-case and IUPAC bytes; references with N;
mismatches inside, outside and at the 28-base seed boundary; poly-T tails of every length for round 3 and the end trims
of round 8; hits at the first and last position of a reference; reference names of 1 to 200 characters; keys of 16 to
512 nt."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from tests.util import host_harness_flags
import mirge_b200
from mirge_b200 import abi
from mirge_b200 import libraries as LB
from mirge_b200.manifoldAlign import round_query_text
from oracle import pyoracle as po
from tests.test_annotate_verify_host import HostLibrary, pack_key

HERE = os.path.dirname(os.path.abspath(__file__))
B = np.array(list("ACGT"))
ODD = list("NnacgtRYKMSWBDHV.")  # bytes a key may carry besides "ACGT": stored as exceptions
NAME_CHARS = np.array(list("abcdefghijklmnopqrstuvwxyzABCDEFGHIJKLMNOPQRSTUVWXYZ0123456789-_.|:"))


@pytest.fixture(scope="module")
def hs(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("hs") / "libsam_format_host.so")
    subprocess.check_call(["g++"] + host_harness_flags() + ["-std=c++17", "-shared", "-fPIC", "-I", os.path.join(mirge_b200.PACKAGE_DIR, "csrc"),
                           "-o", so, os.path.join(HERE, "sam_format_harness.cpp")])
    lib = C.CDLL(so)
    lib.hs_record.restype = C.c_uint32
    lib.hs_record.argtypes = [C.c_void_p, C.c_uint64, C.POINTER(abi.Library), C.POINTER(abi.RoundPolicy), C.c_void_p, C.c_void_p,
                              C.c_void_p]
    return lib


def rnd(rng, n):
    return "".join(rng.choice(B, n))


def make_refs(rng):
    """References of 20 to 700 bases (long enough for 512-nt queries), every third one with N; names of 1 to 200
    characters."""
    lens = [700, 530] + rng.choice([20, 24, 30, 45, 80, 150, 530, 700], size=int(rng.integers(4, 10))).tolist()
    refs = [rnd(rng, int(L)) for L in lens]
    for i in range(0, len(refs), 3):  # ambiguous reference bases
        s = list(refs[i])
        for j in rng.choice(len(s), size=int(rng.integers(1, 4)), replace=False):
            s[j] = "N"
        refs[i] = "".join(s)
    names = ["".join(rng.choice(NAME_CHARS, int(L))) for L in rng.choice([1, 2, 7, 20, 63, 64, 65, 128, 199, 200], size=len(refs))]
    return names, refs


def make_query(rng, ref: str, n: int):
    """(offset, query text) of n bases on ``ref``: first / last position or anywhere, with mismatches (substitutions
    and non-"ACGT" bytes) inside, outside and at the 28-base seed boundary, and lower-case matches."""
    m = rng.random()
    o = 0 if m < 0.2 else len(ref) - n if m < 0.4 else int(rng.integers(0, len(ref) - n + 1))
    q = list(ref[o : o + n].replace("N", str(rng.choice(B))))
    spots = [p for p in (26, 27, 28, 29) if p < n] if rng.random() < 0.5 else []
    spots += [int(p) for p in rng.choice(n, size=min(n, int(rng.choice([0, 0, 1, 2, 3, 6]))), replace=False)]
    for p in spots:
        r = rng.random()
        q[p] = str(rng.choice(ODD)) if r < 0.3 else str(rng.choice([c for c in "ACGT" if c != q[p]]))
    for p in rng.choice(n, size=min(n, int(rng.choice([0, 0, 0, 2]))), replace=False):
        q[p] = q[p].lower()
    return o, "".join(q)


def key_text(rng, q: str, rnd_i: int):
    """The sequence (QNAME) whose round-``rnd_i`` query window is about q: a T tail of 0 to 12 for round 3 (sometimes
    behind a lower-case 't'), one and two extra bases for round 8, as is otherwise."""
    if rnd_i == 3:
        tail = "T" * int(rng.choice([0, 1, 2, 3, 4, 5, 8, 12]))
        return q + ("t" if rng.random() < 0.15 else "") + tail
    if rnd_i == 8:
        return str(rng.choice(B)) + q + rnd(rng, 2)
    return q


@pytest.mark.parametrize("seed", range(8))
def test_records_equal_the_oracle(hs, seed):
    rng = np.random.default_rng(8800 + seed)
    names, refs = make_refs(rng)
    lib = HostLibrary(refs)
    enc = [nm.encode("latin-1") for nm in names]
    blob = np.frombuffer(b"".join(enc), dtype=np.uint8).copy()
    name_off = np.zeros(len(enc) + 1, dtype=np.uint64)
    name_off[1:] = np.cumsum([len(b) for b in enc])
    pols = LB.round_policies()
    out = np.zeros(8192, dtype=np.uint8)
    n_rec = n_mm = 0
    lengths = set()
    for i in range(300):
        rnd_i = int(rng.integers(0, 10))
        r = int(rng.integers(len(refs))) if i >= 10 else i % 2  # (the first ten: keys of about 512 nt)
        n = int(min(len(refs[r]), rng.choice([1, 5, 16, 18, 22, 25, 26, 28, 29, 30, 40, 100, 509]) if i >= 10 else 509))
        o, q = make_query(rng, refs[r], n)
        seq = key_text(rng, q, rnd_i)
        if len(seq) > abi.MAX_READ_LEN:
            seq = seq[: abi.MAX_READ_LEN]
        query = round_query_text(seq, pols[rnd_i])
        if len(query) > len(refs[r]):  # (a 't' behind the query of a whole reference)
            continue
        o = min(o, len(refs[r]) - len(query))
        key = pack_key(seq)
        hit = (int(rng.integers(0, 3)) << 56) | (r << 28) | o
        exp = (po.sam_line(seq, query, names[r], refs[r], o, po.ROUND_POLICIES[rnd_i]) + "\n").encode("latin-1")
        size = hs.hs_record(key.ctypes.data, hit, C.byref(lib.struct), C.byref(pols[rnd_i]), blob.ctypes.data, name_off.ctypes.data, None)
        out[: size + 1] = 0xAA
        wrote = hs.hs_record(key.ctypes.data, hit, C.byref(lib.struct), C.byref(pols[rnd_i]), blob.ctypes.data, name_off.ctypes.data,
                             out.ctypes.data)
        assert size == wrote == len(exp), (seq, rnd_i, size, len(exp))
        assert out[:size].tobytes() == exp, (out[:size].tobytes(), exp)
        assert out[size] == 0xAA  # nothing written past the record
        n_rec += 1
        n_mm += exp.count(b"NM:i:0") == 0
        lengths.add(len(seq))
    assert n_rec > 280 and n_mm > 50 and max(lengths) >= 500 and min(lengths) <= 20


def test_poly_t_tails_and_trims(hs):
    """Every T-run length 0..14 on round 3 (the query keeps what precedes the run, a lower-case 't' ends it), and round
    8's -5 1 -3 2 on keys down to nothing left."""
    rng = np.random.default_rng(77)
    names, refs = ["tRNA-Ala-AGC-1-1", "x"], [rnd(rng, 60), rnd(rng, 40)]
    lib = HostLibrary(refs)
    blob = np.frombuffer("".join(names).encode(), dtype=np.uint8).copy()
    name_off = np.array([0, len(names[0]), len(names[0]) + 1], dtype=np.uint64)
    pols = LB.round_policies()
    out = np.zeros(2048, dtype=np.uint8)
    cases = []
    for k in range(15):
        for body in (refs[0][:20], refs[0][:19] + "T", refs[0][:19] + "t", "TTT"[: k % 4]):
            cases.append((3, body + "T" * k))
    for L in range(0, 8):
        cases.append((8, refs[1][:L]))
    for rnd_i, seq in cases:
        query = round_query_text(seq, pols[rnd_i])
        r = 0 if rnd_i == 3 else 1
        exp = (po.sam_line(seq, query, names[r], refs[r], 0, po.ROUND_POLICIES[rnd_i]) + "\n").encode()
        key = pack_key(seq)
        size = hs.hs_record(key.ctypes.data, r << 28, C.byref(lib.struct), C.byref(pols[rnd_i]), blob.ctypes.data, name_off.ctypes.data,
                            out.ctypes.data)
        assert out[:size].tobytes() == exp, (rnd_i, seq, out[:size].tobytes(), exp)
