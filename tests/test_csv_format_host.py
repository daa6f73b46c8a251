"""The rows of mapped.csv / unmapped.csv / complete_set.csv (mirge3.0_b200/csrc/csv_format.cuh) compiled for the host
and held byte for byte against pandas' DataFrame.to_csv of the same one-row frames, on seeded adversarial cases: keys
with ',', '"', N, lower case, IUPAC and bytes >= 0x80; reference names with ',', '"', newlines and non-ASCII
characters; counts 0 and 2^32 - 1; 0, 1 and many samples; 9 and 10 annotation columns and the unannotated form.  The
header line (outputs.table_csv_header) is held against to_csv too, with sample names that need quoting."""
import ctypes as C
import io
import os
import subprocess

import numpy as np
import pandas as pd
import pytest

import mirge_b200
from mirge_b200.libraries import ROUND_COLUMNS
from mirge_b200.outputs import csv_field, table_csv_header
from tests.test_annotate_verify_host import pack_key
from tests.util import host_harness_flags

HERE = os.path.dirname(os.path.abspath(__file__))
KEY_BYTES = list("ACGT") * 6 + list("NnacgtRYKMSWBDHV.") + [",", '"', "\xe9", "\xff", "\x80", "\xc3"]
NAME_CHARS = list("abcXYZ019-_.|: ") + [",", '"', "\n", "\r", "\xe9", "µ", "–", "\U0001f9ec"]


@pytest.fixture(scope="module")
def hc(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("hc") / "libcsv_format_host.so")
    subprocess.check_call(["g++"] + host_harness_flags() + ["-std=c++17", "-shared", "-fPIC", "-I", os.path.join(mirge_b200.PACKAGE_DIR, "csrc"),
                           "-o", so, os.path.join(HERE, "csv_format_harness.cpp")])
    lib = C.CDLL(so)
    lib.hc_row.restype = C.c_uint32
    lib.hc_row.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p,
                           C.c_int, C.c_uint64, C.c_void_p]
    return lib


def to_csv(frame: pd.DataFrame) -> bytes:
    buf = io.BytesIO()
    frame.to_csv(buf)
    return buf.getvalue()


def frame(seq, cols, flag, names, counts):
    """The one-row frame bwtAlign (or baking) would hand to to_csv."""
    data = {"annotFlag": [flag]}
    data.update((c, [v]) for c, v in cols.items())
    data.update((s, [int(v)]) for s, v in zip(names, counts))
    return pd.DataFrame(data, index=pd.Index([seq], name="Sequence"))


def libraries(rng, n_cols):
    """Reference names per round (round 8 shares round 0's library, as the miRNA rounds do) as the kernel takes them:
    finished CSV fields back to back, offsets, a base per round."""
    per_round, fields, base = [], [], []
    for c in range(n_cols):
        if c == 8:
            per_round.append(per_round[0])
            base.append(base[0])
            continue
        names = ["".join(rng.choice(NAME_CHARS, int(rng.integers(1, 40)))) for _ in range(int(rng.integers(1, 12)))]
        per_round.append(names)
        base.append(len(fields))
        fields += [csv_field(nm).encode("utf-8") for nm in names]
    blob = np.frombuffer(b"".join(fields), dtype=np.uint8).copy()
    off = np.zeros(len(fields) + 1, dtype=np.uint64)
    off[1:] = np.cumsum([len(f) for f in fields])
    return per_round, blob, off, np.array(base, dtype=np.uint32)


def row(hc, key, kid, annot, hit, blob, off, base, n_cols, counts):
    S, n_keys = counts.shape
    cnt = np.ascontiguousarray(counts, dtype=np.uint32)
    args = (key.ctypes.data, kid, annot, hit, blob.ctypes.data, off.ctypes.data, base.ctypes.data, n_cols,
            cnt.ctypes.data if S else None, S, n_keys)
    size = hc.hc_row(*args, None)
    out = np.full(size + 1, 0xAA, dtype=np.uint8)
    wrote = hc.hc_row(*args, out.ctypes.data)
    assert wrote == size and out[size] == 0xAA  # sizing and fill agree, nothing written past the row
    return out[:size].tobytes()


@pytest.mark.parametrize("n_cols,annotated", [(9, True), (10, True), (10, False)])
@pytest.mark.parametrize("seed", range(4))
def test_rows_equal_to_csv(hc, n_cols, annotated, seed):
    rng = np.random.default_rng(4100 + 10 * seed + n_cols + annotated)
    per_round, blob, off, base = libraries(rng, n_cols)
    n_quoted = n_utf8 = 0
    for i in range(150):
        S = int(rng.choice([0, 1, 2, 3, 17]))
        names = ["s%d" % j for j in range(S)]
        L = int(rng.choice([1, 2, 16, 17, 30, 64, 200, 512]))
        seq = "".join(rng.choice(KEY_BYTES, L))
        n_keys = int(rng.integers(1, 6))
        kid = int(rng.integers(0, n_keys))
        counts = rng.choice([0, 1, 9, 10, 99, 12345, 2**31 - 1, 2**31, 2**32 - 1], size=(S, n_keys)).astype(np.uint64)
        annot, hit = 0xFF, 0
        cols = {c: "" for c in ROUND_COLUMNS[:n_cols]}
        if annotated and rng.random() < 0.8:
            annot = int(rng.integers(0, n_cols))
            r = int(rng.integers(0, len(per_round[annot])))
            hit = (int(rng.integers(0, 3)) << 56) | (r << 28) | int(rng.integers(0, 1 << 28))
            cols[ROUND_COLUMNS[annot]] = per_round[annot][r]
        flag = int(annot != 0xFF)
        exp = to_csv(frame(seq, cols, flag, names, counts[:, kid])).split(b"\n", 1)[1]
        got = row(hc, pack_key(seq), kid, annot, hit, blob, off, base, n_cols, counts)
        assert got == exp, (seq, annot, got, exp)
        n_quoted += got.startswith(b'"')
        n_utf8 += any(ord(c) >= 0x80 for c in seq)
    assert n_quoted > 20 and n_utf8 > 20


def test_special_keys_and_names(hc):
    """Hand-picked: a key that is a single '"', keys with ',' at either end, all four special-looking bytes at once,
    a name that is only '"', a name with CRLF."""
    per_round = [['"'], ["a\r\nb"], ["x,y"], ["été"], ["p"], ["q"], ["r"], ["s"], ['"'], ['""q']]
    fields = [csv_field(n[0]).encode("utf-8") for n in per_round]
    blob = np.frombuffer(b"".join(fields), dtype=np.uint8).copy()
    off = np.zeros(len(fields) + 1, dtype=np.uint64)
    off[1:] = np.cumsum([len(f) for f in fields])
    base = np.arange(10, dtype=np.uint32)
    counts = np.array([[0], [2**32 - 1]], dtype=np.uint64)
    for seq in ['"', ",ACGT", "ACGT,", '",\xe9"', "\xe9", "ACGTN", "acgt"]:
        for annot in list(range(10)) + [0xFF]:
            cols = {c: "" for c in ROUND_COLUMNS}
            if annot != 0xFF:
                cols[ROUND_COLUMNS[annot]] = per_round[annot][0]
            exp = to_csv(frame(seq, cols, int(annot != 0xFF), ["a", "b"], counts[:, 0])).split(b"\n", 1)[1]
            assert row(hc, pack_key(seq), 0, annot, 0, blob, off, base, 10, counts) == exp, (seq, annot)


@pytest.mark.parametrize("n_cols", [9, 10])
def test_header_equals_to_csv(n_cols):
    for names in ([], ["s1"], ["sampleA", "sampleB"], ["a,b", 'say "hi"', "line\nbreak", "cr\rx", "café", " sp "]):
        data = {"annotFlag": []}
        data.update((c, []) for c in ROUND_COLUMNS[:n_cols])
        data.update((s, []) for s in names)
        exp = to_csv(pd.DataFrame(data, index=pd.Index([], name="Sequence")))
        assert table_csv_header(names, n_cols) == exp, names
