"""The NextSeq / quality scans of the trim kernels (nextseq_trim_index / quality_trim_index in
mirge3.0_b200/csrc/adapter_search.cuh, four bytes per step) compiled for the host and held against cutadapt's byte loop
(oracle/pyoracle.py) where the word-at-a-time form can go wrong: every read length up to MIRGE_MAX_READ_LEN at every
byte alignment of the two lines, the first negative sum in each byte of a word, ties of the maximum across words, poly-G
runs, scans that never go negative, any byte value, both Phred offsets and the cutoffs / bases at the accepted limits.

Each line lives in an allocation of its own that ends with the last aligned 32-bit word holding a byte of the line and
starts with the first one; the bytes of those words outside the line are random guard bytes.  A scan that read a byte
outside the line would mostly disagree with the oracle, and under MIRGE_TEST_SANITIZE=1 (see tests/util.py) AddressSanitizer
reports a read of any word outside the allocation."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import mirge_b200
from mirge_b200 import abi
from mirge_b200 import params as P
from oracle import pyoracle as po
from tests.util import host_harness_flags

HERE = os.path.dirname(os.path.abspath(__file__))
MAX_LEN = 512  # MIRGE_MAX_READ_LEN
LIMIT = 1000  # largest cutoff / quality base the trim parameters accept

libc = C.CDLL(None)  # the process's malloc: the sanitizer's when its runtime is preloaded
libc.malloc.restype = C.c_void_p
libc.malloc.argtypes = [C.c_size_t]
libc.free.argtypes = [C.c_void_p]


@pytest.fixture(scope="module")
def hs(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("qs") / "libquality_scans_host.so")
    subprocess.check_call(["g++"] + host_harness_flags() + ["-std=c++17", "-shared", "-fPIC", "-I", os.path.join(mirge_b200.PACKAGE_DIR, "csrc"),
                           "-o", so, os.path.join(HERE, "adapter_search_harness.cpp")])
    lib = C.CDLL(so)
    lib.hs_set_params.argtypes = [C.POINTER(abi.TrimParams), C.POINTER(C.c_int), C.c_char_p, C.c_int]
    lib.hs_nextseq.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int]
    lib.hs_quality.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    return lib


class Line:
    """`data` at byte `align` of a fresh allocation of the aligned words that hold it, the rest of them guard bytes."""

    def __init__(self, data: bytes, align: int, rng):
        self.size = (align + len(data) + 3) & ~3
        self.mem = libc.malloc(max(self.size, 1))
        assert self.mem and self.mem % 16 == 0
        buf = bytes(rng.integers(0, 256, self.size, dtype=np.uint8))
        buf = buf[:align] + data + buf[align + len(data):]
        C.memmove(self.mem, buf, self.size)
        self.ptr = self.mem + align

    def free(self):
        libc.free(self.mem)


def check(hs, rng, seq: bytes, qual: bytes, cutoff: int, q5: int, base: int, a_seq: int, a_qual: int):
    assert len(seq) == len(qual)
    s_txt, q_txt = seq.decode("latin-1"), qual.decode("latin-1")
    ls, lq = Line(seq, a_seq, rng), Line(qual, a_qual, rng)
    try:
        got = hs.hs_nextseq(ls.ptr, lq.ptr, len(qual), cutoff, base)
        exp = po.nextseq_trim_index(s_txt, q_txt, cutoff, base)
        assert got == exp, ("nextseq", seq, qual, cutoff, base, a_seq, a_qual, got, exp)
        s, e = C.c_int(-1), C.c_int(-1)
        hs.hs_quality(lq.ptr, len(qual), q5, cutoff, base, C.byref(s), C.byref(e))
        exp = tuple(po.quality_trim_index(q_txt, q5, cutoff, base))
        assert (s.value, e.value) == exp, ("quality", qual, q5, cutoff, base, a_qual, (s.value, e.value), exp)
    finally:
        ls.free()
        lq.free()


def random_case(rng, L, base, cb):
    """seq / qual of length L in one of several shapes around the per-byte step cb - qual (cb = cutoff + base)."""
    mode = int(rng.integers(0, 7))
    if mode == 0:  # any byte value
        qual = rng.integers(0, 256, L)
    elif mode == 1:  # decaying qualities
        qual = base + np.clip(38 - (np.arange(L) * rng.integers(0, 50) // max(L, 1)) + rng.integers(-5, 6, L), 0, 41)
    elif mode == 2:  # steps of -1 / 0 / +1: the running sum revisits its maximum, ties everywhere
        qual = cb + rng.integers(-1, 2, L)
    elif mode == 3:  # never negative: every step >= 0
        qual = cb - rng.integers(0, 4, L)
    elif mode == 4:  # one level
        qual = np.full(L, int(rng.integers(0, 256)))
    elif mode == 5:  # good 5' part, bad 3' tail
        k = int(rng.integers(0, L + 1))
        qual = np.concatenate([cb - 1 - rng.integers(0, 10, k), cb + 1 + rng.integers(0, 5, L - k)]).astype(np.int64)
        if rng.random() < 0.5:
            qual = qual[::-1]
    else:
        qual = base + rng.integers(0, 42, L)
    qual = np.clip(qual, 0, 255)
    smode = int(rng.integers(0, 4))
    if smode == 0:
        seq = rng.choice(np.frombuffer(b"ACGTGGN", dtype=np.uint8), L)
    elif smode == 1:  # poly-G tail (NextSeq's dark cycles), sometimes with gaps
        k = int(rng.integers(0, L + 1))
        seq = np.concatenate([rng.choice(np.frombuffer(b"ACGT", dtype=np.uint8), L - k), np.full(k, ord("G"))]).astype(np.uint8)
        if k and rng.random() < 0.3:
            seq[L - k + int(rng.integers(0, k))] = ord("A")
    elif smode == 2:
        seq = np.full(L, ord("G"))
    else:  # any byte value ('G' with bit 7 set, 'g', ... are not G)
        seq = rng.choice(np.array([0x47, 0xC7, 0x67, 0x46, 0x48, 0x07, 0x00, 0xFF] + list(range(256))), L)
    return bytes(seq.astype(np.uint8)), bytes(qual.astype(np.uint8))


def test_every_length_and_alignment(hs):
    rng = np.random.default_rng(91)
    for L in range(MAX_LEN + 1):
        for a_qual in range(4):
            base = 33 if rng.random() < 0.7 else 64
            cutoff = int(rng.integers(0, 41))
            q5 = int(rng.integers(0, 41)) if rng.random() < 0.5 else 0
            seq, qual = random_case(rng, L, base, cutoff + base)
            check(hs, rng, seq, qual, cutoff, q5, base, int(rng.integers(0, 4)), a_qual)


@pytest.mark.parametrize("direction", ["3'", "5'"])
def test_first_negative_sum_in_each_byte_of_a_word(hs, direction):
    """Steps of +1 up to scan position p, then one step that takes the sum to -1: the scan must stop exactly at p, for
    p in every byte of a group of four, for every alignment, in both scan directions."""
    rng = np.random.default_rng(92)
    cutoff, base = 20, 33
    cb = cutoff + base
    for L in (4, 5, 7, 8, 9, 16, 33, 64, 131):
        for p in range(min(L, 40)):
            for a in range(4):
                steps = np.zeros(L, dtype=np.int64)  # step of scan position t
                steps[:p] = 1
                steps[p] = -(p + 1)
                steps[p + 1:] = rng.integers(-3, 4, L - p - 1)
                qual = cb - steps  # the step of a byte is cb - qual
                if direction == "3'":
                    qual = qual[::-1]
                qual = bytes(np.clip(qual, 0, 255).astype(np.uint8))
                seq = bytes(rng.choice(np.frombuffer(b"ACT", dtype=np.uint8), L))
                q5 = cutoff if direction == "5'" else 0
                check(hs, rng, seq, qual, cutoff, q5, base, (a + 1) % 4, a)


def test_ties_of_the_maximum_across_words(hs):
    """The sum reaches its maximum, then stays there or comes back to it in later words: the first position in scan
    order that reaches it must win (for the 3' scans the largest index, for the 5' scan the smallest)."""
    rng = np.random.default_rng(93)
    cutoff, base = 20, 64
    cb = cutoff + base
    for L in range(1, 70):
        for a in range(4):
            for first in range(min(L, 9)):
                steps = np.zeros(L, dtype=np.int64)
                steps[first] = 2
                if L > first + 2:
                    j = int(rng.integers(first + 1, L))
                    steps[j] = -1
                    if j + 1 < L:
                        steps[j + 1] = 1  # back to the maximum
                for qual in (cb - steps, (cb - steps)[::-1]):
                    check(hs, rng, b"A" * L, bytes(qual.astype(np.uint8)), cutoff, cutoff, base, a, (a + int(rng.integers(0, 4))) % 4)


def test_poly_g_and_limits_of_the_parameters(hs):
    """NextSeq poly-G tails with low qualities (the G step is +1 whatever the quality), and cutoffs / bases at the
    limits the trim parameters accept: 0 / LIMIT for the cutoffs, 1 / LIMIT for the base (a G byte then stands for a
    quality above 255)."""
    rng = np.random.default_rng(94)
    limits = [(0, 1), (0, LIMIT), (LIMIT, 1), (LIMIT, LIMIT), (LIMIT, 33), (255, 1), (256, 1), (0, 256), (1, 255), (20, 33), (20, 64)]
    for cutoff, base in limits:
        for it in range(120):
            L = int(rng.integers(0, MAX_LEN + 1)) if it % 4 else MAX_LEN
            seq, qual = random_case(rng, L, min(base, 255), cutoff + base)
            if it % 3 == 0:  # low-quality poly-G tail
                k = int(rng.integers(0, L + 1))
                seq = seq[: L - k] + b"G" * k
                qual = qual[: L - k] + bytes(rng.integers(0, 256, k, dtype=np.uint8))
            q5 = int(rng.choice([0, cutoff, LIMIT]))
            check(hs, rng, seq, qual, cutoff, q5, base, int(rng.integers(0, 4)), int(rng.integers(0, 4)))


@pytest.mark.parametrize("kind,a,b,ok", [
    ("nextseq", 0, 1, True), ("nextseq", LIMIT, LIMIT, True), ("nextseq", LIMIT + 1, 33, False), ("nextseq", -1, 33, False),
    ("nextseq", 20, 0, False), ("nextseq", 20, LIMIT + 1, False),
    ("quality", (0, LIMIT), 1, True), ("quality", (LIMIT, 0), LIMIT, True), ("quality", (0, LIMIT + 1), 33, False),
    ("quality", (LIMIT + 1, 20), 33, False), ("quality", (-1, 20), 33, False), ("quality", (0, 20), 0, False),
    ("quality", (0, 20), LIMIT + 1, False),
])
def test_quality_parameters_outside_the_limits_are_rejected(hs, kind, a, b, ok):
    if kind == "nextseq":
        cfg = P.TrimConfig(adapters=[("back", "TGGAATTCTCGGGTGCC")], nextseq_trim=a, quality_base=b)
    else:
        cfg = P.TrimConfig(adapters=[("back", "TGGAATTCTCGGGTGCC")], quality_cutoff="%d,%d" % a, quality_base=b)
    cp = P.build_trim_params(cfg)
    fast_ok = C.c_int(0)
    err = C.create_string_buffer(512)
    rc = hs.hs_set_params(C.byref(cp), C.byref(fast_ok), err, 512)
    if ok:
        assert rc == 0, err.value
    else:
        assert rc != 0 and b"trimming: quality cutoffs must lie in 0..1000 and the quality base in 1..1000" in err.value, (rc, err.value)
