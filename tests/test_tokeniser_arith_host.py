"""Host check of the tokeniser's newline-mask arithmetic (csrc/common.cuh::newline_mask, used by tokenise.cu; the kernel replaces the
line splitting of dnaio's FastqIter, reference call site mirge/libs/digest.py:324) against a plain byte compare.
It is a pure integer trick, so it is restated with numpy and swept over random words: any byte values, dense
newlines, bytes >= 128."""
import os

import numpy as np

import mirge_b200

CSRC = os.path.join(mirge_b200.PACKAGE_DIR, "csrc")


def test_newline_mask_arithmetic():
    """newline_mask(): exact zero-byte flags of w ^ '\\n' x 4, two words per multiply by 0x00204081."""
    src = open(os.path.join(CSRC, "common.cuh")).read()
    assert "0x00204081u" in src and "0x7F7F7F7Fu" in src  # the constants restated below are the kernel's
    rng = np.random.default_rng(1)
    n = 200000
    b = rng.integers(0, 256, size=(n, 8, 4), dtype=np.uint8)
    b[rng.random((n, 8, 4)) < 0.3] = 0x0A
    w = (b.astype(np.uint32) << (8 * np.arange(4, dtype=np.uint32))).sum(axis=2, dtype=np.uint32)

    def flags(x):
        x = x ^ np.uint32(0x0A0A0A0A)
        t = ((x & np.uint32(0x7F7F7F7F)) + np.uint32(0x7F7F7F7F)).astype(np.uint32)
        return ~(t | x) & np.uint32(0x80808080)

    mask = np.zeros(n, dtype=np.uint32)
    for k in range(0, 8, 2):
        q = flags(w[:, k + 1]) | (flags(w[:, k]) >> np.uint32(4))
        r = (q.astype(np.uint64) * np.uint64(0x00204081)).astype(np.uint32)
        mask |= ((r >> np.uint32(24)) << np.uint32(4 * k)).astype(np.uint32)
    flat = b.reshape(n, 32)
    exp = np.zeros(n, dtype=np.uint32)
    for i in range(32):
        exp |= (flat[:, i] == 0x0A).astype(np.uint32) << np.uint32(i)
    assert np.array_equal(mask, exp)
