"""CPU-side checks of the drop-in boundary: the C-ABI library builds, loads and exports every
symbol include/mirge_b200.h declares (no compute calls without a GPU)."""
import ctypes
import os
import re

import mirge_b200
from mirge_b200 import abi


def test_library_matches_declared_abi():
    """Every symbol the header declares is exported and bound, and library, header and bindings agree on the ABI
    version."""
    import __graft_entry__ as g

    g.build()
    lib = abi.load_library()
    hdr = open(os.path.join(mirge_b200.REPO_ROOT, "include", "mirge_b200.h")).read()
    declared = set(re.findall(r"\b(mirge_[a-z0-9_]+)\s*\(", hdr))
    assert declared == set(abi.SYMBOLS), declared ^ set(abi.SYMBOLS)
    for name in declared:
        assert getattr(lib, name) is not None
    hdr_version = int(re.search(r"#define MIRGE_ABI_VERSION (\d+)", hdr).group(1))
    assert lib.mirge_abi_version() == abi.ABI_VERSION == hdr_version == 4


def test_struct_sizes_match_header():
    # sizes derived from the header's field lists
    assert ctypes.sizeof(abi.Adapter) == 9 * 4 + 64 + 64 + 65 * 4 + 65 * 4  # + wildcard_read (ABI v3)
    assert ctypes.sizeof(abi.TrimParams) == 4 * (1 + 8 * 4 + 9) + 16 * ctypes.sizeof(abi.Adapter)  # + compat (ABI v2), 16 adapters (v3)
    assert ctypes.sizeof(abi.Table) == 56
    assert ctypes.sizeof(abi.RoundPolicy) == 32
    assert ctypes.sizeof(abi.Library) == 104  # + filter16_bits, max_ref_len, d_filter16 (ABI v2)


def test_no_device_fails_loudly():
    import torch

    if torch.cuda.is_available():
        return
    lib = abi.load_library()
    ctx = ctypes.c_void_p()
    assert lib.mirge_ctx_create(0, ctypes.byref(ctx)) == abi.ERR_NODEVICE
    from mirge_b200 import device as D
    import pytest

    with pytest.raises(D.MirgeError):
        D.Device(0)
