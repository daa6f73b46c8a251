"""ctypes mirror of ``include/mirge_b200.h`` and loader of ``libmirge_b200.so``.

The structures here are the single host-side description of the trim parameters; the CUDA
library (product) and the C oracle (test infrastructure) both take them by pointer."""
import ctypes as C
import os

from . import LIB_PATH

MAX_ADAPTERS = 16
MAX_ADAPTER_LEN = 64
MAX_MODS = 8
MAX_READ_LEN = 512
LIB_PAD_WORDS = 40  # MIRGE_LIB_PAD_WORDS

MOD_NEXTSEQ, MOD_QUALITY, MOD_ADAPTER, MOD_NEND, MOD_CUT = 1, 2, 3, 4, 5
UMI_NONE, UMI_FLANKS, UMI_QIAGEN = 0, 1, 2
COMPAT_CUTADAPT23, COMPAT_CUTADAPT4 = 0, 1
LINK_BACK_HALF = 0x100  # MIRGE_LINK_BACK_HALF
LINK_INDEX_MASK, LINK_FRONT_OPTIONAL, LINK_BACK_OPTIONAL = 0xFF, 0x1000, 0x2000  # MIRGE_LINK_*
# MIRGE_WHERE_*
WHERE = {"back": 0, "front": 1, "suffix": 2, "prefix": 3, "back_not_internal": 4, "front_not_internal": 5}
COUNT_HEAD, COUNT_RELEASE = 0, 1
SELECT_LEN_LT26, SELECT_LEN_GT25, SELECT_UNANNOTATED = 0, 1, 2

OK, ERR_CUDA, ERR_ARG, ERR_FORMAT, ERR_CAPACITY, ERR_NODEVICE = 0, -1, -2, -3, -4, -5
NO_HIT = 0xFFFFFFFFFFFFFFFF
NO_KEY = 0xFFFFFFFF


class Adapter(C.Structure):
    _fields_ = [
        ("where", C.c_int32),
        ("m", C.c_int32),
        ("min_overlap", C.c_int32),
        ("indel_cost", C.c_int32),
        ("wildcard_ref", C.c_int32),
        ("wildcard_read", C.c_int32),
        ("k", C.c_int32),
        ("effective_length", C.c_int32),
        ("link", C.c_int32),
        ("mask", C.c_uint8 * MAX_ADAPTER_LEN),
        ("ascii", C.c_uint8 * MAX_ADAPTER_LEN),
        ("n_counts", C.c_int32 * (MAX_ADAPTER_LEN + 1)),
        ("max_err", C.c_int32 * (MAX_ADAPTER_LEN + 1)),
    ]


class TrimParams(C.Structure):
    _fields_ = [
        ("n_mods", C.c_int32),
        ("mod_kind", C.c_int32 * MAX_MODS),
        ("mod_a", C.c_int32 * MAX_MODS),
        ("mod_b", C.c_int32 * MAX_MODS),
        ("mod_c", C.c_int32 * MAX_MODS),
        ("n_adapters", C.c_int32),
        ("times", C.c_int32),
        ("min_len", C.c_int32),
        ("umi_mode", C.c_int32),
        ("umi5", C.c_int32),
        ("umi3", C.c_int32),
        ("qia_adapter_len", C.c_int32),
        ("count_mode", C.c_int32),
        ("compat", C.c_int32),
        ("adapters", Adapter * MAX_ADAPTERS),
    ]


class Table(C.Structure):
    _fields_ = [
        ("d_slots", C.c_void_p),
        ("capacity", C.c_uint64),
        ("d_arena", C.c_void_p),
        ("arena_words", C.c_uint64),
        ("d_key_ref", C.c_void_p),
        ("max_keys", C.c_uint64),
        ("d_ctrl", C.c_void_p),
    ]


class Library(C.Structure):
    _fields_ = [
        ("d_packed", C.c_void_p),
        ("d_nmask", C.c_void_p),
        ("d_ref_off", C.c_void_p),
        ("n_refs", C.c_uint32),
        ("n_bases", C.c_uint32),
        ("d_idx_kmer", C.c_void_p),
        ("d_idx_pos", C.c_void_p),
        ("n_idx", C.c_uint32),
        ("bucket_bits", C.c_uint32),
        ("d_idx_bucket", C.c_void_p),
        ("d_ref_block", C.c_void_p),
        ("ref_block_shift", C.c_uint32),
        ("filter_bases", C.c_uint32),
        ("d_filter", C.c_void_p),
        ("filter16_bits", C.c_uint32),
        ("max_ref_len", C.c_uint32),
        ("d_filter16", C.c_void_p),
    ]


class RoundPolicy(C.Structure):
    _fields_ = [
        ("round", C.c_int32),
        ("select", C.c_int32),
        ("seed_len", C.c_int32),
        ("seed_mm", C.c_int32),
        ("total_mm", C.c_int32),
        ("trim5", C.c_int32),
        ("trim3", C.c_int32),
        ("strip_polyT", C.c_int32),
    ]


ABI_VERSION = 4  # MIRGE_ABI_VERSION of include/mirge_b200.h

# name -> (restype, argtypes); every symbol include/mirge_b200.h declares
_P = C.c_void_p
_U64 = C.c_uint64
_PU64 = C.POINTER(C.c_uint64)
SYMBOLS = {
    "mirge_abi_version": (C.c_int, []),
    "mirge_ctx_create": (C.c_int, [C.c_int, C.POINTER(_P)]),
    "mirge_ctx_destroy": (None, [_P]),
    "mirge_last_error": (C.c_char_p, [_P]),
    "mirge_set_trim_params": (C.c_int, [_P, C.POINTER(TrimParams)]),
    "mirge_trim_slots": (C.c_int, [_P]),
    "mirge_tokenise_scratch_bytes": (_U64, [_U64]),
    "mirge_tokenise_sync": (C.c_int, [_P, _P, _U64, C.c_int, _P, _PU64, _PU64, _P]),
    "mirge_line_index": (C.c_int, [_P, _P, _U64, _P, _P, _U64, _P]),
    "mirge_trim_scratch_bytes": (_U64, [_U64]),
    "mirge_trim": (C.c_int, [_P, _P, _U64, _P, _U64, _P, _P, _P, _U64, _P, _P, _P, _U64, _P]),
    "mirge_trim_mode": (C.c_int, [_P, C.c_int]),
    "mirge_table_reset": (C.c_int, [_P, C.POINTER(Table), _P]),
    "mirge_collapse_insert_list": (C.c_int, [_P, C.POINTER(Table), _P, _P, _U64, _P, _P]),
    "mirge_collapse_merge_inplace": (C.c_int, [_P, C.POINTER(Table), _P, _U64, _P, _P]),
    "mirge_table_rehash": (C.c_int, [_P, C.POINTER(Table), C.POINTER(Table), _P]),
    "mirge_table_check_sync":(C.c_int, [_P, C.POINTER(Table), _PU64, _PU64, _P]),
    "mirge_table_drain": (C.c_int, [_P, C.POINTER(Table), _P, _P, _U64, _P, _P]),
    "mirge_umi_collapse": (
        C.c_int,
        [_P, C.POINTER(Table), _P, _P, _U64, C.POINTER(Table), C.c_int, C.c_int, C.c_int, C.c_int, _P, _P],
    ),
    "mirge_table_export_keys": (C.c_int, [_P, C.POINTER(Table), _U64, _U64, _P, C.c_uint32, _P, _P]),
    "mirge_key_sizes": (C.c_int, [_P, _P, _P, _U64, _P, _P]),
    "mirge_pack_keys": (C.c_int, [_P, _P, _P, _U64, _P, _P, _P]),
    "mirge_partition_plan": (
        C.c_int,
        [_P, C.POINTER(Table), _P, _U64, C.c_int, C.c_int, C.c_uint32, _P, _P, _P],
    ),
    "mirge_partition_totals": (C.c_int, [_P, _P, _P, _U64, C.c_uint32, _P, _P]),
    "mirge_partition_scatter": (C.c_int, [_P, C.POINTER(Table), _P, _P, _P, _P, _U64, C.c_uint32, _P, _P, _P, _P]),
    "mirge_shard_scatter": (C.c_int, [_P, _P, _P, _U64, C.c_uint32, C.c_uint32, C.c_uint32, _P, _P, _P, _P]),
    "mirge_shard_rebase": (C.c_int, [_P, _P, C.c_uint32, _PU64, _PU64, _P]),
    "mirge_shard_scatter_centre": (
        C.c_int,
        [_P, _P, _P, _U64, C.c_uint32, C.c_int, C.c_int, C.c_uint32, C.c_uint32, _P, _P, _P, _P],
    ),
    "mirge_lib_kmers": (C.c_int, [_P, C.POINTER(Library), _P, _P, _P]),
    "mirge_lib_filter": (C.c_int, [_P, _P, _P, C.c_uint32, C.c_uint32, _P, _P]),
    "mirge_lib_filter16": (C.c_int, [_P, _P, _P, C.c_uint32, C.c_uint32, _P, _P]),
    "mirge_annotate_scratch_bytes": (_U64, [_U64]),
    "mirge_annotate_rounds": (
        C.c_int,
        [_P, C.POINTER(Library), C.POINTER(RoundPolicy), C.c_int, C.POINTER(Table), _U64, _P, _P, _P, _P],
    ),
    "mirge_annotate_allhits": (
        C.c_int,
        [_P, C.POINTER(Library), C.POINTER(RoundPolicy), C.POINTER(Table), _P, _U64, _P, C.c_int, _P, _P, _P, _P],
    ),
    "mirge_sam_format": (
        C.c_int,
        [_P, C.POINTER(Library), C.POINTER(RoundPolicy), C.POINTER(Table), _P, _P, _U64, _P, _P, C.c_int, _P, _P, _P, _P],
    ),
    "mirge_table_csv_format": (
        C.c_int,
        [_P, C.POINTER(Table), _P, _U64, _P, _P, _P, _P, _P, C.c_int, _P, C.c_int, _U64, C.c_int, _P, _P, _P, _P],
    ),
    "mirge_report_reduce":(C.c_int, [_P, _P, _P, _P, _P, _U64, C.c_uint32, _P, _P, _P, _P]),
    "mirge_annotate_round": (
        C.c_int,
        [_P, C.POINTER(Library), C.POINTER(RoundPolicy), C.POINTER(Table), _U64, _P, _P, _P],
    ),
}

_lib = None


def load_library(path: str = None):
    """dlopen libmirge_b200.so and bind every declared symbol.  Raises (never falls back) when the
    library has not been built -- run ``python -c 'import __graft_entry__ as g; g.build()'``."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or LIB_PATH
    if not os.path.exists(p):
        raise RuntimeError(
            "mirge_b200: native library %s is missing; build it with __graft_entry__.build(). "
            "There is no CPU fallback." % p
        )
    lib = C.CDLL(p)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError if the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    if lib.mirge_abi_version() != ABI_VERSION:
        raise RuntimeError("mirge_b200: ABI version mismatch")
    if path is None:
        _lib = lib
    return lib
