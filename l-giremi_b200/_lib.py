"""ctypes binding of liblgmi.so (include/lgmi.h).  This is the stub a reference
maintainer would add next to giremi/mutual_information.py; see INTEGRATION.md.

Loading never falls back to anything: a missing library raises, and creating a
context without a CUDA device raises (LGMI_ERR_NODEVICE)."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
# LGMI_LIB: another build of the same library (kernel experiments: tools/build_variant.py); default in-tree
LIB_PATH = os.environ.get("LGMI_LIB") or os.path.join(HERE, "liblgmi.so")

# numpy mirrors of the ABI structs
UNIT_DESC = np.dtype([("plane_off", "<u8"), ("n_sites", "<u4"), ("n_reads", "<u4"),
                      ("row_words", "<u4"), ("site_off", "<u4")], align=True)
PAIR_REC = np.dtype([("unit", "<u4"), ("i", "<u2"), ("j", "<u2"), ("mi", "<f8")], align=True)
assert UNIT_DESC.itemsize == 24 and PAIR_REC.itemsize == 16

SITE_MISMATCH, SITE_SNP, SITE_HET_SNP = 0, 1, 2
SITE_TYPE_MASK = 0x03
SITE_HAS_OTHER = 0x04
SITE_TYPE_NAMES = ("mismatch", "snp", "het_snp")
SITE_TYPE_CODE = {"mismatch": SITE_MISMATCH, "snp": SITE_SNP, "het_snp": SITE_HET_SNP}

MODE_ALL_PAIRS = 0x0
MODE_HET_ONLY = 0x1
MODE_EMIT_COUNTS = 0x2
MODE_SKIP_NONHET = 0x4
MODE_SPLIT_RECORDS = 0x8
MODE_GRAPH = 0x10
MODE_TIGHT_INPUT = 0x20
MODE_COMPACT_OUTPUT = 0x40

ERR_NODEVICE = -5
DENSE_DEFAULT = (48, 8192)    # lgmi_set_dense_threshold defaults: (min_sites, min_reads)

EXPORTS = (
    "lgmi_version", "lgmi_create", "lgmi_destroy", "lgmi_last_error", "lgmi_set_stream",
    "lgmi_pinned_alloc", "lgmi_pinned_free", "lgmi_launch_count", "lgmi_set_dense_threshold",
    "lgmi_set_tile_path", "lgmi_set_dense_path",
    "lgmi_batch_create", "lgmi_batch_destroy", "lgmi_batch_upload", "lgmi_batch_run",
    "lgmi_batch_download", "lgmi_batch_sync", "lgmi_batch_device_ptrs",
    "lgmi_batch_create_rows", "lgmi_batch_upload_rows", "lgmi_batch_copy_planes", "lgmi_split_means",
    "lgmi_piece_export", "lgmi_batch_copy_planes_ipc", "lgmi_split_means_ipc",
    "lgmi_batch_algorithmic_bytes", "lgmi_pipeline_create", "lgmi_pipeline_step", "lgmi_pipeline_step_packed",
    "lgmi_pipeline_begin", "lgmi_pipeline_begin_packed", "lgmi_pipeline_collect", "lgmi_pipeline_finish",
    "lgmi_pipeline_destroy",
    "lgmi_submit", "lgmi_wait", "lgmi_site_mean_csr",
    "lgmi_ecdf", "lgmi_ecdf_eval", "lgmi_ecdf_table", "lgmi_site_splice_mi", "lgmi_device_count", "lgmi_cs_scan", "lgmi_encode_unit", "lgmi_unit_cost", "lgmi_partition_lpt",
)


class Result(C.Structure):
    _fields_ = [
        ("n_candidates", C.c_uint64),
        ("n_evaluated", C.c_uint64),
        ("n_records", C.c_uint64),
        ("records", C.c_void_p),
        ("counts", C.c_void_p),
        ("n_sites", C.c_uint64),
        ("site_mean", C.c_void_p),
        ("site_cnt", C.c_void_p),
        ("unit_rec_off", C.c_void_p),
        ("kernel_ms", C.c_float),
        ("pairs_kernel_ms", C.c_float),
        ("dense_kernel_ms", C.c_float),
        ("n_dense_units", C.c_uint32),
        ("dense_macs", C.c_uint64),
        ("gram_kernel_ms", C.c_float),
        ("rec_ij_bytes", C.c_uint32),
        ("gram_macs", C.c_uint64),
        ("rec_mi", C.c_void_p),
        ("rec_ij", C.c_void_p),
        ("n_dense_four", C.c_uint32),
    ]


class PieceIpc(C.Structure):
    """lgmi_piece_ipc: one piece of a split unit as another process imports it (plain bytes, 288 of them)."""
    _fields_ = [
        ("plane_mem", C.c_uint8 * 64),
        ("dense_mem", C.c_uint8 * 64),
        ("event", C.c_uint8 * 64),
        ("plane_word", C.c_uint64),
        ("plane_words", C.c_uint64),
        ("dense_off", C.c_uint64),
        ("dense_pairs", C.c_uint64),
        ("batch_id", C.c_uint64),
        ("unit", C.c_uint32),
        ("n_sites", C.c_uint32),
        ("row_limit", C.c_uint32),
        ("ran", C.c_uint32),
        ("pid", C.c_int32),
        ("pci_bus_id", C.c_char * 36),
    ]


class LgmiError(RuntimeError):
    def __init__(self, code, message):
        super().__init__("liblgmi error %d: %s" % (code, message))
        self.code = code


_lib = None


def load():
    """dlopen liblgmi.so and declare every prototype of include/lgmi.h."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "liblgmi.so is not built (%s). Run `python -c 'import __graft_entry__ as g; g.build()'` "
            "at the repo root. There is no CPU fallback for the MI step." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    vp, u64, u32, i32 = C.c_void_p, C.c_uint64, C.c_uint32, C.c_int
    pvp = C.POINTER(C.c_void_p)
    sig = {
        "lgmi_version": (i32, []),
        "lgmi_create": (i32, [i32, pvp]),
        "lgmi_destroy": (None, [vp]),
        "lgmi_last_error": (C.c_char_p, [vp]),
        "lgmi_set_stream": (i32, [vp, vp]),
        "lgmi_pinned_alloc": (i32, [vp, C.c_size_t, pvp]),
        "lgmi_pinned_free": (i32, [vp, vp]),
        "lgmi_launch_count": (u64, [vp]),
        "lgmi_set_dense_threshold": (i32, [vp, u32, u32]),
        "lgmi_set_tile_path": (i32, [vp, i32]),
        "lgmi_set_dense_path": (i32, [vp, i32]),
        "lgmi_batch_create": (i32, [vp, vp, u32, u64, u64, pvp]),
        "lgmi_batch_destroy": (None, [vp]),
        "lgmi_batch_upload": (i32, [vp, vp, vp]),
        "lgmi_batch_run": (i32, [vp, i32, u32]),
        "lgmi_batch_download": (i32, [vp, C.POINTER(Result)]),
        "lgmi_batch_sync": (i32, [vp, C.POINTER(Result)]),
        "lgmi_batch_device_ptrs": (i32, [vp, pvp, pvp, pvp, pvp]),
        "lgmi_batch_algorithmic_bytes": (i32, [vp, C.POINTER(u64)]),
        "lgmi_batch_create_rows": (i32, [vp, vp, u32, vp, u64, u64, pvp]),
        "lgmi_batch_upload_rows": (i32, [vp, vp, u64, u64, vp]),
        "lgmi_batch_copy_planes": (i32, [vp, u64, vp, u64, u64]),
        "lgmi_split_means": (i32, [vp, u32, vp, u32, vp, vp, vp, vp]),
        "lgmi_piece_export": (i32, [vp, u32, C.POINTER(PieceIpc)]),
        "lgmi_batch_copy_planes_ipc": (i32, [vp, u64, C.POINTER(PieceIpc), u64, u64]),
        "lgmi_split_means_ipc": (i32, [vp, u32, vp, u32, vp, vp, vp]),
        "lgmi_pipeline_create": (i32, [vp, vp, u32, u64, u64, u32, pvp]),
        "lgmi_pipeline_step": (i32, [vp, vp, vp, i32, u32, C.POINTER(Result)]),
        "lgmi_pipeline_step_packed": (i32, [vp, vp, vp, i32, u32, C.POINTER(Result)]),
        "lgmi_pipeline_begin": (i32, [vp, vp, vp, i32, u32]),
        "lgmi_pipeline_begin_packed": (i32, [vp, vp, vp, i32, u32]),
        "lgmi_pipeline_collect": (i32, [vp]),
        "lgmi_pipeline_finish": (i32, [vp, C.POINTER(Result)]),
        "lgmi_pipeline_destroy": (None, [vp]),
        "lgmi_submit": (i32, [vp, vp, u32, vp, u64, vp, u64, i32, u32]),
        "lgmi_wait": (i32, [vp, C.POINTER(Result)]),
        "lgmi_site_mean_csr": (i32, [vp, vp, vp, u64, vp]),
        "lgmi_ecdf": (i32, [vp, vp, vp, u64, C.c_double, vp, vp]),
        "lgmi_ecdf_eval": (i32, [vp, vp, u64, vp, u64, vp]),
        "lgmi_ecdf_table": (i32, [vp, vp, u64, vp, vp]),
        "lgmi_site_splice_mi": (i32, [vp, u32, vp, vp, vp, u32, vp, vp, u64, vp, vp, vp, vp, vp]),
        "lgmi_device_count": (i32, []),
        "lgmi_cs_scan": (i32, [C.c_char_p, u64, C.c_int64, i32, u32, vp, vp, vp, C.POINTER(u32), u32, vp, vp,
                               C.POINTER(u32)]),
        "lgmi_encode_unit": (i32, [u32, vp, vp, vp, vp, vp, vp, vp, C.c_char_p, u64, u64, vp, vp, vp,
                                   C.POINTER(u32), C.POINTER(u32)]),
        "lgmi_unit_cost": (u64, [u32, u32]),
        "lgmi_partition_lpt": (i32, [vp, u32, u32, vp, vp]),
    }
    for name in EXPORTS:
        fn = getattr(lib, name)            # AttributeError == missing export
        fn.restype, fn.argtypes = sig[name]
    _lib = lib
    return lib


def check(rc, handle=None):
    if rc != 0:
        msg = load().lgmi_last_error(handle)
        raise LgmiError(rc, msg.decode("utf-8", "replace") if msg else "")


def ptr(a):
    """Address of a C-contiguous numpy array (or None)."""
    if a is None:
        return None
    assert a.flags["C_CONTIGUOUS"]
    return a.ctypes.data


def array_at(address, dtype, count):
    """numpy view of `count` items of `dtype` at a raw host address."""
    dtype = np.dtype(dtype)
    if not address or count == 0:
        return np.empty(0, dtype=dtype)
    buf = (C.c_char * (dtype.itemsize * count)).from_address(address)
    return np.frombuffer(buf, dtype=dtype, count=count)
