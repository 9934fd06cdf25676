"""ctypes binding of libpgtscan.so (include/pgt_scan.h, include/pgt_extreme.h).

The shared library is built in-tree (popgenomicstools_b200/csrc/Makefile, or
``__graft_entry__.build()``).  There is no Python/CPU fallback: a missing library raises
ImportError here, and a missing CUDA device makes every scan call raise PgtError.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# PGT_LIB: another build of the same library, e.g. libpgtscan_bounds.so (-DPGT_BOUNDS: every kernel index checked)
LIB_PATH = os.environ.get("PGT_LIB") or os.path.join(_HERE, "libpgtscan.so")

PGT_OK, PGT_ERR_ARGS, PGT_ERR_CUDA, PGT_ERR_NOMEM, PGT_ERR_INPUT = 0, -1, -2, -3, -4
PGT_MEM_DEVICE, PGT_MEM_HOST = 0, 1
PGT_MODE_SITES, PGT_MODE_BP = 0, 1


class PgtError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libpgtscan error {code}: {msg}")
        self.code = code


PGT_STAT_FST, PGT_STAT_HET, PGT_STAT_DXY, PGT_STAT_FUSED = 0, 1, 2, 3


class PgtRange(C.Structure):
    _fields_ = [("w_lo", C.c_uint64), ("w_hi", C.c_uint64), ("site_origin", C.c_uint64), ("site_count", C.c_uint64)]


COLUMN_FIELDS = ("pos", "a", "b", "geno", "f1", "f2", "n1", "n2")
WINDOW_FIELDS = ("label", "start_pos", "end_pos", "mid_pos", "nsites", "sum_a", "sum_b", "fst", "nhet", "nonmissing",
                 "het", "dxy", "neffective", "nskip", "dxy_global")


XWINDOW_FIELDS = ("ext_value", "ext_pos", "ext_site", "nbig", "nsites", "prop")
PGT_XSTAT_IHS, PGT_XSTAT_XPEHH = 0, 1


class PgtXWindows(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in XWINDOW_FIELDS]


class PgtColumns(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in COLUMN_FIELDS]


class PgtWindows(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in WINDOW_FIELDS]


_u64p = C.POINTER(C.c_uint64)
_u32p = C.POINTER(C.c_uint32)

# name -> (restype, argtypes); every symbol include/pgt_scan.h and include/pgt_extreme.h declare
PROTOTYPES = {
    "pgt_last_error": (C.c_char_p, []),
    "pgt_abi_version": (C.c_int, []),
    "pgt_device_count": (C.c_int, []),
    "pgt_set_device": (C.c_int, [C.c_int]),
    "pgt_host_alloc": (C.c_int, [C.POINTER(C.c_void_p), C.c_size_t]),
    "pgt_host_free": (C.c_int, [C.c_void_p]),
    "pgt_host_register": (C.c_int, [C.c_void_p, C.c_size_t]),
    "pgt_host_unregister": (C.c_int, [C.c_void_p]),
    "pgt_device_alloc": (C.c_int, [C.POINTER(C.c_void_p), C.c_size_t]),
    "pgt_device_free": (C.c_int, [C.c_void_p]),
    "pgt_ipc_export": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t]),
    "pgt_ipc_open": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "pgt_ipc_close": (C.c_int, [C.c_void_p]),
    "pgt_uploader_pinned_bytes": (C.c_size_t, [C.c_uint32, C.c_size_t]),
    "pgt_uploader_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_void_p, C.c_size_t, C.c_uint32, C.c_size_t, C.c_uint32]),
    "pgt_uploader_put": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "pgt_uploader_put_file": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_uint64, C.c_size_t]),
    "pgt_uploader_drain": (C.c_int, [C.c_void_p, _u64p]),
    "pgt_uploader_destroy": (None, [C.c_void_p]),
    "pgt_memcpy_to_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t]),
    "pgt_device_mem_info": (C.c_int, [C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]),
    "pgt_plan_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32,
                                  C.c_uint32]),
    "pgt_plan_destroy": (None, [C.c_void_p]),
    "pgt_plan_num_windows": (C.c_uint64, [C.c_void_p]),
    "pgt_plan_num_units": (C.c_uint64, [C.c_void_p]),
    "pgt_plan_num_segments": (C.c_uint32, [C.c_void_p]),
    "pgt_plan_num_sites": (C.c_uint64, [C.c_void_p]),
    "pgt_plan_window": (C.c_int, [C.c_void_p, C.c_uint64, _u64p, _u64p, _u32p]),
    "pgt_plan_windows": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "pgt_plan_unit": (C.c_int, [C.c_void_p, C.c_uint64, _u64p, _u32p]),
    "pgt_plan_window_units": (C.c_int, [C.c_void_p, C.c_uint64, _u64p, _u64p]),
    "pgt_plan_shard": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, _u64p, _u64p, _u64p, _u64p]),
    "pgt_plan_device_bytes": (C.c_size_t, [C.c_void_p]),
    "pgt_plan_bind_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "pgt_plan_scan_path": (C.c_int, [C.c_void_p, C.c_int]),
    "pgt_scan_workspace_bytes": (C.c_size_t, [C.c_void_p, C.POINTER(PgtRange), C.c_int, C.c_int]),
    "pgt_scan": (C.c_int, [C.c_void_p, C.POINTER(PgtRange), C.c_int, C.POINTER(PgtColumns), C.c_int, C.c_void_p,
                           C.POINTER(PgtWindows), C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]),
    "pgt_scan_bp_sites_workspace_bytes": (C.c_size_t, [C.c_void_p, C.POINTER(PgtRange), C.c_void_p, C.c_int]),
    "pgt_scan_bp_sites": (C.c_int, [C.c_void_p, C.POINTER(PgtRange), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t,
                                    C.c_int, C.c_void_p]),
    "pgt_scan_sharded_workspace_bytes": (C.c_size_t, [C.c_void_p, C.c_int, C.c_uint32, C.c_uint32]),
    "pgt_scan_sharded": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(PgtColumns), C.c_int, C.c_void_p, C.POINTER(PgtWindows),
                                   C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p]),
    "pgt_scan_fst": (C.c_int, [C.c_void_p, C.POINTER(PgtRange), C.POINTER(PgtColumns), C.POINTER(PgtWindows),
                               C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]),
    "pgt_scan_het": (C.c_int, [C.c_void_p, C.POINTER(PgtRange), C.POINTER(PgtColumns), C.POINTER(PgtWindows),
                               C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]),
    "pgt_scan_dxy": (C.c_int, [C.c_void_p, C.POINTER(PgtRange), C.POINTER(PgtColumns), C.c_int, C.c_void_p,
                               C.POINTER(PgtWindows), C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]),
    "pgt_scan_fused": (C.c_int, [C.c_void_p, C.POINTER(PgtRange), C.POINTER(PgtColumns), C.c_int,
                                 C.POINTER(PgtWindows), C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]),
    "pgt_synth_fst": (C.c_int, [C.c_uint64, C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "pgt_synth_het": (C.c_int, [C.c_uint64, C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p]),
    "pgt_synth_dxy": (C.c_int, [C.c_uint64, C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                C.c_void_p]),
    "pgt_synth_pos": (C.c_int, [C.c_uint64, C.c_uint64, C.c_uint64, C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p,
                                C.c_void_p]),
    "pgt_profile": (C.c_int, [C.c_int]),
    "pgt_profile_read": (C.c_int, [C.POINTER(C.c_double), _u64p, C.POINTER(C.c_double), _u64p]),
    "pgt_tune": (C.c_int, [C.c_char_p, C.c_int]),
    "pgt_kernel_launch_count": (C.c_uint64, []),
    # include/pgt_extreme.h
    "pgt_xplan_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32,
                                   C.c_uint32]),
    "pgt_xplan_destroy": (None, [C.c_void_p]),
    "pgt_xplan_num_windows": (C.c_uint64, [C.c_void_p]),
    "pgt_xplan_num_units": (C.c_uint64, [C.c_void_p]),
    "pgt_xplan_num_sites": (C.c_uint64, [C.c_void_p]),
    "pgt_xplan_windows": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "pgt_xplan_shard": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, _u64p, _u64p, _u64p, _u64p]),
    "pgt_xplan_device_bytes": (C.c_size_t, [C.c_void_p]),
    "pgt_xplan_bind_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "pgt_scan_extreme_workspace_bytes": (C.c_size_t, [C.c_void_p, C.POINTER(PgtRange), C.c_int]),
    "pgt_scan_extreme": (C.c_int, [C.c_void_p, C.POINTER(PgtRange), C.c_int, C.c_double, C.c_void_p, C.c_void_p,
                                   C.POINTER(PgtXWindows), C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]),
    "pgt_scan_extreme_sharded": (C.c_int, [C.c_void_p, C.c_int, C.c_double, C.c_void_p, C.c_void_p, C.POINTER(PgtXWindows), C.c_void_p,
                                           C.c_uint32]),
    "pgt_scan_plan_extreme_workspace_bytes": (C.c_size_t, [C.c_void_p, C.POINTER(PgtRange), C.c_int]),
    "pgt_scan_plan_extreme": (C.c_int, [C.c_void_p, C.POINTER(PgtRange), C.c_int, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.POINTER(PgtWindows), C.POINTER(PgtXWindows), C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]),
    "pgt_scan_plan_extreme_sharded": (C.c_int, [C.c_void_p, C.c_int, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p,
                                                C.POINTER(PgtWindows), C.POINTER(PgtXWindows), C.c_void_p, C.c_uint32]),
    "pgt_synth_score": (C.c_int, [C.c_uint64, C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p]),
    "pgt_profile_read_extreme": (C.c_int, [C.POINTER(C.c_double), _u64p, C.POINTER(C.c_double), _u64p]),
}

_lib = None


def load():
    """Load libpgtscan.so (once) and attach prototypes.  Raises ImportError if it is not built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is not built (run `make -C popgenomicstools_b200/csrc` or __graft_entry__.build()); "
                "popgenomicstools_b200 has no CPU fallback")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(lib, name)  # AttributeError = header/library mismatch
            fn.restype = res
            fn.argtypes = args
        # PGT_TUNE="key=value,..." applies pgt_tune knobs at load time (experiments and forced-path test runs)
        for kv in filter(None, os.environ.get("PGT_TUNE", "").split(",")):
            key, _, val = kv.partition("=")
            if lib.pgt_tune(key.strip().encode(), int(val)) != 0:
                raise ValueError(f"PGT_TUNE: unknown knob or value {kv!r}")
        _lib = lib
    return _lib


def check(rc):
    if rc < 0:
        raise PgtError(rc, load().pgt_last_error().decode(errors="replace"))
    return rc
