"""ctypes binding of libphylomap_b200.so (include/phylomap_b200.h).

This is the harness-side twin of the Rcpp shim shown in INTEGRATION.md: it flattens a tree list into `pm_tree`
and calls the same extern "C" entries.  There is no fallback: if the shared library is missing the import of
`lib()` raises, and every compute entry fails with PM_ERR_CUDA when no sm_100 device is present.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libphylomap_b200.so")

PM_OK, PM_ERR_ARG, PM_ERR_CUDA, PM_ERR_SAMPLE, PM_ERR_CAPACITY, PM_ERR_REPLAY = range(6)
PM_F64, PM_F32 = 0, 1
PM_MODE_PRODUCTION, PM_MODE_DETERMINISTIC = 0, 1
PM_RNG_PHILOX, PM_RNG_TABLE = 0, 1
PM_V_PLAIN, PM_V_SPARSE, PM_V_BIGTREE, PM_V_BF, PM_V_KS, PM_V_MT, PM_V_KSMT, PM_V_DIC2S, PM_V_DICKS, PM_V_EXP = range(10)

ALLREDUCE_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_int32)


class PmTree(C.Structure):
    _fields_ = [("n_tips", C.c_int32), ("n_edges", C.c_int32), ("edge", C.c_void_p), ("nen", C.c_void_p),
                ("nodelist", C.c_void_p), ("root", C.c_int32), ("maps_off", C.c_void_p), ("maps_len", C.c_void_p),
                ("maps_state", C.c_void_p), ("states", C.c_void_p), ("states_u8", C.c_void_p),
                ("n_sites", C.c_int64), ("edge_length", C.c_void_p)]


class PmOptions(C.Structure):
    _fields_ = [("device", C.c_int32), ("precision", C.c_int32), ("mode", C.c_int32), ("rng", C.c_int32),
                ("seed", C.c_uint64), ("site_offset", C.c_int64), ("path_capacity", C.c_int32),
                ("power_capacity", C.c_int32), ("tab_off", C.c_void_p), ("tab_u", C.c_void_p),
                ("host_tab", C.c_void_p), ("host_tab_n", C.c_int64), ("allreduce", ALLREDUCE_FN),
                ("allreduce_ctx", C.c_void_p), ("cuda_stream", C.c_void_p), ("progress", C.c_int32),
                ("nccl_world", C.c_int32), ("nccl_rank", C.c_int32), ("reserved", C.c_int32), ("nccl_id", C.c_void_p)]


EXPORTS = ["pm_default_options", "pm_nccl_unique_id", "pm_maketreelistMCMC", "pm_SPARSEmaketreelistMCMC", "pm_maketreelistMCMC_bigtree",
           "pm_maketreelistMCMCbf", "pm_maketreelistMCMCks", "pm_maketreelistMCMCmt", "pm_maketreelistMCMCksmt",
           "pm_maketreelistMCMC2sDICt", "pm_maketreelistMCMCksDICt", "pm_maketreelistEXP", "pm_loglik", "pm_expected_sumstats",
           "pm_ncols", "pm_tree_order", "pm_debug_clade_schedule", "pm_chain_create", "pm_chain_run", "pm_chain_state_bytes",
           "pm_chain_export_state", "pm_chain_import_state", "pm_chain_time_prune",
           "pm_chain_kernel_times", "pm_chain_enable_timing", "pm_chain_overheads", "pm_chain_get_node_states", "pm_chain_get_piece_counts",
           "pm_chain_get_path", "pm_chain_get_maps", "pm_chain_get_partials", "pm_chain_device_bytes", "pm_chain_acceptance", "pm_chain_destroy",
           "pm_rng_probe", "pm_release_cached_memory", "pm_device_count", "pm_version"]

_LIB = None


class PhylomapError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("phylomap_b200 error %d: %s" % (code, msg))
        self.code = code
        self.msg = msg


def lib():
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(LIB_PATH):
        raise ImportError("libphylomap_b200.so is not built (run `python -m phylomap_b200.build`); "
                          "there is no CPU fallback for the sampler")
    L = C.CDLL(LIB_PATH)
    vp, i32, i64, dbl = C.c_void_p, C.c_int32, C.c_int64, C.c_double
    L.pm_default_options.argtypes = [vp]
    L.pm_default_options.restype = None
    fixed = [vp, i32, vp, vp, vp, dbl, i32, vp, vp, C.c_char_p, C.c_size_t]
    for f in ("pm_maketreelistMCMC", "pm_SPARSEmaketreelistMCMC", "pm_maketreelistMCMC_bigtree"):
        getattr(L, f).argtypes = fixed
    rated = [vp, i32, vp, vp, vp, dbl, i32, vp, i32, vp, vp, C.c_char_p, C.c_size_t]
    for f in ("pm_maketreelistMCMCbf", "pm_maketreelistMCMCks", "pm_maketreelistMCMC2sDICt", "pm_maketreelistMCMCksDICt"):
        getattr(L, f).argtypes = rated
    multi = [vp, i32, i32, vp, vp, vp, dbl, i32, vp, i32, vp, vp, C.c_char_p, C.c_size_t]
    for f in ("pm_maketreelistMCMCmt", "pm_maketreelistMCMCksmt"):
        getattr(L, f).argtypes = multi
    L.pm_maketreelistEXP.argtypes = [vp, i32, vp, vp, i32, vp, vp, vp, vp, vp, C.c_char_p, C.c_size_t]
    L.pm_loglik.argtypes = [vp, i32, vp, vp, i32, vp, vp, C.c_char_p, C.c_size_t]
    L.pm_expected_sumstats.argtypes = [vp, i32, vp, vp, i32, vp, i64, vp, vp, vp, vp, vp, C.c_char_p, C.c_size_t]
    L.pm_ncols.argtypes = [i32, i32]
    L.pm_tree_order.argtypes = [vp, i32, i32, vp, vp, vp, C.c_char_p, C.c_size_t]
    L.pm_debug_clade_schedule.argtypes = [vp, i32, i32, vp, vp, i32, i32, i32, vp, C.c_char_p, C.c_size_t]
    L.pm_chain_create.argtypes = [i32, vp, i32, i32, vp, vp, vp, dbl, vp, i32, i32, vp, vp, C.c_char_p, C.c_size_t]
    L.pm_chain_run.argtypes = [vp, i32, vp, i64, C.c_char_p, C.c_size_t]
    L.pm_chain_state_bytes.argtypes = [vp]
    L.pm_chain_state_bytes.restype = i64
    L.pm_chain_export_state.argtypes = [vp, vp, i64, C.c_char_p, C.c_size_t]
    L.pm_chain_import_state.argtypes = [vp, vp, i64, C.c_char_p, C.c_size_t]
    L.pm_chain_time_prune.argtypes = [vp, i32, i32, vp, C.c_char_p, C.c_size_t]
    L.pm_chain_kernel_times.argtypes = [vp, vp, vp]
    L.pm_chain_kernel_times.restype = None
    L.pm_chain_enable_timing.argtypes = [vp, i32]
    L.pm_chain_enable_timing.restype = None
    L.pm_chain_overheads.argtypes = [vp, vp]
    L.pm_chain_overheads.restype = None
    L.pm_chain_get_node_states.argtypes = [vp, i32, vp]
    L.pm_chain_get_piece_counts.argtypes = [vp, i32, vp]
    L.pm_chain_get_path.argtypes = [vp, i32, i64, i32, vp, vp, i32]
    L.pm_chain_get_maps.argtypes = [vp, i32, vp, i64, vp, vp, vp, i64, C.c_char_p, C.c_size_t]
    L.pm_chain_get_partials.argtypes = [vp, i32, i64, vp]
    L.pm_chain_device_bytes.argtypes = [vp]
    L.pm_chain_device_bytes.restype = i64
    L.pm_chain_acceptance.argtypes = [vp, vp, vp, i32]
    L.pm_chain_acceptance.restype = i32
    L.pm_chain_destroy.argtypes = [vp]
    L.pm_chain_destroy.restype = None
    L.pm_rng_probe.argtypes = [C.c_uint32, i32, i32, dbl, dbl, vp]
    L.pm_rng_probe.restype = None
    L.pm_release_cached_memory.restype = None
    L.pm_device_count.restype = C.c_int
    L.pm_version.restype = C.c_char_p
    _LIB = L
    return L


def ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def default_options():
    o = PmOptions()
    lib().pm_default_options(C.byref(o))
    return o


def check(rc, err):
    if rc != PM_OK:
        raise PhylomapError(rc, err.value.decode(errors="replace"))
