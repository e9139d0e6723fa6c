"""ctypes binding of libpmmh_qn_b200.so (the C ABI declared in include/pmmh_qn.h).

There is NO CPU fallback: if the library is missing or cannot be loaded, importing the
kernels raises.  PyTorch is used elsewhere only as device allocator and stream owner.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libpmmh_qn_b200.so")

c_double_p = ctypes.c_void_p   # device / host pointers are passed as raw addresses
c_int = ctypes.c_int
c_ll = ctypes.c_longlong
c_ull = ctypes.c_ulonglong
c_size = ctypes.c_size_t
c_vp = ctypes.c_void_p
c_dbl = ctypes.c_double

DIAG_NEAR_TIES, DIAG_MAX_BIN, DIAG_STATUS, DIAG_KEY_TIES, DIAG_WAVEFRONT, DIAG_TRAJ_IDX, DIAG_KERNEL = range(7)
DIAG_SOFT_TIES = 4   # flps on the grid kernel (same slot as the bpf wave-front depth)
DIAG_COUNT = 8
MODEL_SV_LEVERAGE, MODEL_LINEAR_GAUSSIAN, MODEL_LINEAR_GAUSSIAN_FA, MODEL_LINEAR_GAUSSIAN_FA_GRAD = 0, 1, 2, 4
MODEL_LINEAR_GAUSSIAN_FA_HESS = 6
MODEL_SV_LEVERAGE_EXACT = 8
BPF_PARITY, BPF_INTENDED = 0, 1

# name -> (restype, argtypes); mirrors include/pmmh_qn.h one to one
SIGNATURES = {
    "pmmh_version": (c_int, []),
    "pmmh_last_error": (ctypes.c_char_p, []),
    "pmmh_device_info": (c_int, [ctypes.POINTER(c_int)] * 3),
    "pmmh_sv_set_algorithm": (c_int, [c_int]),
    "pmmh_sv_debug_profile": (c_int, [c_vp]),
    "pmmh_sv_workspace_bytes": (c_int, [c_int] * 8 + [ctypes.POINTER(c_size)]),
    "pmmh_flps_sv_corr": (c_int, [c_vp, c_ll, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_int, c_int,
                                  c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp,
                                  c_vp, c_size, c_int, c_vp]),
    "pmmh_flps_model_workspace_bytes": (c_int, [c_int, c_int, c_int, c_int, ctypes.POINTER(c_size)]),
    "pmmh_flps_model_corr": (c_int, [c_int, c_vp, c_ll, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_int,
                                     c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_size, c_vp]),
    "pmmh_filter_model_workspace_bytes": (c_int, [c_int, c_int, c_int, ctypes.POINTER(c_size)]),
    "pmmh_filter_model_corr": (c_int, [c_int, c_vp, c_ll, c_vp, c_vp, c_vp, c_int, c_int, c_int,
                                       c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_size, c_vp]),
    "pmmh_flps_model_batch_workspace_bytes": (c_int, [c_int, c_int, c_int, c_int, c_int, ctypes.POINTER(c_size)]),
    "pmmh_flps_model_batch_corr": (c_int, [c_int, c_vp, c_ll, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_int, c_int,
                                           c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_size,
                                           c_vp]),
    "pmmh_filter_model_batch_workspace_bytes": (c_int, [c_int, c_int, c_int, ctypes.POINTER(c_size)]),
    "pmmh_filter_model_batch_corr": (c_int, [c_int, c_vp, c_ll, c_vp, c_vp, c_vp, c_int, c_int, c_int,
                                             c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_size, c_vp]),
    "pmmh_sv_stage_bytes": (c_int, [c_int, c_int, ctypes.POINTER(c_size)]),
    "pmmh_sv_stream_schedule": (c_int, [c_int, c_vp, c_int]),
    "pmmh_sv_streamed_workspace_bytes": (c_int, [c_int, c_int, c_int, c_int, ctypes.POINTER(c_size)]),
    "pmmh_sv_streamed_eligible": (c_int, [c_int, c_int, c_int, c_int]),
    "pmmh_flps_sv_corr_streamed": (c_int, [c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_vp, c_size,
                                           c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_size,
                                           c_int, c_vp]),
    "pmmh_flps_sv_corr_philox_workspace_bytes": (c_int, [c_int, c_int, c_int, ctypes.POINTER(c_size)]),
    "pmmh_flps_sv_corr_philox": (c_int, [c_vp, c_vp, c_vp, c_ull, c_ull, c_int, c_int, c_int, c_vp, c_vp, c_vp,
                                         c_vp, c_vp, c_vp, c_vp, c_size, c_vp]),
    "pmmh_bpf_sv_corr": (c_int, [c_vp, c_ll, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_int,
                                 c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_size, c_int, c_vp]),
    "pmmh_split_rvs": (c_int, [c_vp, c_int, c_int, c_int, c_vp, c_vp, c_vp]),
    "pmmh_norm_cdf": (c_int, [c_vp, c_vp, c_ll, c_vp]),
    "pmmh_importance_discrete": (c_int, [c_vp, c_ll, c_vp, c_vp, c_vp, c_int, c_int, c_int,
                                         c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "pmmh_crank_nicolson": (c_int, [c_vp, c_vp, c_vp, c_ll, c_dbl, c_ull, c_ull, c_vp]),
    "pmmh_subsample_workspace_bytes": (c_int, [c_int, ctypes.POINTER(c_size)]),
    "pmmh_subsample_indices": (c_int, [c_vp, c_int, c_int, c_int, c_vp, c_vp, c_vp, c_size, c_vp]),
    "pmmh_logistic_workspace_bytes": (c_int, [c_int, c_int, c_int, ctypes.POINTER(c_size)]),
    "pmmh_logistic_loglike": (c_int, [c_vp, c_vp, c_vp, c_int, c_int, c_ll, c_ll, c_vp, c_int,
                                      c_vp, c_vp, c_size, c_vp]),
    "pmmh_svsplit_workspace_bytes": (c_int, [c_ll, c_ll, ctypes.POINTER(c_size)]),
    "pmmh_svsplit_init": (c_int, [c_vp, c_size, c_ll, c_int, c_int, c_int, c_int, c_ll, c_ll, c_int,
                                  c_vp, c_vp, c_vp, c_vp, c_vp]),
    "pmmh_svsplit_weights": (c_int, [c_vp, c_size, c_ll, c_ll, c_int, c_int, c_int, c_int, c_vp,
                                     c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "pmmh_svsplit_children": (c_int, [c_vp, c_size, c_ll, c_ll, c_int, c_int, c_vp, c_vp, c_vp, c_vp,
                                      c_ull, c_ull, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "pmmh_svsplit_plan": (c_int, [c_vp, c_size, c_ll, c_ll, c_int, c_vp, c_vp, c_vp]),
    "pmmh_svsplit_pack": (c_int, [c_vp, c_size, c_ll, c_ll, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "pmmh_svsplit_pack_direct": (c_int, [c_vp, c_size, c_ll, c_ll, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "pmmh_svsplit_sort": (c_int, [c_vp, c_size, c_ll, c_ll, c_int, c_int, c_int, c_vp, c_vp, c_int, c_vp, c_vp, c_vp]),
    "pmmh_svsplit_normalise": (c_int, [c_vp, c_int, c_vp, c_vp, c_vp]),
    "pmmh_svsplit_tail": (c_int, [c_vp, c_size, c_ll, c_ll, c_int, c_int, c_int, c_vp, c_vp, c_vp, c_vp,
                                  c_vp, c_vp, c_ll, c_vp, c_vp]),
    "pmmh_svsplit_finish": (c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_int, c_vp, c_int, c_int, c_ll,
                                    c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "pmmh_svsplit_diag": (c_int, [c_vp, c_size, c_ll, c_ll, c_vp]),
    "pmmh_flps_sv_corr_host": (c_int, [c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_int,
                                       c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "pmmh_bpf_sv_corr_host": (c_int, [c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_int,
                                      c_vp, c_vp, c_vp, c_vp]),
    "pmmh_importance_discrete_host": (c_int, [c_vp, c_vp, c_dbl, c_vp, c_int, c_int,
                                              c_vp, c_vp, c_vp, c_vp]),
    "pmmh_stratified_host": (c_int, [c_vp, c_int, c_int, c_vp]),
}

_lib = None


class PmmhError(RuntimeError):
    pass


def load():
    """Load the shared library (once) and attach the prototypes."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise PmmhError(
            "libpmmh_qn_b200.so is missing (%s). Build it with `python __graft_entry__.py` or "
            "`python pmmh-qn_b200/_build.py`; there is no CPU fallback." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)   # raises AttributeError if a declared symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc, what=""):
    if rc != 0:
        msg = load().pmmh_last_error()
        raise PmmhError("%s failed with status %d: %s" % (what or "pmmh call", rc,
                                                          msg.decode() if msg else ""))
