"""ctypes binding of the C ABI declared in ``include/mentflow_b200.h``.

The library is the product: there is no CPU or PyTorch fallback.  If the shared object is
missing (or a symbol is), importing the ops fails loudly.
"""
import ctypes
import os
from ctypes import c_char_p, c_double, c_float, c_int, c_int64, c_uint64, c_void_p

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
# MENTFLOW_B200_LIB overrides the library path (A/B runs of differently built kernels)
LIB_PATH = os.environ.get("MENTFLOW_B200_LIB") or os.path.join(PKG_DIR, "libmentflow_b200.so")

P = c_void_p  # every device pointer crosses the ABI as a plain address

ABI_VERSION = 5  # MFB_ABI_VERSION of the header SIGNATURES mirrors

# name -> (restype, argtypes); mirrors include/mentflow_b200.h line by line
SIGNATURES = {
    "mfb_abi_version": (c_int, []),
    "mfb_error_string": (c_char_p, [c_int]),
    "mfb_sm_count": (c_int, []),
    "mfb_kde1d_workspace_bytes": (c_int64, [c_int64, c_int, c_int, c_int]),
    "mfb_project_kde1d_fwd": (c_int, [P, c_int64, c_int, P, P, P, c_int, c_int, c_float, c_double, P, c_float, P, P, P,
                                      P, c_int64, P]),
    "mfb_kde1d_finish": (c_int, [P, c_double, P, c_int, c_int, P, c_float, P, P, P]),
    "mfb_kde1d_p2p_block_floats": (c_int64, [c_int, c_int, c_int]),
    "mfb_kde1d_finish_p2p": (c_int, [P, c_int, c_int, P, P, P, c_int, c_double, P, c_int, c_int, P, c_float, P, P, P, P, P]),
    "mfb_project_kde1d_loss_fwd_p2p": (c_int, [P, c_int64, c_int, P, P, c_int, c_int, c_float, c_double, P, c_float, P,
                                               c_int, c_int, P, P, c_int, P, P, P, P, P, c_int64, P]),
    "mfb_kde1d_finish_bwd": (c_int, [P, c_double, P, c_int, c_int, P, c_float, P, P, P, P]),
    "mfb_project_kde1d_bwd": (c_int, [P, c_int64, c_int, P, P, P, c_int, c_int, c_float, P, P, c_int, P]),
    "mfb_project_hist1d": (c_int, [P, c_int64, c_int, P, P, P, c_int, c_int, P, P]),
    "mfb_kde2d_workspace_bytes": (c_int64, [c_int64, c_int, c_int, c_int, c_int]),
    "mfb_project_kde2d_fwd": (c_int, [P, c_int64, c_int, P, P, c_int, c_int, c_int, c_float, P, P, c_int64, c_int, P]),
    "mfb_kde2d_uses_tensor_cores": (c_int, [c_int64, c_int, c_int, c_int, c_int]),
    "mfb_kde2d_normalize": (c_int, [P, P, c_int, c_int, c_int, P, P]),
    "mfb_kde2d_normalize_bwd": (c_int, [P, P, c_int, c_int, c_int, P, P, P]),
    "mfb_project_kde2d_bwd": (c_int, [P, c_int64, c_int, P, P, c_int, c_int, c_int, c_float, P, P, c_int, P]),
    "mfb_project_hist2d": (c_int, [P, c_int64, c_int, P, P, P, c_int, c_int, c_int, P, P]),
    "mfb_nsf_layer_param_floats": (c_int64, [c_int, c_int, c_int, c_int]),
    "mfb_nsf_tc_supported": (c_int, [c_int, c_int, c_int, c_int]),
    "mfb_nsf_tc_image_bytes": (c_int64, [c_int, c_int]),
    "mfb_nsf_tc_prepare": (c_int, [P, c_int64, c_int, c_int, c_int, c_int, c_int, P, P, P]),
    "mfb_nsf_layer_fwd": (c_int, [P, c_int64, c_int, c_int, c_int, c_int, P, P, P, P, c_int, P, P, P]),
    "mfb_nsf_layer_inv": (c_int, [P, c_int64, c_int, c_int, c_int, c_int, P, P, P, P, c_int, P, P, P]),
    "mfb_nsf_layer_param_om_floats": (c_int64, [c_int, c_int, c_int]),
    "mfb_nsf_layer_bwd_workspace_bytes": (c_int64, [c_int64, c_int, c_int]),
    "mfb_nsf_layer_bwd": (c_int, [P, P, P, c_int64, c_int, c_int, c_int, c_int, P, P, P, P, c_int, P, P, c_int, P,
                                  c_int64, P]),
    "mfb_ment_prob": (c_int, [P, c_int64, c_int, P, P, P, c_int, c_int, P, P, P, P, P, c_int, c_int, c_int, P, c_float,
                              c_float, P, P]),
    "mfb_ment_prob_grid": (c_int, [c_int, P, P, P, P, P, P, c_int, c_int, P, P, P, P, P, c_int, c_int, c_int, P, c_float,
                                   c_float, P, P]),
    "mfb_ment_integrate": (c_int, [c_int, P, c_int, c_int, P, c_int, c_int, c_int, P, P, P, P, P, P, P, P, c_int, c_int,
                                   P, P, P, P, P, c_int, c_int, c_int, P, c_float, c_float, P, P]),
    "mfb_randn_offset_increment": (c_int64, [c_int64]),
    "mfb_randn_philox": (c_int, [P, c_int64, c_uint64, c_uint64, P]),
    "mfb_randn_philox_state": (c_int, [P, c_int64, P, c_int, P]),
    "mfb_cdf_workspace_bytes": (c_int64, [c_int64]),
    "mfb_cdf_build": (c_int, [P, c_int64, c_double, P, P, c_int64, P]),
    "mfb_cdf_sample": (c_int, [P, c_int64, P, c_int, P, P, P, c_int, c_uint64, c_uint64, c_int64, P, P]),
    "mfb_gs_update": (c_int, [P, P, P, c_int, c_float, c_float, P]),
    "mfb_selftest_umma": (c_int, [P, P, c_int, P, P, P]),
    "mfb_selftest_umma_ts": (c_int, [P, P, c_int, P, P, P]),
    "mfb_selftest_umma_sw32": (c_int, [P, P, c_int, c_int, c_int, P, P, P]),
    "mfb_selftest_umma_pair": (c_int, [P, P, c_int, P, P, P]),
    "mfb_nsf_pack_params": (c_int, [P, P, P, P, P, P, P, P, P, c_int, c_int, c_int, c_int, c_int, P, P, P]),
    "mfb_nsf_unpack_grads": (c_int, [P, P, P, P, c_int, c_int, c_int, c_int, c_int, P, P, P, P, P, P, P]),
    "mfb_moments_workspace_bytes": (c_int64, [c_int64, c_int]),
    "mfb_moments": (c_int, [P, P, c_int64, c_int, c_int, P, P, c_int64, P]),
    "mfb_f64_split": (c_int, [P, c_int, P, P]),
    "mfb_f64_join": (c_int, [P, c_int, P, P]),
    "mfb_mc_entropy": (c_int, [P, c_double, c_double, c_double, P, P]),
    "mfb_loss_tail": (c_int, [P, c_int, P, c_float, P, P]),
    "mfb_knn_workspace_bytes": (c_int64, [c_int64, c_int, c_int]),
    "mfb_knn_kth": (c_int, [P, c_int64, c_int, c_int, c_double, P, P, P, P, c_int64, P]),
    "mfb_knn_kth_bwd": (c_int, [P, c_int64, c_int, P, P, P, P, c_double, P, P, P]),
    "mfb_knn_rows_workspace_bytes": (c_int64, [c_int64, c_int64, c_int, c_int]),
    "mfb_knn_kth_rows": (c_int, [P, c_int64, c_int, c_int, c_int64, c_int64, P, P, P, c_int64, P]),
    "mfb_knn_logsum": (c_int, [P, c_int64, c_double, P, P, c_int64, P]),
    "mfb_knn_kth_bwd_rows": (c_int, [P, c_int64, c_int, P, P, P, P, c_int64, c_int64, c_double, P, P, P]),
    "mfb_swd_workspace_bytes": (c_int64, [c_int64, c_int]),
    "mfb_swd_sort": (c_int, [P, c_int64, c_int, P, c_int, P, P, P, c_int64, P]),
    "mfb_swd_wpp": (c_int, [P, c_int64, c_int, P, c_int, P, c_int64, c_double, P, P, P, c_int64, P]),
    "mfb_swd_bwd": (c_int, [P, c_int64, c_int, P, c_int, P, P, P]),
    "mfb_nn_supported": (c_int, [c_int, c_int, c_int, c_int]),
    "mfb_nn_fwd": (c_int, [P, c_int64, c_int, c_int, c_int, c_int, P, P, P, P, P, P, P, P]),
    "mfb_nn_bwd_workspace_bytes": (c_int64, [c_int64, c_int, c_int, c_int, c_int]),
    "mfb_nn_bwd": (c_int, [P, P, c_int64, c_int, c_int, c_int, c_int, P, P, P, P, P, P, P, P, P, P, P, P, P, P,
                           c_int64, P]),
}

_lib = None


class LibraryMissing(RuntimeError):
    pass


def load():
    """Load ``libmentflow_b200.so`` (built by ``python -m mentflow_b200.build``)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise LibraryMissing(
            f"{LIB_PATH} not found. mentflow_b200 has no CPU/PyTorch fallback: build the CUDA "
            "library first with `python -m mentflow_b200.build` (needs nvcc, targets sm_100a).")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as e:
            raise LibraryMissing(f"{LIB_PATH} does not export {name}; rebuild it") from e
        fn.restype = res
        fn.argtypes = args
    # a library built from other sources may export the same names with other argument lists
    version = lib.mfb_abi_version()
    if version != ABI_VERSION:
        raise LibraryMissing(f"{LIB_PATH} has ABI version {version}, this package needs {ABI_VERSION}; rebuild it")
    _lib = lib
    return lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load().mfb_error_string(rc).decode()
        raise RuntimeError(f"mentflow_b200 {what} failed: {msg} (code {rc})")
