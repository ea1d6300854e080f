"""
ctypes binding of libava_b200.so (the C ABI declared in include/ava_b200.h).

There is no CPU fallback: if the library is missing, or a call fails, this raises.
"""
import ctypes
import os
from ctypes import c_double, c_float, c_int, c_longlong, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libava_b200.so")

_lib = None

I, LL, F, D, P = c_int, c_longlong, c_float, c_double, c_void_p

# name -> (argtypes); every entry returns int unless listed in _RESTYPES
SIGNATURES = {
    "ava_b200_channel_stats": (P, I, I, I, P, P),
    "ava_b200_bn_update_running": (P, P, P, P, P, P, P, F, P),
    "ava_b200_bnconv_fwd": (I, I, P, P, P, P, P, P, P, P, P, I, P, P),
    "ava_b200_dz_border_sums": (P, I, I, I, I, I, P, P),
    "ava_b200_bnconv_bwd_data": (I, I, P, P, P, P, P, P, I, P, P, P),
    "ava_b200_bnconv_bwd_weight": (I, I, P, P, P, P, P, P, P, P, P, P, P, P),
    "ava_b200_bnconv_bwd_weight_ws": (I, I),
    "ava_b200_bnconv_bwd_data_ex": (I, I, P, P, P, P, P, P, I, P, I, P, P, P),
    "ava_b200_bnconv_bwd_weight_ex": (I, I, P, P, P, P, P, P, P, P, I, P, P, P, P, P, P),
    "ava_b200_set_conv_precision": (I,),
    "ava_b200_get_conv_precision": (),
    "ava_b200_bn_param_grads": (P, P, P, P, P, P, P, P),
    "ava_b200_bn_param_grads_ex": (P, P, P, P, P, P, P, P, P, I, P),
    "ava_b200_bn_relu_bwd_apply": (P, P, P, P, P, I, I, I, I, P, P, I, P),
    "ava_b200_linear_fwd": (P, I, P, P, P, I, I, I, I, I, I, LL, LL, LL, LL, I, P, LL, P),
    "ava_b200_linear_bwd_data": (P, I, P, P, P, I, I, I, I, I, LL, LL, LL, I, I, P, LL, P),
    "ava_b200_linear_bwd_weight": (P, I, P, P, I, P, P, I, I, I, I, LL, LL, LL, LL, I, P, LL, P),
    "ava_b200_linear_ws_bytes": (I, I, I),
    "ava_b200_bias_grads": (P, I, P, LL, P),
    "ava_b200_bias_grads_ws_bytes": (P, I),
    "ava_b200_latent_fwd": (P, P, P, I, I, P, P, P, P),
    "ava_b200_latent_bwd": (P, P, P, P, P, I, I, P, P),
    "ava_b200_latent_heads_grad": (P, P, P, P, I, I, P, P),
    "ava_b200_recon_input_grad": (P, P, P, LL, F, P, P),
    "ava_b200_recon": (P, P, LL, F, P, P, P, I, I, P),
    "ava_b200_elbo_finalize": (P, I, I, F, P, P, P),
    "ava_b200_adam_step": (P, P, P, P, LL, P, D, D, D, D, F, P),
    "ava_b200_adam_step_dev": (P, P, P, P, LL, P, P, F, P),
    "ava_b200_adam_step_dp": (P, I, I, P, P, LL, P, P, F, P, P),
    "ava_b200_bn_stats_exchange": (P, I, I, P, I, LL, P, I, I, P, F, P, P),
    "ava_b200_get_spec_batch": (P, I, P, P, I, I, I, I, P, D, P, P, I, P, P, I, I, D, D, P, P, P),
    "ava_b200_quantile_normalize": (P, P, I, I, D, P),
    "ava_b200_window_time_tables": (P, P, P, I, P, P, I, I, P, P, P),
    "ava_b200_mmd_block_sums": (P, I, I, P, I, D, P, P),
    "ava_b200_pair_kernel": (P, I, P, P, LL, D, I, P, P),
    "ava_b200_pca_ws_bytes": (I,),
    "ava_b200_pca_fit": (P, I, LL, I, P, P, P, P, P, LL, P),
    "ava_b200_pca_transform": (P, I, LL, I, P, P, I, P, P),
    "ava_b200_umap_knn_ws_bytes": (I, I, I),
    "ava_b200_umap_knn": (P, I, I, I, I, P, P, P, LL, P),
    "ava_b200_umap_smooth_knn": (P, P, I, I, D, P, P, P, P, P),
    "ava_b200_umap_edge_keys": (P, I, I, P, P),
    "ava_b200_umap_graph": (P, LL, I, P, P, I, P, P, P, P, P),
    "ava_b200_umap_epochs_per_sample": (P, LL, P, I, D, P, P, P, P, P),
    "ava_b200_umap_components_step": (P, P, I, P, P, P),
    "ava_b200_umap_degree": (P, P, I, P, P),
    "ava_b200_umap_spmm": (P, P, P, P, I, P, P, P, I, P, P),
    "ava_b200_umap_gram_ws_bytes": (I, I),
    "ava_b200_umap_gram": (P, I, P, I, I, P, P, LL, P),
    "ava_b200_umap_combine": (P, I, P, I, I, P, P),
    "ava_b200_umap_random": (ctypes.c_ulonglong, ctypes.c_ulonglong, LL, I, D, P, P),
    "ava_b200_umap_init_layout": (P, P, D, I, I, P, P),
    "ava_b200_umap_sgd_epoch": (P, I, I, P, P, P, P, P, P, LL, LL, I, D, D, D, D, ctypes.c_ulonglong, P),
    "ava_b200_umap_knn_query_ws_bytes": (I, I, I, I),
    "ava_b200_umap_knn_query": (P, I, P, I, I, I, I, P, P, P, LL, P),
    "ava_b200_umap_smooth_knn_query": (P, P, I, I, D, P, P, P, P, P),
    "ava_b200_umap_init_transform": (P, P, I, I, P, I, I, P, P),
    "ava_b200_umap_sgd_transform": (P, I, P, I, I, P, P, P, P, P, P, I, D, D, D, D, ctypes.c_ulonglong, P),
    "ava_b200_last_error": (),
    "ava_b200_abi_version": (),
    "ava_b200_launch_count": (),
}
_RESTYPES = {
    "ava_b200_last_error": ctypes.c_char_p,
    "ava_b200_launch_count": LL,
    "ava_b200_bnconv_bwd_weight_ws": LL,
    "ava_b200_linear_ws_bytes": LL,
    "ava_b200_bias_grads_ws_bytes": LL,
    "ava_b200_pca_ws_bytes": LL,
    "ava_b200_umap_knn_ws_bytes": LL,
    "ava_b200_umap_gram_ws_bytes": LL,
    "ava_b200_umap_knn_query_ws_bytes": LL,
}
# entry points whose int return value is a status code
_STATUS = {n for n in SIGNATURES if n not in _RESTYPES and n not in ("ava_b200_abi_version", "ava_b200_get_conv_precision")}


class AvaB200Error(RuntimeError):
    pass


def lib():
    """Load (once) and return the ctypes handle; raise if the library is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise AvaB200Error(
            "libava_b200.so not found at %s -- build it with "
            "`python __graft_entry__.py` (nvcc, sm_100a). There is no CPU fallback." % LIB_PATH)
    handle = ctypes.CDLL(LIB_PATH)
    for name, args in SIGNATURES.items():
        fn = getattr(handle, name)  # AttributeError if the header and the .so disagree
        fn.argtypes = list(args)
        fn.restype = _RESTYPES.get(name, c_int)
    _lib = handle
    return _lib


def last_error():
    return lib().ava_b200_last_error().decode("utf-8", "replace")


def launch_count():
    return int(lib().ava_b200_launch_count())


# Optional per-call hook used by bench.py to time each native call with CUDA events on
# the launching stream: an object with begin(name, args) / end(name, args).
PROFILER = None


def call(name, *args):
    """Call a status-returning entry point; raise AvaB200Error on failure."""
    prof = PROFILER
    if prof is not None:
        prof.begin(name, args)
    rc = getattr(lib(), name)(*args)
    if prof is not None:
        prof.end(name, args)
    if rc != 0:
        raise AvaB200Error("%s failed: %s" % (name, last_error()))


def ptr(t):
    """Device pointer of a torch tensor (or None -> NULL)."""
    if t is None:
        return None
    return t.data_ptr()
