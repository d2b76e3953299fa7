"""ctypes binding of libalabi_b200.so (include/alabi_b200.h).

This is the thin C-ABI layer north_star asks for: Python host code reaches the
sm_100a kernels only through the ``extern "C"`` entry points below; torch
tensors are nothing but the carrier of device buffers (``data_ptr()``) and of
the current stream.  There is no CPU fallback: ``load()`` raises if the
library has not been built and every compute call needs a CUDA device.
"""
import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# ALABI_B200_LIB: load another build of the library instead (compare two builds from one tree)
LIB_PATH = os.environ.get("ALABI_B200_LIB") or os.path.join(HERE, "libalabi_b200.so")

c_double_p = ctypes.POINTER(ctypes.c_double)
c_int64_p = ctypes.POINTER(ctypes.c_int64)
MAX_DIM = 32
MAX_PEERS = 15
PEER_HANDLE_BYTES = 64


class EnsembleConfig(ctypes.Structure):
    """Mirror of ``ab_ensemble_config``."""
    _fields_ = [("nwalkers", ctypes.c_int), ("nsteps", ctypes.c_int), ("thin_by", ctypes.c_int),
                ("init_logp", ctypes.c_int), ("randomize_split", ctypes.c_int),
                ("warps_per_unit", ctypes.c_int), ("y_kind", ctypes.c_int), ("reserved", ctypes.c_int),
                ("a", ctypes.c_double), ("seed", ctypes.c_uint64), ("first_step", ctypes.c_int64),
                ("walker_offset", ctypes.c_int64), ("y_scale", ctypes.c_double), ("y_offset", ctypes.c_double),
                ("lo", ctypes.c_double * MAX_DIM), ("hi", ctypes.c_double * MAX_DIM),
                ("theta_scale", ctypes.c_double * MAX_DIM), ("theta_offset", ctypes.c_double * MAX_DIM),
                ("use_normal_prior", ctypes.c_int), ("schedule", ctypes.c_int),
                ("prior_mu", ctypes.c_double * MAX_DIM), ("prior_sd", ctypes.c_double * MAX_DIM),
                ("chain_row_walkers", ctypes.c_int64), ("chain_walker_offset", ctypes.c_int64),
                ("n_chain_peers", ctypes.c_int), ("reserved3", ctypes.c_int),
                ("chain_peers", ctypes.c_void_p * MAX_PEERS), ("logp_chain_peers", ctypes.c_void_p * MAX_PEERS)]


class NestedConfig(ctypes.Structure):
    """Mirror of ``ab_nested_config``."""
    _fields_ = [("nchains", ctypes.c_int), ("walks", ctypes.c_int), ("y_kind", ctypes.c_int),
                ("use_normal_prior", ctypes.c_int), ("scale", ctypes.c_double), ("lmin", ctypes.c_double),
                ("seed", ctypes.c_uint64), ("counter", ctypes.c_int64), ("chain_offset", ctypes.c_int64),
                ("y_scale", ctypes.c_double), ("y_offset", ctypes.c_double),
                ("lo", ctypes.c_double * MAX_DIM), ("hi", ctypes.c_double * MAX_DIM),
                ("prior_mu", ctypes.c_double * MAX_DIM), ("prior_sd", ctypes.c_double * MAX_DIM),
                ("theta_scale", ctypes.c_double * MAX_DIM), ("theta_offset", ctypes.c_double * MAX_DIM),
                ("chol", ctypes.c_double * (MAX_DIM * MAX_DIM))]


# name -> (restype, argtypes); every symbol include/alabi_b200.h declares
_P = ctypes.c_void_p
SIGNATURES = {
    "ab_version": (ctypes.c_int, []),
    "ab_sizeof_ensemble_config": (ctypes.c_int, []),
    "ab_last_error": (ctypes.c_char_p, []),
    "ab_device_sm_count": (ctypes.c_int, [ctypes.c_int]),
    "ab_launch_counter": (ctypes.c_longlong, []),
    "ab_fp64_tensor_peak": (ctypes.c_int, [ctypes.c_int, c_double_p]),
    "ab_fp64_fma_peak": (ctypes.c_int, [ctypes.c_int, c_double_p]),
    "ab_gp_set_profiling": (ctypes.c_int, [_P, ctypes.c_int]),
    "ab_gp_profile_read": (ctypes.c_int, [_P, ctypes.c_int, c_double_p, ctypes.POINTER(ctypes.c_longlong)]),
    "ab_gp_create": (ctypes.c_int, [ctypes.POINTER(_P), ctypes.c_int, _P]),
    "ab_gp_destroy": (ctypes.c_int, [_P]),
    "ab_gp_set_few_query_path": (ctypes.c_int, [_P, ctypes.c_int]),
    "ab_gp_append_point": (ctypes.c_int, [_P, _P]),
    "ab_gp_predict_grad": (ctypes.c_int, [_P, _P, ctypes.c_int64, _P, _P, _P, _P]),
    "ab_gp_set_inputs": (ctypes.c_int, [_P, _P, ctypes.c_int64, ctypes.c_int]),
    "ab_gp_set_kernel": (ctypes.c_int, [_P, ctypes.c_int, ctypes.c_double, c_double_p, ctypes.c_double,
                                        ctypes.c_double, ctypes.c_double]),
    "ab_gp_set_kernel_rq": (ctypes.c_int, [_P, ctypes.c_double, ctypes.c_double, c_double_p, ctypes.c_double,
                                           ctypes.c_double, ctypes.c_double]),
    "ab_gp_build_cov": (ctypes.c_int, [_P, _P, ctypes.c_int]),
    "ab_gp_cross_cov": (ctypes.c_int, [_P, _P, ctypes.c_int64, _P, ctypes.c_int64, _P]),
    "ab_gp_factor": (ctypes.c_int, [_P]),
    "ab_gp_log_determinant": (ctypes.c_int, [_P, c_double_p]),
    "ab_gp_set_targets": (ctypes.c_int, [_P, _P]),
    "ab_gp_log_likelihood": (ctypes.c_int, [_P, _P, c_double_p]),
    "ab_gp_grad_log_likelihood": (ctypes.c_int, [_P, _P, c_double_p]),
    "ab_gp_predict": (ctypes.c_int, [_P, _P, ctypes.c_int64, _P, _P]),
    "ab_gp_predict_cov": (ctypes.c_int, [_P, _P, ctypes.c_int64, _P, _P, ctypes.c_int64]),
    "ab_mvn_sample": (ctypes.c_int, [_P, _P, ctypes.c_int64, ctypes.c_int64, _P, ctypes.c_double, ctypes.c_int64,
                                     ctypes.c_uint64, _P, ctypes.POINTER(ctypes.c_int)]),
    "ab_gp_predict_host": (ctypes.c_int, [_P, _P, ctypes.c_int64, _P, _P]),
    "ab_gp_utility_argmin": (ctypes.c_int, [_P, ctypes.c_int, _P, ctypes.c_int64, c_double_p, ctypes.c_double,
                                            ctypes.c_double, _P, c_int64_p, c_double_p]),
    "ab_utility_eval": (ctypes.c_int, [_P, ctypes.c_int, _P, _P, _P, ctypes.c_int64, c_double_p, ctypes.c_double,
                                       ctypes.c_double, _P, c_int64_p, c_double_p]),
    "ab_gp_padded_size": (ctypes.c_int64, [_P]),
    "ab_gp_get_factor": (ctypes.c_int, [_P, _P]),
    "ab_gp_get_alpha": (ctypes.c_int, [_P, _P]),
    "ab_gp_get_inverse": (ctypes.c_int, [_P, _P]),
    "ab_gp_import_state": (ctypes.c_int, [_P, _P, _P]),
    "ab_gp_get_block_inverses": (ctypes.c_int, [_P, _P]),
    "ab_gp_import_state_full": (ctypes.c_int, [_P, _P, _P, _P]),
    "ab_ensemble_run": (ctypes.c_int, [_P, ctypes.POINTER(EnsembleConfig), _P, _P, _P, _P, _P, _P, _P]),
    "ab_ensemble_launch": (ctypes.c_int, [_P, ctypes.POINTER(EnsembleConfig), _P, _P, _P, _P, _P, _P, _P]),
    "ab_ensemble_finish": (ctypes.c_int, [_P]),
    "ab_gp_cv_batch": (ctypes.c_int, [_P, _P, _P, ctypes.c_int64, ctypes.c_int, ctypes.c_int, ctypes.c_int, c_double_p,
                                      ctypes.c_int, ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int),
                                      ctypes.POINTER(ctypes.c_int), _P, ctypes.c_int, _P, ctypes.c_int, _P, c_double_p,
                                      ctypes.POINTER(ctypes.c_int), _P, ctypes.c_size_t]),
    "ab_gp_cv_workspace_bytes": (ctypes.c_size_t, [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int]),
    "ab_nccl_unique_id": (ctypes.c_int, [ctypes.POINTER(ctypes.c_ubyte)]),
    "ab_nccl_init": (ctypes.c_int, [ctypes.POINTER(_P), ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_ubyte),
                                    ctypes.c_int, _P]),
    "ab_nccl_destroy": (ctypes.c_int, [_P]),
    "ab_nccl_sync": (ctypes.c_int, [_P]),
    "ab_nccl_broadcast": (ctypes.c_int, [_P, _P, ctypes.c_int64, ctypes.c_int]),
    "ab_nccl_allgather": (ctypes.c_int, [_P, _P, _P, ctypes.c_int64]),
    "ab_nccl_broadcast_gp": (ctypes.c_int, [_P, _P, ctypes.c_int]),
    "ab_peer_alloc": (ctypes.c_int, [ctypes.c_int, ctypes.c_size_t, ctypes.POINTER(_P), ctypes.POINTER(ctypes.c_ubyte)]),
    "ab_peer_open": (ctypes.c_int, [ctypes.c_int, ctypes.POINTER(ctypes.c_ubyte), ctypes.POINTER(_P)]),
    "ab_peer_close": (ctypes.c_int, [ctypes.c_int, _P]),
    "ab_peer_free": (ctypes.c_int, [ctypes.c_int, _P]),
    "ab_sizeof_nested_config": (ctypes.c_int, []),
    "ab_nested_walk": (ctypes.c_int, [_P, ctypes.POINTER(NestedConfig), _P, _P, _P, _P]),
    "ab_nested_rslice": (ctypes.c_int, [_P, ctypes.POINTER(NestedConfig), _P, _P, _P, _P]),
    "ab_ensemble_run_host": (ctypes.c_int, [_P, ctypes.POINTER(EnsembleConfig), _P, _P, _P, _P, _P, _P, _P, ctypes.c_int]),
}

_lib = None


class AlabiB200Error(RuntimeError):
    pass


def load():
    """Load the shared library (once).  Raises if it is missing: the product
    path never falls back to a CPU implementation."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise AlabiB200Error(f"{LIB_PATH} not found — build it with `python -m alabi_b200.build` "
                             "(nvcc, sm_100a); there is no CPU fallback")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.ab_sizeof_ensemble_config() != ctypes.sizeof(EnsembleConfig):
        raise AlabiB200Error(f"{LIB_PATH} is stale: ab_ensemble_config is {lib.ab_sizeof_ensemble_config()} bytes there, "
                             f"{ctypes.sizeof(EnsembleConfig)} here — rebuild with `python -m alabi_b200.build`")
    if lib.ab_sizeof_nested_config() != ctypes.sizeof(NestedConfig):
        raise AlabiB200Error(f"{LIB_PATH} is stale: ab_nested_config size mismatch — rebuild with `python -m alabi_b200.build`")
    _lib = lib
    return lib


def last_error():
    return load().ab_last_error().decode("utf-8", "replace")


def check(rc, what):
    """Negative return codes are errors; positive ones are numerical statuses
    handled by the caller."""
    if rc < 0:
        raise AlabiB200Error(f"{what} failed (code {rc}): {last_error()}")
    return rc


def ptr(t):
    """Device (or host) address of a torch tensor / numpy array, or NULL."""
    if t is None:
        return None
    if hasattr(t, "data_ptr"):
        return ctypes.c_void_p(t.data_ptr())
    return ctypes.c_void_p(t.ctypes.data)
