"""ctypes binding of the C ABI (include/limbo_b200.h).  There is no CPU fallback:
if the CUDA library is missing or no device is present every call fails loudly."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "lib", "liblimbo_b200.so")

LB_OK = 0
ERR_NAMES = {-1: "LB_ERR_ARG", -2: "LB_ERR_CUDA", -3: "LB_ERR_STATE", -4: "LB_ERR_ALLOC", -5: "LB_ERR_UNSUPPORTED",
             -6: "LB_ERR_TIMEOUT"}

KERNEL_SQUARED_EXP_ARD, KERNEL_MATERN_FIVE_HALVES, KERNEL_MATERN_THREE_HALVES, KERNEL_EXP = 0, 1, 2, 3
ACQ_UCB, ACQ_EI = 0, 1
GET_K, GET_L, GET_ALPHA, GET_KINV = 0, 1, 2, 3

# every symbol include/limbo_b200.h declares
DECLARED_SYMBOLS = [
    "lb_create", "lb_destroy", "lb_clone", "lb_set_stream", "lb_sync", "lb_launch_count", "lb_set_data",
    "lb_set_data_dev", "lb_set_kernel", "lb_fit", "lb_load_factor", "lb_refit_alpha", "lb_append", "lb_query", "lb_query_dev",
    "lb_acq_argmax", "lb_acq_argmax_dev", "lb_log_lik", "lb_kernel_grad_log_lik", "lb_compute_inv_kernel", "lb_log_loo_cv",
    "lb_kernel_grad_log_loo_cv", "lb_kinv_obs_mean", "lb_sparsify", "lb_get",
    "lb_nb_samples", "lb_strerror", "lb_last_cuda_error",
]

_lib = None


class LimboB200Error(RuntimeError):
    def __init__(self, code: int, where: str):
        self.code = code
        lib = load()
        msg = lib.lb_strerror(code).decode()
        cuda = lib.lb_last_cuda_error().decode() if code == -2 else ""
        super().__init__(f"{where}: {ERR_NAMES.get(code, code)}: {msg} {cuda}".strip())


class NotPositiveDefinite(LimboB200Error):
    """lb_fit / lb_append returned info > 0 (1-based index of the failing pivot)."""


def load() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(limbo_b200 has no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    p, i64, i32, dbl = C.c_void_p, C.c_int64, C.c_int, C.c_double
    dp = C.c_void_p  # raw addresses (numpy / torch data_ptr)
    sig = {
        "lb_create": ([C.POINTER(p), i32, i32], i32),
        "lb_destroy": ([p], i32),
        "lb_clone": ([p, C.POINTER(p)], i32),
        "lb_set_stream": ([p, p], i32),
        "lb_sync": ([p], i32),
        "lb_launch_count": ([p], C.c_longlong),
        "lb_debug_append_count": ([p], C.c_longlong),
        "lb_debug_pool_mallocs": ([], C.c_longlong),
        "lb_debug_pool_hits": ([], C.c_longlong),
        "lb_pool_trim": ([], i32),
        "lb_debug_set_query_panel_min": ([C.c_longlong], i32),
        "lb_debug_set_query_int8": ([C.c_int, C.c_longlong], i32),
        "lb_set_data": ([p, i64, i32, i32, dp, dp], i32),
        "lb_set_data_dev": ([p, i64, i32, i32, dp, dp], i32),
        "lb_set_kernel": ([p, i32, dp, i32, dbl], i32),
        "lb_fit": ([p], i32),
        "lb_fit_async": ([p], i32),
        "lb_check_info": ([p], i32),
        "lb_stage_kbuild": ([p], i32),
        "lb_stage_potrf": ([p], i32),
        "lb_stage_alpha": ([p], i32),
        "lb_refit_alpha": ([p, dp], i32),
        "lb_load_factor": ([p, dp, dp], i32),
        "lb_append": ([p, dp, dp], i32),
        "lb_query": ([p, i64, dp, dp, dp], i32),
        "lb_query_dev": ([p, i64, dp, dp, dp], i32),
        "lb_acq_argmax": ([p, i32, dp, i64, dp, dp, dbl, dp, dp, dp], i32),
        "lb_acq_argmax_dev": ([p, i32, dp, i64, dp, dp, dbl, dp, dp, dp], i32),
        "lb_log_lik": ([p, dp], i32),
        "lb_kernel_grad_log_lik": ([p, i32, dp], i32),
        "lb_compute_inv_kernel": ([p], i32),
        "lb_log_loo_cv": ([p, dp], i32),
        "lb_kernel_grad_log_loo_cv": ([p, i32, dp], i32),
        "lb_kinv_obs_mean": ([p, dp], i32),
        "lb_sparsify": ([p, i64, i32, dp, i64, dp, dp, dp], i32),
        "lb_get": ([p, i32, dp], i32),
        "lb_nb_samples": ([p], i64),
        "lb_strerror": ([i32], C.c_char_p),
        "lb_last_cuda_error": ([], C.c_char_p),
    }
    for name, (argtypes, restype) in sig.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = restype
    _lib = lib
    return lib


def check(code: int, where: str) -> None:
    if code == LB_OK:
        return
    if code > 0:
        raise NotPositiveDefinite(code, where)
    raise LimboB200Error(code, where)
