"""ctypes binding of libkrylov_b200.so (C ABI in include/krylov_b200.h).

The shared library is built in-tree by ``__graft_entry__.build()`` /
``krylov_robustness_b200/csrc/build.sh``.  There is NO CPU fallback: if the library is missing,
or no B200 is visible, every entry point raises.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("KR_B200_LIB", os.path.join(_HERE, "libkrylov_b200.so"))   # override: tuning builds

c_i64 = C.c_int64
c_dp = C.POINTER(C.c_double)
c_ip = C.POINTER(C.c_int64)
c_intp = C.POINTER(C.c_int)
VP = C.c_void_p

# name -> argtypes (restype is int unless listed in _RESTYPE)
PROTOTYPES = {
    "kr_last_error": [],
    "kr_version": [],
    "kr_ctx_create": [C.c_int, C.POINTER(VP)],
    "kr_ctx_destroy": [VP],
    "kr_ctx_sync": [VP],
    "kr_ctx_counters": [VP, c_ip],
    "kr_ctx_set_timing": [VP, C.c_int],
    "kr_ctx_spmm_time": [VP, C.c_int, c_dp, c_ip],
    "kr_ctx_stream": [VP],
    "kr_matrix_create": [VP, c_i64, c_i64, VP, VP, VP, C.POINTER(VP)],
    "kr_matrix_destroy": [VP],
    "kr_matrix_info": [VP, c_ip, c_ip, c_intp, c_intp, c_intp],
    "kr_matrix_set_edges": [VP, c_i64, VP, VP, VP],
    "kr_dense_create": [VP, c_i64, c_i64, C.POINTER(VP)],
    "kr_dense_destroy": [VP],
    "kr_dense_upload": [VP, VP, c_i64],
    "kr_dense_download": [VP, VP, c_i64],
    "kr_dense_fill_rademacher": [VP, C.c_uint64, c_i64],
    "kr_spmm": [VP, VP, c_i64, VP, c_i64, VP, c_i64],
    "kr_matrix_replicate": [VP, C.c_int, VP],
    "kr_matrix_replicas": [VP],
    "kr_spmm_dev": [VP, VP, VP, VP],
    "kr_krylov_start": [VP, VP, C.c_int, c_i64, VP, c_i64, C.POINTER(VP), c_intp],
    "kr_krylov_extend": [VP, c_intp],
    "kr_krylov_dims": [VP, c_ip],
    "kr_krylov_get": [VP, VP, c_i64, VP, c_i64, VP, c_i64, VP, c_i64],
    "kr_krylov_destroy": [VP],
    "kr_trace_fun_update": [VP, VP, c_i64, VP, c_i64, VP, c_i64, C.c_double, c_i64, C.c_int,
                            c_dp, c_ip, c_intp],
    "kr_trace_fun_update_edges": [VP, VP, c_i64, VP, C.c_double, C.c_double, c_i64, C.c_int,
                                  VP, VP, VP],
    "kr_trace_fun_update_edges_ex": [VP, VP, c_i64, VP, C.c_double, C.c_double, C.c_double, c_i64, C.c_int,
                                     VP, VP, VP],
    "kr_trace_fun_update_nodes": [VP, VP, c_i64, VP, C.c_double, c_i64, C.c_int, VP, VP, VP],
    "kr_greedy_round": [VP, VP, c_i64, VP, C.c_double, C.c_double, C.c_double, c_i64, C.c_int, C.c_int, C.c_int,
                        c_ip, c_dp, VP, VP, VP],
    "kr_fun_update": [VP, VP, c_i64, VP, c_i64, VP, c_i64, C.c_int, C.c_double, c_i64, C.c_int,
                      c_ip, c_ip, c_intp, c_intp],
    "kr_fun_update_fetch": [VP, VP, c_i64, VP, c_i64],
    "kr_function_multiple_entries": [VP, VP, c_i64, VP, C.c_int, C.c_double, c_i64, VP, c_ip],
    "kr_trace_fun_sparse_update": [VP, VP, c_i64, VP, VP, C.c_int, C.c_double, c_i64, c_i64, VP, VP, VP, VP],
    "kr_fun_and_grad_krylov": [VP, VP, c_i64, VP, VP, C.c_int, C.c_int, VP, C.c_double, c_i64,
                               c_dp, VP],
    "kr_frechet_hessian": [VP, VP, c_i64, VP, C.c_int, C.c_double, c_i64, VP, c_ip],
    "kr_frechet_hessian_multiply": [VP, VP, c_i64, VP, c_i64, VP, c_i64, C.c_int, C.c_int, C.c_double, c_i64, VP,
                                    c_i64, c_ip, VP],
    "kr_normest": [VP, VP, C.c_double, c_dp, c_ip],
    "kr_compute_centrality": [VP, VP, C.c_int, C.c_double, c_i64, VP, c_ip, c_intp],
    "kr_normAm": [VP, VP, C.c_double, c_i64, c_dp, c_ip],
    "kr_select_taylor_degree": [VP, VP, C.c_double, c_i64, c_i64, c_i64, C.c_int, C.c_int,
                                VP, c_ip, VP, c_intp],
    "kr_expmv": [VP, VP, C.c_double, c_i64, VP, c_i64, VP, c_i64, c_i64, C.c_int, C.c_int,
                 VP, c_i64, c_ip, c_ip, c_ip, c_ip, c_intp],
    "kr_theta": [VP],
    "kr_mc_trace": [VP, VP, C.c_int, C.c_double, c_i64, VP, c_dp, c_dp, c_ip],
    "kr_slq_trace": [VP, VP, c_i64, VP, c_i64, c_i64, C.c_int, c_dp, VP, VP, VP],
    "kr_slq_trace_sign": [VP, VP, c_i64, VP, c_i64, c_i64, C.c_int, c_dp, VP, VP, VP],
    "kr_slq_trace_dev": [VP, VP, VP, c_i64, C.c_int, c_dp, VP, VP, VP],
}
_RESTYPE = {"kr_last_error": C.c_char_p, "kr_version": C.c_char_p, "kr_ctx_destroy": None,
            "kr_matrix_destroy": None, "kr_dense_destroy": None, "kr_krylov_destroy": None,
            "kr_ctx_stream": VP}

_lib = None


class KrylovB200Error(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(msg)
        self.code = code


def load():
    """Load the shared library (idempotent).  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise KrylovB200Error(-2, "libkrylov_b200.so not built (%s); run __graft_entry__.build() - "
                                  "there is no CPU fallback" % LIB_PATH)
    lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    for name, args in PROTOTYPES.items():
        fn = getattr(lib, name)          # AttributeError if the header and the library disagree
        fn.argtypes = args
        fn.restype = _RESTYPE.get(name, C.c_int)
    _lib = lib
    return lib


def check(status):
    if status != 0:
        msg = load().kr_last_error()
        raise KrylovB200Error(status, msg.decode() if msg else "krylov_b200 error %d" % status)
