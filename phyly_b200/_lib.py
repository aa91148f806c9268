"""
ctypes loader for libarbplf_b200.so (built in-tree by phyly_b200/csrc/Makefile
or __graft_entry__.build()).  There is no fallback: if the CUDA library is
missing, importing anything that needs it raises.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libarbplf_b200.so")

_lib = None


class EngineUnavailable(RuntimeError):
    pass


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise EngineUnavailable(
            "%s not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(there is no CPU fallback)" % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH, mode=ctypes.RTLD_GLOBAL)
    c = ctypes
    P = c.c_void_p
    lib.plf_create.argtypes = [c.POINTER(P), c.c_int]
    lib.plf_create.restype = c.c_int
    lib.plf_destroy.argtypes = [P]
    lib.plf_destroy.restype = None
    lib.plf_last_error.argtypes = [P]
    lib.plf_last_error.restype = c.c_char_p
    lib.plf_set_path.argtypes = [P, c.c_int]
    lib.plf_set_tree.argtypes = [P, c.c_int, P, P, P]
    lib.plf_set_model.argtypes = [P, c.c_int, c.c_int, P, P, P, P, P, c.c_int, P]
    lib.plf_set_edge_rates.argtypes = [P, P]
    lib.plf_set_data.argtypes = [P, c.c_int64, c.c_int, P, P, c.c_int]
    lib.plf_set_data_async.argtypes = [P, c.c_int64, c.c_int, P, P, c.c_int, P]
    lib.plf_set_site_weights.argtypes = [P, P]
    lib.plf_ll.argtypes = [P, P, P]
    lib.plf_deriv.argtypes = [P, P, P, P, P, P]
    lib.plf_marginal.argtypes = [P, P, P]
    lib.plf_edge_expect.argtypes = [P, c.c_int, P, P, P, P, P]
    lib.plf_edge_expect_all.argtypes = [P, P, P, P]
    lib.plf_get_transition_matrices.argtypes = [P, P]
    lib.plf_get_derivative_matrices.argtypes = [P, P]
    lib.plf_get_frechet_matrices.argtypes = [P, P, P, P]
    lib.plf_last_timing.argtypes = [P, c.POINTER(c.c_float), c.POINTER(c.c_float)]
    lib.plf_last_kernel_ms.argtypes = [P, c.POINTER(c.c_float)]
    lib.plf_last_kernel_ms.restype = c.c_int
    lib.plf_launch_count.argtypes = [P, c.c_int]
    lib.plf_launch_count.restype = c.c_int64
    lib.plf_last_kernel_name.argtypes = [P]
    lib.plf_last_kernel_name.restype = c.c_char_p
    lib.plf_comm_pause.argtypes = [P, c.c_int]
    lib.plf_comm_pause.restype = c.c_int
    lib.plf_compress_patterns.argtypes = [P, c.c_int64, c.c_int, P, c.c_int, c.POINTER(c.c_int64), P, P, P]
    lib.plf_compress_patterns.restype = c.c_int
    lib.plf_ll_certified.argtypes = [P, c.c_double, c.c_double, P, P, P, P]
    lib.plf_ll_certified.restype = c.c_int
    lib.plf_deriv_certified.argtypes = [P, c.c_double, c.c_double, P, P, P, P, P]
    lib.plf_deriv_certified.restype = c.c_int
    lib.plf_marginal_certified.argtypes = [P, c.c_double, c.c_double, P, P, P, P]
    lib.plf_marginal_certified.restype = c.c_int
    lib.plf_edge_expect_certified.argtypes = [P, c.c_double, c.c_double, c.c_int, P, P, P, P, P, P, P]
    lib.plf_edge_expect_certified.restype = c.c_int
    lib.plf_hess.argtypes = [P, P, P, P]
    lib.plf_hess.restype = c.c_int
    lib.plf_comm_unique_id.argtypes = [c.c_char_p]
    lib.plf_comm_init.argtypes = [P, c.c_int, c.c_int, c.c_char_p]
    lib.plf_stream.argtypes = [P]
    lib.plf_stream.restype = P
    lib.plf_synchronize.argtypes = [P]
    for name in ("plf_set_path", "plf_set_tree", "plf_set_model", "plf_set_edge_rates", "plf_set_data", "plf_set_data_async",
                 "plf_set_site_weights", "plf_ll", "plf_deriv", "plf_marginal", "plf_edge_expect", "plf_edge_expect_all",
                 "plf_get_transition_matrices", "plf_get_derivative_matrices", "plf_get_frechet_matrices",
                 "plf_last_timing", "plf_comm_unique_id", "plf_comm_init", "plf_synchronize"):
        getattr(lib, name).restype = c.c_int
    _lib = lib
    return lib
