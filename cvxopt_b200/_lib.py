"""ctypes binding of the C-ABI shared library (include/cvxopt_b200.h).

The library is the product: there is NO CPU fallback.  If the shared object is
missing, or no sm_100 GPU is visible when a compute entry point is called, the
call fails loudly (RuntimeError) instead of routing anywhere else.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libcvxopt_b200.so")

HOST, DEVICE = 0, 1
E_ARG, E_CUDA, E_NOMEM, E_NOGPU, E_UNSUP = -1, -2, -3, -4, -5

c_double_p = C.POINTER(C.c_double)
c_int_p = C.POINTER(C.c_int)


class Dims(C.Structure):
    _fields_ = [("mnl", C.c_int), ("ml", C.c_int), ("nq", C.c_int), ("q", c_int_p),
                ("ns", C.c_int), ("s", c_int_p)]


class Scaling(C.Structure):
    _fields_ = [(name, C.c_void_p) for name in
                ("dnl", "dnli", "d", "di", "v", "beta", "r", "rti")]


_SIGS = {
    # name: (restype, argtypes)
    "cvxb_last_error": (C.c_char_p, []),
    "cvxb_device_count": (C.c_int, []),
    "cvxb_version": (C.c_int, []),
    "cvxb_launch_count": (C.c_ulonglong, []),
    "cvxb_malloc": (C.c_int, [C.POINTER(C.c_void_p), C.c_ulonglong]),
    "cvxb_free": (C.c_int, [C.c_void_p]),
    "cvxb_memcpy_h2d": (C.c_int, [C.c_void_p, C.c_void_p, C.c_ulonglong]),
    "cvxb_memcpy_d2h": (C.c_int, [C.c_void_p, C.c_void_p, C.c_ulonglong]),
    "cvxb_sync": (C.c_int, []),
    "cvxb_kkt_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_int, C.POINTER(Dims),
                                  C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int]),
    "cvxb_kkt_destroy": (None, [C.c_void_p]),
    "cvxb_kkt_reset": (C.c_int, [C.c_void_p]),
    "cvxb_kkt_set_method": (C.c_int, [C.c_void_p, C.c_int, C.c_double]),
    "cvxb_kkt_set_H": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int]),
    "cvxb_kkt_factor": (C.c_int, [C.c_void_p, C.POINTER(Scaling), C.c_void_p, C.c_int,
                                  C.c_void_p, C.c_int, C.c_int, C.c_int]),
    "cvxb_kkt_solve": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    "cvxb_kkt_get_L": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int]),
    "cvxb_kkt_last_ms": (C.c_int, [C.c_void_p, c_double_p, c_double_p]),
    "cvxb_kkt_timer_start": (C.c_int, [C.c_void_p]),
    "cvxb_kkt_timer_stop": (C.c_int, [C.c_void_p, c_double_p]),
    "cvxb_kkt_trace": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int]),
    "cvxb_kkt_last_breakdown": (C.c_int, [C.c_void_p, c_double_p]),
    "cvxb_kkt_syrk_mma_ms": (C.c_int, [C.c_void_p, c_double_p]),
    "cvxb_kkt_syrk_path": (C.c_int, [C.c_void_p]),
    "cvxb_kkt_qr_passes": (C.c_int, [C.c_void_p]),
    "cvxb_kkt_gemv_G": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_double,
                                  C.c_int, C.c_int]),
    "cvxb_kkt_gemv_A": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_double,
                                  C.c_int, C.c_int]),
    "cvxb_kkt_symv_H": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_double,
                                  C.c_int]),
    "cvxb_scale": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(Dims), C.POINTER(Scaling),
                             C.c_int, C.c_int, C.c_int]),
    "cvxb_scale2": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(Dims), C.c_int, C.c_int]),
    "cvxb_pack": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(Dims), C.c_int]),
    "cvxb_pack2": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(Dims), C.c_int]),
    "cvxb_unpack": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(Dims), C.c_int]),
    "cvxb_symm": (C.c_int, [C.c_void_p, C.c_int, C.c_int]),
    "cvxb_sprod": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(Dims), C.c_int, C.c_int]),
    "cvxb_sinv": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(Dims), C.c_int]),
    "cvxb_trisc": (C.c_int, [C.c_void_p, C.POINTER(Dims), C.c_int]),
    "cvxb_triusc": (C.c_int, [C.c_void_p, C.POINTER(Dims), C.c_int]),
    "cvxb_sdot": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(Dims), c_double_p, C.c_int]),
    "cvxb_max_step": (C.c_int, [C.c_void_p, C.POINTER(Dims), c_double_p, c_double_p, C.c_int]),
    "cvxb_compute_scaling": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(Dims), C.POINTER(Scaling),
                                       C.c_int]),
    "cvxb_update_scaling": (C.c_int, [C.POINTER(Scaling), C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(Dims),
                                      C.c_int]),
    "cvxb_syrk_scaled": (C.c_int, [C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                   C.c_int, C.c_void_p, C.c_int, C.c_int]),
    "cvxb_syrk_scaled_i8": (C.c_int, [C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                      C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int]),
    "cvxb_potrf": (C.c_int, [C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int]),
    "cvxb_potrs": (C.c_int, [C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int]),
    "cvxb_gemm": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, C.c_void_p,
                            C.c_int, C.c_void_p, C.c_int, C.c_double, C.c_void_p, C.c_int, C.c_int]),
    "cvxb_batch_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_int, C.c_int]),
    "cvxb_batch_create_eq": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]),
    "cvxb_batch_create_cones": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                          C.c_int, C.c_int]),
    "cvxb_batch_solve_ref": (C.c_int, [C.c_void_p, C.c_int, C.c_double, C.c_double, C.c_double, C.c_int]),
    "cvxb_batch_phase_ms_cones": (C.c_int, [C.c_void_p, c_double_p]),
    "cvxb_batch_destroy": (None, [C.c_void_p]),
    "cvxb_batch_load_eq": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    "cvxb_batch_results_y": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int]),
    "cvxb_batch_singular": (C.c_int, [C.c_void_p, C.c_void_p]),
    "cvxb_batch_phase_ms": (C.c_int, [C.c_void_p, c_double_p]),
    "cvxb_batch_load": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                  C.c_int]),
    "cvxb_batch_solve": (C.c_int, [C.c_void_p, C.c_int, C.c_double, C.c_double, C.c_double]),
    "cvxb_batch_stats": (C.c_int, [C.c_void_p, c_double_p, c_int_p]),
    "cvxb_batch_syrk_path": (C.c_int, [C.c_void_p]),
    "cvxb_batch_results": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
}

_lib = None


def load():
    """Load libcvxopt_b200.so (built by `make` / __graft_entry__.build())."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "cvxopt_b200: %s is missing — build it with `make` (nvcc, sm_100a). "
            "There is no CPU fallback for the KKT path." % LIB_PATH)
    lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    for name, (res, args) in _SIGS.items():
        fn = getattr(lib, name)          # AttributeError if the header and the .so diverge
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def exported_symbols():
    return sorted(_SIGS)


def last_error():
    return load().cvxb_last_error().decode("utf-8", "replace")


def check(rc, what=""):
    """Map a C return code onto the exception the reference raises for it."""
    if rc == 0:
        return
    msg = "%s%s" % (what + ": " if what else "", last_error())
    if rc > 0:
        # LAPACK info > 0: reference raises ArithmeticError (src/C/lapack.c:32-34)
        raise ArithmeticError(rc)
    if rc == E_ARG:
        raise ValueError(msg)
    if rc == E_UNSUP:
        raise NotImplementedError(msg)
    if rc == E_NOMEM:
        raise MemoryError(msg)
    raise RuntimeError(msg)
