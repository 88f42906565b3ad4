"""ctypes loader of libb200pde.so (the C ABI of include/b200pde.h).

There is no CPU fallback: if the CUDA library is missing this raises, and every
call that needs a device fails loudly when none is present."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libb200pde.so")

# every symbol include/b200pde.h declares: (restype, argtypes)
_P = C.c_void_p
_PP = C.POINTER(C.c_void_p)
_D = C.c_double
_DP = C.POINTER(C.c_double)
_I = C.c_int
_IP = C.POINTER(C.c_int)
_SZ = C.c_size_t
SYMBOLS = {
    "b2_last_error": (C.c_char_p, []),
    "b2_version": (_I, []),
    "b2_ctx_create": (_I, [_I, _I, _I, _SZ, _PP]),
    "b2_ctx_destroy": (_I, [_P]),
    "b2_ctx_sync": (_I, [_P]),
    "b2_ctx_timer_start": (_I, [_P]),
    "b2_ctx_timer_stop": (_I, [_P, _DP]),
    "b2_ctx_launch_count": (_I, [_P, C.POINTER(C.c_longlong)]),
    "b2_ctx_profile": (_I, [_P, _I, _DP]),
    "b2_ctx_opprof": (_I, [_P, _I, C.POINTER(C.c_ulonglong)]),
    "b2_debug_copy": (_I, [_P, _I, _I, C.POINTER(C.c_double)]),
    "b2_ctx_heap_handle": (_I, [_P, _P]),
    "b2_ctx_attach_peers": (_I, [_P, _P]),
    "b2_ctx_nranks": (_I, [_P]),
    "b2_ctx_barrier": (_I, [_P]),
    "b2_space2_create": (_I, [_P, _I, _I, _I, _I, _PP]),
    "b2_space_destroy": (_I, [_P]),
    "b2_space_shape": (_I, [_P, _I, _IP, _IP, _IP]),
    "b2_space_coords": (_I, [_P, _I, _DP]),
    "b2_space_lane_layout": (_I, [_P, _I, _IP]),
    "b2_array_create": (_I, [_P, _I, _PP]),
    "b2_array_destroy": (_I, [_P]),
    "b2_array_local_rows": (_I, [_P, _IP, _IP]),
    "b2_array_sumsq_local": (_I, [_P, _DP]),
    "b2_array_set_host": (_I, [_P, _P, _SZ]),
    "b2_array_get_host": (_I, [_P, _P, _SZ]),
    "b2_array_axpy": (_I, [_P, _D, _P]),
    "b2_array_norm2": (_I, [_P, _DP]),
    "b2_field_array": (_I, [_P, _I, _PP]),
    "b2_array_copy": (_I, [_P, _P]),
    "b2_array_combine": (_I, [_P, _P, _P, _I, _D]),
    "b2_array_weighted_sum": (_I, [_P, _DP, _DP, _I, _DP]),
    "b2_field_create": (_I, [_P, _PP]),
    "b2_field_destroy": (_I, [_P]),
    "b2_field_set_v_host": (_I, [_P, _P, _SZ]),
    "b2_field_get_v_host": (_I, [_P, _P, _SZ]),
    "b2_field_set_vhat_host": (_I, [_P, _P, _SZ]),
    "b2_field_get_vhat_host": (_I, [_P, _P, _SZ]),
    "b2_field_local_rows": (_I, [_P, _I, _IP, _IP]),
    "b2_forward": (_I, [_P]),
    "b2_backward": (_I, [_P]),
    "b2_to_ortho": (_I, [_P, _P]),
    "b2_from_ortho": (_I, [_P, _P]),
    "b2_gradient": (_I, [_P, _I, _I, _DP, _P]),
    "b2_field_dealias": (_I, [_P]),
    "b2_hholtz_adi_create": (_I, [_P, _D, _D, _PP]),
    "b2_poisson_create": (_I, [_P, _D, _D, _DP, _DP, _DP, _PP]),
    "b2_hholtz_create": (_I, [_P, _D, _D, _DP, _DP, _DP, _PP]),
    "b2_solver_destroy": (_I, [_P]),
    "b2_solve": (_I, [_P, _P, _P]),
    "b2_poisson_axis0_matrices": (_I, [_P, _D, _DP, _DP]),
    "b2_host_poisson_matrices": (_I, [_I, _I, _D, _DP, _DP]),
    "b2_navier2d_create": (_I, [_P, _I, _I, _D, _D, _D, _D, C.c_char_p, _I, _DP, _DP, _DP, _PP]),
    "b2_navier_destroy": (_I, [_P]),
    "b2_navier_field": (_I, [_P, _I, _PP]),
    "b2_navier_update": (_I, [_P, _I]),
    "b2_navier_div_norm": (_I, [_P, _DP]),
    "b2_navier_get_time": (_I, [_P, _DP]),
    "b2_navier_set_time": (_I, [_P, _D]),
    "b2_navier_set_mode": (_I, [_P, _I]),
    "b2_navier_launch_count": (_I, [_P, C.POINTER(C.c_longlong)]),
    "b2_navier_info": (_I, [_P, C.POINTER(C.c_longlong)]),
    "b2_navier_poisson_matrices": (_I, [_P, _DP, _DP, _IP]),
}

_lib = None


class B2Error(RuntimeError):
    pass


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise B2Error(f"{LIB_PATH} is missing: build it with `python -m rustpde_mpi_b200.build` "
                          "(there is no CPU fallback)")
        _lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(_lib, name)  # raises AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
    return _lib


def check(status):
    if status != 0:
        raise B2Error(f"b200pde error {status}: {lib().b2_last_error().decode()}")
