"""ctypes binding of librtb200.so -- the C-ABI declared in include/rtb200.h.

The product path has no CPU fallback: if the CUDA library is missing or no CUDA device is present, loading or
`rtb200_create` fails loudly.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "librtb200.so")
_lib = None

# name -> (restype, argtypes); mirrors include/rtb200.h one to one (tests check that every symbol is exported)
P = C.c_void_p
SIGNATURES = {
    "rtb200_version": (C.c_int, []),
    "rtb200_status_string": (C.c_char_p, [C.c_int]),
    "rtb200_create": (C.c_int, [C.c_int, C.POINTER(P)]),
    "rtb200_destroy": (C.c_int, [P]),
    "rtb200_comm_unique_id": (C.c_int, [P]),
    "rtb200_create_multi": (C.c_int, [C.c_int, P, C.POINTER(P)]),
    "rtb200_create_rank": (C.c_int, [C.c_int, C.c_int, C.c_int, P, C.POINTER(P)]),
    "rtb200_multi_info": (C.c_int, [P, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                                    C.POINTER(C.c_int64), C.POINTER(C.c_int32)]),
    "rtb200_shard_directions": (C.c_int, [C.c_int, C.c_int, C.c_int, P, C.c_int, P, C.c_int32, C.POINTER(C.c_int32)]),
    "rtb200_multi_shard": (C.c_int, [P, C.c_int, C.c_int, P, C.c_int32, C.POINTER(C.c_int32)]),
    "rtb200_multi_diffuse_resident": (C.c_int, [P, C.c_int, P, P, P, C.c_int, P, C.POINTER(C.c_int64)]),
    "rtb200_multi_point_resident": (C.c_int, [P, C.c_int, P, P, P, C.c_double, P, C.c_int, C.c_int, C.c_int32, P, P, P, P,
                                              P, P, P, P, C.POINTER(C.c_int64)]),
    "rtb200_multi_slab": (C.c_int, [P, C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(P), C.POINTER(P),
                                    C.POINTER(P)]),
    "rtb200_multi_sync": (C.c_int, [P]),
    "rtb200_multi_slab_get": (C.c_int, [P, C.c_int, P, P, P]),
    "rtb200_set_math": (C.c_int, [P, C.c_int]),
    "rtb200_set_tuning": (C.c_int, [P, C.c_char_p, C.c_double]),
    "rtb200_device_error": (C.c_int, [P]),
    "rtb200_grid_set": (C.c_int, [P, C.c_int, C.c_int64, P, P, P, P, P, P, C.c_double]),
    "rtb200_grid_update_species": (C.c_int, [P, P, P, P]),
    "rtb200_grid_set_emission": (C.c_int, [P, P]),
    "rtb200_grid_set_emission_device": (C.c_int, [P, P, P]),
    "rtb200_grid_set_scattering": (C.c_int, [P, P, C.c_int32, C.c_double]),
    "rtb200_last_scattering": (C.c_int, [P, C.POINTER(C.c_int32), C.POINTER(C.c_double)]),
    "rtb200_grid_set_scattering_acceleration": (C.c_int, [P, C.c_int32]),
    "rtb200_last_scattering_acceleration": (C.c_int, [P, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "rtb200_grid_set_dust": (C.c_int, [P, C.c_int, P, P, C.c_int32, C.c_double]),
    "rtb200_diffuse": (C.c_int, [P, C.c_int, P, P, P, C.c_int32, P, P, P, C.POINTER(C.c_int64)]),
    "rtb200_diffuse_device": (C.c_int, [P, C.c_int, P, P, P, C.c_int32, P, P, C.POINTER(C.c_int64)]),
    "rtb200_diffuse_rates_device": (C.c_int, [P, P, P, P, P, P, P, P, P]),
    "rtb200_uvb_amplitudes": (C.c_int, [C.c_double, C.c_double, P, P]),
    "rtb200_uvb_beta_table": (C.c_int, [C.c_int, C.c_double, P, P]),
    "rtb200_uvb_dust_beta": (C.c_int, [C.c_int, C.c_double, P, P, P]),
    "rtb200_uvb_background": (C.c_int, [C.c_double, C.c_double, C.c_int, C.c_double, P, P, P, P, P, P, P]),
    "rtb200_point": (C.c_int, [P, C.c_int, P, P, P, C.c_double, P, C.c_int, C.c_int, C.c_int32, P, P, P, P, P, P, P, P,
                              P, P, P, P, P, C.POINTER(C.c_int64)]),
    "rtb200_point_device": (C.c_int, [P, C.c_int, P, P, P, C.c_double, P, C.c_int, C.c_int, C.c_int32, P, P, P, P, P,
                                     P, P, P, P, C.POINTER(C.c_int64)]),
    "rtb200_point_trace": (C.c_int, [P, C.c_int, P, P, P, C.c_double, P, C.c_int, C.c_int, C.c_int32, P, P, P,
                                    C.POINTER(C.c_int64), P, C.c_int64, C.POINTER(C.c_int64)]),
    "rtb200_point_tables": (C.c_int, [P, C.c_int, P, P, P, C.c_double, P, C.c_int, C.c_double, P]),
    "rtb200_chemistry_tables": (C.c_int, [P, C.c_int, C.c_double, C.c_double, C.c_double, P, P, P, P, P, P]),
    "rtb200_chemistry_temperature": (C.c_int, [P, P]),
    "rtb200_compute_mass": (C.c_int, [P, C.POINTER(C.c_double), C.POINTER(C.c_double), P]),
    "rtb200_chemistry_device": (C.c_int, [P, P, P, P, P, C.POINTER(C.c_double), P]),
    "rtb200_grid_get_species": (C.c_int, [P, P, P, P]),
    "rtb200_octree_build": (C.c_int, [C.c_int, C.c_int, P, P, P, P, P, P, C.POINTER(C.c_int64), C.POINTER(C.c_int32),
                                      C.POINTER(C.c_double), C.POINTER(P)]),
    "rtb200_octree_get": (C.c_int, [P, P, P, P, P, P, P, P]),
    "rtb200_octree_free": (C.c_int, [P]),
    "rtb200_direction": (C.c_int, [C.c_int, C.c_int64, C.POINTER(C.c_int32), C.POINTER(C.c_double),
                                   C.POINTER(C.c_double)]),
    "rtb200_patterns": (C.c_int, [C.c_int, C.c_int64, C.c_int, P]),
    "rtb200_neighbours": (C.c_int, [P, C.c_int, C.c_int64, P]),
    "rtb200_debug_waves": (C.c_int, [P, C.c_int, C.c_int64, P, P]),
    "rtb200_debug_portable_math": (C.c_int, [P, C.c_int64, P, P, P]),
    "rtb200_debug_fast_exp": (C.c_int, [P, C.c_int64, P, P, P]),
    "rtb200_last_stats": (C.c_int, [P, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_int64),
                                    C.POINTER(C.c_int64), C.POINTER(C.c_double)]),
}


class RTB200Error(RuntimeError):
    def __init__(self, status, where=""):
        self.status = int(status)
        msg = lib().rtb200_status_string(self.status).decode()
        super().__init__(f"{where}: rtb200 status {self.status}: {msg}")


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} not found: build it with `python -m radiativetransfer_b200.build` "
                "(nvcc, sm_100a). There is no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)  # AttributeError if the library lacks a declared entry point
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(status, where):
    if status != 0:
        raise RTB200Error(status, where)
