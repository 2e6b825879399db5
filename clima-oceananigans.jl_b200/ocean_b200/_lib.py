"""ctypes binding of libocean_b200.so (include/ocean_b200.h).  There is no fallback: if the
shared library is missing the import fails, and every entry point fails without a CUDA device."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libocean_b200.so")

F32, F64 = 0, 1
PERIODIC, BOUNDED, FLAT, FULLY_CONNECTED = 0, 1, 2, 3
CENTER, FACE = 0, 1
BC_NONE, BC_PERIODIC, BC_FLUX, BC_VALUE, BC_GRADIENT, BC_OPEN = range(6)
ADV = {"none": 0, "CenteredSecondOrder": 1, "CenteredFourthOrder": 2, "UpwindBiasedFirstOrder": 3,
       "UpwindBiasedThirdOrder": 4, "UpwindBiasedFifthOrder": 5, "WENO5": 6}
CLOSURE = {"none": 0, "ThreeDimensional": 1, "Horizontal": 2, "Vertical": 3, "SmagorinskyLilly": 4, "AnisotropicMinimumDissipation": 5}
TS = {"QuasiAdamsBashforth2": 0, "RungeKutta3": 1}
SOLVER_AUTO, SOLVER_FFT, SOLVER_FT = 0, 1, 2
MAX_TRACERS = 8


class GridDesc(C.Structure):
    _fields_ = [("ftype", C.c_int32), ("N", C.c_int32 * 3), ("H", C.c_int32 * 3),
                ("topology", C.c_int32 * 3), ("L", C.c_double * 3), ("regular", C.c_int32 * 3),
                ("delta", C.c_double * 3),
                ("dC", C.POINTER(C.c_double) * 3), ("dC_first", C.c_int32 * 3), ("dC_len", C.c_int32 * 3),
                ("dF", C.POINTER(C.c_double) * 3), ("dF_first", C.c_int32 * 3), ("dF_len", C.c_int32 * 3)]


class BC(C.Structure):
    _fields_ = [("kind", C.c_int32), ("value", C.c_double)]


class Forcing(C.Structure):
    _fields_ = [("active", C.c_int32), ("mask_dim", C.c_int32), ("rate", C.c_double), ("mask", C.POINTER(C.c_double)),
                ("target_dim", C.c_int32), ("target_value", C.c_double), ("target", C.POINTER(C.c_double))]


class ModelDesc(C.Structure):
    _fields_ = [("grid", C.c_void_p), ("timestepper", C.c_int32), ("chi", C.c_double),
                ("advection", C.c_int32), ("weno_zweno", C.c_int32),
                ("weno_coeff", (C.POINTER(C.c_double) * 2) * 3),
                ("closure", C.c_int32), ("nu", C.c_double), ("kappa", C.c_double * MAX_TRACERS),
                ("coriolis_fplane", C.c_int32), ("f", C.c_double),
                ("buoyancy_tracer", C.c_int32), ("gravity_tilted", C.c_int32), ("g_hat", C.c_double * 3),
                ("ntracers", C.c_int32), ("bcs", (BC * 6) * (3 + MAX_TRACERS)),
                ("pressure_solver", C.c_int32),
                ("buoyancy_kind", C.c_int32), ("temperature_tracer", C.c_int32), ("salinity_tracer", C.c_int32),
                ("gravitational_acceleration", C.c_double), ("thermal_expansion", C.c_double),
                ("haline_contraction", C.c_double),
                ("smagorinsky_C", C.c_double), ("smagorinsky_Cb", C.c_double), ("prandtl", C.c_double * MAX_TRACERS),
                ("amd_Cnu", C.c_double), ("amd_Ckappa", C.c_double * MAX_TRACERS), ("amd_Cb", C.c_double),
                ("amd_has_Cb", C.c_int32), ("closure_vertically_implicit", C.c_int32),
                ("forcing", Forcing * (3 + MAX_TRACERS)),
                ("background", C.c_void_p * (3 + MAX_TRACERS))]


#: every symbol include/ocean_b200.h declares: name -> (restype, argtypes)
SYMBOLS = {
    "ob200_version": (C.c_int32, []),
    "ob200_init": (C.c_int32, [C.c_int32]),
    "ob200_set_stream": (C.c_int32, [C.c_void_p]),
    "ob200_sync": (C.c_int32, []),
    "ob200_last_error": (C.c_size_t, [C.c_char_p, C.c_size_t]),
    "ob200_launch_count": (C.c_int64, []),
    "ob200_malloc": (C.c_int32, [C.POINTER(C.c_void_p), C.c_size_t]),
    "ob200_free": (C.c_int32, [C.c_void_p]),
    "ob200_memset": (C.c_int32, [C.c_void_p, C.c_int32, C.c_size_t]),
    "ob200_upload": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_size_t]),
    "ob200_download": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_size_t]),
    "ob200_grid_create": (C.c_int32, [C.POINTER(GridDesc), C.POINTER(C.c_void_p)]),
    "ob200_grid_destroy": (C.c_int32, [C.c_void_p]),
    "ob200_field_create": (C.c_int32, [C.c_void_p, C.POINTER(C.c_int32), C.POINTER(BC), C.POINTER(C.c_void_p)]),
    "ob200_field_destroy": (C.c_int32, [C.c_void_p]),
    "ob200_field_parent_size": (C.c_int32, [C.c_void_p, C.POINTER(C.c_int32)]),
    "ob200_field_set_parent": (C.c_int32, [C.c_void_p, C.c_void_p]),
    "ob200_field_get_parent": (C.c_int32, [C.c_void_p, C.c_void_p]),
    "ob200_field_set_parent_async": (C.c_int32, [C.c_void_p, C.c_void_p]),
    "ob200_mark_download_batch": (C.c_int32, []),
    "ob200_sync_downloads": (C.c_int32, [C.c_int32]),
    "ob200_field_get_parent_async": (C.c_int32, [C.c_void_p, C.c_void_p]),
    "ob200_field_device_view": (C.c_int32, [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "ob200_fill_halo_regions": (C.c_int32, [C.POINTER(C.c_void_p), C.c_int32]),
    "ob200_field_set_boundary_values": (C.c_int32, [C.c_void_p, C.c_int32, C.c_void_p]),
    "ob200_field_reduce": (C.c_int32, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double),
                                       C.POINTER(C.c_double), C.POINTER(C.c_int32)]),
    "ob200_poisson_create": (C.c_int32, [C.c_void_p, C.c_int32, C.POINTER(C.c_void_p)]),
    "ob200_poisson_destroy": (C.c_int32, [C.c_void_p]),
    "ob200_poisson_solve": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "ob200_solve_for_pressure": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ob200_batched_tridiagonal_solve": (C.c_int32, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                                    C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ob200_model_create": (C.c_int32, [C.POINTER(ModelDesc), C.POINTER(C.c_void_p)]),
    "ob200_model_destroy": (C.c_int32, [C.c_void_p]),
    "ob200_model_field": (C.c_int32, [C.c_void_p, C.c_char_p, C.POINTER(C.c_void_p)]),
    "ob200_model_update_state": (C.c_int32, [C.c_void_p]),
    "ob200_model_calculate_tendencies": (C.c_int32, [C.c_void_p]),
    "ob200_model_pressure_project": (C.c_int32, [C.c_void_p, C.c_double]),
    "ob200_model_time_step": (C.c_int32, [C.c_void_p, C.c_double, C.c_int32]),
    "ob200_model_clock": (C.c_int32, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int64)]),
    "ob200_model_set_clock": (C.c_int32, [C.c_void_p, C.c_double, C.c_int64, C.c_double]),
    "ob200_model_previous_time_step": (C.c_int32, [C.c_void_p, C.POINTER(C.c_double)]),
    "ob200_field_slice_async": (C.c_int32, [C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.c_void_p]),
    "ob200_field_average_async": (C.c_int32, [C.c_void_p, C.POINTER(C.c_int32), C.c_void_p]),
    "ob200_model_diagnostics": (C.c_int32, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "ob200_model_max_abs_velocities": (C.c_int32, [C.c_void_p, C.POINTER(C.c_double)]),
    "ob200_debug_cached_tensor_maps": (C.c_int64, []),
    "ob200_comm_unique_id": (C.c_int32, [C.c_char_p]),
    "ob200_comm_init": (C.c_int32, [C.c_int32, C.c_int32, C.c_char_p]),
    "ob200_comm_destroy": (C.c_int32, []),
    "ob200_comm_allreduce": (C.c_int32, [C.POINTER(C.c_double), C.c_int32, C.c_int32]),
    "ob200_model_use_fast_kernels": (C.c_int32, [C.c_void_p, C.c_int32]),
    "ob200_profile_enable": (C.c_int32, [C.c_int32]),
    "ob200_profile_reset": (C.c_int32, []),
    "ob200_profile_query": (C.c_int32, [C.c_char_p, C.POINTER(C.c_double), C.POINTER(C.c_int64)]),
}
EXTRA_SYMBOLS = {}

if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} is missing: build it with `python __graft_entry__.py` (or `make -C "
        "clima-oceananigans.jl_b200/csrc`).  ocean_b200 has no CPU fallback.")

lib = C.CDLL(LIB_PATH)
for _name, (_res, _args) in {**SYMBOLS, **EXTRA_SYMBOLS}.items():
    _fn = getattr(lib, _name)
    _fn.restype = _res
    _fn.argtypes = _args


class B200Error(RuntimeError):
    pass


def last_error():
    n = lib.ob200_last_error(None, 0)
    buf = C.create_string_buffer(n + 1)
    lib.ob200_last_error(buf, n + 1)
    return buf.value.decode(errors="replace")


def check(status):
    if status != 0:
        raise B200Error(last_error())
