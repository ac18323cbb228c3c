"""ctypes binding of include/sri.h.  Fails loudly when the CUDA library is missing: there is no CPU fallback."""
from __future__ import annotations

import ctypes
from ctypes import POINTER, c_char_p, c_double, c_int, c_int64, c_uint64, c_void_p
from pathlib import Path

import os

# SRI_LIB_PATH lets kernel experiments (tools/) load an alternative build of the same C ABI
LIB_PATH = Path(os.environ.get("SRI_LIB_PATH", Path(__file__).resolve().parent / "libsri_cuda.so"))

SRI_OK = 0
STATUS_NAMES = {
    0: "SRI_OK",
    -1: "SRI_ERR_INVALID_ARGUMENT",
    -2: "SRI_ERR_UNSUPPORTED_N",
    -3: "SRI_ERR_CUDA",
    -4: "SRI_ERR_ALLOC",
    -5: "SRI_ERR_SINGULAR",
}


class SriError(RuntimeError):
    def __init__(self, code: int, where: str, detail: str):
        self.code = code
        super().__init__(f"{where}: {STATUS_NAMES.get(code, code)}: {detail}")


class RodBatch(ctypes.Structure):
    """struct sri_rod_batch (include/sri.h)."""

    _fields_ = [
        ("batch", c_int64),
        ("K", c_void_p), ("q0", c_void_p), ("r0", c_void_p), ("Gamma", c_void_p),
        ("fbar", c_void_p), ("lbar", c_void_p), ("F_tip", c_void_p), ("M_tip", c_void_p),
        ("Q", c_void_p), ("r", c_void_p), ("n", c_void_p), ("m", c_void_p),
        ("info", c_void_p),
    ]


class RodBatchGrad(ctypes.Structure):
    """struct sri_rod_batch_grad (include/sri.h)."""

    _fields_ = [
        ("gQ", c_void_p), ("gr", c_void_p), ("gn", c_void_p), ("gm", c_void_p),
        ("gK", c_void_p), ("gq0", c_void_p), ("gr0", c_void_p), ("gGamma", c_void_p),
        ("gfbar", c_void_p), ("glbar", c_void_p), ("gF_tip", c_void_p), ("gM_tip", c_void_p),
    ]


class NewtonReport(ctypes.Structure):
    """struct sri_newton_report (include/sri.h)."""

    _fields_ = [
        ("iterations", c_int), ("converged", c_int), ("integrations", c_int64),
        ("rms", c_double), ("max_abs", c_double), ("rms_history", c_double * 64), ("history_len", c_int),
        ("singular_solves", c_int64),
    ]


class StaticProblem(ctypes.Structure):
    """struct sri_static_problem (include/sri.h)."""

    _fields_ = [
        ("batch", c_int64), ("ne", c_int),
        ("H_diag", c_void_p), ("F_tip", c_void_p), ("M_tip", c_void_p), ("K0", c_void_p),
        ("q0", c_void_p), ("Gamma", c_void_p), ("fbar", c_void_p), ("lbar", c_void_p),
    ]


class StaticProblemGrad(ctypes.Structure):
    """struct sri_static_problem_grad (include/sri.h)."""

    _fields_ = [
        ("gF_tip", c_void_p), ("gM_tip", c_void_p), ("gK0", c_void_p), ("gH", c_void_p),
        ("gq0", c_void_p), ("gGamma", c_void_p), ("gfbar", c_void_p), ("glbar", c_void_p),
        ("lambda_", c_void_p), ("resid", c_void_p), ("info", c_void_p),
    ]


ALLREDUCE_FN = ctypes.CFUNCTYPE(c_int, POINTER(c_double), c_void_p)  # sri_allreduce_fn

# every symbol include/sri.h declares: name -> (restype, argtypes)
SYMBOLS = {
    "sri_chebyshev_points": (c_int, [c_int, c_double, c_void_p]),
    "sri_chebyshev_coefficients": (c_int, [c_int, c_void_p]),
    "sri_chebyshev_dn": (c_int, [c_int, c_void_p]),
    "sri_phi": (c_int, [c_int, c_int, c_double, c_double, c_double, c_void_p]),
    "sri_create": (c_int, [c_int, c_int, POINTER(c_void_p)]),
    "sri_destroy": (c_int, [c_void_p]),
    "sri_set_stream": (c_int, [c_void_p, c_void_p]),
    "sri_reset_stream": (c_int, [c_void_p]),
    "sri_synchronize": (c_int, [c_void_p]),
    "sri_get_N": (c_int, [c_void_p, POINTER(c_int)]),
    "sri_get_operator": (c_int, [c_void_p, c_int, c_void_p]),
    "sri_strain_from_modes": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_void_p]),
    "sri_strain_from_modes_transpose": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_void_p]),
    "sri_assemble_A": (c_int, [c_void_p, c_int64, c_void_p, c_void_p]),
    "sri_scale_for_length": (c_int, [c_void_p, c_int64, c_void_p, c_double, c_void_p, c_void_p, c_void_p, c_void_p]),
    "sri_device_count": (c_int, [POINTER(c_int)]),
    "sri_create_multi": (c_int, [c_int, POINTER(c_int), c_int, POINTER(c_void_p)]),
    "sri_destroy_multi": (c_int, [c_void_p]),
    "sri_multi_device_count": (c_int, [c_void_p, POINTER(c_int)]),
    "sri_multi_get_handle": (c_int, [c_void_p, c_int, POINTER(c_void_p)]),
    "sri_shard_range": (c_int, [c_int64, c_int, c_int, POINTER(c_int64), POINTER(c_int64)]),
    "sri_integrate_all_sharded": (c_int, [c_void_p, POINTER(RodBatch)]),
    "sri_integrate_all_per_device": (c_int, [c_void_p, POINTER(RodBatch)]),
    "sri_newton_static_shape_sharded": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_double,
                                                c_int, c_double, POINTER(NewtonReport)]),
    "sri_newton_static_problem_sharded": (c_int, [c_void_p, POINTER(StaticProblem), c_void_p, c_double, c_int, c_double,
                                                  POINTER(NewtonReport)]),
    "sri_nccl_unique_id": (c_int, [c_void_p]),
    "sri_nccl_init": (c_int, [c_void_p, c_int, c_int, c_void_p]),
    "sri_nccl_finalize": (c_int, [c_void_p]),
    "sri_nccl_allreduce_norms": (c_int, [c_void_p, c_void_p]),
    "sri_integrate_quaternions": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p]),
    "sri_integrate_position": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p]),
    "sri_integrate_stress": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p]),
    "sri_integrate_couple": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "sri_integrate_all": (c_int, [c_void_p, POINTER(RodBatch)]),
    "sri_integrate_all_vjp": (c_int, [c_void_p, POINTER(RodBatch), POINTER(RodBatchGrad)]),
    "sri_shape_residual": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "sri_wrench_local": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "sri_integrate_wrench_local": (c_int, [c_void_p, c_int64] + [c_void_p] * 10),
    "sri_project_onto_modes": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_void_p]),
    "sri_galerkin_residual": (c_int, [c_void_p, c_int64, c_int] + [c_void_p] * 9),
    "sri_galerkin_residual_vjp": (c_int, [c_void_p, c_int64, c_int] + [c_void_p] * 15),
    "sri_static_shape_vjp": (c_int, [c_void_p, c_int64, c_int] + [c_void_p] * 6 + [c_int] + [c_void_p] * 7),
    "sri_static_problem_vjp": (c_int, [c_void_p, POINTER(StaticProblem), c_void_p, c_void_p, c_int, POINTER(StaticProblemGrad)]),
    "sri_generalised_forces": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_void_p]),
    "sri_shape_jacobian": (c_int, [c_void_p, c_int64, c_int] + [c_void_p] * 8),
    "sri_solve_small_batched": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "sri_newton_static_shape": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_double,
                                        c_int, c_double, c_int64, ALLREDUCE_FN, c_void_p, POINTER(NewtonReport)]),
    "sri_newton_static_problem": (c_int, [c_void_p, POINTER(StaticProblem), c_void_p, c_double, c_int, c_double, c_int64,
                                          ALLREDUCE_FN, c_void_p, POINTER(NewtonReport)]),
    "sri_generate_rods": (c_int, [c_void_p, c_uint64, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_void_p]),
    "sri_last_error_string": (c_char_p, []),
    "sri_set_timing": (c_int, [c_void_p, c_int]),
    "sri_get_last_timing": (c_int, [c_void_p, POINTER(ctypes.c_float), POINTER(c_char_p)]),
    "sri_kernel_launch_count": (c_int64, []),
    "sri_get_handback_count": (c_int, [c_void_p, POINTER(c_int64)]),
    "sri_measure_fp64_peak": (c_int, [c_void_p, POINTER(c_double)]),
    "sri_measure_dmma_peak": (c_int, [c_void_p, POINTER(c_double)]),
}

_lib = None


def load() -> ctypes.CDLL:
    """Load libsri_cuda.so and bind every declared symbol; raises if the library has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(there is no CPU fallback for the integration path)"
        )
    lib = ctypes.CDLL(str(LIB_PATH))
    for name, (restype, argtypes) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError if the .so does not export a declared symbol
        fn.restype = restype
        fn.argtypes = argtypes
    _lib = lib
    return lib


def check(code: int, where: str) -> None:
    if code != SRI_OK:
        detail = load().sri_last_error_string()
        raise SriError(code, where, detail.decode() if detail else "")
