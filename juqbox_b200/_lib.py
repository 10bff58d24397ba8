"""ctypes binding of the C ABI in include/juqbox_b200.h.

The CUDA library is the only implementation of the hot path: if it cannot be built or loaded this module
raises — there is deliberately no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build


class jq_operator(C.Structure):
    _fields_ = [("format", C.c_int32), ("nnz", C.c_int64), ("colptr", C.c_void_p), ("rowval", C.c_void_p),
                ("nzval", C.c_void_p)]


class jq_problem(C.Structure):
    _fields_ = [("n", C.c_int32), ("m", C.c_int32), ("ncoupled", C.c_int32), ("nfreq", C.c_int32),
                ("neumann_terms", C.c_int32), ("obj_func_type", C.c_int32), ("pfid_type", C.c_int32),
                ("linear_solver", C.c_int32), ("nsteps", C.c_int64), ("T", C.c_double),
                ("uinit", C.c_void_p), ("vtarget_r", C.c_void_p), ("vtarget_i", C.c_void_p), ("wdiag", C.c_void_p),
                ("cfreq", C.c_void_p), ("h0", jq_operator), ("hsym", C.POINTER(jq_operator)),
                ("hanti", C.POINTER(jq_operator)), ("solver_tol", C.c_double),
                ("global_phase", C.c_double), ("wmat_real", C.c_void_p), ("wmat_imag", C.c_void_p),
                ("nuncoupled", C.c_int32), ("reserved0", C.c_int32), ("hunc", C.POINTER(jq_operator)),
                ("unc_is_symm", C.c_void_p), ("unc_rfreq", C.c_void_p)]


JQ_DENSE, JQ_CSC = 0, 1
JQ_ERR_PCOF_LENGTH = -2

EXPORTS = ["jq_create", "jq_destroy", "jq_update_target", "jq_traceobjgrad_batch", "jq_traceobjgrad_batch_device", "jq_eval_f_grad",
           "jq_cache_invalidate", "jq_eval_forward", "jq_eval_controls", "jq_forward_sensitivity",
           "jq_set_kernel", "jq_set_time_segments", "jq_time_segments", "jq_query", "jq_fp64_peak", "jq_fp64_peak_3op", "jq_fp64_peak_dmma", "jq_comm_unique_id", "jq_comm_init", "jq_comm_destroy", "jq_comm_set_cooperative",
           "jq_abi_info", "jq_last_error", "jq_version"]
ABI_VERSION = 2

_lib = None


class JuqboxCudaError(RuntimeError):
    pass


def library_path() -> str:
    return _build.LIB


def load(build_if_missing: bool = True):
    """Load (building first if the .so is stale and nvcc is present) libjuqbox_b200.so."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB
    if build_if_missing and _build.needs_build():
        try:
            _build.build_library()
        except Exception as e:
            # never load a stale binary silently: its structs may no longer match the ctypes definitions above
            raise JuqboxCudaError(f"libjuqbox_b200.so is {'stale' if os.path.exists(path) else 'missing'} and could not be rebuilt: {e}") from e
    if not os.path.exists(path):
        raise JuqboxCudaError(f"{path} not found: run `python -m juqbox_b200.build` (there is no CPU fallback)")
    lib = C.CDLL(path)
    vp, i32, dp = C.c_void_p, C.c_int32, C.c_void_p
    lib.jq_create.argtypes = [C.POINTER(jq_problem), C.c_int, C.POINTER(vp)]
    lib.jq_destroy.argtypes = [vp]
    lib.jq_update_target.argtypes = [vp, dp, dp]
    lib.jq_traceobjgrad_batch.argtypes = [vp, i32, dp, i32, i32, dp, dp, i32, dp, dp, dp, dp, dp, dp]
    lib.jq_traceobjgrad_batch_device.argtypes = [vp, i32, dp, i32, i32, dp, dp, i32, dp, dp, dp, dp, dp, dp, vp]
    lib.jq_eval_forward.argtypes = [vp, i32, dp, i32, i32, dp, i32, dp, dp, dp, dp]
    lib.jq_eval_controls.argtypes = [vp, dp, i32, i32, dp, dp, dp]
    lib.jq_forward_sensitivity.argtypes = [vp, i32, dp, i32, i32, dp, dp, i32, dp, dp, dp, dp, dp, dp, dp]
    lib.jq_set_kernel.argtypes = [vp, i32]
    lib.jq_set_time_segments.argtypes = [vp, i32]
    lib.jq_comm_set_cooperative.argtypes = [vp, i32]
    lib.jq_time_segments.argtypes = [C.c_double, C.c_int64, i32, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    lib.jq_time_segments.restype = C.c_int64
    lib.jq_query.argtypes = [vp, i32, C.POINTER(C.c_double)]
    lib.jq_fp64_peak.argtypes = [C.c_int, C.POINTER(C.c_double)]
    lib.jq_fp64_peak_3op.argtypes = [C.c_int, C.POINTER(C.c_double)]
    lib.jq_fp64_peak_dmma.argtypes = [C.c_int, C.POINTER(C.c_double)]
    lib.jq_comm_unique_id.argtypes = [vp]
    lib.jq_comm_init.argtypes = [vp, i32, i32, vp]
    lib.jq_comm_destroy.argtypes = [vp]
    lib.jq_eval_f_grad.argtypes = [vp, dp, i32, i32, dp, dp, C.c_double, dp, dp, dp, dp, dp, dp, C.POINTER(C.c_int32)]
    lib.jq_cache_invalidate.argtypes = [vp]
    lib.jq_abi_info.argtypes = [i32]
    lib.jq_abi_info.restype = C.c_int64
    for name in EXPORTS[:-3]:
        getattr(lib, name).restype = C.c_int
    # the hand-written struct mirrors above must match the binary (guards against a stale or foreign .so)
    got = (lib.jq_abi_info(0), lib.jq_abi_info(1), lib.jq_abi_info(2))
    want = (ABI_VERSION, C.sizeof(jq_problem), C.sizeof(jq_operator))
    if got != want:
        raise JuqboxCudaError(f"{path}: ABI mismatch (version, sizeof(jq_problem), sizeof(jq_operator)) = {got}, this package expects {want}")
    lib.jq_last_error.restype = C.c_char_p
    lib.jq_version.restype = C.c_char_p
    _lib = lib
    return lib


def last_error() -> str:
    return load().jq_last_error().decode()


def check(rc: int):
    if rc == 0:
        return
    msg = last_error()
    if rc == JQ_ERR_PCOF_LENGTH:
        raise ValueError(msg)          # the reference raises error()/DimensionMismatch here
    raise JuqboxCudaError(f"juqbox_b200 error {rc}: {msg}")


def fp64_peak_tflops(device: int = 0, three_operand: bool = False, tensor: bool = False) -> float:
    v = C.c_double()
    fn = load().jq_fp64_peak_dmma if tensor else load().jq_fp64_peak_3op if three_operand else load().jq_fp64_peak
    check(fn(device, C.byref(v)))
    return v.value
