"""ctypes binding of ``include/mafed_distill.h`` (the C ABI under the ``mafed.methods`` mirror).

There is no CPU fallback: if the shared library is missing or a call fails, this raises.
"""
from __future__ import annotations

import contextlib
import ctypes
import os
import threading

MAX_LAYERS = 64
F32, BF16, F16 = 0, 1, 2
LOSS_MSE, LOSS_COSINE = 0, 1
MODW_EQUAL, MODW_TABLE, MODW_CLS, MODW_TEXT_ONLY = 0, 1, 2, 3
VARIANT_DEFAULT, VARIANT_LDG, VARIANT_TMA = 0, 1, 2
STAGE_REDUCE, STAGE_COUNTS, STAGE_LOSSES, STAGE_SCALE = 1, 2, 4, 8
COMM_SUMS, COMM_COUNTS = 1, 2
ABI_VERSION = 4
# indices of mafed_tuning_t::v the library reads (MAFED_TUNE_* of the header; it ignores every other index)
TUNE_NO_TAIL = 17       # 1: separate epilogue launch instead of the in-kernel tail
TUNE_VARIANT_ALL = 18   # kernel family of every pass: 1 ldg, 2 tma (0 = default)
TUNE_NO_GATE = 19       # 1: backward fix-up as a full grid that returns at once (round-1 form)
TUNE_KEYS = {"TUNE_NO_TAIL": TUNE_NO_TAIL, "TUNE_VARIANT_ALL": TUNE_VARIANT_ALL, "TUNE_NO_GATE": TUNE_NO_GATE}
N_TUNE_KEYS = 24

# MAFED_B200_LIB: another build of the same C ABI (A/B measurements of two kernel versions, tools/ab_lib.py)
LIB_PATH = os.environ.get("MAFED_B200_LIB") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "_lib",
                                                            "libmafed_distill.so")

EXPORTS = (
    "mafed_distill_abi_version", "mafed_distill_error_string", "mafed_distill_ws_bytes",
    "mafed_distill_sums_len", "mafed_distill_out_len",
    "mafed_distill_step", "mafed_distill_fwd_step", "mafed_distill_bwd", "mafed_distill_prefetch_counts",
    "mafed_distill_fwd", "mafed_distill_fused", "mafed_distill_scalar_stage",
    "mafed_distill_modality_masks", "mafed_distill_token_norm_sums",
    "mafed_comm_handle_bytes", "mafed_comm_create", "mafed_comm_connect", "mafed_comm_status", "mafed_comm_trace",
    "mafed_comm_trace_async",
    "mafed_comm_set_timeout", "mafed_comm_destroy",
    "mafed_host_step_device_bytes", "mafed_host_step_create", "mafed_host_step_run", "mafed_host_step_destroy",
    "mafed_host_register", "mafed_host_unregister",
)


class Tuning(ctypes.Structure):
    """mafed_tuning_t"""
    _fields_ = [("v", ctypes.c_int32 * N_TUNE_KEYS)]


class Shape(ctypes.Structure):
    """mafed_shape_t"""
    _fields_ = [(n, ctypes.c_int32) for n in ("n_layers", "B", "T", "n_vis", "D", "dtype", "loss_kind", "cls")] + \
               [("tuning", ctypes.POINTER(Tuning))]


# Overrides travel with each call (mafed_shape_t::tuning); the library itself keeps no mutable state.
# Benchmarks and tests install a Tuning for the calls made inside a `with cabi.tuning(...)` block of THIS process.
_active_tuning = None


def active_tuning_address() -> int:
    """Address of the Tuning installed by `tuning(...)`, 0 if none (what the torch extension is handed)."""
    return ctypes.addressof(_active_tuning) if _active_tuning is not None else 0


@contextlib.contextmanager
def tuning(variant: int = 0, **keys):
    """``with cabi.tuning(variant=cabi.VARIANT_LDG, TUNE_NO_TAIL=1): ...`` -- overrides for the calls inside the block.
    Keys are the names of TUNE_KEYS; any other keyword raises TypeError."""
    global _active_tuning
    unknown = sorted(set(keys) - set(TUNE_KEYS))
    if unknown:
        raise TypeError(f"unknown tuning key(s) {unknown}; the library reads {sorted(TUNE_KEYS)}")
    t = Tuning()
    if _active_tuning is not None:
        ctypes.memmove(ctypes.addressof(t), ctypes.addressof(_active_tuning), ctypes.sizeof(Tuning))
    if variant:
        t.v[TUNE_VARIANT_ALL] = int(variant)
    for name, value in keys.items():
        t.v[TUNE_KEYS[name]] = int(value)
    prev, _active_tuning = _active_tuning, t
    try:
        yield t
    finally:
        _active_tuning = prev


class Weights(ctypes.Structure):
    """mafed_weights_t"""
    _fields_ = [
        ("modality_kind", ctypes.c_int32),
        ("distill_coeff", ctypes.c_float),
        ("layer_coeff", ctypes.c_float * MAX_LAYERS),
        ("lang_weight", ctypes.c_float * MAX_LAYERS),
    ]


class MafedDistillError(RuntimeError):
    pass


_lib = None
_lock = threading.Lock()


def load():
    """Load libmafed_distill.so (built in-tree by ``mafed_b200.build``); raise if it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise MafedDistillError(
                f"{LIB_PATH} not found: build it with `python -m mafed_b200.build` "
                "(the distillation path has no CPU / eager fallback)")
        lib = ctypes.CDLL(LIB_PATH)
        vp, i32 = ctypes.c_void_p, ctypes.c_int
        pp = ctypes.POINTER(ctypes.c_void_p)
        sh, wt = ctypes.POINTER(Shape), ctypes.POINTER(Weights)
        lib.mafed_distill_abi_version.restype = i32
        lib.mafed_distill_error_string.restype = ctypes.c_char_p
        lib.mafed_distill_error_string.argtypes = [i32]
        lib.mafed_distill_ws_bytes.restype = ctypes.c_size_t
        lib.mafed_distill_ws_bytes.argtypes = [i32]
        lib.mafed_distill_sums_len.restype = i32
        lib.mafed_distill_sums_len.argtypes = [i32]
        lib.mafed_distill_out_len.restype = i32
        lib.mafed_distill_out_len.argtypes = [i32]
        fp = ctypes.POINTER(ctypes.c_float)
        lib.mafed_distill_fwd.restype = i32
        lib.mafed_distill_fwd.argtypes = [sh, pp, pp, vp, vp, vp]
        lib.mafed_distill_scalar_stage.restype = i32
        lib.mafed_distill_scalar_stage.argtypes = [sh, wt, i32, vp, vp, vp, vp, vp, vp, i32, vp]
        lib.mafed_distill_bwd.restype = i32
        lib.mafed_distill_bwd.argtypes = [sh, pp, pp, pp, vp, vp, vp, ctypes.c_float, fp, vp, vp]
        lib.mafed_distill_fused.restype = i32
        lib.mafed_distill_fused.argtypes = [sh, pp, pp, pp, vp, wt, vp, ctypes.c_float, vp, vp, vp]
        lib.mafed_distill_step.restype = i32
        lib.mafed_distill_step.argtypes = [sh, pp, pp, pp, vp, wt, ctypes.c_float, vp, vp, vp, vp, vp, vp, vp, vp, vp]
        lib.mafed_distill_fwd_step.restype = i32
        lib.mafed_distill_fwd_step.argtypes = [sh, pp, pp, vp, wt, vp, vp, vp, vp, vp, vp]
        lib.mafed_distill_prefetch_counts.restype = i32
        lib.mafed_distill_prefetch_counts.argtypes = [sh, vp, vp, vp, vp]
        lib.mafed_comm_handle_bytes.restype = i32
        lib.mafed_comm_create.restype = i32
        lib.mafed_comm_create.argtypes = [i32, i32, ctypes.c_char_p, ctypes.POINTER(vp)]
        lib.mafed_comm_connect.restype = i32
        lib.mafed_comm_connect.argtypes = [vp, ctypes.c_char_p]
        lib.mafed_comm_status.restype = i32
        lib.mafed_comm_status.argtypes = [vp, ctypes.POINTER(i32)]
        lib.mafed_comm_trace.restype = i32
        lib.mafed_comm_trace.argtypes = [vp, ctypes.POINTER(ctypes.c_ulonglong)]
        lib.mafed_comm_trace_async.restype = i32
        lib.mafed_comm_trace_async.argtypes = [vp, vp, vp]
        lib.mafed_comm_set_timeout.restype = i32
        lib.mafed_comm_set_timeout.argtypes = [vp, ctypes.c_double]
        lib.mafed_comm_destroy.restype = i32
        lib.mafed_comm_destroy.argtypes = [vp]
        lib.mafed_host_step_device_bytes.restype = ctypes.c_size_t
        lib.mafed_host_step_device_bytes.argtypes = [sh]
        lib.mafed_host_step_create.restype = i32
        lib.mafed_host_step_create.argtypes = [sh, ctypes.POINTER(vp)]
        lib.mafed_host_step_run.restype = i32
        lib.mafed_host_step_run.argtypes = [vp, wt, pp, pp, pp, vp, ctypes.c_float, vp, vp]
        lib.mafed_host_step_destroy.restype = i32
        lib.mafed_host_step_destroy.argtypes = [vp]
        lib.mafed_host_register.restype = i32
        lib.mafed_host_register.argtypes = [vp, ctypes.c_size_t]
        lib.mafed_host_unregister.restype = i32
        lib.mafed_host_unregister.argtypes = [vp]
        lib.mafed_distill_token_norm_sums.restype = i32
        lib.mafed_distill_token_norm_sums.argtypes = [sh, pp, vp, vp, vp]
        lib.mafed_distill_modality_masks.restype = i32
        lib.mafed_distill_modality_masks.argtypes = [sh, vp, vp, vp, vp]
        for name in EXPORTS:
            getattr(lib, name)
        if lib.mafed_distill_abi_version() != ABI_VERSION:
            raise MafedDistillError("libmafed_distill.so ABI version mismatch; rebuild")
        _lib = lib
    return _lib


def check(rc: int, what: str):
    if rc != 0:
        msg = load().mafed_distill_error_string(rc).decode()
        raise MafedDistillError(f"{what} failed: {msg} (code {rc})")


def ptr_array(ptrs):
    """Host array of device pointers (``const void* const*``)."""
    return (ctypes.c_void_p * len(ptrs))(*ptrs)


def make_shape(n_layers, B, T, n_vis, D, dtype, loss_kind, cls=False):
    """mafed_shape_t of one call; carries the Tuning installed by `tuning(...)`, if any (kept alive by the shape)."""
    sh = Shape(n_layers, B, T, n_vis, D, dtype, loss_kind, 1 if cls else 0, None)
    if _active_tuning is not None:
        sh.tuning = ctypes.pointer(_active_tuning)
    return sh


# ---- the stage combinations the path uses (one flag set each of mafed_distill_scalar_stage)
def reduce_stage(lib, shape_ref, mask_ptr, ws_ptr, sums_ptr, stream):
    """REDUCE|COUNTS: the rank-local sums vector before an allreduce."""
    return lib.mafed_distill_scalar_stage(shape_ref, None, STAGE_REDUCE | STAGE_COUNTS, mask_ptr, ws_ptr, sums_ptr,
                                          None, None, None, 0, stream)


def finalize_stage(lib, shape_ref, weights_ref, sums_ptr, out_ptr, bwd_scale_ptr, stream):
    """LOSSES (|SCALE) from (global) sums."""
    flags = STAGE_LOSSES | (STAGE_SCALE if bwd_scale_ptr else 0)
    return lib.mafed_distill_scalar_stage(shape_ref, weights_ref, flags, None, None, sums_ptr, out_ptr,
                                          bwd_scale_ptr, None, 0, stream)


def make_weights(modality_kind, distill_coeff, layer_coeffs, lang_weights=None):
    w = Weights()
    w.modality_kind = modality_kind
    w.distill_coeff = float(distill_coeff)
    for i, c in enumerate(layer_coeffs):
        w.layer_coeff[i] = float(c)
    if lang_weights is not None:
        for i, c in enumerate(lang_weights):
            w.lang_weight[i] = float(c)
    return w
