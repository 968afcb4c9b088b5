"""ctypes binding of libmbd_b200.so (the C ABI in include/mbd_b200.h).

The product path has NO CPU fallback: if the library is missing and cannot be built, or no
CUDA device is present when a device entry point is called, this module raises.
"""
from __future__ import annotations

import ctypes
import os

import numpy as np

from . import build as _build

_LIB = None
c_f32p = ctypes.POINTER(ctypes.c_float)
c_u32p = ctypes.POINTER(ctypes.c_uint32)
c_i32p = ctypes.POINTER(ctypes.c_int32)
c_vp = ctypes.c_void_p


class MbdError(RuntimeError):
    pass


class StepParams(ctypes.Structure):
    """mbd_step_params (include/mbd_b200.h): one row per diffusion step index, 32 bytes"""
    _fields_ = [("key", ctypes.c_uint32 * 2), ("sigma", ctypes.c_float), ("coef", ctypes.c_float * 5)]


class StepPlan(ctypes.Structure):
    """mbd_step_plan (include/mbd_b200.h), field for field"""
    _fields_ = [
        ("model", c_vp), ("car_params_dev", c_vp), ("state_init_dev", c_vp), ("params_dev", c_vp), ("ctl_dev", c_vp),
        ("Ybars_dev", c_vp), ("rew_hist_dev", c_vp),
        ("n_total", ctypes.c_int32), ("n_begin", ctypes.c_int32), ("n_local", ctypes.c_int32), ("H", ctypes.c_int32), ("nu", ctypes.c_int32),
        ("temp", ctypes.c_float), ("rew_xref", ctypes.c_float),
        ("xref_dev", c_vp), ("href", ctypes.c_int32), ("env_kind", ctypes.c_int32),
        ("Y0s_dev", c_vp), ("rews_dev", c_vp), ("logpd_dev", c_vp), ("rews_all_dev", c_vp), ("logpd_all_dev", c_vp), ("logp_dev", c_vp),
        ("weights_dev", c_vp), ("runs_dev", c_vp), ("partial_dev", c_vp), ("scalars_dev", c_vp),
        ("P", ctypes.c_int32), ("rank", ctypes.c_int32),
        ("peer_base_ptrs", ctypes.POINTER(ctypes.c_uint64)),
        ("off_rews_words", ctypes.c_uint64), ("off_logpd_words", ctypes.c_uint64), ("off_partial_words", ctypes.c_uint64),
        ("off_flags_words", ctypes.c_uint64), ("timeout_cycles", ctypes.c_uint64),
        # batched solves (appended): n_solves 0/1 = one solve; n_diffuse = rows per solve; temps_dev [n_solves]
        ("n_solves", ctypes.c_int32), ("n_diffuse", ctypes.c_int32), ("temps_dev", c_vp),
    ]


STEP_PARAMS_WORDS = 8    # sizeof(mbd_step_params) / 4
STEP_CTL_WORDS = 32      # sizeof(mbd_step_ctl) / 4
ENV_CAR2D, ENV_PUSHT = 0, 1   # mbd_step_plan.env_kind (model == NULL)


def lib():
    global _LIB
    if _LIB is not None:
        return _LIB
    path = _build.OUT
    # Build when the library is missing OR was built from other sources (content hash stored beside the .so: copied
    # trees carry arbitrary mtimes, so mtimes are not consulted).  build(force=False) re-checks inside an exclusive file
    # lock, so of N ranks starting together exactly one compiles and the others load the finished file.
    if _build.is_stale():
        try:
            path = _build.build(force=False)
        except Exception as e:  # noqa: BLE001
            raise MbdError(f"libmbd_b200.so is missing or stale and could not be built ({e}); there is no CPU fallback") from e
    L = ctypes.CDLL(path)
    L.mbd_last_error.restype = ctypes.c_char_p
    L.mbd_device_count.restype = ctypes.c_int
    L.mbd_layout_info.argtypes = [c_i32p, ctypes.c_int]
    L.mbd_model_create.restype = c_vp
    L.mbd_model_create.argtypes = [c_u32p, ctypes.c_size_t]
    L.mbd_model_destroy.argtypes = [c_vp]
    L.mbd_sample.argtypes = [c_u32p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_float, c_vp, c_vp, c_vp]
    L.mbd_rollout.argtypes = [c_vp, c_vp, c_vp, ctypes.c_int, ctypes.c_int, c_vp, c_vp, c_vp, ctypes.c_int, c_vp, c_vp, c_vp,
                              ctypes.c_int, c_vp]
    L.mbd_sample_rollout.argtypes = [c_vp, c_vp, c_u32p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_float,
                                     c_vp, c_vp, c_vp, c_vp, ctypes.c_int, c_vp, c_vp]
    L.mbd_reverse_step.argtypes = [c_vp, c_vp, c_u32p, ctypes.c_int, ctypes.c_int, ctypes.c_float, c_vp, ctypes.c_float, c_f32p,
                                   c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]
    L.mbd_car2d_rollout.argtypes = [c_vp, c_vp, c_u32p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_float,
                                    c_vp, c_vp, c_vp, c_vp, c_vp, ctypes.c_int, c_vp, c_vp, c_vp]
    L.mbd_pusht_rollout.argtypes = [c_vp, c_vp, c_u32p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_float,
                                    c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]
    L.mbd_softmax_weights.argtypes = [c_vp, c_vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_float, ctypes.c_float,
                                      c_vp, c_vp, c_vp, c_vp]
    L.mbd_weighted_sum.argtypes = [c_vp, c_vp, ctypes.c_int, ctypes.c_int, c_vp, c_vp, c_vp]
    L.mbd_weighted_sum_runs.argtypes = [c_vp, c_vp, ctypes.c_int, ctypes.c_int, c_vp, c_vp]
    L.mbd_weighted_sqerr_sum.argtypes = [c_vp, c_vp, c_vp, ctypes.c_int, ctypes.c_int, c_vp, c_vp, c_vp]
    L.mbd_peer_gather.argtypes = [ctypes.POINTER(ctypes.c_uint64), ctypes.c_int, ctypes.c_int, ctypes.c_size_t, ctypes.c_int,
                                  ctypes.c_size_t, ctypes.c_uint32, c_vp, c_vp, c_vp]
    L.mbd_test_arith.argtypes = [ctypes.c_int, c_vp, c_vp, c_vp, ctypes.c_int, c_vp]
    L.mbd_update.argtypes = [c_vp, ctypes.c_int, ctypes.c_int, c_vp, c_f32p, c_vp, c_vp]
    L.mbd_step_launch.argtypes = [ctypes.POINTER(StepPlan), c_vp]
    L.mbd_step_launch_ev.argtypes = [ctypes.POINTER(StepPlan), c_vp, c_vp, c_vp, c_vp, c_vp]
    L.mbd_event_create.restype = c_vp
    L.mbd_event_destroy.argtypes = [c_vp]
    L.mbd_event_record.argtypes = [c_vp, c_vp]
    L.mbd_event_sync.argtypes = [c_vp]
    L.mbd_event_elapsed_ms.restype = ctypes.c_float
    L.mbd_event_elapsed_ms.argtypes = [c_vp, c_vp]
    L.mbd_ffma_peak.argtypes = [c_vp, ctypes.c_int, c_f32p, c_vp]
    L.mbd_abi_sizes.argtypes = [c_i32p, ctypes.c_int]
    L.mbd_abi_batch_offsets.argtypes = [c_i32p, ctypes.c_int]
    _LIB = L
    return L


EXPORTS = ["mbd_set_kernel_variant", "mbd_set_prng_layout", "mbd_model_set_warp_order", "mbd_model_set_group_map", "mbd_set_group_stagger", "mbd_layout_info", "mbd_last_error", "mbd_device_count", "mbd_model_create", "mbd_model_destroy", "mbd_sample",
           "mbd_rollout", "mbd_sample_rollout", "mbd_reverse_step", "mbd_car2d_rollout", "mbd_pusht_rollout", "mbd_softmax_weights", "mbd_weighted_sum", "mbd_weighted_sum_runs", "mbd_weighted_sqerr_sum", "mbd_peer_gather", "mbd_test_arith", "mbd_update", "mbd_step_launch", "mbd_step_launch_ev", "mbd_event_create", "mbd_event_destroy", "mbd_event_record",
           "mbd_event_sync", "mbd_event_elapsed_ms", "mbd_ffma_peak", "mbd_abi_sizes", "mbd_abi_batch_offsets"]


def check(rc: int, what: str):
    if rc != 0:
        raise MbdError(f"{what} failed (rc={rc}): {lib().mbd_last_error().decode()}")


def key_ptr(key):
    k = np.ascontiguousarray(key, dtype=np.uint32)
    return k, k.ctypes.data_as(c_u32p)


def require_gpu():
    if lib().mbd_device_count() <= 0:
        raise MbdError("no CUDA device visible: the MBD hot path has no CPU fallback")
