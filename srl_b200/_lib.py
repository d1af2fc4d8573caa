"""ctypes binding of the C-ABI in include/srl_b200.h (libsrl_b200.so).

This is the only place Python touches the native library.  There is deliberately no fallback: if
the shared object is missing, `load_library()` raises `MissingCudaLibrary`; if a call returns a
non-zero status, `check()` raises `SrlCudaError` carrying `srl_last_error()` -- the reference's
convention at this boundary is that exceptions propagate out of `Trainer.step`
(distributed/system/trainer_worker.py:171,496-498).
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_int, c_int32, c_int64, c_size_t, c_uint32, c_uint64, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_NAME = "libsrl_b200.so"

SRL_LANE_PART = 8
SRL_LOSS_OUT_LEN = 16
SRL_MAX_LEAVES = 32
SRL_MAX_HEADS = 8
SRL_K4B_MAX_SUM_K = 199
SRL_K4B_MAX_SUM_K_MASKED = 159
SRL_MAX_LOSS_BATCH = 32
ABI_VERSION = 12

# enum srl_loss_out
OUT_LOSS, OUT_POLICY_LOSS, OUT_VALUE_LOSS, OUT_ENTROPY_LOSS = 0, 1, 2, 3
OUT_ADVANTAGE, OUT_IMPORTANCE_WEIGHT, OUT_CLIP_RATIO, OUT_VALUE_TARGETS, OUT_DENORM_VALUE, OUT_MASK_SUM = 4, 5, 6, 7, 8, 9
VALUE_LOSS_CODES = {"mse": 0, "huber": 1, "smoothl1": 2}


class MissingCudaLibrary(RuntimeError):
    """libsrl_b200.so has not been built; run `python -m srl_b200.build` (needs nvcc)."""


class SrlCudaError(RuntimeError):
    """A C-ABI entry point returned a non-zero status."""

    def __init__(self, fn: str, status: int, message: str):
        super().__init__(f"{fn} failed with status {status}: {message}")
        self.fn, self.status, self.message = fn, status, message


class PpoHyper(ctypes.Structure):
    """struct srl_ppo_hyper"""
    _fields_ = [
        ("eps_clip", c_double),
        ("value_eps_clip", c_double),
        ("c_clip", c_double),
        ("value_loss_weight", c_double),
        ("entropy_bonus_weight", c_double),
        ("vl_param", c_double),
        ("adv_eps", c_double),
        ("value_loss", c_int32),
        ("clip_value", c_int32),
        ("dual_clip", c_int32),
        ("normalize_old_value", c_int32),
    ]


class LossProblem(ctypes.Structure):
    """struct srl_loss_problem"""
    _fields_ = [(k, c_void_p) for k in ("new_logp", "v_pred", "entropy", "lane_idx", "norm_stats", "local_stats",
                                        "g_logp", "g_value", "g_entropy", "out", "out_f32", "workspace")]


class LeafDesc(ctypes.Structure):
    """struct srl_leaf_desc"""
    _fields_ = [("src", c_void_p), ("dst", c_void_p), ("row_bytes", c_int64), ("src_slots", c_int64),
                ("src_t_stride", c_int64), ("src_slot_stride", c_int64)]


# name -> (restype, argtypes); must list every symbol include/srl_b200.h declares
SIGNATURES = {
    "srl_last_error": (c_char_p, []),
    "srl_abi_version": (c_int, []),
    "srl_pdl_enabled": (c_int, []),
    "srl_set_pdl": (c_int, [c_int]),
    "srl_device_info": (c_int, [POINTER(c_int), POINTER(c_int), POINTER(c_int)]),
    "srl_gae_scan": (c_int, [c_void_p] * 9 + [c_int, c_int, c_int, c_int, c_double, c_double, c_double, c_double] +
                     [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "srl_gae_scan_perm": (c_int, [c_void_p] * 9 + [c_int, c_int, c_int, c_int, c_double, c_double, c_double, c_double] +
                          [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p] +
                          [ctypes.c_uint64, ctypes.c_uint32, c_int, c_int, c_int, c_void_p, c_int, c_void_p, c_void_p,
                           c_void_p]),
    "srl_gae_trace": (c_int, [c_void_p] * 8 + [c_int, c_int, c_int, c_double, c_double, c_double, c_double, c_int,
                              c_void_p, c_void_p, c_void_p]),
    "srl_traj_gae": (c_int, [c_void_p] * 5 + [c_int, c_int, c_int, c_double, c_double, c_void_p, c_void_p, c_void_p]),
    "srl_n_step_return": (c_int, [c_void_p] * 4 + [c_int, c_int, c_int, c_double, c_void_p, c_void_p]),
    "srl_lane_stats": (c_int, [c_void_p] * 5 + [c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "srl_group_stats_workspace_bytes": (c_size_t, [c_int, c_int]),
    "srl_group_stats": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_size_t, c_void_p]),
    "srl_popart_update": (c_int, [c_void_p, c_void_p, c_double, c_double, c_void_p, c_void_p]),
    "srl_ppo_loss_workspace_bytes": (c_size_t, [c_int, c_int]),
    "srl_ppo_loss_finalize": (c_int, [c_void_p, c_size_t, c_int, c_void_p, c_void_p, c_void_p]),
    "srl_ppo_loss_fwd_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_int64,  # policy side
                                     c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p,  # sample side
                                     c_int, c_int, c_void_p, c_void_p, c_void_p, POINTER(PpoHyper),
                                     c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_size_t,
                                     c_void_p]),
    "srl_ppo_loss_fwd_bwd_batched": (c_int, [POINTER(LossProblem), c_int, c_int64, c_int64,
                                             c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p,
                                             c_int, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, POINTER(PpoHyper),
                                             c_size_t, c_void_p, c_void_p]),
    "srl_ppo_loss_from_logits": (c_int, [c_void_p, c_void_p, POINTER(c_int32), c_int, c_void_p,
                                         c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p,
                                         c_int, c_int, c_void_p, c_void_p, c_void_p, POINTER(PpoHyper),
                                         c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                         c_size_t, c_void_p]),
    "srl_ppo_loss_from_logits_masked": (c_int, [c_void_p, c_void_p, c_void_p, POINTER(c_int32), c_int, c_void_p,
                                                c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p,
                                                c_int, c_int, c_void_p, c_void_p, c_void_p, POINTER(PpoHyper),
                                                c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                                c_size_t, c_void_p]),
    # the _bf16 twins take the same arguments (logits, v_pred, g_logits, g_value: bfloat16 device pointers)
    "srl_ppo_loss_from_logits_bf16": (c_int, [c_void_p, c_void_p, POINTER(c_int32), c_int, c_void_p,
                                              c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p,
                                              c_int, c_int, c_void_p, c_void_p, c_void_p, POINTER(PpoHyper),
                                              c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                              c_size_t, c_void_p]),
    "srl_ppo_loss_from_logits_masked_bf16": (c_int, [c_void_p, c_void_p, c_void_p, POINTER(c_int32), c_int, c_void_p,
                                                     c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p,
                                                     c_int, c_int, c_void_p, c_void_p, c_void_p, POINTER(PpoHyper),
                                                     c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                                     c_size_t, c_void_p]),
    "srl_ppo_loss_gaussian_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_int]),
    "srl_ppo_loss_from_gaussian": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_int, c_void_p,
                                           c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p,
                                           c_int, c_int, c_void_p, c_void_p, c_void_p, POINTER(PpoHyper),
                                           c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                           c_void_p, c_size_t, c_void_p]),
    # mean, v_pred, g_mean, g_value: bfloat16 device pointers; log_std, g_log_std: bfloat16 per row, float32 when shared
    "srl_ppo_loss_from_gaussian_bf16": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_int, c_void_p,
                                                c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p,
                                                c_int, c_int, c_void_p, c_void_p, c_void_p, POINTER(PpoHyper),
                                                c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                                c_void_p, c_size_t, c_void_p]),
    "srl_philox_perm": (c_int, [c_uint64, c_uint32, c_int, c_int, c_int, c_void_p, c_void_p]),
    "srl_philox4x32_10": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    "srl_batch_gather": (c_int, [POINTER(LeafDesc), c_int, c_void_p, c_int, c_int, c_void_p]),
    "srl_rnn_chunk_prep": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p,
                                   c_void_p, c_void_p]),
    "srl_host_copy": (c_int, [c_void_p, c_void_p, c_size_t, c_int]),
    "srl_blosc1_info": (c_int, [c_void_p, c_size_t, POINTER(c_size_t), POINTER(c_size_t), POINTER(c_size_t), POINTER(c_int),
                                POINTER(c_int)]),
    "srl_blosc1_decompress": (c_int, [c_void_p, c_size_t, c_void_p, c_size_t, c_int]),
    "srl_lz4_block_decompress": (c_int, [c_void_p, c_size_t, c_void_p, c_size_t, POINTER(c_size_t)]),
    "srl_group_stats_xchg": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_size_t,
                                     c_void_p, c_void_p]),
    "srl_xchg_create": (c_int, [c_int, c_int, c_int, POINTER(c_void_p)]),
    "srl_xchg_local_handle": (c_int, [c_void_p, c_void_p]),
    "srl_xchg_connect": (c_int, [c_void_p, c_void_p]),
    "srl_xchg_allreduce_sum": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    "srl_xchg_status": (c_int, [c_void_p, POINTER(c_int)]),
    "srl_xchg_status_async": (c_int, [c_void_p, c_void_p, c_void_p]),
    "srl_xchg_set_timeout": (c_int, [c_void_p, c_double]),
    "srl_xchg_destroy": (c_int, [c_void_p]),
}

_lib = None


def lib_path() -> str:
    return os.environ.get("SRL_B200_LIB", os.path.join(_HERE, _LIB_NAME))


def load_library() -> ctypes.CDLL:
    """Loads libsrl_b200.so once and attaches the signatures above.  Raises MissingCudaLibrary."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not os.path.isfile(path):
        raise MissingCudaLibrary(
            f"{path} not found. srl_b200 has no CPU fallback: build the CUDA library with "
            f"`python -m srl_b200.build` (nvcc, sm_100a).")
    lib = ctypes.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here means header and library disagree
        fn.restype = res
        fn.argtypes = args
    got = lib.srl_abi_version()
    if got != ABI_VERSION:
        raise MissingCudaLibrary(f"{path} has ABI version {got}, python side expects {ABI_VERSION}; rebuild it")
    _lib = lib
    return lib


def check(fn_name: str, status: int) -> None:
    if status != 0:
        msg = load_library().srl_last_error()
        raise SrlCudaError(fn_name, status, msg.decode("utf-8", "replace") if msg else "")


_recording = None  # a list while HotPath records a launch plan (record_calls)


def call(fn_name: str, *args) -> None:
    """Calls a status-returning entry point and raises on failure."""
    if _recording is not None:
        _recording.append((fn_name, args))
    check(fn_name, getattr(load_library(), fn_name)(*args))


class record_calls:
    """Context manager: every `call()` inside is also appended to `calls` as (entry point, ctypes arguments) -- the launch plan
    HotPath replays with `replay_calls` (the same C-ABI calls on the same buffers, none of the Python-side checking)."""

    def __init__(self, calls: list):
        self.calls = calls

    def __enter__(self):
        global _recording
        if _recording is not None:
            raise RuntimeError("record_calls does not nest")
        _recording = self.calls
        return self.calls

    def __exit__(self, *exc):
        global _recording
        _recording = None
        return False


def bind_calls(calls):
    """[(entry point name, args)] -> [(name, bound foreign function, args)] for replay_calls."""
    lib = load_library()
    return [(name, getattr(lib, name), args) for name, args in calls]


def replay_calls(bound) -> None:
    for name, fn, args in bound:
        status = fn(*args)
        if status != 0:
            check(name, status)
