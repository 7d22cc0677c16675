# -*- coding: utf-8 -*-
"""ctypes binding of libstoke_b200.so (include/stoke_b200.h).  The library is the product: there is no Python or torch
fallback for any entry point -- a missing library or a failing call raises."""
import ctypes as C
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libstoke_b200.so")

STK_MAX_WORLD = 8
STK_IPC_HANDLE_BYTES = 64
F32, BF16, F16 = 0, 1, 2
REDUCE_ALL, REDUCE_SCATTER = 0, 1
NORM_NONE, NORM_L2, NORM_INF, NORM_P = 0, 1, 2, 3
CLIP_NONE, CLIP_NORM, CLIP_VALUE = 0, 1, 2
OPT_ADAM, OPT_ADAMW, OPT_SGD = 0, 1, 2
RF_FINAL, RF_ZERO_INPUT, RF_UNSCALE = 1, 2, 4
OPT_K1_ALGO, OPT_MEM_MODE, OPT_K1_MAX_BLOCKS, OPT_NVLS_MAX_BLOCKS = 1, 2, 3, 5
K1_ALGO_LDG, K1_ALGO_BULK, K1_ALGO_NVLS = 0, 1, 2
MAX_GROUPS, MAX_SEGMENTS, LOSS_RING = 8, 64, 256
ERR_INVALID, ERR_CUDA, ERR_STATE, ERR_PEER, ERR_UNSUPPORTED = -1, -2, -3, -4, -5


class StokeB200Error(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libstoke_b200: {msg} (status {code})")
        self.code = code


class Caps(C.Structure):
    _fields_ = [("sm_major", C.c_int), ("sm_minor", C.c_int), ("sm_count", C.c_int), ("rank", C.c_int),
                ("world", C.c_int), ("device", C.c_int), ("peer_access", C.c_int), ("multicast", C.c_int),
                ("hbm_bytes", C.c_size_t)]


class ScalerState(C.Structure):
    _fields_ = [("scale", C.c_float), ("growth_factor", C.c_float), ("backoff_factor", C.c_float),
                ("growth_interval", C.c_int32), ("growth_tracker", C.c_int32), ("enabled", C.c_int32),
                ("found_inf", C.c_int32), ("grad_norm", C.c_float), ("opt_steps", C.c_int64),
                ("skipped_steps", C.c_int64)]


class OptimHyper(C.Structure):
    _fields_ = [("kind", C.c_int), ("lr", C.c_double), ("beta1", C.c_double), ("beta2", C.c_double),
                ("eps", C.c_double), ("weight_decay", C.c_double), ("momentum", C.c_double),
                ("dampening", C.c_double), ("nesterov", C.c_int), ("maximize", C.c_int), ("clip_kind", C.c_int),
                ("clip_max_norm", C.c_double), ("clip_value", C.c_double)]


class OptimArgs(C.Structure):
    _fields_ = [("hyper", C.POINTER(OptimHyper)), ("n_groups", C.c_int), ("master", C.c_void_p), ("exp_avg", C.c_void_p),
                ("exp_avg_sq", C.c_void_p), ("grad", C.c_void_p), ("grad_dtype", C.c_int), ("grad_raw", C.c_int),
                ("acc", C.c_void_p), ("grad_mul", C.c_double), ("n_local", C.c_size_t),
                ("lp_ptrs", C.POINTER(C.c_void_p)), ("lp_world", C.c_int), ("lp_dtype", C.c_int), ("lp_offset", C.c_size_t),
                ("n_seg", C.c_int), ("seg_local", C.POINTER(C.c_size_t)), ("seg_global", C.POINTER(C.c_size_t)),
                ("n_ranges", C.c_int), ("range_end_vec", C.c_void_p), ("range_group", C.c_void_p),
                ("grid_n", C.c_size_t), ("range_bc", C.c_void_p)]


class SamplerPlan(C.Structure):
    _fields_ = [("n", C.c_int64), ("buckets", C.c_int64), ("batch_size", C.c_int64), ("world", C.c_int64),
                ("rank", C.c_int64), ("drop_last", C.c_int32), ("allow_bucket_overlap", C.c_int32),
                ("shuffle", C.c_int32), ("slice_size", C.c_int64), ("per_bucket", C.c_int64),
                ("slices_per_bucket", C.c_int64), ("rounded_per_bucket", C.c_int64),
                ("rounded_per_replica", C.c_int64), ("bucket_base", C.c_int64), ("bucket_rem", C.c_int64),
                ("n_bucket_batches", C.c_int64), ("n_overlap_batches", C.c_int64), ("n_batches", C.c_int64),
                ("needs_padding", C.c_int32)]


_P = C.c_void_p
_PP = C.POINTER(C.c_void_p)
_SIGNATURES = {
    "stk_version": (C.c_int, []),
    "stk_last_error": (C.c_char_p, [_P]),
    "stk_ctx_create": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_uint, _PP]),
    "stk_ctx_destroy": (C.c_int, [_P]),
    "stk_caps": (C.c_int, [_P, C.POINTER(Caps)]),
    "stk_mem_alloc_shared": (C.c_int, [_P, C.c_size_t, _PP, C.c_char_p]),
    "stk_mem_open_peers": (C.c_int, [_P, _P, C.c_char_p, _PP]),
    "stk_mem_free_shared": (C.c_int, [_P, _P]),
    "stk_comm_local": (C.c_int, [_P, C.c_char_p]),
    "stk_comm_connect": (C.c_int, [_P, C.c_char_p]),
    "stk_comm_check": (C.c_int, [_P, _P]),
    "stk_comm_poll": (C.c_int, [_P]),
    "stk_multicast_try_bind": (C.c_int, [_P, _P, _PP]),
    "stk_multicast_release": (C.c_int, [_P, _P]),
    "stk_state_create": (C.c_int, [_P, C.POINTER(C.c_int)]),
    "stk_state_select": (C.c_int, [_P, C.c_int]),
    "stk_state_destroy": (C.c_int, [_P, C.c_int]),
    "stk_option_set": (C.c_int, [_P, C.c_int, C.c_int]),
    "stk_option_get": (C.c_int, [_P, C.c_int, C.POINTER(C.c_int)]),
    "stk_profile_enable": (C.c_int, [_P, C.c_int]),
    "stk_profile_read": (C.c_int, [_P, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_int)]),
    "stk_profile_read_k1_device": (C.c_int, [_P, C.POINTER(C.c_double), C.POINTER(C.c_int), C.POINTER(C.c_double), _P]),
    "stk_profile_read_k2_device": (C.c_int, [_P, C.POINTER(C.c_double), C.POINTER(C.c_int), _P]),
    "stk_scaler_set": (C.c_int, [_P, C.POINTER(ScalerState), _P]),
    "stk_scaler_get": (C.c_int, [_P, C.POINTER(ScalerState), _P]),
    "stk_scaler_scale_ptr": (_P, [_P]),
    "stk_grad_accumulate": (C.c_int, [_P, _P, C.c_int, _P, C.c_size_t, C.c_int, C.c_int, _P]),
    "stk_grad_reduce": (C.c_int, [_P, C.c_int, _PP, C.c_int, _PP, _PP, C.c_int, C.c_size_t, C.c_double, C.c_int,
                                  C.c_double, C.c_uint, _P]),
    "stk_grad_norm": (C.c_int, [_P, _P, C.c_int, _P, C.c_size_t, C.c_double, C.c_int, C.c_double, C.c_uint, _P]),
    "stk_grad_scale": (C.c_int, [_P, _P, C.c_size_t, C.c_int, C.c_double, C.c_double, _P]),
    "stk_shard_range": (C.c_int, [C.c_size_t, C.c_int, C.c_int, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]),
    "stk_optim_step": (C.c_int, [_P, C.POINTER(OptimHyper), _P, _P, _P, _P, C.c_size_t, _PP, C.c_int, C.c_int,
                                 C.c_size_t, _P]),
    "stk_optim_step_ex": (C.c_int, [_P, C.POINTER(OptimArgs), _P]),
    "stk_optim_range_prologue": (C.c_int, [_P, C.POINTER(OptimHyper), C.c_int, C.c_int, _P, _P, _P, _P]),
    "stk_step_epilogue": (C.c_int, [_P, _P]),
    "stk_loss_sync": (C.c_int, [_P, _P, C.c_int, C.POINTER(C.c_double), _P]),
    "stk_loss_sync_begin": (C.c_int, [_P, _P, C.c_int, C.POINTER(C.c_int64), _P]),
    "stk_loss_sync_wait": (C.c_int, [_P, C.c_int64, C.POINTER(C.c_double)]),
    "stk_barrier": (C.c_int, [_P, _P]),
    "stk_bcast": (C.c_int, [_P, _PP, C.c_size_t, C.c_int, _P]),
    "stk_randperm": (C.c_int, [C.c_uint64, C.POINTER(C.c_int64), C.c_int, _P]),
    "stk_sampler_plan": (C.c_int, [C.POINTER(SamplerPlan)]),
    "stk_sampler_last_slice": (C.c_int, [C.POINTER(SamplerPlan), C.c_int64, _P]),
    "stk_argsort_tmp_bytes": (C.c_size_t, [C.c_size_t]),
    "stk_argsort_u32": (C.c_int, [_P, _P, C.c_size_t, _P, _P, _P]),
    "stk_sampler_indices": (C.c_int, [_P, C.POINTER(SamplerPlan), _P, _P, _P, _P, _P, _P]),
}
EXPORTS = tuple(_SIGNATURES)

_lib = None
_lock = threading.Lock()


def load():
    """Loads libstoke_b200.so (built in-tree by ``stoke_b200/csrc/build.py`` / ``__graft_entry__.build()``)."""
    global _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                # not a fallback: the only way forward is the CUDA library, so try to compile it in-tree (nvcc, sm_100a)
                try:
                    from .csrc.build import build as _build

                    _build()
                except Exception as e:  # noqa: BLE001
                    raise StokeB200Error(
                        ERR_STATE, f"{LIB_PATH} is missing and could not be built ({type(e).__name__}: {e}) -- build it "
                        f"with `python stoke_b200/csrc/build.py` (there is no non-CUDA fallback)") from e
            lib = C.CDLL(LIB_PATH)
            for name, (res, args) in _SIGNATURES.items():
                fn = getattr(lib, name)
                fn.restype = res
                fn.argtypes = args
            _lib = lib
    return _lib


def check(code, ctx=None):
    if code != 0:
        msg = load().stk_last_error(ctx)
        raise StokeB200Error(code, msg.decode() if msg else "unknown error")


def ptr_array(ptrs):
    arr = (C.c_void_p * len(ptrs))()
    for i, p in enumerate(ptrs):
        arr[i] = p
    return arr
