"""ctypes binding of libseqdiff_b200.so (include/seqdiff_b200.h).  No fallback: if the library is not
built or does not load, every entry point raises."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# SEQDIFF_DEBUG_BOUNDS=1 selects the debug build (device-side asserts + workspace guard bands; build.py with the same variable)
LIB_PATH = os.environ.get("SEQDIFF_LIB") or os.path.join(HERE, "libseqdiff_b200_dbg.so" if os.environ.get("SEQDIFF_DEBUG_BOUNDS") == "1" else "libseqdiff_b200.so")

FP32, BF16, FP16 = 0, 1, 2
PRECISIONS = {"fp32": FP32, "bf16": BF16, "fp16": FP16}


class SeqdiffConfig(C.Structure):
    _fields_ = [
        ("hidden_size", C.c_int32),
        ("num_attention_heads", C.c_int32),
        ("intermediate_size", C.c_int32),
        ("num_hidden_layers", C.c_int32),
        ("max_position_embeddings", C.c_int32),
        ("feature_size", C.c_int32),
        ("relative_key", C.c_int32),
        ("layer_norm_eps", C.c_float),
    ]


# name -> (restype, argtypes): one entry per symbol declared in include/seqdiff_b200.h
_vp, _i, _u64, _u32, _i64 = C.c_void_p, C.c_int, C.c_uint64, C.c_uint32, C.c_int64
PROTOTYPES = {
    "seqdiff_abi_version": (_i, []),
    "seqdiff_last_error": (C.c_char_p, []),
    "seqdiff_launch_count": (_u64, []),
    "seqdiff_profile_begin": (_i, [_vp]),
    "seqdiff_profile_end": (_i, [C.c_char_p, _i, C.POINTER(C.c_float), C.POINTER(C.c_int), _i]),
    "seqdiff_debug_attn_trace": (_i, [_vp]),
    "seqdiff_debug_check_guards": (_i, [C.POINTER(_i), C.POINTER(_i), _vp]),
    "seqdiff_model_create": (_i, [C.POINTER(SeqdiffConfig), _i, C.POINTER(_vp)]),
    "seqdiff_model_destroy": (_i, [_vp]),
    "seqdiff_model_set_tensor": (_i, [_vp, C.c_char_p, _vp, _i64, _vp]),
    "seqdiff_model_finalize": (_i, [_vp, _vp]),
    "seqdiff_forward": (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "seqdiff_reverse_step": (_i, [_vp, _i, _i, _i, _vp, _vp, _i, _vp, _u64, _u64, _u32, _vp, _vp, _vp]),
    "seqdiff_apply_aa_noise": (_i, [_vp, _i, _i, _vp, _vp, _u64, _u64, _u32, _vp, _vp, _vp]),
    "seqdiff_collate": (_i, [_i, _vp, _vp, _vp, _vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "seqdiff_sample": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _u64, _u64, _vp, _vp]),
    "seqdiff_sample_ex": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _u64, _u64, _i, _vp, _vp]),
    "seqdiff_sample_multi": (_i, [_vp, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _u64, _u64, _i, _vp, _vp]),
    "seqdiff_decode": (_i, [_i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "seqdiff_loss_terms": (_i, [_i, _vp, _vp, _vp, _vp, _vp, _vp]),
    "seqdiff_train_param_count": (_i64, [_vp]),
    "seqdiff_train_param_table": (_i, [_vp, C.c_char_p, _i, C.POINTER(_i64), C.POINTER(_i64), _i]),
    "seqdiff_op_gemm_tn": (_i, [_i, _i, _i, _i, _vp, _vp, _vp, _i, _vp]),
    "seqdiff_train_grad_buckets": (_i, [_vp, C.POINTER(_i64), _i]),
    "seqdiff_train_set_bucket_events": (_i, [_vp, C.POINTER(_vp), _i]),
    "seqdiff_train_step": (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, C.c_float, C.c_float, _u64, _u32, _vp, _vp, _vp, _vp]),
    "seqdiff_adamw_step": (_i, [_vp, _vp, _vp, _vp, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, _i, _vp, _vp]),
    "seqdiff_model_get_tensor": (_i, [_vp, C.c_char_p, _vp, _i64, _vp]),
    "seqdiff_struct_train_step": (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, C.c_float, C.c_float, _u64, _u32, _vp, _vp, _vp, _vp]),
    "seqdiff_struct_loss_terms": (_i, [_i, _i, _vp, _vp, _vp, _vp, _vp]),
    "seqdiff_struct_model_create": (_i, [C.POINTER(SeqdiffConfig), _i, C.POINTER(_vp)]),
    "seqdiff_struct_forward": (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "seqdiff_struct_p_sample": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _u64, _u64, _i, _vp, _vp]),
    "seqdiff_struct_sample": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _u64, _u64, _vp, _vp, _vp]),
    "seqdiff_struct_sample_ex": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _u64, _u64, _i, _vp, _vp, _vp]),
    "seqdiff_struct_sample_multi": (_i, [_vp, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _u64, _u64, _i, _vp, _vp, _vp]),
    "seqdiff_op_gemm": (_i, [_i, _i, _i, _i, _vp, _vp, _vp, _vp, _i, _vp, _vp]),
    "seqdiff_op_attention": (_i, [_i, _i, _i, _i, _i, _vp, _i, _vp, _i, _vp, _i, _vp, _i, _vp, _vp, _vp]),
    "seqdiff_op_attention_train_fwd": (_i, [_i, _i, _i, _i, _i, _i, _vp, _i, _vp, _i, _vp, _i, _vp, _i, _vp, C.c_float, _u64, _u32, _u32, _vp, _vp]),
    "seqdiff_op_attention_train_bwd": (_i, [_i, _i, _i, _i, _i, _i, _vp, _i, _vp, _i, _vp, _i, _vp, _i, _vp, C.c_float, _u64, _u32, _u32, _vp, _vp, _vp, _vp, _vp, _vp]),
    "seqdiff_op_layernorm": (_i, [_i, _i, _i, _vp, _vp, _vp, C.c_float, _vp, _vp, _vp, _vp]),
    "seqdiff_op_philox_u32": (_i, [_u64, _u64, _u32, _i, _i, _vp, _vp]),
    "seqdiff_op_gemm_ex": (_i, [_i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp]),
    "seqdiff_op_attention_packed": (_i, [_i, _i, _i, _i, _i, _vp, _i, _vp, _i, _vp, _i, _vp, _i, _vp, _i, _vp, _vp, _vp, _i, _i, _i, _vp, _vp]),
}

_LIB = None


class SeqdiffError(RuntimeError):
    pass


def lib():
    """Loads the CUDA library.  Raises if it has not been built (python __graft_entry__.py build)."""
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            raise SeqdiffError(
                f"{LIB_PATH} is missing: build it with `python e3-invaraint-diffusion-model_b200/build.py` "
                "(there is no CPU / PyTorch fallback for this path)")
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(l, name)
            fn.restype = res
            fn.argtypes = args
        if l.seqdiff_abi_version() != 1:
            raise SeqdiffError("libseqdiff_b200.so ABI version mismatch")
        _LIB = l
    return _LIB


def check(rc: int):
    if rc != 0:
        msg = lib().seqdiff_last_error()
        raise SeqdiffError(f"seqdiff error {rc}: {msg.decode() if msg else '?'}")


def profile(fn, stream=None):
    """Runs fn() with the library's event profiler on; returns {tag: (total_ms, launches)}."""
    l = lib()
    check(l.seqdiff_profile_begin(stream))
    try:
        fn()
    finally:
        cap, stride = 64, 48
        tags = C.create_string_buffer(cap * stride)
        ms = (C.c_float * cap)()
        cnt = (C.c_int * cap)()
        n = l.seqdiff_profile_end(tags, stride, ms, cnt, cap)
    if n < 0:
        raise SeqdiffError("profiler failed")
    return {tags.raw[i * stride:(i + 1) * stride].split(b"\0")[0].decode(): (float(ms[i]), int(cnt[i])) for i in range(n)}


class _GraphIds:
    """Position of this process in the global stream of in-kernel sampling noise.  The Philox noise of the samplers is keyed by
    (seed, GLOBAL graph id, residue / element, step); every stochastic call that is not handed an explicit `graph_id0` takes the
    next block of ids from here, so consecutive batches / repeated calls draw fresh noise (as the reference does from torch's
    global generator) while one cached CUDA graph keeps serving them (the key lives in device memory).  Sharded front ends take
    ONE block for the whole batch on every rank, which keeps the ranks' counters in step."""

    def __init__(self):
        self.next = 0

    def take(self, n: int) -> int:
        lo = self.next
        self.next += int(n)
        return lo

    def reset(self, value: int = 0):
        self.next = int(value)


GRAPH_IDS = _GraphIds()


def ptr(t):
    """Device pointer of a torch tensor (None -> NULL)."""
    return None if t is None else C.c_void_p(t.data_ptr())
