"""ctypes binding of libdkb200.so (the C ABI declared in include/dkb200.h).

There is no CPU fallback: if the library is missing, or a call fails, this module raises.
"""
from __future__ import annotations

import ctypes as C
import os
import re
from typing import Optional

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libdkb200.so")
HEADER_PATH = os.path.join(_HERE, "..", "include", "dkb200.h")

DK_BF16, DK_FP16 = 0, 1
ACT_NONE, ACT_GELU_ERF, ACT_SILU, ACT_QUICK_GELU = 0, 1, 2, 3

vp = C.c_void_p
i32 = C.c_int
i64 = C.c_longlong
f32 = C.c_float


class GemmArgs(C.Structure):
    _fields_ = [
        ("dtype", i32), ("M", i32), ("N", i32), ("K", i32),
        ("A", vp), ("lda", i64),
        ("W", vp), ("ldw", i64),
        ("out", vp), ("ldc", i64),
        ("bias", vp),
        ("gate", vp), ("gate_ld", i64),
        ("res", vp), ("ldres", i64),
        ("rows_per_batch", i32),
        ("out_batch_rows", i32), ("out_row_off", i32),
        ("res_batch_rows", i32), ("res_row_off", i32),
        ("act", i32), ("w_n_major", i32),
        ("qk_q_weight", vp), ("qk_k_weight", vp), ("qk_rope", vp),
        ("qk_heads", i32), ("qk_head_dim", i32), ("qk_eps", f32),
    ]


# name -> (restype, argtypes); must list every symbol include/dkb200.h declares (tests check this)
SIGNATURES = {
    "dk_version": (C.c_char_p, []),
    "dk_last_error": (C.c_char_p, []),
    "dk_ctx_create": (i32, [i32, C.POINTER(vp)]),
    "dk_ctx_destroy": (None, [vp]),
    "dk_ctx_launch_count": (i64, [vp]),
    "dk_gemm": (i32, [vp, C.POINTER(GemmArgs), vp]),
    "dk_ln_modulate": (i32, [vp, i32, vp, vp, vp, vp, i64, i32, i32, i32, f32, vp]),
    "dk_qk_norm_rope": (i32, [vp, i32, vp, i32, i32, i32, i32, i32, vp, vp, vp, vp, vp, f32, vp]),
    "dk_attention_fwd": (i32, [vp, i32, vp, i32, i32, i32, i32, f32, i32, vp, i64, vp, i64, vp]),
    "dk_attention_tuning": (i32, [i32, i32, i32]),
    "dk_silu_add": (i32, [vp, i32, vp, vp, vp, i32, i32, i32, vp]),
    "dk_act": (i32, [vp, i32, vp, vp, i64, i32, vp]),
    "dk_patchify": (i32, [vp, i32, vp, vp, i32, i32, i32, i32, i32, vp]),
    "dk_unpatchify": (i32, [vp, i32, vp, vp, i32, i32, i32, i32, i32, vp]),
    "dk_pos_embed_crop": (i32, [vp, i32, vp, vp, i32, i32, i32, i32, vp]),
    "dk_copy_rows": (i32, [vp, i32, vp, vp, i32, i32, i32, i32, i32, i32, i32, vp]),
    "dk_sampler_prepare": (i32, [vp, i32, vp, vp, i64, i32, vp]),
    "dk_sampler_step": (i32, [vp, i32, vp, vp, vp, i64, f32, f32, f32, vp]),
    "dk_axpb_f32": (i32, [vp, vp, vp, i64, f32, f32, vp]),
    "dk_embedding": (i32, [vp, i32, vp, vp, vp, vp, i64, i32, i32, i32, vp]),
    "dk_layernorm": (i32, [vp, i32, vp, vp, vp, vp, i32, i32, f32, vp]),
    "dk_rmsnorm_f32": (i32, [vp, i32, vp, vp, vp, i32, i32, f32, vp]),
    "dk_add_f32_16": (i32, [vp, i32, vp, vp, i64, vp]),
    "dk_glu_gelu": (i32, [vp, i32, vp, vp, i64, i32, vp]),
    "dk_attention_small": (i32, [vp, i32, vp, vp, vp, i32, i32, i32, i32, f32, i32, vp]),
    "dk_dequant_q4": (i32, [vp, i32, vp, vp, vp, vp, i64, i32, i32, vp]),
    "dk_image_pre": (i32, [vp, i32, vp, vp, i64, i32, i32, vp]),
    "dk_axpby_f32": (i32, [vp, vp, vp, vp, i64, f32, f32, vp]),
    "dk_vae_sample_latent": (i32, [vp, i32, vp, vp, vp, i64, i32, f32, f32, vp]),
    "dk_cast_f32_to_16": (i32, [vp, i32, vp, vp, i64, vp]),
    "dk_cast_16_to_f32": (i32, [vp, i32, vp, vp, i64, vp]),
    "dk_groupnorm_ws_floats": (i32, [i32, i32]),
    "dk_groupnorm_stats": (i32, [vp, i32, vp, vp, vp, i32, i32, i32, i32, f32, vp]),
    "dk_groupnorm_apply": (i32, [vp, i32, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, vp]),
    "dk_conv3x3": (i32, [vp, i32, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, vp]),
    "dk_conv3x3_s2": (i32, [vp, i32, vp, vp, vp, vp, i32, i32, i32, i32, i32, vp]),
    "dk_conv_fused_supported": (i32, [i32, i32, i32, i32]),
    "dk_conv3x3_fused": (i32, [vp, i32, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, vp, vp, vp, i32, i32, vp, i32, vp]),
    "dk_conv_up_weights": (i32, [vp, i32, vp, vp, i32, i32, vp]),
    "dk_groupnorm_finalize": (i32, [vp, vp, vp, i32, i32, i32, C.c_double, f32, vp]),
    "dk_upsample_nearest2x": (i32, [vp, i32, vp, vp, i32, i32, i32, i32, vp]),
    "dk_softmax_rows": (i32, [vp, i32, vp, i64, i32, i64, f32, vp]),
    "dk_image_post": (i32, [vp, i32, vp, i32, vp, vp, i64, vp]),
    "dk_inpaint_blend": (i32, [vp, vp, vp, vp, vp, i64, i32, f32, vp]),
    "dk_image_post_masked": (i32, [vp, i32, vp, i32, vp, vp, vp, i64, vp]),
    "dk_comm_unique_id": (i32, [vp]),
    "dk_comm_init": (i32, [vp, i32, i32, vp]),
    "dk_comm_broadcast": (i32, [vp, vp, C.c_size_t, i32, vp]),
    "dk_comm_destroy": (i32, [vp]),
}


def header_symbols() -> list:
    """Function names declared in include/dkb200.h."""
    text = open(HEADER_PATH).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(dk_[a-z0-9_]+)\s*\(", text)))


class DkError(RuntimeError):
    pass


_lib = None


def load() -> C.CDLL:
    """Load libdkb200.so; raises if it has not been built (python -m diffusionkit_b200.build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise DkError(
            f"{LIB_PATH} not found: the CUDA library must be built first (python -m diffusionkit_b200.build). "
            "There is no CPU fallback."
        )
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the export is missing
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def dtype_code(dt: torch.dtype) -> int:
    if dt == torch.bfloat16:
        return DK_BF16
    if dt == torch.float16:
        return DK_FP16
    raise DkError(f"unsupported 16-bit dtype {dt}")


def ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    if t is None:
        return None
    return t.data_ptr()


class Context:
    """One dk_ctx per (process, device)."""

    def __init__(self, device: int = 0):
        self.lib = load()
        if not torch.cuda.is_available():
            raise DkError("no CUDA device: diffusionkit_b200 runs on B200 (sm_100a) only; there is no CPU fallback")
        h = vp()
        rc = self.lib.dk_ctx_create(device, C.byref(h))
        if rc != 0:
            raise DkError(self.lib.dk_last_error().decode())
        self.handle = h
        self.device = device

    def close(self):
        if getattr(self, "handle", None):
            self.lib.dk_ctx_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def check(self, rc: int):
        if rc != 0:
            raise DkError(self.lib.dk_last_error().decode())

    @property
    def stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream   # the stream of THIS context's device

    @property
    def launches(self) -> int:
        return int(self.lib.dk_ctx_launch_count(self.handle))

    def call(self, name: str, *args):
        """Call lib.<name>(ctx, *args, stream)."""
        fn = getattr(self.lib, name)
        self.check(fn(self.handle, *args, self.stream))
