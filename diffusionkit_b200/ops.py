"""Typed Python wrappers over the C ABI (torch tensors are only the device-memory containers).

Every function launches hand-written sm_100a kernels from libdkb200.so asynchronously on the current
torch CUDA stream.  Nothing here has a torch / CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Optional

import torch

from . import _lib
from ._lib import ACT_GELU_ERF, ACT_NONE, ACT_QUICK_GELU, ACT_SILU, Context, GemmArgs, dtype_code, ptr

_ctx = {}


def ctx(device: Optional[int] = None) -> Context:
    if device is None:
        device = torch.cuda.current_device()
    c = _ctx.get(device)
    if c is None:
        c = Context(device)
        _ctx[device] = c
    return c


_graph_launches = 0


def note_graph_launches(n: int):
    """kernels replayed from a captured CUDA graph (the C-side counter only sees the capture pass)"""
    global _graph_launches
    _graph_launches += n


def launch_count() -> int:
    return sum(c.launches for c in _ctx.values()) + _graph_launches


def _chk16(t: torch.Tensor, name: str):
    if t.dtype not in (torch.bfloat16, torch.float16):
        raise _lib.DkError(f"{name}: expected a bf16/fp16 tensor, got {t.dtype}")
    if not t.is_cuda:
        raise _lib.DkError(f"{name}: expected a CUDA tensor (there is no CPU fallback)")


def gemm(
    A: torch.Tensor,
    W: torch.Tensor,
    out: Optional[torch.Tensor] = None,
    bias: Optional[torch.Tensor] = None,
    act: int = ACT_NONE,
    gate: Optional[torch.Tensor] = None,
    res: Optional[torch.Tensor] = None,
    rows_per_batch: int = 0,
    out_batch_rows: int = 0,
    out_row_off: int = 0,
    res_batch_rows: Optional[int] = None,
    res_row_off: int = 0,
    w_n_major: bool = False,
    N: Optional[int] = None,
    qk: Optional[tuple] = None,
) -> torch.Tensor:
    """out = res + gate * act(A @ W.T + bias)   (see include/dkb200.h, dk_gemm).

    A: [M, K] (row stride may exceed K), W: [N, K] (nn.Linear layout) or [K, N] when w_n_major.
    out: 2-D view [rows, >=N] whose row stride is the leading dimension.
    """
    _chk16(A, "gemm.A")
    _chk16(W, "gemm.W")
    assert A.dim() == 2 and W.dim() == 2 and A.stride(1) == 1 and W.stride(1) == 1
    M, K = A.shape
    if w_n_major:
        assert W.shape[0] == K
        n = W.shape[1]
    else:
        assert W.shape[1] == K, f"K mismatch {A.shape} x {W.shape}"
        n = W.shape[0]
    if N is not None:
        n = N
    if out is None:
        out = torch.empty((M, n), dtype=A.dtype, device=A.device)
    assert out.dim() == 2 and out.stride(1) == 1
    a = GemmArgs()
    a.dtype = dtype_code(A.dtype)
    a.M, a.N, a.K = M, n, K
    a.A, a.lda = ptr(A), A.stride(0)
    a.W, a.ldw = ptr(W), W.stride(0)
    a.out, a.ldc = ptr(out), out.stride(0)
    a.bias = ptr(bias)
    a.gate = ptr(gate)
    a.gate_ld = gate.stride(0) if gate is not None else 0
    a.res = ptr(res)
    a.ldres = res.stride(0) if res is not None else 0
    a.rows_per_batch = rows_per_batch
    a.out_batch_rows = out_batch_rows if rows_per_batch else 0
    a.out_row_off = out_row_off
    if res_batch_rows is None:
        res_batch_rows = rows_per_batch
    a.res_batch_rows = res_batch_rows if rows_per_batch else 0
    a.res_row_off = res_row_off
    a.act = act
    a.w_n_major = 1 if w_n_major else 0
    if qk is not None:
        # (heads, head_dim, q_norm_weight | None, k_norm_weight | None, rope table | None, eps)
        heads, hd, qw, kw, rope, eps = qk
        a.qk_heads, a.qk_head_dim, a.qk_eps = heads, hd, eps
        a.qk_q_weight, a.qk_k_weight, a.qk_rope = ptr(qw), ptr(kw), ptr(rope)
    c = ctx(A.device.index)
    c.check(c.lib.dk_gemm(c.handle, C.byref(a), c.stream))
    return out


def ln_modulate(x, shift, scale, rows_per_batch: int, eps: float = 1e-6, out=None):
    """y = LN(x) * (1 + scale[b]) + shift[b]; x [rows, h]; shift/scale 2-D views [B, h] (row stride = mod_ld)."""
    _chk16(x, "ln_modulate.x")
    rows, h = x.shape
    assert x.is_contiguous() and shift.stride(0) == scale.stride(0) and shift.stride(1) == 1
    if out is None:
        out = torch.empty_like(x)
    c = ctx(x.device.index)
    c.call("dk_ln_modulate", dtype_code(x.dtype), ptr(x), ptr(out), ptr(shift), ptr(scale), shift.stride(0), rows,
           rows_per_batch, h, eps)
    return out


def qk_norm_rope(qkv, S: int, heads: int, d: int, split: int, q_w=None, k_w=None, q_w2=None, k_w2=None, rope=None,
                 eps: float = 1e-6):
    _chk16(qkv, "qk_norm_rope.qkv")
    assert qkv.is_contiguous() and qkv.shape[1] == 3 * heads * d
    if rope is not None:
        assert rope.dtype == torch.float32 and rope.is_contiguous() and rope.numel() == S * d
    c = ctx(qkv.device.index)
    c.call("dk_qk_norm_rope", dtype_code(qkv.dtype), ptr(qkv), qkv.shape[0], S, heads, d, split, ptr(q_w), ptr(k_w),
           ptr(q_w2), ptr(k_w2), ptr(rope), eps)
    return qkv


def attention(qkv, B: int, S: int, heads: int, d: int, out0, split: Optional[int] = None, out1=None,
              scale: Optional[float] = None):
    """softmax(scale q k^T) v over the packed [B*S, 3*heads*d] buffer; rows < split go to out0, the rest to out1."""
    _chk16(qkv, "attention.qkv")
    assert qkv.is_contiguous() and qkv.shape == (B * S, 3 * heads * d)
    if split is None:
        split = S
    if scale is None:
        scale = 1.0 / math.sqrt(d)
    c = ctx(qkv.device.index)
    c.call("dk_attention_fwd", dtype_code(qkv.dtype), ptr(qkv), B, S, heads, d, scale, split, ptr(out0),
           out0.stride(0) if out0 is not None else 0, ptr(out1), out1.stride(0) if out1 is not None else 0)
    return out0, out1


def silu_add(y, temb, out=None):
    """out[t*B + b] = silu(y[b] + temb[t])."""
    _chk16(y, "silu_add.y")
    B, h = y.shape
    n_t = temb.shape[0]
    if out is None:
        out = torch.empty((n_t * B, h), dtype=y.dtype, device=y.device)
    c = ctx(y.device.index)
    c.call("dk_silu_add", dtype_code(y.dtype), ptr(y), ptr(temb), ptr(out), n_t, B, h)
    return out


def act(x, kind: int, out=None):
    _chk16(x, "act.x")
    if out is None:
        out = torch.empty_like(x)
    c = ctx(x.device.index)
    c.call("dk_act", dtype_code(x.dtype), ptr(x), ptr(out), x.numel(), kind)
    return out


def patchify(latent, order: int, out=None):
    _chk16(latent, "patchify.latent")
    B, H, W, Cc = latent.shape
    if out is None:
        out = torch.empty((B * (H // 2) * (W // 2), 4 * Cc), dtype=latent.dtype, device=latent.device)
    c = ctx(latent.device.index)
    c.call("dk_patchify", dtype_code(latent.dtype), ptr(latent), ptr(out), B, H, W, Cc, order)
    return out


def unpatchify(rows, B: int, H: int, W: int, Cc: int, order: int, out=None):
    _chk16(rows, "unpatchify.rows")
    if out is None:
        out = torch.empty((B, H, W, Cc), dtype=rows.dtype, device=rows.device)
    c = ctx(rows.device.index)
    c.call("dk_unpatchify", dtype_code(rows.dtype), ptr(rows), ptr(out), B, H, W, Cc, order)
    return out


def pos_embed_crop(table, max_hw: int, hp: int, wp: int):
    _chk16(table, "pos_embed_crop.table")
    h = table.shape[1]
    out = torch.empty((hp * wp, h), dtype=table.dtype, device=table.device)
    c = ctx(table.device.index)
    c.call("dk_pos_embed_crop", dtype_code(table.dtype), ptr(table), ptr(out), max_hw, hp, wp, h)
    return out


def copy_rows(src, dst, B: int, rows: int, h: int, dst_rows: int, dst_off: int, src_rows: int, src_off: int):
    _chk16(src, "copy_rows.src")
    c = ctx(src.device.index)
    c.call("dk_copy_rows", dtype_code(src.dtype), ptr(src), ptr(dst), B, rows, h, dst_rows, dst_off, src_rows, src_off)
    return dst


def sampler_prepare(x, xin, reps: int):
    assert x.dtype == torch.float32 and x.is_contiguous()
    c = ctx(x.device.index)
    c.call("dk_sampler_prepare", dtype_code(xin.dtype), ptr(x), ptr(xin), x.numel(), reps)
    return xin


def sampler_step(x, xin, out, sigma: float, sigma_next: float, cfg_weight: float):
    assert x.dtype == torch.float32 and x.is_contiguous()
    c = ctx(x.device.index)
    c.call("dk_sampler_step", dtype_code(xin.dtype), ptr(x), ptr(xin), ptr(out), x.numel(), sigma, sigma_next,
           cfg_weight)
    return x


def axpb(x, a: float, b: float, out=None):
    assert x.dtype == torch.float32 and x.is_contiguous()
    if out is None:
        out = torch.empty_like(x)
    c = ctx(x.device.index)
    c.call("dk_axpb_f32", ptr(x), ptr(out), x.numel(), a, b)
    return out


# ------------------------------------------------------------------------------------------------ text encoders
def embedding(table, ids, pos=None, out=None):
    """out[i] = table[ids[i]] (+ pos[i % len(pos)]); ids int32 (any shape, flattened)"""
    _chk16(table, "embedding.table")
    assert table.is_contiguous() and ids.dtype == torch.int32 and ids.is_contiguous() and ids.is_cuda
    n, d = ids.numel(), table.shape[1]
    if out is None:
        out = torch.empty((n, d), dtype=table.dtype, device=table.device)
    c = ctx(table.device.index)
    c.call("dk_embedding", dtype_code(table.dtype), ptr(table), ptr(ids), ptr(pos), ptr(out), n, d, table.shape[0],
           0 if pos is None else pos.shape[0])
    return out


def layernorm(x, weight, bias, eps: float = 1e-5, out=None):
    _chk16(x, "layernorm.x")
    rows, h = x.shape
    assert x.is_contiguous() and weight.is_contiguous() and bias.is_contiguous()
    if out is None:
        out = torch.empty_like(x)
    c = ctx(x.device.index)
    c.call("dk_layernorm", dtype_code(x.dtype), ptr(x), ptr(out), ptr(weight), ptr(bias), rows, h, eps)
    return out


def rmsnorm_f32(x, weight, eps: float = 1e-6, out=None):
    """x fp32 [rows, d] -> 16-bit (weight's dtype) weight * x * rsqrt(mean(x^2) + eps)"""
    _chk16(weight, "rmsnorm_f32.weight")
    assert x.dtype == torch.float32 and x.is_contiguous() and x.dim() == 2
    if out is None:
        out = torch.empty(x.shape, dtype=weight.dtype, device=x.device)
    c = ctx(x.device.index)
    c.call("dk_rmsnorm_f32", dtype_code(weight.dtype), ptr(x), ptr(weight), ptr(out), x.shape[0], x.shape[1], eps)
    return out


def add_f32_16(x, y):
    _chk16(y, "add_f32_16.y")
    assert x.dtype == torch.float32 and x.is_contiguous() and y.is_contiguous() and x.numel() == y.numel()
    c = ctx(x.device.index)
    c.call("dk_add_f32_16", dtype_code(y.dtype), ptr(x), ptr(y), x.numel())
    return x


def glu_gelu(h, out=None):
    _chk16(h, "glu_gelu.h")
    rows, F2 = h.shape
    assert h.is_contiguous() and F2 % 2 == 0
    if out is None:
        out = torch.empty((rows, F2 // 2), dtype=h.dtype, device=h.device)
    c = ctx(h.device.index)
    c.call("dk_glu_gelu", dtype_code(h.dtype), ptr(h), ptr(out), rows, F2 // 2)
    return out


def attention_small(qkv, B: int, S: int, heads: int, scale: float, rel_bias=None, causal: bool = False, out=None):
    """packed (q | k | v) [B*S, 3*heads*64] -> [B*S, heads*64]; rel_bias [heads, 2S-1] or None"""
    _chk16(qkv, "attention_small.qkv")
    assert qkv.is_contiguous() and tuple(qkv.shape) == (B * S, 3 * heads * 64)
    if rel_bias is not None:
        assert rel_bias.dtype == qkv.dtype and rel_bias.is_contiguous() and tuple(rel_bias.shape) == (heads, 2 * S - 1)
    if out is None:
        out = torch.empty((B * S, heads * 64), dtype=qkv.dtype, device=qkv.device)
    c = ctx(qkv.device.index)
    c.call("dk_attention_small", dtype_code(qkv.dtype), ptr(qkv), ptr(rel_bias), ptr(out), B, S, heads, 64, scale,
           1 if causal else 0)
    return out


def dequant_q4(wq, scales, biases, group_size: int = 64, out=None):
    """MLX affine 4-bit weight (wq [N, K/8] uint32 stored as int32/uint32, scales/biases [N, K/group] 16-bit) ->
    dense [N, K] in the scales' dtype"""
    _chk16(scales, "dequant_q4.scales")
    assert wq.dtype in (torch.int32, torch.uint32) and wq.dim() == 2 and wq.is_contiguous() and wq.is_cuda
    assert scales.is_contiguous() and biases.is_contiguous() and biases.dtype == scales.dtype
    N, K = wq.shape[0], wq.shape[1] * 8
    assert tuple(scales.shape) == tuple(biases.shape) == (N, K // group_size)
    if out is None:
        out = torch.empty((N, K), dtype=scales.dtype, device=wq.device)
    c = ctx(wq.device.index)
    c.call("dk_dequant_q4", dtype_code(scales.dtype), ptr(wq), ptr(scales), ptr(biases), ptr(out), N, K, group_size)
    return out


def image_pre(img_u8, dtype, cpad: int = 64):
    """uint8 NHWC [B,H,W,>=3] -> 16-bit NHWC [B,H,W,cpad] in [-1, 1] (channels 3.. zero)"""
    assert img_u8.dtype == torch.uint8 and img_u8.is_contiguous() and img_u8.dim() == 4 and img_u8.is_cuda
    B, H, W, Cs = img_u8.shape
    out = torch.empty((B, H, W, cpad), dtype=dtype, device=img_u8.device)
    c = ctx(img_u8.device.index)
    c.call("dk_image_pre", dtype_code(dtype), ptr(img_u8), ptr(out), B * H * W, Cs, cpad)
    return out


def axpby(x, y, a: float, b: float, out=None):
    assert x.dtype == torch.float32 and y.dtype == torch.float32 and x.is_contiguous() and y.is_contiguous()
    if out is None:
        out = torch.empty_like(x)
    c = ctx(x.device.index)
    c.call("dk_axpby_f32", ptr(x), ptr(y), ptr(out), x.numel(), a, b)
    return out


def vae_sample_latent(hidden, noise, shift: float, scale: float, out=None):
    """hidden NHWC [B,H,W,2C] 16-bit (mean | logvar), noise fp32 [B,H,W,C] -> process_in(mean + std * noise) fp32"""
    _chk16(hidden, "vae_sample_latent.hidden")
    B, H, W, C2 = hidden.shape
    assert hidden.is_contiguous() and noise.dtype == torch.float32 and noise.is_contiguous()
    assert tuple(noise.shape) == (B, H, W, C2 // 2)
    if out is None:
        out = torch.empty((B, H, W, C2 // 2), dtype=torch.float32, device=hidden.device)
    assert out.dtype == torch.float32 and out.is_contiguous()
    c = ctx(hidden.device.index)
    c.call("dk_vae_sample_latent", dtype_code(hidden.dtype), ptr(hidden), ptr(noise), ptr(out), B * H * W, C2 // 2,
           shift, scale)
    return out


def cast_to_16(x, dtype, out=None):
    assert x.dtype == torch.float32 and x.is_contiguous()
    if out is None:
        out = torch.empty(x.shape, dtype=dtype, device=x.device)
    c = ctx(x.device.index)
    c.call("dk_cast_f32_to_16", dtype_code(dtype), ptr(x), ptr(out), x.numel())
    return out


def cast_to_f32(x, out=None):
    _chk16(x, "cast_to_f32.x")
    if out is None:
        out = torch.empty(x.shape, dtype=torch.float32, device=x.device)
    c = ctx(x.device.index)
    c.call("dk_cast_16_to_f32", dtype_code(x.dtype), ptr(x), ptr(out), x.numel())
    return out


def groupnorm_stats(x, G: int, eps: float = 1e-5, ws=None):
    """x NHWC [B, H, W, C] -> stats [B, G, 2] (mean, rstd)."""
    _chk16(x, "groupnorm_stats.x")
    B, H, W, Cc = x.shape
    c = ctx(x.device.index)
    n_ws = c.lib.dk_groupnorm_ws_floats(B, G)
    if ws is None:
        ws = torch.empty(n_ws, dtype=torch.float32, device=x.device)
    assert ws.numel() >= n_ws
    stats = torch.empty((B, G, 2), dtype=torch.float32, device=x.device)
    c.call("dk_groupnorm_stats", dtype_code(x.dtype), ptr(x), ptr(stats), ptr(ws), B, H * W, Cc, G, eps)
    return stats


def groupnorm_apply(x, stats, gamma, beta, G: int, silu: bool, out=None):
    _chk16(x, "groupnorm_apply.x")
    B, H, W, Cc = x.shape
    if out is None:
        out = torch.empty_like(x)
    c = ctx(x.device.index)
    c.call("dk_groupnorm_apply", dtype_code(x.dtype), ptr(x), ptr(out), ptr(stats), ptr(gamma), ptr(beta), B, H * W, Cc,
           G, 1 if silu else 0)
    return out


def conv3x3(x, w, bias=None, res=None, out=None):
    """x NHWC [B,H,W,Cin], w [Cout,3,3,Cin] -> NHWC [B,H,W,Cout] (+ res)."""
    _chk16(x, "conv3x3.x")
    B, H, W, Cin = x.shape
    Cout = w.shape[0]
    assert w.shape == (Cout, 3, 3, Cin) and x.is_contiguous() and w.is_contiguous()
    if out is None:
        out = torch.empty((B, H, W, Cout), dtype=x.dtype, device=x.device)
    c = ctx(x.device.index)
    c.call("dk_conv3x3", dtype_code(x.dtype), ptr(x), ptr(w), ptr(bias), ptr(res), ptr(out), B, H, W, Cin, Cout)
    return out


def conv3x3_s2(x, w, bias=None, out=None):
    """stride-2 3x3 conv with bottom/right zero padding: x NHWC [B,H,W,Cin] -> [B,H/2,W/2,Cout]"""
    _chk16(x, "conv3x3_s2.x")
    B, H, W, Cin = x.shape
    Cout = w.shape[0]
    assert w.shape == (Cout, 3, 3, Cin) and x.is_contiguous() and w.is_contiguous()
    if out is None:
        out = torch.empty((B, H // 2, W // 2, Cout), dtype=x.dtype, device=x.device)
    c = ctx(x.device.index)
    c.call("dk_conv3x3_s2", dtype_code(x.dtype), ptr(x), ptr(w), ptr(bias), ptr(out), B, H, W, Cin, Cout)
    return out


def conv_fused_supported(H: int, W: int, Cin: int, Cout: int) -> bool:
    return bool(_lib.load().dk_conv_fused_supported(H, W, Cin, Cout))


def conv_up_weights(w):
    """w [Cout,3,3,Cin] -> phase weights [4*Cout, 4*Cin] of conv3x3(nearest2x(.)) (see dk_conv_up_weights)"""
    _chk16(w, "conv_up_weights.w")
    Cout, _, _, Cin = w.shape
    assert w.shape == (Cout, 3, 3, Cin) and w.is_contiguous()
    wp = torch.empty((4 * Cout, 4 * Cin), dtype=w.dtype, device=w.device)
    c = ctx(w.device.index)
    c.call("dk_conv_up_weights", dtype_code(w.dtype), ptr(w), ptr(wp), Cout, Cin)
    return wp


def conv3x3_fused(x, w, bias=None, res=None, out=None, up: bool = False, gn=None, silu: bool = False,
                  out_partial=None, out_G: int = 32):
    """fused [GroupNorm+SiLU] -> [nearest 2x] -> conv3x3 (+bias, +res) -> out (+ output GroupNorm partial sums).
    gn = (stats [B,G,2] fp32, gamma [Cin], beta [Cin], G) or None; up: w must be conv_up_weights(w3x3)."""
    _chk16(x, "conv3x3_fused.x")
    B, H, W, Cin = x.shape
    if up:
        Cout = w.shape[0] // 4
        assert tuple(w.shape) == (4 * Cout, 4 * Cin)
        Ho, Wo = 2 * H, 2 * W
    else:
        Cout = w.shape[0]
        assert tuple(w.shape) == (Cout, 3, 3, Cin)
        Ho, Wo = H, W
    assert x.is_contiguous() and w.is_contiguous()
    if out is None:
        out = torch.empty((B, Ho, Wo, Cout), dtype=x.dtype, device=x.device)
    assert tuple(out.shape) == (B, Ho, Wo, Cout) and out.is_contiguous()
    if res is not None:
        assert tuple(res.shape) == tuple(out.shape) and res.is_contiguous()
    stats = gamma = beta = None
    G = 0
    if gn is not None:
        stats, gamma, beta, G = gn
        assert stats.dtype == torch.float32 and stats.is_contiguous() and tuple(stats.shape) == (B, G, 2)
    if out_partial is not None:
        assert out_partial.dtype == torch.float32 and out_partial.is_contiguous()
        assert out_partial.numel() >= B * (Ho * Wo // 128) * out_G * 2
    c = ctx(x.device.index)
    c.call("dk_conv3x3_fused", dtype_code(x.dtype), ptr(x), ptr(w), ptr(bias), ptr(res), ptr(out), B, H, W, Cin, Cout,
           1 if up else 0, ptr(stats), ptr(gamma), ptr(beta), G, 1 if silu else 0, ptr(out_partial), out_G)
    return out


def groupnorm_finalize(partial, B: int, G: int, slots: int, count: float, eps: float = 1e-5, stats=None):
    """partial [B, slots, G, 2] (sum, sumsq) -> stats [B, G, 2] (mean, rstd)"""
    assert partial.dtype == torch.float32 and partial.is_contiguous()
    if stats is None:
        stats = torch.empty((B, G, 2), dtype=torch.float32, device=partial.device)
    c = ctx(partial.device.index)
    c.call("dk_groupnorm_finalize", ptr(partial), ptr(stats), B, G, slots, float(count), eps)
    return stats


def upsample_nearest2x(x, out=None):
    _chk16(x, "upsample.x")
    B, H, W, Cc = x.shape
    if out is None:
        out = torch.empty((B, 2 * H, 2 * W, Cc), dtype=x.dtype, device=x.device)
    c = ctx(x.device.index)
    c.call("dk_upsample_nearest2x", dtype_code(x.dtype), ptr(x), ptr(out), B, H, W, Cc)
    return out


def softmax_rows(x, scale: float = 1.0):
    _chk16(x, "softmax_rows.x")
    assert x.dim() == 2 and x.stride(1) == 1
    c = ctx(x.device.index)
    c.call("dk_softmax_rows", dtype_code(x.dtype), ptr(x), x.shape[0], x.shape[1], x.stride(0), scale)
    return x


def image_post(x, want_u8: bool = True):
    """decoder output NHWC [B,H,W,Cpad] -> (float [B,H,W,3] in [0,1], uint8 [B,H,W,3])."""
    _chk16(x, "image_post.x")
    B, H, W, Cp = x.shape
    f = torch.empty((B, H, W, 3), dtype=torch.float32, device=x.device)
    u = torch.empty((B, H, W, 3), dtype=torch.uint8, device=x.device) if want_u8 else None
    c = ctx(x.device.index)
    c.call("dk_image_post", dtype_code(x.dtype), ptr(x), Cp, ptr(f), ptr(u), B * H * W)
    return f, u


def _chk_mask(mask, shape, name: str):
    if mask.dtype != torch.uint8 or not mask.is_cuda or not mask.is_contiguous() or tuple(mask.shape) != tuple(shape):
        raise _lib.DkError(f"{name}: expected a contiguous CUDA uint8 tensor of shape {tuple(shape)}, got "
                           f"{mask.dtype} {tuple(mask.shape)} on {mask.device}")


def inpaint_blend(x, x0, noise, mask, sigma_next: float):
    """in place on x: x = mask ? x : sigma_next * noise + (1 - sigma_next) * x0.  x, x0, noise fp32 NHWC [B,H,W,C]
    (C % 4 == 0); mask uint8 [B,H,W], non-zero = the cell is being regenerated (left untouched)."""
    for t, n in ((x, "x"), (x0, "x0"), (noise, "noise")):
        if t.dtype != torch.float32 or not t.is_cuda or not t.is_contiguous() or t.shape != x.shape:
            raise _lib.DkError(f"inpaint_blend.{n}: expected a contiguous CUDA fp32 tensor of shape {tuple(x.shape)}")
    _chk_mask(mask, x.shape[:-1], "inpaint_blend.mask")
    c = ctx(x.device.index)
    c.call("dk_inpaint_blend", ptr(x0), ptr(noise), ptr(mask), ptr(x), mask.numel(), x.shape[-1], sigma_next)
    return x


def image_post_masked(x, orig, mask):
    """decoder output NHWC [B,H,W,Cpad] 16-bit, orig uint8 [B,H,W,3], pixel mask uint8 [B,H,W] -> uint8 [B,H,W,3]:
    image_post's uint8 where the mask is non-zero, orig where it is zero."""
    _chk16(x, "image_post_masked.x")
    B, H, W, Cp = x.shape
    _chk_mask(orig, (B, H, W, 3), "image_post_masked.orig")
    _chk_mask(mask, (B, H, W), "image_post_masked.mask")
    u = torch.empty((B, H, W, 3), dtype=torch.uint8, device=x.device)
    c = ctx(x.device.index)
    c.call("dk_image_post_masked", dtype_code(x.dtype), ptr(x), Cp, ptr(orig), ptr(mask), ptr(u), B * H * W)
    return u
