"""MMDiT (SD3 dual-stream / FLUX dual + single-stream) forward on B200.

Host-side mirror of the reference module (python/src/diffusionkit/mlx/mmdit.py:22-266): same public methods
(`cache_modulation_params`, `__call__(latent_image_embeddings, token_level_text_embeddings, timestep)`,
`clear_modulation_params_cache`), same parameter names.  Every FLOP runs in hand-written sm_100a kernels reached
through the C ABI (ops.py -> libdkb200.so); torch tensors are only the HBM containers.

B200 layout decisions (vs. the reference's per-module MLX graph):
  * q/k/v projections of a stream are ONE GEMM (packed [3h, h] weight; k has no bias — quirk Q3) whose epilogue applies
    the per-head QK-RMSNorm and RoPE (FLUX) and scatters rows straight into the joint [text|image] (FLUX) /
    [image|text] (SD3) sequence buffer — no norm / rope / concat kernels.
  * adaLN gate * (.) + residual is fused into the o_proj / fc2 GEMM epilogues (in place on the residual stream);
    bias + exact-erf GELU into fc1's.
  * FLUX single-stream blocks: attention output and GELU(fc1) land in one [B*S, 5h] buffer and
    o_proj + fc2 run as ONE K=5h GEMM with the packed [Wo | W2] weight (upstream `linear2`, mlx/model_io.py:253-259).
  * all adaLN modulations for all timesteps and all blocks are ONE batched GEMM (replaces the reference's
    per-timestep, per-block loop, mmdit.py:91-175); a step selects its rows with one small D2D copy, which keeps the
    forward's launch sequence timestep-invariant (CUDA-graph capturable).
"""
from __future__ import annotations

import math
import os
from collections import OrderedDict
from typing import Dict, List, Optional, Tuple

import torch

from . import ops
from ._lib import ACT_GELU_ERF, ACT_NONE, ACT_SILU, DkError
from .config import MMDiTConfig, PositionalEncoding


class _Stream:
    """Packed weights of one TransformerBlock (reference mmdit.py:395-548)."""

    __slots__ = ("name", "n_mod", "mod_off", "w_qkv", "b_qkv", "w_o", "b_o", "w_fc1", "b_fc1", "w_fc2", "b_fc2",
                 "w_out", "q_norm", "k_norm", "skip_post")


class MMDiT:
    def __init__(self, config: MMDiTConfig, params: Dict[str, torch.Tensor], device=None):
        self.config = config
        c = config
        any_p = next(iter(params.values()))
        self.device = torch.device(device) if device is not None else any_p.device
        if self.device.type != "cuda":
            raise DkError("MMDiT: parameters must live on a CUDA device (no CPU fallback)")
        self.dtype = any_p.dtype
        if self.dtype not in (torch.bfloat16, torch.float16):
            raise DkError(f"MMDiT: weights must be bf16 or fp16 (w16), got {self.dtype}")
        if c.pos_embed_type not in (PositionalEncoding.LearnedInputEmbedding, PositionalEncoding.PreSDPARope):
            raise ValueError(f"Unsupported positional encoding type: {c.pos_embed_type}")  # mmdit.py:50-52
        self.h = c.hidden_size
        self.heads = c.num_heads
        self.d = c.head_dim
        if self.d not in (64, 128):
            raise DkError(f"MMDiT: head dim {self.d} unsupported by the attention kernel (64 or 128)")
        self.is_flux = c.depth_unified > 0
        self._pack(params)
        self._mod_index: Dict[float, int] = {}
        self._mod_all: Optional[torch.Tensor] = None
        self._mod_cur: Optional[torch.Tensor] = None
        self._mod_batch = 0
        # Everything a captured forward bakes device pointers of — workspace, RoPE table, cropped positional embedding —
        # is owned PER SHAPE KEY together with the graph that uses it, so a graph can never outlive its buffers when one
        # model serves several resolutions / text lengths (LRU-bounded: evicting a shape drops its graph with it).
        self._shapes: "OrderedDict[tuple, dict]" = OrderedDict()
        self.max_cached_shapes = int(os.environ.get("DK_MAX_CACHED_SHAPES", "4"))
        # CUDA-graph replay of the (timestep-invariant) forward: one captured graph per input shape
        self.use_cuda_graphs = os.environ.get("DK_CUDA_GRAPHS", "1") != "0"

    # ------------------------------------------------------------------------------------------ weight packing
    def _pack(self, P: Dict[str, torch.Tensor]):
        c, h = self.config, self.h
        dev, dt = self.device, self.dtype

        def get(name):
            t = P[name]
            if t.device != dev or t.dtype != dt:
                t = t.to(device=dev, dtype=dt)
            return t.contiguous()

        # reference weight name -> the tensor or window of a packed buffer holding it (2-D [out, in]); in-place
        # weight edits (lora.py) go through these views so captured graphs keep their pointers
        views: Dict[str, torch.Tensor] = {}
        self.weight_views = views
        self.w_x = get("x_embedder.proj.weight").reshape(h, -1).contiguous()          # (h, 64)
        self.b_x = get("x_embedder.proj.bias")
        self.pos_table = get("x_pos_embedder.pos_embed.weight") if "x_pos_embedder.pos_embed.weight" in P else None
        self.y0 = (get("y_embedder.mlp.layers.0.weight"), get("y_embedder.mlp.layers.0.bias"))
        self.y2 = (get("y_embedder.mlp.layers.2.weight"), get("y_embedder.mlp.layers.2.bias"))
        self.t0 = (get("t_embedder.mlp.layers.0.weight"), get("t_embedder.mlp.layers.0.bias"))
        self.t2 = (get("t_embedder.mlp.layers.2.weight"), get("t_embedder.mlp.layers.2.bias"))
        self.w_ctx, self.b_ctx = get("context_embedder.weight"), get("context_embedder.bias")
        self.w_final, self.b_final = get("final_layer.linear.weight"), get("final_layer.linear.bias")
        views["x_embedder.proj.weight"] = self.w_x
        for name, w in (("y_embedder.mlp.layers.0", self.y0[0]), ("y_embedder.mlp.layers.2", self.y2[0]),
                        ("t_embedder.mlp.layers.0", self.t0[0]), ("t_embedder.mlp.layers.2", self.t2[0]),
                        ("context_embedder", self.w_ctx), ("final_layer.linear", self.w_final)):
            views[name + ".weight"] = w

        mod_w, mod_b, mod_rows = [], [], {}
        self.mod_total = 0

        def add_mod(prefix) -> int:
            off = self.mod_total
            w = get(prefix + ".adaLN_modulation.layers.1.weight")
            mod_rows[prefix + ".adaLN_modulation.layers.1.weight"] = (off, off + w.shape[0])
            mod_w.append(w)
            mod_b.append(get(prefix + ".adaLN_modulation.layers.1.bias"))
            self.mod_total += w.shape[0]
            return off

        def stream(prefix, n_mod, skip_post=False, parallel=False) -> _Stream:
            s = _Stream()
            s.name, s.n_mod, s.skip_post = prefix, n_mod, skip_post
            s.mod_off = add_mod(prefix)
            wq, wk, wv = get(prefix + ".attn.q_proj.weight"), get(prefix + ".attn.k_proj.weight"), get(
                prefix + ".attn.v_proj.weight")
            s.w_qkv = torch.cat([wq, wk, wv], dim=0).contiguous()
            for j, n in enumerate("qkv"):
                views[f"{prefix}.attn.{n}_proj.weight"] = s.w_qkv[j * h:(j + 1) * h]
            bq, bv = get(prefix + ".attn.q_proj.bias"), get(prefix + ".attn.v_proj.bias")
            s.b_qkv = torch.cat([bq, torch.zeros_like(bq), bv]).contiguous()          # no k bias (quirk Q3)
            s.w_o = s.b_o = s.w_fc1 = s.b_fc1 = s.w_fc2 = s.b_fc2 = s.w_out = None
            if not skip_post:
                s.b_o = get(prefix + ".attn.o_proj.bias")
                s.w_fc1, s.b_fc1 = get(prefix + ".mlp.fc1.weight"), get(prefix + ".mlp.fc1.bias")
                if parallel:
                    # u += gate * ([attn | gelu(fc1)] @ [Wo | W2]^T + bo); fc2.bias is zeroed (mmdit.py:742)
                    s.w_out = torch.cat([get(prefix + ".attn.o_proj.weight"), get(prefix + ".mlp.fc2.weight")],
                                        dim=1).contiguous()
                    views[prefix + ".attn.o_proj.weight"] = s.w_out[:, :h]
                    views[prefix + ".mlp.fc2.weight"] = s.w_out[:, h:]
                else:
                    s.w_o = get(prefix + ".attn.o_proj.weight")
                    s.w_fc2, s.b_fc2 = get(prefix + ".mlp.fc2.weight"), get(prefix + ".mlp.fc2.bias")
                    views[prefix + ".attn.o_proj.weight"] = s.w_o
                    views[prefix + ".mlp.fc2.weight"] = s.w_fc2
                views[prefix + ".mlp.fc1.weight"] = s.w_fc1
            s.q_norm = s.k_norm = None
            if c.use_qk_norm:
                s.q_norm = get(prefix + ".qk_norm.q_norm.weight")
                s.k_norm = get(prefix + ".qk_norm.k_norm.weight")
            return s

        self.double: List[Tuple[_Stream, _Stream]] = []
        for i in range(c.depth_multimodal):
            skip_text = (i == c.depth_multimodal - 1) and (c.depth_unified < 1)       # mmdit.py:62-66
            img = stream(f"multimodal_transformer_blocks.{i}.image_transformer_block", 6)
            txt = stream(f"multimodal_transformer_blocks.{i}.text_transformer_block", 2 if skip_text else 6,
                         skip_post=skip_text)
            self.double.append((img, txt))
        self.single: List[_Stream] = []
        par = c.parallel_mlp_for_unified_blocks
        if c.depth_unified > 0 and not par:
            raise DkError("MMDiT: unified blocks without parallel MLP are not used by any reference preset")
        for i in range(c.depth_unified):
            self.single.append(stream(f"unified_transformer_blocks.{i}.transformer_block", 3, parallel=True))
        self.final_mod_off = add_mod("final_layer")
        self.w_mod = torch.cat(mod_w, dim=0).contiguous()                             # (mod_total, h)
        self.b_mod = torch.cat(mod_b, dim=0).contiguous()
        for name, (r0, r1) in mod_rows.items():
            views[name] = self.w_mod[r0:r1]

    # ------------------------------------------------------------------------------------------ modulation cache
    def timestep_embedding(self, t: torch.Tensor) -> torch.Tensor:
        """Sinusoid in config.dtype arithmetic, cos first (reference mmdit.py:379-389, quirk Q5).  Tiny host math."""
        c = self.config
        half = c.frequency_embed_dim // 2
        cd = c.dtype
        ar = torch.arange(0, half, dtype=torch.float32).to(cd)
        freqs = torch.exp(-math.log(c.max_period) * ar.float() / half).to(cd)
        args = (t.reshape(-1, 1).float().to(cd).float() * freqs.float()[None]).to(cd)
        return torch.cat([torch.cos(args.float()).to(cd), torch.sin(args.float()).to(cd)], dim=-1)

    def cache_modulation_params(self, pooled_text_embeddings: torch.Tensor, timesteps):
        """All adaLN modulation vectors for every timestep and every block in one batched GEMM
        (reference mmdit.py:77-180).  pooled: (B, P); timesteps: iterable of floats already rounded to the activation
        dtype by the caller (mlx/__init__.py:769-771)."""
        pooled = pooled_text_embeddings.reshape(pooled_text_embeddings.shape[0], -1)
        pooled = pooled.to(device=self.device, dtype=self.dtype).contiguous()
        B = pooled.shape[0]
        ts = [float(t) for t in (timesteps.tolist() if hasattr(timesteps, "tolist") else timesteps)]
        n_t = len(ts)
        y = ops.gemm(ops.gemm(pooled, self.y0[0], bias=self.y0[1], act=ACT_SILU), self.y2[0], bias=self.y2[1])
        temb = self.timestep_embedding(torch.tensor(ts, dtype=torch.float32)).to(device=self.device, dtype=self.dtype)
        tvec = ops.gemm(ops.gemm(temb.contiguous(), self.t0[0], bias=self.t0[1], act=ACT_SILU), self.t2[0],
                        bias=self.t2[1])
        cin = ops.silu_add(y, tvec)                                                    # (n_t * B, h)
        self._mod_all = ops.gemm(cin, self.w_mod, bias=self.b_mod)                    # (n_t * B, mod_total)
        if self._mod_cur is None or self._mod_batch != B:
            # persistent buffer: captured graphs read the current step's modulation rows from this address
            self._mod_cur = torch.empty((B, self.mod_total), dtype=self.dtype, device=self.device)
            for st in self._shapes.values():
                st["graph"] = None
        self._mod_batch = B
        self._mod_index = {}
        for i, t in enumerate(ts):
            self._mod_index.setdefault(t, i)
        self._cur_t = None

    def clear_modulation_params_cache(self):
        self._mod_index, self._mod_all = {}, None

    def invalidate_modulation_cache(self):
        """after a weight edit: drop the cached rows AND the current timestep, so a forward without a fresh
        cache_modulation_params raises KeyError instead of reusing rows of the old adaLN weights"""
        self.clear_modulation_params_cache()
        self._cur_t = None

    def select_timestep(self, timestep: float):
        """Make `timestep`'s modulation rows current (one D2D copy; keeps the forward timestep-invariant)."""
        key = float(timestep)
        if key not in self._mod_index:
            raise KeyError(f"timestep {key} not in the modulation cache (call cache_modulation_params first)")
        i = self._mod_index[key]
        B = self._mod_batch
        self._mod_cur.copy_(self._mod_all[i * B:(i + 1) * B])
        self._cur_t = key

    def _mod(self, s_off: int, k: int) -> torch.Tensor:
        """k-th h-wide modulation vector of a block: view (B, h) with row stride mod_total."""
        return self._mod_cur[:, s_off + k * self.h: s_off + (k + 1) * self.h]

    # ------------------------------------------------------------------------------------------ workspace
    def _shape_state(self, key: tuple) -> dict:
        st = self._shapes.get(key)
        if st is None:
            while len(self._shapes) >= max(1, self.max_cached_shapes):
                self._shapes.popitem(last=False)            # least recently used shape: buffers AND graph go together
            st = {"ws": None, "rope": None, "pos": None, "graph": None}
            self._shapes[key] = st
        else:
            self._shapes.move_to_end(key)
        return st

    def _workspace(self, st: dict, B: int, N: int, T: int):
        if st["ws"] is not None:
            return st["ws"]
        h, dt, dev = self.h, self.dtype, self.device
        S = N + T
        r = self.config.mlp_ratio

        def buf(*shape):
            return torch.empty(shape, dtype=dt, device=dev)

        ws = {
            "img": buf(B * N, h), "txt": buf(B * T, h),
            "m_img": buf(B * N, h), "m_txt": buf(B * T, h),
            "qkv": buf(B * S, 3 * h),
            "o_img": buf(B * N, h), "o_txt": buf(B * T, h),
            "hid_img": buf(B * N, r * h), "hid_txt": buf(B * T, r * h),
            "rows_in": buf(B * N, self.w_x.shape[1]), "rows_out": buf(B * N, self.w_final.shape[0]),
        }
        if self.is_flux:
            ws["u"] = buf(B * S, h)
            ws["m_u"] = buf(B * S, h)
            ws["cat"] = buf(B * S, (1 + r) * h)
        st["ws"] = ws
        return ws

    def _rope_table(self, st: dict, T: int, hp: int, wp: int) -> torch.Tensor:
        """(S, d/2, 2) fp32 cos/sin; text tokens at position (0,0,0), image token (r, c) at (0, r, c)
        (reference mmdit.py:865-911).  Cached across calls like the reference (:916-932)."""
        if st["rope"] is not None:
            return st["rope"]
        axes = self.config.rope_axes_dim
        S = T + hp * wp
        pos = torch.zeros((S, 3), dtype=torch.float32)
        pos[T:, 1] = torch.arange(hp, dtype=torch.float32)[:, None].expand(hp, wp).reshape(-1)
        pos[T:, 2] = torch.arange(wp, dtype=torch.float32)[None, :].expand(hp, wp).reshape(-1)
        parts = []
        for a, dim in enumerate(axes):
            scale = torch.arange(0, dim, 2, dtype=torch.float32) / dim
            omega = 1.0 / (10000.0 ** scale)
            parts.append(pos[:, a:a + 1] * omega[None, :])
        ang = torch.cat(parts, dim=-1)
        assert ang.shape[1] == self.d // 2, "sum(rope_axes_dim) must equal the head dim"
        st["rope"] = torch.stack([torch.cos(ang), torch.sin(ang)], dim=-1).contiguous().to(self.device)
        return st["rope"]

    # ------------------------------------------------------------------------------------------ forward
    def _qk_fused(self, s: _Stream, rope):
        """epilogue spec for the packed QKV GEMM: per-head QK-RMSNorm (+ RoPE) fused in (None: nothing to fuse)"""
        if s.q_norm is None and rope is None:
            return None
        return (self.heads, self.d, s.q_norm, s.k_norm, rope, 1e-6)

    def _attn_stream_pre(self, s: _Stream, x, m, rows_per_batch, S, row_off, qkv, rope):
        ops.ln_modulate(x, self._mod(s.mod_off, 0), self._mod(s.mod_off, 1), rows_per_batch,
                        self.config.layer_norm_eps, out=m)
        ops.gemm(m, s.w_qkv, out=qkv, bias=s.b_qkv, rows_per_batch=rows_per_batch, out_batch_rows=S,
                 out_row_off=row_off, qk=self._qk_fused(s, rope))

    def _stream_post(self, s: _Stream, x, o, m, hid, rows_per_batch):
        """x += gate1 * o_proj(o); x += gate2 * fc2(gelu(fc1(LN(x)(1+scale2)+shift2)))  (mmdit.py:521-548)"""
        ops.gemm(o, s.w_o, out=x, bias=s.b_o, gate=self._mod(s.mod_off, 2), res=x, rows_per_batch=rows_per_batch,
                 out_batch_rows=rows_per_batch)
        ops.ln_modulate(x, self._mod(s.mod_off, 3), self._mod(s.mod_off, 4), rows_per_batch,
                        self.config.layer_norm_eps, out=m)
        ops.gemm(m, s.w_fc1, out=hid, bias=s.b_fc1, act=ACT_GELU_ERF)
        ops.gemm(hid, s.w_fc2, out=x, bias=s.b_fc2, gate=self._mod(s.mod_off, 5), res=x,
                 rows_per_batch=rows_per_batch, out_batch_rows=rows_per_batch)

    def __call__(self, latent_image_embeddings: torch.Tensor, token_level_text_embeddings: torch.Tensor,
                 timestep=None) -> torch.Tensor:
        """latent (B, H, W, 16) NHWC, text (B, T, 1, 4096) or (B, T, 4096), timestep (B,) tensor / float
        (all entries equal, as in the reference which reads timestep[0], mmdit.py:445-447) -> (B, H, W, 16)."""
        c = self.config
        x = latent_image_embeddings
        if x.dim() != 4:
            raise ValueError(f"Input tensor must have rank 4, got {x.dim()}")
        B, H, W, Cl = x.shape
        if H % c.patch_size or W % c.patch_size:
            raise DkError("latent height/width must be divisible by the patch size")
        text = token_level_text_embeddings
        if text.dim() == 4:
            text = text.squeeze(2)
        T = text.shape[1]
        text = text.reshape(B * T, -1).to(dtype=self.dtype)
        if not text.is_contiguous():
            text = text.contiguous()
        x = x.to(dtype=self.dtype)
        if not x.is_contiguous():
            x = x.contiguous()
        if timestep is not None:
            tval = float(timestep.reshape(-1)[0]) if torch.is_tensor(timestep) else float(timestep)
            if tval != getattr(self, "_cur_t", None):
                self.select_timestep(tval)
        if self._mod_cur is None or self._mod_batch != B:
            raise DkError(f"modulation cache holds batch {self._mod_batch}, forward got batch {B}")
        state = self._shape_state((B, H, W, Cl, T))
        if not self.use_cuda_graphs:
            return self._forward_impl(state, x, text, B, H, W, Cl, T)
        entry = state["graph"]
        if entry is None:
            sx, stx = x.clone(), text.clone()
            self._forward_impl(state, sx, stx, B, H, W, Cl, T)    # eager warm-up: workspaces, tables, func attributes
            torch.cuda.current_stream().synchronize()
            n0 = ops.launch_count()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                so = self._forward_impl(state, sx, stx, B, H, W, Cl, T)
            entry = (graph, sx, stx, so, ops.launch_count() - n0)
            state["graph"] = entry
        graph, sx, stx, so, n_launch = entry
        sx.copy_(x)
        stx.copy_(text)
        graph.replay()
        ops.note_graph_launches(n_launch)
        return so

    def _forward_impl(self, state, x, text, B, H, W, Cl, T):
        c = self.config
        hp, wp = H // c.patch_size, W // c.patch_size
        N = hp * wp
        S = N + T
        h, heads, d = self.h, self.heads, self.d
        ws = self._workspace(state, B, N, T)
        img, txt, qkv = ws["img"], ws["txt"], ws["qkv"]

        # ---- input adapters (mmdit.py:195-206)
        ops.gemm(text, self.w_ctx, out=txt, bias=self.b_ctx)
        if c.patchify_via_reshape:
            ops.patchify(x, 0, out=ws["rows_in"])
            ops.gemm(ws["rows_in"], self.w_x, out=img, bias=self.b_x)
        else:
            ops.patchify(x, 1, out=ws["rows_in"])
            if state["pos"] is None:
                state["pos"] = ops.pos_embed_crop(self.pos_table, c.max_latent_resolution, hp, wp)
            ops.gemm(ws["rows_in"], self.w_x, out=img, bias=self.b_x, res=state["pos"], rows_per_batch=N,
                     out_batch_rows=N, res_batch_rows=0)

        rope = self._rope_table(state, T, hp, wp) if c.pos_embed_type == PositionalEncoding.PreSDPARope else None
        # joint sequence order: FLUX [text, image] (mmdit.py:594-606), SD3 [image, text] (:608-625)
        if self.is_flux:
            off_img, off_txt, split = T, 0, T
        else:
            off_img, off_txt, split = 0, N, N

        for (si, st) in self.double:
            self._attn_stream_pre(si, img, ws["m_img"], N, S, off_img, qkv, rope)
            self._attn_stream_pre(st, txt, ws["m_txt"], T, S, off_txt, qkv, rope)
            if self.is_flux:
                ops.attention(qkv, B, S, heads, d, ws["o_txt"], split=split, out1=ws["o_img"])
            else:
                ops.attention(qkv, B, S, heads, d, ws["o_img"], split=split, out1=ws["o_txt"])
            self._stream_post(si, img, ws["o_img"], ws["m_img"], ws["hid_img"], N)
            if not st.skip_post:
                self._stream_post(st, txt, ws["o_txt"], ws["m_txt"], ws["hid_txt"], T)

        if self.is_flux:
            u, m_u, cat = ws["u"], ws["m_u"], ws["cat"]
            ops.copy_rows(txt, u, B, T, h, S, 0, T, 0)                                 # u = [text | image] (:234-236)
            ops.copy_rows(img, u, B, N, h, S, T, N, 0)
            for s in self.single:                                                      # mmdit.py:693-751
                ops.ln_modulate(u, self._mod(s.mod_off, 0), self._mod(s.mod_off, 1), S, c.layer_norm_eps, out=m_u)
                ops.gemm(m_u, s.w_qkv, out=qkv, bias=s.b_qkv, rows_per_batch=S, out_batch_rows=S,
                         qk=self._qk_fused(s, rope))
                ops.attention(qkv, B, S, heads, d, cat[:, :h])
                ops.gemm(m_u, s.w_fc1, out=cat[:, h:], bias=s.b_fc1, act=ACT_GELU_ERF)
                ops.gemm(cat, s.w_out, out=u, bias=s.b_o, gate=self._mod(s.mod_off, 2), res=u, rows_per_batch=S,
                         out_batch_rows=S)
            ops.copy_rows(u, img, B, N, h, N, 0, S, T)                                 # image part (:245-247)

        # ---- final layer (mmdit.py:780-796) + unpatchify / unpack
        ops.ln_modulate(img, self._mod(self.final_mod_off, 0), self._mod(self.final_mod_off, 1), N, c.layer_norm_eps,
                        out=ws["m_img"])
        ops.gemm(ws["m_img"], self.w_final, out=ws["rows_out"], bias=self.b_final)
        out = ops.unpatchify(ws["rows_out"], B, H, W, Cl, 0 if c.patchify_via_reshape else 1)
        return out
