"""LoRA adapters for the MMDiT, merged in place into its packed weights.

A LoRA file names its target modules the way the upstream checkpoint does (BFL names for FLUX, SAI names for SD3 /
SD3.5, the names model_io already converts), in either of two spellings, mixed freely:
  PEFT   <module>.lora_A.weight [r, in], <module>.lora_B.weight [out, r], optional <module>.alpha
         (an optional `diffusion_model.` / `model.diffusion_model.` prefix is stripped)
  kohya  lora_unet_<module with "." -> "_">.lora_down.weight, .lora_up.weight, .alpha
The kohya form is ambiguous (`single_blocks_1_linear1` vs `single_blocks_11_linear1`), so it is resolved by lookup in
the flattened names of the model's own module list, never by splitting on "_".

Routing has one source of truth per step: upstream module -> reference weights is model_io's Linear route table (the
same splits the checkpoint converters apply), and reference weight -> packed device window is MMDiT.weight_views,
recorded by MMDiT._pack.  This module holds the parsing, the scale bookkeeping, the pristine copies and the merge.

Every touched weight is always  W = W0 + sum_i s_i * (alpha_i / r_i) * B_i @ A_i  with W0 the pristine weight, so the
result does not depend on the order of loads and unloads (the terms are concatenated in adapter-name order, which
makes it bit-for-bit independent of that order too).  One merge of one weight is ONE dk_gemm with the residual
epilogue, writing straight into the packed window the captured CUDA graphs read:
  out = view,  res = W0,  A_op = [c_1 B_1 | c_2 B_2 | ...] [out, R],  W_op = [A_1; A_2; ...]^T [in, R]
with c_i = s_i * alpha_i / r_i folded into B in fp32 before the cast to the model dtype, and R = sum r_i zero-padded to a
multiple of 8 (dk_gemm's K granularity).  The product accumulates in fp32 and is rounded once.
"""
from __future__ import annotations

import os
import re
import time
from typing import Dict, NamedTuple, Optional, Tuple

import torch

from . import model_io, ops
from .config import MMDiTConfig

Tensor = torch.Tensor


class LoraInfo(NamedTuple):
    """what load_lora applied"""
    name: str                    # the adapter's name (file stem, or "lora<N>" for a dict)
    rank: int                    # largest rank in the file (ranks may differ per module)
    n_targets: int               # model weights it changed
    skipped: Tuple[str, ...]     # modules recognised but not applied (text encoders, FLUX.1-dev's guidance_in)


class LoraPair(NamedTuple):
    A: Tensor                    # lora_A / lora_down  [r, in]
    B: Tensor                    # lora_B / lora_up    [out, r]
    alpha_over_rank: float       # alpha / r (alpha defaults to r)


_SUFFIX_PEFT = {".lora_A.weight": "A", ".lora_B.weight": "B", ".alpha": "alpha"}
_SUFFIX_KOHYA = {"lora_down.weight": "A", "lora_up.weight": "B", "alpha": "alpha"}
_UNSUPPORTED = ("hada_", "lokr_", "dora_scale")


class _Family:
    """module names of one model (from its config): Linear routes, kohya lookup table, skipped and conv modules"""

    def __init__(self, cfg: MMDiTConfig):
        self.is_flux = cfg.depth_unified > 0
        if self.is_flux:
            self.name = "FLUX"
            self.modules = model_io.flux_linear_modules(cfg.depth_multimodal, cfg.depth_unified)
            self.route = lambda m: model_io.flux_linear_route(m, cfg.mlp_ratio)
            self.skip = ("guidance_in.in_layer", "guidance_in.out_layer")     # FLUX.1-dev only (quirk Q1)
            self.conv: Tuple[str, ...] = ()
        else:
            self.name = "SD3"
            self.modules = model_io.sd3_linear_modules(cfg.depth_multimodal)
            self.route = model_io.sd3_linear_route
            self.skip = ()
            self.conv = ("x_embedder.proj",)                                  # the 2x2 patch conv
        self.flat = {m.replace(".", "_"): m for m in list(self.modules) + list(self.skip) + list(self.conv)}
        self.known = set(self.flat.values())

    def unknown(self, key: str, module: str) -> ValueError:
        flat = module.replace(".", "_")
        if re.match(r"(double_blocks|single_blocks)_\d+_|(img_in|txt_in|time_in|vector_in|guidance_in)(_|$)", flat):
            other = "FLUX"
        elif re.match(r"joint_blocks_\d+_|(x_embedder|t_embedder|y_embedder)(_|$)", flat):
            other = "SD3"
        else:
            other = None
        if other is not None and other != self.name:
            why = f"it is a {other} module and this is a {self.name} model"
        elif flat.startswith(("transformer_", "lora_transformer_")) or "transformer_blocks" in flat:
            why = "diffusers-named modules are not supported; name the targets like the upstream checkpoint"
        else:
            why = f"no {self.name} module of this model is named {module!r}"
        return ValueError(f"LoRA key {key!r}: {why}")


def _split_key(key: str, fam: _Family, skipped: set) -> Optional[Tuple[str, str]]:
    """one LoRA key -> (upstream module, "A" | "B" | "alpha"), or None for a recognised-but-skipped key"""
    if any(u in key for u in _UNSUPPORTED):
        raise ValueError(f"LoRA key {key!r}: LoHa / LoKr / DoRA tensors are not supported (plain LoRA only)")
    if key.endswith((".diff", ".diff_b")):
        raise ValueError(f"LoRA key {key!r}: full-difference tensors are not supported (plain LoRA only)")
    if key.startswith(("lora_te_", "lora_te1_", "lora_te2_", "lora_te3_")):
        skipped.add(key.split(".", 1)[0])                                     # kohya text-encoder module
        return None
    if key.startswith("text_encoder"):
        skipped.add(next((key[:-len(s)] for s in _SUFFIX_PEFT if key.endswith(s)), key))
        return None
    if key.startswith("lora_unet_"):
        stem, _, suffix = key[len("lora_unet_"):].partition(".")
        kind = _SUFFIX_KOHYA.get(suffix)
        if kind is None:
            raise ValueError(f"LoRA key {key!r}: expected .lora_down.weight, .lora_up.weight or .alpha")
        module = fam.flat.get(stem)
        if module is None:
            raise fam.unknown(key, stem)
        return module, kind
    k = key
    for pre in ("model.diffusion_model.", "diffusion_model."):
        if k.startswith(pre):
            k = k[len(pre):]
            break
    for suffix, kind in _SUFFIX_PEFT.items():
        if k.endswith(suffix):
            module = k[:-len(suffix)]
            if module not in fam.known:
                raise fam.unknown(key, module)
            return module, kind
    raise ValueError(f"LoRA key {key!r}: expected <module>.lora_A.weight, .lora_B.weight or .alpha "
                     "(or the kohya lora_unet_* spelling)")


def weight_shapes(cfg: MMDiTConfig) -> Dict[str, Tuple[int, int]]:
    """reference weight name -> (out, in) of every 2-D-viewable weight (the shapes of MMDiT.weight_views)"""
    from .weights import mmdit_param_specs

    out = {}
    for name, shape, kind in mmdit_param_specs(cfg):
        if kind == "w":
            k = 1
            for s in shape[1:]:
                k *= s
            out[name] = (shape[0], k)
    return out


def parse_lora(sd: Dict[str, Tensor], cfg: MMDiTConfig,
               shapes: Dict[str, Tuple[int, int]]) -> Tuple[Dict[str, LoraPair], Tuple[str, ...]]:
    """LoRA state dict -> ({upstream module: LoraPair}, skipped modules).  Raises ValueError naming the offending key
    for an unknown module, a missing half, mismatched ranks, a conv LoRA or a shape that does not match the model
    (`shapes`: reference weight name -> (out, in), see weight_shapes)."""
    fam = _Family(cfg)
    skipped: set = set()
    parts: Dict[str, Dict[str, Tuple[str, Tensor]]] = {}
    for key, t in sd.items():
        mk = _split_key(key, fam, skipped)
        if mk is None:
            continue
        module, kind = mk
        if module in fam.skip:
            skipped.add(module)
            continue
        if module in fam.conv:
            raise ValueError(f"LoRA key {key!r}: {module} is a convolution; conv LoRAs are not supported")
        slot = parts.setdefault(module, {})
        if kind in slot:
            raise ValueError(f"LoRA key {key!r}: {module}.{kind} is given twice (as {slot[kind][0]!r})")
        slot[kind] = (key, t)
    pairs: Dict[str, LoraPair] = {}
    for module, slot in parts.items():
        any_key = next(iter(slot.values()))[0]
        if "A" not in slot or "B" not in slot:
            raise ValueError(f"LoRA key {any_key!r}: module {module} has no "
                             f"{'down (lora_A)' if 'A' not in slot else 'up (lora_B)'} matrix")
        (ka, A), (kb, B) = slot["A"], slot["B"]
        if A.dim() != 2 or B.dim() != 2:
            bad = ka if A.dim() != 2 else kb
            raise ValueError(f"LoRA key {bad!r}: {tuple((A if bad == ka else B).shape)} is not a Linear LoRA matrix "
                             "(conv LoRAs are not supported)")
        r = A.shape[0]
        if B.shape[1] != r:
            raise ValueError(f"LoRA key {kb!r}: rank {B.shape[1]} does not match {ka!r}'s rank {r}")
        dim, route = fam.route(module)
        ws = [shapes[name + ".weight"] for name, _ in route]
        want = (sum(s[0] for s in ws), ws[0][1]) if dim == 0 else (ws[0][0], sum(s[1] for s in ws))
        if (B.shape[0], A.shape[1]) != want:
            raise ValueError(f"LoRA key {ka!r}: adapter is {B.shape[0]}x{A.shape[1]} (out x in), the model's {module} "
                             f"is {want[0]}x{want[1]}")
        alpha = float(slot["alpha"][1]) if "alpha" in slot else float(r)
        pairs[module] = LoraPair(A, B, alpha / r)
    return pairs, tuple(sorted(skipped))


def route_pairs(pairs: Dict[str, LoraPair], cfg: MMDiTConfig) -> Dict[str, LoraPair]:
    """{upstream module: pair} -> {reference weight name: pair} (slices of the upstream factors, model_io's splits)"""
    fam = _Family(cfg)
    out: Dict[str, LoraPair] = {}
    for module, p in pairs.items():
        for name, a, b in model_io.lora_to_params(fam.route(module), p.A, p.B, module):
            out[name] = LoraPair(a, b, p.alpha_over_rank)
    return out


def read_lora(lora) -> Tuple[Dict[str, Tensor], Optional[str]]:
    """a .safetensors path or a dict str -> tensor -> (state dict, default name or None)"""
    if isinstance(lora, dict):
        return lora, None
    if isinstance(lora, (str, bytes)) or hasattr(lora, "__fspath__"):
        path = os.fsdecode(lora)
        return model_io.load_safetensors(path), os.path.splitext(os.path.basename(path))[0]
    raise TypeError(f"lora must be a .safetensors path or a dict of tensors, got {type(lora).__name__}")


class _Adapter(NamedTuple):
    scale: float
    targets: Dict[str, LoraPair]          # reference weight name -> device fp32 factors


class LoraMerger:
    """Active adapters of one MMDiT and the pristine copies of the weights they touch.

    Pristine copies stay on the device (up to the whole 23.8 GB of FLUX's Linear weights for a LoRA that touches all of
    them); a weight no active adapter touches any more gets its copy back and the copy is freed, which restores it bit
    for bit.  Weights the model shares with the caller's `params` tensors (device tensors already in the model's dtype
    are packed without a copy) change with it.  `timing`: set to a dict to record per-stage milliseconds of the next
    calls (synchronising between stages; for measurement only)."""

    def __init__(self, mmdit):
        self.mmdit = mmdit
        self.cfg = mmdit.config
        self.views: Dict[str, Tensor] = mmdit.weight_views
        self.shapes = {n: (v.shape[0], v.shape[1]) for n, v in self.views.items()}
        self.adapters: Dict[str, _Adapter] = {}
        self.pristine: Dict[str, Tensor] = {}
        self._n_unnamed = 0
        self.timing: Optional[dict] = None

    def _mark(self, stage: str, t0: float) -> float:
        if self.timing is None:
            return t0
        torch.cuda.synchronize(self.mmdit.device)
        t1 = time.perf_counter()
        self.timing[stage] = self.timing.get(stage, 0.0) + 1e3 * (t1 - t0)
        return t1

    def load(self, lora, scale: float = 1.0, name: Optional[str] = None) -> LoraInfo:
        t0 = time.perf_counter()
        sd, stem = read_lora(lora)
        if name is None:
            if stem is None:
                stem = f"lora{self._n_unnamed}"
                self._n_unnamed += 1
            name = stem
        pairs, skipped = parse_lora(sd, self.cfg, self.shapes)
        t0 = self._mark("parse_ms", t0)
        dev = self.mmdit.device
        pairs = {m: LoraPair(p.A.to(dev, torch.float32), p.B.to(dev, torch.float32), p.alpha_over_rank)
                 for m, p in pairs.items()}
        targets = route_pairs(pairs, self.cfg)
        t0 = self._mark("h2d_ms", t0)
        old = self.adapters.get(name)
        self.adapters[name] = _Adapter(float(scale), targets)
        self._remerge(set(targets) | (set(old.targets) if old is not None else set()), t0)
        rank = max((p.A.shape[0] for p in pairs.values()), default=0)
        return LoraInfo(name, rank, len(targets), skipped)

    def unload(self, name: Optional[str] = None) -> None:
        names = list(self.adapters) if name is None else [name]
        if name is not None and name not in self.adapters:
            raise KeyError(f"no active LoRA named {name!r} (active: {sorted(self.adapters)})")
        touched = set()
        for n in names:
            touched |= set(self.adapters.pop(n).targets)
        self._remerge(touched, time.perf_counter())

    def _remerge(self, weights, t0: float) -> None:
        plan = []
        for w in sorted(weights):
            view = self.views[w]
            terms = [(a.scale * p.alpha_over_rank, p) for _, a in sorted(self.adapters.items())
                     if a.scale != 0.0 and (p := a.targets.get(w)) is not None]
            w0 = self.pristine.get(w)
            if not terms:
                if w0 is not None:                          # nothing active on it any more: restore and free
                    view.copy_(w0)
                    del self.pristine[w]
                continue
            if w0 is None:
                w0 = self.pristine[w] = view.clone(memory_format=torch.contiguous_format)
            plan.append((view, w0, terms))
        t0 = self._mark("pristine_ms", t0)
        dt = self.mmdit.dtype
        for view, w0, terms in plan:
            R = sum(p.A.shape[0] for _, p in terms)
            Rp = -(-R // 8) * 8
            a_op = torch.zeros((view.shape[0], Rp), dtype=torch.float32, device=view.device)
            w_op = torch.zeros((view.shape[1], Rp), dtype=torch.float32, device=view.device)
            col = 0
            for c, p in terms:
                r = p.A.shape[0]
                a_op[:, col:col + r] = p.B * c
                w_op[:, col:col + r] = p.A.t()
                col += r
            ops.gemm(a_op.to(dt), w_op.to(dt), out=view, res=w0)
        self._mark("merge_ms", t0)
        self.mmdit.invalidate_modulation_cache()
