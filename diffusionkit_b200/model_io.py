"""Checkpoint key remapping: upstream (BFL FLUX / Stability SD3 / LDM VAE) safetensors layouts -> the parameter tree
this engine consumes (the reference's module-tree names, SURVEY.md App. C).

Restates the rules of the reference loaders (python/src/diffusionkit/mlx/model_io.py):
  flux_state_dict_adjustments        :130-311
  mmdit_state_dict_adjustments       :314-408
  vae_decoder_state_dict_adjustments :411-486, vae_encoder_state_dict_adjustments :489-571
as table-driven converters over torch tensors.  SURVEY.md §8 "next" row f1.  Downloading (huggingface_hub) is out of
scope — callers pass a local .safetensors path (the reference's `local_ckpt`).
"""
from __future__ import annotations

import re
from typing import Callable, Dict, Iterable, List, Optional, Tuple

import torch

Tensor = torch.Tensor


def load_safetensors(path: str) -> Dict[str, Tensor]:
    from safetensors.torch import load_file

    return load_file(path)


def _conv_oihw_to_ohwi(w: Tensor) -> Tensor:
    """PyTorch conv weight (O, I, kh, kw) -> mlx nn.Conv2d weight (O, kh, kw, I)"""
    return w.permute(0, 2, 3, 1).contiguous()


# ------------------------------------------------------------------------------------------------ Linear routing
# An upstream Linear module -> the reference Linear modules its weight is split into:
#   (split dim, ((reference module, width in units), ...))
# dim 0 splits the weight's rows (output features), dim 1 its columns (input features); the widths are in units of
# size / sum(units).  One table serves both the checkpoint converters below and the LoRA converter (lora_to_params), so
# a split rule cannot differ between a base weight and an adapter on it.
Route = Tuple[int, Tuple[Tuple[str, int], ...]]

_FLUX_STREAM = {"img": "image_transformer_block", "txt": "text_transformer_block"}
_FLUX_FIXED = {
    "img_in": "x_embedder.proj", "txt_in": "context_embedder",
    "time_in.in_layer": "t_embedder.mlp.layers.0", "time_in.out_layer": "t_embedder.mlp.layers.2",
    "vector_in.in_layer": "y_embedder.mlp.layers.0", "vector_in.out_layer": "y_embedder.mlp.layers.2",
    "final_layer.linear": "final_layer.linear", "final_layer.adaLN_modulation.1": "final_layer.adaLN_modulation.layers.1",
}
_SD3_FIXED = {
    "context_embedder": "context_embedder", "final_layer.linear": "final_layer.linear",
    "final_layer.adaLN_modulation.1": "final_layer.adaLN_modulation.layers.1",
    "t_embedder.mlp.0": "t_embedder.mlp.layers.0", "t_embedder.mlp.2": "t_embedder.mlp.layers.2",
    "y_embedder.mlp.0": "y_embedder.mlp.layers.0", "y_embedder.mlp.2": "y_embedder.mlp.layers.2",
}
_BLOCK_PARTS = {"qkv": ("attn.q_proj", "attn.k_proj", "attn.v_proj"), "proj": ("attn.o_proj",),
                "fc1": ("mlp.fc1",), "fc2": ("mlp.fc2",), "mod": ("adaLN_modulation.layers.1",)}


def _block_route(base: str, part: str) -> Route:
    return 0, tuple((f"{base}.{n}", 1) for n in _BLOCK_PARTS[part])


def flux_linear_route(module: str, mlp_ratio: int = 4) -> Optional[Route]:
    """BFL FLUX Linear module name (no `.weight`) -> Route, or None if `module` is not one of the model's Linears.
      double_blocks.i.{img,txt}_attn.qkv -> rows [h, h, h] of {q,k,v}_proj;  _attn.proj / _mlp.{0,2} / _mod.lin -> 1:1
      single_blocks.i.linear1 -> rows [h, h, h, r*h] of {q,k,v}_proj, mlp.fc1
      single_blocks.i.linear2 -> cols [h, r*h] of o_proj, mlp.fc2;  single_blocks.i.modulation.lin -> 1:1
      img_in / txt_in / time_in / vector_in / final_layer.* -> embedders / final layer"""
    m = re.fullmatch(r"double_blocks\.(\d+)\.(img|txt)_(attn\.qkv|attn\.proj|mlp\.0|mlp\.2|mod\.lin)", module)
    if m:
        i, stream, part = m.groups()
        part = {"attn.qkv": "qkv", "attn.proj": "proj", "mlp.0": "fc1", "mlp.2": "fc2", "mod.lin": "mod"}[part]
        return _block_route(f"multimodal_transformer_blocks.{i}.{_FLUX_STREAM[stream]}", part)
    m = re.fullmatch(r"single_blocks\.(\d+)\.(linear1|linear2|modulation\.lin)", module)
    if m:
        i, part = m.groups()
        base = f"unified_transformer_blocks.{i}.transformer_block"
        if part == "linear1":
            return 0, tuple((f"{base}.{n}", w) for n, w in
                            (("attn.q_proj", 1), ("attn.k_proj", 1), ("attn.v_proj", 1), ("mlp.fc1", mlp_ratio)))
        if part == "linear2":
            return 1, ((f"{base}.attn.o_proj", 1), (f"{base}.mlp.fc2", mlp_ratio))
        return _block_route(base, "mod")
    if module in _FLUX_FIXED:
        return 0, ((_FLUX_FIXED[module], 1),)
    return None


def sd3_linear_route(module: str) -> Optional[Route]:
    """Stability SD3 / SD3.5 Linear module name (no `model.diffusion_model.` prefix, no `.weight`) -> Route or None.
      joint_blocks.i.{x_block,context_block}.attn.qkv -> rows [h, h, h] of {q,k,v}_proj;  attn.proj, mlp.fc1,
      mlp.fc2, adaLN_modulation.1 -> 1:1;  context_embedder, {t,y}_embedder.mlp.{0,2}, final_layer.* -> 1:1.
    x_embedder.proj is a 2x2 conv, not a Linear."""
    m = re.fullmatch(r"joint_blocks\.(\d+)\.(context_block|x_block)\.(attn\.qkv|attn\.proj|mlp\.fc1|mlp\.fc2|"
                     r"adaLN_modulation\.1)", module)
    if m:
        i, blk, part = m.groups()
        stream = "text_transformer_block" if blk == "context_block" else "image_transformer_block"
        part = {"attn.qkv": "qkv", "attn.proj": "proj", "mlp.fc1": "fc1", "mlp.fc2": "fc2",
                "adaLN_modulation.1": "mod"}[part]
        return _block_route(f"multimodal_transformer_blocks.{i}.{stream}", part)
    if module in _SD3_FIXED:
        return 0, ((_SD3_FIXED[module], 1),)
    return None


def flux_linear_modules(depth_multimodal: int, depth_unified: int) -> List[str]:
    """every upstream Linear module of a FLUX model with these depths (the names flux_linear_route accepts)"""
    mods = list(_FLUX_FIXED)
    for i in range(depth_multimodal):
        for s in _FLUX_STREAM:
            mods += [f"double_blocks.{i}.{s}_{p}" for p in ("attn.qkv", "attn.proj", "mlp.0", "mlp.2", "mod.lin")]
    for i in range(depth_unified):
        mods += [f"single_blocks.{i}.{p}" for p in ("linear1", "linear2", "modulation.lin")]
    return mods


def sd3_linear_modules(depth_multimodal: int) -> List[str]:
    """every upstream Linear module of an SD3 / SD3.5 model with this depth; the last context block stops after its
    qkv projection (reference mmdit.py:62-66), so it has no attn.proj / mlp"""
    mods = list(_SD3_FIXED)
    for i in range(depth_multimodal):
        for blk in ("x_block", "context_block"):
            last_ctx = blk == "context_block" and i == depth_multimodal - 1
            parts = ("attn.qkv", "adaLN_modulation.1") if last_ctx else (
                "attn.qkv", "attn.proj", "mlp.fc1", "mlp.fc2", "adaLN_modulation.1")
            mods += [f"joint_blocks.{i}.{blk}.{p}" for p in parts]
    return mods


def _split_sizes(n: int, parts, what: str) -> List[int]:
    units = sum(w for _, w in parts)
    if n % units:
        raise ValueError(f"{what}: size {n} does not split into {[name for name, _ in parts]} ({units} equal units)")
    return [n // units * w for _, w in parts]


def _convert_linear(route: Route, leaf: str, v: Tensor, out: Dict[str, Tensor], what: str) -> None:
    """one upstream Linear tensor (`leaf` = weight / bias) -> its reference tensors in `out`"""
    dim, parts = route
    if len(parts) == 1:
        out[f"{parts[0][0]}.{leaf}"] = v
        return
    if leaf == "bias" and dim == 1:
        chunks = [v] * len(parts)            # a column split keeps ONE bias: the reference gives it to every part
    else:
        chunks = [c.contiguous() for c in torch.split(v, _split_sizes(v.shape[dim], parts, what), dim=dim)]
    for (name, _), c in zip(parts, chunks):
        if leaf == "bias" and name.endswith(".attn.k_proj"):
            continue                         # no K-projection bias (quirk Q3)
        out[f"{name}.{leaf}"] = c


def lora_to_params(route: Route, A: Tensor, B: Tensor, what: str = "lora") -> List[Tuple[str, Tensor, Tensor]]:
    """a LoRA pair on one upstream Linear (A = down [r, in], B = up [out, r]; delta = B @ A) -> one
    (reference weight name, A, B) per reference weight: a row split slices B by rows, a column split slices A by
    columns, with the same widths the checkpoint converters use for the base weight"""
    dim, parts = route
    if len(parts) == 1:
        return [(parts[0][0] + ".weight", A, B)]
    if dim == 0:
        return [(name + ".weight", A, b) for (name, _), b in
                zip(parts, torch.split(B, _split_sizes(B.shape[0], parts, what), dim=0))]
    return [(name + ".weight", a, B) for (name, _), a in
            zip(parts, torch.split(A, _split_sizes(A.shape[1], parts, what), dim=1))]


# ------------------------------------------------------------------------------------------------ FLUX (BFL layout)


def flux_checkpoint_to_params(sd: Dict[str, Tensor], hidden_size: int = 3072, mlp_ratio: int = 4) -> Dict[str, Tensor]:
    """BFL `flux1-*.safetensors` -> MMDiT parameter tree (reference model_io.py:130-311).

    double_blocks.i.{img,txt}_attn.qkv        -> split 3 (rows)  -> ...{image,text}_transformer_block.attn.{q,k,v}_proj
    double_blocks.i.{img,txt}_attn.proj       -> ...attn.o_proj
    double_blocks.i.{img,txt}_attn.norm.*     -> ...qk_norm.{q,k}_norm.weight
    double_blocks.i.{img,txt}_mlp.{0,2}       -> ...mlp.{fc1,fc2}
    double_blocks.i.{img,txt}_mod.lin         -> ...adaLN_modulation.layers.1
    single_blocks.i.linear1                   -> split rows [h, h, h, r*h] -> attn.{q,k,v}_proj, mlp.fc1
    single_blocks.i.linear2.weight            -> split cols [h, r*h]       -> attn.o_proj.weight, mlp.fc2.weight
    single_blocks.i.linear2.bias              -> attn.o_proj.bias (and mlp.fc2.bias, which the forward zeroes, mmdit.py:742)
    img_in / txt_in / time_in / vector_in / final_layer.adaLN_modulation.1 -> embedders / final layer
    The K-projection bias is dropped (quirk Q3) and guidance_in.* is ignored (quirk Q1).  The Linear splits come from
    flux_linear_route; `hidden_size` is implied by the tensor sizes and kept for existing callers.
    """
    out: Dict[str, Tensor] = {}
    for key, v in sd.items():
        module, _, leaf = key.rpartition(".")
        route = flux_linear_route(module, mlp_ratio) if leaf in ("weight", "bias") else None
        if route is not None:
            if module == "img_in" and leaf == "weight":
                v = v.reshape(v.shape[0], 1, 1, v.shape[1]).contiguous()    # patchify-as-reshape conv weight
            _convert_linear(route, leaf, v, out, key)
            continue
        m = re.fullmatch(r"(double_blocks\.(\d+)\.(img|txt)_attn|single_blocks\.(\d+))\.norm\.(query|key)_norm\.scale", key)
        if m:
            _, i, stream, j, qk = m.groups()
            base = (f"multimodal_transformer_blocks.{i}.{_FLUX_STREAM[stream]}" if i is not None
                    else f"unified_transformer_blocks.{j}.transformer_block")
            out[f"{base}.qk_norm.{qk[0]}_norm.weight"] = v
        elif key.startswith("guidance_in."):
            continue  # quirk Q1: the reference ignores the guidance embedder (model_io.py:756,783)
        else:
            raise KeyError(f"unrecognised FLUX key {key}")
    return out


# ------------------------------------------------------------------------------------------------ SD3 (SAI layout)
def sd3_checkpoint_to_params(sd: Dict[str, Tensor], prefix: str = "model.diffusion_model.") -> Dict[str, Tensor]:
    """Stability `sd3_medium.safetensors` -> MMDiT parameter tree (reference model_io.py:314-408).
    VAE (`first_stage_model.` / `decoder.` / `encoder.`) and `teacher_model.` tensors are skipped here."""
    out: Dict[str, Tensor] = {}
    for key, v in sd.items():
        if "decoder." in key or "encoder." in key or "teacher_model." in key:
            continue
        if key.startswith(prefix):
            key = key[len(prefix):]
        module, _, leaf = key.rpartition(".")
        route = sd3_linear_route(module) if leaf in ("weight", "bias") else None
        if route is not None:
            _convert_linear(route, leaf, v, out, key)          # qkv: the k bias is dropped (model_io.py:389-390)
            continue
        m = re.fullmatch(r"joint_blocks\.(\d+)\.(context_block|x_block)\.(.+)", key)
        if m:
            i, blk, rest = m.groups()
            stream = "text_transformer_block" if blk == "context_block" else "image_transformer_block"
            base = f"multimodal_transformer_blocks.{i}.{stream}"
            if rest.startswith("attn.ln_q."):
                out[f"{base}.qk_norm.q_norm.{rest[10:]}"] = v
            elif rest.startswith("attn.ln_k."):
                out[f"{base}.qk_norm.k_norm.{rest[10:]}"] = v
            elif rest.startswith("adaLN_modulation."):
                out[f"{base}.adaLN_modulation.layers.{rest[17:]}"] = v
            else:                                    # any other block tensor keeps its name
                out[f"{base}.{rest}"] = v
            continue
        if key == "pos_embed":
            out["x_pos_embedder.pos_embed.weight"] = v[0].contiguous()       # (1, N, h) buffer -> (N, h) table
        elif key == "x_embedder.proj.weight":
            out[key] = _conv_oihw_to_ohwi(v)
        elif key.startswith(("y_embedder.mlp.", "t_embedder.mlp.")):
            emb, _, idx, leaf = key.split(".")
            out[f"{emb}.mlp.layers.{idx}.{leaf}"] = v
        elif key.startswith("final_layer.adaLN_modulation."):
            out["final_layer.adaLN_modulation.layers." + key[len("final_layer.adaLN_modulation."):]] = v
        elif key.startswith(("x_embedder.", "context_embedder.", "final_layer.linear.")):
            out[key] = v
        else:
            raise KeyError(f"unrecognised SD3 key {key}")
    return out


# ------------------------------------------------------------------------------------------------ VAE (LDM layout)
def _vae_checkpoint_to_params(sd: Dict[str, Tensor], prefix: str, side: str) -> Dict[str, Tensor]:
    """LDM autoencoder `<prefix>*` -> VAEDecoder / VAEEncoder parameter tree.  side = "up" (decoder: up.N.block.M,
    up.N.upsample.conv) or "down" (encoder: down.N.block.M, down.N.downsample.conv)."""
    blocks, sample = f"{side}_blocks", f"{side}sample"
    out: Dict[str, Tensor] = {}
    for key, v in sd.items():
        pos = key.find(prefix)
        if pos < 0 or "diffusion_model." in key:
            continue
        k = key[pos + len(prefix):]
        leaf = k.rsplit(".", 1)[1]
        m = re.fullmatch(side + r"\.(\d+)\.block\.(\d+)\.(norm1|conv1|norm2|conv2|nin_shortcut)\.(weight|bias)", k)
        if m:
            j, l, mod, _ = m.groups()
            if mod == "nin_shortcut":
                name, val = f"{blocks}.{j}.resnets.{l}.conv_shortcut.{leaf}", (v[:, :, 0, 0].contiguous() if leaf == "weight" else v)
            elif mod.startswith("conv"):
                name, val = f"{blocks}.{j}.resnets.{l}.{mod}.{leaf}", (_conv_oihw_to_ohwi(v) if leaf == "weight" else v)
            else:
                name, val = f"{blocks}.{j}.resnets.{l}.{mod}.{leaf}", v
            out[name] = val
            continue
        m = re.fullmatch(side + r"\.(\d+)\." + sample + r"\.conv\.(weight|bias)", k)
        if m:
            out[f"{blocks}.{m.group(1)}.{sample}.{leaf}"] = _conv_oihw_to_ohwi(v) if leaf == "weight" else v
            continue
        m = re.fullmatch(r"mid\.block_(1|2)\.(norm1|conv1|norm2|conv2)\.(weight|bias)", k)
        if m:
            idx = 0 if m.group(1) == "1" else 2
            mod = m.group(2)
            out[f"mid_blocks.{idx}.{mod}.{leaf}"] = _conv_oihw_to_ohwi(v) if (mod.startswith("conv") and leaf == "weight") else v
            continue
        m = re.fullmatch(r"mid\.attn_1\.(norm|q|k|v|proj_out)\.(weight|bias)", k)
        if m:
            mod = {"norm": "group_norm", "q": "query_proj", "k": "key_proj", "v": "value_proj",
                   "proj_out": "out_proj"}[m.group(1)]
            val = v[:, :, 0, 0].contiguous() if (leaf == "weight" and v.dim() == 4) else v
            out[f"mid_blocks.1.{mod}.{leaf}"] = val
            continue
        if k.startswith(("conv_in.", "conv_out.")):
            out[k] = _conv_oihw_to_ohwi(v) if leaf == "weight" else v
        elif k.startswith("norm_out."):
            out["conv_norm_out." + leaf] = v
        else:
            raise KeyError(f"unrecognised VAE {'decoder' if side == 'up' else 'encoder'} key {key}")
    return out


def vae_decoder_checkpoint_to_params(sd: Dict[str, Tensor], prefix: str = "decoder.") -> Dict[str, Tensor]:
    """LDM autoencoder `decoder.*` -> VAEDecoder parameter tree (reference model_io.py:411-486).
    `prefix` may sit behind another prefix (e.g. `first_stage_model.decoder.`): everything up to and including the first
    occurrence of `prefix` is stripped."""
    return _vae_checkpoint_to_params(sd, prefix, "up")


def vae_encoder_checkpoint_to_params(sd: Dict[str, Tensor], prefix: str = "encoder.") -> Dict[str, Tensor]:
    """LDM autoencoder `encoder.*` -> VAEEncoder parameter tree (reference model_io.py:489-571)."""
    return _vae_checkpoint_to_params(sd, prefix, "down")


# ------------------------------------------------------------------------------------------------ text encoders
def clip_checkpoint_to_params(sd: Dict[str, Tensor]) -> Dict[str, Tensor]:
    """HF CLIPTextModel(WithProjection) safetensors -> CLIPTextModel parameter tree
    (reference map_clip_text_encoder_weights, model_io.py:611-636)."""
    out: Dict[str, Tensor] = {}
    for key, v in sd.items():
        k = key
        for pre in ("text_model.", "embeddings.", "encoder."):
            if k.startswith(pre):
                k = k[len(pre):]
        if k == "position_ids":
            continue                                      # a buffer older checkpoints carry; not a parameter
        k = k.replace("self_attn.", "attention.")
        k = k.replace("q_proj.", "query_proj.").replace("k_proj.", "key_proj.").replace("v_proj.", "value_proj.")
        k = k.replace("mlp.fc1", "linear1").replace("mlp.fc2", "linear2")
        out[k] = v
    return out


def t5_checkpoint_to_params(sd: Dict[str, Tensor], prefix: str = "") -> Dict[str, Tensor]:
    """HF T5EncoderModel (t5xxl.safetensors) -> SD3T5Encoder parameter tree
    (reference t5_encoder_state_dict_adjustments, model_io.py:565-608)."""
    out: Dict[str, Tensor] = {}
    attn = {"q": "query_proj", "k": "key_proj", "v": "value_proj", "o": "out_proj"}
    for key, v in sd.items():
        k = key[len(prefix):] if prefix and key.startswith(prefix) else key
        if k in ("shared.weight",):
            continue                                      # same tensor as encoder.embed_tokens.weight (:601-603)
        if k == "encoder.embed_tokens.weight":
            out["wte.weight"] = v
        elif k == "encoder.final_layer_norm.weight":
            out["encoder.ln.weight"] = v
        elif k == "encoder.block.0.layer.0.SelfAttention.relative_attention_bias.weight":
            out["encoder.relative_attention_bias.embeddings.weight"] = v
        else:
            m = re.fullmatch(r"encoder\.block\.(\d+)\.layer\.(0|1)\.(.+)", k)
            if not m:
                raise KeyError(f"unrecognised T5 key {key}")
            i, sub, rest = m.groups()
            base = f"encoder.layers.{i}."
            if rest == "layer_norm.weight":
                out[base + f"ln{int(sub) + 1}.weight"] = v
            elif rest.startswith("SelfAttention."):
                out[base + f"attention.{attn[rest.split('.')[1]]}.weight"] = v
            elif rest.startswith("DenseReluDense."):
                out[base + "dense." + rest[len("DenseReluDense."):]] = v
            else:
                raise KeyError(f"unrecognised T5 key {key}")
    if "wte.weight" not in out and "shared.weight" in sd:
        out["wte.weight"] = sd["shared.weight"]
    return out


# ------------------------------------------------------------------------------------------------ 4-bit variants
def is_q4_checkpoint(sd: Dict[str, Tensor]) -> bool:
    return any(k.endswith(".scales") for k in sd)


def preadjusted_checkpoint_to_params(sd: Dict[str, Tensor], prefix: str = "") -> Dict[str, Tensor]:
    """The `*-4bit-quantized` checkpoints were saved from the reference's own module tree, so their keys already are
    the App. C names (behind `prefix` for the single-file SD3.5 checkpoint): keep the keys that contain the prefix and
    strip it (reference model_io.py:733-734, 772-775 "4-bit ckpt already adjusted")."""
    if not prefix:
        return dict(sd)
    return {k.replace(prefix, ""): v for k, v in sd.items() if prefix in k}


def dequantize_q4_params(sd: Dict[str, Tensor], device, dtype: torch.dtype, group_size: int = 64) -> Dict[str, Tensor]:
    """MLX QuantizedLinear triples (`X.weight` uint32 [N, K/8], `X.scales`, `X.biases` [N, K/64]) -> dense 16-bit
    `X.weight` [N, K] on `device` (dk_dequant_q4).  On B200 the denoise GEMMs are tensor-pipe bound at M >= 1024 rows
    and the dense FLUX weights are 13 % of HBM, so the 4-bit form is expanded once at load instead of inside every GEMM
    (DESIGN.md §7).  Every other tensor is passed through (cast to `dtype` like the reference, :736-738)."""
    from . import ops

    out: Dict[str, Tensor] = {}
    for k, v in sd.items():
        if k.endswith((".scales", ".biases")) and (k.rsplit(".", 1)[0] + ".weight") in sd:
            continue
        base = k[:-7] if k.endswith(".weight") else None
        if base is not None and (base + ".scales") in sd:
            if v.dtype not in (torch.uint32, torch.int32):
                raise ValueError(f"{k}: quantised weight must be uint32, got {v.dtype}")
            wq = v.contiguous().view(torch.int32).to(device)
            sc = sd[base + ".scales"].to(device=device, dtype=dtype).contiguous()
            bi = sd[base + ".biases"].to(device=device, dtype=dtype).contiguous()
            out[k] = ops.dequant_q4(wq, sc, bi, group_size)
        else:
            out[k] = v.to(device=device, dtype=dtype) if v.is_floating_point() else v.to(device)
    return out


def check_against_specs(params: Dict[str, Tensor], specs: Iterable[Tuple[str, Tuple[int, ...], str]],
                        allow_extra: Iterable[str] = ()) -> None:
    """Raise if the converted tree does not match the engine's parameter specs (names and shapes)."""
    want = {n: tuple(s) for n, s, _ in specs}
    missing = sorted(set(want) - set(params))
    extra = sorted(k for k in set(params) - set(want) if not any(k.endswith(a) for a in allow_extra))
    bad = sorted(n for n in want if n in params and tuple(params[n].shape) != want[n])
    if missing or extra or bad:
        raise ValueError(f"checkpoint does not match the model: missing {missing[:5]} (+{max(0, len(missing) - 5)}), "
                         f"unexpected {extra[:5]} (+{max(0, len(extra) - 5)}), wrong shape {bad[:5]}")
