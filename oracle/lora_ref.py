"""ORACLE (test infrastructure — never imported by the product path).

LoRA merge in UPSTREAM key space, an extension: the reference has no LoRA support.  The product routes every adapter
onto the reference weights and merges into packed device windows; this restatement instead merges into the upstream
checkpoint tensors, in fp64 on the CPU,
    W_up += scale * (alpha / r) * B @ A          (alpha defaults to r)
and leaves the routing to the existing upstream -> reference converters (model_io.*_checkpoint_to_params), so comparing
the two checks the routing end to end.  Keys: PEFT `<module>.lora_A.weight` / `.lora_B.weight` / `.alpha` (optional
`diffusion_model.` / `model.diffusion_model.` prefix) or kohya `lora_unet_<module with . -> _>.lora_down.weight` /
`.lora_up.weight` / `.alpha`, resolved against the upstream tree's own module names.  Keys for modules the tree does
not have (text encoders, guidance_in on a checkpoint without it) are left out.
"""
from __future__ import annotations

from typing import Dict, Iterable, Tuple

import torch


def merge_upstream(sd_up: Dict[str, torch.Tensor], adapters: Iterable[Tuple[Dict[str, torch.Tensor], float]],
                   prefix: str = "") -> Dict[str, torch.Tensor]:
    """sd_up: upstream checkpoint tree whose keys are `prefix + module + .weight`; adapters: (LoRA state dict, scale)
    pairs -> a copy of sd_up with every adapted 2-D weight merged, in float64"""
    weights = {k[len(prefix):-len(".weight")]: k for k, v in sd_up.items()
               if k.startswith(prefix) and k.endswith(".weight") and v.dim() == 2}
    by_flat = {m.replace(".", "_"): m for m in weights}
    out = dict(sd_up)
    for lora, scale in adapters:
        factors: Dict[str, Dict[str, torch.Tensor]] = {}
        for key, t in lora.items():
            if key.startswith("lora_unet_"):
                stem, _, suffix = key[len("lora_unet_"):].partition(".")
                module = by_flat.get(stem)
                part = {"lora_down.weight": "down", "lora_up.weight": "up", "alpha": "alpha"}.get(suffix)
            else:
                k = key
                for pre in ("model.diffusion_model.", "diffusion_model."):
                    if k.startswith(pre):
                        k = k[len(pre):]
                        break
                module, part = None, None
                for suffix, name in ((".lora_A.weight", "down"), (".lora_B.weight", "up"), (".alpha", "alpha")):
                    if k.endswith(suffix) and k[:-len(suffix)] in weights:
                        module, part = k[:-len(suffix)], name
            if module is not None and part is not None:
                factors.setdefault(module, {})[part] = t
        for module, f in factors.items():
            down, up = f["down"].double(), f["up"].double()
            r = down.shape[0]
            alpha = float(f["alpha"]) if "alpha" in f else float(r)
            key = weights[module]
            out[key] = out[key].double() + scale * (alpha / r) * (up @ down)
    return out
