"""ORACLE (test infrastructure — never imported by the product path).

Latent-blend inpainting (masked img2img), an extension: the reference has no inpainting.  It composes with the
reference's img2img flow (mlx/__init__.py:270-285, 586-594; sampler.py:41-42), restated in sampler_ref / vae_ref:
  * inpaint_masks: the mask rules, in numpy without PIL
  * inpaint_blend: the select that puts the kept latent cells back on the input image's noised trajectory
  * sample_euler_inpaint: sampler_ref.sample_euler with inpaint_blend after every Euler step
"""
from __future__ import annotations

from typing import Callable, Optional, Tuple

import numpy as np
import torch

from . import sampler_ref as sr


def inpaint_masks(mask_u8: np.ndarray, size_hw: Tuple[int, int]) -> Tuple[np.ndarray, np.ndarray]:
    """mask_u8: uint8 (H0, W0), (H0, W0, 1), RGB or RGBA at the original size of its image; size_hw: read_image's
    target size (H0, W0 cut down to multiples of 64).
      greyscale  L = (19595 R + 38470 G + 7471 B + 2^15) >> 16   (ITU-R 601-2 luma in PIL's integer form; alpha ignored)
      NEAREST    out[i] = in[floor(u_i)], u_0 = (H0 / H) / 2, u_{i+1} = u_i + H0 / H   (per axis, float64, as PIL)
      pixel mask p = L >= 128 (white = regenerate); latent mask m[y, x] = any(p[8y:8y+8, 8x:8x+8])
    -> (p (H, W), m (H/8, W/8)), uint8 in {0, 1}"""
    a = np.asarray(mask_u8)
    if a.ndim == 3 and a.shape[2] == 1:
        a = a[:, :, 0]
    if a.ndim == 3:
        rgb = a[:, :, :3].astype(np.int64)
        a = ((19595 * rgb[..., 0] + 38470 * rgb[..., 1] + 7471 * rgb[..., 2] + 32768) >> 16).astype(np.uint8)
    H, W = size_hw

    def nearest(n_in, n_out):
        step = n_in / n_out
        idx, u = [], step / 2
        for _ in range(n_out):
            idx.append(int(u))
            u += step
        return np.asarray(idx)

    if a.shape != (H, W):
        a = a[nearest(a.shape[0], H)][:, nearest(a.shape[1], W)]
    p = (a >= 128).astype(np.uint8)
    m = np.zeros((H // 8, W // 8), dtype=np.uint8)
    for y in range(H // 8):
        for x in range(W // 8):
            m[y, x] = p[8 * y:8 * y + 8, 8 * x:8 * x + 8].any()
    return p, m


def inpaint_blend(x: torch.Tensor, x0: torch.Tensor, noise: torch.Tensor, mask: torch.Tensor,
                  sigma_next: float) -> torch.Tensor:
    """After the Euler step to sigma_next, the kept cells are set to noise_scaling(sigma_next, noise, x0)
    (sampler.py:41-42); the cells being regenerated keep the sampler's x.  A select, not a blend of the two.
    x, x0, noise: (B, H, W, C) fp32 with x0 = process_in(encoded image); mask: (B, H, W), non-zero = regenerate."""
    kept = sigma_next * noise + (1.0 - sigma_next) * x0
    return torch.where(mask.bool()[..., None], x, kept)


def sample_euler_inpaint(
    mmdit_call: Callable[[torch.Tensor, torch.Tensor, torch.Tensor], torch.Tensor],
    cache_modulation: Callable[[torch.Tensor, torch.Tensor], None],
    x: torch.Tensor,
    sigmas: torch.Tensor,
    conditioning: torch.Tensor,
    pooled: torch.Tensor,
    cfg_weight: float,
    act_dtype: Optional[torch.dtype],
    x0: torch.Tensor,
    noise: torch.Tensor,
    mask: torch.Tensor,
) -> torch.Tensor:
    """sampler_ref.sample_euler (same arguments) with inpaint_blend(x, x0, noise, mask, sigma_next) after every step,
    the last one included.  Each step is one call of sample_euler over (sigma_i, sigma_i+1): the modulation table is
    computed per timestep value, so this is the same arithmetic as the whole loop, step for step."""
    for i in range(len(sigmas) - 1):
        x = sr.sample_euler(mmdit_call, cache_modulation, x, sigmas[i:i + 2], conditioning, pooled, cfg_weight,
                            act_dtype)
        x = inpaint_blend(x, x0, noise, mask, float(sigmas[i + 1]))
    return x
