"""Golden vectors from the REFERENCE'S OWN PyTorch modules (python/src/diffusionkit/torch/mmdit.py, vae.py), run in
plain PyTorch from a reference checkout ($DIFFUSIONKIT_REFERENCE) with the stand-ins of tests/golden/reference_shims.py for the four argmaxtools
building blocks they import.  Writes tests/golden/reference_torch_mmdit.npz and reference_torch_vae_decoder.npz.

The weights are not stored: they are the deterministic initialiser of diffusionkit_b200/weights.py (seeds below),
converted into the reference modules' state_dict layout here and loaded with strict=True.

Run from the repo root:
    DIFFUSIONKIT_REFERENCE=<argmaxinc/DiffusionKit checkout> python tests/golden/make_reference_golden.py
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
HERE = os.path.dirname(os.path.abspath(__file__))

from diffusionkit_b200.config import MMDiTConfig, VAEDecoderConfig  # noqa: E402
from diffusionkit_b200.weights import init_params, mmdit_param_specs, vae_decoder_param_specs  # noqa: E402
from tests.golden import reference_shims as rs  # noqa: E402

MMDIT_SEED, VAE_SEED = 17, 18


def pin_mmdit_config() -> MMDiTConfig:
    """SD3-shaped, 2 blocks: hidden = 64 * depth = 128, heads = depth = 2 (reference torch/mmdit.py:22-24, 227)"""
    return MMDiTConfig(num_heads=2, depth_multimodal=2, max_latent_resolution=24, pooled_text_embed_dim=64,
                       token_level_text_embed_dim=128, dtype=torch.float32, float16_dtype=torch.float32)


def pin_vae_config() -> VAEDecoderConfig:
    return VAEDecoderConfig(block_out_channels=(32, 64, 128, 128), layers_per_block=3)


def mmdit_params_to_reference_state_dict(params):
    """App. C names -> the reference torch module's state_dict (1x1 Conv2d weights, nn.Sequential indices, OIHW)"""
    sd = {}
    for k, v in params.items():
        k = k.replace(".mlp.layers.", ".mlp.").replace("adaLN_modulation.layers.", "adaLN_modulation.")
        if k == "x_embedder.proj.weight":
            v = v.permute(0, 3, 1, 2).contiguous()                       # OHWI -> OIHW
        elif k.endswith(".weight") and v.dim() == 2 and "pos_embed" not in k:
            v = v[:, :, None, None]                                      # nn.Linear -> 1x1 nn.Conv2d
        sd[k] = v
    return sd


def vae_params_to_reference_state_dict(params):
    sd = {}
    for k, v in params.items():
        leaf = k.rsplit(".", 1)[1]
        k = k.replace("conv_norm_out.", "norm_out.")
        k = k.replace("mid_blocks.0.", "mid.block_1.").replace("mid_blocks.2.", "mid.block_2.")
        if k.startswith("mid_blocks.1."):
            k = k.replace("mid_blocks.1.", "mid.attn_1.").replace("group_norm", "norm").replace("query_proj", "q_proj")
            k = k.replace("key_proj", "k_proj").replace("value_proj", "v_proj")
        k = k.replace("up_blocks.", "up.").replace(".resnets.", ".block.").replace(".conv_shortcut.", ".nin_shortcut.")
        k = k.replace(".upsample.", ".upsample.conv.")
        if leaf == "weight" and v.dim() == 4:
            v = v.permute(0, 3, 1, 2).contiguous()                       # OHWI -> OIHW
        elif leaf == "weight" and v.dim() == 2:
            v = v[:, :, None, None]                                      # Linear -> 1x1 conv
        sd[k] = v
    return sd


def run_reference_mmdit(latent_nhwc, text, pooled, timestep):
    m = rs.load_reference_module("mmdit")
    cfg = pin_mmdit_config()
    rcfg = m.MMDiTConfig(depth=cfg.depth_multimodal, max_latent_resolution=cfg.max_latent_resolution,
                         pooled_text_embed_dim=cfg.pooled_text_embed_dim,
                         token_level_text_embed_dim=cfg.token_level_text_embed_dim)
    net = m.MMDiT(rcfg).eval()
    params = init_params(mmdit_param_specs(cfg), seed=MMDIT_SEED, dtype=torch.float32)
    net.load_state_dict(mmdit_params_to_reference_state_dict(params), strict=True)
    B = latent_nhwc.shape[0]
    with torch.no_grad():
        (out,) = net(latent_nhwc.permute(0, 3, 1, 2).contiguous(),              # (B, 16, H, W)
                     text.permute(0, 2, 1)[:, :, None, :].contiguous(),          # (B, E, 1, T)
                     pooled[:, :, None, None], timestep.reshape(B))
    return out.permute(0, 2, 3, 1).contiguous()                                   # back to NHWC


def run_reference_vae(latent_nhwc):
    v = rs.load_reference_module("vae")
    cfg = pin_vae_config()
    boc = cfg.block_out_channels
    rcfg = v.VAEDecoderConfig(resolution=latent_nhwc.shape[1] * 8, base_channels=boc[0],
                              channel_multipliers=[c // boc[0] for c in boc], num_res_blocks=cfg.layers_per_block - 1)
    net = v.VAEDecoder(rcfg).eval()
    params = init_params(vae_decoder_param_specs(cfg), seed=VAE_SEED, dtype=torch.float32)
    net.load_state_dict(vae_params_to_reference_state_dict(params), strict=True)
    with torch.no_grad():
        out = net(latent_nhwc.permute(0, 3, 1, 2).contiguous())
    return out.permute(0, 2, 3, 1).contiguous()


def make_inputs():
    cfg = pin_mmdit_config()
    g = torch.Generator().manual_seed(23)
    latent = torch.randn((2, 12, 8, 16), generator=g)
    text = torch.randn((2, 20, cfg.token_level_text_embed_dim), generator=g)
    pooled = torch.randn((2, cfg.pooled_text_embed_dim), generator=g)
    timestep = torch.tensor([637.0, 637.0])
    z = torch.randn((1, 6, 4, 16), generator=g)
    return latent, text, pooled, timestep, z


if __name__ == "__main__":
    assert rs.reference_available(), "set DIFFUSIONKIT_REFERENCE to an argmaxinc/DiffusionKit checkout"
    latent, text, pooled, timestep, z = make_inputs()
    y = run_reference_mmdit(latent, text, pooled, timestep)
    np.savez_compressed(os.path.join(HERE, "reference_torch_mmdit.npz"), latent=latent.numpy(), text=text.numpy(),
                        pooled=pooled.numpy(), timestep=timestep.numpy(), out=y.numpy())
    img = run_reference_vae(z)
    np.savez_compressed(os.path.join(HERE, "reference_torch_vae_decoder.npz"), latent=z.numpy(), out=img.numpy())
    print("mmdit out", tuple(y.shape), float(y.abs().mean()), "| vae out", tuple(img.shape), float(img.abs().mean()))
