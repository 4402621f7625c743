"""Golden vectors from the reference's MLX SOURCE files (python/src/diffusionkit/mlx/mmdit.py, config.py, sampler.py,
vae.py), imported from a reference checkout ($DIFFUSIONKIT_REFERENCE) and executed on tests/golden/mlx_standin.py — a torch-backed stand-in for the MLX
primitives they call (MLX itself runs on Apple silicon only).  This pins the oracle's wiring of the FLUX path (single-
stream blocks, RoPE, QK-RMSNorm, reshape-patchify, [text | image] order, modulation cache) and of the SD3 path against
the reference's own code; the fixtures are fp32.

Writes tests/golden/reference_mlxsrc_{flux,sd3}_mmdit.npz, reference_mlxsrc_vae.npz, reference_mlxsrc_sampler.json.
Run from the repo root:
    DIFFUSIONKIT_REFERENCE=<argmaxinc/DiffusionKit checkout> python tests/golden/make_reference_mlx_golden.py
"""
import importlib
import json
import os
import sys
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
HERE = os.path.dirname(os.path.abspath(__file__))

from diffusionkit_b200.config import (PositionalEncoding, VAEDecoderConfig, VAEEncoderConfig,  # noqa: E402
                                      tiny_flux_config, tiny_sd3_config)
from diffusionkit_b200.weights import (init_params, mmdit_param_specs, vae_decoder_param_specs,  # noqa: E402
                                       vae_encoder_param_specs)
from tests.golden import mlx_standin, reference_shims  # noqa: E402

REF_MLX_DIR = os.path.join(reference_shims.REFERENCE_SRC, "diffusionkit", "mlx")

SEEDS = {"flux": 41, "sd3": 42, "vae_dec": 43, "vae_enc": 44, "sd35": 45}


def reference_mlx_available() -> bool:
    return reference_shims.reference_available() and os.path.exists(os.path.join(REF_MLX_DIR, "mmdit.py"))


def load_reference_mlx(name: str):
    """import <reference>/python/src/diffusionkit/mlx/<name>.py as `_refmlx.<name>` without running the package's __init__ (which pulls
    in tokenizers, PIL pipelines and Hugging Face downloads)"""
    mlx_standin.install()
    reference_shims.install()            # argmaxtools.utils.get_logger
    if "_refmlx" not in sys.modules:
        pkg = types.ModuleType("_refmlx")
        pkg.__path__ = [REF_MLX_DIR]
        sys.modules["_refmlx"] = pkg
    return importlib.import_module(f"_refmlx.{name}")


def pin_configs():
    flux = tiny_flux_config(hidden=256, heads=2, depth_mm=2, depth_uni=2)
    sd3 = tiny_sd3_config(hidden=128, heads=2, depth_mm=3)
    from dataclasses import replace

    # fp32 everywhere: the fixture pins wiring, not 16-bit rounding
    return (replace(flux, dtype=torch.float32, float16_dtype=torch.float32),
            replace(sd3, dtype=torch.float32, float16_dtype=torch.float32))


def pin_config(kind):
    """kind in flux / sd3 / sd35 (SD3.5 shape: learned positional embedding + QK-RMSNorm, row f4)"""
    from dataclasses import replace

    from diffusionkit_b200.config import tiny_sd35_config

    if kind == "sd35":
        return replace(tiny_sd35_config(), dtype=torch.float32, float16_dtype=torch.float32)
    flux, sd3 = pin_configs()
    return flux if kind == "flux" else sd3


def reference_config(rcfg_mod, cfg):
    mx = sys.modules["mlx.core"]
    return rcfg_mod.MMDiTConfig(
        num_heads=cfg.num_heads, depth_multimodal=cfg.depth_multimodal, depth_unified=cfg.depth_unified,
        parallel_mlp_for_unified_blocks=cfg.parallel_mlp_for_unified_blocks, mlp_ratio=cfg.mlp_ratio,
        vae_latent_dim=cfg.vae_latent_dim, layer_norm_eps=cfg.layer_norm_eps,
        pos_embed_type=(rcfg_mod.PositionalEncoding.PreSDPARope if cfg.pos_embed_type == PositionalEncoding.PreSDPARope
                        else rcfg_mod.PositionalEncoding.LearnedInputEmbedding),
        rope_axes_dim=cfg.rope_axes_dim, use_qk_norm=cfg.use_qk_norm, hidden_size_override=cfg.hidden_size,
        max_latent_resolution=cfg.max_latent_resolution, patch_size=cfg.patch_size,
        patchify_via_reshape=cfg.patchify_via_reshape, pooled_text_embed_dim=cfg.pooled_text_embed_dim,
        token_level_text_embed_dim=cfg.token_level_text_embed_dim, frequency_embed_dim=cfg.frequency_embed_dim,
        max_period=cfg.max_period, dtype=mx.float32, float16_dtype=mx.float32, low_memory_mode=True)


def to_mx(params):
    mx = sys.modules["mlx.core"]
    return [(k, mx.array(v.clone())) for k, v in params.items()]


def run_reference_mmdit(kind, latent, text, pooled, timesteps, t_index):
    mx = sys.modules.get("mlx.core") or (mlx_standin.install() or sys.modules["mlx.core"])
    rcfg_mod = load_reference_mlx("config")
    rmm = load_reference_mlx("mmdit")
    cfg = pin_config(kind)
    params = init_params(mmdit_param_specs(cfg), seed=SEEDS[kind], dtype=torch.float32)
    model = rmm.MMDiT(reference_config(rcfg_mod, cfg))
    model.load_weights(to_mx(params), strict=True)          # the reference module tree takes exactly our parameter names
    ts = mx.array(timesteps.clone())
    model.cache_modulation_params(mx.array(pooled.clone()), ts)
    B = latent.shape[0]
    out = model(latent_image_embeddings=mx.array(latent.clone()),
                token_level_text_embeddings=mx.array(text.clone()[:, :, None, :]),       # (B, T, 1, E)
                timestep=mx.repeat(ts[t_index][None], B, axis=0))
    return out.t.clone()


def run_reference_vae(latent, image):
    mx = sys.modules["mlx.core"]
    rvae = load_reference_mlx("vae")
    dcfg = VAEDecoderConfig(block_out_channels=(32, 64, 64, 64), layers_per_block=3)
    ecfg = VAEEncoderConfig(block_out_channels=(32, 64, 64, 64), layers_per_block=2)
    dec = rvae.VAEDecoder(in_channels=16, out_channels=3, block_out_channels=list(dcfg.block_out_channels),
                          layers_per_block=dcfg.layers_per_block, resnet_groups=32)
    dec.load_weights(to_mx(init_params(vae_decoder_param_specs(dcfg), seed=SEEDS["vae_dec"], dtype=torch.float32)),
                     strict=True)
    enc = rvae.VAEEncoder(in_channels=3, out_channels=32, block_out_channels=list(ecfg.block_out_channels),
                          layers_per_block=ecfg.layers_per_block, resnet_groups=32)
    enc.load_weights(to_mx(init_params(vae_encoder_param_specs(ecfg), seed=SEEDS["vae_enc"], dtype=torch.float32)),
                     strict=True)
    return dec(mx.array(latent.clone())).t.clone(), enc(mx.array(image.clone())).t.clone(), dcfg, ecfg


def run_reference_vae_fullwidth(latent, image_u8):
    """the reference VAE decoder / encoder at their REAL widths (128, 256, 512, 512) — the product's tensor-core convs
    need Cin % 64 == 0, so the GPU checks compare against these — on a small image; read_image's scaling included"""
    mx = sys.modules.get("mlx.core") or (mlx_standin.install() or sys.modules["mlx.core"])
    rvae = load_reference_mlx("vae")
    dcfg, ecfg = VAEDecoderConfig(), VAEEncoderConfig()
    dec = rvae.VAEDecoder(in_channels=16, out_channels=3, block_out_channels=list(dcfg.block_out_channels),
                          layers_per_block=dcfg.layers_per_block, resnet_groups=32)
    dec.load_weights(to_mx(init_params(vae_decoder_param_specs(dcfg), seed=SEEDS["vae_dec"], dtype=torch.float32)),
                     strict=True)
    enc = rvae.VAEEncoder(in_channels=3, out_channels=32, block_out_channels=list(ecfg.block_out_channels),
                          layers_per_block=ecfg.layers_per_block, resnet_groups=32)
    enc.load_weights(to_mx(init_params(vae_encoder_param_specs(ecfg), seed=SEEDS["vae_enc"], dtype=torch.float32)),
                     strict=True)
    img = (mx.array(image_u8.clone())[:, :, :3].astype(mx.float32) / 255) * 2 - 1.0      # mlx/__init__.py:548-549
    decoded = dec(mx.array(latent.clone()))
    decoded_image = mx.clip(decoded / 2 + 0.5, 0, 1)                                       # :581-584
    return decoded.t.clone(), decoded_image.t.clone(), enc(mx.expand_dims(img, axis=0)).t.clone()


def run_reference_sampler():
    mx = sys.modules["mlx.core"]
    rs = load_reference_mlx("sampler")
    out = {}
    for name, cls, shift in (("sd3_shift3", rs.ModelSamplingDiscreteFlow, 3.0), ("flux_shift1", rs.FluxSampler, 1.0),
                             ("flux_shift3", rs.FluxSampler, 3.0)):
        s = cls(shift=shift)
        sig = mx.array(np.array([0.25, 0.5, 1.0], dtype=np.float32))
        out[name] = {"sigma_min": float(s.sigma_min.item()), "sigma_max": float(s.sigma_max.item()),
                     "sigma_of_t": [float(s.sigma(mx.array(float(t))).item()) for t in (1.0, 250.0, 999.0)],
                     "timestep_of_sigma": [float(v) for v in s.timestep(sig).tolist()],
                     "noise_scaling_0.7": float(s.noise_scaling(mx.array(0.7), mx.array(2.0), mx.array(-1.0)).item())}
    return out


def load_reference_pipeline_package():
    """import the reference's real `diffusionkit.mlx` package (pipeline classes, CFGDenoiser, sample_euler) on the
    stand-in; its two remaining imports from argmaxtools.test_utils are empty base classes here"""
    import transformers  # noqa: F401  (before the stand-in: it probes for an installed mlx)

    mlx_standin.install()
    reference_shims.install()
    if "argmaxtools.test_utils" not in sys.modules:
        tu = types.ModuleType("argmaxtools.test_utils")
        tu.AppleSiliconContextMixin = type("AppleSiliconContextMixin", (), {})
        tu.InferenceContextSpec = type("InferenceContextSpec", (), {})
        sys.modules["argmaxtools.test_utils"] = tu
        sys.modules["argmaxtools"].test_utils = tu
    src = reference_shims.REFERENCE_SRC
    if src not in sys.path:
        sys.path.insert(0, src)
    return importlib.import_module("diffusionkit.mlx")


def run_reference_pipeline(kind, cond, pooled, num_steps, cfg_weight, shift, latent_size, seed):
    """the reference's own denoise_latents -> sample_euler -> CFGDenoiser -> MMDiT loop (mlx/__init__.py:253-292, 674-788)
    on a pipeline object assembled by hand (its constructor downloads checkpoints), then decode_latents_to_image"""
    mx = sys.modules.get("mlx.core") or (mlx_standin.install() or sys.modules["mlx.core"])
    dm = load_reference_pipeline_package()
    flux, sd3 = pin_configs()
    cfg = flux if kind == "flux" else sd3
    params = init_params(mmdit_param_specs(cfg), seed=SEEDS[kind], dtype=torch.float32)
    Pipe = dm.FluxPipeline if kind == "flux" else dm.DiffusionPipeline
    pipe = object.__new__(Pipe)
    from diffusionkit.mlx import config as rcfg_mod, mmdit as rmm, vae as rvae

    pipe.mmdit = rmm.MMDiT(reference_config(rcfg_mod, cfg))
    pipe.mmdit.load_weights(to_mx(params), strict=True)
    pipe.sampler = (dm.FluxSampler if kind == "flux" else dm.ModelSamplingDiscreteFlow)(shift=shift)
    pipe.latent_format = (dm.FluxLatentFormat if kind == "flux" else dm.SD3LatentFormat)()
    pipe.activation_dtype = pipe.dtype = pipe.float16_dtype = mx.float32
    # clear_cache() re-reads the adaLN weights it "offloaded" (mlx/__init__.py:686-689): hand them back from memory
    pipe.load_mmdit = lambda only_modulation_dict=False: [(k, mx.array(v.clone())) for k, v in params.items()
                                                          if "adaLN" in k]
    dcfg = VAEDecoderConfig(block_out_channels=(32, 64, 64, 64), layers_per_block=3)
    pipe.decoder = rvae.VAEDecoder(in_channels=16, out_channels=3, block_out_channels=list(dcfg.block_out_channels),
                                   layers_per_block=dcfg.layers_per_block, resnet_groups=32)
    pipe.decoder.load_weights(to_mx(init_params(vae_decoder_param_specs(dcfg), seed=SEEDS["vae_dec"],
                                                dtype=torch.float32)), strict=True)
    latent, iter_time = pipe.denoise_latents(mx.array(cond.clone()), mx.array(pooled.clone()), num_steps=num_steps,
                                             cfg_weight=cfg_weight, latent_size=latent_size, seed=seed)
    image = pipe.decode_latents_to_image(latent)
    sig = pipe.get_sigmas(pipe.sampler, num_steps)
    return latent.t.clone(), image.t.clone(), sig.t.clone(), len(iter_time)


PIPELINE_CASES = {
    # kind: (num_steps, cfg_weight, shift, latent_size, seed, text_len)
    "flux": (3, 0.0, 1.0, (8, 12), 7, 10),
    "sd3": (4, 4.5, 3.0, (12, 8), 11, 14),
}


def make_pipeline_inputs(kind):
    flux, sd3 = pin_configs()
    cfg = flux if kind == "flux" else sd3
    T = PIPELINE_CASES[kind][5]
    n = 1 if kind == "flux" else 2                 # SD3 with CFG: [positive | negative] rows
    g = torch.Generator().manual_seed(61 if kind == "flux" else 62)
    return (torch.randn((n, T, cfg.token_level_text_embed_dim), generator=g),
            torch.randn((n, cfg.pooled_text_embed_dim), generator=g))


def make_inputs(kind):
    cfg = pin_config(kind)
    g = torch.Generator().manual_seed({"flux": 51, "sd3": 52, "sd35": 56}[kind])
    B, H, W, T = {"flux": (2, 8, 12, 10), "sd3": (2, 12, 8, 14), "sd35": (1, 10, 6, 9)}[kind]
    latent = torch.randn((B, H, W, 16), generator=g)
    text = torch.randn((B, T, cfg.token_level_text_embed_dim), generator=g)
    pooled = torch.randn((B, cfg.pooled_text_embed_dim), generator=g)
    timesteps = torch.tensor([1000.0, 613.0, 250.0])
    return latent, text, pooled, timesteps, 1


if __name__ == "__main__":
    assert reference_mlx_available(), "set DIFFUSIONKIT_REFERENCE to an argmaxinc/DiffusionKit checkout"
    for kind in ("flux", "sd3", "sd35"):
        latent, text, pooled, timesteps, ti = make_inputs(kind)
        y = run_reference_mmdit(kind, latent, text, pooled, timesteps, ti)
        np.savez_compressed(os.path.join(HERE, f"reference_mlxsrc_{kind}_mmdit.npz"), latent=latent.numpy(),
                            text=text.numpy(), pooled=pooled.numpy(), timesteps=timesteps.numpy(), t_index=ti,
                            out=y.numpy())
        print(kind, tuple(y.shape), float(y.abs().mean()))
    g = torch.Generator().manual_seed(53)
    z = torch.randn((1, 4, 6, 16), generator=g)
    img = torch.rand((1, 32, 48, 3), generator=g) * 2 - 1
    d, e, _, _ = run_reference_vae(z, img)
    np.savez_compressed(os.path.join(HERE, "reference_mlxsrc_vae.npz"), latent=z.numpy(), image=img.numpy(),
                        decoded=d.numpy(), encoded=e.numpy())
    print("vae", tuple(d.shape), tuple(e.shape))
    with open(os.path.join(HERE, "reference_mlxsrc_sampler.json"), "w") as f:
        json.dump(run_reference_sampler(), f, indent=1)
    zf = torch.randn((1, 8, 8, 16), generator=torch.Generator().manual_seed(54))
    img_u8 = torch.from_numpy(np.random.RandomState(55).randint(0, 256, (64, 64, 3)).astype(np.uint8))
    draw, dimg, ehid = run_reference_vae_fullwidth(zf, img_u8)
    np.savez_compressed(os.path.join(HERE, "reference_mlxsrc_vae_fullwidth.npz"), latent=zf.numpy(),
                        image_u8=img_u8.numpy(), decoded=draw.numpy().astype(np.float16),
                        decoded_image=dimg.numpy().astype(np.float16), encoded=ehid.numpy())
    print("vae full width", tuple(draw.shape), tuple(ehid.shape))
    for kind, (steps, cfgw, shift, lat, seed, _) in PIPELINE_CASES.items():
        cond, pooled = make_pipeline_inputs(kind)
        latent, image, sig, n_iter = run_reference_pipeline(kind, cond, pooled, steps, cfgw, shift, lat, seed)
        np.savez_compressed(os.path.join(HERE, f"reference_mlxsrc_{kind}_pipeline.npz"), cond=cond.numpy(),
                            pooled=pooled.numpy(), latent=latent.numpy(), image=image.numpy(), sigmas=sig.numpy())
        print("pipeline", kind, tuple(latent.shape), tuple(image.shape), sig.tolist(), n_iter)
