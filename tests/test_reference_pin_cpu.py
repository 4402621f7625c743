"""CPU: the oracle pinned against the REFERENCE'S OWN code.

argmaxinc/DiffusionKit ships a PyTorch twin of its SD3 MMDiT and VAE decoder (python/src/diffusionkit/torch/mmdit.py,
vae.py — the sources of its Core ML conversion).  Unlike the MLX path they can execute under plain PyTorch once the four
generic argmaxtools layers they import are supplied (tests/golden/reference_shims.py).  tests/golden/
make_reference_golden.py ran them on the deterministic synthetic weights and committed inputs + outputs
(reference_torch_*.npz); here the oracle has to reproduce those outputs.  The two documented differences between the
twins are switched on the oracle side: tanh GELU (torch/mmdit.py:242 vs mlx/mmdit.py:421) and GroupNorm eps 1e-6
(torch/vae.py:20 vs the MLX default 1e-5).

The checkpoint-loader and PSNR pins compare with reference outputs stored by tests/golden/make_reference_pins.py.
"""
import json
import os

import numpy as np
import torch

from diffusionkit_b200.weights import init_params, mmdit_param_specs, vae_decoder_param_specs
from oracle.mmdit_ref import MMDiTRef
from oracle.vae_ref import VAEDecoderRef
from tests.golden import make_reference_golden as mk
from tests.golden import make_reference_pins as pins
from tests.oracle_bridge import ref_config

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _oracle_mmdit(latent, text, pooled, timestep):
    cfg = mk.pin_mmdit_config()
    params = init_params(mmdit_param_specs(cfg), seed=mk.MMDIT_SEED, dtype=torch.float32)
    rc = ref_config(cfg)
    rc.gelu_tanh = True
    ref = MMDiTRef(rc, params, act_dtype=None)
    ref.cache_modulation_params(pooled, timestep[:1])
    return ref(latent, text, timestep)


def _oracle_vae(z):
    cfg = mk.pin_vae_config()
    params = init_params(vae_decoder_param_specs(cfg), seed=mk.VAE_SEED, dtype=torch.float32)
    dec = VAEDecoderRef(params, None, cfg.block_out_channels, cfg.layers_per_block)
    dec.gn_eps = 1e-6
    return dec(z)


def test_oracle_mmdit_matches_reference_torch_module():
    g = np.load(os.path.join(GOLD, "reference_torch_mmdit.npz"))
    latent, text, pooled, timestep = [torch.from_numpy(g[k]) for k in ("latent", "text", "pooled", "timestep")]
    got = _oracle_mmdit(latent, text, pooled, timestep)
    want = torch.from_numpy(g["out"])
    assert got.shape == want.shape == (2, 12, 8, 16)
    assert torch.allclose(got, want, atol=2e-4, rtol=1e-4), float((got - want).abs().max())
    # the pin is sensitive to exactly the things a restatement gets wrong: activation flavour ...
    cfg = mk.pin_mmdit_config()
    params = init_params(mmdit_param_specs(cfg), seed=mk.MMDIT_SEED, dtype=torch.float32)
    erf = MMDiTRef(ref_config(cfg), params, act_dtype=None)
    erf.cache_modulation_params(pooled, timestep[:1])
    assert not torch.allclose(erf(latent, text, timestep), want, atol=2e-4, rtol=1e-4)


def test_oracle_vae_decoder_matches_reference_torch_module():
    g = np.load(os.path.join(GOLD, "reference_torch_vae_decoder.npz"))
    z, want = torch.from_numpy(g["latent"]), torch.from_numpy(g["out"])
    got = _oracle_vae(z)
    assert got.shape == want.shape == (1, 48, 32, 3)
    assert torch.allclose(got, want, atol=2e-4, rtol=1e-4), float((got - want).abs().max())


def test_fixtures_are_what_the_reference_produces_today():
    """the fixtures hold the reference's outputs for the inputs make_inputs() draws today (to the last bits, which
    torch.randn's CPU kernels vary between instruction sets); re-running
    tests/golden/make_reference_golden.py against a reference checkout and diffing the fixtures checks the outputs"""
    latent, text, pooled, timestep, z = mk.make_inputs()
    g = np.load(os.path.join(GOLD, "reference_torch_mmdit.npz"))
    for k, v in (("latent", latent), ("text", text), ("pooled", pooled), ("timestep", timestep)):
        assert np.allclose(g[k], v.numpy(), rtol=1e-5, atol=1e-5), k
    gv = np.load(os.path.join(GOLD, "reference_torch_vae_decoder.npz"))
    assert np.allclose(gv["latent"], z.numpy(), rtol=1e-5, atol=1e-5)
    assert g["out"].shape == (2, 12, 8, 16) and gv["out"].shape == (1, 48, 32, 3)


def test_checkpoint_loaders_match_the_reference_loaders():
    """SURVEY.md §8 row f1 pinned by reference code: an upstream-layout (Stability SD3 / LDM) checkpoint went through the
    REFERENCE's own key adjustments (torch/mmdit.py:424-497, torch/model_io.py:90-122) into the reference modules with
    strict=True (tests/golden/make_reference_pins.py stored their outputs); through diffusionkit_b200.model_io into the
    oracle it has to give the same outputs"""
    from diffusionkit_b200 import model_io

    g = np.load(os.path.join(GOLD, "reference_pins.npz"))
    latent, text, pooled, timestep, z = mk.make_inputs()
    upstream, vup = pins.torch_loader_checkpoints()

    # ---- SD3 MMDiT
    cfg = mk.pin_mmdit_config()
    mine = model_io.sd3_checkpoint_to_params(upstream)
    model_io.check_against_specs(mine, mmdit_param_specs(cfg))
    rc = ref_config(cfg)
    rc.gelu_tanh = True
    ref = MMDiTRef(rc, mine, act_dtype=None)
    ref.cache_modulation_params(pooled, timestep[:1])
    pins.assert_close(g, "torch_loader_mmdit", ref(latent, text, timestep), atol=2e-4, rtol=1e-4)

    # ---- VAE decoder
    vcfg = mk.pin_vae_config()
    vmine = model_io.vae_decoder_checkpoint_to_params(vup)
    model_io.check_against_specs(vmine, vae_decoder_param_specs(vcfg))
    dec = VAEDecoderRef(vmine, None, vcfg.block_out_channels, vcfg.layers_per_block)
    dec.gn_eps = 1e-6
    pins.assert_close(g, "torch_loader_vae", dec(z), atol=2e-4, rtol=1e-4)


def test_psnr_metric_is_the_reference_metric():
    """the parity metric itself (tests use oracle.sampler_ref.compute_psnr): reference diffusionkit/utils.py:70-82"""
    from oracle.sampler_ref import compute_psnr

    want = json.load(open(os.path.join(GOLD, "reference_pins.json")))["psnr"]
    assert abs(compute_psnr(*pins.psnr_inputs()) - want) < 1e-3
