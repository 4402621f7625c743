"""CPU: the oracle against the reference's MLX SOURCE (mlx/mmdit.py, vae.py, sampler.py, clip.py, t5.py, tokenizer.py,
model_io.py, __init__.py), executed from a reference checkout on tests/golden/mlx_standin.py — a torch-backed stand-in
for the MLX primitives those files call.  Fixtures committed by tests/golden/make_reference_mlx_golden.py (fp32) and
tests/golden/make_reference_pins.py; re-running those against a reference checkout and diffing the fixtures checks that
the reference has not drifted.

What this pins: every line of the reference above the primitive level, for BOTH model families — FLUX (dual + single-
stream blocks, RoPE tables and rotation, QK-RMSNorm, reshape patchify / unpack, [text | image] order, shared fc2/o_proj
bias zeroing, parallel MLP) and SD3 (learned positional embedding crop, conv patchify, [image | text] order, skipped text
post-path of the last block) — plus the modulation cache keyed by timestep, the VAE decoder AND encoder stacks, and the
sampler formulas.  What it cannot pin: the numerics of MLX's own kernels (the stand-in computes in fp32 torch).
"""
import json
import os

import numpy as np
import pytest
import torch

from diffusionkit_b200.weights import (init_params, mmdit_param_specs, vae_decoder_param_specs,
                                       vae_encoder_param_specs)
from oracle import sampler_ref as sr
from oracle.mmdit_ref import MMDiTRef
from oracle.vae_ref import VAEDecoderRef, VAEEncoderRef
from tests.golden import make_reference_mlx_golden as mk
from tests.golden import make_reference_pins as pins
from tests.oracle_bridge import ref_config

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _pins():
    return np.load(os.path.join(GOLD, "reference_pins.npz")), json.load(open(os.path.join(GOLD, "reference_pins.json")))


def _oracle_mmdit(kind, latent, text, pooled, timesteps, ti):
    cfg = mk.pin_config(kind)
    params = init_params(mmdit_param_specs(cfg), seed=mk.SEEDS[kind], dtype=torch.float32)
    ref = MMDiTRef(ref_config(cfg), params, act_dtype=None)
    ref.cache_modulation_params(pooled, timesteps)
    return ref(latent, text, timesteps[ti].repeat(latent.shape[0]))


@pytest.mark.parametrize("kind", ["flux", "sd3", "sd35"])
def test_oracle_mmdit_matches_reference_mlx_source(kind):
    g = np.load(os.path.join(GOLD, f"reference_mlxsrc_{kind}_mmdit.npz"))
    latent, text, pooled, timesteps = [torch.from_numpy(g[k]) for k in ("latent", "text", "pooled", "timesteps")]
    got = _oracle_mmdit(kind, latent, text, pooled, timesteps, int(g["t_index"]))
    want = torch.from_numpy(g["out"])
    assert got.shape == want.shape
    assert torch.allclose(got, want, atol=3e-4, rtol=1e-4), float((got - want).abs().max())
    # and it is the cached modulation of THAT timestep which is used, not another one
    other = _oracle_mmdit(kind, latent, text, pooled, timesteps, 0)
    assert not torch.allclose(other, want, atol=1e-3)


def test_oracle_vae_matches_reference_mlx_source():
    g = np.load(os.path.join(GOLD, "reference_mlxsrc_vae.npz"))
    from diffusionkit_b200.config import VAEDecoderConfig, VAEEncoderConfig

    dcfg = VAEDecoderConfig(block_out_channels=(32, 64, 64, 64), layers_per_block=3)
    ecfg = VAEEncoderConfig(block_out_channels=(32, 64, 64, 64), layers_per_block=2)
    dec = VAEDecoderRef(init_params(vae_decoder_param_specs(dcfg), seed=mk.SEEDS["vae_dec"], dtype=torch.float32), None,
                        dcfg.block_out_channels, dcfg.layers_per_block)
    enc = VAEEncoderRef(init_params(vae_encoder_param_specs(ecfg), seed=mk.SEEDS["vae_enc"], dtype=torch.float32), None,
                        ecfg.block_out_channels, ecfg.layers_per_block)
    d = dec(torch.from_numpy(g["latent"]))
    e = enc(torch.from_numpy(g["image"]))
    assert torch.allclose(d, torch.from_numpy(g["decoded"]), atol=3e-4, rtol=1e-4)
    assert torch.allclose(e, torch.from_numpy(g["encoded"]), atol=3e-4, rtol=1e-4)


def test_oracle_sampler_matches_reference_mlx_source():
    want = json.load(open(os.path.join(GOLD, "reference_mlxsrc_sampler.json")))
    for name, cls, shift in (("sd3_shift3", sr.ModelSamplingDiscreteFlowRef, 3.0), ("flux_shift1", sr.FluxSamplerRef, 1.0),
                             ("flux_shift3", sr.FluxSamplerRef, 3.0)):
        s = cls(shift)
        w = want[name]
        assert abs(float(s.sigma_min) - w["sigma_min"]) < 1e-7 and abs(float(s.sigma_max) - w["sigma_max"]) < 1e-7
        got = [float(s.sigma(torch.tensor(t))) for t in (1.0, 250.0, 999.0)]
        assert np.allclose(got, w["sigma_of_t"], rtol=1e-6, atol=1e-8), name
        ts = s.timestep(torch.tensor([0.25, 0.5, 1.0]))
        assert np.allclose(np.asarray(ts, dtype=np.float64), w["timestep_of_sigma"], rtol=1e-6)
        ns = s.noise_scaling(0.7, torch.tensor(2.0), torch.tensor(-1.0))
        assert abs(float(ns) - w["noise_scaling_0.7"]) < 1e-6


def test_mlxsrc_fixtures_are_what_the_reference_source_produces_today():
    """the MMDiT fixtures hold the reference's outputs for the inputs make_inputs() draws today (to the last bits, which
    torch.randn's CPU kernels vary between instruction sets)"""
    for kind in ("flux", "sd3", "sd35"):
        latent, text, pooled, timesteps, ti = mk.make_inputs(kind)
        g = np.load(os.path.join(GOLD, f"reference_mlxsrc_{kind}_mmdit.npz"))
        for k, v in (("latent", latent), ("text", text), ("pooled", pooled), ("timesteps", timesteps)):
            assert np.allclose(g[k], v.numpy(), rtol=1e-5, atol=1e-5), (kind, k)
        assert int(g["t_index"]) == ti and g["out"].shape == latent.shape, kind
    assert set(json.load(open(os.path.join(GOLD, "reference_mlxsrc_sampler.json")))) == {"sd3_shift3", "flux_shift1",
                                                                                        "flux_shift3"}


def test_reference_16bit_quirks_match_the_oracle_flags():
    """the reference source run with 16-bit activations on the stand-in (bf16 sinusoid, Q5; per-op rounding) stays within
    16-bit tolerance of the oracle's act_dtype emulation — a looser check that the dtype plumbing is the same"""
    from dataclasses import replace

    g, _ = _pins()
    out = torch.from_numpy(g["mlx_16bit_flux_mmdit"])
    flux, _ = mk.pin_configs()
    cfg16 = replace(flux, dtype=torch.bfloat16, float16_dtype=torch.bfloat16)
    params = init_params(mmdit_param_specs(cfg16), seed=mk.SEEDS["flux"], dtype=torch.float32)
    p16 = {k: v.to(torch.bfloat16) for k, v in params.items()}
    latent, text, pooled, timesteps, ti = mk.make_inputs("flux")
    l16, t16, pl16 = [x.to(torch.bfloat16) for x in (latent, text, pooled)]
    ref = MMDiTRef(ref_config(cfg16), {k: v.float() for k, v in p16.items()}, act_dtype=torch.bfloat16)
    tsf = timesteps.to(torch.bfloat16).float()
    ref.cache_modulation_params(pl16.float(), tsf)
    got = ref(l16.float(), t16.float(), tsf[ti].repeat(2))
    assert got.shape == out.shape
    rel = float((got - out).norm() / out.norm())
    assert rel < 2e-2, rel


@pytest.mark.parametrize("kind", ["flux", "sd3"])
def test_oracle_denoise_loop_matches_reference_pipeline_source(kind):
    """the reference's own denoise_latents -> sample_euler -> CFGDenoiser loop and decode_latents_to_image
    (mlx/__init__.py:253-292, 581-584, 674-788), run on the stand-in, vs the oracle's loop: schedule, seeded noise,
    noise_scaling, timestep rounding, CFG row order and mix, Euler update, process_out, decode + clip"""
    from diffusionkit_b200.config import VAEDecoderConfig
    from oracle.vae_ref import decode_latents_to_image

    steps, cfgw, shift, lat, seed, _ = mk.PIPELINE_CASES[kind]
    g = np.load(os.path.join(GOLD, f"reference_mlxsrc_{kind}_pipeline.npz"))
    cond, pooled = torch.from_numpy(g["cond"]), torch.from_numpy(g["pooled"])
    flux, sd3 = mk.pin_configs()
    cfg = flux if kind == "flux" else sd3
    params = init_params(mmdit_param_specs(cfg), seed=mk.SEEDS[kind], dtype=torch.float32)
    sampler = sr.FluxSamplerRef(shift) if kind == "flux" else sr.ModelSamplingDiscreteFlowRef(shift)
    sig = sr.get_sigmas(sampler, steps)
    assert np.allclose(np.asarray(sig, dtype=np.float64), g["sigmas"], rtol=1e-6, atol=1e-8)
    ref = MMDiTRef(ref_config(cfg), params, act_dtype=None)
    x0 = sampler.noise_scaling(float(sig[0]), sr.get_noise(seed, lat[0], lat[1]), sr.get_empty_latent(lat[0], lat[1]))
    x = sr.sample_euler(lambda xin, c, t: ref(xin, c, t), ref.cache_modulation_params, x0, sig, cond, pooled, cfgw,
                        torch.float32)
    latent = sr.process_out(x, "flux" if kind == "flux" else "sd3")
    want = torch.from_numpy(g["latent"])
    assert latent.shape == want.shape
    assert torch.allclose(latent, want, atol=2e-3, rtol=1e-3), float((latent - want).abs().max())
    dcfg = VAEDecoderConfig(block_out_channels=(32, 64, 64, 64), layers_per_block=3)
    dec = VAEDecoderRef(init_params(vae_decoder_param_specs(dcfg), seed=mk.SEEDS["vae_dec"], dtype=torch.float32), None,
                        dcfg.block_out_channels, dcfg.layers_per_block)
    img = decode_latents_to_image(dec, want)
    assert torch.allclose(img, torch.from_numpy(g["image"]), atol=5e-4), float((img - torch.from_numpy(g["image"])).abs().max())


def test_pipeline_fixtures_are_what_the_reference_source_produces_today():
    """the pipeline fixtures hold the reference's outputs for the inputs make_pipeline_inputs() draws today, and
    the reference loop ran one iteration per step"""
    _, meta = _pins()
    for kind, (steps, cfgw, shift, lat, seed, _) in mk.PIPELINE_CASES.items():
        cond, pooled = mk.make_pipeline_inputs(kind)
        g = np.load(os.path.join(GOLD, f"reference_mlxsrc_{kind}_pipeline.npz"))
        assert np.allclose(g["cond"], cond.numpy(), rtol=1e-5, atol=1e-5), kind
        assert np.allclose(g["pooled"], pooled.numpy(), rtol=1e-5, atol=1e-5), kind
        assert meta["pipeline_iterations"][kind] == steps
        assert g["latent"].shape == (1, lat[0], lat[1], 16), kind


def test_text_encoder_oracles_match_reference_mlx_source():
    """CLIPTextModel (mlx/clip.py) and SD3T5Encoder (mlx/t5.py) of the reference, run on the stand-in, vs oracle/text_ref.py
    (which tests/test_text_cpu.py separately pins against transformers)"""
    from oracle.text_ref import CLIPTextModelRef, T5EncoderRef

    g, _ = _pins()
    clip, (tc, tparams, ttokens) = pins.text_encoder_cases()
    for name, cfg, params, tokens in clip:
        pooled, last, hidden = CLIPTextModelRef(params, cfg.num_layers, cfg.num_heads, cfg.hidden_act)(tokens)
        for got, key in ((last, "last"), (pooled, "pooled"), (hidden[-2], "hidden_m2")):
            pins.assert_close(g, f"{name}_{key}", got, atol=3e-4, rtol=1e-4)
    pins.assert_close(g, "t5_out", T5EncoderRef(tparams, tc.num_layers, tc.num_heads)(ttokens), atol=5e-4, rtol=1e-4)


def test_checkpoint_key_maps_match_reference_mlx_loaders():
    """SURVEY.md §8 row f1 against the reference's own MLX loader functions (mlx/model_io.py:130-636), run on the stand-in:
    an upstream-layout checkpoint (BFL FLUX, Stability SD3, LDM VAE, HF T5) goes through the reference's
    *_state_dict_adjustments (for FLUX: what Module.update leaves in the reference module tree) and through
    diffusionkit_b200.model_io; both must give the same names and bit-identical tensors"""
    from diffusionkit_b200 import model_io

    _, meta = _pins()
    flux, _ = mk.pin_configs()
    ck = pins.key_map_checkpoints()
    mine = {"flux": model_io.flux_checkpoint_to_params(ck["flux"], flux.hidden_size, flux.mlp_ratio),
            "sd3": model_io.sd3_checkpoint_to_params(ck["sd3"]),
            "vae_decoder": model_io.vae_decoder_checkpoint_to_params(ck["vae_decoder"]),
            "vae_encoder": model_io.vae_encoder_checkpoint_to_params(ck["vae_encoder"]),
            "t5": model_io.t5_checkpoint_to_params(ck["t5"])}
    assert set(mine) == set(meta["key_maps"])
    for part, params in mine.items():
        want = meta["key_maps"][part]
        assert set(want) == set(params), (part, sorted(set(want) ^ set(params))[:6])
        for k, v in params.items():
            assert pins.digest(v) == want[k], (part, k)


def test_clip_tokenizer_matches_reference_tokenizer(tmp_path):
    """diffusionkit_b200.tokenizer.Tokenizer vs the reference's own class (mlx/tokenizer.py:14-122) on the synthetic
    vocabulary (tests/test_text_cpu.py also checks it against transformers' CLIPTokenizer)"""
    from diffusionkit_b200.tokenizer import load_tokenizer
    from tests.test_text_cpu import _synthetic_clip_vocab

    want = _pins()[1]["tokenizer"]
    vf, mf, vocab = _synthetic_clip_vocab(tmp_path)
    mine = load_tokenizer(vf, mf, pad_with_eos=True)
    assert len(want["tokens"]) == len(pins.TOKENIZER_TEXTS)
    for text, ref_tokens in zip(pins.TOKENIZER_TEXTS, want["tokens"]):
        assert [int(t) for t in mine.tokenize(text)] == ref_tokens, text
    assert mine.eos_token == want["eos_token"] and mine.bos_token == want["bos_token"]


def test_encode_text_composition_matches_reference_pipeline_source():
    """the reference's own _tokenize / encode_text of both pipelines (mlx/__init__.py:174-251, 642-671) on the stand-in, vs
    the product's host-side _tokenize and the oracle's encode_text_* composition"""
    from diffusionkit_b200.pipeline import DiffusionPipeline as OurPipe
    from oracle.text_ref import CLIPTextModelRef, T5EncoderRef, encode_text_flux, encode_text_sd3, tokenize_pair

    g, meta = _pins()
    s = pins.encode_text_setup()
    cl, cg, tc = s["cl"], s["cg"], s["tc"]
    o_l = CLIPTextModelRef(s["pl"], cl.num_layers, cl.num_heads, cl.hidden_act)
    o_g = CLIPTextModelRef(s["pg"], cg.num_layers, cg.num_heads, cg.hidden_act)
    o_t = T5EncoderRef(s["pt"], tc.num_layers, tc.num_heads)
    tok_l, tok_g, text, neg = s["tok_l"], s["tok_g"], s["text"], s["neg"]

    for kind in ("sd3", "flux"):
        t5_len = s["t5_len"][kind]
        tok_t5 = pins.WordTokenizer(t5_len, False, eos=1)
        for cfgw in (5.0, 0.0):
            case = f"{kind}_cfg{int(cfgw)}"
            # token batching: reference _tokenize == product _tokenize == oracle tokenize_pair
            n = neg if cfgw > 1 else None
            for tk, want in zip((tok_l, tok_g, tok_t5), meta["encode_text_tokens"][case]):
                want_tok = torch.tensor(want)
                assert torch.equal(OurPipe._tokenize(None, tk, text, n), want_tok), case
                assert torch.equal(tokenize_pair(tk, text, n), want_tok), case
            tl, tg, tt = [tokenize_pair(tk, text, n) for tk in (tok_l, tok_g, tok_t5)]
            if kind == "sd3":
                got_c, got_p = encode_text_sd3(o_l, o_g, o_t, tl, tg, tt)
                assert got_c.shape == (2, 77 + t5_len, 4096) and got_p.shape == (2, 128 + 192)
            else:
                got_c, got_p = encode_text_flux(o_l, o_t, tl, tt, t5_len)
                assert got_c.shape == (1, t5_len, 4096) and got_p.shape == (1, 128)
            pins.assert_close(g, f"encode_text_{case}_cond", got_c, atol=5e-4, rtol=1e-4)
            pins.assert_close(g, f"encode_text_{case}_pooled", got_p, atol=5e-4, rtol=1e-4)


def test_img2img_flow_matches_reference_pipeline_source(tmp_path):
    """image_path / denoise arguments (mlx/__init__.py:270-285, 536-551, 586-594): read_image incl. the LANCZOS resize to
    multiples of 64, VAE encoder, clipped-logvar posterior sample drawn with the SAME seeded noise as the diffusion
    noise, process_in, schedule trimming, noise_scaling with a tensor x_T — reference source on the stand-in vs the
    oracle composition the GPU check (tests/model_checks.py::check_pipeline_img2img) compares the product against"""
    from PIL import Image

    from diffusionkit_b200.config import VAEEncoderConfig
    from diffusionkit_b200.pipeline import DiffusionPipeline as OurPipe
    from oracle.vae_ref import encode_image_to_latents, read_image_array

    g, meta = _pins()
    steps, denoise, seed = pins.IMG2IMG["steps"], pins.IMG2IMG["denoise"], pins.IMG2IMG["seed"]
    latent = torch.from_numpy(g["img2img_latent"])
    assert meta["img2img_iterations"] == steps - int(steps * (1 - denoise)) and latent.shape == (1, 8, 16, 16)
    flux, _ = mk.pin_configs()
    params = init_params(mmdit_param_specs(flux), seed=mk.SEEDS["flux"], dtype=torch.float32)
    ecfg = VAEEncoderConfig(block_out_channels=(32, 64, 64, 64), layers_per_block=2)
    eparams = init_params(vae_encoder_param_specs(ecfg), seed=mk.SEEDS["vae_enc"], dtype=torch.float32)
    path = str(tmp_path / "in.png")
    Image.fromarray(pins.img2img_image()).save(path)
    cond, pooled = mk.make_pipeline_inputs("flux")

    # product host side: the same pixels after the resize rule
    ours_u8 = OurPipe._load_image_u8(None, path)
    assert ours_u8.shape == (64, 128, 3)
    pins.assert_close(g, "img2img_read_image", read_image_array(torch.from_numpy(ours_u8)), atol=1e-6, rtol=0)

    # oracle composition
    enc = VAEEncoderRef(eparams, None, ecfg.block_out_channels, ecfg.layers_per_block)
    sampler = sr.FluxSamplerRef(1.0)
    sig = sr.get_sigmas(sampler, steps)[int(steps * (1 - denoise)):]
    noise = sr.get_noise(seed, 8, 16)
    z = encode_image_to_latents(enc, read_image_array(torch.from_numpy(ours_u8)), noise)
    x_T = (z - 0.1159) * 0.3611
    ref = MMDiTRef(ref_config(flux), params, act_dtype=None)
    x = sr.sample_euler(lambda xin, c, t: ref(xin, c, t), ref.cache_modulation_params,
                        sampler.noise_scaling(float(sig[0]), noise, x_T), sig, cond, pooled, 0.0, torch.float32)
    got = sr.process_out(x, "flux")
    assert torch.allclose(got, latent, atol=2e-3, rtol=1e-3), float((got - latent).abs().max())


def test_oracle_fullwidth_vae_matches_reference_mlx_source():
    """the real-width decoder / encoder fixture the GPU check compares the product against, reproduced by the oracle"""
    from diffusionkit_b200.config import VAEDecoderConfig, VAEEncoderConfig
    from oracle.vae_ref import decode_latents_to_image, read_image_array

    g = np.load(os.path.join(GOLD, "reference_mlxsrc_vae_fullwidth.npz"))
    dcfg, ecfg = VAEDecoderConfig(), VAEEncoderConfig()
    dec = VAEDecoderRef(init_params(vae_decoder_param_specs(dcfg), seed=mk.SEEDS["vae_dec"], dtype=torch.float32), None,
                        dcfg.block_out_channels, dcfg.layers_per_block)
    z = torch.from_numpy(g["latent"])
    assert torch.allclose(dec(z), torch.from_numpy(g["decoded"].astype(np.float32)), atol=2e-2, rtol=2e-3)   # fp16 store
    assert torch.allclose(decode_latents_to_image(dec, z), torch.from_numpy(g["decoded_image"].astype(np.float32)),
                          atol=2e-3)
    enc = VAEEncoderRef(init_params(vae_encoder_param_specs(ecfg), seed=mk.SEEDS["vae_enc"], dtype=torch.float32), None,
                        ecfg.block_out_channels, ecfg.layers_per_block)
    e = enc(read_image_array(torch.from_numpy(g["image_u8"])))
    assert torch.allclose(e, torch.from_numpy(g["encoded"]), atol=5e-4, rtol=1e-4)


@pytest.mark.parametrize("kind", ["flux", "sd3"])
def test_16bit_denoise_loop_emulation_tracks_reference_source(kind):
    """The GPU tests compare the product with the oracle run in 16-bit EMULATION (act_dtype).  The reference's own
    pipeline source ran with real 16-bit arrays on the stand-in (bf16 FLUX / fp16 SD3: timestep rounding and the
    config.dtype sinusoid of quirk Q5, the rounding residue of quirk Q6, per-op rounding; stored by
    tests/golden/make_reference_pins.py) and the oracle's emulation has to land on the same final latent.  Measured:
    5.3e-3 (FLUX) / 2.0e-3 (SD3) rel-L2 — while the reference's 16-bit run is 1.1e-1 / 2.7e-2 away from its own fp32 run,
    i.e. the emulation reproduces the reference's 16-bit behaviour, not just the fp32 math."""
    from dataclasses import replace

    g, _ = _pins()
    want = torch.from_numpy(g[f"mlx_16bit_{kind}_pipeline_latent"])
    dt = torch.bfloat16 if kind == "flux" else torch.float16
    steps, cfgw, shift, lat, seed, _ = mk.PIPELINE_CASES[kind]
    cfg = replace(mk.pin_config(kind), dtype=dt, float16_dtype=dt)
    p16 = {k: v.to(dt) for k, v in init_params(mmdit_param_specs(cfg), seed=mk.SEEDS[kind], dtype=torch.float32).items()}
    cond, pooled = mk.make_pipeline_inputs(kind)
    c16, pl16 = cond.to(dt), pooled.to(dt)
    sampler = sr.FluxSamplerRef(shift) if kind == "flux" else sr.ModelSamplingDiscreteFlowRef(shift)
    sig = sr.get_sigmas(sampler, steps)
    ref = MMDiTRef(ref_config(cfg), {k: v.float() for k, v in p16.items()}, act_dtype=dt)
    x0 = sampler.noise_scaling(float(sig[0]), sr.get_noise(seed, lat[0], lat[1]), sr.get_empty_latent(lat[0], lat[1]))
    x = sr.sample_euler(lambda xin, c, t: ref(xin, c, t), ref.cache_modulation_params, x0, sig, c16.float(), pl16.float(),
                        cfgw, dt)
    got = sr.process_out(x, "flux" if kind == "flux" else "sd3")
    assert got.shape == want.shape
    rel = float((got - want).norm() / want.norm())
    assert rel < 2e-2, rel
