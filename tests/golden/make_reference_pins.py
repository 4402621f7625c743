"""Golden data for the reference pins beyond the model forward passes: the checkpoint loaders, the PSNR metric, the CLIP
tokenizer, the text encoders and their composition, the img2img flow and the 16-bit denoise loop.  The reference runs
as in make_reference_golden.py (its PyTorch modules) and make_reference_mlx_golden.py (its MLX source on the torch
stand-in); what it produced is stored here, so the tests (tests/test_reference_pin_cpu.py,
tests/test_reference_mlxsrc_pin_cpu.py) run without a reference checkout.  The inputs are not stored: they come from the
seeded helpers below, which the tests call too.

Writes tests/golden/reference_pins.npz and reference_pins.json.  Re-running it against the reference and diffing the
two files is the check that the reference has not drifted from what the tests compare against.  Run from the repo root:
    DIFFUSIONKIT_REFERENCE=<argmaxinc/DiffusionKit checkout> python tests/golden/make_reference_pins.py
"""
import hashlib
import importlib.util
import json
import os
import sys
import tempfile
from dataclasses import replace

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
HERE = os.path.dirname(os.path.abspath(__file__))
NPZ = os.path.join(HERE, "reference_pins.npz")
JSON = os.path.join(HERE, "reference_pins.json")

from diffusionkit_b200.config import (CLIPTextModelConfig, T5EncoderConfig, VAEDecoderConfig,  # noqa: E402
                                      VAEEncoderConfig, tiny_clip_config, tiny_t5_config)
from diffusionkit_b200.text_encoders import clip_param_specs, t5_param_specs  # noqa: E402
from diffusionkit_b200.weights import (init_params, mmdit_param_specs, vae_decoder_param_specs,  # noqa: E402
                                       vae_encoder_param_specs)
from tests.golden import make_reference_golden as mkt  # noqa: E402
from tests.golden import make_reference_mlx_golden as mk  # noqa: E402
from tests.golden import reference_shims as rs  # noqa: E402

FULL_MAX, SAMPLE = 4096, 1024      # arrays over FULL_MAX elements are stored as a SAMPLE of values + row sums


def digest(t: torch.Tensor):
    """[shape, 64-bit sha256 prefix of the float32 bytes]: exact equality of two tensors without storing them"""
    a = np.ascontiguousarray(t.detach().to(torch.float32).numpy())
    return [list(a.shape), hashlib.sha256(a.tobytes()).hexdigest()[:16]]


def sample_index(shape):
    """the fixed positions (in the flattened array) stored for a large array"""
    n = int(np.prod(shape))
    return np.sort(np.random.RandomState(0).choice(n, min(n, SAMPLE), replace=False))


def shrink(arrays):
    """what is stored for each array: itself, or <name>_shape, <name>_sample and <name>_sums (float64 sums over the
    last axis) when it has more than FULL_MAX elements"""
    out = {}
    for name, a in arrays.items():
        if a.size <= FULL_MAX:
            out[name] = np.ascontiguousarray(a)
        else:
            out[name + "_shape"] = np.asarray(a.shape, dtype=np.int64)
            out[name + "_sample"] = a.reshape(-1)[sample_index(a.shape)]
            out[name + "_sums"] = a.astype(np.float64).sum(-1)
    return out


def assert_close(g, name, got, atol, rtol):
    """got (a tensor) against the stored reference array `name`: elementwise when stored whole; else the shape, the
    sampled values elementwise and the row sums (to atol * sqrt(row length), as for independent elementwise errors)"""
    got = got.detach().to(torch.float32).numpy()
    if name in g:
        want = g[name]
        assert got.shape == want.shape, (name, got.shape, want.shape)
        assert np.allclose(got, want, atol=atol, rtol=rtol), (name, float(np.abs(got - want).max()))
        return
    assert list(got.shape) == g[name + "_shape"].tolist(), (name, got.shape)
    got_s, want_s = got.reshape(-1)[sample_index(got.shape)], g[name + "_sample"]
    assert np.allclose(got_s, want_s, atol=atol, rtol=rtol), (name, float(np.abs(got_s - want_s).max()))
    sums, want_sums = got.astype(np.float64).sum(-1), g[name + "_sums"]
    assert np.allclose(sums, want_sums, atol=atol * got.shape[-1] ** 0.5, rtol=rtol), \
        (name, float(np.abs(sums - want_sums).max()))


# ------------------------------------------------------------------------------------------------ seeded inputs
def torch_loader_checkpoints():
    """upstream-layout checkpoints (Stability SD3 MMDiT, LDM VAE decoder) of the pin configs"""
    from tests.test_model_io_cpu import _sd3_upstream, _vae_upstream

    cfg = mkt.pin_mmdit_config()
    upstream = _sd3_upstream(init_params(mmdit_param_specs(cfg), seed=31, dtype=torch.float32), cfg)
    for k in list(upstream):                        # a real checkpoint has a k bias; both loaders must drop it
        if k.endswith("attn.qkv.bias"):
            upstream[k] = upstream[k] + 0.3
    vparams = init_params(vae_decoder_param_specs(mkt.pin_vae_config()), seed=32, dtype=torch.float32)
    return upstream, _vae_upstream(vparams, prefix="first_stage_model.decoder.")


def psnr_inputs():
    rng = np.random.RandomState(0)
    a = rng.randn(3, 8, 8).astype(np.float32)
    return a, a + 0.01 * rng.randn(3, 8, 8).astype(np.float32)


def text_encoder_cases():
    """(name, config, params, tokens) of the CLIP cases, then the T5 case"""
    clip = []
    for act, proj in (("quick_gelu", True), ("gelu", False)):
        cfg = tiny_clip_config(projection=proj, act=act)
        params = init_params(clip_param_specs(cfg), seed=71, dtype=torch.float32)
        tokens = torch.randint(1, cfg.vocab_size - 1, (2, 24), generator=torch.Generator().manual_seed(5))
        tokens[0, 9] = tokens[1, 23] = cfg.vocab_size - 1
        clip.append((f"clip_{act}", cfg, params, tokens))
    tc = tiny_t5_config()
    tparams = init_params(t5_param_specs(tc), seed=72, dtype=torch.float32)
    tparams["encoder.relative_attention_bias.embeddings.weight"] *= 30.0
    tparams["wte.weight"] *= 30.0
    tokens = torch.randint(0, tc.vocab_size, (2, 160), generator=torch.Generator().manual_seed(6))
    return clip, (tc, tparams, tokens)


def exact_params(specs, salt: int):
    """RNG-free parameters for the bit-exact key-map pins: integers below 2^24 (exact in float32, so the same on every
    CPU, unlike torch.randn whose CPU kernels differ in the last bits between instruction sets), distinct within a tensor
    and offset per tensor, so a tensor or slice put in the wrong place cannot match"""
    out = {}
    for i, (name, shape, _) in enumerate(specs):
        n = int(np.prod(shape))
        v = (torch.arange(n, dtype=torch.int64) * 7 + (salt * 1009 + i) * 7919) % (1 << 24)
        out[name] = v.to(torch.float32).reshape(shape)
    return out


def key_map_checkpoints():
    """upstream-layout checkpoints for the MLX loaders: BFL FLUX, Stability SD3, LDM VAE decoder / encoder, HF T5"""
    from tests.test_model_io_cpu import _flux_upstream, _sd3_upstream, _vae_upstream

    flux, sd3 = mk.pin_configs()
    out = {"flux": _flux_upstream(exact_params(mmdit_param_specs(flux), 81), flux),
           "sd3": _sd3_upstream(exact_params(mmdit_param_specs(sd3), 82), sd3),
           "vae_decoder": _vae_upstream(exact_params(vae_decoder_param_specs(VAEDecoderConfig()), 83),
                                        prefix="first_stage_model.decoder."),
           "vae_encoder": _vae_upstream(exact_params(vae_encoder_param_specs(VAEEncoderConfig()), 84),
                                        prefix="first_stage_model.encoder.")}
    tc = tiny_t5_config()
    hf = {}
    for k, v in exact_params(t5_param_specs(tc), 85).items():
        if k == "wte.weight":
            hf["encoder.embed_tokens.weight"] = v
            hf["shared.weight"] = v
        elif k == "encoder.ln.weight":
            hf["encoder.final_layer_norm.weight"] = v
        elif k == "encoder.relative_attention_bias.embeddings.weight":
            hf["encoder.block.0.layer.0.SelfAttention.relative_attention_bias.weight"] = v
        else:
            i, rest = k.split(".")[2], ".".join(k.split(".")[3:])
            rest = (rest.replace("attention.query_proj", "layer.0.SelfAttention.q")
                    .replace("attention.key_proj", "layer.0.SelfAttention.k")
                    .replace("attention.value_proj", "layer.0.SelfAttention.v")
                    .replace("attention.out_proj", "layer.0.SelfAttention.o").replace("ln1", "layer.0.layer_norm")
                    .replace("ln2", "layer.1.layer_norm").replace("dense.", "layer.1.DenseReluDense."))
            hf[f"encoder.block.{i}.{rest}"] = v
    out["t5"] = hf
    return out


TOKENIZER_TEXTS = ["a photo of a cat", "The  astronaut riding a horse on Mars!!", "cats, cats , 42 cats!", "a",
                   " ".join(["cat"] * 200)]


class WordTokenizer:
    """minimal object with the interface the pipelines' _tokenize uses (tokenize / max_length / pad flags / eos_token)"""

    def __init__(self, max_length, pad_with_eos, eos=99, bos=None, vocab_size=100):
        self.max_length, self.pad_with_eos, self.pad_to_max_length = max_length, pad_with_eos, True
        self.eos_token, self._bos, self._v = eos, bos, vocab_size

    def tokenize(self, text):
        ids = [1 + (sum(map(ord, w)) % (self._v - 3)) for w in text.split()][: self.max_length - 2]
        return ([self._bos] if self._bos is not None else []) + ids + [self.eos_token]


def encode_text_setup():
    """encoders, tokenizers and prompts of the encode_text composition case; T5 lengths per pipeline kind"""
    cl = CLIPTextModelConfig(num_layers=2, model_dims=128, num_heads=2, vocab_size=100, projection_dim=None)
    cg = CLIPTextModelConfig(num_layers=2, model_dims=192, num_heads=3, vocab_size=100, projection_dim=192,
                             hidden_act="gelu")
    tc = T5EncoderConfig(vocab_size=100, d_model=4096, d_kv=64, d_ff=128, num_layers=1, num_heads=2)
    pl = init_params(clip_param_specs(cl), seed=91, dtype=torch.float32)
    pg = init_params(clip_param_specs(cg), seed=92, dtype=torch.float32)
    pt = init_params(t5_param_specs(tc), seed=93, dtype=torch.float32)
    pt["wte.weight"] *= 30.0
    return dict(cl=cl, cg=cg, tc=tc, pl=pl, pg=pg, pt=pt, tok_l=WordTokenizer(77, True, bos=98),
                tok_g=WordTokenizer(77, False, bos=98), t5_len={"sd3": 64, "flux": 48},
                text="a photo of an astronaut riding a horse on mars", neg="blurry low quality")


def img2img_image():
    """100 x 150 RGB, not a multiple of 64: read_image resizes it to 64 x 128"""
    return (np.random.RandomState(3).rand(100, 150, 3) * 255).astype(np.uint8)


IMG2IMG = {"steps": 4, "denoise": 0.5, "seed": 9}


# ------------------------------------------------------------------------------------------------ the reference side
def run_torch_loaders(arrays):
    """SD3 MMDiT and VAE decoder: upstream checkpoint -> the reference's own key adjustments (torch/mmdit.py:424-497,
    torch/model_io.py:90-122) -> the reference modules, strict=True"""
    m, v, mio = rs.load_reference_module("mmdit"), rs.load_reference_module("vae"), rs.load_reference_module("model_io")
    latent, text, pooled, timestep, z = mkt.make_inputs()
    upstream, vup = torch_loader_checkpoints()
    cfg = mkt.pin_mmdit_config()
    # the reference loader's own prefix rule (torch/model_io.py:67-71): drop "model.diffusion_model", skip the VAE
    stripped = {".".join(k.rsplit(".")[2:]): t for k, t in upstream.items()
                if all(s not in k for s in ["encoder", "decoder"])}
    rcfg = m.MMDiTConfig(depth=cfg.depth_multimodal, max_latent_resolution=cfg.max_latent_resolution,
                         pooled_text_embed_dim=cfg.pooled_text_embed_dim,
                         token_level_text_embed_dim=cfg.token_level_text_embed_dim)
    net = m.MMDiT(rcfg).eval()
    net.load_state_dict(m.mmdit_state_dict_adjustments(stripped), strict=True)
    with torch.no_grad():
        (want,) = net(latent.permute(0, 3, 1, 2).contiguous(), text.permute(0, 2, 1)[:, :, None, :].contiguous(),
                      pooled[:, :, None, None], timestep)
    arrays["torch_loader_mmdit"] = want.permute(0, 2, 3, 1).numpy()
    vcfg = mkt.pin_vae_config()
    boc = vcfg.block_out_channels
    vnet = v.VAEDecoder(v.VAEDecoderConfig(resolution=z.shape[1] * 8, base_channels=boc[0],
                                           channel_multipliers=[c // boc[0] for c in boc],
                                           num_res_blocks=vcfg.layers_per_block - 1)).eval()
    vnet.load_state_dict(mio.vae_decoder_state_dict_adjustments(dict(vup)), strict=True)
    with torch.no_grad():
        arrays["torch_loader_vae"] = vnet(z.permute(0, 3, 1, 2).contiguous()).permute(0, 2, 3, 1).numpy()


def run_psnr():
    """diffusionkit/utils.py:70-82"""
    rs.install()
    spec = importlib.util.spec_from_file_location("_reference_utils",
                                                  os.path.join(rs.REFERENCE_SRC, "diffusionkit", "utils.py"))
    utils = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(utils)
    return float(utils.compute_psnr(*psnr_inputs()))


def run_mlx_16bit_mmdit(arrays):
    """the FLUX pin MMDiT with bf16 weights and activations (bf16 sinusoid: quirk Q5; per-op rounding)"""
    rcfg_mod, rmm = mk.load_reference_mlx("config"), mk.load_reference_mlx("mmdit")
    mx = sys.modules["mlx.core"]
    flux, _ = mk.pin_configs()
    cfg16 = replace(flux, dtype=torch.bfloat16, float16_dtype=torch.bfloat16)
    params = init_params(mmdit_param_specs(cfg16), seed=mk.SEEDS["flux"], dtype=torch.float32)
    p16 = {k: v.to(torch.bfloat16) for k, v in params.items()}
    rc = mk.reference_config(rcfg_mod, cfg16)
    rc.dtype = rc.float16_dtype = mx.bfloat16
    model = rmm.MMDiT(rc)
    model.load_weights([(k, mx.array(v.clone())) for k, v in p16.items()], strict=True)
    latent, text, pooled, timesteps, ti = mk.make_inputs("flux")
    l16, t16, pl16 = [x.to(torch.bfloat16) for x in (latent, text, pooled)]
    ts16 = timesteps.to(torch.bfloat16)
    model.cache_modulation_params(mx.array(pl16.clone()), mx.array(ts16.clone()))
    out = model(latent_image_embeddings=mx.array(l16.clone()),
                token_level_text_embeddings=mx.array(t16.clone()[:, :, None, :]),
                timestep=mx.repeat(mx.array(ts16.clone())[ti][None], 2, axis=0)).t.float()
    arrays["mlx_16bit_flux_mmdit"] = out.numpy()


def run_mlx_pipeline_iterations():
    out = {}
    for kind, (steps, cfgw, shift, lat, seed, _) in mk.PIPELINE_CASES.items():
        cond, pooled = mk.make_pipeline_inputs(kind)
        latent, _, _, n_iter = mk.run_reference_pipeline(kind, cond, pooled, steps, cfgw, shift, lat, seed)
        g = np.load(os.path.join(HERE, f"reference_mlxsrc_{kind}_pipeline.npz"))
        assert np.allclose(latent.numpy(), g["latent"], atol=1e-5), f"reference_mlxsrc_{kind}_pipeline.npz is stale"
        out[kind] = n_iter
    return out


def run_mlx_text_encoders(arrays):
    """CLIPTextModel (mlx/clip.py) and SD3T5Encoder (mlx/t5.py)"""
    from transformers import T5Config

    mk.load_reference_pipeline_package()
    mx = sys.modules["mlx.core"]
    from diffusionkit.mlx import clip as rclip, config as rcfg, t5 as rt5

    clip, (tc, tparams, ttokens) = text_encoder_cases()
    for name, cfg, params, tokens in clip:
        model = rclip.CLIPTextModel(rcfg.CLIPTextModelConfig(
            num_layers=cfg.num_layers, model_dims=cfg.model_dims, num_heads=cfg.num_heads, max_length=cfg.max_length,
            vocab_size=cfg.vocab_size, projection_dim=cfg.projection_dim, hidden_act=cfg.hidden_act))
        model.load_weights(mk.to_mx(params), strict=True)
        out = model(mx.array(tokens.to(torch.int32)))
        arrays[f"{name}_last"] = out.last_hidden_state.t.numpy()
        arrays[f"{name}_pooled"] = out.pooled_output.t.numpy()
        arrays[f"{name}_hidden_m2"] = out.hidden_states[-2].t.numpy()
    hf_cfg = T5Config(vocab_size=tc.vocab_size, d_model=tc.d_model, d_kv=tc.d_kv, d_ff=tc.d_ff, num_layers=tc.num_layers,
                      num_heads=tc.num_heads, feed_forward_proj="gated-gelu", relative_attention_num_buckets=32,
                      relative_attention_max_distance=128, layer_norm_epsilon=1e-6)
    enc = rt5.SD3T5Encoder(hf_cfg, low_memory_mode=False)
    enc.load_weights(mk.to_mx(tparams), strict=True)
    arrays["t5_out"] = enc(mx.array(ttokens.to(torch.int32))).t.numpy()


def run_mlx_key_maps():
    """the reference's *_state_dict_adjustments (mlx/model_io.py:130-636): per resulting key, shape + digest"""
    dm = mk.load_reference_pipeline_package()
    mx = sys.modules["mlx.core"]
    rio = dm.model_io
    flux, _ = mk.pin_configs()
    ck = key_map_checkpoints()

    def as_mx(d):
        return {k: mx.array(v.clone()) for k, v in d.items()}

    def digests(d):
        return {k: digest(v.t) for k, v in d.items()}

    ref_flux = rio.flux_state_dict_adjustments(as_mx(ck["flux"]), prefix="", hidden_size=flux.hidden_size,
                                               mlp_ratio=flux.mlp_ratio)
    # the reference loads FLUX with Module.update (model_io.py:776), which ignores keys its module tree does not have
    # (k_proj.bias: quirk Q3; guidance_in.*: quirk Q1): what ends up in the model is what the product must produce
    from diffusionkit.mlx import config as rcfg_mod, mmdit as rmm
    from mlx.utils import tree_flatten, tree_unflatten

    model = rmm.MMDiT(mk.reference_config(rcfg_mod, flux))
    untouched = {k for k, _ in tree_flatten(model.parameters())}
    model.update(tree_unflatten(list(ref_flux.items())))
    effective = dict(tree_flatten(model.parameters()))
    assert set(effective) == untouched                       # update added nothing
    assert any(k.endswith("k_proj.bias") for k in ref_flux) and not any(k.endswith("k_proj.bias") for k in effective)
    return {"flux": digests(effective),
            "sd3": digests(rio.mmdit_state_dict_adjustments(as_mx(ck["sd3"]), prefix="model.diffusion_model.")),
            "vae_decoder": digests(rio.vae_decoder_state_dict_adjustments(as_mx(ck["vae_decoder"]),
                                                                          prefix="first_stage_model.decoder.")),
            "vae_encoder": digests(rio.vae_encoder_state_dict_adjustments(as_mx(ck["vae_encoder"]),
                                                                          prefix="first_stage_model.encoder.")),
            "t5": digests(rio.t5_encoder_state_dict_adjustments(as_mx(ck["t5"]), prefix=""))}


def run_mlx_tokenizer():
    """mlx/tokenizer.py:14-122 on the synthetic vocabulary of tests/test_text_cpu.py"""
    import pathlib

    from diffusionkit_b200.tokenizer import load_tokenizer
    from tests.test_text_cpu import _synthetic_clip_vocab

    mk.load_reference_pipeline_package()
    from diffusionkit.mlx import tokenizer as rtok

    with tempfile.TemporaryDirectory() as d:
        vf, mf, _ = _synthetic_clip_vocab(pathlib.Path(d))
        mine = load_tokenizer(vf, mf, pad_with_eos=True)
    ref = rtok.Tokenizer(mine.bpe_ranks, mine.vocab, pad_with_eos=True)
    return {"tokens": [[int(t) for t in ref.tokenize(text)] for text in TOKENIZER_TEXTS],
            "eos_token": int(ref.eos_token), "bos_token": int(ref.bos_token)}


def run_mlx_encode_text(arrays):
    """_tokenize / encode_text of both pipelines (mlx/__init__.py:174-251, 642-671): token batches, conditioning, pooled"""
    from transformers import T5Config

    dm = mk.load_reference_pipeline_package()
    from diffusionkit.mlx import clip as rclip, config as rcfg, t5 as rt5

    s = encode_text_setup()
    tc = s["tc"]

    def ref_clip(c, p):
        m = rclip.CLIPTextModel(rcfg.CLIPTextModelConfig(num_layers=c.num_layers, model_dims=c.model_dims,
                                                         num_heads=c.num_heads, max_length=c.max_length,
                                                         vocab_size=c.vocab_size, projection_dim=c.projection_dim,
                                                         hidden_act=c.hidden_act))
        m.load_weights(mk.to_mx(p), strict=True)
        return m

    t5 = rt5.SD3T5Encoder(T5Config(vocab_size=tc.vocab_size, d_model=tc.d_model, d_kv=tc.d_kv, d_ff=tc.d_ff,
                                   num_layers=tc.num_layers, num_heads=tc.num_heads, feed_forward_proj="gated-gelu",
                                   relative_attention_num_buckets=32, relative_attention_max_distance=128,
                                   layer_norm_epsilon=1e-6), low_memory_mode=False)
    t5.load_weights(mk.to_mx(s["pt"]), strict=True)
    tokens = {}
    for kind in ("sd3", "flux"):
        pipe = object.__new__(dm.DiffusionPipeline if kind == "sd3" else dm.FluxPipeline)
        pipe.clip_l, pipe.clip_g, pipe.t5_encoder = ref_clip(s["cl"], s["pl"]), ref_clip(s["cg"], s["pg"]), t5
        pipe.tokenizer_l, pipe.tokenizer_g = s["tok_l"], s["tok_g"]
        pipe.t5_tokenizer = WordTokenizer(s["t5_len"][kind], False, eos=1)
        pipe.use_t5 = True
        pipe.model_version = "pin"
        dm.T5_MAX_LENGTH["pin"] = s["t5_len"][kind]
        for cfgw in (5.0, 0.0):
            n = s["neg"] if cfgw > 1 else None
            case = f"{kind}_cfg{int(cfgw)}"
            tokens[case] = [pipe._tokenize(tk, s["text"], n).tolist()
                            for tk in (s["tok_l"], s["tok_g"], pipe.t5_tokenizer)]
            cond, pooled = pipe.encode_text(s["text"], cfgw, s["neg"])
            arrays[f"encode_text_{case}_cond"] = cond.t.numpy()
            arrays[f"encode_text_{case}_pooled"] = pooled.t.numpy()
    return tokens


def run_mlx_img2img(arrays):
    """image_path / denoise (mlx/__init__.py:270-285, 536-551, 586-594) through the reference FluxPipeline"""
    from PIL import Image

    dm = mk.load_reference_pipeline_package()
    mx = sys.modules["mlx.core"]
    from diffusionkit.mlx import config as rcfg_mod, mmdit as rmm, vae as rvae

    flux, _ = mk.pin_configs()
    params = init_params(mmdit_param_specs(flux), seed=mk.SEEDS["flux"], dtype=torch.float32)
    ecfg = VAEEncoderConfig(block_out_channels=(32, 64, 64, 64), layers_per_block=2)
    eparams = init_params(vae_encoder_param_specs(ecfg), seed=mk.SEEDS["vae_enc"], dtype=torch.float32)
    pipe = object.__new__(dm.FluxPipeline)
    pipe.mmdit = rmm.MMDiT(mk.reference_config(rcfg_mod, flux))
    pipe.mmdit.load_weights(mk.to_mx(params), strict=True)
    pipe.encoder = rvae.VAEEncoder(in_channels=3, out_channels=32, block_out_channels=list(ecfg.block_out_channels),
                                   layers_per_block=ecfg.layers_per_block, resnet_groups=32)
    pipe.encoder.load_weights(mk.to_mx(eparams), strict=True)
    pipe.sampler, pipe.latent_format = dm.FluxSampler(shift=1.0), dm.FluxLatentFormat()
    pipe.activation_dtype = pipe.dtype = pipe.float16_dtype = mx.float32
    pipe.load_mmdit = lambda only_modulation_dict=False: [(k, mx.array(v.clone())) for k, v in params.items()
                                                          if "adaLN" in k]
    cond, pooled = mk.make_pipeline_inputs("flux")
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "in.png")
        Image.fromarray(img2img_image()).save(path)
        latent, iter_time = pipe.denoise_latents(mx.array(cond.clone()), mx.array(pooled.clone()),
                                                 num_steps=IMG2IMG["steps"], cfg_weight=0.0, latent_size=(2, 2),
                                                 seed=IMG2IMG["seed"], image_path=path, denoise=IMG2IMG["denoise"])
        arrays["img2img_read_image"] = pipe.read_image(path).t.numpy()
    arrays["img2img_latent"] = latent.t.numpy()
    return len(iter_time)


def run_mlx_16bit_pipelines(arrays):
    """the denoise loop with real 16-bit arrays (bf16 FLUX / fp16 SD3: timestep rounding and the config.dtype
    sinusoid of quirk Q5, the rounding residue of quirk Q6, per-op rounding)"""
    dm = mk.load_reference_pipeline_package()
    mx = sys.modules["mlx.core"]
    from diffusionkit.mlx import config as rcfg_mod, mmdit as rmm

    for kind in ("flux", "sd3"):
        dt = torch.bfloat16 if kind == "flux" else torch.float16
        mdt = mx.bfloat16 if kind == "flux" else mx.float16
        steps, cfgw, shift, lat, seed, _ = mk.PIPELINE_CASES[kind]
        cfg = replace(mk.pin_config(kind), dtype=dt, float16_dtype=dt)
        p16 = {k: v.to(dt) for k, v in init_params(mmdit_param_specs(cfg), seed=mk.SEEDS[kind],
                                                   dtype=torch.float32).items()}
        rc = mk.reference_config(rcfg_mod, cfg)
        rc.dtype = rc.float16_dtype = mdt
        pipe = object.__new__(dm.FluxPipeline if kind == "flux" else dm.DiffusionPipeline)
        pipe.mmdit = rmm.MMDiT(rc)
        pipe.mmdit.load_weights([(k, mx.array(v.clone())) for k, v in p16.items()], strict=True)
        pipe.sampler = (dm.FluxSampler if kind == "flux" else dm.ModelSamplingDiscreteFlow)(shift=shift)
        pipe.latent_format = (dm.FluxLatentFormat if kind == "flux" else dm.SD3LatentFormat)()
        pipe.activation_dtype = pipe.dtype = pipe.float16_dtype = mdt
        pipe.load_mmdit = lambda only_modulation_dict=False, p16=p16: [(k, mx.array(v.clone())) for k, v in p16.items()
                                                                       if "adaLN" in k]
        cond, pooled = mk.make_pipeline_inputs(kind)
        latent, _ = pipe.denoise_latents(mx.array(cond.to(dt).clone()), mx.array(pooled.to(dt).clone()),
                                         num_steps=steps, cfg_weight=cfgw, latent_size=lat, seed=seed)
        arrays[f"mlx_16bit_{kind}_pipeline_latent"] = latent.t.float().numpy()


if __name__ == "__main__":
    assert rs.reference_available() and mk.reference_mlx_available(), \
        "set DIFFUSIONKIT_REFERENCE to an argmaxinc/DiffusionKit checkout"
    arrays = {}
    run_torch_loaders(arrays)
    meta = {"psnr": run_psnr()}
    mk.load_reference_pipeline_package()
    run_mlx_16bit_mmdit(arrays)
    meta["pipeline_iterations"] = run_mlx_pipeline_iterations()
    run_mlx_text_encoders(arrays)
    meta["key_maps"] = run_mlx_key_maps()
    meta["tokenizer"] = run_mlx_tokenizer()
    meta["encode_text_tokens"] = run_mlx_encode_text(arrays)
    meta["img2img_iterations"] = run_mlx_img2img(arrays)
    run_mlx_16bit_pipelines(arrays)
    np.savez_compressed(NPZ, **dict(sorted(shrink(arrays).items())))
    with open(JSON, "w") as f:
        json.dump(meta, f, indent=0, sort_keys=True)
        f.write("\n")
    print(os.path.getsize(NPZ), os.path.getsize(JSON))
