"""-m gpu: LoRA adapters merged in place into the packed MMDiT weights — merge exactness on every window type (full
matrix, row windows of w_qkv / w_mod, column windows of w_out) against an fp64 merge of the file factors, bit-exact
state changes (unload, stacking, scale 0, reload), the denoise loop against the oracle loop on upstream-merged
weights, captured CUDA graphs reading the merged weights, the stale modulation cache and the family check."""
import os
from dataclasses import replace

import pytest
import torch

import diffusionkit_b200 as dk
from diffusionkit_b200 import model_io
from diffusionkit_b200.config import FLUX_SCHNELL, VAEDecoderConfig, tiny_flux_config, tiny_sd3_config
from diffusionkit_b200.lora import LoraMerger
from diffusionkit_b200.weights import init_params, mmdit_param_specs, vae_decoder_param_specs
from oracle import sampler_ref as sr
from oracle.lora_ref import merge_upstream
from oracle.mmdit_ref import MMDiTRef
from tests.model_checks import rel_l2
from tests.oracle_bridge import ref_config
from tests.test_model_io_cpu import _flux_upstream, _sd3_upstream

pytestmark = pytest.mark.gpu


def _route(cfg, module):
    return (model_io.flux_linear_route(module, cfg.mlp_ratio) if cfg.depth_unified > 0
            else model_io.sd3_linear_route(module))


def _upstream_weight(views, cfg, module):
    """the packed windows of an upstream Linear, reassembled in the upstream layout (a copy)"""
    dim, parts = _route(cfg, module)
    return torch.cat([views[n + ".weight"] for n, _ in parts], dim=dim).clone()


def _lora(views, cfg, spec, seed, dtype, amp=1.0):
    """spec: {module: rank} -> PEFT state dict with N(0, 1) / sqrt(fan) factors in `dtype`, alpha = 2 r on odd ranks"""
    g = torch.Generator().manual_seed(seed)
    sd = {}
    for m, r in spec.items():
        out_f, in_f = _upstream_weight(views, cfg, m).shape
        sd[m + ".lora_A.weight"] = (torch.randn((r, in_f), generator=g) / in_f ** 0.5).to(dtype)
        sd[m + ".lora_B.weight"] = (amp * torch.randn((out_f, r), generator=g) / r ** 0.5).to(dtype)
        if r % 2:
            sd[m + ".alpha"] = torch.tensor(2.0 * r)
    return sd


def _ulp(x, dtype):
    e = torch.floor(torch.log2(x.abs().clamp_min(1e-300)))
    if dtype == torch.bfloat16:
        return torch.exp2(e.clamp_min(-126) - 7)
    return torch.exp2(e.clamp_min(-14) - 10)


def _check_merge(m, cfg, adapters, w0_up):
    """every adapted upstream weight within ulp(W_ref) + c * sum |s B| |A| of the fp64 merge"""
    c = 2.0 ** -7 if m.dtype == torch.bfloat16 else 2.0 ** -10
    worst = 0.0
    for module, w0 in w0_up.items():
        ref = w0.double()
        absprod = torch.zeros_like(ref)
        for sd, scale in adapters:
            if module + ".lora_A.weight" not in sd:
                continue
            A, B = sd[module + ".lora_A.weight"].double().cuda(), sd[module + ".lora_B.weight"].double().cuda()
            r = A.shape[0]
            alpha = float(sd[module + ".alpha"]) if module + ".alpha" in sd else float(r)
            sB = scale * alpha / r * B
            ref = ref + sB @ A
            absprod = absprod + sB.abs() @ A.abs()
        got = _upstream_weight(m.weight_views, cfg, module).double()
        err = (got - ref).abs()
        bound = _ulp(ref, m.dtype) + c * absprod
        assert bool((err <= bound).all()), f"{module}: max err/bound {float((err / bound).max()):.3f}"
        worst = max(worst, float((err / bound).max()))
    return worst


TINY_SPEC_1 = {"double_blocks.0.img_attn.qkv": 1, "double_blocks.1.txt_mod.lin": 16, "single_blocks.0.linear2": 64,
               "double_blocks.0.img_mlp.0": 100, "single_blocks.1.linear1": 16, "final_layer.adaLN_modulation.1": 1,
               "img_in": 16}
TINY_SPEC_2 = {"double_blocks.0.img_attn.qkv": 16, "single_blocks.0.linear2": 100, "double_blocks.0.img_mlp.0": 1,
               "single_blocks.1.modulation.lin": 64}


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
def test_merge_exactness_tiny(cuda, dtype):
    cfg = tiny_flux_config()
    m = dk.MMDiT(cfg, {k: v.to(cuda) for k, v in init_params(mmdit_param_specs(cfg), seed=3, dtype=dtype).items()})
    a1 = _lora(m.weight_views, cfg, TINY_SPEC_1, 1, dtype)
    a2 = _lora(m.weight_views, cfg, TINY_SPEC_2, 2, dtype)
    w0 = {mod: _upstream_weight(m.weight_views, cfg, mod) for mod in set(TINY_SPEC_1) | set(TINY_SPEC_2)}
    lm = LoraMerger(m)
    info = lm.load(a1, scale=0.8)
    assert info.name == "lora0" and info.rank == 100 and info.skipped == ()
    assert info.n_targets == 3 + 1 + 2 + 1 + 4 + 1 + 1
    w1 = _check_merge(m, cfg, [(a1, 0.8)], w0)
    lm.load(a2, scale=-1.5, name="second")
    w2 = _check_merge(m, cfg, [(a1, 0.8), (a2, -1.5)], w0)
    print(f"{dtype}: worst err/bound one adapter {w1:.3f}, two stacked {w2:.3f}")


def test_merge_exactness_full_width(cuda):
    """the same windows at full FLUX width: w_qkv [9216, 3072], w_out [3072, 15360], w_mod row windows"""
    cfg = replace(FLUX_SCHNELL, depth_multimodal=1, depth_unified=1)
    dtype = torch.bfloat16
    m = dk.MMDiT(cfg, init_params(mmdit_param_specs(cfg), seed=4, dtype=dtype, device=cuda))
    assert tuple(m.single[0].w_out.shape) == (3072, 15360) and tuple(m.double[0][0].w_qkv.shape) == (9216, 3072)
    spec1 = {"double_blocks.0.img_attn.qkv": 16, "single_blocks.0.linear2": 64, "single_blocks.0.linear1": 64,
             "double_blocks.0.txt_mod.lin": 16, "single_blocks.0.modulation.lin": 1}
    spec2 = {"double_blocks.0.img_attn.qkv": 64, "single_blocks.0.linear2": 100}
    a1 = _lora(m.weight_views, cfg, spec1, 5, dtype)
    a2 = _lora(m.weight_views, cfg, spec2, 6, dtype)
    w0 = {mod: _upstream_weight(m.weight_views, cfg, mod) for mod in set(spec1) | set(spec2)}
    lm = LoraMerger(m)
    lm.load(a1, scale=1.0, name="a")
    lm.load(a2, scale=0.5, name="b")
    worst = _check_merge(m, cfg, [(a1, 1.0), (a2, 0.5)], w0)
    print(f"full width bf16: worst err/bound {worst:.3f}")


def _snapshot(m):
    return {n: v.clone() for n, v in m.weight_views.items()}


def _same(a, b):
    return all(torch.equal(a[n].view(torch.int16), b[n].view(torch.int16)) for n in a)


def test_state_changes_bit_exact(cuda):
    cfg = tiny_flux_config()
    pipe = dk.FluxPipeline(w16=True, a16=True, mmdit_config=cfg, load_decoder=False)
    m = pipe.mmdit
    full = {mod: 8 for mod in model_io.flux_linear_modules(cfg.depth_multimodal, cfg.depth_unified)}
    a = _lora(m.weight_views, cfg, full, 1, torch.bfloat16)
    b = _lora(m.weight_views, cfg, dict(TINY_SPEC_2, **{"txt_in": 4}), 2, torch.bfloat16)
    s0 = _snapshot(m)
    pipe.load_lora(b, scale=0.7, name="B")
    sb = _snapshot(m)
    assert not _same(sb, s0)
    pipe.unload_lora()
    assert _same(_snapshot(m), s0) and not pipe._lora.pristine              # restored bit for bit, copies freed
    pipe.load_lora(a, scale=1.3, name="A")
    pipe.load_lora(b, scale=0.7, name="B")
    pipe.unload_lora("A")
    assert _same(_snapshot(m), sb)                                          # = B alone
    pipe.unload_lora("B")
    pipe.load_lora(a, scale=0.0, name="A")
    assert _same(_snapshot(m), s0)                                          # scale 0 = no adapter
    pipe.load_lora(a, scale=0.5, name="A")
    sa = _snapshot(m)
    pipe.load_lora(a, scale=2.0, name="A")
    pipe.load_lora(a, scale=0.5, name="A")
    assert _same(_snapshot(m), sa)                                          # reload at a scale = fresh load at it
    pipe.unload_lora()
    pipe.load_lora(a, scale=0.5, name="A")
    assert _same(_snapshot(m), sa)
    with pytest.raises(KeyError):
        pipe.unload_lora("nope")


def _pipe(kind, graphs=True):
    if kind == "flux":
        cfg, dtype, Pipe, mv, shift = tiny_flux_config(), torch.bfloat16, dk.FluxPipeline, "argmaxinc/mlx-FLUX.1-schnell", 1.0
    else:
        cfg, dtype, Pipe, mv = tiny_sd3_config(), torch.float16, dk.DiffusionPipeline, "argmaxinc/mlx-stable-diffusion-3-medium"
        shift = 3.0
    p16 = {k: v.to(dtype) for k, v in init_params(mmdit_param_specs(cfg), seed=7, dtype=torch.float32).items()}
    vp16 = {k: v.to(dtype) for k, v in init_params(vae_decoder_param_specs(VAEDecoderConfig()), seed=8,
                                                     dtype=torch.float32).items()}
    old = os.environ.get("DK_CUDA_GRAPHS")
    os.environ["DK_CUDA_GRAPHS"] = "1" if graphs else "0"
    try:
        pipe = Pipe(w16=True, a16=True, shift=shift, model_version=mv, mmdit_config=cfg,
                    params={k: v.to("cuda") for k, v in p16.items()},
                    vae_params={k: v.to("cuda") for k, v in vp16.items()})
    finally:
        if old is None:
            del os.environ["DK_CUDA_GRAPHS"]
        else:
            os.environ["DK_CUDA_GRAPHS"] = old
    assert pipe.mmdit.use_cuda_graphs == graphs
    return pipe, cfg, dtype, p16, shift


def _full_lora(pipe, cfg, dtype, seed, rank=8):
    mods = (model_io.flux_linear_modules(cfg.depth_multimodal, cfg.depth_unified) if cfg.depth_unified > 0
            else model_io.sd3_linear_modules(cfg.depth_multimodal))
    return _lora(pipe.mmdit.weight_views, cfg, {m: rank for m in mods}, seed, dtype, amp=0.5)


@pytest.mark.parametrize("kind", ["flux", "sd3"])
def test_denoise_with_lora_vs_oracle(cuda, kind):
    pipe, cfg, dtype, p16, shift = _pipe(kind)
    steps, cfgw, T, fmt = (4, 0.0, 16, "flux") if kind == "flux" else (6, 5.0, 24, "sd3")
    seeds, H, W = [11, 12], 8, 12
    n = len(seeds)
    cond, pooled = pipe.synthetic_text_embeddings(n_images=n, text_len=T)

    def run():
        return pipe.denoise_latents(cond, pooled, num_steps=steps, cfg_weight=cfgw, latent_size=(H, W), seed=seeds)[0]

    plain = run()
    lora, scale = _full_lora(pipe, cfg, dtype, 3), 0.75
    info = pipe.load_lora(lora, scale=scale)
    assert info.n_targets == len(pipe.mmdit.weight_views) - (kind == "sd3")
    latent = run()
    moved = rel_l2(latent, plain)
    assert moved >= 0.1, f"{kind}: the adapter moved the latent by rel_l2 {moved:.3e} only"
    # oracle: merge in upstream key space (fp64), convert with model_io, run the oracle loop
    p64 = {k: v.double() for k, v in p16.items()}
    if kind == "flux":
        merged = model_io.flux_checkpoint_to_params(merge_upstream(_flux_upstream(p64, cfg), [(lora, scale)]),
                                                    cfg.hidden_size, cfg.mlp_ratio)
    else:
        pre = "model.diffusion_model."
        merged = model_io.sd3_checkpoint_to_params(merge_upstream(_sd3_upstream(p64, cfg, pre), [(lora, scale)], pre),
                                                   pre)
    merged = {k: (merged[k] if k.endswith(".weight") else p64[k]).float() for k in p16}
    sampler = sr.FluxSamplerRef(shift) if kind == "flux" else sr.ModelSamplingDiscreteFlowRef(shift)
    sig = sr.get_sigmas(sampler, steps)
    reps = 2 if cfgw > 0 else 1
    outs = []
    for i, s in enumerate(seeds):
        ref = MMDiTRef(ref_config(cfg), merged)
        idx = [i + k * n for k in range(reps)]
        x0 = sampler.noise_scaling(float(sig[0]), sr.get_noise(s, H, W), sr.get_empty_latent(H, W))
        x = sr.sample_euler(lambda xin, c, t: ref(xin, c, t), ref.cache_modulation_params, x0, sig, cond[idx].float(),
                            pooled[idx].float(), cfgw, dtype)
        outs.append(sr.process_out(x, fmt))
    r = rel_l2(latent, torch.cat(outs))
    assert r <= 5e-2, f"{kind} with LoRA: final latent rel_l2 {r:.3e} vs the oracle"
    pipe.unload_lora()
    assert torch.equal(run(), plain)
    print(f"{kind} with LoRA: latent rel_l2 vs oracle {r:.3e}; moved by the adapter {moved:.3e}")


def test_captured_graph_reads_merged_weights(cuda):
    runs = {}
    for graphs in (True, False):
        pipe, cfg, dtype, _, _ = _pipe("flux", graphs=graphs)
        cond, pooled = pipe.synthetic_text_embeddings(n_images=2, text_len=16)
        kw = dict(num_steps=4, latent_size=(8, 12), seed=[3, 4])
        if graphs:
            pipe.denoise_latents(cond, pooled, **kw)                        # captures the forward's graph
            assert all(st["graph"] is not None for st in pipe.mmdit._shapes.values())
        pipe.load_lora(_full_lora(pipe, cfg, dtype, 9), scale=1.0)
        runs[graphs] = pipe.denoise_latents(cond, pooled, **kw)[0]
    assert torch.equal(runs[True], runs[False])


def test_stale_modulation_cache_raises(cuda):
    pipe, cfg, dtype, _, _ = _pipe("flux")
    cond, pooled = pipe.synthetic_text_embeddings(n_images=1, text_len=16)
    pipe.mmdit.cache_modulation_params(pooled.to(cuda), [500.0])
    x = torch.zeros((1, 8, 12, 16), dtype=dtype, device=cuda)
    pipe.mmdit(x, cond.to(cuda), 500.0)
    pipe.load_lora(_lora(pipe.mmdit.weight_views, cfg, {"double_blocks.0.img_mod.lin": 4}, 1, dtype))
    with pytest.raises(KeyError):
        pipe.mmdit(x, cond.to(cuda), 500.0)
    pipe.mmdit.cache_modulation_params(pooled.to(cuda), [500.0])
    pipe.mmdit(x, cond.to(cuda), 500.0)
    pipe.unload_lora()
    with pytest.raises(KeyError):
        pipe.mmdit(x, cond.to(cuda), 500.0)


def test_flux_lora_on_sd3_pipeline_raises(cuda):
    flux, fcfg, fdt, _, _ = _pipe("flux")
    lora = _lora(flux.mmdit.weight_views, fcfg, {"double_blocks.0.img_attn.qkv": 4}, 1, fdt)
    sd3, *_ = _pipe("sd3")
    snap = _snapshot(sd3.mmdit)
    with pytest.raises(ValueError, match="FLUX module"):
        sd3.load_lora(lora)
    assert _same(_snapshot(sd3.mmdit), snap)
