"""-m gpu: inpainting (masked img2img) — the two kernels against their fp32 / uint8 definitions, the pipeline's masked
denoise loop against the oracle loop for tiny FLUX and tiny SD3 + CFG, the uint8 composite of generate_image, batches
of distinct edits, and the argument errors."""
import numpy as np
import pytest
import torch

import diffusionkit_b200 as dk
from diffusionkit_b200 import ops
from diffusionkit_b200.config import VAEDecoderConfig, VAEEncoderConfig, tiny_flux_config, tiny_sd3_config
from diffusionkit_b200.pipeline import load_image_u8
from diffusionkit_b200.weights import init_params, mmdit_param_specs, vae_decoder_param_specs, vae_encoder_param_specs
from oracle import sampler_ref as sr
from oracle.inpaint_ref import inpaint_masks, sample_euler_inpaint
from oracle.mmdit_ref import MMDiTRef
from oracle.vae_ref import VAEEncoderRef, encode_image_to_latents, read_image_array
from tests.model_checks import _test_image, rel_l2
from tests.oracle_bridge import ref_config

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
def test_inpaint_blend_kernel(cuda, dtype):
    """fp32 state; `dtype` only picks the 16-bit rounding of x0 / noise so both pipelines' value grids are covered"""
    g = torch.Generator().manual_seed(1)
    B, H, W, C = 3, 17, 23, 16                                   # 1173 pixels: not a multiple of any block size
    x0, noise, x = [torch.randn((B, H, W, C), generator=g).to(dtype).float().to(cuda) for _ in range(3)]
    mask = (torch.rand((B, H, W), generator=g) > 0.4).to(torch.uint8).to(cuda)
    for s in (0.75, 0.3125, 0.0):
        got = x.clone()
        ops.inpaint_blend(got, x0, noise, mask, s)
        torch.cuda.synchronize()
        keep = mask == 0
        assert torch.equal(got.view(torch.int32)[~keep], x.view(torch.int32)[~keep])     # regenerated: untouched
        want = s * noise.double() + (1.0 - s) * x0.double()
        bound = 1e-6 * (s * noise.double().abs() + (1.0 - s) * x0.double().abs()) + 1e-30
        assert bool(((got.double() - want).abs() <= bound)[keep].all())
        if s == 0.0:
            assert torch.equal(got[keep], x0[keep])
    with pytest.raises(dk.DkError):
        ops.inpaint_blend(x, x0, noise, mask[:, :, :-1].contiguous(), 0.5)


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
def test_image_post_masked_kernel(cuda, dtype):
    g = torch.Generator().manual_seed(2)
    B, H, W, Cp = 2, 24, 40, 8
    x = (torch.randn((B, H, W, Cp), generator=g) * 1.5).to(dtype).to(cuda)
    orig = torch.randint(0, 256, (B, H, W, 3), generator=g, dtype=torch.uint8).to(cuda)
    mask = (torch.rand((B, H, W), generator=g) > 0.5).to(torch.uint8).to(cuda)
    _, u8 = ops.image_post(x)
    got = ops.image_post_masked(x, orig, mask)
    torch.cuda.synchronize()
    m = mask.bool()
    assert torch.equal(got[m], u8[m]) and torch.equal(got[~m], orig[~m])


def _params(cfg, dtype):
    f = lambda specs, seed: {k: v.to(dtype) for k, v in init_params(specs, seed=seed, dtype=torch.float32).items()}
    return (f(mmdit_param_specs(cfg), 7), f(vae_decoder_param_specs(VAEDecoderConfig()), 8),
            f(vae_encoder_param_specs(VAEEncoderConfig()), 9))


def _pipe(kind):
    if kind == "flux":
        cfg, dtype, Pipe, mv, shift = tiny_flux_config(), torch.bfloat16, dk.FluxPipeline, "argmaxinc/mlx-FLUX.1-schnell", 1.0
    else:
        cfg, dtype, Pipe, mv = tiny_sd3_config(), torch.float16, dk.DiffusionPipeline, "argmaxinc/mlx-stable-diffusion-3-medium"
        shift = 3.0
    p16, vp16, ep16 = _params(cfg, dtype)
    pipe = Pipe(w16=True, a16=True, shift=shift, model_version=mv, mmdit_config=cfg,
                params={k: v.to("cuda") for k, v in p16.items()}, vae_params={k: v.to("cuda") for k, v in vp16.items()},
                vae_encoder_params={k: v.to("cuda") for k, v in ep16.items()})
    return pipe, cfg, dtype, p16, ep16, shift


def _mask(H, W):
    """a rectangle plus a thin diagonal stroke, uint8 (H, W) in {0, 255}"""
    a = np.zeros((H, W), dtype=np.uint8)
    a[H // 4:H // 2, W // 8:W // 3] = 255
    for i in range(min(H, W)):
        a[i, W - 1 - i] = 255
    return a


@pytest.mark.parametrize("kind,denoise", [("flux", 1.0), ("flux", 0.75), ("sd3", 1.0)])
def test_pipeline_inpaint_vs_oracle(cuda, kind, denoise):
    pipe, cfg, dtype, p16, ep16, shift = _pipe(kind)
    steps, cfgw, T, fmt = (4, 0.0, 16, "flux") if kind == "flux" else (6, 5.0, 24, "sd3")
    lf = pipe.latent_format
    img, mask_u8 = _test_image(64, 128), _mask(64, 128)
    H, W = 8, 16
    _, m = inpaint_masks(mask_u8, (64, 128))
    seeds = [11, 12]
    n = len(seeds)
    cond, pooled = pipe.synthetic_text_embeddings(n_images=n, text_len=T)
    latent, iter_time = pipe.denoise_latents(cond, pooled, num_steps=steps, cfg_weight=cfgw, seed=seeds,
                                             image_path=img, denoise=denoise, mask_path=mask_u8)
    assert latent.shape == (n, H, W, 16) and len(iter_time) == steps - int(steps * (1 - denoise))
    sampler = sr.FluxSamplerRef(shift) if kind == "flux" else sr.ModelSamplingDiscreteFlowRef(shift)
    sig = sr.get_sigmas(sampler, steps)[int(steps * (1 - denoise)):]
    enc_ref = VAEEncoderRef({k: v.float() for k, v in ep16.items()})
    image = read_image_array(torch.from_numpy(img))
    mt = torch.from_numpy(m)[None]
    reps = 2 if cfgw > 0 else 1
    outs = []
    for i, s in enumerate(seeds):
        ref = MMDiTRef(ref_config(cfg), {k: v.float() for k, v in p16.items()})
        noise = sr.get_noise(s, H, W)
        x_T = (encode_image_to_latents(enc_ref, image, noise) - lf.shift_factor) * lf.scale_factor   # process_in
        x0 = sampler.noise_scaling(float(sig[0]), noise, x_T)
        idx = [i + k * n for k in range(reps)]
        x = sample_euler_inpaint(lambda xin, c, t: ref(xin, c, t), ref.cache_modulation_params, x0, sig,
                                 cond[idx].float(), pooled[idx].float(), cfgw, dtype, x_T, noise, mt)
        outs.append(sr.process_out(x, fmt))
    r = rel_l2(latent, torch.cat(outs))
    assert r <= 5e-2, f"{kind} inpaint final latent rel_l2 {r:.3e}"
    # kept cells end exactly at the image's encoding whatever the prompt says
    cond2, pooled2 = pipe.synthetic_text_embeddings(n_images=n, seed=99, text_len=T)
    other, _ = pipe.denoise_latents(cond2, pooled2, num_steps=steps, cfg_weight=cfgw, seed=seeds, image_path=img,
                                    denoise=denoise, mask_path=mask_u8)
    keep = torch.from_numpy(m == 0).to(cuda)[None].expand(n, H, W)
    assert torch.equal(other[keep], latent[keep]) and not torch.equal(other[~keep], latent[~keep])
    # an all-ones mask is plain img2img, bit for bit
    ones, _ = pipe.denoise_latents(cond, pooled, num_steps=steps, cfg_weight=cfgw, seed=seeds, image_path=img,
                                   denoise=denoise, mask_path=np.full((64, 128), 255, dtype=np.uint8))
    plain, _ = pipe.denoise_latents(cond, pooled, num_steps=steps, cfg_weight=cfgw, seed=seeds, image_path=img,
                                    denoise=denoise)
    assert torch.equal(ones, plain)
    print(f"{kind} denoise={denoise}: latent rel_l2 vs oracle {r:.3e}")


def test_generate_image_composite(cuda, tmp_path):
    from PIL import Image

    pipe, cfg, dtype, *_ = _pipe("flux")
    img_path, mask_path = str(tmp_path / "in.png"), str(tmp_path / "mask.png")
    Image.fromarray(_test_image(100, 150)).save(img_path)
    Image.fromarray(_mask(100, 150)).save(mask_path)
    cond, pooled = pipe.synthetic_text_embeddings(n_images=1, text_len=16)
    out, log = pipe.generate_image("", num_steps=4, seed=5, verbose=False, conditioning=cond, pooled_conditioning=pooled,
                                   image_path=img_path, denoise=1.0, mask_path=mask_path)
    assert out.size == (128, 64) and len(log["denoising"]["iter_time"]) == 4
    orig = load_image_u8(img_path)[0][:, :, :3]
    p, _ = inpaint_masks(_mask(100, 150), (64, 128))
    u8 = np.asarray(out)
    assert np.array_equal(u8[p == 0], orig[p == 0]) and p.any() and not p.all()
    # inside the mask: the decode of the (uncomposited) latent
    lat, _ = pipe.denoise_latents(cond, pooled, num_steps=4, seed=5, image_path=img_path, mask_path=mask_path)
    dec = (pipe.decode_latents_to_image(lat)[0].cpu() * 255).to(dtype).float().to(torch.uint8).numpy()
    assert np.array_equal(u8[p == 1], dec[p == 1])
    outs, _ = pipe.generate_image("", num_steps=4, seed=[5, 6], verbose=False, conditioning=cond,
                                  pooled_conditioning=pooled, image_path=img_path, mask_path=mask_path)
    assert isinstance(outs, list) and len(outs) == 2 and all(o.size == (128, 64) for o in outs)
    assert all(np.array_equal(np.asarray(o)[p == 0], orig[p == 0]) for o in outs)


def test_batch_of_distinct_edits(cuda):
    pipe, *_ = _pipe("flux")
    imgs = [_test_image(64, 128, seed=5), _test_image(64, 128, seed=6)]
    m2 = np.zeros((64, 128), dtype=np.uint8)
    m2[8:40, 64:120] = 255
    masks = [_mask(64, 128), m2]
    seeds = [21, 22]
    cond, pooled = pipe.synthetic_text_embeddings(n_images=2, text_len=16)
    both, _ = pipe.denoise_latents(cond, pooled, num_steps=4, seed=seeds, image_path=imgs, denoise=0.75,
                                   mask_path=masks)
    alone = torch.cat([pipe.denoise_latents(cond[[i]], pooled[[i]], num_steps=4, seed=seeds[i], image_path=imgs[i],
                                            denoise=0.75, mask_path=masks[i])[0] for i in range(2)])
    r = rel_l2(both, alone)
    assert r <= 1e-3, f"batch of edits vs one at a time rel_l2 {r:.3e}"
    print(f"batch of 2 edits vs one at a time: rel_l2 {r:.3e}, bitwise {torch.equal(both, alone)}")
    # plain img2img with a list of images, same rule
    both, _ = pipe.denoise_latents(cond, pooled, num_steps=4, seed=seeds, image_path=imgs, denoise=0.75)
    alone = torch.cat([pipe.denoise_latents(cond[[i]], pooled[[i]], num_steps=4, seed=seeds[i], image_path=imgs[i],
                                            denoise=0.75)[0] for i in range(2)])
    r = rel_l2(both, alone)
    assert r <= 1e-3, f"img2img batch of images vs one at a time rel_l2 {r:.3e}"
    print(f"img2img batch of 2 images vs one at a time: rel_l2 {r:.3e}, bitwise {torch.equal(both, alone)}")


def test_inpaint_argument_errors_on_the_pipeline(cuda):
    pipe, *_ = _pipe("flux")
    cond, pooled = pipe.synthetic_text_embeddings(n_images=2, text_len=16)
    img, mask = _test_image(100, 150), _mask(100, 150)
    calls = [
        dict(image_path=None, mask_path=mask),                                  # a mask without an image
        dict(image_path=img, mask_path=_mask(64, 128)),                         # mask size != image's original size
        dict(image_path=[img, img, img], mask_path=mask),                       # list length != number of seeds
        dict(image_path=img, mask_path=[mask]),
        dict(image_path=[img, _test_image(64, 64)], mask_path=None),            # list images of different sizes
    ]
    for kw in calls:
        with pytest.raises(ValueError):
            pipe.denoise_latents(cond, pooled, num_steps=2, seed=[1, 2], **kw)
        with pytest.raises(ValueError):
            pipe.generate_image("", num_steps=2, seed=[1, 2], verbose=False, conditioning=cond,
                                pooled_conditioning=pooled, **kw)
