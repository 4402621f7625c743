"""Inpainting (masked img2img) host logic and oracle loop, no device needed: the product's mask preparation against the
oracle's numpy restatement, the oracle loop's two limits (all-ones mask = img2img, all-zeros mask = the image), and
the argument errors raised before anything reaches the GPU."""
import numpy as np
import pytest
import torch
from PIL import Image

from diffusionkit_b200.config import tiny_flux_config
from diffusionkit_b200.pipeline import prepare_image_inputs, prepare_inpaint_mask
from diffusionkit_b200.weights import init_params, mmdit_param_specs
from oracle import sampler_ref as sr
from oracle.mmdit_ref import MMDiTRef
from oracle.inpaint_ref import inpaint_masks, sample_euler_inpaint
from tests.oracle_bridge import ref_config


def _both(mask, size_wh):
    """product (PIL) and oracle (numpy) masks of the same input; asserts they agree"""
    p, m = prepare_inpaint_mask(mask, size_wh)
    W, H = (d - d % 64 for d in size_wh)
    po, mo = inpaint_masks(np.asarray(mask), (H, W))
    assert p.dtype == m.dtype == np.uint8 and p.shape == (H, W) and m.shape == (H // 8, W // 8)
    assert np.array_equal(p, po) and np.array_equal(m, mo)
    return p, m


def test_one_pixel_stroke_sets_exactly_the_cells_it_touches():
    a = np.zeros((64, 128), dtype=np.uint8)
    a[5:60, 37] = 255                            # vertical 1-pixel stroke in latent column 4
    a[20, 64:100] = 200                          # horizontal stroke across latent columns 8..12 of latent row 2
    p, m = _both(a, (128, 64))
    assert np.array_equal(p, (a >= 128).astype(np.uint8))
    want = np.zeros((8, 16), dtype=np.uint8)
    want[0:8, 4] = 1                             # rows 5..59 touch latent rows 0..7
    want[2, 8:13] = 1                            # columns 64..99 touch latent columns 8..12
    assert np.array_equal(m, want)


@pytest.mark.parametrize("mode", ["L", "RGB", "RGBA"])
def test_greyscale_conversion_of_each_input_kind(mode, tmp_path):
    rng = np.random.RandomState(3)
    shape = {"L": (64, 64), "RGB": (64, 64, 3), "RGBA": (64, 64, 4)}[mode]
    a = rng.randint(0, 256, shape, dtype=np.uint8)
    p, _ = _both(a, (64, 64))
    assert np.array_equal(p, (np.asarray(Image.fromarray(a).convert("L")) >= 128).astype(np.uint8))
    path = str(tmp_path / f"mask_{mode}.png")
    Image.fromarray(a).save(path)                # the same mask as a file and as a PIL image
    for kind in (path, Image.open(path)):
        q, _ = prepare_inpaint_mask(kind, (64, 64))
        assert np.array_equal(q, p)


def test_threshold_is_128():
    a = np.full((64, 64), 127, dtype=np.uint8)
    a[:, 32:] = 128
    p, m = _both(a, (64, 64))
    assert not p[:, :32].any() and p[:, 32:].all()
    assert not m[:, :4].any() and m[:, 4:].all()


def test_mask_resizes_with_the_image():
    rng = np.random.RandomState(4)
    a = (rng.rand(100, 150) > 0.7).astype(np.uint8) * 255
    p, m = _both(a, (150, 100))                  # 100 x 150 -> 64 x 128, like read_image's image
    assert p.shape == (64, 128) and m.shape == (8, 16)
    assert np.array_equal(p, (np.asarray(Image.fromarray(a).resize((128, 64), Image.NEAREST)) >= 128).astype(np.uint8))


def _oracle_img2img(mask, steps=4, denoise=0.75, seed=11):
    """the oracle img2img loop of one tiny FLUX image; with a mask, the inpainting blend runs after every step"""
    cfg = tiny_flux_config()
    p = init_params(mmdit_param_specs(cfg), seed=7, dtype=torch.float32)
    ref = MMDiTRef(ref_config(cfg), p)
    H, W = 8, 16
    g = torch.Generator().manual_seed(2)
    cond = torch.randn((1, 16, cfg.token_level_text_embed_dim), generator=g)
    pooled = torch.randn((1, cfg.pooled_text_embed_dim), generator=g)
    x_T = torch.randn((1, H, W, 16), generator=g)            # stands in for process_in(encoded image)
    sampler = sr.FluxSamplerRef(1.0)
    sig = sr.get_sigmas(sampler, steps)[int(steps * (1 - denoise)):]
    noise = sr.get_noise(seed, H, W)
    x0 = sampler.noise_scaling(float(sig[0]), noise, x_T)
    args = (lambda xin, c, t: ref(xin, c, t), ref.cache_modulation_params, x0, sig, cond, pooled, 0.0, torch.bfloat16)
    x = sr.sample_euler(*args) if mask is None else sample_euler_inpaint(*args, x_T, noise, mask)
    return x, x_T


def test_oracle_all_ones_mask_is_img2img():
    plain, _ = _oracle_img2img(None)
    ones, _ = _oracle_img2img(torch.ones((1, 8, 16), dtype=torch.uint8))
    assert torch.equal(ones, plain)


def test_oracle_all_zeros_mask_ends_at_the_image():
    zeros, x_T = _oracle_img2img(torch.zeros((1, 8, 16), dtype=torch.uint8), denoise=1.0)
    assert torch.equal(zeros, x_T)
    m = torch.zeros((1, 8, 16), dtype=torch.uint8)
    m[:, 2:6, 3:9] = 1
    part, _ = _oracle_img2img(m, denoise=1.0)
    keep = ~m.bool()
    assert torch.equal(part[keep], x_T[keep]) and not torch.equal(part[~keep], x_T[~keep])


def test_inpaint_argument_errors():
    img = np.zeros((100, 150, 3), dtype=np.uint8)
    with pytest.raises(ValueError, match="needs an image_path"):
        prepare_image_inputs(None, np.zeros((100, 150), dtype=np.uint8), 1)
    with pytest.raises(ValueError, match="same original size"):
        prepare_image_inputs(img, np.zeros((64, 128), dtype=np.uint8), 1)     # the image's resized size is not enough
    with pytest.raises(ValueError, match="one per seed"):
        prepare_image_inputs([img, img], None, 3)
    with pytest.raises(ValueError, match="one per seed"):
        prepare_image_inputs(img, [np.zeros((100, 150), dtype=np.uint8)] * 3, 2)
    with pytest.raises(ValueError, match="different sizes"):
        prepare_image_inputs([img, np.zeros((64, 64, 3), dtype=np.uint8)], None, 2)
    with pytest.raises(ValueError, match="mask array"):
        prepare_image_inputs(img, np.zeros((100, 150), dtype=np.float32), 1)
    # what is accepted: one shared image and mask, per-seed lists, and plain img2img (no mask)
    src = prepare_image_inputs(img, np.zeros((100, 150), dtype=np.uint8), 3)
    assert src.images.shape == (1, 64, 128, 3) and src.pixel_mask.shape == (3, 64, 128)
    assert src.latent_mask.shape == (3, 8, 16)
    src = prepare_image_inputs([img, img + 1], [np.zeros((100, 150), dtype=np.uint8)] * 2, 2)
    assert src.images.shape == (2, 64, 128, 3) and src.latent_mask.shape == (2, 8, 16)
    src = prepare_image_inputs(img, None, 2)
    assert src.images.shape == (1, 64, 128, 3) and src.pixel_mask is None and src.latent_mask is None
    assert prepare_image_inputs(None, None, 2) is None
