"""DiffusionPipeline / FluxPipeline — the reference's Python surface (python/src/diffusionkit/mlx/__init__.py:64-788)
over the B200 engine.  Same constructor arguments, method names, defaults and return structures; the denoise loop and
the decode run entirely in the CUDA kernels of libdkb200.so.

Differences that are deliberate (documented in DESIGN.md):
  * 16-bit only (w16 = a16 = True, what the reference CLI forces, scripts/generate_images.py:117-118);
    fp32 weights/activations raise NotImplementedError.
  * nothing is downloaded (the reference pulls checkpoints, text encoders and vocabularies from the Hugging Face hub in
    its constructor): weights are the deterministic synthetic initialiser of weights.py unless a `params` dict
    (reference parameter names) or `local_ckpt=` (upstream .safetensors, model_io.py) is passed, and `encode_text` works
    once `load_text_encoders(...)` has attached CLIP / T5 weights and tokenizers built from local files — otherwise pass
    `conditioning` / `pooled_conditioning` to generate_image or call denoise_latents.
  * img2img (`image_path`, `denoise`): the VAE encoder is built on first use.
  * batch-N extension: `seed` may be a list of ints — one independent image per seed (the reference is batch 1);
    a scalar seed behaves exactly like the reference.  `image_path` may then be a list too, one image per seed.
  * inpainting extension (`mask_path`, the reference has none): latent-blend inpainting on the img2img flow.  After
    every Euler step the latent cells outside the mask are reset to sigma_next * noise + (1 - sigma_next) * x_T
    (dk_inpaint_blend), and generate_image restores the pixels outside the mask from the input image in uint8
    (dk_image_post_masked).  A call without a mask launches exactly what it did before.
  * LoRA extension (`load_lora` / `unload_lora`, lora.py; the reference has none): adapters keyed by the upstream
    module names are merged in place into the packed MMDiT weights with dk_gemm's residual epilogue, so the denoise
    loop runs the same kernels and captured graphs.  A pipeline without an adapter launches exactly what it did before.
"""
from __future__ import annotations

import math
import time
from typing import Dict, List, NamedTuple, Optional, Sequence, Tuple, Union

import numpy as np
import torch

from . import ops
from ._lib import DkError
from .config import MODEL_CONFIGS, T5_MAX_LENGTH, MMDiTConfig, VAEDecoderConfig, VAEEncoderConfig
from .mmdit import MMDiT
from .sampler import FluxSampler, ModelSamplingDiscreteFlow
from .vae import VAEDecoder, VAEEncoder
from .weights import init_params, mmdit_param_specs, vae_decoder_param_specs, vae_encoder_param_specs

MMDIT_CKPT = {  # reference mlx/__init__.py:37-44
    "argmaxinc/mlx-stable-diffusion-3-medium": "argmaxinc/mlx-stable-diffusion-3-medium",
    "argmaxinc/mlx-stable-diffusion-3.5-large": "argmaxinc/mlx-stable-diffusion-3.5-large",
    "argmaxinc/mlx-stable-diffusion-3.5-large-4bit-quantized": "argmaxinc/mlx-stable-diffusion-3.5-large-4bit-quantized",
    "argmaxinc/mlx-FLUX.1-schnell": "argmaxinc/mlx-FLUX.1-schnell",
    "argmaxinc/mlx-FLUX.1-schnell-4bit-quantized": "argmaxinc/mlx-FLUX.1-schnell-4bit-quantized",
    "argmaxinc/mlx-FLUX.1-dev": "argmaxinc/mlx-FLUX.1-dev",
}


class LatentFormat:
    """Base class for latent format conversion (reference mlx/__init__.py:722-733)"""

    def __init__(self):
        self.scale_factor = 1.0
        self.shift_factor = 0.0

    def process_in(self, latent):
        return (latent - self.shift_factor) * self.scale_factor

    def process_out(self, latent):
        return (latent / self.scale_factor) + self.shift_factor


class SD3LatentFormat(LatentFormat):
    def __init__(self):
        super().__init__()
        self.scale_factor = 1.5305
        self.shift_factor = 0.0609


class FluxLatentFormat(LatentFormat):
    def __init__(self):
        super().__init__()
        self.scale_factor = 0.3611
        self.shift_factor = 0.1159


def _bytes2gigabytes(n: int) -> float:
    return n / 1024 ** 3


def _open_image(image, what: str):
    """a file path, a PIL image or a uint8 array -> PIL image"""
    from PIL import Image

    if isinstance(image, (str, bytes)) or hasattr(image, "__fspath__"):
        return Image.open(image)
    if isinstance(image, np.ndarray):
        if what == "image" and (image.dtype != np.uint8 or image.ndim != 3 or image.shape[2] < 3):
            raise ValueError("image array must be uint8 (H, W, >=3)")
        if what == "mask":
            if image.ndim == 3 and image.shape[2] == 1:
                image = image[:, :, 0]
            if image.dtype != np.uint8 or not (image.ndim == 2 or (image.ndim == 3 and image.shape[2] in (3, 4))):
                raise ValueError("mask array must be uint8 (H, W), (H, W, 1), (H, W, 3) or (H, W, 4)")
            return Image.fromarray(image)
        return Image.fromarray(image[:, :, :3])
    return image


def load_image_u8(image) -> Tuple[np.ndarray, Tuple[int, int]]:
    """read_image's resize rule (reference mlx/__init__.py:540-546) -> (uint8 (H, W, >=3) with H, W the original size
    cut down to multiples of 64 by a LANCZOS resize, original (width, height))"""
    from PIL import Image

    image = _open_image(image, "image")
    size = (image.width, image.height)
    W, H = (dim - dim % 64 for dim in size)
    if W == 0 or H == 0:
        raise ValueError(f"image {image.width}x{image.height} is smaller than 64x64")
    if W != image.width or H != image.height:
        image = image.resize((W, H), Image.LANCZOS)
    arr = np.asarray(image)
    if arr.ndim == 2:
        raise ValueError("greyscale images are not supported (the reference indexes img[:, :, :3])")
    return np.ascontiguousarray(arr), size


def prepare_inpaint_mask(mask, image_size: Tuple[int, int]) -> Tuple[np.ndarray, np.ndarray]:
    """Inpainting mask (a path, a PIL image or a uint8 array) -> (pixel mask p (H, W), latent mask m (H/8, W/8)), both
    uint8 in {0, 1}; 1 = regenerate.  image_size = (width, height) of the image the mask belongs to BEFORE read_image's
    resize; the mask must have that size and is resized with NEAREST to the image's target size.
      p = greyscale(mask) >= 128 (white = regenerate);  m[y, x] = any(p[8y:8y+8, 8x:8x+8])
    so a latent cell that touches any repainted pixel is repainted and thin strokes survive the 8x downsampling."""
    from PIL import Image

    mask = _open_image(mask, "mask")
    if (mask.width, mask.height) != tuple(image_size):
        raise ValueError(f"mask is {mask.width}x{mask.height}, its image is {image_size[0]}x{image_size[1]}: "
                         "they must have the same original size")
    W, H = (dim - dim % 64 for dim in image_size)
    mask = mask.convert("L")
    if (W, H) != tuple(image_size):
        mask = mask.resize((W, H), Image.NEAREST)
    p = (np.asarray(mask) >= 128).astype(np.uint8)
    m = p.reshape(H // 8, 8, W // 8, 8).max(axis=(1, 3))
    return p, np.ascontiguousarray(m)


class ImageInputs(NamedTuple):
    """Host-side inputs of an img2img / inpainting call, prepared by prepare_image_inputs."""
    images: np.ndarray                   # (1 or B, H, W, >=3) uint8, resized; one entry is shared by every seed
    pixel_mask: Optional[np.ndarray]     # (B, H, W) uint8 or None (plain img2img)
    latent_mask: Optional[np.ndarray]    # (B, H/8, W/8) uint8 or None


def prepare_image_inputs(image_path, mask_path, n: int) -> Optional[ImageInputs]:
    """image_path / mask_path: one image (or mask) shared by all n seeds, or a list with one entry per seed; every
    image must resize to the same size and every mask must have its image's original size.  None without an image."""
    if image_path is None:
        if mask_path is not None:
            raise ValueError("mask_path needs an image_path: inpainting regenerates part of an input image")
        return None

    def per_seed(v, name):
        if not isinstance(v, (list, tuple)):
            return None
        if len(v) != n:
            raise ValueError(f"{name} is a list of {len(v)} entries for {n} seed(s): give one per seed, or one shared")
        return list(v)

    images = per_seed(image_path, "image_path")
    loaded = [load_image_u8(im) for im in (images if images is not None else [image_path])]
    if len({a.shape[:2] for a, _ in loaded}) > 1:
        raise ValueError("the images of a list resize to different sizes "
                         f"{sorted({a.shape[:2] for a, _ in loaded})}: a batch needs one latent size")
    if len(loaded) == 1:
        arr = loaded[0][0][None]                                  # as the single-image img2img path always was
    else:
        arr = np.stack([a[:, :, :3] for a, _ in loaded])
    if mask_path is None:
        return ImageInputs(arr, None, None)
    masks = per_seed(mask_path, "mask_path")
    sizes = [s for _, s in loaded]
    if masks is None:
        prepared = [prepare_inpaint_mask(mask_path, s) for s in sizes]
    else:
        prepared = [prepare_inpaint_mask(mk, sizes[i if len(sizes) > 1 else 0]) for i, mk in enumerate(masks)]
    if len(prepared) == 1:
        prepared = prepared * n
    return ImageInputs(arr, np.stack([p for p, _ in prepared]), np.stack([m for _, m in prepared]))


class CFGDenoiser:
    """Helper for applying CFG scaling to diffusion outputs (reference mlx/__init__.py:674-719).
    x_t is the fp32 sampler state on the device; one call = prepare (cast / CFG doubling) + MMDiT forward; the
    denoised estimate and the Euler update are fused in dk_sampler_step (see sample_euler)."""

    def __init__(self, model: "DiffusionPipeline"):
        self.model = model

    def cache_modulation_params(self, pooled_text_embeddings, sigmas):
        self.model.mmdit.cache_modulation_params(pooled_text_embeddings, sigmas)

    def clear_cache(self):
        # the reference re-reads the adaLN weights it dropped (:686-689); nothing was dropped here
        pass

    def __call__(self, x_t, timestep, sigma, conditioning, cfg_weight: float = 7.5, pooled_conditioning=None):
        m = self.model
        reps = 1 if cfg_weight <= 0 else 2
        B = x_t.shape[0]
        xin = torch.empty((reps * B,) + tuple(x_t.shape[1:]), dtype=m.activation_dtype, device=x_t.device)
        ops.sampler_prepare(x_t, xin, reps)
        out = m.mmdit(latent_image_embeddings=xin, token_level_text_embeddings=conditioning, timestep=timestep)
        return xin, out


def sample_euler(model: CFGDenoiser, x, sigmas, extra_args=None):
    """Implements Algorithm 2 (Euler steps) from Karras et al. (2022) — reference mlx/__init__.py:761-788.
    x: (B, H, W, 16) fp32 device tensor (updated in place); sigmas: 1-D float32 numpy/torch array.
    extra_args["inpaint"] (optional, an extension): (x0, noise, latent mask) of a masked img2img run; after every step
    the kept cells (mask 0) are set to sigma_next * noise + (1 - sigma_next) * x0 (dk_inpaint_blend)."""
    extra_args = {} if extra_args is None else dict(extra_args)
    pipe = model.model
    sig = np.asarray(sigmas, dtype=np.float32)
    # timesteps = sampler.timestep(sigmas).astype(activation_dtype)  (:769-771; quirk Q5)
    timesteps = torch.from_numpy(np.asarray(pipe.sampler.timestep(sig), dtype=np.float32)).to(
        pipe.activation_dtype).to(torch.float32).tolist()
    pooled = extra_args.pop("pooled_conditioning")
    inpaint = extra_args.pop("inpaint", None)
    model.cache_modulation_params(pooled, timesteps)
    cfg_weight = float(extra_args.get("cfg_weight", 0.0))
    conditioning = extra_args["conditioning"]
    events = [torch.cuda.Event(enable_timing=True) for _ in range(len(sig))]
    events[0].record()
    for i in range(len(sig) - 1):
        xin, out = model(x, timesteps[i], float(sig[i]), conditioning, cfg_weight)
        # denoised = xin - out * sigma; CFG mix; d = (x - denoised) / sigma; x += d * (sigma_next - sigma)
        ops.sampler_step(x, xin, out, float(sig[i]), float(sig[i + 1]), cfg_weight)
        if inpaint is not None:
            ops.inpaint_blend(x, *inpaint, float(sig[i + 1]))
        events[i + 1].record()
    model.clear_cache()
    torch.cuda.current_stream().synchronize()  # the reference syncs every step (mx.eval, :782); once is enough here
    iter_time = [round(events[i].elapsed_time(events[i + 1]) / 1e3, 3) for i in range(len(sig) - 1)]
    return x, iter_time


class DiffusionPipeline:
    _default_model = "argmaxinc/mlx-stable-diffusion-3-medium"

    def __init__(
        self,
        w16: bool = False,
        shift: float = 1.0,
        use_t5: bool = True,
        model_version: str = "argmaxinc/mlx-stable-diffusion-3-medium",
        low_memory_mode: bool = True,
        a16: bool = False,
        local_ckpt=None,
        *,
        device: Optional[Union[int, str, torch.device]] = None,
        params: Optional[Dict[str, torch.Tensor]] = None,
        vae_params: Optional[Dict[str, torch.Tensor]] = None,
        mmdit_config: Optional[MMDiTConfig] = None,
        weight_seed: int = 0,
        load_decoder: bool = True,
        vae_encoder_params: Optional[Dict[str, torch.Tensor]] = None,
        load_encoder: bool = False,
    ):
        self.float16_dtype = torch.float16                                  # :76 (quirk Q10)
        self._vae_encoder_params, self._load_encoder = vae_encoder_params, load_encoder
        self._setup(w16, a16, shift, model_version, low_memory_mode, local_ckpt, device, params, vae_params,
                    mmdit_config, weight_seed, load_decoder)
        self.use_t5 = use_t5
        self.sampler = ModelSamplingDiscreteFlow(shift=shift)
        self.latent_format = SD3LatentFormat()
        self.use_clip_g = True

    def _setup(self, w16, a16, shift, model_version, low_memory_mode, local_ckpt, device, params, vae_params,
               mmdit_config, weight_seed, load_decoder):
        self.mmdit_ckpt = MMDIT_CKPT[model_version]                          # KeyError on unknown model (:81)
        if not (w16 and a16):
            raise NotImplementedError(
                "the B200 engine computes in 16-bit only: pass w16=True, a16=True (what the reference CLI forces, "
                "scripts/generate_images.py:117-118)")
        self._local_ckpt = local_ckpt
        self.dtype = self.float16_dtype
        self.activation_dtype = self.float16_dtype
        self.low_memory_mode = low_memory_mode
        self.model_version = model_version
        if device is None:
            device = torch.device("cuda", torch.cuda.current_device()) if torch.cuda.is_available() else None
        if device is None:
            raise DkError("no CUDA device: diffusionkit_b200 runs on B200 only; there is no CPU fallback")
        self.device = torch.device(device) if not isinstance(device, int) else torch.device("cuda", device)
        self.config = mmdit_config if mmdit_config is not None else MODEL_CONFIGS[model_version]
        self._weight_seed = weight_seed
        self._params, self._vae_params = params, vae_params
        self._load_decoder = load_decoder
        self.check_and_load_models()
        self._params = self._vae_params = None      # the models hold packed copies; drop the caller's tensors
        if hasattr(self, "encoder"):
            self._vae_encoder_params = None

    # ------------------------------------------------------------------ model loading (:90-143)
    def _load_local_ckpt(self):
        """`local_ckpt`: path of an upstream .safetensors file (BFL FLUX / Stability SD3 layout), or a dict
        {"mmdit": path, "vae": path}.  Key remapping: model_io.py (reference mlx/model_io.py:130-486)."""
        from . import model_io

        ck = self._local_ckpt
        paths = ck if isinstance(ck, dict) else {"mmdit": ck}
        out = {}
        if paths.get("mmdit"):
            sd = model_io.load_safetensors(paths["mmdit"])
            if self.model_version.endswith("-4bit-quantized"):
                # saved from the reference's own module tree: names already final, Linear weights as MLX 4-bit triples
                # (reference model_io.py:728-734 SD3.5, :772-775 FLUX); expanded to dense 16-bit once, here
                flux = isinstance(self, FluxPipeline)
                tree = model_io.preadjusted_checkpoint_to_params(sd, "" if flux else "model.diffusion_model.")
                if flux:
                    tree = {k: v for k, v in tree.items() if not k.startswith(("decoder.", "encoder."))}
                params = model_io.dequantize_q4_params(tree, self.device, self.dtype)
                if not flux and "vae" not in paths:
                    for part, pref in (("vae", "first_stage_model.decoder."), ("vae_encoder", "first_stage_model.encoder.")):
                        sub = model_io.preadjusted_checkpoint_to_params(sd, pref)
                        if sub:
                            out[part] = sub
            elif isinstance(self, FluxPipeline):
                params = model_io.flux_checkpoint_to_params(sd, self.config.hidden_size, self.config.mlp_ratio)
            else:
                params = model_io.sd3_checkpoint_to_params(sd)
                if "vae" not in paths and any("decoder." in k for k in sd):
                    out["vae"] = model_io.vae_decoder_checkpoint_to_params(sd)     # single-file SD3 checkpoints
                if "vae" not in paths and any("encoder.down." in k for k in sd):
                    out["vae_encoder"] = model_io.vae_encoder_checkpoint_to_params(sd)
            model_io.check_against_specs(params, mmdit_param_specs(self.config))
            out["mmdit"] = params
        if paths.get("vae"):
            vsd = model_io.load_safetensors(paths["vae"])
            out["vae"] = model_io.vae_decoder_checkpoint_to_params(vsd)
            if any("encoder.down." in k for k in vsd):                             # ae.safetensors holds both halves
                out["vae_encoder"] = model_io.vae_encoder_checkpoint_to_params(vsd)
        if "vae" in out:
            model_io.check_against_specs(out["vae"], vae_decoder_param_specs(VAEDecoderConfig()))
        if "vae_encoder" in out:
            model_io.check_against_specs(out["vae_encoder"], vae_encoder_param_specs(VAEEncoderConfig()))
        return out

    def load_mmdit(self, only_modulation_dict=False):
        params = self._params
        if params is None and self._local_ckpt is not None:
            loaded = self._load_local_ckpt()
            params = loaded.get("mmdit")
            if self._vae_params is None:
                self._vae_params = loaded.get("vae")
            if self._vae_encoder_params is None:
                self._vae_encoder_params = loaded.get("vae_encoder")
            if params is not None:
                params = {k: v.to(device=self.device, dtype=self.dtype) for k, v in params.items()}
        if params is None:
            params = init_params(mmdit_param_specs(self.config), seed=self._weight_seed, dtype=self.dtype,
                                 device=self.device)
        self.mmdit = MMDiT(self.config, params, device=self.device)

    def check_and_load_models(self):
        if not hasattr(self, "mmdit"):
            self.load_mmdit()
        if not hasattr(self, "decoder") and self._load_decoder:
            vp = self._vae_params
            if vp is None:
                vp = init_params(vae_decoder_param_specs(VAEDecoderConfig()), seed=self._weight_seed + 1,
                                 dtype=self.dtype, device=self.device)
            self.decoder = VAEDecoder(vp, VAEDecoderConfig(), device=self.device)
        if not hasattr(self, "encoder") and self._load_encoder:
            self.load_encoder()

    def load_encoder(self):
        """reference check_and_load_models (:115-116) loads the encoder eagerly; here it is built on the first img2img
        call (or at construction with load_encoder=True) so text-to-image runs do not carry its 34 M parameters."""
        ep = self._vae_encoder_params
        if ep is None:
            ep = init_params(vae_encoder_param_specs(VAEEncoderConfig()), seed=self._weight_seed + 2,
                             dtype=self.dtype, device=self.device)
        else:
            ep = {k: v.to(device=self.device, dtype=self.dtype) for k, v in ep.items()}
        self.encoder = VAEEncoder(ep, VAEEncoderConfig(), device=self.device)
        self._vae_encoder_params = None

    # ------------------------------------------------------------------ LoRA adapters (an extension)
    def load_lora(self, lora, scale: float = 1.0, name: Optional[str] = None):
        """Merge a LoRA adapter into the MMDiT weights in place -> lora.LoraInfo(name, rank, n_targets, skipped).
        `lora`: a .safetensors path or a dict str -> tensor, keyed by the upstream module names (BFL for FLUX, SAI for
        SD3; PEFT lora_A / lora_B or kohya lora_unet_* lora_down / lora_up, optional .alpha).  `name` defaults to the
        file stem ("lora<N>" for a dict); loading under an active name replaces that adapter, which is how its scale
        is changed.  Every touched weight is W0 + sum_i scale_i * alpha_i / r_i * B_i @ A_i over the active adapters.
        The merge runs on the device (one dk_gemm per weight); the denoise loop and its captured graphs are unchanged."""
        from .lora import LoraMerger

        if getattr(self, "_lora", None) is None:
            self._lora = LoraMerger(self.mmdit)
        return self._lora.load(lora, scale=scale, name=name)

    def unload_lora(self, name: Optional[str] = None):
        """Remove the adapter `name` (None: every adapter); weights no adapter touches any more are restored bit for
        bit."""
        if getattr(self, "_lora", None) is not None:
            self._lora.unload(name)
        elif name is not None:
            raise KeyError(f"no active LoRA named {name!r} (active: [])")

    # ------------------------------------------------------------------ text (SURVEY.md §8 row f2)
    def load_text_encoders(self, clip_l=None, clip_g=None, t5=None, *, tokenizer_l=None, tokenizer_g=None,
                           t5_tokenizer=None, clip_l_config=None, clip_g_config=None, t5_config=None):
        """Build CLIP-L (+ CLIP-G for SD3) and the T5 encoder on the device, and attach their tokenizers.
        clip_l / clip_g / t5: parameter dicts with the reference's names (model_io.clip_checkpoint_to_params /
        t5_checkpoint_to_params convert upstream safetensors), or None for the deterministic synthetic initialiser.
        tokenizer_*: tokenizer.Tokenizer / tokenizer.T5Tokenizer objects built from local vocabulary files (the
        reference downloads all of this in check_and_load_models, :118-143; no network here)."""
        from .config import CLIP_G, CLIP_L, T5EncoderConfig
        from .text_encoders import CLIPTextModel, SD3T5Encoder, clip_param_specs, t5_param_specs

        def build(cls, params, cfg, specs, seed, dtype=None):
            dtype = dtype or self.dtype
            if params is None:
                params = init_params(specs(cfg), seed=self._weight_seed + seed, dtype=dtype, device=self.device)
            return cls({k: v.to(device=self.device, dtype=dtype) for k, v in params.items()}, cfg, device=self.device)

        self.clip_l = build(CLIPTextModel, clip_l, clip_l_config or CLIP_L, clip_param_specs, 3)
        if self.use_clip_g:
            self.clip_g = build(CLIPTextModel, clip_g, clip_g_config or CLIP_G, clip_param_specs, 4)
        if self.use_t5:
            # T5-XXL's feed-forward overflows fp16 — the reference runs it in fp32 for that reason (t5.py:214-224).
            # Here its GEMMs take 16-bit inputs, so the T5 stack always computes in bf16 (fp32's range), also
            # inside the fp16 SD3 pipeline; the output is cast to the activation dtype.
            self.t5_encoder = build(SD3T5Encoder, t5, t5_config or T5EncoderConfig(), t5_param_specs, 5,
                                    dtype=torch.bfloat16)
        self.tokenizer_l, self.tokenizer_g, self.t5_tokenizer = tokenizer_l, tokenizer_g, t5_tokenizer

    def _need_text_stack(self, *names):
        missing = [n for n in names if getattr(self, n, None) is None]
        if missing:
            raise DkError(
                f"encode_text needs {', '.join(missing)}: call load_text_encoders(...) with local weights and "
                "tokenizer files first (nothing can be downloaded here), or pass `conditioning` / `pooled_conditioning`")

    def _tokenize(self, tokenizer, text: str, negative_text: Optional[str] = None):
        """reference :174-195 — note that a None negative prompt becomes "" first, so two rows always come back (Q11)"""
        if negative_text is None:
            negative_text = ""
        pad_token = tokenizer.eos_token if tokenizer.pad_with_eos else 0
        tokens = [list(tokenizer.tokenize(text))]
        if tokenizer.pad_to_max_length:
            tokens[0].extend([pad_token] * (tokenizer.max_length - len(tokens[0])))
        tokens += [list(tokenizer.tokenize(negative_text))]
        N = max(len(t) for t in tokens)
        tokens = [t + [pad_token] * (N - len(t)) for t in tokens]
        return torch.tensor(tokens, dtype=torch.int64)

    def encode_text(self, text: str, cfg_weight: float = 7.5, negative_text: str = ""):
        """reference :197-251 -> (conditioning (2, 77 + T5, 4096), pooled (2, 2048)) in the activation dtype"""
        need = ["clip_l", "tokenizer_l", "clip_g", "tokenizer_g"] + (["t5_encoder", "t5_tokenizer"] if self.use_t5 else [])
        self._need_text_stack(*need)
        neg = negative_text if cfg_weight > 1 else None
        cl = self.clip_l(self._tokenize(self.tokenizer_l, text, neg))
        cg = self.clip_g(self._tokenize(self.tokenizer_g, text, neg))
        conditioning = torch.cat([cl.hidden_states[-2], cg.hidden_states[-2]], dim=-1)
        pooled_conditioning = torch.cat([cl.pooled_output, cg.pooled_output], dim=-1)
        pad = torch.zeros((conditioning.shape[0], conditioning.shape[1], 4096 - conditioning.shape[2]),
                          dtype=conditioning.dtype, device=self.device)
        conditioning = torch.cat([conditioning, pad], dim=-1)
        if self.use_t5:
            t5_conditioning = self.t5_encoder(self._tokenize(self.t5_tokenizer, text, neg)).to(conditioning.dtype)
        else:
            t5_conditioning = torch.zeros_like(conditioning)
        conditioning = torch.cat([conditioning, t5_conditioning], dim=1)
        return conditioning, pooled_conditioning

    def text_shapes(self, cfg_weight: float) -> Tuple[Tuple[int, int], Tuple[int, int]]:
        """(conditioning (Bc, T, 4096), pooled (Bc, P)) shapes the reference produces for ONE image."""
        c = self.config
        if isinstance(self, FluxPipeline):
            return (1, T5_MAX_LENGTH.get(self.model_version, 256), c.token_level_text_embed_dim), (
                1, c.pooled_text_embed_dim)
        T = 77 + (T5_MAX_LENGTH.get(self.model_version, 512) if self.use_t5 else 77)    # :186-187, :239-249 (Q2)
        return (2, T, c.token_level_text_embed_dim), (2, c.pooled_text_embed_dim)        # always 2 (Q11)

    def synthetic_text_embeddings(self, n_images: int = 1, seed: int = 1234, text_len: Optional[int] = None):
        """N(0,1) stand-ins for encode_text's outputs (SURVEY.md §8d), laid out [positive(n) | negative(n)] for SD3."""
        (bc, T, E), (_, P) = self.text_shapes(1.0)
        if text_len is not None:
            T = text_len
        g = torch.Generator(device="cpu").manual_seed(seed)
        cond = torch.randn((bc * n_images, T, E), generator=g, dtype=torch.float32)
        pooled = torch.randn((bc * n_images, P), generator=g, dtype=torch.float32)
        return cond.to(self.activation_dtype), pooled.to(self.activation_dtype)

    # ------------------------------------------------------------------ denoise (:253-292)
    def denoise_latents(
        self,
        conditioning,
        pooled_conditioning,
        num_steps: int = 2,
        cfg_weight: float = 0.0,
        latent_size: Tuple[int, int] = (64, 64),
        seed=None,
        image_path: Optional[str] = None,
        denoise: float = 1.0,
        mask_path=None,
        *,
        noise: Optional[torch.Tensor] = None,
    ):
        """-> (latent NHWC (B, H, W, 16) fp32 on the device, iter_time list).  `noise` (optional, device fp32
        (B, H, W, 16)) replaces the host-side numpy draw of get_noise for callers whose inputs already live in HBM.
        `image_path` (img2img): a file path, a PIL image or a uint8 HWC array; the latent size then follows the image
        (the reference ignores latent_size in that case too, :273).  A list gives one image per seed (all must resize
        to the same size); a single image is shared by every seed.
        `mask_path` (inpainting, an extension): same kinds of value as `image_path`, one shared or a list with one per
        seed, at the original size of its image; white (>= 128) = regenerate.  Latent cells outside the mask follow the
        image's noised trajectory after every step and end exactly at its encoding (prepare_inpaint_mask)."""
        if image_path is None:
            denoise = 1.0                                                   # :270-271
        elif not (0.0 <= denoise <= 1.0):
            raise ValueError(f"denoise must be in [0, 1], got {denoise}")
        n = len(seed) if isinstance(seed, (list, tuple)) else 1
        src = prepare_image_inputs(image_path, mask_path, n)
        return self._denoise_latents(conditioning, pooled_conditioning, num_steps, cfg_weight, latent_size, seed, src,
                                     denoise, noise)

    def _denoise_latents(self, conditioning, pooled_conditioning, num_steps, cfg_weight, latent_size, seed,
                         src: Optional[ImageInputs], denoise, noise):
        seeds: List[int]
        if seed is None:
            seeds = [int(time.time())]
        elif isinstance(seed, (list, tuple)):
            seeds = [int(s) for s in seed]
        else:
            seeds = [int(seed)]
        B = len(seeds)
        H, W = latent_size
        conditioning = torch.as_tensor(conditioning).to(device=self.device, dtype=self.activation_dtype)
        pooled_conditioning = torch.as_tensor(pooled_conditioning).to(device=self.device, dtype=self.activation_dtype)
        if conditioning.dim() == 4:
            conditioning = conditioning.squeeze(2)
        reps = 2 if cfg_weight > 0 else 1
        if B > 1 and conditioning.shape[0] == reps and pooled_conditioning.shape[0] == reps:
            # one prompt (what encode_text returns: [positive] or [positive | negative]), several seeds: every image of
            # the batch shares it -> [positive x B | negative x B], the layout CFGDenoiser splits (:718)
            conditioning = conditioning.repeat_interleave(B, dim=0)
            pooled_conditioning = pooled_conditioning.repeat_interleave(B, dim=0)
        if conditioning.shape[0] != reps * B:
            raise DkError(
                f"conditioning has batch {conditioning.shape[0]}, expected {reps * B} "
                f"({'[positive | negative] x ' if reps == 2 else ''}{B} image(s)) for cfg_weight={cfg_weight}")

        hidden = None
        if src is not None:
            hidden = self._encode_u8(src.images)                            # (1 or B, H, W, 32) = (mean | logvar)
            H, W = hidden.shape[1], hidden.shape[2]
        x_T = self.get_empty_latent(H, W)                                   # (1, H, W, 16) host
        if noise is None:
            noise = self._get_noise_batch(seeds, x_T)                              # (B, H, W, 16) host fp32
        elif tuple(noise.shape) != (B, H, W, 16):
            raise DkError(f"noise has shape {tuple(noise.shape)}, expected {(B, H, W, 16)}")
        sigmas = self.get_sigmas(self.sampler, num_steps)
        sigmas = sigmas[int(num_steps * (1 - denoise)):]
        s0 = float(sigmas[0])
        if hidden is None:
            x = noise.to(self.device, dtype=torch.float32, non_blocking=True).clone()
            # noise_scaling: sigma0 * noise + (1 - sigma0) * x_T (sampler.py:41-42); x_T is the constant 0.0609
            x = ops.axpb(x.contiguous(), s0, (1.0 - s0) * 0.0609)
        else:
            # x_T = process_in(mean + std * noise), with the SAME seeded draw the diffusion noise uses (:273-275,
            # :586-594: both get_noise(seed, .) calls see the same shape); then sigma0 * noise + (1 - sigma0) * x_T
            noise = noise.to(self.device, dtype=torch.float32, non_blocking=True).contiguous()
            lf = self.latent_format
            x_T = torch.empty_like(noise)
            if hidden.shape[0] == B:                                        # one image per seed: one launch
                ops.vae_sample_latent(hidden, noise, lf.shift_factor, lf.scale_factor, out=x_T)
            else:                                                           # one image shared by every seed
                for b in range(B):
                    ops.vae_sample_latent(hidden, noise[b:b + 1], lf.shift_factor, lf.scale_factor, out=x_T[b:b + 1])
            x = ops.axpby(noise, x_T, s0, 1.0 - s0)
        extra_args = {"conditioning": conditioning, "cfg_weight": cfg_weight,
                      "pooled_conditioning": pooled_conditioning}
        if src is not None and src.latent_mask is not None:
            mask = torch.from_numpy(src.latent_mask).pin_memory().to(self.device, non_blocking=True)
            extra_args["inpaint"] = (x_T, noise, mask)
        latent, iter_time = sample_euler(CFGDenoiser(self), x, sigmas, extra_args=extra_args)
        latent = ops.axpb(latent, 1.0 / self.latent_format.scale_factor, self.latent_format.shift_factor)  # process_out
        return latent, iter_time

    # ------------------------------------------------------------------ generate (:294-534)
    def generate_image(
        self,
        text: str,
        num_steps: int = 2,
        cfg_weight: float = 0.0,
        negative_text: str = "",
        latent_size: Tuple[int, int] = (64, 64),
        seed=None,
        verbose: bool = True,
        image_path: Optional[str] = None,
        denoise: float = 1.0,
        mask_path=None,
        *,
        conditioning=None,
        pooled_conditioning=None,
    ):
        """With `mask_path` (inpainting, see denoise_latents) the decoded image is composited in uint8: pixels outside
        the mask are the resized input image, bit for bit."""
        assert latent_size[0] % 2 == 0, f"Height must be divisible by 16 ({latent_size[0]*8}/16={latent_size[0]/2})"
        assert latent_size[1] % 2 == 0, f"Width must be divisible by 16 ({latent_size[1]*8}/16={latent_size[1]/2})"
        if image_path is not None and not (0.0 <= denoise <= 1.0):
            raise ValueError(f"denoise must be in [0, 1], got {denoise}")
        src = prepare_image_inputs(image_path, mask_path, len(seed) if isinstance(seed, (list, tuple)) else 1)
        self.check_and_load_models()
        start_time = time.time()

        def mem():
            return {"peak_memory": round(_bytes2gigabytes(torch.cuda.max_memory_allocated(self.device)), 3),
                    "active_memory": round(_bytes2gigabytes(torch.cuda.memory_allocated(self.device)), 3)}

        log = {
            "text_encoding": {"pre": mem(), "post": {"peak_memory": None, "active_memory": None}},
            "denoising": {"pre": {"peak_memory": None, "active_memory": None},
                          "post": {"peak_memory": None, "active_memory": None}},
            "decoding": {"pre": {"peak_memory": None, "active_memory": None},
                         "post": {"peak_memory": None, "active_memory": None}},
            "peak_memory": 0.0,
        }
        t0 = time.time()
        if conditioning is None or pooled_conditioning is None:
            conditioning, pooled_conditioning = self.encode_text(text, cfg_weight, negative_text)
        log["text_encoding"]["post"] = mem()
        log["text_encoding"]["time"] = round(time.time() - t0, 3)
        log["peak_memory"] = max(log["peak_memory"], log["text_encoding"]["post"]["peak_memory"])

        torch.cuda.reset_peak_memory_stats(self.device)
        t0 = time.time()
        log["denoising"]["pre"] = mem()
        latents, iter_time = self._denoise_latents(conditioning, pooled_conditioning, num_steps, cfg_weight,
                                                   latent_size, seed, src, denoise if src is not None else 1.0, None)
        torch.cuda.synchronize(self.device)
        log["denoising"]["post"] = mem()
        log["denoising"]["time"] = round(time.time() - t0, 3)
        log["denoising"]["iter_time"] = iter_time
        log["peak_memory"] = max(log["peak_memory"], log["denoising"]["post"]["peak_memory"])

        torch.cuda.reset_peak_memory_stats(self.device)
        t0 = time.time()
        log["decoding"]["pre"] = mem()
        latents16 = ops.cast_to_16(latents, self.activation_dtype)          # latents.astype(activation_dtype) (:459)
        if src is not None and src.pixel_mask is not None:
            u8 = self._decode_composite(latents16, src)
        else:
            _, u8 = self._decode(latents16, want_u8=True)
        host = getattr(self, "_host_u8", None)                              # pinned staging, reused across calls
        if host is None or host.shape != u8.shape:
            host = self._host_u8 = torch.empty(u8.shape, dtype=torch.uint8, pin_memory=True)
        host.copy_(u8, non_blocking=True)                                   # device -> host: the result
        torch.cuda.current_stream().synchronize()
        images_u8 = host.numpy()         # Image.fromarray copies RGB data, so reusing the staging buffer is safe
        log["decoding"]["post"] = mem()
        log["decoding"]["time"] = round(time.time() - t0, 3)
        log["peak_memory"] = max(log["peak_memory"], log["decoding"]["post"]["peak_memory"])
        log["total_time"] = round(time.time() - start_time, 3)

        from PIL import Image

        images = [Image.fromarray(images_u8[i]) for i in range(images_u8.shape[0])]
        # batch 1 returns a single image like the reference; a list of seeds returns a list (quirk Q9)
        return (images[0] if not isinstance(seed, (list, tuple)) else images), log

    # ------------------------------------------------------------------ helpers (:553-584)
    def get_noise(self, seed, x_T):
        # np.random.seed(seed); np.random.randn(...) of the reference (:553-557).  RandomState(seed) is the same
        # MT19937 stream as the seeded global generator, without the global state (thread-safe for batches).
        shape = tuple(x_T.shape)
        noise = np.random.RandomState(seed).randn(shape[0], shape[3], shape[1], shape[2])
        # float64 -> float32 and NCHW -> NHWC in numpy: the same values as mx.array(noise).transpose(0, 2, 3, 1), and
        # ~100x cheaper on a many-core host than a strided multi-threaded torch CPU copy
        return torch.from_numpy(np.ascontiguousarray(noise.astype(np.float32).transpose(0, 2, 3, 1)))

    def _get_noise_batch(self, seeds, x_T):
        if len(seeds) == 1:
            return self.get_noise(seeds[0], x_T)
        from concurrent.futures import ThreadPoolExecutor

        with ThreadPoolExecutor(max_workers=min(len(seeds), 8)) as ex:   # numpy releases the GIL while drawing
            parts = list(ex.map(lambda sd: self.get_noise(sd, x_T), seeds))
        return torch.cat(parts, dim=0)

    def get_sigmas(self, sampler, num_steps: int):
        start = float(sampler.timestep(sampler.sigma_max))
        end = float(sampler.timestep(sampler.sigma_min))
        if isinstance(sampler, FluxSampler):
            num_steps += 1
        timesteps = np.linspace(start, end, num_steps, dtype=np.float32)
        sigs = [float(sampler.sigma(ts)) for ts in timesteps]
        if not isinstance(sampler, FluxSampler):
            sigs += [0.0]
        return np.asarray(sigs, dtype=np.float32)

    def _load_image_u8(self, image) -> np.ndarray:
        """-> uint8 (H, W, >=3) with H, W multiples of 64 (read_image's resize rule, :540-546)"""
        return load_image_u8(image)[0]

    def read_image(self, image_path):
        """-> (1, H, W, 3) float32 in [-1, 1] on the host (reference :536-551)"""
        arr = self._load_image_u8(image_path)
        return (torch.from_numpy(arr[:, :, :3].astype(np.float32)) / 255 * 2 - 1.0).unsqueeze(0)

    def _encode_image_hidden(self, image_path) -> torch.Tensor:
        return self._encode_u8(self._load_image_u8(image_path)[None])

    def _encode_u8(self, arr: np.ndarray) -> torch.Tensor:
        """uint8 (N, H, W, >=3) resized images -> encoder hidden (N, H/8, W/8, 32), one encoder run at batch N"""
        if not hasattr(self, "encoder"):
            self.load_encoder()
        host = torch.from_numpy(arr).pin_memory()
        return self.encoder(host.to(self.device, non_blocking=True))       # the /255*2-1 runs in dk_image_pre

    def encode_image_to_latents(self, image_path, seed):
        """mean + exp(0.5 * clip(logvar, -30, 20)) * get_noise(seed)  (reference :586-594) -> (1, H/8, W/8, 16) fp32"""
        hidden = self._encode_image_hidden(image_path)
        mean_like = torch.empty((1, hidden.shape[1], hidden.shape[2], hidden.shape[3] // 2))
        noise = self.get_noise(seed, mean_like).to(self.device)
        return ops.vae_sample_latent(hidden, noise.contiguous(), 0.0, 1.0)

    def get_empty_latent(self, *shape):
        return torch.ones([1, *shape, 16], dtype=torch.float32) * 0.0609

    def max_denoise(self, sigmas):
        max_sigma = float(self.sampler.sigma_max)
        sigma = float(sigmas[0])
        return math.isclose(max_sigma, sigma, rel_tol=1e-05) or sigma > max_sigma

    def _decode(self, x_t, want_u8: bool):
        x = self.decoder(x_t)                                               # (B, 8H, 8W, 3) view of a padded buffer
        B, Ho, Wo, _ = x.shape
        padded = x.as_strided((B, Ho, Wo, x.stride(2)), (x.stride(0), x.stride(1), x.stride(2), 1))
        return ops.image_post(padded, want_u8=want_u8)

    def _decode_composite(self, x_t, src: ImageInputs) -> torch.Tensor:
        """decode, then uint8 = pixel mask ? decoded : resized input image  (inpainting)"""
        x = self.decoder(x_t)
        B, Ho, Wo, _ = x.shape
        padded = x.as_strided((B, Ho, Wo, x.stride(2)), (x.stride(0), x.stride(1), x.stride(2), 1))
        orig = np.ascontiguousarray(np.broadcast_to(src.images[:, :, :, :3], (B, Ho, Wo, 3)))
        orig = torch.from_numpy(orig).pin_memory().to(self.device, non_blocking=True)
        mask = torch.from_numpy(src.pixel_mask).pin_memory().to(self.device, non_blocking=True)
        return ops.image_post_masked(padded, orig, mask)

    def decode_latents_to_image(self, x_t):
        """x = decoder(x_t); clip(x / 2 + 0.5, 0, 1)  (:581-584) -> (B, 8H, 8W, 3) float in [0, 1]"""
        x_t = torch.as_tensor(x_t).to(device=self.device)
        if x_t.dtype == torch.float32:
            x_t = ops.cast_to_16(x_t.contiguous(), self.activation_dtype)
        f, _ = self._decode(x_t, want_u8=False)
        return f


class FluxPipeline(DiffusionPipeline):
    _default_model = "argmaxinc/mlx-FLUX.1-schnell"

    def __init__(
        self,
        w16: bool = False,
        shift: float = 1.0,
        use_t5: bool = True,
        model_version: str = "argmaxinc/mlx-FLUX.1-schnell",
        low_memory_mode: bool = True,
        a16: bool = False,
        local_ckpt=None,
        quantize_mmdit: bool = False,
        *,
        device=None,
        params=None,
        vae_params=None,
        mmdit_config=None,
        weight_seed: int = 0,
        load_decoder: bool = True,
        vae_encoder_params=None,
        load_encoder: bool = False,
    ):
        self.float16_dtype = torch.bfloat16                                 # :610
        self._vae_encoder_params, self._load_encoder = vae_encoder_params, load_encoder
        self._setup(w16, a16, shift, model_version, low_memory_mode, local_ckpt, device, params, vae_params,
                    mmdit_config, weight_seed, load_decoder)
        self.sampler = FluxSampler(shift=shift)
        self.latent_format = FluxLatentFormat()
        self.use_t5 = True
        self.use_clip_g = False
        self.quantize_mmdit = quantize_mmdit

    def encode_text(self, text: str, cfg_weight: float = 7.5, negative_text: str = ""):
        """reference :642-671: CLIP-L pooled output + T5 sequence of the POSITIVE prompt only, T5 padded with zeros to
        T5_MAX_LENGTH -> (conditioning (1, T5, 4096), pooled (1, 768))"""
        self._need_text_stack("clip_l", "tokenizer_l", "t5_encoder", "t5_tokenizer")
        neg = negative_text if cfg_weight > 1 else None
        tokens_l = self._tokenize(self.tokenizer_l, text, neg)
        pooled_conditioning = self.clip_l(tokens_l[[0], :]).pooled_output
        tokens_t5 = self._tokenize(self.t5_tokenizer, text, neg)
        padded = torch.zeros((1, T5_MAX_LENGTH[self.model_version]), dtype=tokens_t5.dtype)
        padded[:, : tokens_t5.shape[1]] = tokens_t5[[0], :]
        conditioning = self.t5_encoder(padded).to(self.activation_dtype)
        return conditioning, pooled_conditioning
