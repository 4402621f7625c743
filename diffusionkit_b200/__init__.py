"""diffusionkit_b200 — B200-native denoise + decode engine behind DiffusionKit's `diffusionkit.mlx`
DiffusionPipeline / FluxPipeline API (reference: argmaxinc/DiffusionKit, python/src/diffusionkit/mlx/__init__.py).

    from diffusionkit_b200 import FluxPipeline
    pipe = FluxPipeline(w16=True, a16=True, shift=1.0, model_version="argmaxinc/mlx-FLUX.1-schnell")
    cond, pooled = pipe.synthetic_text_embeddings()
    image, log = pipe.generate_image("", num_steps=4, cfg_weight=0.0, latent_size=(64, 64), seed=0,
                                     conditioning=cond, pooled_conditioning=pooled)
"""
from ._lib import DkError  # noqa: F401
from .config import FLUX_DEV, FLUX_SCHNELL, SD3_2b, SD3_8b, MMDiTConfig, VAEDecoderConfig, VAEEncoderConfig  # noqa: F401
from .lora import LoraInfo  # noqa: F401
from .mmdit import MMDiT  # noqa: F401
from .pipeline import (CFGDenoiser, DiffusionPipeline, FluxLatentFormat, FluxPipeline, LatentFormat,  # noqa: F401
                       SD3LatentFormat, sample_euler)
from .sampler import FluxSampler, ModelSamplingDiscreteFlow  # noqa: F401
from .vae import VAEDecoder, VAEEncoder  # noqa: F401

__version__ = "0.1.0"
