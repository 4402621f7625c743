"""Stand-ins that let the reference's OWN PyTorch modules (python/src/diffusionkit/torch/mmdit.py and vae.py — real
reference code, imported from a checkout named by $DIFFUSIONKIT_REFERENCE, never copied) run under plain PyTorch.

Those two files import four generic building blocks from the un-vendored dependency `argmaxtools>=0.1.13`
(setup.py:29), which is not installed here:
    argmaxtools.nn.LayerNorm / Attention / FFN / AttentionType   (torch/mmdit.py:221-243, 390)
    argmaxtools._sdpa.Cat                                         (torch/mmdit.py:325-326, torch/vae.py:57-61)
The classes below restate them from how the reference uses them and from the checkpoint shapes its loader produces
(torch/mmdit.py:424-497: every projection is a 1x1 Conv2d over the (batch, channels, 1, sequence) layout, k_proj has no
bias).  Everything else that executes — patch embedding, positional-embedding crop, timestep / pooled adapters, adaLN
chunk order, pre/post-SDPA wiring, gating, final layer, unpatchify, the whole VAE decoder topology — is the reference's
code.  Test infrastructure only (tests/golden/make_reference_golden.py, make_reference_pins.py).
"""
import enum
import importlib.util
import logging
import os
import sys
import types

import torch
import torch.nn as nn

# python/src of an argmaxinc/DiffusionKit checkout; only the golden-data generators under tests/golden/ read it
REFERENCE_SRC = os.path.join(os.environ.get("DIFFUSIONKIT_REFERENCE", ""), "python", "src")
REFERENCE_TORCH_DIR = os.path.join(REFERENCE_SRC, "diffusionkit", "torch")


class LayerNorm(nn.Module):
    """LayerNorm over the channel axis (dim 1) of a (B, C, 1, S) tensor, biased variance, optional affine"""

    def __init__(self, num_channels, eps=1e-5, elementwise_affine=True):
        super().__init__()
        self.eps = eps
        if elementwise_affine:
            self.weight = nn.Parameter(torch.ones(num_channels))
            self.bias = nn.Parameter(torch.zeros(num_channels))
        else:
            self.weight = self.bias = None

    def forward(self, x):
        mu = x.mean(dim=1, keepdim=True)
        var = (x - mu).pow(2).mean(dim=1, keepdim=True)
        y = (x - mu) * torch.rsqrt(var + self.eps)
        if self.weight is not None:
            y = y * self.weight.view(1, -1, 1, 1) + self.bias.view(1, -1, 1, 1)
        return y


class AttentionType(enum.Enum):
    SelfAttention = 1
    KVCachedSelfAttention = 2
    EncoderDecoderCrossAttention = 3


class Attention(nn.Module):
    """Holder of the four 1x1-conv projections the reference calls directly (q/v/o with bias, k without)"""

    def __init__(self, embed_dim, n_heads, attention_type=AttentionType.SelfAttention):
        super().__init__()
        self.embed_dim, self.n_heads = embed_dim, n_heads
        self.q_proj = nn.Conv2d(embed_dim, embed_dim, 1)
        self.k_proj = nn.Conv2d(embed_dim, embed_dim, 1, bias=False)
        self.v_proj = nn.Conv2d(embed_dim, embed_dim, 1)
        self.o_proj = nn.Conv2d(embed_dim, embed_dim, 1)


class FFN(nn.Module):
    def __init__(self, embed_dim, expansion_factor, activation_fn):
        super().__init__()
        self.fc1 = nn.Conv2d(embed_dim, embed_dim * expansion_factor, 1)
        self.act_fn = activation_fn
        self.fc2 = nn.Conv2d(embed_dim * expansion_factor, embed_dim, 1)

    def forward(self, x):
        return self.fc2(self.act_fn(self.fc1(x)))


class Cat:
    """Multi-head scaled-dot-product attention on (B, C, 1, S) tensors; head h owns channels [h*d, (h+1)*d)"""

    def __init__(self, embed_dim, n_heads):
        self.embed_dim, self.n_heads = embed_dim, n_heads
        self.dim_head = embed_dim // n_heads

    def sdpa(self, query, key, value, key_padding_mask=None, causal=False):
        assert key_padding_mask is None and not causal
        B, C, _, Sq = query.shape
        Sk = key.shape[-1]
        H, d = self.n_heads, self.dim_head
        q = query.reshape(B, H, d, Sq)
        k = key.reshape(B, H, d, Sk)
        v = value.reshape(B, H, d, Sk)
        w = torch.softmax(torch.einsum("bhdq,bhdk->bhqk", q, k) * d ** -0.5, dim=-1)
        return torch.einsum("bhqk,bhdk->bhdq", w, v).reshape(B, C, 1, Sq)


def install():
    """register the stand-in `argmaxtools` package (idempotent)"""
    if "argmaxtools" in sys.modules and getattr(sys.modules["argmaxtools"], "_dkb200_shim", False):
        return
    pkg = types.ModuleType("argmaxtools")
    pkg._dkb200_shim = True
    nn_mod = types.ModuleType("argmaxtools.nn")
    nn_mod.LayerNorm, nn_mod.Attention, nn_mod.FFN, nn_mod.AttentionType = LayerNorm, Attention, FFN, AttentionType
    sdpa_mod = types.ModuleType("argmaxtools._sdpa")
    sdpa_mod.Cat = Cat
    utils_mod = types.ModuleType("argmaxtools.utils")
    utils_mod.get_logger = logging.getLogger
    pkg.nn, pkg._sdpa, pkg.utils = nn_mod, sdpa_mod, utils_mod
    sys.modules.update({"argmaxtools": pkg, "argmaxtools.nn": nn_mod, "argmaxtools._sdpa": sdpa_mod,
                        "argmaxtools.utils": utils_mod})


def load_reference_module(name: str):
    """import <reference>/python/src/diffusionkit/torch/<name>.py by path (no package __init__ side effects)"""
    install()
    path = os.path.join(REFERENCE_TORCH_DIR, name + ".py")
    spec = importlib.util.spec_from_file_location(f"_reference_torch_{name}", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def reference_available() -> bool:
    return bool(os.environ.get("DIFFUSIONKIT_REFERENCE")) and os.path.exists(os.path.join(REFERENCE_TORCH_DIR, "mmdit.py"))
