"""CPU: LoRA parsing and routing (lora.py, model_io's Linear route table) against the upstream-space oracle merge
(oracle/lora_ref.py).  The factors are small integers and the scales powers of two, so every fp64 product and sum is
exact and the product's per-reference-weight deltas must equal the oracle's upstream merge bit for bit."""
import pytest
import torch

from diffusionkit_b200 import lora as L
from diffusionkit_b200 import model_io
from diffusionkit_b200.config import FLUX_SCHNELL, SD3_8b, tiny_flux_config, tiny_sd3_config
from diffusionkit_b200.weights import init_params, mmdit_param_specs
from oracle.lora_ref import merge_upstream
from tests.test_model_io_cpu import _flux_upstream, _sd3_upstream


def _modules(cfg):
    if cfg.depth_unified > 0:
        return model_io.flux_linear_modules(cfg.depth_multimodal, cfg.depth_unified)
    return model_io.sd3_linear_modules(cfg.depth_multimodal)


def _upstream_shape(cfg, module):
    """(out, in) of an upstream Linear from the route table and the reference shapes"""
    shapes = L.weight_shapes(cfg)
    route = (model_io.flux_linear_route(module, cfg.mlp_ratio) if cfg.depth_unified > 0
             else model_io.sd3_linear_route(module))
    dim, parts = route
    ws = [shapes[n + ".weight"] for n, _ in parts]
    return (sum(s[0] for s in ws), ws[0][1]) if dim == 0 else (ws[0][0], sum(s[1] for s in ws))


def _int_lora(cfg, seed, rank_of, spelling_of, alpha_of, modules=None, dtype=torch.float64):
    """full-coverage LoRA with small-integer factors; rank_of / spelling_of / alpha_of: callables of the module index"""
    g = torch.Generator().manual_seed(seed)
    sd = {}
    for i, m in enumerate(modules if modules is not None else _modules(cfg)):
        out_f, in_f = _upstream_shape(cfg, m)
        r = rank_of(i)
        A = torch.randint(-3, 4, (r, in_f), generator=g).to(dtype)
        B = torch.randint(-3, 4, (out_f, r), generator=g).to(dtype)
        sp = spelling_of(i)
        if sp == "kohya":
            base = "lora_unet_" + m.replace(".", "_")
            ka, kb, kal = base + ".lora_down.weight", base + ".lora_up.weight", base + ".alpha"
        else:
            base = {"peft": "", "dm": "diffusion_model.", "mdm": "model.diffusion_model."}[sp] + m
            ka, kb, kal = base + ".lora_A.weight", base + ".lora_B.weight", base + ".alpha"
        sd[ka], sd[kb] = A, B
        alpha = alpha_of(i, r)
        if alpha is not None:
            sd[kal] = torch.tensor(float(alpha))
    return sd


def _product_merge(params, cfg, adapters):
    """the product's routing in fp64: upstream modules -> reference weights, W += scale * alpha/r * B @ A per weight"""
    out = dict(params)
    shapes = L.weight_shapes(cfg)
    for sd, scale in adapters:
        pairs, _ = L.parse_lora(sd, cfg, shapes)
        for name, p in L.route_pairs(pairs, cfg).items():
            d = (scale * p.alpha_over_rank) * (p.B.double() @ p.A.double())
            out[name] = out[name].double() + d.reshape(out[name].shape)
    return out


SPELLINGS = ("peft", "kohya", "dm", "mdm")


@pytest.mark.parametrize("kind", ["flux", "sd3"])
def test_routing_matches_upstream_merge(kind):
    cfg = tiny_flux_config() if kind == "flux" else tiny_sd3_config()
    params = {k: v.double() for k, v in init_params(mmdit_param_specs(cfg), seed=3, dtype=torch.float32).items()}
    a1 = _int_lora(cfg, 1, lambda i: (1, 4, 8, 5)[i % 4], lambda i: SPELLINGS[i % 4],
                   lambda i, r: (None, 2 * r, r / 2)[i % 3])
    a2 = _int_lora(cfg, 2, lambda i: 3, lambda i: SPELLINGS[(i + 1) % 4], lambda i, r: None)
    adapters = [(a1, 0.5), (a2, -2.0)]
    got = _product_merge(params, cfg, adapters)
    if kind == "flux":
        up = merge_upstream(_flux_upstream(params, cfg), adapters)
        want = model_io.flux_checkpoint_to_params(up, cfg.hidden_size, cfg.mlp_ratio)
    else:
        prefix = "model.diffusion_model."
        up = merge_upstream(_sd3_upstream(params, cfg, prefix), adapters, prefix)
        want = model_io.sd3_checkpoint_to_params(up, prefix)
    n_changed = 0
    for name, p in params.items():
        if name.startswith("unified") and name.endswith("mlp.fc2.bias"):
            continue                                        # linear2's one bias (see test_flux_checkpoint_roundtrip)
        assert torch.equal(got[name].double(), want[name].double()), name
        n_changed += not torch.equal(got[name].double(), p)
    # every 2-D weight the model has was adapted
    assert n_changed == len(L.weight_shapes(cfg)) - (kind == "sd3")    # SD3's x_embedder is a conv: no LoRA


def test_parse_spellings_prefixes_alpha():
    cfg = tiny_flux_config()
    mods = ["double_blocks.0.img_attn.qkv", "single_blocks.1.linear2", "img_in", "final_layer.adaLN_modulation.1"]
    ranks = [2, 3, 4, 8]
    sd = _int_lora(cfg, 5, lambda i: ranks[i], lambda i: SPELLINGS[i], lambda i, r: (None, 6.0, None, 2.0)[i],
                   modules=mods, dtype=torch.bfloat16)
    pairs, skipped = L.parse_lora(sd, cfg, L.weight_shapes(cfg))
    assert sorted(pairs) == sorted(mods) and skipped == ()
    assert [pairs[m].alpha_over_rank for m in mods] == [1.0, 2.0, 1.0, 0.25]     # alpha absent -> alpha = r
    assert torch.equal(pairs["single_blocks.1.linear2"].A,
                       sd["lora_unet_single_blocks_1_linear2.lora_down.weight"])
    assert torch.equal(pairs["img_in"].B, sd["diffusion_model.img_in.lora_B.weight"])
    routed = L.route_pairs(pairs, cfg)
    h = cfg.hidden_size
    q = routed["multimodal_transformer_blocks.0.image_transformer_block.attn.k_proj.weight"]
    assert torch.equal(q.B, pairs["double_blocks.0.img_attn.qkv"].B[h:2 * h])                    # row split: B rows
    fc2 = routed["unified_transformer_blocks.1.transformer_block.mlp.fc2.weight"]
    assert torch.equal(fc2.A, pairs["single_blocks.1.linear2"].A[:, h:])                           # column split: A cols
    assert len(routed) == 3 + 2 + 1 + 1


@pytest.mark.parametrize("cfg", [FLUX_SCHNELL, SD3_8b], ids=["flux_19_38", "sd35_large_38"])
def test_kohya_names_resolve_full_size(cfg):
    """every module of the full-size module lists resolves from its flattened name, no ambiguity, no miss"""
    mods = _modules(cfg)
    flat = [m.replace(".", "_") for m in mods]
    assert len(set(flat)) == len(flat) == len(set(mods))
    sd = _int_lora(cfg, 0, lambda i: 1, lambda i: "kohya", lambda i, r: None, dtype=torch.bfloat16)
    pairs, _ = L.parse_lora(sd, cfg, L.weight_shapes(cfg))
    assert sorted(pairs) == sorted(mods)
    for m in mods:
        base = "lora_unet_" + m.replace(".", "_")
        assert torch.equal(pairs[m].A, sd[base + ".lora_down.weight"]), m
    if cfg is FLUX_SCHNELL:
        assert "single_blocks.1.linear1" in pairs and "single_blocks.11.linear1" in pairs
        assert len(mods) == 8 + 19 * 10 + 38 * 3


def _one(module, r=2, cfg=None, kohya=False):
    cfg = cfg or tiny_flux_config()
    out_f, in_f = _upstream_shape(cfg, module)
    if kohya:
        b = "lora_unet_" + module.replace(".", "_")
        return {b + ".lora_down.weight": torch.ones(r, in_f), b + ".lora_up.weight": torch.ones(out_f, r)}
    return {module + ".lora_A.weight": torch.ones(r, in_f), module + ".lora_B.weight": torch.ones(out_f, r)}


def test_skipped_modules():
    cfg = tiny_flux_config()
    sd = _one("double_blocks.0.txt_mlp.0")
    sd["lora_te1_text_model_encoder_layers_0_mlp_fc1.lora_down.weight"] = torch.ones(2, 8)
    sd["lora_te1_text_model_encoder_layers_0_mlp_fc1.lora_up.weight"] = torch.ones(8, 2)
    sd["lora_te2_encoder_block_0_layer_0_SelfAttention_q.alpha"] = torch.tensor(1.0)
    sd["text_encoder.text_model.encoder.layers.0.self_attn.q_proj.lora_A.weight"] = torch.ones(2, 8)
    sd["lora_unet_guidance_in_in_layer.lora_down.weight"] = torch.ones(2, 256)
    sd["lora_unet_guidance_in_in_layer.lora_up.weight"] = torch.ones(256, 2)
    sd["guidance_in.out_layer.lora_A.weight"] = torch.ones(2, 256)
    pairs, skipped = L.parse_lora(sd, cfg, L.weight_shapes(cfg))
    assert list(pairs) == ["double_blocks.0.txt_mlp.0"]
    assert skipped == ("guidance_in.in_layer", "guidance_in.out_layer",
                       "lora_te1_text_model_encoder_layers_0_mlp_fc1", "lora_te2_encoder_block_0_layer_0_SelfAttention_q",
                       "text_encoder.text_model.encoder.layers.0.self_attn.q_proj")


def _raises(sd, match, cfg=None):
    cfg = cfg or tiny_flux_config()
    with pytest.raises(ValueError, match=match):
        L.parse_lora(sd, cfg, L.weight_shapes(cfg))


def test_errors():
    flux, sd3 = tiny_flux_config(), tiny_sd3_config()
    _raises({"double_blocks.0.img_attn.mystery.lora_A.weight": torch.ones(2, 8)}, "mystery")
    _raises({"double_blocks.9.img_attn.qkv.lora_A.weight": torch.ones(2, 8)}, "double_blocks.9")   # beyond the depth
    _raises({"lora_unet_single_blocks_7_linear1.lora_down.weight": torch.ones(2, 8)}, "single_blocks_7_linear1")
    _raises({"transformer.transformer_blocks.0.attn.to_q.lora_A.weight": torch.ones(2, 8)}, "diffusers")
    _raises({"lora_transformer_single_transformer_blocks_0_attn_to_q.lora_down.weight": torch.ones(2, 8)},
            "lora_transformer_single")
    # a missing half, by either spelling
    sd = _one("img_in")
    del sd["img_in.lora_B.weight"]
    _raises(sd, "img_in.lora_A.weight")
    sd = _one("txt_in", kohya=True)
    del sd["lora_unet_txt_in.lora_down.weight"]
    _raises(sd, "lora_unet_txt_in.lora_up.weight")
    # mismatched ranks; wrong shapes
    sd = _one("txt_in")
    sd["txt_in.lora_B.weight"] = torch.ones(sd["txt_in.lora_B.weight"].shape[0], 3)
    _raises(sd, "txt_in.lora_B.weight.*rank")
    sd = _one("txt_in")
    sd["txt_in.lora_A.weight"] = torch.ones(2, 100)
    _raises(sd, "txt_in.lora_A.weight")
    sd = _one("single_blocks.0.linear1")
    sd["single_blocks.0.linear1.lora_B.weight"] = torch.ones(3 * flux.hidden_size, 2)         # no fc1 rows
    _raises(sd, "single_blocks.0.linear1")
    # the other family, both ways and both spellings
    _raises(_one("double_blocks.0.img_attn.qkv"), "FLUX module", cfg=sd3)
    _raises(_one("single_blocks.0.linear2", kohya=True), "FLUX module", cfg=sd3)
    _raises(_one("joint_blocks.0.x_block.attn.qkv", cfg=sd3), "SD3 module", cfg=flux)
    _raises(_one("joint_blocks.0.context_block.mlp.fc2", cfg=sd3, kohya=True), "SD3 module", cfg=flux)
    # LoHa / LoKr / DoRA, full-diff keys, conv LoRAs
    _raises({"lora_unet_img_in.hada_w1_a": torch.ones(2, 2)}, "LoHa")
    _raises({"lora_unet_img_in.lokr_w1": torch.ones(2, 2)}, "LoKr")
    sd = _one("txt_in")
    sd["txt_in.dora_scale"] = torch.ones(1, 128)
    _raises(sd, "DoRA")
    _raises({"double_blocks.0.img_attn.qkv.diff": torch.ones(2, 2)}, "full-difference")
    _raises({"double_blocks.0.img_attn.qkv.diff_b": torch.ones(2)}, "full-difference")
    _raises({"x_embedder.proj.lora_A.weight": torch.ones(2, 16, 2, 2),
             "x_embedder.proj.lora_B.weight": torch.ones(sd3.hidden_size, 2, 1, 1)}, "conv", cfg=sd3)
    _raises({"lora_unet_x_embedder_proj.lora_down.weight": torch.ones(2, 64)}, "conv", cfg=sd3)
    sd = _one("txt_in")
    sd["txt_in.lora_A.weight"] = sd["txt_in.lora_A.weight"][:, :, None, None]
    _raises(sd, "conv")
    _raises({"double_blocks.0.img_attn.qkv.weight": torch.ones(2, 2)}, "lora_A")             # not a LoRA key
    sd = _one("txt_in")
    sd["lora_unet_txt_in.lora_down.weight"] = sd["txt_in.lora_A.weight"]
    _raises(sd, "twice")


def test_read_lora_names(tmp_path):
    from safetensors.torch import save_file

    path = tmp_path / "my_style.safetensors"
    sd = _one("txt_in")
    save_file(sd, str(path))
    got, stem = L.read_lora(str(path))
    assert stem == "my_style" and sorted(got) == sorted(sd)
    assert L.read_lora(sd) == (sd, None)
    with pytest.raises(TypeError):
        L.read_lora(3)
