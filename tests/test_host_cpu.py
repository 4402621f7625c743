"""CPU: host logic, config/parameter trees, C-ABI surface (no compute calls without a GPU)."""
import ctypes
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import diffusionkit_b200 as dk
from diffusionkit_b200 import _lib, dist as dkdist
from diffusionkit_b200.config import FLUX_SCHNELL, MODEL_CONFIGS, SD3_2b, PositionalEncoding, VAEDecoderConfig
from diffusionkit_b200.pipeline import DiffusionPipeline, FluxPipeline
from diffusionkit_b200.sampler import FluxSampler, ModelSamplingDiscreteFlow
from diffusionkit_b200.weights import init_params, mmdit_param_specs, param_count, vae_decoder_param_specs

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KATS = json.load(open(os.path.join(ROOT, "tests", "golden", "schedule_kats.json")))


def test_header_and_binding_agree():
    hs = set(_lib.header_symbols())
    assert hs == set(_lib.SIGNATURES), (hs - set(_lib.SIGNATURES), set(_lib.SIGNATURES) - hs)


def test_library_loads_and_exports_every_symbol():
    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__

        __graft_entry__.build()
    lib = _lib.load()
    for name in _lib.header_symbols():
        assert hasattr(lib, name), name
    assert b"sm_100a" in lib.dk_version()
    # error path without a GPU: create must fail cleanly with a message, not crash
    if not torch.cuda.is_available():
        h = ctypes.c_void_p()
        rc = lib.dk_ctx_create(0, ctypes.byref(h))
        assert rc != 0 and len(lib.dk_last_error()) > 0


def test_no_cpu_fallback():
    """without a CUDA device the pipeline and the ops refuse with DkError; the devices are hidden from a child process,
    so this is checked on a machine with a GPU too"""
    code = ("import sys\nsys.path.insert(0, sys.argv[1])\nimport torch\nimport diffusionkit_b200 as dk\n"
            "from diffusionkit_b200 import ops\nassert not torch.cuda.is_available()\n"
            "for call in (lambda: dk.FluxPipeline(w16=True, a16=True),\n"
            "             lambda: ops.gemm(torch.zeros(8, 8, dtype=torch.bfloat16), torch.zeros(8, 8, dtype=torch.bfloat16))):\n"
            "    try:\n        call()\n    except dk.DkError as e:\n        print('DkError:', e)\n")
    out = subprocess.run([sys.executable, "-c", code, ROOT], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and out.stdout.count("DkError:") == 2, out.stdout + out.stderr


def test_pipeline_argument_errors():
    with pytest.raises(KeyError):
        DiffusionPipeline(w16=True, a16=True, model_version="no/such-model")
    with pytest.raises(NotImplementedError):
        DiffusionPipeline(w16=False, a16=False)          # fp32 path not provided
    # valid arguments, but no CUDA device: refuses loudly.  The devices are hidden from a child process, so this is
    # checked on a machine with a GPU too (where the same call would build the model).
    code = ("import sys\nsys.path.insert(0, sys.argv[1])\nfrom diffusionkit_b200 import FluxPipeline\n"
            "from diffusionkit_b200._lib import DkError\ntry:\n"
            "    FluxPipeline(w16=True, a16=True, quantize_mmdit=True,\n"
            "                 model_version='argmaxinc/mlx-FLUX.1-schnell-4bit-quantized')\n"
            "except DkError as e:\n    print('DkError:', e)\n")
    out = subprocess.run([sys.executable, "-c", code, ROOT], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "DkError:" in out.stdout, out.stdout + out.stderr


def test_presets_match_reference_values():
    # reference mlx/config.py:78-95
    assert SD3_2b.hidden_size == 1536 and SD3_2b.num_heads == 24 and SD3_2b.depth_multimodal == 24
    assert SD3_2b.depth_unified == 0 and SD3_2b.dtype == torch.float16 and not SD3_2b.use_qk_norm
    assert SD3_2b.pos_embed_type == PositionalEncoding.LearnedInputEmbedding and SD3_2b.max_latent_resolution == 192
    f = FLUX_SCHNELL
    assert (f.hidden_size, f.num_heads, f.depth_multimodal, f.depth_unified) == (3072, 24, 19, 38)
    assert f.rope_axes_dim == (16, 56, 56) and f.pooled_text_embed_dim == 768 and f.use_qk_norm
    assert f.patchify_via_reshape and f.pos_embed_type == PositionalEncoding.PreSDPARope and f.dtype == torch.bfloat16
    assert MODEL_CONFIGS["argmaxinc/mlx-FLUX.1-dev"] is FLUX_SCHNELL      # quirk Q1
    from diffusionkit_b200.config import SD3_8b

    assert (SD3_8b.hidden_size, SD3_8b.num_heads, SD3_8b.head_dim, SD3_8b.depth_multimodal) == (2432, 38, 64, 38)
    assert SD3_8b.use_qk_norm and SD3_8b.dtype == torch.bfloat16          # reference mlx/config.py:74-76
    assert MODEL_CONFIGS["argmaxinc/mlx-stable-diffusion-3.5-large-4bit-quantized"] is SD3_8b
    assert MODEL_CONFIGS["argmaxinc/mlx-FLUX.1-schnell-4bit-quantized"] is FLUX_SCHNELL


def test_parameter_trees():
    fs = mmdit_param_specs(FLUX_SCHNELL)
    names = {n for n, _, _ in fs}
    assert "multimodal_transformer_blocks.18.text_transformer_block.qk_norm.k_norm.weight" in names
    assert "unified_transformer_blocks.37.transformer_block.adaLN_modulation.layers.1.weight" in names
    assert not any(n.endswith("k_proj.bias") for n in names)               # quirk Q3
    shapes = {n: s for n, s, _ in fs}
    assert shapes["x_embedder.proj.weight"] == (3072, 1, 1, 64)
    assert shapes["unified_transformer_blocks.0.transformer_block.adaLN_modulation.layers.1.weight"] == (9216, 3072)
    assert 11.8e9 < param_count(fs) < 12.0e9                                # SURVEY.md App. B.1: ~11.9 B
    ss = mmdit_param_specs(SD3_2b)
    sn = {n: s for n, s, _ in ss}
    assert sn["x_pos_embedder.pos_embed.weight"] == (36864, 1536) and sn["x_embedder.proj.weight"] == (1536, 2, 2, 16)
    last_txt = "multimodal_transformer_blocks.23.text_transformer_block"
    assert sn[last_txt + ".adaLN_modulation.layers.1.weight"] == (2 * 1536, 1536)       # skip_post_sdpa
    assert (last_txt + ".attn.o_proj.weight") not in sn and (last_txt + ".mlp.fc1.weight") not in sn
    assert 2.0e9 < param_count(ss) < 2.2e9
    vs = {n: s for n, s, _ in vae_decoder_param_specs(VAEDecoderConfig())}
    # up_blocks[0] is the 256->128 full-resolution block and has no upsample (vae.py:367-379)
    assert vs["up_blocks.0.resnets.0.conv1.weight"] == (128, 3, 3, 256) and "up_blocks.0.upsample.weight" not in vs
    assert vs["up_blocks.0.resnets.0.conv_shortcut.weight"] == (128, 256)
    assert vs["up_blocks.3.upsample.weight"] == (512, 3, 3, 512) and vs["conv_out.weight"] == (3, 3, 3, 128)
    assert vs["mid_blocks.1.query_proj.weight"] == (512, 512)


def test_synthetic_init_is_deterministic():
    specs = mmdit_param_specs(dk.config.tiny_sd3_config())
    a = init_params(specs, seed=3, dtype=torch.float32)
    b = init_params(specs, seed=3, dtype=torch.float32)
    c = init_params(specs, seed=4, dtype=torch.float32)
    assert all(torch.equal(a[k], b[k]) for k in a) and not torch.equal(a["context_embedder.weight"],
                                                                       c["context_embedder.weight"])
    w = a["context_embedder.weight"]
    assert abs(float(w.std()) - 1 / np.sqrt(w.shape[1])) < 0.02 / np.sqrt(w.shape[1]) * 10


def _bare(cls, sampler):
    p = object.__new__(cls)
    p.sampler = sampler
    return p


def test_product_schedules_match_kats():
    for key, val in KATS.items():
        if not key.startswith(("flux_n", "sd3_n")):
            continue
        fam, n, shift = key.split("_")
        n, shift = int(n[1:]), float(shift[5:])
        if fam == "flux":
            p = _bare(FluxPipeline, FluxSampler(shift))
        else:
            p = _bare(DiffusionPipeline, ModelSamplingDiscreteFlow(shift))
        sig = p.get_sigmas(p.sampler, n)
        assert sig.dtype == np.float32 and len(sig) == n + 1
        assert np.allclose(sig, np.array(val["sigmas"]), rtol=2e-6, atol=1e-7), key
        assert p.max_denoise(sig)
    p = _bare(DiffusionPipeline, ModelSamplingDiscreteFlow(3.0))
    nz = p.get_noise(0, p.get_empty_latent(4, 4))
    assert np.allclose(nz[0, 0, 0, :].numpy(), np.array(KATS["noise_seed0_4x4_nhwc_0_0_0_c"]), atol=1e-6)
    assert float(p.get_empty_latent(2, 2)[0, 0, 0, 0]) == np.float32(0.0609)


def test_get_noise_equals_global_numpy_rng():
    """RandomState(seed) reproduces the reference's np.random.seed(seed); np.random.randn(...) draw exactly, and the
    threaded batch path equals per-seed draws"""
    p = _bare(DiffusionPipeline, ModelSamplingDiscreteFlow(3.0))
    x_T = p.get_empty_latent(6, 10)
    for seed in (0, 7, 123456):
        np.random.seed(seed)
        want = torch.from_numpy(np.random.randn(1, 16, 6, 10)).permute(0, 2, 3, 1).to(torch.float32)
        assert torch.equal(p.get_noise(seed, x_T), want)
    batch = p._get_noise_batch([3, 4, 5], x_T)
    assert torch.equal(batch, torch.cat([p.get_noise(s, x_T) for s in (3, 4, 5)]))


def test_latent_formats():
    assert dk.SD3LatentFormat().process_out(0.0) == 0.0609 and abs(dk.FluxLatentFormat().process_out(0.3611) - 1.1159) < 1e-12
    lf = dk.FluxLatentFormat()
    assert abs(lf.process_in(lf.process_out(0.7)) - 0.7) < 1e-12


def test_shard_range_partitions_the_batch():
    for n, w in [(32, 8), (8, 8), (5, 4), (3, 8), (0, 2)]:
        parts = [list(dkdist.shard_range(n, r, w)) for r in range(w)]
        assert sum(parts, []) == list(range(n))
        assert max(len(p) for p in parts) - min(len(p) for p in parts) <= 1


_GLOO_WORKER = r'''
import os, sys, torch
sys.path.insert(0, os.environ["DK_ROOT"])
import torch.distributed as dist
from diffusionkit_b200 import dist as dkd
from diffusionkit_b200.config import tiny_sd3_config
from diffusionkit_b200.weights import init_params, mmdit_param_specs
rank, world, _ = dkd.init_distributed("gloo")
specs = mmdit_param_specs(tiny_sd3_config())
called = []
def init_fn():
    called.append(rank)
    return init_params(specs, seed=11, dtype=torch.bfloat16)
views = dkd.replicate_params(specs, init_fn, torch.bfloat16, "cpu", src=0)
ref = init_params(specs, seed=11, dtype=torch.bfloat16)
assert all(torch.equal(views[k], ref[k]) for k in ref), "broadcast mismatch"
assert called == ([0] if rank == 0 else []), called           # only rank 0 materialises weights
mine = list(dkd.shard_range(5, rank, world))
t = torch.full((2,), float(rank))
g = dkd.gather_to_rank0(t)
assert (g is not None) == (rank == 0)
assert dkd.max_over_ranks(float(rank), "cpu") == world - 1
print("OK", rank, mine)
'''


def test_gloo_world2_weight_broadcast_and_sharding(tmp_path):
    script = tmp_path / "w.py"
    script.write_text(_GLOO_WORKER)
    import socket

    outs, ok = [], False
    for attempt in range(2):                               # one retry: the rendezvous can lose a race on a loaded host
        with socket.socket() as sock:                      # a free port: a fixed one can still be in TIME_WAIT
            sock.bind(("127.0.0.1", 0))
            port = sock.getsockname()[1]
        env = dict(os.environ, DK_ROOT=ROOT, MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), WORLD_SIZE="2")
        procs = [subprocess.Popen([sys.executable, str(script)], env=dict(env, RANK=str(r), LOCAL_RANK=str(r)),
                                  stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True) for r in range(2)]
        outs = [p.communicate(timeout=180)[0] for p in procs]
        ok = all(p.returncode == 0 for p in procs)
        if ok:
            break
    assert ok, outs
    assert "OK 0 [0, 1, 2]" in outs[0] and "OK 1 [3, 4]" in outs[1]


def test_read_image_resize_rule(tmp_path):
    """read_image (reference mlx/__init__.py:536-551): sizes are cut to multiples of 64 with a LANCZOS resize, RGB(A)
    uint8 -> [-1, 1] float; host-only logic, no device needed"""
    import numpy as np
    from PIL import Image

    from diffusionkit_b200.pipeline import DiffusionPipeline

    rng = np.random.RandomState(0)
    arr = rng.randint(0, 256, (130, 200, 4), dtype=np.uint8)
    path = str(tmp_path / "im.png")
    Image.fromarray(arr).save(path)
    u8 = DiffusionPipeline._load_image_u8(None, path)
    assert u8.shape == (128, 192, 4) and u8.dtype == np.uint8
    same = DiffusionPipeline._load_image_u8(None, arr[:128, :192])
    assert same.shape == (128, 192, 3) and np.array_equal(same, arr[:128, :192, :3])   # already aligned: untouched
    f = DiffusionPipeline.read_image(DiffusionPipeline.__new__(DiffusionPipeline), arr[:64, :64])
    assert tuple(f.shape) == (1, 64, 64, 3) and abs(float(f[0, 0, 0, 0]) - (arr[0, 0, 0] / 255 * 2 - 1)) < 1e-6
    import pytest

    with pytest.raises(ValueError):
        DiffusionPipeline._load_image_u8(None, arr[:40, :40])
    with pytest.raises(ValueError):
        DiffusionPipeline._load_image_u8(None, arr[:64, :64, 0])


def test_header_is_plain_c(tmp_path):
    """include/dkb200.h is the FFI contract: it has to compile as C99 and as C++ on its own, and a C program that only
    includes it must link against the shared library"""
    import shutil

    hdr = os.path.join(ROOT, "include", "dkb200.h")
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-fsyntax-only", "-x", "c", hdr])
    subprocess.check_call(["g++", "-std=c++17", "-Wall", "-fsyntax-only", "-x", "c++", hdr])
    if not os.path.exists(_lib.LIB_PATH):
        pytest.skip("library not built")
    src = tmp_path / "abi.c"
    src.write_text('#include <stdio.h>\n#include "dkb200.h"\n'
                   'int main(void) { dk_ctx* c = NULL; int rc = dk_ctx_create(0, &c);\n'
                   '  printf("%s|%d|%s\\n", dk_version(), rc, rc ? dk_last_error() : "");\n'
                   '  if (c) dk_ctx_destroy(c); return 0; }\n')
    exe = tmp_path / "abi"
    libdir = os.path.dirname(_lib.LIB_PATH)
    subprocess.check_call(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe),
                           "-L", libdir, "-ldkb200", f"-Wl,-rpath,{libdir}"])
    out = subprocess.run([str(exe)], capture_output=True, text=True, timeout=60)
    assert out.returncode == 0 and "sm_100a" in out.stdout, out.stdout + out.stderr
    if not torch.cuda.is_available():
        assert "|0|" not in out.stdout          # no device here: create fails with a message instead of crashing


def test_integration_doc_struct_is_current():
    """INTEGRATION.md's ctypes stub of struct dk_gemm_args is the generated one (a stale, shorter stub makes dk_gemm read
    past the end of the caller's struct), and the binding it is generated from has the header's fields in the header's order"""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import re

    import gen_integration_stub as gen

    doc = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    assert gen.block() in doc, "run tools/gen_integration_stub.py and paste its output into INTEGRATION.md section 2"
    hdr = open(os.path.join(ROOT, "include", "dkb200.h")).read()
    body = hdr[hdr.index("typedef struct dk_gemm_args"):hdr.index("} dk_gemm_args;")]
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = []
    for decl in body.split("{", 1)[1].split(";"):
        decl = decl.strip()
        if not decl:
            continue
        first, *rest = decl.split(",")
        names.append(re.findall(r"([A-Za-z_][A-Za-z0-9_]*)\s*$", first.strip())[0])
        names += [r.strip().lstrip("*").strip() for r in rest]
    assert names == [n for n, _ in _lib.GemmArgs._fields_], (names, [n for n, _ in _lib.GemmArgs._fields_])


def test_bench_vae_roofline_helper():
    """bench.py's VAE roofline object: pure arithmetic on the decode time of the last step"""
    import importlib.util

    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    peaks = {"bf16_tflops": 1736.7, "bf16_tflops_sustained": 1473.8, "hbm_gbs": 6484.6, "source": "measured"}
    r = bench.vae_roofline(40.4, 4, 128, peaks)
    assert abs(r["ms_per_image"] - 10.1) < 1e-9 and abs(r["tensor_frac"] - 10.472 / 10.1e-3 / 1736.7) < 1e-9
    assert 0.9 < r["dram_over_model"] < 1.0 and 0.15 < r["hbm_frac"] < 0.25
    r2 = bench.vae_roofline(3.4, 1, 64, peaks)                       # C2: 512^2, a quarter of the pixels
    assert abs(r2["tflop_per_image"] - 10.472 / 4) < 1e-9 and abs(r2["dram_gb_model"] - 13.46 / 4) < 1e-9


def test_bench_dump_outputs(tmp_path):
    """bench.py --dump-outputs: float32 .npy files under 64 MB in all; arrays over their share are sampled at the same
    positions in every run (C4 shapes: 4 images of 1024^2)"""
    import importlib.util

    import numpy as np

    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    g = torch.Generator().manual_seed(0)
    images = torch.rand((4, 1024, 1024, 3), generator=g)
    arrays = {"latents": torch.randn((4, 128, 128, 16), generator=g), "images": images,
              "images_uint8": (images * 255).to(torch.uint8)}
    a = bench.dump_outputs(str(tmp_path / "a"), arrays)
    b = bench.dump_outputs(str(tmp_path / "b"), arrays)
    assert a == b == {"latents.npy": [4, 128, 128, 16], "images_sample.npy": [a["images_sample.npy"][0]],
                      "images_uint8_sample.npy": [a["images_sample.npy"][0]]}
    assert sum(os.path.getsize(p) for p in (tmp_path / "a").iterdir()) < 64e6
    for name in a:
        x, y = np.load(tmp_path / "a" / name), np.load(tmp_path / "b" / name)
        assert x.dtype == np.float32 and np.array_equal(x, y), name
    assert np.array_equal(np.load(tmp_path / "a" / "latents.npy"), arrays["latents"].numpy())
    img, u8 = np.load(tmp_path / "a" / "images_sample.npy"), np.load(tmp_path / "a" / "images_uint8_sample.npy")
    assert np.array_equal((img * 255).astype(np.uint8).astype(np.float32), u8)     # same positions in both arrays


def test_attention_trace_numbers_quoted_in_design():
    """DESIGN.md §8's clock table is regenerated from the committed timestamp traces (tools/analyze_att_trace.py)"""
    import importlib.util

    spec = importlib.util.spec_from_file_location("att_trace", os.path.join(ROOT, "tools", "analyze_att_trace.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    base = mod.summarize(os.path.join(ROOT, "profiles", "r02_att_trace_call21.txt"))
    streamed = mod.summarize(os.path.join(ROOT, "profiles", "r02_att_trace_streamed_call22.txt"))
    assert 3250 <= base["period"] <= 3350 and 3100 <= streamed["period"] <= 3200
    assert 2080 <= base["tiles"][0]["softmax_total"] <= 2180 and 1860 <= streamed["tiles"][0]["softmax_total"] <= 1960
    assert 650 <= streamed["tiles"][0]["pv1_qk_issue"] <= 800          # 12 MMAs = 768 tensor clocks, issue is back-pressured
    design = open(os.path.join(ROOT, "DESIGN.md")).read()
    assert "**3300 (62 %)**" in design and "**3144 (65 %)**" in design
