#!/usr/bin/env python
"""bench.py — images/sec of the denoise + decode hot path (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W [--impl ours|reference] [--workload C4|C2|C3] [--dump-outputs DIR]
  (N > 1: launched by torchrun, one rank per GPU; batch sharded by image, no per-step collective.)

--dump-outputs DIR writes what the last timed step returned (rank 0's shard) as DIR/<name>.npy, float32; the inputs are
seeded, so two builds run with the same arguments can be compared output for output (see dump_outputs).

A "step" = one batch of images through the whole hot path (sample_euler over all denoise steps + VAE decode).
Default workload C4: FLUX.1-schnell, 1024x1024 (latent 128x128), 4 steps, cfg 0, batch 4 images per GPU
(BASELINE.json configs[3] sharded 32 / 8 GPUs; SURVEY.md §8 table row C4), synthetic weights and embeddings.

Printed JSON (rank 0, one line): metric/value/unit/... per the driver contract, plus
  e2e          same metric through the public API with HOST inputs (pinned text embeddings -> H2D, host numpy noise
               -> H2D, uint8 images -> D2H) every step
  roofline     the tcgen05 GEMM kernel (dominant: 81% of C4 FLOPs): algorithmic FLOPs / CUDA-event time of every
               GEMM launch of one instrumented step, vs the measured bf16 peak (MEASURED_PEAKS.json)
  cpu_baseline the oracle (CPU restatement of the reference MLX path, "port") timed on the host cores on a bounded
               sample, extrapolated to images/sec (rank 0, N = 1 only)
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

WORKLOADS = {
    # name: (pipeline, model_version, latent, steps, cfg, shift, images per GPU, text_len)
    "C4": ("flux", "argmaxinc/mlx-FLUX.1-schnell", 128, 4, 0.0, 1.0, 4, 256),
    "C2": ("flux", "argmaxinc/mlx-FLUX.1-schnell", 64, 4, 0.0, 1.0, 1, 256),
    "C3": ("sd3", "argmaxinc/mlx-stable-diffusion-3-medium", 128, 50, 5.0, 3.0, 4, 589),
    # BASELINE.json configs[4]: FLUX.1-dev (loaded with the schnell config, quirk Q1), 50 steps, 8 images / 8 GPUs
    "C5": ("flux", "argmaxinc/mlx-FLUX.1-dev", 128, 50, 0.0, 1.0, 1, 512),
    # SURVEY §8 row f4 (not a BASELINE.json config): SD3.5-large, CLI defaults 1024x1024, 50 steps, cfg 5, shift 3
    "SD35": ("sd3", "argmaxinc/mlx-stable-diffusion-3.5-large", 128, 50, 5.0, 3.0, 2, 589),
}


def mmdit_flops_per_forward(cfg, n_img, n_txt):
    """SURVEY.md §8d: multiply-add = 2 FLOPs; per sample."""
    h = cfg.hidden_size
    S = n_img + n_txt
    total = 0.0
    for i in range(cfg.depth_multimodal):
        last_sd3 = (i == cfg.depth_multimodal - 1) and cfg.depth_unified == 0
        total += 24 * n_img * h * h + (6 if last_sd3 else 24) * n_txt * h * h + 4 * S * S * h
    total += cfg.depth_unified * (24 * S * h * h + 4 * S * S * h)
    total += 2 * n_img * 64 * h * 2 + 2 * n_txt * cfg.token_level_text_embed_dim * h
    return total


def workload_config(workload, per_gpu, world):
    """the `config` object of the JSON line: a function of the command line only, so both arms print the same one"""
    kind, mv, lat, steps, cfgw, shift, _, T = WORKLOADS[workload]
    global_batch = per_gpu * world
    return {"workload": f"{workload}: {mv} {lat * 8}x{lat * 8}, {steps} steps, cfg {cfgw}, "
                        f"{per_gpu} images/GPU (global batch {global_batch}), text len {T}; "
                        f"denoise (sample_euler) + VAE decode per step",
            "global_batch": global_batch, "parallelism": f"batch-sharded dp{world}, weights replicated",
            "l2": "inputs larger than L2 (the MMDiT weights, 23.8 GB for FLUX, are streamed once per forward)"}


def committed_gemm_traffic():
    """dram__bytes_read + dram__bytes_write of ONE launch of the dominant kernel (gemm2_tc_kernel, default configuration,
    on the largest C4 shape, 16384 x 12288 x 3072 + GELU) from the committed ncu capture of the kernel as it is timed
    here; algorithmic bytes of that launch are (16384 + 12288) * 3072 * 2 + 16384 * 12288 * 2 = 579 MB."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "r02_ncu_gemm_dram.json")))
        for r in d["rows"]:
            if r["config"] == "base" and r["shape_MNK"].startswith("16384 12288 3072"):
                return float(r["dram_bytes_total"]), ("profiles/r02_ncu_gemm_dram.json: gemm2_tc_kernel (default config) "
                                                      "16384x12288x3072+GELU, bytes per launch")
    except Exception:
        pass
    return None, None


def vae_roofline(decode_ms, images, lat, peaks):
    """The decode of the last timed step against both roofs (SURVEY.md §8d: 10.472 TFLOP and a 13.46 GB fusion model per
    1024^2 image, both linear in pixels).  HBM bytes per image are the ncu-measured dram__bytes of one whole decode
    (profiles/r02_vae_dram_B{1,4}_norm1.txt: 12.44 GB at batch 1, 13.36 GB at batch 4 for 1024^2), not re-measured here."""
    px = (lat / 128.0) ** 2
    ms_img = decode_ms / max(images, 1)
    tflop = 10.472 * px
    gb = (12.44 if images == 1 else 13.36) * px
    return {"ms_per_image": ms_img, "tflop_per_image": tflop, "tensor_tflops": tflop / (ms_img * 1e-3),
            "tensor_frac": tflop / (ms_img * 1e-3) / peaks["bf16_tflops"],
            "dram_gb_per_image": gb, "dram_gb_model": 13.46 * px, "dram_over_model": gb / (13.46 * px),
            "dram_gbs": gb / (ms_img * 1e-3), "hbm_frac": gb / (ms_img * 1e-3) / peaks["hbm_gbs"],
            "dram_source": "profiles/r02_vae_dram_B{1,4}_norm1.txt (ncu dram__bytes_read+write of one decode)",
            "bound": "tensor (3x3 convs at ~780 FLOP/B); the HBM-bound kernels are listed in DESIGN.md §5"}


DUMP_BYTES = 60 << 20      # all dumped arrays together stay under 64 MB


def dump_outputs(out_dir, arrays):
    """Writes each array as out_dir/<name>.npy in float32.  An array larger than its equal share of DUMP_BYTES is cut to
    a fixed sample: the elements at np.sort(np.random.RandomState(0).choice(numel, k, replace=False)) of the flattened
    array, written flat as <name>_sample.npy, so arrays of the same shape are sampled at the same positions in every
    run.  Returns {file name: shape written}."""
    os.makedirs(out_dir, exist_ok=True)
    cap = DUMP_BYTES // max(len(arrays), 1) // 4
    written = {}
    for name, t in arrays.items():
        a = t.detach().to(device="cpu", dtype=torch.float32).numpy()
        if a.size > cap:
            idx = np.sort(np.random.RandomState(0).choice(a.size, cap, replace=False))
            a, name = a.reshape(-1)[idx], name + "_sample"
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a))
        written[name + ".npy"] = list(a.shape)
    return written


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"bf16_tflops": d["bf16_tflops"], "bf16_tflops_sustained": d["bf16_tflops_sustained"],
                "hbm_gbs": d["hbm_gbs"], "source": "measured"}
    return {"bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "hbm_gbs": 6650.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md clocks line)."""

    def __init__(self, index: int):
        self.index = index
        self.lines = []
        self.proc = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for l in self.lines:
            parts = [p.strip() for p in l.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx = float(parts[1])
            except ValueError:
                continue
            for n, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ CPU baseline
def _host_threads() -> int:
    """physical cores when psutil can tell (SMT siblings only add contention to fp32 GEMMs), else the logical count"""
    try:
        import psutil

        n = psutil.cpu_count(logical=False)
        if n:
            return int(n)
    except Exception:
        pass
    return os.cpu_count() or 1


def cpu_baseline(workload: str, repeats: int = 2, budget_s: float = 40.0):
    """Times the oracle (CPU port of the reference MLX path) on a BOUNDED sample of the workload and extrapolates:
    ONE MMDiT forward for one image at the workload's full sequence length and width through a model with one block of
    each kind, scaled to the real depth by the algorithmic FLOP ratio (SURVEY.md §8d formula; the per-block GEMMs are
    > 99 % of the work); plus one VAE decode at 1/16 of the pixels scaled x16.  About 10-30 s of CPU work."""
    from dataclasses import replace

    from diffusionkit_b200.config import MODEL_CONFIGS, VAEDecoderConfig
    from diffusionkit_b200.weights import init_params, mmdit_param_specs, vae_decoder_param_specs
    from oracle.mmdit_ref import MMDiTRef
    from oracle.vae_ref import VAEDecoderRef, decode_latents_to_image
    from tests.oracle_bridge import ref_config

    kind, mv, lat, steps, cfgw, shift, per_gpu, T = WORKLOADS[workload]
    cores = _host_threads()
    torch.set_num_threads(cores)
    full = MODEL_CONFIGS[mv]
    g = torch.Generator().manual_seed(0)
    pooled = torch.randn((1, full.pooled_text_embed_dim), generator=g)
    t = torch.tensor([1000.0])
    ns = 1 if full.depth_unified > 0 else 0
    small = replace(full, depth_multimodal=2 if ns == 0 else 1, depth_unified=ns,
                    hidden_size_override=full.hidden_size)     # SD3: 2 blocks (the last one skips the text post-path)
    params = init_params(mmdit_param_specs(small), seed=0, dtype=torch.float32)
    ref = MMDiTRef(ref_config(small), params)
    ref.cache_modulation_params(pooled, t)

    def forward(lat_side, n_txt):
        latent = torch.randn((1, lat_side, lat_side, 16), generator=g)
        text = torch.randn((1, n_txt, full.token_level_text_embed_dim), generator=g)
        with torch.no_grad():
            t0 = time.time()
            ref(latent, text, t)
            return time.time() - t0

    t_begin = time.time()
    forward(max(lat // 4, 8), 32)                              # untimed: thread pool / allocator warm-up, 1/16 size
    t_small = forward(lat, T)
    n_fwd = 1
    while n_fwd < max(1, repeats) and time.time() - t_begin + t_small < budget_s:   # min over repeats: first-touch page
        t_small = min(t_small, forward(lat, T))                                     # faults / scheduler noise go away
        n_fwd += 1
    n_img = lat * lat // 4
    t_fwd = t_small * mmdit_flops_per_forward(full, n_img, T) / mmdit_flops_per_forward(small, n_img, T)
    del ref, params
    vp = init_params(vae_decoder_param_specs(VAEDecoderConfig()), seed=1, dtype=torch.float32)
    z = torch.randn((1, lat // 4, lat // 4, 16), generator=g)
    with torch.no_grad():
        t0 = time.time()
        decode_latents_to_image(VAEDecoderRef(vp), z)
        t_vae = (time.time() - t0) * 16
    reps = 2 if cfgw > 0 else 1
    sec_per_image = steps * reps * t_fwd + t_vae
    return {
        "value": 1.0 / sec_per_image, "unit": "images/s", "cores": cores, "kind": "port",
        "sample": (f"oracle fp32 torch-CPU, {cores} threads: 1 image, one MMDiT forward at full S={n_img}+{T}, "
                   f"h={full.hidden_size} through {small.depth_multimodal}+{small.depth_unified} blocks "
                   f"({t_small:.1f} s), scaled by the algorithmic FLOP ratio to "
                   f"{full.depth_multimodal}+{full.depth_unified} blocks -> {t_fwd:.1f} s/forward x {steps * reps} "
                   f"forwards; VAE decode at latent {lat // 4} x16 (linear in pixels) -> {t_vae:.1f} s"),
        "sec_per_image": sec_per_image, "forwards_timed": n_fwd,
    }


# ------------------------------------------------------------------------------------------------ our arm
def run_ours(args):
    import diffusionkit_b200 as dk
    from diffusionkit_b200 import dist as dkd, ops
    from diffusionkit_b200.config import MODEL_CONFIGS, VAEDecoderConfig
    from diffusionkit_b200.weights import init_params, mmdit_param_specs, vae_decoder_param_specs

    rank, world, local = dkd.init_distributed()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    kind, mv, lat, steps, cfgw, shift, per_gpu, T = WORKLOADS[args.workload]
    if args.images_per_gpu:
        per_gpu = args.images_per_gpu
    cfg = MODEL_CONFIGS[mv]
    dtype = torch.bfloat16 if kind == "flux" else torch.float16

    # weights: rank 0 materialises the synthetic parameters, one NCCL broadcast replicates them (the only collective)
    specs = mmdit_param_specs(cfg)
    t0 = time.time()
    wt = {}
    params = dkd.replicate_params(specs, lambda: init_params(specs, seed=0, dtype=dtype, device=dev), dtype, dev,
                                  timings=wt)
    vspecs = vae_decoder_param_specs(VAEDecoderConfig())
    vparams = dkd.replicate_params(vspecs, lambda: init_params(vspecs, seed=1, dtype=dtype, device=dev), dtype, dev,
                                   timings=wt)
    torch.cuda.synchronize()
    t_weights = time.time() - t0
    Pipe = dk.FluxPipeline if kind == "flux" else dk.DiffusionPipeline
    pipe = Pipe(w16=True, a16=True, shift=shift, model_version=mv, device=dev, params=params, vae_params=vparams)
    del params, vparams
    torch.cuda.empty_cache()

    # inputs: this rank's slice of the global batch (independent seeds / prompts per image)
    global_batch = per_gpu * world
    mine = list(dkd.shard_range(global_batch, rank, world))
    seeds = [1000 + i for i in mine]
    cond_all, pooled_all = pipe.synthetic_text_embeddings(n_images=global_batch, text_len=T)
    reps = 2 if cfgw > 0 else 1
    idx = [i + k * global_batch for k in range(reps) for i in mine]
    cond_host = cond_all[idx].contiguous().pin_memory()
    pooled_host = pooled_all[idx].contiguous().pin_memory()
    cond_dev, pooled_dev = cond_host.to(dev), pooled_host.to(dev)
    x_T = pipe.get_empty_latent(lat, lat)
    noise_dev = torch.cat([pipe.get_noise(s, x_T) for s in seeds]).to(dev)

    split = {"denoise": 0.0, "decode": 0.0}

    def step_device():
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        ev[0].record()
        latent, _ = pipe.denoise_latents(cond_dev, pooled_dev, num_steps=steps, cfg_weight=cfgw,
                                         latent_size=(lat, lat), seed=seeds, noise=noise_dev)
        ev[1].record()
        lat16 = ops.cast_to_16(latent, pipe.activation_dtype)
        images, images_u8 = pipe._decode(lat16, want_u8=True)
        ev[2].record()
        split["ev"] = ev
        return {"latents": latent, "images": images, "images_uint8": images_u8}

    def step_e2e():
        imgs, log = pipe.generate_image("", num_steps=steps, cfg_weight=cfgw, latent_size=(lat, lat), seed=seeds,
                                        verbose=False, conditioning=cond_host, pooled_conditioning=pooled_host)
        return imgs

    def barrier():
        if world > 1:
            torch.distributed.barrier()

    for _ in range(args.warmup):
        step_device()
    torch.cuda.synchronize()

    # ---- timed region 1: inputs resident in HBM
    clocks = ClockSampler(local)
    barrier()
    torch.cuda.synchronize()
    clocks.start()
    launches0 = ops.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        last = step_device()
    e1.record()
    torch.cuda.synchronize()
    barrier()
    launches = ops.launch_count() - launches0
    clk = clocks.stop()
    if args.dump_outputs and rank == 0:        # before anything else runs on the buffers the last step returned
        dumped = dump_outputs(args.dump_outputs, last)
        print(f"bench: wrote {dumped} to {args.dump_outputs}", file=sys.stderr, flush=True)
    del last
    split["denoise"] = split["ev"][0].elapsed_time(split["ev"][1])
    split["decode"] = split["ev"][1].elapsed_time(split["ev"][2])
    t_mine = e0.elapsed_time(e1) / 1e3
    t_dev = dkd.max_over_ranks(t_mine, dev)
    # per-rank device times of the timed region (the max is the metric; the spread attributes the N > 1 efficiency loss)
    per_rank = [t_mine]
    if world > 1:
        import torch.distributed as tdist

        buf = [torch.zeros(1, dtype=torch.float64, device=dev) for _ in range(world)]
        tdist.all_gather(buf, torch.tensor([t_mine], dtype=torch.float64, device=dev))
        per_rank = [float(b.item()) for b in buf]

    # ---- timed region 2: end to end through the public API with host inputs / outputs
    step_e2e()  # warm the host-side path (pinned staging, PIL)
    barrier()
    torch.cuda.synchronize()
    w0 = time.perf_counter()
    for _ in range(args.steps):
        step_e2e()
    torch.cuda.synchronize()
    t_e2e = dkd.max_over_ranks(time.perf_counter() - w0, dev)
    barrier()

    # ---- instrumented step: CUDA events around every GEMM launch (roofline of the dominant kernel)
    gemm_stats = {"flops": 0.0, "events": []}
    orig_gemm = ops.gemm

    def timed_gemm(A, W, *a, **kw):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        out = orig_gemm(A, W, *a, **kw)
        e.record()
        n = kw.get("N") or (W.shape[1] if kw.get("w_n_major") else W.shape[0])
        gemm_stats["flops"] += 2.0 * A.shape[0] * A.shape[1] * n
        gemm_stats["events"].append((s, e))
        return out

    ops.gemm = timed_gemm
    graphs_were = pipe.mmdit.use_cuda_graphs
    pipe.mmdit.use_cuda_graphs = False          # the instrumented step must launch kernel by kernel
    try:
        latent, _ = pipe.denoise_latents(cond_dev, pooled_dev, num_steps=steps, cfg_weight=cfgw,
                                         latent_size=(lat, lat), seed=seeds, noise=noise_dev)
    finally:
        ops.gemm = orig_gemm
        pipe.mmdit.use_cuda_graphs = graphs_were
    torch.cuda.synchronize()
    t_gemm = sum(s.elapsed_time(e) for s, e in gemm_stats["events"]) / 1e3
    n_gemm = len(gemm_stats["events"])

    peaks = load_peaks()
    n_images = global_batch * args.steps
    value = n_images / t_dev
    n_img_tok, hp = (lat // 2) ** 2, lat // 2
    flops_img = mmdit_flops_per_forward(cfg, n_img_tok, T) * steps * reps
    mmdit_frac = (flops_img * per_gpu * args.steps / t_dev) / (peaks["bf16_tflops_sustained"] * 1e12)
    achieved = gemm_stats["flops"] / t_gemm / 1e12 if t_gemm > 0 else 0.0
    h2d = cond_host.numel() * cond_host.element_size() + pooled_host.numel() * pooled_host.element_size() + \
        noise_dev.numel() * 4
    d2h = len(seeds) * (lat * 8) * (lat * 8) * 3

    if rank != 0:
        return
    line = {
        "metric": "images/sec at 1024x1024 (FLUX.1-schnell 4-step)" if args.workload == "C4" else f"images/sec ({args.workload})",
        "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": t_dev / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16" if dtype == torch.bfloat16 else "fp16", "data": "synthetic",
        "config": workload_config(args.workload, per_gpu, world),
        "e2e": {"value": n_images / t_e2e, "unit": "images/s", "h2d_bytes_per_step": int(h2d),
                "d2h_bytes_per_step": int(d2h)},
        "gpu_launches": int(launches),
        "clocks": clk,
        "roofline": {"bound": "tensor",
                     "kernel": "gemm2_tc_kernel / gemm_tc_kernel (tcgen05 GEMMs: every nn.Linear of the MMDiT)",
                     "achieved": achieved, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
                     "frac": achieved / peaks["bf16_tflops"], "traffic": committed_gemm_traffic()[0],
                     "traffic_source": committed_gemm_traffic()[1],
                     "peak_source": f"{peaks['source']} bf16 burst (sustained {peaks['bf16_tflops_sustained']})",
                     "launches_timed": n_gemm, "gemm_seconds_of_one_step": t_gemm},
        "mmdit_tensor_frac_sustained": mmdit_frac,
        "last_step_ms": {"denoise": split["denoise"], "decode": split["decode"]},
        "denoise_tflops_per_image": flops_img / 1e12,
        "per_rank_step_ms": [round(t / args.steps * 1e3, 3) for t in per_rank],
        "weights_init_broadcast_s": t_weights,
        # the one-time weight replication, split: lazy NCCL communicator creation / rank-0 init / the broadcast itself
        "weights_timing": {k: (round(v, 4) if isinstance(v, float) else v) for k, v in wt.items()},
    }
    try:
        line["vae_roofline"] = vae_roofline(split["decode"], per_gpu, lat, peaks)
    except Exception:  # informational only
        pass
    if world == 1 and not args.no_cpu_baseline:
        try:
            line["cpu_baseline"] = cpu_baseline(args.workload)
        except Exception as ex:  # the baseline is reported, never load-bearing
            line["cpu_baseline"] = {"value": None, "unit": "images/s", "cores": os.cpu_count(), "kind": "port",
                                    "sample": f"failed: {ex!r}"}
    print(json.dumps(line), flush=True)


def run_reference(args):
    """Reference arm: the reference's own implementation cannot run here (MLX is Apple-only and absent; its torch
    modules need argmaxtools/coremltools), so this times the oracle port on the host cores, all threads."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    kind, mv, lat, steps, cfgw, shift, per_gpu, T = WORKLOADS[args.workload]
    world = int(os.environ.get("WORLD_SIZE", "1"))
    # one bounded sample, min over `--steps` timed forwards (after the untimed warm-up forward) within a time budget
    best = cpu_baseline(args.workload, repeats=max(1, args.steps), budget_s=150.0)
    global_batch = (args.images_per_gpu or per_gpu) * world
    line = {
        "impl": "reference",
        "metric": "images/sec at 1024x1024 (FLUX.1-schnell 4-step)" if args.workload == "C4" else f"images/sec ({args.workload})",
        "value": best["value"], "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": best["sec_per_image"] * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        # the same workload description as the GPU arm prints for these arguments
        "config": workload_config(args.workload, args.images_per_gpu or per_gpu, world),
        # how the number was obtained: NOT a full run of the workload — see cpu_baseline.sample
        "extrapolated": True,
        "extrapolation": ("CPU oracle port (fp32 torch, all host threads): one image, one full-sequence MMDiT forward "
                          "through a truncated depth scaled by the algorithmic FLOP ratio + a 1/16-pixel VAE decode x16; "
                          f"min of {best['forwards_timed']} timed forward(s)"),
        "cpu_baseline": {k: best[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": best["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="C4", choices=sorted(WORKLOADS))
    ap.add_argument("--images-per-gpu", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (float32, at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)
    if torch.distributed.is_available() and torch.distributed.is_initialized():
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
