"""LoRA merge cost at full size: FLUX.1-schnell (synthetic weights, bf16) with a synthetic full-coverage LoRA (one
adapter on every Linear of the model) at ranks 16 and 64.

One process, one card.  Per rank it times, with the merger's stage timer (CUDA synchronise between stages):
  the first load_lora  split into parse / H2D (factors to the device, fp32) / pristine copies / merge GEMMs
  a reload under the same name with a new scale (pristine copies already exist: parse + H2D + re-merge)
  unload_lora          copies the pristine weights back and frees them
The merge GEMMs are compared with the HBM floor of the data they must move: every adapted weight's W0 read plus its W
written, 2 x 2 bytes per element, at the 6.48 TB/s DESIGN.md §5 uses.  Then the C4 step time (1024^2, 4 steps,
4 images) with and without a rank-16 adapter, runs alternating: the merged model runs the same kernels and shapes.
The card's name and power limit are read in the same run.

  python tools/bench_lora.py [--rounds 4] [--out FILE]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_TBPS = 6.48


def card_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["sm_clock_max"] = [s.strip() for s in q.split(",")]
    except Exception as e:                                        # the name above still identifies the card
        info["power_limit"] = f"unavailable ({e})"
    return info


def synthetic_lora(pipe, rank, seed):
    """PEFT-style bf16 LoRA on every upstream Linear of the pipeline's FLUX model"""
    from diffusionkit_b200 import model_io

    cfg, views = pipe.config, pipe.mmdit.weight_views
    g = torch.Generator().manual_seed(seed)
    sd = {}
    for m in model_io.flux_linear_modules(cfg.depth_multimodal, cfg.depth_unified):
        dim, parts = model_io.flux_linear_route(m, cfg.mlp_ratio)
        ws = [views[n + ".weight"].shape for n, _ in parts]
        out_f, in_f = (sum(s[0] for s in ws), ws[0][1]) if dim == 0 else (ws[0][0], sum(s[1] for s in ws))
        sd[m + ".lora_A.weight"] = (torch.randn((rank, in_f), generator=g) / in_f ** 0.5).to(torch.bfloat16)
        sd[m + ".lora_B.weight"] = (0.1 * torch.randn((out_f, rank), generator=g) / rank ** 0.5).to(torch.bfloat16)
    return sd


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=4, help="timed (plain, adapter) C4 pairs, order alternating")
    ap.add_argument("--out", default=None, help="also write the JSON result here")
    args = ap.parse_args()

    import diffusionkit_b200 as dk
    from diffusionkit_b200.config import MODEL_CONFIGS
    from diffusionkit_b200.weights import init_params, mmdit_param_specs

    if not torch.cuda.is_available():
        raise SystemExit("bench_lora needs a CUDA device")
    dev = torch.device("cuda", 0)
    mv, steps, images, lat, T = "argmaxinc/mlx-FLUX.1-schnell", 4, 4, 128, 256
    cfg = MODEL_CONFIGS[mv]
    params = init_params(mmdit_param_specs(cfg), seed=0, dtype=torch.bfloat16, device=dev)
    pipe = dk.FluxPipeline(w16=True, a16=True, model_version=mv, device=dev, params=params, load_decoder=False)
    del params
    torch.cuda.synchronize()

    def timed(fn):
        pipe._lora.timing = {} if pipe._lora is not None else None
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        total = 1e3 * (time.perf_counter() - t0)
        stages = {k: round(v, 2) for k, v in (pipe._lora.timing or {}).items()}
        pipe._lora.timing = None
        return out, dict(stages, total_ms=round(total, 2))

    pipe._lora = None
    merges = {}
    for rank in (16, 64):
        t0 = time.perf_counter()
        lora = synthetic_lora(pipe, rank, seed=rank)
        gen_s = time.perf_counter() - t0
        if pipe._lora is None:                                    # the merger is built by the first load_lora
            from diffusionkit_b200.lora import LoraMerger

            pipe._lora = LoraMerger(pipe.mmdit)
        info, first = timed(lambda: pipe.load_lora(lora, scale=1.0, name="bench"))
        mem_gb = torch.cuda.memory_allocated(dev) / 1e9
        pristine_gb = sum(t.numel() * t.element_size() for t in pipe._lora.pristine.values()) / 1e9
        _, reload = timed(lambda: pipe.load_lora(lora, scale=0.5, name="bench"))
        _, unload = timed(lambda: pipe.unload_lora())
        n_el = sum(v.numel() for n, v in pipe.mmdit.weight_views.items())
        floor_ms = 2 * 2 * n_el / (HBM_TBPS * 1e12) * 1e3
        merges[f"rank{rank}"] = {
            "lora_params": sum(t.numel() for t in lora.values()), "synthetic_generation_s": round(gen_s, 1),
            "info": info._asdict(), "first_load": first, "reload_new_scale": reload, "unload": unload,
            "device_memory_after_first_load_GB": round(mem_gb, 2), "pristine_copies_GB": round(pristine_gb, 2),
            "hbm_floor_ms": round(floor_ms, 2), "hbm_floor_bytes": 4 * n_el,
            "merge_over_floor_first": round(first["merge_ms"] / floor_ms, 2),
            "merge_over_floor_reload": round(reload["merge_ms"] / floor_ms, 2),
        }
        del lora
        print(json.dumps({f"rank{rank}": merges[f"rank{rank}"]}), flush=True)

    # C4 step time with and without an adapter, alternating
    lora16 = synthetic_lora(pipe, 16, seed=16)
    cond, pooled = pipe.synthetic_text_embeddings(n_images=images, text_len=T)
    cond, pooled = cond.to(dev), pooled.to(dev)
    seeds = [1000 + i for i in range(images)]

    def run(with_lora):
        if with_lora:
            pipe.load_lora(lora16, name="c4")
        else:
            pipe.unload_lora()
        _, it = pipe.denoise_latents(cond, pooled, num_steps=steps, latent_size=(lat, lat), seed=seeds)
        return [1e3 * t for t in it]

    for w in (False, True):                                       # warm-up
        run(w)
    step_ms = {"plain": [], "lora_r16": []}
    for r in range(args.rounds):
        for w in ((False, True) if r % 2 == 0 else (True, False)):
            step_ms["lora_r16" if w else "plain"] += run(w)
    pipe.unload_lora()

    def summary(v):
        return {"mean": round(statistics.mean(v), 2), "stdev": round(statistics.stdev(v), 2), "min": round(min(v), 2),
                "max": round(max(v), 2), "n": len(v)}

    a, b = summary(step_ms["plain"]), summary(step_ms["lora_r16"])
    res = {
        "card": card_info(),
        "model": "FLUX.1-schnell synthetic weights (bf16), full-coverage synthetic LoRA (every Linear)",
        "timing_note": "host wall clock with a CUDA synchronise after each stage; parse reads an in-memory dict",
        "hbm_floor_note": f"bytes of W0 read + W written over every adapted weight at {HBM_TBPS} TB/s (arithmetic)",
        "merge": merges,
        "c4": {"workload": f"{lat * 8}x{lat * 8}, {steps} steps, {images} images", "step_ms_note":
               "CUDA events around each Euler step, warm-up excluded, runs alternating", "plain": a, "lora_r16": b,
               "lora_minus_plain_ms": round(b["mean"] - a["mean"], 2)},
    }
    print(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
