"""Inpainting cost at full size: FLUX.1-schnell (synthetic weights), 1024^2, 4 steps, 4 images, denoise = 1.0.

One process, one card.  Alternates plain img2img and inpainting runs with the same seeds, noise and image, and reports
the CUDA-event step times of each (sample_euler's per-step events, which include the blend after each step), then
times dk_inpaint_blend on its own at the run's shape and mask, and computes its bytes from the shapes:
  mask (1 B / latent pixel) + for every kept cell: read x0, read noise, write x (3 x 4 B x C)
The regenerated cells read only their mask byte.  The card's name and power limit are read in the same run.

  python tools/bench_inpaint.py [--rounds 6] [--out FILE]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["sm_clock_max"] = [s.strip() for s in q.split(",")]
    except Exception as e:                                        # the name above still identifies the card
        info["power_limit"] = f"unavailable ({e})"
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=6, help="timed (img2img, inpaint) pairs, order alternating")
    ap.add_argument("--out", default=None, help="also write the JSON result here")
    args = ap.parse_args()

    import diffusionkit_b200 as dk
    from diffusionkit_b200 import ops
    from diffusionkit_b200.config import MODEL_CONFIGS, VAEEncoderConfig
    from diffusionkit_b200.pipeline import prepare_inpaint_mask
    from diffusionkit_b200.weights import init_params, mmdit_param_specs, vae_encoder_param_specs

    if not torch.cuda.is_available():
        raise SystemExit("bench_inpaint needs a CUDA device")
    dev = torch.device("cuda", 0)
    mv, steps, images, side, T = "argmaxinc/mlx-FLUX.1-schnell", 4, 4, 1024, 256
    cfg, dtype = MODEL_CONFIGS[mv], torch.bfloat16
    t0 = time.time()
    params = init_params(mmdit_param_specs(cfg), seed=0, dtype=dtype, device=dev)
    eparams = init_params(vae_encoder_param_specs(VAEEncoderConfig()), seed=2, dtype=dtype, device=dev)
    pipe = dk.FluxPipeline(w16=True, a16=True, model_version=mv, device=dev, params=params, load_decoder=False,
                           vae_encoder_params=eparams, load_encoder=True)
    del params, eparams
    torch.cuda.synchronize()
    t_init = time.time() - t0

    rng = np.random.RandomState(0)
    yy, xx = np.meshgrid(np.linspace(0, 1, side), np.linspace(0, 1, side), indexing="ij")
    img = np.stack([0.5 + 0.4 * np.sin(2 * np.pi * (a * xx + b * yy)) for a, b in rng.uniform(0.5, 3, (3, 2))], -1)
    img = (np.clip(img + 0.03 * rng.randn(side, side, 3), 0, 1) * 255).astype(np.uint8)
    mask = np.zeros((side, side), dtype=np.uint8)
    mask[side // 4:3 * side // 4, :] = 255                       # regenerate the middle half of the picture
    seeds = [1000 + i for i in range(images)]
    cond, pooled = pipe.synthetic_text_embeddings(n_images=images, text_len=T)
    cond, pooled = cond.to(dev), pooled.to(dev)
    lat = side // 8
    x_T = pipe.get_empty_latent(lat, lat)
    noise = torch.cat([pipe.get_noise(s, x_T) for s in seeds]).to(dev)

    def run(masked):
        latent, it = pipe.denoise_latents(cond, pooled, num_steps=steps, seed=seeds, image_path=img, denoise=1.0,
                                          mask_path=mask if masked else None, noise=noise)
        return latent, [1e3 * t for t in it]

    for masked in (False, True):                                 # warm-up: every shape of the timed runs
        run(masked)
    step_ms = {"img2img": [], "inpaint": []}
    for r in range(args.rounds):
        for masked in ((False, True) if r % 2 == 0 else (True, False)):
            _, it = run(masked)
            step_ms["inpaint" if masked else "img2img"] += it

    # the blend kernel alone, at the run's shape and mask
    _, m = prepare_inpaint_mask(mask, (side, side))
    m_dev = torch.from_numpy(np.ascontiguousarray(np.broadcast_to(m, (images, lat, lat)))).to(dev)
    g = torch.Generator(device=dev).manual_seed(0)
    x0, nz, x = [torch.randn((images, lat, lat, 16), generator=g, device=dev) for _ in range(3)]
    kept = int((m_dev == 0).sum())
    bytes_moved = m_dev.numel() + kept * 16 * 4 * 3
    bytes_dense = m_dev.numel() + x.numel() * 4 * 4               # if every cell read x, x0, noise and wrote x
    n_warm = 500
    for _ in range(20):
        ops.inpaint_blend(x, x0, nz, m_dev, 0.5)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n_warm):
        ops.inpaint_blend(x, x0, nz, m_dev, 0.5)
    e1.record()
    torch.cuda.synchronize()
    warm_us = 1e3 * e0.elapsed_time(e1) / n_warm
    flush = torch.empty(512 * 1024 * 1024, dtype=torch.uint8, device=dev)     # 4x the L2: evicts the working set
    cold = []
    for _ in range(50):
        flush.zero_()
        e0.record()
        ops.inpaint_blend(x, x0, nz, m_dev, 0.5)
        e1.record()
        torch.cuda.synchronize()
        cold.append(1e3 * e0.elapsed_time(e1))
    cold_us = statistics.median(cold)

    def summary(v):
        return {"mean": round(statistics.mean(v), 2), "stdev": round(statistics.stdev(v), 2), "min": round(min(v), 2),
                "max": round(max(v), 2), "n": len(v)}

    a, b = summary(step_ms["img2img"]), summary(step_ms["inpaint"])
    res = {
        "card": card_info(),
        "workload": f"FLUX.1-schnell synthetic weights, {side}x{side}, {steps} steps, {images} images, denoise 1.0, "
                    f"mask = middle half of the picture ({100 * float(m.mean()):.1f} % of latent cells regenerated)",
        "init_s": round(t_init, 1),
        "step_ms_note": "CUDA events around each Euler step (1 ms resolution), warm-up excluded, runs alternating",
        "step_ms": {"img2img": a, "inpaint": b},
        "inpaint_minus_img2img_ms": round(b["mean"] - a["mean"], 2),
        "blend_kernel": {
            "shape": [images, lat, lat, 16], "kept_cells": kept,
            "bytes": bytes_moved, "bytes_if_dense": bytes_dense,
            "warm_us": round(warm_us, 2), "warm_note": f"{n_warm} back-to-back launches: working set L2-resident",
            "warm_GBps": round(bytes_moved / warm_us / 1e3, 1),
            "cold_us": round(cold_us, 2), "cold_note": "median of 50 launches, each after a 512 MB write evicting L2",
            "cold_GBps": round(bytes_moved / cold_us / 1e3, 1),
            "share_of_step": round(cold_us / 1e3 / a["mean"], 6),
        },
    }
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
