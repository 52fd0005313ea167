"""Denoiser probe: device times of the feature pass, each à-trous level and the whole post-pass (CUDA events), the bytes
they move, the quality of denoised low-sample frames against a 4096-spp frame, and a sigma sweep.

    python tools/denoise_probe.py [--reps 50] [--out results.json]

Timings: C1 at 1200x600 (accumulator + features + two scratch planes = 1200*600*(16 + 32 + 32) B = 58 MB, below the
126 MB L2 of a B200: after the warm-up every level is served from L2) and a 7680x4320 frame (2.65 GB: streamed from
HBM).  Level i's time is T(rt_denoise_device with i + 1 levels) - T(with i levels); T(0 levels) is the finalisation.
Each level reads at least 16 B of colour and 32 B of features per pixel and writes 16 B: 64 B/pixel, set against the
device-to-device copy bandwidth measured in the same run.  The card's name and power limit are read with nvidia-smi
(query only)."""
from __future__ import annotations

import argparse
import itertools
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import raytracing_renderer_cuda_b200 as rt  # noqa: E402
from raytracing_renderer_cuda_b200.assets import load_earth  # noqa: E402


def gpu_info() -> str:
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def events_ms(fn, reps: int, warmup: int = 5) -> float:
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def copy_bandwidth(reps: int) -> float:
    """GB/s of a device-to-device copy of 2 GiB (read + write counted)."""
    x = torch.empty(1 << 29, dtype=torch.float32, device="cuda")
    y = torch.empty_like(x)
    ms = events_ms(lambda: y.copy_(x), reps)
    return 2 * x.numel() * 4 / ms / 1e6


def timings(ctx, scene, w, h, reps, levels=5):
    # the library runs on torch's current stream, so the events below bracket its kernels
    ctx.set_stream(torch.cuda.current_stream().cuda_stream)
    acc = torch.zeros((h, w, 4), dtype=torch.float32, device="cuda")
    feat = torch.empty((2, h, w, 4), dtype=torch.float32, device="cuda")
    rgb = torch.empty((h, w, 3), dtype=torch.float32, device="cuda")
    p = rt.default_params(width=w, height=h, spp=1)
    scene.render_accum_device(p, acc.data_ptr())
    k = rt.default_denoise_params().feature_spp
    t_feat = events_ms(lambda: scene.render_features_device(p, k, feat.data_ptr()), reps)
    tot = []
    for L in range(levels + 1):
        d = rt.default_denoise_params(iterations=L)
        tot.append(events_ms(lambda: rt.denoise_device(ctx, acc.data_ptr(), feat.data_ptr(), w, h, d, rgb.data_ptr()), reps))
    npix = w * h
    per_level = [tot[i + 1] - tot[i] for i in range(levels)]
    return {"size": f"{w}x{h}", "feature_spp": k, "ms_features": t_feat, "ms_finalise": tot[0], "ms_levels": per_level,
            "ms_total_5_levels": t_feat + tot[levels], "ms_total_default": t_feat + tot[rt.default_denoise_params().iterations],
            "bytes_per_level": 64 * npix, "working_set_mb": npix * 80 / 1e6,
            "gbs_per_level": [64 * npix / t / 1e6 for t in per_level]}


def quality(ctx, scene, w, h, sweep):
    ref, _ = scene.render(rt.default_params(width=w, height=h, spp=4096, sample_offset=1 << 20))
    rows = []
    for spp in (1, 4, 16, 64):
        raw, _ = scene.render(rt.default_params(width=w, height=h, spp=spp))
        den, _ = scene.render_denoised(rt.default_params(width=w, height=h, spp=spp))
        rows.append({"spp": spp, "psnr_raw": rt.psnr(raw, ref), "psnr_denoised": rt.psnr(den, ref)})
    best = []
    if sweep:
        p4 = rt.default_params(width=w, height=h, spp=4)
        for L, sc, sn, sz, sa in itertools.product([3, 5], [0.25, 0.5, 1.0], [0.3, 1.0], [0.3, 1.0], [0.3, 1.0]):
            d = rt.default_denoise_params(iterations=L, sigma_color=sc, sigma_normal=sn, sigma_depth=sz, sigma_albedo=sa)
            den, _ = scene.render_denoised(p4, d)
            best.append({"iterations": L, "sigmas": [sc, sn, sz, sa], "psnr_denoised4": rt.psnr(den, ref)})
        best.sort(key=lambda r: -r["psnr_denoised4"])
    return rows, best[:10]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--out", default="", help="also write the results as JSON to this file")
    ap.add_argument("--no-sweep", action="store_true")
    a = ap.parse_args()
    info = gpu_info()
    print("device:", info)
    ctx = rt.Context(0)
    scene = rt.Scene(ctx, rt.SceneDesc.builtin("earth_emitter", load_earth()))
    res = {"device": info, "copy_gbs": copy_bandwidth(a.reps)}
    print(f"copy bandwidth {res['copy_gbs']:.0f} GB/s")
    res["c1_1200x600"] = timings(ctx, scene, 1200, 600, a.reps)
    res["c1_7680x4320"] = timings(ctx, scene, 7680, 4320, a.reps)
    for k in ("c1_1200x600", "c1_7680x4320"):
        t = res[k]
        print(f"{t['size']}: features(K={t['feature_spp']}) {t['ms_features']:.4f} ms, finalise {t['ms_finalise']:.4f} ms, levels "
              + ", ".join(f"{x:.4f}" for x in t["ms_levels"]) + f" ms ({', '.join(f'{g:.0f}' for g in t['gbs_per_level'])} GB/s at 64 B/px), "
              f"total 5 levels {t['ms_total_5_levels']:.4f} ms, default {t['ms_total_default']:.4f} ms")
    ctx.set_stream(torch.cuda.current_stream().cuda_stream)
    res["psnr_c1_1200x600"], res["sweep_c1_1200x600"] = quality(ctx, scene, 1200, 600, not a.no_sweep)
    for r in res["psnr_c1_1200x600"]:
        print(f"{r['spp']:3d} spp: raw {r['psnr_raw']:.2f} dB, denoised {r['psnr_denoised']:.2f} dB")
    for r in res["sweep_c1_1200x600"]:
        print("sweep", r)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
