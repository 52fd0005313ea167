"""Adaptive sampling probe: equal-budget quality, time to quality, selection overhead and a parameter sweep
(profiles/r04_adaptive.md).

    python tools/adaptive_probe.py [--out results.json] [--no-sweep]

Equal budget: for C1 (1200x600), C2 (1920x1080) and C3 (1200x600), the adaptive frame with the default parameters, its mean
spp S, and the uniform frame at S rounded up to an even count, both against a 4096-spp frame of this renderer with
independent samples (sample indices from 2^20 on).  Time to quality: the device time of the whole adaptive call
(rt_stats.ms_total: every pass, its tail and every selection step) against the device time of the smallest uniform frame
(even spp, in steps of 8) whose PSNR is at least the adaptive frame's.  Per-pass times: T(max_spp = min + k step) -
T(max_spp = min + (k - 1) step) at the same threshold, which is pass k plus the selection before it; a pass carries fewer
paths than one resident wave when (pixels listed) x step_spp < SMs x 2048.  Selection: the k_adapt_* and scan kernels of
one adaptive call under torch.profiler, per selection step, at 1200x600 and 7680x4320, against ~45 B/pixel at the
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

SCENES = {"c1": ("earth_emitter", 1200, 600), "c2": ("book1_final", 1920, 1080), "c3": ("perlin_motion", 1200, 600)}
SELECT_BYTES_PER_PIXEL = 45  # 32 B of planes read, the error map written (4 B) and its window read from cache, list + flags


def gpu_info() -> str:
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def copy_bandwidth() -> float:
    x = torch.empty(1 << 29, dtype=torch.float32, device="cuda")
    y = torch.empty_like(x)
    for _ in range(3):
        y.copy_(x)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(20):
        y.copy_(x)
    b.record()
    torch.cuda.synchronize()
    return 2 * x.numel() * 4 / (a.elapsed_time(b) / 20) / 1e6


def scene(ctx, name):
    return rt.Scene(ctx, rt.SceneDesc.builtin(name, load_earth()) if name == "earth_emitter" else rt.SceneDesc.builtin(name))


def even_up(x: float) -> int:
    return int(np.ceil(x / 2.0) * 2)


def equal_budget(sc, w, h, ref, a, sm_count):
    img, spp, st, passes = sc.render_adaptive(rt.default_params(width=w, height=h), a)
    sc.render_adaptive(rt.default_params(width=w, height=h), a)  # (warm: pool and scratch allocated)
    img, spp, st, passes = sc.render_adaptive(rt.default_params(width=w, height=h), a)
    mean = float(spp.mean())
    s_uni = even_up(mean)
    uni, st_u = sc.render(rt.default_params(width=w, height=h, spp=s_uni))
    pa, pu = rt.psnr(img, ref), rt.psnr(uni, ref)
    row = {"mean_spp": mean, "uniform_spp": s_uni, "passes": passes, "frac_at_min": float((spp == a.min_spp).mean()),
           "frac_at_max": float((spp == a.max_spp).mean()), "psnr_adaptive": pa, "psnr_uniform": pu, "gain_db": pa - pu,
           "ms_adaptive": st.ms_total, "ms_uniform_equal_budget": st_u.ms_total, "paths": int(st.paths)}
    # time to quality: the smallest uniform frame (even spp, steps of 8) at least as close to the reference
    s = 8
    while s <= 4 * a.max_spp:
        u, st_s = sc.render(rt.default_params(width=w, height=h, spp=s))
        if rt.psnr(u, ref) >= pa:
            row.update(uniform_spp_same_psnr=s, ms_uniform_same_psnr=st_s.ms_total, psnr_uniform_same=rt.psnr(u, ref))
            break
        s += 8
    # per-pass device times (pass k + the selection before it) and the share in passes thinner than one resident wave
    wave = sm_count * 2048
    times, prev = [], 0.0
    for k in range(passes):
        ak = rt.default_adaptive_params(min_spp=a.min_spp, step_spp=a.step_spp, max_spp=a.min_spp + k * a.step_spp,
                                        threshold=a.threshold)
        ms = min(sc.render_adaptive(rt.default_params(width=w, height=h), ak)[2].ms_total for _ in range(3))
        n_k = int((spp >= a.min_spp + k * a.step_spp).sum())
        paths_k = n_k * (a.min_spp if k == 0 else a.step_spp)
        times.append({"pass": k, "pixels": n_k, "paths": paths_k, "ms": ms - prev, "thin": paths_k < wave})
        prev = ms
    total = sum(t["ms"] for t in times)
    row["passes_detail"] = times
    row["share_thin_passes"] = sum(t["ms"] for t in times if t["thin"]) / total if total > 0 else 0.0
    return row


def selection_time(ctx, sc, w, h, a):
    """Device time of the selection kernels (k_adapt_error / k_adapt_select / scan / k_adapt_compact) per selection step."""
    acc = torch.empty((h, w, 4), dtype=torch.float32, device="cuda")
    p = rt.default_params(width=w, height=h)
    ctx.set_stream(torch.cuda.current_stream().cuda_stream)
    sc.render_adaptive_device(p, a, acc.data_ptr())
    torch.cuda.synchronize()
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        passes, _ = sc.render_adaptive_device(p, a, acc.data_ptr())
        torch.cuda.synchronize()
    sel_us, other = 0.0, {}
    for ev in prof.key_averages():
        name = ev.key
        t = ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
        if any(k in name for k in ("k_adapt_error", "k_adapt_select", "k_scan_tiles", "k_scan_add", "k_adapt_compact")):
            sel_us += t
        other[name[:60]] = t
    steps = max(passes - 1, 1)
    return {"size": f"{w}x{h}", "passes": passes, "selection_ms_per_step": sel_us / 1e3 / steps,
            "bytes_per_step": SELECT_BYTES_PER_PIXEL * w * h}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="")
    ap.add_argument("--no-sweep", action="store_true")
    args = ap.parse_args()
    info = gpu_info()
    print("device:", info, flush=True)
    ctx = rt.Context(0)
    sm_count = torch.cuda.get_device_properties(0).multi_processor_count
    res = {"device": info, "copy_gbs": copy_bandwidth(), "defaults": {}}
    d = rt.default_adaptive_params()
    res["defaults"] = {"min_spp": d.min_spp, "step_spp": d.step_spp, "max_spp": d.max_spp, "threshold": d.threshold}
    print(f"copy bandwidth {res['copy_gbs']:.0f} GB/s", flush=True)
    refs, scenes = {}, {}
    for key, (name, w, h) in SCENES.items():
        scenes[key] = scene(ctx, name)
        refs[key], st = scenes[key].render(rt.default_params(width=w, height=h, spp=4096, sample_offset=1 << 20))
        print(f"{key} reference 4096 spp: {st.ms_total:.1f} ms", flush=True)
    for key, (name, w, h) in SCENES.items():
        row = equal_budget(scenes[key], w, h, refs[key], d, sm_count)
        res[f"equal_budget_{key}"] = row
        print(key, json.dumps({k: v for k, v in row.items() if k != "passes_detail"}), flush=True)
    sc1 = scenes["c1"]
    for w, h in ((1200, 600), (7680, 4320)):
        a = d if w == 1200 else rt.default_adaptive_params(min_spp=8, step_spp=8, max_spp=32, threshold=d.threshold)
        r = selection_time(ctx, sc1, w, h, a)
        r["byte_bound_ms"] = r["bytes_per_step"] / (res["copy_gbs"] * 1e6)
        res[f"selection_{w}x{h}"] = r
        print("selection", json.dumps(r), flush=True)
    if not args.no_sweep:
        rows = []
        for tau255, step, mn in itertools.product([0.5, 1.0, 2.0, 4.0], [8, 16, 32], [8, 16, 32]):
            mx = mn + step * ((256 - mn) // step)
            a = rt.default_adaptive_params(min_spp=mn, step_spp=step, max_spp=mx, threshold=tau255 / 255.0)
            r = {"tau_x255": tau255, "min_spp": mn, "step_spp": step, "max_spp": mx}
            for key, (name, w, h) in SCENES.items():
                img, spp, st, passes = scenes[key].render_adaptive(rt.default_params(width=w, height=h), a)
                s_uni = even_up(float(spp.mean()))
                uni, _ = scenes[key].render(rt.default_params(width=w, height=h, spp=s_uni))
                r[key] = {"mean_spp": float(spp.mean()), "psnr": rt.psnr(img, refs[key]), "gain_db": rt.psnr(img, refs[key]) - rt.psnr(uni, refs[key]),
                          "passes": passes, "ms": st.ms_total}
            r["worst_gain_db"] = min(r[k]["gain_db"] for k in SCENES)
            rows.append(r)
            print("sweep", json.dumps(r), flush=True)
        res["sweep"] = rows
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
