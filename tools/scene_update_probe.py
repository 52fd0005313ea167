"""Scene-update probe: device time of rt_scene_update, split by phase, against rt_scene_create of the same description, and
the frame-time cost of rendering through a refitted tree instead of a fresh one (profiles/r10_scene_update.md).

    python tools/scene_update_probe.py [--out results.json] [--reps 5] [--scenes c2,c4]

Update time: C2 (book-1 final, host SAH) and C4 (1 M random spheres, GPU LBVH); 1 sphere, 1 %, 10 % and 100 % of the
spheres moved by a jitter of up to one radius per axis (a moving sphere keeps its motion).  `ms_device` is the entry's own
device time (events around its work on the context stream), median of `reps` updates after one warm-up update (the first
update of a scene also builds its parent table: reported separately).  The phase split comes from one extra update under
torch.profiler (CUDA activities): kernel and copy time grouped by the phase that issues them.  Creation: host wall clock of
rt_scene_create (which ends in a synchronise), median of 3, with rt_scene_info's build and upload figures.

Tree quality: the scene is refitted after 1, 10 and 100 steps of a random walk (every sphere jittered by up to one radius
per step); rt_stats.ms_total of rt_render_accum_device (device events, wavefront pipeline) at 1920x1080, 16 spp, against a
scene created fresh from the same spheres, median of `reps` alternated renders each.  The card's name and power limit are
read with nvidia-smi (query only)."""
from __future__ import annotations

import argparse
import ctypes as C
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import raytracing_renderer_cuda_b200 as rt  # noqa: E402
from raytracing_renderer_cuda_b200 import capi  # noqa: E402

SCENES = {"c2": dict(name="book1_final", n=0), "c4": dict(name="random_spheres", n=1_000_000)}
FRACTIONS = [("1 sphere", None), ("1 %", 0.01), ("10 %", 0.10), ("100 %", 1.0)]
WALK_STEPS = (1, 10, 100)
FRAME = dict(width=1920, height=1080, spp=16)
PHASES = [  # (phase, substrings of the kernel / activity names it issues)
    ("records (copies + scatter)", ("k_scatter", "Memcpy HtoD")),
    ("refit", ("k_refit_all", "k_parents", "k_depth", "Memset")),
    ("centre/half-extent nodes", ("k_nodes_ch",)),
    ("4-wide collapse", ("k_collapse4", "k_mark4", "k_used4", "k_compact4", "scan", "Memcpy DtoD", "Memcpy DtoH")),
    ("quantisation", ("k_quantize4",)),
]


def gpu_info() -> str:
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else torch.cuda.get_device_name(0)


def with_spheres(desc, sph):
    """`desc` with its sphere array replaced (the description an update of every sphere must match)."""
    sph = np.ascontiguousarray(sph)
    out = capi.rt_scene_desc()
    C.memmove(C.byref(out), C.byref(desc.desc), C.sizeof(out))
    out.spheres = sph.ctypes.data_as(C.POINTER(capi.rt_sphere))
    return rt.SceneDesc(C.pointer(out), desc._lib, keepalive=(sph, desc, out))


def jitter(sph, idx, rng):
    new = sph[idx].copy()
    j = (rng.uniform(-1, 1, (len(idx), 3)) * np.abs(new["radius"])[:, None]).astype(np.float32)
    new["center0"] = new["center0"] + j
    new["center1"] = new["center1"] + j
    return new


def phase_split(sc, idx, new) -> dict:
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        sc.update(idx, new)
        torch.cuda.synchronize()
    per_name: dict[str, float] = {}
    for ev in prof.key_averages():
        us = getattr(ev, "device_time_total", None)
        if us is None:
            us = getattr(ev, "cuda_time_total", 0.0)
        if us:
            per_name[ev.key] = per_name.get(ev.key, 0.0) + us / 1000.0
    split = {p: 0.0 for p, _ in PHASES}
    split["other"] = 0.0
    for name, ms in per_name.items():
        for p, keys in PHASES:
            if any(k in name for k in keys):
                split[p] += ms
                break
        else:
            split["other"] += ms
    return {"phases_ms": split, "activities_ms": per_name}


def create_ms(ctx, desc):
    times, info = [], None
    for _ in range(3):
        t0 = time.perf_counter()
        sc = rt.Scene(ctx, desc)
        times.append((time.perf_counter() - t0) * 1e3)
        info = sc.info()
        sc.close()
    return float(np.median(times)), {"ms_build": info.ms_build, "ms_upload": info.ms_upload, "bvh_mode": info.bvh_mode,
                                     "n_nodes": info.n_nodes, "bvh_depth": info.bvh_depth}


def frame_ms(ctx, scenes, reps):
    p = rt.default_params(**FRAME)
    acc = torch.zeros((p.height, p.width, 4), dtype=torch.float32, device="cuda")
    out = {k: [] for k in scenes}
    for sc in scenes.values():  # warm-up
        sc.render_accum_device(p, acc.data_ptr(), want_stats=True)
    for _ in range(reps):
        for k, sc in scenes.items():
            out[k].append(sc.render_accum_device(p, acc.data_ptr(), want_stats=True).ms_total)
    return {k: float(np.median(v)) for k, v in out.items()}


def probe_scene(ctx, key, reps, rng):
    cfg = SCENES[key]
    desc = rt.SceneDesc.builtin(cfg["name"], n=cfg["n"])
    sph = desc.spheres()
    n = len(sph)
    res = {"spheres": n}
    res["create_wall_ms"], res["create_info"] = create_ms(ctx, desc)
    sc = rt.Scene(ctx, desc)
    first = sc.update(np.arange(1, dtype=np.uint32), sph[:1])  # builds the parent table
    res["first_update_ms_device"] = first
    res["update"] = {}
    for label, frac in FRACTIONS:
        m = 1 if frac is None else max(1, int(round(frac * n)))
        idx = np.sort(rng.choice(n, m, replace=False)).astype(np.uint32)
        new = jitter(sph, idx, rng)
        sc.update(idx, sph[idx])  # warm-up
        dev, wall = [], []
        for _ in range(reps):
            t0 = time.perf_counter()
            dev.append(sc.update(idx, new))
            wall.append((time.perf_counter() - t0) * 1e3)
        res["update"][label] = {"spheres": m, "ms_device": float(np.median(dev)), "wall_ms": float(np.median(wall)),
                                **phase_split(sc, idx, new)}
    sc.close()
    # tree quality after a random walk
    walked = rt.Scene(ctx, desc)
    cur = sph.copy()
    every = np.arange(n, dtype=np.uint32)
    res["walk"] = {}
    done = 0
    for steps in WALK_STEPS:
        while done < steps:
            cur[every] = jitter(cur, every, rng)
            walked.update(every, cur)
            done += 1
        fresh = rt.Scene(ctx, with_spheres(desc, cur))
        ms = frame_ms(ctx, {"refit": walked, "fresh": fresh}, reps)
        res["walk"][str(steps)] = {**ms, "ratio": ms["refit"] / ms["fresh"]}
        fresh.close()
    walked.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="", help="also write the results as JSON to this file")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--scenes", default="c2,c4")
    a = ap.parse_args()
    ctx = rt.Context(0)
    rng = np.random.default_rng(10)
    res = {"gpu": gpu_info(), "frame": FRAME, "scenes": {}}
    for key in a.scenes.split(","):
        res["scenes"][key] = probe_scene(ctx, key, a.reps, rng)
        r = res["scenes"][key]
        print(f"{key}: {r['spheres']} spheres, create {r['create_wall_ms']:.2f} ms wall, first update {r['first_update_ms_device']:.3f} ms")
        for label, u in r["update"].items():
            ph = ", ".join(f"{p} {v:.3f}" for p, v in u["phases_ms"].items())
            print(f"  {label:>8}: {u['ms_device']:.3f} ms device, {u['wall_ms']:.3f} ms wall  [{ph}]")
        for steps, w in r["walk"].items():
            print(f"  walk {steps:>3}: refit {w['refit']:.3f} ms, fresh {w['fresh']:.3f} ms, ratio {w['ratio']:.3f}")
    print("gpu:", res["gpu"])
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
