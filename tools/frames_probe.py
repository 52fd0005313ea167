"""Frame-sequence probe: device time per frame of one batch (rt_render_frames_device) against K separate renders
(rt_render_accum_device) with the same cameras and sample offsets (profiles/r05_frames.md).

    python tools/frames_probe.py [--out results.json] [--reps 7]

Settings: C1 1200x600x100 spp, K = 8; the C1 preview 640x360x4 spp, K = 32; C2 960x540x64 spp, K = 8.  The cameras orbit
the scene's lookat by 30 degrees over the K frames (rt_orbit_cameras).  The separate form renders frame f through a scene
of its own whose camera is cameras[f] (all K scenes resident before timing), with sample_offset = f * spp.  Both forms are
timed by rt_stats.ms_total (device events around the render on the context stream, wavefront pipeline), warmed up once,
and alternated `reps` times; the separate form's time is the sum of its K calls' device times (host gaps between calls are
not counted).  Each setting also checks the batch's accumulators against the separate ones: equal sample counts, equal
summed ray counts, sums within float-addition order.  The card's name and power limit are read with nvidia-smi (query
only)."""
from __future__ import annotations

import argparse
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

SETTINGS = [  # name, scene, width, height, spp, frames
    ("c1", "earth_emitter", 1200, 600, 100, 8),
    ("c1_preview", "earth_emitter", 640, 360, 4, 32),
    ("c2", "book1_final", 960, 540, 64, 8),
]
ORBIT_DEGREES = 30.0


def gpu_info() -> str:
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="")
    ap.add_argument("--reps", type=int, default=7)
    args = ap.parse_args()
    ctx = rt.Context(0)
    earth = load_earth()
    res = {"gpu": gpu_info(), "orbit_degrees": ORBIT_DEGREES, "reps": args.reps, "settings": []}
    print("gpu:", res["gpu"], flush=True)
    for name, scene, w, h, spp, k in SETTINGS:
        desc = rt.SceneDesc.builtin(scene, earth) if scene == "earth_emitter" else rt.SceneDesc.builtin(scene)
        base = desc.desc.camera
        cams = rt.orbit_cameras(base, k, ORBIT_DEGREES)
        batch_scene = rt.Scene(ctx, desc)
        singles = []
        for cam in cams:
            desc.desc.camera = cam
            singles.append(rt.Scene(ctx, desc))
        p = rt.default_params(width=w, height=h, spp=spp)
        qs = [rt.default_params(width=w, height=h, spp=spp, sample_offset=f * spp) for f in range(k)]
        acc_b = torch.zeros((k, h, w, 4), dtype=torch.float32, device="cuda")
        acc_s = torch.zeros((k, h, w, 4), dtype=torch.float32, device="cuda")
        torch.cuda.synchronize()

        def run_batch():
            acc_b.zero_()
            torch.cuda.synchronize()
            st = batch_scene.render_frames_device(p, cams, acc_b.data_ptr(), want_stats=True)
            return st.ms_total, st.rays, st.iterations, st.launches

        def run_singles():
            acc_s.zero_()
            torch.cuda.synchronize()
            ms, rays, iters, launches = 0.0, 0, 0, 0
            for f in range(k):
                st = singles[f].render_accum_device(qs[f], acc_s[f].data_ptr(), want_stats=True)
                ms += st.ms_total
                rays += st.rays
                iters += st.iterations
                launches += st.launches
            return ms, rays, iters, launches

        run_batch()  # warm-up: modules, the path pool at its size, both forms
        run_singles()
        tb, ts = [], []
        for _ in range(args.reps):
            b = run_batch()
            s = run_singles()
            tb.append(b[0])
            ts.append(s[0])
        ctx.synchronize()
        gb, gs = acc_b.cpu().numpy(), acc_s.cpu().numpy()
        same_counts = bool(np.array_equal(gb[..., 3], gs[..., 3]))
        max_rel = float(np.max(np.abs(gb - gs) / np.maximum(np.abs(gs), 1e-3)))
        row = {
            "setting": name, "scene": scene, "width": w, "height": h, "spp": spp, "frames": k,
            "batch_ms": tb, "separate_ms": ts,
            "batch_ms_per_frame_median": float(np.median(tb)) / k, "separate_ms_per_frame_median": float(np.median(ts)) / k,
            "batch_ms_per_frame_min": float(np.min(tb)) / k, "separate_ms_per_frame_min": float(np.min(ts)) / k,
            "speedup_median": float(np.median(ts) / np.median(tb)),
            "batch_iterations": b[2], "separate_iterations": s[2], "batch_launches": b[3], "separate_launches": s[3],
            "rays_equal": b[1] == s[1], "counts_equal": same_counts, "max_rel_diff": max_rel,
        }
        res["settings"].append(row)
        print(json.dumps({kk: vv for kk, vv in row.items() if kk not in ("batch_ms", "separate_ms")}), flush=True)
        for sc in singles:
            sc.close()
        batch_scene.close()
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
