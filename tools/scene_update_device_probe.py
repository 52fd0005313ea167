"""Device-update probe: rt_scene_update_device (records read from device memory) against rt_scene_update of the same records
(packed on the host), and a simulation step through each (profiles/r12_scene_update_device.md).

    python tools/scene_update_device_probe.py [--out results.json] [--md results.md] [--reps 5] [--scenes c2,c4]

Update time: C2 (book-1 final, host SAH) and C4 (1 M random spheres, GPU LBVH); 1 sphere, 1 %, 10 % and 100 % of the
spheres moved by a jitter of up to one radius per axis.  Both entries update the same scene with the same records (the
host entry from a numpy array, the device entry from CUDA tensors that already hold them); `ms_device` is each entry's
own device time, `wall` the host clock around the call (both entries return when the update is complete).  One warm-up
of each entry, then `reps` rounds alternating the two; medians.

Simulation step on C4: a torch kernel jitters every sphere (a random step of up to 0.05 radius per axis on the sphere
state kept in a CUDA tensor), the scene is updated with all 10^6 spheres, then rt_render_accum_device renders 1920x1080 at
4 spp.  Device path: Scene.update_device on the tensor.  Host path: the tensor is copied to the host and passed to
Scene.update.  Host clock per step, ending in a synchronise; medians of `reps` steps after one warm-up step each,
alternated.  The card's name and power limit are read with nvidia-smi (query only) in the same run."""
from __future__ import annotations

import argparse
import json
import sys
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))
import raytracing_renderer_cuda_b200 as rt  # noqa: E402
from raytracing_renderer_cuda_b200 import capi  # noqa: E402
from scene_update_probe import FRACTIONS, SCENES, gpu_info, jitter  # noqa: E402

STEP_FRAME = dict(width=1920, height=1080, spp=4)


def records(sph):
    """The float32 (n, 12) tensor of SPHERE_DTYPE records, on the device."""
    return torch.from_numpy(np.ascontiguousarray(sph).view(np.uint8).reshape(len(sph), 48).view(np.float32).copy()).cuda()


def timed(fn):
    t0 = time.perf_counter()
    ms = fn()
    return ms, (time.perf_counter() - t0) * 1e3


def probe_updates(ctx, key, reps, rng):
    cfg = SCENES[key]
    desc = rt.SceneDesc.builtin(cfg["name"], n=cfg["n"])
    sph = desc.spheres()
    n = len(sph)
    sc = rt.Scene(ctx, desc)
    sc.update(np.arange(1, dtype=np.uint32), sph[:1])  # the parent table
    sc.update_device(torch.zeros(1, dtype=torch.int32, device="cuda"), records(sph[:1]))  # the device index table
    res = {"spheres": n, "update": {}}
    for label, frac in FRACTIONS:
        m = 1 if frac is None else max(1, int(round(frac * n)))
        idx = np.sort(rng.choice(n, m, replace=False)).astype(np.uint32)
        new = jitter(sph, idx, rng)
        i_dev, r_dev = torch.from_numpy(idx.astype(np.int32)).cuda(), records(new)
        torch.cuda.synchronize()
        sc.update(idx, new)
        sc.update_device(i_dev, r_dev)
        rows = {"host": [], "device": []}
        for _ in range(reps):
            rows["host"].append(timed(lambda: sc.update(idx, new)))
            rows["device"].append(timed(lambda: sc.update_device(i_dev, r_dev)))
        res["update"][label] = {"spheres": m, **{k: {"ms_device": float(np.median([r[0] for r in v])),
                                                       "wall_ms": float(np.median([r[1] for r in v]))} for k, v in rows.items()}}
    sc.close()
    return res


def probe_step(ctx, reps):
    cfg = SCENES["c4"]
    desc = rt.SceneDesc.builtin(cfg["name"], n=cfg["n"])
    sph = desc.spheres()
    n = len(sph)
    p = rt.default_params(**STEP_FRAME)
    acc = torch.zeros((p.height, p.width, 4), dtype=torch.float32, device="cuda")
    idx_dev = torch.arange(n, dtype=torch.int32, device="cuda")
    idx_host = np.arange(n, dtype=np.uint32)
    paths = {}
    for name in ("host", "device"):
        state = records(sph)
        paths[name] = dict(scene=rt.Scene(ctx, desc), state=state, times=[], gen=torch.Generator(device="cuda").manual_seed(3))
    torch.cuda.synchronize()

    def step(name):
        s = paths[name]
        st, g = s["state"], s["gen"]
        t0 = time.perf_counter()
        j = (torch.rand((n, 3), device="cuda", generator=g) * 2 - 1) * st[:, 3:4].abs() * 0.05
        st[:, 0:3] += j
        st[:, 4:7] += j
        if name == "device":
            torch.cuda.current_stream().synchronize()  # the context runs on its own stream: order the records first
            s["scene"].update_device(idx_dev, st)
        else:
            s["scene"].update(idx_host, st.cpu().numpy().view(np.uint8).reshape(-1).view(capi.SPHERE_DTYPE))
        s["scene"].render_accum_device(p, acc.data_ptr())
        ctx.synchronize()
        return (time.perf_counter() - t0) * 1e3

    for name in paths:
        step(name)  # warm-up
    for _ in range(reps):
        for name in paths:
            paths[name]["times"].append(step(name))
    out = {"frame": STEP_FRAME, "spheres": n}
    for name, s in paths.items():
        out[name] = {"step_ms": float(np.median(s["times"])), "all_ms": s["times"]}
    # the two paths stepped the same seeded random walk (equal inputs by construction): the scenes the two entries made
    # from it must give the same hits
    rays = np.zeros(4096, capi.RAY_DTYPE)
    cam = desc.desc.camera
    rng = np.random.default_rng(4)
    rays["origin"] = np.array(cam.lookfrom, np.float32)
    rays["direction"] = (np.array(cam.lookat, np.float32) - np.array(cam.lookfrom, np.float32) + rng.normal(scale=0.3, size=(4096, 3))).astype(np.float32)
    rays["time"] = rng.random(4096).astype(np.float32)
    ha, hb = (paths[k]["scene"].trace_primary(rays, use_bvh=1) for k in ("host", "device"))
    out["same_hits"] = bool(np.array_equal(ha.view(np.uint8), hb.view(np.uint8)))
    for s in paths.values():
        s["scene"].close()
    return out


def markdown(res) -> str:
    lines = [f"Measured on {res['gpu']} (`nvidia-smi` name, power limit, max SM clock, read in the same run).", "",
             "| scene | edit | spheres | host `ms_device` | host wall | device `ms_device` | device wall | wall, host / device |",
             "|---|---|---|---|---|---|---|---|"]
    for key, r in res["scenes"].items():
        for label, u in r["update"].items():
            h, d = u["host"], u["device"]
            lines.append(f"| {key.upper()} | {label} | {u['spheres']} | {h['ms_device']:.3f} | {h['wall_ms']:.3f} | {d['ms_device']:.3f} | "
                         f"{d['wall_ms']:.3f} | {h['wall_ms'] / d['wall_ms']:.1f}× |")
    s = res.get("step")
    if s:
        lines += ["", f"Simulation step on C4 ({s['spheres']} spheres; jitter, update of every sphere, "
                      f"{s['frame']['width']}x{s['frame']['height']} at {s['frame']['spp']} spp):", "",
                  "| path | step (ms, median) |", "|---|---|",
                  f"| host entry (`Scene.update` of the tensor copied to the host) | {s['host']['step_ms']:.2f} |",
                  f"| device entry (`Scene.update_device`) | {s['device']['step_ms']:.2f} |", "",
                  f"Closest hits of the two scenes after the steps (4096 camera rays, binary BVH) bit-identical: {s['same_hits']}."]
    return "\n".join(lines) + "\n"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="", help="also write the results as JSON to this file")
    ap.add_argument("--md", default="", help="also write the tables as markdown to this file")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--scenes", default="c2,c4")
    a = ap.parse_args()
    ctx = rt.Context(0)
    rng = np.random.default_rng(12)
    res = {"gpu": gpu_info(), "reps": a.reps, "scenes": {}}
    for key in a.scenes.split(","):
        res["scenes"][key] = probe_updates(ctx, key, a.reps, rng)
    if "c4" in a.scenes.split(","):
        res["step"] = probe_step(ctx, a.reps)
    text = markdown(res)
    print(text)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(json.dumps(res, indent=1))
    if a.md:
        Path(a.md).parent.mkdir(parents=True, exist_ok=True)
        Path(a.md).write_text(text)


if __name__ == "__main__":
    main()
