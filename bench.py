#!/usr/bin/env python
"""bench.py — the driver's measurement contract for the per-pixel render path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config c1|c2|c3|c4|c5] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one frame of the configured scene: zero the float4 accumulator, render `spp` samples per pixel into it
(wavefront pipeline, librt_b200.so), sum the accumulators of all ranks and finalise (/spp, saturate, sqrt, Y-flip +
quantise) on the device.  N > 1 shards SAMPLES through the C-ABI's rt_group_* entries (one process per GPU, CUDA IPC peer
mappings, flag barriers, one fused peer-load reduce + finalisation kernel per GPU over NVLink): rank r renders sample
indices [r*spp, (r+1)*spp) of every pixel, so the job renders N*spp samples per pixel ("weak" scaling: per-GPU work fixed).
torch / torch.distributed are plumbing only: device selection, the stream, timing events, the barrier around the timed
region and the all_gather that carries the IPC handles.

`value` is device-timed (CUDA events on the stream the kernels run on) with the scene resident in HBM; `e2e` goes through
the C-ABI with HOST buffers: scene upload (H2D) + render + read-back of the finished frame (D2H) inside the timed region.
The N = 1 line also carries `other_configs` (short C2 / C3 / C4 lines, each with the roofline that bounds it); an N > 1 line
carries `c5` (the 8K frame: 531 MB accumulators, reduce time and NVLink GB/s broken out) and `strong` (a FIXED number of
samples per pixel split across the ranks).

`--impl reference` times the reference's own main.cu rebuilt unchanged for sm_100 (oracle/_ref/ref_main: BASELINE.json's
stated baseline — the reference ships no CPU renderer) for c1, and the reference harness for the other configs; that arm
never loads librt_b200.so: the scenes are flat files written at build time (oracle/_ref/scenes/) and read with pure ctypes.
The `cpu_baseline` leg times the reference headers compiled for the host cores on a bounded sample.

`--dump-outputs DIR` writes what the last timed step handed its caller on rank 0 as DIR/<name>.npy (float32): `rgb` (the
finished frame), `rgb8` (its 8-bit pixels) and, with one GPU, `accum` (the float4 accumulator).  The scenes are built in and
the random numbers are keyed on pixel, sample and bounce, so the same arguments give the same inputs on every run and two
builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import re
import subprocess
import sys
import tempfile
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

# config -> (builtin scene, width, height, spp per step and GPU, sphere count for random_spheres)
CONFIGS = {
    "c1": dict(scene="earth_emitter", width=1200, height=600, spp=100, n=0,
               name="C1 earth_emitter 1200x600x100spp depth 50 (reference main.cu:188-356)"),
    "c2": dict(scene="book1_final", width=1920, height=1080, spp=256, n=0, name="C2 book-1 final ~485 spheres 1920x1080x256spp"),
    "c3": dict(scene="perlin_motion", width=1200, height=600, spp=1024, n=0,
               name="C3 perlin/checker/wood + moving spheres + emitters 1200x600x1024spp"),
    "c4": dict(scene="random_spheres", width=3840, height=2160, spp=64, n=1_000_000, name="C4 1M random spheres (GPU LBVH) 3840x2160x64spp"),
    "c5": dict(scene="book1_final", width=7680, height=4320, spp=16, n=0,
               name="C5 book-1 final 7680x4320, 16 spp per step and GPU (4096 spp = 256 steps)"),
}
FLOP_PER_RAY = {"c1": 420.0, "c2": 420.0, "c3": 615.0, "c4": 815.0, "c5": 420.0}  # SURVEY.md §8(d), frozen
NODE_BYTES_PER_RAY_C4 = 1340.0                                                     # SURVEY.md §8(d): BVH node traffic of a C4 ray
STATE_BYTES_PER_RAY = 120.0                                                        # SURVEY.md §8(d)
NVLINK_PEER_GBS = 770.0  # measured peer copy per direction per GPU on this pool (B200_PROFILING.md)


def load_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return {"hbm_gbs": float(d["hbm_gbs"]), "sm_max_mhz": float(d.get("sm_max_mhz", 1965.0)), "source": "measured"}
    return {"hbm_gbs": 6650.0, "sm_max_mhz": 1965.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device: int):
        self.device, self.proc, self.lines = device, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.device}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        self.thread.join(timeout=2)
        sm, smax, reasons, power = [], [], set(), []
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
                power.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


def cpu_baseline(cfg_key: str, desc, target_s: float = 12.0) -> dict:
    """Host-core baseline on a bounded sample of the same workload: the reference's own headers compiled
    for the host (oracle/_ref/libref_cpu_rn.so, kind "reference"), else the oracle port (kind "port")."""
    from tests import oracle_api as oa

    cfg = CONFIGS[cfg_key]
    cores = os.cpu_count() or 1
    w, h = cfg["width"] // 4, cfg["height"] // 4
    rt = None
    if not oa.REFCPU_RN_SO.exists():
        import raytracing_renderer_cuda_b200 as rt  # (the oracle port's parameter block comes from the product's defaults)

    if oa.REFCPU_RN_SO.exists():
        kind = "reference"
        sc = oa.RefCpu(oa.REFCPU_RN_SO).scene(desc, use_bvh=True)
        run = lambda spp: sc.render(w, h, spp, nthreads=cores, want_fb=False)[2]  # noqa: E731
    else:
        kind = "port"
        sc = oa.Oracle().scene(desc)
        run = lambda spp: sc.render(rt.default_params(width=w, height=h, spp=spp), sampler=0, arith=0, nthreads=cores)[1]  # noqa: E731
    t0 = time.perf_counter()
    run(1)
    probe = max(time.perf_counter() - t0, 1e-4)  # one sample per pixel at 1/16 of the frame
    rate = w * h / probe
    if rate * target_s > 4 * w * h * 4:  # fast enough: use the full frame
        w, h = cfg["width"], cfg["height"]
        sc = None
        if kind == "reference":
            sc = oa.RefCpu(oa.REFCPU_RN_SO).scene(desc, use_bvh=True)
            run = lambda spp: sc.render(w, h, spp, nthreads=cores, want_fb=False)[2]  # noqa: E731
        else:
            sc = oa.Oracle().scene(desc)
            run = lambda spp: sc.render(rt.default_params(width=w, height=h, spp=spp), sampler=0, arith=0, nthreads=cores)[1]  # noqa: E731
    spp = int(max(1, min(cfg["spp"], rate * target_s / (w * h))))
    t0 = time.perf_counter()
    rays = run(spp)
    dt = time.perf_counter() - t0
    paths = w * h * spp
    return {"value": paths / dt / 1e6, "unit": "Mpaths/s", "cores": cores, "kind": kind, "mrays_per_s": rays / dt / 1e6,
            "seconds": dt, "sample": f"{cfg['scene']} {w}x{h}x{spp}spp ({paths} paths) on {cores} host threads; "
            + ("reference headers via oracle/shim, _rz intrinsics rounding to nearest" if kind == "reference" else "oracle/rt_oracle.cpp")}


def build_desc(cfg_key: str, n_override: int = 0):
    import raytracing_renderer_cuda_b200 as rt
    from raytracing_renderer_cuda_b200.assets import load_earth

    cfg = CONFIGS[cfg_key]
    image = load_earth() if cfg["scene"] == "earth_emitter" else None
    return rt.SceneDesc.builtin(cfg["scene"], image, n=n_override or cfg["n"])


def desc_h2d_bytes(desc) -> int:
    from raytracing_renderer_cuda_b200 import capi

    d = desc.desc
    b = d.n_spheres * C.sizeof(capi.rt_sphere) + d.n_materials * C.sizeof(capi.rt_material) + d.n_textures * C.sizeof(capi.rt_texture)
    for i in range(d.n_images):
        b += d.images[i].width * d.images[i].height * 3 * 4
    return int(b)


def kernel_name_of(info) -> str:
    return ("k_wf_step_pt" if int(info.n_spheres) >= 4096 else "k_wf_step_warp") if int(info.n_nodes) else "k_wf_step_cta"


def measure_l2_gbs(torch, stream) -> float:
    """L2 bandwidth the way MEASURED_PEAKS.json measures HBM: a plain device copy, here of a working set that stays in the
    126 MB L2 (2 x 16 MiB), read + write bytes, best of 5 batches of 50 copies."""
    a = torch.empty(16 << 20, dtype=torch.uint8, device="cuda")
    b = torch.empty_like(a)
    a.fill_(1)
    for _ in range(10):
        b.copy_(a)
    best = 0.0
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(50):
            b.copy_(a)
        e1.record(stream)
        e1.synchronize()
        best = max(best, 50 * 2 * a.numel() / (e0.elapsed_time(e1) / 1e3) / 1e9)
    return best


# ------------------------------------------------------------------------------------------ ours
class FrameLoop:
    """One configuration on this rank: scene, accumulator, the per-step sequence, device timing."""

    def __init__(self, torch, dist, rt, ctx, stream, cfg_key, spp_rank, sample_offset, rank, world, collective, n_override=0):
        self.torch, self.dist, self.rt, self.ctx, self.stream = torch, dist, rt, ctx, stream
        self.cfg_key, self.cfg, self.rank, self.world = cfg_key, CONFIGS[cfg_key], rank, world
        self.W, self.H, self.spp = self.cfg["width"], self.cfg["height"], spp_rank
        self.desc = build_desc(cfg_key, n_override)
        self.scene = rt.Scene(ctx, self.desc)
        self.info = self.scene.info()
        self.params = rt.default_params(width=self.W, height=self.H, spp=spp_rank, sample_offset=sample_offset)
        self.group, self.symm = None, None
        self.collective = "none"
        H, W = self.H, self.W
        if world > 1 and collective in ("auto", "ipc"):
            def exchange(blob):
                table = [None] * world
                dist.all_gather_object(table, blob)
                return table

            self.group = rt.Group(ctx, rank, world, W, H, exchange)
            self.accum_ptr = self.group.accum_ptr
            self.collective = "rt_group (C-ABI): CUDA IPC peer mappings + flag barriers + fused peer-load reduce/finalise kernel over NVLink"
        elif world > 1 and collective in ("multimem", "peer"):
            import torch.distributed._symmetric_memory as symm

            dev = torch.device("cuda", torch.cuda.current_device())
            self.accum = symm.empty((H, W, 4), dtype=torch.float32, device=dev)
            self.rgb = symm.empty((H, W, 3), dtype=torch.float32, device=dev)
            self.rgb8 = symm.empty((H, W, 3), dtype=torch.uint8, device=dev)
            hdl = symm.rendezvous(self.accum, dist.group.WORLD)
            h_rgb, h_rgb8 = symm.rendezvous(self.rgb, dist.group.WORLD), symm.rendezvous(self.rgb8, dist.group.WORLD)
            mc = int(hdl.multicast_ptr or 0) if collective == "multimem" else 0
            self.symm = dict(hdl=hdl, peers=[int(p) for p in hdl.buffer_ptrs], mc=mc, rgb=int(h_rgb.buffer_ptrs[0]), rgb8=int(h_rgb8.buffer_ptrs[0]),
                             rows=rt.shard_rows(H, rank, world))
            self.accum_ptr = self.accum.data_ptr()
            self.collective = "A/B: torch symmetric memory + " + ("NVLS multimem.ld_reduce" if mc else "NVLink peer loads") + " in the fused kernel"
        else:
            self.accum = torch.zeros((H, W, 4), dtype=torch.float32, device="cuda")
            self.rgb = torch.empty((H, W, 3), dtype=torch.float32, device="cuda")
            self.rgb8 = torch.empty((H, W, 3), dtype=torch.uint8, device="cuda")
            self.accum_ptr = self.accum.data_ptr()
            if world > 1:
                self.collective = "A/B: NCCL reduce(SUM) to rank 0 + tonemap"

    # -- the step --
    def begin(self):
        if self.group is not None:
            self.group.begin_frame()
        else:
            self.accum.zero_()

    def render(self, want_stats=False):
        return self.scene.render_accum_device(self.params, self.accum_ptr, want_stats=want_stats)

    def finish(self):
        """sum over ranks + pixel finalisation; the frame ends up on rank 0"""
        rt = self.rt
        if self.group is not None:
            self.group.finish_frame(want_rgb8=True)
        elif self.symm is not None:
            s = self.symm
            s["hdl"].barrier(0)
            rt.reduce_tonemap_peers(self.ctx, s["peers"], s["mc"], self.W, self.H, s["rows"][0], s["rows"][1], s["rgb"], s["rgb8"])
            s["hdl"].barrier(1)
        else:
            if self.world > 1:
                self.dist.reduce(self.accum, dst=0, op=self.dist.ReduceOp.SUM)
            if self.rank == 0:
                rt.tonemap_device(self.ctx, self.accum_ptr, self.W, self.H, self.rgb.data_ptr(), self.rgb8.data_ptr())

    def step(self):
        self.begin()
        self.render()
        self.finish()

    def sync_all(self):
        self.stream.synchronize()
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def timed(self, steps, warmup, flush):
        """-> (ms per step, ms of the render span, ms of the finish span, rays of this rank per step, launches, iterations)"""
        torch, stream = self.torch, self.stream
        self.begin()
        st = self.render(want_stats=True)  # deterministic: the RNG is keyed on pixel/sample/bounce
        self.finish()
        rays, launches, iters = int(st.rays), int(st.launches), int(st.iterations)
        for _ in range(warmup):
            self.step()
        self.sync_all()
        ev = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(steps)]
        for k in range(steps):
            flush.fill_(k & 255)  # L2 flush between timed iterations, outside the timed span
            ev[k][0].record(stream)
            self.begin()
            ev[k][1].record(stream)
            self.render()
            ev[k][2].record(stream)
            self.finish()
            ev[k][3].record(stream)
        self.sync_all()
        ms = float(np.mean([e[0].elapsed_time(e[3]) for e in ev]))
        ms_render = float(np.mean([e[1].elapsed_time(e[2]) for e in ev]))
        ms_finish = float(np.mean([e[2].elapsed_time(e[3]) for e in ev]))
        return ms, ms_render, ms_finish, rays, launches, iters

    def outputs(self) -> dict:
        """what the last step handed its caller on rank 0: the frame as floats and as 8-bit pixels, and with one rank the
        accumulator it was finalised from (with several, each rank's accumulator holds only its own samples)"""
        if self.group is not None:
            rgb, rgb8 = np.empty((self.H, self.W, 3), np.float32), np.empty((self.H, self.W, 3), np.uint8)
            self.group.read_frame(rgb, rgb8)
            out = {"rgb": rgb, "rgb8": rgb8}
        else:
            self.stream.synchronize()
            out = {"rgb": self.rgb.cpu().numpy(), "rgb8": self.rgb8.cpu().numpy()}
        if self.world == 1:
            out["accum"] = self.accum.cpu().numpy()
        return out

    def close(self):
        if self.group is not None:
            self.group.close()
        self.scene.close()


DUMP_BYTES = 64_000_000


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """Writes [H, W, C] arrays as <name>.npy in float32.  When they exceed DUMP_BYTES together, every array keeps the
    same fixed, seeded sample of pixels in ascending order ([n, C]), so that dumps of two builds still line up."""
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    h, w = next(iter(arrays.values())).shape[:2]
    bytes_per_pixel = 4 * sum(a.shape[2] for a in arrays.values())
    n = min(h * w, (DUMP_BYTES - 4096) // bytes_per_pixel)  # (4096: room for the .npy headers)
    pick = None if n == h * w else np.sort(np.random.default_rng(0).choice(h * w, n, replace=False))
    for name, a in arrays.items():
        a = a.astype(np.float32)
        np.save(out / f"{name}.npy", a if pick is None else a.reshape(h * w, -1)[pick])


def roofline_of(cfg_key, rays_rank, ms_render, n_step_launches, peaks, l2_gbs, kernel_name):
    fp32_peak = peaks["sm_count"] * 128 * 2 * peaks["sm_max_mhz"] * 1e6 / 1e12  # TFLOP/s at the measured max SM clock
    flop_launch = rays_rank / n_step_launches * FLOP_PER_RAY[cfg_key]
    dur_launch_s = ms_render / 1e3 / n_step_launches
    fp32 = flop_launch / dur_launch_s / 1e12
    hbm = rays_rank * STATE_BYTES_PER_RAY / (ms_render / 1e3) / 1e9
    common = {"kernel": kernel_name, "launches_per_step": n_step_launches, "avg_launch_ms": dur_launch_s * 1e3}
    if cfg_key == "c4":
        # SURVEY 8d: a C4 ray is bound by the L2 -> SM bandwidth of its BVH node fetches (1.34 KB of nodes per ray, served by L2:
        # the node array is pinned there), not by FP32 issue
        l2 = rays_rank * NODE_BYTES_PER_RAY_C4 / (ms_render / 1e3) / 1e9
        return {"bound": "l2", "achieved": l2, "peak": l2_gbs, "unit": "GB/s", "frac": l2 / l2_gbs if l2_gbs else None, "traffic": None,
                "bytes_per_ray": NODE_BYTES_PER_RAY_C4,
                "peak_source": "L2-resident device copy (2 x 16 MiB, read + write) measured by this run, the method of MEASURED_PEAKS.json's hbm_gbs",
                "fp32": {"achieved": fp32, "peak": fp32_peak, "unit": "TFLOP/s", "frac": fp32 / fp32_peak, "flop_per_ray": FLOP_PER_RAY[cfg_key]},
                **common}
    return {"bound": "fp32", "achieved": fp32, "peak": fp32_peak, "unit": "TFLOP/s", "frac": fp32 / fp32_peak, "traffic": None,
            "flop_per_ray": FLOP_PER_RAY[cfg_key],
            "peak_source": f"{peaks['sm_count']} SM x 128 lanes x 2 flop x {peaks['sm_max_mhz']:.0f} MHz (MEASURED_PEAKS.json sm_max_mhz, {peaks['source']})",
            "note": "no dense contraction and L2-resident state: the bounding roofline is FP32 issue (SURVEY.md 8d), not hbm/tensor",
            "hbm": {"achieved": hbm, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": hbm / peaks["hbm_gbs"],
                    "bytes_per_ray": STATE_BYTES_PER_RAY, "peak_source": f"MEASURED_PEAKS.json ({peaks['source']})"},
            **common}


def run_ours(args) -> None:
    import torch
    import torch.distributed as dist

    import raytracing_renderer_cuda_b200 as rt

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch N > 1 through torch.distributed.run")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; librt_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    cfg = CONFIGS[args.config]
    W, H = cfg["width"], cfg["height"]
    spp = args.spp or cfg["spp"]
    ctx = rt.Context(local_rank)
    stream = torch.cuda.Stream()
    ctx.set_stream(stream.cuda_stream)
    peaks = load_peaks()
    peaks["sm_count"] = torch.cuda.get_device_properties(local_rank).multi_processor_count

    with torch.cuda.stream(stream):
        flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB L2
        loop = FrameLoop(torch, dist, rt, ctx, stream, args.config, spp, rank * spp, rank, world, args.collective)
        sampler = ClockSampler(local_rank) if rank == 0 else None
        # (the warm-up, incl. one instrumented step, runs before the clock sampler starts)
        loop.step()
        loop.sync_all()
        if sampler:
            sampler.start()
        t_wall0 = time.perf_counter()
        ms_step, ms_render, ms_finish, rays_rank, launches_render, iters = loop.timed(args.steps, args.warmup, flush)
        t_wall = time.perf_counter() - t_wall0
        clocks = sampler.stop() if sampler else None
        if args.dump_outputs:
            if rank == 0:
                dump_outputs(args.dump_outputs, loop.outputs())
            if world > 1:
                dist.barrier()  # the other ranks' next rt_group barrier waits a bounded time only
        launches_finish = (3 if loop.group is not None or loop.symm is not None else 1) if (world > 1 or rank == 0) else 0
        launches_step = launches_render + launches_finish

        # ---- end to end through the C-ABI with HOST buffers: scene upload + render + read-back each step ----
        desc = loop.desc
        h2d = desc_h2d_bytes(desc)
        out_host = torch.empty((H, W, 3), dtype=torch.float32).pin_memory()
        cudart = torch.cuda.cudart()
        for i in range(desc.desc.n_images):  # pin the host image the scene upload reads
            im = desc.desc.images[i]
            cudart.cudaHostRegister(C.cast(im.rgb, C.c_void_p).value, im.width * im.height * 12, 0)

        def e2e_step():
            sc = rt.Scene(ctx, desc)  # H2D: spheres, materials, textures, image; BVH build
            if world == 1:
                sc.render(loop.params, out_host.numpy())  # render + tonemap + D2H, synchronous
            else:
                loop.begin()
                sc.render_accum_device(loop.params, loop.accum_ptr)
                loop.finish()
                if loop.group is not None:
                    loop.group.read_frame(out_host.numpy() if rank == 0 else None)
                else:
                    if rank == 0:
                        out_host.copy_(loop.rgb, non_blocking=True)
                    stream.synchronize()
            sc.close()

        for _ in range(min(args.warmup, 2)):
            e2e_step()
        loop.sync_all()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            e2e_step()
        torch.cuda.synchronize()
        e2e_serial_s = (time.perf_counter() - t0) / args.steps
        e2e_s = e2e_serial_s

        # The same work as a two-deep frame pipeline (N = 1), all through public entry points: an uploader thread creates
        # scene k+1 on a second context (H2D on its own stream) while this thread renders frame k into device buffers
        # (rt_render_accum_device + rt_tonemap_device) and a copy stream reads frame k-1 back into pinned host memory.  Every
        # step still uploads its scene and reads its frame back inside the timed region; only the waiting is overlapped.
        e2e_pipe = None
        if world == 1:
            import queue as _queue
            import threading as _threading

            ctx_up = rt.Context(local_rank)
            copy_stream = torch.cuda.Stream()
            rgb_dev = [torch.empty((H, W, 3), dtype=torch.float32, device="cuda") for _ in range(2)]
            out_pin = [torch.empty((H, W, 3), dtype=torch.float32).pin_memory() for _ in range(2)]
            acc_dev = [torch.empty((H, W, 4), dtype=torch.float32, device="cuda") for _ in range(2)]

            def pipelined(n_steps):
                ready = _queue.Queue(maxsize=2)

                def uploader():
                    for _ in range(n_steps):
                        ready.put(rt.Scene(ctx_up, desc))  # blocks in rt_scene_create (the GIL is released), not in Python

                th = _threading.Thread(target=uploader)
                th.start()
                done_ev, old = [None, None], []
                for k in range(n_steps):
                    sc_k = ready.get()
                    b = k & 1
                    if done_ev[b] is not None:
                        done_ev[b].synchronize()  # frame k-2 has been read back: its buffers and its scene are free
                        old.pop(0).close()
                    acc_dev[b].zero_()
                    sc_k.render_accum_device(loop.params, acc_dev[b].data_ptr(), ctx=ctx)  # rendered through the main context
                    rt.tonemap_device(ctx, acc_dev[b].data_ptr(), W, H, rgb_dev[b].data_ptr(), 0)
                    rendered = torch.cuda.Event()
                    rendered.record(stream)
                    copy_stream.wait_event(rendered)
                    with torch.cuda.stream(copy_stream):
                        out_pin[b].copy_(rgb_dev[b], non_blocking=True)
                        done_ev[b] = torch.cuda.Event()
                        done_ev[b].record(copy_stream)
                    old.append(sc_k)
                th.join()
                torch.cuda.synchronize()
                for sc_k in old:
                    sc_k.close()

            try:
                pipelined(3)
                t0 = time.perf_counter()
                pipelined(args.steps)
                e2e_pipe = (time.perf_counter() - t0) / args.steps
            except Exception as ex:  # the serial measurement above stands; say why the pipelined one is missing
                print(f"bench.py: pipelined e2e leg failed ({ex!r}); reporting the serial call sequence", file=sys.stderr)
                e2e_pipe = None
                torch.cuda.synchronize()
            # The pipeline needs two host threads that keep up with ~40 launches per 7 ms frame; on a box whose host cores are busy
            # or slow the plain serial call sequence is the faster of the two.  Both are end-to-end runs of the same per-step
            # work through the public API: the headline is the better one, and the line says which and carries both.
            e2e_s = min(e2e_pipe, e2e_serial_s) if e2e_pipe is not None else e2e_serial_s

        # ---- output stage on the device (SURVEY 8f-1): render + finalise + flip/quantise + JPEG, only the file is read back ----
        jpeg = None
        if world == 1:
            file_host = torch.empty(int(ctx.lib.rt_jpeg_max_bytes(W, H)), dtype=torch.uint8).pin_memory()
            for _ in range(min(args.warmup, 2)):
                loop.scene.render_jpeg(loop.params, 100, file_host.numpy())
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(args.steps):
                f_bytes, st_j = loop.scene.render_jpeg(loop.params, 100, file_host.numpy())
            t_j = (time.perf_counter() - t0) / args.steps
            jpeg = {"value": float(W) * H * spp / t_j / 1e6, "unit": "Mpaths/s", "ms_per_step": t_j * 1e3,
                    "ms_device_jpeg": float(st_j.ms_d2h), "d2h_bytes_per_step": int(f_bytes.size), "quality": 100,
                    "gb_per_s_pixels": W * H * 3 / (float(st_j.ms_d2h) / 1e3) / 1e9 if st_j.ms_d2h > 0 else None,
                    "what": "rt_render_jpeg: render + finalise + Y-flip/quantise + baseline JPEG (byte-identical to the reference's "
                            "stbi_write_jpg, main.cu:475-491) on the device; the D2H copy moves the finished file only"}
        info, kernel_name = loop.info, kernel_name_of(loop.info)
        collective = loop.collective
        loop.close()

        def reduce_max(*xs):
            t = torch.tensor(xs, dtype=torch.float64, device="cuda")
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return [float(x) for x in t.tolist()]

        def reduce_sum(x):
            t = torch.tensor([x], dtype=torch.float64, device="cuda")
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.SUM)
            return float(t.item())

        ms_step, ms_render, ms_finish, e2e_ms = reduce_max(ms_step, ms_render, ms_finish, e2e_s * 1e3)
        rays_total = reduce_sum(rays_rank)

        # ---- the other configurations, short (N = 1), each with the roofline that bounds it ----
        other = {}
        l2_gbs = None
        if world == 1 and not args.no_other_configs and args.config == "c1":
            l2_gbs = measure_l2_gbs(torch, stream)
            for key in ("c2", "c3", "c4"):
                lp = FrameLoop(torch, dist, rt, ctx, stream, key, CONFIGS[key]["spp"], 0, 0, 1, "none")
                lp.step()
                m, mr, mf, rays_k, launches_k, it_k = lp.timed(2, 1, flush)
                c = CONFIGS[key]
                paths = float(c["width"]) * c["height"] * c["spp"]
                other[key] = {"workload": c["name"], "value": paths / m / 1e3, "unit": "Mpaths/s", "ms_per_step": m, "steps": 2, "warmup": 3,
                              "mrays_per_s": rays_k / m / 1e3, "rays_per_path": rays_k / paths, "n_spheres": int(lp.info.n_spheres),
                              "bvh_nodes": int(lp.info.n_nodes), "wavefront_iterations": it_k,
                              "roofline": roofline_of(key, rays_k, mr, max(1, launches_k - 1), peaks, l2_gbs, kernel_name_of(lp.info))}
                lp.close()

        # ---- N > 1: the 8K frame (C5) and strong scaling, through the same rt_group path ----
        c5 = strong = None
        if world > 1 and not args.no_other_configs and args.config == "c1":
            lp = FrameLoop(torch, dist, rt, ctx, stream, "c5", CONFIGS["c5"]["spp"], rank * CONFIGS["c5"]["spp"], rank, world, args.collective)
            lp.step()
            m, mr, mf = reduce_max(*lp.timed(2, 1, flush)[:3])
            c = CONFIGS["c5"]
            npix = float(c["width"]) * c["height"]
            # every GPU pulls its band of the other N-1 accumulators over NVLink: (N-1)/N x 16 B x pixels per GPU
            link_bytes = npix * 16.0 * (world - 1) / world
            c5 = {"workload": c["name"], "value": npix * c["spp"] * world / m / 1e3, "unit": "Mpaths/s", "ms_per_step": m, "ms_render": mr,
                  "ms_reduce_finalise": mf, "steps": 2, "spp_per_gpu": c["spp"], "spp_total": c["spp"] * world, "scaling": "weak",
                  "accumulator_bytes_per_gpu": npix * 16.0, "nvlink_bytes_in_per_gpu": link_bytes,
                  "nvlink_gbs_per_gpu": link_bytes / (mf / 1e3) / 1e9, "nvlink_peak_gbs": NVLINK_PEER_GBS,
                  "nvlink_frac": link_bytes / (mf / 1e3) / 1e9 / NVLINK_PEER_GBS,
                  "note": "ms_reduce_finalise spans barrier + fused reduce/finalise kernel + barrier, i.e. it includes the skew between the ranks' renders"}
            lp.close()
            strong = {}
            for key, total in (("c1", CONFIGS["c1"]["spp"]), ("c5", 64)):
                first, count = rt.shard_samples(total, rank, world)
                lp = FrameLoop(torch, dist, rt, ctx, stream, key, count, first, rank, world, args.collective)
                lp.step()
                m, mr, mf = reduce_max(*lp.timed(3 if key == "c1" else 2, 1, flush)[:3])
                c = CONFIGS[key]
                strong[key] = {"workload": f"{c['scene']} {c['width']}x{c['height']}, {total} spp in TOTAL split over {world} GPUs", "scaling": "strong",
                               "value": float(c["width"]) * c["height"] * total / m / 1e3, "unit": "Mpaths/s", "ms_per_step": m, "ms_render": mr,
                               "ms_reduce_finalise": mf, "spp_total": total}
                lp.close()

    if rank == 0:
        paths_total = float(W) * H * spp * world
        value = paths_total / ms_step / 1e3
        n_step_launches = max(1, launches_render - 1)  # k_wf_step launches (excl. k_wf_init)
        roof = roofline_of(args.config, rays_rank, ms_render, n_step_launches, peaks, l2_gbs or 0.0, kernel_name)
        tp = ROOT / "profiles" / "traffic.json"
        if tp.exists():  # DRAM bytes per launch of the dominant kernel from the committed ncu --set full capture (static)
            ent = json.loads(tp.read_text()).get(args.config) or {}
            roof["traffic"] = ent.get("bytes_per_launch")
            roof["ncu"] = ent.get("ncu")
        line = {
            "metric": "Mpaths/s", "value": value, "unit": "Mpaths/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "mrays_per_s": rays_total / ms_step / 1e3, "ms_per_frame": ms_step, "ms_render": ms_render,
            "ms_reduce_finalise": ms_finish, "rays_per_path": rays_total / paths_total,
            "config": {"workload": cfg["name"], "scene": cfg["scene"], "width": W, "height": H, "spp_per_gpu": spp,
                       "spp_total": spp * world, "max_depth": 50, "n_spheres": int(info.n_spheres), "bvh_nodes": int(info.n_nodes),
                       "bvh_mode": int(info.bvh_mode), "pipeline": "wavefront", "parallelism": f"samples x{world}", "collective": collective,
                       "l2": "flushed between timed steps (256 MiB fill, outside the timed spans)",
                       "timing": "mean of per-step CUDA-event spans on the launching stream, max over ranks"},
            "roofline": roof,
            "e2e": {"value": paths_total / e2e_ms / 1e3, "unit": "Mpaths/s", "ms_per_step": e2e_ms, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": W * H * 3 * 4,
                    "what": (("two-deep frame pipeline over the public C-ABI entries: every step uploads its scene (rt_scene_create on a second "
                              "context / stream, H2D scene + texture, BVH build), renders (rt_render_accum_device + rt_tonemap_device) and reads "
                              "its frame back into pinned host memory (copy stream); uploads and read-backs overlap the neighbouring frames' "
                              "renders; wall clock over the whole loop") if e2e_pipe is not None and e2e_pipe <= e2e_serial_s else
                             "serial call sequence per step: rt_scene_create (H2D scene + texture, BVH build), then rt_render to a pinned host buffer (synchronous); wall clock")
                    if world == 1 else "rt_scene_create (H2D) on every rank + rt_group frame + D2H of the root's frame, wall clock, max over ranks",
                    "mode": None if world > 1 else ("pipelined" if e2e_pipe is not None and e2e_pipe <= e2e_serial_s else "serial"),
                    "pipelined": None if world > 1 or e2e_pipe is None else {"value": paths_total / (e2e_pipe * 1e3) / 1e3, "ms_per_step": e2e_pipe * 1e3},
                    "serial": None if world > 1 else {
                        "value": paths_total / (e2e_serial_s * 1e3) / 1e3, "ms_per_step": e2e_serial_s * 1e3,
                        "what": "the same per-step work without overlap: rt_scene_create, then rt_render to a pinned host buffer (synchronous)"}},
            "gpu_launches": int(args.steps * launches_step),  # k_wf_init + k_wf_step x iterations + tonemap / barrier-reduce-barrier
            "wavefront_iterations": iters, "clocks": clocks, "wall_s_timed_region": t_wall,
        }
        if jpeg is not None:
            line["output_stage"] = jpeg
        if other:
            line["other_configs"] = other
            line["l2_gbs_measured"] = l2_gbs
        if c5 is not None:
            line["c5"] = c5
        if strong is not None:
            line["strong"] = strong
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(args.config, desc)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------ reference
def child_json(*argv, timeout=900):
    """Runs this script in a CHILD process (which may load librt_b200.so and the oracle) and returns the JSON it prints: the
    reference arm's own process stays free of the product library."""
    o = subprocess.run([sys.executable, str(Path(__file__).resolve()), *argv], capture_output=True, text=True, timeout=timeout)
    if o.returncode != 0:
        return None
    try:
        return json.loads(o.stdout.strip().splitlines()[-1])
    except (ValueError, IndexError):
        return None


def run_reference(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return  # the reference is single-GPU: rank 0 alone runs and prints it
    cfg = CONFIGS[args.config]
    ref = ROOT / "oracle" / "_ref"
    W, H = cfg["width"], cfg["height"]
    # the scene of the configuration as a flat file written at build time (oracle/_ref/scenes/, __graft_entry__.build()),
    # read with pure ctypes: nothing in this arm's process tree loads librt_b200.so.  Without the file (build() not run)
    # a child process writes it.
    scene_file = ref / "scenes" / f"{args.config}.rtsc"

    def host_core_baseline():
        if scene_file.exists():
            from tests import oracle_api as oa

            if oa.REFCPU_RN_SO.exists():
                return cpu_baseline(args.config, oa.FileDesc(scene_file))
        return child_json("--child", "cpu-baseline", "--config", args.config)

    cb = None if args.no_cpu_baseline else host_core_baseline()
    if args.ref_device == "cpu":
        v = cb or host_core_baseline()
        if not v:
            print(json.dumps({"impl": "reference", "unavailable": "host-core baseline failed"}))
            return
        line = {"impl": "reference", "metric": "Mpaths/s", "value": v["value"], "unit": "Mpaths/s", "n_gpus": args.gpus, "steps": 1,
                "warmup": 0, "ms_per_step": v["seconds"] * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic", "config": {"workload": cfg["name"], "device": "host cores"},
                "cpu_baseline": v, "e2e": {"value": v["value"], "unit": "Mpaths/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line), flush=True)
        return
    if not (ref / "ref_main").exists() or not (ref / "ref_harness").exists():
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/ref_main not built (needs the reference's sources: make -C oracle ref REF=<dir>)"}))
        return
    spp = args.spp or cfg["spp"]
    took_ms, kernel_ms, rays = [], None, None
    steps = args.steps
    how = ""
    if args.config == "c1" and not args.spp:
        # the UNCHANGED binary: its own timing window (init_rand_state + render + syncs, main.cu:431-454)
        for k in range(args.warmup + args.steps):
            o = subprocess.run([str(ref / "ref_main")], cwd=str(ref), capture_output=True, text=True, timeout=600)
            m = re.search(r"took (\d+)us", o.stdout)
            if o.returncode != 0 or not m:
                print(json.dumps({"impl": "reference", "unavailable": f"ref_main failed rc={o.returncode}: {o.stderr[-200:]}"}))
                return
            if k >= args.warmup:
                took_ms.append(int(m.group(1)) / 1e3)
        how = "reference src/main.cu rebuilt unchanged (-arch=sm_100), its own chrono window (init_rand_state + render + syncs)"
    else:
        with tempfile.TemporaryDirectory() as td:
            # the reference builds its BVH on ONE device thread, O(N log^2 N) with virtual calls (bvh.h:75-113): 10^5 spheres did
            # not finish in 20 minutes on a B200, 10^6 is out of reach -> C4 is run at 10^4
            n_over = 10_000 if args.config == "c4" else 0
            sp = scene_file
            if not sp.exists():
                sp = Path(td) / "scene.rtsc"
                if child_json("--child", "dump-scene", "--config", args.config, "--scene-n", str(n_over), "--out", str(sp)) is None:
                    print(json.dumps({"impl": "reference", "unavailable": "could not write the scene file"}))
                    return
            steps = min(args.steps, 3)  # the reference's frames of the larger configs take seconds to minutes each
            o = subprocess.run([str(ref / "ref_harness"), "render", str(sp), str(W), str(H), str(spp), str(Path(td) / "o.f32"), "1", "1",
                                str(steps)], capture_output=True, text=True, timeout=1500)
            if o.returncode != 0:
                print(json.dumps({"impl": "reference", "unavailable": "ref_harness failed: " + o.stderr[-200:]}))
                return
            info = json.loads(o.stdout.strip().splitlines()[-1])
            kernel_ms, rays = info["ms_render"] + info["ms_init_rand"], info["rays"]
            took_ms = [kernel_ms]
            how = "reference translation unit through oracle/ref_harness.cu (runtime sizes), CUDA events around init_rand_state + render" + (
                "; scene reduced to 10^4 spheres (the reference cannot build its BVH for more)" if n_over else "")
    ms = float(np.mean(took_ms))
    paths = float(W) * H * spp
    value = paths / ms / 1e3
    line = {"impl": "reference", "metric": "Mpaths/s", "value": value, "unit": "Mpaths/s", "n_gpus": args.gpus, "steps": steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "ms_per_frame": ms, "mrays_per_s": (rays / ms / 1e3) if rays else None,
            "kernel_ms_cuda_events": kernel_ms,
            "config": {"workload": cfg["name"], "device": "1x B200 (the reference is single-GPU; it ships no CPU renderer)", "how": how,
                       "spp": spp},
            "e2e": {"value": value, "unit": "Mpaths/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    if cb:
        line["cpu_baseline"] = cb
    print(json.dumps(line), flush=True)


def run_child(args) -> None:
    """helper modes executed in a child process of the reference arm"""
    if args.child == "cpu-baseline":
        print(json.dumps(cpu_baseline(args.config, build_desc(args.config))), flush=True)
    elif args.child == "dump-scene":
        build_desc(args.config, args.scene_n).save(args.out)
        print(json.dumps({"ok": True}), flush=True)


def main() -> None:
    # stdout carries exactly ONE JSON line: anything libraries print on fd 1 (NCCL's version banner, ...) goes to stderr
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    sys.stdout = real_stdout
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--config", choices=sorted(CONFIGS), default="c1")
    ap.add_argument("--spp", type=int, default=0, help="override samples per pixel per step and GPU")
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--ref-device", choices=["gpu", "cpu"], default="gpu")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-other-configs", action="store_true", help="skip the other_configs / c5 / strong sub-records")
    ap.add_argument("--collective", choices=["auto", "ipc", "multimem", "peer", "nccl"], default="auto",
                    help="N > 1: rt_group of the C-ABI (auto / ipc), or the A/B forms: torch symmetric memory with NVLS multimem / "
                         "peer loads in the fused kernel, or the plain NCCL reduce")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the frame (and, with one GPU, the accumulator) of the last timed step as DIR/<name>.npy")
    ap.add_argument("--child", choices=["cpu-baseline", "dump-scene"], default=None, help=argparse.SUPPRESS)
    ap.add_argument("--scene-n", type=int, default=0, help=argparse.SUPPRESS)
    ap.add_argument("--out", default="", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if args.child:
        run_child(args)
        return
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3  # timing rule: W >= 3
    if args.gpus > 1 and "WORLD_SIZE" not in os.environ:
        # convenience: re-launch under torchrun, one rank per GPU
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}", "--master-addr", "127.0.0.1",
               "--master-port", str(29500 + os.getpid() % 1000), str(Path(__file__).resolve())] + sys.argv[1:]
        raise SystemExit(subprocess.call(cmd))
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
