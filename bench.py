#!/usr/bin/env python
"""bench.py — Mrays/s of the NeRFshop render path at 1920x1080 on the synthetic nerf/fox-shaped workload.

  python bench.py --gpus N --steps K --warmup W [--impl native|reference] [--dump-outputs DIR]

--dump-outputs DIR writes what the last timed step computed, as a caller of the render path receives it, to DIR/rgba.npy
([1080, 1920, 4] float32) and DIR/depth.npy ([1080, 1920] float32). The inputs depend on the arguments only (seeded parameters,
camera index 7*step mod 120), so two builds run with the same arguments can be compared output for output.

A "step" is one frame: Testbed::render_nerf of one camera of a 120-view orbit (a different camera every
step = free-viewpoint orbit), base.json network (hash L=16 F=2 T=2^19, MLPs 64x1 / 64x2), synthetic seeded
parameters (no checkpoint ships with the reference). N > 1: image-plane tiles are partitioned across ranks and
one NCCL all-gather assembles the framebuffer inside the step.

value      : whole-job Mrays/s with the output staying in HBM (per-step CUDA-event time, max over ranks)
e2e.value  : the same with every frame delivered to pinned HOST memory inside the timed region, through the C ABI's host-buffer entry point
             nsb_render_host_async / nsb_host_frame_wait (frame description host->device, RGBA+depth device->host; two frames in flight, so
             the 41.5 MB copy of frame k overlaps the render of frame k+1; N > 1: rank 0 copies the gathered frame on a second stream)
roofline   : the one kernel of the step (k_render_fused): algorithmic 512 B hash-grid gather per sample
             (SURVEY.md §8d) x samples of the frame / its CUDA-event duration, against measured HBM peak
gpu_baseline: (N = 1) the reference's OWN CUDA path — Testbed::render_nerf, NerfTracer::trace and every kernel they launch, compiled
             by nvcc for sm_100a from /root/reference (oracle/_ref, built where the reference exists; only tiny-cuda-nn's network, an
             absent submodule, is replaced by this repository's nsb_inference) — timed in the same process on the same cameras.
configs    : (N = 1) BASELINE.json configs[2] (one cage, 3,072 tets) and configs[3] (unit-cube scene, 3 cages + membrane, poisson target)
             at 1920x1080: native and reference-CUDA Mrays/s, samples, roofline fraction, L-inf between the two.
cpu_baseline / --impl reference: the reference's Testbed::render_nerf compiled for the CPU (oracle/_ref/libnerfshop_ref.so: its own host
             loop and kernels, OpenMP over the kernels' grids; the network is the oracle's CPU restatement) when that library is present,
             else the oracle port; all host cores, bounded sample (a 1/64-resolution frame of the same orbit), median over the steps.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

W, H = 1920, 1080
CPU_W, CPU_H = 240, 135  # bounded CPU sample: 1/64 of the pixels of the same camera
N_ORBIT = 120
METRIC = "Mrays/s @1920x1080 nerf/fox render (synthetic params)"
BYTES_PER_SAMPLE = 512   # 16 levels x 8 corners x 2 fp16 (SURVEY.md §8d)
FLOP_PER_SAMPLE = 20480  # both MLPs


_REAL_STDOUT = None


def emit(line: str) -> None:
    """The one JSON line, on the process's original stdout."""
    out = _REAL_STDOUT or sys.stdout
    out.write(line + "\n")
    out.flush()


def load_traffic():
    """DRAM bytes per launch of k_render_fused from the committed `ncu --set full` digest (profiles/), or None."""
    import glob
    import re

    best = None
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_ncu_render_fused*.txt"))):
        txt = open(path).read()
        rd = re.search(r"dram__bytes_read\.sum\s+([0-9.]+)\s+(\w+)", txt)
        wr = re.search(r"dram__bytes_write\.sum\s+([0-9.]+)\s+(\w+)", txt)
        if rd and wr:
            scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
            best = (float(rd.group(1)) * scale.get(rd.group(2), 1.0) + float(wr.group(1)) * scale.get(wr.group(2), 1.0), os.path.basename(path))
    return best


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["hbm_gbs"]), float(d.get("bf16_tflops_sustained", d.get("bf16_tflops", 1590.0))), "measured"
        except Exception:
            pass
    return 6650.0, 1590.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.index), "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            parts = [p.strip() for p in r.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm)}


def cpu_reference_run(steps: int, warmup: int, threads: int | None = None):
    """The CPU arm: the reference's own render_nerf compiled for the CPU (oracle/_ref) when available, else the oracle port.
    All host cores, threads pinned (OMP_PROC_BIND / OMP_PLACES are set by main() before any OpenMP runtime starts), bounded sample per step.
    Returns (Mrays/s from the MEDIAN step, median ms, cores, samples per frame, kind, (p10, p90) ms)."""
    from nerfshop_b200 import synthetic as syn
    from oracle import oracle as orc

    model = syn.make_model(seed=1337)
    occ = syn.make_occupancy(model)
    o = orc.Oracle(model.desc, model.params, occ)
    cores = orc.set_threads(threads or (os.cpu_count() or 1))
    kind = "port"
    ref = None
    try:
        from oracle import ref as _ref

        if _ref.available():
            ref, kind = _ref, "reference"
    except Exception:
        ref = None
    cams = syn.orbit_cameras(N_ORBIT)
    times, samples = [], 0
    for i in range(warmup + steps):
        f = syn.make_frame(model, cams[(i * 7) % N_ORBIT], CPU_W, CPU_H)
        t0 = time.perf_counter()
        if ref is not None:
            _, _, info = ref.render(f, occ, o.inference)
            n = info["n_inferred"] // 2  # the reference infers every (padded) batch twice
        else:
            _, _, st, _ = o.render(f)
            n = st.n_samples
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
            samples += n
    med = float(np.median(times))
    mrays = CPU_W * CPU_H / med / 1e6
    return mrays, med * 1e3, cores, samples / max(len(times), 1), kind, (float(np.percentile(times, 10)) * 1e3, float(np.percentile(times, 90)) * 1e3)


def measure_reference_cuda_and_edit_configs(r, model, occ, cams, fb, depth, flush, steps, dev):
    """N = 1 only. (1) gpu_baseline: the reference's CUDA path (oracle/_ref, nvcc build of /root/reference's render path; network = nsb_inference)
    on the orbit cameras of configs[1]. (2) configs[2] / configs[3] at 1080p, native and reference-CUDA. CUDA events around each frame, L2 flushed
    between frames, 3 warm-up frames, median over the timed frames (both arms)."""
    import torch

    from nerfshop_b200 import editing, synthetic as syn
    from nerfshop_b200.renderer import NerfRenderer

    try:
        from oracle import ref

        ref.cuda_lib()
    except Exception as e:  # the library is built where /root/reference exists and travels with the repo
        return {"unavailable": f"oracle/_ref/libnerfshop_ref_cuda.so not loadable: {e}"}, None

    def time_frames(render_fn, frames, n):
        ms = []
        for i in range(3 + n):
            flush.zero_()
            fb.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            render_fn(frames[i % len(frames)])
            e1.record()
            torch.cuda.synchronize(dev)
            if i >= 3:
                ms.append(e0.elapsed_time(e1))
        return float(np.median(ms)), ms  # median: the reference arm syncs with the host every round, one descheduled host thread would own a mean

    def both_arms(rr, rc, frames, n):
        nat_ms, _ = time_frames(lambda f: rr.render(f, fb, depth), frames, n)
        smp, kms = [], []
        for f in frames:  # samples + fused-kernel time per camera (own events inside nsb_render)
            rr.render(f, fb, depth)
            st = rr.stats()
            smp.append(st.n_samples)
            kms.append(st.fused_ms)
        ref_ms, _ = time_frames(lambda f: rc.render(f, rr, fb, depth), frames, n)
        a = torch.zeros_like(fb)
        b = torch.zeros_like(fb)
        rr.render(frames[0], a, depth)
        _, _, info = rc.render(frames[0], rr, b, depth)
        torch.cuda.synchronize(dev)
        hbm, _, _ = load_peaks()
        s_mean, k_mean = float(np.mean(smp)), float(np.mean(kms))
        return {
            "native": {"value": W * H / nat_ms / 1e3, "unit": "Mrays/s", "ms_per_step": nat_ms, "samples_per_frame": s_mean, "kernel_ms": k_mean,
                       "roofline_frac": s_mean * BYTES_PER_SAMPLE / (k_mean * 1e-3) / 1e9 / hbm},
            "reference_cuda": {"value": W * H / ref_ms / 1e3, "unit": "Mrays/s", "ms_per_step": ref_ms, "inference_rows_frame0": info["n_inferred"], "inference_calls_frame0": info["n_calls"],
                               "rounds_frame0": info["n_calls"] // 2},
            "native_over_reference_cuda": ref_ms / nat_ms, "linf_rgba_native_vs_reference_cuda_frame0": float((a - b).abs().max().item()), "steps": n,
        }

    what = ("the reference's own CUDA render path (Testbed::render_nerf, NerfTracer::trace, compact/generate/composite/shade kernels; >= 12 launches + 3 host syncs per round, "
            "every batch inferred twice) compiled by nvcc for sm_100a from /root/reference; tiny-cuda-nn's network (absent submodule) replaced by this repository's nsb_inference kernel")
    frames = [syn.make_frame(model, cams[(i * 7) % N_ORBIT], W, H) for i in range(steps)]
    rc = ref.RefCuda(occ)
    res = both_arms(r, rc, frames, steps)
    rc.close()
    gpu_baseline = dict(res["reference_cuda"], kind="reference kernels + host loop, nvcc sm_100a", what=what, native_ms_same_cameras=res["native"]["ms_per_step"],
                        linf_rgba_native_vs_reference_cuda_frame0=res["linf_rgba_native_vs_reference_cuda_frame0"], steps=steps, warmup=3)

    extra = {}
    # configs[2]: nerf/fox scale, ONE cage-deform operator (box cage, 8^3 lattice = 3,072 tets, MVC, +x face pulled), local rotations on
    cage = editing.lattice_cage(model, (0.5, 0.62, 0.78), (0.17, 0.17, 0.17), n_lattice=8)
    ops = [cage.to_op()]
    r.set_edit_operators(ops)
    rc = ref.RefCuda(occ, ops)
    fr = [syn.make_frame(model, cams[(i * 7) % N_ORBIT], W, H, apply_operators=True) for i in range(4)]
    extra["configs[2]"] = dict(both_arms(r, rc, fr, 6), workload=f"nerf/fox scale, one cage ({cage.tets.shape[0]} tets, {cage.lut_idx.size} CSR entries), 1080p, 4 orbit cameras")
    rc.close()
    r.set_edit_operators([])
    # configs[3]: unit-cube scene (aabb_scale 1, cone angle 0: the reference's synthetic-Lego shape), 3 concurrent cages (6^3 lattices), membrane on the first, poisson target on
    m1 = syn.make_model(seed=7, aabb_scale=1)
    occ1 = syn.make_occupancy(m1)
    r1 = NerfRenderer(r.device)
    r1.upload_model(m1.desc, m1.params)
    r1.upload_occupancy(occ1)
    cages = [editing.lattice_cage(m1, (0.5, 0.62, 0.78), (0.17, 0.17, 0.17), n_lattice=6, membrane_seed=5),
             editing.lattice_cage(m1, (0.5, 0.55, 0.27), (0.12, 0.12, 0.15), pull=(0.0, 0.08, 0.0), n_lattice=6),
             editing.lattice_cage(m1, (0.41, 0.30, 0.42), (0.08, 0.14, 0.08), pull=(0.05, 0.0, 0.05), n_lattice=6, copy=True)]
    ops = [c.to_op() for c in cages]
    r1.set_edit_operators(ops)
    rc = ref.RefCuda(occ1, ops)
    fr = [syn.make_frame(m1, cams[(i * 7) % N_ORBIT], W, H, apply_operators=True, poisson_target=True) for i in range(4)]
    extra["configs[3]"] = dict(both_arms(r1, rc, fr, 6), workload=f"unit-cube scene (aabb_scale 1, constant step), 3 cages ({sum(c.tets.shape[0] for c in cages)} tets) + membrane + poisson target, 1080p, 4 orbit cameras")
    rc.close()
    r1.close()
    return gpu_baseline, extra


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-baseline", action="store_true", help="skip the reference-CUDA arm and the edit configurations (N = 1 extras)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's RGBA and depth as DIR/rgba.npy and DIR/depth.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs applies to --impl native")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world == 1:
        # pin the CPU arm's OpenMP threads (the round-1 arm swung 3.4x between two boxes with free-floating threads). Single-process runs only:
        # under torchrun every rank would bind its main thread to the same first core and the ranks' launch loops would time-share it.
        os.environ.setdefault("OMP_PROC_BIND", "close")
        os.environ.setdefault("OMP_PLACES", "cores")
    else:
        # rank 0 prints ONE JSON line: NCCL's version banner (NCCL_DEBUG=VERSION or higher, set by some boxes) goes to stdout, so it is switched off
        os.environ.pop("NCCL_DEBUG", None)
        if os.environ.get("NSB_NCCL_DEBUG"):
            os.environ["NCCL_DEBUG"] = os.environ["NSB_NCCL_DEBUG"]
    # ... and whatever else a library writes to file descriptor 1 goes to stderr: the JSON line is the only thing on the real stdout
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    config = {"workload": "nerf/fox 1080p free-viewpoint orbit, hash L=16 F=2 T=2^19, MLP 64x1 + 64x2 (configs[1])", "resolution": [W, H],
              "cameras": f"{N_ORBIT}-view orbit about (0.5, 0.5, 0.5), radius 1.45, height +0.35 (NGP units; closer than BASELINE.md's radius 2.0: more covered pixels, more samples per frame), look-at centre, focal 1080 px, one camera per step (index 7*step mod {N_ORBIT})", "parallelism": f"image-tile partition x{world}" if world > 1 else "single GPU"}

    if args.impl == "reference":
        if rank != 0:
            return
        steps, warm = args.steps, args.warmup
        mrays, ms, cores, spf, kind, (p10, p90) = cpu_reference_run(steps, warm)
        sample = f"{CPU_W}x{CPU_H} frame (1/64 of the 1080p pixels) of the same orbit per step, {cores} pinned threads, median of {steps} steps (p10 {p10:.0f} ms, p90 {p90:.0f} ms), {warm} warm-up"
        note = ("the reference's Testbed::render_nerf / NerfTracer::trace / kernels compiled for the CPU from /root/reference (oracle/_ref); tiny-cuda-nn's network (absent submodule) = the oracle's CPU restatement"
                if kind == "reference" else "CPU oracle port of the reference path (oracle/_ref/libnerfshop_ref.so not present)")
        emit(json.dumps({
            "impl": "reference", "metric": METRIC, "value": mrays, "unit": "Mrays/s", "n_gpus": 0, "steps": steps, "warmup": warm,
            "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f16/f32", "data": "synthetic",
            "config": dict(config, note=note),
            "cpu_baseline": {"value": mrays, "unit": "Mrays/s", "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": mrays, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }))
        return

    import torch
    import torch.distributed as dist

    from nerfshop_b200 import abi, parallel, synthetic as syn
    from nerfshop_b200.renderer import NerfRenderer

    assert torch.cuda.is_available(), "bench.py needs a GPU; there is no CPU fallback"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    model = syn.make_model(seed=1337)
    occ = syn.make_occupancy(model)
    r = NerfRenderer(local_rank)
    r.upload_model(model.desc, model.params)
    r.upload_occupancy(occ)
    cams = syn.orbit_cameras(N_ORBIT)

    fb = torch.zeros((H, W, 4), dtype=torch.float32, device=dev)
    depth = torch.zeros((H, W), dtype=torch.float32, device=dev)
    n_tiles = [r.tiles_for_rank(W, H, k, world) for k in range(world)]
    max_tiles = max(n_tiles)
    if world > 1:
        shard = torch.zeros(max_tiles * 128 * 5, dtype=torch.float32, device=dev)            # [tiles*128 float4 | tiles*128 depth]
        gathered = torch.zeros((world, max_tiles * 128 * 5), dtype=torch.float32, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    host_fb = torch.zeros((H, W, 4), dtype=torch.float32).pin_memory()
    host_depth = torch.zeros((H, W), dtype=torch.float32).pin_memory()
    stream = torch.cuda.current_stream(dev)
    launches_per_step = 2 + (2 if world > 1 else 0)  # k_prepare_rays + k_render_fused (+ k_pack_tiles + k_unpack_gathered; the all-gather is NCCL's)

    def device_step(i, fb=fb, depth=depth):
        """One frame, output left in HBM (for N > 1: render own tiles, pack, all-gather, unpack every shard)."""
        f = syn.make_frame(model, cams[(i * 7) % N_ORBIT], W, H, rank=rank, world=world)
        fb.zero_()  # render_buffer.clear_frame
        r.render(f, fb, depth)
        if world > 1:
            parallel.gather_framebuffer(r, fb, rank, world, shard, gathered, depth)

    def timed(step_fn, n_warm, n_steps):
        for i in range(n_warm):
            step_fn(i)
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        evs = []
        kern_ms, samples = [], []
        wall0 = time.perf_counter()
        for i in range(n_steps):
            flush.zero_()  # L2 flush between timed iterations, outside the per-step event bracket
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            step_fn(n_warm + i)
            e1.record(stream)
            evs.append((e0, e1))
            st = r.stats()  # synchronises on the render kernel's own events
            kern_ms.append(st.fused_ms)
            samples.append(st.n_samples)
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        wall = time.perf_counter() - wall0
        total_ms = sum(a.elapsed_time(b) for a, b in evs)
        t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), wall, kern_ms, samples

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    total_ms, wall, kern_ms, samples = timed(device_step, args.warmup, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:  # fb / depth still hold the last timed step (for N > 1: the gathered frame)
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "rgba.npy"), fb.cpu().numpy())
        np.save(os.path.join(args.dump_outputs, "depth.npy"), depth.cpu().numpy())

    # ---- e2e: every step's frame ends in (pinned) HOST memory; the copy of frame k overlaps the render of frame k+1, two frames in flight ----
    # N = 1: the C ABI's host-buffer entry point nsb_render_host_async / nsb_host_frame_wait (the consumer takes frame k-1 while frame k renders).
    # N > 1: render + gather into one of two device framebuffers, rank 0 copies it out on a second stream.
    host_fbs = [host_fb, torch.zeros((H, W, 4), dtype=torch.float32).pin_memory()]
    host_depths = [host_depth, torch.zeros((H, W), dtype=torch.float32).pin_memory()]
    pending = {}
    if world > 1:
        fbs, depths = [fb, torch.zeros_like(fb)], [depth, torch.zeros_like(depth)]
        copy_stream = torch.cuda.Stream(dev)
        copy_done = [torch.cuda.Event(), torch.cuda.Event()]

    def e2e_step(i):
        b = i & 1
        f = syn.make_frame(model, cams[(i * 7) % N_ORBIT], W, H, rank=rank, world=world)
        if world == 1:
            pending[b] = r.render_to_cpu_async(f, host_fbs[b], host_depths[b])
            if (b ^ 1) in pending:
                r.wait_host_frame(pending.pop(b ^ 1))  # frame i-1 is now in host_fbs[b ^ 1]
        else:
            stream.wait_event(copy_done[b])  # the copy that last read this framebuffer (two steps ago)
            device_step(i, fbs[b], depths[b])
            if rank == 0:
                done = torch.cuda.Event()
                done.record(stream)
                with torch.cuda.stream(copy_stream):
                    copy_stream.wait_event(done)
                    host_fbs[b].copy_(fbs[b], non_blocking=True)
                    host_depths[b].copy_(depths[b], non_blocking=True)
                    copy_done[b].record(copy_stream)

    def e2e_drain():
        for t in list(pending.values()):
            r.wait_host_frame(t)
        pending.clear()

    def timed_wall(step_fn, n_warm, n_steps):
        for i in range(n_warm):
            step_fn(i)
        e2e_drain()
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        for i in range(n_steps):
            step_fn(n_warm + i)
        e2e_drain()  # the last frames' copies are inside the timed region
        torch.cuda.synchronize(dev)
        dt = time.perf_counter() - t0
        t = torch.tensor([dt], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    e2e_s = timed_wall(e2e_step, max(3, args.warmup // 2), args.steps)

    # ---- N = 1 extras: the reference's own CUDA path on the same cameras, and the edit configurations ----
    gpu_baseline, extra_configs = None, None
    if world == 1 and not args.no_gpu_baseline:
        gpu_baseline, extra_configs = measure_reference_cuda_and_edit_configs(r, model, occ, cams, fb, depth, flush, min(args.steps, 8), dev)

    if rank == 0:
        hbm_gbs, tflops, peak_kind = load_peaks()
        traffic = load_traffic()
        ms_per_step = total_ms / args.steps
        value = W * H / (ms_per_step * 1e-3) / 1e6
        e2e_value = W * H * args.steps / e2e_s / 1e6
        k_ms = float(np.mean(kern_ms))
        s_mean = float(np.mean(samples))  # this rank's samples per frame
        achieved = s_mean * BYTES_PER_SAMPLE / (k_ms * 1e-3) / 1e9
        out = {
            "metric": METRIC, "value": value, "unit": "Mrays/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f16 (hash features, MLP operands and tcgen05 accumulators, as the reference's wmma half fragments; fp32 march / deform / composite)",
            "data": "synthetic", "fps": 1e3 / ms_per_step,
            "config": dict(config, l2="flushed between timed steps (256 MiB memset outside the per-step event bracket)",
                           samples_per_frame=s_mean * world, samples_per_ray=s_mean * world / (W * H)),
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "Mrays/s", "h2d_bytes_per_step": int(np.dtype(np.uint8).itemsize * __import__("ctypes").sizeof(abi.NsbFrame)),
                    "d2h_bytes_per_step": W * H * 20, "ms_per_step": e2e_s / args.steps * 1e3},
            "gpu_launches": launches_per_step * args.steps,
            "roofline": {"kernel": "k_render_fused", "bound": "hbm", "achieved": achieved, "peak": hbm_gbs, "unit": "GB/s", "frac": achieved / hbm_gbs,
                         "traffic": traffic[0] if traffic else None, "traffic_source": traffic[1] if traffic else None, "peak_source": peak_kind, "kernel_ms": k_ms, "kernel_share_of_step": k_ms / ms_per_step if world == 1 else None, "samples_per_launch": s_mean,
                         "tensor_tflops": s_mean * FLOP_PER_SAMPLE / (k_ms * 1e-3) / 1e12, "tensor_frac": s_mean * FLOP_PER_SAMPLE / (k_ms * 1e-3) / 1e12 / tflops},
        }
        if world == 1:
            out["gpu_baseline"] = gpu_baseline
            if gpu_baseline and gpu_baseline.get("value"):
                out["vs_gpu_baseline"] = {"device": value / gpu_baseline["value"], "north_star_target": 1.5}
            out["configs"] = extra_configs
        if world == 1 and not args.no_cpu_baseline:
            mrays, ms, cores, _, kind, (p10, p90) = cpu_reference_run(3, 1)
            out["cpu_baseline"] = {"value": mrays, "unit": "Mrays/s", "cores": cores, "kind": kind,
                                   "sample": f"median of 3 frames of {CPU_W}x{CPU_H} (1/64 of the 1080p pixels) of the same orbit after 1 warm-up, {cores} pinned threads (p10 {p10:.0f} / p90 {p90:.0f} ms)"}
        emit(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()
    r.close()


if __name__ == "__main__":
    main()
