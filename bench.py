#!/usr/bin/env python
"""bench.py -- Mpixels/s of the projection-remap hot path on synthetic 8K equirect frames (BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config cfg2|cfg3|cfg4] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A step = one yuv420p frame (3 planes) through the hot path ([segmented low-pass] -> gather).  Default
workload = BASELINE.json configs[1] ("cfg2": MONO 7680x3840 equirect -> CUBEMAP_32 edge 1280 = 3840x2560,
bicubic, low-pass off).  Mpx/s counts INPUT-plane pixels consumed (SURVEY.md 8d).

Legs (one JSON line on rank 0):
  value         frames resident in HBM, one T360B200_transformFrameAsync per frame, CUDA events on the launch
                stream, barrier + synchronize on both sides, max over ranks.  Inputs rotate through a ring larger
                than L2 so every step reads its frame from HBM.
  e2e           same metric through the reference's own C-ABI (VideoFrameTransform_transformFramePlane) with
                pinned HOST planes: H2D of the inputs and D2H of the outputs are inside the timed region.
  roofline      the frame gather kernel (all three planes in one launch): algorithmic bytes (input + output
                plane bytes, SURVEY.md 8d) / its CUDA-event duration / measured HBM peak (MEASURED_PEAKS.json).
  cpu_baseline  the reference's own CPU path (oracle/_ref: unmodified reference sources driving cv2) on this
                box's host cores, bounded sample (N=1, rank 0 only).
  --impl reference   only that CPU path, as its own JSON line.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

METRIC = "Mpixels/s 8K equirect->cubemap bicubic (input-plane pixels consumed per second)"

CONFIGS = {  # BASELINE.json configs[1..3]
    "cfg2": dict(desc="MONO 7680x3840 equirect -> CUBEMAP_32 edge 1280 (3840x2560), bicubic, low-pass off, yuv420p frame (3 planes)",
                 ov=dict(interpolation_alg=2, enable_low_pass_filter=0), inp=(7680, 3840), out=(3840, 2560)),
    "cfg3": dict(desc="cfg2 + low-pass: num_horizontal_segments=32 num_vertical_segments=15 adjust_kernel=1",
                 ov=dict(interpolation_alg=2, enable_low_pass_filter=1, num_horizontal_segments=32, num_vertical_segments=15,
                         adjust_kernel=1), inp=(7680, 3840), out=(3840, 2560)),
    "cfg4": dict(desc="TOP_BOTTOM stereo 7680x7680 equirect -> EAC_32 (3840x5120), Lanczos4, low-pass on, yuv420p frame",
                 ov=dict(input_stereo_format=0, output_stereo_format=0, output_layout=6, interpolation_alg=4,
                         enable_low_pass_filter=1, num_horizontal_segments=32, num_vertical_segments=15, adjust_kernel=1),
                 inp=(7680, 7680), out=(3840, 5120)),
}


def measured_hbm_peak():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons while the timed regions run."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,utilization.gpu,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "50"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.split(",") for r in Path(self.f.name).read_text().splitlines() if r.count(",") >= 7]
        os.unlink(self.f.name)
        sm, reasons, busy = [], set(), []
        for r in rows:
            try:
                r = [c.strip() for c in r]
                clk, mx, util = float(r[0]), float(r[1]), float(r[3])
            except ValueError:
                continue
            sm.append(clk)
            if util > 0:
                busy.append(clk)
            out["sm_max_mhz"] = mx
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        use = busy or sm
        if use:
            out["sm_mhz"] = statistics.median(use)
        out["samples"] = len(sm)
        out["samples_under_load"] = len(busy)
        out["reasons"] = sorted(reasons)
        return out


# ------------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the reference's own CPU implementation of the path on the host cores
# ------------------------------------------------------------------------------------------------------
def reference_cpu_run(cfg, steps, warmup, budget_s=None):
    """Times `steps` frames (3 planes each) through oracle/_ref + cv2 (kind 'reference'), or through the plain-C
    oracle port when the compiled reference is absent (kind 'port').  Plans are built outside the timed region,
    like on the GPU side.  Returns (seconds_per_step list, kind, cores, sample description)."""
    from oracle import ref_harness as rh
    from transform360_b200 import synth
    from transform360_b200.stream import StreamSpec
    spec = StreamSpec(cfg["inp"][0], cfg["inp"][1], cfg["out"][0], cfg["out"][1])
    frames = [[synth.noise_plane(*spec.plane_dims(p)[:2], plane=p, frame=f) for p in range(3)] for f in range(2)]
    cores = os.cpu_count() or 1
    if rh.ref_available():
        import cv2
        cv2.setNumThreads(cores)
        ref = rh.RefTransform(rh.default_context(**cfg["ov"]))
        for idx, plane in ((0, 0), (1, 1)):
            iw, ih, ow, oh, _ = spec.plane_dims(plane)
            assert ref.generate_map(iw, ih, ow, oh, idx)

        def one(frame):
            for p in range(3):
                iw, ih, ow, oh, idx = spec.plane_dims(p)
                ref.transform_plane(frame[p], ow, oh, idx, image_plane=p)
        kind, used = "reference", cores
    else:
        from oracle import c_oracle as co
        octx = rh.default_context(**cfg["ov"])
        plans = [co.OraclePlan(octx, *spec.plane_dims(p)[:4]) for p in (0, 1)]

        def one(frame):
            for p in range(3):
                iw, ih, ow, oh, idx = spec.plane_dims(p)
                co.transform_plane(octx, plans[idx], frame[p], ow, oh, map_index=idx)
        kind, used = "port", 1
    for i in range(warmup):
        one(frames[i % 2])
    times = []
    t_begin = time.perf_counter()
    for i in range(steps):
        t0 = time.perf_counter()
        one(frames[i % 2])
        times.append(time.perf_counter() - t0)
        if budget_s and time.perf_counter() - t_begin > budget_s:
            break
    sample = (f"{len(times)} yuv420p frames of the workload ({'unmodified reference sources + cv2 ' + __import__('cv2').__version__ if kind == 'reference' else 'plain-C oracle port'}), "
              f"{used} host thread(s), plans prebuilt, noise frames")
    return times, kind, used, sample


def run_reference_arm(args, cfg, rank):
    if rank != 0:
        return
    times, kind, cores, sample = reference_cpu_run(cfg, args.steps, max(args.warmup, 1))
    from transform360_b200.stream import StreamSpec
    spec = StreamSpec(cfg["inp"][0], cfg["inp"][1], cfg["out"][0], cfg["out"][1])
    px = spec.input_pixels_per_frame()
    total = sum(times)
    v = px * len(times) / total / 1e6
    line = {
        "impl": "reference", "metric": METRIC, "value": round(v, 2), "unit": "Mpx/s", "n_gpus": args.gpus, "steps": len(times),
        "warmup": max(args.warmup, 1), "ms_per_step": round(1e3 * total / len(times), 3), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": f"{args.config}: {cfg['desc']}", "engine": "reference CPU path on host cores"},
        "cpu_baseline": {"value": round(v, 2), "unit": "Mpx/s", "cores": cores, "kind": kind, "sample": sample,
                         "best_ms_per_step": round(1e3 * min(times), 3), "median_ms_per_step": round(1e3 * statistics.median(times), 3)},
        "e2e": {"value": round(v, 2), "unit": "Mpx/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------
class DeviceFrames:
    """Synthetic frames of one config resident in HBM: a ring of input frames larger than L2 and two output frames."""

    def __init__(self, spec, dev, rank, world, synth):
        self.spec = spec
        frame_bytes = spec.input_pixels_per_frame()
        self.ring = max(4, -(-200_000_000 // frame_bytes))
        pitch = lambda w: (w + 255) // 256 * 256
        self.d_in, self.d_out = [], []
        for f in range(self.ring):
            gframe = rank + f * world  # global frame index handled by this rank (round-robin sharding)
            self.d_in.append([synth.noise_plane_torch(*spec.plane_dims(p)[:2], plane=p, frame=gframe, device=dev, pitch=pitch(spec.plane_dims(p)[0]))
                              for p in range(3)])
        import torch
        for f in range(2):
            self.d_out.append([torch.zeros((spec.plane_dims(p)[3], pitch(spec.plane_dims(p)[2])), dtype=torch.uint8, device=dev) for p in range(3)])
        self.in_args = [[(t.data_ptr(), t.stride(0)) for t in fr] for fr in self.d_in]
        self.out_args = [[(t.data_ptr(), t.stride(0)) for t in fr] for fr in self.d_out]


DUMP_LIMIT_BYTES = 64_000_000 - 4096  # --dump-outputs: at most 64 MB in all, .npy headers included


def dump_outputs(dump_dir, spec, planes):
    """Writes the output planes of one frame as float32 DIR/out_{y,u,v}.npy: whole planes while the frame fits
    DUMP_LIMIT_BYTES as float32 (cfg2 does), else the same seeded sample of rows of every plane in every run."""
    import numpy as np
    import torch
    total = spec.output_pixels_per_frame() * 4
    frac = min(1.0, DUMP_LIMIT_BYTES / total)
    rng = np.random.default_rng(0)
    out = Path(dump_dir)
    out.mkdir(parents=True, exist_ok=True)
    for p, t in enumerate(planes):
        ow, oh = spec.plane_dims(p)[2:4]
        a = t[:, :ow]
        if frac < 1.0:
            rows = np.sort(rng.choice(oh, int(oh * frac), replace=False))
            a = a[torch.from_numpy(rows).to(a.device)]
        np.save(out / f"out_{'yuv'[p]}.npy", a.cpu().numpy().astype(np.float32))


def measure_config(name, cfg, ctx, spec, K, warmup, dev, rank, world, barrier, want_e2e, e2e_steps, dump_dir=None):
    """Device-resident leg, roofline leg (the frame gather kernel alone: isolated launches and a back-to-back stream) and,
    optionally, the end-to-end leg of one config.  Returns a dict of raw measurements (this rank's; times are reduced
    with MAX over ranks by the caller where the contract asks for it).  dump_dir: where the output frame of the last timed
    step goes (dump_outputs)."""
    import torch
    import transform360_b200 as t360
    from transform360_b200 import synth
    from transform360_b200.stream import FrameTransformer
    t_plan = time.perf_counter()
    ft = FrameTransformer(ctx, spec)
    plan_seconds = time.perf_counter() - t_plan
    fr = DeviceFrames(spec, dev, rank, world, synth)
    ring = fr.ring
    tstream = torch.cuda.Stream(device=dev)  # a real (non-default) stream: the events below bracket the library's kernels
    stream = tstream.cuda_stream
    assert stream != 0
    calls = [[ft.frame_call(fr.in_args[i], fr.out_args[o]) for o in range(2)] for i in range(ring)]

    def run(call_table, n, first=0):
        for i in range(first, first + n):
            if not call_table[i % ring][i % 2](stream):
                raise RuntimeError("T360B200_transformFrameAsync failed")

    torch.cuda.synchronize()  # the ring was filled on torch's default stream
    run(calls, warmup)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches0 = t360.kernel_launch_count()
    e0.record(tstream)
    run(calls, K)
    e1.record(tstream)
    barrier()
    out = {"ms_total": e0.elapsed_time(e1), "launches": t360.kernel_launch_count() - launches0, "ring": ring,
           "plan_seconds": plan_seconds, "tiles": [list(ft.vft.plan_tile_counts(0)), list(ft.vft.plan_tile_counts(1))]}
    if dump_dir is not None:  # before the legs below overwrite the output frames
        dump_outputs(dump_dir, spec, fr.d_out[(K - 1) % 2])

    # ---- the dominant kernel alone: with the low-pass enabled a frame call also launches the blur kernels, so the gather
    # is timed through a second transform with the same geometry and the low-pass switched off (same jobs, same records)
    ft_gather = ft
    if cfg["ov"].get("enable_low_pass_filter"):
        ft_gather = FrameTransformer(t360.make_context(**dict(cfg["ov"], enable_low_pass_filter=0)), spec)
    gcalls = [[ft_gather.frame_call(fr.in_args[i], fr.out_args[o]) for o in range(2)] for i in range(ring)]
    run(gcalls, 3)
    barrier()
    Kl = min(K, 200)
    gl0 = t360.kernel_launch_count()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(Kl)]
    for i in range(Kl):
        ev[i][0].record(tstream)
        run(gcalls, 1, i)
        ev[i][1].record(tstream)
    barrier()
    out["gather_launches_per_call"] = (t360.kernel_launch_count() - gl0) / Kl
    out["gather_ms"] = [a.elapsed_time(b) for a, b in ev]
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g0.record(tstream)
    run(gcalls, Kl)
    g1.record(tstream)
    barrier()
    out["gather_streamed_ms"] = g0.elapsed_time(g1) / Kl

    # ---- a frame every rank has in common (global frame 0), for the cross-rank identity check
    common = [synth.noise_plane_torch(*spec.plane_dims(p)[:2], plane=p, frame=0, device=dev, pitch=fr.d_in[0][p].stride(0)) for p in range(3)]
    torch.cuda.synchronize()
    if not ft.frame_call([(t.data_ptr(), t.stride(0)) for t in common], fr.out_args[0])(stream):
        raise RuntimeError("T360B200_transformFrameAsync failed")
    torch.cuda.synchronize()
    import hashlib
    hsh = hashlib.sha256()
    for p in range(3):
        hsh.update(fr.d_out[0][p][:, :spec.plane_dims(p)[2]].contiguous().cpu().numpy().tobytes())
    out["common_frame_sha"] = hsh.hexdigest()[:16]

    # ---- end to end through the reference-facing C-ABI with pinned host planes ------------------------------------
    if want_e2e:
        Ke = e2e_steps
        h_ring = 2
        h_in = [[torch.empty((spec.plane_dims(p)[1], spec.plane_dims(p)[0]), dtype=torch.uint8).pin_memory() for p in range(3)]
                for _ in range(h_ring)]
        for f in range(h_ring):
            for p in range(3):
                h_in[f][p].copy_(fr.d_in[f][p][:, :spec.plane_dims(p)[0]].cpu())
        h_out = [[torch.empty((spec.plane_dims(p)[3], spec.plane_dims(p)[2]), dtype=torch.uint8).pin_memory() for p in range(3)]
                 for _ in range(h_ring)]
        hin_args = [[(t.data_ptr(), t.stride(0)) for t in f] for f in h_in]
        hout_args = [[(t.data_ptr(), t.stride(0)) for t in f] for f in h_out]
        lib_stream = torch.cuda.ExternalStream(ft.vft.stream, device=dev)
        for i in range(3):
            ft.transform_frame_host(hin_args[i % h_ring], hout_args[i % h_ring])
        barrier()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        per_step = []
        w0 = time.perf_counter()
        s0.record(lib_stream)
        for i in range(Ke):
            t0 = time.perf_counter()
            ft.transform_frame_host(hin_args[i % h_ring], hout_args[i % h_ring])  # synchronous: output complete on return
            per_step.append((time.perf_counter() - t0) * 1e3)
        s1.record(lib_stream)
        barrier()
        wall_ms = (time.perf_counter() - w0) * 1e3
        ms_e2e = s0.elapsed_time(s1)
        if ms_e2e <= 0:
            ms_e2e = wall_ms
        # sanity: the host path and the device path produce the same bytes for the same frame
        ft.transform_frame_host(hin_args[0], hout_args[0])
        run(calls, 1, 0)
        torch.cuda.synchronize()
        same = all(torch.equal(h_out[0][p], fr.d_out[0][p][:, :spec.plane_dims(p)[2]].cpu()) for p in range(3))
        out["e2e"] = {"ms_total": ms_e2e, "wall_ms": wall_ms, "steps": Ke, "median_ms": statistics.median(per_step), "best_ms": min(per_step),
                      "matches_device_leg": bool(same)}
    ft.close()
    if ft_gather is not ft:
        ft_gather.close()
    del fr
    torch.cuda.empty_cache()
    return out


def kernel_size_of(cfg):
    return {1: 2, 2: 4, 4: 8}.get(cfg["ov"]["interpolation_alg"], 0)


def roofline_of(name, cfg, spec, m, ms_per_step):
    peak, peak_src = measured_hbm_peak()
    in_px, out_px = spec.input_pixels_per_frame(), spec.output_pixels_per_frame()
    gather_bytes = in_px + out_px  # every input byte read once, every output byte written once (SURVEY.md 8d)
    avg = statistics.mean(m["gather_ms"])
    achieved = gather_bytes / (avg * 1e-3) / 1e9
    traffic = None
    tp = ROOT / "profiles" / "traffic.json"
    if tp.exists():
        try:
            traffic = json.loads(tp.read_text()).get(name, {}).get("frame_gather_dram_bytes_per_launch")
        except Exception:
            traffic = None
    k = kernel_size_of(cfg)
    return {"bound": "hbm", "kernel": f"gatherFrameKernel<{k}> (Y+U+V jobs of one frame, one persistent warp-specialised launch)",
            "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s", "frac": round(achieved / peak, 4),
            "traffic": traffic, "algorithmic_bytes_per_launch": gather_bytes, "avg_launch_ms": round(avg, 5),
            "median_launch_ms": round(statistics.median(m["gather_ms"]), 5),
            "streamed_launch_ms": round(m["gather_streamed_ms"], 5),
            "frac_streamed": round(gather_bytes / (m["gather_streamed_ms"] * 1e-3) / 1e9 / peak, 4),
            "share_of_step": round(m["gather_streamed_ms"] / ms_per_step, 3),
            "launches_per_timed_call": m["gather_launches_per_call"],
            "read_only_frac": round(in_px / (avg * 1e-3) / 1e9 / peak, 4), "peak_source": peak_src,
            "timing": f"{len(m['gather_ms'])} launches each bracketed by CUDA events on the launch stream (avg/median_launch_ms, frac), and the "
                      f"same launches back to back between two events (streamed_launch_ms, frac_streamed, share_of_step); inputs from the >L2 ring"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--config", default="cfg2", choices=sorted(CONFIGS))
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--e2e-steps", type=int, default=0, help="steps of the host-pointer leg (default min(steps, 100))")
    ap.add_argument("--skip-e2e", action="store_true")
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--skip-other-configs", action="store_true", help="do not add the short cfg3 / cfg4 legs (N=1 only)")
    ap.add_argument("--cpu-steps", type=int, default=12)
    ap.add_argument("--no-numa-bind", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the output frame of the last timed step to DIR/out_{y,u,v}.npy "
                    "(float32; a fixed sample of rows where the frame exceeds 64 MB), rank 0")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path; the reference arm has none")
    cfg = CONFIGS[args.config]
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    args.warmup = max(args.warmup, 3)

    if args.impl == "reference":
        run_reference_arm(args, cfg, rank)
        return

    # Page-locked frame buffers must live on the GPU's own NUMA node (20 vs 55 GB/s H2D on these 2-socket boxes): bind
    # the rank to that node's CPUs before anything is allocated; the original affinity comes back for the CPU baseline.
    from transform360_b200.stream import bind_to_gpu_numa_node
    affinity0 = os.sched_getaffinity(0)
    numa = None if args.no_numa_bind else bind_to_gpu_numa_node(local_rank)

    import torch
    import transform360_b200 as t360
    from transform360_b200.stream import StreamSpec, broadcast_parameters

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product has no CPU fallback; use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    if world != args.gpus and rank == 0:
        print(f"bench.py: note: WORLD_SIZE={world} but --gpus {args.gpus}; using WORLD_SIZE", file=sys.stderr)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(values):
        t = torch.tensor(values, dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(v) for v in t.tolist()]

    # ---- parameters: rank 0 decides, one NCCL broadcast of 112 + 28 bytes (the path's only collective) -----
    ctx = spec = None
    if rank == 0:
        ctx = t360.make_context(**cfg["ov"])
        spec = StreamSpec(cfg["inp"][0], cfg["inp"][1], cfg["out"][0], cfg["out"][1])
    ctx, spec = broadcast_parameters(ctx, spec, rank, world, device=dev)
    in_px, out_px = spec.input_pixels_per_frame(), spec.output_pixels_per_frame()
    K = args.steps
    sampler = ClockSampler(local_rank) if rank == 0 else None
    m = measure_config(args.config, cfg, ctx, spec, K, args.warmup, dev, rank, world, barrier, not args.skip_e2e,
                       args.e2e_steps or min(K, 100), args.dump_outputs if rank == 0 else None)
    (ms_total_max,) = max_over_ranks([m["ms_total"]])
    ms_per_step = ms_total_max / K
    value = in_px * K * world / (ms_total_max * 1e-3) / 1e6
    e2e = None
    if "e2e" in m:
        ms_e2e, wall_ms, med, best = max_over_ranks([m["e2e"]["ms_total"], m["e2e"]["wall_ms"], m["e2e"]["median_ms"], m["e2e"]["best_ms"]])
        Ke = m["e2e"]["steps"]
        e2e = {"value": round(in_px * Ke * world / (ms_e2e * 1e-3) / 1e6, 1), "unit": "Mpx/s", "steps": Ke,
               "ms_per_step": round(ms_e2e / Ke, 4), "wall_ms_per_step": round(wall_ms / Ke, 4),
               "median_ms_per_step": round(med, 4), "best_ms_per_step": round(best, 4),
               "h2d_bytes_per_step": in_px, "d2h_bytes_per_step": out_px,
               "api": "VideoFrameTransform_transformFramePlane x3 planes, pinned host planes (on the GPU's NUMA node), synchronous; large "
                      "planes are streamed: chunked H2D || gather waves || D2H of finished rectangles",
               "matches_device_leg": m["e2e"]["matches_device_leg"]}
    cross_rank_identical = None
    if world > 1:
        shas = [None] * world
        dist.all_gather_object(shas, m["common_frame_sha"])
        cross_rank_identical = len(set(shas)) == 1

    # ---- the other BASELINE configs, short legs in the same process (N = 1 only) -------------------------------------
    others = {}
    if world == 1 and not args.skip_other_configs:
        for name in ("cfg3", "cfg4"):
            if name == args.config:
                continue
            c2 = CONFIGS[name]
            spec2 = StreamSpec(c2["inp"][0], c2["inp"][1], c2["out"][0], c2["out"][1])
            K2 = min(K, 60)
            m2 = measure_config(name, c2, t360.make_context(**c2["ov"]), spec2, K2, 3, dev, 0, 1, barrier, False, 0)
            ms2 = m2["ms_total"] / K2
            others[name] = {"workload": c2["desc"], "steps": K2, "ms_per_step": round(ms2, 5),
                            "value": round(spec2.input_pixels_per_frame() / (ms2 * 1e-3) / 1e6, 1), "unit": "Mpx/s",
                            "gpu_launches_per_step": m2["launches"] / K2, "roofline": roofline_of(name, c2, spec2, m2, ms2)}
    clocks = sampler.stop() if sampler else None

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    cpu_baseline = None
    if world == 1 and not args.skip_cpu_baseline:
        os.sched_setaffinity(0, affinity0)  # the CPU path gets every core again
        times, kind, cores, sample = reference_cpu_run(cfg, args.cpu_steps, 2, budget_s=30.0)
        cpu_baseline = {"value": round(in_px * len(times) / sum(times) / 1e6, 1), "unit": "Mpx/s", "cores": cores, "kind": kind,
                        "sample": sample, "median": round(in_px / statistics.median(times) / 1e6, 1), "best": round(in_px / min(times) / 1e6, 1)}

    line = {
        "metric": METRIC, "value": round(value, 1), "unit": "Mpx/s", "n_gpus": world, "steps": K, "warmup": args.warmup,
        "ms_per_step": round(ms_per_step, 5), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic",
        "config": {"workload": f"{args.config}: {cfg['desc']}", "frames_resident_ring": m["ring"],
                   "l2": f"inputs larger than L2: ring of {m['ring']} x {in_px / 1e6:.1f} MB frames per GPU",
                   "sharding": "frames round-robin over ranks; one NCCL broadcast of context+dims; no pixel traffic",
                   "numa": f"rank bound to NUMA node {numa[0]} ({numa[1]} CPUs) of its GPU" if numa else "no NUMA binding",
                   "output_mpx_per_s": round(out_px * K * world / (ms_total_max * 1e-3) / 1e6, 1),
                   "frames_per_s": round(K * world / (ms_total_max * 1e-3), 1), "plan_seconds": round(m["plan_seconds"], 3),
                   "jobs_luma[gather_staged,gather_general,lowpass_strip_jobs,lowpass_general_jobs]": m["tiles"][0],
                   "jobs_chroma": m["tiles"][1]},
        "e2e": e2e, "gpu_launches": int(m["launches"]), "roofline": roofline_of(args.config, cfg, spec, m, ms_per_step),
        "configs": others or None, "cross_rank_identical": cross_rank_identical, "cpu_baseline": cpu_baseline, "clocks": clocks,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
