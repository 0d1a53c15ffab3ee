#!/usr/bin/env python
"""bench.py -- throughput of the V-PCC rec0 reconstruction hot path on B200.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --steps K --warmup W    # the reference algorithm on the host CPU (oracle port)
    torchrun ... bench.py --gpus N ...                       # one rank per GPU, frames sharded, no collective
    python bench.py ... --dump-outputs DIR                   # + the frames of the last timed step as DIR/*.npy (see dump_outputs)

Workload (`config.workload`; the same for both arms):
  N = 1   BASELINE config 2: a 32-frame GOF, 1024x1024 atlas, 10-bit geometry, 2 maps, occupancy precision 4, grid geometry
          smoothing + colour smoothing ON.  A step = one pass of the hot path over a batch of GOFS_PER_STEP such GOFs.
  N > 1   BASELINE config 3, STRONG scaling: a 300-frame sequence (1280x1344, ~1.1 M points per frame, smoothing ON) as ten
          30-frame GOFs, sharded frame-wise over the N ranks with shard.frames_for_rank (contiguous slices, no collective:
          frames and GOFs are independent, src/lib.rs:114-120).  A step = one pass over the whole sequence.
          (--config c3s runs this workload on one GPU as well: the N = 1 point of the scaling curve.)

  value  points/s with the planes already resident in HBM (kernels only, CUDA events on the launching streams); the resident
         GOFs of a rank go round-robin over three streams, like the three GOFs in flight of the streaming path
  e2e    points/s through the public C ABI (tmc2gpu_submit_gof / tmc2gpu_next_frame) from PINNED HOST planes:
         H2D of every plane and D2H of every reconstructed frame inside the timed region; `e2e.host_ceiling` is the same
         byte traffic as bare pinned copies on two streams (all ranks at once), `e2e.frac_of_host_ceiling` the ratio
  e2e_pageable (N = 1)  the same with the planes in ordinary (pageable) memory, like the reference's `Vec<u8>`
  one_context (N > 1)   rank 0 alone drives ONE tmc2gpu context over all N devices (the topology behind the unchanged
         `Decoder` API): frames sharded inside the library, handed back in order
  roofline  algorithmic bytes of the dominant kernel (fused unpack) / its device time, against the measured HBM peak
  cpu_baseline  the reference's single-threaded algorithm (C restatement, oracle/) on this box's host cores
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the benchmark leaves the tree as it found it (which may be read-only)

import numpy as np  # noqa: E402

import tmc2rs_b200  # noqa: E402,F401
from tmc2rs_b200 import abi, shard, synth  # noqa: E402

METRIC = "reconstructed_points_per_sec"
UNIT = "points/s"


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def build_workload(name: str, frames: int, distinct: int):
    """GOF of `frames` frames cycling `distinct` distinct synthetic frames (generation cost only)."""
    cfg = synth.config(name, frames=min(distinct, frames))
    base = synth.make_gof(cfg)
    return synth.replicate_gof(base, frames), cfg


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows, self.proc, self.idx = [], None, gpu_index
        self.paused = False

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.idx)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            if not self.paused:
                self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7),
                              ("sw_power_cap", 8)):
                if len(r) > col and r[col].lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def bind_to_gpu_numa_node(gpu_index: int):
    """Pin this rank to the CPU cores next to its GPU (NVML affinity) before any pinned memory is allocated, so that the
    staging buffers land on the GPU's own NUMA node.  Best effort: silently keeps the inherited affinity on failure."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = {64 * w + b for w, word in enumerate(words) for b in range(64) if (word >> b) & 1}
        allowed = os.sched_getaffinity(0)
        target = cpus & allowed
        if target:
            os.sched_setaffinity(0, target)
        return sorted(target) if target else None
    except Exception:
        return None


def cpu_reference_run(gof, frames_per_step: int, steps: int, warmup: int, threads: int):
    """The reference algorithm on host cores: oracle port (the Rust reference cannot be built here), single-threaded
    like the reference (README.md:7, src/lib.rs:113) unless --ref-threads asks for frame-parallel workers."""
    from oracle import oracle
    view = abi.GofView(gof)
    F = gof.frame_count

    def one_step(step):
        lo = (step * frames_per_step) % F
        idx = [(lo + k) % F for k in range(frames_per_step)]
        if threads <= 1:
            return sum(oracle.time_frames(view, f, 1) for f in idx)
        from concurrent.futures import ThreadPoolExecutor
        with ThreadPoolExecutor(threads) as ex:     # ctypes releases the GIL
            return sum(ex.map(lambda f: oracle.time_frames(view, f, 1), idx))
    for w in range(warmup):
        one_step(w)
    t0 = time.perf_counter()
    pts = sum(one_step(s) for s in range(steps))
    dt = time.perf_counter() - t0
    return pts, dt


GOFS_PER_STEP = 64          # N = 1: GOFs per step (a step of 64 x 0.5 ms keeps the timed region of 10 steps above 0.3 s)
SEQ_FRAMES, SEQ_GOF = 300, 30   # N > 1: BASELINE config 3


def workload(args, world):
    """(mode, synthetic config name, smoothing, config dict).  The dict depends on the arguments only, so both arms print the
    same one."""
    name = args.config
    if name == "auto":
        name = "c2" if max(world, args.gpus) <= 1 else "c3s"
    strong = name == "c3s"
    sname = "c3" if strong else name
    cfg = synth.config(sname)
    frames = args.frames or (SEQ_GOF if strong else {"c1": 1, "c2": 32, "c3": 32, "c4": 8}.get(sname, 32))
    smoothing = sname != "c1" and not args.no_smoothing
    n = max(world, args.gpus, 1)
    if strong:
        desc = {"workload": f"c3 strong scaling: {SEQ_FRAMES}-frame sequence as {SEQ_FRAMES // SEQ_GOF} GOFs of {SEQ_GOF} frames, "
                            f"synthetic decoded planes + patch metadata, sharded frame-wise over {n} GPU(s)",
                "frames_per_step": SEQ_FRAMES, "frames_per_gof": SEQ_GOF}
    else:
        per = 1 if sname == "c1" else GOFS_PER_STEP
        desc = {"workload": f"{sname}: {frames}-frame GOF, synthetic decoded planes + patch metadata, {per} GOF(s) per step",
                "frames_per_step": frames * per, "frames_per_gof": frames}
    desc.update({"atlas": f"{cfg.width}x{cfg.height}", "maps": 2, "occupancy_precision": cfg.occupancy_precision,
                 "bitdepth_3d": cfg.bitdepth_3d, "smoothing": smoothing,
                 "sharding": (f"{n} rank(s), contiguous frame slices of the sequence, no collective" if strong else
                              f"{n} rank(s), every rank its own GOFs, no collective"),
                 "l2": "inputs of a step exceed the 126 MB L2 (no flush needed)"})
    return ("strong" if strong else "weak"), sname, frames, smoothing, desc


def rank_gofs(mode, frames, rank, world):
    """Frame counts of the GOFs rank `rank` reconstructs per step."""
    if mode == "weak":
        return [frames] * (1 if frames == 1 else GOFS_PER_STEP)
    lo, hi = shard.frames_for_rank(SEQ_FRAMES, rank, world)
    out, f = [], lo
    while f < hi:                      # the rank's slice, cut at the sequence's GOF boundaries
        nxt = min(hi, (f // SEQ_GOF + 1) * SEQ_GOF)
        out.append(nxt - f)
        f = nxt
    return out


def host_copy_ceiling(torch, dev, h2d_bytes, d2h_bytes, iters, barrier):
    """The step's byte traffic as bare pinned copies (H2D and D2H on two streams): what the host side of this box can move
    with every rank busy.  Returns seconds per step."""
    hi = torch.empty(max(h2d_bytes, 1), dtype=torch.uint8).pin_memory()
    di = torch.empty(max(h2d_bytes, 1), dtype=torch.uint8, device=dev)
    ho = torch.empty(max(d2h_bytes, 1), dtype=torch.uint8).pin_memory()
    do = torch.empty(max(d2h_bytes, 1), dtype=torch.uint8, device=dev)
    s1, s2 = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)

    def it():
        with torch.cuda.stream(s1):
            di.copy_(hi, non_blocking=True)
        with torch.cuda.stream(s2):
            ho.copy_(do, non_blocking=True)
    it()
    barrier()
    t0 = time.perf_counter()
    for _ in range(iters):
        it()
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / iters
    del hi, di, ho, do
    return dt


DUMP_POINTS = 1 << 20       # --dump-outputs: sampled points over all ranks (40 bytes each below, so DIR stays well under 64 MB)
DUMP_SEED = 0x7C2D


def dump_outputs(out_dir, frames, rank=0, world=1):
    """Writes the frames a caller of the timed path receives, `frames` = [(positions u16 [n,3], colours u8 [n,3])], as .npy files:
    every frame's point count and column sums over all of its points (float64), and a seeded sample of its points (float32)
    with their (frame, point) indices.  A frame's sample depends on its place in `frames` and its point count only, so two
    builds that agree on the counts sample the same points.  Under several ranks each rank writes rank<R>_*.npy and samples
    its share of DUMP_POINTS."""
    os.makedirs(out_dir, exist_ok=True)
    prefix = f"rank{rank}_" if world > 1 else ""
    per_frame = max(1, DUMP_POINTS // max(1, world) // max(1, len(frames)))
    counts, sums, index, pos, col = [], [], [], [], []
    for j, (p, c) in enumerate(frames):
        n = len(p)
        pick = np.arange(n)
        if n > per_frame:
            pick = np.sort(np.random.default_rng([DUMP_SEED, j]).choice(n, per_frame, replace=False))
        counts.append(n)
        sums.append(np.concatenate([p.sum(0, dtype=np.float64), c.sum(0, dtype=np.float64)]))
        index.append(np.stack([np.full(len(pick), j), pick], 1))
        pos.append(p[pick])
        col.append(c[pick])
    out = {"points_per_frame": np.array(counts, np.float64), "frame_sums": np.array(sums, np.float64).reshape(-1, 6),
           "sample_index": np.concatenate(index).astype(np.float64).reshape(-1, 2),
           "sample_positions": np.concatenate(pos).astype(np.float32).reshape(-1, 3),
           "sample_colors": np.concatenate(col).astype(np.float32).reshape(-1, 3)}
    for name, a in out.items():
        np.save(os.path.join(out_dir, prefix + name + ".npy"), a)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="auto", help="auto (c2 on one GPU, c3s = config 3 strong scaling on several), c1, c2, c3, c3s, c4")
    ap.add_argument("--frames", type=int, default=0, help="frames per GOF (default: the config's)")
    ap.add_argument("--distinct", type=int, default=8, help="distinct synthetic frames cycled inside the GOF")
    ap.add_argument("--ref-threads", type=int, default=1)
    ap.add_argument("--cpu-sample-frames", type=int, default=0, help="frames in the cpu_baseline sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-smoothing", action="store_true", help="reference-exact rec0 path only (no post-processing)")
    ap.add_argument("--resident-gofs", type=int, default=3,
                    help="streams the kernel-only loop spreads its GOFs over (consecutive GOFs of a stream overlap: the small "
                         "latency-bound passes of one run under the emit of the other)")
    ap.add_argument("--quick", action="store_true", help="skip the secondary measurements (pageable e2e, one-context, host ceiling)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the frames the last timed kernel-only step computed to DIR/*.npy "
                                                          "(under several ranks: DIR/rank<R>_*.npy)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to the CUDA path (--impl b200)")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    mode, sname, frames, smoothing, cfg_desc = workload(args, world)
    cfg = synth.config(sname)

    # ------------------------------------------------------------------------------------------------ reference arm
    if args.impl == "reference":
        if rank != 0:
            return 0
        gof, _ = build_workload(sname, frames, min(args.distinct, 4))
        gof.params.geometry_smoothing = smoothing
        gof.params.color_smoothing = smoothing
        sample = max(1, min(frames, 2))                   # frames per step: bounded so K steps end within minutes
        pts, dt = cpu_reference_run(gof, sample, args.steps, args.warmup, args.ref_threads)
        v = pts / dt
        line = {"metric": METRIC, "value": v, "unit": UNIT, "impl": "reference", "n_gpus": args.gpus, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
                "scaling": "strong" if mode == "strong" else "weak",
                "vs_baseline": None, "dtype": "u16", "data": "synthetic", "config": cfg_desc,
                "frames_per_sec": sample * args.steps / dt,
                "cpu_baseline": {"value": v, "unit": UNIT, "cores": args.ref_threads, "kind": "port",
                                 "sample": f"{sample} frames/step x {args.steps} steps of the same workload; C restatement of "
                                           "tmc2-rs src/codec.rs (the Rust reference cannot be built: no cargo/rustc)",
                                 "host_cores": os.cpu_count()},
                "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        # context only: the same port with one worker per host core, frames in parallel (the reference itself reconstructs on
        # one thread, src/lib.rs:113 -- the headline `value` above is that)
        cores = len(os.sched_getaffinity(0))
        if cores > 1 and args.ref_threads <= 1:
            par = min(cores, max(frames, 1))
            pts2, dt2 = cpu_reference_run(gof, par, 2, 1, par)
            line["cpu_baseline"]["frame_parallel"] = {"value": pts2 / dt2, "unit": UNIT, "cores": par,
                                                      "sample": f"{par} frames at once x 2 steps"}
        print(json.dumps(line))
        return 0

    # ------------------------------------------------------------------------------------------------ B200 arm
    import torch
    import torch.distributed as dist
    from tmc2rs_b200 import codec

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the reconstruction path is CUDA-only (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    cpus = bind_to_gpu_numa_node(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # the GOFs this rank reconstructs per step, by size; one pinned copy of the planes per distinct size
    sizes = rank_gofs(mode, frames, rank, world)
    base, _ = build_workload(sname, max(sizes), args.distinct)
    base.params.geometry_smoothing = smoothing
    base.params.color_smoothing = smoothing
    depth = 3                                             # GOFs in flight on the streaming path (keeps both DMA engines busy)
    ctx = codec.Context(devices=(local_rank,), gofs_in_flight=depth)
    pinned, views = {}, {}
    for sz in sorted(set(sizes), reverse=True):
        pinned[sz] = codec.pinned_copy_of(base if sz == base.frame_count else base.subset(range(sz)))
        views[sz] = abi.GofView(pinned[sz])
    frames_per_step_rank = sum(sizes)

    # ---- value: planes resident in HBM, kernels only -----------------------------------------------------------------
    n_res = max(1, args.resident_gofs)
    main_sz = max(sizes)
    residents = {sz: [ctx.upload_gof(views[sz]) for _ in range(n_res if sz == main_sz else 1)] for sz in views}
    # dedicated torch streams: torch.cuda.Event only sees the stream it is recorded on, and torch's default stream
    # has handle 0, which the C ABI reads as "use the library's own stream"
    tstreams = [torch.cuda.Stream(device=dev) for _ in range(n_res)]
    tstream = tstreams[0]
    torch.cuda.set_stream(tstream)
    assert all(t.cuda_stream != 0 for t in tstreams)
    # a kernel-only step repeats the rank's GOF list until it holds at least `inner` GOFs (strong scaling at N = 8 leaves a
    # rank two GOFs of ~1 ms in total: far too short to time)
    inner = max(1, -(-32 // len(sizes))) if mode == "strong" else 1
    # every resident GOF keeps ONE stream for all of its launches (two launches of the same resident on different streams
    # would not be ordered with respect to each other)
    stream_of, nth = {}, 0
    for sz in sorted(residents, reverse=True):
        for r in residents[sz]:
            stream_of[id(r)] = tstreams[nth % n_res]
            nth += 1
    plan = []                                            # (resident, stream) of one kernel-only step
    k = 0
    for _ in range(inner):
        for sz in sizes:
            rs = residents[sz]
            r = rs[k % len(rs)]
            plan.append((r, stream_of[id(r)]))
            k += 1
    for rs in residents.values():                        # every resident once (buffers, tables), then the usual warm-up
        for r in rs:
            r.reconstruct(stream_of[id(r)].cuda_stream)
    for _ in range(max(1, min(args.warmup, 3))):
        for r, t in plan[:3 * n_res]:
            r.reconstruct(t.cuda_stream)
    points_by_size = {sz: int(residents[sz][0].counts().sum()) for sz in views}
    points_per_step = sum(points_by_size[sz] for sz in sizes)            # this rank, one pass
    residents[main_sz][0].reconstruct(tstream.cuda_stream, timed=True)
    launches_per_gof, alg_bytes, _ = ctx.last_launch_info()
    sampler = ClockSampler(local_rank)
    barrier()
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(tstream)
    for t in tstreams[1:]:
        t.wait_event(e0)
    for i in range(args.steps):
        for r, t in plan:
            r.reconstruct(t.cuda_stream)
    for t in tstreams[1:]:
        done = torch.cuda.Event()
        done.record(t)
        tstream.wait_event(done)
    e1.record(tstream)
    barrier()
    kernel_ms = e0.elapsed_time(e1) / inner               # per pass over the rank's GOF list
    if args.dump_outputs:
        # every resident of the plan was last launched in the last timed step: read them before anything relaunches one
        last = list(dict.fromkeys(r for r, _ in plan))
        sampler.paused = True                              # the clocks block covers the timed regions only
        dump_outputs(args.dump_outputs, [r.fetch(f, int(n)) for r in last for f, n in enumerate(r.counts())], rank, world)
        sampler.paused = False
    # per-stage device times (library-recorded CUDA events on the same stream), measured on separate launches so that
    # reading them does not serialise the timed loop above
    unpack_ms, stage_acc = [], {}
    for _ in range(5):
        residents[main_sz][0].reconstruct(tstream.cuda_stream, timed=True)
        st = ctx.last_stage_ms()
        unpack_ms.append(st["unpack"])
        for kk, v in st.items():
            stage_acc.setdefault(kk, []).append(v)
    kernel_ms_max, pts_all, frames_all = shard.reduce_metrics(kernel_ms, points_per_step * args.steps,
                                                              frames_per_step_rank * args.steps, dev)
    value = pts_all / (kernel_ms_max * 1e-3)
    for rs in residents.values():
        for r in rs:
            r.free()

    # ---- e2e: public C ABI, pinned host planes in, pinned host frames out, three GOFs in flight ---------------------------
    def e2e_run(c, vws, gof_sizes, steps, warm):
        return e2e_loop(c, vws, gof_sizes, steps, warm, depth, barrier)

    e2e_sizes = sizes if mode == "strong" else sizes[:max(1, min(len(sizes), 8))]   # N = 1: 8 GOFs per e2e step (same rate, shorter run)
    e2e_scale = len(sizes) / len(e2e_sizes)
    warm_e2e = max(1, -(-(depth + 1) // len(e2e_sizes)))
    dt_e2e, got_all = e2e_run(ctx, views, e2e_sizes, args.steps, warm_e2e)
    pts_e2e_step = sum(points_by_size[sz] for sz in e2e_sizes)
    clocks = sampler.stop()            # sampled over both timed regions (kernel-only steps and the end-to-end steps)
    barrier()
    e2e_ms_max, e2e_pts, e2e_frames = shard.reduce_metrics(dt_e2e * 1e3, pts_e2e_step * args.steps, sum(e2e_sizes) * args.steps, dev)
    e2e_value = e2e_pts / (e2e_ms_max * 1e-3)
    h2d = int(sum(pinned[sz].input_bytes() for sz in e2e_sizes) * e2e_scale)
    d2h = int(pts_e2e_step * 9 * e2e_scale)
    e2e = {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
           "frames_per_sec": e2e_frames / (e2e_ms_max * 1e-3), "ms_per_step": e2e_ms_max / args.steps * e2e_scale,
           "gofs_in_flight": depth, "input_memory": "pinned (tmc2gpu_alloc_pinned)"}
    extra = {}
    if not args.quick:
        # the same bytes as bare pinned copies, every rank at once: the ceiling the host side of this box puts on e2e
        dt_copy = host_copy_ceiling(torch, dev, int(h2d / e2e_scale), int(d2h / e2e_scale), 5, barrier)
        copy_ms_max, _, _ = shard.reduce_metrics(dt_copy * 1e3, 0, 0, dev)
        ceiling = e2e_pts / args.steps / (copy_ms_max * 1e-3)
        e2e["host_ceiling"] = {"value": ceiling, "unit": UNIT, "ms_per_step": copy_ms_max * e2e_scale,
                               "what": "the step's H2D + D2H bytes as bare pinned cudaMemcpyAsync on two streams, all ranks at once",
                               "aggregate_GBps": (h2d + d2h) / e2e_scale * world / (copy_ms_max * 1e-3) / 1e9}
        e2e["frac_of_host_ceiling"] = e2e_value / ceiling
        if world == 1:
            # planes in ordinary memory, like the reference's Vec<u8> (src/decoder.rs:1136-1140): staged by the library
            pageable = {sz: abi.GofView(base if sz == base.frame_count else base.subset(range(sz))) for sz in set(e2e_sizes)}
            dt_p, got_p = e2e_run(ctx, pageable, e2e_sizes, max(2, args.steps // 2), warm_e2e)
            extra["e2e_pageable"] = {"value": pts_e2e_step * max(2, args.steps // 2) / dt_p, "unit": UNIT,
                                     "frames_per_sec": sum(e2e_sizes) * max(2, args.steps // 2) / dt_p,
                                     "input_memory": "pageable numpy arrays, staged by the library's thread pool",
                                     "stage_threads": os.environ.get("TMC2_STAGE_THREADS", "default")}
    ctx.close()
    if world > 1 and not args.quick:
        # ONE context over all N devices, driven by rank 0 alone (the other ranks wait): the topology behind the unchanged
        # Decoder API -- tmc2gpu_create(ids, N), frames of every GOF sharded inside the library, handed back in order
        barrier()
        if rank == 0:
            full, _ = build_workload(sname, SEQ_GOF, args.distinct)
            full.params.geometry_smoothing = smoothing
            full.params.color_smoothing = smoothing
            pfull = codec.pinned_copy_of(full)
            vfull = {SEQ_GOF: abi.GofView(pfull)}
            octx = codec.Context(devices=tuple(range(world)), gofs_in_flight=depth)
            try:
                seq = [SEQ_GOF] * (SEQ_FRAMES // SEQ_GOF)
                dt_o, got_o = e2e_loop(octx, vfull, seq, max(2, args.steps // 2), 1, depth)
                extra["one_context"] = {"value": got_o / dt_o, "unit": UNIT, "devices": world,
                                        "frames_per_sec": SEQ_FRAMES * max(2, args.steps // 2) / dt_o,
                                        "what": "e2e through ONE tmc2gpu context over all devices, one host thread, frames in order"}
            finally:
                octx.close()
        barrier()

    # ---- roofline of the dominant kernel -------------------------------------------------------------------------------
    peak, peak_src = measured_peak()
    t_unpack = statistics.mean(unpack_ms) if unpack_ms else float("nan")
    # the emit kernel is launched once per smoothing frame group (the whole GOF unless the tables do not fit); algorithmic bytes
    # and device time are per launch (SURVEY.md 8d figure x the frames one launch processes)
    group = int(os.environ.get("TMC2_SMOOTH_GROUP", "32")) if smoothing else main_sz
    n_emit = max(1, -(-main_sz // max(group, 1)))
    achieved = alg_bytes / (t_unpack * 1e-3) / 1e9 if t_unpack and t_unpack > 0 else 0.0
    roofline = {"bound": "hbm", "kernel": "emit_kernel (fused occupancy upsample / unpack / attribute fetch / YUV->RGB; + boundary + cell statistics when smoothing)",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "peak_source": peak_src,
                "frac_of_nominal_8TBps": achieved / 8000.0,
                "launches_per_gof": n_emit, "frames_per_launch": min(group, main_sz),
                "algorithmic_bytes_per_launch": alg_bytes / n_emit, "ms_per_launch": t_unpack / n_emit, "traffic": None,
                "stage_ms": {kk: statistics.mean(v) for kk, v in stage_acc.items()}}
    # the other HBM-streaming kernel of the path: the count pass reads the occupancy video and both geometry planes once
    # (its stage time also holds the tiny per-frame scan launch, so the fraction is a lower bound)
    t_count = statistics.mean(stage_acc.get("count_scan", [0.0])) if stage_acc else 0.0
    count_bytes = main_sz * (cfg.width // cfg.occupancy_precision) * (cfg.height // cfg.occupancy_precision) + main_sz * 2 * cfg.width * cfg.height * 2
    if t_count > 0:
        roofline["other_kernels"] = {"count_kernel+slot_scan_kernel": {
            "algorithmic_bytes_per_launch": count_bytes, "ms_per_launch": t_count,
            "achieved": count_bytes / (t_count * 1e-3) / 1e9, "frac": count_bytes / (t_count * 1e-3) / 1e9 / peak}}
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            roofline["traffic"] = json.load(f).get(sname + ("" if smoothing else "_nosmooth"))
    except Exception:
        pass

    gofs_per_step_all = len(sizes) if mode == "weak" else SEQ_FRAMES // SEQ_GOF
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": kernel_ms_max / args.steps, "higher_is_better": True,
            "scaling": "strong" if mode == "strong" else "weak", "vs_baseline": None,
            "dtype": "u16", "data": "synthetic", "config": cfg_desc,
            "frames_per_sec": frames_all / (kernel_ms_max * 1e-3), "points_per_step_rank0": points_per_step,
            "e2e": e2e,
            "gpu_launches": launches_per_gof * len(sizes) * inner * args.steps, "gpu_launches_per_gof": launches_per_gof,
            "roofline": roofline, "clocks": clocks,
            "timing": {"kernel_only_passes_per_step": inner, "resident_streams": n_res,
                       "e2e_gofs_per_step_rank0": len(e2e_sizes), "timed_kernel_region_ms": kernel_ms_max * inner,
                       "host_cpus_of_rank0": (f"{cpus[0]}-{cpus[-1]} ({len(cpus)})" if cpus else "inherited")}}
    line.update(extra)

    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        # ~10-20 s of single-threaded CPU work: 64 frames (two passes over the GOF) with smoothing, 128 without
        sample = args.cpu_sample_frames or ((64 if smoothing else 128) if frames > 1 else 16)
        if frames > 1:
            per, reps = min(sample, frames), max(1, sample // min(sample, frames))
        else:
            per, reps = 1, sample
        sample = per * reps
        pts, dt = cpu_reference_run(base, per, reps, 0, 1)
        line["cpu_baseline"] = {"value": pts / dt, "unit": UNIT, "cores": 1, "kind": "port",
                                "sample": f"{sample} frame(s) of the same workload, {dt:.1f} s; single-threaded C restatement "
                                          "of tmc2-rs src/codec.rs (+ this repo's smoothing spec) -- the Rust reference "
                                          "cannot be built in this image",
                                "host_cores": os.cpu_count(), "ms_per_frame": dt / sample * 1e3}
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


def e2e_loop(c, vws, gof_sizes, steps, warm, depth, barrier=None):
    """`warm` untimed + `steps` timed passes over `gof_sizes` through submit_gof / next_frame with `depth` GOFs in flight (the
    warm-up GOFs are drained before the clock starts).  Returns (seconds, points of the timed passes)."""
    # warm-up: first `depth` GOFs of the largest size, so that every GOF slot of the context has its device buffers, cell tables
    # and pinned result slab sized for the largest GOF before the clock starts; then `warm` ordinary passes
    head = [max(gof_sizes)] * depth
    seq = head + [sz for _ in range(warm + steps) for sz in gof_sizes]
    n_warm = len(head) + warm * len(gof_sizes)
    got, t0, pending = 0, None, []
    for i, sz in enumerate(seq):
        if i == n_warm:
            while pending:
                for _ in range(pending.pop(0)):
                    c.next_frame_raw()
            if barrier:
                barrier()
            t0 = time.perf_counter()
        c.submit_gof(vws[sz])
        pending.append(sz)
        if len(pending) >= depth:
            for _ in range(pending.pop(0)):
                n = c.next_frame_raw()[0]
                if i >= n_warm:
                    got += n
    while pending:
        for _ in range(pending.pop(0)):
            got += c.next_frame_raw()[0]
    return time.perf_counter() - t0, got


if __name__ == "__main__":
    sys.exit(main())
