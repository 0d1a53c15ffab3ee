#!/usr/bin/env python
"""End-to-end rate of a BASELINE config-2 GOF (32 frames of 1024x1024, smoothing on) by where its planes come from, and the
time of the kernel that gathers device-resident planes (ingest_planes_kernel).  One GPU, three GOFs in flight.

  host_pinned     planes in tmc2gpu_alloc_pinned memory, frames copied back to pinned host memory (bench.py's `e2e`)
  device_planar   planes in HBM (torch tensors, TMC2_INPUT_DEVICE), frames left in HBM (TMC2_CTX_DEVICE_OUTPUT)
  device_p010     the same with the planes in NVDEC's P010 layout (TMC2_INPUT_P010)
  ingest_kernel   torch.profiler (CUDA activities, a pass of its own): kernel time, bytes read + written over it, against the
                  project's measured HBM copy peak

The frames of one GOF of each device leg are compared with the host leg's (counts and full arrays).

    python tools/device_input_bench.py [--seconds 0.3] [--trace-dir DIR]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tmc2rs_b200 import abi, codec, synth  # noqa: E402

IN_FLIGHT = 3
HBM_COPY_PEAK_GBS = 6500.0      # device-to-device copy rate the project measured on B200 (README, DESIGN section 4)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception as e:                                  # the numbers still stand, without the card's description
        return f"nvidia-smi unavailable ({e})"


def plane_bytes(g):
    """Bytes of samples the ingest kernel reads for one GOF (it writes as many)."""
    F, H, W = g.frame_count, g.height, g.width
    n = F * g.occ.shape[1] * g.occ.shape[2] + F * 2 * H * W * 2
    if g.attr_y is not None:
        n += F * 2 * (H * W + 2 * (H // 2) * (W // 2)) * 2
    return n


def drain_host(ctx, frames):
    for _ in range(frames):
        ctx.next_frame_raw()


def drain_device(ctx, frames):
    fo = abi.CFrameOut()
    for _ in range(frames):
        ctx.check(ctx.lib.tmc2gpu_next_frame(ctx.h, C.byref(fo)), "next_frame")
        ctx.check(ctx.lib.tmc2gpu_release_frame(ctx.h, C.byref(fo)), "release_frame")


def timed(ctx, view, drain, frames, seconds, warmup=3):
    """GOFs per second with IN_FLIGHT GOFs submitted ahead of the one being drained."""
    for _ in range(warmup):
        ctx.submit_gof(view)
        drain(ctx, frames)
    in_flight, done = 0, 0
    t0 = time.perf_counter()
    while True:
        while in_flight < IN_FLIGHT:
            ctx.submit_gof(view)
            in_flight += 1
        drain(ctx, frames)
        in_flight -= 1
        done += 1
        el = time.perf_counter() - t0
        if el >= seconds and done >= 2 * IN_FLIGHT:
            break
    for _ in range(in_flight):
        drain(ctx, frames)
    return done / el, el, done


def device_frames(ctx, view, frames):
    """The frames of one GOF of a device-output context, copied to numpy."""
    import torch

    class Raw:
        def __init__(self, ptr, n):
            self.__cuda_array_interface__ = {"shape": (n,), "typestr": "|u1", "data": (ptr, False), "version": 2}
    ctx.submit_gof(view)
    out = []
    for _ in range(frames):
        n, pp, pc, dev, release = ctx.next_frame_device()
        pos = torch.as_tensor(Raw(pp, n * 6), device=f"cuda:{dev}").cpu().numpy().view(np.uint16).reshape(n, 3) if n else np.zeros((0, 3), np.uint16)
        col = torch.as_tensor(Raw(pc, n * 3), device=f"cuda:{dev}").cpu().numpy().reshape(n, 3) if n else np.zeros((0, 3), np.uint8)
        out.append((pos, col))
        release()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=0.3, help="least length of every timed window")
    ap.add_argument("--distinct", type=int, default=8, help="distinct synthetic frames cycled inside the GOF (as bench.py)")
    ap.add_argument("--trace-dir", help="also write the profiler traces of the ingest pass there")
    args = ap.parse_args()
    import torch
    from torch.profiler import ProfilerActivity, profile

    base = synth.make_gof(synth.config("c2", frames=args.distinct))
    g = synth.replicate_gof(base, 32)
    g.params = base.params
    F = g.frame_count
    res = {"card": card(), "workload": f"c2: {F}-frame GOF of {g.width}x{g.height}, smoothing on, {IN_FLIGHT} GOFs in flight"}

    # leg 1: pinned host planes, host frames
    hv = abi.GofView(codec.pinned_copy_of(g))
    hctx = codec.Context(gofs_in_flight=IN_FLIGHT)
    ref = hctx.decode_gof(hv)
    points = sum(len(f) for f in ref)
    res["points_per_gof"] = points
    # legs 2 and 3: device planes, device frames
    dctx = codec.Context(gofs_in_flight=IN_FLIGHT, device_output=True)
    views = {"device_planar": abi.GofView(synth.to_device(g, "cuda:0")),
             "device_p010": abi.GofView(synth.to_device(g, "cuda:0", p010=True, seed=1))}
    check = {}
    for name, v in views.items():
        got = device_frames(dctx, v, F)
        check[name] = all(len(p) == len(r) and np.array_equal(p, r.positions) and np.array_equal(c, r.colors)
                          for (p, c), r in zip(got, ref))
    res["frames_equal_host_leg"] = check

    legs = [("host_pinned", hctx, hv, drain_host)] + [(n, dctx, v, drain_device) for n, v in views.items()]
    for rnd in range(2):                                    # two rounds, legs alternating: the spread shows in the numbers
        for name, ctx, v, drain in legs:
            rate, el, done = timed(ctx, v, drain, F, args.seconds)
            res.setdefault(name, []).append({"gofs_per_s": round(rate, 1), "gpoints_per_s": round(rate * points / 1e9, 3),
                                             "window_s": round(el, 3), "gofs": done})

    # leg 4: the ingest kernel alone, from the profiler
    nbytes = plane_bytes(g)
    res["ingest_kernel"] = {}
    for name, v in views.items():
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(6):
                dctx.submit_gof(v)
                drain_device(dctx, F)
            torch.cuda.synchronize()
        us = [e.device_time_total for e in prof.events() if "ingest_planes_kernel" in e.name]
        if not us:
            raise RuntimeError("ingest_planes_kernel not found in the profile")
        us = sorted(us)[1:-1] if len(us) > 3 else us
        ms = float(np.mean(us)) / 1e3
        gbs = 2 * nbytes / (ms * 1e-3) / 1e9
        res["ingest_kernel"][name] = {"ms": round(ms, 4), "kernels": len(us), "bytes_read_plus_written": 2 * nbytes,
                                      "gb_per_s": round(gbs, 1), "share_of_copy_peak": round(gbs / HBM_COPY_PEAK_GBS, 3)}
        if args.trace_dir:
            os.makedirs(args.trace_dir, exist_ok=True)
            prof.export_chrome_trace(os.path.join(args.trace_dir, f"device_input_{name}.pt.trace.json"))
    hctx.close()
    dctx.close()
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
