"""Every generator case through every emit instantiation that produces frames for users.

`launch_emit` (kernels.cu) picks one of five `emit_kernel<smooth, debug, fast>` instantiations, each with and without
attributes, and inside each one a slot takes one of three paths: the TMA path with the occupancy box (resolution 16,
precision 4), the TMA path reading the occupancy video (`occupancy_mask`, other powers of two) or the per-pixel
`generic_slot_emit` (other resolutions and precisions, reference-mode rotations that are not block-aligned).  The stage API
with its debug streams always runs the debug instantiation; these tests run the instantiations behind `submit_gof` /
`next_frame`, the resident path, device-output contexts and the stage API without debug streams, on the same cases:

  off            no smoothing: the plain instantiation
  g8c4           dense power-of-two grids, geometry edge <= 8: the fast smoothing instantiation
  g6c3, g16c8    a cell edge that is not a power of two, and a geometry edge of 16: the generic smoothing instantiation
  hashed         hashed cell tables (TMC2_FORCE_HASH): the generic smoothing instantiation

A CPU test mirrors the selection rules and checks that the cases reach every (instantiation, slot path, attributes) cell;
the GPU tests check the instantiation a launch actually ran against that mirror.
"""
import ctypes as C
import re

import numpy as np
import pytest

import util
from oracle import oracle
from tmc2rs_b200 import abi

ALL_CASES = util.CASES + util.FAST_CASES
MODES = {"off": None, "g8c4": (8, 4), "g6c3": (6, 3), "g16c8": (16, 8), "hashed": (8, 4)}
FRAMES = 3


def make_gof(case, mode):
    """The case with three frames (each its own patch list); smoothing modes crowd the patches into one 3D region and use
    low thresholds so that the filters have work."""
    g = util.random_small_gof(frames=FRAMES, **case)
    if MODES[mode] is not None:
        util.crowd_into_one_region(g)
        g.params.geometry_smoothing = True
        g.params.color_smoothing = True
        g.params.grid_size, g.params.cgrid_size = MODES[mode]
        g.params.threshold_smoothing = 4
        g.params.threshold_color_smoothing = 2
        g.params.threshold_color_variation = 200
        g.params.threshold_color_difference = 200
    return g


# ---- the selection rules, mirrored ------------------------------------------------------------------------------------
def _pow2(x):
    return x > 0 and x & (x - 1) == 0


def grid_fast(params, g, hashed):
    """GridDesc.fast of a grid of edge g (tmc2gpu.cu make_args): 0 generic grid, 1 packed 8-bit cell keys, 2 wider."""
    w = -(-(1 << params.geometry_bitdepth_3d) // g)
    if hashed or not (_pow2(g) and _pow2(w) and w <= 1024 and g * w <= 65536):
        return 0
    return 1 if w <= 256 else 2


def emit_instantiation(params, hashed):
    """launch_emit for a launch without debug streams (tmc2gpu.cu fills the GridDesc `fast` field that it reads)."""
    geo = bool(params.geometry_smoothing)
    col = bool(params.color_smoothing) and params.attribute_count != 0
    if not (geo or col):
        return "plain"
    fast = (not geo or (grid_fast(params, params.grid_size, hashed) == 1 and params.grid_size <= 8)) and \
           (not col or grid_fast(params, params.cgrid_size, hashed) != 0)
    return "fast" if fast else "generic"


def slot_path(params, width, height, orientation):
    """slot_is_fast / occ_by_tma (kernels.cu), with the block-alignment rule that tmc2gpu.cu applies to the slot's
    affine steps (DevPatch.aligned)."""
    aligned = params.orientation_mode == abi.ORIENTATION_SPEC or orientation <= 1 or orientation == 8
    prec = params.occupancy_precision
    if params.occupancy_resolution != 16 or not _pow2(prec) or not aligned:
        return "generic-slot"
    return "tma-box" if prec == 4 and width % 4 == 0 and height % 4 == 0 else "tma-mask"


def emitting_slots(g):
    """(frame, patch, slot path) of every slot that emits points: owned by its patch and with an occupied pixel."""
    view = abi.GofView(g)
    res = g.params.occupancy_resolution
    bw = g.width // res
    out = []
    for f in range(g.frame_count):
        b2p = oracle.block_to_patch(view, f)
        for i, p in enumerate(g.patches[f]):
            path = slot_path(g.params, g.width, g.height, int(p["patch_orientation"]))
            owned = any(b2p[by * bw + bx] == i + 1
                        for v0b in range(int(p["size_v0"])) for u0b in range(int(p["size_u0"]))
                        for bx, by in [util._helper(p, u0b, v0b, 1, 1)])
            if owned:
                out.append((f, p, path))
    return out


def cells_of(case, mode):
    g = make_gof(case, mode)
    inst = emit_instantiation(g.params, mode == "hashed")
    attr = "attr" if g.params.attribute_count else "no-attr"
    cells = set()
    for _, p, path in emitting_slots(g):
        cells.add((inst, path, attr))
        if path == "generic-slot" and p["lod_x"] != p["lod_y"]:
            cells.add((inst, path, "lod_x != lod_y"))
    return cells


def test_cases_reach_every_instantiation_and_slot_path():
    """Each of {plain, fast, generic} x {TMA + occupancy box, TMA + occupancy_mask, generic slot} x {attributes, none} is
    reached by some case, and so is a generic slot of the plain instantiation whose patch scales u and v differently
    (level of detail 2 on one axis only).  Fails when an edit of the case lists drops the only case of a cell."""
    reached = set()
    for case in ALL_CASES:
        for mode in MODES:
            reached |= cells_of(case, mode)
    want = {(i, s, a) for i in ("plain", "fast", "generic") for s in ("tma-box", "tma-mask", "generic-slot")
            for a in ("attr", "no-attr")}
    want.add(("plain", "generic-slot", "lod_x != lod_y"))
    assert not want - reached, f"cells no case reaches: {sorted(want - reached)}"


def test_mode_selection_rules():
    """The modes select what their names say (the GPU tests also read the instantiation off the launch)."""
    g = util.random_small_gof(seed=1)
    assert emit_instantiation(g.params, False) == "plain"
    for mode, want in (("g8c4", "fast"), ("g6c3", "generic"), ("g16c8", "generic"), ("hashed", "generic")):
        assert emit_instantiation(make_gof(util.CASES[0], mode).params, mode == "hashed") == want, mode


# ---- GPU ------------------------------------------------------------------------------------------------------------
def _expect(got_n, pos, col, want, what, smoothed=None):
    assert got_n == want["point_count"], f"{what}: point count {got_n} != {want['point_count']}"
    assert np.array_equal(pos, want["positions"]), f"{what}: positions"
    if want["with_colors"]:
        assert np.array_equal(col, want["colors"]), f"{what}: colours"
    if smoothed is not None:
        assert smoothed == (want["smoothed_positions"], want["smoothed_colors"]), f"{what}: smoothed counts"


def _cuda_kernels(fn):
    """Names of the CUDA kernels that ran while fn() did (fn must synchronise the device)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
    return sorted(e.name for e in prof.events() if "kernel" in e.name)


def _emit_of(names):
    """(instantiation, attributes) of the emit kernels in a launch."""
    found = set()
    for n in names:
        m = re.search(r"emit_kernel<(\w+), (\w+), (\w+), (\w+)>", n)
        if m:
            smooth, debug, fast, attr = (x == "true" for x in m.groups())
            assert not debug, n
            found.add(("plain" if not smooth else "fast" if fast else "generic", attr))
    return found


@pytest.fixture(scope="module")
def device_ctx():
    from tmc2rs_b200 import codec
    ctx = codec.Context(device_output=True)
    yield ctx
    ctx.close()


def _device_frames(ctx, view):
    import torch

    class Dev:                                             # zero-copy torch view of a raw device range
        def __init__(self, ptr, nbytes):
            self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 2}
    ctx.submit_gof(view)
    got = [ctx.next_frame_device() for _ in range(view.c.frame_count)]
    assert ctx.next_frame_device() is None
    out = []
    for n, ppos, pcol, dev, _ in got:
        pos = np.zeros((0, 3), np.uint16)
        col = None
        if n:
            pos = torch.as_tensor(Dev(ppos, n * 6), device=f"cuda:{dev}").cpu().numpy().view(np.uint16).reshape(n, 3)
            if pcol:
                col = torch.as_tensor(Dev(pcol, n * 3), device=f"cuda:{dev}").cpu().numpy().reshape(n, 3)
        out.append((n, pos, col))
    for *_, release in got:
        release()
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("case", ALL_CASES, ids=util.case_id)
def test_production_instantiations_match_oracle(gpu_ctx, device_ctx, monkeypatch, case, mode):
    from tmc2rs_b200 import codec
    g = make_gof(case, mode)
    view = abi.GofView(g)
    want = [oracle.reconstruct_frame(view, f) for f in range(FRAMES)]
    inst = emit_instantiation(g.params, mode == "hashed")
    attr = g.params.attribute_count != 0
    ctx = gpu_ctx
    if mode == "hashed":
        monkeypatch.setenv("TMC2_FORCE_HASH", "1")
        ctx = codec.Context()
    try:
        # stage API without debug streams
        for f in range(FRAMES):
            st = ctx.generate_point_cloud(view, f, debug=False)
            _expect(st["point_count"], st["positions"], st["colors"], want[f], f"{mode} stage frame {f}",
                    (st["smoothed_positions"], st["smoothed_colors"]))
        # streaming
        for f, fr in enumerate(ctx.decode_gof(view)):
            assert fr.with_colors == attr
            _expect(len(fr), fr.positions, fr.colors, want[f], f"{mode} streaming frame {f}",
                    (fr.smoothed_positions, fr.smoothed_colors))
        # resident: the first launch runs directly; without smoothing the second is captured into a CUDA graph (and runs
        # nothing) and the third replays it
        r = ctx.upload_gof(view)
        try:
            def fetch_all(what):
                counts = r.counts()
                for f in range(FRAMES):
                    pos, col = r.fetch(f, int(counts[f]))
                    _expect(int(counts[f]), pos, col, want[f], f"{mode} resident {what} frame {f}")
            first = _cuda_kernels(lambda: (r.reconstruct(), r.counts()))
            assert _emit_of(first) == {(inst, attr)}, first
            fetch_all("first launch")
            r.reconstruct()
            replay = _cuda_kernels(lambda: (r.reconstruct(), r.counts()))
            fetch_all("third launch")
            if mode == "off":
                timed = _cuda_kernels(lambda: (r.reconstruct(timed=True), r.counts()))
                assert replay == timed, (replay, timed)
                for k in ("count_kernel", "slot_scan_kernel", "emit_kernel"):
                    assert any(k in n for n in replay), (k, replay)
        finally:
            r.free()
    finally:
        if ctx is not gpu_ctx:
            ctx.close()
    if mode in ("off", "g8c4"):
        for f, (n, pos, col) in enumerate(_device_frames(device_ctx, view)):
            _expect(n, pos, col, want[f], f"{mode} device output frame {f}")
