"""What one launch leaves behind for the next: a batch decodes GOF after GOF, and its cell tables, keys and bitmaps are only
re-zeroed when their layout changes (Batch::prepare); otherwise every launch relies on the previous one's clear pass.  The
same GOF decoded twice cannot show a colour table that was never cleared (every colour decision is unchanged when all the
cell statistics double), so the sequences here give one batch different GOFs in a row.

CPU part: a mirror of the table decisions of Batch::prepare / launch shows that the sequences reach every kind of table
hand-over (reuse, re-layout, reset, groups, idle tables, failures), and names, for every frame of every batch the GPU tests
drive, the earlier frame that last wrote its table frame of each kind without a reset in between.  The leftover-statistics
model (smoothmodel.smooth(prior=...)) shows that each such frame would decode differently on a table that was not cleared.
GPU part: every GOF of every sequence equals the oracle, streamed through one GOF slot, through the stage API, and with
three slots in flight.
"""
import functools
import os

import numpy as np
import pytest

import tmc2rs_b200  # noqa: F401
from tmc2rs_b200 import abi, codec, synth
from oracle import oracle

import smoothmodel
import util
from test_smoothing_limits import c_atlas

BUDGET_MB = "1024"      # per cell table: a grid of 32-byte cells is dense up to 2^25 cells


# ---- the GOFs ------------------------------------------------------------------------------------------------------------
def crowded(seed=1, frames=2, bitdepth=10, grid=8, cgrid=8, W=128, H=64):
    """Patches crowded into one region (many multi-patch cells); grid / cgrid None = that smoothing off.  At bit depth 11
    the region sits at twice the coordinates, so that its cells of edge 16 have the coordinates of the bit-depth-10
    region's cells of edge 8 (a leftover cell lands on a cell of this GOF)."""
    g = util.random_small_gof(seed, W=W, H=H, frames=frames, n_patches=6)
    util.crowd_into_one_region(g)
    vary_colours(g, seed)
    if bitdepth == 11:
        for p in g.patches:
            p["u1"] += 100
            p["v1"] += 100
            p["d1"] = np.where(p["projection_mode"] == 0, 224, 1214)
    P = g.params
    P.geometry_bitdepth_3d = bitdepth
    P.geometry_smoothing, P.color_smoothing = grid is not None, cgrid is not None
    P.grid_size, P.cgrid_size = grid or 8, cgrid or 4
    return g


def vary_colours(g, seed):
    """crowd_into_one_region gives every GOF and every frame the same colours; offset them per GOF and per frame, so that
    what one frame leaves in a colour table differs from what the next frame puts there."""
    for f in range(g.frame_count):
        g.attr_y[f] += (53 * seed + 97 * f) % 300
        g.attr_u[f] += (29 * seed + 41 * f) % 200
        g.attr_v[f] -= (31 * seed + 43 * f) % 200


def inverted_colours(g):
    """Same geometry, colours mirrored: a leftover colour table changes the blend of many points."""
    for a in (g.attr_y, g.attr_u, g.attr_v):
        a[...] = 1023 - a
    return g


def shifted_depth(g, units=3):
    g.geo[...] += 4 * units
    return g


def saturated(W=256, H=160, frames=2):
    """Every plane at its maximum: occupancy 1 everywhere, geometry and attribute samples 65535.  Every row of every plane is
    as wide as its pitch (no padding of its own), so whatever a later, smaller GOF finds in the padding of its rows was
    written here."""
    g = util.random_small_gof(31, W=W, H=H, frames=frames, n_patches=12)
    g.occ[...] = 1
    g.geo[...] = 65535
    for a in (g.attr_y, g.attr_u, g.attr_v):
        a[...] = 65535
    return g


def edge_reaching(W=208, H=112, frames=2):
    """W not a multiple of 64, an occupancy video 52 samples wide (not a multiple of 16), and patches over the last block
    column and the last block row, fully occupied there: points at x = W - 1 and y = H - 1."""
    g = util.random_small_gof(32, W=W, H=H, frames=frames, n_patches=8)
    bw, bh = W // 16, H // 16
    n, t, b, mode = synth.VIEW_AXES[0]
    extra = [(bw - 2, 0, 2, bh, 100, 200, 64, 1, 1, n, t, b, mode, 0, 0, (0, 0)),
             (0, bh - 2, bw - 2, 2, 300, 50, 64, 1, 1, n, t, b, mode, 0, 0, (0, 0))]
    g.patches = [np.concatenate([p, np.array(extra, dtype=abi.PATCH_DTYPE)]) for p in g.patches]
    g.occ[:, -8:, :] = 1
    g.occ[:, :, -8:] = 1
    return g


# name -> builder; every GOF is built once per session (the oracle frames are cached with it)
GOFS = {
    "A": lambda: crowded(),
    "A-inv": lambda: inverted_colours(crowded()),
    "A-shift": lambda: shifted_depth(crowded()),
    "B11": lambda: crowded(seed=2, bitdepth=11, grid=16, cgrid=16),           # both grids 128 cells wide, as in "A"
    "B11-5f": lambda: crowded(seed=3, frames=5, bitdepth=11, grid=16, cgrid=16),
    "B11-shift": lambda: shifted_depth(crowded(seed=2, bitdepth=11, grid=16, cgrid=16), 2),
    "B11-inv": lambda: inverted_colours(crowded(seed=2, bitdepth=11, grid=16, cgrid=16)),
    "off": lambda: crowded(seed=4, grid=None, cgrid=None),
    "B11-geo": lambda: crowded(seed=5, bitdepth=11, grid=16, cgrid=None),
    "B11-col": lambda: crowded(seed=6, bitdepth=11, grid=None, cgrid=16),
    "A-c2": lambda: crowded(seed=7, cgrid=2),                                   # colour grid of 2^27 cells: hashed
    "B11-c4": lambda: crowded(seed=8, bitdepth=11, grid=16, cgrid=4),           # hashed (2^27 cells), another grid
    "A-c8": lambda: inverted_colours(crowded(seed=8)),
    "cell-65537": lambda: c_atlas(65537, "uv"),                                 # fails in the emit (status 6)
    "cell-65536": lambda: c_atlas(65536, "uv"),                                 # the same cells, at the limit
    "small3": lambda: _small3(),
    "sat": lambda: saturated(),
    "edge": lambda: edge_reaching(),
}


def _small3():
    g = synth.make_gof(synth.config("small", frames=3))
    util.crowd_into_one_region(g)
    vary_colours(g, 9)
    g.params.geometry_smoothing = g.params.color_smoothing = True
    return g


@functools.lru_cache(maxsize=None)
def gof(name):
    return GOFS[name]()


@functools.lru_cache(maxsize=None)
def oracle_frames(name):
    view = abi.GofView(gof(name))
    return [oracle.reconstruct_frame(view, f) for f in range(gof(name).frame_count)]


# ---- the sequences: (env of the context, [(GOF, env of that step only, fails)]) ------------------------------------------
def step(name, env=None, fails=False):
    return (name, env or {}, fails)


SEQUENCES = {
    "S1-colour-leak": ({"TMC2_TABLE_BUDGET_MB": BUDGET_MB}, [step("A"), step("A-inv"), step("A")]),
    "S2-geometry-leak": ({"TMC2_TABLE_BUDGET_MB": BUDGET_MB}, [step("A"), step("A-shift")]),
    "S3-layouts": ({"TMC2_TABLE_BUDGET_MB": BUDGET_MB, "TMC2_SMOOTH_GROUP": "2"}, [
        step("A"), step("A-inv"),           # identical layout
        step("B11"),                        # other grids, same slot count: no reset
        step("B11-5f"),                     # three groups over two table sets (TF grows: reset)
        step("B11-shift"),                  # one group again, TF shrinks: no reset
        step("off"),                        # no smoothing: the clear of B11-shift stays pending ...
        step("B11-inv"),                    # ... until this launch
        step("B11-geo"), step("B11-col"), step("B11"),     # one table idle, then reused
        step("A-c2"),                       # colour dense -> hashed: reset
        step("B11-c4"),                     # hashed -> hashed, other grid: no reset
        step("A-c8"),                       # hashed -> dense: reset
    ]),
    "S4-failure-one-group": ({"TMC2_TABLE_BUDGET_MB": BUDGET_MB}, [
        step("cell-65536"), step("cell-65537", fails=True), step("cell-65536")]),
    "S4-failure-groups": ({"TMC2_TABLE_BUDGET_MB": BUDGET_MB, "TMC2_SMOOTH_GROUP": "1"}, [
        step("small3"), step("small3", env={"TMC2_TEST_BLIST_CAP": "16"}, fails=True), step("small3")]),
    "S5-plane-padding": ({}, [step("sat"), step("edge")]),
}

# six different GOFs over three GOF slots in flight: slot k decodes GOF k, then GOF k + 3
THREE_SLOTS = ["A", "A-inv", "A-shift", "B11", "B11-shift", "A-c8"]


# ---- CPU: mirror of the table decisions of Batch::prepare and launch ----------------------------------------------------
class TablesMirror:
    """Batch::prepare's cell-table layout (dense or hashed, slots, table frames TF, frame groups) and what launch leaves
    pending, for one batch.  `submit` returns the kinds of hand-over a launch makes, and leaves in `on`, `reset` and `GF`
    which tables it used, which of them prepare re-zeroed, and its frames per group."""
    CELL_BYTES = 32

    def __init__(self, env):
        self.env = dict(env)
        self.budget = 0
        self.group_frames = 32
        self.tabs = {"geo": dict(slots=0, frames=0, hashed=False, grid=None), "col": dict(slots=0, frames=0, hashed=False, grid=None)}
        self.clear_pending = False
        self.n_groups = 1
        self.last_on = None
        self.skipped_since_clear = False

    def submit(self, g, step_env=None, fails=False, F=None):
        env = {**self.env, **(step_env or {})}
        P, F = g.params, g.frame_count if F is None else F
        on = {"geo": bool(P.geometry_smoothing), "col": bool(P.color_smoothing and P.attribute_count)}
        self.on, self.reset, self.GF = on, {"geo": False, "col": False}, max(F, 1)
        seen = set()
        if not (on["geo"] or on["col"]):
            if self.clear_pending:
                self.skipped_since_clear = True
            return seen
        if "TMC2_SMOOTH_GROUP" in env:
            self.group_frames = max(1, int(env["TMC2_SMOOTH_GROUP"]))
        if self.budget == 0:
            assert "TMC2_TABLE_BUDGET_MB" in env, "the default budget depends on the free device memory"
            self.budget = max(1, int(env["TMC2_TABLE_BUDGET_MB"])) << 20
        maxs = 1 << P.geometry_bitdepth_3d
        cap = -(-2 * g.width * g.height // 16) * 16
        force = "TMC2_FORCE_HASH" in env
        grids = {"geo": P.grid_size, "col": P.cgrid_size}
        cells_of = lambda s: (-(-maxs // s)) ** 3

        def fit(GF, sets):
            for k in ("geo", "col"):
                per_frame = cells_of(grids[k]) * self.CELL_BYTES
                if on[k] and not force and per_frame <= self.budget:
                    GF = min(GF, max(1, self.budget // (sets * per_frame)))
            return GF
        GF = fit(min(self.group_frames, max(F, 1)), 1)
        n_sets = 1
        if GF < F:
            GF, n_sets = fit(min(self.group_frames, max(F, 1)), 2), 2
        TF = n_sets * GF
        for k in ("geo", "col"):
            if not on[k]:
                continue
            t = self.tabs[k]
            hashed = force or cells_of(grids[k]) * self.CELL_BYTES > self.budget
            slots = 1 << max(0, (2 * cap - 1).bit_length()) if hashed else cells_of(grids[k])
            grid = (grids[k], P.geometry_bitdepth_3d)
            if slots != t["slots"] or TF > t["frames"] or hashed != t["hashed"]:
                self.reset[k] = True
                if t["slots"] == 0 and t["grid"] is not None:
                    seen.add("reset after a failure")
                elif t["slots"] and hashed != t["hashed"]:
                    # every flip these sequences make also changes the slot count, which resets on its own: a prepare that
                    # ignored the dense / hashed flip would decode them the same (and equal slot counts would meet a key
                    # array that was never filled)
                    flip = "hashed -> dense" if t["hashed"] else "dense -> hashed"
                    seen.add(f"{flip} reset" + (", slot count changes too" if slots != t["slots"] else ", flip only"))
                t.update(slots=slots, frames=TF, hashed=hashed)
            else:
                if grid == t["grid"]:
                    seen.add("reuse, identical layout")
                elif hashed:
                    seen.add("hashed reuse, other grid")
                else:
                    seen.add("dense reuse, other grid with the same slot count")
                if TF < t["frames"]:
                    seen.add("TF shrinks without a reset")
                if self.last_on is not None and not self.last_on[k]:
                    seen.add("idle table reused")
            t["grid"] = grid
        n_groups = -(-F // GF)
        if self.n_groups == 1 and n_groups > 1:
            seen.add("one group -> several groups")
        if self.n_groups > 1 and n_groups == 1:
            seen.add("several groups -> one group")
        if self.clear_pending and self.skipped_since_clear:
            seen.add("clear pending across a GOF without smoothing")
        self.n_groups, self.last_on, self.GF = n_groups, on, GF
        self.clear_pending, self.skipped_since_clear = n_groups == 1, False
        if fails:
            for t in self.tabs.values():     # finish_counts: the next prepare starts from zeroed tables
                t.update(slots=0, frames=0)
        return seen


TRANSITIONS = {"reuse, identical layout", "dense reuse, other grid with the same slot count", "hashed reuse, other grid",
               "dense -> hashed reset, slot count changes too", "hashed -> dense reset, slot count changes too",
               "TF shrinks without a reset", "one group -> several groups", "several groups -> one group",
               "clear pending across a GOF without smoothing", "idle table reused", "reset after a failure"}


def batch_launches():
    """Every batch the GPU tests drive, as (env, [(GOF, step env, fails, frames of the GOF in one launch)])."""
    out = []
    for name, (env, steps) in SEQUENCES.items():
        out.append((f"{name}/stream", env, [(g, e, x, list(range(gof(g).frame_count))) for g, e, x in steps]))
        out.append((f"{name}/stage", env, [(g, e, x, [f]) for g, e, x in steps for f in range(gof(g).frame_count)]))
    for k in range(3):
        out.append((f"three-slots/{k}", {"TMC2_TABLE_BUDGET_MB": BUDGET_MB},
                    [(g, {}, False, list(range(gof(g).frame_count))) for g in THREE_SLOTS[k::3]]))
    return out


def handovers(env, launches):
    """(kind, (A, frame), (B, frame)) for every frame of a launch whose table frame of that kind was last written by an
    earlier frame (of an earlier GOF, or of an earlier group of the same GOF) and not re-zeroed by prepare since.  Frame j
    of a launch sits in group j // GF, table set group & 1, table frame set * GF + j % GF; a table a GOF does not use keeps
    what its last writer left."""
    m = TablesMirror(env)
    writer = {"geo": {}, "col": {}}
    for name, senv, fails, frames in launches:
        m.submit(gof(name), senv, fails, len(frames))
        for k in writer:
            if m.reset[k]:
                writer[k] = {}
        for j, f in enumerate(frames):
            gi = j // m.GF
            tf = (gi & 1) * m.GF + j - gi * m.GF
            for k in writer:
                if m.on[k]:
                    if tf in writer[k] and not fails:
                        yield k, writer[k][tf], (name, f)
                    writer[k][tf] = (name, f)
        if fails:
            writer = {"geo": {}, "col": {}}


HANDOVERS = sorted({h for _, env, launches in batch_launches() for h in handovers(env, launches)})


def test_sequences_reach_every_table_hand_over():
    reached = set()
    for _, env, launches in batch_launches():
        m = TablesMirror(env)
        for name, senv, fails, frames in launches:
            reached |= m.submit(gof(name), senv, fails, len(frames))
    assert TRANSITIONS <= reached, f"not reached: {sorted(TRANSITIONS - reached)}"


def test_mirror_layouts_of_the_layout_sequence():
    """Spot checks of the mirror on S3: the grids of 'A' and 'B11' have the same slot count, the 2^27-cell colour grid is
    hashed with 2 * cap slots, and the first frame after the three groups of 'B11-5f' reads what its frame 4 left."""
    m = TablesMirror(SEQUENCES["S3-layouts"][0])
    m.submit(gof("A"))
    assert m.tabs["geo"]["slots"] == m.tabs["col"]["slots"] == 128 ** 3 and m.n_groups == 1
    m.submit(gof("B11"))
    assert m.tabs["geo"]["slots"] == 128 ** 3 and m.tabs["geo"]["grid"] == (16, 11)
    m.submit(gof("B11-5f"))
    assert m.n_groups == 3 and m.tabs["geo"]["frames"] == 4
    m.submit(gof("A-c2"))
    assert m.tabs["col"]["hashed"] and m.tabs["col"]["slots"] == 32768
    h = set(handovers(*batch_launches()[4][1:]))
    assert ("geo", ("B11-5f", 4), ("B11-shift", 0)) in h and ("geo", ("B11-5f", 1), ("B11-shift", 1)) in h
    assert ("geo", ("B11-5f", 0), ("B11-5f", 4)) in h                    # group 2 reuses the set of group 0
    assert ("geo", ("B11-geo", 0), ("B11", 0)) in h and ("col", ("B11-inv", 0), ("B11-col", 0)) in h   # idle tables


# ---- CPU: the leak model is decisive on every hand-over ----------------------------------------------------------------
def _differing(m0, m1, key):
    a, b = np.array(m0[key], np.int64).reshape(-1, 3), np.array(m1[key], np.int64).reshape(-1, 3)
    return int((a != b).any(axis=1).sum())


@functools.lru_cache(maxsize=None)
def _statistics(name, f):
    return smoothmodel.oracle_frame_statistics(gof(name).params, oracle_frames(name)[f])


@functools.lru_cache(maxsize=None)
def _clean(name, f):
    m = smoothmodel.smooth_oracle_frame(gof(name).params, oracle_frames(name)[f])
    assert np.array_equal(np.array(m["positions"], np.int64).reshape(-1, 3), oracle_frames(name)[f]["positions"])
    return m


@pytest.mark.parametrize("kind,left,right", HANDOVERS, ids=[f"{k}-{a[0]}.{a[1]}-{b[0]}.{b[1]}" for k, a, b in HANDOVERS])
def test_leftover_statistics_change_the_next_frame(kind, left, right):
    """For every hand-over of a table the GPU sequences make without a reset, smooth(B, prior = what A left in that table)
    differs from smooth(B) on at least five points: a clear that missed that table would fail the oracle comparison."""
    (a, fa), (b, fb) = left, right
    prior = _statistics(a, fa)[kind]
    assert prior, f"{a} frame {fa} leaves no {kind} cells"
    leaked = smoothmodel.smooth_oracle_frame(gof(b).params, oracle_frames(b)[fb], prior={kind: prior})
    n = _differing(_clean(b, fb), leaked, "positions" if kind == "geo" else "colors")
    assert n >= 5, f"{a} frame {fa} -> {b} frame {fb}: a leftover {kind} table changes only {n} points"


def test_same_gof_twice_hides_a_leftover_colour_table():
    """The blind spot of decoding one GOF twice: with its own colour statistics left over, every colour cell holds twice its
    count and sums, and the variance test, the Q8 means and the patch sets all come out the same."""
    g = gof("A")
    for f, o in enumerate(oracle_frames("A")):
        left = smoothmodel.oracle_frame_statistics(g.params, o)
        clean = smoothmodel.smooth_oracle_frame(g.params, o)
        doubled = smoothmodel.smooth_oracle_frame(g.params, o, prior={"col": left["col"]})
        assert clean["recoloured"] > 0, f"frame {f}"
        assert _differing(clean, doubled, "colors") == 0, f"frame {f}"
        assert _differing(clean, smoothmodel.smooth_oracle_frame(g.params, o, prior={"geo": left["geo"]}), "positions") > 0


def _plane_layout(g, kind):
    """(w, h, pitch, bytes per sample, maps) of a batch plane, as Batch::prepare describes it."""
    occ_w, occ_h = g.occ.shape[2], g.occ.shape[1]
    return {"occ": (occ_w, occ_h, -(-occ_w // 16) * 16, 1, 1),
            "geo": (g.width, g.height, -(-g.width // 64) * 64, 2, 2),
            "attr_y": (g.width, g.height, -(-g.width // 64) * 64, 2, 2),
            "attr_u": (g.width // 2, g.height // 2, -(-(g.width // 2) // 64) * 64, 2, 2)}[kind]


@pytest.mark.parametrize("kind", ["occ", "geo", "attr_y", "attr_u"])
def test_edge_gof_padding_holds_what_the_wide_gof_wrote(kind):
    """S5 precondition: 'sat' has no padding of its own (every row as wide as its pitch), and the padding right of every row
    of 'edge' (between w and the pitch) lies inside the bytes 'sat' wrote, so it holds saturated samples.  S5 is a
    regression guard: at the block-aligned widths the TMA path sees, no kernel is known to read that padding."""
    a, b = gof("sat"), gof("edge")
    wa, ha, pa, esz, maps = _plane_layout(a, kind)
    wb, hb, pb, _, _ = _plane_layout(b, kind)
    assert wa == pa, f"{kind}: the wide GOF has padding of its own"
    assert wb < pb, f"{kind}: no padding in the rows of the edge GOF"
    assert b.frame_count * maps * hb * pb <= a.frame_count * maps * ha * pa, f"{kind}: the edge GOF's planes reach past the wide GOF's"


# ---- GPU -----------------------------------------------------------------------------------------------------------------
def _check(got, name, f, what):
    want = oracle_frames(name)[f]
    assert len(got["positions"]) == want["point_count"], f"{what}: {len(got['positions'])} points, oracle {want['point_count']}"
    util.assert_same(got, want, keys=("positions", "colors"), what=what)
    assert (got["smoothed_positions"], got["smoothed_colors"]) == (want["smoothed_positions"], want["smoothed_colors"]), what


def _frame(fr):
    return {"point_count": len(fr), "positions": fr.positions, "colors": fr.colors if fr.with_colors else np.zeros((0, 3)),
            "smoothed_positions": fr.smoothed_positions, "smoothed_colors": fr.smoothed_colors}


class _StepEnv:
    def __init__(self, env):
        self.env = env

    def __enter__(self):
        os.environ.update(self.env)

    def __exit__(self, *exc):
        for k in self.env:
            os.environ.pop(k, None)


def _streamed(ctx, name, view, fails, what):
    if fails:
        ctx.submit_gof(view)
        with pytest.raises(abi.Tmc2Error):
            ctx.next_frame()
        assert ctx.next_frame() is None, f"{what}: frames of the failed GOF were handed out"
        return
    for f, fr in enumerate(ctx.decode_gof(view)):
        _check(_frame(fr), name, f, f"{what} frame {f}")


def _staged(ctx, name, view, fails, what):
    for f in range(gof(name).frame_count):
        if fails:
            with pytest.raises(abi.Tmc2Error):
                ctx.generate_point_cloud(view, f)
            continue
        _check(ctx.generate_point_cloud(view, f), name, f, f"{what} frame {f}")


@pytest.fixture
def seq_env(monkeypatch):
    def apply(env):
        for k in ("TMC2_TABLE_BUDGET_MB", "TMC2_SMOOTH_GROUP", "TMC2_FORCE_HASH", "TMC2_TEST_BLIST_CAP"):
            monkeypatch.delenv(k, raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
    return apply


@pytest.mark.gpu
@pytest.mark.parametrize("api", ["stream", "stage"])
@pytest.mark.parametrize("seq", list(SEQUENCES))
def test_sequence_matches_oracle(seq_env, seq, api):
    """Every GOF of the sequence, on one batch (one GOF slot, or the stage API's batch), equals the oracle."""
    env, steps = SEQUENCES[seq]
    seq_env(env)
    ctx = codec.Context(gofs_in_flight=1)
    try:
        for i, (name, senv, fails) in enumerate(steps):
            with _StepEnv(senv):
                (_streamed if api == "stream" else _staged)(ctx, name, abi.GofView(gof(name)), fails,
                                                            f"{seq}/{api} step {i} ({name})")
    finally:
        ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["planar", "p010"])
def test_edge_gof_from_device_planes_after_a_saturated_gof(seq_env, fmt):
    """S5 with the edge GOF's planes already in device memory (gathered by the ingest kernel into the batch layout)."""
    import torch
    seq_env({})
    ctx = codec.Context(gofs_in_flight=1)
    try:
        _streamed(ctx, "sat", abi.GofView(gof("sat")), False, "sat")
        view = abi.GofView(synth.to_device(gof("edge"), torch.device("cuda", 0), p010=fmt == "p010", seed=5))
        for f, fr in enumerate(ctx.decode_gof(view)):
            _check(_frame(fr), "edge", f, f"edge/{fmt} frame {f}")
    finally:
        ctx.close()


@pytest.mark.gpu
def test_three_slots_six_gofs(seq_env):
    """Three GOF slots in flight and six different GOFs: each slot decodes two of them, while the other slots run."""
    names = THREE_SLOTS
    seq_env({"TMC2_TABLE_BUDGET_MB": BUDGET_MB})
    ctx = codec.Context(gofs_in_flight=3)
    try:
        views = [abi.GofView(gof(n)) for n in names]
        for v in views[:3]:
            ctx.submit_gof(v)
        for i, name in enumerate(names):
            for f in range(gof(name).frame_count):
                _check(_frame(ctx.next_frame()), name, f, f"GOF {i} ({name}) frame {f}")
            if i + 3 < len(names):
                ctx.submit_gof(views[i + 3])
        assert ctx.next_frame() is None
    finally:
        ctx.close()


@pytest.mark.gpu
def test_resident_relaunch_after_a_failure_fails_again(seq_env):
    """A resident relaunch does not go through prepare, so nothing resets its tables after a failure: the relaunch must
    report the failure again, never counts."""
    seq_env({"TMC2_TABLE_BUDGET_MB": BUDGET_MB})
    ctx = codec.Context(gofs_in_flight=1)
    r = ctx.upload_gof(abi.GofView(gof("cell-65537")))
    try:
        for attempt in range(2):
            r.reconstruct()
            with pytest.raises(abi.Tmc2Error) as e:
                r.counts()
            assert e.value.status == 6, f"attempt {attempt}: status {e.value.status}"
    finally:
        r.free()
        ctx.close()
