"""The unpack across occupancy resolutions, precisions and canvas sizes, on its image-edge inputs and at the limits of its
index widths.

* A matrix of (resolution, precision, W x H, attributes, orientations, occupancy slack) runs through the debug stage API,
  streaming, the resident path, a device-output context and the device-plane ingest (planar and P010) against the oracle,
  without smoothing and with the `g8c4` (fast) and `g6c3` (generic) smoothing settings of test_emit_instantiations.py.  A
  CPU mirror of the kernels' selection rules labels every entry by the branches it takes (block ownership, occupancy
  source, boundary-class path) and by what its canvas has at the right and bottom edges; it fails when an edit of the
  matrix leaves a label unreached.
* Decisive image-edge inputs, each a pair of GOFs that differ only in the samples that decide: occupancy slack beyond
  the image (E1), the strip of pixels right of / below the last block (E2, E3) and a last occupancy cell that reaches past
  the image (E4).  A CPU assertion keeps each pair decisive.
* Limits: 32 767-pixel frames (point_to_pixel x / y >= 2^14 in its 15-bit fields), 65 535 patches (partition indices
  near 2^16), resolution 64 and a patch 4 096 blocks wide are accepted; one more of each is refused.

On the CPU the oracle is checked against tests/refmodel.py and its boundary classes against util.boundary_spec on every
matrix entry.
"""
import numpy as np
import pytest

import refmodel
import test_emit_instantiations as tei
import util
from oracle import oracle
from test_smoothing_limits import assert_refused
from tmc2rs_b200 import abi, synth

ALL9 = tuple(range(9))

# ---- the matrix -----------------------------------------------------------------------------------------------------------
# (id, util.random_small_gof arguments).  Widths and heights are picked for what lies beyond the last block and the last
# whole occupancy cell; the comment names what the entry is there for.
MATRIX = [
    # block-aligned side: resolution 16
    ("r16p8", dict(seed=101, res=16, prec=8, W=80, H=72, orientations=(0, 1, 8))),          # mask lp 3, bitmap_row
    ("r16p16-spec", dict(seed=102, res=16, prec=16, W=96, H=56, orientations=ALL9, spec=True)),   # cell > strip
    ("r16p32", dict(seed=103, res=16, prec=32, W=80, H=64, orientations=ALL9)),             # W = 16 mod 32: half a cell
    ("r16p64-spec", dict(seed=104, res=16, prec=64, W=96, H=80, orientations=ALL9, spec=True)),   # cell > block
    ("r16p4-w66", dict(seed=105, res=16, prec=4, W=66, H=48, orientations=(0, 1, 8))),      # W = 2 mod 4: mask path
    ("r16p4-w68-spec", dict(seed=106, res=16, prec=4, W=68, H=52, orientations=ALL9, spec=True)),  # TMA box + strip
    ("r16p2-odd", dict(seed=107, res=16, prec=2, W=65, H=49, orientations=(0, 1, 2, 5), attr=False)),
    ("r16p1-slack", dict(seed=108, res=16, prec=1, W=48, H=48, orientations=(0, 1), slack=(3, 2), slack_fill=255)),
    # generic side
    ("r1p1-spec", dict(seed=111, res=1, prec=1, W=24, H=20, orientations=ALL9, spec=True)),
    ("r2p2-odd", dict(seed=112, res=2, prec=2, W=35, H=30, orientations=(0, 1, 3), attr=False)),
    ("r4p4", dict(seed=113, res=4, prec=4, W=42, H=40, orientations=ALL9)),
    ("r8p16-spec", dict(seed=114, res=8, prec=16, W=72, H=56, orientations=(0, 1, 8), spec=True)),
    ("r12p12-slack", dict(seed=115, res=12, prec=12, W=60, H=50, orientations=ALL9, slack=(1, 1))),
    ("r48p4-spec", dict(seed=116, res=48, prec=4, W=100, H=96, orientations=(0, 1, 5), spec=True)),
    ("r64p4", dict(seed=117, res=64, prec=4, W=136, H=128, orientations=ALL9)),
    ("r64p64-spec", dict(seed=118, res=64, prec=64, W=128, H=70, orientations=(0, 1, 8), spec=True)),
    ("r16p3", dict(seed=119, res=16, prec=3, W=50, H=48, orientations=(0, 1, 8))),
    ("r16p12-spec", dict(seed=120, res=16, prec=12, W=64, H=44, orientations=ALL9, spec=True)),
]
IDS = [e[0] for e in MATRIX]
MODES = ("off", "g8c4", "g6c3")


def matrix_gof(entry, mode="off"):
    return tei.make_gof(entry[1], mode)


def narrow_tails(g):
    """Rows of some plane are not whole 16-byte vectors: the ingest kernel's narrow tails copy them."""
    W, ow = g.width, g.occ.shape[2]
    return W % 8 != 0 or (W // 2) % 8 != 0 or ow % 8 != 0


# ---- the selection rules, mirrored ------------------------------------------------------------------------------------------
def _lp(prec):
    return prec.bit_length() - 1 if tei._pow2(prec) else None


def b2p_branch(params, p, bx):
    """block_to_patch_kernel (kernels.cu): which loop decides whether block column bx of patch p is occupied."""
    res, prec = params.occupancy_resolution, params.occupancy_precision
    aligned = params.orientation_mode == abi.ORIENTATION_SPEC or int(p["patch_orientation"]) in (0, 1, 8)
    if not aligned:
        return "b2p:reference-literal"
    cxa, cxb = bx * res // prec, (bx * res + res - 1) // prec
    return "b2p:aligned-words" if (cxa | (cxb + 1)) & 3 == 0 else "b2p:aligned-bytes"


def slot_branches(params, W, H, orientation):
    """(occupancy source, boundary-class path) of a slot: tei.slot_path refined by occupancy_mask's precision branches and
    by boundary_masks (the 6 x 6 TMA window needs the same frame shape as the occupancy box)."""
    path = tei.slot_path(params, W, H, orientation)
    if path == "generic-slot":
        return "occ:generic", "bt:per-pixel"
    if path == "tma-box":
        return "occ:tma-box", "bt:tma-6x6"
    lp = _lp(params.occupancy_precision)
    return ("occ:mask-lp>=3" if lp >= 3 else f"occ:mask-lp{lp}"), "bt:bitmap_row"


def canvas_labels(g):
    P = g.params
    res, prec = P.occupancy_resolution, P.occupancy_precision
    out = set()
    for axis, n, on in (("W", g.width, g.occ.shape[2]), ("H", g.height, g.occ.shape[1])):
        out.add(f"{axis}:last block touches {axis}-1" if n % res == 0 else f"{axis}:strip beyond the blocks")
        if n % prec:
            out.add(f"{axis}:partial cell")
        if on > -(-n // prec):
            out.add(f"{axis}:slack")
        if n % 2:
            out.add(f"{axis}:odd")
    if prec > res:
        out.add("prec > res")
    return out


def labels(g):
    """Every branch label of one GOF: block ownership over all slots, occupancy source and boundary path over the slots
    that own their block, and the canvas labels; boundary paths combined with a partial edge cell are labelled too."""
    P = g.params
    out = canvas_labels(g)
    for f in range(g.frame_count):
        for p in g.patches[f]:
            for v0b in range(int(p["size_v0"])):
                for u0b in range(int(p["size_u0"])):
                    bx, _ = util._helper(p, u0b, v0b, 1, 1)
                    out.add(b2p_branch(P, p, bx))
    for _, p, _ in tei.emitting_slots(g):
        occ, bt = slot_branches(P, g.width, g.height, int(p["patch_orientation"]))
        out |= {occ, bt}
        if g.width % P.occupancy_precision or g.height % P.occupancy_precision:
            out.add(bt + " + partial cell")
    return out


WANT_LABELS = {
    "b2p:aligned-words", "b2p:aligned-bytes", "b2p:reference-literal",
    "occ:tma-box", "occ:mask-lp0", "occ:mask-lp1", "occ:mask-lp2", "occ:mask-lp>=3", "occ:generic",
    "bt:tma-6x6", "bt:bitmap_row", "bt:per-pixel", "bt:bitmap_row + partial cell", "bt:per-pixel + partial cell",
    "prec > res",
} | {f"{a}:{what}" for a in "WH" for what in (f"last block touches {a}-1", "strip beyond the blocks", "partial cell",
                                            "slack", "odd")}


def test_matrix_reaches_every_branch():
    """Fails when an edit of MATRIX leaves a branch or canvas label unreached, or drops a resolution / precision the issue
    of this file is about."""
    reached = set()
    for entry in MATRIX:
        reached |= labels(matrix_gof(entry))
    assert not WANT_LABELS - reached, f"not reached: {sorted(WANT_LABELS - reached)}"
    pairs = {(e[1]["res"], e[1]["prec"]) for e in MATRIX}
    assert {p for r, p in pairs if r == 16} >= {1, 2, 3, 4, 8, 12, 16, 32, 64}
    assert {r for r, _ in pairs} >= {1, 2, 4, 8, 12, 16, 48, 64}
    assert {e[1].get("spec", False) for e in MATRIX} == {False, True}
    assert any(narrow_tails(matrix_gof(e)) and e[1].get("attr", True) for e in MATRIX)


# ---- CPU: the oracle on every entry -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("entry", MATRIX, ids=IDS)
def test_oracle_matches_refmodel(entry):
    g = matrix_gof(entry)
    view = abi.GofView(g)
    points = 0
    for f in range(g.frame_count):
        want = refmodel.reconstruct(g, f)
        got = oracle.reconstruct_frame(view, f)
        assert got["point_count"] == len(want["positions"]), f
        for k in ("block_to_patch", "occupancy_map", "positions", "partition", "point_to_pixel"):
            assert got[k].tolist() == want[k], (f, k)
        if g.params.attribute_count:
            assert got["colors16bit"].tolist() == want["colors16bit"], f
            assert got["colors"].tolist() == want["colors"], f
        points += got["point_count"]
    assert points > 0


@pytest.mark.parametrize("entry", MATRIX, ids=IDS)
def test_oracle_boundary_classes_match_the_spec(entry):
    g = matrix_gof(entry)
    g.params.geometry_smoothing = True
    seen = set()
    for f in range(g.frame_count):
        a = oracle.reconstruct_frame(abi.GofView(g), f)
        px = a["point_to_pixel"]
        assert np.array_equal(a["boundary_type"], util.boundary_spec(a["occupancy_map"])[px[:, 1], px[:, 0]]), f
        seen |= set(a["boundary_type"].tolist())
    assert seen >= {1, 2}


# ---- decisive image-edge inputs -------------------------------------------------------------------------------------------
def edge_gof(W, H, res, prec, attr=True, slack=(0, 0), slack_fill=0, seed=0):
    """One patch over every block (orientation 0, projection 0), every occupancy sample of the image occupied, geometry
    smoothing on so that the boundary classes are computed and used."""
    g = util.random_small_gof(seed=seed, W=W, H=H, res=res, prec=prec, attr=attr, orientations=(0,), n_patches=0,
                              slack=slack, slack_fill=slack_fill)
    n, t, b, mode = synth.VIEW_AXES[0]
    g.patches = [np.array([(0, 0, W // res, H // res, 0, 0, 0, 1, 1, n, t, b, mode, 0, 0, (0, 0))], dtype=abi.PATCH_DTYPE)]
    oh, ow = -(-H // prec), -(-W // prec)
    g.occ[:, :oh, :ow] = 1
    g.params.geometry_smoothing = True
    g.params.grid_size = 8
    return g


def classes(frame):
    """{(x, y): boundary class} of the points of an oracle frame."""
    return {(int(x), int(y)): int(b) for (x, y, _), b in zip(frame["point_to_pixel"].tolist(), frame["boundary_type"])}


def _frame(g):
    return oracle.reconstruct_frame(abi.GofView(g), 0)


# E1: (resolution, precision) of the TMA 6x6 window, bitmap_row and the per-pixel path; W = res * 4, two slack columns
E1 = {"tma-6x6": (16, 4), "bitmap_row": (16, 8), "per-pixel": (12, 4)}


def e1_pair(which):
    res, prec = E1[which]
    W, H = 4 * res, 48
    return [edge_gof(W, H, res, prec, slack=(2, 2), slack_fill=fill, seed=41) for fill in (0, 255)]


def test_e1_slack_is_not_image():
    """Slack samples of 0 and of 255 give the same frames; a spec that read the slack as image would class x = W - 2
    differently (type 2, not 0)."""
    for which in E1:
        g0, g1 = e1_pair(which)
        f0, f1 = _frame(g0), _frame(g1)
        for k in ("positions", "boundary_type", "point_to_pixel"):
            assert np.array_equal(f0[k], f1[k]), (which, k)
        W, H, prec = g0.width, g0.height, g0.params.occupancy_precision
        as_image = np.kron(g0.occ[0], np.ones((prec, prec), np.uint8))     # the slack upsampled as if it were image
        wrong = util.boundary_spec(as_image)[:H, :W]
        got = classes(f0)
        assert got[(W - 2, H // 2)] == 0 and wrong[H // 2, W - 2] == 2, which
    assert slot_branches(e1_pair("tma-6x6")[0].params, 64, 48, 0)[1] == "bt:tma-6x6"
    assert slot_branches(e1_pair("bitmap_row")[0].params, 64, 48, 0)[1] == "bt:bitmap_row"
    assert slot_branches(e1_pair("per-pixel")[0].params, 48, 48, 0)[1] == "bt:per-pixel"


# E2 / E3: the strip beyond the last block column (row), 4 or 2 pixels wide, occupied and then empty (precision 4: the
# TMA 6x6 window at + 4, bitmap_row with a cell that straddles the image edge at + 2)
STRIPS = [("x", 4), ("x", 2), ("y", 4), ("y", 2)]


def strip_pair(axis, extra):
    W, H = (64 + extra, 48) if axis == "x" else (64, 48 + extra)
    out = []
    for fill in (1, 0):
        g = edge_gof(W, H, 16, 4, seed=43)
        if axis == "x":
            g.occ[:, :, 16:] = fill
        else:
            g.occ[:, 12:, :] = fill
        out.append(g)
    return out


def last_block_classes(g, frame, axis):
    lo = (g.width // 16 - 1) * 16 if axis == "x" else (g.height // 16 - 1) * 16
    return {p: c for p, c in classes(frame).items() if p[0 if axis == "x" else 1] >= lo}


@pytest.mark.parametrize("axis,extra", STRIPS)
def test_e2_e3_the_strip_decides_the_last_block(axis, extra):
    occupied, empty = strip_pair(axis, extra)
    a, b = (last_block_classes(g, _frame(g), axis) for g in (occupied, empty))
    assert a.keys() == b.keys() and a != b
    edge = 63 if axis == "x" else 47
    assert {c for p, c in b.items() if p[0 if axis == "x" else 1] == edge} == {1}
    assert slot_branches(occupied.params, occupied.width, occupied.height, 0)[1] == \
        ("bt:tma-6x6" if extra == 4 else "bt:bitmap_row")


# E4: a last occupancy cell that reaches past the image, occupied and then empty: precision 32 (W = 80, the cell covers
# the last block column and 16 pixels beyond the image) and 3 (W = 49, the cell holds the one strip pixel x = 48)
E4 = {"p32": dict(W=80, H=64, res=16, prec=32, attr=True), "p3": dict(W=49, H=48, res=16, prec=3, attr=False)}


def e4_pair(which):
    out = []
    for fill in (255, 0):
        g = edge_gof(seed=44, **E4[which])
        g.occ[:, :, -1] = fill
        out.append(g)
    return out


@pytest.mark.parametrize("which", E4)
def test_e4_partial_last_cell_decides(which):
    occupied, empty = e4_pair(which)
    a, b = _frame(occupied), _frame(empty)
    assert occupied.width % occupied.params.occupancy_precision != 0
    x = (occupied.occ.shape[2] - 1) * occupied.params.occupancy_precision - 1     # the pixel left of the last cell
    ca, cb = classes(a), classes(b)
    assert cb[(x, occupied.height // 2)] == 1 and ca[(x, occupied.height // 2)] == 0
    if which == "p32":
        assert a["point_count"] > b["point_count"]


def edge_cases():
    out = []
    for which in E1:
        out += [(f"E1-{which}-slack{fill}", g) for fill, g in zip((0, 255), e1_pair(which))]
    for axis, extra in STRIPS:
        out += [(f"E{2 if axis == 'x' else 3}-{extra}-{what}", g) for what, g in zip(("occupied", "empty"),
                                                                                      strip_pair(axis, extra))]
    for which in E4:
        out += [(f"E4-{which}-{what}", g) for what, g in zip(("occupied", "empty"), e4_pair(which))]
    return out


EDGE_IDS = [name for name, _ in edge_cases()]


# ---- limits ------------------------------------------------------------------------------------------------------------------
# L1: the largest frames.  (W, H, precision, attributes)
L1 = [(32767, 32, 1, False), (32766, 32, 2, True), (32, 32767, 1, False), (32, 32766, 2, True)]


def l1_gof(W, H, prec, attr, smooth):
    g = util.random_small_gof(seed=51, W=W, H=H, res=16, prec=prec, attr=attr, orientations=(0, 1), n_patches=12)
    g.params.geometry_smoothing = smooth
    g.params.color_smoothing = smooth and attr
    return g


def test_l1_point_to_pixel_reaches_the_top_bit_of_its_fields():
    for W, H, prec, attr in L1:
        ptp = _frame(l1_gof(W, H, prec, attr, False))["point_to_pixel"]
        assert ptp[:, 0 if W > H else 1].max() >= 1 << 14, (W, H)


L2_PATCHES = 65535


def l2_gof(n_patches=L2_PATCHES):
    """n one-block patches cycling over the 256 blocks of a 256 x 256 canvas: the last 256 own every block."""
    n, t, b, mode = synth.VIEW_AXES[0]
    i = np.arange(n_patches)
    p = np.zeros(n_patches, abi.PATCH_DTYPE)
    p["u0"], p["v0"] = i % 16, (i // 16) % 16
    p["size_u0"] = p["size_v0"] = 1
    p["u1"], p["v1"], p["d1"] = 16 * (i % 16), 16 * ((i // 16) % 16), i % 64
    p["lod_x"] = p["lod_y"] = 1
    p["normal_axis"], p["tangent_axis"], p["bitangent_axis"], p["projection_mode"] = n, t, b, mode
    rng = np.random.RandomState(52)
    occ = (rng.rand(1, 64, 64) < 0.8).astype(np.uint8)
    geo = rng.randint(0, 1024, (1, 2, 256, 256)).astype(np.uint16)
    params = abi.Params(occupancy_resolution=16, occupancy_precision=4, attribute_count=0)
    return abi.Gof(256, 256, occ, geo, None, None, None, [p], params)


def test_l2_partition_reaches_65534():
    f = _frame(l2_gof())
    assert int(f["partition"].max()) == L2_PATCHES - 1
    assert int(f["block_to_patch"].min()) == L2_PATCHES - 255


def l4_gof(size_u0):
    """Resolution 1: one patch size_u0 blocks (pixels) wide on a 4100 x 2 canvas."""
    g = util.random_small_gof(seed=54, W=4100, H=2, res=1, prec=1, orientations=(0,), n_patches=0)
    n, t, b, mode = synth.VIEW_AXES[0]
    g.patches = [np.array([(0, 0, size_u0, 2, 0, 0, 0, 1, 1, n, t, b, mode, 0, 0, (0, 0))], dtype=abi.PATCH_DTYPE)]
    return g


def test_l4_widest_patch_is_inside_the_canvas():
    """4 097 blocks still fit the canvas: the library's refusal is its size limit, not the canvas check."""
    assert _frame(l4_gof(4096))["point_count"] > 0
    assert _frame(l4_gof(4097))["point_count"] > 0


# ---- GPU ------------------------------------------------------------------------------------------------------------------
device_ctx = tei.device_ctx                 # one device-output context for the module
DEBUG_PRE = ("boundary_type", "positions_presmooth", "colors16bit_presmooth")


def stream_keys(g):
    keys = [k for k in util.STREAMS if g.params.attribute_count or k not in ("colors", "colors16bit")]
    if g.params.geometry_smoothing or g.params.color_smoothing:
        keys += [k for k in DEBUG_PRE if k != "colors16bit_presmooth" or (g.params.attribute_count and g.params.color_smoothing)]
    return keys


def check_stage_and_streaming(ctx, g, what, want=None):
    view = abi.GofView(g)
    want = want or [oracle.reconstruct_frame(view, f) for f in range(g.frame_count)]
    for f in range(g.frame_count):
        got = ctx.generate_point_cloud(view, f)
        util.assert_same(got, want[f], keys=stream_keys(g), what=f"{what} stage frame {f}")
        assert (got["smoothed_positions"], got["smoothed_colors"]) == \
            (want[f]["smoothed_positions"], want[f]["smoothed_colors"]), f"{what} stage frame {f}: counts"
    for f, fr in enumerate(ctx.decode_gof(view)):
        tei._expect(len(fr), fr.positions, fr.colors, want[f], f"{what} streaming frame {f}",
                    (fr.smoothed_positions, fr.smoothed_colors))
    return want


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("entry", MATRIX, ids=IDS)
def test_matrix_matches_oracle(gpu_ctx, device_ctx, entry, mode):
    """Debug stage API, streaming, resident (with the emit instantiation read off the launch), device output and device
    planes, planar and P010, where a plane row ends in a narrow tail."""
    import torch
    g = matrix_gof(entry, mode)
    what = f"{entry[0]} {mode}"
    want = check_stage_and_streaming(gpu_ctx, g, what)
    view = abi.GofView(g)
    attr = g.params.attribute_count != 0
    r = gpu_ctx.upload_gof(view)
    try:
        names = tei._cuda_kernels(lambda: (r.reconstruct(), r.counts()))
        assert tei._emit_of(names) == {(tei.emit_instantiation(g.params, False), attr)}, names
        counts = r.counts()
        for f in range(g.frame_count):
            pos, col = r.fetch(f, int(counts[f]))
            tei._expect(int(counts[f]), pos, col, want[f], f"{what} resident frame {f}")
    finally:
        r.free()
    for f, (n, pos, col) in enumerate(tei._device_frames(device_ctx, view)):
        tei._expect(n, pos, col, want[f], f"{what} device output frame {f}")
    if narrow_tails(g):
        for fmt in ("planar", "p010") if attr else ("planar",):
            dv = abi.GofView(synth.to_device(g, "cuda:0", p010=fmt == "p010", seed=7))
            for f in range(g.frame_count):
                got = gpu_ctx.generate_point_cloud(dv, f)
                util.assert_same(got, want[f], keys=stream_keys(g), what=f"{what} device planes {fmt} frame {f}")
            torch.cuda.synchronize()


@pytest.mark.gpu
@pytest.mark.parametrize("index", range(len(EDGE_IDS)), ids=EDGE_IDS)
def test_edge_inputs_match_oracle(gpu_ctx, index):
    name, g = edge_cases()[index]
    check_stage_and_streaming(gpu_ctx, g, name)


@pytest.mark.gpu
@pytest.mark.parametrize("smooth", [False, True], ids=["plain", "smoothing"])
@pytest.mark.parametrize("shape", L1, ids=[f"{w}x{h}-p{p}" for w, h, p, _ in L1])
def test_l1_largest_frames_match_oracle(gpu_ctx, shape, smooth):
    g = l1_gof(*shape, smooth)
    check_stage_and_streaming(gpu_ctx, g, f"L1 {shape}")


@pytest.mark.gpu
def test_l1_width_or_height_32768_is_refused(gpu_ctx):
    for W, H in ((32768, 32), (32, 32768)):
        g = util.random_small_gof(seed=53, W=W, H=H, res=16, prec=1, attr=False, orientations=(0,), n_patches=2)
        assert_refused(gpu_ctx, abi.GofView(g), abi.ERR_CAPACITY)


@pytest.mark.gpu
def test_l2_65535_patches(gpu_ctx):
    """The partition stream (u16 on the device) reaches 65 534 and block_to_patch 65 535; 65 536 patches are refused."""
    g = l2_gof()
    want = check_stage_and_streaming(gpu_ctx, g, "L2")
    assert int(want[0]["partition"].max()) == L2_PATCHES - 1
    assert_refused(gpu_ctx, abi.GofView(l2_gof(L2_PATCHES + 1)), abi.ERR_CAPACITY)


@pytest.mark.gpu
def test_l3_resolution_64_accepted_65_refused(gpu_ctx):
    g = util.random_small_gof(seed=55, W=130, H=130, res=64, prec=2, orientations=ALL9)
    check_stage_and_streaming(gpu_ctx, g, "L3 resolution 64")
    g.params.occupancy_resolution = 65
    assert_refused(gpu_ctx, abi.GofView(g), abi.ERR_CAPACITY)


@pytest.mark.gpu
def test_l4_patch_4096_blocks_wide(gpu_ctx):
    check_stage_and_streaming(gpu_ctx, l4_gof(4096), "L4 4096 blocks")
    assert_refused(gpu_ctx, abi.GofView(l4_gof(4097)), abi.ERR_PATCH_OUT_OF_CANVAS)
