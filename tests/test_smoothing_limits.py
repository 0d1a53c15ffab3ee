"""Grid smoothing across its parameter range, on its decisive inputs and at the limits of its packed cell sums.

* A parameter matrix (attribute and geometry bit depths 8 / 9 / 12 / 16, cell edges 1, 5, 7, 9, 64, 255, 256, every
  threshold at 0, 1 and 65535) runs through the debug stage API and the streaming path against the oracle; grids wider
  than 1024 cells must be refused by both.  A CPU mirror of the selection rules checks that the matrix reaches every
  geometry statistics path, every colour table kind and both probes.
* Decisive inputs put each comparison of the filter exactly on equality (geometry, luminance variance, luminance
  difference, colour distance); a ramp atlas puts type-1 points on the border margin's exact coordinates.  Each runs one below, on and one above.
* Packed sums at their limits: a geometry cell whose offset sums need 64-bit means, the largest atlas smoothing accepts
  (4096 x 2032, 15 * 2^20 points in one cell), a colour cell with exactly 65 536 type-2 points at 16-bit samples, and the
  refusal of 65 537.
* `attribute_bitdepth` above 16 is refused by every entry point and by the oracle.

tests/smoothmodel.py restates the specification from DESIGN.md section 5; CPU tests check it against the oracle on these
cases and use it to assert that every equality, margin coordinate and limit count is still hit.
"""
import numpy as np
import pytest

import smoothmodel
import test_emit_instantiations as tei
import util
from oracle import oracle
from tmc2rs_b200 import abi, synth


# ---- content ---------------------------------------------------------------------------------------------------------
def scaled_crowd(seed, gbd, abd, frames=2, **kw):
    """util.crowd_into_one_region scaled to a volume of 2^gbd (patches overlap in 3D at any bit depth) with attribute
    samples scaled to abd bits; a sparse lattice of 0 and 2^abd - 1 samples covers the whole sample range."""
    g = util.random_small_gof(seed=seed, frames=frames, **kw)
    util.crowd_into_one_region(g)
    s = 2.0 ** (gbd - 10)
    for p in g.patches:
        n = len(p)
        p["u1"] = round(100 * s) + np.arange(n) % 3
        p["v1"] = round(100 * s) + np.arange(n) % 2
        p["d1"] = np.where(p["projection_mode"] == 0, round(64 * s), (1 << gbd) - round(364 * s))
    F, _, H, W = g.geo.shape
    yy, xx = np.mgrid[0:H, 0:W]
    rng = np.random.RandomState(seed)
    d0 = round(100 * s) + ((xx // 5 + yy // 7) % 9)
    delta = np.where(rng.rand(F, H, W) < 0.4, 0, rng.randint(1, 5, (F, H, W)))
    g.geo[:, 0] = (4 * d0 + rng.randint(0, 4, (F, H, W))).astype(np.uint16)
    g.geo[:, 1] = (4 * (d0 + delta) + rng.randint(0, 4, (F, H, W))).astype(np.uint16)
    if g.attr_y is not None:
        top, sa = (1 << abd) - 1, 2.0 ** (abd - 10)
        for a in (g.attr_y, g.attr_u, g.attr_v):
            a[...] = np.minimum(np.round(a * sa), top).astype(np.uint16)
            a[:, :, 3::11, 5::13] = top
            a[:, :, 7::11, 2::13] = 0
    g.params.geometry_bitdepth_3d = gbd
    g.params.attribute_bitdepth = abd
    return g


def set_smoothing(g, grid=None, cgrid=None, thr=(4, 2, 200, 200)):
    """thr = (threshold_smoothing, threshold_color_smoothing, threshold_color_difference, threshold_color_variation)."""
    P = g.params
    P.geometry_smoothing, P.color_smoothing = grid is not None, cgrid is not None
    P.grid_size, P.cgrid_size = grid or 8, cgrid or 4
    (P.threshold_smoothing, P.threshold_color_smoothing, P.threshold_color_difference,
     P.threshold_color_variation) = thr
    return g


# ---- the parameter matrix -----------------------------------------------------------------------------------------------
# (id, geometry bit depth, attribute bit depth, geometry edge, colour edge, hashed tables)
MATRIX = [
    ("g1-bd8", 8, 8, 1, 5, False),          # g = 1 on a 256-wide grid, colour generic: fast8 keys in the generic instantiation
    ("g1-bd9", 9, 9, 1, 7, False),          # g = 1 on a 512-wide grid (fast == 2): the scan of a power-of-two edge <= 8
    ("g1-bd12", 12, 12, 1, 9, False),       # 4096 cells wide: refused
    ("g5-bd12-hashed", 12, 12, 5, 9, True),
    ("g5c64-bd10-a8", 10, 8, 5, 64, False),
    ("g7c1-bd8-a16", 8, 16, 7, 1, False),   # th = 259 > 2^8; colour g = 1
    ("g64c255-bd12-a9", 12, 9, 64, 255, False),
    ("g256c256-bd16", 16, 16, 256, 256, False),
    ("g255c128-bd16-a12", 16, 12, 255, 128, False),   # colour grid 512 wide, dense: fast == 2
    ("g64c64-bd16-a8-hashed", 16, 8, 64, 64, True),   # 1024 wide: hashed only
    ("g8c4-bd9-a12", 9, 12, 8, 4, False),   # the fast instantiation
    ("g8c255-bd12-a16", 12, 16, 8, 255, False),       # power-of-two g <= 8 on a 512-wide geometry grid
    ("g9c9-bd9-a8", 9, 8, 9, 9, False),
    ("g9c7-bd12-a16-hashed", 12, 16, 9, 7, True),
    ("c5-bd16-a9", 16, 9, 255, 5, False),   # colour grid 13108 wide: refused
    ("g1-bd16", 16, 16, 1, 256, False),     # refused
]
THRESHOLDS = [(f"{name}={v}-a{abd}", abd, tuple(v if i == k else d for i, d in enumerate((4, 2, 200, 200))))
              for abd in (8, 16) for k, name in enumerate(("geo", "smooth", "diff", "var")) for v in (0, 1, 65535)]


def matrix_gof(entry, seed):
    _, gbd, abd, ge, ce, _ = entry
    return set_smoothing(scaled_crowd(seed, gbd, abd), ge, ce)


def threshold_gof(entry, seed):
    _, abd, thr = entry
    return set_smoothing(scaled_crowd(seed, 10, abd), 8, 5, thr)


def grid_width(params, g):
    return -(-(1 << params.geometry_bitdepth_3d) // g)


def refused(params):
    return any(on and grid_width(params, g) > 1024 for on, g in ((params.geometry_smoothing, params.grid_size),
                                                                 (params.color_smoothing, params.cgrid_size)))


def paths(params, hashed):
    """Which statistics branch, table kind and probe a launch takes: emit_instantiation (test_emit_instantiations.py)
    refined by the branches of the generic instantiation's `point()` and of the probe (kernels.cu)."""
    inst = tei.emit_instantiation(params, hashed)
    out = set()
    grids = []
    if params.geometry_smoothing:
        g = params.grid_size
        f = tei.grid_fast(params, g, hashed)
        grids.append(f)
        if hashed:
            out.add("geo:hashed")
        if inst == "fast":
            out.add("geo:fast8")                                  # the slot's shared-memory cell table
        elif f == 1 and g <= 8:
            out.add("geo:fast8-in-generic")                       # `fast8`: keys straight from the packed words
        elif g <= 8:                                              # one 8-bit scan word
            out.add(("geo:pow2<=8-" + ("hashed" if hashed else "fast2")) if tei._pow2(g) else "geo:npow2<=8")
        else:                                                     # the 16-bit scan word `1 | rx << 16`
            out.add("geo:pow2>8" if tei._pow2(g) else "geo:npow2>8")
    if params.color_smoothing and params.attribute_count:
        f = tei.grid_fast(params, params.cgrid_size, hashed)
        grids.append(f)
        out.add("col:hashed" if hashed else f"col:fast{f}" if f else "col:generic")
    out |= {"probe:fast" if f else "probe:generic" for f in grids}
    return out


def test_matrix_reaches_every_path():
    """Fails when an edit of MATRIX drops the only entry that reaches a statistics path, table kind or probe, a bit depth
    or a cell edge, or when a dense table would be wider than 512 cells (those are 4 GiB and more per frame)."""
    reached = set()
    for entry in MATRIX:
        g = matrix_gof(entry, 1)
        if refused(g.params):
            reached.add("refused")
            continue
        reached |= paths(g.params, entry[5])
        if g.params.grid_size == 1:
            reached.add("geo:g1 " + ",".join(sorted(p for p in paths(g.params, entry[5]) if p.startswith("geo:"))))
        for on, e in ((g.params.geometry_smoothing, g.params.grid_size), (g.params.color_smoothing, g.params.cgrid_size)):
            if on and not entry[5]:
                assert grid_width(g.params, e) <= 512, entry
    # g = 1 is no branch of its own: it runs the fast8 keys on a 256-wide grid and the power-of-two scan on a 512-wide one
    want = {"geo:fast8", "geo:fast8-in-generic", "geo:pow2<=8-fast2", "geo:pow2>8", "geo:npow2<=8", "geo:npow2>8",
            "geo:hashed", "geo:g1 geo:fast8-in-generic", "geo:g1 geo:pow2<=8-fast2",
            "col:fast1", "col:fast2", "col:generic", "col:hashed", "probe:fast", "probe:generic", "refused"}
    assert not want - reached, f"not reached: {sorted(want - reached)}"
    assert {e[1] for e in MATRIX} >= {8, 9, 12, 16} and {e[2] for e in MATRIX} >= {8, 9, 12, 16}
    edges = {1, 5, 7, 9, 64, 255, 256}
    assert {e[3] for e in MATRIX} >= edges and {e[4] for e in MATRIX} >= edges
    for abd in (8, 16):
        for k in range(4):
            assert {t[2][k] for t in THRESHOLDS if t[1] == abd} >= {0, 1, 65535}, (abd, k)


# ---- decisive inputs ------------------------------------------------------------------------------------------------------
A, T = 128, 20          # the luma level of the colour cells and the distance that decides (8-bit samples)


def _recolour(g, frame, rule):
    """Set the luma of every point of frame 0 by rule(boundary type, k) from the oracle's point_to_pixel."""
    for k, (x, y, m) in enumerate(frame["point_to_pixel"].tolist()):
        g.attr_y[0, m, y, x] = rule(int(frame["boundary_type"][k]), k)


def _cells_of(g, frame):
    G = smoothmodel.Grid(g.params.cgrid_size, g.params.geometry_bitdepth_3d)
    return [G.cell(tuple(p)) for p in frame["positions_presmooth"].tolist()]


def decisive_variance():
    """Type-2 lumas A - T and A + T in equal numbers per colour cell (a cell with an odd count has one A): the variance is
    exactly T^2.  Type-1 points sit at A + 3T, so a usable cell changes their colour."""
    g = set_smoothing(scaled_crowd(31, 10, 8, frames=1), None, 4, (0, 0, 255, T))
    f = oracle.reconstruct_frame(abi.GofView(g), 0)
    cells, seen, total = _cells_of(g, f), {}, {}
    for c, bt in zip(cells, f["boundary_type"].tolist()):
        if bt == 2:
            total[c] = total.get(c, 0) + 1

    def rule(bt, k):
        if bt != 2:
            return A + 3 * T
        c = cells[k]
        i = seen[c] = seen.get(c, -1) + 1
        if total[c] % 2 and i == total[c] - 1:
            return A
        return A - T if i % 2 == 0 else A + T
    _recolour(g, f, rule)
    return g


def decisive_difference():
    """Every type-2 luma is A (exact Q8 means), type-1 lumas alternate A + T and A - T: |meanY - 256 Y| = 256 T."""
    g = set_smoothing(scaled_crowd(32, 10, 8, frames=1), None, 4, (0, 0, T, 0))
    f = oracle.reconstruct_frame(abi.GofView(g), 0)
    _recolour(g, f, lambda bt, k: A if bt != 1 else (A + T if k % 2 else A - T))
    return g


def decisive_distance():
    """Crowded colours at 8 bits; t_smooth is set to a survivor's distance."""
    g = set_smoothing(scaled_crowd(33, 10, 8, frames=1), None, 4, (0, 0, 255, 255))
    m = smoothmodel.smooth_oracle_frame(g.params, oracle.reconstruct_frame(abi.GofView(g), 0))
    d = sorted(e["dist"][0] for e in m["col"].values() if e["dist"][0] > 1)
    g.params.threshold_color_smoothing = d[len(d) // 2]
    return g


def lattice_atlas(seed, edge):
    """128 x 128 at precision 1 with a hole every fifth pixel in x and y (a fifth of the points are type 1), four 64 x 64
    patches on top of each other in 3D (x, z in [128, 191]) with seeded rough depths around y = 100: thousands of type-1
    survivors per grid, each with its own weighted count and |d|^2."""
    rng = np.random.RandomState(seed)
    n, t, b, mode = synth.VIEW_AXES[1]
    W = H = 128
    patches = [(px // 16, py // 16, 4, 4, 128, 128, 0, 1, 1, n, t, b, mode, 0, 0, (0, 0))
               for py in range(0, H, 64) for px in range(0, W, 64)]
    yy, xx = np.mgrid[0:H, 0:W]
    occ = (~((xx % 5 == 2) & (yy % 5 == 2))).astype(np.uint8)[None]
    d0 = 100 + ((xx // 3 + yy // 4 + rng.randint(0, 3, (H, W))) % 12)
    geo = np.empty((1, 2, H, W), np.uint16)
    geo[0, 0] = 4 * d0
    geo[0, 1] = 4 * (d0 + rng.randint(0, 4, (H, W)))
    params = abi.Params(occupancy_resolution=16, occupancy_precision=1, geometry_bitdepth_3d=9, attribute_count=0)
    g = abi.Gof(W, H, occ, geo, None, None, None, [np.array(patches, dtype=abi.PATCH_DTYPE)], params)
    return set_smoothing(g, edge, None, (0, 0, 0, 0))


# Found by a search of lattice atlases (seeds 0-8, edges 4, 8, 16 and 32) for a type-1 point where 2 count |d|^2 + 65536 is
# an exact multiple of 262144 with a quotient >= count: seed 3, edge 8, point 19296, count 128, |d|^2 = 252672, quotient
# 247.  (An earlier search of 1 500 crowded atlases found none: their survivors have too few type-1 points each.)
GEO_EQUALITY = dict(seed=3, edge=8, threshold=247)


def decisive_geometry():
    """threshold_smoothing = 247 puts point 19296 exactly on lhs == rhs: it moves at 247, not at 248."""
    g = lattice_atlas(GEO_EQUALITY["seed"], GEO_EQUALITY["edge"])
    g.params.threshold_smoothing = GEO_EQUALITY["threshold"]
    return g


def _thr_index(what):
    return {"var": "threshold_color_variation", "diff": "threshold_color_difference", "dist": "threshold_color_smoothing",
            "geo": "threshold_smoothing"}[what]


DECISIVE = {"var": decisive_variance, "diff": decisive_difference, "dist": decisive_distance, "geo": decisive_geometry}


def decisive_hits(what, g):
    """How many comparisons of `what` fall on equality in frame 0."""
    m = smoothmodel.smooth_oracle_frame(g.params, oracle.reconstruct_frame(abi.GofView(g), 0))
    if what == "var":
        return sum(num == lim and lim > 0 for e in m["col"].values() for num, lim in e["var"])
    if what == "diff":
        return sum(dy == lim for e in m["col"].values() for dy, lim in e["diff"])
    if what == "dist":
        return sum(d == t and d > 0 for d, t in (e["dist"] for e in m["col"].values()))
    return sum(e["lhs"] == e["rhs"] for e in m["geo"].values())


def margin_atlas(gbd, edge):
    """Type-1 points on the border margin's exact coordinates along every axis.  Twelve 32 x 32 patches: for each normal
    axis a low twin pair (coordinates from 0) and a high pair (up to th - 1, past 2^gbd when th is larger); occupancy holes
    on every fourth diagonal make half of the pixels type 1 and a quarter type 2."""
    Gd = smoothmodel.Grid(edge, gbd)
    W, H, prec = 256, 96, 1
    patches = []
    slot = 0
    for proj in (0, 1, 2):
        n, t, b, mode = synth.VIEW_AXES[proj]
        for lo_hi in (0, 1):
            for twin in (0, 1):
                base = 0 if lo_hi == 0 else Gd.th - 32
                d1 = (twin if lo_hi == 0 else Gd.th - 34 - 2 * twin)
                u0, v0 = 2 * (slot % 8), 2 * (slot // 8)
                patches.append((u0, v0, 2, 2, base, base, d1, 1, 1, n, t, b, 0, 0, 0, (0, 0)))
                slot += 1
    yy, xx = np.mgrid[0:H, 0:W]
    occ = ((xx + yy) % 4 != 0).astype(np.uint8)[None]
    rng = np.random.RandomState(gbd * 1000 + edge)
    depth = yy % 32
    geo = np.empty((1, 2, H, W), np.uint16)
    geo[0, 0] = 4 * depth
    geo[0, 1] = 4 * (depth + rng.randint(0, 3, (H, W)))
    ay = rng.randint(0, 256, (1, 2, H, W)).astype(np.uint16)
    au = rng.randint(0, 256, (1, 2, H // 2, W // 2)).astype(np.uint16)
    av = rng.randint(0, 256, (1, 2, H // 2, W // 2)).astype(np.uint16)
    params = abi.Params(occupancy_resolution=16, occupancy_precision=prec, geometry_bitdepth_3d=gbd, attribute_bitdepth=8)
    g = abi.Gof(W, H, occ, geo, ay, au, av, [np.array(patches, dtype=abi.PATCH_DTYPE)], params)
    return set_smoothing(g, edge, edge, (0, 0, 255, 255))


MARGINS = [(8, 7), (9, 6), (8, 4)]


def margin_coordinates(gbd, edge):
    G = smoothmodel.Grid(edge, gbd)
    want = {G.disth - 1, G.disth, G.th - G.disth - 1, G.th - G.disth}
    if G.th > (1 << gbd):
        want.add(1 << gbd)
    return G, want


def margin_hits(g, gbd, edge):
    """{(axis, coordinate)} of type-1 points whose other two coordinates lie inside the margin."""
    G, want = margin_coordinates(gbd, edge)
    f = oracle.reconstruct_frame(abi.GofView(g), 0)
    hit = set()
    for p, bt in zip(f["positions_presmooth"].tolist(), f["boundary_type"].tolist()):
        if bt != 1:
            continue
        for a in range(3):
            if p[a] in want and all(G.disth <= p[b] and p[b] + G.disth < G.th for b in range(3) if b != a):
                hit.add((a, p[a]))
    return hit, {(a, c) for a in range(3) for c in want}


# ---- packed-sum limits --------------------------------------------------------------------------------------------------
def one_cell_atlas(W, H, occ=None, dedup_rows=0, prec=4):
    """Every point in geometry / colour cell (0,0,0) of edge 256 at bit depth 9: 128 x 128 patches (projection 1: normal y,
    tangent z, bitangent x) with u1 = v1 = 128, so x, z in [128, 255]; map 0 at y = 255, map 1 at y = 254 (the two maps
    give two points), except in the first `dedup_rows` canvas rows, where map 1 repeats map 0 (one point)."""
    n, t, b, mode = synth.VIEW_AXES[1]
    patches = []
    for py in list(range(0, H - 127, 128)) + ([H - 128] if H % 128 else []):
        for px in list(range(0, W - 127, 128)) + ([W - 128] if W % 128 else []):
            patches.append((px // 16, py // 16, 8, 8, 128, 128, 0, 1, 1, n, t, b, mode, 0, 0, (0, 0)))
    if occ is None:
        occ = np.ones((1, H // prec, W // prec), np.uint8)
    geo = np.empty((1, 2, H, W), np.uint16)
    geo[0, 0] = 4 * 255
    geo[0, 1] = 4 * 254
    geo[0, 1, :dedup_rows] = 4 * 255
    params = abi.Params(occupancy_resolution=16, occupancy_precision=prec, geometry_bitdepth_3d=9, attribute_count=0)
    g = abi.Gof(W, H, occ, geo, None, None, None, [np.array(patches, dtype=abi.PATCH_DTYPE)], params)
    return set_smoothing(g, 256, None, (0, 0, 0, 0))


def g1_atlas():
    """512 x 512: 524 288 points in one cell, offsets along y summing to 133 M >= 2^24: 256 * sum >= 2^32."""
    return one_cell_atlas(512, 512)


G2_POINTS = 15 << 20


def g2_atlas(H=2032):
    """The largest accepted atlas, 4096 x 2032 (2 W H = 16 646 144 < 2^24), with exactly 15 * 2^20 points in one cell: a
    count field narrower than 24 bits reads 0 there.  The sum of y offsets is 0.93 * 2^32."""
    W = 4096
    dedup = (2 * W * H - G2_POINTS) // W if H == 2032 else 0
    return one_cell_atlas(W, H, dedup_rows=dedup)


def type2_map(occ):
    """Boundary type 2 of every pixel of a full-resolution occupancy map (DESIGN section 5), for sizing the fixtures."""
    H, W = occ.shape
    z = np.pad(occ == 0, 2, constant_values=False)
    four = z[1:-3, 2:-2] | z[3:-1, 2:-2] | z[2:-2, 1:-3] | z[2:-2, 3:-1]
    border = np.zeros_like(occ, bool)
    border[0, :] = border[-1, :] = border[:, 0] = border[:, -1] = True
    any5 = np.zeros_like(occ, bool)
    for dy in range(5):
        for dx in range(5):
            any5 |= z[dy:dy + H, dx:dx + W]
    return (occ != 0) & ~border & ~four & any5


def c_atlas(points, variant):
    """256 x 256, holes every fifth pixel in x and y (prec 1): one colour cell of edge 256 at bit depth 9 holds `points`
    type-2 points (a type-2 pixel gives two points where map 1 differs from map 0, one elsewhere); attribute_bitdepth 16.
    variant "uv": type-2 luma 40000, U = V = 65535 (sum U = 65536 * 65535 < 2^32, sum Y >= 2^24);
    variant "y0": type-2 luma 0, U = 60000, V = 1000 (sum Y < 2^24: the 32-bit branch, whose U mean needs 64 bits).
    Type-1 lumas are 1000 / 5000, so the blend recolours them."""
    W = H = 256
    yy, xx = np.mgrid[0:H, 0:W]
    occ = ~((xx % 5 == 2) & (yy % 5 == 2))
    t2 = type2_map(occ.astype(np.uint8))
    extra = points - int(t2.sum())
    assert 0 <= extra <= int(t2.sum()), extra
    g = one_cell_atlas(W, H, occ=occ.astype(np.uint8)[None], prec=1)
    g.geo[0, 1] = 4 * 255                                     # one point per pixel ...
    ys, xs = np.nonzero(t2)
    g.geo[0, 1, ys[:extra], xs[:extra]] = 4 * 254             # ... two on the first `extra` type-2 pixels
    y2, y1, u, v = (40000, 1000, 65535, 65535) if variant == "uv" else (0, 5000, 60000, 1000)
    ay = np.where(t2, y2, y1).astype(np.uint16)
    g.attr_y = np.stack([ay, ay])[None]
    g.attr_u = np.full((1, 2, H // 2, W // 2), u, np.uint16)
    g.attr_v = np.full((1, 2, H // 2, W // 2), v, np.uint16)
    g.params.attribute_count = 1
    g.params.attribute_bitdepth = 16
    return set_smoothing(g, 256, 256, (0, 0, 65535, 0))


# ---- CPU: the model against the oracle, and the presence of every decisive and limit case ------------------------------
def _model_matches_oracle(g, frames=None):
    view = abi.GofView(g)
    for f in range(g.frame_count if frames is None else frames):
        o = oracle.reconstruct_frame(view, f)
        m = smoothmodel.smooth_oracle_frame(g.params, o)
        assert np.array_equal(np.array(m["positions"], np.int64).reshape(-1, 3), o["positions"]), f"frame {f} positions"
        if o["with_colors"]:
            assert np.array_equal(np.array(m["colors"], np.int64).reshape(-1, 3), o["colors16bit"]), f"frame {f} colours"
        assert (m["moved"], m["recoloured"]) == (o["smoothed_positions"], o["smoothed_colors"]), f"frame {f} counts"


@pytest.mark.parametrize("entry", MATRIX, ids=[e[0] for e in MATRIX])
def test_model_matches_oracle_on_the_matrix(entry):
    g = matrix_gof(entry, 1)
    if refused(g.params):
        with pytest.raises(smoothmodel.Unsupported):
            for on, e in ((g.params.geometry_smoothing, g.params.grid_size), (g.params.color_smoothing, g.params.cgrid_size)):
                if on:
                    smoothmodel.Grid(e, g.params.geometry_bitdepth_3d)
        with pytest.raises(oracle.OracleError) as e:
            oracle.reconstruct_frame(abi.GofView(g), 0)
        assert e.value.status == abi.ERR_UNSUPPORTED
        return
    _model_matches_oracle(g)


@pytest.mark.parametrize("entry", THRESHOLDS, ids=[t[0] for t in THRESHOLDS])
def test_model_matches_oracle_on_the_thresholds(entry):
    _model_matches_oracle(threshold_gof(entry, 2))


def _around(g, what, delta):
    name = _thr_index(what)
    setattr(g.params, name, getattr(g.params, name) + delta)
    return g


@pytest.mark.parametrize("what", DECISIVE)
def test_decisive_cases_hit_their_equalities(what):
    """Each decisive atlas still puts its comparison on equality, and the model equals the oracle one below, on and one
    above the threshold."""
    g = DECISIVE[what]()
    assert decisive_hits(what, g) > 0
    for delta in (-1, 0, 1):
        _model_matches_oracle(_around(DECISIVE[what](), what, delta))
    # the equality decides something: the answer on the threshold differs from the one on its strict side
    strict = {"var": -1, "diff": -1, "dist": 1, "geo": 1}[what]
    on, off = (oracle.reconstruct_frame(abi.GofView(_around(DECISIVE[what](), what, d)), 0) for d in (0, strict))
    assert (on["smoothed_positions"], on["smoothed_colors"]) != (off["smoothed_positions"], off["smoothed_colors"])


@pytest.mark.parametrize("gbd,edge", MARGINS)
def test_margin_atlas_hits_every_margin_coordinate(gbd, edge):
    g = margin_atlas(gbd, edge)
    hit, want = margin_hits(g, gbd, edge)
    assert not want - hit, f"margin coordinates not hit: {sorted(want - hit)}"
    _model_matches_oracle(g)


def test_limit_fixtures_have_their_counts():
    """G1 / G2 hold what their names promise, and the C1 / C2 colour cells hold exactly 65 536 and 65 537 type-2 points
    (counted by the model on the oracle's boundary types)."""
    g1 = oracle.reconstruct_frame(abi.GofView(g1_atlas()), 0)
    offs = g1["positions_presmooth"].astype(np.int64) % 256
    assert g1["point_count"] >= 65794 and max(offs[:, a].sum() for a in range(3)) >= 1 << 24
    g2 = g2_atlas()
    assert 2 * g2.width * g2.height < 1 << 24 <= 2 * g2.width * 2048
    assert int((g2.geo[0, 1] != g2.geo[0, 0]).sum()) + g2.width * g2.height == G2_POINTS
    assert 0.9 * 2 ** 32 < (g2.width * g2.height * 255 + int((g2.geo[0, 1] != g2.geo[0, 0]).sum()) * 254) < 2 ** 32
    for points in (65536, 65537):
        g = c_atlas(points, "uv")
        m = smoothmodel.smooth_oracle_frame(g.params, oracle.reconstruct_frame(abi.GofView(g), 0))
        assert m["type2_per_cell"] == {(0, 0, 0): points}
        assert m["recoloured"] > 0


def test_limit_cases_model_matches_oracle():
    _model_matches_oracle(g1_atlas())
    for variant in ("uv", "y0"):
        _model_matches_oracle(c_atlas(65536, variant))
    _model_matches_oracle(c_atlas(65537, "uv"))


@pytest.mark.parametrize("bd", [17, 32, 255])
def test_oracle_refuses_attribute_bitdepth_above_16(bd):
    """Samples are u16: a deeper attribute bit depth with colour smoothing on is an invalid argument, also on a frame
    without points."""
    g = set_smoothing(scaled_crowd(3, 10, 10, frames=2), 8, 4)
    g.params.attribute_bitdepth = bd
    g.patches[1] = g.patches[1][:0]
    for f in (0, 1):
        with pytest.raises(oracle.OracleError) as e:
            oracle.reconstruct_frame(abi.GofView(g), f)
        assert e.value.status == abi.ERR_INVALID_ARG
    g.params.geometry_bitdepth_3d, g.params.grid_size = 12, 1     # a refused geometry grid too: the bit depth is reported
    with pytest.raises(oracle.OracleError) as e:
        oracle.reconstruct_frame(abi.GofView(g), 0)
    assert e.value.status == abi.ERR_INVALID_ARG
    g.params.geometry_bitdepth_3d, g.params.grid_size = 10, 8
    g.params.color_smoothing = False                      # without colour smoothing the bit depth scales nothing
    oracle.reconstruct_frame(abi.GofView(g), 0)


# ---- GPU ------------------------------------------------------------------------------------------------------------------
PRE = ("positions_presmooth", "boundary_type", "partition")


def check_all_paths(ctx, g, what):
    """Every frame through the debug stage API (pre-smoothing streams, boundary types, counts, results) and the streaming
    path, against the oracle."""
    view = abi.GofView(g)
    want = [oracle.reconstruct_frame(view, f) for f in range(g.frame_count)]
    attr = g.params.attribute_count != 0
    for f in range(g.frame_count):
        got = ctx.generate_point_cloud(view, f)
        keys = PRE + (("colors16bit_presmooth",) if attr and g.params.color_smoothing else ())
        util.assert_same(got, want[f], keys=keys, what=f"{what} frame {f} pre-smoothing")
        util.assert_same(got, want[f], keys=("positions",) + (("colors16bit", "colors") if attr else ()),
                         what=f"{what} frame {f}")
        assert (got["smoothed_positions"], got["smoothed_colors"]) == \
            (want[f]["smoothed_positions"], want[f]["smoothed_colors"]), f"{what} frame {f}: counts"
    for f, fr in enumerate(ctx.decode_gof(view)):
        assert np.array_equal(fr.positions, want[f]["positions"]), f"{what} streaming frame {f}: positions"
        if attr:
            assert np.array_equal(fr.colors, want[f]["colors"]), f"{what} streaming frame {f}: colours"
        assert (fr.smoothed_positions, fr.smoothed_colors) == \
            (want[f]["smoothed_positions"], want[f]["smoothed_colors"]), f"{what} streaming frame {f}: counts"
    return want


def assert_refused(ctx, view, status):
    """Stage, streaming and resident entry points refuse the GOF with `status` before any launch."""
    for call in (lambda: ctx.generate_point_cloud(view, 0), lambda: ctx.submit_gof(view), lambda: ctx.upload_gof(view)):
        with pytest.raises(abi.Tmc2Error) as e:
            call()
        assert e.value.status == status, e.value


def _ctx_for(gpu_ctx, hashed, monkeypatch):
    from tmc2rs_b200 import codec
    if not hashed:
        return gpu_ctx
    monkeypatch.setenv("TMC2_FORCE_HASH", "1")
    return codec.Context()


@pytest.mark.gpu
@pytest.mark.parametrize("entry", MATRIX, ids=[e[0] for e in MATRIX])
def test_parameter_matrix_matches_oracle(gpu_ctx, monkeypatch, entry):
    g = matrix_gof(entry, 1)
    ctx = _ctx_for(gpu_ctx, entry[5], monkeypatch)
    try:
        if refused(g.params):
            assert_refused(ctx, abi.GofView(g), abi.ERR_UNSUPPORTED)
            with pytest.raises(oracle.OracleError) as e:
                oracle.reconstruct_frame(abi.GofView(g), 0)
            assert e.value.status == abi.ERR_UNSUPPORTED
            return
        want = check_all_paths(ctx, g, entry[0])
        assert sum(w["smoothed_positions"] + w["smoothed_colors"] for w in want) > 0, entry
    finally:
        if ctx is not gpu_ctx:
            ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("entry", THRESHOLDS, ids=[t[0] for t in THRESHOLDS])
def test_thresholds_match_oracle(gpu_ctx, entry):
    check_all_paths(gpu_ctx, threshold_gof(entry, 2), entry[0])


@pytest.mark.gpu
@pytest.mark.parametrize("delta", [-1, 0, 1], ids=["below", "on", "above"])
@pytest.mark.parametrize("what", DECISIVE)
def test_decisive_inputs_match_oracle(gpu_ctx, what, delta):
    g = _around(DECISIVE[what](), what, delta)
    check_all_paths(gpu_ctx, g, f"{what} {delta:+d}")


@pytest.mark.gpu
@pytest.mark.parametrize("gbd,edge", MARGINS)
def test_margin_coordinates_match_oracle(gpu_ctx, gbd, edge):
    want = check_all_paths(gpu_ctx, margin_atlas(gbd, edge), f"margin bd {gbd} g {edge}")
    assert want[0]["smoothed_positions"] + want[0]["smoothed_colors"] > 0


@pytest.mark.gpu
def test_g1_geometry_mean_above_32_bits(gpu_ctx):
    want = check_all_paths(gpu_ctx, g1_atlas(), "G1")
    assert want[0]["smoothed_positions"] > 0


@pytest.mark.gpu
def test_g2_largest_accepted_atlas(gpu_ctx):
    """15 * 2^20 points in one cell of a 4096 x 2032 atlas; the same content at 4096 x 2048 is refused everywhere."""
    g = g2_atlas()
    view = abi.GofView(g)
    want = oracle.reconstruct_frame(view, 0)
    assert want["point_count"] == G2_POINTS and want["smoothed_positions"] > 0
    got = gpu_ctx.generate_point_cloud(view, 0)
    util.assert_same(got, want, keys=("positions", "boundary_type"), what="G2 stage")
    assert got["smoothed_positions"] == want["smoothed_positions"]
    fr = gpu_ctx.decode_gof(view)[0]
    assert np.array_equal(fr.positions, want["positions"]) and fr.smoothed_positions == want["smoothed_positions"]
    del got, fr, want
    assert_refused(gpu_ctx, abi.GofView(g2_atlas(2048)), abi.ERR_UNSUPPORTED)


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["uv", "y0"])
def test_c1_colour_sums_at_their_limit(gpu_ctx, variant):
    want = check_all_paths(gpu_ctx, c_atlas(65536, variant), f"C1 {variant}")
    assert want[0]["smoothed_colors"] > 0


@pytest.mark.gpu
def test_c2_more_than_65536_type2_points_is_refused():
    """65 537 type-2 points in a colour cell: the launch fails with UNSUPPORTED on the stage and resident paths, the
    streaming path drops the GOF whole, and the next GOF on the context equals the oracle (its tables were reset).  The
    oracle has no such limit and answers the case."""
    from tmc2rs_b200 import codec
    bad, good = abi.GofView(c_atlas(65537, "uv")), abi.GofView(c_atlas(65536, "uv"))
    assert oracle.reconstruct_frame(bad, 0)["smoothed_colors"] > 0        # the oracle answers; the runtime refuses
    want = oracle.reconstruct_frame(good, 0)
    ctx = codec.Context(gofs_in_flight=1)
    try:
        with pytest.raises(abi.Tmc2Error) as e:
            ctx.generate_point_cloud(bad, 0)
        assert e.value.status == abi.ERR_UNSUPPORTED
        r = ctx.upload_gof(bad)
        try:
            r.reconstruct()
            with pytest.raises(abi.Tmc2Error) as e:
                r.counts()
            assert e.value.status == abi.ERR_UNSUPPORTED
        finally:
            r.free()
        ctx.submit_gof(bad)
        with pytest.raises(abi.Tmc2Error) as e:
            ctx.next_frame()
        assert e.value.status == abi.ERR_UNSUPPORTED
        assert ctx.next_frame() is None
        fr = ctx.decode_gof(good)[0]
        assert np.array_equal(fr.positions, want["positions"]) and np.array_equal(fr.colors, want["colors"])
        assert fr.smoothed_colors == want["smoothed_colors"]
        got = ctx.generate_point_cloud(good, 0)
        util.assert_same(got, want, keys=("colors16bit", "colors"), what="C1 after C2")
    finally:
        ctx.close()


@pytest.mark.gpu
def test_attribute_bitdepth_above_16_is_refused(gpu_ctx):
    """attribute_bitdepth 17 and 32 (which wrapped the 32-bit threshold scaling to 0) are invalid with colour smoothing;
    16 is accepted with every threshold at 65535 (scaled to 2^24 - 256)."""
    g = set_smoothing(scaled_crowd(3, 10, 16, frames=2), 8, 4, (65535, 65535, 65535, 65535))
    check_all_paths(gpu_ctx, g, "bit depth 16")
    g.params.threshold_color_smoothing = 256
    for bd in (17, 32):
        g.params.attribute_bitdepth = bd
        assert_refused(gpu_ctx, abi.GofView(g), abi.ERR_INVALID_ARG)
        with pytest.raises(oracle.OracleError) as e:
            oracle.reconstruct_frame(abi.GofView(g), 0)
        assert e.value.status == abi.ERR_INVALID_ARG
    # with a geometry grid wider than 1024 cells as well, both report the bit depth (the same status)
    g.params.geometry_bitdepth_3d, g.params.grid_size = 12, 1
    assert_refused(gpu_ctx, abi.GofView(g), abi.ERR_INVALID_ARG)
    with pytest.raises(oracle.OracleError) as e:
        oracle.reconstruct_frame(abi.GofView(g), 0)
    assert e.value.status == abi.ERR_INVALID_ARG
