"""Shared helpers for the tests: small random GOFs exercising every orientation / mode."""
import numpy as np

import tmc2rs_b200  # noqa: F401
from tmc2rs_b200 import abi, synth


def random_small_gof(seed, W=64, H=48, frames=1, orientations=(0, 1), spec=False, absolute_d1=True, res=16, prec=4,
                     n_patches=5, attr=True, depth_max=250, extreme=False, slack=(0, 0), slack_fill=0):
    """A small atlas with random (possibly overlapping) patches of the given orientations.

    The occupancy video is ceil(W / prec) x ceil(H / prec) samples, plus `slack` = (columns, rows) more filled with
    `slack_fill`: a decoder's occupancy video may be larger than the atlas needs, and those samples are not image.  W and
    H may be odd (then without attributes: 4:2:0 planes need even sizes).

    Patch placement keeps every pixel of every patch inside the canvas under the chosen orientation mode (in REFERENCE
    mode the rotated orientations use the reference's un-scaled sizes, so their pixel footprint differs from the block
    footprint -- the generator checks the four corners exactly like the reference's asserts would)."""
    rng = np.random.RandomState(seed)
    bw, bh = W // res, H // res
    sscale = res if spec else 1
    patch_lists = []
    for f in range(frames):
        plist = []
        tries = 0
        while len(plist) < n_patches and tries < 2000:
            tries += 1
            o = int(orientations[rng.randint(len(orientations))])
            su, sv = int(rng.randint(1, max(2, bw))), int(rng.randint(1, max(2, bh)))
            u0, v0 = int(rng.randint(0, bw)), int(rng.randint(0, bh))
            proj = int(rng.randint(6))
            n, t, b, mode = synth.VIEW_AXES[proj]
            if extreme and rng.randint(3) == 0:
                d1 = int(rng.randint(0, 200))          # exercises max(d1, depth) - depth clamping / small values
                u1, v1 = int(rng.randint(65000, 65536)), int(rng.randint(0, 70000))   # u16 truncation
            else:
                d1 = int(16 * rng.randint(0, 40)) if mode == 0 else 1024 - int(16 * rng.randint(0, 40))
                u1, v1 = int(rng.randint(0, 700)), int(rng.randint(0, 700))
            p = dict(u0=u0, v0=v0, size_u0=su, size_v0=sv, patch_orientation=o)
            ok = True
            for cu in (0, su - 1):
                for cv in (0, sv - 1):
                    x, y = _helper(p, cu, cv, 1, 1)
                    ok &= 0 <= x < bw and 0 <= y < bh
            for cu in (0, su * res - 1):
                for cv in (0, sv * res - 1):
                    x, y = _helper(p, cu, cv, res, sscale)
                    ok &= 0 <= x < W and 0 <= y < H
            if not ok:
                continue
            lod = (1, 1) if not extreme else (int(rng.randint(1, 3)), int(rng.randint(1, 3)))
            plist.append((u0, v0, su, sv, u1, v1, d1, lod[0], lod[1], n, t, b, mode, o, 0, (0, 0)))
        patch_lists.append(np.array(plist, dtype=abi.PATCH_DTYPE))
    oh, ow = -(-H // prec), -(-W // prec)
    occ = (rng.rand(frames, oh, ow) < 0.6).astype(np.uint8) * rng.randint(1, 256, (frames, oh, ow)).astype(np.uint8)
    if slack != (0, 0):
        occ = np.pad(occ, ((0, 0), (0, slack[1]), (0, slack[0])), constant_values=slack_fill)
    d0 = rng.randint(0, depth_max, (frames, H, W))
    delta = np.where(rng.rand(frames, H, W) < 0.4, 0, rng.randint(1, 5, (frames, H, W)))
    geo = np.empty((frames, 2, H, W), np.uint16)
    geo[:, 0] = 4 * d0 + rng.randint(0, 4, (frames, H, W))
    geo[:, 1] = 4 * (d0 + delta) + rng.randint(0, 4, (frames, H, W))
    if extreme:
        geo[:, :, ::7, ::5] = 65535
    if attr:
        hi = 65536 if extreme else 1024
        ay = rng.randint(0, hi, (frames, 2, H, W)).astype(np.uint16)
        au = rng.randint(0, hi, (frames, 2, H // 2, W // 2)).astype(np.uint16)
        av = rng.randint(0, hi, (frames, 2, H // 2, W // 2)).astype(np.uint16)
    else:
        ay = au = av = None
    params = abi.Params(occupancy_resolution=res, occupancy_precision=prec, absolute_d1=absolute_d1,
                        orientation_mode=1 if spec else 0, attribute_count=1 if attr else 0)
    return abi.Gof(W, H, occ, geo, ay, au, av, patch_lists, params)


def _helper(p, u, v, res, sscale):
    u0, v0 = p["u0"] * res, p["v0"] * res
    su, sv = p["size_u0"] * sscale, p["size_v0"] * sscale
    o = p["patch_orientation"]
    if o == 0: return u + u0, v + v0
    if o == 2: return sv - 1 - v + u0, u + v0
    if o == 3: return su - 1 - u + u0, sv - 1 - v + v0
    if o == 4: return v + u0, su - 1 - u + v0
    if o == 5: return su - 1 - u + u0, v + v0
    if o == 6: return sv - 1 - v + u0, su - 1 - u + v0
    if o == 7: return u + u0, sv - 1 - v + v0
    return v + u0, u + v0


# Generator cases: every orientation of both orientation modes, precisions 1-4, resolutions 8 / 16 / 32, widths that are
# not a multiple of 64, differential D1, u16 wrap and level of detail 2 (`extreme`), and atlases without attributes.
# tests/test_emit_instantiations.py checks that they reach every emit instantiation and slot path.
CASES = [
    dict(seed=1, orientations=(0, 1)),
    dict(seed=2, orientations=(0, 1), absolute_d1=False),
    dict(seed=3, orientations=(0, 1, 8), extreme=True),
    dict(seed=4, orientations=tuple(range(9)), spec=True),
    dict(seed=5, orientations=tuple(range(9)), spec=False, n_patches=6),
    dict(seed=6, orientations=(0, 1), prec=2),
    dict(seed=7, orientations=(0, 1), prec=1, W=48, H=32),
    dict(seed=8, orientations=(0, 1, 3, 5), spec=True, res=8, prec=4, W=40, H=32),
    dict(seed=9, orientations=(0, 1), attr=False),
    dict(seed=10, orientations=tuple(range(9)), spec=True, absolute_d1=False, extreme=True),
    dict(seed=11, orientations=(0, 1), W=208, H=112, n_patches=14),
    dict(seed=12, orientations=tuple(range(9)), spec=True, W=208, H=112, n_patches=14, extreme=True),
    dict(seed=13, orientations=(0, 1), prec=3, W=48, H=48),
    dict(seed=14, orientations=(0, 1, 2, 4, 6), spec=False, res=32, W=128, H=96, prec=4),
    # level of detail 2 on the per-pixel slot path (reference-mode rotations are not block-aligned)
    dict(seed=15, orientations=tuple(range(2, 8)), extreme=True, W=96, H=64, n_patches=8),
    # no attributes on the occupancy-mask and per-pixel slot paths
    dict(seed=16, orientations=(0, 1, 2, 5), prec=2, attr=False),
]

SMOOTH_CASES = [CASES[i] for i in (0, 2, 3, 4, 5, 6, 7, 9, 11, 12, 13)]

FAST_CASES = [
    dict(seed=21, orientations=(0, 1), W=208, H=112, n_patches=14),
    dict(seed=22, orientations=tuple(range(9)), spec=True, W=208, H=112, n_patches=14),
    dict(seed=23, orientations=(0, 1, 8), extreme=True, W=96, H=64, n_patches=8),
    dict(seed=24, orientations=(0, 1), prec=2, W=64, H=64),
    dict(seed=25, orientations=(0, 1), absolute_d1=False, W=96, H=64, n_patches=8),
]


def case_id(case):
    return "-".join(f"{k}{v}" for k, v in case.items() if k != "orientations")


STREAMS = ("positions","colors", "colors16bit", "partition", "point_to_pixel", "block_to_patch", "occupancy_map")


def assert_same(gpu, orc, keys=STREAMS, what=""):
    assert gpu["point_count"] == orc["point_count"], f"{what}: point count {gpu['point_count']} != {orc['point_count']}"
    for k in keys:
        a, b = np.asarray(gpu[k]), np.asarray(orc[k])
        if b.size == 0 and a.size == 0:
            continue
        assert a.shape == b.shape, f"{what}: {k} shape {a.shape} != {b.shape}"
        if not np.array_equal(a.astype(np.int64), b.astype(np.int64)):
            bad = np.argwhere(a.astype(np.int64) != b.astype(np.int64))
            raise AssertionError(f"{what}: {k} differs at {len(bad)} entries, first {bad[0].tolist()}: "
                                 f"gpu {a[tuple(bad[0])]} oracle {b[tuple(bad[0])]}")


def boundary_spec(occ):
    """Boundary class of every pixel of a full-resolution occupancy map (H x W, the image only), straight from the
    specification (DESIGN.md section 5): 1 = occupied on the image border or with an unoccupied 4-neighbour, 2 = another
    occupied pixel with an unoccupied pixel in its 5 x 5 window (clipped to the image), 0 = the rest."""
    occ = occ != 0
    H, W = occ.shape
    pad = np.pad(occ, 1, constant_values=False)
    four = pad[1:-1, :-2] & pad[1:-1, 2:] & pad[:-2, 1:-1] & pad[2:, 1:-1]
    border = np.zeros_like(occ)
    border[0, :] = border[-1, :] = border[:, 0] = border[:, -1] = True
    t1 = occ & (border | ~four)
    pad2 = np.pad(occ, 2, constant_values=True)
    all5 = np.ones_like(occ)
    for dy in range(5):
        for dx in range(5):
            all5 &= pad2[dy:dy + H, dx:dx + W]
    return np.where(t1, 1, np.where(occ & ~all5, 2, 0))


def crowd_into_one_region(g):
    """Rewrite a GOF in place so that its patches overlap in 3D (same axes, nearly the same offsets, slowly varying depth):
    many voxel cells then hold points of several patches, which is what triggers the smoothing filters."""
    for p in g.patches:
        n = len(p)
        p["u1"] = 100 + (np.arange(n) % 3)
        p["v1"] = 100 + (np.arange(n) % 2)
        p["lod_x"] = 1
        p["lod_y"] = 1
        p["d1"] = np.where(p["projection_mode"] == 0, 64, 1024 - 64 - 300)
        p["normal_axis"], p["tangent_axis"], p["bitangent_axis"] = 0, 2, 1
    F, _, H, W = g.geo.shape
    yy, xx = np.mgrid[0:H, 0:W]
    rng = np.random.RandomState(1234)
    d0 = 100 + ((xx // 5 + yy // 7) % 9)
    delta = np.where(rng.rand(F, H, W) < 0.4, 0, rng.randint(1, 5, (F, H, W)))
    g.geo[:, 0] = (4 * d0 + rng.randint(0, 4, (F, H, W))).astype(np.uint16)
    g.geo[:, 1] = (4 * (d0 + delta) + rng.randint(0, 4, (F, H, W))).astype(np.uint16)
    if g.attr_y is not None:                   # smooth colours with a few outliers (so that the variance test passes)
        base = (400 + 2 * (xx % 50)).astype(np.uint16)
        g.attr_y[:, :] = base
        g.attr_y[:, :, ::9, ::4] += 150
        g.attr_u[:, :] = 500
        g.attr_v[:, :] = 530
