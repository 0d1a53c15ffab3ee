"""Seeded synthetic decoded planes + patch/atlas metadata at the codec boundary (SURVEY.md section 8d).

The reference ships no bitstream, YUV or PLY fixture, and neither rustc nor ffmpeg exist in this image, so every
BASELINE config is fed with synthetic data of the named atlas shape:

* patches: random guillotine partition of the occupancy-block grid into rectangles of 2..12 x 2..12 blocks, ~10 % of
  them dropped (=> ~90 % canvas coverage), plus ~10 % extra patches that overlap earlier ones by 1..3 blocks
  (exercises the block-to-patch precedence of src/codec.rs:242-244); orientation Default/Swap; projection 0..5;
* occupancy (low-res u8): one ellipse per primary rectangle at occupancy-precision granularity, values drawn from
  {1, 255, random 1..255} (the reference tests ``!= 0``, src/codec.rs:393-396);
* geometry Y (u16): map0 = 4*d0 + U{0..3}, map1 = 4*(d0+delta) + U{0..3}, delta = 0 w.p. 0.4 (duplicate-skip path,
  src/codec.rs:421-428) else U{1..4}; depth is sample/4 (src/codec.rs:534,548);
* attribute YUV 4:2:0 u16 in [0, 1023]: low-frequency gradient + noise, extreme values seeded in so that both clamps of
  src/codec.rs:663-671 are hit.

Randomness is a counter-based SplitMix64 (vectorised), seed = 0x7C2D5EED + 1000*config + frame, so the same arrays
come out on every machine and numpy version.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, Tuple

import numpy as np

from .abi import Gof, Params, PATCH_DTYPE, ORIENT_DEFAULT, ORIENT_SWAP

BASE_SEED = 0x7C2D5EED
_M64 = np.uint64(0xFFFFFFFFFFFFFFFF)

# projection_id -> (normal, tangent, bitangent, projection_mode): Patch::set_view_id, src/decoder.rs:788-796
VIEW_AXES = {0: (0, 2, 1, 0), 1: (1, 2, 0, 0), 2: (2, 0, 1, 0), 3: (0, 2, 1, 1), 4: (1, 2, 0, 1), 5: (2, 0, 1, 1)}


def splitmix64(x: np.ndarray) -> np.ndarray:
    with np.errstate(over="ignore"):
        z = (x + np.uint64(0x9E3779B97F4A7C15)) & _M64
        z = ((z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)) & _M64
        z = ((z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)) & _M64
        return z ^ (z >> np.uint64(31))


class Rng:
    """Counter-based stream: value i of stream s is splitmix64(splitmix64(seed + s) + i)."""

    def __init__(self, seed: int):
        self.seed = np.uint64(seed & 0xFFFFFFFFFFFFFFFF)
        self._stream = 0

    def _key(self) -> np.uint64:
        self._stream += 1
        with np.errstate(over="ignore"):
            return splitmix64(np.array([self.seed + np.uint64(self._stream)], dtype=np.uint64))[0]

    def u64(self, n) -> np.ndarray:
        shape = (n,) if np.isscalar(n) else tuple(n)
        cnt = int(np.prod(shape))
        with np.errstate(over="ignore"):
            v = splitmix64(self._key() + np.arange(cnt, dtype=np.uint64))
        return v.reshape(shape)

    def integers(self, lo: int, hi: int, n) -> np.ndarray:
        """uniform int64 in [lo, hi] (inclusive)."""
        span = np.uint64(hi - lo + 1)
        return ((self.u64(n) >> np.uint64(11)) % span).astype(np.int64) + lo

    def uniform(self, n) -> np.ndarray:
        return (self.u64(n) >> np.uint64(11)).astype(np.float64) * (1.0 / (1 << 53))

    def randint(self, lo: int, hi: int) -> int:
        return int(self.integers(lo, hi, 1)[0])


@dataclass
class SynthConfig:
    name: str
    width: int
    height: int
    frames: int
    bitdepth_3d: int = 10
    occupied_ratio: float = 0.48
    depth_max: int = 250           # d0 range [0, depth_max]; samples are 4*d + noise
    config_id: int = 1
    occupancy_resolution: int = 16
    occupancy_precision: int = 4
    absolute_d1: bool = True
    geometry_smoothing: bool = False
    color_smoothing: bool = False
    orientations: Tuple[int, ...] = (ORIENT_DEFAULT, ORIENT_SWAP)


# BASELINE.json configs (SURVEY.md 8d)
def config(name: str, frames: int | None = None) -> SynthConfig:
    table = {
        "c1": SynthConfig("c1", 1024, 1024, 1, 10, 0.48, 250, 1),
        "c2": SynthConfig("c2", 1024, 1024, 32, 10, 0.48, 250, 2, geometry_smoothing=True, color_smoothing=True),
        "c3": SynthConfig("c3", 1280, 1344, 32, 10, 0.40, 250, 3, geometry_smoothing=True, color_smoothing=True),
        "c4": SynthConfig("c4", 2048, 2048, 8, 11, 0.60, 500, 4, geometry_smoothing=True, color_smoothing=True),
        "tiny": SynthConfig("tiny", 128, 96, 2, 10, 0.5, 250, 9),
        "small": SynthConfig("small", 256, 256, 3, 10, 0.48, 250, 8),
    }
    c = table[name]
    if frames is not None:
        c = SynthConfig(**{**c.__dict__, "frames": frames})
    return c


def _guillotine(rng: Rng, bw: int, bh: int, max_side: int = 12, min_side: int = 2) -> List[Tuple[int, int, int, int]]:
    """Split the bw x bh block grid into rectangles (x, y, w, h) with sides in [min_side, max_side] where possible."""
    out, stack = [], [(0, 0, bw, bh)]
    while stack:
        x, y, w, h = stack.pop()
        if w <= max_side and h <= max_side:
            # occasionally split further for size variety
            if (w >= 2 * min_side or h >= 2 * min_side) and rng.randint(0, 3) == 0:
                pass
            else:
                out.append((x, y, w, h))
                continue
        split_w = (w > h) if (w > max_side or h > max_side) else (rng.randint(0, 1) == 0)
        if split_w and w >= 2 * min_side:
            c = rng.randint(min_side, w - min_side)
            stack.append((x, y, c, h)); stack.append((x + c, y, w - c, h))
        elif h >= 2 * min_side:
            c = rng.randint(min_side, h - min_side)
            stack.append((x, y, w, c)); stack.append((x, y + c, w, h - c))
        elif w >= 2 * min_side:
            c = rng.randint(min_side, w - min_side)
            stack.append((x, y, c, h)); stack.append((x + c, y, w - c, h))
        else:
            out.append((x, y, w, h))
    out.sort(key=lambda r: (r[1], r[0]))
    return out


def _make_patch(rng: Rng, rect, orientation: int, bitdepth: int, res: int, depth_max: int) -> tuple:
    x, y, w, h = rect
    proj = rng.randint(0, 5)
    normal, tangent, bitangent, mode = VIEW_AXES[proj]
    if orientation == ORIENT_SWAP:      # canvas x runs along v, canvas y along u (src/decoder.rs:865)
        size_u0, size_v0 = h, w
    else:
        size_u0, size_v0 = w, h
    maxc = 1 << bitdepth
    u1 = rng.randint(0, max(0, maxc - res * size_u0 - 1))
    v1 = rng.randint(0, max(0, maxc - res * size_v0 - 1))
    kmax = max(1, (maxc - depth_max - 16) // 16)
    k = rng.randint(0, kmax - 1)
    d1 = 16 * k if mode == 0 else maxc - 16 * k
    return (x, y, size_u0, size_v0, u1, v1, d1, 1, 1, normal, tangent, bitangent, mode, orientation, 0, (0, 0))


def make_frame(cfg: SynthConfig, frame: int):
    """Returns (occ u8 [oh,ow], geo u16 [2,H,W], attr_y [2,H,W], attr_u [2,H/2,W/2], attr_v, patches PATCH_DTYPE[])."""
    W, H, res, prec = cfg.width, cfg.height, cfg.occupancy_resolution, cfg.occupancy_precision
    rng = Rng(BASE_SEED + 1000 * cfg.config_id + frame)
    bw, bh = W // res, H // res
    ow, oh = W // prec, H // prec
    rects = _guillotine(rng, bw, bh)
    keep = rng.uniform(len(rects)) < 0.90
    primary = [r for r, k in zip(rects, keep) if k] or rects[:1]
    patches, footprint = [], []
    orient_pick = rng.integers(0, len(cfg.orientations) - 1, len(primary) * 2 + 8)
    for i, r in enumerate(primary):
        o = cfg.orientations[int(orient_pick[i])]
        patches.append(_make_patch(rng, r, o, cfg.bitdepth_3d, res, cfg.depth_max)); footprint.append(r)
    # ~10 % extra patches overlapping an earlier one by 1..3 blocks
    n_extra = max(1, len(primary) // 10)
    for j in range(n_extra):
        bx, by, w0, h0 = primary[rng.randint(0, len(primary) - 1)]
        w, h = rng.randint(2, 6), rng.randint(2, 6)
        ov = rng.randint(1, 3)
        if rng.randint(0, 1) == 0:
            x, y = bx + w0 - ov, by + rng.randint(0, max(0, h0 - 1))
        else:
            x, y = bx + rng.randint(0, max(0, w0 - 1)), by + h0 - ov
        x = min(max(x, 0), bw - 1); y = min(max(y, 0), bh - 1)
        w = min(w, bw - x); h = min(h, bh - y)
        o = cfg.orientations[int(orient_pick[len(primary) + j])]
        patches.append(_make_patch(rng, (x, y, w, h), o, cfg.bitdepth_3d, res, cfg.depth_max)); footprint.append((x, y, w, h))
    patch_arr = np.array(patches, dtype=PATCH_DTYPE)

    # ---- per-primary-rectangle parameter maps at low (occupancy) resolution ---------------------------------------
    s = res // prec if res % prec == 0 else 1
    nrect = len(primary)
    rect_id = np.full((oh, ow), -1, dtype=np.int32)
    for i, (x, y, w, h) in enumerate(primary):
        rect_id[y * s:(y + h) * s, x * s:(x + w) * s] = i
    rx = np.array([r[0] for r in primary], dtype=np.float64) * s
    ry = np.array([r[1] for r in primary], dtype=np.float64) * s
    rw = np.array([r[2] for r in primary], dtype=np.float64) * s
    rh = np.array([r[3] for r in primary], dtype=np.float64) * s
    jitter = 0.9 + 0.2 * rng.uniform(nrect)
    ax, ay = 0.5 * rw * jitter, 0.5 * rh * (1.8 - jitter)
    cx, cy = rx + 0.5 * rw, ry + 0.5 * rh
    yy, xx = np.mgrid[0:oh, 0:ow]
    rid = np.clip(rect_id, 0, None)
    e = ((xx + 0.5 - cx[rid]) / ax[rid]) ** 2 + ((yy + 0.5 - cy[rid]) / ay[rid]) ** 2
    e = np.where(rect_id >= 0, e, np.inf)
    # ellipse scale chosen so that the occupied fraction of the canvas hits the target ratio
    level = np.quantile(e, min(cfg.occupied_ratio, float((rect_id >= 0).mean()) * 0.98))
    mask = (e <= level) & (rect_id >= 0)
    vals_kind = rng.integers(0, 2, (oh, ow))
    vals_rand = rng.integers(1, 255, (oh, ow)).astype(np.uint8)
    occ = np.where(vals_kind == 0, 1, np.where(vals_kind == 1, 255, vals_rand)).astype(np.uint8)
    occ = np.where(mask, occ, 0).astype(np.uint8)

    # ---- geometry: smooth depth per rectangle ----------------------------------------------------------------------
    Y, X = np.mgrid[0:H, 0:W]
    rid_full = np.clip(np.repeat(np.repeat(rect_id, prec, axis=0), prec, axis=1)[:H, :W], 0, None)
    # depth slope stays around <= 1.5 units / pixel: steeper surfaces are projected onto another plane by a V-PCC
    # encoder (max gradient = 2*pi*f*amp)
    fx = (0.0008 + 0.0027 * rng.uniform(nrect))[rid_full]
    fy = (0.0008 + 0.0027 * rng.uniform(nrect))[rid_full]
    ph = (2 * np.pi * rng.uniform(nrect))[rid_full]
    mid = (0.3 + 0.4 * rng.uniform(nrect))[rid_full] * cfg.depth_max
    amp = 0.28 * cfg.depth_max
    d0 = np.clip(np.rint(mid + amp * np.sin(2 * np.pi * (fx * X + fy * Y) + ph)), 0, cfg.depth_max).astype(np.int64)
    dup = rng.uniform((H, W)) < 0.4
    delta = np.where(dup, 0, rng.integers(1, 4, (H, W)).astype(np.int64))
    geo = np.empty((2, H, W), dtype=np.uint16)
    geo[0] = (4 * d0 + rng.integers(0, 3, (H, W)).astype(np.int64)).astype(np.uint16)
    geo[1] = (4 * (d0 + delta) + rng.integers(0, 3, (H, W)).astype(np.int64)).astype(np.uint16)

    # ---- attribute YUV 4:2:0, 10-bit --------------------------------------------------------------------------------
    attr_y = np.empty((2, H, W), dtype=np.uint16)
    attr_u = np.empty((2, H // 2, W // 2), dtype=np.uint16)
    attr_v = np.empty((2, H // 2, W // 2), dtype=np.uint16)
    Yc, Xc = np.mgrid[0:H // 2, 0:W // 2]
    for m in range(2):
        base = 512 + 380 * np.sin(2 * np.pi * (X / (W * 0.37) + Y / (H * 0.53)) + 0.3 * m + 0.1 * frame)
        noise = rng.integers(0, 16, (H, W)).astype(np.int64) - 8
        attr_y[m] = np.clip(np.rint(base) + noise, 0, 1023).astype(np.uint16)
        bu = 512 + 300 * np.cos(2 * np.pi * (Xc / (W * 0.21)) + 0.2 * m)
        bv = 512 + 300 * np.sin(2 * np.pi * (Yc / (H * 0.17)) + 0.5 * m)
        attr_u[m] = np.clip(np.rint(bu) + rng.integers(0, 16, Xc.shape).astype(np.int64) - 8, 0, 1023).astype(np.uint16)
        attr_v[m] = np.clip(np.rint(bv) + rng.integers(0, 16, Xc.shape).astype(np.int64) - 8, 0, 1023).astype(np.uint16)
        # seed extremes (hits both clamps of the colour conversion) on a sparse lattice
        attr_y[m, 0::64, 0::64] = 1023; attr_y[m, 32::64, 32::64] = 0
        attr_u[m, 0::32, 0::32] = 1023; attr_u[m, 16::32, 16::32] = 0
        attr_v[m, 0::32, 16::32] = 1023; attr_v[m, 16::32, 0::32] = 0
    return occ, geo, attr_y, attr_u, attr_v, patch_arr


def make_gof(cfg: SynthConfig, first_frame: int = 0) -> Gof:
    F = cfg.frames
    W, H, prec = cfg.width, cfg.height, cfg.occupancy_precision
    occ = np.empty((F, H // prec, W // prec), dtype=np.uint8)
    geo = np.empty((F, 2, H, W), dtype=np.uint16)
    ay = np.empty((F, 2, H, W), dtype=np.uint16)
    au = np.empty((F, 2, H // 2, W // 2), dtype=np.uint16)
    av = np.empty((F, 2, H // 2, W // 2), dtype=np.uint16)
    patches = []
    for f in range(F):
        o, g, y, u, v, p = make_frame(cfg, first_frame + f)
        occ[f], geo[f], ay[f], au[f], av[f] = o, g, y, u, v
        patches.append(p)
    params = Params(occupancy_resolution=cfg.occupancy_resolution, occupancy_precision=prec,
                    absolute_d1=cfg.absolute_d1, geometry_bitdepth_3d=cfg.bitdepth_3d,
                    geometry_smoothing=cfg.geometry_smoothing, color_smoothing=cfg.color_smoothing)
    return Gof(W, H, occ, geo, ay, au, av, patches, params)


def replicate_gof(gof: Gof, frames: int) -> Gof:
    """Cycle the frames of ``gof`` to a GOF of ``frames`` frames (cheap way to build long sequences)."""
    idx = [i % gof.frame_count for i in range(frames)]
    return gof.subset(idx)


def kat_appendix_c() -> Gof:
    """The hand-derived known-answer atlas of SURVEY.md Appendix C (32x16, two patches)."""
    W, H = 32, 16
    occ = np.zeros((1, 4, 8), dtype=np.uint8)
    occ[0, 0, 0] = 1
    occ[0, 1, 4] = 255
    Y, X = np.mgrid[0:H, 0:W]
    geo = np.empty((1, 2, H, W), dtype=np.uint16)
    geo[0, 0] = 4 * (X + Y) + 3
    geo[0, 1] = 4 * (X + Y + (X & 1))
    ay = np.full((1, 2, H, W), 512, dtype=np.uint16)
    au = np.full((1, 2, H // 2, W // 2), 512, dtype=np.uint16)
    av = np.full((1, 2, H // 2, W // 2), 512, dtype=np.uint16)
    patches = np.zeros(2, dtype=PATCH_DTYPE)
    patches[0] = (0, 0, 1, 1, 100, 200, 16, 1, 1, 0, 2, 1, 0, ORIENT_DEFAULT, 0, (0, 0))
    patches[1] = (1, 0, 1, 1, 10, 20, 1024 - 64, 1, 1, 1, 2, 0, 1, ORIENT_SWAP, 0, (0, 0))
    return Gof(W, H, occ, geo, ay, au, av, [patches], Params())


def to_device(gof: Gof, device, pad: int = 0, p010: bool = False, seed: int = 0, offset: int = 0) -> Gof:
    """Device copy of a host GOF as torch CUDA tensors, the way a GPU video decoder would hand its planes over.

    pad: extra samples at the end of every row (row pitch = width + pad); offset: the planes start `offset` samples into
    their allocation (a base address that is not 16-byte aligned).  p010: 16-bit samples become ``v << 6`` with seeded noise
    in the low 6 bits, and U / V are interleaved into one [F, 2, H/2, W] plane (NVDEC / ffmpeg ``p010le``); 16-bit planes
    are int16 tensors (torch has no full uint16 support), read bit for bit as u16."""
    import torch
    gen = torch.Generator(device=device)
    gen.manual_seed(seed)

    def put(a: np.ndarray, shift: bool):
        lead, w = a.shape[:-1], a.shape[-1]
        n = int(np.prod(lead)) * (w + pad)
        store = torch.zeros(n + offset, dtype=torch.int16 if a.itemsize == 2 else torch.uint8, device=device)
        t = store[offset:].view(*lead, w + pad)[..., :w]
        host = a.view(np.int16) if a.itemsize == 2 else a
        if shift:
            host = (a.astype(np.uint16) << 6).view(np.int16)
        t.copy_(torch.from_numpy(np.ascontiguousarray(host)).to(device))
        if shift:
            t |= torch.randint(0, 64, t.shape, generator=gen, device=device, dtype=torch.int16)
        return t

    if gof.attr_y is None:
        ay = au = av = None
    elif p010:
        uv = np.empty(gof.attr_u.shape[:-1] + (2 * gof.attr_u.shape[-1],), np.uint16)
        uv[..., 0::2], uv[..., 1::2] = gof.attr_u, gof.attr_v
        ay, au, av = put(gof.attr_y, True), put(uv, True), None
    else:
        ay, au, av = put(gof.attr_y, False), put(gof.attr_u, False), put(gof.attr_v, False)
    return Gof(gof.width, gof.height, put(gof.occ, False), put(gof.geo, p010), ay, au, av, gof.patches, gof.params,
               gof.geo_video_frames, gof.attr_video_frames, "p010" if p010 else "planar")
