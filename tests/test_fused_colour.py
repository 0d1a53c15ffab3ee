"""The YUV -> RGB conversion fused into the emit kernel, on the inputs where its shortcuts decide the answer.

The emit converts a point's colour from per-chroma-sample integer terms I_c = floor(255 * k_c * d) (kernels.cu
`chroma_term_fast`, 21 fractional bits; a sample it flags is recomputed by `chroma_term`, 32.32).  A warp vote
(`slot_flagged`) sends the points of flagged samples to `yuv_to_rgb_flagged`, which falls back to the reference's literal
float64 chain when 255 * Y + I_c is congruent to 0 or 1022 modulo 1023.  Only there can the float64 chain and the exact
floor disagree, and random content reaches such a point with a probability of about 2e-8, so these tests build the
points instead: for every 10-bit (U, V) pair, the Y that put each channel just above and just below a multiple of 1023.

The reference for every result is the float64 chain of codec.rs:661-687 evaluated by numpy (which never fuses a
multiply-add): r = y + 1.5748 v, g = (y - 0.18733 u) - 0.46813 v, b = y + 1.85563 u, then clamp(floor(c / 1023 * 255)).
The CPU tests check that the generated set still discriminates; the GPU tests run it through every entry point that
produces colours, and through the flat conversion kernel.
"""
import dataclasses
import functools
from fractions import Fraction

import numpy as np
import pytest

import tmc2rs_b200  # noqa: F401
from tmc2rs_b200 import abi

W = H = 1024                       # one 64 x 64-block patch, res 16, precision 4, every pixel occupied, two points each
CW, CH = W // 2, H // 2
SLOTS_PER_FRAME = 2 * CH * CW      # chroma samples of both maps of one frame

# float64 constants of codec.rs:661-687, as exact rationals
_KR, _KGU, _KGV, _KB = (Fraction(k) for k in (1.57480, 0.18733, 0.46813, 1.85563))
_DEN = max(k.denominator for k in (_KR, _KGU, _KGV, _KB))     # all powers of two
_NR, _NGU, _NGV, _NB = (int(k * _DEN) for k in (_KR, _KGU, _KGV, _KB))

# (Y, U, V) -> float64 RGB against exact RGB, found by modelling the conversion; all in the green channel
KNOWN_DECISIVE = [((5, 132, 92), (0, 68, 0), (0, 67, 0)),
                  ((241, 249, 695), (131, 50, 0), (131, 51, 0)),
                  ((336, 892, 932), (248, 16, 255), (248, 17, 255))]


@functools.lru_cache(maxsize=None)
def _term_tables():
    """Exact floor(255 * k * d) pieces for every 16-bit sample value, d = sample - 512.  Red and blue depend on one sample;
    green = floor((a(du) + b(dv)) / den) is assembled from the quotient and remainder of each half."""
    d = [s - 512 for s in range(65536)]
    ir = np.array([(255 * _NR * x) // _DEN for x in d], np.int64)
    ib = np.array([(255 * _NB * x) // _DEN for x in d], np.int64)
    qa, ra = zip(*(divmod(-255 * _NGU * x, _DEN) for x in d))
    qb, rb = zip(*(divmod(-255 * _NGV * x, _DEN) for x in d))
    return ir, ib, np.array(qa, np.int64), np.array(ra, np.int64), np.array(qb, np.int64), np.array(rb, np.int64)


def exact_terms(U, V):
    """[3, n] int64: I_r, I_g, I_b = floor(255 * k * d) in exact arithmetic on the float64 constants."""
    ir, ib, qa, ra, qb, rb = _term_tables()
    U, V = np.asarray(U, np.int64), np.asarray(V, np.int64)
    ig = qa[U] + qb[V] + (ra[U] + rb[V] >= _DEN)
    return np.stack([ir[V], ig, ib[U]])


def exact_rgb(Y, U, V):
    m = 255 * np.asarray(Y, np.int64)[:, None] + exact_terms(U, V).T
    return np.clip(m // 1023, 0, 255).astype(np.uint8)


def chain_rgb(Y, U, V):
    """The reference's float64 sequence, operation by operation."""
    y = np.asarray(Y, np.float64)
    u = np.asarray(U, np.float64) - 512.0
    v = np.asarray(V, np.float64) - 512.0
    r = y + 1.57480 * v
    g = (y - 0.18733 * u) - 0.46813 * v
    b = y + 1.85563 * u
    return np.stack([np.clip(np.floor(c / 1023.0 * 255.0), 0, 255) for c in (r, g, b)], 1).astype(np.uint8)


def _critical_y(I, side, smallest):
    """For each term I, a Y with (255 Y + I) mod 1023 in {0, 1, 2} (side 0) or {1020, 1021, 1022} (side 1).  255 and 1023
    share the factor 3, so exactly one residue of each window is reachable: t = 1020 * side + (I mod 3)."""
    t = 1020 * side + I % 3
    return smallest[(t - I) % 1023]


@functools.lru_cache(maxsize=None)
def adversarial_10bit():
    """[2^20, 8] Y for the pairs (U, V) = divmod(p, 1024): per channel one Y on each side of a multiple of 1023, then 0 and
    1023 for the clamps.  Y is the smallest one in [0, 1023] with the wanted residue."""
    p = np.arange(1 << 20)
    U, V = p >> 10, p & 1023
    I = exact_terms(U, V)
    res = (255 * np.arange(1024)) % 1023
    smallest = np.full(1023, -1, np.int64)
    for y in range(1023, -1, -1):
        smallest[res[y]] = y
    cols = [_critical_y(I[c], side, smallest) for c in range(3) for side in (0, 1)]
    Y = np.stack(cols + [np.zeros_like(U), np.full_like(U, 1023)], 1)
    return Y, U, V


@functools.lru_cache(maxsize=None)
def adversarial_16bit(n=1 << 20, seed=5):
    """n chroma samples with 16-bit (U, V), an eighth of them 10-bit, and four Y each.  Each Y puts a random one of the
    channels that a Y in 0..65535 can place on the critical residues inside the unclamped range [0, 261887] (red or blue
    when their chroma is below 512, otherwise green: large Y against large U and V, green cancellation).  No known point
    of this set separates the float64 chain from the exact floor: it guards the 32.32 terms of `chroma_term` and their
    flag margin `eps`, not a known answer."""
    rng = np.random.default_rng(seed)
    U = rng.integers(0, 65536, n)
    V = rng.integers(0, 65536, n)
    U[: n // 8] = rng.integers(0, 1024, n // 8)
    I = exact_terms(U, V)
    inv85 = pow(85, -1, 341)
    Y = np.empty((n, 4), np.int64)
    for j in range(4):
        t = 1020 * rng.integers(0, 2, (3, n)) + I % 3
        y0 = ((t - I) // 3 * inv85) % 341                # 255 Y = t - I (mod 1023)  <=>  85 Y = (t - I) / 3 (mod 341)
        m0 = 255 * y0 + I                                # the next Y with that residue is 341 higher: m grows by 85 * 1023
        lo = np.maximum(-(m0 // 86955), 0)               # m >= 0
        hi = np.minimum((261887 - m0) // 86955, (65535 - y0) // 341)
        k = lo + (rng.random((3, n)) * np.maximum(hi - lo + 1, 1)).astype(np.int64)
        ch = np.argmax(rng.random((3, n)) + (hi >= lo), 0)   # a random channel among those that can be placed
        Y[:, j] = (y0 + 341 * k)[ch, np.arange(n)]
    return Y, U, V


# ---- CPU: the generated sets still discriminate ---------------------------------------------------------------------
def test_adversarial_set_discriminates():
    Y, U, V = adversarial_10bit()
    assert np.array_equal(np.sort(U * 1024 + V), np.arange(1 << 20))          # every 10-bit pair
    assert Y.min() >= 0 and Y.max() <= 1023
    I = exact_terms(U, V)                                                      # [3, 2^20]
    rem = (255 * Y[:, :, None] + I.T[:, None, :]) % 1023                       # [pair, Y, channel]
    assert np.isin(rem, (0, 1, 2)).any(1).all(), "a (pair, channel) misses the residues just above a multiple of 1023"
    assert np.isin(rem, (1020, 1021, 1022)).any(1).all(), "a (pair, channel) misses the residues just below a multiple"
    y, u, v = Y.ravel(), np.repeat(U, 8), np.repeat(V, 8)
    chain, exact = chain_rgb(y, u, v), exact_rgb(y, u, v)
    bad = np.nonzero((chain != exact).any(1))[0]
    assert len(bad) >= 19, f"only {len(bad)} points where the float64 chain and the exact floor differ"
    got = {(int(y[i]), int(u[i]), int(v[i])): (tuple(chain[i].tolist()), tuple(exact[i].tolist())) for i in bad}
    for yuv, f64, ex in KNOWN_DECISIVE:
        assert got.get(yuv) == (f64, ex), (yuv, got.get(yuv))


def chroma_term_fast_model(U, V):
    """kernels.cu `chroma_term_fast` in numpy, 32-bit wrapping arithmetic: ([3, n] terms, flagged)."""
    u32 = lambda x: x & 0xFFFFFFFF
    s32 = lambda x: np.where(x >= 1 << 31, x - (1 << 32), x)
    du, dv = u32(np.asarray(U, np.int64) - 512), u32(np.asarray(V, np.int64) - 512)
    M = (1 << 21) - 1
    sr, sb, sg = u32(1203765 * dv), u32(389336 * du), u32(-1613024 * du - 782552 * dv)
    ir = s32(u32(401 * dv)) + (s32(sr) >> 21)
    ib = s32(u32(473 * du)) + (s32(sb) >> 21)
    ig = s32(u32(-47 * du - 119 * dv)) + (s32(sg) >> 21)
    near = (((sr & M) + 264) & M < 528) | (((sb & M) + 264) & M < 528) | (((sg & M) + 520) & M < 1040)
    return np.stack([ir, ig, ib]), near | ((np.asarray(U) | np.asarray(V)) > 1023)


def test_fast_chroma_terms_exact_unless_flagged():
    """The 21-bit terms on all 2^20 10-bit pairs: equal to the exact terms wherever they do not flag themselves, flagged
    for 4 603 pairs (44 in 10 000) and for every neutral component."""
    p = np.arange(1 << 20)
    U, V = p >> 10, p & 1023
    terms, flagged = chroma_term_fast_model(U, V)
    wrong = (terms != exact_terms(U, V)).any(0) & ~flagged
    assert not wrong.any(), f"unflagged wrong terms at (U, V) = {list(zip(U[wrong][:5], V[wrong][:5]))}"
    assert flagged[(U == 512) | (V == 512)].all()
    assert flagged.sum() == 4603, flagged.sum()


def test_16bit_set_lands_on_critical_residues():
    Y, U, V = adversarial_16bit()
    assert Y.min() >= 0 and Y.max() <= 65535 and (U < 1024).mean() > 0.12
    m = 255 * Y[:, :, None] + exact_terms(U, V).T[:, None, :]
    crit = np.isin(m % 1023, (0, 1, 2, 1020, 1021, 1022)) & (m >= 0) & (m <= 261887)
    assert crit.any(2).all(), "a Y of the 16-bit set puts no channel on a critical residue"
    # green cancellation: 16-bit Y, U and V with the green channel still inside its unclamped range
    g_in = crit[:, :, 1] & (Y >= 32768) & (U[:, None] >= 32768) & (V[:, None] >= 32768)
    assert g_in.sum() > 1000, g_in.sum()


# ---- the atlas ------------------------------------------------------------------------------------------------------
def _point_order():
    """(y, x, map) of the points of a frame in emission order: blocks in raster order, pixels in raster order inside a
    block, map 0 before map 1 (codec.rs:371-384, :422-428)."""
    by, bx, v1, u1, m = np.meshgrid(np.arange(64), np.arange(64), np.arange(16), np.arange(16), np.arange(2), indexing="ij")
    return (by * 16 + v1).ravel(), (bx * 16 + u1).ravel(), m.ravel()


def _atlas(sU, sV, sY):
    """A GOF whose chroma sample s (frame, map, row, column in C order) carries (sU[s], sV[s]) and whose 2 x 2 luma pixels
    carry sY[s]; returns the GOF and the (Y, U, V) of every point, [F, 2 W H, 3], in emission order."""
    F = len(sU) // SLOTS_PER_FRAME
    au = sU.reshape(F, 2, CH, CW).astype(np.uint16)
    av = sV.reshape(F, 2, CH, CW).astype(np.uint16)
    ay = sY.reshape(F, 2, CH, CW, 2, 2).transpose(0, 1, 2, 4, 3, 5).reshape(F, 2, H, W).astype(np.uint16)
    occ = np.ones((F, H // 4, W // 4), np.uint8)
    geo = np.empty((F, 2, H, W), np.uint16)
    geo[:, 0], geo[:, 1] = 4 * 10, 4 * 11                  # absolute D1, map 1 one deeper: two points per pixel
    patch = np.zeros(1, abi.PATCH_DTYPE)
    patch["size_u0"] = patch["size_v0"] = 64
    patch["lod_x"] = patch["lod_y"] = 1
    patch["normal_axis"], patch["tangent_axis"], patch["bitangent_axis"] = 0, 2, 1
    g = abi.Gof(W, H, occ, geo, ay, au, av, [patch.copy() for _ in range(F)], abi.Params())
    y, x, m = _point_order()
    yuv = np.stack([np.stack([ay[f, m, y, x], au[f, m, y >> 1, x >> 1], av[f, m, y >> 1, x >> 1]], 1) for f in range(F)])
    return g, yuv


@functools.lru_cache(maxsize=None)
def atlas_10bit():
    """Four frames; every pair twice.  Pair p's first sample is chroma slot p (frames 0-1) with Y 0-3 of its eight, the
    second lies in frames 2-3 on the other map, 9 samples further right and down (another block, another term-table
    entry) with Y 4-7."""
    Y, U, V = adversarial_10bit()
    p = np.arange(1 << 20)
    f, m, cy, cx = p >> 19, (p >> 18) & 1, (p >> 9) & 511, p & 511
    second = ((((f + 2) * 2 + (1 - m)) * CH + (cy + 9) % CH) * CW + (cx + 9) % CW)
    n = 4 * SLOTS_PER_FRAME
    sU, sV, sY = np.empty(n, np.int64), np.empty(n, np.int64), np.empty((n, 4), np.int64)
    sU[p], sV[p], sY[p] = U, V, Y[:, :4]
    sU[second], sV[second], sY[second] = U, V, Y[:, 4:]
    return _expected(*_atlas(sU, sV, sY))


@functools.lru_cache(maxsize=None)
def atlas_16bit():
    Y, U, V = adversarial_16bit(2 * SLOTS_PER_FRAME)
    return _expected(*_atlas(U, V, Y))


def _expected(g, yuv):
    want = np.stack([chain_rgb(*yuv[f].T) for f in range(len(yuv))])
    return g, yuv, want


ATLASES = {"10bit": atlas_10bit, "16bit": atlas_16bit}


def check_colours(got, want, yuv, what):
    assert got.shape == want.shape, f"{what}: {got.shape} != {want.shape}"
    bad = np.nonzero((got != want).any(1))[0]
    if len(bad):
        first = [f"(Y, U, V) = {tuple(yuv[i].tolist())}: got {tuple(got[i].tolist())}, want {tuple(want[i].tolist())}"
                 for i in bad[:5]]
        raise AssertionError(f"{what}: {len(bad)} of {len(want)} colours differ; " + "; ".join(first))


# ---- GPU ----------------------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def _positions(name):
    """Positions of every frame (the geometry is the same in all of them), from the oracle, whose colours must equal the
    numpy chain too."""
    from oracle import oracle
    g, yuv, want = ATLASES[name]()
    o = oracle.reconstruct_frame(abi.GofView(g), 0)
    assert o["point_count"] == 2 * W * H
    assert np.array_equal(o["colors16bit"], yuv[0])
    check_colours(o["colors"], want[0], yuv[0], f"{name}: oracle, frame 0")
    return o["positions"]


def _with(g, **params):
    return dataclasses.replace(g, params=dataclasses.replace(g.params, **params))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ATLASES)
def test_stage_api_debug(gpu_ctx, name):
    """The debug instantiation; its `colors16bit` must be the samples of the planes."""
    g, yuv, want = ATLASES[name]()
    view = abi.GofView(g)
    pos = _positions(name)
    for f in range(len(yuv)):
        got = gpu_ctx.generate_point_cloud(view, f, debug=True)
        assert got["point_count"] == len(yuv[f])
        assert np.array_equal(got["colors16bit"], yuv[f]), f"{name}: frame {f} colors16bit"
        assert np.array_equal(got["positions"], pos), f"{name}: frame {f} positions"
        check_colours(got["colors"], want[f], yuv[f], f"{name}: stage API debug, frame {f}")


@pytest.mark.gpu
@pytest.mark.parametrize("name", ATLASES)
@pytest.mark.parametrize("path", ["stage", "streaming", "geo-smoothing-g8", "geo-smoothing-g6", "resident"])
def test_production_paths(gpu_ctx, name, path):
    """The non-debug instantiations: plain (stage API without debug streams, streaming, resident) and, with geometry
    smoothing on and colour smoothing off, the fast (grid 8) and generic (grid 6) smoothing emits."""
    g, yuv, want = ATLASES[name]()
    pos = _positions(name)
    F = len(yuv)
    smoothing = path.startswith("geo-smoothing")
    if smoothing:
        g = _with(g, geometry_smoothing=True, color_smoothing=False, grid_size=int(path[-1]))
    view = abi.GofView(g)
    if path == "stage":
        frames = [gpu_ctx.generate_point_cloud(view, f, debug=False) for f in range(F)]
        frames = [(fr["point_count"], fr["positions"], fr["colors"], fr["smoothed_colors"]) for fr in frames]
    elif path == "resident":
        r = gpu_ctx.upload_gof(view)
        try:
            r.reconstruct()
            counts = r.counts()
            frames = [(int(counts[f]),) + r.fetch(f, int(counts[f])) + (0,) for f in range(F)]
        finally:
            r.free()
    else:
        frames = [(len(fr), fr.positions, fr.colors, fr.smoothed_colors) for fr in gpu_ctx.decode_gof(view)]
    for f, (n, p, c, smoothed_colors) in enumerate(frames):
        assert n == len(yuv[f]), f"{name} {path}: frame {f} has {n} points"
        assert smoothed_colors == 0
        if not smoothing:
            assert np.array_equal(p, pos), f"{name} {path}: frame {f} positions"
        check_colours(c, want[f], yuv[f], f"{name} {path}: frame {f}")


@pytest.mark.gpu
@pytest.mark.parametrize("name", ATLASES)
def test_flat_conversion_kernel(gpu_ctx, name):
    _, yuv, want = ATLASES[name]()
    flat = yuv.reshape(-1, 3)
    check_colours(gpu_ctx.convert_yuv16_to_rgb8(flat), want.reshape(-1, 3), flat, f"{name}: convert_yuv16_to_rgb8")
