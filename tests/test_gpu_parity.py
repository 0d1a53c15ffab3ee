"""Parity of the CUDA path (through the C ABI) against the CPU oracle.  Run on a B200: pytest -m gpu."""
import hashlib
import os

import numpy as np
import pytest

import kats
import util
from oracle import oracle
from tmc2rs_b200 import abi, codec, synth

pytestmark = pytest.mark.gpu


def both(ctx, gof, frame=0):
    view = abi.GofView(gof)
    return ctx.generate_point_cloud(view, frame), oracle.reconstruct_frame(view, frame)


def test_appendix_c_known_answer(gpu_ctx):
    g = synth.kat_appendix_c()
    got, want = both(gpu_ctx, g)
    util.assert_same(got, want, what="appendix C")
    assert got["block_to_patch"].tolist() == [1, 2] and got["point_count"] == 48
    assert got["positions"][24].tolist() == [20, 940, 14] and got["positions"][29].tolist() == [21, 938, 14]
    b2p = gpu_ctx.generate_block_to_patch_from_occupancy_map_video(abi.GofView(g), 0)
    assert b2p.tolist() == [1, 2]


@pytest.mark.parametrize("case", util.CASES, ids=util.case_id)
def test_random_small_atlases_bit_exact(gpu_ctx, case):
    g = util.random_small_gof(**case)
    got, want = both(gpu_ctx, g)
    keys = [k for k in util.STREAMS if g.params.attribute_count or k not in ("colors", "colors16bit")]
    util.assert_same(got, want, keys=keys, what=str(case))


def test_config1_full_frame_bit_exact(gpu_ctx):
    """BASELINE config 1: 1024x1024, 2 maps, precision 4, no smoothing, ~800k points."""
    g = synth.make_gof(synth.config("c1"))
    got, want = both(gpu_ctx, g)
    assert 700_000 < want["point_count"] < 900_000
    util.assert_same(got, want, what="c1")


def test_two_contexts_agree(gpu_ctx):
    """A second, independent context (own streams, own device buffers; created with the reserved legacy flag) gives the
    same frames as the session context, and both equal the oracle."""
    g = synth.make_gof(synth.config("small"))
    view = abi.GofView(g)
    ctx2 = codec.Context(two_pass_scan=True)
    try:
        for f in range(g.frame_count):
            a = gpu_ctx.generate_point_cloud(view, f)
            b = ctx2.generate_point_cloud(view, f)
            util.assert_same(a, b, what=f"second context, frame {f}")
            util.assert_same(a, oracle.reconstruct_frame(view, f), what=f"frame {f}")
    finally:
        ctx2.close()


def test_streaming_gof_in_order_and_deterministic(gpu_ctx):
    """submit_gof / next_frame: frames come back in order (src/lib.rs:81), identical on every run."""
    g = synth.make_gof(synth.config("small", frames=5))
    view = abi.GofView(g)
    first = gpu_ctx.decode_gof(view)
    second = gpu_ctx.decode_gof(view)
    assert gpu_ctx.next_frame() is None
    for f, (a, b) in enumerate(zip(first, second)):
        want = oracle.reconstruct_frame(view, f)
        assert len(a) == want["point_count"]
        assert np.array_equal(a.positions, want["positions"]) and np.array_equal(a.colors, want["colors"])
        assert np.array_equal(a.positions, b.positions) and np.array_equal(a.colors, b.colors)
        assert a.with_colors


def test_streaming_pinned_zero_staging_and_two_gofs_in_flight(gpu_ctx):
    g = synth.make_gof(synth.config("small", frames=4))
    gp = codec.pinned_copy_of(g)
    v, vp = abi.GofView(g), abi.GofView(gp)
    gpu_ctx.submit_gof(vp)
    gpu_ctx.submit_gof(v)                      # second GOF while the first is still in flight
    with pytest.raises(abi.Tmc2Error) as e:    # third one would need a third slot
        gpu_ctx.submit_gof(v)
    assert e.value.status == abi.ERR_STATE
    frames = [gpu_ctx.next_frame() for _ in range(8)]
    assert gpu_ctx.next_frame() is None
    for k, fr in enumerate(frames):
        want = oracle.reconstruct_frame(v, k % 4)
        assert np.array_equal(fr.positions, want["positions"]) and np.array_equal(fr.colors, want["colors"])


def test_resident_path_matches(gpu_ctx):
    g = synth.make_gof(synth.config("small", frames=3))
    view = abi.GofView(g)
    r = gpu_ctx.upload_gof(view)
    try:
        r.reconstruct()
        r.reconstruct()                       # relaunch on resident planes: same answer
        counts = r.counts()
        for f in range(3):
            want = oracle.reconstruct_frame(view, f)
            assert int(counts[f]) == want["point_count"]
            pos, col = r.fetch(f, int(counts[f]))
            assert np.array_equal(pos, want["positions"]) and np.array_equal(col, want["colors"])
        k, nbytes, total = gpu_ctx.last_launch_info()
        assert k >= 2 and total == int(counts.sum()) and nbytes > 0
    finally:
        r.free()


def test_color_conversion_bit_exact(gpu_ctx):
    rng = np.random.RandomState(3)
    yuv = np.concatenate([rng.randint(0, 1024, (200000, 3)), rng.randint(0, 65536, (50000, 3)),
                          [[512, 512, 512], [1023, 512, 512], [0, 512, 512], [512, 512, 1023], [0, 0, 0],
                           [1023, 1023, 1023], [65535, 0, 65535]]]).astype(np.uint16)
    got = gpu_ctx.convert_yuv16_to_rgb8(yuv)
    want = oracle.convert_yuv10_to_rgb8(yuv)
    assert np.array_equal(got, want)
    assert got[-7:].tolist() == [[127, 127, 127], [255, 255, 255], [0, 0, 0], [255, 67, 127], [0, 83, 0],
                                 [255, 171, 255], [255, 255, 255]]


def test_exhaustive_10bit_luma_chroma_slices(gpu_ctx):
    """Every (Y, V) pair at U=512 and every (Y, U) pair at V=512 for 10-bit input: 2 M colours, bit-exact."""
    y, c = np.meshgrid(np.arange(1024), np.arange(1024), indexing="ij")
    a = np.stack([y.ravel(), np.full(y.size, 512), c.ravel()], 1)
    b = np.stack([y.ravel(), c.ravel(), np.full(y.size, 512)], 1)
    yuv = np.concatenate([a, b]).astype(np.uint16)
    got = gpu_ctx.convert_yuv16_to_rgb8(yuv)
    # the oracle's scalar loop through ctypes is slow: check a strided sample exactly, and the full set by checksum of
    # a vectorised float64 numpy evaluation (numpy does not fuse multiply-add either)
    yy, uu, vv = (yuv[:, i].astype(np.float64) for i in range(3))
    r = yy + 1.57480 * (vv - 512.0)
    gg = yy - 0.18733 * (uu - 512.0) - (0.46813 * (vv - 512.0))
    bb = yy + 1.85563 * (uu - 512.0)
    want = np.stack([np.clip(np.floor(ch / 1023.0 * 255.0), 0, 255) for ch in (r, gg, bb)], 1).astype(np.uint8)
    assert np.array_equal(got, want)
    idx = np.arange(0, len(yuv), 997)
    assert np.array_equal(got[idx], oracle.convert_yuv10_to_rgb8(yuv[idx]))


@pytest.mark.parametrize("name", ["small", "c1"])
def test_smoothing_matches_own_spec_oracle(gpu_ctx, name):
    """Boundary detection + grid geometry smoothing + grid colour smoothing: the reference has only stubs for these
    (parity unpinned upstream); the CUDA kernels must equal the repository's integer spec exactly.  The +-1 report that
    north_star asks for is printed as well (expected: 0 differing points)."""
    g = synth.make_gof(synth.config(name))
    g.params.geometry_smoothing = True
    g.params.color_smoothing = True
    got, want = both(gpu_ctx, g)
    util.assert_same(got, want, keys=("positions_presmooth", "colors16bit_presmooth", "partition", "boundary_type"),
                     what=name + " pre-smoothing")
    dpos = np.abs(got["positions"].astype(int) - want["positions"].astype(int)).max(axis=1)
    dcol = np.abs(got["colors"].astype(int) - want["colors"].astype(int)).max(axis=1)
    print(f"{name}: points {want['point_count']}, moved gpu/oracle {got['smoothed_positions']}/{want['smoothed_positions']}, "
          f"recoloured {got['smoothed_colors']}/{want['smoothed_colors']}, |dpos|>0: {(dpos > 0).sum()}, "
          f"|dpos|>1: {(dpos > 1).sum()}, |dcol|>0: {(dcol > 0).sum()}, |dcol|>1: {(dcol > 1).sum()}")
    assert (dpos <= 1).all() and (dcol <= 1).all()        # north_star tolerance
    util.assert_same(got, want, keys=("positions", "colors16bit", "colors"), what=name + " smoothed")   # own spec: exact
    assert got["smoothed_positions"] == want["smoothed_positions"]
    assert got["smoothed_colors"] == want["smoothed_colors"]


def test_smoothing_golden_fixture(gpu_ctx):
    """The CUDA path against the committed smoothing fixture (tests/golden/small_smooth_f1.npz), without the oracle in between."""
    import importlib.util
    gold = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    spec = importlib.util.spec_from_file_location("make_golden", os.path.join(gold, "make_golden.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    z = np.load(os.path.join(gold, "small_smooth_f1.npz"))
    fr = gpu_ctx.decode_gof(abi.GofView(m.smoothing_case()))[1]
    sha = lambda a: hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()
    assert len(fr) == int(z["point_count"])
    assert fr.smoothed_positions == int(z["smoothed_positions"]) and fr.smoothed_colors == int(z["smoothed_colors"])
    assert sha(fr.positions) == z["sha_positions"].item() and sha(fr.colors) == z["sha_colors"].item()
    assert np.array_equal(z["moved_positions_head"], fr.positions[z["moved_index_head"]])


def test_smoothing_dense_overlap_case(gpu_ctx):
    """Patches forced into the same 3D region so that many cells hold several patches (lots of smoothing work)."""
    g = synth.make_gof(synth.config("small"))
    for p in g.patches:
        p["u1"] = 100 + (np.arange(len(p)) % 3)
        p["v1"] = 100 + (np.arange(len(p)) % 2)
        p["d1"] = np.where(p["projection_mode"] == 0, 64, 1024 - 64 - 300)
        p["normal_axis"], p["tangent_axis"], p["bitangent_axis"] = 0, 2, 1
    g.params.geometry_smoothing = True
    g.params.color_smoothing = True
    got, want = both(gpu_ctx, g, 1)
    assert want["smoothed_positions"] > 20 and want["smoothed_colors"] > 20
    util.assert_same(got, want, keys=("positions", "colors16bit", "colors", "boundary_type"), what="dense overlap")
    # streaming path with smoothing gives the same frames
    frames = gpu_ctx.decode_gof(abi.GofView(g))
    assert np.array_equal(frames[1].positions, want["positions"]) and np.array_equal(frames[1].colors, want["colors"])
    assert frames[1].smoothed_positions == want["smoothed_positions"]


@pytest.mark.parametrize("env", [{"TMC2_FORCE_HASH": "1", "TMC2_SMOOTH_GROUP": "2"}, {"TMC2_SMOOTH_GROUP": "2"},
                                 {"TMC2_TABLE_BUDGET_MB": "600"}, {"TMC2_TABLE_BUDGET_MB": "100"}],
                         ids=["hashed-groups-of-2", "dense-groups-of-2", "budget-600MB", "budget-100MB"])
def test_smoothing_hashed_tables_and_small_groups(monkeypatch, env):
    """Same answers when the voxel-cell tables are hashed (grids too large for a dense table), when a GOF is cut into frame
    groups with two alternating table sets (dense tables: the fast instantiation, as for config 4), and when the per-table
    memory budget is small (600 MB: one-frame groups; 100 MB: the colour grid no longer fits and is hashed)."""
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    g = synth.make_gof(synth.config("small", frames=5))
    for p in g.patches:
        p["u1"] = 100 + (np.arange(len(p)) % 3)
        p["v1"] = 100 + (np.arange(len(p)) % 2)
        p["d1"] = np.where(p["projection_mode"] == 0, 64, 1024 - 64 - 300)
        p["normal_axis"], p["tangent_axis"], p["bitangent_axis"] = 0, 2, 1
    g.params.geometry_smoothing = True
    g.params.color_smoothing = True
    view = abi.GofView(g)
    ctx = codec.Context()
    try:
        frames = ctx.decode_gof(view)
        frames2 = ctx.decode_gof(view)          # tables must come back clean for the next GOF
        for f in range(5):
            want = oracle.reconstruct_frame(view, f)
            for fr in (frames[f], frames2[f]):
                assert np.array_equal(fr.positions, want["positions"]) and np.array_equal(fr.colors, want["colors"])
                assert fr.smoothed_positions == want["smoothed_positions"] and fr.smoothed_colors == want["smoothed_colors"]
    finally:
        ctx.close()


def test_error_codes_where_the_reference_panics(gpu_ctx):
    g = util.random_small_gof(seed=11)
    mk = lambda **kw: abi.GofView(abi.Gof(g.width, g.height, kw.get("occ", g.occ), g.geo, g.attr_y, g.attr_u, g.attr_v,
                                          kw.get("patches", g.patches), kw.get("params", g.params),
                                          kw.get("geo_video_frames"), kw.get("attr_video_frames")))
    bad = g.patches[0].copy(); bad["u0"][0] = 1000
    cases = [(mk(patches=[bad]), abi.ERR_PATCH_OUT_OF_CANVAS), (mk(geo_video_frames=1), abi.ERR_SHORT_VIDEO),
             (mk(attr_video_frames=1), abi.ERR_SHORT_VIDEO),
             (mk(params=abi.Params(**{**g.params.__dict__, "map_count_minus1": 0})), abi.ERR_MAP_COUNT),
             (mk(params=abi.Params(**{**g.params.__dict__, "enhanced_occupancy_map": True})), abi.ERR_UNSUPPORTED),
             (mk(params=abi.Params(**{**g.params.__dict__, "occupancy_precision": 2})), abi.ERR_INVALID_ARG)]
    for view, code in cases:
        with pytest.raises(abi.Tmc2Error) as e:
            gpu_ctx.generate_point_cloud(view, 0)
        assert e.value.status == code
        with pytest.raises(abi.Tmc2Error) as e:
            gpu_ctx.submit_gof(view)
        assert e.value.status == code
    # the context is still usable afterwards
    got, want = both(gpu_ctx, g)
    util.assert_same(got, want, what="after errors")


def test_empty_and_blank_frames(gpu_ctx):
    g = util.random_small_gof(seed=12, frames=3)
    patches = [g.patches[0][:0], g.patches[1], g.patches[2]]
    occ = g.occ.copy(); occ[1] = 0
    g2 = abi.Gof(g.width, g.height, occ, g.geo, g.attr_y, g.attr_u, g.attr_v, patches, g.params)
    view = abi.GofView(g2)
    frames = gpu_ctx.decode_gof(view)
    assert len(frames[0]) == 0 and len(frames[1]) == 0
    want = oracle.reconstruct_frame(view, 2)
    assert np.array_equal(frames[2].positions, want["positions"]) and np.array_equal(frames[2].colors, want["colors"])


def test_config2_gof_properties_at_full_size(gpu_ctx):
    """BASELINE config 2 (32 frames, 1024x1024, smoothing on) through the resident path: size-independent properties
    (determinism, per-frame independence, counts) + exact oracle parity on a sample of frames."""
    cfg = synth.config("c2", frames=8)
    base = synth.make_gof(cfg)
    g = synth.replicate_gof(base, 32)          # 32 frames cycling 8 distinct ones
    view = abi.GofView(g)
    r = gpu_ctx.upload_gof(view)
    try:
        r.reconstruct()
        counts = r.counts()
        assert (counts.reshape(4, 8) == counts[:8]).all()          # replicated frames -> identical counts
        sha = lambda f: hashlib.sha256(b"".join(a.tobytes() for a in r.fetch(f, int(counts[f])))).hexdigest()
        assert sha(3) == sha(11) == sha(27)                        # frame independence inside the batch
        r.reconstruct()
        assert (r.counts() == counts).all() and sha(5) == sha(13)  # deterministic relaunch
        for f in (0, 7, 30):
            want = oracle.reconstruct_frame(view, f)
            pos, col = r.fetch(f, int(counts[f]))
            assert np.array_equal(pos, want["positions"]) and np.array_equal(col, want["colors"])
    finally:
        r.free()


@pytest.mark.parametrize("name", ["c3", "c4"])
def test_config3_config4_frame_bit_exact_with_smoothing(gpu_ctx, name):
    """BASELINE configs 3 (1280x1344, width not a power of two) and 4 (2048x2048, 11-bit geometry, ~4M points): one full-size
    frame, every stream against the oracle, smoothing on."""
    g = synth.make_gof(synth.config(name, frames=1))
    assert g.params.geometry_smoothing and g.params.color_smoothing
    got, want = both(gpu_ctx, g)
    lo, hi = (900_000, 1_300_000) if name == "c3" else (3_400_000, 4_600_000)
    assert lo < want["point_count"] < hi, want["point_count"]
    util.assert_same(got, want, what=name)
    util.assert_same(got, want, keys=("positions_presmooth", "colors16bit_presmooth", "boundary_type"), what=name + " pre-smoothing")
    assert got["smoothed_positions"] == want["smoothed_positions"] and got["smoothed_colors"] == want["smoothed_colors"]
    assert want["smoothed_positions"] > 0
    # the production instantiation (streaming path; c4: colour grid 512 cells wide, beyond the packed cell keys)
    fr = gpu_ctx.decode_gof(abi.GofView(g))[0]
    assert np.array_equal(fr.positions, want["positions"]) and np.array_equal(fr.colors, want["colors"])
    assert fr.smoothed_positions == want["smoothed_positions"] and fr.smoothed_colors == want["smoothed_colors"]


def test_three_entry_points_agree_at_full_size(gpu_ctx):
    """Size-independent property at BASELINE size: the stage API, the streaming API (pinned host planes) and the resident
    path give byte-identical frames for a C3-shaped GOF, and the frames arrive in order."""
    g = synth.replicate_gof(synth.make_gof(synth.config("c3", frames=2)), 5)
    view = abi.GofView(g)
    frames = gpu_ctx.decode_gof(view)
    assert len(frames) == 5
    r = gpu_ctx.upload_gof(view)
    try:
        r.reconstruct()
        counts = r.counts()
        for f, fr in enumerate(frames):
            assert len(fr) == counts[f]
            pos, col = r.fetch(f, int(counts[f]))
            assert np.array_equal(pos, fr.positions) and np.array_equal(col, fr.colors)
    finally:
        r.free()
    st = gpu_ctx.generate_point_cloud(view, 3, debug=False)
    assert np.array_equal(st["positions"], frames[3].positions) and np.array_equal(st["colors"], frames[3].colors)
    assert np.array_equal(frames[0].positions, frames[2].positions) and np.array_equal(frames[1].colors, frames[3].colors)


@pytest.mark.parametrize("case", util.SMOOTH_CASES, ids=util.case_id)
@pytest.mark.parametrize("grids", [(8, 4), (6, 3)], ids=["g8c4", "g6c3"])
def test_random_small_atlases_with_smoothing(gpu_ctx, case, grids):
    """Every orientation / precision / resolution / no-attribute case again with boundary detection + both smoothing stages
    on (power-of-two and non-power-of-two cell edges): all streams, pre- and post-smoothing, equal the oracle."""
    g = util.random_small_gof(**case)
    util.crowd_into_one_region(g)              # patches overlap in 3D -> multi-patch cells -> the filters have work
    g.params.geometry_smoothing = True
    g.params.color_smoothing = True
    g.params.grid_size, g.params.cgrid_size = grids
    g.params.threshold_smoothing = 4          # low thresholds: plenty of points move / get recoloured on random content
    g.params.threshold_color_smoothing = 2
    g.params.threshold_color_variation = 200
    g.params.threshold_color_difference = 200
    got, want = both(gpu_ctx, g)
    keys = [k for k in util.STREAMS if g.params.attribute_count or k not in ("colors", "colors16bit")]
    util.assert_same(got, want, keys=keys, what=str(case))
    pre = ["positions_presmooth", "boundary_type"] + (["colors16bit_presmooth"] if g.params.attribute_count else [])
    util.assert_same(got, want, keys=pre, what=str(case) + " pre-smoothing")
    assert got["smoothed_positions"] == want["smoothed_positions"] and got["smoothed_colors"] == want["smoothed_colors"]


@pytest.mark.parametrize("case", util.FAST_CASES, ids=util.case_id)
@pytest.mark.parametrize("content", ["smooth", "noisy", "asis"])
@pytest.mark.parametrize("grids", [(8, 4), (4, 2), (2, 8)], ids=["g8c4", "g4c2", "g2c8"])
def test_streaming_smoothing_fast_grids(gpu_ctx, case, content, grids):
    """The production (non-debug) smoothing instantiation for dense power-of-two grids keeps per-slot cell tables in shared
    memory: frames from submit_gof / next_frame must equal the oracle on slowly varying depth (everything lands in the
    table), on noisy depth (a slot spans more cells along the projection axis than its table holds: per-point path) and on
    the generator's own patches (level of detail 2, 16-bit wrap of the tangential coordinates: no table at all)."""
    g = util.random_small_gof(frames=2, **case)
    if content != "asis":
        geo = g.geo.copy()
        util.crowd_into_one_region(g)
        if content == "noisy":
            g.geo[:] = geo
    g.params.geometry_smoothing = True
    g.params.color_smoothing = True
    g.params.grid_size, g.params.cgrid_size = grids
    g.params.threshold_smoothing = 4
    g.params.threshold_color_smoothing = 2
    g.params.threshold_color_variation = 200
    g.params.threshold_color_difference = 200
    view = abi.GofView(g)
    frames = gpu_ctx.decode_gof(view)
    for f, fr in enumerate(frames):
        want = oracle.reconstruct_frame(view, f)
        assert len(fr) == want["point_count"]
        assert np.array_equal(fr.positions, want["positions"]), (case, content, f)
        assert np.array_equal(fr.colors, want["colors"]), (case, content, f)
        assert fr.smoothed_positions == want["smoothed_positions"] and fr.smoothed_colors == want["smoothed_colors"]


def test_row_padded_planes_like_ffmpeg_linesize(gpu_ctx):
    """Planes whose row pitch exceeds the width (libavcodec pads linesize; the reference ignores it, decoder.rs:976-978): the
    C ABI takes the pitch per plane kind and must give the same frames as tight copies, whatever sits in the padding."""
    g = util.random_small_gof(seed=31, W=208, H=112, n_patches=14, frames=2)
    util.crowd_into_one_region(g)
    g.params.geometry_smoothing = True
    g.params.color_smoothing = True
    rng = np.random.RandomState(7)

    def padded(a, pad):
        big = rng.randint(0, 256 if a.dtype == np.uint8 else 65536, a.shape[:-1] + (a.shape[-1] + pad,)).astype(a.dtype)
        big[..., :a.shape[-1]] = a
        return big[..., :a.shape[-1]]

    gp = abi.Gof(g.width, g.height, padded(g.occ, 12), padded(g.geo, 48), padded(g.attr_y, 48), padded(g.attr_u, 24),
                 padded(g.attr_v, 24), g.patches, g.params)
    vp = abi.GofView(gp)
    assert vp.c.frames[0].geo_stride == g.width + 48 and vp.c.frames[0].attr_stride_c == g.width // 2 + 24
    tight = gpu_ctx.decode_gof(abi.GofView(g))
    pad = gpu_ctx.decode_gof(vp)
    for a, b in zip(tight, pad):
        assert np.array_equal(a.positions, b.positions) and np.array_equal(a.colors, b.colors)
    want = oracle.reconstruct_frame(abi.GofView(g), 1)
    assert np.array_equal(pad[1].positions, want["positions"]) and np.array_equal(pad[1].colors, want["colors"])
    st = gpu_ctx.generate_point_cloud(vp, 1, debug=True)
    assert np.array_equal(st["positions"], want["positions"]) and np.array_equal(st["occupancy_map"], want["occupancy_map"])


def test_mixed_pinned_and_pageable_planes(gpu_ctx):
    """Pinned-ness is decided per plane on its full extent (ADVICE r1): geometry map 0 pinned, everything else pageable --
    must stage exactly the unpinned planes."""
    g = synth.make_gof(synth.config("small", frames=3))
    want = [oracle.reconstruct_frame(abi.GofView(g), f) for f in range(3)]
    F, _, H, W = g.geo.shape
    geo0 = codec.pinned_empty((F, H, W), np.uint16)                      # map 0 of every frame pinned, map 1 pageable
    geo0[...] = g.geo[:, 0]
    geo = [[geo0[f], np.ascontiguousarray(g.geo[f, 1])] for f in range(F)]
    gm = abi.Gof(g.width, g.height, g.occ, g.geo, g.attr_y, g.attr_u, g.attr_v, g.patches, g.params)
    vm = abi.GofView(gm)
    keep = []
    for f in range(F):
        for m in range(2):
            keep.append(geo[f][m])
            vm.c.frames[f].geo[m] = geo[f][m].ctypes.data
    frames = gpu_ctx.decode_gof(vm)
    for f in range(F):
        assert np.array_equal(frames[f].positions, want[f]["positions"]) and np.array_equal(frames[f].colors, want[f]["colors"])
    # all planes pinned except the chroma planes
    gp = codec.pinned_copy_of(g)
    gq = abi.Gof(g.width, g.height, gp.occ, gp.geo, gp.attr_y, g.attr_u.copy(), g.attr_v.copy(), g.patches, g.params)
    frames = gpu_ctx.decode_gof(abi.GofView(gq))
    for f in range(F):
        assert np.array_equal(frames[f].positions, want[f]["positions"]) and np.array_equal(frames[f].colors, want[f]["colors"])


def test_wait_inputs_then_overwrite_pinned_planes(gpu_ctx):
    """Input ownership (include/tmc2gpu.h, INPUT LIFETIME): after wait_inputs the caller may decode the next GOF into the
    same pinned planes; the frames of the GOF in flight must not change."""
    g = synth.make_gof(synth.config("small", frames=4))
    g2 = synth.make_gof(synth.config("small", frames=4, seed_offset=77)) if "seed_offset" in synth.config.__code__.co_varnames else None
    gp = codec.pinned_copy_of(g)
    v, vp = abi.GofView(g), abi.GofView(gp)
    want = [oracle.reconstruct_frame(v, f) for f in range(4)]
    gpu_ctx.submit_gof(vp)
    gpu_ctx.wait_inputs()
    rng = np.random.RandomState(5)
    gp.geo[...] = rng.randint(0, 1024, gp.geo.shape).astype(np.uint16)     # "decode the next GOF" into the same buffers
    gp.attr_y[...] = rng.randint(0, 1024, gp.attr_y.shape).astype(np.uint16)
    gp.occ[...] = 0
    for f in range(4):
        fr = gpu_ctx.next_frame()
        assert np.array_equal(fr.positions, want[f]["positions"]) and np.array_equal(fr.colors, want[f]["colors"])
    assert gpu_ctx.next_frame() is None


def test_rejected_inputs_odd_size_and_degenerate_axes(gpu_ctx):
    """ADVICE r1: odd width / height with 4:2:0 attributes, and patches whose axes are not a permutation (the reference's
    duplicate test and differential D1 then act on an overwritten coordinate), are refused with a status code."""
    g = util.random_small_gof(seed=3, W=64, H=48)
    odd = abi.Gof(63, 48, g.occ, np.ascontiguousarray(g.geo[..., :63]), np.ascontiguousarray(g.attr_y[..., :63]),
                  np.ascontiguousarray(g.attr_u[..., :31]), np.ascontiguousarray(g.attr_v[..., :31]),
                  [p[:0] for p in g.patches], g.params)
    with pytest.raises(abi.Tmc2Error) as e:
        gpu_ctx.submit_gof(abi.GofView(odd))
    assert e.value.status == abi.ERR_INVALID_ARG
    for absolute in (False, True):
        gd = util.random_small_gof(seed=4, absolute_d1=absolute)
        for p in gd.patches:
            p["tangent_axis"] = p["normal_axis"]
        with pytest.raises(abi.Tmc2Error) as e:
            gpu_ctx.submit_gof(abi.GofView(gd))
        assert e.value.status == abi.ERR_UNSUPPORTED
        with pytest.raises(abi.Tmc2Error) as e:
            gpu_ctx.generate_point_cloud(abi.GofView(gd), 0)
        assert e.value.status == abi.ERR_UNSUPPORTED


def test_failed_gof_is_dropped_whole_and_slot_is_freed():
    """ADVICE r1: a device-side failure (here: the boundary list capacity, forced tiny) is reported once by next_frame, no frame
    of that GOF is handed out afterwards, and the GOF slot is free again."""
    import os
    g = synth.make_gof(synth.config("small", frames=3))
    g.params.geometry_smoothing = True
    g.params.color_smoothing = True
    view = abi.GofView(g)
    os.environ["TMC2_TEST_BLIST_CAP"] = "16"
    ctx = codec.Context(gofs_in_flight=1)
    try:
        ctx.submit_gof(view)
        with pytest.raises(abi.Tmc2Error):
            ctx.next_frame()
        assert ctx.next_frame() is None                                    # nothing of the failed GOF is left
        os.environ.pop("TMC2_TEST_BLIST_CAP")
        frames = ctx.decode_gof(view)          # the single slot is usable again, and smoothing on it is right
        for f, fr in enumerate(frames):
            want = oracle.reconstruct_frame(view, f)
            assert np.array_equal(fr.positions, want["positions"]) and np.array_equal(fr.colors, want["colors"]), f
            assert (fr.smoothed_positions, fr.smoothed_colors) == (want["smoothed_positions"], want["smoothed_colors"]), f
    finally:
        os.environ.pop("TMC2_TEST_BLIST_CAP", None)
        ctx.close()


@pytest.mark.parametrize("name,make", kats.ALL, ids=[n for n, _ in kats.ALL])
def test_hand_derived_kats_on_gpu(gpu_ctx, name, make):
    """The CUDA path against the hand-derived vectors of tests/kats.py (stage API and streaming API)."""
    g, want = make()
    view = abi.GofView(g)
    kats.check(gpu_ctx.generate_point_cloud(view, 0), want, name)
    fr = gpu_ctx.decode_gof(view)[0]
    assert fr.positions.tolist() == want["positions"] and (fr.colors == 127).all()


def test_device_resident_hand_off_matches_host_frames(gpu_ctx):
    """SURVEY 8f-4: a context created with TMC2_CTX_DEVICE_OUTPUT hands frames out as device pointers (no D2H copy); what
    sits behind them equals the frames of the ordinary context and the oracle."""
    import torch
    g = synth.make_gof(synth.config("small", frames=3))
    g.params.geometry_smoothing = True
    g.params.color_smoothing = True
    view = abi.GofView(g)
    host = gpu_ctx.decode_gof(view)
    dctx = codec.Context(device_output=True)

    class Dev:                                             # zero-copy torch view of a raw device range
        def __init__(self, ptr, nbytes):
            self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 2}
    try:
        dctx.submit_gof(view)
        got = [dctx.next_frame_device() for _ in range(3)]
        assert dctx.next_frame_device() is None
        for f, (n, ppos, pcol, dev, release) in enumerate(got):
            want = oracle.reconstruct_frame(view, f)
            assert n == want["point_count"] == len(host[f]) and dev == 0
            pos = torch.as_tensor(Dev(ppos, n * 6), device="cuda:0").cpu().numpy().view(np.uint16).reshape(n, 3)
            col = torch.as_tensor(Dev(pcol, n * 3), device="cuda:0").cpu().numpy().reshape(n, 3)
            assert np.array_equal(pos, want["positions"]) and np.array_equal(col, want["colors"])
            assert np.array_equal(pos, host[f].positions) and np.array_equal(col, host[f].colors)
        for *_, release in got:
            release()
        dctx.submit_gof(view)                               # the slot is free again
        assert dctx.next_frame_device()[0] == len(host[0])
    finally:
        dctx.close()


def _ply_frames(ctx, view, n, fmt, **kw):
    ctx.submit_gof(view)
    out = [ctx.next_frame_ply(fmt, **kw) for _ in range(n)]
    assert ctx.next_frame() is None
    return out


@pytest.mark.parametrize("device_output", [False, True], ids=["host-frames", "device-frames"])
def test_frame_to_ply_equals_the_reference_writer(gpu_ctx, device_output):
    """SURVEY 8f-4: tmc2gpu_frame_to_ply formats a frame on the device; the ASCII file equals, byte for byte, what the
    reference's PlyWriter (src/writer.rs:24-75, restated in tmc2rs_b200/ply.py) writes for the oracle's PointSet3, and the
    binary_little_endian file holds the same points."""
    from tmc2rs_b200 import ply
    g = synth.make_gof(synth.config("small", frames=3))
    g.params.geometry_smoothing = True
    g.params.color_smoothing = True
    view = abi.GofView(g)
    ctx = codec.Context(device_output=True) if device_output else gpu_ctx
    try:
        asc = _ply_frames(ctx, view, 3, abi.PLY_ASCII)
        binr = _ply_frames(ctx, view, 3, abi.PLY_BINARY_LE)
        for f in range(3):
            want = oracle.reconstruct_frame(view, f)
            assert want["point_count"] > 1000
            assert asc[f] == ply.ascii_ply(want["positions"], want["colors"])
            assert binr[f] == ply.binary_ply(want["positions"], want["colors"])
            pos, col = ply.read_ply(binr[f])
            assert np.array_equal(pos, want["positions"]) and np.array_equal(col, want["colors"])
    finally:
        if device_output:
            ctx.close()


def test_frame_to_ply_digit_widths_empty_frames_no_colours_and_capacity(gpu_ctx):
    from tmc2rs_b200 import ply
    # five-digit coordinates: the differential-D1 wrap vector (positions up to 65 5xx), colours 127
    for absolute in (False, True):
        g, want = kats.d1_wrap_and_mode1_clamp(absolute)
        view = abi.GofView(g)
        pos = np.array(want["positions"], np.uint16).reshape(-1, 3)
        col = np.full((len(pos), 3), 127, np.uint8)
        assert max(len(str(v)) for v in pos.ravel().tolist()) == 5 and min(len(str(v)) for v in pos.ravel().tolist()) == 1
        assert _ply_frames(gpu_ctx, view, 1, abi.PLY_ASCII)[0] == ply.ascii_ply(pos, col)
        assert _ply_frames(gpu_ctx, view, 1, abi.PLY_BINARY_LE)[0] == ply.binary_ply(pos, col)
    # a frame without points is a header and nothing else; positions only (attribute_count == 0): three columns
    g = util.random_small_gof(seed=12, frames=3)
    occ = g.occ.copy(); occ[1] = 0
    g.params.attribute_count = 0
    g2 = abi.Gof(g.width, g.height, occ, g.geo, g.attr_y, g.attr_u, g.attr_v, [g.patches[0][:0], g.patches[1], g.patches[2]], g.params)
    view = abi.GofView(g2)
    files = _ply_frames(gpu_ctx, view, 3, abi.PLY_ASCII)
    empty = np.zeros((0, 3), np.uint16)
    assert files[0] == files[1] == ply.ascii_ply(empty, None) and b"red" not in files[0]
    want = oracle.reconstruct_frame(view, 2)
    assert files[2] == ply.ascii_ply(want["positions"], None)
    assert _ply_frames(gpu_ctx, view, 3, abi.PLY_BINARY_LE)[2] == ply.binary_ply(want["positions"], None)
    # destination too small: TMC2_ERR_CAPACITY, the frame is released all the same and the context goes on
    gpu_ctx.submit_gof(view)
    with pytest.raises(abi.Tmc2Error) as e:
        gpu_ctx.next_frame_ply(abi.PLY_ASCII, capacity=64)
    assert e.value.status == abi.ERR_CAPACITY
    assert gpu_ctx.next_frame_ply(abi.PLY_ASCII) == files[1]
    assert gpu_ctx.next_frame_ply(abi.PLY_ASCII, capacity=len(files[2])) == files[2]
    assert gpu_ctx.next_frame_ply() is None


def test_frame_to_ply_full_size_frame_round_trip(gpu_ctx):
    """BASELINE config 1 (0.8 M points): the ASCII file parses back to the frame, the binary one equals the host writer."""
    from tmc2rs_b200 import ply
    g = synth.make_gof(synth.config("c1"))
    view = abi.GofView(g)
    fr = gpu_ctx.decode_gof(view)[0]
    asc = _ply_frames(gpu_ctx, view, 1, abi.PLY_ASCII)[0]
    pos, col = ply.read_ply(asc)
    assert np.array_equal(pos, fr.positions) and np.array_equal(col, fr.colors)
    assert hashlib.sha256(asc).digest() == hashlib.sha256(ply.ascii_ply(fr.positions, fr.colors)).digest()
    assert _ply_frames(gpu_ctx, view, 1, abi.PLY_BINARY_LE)[0] == ply.binary_ply(fr.positions, fr.colors)


def test_one_process_two_devices_shard_frames_in_order():
    """SURVEY 8e inside ONE process: a context over two devices shards the frames of a GOF frame-wise (contiguous halves, no
    collective) and hands them back in order; results equal the single-device context.  Skipped on a one-GPU box."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    g = synth.replicate_gof(synth.make_gof(synth.config("small")), 7)      # odd frame count: slices of 3 and 4
    g.params.geometry_smoothing = True
    g.params.color_smoothing = True
    view = abi.GofView(g)
    one, two = codec.Context(devices=(0,)), codec.Context(devices=(0, 1))
    try:
        a = one.decode_gof(view)
        b = two.decode_gof(view)
        b2 = two.decode_gof(view)                                           # second GOF through the same two-device context
        assert len(a) == len(b) == len(b2) == 7
        for x, y, z in zip(a, b, b2):
            assert np.array_equal(x.positions, y.positions) and np.array_equal(x.colors, y.colors)
            assert np.array_equal(x.positions, z.positions) and np.array_equal(x.colors, z.colors)
        want = oracle.reconstruct_frame(view, 5)
        assert np.array_equal(b[5].positions, want["positions"]) and np.array_equal(b[5].colors, want["colors"])
    finally:
        one.close()
        two.close()


def test_one_context_over_all_devices_in_order():
    """The product topology behind the unchanged `Decoder` API (src/lib.rs:81): ONE context over every GPU of the box, frames of
    each GOF sharded frame-wise inside the library and handed back in order, several GOFs in flight.  Needs >= 2 GPUs (runs on
    the multi-GPU scaling box; skipped on a one-GPU box)."""
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs at least two GPUs")
    g = synth.replicate_gof(synth.make_gof(synth.config("small")), 2 * n + 3)      # uneven slices
    g.params.geometry_smoothing = True
    g.params.color_smoothing = True
    view = abi.GofView(g)
    F = g.frame_count
    want = {f: oracle.reconstruct_frame(view, f) for f in (0, F // 2, F - 1)}
    ctx = codec.Context(devices=tuple(range(n)), gofs_in_flight=2)
    try:
        ctx.submit_gof(view)
        ctx.submit_gof(view)                                                        # two GOFs in flight on every device
        frames = [ctx.next_frame() for _ in range(2 * F)]
        assert ctx.next_frame() is None
        for k, fr in enumerate(frames):
            f = k % F
            if f in want:
                assert np.array_equal(fr.positions, want[f]["positions"]) and np.array_equal(fr.colors, want[f]["colors"]), (k, f)
        for a, b in zip(frames[:F], frames[F:]):
            assert np.array_equal(a.positions, b.positions) and np.array_equal(a.colors, b.colors)
    finally:
        ctx.close()
