"""Pins for the CPU oracle (no GPU needed): the hand-derived known-answer vector of SURVEY.md Appendix C, colour KATs
derived from src/codec.rs:661-687, and differential tests against the independent Python model tests/refmodel.py."""
import numpy as np
import pytest

import kats
import refmodel
import util
from oracle import oracle
from tmc2rs_b200 import abi, synth


def test_appendix_c_known_answer():
    g = synth.kat_appendix_c()
    r = oracle.reconstruct_frame(abi.GofView(g), 0)
    assert r["block_to_patch"].tolist() == [1, 2]
    assert r["point_count"] == 48
    pos = r["positions"].tolist()
    assert pos[0] == [16, 200, 100]
    assert pos[1] == [17, 200, 101] and pos[2] == [18, 200, 101]
    assert pos[3] == [18, 200, 102]
    assert pos[4] == [19, 200, 103] and pos[5] == [20, 200, 103]
    assert pos[6] == [17, 201, 100]
    assert pos[24] == [20, 940, 14] and pos[25] == [20, 939, 15] and pos[26] == [20, 938, 16] and pos[27] == [20, 937, 17]
    assert pos[28] == [21, 939, 14] and pos[29] == [21, 938, 14]
    assert r["point_to_pixel"][28].tolist() == [17, 4, 0] and r["point_to_pixel"][29].tolist() == [17, 4, 1]
    assert r["partition"].tolist() == [0] * 24 + [1] * 24
    # every pixel group of 4 sharing a canvas row yields 1+2+1+2 points (x&1 adds one to the second map's depth)
    assert (r["colors"] == 127).all()          # Y=U=V=512 -> (127,127,127)


@pytest.mark.parametrize("name,make", kats.ALL, ids=[n for n, _ in kats.ALL])
def test_hand_derived_kats(name, make):
    """tests/kats.py: rotated orientation in the reference's own pixel mapping, differential-D1 wrap, mode-1 clamp, duplicate
    skip, precedence of overlapping patches -- expected values derived by hand from the reference text."""
    g, want = make()
    kats.check(oracle.reconstruct_frame(abi.GofView(g), 0), want, name)
    m = refmodel.reconstruct(g, 0)                       # the independent Python model of the same lines agrees too
    m = {k: np.asarray(v) for k, v in m.items()}
    m["point_count"] = len(m["positions"])
    kats.check(m, want, name + " (refmodel)")


@pytest.mark.parametrize("yuv,rgb", [((512, 512, 512), (127, 127, 127)), ((1023, 512, 512), (255, 255, 255)),
                                     ((0, 512, 512), (0, 0, 0)), ((512, 512, 1023), (255, 67, 127)),
                                     ((0, 0, 0), (0, 83, 0)), ((1023, 1023, 1023), (255, 171, 255)),
                                     ((65535, 0, 65535), (255, 255, 255))])
def test_color_kats(yuv, rgb):
    # (0,0,0): g = 0 + 0.18733*512 + 0.46813*512 = 335.5955.. -> /1023*255 = 83.65 -> 83 ; r,b negative -> 0
    # (1023,1023,1023): g = 1023 - 0.18733*511 - 0.46813*511 = 688.06.. -> 171.5 -> 171
    assert oracle.convert_yuv10_to_rgb8([yuv]).tolist() == [list(rgb)]
    assert refmodel.yuv_to_rgb(yuv) == list(rgb)


def test_color_oracle_vs_model_random():
    rng = np.random.RandomState(7)
    yuv = np.concatenate([rng.randint(0, 1024, (3000, 3)), rng.randint(0, 65536, (1000, 3))]).astype(np.uint16)
    got = oracle.convert_yuv10_to_rgb8(yuv)
    want = np.array([refmodel.yuv_to_rgb(c) for c in yuv.tolist()], dtype=np.uint8)
    assert np.array_equal(got, want)


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
]


@pytest.mark.parametrize("case", CASES, ids=lambda c: "-".join(f"{k}{v}" for k, v in c.items() if k != "orientations"))
def test_oracle_matches_python_model(case):
    g = util.random_small_gof(**case)
    view = abi.GofView(g)
    want = refmodel.reconstruct(g, 0)
    got = oracle.reconstruct_frame(view, 0)
    assert got["block_to_patch"].tolist() == want["block_to_patch"]
    assert got["occupancy_map"].tolist() == want["occupancy_map"]
    assert got["point_count"] == len(want["positions"])
    assert got["positions"].tolist() == want["positions"]
    assert got["partition"].tolist() == want["partition"]
    assert got["point_to_pixel"].tolist() == want["point_to_pixel"]
    if g.params.attribute_count:
        assert got["colors16bit"].tolist() == want["colors16bit"]
        assert got["colors"].tolist() == want["colors"]
    assert oracle.block_to_patch(view, 0).tolist() == want["block_to_patch"]


def test_oracle_error_codes_mirror_reference_panics():
    g = util.random_small_gof(seed=11)
    # patch sticking out of the canvas -> assert at decoder.rs:835/848
    bad = g.patches[0].copy()
    bad["u0"][0] = 1000
    g2 = abi.Gof(g.width, g.height, g.occ, g.geo, g.attr_y, g.attr_u, g.attr_v, [bad], g.params)
    with pytest.raises(oracle.OracleError) as e:
        oracle.reconstruct_frame(abi.GofView(g2), 0)
    assert e.value.status == abi.ERR_PATCH_OUT_OF_CANVAS
    with pytest.raises(refmodel.Panic):
        refmodel.reconstruct(g2, 0)
    # short geometry video -> codec.rs:318-320
    g3 = abi.Gof(g.width, g.height, g.occ, g.geo, g.attr_y, g.attr_u, g.attr_v, g.patches, g.params, geo_video_frames=1)
    with pytest.raises(oracle.OracleError) as e:
        oracle.reconstruct_frame(abi.GofView(g3), 0)
    assert e.value.status == abi.ERR_SHORT_VIDEO
    # single map -> codec.rs:432 unwrap of None
    p = abi.Params(**{**g.params.__dict__, "map_count_minus1": 0})
    g4 = abi.Gof(g.width, g.height, g.occ, g.geo, g.attr_y, g.attr_u, g.attr_v, g.patches, p)
    with pytest.raises(oracle.OracleError) as e:
        oracle.reconstruct_frame(abi.GofView(g4), 0)
    assert e.value.status == abi.ERR_MAP_COUNT
    # unimplemented!() switches
    p = abi.Params(**{**g.params.__dict__, "pbf_enabled": True})
    g5 = abi.Gof(g.width, g.height, g.occ, g.geo, g.attr_y, g.attr_u, g.attr_v, g.patches, p)
    with pytest.raises(oracle.OracleError) as e:
        oracle.reconstruct_frame(abi.GofView(g5), 0)
    assert e.value.status == abi.ERR_UNSUPPORTED


def test_empty_and_ragged_inputs():
    # no patches at all; a patch of size zero; a fully unoccupied frame
    g = util.random_small_gof(seed=12)
    empty = abi.Gof(g.width, g.height, g.occ, g.geo, g.attr_y, g.attr_u, g.attr_v, [g.patches[0][:0]], g.params)
    r = oracle.reconstruct_frame(abi.GofView(empty), 0)
    assert r["point_count"] == 0 and not r["block_to_patch"].any()
    z = g.patches[0].copy()
    z["size_u0"][0] = 0
    r = oracle.reconstruct_frame(abi.GofView(abi.Gof(g.width, g.height, g.occ, g.geo, g.attr_y, g.attr_u, g.attr_v, [z], g.params)), 0)
    assert r["point_count"] == len(refmodel.reconstruct(abi.Gof(g.width, g.height, g.occ, g.geo, g.attr_y, g.attr_u, g.attr_v, [z], g.params), 0)["positions"])
    blank = abi.Gof(g.width, g.height, np.zeros_like(g.occ), g.geo, g.attr_y, g.attr_u, g.attr_v, g.patches, g.params)
    r = oracle.reconstruct_frame(abi.GofView(blank), 0)
    assert r["point_count"] == 0 and not r["block_to_patch"].any()


def test_smoothing_spec_invariants():
    """Own-spec post-processing: deterministic, only boundary points move, counts are consistent."""
    cfg = synth.config("small")
    g = synth.make_gof(cfg)
    g.params.geometry_smoothing = True
    g.params.color_smoothing = True
    v = abi.GofView(g)
    a = oracle.reconstruct_frame(v, 0)
    b = oracle.reconstruct_frame(v, 0)
    assert np.array_equal(a["positions"], b["positions"]) and np.array_equal(a["colors"], b["colors"])
    moved = (a["positions"] != a["positions_presmooth"]).any(axis=1)
    assert moved.sum() == a["smoothed_positions"]
    assert (a["boundary_type"][moved] == 1).all()
    rec = (a["colors16bit"] != a["colors16bit_presmooth"]).any(axis=1)
    assert rec.sum() == a["smoothed_colors"]
    assert (a["boundary_type"][rec] == 1).all()
    # boundary types against a direct numpy evaluation of the spec
    expect = util.boundary_spec(a["occupancy_map"])
    px = a["point_to_pixel"]
    assert np.array_equal(a["boundary_type"], expect[px[:, 1], px[:, 0]])
