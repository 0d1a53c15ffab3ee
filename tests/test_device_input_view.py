"""GofView over device planes (``__cuda_array_interface__``), without a GPU: pointers, element strides and input_flags of
the C view, for padded pitches and the P010 layout; mixed host / device planes are refused."""
import numpy as np
import pytest

import util
from tmc2rs_b200 import abi


class FakeDev:
    """A device array as torch / cupy describe one: shape, strides in bytes, base address, no memory behind it."""

    def __init__(self, shape, typestr, base, strides=None):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (base, False),
                                         "strides": None if strides is None else tuple(strides), "version": 3}


def padded(shape, itemsize, base, pad, typestr):
    """C-ordered array whose rows are `pad` samples longer than the shape says."""
    row = (shape[-1] + pad) * itemsize
    strides = [row, itemsize]
    for n in reversed(shape[1:-1]):
        strides.insert(0, strides[0] * n)
    return FakeDev(shape, typestr, base, strides), row


def test_device_planar_view_pointers_strides_and_flags():
    g = util.random_small_gof(1, W=64, H=48, frames=2)
    F, W, H = 2, 64, 48
    occ, occ_row = padded((F, H // 4, W // 4), 1, 0x1000_0000, 16, "|u1")
    geo, geo_row = padded((F, 2, H, W), 2, 0x2000_0000, 64, "<u2")
    ay, ay_row = padded((F, 2, H, W), 2, 0x3000_0000, 3, "<i2")              # odd pad: a pitch that is no 16-byte multiple
    au, c_row = padded((F, 2, H // 2, W // 2), 2, 0x4000_0002, 0, "<u2")     # tight, base one sample into its allocation
    av, _ = padded((F, 2, H // 2, W // 2), 2, 0x5000_0000, 0, "<u2")
    dg = abi.Gof(W, H, occ, geo, ay, au, av, g.patches, g.params)
    v = abi.GofView(dg)
    c = v.c
    assert c.input_flags == abi.INPUT_DEVICE and v.device_input
    assert (c.width, c.height, c.occ_width, c.occ_height, c.frame_count) == (W, H, W // 4, H // 4, F)
    assert c.geo_video_frames == c.attr_video_frames == 2 * F
    for f in range(F):
        fr = c.frames[f]
        assert (fr.occ_stride, fr.geo_stride, fr.attr_stride_y, fr.attr_stride_c) == (W // 4 + 16, W + 64, W + 3, W // 2)
        assert fr.occ == 0x1000_0000 + f * (H // 4) * occ_row
        for m in range(2):
            assert fr.geo[m] == 0x2000_0000 + (f * 2 + m) * H * geo_row
            assert fr.attr_y[m] == 0x3000_0000 + (f * 2 + m) * H * ay_row
            assert fr.attr_u[m] == 0x4000_0002 + (f * 2 + m) * (H // 2) * c_row
            assert fr.attr_v[m] == 0x5000_0000 + (f * 2 + m) * (H // 2) * c_row
        assert fr.patch_count == len(g.patches[f])


def test_device_p010_view_interleaved_uv_and_no_v_plane():
    g = util.random_small_gof(2, W=64, H=48)
    W, H = 64, 48
    occ = FakeDev((1, H // 4, W // 4), "|u1", 0x1000_0000)
    geo, geo_row = padded((1, 2, H, W), 2, 0x2000_0000, 192, "<u2")        # NVDEC-like 256-byte pitch multiple
    ay, _ = padded((1, 2, H, W), 2, 0x3000_0000, 192, "<u2")
    uv, uv_row = padded((1, 2, H // 2, W), 2, 0x4000_0000, 192, "<u2")
    v = abi.GofView(abi.Gof(W, H, occ, geo, ay, uv, None, g.patches, g.params, plane_format="p010"))
    fr = v.c.frames[0]
    assert v.c.input_flags == abi.INPUT_DEVICE | abi.INPUT_P010
    assert fr.attr_stride_c == W + 192 and fr.geo_stride == W + 192 and uv_row == 512
    assert fr.attr_u[1] == 0x4000_0000 + (H // 2) * uv_row
    assert not fr.attr_v[0] and not fr.attr_v[1]
    assert fr.geo[1] == 0x2000_0000 + H * geo_row


def test_host_planes_keep_flag_word_zero():
    v = abi.GofView(util.random_small_gof(3))
    assert v.c.input_flags == 0 and not v.device_input


def test_mixed_host_and_device_planes_are_refused():
    g = util.random_small_gof(4, W=64, H=48)
    g.geo = FakeDev(g.geo.shape, "<u2", 0x2000_0000)
    with pytest.raises(ValueError, match="mixed"):
        abi.GofView(g)


def test_p010_layout_errors():
    g = util.random_small_gof(5, W=64, H=48)
    g.plane_format = "p010"
    with pytest.raises(ValueError, match="attr_v"):               # P010 carries no separate V plane
        abi.GofView(g)
    g.attr_v = None
    g.attr_u = np.zeros((1, 2, 24, 64), np.uint16)
    with pytest.raises(ValueError, match="device"):               # host P010 is not supported
        abi.GofView(g)
    g.plane_format = "nv12"
    with pytest.raises(ValueError, match="plane_format"):
        abi.GofView(g)


def test_device_plane_with_non_contiguous_rows_is_refused():
    g = util.random_small_gof(6, W=64, H=48)
    g.occ = FakeDev(g.occ.shape, "|u1", 0x1000_0000)
    g.geo = FakeDev(g.geo.shape, "<u2", 0x2000_0000, strides=(2 * 48 * 128 * 2, 48 * 128 * 2, 128 * 2, 4))   # every other sample
    for n in ("attr_y", "attr_u", "attr_v"):
        setattr(g, n, FakeDev(getattr(g, n).shape, "<u2", 0x3000_0000))
    with pytest.raises(ValueError, match="geo: rows must be contiguous"):
        abi.GofView(g)
