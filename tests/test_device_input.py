"""Planes that already sit in GPU memory (TMC2_INPUT_DEVICE), planar and in the P010 layout of hardware video decoders
(TMC2_INPUT_P010): every entry point gives the oracle's answer for the host planes, bit for bit.  Run on a B200."""
import numpy as np
import pytest

import util
from oracle import oracle
from tmc2rs_b200 import abi, codec, synth

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
# row pitch and base address of the device planes: tight; padded to a 16-byte multiple (vector path); padded by an odd
# number of samples (narrow path); based one sample into the allocation (narrow path, 2-byte aligned base)
LAYOUTS = {"tight": {}, "pad64": {"pad": 64}, "pad3": {"pad": 3}, "offset1": {"offset": 1}}
FORMATS = ("planar", "p010")
SMOOTH_KEYS = ("boundary_type", "positions_presmooth", "colors16bit_presmooth")


def small_smooth(frames=3):
    g = synth.make_gof(synth.config("small", frames=frames))
    g.params.geometry_smoothing = True
    g.params.color_smoothing = True
    return g


# 10-bit samples only (P010 holds 10 bits): the `extreme` generator cases are left to the host-plane tests
CASES = {
    "rand1": lambda: util.random_small_gof(1, orientations=(0, 1)),
    "rand4-spec": lambda: util.random_small_gof(4, orientations=tuple(range(9)), spec=True),
    "rand8-res8": lambda: util.random_small_gof(8, orientations=(0, 1, 3, 5), spec=True, res=8, prec=4, W=40, H=32),
    "rand9-noattr": lambda: util.random_small_gof(9, orientations=(0, 1), attr=False),
    "rand11-wide": lambda: util.random_small_gof(11, orientations=(0, 1), W=208, H=112, n_patches=14),
    "small-smooth": small_smooth,
    "c1": lambda: synth.make_gof(synth.config("c1")),
}
_host, _want = {}, {}


def host_case(name):
    if name not in _host:
        g = CASES[name]()
        v = abi.GofView(g)
        _host[name] = (g, v)
        _want[name] = [oracle.reconstruct_frame(v, f) for f in range(g.frame_count)]
    return _host[name][0], _want[name]


def keys_of(g):
    keys = list(util.STREAMS)
    if not g.params.attribute_count:
        keys = [k for k in keys if k not in ("colors", "colors16bit")]
    if g.params.geometry_smoothing or g.params.color_smoothing:
        keys += list(SMOOTH_KEYS)
    return keys


def device_view(g, fmt="planar", device=DEV, **layout):
    if fmt == "p010" and g.attr_y is None:
        pytest.skip("P010 needs attribute planes in this test")
    return abi.GofView(synth.to_device(g, device, p010=fmt == "p010", seed=7, **layout))


def same_frame(pos, col, want, what):
    assert len(pos) == want["point_count"], what
    assert np.array_equal(pos, want["positions"]), what
    if col is not None:
        assert np.array_equal(col, want["colors"]), what


@pytest.mark.parametrize("fmt", FORMATS)
@pytest.mark.parametrize("layout", list(LAYOUTS))
@pytest.mark.parametrize("case", list(CASES))
def test_stage_api_device_planes_bit_exact(gpu_ctx, case, layout, fmt):
    g, want = host_case(case)
    v = device_view(g, fmt, **LAYOUTS[layout])
    assert v.c.input_flags == abi.INPUT_DEVICE | (abi.INPUT_P010 if fmt == "p010" else 0)
    for f in range(g.frame_count):
        got = gpu_ctx.generate_point_cloud(v, f)
        util.assert_same(got, want[f], keys=keys_of(g), what=f"{case}/{layout}/{fmt} frame {f}")
        assert got["smoothed_positions"] == want[f]["smoothed_positions"]
        assert got["smoothed_colors"] == want[f]["smoothed_colors"]
        b2p = gpu_ctx.generate_block_to_patch_from_occupancy_map_video(v, f)
        assert np.array_equal(b2p.astype(np.int64), want[f]["block_to_patch"].astype(np.int64))


@pytest.mark.parametrize("fmt", FORMATS)
@pytest.mark.parametrize("layout", list(LAYOUTS))
def test_streaming_and_resident_device_planes(gpu_ctx, layout, fmt):
    g, want = host_case("small-smooth")
    v = device_view(g, fmt, **LAYOUTS[layout])
    frames = gpu_ctx.decode_gof(v)
    assert gpu_ctx.next_frame() is None
    for f, fr in enumerate(frames):
        same_frame(fr.positions, fr.colors, want[f], f"streaming {layout}/{fmt} frame {f}")
    r = gpu_ctx.upload_gof(v)
    try:
        r.reconstruct()
        r.reconstruct()
        counts = r.counts()
        for f in range(g.frame_count):
            pos, col = r.fetch(f, int(counts[f]))
            same_frame(pos, col, want[f], f"resident {layout}/{fmt} frame {f}")
    finally:
        r.free()


def test_full_size_streaming_device_planes(gpu_ctx):
    g, want = host_case("c1")
    for fmt in FORMATS:
        fr = gpu_ctx.decode_gof(device_view(g, fmt, pad=192))      # NVDEC-like pitch: a multiple of 256 bytes
        same_frame(fr[0].positions, fr[0].colors, want[0], fmt)
        k, _, total = gpu_ctx.last_launch_info()
        assert total == want[0]["point_count"] and k >= 3          # the ingest launch is counted with the others


class _Raw:                                               # zero-copy torch view of a raw device range
    def __init__(self, ptr, nbytes):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 2}


def test_device_planes_in_device_frames_out():
    import torch
    g, want = host_case("small-smooth")
    ctx = codec.Context(device_output=True)
    try:
        for fmt in FORMATS:
            ctx.submit_gof(device_view(g, fmt))
            got = [ctx.next_frame_device() for _ in range(g.frame_count)]
            assert ctx.next_frame_device() is None
            for f, (n, ppos, pcol, dev, release) in enumerate(got):
                pos = torch.as_tensor(_Raw(ppos, n * 6), device=DEV).cpu().numpy().view(np.uint16).reshape(n, 3)
                col = torch.as_tensor(_Raw(pcol, n * 3), device=DEV).cpu().numpy().reshape(n, 3)
                same_frame(pos, col, want[f], f"{fmt} frame {f}")
            for *_, release in got:
                release()
    finally:
        ctx.close()


def test_planes_may_be_overwritten_after_wait_inputs(gpu_ctx):
    import torch
    g, want = host_case("small-smooth")
    for fmt in FORMATS:
        dg = synth.to_device(g, DEV, p010=fmt == "p010", seed=3)
        gpu_ctx.submit_gof(abi.GofView(dg))
        gpu_ctx.wait_inputs()
        for t in (dg.occ, dg.geo, dg.attr_y, dg.attr_u, dg.attr_v):
            if t is not None:
                t.fill_(77)
        torch.cuda.synchronize()
        for f in range(g.frame_count):
            fr = gpu_ctx.next_frame()
            same_frame(fr.positions, fr.colors, want[f], f"{fmt} frame {f}")
        assert gpu_ctx.next_frame() is None


def test_host_device_and_p010_gofs_back_to_back():
    g, want = host_case("small-smooth")
    views = [abi.GofView(g), device_view(g, "planar", pad=3), device_view(g, "p010", offset=1)]
    ctx = codec.Context(gofs_in_flight=3)
    try:
        for v in views:
            ctx.submit_gof(v)
        for k in range(3 * g.frame_count):
            fr = ctx.next_frame()
            same_frame(fr.positions, fr.colors, want[k % g.frame_count], f"GOF {k // g.frame_count} frame {k % g.frame_count}")
        assert ctx.next_frame() is None
    finally:
        ctx.close()


def refused(ctx, view, status):
    with pytest.raises(abi.Tmc2Error) as e:
        ctx.submit_gof(view)
    assert e.value.status == status, str(e.value)
    with pytest.raises(abi.Tmc2Error) as e:
        ctx.generate_point_cloud(view, 0)
    assert e.value.status == status, str(e.value)
    return str(e.value)


def still_usable(ctx, g, want):
    fr = ctx.decode_gof(device_view(g, "p010"))
    assert ctx.next_frame() is None
    for f in range(g.frame_count):
        same_frame(fr[f].positions, fr[f].colors, want[f], f"after a refusal, frame {f}")


def test_refusals_leave_a_usable_context(gpu_ctx):
    g, want = host_case("small-smooth")
    W = g.width

    v = abi.GofView(g)
    v.c.input_flags = 4                                           # unknown bit
    refused(gpu_ctx, v, abi.ERR_INVALID_ARG)
    v.c.input_flags = abi.INPUT_P010                              # P010 from host planes
    refused(gpu_ctx, v, abi.ERR_UNSUPPORTED)
    v.c.input_flags = abi.INPUT_DEVICE                            # "device" planes that are numpy arrays
    assert "host memory" in refused(gpu_ctx, v, abi.ERR_INVALID_ARG)
    vp = abi.GofView(codec.pinned_copy_of(g))                     # ... or tmc2gpu_alloc_pinned blocks
    vp.c.input_flags = abi.INPUT_DEVICE
    assert "host memory" in refused(gpu_ctx, vp, abi.ERR_INVALID_ARG)
    still_usable(gpu_ctx, g, want)

    dg = synth.to_device(g, DEV, p010=True, seed=1)
    v = abi.GofView(dg)
    v.c.frames[0].attr_v[1] = v.c.frames[0].attr_u[1]             # P010 with a V plane
    refused(gpu_ctx, v, abi.ERR_INVALID_ARG)
    v = abi.GofView(dg)
    v.c.frames[0].attr_stride_c = W - 1                           # interleaved UV rows hold W samples
    assert "stride smaller than width" in refused(gpu_ctx, v, abi.ERR_INVALID_ARG)
    v = abi.GofView(synth.to_device(g, DEV))
    v.c.frames[0].geo_stride = 1 << 31                            # the plane would run far past its tensor
    assert "past the end" in refused(gpu_ctx, v, abi.ERR_INVALID_ARG)
    still_usable(gpu_ctx, g, want)


def test_plane_on_a_device_outside_the_context(gpu_ctx):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    g, want = host_case("small-smooth")
    assert "not a device of the context" in refused(gpu_ctx, device_view(g, "planar", device="cuda:1"), abi.ERR_INVALID_ARG)
    still_usable(gpu_ctx, g, want)


@pytest.mark.parametrize("plane_device", [0, 1])
def test_two_device_context_reads_planes_of_either_device(plane_device):
    """Frames of a GOF are sharded over devices 0 and 1; every plane sits on one of them, the other device reads them by
    peer access."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    g = synth.replicate_gof(small_smooth(), 7)
    hv = abi.GofView(g)
    want = [oracle.reconstruct_frame(hv, f) for f in range(7)]
    ctx = codec.Context(devices=(0, 1))
    try:
        for fmt in FORMATS:
            v = device_view(g, fmt, device=f"cuda:{plane_device}", pad=3)
            frames = ctx.decode_gof(v) + ctx.decode_gof(v)
            assert ctx.next_frame() is None
            for k, fr in enumerate(frames):
                same_frame(fr.positions, fr.colors, want[k % 7], f"{fmt} frame {k}")
    finally:
        ctx.close()
