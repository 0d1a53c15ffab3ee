"""Host-side mirror of the reference's reconstruction interface (``src/codec.rs`` + the frame loop of
``src/decoder.rs:188-314``), implemented by calling the CUDA library through the C ABI.

Names follow the reference: :func:`Context.generate_block_to_patch_from_occupancy_map_video` (src/codec.rs:205),
:func:`Context.generate_point_cloud` (src/codec.rs:256), :func:`Context.convert_yuv16_to_rgb8` (src/codec.rs:88),
:class:`PointSet3` (src/codec.rs:20-36).  Where the reference panics, these raise :class:`abi.Tmc2Error` carrying the
status code.  Nothing here computes on the CPU and nothing imports ``oracle/``.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence

import numpy as np

from . import abi
from ._lib import load


@dataclass
class PointSet3:
    """src/codec.rs:20-36: ``positions`` [n,3] u16, ``colors`` [n,3] u8, ``with_colors``."""
    positions: np.ndarray
    colors: Optional[np.ndarray]
    with_colors: bool
    smoothed_positions: int = 0
    smoothed_colors: int = 0

    def __len__(self) -> int:          # PointSet3::len, src/codec.rs:108-111
        assert not self.with_colors or len(self.positions) == len(self.colors)
        return len(self.positions)


class Context:
    """Owns a ``tmc2gpu_ctx`` (device buffers, streams, pinned staging).  ``two_pass_scan`` sets a reserved legacy flag that
    the library accepts and ignores (the unpack is always count / scan / emit)."""

    def __init__(self, devices: Sequence[int] = (0,), max_frames: int = 0, gofs_in_flight: int = 2,
                 two_pass_scan: bool = False, device_output: bool = False):
        self.h = None
        self.lib = load()
        if self.lib.tmc2gpu_device_count() <= 0:
            raise abi.Tmc2Error(abi.ERR_NO_DEVICE, "tmc2gpu_create", "no CUDA device (there is no CPU fallback)")
        lim = abi.CLimits(0, 0, max_frames, 0, gofs_in_flight,
                          (abi.CTX_TWO_PASS_SCAN if two_pass_scan else 0) | (abi.CTX_DEVICE_OUTPUT if device_output else 0))
        ids = (C.c_int * len(devices))(*devices)
        h = C.c_void_p()
        st = self.lib.tmc2gpu_create(ids, len(devices), C.byref(lim), C.byref(h))
        if st:
            raise abi.Tmc2Error(st, "tmc2gpu_create")
        self.h = h
        self.devices = list(devices)
        self._fo = abi.CFrameOut()

    def close(self):
        if getattr(self, "h", None):
            self.lib.tmc2gpu_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def check(self, st: int, where: str):
        if st != abi.OK:
            msg = self.lib.tmc2gpu_last_error(self.h)
            raise abi.Tmc2Error(st, where, msg.decode() if msg else "")

    @staticmethod
    def _inputs_written(view: abi.GofView):
        """Device planes must be completely written when the library is called (it does not wait on the caller's stream):
        synchronise torch's current stream on every device that holds planes of the GOF."""
        if view.device_input and view.devices:
            import torch
            for d in view.devices:
                torch.cuda.current_stream(d).synchronize()

    # ---- stage API (one frame, synchronous) -----------------------------------------------------------------
    def generate_block_to_patch_from_occupancy_map_video(self, view: abi.GofView, frame_index: int) -> np.ndarray:
        """src/codec.rs:205-250.  Returns ``block_to_patch`` (patch index + 1, 0 = unowned)."""
        g = view.c
        res = max(g.params.occupancy_resolution, 1)
        out = np.zeros(max((g.width // res) * (g.height // res), 1), dtype=np.uint32)
        self._inputs_written(view)
        self.check(self.lib.tmc2gpu_generate_block_to_patch_from_occupancy_map_video(
            self.h, view.ref(), frame_index, out.ctypes.data), "generate_block_to_patch_from_occupancy_map_video")
        return out[:(g.width // res) * (g.height // res)]

    def generate_point_cloud(self, view: abi.GofView, frame_index: int, debug: bool = True) -> Dict[str, np.ndarray]:
        """src/codec.rs:256-514 for one frame, plus the post-processing / colour conversion the reference's caller does
        (src/decoder.rs:281-305).  With ``debug`` every intermediate the reference materialises is returned too."""
        g = view.c
        cap = max(2 * g.width * g.height, 1)
        res = max(g.params.occupancy_resolution, 1)
        o = abi.CPointCloudOut()
        o.capacity_points = cap
        bufs = {"positions": np.zeros((cap, 3), np.uint16), "colors": np.zeros((cap, 3), np.uint8)}
        if debug:
            bufs.update({"colors16bit": np.zeros((cap, 3), np.uint16), "partition": np.zeros(cap, np.uint32),
                         "point_to_pixel": np.zeros((cap, 3), np.uint32),
                         "occupancy_map": np.zeros((g.height, g.width), np.uint8),
                         "boundary_type": np.zeros(cap, np.uint8),
                         "positions_presmooth": np.zeros((cap, 3), np.uint16),
                         "colors16bit_presmooth": np.zeros((cap, 3), np.uint16)})
        bufs["block_to_patch"] = np.zeros(max((g.width // res) * (g.height // res), 1), np.uint32)
        for k, v in bufs.items():
            setattr(o, k, v.ctypes.data)
        self._inputs_written(view)
        self.check(self.lib.tmc2gpu_generate_point_cloud(self.h, view.ref(), frame_index, C.byref(o)),
                   "generate_point_cloud")
        n = int(o.point_count)
        out = {"point_count": n, "smoothed_positions": int(o.smoothed_positions),
               "smoothed_colors": int(o.smoothed_colors)}
        per_point = {"positions", "colors", "colors16bit", "partition", "point_to_pixel", "boundary_type",
                     "positions_presmooth", "colors16bit_presmooth"}
        for k, v in bufs.items():
            out[k] = v[:n].copy() if k in per_point else v
        out["block_to_patch"] = out["block_to_patch"][:(g.width // res) * (g.height // res)]
        return out

    def convert_yuv16_to_rgb8(self, yuv16: np.ndarray) -> np.ndarray:
        """src/codec.rs:88-94 / :661-687 on the GPU."""
        yuv = np.ascontiguousarray(yuv16, dtype=np.uint16).reshape(-1, 3)
        rgb = np.zeros((len(yuv), 3), np.uint8)
        self.check(self.lib.tmc2gpu_convert_yuv16_to_rgb8(self.h, yuv.ctypes.data, len(yuv), rgb.ctypes.data),
                   "convert_yuv16_to_rgb8")
        return rgb

    # ---- streaming API: the frame loop src/decoder.rs:188-314 -------------------------------------------------
    def submit_gof(self, view: abi.GofView):
        self._inputs_written(view)
        self.check(self.lib.tmc2gpu_submit_gof(self.h, view.ref()), "submit_gof")

    def wait_inputs(self):
        """Blocks until the inputs of every submitted GOF have been read (H2D copies, or the gather kernel of device planes):
        pinned or device input planes may be overwritten again."""
        self.check(self.lib.tmc2gpu_wait_inputs(self.h), "wait_inputs")

    def next_frame(self, copy: bool = True) -> Optional[PointSet3]:
        fo = abi.CFrameOut()
        st = self.lib.tmc2gpu_next_frame(self.h, C.byref(fo))
        if st == abi.END:
            return None
        self.check(st, "next_frame")
        n = int(fo.point_count)
        pos = np.ctypeslib.as_array(C.cast(fo.positions, C.POINTER(C.c_uint16)), shape=(n, 3)) if n else \
            np.zeros((0, 3), np.uint16)
        col = None
        if fo.with_colors:
            col = np.ctypeslib.as_array(C.cast(fo.colors, C.POINTER(C.c_uint8)), shape=(n, 3)) if n else \
                np.zeros((0, 3), np.uint8)
        if copy:
            pos = pos.copy()
            col = None if col is None else col.copy()
        ps = PointSet3(pos, col, bool(fo.with_colors), int(fo.smoothed_positions), int(fo.smoothed_colors))
        self.check(self.lib.tmc2gpu_release_frame(self.h, C.byref(fo)), "release_frame")
        return ps

    def next_frame_ply(self, fmt: int = abi.PLY_ASCII, capacity: Optional[int] = None) -> Optional[bytes]:
        """The next frame as a finished PLY file (``src/writer.rs:15-75``), formatted on the device
        (``tmc2gpu_frame_to_ply``); None at the end.  ``capacity``: size of the destination buffer (default: ask first)."""
        fo = abi.CFrameOut()
        st = self.lib.tmc2gpu_next_frame(self.h, C.byref(fo))
        if st == abi.END:
            return None
        self.check(st, "next_frame")
        try:
            size = C.c_uint64(0)
            if capacity is None:
                self.check(self.lib.tmc2gpu_frame_to_ply(self.h, C.byref(fo), fmt, None, 0, C.byref(size)), "frame_to_ply")
                capacity = int(size.value)
            buf = np.empty(max(capacity, 1), np.uint8)
            self.check(self.lib.tmc2gpu_frame_to_ply(self.h, C.byref(fo), fmt, buf.ctypes.data, capacity, C.byref(size)),
                       "frame_to_ply")
            return buf[:int(size.value)].tobytes()
        finally:
            self.lib.tmc2gpu_release_frame(self.h, C.byref(fo))

    def next_frame_device(self):
        """Device-resident hand-off (contexts created with ``device_output=True``): ``(point_count, positions device pointer,
        colours device pointer, device ordinal, release)`` of the next frame, or None at the end.  The pointers stay valid until
        ``release()`` has been called for every frame of that GOF."""
        fo = abi.CFrameOut()
        st = self.lib.tmc2gpu_next_frame(self.h, C.byref(fo))
        if st == abi.END:
            return None
        self.check(st, "next_frame")
        assert fo.memory_space == 1, "context was not created with device_output=True"

        def release(fo=fo):
            self.check(self.lib.tmc2gpu_release_frame(self.h, C.byref(fo)), "release_frame")
        return int(fo.point_count), int(fo.positions or 0), int(fo.colors or 0), int(fo.device), release

    def next_frame_raw(self):
        """Lean variant of next_frame for tight loops: (point_count, positions address, colours address) of the next frame in
        the library's pinned host buffers, already released (valid until the GOF slot is reused); None at the end."""
        fo = self._fo
        st = self.lib.tmc2gpu_next_frame(self.h, C.byref(fo))
        if st == abi.END:
            return None
        if st:
            self.check(st, "next_frame")
        r = (fo.point_count, fo.positions, fo.colors)
        st = self.lib.tmc2gpu_release_frame(self.h, C.byref(fo))
        if st:
            self.check(st, "release_frame")
        return r

    def decode_gof(self, view: abi.GofView) -> List[PointSet3]:
        self.submit_gof(view)
        return [self.next_frame() for _ in range(view.c.frame_count)]

    # ---- resident path (planes stay in HBM) -------------------------------------------------------------------
    def upload_gof(self, view: abi.GofView) -> "Resident":
        h = C.c_void_p()
        self._inputs_written(view)
        self.check(self.lib.tmc2gpu_upload_gof(self.h, view.ref(), C.byref(h)), "upload_gof")
        return Resident(self, h, view.c.frame_count)

    def last_launch_info(self):
        k, b, t = C.c_uint32(), C.c_uint64(), C.c_uint64()
        self.check(self.lib.tmc2gpu_last_launch_info(self.h, C.byref(k), C.byref(b), C.byref(t)), "last_launch_info")
        return int(k.value), int(b.value), int(t.value)

    def last_stage_ms(self):
        ms = (C.c_float * 5)()
        self.check(self.lib.tmc2gpu_last_stage_ms(self.h, ms), "last_stage_ms")
        return dict(zip(("block_to_patch", "unpack", "smoothing", "count_scan", "yuv_to_rgb"), list(ms)))


class Resident:
    def __init__(self, ctx: Context, h, frames: int):
        self.ctx, self.h, self.frames = ctx, h, frames

    def reconstruct(self, cuda_stream: int = 0, timed: bool = False):
        """Launch the reconstruction of the resident GOF on `cuda_stream`.  `timed`: take the ordinary launch sequence (which
        records the stage-timing events) even where a CUDA-graph replay would be used."""
        self.ctx.check(self.ctx.lib.tmc2gpu_reconstruct_resident_ex(self.ctx.h, self.h, C.c_void_p(cuda_stream),
                                                                    abi.LAUNCH_TIMED if timed else 0), "reconstruct_resident")

    def counts(self) -> np.ndarray:
        out = (C.c_uint64 * max(self.frames, 1))()
        self.ctx.check(self.ctx.lib.tmc2gpu_resident_counts(self.ctx.h, self.h, out), "resident_counts")
        return np.array(list(out)[:self.frames], dtype=np.uint64)

    def fetch(self, frame: int, n: int):
        pos = np.zeros((max(n, 1), 3), np.uint16)
        col = np.zeros((max(n, 1), 3), np.uint8)
        self.ctx.check(self.ctx.lib.tmc2gpu_resident_fetch(self.ctx.h, self.h, frame, pos.ctypes.data, col.ctypes.data,
                                                           max(n, 1)), "resident_fetch")
        return pos[:n], col[:n]

    def free(self):
        if self.h:
            self.ctx.lib.tmc2gpu_free_resident(self.ctx.h, self.h)
            self.h = None


_PINNED: Dict[int, int] = {}


def pinned_empty(shape, dtype) -> np.ndarray:
    """numpy array over memory from ``tmc2gpu_alloc_pinned`` (submits from it skip the staging copy)."""
    lib = load()
    dtype = np.dtype(dtype)
    count = int(np.prod(shape))
    n = count * dtype.itemsize
    p = lib.tmc2gpu_alloc_pinned(max(n, 1))
    if not p:
        raise MemoryError("tmc2gpu_alloc_pinned failed")
    buf = (C.c_uint8 * max(n, 1)).from_address(p)
    arr = np.frombuffer(buf, dtype=dtype, count=count).reshape(shape)
    _PINNED[arr.ctypes.data] = p
    return arr


def pinned_copy_of(gof: abi.Gof) -> abi.Gof:
    """Copy a GOF's planes into pinned memory."""
    def pc(a):
        if a is None:
            return None
        b = pinned_empty(a.shape, a.dtype)
        b[...] = a
        return b
    return abi.Gof(gof.width, gof.height, pc(gof.occ), pc(gof.geo), pc(gof.attr_y), pc(gof.attr_u), pc(gof.attr_v),
                   gof.patches, gof.params, gof.geo_video_frames, gof.attr_video_frames)
