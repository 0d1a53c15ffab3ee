"""ctypes mirror of ``include/tmc2gpu.h`` (the C ABI of the reconstruction path).

Every structure here has the same field order, types and size as its C counterpart; ``tests/test_abi.py``
checks sizes/offsets against a table emitted by the C compiler.  The numpy ``PATCH_DTYPE`` is the same
40-byte record as ``tmc2_patch`` so patch lists travel as plain arrays.

Reference counterparts: ``Patch`` src/decoder.rs:711-783, ``GeneratePointCloudParams`` src/codec.rs:140-170,
``PointSet3`` src/codec.rs:20-36, ``Video``/``Image`` src/decoder.rs:913-1021.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import List, Optional, Sequence

import numpy as np

ABI_VERSION = 1

# ---- status codes (tmc2_status) ---------------------------------------------------------------------------------
OK, END, ERR_INVALID_ARG, ERR_PATCH_OUT_OF_CANVAS, ERR_SHORT_VIDEO, ERR_MAP_COUNT, ERR_UNSUPPORTED, \
    ERR_CAPACITY, ERR_STATE, ERR_NO_DEVICE, ERR_CUDA, ERR_INTERNAL = range(12)
STATUS_NAMES = ["OK", "END", "ERR_INVALID_ARG", "ERR_PATCH_OUT_OF_CANVAS", "ERR_SHORT_VIDEO", "ERR_MAP_COUNT",
                "ERR_UNSUPPORTED", "ERR_CAPACITY", "ERR_STATE", "ERR_NO_DEVICE", "ERR_CUDA", "ERR_INTERNAL"]

# ---- PatchOrientation (src/decoder.rs:694-707) ------------------------------------------------------------------
ORIENT_DEFAULT, ORIENT_SWAP, ORIENT_ROT90, ORIENT_ROT180, ORIENT_ROT270, ORIENT_MIRROR, ORIENT_MROT90, \
    ORIENT_MROT180, ORIENT_MROT270 = range(9)
ORIENTATION_REFERENCE, ORIENTATION_SPEC = 0, 1

CTX_TWO_PASS_SCAN = 1
CTX_DEVICE_OUTPUT = 2
LAUNCH_TIMED = 1
INPUT_DEVICE, INPUT_P010 = 1, 2          # tmc2_gof.input_flags: planes in CUDA device memory / P010 layout
PLY_ASCII, PLY_BINARY_LE = 0, 1          # tmc2gpu_frame_to_ply formats (src/writer.rs:8-12)


class Tmc2Error(RuntimeError):
    """Raised where the reference would panic; carries the C status code."""

    def __init__(self, status: int, where: str = "", detail: str = ""):
        self.status = int(status)
        name = STATUS_NAMES[status] if 0 <= status < len(STATUS_NAMES) else str(status)
        super().__init__(f"{where}: {name}" + (f" ({detail})" if detail else ""))


class CPatch(C.Structure):
    _fields_ = [("u0", C.c_uint32), ("v0", C.c_uint32), ("size_u0", C.c_uint32), ("size_v0", C.c_uint32),
                ("u1", C.c_uint32), ("v1", C.c_uint32), ("d1", C.c_uint32),
                ("lod_x", C.c_uint16), ("lod_y", C.c_uint16),
                ("normal_axis", C.c_uint8), ("tangent_axis", C.c_uint8), ("bitangent_axis", C.c_uint8),
                ("projection_mode", C.c_uint8), ("patch_orientation", C.c_uint8),
                ("axis_of_additional_plane", C.c_uint8), ("_reserved", C.c_uint8 * 2)]


PATCH_DTYPE = np.dtype([("u0", "<u4"), ("v0", "<u4"), ("size_u0", "<u4"), ("size_v0", "<u4"),
                        ("u1", "<u4"), ("v1", "<u4"), ("d1", "<u4"), ("lod_x", "<u2"), ("lod_y", "<u2"),
                        ("normal_axis", "u1"), ("tangent_axis", "u1"), ("bitangent_axis", "u1"),
                        ("projection_mode", "u1"), ("patch_orientation", "u1"),
                        ("axis_of_additional_plane", "u1"), ("_reserved", "u1", (2,))])
assert PATCH_DTYPE.itemsize == C.sizeof(CPatch) == 40


class CParams(C.Structure):
    _fields_ = [("occupancy_resolution", C.c_uint32), ("occupancy_precision", C.c_uint32),
                ("map_count_minus1", C.c_uint8), ("absolute_d1", C.c_uint8), ("geometry_bitdepth_3d", C.c_uint8),
                ("attribute_count", C.c_uint8), ("orientation_mode", C.c_uint8),
                ("enable_size_quantization", C.c_uint8), ("multiple_streams", C.c_uint8), ("pbf_enabled", C.c_uint8),
                ("enhanced_occupancy_map", C.c_uint8), ("point_local_reconstruction", C.c_uint8),
                ("single_map_pixel_interleaving", C.c_uint8), ("use_additional_points_patch", C.c_uint8),
                ("geometry_smoothing", C.c_uint8), ("color_smoothing", C.c_uint8), ("attribute_bitdepth", C.c_uint8),
                ("_reserved0", C.c_uint8),
                ("grid_size", C.c_uint16), ("threshold_smoothing", C.c_uint16), ("cgrid_size", C.c_uint16),
                ("threshold_color_smoothing", C.c_uint16), ("threshold_color_difference", C.c_uint16),
                ("threshold_color_variation", C.c_uint16)]


class CFrame(C.Structure):
    _fields_ = [("occ", C.c_void_p), ("geo", C.c_void_p * 2), ("attr_y", C.c_void_p * 2),
                ("attr_u", C.c_void_p * 2), ("attr_v", C.c_void_p * 2), ("patches", C.c_void_p),
                ("patch_count", C.c_uint32), ("occ_stride", C.c_uint32), ("geo_stride", C.c_uint32),
                ("attr_stride_y", C.c_uint32), ("attr_stride_c", C.c_uint32), ("_reserved", C.c_uint32)]


class CGof(C.Structure):
    _fields_ = [("width", C.c_uint32), ("height", C.c_uint32), ("occ_width", C.c_uint32), ("occ_height", C.c_uint32),
                ("frame_count", C.c_uint32), ("geo_video_frames", C.c_uint32), ("attr_video_frames", C.c_uint32),
                ("input_flags", C.c_uint32), ("frames", C.POINTER(CFrame)), ("params", CParams)]


class CFrameOut(C.Structure):
    _fields_ = [("frame_index", C.c_uint64), ("point_count", C.c_uint64), ("positions", C.c_void_p),
                ("colors", C.c_void_p), ("with_colors", C.c_uint8), ("memory_space", C.c_uint8), ("device", C.c_uint8),
                ("_reserved", C.c_uint8 * 5),
                ("smoothed_positions", C.c_uint64), ("smoothed_colors", C.c_uint64), ("_handle", C.c_void_p)]


class CLimits(C.Structure):
    _fields_ = [("max_width", C.c_uint32), ("max_height", C.c_uint32), ("max_frames", C.c_uint32),
                ("max_patches_per_frame", C.c_uint32), ("gofs_in_flight", C.c_uint32), ("flags", C.c_uint32)]


class CPointCloudOut(C.Structure):
    _fields_ = [("capacity_points", C.c_uint64), ("point_count", C.c_uint64), ("positions", C.c_void_p),
                ("colors", C.c_void_p), ("colors16bit", C.c_void_p), ("partition", C.c_void_p),
                ("point_to_pixel", C.c_void_p), ("occupancy_map", C.c_void_p), ("block_to_patch", C.c_void_p),
                ("boundary_type", C.c_void_p), ("positions_presmooth", C.c_void_p),
                ("colors16bit_presmooth", C.c_void_p), ("smoothed_positions", C.c_uint64),
                ("smoothed_colors", C.c_uint64)]


# ---- host-side descriptions -------------------------------------------------------------------------------------
@dataclass
class Params:
    """Mirror of ``GeneratePointCloudParams`` (src/codec.rs:140-170) + smoothing parameter surface."""
    occupancy_resolution: int = 16
    occupancy_precision: int = 4
    map_count_minus1: int = 1
    absolute_d1: bool = True
    geometry_bitdepth_3d: int = 10
    attribute_count: int = 1
    orientation_mode: int = ORIENTATION_REFERENCE
    enable_size_quantization: bool = False
    multiple_streams: bool = False
    pbf_enabled: bool = False
    enhanced_occupancy_map: bool = False
    point_local_reconstruction: bool = False
    single_map_pixel_interleaving: bool = False
    use_additional_points_patch: bool = False
    geometry_smoothing: bool = False
    color_smoothing: bool = False
    attribute_bitdepth: int = 10
    grid_size: int = 8
    threshold_smoothing: int = 64
    cgrid_size: int = 4
    threshold_color_smoothing: int = 10
    threshold_color_difference: int = 10
    threshold_color_variation: int = 6

    def to_c(self) -> CParams:
        c = CParams()
        for name, _ in CParams._fields_:
            if name.startswith("_"):
                continue
            setattr(c, name, int(getattr(self, name)))
        return c


@dataclass
class Gof:
    """Decoded planes + patch lists of one group of frames.

    occ    [F, occH, occW] u8      reference ``atlas.occ_frames``           (Video<u8>)
    geo    [F, 2, H, W]   u16      reference ``atlas.geo_frames[0]``  frame f*2+m, channel 0
    attr_y [F, 2, H, W]   u16      reference ``atlas.attr_frames[0]`` frame f*2+m, channel 0
    attr_u/attr_v [F, 2, H/2, W/2] u16  channels 1, 2 (4:2:0)
    patches: one PATCH_DTYPE array per frame (``tile.patches``)

    Planes are numpy arrays (host memory) or, all of them, objects exposing ``__cuda_array_interface__`` such as torch
    CUDA tensors (device memory, ``TMC2_INPUT_DEVICE``; 16-bit planes may be int16 tensors, their bits are read as u16).
    ``plane_format="p010"`` (device planes only): geo / attr_y samples hold the value in bits 15..6, ``attr_u`` is the
    interleaved UV array [F, 2, H/2, W] (U first) and ``attr_v`` is None.
    """
    width: int
    height: int
    occ: np.ndarray
    geo: np.ndarray
    attr_y: Optional[np.ndarray]
    attr_u: Optional[np.ndarray]
    attr_v: Optional[np.ndarray]
    patches: List[np.ndarray]
    params: Params = field(default_factory=Params)
    geo_video_frames: Optional[int] = None
    attr_video_frames: Optional[int] = None
    plane_format: str = "planar"

    @property
    def frame_count(self) -> int:
        iface = getattr(self.occ, "__cuda_array_interface__", None)
        return int(iface["shape"][0] if iface is not None else self.occ.shape[0])

    def input_bytes(self) -> int:
        n = self.occ.nbytes + self.geo.nbytes
        for a in (self.attr_y, self.attr_u, self.attr_v):
            if a is not None:
                n += a.nbytes
        return n + sum(p.nbytes for p in self.patches)

    def subset(self, frames: Sequence[int]) -> "Gof":
        idx = list(frames)
        sel = lambda a: None if a is None else np.ascontiguousarray(a[idx])
        return Gof(self.width, self.height, sel(self.occ), sel(self.geo), sel(self.attr_y), sel(self.attr_u),
                   sel(self.attr_v), [self.patches[i] for i in idx], self.params)


class _Plane:
    """Address arithmetic over a plane array: numpy (host) or ``__cuda_array_interface__`` (device)."""

    def __init__(self, name, a):
        self.name = name
        iface = getattr(a, "__cuda_array_interface__", None)
        self.device = iface is not None
        if self.device:
            self.shape = tuple(iface["shape"])
            self.itemsize = int(iface["typestr"][2:])
            if iface["typestr"][1] not in "ui":
                raise ValueError(f"{name}: integer samples expected, got {iface['typestr']}")
            strides = iface.get("strides")
            if strides is None:                   # C-contiguous
                strides, acc = [], self.itemsize
                for n in reversed(self.shape):
                    strides.insert(0, acc)
                    acc *= n
            self.strides = tuple(strides)
            self.base = int(iface["data"][0])
            self.torch_device = getattr(getattr(a, "device", None), "index", None)
        else:
            self.shape, self.strides, self.itemsize = a.shape, a.strides, a.itemsize
            self.base = a.ctypes.data

    def ptr(self, *idx):
        return self.base + sum(i * s for i, s in zip(idx, self.strides))

    def pitch(self):
        # rows may be padded (ffmpeg's linesize > width): samples of a row contiguous, row pitch a multiple of the sample size
        # -- the pitch travels in the *_stride fields (the reference itself assumes tight planes)
        s, isz = self.strides, self.itemsize
        if s[-1] != isz or s[-2] % isz or s[-2] < self.shape[-1] * isz:
            raise ValueError(f"{self.name}: rows must be contiguous runs of samples (row pitch >= width)")
        return s[-2] // isz


class GofView:
    """Builds (and keeps alive) the ``tmc2_gof`` C view of a :class:`Gof`."""

    def __init__(self, gof: Gof):
        self.gof = gof
        F = gof.frame_count
        if gof.plane_format not in ("planar", "p010"):
            raise ValueError(f"plane_format {gof.plane_format!r}: 'planar' or 'p010'")
        p010 = gof.plane_format == "p010"
        names = ["occ", "geo"] + (["attr_y", "attr_u"] + ([] if p010 else ["attr_v"]) if gof.attr_y is not None else [])
        if p010 and gof.attr_v is not None:
            raise ValueError("p010: attr_u is the interleaved UV array and attr_v must be None")
        pl = {n: _Plane(n, getattr(gof, n)) for n in names}
        on_device = {p.device for p in pl.values()}
        if len(on_device) > 1:
            raise ValueError("host (numpy) and device (__cuda_array_interface__) planes mixed in one GOF")
        self.device_input = on_device == {True}
        if p010 and not self.device_input:
            raise ValueError("p010 planes must be device arrays (host P010 is not supported)")
        if pl["occ"].itemsize != 1 or any(pl[n].itemsize != 2 for n in names[1:]):
            raise ValueError("occ must hold 8-bit samples, geo / attr_* 16-bit samples")
        # CUDA devices of the planes, where the producer tells (torch tensors): codec synchronises their current streams
        self.devices = sorted({p.torch_device for p in pl.values() if self.device_input and p.torch_device is not None})
        self._frames = (CFrame * max(F, 1))()
        self._keep = []
        for f in range(F):
            fr = self._frames[f]
            fr.occ = pl["occ"].ptr(f)
            fr.occ_stride = pl["occ"].pitch()
            for m in range(2):
                fr.geo[m] = pl["geo"].ptr(f, m) if pl["geo"].shape[1] > m else None
                if gof.attr_y is not None:
                    fr.attr_y[m] = pl["attr_y"].ptr(f, m)
                    fr.attr_u[m] = pl["attr_u"].ptr(f, m)
                    fr.attr_v[m] = None if p010 else pl["attr_v"].ptr(f, m)
            fr.geo_stride = pl["geo"].pitch()
            if gof.attr_y is not None:
                fr.attr_stride_y = pl["attr_y"].pitch()
                fr.attr_stride_c = pl["attr_u"].pitch()
                if not p010 and pl["attr_v"].pitch() != fr.attr_stride_c:
                    raise ValueError("attr_u and attr_v must share one row pitch")
            p = np.ascontiguousarray(gof.patches[f], dtype=PATCH_DTYPE)
            self._keep.append(p)
            fr.patches = p.ctypes.data if len(p) else None
            fr.patch_count = len(p)
        g = CGof()
        g.width, g.height = gof.width, gof.height
        g.occ_height, g.occ_width = pl["occ"].shape[1], pl["occ"].shape[2]
        g.frame_count = F
        g.geo_video_frames = gof.geo_video_frames if gof.geo_video_frames is not None else F * pl["geo"].shape[1]
        if gof.attr_video_frames is not None:
            g.attr_video_frames = gof.attr_video_frames
        else:
            g.attr_video_frames = 0 if gof.attr_y is None else F * pl["attr_y"].shape[1]
        g.input_flags = (INPUT_DEVICE if self.device_input else 0) | (INPUT_P010 if p010 else 0)
        g.frames = C.cast(self._frames, C.POINTER(CFrame))
        g.params = gof.params.to_c()
        self.c = g

    def ref(self):
        return C.byref(self.c)
