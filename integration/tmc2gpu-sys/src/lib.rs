//! Raw bindings of `include/tmc2gpu.h` (ABI version 1) plus a small safe wrapper shaped for
//! tmc2-rs `decoder::Decoder::decode` (src/decoder.rs:185-314).  See INTEGRATION.md.
#![allow(non_camel_case_types)]
use std::ffi::CStr;
use std::os::raw::{c_char, c_int, c_void};

pub const TMC2GPU_ABI_VERSION: u32 = 1;
pub const TMC2_OK: c_int = 0;
pub const TMC2_END: c_int = 1;

#[repr(C)]
#[derive(Clone, Copy, Default, Debug)]
pub struct tmc2_patch {
    pub u0: u32,
    pub v0: u32,
    pub size_u0: u32,
    pub size_v0: u32,
    pub u1: u32,
    pub v1: u32,
    pub d1: u32,
    pub lod_x: u16,
    pub lod_y: u16,
    pub normal_axis: u8,
    pub tangent_axis: u8,
    pub bitangent_axis: u8,
    pub projection_mode: u8,
    pub patch_orientation: u8,
    pub axis_of_additional_plane: u8,
    pub _reserved: [u8; 2],
}

#[repr(C)]
#[derive(Clone, Copy, Default, Debug)]
pub struct tmc2_params {
    pub occupancy_resolution: u32,
    pub occupancy_precision: u32,
    pub map_count_minus1: u8,
    pub absolute_d1: u8,
    pub geometry_bitdepth_3d: u8,
    pub attribute_count: u8,
    pub orientation_mode: u8,
    pub enable_size_quantization: u8,
    pub multiple_streams: u8,
    pub pbf_enabled: u8,
    pub enhanced_occupancy_map: u8,
    pub point_local_reconstruction: u8,
    pub single_map_pixel_interleaving: u8,
    pub use_additional_points_patch: u8,
    pub geometry_smoothing: u8,
    pub color_smoothing: u8,
    pub attribute_bitdepth: u8,
    pub _reserved0: u8,
    pub grid_size: u16,
    pub threshold_smoothing: u16,
    pub cgrid_size: u16,
    pub threshold_color_smoothing: u16,
    pub threshold_color_difference: u16,
    pub threshold_color_variation: u16,
}

#[repr(C)]
pub struct tmc2_frame {
    pub occ: *const u8,
    pub geo: [*const u16; 2],
    pub attr_y: [*const u16; 2],
    pub attr_u: [*const u16; 2],
    pub attr_v: [*const u16; 2],
    pub patches: *const tmc2_patch,
    pub patch_count: u32,
    pub occ_stride: u32,
    pub geo_stride: u32,
    pub attr_stride_y: u32,
    pub attr_stride_c: u32,
    pub _reserved: u32,
}

#[repr(C)]
pub struct tmc2_gof {
    pub width: u32,
    pub height: u32,
    pub occ_width: u32,
    pub occ_height: u32,
    pub frame_count: u32,
    pub geo_video_frames: u32,
    pub attr_video_frames: u32,
    pub input_flags: u32, // TMC2_INPUT_* bits; 0 = every plane in host memory
    pub frames: *const tmc2_frame,
    pub params: tmc2_params,
}

#[repr(C)]
pub struct tmc2_frame_out {
    pub frame_index: u64,
    pub point_count: u64,
    pub positions: *const u16,
    pub colors: *const u8,
    pub with_colors: u8,
    pub memory_space: u8, // 0 = pinned host memory, 1 = device memory (TMC2_CTX_DEVICE_OUTPUT)
    pub device: u8,
    pub _reserved: [u8; 5],
    pub smoothed_positions: u64,
    pub smoothed_colors: u64,
    pub _handle: *mut c_void,
}

#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct tmc2_limits {
    pub max_width: u32,
    pub max_height: u32,
    pub max_frames: u32,
    pub max_patches_per_frame: u32,
    pub gofs_in_flight: u32,
    pub flags: u32,
}

pub enum tmc2gpu_ctx {}

extern "C" {
    pub fn tmc2gpu_abi_version() -> u32;
    pub fn tmc2gpu_device_count() -> c_int;
    pub fn tmc2gpu_create(device_ids: *const c_int, device_count: c_int, limits: *const tmc2_limits, out_ctx: *mut *mut tmc2gpu_ctx) -> c_int;
    pub fn tmc2gpu_destroy(ctx: *mut tmc2gpu_ctx);
    pub fn tmc2gpu_last_error(ctx: *const tmc2gpu_ctx) -> *const c_char;
    pub fn tmc2gpu_status_string(s: c_int) -> *const c_char;
    pub fn tmc2gpu_alloc_pinned(bytes: usize) -> *mut c_void;
    pub fn tmc2gpu_free_pinned(p: *mut c_void);
    pub fn tmc2gpu_submit_gof(ctx: *mut tmc2gpu_ctx, gof: *const tmc2_gof) -> c_int;
    pub fn tmc2gpu_wait_inputs(ctx: *mut tmc2gpu_ctx) -> c_int;
    pub fn tmc2gpu_next_frame(ctx: *mut tmc2gpu_ctx, out: *mut tmc2_frame_out) -> c_int;
    pub fn tmc2gpu_release_frame(ctx: *mut tmc2gpu_ctx, out: *mut tmc2_frame_out) -> c_int;
    pub fn tmc2gpu_frame_to_ply(ctx: *mut tmc2gpu_ctx, frame: *const tmc2_frame_out, format: u32, dst: *mut c_void, dst_capacity: u64, file_bytes: *mut u64) -> c_int;
}
pub const TMC2_INPUT_DEVICE: u32 = 1; // every plane of the GOF is CUDA device memory (NVDEC / ffmpeg CUDA hwaccel)
pub const TMC2_INPUT_P010: u32 = 2; // 16-bit planes in P010 layout (value in bits 15..6, interleaved UV in attr_u)
pub const TMC2_PLY_ASCII: u32 = 0;
pub const TMC2_PLY_BINARY_LE: u32 = 1;

/// One reconstructed frame: the payload of reference `PointSet3` (src/codec.rs:20-36).
pub struct Frame {
    pub positions: Vec<[u16; 3]>,
    pub colors: Option<Vec<[u8; 3]>>,
}

/// Owns a `tmc2gpu_ctx`; one per decoder worker thread (src/lib.rs:113).  `!Sync` like the reference's `Context`.
pub struct Reconstructor {
    ctx: *mut tmc2gpu_ctx,
}

impl Reconstructor {
    pub fn new(devices: &[c_int]) -> Result<Self, String> {
        let mut ctx = std::ptr::null_mut();
        let lim = tmc2_limits { gofs_in_flight: 2, ..Default::default() };
        let st = unsafe { tmc2gpu_create(devices.as_ptr(), devices.len() as c_int, &lim, &mut ctx) };
        if st != TMC2_OK {
            return Err(unsafe { CStr::from_ptr(tmc2gpu_status_string(st)) }.to_string_lossy().into_owned());
        }
        Ok(Self { ctx })
    }

    fn check(&self, st: c_int) -> Result<(), String> {
        if st == TMC2_OK {
            Ok(())
        } else {
            Err(unsafe { CStr::from_ptr(tmc2gpu_last_error(self.ctx)) }.to_string_lossy().into_owned())
        }
    }

    /// Replaces the frame loop src/decoder.rs:188-305 for one GOF.
    ///
    /// Lifetime of the inputs (see "INPUT LIFETIME" in include/tmc2gpu.h): the `tmc2_gof` / `tmc2_frame` structs and the
    /// patch lists are only read during this call.  Planes in ordinary memory (`Vec<u8>`, src/decoder.rs:1136-1140) are
    /// copied into the library's staging area before this returns and may be dropped at once.  Planes inside a
    /// `tmc2gpu_alloc_pinned` block are read by the DMA engine AFTER this returns: keep them unmodified until
    /// [`Reconstructor::wait_inputs`] has returned (or the first frame of the GOF has come back from `next_frame`).
    pub fn submit_gof(&mut self, gof: &tmc2_gof) -> Result<(), String> {
        self.check(unsafe { tmc2gpu_submit_gof(self.ctx, gof) })
    }

    /// Blocks until the host-to-device copies of every GOF submitted so far are done: pinned input planes may then be
    /// overwritten with the samples of the next GOF.
    pub fn wait_inputs(&mut self) -> Result<(), String> {
        self.check(unsafe { tmc2gpu_wait_inputs(self.ctx) })
    }

    /// Next frame in order (src/lib.rs:81); `None` when every submitted frame has been returned.
    pub fn next_frame(&mut self) -> Result<Option<Frame>, String> {
        let mut out: tmc2_frame_out = unsafe { std::mem::zeroed() };
        let st = unsafe { tmc2gpu_next_frame(self.ctx, &mut out) };
        if st == TMC2_END {
            return Ok(None);
        }
        self.check(st)?;
        let n = out.point_count as usize;
        // cgmath Vector3<T> is #[repr(C)]: [T; 3] has the same layout
        let positions = unsafe { std::slice::from_raw_parts(out.positions as *const [u16; 3], n) }.to_vec();
        let colors = if out.with_colors != 0 {
            Some(unsafe { std::slice::from_raw_parts(out.colors as *const [u8; 3], n) }.to_vec())
        } else {
            None
        };
        self.check(unsafe { tmc2gpu_release_frame(self.ctx, &mut out) })?;
        Ok(Some(Frame { positions, colors }))
    }
}

impl Reconstructor {
    /// Next frame in order as a finished PLY file (what `PlyWriter::write`, src/writer.rs:24-75, would put on disk for it),
    /// formatted on the GPU; `None` when every submitted frame has been returned.
    pub fn next_frame_ply(&mut self, format: u32) -> Result<Option<Vec<u8>>, String> {
        let mut out: tmc2_frame_out = unsafe { std::mem::zeroed() };
        let st = unsafe { tmc2gpu_next_frame(self.ctx, &mut out) };
        if st == TMC2_END {
            return Ok(None);
        }
        self.check(st)?;
        let mut size: u64 = 0;
        let mut st = unsafe { tmc2gpu_frame_to_ply(self.ctx, &out, format, std::ptr::null_mut(), 0, &mut size) };
        let mut file = vec![0u8; size as usize];
        if st == TMC2_OK {
            st = unsafe { tmc2gpu_frame_to_ply(self.ctx, &out, format, file.as_mut_ptr() as *mut c_void, size, &mut size) };
        }
        let released = unsafe { tmc2gpu_release_frame(self.ctx, &mut out) };
        self.check(st)?;
        self.check(released)?;
        Ok(Some(file))
    }
}

impl Drop for Reconstructor {
    fn drop(&mut self) {
        unsafe { tmc2gpu_destroy(self.ctx) }
    }
}
