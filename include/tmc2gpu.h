/*
 * tmc2gpu.h -- C ABI of the B200-native V-PCC rec0 reconstruction path.
 *
 * This is the drop-in boundary for the code tmc2-rs runs between "all three videos of the
 * GOF are decoded" (reference src/decoder.rs:180) and `tx.send(reconstruct)` (src/decoder.rs:311):
 *
 *   src/codec.rs:205-250    generate_block_to_patch_from_occupancy_map_video
 *   src/codec.rs:256-514    generate_point_cloud (occupancy upsample, unpack loop, attribute fetch)
 *   src/codec.rs:517-565    generate_points
 *   src/codec.rs:569-658    color_point_cloud
 *   src/codec.rs:661-687    convert_yuv10_to_rgb8   (through PointSet3::convert_yuv16_to_rgb8, :88-94)
 *   src/decoder.rs:827-888  Patch::{patch_block_to_canvas_block, patch_to_canvas, generate_point}
 *   src/decoder.rs:973-1020 Image::get (plane indexing, 4:2:0 nearest chroma, native-endian u16)
 *   src/decoder.rs:188-314  per-frame driver (the caller this library replaces)
 *
 * plus the three post-processing stages the reference only stubs (`unimplemented!`,
 * src/decoder.rs:291-299, src/codec.rs:498-500): boundary-point detection, grid geometry
 * smoothing, grid colour smoothing.  Their arithmetic is this repository's own frozen integer
 * specification (DESIGN.md, "Smoothing specification"); upstream parity for them is unpinned.
 *
 * Plain C: pointers, sizes, PODs.  No torch / CUDA types cross this boundary (a CUDA stream is
 * passed as an opaque `void*`).  Every entry point returns a tmc2_status; nothing aborts.  Where the
 * reference panics (assert!/unwrap/unimplemented!) the matching status code is documented below.
 */
#ifndef TMC2GPU_H
#define TMC2GPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TMC2GPU_ABI_VERSION 1u

#if defined(_WIN32)
#define TMC2_API
#else
#define TMC2_API __attribute__((visibility("default")))
#endif

/* ------------------------------------------------------------------------------------------------
 * Status codes.  0 == success; TMC2_END is the non-error "no more frames" answer of next_frame.
 * ---------------------------------------------------------------------------------------------- */
typedef enum tmc2_status {
  TMC2_OK                      = 0,
  TMC2_END                     = 1,  /* next_frame: every submitted frame was already returned            */
  TMC2_ERR_INVALID_ARG         = 2,  /* NULL pointer, zero size, stride < width, ...                      */
  TMC2_ERR_PATCH_OUT_OF_CANVAS = 3,  /* reference: assert! in decoder.rs:835 / :848                       */
  TMC2_ERR_SHORT_VIDEO         = 4,  /* reference: codec.rs:318-320 returns None -> unwrap panic at       */
                                     /*            decoder.rs:271; attribute video < 2 frames codec.rs:589 */
  TMC2_ERR_MAP_COUNT           = 5,  /* reference: map_count != 2 panics at codec.rs:415/:432             */
  TMC2_ERR_UNSUPPORTED         = 6,  /* reference: unimplemented!() branch (pbf, eom, plr, raw, ...)      */
  TMC2_ERR_CAPACITY            = 7,  /* GOF larger than the limits given to tmc2gpu_create                */
  TMC2_ERR_STATE               = 8,  /* call order violated (e.g. release of a frame not handed out)      */
  TMC2_ERR_NO_DEVICE           = 9,  /* no CUDA device / bad device id.  There is NO CPU fallback.        */
  TMC2_ERR_CUDA                = 10, /* a CUDA call or kernel failed; see tmc2gpu_last_error              */
  TMC2_ERR_INTERNAL            = 11  /* watchdog tripped inside a kernel (should never happen)            */
} tmc2_status;

/* ------------------------------------------------------------------------------------------------
 * Patch: the fields of reference `Patch` (src/decoder.rs:711-783) that the hot path reads, as filled
 * by create_patch_frame (src/decoder.rs:427-473).  Field names follow the reference.
 * ---------------------------------------------------------------------------------------------- */
typedef enum tmc2_patch_orientation { /* src/decoder.rs:694-707 */
  TMC2_ORIENT_DEFAULT = 0, TMC2_ORIENT_SWAP = 1, TMC2_ORIENT_ROT90 = 2, TMC2_ORIENT_ROT180 = 3,
  TMC2_ORIENT_ROT270 = 4, TMC2_ORIENT_MIRROR = 5, TMC2_ORIENT_MROT90 = 6, TMC2_ORIENT_MROT180 = 7,
  TMC2_ORIENT_MROT270 = 8
} tmc2_patch_orientation;

typedef struct tmc2_patch {
  uint32_t u0, v0;            /* uv0: location in the packed image, in occupancy blocks (pdu.pos_2d)      */
  uint32_t size_u0, size_v0;  /* size_uv0: size in occupancy blocks (size_2d_minus1 + 1)                  */
  uint32_t u1, v1;            /* uv1: tangential / bitangential shift (pdu.pos_3d_offset)                 */
  uint32_t d1;                /* depth shift, already mode-adjusted (decoder.rs:468-473)                  */
  uint16_t lod_x, lod_y;      /* level_of_detail; the reference always has (1,1) (decoder.rs:432-436)     */
  uint8_t  normal_axis;       /* axes.0  in {0,1,2}                                                       */
  uint8_t  tangent_axis;      /* axes.1                                                                   */
  uint8_t  bitangent_axis;    /* axes.2                                                                   */
  uint8_t  projection_mode;   /* 0: depth + d1 ; 1: max(d1,depth) - depth (decoder.rs:881-888)            */
  uint8_t  patch_orientation; /* tmc2_patch_orientation                                                   */
  uint8_t  axis_of_additional_plane; /* must be 0 (codec.rs:429-439 unimplemented otherwise)              */
  uint8_t  _reserved[2];
} tmc2_patch;

/* How the six rotated / mirrored orientations are evaluated at PIXEL level (SURVEY.md Appendix B):
 * REFERENCE reproduces decoder.rs:853-866 literally (size_uv0 stays in blocks -> the reference's quirk,
 * bit-exact with tmc2-rs); SPEC multiplies size_uv0 by the occupancy resolution (ISO/IEC 23090-5).
 * Default and Swap are identical in both modes. */
typedef enum tmc2_orientation_mode { TMC2_ORIENTATION_REFERENCE = 0, TMC2_ORIENTATION_SPEC = 1 } tmc2_orientation_mode;

/* ------------------------------------------------------------------------------------------------
 * Parameters: reference `GeneratePointCloudParams` (src/codec.rs:140-170) + the smoothing parameter
 * surface (GeometrySmoothingParams :188-193, ColorSmoothingParams :180-186).
 * ---------------------------------------------------------------------------------------------- */
typedef struct tmc2_params {
  uint32_t occupancy_resolution;   /* 1 << log2_patch_packing_block_size (decoder.rs:252,602)              */
  uint32_t occupancy_precision;    /* vps.frame_width / occ.width() (decoder.rs:194)                       */
  uint8_t  map_count_minus1;       /* must be 1 (two maps) -> else TMC2_ERR_MAP_COUNT                      */
  uint8_t  absolute_d1;            /* decoder.rs:605                                                       */
  uint8_t  geometry_bitdepth_3d;   /* gi.geometry_3d_coordinates_bitdepth_minus1 + 1 (decoder.rs:625)      */
  uint8_t  attribute_count;        /* 0: positions only; 1: colours too (decoder.rs:133 asserts == 1)      */
  uint8_t  orientation_mode;       /* tmc2_orientation_mode                                                */
  /* Switches whose reference branch is unimplemented!(): any non-zero -> TMC2_ERR_UNSUPPORTED.            */
  uint8_t  enable_size_quantization;       /* codec.rs:303 */
  uint8_t  multiple_streams;               /* codec.rs:314 */
  uint8_t  pbf_enabled;                    /* codec.rs:285 */
  uint8_t  enhanced_occupancy_map;         /* codec.rs:399 */
  uint8_t  point_local_reconstruction;     /* codec.rs:402 */
  uint8_t  single_map_pixel_interleaving;  /* codec.rs:454 */
  uint8_t  use_additional_points_patch;    /* codec.rs:494 */
  /* Post-processing (hook points decoder.rs:291-299). 0 = off, exactly the reference's behaviour.         */
  uint8_t  geometry_smoothing;             /* 1: grid geometry smoothing (needs boundary detection)        */
  uint8_t  color_smoothing;                /* 1: grid colour smoothing on the 16-bit YUV colours           */
  uint8_t  attribute_bitdepth;             /* nominal bit depth of attribute samples (10); scales the      */
                                           /* colour-smoothing thresholds, which are in 8-bit units        */
  uint8_t  _reserved0;
  uint16_t grid_size;                      /* GeometrySmoothingParams._grid_size (SEI grid_size_minus_2+2) */
  uint16_t threshold_smoothing;            /* GeometrySmoothingParams._threshold_smoothing                 */
  uint16_t cgrid_size;                     /* ColorSmoothingParams._cgrid_size                             */
  uint16_t threshold_color_smoothing;      /* ColorSmoothingParams._threshold_color_smoothing              */
  uint16_t threshold_color_difference;     /* ColorSmoothingParams._threshold_color_difference             */
  uint16_t threshold_color_variation;      /* ColorSmoothingParams._threshold_color_variation              */
} tmc2_params;

/* ------------------------------------------------------------------------------------------------
 * Decoded planes of one atlas frame (tile == frame, decoder.rs:200-206) and its patch list.
 * Reference containers: atlas.occ_frames (Video<u8>), atlas.geo_frames[0] / atlas.attr_frames[0]
 * (Video<u16>, frame index f*M+m, codec.rs:317,545,620-624).  Only channel 0 of geometry is read
 * (codec.rs:534,548).  u16 samples are native-endian (decoder.rs:1014).  Strides are in ELEMENTS;
 * the reference assumes stride == width (decoder.rs:976-978) -- pass tight planes for bit parity.
 * ---------------------------------------------------------------------------------------------- */
typedef struct tmc2_frame {
  const uint8_t*    occ;          /* occupancy video frame f, channel 0, occ_width x occ_height u8         */
  const uint16_t*   geo[2];       /* geometry video frames f*2+0 / f*2+1, channel 0, width x height        */
  const uint16_t*   attr_y[2];    /* attribute video frames f*2+m, channel 0, width x height               */
  const uint16_t*   attr_u[2];    /* channel 1, (width/2) x (height/2), 4:2:0                              */
  const uint16_t*   attr_v[2];    /* channel 2                                                             */
  const tmc2_patch* patches;      /* tile.patches, ascending patch index                                   */
  uint32_t          patch_count;
  uint32_t          occ_stride;   /* >= occ_width                                                          */
  uint32_t          geo_stride;   /* >= width                                                              */
  uint32_t          attr_stride_y;/* >= width                                                              */
  uint32_t          attr_stride_c;/* >= width/2                                                            */
  uint32_t          _reserved;
} tmc2_frame;

typedef struct tmc2_gof {
  uint32_t          width, height;         /* tile.width / tile.height == atlas frame size                 */
  uint32_t          occ_width, occ_height; /* size of the occupancy video                                  */
  uint32_t          frame_count;           /* frames to reconstruct (decoder.rs:188)                       */
  uint32_t          geo_video_frames;      /* atlas.geo_frames[0].frame_count(); must be >= 2*frame_count   */
  uint32_t          attr_video_frames;     /* atlas.attr_frames[0].frame_count()                           */
  uint32_t          input_flags;           /* TMC2_INPUT_* bits; 0 = every plane in host memory            */
  const tmc2_frame* frames;                /* frame_count entries                                          */
  tmc2_params       params;
} tmc2_gof;

/* Where the planes of a GOF live and how they are laid out (tmc2_gof.input_flags).  Unknown bits -> TMC2_ERR_INVALID_ARG.
 * TMC2_INPUT_DEVICE: every plane pointer of the GOF (occ, geo, attr_*) is CUDA device (or managed) memory on one of the
 *   context's devices -- what NVDEC or ffmpeg's CUDA hwaccel hands out.  The planes are not copied through the host: one
 *   kernel gathers them into the library's own layout.  Each plane is checked: host memory (tmc2gpu_alloc_pinned blocks
 *   included) and a plane whose extent ((rows-1)*stride + row) runs past the end of its allocation -> TMC2_ERR_INVALID_ARG;
 *   a plane on a device that the reconstructing device cannot reach by peer access -> TMC2_ERR_UNSUPPORTED.
 * TMC2_INPUT_P010 (needs TMC2_INPUT_DEVICE, else TMC2_ERR_UNSUPPORTED): the 16-bit planes use the P010 layout that NVDEC
 *   and ffmpeg's p010le write.  A sample's 10-bit value sits in bits 15..6 (the library reads raw >> 6, the low 6 bits are
 *   ignored).  attr_u[m] is the interleaved UV plane, (width/2) x (height/2) pairs with U first, attr_stride_c counts u16
 *   elements and must be >= width; attr_v[m] must be NULL.  geo[m] is the Y plane of the geometry frame (its chroma is
 *   never read).  The occupancy plane stays plain u8 (the luma plane of an nv12 frame).
 *
 * Feeding AVFrames of ffmpeg's CUDA hwaccel (AV_PIX_FMT_CUDA, sw_format p010le for geometry / attributes, nv12 for
 * occupancy): plane pointer = frame->data[0] (Y) / frame->data[1] (interleaved UV), stride in ELEMENTS = linesize[i] / 2
 * for p010le and linesize[0] for the nv12 occupancy luma; set input_flags = TMC2_INPUT_DEVICE | TMC2_INPUT_P010.       */
#define TMC2_INPUT_DEVICE 1u
#define TMC2_INPUT_P010   2u

/* ------------------------------------------------------------------------------------------------
 * One reconstructed frame == reference `PointSet3` (src/codec.rs:20-36): positions are
 * cgmath Vector3<u16> (x,y,z interleaved, 6 B), colors Vector3<u8> (r,g,b, 3 B); both #[repr(C)].
 * The buffers are pinned host memory owned by the library until tmc2gpu_release_frame.
 * ---------------------------------------------------------------------------------------------- */
typedef struct tmc2_frame_out {
  uint64_t        frame_index;    /* running index over all submitted GOFs (frames come back in order)     */
  uint64_t        point_count;    /* PointSet3::len()                                                      */
  const uint16_t* positions;      /* point_count * 3                                                       */
  const uint8_t*  colors;         /* point_count * 3 ; NULL when attribute_count == 0                      */
  uint8_t         with_colors;    /* PointSet3.with_colors                                                 */
  uint8_t         memory_space;   /* 0: positions / colors are pinned HOST memory; 1: DEVICE memory (TMC2_CTX_DEVICE_OUTPUT) */
  uint8_t         device;         /* CUDA device ordinal that reconstructed the frame (and holds it when memory_space == 1)  */
  uint8_t         _reserved[5];
  uint64_t        smoothed_positions; /* points moved by geometry smoothing (0 when off)                   */
  uint64_t        smoothed_colors;    /* points recoloured by colour smoothing (0 when off)                */
  void*           _handle;        /* library cookie                                                        */
} tmc2_frame_out;

typedef struct tmc2_limits {
  uint32_t max_width, max_height;  /* largest atlas frame the context must accept                          */
  uint32_t max_frames;             /* largest GOF (frames) accepted by one submit                          */
  uint32_t max_patches_per_frame;  /* 0 -> default 4096                                                    */
  uint32_t gofs_in_flight;         /* submit/next_frame pipelining depth, 0 -> default 2                   */
  uint32_t flags;                  /* TMC2_CTX_* bits                                                      */
} tmc2_limits;

#define TMC2_CTX_TWO_PASS_SCAN 1u  /* accepted for compatibility; the unpack is always count / scan / emit   */
/* Device-resident hand-off (SURVEY.md 8f-4): frames are NOT copied to the host; next_frame returns device pointers
 * (frame_out.memory_space == 1, on frame_out.device) that stay valid until every frame of that GOF has been released.
 * For consumers on the same GPU (renderer, encoder, a PLY formatter): the 9 bytes per point of D2H -- 41 % of the PCIe
 * traffic that bounds the streaming path -- are not moved at all.                                                 */
#define TMC2_CTX_DEVICE_OUTPUT 2u

typedef struct tmc2gpu_ctx tmc2gpu_ctx;

/* ---- lifetime ---------------------------------------------------------------------------------- */
TMC2_API uint32_t    tmc2gpu_abi_version(void);
TMC2_API int         tmc2gpu_device_count(void);
TMC2_API tmc2_status tmc2gpu_create(const int* device_ids, int device_count, const tmc2_limits* limits,
                                    tmc2gpu_ctx** out_ctx);
TMC2_API void        tmc2gpu_destroy(tmc2gpu_ctx* ctx);
TMC2_API const char* tmc2gpu_last_error(const tmc2gpu_ctx* ctx);
TMC2_API const char* tmc2gpu_status_string(tmc2_status s);

/* Pinned host memory for zero-staging submits (decode straight into these; SURVEY.md section 8f-2).
 * INPUT LIFETIME.  Planes in ordinary (pageable) memory are copied into the library's own staging area before
 * tmc2gpu_submit_gof returns: the caller may reuse them at once (the reference's `Vec<u8>` planes,
 * src/decoder.rs:1136-1140).  Planes inside a tmc2gpu_alloc_pinned block are read by the DMA engine IN PLACE after
 * submit_gof has returned: they must stay unmodified until tmc2gpu_wait_inputs returns (or until the first frame of that
 * GOF has been handed out by tmc2gpu_next_frame).  The patch lists and the tmc2_gof / tmc2_frame structs themselves are
 * only read during submit_gof.
 * DEVICE PLANES (TMC2_INPUT_DEVICE).  They must be completely written before submit_gof / upload_gof / the stage entry points
 * are called: the library does not wait on the caller's stream (synchronise it first).  They are read on the device after
 * submit_gof has returned and must stay unmodified until tmc2gpu_wait_inputs returns.                                */
TMC2_API void*       tmc2gpu_alloc_pinned(size_t bytes);
TMC2_API void        tmc2gpu_free_pinned(void* p);

/* ---- streaming path: replaces the frame loop src/decoder.rs:188-314 ----------------------------
 * submit_gof validates (everything the reference asserts), stages the planes through pinned memory,
 * and enqueues H2D + kernels + D2H; frames of the GOF are sharded frame-wise over the context's
 * devices.  next_frame blocks until the next frame IN ORDER (src/lib.rs:81) is on the host.
 * A GOF is delivered whole or not at all: when submit_gof fails nothing of it is queued; when a launch fails on the
 * device, next_frame reports the error ONCE, drops every frame of that GOF and frees its slot -- the next call
 * continues with the following GOF (or returns TMC2_END).
 * wait_inputs blocks until the host-to-device copies (device planes: the gather kernel) of every GOF submitted so far have
 * finished, i.e. until pinned or device input planes may be overwritten with the next GOF's samples.  */
TMC2_API tmc2_status tmc2gpu_submit_gof(tmc2gpu_ctx* ctx, const tmc2_gof* gof);
TMC2_API tmc2_status tmc2gpu_wait_inputs(tmc2gpu_ctx* ctx);
TMC2_API tmc2_status tmc2gpu_next_frame(tmc2gpu_ctx* ctx, tmc2_frame_out* out);
TMC2_API tmc2_status tmc2gpu_release_frame(tmc2gpu_ctx* ctx, tmc2_frame_out* out);

/* ---- PLY output: the reference's consumer of a PointSet3 (src/writer.rs:15-75 PlyWriter::write) -------------------
 * The frame `frame` -- as handed out by tmc2gpu_next_frame and not yet released, host or device memory space -- is formatted
 * ON ITS DEVICE from the copy that still sits in HBM, header (write_header, :31-60) and body (write_body, :62-75), and the
 * finished file is copied to `dst` (host memory, pinned or not; or device memory on frame->device).  TMC2_PLY_ASCII is byte for
 * byte the file the reference writes (Format::Ascii); TMC2_PLY_BINARY_LE is the binary_little_endian form the reference lists
 * but leaves commented out (:10-11, :41-46): the same properties (uint x y z, uchar red green blue), 15 bytes per point.
 * *file_bytes receives the size of the file; with dst == NULL nothing is written (size query); a destination that is too
 * small gives TMC2_ERR_CAPACITY (and the size).  Synchronous.                                                          */
#define TMC2_PLY_ASCII     0u
#define TMC2_PLY_BINARY_LE 1u
TMC2_API tmc2_status tmc2gpu_frame_to_ply(tmc2gpu_ctx* ctx, const tmc2_frame_out* frame, uint32_t format,
                                          void* dst, uint64_t dst_capacity, uint64_t* file_bytes);

/* ---- resident path: planes stay in HBM, kernels only (what bench.py's `value` times) ------------
 * upload copies a GOF to device 0 of the context once; reconstruct_resident launches the whole
 * reconstruction on `cuda_stream` (a cudaStream_t, NULL = the context's own stream) and returns
 * without synchronising; resident_counts / resident_fetch read results back (they synchronise).    */
typedef struct tmc2_resident tmc2_resident;
TMC2_API tmc2_status tmc2gpu_upload_gof(tmc2gpu_ctx* ctx, const tmc2_gof* gof, tmc2_resident** out);
TMC2_API tmc2_status tmc2gpu_reconstruct_resident(tmc2gpu_ctx* ctx, tmc2_resident* r, void* cuda_stream);
/* Same with flags.  Relaunches of a resident GOF without smoothing are replayed from a CUDA graph (one API call instead of
 * a dozen); TMC2_LAUNCH_TIMED forces the ordinary launch sequence, which records the events tmc2gpu_last_stage_ms reads. */
#define TMC2_LAUNCH_TIMED 1u
TMC2_API tmc2_status tmc2gpu_reconstruct_resident_ex(tmc2gpu_ctx* ctx, tmc2_resident* r, void* cuda_stream, uint32_t flags);
TMC2_API tmc2_status tmc2gpu_resident_counts(tmc2gpu_ctx* ctx, tmc2_resident* r, uint64_t* point_counts /*[frame_count]*/);
TMC2_API tmc2_status tmc2gpu_resident_fetch(tmc2gpu_ctx* ctx, tmc2_resident* r, uint32_t frame,
                                            uint16_t* positions, uint8_t* colors, uint64_t capacity_points);
TMC2_API tmc2_status tmc2gpu_free_resident(tmc2gpu_ctx* ctx, tmc2_resident* r);
/* Launch bookkeeping of the last reconstruct_resident / submit_gof: number of kernel launches and the
 * algorithmic bytes (SURVEY.md 8d) of the dominant (unpack) kernel for that GOF.                    */
TMC2_API tmc2_status tmc2gpu_last_launch_info(tmc2gpu_ctx* ctx, uint32_t* kernel_launches,
                                              uint64_t* unpack_algorithmic_bytes, uint64_t* total_points);
/* Device time of the unpack kernel alone over the last reconstruct_resident, measured with CUDA
 * events recorded on the launching stream (synchronises). */
TMC2_API tmc2_status tmc2gpu_last_unpack_ms(tmc2gpu_ctx* ctx, float* ms);
/* All stage times of the last launch: ms[0] block_to_patch + owned-slot compaction, [1] unpack emit launches, [2] smoothing
 * finalize / filter / clear launches (geometry + colour), [3] unpack count + slot-scan launches, [4] separate YUV->RGB
 * pass (0: fused into the emit). */
TMC2_API tmc2_status tmc2gpu_last_stage_ms(tmc2gpu_ctx* ctx, float* ms5);

/* ---- stage entry points: one frame, host buffers in and out, synchronous ------------------------
 * These mirror the reference's own function boundaries so parity tests read like the reference.
 * All `out` pointers are optional (NULL = not wanted) unless noted.                                  */

/* src/codec.rs:205 generate_block_to_patch_from_occupancy_map_video.
 * block_to_patch: (width/res)*(height/res) entries, value = patch index + 1, 0 = unowned.            */
TMC2_API tmc2_status tmc2gpu_generate_block_to_patch_from_occupancy_map_video(
    tmc2gpu_ctx* ctx, const tmc2_gof* gof, uint32_t frame_index, uint32_t* block_to_patch);

typedef struct tmc2_point_cloud_out {
  uint64_t  capacity_points;   /* in: room in every per-point array below (worst case 2*width*height)     */
  uint64_t  point_count;       /* out: tile.total_number_of_regular_points (codec.rs:482)                 */
  uint16_t* positions;         /* [n][3]  PointSet3.positions after all enabled post-processing           */
  uint8_t*  colors;            /* [n][3]  PointSet3.colors (RGB8 after convert_yuv16_to_rgb8)             */
  uint16_t* colors16bit;       /* [n][3]  PointSet3.colors16bit (YUV, after colour smoothing if enabled)  */
  uint32_t* partition;         /* [n]     patch index per point (codec.rs:452)                            */
  uint32_t* point_to_pixel;    /* [n][3]  (x, y, map) in tile coordinates (codec.rs:463-472)              */
  uint8_t*  occupancy_map;     /* [height*width] tile.occupancy_map (codec.rs:288-300)                    */
  uint32_t* block_to_patch;    /* [(width/res)*(height/res)]                                              */
  /* post-processing intermediates (only filled when smoothing is enabled) */
  uint8_t*  boundary_type;     /* [n]     0 interior, 1 boundary, 2 second ring                           */
  uint16_t* positions_presmooth;   /* [n][3] positions before geometry smoothing                          */
  uint16_t* colors16bit_presmooth; /* [n][3] YUV before colour smoothing                                  */
  uint64_t  smoothed_positions;    /* out: points moved by geometry smoothing                             */
  uint64_t  smoothed_colors;       /* out: points recoloured by colour smoothing                          */
} tmc2_point_cloud_out;

/* src/codec.rs:256 generate_point_cloud (+ the post-processing and colour conversion the caller does
 * at src/decoder.rs:281-305) for ONE frame of the GOF.                                               */
TMC2_API tmc2_status tmc2gpu_generate_point_cloud(tmc2gpu_ctx* ctx, const tmc2_gof* gof, uint32_t frame_index,
                                                  tmc2_point_cloud_out* out);

/* src/codec.rs:88 PointSet3::convert_yuv16_to_rgb8 over n colours (yuv16 [n][3] -> rgb8 [n][3]). */
TMC2_API tmc2_status tmc2gpu_convert_yuv16_to_rgb8(tmc2gpu_ctx* ctx, const uint16_t* yuv16, uint64_t n, uint8_t* rgb8);

#ifdef __cplusplus
} /* extern "C" */
#endif
#endif /* TMC2GPU_H */
