// device_types.h -- PODs shared by the host runtime (tmc2gpu.cu) and the sm_100a kernels (kernels.cu).
//
// HBM layout of one batch (a GOF, or the slice of a GOF given to one GPU); F frames, M = 2 maps:
//   occ    [F][occ_h][occ_pitch]       u8   low-resolution occupancy video     (reference atlas.occ_frames)
//   geo    [F][2][H][pitch]            u16  geometry video, channel 0 only     (reference atlas.geo_frames[0], frame f*2+m)
//   attr_y [F][2][H][pitch]            u16  attribute video, channel 0         (reference atlas.attr_frames[0])
//   attr_u [F][2][H/2][pitch_c]        u16  channel 1 (4:2:0)      attr_v likewise
//   patches[total]  DevPatch ; slot_rec[n_tiles*kWarpsPerTile] SlotRec ; tile_frame[n_tiles] ; frame_tile_begin[F+1]
//   block_to_patch [F][bw*bh] u32 ; work[n_tiles*kWarpsPerTile] WorkRec (per frame: its owned slots, compacted, in order)
// Pitches are multiples of 64 elements so every 16x16 canvas block row starts on a 32-byte boundary.
// Outputs are per-frame slabs of `cap` points (cap % 16 == 0):  pos [F][cap][3] u16, rgb [F][cap][3] u8, and (debug /
// stage API only) yuv [F][cap][3] u16, partition [F][cap] u16, pixel [F][cap] u32 (x | y<<15 | map<<30), btype [F][cap] u8;
// count [F] u32.
// Smoothing state (per group of frames): voxel-cell tables (GeoCell / ColCell, dense or hashed), per frame two bitmaps over
// the table slots (touched / multi-patch) and a compact list of type-1 boundary points.
#pragma once
#include <cstdint>

namespace tmc2 {

#ifndef TMC2_WARPS_PER_TILE
#define TMC2_WARPS_PER_TILE 8
#endif
constexpr int kWarpsPerTile = TMC2_WARPS_PER_TILE;   // one warp per 16x16 patch block ("slot"); one CTA per tile of slots
constexpr uint32_t kNoPatch = 0xFFFFFFFFu;  // padding slot
constexpr int kSlotPoints = 512;            // max points of a 16x16 block (2 maps)

struct alignas(16) DevPatch { // reference Patch (src/decoder.rs:711-783), pre-digested on the host (64 B = four 16-byte vectors)
  uint32_t u0, v0;           // uv0 (blocks)
  uint32_t size_u0, size_v0; // size_uv0 (blocks)
  // ---- vector 1
  uint32_t u1, v1, d1;       // 3D shifts
  uint16_t lod_x, lod_y;
  // ---- vector 2: everything else the block-aligned unpack path needs
  uint8_t  normal, tangent, bitangent, mode;
  uint8_t  orient;
  uint8_t  aligned;          // 1: a 16x16 patch block is exactly one canvas block and (u,v) -> (x,y) is the affine map
                             //    below (Default / Swap / MRot270 always; the other six in SPEC orientation mode)
  int8_t   ax, ay;           // canvas step per +1 in patch u   (one of them is 0, the other +-1)
  uint32_t sel;              // byte-permute selectors of generate_point (decoder.rs:871-878): selA | selB << 16, see
                             // position_selectors() -- which of normal / tangent / bitangent lands in x, y, z
  uint32_t local_index;      // patch index inside its frame (partition value; block_to_patch holds local_index+1)
  // ---- vector 3
  int8_t   rx, ry;           // canvas step per +1 in patch v
  uint8_t  _pad[2];
  uint32_t slot_base;        // index of this patch's first slot in slot_rec[]
  uint32_t frame;            // frame inside the batch
  uint32_t _pad2;
};
static_assert(sizeof(DevPatch) == 64, "DevPatch is four 16-byte vectors");

// generate_point (decoder.rs:871-878) stores point[normal], point[tangent], point[bitangent] in that order, so a later axis
// overwrites an earlier one if they coincide, and an axis nobody names stays 0.  With A = n | t << 16 and B = b (upper half
// zero) as the two byte-permute operands (bytes 0,1 = n; 2,3 = t; 4,5 = b; 6,7 = zero):
//   word 0 = x | y << 16 = prmt(A, B, selA),  word 1 = z = prmt(A, B, selB).   Host and device share this one definition.
inline __host__ __device__ uint32_t position_selectors(uint32_t normal, uint32_t tangent, uint32_t bitangent) {
  uint32_t s[3];
  for (uint32_t a = 0; a < 3; ++a)
    s[a] = bitangent == a ? 0x54u : tangent == a ? 0x32u : normal == a ? 0x10u : 0x76u;
  return (s[0] | (s[1] << 8)) | ((s[2] | 0x7600u) << 16);
}

// One 16x16 block of one patch ("slot"), in the reference's iteration order (patch, v0, u0): everything the unpack
// kernel needs to start loading planes, digested on the host.
struct alignas(16) SlotRec {
  uint32_t pid;              // index into patches[], kNoPatch = padding
  uint16_t u0b, v0b;         // block inside the patch
  uint16_t bx, by;           // canvas block it maps to (src/decoder.rs:827-837)
  int8_t   ax, ay, rx, ry;   // copy of the patch's affine steps
};

// One owned slot at its position in the frame's compacted list: everything the count / emit warps need in two 16-byte
// loads.  compact_owned_kernel fills the slot part (pid = kNoPatch for the unused tail of a frame's region), count_kernel
// `total`, slot_scan_kernel `base`.
struct alignas(16) WorkRec {
  uint32_t pid;
  uint16_t u0b, v0b;
  uint16_t bx, by;
  int8_t   ax, ay, rx, ry;
  uint32_t frame;            // frame inside the batch (in memory: | projection mode << 31)
  uint32_t total;            // points this slot emits
  uint32_t base;             // first point of its run inside the frame
  uint32_t d1;               // the patch's depth shift (copy, so that count_kernel needs no patch load)
};
static_assert(sizeof(WorkRec) == 32, "WorkRec is two 16-byte vectors");

struct Planes {
  const uint8_t*  occ;
  const uint16_t* geo;
  const uint16_t* attr_y;
  const uint16_t* attr_u;
  const uint16_t* attr_v;
  uint32_t occ_pitch, occ_w, occ_h;
  uint32_t geo_pitch, attr_pitch_y, attr_pitch_c;
  uint64_t occ_frame_stride;     // elements between frames
  uint64_t geo_map_stride;       // elements between maps (frame stride = 2x)
  uint64_t attr_y_map_stride;
  uint64_t attr_c_map_stride;
};

struct Outputs {                // any pointer may be null = stream not wanted
  uint16_t* pos;
  uint8_t*  rgb;
  uint16_t* yuv;
  uint16_t* part;
  uint32_t* pix;
  uint8_t*  btype;
  uint64_t  cap;                // points per frame slab (multiple of 16)
};

// ---- voxel-cell tables of the grid smoothing stages (own spec, DESIGN.md) ------------------------------------------
// The sums of a cell are written only with fire-and-forget reductions (RED): two / three 64-bit adds.  All-zero == empty.
// "multi-patch" (the smoothing trigger) <=> two different patches touched the cell: the first toucher claims `first1` with
// a compare-and-swap (0 -> patch + 1); whoever finds another patch's claim stores 1 into `multi` (idempotent).
// The apply pass computes Q8 means from the sums on the fly (there is no finalize pass).
#ifndef TMC2_TOUCH_SHIFT
#define TMC2_TOUCH_SHIFT 2
#endif
constexpr uint32_t kTouchShift = TMC2_TOUCH_SHIFT;   // log2(cells per bit of the touched bitmap)
constexpr uint32_t kCellEmpty = 0xFFFFFFFFu;      // free slot of a hashed table's key array
struct GeoCell {     // 32 B = one DRAM sector
  uint32_t first1;              // patch index + 1 of the first toucher, 0 = untouched
  uint32_t multi;               // 1 = touched by more than one patch
  unsigned long long cnt_sx;    // count | sum(x - cell origin) << 32
  unsigned long long sy_sz;     // sum(y - origin) | sum(z - origin) << 32
  unsigned long long mean;      // unused (pads the cell to one 32-byte sector)
};
struct ColCell {     // 32 B
  uint32_t first1, multi;
  unsigned long long cnt_sy;    // count (24 bits) | sum(Y) << 24
  unsigned long long su_sv;     // sum(U) | sum(V) << 32
  unsigned long long sy2;       // sum(Y*Y)
};
struct alignas(16) BoundaryEntry {  // one type-1 boundary point (16 B)
  uint32_t idx;         // point index inside its frame
  uint16_t pos[3];      // reconstructed (pre-smoothing) position
  uint16_t yuv[3];      // 16-bit colour
};

struct GridDesc {               // geometry of one voxel grid
  uint32_t on;
  uint32_t g, w, disth, th;     // cell edge, cells per axis, border margin, g*w
  uint32_t magic;               // ceil(2^32 / g): x / g == umulhi(x, magic) for x < 65536
  int32_t  g_shift;             // log2(g) when g is a power of two, else -1
  uint32_t identity;            // 1: slot = dense cell index (table covers the whole grid)
  // fast: dense table, g and w powers of two, g * w == 2^bitdepth (1: w <= 256, cell keys pack into bytes; 2: w <= 1024,
  // direct slot arithmetic only -- colour statistics and the probe).  Then cell coordinates come from shifts and
  // masks on the packed position words (x | y << 16, z): oob_mask = bits that must be zero in every coordinate, replicated
  // in both halves; cmask = (w - 1) in both halves; w_shift = log2(w).
  uint32_t fast, w_shift, oob_mask, cmask;
  uint64_t slots;               // table slots per frame-in-group (power of two unless identity)
  void*    table;               // GeoCell / ColCell [frames_in_group][slots]
  uint32_t* keys;               // hashed tables only: [frames_in_group][slots], kCellEmpty = free
  uint32_t* tbits;              // [frames_in_group][twords] one bit per 4 consecutive table slots (one 128-byte line of cells): some
                                // cell of the quad was touched (set by its first toucher; what the clear pass walks)
  uint32_t* mbits;              // [frames_in_group][mwords] ... the cell is multi-patch (set by whoever finds another patch's claim, read by the probe)
  uint64_t mwords;
  uint64_t twords;              // words per frame of tbits = ceil(slots / 128)
};

struct SmoothArgs {
  GridDesc geo, col;
  BoundaryEntry* blist;         // [F][blist_cap]
  uint32_t* blist_count;        // [F]
  uint64_t blist_cap;
  uint32_t* slist;              // [F][blist_cap] survivors of the probe pass: list index | grids-to-filter << 30
  uint32_t* slist_count;        // [F]
  uint32_t group_first_frame;   // tables are indexed by (frame - group_first_frame)
  uint32_t group_frames;
  uint32_t thr_geo;             // threshold_smoothing
  uint32_t thr_col_smooth, thr_col_diff, thr_col_var;   // colour thresholds, already scaled to the sample bit depth
  unsigned long long* changed;  // [2][F] moved / recoloured points
};

struct UnpackArgs {
  Planes   in;
  Outputs  out;
  uint32_t W, H, res, prec;
  int32_t  prec_shift;          // log2(prec) or -1 when prec is not a power of two
  uint32_t bw, bh;              // block grid (W/res, H/res)
  uint32_t n_frames, n_tiles;
  uint8_t  absolute_d1, spec_orientation, has_attr, want_btype;
  const DevPatch* patches;
  const SlotRec*  slot_rec;
  const uint32_t* tile_frame;
  const uint32_t* frame_tile_begin;   // [F+1]
  const uint32_t* block_to_patch;     // [F][bw*bh]
  WorkRec*        work;               // [n_tiles*kWarpsPerTile] compacted owned slots of each frame, from frame_tile_begin[f]*8
  uint32_t*       owned_count;        // [F]
  uint16_t*       slot_bt;            // [n_tiles*kWarpsPerTile][32] boundary classes of a slot's pixels in canvas layout (lane = row, half):
                                      // type-1 mask | type-2 mask << 8, written by count_kernel when want_btype
  uint16_t*       slot_nmin;          // [n_tiles*kWarpsPerTile] smallest normal coordinate among the slot's points (origin of its cell table)
  uint32_t*       slot_bbase;         // [n_tiles*kWarpsPerTile] count_kernel: type-1 boundary points of the slot; slot_scan_kernel: where its
                                      // entries start in the frame's boundary list (exclusive prefix in slot order)
  uint32_t*       frame_count;        // [F] points per frame
  int*            err;                // device error flag (0 ok)
  SmoothArgs sm;                      // used by the smoothing instantiation only
};

// Shared memory of one warp of emit_kernel (one warp = one slot; warps never talk to each other).
//   RAW area: the plane tiles of the canvas block, written by the TMA unit (cp.async.bulk.tensor, 128-byte aligned boxes,
//   completion on the warp's mbarrier).  It is dead once the tables below have been built; the smoothing instantiations
//   then reuse it for their per-slot state.
constexpr uint32_t kOffRawGeo = 0;                               // [2 maps][16 rows][16] u16  geometry samples of the canvas block
constexpr uint32_t kOffRawY = kOffRawGeo + 1024;                 // [2][16][16] u16            attribute luma
constexpr uint32_t kOffRawU = kOffRawY + 1024;                   // [2][8][8] u16              4:2:0 chroma
constexpr uint32_t kOffRawV = kOffRawU + 256;
constexpr uint32_t kOffRawOcc = kOffRawV + 256;                  // [8 rows][32] u8: occupancy samples from (ox, by*4-2), ox = (bx*4-1) rounded
                                                                 // down to a multiple of 16 (the TMA unit wants the first byte of a box
                                                                 // row 16-byte aligned): the block's 4x4 samples plus the ring around
                                                                 // them that the boundary classes look at
constexpr uint32_t kRawBytes = kOffRawOcc + 256;
constexpr uint32_t kListEntries = 520;
constexpr uint32_t kSrcBytes = 1040;
// The rest of a warp's shared memory depends on the instantiation (byte offsets inside the warp's region):
//   pt    [16 rows][17][2] u32: per-pixel table in PATCH raster order (rank = v1*16 + u1): n | Y << 16 of map 0 / map 1; the 17th
//         pair of a row is padding (bank conflicts), and the warp's mbarrier (`bar`) sits in the padding pair of the last row
//   term  [64][2] uint4: chroma term of (chroma sample, map)
//   src   [3 + 512 (+ slack)] u16: output point -> rank << 1 | map | term << 9; entry i = point i - (run_base & 3) of the run
//         (the run starts at the same phase of a 4-point group as in the frame)
//   cnt   [256] u8: points of the pixel (0..2) | boundary class << 2
//   bmp   [32] u32: 20x20 occupancy bitmap rows (canvas axes); later the list of non-empty cell-table entries
//   memo  [2][32] u32: cells the slot has already claimed (smoothing)
//   tab   [128] uint2: the slot's geometry-cell table; list [520] u16: run-relative indices of the slot's type-1 boundary points
//         from the front, type-2 from the back (fast smoothing grids)
// Whatever is only needed AFTER the tables have been built lives in the RAW area (dead by then):
//   plain  (no smoothing, no debug streams): src and cnt in the RAW area                                         7 040 B
//   fast   (smoothing, dense power-of-two grids): RAW region of 3 104 B holds tab, list and src; memo takes the place of
//          cnt once the point list has been built                                                                7 808 B
//   wide   (debug streams, generic smoothing grids: boundary classes are looked up per point): memo in the RAW area 8 576 B
struct EmitLayout { uint32_t raw, pt, bar, term, src, cnt, bmp, memo, tab, list, bytes; };
__host__ __device__ constexpr EmitLayout emit_layout(bool smooth, bool debug, bool fast) {
  EmitLayout l{};
  const bool compact = smooth && fast && !debug, plain = !smooth && !debug;
  l.raw = compact ? 1024 + 2 * kListEntries + kSrcBytes : kRawBytes;
  l.pt = l.raw; l.bar = l.pt + 2176 - 8; l.term = l.pt + 2176;
  uint32_t end = l.term + 2048;
  if (plain) { l.src = 0; l.cnt = kSrcBytes; l.bmp = 0; l.memo = 0; l.tab = 0; l.list = 0; }
  else if (compact) { l.tab = 0; l.list = 1024; l.src = 1024 + 2 * kListEntries; l.cnt = end; l.memo = l.cnt; l.bmp = end + 256; end += 256 + 128; }
  else { l.memo = 0; l.tab = 256; l.list = 1280; l.src = end; l.cnt = end + kSrcBytes; l.bmp = l.cnt + 256; end = l.bmp + 128; }
  l.bytes = (end + 127) / 128 * 128;
  return l;
}
static_assert(emit_layout(false, false, false).bytes == 7040 && emit_layout(true, false, true).bytes == 7808 && emit_layout(true, true, false).bytes == 8576, "layout sizes");
static_assert(emit_layout(false, false, false).cnt + 256 <= kOffRawU, "plain layout: list and counts overwrite only the geometry / luma tiles");
static_assert(emit_layout(true, false, true).raw >= kRawBytes && emit_layout(true, false, true).src % 16 == 0, "fast layout");
#ifndef TMC2_EMIT_WARPS
#define TMC2_EMIT_WARPS 4
#endif
constexpr int kEmitWarps = TMC2_EMIT_WARPS;                      // warps per CTA of emit_kernel

// TMA descriptors (CUtensorMap, 128 B each) of the five plane arrays of a batch; tiled, no swizzle, u16 / u8 elements:
//   geo, attr_y: (x, y, map, frame) box 16 x 16 x 2 x 1      attr_u, attr_v: box 8 x 8 x 2 x 1      occ: (x, y, frame) box 32 x 8 x 1
struct alignas(64) TileMaps { unsigned long long geo[16], attr_y[16], attr_u[16], attr_v[16], occ[16]; };

// Device-resident input (TMC2_INPUT_DEVICE): one entry per (frame, plane kind, map) of the caller's planes, gathered by
// ingest_planes_kernel into the batch layout above.  The table travels at the end of the batch's metadata block.
enum IngestOp : uint32_t {
  kIngestCopy8 = 0,        // u8 samples, copied
  kIngestCopy16 = 1,       // u16 samples, copied
  kIngestShr16 = 2,        // P010 u16 samples: raw >> 6
  kIngestUv16 = 3,         // P010 interleaved UV pairs: U >> 6 to dst, V >> 6 to dst2
  kIngestVec = 0x100u,     // flag: source base and pitch are 16-byte aligned -> 16-byte vector loads
};
struct alignas(16) IngestPlane {
  const uint8_t* src;      // caller's plane (this device, or a peer device of the context)
  uint8_t* dst;            // plane in the batch layout
  uint8_t* dst2;           // kIngestUv16: the V plane
  uint32_t spitch;         // source row pitch, bytes
  uint32_t dpitch;         // destination row pitch, bytes (a multiple of 64)
  uint32_t rows;
  uint32_t row_bytes;      // source bytes per row
  uint32_t op;             // IngestOp (| kIngestVec)
  uint32_t _pad;
};
static_assert(sizeof(IngestPlane) == 48, "IngestPlane is three 16-byte vectors");

// launch wrappers (kernels.cu); every one enqueues on `stream` and returns the cudaGetLastError() code
int launch_block_to_patch(const UnpackArgs& a, uint32_t n_slots, void* stream);
int launch_compact_owned(const UnpackArgs& a, void* stream);   // after block_to_patch: per-frame list of owned slots
// unpack = count (points per owned slot) -> slot_scan (run starts, per frame) -> emit.  Tiles [tile_begin, tile_end).
// smooth: the emit also accumulates the cell tables and writes the boundary lists of the current frame group.
int launch_count(const UnpackArgs& a, uint32_t tile_begin, uint32_t tile_end, void* stream);
int launch_slot_scan(const UnpackArgs& a, void* stream);
int launch_emit(const UnpackArgs& a, const TileMaps& tm, bool smooth, uint32_t tile_begin, uint32_t tile_end, void* stream);
int launch_upsample(const UnpackArgs& a, uint8_t* occ_full /*[F][H][W]*/, void* stream);
int launch_smooth_filter(const UnpackArgs& a, void* stream);   // boundary points of the current frame group
int launch_smooth_clear(const UnpackArgs& a, void* stream);    // reset touched cells (+ keys) of the group
int launch_yuv_to_rgb_flat(const uint16_t* yuv, uint8_t* rgb, uint64_t n, void* stream);
int launch_fill_u32(uint32_t* p, uint64_t n, uint32_t v, void* stream);
// every plane of `table` (device memory, n_planes entries); max_rows / max_row_bytes over the table size the grid
int launch_ingest_planes(const IngestPlane* table, uint32_t n_planes, uint32_t max_rows, uint32_t max_row_bytes, void* stream);
int kernel_launch_count_reset();   // returns launches since the last reset

// ply.cu: a frame in HBM formatted as the body of a PLY file (src/writer.rs:62-75).  measure -> scan -> write for the ASCII
// form (block_sums / block_offs: one entry per 1024 points; *total = body bytes), write alone for the binary records.
constexpr uint64_t ply_blocks(uint64_t n_points) { return (n_points + 1023u) / 1024u; }
int launch_ply_measure(const uint16_t* pos, const uint8_t* rgb, uint64_t n, uint32_t* block_sums, void* stream);
int launch_ply_scan(const uint32_t* block_sums, uint64_t n, unsigned long long* block_offs, unsigned long long* total, void* stream);
int launch_ply_write(const uint16_t* pos, const uint8_t* rgb, uint64_t n, const unsigned long long* block_offs, uint8_t* body,
                     bool ascii, void* stream);

}  // namespace tmc2
