// kernels.cu -- hand-written sm_100a kernels of the V-PCC rec0 reconstruction path.
//
//   K2  block_to_patch_kernel     src/codec.rs:205-250   (atomicMax == "later patch overwrites", :242-244)
//   K1  upsample_kernel           src/codec.rs:288-300   (materialised only for the stage API; fused otherwise)
//   K3+K4 count_kernel / slot_scan_kernel / emit_kernel
//                                 src/codec.rs:352-480 (unpack loop, order, dedup), :517-565 (generate_points),
//                                 :569-658 (attribute fetch), :661-687 (YUV->RGB), src/decoder.rs:827-888 (patch maths)
//       + K5 boundary class per pixel, K6/K7 cell statistics (own spec) in the smoothing instantiation of emit_kernel
//   K6/K7 smooth_probe_kernel / smooth_apply_kernel / smooth_clear_kernel
//                                 grid geometry + colour smoothing of the boundary points (own integer spec, DESIGN.md;
//                                 the reference has only stubs: decoder.rs:291-299)
//
// Ordering.  The reference emits points in (patch, v0, u0, v1, u1, map) order.  A 16x16 patch block ("slot") that
// owns its canvas block emits one contiguous run, so the output position of a run is an exclusive prefix sum of
// per-slot counts in slot order: count_kernel (points per owned slot), slot_scan_kernel (prefix per frame), emit_kernel
// (a warp per slot writes its run at its final place).  Warps never talk to each other.
//
// A block-aligned slot is loaded in CANVAS layout (lane = canvas row + half: one 16-byte vector per plane, whatever the
// patch orientation), spilled into per-pixel tables in shared memory in PATCH raster order, and emitted by a
// point-parallel loop (lane == point index mod 32) that writes aligned 32-bit words assembled from neighbouring lanes.
//
// All arithmetic on the bit-exact path is integer.  The colour conversion of the reference is IEEE f64; it is evaluated
// here in 32.32 fixed point with a proven error margin, and re-done with the literal f64 sequence (__dmul_rn/__dadd_rn/
// __ddiv_rn, every operation rounded on its own like rustc's code) whenever the fixed-point value is within that margin
// of an integer boundary, so the result is bit-exact for every u16 input.
#include <cuda_runtime.h>
#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <type_traits>

#include "device_types.h"

namespace tmc2 {

static thread_local int g_launches = 0;   // per host thread: the pieces of a GOF are launched from one thread per device
int kernel_launch_count_reset() { int n = g_launches; g_launches = 0; return n; }

constexpr uint32_t kFull = 0xFFFFFFFFu;

// ----------------------------------------------------------------------------------------------------------------
// small helpers
// ----------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31u; }

__device__ __forceinline__ uint32_t div_prec(uint32_t x, uint32_t prec, int shift) {
  return shift >= 0 ? (x >> shift) : (x / prec);
}

__device__ __forceinline__ uint4 ldg_nc_v4(const void* p) {   // streaming 16-byte load, no L1 allocation
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ uint2 ldg_nc_v2(const void* p) {
  uint2 r;
  asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p));
  return r;
}
__device__ __forceinline__ uint32_t ldg_nc_u16(const uint16_t* p) {
  uint16_t r;
  asm volatile("ld.global.nc.u16 %0, [%1];" : "=h"(r) : "l"(p));
  return r;
}
__device__ __forceinline__ unsigned long long ld_relaxed_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_relaxed_u64(unsigned long long* p, unsigned long long v) {
  asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" :: "l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ void stg_cs_v4(void* p, const uint4& v) {   // streaming store: output is never re-read here
  asm volatile("st.global.cs.v4.u32 [%0], {%1,%2,%3,%4};" :: "l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ uint32_t word_of(const uint4& v, int i) { return i == 0 ? v.x : i == 1 ? v.y : i == 2 ? v.z : v.w; }
__device__ __forceinline__ uint32_t word_of(const uint2& v, int i) { return i == 0 ? v.x : v.y; }

// ---- Patch maths, src/decoder.rs:853-888 --------------------------------------------------------------------------
// Forward map patch (u,v) -> canvas (x,y), decoder.rs:853-867.  `sscale` multiplies size_uv0: 1 reproduces the
// reference (sizes stay in blocks even at pixel level), `res` is the spec-correct form.  Signed 64-bit arithmetic: the
// host has verified that every pixel of the patch lands inside the canvas, where wrapping usize and i64 agree.
__device__ __forceinline__ void patch_to_canvas(const DevPatch& P, int64_t u, int64_t v, int64_t res, int64_t sscale,
                                                int64_t& x, int64_t& y) {
  const int64_t u0 = (int64_t)P.u0 * res, v0 = (int64_t)P.v0 * res;
  const int64_t su = (int64_t)P.size_u0 * sscale, sv = (int64_t)P.size_v0 * sscale;
  switch (P.orient) {
    case 0:  x = u + u0;           y = v + v0;           break;   // Default
    case 2:  x = sv - 1 - v + u0;  y = u + v0;           break;   // Rot90
    case 3:  x = su - 1 - u + u0;  y = sv - 1 - v + v0;  break;   // Rot180
    case 4:  x = v + u0;           y = su - 1 - u + v0;  break;   // Rot270
    case 5:  x = su - 1 - u + u0;  y = v + v0;           break;   // Mirror
    case 6:  x = sv - 1 - v + u0;  y = su - 1 - u + v0;  break;   // MRot90
    case 7:  x = u + u0;           y = sv - 1 - v + v0;  break;   // MRot180
    default: x = v + u0;           y = u + v0;           break;   // Swap (1) and MRot270 (8)
  }
}

// generate_normal_coordinate (decoder.rs:881-888), truncated to u16 like the `as u16` cast at :874
__device__ __forceinline__ uint32_t normal_coord(const DevPatch& P, uint32_t depth) {
  const uint32_t n = P.mode == 0 ? depth + P.d1 : (P.d1 > depth ? P.d1 : depth) - depth;
  return n & 0xFFFFu;
}
// generate_point (decoder.rs:871-878) writes point[normal], point[tangent], point[bitangent] in that order, so a later
// axis overwrites an earlier one if they coincide.  axis_source() returns, for output axis `a`, which value lands there:
// 0 nothing, 1 normal, 2 tangent, 3 bitangent.
__device__ __forceinline__ uint32_t axis_source(const DevPatch& P, uint32_t a) {
  return P.bitangent == a ? 3u : P.tangent == a ? 2u : P.normal == a ? 1u : 0u;
}
__device__ __forceinline__ uint32_t pick(uint32_t src, uint32_t n, uint32_t t, uint32_t b) {
  return src == 3u ? b : src == 2u ? t : src == 1u ? n : 0u;
}
// byte-permute selectors that build a staged position from A = n | t << 16 and Bv = b (upper half zero):
// word 0 = pos[0] | pos[1] << 16, word 1 = pos[2].   source nibbles: n -> bytes 0,1 ; t -> 2,3 ; b -> 4,5 ; none -> 6,7
__device__ __forceinline__ uint32_t sel_of_src(uint32_t src) { return src == 1u ? 0x10u : src == 2u ? 0x32u : src == 3u ? 0x54u : 0x76u; }

// ---- convert_yuv10_to_rgb8, src/codec.rs:661-687 ---------------------------------------------------------------------
// literal f64 sequence: one channel = clamp(floor(c / 1023 * 255))
__device__ __forceinline__ uint32_t quant_channel_f64(double c) {
  const double q = floor(__dmul_rn(__ddiv_rn(c, 1023.0), 255.0));
  if (q < 0.0) return 0u;
  if (q > 255.0) return 255u;
  return (uint32_t)q;
}
__device__ __noinline__ uint32_t yuv_to_rgb_f64(uint32_t Y, uint32_t U, uint32_t V) {
  const double y = (double)Y, u = __dsub_rn((double)U, 512.0), v = __dsub_rn((double)V, 512.0);
  const double r = __dadd_rn(y, __dmul_rn(1.57480, v));
  const double g = __dsub_rn(__dsub_rn(y, __dmul_rn(0.18733, u)), __dmul_rn(0.46813, v));
  const double b = __dadd_rn(y, __dmul_rn(1.85563, u));
  return quant_channel_f64(r) | (quant_channel_f64(g) << 8) | (quant_channel_f64(b) << 16);
}
// Exact integer evaluation.  With d = chroma - 512 and t = k*d, a channel is floor(T), T = 255*(Y + t)/1023.
// Write 255*t = I + f with I integer and 0 <= f < 1: then floor((255*Y + I + f)/1023) == floor((255*Y + I)/1023), because
// (255*Y + I)/1023 has a fractional part <= 1022/1023 and f/1023 < 1/1023.  So the chroma-dependent work is done ONCE per
// chroma sample (ChromaTerm: three integers), and a point costs three 32-bit multiply-high divisions.
// Exactness versus the reference's f64 chain: the chain deviates from the real value by < 2e-11, and I, f are computed
// from the f64 constants rounded to 32 fractional bits (error <= 255*|d|/2^33), so floor() can only differ when f is
// within `eps` = 255*|d|/2^33 + 2^-24 of 0 or 1 AND 255*Y + I is congruent to 0 / 1022 mod 1023.  Such chroma samples are
// flagged (a few per million for 10-bit content) and their points take the literal f64 path.
constexpr long long kKr = 6763714498LL;   // 1.57480 * 2^32
constexpr long long kKgu = 804576224LL;   // 0.18733 * 2^32
constexpr long long kKgv = 2010603040LL;  // 0.46813 * 2^32
constexpr long long kKb = 7969870163LL;   // 1.85563 * 2^32
struct ChromaTerm { int32_t ir, ig, ib; uint32_t flagged; };   // flagged: some channel's f is within eps of 0 or 1
__device__ __forceinline__ int32_t chroma_floor(long long p32 /* 255*k*d in 32.32 */, uint32_t eps, uint32_t& flagged) {
  const uint32_t f = (uint32_t)p32;                         // fractional part, units of 2^-32
  flagged |= (f + eps <= 2u * eps) ? 1u : 0u;               // f < eps or f > 2^32 - 1 - eps (unsigned wrap)
  return (int32_t)(p32 >> 32);                              // floor (arithmetic shift)
}
__device__ __forceinline__ ChromaTerm chroma_term(uint32_t U, uint32_t V) {
  const int32_t du = (int32_t)U - 512, dv = (int32_t)V - 512;
  const uint32_t adu = (uint32_t)abs(du), adv = (uint32_t)abs(dv);
  ChromaTerm c;
  c.flagged = 0;
  c.ir = chroma_floor(255LL * kKr * dv, 128u * adv + 256u, c.flagged);
  c.ig = chroma_floor(-(255LL * kKgu) * du - (255LL * kKgv) * dv, 128u * (adu + adv) + 256u, c.flagged);
  c.ib = chroma_floor(255LL * kKb * du, 128u * adu + 256u, c.flagged);
  return c;
}
// The same three integers for 10-bit chroma from 32-bit arithmetic: 255*k = Cint + Cfrac, Cfrac rounded to 21 fractional bits
// (error <= 2^-22 per unit of d, so <= 2^-13 over |d| <= 512; the green channel adds two such terms).  The result is exact
// unless the fraction lands within that error (plus a margin) of 0 or 1 -- 4 603 of the 2^20 chroma pairs, and always for a
// neutral component (d == 0) -- or the sample is not a 10-bit value; then `flagged` is set and the caller takes chroma_term().
// Verified exhaustively over all 2^20 (U, V) pairs against exact rational arithmetic in tests/test_fused_colour.py, which
// also runs every pair through the emit on the luma values where the result turns on these terms.
__device__ __forceinline__ ChromaTerm chroma_term_fast(uint32_t U, uint32_t V) {
  const uint32_t du = U - 512u, dv = V - 512u;                              // two's complement
  constexpr uint32_t M = (1u << 21) - 1u;
  const int32_t sr = (int32_t)(1203765u * dv), sb = (int32_t)(389336u * du);
  const int32_t sg = (int32_t)(0u - 1613024u * du - 782552u * dv);
  ChromaTerm c;
  c.ir = (int32_t)(401u * dv) + (sr >> 21);
  c.ib = (int32_t)(473u * du) + (sb >> 21);
  c.ig = (int32_t)(0u - 47u * du - 119u * dv) + (sg >> 21);
  const bool near = ((((uint32_t)sr & M) + 264u) & M) < 528u || ((((uint32_t)sb & M) + 264u) & M) < 528u ||
                    ((((uint32_t)sg & M) + 520u) & M) < 1040u;
  c.flagged = (near || (U | V) > 1023u) ? 1u : 0u;
  return c;
}
// clamp(floor(m / 1023), 0, 255): clamp m to [0, 255*1023 + 1022] first, then floor(m / 1023) == umulhi(m, ceil(2^32/1023))
// (exact while m * 1019 < 2^32, i.e. m < 4.2e6)
__device__ __forceinline__ uint32_t quant_int(int32_t m) {
  int32_t c;
  asm("min.s32.relu %0, %1, %2;" : "=r"(c) : "r"(m), "r"(261887));   // clamp to [0, 261887] in one instruction
  return __umulhi((uint32_t)c, 4198405u);
}
// A flagged chroma sample only matters when 255*Y + I sits right at a multiple of 1023: then the f64 chain decides.
__device__ __noinline__ uint32_t yuv_to_rgb_flagged(uint32_t Y, uint32_t U, uint32_t V, int32_t ir, int32_t ig, int32_t ib) {
  const int32_t y255 = (int32_t)(255u * Y);
  const int32_t m[3] = {y255 + ir, y255 + ig, y255 + ib};
  bool unc = false;
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    if (m[i] <= 0) continue;
    const uint32_t rem = (uint32_t)m[i] % 1023u;
    unc |= rem == 0u || rem == 1022u;
  }
  if (unc) return yuv_to_rgb_f64(Y, U, V);
  return quant_int(m[0]) | (quant_int(m[1]) << 8) | (quant_int(m[2]) << 16);
}
__device__ __forceinline__ uint32_t yuv_to_rgb_term(uint32_t Y, uint32_t U, uint32_t V, const ChromaTerm& c) {
  if (c.flagged) return yuv_to_rgb_flagged(Y, U, V, c.ir, c.ig, c.ib);   // rare unless the chroma is exactly neutral
  const int32_t y255 = (int32_t)(255u * Y);
  return quant_int(y255 + c.ir) | (quant_int(y255 + c.ig) << 8) | (quant_int(y255 + c.ib) << 16);
}
__device__ __forceinline__ uint32_t yuv_to_rgb_fast(uint32_t Y, int32_t ir, int32_t ig, int32_t ib) {
  const uint32_t r = quant_int((int32_t)(255u * Y) + ir), g = quant_int((int32_t)(255u * Y) + ig), b = quant_int((int32_t)(255u * Y) + ib);
  return (b * 256u + g) * 256u + r;
}
__device__ __forceinline__ uint32_t yuv_to_rgb_packed(uint32_t Y, uint32_t U, uint32_t V) {
  return yuv_to_rgb_term(Y, U, V, chroma_term(U, V));
}

// occupancy of the full-resolution pixel (x,y) straight from the low-resolution video (codec.rs:294-298)
__device__ __forceinline__ uint32_t occ_at(const UnpackArgs& a, const uint8_t* occ_f, uint32_t x, uint32_t y) {
  return occ_f[(uint64_t)div_prec(y, a.prec, a.prec_shift) * a.in.occ_pitch + div_prec(x, a.prec, a.prec_shift)];
}

// K5: boundary type of an occupied pixel (own spec): 1 = image border or an unoccupied 4-neighbour, 2 = an unoccupied
// pixel inside the 5x5 window (clipped to the image), 0 = interior.  Per-pixel form (generic slots only).
__device__ uint32_t boundary_type(const UnpackArgs& a, const uint8_t* occ_f, int32_t x, int32_t y) {
  const int32_t W = (int32_t)a.W, H = (int32_t)a.H;
  if (x == 0 || y == 0 || x == W - 1 || y == H - 1) return 1;
  if (!occ_at(a, occ_f, x - 1, y) || !occ_at(a, occ_f, x + 1, y) || !occ_at(a, occ_f, x, y - 1) ||
      !occ_at(a, occ_f, x, y + 1))
    return 1;
  const int32_t xa = max(x - 2, 0), xb = min(x + 2, W - 1), ya = max(y - 2, 0), yb = min(y + 2, H - 1);
  const uint32_t cxa = div_prec(xa, a.prec, a.prec_shift), cxb = div_prec(xb, a.prec, a.prec_shift);
  const uint32_t cya = div_prec(ya, a.prec, a.prec_shift), cyb = div_prec(yb, a.prec, a.prec_shift);
  for (uint32_t cy = cya; cy <= cyb; ++cy)
    for (uint32_t cx = cxa; cx <= cxb; ++cx)
      if (occ_f[(uint64_t)cy * a.in.occ_pitch + cx] == 0) return 2;
  return 0;
}

// ----------------------------------------------------------------------------------------------------------------
// voxel-cell tables (own spec; see DESIGN.md "Smoothing specification")
// ----------------------------------------------------------------------------------------------------------------
// x / G.g for x < 65536 by multiply-high (magic = ceil(2^32 / g); exact while x * g < 2^32)
__device__ __forceinline__ uint32_t cell_div(uint32_t x, const GridDesc& G) {
  return G.g_shift >= 0 ? (x >> G.g_shift) : __umulhi(x, G.magic);
}

__device__ __forceinline__ uint64_t hash_slot0(uint32_t key, const GridDesc& G) {
  const uint32_t cx = key & 1023u, cy = (key >> 10) & 1023u, cz = key >> 20;
  // 2x2x2 neighbouring cells share one 8-slot group: the filter's neighbourhood lookups stay within a few lines
  const uint32_t grp = (cx >> 1) | ((cy >> 1) << 9) | ((cz >> 1) << 18);
  const uint64_t h = ((uint64_t)grp * 0x9E3779B97F4A7C15ull) >> 24;
  return ((h << 3) | ((cx & 1u) | ((cy & 1u) << 1) | ((cz & 1u) << 2))) & (G.slots - 1);
}
// table slot of cell `key` (cx | cy<<10 | cz<<20) in the table of frame-in-group `fig`: the dense index, or find-or-claim
// in the key array of a hashed table.  kCellEmpty on failure (table full: cannot happen, slots >= 2 * points).
__device__ __noinline__ uint32_t cell_slot_hashed(const GridDesc& G, uint32_t fig, uint32_t key, int* err) {
  uint32_t* keys = G.keys + (uint64_t)fig * G.slots;
  uint64_t i = hash_slot0(key, G);
  for (uint64_t probe = 0; probe < G.slots; ++probe) {
    uint32_t cur = *reinterpret_cast<volatile uint32_t*>(&keys[i]);
    if (cur == kCellEmpty) cur = atomicCAS(&keys[i], kCellEmpty, key);
    if (cur == kCellEmpty || cur == key) return (uint32_t)i;
    i = (i + 1) & (G.slots - 1);
  }
  atomicExch(err, 11);
  return kCellEmpty;
}
__device__ __forceinline__ uint32_t cell_slot(const GridDesc& G, uint32_t fig, uint32_t key, int* err) {
  if (G.identity) return (key & 1023u) + G.w * (((key >> 10) & 1023u) + G.w * (key >> 20));
  return cell_slot_hashed(G, fig, key, err);          // rare (grids too large for a dense table): kept out of the hot loops
}
__device__ __noinline__ uint32_t cell_find_hashed(const GridDesc& G, uint32_t fig, uint32_t key) {
  const uint32_t* keys = G.keys + (uint64_t)fig * G.slots;
  uint64_t i = hash_slot0(key, G);
  for (uint64_t probe = 0; probe < G.slots; ++probe) {
    const uint32_t k = keys[i];
    if (k == key) return (uint32_t)i;
    if (k == kCellEmpty) return kCellEmpty;
    i = (i + 1) & (G.slots - 1);
  }
  return kCellEmpty;
}
__device__ __forceinline__ uint32_t cell_find(const GridDesc& G, uint32_t fig, uint32_t key) {
  if (G.identity) return (key & 1023u) + G.w * (((key >> 10) & 1023u) + G.w * (key >> 20));
  return cell_find_hashed(G, fig, key);
}

// ----------------------------------------------------------------------------------------------------------------
// K2: block-to-patch map.  One thread per slot (= one 16x16 block of one patch).
// ----------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ SlotRec load_slot_rec(const SlotRec* p) {
  const uint4 v = __ldg(reinterpret_cast<const uint4*>(p));
  SlotRec r;
  r.pid = v.x; r.u0b = (uint16_t)v.y; r.v0b = (uint16_t)(v.y >> 16); r.bx = (uint16_t)v.z; r.by = (uint16_t)(v.z >> 16);
  r.ax = (int8_t)v.w; r.ay = (int8_t)(v.w >> 8); r.rx = (int8_t)(v.w >> 16); r.ry = (int8_t)(v.w >> 24);
  return r;
}

__global__ void __launch_bounds__(256) block_to_patch_kernel(const UnpackArgs a, uint32_t n_slots,
                                                             uint32_t* __restrict__ b2p) {
  const uint32_t slot = blockIdx.x * blockDim.x + threadIdx.x;
  if (slot >= n_slots) return;
  const SlotRec R = load_slot_rec(a.slot_rec + slot);
  if (R.pid == kNoPatch) return;
  const uint32_t frame = a.tile_frame[slot / kWarpsPerTile];
  const uint8_t* occ_f = a.in.occ + (uint64_t)frame * a.in.occ_frame_stride;
  const uint32_t res = a.res;
  const uint32_t packed = __ldg(reinterpret_cast<const uint32_t*>(&a.patches[R.pid].orient));   // orient | aligned << 8 | ...
  bool nz = false;
  if ((packed >> 8) & 0xFFu) {
    // the res x res patch pixels are exactly the canvas block: test the low-resolution samples that cover it
    const uint32_t x0 = (uint32_t)R.bx * res, y0 = (uint32_t)R.by * res;
    const uint32_t cxa = div_prec(x0, a.prec, a.prec_shift), cxb = div_prec(x0 + res - 1, a.prec, a.prec_shift);
    const uint32_t cya = div_prec(y0, a.prec, a.prec_shift), cyb = div_prec(y0 + res - 1, a.prec, a.prec_shift);
    for (uint32_t cy = cya; cy <= cyb && !nz; ++cy) {
      const uint8_t* row = occ_f + (uint64_t)cy * a.in.occ_pitch;
      if (((cxa | (cxb + 1)) & 3u) == 0) {                           // whole aligned words (precision 4, resolution 16)
        for (uint32_t cx = cxa; cx <= cxb; cx += 4) nz |= *reinterpret_cast<const uint32_t*>(row + cx) != 0u;
      } else {
        for (uint32_t cx = cxa; cx <= cxb; ++cx) nz |= row[cx] != 0;
      }
    }
  } else {
    // reference-literal pixel mapping for the rotated / mirrored orientations (codec.rs:227-241)
    const DevPatch P = a.patches[R.pid];
    for (uint32_t i = 0; i < res * res && !nz; ++i) {
      const uint32_t v1 = i / res, u1 = i - v1 * res;
      int64_t x, y;
      patch_to_canvas(P, (int64_t)R.u0b * res + u1, (int64_t)R.v0b * res + v1, res, 1, x, y);
      nz |= occ_at(a, occ_f, (uint32_t)x, (uint32_t)y) != 0;
    }
  }
  if (nz) {
    const uint32_t local_index = __ldg(&a.patches[R.pid].local_index);
    atomicMax(&b2p[(uint64_t)frame * a.bw * a.bh + (uint64_t)R.by * a.bw + (uint64_t)R.bx], local_index + 1);
  }
}

// After K2: the slots that own their canvas block (codec.rs:379), compacted per frame in slot order.  One CTA per frame.
// The unpack kernel walks this list, so every warp of a tile has work and no plane is touched for a block that is
// skipped.
// exclusive prefix of `v` over the CTA (1024 threads) + the CTA total; s_w: 32 words of shared memory
__device__ __forceinline__ uint32_t cta_exclusive_scan(uint32_t v, uint32_t* s_w, uint32_t& total) {
  const uint32_t lane = lane_id(), warp = threadIdx.x >> 5;
  uint32_t incl = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t t = __shfl_up_sync(kFull, incl, d);
    if (lane >= (uint32_t)d) incl += t;
  }
  if (lane == 31) s_w[warp] = incl;
  __syncthreads();
  uint32_t w = lane < (blockDim.x >> 5) ? s_w[lane] : 0u, wincl = w;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t t = __shfl_up_sync(kFull, wincl, d);
    if (lane >= (uint32_t)d) wincl += t;
  }
  total = __shfl_sync(kFull, wincl, 31);
  const uint32_t wbase = __shfl_sync(kFull, wincl - w, warp);
  __syncthreads();
  return wbase + incl - v;
}

constexpr int kPerThread = 8;   // slots per thread and pass of the per-frame kernels (all loads of a pass are in flight together)

__global__ void __launch_bounds__(1024) compact_owned_kernel(const UnpackArgs a) {
  const uint32_t f = blockIdx.x;
  const uint32_t s0 = a.frame_tile_begin[f] * kWarpsPerTile, s1 = a.frame_tile_begin[f + 1] * kWarpsPerTile;
  __shared__ uint32_t s_w[32];
  uint32_t carry = 0;
  for (uint32_t b = s0; b < s1; b += 1024 * kPerThread) {
    // thread t owns the kPerThread consecutive slots from b + t * kPerThread (slot order == thread order)
    const uint32_t first = b + threadIdx.x * kPerThread;
    uint4 rec[kPerThread];
    uint32_t li[kPerThread], d1m[kPerThread][2];
#pragma unroll
    for (int i = 0; i < kPerThread; ++i) {
      rec[i] = make_uint4(kNoPatch, 0, 0, 0);
      if (first + i < s1) rec[i] = __ldg(reinterpret_cast<const uint4*>(a.slot_rec + first + i));
    }
#pragma unroll
    for (int i = 0; i < kPerThread; ++i) {
      li[i] = 0; d1m[i][0] = d1m[i][1] = 0;
      if (rec[i].x != kNoPatch) {
        const DevPatch* p = a.patches + rec[i].x;
        li[i] = __ldg(&p->local_index);
        d1m[i][0] = __ldg(&p->d1);
        d1m[i][1] = __ldg(reinterpret_cast<const uint32_t*>(&p->normal)) >> 24;     // projection mode
      }
    }
    uint32_t own = 0;
#pragma unroll
    for (int i = 0; i < kPerThread; ++i) {
      if (rec[i].x == kNoPatch) continue;
      const uint32_t bx = rec[i].z & 0xFFFFu, by = rec[i].z >> 16;
      if (a.block_to_patch[(uint64_t)f * a.bw * a.bh + (uint64_t)by * a.bw + bx] == li[i] + 1) own |= 1u << i;
    }
    uint32_t total;
    uint32_t pos = carry + cta_exclusive_scan(__popc(own), s_w, total);
#pragma unroll
    for (int i = 0; i < kPerThread; ++i) {
      if (!((own >> i) & 1u)) continue;
      uint4* dst = reinterpret_cast<uint4*>(a.work + s0 + pos);
      dst[0] = rec[i];
      dst[1] = make_uint4(f | (d1m[i][1] << 31), 0, 0, d1m[i][0]);      // frame | mode << 31, total, base, d1
      ++pos;
    }
    carry += total;
  }
  // the unused tail of the frame's region: inactive records
  for (uint32_t i = s0 + carry + threadIdx.x; i < s1; i += blockDim.x) {
    uint4* dst = reinterpret_cast<uint4*>(a.work + i);
    dst[0] = make_uint4(kNoPatch, 0, 0, 0);
    dst[1] = make_uint4(f, 0, 0, 0);
  }
  if (threadIdx.x == 0) a.owned_count[f] = carry;
}

// ----------------------------------------------------------------------------------------------------------------
// K1: occupancy upsample (codec.rs:288-300), materialised only when the caller asks for tile.occupancy_map.
// ----------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) upsample_kernel(const UnpackArgs a, uint8_t* __restrict__ occ_full) {
  const uint64_t total = (uint64_t)a.n_frames * a.W * a.H;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (uint64_t)gridDim.x * blockDim.x) {
    const uint64_t f = i / ((uint64_t)a.W * a.H);
    const uint32_t r = (uint32_t)(i - f * a.W * a.H);
    const uint32_t y = r / a.W, x = r - y * a.W;
    occ_full[i] = (uint8_t)occ_at(a, a.in.occ + f * a.in.occ_frame_stride, x, y);
  }
}

// ----------------------------------------------------------------------------------------------------------------
// K3+K4(+K5, + K6/K7 statistics): unpack.  Three launches:
//   count_kernel      per owned slot: how many points it emits (reads occupancy + the two geometry planes only)
//   slot_scan_kernel  per frame: exclusive prefix of those counts in slot order == where every run starts (codec.rs:482)
//   emit_kernel       per owned slot: reload, build positions + colours, write the run at its final place
// A warp owns a slot; warps never talk to each other, so there is no barrier, flag or look-back anywhere.
//
// A block-aligned slot (16x16 block == one canvas block, every orientation whose pixel map is the affine one) is always
// LOADED in canvas layout -- lane (r, h) = canvas row r, columns 8h..8h+7, one 16-byte vector per plane -- whatever the
// patch orientation.  The orientation only decides where a pixel lands in the per-pixel tables in shared memory, which
// are in PATCH raster order (rank = v1*16 + u1, the reference's emission order).
// ----------------------------------------------------------------------------------------------------------------

// normal coordinates (n0 | n1 << 16) of one pixel from its two geometry samples (codec.rs:534-558)
__device__ __forceinline__ uint32_t normals_of(const DevPatch& P, uint32_t s0, uint32_t s1, bool absolute_d1) {
  const uint32_t d0 = s0 >> 2, d1 = s1 >> 2;                                     // depth = sample / 4
  const uint32_t n0 = normal_coord(P, d0);
  const uint32_t n1 = absolute_d1 ? normal_coord(P, d1) : ((P.mode == 0 ? n0 + d1 : n0 - d1) & 0xFFFFu);
  return n0 | (n1 << 16);
}

__device__ __forceinline__ uint32_t cell_key_of(const GridDesc& G, uint32_t x, uint32_t y, uint32_t z) {
  if (!(x < G.th && y < G.th && z < G.th)) return kCellEmpty;
  return cell_div(x, G) | (cell_div(y, G) << 10) | (cell_div(z, G) << 20);
}

__device__ __forceinline__ WorkRec load_work(const WorkRec* p, uint32_t* mode = nullptr) {
  const uint4 v = *reinterpret_cast<const uint4*>(p), w = *(reinterpret_cast<const uint4*>(p) + 1);
  WorkRec r;
  r.pid = v.x; r.u0b = (uint16_t)v.y; r.v0b = (uint16_t)(v.y >> 16); r.bx = (uint16_t)v.z; r.by = (uint16_t)(v.z >> 16);
  r.ax = (int8_t)v.w; r.ay = (int8_t)(v.w >> 8); r.rx = (int8_t)(v.w >> 16); r.ry = (int8_t)(v.w >> 24);
  r.frame = w.x & 0x7FFFFFFFu; r.total = w.y; r.base = w.z; r.d1 = w.w;
  if (mode) *mode = w.x >> 31;                                     // projection mode travels in the top bit of `frame`
  return r;
}

// Is the block-aligned layout usable for this slot?  (16x16 blocks, power-of-two precision, affine steps present: the
// host zeroes the steps of reference-literal rotated patches, which take the generic per-pixel path.)
__device__ __forceinline__ bool slot_is_fast(const UnpackArgs& a, const WorkRec& R) {
  return a.res == 16 && a.prec_shift >= 0 && (R.ax != 0 || R.ay != 0);
}

// the fields of a DevPatch that the block-aligned path needs (two 16-byte loads, registers only)
__device__ __forceinline__ void load_patch_fields(const DevPatch* p, DevPatch& P) {
  const uint4 b = __ldg(reinterpret_cast<const uint4*>(p) + 1), c = __ldg(reinterpret_cast<const uint4*>(p) + 2);
  P.u1 = b.x; P.v1 = b.y; P.d1 = b.z; P.lod_x = (uint16_t)b.w; P.lod_y = (uint16_t)(b.w >> 16);
  P.normal = (uint8_t)c.x; P.tangent = (uint8_t)(c.x >> 8); P.bitangent = (uint8_t)(c.x >> 16); P.mode = (uint8_t)(c.x >> 24);
  P.sel = c.z; P.local_index = c.w;
}

// Canvas-layout view of a block: lane (r = lane >> 1, h = lane & 1) holds canvas row r, columns 8h .. 8h+7.
struct CanvasBlock {
  uint32_t n0p[4], n1p[4];   // normal coordinates of map 0 / map 1, two pixels per word (pixel 2q in the low half)
  uint32_t m1, m2;           // bit j set = pixel j of this lane emits >= 1 / 2 points
};

// occupancy of the lane's 8 pixels straight from the low-resolution video: bit j set = pixel j is occupied
__device__ __forceinline__ uint32_t occupancy_mask(const UnpackArgs& a, const WorkRec& R, uint32_t lane) {
  const uint32_t h = lane & 1u, r = lane >> 1;
  const uint32_t x0 = (uint32_t)R.bx * 16u + 8u * h, y = (uint32_t)R.by * 16u + r;
  // occupancy of the 8 pixels (codec.rs:393-396: any non-zero sample counts).  Pixels j*p .. j*p+p-1 share a sample.
  uint32_t m1 = 0;
  {
    const uint8_t* occ_f = a.in.occ + (uint64_t)R.frame * a.in.occ_frame_stride;
    const int32_t lp = a.prec_shift;
    const uint8_t* row = occ_f + (uint64_t)(y >> lp) * a.in.occ_pitch;
    if (lp == 2) {
      const uint32_t o = *reinterpret_cast<const uint16_t*>(row + (x0 >> 2));     // two samples, 2-byte aligned (x0 % 8 == 0)
      m1 = ((o & 0xFFu) ? 0x0Fu : 0u) | ((o >> 8) ? 0xF0u : 0u);
    } else {
      const int32_t nb = lp >= 3 ? 1 : (8 >> lp);
      const uint32_t ones = lp >= 3 ? 0xFFu : ((1u << (1 << lp)) - 1u);
      for (int32_t k = 0; k < nb; ++k) {
        const int32_t j = k << lp;
        if (row[(x0 + j) >> lp] != 0) m1 |= ones << j;
      }
    }
  }
  return m1;
}

// the lane's 8 pixels: geometry samples of both maps + occupancy mask -> normals and the two emission masks
__device__ __forceinline__ void geometry_digest(const UnpackArgs& a, const DevPatch& P, const uint4& g0, const uint4& g1, uint32_t m1,
                                                CanvasBlock& L) {
  uint32_t m2 = 0;
  if (P.d1 <= 0xFFFFu) {
    // codec.rs:534-558 + decoder.rs:881-888 on two pixels per instruction (16-bit lanes: VIADD.16x2 / VIMNMX.U16x2 wrap and
    // compare per half, exactly the reference's `as u16`).  depth = sample / 4 <= 16383.
    //   mode 0: n = depth + d1            mode 1: n = max(d1, depth) - depth   (never negative: a plain subtract cannot borrow)
    //   differential D1 (codec.rs:551-558): n1 = n0 +- depth1 in wrapping u16
    const uint32_t dd = P.d1 * 0x10001u;
    const bool mode0 = P.mode == 0, absd1 = a.absolute_d1 != 0;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const uint32_t e0 = (word_of(g0, q) >> 2) & 0x3FFF3FFFu, e1 = (word_of(g1, q) >> 2) & 0x3FFF3FFFu;
      const uint32_t n0 = mode0 ? __vadd2(e0, dd) : __vmaxu2(e0, dd) - e0;
      L.n0p[q] = n0;
      L.n1p[q] = absd1 ? (mode0 ? __vadd2(e1, dd) : __vmaxu2(e1, dd) - e1) : (mode0 ? __vadd2(n0, e1) : __vsub2(n0, e1));
    }
  } else {                                                          // d1 beyond 16 bits: one pixel at a time
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const uint32_t w0 = word_of(g0, q), w1 = word_of(g1, q);
      const uint32_t na = normals_of(P, w0 & 0xFFFFu, w1 & 0xFFFFu, a.absolute_d1);      // n0 | n1 << 16 of pixel 2q
      const uint32_t nb = normals_of(P, w0 >> 16, w1 >> 16, a.absolute_d1);              // pixel 2q + 1
      L.n0p[q] = __byte_perm(na, nb, 0x5410);
      L.n1p[q] = __byte_perm(na, nb, 0x7632);
    }
  }
#pragma unroll
  for (int q = 0; q < 4; ++q) {                                     // codec.rs:422-428 duplicate skip
    const uint32_t diff = L.n0p[q] ^ L.n1p[q];
    if (diff & 0xFFFFu) m2 |= 1u << (2 * q);
    if (diff >> 16) m2 |= 2u << (2 * q);
  }
  L.m1 = m1; L.m2 = m2 & m1;
}


// geometry + occupancy of the lane's 8 pixels with ordinary loads (the count pass)
__device__ __forceinline__ void load_geometry(const UnpackArgs& a, const WorkRec& R, const DevPatch& P, uint32_t lane,
                                              CanvasBlock& L) {
  const uint32_t h = lane & 1u, r = lane >> 1;
  const uint32_t x0 = (uint32_t)R.bx * 16u + 8u * h, y = (uint32_t)R.by * 16u + r;
  const uint16_t* geo0 = a.in.geo + (uint64_t)R.frame * 2 * a.in.geo_map_stride;
  const uint32_t goff = y * a.in.geo_pitch + x0;
  const uint4 g0 = ldg_nc_v4(geo0 + goff);
  const uint4 g1 = ldg_nc_v4(geo0 + a.in.geo_map_stride + goff);
  geometry_digest(a, P, g0, g1, occupancy_mask(a, R, lane), L);
}

// points of a generic slot (any resolution / precision, reference-literal rotated orientations): lane = pixel
__device__ __noinline__ uint32_t generic_slot_count(const UnpackArgs& a, uint32_t pid, uint32_t frame, uint32_t u0b,
                                                    uint32_t v0b) {
  const DevPatch P = a.patches[pid];
  const uint32_t lane = lane_id(), res = a.res;
  const uint8_t* occ_f = a.in.occ + (uint64_t)frame * a.in.occ_frame_stride;
  const uint16_t* geo0 = a.in.geo + (uint64_t)frame * 2 * a.in.geo_map_stride;
  const uint16_t* geo1 = geo0 + a.in.geo_map_stride;
  const int64_t sscale = a.spec_orientation ? res : 1;
  uint32_t total = 0;
  for (uint32_t base = 0; base < res * res; base += 32) {
    const uint32_t i = base + lane;
    uint32_t c = 0;
    if (i < res * res) {
      const uint32_t v1 = i / res, u1 = i - v1 * res;
      int64_t x, y;
      patch_to_canvas(P, (int64_t)u0b * res + u1, (int64_t)v0b * res + v1, res, sscale, x, y);
      if (occ_at(a, occ_f, (uint32_t)x, (uint32_t)y)) {
        const uint64_t off = (uint64_t)y * a.in.geo_pitch + (uint64_t)x;
        const uint32_t n = normals_of(P, geo0[off], geo1[off], a.absolute_d1);
        c = (n >> 16) != (n & 0xFFFFu) ? 2u : 1u;
      }
    }
    total += __reduce_add_sync(kFull, c);
  }
  return total;
}

// ---- smoothing: accumulate into a cell.  The sums are fire-and-forget reductions (two / three 64-bit adds).  Who touched a
// cell is settled by a CLAIM: compare-and-swap 0 -> patch + 1 on the cell's first word.  The first toucher (old value 0) sets
// the cell's bit in the frame's "touched" bitmap (what the clear pass walks); whoever finds another patch's claim marks the
// cell multi-patch (idempotent flag word in the cell + its bit in the frame's multi-patch bitmap, which the probe reads).
__device__ __forceinline__ void claim_result(const GridDesc& G, uint32_t fig, uint32_t cs, uint32_t old, uint32_t patch) {
  if (old == 0u) {
    atomicOr(G.tbits + (uint64_t)fig * G.twords + (cs >> (5u + kTouchShift)), 1u << ((cs >> kTouchShift) & 31u));
  } else if (old != patch + 1u) {
    reinterpret_cast<volatile uint32_t*>(static_cast<uint8_t*>(G.table) + ((uint64_t)fig * G.slots + cs) * 32u)[1] = 1u;
    atomicOr(G.mbits + (uint64_t)fig * G.mwords + (cs >> 5), 1u << (cs & 31u));
  }
}
__device__ __forceinline__ uint32_t claim_issue(const GridDesc& G, uint32_t fig, uint32_t cs, uint32_t patch) {
  return atomicCAS(reinterpret_cast<uint32_t*>(static_cast<uint8_t*>(G.table) + ((uint64_t)fig * G.slots + cs) * 32u), 0u, patch + 1u);
}
// claim and wait for the answer (the rare paths)
__device__ __forceinline__ void cell_claim_now(const GridDesc& G, uint32_t fig, uint32_t cs, uint32_t patch) {
  claim_result(G, fig, cs, claim_issue(G, fig, cs, patch), patch);
}
__device__ __forceinline__ void geo_cell_add(const GridDesc& G, uint32_t fig, uint32_t slot, uint32_t patch, uint32_t cnt,
                                             uint32_t sx, uint32_t sy, uint32_t sz) {
  GeoCell* c = reinterpret_cast<GeoCell*>(G.table) + (uint64_t)fig * G.slots + slot;
  cell_claim_now(G, fig, slot, patch);
  atomicAdd(&c->cnt_sx, (unsigned long long)cnt | ((unsigned long long)sx << 32));
  atomicAdd(&c->sy_sz, (unsigned long long)sy | ((unsigned long long)sz << 32));
}
__device__ __forceinline__ void col_cell_add(const GridDesc& G, uint32_t fig, uint32_t slot, uint32_t patch, uint32_t cnt,
                                             uint32_t sy, uint32_t su, uint32_t sv, unsigned long long sy2) {
  ColCell* c = reinterpret_cast<ColCell*>(G.table) + (uint64_t)fig * G.slots + slot;
  cell_claim_now(G, fig, slot, patch);
  atomicAdd(&c->cnt_sy, (unsigned long long)cnt | ((unsigned long long)sy << 24));
  atomicAdd(&c->su_sv, (unsigned long long)su | ((unsigned long long)sv << 32));
  atomicAdd(&c->sy2, sy2);
}

// Generic slot path: lane = pixel, 32 at a time in patch raster order, everything straight to global memory.  Rare.
template <bool kSmooth, bool kDebug>
__device__ __noinline__ void generic_slot_emit(const UnpackArgs& a, uint32_t pid, uint32_t frame, uint32_t fig, uint32_t u0b,
                                               uint32_t v0b, uint64_t gidx) {
  const DevPatch P = a.patches[pid];
  const uint32_t lane = lane_id(), res = a.res;
  const uint8_t* occ_f = a.in.occ + (uint64_t)frame * a.in.occ_frame_stride;
  const uint16_t* geo0 = a.in.geo + (uint64_t)frame * 2 * a.in.geo_map_stride;
  const uint16_t* geo1 = geo0 + a.in.geo_map_stride;
  const int64_t sscale = a.spec_orientation ? res : 1;
  const uint32_t srcx = axis_source(P, 0), srcy = axis_source(P, 1), srcz = axis_source(P, 2);
  uint64_t run = gidx;
  for (uint32_t base = 0; base < res * res; base += 32) {
    const uint32_t i = base + lane;
    uint32_t c = 0, n0 = 0, n1 = 0, t = 0, b = 0;
    int64_t x = 0, y = 0;
    if (i < res * res) {
      const uint32_t v1 = i / res, u1 = i - v1 * res;
      const uint32_t u = u0b * res + u1, v = v0b * res + v1;
      patch_to_canvas(P, u, v, res, sscale, x, y);
      if (occ_at(a, occ_f, (uint32_t)x, (uint32_t)y)) {
        const uint64_t off = (uint64_t)y * a.in.geo_pitch + (uint64_t)x;
        const uint32_t nn = normals_of(P, geo0[off], geo1[off], a.absolute_d1);
        n0 = nn & 0xFFFFu; n1 = nn >> 16;
        c = n1 != n0 ? 2u : 1u;
        t = (u * P.lod_x + P.u1) & 0xFFFFu;
        b = (v * P.lod_y + P.v1) & 0xFFFFu;
      }
    }
    uint32_t incl = c;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const uint32_t tt = __shfl_up_sync(kFull, incl, d);
      if (lane >= (uint32_t)d) incl += tt;
    }
    const uint32_t chunk_total = __shfl_sync(kFull, incl, 31);
    uint64_t k = run + (incl - c);
    uint32_t bt = 0;
    if (c && ((kDebug && a.out.btype) || kSmooth)) bt = boundary_type(a, occ_f, (int32_t)x, (int32_t)y);
    for (uint32_t m = 0; m < 2; ++m) {
      const bool on = m < c;
      const uint32_t n = m == 0 ? n0 : n1;
      const uint32_t X = pick(srcx, n, t, b), Yc = pick(srcy, n, t, b), Z = pick(srcz, n, t, b);
      uint32_t Y = 0, U = 0, V = 0;
      if (on) {
        if (a.out.pos) { uint16_t* d = a.out.pos + k * 3; d[0] = (uint16_t)X; d[1] = (uint16_t)Yc; d[2] = (uint16_t)Z; }
        if (a.has_attr) {
          const uint64_t fm = (uint64_t)frame * 2 + m;
          Y = a.in.attr_y[fm * a.in.attr_y_map_stride + (uint64_t)y * a.in.attr_pitch_y + (uint64_t)x];
          const uint64_t co = fm * a.in.attr_c_map_stride + (uint64_t)(y >> 1) * a.in.attr_pitch_c + (uint64_t)(x >> 1);
          U = a.in.attr_u[co]; V = a.in.attr_v[co];
          if (kDebug && a.out.yuv) { uint16_t* d = a.out.yuv + k * 3; d[0] = (uint16_t)Y; d[1] = (uint16_t)U; d[2] = (uint16_t)V; }
          if (a.out.rgb) {
            const uint32_t cc = yuv_to_rgb_packed(Y, U, V);
            uint8_t* d = a.out.rgb + k * 3; d[0] = (uint8_t)cc; d[1] = (uint8_t)(cc >> 8); d[2] = (uint8_t)(cc >> 16);
          }
        }
        if (kDebug && a.out.part) a.out.part[k] = (uint16_t)P.local_index;
        if (kDebug && a.out.pix) a.out.pix[k] = (uint32_t)x | ((uint32_t)y << 15) | (m << 30);
        if (kDebug && a.out.btype) a.out.btype[k] = (uint8_t)bt;
      }
      if (kSmooth) {
        if (a.sm.geo.on) {
          const uint32_t key = on ? cell_key_of(a.sm.geo, X, Yc, Z) : kCellEmpty;
          if (key != kCellEmpty) {
            const uint32_t cs = cell_slot(a.sm.geo, fig, key, a.err);
            if (cs != kCellEmpty) {
              const uint32_t g = a.sm.geo.g;
              geo_cell_add(a.sm.geo, fig, cs, P.local_index, 1, X - (key & 1023u) * g, Yc - ((key >> 10) & 1023u) * g,
                           Z - (key >> 20) * g);
            }
          }
        }
        if (a.sm.col.on && a.has_attr) {
          const uint32_t key = (on && bt == 2) ? cell_key_of(a.sm.col, X, Yc, Z) : kCellEmpty;
          if (key != kCellEmpty) {
            const uint32_t cs = cell_slot(a.sm.col, fig, key, a.err);
            if (cs != kCellEmpty) col_cell_add(a.sm.col, fig, cs, P.local_index, 1, Y, U, V, (unsigned long long)Y * Y);
          }
        }
        if (on && bt == 1) {
          const uint32_t li = atomicAdd(&a.sm.blist_count[frame], 1u);
          if (li < a.sm.blist_cap) {
            BoundaryEntry e;
            e.idx = (uint32_t)(k - (uint64_t)frame * a.out.cap);
            e.pos[0] = (uint16_t)X; e.pos[1] = (uint16_t)Yc; e.pos[2] = (uint16_t)Z;
            e.yuv[0] = (uint16_t)Y; e.yuv[1] = (uint16_t)U; e.yuv[2] = (uint16_t)V;
            a.sm.blist[(uint64_t)frame * a.sm.blist_cap + li] = e;
          } else atomicExch(a.err, 7);
        }
      }
      if (on) ++k;
    }
    run += chunk_total;
  }
}

// ---- pass 1: points per owned slot ---------------------------------------------------------------------------------------
#ifndef TMC2_COUNT_MINCTA
#define TMC2_COUNT_MINCTA 8
#endif
__device__ __forceinline__ void boundary_masks(const UnpackArgs& a, const WorkRec& R, uint32_t lane, uint32_t* s_bmp, uint32_t& bt1,
                                               uint32_t& bt2);   // below
__global__ void __launch_bounds__(kWarpsPerTile * 32, TMC2_COUNT_MINCTA) count_kernel(const __grid_constant__ UnpackArgs a, uint32_t tile_offset) {
  __shared__ uint32_t s_bmp_all[kWarpsPerTile][32];
  const uint32_t lane = lane_id();
  const uint32_t lpos = (blockIdx.x + tile_offset) * kWarpsPerTile + (threadIdx.x >> 5);
  uint32_t mode;
  const WorkRec R = load_work(a.work + lpos, &mode);
  if (R.pid == kNoPatch) return;                                   // unused tail of the frame's region (total stays 0)
  uint32_t total, n_boundary = 0, nmin = 0;
  if (slot_is_fast(a, R)) {
    DevPatch P;
    P.d1 = R.d1; P.mode = (uint8_t)mode;                 // copied into the work record: no patch load on this path
    CanvasBlock L;
    load_geometry(a, R, P, lane, L);
    total = __reduce_add_sync(kFull, __popc(L.m1) + __popc(L.m2));
    if (a.want_btype) {
      // K5 here, where registers and warps are plentiful: the emit pass only reads the two 8-bit masks of its lane back.  The
      // type-1 points of the slot are counted as well, so that the scan can hand every slot its place in the frame's boundary list.
      uint32_t bt1, bt2;
      boundary_masks(a, R, lane, s_bmp_all[threadIdx.x >> 5], bt1, bt2);
      a.slot_bt[(uint64_t)lpos * 32u + lane] = (uint16_t)(bt1 | (bt2 << 8));
      const uint32_t b1 = L.m1 & bt1;
      n_boundary = __reduce_add_sync(kFull, __popc(b1) + __popc(b1 & L.m2));
      // smallest normal coordinate among the slot's points (both maps; a skipped duplicate equals its map-0 point): origin
      // of the slot's cell table along the projection axis
      uint32_t lo = 0xFFFFFFFFu;
      const uint32_t inv = ~L.m1;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const uint32_t off = (((inv >> (2 * q)) & 1u) * 0xFFFFu) | (((inv >> (2 * q + 1)) & 1u) * 0xFFFF0000u);
        lo = __vminu2(lo, __vminu2(L.n0p[q] | off, L.n1p[q] | off));
      }
      nmin = __reduce_min_sync(kFull, min(lo & 0xFFFFu, lo >> 16));
    }
  } else {
    total = generic_slot_count(a, R.pid, R.frame, R.u0b, R.v0b);   // (generic slots append to the boundary list with atomics)
  }
  if (lane == 0) {
    a.work[lpos].total = total;
    if (a.want_btype) { a.slot_bbase[lpos] = n_boundary; a.slot_nmin[lpos] = (uint16_t)nmin; }
  }
}

// ---- pass 2: where every run starts.  One CTA per frame; the scan domain is the frame's owned-slot list ---------------------
__global__ void __launch_bounds__(1024) slot_scan_kernel(const UnpackArgs a) {
  const uint32_t f = blockIdx.x;
  const uint32_t s0 = a.frame_tile_begin[f] * kWarpsPerTile, n = a.owned_count[f];
  __shared__ uint32_t s_w[32];
  uint32_t carry = 0;
  for (uint32_t b = 0; b < n; b += 1024 * kPerThread) {
    const uint32_t first = b + threadIdx.x * kPerThread;
    uint32_t v[kPerThread], sum = 0;
#pragma unroll
    for (int i = 0; i < kPerThread; ++i) {
      v[i] = first + i < n ? a.work[s0 + first + i].total : 0u;
      sum += v[i];
    }
    uint32_t total;
    uint32_t base = carry + cta_exclusive_scan(sum, s_w, total);
#pragma unroll
    for (int i = 0; i < kPerThread; ++i) {
      if (first + i < n) a.work[s0 + first + i].base = base;
      base += v[i];
    }
    carry += total;
  }
  if (threadIdx.x == 0) a.frame_count[f] = carry;                // tile.total_number_of_regular_points, codec.rs:482
  if (a.want_btype && a.sm.blist_count != nullptr) {
    // the same for the type-1 boundary points: every block-aligned slot gets a fixed range of the frame's boundary list (no
    // atomics, and the list comes out in slot order); generic slots append behind it
    __syncthreads();
    uint32_t bcarry = 0;
    for (uint32_t b = 0; b < n; b += 1024 * kPerThread) {
      const uint32_t first = b + threadIdx.x * kPerThread;
      uint32_t v[kPerThread], sum = 0;
#pragma unroll
      for (int i = 0; i < kPerThread; ++i) {
        v[i] = first + i < n ? a.slot_bbase[s0 + first + i] : 0u;
        sum += v[i];
      }
      uint32_t total;
      uint32_t base = bcarry + cta_exclusive_scan(sum, s_w, total);
#pragma unroll
      for (int i = 0; i < kPerThread; ++i) {
        if (first + i < n) a.slot_bbase[s0 + first + i] = base;
        base += v[i];
      }
      bcarry += total;
    }
    if (threadIdx.x == 0) a.sm.blist_count[f] = bcarry;
  }
}

// one row of the 20x20 occupancy bitmap (block + 2-pixel margin): bit cc = pixel (x0 + sx*cc, y0 + sy*cc) is occupied, or
// lies outside the image (the 5x5 test ignores those).  Walks the row one occupancy cell at a time.  Any precision.
__device__ __forceinline__ uint32_t bitmap_row(const UnpackArgs& a, const uint8_t* occ_f, int32_t x0, int32_t y0, int32_t sx,
                                               int32_t sy) {
  // pixel cc of the row is (x0 + sx*cc, y0 + sy*cc); exactly one of sx, sy is non-zero
  const int32_t W = (int32_t)a.W, H = (int32_t)a.H, lp = a.prec_shift;
  const bool along_x = sx != 0;
  const int32_t fixed = along_x ? y0 : x0, flim = along_x ? H : W;
  if (fixed < 0 || fixed >= flim) return 0xFFFFFu;
  const int32_t m0 = along_x ? x0 : y0, st = along_x ? sx : sy, mlim = along_x ? W : H;
  const uint8_t* rowp = along_x ? occ_f + (uint64_t)(fixed >> lp) * a.in.occ_pitch : occ_f + (fixed >> lp);
  const uint32_t cell_stride = along_x ? 1u : a.in.occ_pitch;
  const int32_t pm = (1 << lp) - 1;
  uint32_t bits = 0;
  int32_t cc = 0;
  while (cc < 20) {
    const int32_t m = m0 + st * cc;
    if (m < 0 || m >= mlim) { bits |= 1u << cc; ++cc; continue; }
    const int32_t run = min(20 - cc, st > 0 ? (pm + 1) - (m & pm) : (m & pm) + 1);     // pixels left inside this cell
    if (rowp[(uint64_t)(m >> lp) * cell_stride] != 0) bits |= ((1u << run) - 1u) << cc;
    cc += run;
  }
  // a cell run may have crossed the image edge (image size not a multiple of the precision): those pixels count as set
  return bits | (st > 0 ? (m0 + 19 >= mlim ? (0xFFFFFu << max(mlim - m0, 0)) & 0xFFFFFu : 0u)
                        : (m0 - 19 < 0 ? (0xFFFFFu << max(m0 + 1, 0)) & 0xFFFFFu : 0u));
}

// K5 for a block-aligned slot, canvas axes: boundary classes of the lane's 8 pixels (bit j of bt1 / bt2 = type 1 / type 2;
// meaningful where the pixel is occupied).  s_bmp: 32 words of warp-private shared memory.
__device__ __forceinline__ void boundary_masks(const UnpackArgs& a, const WorkRec& R, uint32_t lane, uint32_t* s_bmp,
                                               uint32_t& bt1, uint32_t& bt2) {
  const int32_t W = (int32_t)a.W, H = (int32_t)a.H;
  const uint8_t* occ_f = a.in.occ + (uint64_t)R.frame * a.in.occ_frame_stride;
  const int32_t h = (int32_t)(lane & 1u), r = (int32_t)(lane >> 1);
  const int32_t bx16 = (int32_t)R.bx * 16, by16 = (int32_t)R.by * 16;
  if (a.prec_shift == 2 && ((a.W | a.H) & 3u) == 0) {
    // precision 4: the 20x20 window is a 6x6 patch of occupancy samples (cells bx*4-1 .. bx*4+4); lane i < 30 fetches
    // cell (row i / 6, column i % 6), lanes 0..5 then fetch row 5; cells outside the image count as occupied
    const int32_t cw = W >> 2, ch = H >> 2, cxb = (int32_t)R.bx * 4 - 1, cyb = (int32_t)R.by * 4 - 1;
    auto cell = [&](int32_t row, int32_t col) -> bool {
      const int32_t cx = cxb + col, cy = cyb + row;
      if (cx < 0 || cy < 0 || cx >= cw || cy >= ch) return true;
      return occ_f[(uint64_t)cy * a.in.occ_pitch + cx] != 0;
    };
    const int32_t i = (int32_t)lane;
    const uint32_t b0 = __ballot_sync(kFull, i < 30 ? cell(i / 6, i % 6) : false);
    const uint32_t b1 = __ballot_sync(kFull, i < 6 ? cell(5, i) : false);
    // lane = bitmap row rr (pixel row rr - 2): its cell row is (rr + 2) / 4
    const uint32_t crow = (lane + 2u) >> 2;
    const uint32_t m6 = crow < 5u ? (b0 >> (6u * crow)) & 63u : (b1 & 63u);
    const uint32_t row20 = ((m6 & 1u) ? 0x3u : 0u) | ((m6 & 2u) ? 0x3Cu : 0u) | ((m6 & 4u) ? 0x3C0u : 0u) |
                           ((m6 & 8u) ? 0x3C00u : 0u) | ((m6 & 16u) ? 0x3C000u : 0u) | ((m6 & 32u) ? 0xC0000u : 0u);
    if (lane < 20) s_bmp[lane] = row20;
  } else if (lane < 20) {
    s_bmp[lane] = bitmap_row(a, occ_f, bx16 - 2, by16 + (int32_t)lane - 2, 1, 0);
  }
  __syncwarp();
  const uint32_t r0 = s_bmp[r], r1 = s_bmp[r + 1], r2 = s_bmp[r + 2], r3 = s_bmp[r + 3], r4 = s_bmp[r + 4];
  const uint32_t cross = r1 & r3 & (r2 >> 1) & (r2 << 1);    // bit c: the four neighbours of column c are occupied
  const uint32_t all5 = r0 & r1 & r2 & r3 & r4;
  const uint32_t full = all5 & (all5 >> 1) & (all5 >> 2) & (all5 << 1) & (all5 << 2);
  const uint32_t sh = 8u * (uint32_t)h + 2u;
  uint32_t border = 0;
  if (R.bx == 0 || R.by == 0 || bx16 + 16 >= W || by16 + 16 >= H) {
    const int32_t y = by16 + r;
#pragma unroll 1
    for (int j = 0; j < 8; ++j) {
      const int32_t x = bx16 + 8 * h + j;
      if (x == 0 || y == 0 || x == W - 1 || y == H - 1) border |= 1u << j;
    }
  }
  bt1 = ((~(cross >> sh)) & 0xFFu) | border;
  bt2 = (~(full >> sh)) & 0xFFu & ~bt1;
}

__device__ __forceinline__ void stg_u32(void* p, uint32_t v) { *reinterpret_cast<uint32_t*>(p) = v; }
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" :: "l"(p)); }

// ---- smoothing work of the emit loop (K6 / K7 statistics + boundary list), one call per 32-point window -----------------
// The sums are fire-and-forget reductions, so nothing in the loop waits for the memory system.  A slot claims each cell once,
// and (fast grids) only after its point loop: geometry cells sit in the slot's shared-memory table anyway, colour cells are
// remembered in a warp-local memo; all claims of the slot are then issued together and their answers looked at together.
struct SmoothState {
  uint32_t frame, fig, patch, lane, lbase, n_done;
  uint32_t* memo;                // [2][32] cells this warp has already claimed for its slot (direct-mapped, geometry / colour)
  uint8_t* scratch;              // 128 bytes (the bitmap rows of the boundary pass, free by then)
  GeoCell* geo_tab;              // this frame's tables
  ColCell* col_tab;
  uint32_t pend_cs, pend_old;    // a claim issued in the loop (memo entry taken by another cell); bit 31 of pend_cs: colour grid
  // kFast only: the slot's own geometry-cell table in shared memory, [4 bitangent][4 tangent][8 normal] cells from the slot's
  // lowest cell (kmin, in packed-key form) -- a 16x16 block with lod 1 spans at most 3 cells of edge 8 along either tangential
  // axis.  Entry = {count | sum x << 10, sum y | sum z << 12} (at most 512 points of offsets <= 7: 10 + 12 bits).
  uint32_t* tab;
  uint32_t kmin, bad, mul;       // local cell = key - kmin (valid iff no bit of `bad`); entry = (local * mul) >> 24

  __device__ __forceinline__ void init(const UnpackArgs& a, uint32_t frame_, uint32_t fig_, uint32_t patch_, uint32_t lane_,
                                       uint32_t* memo_, uint32_t* tab_, uint8_t* scratch_, bool with_table) {
    frame = frame_; fig = fig_; patch = patch_; lane = lane_; lbase = 0; n_done = 0;
    memo = memo_; scratch = scratch_;
    memo[lane] = kCellEmpty; memo[32 + lane] = kCellEmpty;
    tab = tab_;
    if (with_table) {
      reinterpret_cast<uint4*>(tab)[lane] = make_uint4(0, 0, 0, 0);
      reinterpret_cast<uint4*>(tab)[32 + lane] = make_uint4(0, 0, 0, 0);
    }
    kmin = 0xFF000000u; bad = 0xFFFFFFFFu; mul = 0;                  // no table until table_origin() says otherwise
    pend_cs = kCellEmpty; pend_old = 0;
    __syncwarp();
    geo_tab = reinterpret_cast<GeoCell*>(a.sm.geo.table) + (uint64_t)fig * a.sm.geo.slots;
    col_tab = reinterpret_cast<ColCell*>(a.sm.col.table) + (uint64_t)fig * a.sm.col.slots;
  }
  // true when this warp claimed `cs` before (then the claim is skipped); remembers it otherwise.  Two lanes of one window may
  // both miss on the same cell: the claim is then simply issued twice (it is idempotent).
  __device__ __forceinline__ bool claimed_before(uint32_t* m, uint32_t cs) const {
    const uint32_t e = (cs ^ (cs >> 7) ^ (cs >> 14)) & 31u;
    if (m[e] == cs) return true;
    m[e] = cs;
    return false;
  }
  // fast grids: remember `cs` for the claims after the loop.  Its memo entry may hold another cell: then this one is claimed
  // right away, but the answer is looked at only when the next such claim comes up (or after the loop).
  __device__ __forceinline__ void retire_pending(const UnpackArgs& a) {
    if (pend_cs != kCellEmpty) {
      claim_result((pend_cs >> 31) ? a.sm.col : a.sm.geo, fig, pend_cs & 0x7FFFFFFFu, pend_old, patch);
      pend_cs = kCellEmpty;
    }
  }
  __device__ __forceinline__ void claim_later(const UnpackArgs& a, uint32_t colour, uint32_t cs) {
    const uint32_t prev = atomicCAS(memo + 32u * colour + ((cs ^ (cs >> 7) ^ (cs >> 14)) & 31u), kCellEmpty, cs);
    if (prev != kCellEmpty && prev != cs) {
      retire_pending(a);
      pend_cs = cs | (colour << 31);
      pend_old = claim_issue(colour ? a.sm.col : a.sm.geo, fig, cs, patch);
    }
  }
  // dense slot of a cell from the packed key cx | cz << 8 | cy << 16 of a fast grid
  static __device__ __forceinline__ uint32_t fast_slot(const GridDesc& G, uint32_t key) {
    return (key & 0xFFu) | ((key >> 16) << G.w_shift) | (((key >> 8) & 0xFFu) << (2u * G.w_shift));
  }

  // byte of a packed cell key (cx | cz << 8 | cy << 16) that holds the cell coordinate of position axis `ax` (0 x, 1 y, 2 z)
  static __device__ __forceinline__ uint32_t key_byte(uint32_t ax) { return ax == 0u ? 0u : ax == 2u ? 1u : 2u; }
  // kFast: place the slot's table.  nmin = smallest normal coordinate of the slot's points, t0 / b0 = tangent / bitangent of
  // pixel (0, 0) of the block, t_hi / b_hi of pixel (15, 15).  Without a table (degenerate axes, 16-bit wrap) every point takes
  // the per-point path.
  __device__ __forceinline__ void table_origin(const GridDesc& G, const DevPatch& P, uint32_t nmin, uint32_t t0, uint32_t b0,
                                               uint32_t t_hi, uint32_t b_hi) {
    const uint32_t an = P.normal, at = P.tangent, ab = P.bitangent;
    const bool ok = an < 3u && at < 3u && ab < 3u && an != at && an != ab && at != ab && t_hi < 65536u && b_hi < 65536u;
    if (!ok) return;
    const uint32_t sn = 8u * key_byte(an), st = 8u * key_byte(at), sb = 8u * key_byte(ab);
    kmin = (((nmin >> G.g_shift) & 0xFFu) << sn) | (((t0 >> G.g_shift) & 0xFFu) << st) | (((b0 >> G.g_shift) & 0xFFu) << sb);
    bad = ~((7u << sn) | (3u << st) | (3u << sb));
    mul = (1u << (24u - sn)) | (8u << (24u - st)) | (32u << (24u - sb));
  }
  // kFast, after the point loop: every non-empty entry of the slot's table goes to its cell (two reductions), and all claims
  // of the slot -- table entries, memo entries of both grids, the pending one -- are issued before any answer is looked at
  __device__ __forceinline__ void finish(const UnpackArgs& a, const DevPatch& P) {
    __syncwarp();
    const GridDesc& G = a.sm.geo;
    const uint32_t sn = 8u * key_byte(P.normal), st = 8u * key_byte(P.tangent), sb = 8u * key_byte(P.bitangent);
    // the non-empty entries of the table (a handful out of 128), compacted: the bitmap rows of the boundary pass are free by now
    uint8_t* idx8 = scratch;
    uint32_t n_ne = 0;
    if (G.on) {
      const uint32_t lt = (1u << lane) - 1u;
#pragma unroll
      for (uint32_t i = 0; i < 4; ++i) {
        const uint32_t ent = 32u * i + lane;
        const bool ne = tab[2u * ent] != 0u;
        const uint32_t b = __ballot_sync(kFull, ne);
        if (ne) idx8[n_ne + __popc(b & lt)] = (uint8_t)ent;
        n_ne += __popc(b);
      }
      __syncwarp();
    }
    // claims of the cells that did not go through the table (memo entries of both grids, the pending one) are issued first,
    // their answers looked at last
    const uint32_t cs4 = G.on ? memo[lane] : kCellEmpty;
    const uint32_t old4 = cs4 != kCellEmpty ? claim_issue(G, fig, cs4, patch) : 0u;
    const uint32_t cs5 = a.sm.col.on ? memo[32u + lane] : kCellEmpty;
    const uint32_t old5 = cs5 != kCellEmpty ? claim_issue(a.sm.col, fig, cs5, patch) : 0u;
#pragma unroll 1
    for (uint32_t base = 0; base < n_ne; base += 32) {
      uint32_t cs = kCellEmpty, old = 0;
      if (base + lane < n_ne) {
        const uint32_t ent = idx8[base + lane];
        const uint2 e = reinterpret_cast<const uint2*>(tab)[ent];
        const uint32_t key = kmin + (((ent & 7u) << sn) | (((ent >> 3) & 3u) << st) | ((ent >> 5) << sb));
        cs = fast_slot(G, key);
        GeoCell* c = geo_tab + cs;
        old = atomicCAS(&c->first1, 0u, patch + 1u);
        atomicAdd(&c->cnt_sx, (unsigned long long)(e.x & 1023u) | ((unsigned long long)(e.x >> 10) << 32));
        atomicAdd(&c->sy_sz, (unsigned long long)(e.y & 4095u) | ((unsigned long long)(e.y >> 12) << 32));
      }
      if (cs != kCellEmpty) claim_result(G, fig, cs, old, patch);
    }
    retire_pending(a);
    if (cs4 != kCellEmpty) claim_result(G, fig, cs4, old4, patch);
    if (cs5 != kCellEmpty) claim_result(a.sm.col, fig, cs5, old5, patch);
  }

  // ---- fast grids (dense power-of-two grids, geometry cell edge <= 8), used by the instantiation without generic branches ----
  // K6 statistics of the lane's two points (all points count).  Into the slot's shared-memory table (flushed once per slot);
  // two points of one cell -- the usual case, they are neighbours in the run -- share one pair of atomics.  The rare point
  // outside the table goes to its global cell directly.
  __device__ __forceinline__ void geo_pair(const UnpackArgs& a, bool v0, uint32_t w00, uint32_t w10, bool v1, uint32_t w01, uint32_t w11) {
    const GridDesc& G = a.sm.geo;
    const uint32_t m2 = (G.g - 1u) * 0x10001u;
    uint32_t ent[2], va[2], vb[2];
    bool ok[2];
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const uint32_t w0 = j ? w01 : w00, w1 = j ? w11 : w10;
      const bool valid = j ? v1 : v0;
      const bool in_grid = valid && ((w0 | w1) & G.oob_mask) == 0u;
      const uint32_t key = ((w0 >> G.g_shift) & G.cmask) | ((w1 >> G.g_shift) << 8);          // cx | cz << 8 | cy << 16
      const uint32_t rel = w0 & m2, relz = w1 & m2;                                           // w1's upper half is zero
      const uint32_t d = key - kmin;
      ok[j] = in_grid && (d & bad) == 0u;
      ent[j] = (d * mul) >> 24;
      va[j] = 1u | ((rel & 0xFFFFu) << 10);
      vb[j] = (rel >> 16) | (relz << 12);
      if (in_grid && !ok[j]) {
        const uint32_t cs = fast_slot(G, key);
        GeoCell* c = geo_tab + cs;
        claim_later(a, 0u, cs);
        atomicAdd(&c->cnt_sx, 1ull | ((unsigned long long)(rel & 0xFFFFu) << 32));
        atomicAdd(&c->sy_sz, (unsigned long long)(rel >> 16) | ((unsigned long long)relz << 32));
      }
    }
    const bool same = ok[0] && ok[1] && ent[0] == ent[1];
    if (ok[0]) {
      uint32_t* e = tab + 2u * ent[0];
      atomicAdd(e, same ? va[0] + va[1] : va[0]);
      atomicAdd(e + 1, same ? vb[0] + vb[1] : vb[0]);
    }
    if (ok[1] && !same) {
      uint32_t* e = tab + 2u * ent[1];
      atomicAdd(e, va[1]);
      atomicAdd(e + 1, vb[1]);
    }
  }
  // K7 statistics of one type-2 (second ring) point: three fire-and-forget reductions into its colour cell
  __device__ __forceinline__ void colour_point(const UnpackArgs& a, uint32_t w0, uint32_t w1, uint32_t Y, uint32_t uv) {
    const GridDesc& G = a.sm.col;
    if (((w0 | w1) & G.oob_mask) != 0u) return;
    const uint32_t cs = ((w0 & 0xFFFFu) >> G.g_shift) | (((w0 >> 16) >> G.g_shift) << G.w_shift) | ((w1 >> G.g_shift) << (2u * G.w_shift));
    ColCell* c = col_tab + cs;
    claim_later(a, 1u, cs);
    atomicAdd(&c->cnt_sy, 1ull | ((unsigned long long)Y << 24));
    atomicAdd(&c->su_sv, (unsigned long long)(uv & 0xFFFFu) | ((unsigned long long)(uv >> 16) << 32));
    atomicAdd(&c->sy2, (unsigned long long)Y * Y);
  }

  // ---- generic grids (non-power-of-two edges, hashed tables, wide geometry grids) and the debug instantiation: everything
  // per point inside the emit loop
  __device__ __forceinline__ void point(const UnpackArgs& a, bool valid, uint32_t g, uint32_t w0, uint32_t w1, uint32_t Y,
                                        uint32_t uv, uint32_t bt, bool has_attr) {
    constexpr bool kFast = false;
    const uint32_t X = w0 & 0xFFFFu, Yc = w0 >> 16, Z = w1 & 0xFFFFu;
    // K6 statistics: geometry cells over ALL points
    if (a.sm.geo.on) {
      // generic grids: segmented scan over runs of equal cell, see below
      const GridDesc& G = a.sm.geo;
      const bool fast8 = G.fast == 1u && G.g <= 8u;                     // packed single-word sums need 32 * (g - 1) < 256
      uint32_t key = kCellEmpty, rx_ = 0, ry_ = 0, rz_ = 0, vfast = 0;
      if (fast8) {
        // cell coordinates straight from the packed position words (w1's upper half is zero)
        if (valid && ((w0 | w1) & G.oob_mask) == 0u) {
          const uint32_t m2 = (G.g - 1u) * 0x10001u;
          key = ((w0 >> G.g_shift) & G.cmask) | ((w1 >> G.g_shift) << 8);          // cx | cz << 8 | cy << 16
          vfast = __byte_perm(w0 & m2, (w1 & m2) | 0x100u, 0x4205);                // 1 | rel x << 8 | rel y << 16 | rel z << 24
        }
      } else if (valid && X < G.th && Yc < G.th && Z < G.th) {
        if (G.g_shift >= 0) {
          const uint32_t m = G.g - 1u;
          key = (X >> G.g_shift) | ((Yc >> G.g_shift) << 10) | ((Z >> G.g_shift) << 20);
          rx_ = X & m; ry_ = Yc & m; rz_ = Z & m;
        } else {
          const uint32_t cx = __umulhi(X, G.magic), cy = __umulhi(Yc, G.magic), cz = __umulhi(Z, G.magic);
          key = cx | (cy << 10) | (cz << 20);
          rx_ = X - cx * G.g; ry_ = Yc - cy * G.g; rz_ = Z - cz * G.g;
        }
      }
      // Points are in patch raster order, so the lanes of a cell are (mostly) a run of consecutive lanes: segmented inclusive
      // scan over runs of equal key, the last lane of a run issues the reductions (a cell split into several runs just
      // gets several reductions).
      const uint32_t kprev = __shfl_up_sync(kFull, key, 1);
      const uint32_t heads = __ballot_sync(kFull, lane == 0 || kprev != key);
      const uint32_t dist = lane - (31u - (uint32_t)__clz(heads & (0xFFFFFFFFu >> (31u - lane))));   // lanes since the run began
      uint32_t cnt, sx, sy, sz;
      if (G.g <= 8u) {             // one packed word: count | three sums of at most 32 * 7 (8 bits each)
        uint32_t v = fast8 ? vfast : (key != kCellEmpty ? (1u | (rx_ << 8) | (ry_ << 16) | (rz_ << 24)) : 0u);
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
          const uint32_t t = __shfl_up_sync(kFull, v, d);
          if (dist >= (uint32_t)d) v += t;
        }
        cnt = v & 0xFFu; sx = (v >> 8) & 0xFFu; sy = (v >> 16) & 0xFFu; sz = v >> 24;
      } else {                              // sums of at most 32 * 255
        uint32_t v0 = key != kCellEmpty ? (1u | (rx_ << 16)) : 0u, v1 = ry_ | (rz_ << 16);
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
          const uint32_t t0 = __shfl_up_sync(kFull, v0, d), t1 = __shfl_up_sync(kFull, v1, d);
          if (dist >= (uint32_t)d) { v0 += t0; v1 += t1; }
        }
        cnt = v0 & 0xFFFFu; sx = v0 >> 16; sy = v1 & 0xFFFFu; sz = v1 >> 16;
      }
      const bool tail = key != kCellEmpty && (lane == 31u || ((heads >> 1) >> lane) & 1u);
      if (tail) {
        const uint32_t cs = fast8 ? fast_slot(G, key) : cell_slot(G, fig, key, a.err);
        if (cs != kCellEmpty) {
          GeoCell* c = geo_tab + cs;
          if (!claimed_before(memo, cs)) cell_claim_now(G, fig, cs, patch);
          atomicAdd(&c->cnt_sx, (unsigned long long)cnt | ((unsigned long long)sx << 32));
          atomicAdd(&c->sy_sz, (unsigned long long)sy | ((unsigned long long)sz << 32));
        }
      }
    }
    // K7 statistics: colour cells over the type-2 (second ring) points
    if (a.sm.col.on && has_attr) {
      const GridDesc& G = a.sm.col;
      if (bt == 2u) {
        uint32_t cs = kCellEmpty;
        if (kFast || G.fast) {
          // dense slot cx + w * (cy + w * cz) straight from the packed position words (any power-of-two width)
          if (((w0 | w1) & G.oob_mask) == 0u)
            cs = ((w0 & 0xFFFFu) >> G.g_shift) | (((w0 >> 16) >> G.g_shift) << G.w_shift) | ((w1 >> G.g_shift) << (2u * G.w_shift));
        } else {
          const uint32_t key = cell_key_of(G, X, Yc, Z);
          if (key != kCellEmpty) cs = cell_slot(G, fig, key, a.err);
        }
        if (cs != kCellEmpty) {
          ColCell* c = col_tab + cs;
          if (kFast) claim_later(a, 1u, cs);
          else if (!claimed_before(memo + 32, cs)) cell_claim_now(G, fig, cs, patch);
          atomicAdd(&c->cnt_sy, 1ull | ((unsigned long long)Y << 24));
          atomicAdd(&c->su_sv, (unsigned long long)(uv & 0xFFFFu) | ((unsigned long long)(uv >> 16) << 32));
          atomicAdd(&c->sy2, (unsigned long long)Y * Y);
        }
      }
    }
    // compact list of the type-1 boundary points (order inside the list is irrelevant)
    const uint32_t bm = __ballot_sync(kFull, bt == 1u);
    if (bt == 1u) {
      uint4 ent;
      ent.x = g;
      ent.y = w0;                                  // pos[0] | pos[1] << 16
      ent.z = (w1 & 0xFFFFu) | (Y << 16);          // pos[2] | Y << 16
      ent.w = uv;                                  // U | V << 16
      reinterpret_cast<uint4*>(a.sm.blist + (uint64_t)frame * a.sm.blist_cap)[lbase + n_done + __popc(bm & ((1u << lane) - 1u))] = ent;
    }
    n_done += __popc(bm);
  }

};

// ---- pass 3: emit ------------------------------------------------------------------------------------------------------------
// PERSISTENT: a warp walks a strided sequence of the frame group's slots.  Per slot: (1) the plane tiles of the block -- fetched
// by the TMA unit into the warp's RAW area while the warp was still busy with its previous slot -- are read in canvas layout,
// (2) spilled into per-pixel tables in shared memory in patch raster order together with the list "output point k <- (pixel
// rank, map)"; as soon as the RAW area has been read, the tiles of the warp's NEXT slot are requested (work record and patch
// fields by cp.async, planes by cp.async.bulk.tensor on the warp's mbarrier), so that no global load is ever waited for;
// (3) POINT-parallel loop, two points per lane, over groups of 64 points aligned to multiples of four in the frame's
// numbering: position, colour, straight to global memory as aligned 32-bit words (two positions = three words, four
// colours = three words); only the ragged ends of a run use 16-bit / 8-bit stores; (4) smoothing: cell statistics and
// the boundary list.
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(void* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(void* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(void* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" :: "r"(smem_u32(bar)), "r"(parity) : "memory");
}
// one box of a tiled tensor map -> shared memory, completion counted in bytes on `bar`
__device__ __forceinline__ void tma_load_4d(void* dst, const void* tmap, void* bar, int32_t c0, int32_t c1, int32_t c2, int32_t c3) {
  asm volatile("cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
               :: "r"(smem_u32(dst)), "l"(tmap), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* dst, const void* tmap, void* bar, int32_t c0, int32_t c1, int32_t c2) {
  asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
               :: "r"(smem_u32(dst)), "l"(tmap), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
// Can the occupancy samples of a block (and the ring around it that the boundary classes look at) come from the 16 x 8 box
// of the occupancy tensor map?  (precision 4 and a frame that is whole samples wide and high; anything else reads the
// occupancy video with ordinary loads)
__device__ __forceinline__ bool occ_by_tma(const UnpackArgs& a) { return a.prec_shift == 2 && ((a.W | a.H) & 3u) == 0u; }

// first sample column of the occupancy box of block column bx (a multiple of 16 samples: the TMA unit wants the first byte
// of a box row 16-byte aligned)
__device__ __forceinline__ int32_t occ_box_x(uint32_t bx) { return ((int32_t)bx * 4 - 1) & ~15; }

#ifndef TMC2_EMIT_CTAS
#define TMC2_EMIT_CTAS 8
#endif
#ifndef TMC2_EMIT_CTAS_SMOOTH
#define TMC2_EMIT_CTAS_SMOOTH 7
#endif

// One block-aligned slot.  `release_raw()` is called exactly when the RAW area has been read for the last time.
// One block-aligned slot whose tiles have landed in the RAW area.
template <bool kSmooth, bool kDebug, bool kFast, bool kAttr>
__device__ __forceinline__ void emit_fast_slot(const UnpackArgs& a, const WorkRec& R, const DevPatch& P, uint8_t* wsm, uint32_t lane,
                                               uint32_t bt_word, uint32_t blist_base, uint32_t nmin) {
  const uint32_t total = R.total, run_base = R.base, frame = R.frame;
  const uint32_t fig = kSmooth ? frame - a.sm.group_first_frame : 0u;   // frame inside the smoothing group
  constexpr EmitLayout LY = emit_layout(kSmooth, kDebug, kFast);
  constexpr bool kWide = kSmooth || kDebug;              // (plain layout: list and counts live in the dead RAW area)
  uint32_t* s_pt = reinterpret_cast<uint32_t*>(wsm + LY.pt);
  uint4* s_term = reinterpret_cast<uint4*>(wsm + LY.term);
  uint16_t* s_src = reinterpret_cast<uint16_t*>(wsm + LY.src);
  uint8_t* s_cnt = wsm + LY.cnt;
  uint32_t* s_bmp = reinterpret_cast<uint32_t*>(wsm + LY.bmp);

  constexpr bool has_attr = kAttr;
  const bool want_bt = kSmooth || (kDebug && a.out.btype != nullptr);
  const uint32_t h = lane & 1u, r = lane >> 1;
  const int32_t ax = R.ax, ay = R.ay, rx = R.rx, ry = R.ry;
  uint32_t n_boundary = 0, any_flag = 0;

  {
    // ---- (1): canvas layout: lane (r, h) = canvas row r, columns 8h .. 8h+7 -------------------------------------------
    const uint4 g0 = *reinterpret_cast<const uint4*>(wsm + kOffRawGeo + 32u * r + 16u * h);
    const uint4 g1 = *reinterpret_cast<const uint4*>(wsm + kOffRawGeo + 512u + 32u * r + 16u * h);
    uint32_t m1 = 0;
    if (occ_by_tma(a)) {
      // occupancy of the 8 pixels (codec.rs:393-396: any non-zero sample counts): two samples of the box row (r >> 2) + 2
      const uint32_t o = *reinterpret_cast<const uint16_t*>(wsm + kOffRawOcc + ((r >> 2) + 2u) * 32u +
                                                            (uint32_t)((int32_t)R.bx * 4 - occ_box_x(R.bx)) + 2u * h);
      m1 = ((o & 0xFFu) ? 0x0Fu : 0u) | ((o >> 8) ? 0xF0u : 0u);
    } else {
      m1 = occupancy_mask(a, R, lane);
    }
    CanvasBlock L;
    geometry_digest(a, P, g0, g1, m1, L);
    // K5: the boundary classes of the lane's 8 pixels were worked out by the count pass (slot_bt)
    const uint32_t bt1 = want_bt ? (bt_word & 0xFFu) : 0u, bt2 = want_bt ? (bt_word >> 8) : 0u;
    if (kSmooth) {
      if (!(kFast)) {                       // generic grids append inside the point loop and check the list capacity up front
        const uint32_t b1 = L.m1 & bt1;
        n_boundary = __reduce_add_sync(kFull, __popc(b1) + __popc(b1 & L.m2));
      }
    }

    // ---- (2): tables in patch raster order -----------------------------------------------------------------------------
    // canvas-local (lx, ly) = (8h + j, r) -> patch-local (u1, v1) through the inverse of the affine map (decoder.rs:853-867)
    uint32_t rank0; int32_t dr;
    if (ax != 0) {                          // u runs along canvas x, v along canvas y
      const uint32_t u1 = ax > 0 ? 8u * h : 15u - 8u * h, v1 = ry > 0 ? r : 15u - r;
      rank0 = v1 * 16u + u1; dr = ax;
    } else {                                // transposed: u runs along canvas y, v along canvas x
      const uint32_t u1 = ay > 0 ? r : 15u - r, v1 = rx > 0 ? 8u * h : 15u - 8u * h;
      rank0 = v1 * 16u + u1; dr = 16 * rx;
    }
    // per-pixel byte = points of the pixel (0..2) | boundary class << 2, for the lane's 8 pixels at once: spread4(m) puts bit i
    // of a 4-bit mask into byte i ((m * 0x00204081) & 0x01010101: the four shifted copies do not overlap)
    uint32_t cb_lo, cb_hi;
    {
      auto spread4 = [](uint32_t m) -> uint32_t { return (m * 0x00204081u) & 0x01010101u; };
      cb_lo = spread4(L.m1 & 15u) + spread4(L.m2 & 15u);
      cb_hi = spread4(L.m1 >> 4) + spread4(L.m2 >> 4);
      if (want_bt) {
        cb_lo += 4u * spread4(bt1 & 15u) + 8u * spread4(bt2 & 15u);
        cb_hi += 4u * spread4((bt1 >> 4) & 15u) + 8u * spread4((bt2 >> 4) & 15u);
      }
    }
    // entry of (pixel, map) = n | Y << 16; a table row (16 pixels) is padded by one entry pair so that neither the row-wise
    // nor the column-wise (transposed patches) stores run into shared-memory bank conflicts
    {
      uint4 ya = {0, 0, 0, 0}, yb = {0, 0, 0, 0};
      if (has_attr) {                                                                // decoder.rs:976-977
        ya = *reinterpret_cast<const uint4*>(wsm + kOffRawY + 32u * r + 16u * h);
        yb = *reinterpret_cast<const uint4*>(wsm + kOffRawY + 512u + 32u * r + 16u * h);
      }
      if (!kWide) __syncwarp();        // plain layout: the per-pixel counts go where the geometry / luma tiles were
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const uint32_t rank = rank0 + (uint32_t)(j * dr);
        const uint32_t sel = (j & 1) ? 0x7632u : 0x5410u;
        *reinterpret_cast<uint2*>(s_pt + 2u * (rank + (rank >> 4))) =
            make_uint2(__byte_perm(L.n0p[j >> 1], word_of(ya, j >> 1), sel), __byte_perm(L.n1p[j >> 1], word_of(yb, j >> 1), sel));
      }
    }
    if (dr == 1) {
      *reinterpret_cast<uint2*>(s_cnt + rank0) = make_uint2(cb_lo, cb_hi);
    } else if (dr == -1) {                                          // descending ranks: rank0 - 7 .. rank0, bytes reversed
      *reinterpret_cast<uint2*>(s_cnt + rank0 - 7u) = make_uint2(__byte_perm(cb_hi, 0, 0x0123), __byte_perm(cb_lo, 0, 0x0123));
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j)
        s_cnt[rank0 + (uint32_t)(j * dr)] = (uint8_t)((j < 4 ? cb_lo : cb_hi) >> (8 * (j & 3)));
    }
    uint2 cu2 = {0, 0}, cv2 = {0, 0};
    if (has_attr) {
      // the two rows of a chroma row pair hold the same 4 samples; the even row evaluates map 0, the odd row map 1
      const uint32_t coff = ((r & 1u) ? 128u : 0u) + 16u * (r >> 1) + 8u * h;
      cu2 = *reinterpret_cast<const uint2*>(wsm + kOffRawU + coff);
      cv2 = *reinterpret_cast<const uint2*>(wsm + kOffRawV + coff);
    }
    __syncwarp();                                                   // the RAW area has been read for the last time: the smoothing state may overwrite it
    if (has_attr) {
      // chroma terms, once per (chroma sample, map).  Entry = {ir, ig, ib << 1 | flagged, U | V << 16}, indexed by the
      // patch-local chroma position (cv * 8 + cu) * 2 + map.
      const bool odd = (r & 1u) != 0;
      const uint32_t ccy = r >> 1;
      auto term_of = [&](int cc) {
        const uint32_t sel = (cc & 1) ? 0x7632u : 0x5410u;
        const uint32_t uv = __byte_perm(word_of(cu2, cc >> 1), word_of(cv2, cc >> 1), sel);
        const uint32_t ccx = 4u * h + (uint32_t)cc;
        uint32_t cu, cv;
        if (ax != 0) { cu = ax > 0 ? ccx : 7u - ccx; cv = ry > 0 ? ccy : 7u - ccy; }
        else { cu = ay > 0 ? ccy : 7u - ccy; cv = rx > 0 ? ccx : 7u - ccx; }
        // no occupied pixel under the sample (the other row of the pair lies in the same occupancy cell unless the
        // precision is 1): nobody will read the term
        if (a.prec_shift >= 1 && !((L.m1 >> (2 * cc)) & 3u)) return;
        ChromaTerm t = chroma_term_fast(uv & 0xFFFFu, uv >> 16);
        if (t.flagged) t = chroma_term(uv & 0xFFFFu, uv >> 16);   // rare (or not 10-bit content): the exact 32.32 evaluation
        any_flag |= t.flagged;
        s_term[((cv * 8u + cu) << 1) | (odd ? 1u : 0u)] = make_uint4((uint32_t)t.ir, (uint32_t)t.ig, ((uint32_t)t.ib << 1) | t.flagged, uv);
      };
      // the smoothing instantiation is large enough for instruction fetch to show up among its stalls (`no_instruction`): there the
      // loop stays rolled (measured: 0.360 -> 0.353 ms; unrolled it is the faster form for the plain kernel, 0.170 against 0.174)
      if (kSmooth) {
#pragma unroll 1
        for (int cc = 0; cc < 4; ++cc) term_of(cc);
      } else {
#pragma unroll
        for (int cc = 0; cc < 4; ++cc) term_of(cc);
      }
    }
  }
  const bool slot_flagged = __any_sync(kFull, any_flag != 0);      // some chroma sample of the block needs the f64 check
  __syncwarp();

  // ---- (2b): patch raster order: lane l owns ranks 8l .. 8l+7; where its points go inside the run --------------------------
  // s_src entry of a point = rank << 1 | map | term << 9, term = index of its chroma term ((cv * 8 + cu) << 1 | map).  Entry i
  // of the list is point i - a4 of the run, a4 = run_base % 4: the point loop works on groups of four points that are
  // groups of four in the FRAME's numbering (12 colour bytes = three aligned words).
  // Fast smoothing grids: the slot's type-1 and type-2 boundary points also go into two compact lists (run-relative index),
  // which two short loops after the point loop work off with full warps -- the point loop itself does not look at classes.
  constexpr bool kLists = kSmooth && kFast;
  const uint32_t a4 = run_base & 3u;
  uint16_t* s_list = reinterpret_cast<uint16_t*>(wsm + LY.list);
  uint32_t n_type1 = 0, n_type2 = 0;
  {
    const uint2 cb = *reinterpret_cast<const uint2*>(s_cnt + 8u * lane);
    const uint32_t c_lo = cb.x & 0x03030303u, c_hi = cb.y & 0x03030303u;
    const uint32_t p_lo = c_lo * 0x01010101u;                       // byte i: points of pixels 0..i (inclusive), <= 8
    const uint32_t p_hi = c_hi * 0x01010101u + (p_lo >> 24) * 0x01010101u;
    uint32_t c = p_hi >> 24;                                        // points of this lane (<= 16)
    // type-1 / type-2 points of the lane: the same byte-parallel prefix over the counts masked by the class
    uint32_t c1_lo = 0, c1_hi = 0, c2_lo = 0, c2_hi = 0, q1_lo = 0, q1_hi = 0, q2_lo = 0, q2_hi = 0;
    if (kLists) {
      c1_lo = c_lo & (((cb.x >> 2) & 0x01010101u) * 3u); c1_hi = c_hi & (((cb.y >> 2) & 0x01010101u) * 3u);
      c2_lo = c_lo & (((cb.x >> 3) & 0x01010101u) * 3u); c2_hi = c_hi & (((cb.y >> 3) & 0x01010101u) * 3u);
      q1_lo = c1_lo * 0x01010101u; q1_hi = c1_hi * 0x01010101u + (q1_lo >> 24) * 0x01010101u;
      q2_lo = c2_lo * 0x01010101u; q2_hi = c2_hi * 0x01010101u + (q2_lo >> 24) * 0x01010101u;
      c |= ((q1_hi >> 24) << 10) | ((q2_hi >> 24) << 20);           // one scan for the three counts (each total <= 512)
    }
    uint32_t incl = c;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const uint32_t t = __shfl_up_sync(kFull, incl, d);
      if (lane >= (uint32_t)d) incl += t;
    }
    const uint32_t excl = incl - c;
    const uint32_t lane_excl = (excl & 1023u) + a4;
    if (kLists) {
      const uint32_t tot = __shfl_sync(kFull, incl, 31);
      n_type1 = (tot >> 10) & 1023u; n_type2 = tot >> 20;
    }
    const uint32_t x1 = (excl >> 10) & 1023u, x2 = excl >> 20;
    // chroma term of pixel j: ((v1 >> 1) * 8 + (u1 >> 1)) << 1, v1 = lane >> 1, u1 = 8 * (lane & 1) + j
    const uint32_t ebase = (16u * lane) | ((((lane >> 2) << 3) + ((lane & 1u) << 2)) << 10);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const uint32_t sh = 8 * (j & 3);
      const uint32_t cj = ((j < 4 ? c_lo : c_hi) >> sh) & 3u;
      const uint32_t ij = ((j < 4 ? p_lo : p_hi) >> sh) & 0xFFu;
      const uint32_t k = lane_excl + ij - cj;
      const uint32_t e = ebase + (uint32_t)((j << 1) | ((j >> 1) << 10));
      if (cj >= 1u) s_src[k] = (uint16_t)e;
      if (cj == 2u) s_src[k + 1] = (uint16_t)(e | 0x201u);           // map 1: bit 0, and bit 0 of the term index (bit 9)
      if (kLists) {
        const uint32_t cls = ((j < 4 ? cb.x : cb.y) >> (sh + 2)) & 3u;
        if (cj >= 1u && cls != 0u) {
          const uint32_t kr = k - a4;                               // run-relative index of the pixel's first point
          if (cls == 1u) {
            const uint32_t pos = x1 + (((j < 4 ? q1_lo : q1_hi) >> sh) & 0xFFu) - cj;
            s_list[pos] = (uint16_t)kr;
            if (cj == 2u) s_list[pos + 1] = (uint16_t)(kr + 1u);
          } else {
            const uint32_t pos = kListEntries - 1u - (x2 + (((j < 4 ? q2_lo : q2_hi) >> sh) & 0xFFu) - cj);
            s_list[pos] = (uint16_t)kr;
            if (cj == 2u) s_list[pos - 1u] = (uint16_t)(kr + 1u);
          }
        }
      }
    }
  }
  __syncwarp();

  // ---- (3): point-parallel, two points per lane ---------------------------------------------------------------------------
  // generate_point (decoder.rs:871-878) stores normal, tangent, bitangent in that order; the selectors (host-made, per patch)
  // reproduce "later stores overwrite earlier ones" and leave unset coordinates at 0
  const uint32_t selA = P.sel & 0xFFFFu, selB = P.sel >> 16;
  const uint32_t T00 = (uint32_t)R.u0b * 16u * P.lod_x + P.u1, B00 = (uint32_t)R.v0b * 16u * P.lod_y + P.v1;   // decoder.rs:875-876
  const uint32_t lodx = P.lod_x, lody = P.lod_y, patch = P.local_index;
  const uint64_t gframe = (uint64_t)frame * a.out.cap;
  const bool odd_lane = (lane & 1u) != 0;

  SmoothState S;
  if (kSmooth) {
    S.init(a, frame, fig, patch, lane, reinterpret_cast<uint32_t*>(wsm + LY.memo), reinterpret_cast<uint32_t*>(wsm + LY.tab),
           reinterpret_cast<uint8_t*>(s_bmp), kFast);
    // the slot's range of the frame's boundary list was fixed by the scan pass
    if (kFast) n_boundary = n_type1;
    if ((uint64_t)blist_base + n_boundary > a.sm.blist_cap) {
      if (lane == 0) atomicExch(a.err, 7);
      return;
    }
    S.lbase = blist_base;
    if (kFast && a.sm.geo.on) S.table_origin(a.sm.geo, P, nmin, T00, B00, T00 + 15u * lodx, B00 + 15u * lody);
  }

  // position words and colour of the point behind list entry `e`
  auto make_point = [&](uint32_t e, uint32_t& w0, uint32_t& w1, uint32_t& Y, uint32_t& c, uint32_t& tz) {
    const uint32_t er = e & 0x1FFu;                                  // rank << 1 | map
    const uint32_t pt = s_pt[er + ((er >> 5) << 1)];                 // n | Y << 16 (rows are padded by one pixel)
    const uint32_t u1 = (er >> 1) & 15u, v1 = er >> 5;
    const uint32_t t = T00 + u1 * lodx, b = (B00 + v1 * lody) & 0xFFFFu;
    const uint32_t A = __byte_perm(pt, t, 0x5410);                   // n | t << 16
    w0 = __byte_perm(A, b, selA); w1 = __byte_perm(A, b, selB);      // x | y << 16 ; z
    Y = pt >> 16;                                                    // codec.rs:637-640
    c = 0; tz = 0;
    if (has_attr) {
      const uint4 te = s_term[e >> 9];
      tz = te.z;
      c = yuv_to_rgb_fast(Y, (int32_t)te.x, (int32_t)te.y, (int32_t)te.z >> 1);
      if (slot_flagged && (te.z & 1u))                               // rare: neutral / borderline chroma
        c = yuv_to_rgb_flagged(Y, te.w & 0xFFFFu, te.w >> 16, (int32_t)te.x, (int32_t)te.y, (int32_t)te.z >> 1);
    }
  };

  const uint32_t n_idx = total + a4;                                 // list entries [a4, n_idx) are this slot's points
  const uint32_t* s_src32 = reinterpret_cast<const uint32_t*>(s_src);
  const uint64_t gq0 = gframe + (run_base - a4);                     // frame-global point index of list entry 0 (multiple of 4)
  uint16_t* ppos = a.out.pos + (gq0 + 2u * lane) * 3;                // this lane's two points: three aligned words
  uint8_t* prgb = has_attr ? a.out.rgb + (gq0 + 2u * (lane & ~1u)) * 3 : nullptr;   // the lane pair's four colours: three aligned words
#pragma unroll 1
  for (uint32_t i0 = 0; i0 < n_idx; i0 += 64, ppos += 192, prgb += 192) {
    const uint32_t idx = i0 + 2u * lane;
    const bool v0 = idx >= a4 && idx < n_idx, v1 = idx + 1u >= a4 && idx + 1u < n_idx;
    const uint32_t ee = s_src32[idx >> 1];
    const uint32_t e0 = v0 ? (ee & 0xFFFFu) : 0u, e1 = v1 ? (ee >> 16) : 0u;
    uint32_t w00, w10, Y0, c0, tz0, w01, w11, Y1, c1, tz1;
    make_point(e0, w00, w10, Y0, c0, tz0);
    make_point(e1, w01, w11, Y1, c1, tz1);
    // two points = three words: [x0 y0] [z0 x1] [y1 z1]
    const uint32_t Wb = __byte_perm(w10, w01, 0x5410), Wc = __byte_perm(w01, w11, 0x5432);
    // four colours (lane pair) = three words: the even lane writes the first two, the odd lane the third
    uint32_t K0 = 0, K1 = 0;
    if (has_attr) {
      const uint32_t nc0 = __shfl_down_sync(kFull, c0, 1);
      K0 = odd_lane ? __byte_perm(c0, c1, 0x6542) : __byte_perm(c0, c1, 0x4210);
      K1 = __byte_perm(c1, nc0, 0x5421);
    }
    if (i0 >= a4 && i0 + 64u <= n_idx) {                             // whole window inside the run (warp-uniform)
      stg_u32(ppos, w00); stg_u32(ppos + 2, Wb); stg_u32(ppos + 4, Wc);
      if (has_attr) {
        stg_u32(prgb + (odd_lane ? 8 : 0), K0);
        if (!odd_lane) stg_u32(prgb + 4, K1);
      }
    } else {
      // ragged end of the run: neighbouring points may belong to another slot
      if (v0) stg_u32(ppos, w00);
      if (v0 && v1) stg_u32(ppos + 2, Wb);
      else if (v0) ppos[2] = (uint16_t)w10;
      else if (v1) ppos[3] = (uint16_t)w01;
      if (v1) stg_u32(ppos + 4, Wc);
      if (has_attr) {
        const uint32_t b0 = __ballot_sync(kFull, v0), b1 = __ballot_sync(kFull, v1);
        const uint32_t le = lane & ~1u;
        if ((((b0 & b1) >> le) & 3u) == 3u) {
          stg_u32(prgb + (odd_lane ? 8 : 0), K0);
          if (!odd_lane) stg_u32(prgb + 4, K1);
        } else {
          uint8_t* q = prgb + (odd_lane ? 6 : 0);
          if (v0) { q[0] = (uint8_t)c0; q[1] = (uint8_t)(c0 >> 8); q[2] = (uint8_t)(c0 >> 16); }
          if (v1) { q[3] = (uint8_t)c1; q[4] = (uint8_t)(c1 >> 8); q[5] = (uint8_t)(c1 >> 16); }
        }
      }
    }
    if (kDebug || (kSmooth && !kFast)) {                             // streams only the stage API / tests ask for; generic grids
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const bool valid = j ? v1 : v0;
        const uint32_t e = j ? e1 : e0, w0 = j ? w01 : w00, w1 = j ? w11 : w10, Y = j ? Y1 : Y0;
        const uint32_t rank = (e >> 1) & 255u, map = e & 1u;
        const uint32_t uv = has_attr ? s_term[e >> 9].w : 0u;
        const uint32_t g = run_base - a4 + idx + (uint32_t)j;        // point index inside the frame
        uint32_t bt = 0;
        if (valid && want_bt) bt = (uint32_t)s_cnt[rank] >> 2;
        if (kDebug && valid) {
          const uint64_t gk = gframe + g;
          if (a.out.yuv && has_attr) {
            uint16_t* qy = a.out.yuv + gk * 3;
            qy[0] = (uint16_t)Y; qy[1] = (uint16_t)(uv & 0xFFFFu); qy[2] = (uint16_t)(uv >> 16);
          }
          if (a.out.part) a.out.part[gk] = (uint16_t)patch;                          // codec.rs:452
          if (a.out.pix) {                                                            // codec.rs:463-472
            const uint32_t u1 = rank & 15u, v1p = rank >> 4;
            const int32_t cx0 = (int32_t)R.bx * 16 + ((ax < 0 || rx < 0) ? 15 : 0), cy0 = (int32_t)R.by * 16 + ((ay < 0 || ry < 0) ? 15 : 0);
            a.out.pix[gk] = (uint32_t)(cx0 + ax * (int32_t)u1 + rx * (int32_t)v1p) |
                            ((uint32_t)(cy0 + ay * (int32_t)u1 + ry * (int32_t)v1p) << 15) | (map << 30);
          }
          if (a.out.btype) a.out.btype[gk] = (uint8_t)bt;
        }
        if (kSmooth && !kFast) S.point(a, valid, g, w0, w1, Y, uv, bt, has_attr);
      }
    }
    if (kSmooth && kFast) {
      if (a.sm.geo.on) S.geo_pair(a, v0, w00, w10, v1, w01, w11);
    }
  }

  if (kLists) {
    // ---- (4): the slot's boundary points, full warps ----------------------------------------------------------------------
    // type 1: entries of the frame's boundary list (what the filter passes read)
    uint4* blist = reinterpret_cast<uint4*>(a.sm.blist + (uint64_t)frame * a.sm.blist_cap) + S.lbase;
#pragma unroll 1
    for (uint32_t i = lane; i - lane < n_type1; i += 32) {
      if (i < n_type1) {
        const uint32_t kr = s_list[i];
        const uint32_t e = s_src[kr + a4];
        uint32_t w0, w1, Y, c, tz;
        make_point(e, w0, w1, Y, c, tz);
        uint4 ent;
        ent.x = run_base + kr;                       // point index inside the frame
        ent.y = w0;                                  // pos[0] | pos[1] << 16
        ent.z = (w1 & 0xFFFFu) | (Y << 16);          // pos[2] | Y << 16
        ent.w = has_attr ? s_term[e >> 9].w : 0u;    // U | V << 16
        blist[i] = ent;
      }
    }
    // type 2: K7 statistics
    if (a.sm.col.on && has_attr) {
#pragma unroll 1
      for (uint32_t i = lane; i - lane < n_type2; i += 32) {
        if (i < n_type2) {
          const uint32_t kr = s_list[kListEntries - 1u - i];
          const uint32_t e = s_src[kr + a4];
          uint32_t w0, w1, Y, c, tz;
          make_point(e, w0, w1, Y, c, tz);
          S.colour_point(a, w0, w1, Y, s_term[e >> 9].w);
        }
      }
    }
    S.finish(a, P);
  }
}

template <bool kSmooth, bool kDebug, bool kFast, bool kAttr>
__global__ void __launch_bounds__(kEmitWarps * 32, kSmooth ? TMC2_EMIT_CTAS_SMOOTH : TMC2_EMIT_CTAS)
emit_kernel(const __grid_constant__ UnpackArgs a, const __grid_constant__ TileMaps tm, uint32_t slot_begin, uint32_t slot_end) {
  extern __shared__ __align__(128) uint8_t smem[];
  const uint32_t warp = threadIdx.x >> 5, lane = lane_id();
  constexpr EmitLayout LY = emit_layout(kSmooth, kDebug, kFast);
  uint8_t* wsm = smem + (size_t)warp * LY.bytes;
  void* bar = wsm + LY.bar;
  const uint32_t lpos = slot_begin + blockIdx.x * kEmitWarps + warp;
  if (lpos >= slot_end) return;
  uint32_t mode;
  const WorkRec R = load_work(a.work + lpos, &mode);
  if (R.pid == kNoPatch || R.total == 0u) return;                // unused tail of the frame's region / nothing to emit
  if ((uint64_t)R.base + R.total > a.out.cap) {                  // cannot happen for footprints inside the canvas
    if (lane == 0) atomicExch(a.err, 7);
    return;
  }
  if (!slot_is_fast(a, R)) {
    const uint32_t fig = kSmooth ? R.frame - a.sm.group_first_frame : 0u;
    generic_slot_emit<kSmooth, kDebug>(a, R.pid, R.frame, fig, R.u0b, R.v0b, (uint64_t)R.frame * a.out.cap + R.base);
    return;
  }
  // the plane tiles of the block: five boxes (three without attributes), one mbarrier
  if (lane == 0) {
    mbar_init(bar, 1);
    const bool occ = occ_by_tma(a);
    mbar_expect_tx(bar, 1024u + (kAttr ? 1536u : 0u) + (occ ? 256u : 0u));
    const int32_t x0 = (int32_t)R.bx * 16, y0 = (int32_t)R.by * 16, f = (int32_t)R.frame;
    tma_load_4d(wsm + kOffRawGeo, tm.geo, bar, x0, y0, 0, f);
    if (kAttr) {
      tma_load_4d(wsm + kOffRawY, tm.attr_y, bar, x0, y0, 0, f);
      tma_load_4d(wsm + kOffRawU, tm.attr_u, bar, x0 >> 1, y0 >> 1, 0, f);
      tma_load_4d(wsm + kOffRawV, tm.attr_v, bar, x0 >> 1, y0 >> 1, 0, f);
    }
    if (occ) tma_load_3d(wsm + kOffRawOcc, tm.occ, bar, occ_box_x(R.bx), (int32_t)R.by * 4 - 2, f);
  }
  DevPatch P;
  load_patch_fields(a.patches + R.pid, P);                       // in flight together with the tiles
  uint32_t bt_word = 0, blist_base = 0, nmin = 0;
  if (kSmooth || kDebug) {                                       // what the count / scan passes left for this slot
    if (a.want_btype) bt_word = __ldg(a.slot_bt + (uint64_t)lpos * 32u + lane);
    if (kSmooth) { blist_base = __ldg(a.slot_bbase + lpos); nmin = __ldg(a.slot_nmin + lpos); }
  }
  __syncwarp();
  mbar_wait(bar, 0);
  emit_fast_slot<kSmooth, kDebug, kFast, kAttr>(a, R, P, wsm, lane, bt_word, blist_base, nmin);
}

// ----------------------------------------------------------------------------------------------------------------
// yuv -> rgb over a flat colour array (codec.rs:88-94)
// ----------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) yuv_to_rgb_flat_kernel(const uint16_t* __restrict__ yuv, uint8_t* __restrict__ rgb,
                                                              uint64_t n) {
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
    const uint32_t c = yuv_to_rgb_packed(yuv[3 * i], yuv[3 * i + 1], yuv[3 * i + 2]);
    rgb[3 * i] = (uint8_t)c; rgb[3 * i + 1] = (uint8_t)(c >> 8); rgb[3 * i + 2] = (uint8_t)(c >> 16);
  }
}

// ----------------------------------------------------------------------------------------------------------------
// K6 / K7 cell summaries: sums -> Q8 means (and the colour cell's luminance-variance verdict).  There is no finalize pass:
// only the boundary points that survive the probe need summaries, and they compute them from the raw accumulators.
// ----------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t mean_q8_u32(uint32_t s, uint32_t cnt) {       // (256*s + cnt/2) / cnt
  const unsigned long long num = 256ull * s + (cnt >> 1);
  return num < (1ull << 32) ? (uint32_t)num / cnt : (uint32_t)(num / cnt);
}
// SUMMARY of a cell, computed on the fly from its accumulators by whoever needs it (only the few boundary points that
// survive the probe pass do):
//   x = kCellMulti (touched by more than one patch) | kCellUsable (colour: luminance variance test passed)
//       | point count (24 bits; a frame has < 2^24 points)
//   geometry: y = mean x | mean y << 16, z = mean z   (Q8, relative to the cell origin, < 256 * g <= 65536)
//   colour:   y = mean Y, z = mean U, w = mean V      (Q8)
constexpr uint32_t kCellMulti = 0x40000000u, kCellUsable = 0x20000000u, kCellCount = 0x00FFFFFFu;
__device__ __forceinline__ uint4 geo_summary(const uint4& v0, const uint4& v1) {   // first1, multi, count, sx ; sy, sz, -, -
  const uint32_t cnt = v0.z;
  if (cnt == 0) return make_uint4(0, 0, 0, 0);
  const uint32_t multi = v0.y != 0u ? kCellMulti : 0u;
  const uint32_t mx = mean_q8_u32(v0.w, cnt), my = mean_q8_u32(v1.x, cnt), mz = mean_q8_u32(v1.y, cnt);
  return make_uint4(multi | (cnt & kCellCount), mx | (my << 16), mz, 0u);
}
__device__ __forceinline__ uint4 col_summary(const uint4& v0, const uint4& v1, uint32_t thr_col_var, int* err) {
  // first1, multi, cnt_sy (lo, hi) ; su, sv, sy2 (lo, hi)
  const unsigned long long w0 = (unsigned long long)v0.z | ((unsigned long long)v0.w << 32);
  const unsigned long long sy2 = (unsigned long long)v1.z | ((unsigned long long)v1.w << 32);
  const unsigned long long cnt = w0 & 0xFFFFFFull, sy = w0 >> 24, su = v1.x, sv = v1.y;
  if (cnt == 0) return make_uint4(0, 0, 0, 0);
  if (cnt > 65536ull) atomicExch(err, 6);       // the packed U / V sums are only exact up to 65536 points per cell
  const uint32_t multi = v0.y != 0u ? kCellMulti : 0u;
  uint32_t my, mu, mv;
  if (sy < (1ull << 24) && cnt < (1ull << 24)) {                          // the usual case fits 32-bit division
    const uint32_t c32 = (uint32_t)cnt;
    my = mean_q8_u32((uint32_t)sy, c32); mu = mean_q8_u32((uint32_t)su, c32); mv = mean_q8_u32((uint32_t)sv, c32);
  } else {
    my = (uint32_t)((256ull * sy + cnt / 2) / cnt); mu = (uint32_t)((256ull * su + cnt / 2) / cnt);
    mv = (uint32_t)((256ull * sv + cnt / 2) / cnt);
  }
  // luminance variation: var(Y) = (cnt*sumY2 - sumY^2)/cnt^2 must not exceed t_var^2
  const unsigned __int128 num = (unsigned __int128)cnt * sy2 - (unsigned __int128)sy * sy;
  const unsigned long long tv = (unsigned long long)thr_col_var * cnt;
  const unsigned __int128 lim = (unsigned __int128)tv * tv;
  const uint32_t usable = num > lim ? 0u : kCellUsable;
  return make_uint4(multi | usable | ((uint32_t)cnt & kCellCount), my, mu, mv);
}

// ----------------------------------------------------------------------------------------------------------------
// K6 / K7: filter the type-1 boundary points against the trilinear blend of the 8 surrounding cell means
// ----------------------------------------------------------------------------------------------------------------
struct Nbhd { uint32_t key[8]; uint32_t wgt[8]; uint32_t w3; };
// weights fit 32 bits: (2g)^3 <= 2^27 for g <= 256
__device__ __forceinline__ bool neighbourhood(const GridDesc& G, const uint32_t p[3], Nbhd& N) {
  if (!(p[0] < G.th && p[1] < G.th && p[2] < G.th)) return false;
#pragma unroll
  for (int a = 0; a < 3; ++a)
    if (p[a] < G.disth || p[a] + G.disth >= G.th) return false;
  int32_t s[3]; uint32_t wa[3];
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    const uint32_t c = cell_div(p[a], G), rem = p[a] - c * G.g;
    s[a] = (int32_t)c + (rem < G.g / 2 ? -1 : 0);
    wa[a] = 2u * (uint32_t)((int32_t)p[a] - s[a] * (int32_t)G.g - (int32_t)(G.g / 2)) + 1u;
  }
  const uint32_t g2 = 2u * G.g;
  N.w3 = g2 * g2 * g2;
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const int dx = k & 1, dy = (k >> 1) & 1, dz = (k >> 2) & 1;
    const int32_t cx = s[0] + dx, cy = s[1] + dy, cz = s[2] + dz;
    const bool valid = cx >= 0 && cy >= 0 && cz >= 0 && (uint32_t)cx < G.w && (uint32_t)cy < G.w && (uint32_t)cz < G.w;
    N.key[k] = valid ? ((uint32_t)cx | ((uint32_t)cy << 10) | ((uint32_t)cz << 20)) : kCellEmpty;
    N.wgt[k] = (dx ? wa[0] : g2 - wa[0]) * (dy ? wa[1] : g2 - wa[1]) * (dz ? wa[2] : g2 - wa[2]);
  }
  return true;
}
// x / w3 where w3 = (2g)^3: a shift when g is a power of two
__device__ __forceinline__ unsigned long long div_w3(unsigned long long x, const GridDesc& G, uint32_t w3) {
  return G.g_shift >= 0 ? (x >> (3 * (G.g_shift + 1))) : (x / w3);
}
// the summaries of the 8 cells of a neighbourhood, from the cells' accumulators (16 independent 16-byte loads in flight)
template <bool kColour>
__device__ __forceinline__ void load_summaries(const UnpackArgs& a, const GridDesc& G, uint32_t fig, const Nbhd& N, uint4 c[8]) {
  const uint8_t* tab = static_cast<const uint8_t*>(G.table) + (uint64_t)fig * G.slots * 32u;      // 32-byte cells
#pragma unroll
  for (int h = 0; h < 2; ++h) {                                      // four cells (eight loads) in flight at a time
    uint4 r0[4], r1[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int j = 4 * h + i;
      r0[i] = make_uint4(0, 0, 0, 0); r1[i] = make_uint4(0, 0, 0, 0);
      if (N.key[j] != kCellEmpty) {
        const uint32_t cs = cell_find(G, fig, N.key[j]);
        if (cs != kCellEmpty) {
          r0[i] = __ldg(reinterpret_cast<const uint4*>(tab + (uint64_t)cs * 32u));
          r1[i] = __ldg(reinterpret_cast<const uint4*>(tab + (uint64_t)cs * 32u) + 1);
        }
      }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i)
      c[4 * h + i] = kColour ? col_summary(r0[i], r1[i], a.sm.thr_col_var, a.err) : geo_summary(r0[i], r1[i]);
  }
}

// One type-1 boundary point against the two grids.  `want` bit 0: geometry, bit 1: colour (the grids whose neighbourhood
// holds a multi-patch cell).  Returns moved | recoloured << 1.
__device__ __forceinline__ uint32_t filter_apply(const UnpackArgs& a, uint32_t fig, uint32_t f, const uint4& raw, uint32_t want) {
  const uint32_t p[3] = {raw.y & 0xFFFFu, raw.y >> 16, raw.z & 0xFFFFu};
  const uint32_t col[3] = {raw.z >> 16, raw.w & 0xFFFFu, raw.w >> 16};
  const uint64_t gi = (uint64_t)f * a.out.cap + raw.x;
  uint32_t result = 0;
  // ---- geometry (K6) ----
  if (want & 1u) {
    const GridDesc& G = a.sm.geo;
    Nbhd Ng;
    neighbourhood(G, p, Ng);
    uint4 cg[8];
    load_summaries<false>(a, G, fig, Ng, cg);
    unsigned long long C[3] = {0, 0, 0}, cntw = 0;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const uint32_t cnt = cg[j].x & kCellCount;
      uint32_t m[3] = {256u * p[0], 256u * p[1], 256u * p[2]};                  // empty cell -> the point itself
      if (cnt > 0) {
        m[0] = 256u * ((Ng.key[j] & 1023u) * G.g) + (cg[j].y & 0xFFFFu);
        m[1] = 256u * (((Ng.key[j] >> 10) & 1023u) * G.g) + (cg[j].y >> 16);
        m[2] = 256u * ((Ng.key[j] >> 20) * G.g) + (cg[j].z & 0xFFFFu);
      }
#pragma unroll
      for (int ax = 0; ax < 3; ++ax) C[ax] += (unsigned long long)Ng.wgt[j] * m[ax];
      cntw += (unsigned long long)Ng.wgt[j] * cnt;
    }
    const unsigned long long count = div_w3(cntw, G, Ng.w3);
    if (count > 0) {
      unsigned long long c4[3], D2 = 0;
#pragma unroll
      for (int ax = 0; ax < 3; ++ax) {
        c4[ax] = div_w3(C[ax] + Ng.w3 / 2, G, Ng.w3);
        const long long d = (long long)(256ull * p[ax]) - (long long)c4[ax];
        D2 += (unsigned long long)(d * d);
      }
      const unsigned long long m = a.sm.thr_geo > count ? a.sm.thr_geo : count;
      const unsigned __int128 lhs = (unsigned __int128)2 * count * D2 + 65536u;
      const unsigned __int128 rhs = (unsigned __int128)262144u * m;
      if (lhs >= rhs) {
        bool changed = false;
        uint16_t q[3];
#pragma unroll
        for (int ax = 0; ax < 3; ++ax) {
          unsigned long long rr = (c4[ax] + 128) >> 8;
          if (rr > 65535) rr = 65535;
          q[ax] = (uint16_t)rr;
          changed |= q[ax] != p[ax];
        }
        if (changed) {
          uint16_t* d = a.out.pos + gi * 3;
          d[0] = q[0]; d[1] = q[1]; d[2] = q[2];
          result |= 1u;
        }
      }
    }
  }
  // ---- colour (K7), on the same pre-smoothing position ----
  if (want & 2u) {
    const GridDesc& G = a.sm.col;
    Nbhd Nc;
    neighbourhood(G, p, Nc);
    uint4 cc[8];
    load_summaries<true>(a, G, fig, Nc, cc);
    unsigned long long C[3] = {0, 0, 0};
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      bool usable = (cc[j].x & kCellCount) != 0 && (cc[j].x & kCellUsable) != 0;
      const uint32_t mean[3] = {cc[j].y, cc[j].z, cc[j].w};
      if (usable) {
        const long long dy = (long long)mean[0] - (long long)(256u * col[0]);
        if ((unsigned long long)(dy < 0 ? -dy : dy) > 256ull * a.sm.thr_col_diff) usable = false;
      }
#pragma unroll
      for (int ax = 0; ax < 3; ++ax) C[ax] += (unsigned long long)Nc.wgt[j] * (usable ? mean[ax] : 256u * col[ax]);
    }
    uint32_t q[3]; unsigned long long dist = 0;
#pragma unroll
    for (int ax = 0; ax < 3; ++ax) {
      const unsigned long long c4 = div_w3(C[ax] + Nc.w3 / 2, G, Nc.w3);
      unsigned long long rr = (c4 + 128) >> 8;
      if (rr > 65535) rr = 65535;
      q[ax] = (uint32_t)rr;
      const long long d = (long long)q[ax] - (long long)col[ax];
      dist += (unsigned long long)(d < 0 ? -d : d) * (ax == 0 ? 10u : 1u);
    }
    if (dist >= a.sm.thr_col_smooth && dist > 0) {
      const uint32_t c = yuv_to_rgb_packed(q[0], q[1], q[2]);
      uint8_t* d = a.out.rgb + gi * 3;
      d[0] = (uint8_t)c; d[1] = (uint8_t)(c >> 8); d[2] = (uint8_t)(c >> 16);
      if (a.out.yuv) { uint16_t* y = a.out.yuv + gi * 3; y[0] = (uint16_t)q[0]; y[1] = (uint16_t)q[1]; y[2] = (uint16_t)q[2]; }
      result |= 2u;
    }
  }
  return result;
}

// The filter is two kernels.  PROBE (every type-1 boundary point, light in registers so that many loads are in flight): fetch
// the multi-patch bits of the 16 neighbouring cells (a bitmap, 32 cells per word) and keep the point if some cell of a grid has it set -- most
// boundary points have none and are done.  APPLY (the survivors): the expensive blend, in full warps.
__device__ __forceinline__ uint32_t probe_multi(const GridDesc& G, uint32_t fig, const uint32_t p[3]) {
  Nbhd N;
  if (!neighbourhood(G, p, N)) return 0u;
  const uint32_t* bits = G.mbits + (uint64_t)fig * G.mwords;         // one bit per table slot: 32 cells per word
  uint32_t any = 0;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    if (N.key[j] == kCellEmpty) continue;
    const uint32_t cs = cell_find(G, fig, N.key[j]);
    if (cs != kCellEmpty) any |= (__ldg(bits + (cs >> 5)) >> (cs & 31u)) & 1u;
  }
  return any;
}

// The same for a dense grid with power-of-two cell edge and width: the neighbourhood's first cell along an axis is
// (p - g/2) >> log2(g) (the margin test guarantees both cells of every axis exist), and the two cells along x are neighbouring
// bits of the bitmap -- four word loads instead of eight (a fifth when the pair straddles a word).
__device__ __forceinline__ uint32_t probe_multi_fast(const GridDesc& G, uint32_t fig, const uint32_t p[3]) {
#pragma unroll
  for (int ax = 0; ax < 3; ++ax)
    if (p[ax] >= G.th || p[ax] < G.disth || p[ax] + G.disth >= G.th) return 0u;
  const uint32_t hg = G.g >> 1, gs = (uint32_t)G.g_shift, ws = G.w_shift;
  const uint32_t sx = (p[0] - hg) >> gs, sy = (p[1] - hg) >> gs, sz = (p[2] - hg) >> gs;
  const uint32_t* bits = G.mbits + (uint64_t)fig * G.mwords;
  const uint32_t c00 = sx + (sy << ws) + (sz << (2u * ws));
  uint32_t any = 0;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const uint32_t cs = c00 + ((k & 1) ? (1u << ws) : 0u) + ((k & 2) ? (1u << (2u * ws)) : 0u);
    const uint32_t b = cs & 31u;
    any |= (__ldg(bits + (cs >> 5)) >> b) & 3u;
    if (b == 31u) any |= __ldg(bits + (cs >> 5) + 1) & 1u;
  }
  return any;
}

#ifndef TMC2_PROBE_MINCTA
#define TMC2_PROBE_MINCTA 8
#endif
__global__ void __launch_bounds__(256, TMC2_PROBE_MINCTA) smooth_probe_kernel(const __grid_constant__ UnpackArgs a) {
  const uint32_t fig = blockIdx.y;
  const uint32_t f = a.sm.group_first_frame + fig;
  const uint32_t n = min((uint64_t)a.sm.blist_count[f], a.sm.blist_cap);
  const BoundaryEntry* L = a.sm.blist + (uint64_t)f * a.sm.blist_cap;
  const uint32_t lane = lane_id();
  const uint32_t n_round = (n + 31u) & ~31u;                                     // whole warps stay in the loop together
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_round; i += gridDim.x * blockDim.x) {
    uint32_t want = 0;
    if (i < n) {
      const uint4 raw = __ldg(reinterpret_cast<const uint4*>(&L[i]));
      const uint32_t p[3] = {raw.y & 0xFFFFu, raw.y >> 16, raw.z & 0xFFFFu};
      if (a.sm.geo.on && (a.sm.geo.fast ? probe_multi_fast(a.sm.geo, fig, p) : probe_multi(a.sm.geo, fig, p))) want |= 1u;
      if (a.sm.col.on && a.has_attr && (a.sm.col.fast ? probe_multi_fast(a.sm.col, fig, p) : probe_multi(a.sm.col, fig, p)))
        want |= 2u;                                                                 // pre-smoothing position
    }
    const uint32_t wm = __ballot_sync(kFull, want != 0u);
    if (wm == 0u) continue;
    uint32_t base = 0;
    if (lane == 0) base = atomicAdd(&a.sm.slist_count[f], (uint32_t)__popc(wm));
    base = __shfl_sync(kFull, base, 0);
    if (want) a.sm.slist[(uint64_t)f * a.sm.blist_cap + base + __popc(wm & ((1u << lane) - 1u))] = i | (want << 30);
  }
}

#ifndef TMC2_APPLY_MINCTA
#define TMC2_APPLY_MINCTA 1
#endif
__global__ void __launch_bounds__(128, TMC2_APPLY_MINCTA) smooth_apply_kernel(const __grid_constant__ UnpackArgs a) {
  const uint32_t fig = blockIdx.y;
  const uint32_t f = a.sm.group_first_frame + fig;
  const uint32_t m = min((uint64_t)a.sm.slist_count[f], a.sm.blist_cap);
  const BoundaryEntry* L = a.sm.blist + (uint64_t)f * a.sm.blist_cap;
  const uint32_t* S = a.sm.slist + (uint64_t)f * a.sm.blist_cap;
  uint32_t moved = 0, recol = 0;
  for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < m; j += gridDim.x * blockDim.x) {
    const uint32_t e = S[j];
    const uint4 raw = __ldg(reinterpret_cast<const uint4*>(&L[e & 0x3FFFFFFFu]));
    const uint32_t r = filter_apply(a, fig, f, raw, e >> 30);
    moved += r & 1u; recol += r >> 1;
  }
  moved = __reduce_add_sync(kFull, moved);
  recol = __reduce_add_sync(kFull, recol);
  if (lane_id() == 0) {
    if (moved) atomicAdd(&a.sm.changed[f], (unsigned long long)moved);
    if (recol) atomicAdd(&a.sm.changed[a.n_frames + f], (unsigned long long)recol);
  }
}

// back to all-zero cells (free keys, clean bitmaps) for the next launch: the touched bitmap names the cells
__global__ void __launch_bounds__(256) smooth_clear_kernel(const __grid_constant__ UnpackArgs a) {
  const uint32_t fig = blockIdx.y;
#pragma unroll
  for (int which = 0; which < 2; ++which) {
    const GridDesc& G = which ? a.sm.col : a.sm.geo;
    if (!G.on) continue;
    uint32_t* tb = G.tbits + (uint64_t)fig * G.twords;
    uint32_t* mb = G.mbits + (uint64_t)fig * G.mwords;
    uint4* tab = reinterpret_cast<uint4*>(G.table) + ((uint64_t)fig * G.slots) * 2;      // 32-byte cells
    // a word of the touched bitmap = 32 quads = 128 cells = four words of the multi-patch bitmap
    for (uint64_t w = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; w < G.twords; w += (uint64_t)gridDim.x * blockDim.x) {
      uint32_t t = tb[w];
      if (t == 0) continue;
      tb[w] = 0;
#pragma unroll
      for (uint32_t i = 0; i < (1u << kTouchShift); ++i)
        if ((w << kTouchShift) + i < G.mwords) mb[(w << kTouchShift) + i] = 0;
      while (t) {
        const uint64_t q = w * 32u + ((uint32_t)__ffs(t) - 1u);                     // quad = cells 4q .. 4q+3 = one 128-byte line
        t &= t - 1u;
#pragma unroll
        for (uint32_t i = 0; i < (1u << kTouchShift); ++i) {
          const uint64_t cs = (q << kTouchShift) + i;
          if (cs >= G.slots) break;
          tab[cs * 2] = make_uint4(0, 0, 0, 0);
          tab[cs * 2 + 1] = make_uint4(0, 0, 0, 0);
          if (!G.identity) G.keys[(uint64_t)fig * G.slots + cs] = kCellEmpty;
        }
      }
    }
  }
}

__global__ void __launch_bounds__(256) fill_u32_kernel(uint32_t* p, uint64_t n, uint32_t v) {
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) p[i] = v;
}

// ----------------------------------------------------------------------------------------------------------------
// ingest_planes_kernel: the caller's device-resident planes (TMC2_INPUT_DEVICE) -> batch layout.  CTA = (row range,
// plane); thread = one 16-byte chunk of a source row at a time, four chunks loaded before any is stored.  A chunk takes
// the vector path when the plane's base and pitch are 16-byte aligned (decided on the host) and the chunk is whole; the
// rest of a row and every chunk of an unaligned plane go sample by sample.  Destination rows are 64-element aligned.
// ----------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t p010_pair(uint32_t w) { return (w >> 6) & 0x03FF03FFu; }   // two samples, raw >> 6

__device__ __forceinline__ void ingest_store_vec(const IngestPlane& p, uint32_t op, uint32_t r, uint32_t c, uint4 v) {
  if (op == kIngestUv16) {                 // u0 v0 u1 v1 | u2 v2 u3 v3 -> u0 u1 u2 u3, v0 v1 v2 v3
    const uint2 u = make_uint2(p010_pair(__byte_perm(v.x, v.y, 0x5410)), p010_pair(__byte_perm(v.z, v.w, 0x5410)));
    const uint2 w = make_uint2(p010_pair(__byte_perm(v.x, v.y, 0x7632)), p010_pair(__byte_perm(v.z, v.w, 0x7632)));
    *reinterpret_cast<uint2*>(p.dst + (size_t)r * p.dpitch + c * 8) = u;
    *reinterpret_cast<uint2*>(p.dst2 + (size_t)r * p.dpitch + c * 8) = w;
    return;
  }
  if (op == kIngestShr16) v = make_uint4(p010_pair(v.x), p010_pair(v.y), p010_pair(v.z), p010_pair(v.w));
  *reinterpret_cast<uint4*>(p.dst + (size_t)r * p.dpitch + c * 16) = v;
}

__device__ __forceinline__ void ingest_narrow(const IngestPlane& p, uint32_t op, uint32_t r, uint32_t c, uint32_t n) {
  const uint8_t* s = p.src + (size_t)r * p.spitch + c * 16;
  if (op == kIngestCopy8) {
    uint8_t* d = p.dst + (size_t)r * p.dpitch + c * 16;
    for (uint32_t j = 0; j < n; ++j) d[j] = __ldg(s + j);
  } else if (op == kIngestUv16) {
    const uint16_t* s16 = reinterpret_cast<const uint16_t*>(s);
    uint16_t* du = reinterpret_cast<uint16_t*>(p.dst + (size_t)r * p.dpitch) + c * 4;
    uint16_t* dv = reinterpret_cast<uint16_t*>(p.dst2 + (size_t)r * p.dpitch) + c * 4;
    for (uint32_t j = 0; j < n / 4; ++j) {
      du[j] = (uint16_t)(__ldg(s16 + 2 * j) >> 6);
      dv[j] = (uint16_t)(__ldg(s16 + 2 * j + 1) >> 6);
    }
  } else {
    const uint16_t* s16 = reinterpret_cast<const uint16_t*>(s);
    uint16_t* d = reinterpret_cast<uint16_t*>(p.dst + (size_t)r * p.dpitch + c * 16);
    const uint32_t sh = op == kIngestShr16 ? 6u : 0u;
    for (uint32_t j = 0; j < n / 2; ++j) d[j] = (uint16_t)(__ldg(s16 + j) >> sh);
  }
}

constexpr uint32_t kIngestThreads = 256, kIngestUnroll = 4;

__global__ void __launch_bounds__(kIngestThreads) ingest_planes_kernel(const IngestPlane* __restrict__ table, uint32_t n_planes,
                                                                     uint32_t rows_per_cta) {
  for (uint32_t pi = blockIdx.y; pi < n_planes; pi += gridDim.y) {
    const IngestPlane p = table[pi];
    const uint32_t r0 = blockIdx.x * rows_per_cta;
    if (r0 >= p.rows) continue;
    const uint32_t rows = min(p.rows - r0, rows_per_cta);
    const uint32_t nch = (p.row_bytes + 15u) >> 4;
    const uint32_t total = rows * nch;
    const uint32_t op = p.op & 0xFFu;
    const bool vec = (p.op & kIngestVec) != 0;
    for (uint32_t i0 = threadIdx.x; i0 < total; i0 += kIngestUnroll * kIngestThreads) {
      uint4 v[kIngestUnroll];
#pragma unroll
      for (uint32_t k = 0; k < kIngestUnroll; ++k) {
        const uint32_t i = i0 + k * kIngestThreads;
        const uint32_t r = r0 + i / nch, c = i % nch;
        v[k] = make_uint4(0, 0, 0, 0);
        if (vec && i < total && c * 16 + 16 <= p.row_bytes) v[k] = ldg_nc_v4(p.src + (size_t)r * p.spitch + c * 16);
      }
#pragma unroll
      for (uint32_t k = 0; k < kIngestUnroll; ++k) {
        const uint32_t i = i0 + k * kIngestThreads;
        if (i >= total) break;
        const uint32_t r = r0 + i / nch, c = i % nch;
        const uint32_t n = min(16u, p.row_bytes - c * 16);
        if (vec && n == 16) ingest_store_vec(p, op, r, c, v[k]);
        else ingest_narrow(p, op, r, c, n);
      }
    }
  }
}

// ----------------------------------------------------------------------------------------------------------------
// launch wrappers
// ----------------------------------------------------------------------------------------------------------------
static inline int after_launch() { ++g_launches; return (int)cudaGetLastError(); }
// grid.x of the per-frame post-pass kernels (grid.y = frames of the group): 16 blocks per SM over all frames (other grids
// measured no different, DESIGN.md section 9)
static unsigned post_blocks(unsigned frames) { return (148u * 16u + frames - 1) / frames; }

int launch_block_to_patch(const UnpackArgs& a, uint32_t n_slots, void* stream) {
  if (n_slots == 0) return 0;
  const uint32_t blocks = (n_slots + 255) / 256;
  block_to_patch_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(a, n_slots, const_cast<uint32_t*>(a.block_to_patch));
  return after_launch();
}

int launch_compact_owned(const UnpackArgs& a, void* stream) {
  if (a.n_frames == 0) return 0;
  compact_owned_kernel<<<a.n_frames, 1024, 0, (cudaStream_t)stream>>>(a);
  return after_launch();
}

template <bool kSmooth, bool kDebug, bool kFast, bool kAttr>
static int launch_emit_t(const UnpackArgs& a, const TileMaps& tm, uint32_t slot_begin, uint32_t slot_end, cudaStream_t s) {
  const size_t smem = (size_t)emit_layout(kSmooth, kDebug, kFast).bytes * kEmitWarps;
  auto kern = emit_kernel<kSmooth, kDebug, kFast, kAttr>;
  static bool configured[64] = {};               // the dynamic shared memory limit is a per-device attribute of the function
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return (int)e;
  if (dev < 0 || dev >= 64) return (int)cudaErrorInvalidDevice;
  if (!configured[dev]) {
    e = cudaFuncSetAttribute((const void*)kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    configured[dev] = true;
  }
  const uint32_t blocks = (slot_end - slot_begin + kEmitWarps - 1) / kEmitWarps;
  kern<<<blocks, kEmitWarps * 32, smem, s>>>(a, tm, slot_begin, slot_end);
  return after_launch();
}

int launch_count(const UnpackArgs& a, uint32_t tile_begin, uint32_t tile_end, void* stream) {
  if (tile_end <= tile_begin) return 0;
  count_kernel<<<tile_end - tile_begin, kWarpsPerTile * 32, 0, (cudaStream_t)stream>>>(a, tile_begin);
  return after_launch();
}

int launch_slot_scan(const UnpackArgs& a, void* stream) {
  if (a.n_frames == 0) return 0;
  slot_scan_kernel<<<a.n_frames, 1024, 0, (cudaStream_t)stream>>>(a);
  return after_launch();
}

int launch_emit(const UnpackArgs& a, const TileMaps& tm, bool smooth, uint32_t tile_begin, uint32_t tile_end, void* stream) {
  if (tile_end <= tile_begin) return 0;
  const cudaStream_t s = (cudaStream_t)stream;
  const uint32_t s0 = tile_begin * kWarpsPerTile, s1 = tile_end * kWarpsPerTile;
  const bool debug = a.out.yuv || a.out.part || a.out.pix || a.out.btype;
  const bool attr = a.has_attr != 0;
#define TMC2_EMIT(S, D, F) (attr ? launch_emit_t<S, D, F, true>(a, tm, s0, s1, s) : launch_emit_t<S, D, F, false>(a, tm, s0, s1, s))
  if (smooth) {
    if (debug) return TMC2_EMIT(true, true, false);
    // the usual grids (dense tables, power-of-two cell edges, geometry edge <= 8) get the instantiation without generic branches
    const bool fast = (!a.sm.geo.on || (a.sm.geo.fast == 1u && a.sm.geo.g <= 8u)) && (!a.sm.col.on || a.sm.col.fast);
    return fast ? TMC2_EMIT(true, false, true) : TMC2_EMIT(true, false, false);
  }
  return debug ? TMC2_EMIT(false, true, false) : TMC2_EMIT(false, false, false);
#undef TMC2_EMIT
}

int launch_upsample(const UnpackArgs& a, uint8_t* occ_full, void* stream) {
  upsample_kernel<<<148 * 8, 256, 0, (cudaStream_t)stream>>>(a, occ_full);
  return after_launch();
}

int launch_smooth_filter(const UnpackArgs& a, void* stream) {
  if (a.sm.group_frames == 0) return 0;
  const unsigned bx = post_blocks(a.sm.group_frames);
  smooth_probe_kernel<<<dim3(bx, a.sm.group_frames), 256, 0, (cudaStream_t)stream>>>(a);
  int e = after_launch();
  if (e) return e;
  smooth_apply_kernel<<<dim3(bx, a.sm.group_frames), 128, 0, (cudaStream_t)stream>>>(a);
  return after_launch();
}

int launch_smooth_clear(const UnpackArgs& a, void* stream) {
  if (a.sm.group_frames == 0) return 0;
  const unsigned bx = post_blocks(a.sm.group_frames);
  smooth_clear_kernel<<<dim3(bx, a.sm.group_frames), 256, 0, (cudaStream_t)stream>>>(a);
  return after_launch();
}

int launch_yuv_to_rgb_flat(const uint16_t* yuv, uint8_t* rgb, uint64_t n, void* stream) {
  if (n == 0) return 0;
  uint64_t blocks = (n + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  yuv_to_rgb_flat_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(yuv, rgb, n);
  return after_launch();
}
int launch_fill_u32(uint32_t* p, uint64_t n, uint32_t v, void* stream) {
  if (n == 0) return 0;
  fill_u32_kernel<<<148 * 8, 256, 0, (cudaStream_t)stream>>>(p, n, v);
  return after_launch();
}

int launch_ingest_planes(const IngestPlane* table, uint32_t n_planes, uint32_t max_rows, uint32_t max_row_bytes, void* stream) {
  if (n_planes == 0 || max_rows == 0 || max_row_bytes == 0) return 0;
  // ~64 KB of source per CTA: enough work per CTA to amortise its start, enough CTAs to fill 148 SMs several times over
  const uint32_t rows_per_cta = std::max(1u, (64u << 10) / max_row_bytes);
  const dim3 grid((max_rows + rows_per_cta - 1) / rows_per_cta, std::min(n_planes, 65535u));
  ingest_planes_kernel<<<grid, kIngestThreads, 0, (cudaStream_t)stream>>>(table, n_planes, rows_per_cta);
  return after_launch();
}

}  // namespace tmc2
