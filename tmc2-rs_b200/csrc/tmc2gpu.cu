// tmc2gpu.cu -- host runtime behind include/tmc2gpu.h: validation (everything the reference asserts), HBM layout,
// pinned staging, stream/event plumbing, frame-wise multi-GPU sharding, and the C ABI entry points.
//
// This file replaces the per-frame driver of the reference, src/decoder.rs:188-314, with a GOF-batched one:
//   submit_gof  = validate + stage + H2D + [K2 block_to_patch] + [fused unpack] + [smoothing] + counts D2H
//   next_frame  = in-order hand-out of PointSet3-compatible buffers (src/lib.rs:81, src/codec.rs:20-36)
// There is no CPU fallback anywhere: without a CUDA device every entry point returns TMC2_ERR_NO_DEVICE.
#include <cuda.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <functional>
#include <thread>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/tmc2gpu.h"
#include "device_types.h"

using namespace tmc2;

namespace {

// ---------------------------------------------------------------------------------------------------------------
// utilities
// ---------------------------------------------------------------------------------------------------------------
struct Err {
  tmc2_status st = TMC2_OK;
  std::string msg;
};

static std::string fmt(const char* f, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, f);
  vsnprintf(buf, sizeof buf, f, ap);
  va_end(ap);
  return buf;
}

#define CU(call)                                                                                      \
  do {                                                                                                \
    cudaError_t _e = (call);                                                                          \
    if (_e != cudaSuccess) {                                                                          \
      err.st = TMC2_ERR_CUDA;                                                                         \
      err.msg = fmt("%s failed: %s (%s:%d)", #call, cudaGetErrorString(_e), __FILE__, __LINE__);      \
      return err.st;                                                                                  \
    }                                                                                                 \
  } while (0)
#define KL(call)                                                                                      \
  do {                                                                                                \
    int _e = (call);                                                                                  \
    if (_e != 0) {                                                                                    \
      err.st = TMC2_ERR_CUDA;                                                                         \
      err.msg = fmt("%s failed: %s", #call, cudaGetErrorString((cudaError_t)_e));                     \
      return err.st;                                                                                  \
    }                                                                                                 \
  } while (0)
#define FAIL(code, ...)            \
  do {                             \
    err.st = (code);               \
    err.msg = fmt(__VA_ARGS__);    \
    return err.st;                 \
  } while (0)

// TMC2_TRACE=1: host-side phase timings of the streaming path on stderr (diagnostics only)
static bool trace_on() { static const bool on = getenv("TMC2_TRACE") != nullptr; return on; }
struct TraceClock {
  std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
  double lap() {
    const auto t1 = std::chrono::steady_clock::now();
    const double ms = std::chrono::duration<double, std::milli>(t1 - t0).count();
    t0 = t1;
    return ms;
  }
};

static inline uint32_t round_up(uint32_t x, uint32_t m) { return (x + m - 1) / m * m; }
static inline uint64_t round_up64(uint64_t x, uint64_t m) { return (x + m - 1) / m * m; }
static inline uint64_t pow2_at_least(uint64_t x) { uint64_t p = 1; while (p < x) p <<= 1; return p; }

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  cudaError_t ensure(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr; cap = 0;
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e == cudaSuccess) cap = bytes;
    return e;
  }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
  template <typename T> T* as() const { return reinterpret_cast<T*>(p); }
};
struct PinBuf {
  void* p = nullptr;
  size_t cap = 0;
  cudaError_t ensure(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFreeHost(p);
    p = nullptr; cap = 0;
    bytes = bytes + bytes / 4;   // head room: later GOFs of the same stream rarely need a re-pin
    cudaError_t e = cudaHostAlloc(&p, bytes, cudaHostAllocDefault);
    if (e == cudaSuccess) cap = bytes;
    return e;
  }
  void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
  template <typename T> T* as() const { return reinterpret_cast<T*>(p); }
};

// registry of memory handed out by tmc2gpu_alloc_pinned: planes inside it are DMA'd without staging
std::mutex g_pin_mu;
std::vector<std::pair<const uint8_t*, size_t>> g_pinned;
static std::vector<std::pair<const uint8_t*, size_t>> pinned_snapshot() {
  std::lock_guard<std::mutex> lk(g_pin_mu);
  return g_pinned;
}
static bool is_pinned(const std::vector<std::pair<const uint8_t*, size_t>>& reg, const void* p, size_t bytes) {
  const uint8_t* q = static_cast<const uint8_t*>(p);
  for (auto& r : reg)
    if (q >= r.first && q + bytes <= r.first + r.second) return true;
  return false;
}

// Staging of pageable planes (what an unmodified tmc2-rs host hands over: `Vec<u8>`, src/decoder.rs:1136-1140) into pinned
// memory runs on a small pool of host threads: one thread moves ~10 GB/s, the PCIe link takes 50+.  TMC2_STAGE_THREADS
// overrides the pool size (1 = the calling thread only).
class StagePool {
 public:
  // never destroyed: the workers wait on its condition variable for the life of the process (destroying a condition
  // variable with waiters at exit would block)
  static StagePool& get() { static StagePool* p = new StagePool(); return *p; }
  unsigned threads() const { return n_; }
  // fn(i) for i in [0, items); returns when all are done.  The calling thread takes part.
  void run(size_t items, const std::function<void(size_t)>& fn) {
    if (items == 0) return;
    if (n_ <= 1 || items == 1) { for (size_t i = 0; i < items; ++i) fn(i); return; }
    std::unique_lock<std::mutex> lk(mu_);
    fn_ = &fn; items_ = items; next_.store(0); left_ = items; finished_ = 0; ++epoch_;
    cv_.notify_all();
    lk.unlock();
    work();
    lk.lock();
    // every worker has passed through this job (none is still inside work() when the next job is set up)
    done_.wait(lk, [&] { return left_ == 0 && finished_ == n_ - 1; });
    fn_ = nullptr;
  }
 private:
  StagePool() {
    unsigned n = std::min(8u, std::max(1u, std::thread::hardware_concurrency() / 2));
    if (const char* e = getenv("TMC2_STAGE_THREADS")) n = (unsigned)std::max(1, atoi(e));
    n_ = n;
    for (unsigned i = 1; i < n_; ++i) std::thread([this] { loop(); }).detach();
  }
  void work() {
    for (;;) {
      const size_t i = next_.fetch_add(1);
      if (i >= items_) break;
      (*fn_)(i);
      std::lock_guard<std::mutex> lk(mu_);
      if (--left_ == 0) done_.notify_all();
    }
  }
  void loop() {
    uint64_t seen = 0;
    for (;;) {
      {
        std::unique_lock<std::mutex> lk(mu_);
        cv_.wait(lk, [&] { return epoch_ != seen; });
        seen = epoch_;
      }
      work();
      std::lock_guard<std::mutex> lk(mu_);
      ++finished_;
      done_.notify_all();
    }
  }
  unsigned n_ = 1;
  std::mutex mu_;
  std::condition_variable cv_, done_;
  const std::function<void(size_t)>* fn_ = nullptr;
  size_t items_ = 0, left_ = 0;
  unsigned finished_ = 0;
  std::atomic<size_t> next_{0};
  uint64_t epoch_ = 0;
};

// TMA descriptors of the plane arrays (device_types.h TileMaps).  cuTensorMapEncodeTiled is reached through the runtime's
// driver entry point lookup, so the library does not link against libcuda.
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) {
      cudaGetLastError();
      p = nullptr;
    }
    return (EncodeTiledFn)p;
  }();
  return fn;
}
// rank-`rank` tensor of `esz`-byte elements: dims[] elements, strides[] bytes of dims 1.., box[] elements
static bool encode_map(unsigned long long* out, void* base, uint32_t esz, uint32_t rank, const uint64_t* dims, const uint64_t* strides,
                       const uint32_t* box) {
  static_assert(sizeof(CUtensorMap) == 128, "CUtensorMap is 128 bytes");
  EncodeTiledFn fn = encode_tiled_fn();
  if (!fn || !base) return false;
  cuuint64_t d[5]; cuuint64_t st[5]; cuuint32_t b[5]; cuuint32_t es[5];
  for (uint32_t i = 0; i < rank; ++i) { d[i] = dims[i]; b[i] = box[i]; es[i] = 1; if (i) st[i - 1] = strides[i - 1]; }
  CUtensorMap m;
  const CUresult r = fn(&m, esz == 1 ? CU_TENSOR_MAP_DATA_TYPE_UINT8 : CU_TENSOR_MAP_DATA_TYPE_UINT16, rank, base, d, st, b, es,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return false;
  memcpy(out, &m, 128);
  return true;
}

// Allocation that holds a device pointer (cuMemGetAddressRange, reached the same way).
typedef CUresult (*AddressRangeFn)(CUdeviceptr*, size_t*, CUdeviceptr);
static AddressRangeFn address_range_fn() {
  static AddressRangeFn fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuMemGetAddressRange", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) {
      cudaGetLastError();
      p = nullptr;
    }
    return (AddressRangeFn)p;
  }();
  return fn;
}

// ---------------------------------------------------------------------------------------------------------------
// validation: everything the reference asserts / unwraps / leaves unimplemented on this path
// ---------------------------------------------------------------------------------------------------------------
static void helper_i64(const tmc2_patch& p, int64_t u, int64_t v, int64_t res, int64_t sscale, int64_t& x, int64_t& y) {
  // src/decoder.rs:853-867 in signed arithmetic (agrees with wrapping usize whenever the result is in range)
  const int64_t u0 = (int64_t)p.u0 * res, v0 = (int64_t)p.v0 * res;
  const int64_t su = (int64_t)p.size_u0 * sscale, sv = (int64_t)p.size_v0 * sscale;
  switch (p.patch_orientation) {
    case TMC2_ORIENT_DEFAULT: x = u + u0; y = v + v0; break;
    case TMC2_ORIENT_ROT90:   x = sv - 1 - v + u0; y = u + v0; break;
    case TMC2_ORIENT_ROT180:  x = su - 1 - u + u0; y = sv - 1 - v + v0; break;
    case TMC2_ORIENT_ROT270:  x = v + u0; y = su - 1 - u + v0; break;
    case TMC2_ORIENT_MIRROR:  x = su - 1 - u + u0; y = v + v0; break;
    case TMC2_ORIENT_MROT90:  x = sv - 1 - v + u0; y = su - 1 - u + v0; break;
    case TMC2_ORIENT_MROT180: x = u + u0; y = sv - 1 - v + v0; break;
    default:                  x = v + u0; y = u + v0; break;  // Swap, MRot270
  }
}

static tmc2_status validate_params(const tmc2_gof* g, Err& err) {
  if (!g) FAIL(TMC2_ERR_INVALID_ARG, "gof is NULL");
  const tmc2_params& P = g->params;
  if (g->frame_count && !g->frames) FAIL(TMC2_ERR_INVALID_ARG, "frames is NULL");
  if (g->width == 0 || g->height == 0 || g->occ_width == 0 || g->occ_height == 0)
    FAIL(TMC2_ERR_INVALID_ARG, "zero-sized frame");
  if (g->width >= 32768 || g->height >= 32768) FAIL(TMC2_ERR_CAPACITY, "frame larger than 32767 pixels");
  if (P.occupancy_resolution == 0 || P.occupancy_precision == 0)
    FAIL(TMC2_ERR_INVALID_ARG, "occupancy resolution / precision must be non-zero");
  if (P.occupancy_resolution > 64) FAIL(TMC2_ERR_CAPACITY, "occupancy resolution > 64");
  if (P.enable_size_quantization || P.multiple_streams || P.pbf_enabled || P.enhanced_occupancy_map ||
      P.point_local_reconstruction || P.single_map_pixel_interleaving || P.use_additional_points_patch)
    FAIL(TMC2_ERR_UNSUPPORTED, "reference branch is unimplemented!() (codec.rs:285,303,314,399,402,454,494)");
  if (P.map_count_minus1 != 1) FAIL(TMC2_ERR_MAP_COUNT, "map_count must be 2 (codec.rs:415-432)");
  if (P.attribute_count > 1) FAIL(TMC2_ERR_UNSUPPORTED, "attribute_count > 1 (decoder.rs:133)");
  if (P.orientation_mode > 1) FAIL(TMC2_ERR_INVALID_ARG, "orientation_mode");
  // 4:2:0 chroma planes hold (W/2) x (H/2) samples (decoder.rs:976-977 indexes them with w/2 and v/2): with an odd width or
  // height the last pixel row / column would read past them
  if (P.attribute_count && ((g->width | g->height) & 1u))
    FAIL(TMC2_ERR_INVALID_ARG, "odd frame width / height with 4:2:0 attributes (decoder.rs:976-977)");
  // Image::get asserts (decoder.rs:974): the upsample touches every pixel of the tile
  if ((g->width - 1) / P.occupancy_precision >= g->occ_width || (g->height - 1) / P.occupancy_precision >= g->occ_height)
    FAIL(TMC2_ERR_INVALID_ARG, "occupancy video smaller than frame / precision (decoder.rs:974 assert)");
  if (P.geometry_smoothing || P.color_smoothing) {
    if (P.geometry_bitdepth_3d == 0 || P.geometry_bitdepth_3d > 16) FAIL(TMC2_ERR_INVALID_ARG, "geometry_bitdepth_3d");
    const uint32_t maxs = 1u << P.geometry_bitdepth_3d;
    if (2ull * g->width * g->height >= (1ull << 24))
      FAIL(TMC2_ERR_UNSUPPORTED, "smoothing supports atlases up to 8.3 M pixels (per-cell sums are 32-bit)");
    if (P.grid_size > 256 || P.cgrid_size > 256) FAIL(TMC2_ERR_UNSUPPORTED, "grid sizes above 256");
    if (P.geometry_smoothing) {
      if (P.grid_size < 1) FAIL(TMC2_ERR_INVALID_ARG, "grid_size");
      if ((maxs + P.grid_size - 1) / P.grid_size > 1024) FAIL(TMC2_ERR_UNSUPPORTED, "geometry grid wider than 1024 cells");
    }
    if (P.color_smoothing && P.attribute_count) {
      if (P.cgrid_size < 1) FAIL(TMC2_ERR_INVALID_ARG, "cgrid_size");
      if ((maxs + P.cgrid_size - 1) / P.cgrid_size > 1024) FAIL(TMC2_ERR_UNSUPPORTED, "colour grid wider than 1024 cells");
    }
  }
  if (g->input_flags & ~(TMC2_INPUT_DEVICE | TMC2_INPUT_P010))
    FAIL(TMC2_ERR_INVALID_ARG, "input_flags 0x%x: unknown bits", g->input_flags);
  if ((g->input_flags & TMC2_INPUT_P010) && !(g->input_flags & TMC2_INPUT_DEVICE))
    FAIL(TMC2_ERR_UNSUPPORTED, "TMC2_INPUT_P010 is only accepted with TMC2_INPUT_DEVICE (host P010 planes are not supported)");
  return TMC2_OK;
}

// Device planes (TMC2_INPUT_DEVICE): the allocations they were found in, with their devices.  A plane inside an allocation
// already seen costs no driver call (a GOF held in one tensor is checked with one query per plane kind).
struct DevRange { uintptr_t base; size_t size; int device; };

static tmc2_status check_device_plane(const void* p, uint32_t rows, size_t pitch_bytes, size_t row_bytes, const std::vector<int>& devices,
                                      std::vector<DevRange>& ranges, uint32_t f, const char* what, Err& err) {
  const uintptr_t a = (uintptr_t)p;
  const size_t extent = (size_t)(rows - 1) * pitch_bytes + row_bytes;
  for (const DevRange& r : ranges)
    if (a >= r.base && a - r.base < r.size) {
      if (extent > r.size - (a - r.base))
        FAIL(TMC2_ERR_INVALID_ARG, "frame %u: %s plane (%zu bytes from its start) runs past the end of its allocation", f, what, extent);
      return TMC2_OK;
    }
  cudaPointerAttributes at{};
  if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
    cudaGetLastError();
    FAIL(TMC2_ERR_INVALID_ARG, "frame %u: %s plane is not CUDA device memory (TMC2_INPUT_DEVICE)", f, what);
  }
  if (at.type != cudaMemoryTypeDevice && at.type != cudaMemoryTypeManaged)
    FAIL(TMC2_ERR_INVALID_ARG, "frame %u: %s plane is host memory, TMC2_INPUT_DEVICE wants device memory", f, what);
  if (std::find(devices.begin(), devices.end(), at.device) == devices.end())
    FAIL(TMC2_ERR_INVALID_ARG, "frame %u: %s plane is on device %d, which is not a device of the context", f, what, at.device);
  AddressRangeFn fn = address_range_fn();
  if (!fn) FAIL(TMC2_ERR_CUDA, "cuMemGetAddressRange is not available from the driver");
  int cur = 0;
  if (cudaGetDevice(&cur) != cudaSuccess || cudaSetDevice(at.device) != cudaSuccess) {
    cudaGetLastError();
    FAIL(TMC2_ERR_CUDA, "cudaSetDevice(%d) failed while checking a device plane", at.device);
  }
  CUdeviceptr base = 0;
  size_t size = 0;
  const CUresult cr = fn(&base, &size, (CUdeviceptr)a);
  cudaSetDevice(cur);
  if (cr != CUDA_SUCCESS) FAIL(TMC2_ERR_INVALID_ARG, "frame %u: %s plane: no device allocation holds it (CUresult %d)", f, what, (int)cr);
  ranges.push_back({(uintptr_t)base, size, at.device});
  if (extent > size - (a - (uintptr_t)base))
    FAIL(TMC2_ERR_INVALID_ARG, "frame %u: %s plane (%zu bytes from its start) runs past the end of its allocation", f, what, extent);
  return TMC2_OK;
}

// `devices` / `ranges`: the context's devices and the allocations of the GOF's device planes seen so far (TMC2_INPUT_DEVICE)
static tmc2_status validate_frame(const tmc2_gof* g, uint32_t f, const std::vector<int>& devices, std::vector<DevRange>& ranges,
                                  Err& err) {
  const tmc2_params& P = g->params;
  const tmc2_frame& fr = g->frames[f];
  const bool p010 = (g->input_flags & TMC2_INPUT_P010) != 0;
  // codec.rs:318-320: geometry video must hold frames f*M .. f*M+M-1
  if ((uint64_t)g->geo_video_frames < (uint64_t)f * 2 + 2)
    FAIL(TMC2_ERR_SHORT_VIDEO, "geometry video has %u frames, frame %u needs %llu (codec.rs:318)", g->geo_video_frames, f,
         (unsigned long long)f * 2 + 2);
  if (P.attribute_count && (uint64_t)g->attr_video_frames < (uint64_t)f * 2 + 2)
    FAIL(TMC2_ERR_SHORT_VIDEO, "attribute video has %u frames, frame %u needs %llu (codec.rs:589,637)",
         g->attr_video_frames, f, (unsigned long long)f * 2 + 2);
  if (!fr.occ || !fr.geo[0] || !fr.geo[1]) FAIL(TMC2_ERR_INVALID_ARG, "frame %u: NULL occupancy / geometry plane", f);
  if (P.attribute_count && (!fr.attr_y[0] || !fr.attr_y[1] || !fr.attr_u[0] || !fr.attr_u[1] ||
                            (!p010 && (!fr.attr_v[0] || !fr.attr_v[1]))))
    FAIL(TMC2_ERR_INVALID_ARG, "frame %u: NULL attribute plane", f);
  if (P.attribute_count && p010 && (fr.attr_v[0] || fr.attr_v[1]))
    FAIL(TMC2_ERR_INVALID_ARG, "frame %u: attr_v must be NULL with TMC2_INPUT_P010 (attr_u is the interleaved UV plane)", f);
  // P010: attr_u rows hold width/2 interleaved (U, V) pairs = width elements
  if (fr.occ_stride < g->occ_width || fr.geo_stride < g->width ||
      (P.attribute_count && (fr.attr_stride_y < g->width || fr.attr_stride_c < (p010 ? g->width : g->width / 2))))
    FAIL(TMC2_ERR_INVALID_ARG, "frame %u: stride smaller than width", f);
  if (fr.patch_count && !fr.patches) FAIL(TMC2_ERR_INVALID_ARG, "frame %u: NULL patch list", f);
  if (fr.patch_count > 65535) FAIL(TMC2_ERR_CAPACITY, "frame %u: more than 65535 patches", f);
  const int64_t res = P.occupancy_resolution;
  const int64_t sscale = P.orientation_mode == TMC2_ORIENTATION_SPEC ? res : 1;
  const int64_t bw = g->width / res, bh = g->height / res;
  for (uint32_t i = 0; i < fr.patch_count; ++i) {
    const tmc2_patch& p = fr.patches[i];
    if (p.patch_orientation > 8) FAIL(TMC2_ERR_INVALID_ARG, "frame %u patch %u: orientation %u", f, i, p.patch_orientation);
    if (p.normal_axis > 2 || p.tangent_axis > 2 || p.bitangent_axis > 2 || p.projection_mode > 1)
      FAIL(TMC2_ERR_INVALID_ARG, "frame %u patch %u: axes / projection mode out of range", f, i);
    // set_axis (decoder.rs:788-821) only ever produces a permutation of (0, 1, 2).  With coinciding axes the reference's
    // duplicate test (codec.rs:425 compares the final points, after a later axis store has overwritten an earlier one) and
    // its differential D1 (codec.rs:551-558 moves point[normal] after all three stores) act on the overwritten coordinate;
    // the kernels compare / move the normal coordinate itself, so such patches are refused instead of silently differing
    if (p.normal_axis == p.tangent_axis || p.normal_axis == p.bitangent_axis || p.tangent_axis == p.bitangent_axis)
      FAIL(TMC2_ERR_UNSUPPORTED, "frame %u patch %u: normal / tangent / bitangent axes are not a permutation (decoder.rs:788-821)", f, i);
    if (p.axis_of_additional_plane != 0)
      FAIL(TMC2_ERR_UNSUPPORTED, "frame %u patch %u: axis_of_additional_plane (codec.rs:437)", f, i);
    if (p.size_u0 == 0 || p.size_v0 == 0) continue;
    if (p.size_u0 > 4096 || p.size_v0 > 4096) FAIL(TMC2_ERR_PATCH_OUT_OF_CANVAS, "frame %u patch %u: size", f, i);
    for (int c = 0; c < 4; ++c) {
      int64_t x, y;
      const int64_t ub = (c & 1) ? p.size_u0 - 1 : 0, vb = (c & 2) ? p.size_v0 - 1 : 0;
      helper_i64(p, ub, vb, 1, 1, x, y);                         // decoder.rs:834-835
      if (x < 0 || y < 0 || x >= bw || y >= bh)
        FAIL(TMC2_ERR_PATCH_OUT_OF_CANVAS, "frame %u patch %u: block (%lld,%lld) outside %lldx%lld (decoder.rs:835)", f, i,
             (long long)x, (long long)y, (long long)bw, (long long)bh);
      const int64_t u = (c & 1) ? (int64_t)p.size_u0 * res - 1 : 0, v = (c & 2) ? (int64_t)p.size_v0 * res - 1 : 0;
      helper_i64(p, u, v, res, sscale, x, y);                    // decoder.rs:847-848
      if (x < 0 || y < 0 || x >= (int64_t)g->width || y >= (int64_t)g->height)
        FAIL(TMC2_ERR_PATCH_OUT_OF_CANVAS, "frame %u patch %u: pixel (%lld,%lld) outside the canvas (decoder.rs:848)", f, i,
             (long long)x, (long long)y);
    }
  }
  if (g->input_flags & TMC2_INPUT_DEVICE) {
    if (check_device_plane(fr.occ, g->occ_height, fr.occ_stride, g->occ_width, devices, ranges, f, "occupancy", err)) return err.st;
    for (int m = 0; m < 2; ++m)
      if (check_device_plane(fr.geo[m], g->height, (size_t)fr.geo_stride * 2, (size_t)g->width * 2, devices, ranges, f, "geometry", err))
        return err.st;
    if (P.attribute_count) {
      const uint32_t hc = g->height / 2;
      for (int m = 0; m < 2; ++m) {
        if (check_device_plane(fr.attr_y[m], g->height, (size_t)fr.attr_stride_y * 2, (size_t)g->width * 2, devices, ranges, f,
                               "attribute Y", err)) return err.st;
        if (check_device_plane(fr.attr_u[m], hc, (size_t)fr.attr_stride_c * 2, (size_t)(p010 ? g->width : g->width / 2) * 2, devices,
                               ranges, f, p010 ? "attribute UV" : "attribute U", err)) return err.st;
        if (!p010 && check_device_plane(fr.attr_v[m], hc, (size_t)fr.attr_stride_c * 2, (size_t)(g->width / 2) * 2, devices, ranges, f,
                                        "attribute V", err)) return err.st;
      }
    }
  }
  return TMC2_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// Batch: the frames of one GOF (or GOF slice) on one device
// ---------------------------------------------------------------------------------------------------------------
enum : uint32_t {
  WANT_DEBUG = 1u,       // partition, point_to_pixel, colors16bit, boundary type, pre-smoothing copies
  WANT_OCC_FULL = 2u,    // materialise tile.occupancy_map (K1)
};

struct StageTimes { float b2p = 0, count = 0, unpack = 0, geo = 0, col = 0, rgb = 0; };

struct Batch {
  int device = 0;
  cudaStream_t stream = nullptr;      // compute + H2D
  cudaStream_t d2h_stream = nullptr;  // result copies
  cudaStream_t aux_stream = nullptr;  // smoothing post-passes of group g overlap the emit of group g+1
  std::vector<cudaEvent_t> ev_emit, ev_post;   // per group: emit done (main stream) / filter+clear done (aux)
  cudaEvent_t ev_tables_clean = nullptr;       // single-group launches: the clear pass runs on aux, off the critical path
  bool clear_pending = false;
  bool two_pass = false;

  // description of the loaded GOF slice
  uint32_t W = 0, H = 0, occ_w = 0, occ_h = 0, F = 0, res = 16, prec = 4;
  uint32_t geo_pitch = 0, attr_pitch_y = 0, attr_pitch_c = 0, occ_pitch = 0, Hc = 0;
  tmc2_params params{};
  uint32_t want = 0;
  uint64_t cap = 0;                   // points per frame slab
  uint32_t n_tiles = 0, n_slots = 0, bw = 0, bh = 0;
  bool smoothing_geo = false, smoothing_col = false;

  std::vector<DevPatch> h_patches;
  std::vector<SlotRec> h_slot_rec;
  std::vector<uint32_t> h_tile_frame, h_ftb;

  DevBuf d_occ, d_geo, d_ay, d_au, d_av, d_meta, d_b2p, d_count, d_err, d_work, d_owned_count, d_slot_bt, d_slot_bbase, d_slot_nmin;
  DevBuf d_pos, d_rgb, d_yuv, d_part, d_pix, d_bt, d_occ_full, d_pos_pre, d_yuv_pre;
  DevBuf d_geotab, d_coltab, d_geokeys, d_colkeys, d_changed, d_blist,
      d_blist_count, d_slist, d_slist_count, d_geombits, d_colmbits, d_geotbits, d_coltbits;
  uint64_t geotab_slots = 0, coltab_slots = 0, geotab_frames = 0, coltab_frames = 0, blist_cap = 0;
  uint64_t table_budget = 0;          // bytes per cell table, decided when the batch first needs tables
  bool geotab_hashed = false, coltab_hashed = false;
  uint32_t group_frames = 32;         // frames per smoothing group (one group = no post-pass tails between groups; a GOF is <= 32 frames)
  uint32_t group_frames_eff = 8;      // after fitting the dense tables into the memory budget
  std::vector<cudaEvent_t> ev_grp;    // 2 per group: around the unpack launch
  PinBuf h_in, h_meta, h_small, h_out, h_ply;
  DevBuf d_ply, d_ply_sums;           // tmc2gpu_frame_to_ply: body scratch, block sums + offsets + total
  size_t meta_patch_off = 0, meta_slot_off = 0, meta_tf_off = 0, meta_ftb_off = 0, meta_ingest_off = 0, meta_bytes = 0;
  uint32_t input_flags = 0;           // tmc2_gof.input_flags of the loaded GOF
  uint32_t n_ingest = 0;              // device planes: entries of the ingest table (end of the metadata block)
  uint32_t ingest_launches = 0;       // ingest kernel launched by upload(), counted with the next launch()

  cudaEvent_t ev[8] = {};             // stage boundaries: 0 start,1 after b2p,2 after unpack,3 geo,4 col,5 rgb
  cudaEvent_t ev_counts = nullptr, ev_inputs_free = nullptr;
  std::vector<cudaEvent_t> ev_frame;  // per-frame D2H completion

  // results on the host after fetch
  std::vector<uint32_t> counts;
  std::vector<uint64_t> moved, recoloured;
  std::vector<size_t> out_pos_off, out_rgb_off;
  bool counts_ready = false, outputs_enqueued = false, counts_enqueued = false;
  uint32_t launches = 0, n_groups = 1;
  uint64_t unpack_alg_bytes = 0;
  uint32_t frames_released = 0;
  bool busy = false;
  std::chrono::steady_clock::time_point t_submit;   // TMC2_TRACE bookkeeping
  uint64_t t_epoch = 0;                             // submit call that made this batch busy
  Err failed_early;                                 // a failure found while this batch was not yet at the head of the queue
  cudaGraphExec_t graph_exec = nullptr;             // resident relaunches without smoothing: the whole launch sequence as one graph
  bool graph_tried = false;
  double trace_wait_ms = 0;

  ~Batch() { destroy(); }
  void destroy() {
    cudaSetDevice(device);
    for (DevBuf* b : {&d_occ, &d_geo, &d_ay, &d_au, &d_av, &d_meta, &d_b2p, &d_count, &d_err, &d_work,
                      &d_owned_count, &d_slot_bt, &d_slot_bbase, &d_slot_nmin, &d_pos,
                      &d_rgb, &d_yuv, &d_part, &d_pix, &d_bt, &d_occ_full, &d_pos_pre, &d_yuv_pre, &d_geotab, &d_coltab,
                      &d_geokeys, &d_colkeys, &d_changed, &d_blist,
                      &d_blist_count, &d_slist, &d_slist_count, &d_geombits, &d_colmbits, &d_geotbits, &d_coltbits, &d_ply, &d_ply_sums})
      b->release();
    for (PinBuf* b : {&h_in, &h_meta, &h_small, &h_out, &h_ply}) b->release();
    for (auto& e : ev) if (e) { cudaEventDestroy(e); e = nullptr; }
    if (ev_counts) cudaEventDestroy(ev_counts), ev_counts = nullptr;
    if (ev_inputs_free) cudaEventDestroy(ev_inputs_free), ev_inputs_free = nullptr;
    for (auto e : ev_frame) cudaEventDestroy(e);
    ev_frame.clear();
    for (auto e : ev_grp) cudaEventDestroy(e);
    ev_grp.clear();
    for (auto e : ev_emit) cudaEventDestroy(e);
    ev_emit.clear();
    for (auto e : ev_post) cudaEventDestroy(e);
    ev_post.clear();
    if (graph_exec) cudaGraphExecDestroy(graph_exec), graph_exec = nullptr;
    if (aux_stream) cudaStreamDestroy(aux_stream), aux_stream = nullptr;
    if (ev_tables_clean) cudaEventDestroy(ev_tables_clean), ev_tables_clean = nullptr;
    if (stream) cudaStreamDestroy(stream), stream = nullptr;
    if (d2h_stream) cudaStreamDestroy(d2h_stream), d2h_stream = nullptr;
  }

  tmc2_status init(int dev, bool two_pass_scan, Err& err) {
    device = dev; two_pass = two_pass_scan;
    CU(cudaSetDevice(device));
    CU(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&d2h_stream, cudaStreamNonBlocking));
    {
      // the auxiliary stream only runs small clean-up kernels under the next launch: let them jump the queue
      int lo = 0, hi = 0;
      CU(cudaDeviceGetStreamPriorityRange(&lo, &hi));
      CU(cudaStreamCreateWithPriority(&aux_stream, cudaStreamNonBlocking, hi));
    }
    CU(cudaEventCreateWithFlags(&ev_tables_clean, cudaEventDisableTiming));
    for (auto& e : ev) CU(cudaEventCreate(&e));
    CU(cudaEventCreateWithFlags(&ev_counts, cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&ev_inputs_free, cudaEventDisableTiming));
    CU(d_err.ensure(sizeof(int)));
    CU(cudaMemset(d_err.p, 0, sizeof(int)));
    return TMC2_OK;
  }

  // ---- host-side digest of the patch lists: DevPatch array, slot list, tile -> frame map ------------------------
  tmc2_status prepare(const tmc2_gof* g, uint32_t first, uint32_t count, uint32_t want_flags, Err& err) {
    CU(cudaSetDevice(device));
    params = g->params;
    W = g->width; H = g->height; occ_w = g->occ_width; occ_h = g->occ_height; F = count;
    res = params.occupancy_resolution; prec = params.occupancy_precision;
    bw = W / res; bh = H / res;
    want = want_flags;
    input_flags = g->input_flags;
    Hc = H / 2;
    geo_pitch = round_up(W, 64); attr_pitch_y = round_up(W, 64); attr_pitch_c = round_up(std::max(W / 2, 1u), 64);
    occ_pitch = round_up(occ_w, 16);
    cap = round_up64(2ull * W * H, 16);   // slabs stay 16-byte aligned for both output streams
    smoothing_geo = params.geometry_smoothing != 0;
    smoothing_col = params.color_smoothing != 0 && params.attribute_count != 0;

    h_patches.clear(); h_slot_rec.clear(); h_tile_frame.clear(); h_ftb.assign(1, 0);
    uint64_t total_points_bound = 0;
    for (uint32_t k = 0; k < count; ++k) {
      const tmc2_frame& fr = g->frames[first + k];
      for (uint32_t i = 0; i < fr.patch_count; ++i) {
        const tmc2_patch& p = fr.patches[i];
        DevPatch d{};
        d.u0 = p.u0; d.v0 = p.v0; d.size_u0 = p.size_u0; d.size_v0 = p.size_v0;
        d.u1 = p.u1; d.v1 = p.v1; d.d1 = p.d1; d.lod_x = p.lod_x; d.lod_y = p.lod_y;
        d.normal = p.normal_axis; d.tangent = p.tangent_axis; d.bitangent = p.bitangent_axis; d.mode = p.projection_mode;
        d.orient = p.patch_orientation;
        d.sel = position_selectors(p.normal_axis, p.tangent_axis, p.bitangent_axis);
        {
          // block-aligned affine form of decoder.rs:853-867: canvas step per +1 in patch u (ax, ay) and per +1 in v (rx, ry)
          static const int8_t kAx[9] = {1, 0, 0, -1, 0, -1, 0, 1, 0}, kAy[9] = {0, 1, 1, 0, -1, 0, -1, 0, 1};
          static const int8_t kRx[9] = {0, 1, -1, 0, 1, 0, -1, 0, 1}, kRy[9] = {1, 0, 0, -1, 0, 1, 0, -1, 0};
          const uint32_t o = p.patch_orientation;
          d.ax = kAx[o]; d.ay = kAy[o]; d.rx = kRx[o]; d.ry = kRy[o];
          d.aligned = (params.orientation_mode == TMC2_ORIENTATION_SPEC || o <= 1 || o == 8) ? 1 : 0;
        }
        d.slot_base = (uint32_t)h_slot_rec.size();
        d.local_index = i; d.frame = k;
        const uint64_t ns = (uint64_t)p.size_u0 * p.size_v0;
        if (h_slot_rec.size() + ns > (1ull << 30)) FAIL(TMC2_ERR_CAPACITY, "too many patch blocks in one GOF");
        const uint32_t pid = (uint32_t)h_patches.size();
        h_patches.push_back(d);
        for (uint32_t v0b = 0; v0b < p.size_v0; ++v0b)
          for (uint32_t u0b = 0; u0b < p.size_u0; ++u0b) {       // the reference's block order, codec.rs:371-372
            int64_t bx, by;
            helper_i64(p, u0b, v0b, 1, 1, bx, by);               // decoder.rs:827-837 (validated to be inside the grid)
            SlotRec r{};
            r.pid = pid; r.u0b = (uint16_t)u0b; r.v0b = (uint16_t)v0b; r.bx = (uint16_t)bx; r.by = (uint16_t)by;
            r.ax = d.ax; r.ay = d.ay; r.rx = d.rx; r.ry = d.ry;
            if (!d.aligned) { r.ax = r.ay = r.rx = r.ry = 0; }   // reference-literal rotated patch: generic device path
            h_slot_rec.push_back(r);
          }
        total_points_bound += ns * res * res * 2;
      }
      // pad the frame's slot list to whole tiles: a tile never straddles two frames (one scan domain per frame)
      while (h_slot_rec.size() % kWarpsPerTile) { SlotRec r{}; r.pid = kNoPatch; h_slot_rec.push_back(r); }
      const uint32_t tiles_now = (uint32_t)(h_slot_rec.size() / kWarpsPerTile);
      h_tile_frame.resize(tiles_now, k);
      h_ftb.push_back(tiles_now);
    }
    n_slots = (uint32_t)h_slot_rec.size();
    n_tiles = n_slots / kWarpsPerTile;
    (void)total_points_bound;

    // device buffers
    const bool attr = params.attribute_count != 0;
    CU(d_occ.ensure((size_t)F * occ_h * occ_pitch));
    CU(d_geo.ensure((size_t)F * 2 * H * geo_pitch * 2));
    if (attr) {
      CU(d_ay.ensure((size_t)F * 2 * H * attr_pitch_y * 2));
      CU(d_au.ensure((size_t)F * 2 * std::max(Hc, 1u) * attr_pitch_c * 2));
      CU(d_av.ensure((size_t)F * 2 * std::max(Hc, 1u) * attr_pitch_c * 2));
    }
    meta_patch_off = 0;
    meta_slot_off = round_up64(h_patches.size() * sizeof(DevPatch), 256);
    meta_tf_off = meta_slot_off + round_up64((uint64_t)n_slots * sizeof(SlotRec), 256);
    meta_ftb_off = meta_tf_off + round_up64((uint64_t)n_tiles * 4, 256);
    meta_ingest_off = meta_ftb_off + round_up64((uint64_t)(F + 1) * 4, 256);
    // one table entry per (frame, kind, map): occupancy, 2 geometry, 2 luma, 2 UV (P010) or 2 U + 2 V
    n_ingest = (input_flags & TMC2_INPUT_DEVICE) ? F * (3 + (attr ? ((input_flags & TMC2_INPUT_P010) ? 4 : 6) : 0)) : 0;
    meta_bytes = meta_ingest_off + (size_t)n_ingest * sizeof(IngestPlane);
    CU(d_meta.ensure(meta_bytes));
    CU(h_meta.ensure(meta_bytes));
    CU(d_b2p.ensure(std::max<size_t>((size_t)F * bw * bh * 4, 4)));
    CU(d_count.ensure(std::max<size_t>((size_t)F * 4, 4)));
    CU(d_work.ensure(std::max<size_t>((size_t)n_slots * sizeof(WorkRec), sizeof(WorkRec))));
    CU(d_owned_count.ensure(std::max<size_t>((size_t)F * 4, 4)));
    if (smoothing_geo || smoothing_col || (want_flags & WANT_DEBUG)) {       // boundary classes per slot (count pass -> emit pass)
      CU(d_slot_bt.ensure(std::max<size_t>((size_t)n_slots * 64, 64)));
      CU(d_slot_bbase.ensure(std::max<size_t>((size_t)n_slots * 4, 4)));
      CU(d_slot_nmin.ensure(std::max<size_t>((size_t)n_slots * 2, 2)));
    }
    CU(d_changed.ensure(std::max<size_t>((size_t)F * 16, 16)));
    CU(d_pos.ensure((size_t)F * cap * 6));
    const bool dbg = (want & WANT_DEBUG) != 0;
    if (attr) CU(d_rgb.ensure((size_t)F * cap * 3));
    if (dbg) {
      if (attr) CU(d_yuv.ensure((size_t)F * cap * 6));
      CU(d_part.ensure((size_t)F * cap * 2));
      CU(d_bt.ensure((size_t)F * cap));
      CU(d_pix.ensure((size_t)F * cap * 4));
      CU(d_pos_pre.ensure((size_t)F * cap * 6));
      if (attr) CU(d_yuv_pre.ensure((size_t)F * cap * 6));
    }
    if (want & WANT_OCC_FULL) CU(d_occ_full.ensure((size_t)F * W * H));
    if (smoothing_geo || smoothing_col) {
      if (const char* e = getenv("TMC2_SMOOTH_GROUP")) group_frames = std::max(1, atoi(e));
      const uint32_t maxs = 1u << params.geometry_bitdepth_3d;
      // boundary-point lists (one per frame) and their counters
      if (blist_cap != cap || d_blist.cap < (size_t)F * cap * sizeof(BoundaryEntry)) {
        CU(d_blist.ensure((size_t)F * cap * sizeof(BoundaryEntry)));
        CU(d_slist.ensure((size_t)F * cap * 4));
        blist_cap = cap;
      }
      CU(d_blist_count.ensure(std::max<size_t>((size_t)F * 4, 4)));
      CU(d_slist_count.ensure(std::max<size_t>((size_t)F * 4, 4)));
      // Cell tables: dense (direct-indexed, no probing) when the whole grid fits the per-table budget for at least one
      // frame, hashed (separate key array) otherwise.  The group size shrinks until the dense tables fit.
      // Budget per table: 40 GB, less when the device is short of memory (a quarter of what is free now, so that the GOFs in
      // flight after this one still find room; at least 1 GB) -- smaller budgets mean smaller frame groups, then hashed tables.
      // Decided once per batch (the tables are kept from GOF to GOF).
      if (table_budget == 0) {
        table_budget = 40ull << 30;
        size_t free_b = 0, total_b = 0;
        if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess)
          table_budget = std::min<uint64_t>(table_budget, std::max<uint64_t>(1ull << 30, (uint64_t)free_b / 4));
        else
          cudaGetLastError();
        if (const char* e = getenv("TMC2_TABLE_BUDGET_MB")) table_budget = std::max<uint64_t>(1, strtoull(e, nullptr, 10)) << 20;
      }
      const uint64_t kTableBudget = table_budget;
      const bool force_hash = getenv("TMC2_FORCE_HASH") != nullptr;        // test hook for the hashed-table path
      auto cells_of = [&](uint32_t g) -> uint64_t { const uint64_t w = (maxs + g - 1) / g; return w * w * w; };
      uint32_t GF = std::min(group_frames, std::max(F, 1u));
      auto fit = [&](bool on, uint32_t g, size_t cell_bytes, uint32_t sets) {
        if (!on || force_hash) return;
        const uint64_t per_frame = cells_of(g) * cell_bytes;
        if (per_frame <= kTableBudget) GF = (uint32_t)std::min<uint64_t>(GF, std::max<uint64_t>(1, kTableBudget / (sets * per_frame)));
      };
      // one table set when the whole batch is a single group, else two alternating sets (post-passes of a group overlap the
      // next group's emit)
      fit(smoothing_geo, params.grid_size, sizeof(GeoCell), 1);
      fit(smoothing_col, params.cgrid_size, sizeof(ColCell), 1);
      uint32_t n_sets = 1;
      if (GF < F) {
        GF = std::min(group_frames, std::max(F, 1u));
        fit(smoothing_geo, params.grid_size, sizeof(GeoCell), 2);
        fit(smoothing_col, params.cgrid_size, sizeof(ColCell), 2);
        n_sets = 2;
      }
      group_frames_eff = GF;
      const uint64_t TF = (uint64_t)n_sets * GF;                              // table frames to hold
      auto table_slots = [&](uint32_t g, size_t cell_bytes, bool& hashed) -> uint64_t {
        const uint64_t cells = cells_of(g);
        hashed = force_hash || cells * cell_bytes > kTableBudget;
        return hashed ? pow2_at_least(2 * cap) : cells;
      };
      auto setup = [&](bool on, uint32_t g, size_t cell_bytes, DevBuf& tab, DevBuf& keys, DevBuf& mbits, DevBuf& tbits, uint64_t& slots_now,
                       uint64_t& frames_now, bool& hashed_now) -> tmc2_status {
        if (!on) return TMC2_OK;
        bool hashed = false;
        const uint64_t slots = table_slots(g, cell_bytes, hashed);
        if (slots != slots_now || TF > frames_now || hashed != hashed_now) {
          CU(tab.ensure((size_t)TF * slots * cell_bytes));
          CU(cudaMemsetAsync(tab.p, 0, (size_t)TF * slots * cell_bytes, stream));     // all-zero == empty cell
          CU(mbits.ensure((size_t)TF * ((slots + 31) / 32) * 4));
          CU(cudaMemsetAsync(mbits.p, 0, (size_t)TF * ((slots + 31) / 32) * 4, stream));
          CU(tbits.ensure((size_t)TF * ((slots + (32u << kTouchShift) - 1) / (32u << kTouchShift)) * 4));
          CU(cudaMemsetAsync(tbits.p, 0, (size_t)TF * ((slots + (32u << kTouchShift) - 1) / (32u << kTouchShift)) * 4, stream));
          if (hashed) {
            CU(keys.ensure((size_t)TF * slots * 4));
            KL(launch_fill_u32(keys.as<uint32_t>(), (uint64_t)TF * slots, kCellEmpty, stream));
          }
          slots_now = slots; frames_now = TF; hashed_now = hashed;
        }
        return TMC2_OK;
      };
      if (setup(smoothing_geo, params.grid_size, sizeof(GeoCell), d_geotab, d_geokeys, d_geombits, d_geotbits, geotab_slots, geotab_frames, geotab_hashed)) return err.st;
      if (setup(smoothing_col, params.cgrid_size, sizeof(ColCell), d_coltab, d_colkeys, d_colmbits, d_coltbits, coltab_slots, coltab_frames, coltab_hashed)) return err.st;
    }
    return make_tile_maps(err);
  }

  // ---- H2D: planes (through pinned staging unless the caller's memory is already pinned) + metadata -------------
  // One row-pitched copy per (frame, map), merged when neighbouring planes are contiguous on both sides.  Whether a plane is
  // DMA'd in place or staged is decided ONCE per plane, on its full extent, and the staging area is sized from exactly
  // those decisions.
  struct Seg {
    const uint8_t* src; size_t spitch; uint8_t* dst; uint32_t rows;
    size_t row_bytes, dpb, plane_dev;      // bytes per row, device pitch in bytes, bytes of the plane on the device
    bool staged; size_t stage_off;
    int kind;                              // runs are only merged inside one device allocation (= one plane kind)
  };
  void plan_plane_set(const tmc2_gof* g, uint32_t first, int kind, const std::vector<std::pair<const uint8_t*, size_t>>& reg,
                      std::vector<Seg>& segs, size_t& stage_bytes) const {
    // kind: 0 occ, 1 geo, 2 attr_y, 3 attr_u, 4 attr_v
    const int maps = kind == 0 ? 1 : 2;
    const uint32_t esz = kind == 0 ? 1 : 2;
    const uint32_t w = kind == 0 ? occ_w : (kind >= 3 ? W / 2 : W);
    const uint32_t h = kind == 0 ? occ_h : (kind >= 3 ? Hc : H);
    const uint32_t dpitch = kind == 0 ? occ_pitch : kind == 1 ? geo_pitch : kind == 2 ? attr_pitch_y : attr_pitch_c;
    uint8_t* dbase = kind == 0 ? d_occ.as<uint8_t>() : kind == 1 ? d_geo.as<uint8_t>() : kind == 2 ? d_ay.as<uint8_t>()
                   : kind == 3 ? d_au.as<uint8_t>() : d_av.as<uint8_t>();
    if (w == 0 || h == 0) return;
    const size_t plane_dev = (size_t)h * dpitch * esz;
    for (uint32_t k = 0; k < F; ++k) {
      const tmc2_frame& fr = g->frames[first + k];
      for (int m = 0; m < maps; ++m) {
        const void* src = kind == 0 ? (const void*)fr.occ : kind == 1 ? (const void*)fr.geo[m]
                        : kind == 2 ? (const void*)fr.attr_y[m] : kind == 3 ? (const void*)fr.attr_u[m] : (const void*)fr.attr_v[m];
        const uint32_t sstride = kind == 0 ? fr.occ_stride : kind == 1 ? fr.geo_stride : kind == 2 ? fr.attr_stride_y : fr.attr_stride_c;
        Seg s{(const uint8_t*)src, (size_t)sstride * esz, dbase + ((size_t)k * maps + m) * plane_dev, h,
              (size_t)w * esz, (size_t)dpitch * esz, plane_dev, false, 0, kind};
        const size_t src_bytes = (size_t)(s.rows - 1) * s.spitch + s.row_bytes;
        s.staged = !is_pinned(reg, s.src, src_bytes);
        if (s.staged) { s.stage_off = stage_bytes; stage_bytes += plane_dev; }
        segs.push_back(s);
      }
    }
  }

  // dev_ranges: allocations of the GOF's device planes (validate_frame), for TMC2_INPUT_DEVICE
  tmc2_status upload(const tmc2_gof* g, uint32_t first, const std::vector<DevRange>& dev_ranges, Err& err, bool use_pool = true) {
    CU(cudaSetDevice(device));
    if (input_flags & TMC2_INPUT_DEVICE) return upload_device(g, first, dev_ranges, err);
    const bool attr = params.attribute_count != 0;
    std::vector<Seg> segs;
    size_t stage_bytes = 0;
    {
      const auto reg = pinned_snapshot();
      for (int kind = 0; kind < (attr ? 5 : 2); ++kind) plan_plane_set(g, first, kind, reg, segs, stage_bytes);
    }
    // the previous GOF of this batch must have finished its H2D copies before its staging area (planes and metadata) is
    // written again
    CU(cudaEventSynchronize(ev_inputs_free));
    if (stage_bytes) CU(h_in.ensure(stage_bytes));
    // current run of planes that are contiguous on both sides -> one cudaMemcpyAsync
    const uint8_t* run_src = nullptr; uint8_t* run_dst = nullptr; size_t run_bytes = 0; int run_kind = -1;
    auto flush = [&]() -> cudaError_t {
      cudaError_t e = cudaSuccess;
      if (run_bytes) e = cudaMemcpyAsync(run_dst, run_src, run_bytes, cudaMemcpyHostToDevice, stream);
      run_bytes = 0;
      return e;
    };
    auto enqueue = [&](const Seg& s) -> tmc2_status {
      const uint8_t* src = s.staged ? h_in.as<uint8_t>() + s.stage_off : s.src;
      const size_t spitch = s.staged ? s.dpb : s.spitch;
      // in-place planes: the last row of a plane may be shorter than the pitch in the SOURCE allocation -- never read past it
      if (spitch == s.dpb && (s.staged || s.row_bytes == s.dpb)) {
        if (run_bytes && s.kind == run_kind && src == run_src + run_bytes && s.dst == run_dst + run_bytes) {
          run_bytes += s.plane_dev;
        } else {
          CU(flush());
          run_src = src; run_dst = s.dst; run_bytes = s.plane_dev; run_kind = s.kind;
        }
      } else {
        CU(flush());
        CU(cudaMemcpy2DAsync(s.dst, s.dpb, src, spitch, s.row_bytes, s.rows, cudaMemcpyHostToDevice, stream));
      }
      return TMC2_OK;
    };
    // Staged planes go in groups of ~1/8 of the staging area: the pool repacks a group (row ranges in parallel) into pinned
    // memory with the device pitch, its copies are enqueued, and the DMA of group i runs under the repacking of group i+1.
    const size_t group_bytes = std::max<size_t>(stage_bytes / 8, 4u << 20);
    size_t i = 0;
    while (i < segs.size()) {
      size_t j = i, bytes = 0;
      while (j < segs.size() && (j == i || bytes < group_bytes)) { if (segs[j].staged) bytes += segs[j].plane_dev; ++j; }
      if (bytes) {
        struct Item { const Seg* s; uint32_t r0, r1; };
        std::vector<Item> items;
        for (size_t k = i; k < j; ++k) {
          if (!segs[k].staged) continue;
          const uint32_t rows_per = std::max<uint32_t>(1, (uint32_t)((1u << 20) / std::max<size_t>(segs[k].dpb, 1)));   // ~1 MB pieces
          for (uint32_t r = 0; r < segs[k].rows; r += rows_per) items.push_back({&segs[k], r, std::min(segs[k].rows, r + rows_per)});
        }
        uint8_t* base = h_in.as<uint8_t>();
        auto stage_item = [&](size_t n) {
          const Item& it = items[n];
          const Seg& sg = *it.s;
          uint8_t* st = base + sg.stage_off;
          if (sg.spitch == sg.dpb && sg.row_bytes == sg.dpb) memcpy(st + (size_t)it.r0 * sg.dpb, sg.src + (size_t)it.r0 * sg.spitch, (size_t)(it.r1 - it.r0) * sg.dpb);
          else for (uint32_t r = it.r0; r < it.r1; ++r) memcpy(st + (size_t)r * sg.dpb, sg.src + (size_t)r * sg.spitch, sg.row_bytes);
        };
        if (use_pool) StagePool::get().run(items.size(), stage_item);
        else for (size_t n = 0; n < items.size(); ++n) stage_item(n);     // already on a pool thread (one per device piece)
      }
      for (size_t k = i; k < j; ++k) { tmc2_status st = enqueue(segs[k]); if (st) return st; }
      i = j;
    }
    CU(flush());
    if (send_meta(err)) return err.st;
    CU(cudaEventRecord(ev_inputs_free, stream));
    return TMC2_OK;
  }

  // metadata block (patches, slots, tile -> frame, frame tile ranges; the ingest table is already in place) -> d_meta
  tmc2_status send_meta(Err& err) {
    uint8_t* m = h_meta.as<uint8_t>();
    if (!h_patches.empty()) memcpy(m + meta_patch_off, h_patches.data(), h_patches.size() * sizeof(DevPatch));
    if (n_slots) memcpy(m + meta_slot_off, h_slot_rec.data(), (size_t)n_slots * sizeof(SlotRec));
    if (n_tiles) memcpy(m + meta_tf_off, h_tile_frame.data(), (size_t)n_tiles * 4);
    memcpy(m + meta_ftb_off, h_ftb.data(), (size_t)(F + 1) * 4);
    CU(cudaMemcpyAsync(d_meta.p, m, meta_bytes, cudaMemcpyHostToDevice, stream));
    return TMC2_OK;
  }

  // TMC2_INPUT_DEVICE: no staging and no H2D of planes.  The planes' table goes with the metadata, and one kernel gathers
  // every plane into the batch layout (the same layout the host path produces, so everything downstream is unchanged).
  tmc2_status upload_device(const tmc2_gof* g, uint32_t first, const std::vector<DevRange>& dev_ranges, Err& err) {
    for (const DevRange& r : dev_ranges) {
      if (r.device == device) continue;
      int can = 0;
      CU(cudaDeviceCanAccessPeer(&can, device, r.device));
      if (!can) FAIL(TMC2_ERR_UNSUPPORTED, "device %d cannot read input planes on device %d (no peer access between them)", device, r.device);
      const cudaError_t e = cudaDeviceEnablePeerAccess(r.device, 0);
      if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
      else CU(e);
    }
    // the previous GOF of this batch must have been read (ingest done, metadata copied) before its table is written again
    CU(cudaEventSynchronize(ev_inputs_free));
    const bool attr = params.attribute_count != 0, p010 = (input_flags & TMC2_INPUT_P010) != 0;
    IngestPlane* tab = reinterpret_cast<IngestPlane*>(h_meta.as<uint8_t>() + meta_ingest_off);
    uint32_t n = 0, max_rows = 0, max_row_bytes = 0;
    auto add = [&](const void* src, size_t spitch, uint32_t rows, uint32_t row_bytes, uint8_t* dst, uint8_t* dst2, uint32_t dpitch,
                   uint32_t op) {
      IngestPlane& e = tab[n++];
      e.src = static_cast<const uint8_t*>(src); e.dst = dst; e.dst2 = dst2;
      e.spitch = (uint32_t)spitch; e.dpitch = dpitch; e.rows = rows; e.row_bytes = row_bytes;
      e.op = op | (((uintptr_t)src % 16 == 0 && spitch % 16 == 0) ? (uint32_t)kIngestVec : 0u);
      e._pad = 0;
      max_rows = std::max(max_rows, rows); max_row_bytes = std::max(max_row_bytes, row_bytes);
    };
    const uint32_t op16 = p010 ? kIngestShr16 : kIngestCopy16;
    const size_t occ_plane = (size_t)occ_h * occ_pitch, geo_plane = (size_t)H * geo_pitch * 2, y_plane = (size_t)H * attr_pitch_y * 2;
    const size_t c_plane = (size_t)std::max(Hc, 1u) * attr_pitch_c * 2;
    for (uint32_t k = 0; k < F; ++k) {
      const tmc2_frame& fr = g->frames[first + k];
      add(fr.occ, fr.occ_stride, occ_h, occ_w, d_occ.as<uint8_t>() + k * occ_plane, nullptr, occ_pitch, kIngestCopy8);
      for (uint32_t m = 0; m < 2; ++m) {
        const size_t km = (size_t)k * 2 + m;
        add(fr.geo[m], (size_t)fr.geo_stride * 2, H, W * 2, d_geo.as<uint8_t>() + km * geo_plane, nullptr, geo_pitch * 2, op16);
        if (!attr) continue;
        add(fr.attr_y[m], (size_t)fr.attr_stride_y * 2, H, W * 2, d_ay.as<uint8_t>() + km * y_plane, nullptr, attr_pitch_y * 2, op16);
        if (p010) {
          add(fr.attr_u[m], (size_t)fr.attr_stride_c * 2, Hc, W * 2, d_au.as<uint8_t>() + km * c_plane, d_av.as<uint8_t>() + km * c_plane,
              attr_pitch_c * 2, kIngestUv16);
        } else {
          add(fr.attr_u[m], (size_t)fr.attr_stride_c * 2, Hc, (W / 2) * 2, d_au.as<uint8_t>() + km * c_plane, nullptr, attr_pitch_c * 2, op16);
          add(fr.attr_v[m], (size_t)fr.attr_stride_c * 2, Hc, (W / 2) * 2, d_av.as<uint8_t>() + km * c_plane, nullptr, attr_pitch_c * 2, op16);
        }
      }
    }
    if (n != n_ingest) FAIL(TMC2_ERR_INTERNAL, "ingest table: %u entries, %u expected", n, n_ingest);
    if (send_meta(err)) return err.st;
    KL(launch_ingest_planes(reinterpret_cast<const IngestPlane*>(d_meta.as<uint8_t>() + meta_ingest_off), n, max_rows, max_row_bytes,
                            stream));
    ingest_launches = 1;
    CU(cudaEventRecord(ev_inputs_free, stream));
    return TMC2_OK;
  }

  // TMA descriptors of this batch's plane arrays (rebuilt by prepare(): they hold device addresses and sizes)
  TileMaps tile_maps{};
  tmc2_status make_tile_maps(Err& err) {
    memset(&tile_maps, 0, sizeof tile_maps);
    if (F == 0 || res != 16) return TMC2_OK;                           // no block-aligned slots: the maps are never used
    const uint64_t gms = (uint64_t)H * geo_pitch * 2, yms = (uint64_t)H * attr_pitch_y * 2, cms = (uint64_t)std::max(Hc, 1u) * attr_pitch_c * 2;
    bool ok = true;
    {
      const uint64_t dims[4] = {W, H, 2, F}, st[3] = {(uint64_t)geo_pitch * 2, gms, 2 * gms};
      const uint32_t box[4] = {16, 16, 2, 1};
      ok &= encode_map(tile_maps.geo, d_geo.p, 2, 4, dims, st, box);
    }
    if (params.attribute_count) {
      const uint64_t dims[4] = {W, H, 2, F}, st[3] = {(uint64_t)attr_pitch_y * 2, yms, 2 * yms};
      const uint32_t box[4] = {16, 16, 2, 1};
      ok &= encode_map(tile_maps.attr_y, d_ay.p, 2, 4, dims, st, box);
      const uint64_t cd[4] = {std::max(W / 2, 1u), std::max(Hc, 1u), 2, F}, cs[3] = {(uint64_t)attr_pitch_c * 2, cms, 2 * cms};
      const uint32_t cbox[4] = {8, 8, 2, 1};
      ok &= encode_map(tile_maps.attr_u, d_au.p, 2, 4, cd, cs, cbox);
      ok &= encode_map(tile_maps.attr_v, d_av.p, 2, 4, cd, cs, cbox);
    }
    {
      const uint64_t dims[3] = {occ_w, occ_h, F}, st[2] = {(uint64_t)occ_pitch, (uint64_t)occ_h * occ_pitch};
      const uint32_t box[3] = {32, 8, 1};
      ok &= encode_map(tile_maps.occ, d_occ.p, 1, 3, dims, st, box);
    }
    if (!ok) FAIL(TMC2_ERR_CUDA, "cuTensorMapEncodeTiled failed (TMA descriptors of the plane arrays)");
    return TMC2_OK;
  }

  UnpackArgs make_args() const {
    UnpackArgs a{};
    a.in.occ = d_occ.as<uint8_t>(); a.in.geo = d_geo.as<uint16_t>();
    a.in.attr_y = d_ay.as<uint16_t>(); a.in.attr_u = d_au.as<uint16_t>(); a.in.attr_v = d_av.as<uint16_t>();
    a.in.occ_pitch = occ_pitch; a.in.occ_w = occ_w; a.in.occ_h = occ_h;
    a.in.geo_pitch = geo_pitch; a.in.attr_pitch_y = attr_pitch_y; a.in.attr_pitch_c = attr_pitch_c;
    a.in.occ_frame_stride = (uint64_t)occ_h * occ_pitch;
    a.in.geo_map_stride = (uint64_t)H * geo_pitch;
    a.in.attr_y_map_stride = (uint64_t)H * attr_pitch_y;
    a.in.attr_c_map_stride = (uint64_t)std::max(Hc, 1u) * attr_pitch_c;
    a.W = W; a.H = H; a.res = res; a.prec = prec;
    a.prec_shift = -1;
    for (int s = 0; s < 16; ++s) if ((1u << s) == prec) a.prec_shift = s;
    a.bw = bw; a.bh = bh; a.n_frames = F; a.n_tiles = n_tiles;
    a.absolute_d1 = params.absolute_d1 ? 1 : 0;
    a.spec_orientation = params.orientation_mode == TMC2_ORIENTATION_SPEC ? 1 : 0;
    a.has_attr = params.attribute_count ? 1 : 0;
    const uint8_t* m = d_meta.as<uint8_t>();
    a.patches = reinterpret_cast<const DevPatch*>(m + meta_patch_off);
    a.slot_rec = reinterpret_cast<const SlotRec*>(m + meta_slot_off);
    a.tile_frame = reinterpret_cast<const uint32_t*>(m + meta_tf_off);
    a.frame_tile_begin = reinterpret_cast<const uint32_t*>(m + meta_ftb_off);
    a.block_to_patch = d_b2p.as<uint32_t>();
    a.work = d_work.as<WorkRec>(); a.owned_count = d_owned_count.as<uint32_t>();
    a.slot_bt = d_slot_bt.as<uint16_t>(); a.slot_bbase = d_slot_bbase.as<uint32_t>(); a.slot_nmin = d_slot_nmin.as<uint16_t>();
    a.frame_count = d_count.as<uint32_t>();
    a.err = d_err.as<int>();
    const bool dbg = (want & WANT_DEBUG) != 0;
    const bool smooth = smoothing_geo || smoothing_col;
    a.out.cap = cap;
    a.out.pos = d_pos.as<uint16_t>();
    a.out.rgb = a.has_attr ? d_rgb.as<uint8_t>() : nullptr;     // pre-smoothing colours; the filter patches recoloured points
    a.out.yuv = (a.has_attr && dbg) ? d_yuv.as<uint16_t>() : nullptr;
    a.out.part = dbg ? d_part.as<uint16_t>() : nullptr;
    a.out.btype = dbg ? d_bt.as<uint8_t>() : nullptr;
    a.out.pix = dbg ? d_pix.as<uint32_t>() : nullptr;
    a.want_btype = a.out.btype != nullptr || smooth;
    if (smooth) {
      const uint32_t maxs = 1u << params.geometry_bitdepth_3d;
      auto grid = [&](GridDesc& G, bool on, uint32_t g, void* table, uint32_t* keys, uint64_t slots, bool hashed, uint32_t* mbits,
                      uint32_t* tbits) {
        G.on = on ? 1 : 0;
        if (!on) return;
        G.g = g; G.w = (maxs + g - 1) / g; G.disth = std::max(g / 2, 1u); G.th = g * G.w;
        G.magic = g > 1 ? (uint32_t)(((1ull << 32) + g - 1) / g) : 0u;
        G.g_shift = -1;
        for (int sft = 0; sft < 16; ++sft) if ((1u << sft) == g) G.g_shift = sft;
        G.slots = slots; G.table = table; G.keys = keys;
        G.identity = hashed ? 0 : 1;
        G.fast = 0; G.w_shift = 0; G.oob_mask = 0; G.cmask = 0;
        {
          int wl = -1;
          for (int sft = 0; sft <= 10; ++sft) if ((1u << sft) == G.w) wl = sft;
          if (!hashed && G.g_shift >= 0 && wl >= 0 && G.th <= 65536u) {
            G.fast = wl <= 8 ? 1 : 2; G.w_shift = (uint32_t)wl;      // 2: wider than the packed 8-bit cell keys (colour / probe only)
            G.oob_mask = (0xFFFFu & ~(G.th - 1u)) * 0x10001u;
            G.cmask = (G.w - 1u) * 0x10001u;
          }
        }
        G.mbits = mbits; G.tbits = tbits; G.mwords = (slots + 31) / 32; G.twords = (slots + (32u << kTouchShift) - 1) / (32u << kTouchShift);
      };
      grid(a.sm.geo, smoothing_geo, params.grid_size, d_geotab.p, d_geokeys.as<uint32_t>(), geotab_slots, geotab_hashed,
           d_geombits.as<uint32_t>(), d_geotbits.as<uint32_t>());
      grid(a.sm.col, smoothing_col, params.cgrid_size, d_coltab.p, d_colkeys.as<uint32_t>(), coltab_slots, coltab_hashed,
           d_colmbits.as<uint32_t>(), d_coltbits.as<uint32_t>());
      a.sm.blist = d_blist.as<BoundaryEntry>(); a.sm.blist_count = d_blist_count.as<uint32_t>(); a.sm.blist_cap = blist_cap;
      if (const char* e = getenv("TMC2_TEST_BLIST_CAP")) a.sm.blist_cap = std::min<uint64_t>(blist_cap, strtoull(e, nullptr, 10));   // test hook: provoke the device-side capacity failure
      a.sm.slist = d_slist.as<uint32_t>(); a.sm.slist_count = d_slist_count.as<uint32_t>();
      const uint32_t sc = params.attribute_bitdepth > 8 ? (1u << (params.attribute_bitdepth - 8)) : 1u;
      a.sm.thr_geo = params.threshold_smoothing;
      a.sm.thr_col_smooth = params.threshold_color_smoothing * sc;
      a.sm.thr_col_diff = params.threshold_color_difference * sc;
      a.sm.thr_col_var = params.threshold_color_variation * sc;
      a.sm.changed = d_changed.as<unsigned long long>();
    }
    return a;
  }

  uint64_t algorithmic_bytes_core(uint64_t total_points) const {
    // SURVEY.md 8(d): occ + geometry Y (2 maps) + attribute YUV 4:2:0 (2 maps) + per-point output streams
    uint64_t b = (uint64_t)F * ((uint64_t)occ_w * occ_h + 2ull * W * H * 2);
    if (params.attribute_count) b += (uint64_t)F * 2ull * ((uint64_t)W * H + 2ull * (W / 2) * (H / 2)) * 2;
    uint64_t per_point = 6;
    const bool dbg = (want & WANT_DEBUG) != 0;
    if (params.attribute_count) per_point += 3;
    if (dbg) per_point += (params.attribute_count ? 6 : 0) + 2 + 1 + 4;
    return b + per_point * total_points;
  }

  // ---- kernels ---------------------------------------------------------------------------------------------------
  // `timed`: record the stage-timing events (not inside a CUDA graph capture: captured events cannot be timed)
  tmc2_status launch(cudaStream_t s, Err& err, bool timed = true) {
    CU(cudaSetDevice(device));
    kernel_launch_count_reset();
    UnpackArgs a = make_args();
    if (timed) CU(cudaEventRecord(ev[0], s));
    CU(cudaMemsetAsync(d_b2p.p, 0, std::max<size_t>((size_t)F * bw * bh * 4, 4), s));
    CU(cudaMemsetAsync(d_count.p, 0, std::max<size_t>((size_t)F * 4, 4), s));
    KL(launch_block_to_patch(a, n_slots, s));
    KL(launch_compact_owned(a, s));
    if (timed) CU(cudaEventRecord(ev[1], s));
    const bool smooth = smoothing_geo || smoothing_col;
    const bool dbg = (want & WANT_DEBUG) != 0;
    CU(cudaMemsetAsync(d_changed.p, 0, std::max<size_t>((size_t)F * 16, 16), s));
    if (smooth) {
      CU(cudaMemsetAsync(d_blist_count.p, 0, std::max<size_t>((size_t)F * 4, 4), s));
      CU(cudaMemsetAsync(d_slist_count.p, 0, std::max<size_t>((size_t)F * 4, 4), s));
    }
    // unpack = count (points per owned slot) -> slot scan (run starts per frame, frame totals) -> emit
    if (timed) CU(cudaEventRecord(ev[6], s));
    KL(launch_count(a, 0, n_tiles, s));
    KL(launch_slot_scan(a, s));
    if (timed) CU(cudaEventRecord(ev[7], s));
    if (!smooth) {
      while (ev_grp.size() < 2) { cudaEvent_t e; CU(cudaEventCreate(&e)); ev_grp.push_back(e); }
      n_groups = 1;
      if (timed) CU(cudaEventRecord(ev_grp[0], s));
      KL(launch_emit(a, tile_maps, false, 0, n_tiles, s));
      if (timed) CU(cudaEventRecord(ev_grp[1], s));
    } else {
      // frame groups: unpack (+ cell statistics + boundary lists) -> filter -> clear, tables stay hot in L2
      const uint32_t GF = group_frames_eff;
      n_groups = (F + GF - 1) / GF;
      while (ev_grp.size() < 2 * (size_t)n_groups) { cudaEvent_t e; CU(cudaEventCreate(&e)); ev_grp.push_back(e); }
      while (ev_emit.size() < n_groups) {
        cudaEvent_t e1, e2;
        CU(cudaEventCreateWithFlags(&e1, cudaEventDisableTiming)); ev_emit.push_back(e1);
        CU(cudaEventCreateWithFlags(&e2, cudaEventDisableTiming)); ev_post.push_back(e2);
      }
      const GridDesc geo0 = a.sm.geo, col0 = a.sm.col;             // table set 0
      auto use_set = [&](GridDesc& G, const GridDesc& G0, uint32_t set, size_t cell_bytes) {
        if (!G0.on) return;
        G.table = static_cast<uint8_t*>(G0.table) + (size_t)set * GF * G0.slots * cell_bytes;
        G.keys = G0.keys ? G0.keys + (size_t)set * GF * G0.slots : nullptr;
        G.mbits = G0.mbits + (size_t)set * GF * G0.mwords;
        G.tbits = G0.tbits + (size_t)set * GF * G0.twords;
      };
      for (uint32_t gi = 0; gi < n_groups; ++gi) {
        const uint32_t f0 = gi * GF, f1 = std::min(F, f0 + GF), set = gi & 1u;
        a.sm.group_first_frame = f0; a.sm.group_frames = f1 - f0;
        use_set(a.sm.geo, geo0, set, sizeof(GeoCell));
        use_set(a.sm.col, col0, set, sizeof(ColCell));
        if (gi >= 2) CU(cudaStreamWaitEvent(s, ev_post[gi - 2], 0));          // this table set has been cleared
        if (clear_pending) { CU(cudaStreamWaitEvent(s, ev_tables_clean, 0)); clear_pending = false; }   // ... by the previous launch
        if (timed) CU(cudaEventRecord(ev_grp[2 * gi], s));
          KL(launch_emit(a, tile_maps, true, h_ftb[f0], h_ftb[f1], s));
        if (timed) CU(cudaEventRecord(ev_grp[2 * gi + 1], s));
        if (dbg) {
          CU(cudaMemcpyAsync(d_pos_pre.as<uint8_t>() + (size_t)f0 * cap * 6, d_pos.as<uint8_t>() + (size_t)f0 * cap * 6,
                             (size_t)(f1 - f0) * cap * 6, cudaMemcpyDeviceToDevice, s));
          if (a.out.yuv)
            CU(cudaMemcpyAsync(d_yuv_pre.as<uint8_t>() + (size_t)f0 * cap * 6, d_yuv.as<uint8_t>() + (size_t)f0 * cap * 6,
                               (size_t)(f1 - f0) * cap * 6, cudaMemcpyDeviceToDevice, s));
        }
        if (n_groups == 1) {
          // one group: filter (probe + apply) in line; the clear pass only matters to the NEXT launch, so it runs on the auxiliary
          // stream under that launch's block-to-patch / count passes (which do not touch the tables)
          KL(launch_smooth_filter(a, s));
          CU(cudaEventRecord(ev_emit[gi], s));
          CU(cudaStreamWaitEvent(aux_stream, ev_emit[gi], 0));
          KL(launch_smooth_clear(a, aux_stream));
          CU(cudaEventRecord(ev_tables_clean, aux_stream));
          clear_pending = true;
        } else {
          // post-passes of this group on the auxiliary stream, while the main stream goes on with the next group's emit
          CU(cudaEventRecord(ev_emit[gi], s));
          CU(cudaStreamWaitEvent(aux_stream, ev_emit[gi], 0));
          KL(launch_smooth_filter(a, aux_stream));
          KL(launch_smooth_clear(a, aux_stream));
          CU(cudaEventRecord(ev_post[gi], aux_stream));
        }
      }
      if (n_groups >= 2)
        for (uint32_t gi = n_groups - 2; gi < n_groups; ++gi) CU(cudaStreamWaitEvent(s, ev_post[gi], 0));
    }
    if (timed) CU(cudaEventRecord(ev[2], s));
    if (want & WANT_OCC_FULL) KL(launch_upsample(a, d_occ_full.as<uint8_t>(), s));
    if (dbg && !smooth) {
      CU(cudaMemcpyAsync(d_pos_pre.p, d_pos.p, (size_t)F * cap * 6, cudaMemcpyDeviceToDevice, s));
      if (a.out.yuv) CU(cudaMemcpyAsync(d_yuv_pre.p, d_yuv.p, (size_t)F * cap * 6, cudaMemcpyDeviceToDevice, s));
    }
    if (timed) CU(cudaEventRecord(ev[3], s)); if (timed) CU(cudaEventRecord(ev[4], s)); if (timed) CU(cudaEventRecord(ev[5], s));
    launches = (uint32_t)kernel_launch_count_reset() + ingest_launches;
    ingest_launches = 0;
    counts_ready = false; outputs_enqueued = false; counts_enqueued = false;
    return TMC2_OK;
  }

  // counts (+ error flag, + smoothing statistics) to the host: enqueue_counts puts the copies behind the kernels on `s`,
  // finish_counts waits for them and reads the result; fetch_counts does both
  tmc2_status enqueue_counts(cudaStream_t s, Err& err) {
    CU(cudaSetDevice(device));
    const size_t bytes = (size_t)F * 4 + (size_t)F * 16 + 16;
    CU(h_small.ensure(bytes));
    uint8_t* hs = h_small.as<uint8_t>();
    CU(cudaMemcpyAsync(hs, d_count.p, (size_t)F * 4, cudaMemcpyDeviceToHost, s));
    CU(cudaMemcpyAsync(hs + (size_t)F * 4, d_changed.p, (size_t)F * 16, cudaMemcpyDeviceToHost, s));
    CU(cudaMemcpyAsync(hs + (size_t)F * 20, d_err.p, 4, cudaMemcpyDeviceToHost, s));
    CU(cudaEventRecord(ev_counts, s));
    counts_enqueued = true;
    return TMC2_OK;
  }
  bool counts_arrived() {                       // non-blocking: have the kernels and the counts copy of this batch finished?
    if (!counts_enqueued) return false;
    cudaSetDevice(device);
    const cudaError_t e = cudaEventQuery(ev_counts);
    if (e != cudaSuccess) cudaGetLastError();
    return e == cudaSuccess;
  }
  tmc2_status finish_counts(cudaStream_t s, Err& err) {
    CU(cudaSetDevice(device));
    uint8_t* hs = h_small.as<uint8_t>();
    CU(cudaEventSynchronize(ev_counts));
    counts_enqueued = false;
    int dev_err = 0;
    memcpy(&dev_err, hs + (size_t)F * 20, 4);
    if (dev_err) {
      CU(cudaMemsetAsync(d_err.p, 0, 4, s));
      // a slot that bailed out may have claimed cells without marking them touched: the clear pass would miss them, so the
      // next launch of this batch starts from freshly zeroed tables
      geotab_slots = coltab_slots = 0; geotab_frames = coltab_frames = 0;
      FAIL((tmc2_status)dev_err, "device-side failure flag %d (7 = output capacity, 11 = watchdog / table)", dev_err);
    }
    counts.assign(F, 0); moved.assign(F, 0); recoloured.assign(F, 0);
    if (F) {
      memcpy(counts.data(), hs, (size_t)F * 4);
      memcpy(moved.data(), hs + (size_t)F * 4, (size_t)F * 8);
      memcpy(recoloured.data(), hs + (size_t)F * 12, (size_t)F * 8);
    }
    uint64_t total = 0;
    for (auto c : counts) total += c;
    unpack_alg_bytes = algorithmic_bytes_core(total);
    counts_ready = true;
    return TMC2_OK;
  }
  tmc2_status fetch_counts(cudaStream_t s, Err& err) {
    if (!counts_enqueued && enqueue_counts(s, err)) return err.st;
    return finish_counts(s, err);
  }

  // enqueue the per-frame result copies into one pinned slab; per-frame events signal completion
  tmc2_status enqueue_outputs(Err& err) {
    CU(cudaSetDevice(device));
    const bool attr = params.attribute_count != 0;
    out_pos_off.assign(F, 0); out_rgb_off.assign(F, 0);
    size_t off = 0;
    for (uint32_t k = 0; k < F; ++k) {
      out_pos_off[k] = off; off += round_up64((uint64_t)counts[k] * 6, 64);
      out_rgb_off[k] = off; if (attr) off += round_up64((uint64_t)counts[k] * 3, 64);
    }
    CU(h_out.ensure(std::max<size_t>(off, 64)));
    while (ev_frame.size() < F) {
      cudaEvent_t e;
      CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
      ev_frame.push_back(e);
    }
    CU(cudaStreamWaitEvent(d2h_stream, ev_counts, 0));
    uint8_t* ho = h_out.as<uint8_t>();
    for (uint32_t k = 0; k < F; ++k) {
      if (counts[k]) {
        CU(cudaMemcpyAsync(ho + out_pos_off[k], d_pos.as<uint8_t>() + (size_t)k * cap * 6, (size_t)counts[k] * 6,
                           cudaMemcpyDeviceToHost, d2h_stream));
        if (attr)
          CU(cudaMemcpyAsync(ho + out_rgb_off[k], d_rgb.as<uint8_t>() + (size_t)k * cap * 3, (size_t)counts[k] * 3,
                             cudaMemcpyDeviceToHost, d2h_stream));
      }
      CU(cudaEventRecord(ev_frame[k], d2h_stream));
    }
    outputs_enqueued = true;
    return TMC2_OK;
  }

  tmc2_status stage_times(StageTimes& t, Err& err) {
    CU(cudaSetDevice(device));
    CU(cudaEventSynchronize(ev[5]));
    CU(cudaEventElapsedTime(&t.b2p, ev[0], ev[1]));
    float whole = 0;
    CU(cudaEventElapsedTime(&whole, ev[1], ev[2]));
    CU(cudaEventElapsedTime(&t.count, ev[6], ev[7]));
    t.unpack = 0;
    for (uint32_t gi = 0; gi < n_groups; ++gi) {
      float ms = 0;
      CU(cudaEventElapsedTime(&ms, ev_grp[2 * gi], ev_grp[2 * gi + 1]));
      t.unpack += ms;
    }
    t.geo = std::max(0.f, whole - t.unpack - t.count);   // filter + clear launches of all groups (both smoothing stages)
    t.col = 0; t.rgb = 0;   // colour smoothing runs inside the same filter launch; RGB conversion is fused into the emit
    return TMC2_OK;
  }
};

}  // namespace

// ---------------------------------------------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------------------------------------------
struct PendingFrame {
  Batch* batch;
  uint32_t local;
  uint64_t global_index;
};

struct tmc2gpu_ctx {
  std::vector<int> devices;
  tmc2_limits limits{};
  std::vector<std::vector<std::unique_ptr<Batch>>> slots;   // [device][gofs_in_flight]
  std::unique_ptr<Batch> stage_batch;                        // single-frame stage API
  std::deque<PendingFrame> pending;
  uint64_t next_global = 0;
  uint64_t submit_epoch = 0;
  Err err;
  std::string last_error;
  Batch* last_batch = nullptr;                               // for launch info / stage times
  bool two_pass = false;
  bool device_output = false;                                // TMC2_CTX_DEVICE_OUTPUT: frames stay in HBM

  tmc2_status fail() { last_error = err.msg; return err.st; }
};

struct tmc2_resident {
  std::unique_ptr<Batch> batch;
};

extern "C" {

uint32_t tmc2gpu_abi_version(void) { return TMC2GPU_ABI_VERSION; }

int tmc2gpu_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

const char* tmc2gpu_status_string(tmc2_status s) {
  static const char* names[] = {"TMC2_OK", "TMC2_END", "TMC2_ERR_INVALID_ARG", "TMC2_ERR_PATCH_OUT_OF_CANVAS",
                                "TMC2_ERR_SHORT_VIDEO", "TMC2_ERR_MAP_COUNT", "TMC2_ERR_UNSUPPORTED", "TMC2_ERR_CAPACITY",
                                "TMC2_ERR_STATE", "TMC2_ERR_NO_DEVICE", "TMC2_ERR_CUDA", "TMC2_ERR_INTERNAL"};
  return (int)s >= 0 && (int)s < 12 ? names[s] : "TMC2_ERR_?";
}

tmc2_status tmc2gpu_create(const int* device_ids, int device_count, const tmc2_limits* limits, tmc2gpu_ctx** out_ctx) {
  if (!out_ctx) return TMC2_ERR_INVALID_ARG;
  *out_ctx = nullptr;
  const int n_dev = tmc2gpu_device_count();
  if (n_dev <= 0) return TMC2_ERR_NO_DEVICE;      // no CPU fallback
  std::unique_ptr<tmc2gpu_ctx> ctx(new tmc2gpu_ctx());
  if (device_ids && device_count > 0) {
    for (int i = 0; i < device_count; ++i) {
      if (device_ids[i] < 0 || device_ids[i] >= n_dev) return TMC2_ERR_NO_DEVICE;
      ctx->devices.push_back(device_ids[i]);
    }
  } else {
    ctx->devices.push_back(0);
  }
  if (limits) ctx->limits = *limits;
  if (ctx->limits.gofs_in_flight == 0) ctx->limits.gofs_in_flight = 2;
  if (ctx->limits.gofs_in_flight > 8) ctx->limits.gofs_in_flight = 8;
  ctx->two_pass = (ctx->limits.flags & TMC2_CTX_TWO_PASS_SCAN) != 0;
  ctx->device_output = (ctx->limits.flags & TMC2_CTX_DEVICE_OUTPUT) != 0;
  ctx->slots.resize(ctx->devices.size());
  for (size_t d = 0; d < ctx->devices.size(); ++d) {
    for (uint32_t k = 0; k < ctx->limits.gofs_in_flight; ++k) {
      std::unique_ptr<Batch> b(new Batch());
      if (b->init(ctx->devices[d], ctx->two_pass, ctx->err)) return ctx->err.st;
      ctx->slots[d].push_back(std::move(b));
    }
  }
  ctx->stage_batch.reset(new Batch());
  if (ctx->stage_batch->init(ctx->devices[0], ctx->two_pass, ctx->err)) return ctx->err.st;
  *out_ctx = ctx.release();
  return TMC2_OK;
}

void tmc2gpu_destroy(tmc2gpu_ctx* ctx) {
  if (!ctx) return;
  for (int d : ctx->devices) { cudaSetDevice(d); cudaDeviceSynchronize(); }
  delete ctx;
}

const char* tmc2gpu_last_error(const tmc2gpu_ctx* ctx) { return ctx ? ctx->last_error.c_str() : "ctx is NULL"; }

void* tmc2gpu_alloc_pinned(size_t bytes) {
  void* p = nullptr;
  if (bytes == 0) return nullptr;
  // TMC2_PINNED_WC=1: write-combined pages (the host only ever writes decoded samples into these planes; the DMA engine
  // reads them without snooping the CPU caches) -- an experiment knob, measured in profiles/
  static const bool wc = [] { const char* e = getenv("TMC2_PINNED_WC"); return e && atoi(e) != 0; }();
  if (cudaHostAlloc(&p, bytes, cudaHostAllocPortable | (wc ? cudaHostAllocWriteCombined : 0)) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  std::lock_guard<std::mutex> lk(g_pin_mu);
  g_pinned.emplace_back((const uint8_t*)p, bytes);
  return p;
}
void tmc2gpu_free_pinned(void* p) {
  if (!p) return;
  {
    std::lock_guard<std::mutex> lk(g_pin_mu);
    for (size_t i = 0; i < g_pinned.size(); ++i)
      if (g_pinned[i].first == p) { g_pinned.erase(g_pinned.begin() + i); break; }
  }
  cudaFreeHost(p);
}

// ---- streaming -----------------------------------------------------------------------------------------------
tmc2_status tmc2gpu_submit_gof(tmc2gpu_ctx* ctx, const tmc2_gof* gof) {
  if (!ctx) return TMC2_ERR_INVALID_ARG;
  Err& err = ctx->err;
  err = Err();
  TraceClock tc;
  if (validate_params(gof, err)) return ctx->fail();
  if (ctx->limits.max_frames && gof->frame_count > ctx->limits.max_frames) {
    err.st = TMC2_ERR_CAPACITY; err.msg = "GOF has more frames than limits.max_frames"; return ctx->fail();
  }
  if ((ctx->limits.max_width && gof->width > ctx->limits.max_width) ||
      (ctx->limits.max_height && gof->height > ctx->limits.max_height)) {
    err.st = TMC2_ERR_CAPACITY; err.msg = "frame larger than limits.max_width/height"; return ctx->fail();
  }
  std::vector<DevRange> dev_ranges;
  for (uint32_t f = 0; f < gof->frame_count; ++f)
    if (validate_frame(gof, f, ctx->devices, dev_ranges, err)) return ctx->fail();
  if (gof->frame_count == 0) return TMC2_OK;

  // Frame-wise sharding: contiguous slices of the GOF, one per device; no collective (SURVEY.md 8e).  A device's slice can
  // be cut further into chunks of TMC2_CHUNK_FRAMES frames, each an independent batch on its own stream (lower latency to
  // the first frame); measured on B200 it does not raise throughput once several GOFs are in flight, so the default is
  // one batch per device slice.
  const uint32_t D = (uint32_t)ctx->devices.size();
  const uint32_t F = gof->frame_count;
  static const uint32_t chunk_frames = [] { const char* e = getenv("TMC2_CHUNK_FRAMES"); return e ? (uint32_t)atoi(e) : 0u; }();
  struct Piece { uint32_t d, lo, hi; Batch* b; };
  std::vector<Piece> pieces;
  for (uint32_t d = 0; d < D; ++d) {
    const uint32_t lo = (uint32_t)((uint64_t)F * d / D), hi = (uint32_t)((uint64_t)F * (d + 1) / D);
    const uint32_t step = chunk_frames ? chunk_frames : std::max(hi - lo, 1u);
    for (uint32_t c = lo; c < hi; c += step) pieces.push_back({d, c, std::min(hi, c + step), nullptr});
  }
  // every piece needs a free batch of its device; batches are created on demand, up to gofs_in_flight GOFs of this shape
  for (uint32_t d = 0; d < D; ++d) {
    uint32_t need = 0;
    for (auto& pc : pieces) need += pc.d == d;
    if (!need) continue;
    std::vector<Batch*> free_list;
    for (auto& b : ctx->slots[d]) if (!b->busy) free_list.push_back(b.get());
    const size_t cap_batches = (size_t)ctx->limits.gofs_in_flight * need;
    while (free_list.size() < need && ctx->slots[d].size() < cap_batches) {
      std::unique_ptr<Batch> b(new Batch());
      if (b->init(ctx->devices[d], ctx->two_pass, err)) return ctx->fail();
      free_list.push_back(b.get());
      ctx->slots[d].push_back(std::move(b));
    }
    if (free_list.size() < need) {
      err.st = TMC2_ERR_STATE;
      err.msg = "all GOF slots in flight: drain frames with tmc2gpu_next_frame / release_frame first";
      return ctx->fail();
    }
    size_t k = 0;
    for (auto& pc : pieces) if (pc.d == d) pc.b = free_list[k++];
  }
  // A failure part-way through leaves no trace: pieces already enqueued are drained and freed, and none of the GOF's frames
  // stays in the hand-out queue (a GOF is delivered whole or not at all).
  const size_t pending_mark = ctx->pending.size();
  const uint64_t global_mark = ctx->next_global;
  auto undo = [&]() {
    for (auto& pc : pieces) {
      if (!pc.b) continue;
      cudaSetDevice(pc.b->device);
      cudaStreamSynchronize(pc.b->stream);           // also the piece that failed: it may have enqueued some copies
      cudaGetLastError();
      if (pc.b->busy && pc.b->t_epoch == ctx->submit_epoch) pc.b->busy = false;
    }
    ctx->pending.resize(pending_mark);
    ctx->next_global = global_mark;
  };
  ++ctx->submit_epoch;
  // The pieces (one per device, or per chunk) are independent batches: digest of the patch lists, staging, H2D and launch
  // enqueue of every piece run on their own host thread when there are several, so that one submitting thread keeps N devices
  // busy (src/lib.rs has exactly one worker thread above this call).
  std::vector<Err> perr(pieces.size());
  auto do_piece = [&](size_t i) {
    Piece& pc = pieces[i];
    Batch* b = pc.b;
    Err& e = perr[i];
    TraceClock pt;
    if (b->prepare(gof, pc.lo, pc.hi - pc.lo, 0, e)) return;
    const double t_prep = pt.lap();
    if (b->upload(gof, pc.lo, dev_ranges, e, pieces.size() == 1)) return;
    const double t_up = pt.lap();
    if (b->launch(b->stream, e)) return;
    if (b->enqueue_counts(b->stream, e)) return;          // counts travel right behind the kernels
    if (trace_on())
      fprintf(stderr, "[tmc2gpu] submit dev %d frames %u..%u: prepare %.3f upload-enqueue %.3f launch-enqueue %.3f ms\n",
              b->device, pc.lo, pc.hi, t_prep, t_up, pt.lap());
  };
  if (pieces.size() == 1) do_piece(0);
  else StagePool::get().run(pieces.size(), do_piece);
  for (size_t i = 0; i < pieces.size(); ++i)
    if (perr[i].st != TMC2_OK) { err = perr[i]; undo(); return ctx->fail(); }
  for (auto& pc : pieces) {
    Batch* b = pc.b;
    // counts travel right behind the kernels; result copies are enqueued when the first frame is asked for
    b->busy = true; b->frames_released = 0; b->t_epoch = ctx->submit_epoch;
    b->t_submit = std::chrono::steady_clock::now(); b->trace_wait_ms = 0;
    ctx->last_batch = b;
    for (uint32_t k = 0; k < pc.hi - pc.lo; ++k) ctx->pending.push_back({b, k, ctx->next_global++});
  }
  if (trace_on()) fprintf(stderr, "[tmc2gpu] submit_gof: %zu piece(s), %.3f ms on the calling thread\n", pieces.size(), tc.lap());
  return TMC2_OK;
}

tmc2_status tmc2gpu_wait_inputs(tmc2gpu_ctx* ctx) {
  if (!ctx) return TMC2_ERR_INVALID_ARG;
  Err& err = ctx->err;
  err = Err();
  auto body = [&]() -> tmc2_status {
    for (auto& v : ctx->slots)
      for (auto& b : v) {
        CU(cudaSetDevice(b->device));
        CU(cudaEventSynchronize(b->ev_inputs_free));
      }
    return TMC2_OK;
  };
  if (body()) return ctx->fail();
  return TMC2_OK;
}

tmc2_status tmc2gpu_next_frame(tmc2gpu_ctx* ctx, tmc2_frame_out* out) {
  if (!ctx || !out) return TMC2_ERR_INVALID_ARG;
  Err& err = ctx->err;
  err = Err();
  if (ctx->pending.empty()) return TMC2_END;
  PendingFrame pf = ctx->pending.front();
  Batch* b = pf.batch;
  TraceClock tc;
  // A GOF whose launch failed on the device (or whose copies failed) is dropped WHOLE: all of its frames leave the queue, its
  // slot is drained and freed, and the error is reported once -- a later call never hands out frames of the failed launch.
  auto drop_gof = [&]() {
    while (!ctx->pending.empty() && ctx->pending.front().batch == b) ctx->pending.pop_front();
    cudaSetDevice(b->device);
    cudaStreamSynchronize(b->stream);
    cudaStreamSynchronize(b->d2h_stream);
    cudaGetLastError();
    b->busy = false; b->counts_ready = false; b->outputs_enqueued = false; b->counts_enqueued = false;
  };
  const bool first = !b->counts_ready;
  if (!b->counts_ready && b->fetch_counts(b->stream, err)) { drop_gof(); return ctx->fail(); }
  // Result copies of the pieces BEHIND this one (other devices of the same GOF, later GOFs) are enqueued as soon as their
  // kernels have finished, not when their turn comes: otherwise the D2H transfers of a GOF sharded over N devices would run
  // one device after the other, in hand-out order.  Failures of those pieces are left for their own turn.
  {
    Batch* seen = b;
    for (const PendingFrame& q : ctx->pending) {
      if (q.batch == seen) continue;
      seen = q.batch;
      if (!seen->counts_ready && !seen->outputs_enqueued && seen->counts_arrived()) {
        Err e2;
        if (seen->finish_counts(seen->stream, e2) == TMC2_OK && !ctx->device_output) seen->enqueue_outputs(e2);
        else if (e2.st != TMC2_OK) { seen->counts_ready = false; seen->failed_early = e2; }
      }
    }
  }
  if (b->failed_early.st != TMC2_OK) { err = b->failed_early; b->failed_early = Err(); drop_gof(); return ctx->fail(); }
  const double t_counts = tc.lap();
  if (ctx->device_output) {
    // device-resident hand-off: the counts copy was enqueued behind the last kernel of the GOF, so every frame is complete
    ctx->pending.pop_front();
    memset(out, 0, sizeof *out);
    out->frame_index = pf.global_index;
    out->point_count = b->counts[pf.local];
    out->positions = reinterpret_cast<const uint16_t*>(b->d_pos.as<uint8_t>() + (size_t)pf.local * b->cap * 6);
    out->with_colors = b->params.attribute_count ? 1 : 0;
    out->colors = out->with_colors ? b->d_rgb.as<uint8_t>() + (size_t)pf.local * b->cap * 3 : nullptr;
    out->memory_space = 1;
    out->device = (uint8_t)b->device;
    out->smoothed_positions = b->moved[pf.local];
    out->smoothed_colors = b->recoloured[pf.local];
    out->_handle = b;
    return TMC2_OK;
  }
  if (!b->outputs_enqueued && b->enqueue_outputs(err)) { drop_gof(); return ctx->fail(); }
  const double t_enq = tc.lap();
  if (cudaSetDevice(b->device) != cudaSuccess || cudaEventSynchronize(b->ev_frame[pf.local]) != cudaSuccess) {
    err.st = TMC2_ERR_CUDA; err.msg = std::string("waiting for frame: ") + cudaGetErrorString(cudaGetLastError());
    drop_gof();
    return ctx->fail();
  }
  if (trace_on()) {
    const double t_wait = tc.lap();
    b->trace_wait_ms += t_counts + t_enq + t_wait;
    if (first || pf.local + 1 == b->F)
      fprintf(stderr, "[tmc2gpu] next_frame local %u: wait-counts %.3f enqueue-d2h %.3f wait-frame %.3f ms | GOF: inside next_frame "
              "%.3f ms, since submit %.3f ms\n", pf.local, t_counts, t_enq, t_wait, b->trace_wait_ms,
              std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - b->t_submit).count());
  }
  ctx->pending.pop_front();
  memset(out, 0, sizeof *out);
  out->frame_index = pf.global_index;
  out->point_count = b->counts[pf.local];
  out->positions = reinterpret_cast<const uint16_t*>(b->h_out.as<uint8_t>() + b->out_pos_off[pf.local]);
  out->with_colors = b->params.attribute_count ? 1 : 0;
  out->colors = out->with_colors ? b->h_out.as<uint8_t>() + b->out_rgb_off[pf.local] : nullptr;
  out->memory_space = 0;
  out->device = (uint8_t)b->device;
  out->smoothed_positions = b->moved[pf.local];
  out->smoothed_colors = b->recoloured[pf.local];
  out->_handle = b;
  return TMC2_OK;
}

tmc2_status tmc2gpu_release_frame(tmc2gpu_ctx* ctx, tmc2_frame_out* out) {
  if (!ctx || !out || !out->_handle) return TMC2_ERR_INVALID_ARG;
  Batch* b = static_cast<Batch*>(out->_handle);
  bool known = false;
  for (auto& v : ctx->slots) for (auto& s : v) known |= s.get() == b;
  if (!known || !b->busy) { ctx->last_error = "release_frame: frame was not handed out by this context"; return TMC2_ERR_STATE; }
  out->_handle = nullptr; out->positions = nullptr; out->colors = nullptr;
  if (++b->frames_released >= b->F) b->busy = false;
  return TMC2_OK;
}

// ---- PLY output (src/writer.rs:15-75), formatted on the device -------------------------------------------------
static std::string ply_header(uint32_t format, uint64_t n, bool colours) {
  std::string h = "ply\n";                                                      // write_header, src/writer.rs:31-60
  h += format == TMC2_PLY_ASCII ? "format ascii 1.0\n" : "format binary_little_endian 1.0\n";
  h += "element vertex " + std::to_string(n) + "\n";
  h += "property uint x\nproperty uint y\nproperty uint z\n";
  if (colours) h += "property uchar red\nproperty uchar green\nproperty uchar blue\n";
  h += "element face 0\nproperty list uint8 int32 vertex_index\nend_header\n";
  return h;
}

tmc2_status tmc2gpu_frame_to_ply(tmc2gpu_ctx* ctx, const tmc2_frame_out* frame, uint32_t format, void* dst, uint64_t dst_capacity,
                                 uint64_t* file_bytes) {
  if (!ctx || !frame || !file_bytes || !frame->_handle || (format != TMC2_PLY_ASCII && format != TMC2_PLY_BINARY_LE))
    return TMC2_ERR_INVALID_ARG;
  *file_bytes = 0;
  Err& err = ctx->err;
  err = Err();
  Batch* b = static_cast<Batch*>(frame->_handle);
  bool known = false;
  for (auto& v : ctx->slots) for (auto& s : v) known |= s.get() == b;
  if (!known || !b->busy || !b->counts_ready) { ctx->last_error = "frame_to_ply: frame was not handed out by this context (or already released)"; return TMC2_ERR_STATE; }
  // which frame of the batch: by its buffer (device slab or offset inside the pinned output area)
  uint32_t local = b->F;
  for (uint32_t k = 0; k < b->F; ++k) {
    const void* p = frame->memory_space == 1 ? static_cast<const void*>(b->d_pos.as<uint8_t>() + (size_t)k * b->cap * 6)
                                              : static_cast<const void*>(b->h_out.as<uint8_t>() + b->out_pos_off[k]);
    if (p == static_cast<const void*>(frame->positions) && b->counts[k] == frame->point_count) { local = k; break; }   // empty frames share an offset
  }
  if (local == b->F) { ctx->last_error = "frame_to_ply: not a frame of this context"; return TMC2_ERR_STATE; }
  auto body = [&]() -> tmc2_status {
    const uint64_t n = frame->point_count;
    const bool colours = b->params.attribute_count != 0;
    const std::string head = ply_header(format, n, colours);
    const uint16_t* dpos = reinterpret_cast<const uint16_t*>(b->d_pos.as<uint8_t>() + (size_t)local * b->cap * 6);
    const uint8_t* drgb = colours ? b->d_rgb.as<uint8_t>() + (size_t)local * b->cap * 3 : nullptr;
    CU(cudaSetDevice(b->device));
    cudaStream_t s = b->stream;                       // idle: the GOF of a handed-out frame is complete, the slot is still taken
    const uint64_t nb = ply_blocks(n);
    uint64_t body_bytes = n * (colours ? 15u : 12u);
    unsigned long long* d_offs = nullptr;
    if (format == TMC2_PLY_ASCII && n) {
      // [block sums u32 x nb, padded][block offsets u64 x nb][total u64]
      const size_t sums_bytes = (nb * 4 + 7) / 8 * 8;
      CU(b->d_ply_sums.ensure(sums_bytes + nb * 8 + 8));
      CU(b->h_ply.ensure(8));
      uint32_t* d_sums = b->d_ply_sums.as<uint32_t>();
      d_offs = reinterpret_cast<unsigned long long*>(b->d_ply_sums.as<uint8_t>() + sums_bytes);
      CU((cudaError_t)launch_ply_measure(dpos, drgb, n, d_sums, s));
      CU((cudaError_t)launch_ply_scan(d_sums, n, d_offs, d_offs + nb, s));
      CU(cudaMemcpyAsync(b->h_ply.p, d_offs + nb, 8, cudaMemcpyDeviceToHost, s));
      CU(cudaStreamSynchronize(s));
      body_bytes = *static_cast<const unsigned long long*>(b->h_ply.p);
    }
    *file_bytes = head.size() + body_bytes;
    if (!dst) return TMC2_OK;                         // size query
    if (dst_capacity < *file_bytes) {
      err.st = TMC2_ERR_CAPACITY;
      err.msg = fmt("frame_to_ply: the file has %llu bytes, the destination %llu", (unsigned long long)*file_bytes, (unsigned long long)dst_capacity);
      return err.st;
    }
    cudaPointerAttributes at{};
    const bool dst_on_device = cudaPointerGetAttributes(&at, dst) == cudaSuccess && at.type == cudaMemoryTypeDevice;
    cudaGetLastError();
    if (dst_on_device && at.device != b->device) {
      err.st = TMC2_ERR_INVALID_ARG; err.msg = "frame_to_ply: device destination is not on the frame's device";
      return err.st;
    }
    uint8_t* out_body = static_cast<uint8_t*>(dst) + head.size();
    if (dst_on_device) {
      CU(cudaMemcpyAsync(dst, head.data(), head.size(), cudaMemcpyHostToDevice, s));
      CU((cudaError_t)launch_ply_write(dpos, drgb, n, d_offs, out_body, format == TMC2_PLY_ASCII, s));
    } else {
      memcpy(dst, head.data(), head.size());
      if (n) {
        CU(b->d_ply.ensure(body_bytes + 16));
        CU((cudaError_t)launch_ply_write(dpos, drgb, n, d_offs, b->d_ply.as<uint8_t>(), format == TMC2_PLY_ASCII, s));
        CU(cudaMemcpyAsync(out_body, b->d_ply.p, body_bytes, cudaMemcpyDeviceToHost, s));
      }
    }
    CU(cudaStreamSynchronize(s));
    return TMC2_OK;
  };
  if (body()) return ctx->fail();
  return TMC2_OK;
}

// ---- resident path -------------------------------------------------------------------------------------------
tmc2_status tmc2gpu_upload_gof(tmc2gpu_ctx* ctx, const tmc2_gof* gof, tmc2_resident** out) {
  if (!ctx || !out) return TMC2_ERR_INVALID_ARG;
  *out = nullptr;
  Err& err = ctx->err;
  err = Err();
  if (validate_params(gof, err)) return ctx->fail();
  std::vector<DevRange> dev_ranges;
  for (uint32_t f = 0; f < gof->frame_count; ++f)
    if (validate_frame(gof, f, ctx->devices, dev_ranges, err)) return ctx->fail();
  std::unique_ptr<tmc2_resident> r(new tmc2_resident());
  r->batch.reset(new Batch());
  Batch* b = r->batch.get();
  if (b->init(ctx->devices[0], ctx->two_pass, err) || b->prepare(gof, 0, gof->frame_count, 0, err) || b->upload(gof, 0, dev_ranges, err))
    return ctx->fail();
  if (cudaStreamSynchronize(b->stream) != cudaSuccess) { err.st = TMC2_ERR_CUDA; err.msg = "upload sync"; return ctx->fail(); }
  b->h_in.release();   // planes now live in HBM; the staging area is not needed again
  *out = r.release();
  return TMC2_OK;
}

tmc2_status tmc2gpu_reconstruct_resident(tmc2gpu_ctx* ctx, tmc2_resident* r, void* cuda_stream) {
  return tmc2gpu_reconstruct_resident_ex(ctx, r, cuda_stream, 0);
}

tmc2_status tmc2gpu_reconstruct_resident_ex(tmc2gpu_ctx* ctx, tmc2_resident* r, void* cuda_stream, uint32_t flags) {
  if (!ctx || !r) return TMC2_ERR_INVALID_ARG;
  Err& err = ctx->err;
  err = Err();
  Batch* b = r->batch.get();
  cudaStream_t s = cuda_stream ? (cudaStream_t)cuda_stream : b->stream;
  // Relaunches of a resident GOF are the same launch sequence every time: without smoothing (no auxiliary stream, nothing
  // that outlives the launch) it is captured once into a CUDA graph and replayed with one API call -- for a small GOF
  // (BASELINE config 1: one frame, 8 launches + 3 memsets of a few microseconds each) the CPU launch cost is what bounds the
  // rate.  The first launch and every TMC2_GRAPH=0 launch take the ordinary path, which also records the stage-timing events.
  static const bool graphs = [] { const char* e = getenv("TMC2_GRAPH"); return !e || atoi(e) != 0; }();
  const bool eligible = graphs && !(flags & TMC2_LAUNCH_TIMED) && !(b->smoothing_geo || b->smoothing_col) && b->want == 0;
  if (eligible && b->graph_exec) {
    auto replay = [&]() -> tmc2_status {
      CU(cudaSetDevice(b->device));
      CU(cudaGraphLaunch(b->graph_exec, s));
      b->counts_ready = false; b->outputs_enqueued = false; b->counts_enqueued = false;
      return TMC2_OK;
    };
    if (replay()) return ctx->fail();
    ctx->last_batch = b;
    return TMC2_OK;
  }
  if (b->launch(s, err)) return ctx->fail();
  if (eligible && !b->graph_tried) {
    // capture the NEXT launches (this one ran directly: buffers, function attributes and stage times are in place)
    b->graph_tried = true;
    cudaGraph_t g = nullptr;
    const uint32_t launches = b->launches;
    if (cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
      Err e2;
      const tmc2_status st = b->launch(s, e2, false);
      const cudaError_t ce = cudaStreamEndCapture(s, &g);
      if (st == TMC2_OK && ce == cudaSuccess && g && cudaGraphInstantiate(&b->graph_exec, g, 0) != cudaSuccess) b->graph_exec = nullptr;
      if (st != TMC2_OK || ce != cudaSuccess) b->graph_exec = nullptr;
      if (g) cudaGraphDestroy(g);
    }
    cudaGetLastError();
    b->launches = launches;
  }
  ctx->last_batch = b;
  return TMC2_OK;
}

tmc2_status tmc2gpu_resident_counts(tmc2gpu_ctx* ctx, tmc2_resident* r, uint64_t* point_counts) {
  if (!ctx || !r || !point_counts) return TMC2_ERR_INVALID_ARG;
  Err& err = ctx->err;
  err = Err();
  Batch* b = r->batch.get();
  if (cudaSetDevice(b->device) != cudaSuccess || cudaDeviceSynchronize() != cudaSuccess) {
    err.st = TMC2_ERR_CUDA; err.msg = std::string("device sync: ") + cudaGetErrorString(cudaGetLastError()); return ctx->fail();
  }
  if (b->fetch_counts(b->stream, err)) return ctx->fail();
  for (uint32_t k = 0; k < b->F; ++k) point_counts[k] = b->counts[k];
  return TMC2_OK;
}

tmc2_status tmc2gpu_resident_fetch(tmc2gpu_ctx* ctx, tmc2_resident* r, uint32_t frame, uint16_t* positions, uint8_t* colors,
                                   uint64_t capacity_points) {
  if (!ctx || !r) return TMC2_ERR_INVALID_ARG;
  Err& err = ctx->err;
  err = Err();
  Batch* b = r->batch.get();
  if (frame >= b->F) return TMC2_ERR_INVALID_ARG;
  if (cudaSetDevice(b->device) != cudaSuccess || cudaDeviceSynchronize() != cudaSuccess) {
    err.st = TMC2_ERR_CUDA; err.msg = "device sync"; return ctx->fail();
  }
  if (!b->counts_ready && b->fetch_counts(b->stream, err)) return ctx->fail();
  const uint64_t n = b->counts[frame];
  if (n > capacity_points) { err.st = TMC2_ERR_CAPACITY; err.msg = "resident_fetch: capacity_points too small"; return ctx->fail(); }
  auto body = [&]() -> tmc2_status {
    if (positions && n)
      CU(cudaMemcpy(positions, b->d_pos.as<uint8_t>() + (size_t)frame * b->cap * 6, n * 6, cudaMemcpyDeviceToHost));
    if (colors && n && b->params.attribute_count)
      CU(cudaMemcpy(colors, b->d_rgb.as<uint8_t>() + (size_t)frame * b->cap * 3, n * 3, cudaMemcpyDeviceToHost));
    return TMC2_OK;
  };
  if (body()) return ctx->fail();
  return TMC2_OK;
}

tmc2_status tmc2gpu_free_resident(tmc2gpu_ctx* ctx, tmc2_resident* r) {
  if (!ctx || !r) return TMC2_ERR_INVALID_ARG;
  if (ctx->last_batch == r->batch.get()) ctx->last_batch = nullptr;
  cudaSetDevice(r->batch->device);
  cudaDeviceSynchronize();
  delete r;
  return TMC2_OK;
}

tmc2_status tmc2gpu_last_launch_info(tmc2gpu_ctx* ctx, uint32_t* kernel_launches, uint64_t* unpack_algorithmic_bytes,
                                     uint64_t* total_points) {
  if (!ctx || !ctx->last_batch) return TMC2_ERR_STATE;
  Batch* b = ctx->last_batch;
  Err& err = ctx->err;
  err = Err();
  if (!b->counts_ready) {
    if (cudaSetDevice(b->device) != cudaSuccess || cudaDeviceSynchronize() != cudaSuccess) return TMC2_ERR_CUDA;
    if (b->fetch_counts(b->stream, err)) return ctx->fail();
  }
  uint64_t total = 0;
  for (auto c : b->counts) total += c;
  if (kernel_launches) *kernel_launches = b->launches;
  if (unpack_algorithmic_bytes) *unpack_algorithmic_bytes = b->unpack_alg_bytes;
  if (total_points) *total_points = total;
  return TMC2_OK;
}

tmc2_status tmc2gpu_last_unpack_ms(tmc2gpu_ctx* ctx, float* ms) {
  if (!ctx || !ctx->last_batch || !ms) return TMC2_ERR_STATE;
  StageTimes t;
  ctx->err = Err();
  if (ctx->last_batch->stage_times(t, ctx->err)) return ctx->fail();
  *ms = t.unpack;
  return TMC2_OK;
}

tmc2_status tmc2gpu_last_stage_ms(tmc2gpu_ctx* ctx, float* ms5) {
  if (!ctx || !ctx->last_batch || !ms5) return TMC2_ERR_STATE;
  StageTimes t;
  ctx->err = Err();
  if (ctx->last_batch->stage_times(t, ctx->err)) return ctx->fail();
  ms5[0] = t.b2p; ms5[1] = t.unpack; ms5[2] = t.geo; ms5[3] = t.count; ms5[4] = t.rgb;
  return TMC2_OK;
}

// ---- stage entry points -----------------------------------------------------------------------------------------
static tmc2_status run_single(tmc2gpu_ctx* ctx, const tmc2_gof* gof, uint32_t frame_index, uint32_t want) {
  Err& err = ctx->err;
  err = Err();
  if (validate_params(gof, err)) return err.st;
  if (frame_index >= gof->frame_count) FAIL(TMC2_ERR_INVALID_ARG, "frame_index %u >= frame_count %u", frame_index, gof->frame_count);
  std::vector<DevRange> dev_ranges;
  if (validate_frame(gof, frame_index, ctx->devices, dev_ranges, err)) return err.st;
  Batch* b = ctx->stage_batch.get();
  if (b->prepare(gof, frame_index, 1, want, err) || b->upload(gof, frame_index, dev_ranges, err) || b->launch(b->stream, err))
    return err.st;
  if (b->fetch_counts(b->stream, err)) return err.st;
  ctx->last_batch = b;
  return TMC2_OK;
}

tmc2_status tmc2gpu_generate_block_to_patch_from_occupancy_map_video(tmc2gpu_ctx* ctx, const tmc2_gof* gof,
                                                                      uint32_t frame_index, uint32_t* block_to_patch) {
  if (!ctx || !block_to_patch) return TMC2_ERR_INVALID_ARG;
  if (run_single(ctx, gof, frame_index, 0)) return ctx->fail();
  Batch* b = ctx->stage_batch.get();
  Err& err = ctx->err;
  if (cudaMemcpy(block_to_patch, b->d_b2p.p, (size_t)b->bw * b->bh * 4, cudaMemcpyDeviceToHost) != cudaSuccess) {
    err.st = TMC2_ERR_CUDA; err.msg = "block_to_patch D2H"; return ctx->fail();
  }
  return TMC2_OK;
}

tmc2_status tmc2gpu_generate_point_cloud(tmc2gpu_ctx* ctx, const tmc2_gof* gof, uint32_t frame_index,
                                         tmc2_point_cloud_out* out) {
  if (!ctx || !out) return TMC2_ERR_INVALID_ARG;
  const bool dbg = out->colors16bit || out->partition || out->point_to_pixel || out->boundary_type ||
                   out->positions_presmooth || out->colors16bit_presmooth;
  const uint32_t want = (dbg ? WANT_DEBUG : 0u) | (out->occupancy_map ? WANT_OCC_FULL : 0u);
  if (run_single(ctx, gof, frame_index, want)) return ctx->fail();
  Batch* b = ctx->stage_batch.get();
  Err& err = ctx->err;
  const uint64_t n = b->counts[0];
  out->point_count = n;
  out->smoothed_positions = b->moved[0];
  out->smoothed_colors = b->recoloured[0];
  if (n > out->capacity_points) { err.st = TMC2_ERR_CAPACITY; err.msg = "capacity_points too small"; return ctx->fail(); }
  const bool attr = b->params.attribute_count != 0;
  auto d2h = [&](void* dst, const void* src, size_t bytes) -> bool {
    if (!dst || !bytes || !src) return true;
    return cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost) == cudaSuccess;
  };
  bool ok = true;
  ok &= d2h(out->positions, b->d_pos.p, n * 6);
  if (attr) ok &= d2h(out->colors, b->d_rgb.p, n * 3);
  if (attr && dbg) ok &= d2h(out->colors16bit, b->d_yuv.p, n * 6);
  if (dbg) {
    ok &= d2h(out->boundary_type, b->d_bt.p, n);
    ok &= d2h(out->positions_presmooth, b->d_pos_pre.p, n * 6);
    if (attr) ok &= d2h(out->colors16bit_presmooth, b->d_yuv_pre.p, n * 6);
    if (out->partition && n) {
      std::vector<uint16_t> tmp(n);
      ok &= d2h(tmp.data(), b->d_part.p, n * 2);
      for (uint64_t i = 0; i < n; ++i) out->partition[i] = tmp[i];
    }
    if (out->point_to_pixel && n) {
      std::vector<uint32_t> tmp(n);
      ok &= d2h(tmp.data(), b->d_pix.p, n * 4);
      for (uint64_t i = 0; i < n; ++i) {
        out->point_to_pixel[3 * i] = tmp[i] & 0x7FFFu;
        out->point_to_pixel[3 * i + 1] = (tmp[i] >> 15) & 0x7FFFu;
        out->point_to_pixel[3 * i + 2] = tmp[i] >> 30;
      }
    }
  }
  if (out->occupancy_map) ok &= d2h(out->occupancy_map, b->d_occ_full.p, (size_t)b->W * b->H);
  if (out->block_to_patch) ok &= d2h(out->block_to_patch, b->d_b2p.p, (size_t)b->bw * b->bh * 4);
  if (!ok) { err.st = TMC2_ERR_CUDA; err.msg = std::string("D2H: ") + cudaGetErrorString(cudaGetLastError()); return ctx->fail(); }
  return TMC2_OK;
}

tmc2_status tmc2gpu_convert_yuv16_to_rgb8(tmc2gpu_ctx* ctx, const uint16_t* yuv16, uint64_t n, uint8_t* rgb8) {
  if (!ctx || (n && (!yuv16 || !rgb8))) return TMC2_ERR_INVALID_ARG;
  if (n == 0) return TMC2_OK;
  Err& err = ctx->err;
  err = Err();
  Batch* b = ctx->stage_batch.get();
  auto body = [&]() -> tmc2_status {
    CU(cudaSetDevice(b->device));
    DevBuf din, dout;
    CU(din.ensure(n * 6));
    CU(dout.ensure(n * 3));
    CU(cudaMemcpyAsync(din.p, yuv16, n * 6, cudaMemcpyHostToDevice, b->stream));
    KL(launch_yuv_to_rgb_flat(din.as<uint16_t>(), dout.as<uint8_t>(), n, b->stream));
    CU(cudaMemcpyAsync(rgb8, dout.p, n * 3, cudaMemcpyDeviceToHost, b->stream));
    CU(cudaStreamSynchronize(b->stream));
    din.release(); dout.release();
    return TMC2_OK;
  };
  if (body()) return ctx->fail();
  return TMC2_OK;
}

}  // extern "C"
