// Shared helpers for libddn_b200.so: error reporting, launch accounting, small device utilities.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <atomic>

#include "../../include/ddn_b200.h"

namespace ddn {

void set_error(const char* fmt, ...);
extern std::atomic<int64_t> g_launches;

inline int check_cuda(cudaError_t e, const char* what) {
  if (e != cudaSuccess) {
    set_error("%s: %s", what, cudaGetErrorString(e));
    return DDN_ERR_CUDA;
  }
  return DDN_OK;
}

// Optional per-launch timing (ddn_profile_enable): an event after every launch that passes its stream.
void profile_mark(const char* name, cudaStream_t st);
extern std::atomic<int> g_profile;

// Call after every kernel launch: counts it and surfaces launch-configuration errors.
inline int after_launch(const char* name) {
  g_launches.fetch_add(1, std::memory_order_relaxed);
  return check_cuda(cudaPeekAtLastError(), name);
}
inline int after_launch(const char* name, cudaStream_t st) {
  if (g_profile.load(std::memory_order_relaxed)) profile_mark(name, st);
  return after_launch(name);
}

#define DDN_REQUIRE(cond, msg)                      \
  do {                                              \
    if (!(cond)) {                                  \
      ::ddn::set_error("invalid argument: %s", msg); \
      return DDN_ERR_INVALID_ARGUMENT;              \
    }                                               \
  } while (0)

#define DDN_TRY(expr)            \
  do {                           \
    int _rc = (expr);            \
    if (_rc != DDN_OK) return _rc; \
  } while (0)

constexpr int kNumSMs = 148;  // B200
// Work units of the ragged layout: the remap kernel's 126 x 32 pixel tile (align.cu) and the consistency kernel's
// points per CTA (filter.cu, kFilterChunk).
constexpr int kRemapTileW = 126, kRemapTileH = 32, kFilterChunkPoints = 1024;

inline int64_t align_up(int64_t x, int64_t a) { return (x + a - 1) / a * a; }

// Host-side validation of a ragged view layout (include/ddn_b200.h, DDN_LAYOUT_COLS) before anything is launched:
// the offsets and work-unit prefixes must be the prefix sums of the sizes, so no layout can send a kernel outside its
// buffers.
inline int check_layout(int64_t n_views, const int64_t* L) {
  DDN_REQUIRE(L != nullptr, "null layout_host");
  DDN_REQUIRE(n_views >= 1 && n_views <= 65535, "a ragged layout holds 1 to 65535 views");
  const int64_t* last = L + n_views * DDN_LAYOUT_COLS;
  const int64_t s = last[0];
  DDN_REQUIRE(s >= 1 && last[1] == n_views, "layout: the last row must hold the stride and the view count");
  int64_t pix = 0, grid = 0, tiles = 0, chunks = 0;
  for (int64_t v = 0; v < n_views; ++v) {
    const int64_t* r = L + v * DDN_LAYOUT_COLS;
    const int64_t h = r[0], w = r[1];
    DDN_REQUIRE(h >= 1 && w >= 1 && h < (1 << 22) && w < (1 << 22) && h * w < (1ll << 31),
                "layout: every side must be 1 .. 2^22 - 1 and every view below 2^31 pixels");
    DDN_REQUIRE(r[2] == pix && r[3] == grid && r[4] == tiles && r[5] == chunks,
                "layout: the offsets are not the prefix sums of the view sizes");
    const int64_t hs = (h + s - 1) / s, ws = (w + s - 1) / s;
    pix += h * w;
    grid += hs * ws;
    tiles += ((h + kRemapTileH - 1) / kRemapTileH) * ((w + kRemapTileW - 1) / kRemapTileW);
    chunks += (hs * ws + kFilterChunkPoints - 1) / kFilterChunkPoints;
  }
  DDN_REQUIRE(last[2] == pix && last[3] == grid && last[4] == tiles && last[5] == chunks,
              "layout: the totals are not the sums of the view sizes");
  DDN_REQUIRE(pix < (1ll << 32), "the views must hold fewer than 2^32 pixels in all (32-bit gather offsets)");
  return DDN_OK;
}

// View of a flat work unit (remap tile or consistency chunk): the last v with layout[v][col] <= unit.  CTA-uniform.
__device__ __forceinline__ int layout_view_of(const int64_t* __restrict__ layout, int n_views, int col, int64_t unit) {
  int lo = 0, hi = n_views - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (__ldg(layout + (size_t)mid * DDN_LAYOUT_COLS + col) <= unit) lo = mid;
    else hi = mid - 1;
  }
  return lo;
}

// Order-preserving float <-> int encoding for atomicMin/atomicMax on floats.
__device__ __forceinline__ int float_to_ordered(float f) {
  int i = __float_as_int(f);
  return i >= 0 ? i : i ^ 0x7fffffff;
}
__device__ __forceinline__ float ordered_to_float(int i) {
  return __int_as_float(i >= 0 ? i : i ^ 0x7fffffff);
}

// Packed FP32 pairs: sm_100's FFMA2 / FMUL2 / FADD2 do two float32 operations per issue slot.  Each lane is exactly
// the IEEE operation of the scalar form (fma.rn, mul.rn, sub.rn, add.rz, no flush to zero), so evaluating two values
// as a pair gives the same bits as evaluating them one by one.  A pair is one 64-bit register pair, first value in
// the low half.
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pack2(float lo, float hi) {
  f32x2 r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ f32x2 splat2(float x) { return pack2(x, x); }
__device__ __forceinline__ void unpack2(f32x2 p, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(p)); }
__device__ __forceinline__ float lane2(f32x2 p, int e) {
  float lo, hi;
  unpack2(p, lo, hi);
  return e ? hi : lo;
}
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) {
  f32x2 r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b) {
  f32x2 r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ f32x2 sub2(f32x2 a, f32x2 b) {
  f32x2 r;
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ f32x2 add_rz2(f32x2 a, f32x2 b) {
  f32x2 r;
  asm("add.rz.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}

// World position of a pixel from P = d*x, Q = d*y, d and the view's 16-float src_table row (rows of
// R_s^T Kinv_s with the camera centre appended; scripts/test.py:79-90 then :233).  K4 (filter.cu) and the
// bounding-box epilogue of K3 (align.cu) both call this, so the box encloses K4's points bit for bit.
__device__ __forceinline__ void backproject_pqd(const float* __restrict__ s, float P, float Q, float d, float& X, float& Y,
                                                float& Z) {
  X = fmaf(s[0], P, fmaf(s[1], Q, fmaf(s[2], d, s[3])));
  Y = fmaf(s[4], P, fmaf(s[5], Q, fmaf(s[6], d, s[7])));
  Z = fmaf(s[8], P, fmaf(s[9], Q, fmaf(s[10], d, s[11])));
}
// The same for a pair of pixels, bit for bit per lane.
__device__ __forceinline__ void backproject_pqd2(const float* __restrict__ s, f32x2 P, f32x2 Q, f32x2 d, f32x2& X, f32x2& Y,
                                                 f32x2& Z) {
  X = fma2(splat2(s[0]), P, fma2(splat2(s[1]), Q, fma2(splat2(s[2]), d, splat2(s[3]))));
  Y = fma2(splat2(s[4]), P, fma2(splat2(s[5]), Q, fma2(splat2(s[6]), d, splat2(s[7]))));
  Z = fma2(splat2(s[8]), P, fma2(splat2(s[9]), Q, fma2(splat2(s[10]), d, splat2(s[11]))));
}

}  // namespace ddn
