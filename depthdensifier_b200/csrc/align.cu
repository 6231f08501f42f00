// Stage 1: per-view alignment of monocular depth to projected COLMAP sparse points.
//
// Reference semantics: src/depthdensifier/depth_refiner.py:92-328 (see include/ddn_b200.h).
//   K1+K2  align_stats_kernel  one CTA per view: project sparse points (float32, :92-115), bounds gate
//          and bilinear sample (:247-288), IQR outlier rejection on z_colmap/z_mono (:117-139),
//          min-count gate and <=500 subsample (:296-306), scale_factor (:315), then the lookup table
//          sorted by x (:148-150) or, in affine mode, the five-sum least squares in float64.
//   K3     remap_median_kernel  fused per-pixel piecewise-linear remap (:157-176), 3x3 replicate
//          median (:194-200) and mask (:203): depth+mask are read once, refined written once
//          (9 B/pixel instead of the reference's 9x unfold blow-up).  The per-pixel searchsorted runs
//          through a 1024-bucket index of the table built by K2, the median through sorted row triples.
#include <stdlib.h>

#include <cuda.h>  // CUtensorMap (types only: the encoder is fetched through cudaGetDriverEntryPoint, no -lcuda)

#include "common.cuh"

namespace ddn {

constexpr int kStatsThreads = 1024;
constexpr int kSortSmemMax = 16384;  // u64 entries sorted in shared memory (128 KB); larger -> global

struct AlignWorkspace {
  float* zd;     // [V,C] sampled mono depth of the surviving pairs
  float* zc;     // [V,C] COLMAP depth of the surviving pairs
  float* ratio;  // [V,C]
  float* tx;     // [V,C] table x (sorted)
  float* ty;     // [V,C] table y
  unsigned long long* sortbuf;  // [V,Cp]
  uint32_t* bucket;             // [V,kBuckets] search acceleration of the table: start | end << 16
  void* tensor_map;             // device copy of the TMA descriptor of the depth maps (use_tma)
  int64_t C, Cp;
};

// Uniform buckets over the table's x range.  bucket_of() is monotone non-decreasing in d (float
// subtract, multiply by a positive constant and truncation all are), so every knot in a lower bucket
// than d's is < d and every knot in a higher bucket is > d: searchsorted_left(xs, d) lies inside the
// knot range of d's own bucket, exactly.
constexpr int kBuckets = 1024;
__device__ __forceinline__ float bucket_scale(float xmin, float xmax) {
  const float w = __fadd_rn(xmax, -xmin);
  return w > 0.f ? __fdiv_rn((float)kBuckets, w) : 0.f;
}
__device__ __forceinline__ int bucket_of(float d, float xmin, float scale) {
  return min(max(__float2int_rz(__fmul_rn(__fadd_rn(d, -xmin), scale)), 0), kBuckets - 1);
}

static int64_t next_pow2(int64_t x) {
  int64_t p = 1;
  while (p < x) p <<= 1;
  return p;
}

static int64_t align_ws_bytes(int64_t V, int64_t C) {
  const int64_t Cp = next_pow2(C > 1 ? C : 2);
  return align_up(V * C * 4, 256) * 5 + align_up(V * Cp * 8, 256) + align_up(V * 1024 * 4, 256) + 256 + 256;  // + a TMA descriptor
}

static AlignWorkspace carve(void* ws, int64_t V, int64_t C) {
  AlignWorkspace w;
  w.C = C;
  w.Cp = next_pow2(C > 1 ? C : 2);
  char* p = reinterpret_cast<char*>(align_up((int64_t)(uintptr_t)ws, 256));
  const int64_t fb = align_up(V * C * 4, 256);
  w.zd = (float*)p; p += fb;
  w.zc = (float*)p; p += fb;
  w.ratio = (float*)p; p += fb;
  w.tx = (float*)p; p += fb;
  w.ty = (float*)p; p += fb;
  w.sortbuf = (unsigned long long*)p; p += align_up(V * w.Cp * 8, 256);
  w.bucket = (uint32_t*)p;
  p += align_up(V * 1024 * 4, 256);
  w.tensor_map = (void*)p;  // 128 bytes, 256-byte aligned
  return w;
}

// ---- block-level primitives (blockDim.x == kStatsThreads) ----------------------------------------

// Order-preserving compaction of one <=blockDim chunk; returns this thread's slot or -1. `base` is
// advanced by the chunk's count (uniform across the block after the call).
__device__ __forceinline__ int block_compact_slot(bool flag, int& base, int* s_warp) {
  const unsigned m = __ballot_sync(0xffffffffu, flag);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (lane == 0) s_warp[wid] = __popc(m);
  __syncthreads();
  if (wid == 0) {
    int v = s_warp[lane];
    int incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      int n = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += n;
    }
    s_warp[lane] = incl - v;
    if (lane == 31) s_warp[32] = incl;
  }
  __syncthreads();
  const int slot = flag ? base + s_warp[wid] + __popc(m & ((1u << lane) - 1)) : -1;
  base += s_warp[32];
  __syncthreads();
  return slot;
}

__device__ void block_bitonic_sort(unsigned long long* buf, int n_pow2) {
  for (int k = 2; k <= n_pow2; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = threadIdx.x; i < n_pow2; i += blockDim.x) {
        const int ixj = i ^ j;
        if (ixj > i) {
          const unsigned long long a = buf[i], b = buf[ixj];
          const bool asc = (i & k) == 0;
          if ((a > b) == asc) {
            buf[i] = b;
            buf[ixj] = a;
          }
        }
      }
      __syncthreads();
    }
  }
}

__device__ __forceinline__ unsigned ordered_bits(float f) {
  const unsigned b = __float_as_uint(f);
  return b ^ ((b >> 31) ? 0xffffffffu : 0x80000000u);
}

__device__ __forceinline__ int pow2_at_least(int n) {
  int p = 2;
  while (p < n) p <<= 1;
  return p;
}

// Sort indices 0..n-1 by (key(i), i) ascending; afterwards low 32 bits of buf[r] = index of rank r.
template <typename KeyFn>
__device__ void block_sort_by(unsigned long long* buf, int n, KeyFn key) {
  const int np = pow2_at_least(n);
  for (int i = threadIdx.x; i < np; i += blockDim.x)
    buf[i] = i < n ? (((unsigned long long)key(i) << 32) | (unsigned)i) : ~0ull;
  __syncthreads();
  block_bitonic_sort(buf, np);
}

__device__ __forceinline__ unsigned mix32(unsigned h) {
  h ^= h >> 16;
  h *= 0x85ebca6bu;
  h ^= h >> 13;
  h *= 0xc2b2ae35u;
  h ^= h >> 16;
  return h;
}

__device__ double block_sum(double v, double* s_red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) s_red[wid] = v;
  __syncthreads();
  if (wid == 0) {
    double t = s_red[lane];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    if (lane == 0) s_red[0] = t;
  }
  __syncthreads();
  const double r = s_red[0];
  __syncthreads();
  return r;
}

// ---- K1+K2 ------------------------------------------------------------------------------------------
// kRagged (ddn_align_views_ragged): the view's H, W and map offset come from the layout.
template <bool kRagged>
__device__ __forceinline__ void align_stats_body(const ddn_align_config& cfg, int H, int W, const float* __restrict__ depth,
                                                 const double* __restrict__ poses, const double* __restrict__ kmat,
                                                 const double* __restrict__ sparse_xyz, const int64_t* __restrict__ offsets,
                                                 const AlignWorkspace& ws, ddn_view_stats* __restrict__ stats, int sort_in_smem,
                                                 int pairs_in_smem, const int64_t* __restrict__ layout) {
  extern __shared__ __align__(16) unsigned long long s_sort[];
  __shared__ int s_warp[33];
  __shared__ double s_red[32];
  __shared__ float s_f[4];

  const int v = blockIdx.x;
  const int tid = threadIdx.x;
  if (kRagged) H = (int)layout[(size_t)v * DDN_LAYOUT_COLS], W = (int)layout[(size_t)v * DDN_LAYOUT_COLS + 1];
  const int64_t lo = offsets[v];
  const int n_sparse = (int)(offsets[v + 1] - lo);
  // The pair arrays of a view (sampled depth, COLMAP depth, ratio, table x / y) live in shared memory next to the
  // sort buffer when they fit (5 x 4 C bytes): the kernel is one long chain of block-wide phases, and every
  // phase that went through the global workspace paid an L2 round trip.  Only the final table goes out.
  float* const s_pairs = reinterpret_cast<float*>(s_sort + (sort_in_smem ? ws.Cp : 0));
  float* const gtx = ws.tx + (size_t)v * ws.C;
  float* const gty = ws.ty + (size_t)v * ws.C;
  float* zd = pairs_in_smem ? s_pairs : ws.zd + (size_t)v * ws.C;
  float* zc = pairs_in_smem ? s_pairs + ws.C : ws.zc + (size_t)v * ws.C;
  float* ratio = pairs_in_smem ? s_pairs + 2 * ws.C : ws.ratio + (size_t)v * ws.C;
  float* tx = pairs_in_smem ? s_pairs + 3 * ws.C : gtx;
  float* ty = pairs_in_smem ? s_pairs + 4 * ws.C : gty;
  unsigned long long* sortbuf = sort_in_smem ? s_sort : ws.sortbuf + (size_t)v * ws.Cp;
  const float* __restrict__ dmap = kRagged ? depth + layout[(size_t)v * DDN_LAYOUT_COLS + 2] : depth + (size_t)v * H * W;

  ddn_view_stats st;
  st.status = DDN_VIEW_REFINED;
  st.num_correspondences = 0;
  st.outliers_removed = 0;
  st.num_table = 0;
  st.scale_factor = 1.0f;
  st.affine_scale = 1.0f;
  st.affine_shift = 0.0f;
  st.reserved = 0;

  if (n_sparse <= 0) {
    if (tid == 0) {
      st.status = DDN_VIEW_NO_SPARSE;
      stats[v] = st;
    }
    return;
  }

  // float32 copies of pose and K (depth_refiner.py:233-236 casts inputs to self.dtype)
  float T[12], Kf[6];
#pragma unroll
  for (int i = 0; i < 12; ++i) T[i] = (float)poses[(size_t)v * 12 + i];
#pragma unroll
  for (int i = 0; i < 6; ++i) Kf[i] = (float)kmat[(size_t)v * 9 + i];
  const float m = (float)cfg.edge_margin;
  const float wlim = (float)(W - cfg.edge_margin), hlim = (float)(H - cfg.edge_margin);

  // -- A1 + A2: project, gate, bilinear sample, keep sampled > 0 (order preserving) --
  int n1 = 0;
  int any_inb = 0;
  for (int c0 = 0; c0 < n_sparse; c0 += kStatsThreads) {
    const int i = c0 + tid;
    bool keep = false;
    float samp = 0.f, z = 0.f;
    if (i < n_sparse) {
      const double* p = sparse_xyz + (size_t)(lo + i) * 3;
      const float x = (float)p[0], y = (float)p[1], zz = (float)p[2];
      const float cxm = fmaf(T[3], 1.f, fmaf(T[2], zz, fmaf(T[1], y, T[0] * x)));
      const float cym = fmaf(T[7], 1.f, fmaf(T[6], zz, fmaf(T[5], y, T[4] * x)));
      z = fmaf(T[11], 1.f, fmaf(T[10], zz, fmaf(T[9], y, T[8] * x)));
      float u = 0.f, w = 0.f;
      if (z > 0.f) {
        const float xn = __fdiv_rn(cxm, z), yn = __fdiv_rn(cym, z);
        u = __fadd_rn(fmaf(Kf[1], yn, Kf[0] * xn), Kf[2]);
        w = __fadd_rn(fmaf(Kf[4], yn, Kf[3] * xn), Kf[5]);
      }
      const bool inb = (u >= m) && (u < wlim) && (w >= m) && (w < hlim) && (z > 0.f);
      if (inb) {
        any_inb = 1;
        // grid_sample(bilinear, zeros, align_corners=True) at pixel coords (u, w): normalise and
        // un-normalise exactly as the reference + ATen do (depth_refiner.py:266-272)
        const float gx = __fadd_rn(__fmul_rn(__fdiv_rn(u, (float)(W - 1)), 2.f), -1.f);
        const float gy = __fadd_rn(__fmul_rn(__fdiv_rn(w, (float)(H - 1)), 2.f), -1.f);
        const float ix = __fmul_rn(__fdiv_rn(__fadd_rn(gx, 1.f), 2.f), (float)(W - 1));
        const float iy = __fmul_rn(__fdiv_rn(__fadd_rn(gy, 1.f), 2.f), (float)(H - 1));
        const float x0 = floorf(ix), y0 = floorf(iy);
        const float x1 = x0 + 1.f, y1 = y0 + 1.f;
        const float wnw = __fmul_rn(x1 - ix, y1 - iy), wne = __fmul_rn(ix - x0, y1 - iy);
        const float wsw = __fmul_rn(x1 - ix, iy - y0), wse = __fmul_rn(ix - x0, iy - y0);
        const int xi0 = (int)x0, yi0 = (int)y0, xi1 = xi0 + 1, yi1 = yi0 + 1;
        auto tap = [&](int xx, int yy) -> float {
          return (xx >= 0 && xx < W && yy >= 0 && yy < H) ? __ldg(dmap + (size_t)yy * W + xx) : 0.f;
        };
        // ATen's CPU kernel accumulates the four taps as one forward FMA chain (verified bit for bit
        // against F.grid_sample on the build host)
        samp = fmaf(tap(xi1, yi1), wse, fmaf(tap(xi0, yi1), wsw, fmaf(tap(xi1, yi0), wne, __fmul_rn(tap(xi0, yi0), wnw))));
        keep = samp > 0.f;
      }
    }
    const int slot = block_compact_slot(keep, n1, s_warp);
    if (slot >= 0) {
      zd[slot] = samp;
      zc[slot] = z;
    }
  }
  any_inb = __syncthreads_or(any_inb);
  if (n1 == 0) {
    if (tid == 0) {
      st.status = any_inb ? DDN_VIEW_NO_POSITIVE_SAMPLES : DDN_VIEW_NO_POINTS_IN_BOUNDS;
      stats[v] = st;
    }
    return;
  }
  __syncthreads();

  // -- A3: IQR rejection on r = z_colmap / (z_mono + 1e-6) --
  int n2 = n1;
  if (cfg.robust && n1 > 10) {
    for (int i = tid; i < n1; i += kStatsThreads) ratio[i] = __fdiv_rn(zc[i], __fadd_rn(zd[i], 1e-6f));
    __syncthreads();
    block_sort_by(sortbuf, n1, [&](int i) { return ordered_bits(ratio[i]); });
    if (tid == 0) {
      auto sorted = [&](int r) { return ratio[(unsigned)(sortbuf[r] & 0xffffffffu)]; };
      const float med = sorted((n1 - 1) >> 1);  // torch.median = lower median
      float q[2];
      const float qs[2] = {0.75f, 0.25f};
      for (int k = 0; k < 2; ++k) {  // torch.quantile, linear interpolation
        const float rank = __fmul_rn(qs[k], (float)(n1 - 1));
        const int rb = (int)rank;
        const int ra = (int)ceilf(rank);
        const float wgt = __fadd_rn(rank, -(float)rb);
        const float a = sorted(rb), b = sorted(ra);
        const float diff = __fadd_rn(b, -a);
        q[k] = (wgt < 0.5f) ? __fadd_rn(a, __fmul_rn(wgt, diff)) : __fadd_rn(b, -__fmul_rn(diff, __fadd_rn(1.f, -wgt)));
      }
      s_f[0] = med;
      s_f[1] = __fmul_rn(cfg.outlier_threshold, __fadd_rn(q[0], -q[1]));
    }
    __syncthreads();
    const float med = s_f[0], thr = s_f[1];
    n2 = 0;
    // in-place order-preserving compaction: slot <= i always, chunks processed in order
    for (int c0 = 0; c0 < n1; c0 += kStatsThreads) {
      const int i = c0 + tid;
      float a = 0.f, b = 0.f;
      bool keep = false;
      if (i < n1) {
        a = zd[i];
        b = zc[i];
        keep = fabsf(__fadd_rn(ratio[i], -med)) < thr;
      }
      const int slot = block_compact_slot(keep, n2, s_warp);  // contains __syncthreads
      if (slot >= 0) {
        zd[slot] = a;
        zc[slot] = b;
      }
      __syncthreads();
    }
    st.outliers_removed = n1 - n2;
  }
  st.num_correspondences = n2;
  if (n2 < cfg.min_correspondences || n2 == 0) {
    if (tid == 0) {
      st.status = DDN_VIEW_TOO_FEW;
      stats[v] = st;
    }
    return;
  }

  // -- A4: subsample to max_pairs with the hash permutation (replaces torch.randperm) --
  int n3 = n2;
  if (cfg.mode == 0 && cfg.adaptive_correspondences && n2 > cfg.max_pairs) {
    const unsigned seed = cfg.subsample_seed;
    block_sort_by(sortbuf, n2, [&](int i) { return mix32((unsigned)i ^ seed); });
    n3 = cfg.max_pairs;
    // gather in permutation order into ratio/tx as temporaries, then copy back
    for (int r = tid; r < n3; r += kStatsThreads) {
      const unsigned i = (unsigned)(sortbuf[r] & 0xffffffffu);
      ratio[r] = zd[i];
      tx[r] = zc[i];
    }
    __syncthreads();
    for (int r = tid; r < n3; r += kStatsThreads) {
      zd[r] = ratio[r];
      zc[r] = tx[r];
    }
    __syncthreads();
  }
  st.num_correspondences = n3;

  // -- A7: scale_factor = lower median of z_colmap / (z_mono + 1e-6) over the final pairs --
  for (int i = tid; i < n3; i += kStatsThreads) ratio[i] = __fdiv_rn(zc[i], __fadd_rn(zd[i], 1e-6f));
  __syncthreads();
  block_sort_by(sortbuf, n3, [&](int i) { return ordered_bits(ratio[i]); });
  if (tid == 0) st.scale_factor = ratio[(unsigned)(sortbuf[(n3 - 1) >> 1] & 0xffffffffu)];
  __syncthreads();

  if (cfg.mode == 1) {
    // -- N1: affine least squares from five float64 sums --
    double sd = 0, sz = 0, sdd = 0, sdz = 0;
    for (int i = tid; i < n3; i += kStatsThreads) {
      const double a = zd[i], b = zc[i];
      sd += a;
      sz += b;
      sdd += a * a;
      sdz += a * b;
    }
    sd = block_sum(sd, s_red);
    sz = block_sum(sz, s_red);
    sdd = block_sum(sdd, s_red);
    sdz = block_sum(sdz, s_red);
    if (tid == 0) {
      const double n = (double)n3;
      const double det = n * sdd - sd * sd;
      if (det > 0) {
        st.affine_scale = (float)((n * sdz - sd * sz) / det);
        st.affine_shift = (float)((sz * sdd - sd * sdz) / det);
      } else {
        st.status = DDN_VIEW_DEGENERATE_FIT;
      }
      stats[v] = st;
    }
    return;
  }

  // -- A5 (table part): pairs sorted by x = z_mono, ties by original order --
  block_sort_by(sortbuf, n3, [&](int i) { return ordered_bits(zd[i]); });
  for (int r = tid; r < n3; r += kStatsThreads) {
    const unsigned i = (unsigned)(sortbuf[r] & 0xffffffffu);
    const float x = zd[i], y = zc[i];
    tx[r] = x;
    ty[r] = y;
    if (pairs_in_smem) gtx[r] = x, gty[r] = y;  // K3 reads the table from the workspace
  }
  if (tid == 0) {
    st.num_table = n3;
    stats[v] = st;
  }
  if (n3 <= 0xffff) {  // bucket b -> [first knot with bucket >= b, first knot with bucket >= b + 1)
    __syncthreads();
    const float xmin = tx[0], scale = bucket_scale(xmin, tx[n3 - 1]);
    for (int b = tid; b < kBuckets; b += kStatsThreads) {
      int lo2[2];
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        int lo_ = 0, len = n3;
        while (len > 0) {
          const int half = len >> 1;
          const bool less = bucket_of(tx[lo_ + half], xmin, scale) < b + e;
          lo_ = less ? lo_ + half + 1 : lo_;
          len = less ? len - half - 1 : half;
        }
        lo2[e] = lo_;
      }
      ws.bucket[(size_t)v * kBuckets + b] = (uint32_t)lo2[0] | ((uint32_t)lo2[1] << 16);
    }
  }
}

__global__ void __launch_bounds__(kStatsThreads, 1)
align_stats_kernel(ddn_align_config cfg, int H, int W, const float* __restrict__ depth,
                   const double* __restrict__ poses, const double* __restrict__ kmat,
                   const double* __restrict__ sparse_xyz, const int64_t* __restrict__ offsets,
                   AlignWorkspace ws, ddn_view_stats* __restrict__ stats, int sort_in_smem, int pairs_in_smem) {
  align_stats_body<false>(cfg, H, W, depth, poses, kmat, sparse_xyz, offsets, ws, stats, sort_in_smem, pairs_in_smem, nullptr);
}

__global__ void __launch_bounds__(kStatsThreads, 1)
align_stats_ragged_kernel(ddn_align_config cfg, const int64_t* __restrict__ layout, const float* __restrict__ depth,
                          const double* __restrict__ poses, const double* __restrict__ kmat,
                          const double* __restrict__ sparse_xyz, const int64_t* __restrict__ offsets,
                          AlignWorkspace ws, ddn_view_stats* __restrict__ stats, int sort_in_smem, int pairs_in_smem) {
  align_stats_body<true>(cfg, 0, 0, depth, poses, kmat, sparse_xyz, offsets, ws, stats, sort_in_smem, pairs_in_smem, layout);
}

// ---- K3 ---------------------------------------------------------------------------------------------
// One CTA = a 128 x 32 pixel tile (+1 replicate halo) of one view.  Phase 1 remaps tile + halo into
// shared memory (lookup table and its bucket index also in shared memory); phase 2 takes the 3x3 median
// with a sliding window down each column: the three values of a row are sorted once and reused by the
// three windows that contain them (median9 = med3(max of the minima, med3 of the middles, min of the
// maxima)), 3 LDS and ~20 min/max per pixel instead of 9 LDS and 38.
constexpr int kTileW = 126, kTileH = 32, kRemapThreads = 256;
static_assert(kTileW == kRemapTileW && kTileH == kRemapTileH, "the ragged layout counts tiles of kRemapTileW x kRemapTileH");
constexpr int kHaloW = kTileW + 2, kHaloH = kTileH + 2;
constexpr int kLutSmemMax = 4096;  // knots kept in shared memory (32 KB); larger tables read global

__device__ __forceinline__ float med3(float a, float b, float c) { return fmaxf(fminf(a, b), fminf(fmaxf(a, b), c)); }

__device__ __forceinline__ float pwl_interp(float d, float x0, float x1, float y0, float y1) {
  float dx = __fadd_rn(x1, -x0);
  dx = dx == 0.f ? 1e-6f : dx;
  float t = __fdiv_rn(__fadd_rn(d, -x0), dx);
  t = fminf(fmaxf(t, 0.f), 1.f);
  return fmaxf(__fadd_rn(y0, __fmul_rn(t, __fadd_rn(y1, -y0))), 1e-3f);
}

// i = clamp(searchsorted_left(xs, d), 1, n-1)  (depth_refiner.py:157-158), binary search
__device__ __forceinline__ float pwl_eval(float d, const float* __restrict__ xs, const float* __restrict__ ys, int n) {
  int lo = 0, len = n;
  while (len > 0) {
    const int half = len >> 1;
    const bool less = xs[lo + half] < d;
    lo = less ? lo + half + 1 : lo;
    len = less ? len - half - 1 : half;
  }
  const int i = min(max(lo, 1), n - 1);
  return pwl_interp(d, xs[i - 1], xs[i], ys[i - 1], ys[i]);
}

// same result through the bucket index: a short linear scan inside d's bucket
__device__ __forceinline__ float pwl_eval_bucketed(float d, const float* __restrict__ xs, const float* __restrict__ ys,
                                                   int n, const uint32_t* __restrict__ bucket, float xmin, float scale) {
  const uint32_t se = bucket[bucket_of(d, xmin, scale)];
  int i = (int)(se & 0xffffu);
  const int end = (int)(se >> 16);
  while (i < end && xs[i] < d) ++i;
  i = min(max(i, 1), n - 1);
  return pwl_interp(d, xs[i - 1], xs[i], ys[i - 1], ys[i]);
}

// Bounding-box epilogue of K3 (called by every thread of the CTA, after a block barrier that made the
// s_dmin / s_dmax initialisation visible).  Every pixel (x, y) of the tile with refined depth d > 0 back-projects
// to X = d * (a x + b y + c) + t per axis - affine in d for a fixed pixel and affine in (x, y) for a fixed d - so all
// points of the tile lie inside the box of the 8 corners {x0, x1} x {y0, y1} x {dmin, dmax}.  The tile's points cost
// two min/max per pixel instead of a full back-projection; the box is a superset of the true one by at most the
// tile's own extent at its largest depth.
__device__ __forceinline__ void tile_bbox_epilogue(int* __restrict__ bbox, const float* __restrict__ src_table, int v, int tx0,
                                                   int ty0, int W, int H, int t_dmin, int t_dmax, int* s_dmin, int* s_dmax) {
  if (bbox == nullptr) return;  // uniform
  const int lo = __reduce_min_sync(0xffffffffu, t_dmin), hi = __reduce_max_sync(0xffffffffu, t_dmax);
  if ((threadIdx.x & 31) == 0 && hi > 0) {
    atomicMin(s_dmin, lo);
    atomicMax(s_dmax, hi);
  }
  __syncthreads();
  if (threadIdx.x != 0 || *s_dmax <= 0) return;
  const float* s = src_table + (size_t)v * 16;
  float row[12];
#pragma unroll
  for (int i = 0; i < 12; ++i) row[i] = __ldg(s + i);
  const float dlim[2] = {__int_as_float(*s_dmin), __int_as_float(*s_dmax)};
  const float xs[2] = {(float)tx0, (float)(min(tx0 + kTileW, W) - 1)};
  const float ys[2] = {(float)ty0, (float)(min(ty0 + kTileH, H) - 1)};
  float bmin[3] = {INFINITY, INFINITY, INFINITY}, bmax[3] = {-INFINITY, -INFINITY, -INFINITY};
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    const float d = dlim[c & 1], x = xs[(c >> 1) & 1], y = ys[c >> 2];
    float p[3];
    backproject_pqd(row, d * x, d * y, d, p[0], p[1], p[2]);
#pragma unroll
    for (int i = 0; i < 3; ++i) bmin[i] = fminf(bmin[i], p[i]), bmax[i] = fmaxf(bmax[i], p[i]);
  }
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    atomicMin(bbox + i, float_to_ordered(bmin[i]));
    atomicMax(bbox + 3 + i, float_to_ordered(bmax[i]));
  }
}

#ifndef DDN_K3_MINB
#define DDN_K3_MINB 8
#endif
// kPacked: the mask is one bit per pixel; kBox: the bounding-box epilogue is on.  Template parameters, not run-time
// flags: the kernel is bound by instruction issue, and a per-pixel branch on either costs 5 % (measured).
// kTma (ddn_align_config.use_tma): the depth tile arrives through ONE cp.async.bulk.tensor (TMA, SASS UTMALDG), is
// remapped in place, and halo positions outside the image take the value of the clamped pixel afterwards (TMA
// zero-fills elements past the far edges; the remap is pointwise, so copying the remapped neighbour is the replicate
// padding).  A tensor copy faults ("illegal instruction") when a start coordinate is negative or the innermost one is
// not a multiple of 16 bytes (scripts/experiments/tma_min2.cu, profiles/r02_tma_min2.log), and the halo starts one pixel
// left of a 126-pixel tile, so the box is 132 x 34: it starts at the 4-pixel boundary at or below max(tx0 - 1, 0), row
// max(ty0 - 1, 0), and the kernel indexes it with the tile's own column / row offset (-1..3 / -1..0; a guard band in
// front of the box takes the two negative cases, whose positions lie outside the image and are filled by the replicate
// pass).  Needs 16-byte multiples for the row pitch, i.e. W % 4 == 0 - cfg 2's 1297-pixel rows do not qualify.
constexpr int kTmaBoxW = 132;                                // 128 halo columns + up to 3 columns of alignment slack, x4 B = 528 B
constexpr int kTmaGuard = 160;                               // floats in front of the box (>= one row + 1; 640 B keeps 128-B alignment)
constexpr int kTmaFloats = kTmaGuard + kHaloH * kTmaBoxW;    // 18,592 B
// kRagged (ddn_align_views_ragged, byte mask, no TMA; layout = the device layout, nullptr otherwise): blockIdx.x runs
// over the tiles of all views; a CTA finds its view from the layout's tile prefix (tiles_y = the number of views) and
// takes H, W, tiles_x and the map offset from there.
template <bool kPacked, bool kBox, bool kTma, bool kRagged>
__global__ void __launch_bounds__(kRemapThreads, DDN_K3_MINB)
remap_median_kernel(ddn_align_config cfg, int H, int W, int tiles_x, int tiles_y, const float* __restrict__ depth,
                    const uint8_t* __restrict__ mask, const ddn_view_stats* __restrict__ stats, AlignWorkspace ws,
                    float* __restrict__ refined, int lut_cap, const float* __restrict__ src_table, int* __restrict__ bbox,
                    const CUtensorMap* __restrict__ depth_map, const int64_t* __restrict__ layout) {
  static_assert(!kRagged || (!kPacked && !kTma), "the ragged remap reads a byte mask with plain loads");
  extern __shared__ __align__(16) float s_dyn[];  // LUT xs | ys | bucket index (when the table fits)
  __shared__ __align__(128) float s_buf[kTma ? kTmaFloats : kHaloH * kHaloW];
  __shared__ __align__(8) unsigned long long s_bar;  // mbarrier of the TMA load (kTma)
  __shared__ uint8_t s_msk[kHaloH][kHaloW + 2];
  // bounding-box epilogue: smallest / largest positive refined depth of the tile (bits of positive floats order as ints)
  __shared__ int s_dmin, s_dmax;
  int t_dmin = 0x7f800000, t_dmax = 0;
  auto fold_depth = [&](float v) {
    if (!kBox) return;
    const int b = __float_as_int(v);
    t_dmax = max(t_dmax, b);
    t_dmin = min(t_dmin, v > 0.f ? b : 0x7f800000);
  };
  if (threadIdx.x == 0) s_dmin = 0x7f800000, s_dmax = 0;

  const int tid = threadIdx.x;
  const int vr = kRagged ? layout_view_of(layout, tiles_y, 4, blockIdx.x) : 0;  // ragged: the view of this tile
  const int64_t* __restrict__ L = layout + (size_t)vr * DDN_LAYOUT_COLS;
  if (kRagged) H = (int)L[0], W = (int)L[1], tiles_x = (W + kTileW - 1) / kTileW;
  const int tile = kRagged ? (int)(blockIdx.x - L[4]) : blockIdx.x;
  const int v = kRagged ? vr : blockIdx.y;
  const int ty0 = (tile / tiles_x) * kTileH, tx0 = (tile % tiles_x) * kTileW;
  const size_t HW = (size_t)H * W;
  const float* __restrict__ dmap = kRagged ? depth + L[2] : depth + (size_t)v * HW;
  // mask: one byte per pixel, or (cfg.mask_packed) one BIT per pixel - bit (g & 7) of byte g >> 3 of the view's
  // ceil(H W / 8) bytes: an eighth of the upload for the host path
  const uint8_t* __restrict__ mmap = mask ? (kRagged ? mask + L[2] : mask + (size_t)v * (kPacked ? (HW + 7) / 8 : HW)) : nullptr;
  auto mask_at = [&](size_t g) -> bool { return kPacked ? ((__ldg(mmap + (g >> 3)) >> (g & 7)) & 1) != 0 : __ldg(mmap + g) != 0; };
  float* __restrict__ out = kRagged ? refined + L[2] : refined + (size_t)v * HW;
  const ddn_view_stats st = stats[v];

  if (st.status != DDN_VIEW_REFINED) {
    // Views the reference returns unchanged (or skips): copy / zero, no remap.
    for (int i = tid; i < kTileW * kTileH; i += kRemapThreads) {
      const int y = ty0 + i / kTileW, x = tx0 + i % kTileW;
      if (y < H && x < W) {
        const size_t g = (size_t)y * W + x;
        float d = dmap[g];
        if (st.status == DDN_VIEW_NO_SPARSE) d = 0.f;
        else if (cfg.zero_unmasked_passthrough && !(mmap ? mask_at(g) : d > 0.f)) d = 0.f;
        out[g] = d;
        fold_depth(d);
      }
    }
    __syncthreads();
    if (kBox) tile_bbox_epilogue(bbox, src_table, v, tx0, ty0, W, H, t_dmin, t_dmax, &s_dmin, &s_dmax);
    return;
  }

  // halo position (hy, hx) <-> pixel (ty0 - 1 + hy, tx0 - 1 + hx); with TMA the box starts at (by0, bx0) instead
  const int bx0 = max(tx0 - 1, 0) & ~3, by0 = max(ty0 - 1, 0);
  const int val_base = kTma ? kTmaGuard + (ty0 - 1 - by0) * kTmaBoxW + (tx0 - 1 - bx0) : 0;
  constexpr int kValPitch = kTma ? kTmaBoxW : kHaloW;
  auto val_at = [&](int hy, int hx) -> float& { return s_buf[val_base + hy * kValPitch + hx]; };
  if (kTma) {
    const uint32_t bar = (uint32_t)__cvta_generic_to_shared(&s_bar), dst = (uint32_t)__cvta_generic_to_shared(s_buf + kTmaGuard);
    if (tid == 0) {
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar) : "memory");
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (tid == 0) {  // the whole box in one request; elements past the right / bottom edge of the image arrive as zeros
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"((uint32_t)(kTmaBoxW * kHaloH * 4)) : "memory");
      asm volatile(
          "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(dst),
          "l"(reinterpret_cast<uint64_t>(depth_map)), "r"(bx0), "r"(by0), "r"(v), "r"(bar)
          : "memory");
    }
  }
  const int n = st.num_table;
  const float* gxs = ws.tx + (size_t)v * ws.C;
  const float* gys = ws.ty + (size_t)v * ws.C;
  const bool bucketed = cfg.mode == 0 && n >= 2 && n <= lut_cap;
  float* const sx = s_dyn;  // shared-memory copies (only valid when `bucketed`)
  float* const sy = s_dyn + lut_cap;
  uint32_t* const sb = reinterpret_cast<uint32_t*>(s_dyn + 2 * lut_cap);
  float xmin = 0.f, bscale = 0.f;
  if (bucketed) {
    for (int i = tid; i < n; i += kRemapThreads) {
      sx[i] = gxs[i];
      sy[i] = gys[i];
    }
    for (int i = tid; i < kBuckets; i += kRemapThreads) sb[i] = ws.bucket[(size_t)v * kBuckets + i];
    xmin = gxs[0];
    bscale = bucket_scale(xmin, gxs[n - 1]);
    __syncthreads();
  }
  const float a_s = st.affine_scale, a_t = st.affine_shift;

  // phase 1: remap tile + 1-pixel replicate halo into shared memory.  The halo is exactly 128 wide: a thread owns
  // halo column hx (clamp hoisted) and every second halo row - no index division, no idle lanes.
  static_assert(kHaloW == 128 && kRemapThreads == 256, "phase 1 maps two halo rows per pass");
  if (kTma) {  // phase 0 of the barrier completes when the box's 17,952 bytes have landed
    const uint32_t bar = (uint32_t)__cvta_generic_to_shared(&s_bar);
    uint32_t ok = 0;
    do {
      asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                   : "=r"(ok)
                   : "r"(bar)
                   : "memory");
    } while (!ok);
  }
  {
    const int hx = tid & (kHaloW - 1);
    const int x = min(max(tx0 + hx - 1, 0), W - 1);
#pragma unroll 1
    for (int hy = tid >> 7; hy < kHaloH; hy += 2) {
      const int y = min(max(ty0 + hy - 1, 0), H - 1);
      const int g = y * W + x;
      if (kTma && (x != tx0 + hx - 1 || y != ty0 + hy - 1)) continue;  // outside the image: filled in below
      const float d = kTma ? val_at(hy, hx) : __ldg(dmap + g);
      const bool mk = mmap ? mask_at((size_t)g) : (d > 0.f);
      float val = 0.f;
      if (mk) {
        if (bucketed) val = pwl_eval_bucketed(d, sx, sy, n, sb, xmin, bscale);
        else if (cfg.mode == 0) val = (n >= 2) ? pwl_eval(d, gxs, gys, n) : __fmul_rn(d, __fdiv_rn(gys[0], __fadd_rn(gxs[0], 1e-6f)));
        else val = fmaxf(__fadd_rn(__fmul_rn(d, a_s), a_t), 1e-3f);
      }
      val_at(hy, hx) = val;
      s_msk[hy][hx] = mk ? 1 : 0;
    }
    if (kTma) {  // replicate padding: positions outside the image <- the (remapped) clamped pixel, which is inside the tile
      __syncthreads();
#pragma unroll 1
      for (int hy = tid >> 7; hy < kHaloH; hy += 2) {
        const int y = min(max(ty0 + hy - 1, 0), H - 1);
        if (x != tx0 + hx - 1 || y != ty0 + hy - 1) {
          const int cx = x - (tx0 - 1), cy = y - (ty0 - 1);
          val_at(hy, hx) = val_at(cy, cx);
          s_msk[hy][hx] = s_msk[cy][cx];
        }
      }
    }
  }
  __syncthreads();

  // phase 2: column lx, rows [ly0, ly0 + 16)
  const int lx = tid & (kHaloW - 1);
  const int x = tx0 + lx;
  const bool active = lx < kTileW && x < W;
  constexpr int kRowsPerThread = kTileH / (kRemapThreads / kHaloW);
  const int ly0 = (tid / kHaloW) * kRowsPerThread;
  if (active && cfg.skip_smoothing) {
#pragma unroll 4
    for (int r = 0; r < kRowsPerThread; ++r) {
      const int y = ty0 + ly0 + r;
      if (y >= H) break;
      const float o = s_msk[ly0 + r + 1][lx + 1] ? val_at(ly0 + r + 1, lx + 1) : 0.f;
      out[(size_t)y * W + x] = o;
      fold_depth(o);
    }
  } else if (active) {
    float lo[3], mi[3], hi[3];
    auto load_row = [&](int hy, int slot) {
      float a = val_at(hy, lx), b = val_at(hy, lx + 1), c = val_at(hy, lx + 2);
      const float ab_lo = fminf(a, b), ab_hi = fmaxf(a, b);
      lo[slot] = fminf(ab_lo, c);
      hi[slot] = fmaxf(ab_hi, c);
      mi[slot] = fmaxf(ab_lo, fminf(ab_hi, c));
    };
    load_row(ly0, 0);
    load_row(ly0 + 1, 1);
#pragma unroll
    for (int r = 0; r < kRowsPerThread; ++r) {
      const int y = ty0 + ly0 + r;
      if (y >= H) break;
      load_row(ly0 + r + 2, (r + 2) % 3);
      float o = med3(fmaxf(fmaxf(lo[0], lo[1]), lo[2]), med3(mi[0], mi[1], mi[2]), fminf(fminf(hi[0], hi[1]), hi[2]));
      o = s_msk[ly0 + r + 1][lx + 1] ? o : 0.f;
      out[(size_t)y * W + x] = o;
      fold_depth(o);
    }
  }
  if (kBox) tile_bbox_epilogue(bbox, src_table, v, tx0, ty0, W, H, t_dmin, t_dmax, &s_dmin, &s_dmax);
}

// What an alignment call derives from its config and sparse-point bound: the carved workspace, where K1+K2 sort and keep
// their pairs (shared or global memory), and how much of K3's lookup table sits in shared memory (lut = 0: none).
struct AlignPlan {
  AlignWorkspace ws;
  int in_smem, pairs_smem, lut;
  size_t smem_sort, smem_lut;
};

// The checks and sizes both entry points share, after each has checked its shapes or layout.  With no views it checks
// the config only and plans nothing.
static int plan_align(const ddn_align_config* cfg, int64_t n_views, const float* depth, const double* cam_from_world,
                      const double* kmat, const int64_t* sparse_offsets, const float* refined, const ddn_view_stats* stats,
                      int64_t max_sparse_per_view, void* workspace, int64_t workspace_bytes, const float* src_table,
                      const float* bbox, AlignPlan& p) {
  DDN_REQUIRE(cfg != nullptr, "null config");
  DDN_REQUIRE((src_table == nullptr) == (bbox == nullptr), "src_table and bbox go together");
  DDN_REQUIRE(cfg->mode == 0 || cfg->mode == 1, "mode");
  DDN_REQUIRE(cfg->max_pairs >= 1, "max_pairs");
  if (n_views == 0) return DDN_OK;
  DDN_REQUIRE(depth && cam_from_world && kmat && sparse_offsets && refined && stats && workspace, "null pointer");
  const int64_t C = max_sparse_per_view > 0 ? max_sparse_per_view : 1;
  DDN_REQUIRE(C < (1ll << 30), "max_sparse_per_view");
  if (workspace_bytes < align_ws_bytes(n_views, C)) {
    set_error("align workspace too small: %lld < %lld", (long long)workspace_bytes, (long long)align_ws_bytes(n_views, C));
    return DDN_ERR_WORKSPACE_TOO_SMALL;
  }
  p.ws = carve(workspace, n_views, C);
  p.in_smem = p.ws.Cp <= kSortSmemMax ? 1 : 0;
  p.pairs_smem = (p.in_smem && (size_t)p.ws.Cp * 8 + (size_t)p.ws.C * 20 <= 200 * 1024) ? 1 : 0;
  p.smem_sort = (p.in_smem ? (size_t)p.ws.Cp * 8 : 0) + (p.pairs_smem ? (size_t)p.ws.C * 20 : 0);
  // largest table any view can have: max_pairs when subsampling, else every surviving pair
  int64_t lut = (cfg->adaptive_correspondences && cfg->max_pairs < C) ? cfg->max_pairs : C;
  if (cfg->mode != 0 || lut > kLutSmemMax) lut = 0;  // affine mode has no table; huge tables stay in global
  p.lut = (int)lut;
  p.smem_lut = lut > 0 ? (size_t)lut * 8 + (size_t)kBuckets * 4 : 0;
  return DDN_OK;
}

template <bool kPacked, bool kBox, bool kTma, bool kRagged>
static int launch_remap(const ddn_align_config& cfg, const AlignPlan& p, dim3 grid, int H, int W, int tiles_x, int tiles_y,
                        const float* depth, const uint8_t* mask, const ddn_view_stats* stats, float* refined,
                        const float* src_table, float* bbox, const CUtensorMap* depth_map, const int64_t* layout, cudaStream_t st) {
  DDN_TRY(check_cuda(cudaFuncSetAttribute(remap_median_kernel<kPacked, kBox, kTma, kRagged>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          (int)p.smem_lut),
                     "cudaFuncSetAttribute(remap_median)"));
  remap_median_kernel<kPacked, kBox, kTma, kRagged><<<grid, kRemapThreads, p.smem_lut, st>>>(
      cfg, H, W, tiles_x, tiles_y, depth, mask, stats, p.ws, refined, p.lut, src_table, reinterpret_cast<int*>(bbox), depth_map, layout);
  return after_launch("remap_median_kernel", st);
}

}  // namespace ddn

extern "C" {

int ddn_align_workspace_bytes(int64_t n_views, int64_t max_sparse_per_view, int64_t* bytes_out) {
  using namespace ddn;
  DDN_REQUIRE(bytes_out != nullptr, "null bytes_out");
  DDN_REQUIRE(n_views >= 0 && max_sparse_per_view >= 0, "negative size");
  *bytes_out = align_ws_bytes(n_views, max_sparse_per_view > 0 ? max_sparse_per_view : 1);
  return DDN_OK;
}

int ddn_align_views(const ddn_align_config* cfg, int64_t n_views, int64_t height, int64_t width,
                    const float* depth, const uint8_t* mask, const double* cam_from_world,
                    const double* kmat, const double* sparse_xyz, const int64_t* sparse_offsets,
                    int64_t max_sparse_per_view, float* refined, ddn_view_stats* stats,
                    void* workspace, int64_t workspace_bytes, const float* src_table, float* bbox, void* stream) {
  using namespace ddn;
  DDN_REQUIRE(n_views >= 0 && height > 1 && width > 1, "shape");
  DDN_REQUIRE(height * width < (1ll << 31), "image too large");
  DDN_REQUIRE(n_views <= 65535, "too many views per call");
  AlignPlan p;
  DDN_TRY(plan_align(cfg, n_views, depth, cam_from_world, kmat, sparse_offsets, refined, stats, max_sparse_per_view, workspace,
                     workspace_bytes, src_table, bbox, p));
  if (n_views == 0) return DDN_OK;
  const bool tma = cfg->use_tma != 0;
  if (tma) {  // tensor-copy form of the remap kernel: checked before anything is launched
    DDN_REQUIRE(width % 4 == 0 && ((uintptr_t)depth & 15) == 0, "use_tma needs W % 4 == 0 and a 16-byte aligned depth pointer");
    DDN_REQUIRE(width >= kTmaBoxW && height >= kHaloH, "use_tma needs an image of at least 132 x 34 pixels");
  }
  cudaStream_t st = (cudaStream_t)stream;
  DDN_TRY(check_cuda(cudaFuncSetAttribute(align_stats_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem_sort),
                     "cudaFuncSetAttribute(align_stats)"));
  align_stats_kernel<<<(unsigned)n_views, kStatsThreads, p.smem_sort, st>>>(*cfg, (int)height, (int)width, depth,
                                                                           cam_from_world, kmat, sparse_xyz,
                                                                           sparse_offsets, p.ws, stats, p.in_smem, p.pairs_smem);
  DDN_TRY(after_launch("align_stats_kernel", st));
  const int tiles_x = (int)((width + kTileW - 1) / kTileW), tiles_y = (int)((height + kTileH - 1) / kTileH);
  dim3 grid((unsigned)(tiles_x * tiles_y), (unsigned)n_views);
  CUtensorMap depth_map;
  memset(&depth_map, 0, sizeof(depth_map));
  if (tma) {
    typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                 const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                 CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    DDN_TRY(check_cuda(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres), "cudaGetDriverEntryPoint"));
    DDN_REQUIRE(fn != nullptr && qres == cudaDriverEntryPointSuccess, "cuTensorMapEncodeTiled not available");
    const cuuint64_t dims[3] = {(cuuint64_t)width, (cuuint64_t)height, (cuuint64_t)n_views};
    const cuuint64_t strides[2] = {(cuuint64_t)width * 4, (cuuint64_t)width * (cuuint64_t)height * 4};
    const cuuint32_t box[3] = {(cuuint32_t)kTmaBoxW, (cuuint32_t)kHaloH, 1};
    const cuuint32_t estr[3] = {1, 1, 1};
    const CUresult r = ((EncodeFn)fn)(&depth_map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(depth), dims, strides, box, estr,
                                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
      set_error("cuTensorMapEncodeTiled failed: %d", (int)r);
      return DDN_ERR_CUDA;
    }
    DDN_TRY(check_cuda(cudaMemcpyAsync(p.ws.tensor_map, &depth_map, sizeof(depth_map), cudaMemcpyHostToDevice, st), "tensor map upload"));
  }
  const bool packed = cfg->mask_packed != 0 && mask != nullptr, with_box = bbox != nullptr;
  const auto launch = packed ? (with_box ? (tma ? &launch_remap<true, true, true, false> : &launch_remap<true, true, false, false>)
                                         : (tma ? &launch_remap<true, false, true, false> : &launch_remap<true, false, false, false>))
                             : (with_box ? (tma ? &launch_remap<false, true, true, false> : &launch_remap<false, true, false, false>)
                                         : (tma ? &launch_remap<false, false, true, false> : &launch_remap<false, false, false, false>));
  return launch(*cfg, p, grid, (int)height, (int)width, tiles_x, tiles_y, depth, mask, stats, refined, src_table, bbox,
                reinterpret_cast<const CUtensorMap*>(p.ws.tensor_map), nullptr, st);
}

int ddn_align_views_ragged(const ddn_align_config* cfg, int64_t n_views, const int64_t* layout, const int64_t* layout_host,
                           const float* depth, const uint8_t* mask, const double* cam_from_world, const double* kmat,
                           const double* sparse_xyz, const int64_t* sparse_offsets, int64_t max_sparse_per_view, float* refined,
                           ddn_view_stats* stats, void* workspace, int64_t workspace_bytes, const float* src_table, float* bbox,
                           void* stream) {
  using namespace ddn;
  DDN_REQUIRE(layout != nullptr, "null layout");
  DDN_TRY(check_layout(n_views, layout_host));
  for (int64_t v = 0; v < n_views; ++v)
    DDN_REQUIRE(layout_host[v * DDN_LAYOUT_COLS] > 1 && layout_host[v * DDN_LAYOUT_COLS + 1] > 1, "every view needs H, W >= 2");
  AlignPlan p;
  DDN_TRY(plan_align(cfg, n_views, depth, cam_from_world, kmat, sparse_offsets, refined, stats, max_sparse_per_view, workspace,
                     workspace_bytes, src_table, bbox, p));
  if (cfg->mask_packed || cfg->use_tma) {
    set_error("ddn_align_views_ragged: mask_packed and use_tma are options of the uniform ddn_align_views only");
    return DDN_ERR_UNSUPPORTED;
  }
  cudaStream_t st = (cudaStream_t)stream;
  DDN_TRY(check_cuda(cudaFuncSetAttribute(align_stats_ragged_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem_sort),
                     "cudaFuncSetAttribute(align_stats_ragged)"));
  align_stats_ragged_kernel<<<(unsigned)n_views, kStatsThreads, p.smem_sort, st>>>(*cfg, layout, depth, cam_from_world, kmat, sparse_xyz,
                                                                                  sparse_offsets, p.ws, stats, p.in_smem, p.pairs_smem);
  DDN_TRY(after_launch("align_stats_ragged_kernel", st));
  const unsigned tiles = (unsigned)layout_host[n_views * DDN_LAYOUT_COLS + 4];
  const auto launch = bbox != nullptr ? &launch_remap<false, true, false, true> : &launch_remap<false, false, false, true>;
  return launch(*cfg, p, dim3(tiles), 0, 0, 1, (int)n_views, depth, mask, stats, refined, src_table, bbox, nullptr, layout, st);
}

}  // extern "C"
