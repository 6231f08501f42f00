// Stages 2+3: fused pixel back-projection and multi-view consistency vote (kernel K4), plus the
// float64 set-up kernel that turns poses into per-(source view, neighbour) float32 tables.
//
// Reference semantics (see include/ddn_b200.h): scripts/test.py:79-90, 205-233 (back-projection),
// scripts/test.py:58-76, 273-330 (reproject, grazing gate, truncating lookup, one-sided floater vote).
//
// HBM-bound design (no dense contraction anywhere on this path, so no tensor cores):
//   * one CTA owns 256*PX consecutive pixels of ONE source view, so the K neighbour tables are
//     CTA-uniform and live in shared memory;
//   * xyz out is AoS float3: it moves through a shared staging buffer as float4 vectors (fully
//     coalesced 16 B per lane) and is written per pixel with stride-3 STS (conflict free); the
//     normal map is only read for vote candidates (rare), not streamed;
//   * pixel groups without any point (sky, masked regions - contiguous in practice) are skipped per
//     warp;
//   * neighbour depth gathers go through the read-only path; consecutive lanes hit consecutive
//     pixels of the neighbour map, and CTAs are scheduled view by view so the K neighbour maps of
//     the views in flight stay L2 resident;
//   * float->int truncation uses FADD.RZ with 2^23 instead of F2I (keeps the XU pipe free for the
//     one MUFU.RCP and one MUFU.SQRT per pair).
#include <string.h>

#include "fuse_common.cuh"

namespace ddn {

#ifndef DDN_K4_MINBLOCKS
#define DDN_K4_MINBLOCKS 5
#endif
#ifndef DDN_K4_SUPPORT_MINBLOCKS
#define DDN_K4_SUPPORT_MINBLOCKS 4
#endif
constexpr int kFilterThreads = 256;
#ifndef DDN_K4_PX
#define DDN_K4_PX 4
#endif
constexpr int kFilterPX = DDN_K4_PX;  // pixels per thread
constexpr int kFilterChunk = kFilterThreads * kFilterPX;
static_assert(kFilterChunk == kFilterChunkPoints, "the ragged layout counts chunks of kFilterChunkPoints points");

// ------------------------------------------------------------------------------------------------
// Table set-up (float64, one thread per (source view, neighbour))
// pair_table[s][k][24]: rows 0..2 of K_t [M | t_ts], M = R_t R_s^T Kinv_s (12 floats) - i.e. the pixel
//   (x, y) at depth d maps to (U, V, Z) = rows * (d x, d y, d, 1) and lands at u = U/Z, v = V/Z;
//   camera centre of t (3), target view index (int bits), fx_t fy_t cx_t cy_t, own-view flag, and (float 21,
//   uint bits) K4's gather offset of the entry: t*H*W - 0x4B000000*(W+1) mod 2^32 (see pair_gather).
//   The entries of a source view are COMPACTED: valid neighbours other than the view itself first
//   (n_hot of them, in table order), then the n_own entries of the view itself (only the
//   reference-parity table K = V lists it); entry 0 carries n_hot and n_own in floats 22, 23 (int bits).  K4's hot loop therefore runs over n_hot entries without any validity test.
// src_table[s][16]: rows of R_s^T Kinv_s with c_s appended (12 floats), cx_s, cy_s, fx_s, fy_s.
// ------------------------------------------------------------------------------------------------
// kRagged (ddn_build_pair_tables_ragged): the views' sizes and offsets come from the layout, and floats 16-19 describe
// the neighbour's map instead of its intrinsics (K4 never reads those).
template <bool kRagged>
__device__ __forceinline__ void build_pair_tables_body(int n_total, int src_begin, int n_src, int k_nbr, unsigned hw, unsigned width,
                                                       const double* __restrict__ poses, const double* __restrict__ intr,
                                                       const int32_t* __restrict__ nbr, float* __restrict__ pair_table,
                                                       float* __restrict__ src_table, const int64_t* __restrict__ layout) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  int n_pairs = n_src * k_nbr;
  if (idx >= n_pairs + n_src) return;
  const bool is_src_row = idx >= n_pairs;
  const int sl = is_src_row ? idx - n_pairs : idx / k_nbr;
  const int s = src_begin + sl;
  const double* Ps = poses + (size_t)s * 12;
  const double fx = intr[s * 4 + 0], fy = intr[s * 4 + 1], cx = intr[s * 4 + 2], cy = intr[s * 4 + 3];
  // Kinv_s columns: (1/fx, 0, 0), (0, 1/fy, 0), (-cx/fx, -cy/fy, 1)
  double Rs[3][3], ts[3];
  for (int i = 0; i < 3; ++i) {
    for (int j = 0; j < 3; ++j) Rs[i][j] = Ps[i * 4 + j];
    ts[i] = Ps[i * 4 + 3];
  }
  if (is_src_row) {
    float* o = src_table + (size_t)sl * 16;
    for (int i = 0; i < 3; ++i) {
      // row i of R_s^T: (Rs[0][i], Rs[1][i], Rs[2][i]);  c_s = -R_s^T t_s
      double r0 = Rs[0][i], r1 = Rs[1][i], r2 = Rs[2][i];
      o[i * 4 + 0] = (float)(r0 / fx);
      o[i * 4 + 1] = (float)(r1 / fy);
      o[i * 4 + 2] = (float)(-r0 * cx / fx - r1 * cy / fy + r2);
      o[i * 4 + 3] = (float)(-(r0 * ts[0] + r1 * ts[1] + r2 * ts[2]));
    }
    o[12] = (float)cx;
    o[13] = (float)cy;
    o[14] = (float)fx;
    o[15] = (float)fy;
    return;
  }
  const int k = idx - sl * k_nbr;
  const int32_t* row = nbr + (size_t)s * k_nbr;
  const int t = row[k];
  int n_hot = 0, n_own = 0, hot_before = 0, own_before = 0;
  for (int q = 0; q < k_nbr; ++q) {
    const int tq = row[q];
    const bool own = tq == s, hot = tq >= 0 && tq < n_total && !own;
    n_hot += hot ? 1 : 0;
    n_own += own ? 1 : 0;
    hot_before += (hot && q < k) ? 1 : 0;
    own_before += (own && q < k) ? 1 : 0;
  }
  if (k == 0) {
    float* e0 = pair_table + (size_t)sl * k_nbr * DDN_PAIR_TABLE_FLOATS;
    e0[22] = __int_as_float(n_hot);
    e0[23] = __int_as_float(n_own);
  }
  if (t < 0 || t >= n_total) return;
  const int pos = (t == s) ? n_hot + own_before : hot_before;
  float* o = pair_table + ((size_t)sl * k_nbr + pos) * DDN_PAIR_TABLE_FLOATS;
  const double* Pt = poses + (size_t)t * 12;
  double Rt[3][3], tt[3];
  for (int i = 0; i < 3; ++i) {
    for (int j = 0; j < 3; ++j) Rt[i][j] = Pt[i * 4 + j];
    tt[i] = Pt[i * 4 + 3];
  }
  double rows[3][4];
  for (int i = 0; i < 3; ++i) {
    double r[3];  // row i of R_t R_s^T
    for (int j = 0; j < 3; ++j) r[j] = Rt[i][0] * Rs[j][0] + Rt[i][1] * Rs[j][1] + Rt[i][2] * Rs[j][2];
    rows[i][0] = r[0] / fx;
    rows[i][1] = r[1] / fy;
    rows[i][2] = -r[0] * cx / fx - r[1] * cy / fy + r[2];
    rows[i][3] = tt[i] - (r[0] * ts[0] + r[1] * ts[1] + r[2] * ts[2]);
  }
  const double fxt = intr[t * 4 + 0], fyt = intr[t * 4 + 1], cxt = intr[t * 4 + 2], cyt = intr[t * 4 + 3];
  for (int j = 0; j < 4; ++j) {
    o[0 * 4 + j] = (float)(fxt * rows[0][j] + cxt * rows[2][j]);
    o[1 * 4 + j] = (float)(fyt * rows[1][j] + cyt * rows[2][j]);
    o[2 * 4 + j] = (float)rows[2][j];
  }
  for (int i = 0; i < 3; ++i)  // c_t = -R_t^T t_t
    o[12 + i] = (float)(-(Rt[0][i] * tt[0] + Rt[1][i] * tt[1] + Rt[2][i] * tt[2]));
  o[15] = __int_as_float(t);
  if (kRagged) {
    const int64_t* Lt = layout + (size_t)t * DDN_LAYOUT_COLS;
    const unsigned ht = (unsigned)Lt[0], wt = (unsigned)Lt[1];
    o[16] = __uint_as_float(wt);
    o[17] = __uint_as_float(ht);
    o[18] = (float)wt;  // K4's bounds test compares the raw bits of u, v with these
    o[19] = (float)ht;
    o[20] = (t == s) ? 1.f : 0.f;
    o[21] = __uint_as_float((unsigned)Lt[2] - 0x4B000000u * (wt + 1u));
    return;
  }
  o[16] = (float)intr[t * 4 + 0];
  o[17] = (float)intr[t * 4 + 1];
  o[18] = (float)intr[t * 4 + 2];
  o[19] = (float)intr[t * 4 + 3];
  o[20] = (t == s) ? 1.f : 0.f;
  o[21] = __uint_as_float((unsigned)t * hw - 0x4B000000u * (width + 1u));
}

__global__ void build_pair_tables_kernel(int n_total, int src_begin, int n_src, int k_nbr, unsigned hw, unsigned width,
                                         const double* __restrict__ poses,
                                         const double* __restrict__ intr,
                                         const int32_t* __restrict__ nbr, float* __restrict__ pair_table,
                                         float* __restrict__ src_table) {
  build_pair_tables_body<false>(n_total, src_begin, n_src, k_nbr, hw, width, poses, intr, nbr, pair_table, src_table, nullptr);
}

__global__ void build_pair_tables_ragged_kernel(int n_views, int k_nbr, const double* __restrict__ poses,
                                                const double* __restrict__ intr, const int32_t* __restrict__ nbr,
                                                float* __restrict__ pair_table, float* __restrict__ src_table,
                                                const int64_t* __restrict__ layout) {
  build_pair_tables_body<true>(n_views, 0, n_views, k_nbr, 0u, 0u, poses, intr, nbr, pair_table, src_table, layout);
}

// ------------------------------------------------------------------------------------------------
// K4
// ------------------------------------------------------------------------------------------------
struct FilterParams {
  const float* refined_all;  // [V,H,W]
  const float* normal;       // [n_src,H,W,3]
  const float* pair_table;   // [n_src,K,24]
  const float* src_table;    // [n_src,16]
  float* xyz;                // [n_src,Hs,Ws,3]
  uint8_t* votes;            // [n_src,Hs,Ws]
  int* bbox;                 // [6] ordered-int encoded, or nullptr
  FuseDev mark;              // occupancy marking of kept points (mark.units == nullptr: off)
  int src_begin, n_src, H, W, Hs, Ws, K, stride;
  int vote_threshold;
  float depth_threshold, grazing_cos, two_sided_tau;
  int normals_in_world;
  unsigned wbits, hbits;  // bit patterns of (float)W, (float)H for the bounds test on raw bits
};

// The arguments only ddn_backproject_filter_support* take: K4's optional third parameter, so that the parameters of the
// plain instantiations keep their layout (and the kernels their code).
struct SupportParams {
  uint8_t* support;  // same grid as votes
  int min_support;
  float support_tau;
};
// The trailing parameter of the reprojection forms (ddn_backproject_filter_support_reproj*): the support arguments and
// rho^2, the square of the round-trip pixel bound (+inf when rho^2 overflows float32: the bound then passes every
// finite error).
struct ReprojParams {
  SupportParams support;
  float reproj_px2;
};
__device__ __forceinline__ SupportParams support_params() { return SupportParams{nullptr, 0, 0.f}; }
__device__ __forceinline__ SupportParams support_params(const SupportParams& s) { return s; }
__device__ __forceinline__ SupportParams support_params(const ReprojParams& r) { return r.support; }
__device__ __forceinline__ float reproj_px2() { return 0.f; }
__device__ __forceinline__ float reproj_px2(const SupportParams&) { return 0.f; }
__device__ __forceinline__ float reproj_px2(const ReprojParams& r) { return r.reproj_px2; }
template <class... S>
struct IsReproj {
  static constexpr bool value = false;
};
template <>
struct IsReproj<ReprojParams> {
  static constexpr bool value = true;
};

__device__ __forceinline__ float rcp_approx(float x) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float sqrt_approx(float x) {
  float r;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
// The bits of u + 2^23 rounded toward zero are trunc(u) biased by kTruncBias, for 0 <= u < 2^22: the truncation
// runs on the FMA pipe (no F2I).
constexpr int kTruncBias = 0x4B000000;

// The (pixel, neighbour) evaluations of a pixel pair, in two steps so that the gathers of a thread's four pixels
// are all in flight before the first one is consumed.  pair_gather: project, bounds test, issue the depth lookups.
// pair_test: the candidate flag ("would vote if the grazing gate passes").
// The projection and the truncation run on both pixels at once (FFMA2, FMUL2, FADD2.RZ), with the scalar order of
// operations in each lane: U = fma(r.x, P, fma(r.y, Q, fma(r.z, d, r.w))), u = U * (1/Z), trunc(u) = u + 2^23 (RZ).
// A pixel without a point (NaN depth) computes along with its partner and fails the bounds test.
template <bool kBilinear, bool kFoldMask>
__device__ __forceinline__ void pixel_gather(float u, float v, unsigned ub, unsigned vb, const float* __restrict__ depth_all,
                                             unsigned off_k, unsigned W, int H, unsigned wbits, unsigned hbits, float& Z,
                                             float& D, bool& inb) {
  // 0 <= u < W and 0 <= v < H on the raw bits (negative floats and NaN compare as huge unsigned);
  // invalid pixels carry NaN depth, so Z > 0 rejects them too.
  inb = (__float_as_uint(u) < wbits) & (__float_as_uint(v) < hbits) & (Z > 0.f);
  if (kFoldMask && !inb) Z = INFINITY;  // folds the bounds mask into the one-sided test: inf < thr*D is false
  if (!kBilinear) {
    // 32-bit element offset from the start of refined_all; off_k = t*H*W - bias*(W+1) removes the 2^23
    // biases by modular arithmetic.  Out-of-bounds lanes read element 0 and are masked by `inb`.
    const unsigned off = inb ? vb * W + ub + off_k : 0u;
    D = __ldg(depth_all + off);
  } else {
    const float* __restrict__ depth_t = depth_all + (off_k + (unsigned)kTruncBias * (W + 1u));
    // N3: 4 taps at floor(u), floor(v), +1 clamped; all taps must be > 0
    const int x0 = inb ? ub - kTruncBias : 0, y0 = inb ? vb - kTruncBias : 0;
    const int x1 = min(x0 + 1, (int)W - 1), y1 = min(y0 + 1, H - 1);
    const float ta = __ldg(depth_t + y0 * W + x0), tb = __ldg(depth_t + y0 * W + x1);
    const float tc = __ldg(depth_t + y1 * W + x0), td = __ldg(depth_t + y1 * W + x1);
    const float fxw = u - (float)x0, fyw = v - (float)y0;
    const float gx = 1.f - fxw, gy = 1.f - fyw;
    const float acc = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(__fmul_rn(gx, gy), ta), __fmul_rn(__fmul_rn(fxw, gy), tb)),
                                          __fmul_rn(__fmul_rn(gx, fyw), tc)),
                                __fmul_rn(__fmul_rn(fxw, fyw), td));
    D = ((ta > 0.f) & (tb > 0.f) & (tc > 0.f) & (td > 0.f)) ? acc : 0.f;
  }
}

__device__ __forceinline__ f32x2 row_dot2(const float4& r, f32x2 P, f32x2 Q, f32x2 d) {
  return fma2(splat2(r.x), P, fma2(splat2(r.y), Q, fma2(splat2(r.z), d, splat2(r.w))));
}

template <bool kBilinear, bool kFoldMask>
__device__ __forceinline__ void pair_gather(const float4& r0, const float4& r1, const float4& r2, f32x2 P, f32x2 Q, f32x2 d,
                                            const float* __restrict__ depth_all, unsigned off_k, unsigned W, int H,
                                            unsigned wbits, unsigned hbits, float* Z, float* D, bool* inb, f32x2& inv) {
  const f32x2 U = row_dot2(r0, P, Q, d), V = row_dot2(r1, P, Q, d);
  unpack2(row_dot2(r2, P, Q, d), Z[0], Z[1]);
  inv = pack2(rcp_approx(Z[0]), rcp_approx(Z[1]));  // 1/Z, before the out-of-bounds lanes' Z becomes +inf
  const f32x2 u = mul2(U, inv), v = mul2(V, inv);
  const f32x2 bias = splat2(8388608.0f);
  const f32x2 ub = add_rz2(u, bias), vb = add_rz2(v, bias);  // trunc(u), trunc(v) + kTruncBias per lane
#pragma unroll
  for (int e = 0; e < 2; ++e)
    pixel_gather<kBilinear, kFoldMask>(lane2(u, e), lane2(v, e), __float_as_uint(lane2(ub, e)), __float_as_uint(lane2(vb, e)),
                                       depth_all, off_k, W, H, wbits, hbits, Z[e], D[e], inb[e]);
}

// cm |= bit when a < b, as one compare and one predicated OR (the compiler would otherwise build the bit with
// two selects)
__device__ __forceinline__ void or_bit_if_less(unsigned& cm, float a, float b, unsigned bit) {
  asm("{\n\t.reg .pred p;\n\tsetp.lt.f32 p, %1, %2;\n\t@p or.b32 %0, %0, %3;\n\t}" : "+r"(cm) : "f"(a), "f"(b), "r"(bit));
}

// Candidate bits of a pixel pair.  kFoldMask: Z is +inf for out-of-bounds lanes, so the bounds mask is already in Z.
template <bool kTwoSided, bool kFoldMask>
__device__ __forceinline__ void pair_test(const float* Z, const float* D, const bool* inb, float thr, float tau, unsigned bit,
                                          unsigned* cm) {
  if (kTwoSided) {
#pragma unroll
    for (int e = 0; e < 2; ++e)
      if (inb[e] & (D[e] > 0.f) & (fabsf(Z[e] - D[e]) > tau * D[e])) cm[e] |= bit;
    return;
  }
  // one-sided floater test z < float32(thr * D) (scripts/test.py:319-321, NEP-50 product in float32).
  // The lookup-valid gate D > 0 (:315) is implied: inb has Z > 0 and thr > 0, so Z < thr*D needs D > 0.
  const f32x2 thrD = mul2(splat2(thr), pack2(D[0], D[1]));
#pragma unroll
  for (int e = 0; e < 2; ++e) {
    if (kFoldMask) or_bit_if_less(cm[e], Z[e], lane2(thrD, e), bit);
    else if (inb[e] & (Z[e] < lane2(thrD, e))) cm[e] |= bit;
  }
}

// Support bits of a pixel pair: neighbour entry `bit` sees the surface of the pixel within the relative depth error
// tau, |Z - D| <= tau*D.  No grazing gate.  kFoldMask: out-of-bounds lanes carry Z = +inf and pixels without a point
// NaN, so both fail the comparison without the bounds mask; D > 0 is implied, since in-bounds lanes have Z > 0.
// kReproj (the reprojection forms): the entry must also pass the forward-backward reprojection test of
// include/ddn_b200.h in its closed form, from t's epipole in s, ep = (e_x, e_y, e_z, -e_z):
//   w = (Z - D)/Z,  z' = d + w (e_z - d),  A = d e_x - P e_z,  B = d e_y - Q e_z,
//   z' > 0  and  w^2 (A^2 + B^2) <= rho^2 (d z')^2.
// inv = 1/Z of pair_gather.  Lanes that fail the depth test (out of bounds: Z = +inf; no point: NaN) fail the
// conjunction whatever this evaluates to.
template <bool kFoldMask, bool kReproj = false>
__device__ __forceinline__ void pair_support(const float* Z, const float* D, const bool* inb, float tau, unsigned bit,
                                             unsigned* sm, f32x2 inv = 0ull, f32x2 d = 0ull, f32x2 P = 0ull, f32x2 Q = 0ull,
                                             float4 ep = float4{}, float rho2 = 0.f) {
  const f32x2 D2 = pack2(D[0], D[1]);
  const f32x2 dz = sub2(pack2(Z[0], Z[1]), D2), tD = mul2(splat2(tau), D2);
  if (kReproj) {
    const f32x2 w = mul2(dz, inv);
    const f32x2 A = fma2(P, splat2(ep.w), mul2(d, splat2(ep.x)));
    const f32x2 B = fma2(Q, splat2(ep.w), mul2(d, splat2(ep.y)));
    const f32x2 zp = fma2(w, sub2(splat2(ep.z), d), d);
    const f32x2 lhs = mul2(mul2(w, w), fma2(A, A, mul2(B, B)));
    const f32x2 dzp = mul2(d, zp);
    const f32x2 rhs = mul2(mul2(splat2(rho2), dzp), dzp);
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const bool ok = (lane2(zp, e) > 0.f) & (lane2(lhs, e) <= lane2(rhs, e)) & (fabsf(lane2(dz, e)) <= lane2(tD, e));
      if (kFoldMask ? ok : (ok & inb[e])) sm[e] |= bit;
    }
  } else {
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      if (kFoldMask) {
        if (fabsf(lane2(dz, e)) <= lane2(tD, e)) sm[e] |= bit;
      } else if (inb[e] & (fabsf(lane2(dz, e)) <= lane2(tD, e))) {
        sm[e] |= bit;
      }
    }
  }
}

// t's epipole in s, e = K_s (R_s c_t + t_s) = K_s R_s (c_t - c_s), as (e_x, e_y, e_z, -e_z): from the source table
// (rows of R_s^T K_s^-1 with c_s, then cx, cy, fx, fy; the rows of R_s^T recovered as load_normal does) and c_t, floats
// 12-14 of t's pair-table entry.  Each rounding written out (no contraction), so tests/reproj_oracle.py replays it
// bit for bit on the host.
__device__ __forceinline__ float4 epipole(const float* __restrict__ src, const float* __restrict__ ct) {
  const float fx = __ldg(src + 14), fy = __ldg(src + 15), cx = __ldg(src + 12), cy = __ldg(src + 13);
  float a0 = 0.f, a1 = 0.f, a2 = 0.f;  // R_s (c_t - c_s) = sum_i (row i of R_s^T) * (c_t - c_s)_i
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const float m0 = __ldg(src + i * 4 + 0), m1 = __ldg(src + i * 4 + 1), m2 = __ldg(src + i * 4 + 2);
    const float ra = __fmul_rn(m0, fx), rb = __fmul_rn(m1, fy);
    const float rc = __fadd_rn(__fadd_rn(m2, __fmul_rn(m0, cx)), __fmul_rn(m1, cy));
    const float c = __fsub_rn(__ldg(ct + i), __ldg(src + i * 4 + 3));
    a0 = __fadd_rn(a0, __fmul_rn(ra, c));
    a1 = __fadd_rn(a1, __fmul_rn(rb, c));
    a2 = __fadd_rn(a2, __fmul_rn(rc, c));
  }
  const float ex = __fadd_rn(__fmul_rn(fx, a0), __fmul_rn(cx, a2)), ey = __fadd_rn(__fmul_rn(fy, a1), __fmul_rn(cy, a2));
  return make_float4(ex, ey, a2, -a2);
}

// Normal of one source pixel for the grazing gate (scripts/test.py:291), read on demand: only vote
// candidates need it, and they are rare (floaters), so the 12 B/pixel normal map is not streamed.
// normals_in_world rotates it by R_s^T (rows recovered from the source table) and divides by (|n| + 1e-8), as
// oracle/restatement_masks.py:transform_normals states it; the default camera-frame normal is used as given.
__device__ __forceinline__ void load_normal(const float* __restrict__ normal_view, size_t pixel, bool in_world,
                                            const float* __restrict__ s_src, float& n0, float& n1, float& n2) {
  const float* np_ = normal_view + pixel * 3;
  n0 = __ldg(np_ + 0);
  n1 = __ldg(np_ + 1);
  n2 = __ldg(np_ + 2);
  if (in_world) {
    const float fx = s_src[14], fy = s_src[15], cx = s_src[12], cy = s_src[13];
    float w[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      const float ra = s_src[i * 4 + 0] * fx, rb = s_src[i * 4 + 1] * fy;
      const float rc = s_src[i * 4 + 2] + s_src[i * 4 + 0] * cx + s_src[i * 4 + 1] * cy;
      w[i] = ra * n0 + rb * n1 + rc * n2;
    }
    const float inv = rcp_approx(sqrt_approx(fmaf(w[0], w[0], fmaf(w[1], w[1], w[2] * w[2]))) + 1e-8f);
    n0 = w[0] * inv, n1 = w[1] * inv, n2 = w[2] * inv;
  }
}

// Bulk asynchronous copy shared -> global (the TMA engine's 1-D form, SASS UBLKCP): with -DDDN_K4_BULK=1 one elected
// lane hands a warp's 1536-byte xyz slice to the copy engine instead of 32 lanes moving it with three LDS.128 + three
// streaming STG.128 each.  Measured at cfg 2 (profiles/README.md, round 2): 2.29 ms against 2.23 ms for the per-lane
// copy (3.03 vs 2.97 ms with the occupancy mark fused in) - the proxy fence and the wait for the engine's read before
// the CTA may retire cost more than the twelve instructions per thread they replace - so the per-lane copy stays.
#ifndef DDN_K4_BULK
#define DDN_K4_BULK 0
#endif
__device__ __forceinline__ void fence_proxy_async_shared() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void bulk_store_shared_to_global(void* gdst, const void* ssrc, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;\n\tcp.async.bulk.commit_group;"
               :
               : "l"(gdst), "r"((uint32_t)__cvta_generic_to_shared(ssrc)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void bulk_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }

// Pixel ownership.  A CTA owns kFilterChunk consecutive source-grid pixels of one view, a warp 128 of them.
//   layout 0 ("strided"):  thread pixel j = warp base + j*32 + lane.  Every load, gather and byte store of a
//                          warp instruction covers 32 consecutive pixels; xyz leaves through a per-warp
//                          shared staging buffer as float4 (no block barrier).
//   layout 1 ("adjacent"): thread pixel j = warp base + lane*4 + j.  One LDG.128 for the depths, one STG.32
//                          for the votes, three STG.128 for xyz straight from registers, no shared staging;
//                          the gathers of one instruction are 4 pixels apart.
// -DDDN_K4_LAYOUT selects the default; both produce identical results.
#ifndef DDN_K4_LAYOUT
#define DDN_K4_LAYOUT 0
#endif
constexpr int kWarpPix = 32 * kFilterPX;
static_assert(kFilterPX == 4, "the layouts below are written for 4 pixels per thread");

// kRagged (ddn_backproject_filter_ragged; layout = the device layout, nullptr otherwise): one flat grid over the chunks
// of all views in view order (the L2 argument above holds unchanged); a CTA finds its view in the layout, and every
// neighbour's W, H and bounds-test bits come from its table entry (floats 16-19) next to the gather offset.
// p.n_src is then the number of views, and p.H, p.W, p.Hs, p.Ws, p.src_begin, p.wbits and p.hbits are not read.
// kSupport (ddn_backproject_filter_support*; Support = SupportParams, the plain kernels have no third parameter): also
// count, per pixel, the neighbour entries that support the point (pair_support), write the count to sp.support and apply
// the keep rule and vote encoding of include/ddn_b200.h.  The support forms take 56 to 64 registers with nearest
// sampling: at 5 CTAs per SM (48 registers) they would spill inside the neighbour loop, at 4 they do not.
// kReproj (ddn_backproject_filter_support_reproj*; Support = ReprojParams): the support test also requires the
// forward-backward reprojection test (pair_support); the epipoles of the hot entries are computed once per CTA into
// shared memory (16 B per entry, after the pair table).  With the support forms' bounds these take 64 registers with
// nearest sampling and 80 with bilinear, and their few spills lie outside the per-neighbour loop.
template <bool kBilinear, bool kStride1, bool kTwoSided, int kLayout, bool kRagged, class... Support>
__global__ void __launch_bounds__(kFilterThreads, kBilinear ? 3 : (sizeof...(Support) ? DDN_K4_SUPPORT_MINBLOCKS : DDN_K4_MINBLOCKS))
    backproject_filter_kernel(const FilterParams p, const int64_t* __restrict__ layout, Support... support) {
  constexpr bool kSupport = sizeof...(Support) != 0;
  constexpr bool kReproj = IsReproj<Support...>::value;
  const SupportParams sp = support_params(support...);
  extern __shared__ __align__(16) float smem[];
  float* s_src = smem;                     // 16 floats
  float* s_pair = s_src + 16;              // K*24 floats
  float4* s_epi = reinterpret_cast<float4*>(s_pair + p.K * DDN_PAIR_TABLE_FLOATS);  // kReproj: K float4
  float* s_stage = s_pair + p.K * (DDN_PAIR_TABLE_FLOATS + (kReproj ? 4 : 0));      // layout 0: 8 warps x 128 px x 3 floats
  __shared__ int s_bbox[6];
  __shared__ int s_marked;

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int sl = kRagged ? layout_view_of(layout, p.n_src, 5, blockIdx.x) : (int)blockIdx.y;
  const int s = kRagged ? sl : p.src_begin + sl;
  const int64_t* __restrict__ L = layout + (size_t)sl * DDN_LAYOUT_COLS;  // ragged: the source view's layout row
  // the source view's full and strided row length, read where the uniform kernel reads p.W / p.Ws
  auto W_src = [&]() -> int { return kRagged ? (int)L[1] : p.W; };
  auto Ws_src = [&]() -> int { return kRagged ? ((int)L[1] + p.stride - 1) / p.stride : p.Ws; };
  const int Ps = kRagged ? ((int)L[0] + p.stride - 1) / p.stride * Ws_src() : p.Hs * p.Ws;  // source-grid pixels per view
  const int chunk0 = kRagged ? (int)(blockIdx.x - L[5]) * kFilterChunk : blockIdx.x * kFilterChunk;
  const size_t HW = (size_t)p.H * p.W;
  const float* __restrict__ depth_s = kRagged ? p.refined_all + L[2] : p.refined_all + (size_t)s * HW;
  const float* __restrict__ normal_s = kRagged ? p.normal + (size_t)L[2] * 3 : p.normal + (size_t)sl * HW * 3;

  // tables -> shared memory, as float4 (entries are 96 bytes; the gather offset t*H*W - bias*(W+1) of every
  // entry was put into float 21 by build_pair_tables_kernel)
  {
    const float4* g4 = reinterpret_cast<const float4*>(p.pair_table + (size_t)sl * p.K * DDN_PAIR_TABLE_FLOATS);
    float4* s4 = reinterpret_cast<float4*>(s_pair);
    for (int i = tid; i < p.K * (DDN_PAIR_TABLE_FLOATS / 4); i += kFilterThreads) s4[i] = __ldg(g4 + i);
    if (tid < 4) reinterpret_cast<float4*>(s_src)[tid] = __ldg(reinterpret_cast<const float4*>(p.src_table + (size_t)sl * 16) + tid);
    if (tid < 6) s_bbox[tid] = tid < 3 ? 0x7fffffff : (int)0x80000000;
    if (tid == 6) s_marked = 0;
    if (kReproj) {  // read from the global tables, so that the barrier below covers them too
      const float* g = p.pair_table + (size_t)sl * p.K * DDN_PAIR_TABLE_FLOATS;
      const int nh = __float_as_int(__ldg(g + 22));
      for (int k = tid; k < nh; k += kFilterThreads) s_epi[k] = epipole(p.src_table + (size_t)sl * 16, g + k * DDN_PAIR_TABLE_FLOATS + 12);
    }
  }

  // first pixel of the thread on the source grid: q0 = y0 * Ws + x0 (one integer division per thread)
  const int wbase = chunk0 + warp * kWarpPix;
  const int q0 = wbase + (kLayout == 1 ? lane * kFilterPX : lane);
  constexpr int kStep = kLayout == 1 ? 1 : 32;
  int ys_run = q0 / Ws_src();
  int xs_run = q0 - ys_run * Ws_src();

  // Per-pixel state kept in registers: depth d (NaN = no point), P = d*x, Q = d*y, vote count.  d, P and Q are held
  // as pairs of pixels (0, 1) and (2, 3) for the packed projection; d(j) reads one pixel's depth.
  constexpr int kPairs = kFilterPX / 2;
  f32x2 d2[kPairs], P2[kPairs], Q2[kPairs];
  int nvotes[kFilterPX];  // kSupport: the count of supporting neighbour entries in bits 16-31 (both counts <= 1024)
  unsigned src_pix[kFilterPX];  // element index of the pixel in its own full-resolution map
  const float qnan = __int_as_float(0x7fc00000);
  {
    float dd[kFilterPX];
    int px[kFilterPX], py[kFilterPX];
#pragma unroll
    for (int j = 0; j < kFilterPX; ++j) {
      px[j] = kStride1 ? xs_run : xs_run * p.stride;
      py[j] = kStride1 ? ys_run : ys_run * p.stride;
      src_pix[j] = kStride1 ? (unsigned)(q0 + j * kStep) : (unsigned)py[j] * (unsigned)W_src() + (unsigned)px[j];
      xs_run += kStep;
      while (xs_run >= Ws_src()) {
        xs_run -= Ws_src();
        ++ys_run;
      }
    }
    if (kLayout == 1 && kStride1 && q0 + kFilterPX <= Ps && ((reinterpret_cast<uintptr_t>(depth_s + q0) & 15) == 0)) {
      const float4 v = __ldg(reinterpret_cast<const float4*>(depth_s + q0));
      dd[0] = v.x, dd[1] = v.y, dd[2] = v.z, dd[3] = v.w;
    } else {
#pragma unroll
      for (int j = 0; j < kFilterPX; ++j) dd[j] = (q0 + j * kStep) < Ps ? __ldg(depth_s + src_pix[j]) : 0.f;
    }
#pragma unroll
    for (int h = 0; h < kPairs; ++h) {
      d2[h] = pack2(dd[2 * h] > 0.f ? dd[2 * h] : qnan, dd[2 * h + 1] > 0.f ? dd[2 * h + 1] : qnan);
      asm volatile("" : "+l"(d2[h]));  // keep the NaN-tagged depths in registers (no per-neighbour recompute)
      P2[h] = mul2(d2[h], pack2((float)px[2 * h], (float)px[2 * h + 1]));
      Q2[h] = mul2(d2[h], pack2((float)py[2 * h], (float)py[2 * h + 1]));
    }
#pragma unroll
    for (int j = 0; j < kFilterPX; ++j) nvotes[j] = 0;
  }
  auto d = [&](int j) { return lane2(d2[j >> 1], j & 1); };
  __syncthreads();  // tables visible
  // warp-uniform flags: pixel pair h of this warp has at least one point (sky / masked regions are
  // contiguous, so whole pairs drop out of the neighbour loop)
  bool live[kPairs];
  bool any_live = false;
#pragma unroll
  for (int h = 0; h < kPairs; ++h) {
    live[h] = __any_sync(0xffffffffu, d(2 * h) > 0.f || d(2 * h + 1) > 0.f);
    any_live |= live[h];
  }

  const unsigned wbits = p.wbits, hbits = p.hbits;
  const float thr = p.depth_threshold, gcos = p.grazing_cos, tau = p.two_sided_tau;
  const float stau = kSupport ? sp.support_tau : 0.f;
  const float rho2 = reproj_px2(support...);
  const bool in_world = p.normals_in_world != 0;
  const int n_hot = __float_as_int(s_pair[22]), n_own = __float_as_int(s_pair[23]);

  // world position of pixel j (scripts/test.py:79-90 then :233), fp32 with float64-precomputed rows;
  // the same expression ddn_align_views' bounding-box epilogue evaluates (backproject_px)
  auto world_of = [&](int j, float& X, float& Y, float& Z) {
    backproject_pqd(s_src, lane2(P2[j >> 1], j & 1), lane2(Q2[j >> 1], j & 1), d(j), X, Y, Z);
  };

  // Hot loop: branch-free candidate test for every (pixel, neighbour); the four gathers of a thread
  // issue back to back.  Candidates ("would vote if the grazing gate passes") are only recorded as a
  // bit per neighbour; the gate itself (scripts/test.py:284-295) needs the pixel's normal and is
  // resolved after each block of 32 neighbours, once per pixel that has a candidate at all.
  if (any_live) {
    bool all_live = true;
#pragma unroll
    for (int h = 0; h < kPairs; ++h) all_live &= live[h];
    for (int k0 = 0; k0 < n_hot; k0 += 32) {
      const int k1 = min(k0 + 32, n_hot);
      unsigned cm[kFilterPX], sm[kFilterPX];  // candidate and support bits of the block
#pragma unroll
      for (int j = 0; j < kFilterPX; ++j) cm[j] = 0u, sm[j] = 0u;
      unsigned bit = 1u;
      for (int k = k0; k < k1; ++k, bit <<= 1) {
        const float4* t4 = reinterpret_cast<const float4*>(s_pair + k * DDN_PAIR_TABLE_FLOATS);
        const float4 r0 = t4[0], r1 = t4[1], r2 = t4[2];
        const unsigned off_k = __float_as_uint(s_pair[k * DDN_PAIR_TABLE_FLOATS + 21]);
        const float4 wh = kRagged ? t4[4] : make_float4(0.f, 0.f, 0.f, 0.f);  // ragged: the neighbour's W, H, (float)W, (float)H
        float Z[kFilterPX], D[kFilterPX];
        bool inb[kFilterPX];
        f32x2 inv[kPairs];
        constexpr bool kFold = !kBilinear && !kTwoSided;
        auto gather = [&](int h) {
          pair_gather<kBilinear, kFold>(r0, r1, r2, P2[h], Q2[h], d2[h], p.refined_all, off_k, kRagged ? __float_as_uint(wh.x) : (unsigned)p.W,
                                        kRagged ? __float_as_int(wh.y) : p.H, kRagged ? __float_as_uint(wh.z) : wbits,
                                        kRagged ? __float_as_uint(wh.w) : hbits, Z + 2 * h, D + 2 * h, inb + 2 * h, inv[h]);
        };
        auto test = [&](int h) {
          pair_test<kTwoSided, kFold>(Z + 2 * h, D + 2 * h, inb + 2 * h, thr, tau, bit, cm + 2 * h);
          if (kReproj)
            pair_support<kFold, true>(Z + 2 * h, D + 2 * h, inb + 2 * h, stau, bit, sm + 2 * h, inv[h], d2[h], P2[h], Q2[h], s_epi[k], rho2);
          else if (kSupport)
            pair_support<kFold>(Z + 2 * h, D + 2 * h, inb + 2 * h, stau, bit, sm + 2 * h);
        };
        if (all_live) {
#pragma unroll
          for (int h = 0; h < kPairs; ++h) gather(h);
#pragma unroll
          for (int h = 0; h < kPairs; ++h) test(h);
        } else {
#pragma unroll
          for (int h = 0; h < kPairs; ++h) {
            if (live[h]) {
              gather(h);
              test(h);
            }
          }
        }
      }
      if (kSupport) {
#pragma unroll
        for (int j = 0; j < kFilterPX; ++j) nvotes[j] += __popc(sm[j]) << 16;
      }
      // dot(n, -(Xw - c_t)/|Xw - c_t|) > cos  <=>  dot(n, c_t - Xw) > cos * |c_t - Xw|
#pragma unroll
      for (int j = 0; j < kFilterPX; ++j) {
        if (cm[j]) {
          float n0, n1, n2, wx, wy, wz;
          load_normal(normal_s, src_pix[j], in_world, s_src, n0, n1, n2);
          world_of(j, wx, wy, wz);
          unsigned m = cm[j];
          while (m) {
            const int k = k0 + __ffs(m) - 1;
            m &= m - 1;
            const float4 cc = reinterpret_cast<const float4*>(s_pair + k * DDN_PAIR_TABLE_FLOATS)[3];
            const float ex = cc.x - wx, ey = cc.y - wy, ez = cc.z - wz;
            const float dn = fmaf(n0, ex, fmaf(n1, ey, n2 * ez));
            const float len = sqrt_approx(fmaf(ex, ex, fmaf(ey, ey, ez * ez)));
            nvotes[j] += (dn > gcos * len) ? 1 : 0;
          }
        }
      }
    }
  }

  // Own view (only present in the reference-parity table K = V).  The reference normalises by (z + 1e-8)
  // before applying K (scripts/test.py:71-75), so u = x * z/(z+1e-8) lands ~x*1e-8/z BELOW the integer x
  // (far above float64 round-off) and the truncation at :308-309 looks up pixel (x-1, y-1) for
  // x, y >= 1.  Reproduced in integer arithmetic; z is the pixel's own depth.  (x == 0 or y == 0 is a
  // round-off tie in the reference.)
  // Bilinear sampling never votes here: the sample at (u, v) puts a weight of about e = (x + y)*1e-8/z on the
  // neighbouring taps and 1 - e on the pixel's own depth z, so z < thr*D needs a tap above (1/thr - 1)/e times z and
  // |z - D| > tau*D one above tau/e times z (a zero tap makes D = 0: no vote).  At x + y < 2^13 and z = 1 that is
  // more than 600 times the pixel's depth for tau = 0.05.  The loop is not compiled into the bilinear instantiations.
  if (!kBilinear && n_own > 0) {
    for (int k = n_hot; k < n_hot + n_own; ++k) {
      const float4* t4 = reinterpret_cast<const float4*>(s_pair + k * DDN_PAIR_TABLE_FLOATS);
      const float4 cc = t4[3];
#pragma unroll
      for (int j = 0; j < kFilterPX; ++j) {
        if (d(j) > 0.f) {
          const int py = (int)(src_pix[j] / (unsigned)W_src()), px = (int)(src_pix[j] - (unsigned)py * (unsigned)W_src());
          const int ux = max(px - 1, 0), vy = max(py - 1, 0);
          const float D = __ldg(depth_s + (size_t)vy * W_src() + ux);
          const bool bad = kTwoSided ? (fabsf(d(j) - D) > tau * D) : (d(j) < __fmul_rn(thr, D));
          if (D > 0.f && bad) {
            float n0, n1, n2, wx, wy, wz;
            load_normal(normal_s, src_pix[j], in_world, s_src, n0, n1, n2);
            world_of(j, wx, wy, wz);
            const float ex = cc.x - wx, ey = cc.y - wy, ez = cc.z - wz;
            const float dn = fmaf(n0, ex, fmaf(n1, ey, n2 * ez));
            const float len = sqrt_approx(fmaf(ex, ex, fmaf(ey, ey, ez * ez)));
            nvotes[j] += (dn > gcos * len) ? 1 : 0;
          }
        }
      }
    }
  }

  // ---- epilogue: world positions (recomputed from the registers), votes, bounding box, occupancy ----
  bool bulk_pending = false;  // lane 0: a bulk copy out of this warp's staging slice is in flight
  float X[kFilterPX], Y[kFilterPX], Zw[kFilterPX];
  bool keep[kFilterPX];
  unsigned vote_bytes = 0, support_bytes = 0;
  // kSupport: a valid point the neighbours do not support stores 254, which no fusion threshold min(thr, 254) passes;
  // a supported one stores its count saturated at 254, or at 253 when every count passes (threshold >= 255)
  const int vote_cap = (kSupport && p.vote_threshold == INT_MAX) ? 253 : 254;
#pragma unroll
  for (int h = 0; h < kPairs; ++h) {
    f32x2 X2, Y2, Z2;
    backproject_pqd2(s_src, P2[h], Q2[h], d2[h], X2, Y2, Z2);
    unpack2(X2, X[2 * h], X[2 * h + 1]);
    unpack2(Y2, Y[2 * h], Y[2 * h + 1]);
    unpack2(Z2, Zw[2 * h], Zw[2 * h + 1]);
  }
#pragma unroll
  for (int j = 0; j < kFilterPX; ++j) {
    const bool valid = d(j) > 0.f;
    if (!valid) X[j] = 0.f, Y[j] = 0.f, Zw[j] = 0.f;
    if (kSupport) {
      const int nv = nvotes[j] & 0xffff, ns = nvotes[j] >> 16;
      const bool supported = ns >= sp.min_support;
      keep[j] = valid && nv < p.vote_threshold && supported;
      vote_bytes |= (valid ? (supported ? (unsigned)min(nv, vote_cap) : 254u) : 255u) << (8 * j);
      support_bytes |= (valid ? (unsigned)min(ns, 254) : 255u) << (8 * j);
    } else {
      keep[j] = valid && nvotes[j] < p.vote_threshold;
      vote_bytes |= (valid ? (unsigned)min(nvotes[j], 254) : 255u) << (8 * j);
    }
  }
  const size_t out0 = kRagged ? (size_t)L[3] : (size_t)sl * Ps;  // first pixel of the view in the outputs
  if (kLayout == 1) {
    uint8_t* vo = p.votes + out0 + q0;
    if (q0 + kFilterPX <= Ps && ((reinterpret_cast<uintptr_t>(vo) & 3) == 0) &&
        (!kSupport || (reinterpret_cast<uintptr_t>(sp.support + out0 + q0) & 3) == 0)) {
      *reinterpret_cast<unsigned*>(vo) = vote_bytes;
      if (kSupport) *reinterpret_cast<unsigned*>(sp.support + out0 + q0) = support_bytes;
    } else {
#pragma unroll
      for (int j = 0; j < kFilterPX; ++j)
        if (q0 + j < Ps) {
          vo[j] = (uint8_t)(vote_bytes >> (8 * j));
          if (kSupport) sp.support[out0 + q0 + j] = (uint8_t)(support_bytes >> (8 * j));
        }
    }
    float* xo = p.xyz + (out0 + q0) * 3;
    if (q0 + kFilterPX <= Ps && ((reinterpret_cast<uintptr_t>(xo) & 15) == 0)) {
      float4* x4 = reinterpret_cast<float4*>(xo);
      __stcs(x4 + 0, make_float4(X[0], Y[0], Zw[0], X[1]));
      __stcs(x4 + 1, make_float4(Y[1], Zw[1], X[2], Y[2]));
      __stcs(x4 + 2, make_float4(Zw[2], X[3], Y[3], Zw[3]));
    } else {
#pragma unroll
      for (int j = 0; j < kFilterPX; ++j)
        if (q0 + j < Ps) {
          __stcs(xo + j * 3 + 0, X[j]);
          __stcs(xo + j * 3 + 1, Y[j]);
          __stcs(xo + j * 3 + 2, Zw[j]);
        }
    }
  } else {
#pragma unroll
    for (int j = 0; j < kFilterPX; ++j)
      if (q0 + j * 32 < Ps) {
        p.votes[out0 + q0 + j * 32] = (uint8_t)(vote_bytes >> (8 * j));
        if (kSupport) sp.support[out0 + q0 + j * 32] = (uint8_t)(support_bytes >> (8 * j));
      }
    // xyz through the warp's staging slice: stride-3 STS (conflict free), float4 out (16 B per lane, coalesced)
    float* sw = s_stage + warp * (kWarpPix * 3);
#pragma unroll
    for (int j = 0; j < kFilterPX; ++j) {
      const int l = j * 32 + lane;
      sw[l * 3 + 0] = X[j];
      sw[l * 3 + 1] = Y[j];
      sw[l * 3 + 2] = Zw[j];
    }
#if DDN_K4_BULK
    fence_proxy_async_shared();  // the slice was written through the generic proxy: make it visible to the copy engine
#endif
    __syncwarp();
    const int n_w = min(kWarpPix, Ps - wbase);  // pixels of this warp that exist (<= 0: none)
    float* xo = p.xyz + (out0 + wbase) * 3;
    if (n_w == kWarpPix && ((reinterpret_cast<uintptr_t>(xo) & 15) == 0)) {
#if DDN_K4_BULK
      if (lane == 0) {
        bulk_store_shared_to_global(xo, sw, kWarpPix * 3 * sizeof(float));
        bulk_pending = true;
      }
#else
      const float4* s4 = reinterpret_cast<const float4*>(sw);
      float4* g4 = reinterpret_cast<float4*>(xo);
#pragma unroll
      for (int q = 0; q < 3; ++q) __stcs(g4 + q * 32 + lane, s4[q * 32 + lane]);
#endif
    } else {
      for (int i = lane; i < n_w * 3; i += 32) __stcs(xo + i, sw[i]);
    }
  }

  if (p.bbox != nullptr && any_live) {
    float bmin[3] = {INFINITY, INFINITY, INFINITY}, bmax[3] = {-INFINITY, -INFINITY, -INFINITY};
#pragma unroll
    for (int j = 0; j < kFilterPX; ++j) {
      if (keep[j]) {
        bmin[0] = fminf(bmin[0], X[j]), bmax[0] = fmaxf(bmax[0], X[j]);
        bmin[1] = fminf(bmin[1], Y[j]), bmax[1] = fmaxf(bmax[1], Y[j]);
        bmin[2] = fminf(bmin[2], Zw[j]), bmax[2] = fmaxf(bmax[2], Zw[j]);
      }
    }
    // warp reduction with REDUX on the order-preserving int encoding, then one shared atomic per warp
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      const int lo = __reduce_min_sync(0xffffffffu, float_to_ordered(bmin[i]));
      const int hi = __reduce_max_sync(0xffffffffu, float_to_ordered(bmax[i]));
      if (lane == 0 && lo <= hi) {
        atomicMin(&s_bbox[i], lo);
        atomicMax(&s_bbox[3 + i], hi);
      }
    }
  }

  // Stage 4's mark pass, fused: the occupancy bit of every kept point.  A cell equal to that of the pixel
  // to the left (same thread, or the neighbouring lane) is already set by that pixel.
  if (p.mark.units != nullptr && any_live) {
    const GridDev g = *p.mark.grid;
    if (g.n_units != 0) {
      const float rv = 1.0f / g.voxel;
      // cell_of_point of every kept pixel, with voxel_coord's quotient evaluated as pairs.  While the estimate of every
      // kept pixel is in voxel_quotient_in_domain (finite, 2^-126 <= |q| < 2^22) the floor converts straight to an
      // integer and the inside test is one unsigned compare per axis.
      int kx[kFilterPX], ky[kFilterPX], kz[kFilterPX];
      bool all_exact = true;
#pragma unroll
      for (int h = 0; h < kPairs; ++h) {
        const bool u0 = keep[2 * h], u1 = keep[2 * h + 1];
        f32x2 q[3];
        q[0] = voxel_quotient2(pack2(X[2 * h], X[2 * h + 1]), g.ox, g.voxel, rv, u0, u1, all_exact);
        q[1] = voxel_quotient2(pack2(Y[2 * h], Y[2 * h + 1]), g.oy, g.voxel, rv, u0, u1, all_exact);
        q[2] = voxel_quotient2(pack2(Zw[2 * h], Zw[2 * h + 1]), g.oz, g.voxel, rv, u0, u1, all_exact);
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          kx[2 * h + e] = __float2int_rd(lane2(q[0], e));
          ky[2 * h + e] = __float2int_rd(lane2(q[1], e));
          kz[2 * h + e] = __float2int_rd(lane2(q[2], e));
        }
      }
      if (!all_exact) {  // a kept point beyond 2^22 voxels of the origin on some axis, or not finite: outside is -1
        auto coord = [&](float p, float o, int n) {
          const float f = voxel_coord(p, o, g.voxel, rv);
          return f >= 0.f && f < (float)n ? (int)f : -1;
        };
#pragma unroll
        for (int j = 0; j < kFilterPX; ++j) {
          kx[j] = coord(X[j], g.ox, g.nx);
          ky[j] = coord(Y[j], g.oy, g.ny);
          kz[j] = coord(Zw[j], g.oz, g.nz);
        }
      }
      uint64_t cell[kFilterPX];
      int mine = 0;
#pragma unroll
      for (int j = 0; j < kFilterPX; ++j) {
        const bool inside = keep[j] & ((unsigned)kx[j] < (unsigned)g.nx) & ((unsigned)ky[j] < (unsigned)g.ny) & ((unsigned)kz[j] < (unsigned)g.nz);
        const uint64_t c = cell_of_index(g, kx[j], ky[j], kz[j]);  // computed for every pixel: a select, no branch
        cell[j] = inside ? c : kNoCell;
        mine += inside ? 1 : 0;
      }
#pragma unroll
      for (int j = 0; j < kFilterPX; ++j) {
        // left neighbour: layout 1 - previous pixel of the thread, or the last pixel of the previous lane;
        // layout 0 - the same group in the previous lane
        uint64_t left = __shfl_up_sync(0xffffffffu, kLayout == 1 ? cell[kFilterPX - 1] : cell[j], 1);
        if (lane == 0) left = kNoCell;
        if (kLayout == 1 && j > 0) left = cell[j - 1];
        if (cell[j] != kNoCell && cell[j] != left) set_cell_bit(p.mark.units, p.mark.dirty, cell[j], left);
      }
      mine = __reduce_add_sync(0xffffffffu, mine);
      if (lane == 0 && mine) atomicAdd(&s_marked, mine);
    }
  }
  __syncthreads();
  if (p.bbox != nullptr && tid < 6) {
    if (tid < 3) {
      if (s_bbox[tid] != 0x7fffffff) atomicMin(p.bbox + tid, s_bbox[tid]);
    } else {
      if (s_bbox[tid] != (int)0x80000000) atomicMax(p.bbox + tid, s_bbox[tid]);
    }
  }
  if (tid == 6 && s_marked) atomicAdd(p.mark.counts, (unsigned long long)s_marked);
  if (bulk_pending) bulk_store_wait_read();  // the staging slice must stay intact until the copy engine has read it
}

__global__ void bbox_init_kernel(int* bbox) {
  if (threadIdx.x < 3) bbox[threadIdx.x] = float_to_ordered(INFINITY);
  else if (threadIdx.x < 6) bbox[threadIdx.x] = float_to_ordered(-INFINITY);
}

// The checks and FilterParams fields both entry points share (everything but the sizes and the source range).
static int fill_filter_params(const ddn_filter_config* cfg, const float* refined_all, const float* normal,
                              const float* pair_table, const float* src_table, int32_t vote_threshold, float* xyz,
                              uint8_t* votes, float* bbox, const ddn_fuse_session* mark, int64_t k_nbr, FilterParams& p) {
  DDN_REQUIRE(cfg != nullptr, "null config");
  DDN_REQUIRE(k_nbr > 0 && k_nbr <= 1024, "view counts (at most 1024 neighbours per view)");
  DDN_REQUIRE(cfg->stride >= 1, "stride");
  DDN_REQUIRE(cfg->pixel_layout == 0 || cfg->pixel_layout == 1, "pixel_layout");
  DDN_REQUIRE(refined_all && normal && pair_table && src_table && xyz && votes, "null pointer");
  DDN_REQUIRE((reinterpret_cast<uintptr_t>(pair_table) & 15) == 0 && (reinterpret_cast<uintptr_t>(src_table) & 15) == 0,
              "pair_table / src_table must be 16-byte aligned");
  p.refined_all = refined_all;
  p.normal = normal;
  p.pair_table = pair_table;
  p.src_table = src_table;
  p.xyz = xyz;
  p.votes = votes;
  p.bbox = reinterpret_cast<int*>(bbox);
  p.mark.grid = nullptr, p.mark.units = nullptr, p.mark.dirty = nullptr, p.mark.counts = nullptr;
  if (mark != nullptr) {
    DDN_REQUIRE(mark->grid && mark->units && mark->counts, "mark session: null buffer");
    p.mark.grid = reinterpret_cast<const GridDev*>(mark->grid);
    p.mark.units = reinterpret_cast<uint32_t*>(mark->units);
    p.mark.dirty = mark->dirty;
    p.mark.counts = reinterpret_cast<unsigned long long*>(mark->counts);
  }
  p.stride = cfg->stride;
  p.K = (int)k_nbr;
  // The vote byte is min(votes, 254) and the callers' clamp makes any threshold >= 255 keep every valid point.  K4
  // decides keep (and the occupancy mark) on the unsaturated count, so such a threshold must keep whatever the count:
  // then keep == (byte < min(threshold, 255)) at every threshold, and fusion and keep_mask agree with the mark.
  p.vote_threshold = vote_threshold < 255 ? vote_threshold : INT_MAX;
  p.depth_threshold = cfg->depth_threshold;
  p.grazing_cos = cfg->grazing_cos;
  p.two_sided_tau = cfg->two_sided_tau;
  p.normals_in_world = cfg->normals_in_world;
  return DDN_OK;
}

// One K4 instantiation: plain (sp == nullptr), with the support count, or with the support count and the reprojection
// test (rp != nullptr).
template <bool kBilinear, bool kStride1, bool kTwoSided, int kLayout, bool kRagged>
static int launch_k4(const FilterParams& p, const SupportParams* sp, const ReprojParams* rp, dim3 grid, const int64_t* layout,
                     size_t smem, cudaStream_t st) {
  if (rp != nullptr) {
    auto* k = backproject_filter_kernel<kBilinear, kStride1, kTwoSided, kLayout, kRagged, ReprojParams>;
    DDN_TRY(check_cuda(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), "cudaFuncSetAttribute"));
    k<<<grid, kFilterThreads, smem, st>>>(p, layout, *rp);
  } else if (sp == nullptr) {
    auto* k = backproject_filter_kernel<kBilinear, kStride1, kTwoSided, kLayout, kRagged>;
    DDN_TRY(check_cuda(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), "cudaFuncSetAttribute"));
    k<<<grid, kFilterThreads, smem, st>>>(p, layout);
  } else {
    auto* k = backproject_filter_kernel<kBilinear, kStride1, kTwoSided, kLayout, kRagged, SupportParams>;
    DDN_TRY(check_cuda(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), "cudaFuncSetAttribute"));
    k<<<grid, kFilterThreads, smem, st>>>(p, layout, *sp);
  }
  return DDN_OK;
}

// Launches the K4 instantiation cfg selects: the uniform kernel (layout == nullptr, grid = chunks x views) or the
// ragged one (grid = all chunks of the layout); sp != nullptr: the support form; rp != nullptr: the reprojection form.
static int launch_filter(const ddn_filter_config* cfg, const FilterParams& p, const SupportParams* sp, const ReprojParams* rp,
                         dim3 grid, const int64_t* layout, cudaStream_t st) {
  const int pl = cfg->pixel_layout;
  const size_t smem = (size_t)(16 + p.K * (DDN_PAIR_TABLE_FLOATS + (rp != nullptr ? 4 : 0)) + (pl == 0 ? kFilterChunk * 3 : 0)) *
                      sizeof(float);
  const bool bil = cfg->sample_mode == 1;
  const bool s1 = cfg->stride == 1;
  const bool two = cfg->two_sided_tau > 0.f;
  DDN_REQUIRE(two || cfg->depth_threshold > 0.f, "depth_threshold must be positive");
#define DDN_LAUNCH_FILTER(B, S, T, L)                                                      \
  do {                                                                                     \
    if (layout != nullptr) DDN_TRY((launch_k4<B, S, T, L, true>(p, sp, rp, grid, layout, smem, st))); \
    else DDN_TRY((launch_k4<B, S, T, L, false>(p, sp, rp, grid, nullptr, smem, st)));      \
  } while (0)
#define DDN_LAUNCH_FILTER_L(B, S, T)       \
  do {                                     \
    if (pl == 1) DDN_LAUNCH_FILTER(B, S, T, 1); \
    else DDN_LAUNCH_FILTER(B, S, T, 0);    \
  } while (0)
  if (two) {
    if (bil && s1) DDN_LAUNCH_FILTER_L(true, true, true);
    else if (bil) DDN_LAUNCH_FILTER_L(true, false, true);
    else if (s1) DDN_LAUNCH_FILTER_L(false, true, true);
    else DDN_LAUNCH_FILTER_L(false, false, true);
  } else {
    if (bil && s1) DDN_LAUNCH_FILTER_L(true, true, false);
    else if (bil) DDN_LAUNCH_FILTER_L(true, false, false);
    else if (s1) DDN_LAUNCH_FILTER_L(false, true, false);
    else DDN_LAUNCH_FILTER_L(false, false, false);
  }
#undef DDN_LAUNCH_FILTER_L
#undef DDN_LAUNCH_FILTER
  return DDN_OK;
}

static int check_support(const SupportParams* sp) {
  if (sp == nullptr) return DDN_OK;
  DDN_REQUIRE(sp->min_support >= 0 && sp->min_support <= 1024, "min_support must be in [0, 1024]");
  DDN_REQUIRE(sp->support_tau > 0.f && isfinite(sp->support_tau), "support_tau must be positive and finite");
  DDN_REQUIRE(sp->support != nullptr, "null support");
  return DDN_OK;
}

// The reprojection form's argument (reproj_px > 0, checked by its entry points: the form is on; 0: off) -> rp, or
// nullptr when off.
static int reproj_params(const SupportParams* sp, float reproj_px, ReprojParams& r, const ReprojParams*& rp) {
  rp = nullptr;
  if (reproj_px == 0.f) return DDN_OK;
  r = ReprojParams{*sp, reproj_px * reproj_px};
  rp = &r;
  return DDN_OK;
}

// The three uniform entry points (sup: nullptr for ddn_backproject_filter; reproj_px: 0 but for the reprojection form).
static int filter_uniform(const SupportParams* sup, float reproj_px, const ddn_filter_config* cfg, int64_t n_views_total, int64_t src_begin,
                          int64_t n_src, int64_t height, int64_t width, int64_t k_nbr, const float* refined_all,
                          const float* normal, const int32_t* nbr, const float* pair_table, const float* src_table,
                          int32_t vote_threshold, float* xyz, uint8_t* votes, float* bbox, const ddn_fuse_session* mark,
                          void* stream) {
  (void)nbr;
  DDN_REQUIRE(n_views_total > 0 && n_src >= 0, "view counts");
  DDN_REQUIRE(src_begin >= 0 && src_begin + n_src <= n_views_total, "source range");
  DDN_REQUIRE(height > 0 && width > 0 && height * width < (1ll << 31), "image size");
  DDN_REQUIRE(n_views_total * height * width < (1ll << 32), "refined_all must hold fewer than 2^32 pixels (32-bit gather offsets)");
  DDN_REQUIRE(width < (1 << 22) && height < (1 << 22), "image side too large for the truncation trick");
  FilterParams p;
  DDN_TRY(fill_filter_params(cfg, refined_all, normal, pair_table, src_table, vote_threshold, xyz, votes, bbox, mark, k_nbr, p));
  DDN_TRY(check_support(sup));
  ReprojParams rpv;
  const ReprojParams* rp;
  DDN_TRY(reproj_params(sup, reproj_px, rpv, rp));
  if (n_src == 0) return DDN_OK;
  p.src_begin = (int)src_begin;
  p.n_src = (int)n_src;
  p.H = (int)height;
  p.W = (int)width;
  p.Hs = (p.H + p.stride - 1) / p.stride;
  p.Ws = (p.W + p.stride - 1) / p.stride;
  {
    const float wf = (float)p.W, hf = (float)p.H;
    memcpy(&p.wbits, &wf, 4);
    memcpy(&p.hbits, &hf, 4);
  }
  const int Ps = p.Hs * p.Ws;
  dim3 grid((Ps + kFilterChunk - 1) / kFilterChunk, (unsigned)n_src);
  DDN_REQUIRE(n_src <= 65535, "too many source views per call");
  DDN_TRY(launch_filter(cfg, p, sup, rp, grid, nullptr, (cudaStream_t)stream));
  return after_launch("backproject_filter_kernel");
}

// The three ragged entry points (sup: nullptr for ddn_backproject_filter_ragged; reproj_px as in filter_uniform).
static int filter_ragged(const SupportParams* sup, float reproj_px, const ddn_filter_config* cfg, int64_t n_views, int64_t k_nbr,
                         const int64_t* layout, const int64_t* layout_host, const float* refined_all, const float* normal,
                         const float* pair_table, const float* src_table, int32_t vote_threshold, float* xyz,
                         uint8_t* votes, float* bbox, const ddn_fuse_session* mark, void* stream) {
  FilterParams p;
  DDN_TRY(fill_filter_params(cfg, refined_all, normal, pair_table, src_table, vote_threshold, xyz, votes, bbox, mark, k_nbr, p));
  DDN_TRY(check_support(sup));
  ReprojParams rpv;
  const ReprojParams* rp;
  DDN_TRY(reproj_params(sup, reproj_px, rpv, rp));
  DDN_REQUIRE(layout != nullptr, "null layout");
  DDN_TRY(check_layout(n_views, layout_host));
  DDN_REQUIRE(cfg->stride == layout_host[n_views * DDN_LAYOUT_COLS], "cfg->stride must be the layout's stride");
  p.src_begin = 0;
  p.n_src = (int)n_views;
  p.H = p.W = p.Hs = p.Ws = 0;  // per view, from the layout and the table entries
  p.wbits = p.hbits = 0;
  const int64_t chunks = layout_host[n_views * DDN_LAYOUT_COLS + 5];  // >= 1: every view has a pixel
  DDN_TRY(launch_filter(cfg, p, sup, rp, dim3((unsigned)chunks), layout, (cudaStream_t)stream));
  return after_launch("backproject_filter_kernel");
}

}  // namespace ddn

extern "C" {

int ddn_build_pair_tables(int64_t n_views_total, int64_t src_begin, int64_t n_src, int64_t k_nbr, int64_t height,
                          int64_t width, const double* cam_from_world, const double* intr, const int32_t* nbr,
                          float* pair_table, float* src_table, void* stream) {
  using namespace ddn;
  DDN_REQUIRE(n_views_total > 0 && n_src >= 0 && k_nbr > 0, "view counts");
  DDN_REQUIRE(height > 0 && width > 0 && height * width < (1ll << 31), "image size");
  DDN_REQUIRE(src_begin >= 0 && src_begin + n_src <= n_views_total, "source range");
  DDN_REQUIRE(cam_from_world && intr && nbr && pair_table && src_table, "null pointer");
  if (n_src == 0) return DDN_OK;
  const int total = (int)(n_src * k_nbr + n_src);
  build_pair_tables_kernel<<<(total + 127) / 128, 128, 0, (cudaStream_t)stream>>>(
      (int)n_views_total, (int)src_begin, (int)n_src, (int)k_nbr, (unsigned)(height * width), (unsigned)width, cam_from_world, intr,
      nbr, pair_table, src_table);
  return after_launch("build_pair_tables_kernel");
}

int ddn_bbox_init(float* bbox, void* stream) {
  using namespace ddn;
  DDN_REQUIRE(bbox != nullptr, "null bbox");
  bbox_init_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(reinterpret_cast<int*>(bbox));
  return after_launch("bbox_init_kernel");
}

int ddn_backproject_filter(const ddn_filter_config* cfg, int64_t n_views_total, int64_t src_begin,
                           int64_t n_src, int64_t height, int64_t width, int64_t k_nbr,
                           const float* refined_all, const float* normal, const int32_t* nbr,
                           const float* pair_table, const float* src_table, int32_t vote_threshold,
                           float* xyz, uint8_t* votes, float* bbox, const ddn_fuse_session* mark, void* stream) {
  return ddn::filter_uniform(nullptr, 0.f, cfg, n_views_total, src_begin, n_src, height, width, k_nbr, refined_all, normal, nbr,
                             pair_table, src_table, vote_threshold, xyz, votes, bbox, mark, stream);
}

int ddn_backproject_filter_support(const ddn_filter_config* cfg, int64_t n_views_total, int64_t src_begin, int64_t n_src,
                                   int64_t height, int64_t width, int64_t k_nbr, const float* refined_all,
                                   const float* normal, const int32_t* nbr, const float* pair_table,
                                   const float* src_table, int32_t vote_threshold, int32_t min_support, float support_tau,
                                   float* xyz, uint8_t* votes, uint8_t* support, float* bbox,
                                   const ddn_fuse_session* mark, void* stream) {
  const ddn::SupportParams sup{support, min_support, support_tau};
  return ddn::filter_uniform(&sup, 0.f, cfg, n_views_total, src_begin, n_src, height, width, k_nbr, refined_all, normal, nbr,
                             pair_table, src_table, vote_threshold, xyz, votes, bbox, mark, stream);
}

int ddn_backproject_filter_support_reproj(const ddn_filter_config* cfg, int64_t n_views_total, int64_t src_begin,
                                          int64_t n_src, int64_t height, int64_t width, int64_t k_nbr,
                                          const float* refined_all, const float* normal, const int32_t* nbr,
                                          const float* pair_table, const float* src_table, int32_t vote_threshold,
                                          int32_t min_support, float support_tau, float reproj_px, float* xyz,
                                          uint8_t* votes, uint8_t* support, float* bbox, const ddn_fuse_session* mark,
                                          void* stream) {
  DDN_REQUIRE(reproj_px > 0.f && isfinite(reproj_px), "reproj_px must be positive and finite");
  const ddn::SupportParams sup{support, min_support, support_tau};
  return ddn::filter_uniform(&sup, reproj_px, cfg, n_views_total, src_begin, n_src, height, width, k_nbr, refined_all, normal,
                             nbr, pair_table, src_table, vote_threshold, xyz, votes, bbox, mark, stream);
}

int ddn_build_pair_tables_ragged(int64_t n_views, int64_t k_nbr, const int64_t* layout, const int64_t* layout_host,
                                 const double* cam_from_world, const double* intr, const int32_t* nbr, float* pair_table,
                                 float* src_table, void* stream) {
  using namespace ddn;
  DDN_REQUIRE(k_nbr > 0, "view counts");
  DDN_REQUIRE(layout != nullptr, "null layout");
  DDN_TRY(check_layout(n_views, layout_host));
  DDN_REQUIRE(cam_from_world && intr && nbr && pair_table && src_table, "null pointer");
  const int total = (int)(n_views * k_nbr + n_views);
  build_pair_tables_ragged_kernel<<<(total + 127) / 128, 128, 0, (cudaStream_t)stream>>>(
      (int)n_views, (int)k_nbr, cam_from_world, intr, nbr, pair_table, src_table, layout);
  return after_launch("build_pair_tables_ragged_kernel");
}

int ddn_backproject_filter_ragged(const ddn_filter_config* cfg, int64_t n_views, int64_t k_nbr, const int64_t* layout,
                                  const int64_t* layout_host, const float* refined_all, const float* normal,
                                  const float* pair_table, const float* src_table, int32_t vote_threshold, float* xyz,
                                  uint8_t* votes, float* bbox, const ddn_fuse_session* mark, void* stream) {
  return ddn::filter_ragged(nullptr, 0.f, cfg, n_views, k_nbr, layout, layout_host, refined_all, normal, pair_table, src_table,
                            vote_threshold, xyz, votes, bbox, mark, stream);
}

int ddn_backproject_filter_support_ragged(const ddn_filter_config* cfg, int64_t n_views, int64_t k_nbr,
                                          const int64_t* layout, const int64_t* layout_host, const float* refined_all,
                                          const float* normal, const float* pair_table, const float* src_table,
                                          int32_t vote_threshold, int32_t min_support, float support_tau, float* xyz,
                                          uint8_t* votes, uint8_t* support, float* bbox, const ddn_fuse_session* mark,
                                          void* stream) {
  const ddn::SupportParams sup{support, min_support, support_tau};
  return ddn::filter_ragged(&sup, 0.f, cfg, n_views, k_nbr, layout, layout_host, refined_all, normal, pair_table, src_table,
                            vote_threshold, xyz, votes, bbox, mark, stream);
}

int ddn_backproject_filter_support_reproj_ragged(const ddn_filter_config* cfg, int64_t n_views, int64_t k_nbr,
                                                 const int64_t* layout, const int64_t* layout_host, const float* refined_all,
                                                 const float* normal, const float* pair_table, const float* src_table,
                                                 int32_t vote_threshold, int32_t min_support, float support_tau,
                                                 float reproj_px, float* xyz, uint8_t* votes, uint8_t* support, float* bbox,
                                                 const ddn_fuse_session* mark, void* stream) {
  DDN_REQUIRE(reproj_px > 0.f && isfinite(reproj_px), "reproj_px must be positive and finite");
  const ddn::SupportParams sup{support, min_support, support_tau};
  return ddn::filter_ragged(&sup, reproj_px, cfg, n_views, k_nbr, layout, layout_host, refined_all, normal, pair_table,
                            src_table, vote_threshold, xyz, votes, bbox, mark, stream);
}

}  // extern "C"
