// Per-point oriented normals on the back-projection grid (include/ddn_b200.h: ddn_point_normals): one streaming pass
// that reads each grid point's vote byte and the camera-frame normal at its pixel, rotates the normal into the world,
// normalises it, turns it toward the camera and writes it in the order of K4's xyz.  The fused-normal forms of the
// fusion paths (fuse.cu, fuse_hash.cu) then sum these per voxel.
#include "common.cuh"

namespace ddn {

constexpr int kNormalThreads = 256;
constexpr int kNormalPX = kFilterChunkPoints / kNormalThreads;  // points per thread: a CTA covers one consistency chunk

// kRagged: one flat grid over the chunks of all views (layout column 5, as K4's ragged form); otherwise blockIdx.y is
// the view and blockIdx.x the chunk.  The normal map may be pinned host memory (read in place over PCIe).
template <bool kRagged>
__global__ void __launch_bounds__(kNormalThreads)
point_normals_kernel(int n_views, int height, int width, int stride, const int64_t* __restrict__ layout, const float* __restrict__ normal,
                     const double* __restrict__ poses, const double* __restrict__ intr, const uint8_t* __restrict__ votes,
                     float* __restrict__ out) {
  __shared__ float s_cam[13];  // R row-major, then fx, fy, cx, cy
  int v, H, W;
  int64_t pix0, grid0, chunk;
  if (kRagged) {
    v = layout_view_of(layout, n_views, 5, blockIdx.x);
    const int64_t* L = layout + (size_t)v * DDN_LAYOUT_COLS;
    H = (int)L[0], W = (int)L[1], pix0 = L[2], grid0 = L[3], chunk = (int64_t)blockIdx.x - L[5];
    stride = (int)layout[(size_t)n_views * DDN_LAYOUT_COLS];
  } else {
    v = (int)blockIdx.y, H = height, W = width, chunk = blockIdx.x;
    const int64_t hs = (H + stride - 1) / stride, ws = (W + stride - 1) / stride;
    pix0 = (int64_t)v * H * W, grid0 = (int64_t)v * hs * ws;
  }
  const int tid = threadIdx.x;
  if (tid < 13) s_cam[tid] = (float)(tid < 9 ? __ldg(poses + (size_t)v * 12 + (tid / 3) * 4 + tid % 3) : __ldg(intr + (size_t)v * 4 + tid - 9));
  __syncthreads();
  const int ws = (W + stride - 1) / stride, ps = (H + stride - 1) / stride * ws;
  const float fx = s_cam[9], fy = s_cam[10], cx = s_cam[11], cy = s_cam[12];
#pragma unroll
  for (int j = 0; j < kNormalPX; ++j) {
    const int q = (int)chunk * kFilterChunkPoints + j * kNormalThreads + tid;
    if (q >= ps) break;
    const int ys = q / ws, xs = q - ys * ws;
    float o0 = 0.f, o1 = 0.f, o2 = 0.f;
    if (__ldg(votes + grid0 + q) != 255) {
      const int x = xs * stride, y = ys * stride;
      const float* np_ = normal + (size_t)(pix0 + (int64_t)y * W + x) * 3;
      const float n0 = __ldg(np_ + 0), n1 = __ldg(np_ + 1), n2 = __ldg(np_ + 2);
      float w[3];
#pragma unroll
      for (int i = 0; i < 3; ++i) w[i] = fmaf(s_cam[i], n0, fmaf(s_cam[3 + i], n1, s_cam[6 + i] * n2));  // R^T n
      const float inv = 1.0f / (sqrtf(fmaf(w[0], w[0], fmaf(w[1], w[1], w[2] * w[2]))) + 1e-8f);
      // facing away from the camera (n_c . ray > 0, ray = ((x - cx) / fx, (y - cy) / fy, 1)): negate
      const float dot = fmaf(n0, ((float)x - cx) / fx, fmaf(n1, ((float)y - cy) / fy, n2));
      const float sgn = dot > 0.f ? -inv : inv;
      o0 = w[0] * sgn, o1 = w[1] * sgn, o2 = w[2] * sgn;
      if (!(isfinite(o0) && isfinite(o1) && isfinite(o2))) o0 = o1 = o2 = 0.f;
    }
    float* op = out + (size_t)(grid0 + q) * 3;
    op[0] = o0, op[1] = o1, op[2] = o2;
  }
}

}  // namespace ddn

extern "C" {

int ddn_point_normals(int64_t n_views, int64_t height, int64_t width, int32_t stride, const float* normal, const double* cam_from_world,
                      const double* intr, const uint8_t* votes, float* normal_out, void* stream) {
  using namespace ddn;
  DDN_REQUIRE(n_views >= 0 && n_views <= 65535, "n_views must be in [0, 65535]");
  DDN_REQUIRE(height >= 1 && width >= 1 && height < (1 << 22) && width < (1 << 22) && height * width < (1ll << 31),
              "every side must be 1 .. 2^22 - 1 and a view below 2^31 pixels");
  DDN_REQUIRE(stride >= 1, "stride must be >= 1");
  if (n_views == 0) return DDN_OK;
  DDN_REQUIRE(normal && cam_from_world && intr && votes && normal_out, "null pointer");
  const int64_t hs = (height + stride - 1) / stride, ws = (width + stride - 1) / stride;
  const dim3 grid((unsigned)((hs * ws + kFilterChunkPoints - 1) / kFilterChunkPoints), (unsigned)n_views);
  point_normals_kernel<false><<<grid, kNormalThreads, 0, (cudaStream_t)stream>>>((int)n_views, (int)height, (int)width, stride, nullptr,
                                                                               normal, cam_from_world, intr, votes, normal_out);
  return after_launch("point_normals_kernel", (cudaStream_t)stream);
}

int ddn_point_normals_ragged(int64_t n_views, const int64_t* layout, const int64_t* layout_host, const float* normal,
                             const double* cam_from_world, const double* intr, const uint8_t* votes, float* normal_out, void* stream) {
  using namespace ddn;
  DDN_TRY(check_layout(n_views, layout_host));
  DDN_REQUIRE(layout && normal && cam_from_world && intr && votes && normal_out, "null pointer");
  const int64_t chunks = layout_host[n_views * DDN_LAYOUT_COLS + 5];
  if (chunks == 0) return DDN_OK;
  point_normals_kernel<true><<<(unsigned)chunks, kNormalThreads, 0, (cudaStream_t)stream>>>((int)n_views, 0, 0, 0, layout, normal,
                                                                                          cam_from_world, intr, votes, normal_out);
  return after_launch("point_normals_kernel", (cudaStream_t)stream);
}

}  // extern "C"
