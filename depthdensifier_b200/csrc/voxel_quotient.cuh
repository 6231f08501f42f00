// The IEEE float32 quotient a / voxel of stage 4's voxel coordinate, without a division on the common path.
// Self-contained (no CUDA headers), so that a host program built with any C++ compiler evaluates exactly what the
// kernels evaluate: tests/test_voxel_quotient.py checks it against a / voxel on the CPU.
#pragma once

#include <math.h>
#include <stdint.h>
#ifndef __CUDACC__
#include <string.h>
#define __host__
#define __device__
#define __forceinline__ inline
#endif

namespace ddn {

__host__ __device__ __forceinline__ uint32_t voxel_f32_bits(float x) {
#ifdef __CUDA_ARCH__
  return __float_as_uint(x);
#else
  uint32_t u;
  memcpy(&u, &x, sizeof(u));
  return u;
#endif
}

// q = fl(a * rvoxel) with rvoxel = fl(1 / voxel) is within an ulp of a / voxel.  Markstein's correction
//   r = fma(-q, voxel, a)   (exact: the residual of a quotient within an ulp)
//   q' = fma(r, rvoxel, q)
// then rounds to the IEEE quotient fl(a / voxel) when no step over- or underflows.  voxel_quotient_in_domain(q)
// is that condition, on the estimate's exponent: 2^-126 <= |q| < 2^22.  Outside it (zero, subnormal, huge, inf or
// NaN - never at a scene's scale) the caller divides.  Up to 2^22 the floors are those of the IEEE quotient by
// tests/test_voxel_quotient.py, exhaustively over every float32 a at the voxel sizes it lists.
__host__ __device__ __forceinline__ bool voxel_quotient_in_domain(float q) {
  return (voxel_f32_bits(q) & 0x7fffffffu) - 0x00800000u < 0x4a800000u - 0x00800000u;
}
__host__ __device__ __forceinline__ float voxel_quotient_fix(float a, float q, float voxel, float rvoxel) {
  return fmaf(fmaf(-q, voxel, a), rvoxel, q);
}
__host__ __device__ __forceinline__ float voxel_divide(float a, float voxel) {
#ifdef __CUDA_ARCH__
  return __fdiv_rn(a, voxel);
#else
  return a / voxel;
#endif
}

// floor(fl(a / voxel)) bit for bit (SURVEY.md N4: numpy divides, and x / v and x * (1 / v) round differently).
__host__ __device__ __forceinline__ float voxel_floor(float a, float voxel, float rvoxel) {
#ifdef __CUDA_ARCH__
  const float q = __fmul_rn(a, rvoxel);
#else
  const float q = a * rvoxel;
#endif
  if (!voxel_quotient_in_domain(q)) return floorf(voxel_divide(a, voxel));
  return floorf(voxel_quotient_fix(a, q, voxel, rvoxel));
}

}  // namespace ddn

#ifndef __CUDACC__
#undef __host__
#undef __device__
#undef __forceinline__
#endif
