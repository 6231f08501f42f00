// Host check of ddn::voxel_floor (depthdensifier_b200/csrc/voxel_quotient.cuh) against floorf(a / v) in IEEE
// float32.  Built and run by tests/test_voxel_quotient.py with -O2 -ffp-contract=off -fopenmp.
//   exhaustive V        every float32 bit pattern of a at voxel size V (given as float32 bits, hex)
//   boundaries N SEED   N random voxel sizes in [1e-4, 10] (and their neighbours at significands 1 and 2):
//                       the 129 floats nearest every boundary k * v, 1 <= |k| <= 2^21
// Prints "checked <count> mismatches <count>" and the first few counterexamples.
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <random>
#include <vector>

#include "../depthdensifier_b200/csrc/voxel_quotient.cuh"

static float from_bits(uint32_t u) {
  float f;
  memcpy(&f, &u, sizeof(f));
  return f;
}

static long long g_bad = 0;

// One a at voxel v; a mismatch is a different bit pattern of the floor (NaN matches NaN).
static inline bool same(float a, float v, float rv) {
  const float got = ddn::voxel_floor(a, v, rv);
  const float want = floorf(a / v);
  if (isnan(got) && isnan(want)) return true;
  return ddn::voxel_f32_bits(got) == ddn::voxel_f32_bits(want);
}

static void report(float a, float v, float rv) {
#pragma omp critical
  {
    if (g_bad < 8)
      printf("counterexample: v=%a a=%a voxel_floor=%a floorf(a/v)=%a\n", v, a, ddn::voxel_floor(a, v, rv), floorf(a / v));
    ++g_bad;
  }
}

static long long exhaustive(float v) {
  const float rv = 1.0f / v;
#pragma omp parallel for schedule(dynamic, 64)
  for (long long hi = 0; hi < (1ll << 16); ++hi) {
    for (uint32_t lo = 0; lo < (1u << 16); ++lo) {
      const float a = from_bits(((uint32_t)hi << 16) | lo);
      if (!same(a, v, rv)) report(a, v, rv);
    }
  }
  return 1ll << 32;
}

static long long boundaries(float v) {
  const float rv = 1.0f / v;
  const int kmax = 1 << 21;
#pragma omp parallel for schedule(dynamic, 64)
  for (int k = 1; k <= kmax; ++k) {
    for (int s = -1; s <= 1; s += 2) {
      const float c = (float)((double)s * (double)k * (double)v);  // nearest float to the boundary
      const uint32_t cb = ddn::voxel_f32_bits(c);
      for (int d = -64; d <= 64; ++d) {
        const float a = from_bits(cb + (uint32_t)d);  // same sign: |c| >= v > 2^-14, far from zero in ulps
        if (!same(a, v, rv)) report(a, v, rv);
      }
    }
  }
  return 2ll * kmax * 129;
}

int main(int argc, char** argv) {
  long long n = 0;
  if (argc == 3 && strcmp(argv[1], "exhaustive") == 0) {
    n = exhaustive(from_bits((uint32_t)strtoul(argv[2], nullptr, 16)));
  } else if (argc == 4 && strcmp(argv[1], "boundaries") == 0) {
    const int nv = atoi(argv[2]);
    std::mt19937 rng((unsigned)atoi(argv[3]));
    std::uniform_real_distribution<double> lg(log(1e-4), log(10.0));
    std::vector<float> vs;
    for (int i = 0; i < nv; ++i) {
      const float v = (float)exp(lg(rng));
      vs.push_back(v);
      // the same exponent with a significand at 1 + ulp and at 2 - ulp
      const uint32_t e = ddn::voxel_f32_bits(v) & 0x7f800000u;
      if (i % 8 == 0) vs.push_back(from_bits(e | 1u)), vs.push_back(from_bits(e | 0x7fffffu));
    }
    for (float v : vs) n += boundaries(v);
  } else {
    fprintf(stderr, "usage: %s exhaustive <v bits hex> | boundaries <n> <seed>\n", argv[0]);
    return 2;
  }
  printf("checked %lld mismatches %lld\n", n, g_bad);
  return g_bad == 0 ? 0 : 1;
}
