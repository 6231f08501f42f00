// Shared definitions of the hashed fusion path: the table, its probe, the radix sort of the voxel keys and the
// finalisation in key order.  Used by the one-GPU form (fuse_hash.cu) and by the multi-GPU form (fuse_hash_peers.cu:
// per-rank partial records, owner-side merge over peer memory).
#pragma once

#include <cooperative_groups.h>

#include "fuse_common.cuh"

namespace ddn {

namespace cg = cooperative_groups;

constexpr uint64_t kEmptyKey = ~0ull;      // also the table index's empty word (all bits set)
constexpr uint64_t kTombBit = 1ull << 63;  // no canonical key (3 x 21 bits) uses bit 63
constexpr uint32_t kNoIndex = 0xffffffffu;  // table index not yet published; slot-list entry unused
constexpr uint32_t kSkipIndex = 0xfffffffeu;  // tombstoned cell (or a full table)
constexpr int kHashAccWords = 5;            // sx, sy, sz, r:g, b:count (u64 each), as in fuse.cu
constexpr int kSortThreads = 512, kSortWarps = kSortThreads / 32, kRadixBins = 256;
constexpr int kSortCtas = kNumSMs;  // one resident CTA per SM (cooperative launch)
constexpr int kHashTilesPerWarp = 8;
constexpr int kHashCtas = kNumSMs * 8;  // persistent grid of the point passes
constexpr int kHashTileW = 16;
constexpr int kCompactPerThread = 8;

// ddn_hash_fuse.state words
enum { kStActive = 0, kStStatus = 1, kStTombs = 2 };

struct HashDev {
  unsigned long long* keys;  // [cap_slots]
  uint32_t* index;           // [cap_slots] voxel index of the slot's key
  uint32_t* slots;           // [cap_voxels]: voxel (= point) i -> its slot, tombstone j -> slot at cap_voxels - 1 - j
  unsigned long long* sort_keys;  // [2, cap_voxels]
  uint32_t* sort_index;           // [2, cap_voxels]
  uint32_t* hist;                 // [kRadixBins, kSortCtas]
  unsigned long long* state;
  long long cap_slots, cap_voxels;
  int shift;  // 64 - log2(cap_slots)
};

// First slot of a key's probe sequence.  The 64 cells of a 4 x 4 x 4 brick share one hashed 64-slot block (in key
// order inside it), so neighbouring points - consecutive pixels, the next tile of a warp - probe the same few cache
// lines instead of random ones.  The tombstone bit does not enter the hash: a cell's live key probes through its
// tombstone.
__device__ __forceinline__ uint64_t hash_slot(const HashDev& h, uint64_t key) {
  const uint64_t kx = key & 0x1fffff, ky = (key >> 21) & 0x1fffff, kz = (key >> 42) & 0x1fffff;
  const uint64_t brick = (kx >> 2) | ((ky >> 2) << 19) | ((kz >> 2) << 38);
  const uint64_t sub = (kx & 3) | ((ky & 3) << 2) | ((kz & 3) << 4);
  return (((brick * 0x9E3779B97F4A7C15ull) >> h.shift) & ~63ull) | sub;
}
__device__ __forceinline__ uint64_t ld_relaxed_u64(const unsigned long long* p) {
  uint64_t v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ uint32_t ld_acquire_u32(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_u32(uint32_t* p, uint32_t v) {
  asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint64_t canonical_key(uint32_t kx, uint32_t ky, uint32_t kz) {
  return (uint64_t)kx | ((uint64_t)ky << 21) | ((uint64_t)kz << 42);
}

// Voxel index of `key`: found, or inserted with `self` (the inserting point's index) as its index.  The inserter
// zeroes the accumulator (kHashAccWords words at accum + self * kStride) before it publishes the index with release
// semantics; the others acquire it before their REDs.  kSkipIndex for a tombstoned cell.
template <int kStride = kHashAccWords>
__device__ __forceinline__ uint32_t hash_voxel_index(const HashDev& h, uint64_t key, uint32_t self, unsigned long long* __restrict__ accum) {
  uint64_t s = hash_slot(h, key);
  const uint64_t mask = (uint64_t)(h.cap_slots - 1);
#pragma unroll 1
  for (long long p = 0; p < h.cap_slots; ++p, s = (s + 1) & mask) {
    uint64_t cur = ld_relaxed_u64(h.keys + s);
    if (cur == kEmptyKey) {
      cur = atomicCAS(h.keys + s, kEmptyKey, key);
      if (cur == kEmptyKey) {
        h.slots[self] = (uint32_t)s;
        unsigned long long* a = accum + (size_t)self * kStride;
#pragma unroll
        for (int q = 0; q < kHashAccWords; ++q) a[q] = 0ull;
        st_release_u32(h.index + s, self);
        return self;
      }
    }
    if (cur == key) {
      uint32_t v;
      while ((v = ld_acquire_u32(h.index + s)) == kNoIndex) {
      }
      return v;
    }
    if (cur == (key | kTombBit)) return kSkipIndex;
  }
  h.state[kStStatus] = 1ull;
  return kSkipIndex;
}

// Radix sort of the step's voxels, then an epilogue in key order; the body of the one cooperative launch of
// kSortCtas x kSortThreads that ends every hashed form.  The sort is LSD over the compact key (kx | ky << bx | kz <<
// (bx + by), which orders as the canonical key: by kz, ky, kx) in 8-bit digits, ceil((bx + by + bz) / 8) passes.  Each
// CTA owns a contiguous chunk of the M (compact key, voxel index) pairs hash_compact left; a pass is: per-CTA digit
// histogram -> grid sync -> every CTA derives its own scatter offsets from all histograms (digit-major prefix) ->
// stable scatter in 512-element tiles (MATCH.ANY rank inside the warp, warp-major prefix inside the tile) -> grid
// sync.  M is read from counts[1], so no host round trip.  Then epi(g, m, ka, va, gtid, gthreads): the sorted pairs
// are (ka, va)[0, m), every thread of the grid takes the elements gtid + k * gthreads.
template <class Epilogue>
__device__ __forceinline__ void hash_sort_body(const GridDev* __restrict__ gp, const HashDev& h, const long long* __restrict__ counts,
                                               Epilogue epi) {
  __shared__ uint32_t s_wcnt[kSortWarps][kRadixBins];
  __shared__ uint32_t s_off[kRadixBins];
  __shared__ uint32_t s_scan[kRadixBins / 32];
  if (h.state[kStActive] == 0) return;  // grid-uniform: no CTA reaches a grid sync
  cg::grid_group grid = cg::this_grid();
  const GridDev g = *gp;
  const long long m = min(counts[1], h.cap_voxels);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const long long gtid = (long long)blockIdx.x * kSortThreads + tid, gthreads = (long long)gridDim.x * kSortThreads;
  const int nbits = g.bx + g.by + g.bz;
  unsigned long long* ka = h.sort_keys;
  unsigned long long* kb = h.sort_keys + h.cap_voxels;
  uint32_t* va = h.sort_index;
  uint32_t* vb = h.sort_index + h.cap_voxels;
  // 1. radix passes
  const long long chunk = (m + gridDim.x - 1) / gridDim.x;
  const long long c0 = min((long long)blockIdx.x * chunk, m), c1 = min(c0 + chunk, m);
  const int passes = (nbits + 7) / 8;
  for (int pass = 0; pass < passes; ++pass) {
    const int shift = 8 * pass;
    if (tid < kRadixBins) s_off[tid] = 0u;
    __syncthreads();
    for (long long i = c0 + tid; i < c1; i += kSortThreads) atomicAdd(&s_off[(ka[i] >> shift) & 0xff], 1u);
    __syncthreads();
    if (tid < kRadixBins) h.hist[tid * gridDim.x + blockIdx.x] = s_off[tid];
    grid.sync();
    if (tid < kRadixBins) {  // offset of (digit tid, this CTA) = elements of smaller digits + of digit tid in earlier CTAs
      uint32_t total = 0, before = 0;
      for (unsigned b = 0; b < gridDim.x; ++b) {
        const uint32_t v = __ldcg(h.hist + tid * gridDim.x + b);
        before += b < blockIdx.x ? v : 0u;
        total += v;
      }
      uint32_t inc = total;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += t;
      }
      if (lane == 31) s_scan[warp] = inc;
      __syncwarp();
      s_off[tid] = inc - total + before;  // warp-local part; the earlier warps' totals are added below
    }
    __syncthreads();
    if (tid < kRadixBins) {
      uint32_t add = 0;
#pragma unroll
      for (int w = 0; w < kRadixBins / 32; ++w) add += w < warp ? s_scan[w] : 0u;
      s_off[tid] += add;
    }
    for (long long base = c0; base < c1; base += kSortThreads) {
      __syncthreads();
#pragma unroll
      for (int q = 0; q < kSortWarps * kRadixBins / kSortThreads; ++q) (&s_wcnt[0][0])[q * kSortThreads + tid] = 0u;
      const long long i = base + tid;
      const bool in = i < c1;
      const unsigned long long k = in ? ka[i] : 0ull;
      const uint32_t v = in ? va[i] : 0u;
      const uint32_t d = in ? (uint32_t)((k >> shift) & 0xff) : (uint32_t)kRadixBins;
      __syncthreads();
      const uint32_t peers = __match_any_sync(0xffffffffu, d);
      const uint32_t rank = __popc(peers & ((1u << lane) - 1u));
      if (in && rank == 0) s_wcnt[warp][d] = (uint32_t)__popc(peers);
      __syncthreads();
      if (tid < kRadixBins) {
        uint32_t run = s_off[tid];
#pragma unroll
        for (int w = 0; w < kSortWarps; ++w) {
          const uint32_t c = s_wcnt[w][tid];
          s_wcnt[w][tid] = run;
          run += c;
        }
        s_off[tid] = run;
      }
      __syncthreads();
      if (in) {
        const uint32_t pos = s_wcnt[warp][d] + rank;
        kb[pos] = k;
        vb[pos] = v;
      }
    }
    grid.sync();
    unsigned long long* tk = ka;
    ka = kb, kb = tk;
    uint32_t* tv = va;
    va = vb, vb = tv;
  }
  // 2. epilogue in key order
  epi(g, m, ka, va, gtid, gthreads);
}

// The finalising epilogue (finalize_kernel's arithmetic, the accumulator read through the sorted index): the voxel of
// sorted element r has its kHashAccWords sums at accum + va[r] * kStride.
template <int kStride>
struct HashFinalize {
  long long* counts;
  long long cap;
  uint64_t* out_keys;
  float* out_xyz;
  uint8_t* out_rgb;
  int32_t* out_count;
  const unsigned long long* accum;
  __device__ __forceinline__ void operator()(const GridDev& g, long long m, const unsigned long long* ka, const uint32_t* va,
                                             long long gtid, long long gthreads) const {
    const int bx = g.bx, by = g.by;
    const uint64_t mx = (1ull << bx) - 1, my = (1ull << by) - 1;
    for (long long r = gtid; r < min(m, cap); r += gthreads) {
      const uint32_t idx = va[r];
      const uint64_t ck = ka[r];
      const uint32_t kx = (uint32_t)(ck & mx), ky = (uint32_t)((ck >> bx) & my), kz = (uint32_t)(ck >> (bx + by));
      out_keys[r] = canonical_key(kx, ky, kz);
      const unsigned long long* a = accum + (size_t)idx * kStride;
      const long long sx = (long long)a[0], sy = (long long)a[1], sz = (long long)a[2];
      const unsigned long long rg = a[3], bn = a[4];
      const uint32_t cnt = (uint32_t)bn;
      if (cnt >= (1u << 24)) counts[0] = -1;
      out_count[r] = (int32_t)cnt;
      finalize_voxel(g, voxel_centre(g.ox, kx, g.voxel), voxel_centre(g.oy, ky, g.voxel), voxel_centre(g.oz, kz, g.voxel), sx, sy, sz,
                     rg >> 32, rg & 0xffffffffull, bn >> 32, (long long)cnt, out_xyz + r * 3, out_rgb + r * 3);
    }
  }
};

// ---- host side (fuse_hash.cu) --------------------------------------------------------------------
int hash_dev(const ddn_hash_fuse* hf, HashDev* h);
// hash_begin (mode as ddn_fuse_finish_hashed), hash_tomb over the dedup points, hash_insert over the points into
// `accum` (kHashAccWords words per point), hash_compact: the step's voxels as unsorted (compact key, index) pairs,
// their number in counts[1]
int hash_launch_points(GridDev* gp, const HashDev& h, unsigned long long* counts, int mode, int64_t n_points, int64_t row_len,
                       const float* xyz, const uint8_t* rgb, const uint8_t* votes, int thr, const float* dedup_xyz, int64_t n_dedup,
                       unsigned long long* accum, cudaStream_t st);
// hash_compact over the first n entries of the slot list
int hash_launch_compact(const GridDev* gp, const HashDev& h, int64_t n, unsigned long long* counts, cudaStream_t st);

}  // namespace ddn
