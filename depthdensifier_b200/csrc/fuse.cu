// Stage 4: voxel-grid fusion (new capability, SURVEY.md §8 row N4; the reference only concatenates
// points, scripts/test.py:353-359).  DENSE-RANK PATH - no sort.
//
// The voxel grid of a scene is small enough for one occupancy BIT per cell (cfg 2: about 2400 x 2400 x 600
// cells = 0.6 GB of occupancy units in 180 GB of HBM).  Bit order == key order (x fastest, then y, then z), so
// the rank of a set bit among all set bits IS the voxel's position in the key-sorted output.  That
// replaces the radix sort of 168 M (key, index) pairs by streaming passes:
//
//   mark        every participating point sets the bit of its cell (RED.OR; a cell equal to the
//               previous point's is skipped).  In the pipeline this happens in K4's epilogue
//               (filter.cu) while the point is still in registers; mark_points_kernel is the
//               stand-alone form.
//   rank        popcount scan over the occupancy: one exclusive prefix per 96-bit unit, stored in the
//               unit's fourth word; the pass also emits the sorted keys
//   accumulate  integer fixed-point sums per voxel with 64-bit RED.ADD.  The L2 atomic units bound this
//               pass, so a warp first merges the points of its 16 x 2 pixel tile that share a cell
//               (MATCH.ANY + shuffles); the group's first lane looks the slot up (ONE 16 B load:
//               96 bits + prefix) and issues the atomics.
//   finalize    one thread per voxel: mean = centre + sum/count, colour = round-half-up
//
// Integer sums make the result independent of the order of points and of how they are split over
// ranks.  THE GRID LIVES IN DEVICE MEMORY (GridDev behind a pointer): a fusion session derives it from
// bounding boxes on the device, every grid-sized pass is a persistent kernel that reads the actual
// extent, so a whole step - and the multi-GPU exchange + merge over peer memory at the end of this
// file - runs without the host looking at any intermediate result.
// The host-grid entry points fuse grids of more than 2^35 cells with the hashed path (fuse_hash.cu).
#include <algorithm>
#include <type_traits>

#include "fuse_hash.cuh"

namespace ddn {

constexpr int kAccWords = 5;  // sx, sy, sz, r:g, b:count (u64 each)
// Partial-sum RECORD exchanged between ranks: {key, sx, sy, sz, r:g, b:count} = DDN_RECORD_WORDS u64 (Record<kW> in
// fuse_common.cuh; the fused-normal form adds the three normal sums and a zero word).  In partial mode the
// accumulators ARE words 1.. of the output records (stride kW), so there is no finalisation pass and a destination's
// share of the sorted records is one contiguous slice.
constexpr int kRecWords = DDN_RECORD_WORDS;
static_assert(kRecWords == kAccWords + 1, "record = key + accumulators");
constexpr uint64_t kDenseMaxCells = 1ull << 35;  // 5.7 GB of units
constexpr int kPersistentCtas = kNumSMs * 8;

__device__ __forceinline__ uint64_t cell_of_key(const GridDev& g, uint64_t key) {
  const uint64_t kx = key & 0x1fffff, ky = (key >> 21) & 0x1fffff, kz = (key >> 42) & 0x1fffff;
  if ((key >> 63) || kx >= (uint64_t)g.nx || ky >= (uint64_t)g.ny || kz >= (uint64_t)g.nz) return kNoCell;
  return kx + (uint64_t)g.nx * (ky + (uint64_t)g.ny * kz);
}

// ---- session set-up -------------------------------------------------------------------------------
struct BoxPtrs {
  const int* p[DDN_MAX_PEERS];
  int n;
};

// Grid from the union of n encoded bounding boxes (possibly in peer memory).  origin = (floor(min / voxel)
// - 1) * voxel, dims = floor((max - origin) / voxel) + 2: one cell of slack on either side, so float32
// rounding of the origin can never push a boxed point out of the grid.
__global__ void grid_from_bbox_kernel(BoxPtrs boxes, float voxel, long long cap_units, GridDev* __restrict__ out,
                                      unsigned long long* __restrict__ counts) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  int lo[3] = {0x7fffffff, 0x7fffffff, 0x7fffffff}, hi[3] = {(int)0x80000000, (int)0x80000000, (int)0x80000000};
  for (int b = 0; b < boxes.n; ++b)
    for (int i = 0; i < 3; ++i) {
      lo[i] = min(lo[i], __ldcv(boxes.p[b] + i));
      hi[i] = max(hi[i], __ldcv(boxes.p[b] + 3 + i));
    }
  GridDev g;
  g.voxel = voxel;
  g.status = DDN_GRID_OK;
  g.reserved = 0;
  float o[3] = {0.f, 0.f, 0.f};
  int dims[3] = {0, 0, 0}, bits[3] = {1, 1, 1};
  for (int i = 0; i < 3; ++i) {
    float flo = ordered_to_float(lo[i]), fhi = ordered_to_float(hi[i]);
    if (!(fabsf(flo) < INFINITY) || !(fabsf(fhi) < INFINITY) || flo > fhi) {
      g.status = DDN_GRID_EMPTY;
      continue;
    }
    // the box may come from another kernel's float32 arithmetic (K3's tile corners): widen it by ~32 ulp
    const float slack = 4e-6f * fmaxf(fabsf(flo), fabsf(fhi));
    flo -= slack, fhi += slack;
    o[i] = __fmul_rn(floorf(__fdiv_rn(flo, voxel)) - 1.f, voxel);
    const float c = floorf(__fdiv_rn(__fsub_rn(fhi, o[i]), voxel)) + 2.f;
    if (!(c <= 2097152.f)) {
      if (g.status == DDN_GRID_OK) g.status = DDN_GRID_TOO_MANY_BITS;
      continue;
    }
    dims[i] = (int)c;
    int bb = 1;
    while ((1 << bb) < dims[i]) ++bb;
    bits[i] = bb;
  }
  g.ox = o[0], g.oy = o[1], g.oz = o[2];
  g.nx = dims[0], g.ny = dims[1], g.nz = dims[2];
  g.bx = bits[0], g.by = bits[1], g.bz = bits[2];
  g.cells = (long long)dims[0] * (long long)dims[1] * (long long)dims[2];
  g.n_units = (g.cells + kUnitBits - 1) / kUnitBits;
  if (g.status == DDN_GRID_OK && g.n_units > cap_units) g.status = DDN_GRID_TOO_LARGE;
  if (g.status != DDN_GRID_OK) g.n_units = 0;
  *out = g;
  counts[0] = 0ull;
  counts[1] = 0ull;
}

__global__ void grid_store_kernel(GridDev g, long long cap_units, GridDev* __restrict__ out, unsigned long long* __restrict__ counts) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  if (g.n_units > cap_units) g.status = DDN_GRID_TOO_LARGE, g.n_units = 0;
  *out = g;
  counts[0] = 0ull;
  counts[1] = 0ull;
}

// Clears the occupancy for a new step.  With dirty flags only the scan tiles the previous step touched are
// cleared (and their flags reset); without, the units the new grid uses.
__global__ void __launch_bounds__(256)
clear_units_kernel(const GridDev* __restrict__ gp, uint4* __restrict__ units, uint8_t* __restrict__ dirty, long long cap_units) {
  if (dirty != nullptr) {
    const long long cap_tiles = (cap_units + kTileUnits - 1) / kTileUnits;
    for (long long t = blockIdx.x; t < cap_tiles; t += gridDim.x) {
      if (dirty[t] == 0) continue;  // CTA-uniform
      const long long u0 = t * kTileUnits, u1 = min(u0 + (long long)kTileUnits, cap_units);
      for (long long u = u0 + threadIdx.x; u < u1; u += blockDim.x) units[u] = make_uint4(0, 0, 0, 0);
      __syncthreads();
      if (threadIdx.x == 0) dirty[t] = 0;
    }
    return;
  }
  const long long n = gp->n_units;
  for (long long u = (long long)blockIdx.x * blockDim.x + threadIdx.x; u < n; u += (long long)gridDim.x * blockDim.x)
    units[u] = make_uint4(0, 0, 0, 0);
}

// ---- mark (stand-alone form) -----------------------------------------------------------------------
constexpr int kMarkPX = 4;  // consecutive points per thread

// A thread owns 4 consecutive points; a cell equal to its predecessor (in the thread, or the last cell
// of the previous lane) is not marked again.  Consecutive pixels of a depth map fall into the same or
// neighbouring voxels, so this removes most of the atomics.
template <bool kVec>
__global__ void __launch_bounds__(256)
mark_points_kernel(FuseDev f, int64_t n, const float* __restrict__ xyz, const uint8_t* __restrict__ votes, int thr) {
  __shared__ int s_count;
  const GridDev g = *f.grid;
  if (g.n_units == 0) return;
  const float rv = 1.0f / g.voxel;
  if (threadIdx.x == 0) s_count = 0;
  __syncthreads();
  const int64_t base = ((int64_t)blockIdx.x * 256 + threadIdx.x) * kMarkPX;
  uint64_t cell[kMarkPX];
  int mine = 0;
  bool take[kMarkPX];
  if (kVec && base + kMarkPX <= n) {
    uint32_t vv = 0;
    if (votes != nullptr) vv = __ldcs(reinterpret_cast<const uint32_t*>(votes + base));
#pragma unroll
    for (int j = 0; j < kMarkPX; ++j) take[j] = votes == nullptr || (int)((vv >> (8 * j)) & 0xff) < thr;
    if (take[0] | take[1] | take[2] | take[3]) {
      const float4* x4 = reinterpret_cast<const float4*>(xyz + base * 3);
      const float4 a = __ldcs(x4), b = __ldcs(x4 + 1), c = __ldcs(x4 + 2);
      const float p[12] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w, c.x, c.y, c.z, c.w};
      uint32_t kx, ky, kz;
#pragma unroll
      for (int j = 0; j < kMarkPX; ++j)
        cell[j] = take[j] ? cell_of_point(g, rv, p[j * 3], p[j * 3 + 1], p[j * 3 + 2], kx, ky, kz) : kNoCell;
    } else {
#pragma unroll
      for (int j = 0; j < kMarkPX; ++j) cell[j] = kNoCell;
    }
  } else {
#pragma unroll
    for (int j = 0; j < kMarkPX; ++j) {
      const int64_t i = base + j;
      cell[j] = kNoCell;
      if (i < n && (votes == nullptr || (int)__ldg(votes + i) < thr)) {
        uint32_t kx, ky, kz;
        cell[j] = cell_of_point(g, rv, __ldg(xyz + i * 3 + 0), __ldg(xyz + i * 3 + 1), __ldg(xyz + i * 3 + 2), kx, ky, kz);
      }
    }
  }
  uint64_t prev = __shfl_up_sync(0xffffffffu, cell[kMarkPX - 1], 1);
  if ((threadIdx.x & 31) == 0) prev = kNoCell;
#pragma unroll
  for (int j = 0; j < kMarkPX; ++j) {
    if (cell[j] != kNoCell) {
      ++mine;
      if (cell[j] != prev) set_cell_bit(f.units, f.dirty, cell[j], prev);
    }
    prev = cell[j];
  }
  mine = __reduce_add_sync(0xffffffffu, mine);
  if ((threadIdx.x & 31) == 0 && mine) atomicAdd(&s_count, mine);
  __syncthreads();
  if (threadIdx.x == 0 && s_count) atomicAdd(f.counts, (unsigned long long)s_count);
}

// records source (legacy merge): cells outside [cell_begin, cell_end) are not owned by this call
__global__ void __launch_bounds__(256)
mark_records_kernel(FuseDev f, int64_t n, const uint64_t* __restrict__ records, uint64_t cell_begin, uint64_t cell_end) {
  __shared__ int s_count;
  const GridDev g = *f.grid;
  if (g.n_units == 0) return;
  if (threadIdx.x == 0) s_count = 0;
  __syncthreads();
  const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
  uint64_t cell = i < n ? cell_of_key(g, __ldg(records + i * kRecWords)) : kNoCell;
  if (cell < cell_begin || cell >= cell_end) cell = kNoCell;
  if (cell != kNoCell) set_cell_bit(f.units, f.dirty, cell);
  const int c = __popc(__ballot_sync(0xffffffffu, cell != kNoCell));
  if ((threadIdx.x & 31) == 0 && c) atomicAdd(&s_count, c);
  __syncthreads();
  if (threadIdx.x == 0 && s_count) atomicAdd(f.counts, (unsigned long long)s_count);
}

// N5 (sparse-cloud merge with de-duplication): clears the occupancy bit of every cell that holds one of the
// given points, so the dense voxel there is never created (the sparse point itself is kept by the caller).
// Runs between the mark and the rank passes; [cell_begin, cell_end): the cells this call may touch.
__global__ void __launch_bounds__(256)
unmark_points_kernel(FuseDev f, int64_t n, const float* __restrict__ xyz, const long long* __restrict__ plan) {
  const GridDev g = *f.grid;
  if (g.n_units == 0) return;
  const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (i >= n) return;
  uint32_t kx, ky, kz;
  const uint64_t cell = cell_of_point(g, 1.0f / g.voxel, __ldg(xyz + i * 3 + 0), __ldg(xyz + i * 3 + 1), __ldg(xyz + i * 3 + 2), kx, ky, kz);
  if (cell == kNoCell) return;
  if (plan != nullptr) {
    const uint64_t cb = (uint64_t)plan[0] * kOwnUnits * kUnitBits, ce = (uint64_t)plan[1] * kOwnUnits * kUnitBits;
    if (cell < cb || cell >= ce) return;
  }
  const uint32_t w32 = (uint32_t)(cell >> 5);
  const uint32_t unit = w32 / 3u;
  atomicAnd(f.units + (size_t)unit * 4 + (w32 - unit * 3u), ~(1u << (cell & 31)));
}

// ---- rank: popcount scan over the units --------------------------------------------------------
__device__ __forceinline__ int popc3(const uint4& u) { return __popc(u.x) + __popc(u.y) + __popc(u.z); }

// Range of scan tiles a rank pass covers: [tile_begin, tile_begin + n_tiles); n_tiles < 0 = every tile of
// the device grid.
struct ScanRange {
  long long tile_begin, n_tiles;
};
__device__ __forceinline__ long long scan_tiles(const ScanRange& r, long long n_units) {
  return r.n_tiles >= 0 ? r.n_tiles : (n_units + kTileUnits - 1) / kTileUnits;
}

__device__ __forceinline__ int block_sum_256(int v, int* s_warp) {
  v = __reduce_add_sync(0xffffffffu, v);
  if ((threadIdx.x & 31) == 0) s_warp[threadIdx.x >> 5] = v;
  __syncthreads();
  int t = 0;
#pragma unroll
  for (int w = 0; w < kScanThreads / 32; ++w) t += s_warp[w];
  __syncthreads();
  return t;
}

__global__ void __launch_bounds__(kScanThreads)
tile_count_kernel(const GridDev* __restrict__ gp, const uint4* __restrict__ units, const uint8_t* __restrict__ dirty,
                  ScanRange range, uint32_t* __restrict__ tile_sums) {
  __shared__ int s_warp[kScanThreads / 32];
  const long long n_units = gp->n_units;
  const long long tiles = scan_tiles(range, n_units);
  for (long long t = blockIdx.x; t < tiles; t += gridDim.x) {
    const long long tile = range.tile_begin + t;
    if (dirty != nullptr && dirty[tile] == 0) {  // untouched since the last clean-up: empty (CTA-uniform)
      if (threadIdx.x == 0) tile_sums[t] = 0u;
      continue;
    }
    const long long base = tile * kTileUnits;
    int sum = 0;
#pragma unroll
    for (int j = 0; j < kUnitsPerThread; ++j) {
      const long long ui = base + j * kScanThreads + threadIdx.x;
      if (ui < n_units) sum += popc3(__ldg(units + ui));
    }
    const int total = block_sum_256(sum, s_warp);
    if (threadIdx.x == 0) tile_sums[t] = (uint32_t)total;
  }
}

// exclusive scan of the tile sums in place (one CTA, four entries per thread and iteration), total ->
// counts[1] and tile_sums[tiles].  plan != nullptr: the number of entries is plan[1] - plan[0] (merge over a
// device-side tile range).
__global__ void __launch_bounds__(1024)
tile_scan_kernel(const GridDev* __restrict__ gp, ScanRange range, const long long* __restrict__ plan,
                 uint32_t* __restrict__ tile_sums, unsigned long long* __restrict__ counts) {
  __shared__ uint32_t s_warp[32];
  __shared__ uint32_t s_carry;
  const long long tiles = plan != nullptr ? plan[1] - plan[0] : scan_tiles(range, gp->n_units);
  if (threadIdx.x == 0) s_carry = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (long long base = 0; base < tiles; base += 4096) {
    const long long i0 = base + 4 * threadIdx.x;
    uint32_t v[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) v[q] = i0 + q < tiles ? tile_sums[i0 + q] : 0u;
    const uint32_t mine = v[0] + v[1] + v[2] + v[3];
    uint32_t inc = mine;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const uint32_t t = __shfl_up_sync(0xffffffffu, inc, d);
      if (lane >= d) inc += t;
    }
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    if (warp == 0) {
      uint32_t w = s_warp[lane];
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, w, d);
        if (lane >= d) w += t;
      }
      s_warp[lane] = w;
    }
    __syncthreads();
    const uint32_t carry = s_carry;
    uint32_t excl = carry + (warp ? s_warp[warp - 1] : 0u) + inc - mine;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      if (i0 + q < tiles) tile_sums[i0 + q] = excl;
      excl += v[q];
    }
    __syncthreads();
    if (threadIdx.x == 1023) s_carry = carry + s_warp[31];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    counts[1] = (unsigned long long)s_carry;
    tile_sums[tiles] = s_carry;  // exclusive prefix with the total appended: [tiles + 1] entries
  }
}

// canonical keys of the set bits of one unit -> keys[slot...] (slots >= cap are dropped)
__device__ __forceinline__ void emit_unit_keys(const GridDev& g, uint64_t nxy, long long ui, const uint4& u, uint32_t slot,
                                               uint64_t* __restrict__ keys, int key_stride, long long cap) {
  const uint64_t cell0 = (uint64_t)ui * kUnitBits;
  uint32_t kz = (uint32_t)(cell0 / nxy);
  const uint64_t rem = cell0 - (uint64_t)kz * nxy;
  uint32_t ky = (uint32_t)(rem / (uint64_t)g.nx);
  const uint32_t kx0 = (uint32_t)(rem - (uint64_t)ky * (uint64_t)g.nx);
  const uint32_t w[3] = {u.x, u.y, u.z};
  uint32_t row_off = 0;  // bits of this unit that belong to earlier rows
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    uint32_t bits = w[i];
    while (bits) {
      const int b = __ffs(bits) - 1;
      bits &= bits - 1;
      uint32_t kx = kx0 + (uint32_t)(i * 32 + b) - row_off;
      while (kx >= (uint32_t)g.nx) {  // the unit straddles a row end
        kx -= (uint32_t)g.nx;
        row_off += (uint32_t)g.nx;
        if (++ky >= (uint32_t)g.ny) ky = 0, ++kz;
      }
      if ((long long)slot < cap) keys[(size_t)slot * key_stride] = (uint64_t)kx | ((uint64_t)ky << 21) | ((uint64_t)kz << 42);
      ++slot;
    }
  }
}

// Per unit: exclusive rank prefix -> word w of the unit.  Per set bit: canonical key of the cell ->
// keys[slot].  own_prefix (optional): record index at every ownership-tile boundary, [own_tiles + 1].
__global__ void __launch_bounds__(kScanThreads)
unit_prefix_kernel(const GridDev* __restrict__ gp, uint4* __restrict__ units, ScanRange range,
                   const uint32_t* __restrict__ tile_excl, uint64_t* __restrict__ keys, int key_stride, long long cap,
                   uint32_t* __restrict__ own_prefix) {
  __shared__ uint32_t s_warp[kScanThreads / 32];
  const GridDev g = *gp;
  const long long n_units = g.n_units;
  const long long tiles = scan_tiles(range, n_units);
  const long long own_tiles = (n_units + kOwnUnits - 1) / kOwnUnits;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint64_t nxy = (uint64_t)g.nx * (uint64_t)g.ny;
  for (long long t = blockIdx.x; t < tiles; t += gridDim.x) {
    const long long tile = range.tile_begin + t;
    const long long base = tile * kTileUnits;
    uint32_t carry = tile_excl[t];
    const long long own0 = tile * kOwnPerScanTile;
    const bool last = t == tiles - 1;
    // empty tile (most of the grid is): its units keep the zero prefix word of the clean-up and are never
    // looked up, nothing to emit
    if (tile_excl[t + 1] == carry) {
      if (own_prefix != nullptr && threadIdx.x <= kOwnPerScanTile && own0 + threadIdx.x <= own_tiles &&
          (threadIdx.x < kOwnPerScanTile || last))
        own_prefix[own0 + threadIdx.x] = carry;
      continue;
    }
#pragma unroll 1
    for (int j = 0; j < kUnitsPerThread; ++j) {
      const long long ui = base + j * kScanThreads + threadIdx.x;
      uint4 u = make_uint4(0, 0, 0, 0);
      if (ui < n_units) u = __ldg(units + ui);
      const uint32_t cnt = (uint32_t)popc3(u);
      uint32_t inc = cnt;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const uint32_t tt = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += tt;
      }
      if (lane == 31) s_warp[warp] = inc;
      __syncthreads();
      uint32_t before = 0, total = 0;
#pragma unroll
      for (int q = 0; q < kScanThreads / 32; ++q) {
        const uint32_t s = s_warp[q];
        before += q < warp ? s : 0u;
        total += s;
      }
      __syncthreads();
      const uint32_t slot = carry + before + inc - cnt;
      if (own_prefix != nullptr && threadIdx.x == 0 && own0 + j <= own_tiles) own_prefix[own0 + j] = carry;
      carry += total;
      if (ui < n_units) units[ui].w = slot;
      if (cnt) emit_unit_keys(g, nxy, ui, u, slot, keys, key_stride, cap);
    }
    if (own_prefix != nullptr && threadIdx.x == 0 && last && own0 + kOwnPerScanTile <= own_tiles)
      own_prefix[own0 + kOwnPerScanTile] = carry;  // total, when the ownership tiles end exactly at this scan tile
  }
}

// accumulators of the min(counts[1], cap) voxels -> 0 (device-side count, no host round trip)
__global__ void __launch_bounds__(256)
zero_accum_kernel(ulonglong2* __restrict__ accum2, const unsigned long long* __restrict__ counts, int words_per_voxel, long long cap) {
  const long long mv = min((long long)counts[1], cap);
  const long long n2 = (mv * words_per_voxel + 1) / 2;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n2; i += (long long)gridDim.x * blockDim.x)
    accum2[i] = make_ulonglong2(0ull, 0ull);
}

// slot of `cell` in the key-sorted output, or kNoSlot when its occupancy bit is not set (a cell that
// ddn_fuse_unmark_points removed: its points do not participate)
constexpr uint32_t kNoSlot = 0xffffffffu;
__device__ __forceinline__ uint32_t slot_from_unit(uint64_t cell, const uint4& u) {
  const uint32_t w32 = (uint32_t)(cell >> 5);
  const int wi = (int)(w32 - (w32 / 3u) * 3u);
  const uint32_t below = (1u << (cell & 31)) - 1u;
  const uint32_t word = wi == 0 ? u.x : (wi == 1 ? u.y : u.z);
  if (((word >> (cell & 31)) & 1u) == 0u) return kNoSlot;
  uint32_t s = u.w;
  s += __popc(u.x & (wi > 0 ? 0xffffffffu : below));
  s += wi > 0 ? __popc(u.y & (wi > 1 ? 0xffffffffu : below)) : 0;
  s += wi > 1 ? __popc(u.z & below) : 0;
  return s;
}
__device__ __forceinline__ uint32_t slot_of_cell(uint64_t cell, const uint4* __restrict__ units) {
  return slot_from_unit(cell, __ldg(units + unit_of_cell(cell)));
}

// accumulate: one point per lane, aggregated ACROSS THE WARP before touching memory.  With a row length
// (points are pixels of [rows, row_len] images) a warp covers a 16 x 2 pixel tile, otherwise 32
// consecutive points.  Lanes whose points fall into the same cell are found with MATCH.ANY; every lane
// walks its peer mask with shuffles (32-bit partial sums: at most 32 points of |offset| <= 2^19 + 1), and
// the lowest lane of each group looks the slot up and issues the five 64-bit REDs.  The L2 atomic units
// are the bound of this pass, so points per RED group is what matters: ~2 at cfg 2.
// (-DDDN_ACC_REDUX sums each group with REDUX over its own peer mask instead of the shuffle walk: the
// hardware serialises the distinct masks of a warp, measured 2.5x SLOWER - profiles/README.md, round 2.)
#ifndef DDN_ACC_TPW
#define DDN_ACC_TPW 8
#endif
constexpr int kAccTilesPerWarp = DDN_ACC_TPW;
constexpr int kAccTileW = 16;  // pixel tile of a warp: 16 x 2 (measured at cfg 2: 4 x 8 4.46, 8 x 4 4.35, 16 x 2 4.34, 32 x 1 4.54 ms)

// The normals form (Normal = const float*, the plain form has no trailing parameter): every point also adds its
// quantised normal (normal_fix; normal [n,3] f32 in the order of xyz) - three more 32-bit words in the shuffle walk and
// three more REDs from the group leader, at accumulator words 5..7 (stride kAccNormalWords).
template <int kTW, class... Normal>  // tile width in pixels (tile = kTW x 32/kTW); 0 = no row structure, 32 consecutive points
__global__ void __launch_bounds__(256)
accumulate_points_kernel(const GridDev* __restrict__ gp, int64_t n, int row_len, const float* __restrict__ xyz,
                         const uint8_t* __restrict__ rgb, const uint8_t* __restrict__ votes, int thr,
                         const uint4* __restrict__ units, unsigned long long* __restrict__ accum, int stride, long long cap,
                         Normal... normal_in) {
  constexpr bool kNormals = sizeof...(Normal) != 0;
  const float* __restrict__ normal = normal_arg(normal_in...);
#if defined(DDN_ACC_REDUX) || defined(DDN_ACC_DEFER)
  static_assert(!kNormals, "the DDN_ACC_REDUX / DDN_ACC_DEFER experiments have no normals form");
#endif
  const GridDev g = *gp;
  if (g.n_units == 0) return;
  const float rv = 1.0f / g.voxel;
  const int lane = threadIdx.x & 31;
  const float fix_scale = voxel_fix_scale(g.voxel);
  // n < 2^31, so tile indices fit 32 bits
  const uint32_t warp = blockIdx.x * 8u + (threadIdx.x >> 5);
  constexpr bool kTiled = kTW > 0;
  constexpr int kTWs = kTiled ? kTW : 32, kTH = 32 / kTWs;
  uint32_t tiles_x = 0, n_tiles;
  if (kTiled) {
    tiles_x = ((uint32_t)row_len + kTWs - 1u) / kTWs;
    const uint32_t n_rows = (uint32_t)((n + row_len - 1) / row_len);
    n_tiles = tiles_x * ((n_rows + kTH - 1u) / kTH);
  } else {
    n_tiles = (uint32_t)((n + 31) / 32);
  }
  const int dx = lane % kTWs, dy = lane / kTWs;
  const uint32_t t_begin = warp * kAccTilesPerWarp;
  if (t_begin >= n_tiles) return;
  const uint32_t t_end = min(t_begin + (uint32_t)kAccTilesPerWarp, n_tiles);
  uint32_t ty = 0, tx = 0;
  if (kTiled) {
    ty = t_begin / tiles_x;
    tx = t_begin - ty * tiles_x;
  }
  // The point of the NEXT tile is loaded (vote, position and colour at once - no dependent round trips)
  // before the current tile is processed, so its latency hides behind the aggregation and the atomics.
  struct InBase {
    float x, y, z;
    uint32_t rg, bb;
    bool take;
  };
  struct InNormal : InBase {
    float nx, ny, nz;
  };
  using In = std::conditional_t<kNormals, InNormal, InBase>;
  auto load_tile = [&](uint32_t t) -> In {
    int64_t i;
    bool in;
    if (kTiled) {
      const int x = (int)tx * kTWs + dx;
      i = (int64_t)(ty * kTH + dy) * row_len + x;
      in = x < row_len && i < n;
      if (++tx == tiles_x) tx = 0, ++ty;
    } else {
      i = (int64_t)t * 32 + lane;
      in = i < n;
    }
    In r{};
    if (in) {
      const int v = votes != nullptr ? (int)__ldg(votes + i) : 0;
      r.x = __ldg(xyz + i * 3 + 0), r.y = __ldg(xyz + i * 3 + 1), r.z = __ldg(xyz + i * 3 + 2);
      r.rg = ((uint32_t)__ldg(rgb + i * 3 + 0) << 16) | (uint32_t)__ldg(rgb + i * 3 + 1);
      r.bb = (uint32_t)__ldg(rgb + i * 3 + 2);
      r.take = v < thr || votes == nullptr;
      if constexpr (kNormals) r.nx = __ldg(normal + i * 3 + 0), r.ny = __ldg(normal + i * 3 + 1), r.nz = __ldg(normal + i * 3 + 2);
    }
    return r;
  };
  In nxt = load_tile(t_begin);
#ifdef DDN_ACC_DEFER
  bool pend = false;
  uint4 pend_unit = make_uint4(0, 0, 0, 0);
  uint64_t pend_cell = 0;
  int psx = 0, psy = 0, psz = 0;
  uint32_t psrg = 0, psb = 0, ppop = 0;
  auto flush = [&]() {
    if (pend) {
      const uint32_t slot = slot_from_unit(pend_cell, pend_unit);
      if ((long long)slot < cap) {
        unsigned long long* a = accum + (size_t)slot * stride;
        atomicAdd(a + 0, (unsigned long long)(long long)psx);
        atomicAdd(a + 1, (unsigned long long)(long long)psy);
        atomicAdd(a + 2, (unsigned long long)(long long)psz);
        atomicAdd(a + 3, ((unsigned long long)(psrg >> 16) << 32) | (psrg & 0xffffu));
        atomicAdd(a + 4, ((unsigned long long)psb << 32) | ppop);
      }
    }
  };
#endif
#pragma unroll 1
  for (uint32_t t = t_begin; t < t_end; ++t) {
    const In cur = nxt;
    if (t + 1 < t_end) nxt = load_tile(t + 1);
    uint64_t cell = kNoCell;
    int ox = 0, oy = 0, oz = 0;
    const uint32_t rg = cur.rg, bb = cur.bb;
    if (cur.take) {
      uint32_t kx, ky, kz;
      cell = cell_of_point(g, rv, cur.x, cur.y, cur.z, kx, ky, kz);
      if (cell != kNoCell) {
        // p - centre is exact in float32 for points inside the voxel
        ox = voxel_offset_fix(cur.x, voxel_centre(g.ox, kx, g.voxel), fix_scale);
        oy = voxel_offset_fix(cur.y, voxel_centre(g.oy, ky, g.voxel), fix_scale);
        oz = voxel_offset_fix(cur.z, voxel_centre(g.oz, kz, g.voxel), fix_scale);
      }
    }
    const bool valid = cell != kNoCell;
    uint32_t peers = __match_any_sync(0xffffffffu, cell);
    if (!valid) peers = 0;
    const bool leader = valid && (__ffs(peers) - 1) == lane;
    int sx = 0, sy = 0, sz = 0;
    uint32_t srg = 0, sb = 0;
    int snx = 0, sny = 0, snz = 0;  // kNormals
#ifndef DDN_ACC_REDUX
    // Three shuffles per step of the walk instead of five: a word per axis holds the offset (|offset| <= 2^19 + 1, far
    // inside 24 signed bits) above one colour byte.  s* sums the offsets (arithmetic shift), t* the whole words modulo
    // 2^32, so a colour sum is t - (s << 8), exact because it is at most 32 * 255 < 2^13.
    const uint32_t wx = ((uint32_t)ox << 8) | (rg >> 16), wy = ((uint32_t)oy << 8) | (rg & 0xffffu), wz = ((uint32_t)oz << 8) | bb;
    uint32_t tx = 0, ty = 0, tz = 0;
    int qx = 0, qy = 0, qz = 0;
    if constexpr (kNormals) {
      if (valid) qx = normal_fix(cur.nx), qy = normal_fix(cur.ny), qz = normal_fix(cur.nz);
    }
    const int iters = __reduce_max_sync(0xffffffffu, __popc(peers));
    uint32_t rest = peers;
#pragma unroll 1
    for (int k = 0; k < iters; ++k) {
      const bool has = rest != 0;
      const int src = has ? __ffs(rest) - 1 : lane;
      rest &= rest - 1;
      const uint32_t ax = __shfl_sync(0xffffffffu, wx, src), ay = __shfl_sync(0xffffffffu, wy, src);
      const uint32_t az = __shfl_sync(0xffffffffu, wz, src);
      if (has) {
        sx += (int)ax >> 8, sy += (int)ay >> 8, sz += (int)az >> 8;
        tx += ax, ty += ay, tz += az;
      }
      if constexpr (kNormals) {
        const int bx = __shfl_sync(0xffffffffu, qx, src), by = __shfl_sync(0xffffffffu, qy, src), bz = __shfl_sync(0xffffffffu, qz, src);
        if (has) snx += bx, sny += by, snz += bz;
      }
    }
    srg = ((tx - ((uint32_t)sx << 8)) << 16) | (ty - ((uint32_t)sy << 8));
    sb = tz - ((uint32_t)sz << 8);
#else
    if (valid) {  // every lane of a group passes the same mask: REDUX over the group only
      sx = __reduce_add_sync(peers, ox);
      sy = __reduce_add_sync(peers, oy);
      sz = __reduce_add_sync(peers, oz);
      srg = __reduce_add_sync(peers, rg);
      sb = __reduce_add_sync(peers, bb);
    }
#endif
#ifndef DDN_ACC_DEFER
    if (leader) {
      const uint32_t slot = slot_of_cell(cell, units);
      if ((long long)slot < cap) {
        unsigned long long* a = accum + (size_t)slot * stride;
        atomicAdd(a + 0, (unsigned long long)(long long)sx);
        atomicAdd(a + 1, (unsigned long long)(long long)sy);
        atomicAdd(a + 2, (unsigned long long)(long long)sz);
        atomicAdd(a + 3, ((unsigned long long)(srg >> 16) << 32) | (srg & 0xffffu));
        atomicAdd(a + 4, ((unsigned long long)sb << 32) | (unsigned)__popc(peers));
        if constexpr (kNormals) {
          atomicAdd(a + 5, (unsigned long long)(long long)snx);
          atomicAdd(a + 6, (unsigned long long)(long long)sny);
          atomicAdd(a + 7, (unsigned long long)(long long)snz);
        }
      }
    }
  }
#else
    // -DDDN_ACC_DEFER: the atomics of a tile are issued one iteration LATER - the leader only requests its unit
    // here, and the 16-byte gather has the whole next tile to arrive.  Measured at cfg 2: 56 registers instead of
    // 38 cost more occupancy than the hidden latency returns (rank + accumulate + finalise 3.62 vs 3.45 ms).
    flush();
    pend = leader;
    if (leader) {
      pend_unit = __ldg(units + unit_of_cell(cell));
      pend_cell = cell;
      psx = sx, psy = sy, psz = sz, psrg = srg, psb = sb, ppop = (uint32_t)__popc(peers);
    }
  }
  flush();
#endif
}

__global__ void __launch_bounds__(256)
accumulate_records_kernel(const GridDev* __restrict__ gp, int64_t n, const unsigned long long* __restrict__ records,
                          const uint4* __restrict__ units, uint64_t cell_begin, uint64_t cell_end,
                          unsigned long long* __restrict__ accum, long long cap) {
  const GridDev g = *gp;
  if (g.n_units == 0) return;
  const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (i >= n) return;
  const unsigned long long* r = records + i * kRecWords;
  const uint64_t cell = cell_of_key(g, __ldg(r));
  if (cell == kNoCell || cell < cell_begin || cell >= cell_end) return;
  const uint32_t slot = slot_of_cell(cell, units);
  if ((long long)slot >= cap) return;
  unsigned long long* a = accum + (size_t)slot * kAccWords;
#pragma unroll
  for (int q = 0; q < kAccWords; ++q) atomicAdd(a + q, __ldg(r + 1 + q));
}

// One thread per voxel.  The colour fields are 32 bits wide: a voxel with 2^24 or more points could
// have overflowed them, which is reported (counts[0] = -1) instead of returned as a wrong colour.
// kNormals (finalize_normals_kernel): accumulators of kAccNormalWords words, whose normal sums finalize_normal turns into
// out_normal.
template <bool kNormals>
__device__ __forceinline__ void finalize_body(const GridDev* __restrict__ gp, const unsigned long long* __restrict__ accum,
                                              const uint64_t* __restrict__ keys, long long* __restrict__ counts, long long cap,
                                              float* __restrict__ out_xyz, uint8_t* __restrict__ out_rgb, int32_t* __restrict__ out_count,
                                              float* __restrict__ out_normal) {
  const GridDev g = *gp;
  const long long mv = min(counts[1], cap);
  for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < mv; r += (long long)gridDim.x * blockDim.x) {
    const unsigned long long* a = accum + (size_t)r * (kNormals ? kAccNormalWords : kAccWords);
    const long long sx = (long long)a[0], sy = (long long)a[1], sz = (long long)a[2];
    const unsigned long long rg = a[3], bn = a[4];
    const uint32_t cnt = (uint32_t)bn;
    if (cnt >= (1u << 24)) counts[0] = -1;
    out_count[r] = (int32_t)cnt;
    const uint64_t key = keys[r];
    const uint32_t kx = (uint32_t)(key & 0x1fffff), ky = (uint32_t)((key >> 21) & 0x1fffff), kz = (uint32_t)((key >> 42) & 0x1fffff);
    finalize_voxel(g, voxel_centre(g.ox, kx, g.voxel), voxel_centre(g.oy, ky, g.voxel), voxel_centre(g.oz, kz, g.voxel), sx, sy, sz,
                   rg >> 32, rg & 0xffffffffull, bn >> 32, (long long)cnt, out_xyz + r * 3, out_rgb + r * 3);
    if constexpr (kNormals) finalize_normal((long long)a[5], (long long)a[6], (long long)a[7], out_normal + r * 3);
  }
}

__global__ void __launch_bounds__(256)
finalize_kernel(const GridDev* __restrict__ gp, const unsigned long long* __restrict__ accum, const uint64_t* __restrict__ keys,
                long long* __restrict__ counts, long long cap, float* __restrict__ out_xyz, uint8_t* __restrict__ out_rgb,
                int32_t* __restrict__ out_count) {
  finalize_body<false>(gp, accum, keys, counts, cap, out_xyz, out_rgb, out_count, nullptr);
}

__global__ void __launch_bounds__(256)
finalize_normals_kernel(const GridDev* __restrict__ gp, const unsigned long long* __restrict__ accum, const uint64_t* __restrict__ keys,
                        long long* __restrict__ counts, long long cap, float* __restrict__ out_xyz, uint8_t* __restrict__ out_rgb,
                        int32_t* __restrict__ out_count, float* __restrict__ out_normal) {
  finalize_body<true>(gp, accum, keys, counts, cap, out_xyz, out_rgb, out_count, out_normal);
}

__global__ void canonical_key_kernel(GridDev g, int64_t n, const float* __restrict__ xyz, uint64_t* __restrict__ keys) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float x = xyz[i * 3 + 0], y = xyz[i * 3 + 1], z = xyz[i * 3 + 2];
  const float rv = 1.0f / g.voxel;
  const int64_t kx = (int64_t)voxel_coord(x, g.ox, g.voxel, rv);
  const int64_t ky = (int64_t)voxel_coord(y, g.oy, g.voxel, rv);
  const int64_t kz = (int64_t)voxel_coord(z, g.oz, g.voxel, rv);
  const bool ok = kx >= 0 && ky >= 0 && kz >= 0 && kx < (1 << 21) && ky < (1 << 21) && kz < (1 << 21);
  keys[i] = ok ? ((uint64_t)kx | ((uint64_t)ky << 21) | ((uint64_t)kz << 42)) : ~0ull;
}

// ====================================================================================================
// Multi-GPU: owner-side exchange + merge over peer memory
// ====================================================================================================
// plan (device, i64): [0] first owned tile, [1] end of owned tiles, [2] records to receive, [3] own tiles,
// [4 + k] first record of this rank's share in the records of rank q = (rank + k) % R, [4 + P + k] its length,
// [4 + 2P + k] exclusive prefix of the lengths (P = DDN_MAX_PEERS).  The shares are walked in this ROTATED order:
// every rank starts with its own records and then reads a different peer than everybody else, so all NVLink
// ports carry traffic at once (in natural order all ranks would pull from rank 0 first, then from rank 1, ...).
#ifndef DDN_PULL_CTAS_PER_SM
#define DDN_PULL_CTAS_PER_SM 8
#endif
constexpr int kPlanWords = 4 + 3 * DDN_MAX_PEERS;
static_assert(kPlanWords <= 64, "plan scratch is 64 words");
static_assert(DDN_MAX_PEERS <= 31, "the plan kernel is one warp");

// Step 0 of the merge: every rank's tile prefix (whole array, n_own + 1 entries) is copied into local memory in
// ONE bulk pass over NVLink - local[q * stride + t] - with their sum over the ranks in row R.  Everything the plan
// and the occupancy merge decide afterwards reads local memory: no chain of dependent remote round trips.
__global__ void __launch_bounds__(256)
merge_gather_prefix_kernel(const GridDev* __restrict__ gp, PeerPtrs prefix, int R, uint32_t* __restrict__ local, long long stride) {
  const long long n = (gp->n_units + kOwnUnits - 1) / kOwnUnits + 1;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    uint32_t v[DDN_MAX_PEERS];
#pragma unroll
    for (int q = 0; q < DDN_MAX_PEERS; ++q) v[q] = q < R ? __ldcv(reinterpret_cast<const uint32_t*>(prefix.p[q]) + i) : 0u;
    uint32_t sum = 0;
#pragma unroll
    for (int q = 0; q < DDN_MAX_PEERS; ++q) {
      if (q < R) local[q * stride + i] = v[q];
      sum += v[q];
    }
    local[(long long)R * stride + i] = sum;
  }
}

// The R ranks cut the ownership tiles into R contiguous ranges that balance the GLOBAL record count:
// cum[t] = sum over ranks of tile_prefix_q[t] is the number of records in tiles [0, t); boundary b is the
// first t with cum[t] >= total * b / R.  Every rank runs the same search on the same numbers, so all agree
// without communicating.  One thread per boundary (binary search in the local cum row).
__global__ void __launch_bounds__(32)
merge_plan_kernel(const GridDev* __restrict__ gp, const uint32_t* __restrict__ local, long long stride, int rank, int R,
                  long long* __restrict__ plan) {
  __shared__ long long s_bnd[DDN_MAX_PEERS + 1];
  const long long n_own = (gp->n_units + kOwnUnits - 1) / kOwnUnits;
  const uint32_t* cum = local + (long long)R * stride;
  const int b = threadIdx.x;
  if (b <= R) {
    // b = 1..R-1: the balanced cuts; b = 0: the first tile that holds a record; b = R: the end of the last one -
    // the empty head and tail of the grid belong to nobody
    const long long total = (long long)cum[n_own];
    const long long target = b == 0 ? 1 : (b == R ? total : total * b / R);
    long long lo = 0, hi = n_own + 1;
    while (lo < hi) {
      const long long mid = (lo + hi) >> 1;
      if ((long long)cum[mid] < target) lo = mid + 1;
      else hi = mid;
    }
    lo = min(lo, n_own);
    if (b == 0) lo = total > 0 ? max(lo - 1, 0ll) : 0;  // cum[lo] >= 1 > cum[lo - 1]: tile lo - 1 is the first with a record
    s_bnd[b] = lo;
  }
  __syncwarp();
  if (threadIdx.x == 0) {
    for (int k = 1; k <= R; ++k) s_bnd[k] = max(s_bnd[k], s_bnd[k - 1]);  // monotone
    plan[0] = s_bnd[rank];
    plan[1] = s_bnd[rank + 1];
    plan[3] = n_own;
  }
  __syncwarp();
  const int lane = threadIdx.x;
  long long begin = 0, count = 0;
  if (lane < R) {
    const int q = (rank + lane) % R;
    begin = (long long)local[q * stride + s_bnd[rank]];
    count = (long long)local[q * stride + s_bnd[rank + 1]] - begin;
  }
  long long inc = count;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const long long t = __shfl_up_sync(0xffffffffu, inc, d);
    if (lane >= d) inc += t;
  }
  if (lane < DDN_MAX_PEERS) {
    plan[4 + lane] = begin;
    plan[4 + DDN_MAX_PEERS + lane] = count;
    plan[4 + 2 * DDN_MAX_PEERS + lane] = inc - count;
  }
  const long long total = __shfl_sync(0xffffffffu, inc, 31);
  if (lane == 0) plan[2] = total;
}

// The owner's units over its own range start empty: its own partial bits are re-marked from its records like
// everybody else's (dirty scan tiles only; the flags stay set for the next step's clean-up).
__global__ void __launch_bounds__(kOwnUnits)
merge_clear_kernel(FuseDev f, const long long* __restrict__ plan) {
  const long long n_units = f.grid->n_units;
  uint4* my_units = reinterpret_cast<uint4*>(f.units);
  for (long long t = plan[0] + blockIdx.x; t < plan[1]; t += gridDim.x) {
    if (f.dirty != nullptr && f.dirty[(t * kOwnUnits) / kTileUnits] == 0) continue;  // CTA-uniform
    const long long ui = t * kOwnUnits + threadIdx.x;
    if (ui < n_units) my_units[ui] = make_uint4(0, 0, 0, 0);
  }
}

// THE exchange: this rank's share of every rank's sorted partial records is pulled straight out of its owner's HBM
// - once - into a local staging array, and the occupancy bit of every record is set on the way.  A warp handles 32
// consecutive records: the 1536 bytes are fetched as three fully coalesced 512-byte requests (lane l takes bytes
// 16 l of each) and re-distributed through shared memory - NVLink moves large requests at full rate, while
// per-thread 48-byte records (three 16-byte pieces at a 48-byte stride) cross it as twice as many half-used
// sectors: measured 140 GB/s that way against 650 GB/s coalesced (scripts/experiments/peer_read_probe.py).
// The shares are walked in rotated rank order, so every rank reads a different peer at any time.
// Work is proportional to the records, which the cuts balance - the unit-driven occupancy merge this replaces cost
// the owner of a sparse key range three times what the others paid (profiles/README.md, round 2).
// merge_pull_mark_normals_kernel is the same loop over the 80-byte records of the fused-normal form (five requests per
// warp step).  Each form spells the loop out: behind a shared inline body the plain form no longer compiled to the same
// instructions.
__global__ void __launch_bounds__(256)
merge_pull_mark_kernel(FuseDev f, PeerPtrs peer_records, int rank, int R, const long long* __restrict__ plan,
                       ulonglong2* __restrict__ staging, long long cap) {
  __shared__ ulonglong2 s_rec[8][16 * DDN_RECORD_WORDS];  // per warp: 32 records
  const GridDev g = *f.grid;
  if (g.n_units == 0) return;
  const long long total = min(plan[2], cap);
  const uint64_t cell_begin = (uint64_t)plan[0] * kOwnUnits * kUnitBits, cell_end = (uint64_t)plan[1] * kOwnUnits * kUnitBits;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long n_warps = (long long)gridDim.x * 8;
  for (long long w0 = ((long long)blockIdx.x * 8 + warp) * 32; w0 < total; w0 += n_warps * 32) {
    const unsigned long long key = pull_share_warp<DDN_RECORD_WORDS>(peer_records, rank, R, plan, staging, w0, total, s_rec[warp], lane);
    uint64_t cell = cell_of_key(g, key);
    if (cell < cell_begin || cell >= cell_end) cell = kNoCell;
    uint64_t left = __shfl_up_sync(0xffffffffu, cell, 1);
    if (lane == 0) left = kNoCell;
    if (cell != kNoCell) set_cell_bit(f.units, f.dirty, cell, left);
  }
}

__global__ void __launch_bounds__(256, DDN_PULL_CTAS_PER_SM)  // 32 registers, as the plain form (40 without the bound: 6 CTAs per SM)
merge_pull_mark_normals_kernel(FuseDev f, PeerPtrs peer_records, int rank, int R, const long long* __restrict__ plan,
                               ulonglong2* __restrict__ staging, long long cap) {
  __shared__ ulonglong2 s_rec[8][16 * DDN_RECORD_NORMAL_WORDS];  // per warp: 32 records
  const GridDev g = *f.grid;
  if (g.n_units == 0) return;
  const long long total = min(plan[2], cap);
  const uint64_t cell_begin = (uint64_t)plan[0] * kOwnUnits * kUnitBits, cell_end = (uint64_t)plan[1] * kOwnUnits * kUnitBits;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long n_warps = (long long)gridDim.x * 8;
  for (long long w0 = ((long long)blockIdx.x * 8 + warp) * 32; w0 < total; w0 += n_warps * 32) {
    const unsigned long long key = pull_share_warp<DDN_RECORD_NORMAL_WORDS>(peer_records, rank, R, plan, staging, w0, total, s_rec[warp], lane);
    uint64_t cell = cell_of_key(g, key);
    if (cell < cell_begin || cell >= cell_end) cell = kNoCell;
    uint64_t left = __shfl_up_sync(0xffffffffu, cell, 1);
    if (lane == 0) left = kNoCell;
    if (cell != kNoCell) set_cell_bit(f.units, f.dirty, cell, left);
  }
}

// occupied cells per ownership tile of the owned range (a tile whose scan tile was never touched is empty)
__global__ void __launch_bounds__(kOwnUnits)
merge_count_kernel(FuseDev f, const long long* __restrict__ plan, uint32_t* __restrict__ tile_sums) {
  __shared__ int s_warp[kScanThreads / 32];
  const long long n_units = f.grid->n_units;
  const long long t0 = plan[0], t1 = plan[1];
  const uint4* my_units = reinterpret_cast<const uint4*>(f.units);
  for (long long t = t0 + blockIdx.x; t < t1; t += gridDim.x) {
    if (f.dirty != nullptr && f.dirty[(t * kOwnUnits) / kTileUnits] == 0) {  // CTA-uniform
      if (threadIdx.x == 0) tile_sums[t - t0] = 0u;
      continue;
    }
    const long long ui = t * kOwnUnits + threadIdx.x;
    const int total = block_sum_256(ui < n_units ? popc3(my_units[ui]) : 0, s_warp);
    if (threadIdx.x == 0) tile_sums[t - t0] = (uint32_t)total;
  }
}

// rank prefix of the merged units + keys of the merged voxels (one ownership tile per CTA iteration)
__global__ void __launch_bounds__(kOwnUnits)
merge_prefix_kernel(FuseDev f, const long long* __restrict__ plan, const uint32_t* __restrict__ tile_excl,
                    uint64_t* __restrict__ keys, long long cap) {
  __shared__ uint32_t s_warp[kScanThreads / 32];
  const GridDev g = *f.grid;
  const long long n_units = g.n_units;
  const long long t0 = plan[0], t1 = plan[1];
  uint4* my_units = reinterpret_cast<uint4*>(f.units);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint64_t nxy = (uint64_t)g.nx * (uint64_t)g.ny;
  for (long long t = t0 + blockIdx.x; t < t1; t += gridDim.x) {
    const uint32_t carry = tile_excl[t - t0];
    if (tile_excl[t - t0 + 1] == carry) continue;  // CTA-uniform
    const long long ui = t * kOwnUnits + threadIdx.x;
    uint4 u = make_uint4(0, 0, 0, 0);
    if (ui < n_units) u = my_units[ui];
    const uint32_t cnt = (uint32_t)popc3(u);
    uint32_t inc = cnt;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const uint32_t tt = __shfl_up_sync(0xffffffffu, inc, d);
      if (lane >= d) inc += tt;
    }
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    uint32_t before = 0;
#pragma unroll
    for (int q = 0; q < kScanThreads / 32; ++q) before += q < warp ? s_warp[q] : 0u;
    __syncthreads();
    const uint32_t slot = carry + before + inc - cnt;
    if (ui < n_units) my_units[ui].w = slot;
    if (cnt) emit_unit_keys(g, nxy, ui, u, slot, keys, 1, cap);
  }
}

// the staged records (local memory now) are looked up in the merged units and added with 64-bit REDs: the kSums words
// of a record into an accumulator of kSums words (kAccWords; kAccNormalWords for the fused-normal records)
template <int kW>
__device__ __forceinline__ void merge_accumulate_body(FuseDev f, const long long* __restrict__ plan, const ulonglong2* __restrict__ staging,
                                                      long long cap_records, unsigned long long* __restrict__ accum, long long cap) {
  constexpr int kP = Record<kW>::kPieces, kSums = Record<kW>::kSums;
  const GridDev g = *f.grid;
  if (g.n_units == 0) return;
  const long long total = min(plan[2], cap_records);
  const uint4* units = reinterpret_cast<const uint4*>(f.units);
  const uint64_t cell_begin = (uint64_t)plan[0] * kOwnUnits * kUnitBits, cell_end = (uint64_t)plan[1] * kOwnUnits * kUnitBits;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    ulonglong2 v[kP];
#pragma unroll
    for (int k = 0; k < kP; ++k) v[k] = __ldg(staging + i * kP + k);
    const uint64_t cell = cell_of_key(g, v[0].x);
    if (cell == kNoCell || cell < cell_begin || cell >= cell_end) continue;
    const uint32_t slot = slot_of_cell(cell, units);
    if ((long long)slot >= cap) continue;
    unsigned long long* o = accum + (size_t)slot * kSums;
#pragma unroll
    for (int q = 0; q < kSums; ++q) atomicAdd(o + q, record_word(v, q + 1));
  }
}

__global__ void __launch_bounds__(256)
merge_accumulate_kernel(FuseDev f, const long long* __restrict__ plan, const ulonglong2* __restrict__ staging, long long cap_records,
                        unsigned long long* __restrict__ accum, long long cap) {
  static_assert(Record<DDN_RECORD_WORDS>::kSums == kAccWords, "record = key + accumulators");
  merge_accumulate_body<DDN_RECORD_WORDS>(f, plan, staging, cap_records, accum, cap);
}

__global__ void __launch_bounds__(256)
merge_accumulate_normals_kernel(FuseDev f, const long long* __restrict__ plan, const ulonglong2* __restrict__ staging, long long cap_records,
                                unsigned long long* __restrict__ accum, long long cap) {
  merge_accumulate_body<DDN_RECORD_NORMAL_WORDS>(f, plan, staging, cap_records, accum, cap);
}

// ---- host side ---------------------------------------------------------------------------------
static uint64_t grid_cells(const GridDev& g) { return (uint64_t)g.nx * (uint64_t)g.ny * (uint64_t)g.nz; }
static bool use_dense(const GridDev& g) { return grid_cells(g) <= kDenseMaxCells; }

static int session_check(const ddn_fuse_session* s) {
  DDN_REQUIRE(s != nullptr, "null session");
  DDN_REQUIRE(s->grid && s->units && s->tile_sums && s->counts, "session: null buffer");
  DDN_REQUIRE(s->cap_units > 0 && s->cap_units <= (int64_t)(kDenseMaxCells / kUnitBits) + 1, "session: cap_units");
  DDN_REQUIRE((uintptr_t)s->units % 16 == 0 && (uintptr_t)s->grid % 8 == 0, "session: alignment");
  return DDN_OK;
}

static FuseDev fuse_dev(const ddn_fuse_session* s) {
  FuseDev f;
  f.grid = reinterpret_cast<const GridDev*>(s->grid);
  f.units = reinterpret_cast<uint32_t*>(s->units);
  f.dirty = s->dirty;
  f.counts = reinterpret_cast<unsigned long long*>(s->counts);
  return f;
}

static int launch_clear(const ddn_fuse_session* s, cudaStream_t st) {
  clear_units_kernel<<<kPersistentCtas, 256, 0, st>>>(reinterpret_cast<const GridDev*>(s->grid), reinterpret_cast<uint4*>(s->units),
                                                      s->dirty, (long long)s->cap_units);
  return after_launch("clear_units_kernel");
}

static int launch_mark_points(const ddn_fuse_session* s, int64_t n, const float* xyz, const uint8_t* votes, int thr, cudaStream_t st) {
  const bool vec = ((uintptr_t)xyz % 16 == 0) && (votes == nullptr || (uintptr_t)votes % 4 == 0);
  const unsigned mblocks = (unsigned)((n + 256 * kMarkPX - 1) / (256 * kMarkPX));
  if (vec) mark_points_kernel<true><<<mblocks, 256, 0, st>>>(fuse_dev(s), n, xyz, votes, thr);
  else mark_points_kernel<false><<<mblocks, 256, 0, st>>>(fuse_dev(s), n, xyz, votes, thr);
  return after_launch("mark_points_kernel");
}

// rank passes over `range` (whole device grid when range.n_tiles < 0): tile counts -> scan -> accumulators
// cleared -> unit prefixes + keys
static int launch_rank(const ddn_fuse_session* s, ScanRange range, uint64_t* keys, int key_stride, unsigned long long* zero_base,
                       int zero_stride, long long cap, uint32_t* own_prefix, cudaStream_t st) {
  const GridDev* gp = reinterpret_cast<const GridDev*>(s->grid);
  uint4* units = reinterpret_cast<uint4*>(s->units);
  unsigned long long* counts = reinterpret_cast<unsigned long long*>(s->counts);
  const unsigned ctas = range.n_tiles >= 0 ? (unsigned)std::max<long long>(1, std::min<long long>(range.n_tiles, kPersistentCtas))
                                            : (unsigned)kPersistentCtas;
  tile_count_kernel<<<ctas, kScanThreads, 0, st>>>(gp, units, s->dirty, range, s->tile_sums);
  DDN_TRY(after_launch("tile_count_kernel", st));
  tile_scan_kernel<<<1, 1024, 0, st>>>(gp, range, nullptr, s->tile_sums, counts);
  DDN_TRY(after_launch("tile_scan_kernel", st));
  zero_accum_kernel<<<kPersistentCtas, 256, 0, st>>>((ulonglong2*)zero_base, counts, zero_stride, cap);
  DDN_TRY(after_launch("zero_accum_kernel", st));
  unit_prefix_kernel<<<ctas, kScanThreads, 0, st>>>(gp, units, range, s->tile_sums, keys, key_stride, cap, own_prefix);
  return after_launch("unit_prefix_kernel", st);
}

// normal != nullptr: the normals form (accumulators of kAccNormalWords words)
static int launch_accumulate_points(const ddn_fuse_session* s, int64_t n, int64_t row_len, const float* xyz, const uint8_t* rgb,
                                    const uint8_t* votes, int thr, unsigned long long* accum, int stride, long long cap,
                                    cudaStream_t st, const float* normal = nullptr) {
  const GridDev* gp = reinterpret_cast<const GridDev*>(s->grid);
  const uint4* units = reinterpret_cast<const uint4*>(s->units);
  const bool tiled = row_len >= 32 && row_len < (1 << 30);
  const int tw = tiled ? kAccTileW : 0;
  const int th = tw ? 32 / tw : 1, twe = tw ? tw : 32;
  const int64_t n_tiles = tiled ? ((row_len + twe - 1) / twe) * (((n + row_len - 1) / row_len + th - 1) / th) : (n + 31) / 32;
  const unsigned ablocks = (unsigned)((n_tiles + 8 * kAccTilesPerWarp - 1) / (8 * kAccTilesPerWarp));
  if (normal != nullptr) {
#if defined(DDN_ACC_REDUX) || defined(DDN_ACC_DEFER)
    set_error("the DDN_ACC_REDUX / DDN_ACC_DEFER builds have no fused-normals form");
    return DDN_ERR_UNSUPPORTED;
#else
    if (tiled)
      accumulate_points_kernel<kAccTileW, const float*><<<ablocks, 256, 0, st>>>(gp, n, (int)row_len, xyz, rgb, votes, thr, units, accum,
                                                                                stride, cap, normal);
    else
      accumulate_points_kernel<0, const float*><<<ablocks, 256, 0, st>>>(gp, n, (int)row_len, xyz, rgb, votes, thr, units, accum, stride,
                                                                        cap, normal);
    return after_launch("accumulate_points_kernel", st);
#endif
  }
  if (tiled)
    accumulate_points_kernel<kAccTileW><<<ablocks, 256, 0, st>>>(gp, n, (int)row_len, xyz, rgb, votes, thr, units, accum, stride, cap);
  else
    accumulate_points_kernel<0><<<ablocks, 256, 0, st>>>(gp, n, (int)row_len, xyz, rgb, votes, thr, units, accum, stride, cap);
  return after_launch("accumulate_points_kernel", st);
}

static int launch_finalize(const ddn_fuse_session* s, const unsigned long long* accum, const uint64_t* keys, long long cap,
                           float* out_xyz, uint8_t* out_rgb, int32_t* out_count, cudaStream_t st, float* out_normal = nullptr) {
  if (out_normal != nullptr) {
    finalize_normals_kernel<<<kPersistentCtas, 256, 0, st>>>(reinterpret_cast<const GridDev*>(s->grid), accum, keys,
                                                             reinterpret_cast<long long*>(s->counts), cap, out_xyz, out_rgb, out_count,
                                                             out_normal);
    return after_launch("finalize_normals_kernel", st);
  }
  finalize_kernel<<<kPersistentCtas, 256, 0, st>>>(reinterpret_cast<const GridDev*>(s->grid), accum, keys,
                                                   reinterpret_cast<long long*>(s->counts), cap, out_xyz, out_rgb, out_count);
  return after_launch("finalize_kernel", st);
}

// ---- legacy host-grid entry points: a session carved out of the caller's workspace -----------------
struct DenseLayout {
  uint64_t cells, n_units, tiles, own_tiles;
  size_t grid, units, tile_sums, accum, total;
};

// consecutive 256-byte aligned pieces of a workspace
struct WorkspaceOffsets {
  size_t off = 0;
  size_t take(size_t bytes) {
    const size_t o = off;
    off += (size_t)align_up((int64_t)bytes, 256);
    return o;
  }
};

// sized for the non-partial form; words: accumulator words per voxel (kAccWords, or kAccNormalWords for the normals form)
static void dense_layout(const GridDev& g, int64_t n, DenseLayout* L, int words = kAccWords) {
  L->cells = grid_cells(g);
  L->n_units = (L->cells + kUnitBits - 1) / kUnitBits;
  L->tiles = (L->n_units + kTileUnits - 1) / kTileUnits;
  L->own_tiles = (L->n_units + kOwnUnits - 1) / kOwnUnits;
  const uint64_t max_vox = (uint64_t)n < L->cells ? (uint64_t)n : L->cells;
  WorkspaceOffsets o;
  L->grid = o.take(sizeof(GridDev));
  L->units = o.take((size_t)L->n_units * 16);
  L->tile_sums = o.take((size_t)(L->own_tiles + 2) * 4);
  L->accum = o.take((size_t)max_vox * words * 8 + 16);
  L->total = o.off + 256;
}

static int carve_session(const GridDev& g, int64_t n, void* workspace, int64_t workspace_bytes, ddn_fuse_session* s,
                         int64_t* counts_out, unsigned long long** accum, DenseLayout* L, int words = kAccWords) {
  dense_layout(g, n, L, words);
  if ((int64_t)L->total > workspace_bytes) {
    set_error("fuse workspace too small: %lld < %lld", (long long)workspace_bytes, (long long)L->total);
    return DDN_ERR_WORKSPACE_TOO_SMALL;
  }
  char* base = reinterpret_cast<char*>(align_up((int64_t)(uintptr_t)workspace, 256));
  s->grid = reinterpret_cast<ddn_grid_state*>(base + L->grid);
  s->units = base + L->units;
  s->cap_units = (int64_t)L->n_units;
  s->dirty = nullptr;
  s->tile_sums = reinterpret_cast<uint32_t*>(base + L->tile_sums);
  s->tile_prefix = nullptr;
  s->counts = counts_out;
  *accum = reinterpret_cast<unsigned long long*>(base + L->accum);
  return DDN_OK;
}

static int begin_with_grid(const ddn_fuse_session* s, const GridDev& g, cudaStream_t st) {
  grid_store_kernel<<<1, 32, 0, st>>>(g, (long long)s->cap_units, reinterpret_cast<GridDev*>(s->grid),
                                      reinterpret_cast<unsigned long long*>(s->counts));
  DDN_TRY(after_launch("grid_store_kernel"));
  return launch_clear(s, st);
}

// Grids of more than 2^35 cells: the hashed path on a session and hash buffers carved out of the caller's workspace.
// One layout serves ddn_voxel_fuse, ddn_voxel_partials and ddn_voxel_merge on n points (or records), so
// ddn_fuse_workspace_bytes is the most any of them needs.
struct HashedWork {
  ddn_fuse_session s;  // grid and counts only
  ddn_hash_fuse hf;
  uint64_t* samples;   // [DDN_HASH_SAMPLES + 1]
  int64_t* plan;       // [64]
  void* scratch;       // the accumulator of fuse and partials, the merge's staging
  int64_t scratch_bytes;
};

// Bytes of the layout for n > 0 points; with a (256-byte aligned) base also the pointers into it.  words: accumulator
// words per point (kAccWords, or kAccNormalWords for the normals form).
static int hashed_layout(int64_t n, char* base, HashedWork* w, int64_t* total, int words = kAccWords) {
  int64_t cap_slots, table_bytes, slots_bytes, sort_bytes, hist_bytes, merge_bytes;
  DDN_TRY(ddn_hash_fuse_sizes(n, &cap_slots, &table_bytes, &slots_bytes, &sort_bytes, &hist_bytes));
  DDN_TRY(ddn_fuse_merge_hashed_scratch_bytes(1, n, &merge_bytes));
  const int64_t scratch_bytes = std::max<int64_t>(n * words * 8 + 16, merge_bytes);
  WorkspaceOffsets o;
  const size_t grid = o.take(sizeof(GridDev)), table = o.take(table_bytes), slots = o.take(slots_bytes),
               sort = o.take(sort_bytes), hist = o.take(hist_bytes), state = o.take(DDN_HASH_STATE_BYTES),
               samples = o.take((DDN_HASH_SAMPLES + 1) * 8), plan = o.take(64 * 8), scratch = o.take(scratch_bytes);
  *total = (int64_t)o.off + 256;
  if (base == nullptr) return DDN_OK;
  w->s = ddn_fuse_session{};
  w->s.grid = reinterpret_cast<ddn_grid_state*>(base + grid);
  w->hf.table = base + table;
  w->hf.slots = reinterpret_cast<uint32_t*>(base + slots);
  w->hf.sort = base + sort;
  w->hf.hist = reinterpret_cast<uint32_t*>(base + hist);
  w->hf.state = reinterpret_cast<int64_t*>(base + state);
  w->hf.cap_slots = cap_slots;
  w->hf.cap_voxels = n;
  w->samples = reinterpret_cast<uint64_t*>(base + samples);
  w->plan = reinterpret_cast<int64_t*>(base + plan);
  w->scratch = base + scratch;
  w->scratch_bytes = scratch_bytes;
  return DDN_OK;
}

// Checks the workspace before anything is enqueued, then stores the grid with cap_units = 0, i.e. as
// DDN_GRID_TOO_LARGE (the status on which the hashed path's mode 0 runs), and empties the hash buffers.
static int carve_hashed(const GridDev& g, int64_t n, void* workspace, int64_t workspace_bytes, int64_t* counts_out, HashedWork* w,
                        cudaStream_t st, int words = kAccWords) {
  int64_t total = 0;
  DDN_TRY(hashed_layout(n, reinterpret_cast<char*>(align_up((int64_t)(uintptr_t)workspace, 256)), w, &total, words));
  if (total > workspace_bytes) {
    set_error("fuse workspace too small: %lld < %lld", (long long)workspace_bytes, (long long)total);
    return DDN_ERR_WORKSPACE_TOO_SMALL;
  }
  w->s.counts = counts_out;
  grid_store_kernel<<<1, 32, 0, st>>>(g, 0, reinterpret_cast<GridDev*>(w->s.grid), reinterpret_cast<unsigned long long*>(counts_out));
  DDN_TRY(after_launch("grid_store_kernel"));
  return ddn_hash_fuse_reset(&w->hf, st);
}

static int fuse_workspace_bytes(const ddn_voxel_grid* grid_host, int64_t n_points, int64_t* bytes_out, int words) {
  DDN_REQUIRE(bytes_out != nullptr, "null bytes_out");
  DDN_REQUIRE(n_points >= 0 && n_points < (1ll << 31) - 1024, "n_points");
  const int64_t n = n_points > 0 ? n_points : 1;
  if (grid_host != nullptr) {
    GridDev g;
    DDN_TRY(grid_from_host(grid_host, &g));
    if (use_dense(g)) {
      DenseLayout L;
      dense_layout(g, n, &L, words);
      *bytes_out = (int64_t)L.total;
      return DDN_OK;
    }
  }
  HashedWork w;
  return hashed_layout(n, nullptr, &w, bytes_out, words);
}

// ddn_voxel_fuse, and with normal / out_normal its normals form
static int voxel_fuse(const ddn_voxel_grid* grid_host, int64_t n_points, int64_t row_len, const float* xyz, const uint8_t* rgb,
                      const uint8_t* votes, int32_t vote_threshold, const float* normal, uint64_t* out_keys, float* out_xyz,
                      uint8_t* out_rgb, int32_t* out_count, float* out_normal, int64_t* counts_out, void* workspace,
                      int64_t workspace_bytes, cudaStream_t st) {
  const bool normals = normal != nullptr;
  const int words = normals ? kAccNormalWords : kAccWords;
  GridDev g;
  DDN_TRY(grid_from_host(grid_host, &g));
  DDN_REQUIRE(n_points >= 0 && n_points < (1ll << 31) - 1024, "n_points");
  DDN_REQUIRE(row_len >= 0, "row_len");
  DDN_REQUIRE(counts_out != nullptr, "null counts_out");
  vote_threshold = std::min(vote_threshold, 255);
  if (n_points == 0) return check_cuda(cudaMemsetAsync(counts_out, 0, 16, st), "memset counts");
  DDN_REQUIRE(xyz && rgb && out_keys && out_xyz && out_rgb && out_count && workspace, "null pointer");
  if (!use_dense(g)) {
    HashedWork w;
    DDN_TRY(carve_hashed(g, n_points, workspace, workspace_bytes, counts_out, &w, st, words));
    if (normals)
      return ddn_fuse_finish_hashed_normals(&w.s, &w.hf, 0, n_points, row_len, xyz, rgb, votes, vote_threshold, normal, nullptr, 0,
                                            out_keys, out_xyz, out_rgb, out_count, out_normal, n_points, w.scratch, w.scratch_bytes, st);
    return ddn_fuse_finish_hashed(&w.s, &w.hf, 0, n_points, row_len, xyz, rgb, votes, vote_threshold, nullptr, 0, out_keys, out_xyz,
                                  out_rgb, out_count, n_points, w.scratch, w.scratch_bytes, st);
  }
  ddn_fuse_session s;
  unsigned long long* accum;
  DenseLayout L;
  DDN_TRY(carve_session(g, n_points, workspace, workspace_bytes, &s, counts_out, &accum, &L, words));
  DDN_TRY(begin_with_grid(&s, g, st));
  DDN_TRY(launch_mark_points(&s, n_points, xyz, votes, vote_threshold, st));
  const long long cap = (long long)std::min<uint64_t>((uint64_t)n_points, L.cells);
  DDN_TRY(launch_rank(&s, ScanRange{0, -1}, out_keys, 1, accum, words, cap, nullptr, st));
  DDN_TRY(launch_accumulate_points(&s, n_points, row_len, xyz, rgb, votes, vote_threshold, accum, words, cap, st, normal));
  return launch_finalize(&s, accum, out_keys, cap, out_xyz, out_rgb, out_count, st, out_normal);
}

// ddn_fuse_finish, and with normal / out_normal its normals form
static int fuse_finish(const ddn_fuse_session* s, int64_t n_points, int64_t row_len, const float* xyz, const uint8_t* rgb,
                       const uint8_t* votes, int32_t vote_threshold, const float* normal, uint64_t* out_keys, float* out_xyz,
                       uint8_t* out_rgb, int32_t* out_count, float* out_normal, int64_t cap_out, void* accum, int64_t accum_bytes,
                       cudaStream_t st) {
  const int words = out_normal != nullptr ? kAccNormalWords : kAccWords;
  DDN_TRY(session_check(s));
  DDN_REQUIRE(n_points >= 0 && n_points < (1ll << 31) - 1024, "n_points");
  DDN_REQUIRE(row_len >= 0, "row_len");
  DDN_REQUIRE(cap_out > 0 && cap_out < (1ll << 31), "cap_out");
  DDN_REQUIRE(out_keys && out_xyz && out_rgb && out_count && accum, "null pointer");
  DDN_REQUIRE(accum_bytes >= cap_out * words * 8 + 16 && (uintptr_t)accum % 16 == 0, "accumulator scratch");
  DDN_REQUIRE(n_points == 0 || (xyz && rgb), "null pointer");
  vote_threshold = std::min(vote_threshold, 255);
  unsigned long long* acc = (unsigned long long*)accum;
  DDN_TRY(launch_rank(s, ScanRange{0, -1}, out_keys, 1, acc, words, cap_out, nullptr, st));
  if (n_points > 0)
    DDN_TRY(launch_accumulate_points(s, n_points, row_len, xyz, rgb, votes, vote_threshold, acc, words, cap_out, st, normal));
  return launch_finalize(s, acc, out_keys, cap_out, out_xyz, out_rgb, out_count, st, out_normal);
}

// ddn_fuse_merge_scratch_bytes for records of rec_words u64: staging [cap_out records], then the gathered tile prefixes
static int merge_scratch_bytes(int64_t cap_units, int32_t n_ranks, int64_t cap_out, int rec_words, int64_t* bytes_out) {
  DDN_REQUIRE(bytes_out != nullptr && cap_units > 0 && n_ranks >= 1 && n_ranks <= DDN_MAX_PEERS && cap_out > 0, "arguments");
  const int64_t stride = cap_units / kOwnUnits + 2;
  *bytes_out = align_up(cap_out * rec_words * 8, 256) + (int64_t)(n_ranks + 1) * stride * 4 + 256;
  return DDN_OK;
}

// ddn_fuse_finish_partial, and with `normals` its normals form: records of DDN_RECORD_NORMAL_WORDS u64, whose zeroed
// pad word the accumulate pass never touches
static int fuse_finish_partial(const ddn_fuse_session* s, int64_t n_points, int64_t row_len, const float* xyz, const uint8_t* rgb,
                               const uint8_t* votes, int32_t vote_threshold, const float* normal, bool normals, uint64_t* records,
                               int64_t cap_records, cudaStream_t st) {
  const int w = normals ? DDN_RECORD_NORMAL_WORDS : kRecWords;
  DDN_TRY(session_check(s));
  DDN_REQUIRE(n_points >= 0 && n_points < (1ll << 31) - 1024, "n_points");
  DDN_REQUIRE(row_len >= 0, "row_len");
  DDN_REQUIRE(cap_records > 0 && cap_records < (1ll << 31), "cap_records");
  DDN_REQUIRE(records != nullptr && (uintptr_t)records % 16 == 0, "records must be 16-byte aligned");
  DDN_REQUIRE(n_points == 0 || (xyz && rgb), "null pointer");
  DDN_REQUIRE(!normals || n_points == 0 || normal != nullptr, "null pointer");
  vote_threshold = std::min(vote_threshold, 255);
  unsigned long long* rec = (unsigned long long*)records;
  DDN_TRY(launch_rank(s, ScanRange{0, -1}, (uint64_t*)rec, w, rec, w, cap_records, s->tile_prefix, st));
  if (n_points == 0) return DDN_OK;
  return launch_accumulate_points(s, n_points, row_len, xyz, rgb, votes, vote_threshold, rec + 1, w, cap_records, st,
                                  normals ? normal : nullptr);
}

// ddn_fuse_merge_peers, and with `normals` its normals form (records of DDN_RECORD_NORMAL_WORDS u64, accumulators of
// kAccNormalWords, out_normal)
static int merge_peers(const ddn_fuse_session* s, int32_t rank, int32_t n_ranks, const void* const* peer_records_host,
                       const void* const* peer_tile_prefix_host, int64_t* plan, void* scratch, int64_t scratch_bytes, const float* drop_xyz,
                       int64_t n_drop, uint64_t* out_keys, float* out_xyz, uint8_t* out_rgb, int32_t* out_count, float* out_normal,
                       bool normals, int64_t cap_out, void* accum, int64_t accum_bytes, cudaStream_t st) {
  const int words = normals ? kAccNormalWords : kAccWords;
  const int rec_words = normals ? DDN_RECORD_NORMAL_WORDS : kRecWords;
  DDN_REQUIRE(n_drop >= 0 && n_drop < (1ll << 31) - 1024 && (n_drop == 0 || drop_xyz != nullptr), "drop points");
  DDN_TRY(session_check(s));
  DDN_REQUIRE(n_ranks >= 1 && n_ranks <= DDN_MAX_PEERS && rank >= 0 && rank < n_ranks, "rank / n_ranks");
  DDN_REQUIRE(peer_records_host && peer_tile_prefix_host && plan && scratch, "null pointer");
  DDN_REQUIRE(cap_out > 0 && cap_out < (1ll << 31), "cap_out");
  DDN_REQUIRE(out_keys && out_xyz && out_rgb && out_count && accum, "null pointer");
  DDN_REQUIRE(!normals || out_normal != nullptr, "null pointer");
  DDN_REQUIRE(accum_bytes >= cap_out * words * 8 + 16 && (uintptr_t)accum % 16 == 0,
              normals ? "accumulator scratch (cap_out * 64 bytes)" : "accumulator scratch");
  int64_t need = 0;
  DDN_TRY(merge_scratch_bytes(s->cap_units, n_ranks, cap_out, rec_words, &need));
  DDN_REQUIRE(scratch_bytes >= need && (uintptr_t)scratch % 16 == 0,
              normals ? "merge scratch too small (ddn_fuse_merge_normals_scratch_bytes)" : "merge scratch too small (ddn_fuse_merge_scratch_bytes)");
  PeerPtrs pr, pp;
  for (int q = 0; q < DDN_MAX_PEERS; ++q) {
    pr.p[q] = q < n_ranks ? peer_records_host[q] : nullptr;
    pp.p[q] = q < n_ranks ? peer_tile_prefix_host[q] : nullptr;
    if (q < n_ranks) DDN_REQUIRE(pr.p[q] && pp.p[q], "null peer pointer");
  }
  if (normals)
    for (int q = 0; q < n_ranks; ++q) DDN_REQUIRE((uintptr_t)pr.p[q] % 16 == 0, "records must be 16-byte aligned");
  DDN_REQUIRE(pp.p[rank] == (const void*)s->tile_prefix, "entry `rank` must be the session's own buffers");
  const GridDev* gp = reinterpret_cast<const GridDev*>(s->grid);
  const FuseDev f = fuse_dev(s);
  unsigned long long* counts = reinterpret_cast<unsigned long long*>(s->counts);
  long long* planll = reinterpret_cast<long long*>(plan);
  unsigned long long* acc = (unsigned long long*)accum;
  const long long stride = (long long)(s->cap_units / kOwnUnits + 2);
  ulonglong2* staging = reinterpret_cast<ulonglong2*>(scratch);                                         // [cap_out] records
  uint32_t* local = reinterpret_cast<uint32_t*>(reinterpret_cast<char*>(scratch) + align_up(cap_out * rec_words * 8, 256));  // [(R + 1) * stride]
  merge_gather_prefix_kernel<<<kNumSMs * 2, 256, 0, st>>>(gp, pp, n_ranks, local, stride);
  DDN_TRY(after_launch("merge_gather_prefix_kernel", st));
  merge_plan_kernel<<<1, 32, 0, st>>>(gp, local, stride, rank, n_ranks, planll);
  DDN_TRY(after_launch("merge_plan_kernel", st));
  merge_clear_kernel<<<kPersistentCtas, kOwnUnits, 0, st>>>(f, planll);
  DDN_TRY(after_launch("merge_clear_kernel", st));
  // (fewer CTAs per SM, to leave room for another stream's kernels, cost the pull 3-14 % on 2 GPUs: -DDDN_PULL_CTAS_PER_SM)
  if (normals) {
    merge_pull_mark_normals_kernel<<<kNumSMs * DDN_PULL_CTAS_PER_SM, 256, 0, st>>>(f, pr, rank, n_ranks, planll, staging, cap_out);
    DDN_TRY(after_launch("merge_pull_mark_normals_kernel", st));
  } else {
    merge_pull_mark_kernel<<<kNumSMs * DDN_PULL_CTAS_PER_SM, 256, 0, st>>>(f, pr, rank, n_ranks, planll, staging, cap_out);
    DDN_TRY(after_launch("merge_pull_mark_kernel", st));
  }
  if (n_drop > 0) {  // N5: the cells of the sparse cloud leave the merged occupancy
    unmark_points_kernel<<<(unsigned)((n_drop + 255) / 256), 256, 0, st>>>(f, n_drop, drop_xyz, planll);
    DDN_TRY(after_launch("unmark_points_kernel", st));
  }
  merge_count_kernel<<<kPersistentCtas, kOwnUnits, 0, st>>>(f, planll, s->tile_sums);
  DDN_TRY(after_launch("merge_count_kernel", st));
  tile_scan_kernel<<<1, 1024, 0, st>>>(gp, ScanRange{0, 0}, planll, s->tile_sums, counts);
  DDN_TRY(after_launch("tile_scan_kernel", st));
  zero_accum_kernel<<<kPersistentCtas, 256, 0, st>>>((ulonglong2*)acc, counts, words, cap_out);
  DDN_TRY(after_launch("zero_accum_kernel", st));
  merge_prefix_kernel<<<kPersistentCtas, kOwnUnits, 0, st>>>(f, planll, s->tile_sums, out_keys, cap_out);
  DDN_TRY(after_launch("merge_prefix_kernel", st));
  if (normals) {
    merge_accumulate_normals_kernel<<<kPersistentCtas, 256, 0, st>>>(f, planll, staging, cap_out, acc, cap_out);
    DDN_TRY(after_launch("merge_accumulate_normals_kernel", st));
  } else {
    merge_accumulate_kernel<<<kPersistentCtas, 256, 0, st>>>(f, planll, staging, cap_out, acc, cap_out);
    DDN_TRY(after_launch("merge_accumulate_kernel", st));
  }
  return launch_finalize(s, acc, out_keys, cap_out, out_xyz, out_rgb, out_count, st, normals ? out_normal : nullptr);
}

}  // namespace ddn

extern "C" {

int ddn_fuse_workspace_bytes(const ddn_voxel_grid* grid_host, int64_t n_points, int64_t* bytes_out) {
  return ddn::fuse_workspace_bytes(grid_host, n_points, bytes_out, ddn::kAccWords);
}

int ddn_fuse_normals_workspace_bytes(const ddn_voxel_grid* grid_host, int64_t n_points, int64_t* bytes_out) {
  return ddn::fuse_workspace_bytes(grid_host, n_points, bytes_out, ddn::kAccNormalWords);
}

int ddn_voxel_fuse(const ddn_voxel_grid* grid_host, int64_t n_points, int64_t row_len, const float* xyz, const uint8_t* rgb,
                   const uint8_t* votes, int32_t vote_threshold, uint64_t* out_keys, float* out_xyz,
                   uint8_t* out_rgb, int32_t* out_count, int64_t* counts_out, void* workspace,
                   int64_t workspace_bytes, void* stream) {
  return ddn::voxel_fuse(grid_host, n_points, row_len, xyz, rgb, votes, vote_threshold, nullptr, out_keys, out_xyz, out_rgb, out_count,
                         nullptr, counts_out, workspace, workspace_bytes, (cudaStream_t)stream);
}

int ddn_voxel_fuse_normals(const ddn_voxel_grid* grid_host, int64_t n_points, int64_t row_len, const float* xyz, const uint8_t* rgb,
                           const uint8_t* votes, int32_t vote_threshold, const float* normal, uint64_t* out_keys, float* out_xyz,
                           uint8_t* out_rgb, int32_t* out_count, float* out_normal, int64_t* counts_out, void* workspace,
                           int64_t workspace_bytes, void* stream) {
  DDN_REQUIRE(n_points == 0 || (normal && out_normal), "null pointer");
  return ddn::voxel_fuse(grid_host, n_points, row_len, xyz, rgb, votes, vote_threshold, normal, out_keys, out_xyz, out_rgb, out_count,
                         out_normal, counts_out, workspace, workspace_bytes, (cudaStream_t)stream);
}

int ddn_fuse_tile_info(const ddn_voxel_grid* grid_host, int64_t* n_tiles, int64_t* cells_per_tile) {
  using namespace ddn;
  DDN_REQUIRE(n_tiles != nullptr && cells_per_tile != nullptr, "null output");
  GridDev g;
  DDN_TRY(grid_from_host(grid_host, &g));
  *n_tiles = 0;
  *cells_per_tile = (int64_t)kOwnUnits * kUnitBits;
  if (use_dense(g)) {
    DenseLayout L;
    dense_layout(g, 1, &L);
    *n_tiles = (int64_t)L.own_tiles;
  }
  return DDN_OK;
}

int ddn_voxel_partials(const ddn_voxel_grid* grid_host, int64_t n_points, int64_t row_len, const float* xyz, const uint8_t* rgb,
                       const uint8_t* votes, int32_t vote_threshold, uint64_t* records, uint32_t* tile_prefix,
                       int64_t* counts_out, void* workspace, int64_t workspace_bytes, void* stream) {
  using namespace ddn;
  GridDev g;
  DDN_TRY(grid_from_host(grid_host, &g));
  DDN_REQUIRE(n_points >= 0 && n_points < (1ll << 31) - 1024, "n_points");
  DDN_REQUIRE(row_len >= 0, "row_len");
  DDN_REQUIRE(counts_out != nullptr, "null counts_out");
  cudaStream_t st = (cudaStream_t)stream;
  vote_threshold = std::min(vote_threshold, 255);
  if (n_points == 0) {
    if (tile_prefix != nullptr && use_dense(g)) {
      DenseLayout L;
      dense_layout(g, 1, &L);
      DDN_TRY(check_cuda(cudaMemsetAsync(tile_prefix, 0, (size_t)(L.own_tiles + 1) * 4, st), "memset tile prefix"));
    }
    return check_cuda(cudaMemsetAsync(counts_out, 0, 16, st), "memset counts");
  }
  DDN_REQUIRE(xyz && rgb && records && workspace, "null pointer");
  DDN_REQUIRE((uintptr_t)records % 16 == 0, "records must be 16-byte aligned");
  if (!use_dense(g)) {  // records sorted by compact key, which orders as the canonical key
    HashedWork w;
    DDN_TRY(carve_hashed(g, n_points, workspace, workspace_bytes, counts_out, &w, st));
    return ddn_fuse_finish_hashed_partial(&w.s, &w.hf, 0, n_points, row_len, xyz, rgb, votes, vote_threshold, nullptr, 0, records,
                                          n_points, w.samples, w.scratch, w.scratch_bytes, st);
  }
  ddn_fuse_session s;
  unsigned long long* accum;
  DenseLayout L;
  DDN_TRY(carve_session(g, n_points, workspace, workspace_bytes, &s, counts_out, &accum, &L));
  DDN_TRY(begin_with_grid(&s, g, st));
  DDN_TRY(launch_mark_points(&s, n_points, xyz, votes, vote_threshold, st));
  unsigned long long* rec = (unsigned long long*)records;
  const long long cap = (long long)n_points;
  DDN_TRY(launch_rank(&s, ScanRange{0, -1}, (uint64_t*)rec, kRecWords, rec, kRecWords, cap, tile_prefix, st));
  return launch_accumulate_points(&s, n_points, row_len, xyz, rgb, votes, vote_threshold, rec + 1, kRecWords, cap, st);
}

int ddn_voxel_merge(const ddn_voxel_grid* grid_host, int64_t n_records, const uint64_t* records, int64_t tile_begin,
                    int64_t tile_end, uint64_t* out_keys, float* out_xyz, uint8_t* out_rgb, int32_t* out_count,
                    int64_t* counts_out, void* workspace, int64_t workspace_bytes, void* stream) {
  using namespace ddn;
  GridDev g;
  DDN_TRY(grid_from_host(grid_host, &g));
  DDN_REQUIRE(n_records >= 0 && n_records < (1ll << 31) - 1024, "n_records");
  DDN_REQUIRE(counts_out != nullptr, "null counts_out");
  cudaStream_t st = (cudaStream_t)stream;
  if (n_records == 0) return check_cuda(cudaMemsetAsync(counts_out, 0, 16, st), "memset counts");
  DDN_REQUIRE(records && out_keys && out_xyz && out_rgb && out_count && workspace, "null pointer");
  if (!use_dense(g)) {
    // The records, in any order, merged as the only rank's: with no splitters the cut is [0, n_records) whatever the
    // sample keys, as long as they stay below ~0.  hash_begin on an empty step arms the path first (and zeroes
    // counts); counts[0] then reports the records, or -1 when the merge finds a voxel of 2^24 or more points.
    HashedWork w;
    DDN_TRY(carve_hashed(g, n_records, workspace, workspace_bytes, counts_out, &w, st));
    HashDev h;
    DDN_TRY(hash_dev(&w.hf, &h));
    DDN_TRY(hash_launch_points(reinterpret_cast<GridDev*>(w.s.grid), h, reinterpret_cast<unsigned long long*>(counts_out), 0, 0, 0,
                               nullptr, nullptr, nullptr, 0, nullptr, 0, nullptr, st));
    const int64_t m = n_records;
    DDN_TRY(check_cuda(cudaMemsetAsync(w.samples, 0, DDN_HASH_SAMPLES * 8, st), "memset samples"));
    DDN_TRY(check_cuda(cudaMemcpyAsync(w.samples + DDN_HASH_SAMPLES, &m, 8, cudaMemcpyHostToDevice, st), "copy record count"));
    DDN_TRY(check_cuda(cudaMemcpyAsync(counts_out, &m, 8, cudaMemcpyHostToDevice, st), "copy record count"));
    const void* rec = records;
    const void* smp = w.samples;
    return ddn_fuse_merge_hashed_peers(&w.s, &w.hf, 0, 1, &rec, &smp, w.plan, w.scratch, w.scratch_bytes, out_keys, out_xyz, out_rgb,
                                       out_count, n_records, st);
  }
  ddn_fuse_session s;
  unsigned long long* accum;
  DenseLayout L;
  DDN_TRY(carve_session(g, n_records, workspace, workspace_bytes, &s, counts_out, &accum, &L));
  // ownership tiles -> owned cell range and the scan tiles that enclose it
  if (tile_end <= 0) tile_begin = 0, tile_end = (int64_t)L.own_tiles;
  DDN_REQUIRE(tile_begin >= 0 && tile_begin <= tile_end && tile_end <= (int64_t)L.own_tiles, "tile range");
  const uint64_t cell_begin = (uint64_t)tile_begin * kOwnUnits * kUnitBits;
  const uint64_t cell_end = (uint64_t)tile_end * kOwnUnits * kUnitBits;
  ScanRange range;
  range.tile_begin = tile_begin / kOwnPerScanTile;
  range.n_tiles = tile_end > tile_begin ? (tile_end + kOwnPerScanTile - 1) / kOwnPerScanTile - range.tile_begin : 0;
  grid_store_kernel<<<1, 32, 0, st>>>(g, (long long)s.cap_units, reinterpret_cast<GridDev*>(s.grid),
                                      reinterpret_cast<unsigned long long*>(s.counts));
  DDN_TRY(after_launch("grid_store_kernel"));
  if (range.n_tiles == 0) return DDN_OK;
  {
    const size_t ub = (size_t)range.tile_begin * kTileUnits;
    const size_t ue = std::min((size_t)(range.tile_begin + range.n_tiles) * kTileUnits, (size_t)L.n_units);
    DDN_TRY(check_cuda(cudaMemsetAsync(reinterpret_cast<uint4*>(s.units) + ub, 0, (ue - ub) * 16, st), "memset occupancy"));
  }
  const unsigned blocks = (unsigned)((n_records + 255) / 256);
  mark_records_kernel<<<blocks, 256, 0, st>>>(fuse_dev(&s), n_records, records, cell_begin, cell_end);
  DDN_TRY(after_launch("mark_records_kernel"));
  const long long cap = (long long)std::min<uint64_t>((uint64_t)n_records, L.cells);
  DDN_TRY(launch_rank(&s, range, out_keys, 1, accum, kAccWords, cap, nullptr, st));
  accumulate_records_kernel<<<blocks, 256, 0, st>>>(reinterpret_cast<const GridDev*>(s.grid), n_records,
                                                    (const unsigned long long*)records, reinterpret_cast<const uint4*>(s.units),
                                                    cell_begin, cell_end, accum, cap);
  DDN_TRY(after_launch("accumulate_records_kernel"));
  return launch_finalize(&s, accum, out_keys, cap, out_xyz, out_rgb, out_count, st);
}

int ddn_voxel_keys(const ddn_voxel_grid* grid_host, int64_t n_points, const float* xyz, uint64_t* keys, void* stream) {
  using namespace ddn;
  DDN_REQUIRE(grid_host != nullptr && grid_host->voxel > 0.f, "grid");
  DDN_REQUIRE(n_points >= 0, "n_points");
  if (n_points == 0) return DDN_OK;
  DDN_REQUIRE(xyz && keys, "null pointer");
  GridDev g;
  g.voxel = grid_host->voxel;
  g.ox = grid_host->origin[0];
  g.oy = grid_host->origin[1];
  g.oz = grid_host->origin[2];
  g.bx = g.by = g.bz = 21;
  g.nx = g.ny = g.nz = 1 << 21;
  canonical_key_kernel<<<(unsigned)((n_points + 255) / 256), 256, 0, (cudaStream_t)stream>>>(g, n_points, xyz, keys);
  return after_launch("canonical_key_kernel");
}

// ---- fusion session ------------------------------------------------------------------------------
int ddn_fuse_session_sizes(int64_t max_cells, int64_t* cap_units, int64_t* units_bytes, int64_t* dirty_bytes,
                           int64_t* tile_sums_bytes, int64_t* tile_prefix_bytes) {
  using namespace ddn;
  DDN_REQUIRE(max_cells > 0 && (uint64_t)max_cells <= kDenseMaxCells, "max_cells must be in (0, 2^35]");
  DDN_REQUIRE(cap_units && units_bytes && dirty_bytes && tile_sums_bytes && tile_prefix_bytes, "null output");
  const int64_t cu = align_up((max_cells + kUnitBits - 1) / kUnitBits, kTileUnits);
  *cap_units = cu;
  *units_bytes = cu * 16;
  *dirty_bytes = align_up(cu / kTileUnits + 1, 256);
  *tile_sums_bytes = align_up((cu / kOwnUnits + 2) * 4, 256);
  *tile_prefix_bytes = align_up((cu / kOwnUnits + 2) * 4, 256);
  return DDN_OK;
}

int ddn_fuse_merge_scratch_bytes(int64_t cap_units, int32_t n_ranks, int64_t cap_out, int64_t* bytes_out) {
  return ddn::merge_scratch_bytes(cap_units, n_ranks, cap_out, ddn::kRecWords, bytes_out);
}

int ddn_fuse_merge_normals_scratch_bytes(int64_t cap_units, int32_t n_ranks, int64_t cap_out, int64_t* bytes_out) {
  return ddn::merge_scratch_bytes(cap_units, n_ranks, cap_out, DDN_RECORD_NORMAL_WORDS, bytes_out);
}

int ddn_fuse_session_reset(const ddn_fuse_session* s, void* stream) {
  using namespace ddn;
  DDN_TRY(session_check(s));
  cudaStream_t st = (cudaStream_t)stream;
  DDN_TRY(check_cuda(cudaMemsetAsync(s->units, 0, (size_t)s->cap_units * 16, st), "memset units"));
  if (s->dirty != nullptr) DDN_TRY(check_cuda(cudaMemsetAsync(s->dirty, 0, (size_t)(s->cap_units / kTileUnits + 1), st), "memset flags"));
  DDN_TRY(check_cuda(cudaMemsetAsync(s->grid, 0, sizeof(ddn_grid_state), st), "memset grid"));
  return check_cuda(cudaMemsetAsync(s->counts, 0, 16, st), "memset counts");
}

int ddn_fuse_begin(const ddn_fuse_session* s, const void* const* bbox_ptrs_host, int32_t n_boxes, float voxel, void* stream) {
  using namespace ddn;
  DDN_TRY(session_check(s));
  DDN_REQUIRE(bbox_ptrs_host != nullptr && n_boxes >= 1 && n_boxes <= DDN_MAX_PEERS, "bounding boxes");
  DDN_REQUIRE(voxel > 0.f, "voxel size");
  cudaStream_t st = (cudaStream_t)stream;
  BoxPtrs boxes;
  boxes.n = n_boxes;
  for (int i = 0; i < DDN_MAX_PEERS; ++i) boxes.p[i] = i < n_boxes ? reinterpret_cast<const int*>(bbox_ptrs_host[i]) : nullptr;
  for (int i = 0; i < n_boxes; ++i) DDN_REQUIRE(boxes.p[i] != nullptr, "null bounding box");
  grid_from_bbox_kernel<<<1, 32, 0, st>>>(boxes, voxel, (long long)s->cap_units, reinterpret_cast<GridDev*>(s->grid),
                                          reinterpret_cast<unsigned long long*>(s->counts));
  DDN_TRY(after_launch("grid_from_bbox_kernel"));
  return launch_clear(s, st);
}

int ddn_fuse_begin_grid(const ddn_fuse_session* s, const ddn_voxel_grid* grid_host, void* stream) {
  using namespace ddn;
  DDN_TRY(session_check(s));
  GridDev g;
  DDN_TRY(grid_from_host(grid_host, &g));
  DDN_REQUIRE(use_dense(g), "grid too large for a fusion session (more than 2^35 cells)");
  return begin_with_grid(s, g, (cudaStream_t)stream);
}

int ddn_fuse_mark_points(const ddn_fuse_session* s, int64_t n_points, const float* xyz, const uint8_t* votes,
                         int32_t vote_threshold, void* stream) {
  using namespace ddn;
  DDN_TRY(session_check(s));
  DDN_REQUIRE(n_points >= 0 && n_points < (1ll << 31) - 1024, "n_points");
  if (n_points == 0) return DDN_OK;
  DDN_REQUIRE(xyz != nullptr, "null pointer");
  return launch_mark_points(s, n_points, xyz, votes, std::min(vote_threshold, 255), (cudaStream_t)stream);
}

int ddn_fuse_unmark_points(const ddn_fuse_session* s, int64_t n_points, const float* xyz, void* stream) {
  using namespace ddn;
  DDN_TRY(session_check(s));
  DDN_REQUIRE(n_points >= 0 && n_points < (1ll << 31) - 1024, "n_points");
  if (n_points == 0) return DDN_OK;
  DDN_REQUIRE(xyz != nullptr, "null pointer");
  unmark_points_kernel<<<(unsigned)((n_points + 255) / 256), 256, 0, (cudaStream_t)stream>>>(fuse_dev(s), n_points, xyz, nullptr);
  return after_launch("unmark_points_kernel");
}

int ddn_fuse_finish(const ddn_fuse_session* s, int64_t n_points, int64_t row_len, const float* xyz, const uint8_t* rgb,
                    const uint8_t* votes, int32_t vote_threshold, uint64_t* out_keys, float* out_xyz, uint8_t* out_rgb,
                    int32_t* out_count, int64_t cap_out, void* accum, int64_t accum_bytes, void* stream) {
  return ddn::fuse_finish(s, n_points, row_len, xyz, rgb, votes, vote_threshold, nullptr, out_keys, out_xyz, out_rgb, out_count, nullptr,
                          cap_out, accum, accum_bytes, (cudaStream_t)stream);
}

int ddn_fuse_finish_normals(const ddn_fuse_session* s, int64_t n_points, int64_t row_len, const float* xyz, const uint8_t* rgb,
                            const uint8_t* votes, int32_t vote_threshold, const float* normal, uint64_t* out_keys, float* out_xyz,
                            uint8_t* out_rgb, int32_t* out_count, float* out_normal, int64_t cap_out, void* accum, int64_t accum_bytes,
                            void* stream) {
  DDN_REQUIRE(out_normal != nullptr && (n_points == 0 || normal != nullptr), "null pointer");
  return ddn::fuse_finish(s, n_points, row_len, xyz, rgb, votes, vote_threshold, normal, out_keys, out_xyz, out_rgb, out_count, out_normal,
                          cap_out, accum, accum_bytes, (cudaStream_t)stream);
}

int ddn_fuse_finish_partial(const ddn_fuse_session* s, int64_t n_points, int64_t row_len, const float* xyz, const uint8_t* rgb,
                            const uint8_t* votes, int32_t vote_threshold, uint64_t* records, int64_t cap_records, void* stream) {
  return ddn::fuse_finish_partial(s, n_points, row_len, xyz, rgb, votes, vote_threshold, nullptr, false, records, cap_records,
                                  (cudaStream_t)stream);
}

int ddn_fuse_finish_partial_normals(const ddn_fuse_session* s, int64_t n_points, int64_t row_len, const float* xyz, const uint8_t* rgb,
                                    const uint8_t* votes, int32_t vote_threshold, const float* normal, uint64_t* records,
                                    int64_t cap_records, void* stream) {
  return ddn::fuse_finish_partial(s, n_points, row_len, xyz, rgb, votes, vote_threshold, normal, true, records, cap_records,
                                  (cudaStream_t)stream);
}

int ddn_fuse_merge_peers(const ddn_fuse_session* s, int32_t rank, int32_t n_ranks, const void* const* peer_records_host,
                         const void* const* peer_tile_prefix_host, int64_t* plan, void* scratch, int64_t scratch_bytes,
                         const float* drop_xyz, int64_t n_drop, uint64_t* out_keys, float* out_xyz, uint8_t* out_rgb,
                         int32_t* out_count, int64_t cap_out, void* accum, int64_t accum_bytes, void* stream) {
  return ddn::merge_peers(s, rank, n_ranks, peer_records_host, peer_tile_prefix_host, plan, scratch, scratch_bytes, drop_xyz, n_drop,
                          out_keys, out_xyz, out_rgb, out_count, nullptr, false, cap_out, accum, accum_bytes, (cudaStream_t)stream);
}

int ddn_fuse_merge_peers_normals(const ddn_fuse_session* s, int32_t rank, int32_t n_ranks, const void* const* peer_records_host,
                                 const void* const* peer_tile_prefix_host, int64_t* plan, void* scratch, int64_t scratch_bytes,
                                 const float* drop_xyz, int64_t n_drop, uint64_t* out_keys, float* out_xyz, uint8_t* out_rgb,
                                 int32_t* out_count, float* out_normal, int64_t cap_out, void* accum, int64_t accum_bytes, void* stream) {
  return ddn::merge_peers(s, rank, n_ranks, peer_records_host, peer_tile_prefix_host, plan, scratch, scratch_bytes, drop_xyz, n_drop,
                          out_keys, out_xyz, out_rgb, out_count, out_normal, true, cap_out, accum, accum_bytes, (cudaStream_t)stream);
}

}  // extern "C"
