// Shared definitions of stage 4 (voxel-grid fusion): grid description, IEEE-exact voxel coordinates,
// the occupancy-unit layout, fixed-point offsets and the finalisation of one voxel.  Used by the
// dense-rank path (fuse.cu), by K4's fused occupancy marking (filter.cu) and by the hashed path for grids
// too large for a dense occupancy bitmap (fuse_hash.cu, fuse_hash_peers.cu).
#pragma once

#include "common.cuh"
#include "voxel_quotient.cuh"

namespace ddn {

// Same layout as ddn_grid_state (include/ddn_b200.h): the grid lives in DEVICE memory, so a step needs no
// host round trip between the bounding box and the fusion passes.  Host-grid entry points fill one on
// the host and pass it by value to a one-thread kernel that stores it.
struct GridDev {
  float voxel, ox, oy, oz;
  int bx, by, bz;     // significant bits per axis (the hashed path's compact key packing)
  int nx, ny, nz;     // cells per axis; a point outside [0, n) on any axis does not participate
  long long n_units;  // ceil(cells / 96); 0 when status != DDN_GRID_OK
  int status, reserved;
  long long cells;
};
static_assert(sizeof(GridDev) == sizeof(ddn_grid_state), "GridDev mirrors ddn_grid_state");

inline int grid_from_host(const ddn_voxel_grid* h, GridDev* g) {
  DDN_REQUIRE(h != nullptr, "null grid");
  DDN_REQUIRE(h->voxel > 0.f, "voxel size");
  for (int i = 0; i < 3; ++i) DDN_REQUIRE(h->bits[i] >= 1 && h->bits[i] <= 21, "bits per axis must be in [1,21]");
  for (int i = 0; i < 3; ++i)
    DDN_REQUIRE(h->dims[i] >= 0 && h->dims[i] <= (1 << h->bits[i]), "dims per axis must be in [0, 2^bits]");
  g->voxel = h->voxel;
  g->ox = h->origin[0];
  g->oy = h->origin[1];
  g->oz = h->origin[2];
  g->bx = h->bits[0];
  g->by = h->bits[1];
  g->bz = h->bits[2];
  g->nx = h->dims[0] > 0 ? h->dims[0] : (1 << h->bits[0]);
  g->ny = h->dims[1] > 0 ? h->dims[1] : (1 << h->bits[1]);
  g->nz = h->dims[2] > 0 ? h->dims[2] : (1 << h->bits[2]);
  g->cells = (long long)g->nx * (long long)g->ny * (long long)g->nz;
  g->n_units = (g->cells + 95) / 96;
  g->status = DDN_GRID_OK;
  g->reserved = 0;
  return DDN_OK;
}

// k = floor((p - o) / voxel) with IEEE float32 sub and div (bit-exact with the numpy definition), through the
// division-free quotient of voxel_quotient.cuh.
__device__ __forceinline__ float voxel_coord(float p, float o, float voxel, float rvoxel) {
  return voxel_floor(__fsub_rn(p, o), voxel, rvoxel);
}
// voxel_coord's quotient for a pair of values (K4's fused mark), before the floor: each lane of the result is
// fl((p - o) / voxel) where voxel_quotient_in_domain holds or the lane's `use` flag is clear.  `all_exact` is cleared
// where neither holds; the caller then takes voxel_coord for those values.
__device__ __forceinline__ f32x2 voxel_quotient2(f32x2 p, float o, float voxel, float rvoxel, bool use0, bool use1,
                                                 bool& all_exact) {
  const f32x2 a = sub2(p, splat2(o));
  const f32x2 rv2 = splat2(rvoxel);
  const f32x2 q = mul2(a, rv2);
  float q0, q1;
  unpack2(q, q0, q1);
  all_exact &= (voxel_quotient_in_domain(q0) | !use0) & (voxel_quotient_in_domain(q1) | !use1);
  return fma2(fma2(q, splat2(-voxel), a), rv2, q);
}

constexpr int kFixShift = 20;  // offsets are stored in units of voxel * 2^-20

__device__ __forceinline__ float voxel_centre(float o, uint32_t k, float voxel) {
  return __fadd_rn(o, __fmul_rn((float)k + 0.5f, voxel));
}

// (p - voxel centre) * fix_scale rounded to nearest, fix_scale = fl(1/voxel) * 2^20: the integer a point
// adds to its voxel's sum (|result| <= 2^19 for a point inside the voxel).  One multiply, no division:
// the value only has to be the SAME everywhere (kernels, ranks, the numpy statement), not a quotient.
__host__ __device__ __forceinline__ float voxel_fix_scale(float voxel) { return (1.0f / voxel) * (float)(1 << kFixShift); }
__device__ __forceinline__ int voxel_offset_fix(float p, float centre, float fix_scale) {
  return __float2int_rn(__fmul_rn(__fsub_rn(p, centre), fix_scale));
}

// mean position = centre + (sum / count) * voxel * 2^-20 (float64, once per voxel); colour = round-half-up
__device__ __forceinline__ void finalize_voxel(const GridDev& g, float cx, float cy, float cz, long long sx, long long sy,
                                               long long sz, unsigned long long sr, unsigned long long sg,
                                               unsigned long long sb, long long cnt, float* __restrict__ oxyz,
                                               uint8_t* __restrict__ orgb) {
  const double inv = (double)g.voxel / ((double)cnt * (double)(1 << kFixShift));
  oxyz[0] = (float)((double)cx + (double)sx * inv);
  oxyz[1] = (float)((double)cy + (double)sy * inv);
  oxyz[2] = (float)((double)cz + (double)sz * inv);
  const unsigned long long c2 = 2ull * (unsigned long long)cnt;
  orgb[0] = (uint8_t)((2 * sr + cnt) / c2);
  orgb[1] = (uint8_t)((2 * sg + cnt) / c2);
  orgb[2] = (uint8_t)((2 * sb + cnt) / c2);
}

// ---- occupancy units (dense-rank path) --------------------------------------------------------------
// Occupancy + rank live in ONE array of 16-byte units: words x, y, z = 96 occupancy bits, word w = the
// exclusive rank prefix of the unit (written by the rank pass).  A slot lookup is a single LDG.128.
constexpr int kUnitBits = 96;
constexpr int kUnitsPerThread = 8;
constexpr int kScanThreads = 256;
constexpr int kTileUnits = kScanThreads * kUnitsPerThread;  // units per "scan tile" (32 KB of units)
// Ownership granularity of the multi-GPU form: a "tile" of the C ABI is kOwnUnits consecutive units
// (24,576 cells in key order), fine enough to cut a dense z-layer of the grid into balanced shares.
constexpr int kOwnUnits = kScanThreads;
constexpr int kOwnPerScanTile = kTileUnits / kOwnUnits;
constexpr uint64_t kNoCell = ~0ull;

// Cell of the integer voxel coordinates (kx, ky, kz) inside the grid.
__device__ __forceinline__ uint64_t cell_of_index(const GridDev& g, uint32_t kx, uint32_t ky, uint32_t kz) {
  return (uint64_t)kx + (uint64_t)g.nx * ((uint64_t)ky + (uint64_t)g.ny * (uint64_t)kz);
}
// Cell of the voxel coordinates (fx, fy, fz), kNoCell outside the grid.
__device__ __forceinline__ uint64_t cell_of_coords(const GridDev& g, float fx, float fy, float fz, uint32_t& kx, uint32_t& ky,
                                                   uint32_t& kz) {
  const bool inside = fx >= 0.f && fy >= 0.f && fz >= 0.f && fx < (float)g.nx && fy < (float)g.ny && fz < (float)g.nz;
  if (!inside) return kNoCell;
  kx = (uint32_t)fx;
  ky = (uint32_t)fy;
  kz = (uint32_t)fz;
  return cell_of_index(g, kx, ky, kz);
}
__device__ __forceinline__ uint64_t cell_of_point(const GridDev& g, float rv, float x, float y, float z, uint32_t& kx,
                                                  uint32_t& ky, uint32_t& kz) {
  return cell_of_coords(g, voxel_coord(x, g.ox, g.voxel, rv), voxel_coord(y, g.oy, g.voxel, rv), voxel_coord(z, g.oz, g.voxel, rv),
                        kx, ky, kz);
}

// Sets the occupancy bit of `cell`.  `dirty` (optional): one byte per scan tile, set when a tile receives a
// bit - the rank passes and the clean-up then only touch the tiles a step has actually used.  The flag is
// looked at only when the cell lies in another scan tile than `left` (the cell the caller marked just before,
// kNoCell if none), through the L1-cached path (a stale 0 only costs one redundant store per SM), and written
// only while it still reads 0.  Measured alternatives (cfg 2, on top of a 2.23 ms K4): an uncached (volatile)
// check on every mark +1.0 ms, an unconditional store on every tile change +3.5 ms (same-address stores
// serialise in L2).
__device__ __forceinline__ uint32_t unit_of_cell(uint64_t cell) { return (uint32_t)(cell >> 5) / 3u; }
__device__ __forceinline__ void set_cell_bit(uint32_t* __restrict__ units, uint8_t* __restrict__ dirty, uint64_t cell,
                                             uint64_t left = kNoCell) {
  const uint32_t w32 = (uint32_t)(cell >> 5);  // word index in a plain bitmap
  const uint32_t unit = w32 / 3u;
  atomicOr(units + (size_t)unit * 4 + (w32 - unit * 3u), 1u << (cell & 31));
  if (dirty != nullptr) {
    const uint32_t tile = unit / (uint32_t)kTileUnits;
    if (left == kNoCell || unit_of_cell(left) / (uint32_t)kTileUnits != tile) {
      if (__ldg(dirty + tile) == 0) dirty[tile] = 1;
    }
  }
}

// The device buffers of one fusion session, as the kernels see them (host struct: ddn_fuse_session).
struct FuseDev {
  const GridDev* grid;
  uint32_t* units;
  uint8_t* dirty;                   // may be nullptr
  unsigned long long* counts;       // [0] participating points, [1] voxels
};

// ---- multi-GPU exchange ------------------------------------------------------------------------------
struct PeerPtrs {
  const void* p[DDN_MAX_PEERS];
};

// One warp's step of the owner-side pull: records w0 .. w0 + 31 of this rank's share, which plan (the layout of
// merge_plan_kernel, include/ddn_b200.h) lays out as the concatenation of its slices of every rank's sorted records
// in rotated rank order, are copied from the peers' memory into staging[w0 ...] (DDN_RECORD_WORDS u64 each).  A warp
// inside one rank's slice (the usual case) moves its 1536 bytes as three fully coalesced 512-byte requests (lane l
// takes bytes 16 l of each) and re-distributes them through s_rec (this warp's 96 entries of shared memory).
// Returns the key of record w0 + lane, ~0 past the end of the share (total).
__device__ __forceinline__ unsigned long long pull_share_warp(const PeerPtrs& peer_records, int rank, int R, const long long* __restrict__ plan,
                                                              ulonglong2* __restrict__ staging, long long w0, long long total,
                                                              ulonglong2* s_rec, int lane) {
  const long long i = w0 + lane;
  const bool in = i < total;
  int kq = 0;
#pragma unroll
  for (int k = 1; k < DDN_MAX_PEERS; ++k) kq += (k < R && i >= plan[4 + 2 * DDN_MAX_PEERS + k]) ? 1 : 0;
  const long long j = plan[4 + kq] + (i - plan[4 + 2 * DDN_MAX_PEERS + kq]);
  int q = rank + kq;
  q -= q >= R ? R : 0;
  const unsigned long long* base = reinterpret_cast<const unsigned long long*>(peer_records.p[q]);
  // whole warp inside one rank's share (the usual case): three coalesced 512-byte loads and stores
  const int kq0 = __shfl_sync(0xffffffffu, kq, 0);
  const bool uniform = __all_sync(0xffffffffu, in && kq == kq0);
  unsigned long long key = ~0ull;
  if (uniform) {
    const long long j0 = __shfl_sync(0xffffffffu, j, 0);
    const ulonglong2* src = reinterpret_cast<const ulonglong2*>(base + j0 * DDN_RECORD_WORDS);
    ulonglong2* dst = staging + w0 * 3;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const ulonglong2 v = __ldcv(src + k * 32 + lane);
      s_rec[k * 32 + lane] = v;
      dst[k * 32 + lane] = v;
    }
    __syncwarp();
    key = s_rec[lane * 3].x;
    __syncwarp();
  } else if (in) {
    const ulonglong2* r = reinterpret_cast<const ulonglong2*>(base + j * DDN_RECORD_WORDS);
    const ulonglong2 a = __ldcv(r), b = __ldcv(r + 1), c = __ldcv(r + 2);
    staging[i * 3 + 0] = a, staging[i * 3 + 1] = b, staging[i * 3 + 2] = c;
    key = a.x;
  }
  return key;
}

}  // namespace ddn
