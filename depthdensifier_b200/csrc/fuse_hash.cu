// Stage 4, HASHED PATH: voxel fusion for grids whose bounding box is too large for the dense occupancy bitmap of
// fuse.cu.  Memory is sized by the points of a step, not by the volume of its box, so one distant surface (or one
// outlier depth) no longer makes a step fail.
//
//   hash_begin        decides whether this path owns the step (from the device grid and the mode), rewrites a
//                     TOO_LARGE grid to DDN_GRID_HASHED and zeroes counts
//   hash_tomb         N5: the cells of the sparse cloud go into the table as TOMBSTONES (key | 2^63)
//   hash_insert       one pass over the points, with accumulate_points_kernel's warp aggregation (16 x 2 pixel
//                     tiles, MATCH.ANY, shuffle walk) and arithmetic; the group leader finds or inserts the cell's
//                     canonical key (open addressing, linear probing, atomicCAS).  The first inserter's own point
//                     index becomes the voxel's index (unique, < n, and no shared counter to contend on): it records
//                     its table slot in the slot list at that index; every leader adds the five 64-bit fixed-point
//                     sums with RED.ADD to the accumulator of that index
//   hash_compact      the M used entries of the slot list -> (compact key, voxel index) pairs, M -> counts[1]; the
//                     slot list and the table slots the step used are cleared on the way (the next step finds them
//                     empty, and no step clears the whole table)
//   hash_sort_final   ONE cooperative kernel: LSD radix sort of the M pairs with the element count read from device
//                     memory, then finalisation in key order with finalize_kernel's arithmetic
//
// Every kernel returns at once unless hash_begin let the path run, so a step enqueues the same launches whatever grid
// the device derives, and nothing is read back.  The results are those of the dense path bit for bit: the same cell
// of every point, the same integer sums (order-independent), the same finalisation, keys ascending.
#include <algorithm>
#include <type_traits>

#include "fuse_hash.cuh"

namespace ddn {

__global__ void hash_begin_kernel(GridDev* __restrict__ gp, HashDev h, unsigned long long* __restrict__ counts, int mode) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const int st = gp->status;
  const bool dims = gp->nx > 0 && gp->ny > 0 && gp->nz > 0;
  const bool hashed = st == DDN_GRID_TOO_LARGE || st == DDN_GRID_HASHED;
  const bool run = dims && (mode == 1 ? (st == DDN_GRID_OK || hashed) : hashed);
  h.state[kStActive] = run ? 1ull : 0ull;
  h.state[kStStatus] = 0ull;
  h.state[kStTombs] = 0ull;
  if (!run) return;
  if (st == DDN_GRID_TOO_LARGE) gp->status = DDN_GRID_HASHED;
  counts[0] = 0ull;  // mode 1: K4's mark has already counted the points of an OK grid
  counts[1] = 0ull;
}

// N5: one thread per sparse point.  A point whose cell is tombstoned is not accumulated (hash_insert), as the dense
// path's unmark_points_kernel clears the cell's occupancy bit.
__global__ void __launch_bounds__(256)
hash_tomb_kernel(const GridDev* __restrict__ gp, HashDev h, int64_t n, const float* __restrict__ xyz) {
  if (h.state[kStActive] == 0) return;
  const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (i >= n) return;
  const GridDev g = *gp;
  uint32_t kx, ky, kz;
  const uint64_t cell = cell_of_point(g, 1.0f / g.voxel, __ldg(xyz + i * 3 + 0), __ldg(xyz + i * 3 + 1), __ldg(xyz + i * 3 + 2), kx, ky, kz);
  if (cell == kNoCell) return;
  // the tombstone of the corner cell of a 2^21 x 2^21 x 2^21 grid would be the empty word; a grid derived from a box
  // never holds a point there (one cell of slack on every side)
  const uint64_t key = canonical_key(kx, ky, kz) | kTombBit;
  if (key == kEmptyKey) return;
  uint64_t s = hash_slot(h, key);
  for (long long p = 0; p < h.cap_slots; ++p, s = (s + 1) & (uint64_t)(h.cap_slots - 1)) {
    const unsigned long long prev = atomicCAS(h.keys + s, kEmptyKey, key);
    if (prev == kEmptyKey) {
      const unsigned long long t = atomicAdd(h.state + kStTombs, 1ull);
      h.slots[h.cap_voxels - 1 - (long long)t] = (uint32_t)s;
      return;
    }
    if (prev == key) return;
  }
  h.state[kStStatus] = 1ull;  // table full (cannot happen with ddn_hash_fuse_sizes' sizing)
}

// accumulate_points_kernel (fuse.cu) with the slot lookup replaced by the table, and the participating points counted
// into counts[0] (what K4's fused mark counts on the dense path: points that pass the vote and fall inside the grid).
// The normals form (Normal = const float*, the plain form has no trailing parameter): also the quantised normals, as
// accumulate_points_kernel's normals form, into accumulators of kAccNormalWords words.
template <int kTW, class... Normal>  // tile width in pixels (tile = kTW x 32/kTW); 0 = no row structure, 32 consecutive points
__global__ void __launch_bounds__(256)
hash_insert_kernel(const GridDev* __restrict__ gp, HashDev h, int64_t n, int row_len, const float* __restrict__ xyz,
                   const uint8_t* __restrict__ rgb, const uint8_t* __restrict__ votes, int thr,
                   unsigned long long* __restrict__ counts, unsigned long long* __restrict__ accum, Normal... normal_in) {
  constexpr bool kNormals = sizeof...(Normal) != 0;
  constexpr int kWords = kNormals ? kAccNormalWords : kHashAccWords;
  const float* __restrict__ normal = normal_arg(normal_in...);
  if (h.state[kStActive] == 0) return;
  const GridDev g = *gp;
  const float rv = 1.0f / g.voxel;
  const int lane = threadIdx.x & 31;
  const float fix_scale = voxel_fix_scale(g.voxel);
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
  uint32_t ty = 0, tx = 0;
  struct InBase {
    float x, y, z;
    uint32_t rg, bb, i;
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
    r.i = (uint32_t)i;
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
  int participating = 0;
  // persistent warps (a grid of fixed size, so the launch costs next to nothing on steps the dense path owns): each
  // takes kHashTilesPerWarp consecutive tiles at a time
#pragma unroll 1
  for (uint32_t t_begin = warp * kHashTilesPerWarp; t_begin < n_tiles; t_begin += gridDim.x * 8u * kHashTilesPerWarp) {
  const uint32_t t_end = min(t_begin + (uint32_t)kHashTilesPerWarp, n_tiles);
  if (kTiled) {
    ty = t_begin / tiles_x;
    tx = t_begin - ty * tiles_x;
  }
  In nxt = load_tile(t_begin);
#pragma unroll 1
  for (uint32_t t = t_begin; t < t_end; ++t) {
    const In cur = nxt;
    if (t + 1 < t_end) nxt = load_tile(t + 1);
    uint64_t cell = kNoCell, key = 0;
    int ox = 0, oy = 0, oz = 0;
    const uint32_t rg = cur.rg, bb = cur.bb;
    if (cur.take) {
      uint32_t kx, ky, kz;
      cell = cell_of_point(g, rv, cur.x, cur.y, cur.z, kx, ky, kz);
      if (cell != kNoCell) {
        ox = voxel_offset_fix(cur.x, voxel_centre(g.ox, kx, g.voxel), fix_scale);
        oy = voxel_offset_fix(cur.y, voxel_centre(g.oy, ky, g.voxel), fix_scale);
        oz = voxel_offset_fix(cur.z, voxel_centre(g.oz, kz, g.voxel), fix_scale);
        key = canonical_key(kx, ky, kz);
      }
    }
    const bool valid = cell != kNoCell;
    participating += valid ? 1 : 0;
    uint32_t peers = __match_any_sync(0xffffffffu, cell);
    if (!valid) peers = 0;
    const bool leader = valid && (__ffs(peers) - 1) == lane;
    int sx = 0, sy = 0, sz = 0;
    uint32_t srg = 0, sb = 0;
    int qx = 0, qy = 0, qz = 0, snx = 0, sny = 0, snz = 0;  // kNormals
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
      const int ax = __shfl_sync(0xffffffffu, ox, src), ay = __shfl_sync(0xffffffffu, oy, src);
      const int az = __shfl_sync(0xffffffffu, oz, src);
      const uint32_t arg = __shfl_sync(0xffffffffu, rg, src), ab = __shfl_sync(0xffffffffu, bb, src);
      if (has) sx += ax, sy += ay, sz += az, srg += arg, sb += ab;
      if constexpr (kNormals) {
        const int bx = __shfl_sync(0xffffffffu, qx, src), by = __shfl_sync(0xffffffffu, qy, src), bz = __shfl_sync(0xffffffffu, qz, src);
        if (has) snx += bx, sny += by, snz += bz;
      }
    }
    if (leader) {
      const uint32_t idx = hash_voxel_index<kWords, kWords>(h, key, cur.i, accum);
      if (idx != kSkipIndex) {
        unsigned long long* a = accum + (size_t)idx * kWords;
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
  }
  participating = __reduce_add_sync(0xffffffffu, participating);
  if (lane == 0 && participating) atomicAdd(counts, (unsigned long long)participating);
}

// The used entries of the slot list (voxel indices; unused entries hold kNoIndex) -> (compact key, voxel index) in
// any order (the keys are distinct, so the sort needs no input order), their number -> counts[1] with one atomic per
// CTA.  The step's table slots, slot-list entries and tombstones are cleared on the way.
__global__ void __launch_bounds__(256)
hash_compact_kernel(const GridDev* __restrict__ gp, HashDev h, int64_t n, unsigned long long* __restrict__ counts) {
  __shared__ uint32_t s_warp[8];
  __shared__ unsigned long long s_base;
  if (h.state[kStActive] == 0) return;
  const GridDev g = *gp;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int64_t base = (int64_t)blockIdx.x * 256 * kCompactPerThread; base < n; base += (int64_t)gridDim.x * 256 * kCompactPerThread) {
  uint32_t slot[kCompactPerThread];
  int mine = 0;
#pragma unroll
  for (int j = 0; j < kCompactPerThread; ++j) {
    const int64_t i = base + j * 256 + threadIdx.x;
    slot[j] = i < n ? h.slots[i] : kNoIndex;
    mine += slot[j] != kNoIndex ? 1 : 0;
  }
  uint32_t inc = (uint32_t)mine;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t t = __shfl_up_sync(0xffffffffu, inc, d);
    if (lane >= d) inc += t;
  }
  if (lane == 31) s_warp[warp] = inc;
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t tot = 0;
    for (int w = 0; w < 8; ++w) tot += s_warp[w];
    s_base = tot ? atomicAdd(counts + 1, (unsigned long long)tot) : 0ull;
  }
  __syncthreads();
  uint32_t before = 0;
  for (int w = 0; w < warp; ++w) before += s_warp[w];
  unsigned long long o = s_base + before + inc - (uint32_t)mine;
#pragma unroll
  for (int j = 0; j < kCompactPerThread; ++j) {
    if (slot[j] == kNoIndex) continue;
    const int64_t i = base + j * 256 + threadIdx.x;
    const uint64_t key = h.keys[slot[j]];
    const uint64_t kx = key & 0x1fffff, ky = (key >> 21) & 0x1fffff, kz = (key >> 42) & 0x1fffff;
    if ((long long)o < h.cap_voxels) {
      h.sort_keys[o] = kx | (ky << g.bx) | (kz << (g.bx + g.by));
      h.sort_index[o] = (uint32_t)i;
    }
    ++o;
    h.keys[slot[j]] = kEmptyKey;
    h.index[slot[j]] = kNoIndex;
    h.slots[i] = kNoIndex;
  }
  __syncthreads();  // s_warp and s_base are rewritten by the next chunk
  }
  if (blockIdx.x == 0) {  // tombstones
    const long long tombs = (long long)h.state[kStTombs];
    for (long long j = threadIdx.x; j < tombs; j += 256) {
      uint32_t* e = h.slots + (h.cap_voxels - 1 - j);
      h.keys[*e] = kEmptyKey;
      *e = kNoIndex;
    }
  }
}

// Radix sort + finalise, one cooperative launch of kSortCtas x kSortThreads (hash_sort_body with the finalising
// epilogue).
__global__ void __launch_bounds__(kSortThreads, 1)
hash_sort_finalize_kernel(const GridDev* __restrict__ gp, HashDev h, long long* __restrict__ counts, long long cap,
                          uint64_t* __restrict__ out_keys, float* __restrict__ out_xyz, uint8_t* __restrict__ out_rgb,
                          int32_t* __restrict__ out_count, const unsigned long long* __restrict__ accum) {
  hash_sort_body(gp, h, counts, HashFinalize<kHashAccWords>{counts, cap, out_keys, out_xyz, out_rgb, out_count, accum});
}

__global__ void __launch_bounds__(kSortThreads, 1)
hash_sort_finalize_normals_kernel(const GridDev* __restrict__ gp, HashDev h, long long* __restrict__ counts, long long cap,
                                  uint64_t* __restrict__ out_keys, float* __restrict__ out_xyz, uint8_t* __restrict__ out_rgb,
                                  int32_t* __restrict__ out_count, const unsigned long long* __restrict__ accum, float* __restrict__ out_normal) {
  hash_sort_body(gp, h, counts,
                 HashFinalize<kAccNormalWords, true>{counts, cap, out_keys, out_xyz, out_rgb, out_count, accum, out_normal});
}

// ---- host side ---------------------------------------------------------------------------------
struct HashSizes {
  int64_t cap_slots, table_bytes, slots_bytes, sort_bytes, hist_bytes;
};

static int hash_sizes(int64_t cap_voxels, HashSizes* z) {
  DDN_REQUIRE(cap_voxels > 0 && cap_voxels < (1ll << 31) - 2, "cap_voxels must be in (0, 2^31 - 2)");
  int64_t p = 1;
  while (p < cap_voxels) p <<= 1;
  z->cap_slots = std::max<int64_t>(2 * p, 64);  // voxels + tombstones <= cap_voxels: the table is never more than half full
  z->table_bytes = z->cap_slots * 12;  // u64 keys, then u32 voxel indices
  z->slots_bytes = align_up(cap_voxels * 4, 256);
  z->sort_bytes = align_up(2 * cap_voxels * 8, 256) + align_up(2 * cap_voxels * 4, 256);
  z->hist_bytes = align_up((int64_t)kRadixBins * kSortCtas * 4, 256);
  return DDN_OK;
}

int hash_dev(const ddn_hash_fuse* hf, HashDev* h) {
  DDN_REQUIRE(hf != nullptr, "null hash buffers");
  DDN_REQUIRE(hf->table && hf->slots && hf->sort && hf->hist && hf->state, "hash buffers: null pointer");
  HashSizes z;
  DDN_TRY(hash_sizes(hf->cap_voxels, &z));
  DDN_REQUIRE(hf->cap_slots == z.cap_slots, "hash buffers: cap_slots does not match ddn_hash_fuse_sizes(cap_voxels)");
  DDN_REQUIRE((uintptr_t)hf->table % 16 == 0 && (uintptr_t)hf->sort % 16 == 0 && (uintptr_t)hf->state % 16 == 0,
              "hash buffers: alignment");
  h->keys = reinterpret_cast<unsigned long long*>(hf->table);
  h->index = reinterpret_cast<uint32_t*>(reinterpret_cast<char*>(hf->table) + hf->cap_slots * 8);
  h->slots = hf->slots;
  h->sort_keys = reinterpret_cast<unsigned long long*>(hf->sort);
  h->sort_index = reinterpret_cast<uint32_t*>(reinterpret_cast<char*>(hf->sort) + align_up(2 * hf->cap_voxels * 8, 256));
  h->hist = hf->hist;
  h->state = reinterpret_cast<unsigned long long*>(hf->state);
  h->cap_slots = hf->cap_slots;
  h->cap_voxels = hf->cap_voxels;
  int lg = 0;
  while ((1ll << lg) < hf->cap_slots) ++lg;
  h->shift = 64 - lg;
  return DDN_OK;
}

int hash_launch_compact(const GridDev* gp, const HashDev& h, int64_t n, unsigned long long* counts, cudaStream_t st) {
  const int64_t n_chunks = (std::max<int64_t>(n, 1) + 256 * kCompactPerThread - 1) / (256 * kCompactPerThread);
  hash_compact_kernel<<<(unsigned)std::min<int64_t>(n_chunks, kHashCtas), 256, 0, st>>>(gp, h, n, counts);  // block 0: tombstones
  return after_launch("hash_compact_kernel", st);
}

int hash_launch_points(GridDev* gp, const HashDev& h, unsigned long long* counts, int mode, int64_t n_points, int64_t row_len,
                       const float* xyz, const uint8_t* rgb, const uint8_t* votes, int thr, const float* dedup_xyz, int64_t n_dedup,
                       unsigned long long* acc, cudaStream_t st, const float* normal) {
  hash_begin_kernel<<<1, 32, 0, st>>>(gp, h, counts, mode);
  DDN_TRY(after_launch("hash_begin_kernel", st));
  if (n_dedup > 0) {
    hash_tomb_kernel<<<(unsigned)((n_dedup + 255) / 256), 256, 0, st>>>(gp, h, n_dedup, dedup_xyz);
    DDN_TRY(after_launch("hash_tomb_kernel", st));
  }
  if (n_points > 0) {
    const bool tiled = row_len >= 32 && row_len < (1 << 30);
    const int tw = tiled ? kHashTileW : 0;
    const int th = tw ? 32 / tw : 1, twe = tw ? tw : 32;
    const int64_t n_tiles = tiled ? ((row_len + twe - 1) / twe) * (((n_points + row_len - 1) / row_len + th - 1) / th) : (n_points + 31) / 32;
    const unsigned blocks = (unsigned)std::min<int64_t>((n_tiles + 8 * kHashTilesPerWarp - 1) / (8 * kHashTilesPerWarp), kHashCtas);
    if (normal != nullptr) {
      if (tiled)
        hash_insert_kernel<kHashTileW, const float*><<<blocks, 256, 0, st>>>(gp, h, n_points, (int)row_len, xyz, rgb, votes, thr, counts, acc,
                                                                             normal);
      else
        hash_insert_kernel<0, const float*><<<blocks, 256, 0, st>>>(gp, h, n_points, (int)row_len, xyz, rgb, votes, thr, counts, acc, normal);
      DDN_TRY(after_launch("hash_insert_kernel", st));
    } else {
      if (tiled)
        hash_insert_kernel<kHashTileW><<<blocks, 256, 0, st>>>(gp, h, n_points, (int)row_len, xyz, rgb, votes, thr, counts, acc);
      else
        hash_insert_kernel<0><<<blocks, 256, 0, st>>>(gp, h, n_points, (int)row_len, xyz, rgb, votes, thr, counts, acc);
      DDN_TRY(after_launch("hash_insert_kernel", st));
    }
  }
  return hash_launch_compact(gp, h, n_points, counts, st);
}

}  // namespace ddn

extern "C" {

int ddn_hash_fuse_sizes(int64_t cap_voxels, int64_t* cap_slots, int64_t* table_bytes, int64_t* slots_bytes, int64_t* sort_bytes,
                        int64_t* hist_bytes) {
  using namespace ddn;
  DDN_REQUIRE(cap_slots && table_bytes && slots_bytes && sort_bytes && hist_bytes, "null output");
  HashSizes z;
  DDN_TRY(hash_sizes(cap_voxels, &z));
  *cap_slots = z.cap_slots;
  *table_bytes = z.table_bytes;
  *slots_bytes = z.slots_bytes;
  *sort_bytes = z.sort_bytes;
  *hist_bytes = z.hist_bytes;
  return DDN_OK;
}

int ddn_hash_fuse_reset(const struct ddn_hash_fuse* hf, void* stream) {
  using namespace ddn;
  HashDev h;
  DDN_TRY(hash_dev(hf, &h));
  cudaStream_t st = (cudaStream_t)stream;
  DDN_TRY(check_cuda(cudaMemsetAsync(hf->table, 0xff, (size_t)hf->cap_slots * 12, st), "memset hash table"));
  DDN_TRY(check_cuda(cudaMemsetAsync(hf->slots, 0xff, (size_t)hf->cap_voxels * 4, st), "memset slot list"));
  return check_cuda(cudaMemsetAsync(hf->state, 0, DDN_HASH_STATE_BYTES, st), "memset hash state");
}

}  // extern "C"

namespace ddn {

// ddn_fuse_finish_hashed, and with out_normal its normals form
static int fuse_finish_hashed(const ddn_fuse_session* s, const struct ddn_hash_fuse* hf, int32_t mode, int64_t n_points, int64_t row_len,
                              const float* xyz, const uint8_t* rgb, const uint8_t* votes, int32_t vote_threshold, const float* normal,
                              const float* dedup_xyz, int64_t n_dedup, uint64_t* out_keys, float* out_xyz, uint8_t* out_rgb,
                              int32_t* out_count, float* out_normal, int64_t cap_out, void* accum, int64_t accum_bytes, cudaStream_t st) {
  const bool normals = out_normal != nullptr;
  const int words = normals ? kAccNormalWords : kHashAccWords;
  DDN_REQUIRE(s != nullptr && s->grid && s->counts, "session: null buffer");
  HashDev h;
  DDN_TRY(hash_dev(hf, &h));
  DDN_REQUIRE(mode == 0 || mode == 1, "mode must be 0 (TOO_LARGE grids only) or 1 (any grid)");
  DDN_REQUIRE(n_points >= 0 && n_points < (1ll << 31) - 1024, "n_points");
  DDN_REQUIRE(n_dedup >= 0 && (n_dedup == 0 || dedup_xyz != nullptr), "dedup points");
  DDN_REQUIRE(n_points + n_dedup <= hf->cap_voxels, "hash buffers too small: n_points + n_dedup > cap_voxels");
  DDN_REQUIRE(row_len >= 0, "row_len");
  DDN_REQUIRE(cap_out > 0 && cap_out < (1ll << 31), "cap_out");
  DDN_REQUIRE(out_keys && out_xyz && out_rgb && out_count && accum, "null pointer");
  DDN_REQUIRE(accum_bytes >= std::max(cap_out, n_points) * words * 8 + 16 && (uintptr_t)accum % 16 == 0,
              normals ? "accumulator scratch (max(cap_out, n_points) * 64 bytes)" : "accumulator scratch (max(cap_out, n_points) * 40 bytes)");
  DDN_REQUIRE(n_points == 0 || (xyz && rgb), "null pointer");
  DDN_REQUIRE(!normals || n_points == 0 || normal != nullptr, "null pointer");
  const int thr = std::min(vote_threshold, 255);
  GridDev* gp = reinterpret_cast<GridDev*>(s->grid);
  unsigned long long* counts = reinterpret_cast<unsigned long long*>(s->counts);
  unsigned long long* acc = reinterpret_cast<unsigned long long*>(accum);
  const long long cap = (long long)cap_out;
  DDN_TRY(hash_launch_points(gp, h, counts, mode, n_points, row_len, xyz, rgb, votes, thr, dedup_xyz, n_dedup, acc, st,
                             normals ? normal : nullptr));
  long long* counts_ll = reinterpret_cast<long long*>(s->counts);
  const unsigned long long* acc_c = acc;
  const GridDev* gpc = gp;
  void* args[] = {(void*)&gpc, (void*)&h, (void*)&counts_ll, (void*)&cap, (void*)&out_keys, (void*)&out_xyz, (void*)&out_rgb,
                  (void*)&out_count, (void*)&acc_c, (void*)&out_normal};
  if (normals) {
    DDN_TRY(check_cuda(cudaLaunchCooperativeKernel((const void*)hash_sort_finalize_normals_kernel, dim3(kSortCtas), dim3(kSortThreads), args,
                                                   0, st),
                       "hash_sort_finalize_normals_kernel"));
    return after_launch("hash_sort_finalize_normals_kernel", st);
  }
  DDN_TRY(check_cuda(cudaLaunchCooperativeKernel((const void*)hash_sort_finalize_kernel, dim3(kSortCtas), dim3(kSortThreads), args, 0, st),
                     "hash_sort_finalize_kernel"));
  return after_launch("hash_sort_finalize_kernel", st);
}

}  // namespace ddn

extern "C" {

int ddn_fuse_finish_hashed(const ddn_fuse_session* s, const struct ddn_hash_fuse* hf, int32_t mode, int64_t n_points, int64_t row_len,
                           const float* xyz, const uint8_t* rgb, const uint8_t* votes, int32_t vote_threshold, const float* dedup_xyz,
                           int64_t n_dedup, uint64_t* out_keys, float* out_xyz, uint8_t* out_rgb, int32_t* out_count, int64_t cap_out,
                           void* accum, int64_t accum_bytes, void* stream) {
  return ddn::fuse_finish_hashed(s, hf, mode, n_points, row_len, xyz, rgb, votes, vote_threshold, nullptr, dedup_xyz, n_dedup, out_keys,
                                 out_xyz, out_rgb, out_count, nullptr, cap_out, accum, accum_bytes, (cudaStream_t)stream);
}

int ddn_fuse_finish_hashed_normals(const ddn_fuse_session* s, const struct ddn_hash_fuse* hf, int32_t mode, int64_t n_points,
                                   int64_t row_len, const float* xyz, const uint8_t* rgb, const uint8_t* votes, int32_t vote_threshold,
                                   const float* normal, const float* dedup_xyz, int64_t n_dedup, uint64_t* out_keys, float* out_xyz,
                                   uint8_t* out_rgb, int32_t* out_count, float* out_normal, int64_t cap_out, void* accum,
                                   int64_t accum_bytes, void* stream) {
  DDN_REQUIRE(out_normal != nullptr, "null pointer");
  return ddn::fuse_finish_hashed(s, hf, mode, n_points, row_len, xyz, rgb, votes, vote_threshold, normal, dedup_xyz, n_dedup, out_keys,
                                 out_xyz, out_rgb, out_count, out_normal, cap_out, accum, accum_bytes, (cudaStream_t)stream);
}

}  // extern "C"
