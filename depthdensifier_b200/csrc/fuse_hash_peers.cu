// Stage 4, HASHED PATH on several GPUs: grids too large for the dense occupancy bitmap, fused by R ranks that each
// hold a share of the views.  The same invariants as the dense peer merge (fuse.cu): the rank-ordered concatenation of
// the owners' voxels is the one-GPU result bit for bit, launch sizes come from capacities, counts are read by the
// kernels, and every kernel returns at once when the dense path owns the step (the HashDev's active word, which the
// partial's hash_begin sets from the device grid).
//
// Per rank (ddn_fuse_finish_hashed_partial), on the rank's own points:
//   hash_begin, hash_tomb, hash_insert, hash_compact   unchanged (fuse_hash.cu)
//   hash_sort_records   the radix sort of hash_sort_finalize; instead of finalising, the M voxels are written as
//                       sorted partial RECORDS (DDN_RECORD_WORDS u64: canonical key + the five sums) into the
//                       caller's peer-visible buffer, and S = DDN_HASH_SAMPLES evenly spaced sample keys
//                       (key[floor(i M / S)]) and M into its peer-visible sample array
// At the owner (ddn_fuse_merge_hashed_peers), after a barrier the caller provides:
//   hash_merge_gather   every rank's samples -> local memory, in one bulk pass over NVLink
//   hash_merge_split    R - 1 splitter keys, the same on every rank: splitter b is the smallest key k with
//                       E(k) >= floor(total b / R), where E(k) = sum over ranks q of p_q(#samples of q below k) and
//                       p_q(j) = floor(j M_q / S) is the record index of q's j-th sample (p_q(S) = M_q): an upper bound
//                       of the records below k that is off by less than ceil(M_q / S) per rank
//   hash_merge_cut      where splitters rank and rank + 1 fall in every peer's sorted records: the samples bound
//                       each cut to a window of fewer than ceil(M_q / S) records, whose keys one CTA reads at once
//                       (no chain of dependent remote reads)
//   hash_merge_plan     the cuts in merge_plan_kernel's layout: begin, count, prefix per peer in rotated order
//   hash_pull           this rank's share of every rank's records -> local staging (merge_pull_mark_kernel's loop)
//   hash_merge_insert   the staged records into the rank's (empty) table: the first copy of a key publishes its
//                       staging index, the others add their five sums into that record with RED.ADD
//   hash_compact        unchanged
//   hash_merge_final    the radix sort, then finalisation with the staged records as the accumulator
// DESIGN.md §6 derives the capacity bound of an owner's share.
#include <algorithm>

#include "fuse_hash.cuh"

namespace ddn {

constexpr int kSamples = DDN_HASH_SAMPLES;
constexpr int kSampleWords = kSamples + 1;  // the samples, then M
constexpr int kCutThreads = 256;

// ---- per rank: sorted partial records + samples ---------------------------------------------------------------
struct HashRecords {
  ulonglong2* records;
  long long cap;
  unsigned long long* samples;
  unsigned long long* state;
  const unsigned long long* accum;
  __device__ __forceinline__ void operator()(const GridDev& g, long long m, const unsigned long long* ka, const uint32_t* va,
                                             long long gtid, long long gthreads) const {
    const long long mv = min(m, cap);
    for (long long r = gtid; r < mv; r += gthreads) {
      const unsigned long long* a = accum + (size_t)va[r] * kHashAccWords;
      ulonglong2* o = records + r * 3;
      o[0] = make_ulonglong2(canonical_of_compact(g, ka[r]), a[0]);
      o[1] = make_ulonglong2(a[1], a[2]);
      o[2] = make_ulonglong2(a[3], a[4]);
    }
    if (gtid < kSamples && mv > 0) samples[gtid] = canonical_of_compact(g, ka[(gtid * mv) / kSamples]);
    if (gtid == 0) {
      samples[kSamples] = (unsigned long long)mv;
      if (m > cap) state[kStStatus] = 1ull;  // cannot happen: records <= points <= cap
    }
  }

  __device__ __forceinline__ static uint64_t canonical_of_compact(const GridDev& g, uint64_t ck) {
    const uint64_t mx = (1ull << g.bx) - 1, my = (1ull << g.by) - 1;
    return canonical_key((uint32_t)(ck & mx), (uint32_t)((ck >> g.bx) & my), (uint32_t)(ck >> (g.bx + g.by)));
  }
};

__global__ void __launch_bounds__(kSortThreads, 1)
hash_sort_records_kernel(const GridDev* __restrict__ gp, HashDev h, const long long* __restrict__ counts, ulonglong2* __restrict__ records,
                         long long cap, unsigned long long* __restrict__ samples, const unsigned long long* __restrict__ accum) {
  hash_sort_body(gp, h, counts, HashRecords{records, cap, samples, h.state, accum});
}

// ---- owner side: plan ------------------------------------------------------------------------------------------
// scratch: staging [cap_out records], then local samples [R][kSampleWords], then splitters [DDN_MAX_PEERS + 1] and
// cuts [DDN_MAX_PEERS][2]
struct MergeScratch {
  ulonglong2* staging;
  unsigned long long* local;
  unsigned long long* split;
  long long* cuts;
};

__device__ __forceinline__ long long sample_pos(long long j, long long m) { return j * m / kSamples; }  // p_q(j)

// number of the (non-decreasing) samples s[0, kSamples) below k
__device__ __forceinline__ int samples_below(const unsigned long long* s, unsigned long long k) {
  int lo = 0, hi = kSamples;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (s[mid] < k) lo = mid + 1;
    else hi = mid;
  }
  return lo;
}

__device__ __forceinline__ long long total_records(const unsigned long long* local, int R) {
  long long t = 0;
  for (int q = 0; q < R; ++q) t += (long long)local[q * kSampleWords + kSamples];
  return t;
}

__global__ void __launch_bounds__(256)
hash_merge_gather_kernel(HashDev h, PeerPtrs samples, int R, MergeScratch ms, unsigned long long* __restrict__ counts) {
  if (h.state[kStActive] == 0) return;
  const long long n = (long long)R * kSampleWords;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const long long q = i / kSampleWords;
    ms.local[i] = __ldcv(reinterpret_cast<const unsigned long long*>(samples.p[q]) + (i - q * kSampleWords));
  }
  if (blockIdx.x == 0 && threadIdx.x <= DDN_MAX_PEERS) ms.split[threadIdx.x] = ~0ull;
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    counts[1] = 0ull;         // the merged voxels (hash_compact counts them); counts[0] keeps the rank's own points
    h.state[kStTombs] = 0ull;  // the partial's tombstones are gone from the table
  }
}

// One thread per candidate splitter k = s + 1 (s: any rank's sample); E(k) only changes at such keys.
__global__ void __launch_bounds__(256)
hash_merge_split_kernel(HashDev h, int R, MergeScratch ms) {
  __shared__ unsigned long long s_min[DDN_MAX_PEERS];
  if (h.state[kStActive] == 0) return;
  if (threadIdx.x < DDN_MAX_PEERS) s_min[threadIdx.x] = ~0ull;
  __syncthreads();
  const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int q = (int)(c / kSamples), i = (int)(c - (long long)q * kSamples);
  if (q < R && ms.local[q * kSampleWords + kSamples] > 0) {
    const unsigned long long k = ms.local[q * kSampleWords + i] + 1ull;
    long long e = 0;
    for (int r = 0; r < R; ++r) {
      const unsigned long long* s = ms.local + r * kSampleWords;
      const long long m = (long long)s[kSamples];
      if (m > 0) e += sample_pos(samples_below(s, k), m);
    }
    const long long total = total_records(ms.local, R);
    for (int b = 1; b < R; ++b) {
      const long long t = total * b / R;
      if (t > 0 && e >= t) atomicMin(&s_min[b], k);
    }
  }
  __syncthreads();
  if (threadIdx.x > 0 && threadIdx.x < R && s_min[threadIdx.x] != ~0ull) atomicMin(ms.split + threadIdx.x, s_min[threadIdx.x]);
}

// splitter b: keys [key_b, key_{b+1}) belong to rank b
__device__ __forceinline__ unsigned long long splitter(const MergeScratch& ms, int b, int R, long long total) {
  if (b == 0 || total * b / R == 0) return 0ull;
  return b == R ? ~0ull : ms.split[b];
}

// CTA (k, side): the cut of splitter rank + side in the sorted records of rank q = (rank + k) % R
__global__ void __launch_bounds__(kCutThreads)
hash_merge_cut_kernel(HashDev h, PeerPtrs records, int rank, int R, MergeScratch ms) {
  __shared__ int s_warp[kCutThreads / 32];
  if (h.state[kStActive] == 0) return;
  const int k = blockIdx.x, side = blockIdx.y;
  int q = rank + k;
  q -= q >= R ? R : 0;
  const unsigned long long* s = ms.local + q * kSampleWords;
  const long long m = (long long)s[kSamples];
  const unsigned long long key = splitter(ms, rank + side, R, total_records(ms.local, R));
  const int j = samples_below(s, key);  // m > 0: records [0, p(j - 1)] are below key, records [p(j), m) are not
  long long lo = 0, hi = 0;
  if (m > 0 && j > 0) lo = sample_pos(j - 1, m) + 1, hi = sample_pos(j, m);
  const unsigned long long* rec = reinterpret_cast<const unsigned long long*>(records.p[q]);
  int below = 0;
  for (long long r = lo + threadIdx.x; r < hi; r += kCutThreads) below += __ldcv(rec + r * DDN_RECORD_WORDS) < key ? 1 : 0;
  below = __reduce_add_sync(0xffffffffu, below);
  if ((threadIdx.x & 31) == 0) s_warp[threadIdx.x >> 5] = below;
  __syncthreads();
  if (threadIdx.x == 0) {
    long long cut = lo;
    for (int w = 0; w < kCutThreads / 32; ++w) cut += s_warp[w];
    ms.cuts[k * 2 + side] = m > 0 && j > 0 ? cut : 0;
  }
}

// plan in merge_plan_kernel's layout; [0], [1] = this rank's key range [begin, end) (end ~0 = unbounded), [3] = the
// records of all ranks
__global__ void __launch_bounds__(32)
hash_merge_plan_kernel(HashDev h, int rank, int R, MergeScratch ms, long long cap, long long* __restrict__ plan) {
  if (h.state[kStActive] == 0) return;
  const int lane = threadIdx.x;
  long long begin = 0, count = 0;
  if (lane < R) {
    begin = ms.cuts[lane * 2];
    count = ms.cuts[lane * 2 + 1] - begin;
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
  if (lane == 0) {
    const long long all = total_records(ms.local, R);
    plan[0] = (long long)splitter(ms, rank, R, all);
    plan[1] = (long long)splitter(ms, rank + 1, R, all);
    plan[2] = total;
    plan[3] = all;
    if (total > cap) h.state[kStStatus] = 1ull;  // cannot happen with the capacity of DESIGN.md §6
  }
}

// ---- owner side: pull, merge, finalise -------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
hash_pull_kernel(HashDev h, PeerPtrs peer_records, int rank, int R, const long long* __restrict__ plan, ulonglong2* __restrict__ staging,
                 long long cap) {
  __shared__ ulonglong2 s_rec[8][96];  // per warp: 32 records x 48 bytes
  if (h.state[kStActive] == 0) return;
  const long long total = min(plan[2], cap);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long n_warps = (long long)gridDim.x * 8;
  for (long long w0 = ((long long)blockIdx.x * 8 + warp) * 32; w0 < total; w0 += n_warps * 32)
    pull_share_warp(peer_records, rank, R, plan, staging, w0, total, s_rec[warp], lane);
}

__global__ void __launch_bounds__(256)
hash_merge_insert_kernel(HashDev h, const long long* __restrict__ plan, ulonglong2* __restrict__ staging, long long cap) {
  if (h.state[kStActive] == 0) return;
  const long long total = min(plan[2], cap);
  unsigned long long* words = reinterpret_cast<unsigned long long*>(staging);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const ulonglong2 a = staging[i * 3], b = staging[i * 3 + 1], c = staging[i * 3 + 2];
    const uint32_t idx = hash_voxel_index<DDN_RECORD_WORDS>(h, a.x, (uint32_t)i, words + 1);
    if (idx == kSkipIndex) continue;
    unsigned long long* o = words + (size_t)idx * DDN_RECORD_WORDS + 1;
    atomicAdd(o + 0, a.y);
    atomicAdd(o + 1, b.x);
    atomicAdd(o + 2, b.y);
    atomicAdd(o + 3, c.x);
    atomicAdd(o + 4, c.y);
  }
}

__global__ void __launch_bounds__(kSortThreads, 1)
hash_merge_finalize_kernel(const GridDev* __restrict__ gp, HashDev h, long long* __restrict__ counts, long long cap,
                           uint64_t* __restrict__ out_keys, float* __restrict__ out_xyz, uint8_t* __restrict__ out_rgb,
                           int32_t* __restrict__ out_count, const unsigned long long* __restrict__ staged) {
  hash_sort_body(gp, h, counts, HashFinalize<DDN_RECORD_WORDS>{counts, cap, out_keys, out_xyz, out_rgb, out_count, staged + 1});
}

static int merge_scratch_layout(int32_t n_ranks, int64_t cap_out, void* scratch, int64_t* bytes, MergeScratch* ms) {
  DDN_REQUIRE(n_ranks >= 1 && n_ranks <= DDN_MAX_PEERS && cap_out > 0 && cap_out < (1ll << 31), "n_ranks / cap_out");
  const int64_t o_local = align_up(cap_out * DDN_RECORD_WORDS * 8, 256);
  const int64_t o_split = o_local + align_up((int64_t)n_ranks * kSampleWords * 8, 256);
  const int64_t o_cuts = o_split + 256;
  *bytes = o_cuts + 256;
  if (ms != nullptr) {
    char* p = reinterpret_cast<char*>(scratch);
    ms->staging = reinterpret_cast<ulonglong2*>(p);
    ms->local = reinterpret_cast<unsigned long long*>(p + o_local);
    ms->split = reinterpret_cast<unsigned long long*>(p + o_split);
    ms->cuts = reinterpret_cast<long long*>(p + o_cuts);
  }
  return DDN_OK;
}

static int launch_sort(const void* kernel, void** args, const char* name, cudaStream_t st) {
  DDN_TRY(check_cuda(cudaLaunchCooperativeKernel(kernel, dim3(kSortCtas), dim3(kSortThreads), args, 0, st), name));
  return after_launch(name, st);
}

}  // namespace ddn

extern "C" {

int ddn_fuse_finish_hashed_partial(const ddn_fuse_session* s, const struct ddn_hash_fuse* hf, int32_t mode, int64_t n_points,
                                   int64_t row_len, const float* xyz, const uint8_t* rgb, const uint8_t* votes, int32_t vote_threshold,
                                   const float* dedup_xyz, int64_t n_dedup, uint64_t* records, int64_t cap_records, uint64_t* samples,
                                   void* accum, int64_t accum_bytes, void* stream) {
  using namespace ddn;
  DDN_REQUIRE(s != nullptr && s->grid && s->counts, "session: null buffer");
  HashDev h;
  DDN_TRY(hash_dev(hf, &h));
  DDN_REQUIRE(mode == 0 || mode == 1, "mode must be 0 (TOO_LARGE grids only) or 1 (any grid)");
  DDN_REQUIRE(n_points >= 0 && n_points < (1ll << 31) - 1024, "n_points");
  DDN_REQUIRE(n_dedup >= 0 && (n_dedup == 0 || dedup_xyz != nullptr), "dedup points");
  DDN_REQUIRE(n_points + n_dedup <= hf->cap_voxels, "hash buffers too small: n_points + n_dedup > cap_voxels");
  DDN_REQUIRE(row_len >= 0, "row_len");
  DDN_REQUIRE(cap_records > 0 && cap_records < (1ll << 31), "cap_records");
  DDN_REQUIRE(records != nullptr && (uintptr_t)records % 16 == 0, "records must be 16-byte aligned");
  DDN_REQUIRE(samples != nullptr && (uintptr_t)samples % 8 == 0, "samples must be 8-byte aligned");
  DDN_REQUIRE(accum != nullptr && accum_bytes >= n_points * kHashAccWords * 8 + 16 && (uintptr_t)accum % 16 == 0,
              "accumulator scratch (n_points * 40 bytes)");
  DDN_REQUIRE(n_points == 0 || (xyz && rgb), "null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  GridDev* gp = reinterpret_cast<GridDev*>(s->grid);
  unsigned long long* counts = reinterpret_cast<unsigned long long*>(s->counts);
  unsigned long long* acc = reinterpret_cast<unsigned long long*>(accum);
  DDN_TRY(hash_launch_points(gp, h, counts, mode, n_points, row_len, xyz, rgb, votes, std::min(vote_threshold, 255), dedup_xyz, n_dedup,
                             acc, st));
  const GridDev* gpc = gp;
  const long long* counts_c = reinterpret_cast<const long long*>(s->counts);
  ulonglong2* rec = reinterpret_cast<ulonglong2*>(records);
  const long long cap = (long long)cap_records;
  unsigned long long* smp = reinterpret_cast<unsigned long long*>(samples);
  const unsigned long long* acc_c = acc;
  void* args[] = {(void*)&gpc, (void*)&h, (void*)&counts_c, (void*)&rec, (void*)&cap, (void*)&smp, (void*)&acc_c};
  return launch_sort((const void*)hash_sort_records_kernel, args, "hash_sort_records_kernel", st);
}

int ddn_fuse_merge_hashed_scratch_bytes(int32_t n_ranks, int64_t cap_out, int64_t* bytes_out) {
  using namespace ddn;
  DDN_REQUIRE(bytes_out != nullptr, "null output");
  return merge_scratch_layout(n_ranks, cap_out, nullptr, bytes_out, nullptr);
}

int ddn_fuse_merge_hashed_peers(const ddn_fuse_session* s, const struct ddn_hash_fuse* hf, int32_t rank, int32_t n_ranks,
                                const void* const* peer_records_host, const void* const* peer_samples_host, int64_t* plan, void* scratch,
                                int64_t scratch_bytes, uint64_t* out_keys, float* out_xyz, uint8_t* out_rgb, int32_t* out_count,
                                int64_t cap_out, void* stream) {
  using namespace ddn;
  DDN_REQUIRE(s != nullptr && s->grid && s->counts, "session: null buffer");
  HashDev h;
  DDN_TRY(hash_dev(hf, &h));
  DDN_REQUIRE(n_ranks >= 1 && n_ranks <= DDN_MAX_PEERS && rank >= 0 && rank < n_ranks, "rank / n_ranks");
  DDN_REQUIRE(peer_records_host && peer_samples_host && plan && scratch, "null pointer");
  DDN_REQUIRE(cap_out > 0 && cap_out < (1ll << 31), "cap_out");
  DDN_REQUIRE(cap_out <= hf->cap_voxels, "hash buffers too small: cap_out > cap_voxels");
  DDN_REQUIRE(out_keys && out_xyz && out_rgb && out_count, "null pointer");
  int64_t need = 0;
  MergeScratch ms;
  DDN_TRY(merge_scratch_layout(n_ranks, cap_out, scratch, &need, &ms));
  DDN_REQUIRE(scratch_bytes >= need && (uintptr_t)scratch % 16 == 0, "merge scratch too small (ddn_fuse_merge_hashed_scratch_bytes)");
  PeerPtrs pr, ps;
  for (int q = 0; q < DDN_MAX_PEERS; ++q) {
    pr.p[q] = q < n_ranks ? peer_records_host[q] : nullptr;
    ps.p[q] = q < n_ranks ? peer_samples_host[q] : nullptr;
    if (q < n_ranks) DDN_REQUIRE(pr.p[q] && ps.p[q], "null peer pointer");
  }
  cudaStream_t st = (cudaStream_t)stream;
  const GridDev* gp = reinterpret_cast<const GridDev*>(s->grid);
  unsigned long long* counts = reinterpret_cast<unsigned long long*>(s->counts);
  long long* planll = reinterpret_cast<long long*>(plan);
  const long long cap = (long long)cap_out;
  hash_merge_gather_kernel<<<kNumSMs, 256, 0, st>>>(h, ps, n_ranks, ms, counts);
  DDN_TRY(after_launch("hash_merge_gather_kernel", st));
  hash_merge_split_kernel<<<(unsigned)((n_ranks * kSamples + 255) / 256), 256, 0, st>>>(h, n_ranks, ms);
  DDN_TRY(after_launch("hash_merge_split_kernel", st));
  hash_merge_cut_kernel<<<dim3(n_ranks, 2), kCutThreads, 0, st>>>(h, pr, rank, n_ranks, ms);
  DDN_TRY(after_launch("hash_merge_cut_kernel", st));
  hash_merge_plan_kernel<<<1, 32, 0, st>>>(h, rank, n_ranks, ms, cap, planll);
  DDN_TRY(after_launch("hash_merge_plan_kernel", st));
  hash_pull_kernel<<<kNumSMs * 8, 256, 0, st>>>(h, pr, rank, n_ranks, planll, ms.staging, cap);
  DDN_TRY(after_launch("hash_pull_kernel", st));
  hash_merge_insert_kernel<<<kNumSMs * 8, 256, 0, st>>>(h, planll, ms.staging, cap);
  DDN_TRY(after_launch("hash_merge_insert_kernel", st));
  DDN_TRY(hash_launch_compact(gp, h, cap_out, counts, st));
  long long* counts_ll = reinterpret_cast<long long*>(s->counts);
  const unsigned long long* staged = reinterpret_cast<const unsigned long long*>(ms.staging);
  void* args[] = {(void*)&gp, (void*)&h, (void*)&counts_ll, (void*)&cap, (void*)&out_keys, (void*)&out_xyz, (void*)&out_rgb,
                  (void*)&out_count, (void*)&staged};
  return launch_sort((const void*)hash_merge_finalize_kernel, args, "hash_merge_finalize_kernel", st);
}

}  // extern "C"
