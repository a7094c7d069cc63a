// Ranking, CMC and mAP (Market-1501 protocol) without sorting the distance rows.
//
// Replaces torchreid/metrics/rank.py:103-171 (eval_market1501) and rank_cylib/rank_cy.pyx:156-243.
// The reference argsorts every row (rank.py:117), drops same-pid-same-camera gallery items (:136-140), then walks
// the kept list.  CMC and AP only depend on the POSITIONS of the relevant items among the kept ones,
//     pos(r) = #{ kept g : (d[q,g], g) <lex (d[q,r], r) },
// so one streaming pass over the row, binning every distance against the (few) sorted relevant distances, gives
// the same numbers: bit-exact CMC, fp64 AP, ties broken by gallery index, and integer partial counts that add up
// across gallery shards.  HBM-bound: 4 bytes per (query, gallery) pair, read once.
#include "common.cuh"

namespace ieee {

static constexpr uint64_t kPadKey = ~uint64_t(0);

// ---------------------------------------------------------------------------------------------------------
// CTA-wide bitonic sort of n (power of two) uint64 keys in shared memory, ascending.
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void block_bitonic_sort(uint64_t* s, int n) {
  for (int k = 2; k <= n; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      __syncthreads();
      for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const int p = i ^ j;
        if (p > i) {
          const uint64_t a = s[i], b = s[p];
          const bool up = (i & k) == 0;
          if ((a > b) == up) { s[i] = b; s[p] = a; }
        }
      }
    }
  }
  __syncthreads();
}
__host__ __device__ __forceinline__ int next_pow2(int x) {
  int p = 1;
  while (p < x) p <<= 1;
  return p;
}

// ---------------------------------------------------------------------------------------------------------
// Gallery grouping: an open-addressing hash table pid -> (offset, count) into `members`, the gallery indices
// grouped by identity.  Four small kernels (insert+count, allocate, fill) instead of a sort; once per gallery
// (shard), reused by every query block.  Order inside a group is arbitrary -- the consumers sort what they take.
// ---------------------------------------------------------------------------------------------------------

struct GroupView {
  long long* keys;     // [T]  pid of the slot or kEmptyPid
  int32_t* cnt;        // [T]  members of that pid
  int32_t* fill;       // [T]  fill cursor (== cnt when built)
  int32_t* cursor;     // [1]  allocation cursor (+ padding)
  int32_t* off;        // [T]  first member
  int32_t* slot_of;    // [G]
  int32_t* members;    // [G]  gallery indices grouped by pid
  int64_t T;
  size_t zero_off, zero_bytes, total;
};
static inline GroupView group_view(const void* blob, int64_t G) {
  GroupView v;
  int64_t T = 16;
  while (T < 2 * G) T <<= 1;
  v.T = T;
  uint8_t* b = static_cast<uint8_t*>(const_cast<void*>(blob));
  size_t o = 0;
  auto take = [&](size_t bytes) { size_t r = o; o += align256(bytes); return r; };
  v.keys = reinterpret_cast<long long*>(b + take(size_t(T) * 8));
  v.zero_off = o;
  v.cnt = reinterpret_cast<int32_t*>(b + take(size_t(T) * 4));
  v.fill = reinterpret_cast<int32_t*>(b + take(size_t(T) * 4));
  v.cursor = reinterpret_cast<int32_t*>(b + take(256));
  v.zero_bytes = o - v.zero_off;
  v.off = reinterpret_cast<int32_t*>(b + take(size_t(T) * 4));
  v.slot_of = reinterpret_cast<int32_t*>(b + take(size_t(G) * 4));
  v.members = reinterpret_cast<int32_t*>(b + take(size_t(G) * 4));
  v.total = o;
  return v;
}
size_t gallery_group_bytes(int64_t G) { return group_view(nullptr, G).total; }

__global__ void group_insert_kernel(const int64_t* __restrict__ g_pids, int64_t G, long long* keys, int32_t* cnt,
                                    int32_t* slot_of, int64_t T) {
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= G) return;
  const long long pid = g_pids[g];
  uint32_t h = hash_pid(pid) & (uint32_t)(T - 1);
  while (true) {
    const long long prev = (long long)atomicCAS(reinterpret_cast<unsigned long long*>(keys + h), (unsigned long long)kEmptyPid,
                                                (unsigned long long)pid);
    if (prev == kEmptyPid || prev == pid) break;
    h = (h + 1) & (uint32_t)(T - 1);
  }
  atomicAdd(cnt + h, 1);
  slot_of[g] = (int32_t)h;
}
__global__ void group_alloc_kernel(const int32_t* __restrict__ cnt, int32_t* off, int32_t* cursor, int64_t T) {
  const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s < T && cnt[s] > 0) off[s] = atomicAdd(cursor, cnt[s]);
}
__global__ void group_fill_kernel(const int32_t* __restrict__ slot_of, const int32_t* __restrict__ off, int32_t* fill,
                                  int32_t* members, int64_t G) {
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= G) return;
  const int s = slot_of[g];
  members[off[s] + atomicAdd(fill + s, 1)] = (int32_t)g;
}

int gallery_group(const int64_t* g_pids, int64_t G, void* blob, cudaStream_t stream) {
  IEEE_REQUIRE(g_pids && blob && G > 0 && G < (int64_t(1) << 30), "gallery_group: bad arguments (G=%lld)", (long long)G);
  IEEE_REQUIRE((reinterpret_cast<uintptr_t>(blob) & 255) == 0, "gallery_group: blob must be 256-byte aligned");
  GroupView v = group_view(blob, G);
  IEEE_CUDA_CHECK(cudaMemsetAsync(v.keys, 0x80, size_t(v.T) * 8, stream));
  IEEE_CUDA_CHECK(cudaMemsetAsync(static_cast<uint8_t*>(blob) + v.zero_off, 0, v.zero_bytes, stream));
  const int th = 256;
  group_insert_kernel<<<(unsigned)((G + th - 1) / th), th, 0, stream>>>(g_pids, G, v.keys, v.cnt, v.slot_of, v.T);
  group_alloc_kernel<<<(unsigned)((v.T + th - 1) / th), th, 0, stream>>>(v.cnt, v.off, v.cursor, v.T);
  group_fill_kernel<<<(unsigned)((G + th - 1) / th), th, 0, stream>>>(v.slot_of, v.off, v.fill, v.members, G);
  count_launch(3);
  IEEE_CUDA_CHECK(cudaGetLastError());
  return IEEE_OK;
}

__global__ void list_cap_kernel(const long long* __restrict__ keys, const int32_t* __restrict__ cnt, int64_t T,
                                const int64_t* __restrict__ q_pids, int64_t Q, int32_t* cap_out) {
  const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int32_t n = 0;
  if (q < Q) {
    const int s = group_find(keys, T, q_pids[q]);
    n = s >= 0 ? cnt[s] : 0;
  }
  for (int o = 16; o > 0; o >>= 1) n = max(n, __shfl_xor_sync(0xffffffffu, n, o));
  if ((threadIdx.x & 31) == 0 && n > 0) atomicMax(cap_out, n);
}

int rank_list_cap(const void* group, int64_t G, const int64_t* q_pids, int64_t Q, int32_t* cap_dev, cudaStream_t stream) {
  GroupView v = group_view(group, G);
  IEEE_CUDA_CHECK(cudaMemsetAsync(cap_dev, 0, 4, stream));
  if (Q > 0) {
    list_cap_kernel<<<(unsigned)((Q + 255) / 256), 256, 0, stream>>>(v.keys, v.cnt, v.T, q_pids, Q, cap_dev);
    count_launch();
  }
  IEEE_CUDA_CHECK(cudaGetLastError());
  return IEEE_OK;
}

// ---------------------------------------------------------------------------------------------------------
// gather: one warp per query.  rank.py:136: junk = same pid AND same camera; relevant = same pid, other camera.
// ---------------------------------------------------------------------------------------------------------
// With a peer exchange the CTA's eight list rows are staged in shared memory and then copied, as ONE contiguous chunk
// of 8 * (cap + 1) words, into slot `my` of every rank's list table: per-lane 8-byte stores over NVLink (one 40 - 70 byte
// transaction per query and peer) made the kernel 45 us at N = 8.  `stage` = 0 when the rows do not fit (cap > 255).
__global__ void __launch_bounds__(256) rank_gather_kernel(const float* __restrict__ distmat, int64_t ld, int64_t Q, int64_t G,
                                                           const int64_t* __restrict__ q_pids, const int64_t* __restrict__ q_camids,
                                                           const int64_t* __restrict__ g_camids, const long long* __restrict__ keys,
                                                           const int32_t* __restrict__ gcnt, const int32_t* __restrict__ goff,
                                                           const int32_t* __restrict__ members, int64_t T, int64_t g_offset,
                                                           int32_t cap, uint64_t* __restrict__ rel, int32_t* __restrict__ n_rel,
                                                           uint64_t* __restrict__ junk, int32_t* __restrict__ n_junk,
                                                           int32_t* __restrict__ overflow, const PeerView pv, int stage) {
  extern __shared__ __align__(16) uint64_t g_stage[];          // [8][cap + 1] when staging
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int64_t q0 = (int64_t)blockIdx.x * (blockDim.x >> 5);
  const int64_t q = q0 + w;
  const bool staged = pv.shards != 0 && stage != 0;
  // peer exchange: this shard's list goes into slot `my` of EVERY rank's list table (posted NVLink stores; the count
  // kernel hands over with the phase-A flags), instead of a local list + all-gather
  auto put_rel = [&](int slot, uint64_t v) {
    if (pv.shards == 0) { rel[q * (cap + 1) + slot] = v; return; }
    if (staged) { g_stage[w * (cap + 1) + slot] = v; return; }
    for (int p = 0; p < pv.shards; ++p)
      (reinterpret_cast<uint64_t*>(pv.base[p] + pv.off_rel) + ((int64_t)pv.my * Q + q) * (cap + 1))[slot] = v;
  };
  if (q < Q) {
    const int64_t cam = q_camids[q];
    int lo = 0, n = 0;
    if (lane == 0) {
      const int s = group_find(keys, T, q_pids[q]);
      if (s >= 0) { lo = goff[s]; n = gcnt[s]; }
    }
    lo = __shfl_sync(0xffffffffu, lo, 0);
    n = __shfl_sync(0xffffffffu, n, 0);
    int nr = 0, nj = 0;
    for (int t0 = 0; t0 < n; t0 += 32) {
      const int t = t0 + lane;
      bool is_rel = false, is_junk = false;
      uint64_t key = 0;
      if (t < n) {
        const int32_t gi = members[lo + t];
        key = pack_key(distmat[q * ld + gi], (uint32_t)(gi + g_offset));
        is_junk = g_camids[gi] == cam;
        is_rel = !is_junk;
      }
      const unsigned mr = __ballot_sync(0xffffffffu, is_rel), mj = __ballot_sync(0xffffffffu, is_junk);
      const unsigned below = (1u << lane) - 1;
      if (is_rel) { const int s = nr + __popc(mr & below); if (s < cap) put_rel(s, key); }
      if (is_junk) { const int s = nj + __popc(mj & below); if (s < cap) junk[q * cap + s] = key; }
      nr += __popc(mr);
      nj += __popc(mj);
    }
    if (lane == 0) {
      if (nr > cap || nj > cap) { atomicMax(overflow, max(nr, nj)); nr = min(nr, cap); nj = min(nj, cap); }
      n_rel[q] = nr;
      put_rel(cap, (uint64_t)nr);                   // the list carries its own length: one exchange moves both
      n_junk[q] = nj;
    }
  }
  if (!staged) return;
  __syncthreads();
  // rows q0 .. q0 + 7 are adjacent in every table: one chunk per peer, 8-byte words, consecutive threads -> consecutive
  // words (entries past a list's length are whatever the staging area held: nobody reads them)
  const int64_t left = Q - q0;
  const int rows = left < (int64_t)(blockDim.x >> 5) ? (int)left : (int)(blockDim.x >> 5);
  const int words = rows * (cap + 1);
  for (int p = 0; p < pv.shards; ++p) {
    uint64_t* dst = reinterpret_cast<uint64_t*>(pv.base[p] + pv.off_rel) + ((int64_t)pv.my * Q + q0) * (cap + 1);
    for (int i = threadIdx.x; i < words; i += blockDim.x) dst[i] = g_stage[i];
  }
}

// ---------------------------------------------------------------------------------------------------------
// count: one CTA per query; single streaming pass over the local distance row.
//
// Every distance is binned against the query's sorted thresholds T_0 < ... < T_{R-1} (the relevant items' packed
// (distance key, global index)): b(e) = #{k : T_k <lex e}.  A 1024-cell table over [d(T_0), d(T_{R-1})] maps a
// distance to its bin with one multiply and one shared-memory load; only cells that contain a threshold need
// exact 64-bit compares.  Bin counters are PRIVATE per thread (32-bit, layout [bin][thread]: conflict-free plain
// read-modify-write, no atomics) and are summed once after the stream; queries whose R + 2 bins do not fit the
// private table, or whose thresholds are not finite, fall back to shared atomics / binary search.
// ---------------------------------------------------------------------------------------------------------
constexpr int kCountThreads = 256;
constexpr int kLutCells = 1024;
constexpr int kPrivateBinBudget = 64 * 1024;   // bytes of private counters per CTA ((R + 2) * 1 KB)

struct CountSmemPlan { size_t hist_off, cell_off, misc_off, priv_off, total; int priv_bins; };
__host__ __device__ inline CountSmemPlan count_smem_plan(int Rp) {
  CountSmemPlan p;
  p.hist_off = size_t(Rp) * 8;                          // after T[Rp] u64
  p.cell_off = p.hist_off + size_t(Rp + 2) * 4;         // hist[Rp + 2] i32
  p.misc_off = p.cell_off + size_t(kLutCells + 2) * 4;  // cell[L + 2] u32 (guard cells at both ends)
  p.priv_off = (p.misc_off + 64 * 4 + 15) & ~size_t(15);
  const int want = Rp + 2;
  p.priv_bins = want * kCountThreads * 4 <= kPrivateBinBudget ? want : kPrivateBinBudget / (kCountThreads * 4);
  p.total = p.priv_off + size_t(p.priv_bins) * kCountThreads * 4;
  return p;
}

enum CountMode { COUNT_LUT_PRIVATE = 0, COUNT_LUT_ATOMIC = 1, COUNT_SEARCH_ATOMIC = 2 };

// Table size for a row of G distances: building it costs O(L) per query, so short rows get short tables.
__host__ __device__ inline int lut_cells_for(int G) {
  int L = 64;
  while (L < kLutCells && L * 8 < G) L <<= 1;
  return L;
}

struct CountCtx {
  const uint64_t* T;
  const uint32_t* cell;
  int32_t* hist;
  int32_t* priv;        // this thread's column: priv[b * kCountThreads]
  float lo, hi, scale;
  uint32_t kmax;
  int R, trash;
  int L;                // live cells of the table (power of two <= kLutCells), chosen from the row length
  uint32_t g_offset;
  int ties;
};

// b(e) = lo + #{k in [lo, lo+n) : T_k <lex e}; ties += #{k : key(T_k) == key(e)} unless e is itself a threshold
__device__ __forceinline__ int exact_bin(CountCtx& c, int lo, int n, uint64_t pe) {
  int b = lo, same = 0;
  bool is_thr = false;
  const uint32_t ke = (uint32_t)(pe >> 32);
  for (int j = lo; j < lo + n; ++j) {
    const uint64_t t = c.T[j];
    b += (t < pe);
    same += ((uint32_t)(t >> 32) == ke);
    is_thr |= (t == pe);
  }
  if (!is_thr) c.ties += same;
  return b;
}

// Branch-free per-element body (the lanes of a warp must stay converged over the 16 elements in flight): every
// element increments exactly one counter -- bin 0 if it precedes all thresholds, the trash bin R + 1 if it follows
// them (or is NaN), else its bin from the cell table; only cells that hold a threshold take a (reconverging) branch.
template <int MODE, int NT>
__device__ __forceinline__ void count_bump(CountCtx& c, int b, int delta) {
  if constexpr (MODE == COUNT_LUT_PRIVATE) c.priv[b * NT] += delta;
  else atomicAdd(&c.hist[b], delta);
}

// Cell of a distance in the guarded table (L = c.L live cells): index 0 = "before every threshold" (bin 0), 1 .. L = the L cells over
// [lo, hi], L + 1 = "after every threshold" (trash bin).  floor() sends d < lo below 0 and d >> hi beyond L; fminf
// returns its non-NaN operand, so a NaN distance goes to the trash guard: NaN ranks after every (finite) threshold,
// as in NumPy's sort (the table is only used when all thresholds are finite).
__device__ __forceinline__ uint32_t count_cell(const CountCtx& c, float d) {
  int ci = __float2int_rd(fminf((d - c.lo) * c.scale, (float)c.L));
  ci = max(min(ci, c.L) + 1, 0);
  return c.cell[ci];
}

// Branch-free per-element body (the lanes of a warp stay converged and the 16 elements in flight interleave): every
// element increments exactly one counter, tentatively the FIRST bin of its cell; the return value says whether the
// cell holds thresholds, in which case count_fix() later moves the count to the exact bin.
template <int MODE, int NT>
__device__ __forceinline__ uint32_t count_visit(CountCtx& c, float d) {
  const uint32_t ce = count_cell(c, d);
  count_bump<MODE, NT>(c, (int)(ce & 0xFFFFFu), 1);
  return (ce >> 20) ? 1u : 0u;
}

// Exact (key, index) placement of an element whose cell holds thresholds (rare).  Must stay inlined: a real call
// would force the context struct into local memory and turn every c.lo / c.scale / c.priv access into a local load.
template <int MODE, int NT>
__device__ __forceinline__ void count_fix(CountCtx& c, float d, uint32_t g) {
  const uint32_t ce = count_cell(c, d);
  const int tent = (int)(ce & 0xFFFFFu);
  const int b = exact_bin(c, tent, (int)(ce >> 20), pack_key(d, g + c.g_offset));
  if (b != tent) {
    count_bump<MODE, NT>(c, tent, -1);
    count_bump<MODE, NT>(c, b, 1);
  }
}

// Generic path (non-finite / degenerate thresholds): binary search over all of T, shared atomics.
template <int NT>
__device__ __forceinline__ void count_visit_search(CountCtx& c, float d, uint32_t g) {
  const uint32_t ke = order_key(d);
  const uint64_t pe = (uint64_t(ke) << 32) | (g + c.g_offset);
  int a = 0, e = c.R;
  while (a < e) { const int m = (a + e) >> 1; if (c.T[m] < pe) a = m + 1; else e = m; }
  int same = 0;
  bool is_thr = false;
  for (int j = a; j < c.R && (uint32_t)(c.T[j] >> 32) == ke; ++j) { same++; is_thr |= (c.T[j] == pe); }
  for (int j = a - 1; j >= 0 && (uint32_t)(c.T[j] >> 32) == ke; --j) same++;
  if (!is_thr) c.ties += same;
  atomicAdd(&c.hist[(ke > c.kmax) ? c.trash : a], 1);
}

// NT threads (a CTA or one warp) stream one row; `tid` is the thread's index among them.
template <int MODE, int NT>
__device__ __forceinline__ void count_stream(CountCtx& c, const float* __restrict__ row, int G, int tid) {
  const uintptr_t addr = reinterpret_cast<uintptr_t>(row);
  int head = (int)(((16 - (addr & 15)) & 15) >> 2);
  if (head > G) head = G;
  const int nvec = (G - head) >> 2;
  const float4* rv = reinterpret_cast<const float4*>(row + head);
  if constexpr (MODE == COUNT_SEARCH_ATOMIC) {      // non-finite thresholds only; still keep four loads in flight
    int g = tid;
    for (; g + 3 * NT < G; g += 4 * NT) {
      const float d0 = row[g], d1 = row[g + NT], d2 = row[g + 2 * NT], d3 = row[g + 3 * NT];
      count_visit_search<NT>(c, d0, (uint32_t)g);
      count_visit_search<NT>(c, d1, (uint32_t)(g + NT));
      count_visit_search<NT>(c, d2, (uint32_t)(g + 2 * NT));
      count_visit_search<NT>(c, d3, (uint32_t)(g + 3 * NT));
    }
    for (; g < G; g += NT) count_visit_search<NT>(c, row[g], (uint32_t)g);
    return;
  } else {
    auto one = [&](float d, uint32_t g) { if (count_visit<MODE, NT>(c, d)) count_fix<MODE, NT>(c, d, g); };
    for (int g = tid; g < head; g += NT) one(row[g], (uint32_t)g);
    int i = tid;
    for (; i + 3 * NT < nvec; i += 4 * NT) {   // 4 independent 16-byte loads in flight
      // (a register double-buffer that keeps the next batch in flight was measured slower: occupancy)
      const float4 a0 = __ldcs(rv + i), a1 = __ldcs(rv + i + NT), a2 = __ldcs(rv + i + 2 * NT), a3 = __ldcs(rv + i + 3 * NT);
      uint32_t g0 = (uint32_t)(head + 4 * i);
      one(a0.x, g0); one(a0.y, g0 + 1); one(a0.z, g0 + 2); one(a0.w, g0 + 3);
      g0 += 4 * NT;
      one(a1.x, g0); one(a1.y, g0 + 1); one(a1.z, g0 + 2); one(a1.w, g0 + 3);
      g0 += 4 * NT;
      one(a2.x, g0); one(a2.y, g0 + 1); one(a2.z, g0 + 2); one(a2.w, g0 + 3);
      g0 += 4 * NT;
      one(a3.x, g0); one(a3.y, g0 + 1); one(a3.z, g0 + 2); one(a3.w, g0 + 3);
    }
    for (; i < nvec; i += NT) {
      const float4 a = __ldcs(rv + i);
      const uint32_t g0 = (uint32_t)(head + 4 * i);
      one(a.x, g0); one(a.y, g0 + 1); one(a.z, g0 + 2); one(a.w, g0 + 3);
    }
    for (int g = head + 4 * nvec + tid; g < G; g += NT) one(row[g], (uint32_t)g);
  }
}

// ---------------------------------------------------------------------------------------------------------
// Streaming body of the warp-per-query kernel.  Per element: 4 float ops to the cell index, one 16-bit table load,
// one fire-and-forget shared atomic on the lane's private counter column (no read-modify-write dependency chain
// between the 16 elements in flight), one mask update.  Elements whose cell holds thresholds are fixed up after
// the batch in ONE rolled loop over the mask (the distance is re-read, an L2 hit): the hot loop stays a few hundred
// instructions long instead of sixteen inlined copies of the exact (key, index) comparison.
//
// Cell word (uint16): bit 0 = the cell holds thresholds, bits 1..6 = (number of thresholds in the cell) - 1,
// bits 7..15 = first bin of the cell * 128 = byte offset of that bin's counter row (bin R + 1 = "after every
// threshold": a real row nobody reads, so the body needs no branch).
// ---------------------------------------------------------------------------------------------------------
struct WarpCount {
  const uint64_t* T;
  const uint16_t* cell;
  uint8_t* col;          // this lane's counter column: *(int32_t*)(col + bin * 128)
  const float* row;
  float lo, scale, top;  // cell index = floor(min((d - lo) * scale + 1, top)), top = L + 1
  uint32_t g_offset;
  int ties;
};

__host__ __device__ __forceinline__ uint16_t warp_cell_word(int first_bin, int n) {
  return (uint16_t)((first_bin << 7) | (n ? (((n - 1) << 1) | 1) : 0));
}

// d < lo (and -inf) -> 0 (float->unsigned conversion saturates), [lo, hi] -> 1 .. L, d >> hi, +inf and NaN -> L + 1
// (fminf returns the non-NaN operand: NaN ranks last, like NumPy's sort).  Monotone in d.
__device__ __forceinline__ uint32_t warp_cell_index(float d, float lo, float scale, float top) {
  return __float2uint_rd(fminf(fmaf(d - lo, scale, 1.0f), top));
}

__device__ __forceinline__ void warp_bump(WarpCount& c, uint32_t row_off, int delta) {
  atomicAdd(reinterpret_cast<int32_t*>(c.col + row_off), delta);   // result unused: fire and forget, nothing waits
}

__device__ __forceinline__ void warp_fix(WarpCount& c, float d, uint32_t g) {
  const uint32_t ce = c.cell[warp_cell_index(d, c.lo, c.scale, c.top)];
  if (!(ce & 1u)) return;
  const int tent = (int)(ce >> 7), n = (int)((ce >> 1) & 63u) + 1;
  const uint64_t pe = pack_key(d, g + c.g_offset);
  const uint32_t ke = (uint32_t)(pe >> 32);
  int b = tent, same = 0;
  bool is_thr = false;
#pragma unroll 1                          // rare, divergent code: keep it small (n is 1 nearly always)
  for (int j = tent; j < tent + n; ++j) {
    const uint64_t t = c.T[j];
    b += (t < pe);
    same += ((uint32_t)(t >> 32) == ke);
    is_thr |= (t == pe);
  }
  if (!is_thr) c.ties += same;
  if (b != tent) {
    warp_bump(c, (uint32_t)tent << 7, -1);
    warp_bump(c, (uint32_t)b << 7, 1);
  }
}

// Eight elements at a time in two phases -- all table loads first, then all counter updates -- because the
// compiler may not move a shared load above a shared atomic it cannot prove disjoint.
__device__ __forceinline__ void warp_visit8(WarpCount& c, const float4& u, const float4& v, uint32_t& mask) {
  const float d[8] = {u.x, u.y, u.z, u.w, v.x, v.y, v.z, v.w};
  uint32_t ce[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) ce[e] = c.cell[warp_cell_index(d[e], c.lo, c.scale, c.top)];
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    warp_bump(c, ce[e] & 0xFF80u, 1);
    mask = mask * 2u + (ce[e] & 1u);
  }
}

// `team` warps stream one row together: warp `wq` of the team takes every team-th group of 32 float4.
__device__ __forceinline__ void warp_count_stream(WarpCount& c, int G, int lane, int wq, int team) {
  const float* __restrict__ row = c.row;
  const uintptr_t addr = reinterpret_cast<uintptr_t>(row);
  int head = (int)(((16 - (addr & 15)) & 15) >> 2);
  if (head > G) head = G;
  const int nvec = (G - head) >> 2;
  const float4* rv = reinterpret_cast<const float4*>(row + head);
  const int S = 32 * team, t0 = wq * 32 + lane;
  auto one = [&](int g) {
    const float d = row[g];
    const uint32_t ce = c.cell[warp_cell_index(d, c.lo, c.scale, c.top)];
    warp_bump(c, ce & 0xFF80u, 1);
    if (ce & 1u) warp_fix(c, d, (uint32_t)g);
  };
  for (int g = t0; g < head; g += S) one(g);
  int i = t0;
  // 4 independent 16-byte loads per lane and batch, software-pipelined: the NEXT batch's loads are issued before the
  // current batch is processed (the compiler places them right after the last use of the current values, a third of
  // the way into the body), so a warp's ~200 instructions of binning overlap its own load latency -- with ~23 warps
  // per SM (3368 rows are 0.7 of a wave) there are not enough other warps to hide it.  ncu at the Market shape:
  // 66.3 -> 60.1 us, issue slots 54 -> 64 % busy.  (Batches of 8 loads: same time for one warp per row, 80 registers
  // and slower teams.)  Plain (L1-allocating) loads: the rare exact pass below re-reads a distance from L1.
  bool have = i + 3 * S < nvec;
  float4 a0, a1, a2, a3;
  if (have) { a0 = __ldg(rv + i); a1 = __ldg(rv + i + S); a2 = __ldg(rv + i + 2 * S); a3 = __ldg(rv + i + 3 * S); }
  while (have) {
    const int in = i + 4 * S;
    const bool more = in + 3 * S < nvec;
    float4 n0 = a0, n1 = a1, n2 = a2, n3 = a3;
    if (more) { n0 = __ldg(rv + in); n1 = __ldg(rv + in + S); n2 = __ldg(rv + in + 2 * S); n3 = __ldg(rv + in + 3 * S); }
    uint32_t mask = 0;
    warp_visit8(c, a0, a1, mask);
    warp_visit8(c, a2, a3, mask);
#pragma unroll 1
    while (mask) {                            // rare: bit (15 - e) <-> element e = 4 * (which load) + component
      const int bit = 31 - __clz(mask);
      mask &= ~(1u << bit);
      const int e = 15 - bit;
      const int g = head + 4 * (i + (e >> 2) * S) + (e & 3);
      warp_fix(c, __ldg(row + g), (uint32_t)g);
    }
    a0 = n0; a1 = n1; a2 = n2; a3 = n3;
    i = in;
    have = more;
  }
  for (; i < nvec; i += S) {
    const int g0 = head + 4 * i;
    one(g0); one(g0 + 1); one(g0 + 2); one(g0 + 3);
  }
  for (int g = head + 4 * nvec + t0; g < G; g += S) one(g);
}

// Where the count kernels put a query's row.  Alone: the caller's table.  With a peer exchange: slot `my` of EVERY
// rank's table (posted stores over NVLink), so that each rank can sum the shards' partial counts itself and the
// evaluation needs no third hand-over (an owner stage + result broadcast was one more flag round trip per step).
struct CountRow {
  int32_t* local;
  const PeerView* pv;
  int64_t slot_row;      // (my * Qb + q) * stride
  __device__ __forceinline__ void put(int idx, int32_t v) const {
    if (pv->shards == 0) { local[idx] = v; return; }
    for (int p = 0; p < pv->shards; ++p) reinterpret_cast<int32_t*>(pv->base[p] + pv->off_cnt)[slot_row + idx] = v;
  }
};
__device__ __forceinline__ CountRow count_row(int32_t* counts, int64_t q, int stride, const PeerView& pv) {
  CountRow r;
  r.local = counts ? counts + q * stride : nullptr;
  r.pv = &pv;
  r.slot_row = ((int64_t)pv.my * pv.Qb + q) * stride;
  return r;
}

// ---------------------------------------------------------------------------------------------------------
// count kernel.  WPQ = warps per query:
//   WPQ = 1  eight queries per CTA, one warp each: short rows (G <= 64K), where a CTA-wide setup would cost more
//            than streaming the row; all setup is done with warp-level primitives.
//   WPQ = 8  one query per CTA: long rows (one C4 shard is 125 000 elements).  Warp 0 does the same setup, then
//            all eight warps stream interleaved groups of the row into their own private counter columns.
// Up to kWarpRmax thresholds per query; non-finite threshold distances or more than 64 thresholds in one cell
// take the generic search with shared atomics.  Longer lists go to rank_count_kernel below.
// ---------------------------------------------------------------------------------------------------------
constexpr int kWarpQ = 8;            // warps per CTA
constexpr int kCountTeamDefault = 1;  // warps per query for rows of 4 K .. 64 K columns
constexpr int kWarpRmax = 128;       // thresholds per query the private table holds (cell words address up to 511 bins)
struct WarpMisc { float lo, scale, top; int R, use_lut, ties; uint32_t kmax; int pad; };   // 32 bytes
// T[rmax] u64 | hist[rmax + 2] | cell[1024 + 4] u16 | misc (32 B) | priv[wpq][rmax + 2][32]   (priv 8-byte aligned: it
// doubles as the u64 staging area of the unsorted thresholds)
__host__ __device__ inline int warp_smem_per_query(int rmax, int wpq) {
  return ((rmax * 8 + (rmax + 2) * 4 + (kLutCells + 4) * 2 + 32 + wpq * (rmax + 2) * 32 * 4) + 15) & ~15;
}

template <int WPQ>
__global__ void __launch_bounds__(32 * kWarpQ)
rank_count_warp_kernel(const float* __restrict__ distmat, int64_t ld, int64_t Q, int G, int64_t g_offset, int shards, int cap,
                       int out_cap, int rmax, const uint64_t* __restrict__ rel_all, const int32_t* __restrict__ n_rel,
                       const uint64_t* __restrict__ junk, const int32_t* __restrict__ n_junk, int32_t* __restrict__ counts,
                       unsigned long long* __restrict__ ties_out, const PeerView pv) {
  static_assert(WPQ == 1 || WPQ == 2 || WPQ == 4 || WPQ == kWarpQ, "1, 2, 4 or all 8 warps of the CTA per query");
  if (pv.shards) peer_signal_and_wait(pv, 0);      // every shard's relevant lists have landed in rel_all
  constexpr bool kTeam = WPQ > 1;
  constexpr int kTeams = kWarpQ / WPQ;             // queries per CTA
  extern __shared__ __align__(16) uint8_t ws_raw[];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int team = w / WPQ, wq = w % WPQ;                                             // this warp's team and place in it
  uint8_t* mine = ws_raw + size_t(team) * warp_smem_per_query(rmax, WPQ);
  uint64_t* T = reinterpret_cast<uint64_t*>(mine);                                   // [rmax]
  int32_t* hist = reinterpret_cast<int32_t*>(mine + rmax * 8);                        // [rmax + 2]
  uint16_t* cell = reinterpret_cast<uint16_t*>(hist + rmax + 2);                      // [1024 + 4]
  WarpMisc* misc = reinterpret_cast<WarpMisc*>(cell + kLutCells + 4);
  int32_t* priv = reinterpret_cast<int32_t*>(misc + 1) + size_t(wq) * (rmax + 2) * 32;   // this warp's [rmax + 2][32]
  // a team's warps meet at their own named barrier (ids 1 .. kTeams; 0 is __syncthreads'): teams run independently
  auto team_sync = [&]() {
    if constexpr (WPQ == kWarpQ) __syncthreads();
    else if constexpr (kTeam) asm volatile("bar.sync %0, %1;" ::"r"(team + 1), "r"(32 * WPQ) : "memory");
    else __syncwarp();
  };
  const int64_t q = (int64_t)blockIdx.x * kTeams + team;
  if (q >= Q) return;
  const int stride = out_cap + 2;
  const CountRow out = count_row(counts, q, stride, pv);
  const int nj = n_junk[q];
  // list lengths of all shards in ONE round of loads (lane s reads shard s), then a warp scan: with 8 shards the
  // set-up used to pay 8 dependent trips to L2 per query, and set-up is what a short (sharded) row costs
  int Rtot = 0, my_n = 0, my_base = 0;
  const bool lanes_cover_shards = shards <= 32;
  if (lanes_cover_shards) {
    if (lane < shards) my_n = (int)rel_all[((int64_t)lane * Q + q) * (cap + 1) + cap];
    int incl = my_n;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
    my_base = incl - my_n;
    Rtot = __shfl_sync(0xffffffffu, incl, 31);
  } else {
    for (int s = 0; s < shards; ++s) Rtot += (int)rel_all[((int64_t)s * Q + q) * (cap + 1) + cap];
  }
  if (lane == 0 && wq == 0) {
    out.put(stride - 1, nj); out.put(stride - 2, n_rel[q]);
    // longest merged list seen: sizes the next call's rows (out_cap); a list longer than this call's is flagged by it
    if (ties_out != nullptr && (unsigned long long)Rtot > ties_out[1]) atomicMax(ties_out + 1, (unsigned long long)Rtot);
  }
  if (Rtot == 0 || Rtot > rmax) return;     // invalid query (rank.py:142-144) / row too small: caller re-runs
  const int R = Rtot;
  const int L = lut_cells_for(G);
  if (wq == 0) {                             // ---- setup by the team's first warp --------------------------------
    // thresholds of all shards, staged in this warp's `priv` (not live yet)
    uint64_t* Tin = reinterpret_cast<uint64_t*>(priv);
    if (lanes_cover_shards) {
      // flattened copy: entry idx of the merged list lives in shard s at position idx - base_s; every lane finds its
      // (s, position) with shuffles only and then issues ONE load, so all entries arrive in one round trip
      for (int idx0 = 0; idx0 < R; idx0 += 32) {
        const int idx = idx0 + lane;
        int s_mine = -1, i_mine = 0;
        for (int s = 0; s < shards; ++s) {
          const int b = __shfl_sync(0xffffffffu, my_base, s), n = __shfl_sync(0xffffffffu, my_n, s);
          if (idx >= b && idx < b + n) { s_mine = s; i_mine = idx - b; }
        }
        if (s_mine >= 0) Tin[idx] = rel_all[((int64_t)s_mine * Q + q) * (cap + 1) + i_mine];
      }
    } else {
      int base = 0;
      for (int s = 0; s < shards; ++s) {
        const uint64_t* src = rel_all + ((int64_t)s * Q + q) * (cap + 1);
        const int n = (int)src[cap];
        for (int i = lane; i < n; i += 32) Tin[base + i] = src[i];
        base += n;
      }
    }
    __syncwarp();
    // rank sort (keys are distinct)
    for (int k = lane; k < R; k += 32) {
      const uint64_t me = Tin[k];
      int pos = 0;
      for (int j = 0; j < R; ++j) pos += (Tin[j] < me);
      T[pos] = me;
    }
    __syncwarp();
    const uint32_t kmin = (uint32_t)(T[0] >> 32), kmax = (uint32_t)(T[R - 1] >> 32);
    const float lo = key_to_float(kmin), hi = key_to_float(kmax);
    const float span = hi - lo;
    bool use_lut = (kmax != 0xFFFFFFFFu) && isfinite(lo) && isfinite(hi);
    // (hi - lo) * scale = L - 0.5: every threshold lands in cells 1 .. L and the map stays monotone (the -0.5 margin
    // dwarfs fp32 rounding); everything else falls into the guard cells 0 and L + 1.  Any finite positive scale is
    // CORRECT (cells only pre-sort, occupied cells compare exactly), so a single threshold or a tiny span (scale
    // would overflow) just clamps it: d == lo -> cell 1, anything above -> beyond the table.
    const float scale = use_lut ? fminf(((float)L - 0.5f) / span, 1.2676506e30f /* 2^100 */) : 0.f;
    const float top = (float)(L + 1);
    if (use_lut) {
      // cell of every (sorted) threshold: non-decreasing in k; kept in `hist` (not live yet)
      uint16_t* tcell = reinterpret_cast<uint16_t*>(hist);
      for (int k = lane; k < R; k += 32) {
        const uint32_t ci = warp_cell_index(key_to_float((uint32_t)(T[k] >> 32)), lo, scale, top);
        tcell[k] = (uint16_t)min(max(ci, 1u), (uint32_t)L);
      }
      __syncwarp();
      // Cell words in three warp-wide steps (O(L / 32) per lane, no per-cell search):
      //   1. clear the table; 2. the first threshold of every run of equal cells writes that cell's word
      //   (first bin = its rank k, count = run length; bit 0 marks the cell as occupied); 3. every empty cell
      //   inherits "first bin" = a + n of the nearest occupied cell below it: each lane owns a contiguous chunk of
      //   cells, finds the last occupied one, the warp passes those values upwards, and a second walk fills in.
      uint32_t* cell32 = reinterpret_cast<uint32_t*>(cell);
      for (int i = lane; i < (L + 4) / 2; i += 32) cell32[i] = 0;
      __syncwarp();
      bool crowded = false;                     // a cell word counts at most 64 thresholds
      for (int k = lane; k < R; k += 32) {
        const int cidx = tcell[k];
        if (k == 0 || (int)tcell[k - 1] != cidx) {
          int n = 1;
          while (k + n < R && (int)tcell[k + n] == cidx) ++n;
          crowded |= n > 64;
          cell[cidx] = warp_cell_word(k, min(n, 64));
        }
      }
      __syncwarp();
      const int chunk = (L + 2 + 31) / 32;
      const int c0 = lane * chunk, c1 = min(c0 + chunk, L + 2);
      int last = -1;                            // first bin that follows this lane's last occupied cell
      for (int i = c0; i < c1; ++i) {
        const uint32_t cw = cell[i];
        if (cw & 1u) last = (int)(cw >> 7) + (int)((cw >> 1) & 63u) + 1;
      }
      const uint32_t have = __ballot_sync(0xffffffffu, last >= 0) & ((1u << lane) - 1u);
      const int src = have ? 31 - __clz(have) : lane;
      const int below = __shfl_sync(0xffffffffu, last, src);
      int run = have ? below : 0;
      for (int i = c0; i < c1; ++i) {
        const uint32_t cw = cell[i];
        if (cw & 1u) run = (int)(cw >> 7) + (int)((cw >> 1) & 63u) + 1;
        else cell[i] = (i == L + 1) ? warp_cell_word(R + 1, 0) : warp_cell_word(run, 0);
      }
      if (__any_sync(0xffffffffu, crowded)) use_lut = false;     // (generic search path below)
      __syncwarp();
    }
    for (int i = lane; i < R + 2; i += 32) hist[i] = 0;
    if (lane == 0) {
      misc->lo = lo; misc->scale = scale; misc->top = top; misc->R = R; misc->use_lut = use_lut ? 1 : 0;
      misc->ties = 0; misc->kmax = kmax;
    }
    __syncwarp();
  }
  // every warp clears its own counter columns (warp 0: after the staging above); own column only: i % 32 == lane
  for (int i = lane; i < (R + 2) * 32; i += 32) priv[i] = 0;
  team_sync();
  const float lo = misc->lo, scale = misc->scale, top = misc->top;
  const bool use_lut = misc->use_lut != 0;
  const uint32_t kmax = misc->kmax;
  const float* row = distmat + q * ld;
  int tie_local = 0;
  if (use_lut) {
    WarpCount c;
    c.T = T; c.cell = cell; c.col = reinterpret_cast<uint8_t*>(priv + lane); c.row = row;
    c.lo = lo; c.scale = scale; c.top = top; c.g_offset = (uint32_t)g_offset; c.ties = 0;
    warp_count_stream(c, G, lane, wq, WPQ);
    tie_local = c.ties;
  } else {
    CountCtx c;
    c.T = T; c.cell = nullptr; c.hist = hist; c.priv = priv + lane;
    c.lo = lo; c.hi = 0.f; c.scale = scale; c.kmax = kmax; c.R = R; c.trash = R + 1; c.L = L;
    c.g_offset = (uint32_t)g_offset; c.ties = 0;
    count_stream<COUNT_SEARCH_ATOMIC, 32 * WPQ>(c, row, G, wq * 32 + lane);
    tie_local = c.ties;
  }
  __syncwarp();
  if (use_lut) {   // fold: lane l sums bins l, l + 32, .. over the warp's 32 private columns (rotated reads: conflict-free)
    for (int b = lane; b <= R; b += 32) {
      int sum = 0;
      for (int j = 0; j < 32; ++j) sum += priv[b * 32 + ((j + lane) & 31)];
      if constexpr (kTeam) atomicAdd(&hist[b], sum); else hist[b] = sum;
    }
  }
  if constexpr (kTeam) {
    for (int o = 16; o > 0; o >>= 1) tie_local += __shfl_xor_sync(0xffffffffu, tie_local, o);
    if (lane == 0 && tie_local != 0) atomicAdd(&misc->ties, tie_local);
    tie_local = 0;
  }
  team_sync();
  if (wq != 0) return;
  for (int i = lane; i < nj; i += 32) {      // junk items were streamed too: take them out (rank.py:136-140)
    const uint64_t pe = junk[q * cap + i];
    const uint32_t ke = (uint32_t)(pe >> 32);
    if (ke > kmax) continue;
    int a = 0, e = R;
    while (a < e) { const int m = (a + e) >> 1; if (T[m] < pe) a = m + 1; else e = m; }
    for (int j = a; j < R && (uint32_t)(T[j] >> 32) == ke; ++j) tie_local--;
    for (int j = a - 1; j >= 0 && (uint32_t)(T[j] >> 32) == ke; --j) tie_local--;
    atomicSub(&hist[a], 1);
  }
  for (int o = 16; o > 0; o >>= 1) tie_local += __shfl_xor_sync(0xffffffffu, tie_local, o);
  if constexpr (kTeam) tie_local += misc->ties;
  __syncwarp();
  // counts[k] = sum_{b <= k} hist[b] - [T_k is a local row entry]
  int carry = 0;
  for (int base = 0; base < R; base += 32) {
    const int k = base + lane;
    const int v = k < R ? hist[k] : 0;
    int incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { int n = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += n; }
    if (k < R) {
      const int64_t gi = (int64_t)(uint32_t)T[k] - g_offset;
      out.put(k, carry + incl - ((gi >= 0 && gi < G) ? 1 : 0));
    }
    carry += __shfl_sync(0xffffffffu, incl, 31);
  }
  if (lane == 0 && ties_out != nullptr && tie_local != 0) atomicAdd(ties_out, (unsigned long long)(long long)tie_local);
}

__global__ void __launch_bounds__(kCountThreads, 6)
rank_count_kernel(const float* __restrict__ distmat, int64_t ld, int64_t Q, int G, int64_t g_offset, int shards, int cap,
                  int out_cap, int Rp, const uint64_t* __restrict__ rel_all, const int32_t* __restrict__ n_rel,
                  const uint64_t* __restrict__ junk, const int32_t* __restrict__ n_junk, int32_t* __restrict__ counts,
                  unsigned long long* __restrict__ ties_out, const PeerView pv) {
  extern __shared__ __align__(16) uint8_t cs_raw[];
  if (pv.shards) peer_signal_and_wait(pv, 0);
  const CountSmemPlan plan = count_smem_plan(Rp);
  uint64_t* T = reinterpret_cast<uint64_t*>(cs_raw);
  int32_t* hist = reinterpret_cast<int32_t*>(cs_raw + plan.hist_off);
  uint32_t* cell = reinterpret_cast<uint32_t*>(cs_raw + plan.cell_off);   // first bin of the cell | (#thresholds in it) << 20
  int32_t* misc = reinterpret_cast<int32_t*>(cs_raw + plan.misc_off);    // [0] R, [1] ties (signed), [2..] scan scratch
  int32_t* priv = reinterpret_cast<int32_t*>(cs_raw + plan.priv_off);    // [bins][kCountThreads]
  const int64_t q = blockIdx.x;
  const int tid = threadIdx.x;
  const int stride = out_cap + 2;
  const CountRow out = count_row(counts, q, stride, pv);
  int Rtot = 0;
  for (int s = 0; s < shards; ++s) Rtot += (int)rel_all[((int64_t)s * Q + q) * (cap + 1) + cap];
  if (tid == 0 && ties_out != nullptr && (unsigned long long)Rtot > ties_out[1]) atomicMax(ties_out + 1, (unsigned long long)Rtot);
  if (Rtot > out_cap) {                      // row too small for this query's merged list: flagged above, caller re-runs
    if (tid == 0) { out.put(stride - 1, n_junk[q]); out.put(stride - 2, n_rel[q]); }
    return;
  }

  // ---- thresholds: union of the shards' relevant lists -------------------------------------------------
  if (tid == 0) { misc[0] = 0; misc[1] = 0; }
  for (int i = tid; i < kLutCells + 2; i += kCountThreads) cell[i] = 0;
  __syncthreads();
  // unsorted staging: the (not yet live) private-bin area when it is large enough, else T itself
  const bool stage_in_priv = size_t(Rp) * 8 <= size_t(plan.priv_bins) * kCountThreads * 4;
  uint64_t* Tin = stage_in_priv ? reinterpret_cast<uint64_t*>(priv) : T;
  for (int s = 0; s < shards; ++s) {
    const uint64_t* src = rel_all + ((int64_t)s * Q + q) * (cap + 1);
    const int n = (int)src[cap];
    __shared__ int base_s;
    if (tid == 0) { base_s = misc[0]; misc[0] += n; }
    __syncthreads();
    for (int i = tid; i < n; i += kCountThreads) Tin[base_s + i] = src[i];
    __syncthreads();
  }
  const int R = misc[0];
  const int nj = n_junk[q];
  if (tid == 0) { out.put(stride - 1, nj); out.put(stride - 2, n_rel[q]); }
  if (R == 0) return;   // invalid query (rank.py:142-144): nothing to rank against
  if (stage_in_priv && R <= 512) {
    // rank sort: keys are distinct (distinct gallery indices), so #smaller is each key's final position
    for (int k = tid; k < R; k += kCountThreads) {
      const uint64_t me = Tin[k];
      int pos = 0;
      for (int j = 0; j < R; ++j) pos += (Tin[j] < me);
      T[pos] = me;
    }
  } else {
    const int np = next_pow2(max(R, 2));
    if (stage_in_priv) {
      for (int i = tid; i < np; i += kCountThreads) T[i] = i < R ? Tin[i] : kPadKey;
    } else {
      for (int i = R + tid; i < np; i += kCountThreads) T[i] = kPadKey;
    }
    block_bitonic_sort(T, np);
  }
  __syncthreads();
  for (int i = tid; i < R + 2; i += kCountThreads) hist[i] = 0;
  const bool priv_ok = R + 2 <= plan.priv_bins;
  if (priv_ok)
    for (int i = tid; i < (R + 2) * kCountThreads; i += kCountThreads) priv[i] = 0;

  // ---- cell table over [lo, hi] of the threshold distances ----------------------------------------------
  const uint32_t kmin = (uint32_t)(T[0] >> 32), kmax = (uint32_t)(T[R - 1] >> 32);
  const float lo = key_to_float(kmin), hi = key_to_float(kmax);
  const float span = hi - lo;
  const int L = lut_cells_for(G);
  const bool use_lut = (kmax != 0xFFFFFFFFu) && isfinite(lo) && isfinite(hi) && R < (1 << 11);
  // (hi - lo) * scale = L - 0.5: every in-range distance lands in cells [0, L) and the map stays monotone (the -0.5
  // margin dwarfs fp32 rounding); out-of-range elements fall into the guard cells.  Clamped for a single threshold /
  // tiny span (any finite positive scale is correct: occupied cells compare exactly).
  const float scale = use_lut ? fminf(((float)L - 0.5f) / span, 1.2676506e30f /* 2^100 */) : 0.f;
  if (use_lut) {
    for (int k = tid; k < R; k += kCountThreads) {
      const float d = key_to_float((uint32_t)(T[k] >> 32));
      atomicAdd(&cell[1 + min(__float2int_rd((d - lo) * scale), L - 1)], 1u << 20);
    }
    __syncthreads();
    // exclusive scan of the per-cell counts -> first bin of each cell (kLutCells == 4 * kCountThreads)
    int v[4], sum = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) { v[j] = (int)(cell[1 + tid * 4 + j] >> 20); sum += v[j]; }
    int incl = sum;
    const int lane = tid & 31, w = tid >> 5;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { int n = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += n; }
    int32_t* wsum = misc + 2;
    if (lane == 31) wsum[w] = incl;
    __syncthreads();
    int woff = 0;
    for (int i = 0; i < w; ++i) woff += wsum[i];
    int run = woff + incl - sum;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int idx = 1 + tid * 4 + j;          // cells beyond L are empty; index L + 1 is the trash guard
      cell[idx] = (idx == L + 1) ? (uint32_t)(R + 1) : ((uint32_t)run | ((uint32_t)v[j] << 20));
      run += v[j];
    }
    if (tid == 0) { cell[0] = 0; if (L == kLutCells) cell[L + 1] = (uint32_t)(R + 1); }   // guards: bin 0 / trash bin
  }
  __syncthreads();

  // ---- stream the row ---------------------------------------------------------------------------------------
  CountCtx c;
  c.T = T; c.cell = cell; c.hist = hist; c.priv = priv + tid;
  c.lo = lo; c.hi = hi; c.scale = scale; c.kmax = kmax; c.R = R; c.trash = R + 1; c.L = L;
  c.g_offset = (uint32_t)g_offset; c.ties = 0;
  const float* row = distmat + q * ld;
  if (!use_lut) count_stream<COUNT_SEARCH_ATOMIC, kCountThreads>(c, row, G, tid);
  else if (priv_ok) count_stream<COUNT_LUT_PRIVATE, kCountThreads>(c, row, G, tid);
  else count_stream<COUNT_LUT_ATOMIC, kCountThreads>(c, row, G, tid);
  int tie_local = c.ties;
  __syncthreads();
  if (use_lut && priv_ok) {   // fold the private counters: warp w sums bins w, w + 8, ...
    const int lane = tid & 31, w = tid >> 5;
    for (int b = w; b <= R; b += kCountThreads / 32) {
      int sum = 0;
#pragma unroll
      for (int j = 0; j < kCountThreads / 32; ++j) sum += priv[b * kCountThreads + j * 32 + lane];
      for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
      if (lane == 0) hist[b] = sum;
    }
    __syncthreads();
  }
  // ---- junk items were streamed like everything else: take them out again (rank.py:136-140) -------------
  for (int i = tid; i < nj; i += kCountThreads) {
    const uint64_t pe = junk[q * cap + i];
    const uint32_t ke = (uint32_t)(pe >> 32);
    if (ke > kmax) continue;
    int a = 0, e = R;
    while (a < e) { const int m = (a + e) >> 1; if (T[m] < pe) a = m + 1; else e = m; }
    for (int j = a; j < R && (uint32_t)(T[j] >> 32) == ke; ++j) tie_local--;
    for (int j = a - 1; j >= 0 && (uint32_t)(T[j] >> 32) == ke; --j) tie_local--;
    atomicSub(&hist[a], 1);
  }
  for (int o = 16; o > 0; o >>= 1) tie_local += __shfl_xor_sync(0xffffffffu, tie_local, o);
  if ((tid & 31) == 0 && tie_local) atomicAdd(&misc[1], tie_local);
  __syncthreads();
  // ---- counts[k] = sum_{b <= k} hist[b] - [T_k is a local row entry (it was binned at b == k)] -----------
  __shared__ int carry;
  if (tid == 0) carry = 0;
  __syncthreads();
  for (int base = 0; base < R; base += kCountThreads) {
    const int k = base + tid;
    int v = (k < R) ? hist[k] : 0;
    const int lane = tid & 31, w = tid >> 5;
    int incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { int n = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += n; }
    int32_t* wsum = misc + 2;
    if (lane == 31) wsum[w] = incl;
    __syncthreads();
    int woff = carry;
    for (int i = 0; i < w; ++i) woff += wsum[i];
    if (k < R) {
      const int64_t gi = (int64_t)(uint32_t)T[k] - g_offset;
      out.put(k, woff + incl - ((gi >= 0 && gi < G) ? 1 : 0));
    }
    __syncthreads();
    if (tid == kCountThreads - 1) carry = woff + incl;
    __syncthreads();
  }
  if (tid == 0 && ties_out != nullptr && misc[1] != 0) atomicAdd(ties_out, (unsigned long long)(long long)misc[1]);
}

// rows up to this length use the warp-per-query kernel (ieee_set_debug_flags bit 4: off; tuning override:
// IEEE_B200_COUNT_WARP_MAX_G)
static int count_warp_max_g() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("IEEE_B200_COUNT_WARP_MAX_G");
    v = e ? atoi(e) : 65536;
    if (v < 0) v = 65536;
  }
  return v;
}

// team size for rows of 4 K .. 64 K columns (ieee_set_count_team / IEEE_B200_COUNT_WPQ = 1 | 2 | 4 | 8)
static int g_count_team = -1;
static int count_team_mid() {
  if (g_count_team < 0) {
    const char* e = getenv("IEEE_B200_COUNT_WPQ");
    const int v = e ? atoi(e) : kCountTeamDefault;
    g_count_team = (v == 1 || v == 2 || v == 4 || v == 8) ? v : kCountTeamDefault;
  }
  return g_count_team;
}
int set_count_team(int wpq) {
  const int prev = count_team_mid();
  if (wpq == 1 || wpq == 2 || wpq == 4 || wpq == 8) g_count_team = wpq;
  return prev;
}

size_t rank_count_smem(int shards, int cap) { return count_smem_plan(next_pow2(max(shards * cap, 2))).total; }

int rank_count(const float* distmat, int64_t ld, int64_t Q, int64_t G, int64_t g_offset, int shards, int cap, int out_cap,
               const uint64_t* rel_all, const int32_t* n_rel, const uint64_t* junk, const int32_t* n_junk,
               int32_t* counts, unsigned long long* ties, cudaStream_t stream, const PeerView* peers) {
  const PeerView pv = peers ? *peers : no_peers();
  IEEE_REQUIRE(distmat && rel_all && n_rel && junk && n_junk && (counts || pv.shards), "rank_count: null pointer");
  IEEE_REQUIRE(Q >= 0 && G > 0 && G < (int64_t(1) << 31) && ld >= G && shards >= 1 && cap >= 1 && out_cap >= 0,
               "rank_count: bad shape");
  if (Q == 0) return IEEE_OK;
  if (out_cap == 0 || out_cap > shards * cap) out_cap = shards * cap;       // a merged list cannot be longer than this
  if (out_cap <= kWarpRmax && !(g_debug_flags & 16)) {
    const int rmax = (out_cap + 1) & ~1;           // even: keeps the 8-byte alignment of every query's T
    // warps per query: long rows (a C4 shard) take the whole CTA; Market-sized rows a team of `count_team_mid()` warps
    // -- 3368 one-warp rows are 0.7 of ONE wave on 148 SMs, so every warp's set-up phase coincided and nothing
    // streamed meanwhile; teams make more, shorter rows of work, and set-up overlaps streaming across waves
    const int wpq = G > count_warp_max_g() ? kWarpQ : (G >= 4096 ? count_team_mid() : 1);
    const int teams = kWarpQ / wpq;
    const size_t wsmem = size_t(teams) * warp_smem_per_query(rmax, wpq);
    const unsigned grid = (unsigned)((Q + teams - 1) / teams);
#define IEEE_COUNT_LAUNCH(W)                                                                                                   \
  do {                                                                                                                         \
    IEEE_ENSURE_DYN_SMEM(rank_count_warp_kernel<W>, wsmem);                                                                    \
    rank_count_warp_kernel<W><<<grid, 32 * kWarpQ, wsmem, stream>>>(distmat, ld, Q, (int)G, g_offset, shards, cap, out_cap, rmax, \
                                                                    rel_all, n_rel, junk, n_junk, counts, ties, pv);           \
  } while (0)
    if (wpq == kWarpQ) IEEE_COUNT_LAUNCH(kWarpQ);
    else if (wpq == 4) IEEE_COUNT_LAUNCH(4);
    else if (wpq == 2) IEEE_COUNT_LAUNCH(2);
    else IEEE_COUNT_LAUNCH(1);
#undef IEEE_COUNT_LAUNCH
    count_launch(1, "rank_count_warp_kernel");
    IEEE_CUDA_CHECK(cudaGetLastError());
    return IEEE_OK;
  }
  const int Rp = next_pow2(max(out_cap, 2));
  const size_t smem = count_smem_plan(Rp).total;
  IEEE_REQUIRE(smem <= 200 * 1024, "rank_count: %d relevant items per query exceed the shared-memory budget", out_cap);
  IEEE_ENSURE_DYN_SMEM(rank_count_kernel, smem);
  rank_count_kernel<<<(unsigned)Q, kCountThreads, smem, stream>>>(distmat, ld, Q, (int)G, g_offset, shards, cap, out_cap, Rp, rel_all,
                                                                  n_rel, junk, n_junk, counts, ties, pv);
  count_launch(1, "rank_count_kernel");
  IEEE_CUDA_CHECK(cudaGetLastError());
  return IEEE_OK;
}

int rank_gather(const float* distmat, int64_t ld, int64_t Q, int64_t G, const int64_t* q_pids, const int64_t* q_camids,
                const int64_t* g_camids, const void* group, int64_t g_offset, int32_t cap, uint64_t* rel, int32_t* n_rel,
                uint64_t* junk, int32_t* n_junk, int32_t* overflow, cudaStream_t stream, const PeerView* peers) {
  const PeerView pv = peers ? *peers : no_peers();
  IEEE_REQUIRE(distmat && q_pids && q_camids && g_camids && group && (rel || pv.shards) && n_rel && junk && n_junk && overflow,
               "rank_gather: null pointer");
  IEEE_REQUIRE(Q >= 0 && G > 0 && ld >= G && cap >= 1, "rank_gather: bad shape");
  IEEE_REQUIRE(g_offset >= 0 && g_offset + G <= (int64_t(1) << 32), "rank_gather: global gallery index must fit 32 bits");
  if (Q == 0) return IEEE_OK;
  GroupView v = group_view(group, G);
  const int stage = (pv.shards != 0 && cap <= 255) ? 1 : 0;
  const size_t smem = stage ? size_t(8) * (cap + 1) * 8 : 0;
  rank_gather_kernel<<<(unsigned)((Q + 7) / 8), 256, smem, stream>>>(distmat, ld, Q, G, q_pids, q_camids, g_camids, v.keys, v.cnt,
                                                                     v.off, v.members, v.T, g_offset, cap, rel, n_rel, junk, n_junk,
                                                                     overflow, pv, stage);
  count_launch(1, "rank_gather_kernel");
  IEEE_CUDA_CHECK(cudaGetLastError());
  return IEEE_OK;
}

// ---------------------------------------------------------------------------------------------------------
// finalize: per-query AP / first hit, then one deterministic CTA-wide reduction.
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void query_metrics(const int32_t* __restrict__ counts, int64_t q, int64_t G_total, int stride,
                                              int max_rank, double* ap, int32_t* first, int32_t* is_short, double* inp) {
  const int32_t* c = counts + q * stride;
  const int R = c[stride - 2];            // relevant items over all shards (summed with the counts)
  if (R == 0) {
    ap[q] = 0.0; first[q] = -1; is_short[q] = 0;
    if (inp) inp[q] = 0.0;
    return;
  }
  // inverse negative penalty (README.rst:45, Ye et al. TPAMI 2021): R / (1-based rank of the hardest relevant item)
  if (inp) inp[q] = (double)R / ((double)c[R - 1] + 1.0);
  // rank.py:155-160: AP = (1/R) sum_k (k+1) / (pos_k + 1), float64
  double s = 0.0;
  for (int k = 0; k < R; ++k) s += (double)(k + 1) / ((double)c[k] + 1.0);
  ap[q] = s / (double)R;
  first[q] = c[0];
  const int64_t kept = G_total - (int64_t)c[stride - 1];
  is_short[q] = kept < max_rank ? 1 : 0;
}

__global__ void __launch_bounds__(256) rank_query_kernel(const int32_t* __restrict__ counts,
                                                          int64_t Q, int64_t G_total, int shards, int cap, int max_rank,
                                                          double* __restrict__ ap, int32_t* __restrict__ first,
                                                          int32_t* __restrict__ is_short, double* __restrict__ inp) {
  const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= Q) return;
  query_metrics(counts, q, G_total, shards * cap + 2, max_rank, ap, first, is_short, inp);
}

// The reduction proper, run by ONE CTA of 1024 threads (a kernel of its own, or the last CTA of the metrics kernels).
// No __restrict__ / read-only loads here: the arrays may have been written earlier in the same kernel.
__device__ __forceinline__ void reduce_body(uint8_t* rs_raw, const double* ap, const int32_t* first, const int32_t* is_short,
                                            int64_t Q, int max_rank, const unsigned long long* ties, float* cmc,
                                            ieee_eval_summary* summary, const double* inp, const int32_t* overflow,
                                            const PeerView& pv, long long* stats_out) {
  double* sd = reinterpret_cast<double*>(rs_raw);                 // [1024] AP partial sums
  double* si = sd + 1024;                                         // [1024] INP partial sums
  int32_t* hfirst = reinterpret_cast<int32_t*>(si + 1024);        // [max_rank + 1]
  __shared__ long long s_valid, s_short;
  const int tid = threadIdx.x;
  for (int i = tid; i <= max_rank; i += 1024) hfirst[i] = 0;
  if (tid == 0) { s_valid = 0; s_short = 0; }
  __syncthreads();
  // fixed assignment of queries to threads + fixed tree => the fp64 sum does not depend on scheduling
  double acc = 0.0, acc_inp = 0.0;
  long long nv = 0, ns = 0;
  for (int64_t q = tid; q < Q; q += 1024) {
    const int f = first[q];
    if (f >= 0) {
      acc += ap[q];
      if (inp) acc_inp += inp[q];
      ++nv;
      ns += is_short[q];
      atomicAdd(&hfirst[f < max_rank ? f : max_rank], 1);   // shared int32 atomics: native, cheap
    }
  }
  sd[tid] = acc;
  si[tid] = acc_inp;
  // counts: warp shuffle first, then one shared atomic per warp (1024 threads CAS-looping on one 64-bit shared
  // word cost 40 us here)
  for (int o = 16; o > 0; o >>= 1) {
    nv += __shfl_xor_sync(0xffffffffu, nv, o);
    ns += __shfl_xor_sync(0xffffffffu, ns, o);
  }
  if ((tid & 31) == 0) {
    if (nv) atomicAdd((unsigned long long*)&s_valid, (unsigned long long)nv);
    if (ns) atomicAdd((unsigned long long*)&s_short, (unsigned long long)ns);
  }
  __syncthreads();
  for (int o = 512; o > 0; o >>= 1) {
    if (tid < o) { sd[tid] += sd[tid + o]; si[tid] += si[tid + o]; }
    __syncthreads();
  }
  if (tid == 0) {
    const long long valid = s_valid;
    // rank.py:167-168: float32 sum of {0,1} rows (exact below 2^24) divided by the float count
    int run = 0;
    for (int j = 0; j < max_rank; ++j) {
      run += hfirst[j];
      cmc[j] = valid > 0 ? __fdiv_rn((float)run, (float)valid) : 0.f;
    }
    summary->sum_ap = sd[0];
    summary->mAP = valid > 0 ? sd[0] / (double)valid : 0.0;
    summary->num_valid = valid;
    long long n_ties = ties ? (long long)*ties : 0, over = overflow ? (long long)*overflow : 0;
    if (pv.shards) {   // statistics of all shards (written into this rank's header with the phase-B hand-over)
      const long long* st = reinterpret_cast<const long long*>(pv.base[pv.my] + 512);
      long long longest = 0;
      n_ties = 0; over = 0;
      for (int s = 0; s < pv.shards; ++s) {
        over = max(over, (long long)(int32_t)st[4 * s]);
        n_ties += st[4 * s + 1];
        longest = max(longest, st[4 * s + 2]);
      }
      if (stats_out) { stats_out[0] = over; stats_out[1] = n_ties; stats_out[2] = longest; }
    }
    summary->num_ties = n_ties;
    summary->num_short = s_short;
    summary->max_rank = max_rank;
    summary->status = valid == 0 ? IEEE_ERR_NO_VALID_QUERY : (s_short > 0 ? IEEE_ERR_SHORT_RANK_LIST : IEEE_OK);
    summary->list_overflow = over;
    summary->mINP = (inp && valid > 0) ? si[0] / (double)valid : 0.0;
  }
}

__global__ void __launch_bounds__(1024) rank_reduce_kernel(const double* __restrict__ ap, const int32_t* __restrict__ first,
                                                            const int32_t* __restrict__ is_short, int64_t Q, int max_rank,
                                                            const unsigned long long* __restrict__ ties, float* __restrict__ cmc,
                                                            ieee_eval_summary* __restrict__ summary,
                                                            const double* __restrict__ inp,
                                                            const int32_t* __restrict__ overflow, const PeerView pv,
                                                            long long* __restrict__ stats_out) {
  extern __shared__ __align__(16) uint8_t rs_raw[];
  reduce_body(rs_raw, ap, first, is_short, Q, max_rank, ties, cmc, summary, inp, overflow, pv, stats_out);
}

// True in exactly one CTA of the grid: the one that finishes last.  Its threads then see every other CTA's global
// writes (fence, ticket, fence).  The ticket word must be zero at launch; the last CTA leaves it zero again.
__device__ __forceinline__ bool last_cta_done(uint32_t* ticket) {
  __shared__ int s_last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const uint32_t t = atomicAdd(ticket, 1u);
    s_last = (t == gridDim.x - 1) ? 1 : 0;
    if (s_last) *ticket = 0u;
  }
  __syncthreads();
  if (!s_last) return false;
  __threadfence();
  return true;
}

// rank_query_kernel and rank_reduce_kernel in ONE launch (a launch boundary is 3 - 6 us of a 0.75 ms step): CTAs of
// 1024 threads derive the per-query results, the CTA that finishes last runs the reduction -- the same fixed
// assignment and tree as rank_reduce_kernel, so the sums come out bit-identical to the two-kernel form.
//
// With a peer exchange (pv.shards > 0) the kernel first hands over / waits for the shards' partial counts (phase B;
// this rank's statistics travel with the signal), sums them per query (integers: exact in any order) and reduces
// over all Qtot queries when `reduce_now` says this was the last block.  Every rank does the same arithmetic on the
// same integers, so (cmc, mAP) come out bit-identical everywhere without a result broadcast.
__global__ void __launch_bounds__(1024) rank_metrics_kernel(const int32_t* __restrict__ counts, int64_t Q, int64_t G_total, int stride,
                                                             int max_rank, double* ap, int32_t* first, int32_t* is_short,
                                                             double* inp, const unsigned long long* ties, float* cmc,
                                                             ieee_eval_summary* summary, const int32_t* overflow, uint32_t* ticket,
                                                             const PeerView pv, const unsigned long long* local_stats,
                                                             long long* stats_out, int reduce_now, int64_t Qred) {
  extern __shared__ __align__(16) uint8_t rs_raw[];
  // one WARP per query: lane k owns the k-th relevant item (its summed position and its term of the AP sum -- the
  // division is the expensive part), then every lane adds the terms in k order: the same sequence of fp64 additions
  // as the one-thread-per-query loop of rank_query_kernel, hence the same bits
  const int lane = threadIdx.x & 31;
  const int64_t q = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (pv.shards) peer_signal_and_wait(pv, 1, local_stats);       // every shard's partial counts (and statistics) have landed here
  if (q < Q) {
    const int shards = pv.shards ? pv.shards : 1;
    const int32_t* part = pv.shards ? reinterpret_cast<const int32_t*>(pv.base[pv.my] + pv.off_cnt) + q * stride : counts + q * stride;
    const int64_t shard_stride = (int64_t)pv.Qb * stride;
    int R = 0, nj = 0;
    if (lane < shards) { R = part[lane * shard_stride + stride - 2]; nj = part[lane * shard_stride + stride - 1]; }
    for (int o = 16; o > 0; o >>= 1) { R += __shfl_xor_sync(0xffffffffu, R, o); nj += __shfl_xor_sync(0xffffffffu, nj, o); }
    double a = 0.0, np = 0.0;
    int32_t f = -1, sh = 0;
    const int width = stride - 2;
    if (R > 0 && R <= width) {                        // (R > width: rows too narrow, flagged through the statistics; rerun)
      double acc = 0.0;
      int last_pos = 0;
      for (int base = 0; base < R; base += 32) {
        const int k = base + lane;
        int pos = 0;
        if (k < R)
          for (int s = 0; s < shards; ++s) pos += part[s * shard_stride + k];
        const double term = k < R ? (double)(k + 1) / ((double)pos + 1.0) : 0.0;          // rank.py:155-160
        const int n = min(32, R - base);
        for (int j = 0; j < n; ++j) acc += __shfl_sync(0xffffffffu, term, j);
        if (base == 0) f = __shfl_sync(0xffffffffu, pos, 0);
        last_pos = __shfl_sync(0xffffffffu, pos, n - 1);
      }
      a = acc / (double)R;
      // inverse negative penalty (README.rst:45, Ye et al. TPAMI 2021): R / (1-based rank of the hardest relevant item)
      np = (double)R / ((double)last_pos + 1.0);
      sh = (G_total - (int64_t)nj) < max_rank ? 1 : 0;
    }
    if (lane == 0) {
      const int64_t gq = pv.q_base + q;
      ap[gq] = a; first[gq] = f; is_short[gq] = sh;
      if (inp) inp[gq] = np;
    }
  }
  if (!reduce_now) return;
  if (!last_cta_done(ticket)) return;
  reduce_body(rs_raw, ap, first, is_short, Qred, max_rank, ties, cmc, summary, inp, overflow, pv, stats_out);
}

// Peer exchange, last stage of a query block (see rank_metrics_kernel).  cmc / summary / stats_out are written when
// the block is the last one of the evaluation (q_base + Qb == Qtot).  ap_out / first_out (arrays of Qtot entries, may
// be null) replace the per-query AP / first-hit arrays of the exchange buffer: the results are local to each rank.
int rank_metrics_peer(const PeerView* peers, int64_t G_total, int32_t max_rank, const unsigned long long* local_stats,
                      float* cmc, ieee_eval_summary* summary, long long* stats_out, int64_t Qtot, cudaStream_t stream,
                      double* ap_out, int32_t* first_out) {
  IEEE_REQUIRE(peers && peers->shards >= 1 && local_stats, "rank_metrics_peer: needs a peer exchange");
  IEEE_REQUIRE(max_rank >= 1 && max_rank <= 8192, "rank_metrics_peer: bad shape (max_rank=%d)", max_rank);
  if (max_rank > G_total) max_rank = (int32_t)G_total;
  const PeerView& v = *peers;
  const int last = (v.q_base + v.Qb == Qtot) ? 1 : 0;
  IEEE_REQUIRE(!last || (cmc && summary), "rank_metrics_peer: the last block needs the result buffers");
  uint8_t* mine = v.base[v.my];
  const size_t smem = 2 * 1024 * 8 + size_t(max_rank + 1) * 4;
  IEEE_ENSURE_DYN_SMEM(rank_metrics_kernel, smem);
  rank_metrics_kernel<<<(unsigned)((v.Qb + 31) / 32), 1024, smem, stream>>>(
      nullptr, v.Qb, G_total, v.W + 2, max_rank, ap_out ? ap_out : reinterpret_cast<double*>(mine + v.off_ap),
      first_out ? first_out : reinterpret_cast<int32_t*>(mine + v.off_first), reinterpret_cast<int32_t*>(mine + v.off_short),
      reinterpret_cast<double*>(mine + v.off_inp), nullptr, cmc, summary, nullptr,
      reinterpret_cast<uint32_t*>(mine + kPeerTicketOffset), v, local_stats, stats_out, last, Qtot);
  count_launch(1, "rank_metrics_kernel (peer)");
  IEEE_CUDA_CHECK(cudaGetLastError());
  return IEEE_OK;
}

size_t rank_finalize_workspace_bytes(int64_t Q) { return 2 * align256(size_t(Q) * 8) + 2 * align256(size_t(Q) * 4); }

int rank_query_metrics(const int32_t* counts, int64_t Q, int64_t G_total, int32_t shards, int32_t cap,
                       int32_t max_rank, double* ap, int32_t* first, int32_t* short_list, double* inp,
                       cudaStream_t stream) {
  IEEE_REQUIRE(counts && ap && first && short_list, "rank_query_metrics: null pointer");
  IEEE_REQUIRE(Q > 0 && G_total > 0 && max_rank >= 1 && shards >= 1 && cap >= 1, "rank_query_metrics: bad shape");
  if (max_rank > G_total) max_rank = (int32_t)G_total;   // rank.py:110-115
  rank_query_kernel<<<(unsigned)((Q + 255) / 256), 256, 0, stream>>>(counts, Q, G_total, shards, cap, max_rank, ap,
                                                                     first, short_list, inp); count_launch(1, "rank_query_kernel");
  IEEE_CUDA_CHECK(cudaGetLastError());
  return IEEE_OK;
}

int rank_reduce(const double* ap, const int32_t* first, const int32_t* short_list, int64_t Q, int32_t max_rank,
                const unsigned long long* ties, float* cmc, ieee_eval_summary* summary, const double* inp,
                const int32_t* overflow, cudaStream_t stream, const PeerView* peers, long long* stats_out) {
  const PeerView pv = peers ? *peers : no_peers();
  IEEE_REQUIRE(ap && first && short_list && cmc && summary, "rank_reduce: null pointer");
  IEEE_REQUIRE(Q > 0 && max_rank >= 1 && max_rank <= 8192, "rank_reduce: bad shape (max_rank=%d)", max_rank);
  const size_t smem = 2 * 1024 * 8 + size_t(max_rank + 1) * 4;
  IEEE_ENSURE_DYN_SMEM(rank_reduce_kernel, smem);
  rank_reduce_kernel<<<1, 1024, smem, stream>>>(ap, first, short_list, Q, max_rank, ties, cmc, summary, inp, overflow, pv, stats_out);
  count_launch(1, "rank_reduce_kernel");
  IEEE_CUDA_CHECK(cudaGetLastError());
  return IEEE_OK;
}

int rank_finalize(const int32_t* counts, int64_t Q, int64_t G_total, int32_t shards, int32_t cap,
                  int32_t max_rank, const unsigned long long* ties, float* cmc, ieee_eval_summary* summary,
                  double* per_query_ap, int32_t* per_query_first, void* workspace, cudaStream_t stream,
                  const int32_t* overflow, uint32_t* ticket) {
  IEEE_REQUIRE(workspace != nullptr, "rank_finalize: null workspace");
  if (max_rank > G_total) max_rank = (int32_t)G_total;   // rank.py:110-115
  uint8_t* w = static_cast<uint8_t*>(workspace);
  double* ap = per_query_ap ? per_query_ap : reinterpret_cast<double*>(w);
  int32_t* first = per_query_first ? per_query_first : reinterpret_cast<int32_t*>(w + align256(size_t(Q) * 8));
  int32_t* is_short = reinterpret_cast<int32_t*>(w + align256(size_t(Q) * 8) + align256(size_t(Q) * 4));
  double* inp = reinterpret_cast<double*>(w + align256(size_t(Q) * 8) + 2 * align256(size_t(Q) * 4));
  if (ticket != nullptr) {       // a zeroed word is at hand: both stages in one launch
    IEEE_REQUIRE(counts && cmc && summary, "rank_finalize: null pointer");
    IEEE_REQUIRE(Q > 0 && G_total > 0 && max_rank >= 1 && max_rank <= 8192 && shards >= 1 && cap >= 1, "rank_finalize: bad shape");
    const size_t smem = 2 * 1024 * 8 + size_t(max_rank + 1) * 4;
    IEEE_ENSURE_DYN_SMEM(rank_metrics_kernel, smem);
    rank_metrics_kernel<<<(unsigned)((Q + 31) / 32), 1024, smem, stream>>>(counts, Q, G_total, shards * cap + 2, max_rank, ap, first,
                                                                                is_short, inp, ties, cmc, summary, overflow, ticket,
                                                                                no_peers(), nullptr, nullptr, 1, Q);
    count_launch(1, "rank_metrics_kernel");
    IEEE_CUDA_CHECK(cudaGetLastError());
    return IEEE_OK;
  }
  int rc = rank_query_metrics(counts, Q, G_total, shards, cap, max_rank, ap, first, is_short, inp, stream);
  if (rc) return rc;
  return rank_reduce(ap, first, is_short, Q, max_rank, ties, cmc, summary, inp, overflow, stream, nullptr, nullptr);
}

// ---------------------------------------------------------------------------------------------------------
// float64 distance matrices.  evaluate_py (rank.py:117, the function this fork runs) argsorts the matrix in the dtype
// it arrives in, so two distances that differ below float32 resolution are ORDERED there, while a float32 copy would
// tie them (and break the tie by index).  This path keeps the float64 order: one CTA per query, the relevant items'
// (64-bit distance key, gallery index) thresholds sorted in shared memory, every row entry placed with a binary
// search.  Not a roofline kernel -- the engine never produces float64 distances -- but the same counting form,
// the same tie rule (NaN last, -0 == +0, equal distances by gallery index) and the same finalize stage.
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t order_key64(double d) {
  if (d != d) return ~uint64_t(0);
  d += 0.0;
  const uint64_t b = (uint64_t)__double_as_longlong(d);
  return (b >> 63) ? ~b : (b | (uint64_t(1) << 63));
}
__device__ __forceinline__ bool key96_less(uint64_t ka, uint32_t ia, uint64_t kb, uint32_t ib) {
  return ka < kb || (ka == kb && ia < ib);
}

constexpr int kF64Threads = 256;

__global__ void __launch_bounds__(kF64Threads) rank_count_f64_kernel(
    const double* __restrict__ distmat, int64_t ld, int64_t Q, int G, const int64_t* __restrict__ q_pids,
    const int64_t* __restrict__ q_camids, const int64_t* __restrict__ g_camids, const long long* __restrict__ keys,
    const int32_t* __restrict__ gcnt, const int32_t* __restrict__ goff, const int32_t* __restrict__ members, int64_t T, int cap,
    int32_t* __restrict__ counts, unsigned long long* __restrict__ ties_out, int32_t* __restrict__ overflow) {
  extern __shared__ __align__(16) uint8_t fs_raw[];
  uint64_t* Uk = reinterpret_cast<uint64_t*>(fs_raw);            // [cap] relevant, unsorted
  uint64_t* Sk = Uk + cap;                                        // [cap] relevant, sorted
  uint64_t* Jk = Sk + cap;                                        // [cap] junk
  uint32_t* Ui = reinterpret_cast<uint32_t*>(Jk + cap);           // [cap]
  uint32_t* Si = Ui + cap;
  uint32_t* Ji = Si + cap;
  int32_t* hist = reinterpret_cast<int32_t*>(Ji + cap);           // [cap + 2]
  __shared__ int s_lo, s_n, s_nr, s_nj, s_ties;
  const int64_t q = blockIdx.x;
  const int tid = threadIdx.x;
  const int stride = cap + 2;
  int32_t* out = counts + q * stride;
  if (tid == 0) {
    const int s = group_find(keys, T, q_pids[q]);
    s_lo = s >= 0 ? goff[s] : 0;
    s_n = s >= 0 ? gcnt[s] : 0;
    s_nr = 0; s_nj = 0; s_ties = 0;
  }
  __syncthreads();
  const int n = s_n, lo = s_lo;
  if (n > cap) {
    if (tid == 0) { atomicMax(overflow, n); out[stride - 2] = 0; out[stride - 1] = 0; }
    return;
  }
  const double* row = distmat + q * ld;
  const long long cam = q_camids[q];
  for (int t = tid; t < n; t += kF64Threads) {
    const int gi = members[lo + t];
    const uint64_t k = order_key64(row[gi]);
    if (g_camids[gi] == cam) { const int p = atomicAdd(&s_nj, 1); Jk[p] = k; Ji[p] = (uint32_t)gi; }
    else { const int p = atomicAdd(&s_nr, 1); Uk[p] = k; Ui[p] = (uint32_t)gi; }
  }
  __syncthreads();
  const int R = s_nr, nj = s_nj;
  if (tid == 0) { out[stride - 2] = R; out[stride - 1] = nj; }
  if (R == 0) return;                                            // invalid query (rank.py:142-144)
  for (int t = tid; t < R; t += kF64Threads) {                   // rank sort: (key, index) pairs are distinct
    int pos = 0;
    for (int j = 0; j < R; ++j) pos += key96_less(Uk[j], Ui[j], Uk[t], Ui[t]);
    Sk[pos] = Uk[t];
    Si[pos] = Ui[t];
  }
  for (int b = tid; b <= R; b += kF64Threads) hist[b] = 0;
  __syncthreads();
  auto place = [&](uint64_t k, uint32_t g, int delta) {
    // lb = #{thresholds < (k, g)}; an entry is before threshold t iff t >= lb, or t >= lb + 1 when it IS threshold lb
    int a = 0, e = R;
    while (a < e) { const int m = (a + e) >> 1; if (key96_less(Sk[m], Si[m], k, g)) a = m + 1; else e = m; }
    const bool is_thr = a < R && Sk[a] == k && Si[a] == g;
    atomicAdd(&hist[a + (is_thr ? 1 : 0)], delta);
    if (!is_thr) {                                               // bit-equal distance with a threshold: a tie pair
      int same = 0;
      for (int j = a; j < R && Sk[j] == k; ++j) ++same;
      for (int j = a - 1; j >= 0 && Sk[j] == k; --j) ++same;
      if (same) atomicAdd(&s_ties, delta * same);
    }
  };
  for (int g = tid; g < G; g += kF64Threads) place(order_key64(row[g]), (uint32_t)g, 1);
  __syncthreads();
  for (int t = tid; t < nj; t += kF64Threads) place(Jk[t], Ji[t], -1);   // junk items were streamed too (rank.py:136-140)
  __syncthreads();
  if (tid == 0) {
    int run = 0;
    for (int k = 0; k < R; ++k) { run += hist[k]; out[k] = run; }
    if (ties_out != nullptr && s_ties != 0) atomicAdd(ties_out, (unsigned long long)(long long)s_ties);
  }
}

int rank_count_f64(const double* distmat, int64_t ld, int64_t Q, int64_t G, const int64_t* q_pids, const int64_t* q_camids,
                   const int64_t* g_camids, const void* group, int32_t cap, int32_t* counts, unsigned long long* ties,
                   int32_t* overflow, cudaStream_t stream) {
  IEEE_REQUIRE(distmat && q_pids && q_camids && g_camids && group && counts && overflow, "rank_count_f64: null pointer");
  IEEE_REQUIRE(Q >= 0 && G > 0 && G < (int64_t(1) << 31) && ld >= G && cap >= 1, "rank_count_f64: bad shape");
  IEEE_REQUIRE(cap <= 4096, "rank_count_f64: %d same-identity gallery items per query exceed the float64 path's limit (4096)", cap);
  if (Q == 0) return IEEE_OK;
  GroupView v = group_view(group, G);
  const size_t smem = size_t(cap) * (3 * 8 + 3 * 4) + size_t(cap + 2) * 4;
  IEEE_ENSURE_DYN_SMEM(rank_count_f64_kernel, smem);
  rank_count_f64_kernel<<<(unsigned)Q, kF64Threads, smem, stream>>>(distmat, ld, Q, (int)G, q_pids, q_camids, g_camids, v.keys, v.cnt,
                                                                    v.off, v.members, v.T, cap, counts, ties, overflow);
  count_launch();
  IEEE_CUDA_CHECK(cudaGetLastError());
  return IEEE_OK;
}

// ---------------------------------------------------------------------------------------------------------
// Junk-masked top-k (ranked list): threshold filter into a shared candidate buffer, compacted by bitonic sort.
// ---------------------------------------------------------------------------------------------------------
constexpr int kTopkThreads = 256;
constexpr int kTopkBuf = 2048;   // candidates; compaction keeps k <= kTopkBuf / 2
constexpr int kTopkFastMaxK = 120;

struct TopkArgs {
  const float* row;
  int64_t G, g_offset;
  bool masked;
  int64_t qp, qc;
  const int64_t* g_pids;
  const int64_t* g_camids;
  int k;
};

// General path: threshold filter into the candidate buffer, compacted by a bitonic sort whenever the next tile
// could overflow it.  Any k <= kTopkBuf / 2.  Returns the number of candidates left in cand[] (unsorted).
__device__ int topk_stream_path(const TopkArgs& a, uint64_t* cand, int* count_s, uint64_t* tau_s) {
  const int tid = threadIdx.x;
  if (tid == 0) { *count_s = 0; *tau_s = kPadKey; }
  __syncthreads();
  constexpr int kTile = kTopkThreads * 4;
  for (int64_t g0 = 0; g0 < a.G; g0 += kTile) {
    const uint64_t tau = *tau_s;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int64_t g = g0 + j * kTopkThreads + tid;
      if (g < a.G) {
        const uint64_t pe = pack_key(__ldcs(a.row + g), (uint32_t)(g + a.g_offset));
        if (pe < tau) {
          const bool is_junk = a.masked && a.g_pids[g] == a.qp && a.g_camids[g] == a.qc;   // rank.py:136
          if (!is_junk) cand[atomicAdd(count_s, 1)] = pe;
        }
      }
    }
    __syncthreads();
    const int filled = *count_s;             // snapshot taken between two barriers: every thread sees the same value
    __syncthreads();                         // (without it fast threads would already be appending the next tile)
    if (filled > kTopkBuf - kTile) {         // next tile could overflow: keep the k best, tighten the threshold
      for (int i = filled + tid; i < kTopkBuf; i += kTopkThreads) cand[i] = kPadKey;
      block_bitonic_sort(cand, kTopkBuf);
      if (tid == 0) { *count_s = min(filled, a.k); if (filled >= a.k) *tau_s = cand[a.k - 1]; }
      __syncthreads();
    }
  }
  return *count_s;
}

// ascending bitonic sort of one 64-bit key per lane across a warp (registers + shuffles, no barrier)
__device__ __forceinline__ uint64_t warp_sort_u64(uint64_t v, int lane) {
#pragma unroll
  for (int k = 2; k <= 32; k <<= 1) {
#pragma unroll
    for (int j = k >> 1; j > 0; j >>= 1) {
      const uint64_t o = __shfl_xor_sync(0xffffffffu, v, j);
      const bool keep_min = ((lane & j) == 0) == ((lane & k) == 0);
      v = keep_min ? (v < o ? v : o) : (v > o ? v : o);
    }
  }
  return v;
}

// Fast path (k <= kTopkFastMaxK): every thread keeps the leader of its strided share of the row (smallest distance,
// lowest index among equals); the m-th smallest of those 256 leaders is >= the m-th smallest element of the row, so
// with m = 2k + 8 (head-room for junk entries) it bounds the k-th smallest kept element unless more than k + 8 of
// the leaders are junk.  A second pass over the (L2-resident) row collects the few elements below that bound.
// Both passes read 16-byte vectors and decide with plain float compares -- a thread walks its share in increasing
// index order, so `d < best` keeps the earliest of equal distances (-0 == +0 as in the key order), NaN never leads
// (it ranks last) -- and only leaders / candidates get a packed 64-bit key: the round-1 version built a key per
// element in both passes (93 M warp instructions for 54 M elements).  Returns the candidate count, or -1 when the
// bound left fewer than k kept candidates / overflowed (the caller then takes the general path).
__device__ int topk_select_path(const TopkArgs& a, uint64_t* cand, int* count_s) {
  const int tid = threadIdx.x;
  const float* __restrict__ row = a.row;
  const int G = (int)a.G;
  const uintptr_t addr = reinterpret_cast<uintptr_t>(row);
  int head = (int)(((16 - (addr & 15)) & 15) >> 2);
  if (head > G) head = G;
  const int nvec = (G - head) >> 2;
  const float4* rv = reinterpret_cast<const float4*>(row + head);
  float bd = __int_as_float(0x7f800000);
  int bg = -1;
  auto lead = [&](float d, int g) { if (d < bd) { bd = d; bg = g; } };
  for (int g = tid; g < head; g += kTopkThreads) lead(row[g], g);
  int i = tid;
  for (; i + 3 * kTopkThreads < nvec; i += 4 * kTopkThreads) {          // four independent 16-byte loads in flight
    const float4 v0 = __ldg(rv + i), v1 = __ldg(rv + i + kTopkThreads), v2 = __ldg(rv + i + 2 * kTopkThreads),
                 v3 = __ldg(rv + i + 3 * kTopkThreads);
    int g = head + 4 * i;
    lead(v0.x, g); lead(v0.y, g + 1); lead(v0.z, g + 2); lead(v0.w, g + 3);
    g += 4 * kTopkThreads;
    lead(v1.x, g); lead(v1.y, g + 1); lead(v1.z, g + 2); lead(v1.w, g + 3);
    g += 4 * kTopkThreads;
    lead(v2.x, g); lead(v2.y, g + 1); lead(v2.z, g + 2); lead(v2.w, g + 3);
    g += 4 * kTopkThreads;
    lead(v3.x, g); lead(v3.y, g + 1); lead(v3.z, g + 2); lead(v3.w, g + 3);
  }
  for (; i < nvec; i += kTopkThreads) {
    const float4 v = __ldg(rv + i);
    const int g = head + 4 * i;
    lead(v.x, g); lead(v.y, g + 1); lead(v.z, g + 2); lead(v.w, g + 3);
  }
  for (int g = head + 4 * nvec + tid; g < G; g += kTopkThreads) lead(row[g], g);
  // (a share that holds nothing below +inf has no leader: a pad key, which can only raise the bound)
  // the m-th smallest leader, without sorting all 256 in shared memory (36 barrier-separated stages were a third of
  // the kernel's instructions): every warp sorts its 32 leaders in registers, the eight sorted runs go to shared
  // memory, and each thread ranks its own leader by binary search in the seven other runs.  Real leaders are distinct
  // (distinct gallery indices), so exactly one thread finds rank m -- unless fewer than m + 1 shares have a leader.
  const int lane = tid & 31, w = tid >> 5;
  const uint64_t mine = warp_sort_u64(bg >= 0 ? pack_key(bd, (uint32_t)(bg + a.g_offset)) : kPadKey, lane);
  __shared__ uint64_t tau_sel;
  cand[tid] = mine;
  if (tid == 0) { *count_s = 0; tau_sel = kPadKey; }
  __syncthreads();
  const int m = min(2 * a.k + 8, kTopkThreads) - 1;
  if (mine != kPadKey) {
    int rank = lane;
    for (int r = 0; r < kTopkThreads / 32; ++r) {
      if (r == w) continue;
      const uint64_t* run = cand + r * 32;
      int lo = 0;
#pragma unroll
      for (int step = 16; step > 0; step >>= 1)
        if (run[lo + step - 1] < mine) lo += step;
      lo += run[lo] < mine ? 1 : 0;             // (lo <= 31 here)
      rank += lo;
    }
    if (rank == m) tau_sel = mine;
  }
  __syncthreads();
  const uint64_t tau = tau_sel;
  __syncthreads();                           // (cand is reused below)
  if (tau == kPadKey) return -1;             // fewer than m+1 leaders (tiny rows, rows of inf / NaN): general path
  const float tau_d = key_to_float((uint32_t)(tau >> 32));
  auto collect = [&](float d, int g) {
    if (!(d > tau_d)) {                      // cheap float pre-filter (NaN passes and is decided by the key compare)
      const uint64_t pe = pack_key(d, (uint32_t)(g + a.g_offset));
      if (pe <= tau) {
        const bool is_junk = a.masked && a.g_pids[g] == a.qp && a.g_camids[g] == a.qc;
        if (!is_junk) {
          const int pos = atomicAdd(count_s, 1);
          if (pos < kTopkBuf) cand[pos] = pe;
        }
      }
    }
  };
  for (int g = tid; g < head; g += kTopkThreads) collect(row[g], g);
  for (i = tid; i < nvec; i += kTopkThreads) {
    const float4 v = __ldg(rv + i);
    const int g = head + 4 * i;
    collect(v.x, g); collect(v.y, g + 1); collect(v.z, g + 2); collect(v.w, g + 3);
  }
  for (int g = head + 4 * nvec + tid; g < G; g += kTopkThreads) collect(row[g], g);
  __syncthreads();
  const int n = *count_s;
  __syncthreads();
  if (n > kTopkBuf) return -1;
  // every kept element below the bound was collected; fewer than k of them means the bound was spent on junk
  // (or the row has fewer than k kept entries in total, which only the general path can tell)
  if (n < a.k) return -1;
  return n;
}

__global__ void __launch_bounds__(kTopkThreads)
topk_kernel(const float* __restrict__ distmat, int64_t ld, int64_t Q, int64_t G, int64_t g_offset,
            const int64_t* __restrict__ q_pids, const int64_t* __restrict__ q_camids, const int64_t* __restrict__ g_pids,
            const int64_t* __restrict__ g_camids, int k, int32_t* __restrict__ idx_out, float* __restrict__ val_out) {
  __shared__ uint64_t cand[kTopkBuf];
  __shared__ int count;
  __shared__ uint64_t tau_s;
  const int64_t q = blockIdx.x;
  const int tid = threadIdx.x;
  TopkArgs a;
  a.row = distmat + q * ld;
  a.G = G;
  a.g_offset = g_offset;
  a.masked = q_pids != nullptr;
  a.qp = a.masked ? q_pids[q] : 0;
  a.qc = a.masked ? q_camids[q] : 0;
  a.g_pids = g_pids;
  a.g_camids = g_camids;
  a.k = k;
  int n = -1;
  if (k <= kTopkFastMaxK && G >= 4 * kTopkThreads) n = topk_select_path(a, cand, &count);
  if (n < 0) {
    __syncthreads();
    n = topk_stream_path(a, cand, &count, &tau_s);
  }
  const uint64_t* sorted = cand;
  if (n <= 128) {
    // few candidates (the usual case: about 2k + 8): every candidate's position is the number of smaller ones
    // (distinct keys) -- one pass of broadcast loads for the first n threads instead of a barrier-separated sort
    __syncthreads();
    if (tid < n) {
      const uint64_t v = cand[tid];
      int pos = 0;
      for (int j = 0; j < n; ++j) pos += cand[j] < v ? 1 : 0;
      cand[kTopkBuf / 2 + pos] = v;
    }
    __syncthreads();
    sorted = cand + kTopkBuf / 2;
  } else {
    const int np = next_pow2(max(n, 2));
    for (int i = n + tid; i < np; i += kTopkThreads) cand[i] = kPadKey;
    block_bitonic_sort(cand, np);
  }
  for (int i = tid; i < k; i += kTopkThreads) {
    if (i < n) {
      const uint32_t gi = (uint32_t)sorted[i];
      idx_out[q * k + i] = (int32_t)gi;
      val_out[q * k + i] = a.row[(int64_t)gi - g_offset];
    } else {
      idx_out[q * k + i] = -1;
      val_out[q * k + i] = __int_as_float(0x7f800000);
    }
  }
}

int topk(const float* distmat, int64_t ld, int64_t Q, int64_t G, int64_t g_offset, const int64_t* q_pids,
         const int64_t* q_camids, const int64_t* g_pids, const int64_t* g_camids, int32_t k, int32_t* idx, float* val,
         cudaStream_t stream) {
  IEEE_REQUIRE(distmat && idx && val, "topk: null pointer");
  IEEE_REQUIRE(Q >= 0 && G > 0 && ld >= G && k >= 1 && k <= kTopkBuf / 2, "topk: bad shape (k=%d, max %d)", k, kTopkBuf / 2);
  IEEE_REQUIRE((q_pids == nullptr) == (q_camids == nullptr) && (q_pids == nullptr || (g_pids && g_camids)),
               "topk: junk masking needs all four label arrays");
  IEEE_REQUIRE(g_offset >= 0 && g_offset + G < (int64_t(1) << 31), "topk: global gallery index must fit int32");
  if (Q == 0) return IEEE_OK;
  topk_kernel<<<(unsigned)Q, kTopkThreads, 0, stream>>>(distmat, ld, Q, G, g_offset, q_pids, q_camids, g_pids, g_camids, k, idx, val); count_launch();
  IEEE_CUDA_CHECK(cudaGetLastError());
  return IEEE_OK;
}

// Merge per-shard lists: the global top-k is the k smallest (distance, index) among the shards' k best.
__global__ void __launch_bounds__(256) topk_merge_kernel(const int32_t* __restrict__ idx_all, const float* __restrict__ val_all,
                                                          int shards, int64_t Q, int k, int np, int32_t* __restrict__ idx,
                                                          float* __restrict__ val) {
  extern __shared__ __align__(16) uint8_t ms_raw[];
  uint64_t* keys = reinterpret_cast<uint64_t*>(ms_raw);   // [np]
  const int64_t q = blockIdx.x;
  const int total = shards * k;
  for (int i = threadIdx.x; i < np; i += blockDim.x) {
    uint64_t key = kPadKey;
    if (i < total) {
      const int s = i / k, j = i - s * k;
      const int32_t gi = idx_all[((int64_t)s * Q + q) * k + j];
      if (gi >= 0) key = pack_key(val_all[((int64_t)s * Q + q) * k + j], (uint32_t)gi);
    }
    keys[i] = key;
  }
  block_bitonic_sort(keys, np);
  for (int i = threadIdx.x; i < k; i += blockDim.x) {
    const uint64_t key = keys[i];
    if (key == kPadKey) { idx[q * k + i] = -1; val[q * k + i] = __int_as_float(0x7f800000); continue; }
    idx[q * k + i] = (int32_t)(uint32_t)key;
    // recover the exact distance bits from the shard list that held this entry
    float v = key_to_float((uint32_t)(key >> 32));
    for (int j = 0; j < total; ++j) {
      const int s = j / k, jj = j - s * k;
      if (idx_all[((int64_t)s * Q + q) * k + jj] == (int32_t)(uint32_t)key) { v = val_all[((int64_t)s * Q + q) * k + jj]; break; }
    }
    val[q * k + i] = v;
  }
}

int topk_merge(const int32_t* idx_all, const float* val_all, int32_t shards, int64_t Q, int32_t k, int32_t* idx, float* val,
               cudaStream_t stream) {
  IEEE_REQUIRE(idx_all && val_all && idx && val && shards >= 1 && k >= 1, "topk_merge: bad arguments");
  const int np = next_pow2(max(shards * k, 2));
  IEEE_REQUIRE(np <= 16384, "topk_merge: shards*k=%d too large", shards * k);
  if (Q == 0) return IEEE_OK;
  const size_t smem = size_t(np) * 8;
  IEEE_ENSURE_DYN_SMEM(topk_merge_kernel, smem);
  topk_merge_kernel<<<(unsigned)Q, 256, smem, stream>>>(idx_all, val_all, shards, Q, k, np, idx, val); count_launch();
  IEEE_CUDA_CHECK(cudaGetLastError());
  return IEEE_OK;
}

}  // namespace ieee
