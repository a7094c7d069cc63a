// Shared helpers for libieee_b200.so (sm_100a only).
#pragma once

#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstring>

#include "../../include/ieee_b200.h"

namespace ieee {

// ---- error plumbing (thread-local text behind ieee_last_error) -------------------------------------
void set_error(const char* fmt, ...);
const char* get_error();

#define IEEE_CUDA_CHECK(expr)                                                                   \
  do {                                                                                          \
    cudaError_t _e = (expr);                                                                    \
    if (_e != cudaSuccess) {                                                                    \
      ::ieee::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return IEEE_ERR_CUDA;                                                                     \
    }                                                                                           \
  } while (0)

#define IEEE_REQUIRE(cond, ...)            \
  do {                                     \
    if (!(cond)) {                         \
      ::ieee::set_error(__VA_ARGS__);      \
      return IEEE_ERR_INVALID;             \
    }                                      \
  } while (0)

// cudaFuncAttributeMaxDynamicSharedMemorySize is a PER-DEVICE attribute of a kernel: remember what was set per device
// (a process may evaluate on cuda:1 after cuda:0), one table per call site.
#define IEEE_ENSURE_DYN_SMEM(kernel, bytes)                                                              \
  do {                                                                                                   \
    static std::atomic<size_t> ieee_smem_set_[64];                                                       \
    int ieee_dev_ = -1;                                                                                  \
    IEEE_CUDA_CHECK(cudaGetDevice(&ieee_dev_));                                                          \
    const size_t ieee_need_ = (size_t)(bytes);                                                           \
    if (ieee_need_ > 48 * 1024 &&                                                                        \
        (ieee_dev_ < 0 || ieee_dev_ >= 64 || ieee_smem_set_[ieee_dev_].load(std::memory_order_relaxed) < ieee_need_)) { \
      IEEE_CUDA_CHECK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ieee_need_)); \
      if (ieee_dev_ >= 0 && ieee_dev_ < 64) ieee_smem_set_[ieee_dev_].store(ieee_need_, std::memory_order_relaxed); \
    }                                                                                                    \
  } while (0)

inline int64_t round_up(int64_t x, int64_t m) { return (x + m - 1) / m * m; }
inline size_t align256(size_t x) { return (x + 255) & ~size_t(255); }
int sm_count();
// Small scratch words a kernel's first CTA clears on behalf of the kernels that follow it on the stream (a
// cudaMemsetAsync node between two kernels costs ~4 us of a step; up to 256 words per region).
struct ZeroJob {
  uint32_t* p[2];
  int n[2];
  __device__ __forceinline__ void run() const {
    if (blockIdx.x != 0) return;
    for (int i = 0; i < 2; ++i)
      if (p[i] != nullptr && (int)threadIdx.x < n[i]) p[i][threadIdx.x] = 0u;
  }
};

void count_launch(int n = 1, const char* name = nullptr);   // a name puts the launch on the step timeline (debug flag 128)
extern int g_debug_flags;       // ieee_set_debug_flags()
extern int g_raster_panel;      // ieee_set_raster_panel(): m tiles per raster panel of the contraction (0 = sized for L2)
extern int g_accum_chunk_kb;    // ieee_set_accum_chunk(): K-slices per tensor-core accumulation chunk (0 = whole K)   // bookkeeping behind ieee_launch_count()

// ---- total order on float distances -----------------------------------------------------------------
// Ascending uint32 key == NumPy's ascending sort order: -0.0 == +0.0, every NaN equal and last.
__host__ __device__ __forceinline__ uint32_t order_key(float d) {
  if (d != d) return 0xFFFFFFFFu;
  d += 0.0f;  // -0.0 -> +0.0
#ifdef __CUDA_ARCH__
  uint32_t b = __float_as_uint(d);
#else
  uint32_t b;
  memcpy(&b, &d, 4);
#endif
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__host__ __device__ __forceinline__ float key_to_float(uint32_t k) {
  uint32_t b = (k & 0x80000000u) ? (k & 0x7FFFFFFFu) : ~k;
#ifdef __CUDA_ARCH__
  return __uint_as_float(b);
#else
  float f;
  memcpy(&f, &b, 4);
  return f;
#endif
}
__host__ __device__ __forceinline__ uint64_t pack_key(float d, uint32_t idx) {
  return (uint64_t(order_key(d)) << 32) | idx;
}

// ---- packed operand layout (ieee_pack_features) ------------------------------------------------------
// [hi plane: rows x Dp 16-bit][lo plane (F16X3 only)][norms: rows fp32][row scale: rows fp32], 256-byte aligned
// sections.  FP32_SIMT: [fp32 plane rows x Dp][norms][row scale].
struct PackedLayout {
  int64_t rows, D, Dp;
  size_t hi_off, lo_off, norm_off, scale_off, total;
  bool has_lo;
};
inline PackedLayout packed_layout(int64_t rows, int64_t D, int precision) {
  PackedLayout L;
  L.rows = rows;
  L.D = D;
  L.Dp = round_up(D, 64);
  L.has_lo = (precision == IEEE_PREC_F16X3);
  const size_t esz = precision == IEEE_PREC_FP32_SIMT ? 4 : 2;
  const size_t plane = align256(size_t(rows) * size_t(L.Dp) * esz);
  L.hi_off = 0;
  L.lo_off = L.has_lo ? plane : 0;
  L.norm_off = L.has_lo ? 2 * plane : plane;
  L.scale_off = L.norm_off + align256(size_t(rows) * 4);
  L.total = L.scale_off + align256(size_t(rows) * 4);
  return L;
}

// Rows [r0, r0 + rows) of a packed operand that holds `total` rows, as pointers into its sections: a contraction over
// them reads the same bytes a contraction over the whole operand reads for those rows.
struct PackedRows {
  const uint8_t *hi, *lo;       // lo == hi when the operand has no lo plane
  const float *norm, *scale;
  int64_t rows, Dp;
};
inline PackedRows packed_rows(const void* packed, int64_t total, int64_t r0, int64_t rows, int64_t D, int precision) {
  const PackedLayout L = packed_layout(total, D, precision);
  const uint8_t* b = static_cast<const uint8_t*>(packed);
  const size_t row_bytes = size_t(L.Dp) * (precision == IEEE_PREC_FP32_SIMT ? 4 : 2);
  PackedRows r;
  r.hi = b + L.hi_off + size_t(r0) * row_bytes;
  r.lo = L.has_lo ? b + L.lo_off + size_t(r0) * row_bytes : r.hi;
  r.norm = reinterpret_cast<const float*>(b + L.norm_off) + r0;
  r.scale = reinterpret_cast<const float*>(b + L.scale_off) + r0;
  r.rows = rows;
  r.Dp = L.Dp;
  return r;
}

// ---- gallery grouping (rank.cu): open-addressing hash pid -> slot; members of a slot = the gallery items of that identity
static constexpr long long kEmptyPid = (long long)0x8080808080808080ull;   // memset(0x80) pattern; not a usable pid

// ---- exchange between the ranks of a sharded gallery over NVLink peer memory ----------------------------------
// Every rank owns one exchange buffer (ieee_peer_alloc) that all ranks of the gallery group map (cudaIpc): the rank
// kernels STORE their lists and partial counts straight into EVERY peer's buffer and hand over with flag words,
// instead of an all-gather + all-reduce per query block; each rank then derives all per-query results itself (the
// same integer sums everywhere, so no result broadcast).  Two hand-overs per block are enough, and they also
// protect the buffers across blocks: a rank that has seen flag B of block n from peer p knows p's count kernel of
// block n is over (p is done reading its lists: they may be overwritten), and flag A of block n + 1 from p says p's
// metrics kernel of block n is over (p's count rows may be overwritten).  Header (first 1 KB of a buffer):
//   [0, 128)    flag A[s]: epoch of the last block whose relevant lists from shard s have landed here
//   [128, 256)  flag B[s]: ... whose partial counts (and statistics) from shard s have landed here
//   [256, 384)  unused (flag C of the three-phase protocol this replaced)
//   [384, 408)  sent[3]:   (local) epoch this rank has already signalled per phase
//   [416, 440)  seen[3]:   (local) epoch for which this rank has already seen every peer's flag of the phase
//   [448, 452)  ticket of the metrics kernel's last-CTA reduction (zero between kernels)
//   [512, ...)  stats[s][4]: shard s' {gather overflow, tie pairs, longest merged list, -}
constexpr int kMaxPeers = 16;
constexpr size_t kPeerHeaderBytes = 1024;
constexpr size_t kPeerTicketOffset = 448;   // a word of the header no flag uses: ticket of the metrics kernel's last-CTA reduction
struct PeerView {
  int shards, my;                  // shards == 0: no peer exchange (single GPU / NCCL path)
  unsigned long long epoch;        // one per query block, increasing
  // device-resident epoch (replayable steps): when set, every kernel of the step reads the epoch from this word instead
  // of `epoch`, and the metrics kernel's last CTA advances it once its reduction is over
  unsigned long long* epoch_dev;
  uint8_t* base[kMaxPeers];        // every rank's buffer as mapped into this process; base[my] is this rank's own
  unsigned long long off_rel;      // uint64 [shards][Qb][cap + 1]   relevant lists (+ length), slot s written by shard s
  unsigned long long off_cnt;      // int32  [shards][Qb][W + 2]     partial counts, slot s written by shard s
  unsigned long long off_ap, off_inp, off_first, off_short;   // per-query results [Qtot]: f64, f64, i32, i32
  long long Qb, q_base;            // rows of this query block; index of its first query in the result arrays
  int cap, W;                      // list capacity; count row width
};
inline PeerView no_peers() { PeerView v; memset(&v, 0, sizeof(v)); return v; }

// ---- raw PTX: mbarrier / TMA / tcgen05 ----------------------------------------------------------------
#ifdef __CUDACC__
__device__ __forceinline__ uint32_t hash_pid(long long pid) {
  uint64_t x = (uint64_t)pid;
  x ^= x >> 33; x *= 0xff51afd7ed558ccdull; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ull; x ^= x >> 33;   // murmur3 finaliser
  return (uint32_t)x;
}
// slot of `pid`, or -1 if the gallery has no such identity
__device__ __forceinline__ int group_find(const long long* __restrict__ keys, int64_t T, long long pid) {
  uint32_t h = hash_pid(pid) & (uint32_t)(T - 1);
  while (true) {
    const long long k = keys[h];
    if (k == pid) return (int)h;
    if (k == kEmptyPid) return -1;
    h = (h + 1) & (uint32_t)(T - 1);
  }
}

__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_sys(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
// Called by every thread of every CTA at the top of the kernel that CONSUMES phase `phase` (0 lists, 1 partial
// counts).  The producing kernel is the previous one on this stream, so all of this rank's stores --
// including the ones into peer buffers -- are complete when any CTA of this kernel runs: the first CTA to get here
// publishes them (fence, then one flag store per peer), then everybody waits until every peer has done the same.
// `stats_src` (4 words, may be null) is copied into this rank's stats slot of every peer before the flags.
// The wait is bounded like mbar_wait: a peer that never arrives traps instead of hanging the box.
__device__ __forceinline__ void peer_signal_and_wait(const PeerView& pv, int phase, const unsigned long long* stats_src = nullptr) {
  if (threadIdx.x < 32) {
    const int lane = threadIdx.x;
    // (a device epoch is written only by the step's last CTA, after every read of it: all CTAs read the same value)
    const unsigned long long epoch = pv.epoch_dev ? *reinterpret_cast<volatile const unsigned long long*>(pv.epoch_dev) : pv.epoch;
    unsigned long long* hdr = reinterpret_cast<unsigned long long*>(pv.base[pv.my] + 384);
    unsigned long long* sent = hdr + phase;          // epoch this rank has signalled
    unsigned long long* seen = hdr + 4 + phase;      // epoch for which all peers' flags were already observed here
    // later CTAs of the kernel (a grid is many waves) find `seen` set and skip the system-scope polling altogether
    unsigned long long have = 0;
    if (lane == 0) have = *reinterpret_cast<volatile unsigned long long*>(seen);
    have = __shfl_sync(0xffffffffu, have, 0);
    if (have < epoch) {
      bool first = false;
      if (lane == 0) first = atomicMax(sent, epoch) < epoch;
      first = __shfl_sync(0xffffffffu, first, 0);
      if (first) {
        if (stats_src != nullptr && lane < pv.shards) {
          unsigned long long* dst = reinterpret_cast<unsigned long long*>(pv.base[lane] + 512) + 4 * pv.my;
          for (int i = 0; i < 4; ++i) dst[i] = stats_src[i];
        }
        __threadfence_system();
        __syncwarp();
        if (lane < pv.shards)
          st_release_sys(reinterpret_cast<unsigned long long*>(pv.base[lane] + 128 * phase) + pv.my, epoch);
      }
      // lane s polls the flag of shard s: the S loads are in flight together
      const unsigned long long* mine = reinterpret_cast<const unsigned long long*>(pv.base[pv.my] + 128 * phase);
      const long long t0 = clock64();
      bool ok = lane >= pv.shards;
      while (!__all_sync(0xffffffffu, ok)) {
        if (!ok) ok = ld_acquire_sys(mine + lane) >= epoch;
        if (clock64() - t0 > 8000000000ll) {
          if (!ok) printf("ieee_b200: rank %d waited in vain for shard %d (phase %d, epoch %llu)\n", pv.my, lane, phase, epoch);
          __trap();
        }
      }
      __threadfence();
      if (lane == 0) atomicMax(seen, epoch);
    } else {
      __threadfence();     // order this CTA's reads of the exchanged data after its read of `seen`
    }
  }
  __syncthreads();
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// Arrive on the barrier at the same smem offset in cluster CTA `cta` (mapa + remote arrive).
__device__ __forceinline__ void mbar_arrive_cluster(uint64_t* bar, uint32_t cta) {
  uint32_t remote;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(smem_u32(bar)), "r"(cta));
  // default semantics (release at CTA scope), as CUTLASS' ClusterBarrier::arrive(cta_id): a cluster-scope release
  // costs a MEMBAR.ALL.CTA + ERRBAR per arrival and starved the cta_group::2 pipeline (ncu: 33 % of stall samples)
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(remote) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Spin on try_wait.  A pipeline bug would otherwise hang the GPU until the host kills the box, so the
// wait traps after ~2 s of SM clocks (IEEE_MBAR_WATCHDOG_CYCLES; 0 disables).
#ifndef IEEE_MBAR_WATCHDOG_CYCLES
#define IEEE_MBAR_WATCHDOG_CYCLES 4000000000ll
#endif
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (IEEE_MBAR_WATCHDOG_CYCLES > 0 && clock64() - t0 > IEEE_MBAR_WATCHDOG_CYCLES) {
      printf("ieee_b200: mbarrier wait timed out (block %d thread %d bar %u parity %u)\n", blockIdx.x, threadIdx.x,
             smem_u32(bar), parity);
      __trap();
    }
  }
}

__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}"
      : "=r"(pred));
  return pred != 0;
}

__device__ __forceinline__ void tma_prefetch_desc(const void* desc) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(desc) : "memory");
}
// 2-D tiled TMA load global -> this CTA's smem, completion on this CTA's mbarrier.
__device__ __forceinline__ void tma_load_2d(const void* desc, uint64_t* bar, void* smem, int32_t c0, int32_t c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(smem)),
      "l"(desc), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
// cta_group::2 form: data lands in the issuing CTA's smem, the transaction bytes are signalled on the
// mbarrier of the PAIR LEADER (peer bit cleared in the barrier address).
__device__ __forceinline__ void tma_load_2d_pair(const void* desc, uint64_t* bar, void* smem, int32_t c0, int32_t c1) {
  uint32_t mbar = smem_u32(bar) & 0xFEFFFFFFu;
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], "
      "[%2];" ::"r"(smem_u32(smem)),
      "l"(desc), "r"(mbar), "r"(c0), "r"(c1)
      : "memory");
}

// smem tile -> global through a tensor map (clips rows / columns outside the tensor); bulk-group completion.
__device__ __forceinline__ void tma_store_2d(const void* desc, const void* smem, int32_t c0, int32_t c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(desc),
               "r"(smem_u32(smem)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void tma_store_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void tma_store_wait() {
  asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}

__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

template <int kCtaGroup>
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t cols) {
  if constexpr (kCtaGroup == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  } else {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
}
template <int kCtaGroup>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
  if constexpr (kCtaGroup == 1)
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
  else
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}

// D[tmem] (+)= A[smem] * B[smem]^T, kind::f16 (bf16 inputs, fp32 accumulate).  One thread issues.
template <int kCtaGroup>
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                          uint32_t accumulate) {
  if constexpr (kCtaGroup == 1) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
  } else {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
  }
}
// Make the mbarrier track completion of all MMAs issued so far by this thread (implies fence::before_thread_sync).
template <int kCtaGroup>
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  if constexpr (kCtaGroup == 1) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
  } else {  // arrive on the barrier at this offset in BOTH CTAs of the pair
    asm volatile(
        "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
            smem_u32(bar)),
        "h"((uint16_t)3)
        : "memory");
  }
}

// 32 lanes x 32 consecutive fp32 columns of TMEM -> 32 registers per thread (thread i <-> lane base+i).
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// K-major, SWIZZLE_128B shared-memory matrix descriptor (sm_100 "version 1"):
//   start address >> 4 in bits [0,14), LBO unused for swizzled K-major (0), SBO = 1024 B (8 rows x 128 B) >> 4
//   in bits [32,46), descriptor version 1 in bits [46,48), layout type SWIZZLE_128B = 2 in bits [61,64).
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
  return uint64_t((smem_addr & 0x3FFFFu) >> 4) | (uint64_t(1024 >> 4) << 32) | (uint64_t(1) << 46) | (uint64_t(2) << 61);
}
// Instruction descriptor, kind::f16: D fp32 (bit 4), A and B format at bits 7 / 10, both K-major, N >> 3 at bit 17,
// M >> 4 at bit 24.
__host__ __device__ constexpr uint32_t umma_idesc_16bit(uint32_t M, uint32_t N, uint32_t fmt /* 0 f16, 1 bf16 */) {
  return (1u << 4) | (fmt << 7) | (fmt << 10) | ((N >> 3) << 17) | ((M >> 4) << 24);
}
#endif  // __CUDACC__

}  // namespace ieee
