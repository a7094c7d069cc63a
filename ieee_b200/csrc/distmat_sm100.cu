// Distance-matrix contraction on the sm_100a tensor cores.
//
// Replaces torchreid/metrics/distance.py:59-64 (out = (|a|^2 + |b|^2) - 2 a b^T via addmm_) and
// distance.py:77-80 (out = 1 - normalize(a) normalize(b)^T via mm).  Both feature matrices are row-major
// [rows, D], i.e. K-major operands of C = A * B^T -- the layout tcgen05.mma consumes directly.
//
// Kernel shape (persistent, warp specialised, one CTA per SM):
//   warp 0   : TMA producer   -- cp.async.bulk.tensor 2-D tiles (SWIZZLE_128B) into a kStages smem ring
//   warp 1   : MMA issuer     -- one elected lane issues tcgen05.mma (kind::f16, fp16/bf16 in, fp32 accumulate in TMEM)
//   warp 2   : TMEM allocator -- 512 columns = two 128 x 256 fp32 accumulator stages
//   warps 4-7: epilogue       -- tcgen05.ld -> d = fma(coef[row] * sg[col], acc, rq[row] + rg[col]) in registers ->
//                                swizzled smem tile -> TMA store (clips the ragged edges); a transposing
//                                st.global path serves outputs whose row pitch is not a multiple of 16 bytes
// kCtaGroup == 2 pairs two SMs on one 256 x 256 tile (tcgen05.mma.cta_group::2): each CTA loads its own 128
// rows of A and HALF of the B tile.
//
// F16X3 (fp32-grade) mode runs three k-passes per 64-wide k block into the same accumulator:
// (A_hi,B_hi), (A_hi,B_lo), (A_lo,B_hi); rows were scaled by powers of two when packed, undone by sq/sg here.
#include <cuda.h>
#include <cuda_fp16.h>

#include "common.cuh"

namespace ieee {

constexpr int BLOCK_M = 128;  // rows of A per CTA == TMEM lanes
constexpr int BLOCK_N = 256;  // columns per tile == UMMA N
constexpr int BLOCK_K = 64;   // 16-bit elements per k block == one 128-byte swizzle span
constexpr int UMMA_K = 16;
constexpr int kEpilogueWarps = 4;
constexpr int kThreads = 128 + 32 * kEpilogueWarps;
constexpr int kStagePitch = 33;  // floats; padded 32 x 32 transpose tile (fallback epilogue)

template <int CG>
struct GemmCfg {
  static constexpr int kStages = (CG == 1) ? 4 : 6;
  static constexpr int kBRows = BLOCK_N / CG;                      // B rows this CTA loads
  static constexpr uint32_t kABytes = BLOCK_M * BLOCK_K * 2;       // 16 KB
  static constexpr uint32_t kBBytes = kBRows * BLOCK_K * 2;        // 32 KB / 16 KB
  static constexpr uint32_t kStageBytes = kABytes + kBBytes;
  // per epilogue warp: 32 x 32 fp32 output tile (4 KB, 1024-aligned for SWIZZLE_128B; the fallback's padded
  // 32 x 33 tile needs 4224 B) + the tile's 256 column terms rg / sg
  static constexpr uint32_t kEpiTileBytes = 5 * 1024;
  static constexpr uint32_t kEpiColBytes = 2 * BLOCK_N * 4;
  static constexpr uint32_t kEpiWarpBytes = 7 * 1024;              // keeps every warp's tile 1024-byte aligned
  static constexpr uint32_t kEpiBytes = kEpilogueWarps * kEpiWarpBytes;
  static constexpr uint32_t kBarBytes = 256;
  static constexpr uint32_t kSmemBytes = kStages * kStageBytes + kEpiBytes + kBarBytes + 1024 /* alignment slack */;
  static_assert(kEpiTileBytes + kEpiColBytes <= kEpiWarpBytes, "epilogue smem carve");
};

struct GemmParams {
  const float* rq;   // per query row additive term (euclidean: squared norm; cosine: nullptr -> 1)
  const float* rg;   // per gallery row additive term (euclidean: squared norm; cosine: nullptr -> 0)
  const float* sq;   // per query row power-of-two scale (F16X3; 1 otherwise)
  const float* sg;   // per gallery row power-of-two scale
  float* out;
  int64_t ldo;
  int Q, G;
  int num_kb;        // Dp / 64
  int nseg;          // 1 (BF16) or 3 (F16X3)
  float alpha;       // -2 (euclidean) or -1 (cosine, negative dot product)
  float base0;       // additive term when there are no row terms: 1 (cosine: 1 - a.b) or 0 (negative dot product)
  int num_m_tiles, num_n_tiles;
  int panel_m;       // m tiles per raster panel: the panel's A rows stay L2-resident while it sweeps all n tiles
  uint32_t idesc;    // tcgen05 instruction descriptor (operand format, M, N)
  int tma_store;     // 1: out is 16-byte aligned with a 16-byte-multiple pitch -> TMA store epilogue
  int debug;         // ieee_set_debug_flags()
  // near-duplicate list (euclidean, chunked kernel): [0] = number of entries, [1 ..] = (row << 32 | first column) of every
  // (row, 128-column span) holding an output with d < fix_tau * (|q|^2 + |g|^2); distmat_fixup_kernel recomputes those
  // outputs in difference form.  May be null.
  unsigned long long* fix_list;
  uint32_t fix_cap;
  float fix_tau;
};

// Tile order.  Inside a panel of `panel_m` m tiles, m runs fastest (the CTAs of one wave share B tiles in L2);
// panels follow each other, so the A rows of a panel are fetched from HBM once however many n tiles there are
// (a tall query block against a narrow gallery shard would otherwise stream all of A once per n tile).
__device__ __forceinline__ void tile_coords(const GemmParams& p, int t, int& m_blk, int& n_blk) {
  const int per_panel = p.panel_m * p.num_n_tiles;
  const int panel = t / per_panel;
  const int r = t - panel * per_panel;
  const int m0 = panel * p.panel_m;
  const int pm = min(p.panel_m, p.num_m_tiles - m0);
  n_blk = r / pm;
  m_blk = m0 + (r - n_blk * pm);
}

template <int CG>
__global__ void __launch_bounds__(kThreads, 1)
distmat_umma_kernel(const __grid_constant__ CUtensorMap tm_a_hi, const __grid_constant__ CUtensorMap tm_a_lo,
                    const __grid_constant__ CUtensorMap tm_b_hi, const __grid_constant__ CUtensorMap tm_b_lo,
                    const __grid_constant__ CUtensorMap tm_out, const GemmParams p) {
  using Cfg = GemmCfg<CG>;
  constexpr int kStages = Cfg::kStages;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + kStages * Cfg::kABytes;
  uint8_t* smem_epi = smem + kStages * Cfg::kStageBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_epi + Cfg::kEpiBytes);
  uint64_t* full_bar = bars;                      // [kStages]  TMA -> MMA   (lives in the pair leader for CG == 2)
  uint64_t* empty_bar = bars + kStages;           // [kStages]  MMA -> TMA   (per CTA)
  uint64_t* tmem_full_bar = bars + 2 * kStages;   // [2]        MMA -> epilogue (per CTA)
  uint64_t* tmem_empty_bar = bars + 2 * kStages + 2;  // [2]    epilogue -> MMA (leader)
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bars + 2 * kStages + 4);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t cta_rank = (CG == 2) ? cluster_ctarank() : 0;
  const bool is_leader = cta_rank == 0;

  if (warp == 0 && elect_one()) {
    tma_prefetch_desc(&tm_a_hi);
    tma_prefetch_desc(&tm_b_hi);
    if (p.nseg == 3) {
      tma_prefetch_desc(&tm_a_lo);
      tma_prefetch_desc(&tm_b_lo);
    }
    if (p.tma_store) tma_prefetch_desc(&tm_out);
  }
  if (warp == 1 && elect_one()) {
    for (int i = 0; i < kStages; ++i) {
      mbar_init(&full_bar[i], CG);   // one arrive(+expect_tx) per producing CTA
      mbar_init(&empty_bar[i], 1);   // one tcgen05.commit
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tmem_full_bar[i], 1);
      mbar_init(&tmem_empty_bar[i], CG * kEpilogueWarps);   // one arrival per epilogue warp
    }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<CG>(tmem_ptr_smem, 512);
  tc_fence_before();
  if constexpr (CG == 2) cluster_sync_all(); else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  // Persistent tile loop shared by all roles: tile t -> (m fastest, so co-resident CTAs share B tiles in L2).
  const int num_tiles = p.num_m_tiles * p.num_n_tiles;
  const int group_id = blockIdx.x / CG;
  const int num_groups = gridDim.x / CG;
  const int total_kb = p.num_kb * p.nseg;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int t = group_id; t < num_tiles; t += num_groups) {
        int m_blk, n_blk;
        tile_coords(p, t, m_blk, n_blk);
        const int row_a = (m_blk * CG + (int)cta_rank) * BLOCK_M;
        const int row_b = n_blk * BLOCK_N + (int)cta_rank * Cfg::kBRows;
        for (int kb = 0; kb < total_kb; ++kb) {
          const int kk = kb / p.nseg, seg = kb - kk * p.nseg;
          mbar_wait(&empty_bar[stage], phase ^ 1);
          const CUtensorMap* ma = (seg == 2) ? &tm_a_lo : &tm_a_hi;
          const CUtensorMap* mb = (seg == 1) ? &tm_b_lo : &tm_b_hi;
          void* sa = smem_a + stage * Cfg::kABytes;
          void* sb = smem_b + stage * Cfg::kBBytes;
          if constexpr (CG == 1) {
            mbar_expect_tx(&full_bar[stage], Cfg::kStageBytes);
            tma_load_2d(ma, &full_bar[stage], sa, kk * BLOCK_K, row_a);
            tma_load_2d(mb, &full_bar[stage], sb, kk * BLOCK_K, row_b);
          } else {
            // Both CTAs' bytes are counted on the leader's barrier; each CTA contributes one arrival.
            if (is_leader) mbar_expect_tx(&full_bar[stage], 2 * Cfg::kStageBytes);
            tma_load_2d_pair(ma, &full_bar[stage], sa, kk * BLOCK_K, row_a);
            tma_load_2d_pair(mb, &full_bar[stage], sb, kk * BLOCK_K, row_b);
            if (!is_leader) mbar_arrive_cluster(&full_bar[stage], 0);
          }
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ===================== MMA issuer (pair leader only) =====================
    if (is_leader && elect_one()) {
      const uint32_t idesc = p.idesc;
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      for (int t = group_id; t < num_tiles; t += num_groups, ++it) {
        const int acc = it & 1;
        const uint32_t acc_phase = (it >> 1) & 1;
        mbar_wait(&tmem_empty_bar[acc], acc_phase ^ 1);   // epilogue drained this accumulator stage
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + acc * BLOCK_N;
        for (int kb = 0; kb < total_kb; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint64_t da = umma_desc_sw128(smem_u32(smem_a + stage * Cfg::kABytes));
          const uint64_t db = umma_desc_sw128(smem_u32(smem_b + stage * Cfg::kBBytes));
#pragma unroll
          for (int k = 0; k < BLOCK_K / UMMA_K; ++k) {
            // advance 16 elements = 32 bytes inside the 128-byte swizzle span: +2 in the (addr >> 4) field
            umma_bf16<CG>(tmem_d, da + 2 * k, db + 2 * k, idesc, (kb | k) != 0);
          }
          umma_commit<CG>(&empty_bar[stage]);                 // smem slot free once these MMAs retire
          if (kb == total_kb - 1) umma_commit<CG>(&tmem_full_bar[acc]);  // accumulator complete
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
    __syncwarp();
  } else if (warp >= 4) {
    // ===================== epilogue =====================
    const int ew = warp - 4;                       // == warp % 4 -> TMEM lane quarter
    uint8_t* my_epi = smem_epi + ew * Cfg::kEpiWarpBytes;
    float* tile = reinterpret_cast<float*>(my_epi);                          // 1024-byte aligned
    float* col_rg = reinterpret_cast<float*>(my_epi + Cfg::kEpiTileBytes);   // [256]
    float* col_sg = col_rg + BLOCK_N;                                        // [256]
    int it = 0;
    for (int t = group_id; t < num_tiles; t += num_groups, ++it) {
      int m_blk, n_blk;
        tile_coords(p, t, m_blk, n_blk);
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      const int row0 = (m_blk * CG + (int)cta_rank) * BLOCK_M + ew * 32;   // first row of this warp
      const int col_tile = n_blk * BLOCK_N;
      // this thread's row terms (thread <-> TMEM lane <-> output row)
      const int my_row = row0 + lane;
      const float rq_row = (p.rq != nullptr) ? (my_row < p.Q ? p.rq[my_row] : 0.0f) : p.base0;
      const float coef_row = p.alpha * ((p.sq != nullptr && my_row < p.Q) ? p.sq[my_row] : 1.0f);
      // the tile's column terms, one private copy per warp (no cross-warp barrier needed)
      __syncwarp();
#pragma unroll
      for (int j = 0; j < BLOCK_N / 32; ++j) {
        const int col = col_tile + j * 32 + lane;
        col_rg[j * 32 + lane] = (p.rg != nullptr && col < p.G) ? p.rg[col] : 0.0f;
        col_sg[j * 32 + lane] = (p.sg != nullptr && col < p.G) ? p.sg[col] : 1.0f;
      }
      __syncwarp();
      mbar_wait(&tmem_full_bar[acc], acc_phase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + acc * BLOCK_N + (uint32_t(ew * 32) << 16);
#pragma unroll 1
      for (int c = 0; c < BLOCK_N / 32; ++c) {
        uint32_t v[32];
        if (!(p.debug & 2)) {
          tmem_ld_32x32(taddr + c * 32, v);
          tmem_ld_wait();
        }
        if (c == BLOCK_N / 32 - 1) {
          // all of this warp's accumulator reads are done: hand the TMEM stage back to the MMA warp
          tc_fence_before();
          __syncwarp();
          if (lane == 0) {
            if constexpr (CG == 1) mbar_arrive(&tmem_empty_bar[acc]); else mbar_arrive_cluster(&tmem_empty_bar[acc], 0);
          }
        }
        if (col_tile + c * 32 >= p.G || row0 >= p.Q || (p.debug & 1)) continue;   // warp-uniform
        if (p.tma_store) {
          // d in registers (thread = row), 16-byte chunks XOR-swizzled by (row & 7) as SWIZZLE_128B expects
          if (lane == 0) tma_store_wait_read<0>();     // the previous store has finished reading `tile`
          __syncwarp();
#pragma unroll
          for (int k = 0; k < 8; ++k) {
            float4 o;
            const float4 g4 = *reinterpret_cast<const float4*>(col_rg + c * 32 + 4 * k);
            const float4 s4 = *reinterpret_cast<const float4*>(col_sg + c * 32 + 4 * k);
            o.x = __fmaf_rn(coef_row * s4.x, __uint_as_float(v[4 * k + 0]), __fadd_rn(rq_row, g4.x));
            o.y = __fmaf_rn(coef_row * s4.y, __uint_as_float(v[4 * k + 1]), __fadd_rn(rq_row, g4.y));
            o.z = __fmaf_rn(coef_row * s4.z, __uint_as_float(v[4 * k + 2]), __fadd_rn(rq_row, g4.z));
            o.w = __fmaf_rn(coef_row * s4.w, __uint_as_float(v[4 * k + 3]), __fadd_rn(rq_row, g4.w));
            *reinterpret_cast<float4*>(reinterpret_cast<uint8_t*>(tile) + lane * 128 + ((k ^ (lane & 7)) << 4)) = o;
          }
          fence_proxy_async();                          // generic-proxy smem writes -> visible to the TMA engine
          __syncwarp();
          if (lane == 0) {
            tma_store_2d(&tm_out, tile, col_tile + c * 32, row0);
            tma_store_commit();
          }
        } else {
          // transpose through smem so that a warp writes 32 consecutive columns of one row per instruction
          const int col = col_tile + c * 32 + lane;
          const float rg_lane = col_rg[c * 32 + lane], sg_lane = col_sg[c * 32 + lane];
          __syncwarp();
#pragma unroll
          for (int j = 0; j < 32; ++j) tile[lane * kStagePitch + j] = __uint_as_float(v[j]);
          __syncwarp();
#pragma unroll 8
          for (int r = 0; r < 32; ++r) {
            const float rq = __shfl_sync(0xffffffffu, rq_row, r);
            const float cf = __shfl_sync(0xffffffffu, coef_row, r);
            const float a = tile[r * kStagePitch + lane];
            const int row = row0 + r;
            if (row < p.Q && col < p.G)
              p.out[(int64_t)row * p.ldo + col] = __fmaf_rn(cf * sg_lane, a, __fadd_rn(rq, rg_lane));
          }
        }
      }
    }
    if (p.tma_store && lane == 0) tma_store_wait<0>();   // all bulk stores complete before smem goes away
    __syncwarp();
  }

  tc_fence_before();
  if constexpr (CG == 2) cluster_sync_all(); else __syncthreads();
  if (warp == 2) tmem_dealloc<CG>(tmem_base, 512);
}

// =====================================================================================================
// Chunked-accumulation variant (cta_group::1).
//
// The tcgen05 fp32 accumulator truncates (measured: the dot product comes out low by up to 1.3e-5 relative after
// the 432 chained MMAs of one F16X3 output, profiles/accuracy_r1.txt).  Here the MMA warp closes an accumulator
// stage every `chunk_kb` K-slices and EIGHT epilogue warps add the chunks into fp32 registers with
// round-to-nearest (128 running sums per thread; 168 registers per thread at 384 threads fill the register file),
// so a truncating chain is only chunk_kb * 4 * nseg MMAs long.  TMEM stages alternate per chunk, so the
// register adds of chunk c overlap the MMAs of chunk c + 1.
// =====================================================================================================
constexpr int kEpiWarpsC = 8;
constexpr int kThreadsC = 128 + 32 * kEpiWarpsC;
constexpr int kPitchC = 17;                      // floats; padded 32 x 16 transpose tile (fallback store path)

template <int CG>
struct GemmCfgC {
  static constexpr int kStages = (CG == 1) ? 4 : 6;
  static constexpr int kBRows = BLOCK_N / CG;
  static constexpr uint32_t kABytes = BLOCK_M * BLOCK_K * 2;
  static constexpr uint32_t kBBytes = kBRows * BLOCK_K * 2;
  static constexpr uint32_t kStageBytes = kABytes + kBBytes;
  // store epilogue: 32 x 16 fp32 (2 KB, SWIZZLE_64B) / 32 x 17 padded (2176 B)
  static constexpr uint32_t kEpiTileBytes = 2560;
  static constexpr uint32_t kEpiColBytes = 2 * 128 * 4;
  static constexpr uint32_t kEpiWarpBytes = 4096;   // keeps every warp's tile 1024-byte aligned
  static constexpr uint32_t kEpiBytes = kEpiWarpsC * kEpiWarpBytes;
  static constexpr uint32_t kBarBytes = 256;
  static constexpr uint32_t kSmemBytes = kStages * kStageBytes + kEpiBytes + kBarBytes + 1024;
  static_assert(kEpiTileBytes + kEpiColBytes <= kEpiWarpBytes, "epilogue smem carve");
  static_assert(kSmemBytes <= 232448, "shared memory budget");
};

// p is __grid_constant__ so that every use reads its field from the parameter bank: taken by value, the compiler
// hoists the fields into registers at kernel entry, and in this kernel, whose 168 registers are full, that adds spills.
template <int CG>
__global__ void __launch_bounds__(kThreadsC, 1)
distmat_umma_chunked_kernel(const __grid_constant__ CUtensorMap tm_a_hi, const __grid_constant__ CUtensorMap tm_a_lo,
                            const __grid_constant__ CUtensorMap tm_b_hi, const __grid_constant__ CUtensorMap tm_b_lo,
                            const __grid_constant__ CUtensorMap tm_out, const __grid_constant__ GemmParams p,
                            const int chunk_kb) {
  using Cfg = GemmCfgC<CG>;
  constexpr int kStages = Cfg::kStages;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + kStages * Cfg::kABytes;
  uint8_t* smem_epi = smem + kStages * Cfg::kStageBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_epi + Cfg::kEpiBytes);
  uint64_t* full_bar = bars;                          // lives in the pair leader for CG == 2
  uint64_t* empty_bar = bars + kStages;               // per CTA
  uint64_t* tmem_full_bar = bars + 2 * kStages;       // per CTA
  uint64_t* tmem_empty_bar = bars + 2 * kStages + 2;  // leader
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bars + 2 * kStages + 4);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t cta_rank = (CG == 2) ? cluster_ctarank() : 0;
  const bool is_leader = cta_rank == 0;

  if (warp == 0 && elect_one()) {
    tma_prefetch_desc(&tm_a_hi);
    tma_prefetch_desc(&tm_b_hi);
    if (p.nseg == 3) {
      tma_prefetch_desc(&tm_a_lo);
      tma_prefetch_desc(&tm_b_lo);
    }
    if (p.tma_store) tma_prefetch_desc(&tm_out);
  }
  if (warp == 1 && elect_one()) {
    for (int i = 0; i < kStages; ++i) {
      mbar_init(&full_bar[i], CG);
      mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tmem_full_bar[i], 1);
      mbar_init(&tmem_empty_bar[i], CG * kEpiWarpsC);   // one arrival per epilogue warp
    }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<CG>(tmem_ptr_smem, 512);
  tc_fence_before();
  if constexpr (CG == 2) cluster_sync_all(); else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  const int num_tiles = p.num_m_tiles * p.num_n_tiles;
  const int group_id = blockIdx.x / CG;
  const int num_groups = gridDim.x / CG;
  const int num_chunks = (p.num_kb + chunk_kb - 1) / chunk_kb;

  if (warp < 4) {
    if (warp == 0) {
      // ===================== TMA producer =====================
      if (elect_one()) {
        int stage = 0;
        uint32_t phase = 0;
        for (int t = group_id; t < num_tiles; t += num_groups) {
          int m_blk, n_blk;
          tile_coords(p, t, m_blk, n_blk);
          const int row_a = (m_blk * CG + (int)cta_rank) * BLOCK_M;
          const int row_b = n_blk * BLOCK_N + (int)cta_rank * Cfg::kBRows;
          for (int c = 0; c < num_chunks; ++c) {
            const int k0 = c * chunk_kb, k1 = min(p.num_kb, k0 + chunk_kb);
            // Inside a chunk the two cross terms (A_hi B_lo, A_lo B_hi: ~2^-11 of the main term) go first and the
            // hi*hi products last: every tcgen05.mma truncates the running sum once, at the magnitude it has reached,
            // so the only full-magnitude truncations left are the (k1 - k0) * 4 hi*hi instructions of the chunk.
            for (int s = 0; s < p.nseg; ++s) {
              const int seg = (p.nseg == 3) ? (s == 2 ? 0 : s + 1) : 0;
              const CUtensorMap* ma = (seg == 2) ? &tm_a_lo : &tm_a_hi;
              const CUtensorMap* mb = (seg == 1) ? &tm_b_lo : &tm_b_hi;
              for (int kk = k0; kk < k1; ++kk) {
                mbar_wait(&empty_bar[stage], phase ^ 1);
                void* sa = smem_a + stage * Cfg::kABytes;
                void* sb = smem_b + stage * Cfg::kBBytes;
                if constexpr (CG == 1) {
                  mbar_expect_tx(&full_bar[stage], Cfg::kStageBytes);
                  tma_load_2d(ma, &full_bar[stage], sa, kk * BLOCK_K, row_a);
                  tma_load_2d(mb, &full_bar[stage], sb, kk * BLOCK_K, row_b);
                } else {
                  if (is_leader) mbar_expect_tx(&full_bar[stage], 2 * Cfg::kStageBytes);
                  tma_load_2d_pair(ma, &full_bar[stage], sa, kk * BLOCK_K, row_a);
                  tma_load_2d_pair(mb, &full_bar[stage], sb, kk * BLOCK_K, row_b);
                  if (!is_leader) mbar_arrive_cluster(&full_bar[stage], 0);
                }
                if (++stage == kStages) { stage = 0; phase ^= 1; }
              }
            }
          }
        }
      }
      __syncwarp();
    } else if (warp == 1) {
      // ===================== MMA issuer (pair leader only) =====================
      if (is_leader && elect_one()) {
        const uint32_t idesc = p.idesc;
        int stage = 0;
        uint32_t phase = 0;
        int ci = 0;   // chunk counter over the whole kernel: TMEM stage = ci & 1
        for (int t = group_id; t < num_tiles; t += num_groups) {
          for (int c = 0; c < num_chunks; ++c, ++ci) {
            const int acc = ci & 1;
            mbar_wait(&tmem_empty_bar[acc], ((ci >> 1) & 1) ^ 1);
            tc_fence_after();
            const uint32_t tmem_d = tmem_base + acc * BLOCK_N;
            const int kb_begin = c * chunk_kb * p.nseg;
            const int kb_end = min(p.num_kb, (c + 1) * chunk_kb) * p.nseg;
            for (int kb = kb_begin; kb < kb_end; ++kb) {
              mbar_wait(&full_bar[stage], phase);
              tc_fence_after();
              const uint64_t da = umma_desc_sw128(smem_u32(smem_a + stage * Cfg::kABytes));
              const uint64_t db = umma_desc_sw128(smem_u32(smem_b + stage * Cfg::kBBytes));
#pragma unroll
              for (int k = 0; k < BLOCK_K / UMMA_K; ++k)
                umma_bf16<CG>(tmem_d, da + 2 * k, db + 2 * k, idesc, (kb != kb_begin) || k != 0);
              umma_commit<CG>(&empty_bar[stage]);
              if (kb == kb_end - 1) umma_commit<CG>(&tmem_full_bar[acc]);
              if (++stage == kStages) { stage = 0; phase ^= 1; }
            }
          }
        }
      }
      __syncwarp();
    }
  } else {
    // ===================== epilogue: 8 warps, thread = (row, 128-column half) =====================
    const int ew = warp - 4;
    const int quarter = ew & 3;                    // TMEM lane quarter == warp % 4
    const int half = ew >> 2;                      // columns [128 * half, 128 * half + 128)
    uint8_t* my_epi = smem_epi + ew * Cfg::kEpiWarpBytes;
    float* tile = reinterpret_cast<float*>(my_epi);
    float* col_rg = reinterpret_cast<float*>(my_epi + Cfg::kEpiTileBytes);   // [128]
    float* col_sg = col_rg + 128;                                            // [128]
    int ci = 0;
    for (int t = group_id; t < num_tiles; t += num_groups) {
      int m_blk, n_blk;
        tile_coords(p, t, m_blk, n_blk);
      const int row0 = (m_blk * CG + (int)cta_rank) * BLOCK_M + quarter * 32;
      const int col0 = n_blk * BLOCK_N + half * 128;
      const int my_row = row0 + lane;
      const float rq_row = (p.rq != nullptr) ? (my_row < p.Q ? p.rq[my_row] : 0.0f) : p.base0;
      const float coef_row = p.alpha * ((p.sq != nullptr && my_row < p.Q) ? p.sq[my_row] : 1.0f);
      __syncwarp();
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int col = col0 + j * 32 + lane;
        col_rg[j * 32 + lane] = (p.rg != nullptr && col < p.G) ? p.rg[col] : 0.0f;
        col_sg[j * 32 + lane] = (p.sg != nullptr && col < p.G) ? p.sg[col] : 1.0f;
      }
      __syncwarp();
      float r[128];
      for (int c = 0; c < num_chunks; ++c, ++ci) {
        const int acc = ci & 1;
        mbar_wait(&tmem_full_bar[acc], (ci >> 1) & 1);
        tc_fence_after();
        const uint32_t taddr = tmem_base + acc * BLOCK_N + half * 128 + (uint32_t(quarter * 32) << 16);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          uint32_t v[32];
          tmem_ld_32x32(taddr + j * 32, v);
          tmem_ld_wait();
          if (c == 0) {
#pragma unroll
            for (int i = 0; i < 32; ++i) r[j * 32 + i] = __uint_as_float(v[i]);
          } else {
#pragma unroll
            for (int i = 0; i < 32; ++i) r[j * 32 + i] = __fadd_rn(r[j * 32 + i], __uint_as_float(v[i]));
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if constexpr (CG == 1) mbar_arrive(&tmem_empty_bar[acc]); else mbar_arrive_cluster(&tmem_empty_bar[acc], 0);
        }
      }
      if (row0 >= p.Q || (p.debug & 1)) continue;
      const bool fix_on = p.fix_list != nullptr && p.rq != nullptr;
      float viol = 0.f;                          // min over this thread's 128 outputs of d - fix_tau * (|q|^2 + |g|^2)
      // d = fma(coef * sg, sum, rq + rg), 16 columns at a time
#pragma unroll
      for (int s16 = 0; s16 < 8; ++s16) {
        const int cbase = col0 + s16 * 16;
        if (cbase >= p.G) break;                 // warp-uniform
        auto out4 = [&](int k) {                 // outputs 4k .. 4k+3 of this 16-column group
          const int i = s16 * 16 + 4 * k;
          float o[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float base = __fadd_rn(rq_row, col_rg[i + j]);
            o[j] = __fmaf_rn(coef_row * col_sg[i + j], r[i + j], base);
            viol = fminf(viol, __fmaf_rn(-p.fix_tau, base, o[j]));    // < 0: a near-duplicate pair (see below)
          }
          return make_float4(o[0], o[1], o[2], o[3]);
        };
        if (p.tma_store) {
          if (lane == 0) tma_store_wait_read<0>();
          __syncwarp();
          // 32 rows x 64 bytes, SWIZZLE_64B: 16-byte chunk k of row r lives at chunk k ^ ((r >> 1) & 3)
#pragma unroll
          for (int k = 0; k < 4; ++k)
            *reinterpret_cast<float4*>(reinterpret_cast<uint8_t*>(tile) + lane * 64 + ((k ^ ((lane >> 1) & 3)) << 4)) = out4(k);
          fence_proxy_async();
          __syncwarp();
          if (lane == 0) {
            tma_store_2d(&tm_out, tile, cbase, row0);
            tma_store_commit();
          }
        } else {
          __syncwarp();
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const float4 o = out4(k);
            tile[lane * kPitchC + 4 * k] = o.x;
            tile[lane * kPitchC + 4 * k + 1] = o.y;
            tile[lane * kPitchC + 4 * k + 2] = o.z;
            tile[lane * kPitchC + 4 * k + 3] = o.w;
          }
          __syncwarp();
          const int cl = lane & 15, rh = lane >> 4;          // 2 rows x 16 columns per instruction
#pragma unroll 4
          for (int rr = 0; rr < 32; rr += 2) {
            const int row = row0 + rr + rh, col = cbase + cl;
            if (row < p.Q && col < p.G) p.out[(int64_t)row * p.ldo + col] = tile[(rr + rh) * kPitchC + cl];
          }
        }
      }
      // Near-duplicate pairs: almost all of |q|^2 + |g|^2 cancels, and what the truncating accumulator lost in the
      // all-positive products is no longer small against d.  Rare: the (row, 128-column span) goes on a list and
      // distmat_fixup_kernel recomputes the outputs below the bound in difference form.
      if (fix_on && viol < 0.f && my_row < p.Q) {
        const unsigned long long slot = atomicAdd(p.fix_list, 1ull);
        if (slot < p.fix_cap) p.fix_list[1 + slot] = ((unsigned long long)(uint32_t)my_row << 32) | (uint32_t)col0;
      }
    }
    if (p.tma_store && lane == 0) tma_store_wait<0>();
    __syncwarp();
  }

  tc_fence_before();
  if constexpr (CG == 2) cluster_sync_all(); else __syncthreads();
  if (warp == 2) tmem_dealloc<CG>(tmem_base, 512);
}

// =====================================================================================================
// Near-duplicate fix-up.  For a pair with |q - g|^2 << |q|^2 + |g|^2 the expansion |q|^2 + |g|^2 - 2 q.g keeps only
// the absolute accuracy of its terms (the reference's fp32 GEMM has the same problem, distance.py:59-64: self
// distances of +-3e-7 (|q|^2 + |g|^2)).  The chunked kernel lists the (row, 128-column span)s in which it saw an output
// below fix_tau of its scale; one warp per entry re-reads that span of the block and recomputes every output below the
// bound as sum_k (q_k - g_k)^2 from the packed planes -- exact operands (hi + lo is the packed value), fp32 FMA chain,
// relative error ~1e-7 of d itself.
// The list holds `cap` entries.  A block with more flagged spans (duplicates scattered through the gallery, or centring
// switched off on a large block) counts past it: then the warps walk every (row, span) of the block instead and apply
// the same re-test, so the same outputs are recomputed, bit for bit, at the cost of one more read of the block.
// =====================================================================================================
__global__ void __launch_bounds__(256) distmat_fixup_kernel(const __half* __restrict__ q_hi, const __half* __restrict__ q_lo,
                                                             const __half* __restrict__ g_hi, const __half* __restrict__ g_lo,
                                                             const float* __restrict__ sq, const float* __restrict__ sg,
                                                             const float* __restrict__ rq, const float* __restrict__ rg, int Dp,
                                                             int Q, int G, float tau, const unsigned long long* __restrict__ list,
                                                             uint32_t cap, float* __restrict__ out, int64_t ldo) {
  const unsigned long long n64 = list[0];
  const bool overflow = n64 > cap;
  const unsigned long long spans = (unsigned long long)((G + 127) / 128);
  const unsigned long long n = overflow ? (unsigned long long)Q * spans : n64;
  const int lane = threadIdx.x & 31;
  const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
  for (unsigned long long e = warp; e < n; e += nwarps) {
    // entry = (row, first column of a 128-column span) in which the contraction saw an output below the bound
    uint32_t row, col0;
    if (overflow) {
      row = (uint32_t)(e / spans);
      col0 = (uint32_t)(e - row * spans) * 128u;
    } else {
      const unsigned long long rc = list[1 + e];
      row = (uint32_t)(rc >> 32);
      col0 = (uint32_t)rc;
    }
    const float a_s = sq[row], a_n = rq[row];
    const uint4* ah = reinterpret_cast<const uint4*>(q_hi + (size_t)row * Dp);
    const uint4* al = reinterpret_cast<const uint4*>(q_lo + (size_t)row * Dp);
    for (int j0 = 0; j0 < 128; j0 += 32) {
      const int colj = (int)col0 + j0 + lane;
      bool hit = false;
      if (colj < G) hit = out[(int64_t)row * ldo + colj] < tau * __fadd_rn(a_n, rg[colj]);
      unsigned todo = __ballot_sync(0xffffffffu, hit);
      while (todo) {
        const int b = __ffs(todo) - 1;
        todo &= todo - 1;
        const uint32_t col = col0 + j0 + b;
        const float b_s = sg[col];
        const uint4* bh = reinterpret_cast<const uint4*>(g_hi + (size_t)col * Dp);
        const uint4* bl = reinterpret_cast<const uint4*>(g_lo + (size_t)col * Dp);
        float acc = 0.f;
        for (int i = lane; i < Dp / 8; i += 32) {      // 8 halves per 16-byte load
          const uint4 x0 = ah[i], x1 = al[i], y0 = bh[i], y1 = bl[i];
          const __half2* xh = reinterpret_cast<const __half2*>(&x0);
          const __half2* xl = reinterpret_cast<const __half2*>(&x1);
          const __half2* yh = reinterpret_cast<const __half2*>(&y0);
          const __half2* yl = reinterpret_cast<const __half2*>(&y1);
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float2 a_hi = __half22float2(xh[j]), a_lo = __half22float2(xl[j]);
            const float2 b_hi = __half22float2(yh[j]), b_lo = __half22float2(yl[j]);
            const float d0 = __fsub_rn(__fadd_rn(a_hi.x, a_lo.x) * a_s, __fadd_rn(b_hi.x, b_lo.x) * b_s);
            const float d1 = __fsub_rn(__fadd_rn(a_hi.y, a_lo.y) * a_s, __fadd_rn(b_hi.y, b_lo.y) * b_s);
            acc = __fmaf_rn(d0, d0, acc);
            acc = __fmaf_rn(d1, d1, acc);
          }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (lane == 0) out[(int64_t)row * ldo + col] = acc;
      }
    }
  }
}

// ---- host side --------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn) return fn;
  void* sym = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres) != cudaSuccess ||
      qres != cudaDriverEntryPointSuccess)
    return nullptr;
  fn = reinterpret_cast<EncodeTiledFn>(sym);
  return fn;
}

// row-major [rows, cols] matrix of `esize`-byte elements -> tiles of box_rows x box_cols, 128-byte swizzle
// (box_cols * esize == swizzle span), zero fill / clipping out of bounds.
static int make_tmap(CUtensorMap* tm, CUtensorMapDataType dt, int esize, const void* base, int64_t rows, int64_t cols,
                     int64_t pitch_elems, int box_rows, int box_cols, CUtensorMapSwizzle swz = CU_TENSOR_MAP_SWIZZLE_128B) {
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) {
    set_error("cuTensorMapEncodeTiled not available from the driver");
    return IEEE_ERR_CUDA;
  }
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)pitch_elems * esize};
  cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(tm, dt, 2, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed with CUresult %d (rows=%lld cols=%lld pitch=%lld)", (int)r, (long long)rows,
              (long long)cols, (long long)pitch_elems);
    return IEEE_ERR_CUDA;
  }
  return IEEE_OK;
}

// Operand tensor maps, epilogue terms and tile raster shared by both kernels.
struct GemmLaunch {
  CUtensorMap ta_hi, ta_lo, tb_hi, tb_lo, t_out;
  GemmParams p;
  int groups;
};

template <int CG>
static int gemm_setup(GemmLaunch& L, const PackedRows& a, const PackedRows& b, int metric, int precision, float* out,
                      int64_t ldo, int out_box_cols, CUtensorMapSwizzle out_swizzle) {
  constexpr int kBRows = BLOCK_N / CG;
  const int64_t Q = a.rows, G = b.rows;
  const CUtensorMapDataType dt16 = CU_TENSOR_MAP_DATA_TYPE_UINT16;   // the copy engine only moves 16-bit words
  int rc;
  if ((rc = make_tmap(&L.ta_hi, dt16, 2, a.hi, Q, a.Dp, a.Dp, BLOCK_M, BLOCK_K))) return rc;
  if ((rc = make_tmap(&L.tb_hi, dt16, 2, b.hi, G, b.Dp, b.Dp, kBRows, BLOCK_K))) return rc;
  if (precision == IEEE_PREC_F16X3) {
    if ((rc = make_tmap(&L.ta_lo, dt16, 2, a.lo, Q, a.Dp, a.Dp, BLOCK_M, BLOCK_K))) return rc;
    if ((rc = make_tmap(&L.tb_lo, dt16, 2, b.lo, G, b.Dp, b.Dp, kBRows, BLOCK_K))) return rc;
  } else {
    L.ta_lo = L.ta_hi;
    L.tb_lo = L.tb_hi;
  }
  GemmParams& p = L.p;
  const bool euclid = metric == IEEE_METRIC_EUCLIDEAN;
  p.rq = euclid ? a.norm : nullptr;
  p.rg = euclid ? b.norm : nullptr;
  p.sq = precision == IEEE_PREC_F16X3 ? a.scale : nullptr;
  p.sg = precision == IEEE_PREC_F16X3 ? b.scale : nullptr;
  p.alpha = euclid ? -2.0f : -1.0f;
  p.base0 = metric == IEEE_METRIC_NEG_DOT ? 0.0f : 1.0f;
  p.out = out;
  p.ldo = ldo;
  p.Q = (int)Q;
  p.G = (int)G;
  p.num_kb = (int)(a.Dp / BLOCK_K);
  p.nseg = precision == IEEE_PREC_F16X3 ? 3 : 1;
  p.num_m_tiles = (int)((Q + BLOCK_M * CG - 1) / (BLOCK_M * CG));
  p.num_n_tiles = (int)((G + BLOCK_N - 1) / BLOCK_N);
  // raster panel: as many m tiles as keep the panel's A planes within ~40 MB of the 126 MB L2
  const double a_tile_bytes = double(BLOCK_M * CG) * double(a.Dp) * 2.0 * (precision == IEEE_PREC_F16X3 ? 2.0 : 1.0);
  int panel = (int)(40.0 * 1024 * 1024 / a_tile_bytes);
  if (g_raster_panel > 0) panel = g_raster_panel;
  p.panel_m = panel < 1 ? 1 : (panel > p.num_m_tiles ? p.num_m_tiles : panel);
  p.idesc = umma_idesc_16bit(BLOCK_M * CG, BLOCK_N, precision == IEEE_PREC_F16X3 ? 0u : 1u);
  p.debug = g_debug_flags;
  p.fix_list = nullptr;
  p.fix_cap = 0;
  p.fix_tau = 0.f;
  p.tma_store = ((reinterpret_cast<uintptr_t>(out) & 15) == 0 && (ldo % 4) == 0 && !(g_debug_flags & 4)) ? 1 : 0;
  if (p.tma_store) {
    if ((rc = make_tmap(&L.t_out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, out, Q, G, ldo, 32, out_box_cols, out_swizzle))) return rc;
  } else {
    L.t_out = L.ta_hi;
  }
  const int num_tiles = p.num_m_tiles * p.num_n_tiles;
  L.groups = sm_count() / CG;
  if (L.groups > num_tiles) L.groups = num_tiles;
  return IEEE_OK;
}

static void cluster_launch_config(cudaLaunchConfig_t& cfg, cudaLaunchAttribute* attr, int grid, int threads, size_t smem,
                                  int cluster, cudaStream_t stream) {
  cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(threads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = cluster;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
}

template <int CG>
static int launch_umma(const PackedRows& a, const PackedRows& b, int metric, int precision, float* out, int64_t ldo,
                       cudaStream_t stream) {
  using Cfg = GemmCfg<CG>;
  GemmLaunch L;
  int rc = gemm_setup<CG>(L, a, b, metric, precision, out, ldo, 32, CU_TENSOR_MAP_SWIZZLE_128B);
  if (rc) return rc;
  IEEE_ENSURE_DYN_SMEM(distmat_umma_kernel<CG>, Cfg::kSmemBytes);
  cudaLaunchConfig_t cfg;
  cudaLaunchAttribute attr[1];
  cluster_launch_config(cfg, attr, L.groups * CG, kThreads, Cfg::kSmemBytes, CG, stream);
  IEEE_CUDA_CHECK(cudaLaunchKernelEx(&cfg, distmat_umma_kernel<CG>, L.ta_hi, L.ta_lo, L.tb_hi, L.tb_lo, L.t_out, L.p));
  count_launch(1, "distmat_umma_kernel");
  return IEEE_OK;
}

// pairs below 2^-6 of their scale are recomputed: above it, what the accumulator can lose (<= ~1.3e-6 of the scale
// at the default chunking, all-positive products) stays under 1e-4 of the distance itself
constexpr float kFixTau = 0.015625f;

size_t distmat_fixup_bytes(int64_t Q) { return align256((size_t(2 * Q + 4096) + 2) * 8); }

template <int CG>
static int launch_umma_chunked(const PackedRows& a, const PackedRows& b, int metric, int precision, float* out, int64_t ldo,
                               cudaStream_t stream, int chunk_kb, void* fix_ws, bool fix_zeroed) {
  using Cfg = GemmCfgC<CG>;
  GemmLaunch L;
  const int64_t Q = a.rows, G = b.rows;
  int rc = gemm_setup<CG>(L, a, b, metric, precision, out, ldo, 16, CU_TENSOR_MAP_SWIZZLE_64B);
  if (rc) return rc;
  const bool fix = fix_ws != nullptr && metric == IEEE_METRIC_EUCLIDEAN && precision == IEEE_PREC_F16X3 &&
                   !(g_debug_flags & 32);
  if (fix) {
    L.p.fix_list = static_cast<unsigned long long*>(fix_ws);
    L.p.fix_cap = (uint32_t)(2 * Q + 4096);
    L.p.fix_tau = kFixTau;
    if (!fix_zeroed) {      // (the one-call entry points have an earlier kernel clear the list header)
      IEEE_CUDA_CHECK(cudaMemsetAsync(fix_ws, 0, 8, stream));
      count_launch(0, "memset fix list");
    }
  }
  IEEE_ENSURE_DYN_SMEM(distmat_umma_chunked_kernel<CG>, Cfg::kSmemBytes);
  cudaLaunchConfig_t cfg;
  cudaLaunchAttribute attr[1];
  cluster_launch_config(cfg, attr, L.groups * CG, kThreadsC, Cfg::kSmemBytes, CG, stream);
  IEEE_CUDA_CHECK(cudaLaunchKernelEx(&cfg, distmat_umma_chunked_kernel<CG>, L.ta_hi, L.ta_lo, L.tb_hi, L.tb_lo, L.t_out, L.p,
                                     chunk_kb));
  count_launch(1, "distmat_umma_chunked_kernel");
  if (fix) {
    distmat_fixup_kernel<<<sm_count(), 256, 0, stream>>>(
        reinterpret_cast<const __half*>(a.hi), reinterpret_cast<const __half*>(a.lo), reinterpret_cast<const __half*>(b.hi),
        reinterpret_cast<const __half*>(b.lo), a.scale, b.scale, a.norm, b.norm, (int)a.Dp, (int)Q, (int)G, kFixTau,
        L.p.fix_list, L.p.fix_cap, out, ldo);
    count_launch(1, "distmat_fixup_kernel");
    IEEE_CUDA_CHECK(cudaGetLastError());
  }
  return IEEE_OK;
}

int distmat_umma_rows(const PackedRows& a, const PackedRows& b, int metric, int precision, float* out, int64_t ldo,
                      cudaStream_t stream, int cta_group, void* fix_ws, bool fix_zeroed) {
  // chunked accumulation serves the fp32-grade mode; the 1-pass BF16 mode keeps the whole K in TMEM (throughput mode)
  if (g_accum_chunk_kb > 0 && (precision == IEEE_PREC_F16X3 || (g_debug_flags & 8))) {
    if (cta_group == 2)
      return launch_umma_chunked<2>(a, b, metric, precision, out, ldo, stream, g_accum_chunk_kb, fix_ws, fix_zeroed);
    return launch_umma_chunked<1>(a, b, metric, precision, out, ldo, stream, g_accum_chunk_kb, fix_ws, fix_zeroed);
  }
  if (cta_group == 2) return launch_umma<2>(a, b, metric, precision, out, ldo, stream);
  return launch_umma<1>(a, b, metric, precision, out, ldo, stream);
}

int distmat_umma(const void* q_packed, int64_t Q, const void* g_packed, int64_t G, int64_t D, int metric, int precision,
                 float* out, int64_t ldo, cudaStream_t stream, int cta_group, void* fix_ws, bool fix_zeroed) {
  return distmat_umma_rows(packed_rows(q_packed, Q, 0, Q, D, precision), packed_rows(g_packed, G, 0, G, D, precision), metric,
                           precision, out, ldo, stream, cta_group, fix_ws, fix_zeroed);
}

}  // namespace ieee
