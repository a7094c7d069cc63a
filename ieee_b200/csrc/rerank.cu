// k-reciprocal re-ranking (Zhong et al., CVPR 2017) -- replaces torchreid/utils/rerank.py:31-113.
//
// Stages (SURVEY.md section 8a, K1-K6), N = Q + G:
//   K1  original_dist[i][j] = raw[j][i]^2 / max_k raw[k][i]^2 over the virtual block matrix
//       raw = [[qq, qg], [qg^T, gg]] (rerank.py:36-46: squared again, column-normalised, transposed)
//   K2  initial_rank = first k1+1 entries of each row's ascending order (rerank.py:48; only those prefixes are read)
//   K3  k-reciprocal sets + half-k expansion + Gaussian weights -> row-sparse V (rerank.py:54-82)
//   K4  query expansion: V_qe[i] = mean of the k2 rows V[initial_rank[i, :k2]] (rerank.py:84-89), still sparse
//   K5  Jaccard distance through the inverted index (rerank.py:91-106), accumulated in ascending column order
//   K6  final = jaccard * (1 - lambda) + original_dist * lambda, rows < Q, columns >= Q (rerank.py:108-113)
// V never exists densely: rows hold at most (k1+1)(round(k1/2)+2) entries, expanded rows k2 times that.
// Ties in K2 are broken by index (the reference's unstable argsort leaves them undefined).
#include "common.cuh"

namespace ieee {

int topk(const float* distmat, int64_t ld, int64_t Q, int64_t G, int64_t g_offset, const int64_t* q_pids,
         const int64_t* q_camids, const int64_t* g_pids, const int64_t* g_camids, int32_t k, int32_t* idx, float* val,
         cudaStream_t stream);

struct RawView {            // the virtual N x N matrix [[qq, qg], [qg^T, gg]]
  const float *qg, *qq, *gg;
  int64_t ld_qg, ld_qq, ld_gg;
  int Q, G;
  __device__ __forceinline__ float at(int r, int c) const {
    if (r < Q) return c < Q ? qq[(int64_t)r * ld_qq + c] : qg[(int64_t)r * ld_qg + (c - Q)];
    return c < Q ? qg[(int64_t)c * ld_qg + (r - Q)] : gg[(int64_t)(r - Q) * ld_gg + (c - Q)];
  }
  // the 32 x 32 tile raw[r0.., c0..] is contiguous in r (the qg^T block: r >= Q, c < Q)
  __device__ __forceinline__ bool contiguous_in_r(int r0, int c0) const { return r0 >= Q && c0 + 31 < Q; }
};

// Columns [c0, c0 + w) of the virtual matrix (a strip, c0 and w counted in the queries or in the gallery, never both),
// held as the two contraction outputs that make them up; `at(r, t)` is raw[r][c0 + t].
//   top: raw rows < Q,  [Q, w]  -- qq[:, I] (A = all queries, B = q_I) or qg[:, I - Q] (A = all queries, B = g_I)
//   bot: raw rows >= Q, [w, G] when the strip lies in the queries -- qg[I, :] (A = q_I, B = all gallery), row t =
//        strip column t -- else [G, w] -- gg[:, I - Q] (A = all gallery, B = g_I)
struct StripView {
  const float *top, *bot;
  int64_t ld_top, ld_bot;
  int Q;
  bool bot_by_row;
  __device__ __forceinline__ float at(int r, int t) const {
    if (r < Q) return top[(int64_t)r * ld_top + t];
    return bot_by_row ? bot[(int64_t)t * ld_bot + (r - Q)] : bot[(int64_t)(r - Q) * ld_bot + t];
  }
  __device__ __forceinline__ bool contiguous_in_r(int r0, int) const { return bot_by_row && r0 >= Q; }
};

// ---- K1a: column maxima of raw^2 ------------------------------------------------------------------------
// values are squares (>= 0), so the float order equals the order of their bit patterns: integer atomicMax.
__global__ void __launch_bounds__(256) rr_colmax_kernel(const float* __restrict__ m, int64_t ld, int rows, int cols,
                                                         int rows_per_block, int* __restrict__ colmax_bits) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= cols) return;
  const int r0 = blockIdx.y * rows_per_block, r1 = min(rows, r0 + rows_per_block);
  float mx = 0.f;
  for (int r = r0; r < r1; ++r) {
    const float x = m[(int64_t)r * ld + c];
    mx = fmaxf(mx, __fmul_rn(x, x));
  }
  atomicMax(colmax_bits + c, __float_as_int(mx));
}
// maxima over the ROWS of qg: the qg^T block's contribution to columns < Q
__global__ void __launch_bounds__(256) rr_rowmax_kernel(const float* __restrict__ m, int64_t ld, int rows, int cols,
                                                         int* __restrict__ colmax_bits) {
  const int r = blockIdx.x;
  float mx = 0.f;
  for (int c = threadIdx.x; c < cols; c += blockDim.x) {
    const float x = m[(int64_t)r * ld + c];
    mx = fmaxf(mx, __fmul_rn(x, x));
  }
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if ((threadIdx.x & 31) == 0) atomicMax(colmax_bits + r, __float_as_int(mx));
}

// ---- K1b: orig[i][j] = raw[j][i]^2 / colmax[i], i < rows, j < N; 32 x 32 tiles transposed through shared memory ----
// View = RawView (all N rows of orig) or StripView (the rows of one strip, colmax and orig offset to its first row)
template <class View>
__global__ void __launch_bounds__(256) rr_build_orig_kernel(View raw, int rows, int N, const float* __restrict__ colmax,
                                                             float* __restrict__ orig, int64_t ldo) {
  __shared__ float tile[32][33];
  const int i0 = blockIdx.y * 32, j0 = blockIdx.x * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;   // 32 x 8
  // raw[j][i] is contiguous in i except where the view says it is contiguous in j
  if (raw.contiguous_in_r(j0, i0)) {
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int i = i0 + ty + 8 * k, j = j0 + tx;
      if (i < rows && j < N) {
        const float x = raw.at(j, i);
        orig[(int64_t)i * ldo + j] = __fdiv_rn(__fmul_rn(x, x), colmax[i]);
      }
    }
    return;
  }
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int j = j0 + ty + 8 * k, i = i0 + tx;
    tile[ty + 8 * k][tx] = (i < rows && j < N) ? raw.at(j, i) : 0.f;
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int i = i0 + ty + 8 * k, j = j0 + tx;
    if (i < rows && j < N) {
      const float x = tile[tx][ty + 8 * k];
      orig[(int64_t)i * ldo + j] = __fdiv_rn(__fmul_rn(x, x), colmax[i]);
    }
  }
}

// ---- K3: k-reciprocal sets, expansion, weights; one warp per row ----------------------------------------
constexpr int kRowWarps = 4;

// members of `row`'s first kk neighbours whose own first kk neighbours contain `row` (rerank.py:56-59, :63-71),
// appended to `out` (shared memory) in neighbour order; returns the new count.
__device__ int reciprocal_append(const int32_t* __restrict__ rank, int ldr, int row, int kk, int lane, int* out, int n_out) {
  for (int t0 = 0; t0 < kk; t0 += 32) {
    const int t = t0 + lane;
    bool ok = false;
    int mine = -1;
    if (t < kk) {
      mine = rank[(int64_t)row * ldr + t];
      if (mine >= 0) {
        const int32_t* back = rank + (int64_t)mine * ldr;
        for (int u = 0; u < kk; ++u) ok |= (back[u] == row);
      }
    }
    const unsigned m = __ballot_sync(0xffffffffu, ok);
    if (ok) out[n_out + __popc(m & ((1u << lane) - 1))] = mine;
    n_out += __popc(m);
  }
  __syncwarp();
  return n_out;
}

// weights of one row of V (rerank.py:81-82): exp(-orig[i, members]) / sum, summed in ascending member order;
// orig_row is row i of orig (the N x N matrix, or the row as one strip holds it)
__device__ void rr_weights(const float* __restrict__ orig_row, const int32_t* __restrict__ cols, float* __restrict__ vals,
                           int nu, int lane) {
  for (int t = lane; t < nu; t += 32) vals[t] = expf(-orig_row[cols[t]]);
  __syncwarp();
  float total = 0.f;
  if (lane == 0)
    for (int t = 0; t < nu; ++t) total = __fadd_rn(total, vals[t]);
  total = __shfl_sync(0xffffffffu, total, 0);
  for (int t = lane; t < nu; t += 32) vals[t] = __fdiv_rn(vals[t], total);
}

// kWeights: also weigh the members from orig (N x N).  Without it only the membership (columns, counts) is written,
// from `rank` alone, and rr_weights_kernel weighs the rows strip by strip.
template <bool kWeights>
__global__ void __launch_bounds__(32 * kRowWarps)
rr_krecip_kernel(const int32_t* __restrict__ rank, int ldr, const float* __restrict__ orig, int N, int k1p, int khp, int cap_v,
                 int cap_pow2, int32_t* __restrict__ v_col, float* __restrict__ v_val, int32_t* __restrict__ v_cnt) {
  extern __shared__ __align__(16) uint8_t kr_raw[];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  int* base_set = reinterpret_cast<int*>(kr_raw) + w * (k1p + khp + cap_pow2);   // R(i), up to k1p
  int* cand_set = base_set + k1p;                                                 // R_half(c), up to khp
  int* members = cand_set + khp;                                                  // expansion list, cap_pow2
  const int i = blockIdx.x * kRowWarps + w;
  if (i >= N) return;
  // R(i)
  const int nb = reciprocal_append(rank, ldr, i, k1p, lane, base_set, 0);
  for (int t = lane; t < nb; t += 32) members[t] = base_set[t];
  int nm = nb;
  __syncwarp();
  // expansion (rerank.py:61-78): candidates in R(i) order; the overlap test is against the UN-expanded R(i)
  for (int j = 0; j < nb; ++j) {
    const int c = base_set[j];
    const int nc = reciprocal_append(rank, ldr, c, khp, lane, cand_set, 0);
    int inter = 0;
    for (int t = lane; t < nc; t += 32) {
      const int x = cand_set[t];
      bool hit = false;
      for (int u = 0; u < nb; ++u) hit |= (base_set[u] == x);
      inter += hit;
    }
    for (int o = 16; o > 0; o >>= 1) inter += __shfl_xor_sync(0xffffffffu, inter, o);
    if (3 * inter > 2 * nc) {          // len(intersect) > 2/3 * len(candidate set), strict
      for (int t = lane; t < nc; t += 32) members[nm + t] = cand_set[t];
      nm += nc;
    }
    __syncwarp();
  }
  // np.unique: sort ascending, drop duplicates (warp bitonic sort in shared memory)
  for (int t = nm + lane; t < cap_pow2; t += 32) members[t] = INT32_MAX;
  __syncwarp();
  for (int k = 2; k <= cap_pow2; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int t = lane; t < cap_pow2; t += 32) {
        const int p = t ^ j;
        if (p > t) {
          const int a = members[t], b = members[p];
          if ((a > b) == ((t & k) == 0)) { members[t] = b; members[p] = a; }
        }
      }
      __syncwarp();
    }
  }
  int nu = 0;
  for (int t0 = 0; t0 < nm; t0 += 32) {
    const int t = t0 + lane;
    const bool keep = t < nm && (t == 0 || members[t] != members[t - 1]);
    const int val = t < nm ? members[t] : 0;
    const unsigned m = __ballot_sync(0xffffffffu, keep);
    __syncwarp();
    if (keep) v_col[(int64_t)i * cap_v + nu + __popc(m & ((1u << lane) - 1))] = val;
    nu += __popc(m);
  }
  __syncwarp();
  if constexpr (kWeights) rr_weights(orig + (int64_t)i * N, v_col + (int64_t)i * cap_v, v_val + (int64_t)i * cap_v, nu, lane);
  if (lane == 0) v_cnt[i] = nu;
}

// weights of rows [row0, row0 + rows) of V from one strip of orig (row t of the strip = row row0 + t of orig)
__global__ void __launch_bounds__(32 * kRowWarps)
rr_weights_kernel(const float* __restrict__ orig, int64_t ldo, int row0, int rows, int cap_v, const int32_t* __restrict__ v_col,
                  float* __restrict__ v_val, const int32_t* __restrict__ v_cnt) {
  const int lane = threadIdx.x & 31, t = blockIdx.x * kRowWarps + (threadIdx.x >> 5);
  if (t >= rows) return;
  const int i = row0 + t;
  rr_weights(orig + (int64_t)t * ldo, v_col + (int64_t)i * cap_v, v_val + (int64_t)i * cap_v, v_cnt[i], lane);
}

// Rows of a gallery window: the Q query rows, then the gallery rows [Q + g0, Q + g0 + Gs).  Window row m is sample
// m < Q ? m : m + g0; with g0 = 0 and Gs = G the window is every sample.
__device__ __forceinline__ int window_sample(int m, int Q, int g0) { return m < Q ? m : m + g0; }

// ---- K4: V_qe[m] = mean_j V[rank[i][j]], j < k2, i the sample of window row m; one CTA per window row ------------
__device__ __forceinline__ void block_sort_u64(uint64_t* s, int n) {
  for (int k = 2; k <= n; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      __syncthreads();
      for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const int p = i ^ j;
        if (p > i) {
          const uint64_t a = s[i], b = s[p];
          if ((a > b) == ((i & k) == 0)) { s[i] = b; s[p] = a; }
        }
      }
    }
  }
  __syncthreads();
}

__global__ void __launch_bounds__(256)
rr_expand_kernel(const int32_t* __restrict__ rank, int ldr, int Q, int g0, int k2, int cap_v, const int32_t* __restrict__ v_col,
                 const float* __restrict__ v_val, const int32_t* __restrict__ v_cnt, int cap_e, int cap_e_pow2,
                 int32_t* __restrict__ e_col, float* __restrict__ e_val, int32_t* __restrict__ e_cnt) {
  extern __shared__ __align__(16) uint8_t ex_raw[];
  uint64_t* keys = reinterpret_cast<uint64_t*>(ex_raw);                  // (col * k2 + j) << 32 | float bits
  __shared__ int n_items, n_out;
  const int i = blockIdx.x;                                              // output row (window row)
  const int sample = window_sample(i, Q, g0);
  if (threadIdx.x == 0) { n_items = 0; n_out = 0; }
  __syncthreads();
  for (int j = 0; j < k2; ++j) {
    const int r = rank[(int64_t)sample * ldr + j];
    if (r < 0) continue;
    const int n = v_cnt[r];
    __shared__ int base;
    if (threadIdx.x == 0) { base = n_items; n_items += n; }
    __syncthreads();
    for (int t = threadIdx.x; t < n; t += blockDim.x) {
      const uint32_t c = (uint32_t)v_col[(int64_t)r * cap_v + t];
      keys[base + t] = (uint64_t(c * (uint32_t)k2 + (uint32_t)j) << 32) | __float_as_uint(v_val[(int64_t)r * cap_v + t]);
    }
    __syncthreads();
  }
  const int n = n_items;
  for (int t = n + threadIdx.x; t < cap_e_pow2; t += blockDim.x) keys[t] = ~uint64_t(0);
  block_sort_u64(keys, cap_e_pow2);
  // segment heads: first entry of each column; each head sums its column's entries in j order (np.add.reduce over
  // the k2 rows, rerank.py:87) and divides by k2 (np.mean)
  for (int t0 = 0; t0 < n; t0 += blockDim.x) {
    const int t = t0 + threadIdx.x;
    bool head = false;
    uint32_t col = 0;
    float sum = 0.f;
    if (t < n) {
      col = (uint32_t)(keys[t] >> 32) / (uint32_t)k2;
      head = (t == 0) || ((uint32_t)(keys[t - 1] >> 32) / (uint32_t)k2 != col);
      if (head) {
        for (int u = t; u < n && (uint32_t)(keys[u] >> 32) / (uint32_t)k2 == col; ++u)
          sum = __fadd_rn(sum, __uint_as_float((uint32_t)keys[u]));
        sum = __fdiv_rn(sum, (float)k2);
      }
    }
    // ordered compaction of the heads
    const unsigned m = __ballot_sync(0xffffffffu, head);
    __shared__ int warp_cnt[8];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    if (lane == 0) warp_cnt[w] = __popc(m);
    __syncthreads();
    int off = n_out;
    for (int x = 0; x < w; ++x) off += warp_cnt[x];
    if (head) {
      const int pos = off + __popc(m & ((1u << lane) - 1));
      e_col[(int64_t)i * cap_e + pos] = (int32_t)col;
      e_val[(int64_t)i * cap_e + pos] = sum;
    }
    __syncthreads();
    if (threadIdx.x == 0) { int tot = 0; for (int x = 0; x < 8; ++x) tot += warp_cnt[x]; n_out += tot; }
    __syncthreads();
  }
  if (threadIdx.x == 0) e_cnt[i] = n_out;
}

// ---- K5a: inverted index (CSC of the row-sparse matrix), zero values excluded (rerank.py:93: V[:, i] != 0) ----
// One CTA per window row r; its entries are read from row window_sample(r, Q, shift) of the row-sparse matrix (shift =
// g0 when that matrix is V, indexed by sample; 0 when it is V_qe, already indexed by window row) and listed as row r.
__global__ void rr_col_count_kernel(int Q, int shift, int cap, const int32_t* __restrict__ col, const float* __restrict__ val,
                                    const int32_t* __restrict__ cnt, int32_t* __restrict__ col_count) {
  const int r = window_sample(blockIdx.x, Q, shift);
  const int n = cnt[r];
  for (int t = threadIdx.x; t < n; t += blockDim.x)
    if (val[(int64_t)r * cap + t] != 0.f) atomicAdd(col_count + col[(int64_t)r * cap + t], 1);
}
// exclusive scan of col_count[N] -> col_ptr[N + 1]; single CTA
__global__ void __launch_bounds__(1024) rr_scan_kernel(const int32_t* __restrict__ in, int N, int32_t* __restrict__ out) {
  __shared__ int wsum[32];
  __shared__ int carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (int base = 0; base < N; base += 1024) {
    const int i = base + threadIdx.x;
    const int v = i < N ? in[i] : 0;
    int incl = v;
    for (int o = 1; o < 32; o <<= 1) { int n = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += n; }
    if (lane == 31) wsum[w] = incl;
    __syncthreads();
    int off = carry;
    for (int x = 0; x < w; ++x) off += wsum[x];
    if (i < N) out[i] = off + incl - v;
    __syncthreads();
    if (threadIdx.x == 1023) carry = off + incl;
    __syncthreads();
  }
  if (threadIdx.x == 0) out[N] = carry;
}
__global__ void rr_col_fill_kernel(int Q, int shift, int cap, const int32_t* __restrict__ col, const float* __restrict__ val,
                                   const int32_t* __restrict__ cnt, const int32_t* __restrict__ col_ptr,
                                   int32_t* __restrict__ cursor, int32_t* __restrict__ inv_row, float* __restrict__ inv_val) {
  const int r = window_sample(blockIdx.x, Q, shift);
  const int n = cnt[r];
  for (int t = threadIdx.x; t < n; t += blockDim.x) {
    const float v = val[(int64_t)r * cap + t];
    if (v == 0.f) continue;
    const int c = col[(int64_t)r * cap + t];
    const int pos = col_ptr[c] + atomicAdd(cursor + c, 1);
    inv_row[pos] = blockIdx.x;
    inv_val[pos] = v;
  }
}

// ---- K5b + K6: Jaccard accumulation for one query per CTA, then the lambda blend ----------------------------
// Query i = row0 + blockIdx.x, output row blockIdx.x of `out`.  Dense (kBlock = false): row0 = 0, the output row
// doubles as the accumulator (acc == out) and the original distance is read from orig.  kBlock: `out` holds the
// query's distances to the gallery (qg rows row0..), accumulation goes to `acc`, and the original distance is
// formed from the distance as rr_build_orig_kernel forms it (qg[i][g] = raw[Q + g][i]).
// The inverted index holds the rows of one gallery window (Q query rows, then Gs gallery rows, see window_sample): row
// r >= Q of the index is column r - Q of the window, so acc and out are Gs wide.  Each acc[g] gets at most one add per
// column of row i (rows are distinct inside a column), in the ascending column order, so a window has the bits of the
// same columns of the whole gallery whatever order the index was filled in.
template <bool kBlock>
__global__ void __launch_bounds__(256)
rr_jaccard_kernel(int Q, int Gs, int N, int cap, const int32_t* __restrict__ col, const float* __restrict__ val,
                  const int32_t* __restrict__ cnt, const int32_t* __restrict__ col_ptr, const int32_t* __restrict__ inv_row,
                  const float* __restrict__ inv_val, const float* __restrict__ orig, const float* __restrict__ colmax, int row0,
                  float* acc_rows, int64_t ld_acc, float w_jaccard, float w_orig, float* out, int64_t ldo) {
  const int i = row0 + blockIdx.x;
  float* acc = acc_rows + (int64_t)blockIdx.x * ld_acc;
  float* dst = out + (int64_t)blockIdx.x * ldo;
  for (int g = threadIdx.x; g < Gs; g += blockDim.x) acc[g] = 0.f;
  __syncthreads();
  const int n = cnt[i];
  for (int t = 0; t < n; ++t) {            // ascending column order (rerank.py:99-105)
    const float vi = val[(int64_t)i * cap + t];
    if (vi == 0.f) continue;               // np.where(V[i, :] != 0)
    const int c = col[(int64_t)i * cap + t];
    const int p0 = col_ptr[c], p1 = col_ptr[c + 1];
    for (int p = p0 + threadIdx.x; p < p1; p += blockDim.x) {
      const int r = inv_row[p];
      if (r >= Q) acc[r - Q] = __fadd_rn(acc[r - Q], fminf(vi, inv_val[p]));   // rows are distinct inside a column
    }
    __syncthreads();
  }
  for (int g = threadIdx.x; g < Gs; g += blockDim.x) {
    const float tmin = acc[g];
    const float jac = __fsub_rn(1.0f, __fdiv_rn(tmin, __fsub_rn(2.0f, tmin)));          // rerank.py:106
    float o;
    if constexpr (kBlock) {
      const float x = dst[g];
      o = __fdiv_rn(__fmul_rn(x, x), colmax[i]);
    } else {
      o = orig[(int64_t)i * N + Q + g];
    }
    dst[g] = __fadd_rn(__fmul_rn(jac, w_jaccard), __fmul_rn(o, w_orig));   // :108
  }
}

// ---- host ----------------------------------------------------------------------------------------------------
int distmat_umma_rows(const PackedRows& a, const PackedRows& b, int metric, int precision, float* out, int64_t ldo,
                      cudaStream_t stream, int cta_group, void* fix_ws, bool fix_zeroed);
size_t distmat_fixup_bytes(int64_t Q);

static inline int pow2_at_least(int x) { int p = 1; while (p < x) p <<= 1; return p; }
static inline int half_k(int k1) {          // int(np.around(k1 / 2.)): round half to even
  const double h = k1 / 2.0;
  double r = floor(h + 0.5);
  if (h + 0.5 == r && (static_cast<long long>(r) & 1)) r -= 1.0;
  return (int)r;
}

// Workspace of both forms.  The dense form holds orig (N x N), colmax, rank and the top-k values; the streamed form
// keeps colmax and rank in caller buffers and only the sparse state here (its strips live in a separate scratch, see
// StripPlan), so its offsets depend on (Q, G, k1, k2, Gs) alone.  V holds all N rows; its query expansion and the
// inverted index hold the M = Q + Gs rows of a gallery window (window_sample): the whole gallery when Gs = G.  V comes
// first, so its offsets do not depend on the window.
struct RerankPlan {
  int N, M, k1p, khp, cap_v, cap_v_pow2, cap_e, cap_e_pow2;
  size_t off_orig, off_colmax, off_rank, off_rank_val, off_vcol, off_vval, off_vcnt, v_end, off_ecol, off_eval, off_ecnt,
      off_colcnt, off_colptr, off_cursor, off_invrow, off_invval, total;
};
static RerankPlan make_plan(int64_t Q, int64_t G, int k1, int k2, bool dense, int64_t Gs) {
  RerankPlan p;
  p.N = (int)(Q + G);
  p.M = (int)(Q + Gs);
  p.k1p = k1 + 1;
  p.khp = half_k(k1) + 1;
  p.cap_v = p.k1p * (p.khp + 1);
  p.cap_v_pow2 = pow2_at_least(p.cap_v);
  p.cap_e = (k2 > 1 ? k2 : 1) * p.cap_v;
  p.cap_e_pow2 = pow2_at_least(p.cap_e);
  size_t o = 0;
  auto take = [&](size_t bytes) { size_t r = o; o += align256(bytes); return r; };
  const size_t N = p.N, M = p.M;
  const size_t dn = dense ? N : 0;
  p.off_orig = take(dn * N * 4);
  p.off_colmax = take(dn * 4);
  p.off_rank = take(dn * p.k1p * 4);
  p.off_rank_val = take(dn * p.k1p * 4);
  p.off_vcol = take(N * p.cap_v * 4);
  p.off_vval = take(N * p.cap_v * 4);
  p.off_vcnt = take(N * 4);
  p.v_end = o;
  p.off_ecol = take(k2 > 1 ? M * p.cap_e * 4 : 0);
  p.off_eval = take(k2 > 1 ? M * p.cap_e * 4 : 0);
  p.off_ecnt = take(k2 > 1 ? M * 4 : 0);
  p.off_colcnt = take(N * 4);                 // the index's columns are samples: all N of them
  p.off_colptr = take((N + 1) * 4);
  p.off_cursor = take(N * 4);
  p.off_invrow = take(M * p.cap_e * 4);
  p.off_invval = take(M * p.cap_e * 4);
  p.total = o + 256;
  return p;
}

// the limits both forms share; returns IEEE_OK or sets the error text
static int check_params(const char* who, int64_t Q, int64_t G, int32_t k1, int32_t k2) {
  IEEE_REQUIRE(Q > 0 && G > 0, "%s: bad shape Q=%lld G=%lld", who, (long long)Q, (long long)G);
  IEEE_REQUIRE(Q + G < (int64_t(1) << 24), "%s: N = Q + G too large", who);
  IEEE_REQUIRE(k1 >= 1 && k1 + 1 <= 512 && k2 >= 1 && k2 <= k1 + 1, "%s: need 1 <= k2 <= k1 + 1 <= 512", who);
  IEEE_REQUIRE(k1 + 1 <= Q + G, "%s: k1 + 1 exceeds the number of samples", who);
  const RerankPlan p = make_plan(Q, G, k1, k2, false, G);
  IEEE_REQUIRE((size_t)p.cap_e_pow2 * 8 <= 160 * 1024, "%s: k2 * (k1+1) * (k1/2+2) = %d entries per row exceed the shared-memory sort",
               who, p.cap_e);
  return IEEE_OK;
}

// The V rows the Jaccard stage reads: V_qe (k2 > 1) or V itself.
struct SparseRows {
  const int32_t* col;
  const float* val;
  const int32_t* cnt;
  int cap;
};
static SparseRows final_rows(const RerankPlan& p, uint8_t* w, int k2) {
  if (k2 != 1)
    return {reinterpret_cast<int32_t*>(w + p.off_ecol), reinterpret_cast<float*>(w + p.off_eval),
            reinterpret_cast<int32_t*>(w + p.off_ecnt), p.cap_e};
  return {reinterpret_cast<int32_t*>(w + p.off_vcol), reinterpret_cast<float*>(w + p.off_vval),
          reinterpret_cast<int32_t*>(w + p.off_vcnt), p.cap_v};
}

// K4 + K5a over the rows of the gallery window that starts at gallery row g0: query expansion of V (built by K3) and
// the inverted index of the result
static int expand_and_index(const RerankPlan& p, uint8_t* w, const int32_t* rank, int k2, int64_t Q, int64_t g0,
                            cudaStream_t stream) {
  const int N = p.N, M = p.M;
  int32_t* vcol = reinterpret_cast<int32_t*>(w + p.off_vcol);
  float* vval = reinterpret_cast<float*>(w + p.off_vval);
  int32_t* vcnt = reinterpret_cast<int32_t*>(w + p.off_vcnt);
  int32_t* colcnt = reinterpret_cast<int32_t*>(w + p.off_colcnt);
  int32_t* colptr = reinterpret_cast<int32_t*>(w + p.off_colptr);
  int32_t* cursor = reinterpret_cast<int32_t*>(w + p.off_cursor);
  int32_t* invrow = reinterpret_cast<int32_t*>(w + p.off_invrow);
  float* invval = reinterpret_cast<float*>(w + p.off_invval);
  // K4
  if (k2 != 1) {
    const size_t smem = size_t(p.cap_e_pow2) * 8;
    IEEE_ENSURE_DYN_SMEM(rr_expand_kernel, smem);
    rr_expand_kernel<<<M, 256, smem, stream>>>(rank, p.k1p, (int)Q, (int)g0, k2, p.cap_v, vcol, vval, vcnt, p.cap_e,
                                               p.cap_e_pow2, reinterpret_cast<int32_t*>(w + p.off_ecol),
                                               reinterpret_cast<float*>(w + p.off_eval), reinterpret_cast<int32_t*>(w + p.off_ecnt));
    count_launch();
  }
  const SparseRows f = final_rows(p, w, k2);
  const int shift = k2 != 1 ? 0 : (int)g0;     // V_qe rows are window rows already, V rows are samples
  // K5a
  IEEE_CUDA_CHECK(cudaMemsetAsync(colcnt, 0, size_t(N) * 4, stream));
  IEEE_CUDA_CHECK(cudaMemsetAsync(cursor, 0, size_t(N) * 4, stream));
  rr_col_count_kernel<<<M, 128, 0, stream>>>((int)Q, shift, f.cap, f.col, f.val, f.cnt, colcnt);
  count_launch();
  rr_scan_kernel<<<1, 1024, 0, stream>>>(colcnt, N, colptr);
  count_launch();
  rr_col_fill_kernel<<<M, 128, 0, stream>>>((int)Q, shift, f.cap, f.col, f.val, f.cnt, colptr, cursor, invrow, invval);
  count_launch();
  return IEEE_OK;
}

// K5b + K6 for query rows [row0, row0 + rows) against the window's p.M - Q gallery rows, written to out (leading dim ldo)
template <bool kBlock>
static void launch_jaccard(const RerankPlan& p, uint8_t* w, int64_t Q, int k2, double lambda_value, const float* orig,
                           const float* colmax, int64_t row0, int64_t rows, float* acc, int64_t ld_acc, float* out, int64_t ldo,
                           cudaStream_t stream) {
  const SparseRows f = final_rows(p, w, k2);
  // (1 - lambda) is formed in double and rounded to float32 once, as NumPy does with the Python float
  rr_jaccard_kernel<kBlock><<<(unsigned)rows, 256, 0, stream>>>(
      (int)Q, p.M - (int)Q, p.N, f.cap, f.col, f.val, f.cnt, reinterpret_cast<int32_t*>(w + p.off_colptr),
      reinterpret_cast<int32_t*>(w + p.off_invrow), reinterpret_cast<float*>(w + p.off_invval), orig, colmax, (int)row0, acc,
      ld_acc, (float)(1.0 - lambda_value), (float)lambda_value, out, ldo);
  count_launch();
}

size_t rerank_workspace_bytes(int64_t Q, int64_t G, int32_t k1, int32_t k2) {
  if (Q <= 0 || G <= 0 || k1 < 1 || k2 < 1) return 0;
  return make_plan(Q, G, k1, k2, true, G).total;
}

int rerank(const float* q_g, int64_t ld_qg, const float* q_q, int64_t ld_qq, const float* g_g, int64_t ld_gg, int64_t Q,
           int64_t G, int32_t k1, int32_t k2, double lambda_value, float* out, int64_t ldo, void* workspace,
           size_t workspace_bytes, cudaStream_t stream) {
  IEEE_REQUIRE(q_g && q_q && g_g && out && workspace, "rerank: null pointer");
  IEEE_REQUIRE(Q > 0 && G > 0 && ld_qg >= G && ld_qq >= Q && ld_gg >= G && ldo >= G, "rerank: bad shape");
  IEEE_REQUIRE(Q + G < (int64_t(1) << 24), "rerank: N = Q + G too large");
  IEEE_REQUIRE(k1 >= 1 && k1 + 1 <= 512 && k2 >= 1 && k2 <= k1 + 1, "rerank: need 1 <= k2 <= k1 + 1 <= 512");
  IEEE_REQUIRE(k1 + 1 <= Q + G, "rerank: k1 + 1 exceeds the number of samples");
  IEEE_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "rerank: workspace must be 256-byte aligned");
  const RerankPlan p = make_plan(Q, G, k1, k2, true, G);
  if (workspace_bytes < p.total) {
    set_error("rerank: workspace too small (%zu < %zu)", workspace_bytes, p.total);
    return IEEE_ERR_WORKSPACE;
  }
  int rc = check_params("rerank", Q, G, k1, k2);
  if (rc) return rc;
  uint8_t* w = static_cast<uint8_t*>(workspace);
  const int N = p.N;
  float* orig = reinterpret_cast<float*>(w + p.off_orig);
  float* colmax = reinterpret_cast<float*>(w + p.off_colmax);
  int32_t* rank = reinterpret_cast<int32_t*>(w + p.off_rank);
  float* rank_val = reinterpret_cast<float*>(w + p.off_rank_val);

  // K1
  IEEE_CUDA_CHECK(cudaMemsetAsync(colmax, 0, size_t(N) * 4, stream));
  int* cm_bits = reinterpret_cast<int*>(colmax);
  const int rpb = 256;
  auto colmax_of = [&](const float* m, int64_t ld, int rows, int cols, int* dst) {
    dim3 grid((cols + 255) / 256, (rows + rpb - 1) / rpb);
    rr_colmax_kernel<<<grid, 256, 0, stream>>>(m, ld, rows, cols, rpb, dst);
    count_launch();
  };
  colmax_of(q_q, ld_qq, (int)Q, (int)Q, cm_bits);
  colmax_of(q_g, ld_qg, (int)Q, (int)G, cm_bits + Q);
  colmax_of(g_g, ld_gg, (int)G, (int)G, cm_bits + Q);
  rr_rowmax_kernel<<<(unsigned)Q, 256, 0, stream>>>(q_g, ld_qg, (int)Q, (int)G, cm_bits);
  count_launch();
  RawView raw{q_g, q_q, g_g, ld_qg, ld_qq, ld_gg, (int)Q, (int)G};
  {
    dim3 grid((N + 31) / 32, (N + 31) / 32);
    rr_build_orig_kernel<<<grid, 256, 0, stream>>>(raw, N, N, colmax, orig, N);
    count_launch();
  }
  // K2: first k1+1 of each row's ascending (value, index) order
  rc = topk(orig, N, N, N, 0, nullptr, nullptr, nullptr, nullptr, p.k1p, rank, rank_val, stream);
  if (rc) return rc;
  // K3
  {
    const size_t smem = size_t(kRowWarps) * (p.k1p + p.khp + p.cap_v_pow2) * 4;
    IEEE_ENSURE_DYN_SMEM(rr_krecip_kernel<true>, smem);
    rr_krecip_kernel<true><<<(N + kRowWarps - 1) / kRowWarps, 32 * kRowWarps, smem, stream>>>(
        rank, p.k1p, orig, N, p.k1p, p.khp, p.cap_v, p.cap_v_pow2, reinterpret_cast<int32_t*>(w + p.off_vcol),
        reinterpret_cast<float*>(w + p.off_vval), reinterpret_cast<int32_t*>(w + p.off_vcnt));
    count_launch();
  }
  // K4 + K5a
  if ((rc = expand_and_index(p, w, rank, k2, Q, 0, stream))) return rc;
  // K5b + K6
  launch_jaccard<false>(p, w, Q, k2, lambda_value, orig, nullptr, 0, Q, out, ldo, out, ldo, stream);
  IEEE_CUDA_CHECK(cudaGetLastError());
  return IEEE_OK;
}

// ---- streamed form: orig in column strips of the virtual matrix, never all of it -------------------------------
// A strip is raw[:, I] for |I| <= W columns, I inside the queries or inside the gallery and starting at a multiple of
// 256 of that operand's index: every contraction output is then computed at the same position inside its tile (and
// its 128-column fix-up span) as in the whole-matrix products, so it has the same bits whatever W (a multiple of 256)
// is and wherever the strips of a sample range start.
// Strip scratch (a buffer of its own: only the prepare call needs it): top [Q, W], bot [max(W x Gp, G x W)], orig rows
// [W, Np], top-k values [W, k1+1], the contraction's fix-up list.
struct StripPlan {
  int64_t W, Gp, Np;
  size_t off_top, off_bot, off_orig, off_val, off_fix, total;
};
static StripPlan make_strip_plan(int64_t Q, int64_t G, int k1, size_t strip_bytes) {
  StripPlan s;
  s.Gp = round_up(G, 32);
  s.Np = round_up(Q + G, 32);
  const int64_t per_col = 4 * (Q + s.Gp + s.Np + k1 + 1);    // scratch bytes per strip column
  const int64_t widest = round_up(Q > G ? Q : G, 256);
  s.W = int64_t(strip_bytes / size_t(per_col)) / 256 * 256;
  s.W = s.W < 256 ? 256 : (s.W > widest ? widest : s.W);
  size_t o = 0;
  auto take = [&](size_t bytes) { size_t r = o; o += align256(bytes); return r; };
  s.off_top = take(size_t(Q) * s.W * 4);
  s.off_bot = take(size_t(s.W) * s.Gp * 4);
  s.off_orig = take(size_t(s.W) * s.Np * 4);
  s.off_val = take(size_t(s.W) * (k1 + 1) * 4);
  s.off_fix = take(distmat_fixup_bytes(Q > G ? Q : G));
  s.total = o + 256;
  return s;
}

size_t rerank_stream_window_workspace_bytes(int64_t Q, int64_t G, int32_t k1, int32_t k2, int64_t Gs) {
  if (check_params("rerank_stream", Q, G, k1, k2) != IEEE_OK) return 0;
  if (Gs < 0 || Gs > G) {
    set_error("rerank_stream: gallery window of %lld rows outside the gallery of %lld", (long long)Gs, (long long)G);
    return 0;
  }
  return make_plan(Q, G, k1, k2, false, Gs).total;
}

size_t rerank_stream_workspace_bytes(int64_t Q, int64_t G, int32_t k1, int32_t k2) {
  return rerank_stream_window_workspace_bytes(Q, G, k1, k2, G);
}

size_t rerank_stream_scratch_bytes(int64_t Q, int64_t G, int32_t k1, size_t strip_bytes) {
  if (check_params("rerank_stream", Q, G, k1, 1) != IEEE_OK) return 0;
  return make_strip_plan(Q, G, k1, strip_bytes).total;
}

int rerank_stream_v_layout(int64_t Q, int64_t G, int32_t k1, int32_t k2, int64_t* cap, size_t* off_col, size_t* off_val,
                           size_t* off_cnt) {
  IEEE_REQUIRE(cap && off_col && off_val && off_cnt, "rerank_stream_v_layout: null pointer");
  int rc = check_params("rerank_stream_v_layout", Q, G, k1, k2);
  if (rc) return rc;
  const RerankPlan p = make_plan(Q, G, k1, k2, false, G);
  *cap = p.cap_v;
  *off_col = p.off_vcol;
  *off_val = p.off_vval;
  *off_cnt = p.off_vcnt;
  return IEEE_OK;
}

// One pass over the strips of the owned samples [q0, q1) and [Q + g0, Q + g1) (each range starting at a multiple of 256
// of its segment and ending at one or at the segment's end).  Pass 0 (K1, K2): colmax and rank of the owned samples.
// Pass 1 (K3): V's membership (columns, counts) of all N rows from `rank`, which must be complete, and the weights of
// the owned rows from their strips, which need their colmax.
int rerank_stream_pass(int pass, const void* q_packed, int64_t Q, const void* g_packed, int64_t G, int64_t D, int metric,
                       int precision, int32_t k1, int32_t k2, size_t strip_bytes, int64_t q0, int64_t q1, int64_t g0, int64_t g1,
                       float* colmax, int32_t* rank, void* workspace, size_t workspace_bytes, void* scratch, size_t scratch_bytes,
                       cudaStream_t stream, int cta_group) {
  IEEE_REQUIRE(pass == 0 || pass == 1, "rerank_stream_pass: pass must be 0 or 1, got %d", pass);
  IEEE_REQUIRE(q_packed && g_packed && colmax && rank && scratch && (pass == 0 || workspace), "rerank_stream_pass: null pointer");
  IEEE_REQUIRE(D > 0, "rerank_stream_pass: bad feature width D=%lld", (long long)D);
  int rc = check_params("rerank_stream_pass", Q, G, k1, k2);
  if (rc) return rc;
  IEEE_REQUIRE(metric == IEEE_METRIC_EUCLIDEAN || metric == IEEE_METRIC_COSINE, "rerank_stream_pass: unknown metric %d", metric);
  IEEE_REQUIRE(precision == IEEE_PREC_F16X3 || precision == IEEE_PREC_BF16,
               "rerank_stream_pass: precision %d has no tensor-core contraction", precision);
  IEEE_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0 && (reinterpret_cast<uintptr_t>(scratch) & 255) == 0,
               "rerank_stream_pass: workspace and scratch must be 256-byte aligned");
  auto range_ok = [](int64_t a, int64_t b, int64_t n) {
    return a == b ? 0 <= a && a <= n : 0 <= a && a < b && b <= n && a % 256 == 0 && (b == n || b % 256 == 0);
  };
  IEEE_REQUIRE(range_ok(q0, q1, Q) && range_ok(g0, g1, G),
               "rerank_stream_pass: owned samples [%lld, %lld) of %lld queries and [%lld, %lld) of %lld gallery rows must start "
               "at a multiple of 256 and end at one or at the end, or be empty", (long long)q0, (long long)q1, (long long)Q, (long long)g0,
               (long long)g1, (long long)G);
  const RerankPlan p = make_plan(Q, G, k1, k2, false, 0);
  const StripPlan s = make_strip_plan(Q, G, k1, strip_bytes);
  if ((pass == 1 && workspace_bytes < p.v_end) || scratch_bytes < s.total) {
    set_error("rerank_stream_pass: workspace or scratch too small (%zu < %zu or %zu < %zu)", workspace_bytes, p.v_end,
              scratch_bytes, s.total);
    return IEEE_ERR_WORKSPACE;
  }
  const int N = p.N;
  uint8_t* w = static_cast<uint8_t*>(workspace);
  uint8_t* sc = static_cast<uint8_t*>(scratch);
  float* top = reinterpret_cast<float*>(sc + s.off_top);
  float* bot = reinterpret_cast<float*>(sc + s.off_bot);
  float* orig = reinterpret_cast<float*>(sc + s.off_orig);
  float* val = reinterpret_cast<float*>(sc + s.off_val);
  void* fix = sc + s.off_fix;
  int32_t* vcol = reinterpret_cast<int32_t*>(w + p.off_vcol);
  float* vval = reinterpret_cast<float*>(w + p.off_vval);
  int32_t* vcnt = reinterpret_cast<int32_t*>(w + p.off_vcnt);
  int* cm_bits = reinterpret_cast<int*>(colmax);
  const int rpb = 256;
  auto rows_of = [&](bool gallery, int64_t r0, int64_t n) {
    return gallery ? packed_rows(g_packed, G, r0, n, D, precision) : packed_rows(q_packed, Q, r0, n, D, precision);
  };
  if (pass == 0) {
    if (q1 > q0) IEEE_CUDA_CHECK(cudaMemsetAsync(colmax + q0, 0, size_t(q1 - q0) * 4, stream));
    if (g1 > g0) IEEE_CUDA_CHECK(cudaMemsetAsync(colmax + Q + g0, 0, size_t(g1 - g0) * 4, stream));
  } else {
    // K3, membership: from rank alone
    const size_t smem = size_t(kRowWarps) * (p.k1p + p.khp + p.cap_v_pow2) * 4;
    IEEE_ENSURE_DYN_SMEM(rr_krecip_kernel<false>, smem);
    rr_krecip_kernel<false><<<(N + kRowWarps - 1) / kRowWarps, 32 * kRowWarps, smem, stream>>>(
        rank, p.k1p, nullptr, N, p.k1p, p.khp, p.cap_v, p.cap_v_pow2, vcol, vval, vcnt);
    count_launch();
  }
  for (int seg = 0; seg < 2; ++seg) {         // strips of the queries, then of the gallery
    const bool gal = seg == 1;
    const int64_t a = gal ? g0 : q0, b = gal ? g1 : q1;
    for (int64_t c0 = a; c0 < b; c0 += s.W) {
      const int64_t wc = (b - c0) < s.W ? (b - c0) : s.W;
      const int64_t i0 = (gal ? Q : 0) + c0;  // first row of orig (column of raw) in the strip
      // the contraction calls of the whole-matrix products, with the same operand roles
      if ((rc = distmat_umma_rows(rows_of(false, 0, Q), rows_of(gal, c0, wc), metric, precision, top, s.W, stream, cta_group,
                                  fix, false)))
        return rc;
      if (!gal) rc = distmat_umma_rows(rows_of(false, c0, wc), rows_of(true, 0, G), metric, precision, bot, s.Gp, stream,
                                       cta_group, fix, false);
      else rc = distmat_umma_rows(rows_of(true, 0, G), rows_of(true, c0, wc), metric, precision, bot, s.W, stream, cta_group,
                                  fix, false);
      if (rc) return rc;
      const StripView view{top, bot, s.W, gal ? s.W : s.Gp, (int)Q, !gal};
      if (pass == 0) {
        rr_colmax_kernel<<<dim3((unsigned)((wc + 255) / 256), (unsigned)((Q + rpb - 1) / rpb)), 256, 0, stream>>>(
            top, s.W, (int)Q, (int)wc, rpb, cm_bits + i0);
        if (!gal) rr_rowmax_kernel<<<(unsigned)wc, 256, 0, stream>>>(bot, s.Gp, (int)wc, (int)G, cm_bits + i0);
        else rr_colmax_kernel<<<dim3((unsigned)((wc + 255) / 256), (unsigned)((G + rpb - 1) / rpb)), 256, 0, stream>>>(
                 bot, s.W, (int)G, (int)wc, rpb, cm_bits + i0);
        count_launch(2);
      }
      rr_build_orig_kernel<<<dim3((unsigned)((N + 31) / 32), (unsigned)((wc + 31) / 32)), 256, 0, stream>>>(
          view, (int)wc, N, colmax + i0, orig, s.Np);
      count_launch();
      if (pass == 0) {
        // K2 for the strip's rows
        if ((rc = topk(orig, s.Np, wc, N, 0, nullptr, nullptr, nullptr, nullptr, p.k1p, rank + i0 * p.k1p, val, stream)))
          return rc;
      } else {
        rr_weights_kernel<<<(unsigned)((wc + kRowWarps - 1) / kRowWarps), 32 * kRowWarps, 0, stream>>>(
            orig, s.Np, (int)i0, (int)wc, p.cap_v, vcol, vval, vcnt);
        count_launch();
      }
    }
  }
  IEEE_CUDA_CHECK(cudaGetLastError());
  return IEEE_OK;
}

// K4 + K5a over the gallery window [g0, g0 + Gs): needs rank and V of every sample
int rerank_stream_finish(void* workspace, size_t workspace_bytes, int64_t Q, int64_t G, int32_t k1, int32_t k2, int64_t g0,
                         int64_t Gs, const int32_t* rank, cudaStream_t stream) {
  IEEE_REQUIRE(workspace && rank, "rerank_stream_finish: null pointer");
  int rc = check_params("rerank_stream_finish", Q, G, k1, k2);
  if (rc) return rc;
  IEEE_REQUIRE(g0 >= 0 && Gs >= 0 && g0 + Gs <= G, "rerank_stream_finish: gallery window [%lld, %lld) outside [0, %lld)",
               (long long)g0, (long long)(g0 + Gs), (long long)G);
  IEEE_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "rerank_stream_finish: workspace must be 256-byte aligned");
  const RerankPlan p = make_plan(Q, G, k1, k2, false, Gs);
  if (workspace_bytes < p.total) {
    set_error("rerank_stream_finish: workspace too small (%zu < %zu)", workspace_bytes, p.total);
    return IEEE_ERR_WORKSPACE;
  }
  if ((rc = expand_and_index(p, static_cast<uint8_t*>(workspace), rank, k2, Q, g0, stream))) return rc;
  IEEE_CUDA_CHECK(cudaGetLastError());
  return IEEE_OK;
}

int rerank_stream_prepare(const void* q_packed, int64_t Q, const void* g_packed, int64_t G, int64_t D, int metric,
                          int precision, int32_t k1, int32_t k2, size_t strip_bytes, float* colmax, int32_t* rank,
                          void* workspace, size_t workspace_bytes, void* scratch, size_t scratch_bytes, cudaStream_t stream,
                          int cta_group) {
  int rc = check_params("rerank_stream_prepare", Q, G, k1, k2);
  if (rc) return rc;
  const size_t need = make_plan(Q, G, k1, k2, false, G).total;
  if (workspace_bytes < need) {                 // before any work is queued
    set_error("rerank_stream_prepare: workspace too small (%zu < %zu)", workspace_bytes, need);
    return IEEE_ERR_WORKSPACE;
  }
  for (int pass = 0; pass < 2; ++pass)
    if ((rc = rerank_stream_pass(pass, q_packed, Q, g_packed, G, D, metric, precision, k1, k2, strip_bytes, 0, Q, 0, G, colmax,
                                 rank, workspace, workspace_bytes, scratch, scratch_bytes, stream, cta_group)))
      return rc;
  return rerank_stream_finish(workspace, workspace_bytes, Q, G, k1, k2, 0, G, rank, stream);
}

// K5b + K6 of queries [row0, row0 + rows) against the gallery window the finish call indexed (Gs columns)
int rerank_stream_block_window(const void* workspace, int64_t Q, int64_t G, int32_t k1, int32_t k2, int64_t Gs,
                               const float* colmax, int64_t row0, int64_t rows, double lambda_value, float* block, int64_t ld,
                               void* scratch, size_t scratch_bytes, cudaStream_t stream) {
  IEEE_REQUIRE(workspace && colmax && block && scratch, "rerank_stream_block: null pointer");
  int rc = check_params("rerank_stream_block", Q, G, k1, k2);
  if (rc) return rc;
  IEEE_REQUIRE(Gs >= 0 && Gs <= G, "rerank_stream_block: gallery window of %lld rows outside the gallery of %lld",
               (long long)Gs, (long long)G);
  IEEE_REQUIRE(row0 >= 0 && rows >= 0 && row0 + rows <= Q && ld >= Gs, "rerank_stream_block: bad block rows [%lld, %lld) of %lld, ld=%lld",
               (long long)row0, (long long)(row0 + rows), (long long)Q, (long long)ld);
  if (scratch_bytes < size_t(rows) * size_t(Gs) * 4) {
    set_error("rerank_stream_block: scratch too small (%zu < %zu)", scratch_bytes, size_t(rows) * size_t(Gs) * 4);
    return IEEE_ERR_WORKSPACE;
  }
  if (rows == 0 || Gs == 0) return IEEE_OK;
  const RerankPlan p = make_plan(Q, G, k1, k2, false, Gs);
  launch_jaccard<true>(p, static_cast<uint8_t*>(const_cast<void*>(workspace)), Q, k2, lambda_value, nullptr, colmax, row0, rows,
                       static_cast<float*>(scratch), Gs, block, ld, stream);
  IEEE_CUDA_CHECK(cudaGetLastError());
  return IEEE_OK;
}

int rerank_stream_block(const void* workspace, int64_t Q, int64_t G, int32_t k1, int32_t k2, const float* colmax, int64_t row0,
                        int64_t rows, double lambda_value, float* block, int64_t ld, void* scratch, size_t scratch_bytes,
                        cudaStream_t stream) {
  return rerank_stream_block_window(workspace, Q, G, k1, k2, G, colmax, row0, rows, lambda_value, block, ld, scratch,
                                    scratch_bytes, stream);
}

// =========================================================================================================
// GNN re-ranking (torchreid/utils/GPU-Re-Ranking/gnn_reranking.py:27-59 and its two CUDA extensions), as an alternative
// `rerank` mode.  Input: the negated similarity matrix -(X_u X_u^T) over queries + gallery (our contraction with the
// NEG_DOT metric).  Steps, all on N x N float32 matrices (N = Q + G; 1.5 GB at Market scale, nothing on a 180 GB part):
//   top-k1 neighbours per row (ieee_topk on the negated scores: largest similarity first, ties by index)  :36-38
//   A[i, rank[i, j]] = 1                              build_adjacency_matrix_kernel.cu:10-17
//   S = S * S                                          :42
//   twice, if k2 != 1:  A = A + A^T;  A[i, :] = sum_{j < k2} S[i, j] * A[rank[i, j], :];  A[i, :] /= |A[i, :]|_2
//                                                      :46-53, gnn_propagate_kernel.cu:8-22
// The caller finishes with cosine = A[:Q] A[Q:]^T (:55) -- again our contraction.
// =========================================================================================================
__global__ void gnn_square_kernel(const float* __restrict__ val, float* __restrict__ S, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) S[i] = val[i] * val[i];                 // (-s)^2 == s^2: the negation of the scores drops out here
}

__global__ void gnn_adjacency_kernel(const int32_t* __restrict__ rank, int k1, int64_t N, float* __restrict__ A, int64_t ld) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= N * k1) return;
  const int64_t i = e / k1;
  const int32_t j = rank[e];
  if (j >= 0) A[i * ld + j] = 1.0f;
}

__global__ void __launch_bounds__(256) gnn_symmetrise_kernel(const float* __restrict__ A, float* __restrict__ B, int64_t N, int64_t ld) {
  __shared__ float t[32][33];
  const int bx = blockIdx.x * 32, by = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;   // 32 x 8
  for (int r = ty; r < 32; r += 8) {
    const int64_t row = bx + r, col = by + tx;             // the transposed tile
    t[r][tx] = (row < N && col < N) ? A[row * ld + col] : 0.f;
  }
  __syncthreads();
  for (int r = ty; r < 32; r += 8) {
    const int64_t row = by + r, col = bx + tx;
    if (row < N && col < N) B[row * ld + col] = A[row * ld + col] + t[tx][r];
  }
}

// out[i, f] = sum_{j < k2} S[i, j] * A[rank[i, j], f], summed in j order like the reference kernel
__global__ void __launch_bounds__(256) gnn_propagate_kernel(const float* __restrict__ A, int64_t ld, const int32_t* __restrict__ rank,
                                                             const float* __restrict__ S, int k1, int k2, int64_t N,
                                                             float* __restrict__ out) {
  const int64_t i = blockIdx.y;
  const int64_t f = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (f >= N) return;
  float sum = 0.f;
  for (int j = 0; j < k2; ++j) {
    const int32_t nb = rank[i * k1 + j];
    if (nb >= 0) sum += A[(int64_t)nb * ld + f] * S[i * k1 + j];
  }
  out[i * ld + f] = sum;
}

__global__ void __launch_bounds__(256) gnn_normalise_kernel(float* __restrict__ A, int64_t ld, int64_t N) {
  __shared__ float red[8];
  __shared__ float inv_s;
  float* row = A + (int64_t)blockIdx.x * ld;
  float s = 0.f;
  for (int64_t f = threadIdx.x; f < N; f += 256) s = __fmaf_rn(row[f], row[f], s);
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int w = 0; w < 8; ++w) t += red[w];
    inv_s = __fsqrt_rn(t);                               // torch.norm(A, p=2, dim=1): no epsilon (gnn_reranking.py:52-53)
  }
  __syncthreads();
  const float nrm = inv_s;
  for (int64_t f = threadIdx.x; f < N; f += 256) row[f] = __fdiv_rn(row[f], nrm);
}

size_t gnn_rerank_workspace_bytes(int64_t N, int32_t k1) {
  if (N <= 0 || k1 <= 0) return 0;
  const int64_t ld = round_up(N, 32);
  return 3 * align256(size_t(N) * k1 * 4) + align256(size_t(N) * ld * 4) + 256;
}

int gnn_rerank(const float* neg_score, int64_t lds, int64_t N, int32_t k1, int32_t k2, float* A, int64_t ldA, void* workspace,
               size_t workspace_bytes, cudaStream_t stream) {
  IEEE_REQUIRE(neg_score && A && workspace, "gnn_rerank: null pointer");
  IEEE_REQUIRE(N > 0 && lds >= N && ldA >= N && k1 >= 1 && k1 <= N && k1 <= 1024 && k2 >= 1 && k2 <= k1,
               "gnn_rerank: bad arguments N=%lld k1=%d k2=%d", (long long)N, k1, k2);
  IEEE_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "gnn_rerank: workspace must be 256-byte aligned");
  if (workspace_bytes < gnn_rerank_workspace_bytes(N, k1)) {
    set_error("gnn_rerank: workspace too small (%zu < %zu)", workspace_bytes, gnn_rerank_workspace_bytes(N, k1));
    return IEEE_ERR_WORKSPACE;
  }
  const int64_t ld = round_up(N, 32);
  IEEE_REQUIRE(ldA == ld, "gnn_rerank: the adjacency matrix must have a row pitch of %lld floats", (long long)ld);
  uint8_t* w = static_cast<uint8_t*>(workspace);
  int32_t* rank = reinterpret_cast<int32_t*>(w);
  w += align256(size_t(N) * k1 * 4);
  float* val = reinterpret_cast<float*>(w);
  w += align256(size_t(N) * k1 * 4);
  float* S = reinterpret_cast<float*>(w);
  w += align256(size_t(N) * k1 * 4);
  float* B = reinterpret_cast<float*>(w);
  int rc = topk(neg_score, lds, N, N, 0, nullptr, nullptr, nullptr, nullptr, k1, rank, val, stream);
  if (rc) return rc;
  const int64_t nk = N * k1;
  gnn_square_kernel<<<(unsigned)((nk + 255) / 256), 256, 0, stream>>>(val, S, nk);
  IEEE_CUDA_CHECK(cudaMemsetAsync(A, 0, size_t(N) * ld * 4, stream));
  gnn_adjacency_kernel<<<(unsigned)((nk + 255) / 256), 256, 0, stream>>>(rank, k1, N, A, ld);
  count_launch(2);
  if (k2 != 1) {
    const dim3 tgrid((unsigned)((N + 31) / 32), (unsigned)((N + 31) / 32)), pgrid((unsigned)((N + 255) / 256), (unsigned)N);
    for (int it = 0; it < 2; ++it) {
      gnn_symmetrise_kernel<<<tgrid, 256, 0, stream>>>(A, B, N, ld);
      gnn_propagate_kernel<<<pgrid, 256, 0, stream>>>(B, ld, rank, S, k1, k2, N, A);
      gnn_normalise_kernel<<<(unsigned)N, 256, 0, stream>>>(A, ld, N);
      count_launch(3);
    }
  }
  IEEE_CUDA_CHECK(cudaGetLastError());
  return IEEE_OK;
}

// =========================================================================================================
// GNN re-ranking, streamed: the same A as gnn_rerank, held sparse, from packed features without any N x N matrix.
//   neighbours  -(X_u X_u^T) in row strips (queries, then gallery; W rows each) -> top-k1 `rank`, S = val^2
//   symbolic    every structure below is decided by `rank` alone; one CTA per row counts it in a shared-memory bitmap
//               of N bits from A0 = rank, its transpose T0 and K2inv (the transpose of the first k2 columns of rank):
//                 B1[r] = A0[r] u T0[r]                 A1[i] = u_{j<k2} B1[rank[i, j]]
//                 A1^T[r] = u_{m in B1[r]} K2inv[m]     B2[r] = A1[r] u A1^T[r]     A2[i] = u_{j<k2} B2[rank[i, j]]
//               (A1^T[r]: r in A1[c] <=> some rank[c, j < k2] lies in B1[r], B1 being structurally symmetric)
//   numeric     B = A + A^T, propagation and normalisation row by row into CSR rows with ascending columns, then the
//               gallery rows of A2 as CSC (rows ascending).  Structural entries whose value is 0 are kept.
// Every value has the dense kernels' bits: the dense sums skip nothing, but an absent entry adds fma(0, s, x) = x or
// 0 + x = x, so summing only the present entries in the same order gives the same float.
// =========================================================================================================
constexpr int kGnnThreads = 256;           // also the residue classes of the normalisation (gnn_normalise_kernel)
constexpr int64_t kGnnMaxN = int64_t(1) << 20;   // the per-row bitmap: N bits of shared memory

struct SpRows {                            // CSR rows (idx = columns) or CSC columns (idx = rows); val == nullptr: all 1
  const int64_t* ptr;
  const int32_t* idx;
  const float* val;
  __device__ __forceinline__ float v(int64_t p) const { return val ? val[p] : 1.0f; }
};

// The rows (or columns) a call covers: [a0, a0 + na), then [b0, b0 + nb) -- a process's queries, then its gallery rows,
// as indices among all N samples.  Block i of a launch over count() rows takes row(i); the whole range is {0, Q, Q, G}.
struct GnnRows {
  int a0, na, b0, nb;
  __host__ __device__ int count() const { return na + nb; }
  __device__ __forceinline__ int row(int i) const { return i < na ? a0 + i : b0 + i - na; }
  __device__ __forceinline__ bool owns(int c) const { return (c >= a0 && c < a0 + na) || (c >= b0 && c < b0 + nb); }
};

__device__ __forceinline__ void bm_set(uint32_t* bm, int c) { atomicOr(bm + (c >> 5), 1u << (c & 31)); }

__device__ void bm_clear(uint32_t* bm, int nw) {
  __syncthreads();
  for (int w = threadIdx.x; w < nw; w += kGnnThreads) bm[w] = 0u;
  __syncthreads();
}

// exclusive scan of one int per thread; wsum: 8 ints of shared memory
__device__ int block_excl_scan(int v, int* wsum) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  int incl = v;
  for (int o = 1; o < 32; o <<= 1) {
    const int y = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += y;
  }
  if (lane == 31) wsum[w] = incl;
  __syncthreads();
  int off = 0;
  for (int x = 0; x < w; ++x) off += wsum[x];
  __syncthreads();
  return off + incl - v;
}

// number of set bits (every thread gets it)
__device__ int bm_count(const uint32_t* bm, int nw, int* wsum) {
  __syncthreads();
  int n = 0;
  for (int w = threadIdx.x; w < nw; w += kGnnThreads) n += __popc(bm[w]);
  for (int o = 16; o > 0; o >>= 1) n += __shfl_xor_sync(0xffffffffu, n, o);
  if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = n;
  __syncthreads();
  int t = 0;
  for (int x = 0; x < kGnnThreads / 32; ++x) t += wsum[x];
  __syncthreads();
  return t;
}

// the set bits in ascending order -> out[0, count); thread t owns a contiguous run of words
__device__ void bm_emit(const uint32_t* bm, int nw, int32_t* out, int* wsum) {
  __syncthreads();
  const int per = (nw + kGnnThreads - 1) / kGnnThreads, w0 = threadIdx.x * per, w1 = min(nw, w0 + per);
  int n = 0;
  for (int w = w0; w < w1; ++w) n += __popc(bm[w]);
  int pos = block_excl_scan(n, wsum);
  for (int w = w0; w < w1; ++w)
    for (uint32_t b = bm[w]; b; b &= b - 1) out[pos++] = w * 32 + __ffs(b) - 1;
  __syncthreads();
}

// position of column c in the ascending run idx[lo, hi) (present by construction)
__device__ __forceinline__ int64_t find_col(const int32_t* __restrict__ idx, int64_t lo, int64_t hi, int c) {
  while (hi - lo > 1) {
    const int64_t mid = (lo + hi) >> 1;
    if (idx[mid] <= c) lo = mid; else hi = mid;
  }
  return lo;
}

// bits of row m of a sparse operand, by worker `id` of `nt`
// (a top-k list pads with -1 only when a row has fewer than k1 candidates, which k1 <= N rules out; skipped anyway)
__device__ __forceinline__ void set_row(uint32_t* bm, const SpRows& a, int m, int id, int nt) {
  for (int64_t p = a.ptr[m] + id; p < a.ptr[m + 1]; p += nt)
    if (a.idx[p] >= 0) bm_set(bm, a.idx[p]);
}
// B1[m] = A0[m] u T0[m]
__device__ __forceinline__ void set_b1(uint32_t* bm, const SpRows& a0, const SpRows& t0, int m, int id, int nt) {
  set_row(bm, a0, m, id, nt);
  set_row(bm, t0, m, id, nt);
}
// A1[m] = u_{j<k2} B1[rank[m, j]]: one warp per j
__device__ void set_a1(uint32_t* bm, const SpRows& a0, const SpRows& t0, int k2, int m) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (int j = w; j < k2; j += kGnnThreads / 32) {
    const int x = a0.idx[a0.ptr[m] + j];
    if (x >= 0) set_b1(bm, a0, t0, x, lane, 32);
  }
}
// A1^T[m] = u_{x in B1[m]} K2inv[x]: one warp per x
__device__ void set_a1t(uint32_t* bm, const SpRows& a0, const SpRows& t0, const SpRows& k2inv, int m) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int64_t na = a0.ptr[m + 1] - a0.ptr[m], nt = t0.ptr[m + 1] - t0.ptr[m];
  for (int64_t u = w; u < na + nt; u += kGnnThreads / 32) {
    const int x = u < na ? a0.idx[a0.ptr[m] + u] : t0.idx[t0.ptr[m] + u - na];
    if (x >= 0) set_row(bm, k2inv, x, lane, 32);
  }
}

// symbolic phase: per row the nnz of B1, A1, B2, A2
__global__ void __launch_bounds__(kGnnThreads) gnn_symbolic_kernel(SpRows a0, SpRows t0, SpRows k2inv, int N, int k2,
                                                                    GnnRows own, int32_t* __restrict__ cnt_b1,
                                                                    int32_t* __restrict__ cnt_a1, int32_t* __restrict__ cnt_b2,
                                                                    int32_t* __restrict__ cnt_a2) {
  extern __shared__ __align__(16) uint32_t bm[];
  __shared__ int wsum[kGnnThreads / 32];
  const int r = own.row(blockIdx.x), nw = (N + 31) >> 5;
  bm_clear(bm, nw);
  set_b1(bm, a0, t0, r, threadIdx.x, kGnnThreads);
  int n = bm_count(bm, nw, wsum);
  if (threadIdx.x == 0) cnt_b1[r] = n;
  bm_clear(bm, nw);
  set_a1(bm, a0, t0, k2, r);
  n = bm_count(bm, nw, wsum);
  if (threadIdx.x == 0) cnt_a1[r] = n;
  set_a1t(bm, a0, t0, k2inv, r);
  n = bm_count(bm, nw, wsum);
  if (threadIdx.x == 0) cnt_b2[r] = n;
  bm_clear(bm, nw);
  for (int j = 0; j < k2; ++j) {
    const int m = a0.idx[a0.ptr[r] + j];
    if (m < 0) continue;
    set_a1(bm, a0, t0, k2, m);
    set_a1t(bm, a0, t0, k2inv, m);
  }
  n = bm_count(bm, nw, wsum);
  if (threadIdx.x == 0) cnt_a2[r] = n;
}

// B = A + A^T row by row: ascending columns of A[r] u T[r]; values (0 + A[r][c]) + A[c][r], which is the dense
// A[r][c] + A[c][r] (gnn_symmetrise_kernel) for every pattern of presence
__global__ void __launch_bounds__(kGnnThreads) gnn_sum_kernel(SpRows a, SpRows t, int N, GnnRows own,
                                                               const int64_t* __restrict__ bptr, int32_t* __restrict__ bcol,
                                                               float* __restrict__ bval) {
  extern __shared__ __align__(16) uint32_t bm[];
  __shared__ int wsum[kGnnThreads / 32];
  const int r = own.row(blockIdx.x), nw = (N + 31) >> 5;
  const int64_t b0 = bptr[r], b1 = bptr[r + 1];
  bm_clear(bm, nw);
  set_row(bm, a, r, threadIdx.x, kGnnThreads);
  if (t.ptr) set_row(bm, t, r, threadIdx.x, kGnnThreads);
  bm_emit(bm, nw, bcol + b0, wsum);
  for (int64_t p = b0 + threadIdx.x; p < b1; p += kGnnThreads) bval[p] = 0.f;
  __syncthreads();
  for (int64_t p = a.ptr[r] + threadIdx.x; p < a.ptr[r + 1]; p += kGnnThreads) {
    if (a.idx[p] < 0) continue;
    const int64_t q = find_col(bcol, b0, b1, a.idx[p]);
    bval[q] = __fadd_rn(bval[q], a.v(p));
  }
  __syncthreads();
  if (t.ptr)
    for (int64_t p = t.ptr[r] + threadIdx.x; p < t.ptr[r + 1]; p += kGnnThreads) {
      const int64_t q = find_col(bcol, b0, b1, t.idx[p]);
      bval[q] = __fadd_rn(bval[q], t.v(p));
    }
}

// A[i] = sum_{j<k2} S[i, j] * B[rank[i, j]] in j order (gnn_propagate_kernel's FFMA chain), then A[i] /= |A[i]|_2 in
// gnn_normalise_kernel's order: thread t sums the squares of columns c = t (mod 256) in ascending order, then the same
// shuffle tree, warp sum and square root
__global__ void __launch_bounds__(kGnnThreads) gnn_propagate_rows_kernel(SpRows b, const int32_t* __restrict__ rank,
                                                                          const float* __restrict__ S, int k1, int k2, int N,
                                                                          GnnRows own, const int64_t* __restrict__ aptr,
                                                                          int32_t* __restrict__ acol, float* __restrict__ aval) {
  extern __shared__ __align__(16) uint32_t bm[];
  __shared__ int wsum[kGnnThreads / 32];
  __shared__ int32_t chunk_c[kGnnThreads];
  __shared__ float chunk_v[kGnnThreads];
  __shared__ float red[kGnnThreads / 32];
  __shared__ float nrm_s;
  const int i = own.row(blockIdx.x), nw = (N + 31) >> 5;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int64_t a0 = aptr[i], a1 = aptr[i + 1];
  const int32_t* nb = rank + (int64_t)i * k1;
  bm_clear(bm, nw);
  for (int j = w; j < k2; j += kGnnThreads / 32)
    if (nb[j] >= 0) set_row(bm, b, nb[j], lane, 32);
  bm_emit(bm, nw, acol + a0, wsum);
  for (int64_t p = a0 + threadIdx.x; p < a1; p += kGnnThreads) aval[p] = 0.f;
  __syncthreads();
  for (int j = 0; j < k2; ++j) {
    const int m = nb[j];
    if (m < 0) continue;
    const float s = S[(int64_t)i * k1 + j];
    for (int64_t p = b.ptr[m] + threadIdx.x; p < b.ptr[m + 1]; p += kGnnThreads) {
      const int64_t q = find_col(acol, a0, a1, b.idx[p]);
      aval[q] = __fmaf_rn(b.val[p], s, aval[q]);
    }
    __syncthreads();
  }
  float s = 0.f;
  for (int64_t base = a0; base < a1; base += kGnnThreads) {
    const int64_t p = base + threadIdx.x;
    chunk_c[threadIdx.x] = p < a1 ? acol[p] : -1;
    chunk_v[threadIdx.x] = p < a1 ? aval[p] : 0.f;
    __syncthreads();
    const int n = a1 - base < kGnnThreads ? (int)(a1 - base) : kGnnThreads;
    for (int u = 0; u < n; ++u)
      if ((chunk_c[u] & (kGnnThreads - 1)) == (int)threadIdx.x) s = __fmaf_rn(chunk_v[u], chunk_v[u], s);
    __syncthreads();
  }
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) red[w] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int x = 0; x < kGnnThreads / 32; ++x) t += red[x];
    nrm_s = __fsqrt_rn(t);
  }
  __syncthreads();
  const float nrm = nrm_s;
  for (int64_t p = a0 + threadIdx.x; p < a1; p += kGnnThreads) aval[p] = __fdiv_rn(aval[p], nrm);
}

// transposes: entries of rows [r0, r1) counted per column, then placed (row - r_base, value) in any order
__global__ void gnn_col_count_kernel(SpRows a, int r0, int r1, int32_t* __restrict__ cnt) {
  const int r = r0 + blockIdx.x * (blockDim.x / 32) + (threadIdx.x >> 5);
  if (r >= r1) return;
  for (int64_t p = a.ptr[r] + (threadIdx.x & 31); p < a.ptr[r + 1]; p += 32) atomicAdd(cnt + a.idx[p], 1);
}
__global__ void gnn_col_fill_kernel(SpRows a, int r0, int r1, int r_base, const int64_t* __restrict__ tptr,
                                    int32_t* __restrict__ cursor, int32_t* __restrict__ tidx, float* __restrict__ tval) {
  const int r = r0 + blockIdx.x * (blockDim.x / 32) + (threadIdx.x >> 5);
  if (r >= r1) return;
  for (int64_t p = a.ptr[r] + (threadIdx.x & 31); p < a.ptr[r + 1]; p += 32) {
    const int c = a.idx[p];
    const int64_t q = tptr[c] + atomicAdd(cursor + c, 1);
    tidx[q] = r - r_base;
    if (tval) tval[q] = a.v(p);
  }
}
// K2inv and the transpose of A0 straight from rank (columns j < kk of every row)
__global__ void gnn_rank_count_kernel(const int32_t* __restrict__ rank, int64_t N, int k1, int kk, int32_t* __restrict__ cnt) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= N * kk) return;
  const int64_t i = e / kk;
  const int32_t c = rank[i * k1 + (e - i * kk)];
  if (c >= 0) atomicAdd(cnt + c, 1);
}
__global__ void gnn_rank_fill_kernel(const int32_t* __restrict__ rank, int64_t N, int k1, int kk, const int64_t* __restrict__ tptr,
                                     int32_t* __restrict__ cursor, int32_t* __restrict__ tidx) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= N * kk) return;
  const int64_t i = e / kk;
  const int32_t c = rank[i * k1 + (e - i * kk)];
  if (c >= 0) tidx[tptr[c] + atomicAdd(cursor + c, 1)] = (int32_t)i;
}
// exclusive scan int32[n] -> int64[n + 1]; single CTA
__global__ void __launch_bounds__(1024) gnn_scan64_kernel(const int32_t* __restrict__ in, int64_t n, int64_t* __restrict__ out) {
  __shared__ long long wsum[32];
  __shared__ long long carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (int64_t base = 0; base < n; base += 1024) {
    const int64_t i = base + threadIdx.x;
    const long long v = i < n ? in[i] : 0;
    long long incl = v;
    for (int o = 1; o < 32; o <<= 1) {
      const long long y = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += y;
    }
    if (lane == 31) wsum[w] = incl;
    __syncthreads();
    long long off = carry;
    for (int x = 0; x < w; ++x) off += wsum[x];
    if (i < n) out[i] = off + incl - v;
    __syncthreads();
    if (threadIdx.x == 1023) carry = off + incl;
    __syncthreads();
  }
  if (threadIdx.x == 0) out[n] = carry;
}
__global__ void gnn_iota_kernel(int64_t* __restrict__ ptr, int64_t n, int step) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i <= n) ptr[i] = i * step;
}
// the gallery CSC: each owned column's rows ascending (a bitmap of G bits), values looked up in the CSR rows; every
// other column's entries are set to 0, so that summing the processes' CSCs as integers assembles the whole one
__global__ void __launch_bounds__(kGnnThreads) gnn_col_sort_kernel(const int64_t* __restrict__ gptr, int32_t* __restrict__ grow,
                                                                    float* __restrict__ gval, SpRows a, int Q, int G, GnnRows own) {
  extern __shared__ __align__(16) uint32_t bm[];
  __shared__ int wsum[kGnnThreads / 32];
  const int c = blockIdx.x, nw = (G + 31) >> 5;
  const int64_t p0 = gptr[c], p1 = gptr[c + 1];
  if (p0 == p1) return;
  if (!own.owns(c)) {
    for (int64_t p = p0 + threadIdx.x; p < p1; p += kGnnThreads) {
      grow[p] = 0;
      gval[p] = 0.f;
    }
    return;
  }
  bm_clear(bm, nw);
  for (int64_t p = p0 + threadIdx.x; p < p1; p += kGnnThreads) bm_set(bm, grow[p]);
  bm_emit(bm, nw, grow + p0, wsum);
  for (int64_t p = p0 + threadIdx.x; p < p1; p += kGnnThreads) {
    const int r = Q + grow[p];
    gval[p] = a.val[find_col(a.idx, a.ptr[r], a.ptr[r + 1], c)];
  }
}
// -(A2[q] . A2[Q + g]) for queries [row0, row0 + rows): scattered through the gallery CSC, columns of A2[q] ascending,
// into a float64 accumulator row (a product of two floats is exact in float64), rounded to float32 once
__global__ void __launch_bounds__(kGnnThreads) gnn_block_kernel(SpRows a, SpRows gcsc, int G, int row0, double* __restrict__ acc_rows,
                                                                 float* __restrict__ block, int64_t ld) {
  const int q = row0 + blockIdx.x;
  double* acc = acc_rows + (int64_t)blockIdx.x * G;
  float* out = block + (int64_t)blockIdx.x * ld;
  for (int g = threadIdx.x; g < G; g += kGnnThreads) acc[g] = 0.0;
  __syncthreads();
  for (int64_t p = a.ptr[q]; p < a.ptr[q + 1]; ++p) {
    const int c = a.idx[p];
    const double x = a.val[p];
    for (int64_t e = gcsc.ptr[c] + threadIdx.x; e < gcsc.ptr[c + 1]; e += kGnnThreads) {
      const int g = gcsc.idx[e];
      acc[g] = __fma_rn(x, (double)gcsc.val[e], acc[g]);      // rows are distinct inside a column
    }
    __syncthreads();
  }
  for (int g = threadIdx.x; g < G; g += kGnnThreads) out[g] = -__double2float_rn(acc[g]);
}

static int gnn_stream_check(const char* who, int64_t Q, int64_t G, int32_t k1, int32_t k2) {
  IEEE_REQUIRE(Q > 0 && G > 0, "%s: bad shape Q=%lld G=%lld", who, (long long)Q, (long long)G);
  IEEE_REQUIRE(Q + G <= kGnnMaxN, "%s: N = Q + G = %lld exceeds %lld", who, (long long)(Q + G), (long long)kGnnMaxN);
  IEEE_REQUIRE(k2 >= 1 && k2 <= k1 && k1 <= 1024, "%s: need 1 <= k2 <= k1 <= 1024, got k1=%d k2=%d", who, k1, k2);
  IEEE_REQUIRE(k1 <= Q + G, "%s: k1 = %d exceeds the %lld query and gallery samples", who, k1, (long long)(Q + G));
  return IEEE_OK;
}

// Scratch of the neighbour and graph calls (one buffer, used by one phase after the other): the strips [W, ld] with
// their top-k values, or the index both graph calls share (A0's row offsets, T0, K2inv, per-row counts and offsets).
struct GnnScratch {
  int64_t N, W, ld;
  size_t off_strip, off_val, strips;
  size_t off_a0p, off_t0p, off_t0i, off_k2p, off_k2i, off_cnt, off_cursor, off_cntr[4], off_ptr[4], off_tot, index;
  size_t total;
};
static GnnScratch gnn_scratch_plan(int64_t Q, int64_t G, int k1, size_t strip_bytes) {
  GnnScratch s;
  s.N = Q + G;
  s.ld = round_up(s.N, 32);
  const int64_t per_row = 4 * (s.ld + k1);
  const int64_t widest = round_up(Q > G ? Q : G, 256);
  s.W = int64_t(strip_bytes / size_t(per_row)) / 256 * 256;
  s.W = s.W < 256 ? 256 : (s.W > widest ? widest : s.W);
  size_t o = 0;
  auto take = [&](size_t bytes) { size_t r = o; o += align256(bytes); return r; };
  s.off_strip = take(size_t(s.W) * s.ld * 4);
  s.off_val = take(size_t(s.W) * k1 * 4);
  s.strips = o;
  o = 0;
  const size_t N = s.N, p8 = (N + 1) * 8;
  s.off_a0p = take(p8);
  s.off_t0p = take(p8);
  s.off_t0i = take(N * k1 * 4);
  s.off_k2p = take(p8);
  s.off_k2i = take(N * k1 * 4);
  s.off_cnt = take(N * 4);
  s.off_cursor = take(N * 4);
  for (int x = 0; x < 4; ++x) s.off_cntr[x] = take(N * 4);
  for (int x = 0; x < 4; ++x) s.off_ptr[x] = take(p8);
  s.off_tot = take(64);
  s.index = o;
  s.total = (s.strips > s.index ? s.strips : s.index) + 256;
  return s;
}

size_t gnn_stream_scratch_bytes(int64_t Q, int64_t G, int32_t k1, size_t strip_bytes) {
  if (gnn_stream_check("gnn_stream", Q, G, k1, 1) != IEEE_OK) return 0;
  return gnn_scratch_plan(Q, G, k1, strip_bytes).total;
}

// The owned rows [q0, q1) and [g0, g1) of the phase calls: each empty, or starting at a multiple of 256 of its segment and
// ending at one or at the segment's end.
static int gnn_owned(const char* who, int64_t Q, int64_t G, int64_t q0, int64_t q1, int64_t g0, int64_t g1, GnnRows* own) {
  auto range_ok = [](int64_t a, int64_t b, int64_t n) {
    return a == b ? 0 <= a && a <= n : 0 <= a && a < b && b <= n && a % 256 == 0 && (b == n || b % 256 == 0);
  };
  IEEE_REQUIRE(range_ok(q0, q1, Q) && range_ok(g0, g1, G),
               "%s: owned rows [%lld, %lld) of %lld queries and [%lld, %lld) of %lld gallery rows must start at a multiple "
               "of 256 and end at one or at the end, or be empty", who, (long long)q0, (long long)q1, (long long)Q, (long long)g0,
               (long long)g1, (long long)G);
  *own = GnnRows{(int)q0, (int)(q1 - q0), (int)(Q + g0), (int)(g1 - g0)};
  return IEEE_OK;
}

int gnn_stream_neighbours_rows(const void* q_packed, int64_t Q, const void* g_packed, int64_t G, int64_t D, int precision,
                               int32_t k1, size_t strip_bytes, int64_t q0, int64_t q1, int64_t g0, int64_t g1, int32_t* rank,
                               float* S, void* scratch, size_t scratch_bytes, cudaStream_t stream, int cta_group) {
  IEEE_REQUIRE(q_packed && g_packed && rank && S && scratch, "gnn_stream_neighbours: null pointer");
  IEEE_REQUIRE(D > 0, "gnn_stream_neighbours: bad feature width D=%lld", (long long)D);
  int rc = gnn_stream_check("gnn_stream_neighbours", Q, G, k1, 1);
  if (rc) return rc;
  GnnRows own;
  if ((rc = gnn_owned("gnn_stream_neighbours", Q, G, q0, q1, g0, g1, &own))) return rc;
  IEEE_REQUIRE(precision == IEEE_PREC_F16X3 || precision == IEEE_PREC_BF16,
               "gnn_stream_neighbours: precision %d has no tensor-core contraction", precision);
  IEEE_REQUIRE((reinterpret_cast<uintptr_t>(scratch) & 255) == 0, "gnn_stream_neighbours: scratch must be 256-byte aligned");
  const GnnScratch s = gnn_scratch_plan(Q, G, k1, strip_bytes);
  if (scratch_bytes < s.total) {
    set_error("gnn_stream_neighbours: scratch too small (%zu < %zu)", scratch_bytes, s.total);
    return IEEE_ERR_WORKSPACE;
  }
  uint8_t* sc = static_cast<uint8_t*>(scratch);
  float* strip = reinterpret_cast<float*>(sc + s.off_strip);
  float* val = reinterpret_cast<float*>(sc + s.off_val);
  const int64_t N = Q + G;
  auto rows_of = [&](bool gallery, int64_t r0, int64_t n) {
    return gallery ? packed_rows(g_packed, G, r0, n, D, precision) : packed_rows(q_packed, Q, r0, n, D, precision);
  };
  // NEG_DOT has no centre and no near-duplicate fix-up, so an output's bits do not depend on where it sits in its
  // tile: the strips give the bits of the whole -(X_u X_u^T) product
  for (int seg = 0; seg < 2; ++seg) {
    const bool gal = seg == 1;
    const int64_t a = gal ? g0 : q0, b = gal ? g1 : q1;
    for (int64_t r0 = a; r0 < b; r0 += s.W) {
      const int64_t wr = (b - r0) < s.W ? (b - r0) : s.W;
      const int64_t i0 = (gal ? Q : 0) + r0;
      if ((rc = distmat_umma_rows(rows_of(gal, r0, wr), rows_of(false, 0, Q), IEEE_METRIC_NEG_DOT, precision, strip, s.ld, stream,
                                  cta_group, nullptr, false)))
        return rc;
      if ((rc = distmat_umma_rows(rows_of(gal, r0, wr), rows_of(true, 0, G), IEEE_METRIC_NEG_DOT, precision, strip + Q, s.ld,
                                  stream, cta_group, nullptr, false)))
        return rc;
      if ((rc = topk(strip, s.ld, wr, N, 0, nullptr, nullptr, nullptr, nullptr, k1, rank + i0 * k1, val, stream))) return rc;
      const int64_t nk = wr * k1;
      gnn_square_kernel<<<(unsigned)((nk + 255) / 256), 256, 0, stream>>>(val, S + i0 * k1, nk);
      count_launch();
    }
  }
  IEEE_CUDA_CHECK(cudaGetLastError());
  return IEEE_OK;
}

int gnn_stream_neighbours(const void* q_packed, int64_t Q, const void* g_packed, int64_t G, int64_t D, int precision, int32_t k1,
                          size_t strip_bytes, int32_t* rank, float* S, void* scratch, size_t scratch_bytes, cudaStream_t stream,
                          int cta_group) {
  return gnn_stream_neighbours_rows(q_packed, Q, g_packed, G, D, precision, k1, strip_bytes, 0, Q, 0, G, rank, S, scratch,
                                    scratch_bytes, stream, cta_group);
}

// The index of the graph calls, and the offsets of the numeric phase's work buffer (B1, A1, A1^T, B2).
struct GnnIndex {
  int64_t *a0p, *t0p, *k2p, *ptr[4], *tot;     // ptr: B1, A1, B2, A2
  int32_t *t0i, *k2i, *cnt, *cursor, *cntr[4];
};
static GnnIndex gnn_index(const GnnScratch& s, void* scratch) {
  uint8_t* b = static_cast<uint8_t*>(scratch);
  GnnIndex x;
  x.a0p = reinterpret_cast<int64_t*>(b + s.off_a0p);
  x.t0p = reinterpret_cast<int64_t*>(b + s.off_t0p);
  x.k2p = reinterpret_cast<int64_t*>(b + s.off_k2p);
  x.t0i = reinterpret_cast<int32_t*>(b + s.off_t0i);
  x.k2i = reinterpret_cast<int32_t*>(b + s.off_k2i);
  x.cnt = reinterpret_cast<int32_t*>(b + s.off_cnt);
  x.cursor = reinterpret_cast<int32_t*>(b + s.off_cursor);
  for (int i = 0; i < 4; ++i) {
    x.cntr[i] = reinterpret_cast<int32_t*>(b + s.off_cntr[i]);
    x.ptr[i] = reinterpret_cast<int64_t*>(b + s.off_ptr[i]);
  }
  x.tot = reinterpret_cast<int64_t*>(b + s.off_tot);
  return x;
}
struct GnnWork {
  size_t off_b1c, off_b1v, off_a1c, off_a1v, off_tp, off_ti, off_tv, off_b2c, off_b2v, total;
};
static GnnWork gnn_work_plan(int64_t N, int k2, int64_t nb1, int64_t na1, int64_t nb2) {
  GnnWork w{};
  size_t o = 0;
  auto take = [&](size_t bytes) { size_t r = o; o += align256(bytes); return r; };
  if (k2 != 1) {
    w.off_b1c = take(size_t(nb1) * 4);
    w.off_b1v = take(size_t(nb1) * 4);
    w.off_a1c = take(size_t(na1) * 4);
    w.off_a1v = take(size_t(na1) * 4);
    w.off_tp = take(size_t(N + 1) * 8);
    w.off_ti = take(size_t(na1) * 4);
    w.off_tv = take(size_t(na1) * 4);
    w.off_b2c = take(size_t(nb2) * 4);
    w.off_b2v = take(size_t(nb2) * 4);
  }
  w.total = o + 256;
  return w;
}

static size_t gnn_bitmap_smem(int64_t n) { return size_t((n + 31) / 32) * 4; }

// counts per column of rank[:, :kk] -> offsets, then the rows of every column (any order)
static int gnn_rank_transpose(const int32_t* rank, int64_t N, int k1, int kk, const GnnIndex& x, int64_t* tptr, int32_t* tidx,
                              cudaStream_t stream) {
  const int64_t nk = N * kk;
  IEEE_CUDA_CHECK(cudaMemsetAsync(x.cnt, 0, size_t(N) * 4, stream));
  IEEE_CUDA_CHECK(cudaMemsetAsync(x.cursor, 0, size_t(N) * 4, stream));
  gnn_rank_count_kernel<<<(unsigned)((nk + 255) / 256), 256, 0, stream>>>(rank, N, k1, kk, x.cnt);
  gnn_scan64_kernel<<<1, 1024, 0, stream>>>(x.cnt, N, tptr);
  gnn_rank_fill_kernel<<<(unsigned)((nk + 255) / 256), 256, 0, stream>>>(rank, N, k1, kk, tptr, x.cursor, tidx);
  count_launch(3);
  return IEEE_OK;
}
// rows [r0, r1) of `a` -> CSC (row indices relative to r_base) with values
static int gnn_sparse_transpose(const SpRows& a, int64_t N, int r0, int r1, int r_base, const GnnIndex& x, int64_t* tptr,
                                int32_t* tidx, float* tval, cudaStream_t stream) {
  IEEE_CUDA_CHECK(cudaMemsetAsync(x.cnt, 0, size_t(N) * 4, stream));
  IEEE_CUDA_CHECK(cudaMemsetAsync(x.cursor, 0, size_t(N) * 4, stream));
  const unsigned blocks = (unsigned)((r1 - r0 + 7) / 8);
  if (blocks) gnn_col_count_kernel<<<blocks, 256, 0, stream>>>(a, r0, r1, x.cnt);
  gnn_scan64_kernel<<<1, 1024, 0, stream>>>(x.cnt, N, tptr);
  if (blocks) gnn_col_fill_kernel<<<blocks, 256, 0, stream>>>(a, r0, r1, r_base, tptr, x.cursor, tidx, tval);
  count_launch(3);
  return IEEE_OK;
}

int gnn_stream_layout(int64_t Q, int64_t G, int32_t k1, int32_t k2, const int64_t* sizes, size_t* off) {
  IEEE_REQUIRE(off, "gnn_stream_layout: null pointer");
  int rc = gnn_stream_check("gnn_stream_layout", Q, G, k1, k2);
  if (rc) return rc;
  const GnnScratch s = gnn_scratch_plan(Q, G, k1, 0);
  for (int i = 0; i < 4; ++i) off[i] = s.off_cntr[i];
  if (sizes) {
    const GnnWork w = gnn_work_plan(Q + G, k2, sizes[3], sizes[4], sizes[5]);
    const size_t o[6] = {w.off_b1c, w.off_b1v, w.off_a1c, w.off_a1v, w.off_b2c, w.off_b2v};
    for (int i = 0; i < 6; ++i) off[4 + i] = o[i];
  }
  return IEEE_OK;
}

// index of the graph calls (A0's row offsets, T0, K2inv; every process builds all of it), then the nnz of B1, A1, B2 and
// A2 of the owned rows; k2 == 1 has nothing to count (A2 = A0)
int gnn_stream_symbolic(const int32_t* rank, int64_t Q, int64_t G, int32_t k1, int32_t k2, int64_t q0, int64_t q1, int64_t g0,
                        int64_t g1, void* scratch, size_t scratch_bytes, cudaStream_t stream) {
  IEEE_REQUIRE(rank && scratch, "gnn_stream_symbolic: null pointer");
  int rc = gnn_stream_check("gnn_stream_symbolic", Q, G, k1, k2);
  if (rc) return rc;
  GnnRows own;
  if ((rc = gnn_owned("gnn_stream_symbolic", Q, G, q0, q1, g0, g1, &own))) return rc;
  IEEE_REQUIRE((reinterpret_cast<uintptr_t>(scratch) & 255) == 0, "gnn_stream_symbolic: scratch must be 256-byte aligned");
  const GnnScratch s = gnn_scratch_plan(Q, G, k1, 0);
  if (scratch_bytes < s.index) {
    set_error("gnn_stream_symbolic: scratch too small (%zu < %zu)", scratch_bytes, s.index);
    return IEEE_ERR_WORKSPACE;
  }
  if (k2 == 1) return IEEE_OK;
  const int64_t N = Q + G;
  const GnnIndex x = gnn_index(s, scratch);
  gnn_iota_kernel<<<(unsigned)((N + 256) / 256), 256, 0, stream>>>(x.a0p, N, k1);
  count_launch();
  if ((rc = gnn_rank_transpose(rank, N, k1, k1, x, x.t0p, x.t0i, stream))) return rc;
  if ((rc = gnn_rank_transpose(rank, N, k1, k2, x, x.k2p, x.k2i, stream))) return rc;
  const SpRows a0{x.a0p, rank, nullptr}, t0{x.t0p, x.t0i, nullptr}, k2inv{x.k2p, x.k2i, nullptr};
  const size_t smem = gnn_bitmap_smem(N);
  IEEE_ENSURE_DYN_SMEM(gnn_symbolic_kernel, smem);
  if (own.count())
    gnn_symbolic_kernel<<<(unsigned)own.count(), kGnnThreads, smem, stream>>>(a0, t0, k2inv, (int)N, k2, own, x.cntr[0], x.cntr[1],
                                                                              x.cntr[2], x.cntr[3]);
  if (own.count()) count_launch();
  IEEE_CUDA_CHECK(cudaGetLastError());
  return IEEE_OK;
}

// row offsets of B1, A1, B2, A2 from the counts of all N rows, and the one wait for their totals
int gnn_stream_sizes_sync(int64_t Q, int64_t G, int32_t k1, int32_t k2, void* scratch, size_t scratch_bytes, int64_t* sizes,
                          cudaStream_t stream) {
  IEEE_REQUIRE(scratch && sizes, "gnn_stream_sizes_sync: null pointer");
  int rc = gnn_stream_check("gnn_stream_sizes_sync", Q, G, k1, k2);
  if (rc) return rc;
  const GnnScratch s = gnn_scratch_plan(Q, G, k1, 0);
  if (scratch_bytes < s.index) {
    set_error("gnn_stream_sizes_sync: scratch too small (%zu < %zu)", scratch_bytes, s.index);
    return IEEE_ERR_WORKSPACE;
  }
  const int64_t N = Q + G;
  const GnnIndex x = gnn_index(s, scratch);
  int64_t tot[4] = {N * k1, N * k1, N * k1, N * k1};     // nnz of B1, A1, B2, A2 (k2 == 1: A2 = A0)
  int64_t nnz_gal = G * k1;
  if (k2 != 1) {
    for (int i = 0; i < 4; ++i) {
      gnn_scan64_kernel<<<1, 1024, 0, stream>>>(x.cntr[i], N, x.ptr[i]);
      count_launch();
    }
    int64_t host[5];
    for (int i = 0; i < 4; ++i) IEEE_CUDA_CHECK(cudaMemcpyAsync(host + i, x.ptr[i] + N, 8, cudaMemcpyDeviceToHost, stream));
    IEEE_CUDA_CHECK(cudaMemcpyAsync(host + 4, x.ptr[3] + Q, 8, cudaMemcpyDeviceToHost, stream));
    IEEE_CUDA_CHECK(cudaStreamSynchronize(stream));
    for (int i = 0; i < 4; ++i) tot[i] = host[i];
    nnz_gal = host[3] - host[4];
  }
  IEEE_REQUIRE(tot[3] < (int64_t(1) << 40), "gnn_stream_sizes_sync: nnz overflow");
  sizes[0] = tot[3];
  sizes[1] = nnz_gal;
  sizes[2] = (int64_t)gnn_work_plan(N, k2, tot[0], tot[1], tot[2]).total;
  sizes[3] = tot[0];
  sizes[4] = tot[1];
  sizes[5] = tot[2];
  return IEEE_OK;
}

int gnn_stream_graph_bytes_sync(const int32_t* rank, int64_t Q, int64_t G, int32_t k1, int32_t k2, void* scratch,
                                size_t scratch_bytes, int64_t* sizes, cudaStream_t stream) {
  IEEE_REQUIRE(sizes, "gnn_stream_graph_bytes_sync: null pointer");
  int rc = gnn_stream_symbolic(rank, Q, G, k1, k2, 0, Q, 0, G, scratch, scratch_bytes, stream);
  if (rc) return rc;
  return gnn_stream_sizes_sync(Q, G, k1, k2, scratch, scratch_bytes, sizes, stream);
}

// One step of the numeric phase over the owned rows: 0 B1 = A0 + A0^T, 1 A1 = P(B1), 2 A1^T (all rows, from the whole
// A1) and B2 = A1 + A1^T, 3 A2 = P(B2) (k2 == 1: A2 = A0) into a_ptr (all rows) and a_col / a_val.  When the owned rows
// are not all N rows, the entries of every other row are set to 0 (see gnn_col_sort_kernel).
int gnn_stream_numeric(int step, const int32_t* rank, const float* S, int64_t Q, int64_t G, int32_t k1, int32_t k2, int64_t q0,
                       int64_t q1, int64_t g0, int64_t g1, void* scratch, size_t scratch_bytes, void* work, size_t work_bytes,
                       const int64_t* sizes, int64_t* a_ptr, int32_t* a_col, float* a_val, cudaStream_t stream) {
  IEEE_REQUIRE(step >= 0 && step <= 3, "gnn_stream_numeric: step must be 0 to 3, got %d", step);
  IEEE_REQUIRE(rank && S && scratch && work && sizes && (step < 3 || (a_ptr && a_col && a_val)), "gnn_stream_numeric: null pointer");
  int rc = gnn_stream_check("gnn_stream_numeric", Q, G, k1, k2);
  if (rc) return rc;
  IEEE_REQUIRE(k2 != 1 || step == 3, "gnn_stream_numeric: with k2 = 1 there is only step 3 (A2 = A0), got step %d", step);
  GnnRows own;
  if ((rc = gnn_owned("gnn_stream_numeric", Q, G, q0, q1, g0, g1, &own))) return rc;
  IEEE_REQUIRE((reinterpret_cast<uintptr_t>(scratch) & 255) == 0 && (reinterpret_cast<uintptr_t>(work) & 255) == 0,
               "gnn_stream_numeric: scratch and work must be 256-byte aligned");
  const int64_t N = Q + G;
  const GnnScratch s = gnn_scratch_plan(Q, G, k1, 0);
  const GnnWork wp = gnn_work_plan(N, k2, sizes[3], sizes[4], sizes[5]);
  if (scratch_bytes < s.index || work_bytes < wp.total) {
    set_error("gnn_stream_numeric: scratch or work too small (%zu < %zu or %zu < %zu)", scratch_bytes, s.index, work_bytes,
              wp.total);
    return IEEE_ERR_WORKSPACE;
  }
  const bool part = own.count() != N;
  const unsigned rows = (unsigned)own.count();
  const GnnIndex x = gnn_index(s, scratch);
  const size_t smem = gnn_bitmap_smem(N);
  uint8_t* w = static_cast<uint8_t*>(work);
  int32_t* b1c = reinterpret_cast<int32_t*>(w + wp.off_b1c);
  float* b1v = reinterpret_cast<float*>(w + wp.off_b1v);
  int32_t* a1c = reinterpret_cast<int32_t*>(w + wp.off_a1c);
  float* a1v = reinterpret_cast<float*>(w + wp.off_a1v);
  int32_t* b2c = reinterpret_cast<int32_t*>(w + wp.off_b2c);
  float* b2v = reinterpret_cast<float*>(w + wp.off_b2v);
  auto clear = [&](void* col, void* val, int64_t nnz) -> int {
    if (part && nnz) {
      IEEE_CUDA_CHECK(cudaMemsetAsync(col, 0, size_t(nnz) * 4, stream));
      IEEE_CUDA_CHECK(cudaMemsetAsync(val, 0, size_t(nnz) * 4, stream));
    }
    return IEEE_OK;
  };
  IEEE_ENSURE_DYN_SMEM(gnn_sum_kernel, smem);
  IEEE_ENSURE_DYN_SMEM(gnn_propagate_rows_kernel, smem);
  if (step == 0) {            // B1 = A0 + A0^T
    if ((rc = clear(b1c, b1v, sizes[3]))) return rc;
    if (rows)
      gnn_sum_kernel<<<rows, kGnnThreads, smem, stream>>>(SpRows{x.a0p, rank, nullptr}, SpRows{x.t0p, x.t0i, nullptr}, (int)N, own,
                                                          x.ptr[0], b1c, b1v);
  } else if (step == 1) {     // A1 = P(B1)
    if ((rc = clear(a1c, a1v, sizes[4]))) return rc;
    if (rows)
      gnn_propagate_rows_kernel<<<rows, kGnnThreads, smem, stream>>>(SpRows{x.ptr[0], b1c, b1v}, rank, S, k1, k2, (int)N, own,
                                                                     x.ptr[1], a1c, a1v);
  } else if (step == 2) {     // B2 = A1 + A1^T
    int64_t* tp = reinterpret_cast<int64_t*>(w + wp.off_tp);
    int32_t* ti = reinterpret_cast<int32_t*>(w + wp.off_ti);
    float* tv = reinterpret_cast<float*>(w + wp.off_tv);
    const SpRows a1{x.ptr[1], a1c, a1v};
    if ((rc = gnn_sparse_transpose(a1, N, 0, (int)N, 0, x, tp, ti, tv, stream))) return rc;
    if ((rc = clear(b2c, b2v, sizes[5]))) return rc;
    if (rows) gnn_sum_kernel<<<rows, kGnnThreads, smem, stream>>>(a1, SpRows{tp, ti, tv}, (int)N, own, x.ptr[2], b2c, b2v);
  } else if (k2 == 1) {       // A2 = A0: the neighbour lists with ascending columns, all values 1
    gnn_iota_kernel<<<(unsigned)((N + 256) / 256), 256, 0, stream>>>(a_ptr, N, k1);
    count_launch();
    if ((rc = clear(a_col, a_val, sizes[0]))) return rc;
    if (rows)
      gnn_sum_kernel<<<rows, kGnnThreads, smem, stream>>>(SpRows{a_ptr, rank, nullptr}, SpRows{nullptr, nullptr, nullptr}, (int)N,
                                                          own, a_ptr, a_col, a_val);
  } else {                    // A2 = P(B2)
    IEEE_CUDA_CHECK(cudaMemcpyAsync(a_ptr, x.ptr[3], size_t(N + 1) * 8, cudaMemcpyDeviceToDevice, stream));
    if ((rc = clear(a_col, a_val, sizes[0]))) return rc;
    if (rows)
      gnn_propagate_rows_kernel<<<rows, kGnnThreads, smem, stream>>>(SpRows{x.ptr[2], b2c, b2v}, rank, S, k1, k2, (int)N, own,
                                                                     a_ptr, a_col, a_val);
  }
  count_launch();
  IEEE_CUDA_CHECK(cudaGetLastError());
  return IEEE_OK;
}

// the gallery rows of A2 (all of them) as CSC, rows ascending in the owned columns (the owned rows' indices)
int gnn_stream_csc(int64_t Q, int64_t G, int32_t k1, int64_t q0, int64_t q1, int64_t g0, int64_t g1, void* scratch,
                   size_t scratch_bytes, const int64_t* a_ptr, const int32_t* a_col, const float* a_val, int64_t* g_ptr,
                   int32_t* g_row, float* g_val, cudaStream_t stream) {
  IEEE_REQUIRE(scratch && a_ptr && a_col && a_val && g_ptr && g_row && g_val, "gnn_stream_csc: null pointer");
  int rc = gnn_stream_check("gnn_stream_csc", Q, G, k1, 1);
  if (rc) return rc;
  GnnRows own;
  if ((rc = gnn_owned("gnn_stream_csc", Q, G, q0, q1, g0, g1, &own))) return rc;
  IEEE_REQUIRE((reinterpret_cast<uintptr_t>(scratch) & 255) == 0, "gnn_stream_csc: scratch must be 256-byte aligned");
  const GnnScratch s = gnn_scratch_plan(Q, G, k1, 0);
  if (scratch_bytes < s.index) {
    set_error("gnn_stream_csc: scratch too small (%zu < %zu)", scratch_bytes, s.index);
    return IEEE_ERR_WORKSPACE;
  }
  const int64_t N = Q + G;
  const GnnIndex x = gnn_index(s, scratch);
  const SpRows a2{a_ptr, a_col, a_val};
  if ((rc = gnn_sparse_transpose(a2, N, (int)Q, (int)N, (int)Q, x, g_ptr, g_row, nullptr, stream))) return rc;
  const size_t gsmem = gnn_bitmap_smem(G);
  IEEE_ENSURE_DYN_SMEM(gnn_col_sort_kernel, gsmem);
  gnn_col_sort_kernel<<<(unsigned)N, kGnnThreads, gsmem, stream>>>(g_ptr, g_row, g_val, a2, (int)Q, (int)G, own);
  count_launch();
  IEEE_CUDA_CHECK(cudaGetLastError());
  return IEEE_OK;
}

int gnn_stream_graph(const int32_t* rank, const float* S, int64_t Q, int64_t G, int32_t k1, int32_t k2, void* scratch,
                     size_t scratch_bytes, void* work, size_t work_bytes, const int64_t* sizes, int64_t* a_ptr, int32_t* a_col,
                     float* a_val, int64_t* g_ptr, int32_t* g_row, float* g_val, cudaStream_t stream) {
  IEEE_REQUIRE(rank && S && scratch && work && sizes && a_ptr && a_col && a_val && g_ptr && g_row && g_val,
               "gnn_stream_graph: null pointer");
  int rc = gnn_stream_check("gnn_stream_graph", Q, G, k1, k2);
  if (rc) return rc;
  for (int step = k2 == 1 ? 3 : 0; step < 4; ++step)
    if ((rc = gnn_stream_numeric(step, rank, S, Q, G, k1, k2, 0, Q, 0, G, scratch, scratch_bytes, work, work_bytes, sizes, a_ptr,
                                 a_col, a_val, stream)))
      return rc;
  return gnn_stream_csc(Q, G, k1, 0, Q, 0, G, scratch, scratch_bytes, a_ptr, a_col, a_val, g_ptr, g_row, g_val, stream);
}

int gnn_stream_block(const int64_t* a_ptr, const int32_t* a_col, const float* a_val, const int64_t* g_ptr, const int32_t* g_row,
                     const float* g_val, int64_t Q, int64_t G, int64_t row0, int64_t rows, float* block, int64_t ld,
                     void* scratch, size_t scratch_bytes, cudaStream_t stream) {
  IEEE_REQUIRE(a_ptr && a_col && a_val && g_ptr && g_row && g_val && block && scratch, "gnn_stream_block: null pointer");
  IEEE_REQUIRE(Q > 0 && G > 0 && Q + G <= kGnnMaxN, "gnn_stream_block: bad shape Q=%lld G=%lld", (long long)Q, (long long)G);
  IEEE_REQUIRE(row0 >= 0 && rows >= 0 && row0 + rows <= Q && ld >= G, "gnn_stream_block: bad block rows [%lld, %lld) of %lld, ld=%lld",
               (long long)row0, (long long)(row0 + rows), (long long)Q, (long long)ld);
  if (scratch_bytes < size_t(rows) * size_t(G) * 8) {
    set_error("gnn_stream_block: scratch too small (%zu < %zu)", scratch_bytes, size_t(rows) * size_t(G) * 8);
    return IEEE_ERR_WORKSPACE;
  }
  if (rows == 0) return IEEE_OK;
  gnn_block_kernel<<<(unsigned)rows, kGnnThreads, 0, stream>>>(SpRows{a_ptr, a_col, a_val}, SpRows{g_ptr, g_row, g_val}, (int)G,
                                                                (int)row0, static_cast<double*>(scratch), block, ld);
  count_launch();
  IEEE_CUDA_CHECK(cudaGetLastError());
  return IEEE_OK;
}

}  // namespace ieee
