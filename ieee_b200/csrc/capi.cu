// extern "C" surface of libieee_b200.so (see include/ieee_b200.h).
#include <atomic>
#include <mutex>

#include "common.cuh"

namespace ieee {

static thread_local char g_error[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_error, sizeof(g_error), fmt, ap);
  va_end(ap);
}
const char* get_error() { return g_error; }

static std::atomic<long long> g_launches{0};
int g_debug_flags = 0;
int g_accum_chunk_kb = 6;
int g_raster_panel = 0;
static int g_centering = 1;

// Step timeline (debug flag 128): every named launch on the traced stream is followed by an event record, so the gaps
// between consecutive marks are kernel time + launch gap as they occur INSIDE a step (ncu serialises and cools the
// caches; this does not).  ieee_debug_timeline() formats the marks.
struct TlMark { cudaEvent_t ev; const char* name; };
static thread_local TlMark tl_marks[96];
static thread_local int tl_n = 0;
static thread_local cudaStream_t tl_stream = nullptr;
static thread_local bool tl_on = false;
static void tl_mark(const char* name) {
  if (!tl_on || tl_n >= 96) return;
  TlMark& m = tl_marks[tl_n];
  if (m.ev == nullptr && cudaEventCreate(&m.ev) != cudaSuccess) return;
  if (cudaEventRecord(m.ev, tl_stream) != cudaSuccess) return;
  m.name = name;
  ++tl_n;
}
static void tl_enter(cudaStream_t stream, const char* what) {
  tl_on = (g_debug_flags & 128) != 0;
  if (!tl_on) return;
  // a captured step gets no marks: they would be events of the capture, which the timeline cannot read back
  cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(stream, &cs) != cudaSuccess || cs != cudaStreamCaptureStatusNone) { tl_on = false; return; }
  tl_stream = stream;
  tl_mark(what);
}
void count_launch(int n, const char* name) {
  g_launches.fetch_add(n, std::memory_order_relaxed);
  if (name != nullptr && tl_on) tl_mark(name);
}

int sm_count() {
  static int cached[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (cached[dev] == 0) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    cached[dev] = n;
  }
  return cached[dev];
}

// implemented in the other translation units
int pack_features(const void* x, int dtype, int64_t ld, int64_t rows, int64_t D, int metric, int normalize, int precision,
                  const float* center, void* packed, cudaStream_t stream, const ZeroJob* zero = nullptr);
size_t feature_center_workspace_bytes(int64_t D);
int feature_center(const void* x, int dtype, int64_t ld, int64_t rows, int64_t D, int normalize, int64_t max_rows,
                   float* center, void* workspace, cudaStream_t stream);
int distmat_umma(const void* q_packed, int64_t Q, const void* g_packed, int64_t G, int64_t D, int metric, int precision,
                 float* out, int64_t ldo, cudaStream_t stream, int cta_group, void* fix_ws, bool fix_zeroed = false);
size_t distmat_fixup_bytes(int64_t Q);
int distmat_simt(const void* q_packed, int64_t Q, const void* g_packed, int64_t G, int64_t D, int metric, float* out,
                 int64_t ldo, cudaStream_t stream);
size_t gallery_group_bytes(int64_t G);
int gallery_group(const int64_t* g_pids, int64_t G, void* blob, cudaStream_t stream);
int rank_list_cap(const void* group, int64_t G, const int64_t* q_pids, int64_t Q, int32_t* cap_dev, cudaStream_t stream);
int rank_gather(const float* distmat, int64_t ld, int64_t Q, int64_t G, const int64_t* q_pids, const int64_t* q_camids,
                const int64_t* g_camids, const void* group, int64_t g_offset, int32_t cap, uint64_t* rel, int32_t* n_rel,
                uint64_t* junk, int32_t* n_junk, int32_t* overflow, cudaStream_t stream, const PeerView* peers = nullptr);
size_t rank_count_smem(int shards, int cap);
int set_count_team(int wpq);
int rank_count(const float* distmat, int64_t ld, int64_t Q, int64_t G, int64_t g_offset, int shards, int cap, int out_cap,
               const uint64_t* rel_all, const int32_t* n_rel, const uint64_t* junk, const int32_t* n_junk,
               int32_t* counts, unsigned long long* ties, cudaStream_t stream, const PeerView* peers = nullptr);
int rank_metrics_peer(const PeerView* peers, int64_t G_total, int32_t max_rank, const unsigned long long* local_stats,
                      float* cmc, ieee_eval_summary* summary, long long* stats_out, int64_t Qtot, cudaStream_t stream,
                      double* ap_out = nullptr, int32_t* first_out = nullptr);
int rank_count_f64(const double* distmat, int64_t ld, int64_t Q, int64_t G, const int64_t* q_pids, const int64_t* q_camids,
                   const int64_t* g_camids, const void* group, int32_t cap, int32_t* counts, unsigned long long* ties,
                   int32_t* overflow, cudaStream_t stream);
size_t rank_finalize_workspace_bytes(int64_t Q);
int rank_query_metrics(const int32_t* counts, int64_t Q, int64_t G_total, int32_t shards, int32_t cap,
                       int32_t max_rank, double* ap, int32_t* first, int32_t* short_list, double* inp,
                       cudaStream_t stream);
int rank_reduce(const double* ap, const int32_t* first, const int32_t* short_list, int64_t Q, int32_t max_rank,
                const unsigned long long* ties, float* cmc, ieee_eval_summary* summary, const double* inp,
                const int32_t* overflow, cudaStream_t stream, const PeerView* peers = nullptr, long long* stats_out = nullptr);
int rank_finalize(const int32_t* counts, int64_t Q, int64_t G_total, int32_t shards, int32_t cap,
                  int32_t max_rank, const unsigned long long* ties, float* cmc, ieee_eval_summary* summary,
                  double* per_query_ap, int32_t* per_query_first, void* workspace, cudaStream_t stream,
                  const int32_t* overflow = nullptr, uint32_t* ticket = nullptr);
int topk(const float* distmat, int64_t ld, int64_t Q, int64_t G, int64_t g_offset, const int64_t* q_pids,
         const int64_t* q_camids, const int64_t* g_pids, const int64_t* g_camids, int32_t k, int32_t* idx, float* val,
         cudaStream_t stream);
int topk_merge(const int32_t* idx_all, const float* val_all, int32_t shards, int64_t Q, int32_t k, int32_t* idx, float* val,
               cudaStream_t stream);
size_t rerank_workspace_bytes(int64_t Q, int64_t G, int32_t k1, int32_t k2);
int rerank(const float* q_g, int64_t ld_qg, const float* q_q, int64_t ld_qq, const float* g_g, int64_t ld_gg, int64_t Q,
           int64_t G, int32_t k1, int32_t k2, double lambda_value, float* out, int64_t ldo, void* workspace,
           size_t workspace_bytes, cudaStream_t stream);

size_t rerank_stream_workspace_bytes(int64_t Q, int64_t G, int32_t k1, int32_t k2);
size_t rerank_stream_scratch_bytes(int64_t Q, int64_t G, int32_t k1, size_t strip_bytes);
int rerank_stream_prepare(const void* q_packed, int64_t Q, const void* g_packed, int64_t G, int64_t D, int metric,
                          int precision, int32_t k1, int32_t k2, size_t strip_bytes, float* colmax, int32_t* rank,
                          void* workspace, size_t workspace_bytes, void* scratch, size_t scratch_bytes, cudaStream_t stream,
                          int cta_group);
int rerank_stream_block(const void* workspace, int64_t Q, int64_t G, int32_t k1, int32_t k2, const float* colmax, int64_t row0,
                        int64_t rows, double lambda_value, float* block, int64_t ld, void* scratch, size_t scratch_bytes,
                        cudaStream_t stream);
size_t rerank_stream_window_workspace_bytes(int64_t Q, int64_t G, int32_t k1, int32_t k2, int64_t Gs);
int rerank_stream_v_layout(int64_t Q, int64_t G, int32_t k1, int32_t k2, int64_t* cap, size_t* off_col, size_t* off_val,
                           size_t* off_cnt);
int rerank_stream_pass(int pass, const void* q_packed, int64_t Q, const void* g_packed, int64_t G, int64_t D, int metric,
                       int precision, int32_t k1, int32_t k2, size_t strip_bytes, int64_t q0, int64_t q1, int64_t g0, int64_t g1,
                       float* colmax, int32_t* rank, void* workspace, size_t workspace_bytes, void* scratch, size_t scratch_bytes,
                       cudaStream_t stream, int cta_group);
int rerank_stream_finish(void* workspace, size_t workspace_bytes, int64_t Q, int64_t G, int32_t k1, int32_t k2, int64_t g0,
                         int64_t Gs, const int32_t* rank, cudaStream_t stream);
int rerank_stream_block_window(const void* workspace, int64_t Q, int64_t G, int32_t k1, int32_t k2, int64_t Gs,
                               const float* colmax, int64_t row0, int64_t rows, double lambda_value, float* block, int64_t ld,
                               void* scratch, size_t scratch_bytes, cudaStream_t stream);
int64_t rerank_stream_part_width(int64_t Q, int64_t G, int32_t k1, int64_t qa, int64_t qb, int64_t ga, int64_t gb,
                                 size_t strip_bytes);
size_t rerank_stream_part_scratch_bytes(int64_t Q, int64_t G, int32_t k1, int64_t qa, int64_t qb, int64_t ga, int64_t gb,
                                        int64_t W);
int rerank_stream_part_contract(int pass, const void* q_packed, int64_t Q, const void* g_part, const void* g_strip, int64_t G,
                                int64_t D, int metric, int precision, int32_t k1, int64_t qa, int64_t qb, int64_t ga, int64_t gb,
                                int64_t W, int64_t i0, int64_t wc, float* colmax, void* scratch, size_t scratch_bytes,
                                cudaStream_t stream, int cta_group);
int rerank_stream_part_topk(int64_t Q, int64_t G, int32_t k1, int64_t qa, int64_t qb, int64_t ga, int64_t gb, int64_t W,
                            int64_t i0, int64_t wc, const float* colmax, int32_t* idx, float* val, void* scratch,
                            size_t scratch_bytes, cudaStream_t stream);
int rerank_stream_part_members(int64_t Q, int64_t G, int32_t k1, int32_t k2, int64_t qa, int64_t qb, int64_t ga, int64_t gb,
                               int64_t W, int64_t i0, int64_t wc, const float* colmax, void* workspace, size_t workspace_bytes,
                               const void* scratch, size_t scratch_bytes, cudaStream_t stream);
int rerank_stream_part_weights(void* workspace, size_t workspace_bytes, int64_t Q, int64_t G, int32_t k1, int32_t k2,
                               int64_t row0, int64_t rows, cudaStream_t stream);

size_t gnn_rerank_workspace_bytes(int64_t N, int32_t k1);
int gnn_rerank(const float* neg_score, int64_t lds, int64_t N, int32_t k1, int32_t k2, float* A, int64_t ldA, void* workspace,
               size_t workspace_bytes, cudaStream_t stream);
size_t gnn_stream_scratch_bytes(int64_t Q, int64_t G, int32_t k1, size_t strip_bytes);
int gnn_stream_neighbours(const void* q_packed, int64_t Q, const void* g_packed, int64_t G, int64_t D, int precision, int32_t k1,
                          size_t strip_bytes, int32_t* rank, float* S, void* scratch, size_t scratch_bytes, cudaStream_t stream,
                          int cta_group);
int gnn_stream_graph_bytes_sync(const int32_t* rank, int64_t Q, int64_t G, int32_t k1, int32_t k2, void* scratch,
                                size_t scratch_bytes, int64_t* sizes, cudaStream_t stream);
int gnn_stream_graph(const int32_t* rank, const float* S, int64_t Q, int64_t G, int32_t k1, int32_t k2, void* scratch,
                     size_t scratch_bytes, void* work, size_t work_bytes, const int64_t* sizes, int64_t* a_ptr, int32_t* a_col,
                     float* a_val, int64_t* g_ptr, int32_t* g_row, float* g_val, cudaStream_t stream);
int gnn_stream_neighbours_rows(const void* q_packed, int64_t Q, const void* g_packed, int64_t G, int64_t D, int precision,
                               int32_t k1, size_t strip_bytes, int64_t q0, int64_t q1, int64_t g0, int64_t g1, int32_t* rank,
                               float* S, void* scratch, size_t scratch_bytes, cudaStream_t stream, int cta_group);
int gnn_stream_layout(int64_t Q, int64_t G, int32_t k1, int32_t k2, const int64_t* sizes, size_t* off);
int gnn_stream_symbolic(const int32_t* rank, int64_t Q, int64_t G, int32_t k1, int32_t k2, int64_t q0, int64_t q1, int64_t g0,
                        int64_t g1, void* scratch, size_t scratch_bytes, cudaStream_t stream);
int gnn_stream_sizes_sync(int64_t Q, int64_t G, int32_t k1, int32_t k2, void* scratch, size_t scratch_bytes, int64_t* sizes,
                          cudaStream_t stream);
int gnn_stream_numeric(int step, const int32_t* rank, const float* S, int64_t Q, int64_t G, int32_t k1, int32_t k2, int64_t q0,
                       int64_t q1, int64_t g0, int64_t g1, void* scratch, size_t scratch_bytes, void* work, size_t work_bytes,
                       const int64_t* sizes, int64_t* a_ptr, int32_t* a_col, float* a_val, cudaStream_t stream);
int gnn_stream_csc(int64_t Q, int64_t G, int32_t k1, int64_t q0, int64_t q1, int64_t g0, int64_t g1, void* scratch,
                   size_t scratch_bytes, const int64_t* a_ptr, const int32_t* a_col, const float* a_val, int64_t* g_ptr,
                   int32_t* g_row, float* g_val, cudaStream_t stream);
int gnn_stream_block(const int64_t* a_ptr, const int32_t* a_col, const float* a_val, const int64_t* g_ptr, const int32_t* g_row,
                     const float* g_val, int64_t Q, int64_t G, int64_t row0, int64_t rows, float* block, int64_t ld,
                     void* scratch, size_t scratch_bytes, cudaStream_t stream);

static int g_cta_group = -1;   // IEEE_B200_CTA_GROUP=1|2 overrides the default (2) pairing of the tensor-core kernel
static int cta_group_default() {
  if (g_cta_group < 0) {
    const char* e = getenv("IEEE_B200_CTA_GROUP");
    g_cta_group = (e && e[0] == '1') ? 1 : 2;
  }
  return g_cta_group;
}

static int check_device() {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) {
    cudaGetLastError();
    set_error("no CUDA device available (libieee_b200 has no CPU fallback)");
    return IEEE_ERR_CUDA;
  }
  return IEEE_OK;
}

// bump allocator over a caller-provided workspace
struct Arena {
  uint8_t* base;
  size_t size, off;
  void* take(size_t bytes) {
    size_t o = align256(off);
    if (o + bytes > size) return nullptr;
    off = o + bytes;
    return base + o;
  }
};


struct SideLane { cudaStream_t stream = nullptr; cudaEvent_t fork = nullptr, join = nullptr; };
static SideLane g_side[64];
static std::mutex g_side_mutex;
static int side_lane(SideLane** out) {
  int dev = 0;
  IEEE_CUDA_CHECK(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64) { set_error("device index %d out of range", dev); return IEEE_ERR_CUDA; }
  std::lock_guard<std::mutex> lock(g_side_mutex);
  SideLane& l = g_side[dev];
  if (l.stream == nullptr) {
    // highest priority: the lane's tiny label-only kernels get the SM slots the bandwidth-bound kernel beside them
    // frees, instead of queueing behind its remaining waves
    int lo = 0, hi = 0;
    IEEE_CUDA_CHECK(cudaDeviceGetStreamPriorityRange(&lo, &hi));
    IEEE_CUDA_CHECK(cudaStreamCreateWithPriority(&l.stream, cudaStreamNonBlocking, hi));
    IEEE_CUDA_CHECK(cudaEventCreateWithFlags(&l.fork, cudaEventDisableTiming));
    IEEE_CUDA_CHECK(cudaEventCreateWithFlags(&l.join, cudaEventDisableTiming));
  }
  *out = &l;
  return IEEE_OK;
}
// `stream` waits for whatever the side lane of the current device was last given (nothing, if it was never used)
static int side_lane_join(cudaStream_t stream) {
  int dev = 0;
  IEEE_CUDA_CHECK(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64) return IEEE_OK;
  cudaEvent_t join = nullptr;
  {
    std::lock_guard<std::mutex> lock(g_side_mutex);
    join = g_side[dev].join;
  }
  if (join == nullptr) return IEEE_OK;
  // under stream capture the event was recorded outside the capture: the graph gets an external wait node, so every
  // replay waits for whatever the side lane was last given, as an eager call does
  cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
  IEEE_CUDA_CHECK(cudaStreamIsCapturing(stream, &cs));
  IEEE_CUDA_CHECK(cudaStreamWaitEvent(stream, join, cs == cudaStreamCaptureStatusActive ? cudaEventWaitExternal : 0));
  return IEEE_OK;
}
}  // namespace ieee

using namespace ieee;

extern "C" {

const char* ieee_last_error(void) { return get_error(); }
int ieee_abi_version(void) { return IEEE_B200_ABI_VERSION; }

int ieee_device_info(int* sm, int* cc) {
  int rc = check_device();
  if (rc) return rc;
  int dev = 0, major = 0, minor = 0;
  IEEE_CUDA_CHECK(cudaGetDevice(&dev));
  IEEE_CUDA_CHECK(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
  IEEE_CUDA_CHECK(cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev));
  if (sm) *sm = sm_count();
  if (cc) *cc = major * 10 + minor;
  return IEEE_OK;
}

int64_t ieee_launch_count(void) { return g_launches.load(); }

int ieee_set_accum_chunk(int k_slices) {
  const int prev = g_accum_chunk_kb;
  if (k_slices >= 0) g_accum_chunk_kb = k_slices;
  return prev;
}

int ieee_set_debug_flags(int flags) {
  const int prev = g_debug_flags;
  g_debug_flags = flags;
  return prev;
}

int64_t ieee_note_launches(int64_t n) { return g_launches.fetch_add(n) + n; }

void ieee_debug_timeline_reset(void) { tl_n = 0; }

// "name<TAB>us since the previous mark<TAB>us since the first mark" per line; returns the number of marks
int ieee_debug_timeline(char* buf, size_t cap) {
  if (buf && cap) buf[0] = 0;
  if (tl_n == 0) return 0;
  if (cudaEventSynchronize(tl_marks[tl_n - 1].ev) != cudaSuccess) return -1;
  size_t off = 0;
  for (int i = 0; i < tl_n; ++i) {
    float d = 0.f, t = 0.f;
    if (i > 0) cudaEventElapsedTime(&d, tl_marks[i - 1].ev, tl_marks[i].ev);
    cudaEventElapsedTime(&t, tl_marks[0].ev, tl_marks[i].ev);
    if (buf && off < cap) off += (size_t)snprintf(buf + off, cap - off, "%s\t%.1f\t%.1f\n", tl_marks[i].name, d * 1e3f, t * 1e3f);
  }
  return tl_n;
}

int ieee_set_raster_panel(int m_tiles) {
  const int prev = g_raster_panel;
  if (m_tiles >= 0) g_raster_panel = m_tiles;
  return prev;
}

int ieee_set_centering(int on) {
  const int prev = g_centering;
  if (on >= 0) g_centering = on ? 1 : 0;
  return prev;
}

int ieee_set_count_team(int warps_per_query) { return set_count_team(warps_per_query); }

int ieee_set_cta_group(int cg) {
  const int prev = cta_group_default();
  if (cg == 1 || cg == 2) g_cta_group = cg;
  return prev;
}

// ---- distance ------------------------------------------------------------------------------------------
size_t ieee_packed_bytes(int64_t rows, int64_t D, int precision) {
  if (rows < 0 || D <= 0) return 0;
  return packed_layout(rows, D, precision).total;
}

int ieee_packed_copy_rows(const void* src, int64_t src_rows, int64_t src_r0, void* dst, int64_t dst_rows, int64_t dst_r0,
                          int64_t n, int64_t D, int precision, ieee_stream_t stream) {
  IEEE_REQUIRE(src && dst, "packed_copy_rows: null pointer");
  IEEE_REQUIRE(D > 0 && precision >= 0 && precision <= IEEE_PREC_FP32_SIMT, "packed_copy_rows: bad D=%lld or precision %d",
               (long long)D, precision);
  IEEE_REQUIRE(n >= 0 && src_r0 >= 0 && src_r0 + n <= src_rows && dst_r0 >= 0 && dst_r0 + n <= dst_rows,
               "packed_copy_rows: rows [%lld, %lld) of %lld to [%lld, %lld) of %lld", (long long)src_r0, (long long)(src_r0 + n),
               (long long)src_rows, (long long)dst_r0, (long long)(dst_r0 + n), (long long)dst_rows);
  if (n == 0) return IEEE_OK;
  const PackedRows a = packed_rows(src, src_rows, src_r0, n, D, precision), b = packed_rows(dst, dst_rows, dst_r0, n, D, precision);
  const size_t plane = size_t(n) * size_t(a.Dp) * (precision == IEEE_PREC_FP32_SIMT ? 4 : 2);
  cudaStream_t st = (cudaStream_t)stream;
  IEEE_CUDA_CHECK(cudaMemcpyAsync(const_cast<uint8_t*>(b.hi), a.hi, plane, cudaMemcpyDeviceToDevice, st));
  if (precision == IEEE_PREC_F16X3)
    IEEE_CUDA_CHECK(cudaMemcpyAsync(const_cast<uint8_t*>(b.lo), a.lo, plane, cudaMemcpyDeviceToDevice, st));
  IEEE_CUDA_CHECK(cudaMemcpyAsync(const_cast<float*>(b.norm), a.norm, size_t(n) * 4, cudaMemcpyDeviceToDevice, st));
  IEEE_CUDA_CHECK(cudaMemcpyAsync(const_cast<float*>(b.scale), a.scale, size_t(n) * 4, cudaMemcpyDeviceToDevice, st));
  return IEEE_OK;
}

int ieee_pack_features(const void* x, int dtype, int64_t ld, int64_t rows, int64_t D, int metric, int normalize,
                       int precision, const float* center, void* packed, ieee_stream_t stream) {
  int rc = check_device();
  if (rc) return rc;
  return pack_features(x, dtype, ld, rows, D, metric, normalize, precision, center, packed, (cudaStream_t)stream);
}

size_t ieee_feature_center_workspace_bytes(int64_t D) { return D > 0 ? feature_center_workspace_bytes(D) : 0; }

int ieee_feature_center(const void* x, int dtype, int64_t ld, int64_t rows, int64_t D, int normalize, int64_t max_rows,
                        float* center, void* workspace, ieee_stream_t stream) {
  int rc = check_device();
  if (rc) return rc;
  return feature_center(x, dtype, ld, rows, D, normalize, max_rows, center, workspace, (cudaStream_t)stream);
}

// whether the one-call entry points centre the operands themselves: euclidean only (cosine is not translation
// invariant), and not the 1-pass BF16 mode (bf16 inputs multiply exactly as they are)
static bool auto_center(int metric, int precision) {
  return g_centering && metric == IEEE_METRIC_EUCLIDEAN && precision != IEEE_PREC_BF16;
}
static size_t center_bytes(int64_t D) { return align256(size_t(D) * 4) + feature_center_workspace_bytes(D); }

size_t ieee_distmat_fixup_bytes(int64_t Q) { return Q > 0 ? distmat_fixup_bytes(Q) : 0; }

static int distmat_packed(const void* q_packed, int64_t Q, const void* g_packed, int64_t G, int64_t D, int metric,
                          int precision, float* out, int64_t ldo, void* fixup_workspace, ieee_stream_t stream, bool fix_zeroed) {
  int rc = check_device();
  if (rc) return rc;
  IEEE_REQUIRE(q_packed && g_packed && out, "distmat: null pointer");
  IEEE_REQUIRE(Q >= 0 && G >= 0 && D > 0 && ldo >= G, "distmat: bad shape Q=%lld G=%lld D=%lld ldo=%lld", (long long)Q,
               (long long)G, (long long)D, (long long)ldo);
  IEEE_REQUIRE(Q < (int64_t(1) << 31) && G < (int64_t(1) << 31), "distmat: Q and G must fit int32");
  IEEE_REQUIRE(metric >= IEEE_METRIC_EUCLIDEAN && metric <= IEEE_METRIC_NEG_DOT, "unknown metric %d", metric);
  if (Q == 0 || G == 0) return IEEE_OK;
  if (precision == IEEE_PREC_FP32_SIMT) return distmat_simt(q_packed, Q, g_packed, G, D, metric, out, ldo, (cudaStream_t)stream);
  IEEE_REQUIRE(precision == IEEE_PREC_F16X3 || precision == IEEE_PREC_BF16, "unknown precision %d", precision);
  IEEE_REQUIRE((reinterpret_cast<uintptr_t>(fixup_workspace) & 7) == 0, "distmat: fix-up workspace must be 8-byte aligned");
  return distmat_umma(q_packed, Q, g_packed, G, D, metric, precision, out, ldo, (cudaStream_t)stream, cta_group_default(),
                      fixup_workspace, fix_zeroed);
}

int ieee_distmat_packed(const void* q_packed, int64_t Q, const void* g_packed, int64_t G, int64_t D, int metric,
                        int precision, float* out, int64_t ldo, void* fixup_workspace, ieee_stream_t stream) {
  return distmat_packed(q_packed, Q, g_packed, G, D, metric, precision, out, ldo, fixup_workspace, stream, false);
}

size_t ieee_distmat_workspace_bytes(int64_t Q, int64_t G, int64_t D, int precision) {
  return align256(ieee_packed_bytes(Q, D, precision)) + align256(ieee_packed_bytes(G, D, precision)) + center_bytes(D) +
         distmat_fixup_bytes(Q) + 512;
}

int ieee_distmat(const void* q, const void* g, int dtype, int64_t ldq, int64_t ldg, int64_t Q, int64_t G, int64_t D,
                 int metric, int normalize, int precision, float* out, int64_t ldo, void* workspace, size_t workspace_bytes,
                 ieee_stream_t stream) {
  int rc = check_device();
  if (rc) return rc;
  IEEE_REQUIRE(workspace != nullptr && (reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "distmat: workspace must be 256-byte aligned");
  if (workspace_bytes < ieee_distmat_workspace_bytes(Q, G, D, precision)) {
    set_error("distmat: workspace too small (%zu < %zu)", workspace_bytes, ieee_distmat_workspace_bytes(Q, G, D, precision));
    return IEEE_ERR_WORKSPACE;
  }
  uint8_t* w = static_cast<uint8_t*>(workspace);
  void* qp = w;
  void* gp = w + align256(ieee_packed_bytes(Q, D, precision));
  float* center = nullptr;
  uint8_t* cbase = static_cast<uint8_t*>(gp) + align256(ieee_packed_bytes(G, D, precision));
  void* fix = cbase + center_bytes(D);
  if (auto_center(metric, precision) && Q > 0 && G > 0) {
    // centre of the first operand (a sample of its rows): both sides are packed relative to it
    center = reinterpret_cast<float*>(cbase);
    void* cws = cbase + align256(size_t(D) * 4);
    if ((rc = feature_center(q, dtype, ldq, Q, D, normalize, 0, center, cws, (cudaStream_t)stream))) return rc;
  }
  if ((rc = ieee_pack_features(q, dtype, ldq, Q, D, metric, normalize, precision, center, qp, stream))) return rc;
  if ((rc = ieee_pack_features(g, dtype, ldg, G, D, metric, normalize, precision, center, gp, stream))) return rc;
  return ieee_distmat_packed(qp, Q, gp, G, D, metric, precision, out, ldo, fix, stream);
}

// ---- ranking -------------------------------------------------------------------------------------------
size_t ieee_gallery_group_bytes(int64_t G) { return G > 0 ? gallery_group_bytes(G) : 0; }

int ieee_gallery_group(const int64_t* g_pids, int64_t G, void* group, ieee_stream_t stream) {
  int rc = check_device();
  if (rc) return rc;
  return gallery_group(g_pids, G, group, (cudaStream_t)stream);
}

int ieee_rank_list_cap(const void* group, int64_t G, const int64_t* q_pids, int64_t Q, int32_t* cap_dev, ieee_stream_t stream) {
  int rc = check_device();
  if (rc) return rc;
  IEEE_REQUIRE(group && q_pids && cap_dev, "rank_list_cap: null pointer");
  return rank_list_cap(group, G, q_pids, Q, cap_dev, (cudaStream_t)stream);
}

int ieee_rank_list_cap_sync(const void* group, int64_t G, const int64_t* q_pids, int64_t Q, int32_t* scratch_dev,
                            int32_t* cap_host, ieee_stream_t stream) {
  int rc = check_device();
  if (rc) return rc;
  IEEE_REQUIRE(group && q_pids && scratch_dev && cap_host, "rank_list_cap: null pointer");
  if ((rc = rank_list_cap(group, G, q_pids, Q, scratch_dev, (cudaStream_t)stream))) return rc;
  IEEE_CUDA_CHECK(cudaMemcpyAsync(cap_host, scratch_dev, 4, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  IEEE_CUDA_CHECK(cudaStreamSynchronize((cudaStream_t)stream));
  return IEEE_OK;
}

int ieee_rank_gather(const float* distmat, int64_t ld, int64_t Q, int64_t G, const int64_t* q_pids, const int64_t* q_camids,
                     const int64_t* g_camids, const void* group, int64_t g_offset, int32_t cap, uint64_t* rel,
                     int32_t* n_rel, uint64_t* junk, int32_t* n_junk, int32_t* overflow_flag, ieee_stream_t stream) {
  int rc = check_device();
  if (rc) return rc;
  return rank_gather(distmat, ld, Q, G, q_pids, q_camids, g_camids, group, g_offset, cap, rel, n_rel, junk, n_junk,
                     overflow_flag, (cudaStream_t)stream);
}

size_t ieee_rank_count_smem_bytes(int32_t shards, int32_t cap) { return rank_count_smem(shards, cap); }

int ieee_rank_count(const float* distmat, int64_t ld, int64_t Q, int64_t G, int64_t g_offset, int32_t shards, int32_t cap,
                    int32_t out_cap, const uint64_t* rel_all, const int32_t* n_rel, const uint64_t* junk, const int32_t* n_junk,
                    int32_t* counts, unsigned long long* ties, ieee_stream_t stream) {
  int rc = check_device();
  if (rc) return rc;
  return rank_count(distmat, ld, Q, G, g_offset, shards, cap, out_cap, rel_all, n_rel, junk, n_junk, counts, ties,
                    (cudaStream_t)stream);
}

int ieee_rank_query_metrics(const int32_t* counts, int64_t Q, int64_t G_total, int32_t shards,
                            int32_t cap, int32_t max_rank, double* ap, int32_t* first, int32_t* short_list,
                            double* inp, ieee_stream_t stream) {
  int rc = check_device();
  if (rc) return rc;
  return rank_query_metrics(counts, Q, G_total, shards, cap, max_rank, ap, first, short_list, inp, (cudaStream_t)stream);
}

int ieee_rank_reduce(const double* ap, const int32_t* first, const int32_t* short_list, int64_t Q, int32_t max_rank,
                     const unsigned long long* ties, float* cmc, ieee_eval_summary* summary, const double* inp,
                     ieee_stream_t stream) {
  int rc = check_device();
  if (rc) return rc;
  return rank_reduce(ap, first, short_list, Q, max_rank, ties, cmc, summary, inp, nullptr, (cudaStream_t)stream);
}

size_t ieee_rank_finalize_workspace_bytes(int64_t Q) { return Q > 0 ? rank_finalize_workspace_bytes(Q) : 0; }

int ieee_rank_finalize(const int32_t* counts, int64_t Q, int64_t G_total, int32_t shards,
                       int32_t cap, int32_t max_rank, const unsigned long long* ties, float* cmc, ieee_eval_summary* summary,
                       double* per_query_ap, int32_t* per_query_first, void* workspace, ieee_stream_t stream) {
  int rc = check_device();
  if (rc) return rc;
  return rank_finalize(counts, Q, G_total, shards, cap, max_rank, ties, cmc, summary, per_query_ap,
                       per_query_first, workspace, (cudaStream_t)stream);
}

// workspace of the one-shot evaluate: group | cap scratch | rel | junk | n_rel | n_junk | counts | ties | finalize ws
size_t ieee_eval_workspace_bytes(int64_t Q, int64_t G, int32_t cap) {
  if (Q <= 0 || G <= 0) return 0;
  if (cap <= 0) cap = (int32_t)(G < 4096 ? G : 4096);
  size_t b = 0;
  b += align256(gallery_group_bytes(G));
  b += 256;                                        // cap scratch + overflow flag + ties
  b += 2 * align256(size_t(Q) * (cap + 1) * 8);    // rel (+ embedded count), junk
  b += 2 * align256(size_t(Q) * 4);                // n_rel, n_junk
  b += align256(size_t(Q) * (cap + 2) * 4);        // counts
  b += align256(rank_finalize_workspace_bytes(Q));
  return b + 256;
}

int ieee_eval_market1501(const float* distmat, int64_t ld, int64_t Q, int64_t G, const int64_t* q_pids,
                         const int64_t* g_pids, const int64_t* q_camids, const int64_t* g_camids, int32_t max_rank,
                         int32_t cap, float* cmc, ieee_eval_summary* summary, void* workspace, size_t workspace_bytes,
                         ieee_stream_t stream_) {
  int rc = check_device();
  if (rc) return rc;
  cudaStream_t stream = (cudaStream_t)stream_;
  IEEE_REQUIRE(distmat && q_pids && g_pids && q_camids && g_camids && cmc && summary && workspace, "eval: null pointer");
  IEEE_REQUIRE(Q > 0 && G > 0 && ld >= G && max_rank >= 1, "eval: bad shape Q=%lld G=%lld ld=%lld max_rank=%d", (long long)Q,
               (long long)G, (long long)ld, max_rank);
  IEEE_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "eval: workspace must be 256-byte aligned");
  Arena a{static_cast<uint8_t*>(workspace), workspace_bytes, 0};
  void* group = a.take(gallery_group_bytes(G));
  int32_t* scratch = static_cast<int32_t*>(a.take(256));   // [0] cap, [1] overflow, [2..3] ties (u64)
  if (!group || !scratch) { set_error("eval: workspace too small"); return IEEE_ERR_WORKSPACE; }
  if ((rc = gallery_group(g_pids, G, group, stream))) return rc;
  int32_t need = 0;
  if ((rc = ieee_rank_list_cap_sync(group, G, q_pids, Q, scratch, &need, stream_))) return rc;
  if (need < 1) need = 1;
  if (cap <= 0) cap = need;
  if (need > cap) {
    set_error("eval: a query has %d same-identity gallery items but list capacity is %d", need, cap);
    return IEEE_ERR_CAPACITY;
  }
  cap = need;   // tight lists: less shared memory in the count kernel
  uint64_t* rel = static_cast<uint64_t*>(a.take(size_t(Q) * (cap + 1) * 8));
  uint64_t* junk = static_cast<uint64_t*>(a.take(size_t(Q) * cap * 8));
  int32_t* n_rel = static_cast<int32_t*>(a.take(size_t(Q) * 4));
  int32_t* n_junk = static_cast<int32_t*>(a.take(size_t(Q) * 4));
  int32_t* counts = static_cast<int32_t*>(a.take(size_t(Q) * (cap + 2) * 4));
  void* fws = a.take(rank_finalize_workspace_bytes(Q));
  if (!rel || !junk || !n_rel || !n_junk || !counts || !fws) {
    set_error("eval: workspace too small (%zu bytes given, need %zu for cap=%d)", workspace_bytes,
              ieee_eval_workspace_bytes(Q, G, cap), cap);
    return IEEE_ERR_WORKSPACE;
  }
  IEEE_CUDA_CHECK(cudaMemsetAsync(scratch, 0, 256, stream));
  unsigned long long* ties = reinterpret_cast<unsigned long long*>(scratch + 2);
  if ((rc = rank_gather(distmat, ld, Q, G, q_pids, q_camids, g_camids, group, 0, cap, rel, n_rel, junk, n_junk, scratch + 1, stream))) return rc;
  if ((rc = rank_count(distmat, ld, Q, G, 0, 1, cap, 0, rel, n_rel, junk, n_junk, counts, ties, stream))) return rc;
  return rank_finalize(counts, Q, G, 1, cap, max_rank, ties, cmc, summary, nullptr, nullptr, fws, stream, nullptr,
                       reinterpret_cast<uint32_t*>(scratch + 8));
}

// ---- gallery preparation in one call ----------------------------------------------------------------------
// A side stream per device for work that only depends on the labels (the grouping's tiny kernels run beside the
// bandwidth-bound feature packing instead of in front of it).

size_t ieee_gallery_prepare_workspace_bytes(int64_t D) { return D > 0 ? feature_center_workspace_bytes(D) : 0; }

int ieee_gallery_prepare(const void* gf, int64_t ldg, int dtype, int64_t G, int64_t D, int metric, int normalize, int precision,
                         const int64_t* g_pids, const void* q, int64_t ldq, int64_t Q, float* center, void* g_packed,
                         void* group, void* q_packed, int flags, void* workspace, ieee_stream_t stream_) {
  int rc = check_device();
  if (rc) return rc;
  cudaStream_t stream = (cudaStream_t)stream_;
  IEEE_REQUIRE(gf && g_packed && G > 0 && D > 0, "gallery_prepare: bad arguments (G=%lld D=%lld)", (long long)G, (long long)D);
  const bool new_center = q != nullptr && !(flags & IEEE_PREPARE_KEEP_CENTER);
  IEEE_REQUIRE(!new_center || (center != nullptr && Q > 0), "gallery_prepare: a centre from the query rows needs the centre buffer");
  IEEE_REQUIRE(q_packed == nullptr || (q != nullptr && Q > 0), "gallery_prepare: packing the queries needs the query rows");
  tl_enter(stream, "enter gallery_prepare");
  SideLane* lane = nullptr;
  const bool grouping = g_pids != nullptr && group != nullptr;
  if (grouping) {
    if ((rc = side_lane(&lane))) return rc;
    IEEE_CUDA_CHECK(cudaEventRecord(lane->fork, stream));
  }
  // the bandwidth-bound kernels are issued FIRST: the six API calls of the side lane took ~25 us of host time during
  // which the GPU had nothing to do (profiles/r2_step_marks_n1_before.txt)
  if (new_center && (rc = feature_center(q, dtype, ldq, Q, D, normalize, 0, center, workspace, stream))) return rc;
  if ((rc = pack_features(gf, dtype, ldg, G, D, metric, normalize, precision, center, g_packed, stream))) return rc;
  // the query block too, when asked: the caller's host work between this call and the evaluation call then hides
  // behind it (with a small gallery shard the gallery pack alone is over before the next call arrives)
  if (q_packed != nullptr && (rc = pack_features(q, dtype, ldq, Q, D, metric, normalize, precision, center, q_packed, stream)))
    return rc;
  if (grouping) {
    IEEE_CUDA_CHECK(cudaStreamWaitEvent(lane->stream, lane->fork, 0));
    if ((rc = gallery_group(g_pids, G, group, lane->stream))) return rc;
    IEEE_CUDA_CHECK(cudaEventRecord(lane->join, lane->stream));
    if (!(flags & IEEE_PREPARE_DEFER_JOIN)) {
      IEEE_CUDA_CHECK(cudaStreamWaitEvent(stream, lane->join, 0));
      count_launch(0, "join grouping (side stream)");
    }
  }
  return IEEE_OK;
}

int ieee_gallery_group_join(ieee_stream_t stream) {
  int rc = check_device();
  if (rc) return rc;
  return side_lane_join((cudaStream_t)stream);
}

// float64 distance matrix: ranked in float64 order (rank.py:117 argsorts whatever dtype it is given)
int ieee_eval_market1501_f64(const double* distmat, int64_t ld, int64_t Q, int64_t G, const int64_t* q_pids,
                             const int64_t* g_pids, const int64_t* q_camids, const int64_t* g_camids, int32_t max_rank,
                             int32_t cap, float* cmc, ieee_eval_summary* summary, void* workspace, size_t workspace_bytes,
                             ieee_stream_t stream_) {
  int rc = check_device();
  if (rc) return rc;
  cudaStream_t stream = (cudaStream_t)stream_;
  IEEE_REQUIRE(distmat && q_pids && g_pids && q_camids && g_camids && cmc && summary && workspace, "eval (f64): null pointer");
  IEEE_REQUIRE(Q > 0 && G > 0 && ld >= G && max_rank >= 1, "eval (f64): bad shape Q=%lld G=%lld ld=%lld max_rank=%d", (long long)Q,
               (long long)G, (long long)ld, max_rank);
  IEEE_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "eval (f64): workspace must be 256-byte aligned");
  Arena a{static_cast<uint8_t*>(workspace), workspace_bytes, 0};
  void* group = a.take(gallery_group_bytes(G));
  int32_t* scratch = static_cast<int32_t*>(a.take(256));   // [0] cap, [1] overflow, [2..3] ties (u64)
  if (!group || !scratch) { set_error("eval (f64): workspace too small"); return IEEE_ERR_WORKSPACE; }
  if ((rc = gallery_group(g_pids, G, group, stream))) return rc;
  int32_t need = 0;
  if ((rc = ieee_rank_list_cap_sync(group, G, q_pids, Q, scratch, &need, stream_))) return rc;
  if (need < 1) need = 1;
  if (cap > 0 && need > cap) {
    set_error("eval (f64): a query has %d same-identity gallery items but list capacity is %d", need, cap);
    return IEEE_ERR_CAPACITY;
  }
  cap = need;
  int32_t* counts = static_cast<int32_t*>(a.take(size_t(Q) * (cap + 2) * 4));
  void* fws = a.take(rank_finalize_workspace_bytes(Q));
  if (!counts || !fws) {
    set_error("eval (f64): workspace too small (%zu bytes given, need %zu for cap=%d)", workspace_bytes,
              ieee_eval_workspace_bytes(Q, G, cap), cap);
    return IEEE_ERR_WORKSPACE;
  }
  IEEE_CUDA_CHECK(cudaMemsetAsync(scratch, 0, 256, stream));
  unsigned long long* ties = reinterpret_cast<unsigned long long*>(scratch + 2);
  if ((rc = rank_count_f64(distmat, ld, Q, G, q_pids, q_camids, g_camids, group, cap, counts, ties, scratch + 1, stream))) return rc;
  return rank_finalize(counts, Q, G, 1, cap, max_rank, ties, cmc, summary, nullptr, nullptr, fws, stream, nullptr,
                       reinterpret_cast<uint32_t*>(scratch + 8));
}

// ---- retrieval + evaluation in one call ----------------------------------------------------------------
static size_t retrieve_rank_bytes(int64_t Q, int32_t cap) {
  size_t b = 256;                                  // cap scratch + overflow flag + ties
  b += 2 * align256(size_t(Q) * (cap + 1) * 8);    // rel (+ embedded count), junk
  b += 2 * align256(size_t(Q) * 4);                // n_rel, n_junk
  b += align256(size_t(Q) * (cap + 2) * 4);        // counts
  b += align256(rank_finalize_workspace_bytes(Q));
  return b;
}

size_t ieee_retrieve_prepared_workspace_bytes(int64_t Q, int64_t D, int precision, int32_t cap) {
  if (Q <= 0 || D <= 0) return 0;
  if (cap <= 0) cap = 4096;
  return align256(ieee_packed_bytes(Q, D, precision)) + retrieve_rank_bytes(Q, cap) + distmat_fixup_bytes(Q) + 256;
}

size_t ieee_retrieve_workspace_bytes(int64_t Q, int64_t G, int64_t D, int precision, int32_t cap) {
  if (Q <= 0 || G <= 0 || D <= 0) return 0;
  if (cap <= 0) cap = (int32_t)(G < 4096 ? G : 4096);
  return align256(ieee_packed_bytes(G, D, precision)) + align256(gallery_group_bytes(G)) + center_bytes(D) +
         ieee_retrieve_prepared_workspace_bytes(Q, D, precision, cap);
}

int ieee_retrieve_eval_prepared(const void* qf, int64_t ldq, int dtype, int64_t Q, int64_t D, int metric, int normalize,
                                int precision, const void* g_packed, const void* group, const float* center, int64_t G,
                                const int64_t* q_pids,
                                const int64_t* q_camids, const int64_t* g_camids, int32_t max_rank, int32_t cap,
                                int32_t* cap_host_out, float* distmat, int64_t ld, float* cmc, ieee_eval_summary* summary,
                                double* per_query_ap, int32_t* per_query_first, const void* q_packed_ready,
                                void* workspace, size_t workspace_bytes, ieee_stream_t stream_) {
  int rc = check_device();
  if (rc) return rc;
  cudaStream_t stream = (cudaStream_t)stream_;
  IEEE_REQUIRE((qf || q_packed_ready) && g_packed && group && q_pids && q_camids && g_camids && distmat && cmc && summary && workspace,
               "retrieve: null pointer");
  IEEE_REQUIRE(Q > 0 && G > 0 && D > 0 && ld >= G && max_rank >= 1, "retrieve: bad shape Q=%lld G=%lld D=%lld ld=%lld max_rank=%d",
               (long long)Q, (long long)G, (long long)D, (long long)ld, max_rank);
  IEEE_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "retrieve: workspace must be 256-byte aligned");
  Arena a{static_cast<uint8_t*>(workspace), workspace_bytes, 0};
  int32_t* scratch = static_cast<int32_t*>(a.take(256));   // [0] cap, [1] overflow, [2..3] ties (u64), [8] metrics ticket
  void* fix = a.take(distmat_fixup_bytes(Q));              // (directly behind the scratch words: one clear covers both)
  const void* q_packed = q_packed_ready;
  if (q_packed == nullptr) q_packed = a.take(ieee_packed_bytes(Q, D, precision));
  if (!q_packed || !scratch || !fix) { set_error("retrieve: workspace too small"); return IEEE_ERR_WORKSPACE; }
  tl_enter(stream, "enter retrieve_eval_prepared");
  if (q_packed_ready != nullptr) {
    // queries packed by ieee_gallery_prepare: clear the scratch words and the fix-up list header in one node
    IEEE_CUDA_CHECK(cudaMemsetAsync(scratch, 0, 256 + 8, stream));
    count_launch(0, "memset scratch + fix list");
  } else {
    // the query pack's first CTA clears the scratch words and the fix-up list header for the kernels behind it
    const ZeroJob zero{{reinterpret_cast<uint32_t*>(scratch), static_cast<uint32_t*>(fix)}, {64, 2}};
    if ((rc = pack_features(qf, dtype, ldq, Q, D, metric, normalize, precision, center, const_cast<void*>(q_packed), stream, &zero)))
      return rc;
  }
  if (cap <= 0) {
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    IEEE_CUDA_CHECK(cudaStreamIsCapturing(stream, &cs));
    IEEE_REQUIRE(cs == cudaStreamCaptureStatusNone,
                 "retrieve: cap <= 0 sizes the lists with a host round trip, which a stream capture cannot hold: pass cap > 0");
    int32_t need = 0;
    if ((rc = ieee_rank_list_cap_sync(group, G, q_pids, Q, scratch, &need, stream_))) return rc;
    cap = need < 1 ? 1 : need;
  }
  if (cap_host_out) *cap_host_out = cap;
  uint64_t* rel = static_cast<uint64_t*>(a.take(size_t(Q) * (cap + 1) * 8));
  uint64_t* junk = static_cast<uint64_t*>(a.take(size_t(Q) * cap * 8));
  int32_t* n_rel = static_cast<int32_t*>(a.take(size_t(Q) * 4));
  int32_t* n_junk = static_cast<int32_t*>(a.take(size_t(Q) * 4));
  int32_t* counts = static_cast<int32_t*>(a.take(size_t(Q) * (cap + 2) * 4));
  void* fws = a.take(rank_finalize_workspace_bytes(Q));
  if (!rel || !junk || !n_rel || !n_junk || !counts || !fws) {
    set_error("retrieve: workspace too small (%zu bytes given, need %zu for cap=%d)", workspace_bytes,
              ieee_retrieve_prepared_workspace_bytes(Q, D, precision, cap), cap);
    return IEEE_ERR_WORKSPACE;
  }
  if ((rc = distmat_packed(q_packed, Q, g_packed, G, D, metric, precision, distmat, ld, fix, stream_, true))) return rc;
  unsigned long long* ties = reinterpret_cast<unsigned long long*>(scratch + 2);
  if ((rc = side_lane_join(stream))) return rc;      // a grouping ieee_gallery_prepare left on the side lane
  if ((rc = rank_gather(distmat, ld, Q, G, q_pids, q_camids, g_camids, group, 0, cap, rel, n_rel, junk, n_junk, scratch + 1, stream))) return rc;
  if ((rc = rank_count(distmat, ld, Q, G, 0, 1, cap, 0, rel, n_rel, junk, n_junk, counts, ties, stream))) return rc;
  // scratch: [0] cap, [1] overflow, [2..3] ties, [8] ticket of the metrics kernel (all cleared by the query pack)
  return rank_finalize(counts, Q, G, 1, cap, max_rank, ties, cmc, summary, per_query_ap, per_query_first, fws, stream,
                       scratch + 1, reinterpret_cast<uint32_t*>(scratch + 8));
}

int ieee_retrieve_eval(const void* qf, int64_t ldq, const void* gf, int64_t ldg, int dtype, int64_t Q, int64_t G, int64_t D,
                       int metric, int normalize, int precision, const int64_t* q_pids, const int64_t* g_pids,
                       const int64_t* q_camids, const int64_t* g_camids, int32_t max_rank, int32_t cap,
                       int32_t* cap_host_out, float* distmat, int64_t ld, float* cmc, ieee_eval_summary* summary,
                       double* per_query_ap, int32_t* per_query_first, void* workspace, size_t workspace_bytes,
                       ieee_stream_t stream_) {
  int rc = check_device();
  if (rc) return rc;
  IEEE_REQUIRE(gf && g_pids && workspace, "retrieve: null pointer");
  IEEE_REQUIRE(Q > 0 && G > 0 && D > 0, "retrieve: bad shape Q=%lld G=%lld D=%lld", (long long)Q, (long long)G, (long long)D);
  IEEE_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "retrieve: workspace must be 256-byte aligned");
  Arena a{static_cast<uint8_t*>(workspace), workspace_bytes, 0};
  void* g_packed = a.take(ieee_packed_bytes(G, D, precision));
  void* group = a.take(gallery_group_bytes(G));
  float* center = static_cast<float*>(a.take(size_t(D) * 4));
  void* cws = a.take(feature_center_workspace_bytes(D));
  if (!g_packed || !group || !center || !cws) { set_error("retrieve: workspace too small"); return IEEE_ERR_WORKSPACE; }
  // the grouping (three tiny label-only kernels) runs on the side lane beside the centre and the feature packing
  const bool centred = auto_center(metric, precision);
  IEEE_REQUIRE(qf != nullptr, "retrieve: null pointer");
  if (!centred) center = nullptr;
  // the evaluation call packs the queries itself (its workspace holds them) and joins the side lane before the gather
  if ((rc = ieee_gallery_prepare(gf, ldg, dtype, G, D, metric, normalize, precision, g_pids, centred ? qf : nullptr, ldq, Q,
                                 center, g_packed, group, nullptr, IEEE_PREPARE_DEFER_JOIN, cws, stream_)))
    return rc;
  const size_t used = align256(a.off);
  return ieee_retrieve_eval_prepared(qf, ldq, dtype, Q, D, metric, normalize, precision, g_packed, group, center, G, q_pids, q_camids,
                                     g_camids, max_rank, cap, cap_host_out, distmat, ld, cmc, summary, per_query_ap,
                                     per_query_first, nullptr, static_cast<uint8_t*>(workspace) + used, workspace_bytes - used,
                                     stream_);
}

int ieee_topk(const float* distmat, int64_t ld, int64_t Q, int64_t G, int64_t g_offset, const int64_t* q_pids,
              const int64_t* q_camids, const int64_t* g_pids, const int64_t* g_camids, int32_t k, int32_t* idx, float* val,
              ieee_stream_t stream) {
  int rc = check_device();
  if (rc) return rc;
  return topk(distmat, ld, Q, G, g_offset, q_pids, q_camids, g_pids, g_camids, k, idx, val, (cudaStream_t)stream);
}

int ieee_topk_merge(const int32_t* idx_all, const float* val_all, int32_t shards, int64_t Q, int32_t k, int32_t* idx,
                    float* val, ieee_stream_t stream) {
  int rc = check_device();
  if (rc) return rc;
  return topk_merge(idx_all, val_all, shards, Q, k, idx, val, (cudaStream_t)stream);
}

size_t ieee_rerank_workspace_bytes(int64_t Q, int64_t G, int32_t k1, int32_t k2) { return rerank_workspace_bytes(Q, G, k1, k2); }

int ieee_rerank(const float* q_g, int64_t ld_qg, const float* q_q, int64_t ld_qq, const float* g_g, int64_t ld_gg, int64_t Q,
                int64_t G, int32_t k1, int32_t k2, double lambda_value, float* out, int64_t ldo, void* workspace,
                size_t workspace_bytes, ieee_stream_t stream) {
  int rc = check_device();
  if (rc) return rc;
  return rerank(q_g, ld_qg, q_q, ld_qq, g_g, ld_gg, Q, G, k1, k2, lambda_value, out, ldo, workspace, workspace_bytes,
                (cudaStream_t)stream);
}

size_t ieee_rerank_stream_workspace_bytes(int64_t Q, int64_t G, int32_t k1, int32_t k2) {
  return rerank_stream_workspace_bytes(Q, G, k1, k2);
}

size_t ieee_rerank_stream_scratch_bytes(int64_t Q, int64_t G, int32_t k1, size_t strip_bytes) {
  return rerank_stream_scratch_bytes(Q, G, k1, strip_bytes);
}

int ieee_rerank_stream_prepare(const void* q_packed, int64_t Q, const void* g_packed, int64_t G, int64_t D, int metric,
                               int precision, int32_t k1, int32_t k2, size_t strip_bytes, float* colmax, int32_t* rank,
                               void* workspace, size_t workspace_bytes, void* scratch, size_t scratch_bytes,
                               ieee_stream_t stream) {
  int rc = check_device();
  if (rc) return rc;
  return rerank_stream_prepare(q_packed, Q, g_packed, G, D, metric, precision, k1, k2, strip_bytes, colmax, rank, workspace,
                               workspace_bytes, scratch, scratch_bytes, (cudaStream_t)stream, cta_group_default());
}

int ieee_rerank_stream_block(const void* workspace, int64_t Q, int64_t G, int32_t k1, int32_t k2, const float* colmax,
                             int64_t row0, int64_t rows, double lambda_value, float* block, int64_t ld, void* scratch,
                             size_t scratch_bytes, ieee_stream_t stream) {
  int rc = check_device();
  if (rc) return rc;
  return rerank_stream_block(workspace, Q, G, k1, k2, colmax, row0, rows, lambda_value, block, ld, scratch, scratch_bytes,
                             (cudaStream_t)stream);
}

size_t ieee_rerank_stream_window_workspace_bytes(int64_t Q, int64_t G, int32_t k1, int32_t k2, int64_t Gs) {
  return rerank_stream_window_workspace_bytes(Q, G, k1, k2, Gs);
}

int ieee_rerank_stream_v_layout(int64_t Q, int64_t G, int32_t k1, int32_t k2, int64_t* cap, size_t* off_col, size_t* off_val,
                                size_t* off_cnt) {
  return rerank_stream_v_layout(Q, G, k1, k2, cap, off_col, off_val, off_cnt);
}

int ieee_rerank_stream_pass(int32_t pass, const void* q_packed, int64_t Q, const void* g_packed, int64_t G, int64_t D, int metric,
                            int precision, int32_t k1, int32_t k2, size_t strip_bytes, int64_t q0, int64_t q1, int64_t g0,
                            int64_t g1, float* colmax, int32_t* rank, void* workspace, size_t workspace_bytes, void* scratch,
                            size_t scratch_bytes, ieee_stream_t stream) {
  int rc = check_device();
  if (rc) return rc;
  return rerank_stream_pass(pass, q_packed, Q, g_packed, G, D, metric, precision, k1, k2, strip_bytes, q0, q1, g0, g1, colmax,
                            rank, workspace, workspace_bytes, scratch, scratch_bytes, (cudaStream_t)stream, cta_group_default());
}

int ieee_rerank_stream_finish(void* workspace, size_t workspace_bytes, int64_t Q, int64_t G, int32_t k1, int32_t k2, int64_t g0,
                              int64_t Gs, const int32_t* rank, ieee_stream_t stream) {
  int rc = check_device();
  if (rc) return rc;
  return rerank_stream_finish(workspace, workspace_bytes, Q, G, k1, k2, g0, Gs, rank, (cudaStream_t)stream);
}

int ieee_rerank_stream_block_window(const void* workspace, int64_t Q, int64_t G, int32_t k1, int32_t k2, int64_t Gs,
                                    const float* colmax, int64_t row0, int64_t rows, double lambda_value, float* block,
                                    int64_t ld, void* scratch, size_t scratch_bytes, ieee_stream_t stream) {
  int rc = check_device();
  if (rc) return rc;
  return rerank_stream_block_window(workspace, Q, G, k1, k2, Gs, colmax, row0, rows, lambda_value, block, ld, scratch,
                                    scratch_bytes, (cudaStream_t)stream);
}

int64_t ieee_rerank_stream_part_width(int64_t Q, int64_t G, int32_t k1, int64_t qa, int64_t qb, int64_t ga, int64_t gb,
                                      size_t strip_bytes) {
  return rerank_stream_part_width(Q, G, k1, qa, qb, ga, gb, strip_bytes);
}

size_t ieee_rerank_stream_part_scratch_bytes(int64_t Q, int64_t G, int32_t k1, int64_t qa, int64_t qb, int64_t ga, int64_t gb,
                                             int64_t width) {
  return rerank_stream_part_scratch_bytes(Q, G, k1, qa, qb, ga, gb, width);
}

int ieee_rerank_stream_part_contract(int32_t pass, const void* q_packed, int64_t Q, const void* g_part, const void* g_strip,
                                     int64_t G, int64_t D, int metric, int precision, int32_t k1, int64_t qa, int64_t qb,
                                     int64_t ga, int64_t gb, int64_t width, int64_t i0, int64_t wc, float* colmax, void* scratch,
                                     size_t scratch_bytes, ieee_stream_t stream) {
  int rc = check_device();
  if (rc) return rc;
  return rerank_stream_part_contract(pass, q_packed, Q, g_part, g_strip, G, D, metric, precision, k1, qa, qb, ga, gb, width, i0,
                                     wc, colmax, scratch, scratch_bytes, (cudaStream_t)stream, cta_group_default());
}

int ieee_rerank_stream_part_topk(int64_t Q, int64_t G, int32_t k1, int64_t qa, int64_t qb, int64_t ga, int64_t gb, int64_t width,
                                 int64_t i0, int64_t wc, const float* colmax, int32_t* idx, float* val, void* scratch,
                                 size_t scratch_bytes, ieee_stream_t stream) {
  int rc = check_device();
  if (rc) return rc;
  return rerank_stream_part_topk(Q, G, k1, qa, qb, ga, gb, width, i0, wc, colmax, idx, val, scratch, scratch_bytes,
                                 (cudaStream_t)stream);
}

int ieee_rerank_stream_part_members(int64_t Q, int64_t G, int32_t k1, int32_t k2, int64_t qa, int64_t qb, int64_t ga, int64_t gb,
                                    int64_t width, int64_t i0, int64_t wc, const float* colmax, void* workspace,
                                    size_t workspace_bytes, const void* scratch, size_t scratch_bytes, ieee_stream_t stream) {
  int rc = check_device();
  if (rc) return rc;
  return rerank_stream_part_members(Q, G, k1, k2, qa, qb, ga, gb, width, i0, wc, colmax, workspace, workspace_bytes, scratch,
                                    scratch_bytes, (cudaStream_t)stream);
}

int ieee_rerank_stream_part_weights(void* workspace, size_t workspace_bytes, int64_t Q, int64_t G, int32_t k1, int32_t k2,
                                    int64_t row0, int64_t rows, ieee_stream_t stream) {
  int rc = check_device();
  if (rc) return rc;
  return rerank_stream_part_weights(workspace, workspace_bytes, Q, G, k1, k2, row0, rows, (cudaStream_t)stream);
}

size_t ieee_gnn_rerank_workspace_bytes(int64_t N, int32_t k1) { return gnn_rerank_workspace_bytes(N, k1); }

int ieee_gnn_rerank(const float* neg_score, int64_t lds, int64_t N, int32_t k1, int32_t k2, float* A, int64_t ldA,
                    void* workspace, size_t workspace_bytes, ieee_stream_t stream) {
  int rc = check_device();
  if (rc) return rc;
  return gnn_rerank(neg_score, lds, N, k1, k2, A, ldA, workspace, workspace_bytes, (cudaStream_t)stream);
}

size_t ieee_gnn_stream_scratch_bytes(int64_t Q, int64_t G, int32_t k1, size_t strip_bytes) {
  return gnn_stream_scratch_bytes(Q, G, k1, strip_bytes);
}

int ieee_gnn_stream_neighbours(const void* q_packed, int64_t Q, const void* g_packed, int64_t G, int64_t D, int precision,
                               int32_t k1, size_t strip_bytes, int32_t* rank, float* S, void* scratch, size_t scratch_bytes,
                               ieee_stream_t stream) {
  int rc = check_device();
  if (rc) return rc;
  return gnn_stream_neighbours(q_packed, Q, g_packed, G, D, precision, k1, strip_bytes, rank, S, scratch, scratch_bytes,
                               (cudaStream_t)stream, cta_group_default());
}

int ieee_gnn_stream_graph_bytes_sync(const int32_t* rank, int64_t Q, int64_t G, int32_t k1, int32_t k2, void* scratch,
                                     size_t scratch_bytes, int64_t* sizes, ieee_stream_t stream) {
  int rc = check_device();
  if (rc) return rc;
  return gnn_stream_graph_bytes_sync(rank, Q, G, k1, k2, scratch, scratch_bytes, sizes, (cudaStream_t)stream);
}

int ieee_gnn_stream_graph(const int32_t* rank, const float* S, int64_t Q, int64_t G, int32_t k1, int32_t k2, void* scratch,
                          size_t scratch_bytes, void* work, size_t work_bytes, const int64_t* sizes, int64_t* a_ptr,
                          int32_t* a_col, float* a_val, int64_t* g_ptr, int32_t* g_row, float* g_val, ieee_stream_t stream) {
  int rc = check_device();
  if (rc) return rc;
  return gnn_stream_graph(rank, S, Q, G, k1, k2, scratch, scratch_bytes, work, work_bytes, sizes, a_ptr, a_col, a_val, g_ptr,
                          g_row, g_val, (cudaStream_t)stream);
}

int ieee_gnn_stream_block(const int64_t* a_ptr, const int32_t* a_col, const float* a_val, const int64_t* g_ptr,
                          const int32_t* g_row, const float* g_val, int64_t Q, int64_t G, int64_t row0, int64_t rows,
                          float* block, int64_t ld, void* scratch, size_t scratch_bytes, ieee_stream_t stream) {
  int rc = check_device();
  if (rc) return rc;
  return gnn_stream_block(a_ptr, a_col, a_val, g_ptr, g_row, g_val, Q, G, row0, rows, block, ld, scratch, scratch_bytes,
                          (cudaStream_t)stream);
}

int ieee_gnn_stream_neighbours_rows(const void* q_packed, int64_t Q, const void* g_packed, int64_t G, int64_t D, int precision,
                                    int32_t k1, size_t strip_bytes, int64_t q0, int64_t q1, int64_t g0, int64_t g1, int32_t* rank,
                                    float* S, void* scratch, size_t scratch_bytes, ieee_stream_t stream) {
  int rc = check_device();
  if (rc) return rc;
  return gnn_stream_neighbours_rows(q_packed, Q, g_packed, G, D, precision, k1, strip_bytes, q0, q1, g0, g1, rank, S, scratch,
                                    scratch_bytes, (cudaStream_t)stream, cta_group_default());
}

int ieee_gnn_stream_layout(int64_t Q, int64_t G, int32_t k1, int32_t k2, const int64_t* sizes, size_t* off) {
  return gnn_stream_layout(Q, G, k1, k2, sizes, off);
}

int ieee_gnn_stream_symbolic(const int32_t* rank, int64_t Q, int64_t G, int32_t k1, int32_t k2, int64_t q0, int64_t q1, int64_t g0,
                             int64_t g1, void* scratch, size_t scratch_bytes, ieee_stream_t stream) {
  int rc = check_device();
  if (rc) return rc;
  return gnn_stream_symbolic(rank, Q, G, k1, k2, q0, q1, g0, g1, scratch, scratch_bytes, (cudaStream_t)stream);
}

int ieee_gnn_stream_sizes_sync(int64_t Q, int64_t G, int32_t k1, int32_t k2, void* scratch, size_t scratch_bytes, int64_t* sizes,
                               ieee_stream_t stream) {
  int rc = check_device();
  if (rc) return rc;
  return gnn_stream_sizes_sync(Q, G, k1, k2, scratch, scratch_bytes, sizes, (cudaStream_t)stream);
}

int ieee_gnn_stream_numeric(int32_t step, const int32_t* rank, const float* S, int64_t Q, int64_t G, int32_t k1, int32_t k2,
                            int64_t q0, int64_t q1, int64_t g0, int64_t g1, void* scratch, size_t scratch_bytes, void* work,
                            size_t work_bytes, const int64_t* sizes, int64_t* a_ptr, int32_t* a_col, float* a_val,
                            ieee_stream_t stream) {
  int rc = check_device();
  if (rc) return rc;
  return gnn_stream_numeric(step, rank, S, Q, G, k1, k2, q0, q1, g0, g1, scratch, scratch_bytes, work, work_bytes, sizes, a_ptr,
                            a_col, a_val, (cudaStream_t)stream);
}

int ieee_gnn_stream_csc(int64_t Q, int64_t G, int32_t k1, int64_t q0, int64_t q1, int64_t g0, int64_t g1, void* scratch,
                        size_t scratch_bytes, const int64_t* a_ptr, const int32_t* a_col, const float* a_val, int64_t* g_ptr,
                        int32_t* g_row, float* g_val, ieee_stream_t stream) {
  int rc = check_device();
  if (rc) return rc;
  return gnn_stream_csc(Q, G, k1, q0, q1, g0, g1, scratch, scratch_bytes, a_ptr, a_col, a_val, g_ptr, g_row, g_val,
                        (cudaStream_t)stream);
}

// ---- peer exchange (gallery sharded over the GPUs of one box) ---------------------------------------------------
// regions are sized for the largest query block (Qb_max); a block of Qb <= Qb_max rows uses a dense prefix of each
static size_t peer_layout(int64_t Qb_max, int64_t Qb, int64_t Qtot, int32_t cap, int32_t W, int32_t shards, PeerView* v) {
  size_t o = kPeerHeaderBytes;
  auto take = [&](size_t bytes) { size_t r = o; o += align256(bytes); return r; };
  const size_t off_rel = take(size_t(shards) * Qb_max * (cap + 1) * 8);
  const size_t off_cnt = take(size_t(shards) * Qb_max * (W + 2) * 4);
  const size_t off_ap = take(size_t(Qtot) * 8), off_inp = take(size_t(Qtot) * 8);
  const size_t off_first = take(size_t(Qtot) * 4), off_short = take(size_t(Qtot) * 4);
  if (v) {
    v->off_rel = off_rel; v->off_cnt = off_cnt; v->off_ap = off_ap; v->off_inp = off_inp;
    v->off_first = off_first; v->off_short = off_short;
    v->Qb = Qb; v->cap = cap; v->W = W;
  }
  return o;
}

size_t ieee_peer_exchange_bytes(int64_t Qb_max, int64_t Qtot, int32_t cap, int32_t W, int32_t shards) {
  if (Qb_max <= 0 || Qtot < Qb_max || cap < 1 || W < 1 || shards < 1 || shards > kMaxPeers) return 0;
  return peer_layout(Qb_max, Qb_max, Qtot, cap, W, shards, nullptr);
}

int ieee_peer_alloc(size_t bytes, void** ptr, void* ipc_handle_out) {
  int rc = check_device();
  if (rc) return rc;
  IEEE_REQUIRE(ptr && ipc_handle_out && bytes >= kPeerHeaderBytes, "peer_alloc: bad arguments");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "ipc handle size");
  IEEE_CUDA_CHECK(cudaMalloc(ptr, bytes));
  IEEE_CUDA_CHECK(cudaMemset(*ptr, 0, bytes));
  IEEE_CUDA_CHECK(cudaDeviceSynchronize());
  IEEE_CUDA_CHECK(cudaIpcGetMemHandle(static_cast<cudaIpcMemHandle_t*>(ipc_handle_out), *ptr));
  return IEEE_OK;
}

int ieee_peer_open(const void* ipc_handle, void** ptr) {
  int rc = check_device();
  if (rc) return rc;
  IEEE_REQUIRE(ipc_handle && ptr, "peer_open: null pointer");
  cudaIpcMemHandle_t h;
  memcpy(&h, ipc_handle, sizeof(h));
  IEEE_CUDA_CHECK(cudaIpcOpenMemHandle(ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return IEEE_OK;
}

int ieee_peer_close(void* ptr) {
  if (ptr) IEEE_CUDA_CHECK(cudaIpcCloseMemHandle(ptr));
  return IEEE_OK;
}

int ieee_peer_free(void* ptr) {
  if (ptr) IEEE_CUDA_CHECK(cudaFree(ptr));
  return IEEE_OK;
}

static int peer_view(const ieee_peer_exchange* ex, PeerView* v, unsigned long long* epoch_dev = nullptr) {
  IEEE_REQUIRE(ex != nullptr, "peer exchange: null descriptor");
  IEEE_REQUIRE(ex->shards >= 1 && ex->shards <= kMaxPeers && ex->my_shard >= 0 && ex->my_shard < ex->shards,
               "peer exchange: bad shard %d of %d", ex->my_shard, ex->shards);
  IEEE_REQUIRE(ex->Qb > 0 && ex->Qb <= ex->Qb_max && ex->q_base >= 0 && ex->q_base + ex->Qb <= ex->Qtot && ex->cap >= 1 &&
                   ex->W >= 1 && (ex->epoch > 0 || epoch_dev != nullptr),
               "peer exchange: bad block (Qb=%lld q_base=%lld Qtot=%lld cap=%d W=%d)", (long long)ex->Qb,
               (long long)ex->q_base, (long long)ex->Qtot, ex->cap, ex->W);
  *v = no_peers();
  v->shards = ex->shards;
  v->my = ex->my_shard;
  v->epoch = ex->epoch;
  v->epoch_dev = epoch_dev;
  for (int s = 0; s < ex->shards; ++s) {
    IEEE_REQUIRE(ex->base[s] != nullptr, "peer exchange: buffer of shard %d is not mapped", s);
    v->base[s] = static_cast<uint8_t*>(ex->base[s]);
  }
  peer_layout(ex->Qb_max, ex->Qb, ex->Qtot, ex->cap, ex->W, ex->shards, v);
  v->q_base = ex->q_base;
  return IEEE_OK;
}

int ieee_rank_gather_peer(const float* distmat, int64_t ld, int64_t G, const int64_t* q_pids, const int64_t* q_camids,
                          const int64_t* g_camids, const void* group, int64_t g_offset, int32_t* n_rel, uint64_t* junk,
                          int32_t* n_junk, unsigned long long* stats, const ieee_peer_exchange* ex, ieee_stream_t stream) {
  int rc = check_device();
  if (rc) return rc;
  PeerView v;
  if ((rc = peer_view(ex, &v))) return rc;
  IEEE_REQUIRE(stats != nullptr, "rank_gather_peer: null pointer");
  return rank_gather(distmat, ld, v.Qb, G, q_pids, q_camids, g_camids, group, g_offset, v.cap, nullptr, n_rel, junk, n_junk,
                     reinterpret_cast<int32_t*>(stats), (cudaStream_t)stream, &v);
}

int ieee_rank_count_peer(const float* distmat, int64_t ld, int64_t G, int64_t g_offset, const int32_t* n_rel,
                         const uint64_t* junk, const int32_t* n_junk, unsigned long long* stats,
                         const ieee_peer_exchange* ex, ieee_stream_t stream) {
  int rc = check_device();
  if (rc) return rc;
  PeerView v;
  if ((rc = peer_view(ex, &v))) return rc;
  IEEE_REQUIRE(stats != nullptr, "rank_count_peer: null pointer");
  const uint64_t* rel_all = reinterpret_cast<const uint64_t*>(v.base[v.my] + v.off_rel);
  return rank_count(distmat, ld, v.Qb, G, g_offset, v.shards, v.cap, v.W, rel_all, n_rel, junk, n_junk, nullptr, stats + 1,
                    (cudaStream_t)stream, &v);
}

int ieee_rank_metrics_peer(int64_t G_total, int32_t max_rank, const unsigned long long* stats, float* cmc,
                           ieee_eval_summary* summary, int64_t* stats_out, const ieee_peer_exchange* ex, ieee_stream_t stream) {
  int rc = check_device();
  if (rc) return rc;
  PeerView v;
  if ((rc = peer_view(ex, &v))) return rc;
  return rank_metrics_peer(&v, G_total, max_rank, stats, cmc, summary, reinterpret_cast<long long*>(stats_out), ex->Qtot,
                           (cudaStream_t)stream);
}

size_t ieee_retrieve_prepared_peer_workspace_bytes(int64_t Q, int64_t D, int precision, int32_t cap) {
  if (Q <= 0 || D <= 0 || cap < 1) return 0;
  return align256(ieee_packed_bytes(Q, D, precision)) + distmat_fixup_bytes(Q) + align256(size_t(Q) * cap * 8) +
         2 * align256(size_t(Q) * 4) + 256 + 256;
}

static int retrieve_eval_prepared_peer(const void* qf, int64_t ldq, int dtype, int64_t Q, int64_t D, int metric, int normalize,
                                     int precision, const void* g_packed, const void* group, const float* center, int64_t G,
                                     int64_t G_total, int64_t g_offset, const int64_t* q_pids, const int64_t* q_camids,
                                     const int64_t* g_camids, int32_t max_rank, float* distmat, int64_t ld, float* cmc,
                                     ieee_eval_summary* summary, int64_t* stats_out, double* per_query_ap,
                                     int32_t* per_query_first, const ieee_peer_exchange* ex, unsigned long long* epoch_dev,
                                     const void* q_packed_ready, void* workspace, size_t workspace_bytes, ieee_stream_t stream_) {
  int rc = check_device();
  if (rc) return rc;
  cudaStream_t stream = (cudaStream_t)stream_;
  IEEE_REQUIRE((qf || q_packed_ready) && g_packed && group && q_pids && q_camids && g_camids && distmat && cmc && summary && workspace && ex,
               "retrieve (peer): null pointer");
  IEEE_REQUIRE(Q > 0 && G > 0 && D > 0 && ld >= G && max_rank >= 1 && G_total >= G && g_offset >= 0,
               "retrieve (peer): bad shape Q=%lld G=%lld D=%lld ld=%lld", (long long)Q, (long long)G, (long long)D, (long long)ld);
  IEEE_REQUIRE(ex->Qb == Q && ex->Qtot == Q && ex->q_base == 0, "retrieve (peer): the exchange must describe one block of Q rows");
  IEEE_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "retrieve (peer): workspace must be 256-byte aligned");
  const int32_t cap = ex->cap;
  Arena a{static_cast<uint8_t*>(workspace), workspace_bytes, 0};
  unsigned long long* stats = static_cast<unsigned long long*>(a.take(256));   // this rank's own statistics
  void* fix = a.take(distmat_fixup_bytes(Q));                                   // (directly behind them: one clear covers both)
  const void* q_packed = q_packed_ready;
  if (q_packed == nullptr) q_packed = a.take(ieee_packed_bytes(Q, D, precision));
  uint64_t* junk = static_cast<uint64_t*>(a.take(size_t(Q) * cap * 8));
  int32_t* n_rel = static_cast<int32_t*>(a.take(size_t(Q) * 4));
  int32_t* n_junk = static_cast<int32_t*>(a.take(size_t(Q) * 4));
  if (!q_packed || !fix || !junk || !n_rel || !n_junk || !stats) {
    set_error("retrieve (peer): workspace too small (%zu bytes given, need %zu for cap=%d)", workspace_bytes,
              ieee_retrieve_prepared_peer_workspace_bytes(Q, D, precision, cap), cap);
    return IEEE_ERR_WORKSPACE;
  }
  tl_enter(stream, "enter retrieve_eval_prepared_peer");
  if (q_packed_ready != nullptr) {
    IEEE_CUDA_CHECK(cudaMemsetAsync(stats, 0, 256 + 8, stream));
    count_launch(0, "memset stats + fix list");
  } else {
    const ZeroJob zero{{reinterpret_cast<uint32_t*>(stats), static_cast<uint32_t*>(fix)}, {64, 2}};
    if ((rc = pack_features(qf, dtype, ldq, Q, D, metric, normalize, precision, center, const_cast<void*>(q_packed), stream, &zero)))
      return rc;
  }
  if ((rc = distmat_packed(q_packed, Q, g_packed, G, D, metric, precision, distmat, ld, fix, stream_, true))) return rc;
  if ((rc = side_lane_join(stream))) return rc;      // a grouping ieee_gallery_prepare left on the side lane
  PeerView v;
  if ((rc = peer_view(ex, &v, epoch_dev))) return rc;
  if ((rc = rank_gather(distmat, ld, v.Qb, G, q_pids, q_camids, g_camids, group, g_offset, v.cap, nullptr, n_rel, junk, n_junk,
                        reinterpret_cast<int32_t*>(stats), stream, &v)))
    return rc;
  const uint64_t* rel_all = reinterpret_cast<const uint64_t*>(v.base[v.my] + v.off_rel);
  if ((rc = rank_count(distmat, ld, v.Qb, G, g_offset, v.shards, v.cap, v.W, rel_all, n_rel, junk, n_junk, nullptr, stats + 1,
                       stream, &v)))
    return rc;
  return rank_metrics_peer(&v, G_total, max_rank, stats, cmc, summary, reinterpret_cast<long long*>(stats_out), ex->Qtot, stream,
                           per_query_ap, per_query_first);
}

int ieee_retrieve_eval_prepared_peer(const void* qf, int64_t ldq, int dtype, int64_t Q, int64_t D, int metric, int normalize,
                                     int precision, const void* g_packed, const void* group, const float* center, int64_t G,
                                     int64_t G_total, int64_t g_offset, const int64_t* q_pids, const int64_t* q_camids,
                                     const int64_t* g_camids, int32_t max_rank, float* distmat, int64_t ld, float* cmc,
                                     ieee_eval_summary* summary, int64_t* stats_out, double* per_query_ap,
                                     int32_t* per_query_first, const ieee_peer_exchange* ex, const void* q_packed_ready,
                                     void* workspace, size_t workspace_bytes, ieee_stream_t stream_) {
  return retrieve_eval_prepared_peer(qf, ldq, dtype, Q, D, metric, normalize, precision, g_packed, group, center, G, G_total,
                                     g_offset, q_pids, q_camids, g_camids, max_rank, distmat, ld, cmc, summary, stats_out,
                                     per_query_ap, per_query_first, ex, nullptr, q_packed_ready, workspace, workspace_bytes,
                                     stream_);
}

int ieee_retrieve_eval_prepared_peer_dev_epoch(const void* qf, int64_t ldq, int dtype, int64_t Q, int64_t D, int metric,
                                               int normalize, int precision, const void* g_packed, const void* group,
                                               const float* center, int64_t G, int64_t G_total, int64_t g_offset,
                                               const int64_t* q_pids, const int64_t* q_camids, const int64_t* g_camids,
                                               int32_t max_rank, float* distmat, int64_t ld, float* cmc, ieee_eval_summary* summary,
                                               int64_t* stats_out, double* per_query_ap, int32_t* per_query_first,
                                               const ieee_peer_exchange* ex, uint64_t* epoch, const void* q_packed_ready,
                                               void* workspace, size_t workspace_bytes, ieee_stream_t stream_) {
  IEEE_REQUIRE(epoch != nullptr, "retrieve (peer, device epoch): null epoch word");
  IEEE_REQUIRE((reinterpret_cast<uintptr_t>(epoch) & 7) == 0, "retrieve (peer, device epoch): the epoch word must be 8-byte aligned");
  return retrieve_eval_prepared_peer(qf, ldq, dtype, Q, D, metric, normalize, precision, g_packed, group, center, G, G_total,
                                     g_offset, q_pids, q_camids, g_camids, max_rank, distmat, ld, cmc, summary, stats_out,
                                     per_query_ap, per_query_first, ex, reinterpret_cast<unsigned long long*>(epoch),
                                     q_packed_ready, workspace, workspace_bytes, stream_);
}

size_t ieee_peer_result_offset(int which, int64_t Qb_max, int64_t Qtot, int32_t cap, int32_t W, int32_t shards) {
  PeerView v = no_peers();
  if (ieee_peer_exchange_bytes(Qb_max, Qtot, cap, W, shards) == 0) return 0;
  peer_layout(Qb_max, Qb_max, Qtot, cap, W, shards, &v);
  return which == 0 ? v.off_ap : (which == 1 ? v.off_first : (which == 2 ? v.off_inp : v.off_short));
}

}  // extern "C"
