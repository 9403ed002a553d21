// C-ABI entry points of libraglite_b200 (see include/raglite_b200.h).
#include <cmath>
#include <cstdarg>
#include <map>
#include <mutex>

#include "scan_common.cuh"
#include "scan_tcgen05.cuh"
#include "select_finalize.cuh"

namespace rl {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

static size_t align_up(size_t x, size_t a = 256) { return (x + a - 1) / a * a; }

// Stage timing events, keyed by workspace pointer (only touched when RL_FLAG_TIME_KERNELS is set): a ring
// of event sets, one per timed call, so that a caller can time N back-to-back calls without
// synchronising in between and read the per-stage average afterwards.
constexpr int kNumStageEvents = 6;
constexpr int kEventRing = 32;
struct StageEvents {
  cudaEvent_t ev[kEventRing][kNumStageEvents];
  int next = 0;    // set used by the next timed call
  int count = 0;   // sets recorded since the last read
  bool valid = false;
};
static std::mutex g_ev_mutex;
static std::map<const void*, StageEvents> g_events;

static cudaEvent_t* stage_events_for(const void* ws) {
  std::lock_guard<std::mutex> lock(g_ev_mutex);
  StageEvents& se = g_events[ws];
  if (!se.valid) {
    for (int r = 0; r < kEventRing; ++r)
      for (int i = 0; i < kNumStageEvents; ++i)
        if (cudaEventCreate(&se.ev[r][i]) != cudaSuccess) return nullptr;
    se.valid = true;
  }
  cudaEvent_t* set = se.ev[se.next];
  se.next = (se.next + 1) % kEventRing;
  if (se.count < kEventRing) ++se.count;
  return set;
}

static int floor_pow2(double x) {
  int p = 1;
  while ((double)(p * 2) <= x) p *= 2;
  return p;
}

int make_layout(const rl_scan_params* p, int sm_count, Layout* L) {
  (void)sm_count;
  RL_REQUIRE(p != nullptr, RL_EINVAL, "null params");
  RL_REQUIRE(p->n_rows >= 0 && p->n_rows < (1ll << 31) - kBlockRows, RL_EINVAL, "n_rows out of range");
  RL_REQUIRE(p->d > 0 && p->d <= 16384 && p->ld >= p->d, RL_EINVAL, "bad d / ld");
  RL_REQUIRE(p->B >= 0 && p->B <= 65535, RL_EINVAL, "bad B");
  RL_REQUIRE(p->k > 0, RL_EINVAL, "k must be positive");
  RL_REQUIRE(p->num_hits >= 0, RL_EINVAL, "num_hits must be >= 0");
  RL_REQUIRE(p->metric >= RL_METRIC_COSINE && p->metric <= RL_METRIC_L2, RL_EINVAL, "unknown metric %d", p->metric);
  RL_REQUIRE(p->max_vecs_per_chunk >= 1, RL_EINVAL, "max_vecs_per_chunk must be >= 1");
  RL_REQUIRE(p->e_dtype == 0 || p->e_dtype == 1, RL_EINVAL, "e_dtype must be 0 (float32) or 1 (float16)");
  memset(L, 0, sizeof(*L));
  L->mode_sql = p->num_hits > 0;
  L->H = L->mode_sql ? p->num_hits : p->k;
  const int64_t sel_final = L->mode_sql ? p->num_hits : (int64_t)(p->k - 1) * p->max_vecs_per_chunk + 1;
  RL_REQUIRE(sel_final <= RL_MAX_SURVIVORS, RL_EUNSUPPORTED,
             "selection size %lld exceeds the %d-survivor finalize window (k=%d num_hits=%d max_vecs=%d)",
             (long long)sel_final, RL_MAX_SURVIVORS, p->k, p->num_hits, p->max_vecs_per_chunk);
  L->sel_k = L->mode_sql ? p->num_hits : p->k;  // order statistic searched in the sample
  L->n_blocks = (p->n_rows + kBlockRows - 1) / kBlockRows;

  int algo = p->algo;
  const bool tc_ok = tcgen05_supported(p);
  if (algo == RL_ALGO_AUTO) algo = tc_ok ? RL_ALGO_TCGEN05 : RL_ALGO_FP32;
  RL_REQUIRE(algo == RL_ALGO_FP32 || algo == RL_ALGO_TCGEN05, RL_EINVAL, "unknown algo %d", p->algo);
  RL_REQUIRE(p->e_dtype == 0 || algo == RL_ALGO_TCGEN05, RL_EUNSUPPORTED,
             "float16 storage needs the tcgen05 scan (d %% 8 == 0, ld %% 8 == 0, 16-byte aligned E)");
  RL_REQUIRE(algo != RL_ALGO_TCGEN05 || tc_ok, RL_EUNSUPPORTED,
             "RL_ALGO_TCGEN05 needs d %% 4 == 0, ld %% 4 == 0, 16-byte aligned E and a supported metric");
  L->algo = algo;

  int S = p->sample_stride;
  if (S <= 0) {
    // Balance the cost of dumping a 1/S sample (B floats per sampled row) against the candidates
    // the main pass then emits (~ sel_k * S per query, 8 bytes each plus select passes).
    const double rows_per_sel = L->mode_sql ? 1.0 : (double)p->max_vecs_per_chunk;
    const double f = std::sqrt((double)L->sel_k * rows_per_sel * 16.0 / ((double)(p->n_rows > 0 ? p->n_rows : 1) * 4.0));
    // The emit pass tightens its thresholds online (histogram refinement), so the sample only has
    // to seed them: 4x sparser than the static optimum.
    S = floor_pow2(f > 0 ? 4.0 / f : 1.0);
    if (S > 256) S = 256;
    while (S > 1 && (L->n_blocks / S) * kBlockRows < 8 * (int64_t)(L->sel_k * rows_per_sel)) S /= 2;
    if (L->n_blocks < 64) S = 1;
  }
  if (S < 1) S = 1;
  L->S = S;
  L->n_sample_blocks = (L->n_blocks + S - 1) / S;
  L->n_main_blocks = L->n_blocks - L->n_sample_blocks;
  L->n_sample_rows = L->n_sample_blocks * kBlockRows;

  int64_t cap = p->cand_cap;
  if (cap <= 0) {
    // ~3-4x sel_final candidates survive the refined thresholds, plus the burst before the first
    // refresh; the static bound (4 * sel_final * S) only applies to the fp32 scan, which does not refine.
    cap = algo == RL_ALGO_TCGEN05 ? 64 * sel_final + 16384 : 4 * sel_final * S + 1024;
    if (cap > p->n_rows + 1024) cap = p->n_rows + 1024;
  }
  if (cap < 256) cap = 256;
  RL_REQUIRE(cap < (1ll << 30), RL_EINVAL, "cand_cap too large");
  L->cap = (int)cap;

  L->d_pad = (p->d + 63) / 64 * 64;
  L->b_pad = (p->B + 15) / 16 * 16;
  const size_t B = (size_t)(p->B > 0 ? p->B : 1);
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes); return o; };
  L->off_hdr = take(sizeof(Header));
  L->off_cnt = take(B * 4);
  L->off_thr = take(B * 4);
  L->off_thr_out = take(B * 4);
  L->off_eps = take(B * 4);
  L->off_qinv = take(B * 4);
  L->off_qsq = take(B * 8);
  L->off_qscale = take(B * 4);
  L->off_nsurv = take(B * 4);
  L->off_hist = take(B * kHistBins * 4);
  L->off_histw = take(B * 4);
  L->off_cntall = take(B * 4);
  L->off_qimg = take(algo == RL_ALGO_TCGEN05 ? tcgen05_qimg_bytes(p->B, p->d) : 0);
  L->off_dump = take(B * (size_t)L->n_sample_rows * 4);
  L->off_cand = take(B * (size_t)L->cap * sizeof(Cand));
  L->total = off;
  return RL_OK;
}

static int device_sm_count(int* out) {
  int dev = 0;
  RL_CUDA_CHECK(cudaGetDevice(&dev));
  RL_CUDA_CHECK(cudaDeviceGetAttribute(out, cudaDevAttrMultiProcessorCount, dev));
  return RL_OK;
}

}  // namespace rl

using namespace rl;

extern "C" int rl_version(void) { return 101; }
extern "C" const char* rl_last_error(void) { return g_err; }

extern "C" int rl_device_info(int* sm_count, int* cc_major, int* cc_minor, size_t* l2_bytes) {
  int dev = 0;
  RL_CUDA_CHECK(cudaGetDevice(&dev));
  cudaDeviceProp prop;
  RL_CUDA_CHECK(cudaGetDeviceProperties(&prop, dev));
  if (sm_count) *sm_count = prop.multiProcessorCount;
  if (cc_major) *cc_major = prop.major;
  if (cc_minor) *cc_minor = prop.minor;
  if (l2_bytes) *l2_bytes = (size_t)prop.l2CacheSize;
  return RL_OK;
}

extern "C" size_t rl_maxsim_workspace_bytes(const rl_scan_params* p) {
  Layout L;
  if (make_layout(p, 148, &L) != RL_OK) return 0;
  return L.total;
}

extern "C" int rl_maxsim_topk(const rl_scan_params* p, float* hit_sim, int64_t* hit_chunk, int32_t* hit_count,
                              int32_t* status, void* workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  int sms = 148;
  int rc = device_sm_count(&sms);
  if (rc != RL_OK) return rc;
  Layout L;
  rc = make_layout(p, sms, &L);
  if (rc != RL_OK) return rc;
  if (p->B == 0) return RL_OK;
  RL_REQUIRE(hit_sim && hit_chunk && hit_count && status && p->Q, RL_EINVAL, "rl_maxsim_topk: null pointer");
  if (p->n_rows == 0) {  // empty shard: no hits (reference: empty database -> ([], []), tests/test_search.py:76-85)
    RL_CUDA_CHECK(cudaMemsetAsync(hit_count, 0, (size_t)p->B * 4, stream));
    RL_CUDA_CHECK(cudaMemsetAsync(status, 0, (size_t)p->B * 4, stream));
    RL_CUDA_CHECK(cudaMemsetAsync(hit_chunk, 0xFF, (size_t)p->B * L.H * 8, stream));
    RL_CUDA_CHECK(cudaMemsetAsync(hit_sim, 0xFF, (size_t)p->B * L.H * 4, stream));
    return RL_OK;
  }
  RL_REQUIRE(p->E && p->inv_norm && p->sq_norm && p->row_chunk, RL_EINVAL, "rl_maxsim_topk: null index pointer");
  RL_REQUIRE(workspace != nullptr && workspace_bytes >= L.total, RL_ENOSPACE,
             "rl_maxsim_topk: workspace %zu < required %zu", workspace_bytes, L.total);
  RL_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, RL_EINVAL, "workspace must be 256-byte aligned");
  unsigned char* ws = static_cast<unsigned char*>(workspace);
  Header* hdr = reinterpret_cast<Header*>(ws + L.off_hdr);
  int32_t* cand_cnt = reinterpret_cast<int32_t*>(ws + L.off_cnt);
  float* thr = reinterpret_cast<float*>(ws + L.off_thr);
  float* thr_out = reinterpret_cast<float*>(ws + L.off_thr_out);
  float* eps = reinterpret_cast<float*>(ws + L.off_eps);
  float* q_inv = reinterpret_cast<float*>(ws + L.off_qinv);
  double* q_sq = reinterpret_cast<double*>(ws + L.off_qsq);
  float* q_scale = reinterpret_cast<float*>(ws + L.off_qscale);
  int32_t* n_surv = reinterpret_cast<int32_t*>(ws + L.off_nsurv);
  int32_t* ghist = reinterpret_cast<int32_t*>(ws + L.off_hist);
  float* hist_inv_w = reinterpret_cast<float*>(ws + L.off_histw);
  int32_t* cnt_all = reinterpret_cast<int32_t*>(ws + L.off_cntall);
  void* qimg = ws + L.off_qimg;
  float* dump = reinterpret_cast<float*>(ws + L.off_dump);
  Cand* cand = reinterpret_cast<Cand*>(ws + L.off_cand);
  const bool reuse = (p->flags & RL_FLAG_REUSE_THRESHOLDS) != 0;
  const bool count_unf = (p->flags & RL_FLAG_COUNT_UNFILTERED) != 0 && p->row_allowed != nullptr && L.algo == RL_ALGO_TCGEN05;
  int launches = 0;
  cudaEvent_t* se = (p->flags & RL_FLAG_TIME_KERNELS) ? stage_events_for(workspace) : nullptr;
  auto mark = [&](int i) { if (se) cudaEventRecord(se[i], stream); };
  mark(0);

  RL_CUDA_CHECK(cudaMemsetAsync(cand_cnt, 0, (size_t)p->B * 4, stream));
  RL_CUDA_CHECK(cudaMemsetAsync(ghist, 0, (size_t)p->B * kHistBins * 4, stream));
  if (count_unf) RL_CUDA_CHECK(cudaMemsetAsync(cnt_all, 0, (size_t)p->B * 4, stream));
  rc = launch_query_prep(p->Q, p->B, p->d, p->metric, L.algo, p->row_stats, q_sq, q_inv, eps, stream);
  if (rc != RL_OK) return rc;
  ++launches;
  if (L.algo == RL_ALGO_TCGEN05) {
    rc = tcgen05_prepare_queries(p, q_inv, q_scale, qimg, stream);
    if (rc != RL_OK) return rc;
    ++launches;
  }

  ScanArgs a;
  memset(&a, 0, sizeof(a));
  a.E = p->E; a.inv_norm = p->inv_norm; a.sq_norm = p->sq_norm; a.row_allowed = p->row_allowed;
  a.Q = p->Q; a.q_inv_norm = q_inv; a.thr = thr; a.dump = dump; a.cand = cand; a.cand_cnt = cand_cnt;
  a.n_rows = p->n_rows; a.ld = p->ld; a.n_sample_rows = L.n_sample_rows;
  a.d = p->d; a.B = p->B; a.metric = p->metric; a.S = L.S; a.cap = L.cap;
  a.ghist = ghist; a.eps = eps; a.hist_inv_w = hist_inv_w;
  a.sel_count = L.mode_sql ? p->num_hits : (p->k - 1) * p->max_vecs_per_chunk + 1;
  a.row_alive = p->row_alive; a.cnt_all = count_unf ? cnt_all : nullptr;

  auto scan = [&](int dump_mode, int64_t n_mode_blocks) -> int {
    if (n_mode_blocks == 0) return RL_OK;
    a.dump_mode = dump_mode;
    a.n_mode_blocks = n_mode_blocks;
    ++launches;
    if (L.algo == RL_ALGO_TCGEN05) return launch_scan_tcgen05(a, p, q_scale, qimg, sms, stream);
    return launch_scan_fp32(a, stream);
  };

  mark(1);
  if (!reuse) {
    rc = scan(1, L.n_sample_blocks);
    if (rc != RL_OK) return rc;
  } else {
    RL_CUDA_CHECK(cudaMemcpyAsync(thr, thr_out, (size_t)p->B * 4, cudaMemcpyDeviceToDevice, stream));
  }
  mark(2);
  SelectArgs s;
  s.dump = dump; s.row_chunk = p->row_chunk; s.eps = eps; s.thr = thr; s.cand = cand; s.cand_cnt = cand_cnt;
  s.ghist = ghist; s.hist_inv_w = hist_inv_w;
  s.n_sample_rows = L.n_sample_rows; s.n_rows = p->n_rows; s.S = L.S; s.cap = L.cap; s.mode_sql = L.mode_sql;
  s.sel_k = L.sel_k; s.reuse_thr = reuse ? 1 : 0;
  rc = launch_select(s, p->B, stream);
  if (rc != RL_OK) return rc;
  ++launches;
  mark(3);
  rc = scan(0, L.n_main_blocks);
  if (rc != RL_OK) return rc;
  mark(4);

  FinalizeArgs f;
  f.E = p->E; f.row_chunk = p->row_chunk; f.Q = p->Q; f.q_sq = q_sq; f.eps = eps; f.cand = cand; f.cand_rw = cand; f.cand_cnt = cand_cnt;
  f.thr_out = thr_out; f.hit_sim = hit_sim; f.hit_chunk = hit_chunk; f.hit_count = hit_count; f.status = status;
  f.n_surv = n_surv; f.header = hdr; f.ld = p->ld; f.chunk_base = p->chunk_base; f.n_sample_rows = L.n_sample_rows;
  f.d = p->d; f.metric = p->metric; f.cap = L.cap; f.mode_sql = L.mode_sql;
  f.sel_k = L.mode_sql ? p->num_hits : (p->k - 1) * p->max_vecs_per_chunk + 1;
  f.H = L.H; f.launches = launches + 1; f.S = L.S; f.algo = L.algo; f.e_f16 = p->e_dtype; f.counted_unfiltered = count_unf ? 1 : 0;
  rc = launch_finalize(f, p->B, stream);
  mark(5);
  return rc;
}

extern "C" int rl_maxsim_count_at_least(const rl_scan_params* p, const float* sim_floor, int bound, int32_t* counts,
                                        void* workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  int sms = 148;
  int rc = device_sm_count(&sms);
  if (rc != RL_OK) return rc;
  Layout L;
  rc = make_layout(p, sms, &L);
  if (rc != RL_OK) return rc;
  if (p->B == 0) return RL_OK;
  RL_REQUIRE(sim_floor && counts && p->Q, RL_EINVAL, "rl_maxsim_count_at_least: null pointer");
  RL_REQUIRE(bound >= -1 && bound <= 1, RL_EINVAL, "rl_maxsim_count_at_least: bound must be -1, 0 or +1");
  if (p->n_rows == 0) {
    RL_CUDA_CHECK(cudaMemsetAsync(counts, 0, (size_t)p->B * 4, stream));
    return RL_OK;
  }
  RL_REQUIRE(p->E && p->inv_norm && p->sq_norm, RL_EINVAL, "rl_maxsim_count_at_least: null index pointer");
  RL_REQUIRE(workspace != nullptr && workspace_bytes >= L.total, RL_ENOSPACE,
             "rl_maxsim_count_at_least: workspace %zu < required %zu", workspace_bytes, L.total);
  RL_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, RL_EINVAL, "workspace must be 256-byte aligned");
  unsigned char* ws = static_cast<unsigned char*>(workspace);
  int32_t* cand_cnt = reinterpret_cast<int32_t*>(ws + L.off_cnt);
  float* thr = reinterpret_cast<float*>(ws + L.off_thr);
  float* eps = reinterpret_cast<float*>(ws + L.off_eps);
  float* q_inv = reinterpret_cast<float*>(ws + L.off_qinv);
  double* q_sq = reinterpret_cast<double*>(ws + L.off_qsq);
  float* q_scale = reinterpret_cast<float*>(ws + L.off_qscale);
  int32_t* ghist = reinterpret_cast<int32_t*>(ws + L.off_hist);
  float* hist_inv_w = reinterpret_cast<float*>(ws + L.off_histw);
  void* qimg = ws + L.off_qimg;

  RL_CUDA_CHECK(cudaMemsetAsync(cand_cnt, 0, (size_t)p->B * 4, stream));
  RL_CUDA_CHECK(cudaMemsetAsync(ghist, 0, (size_t)p->B * kHistBins * 4, stream));
  RL_CUDA_CHECK(cudaMemsetAsync(hist_inv_w, 0, (size_t)p->B * 4, stream));
  rc = launch_query_prep(p->Q, p->B, p->d, p->metric, L.algo, p->row_stats, q_sq, q_inv, eps, stream);
  if (rc != RL_OK) return rc;
  if (L.algo == RL_ALGO_TCGEN05) {
    rc = tcgen05_prepare_queries(p, q_inv, q_scale, qimg, stream);
    if (rc != RL_OK) return rc;
  }
  rc = launch_sim_floor_to_thr(sim_floor, q_sq, eps, p->metric, bound, p->B, thr, stream);
  if (rc != RL_OK) return rc;

  // One emit-mode pass over every block with a zero-capacity candidate list: rows at or above the
  // threshold are counted, nothing is stored, and the online refinement is off (sel_count unreachable).
  ScanArgs a;
  memset(&a, 0, sizeof(a));
  a.E = p->E; a.inv_norm = p->inv_norm; a.sq_norm = p->sq_norm; a.row_allowed = p->row_allowed;
  a.Q = p->Q; a.q_inv_norm = q_inv; a.thr = thr; a.dump = nullptr; a.cand = nullptr; a.cand_cnt = cand_cnt;
  a.n_rows = p->n_rows; a.ld = p->ld; a.n_sample_rows = 0;
  a.d = p->d; a.B = p->B; a.metric = p->metric; a.S = 0; a.cap = 0;
  a.ghist = ghist; a.eps = eps; a.hist_inv_w = hist_inv_w;
  a.sel_count = 0x7fffffff;
  a.dump_mode = 0;
  a.n_mode_blocks = L.n_blocks;
  rc = L.algo == RL_ALGO_TCGEN05 ? launch_scan_tcgen05(a, p, q_scale, qimg, sms, stream) : launch_scan_fp32(a, stream);
  if (rc != RL_OK) return rc;
  RL_CUDA_CHECK(cudaMemcpyAsync(counts, cand_cnt, (size_t)p->B * 4, cudaMemcpyDeviceToDevice, stream));
  return RL_OK;
}

extern "C" int rl_maxsim_kernel_times(const void* workspace, float* ms) {
  RL_REQUIRE(workspace && ms, RL_EINVAL, "rl_maxsim_kernel_times: null pointer");
  std::lock_guard<std::mutex> lock(g_ev_mutex);
  auto it = g_events.find(workspace);
  RL_REQUIRE(it != g_events.end() && it->second.valid && it->second.count > 0, RL_EINVAL,
             "rl_maxsim_kernel_times: no timed call on this workspace");
  StageEvents& se = it->second;
  for (int i = 0; i + 1 < kNumStageEvents; ++i) ms[i] = 0.f;
  const int n = se.count;
  for (int c = 0; c < n; ++c) {
    cudaEvent_t* set = se.ev[(se.next - 1 - c + 2 * kEventRing) % kEventRing];
    RL_CUDA_CHECK(cudaEventSynchronize(set[kNumStageEvents - 1]));
    for (int i = 0; i + 1 < kNumStageEvents; ++i) {
      float t = 0.f;
      RL_CUDA_CHECK(cudaEventElapsedTime(&t, set[i], set[i + 1]));
      ms[i] += t / (float)n;
    }
  }
  se.count = 0;
  return RL_OK;
}

extern "C" int rl_maxsim_release(const void* workspace) {
  // Drops the CUDA events rl_maxsim_topk created for this workspace (RL_FLAG_TIME_KERNELS); call it
  // before the workspace memory is freed or handed to another use.  A workspace never timed is a no-op.
  std::lock_guard<std::mutex> lock(g_ev_mutex);
  auto it = g_events.find(workspace);
  if (it == g_events.end()) return RL_OK;
  if (it->second.valid)
    for (int r = 0; r < kEventRing; ++r)
      for (int i = 0; i < kNumStageEvents; ++i) cudaEventDestroy(it->second.ev[r][i]);
  g_events.erase(it);
  return RL_OK;
}

extern "C" int rl_maxsim_stats(const rl_scan_params* p, const void* workspace, rl_scan_stats* out, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  RL_REQUIRE(p && workspace && out, RL_EINVAL, "rl_maxsim_stats: null pointer");
  Layout L;
  int rc = make_layout(p, 148, &L);
  if (rc != RL_OK) return rc;
  memset(out, 0, sizeof(*out));
  if (p->B == 0 || p->n_rows == 0) return RL_OK;
  const unsigned char* ws = static_cast<const unsigned char*>(workspace);
  Header h;
  RL_CUDA_CHECK(cudaMemcpyAsync(&h, ws + L.off_hdr, sizeof(h), cudaMemcpyDeviceToHost, stream));
  int32_t* cnt = new int32_t[2 * (size_t)p->B];
  cudaError_t e1 = cudaMemcpyAsync(cnt, ws + L.off_cnt, (size_t)p->B * 4, cudaMemcpyDeviceToHost, stream);
  cudaError_t e2 = cudaMemcpyAsync(cnt + p->B, ws + L.off_nsurv, (size_t)p->B * 4, cudaMemcpyDeviceToHost, stream);
  cudaError_t e3 = cudaStreamSynchronize(stream);
  if (e1 != cudaSuccess || e2 != cudaSuccess || e3 != cudaSuccess) {
    delete[] cnt;
    set_error("rl_maxsim_stats: copy failed");
    return RL_ECUDA;
  }
  out->launches = h.launches;
  out->sample_stride = h.sample_stride;
  out->cand_cap = h.cand_cap;
  out->algo = h.algo;
  out->n_sample_rows = h.n_sample_rows;
  for (int b = 0; b < p->B; ++b) {
    out->cand_total += cnt[b];
    if (cnt[b] > out->cand_max) out->cand_max = cnt[b];
    out->survivors_total += cnt[p->B + b];
    if (cnt[p->B + b] > out->survivors_max) out->survivors_max = cnt[p->B + b];
  }
  delete[] cnt;
  return RL_OK;
}

extern "C" int rl_maxsim_copy_dump(const rl_scan_params* p, const void* workspace, float* dst, int64_t* n_sample_rows,
                                   void* stream) {
  RL_REQUIRE(p && workspace && n_sample_rows, RL_EINVAL, "rl_maxsim_copy_dump: null pointer");
  Layout L;
  int rc = make_layout(p, 148, &L);
  if (rc != RL_OK) return rc;
  *n_sample_rows = L.n_sample_rows;
  if (dst != nullptr && p->B > 0 && L.n_sample_rows > 0) {
    RL_CUDA_CHECK(cudaMemcpyAsync(dst, static_cast<const unsigned char*>(workspace) + L.off_dump,
                                  (size_t)p->B * L.n_sample_rows * 4, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  }
  return RL_OK;
}

extern "C" int rl_topk_merge(const float* hit_sim, const int64_t* hit_chunk, const int32_t* hit_count, int R, int B,
                             int H, int num_hits, int k, float* out_sim, int64_t* out_chunk, int32_t* out_count,
                             void* stream) {
  RL_REQUIRE(R >= 1 && B >= 0 && H >= 1 && k >= 1 && num_hits >= 0, RL_EINVAL, "rl_topk_merge: bad sizes");
  if (B == 0) return RL_OK;
  RL_REQUIRE(hit_sim && hit_chunk && hit_count && out_sim && out_chunk && out_count, RL_EINVAL,
             "rl_topk_merge: null pointer");
  MergeArgs m;
  m.hit_sim = hit_sim; m.hit_chunk = hit_chunk; m.hit_count = hit_count; m.out_sim = out_sim;
  m.out_chunk = out_chunk; m.out_count = out_count; m.R = R; m.B = B; m.H = H; m.num_hits = num_hits; m.k = k;
  m.win = 0; m.prefilter = 0; m.sim_rs = 0; m.chunk_rs = 0; m.count_rs = 0;
  return launch_merge(m, (cudaStream_t)stream);
}

extern "C" size_t rl_hits_packed_bytes(int B, int H, int with_status) {
  if (B < 0 || H < 0) return 0;
  const size_t raw = (size_t)B * H * 12 + (size_t)B * 4 * (with_status ? 2 : 1);
  return (raw + 15) / 16 * 16;
}

extern "C" int rl_topk_merge_packed(const void* packed, int64_t rank_stride_bytes, int R, int B, int H, int num_hits, int k,
                                    float* out_sim, int64_t* out_chunk, int32_t* out_count, void* stream) {
  RL_REQUIRE(R >= 1 && B >= 0 && H >= 1 && k >= 1 && num_hits >= 0, RL_EINVAL, "rl_topk_merge_packed: bad sizes");
  if (B == 0) return RL_OK;
  RL_REQUIRE(packed && out_sim && out_chunk && out_count, RL_EINVAL, "rl_topk_merge_packed: null pointer");
  RL_REQUIRE(rank_stride_bytes % 8 == 0 && (reinterpret_cast<uintptr_t>(packed) & 7) == 0 &&
                 rank_stride_bytes >= (int64_t)B * H * 12 + (int64_t)B * 4,
             RL_EINVAL, "rl_topk_merge_packed: rank stride must be a multiple of 8 covering one packed list");
  const unsigned char* base = static_cast<const unsigned char*>(packed);
  MergeArgs m;
  m.hit_chunk = reinterpret_cast<const int64_t*>(base);
  m.hit_sim = reinterpret_cast<const float*>(base + (size_t)B * H * 8);
  m.hit_count = reinterpret_cast<const int32_t*>(base + (size_t)B * H * 12);
  m.out_sim = out_sim; m.out_chunk = out_chunk; m.out_count = out_count;
  m.R = R; m.B = B; m.H = H; m.num_hits = num_hits; m.k = k; m.win = 0; m.prefilter = 0;
  m.chunk_rs = rank_stride_bytes / 8; m.sim_rs = rank_stride_bytes / 4; m.count_rs = rank_stride_bytes / 4;
  return launch_merge(m, (cudaStream_t)stream);
}

namespace rl {
__global__ void unfiltered_bound_kernel(const Header* hdr, const int32_t* cand_cnt, const int32_t* cnt_all, int B,
                                        int64_t* bound) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  // not counted (fp32 scan / flag not set): no bound
  bound[b] = hdr->counted_unfiltered ? (int64_t)cand_cnt[b] + (int64_t)cnt_all[b] + hdr->n_sample_rows : (int64_t)-1;
}
}  // namespace rl

extern "C" int rl_maxsim_unfiltered_bound(const rl_scan_params* p, const void* workspace, int64_t* bound, void* stream) {
  RL_REQUIRE(p && workspace && bound, RL_EINVAL, "rl_maxsim_unfiltered_bound: null pointer");
  Layout L;
  int rc = make_layout(p, 148, &L);
  if (rc != RL_OK) return rc;
  if (p->B == 0) return RL_OK;
  const unsigned char* ws = static_cast<const unsigned char*>(workspace);
  unfiltered_bound_kernel<<<(p->B + 127) / 128, 128, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const Header*>(ws + L.off_hdr), reinterpret_cast<const int32_t*>(ws + L.off_cnt),
      reinterpret_cast<const int32_t*>(ws + L.off_cntall), p->B, bound);
  RL_CUDA_CHECK(cudaGetLastError());
  return RL_OK;
}
