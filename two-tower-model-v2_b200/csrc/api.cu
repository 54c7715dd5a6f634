// C-ABI glue: error reporting and the tt_flat_search orchestration (include/tt_b200.h).
#include "tt_common.cuh"
#include "flat_internal.cuh"
#include <algorithm>
#include <atomic>
#include <vector>

namespace tt {
static thread_local std::string g_last_error;
void set_error(const std::string& msg) { g_last_error = msg; }

static std::atomic<long long> g_launches{0};
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

// scan-kernel timing records (armed by tt_profile_scan_arm)
static std::vector<cudaEvent_t> g_ev;     // 2 events per record
static int g_prof_cap = 0, g_prof_n = 0;
void profile_scan_begin(cudaStream_t st) {
  if (g_prof_n < g_prof_cap) cudaEventRecord(g_ev[2 * g_prof_n], st);
}
void profile_scan_end(cudaStream_t st) {
  if (g_prof_n < g_prof_cap) { cudaEventRecord(g_ev[2 * g_prof_n + 1], st); ++g_prof_n; }
}

struct SearchWs {
  size_t qn, qh, eps, thr, cnt, cand, sample, total;
};

static SearchWs search_ws_layout(const ScanPlan& pl, int D, int nq) {
  SearchWs w{};
  size_t o = 0;
  w.qn = o;     o += align_up((size_t)nq * D * sizeof(float), 256);
  w.qh = o;     o += align_up((size_t)pl.nq_pad * pl.Dp * 2, 256);
  w.eps = o;    o += align_up((size_t)nq * sizeof(float), 256);
  w.thr = o;    o += align_up((size_t)nq * sizeof(float), 256);
  w.cnt = o;    o += align_up((size_t)nq * pl.main_slices * sizeof(unsigned int), 256);
  w.cand = o;   o += align_up((size_t)nq * pl.main_slices * pl.seg_cap * 8, 256);
  w.sample = o; o += align_up((size_t)pl.sample_slots * 8 * pl.nq_pad * sizeof(float), 256);
  w.total = o;
  return w;
}
}  // namespace tt

using namespace tt;

extern "C" __attribute__((visibility("default"))) int tt_abi_version(void) { return TT_B200_ABI_VERSION; }
extern "C" __attribute__((visibility("default"))) const char* tt_last_error(void) { return g_last_error.c_str(); }

extern "C" __attribute__((visibility("default"))) int64_t tt_kernel_launch_count(void) { return g_launches.load(); }

extern "C" __attribute__((visibility("default"))) int tt_profile_scan_arm(int max_records) {
  TT_CHECK_ARG(max_records >= 0 && max_records <= 4096, "max_records out of range");
  while ((int)g_ev.size() < 2 * max_records) {
    cudaEvent_t e;
    TT_CHECK_CUDA(cudaEventCreate(&e));
    g_ev.push_back(e);
  }
  g_prof_cap = max_records;
  g_prof_n = 0;
  return TT_OK;
}

extern "C" __attribute__((visibility("default"))) int tt_profile_scan_read(float* ms_out, int max_out) {
  int n = g_prof_n < max_out ? g_prof_n : max_out;
  for (int i = 0; i < n; ++i) {
    if (cudaEventSynchronize(g_ev[2 * i + 1]) != cudaSuccess) return -1;
    if (cudaEventElapsedTime(ms_out + i, g_ev[2 * i], g_ev[2 * i + 1]) != cudaSuccess) return -1;
  }
  g_prof_cap = 0;
  return n;
}

namespace tt {
__global__ void fill_int_kernel(int* p, int n, int v) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}
}  // namespace tt

extern "C" __attribute__((visibility("default"))) size_t tt_flat_search_workspace_bytes(int64_t N, int D, int nq, int K) {
  if (N < 1 || D < 1 || nq < 1 || K < 1) return 0;
  const ScanPlan pl = make_scan_plan(N, D, nq, K);
  if (pl.route_exact || !pl.supported) return tt_flat_search_exact_workspace_bytes(N, D, nq, K);
  return search_ws_layout(pl, D, nq).total;
}

// The K a search with E exclusions per query plans its scan for: the excluded rows are typically the query's best
// ones, so the candidate budget must cover them (include/tt_b200.h).
static int plan_k(int64_t N, int K, int E) {
  const int64_t k = (int64_t)K + (E > 0 ? E : 0);
  return (int)std::min<int64_t>(std::min<int64_t>(k, N), TT_FLAT_MAX_K);
}

extern "C" __attribute__((visibility("default"))) size_t tt_flat_search_excl_workspace_bytes(int64_t N, int D, int nq, int K, int E) {
  if (E < 0 || E > TT_FLAT_MAX_EXCLUDE || N < 1 || K < 1) return 0;
  return tt_flat_search_workspace_bytes(N, D, nq, plan_k(N, K, E));
}

static int flat_search_impl(const float* q, int nq, const float* Xn, const void* Xh, const float* stats,
                            int64_t N, int D, int K, int64_t id_offset, float* scores, int64_t* ids,
                            int32_t* flags, int32_t* n_uncertified, float* bound, const int64_t* excl, int E,
                            void* workspace, size_t workspace_bytes, void* stream, const LabelArgs& lab = LabelArgs{},
                            const GroupArgs& grp = GroupArgs{}) {
  TT_CHECK_ARG(E >= 0 && E <= TT_FLAT_MAX_EXCLUDE, "need 0 <= E <= TT_FLAT_MAX_EXCLUDE (1024) exclusions per query");
  TT_CHECK_ARG(excl != nullptr || E == 0, "null exclusion list with E > 0");
  TT_CHECK_ARG(q && Xn && Xh && stats && scores && ids && flags && n_uncertified, "null pointer");
  TT_CHECK_ARG(nq >= 0, "nq < 0");
  TT_CHECK_ARG(N >= 1 && N < (1LL << 31), "need 1 <= N < 2^31 rows per shard");
  TT_CHECK_ARG(D >= 1, "D < 1");
  TT_CHECK_ARG(K >= 1 && K <= N && K <= TT_FLAT_MAX_K, "need 1 <= K <= min(N, TT_FLAT_MAX_K)");
  TT_CHECK_ARG((reinterpret_cast<uintptr_t>(Xh) & 15) == 0, "Xh must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  if (nq == 0) { TT_CHECK_CUDA(cudaMemsetAsync(n_uncertified, 0, sizeof(int32_t), st)); return TT_OK; }

  const ScanPlan pl = make_scan_plan(N, D, nq, plan_k(N, K, E));
  TT_CHECK_ARG(workspace != nullptr, "null workspace");
  TT_CHECK_ARG((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "workspace must be 256-byte aligned");
  if (pl.route_exact || !pl.supported) {
    // K is too large a fraction of N for a sampled threshold, or the rows are too wide for the resident-query
    // scan (D > 1024): the fp32 exact path serves the batch.
    TT_CHECK_CUDA(cudaMemsetAsync(n_uncertified, 0, sizeof(int32_t), st));
    fill_int_kernel<<<(nq + 255) / 256, 256, 0, st>>>(flags, nq, 1);
    TT_CHECK_LAUNCH();
    if (bound) {   // the exact path scores every row: nothing is left unbounded
      fill_int_kernel<<<(nq + 255) / 256, 256, 0, st>>>(reinterpret_cast<int*>(bound), nq, (int)0xff800000);
      TT_CHECK_LAUNCH();
    }
    if (grp.groups)
      return tt_flat_search_exact_grouped(q, nq, nullptr, nq, Xn, N, D, K, id_offset, scores, ids, lab.labels, lab.require,
                                          excl, E, grp.groups, grp.n_groups, grp.max_per_group, workspace, workspace_bytes,
                                          stream);
    if (lab.labels)
      return tt_flat_search_exact_filtered(q, nq, nullptr, nq, Xn, N, D, K, id_offset, scores, ids, lab.labels, lab.require,
                                           excl, E, workspace, workspace_bytes, stream);
    return tt_flat_search_exact_excl(q, nq, nullptr, nq, Xn, N, D, K, id_offset, scores, ids, excl, E, workspace,
                                     workspace_bytes, stream);
  }
  const SearchWs w = search_ws_layout(pl, D, nq);
  if (workspace_bytes < w.total) { set_error("tt_flat_search: workspace too small"); return TT_ERR_WORKSPACE; }
  TT_CHECK_ARG((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "workspace must be 256-byte aligned");
  unsigned char* ws = reinterpret_cast<unsigned char*>(workspace);
  float* qn = reinterpret_cast<float*>(ws + w.qn);
  void* qh = ws + w.qh;
  float* eps = reinterpret_cast<float*>(ws + w.eps);
  float* thr = reinterpret_cast<float*>(ws + w.thr);
  unsigned int* cnt = reinterpret_cast<unsigned int*>(ws + w.cnt);
  void* cand = ws + w.cand;
  float* sample = reinterpret_cast<float*>(ws + w.sample);

  if (int e = launch_prep_queries(q, nq, pl.nq_pad, D, pl.Dp, stats, qn, qh, eps, n_uncertified, st)) return e;
  if (int e = launch_scan(pl, qh, Xh, N, nq, thr, cnt, cand, sample, st, lab)) return e;
  if (grp.groups)
    return launch_group_finalize(pl, qn, Xn, N, D, nq, K, id_offset, thr, eps, cnt, cand, scores,
                                 reinterpret_cast<long long*>(ids), flags, n_uncertified, grp, st,
                                 reinterpret_cast<const long long*>(excl), E);
  return launch_finalize(pl, qn, Xn, N, D, nq, K, id_offset, thr, eps, cnt, cand, scores,
                         reinterpret_cast<long long*>(ids), flags, n_uncertified, bound, st,
                         reinterpret_cast<const long long*>(excl), E);
}

extern "C" __attribute__((visibility("default"))) int tt_flat_search(const float* q, int nq, const float* Xn, const void* Xh, const float* stats,
                              int64_t N, int D, int K, int64_t id_offset, float* scores, int64_t* ids,
                              int32_t* flags, int32_t* n_uncertified, void* workspace, size_t workspace_bytes,
                              void* stream) {
  return flat_search_impl(q, nq, Xn, Xh, stats, N, D, K, id_offset, scores, ids, flags, n_uncertified, nullptr,
                          nullptr, 0, workspace, workspace_bytes, stream);
}

extern "C" __attribute__((visibility("default"))) int tt_flat_search_excl(const float* q, int nq, const float* Xn, const void* Xh, const float* stats,
                                   int64_t N, int D, int K, int64_t id_offset, float* scores, int64_t* ids,
                                   int32_t* flags, int32_t* n_uncertified, const int64_t* excl, int E,
                                   void* workspace, size_t workspace_bytes, void* stream) {
  return flat_search_impl(q, nq, Xn, Xh, stats, N, D, K, id_offset, scores, ids, flags, n_uncertified, nullptr,
                          excl, E, workspace, workspace_bytes, stream);
}

// The filter arguments of the *_filtered calls -> lab; nullptr when they are valid, else the error message.
static const char* label_args(const uint32_t* labels, const uint32_t* require, LabelArgs* lab) {
  if (labels == nullptr || require == nullptr)
    return "null labels or require (the unfiltered calls are the ones without _filtered)";
  if ((reinterpret_cast<uintptr_t>(labels) & 15) != 0) return "labels must be 16-byte aligned";
  if ((reinterpret_cast<uintptr_t>(require) & 7) != 0) return "require must be 8-byte aligned";
  lab->labels = labels;
  lab->require = require;
  return nullptr;
}

extern "C" __attribute__((visibility("default"))) int tt_flat_search_filtered(const float* q, int nq, const float* Xn, const void* Xh, const float* stats,
                                       int64_t N, int D, int K, int64_t id_offset, float* scores, int64_t* ids,
                                       int32_t* flags, int32_t* n_uncertified, const uint32_t* labels,
                                       const uint32_t* require, const int64_t* excl, int E, void* workspace,
                                       size_t workspace_bytes, void* stream) {
  LabelArgs lab;
  const char* bad = label_args(labels, require, &lab);
  TT_CHECK_ARG(bad == nullptr, bad);
  return flat_search_impl(q, nq, Xn, Xh, stats, N, D, K, id_offset, scores, ids, flags, n_uncertified, nullptr,
                          excl, E, workspace, workspace_bytes, stream, lab);
}

extern "C" __attribute__((visibility("default"))) size_t tt_flat_search_grouped_workspace_bytes(int64_t N, int D, int nq, int K, int E,
                                                                                      int32_t n_groups) {
  if (E < 0 || E > TT_FLAT_MAX_EXCLUDE || N < 1 || D < 1 || nq < 1 || K < 1 || n_groups < 0) return 0;
  const ScanPlan pl = make_scan_plan(N, D, nq, plan_k(N, K, E));
  if (pl.route_exact || !pl.supported) return exact_workspace_bytes(N, K, n_groups);
  return search_ws_layout(pl, D, nq).total;
}

extern "C" __attribute__((visibility("default"))) int tt_flat_search_grouped(const float* q, int nq, const float* Xn, const void* Xh,
                                                                            const float* stats, int64_t N, int D, int K,
                                                                            int64_t id_offset, float* scores, int64_t* ids,
                                                                            int32_t* flags, int32_t* n_uncertified,
                                                                            const int32_t* groups, int32_t n_groups,
                                                                            int max_per_group, const uint32_t* labels,
                                                                            const uint32_t* require, const int64_t* excl,
                                                                            int E, void* workspace, size_t workspace_bytes,
                                                                            void* stream) {
  TT_CHECK_ARG(groups != nullptr, "null groups");
  TT_CHECK_ARG(n_groups >= 0, "n_groups < 0");
  TT_CHECK_ARG(max_per_group >= 1 && max_per_group <= TT_FLAT_MAX_PER_GROUP,
               "need 1 <= max_per_group <= TT_FLAT_MAX_PER_GROUP (64)");
  TT_CHECK_ARG((labels == nullptr) == (require == nullptr), "labels and require must be both NULL or both non-NULL");
  LabelArgs lab;
  if (labels) {
    const char* bad = label_args(labels, require, &lab);
    TT_CHECK_ARG(bad == nullptr, bad);
  }
  GroupArgs grp;
  grp.groups = groups;
  grp.n_groups = n_groups;
  grp.max_per_group = max_per_group;
  return flat_search_impl(q, nq, Xn, Xh, stats, N, D, K, id_offset, scores, ids, flags, n_uncertified, nullptr,
                          excl, E, workspace, workspace_bytes, stream, lab, grp);
}

extern "C" __attribute__((visibility("default"))) int tt_flat_search_shard(const float* q, int nq, const float* Xn, const void* Xh, const float* stats,
                              int64_t N, int D, int K, int64_t id_offset, float* scores, int64_t* ids,
                              int32_t* flags, int32_t* n_uncertified, float* bound, void* workspace,
                              size_t workspace_bytes, void* stream) {
  TT_CHECK_ARG(bound != nullptr, "null bound");
  return flat_search_impl(q, nq, Xn, Xh, stats, N, D, K, id_offset, scores, ids, flags, n_uncertified, bound,
                          nullptr, 0, workspace, workspace_bytes, stream);
}

extern "C" __attribute__((visibility("default"))) int tt_flat_search_shard_excl(const float* q, int nq, const float* Xn, const void* Xh, const float* stats,
                                         int64_t N, int D, int K, int64_t id_offset, float* scores, int64_t* ids,
                                         int32_t* flags, int32_t* n_uncertified, float* bound, const int64_t* excl,
                                         int E, void* workspace, size_t workspace_bytes, void* stream) {
  TT_CHECK_ARG(bound != nullptr, "null bound");
  return flat_search_impl(q, nq, Xn, Xh, stats, N, D, K, id_offset, scores, ids, flags, n_uncertified, bound,
                          excl, E, workspace, workspace_bytes, stream);
}

extern "C" __attribute__((visibility("default"))) int tt_flat_search_shard_filtered(const float* q, int nq, const float* Xn, const void* Xh,
                                             const float* stats, int64_t N, int D, int K, int64_t id_offset,
                                             float* scores, int64_t* ids, int32_t* flags, int32_t* n_uncertified,
                                             float* bound, const uint32_t* labels, const uint32_t* require,
                                             const int64_t* excl, int E, void* workspace, size_t workspace_bytes,
                                             void* stream) {
  TT_CHECK_ARG(bound != nullptr, "null bound");
  LabelArgs lab;
  const char* bad = label_args(labels, require, &lab);
  TT_CHECK_ARG(bad == nullptr, bad);
  return flat_search_impl(q, nq, Xn, Xh, stats, N, D, K, id_offset, scores, ids, flags, n_uncertified, bound,
                          excl, E, workspace, workspace_bytes, stream, lab);
}

// ------------------------------------------------------------------------------------------
// Sharded catalogs with ONE threshold for the whole catalog (include/tt_b200.h).
extern "C" __attribute__((visibility("default"))) int tt_flat_shard_plan_ok(int64_t N_local, int64_t N_total, int D, int nq, int K) {
  if (N_local < 1 || N_total < N_local || D < 1 || nq < 1 || K < 1) return 0;
  bool ok = false;
  (void)make_shard_plan(N_local, N_total, D, nq, K, &ok);
  return ok ? 1 : 0;
}

extern "C" __attribute__((visibility("default"))) size_t tt_flat_shard_workspace_bytes(int64_t N_local, int64_t N_total, int D, int nq, int K) {
  if (N_local < 1 || N_total < N_local || D < 1 || nq < 1 || K < 1) return 0;
  bool ok = false;
  const ScanPlan pl = make_shard_plan(N_local, N_total, D, nq, K, &ok);
  return ok ? search_ws_layout(pl, D, nq).total : 0;
}

static int flat_shard_sample_impl(const float* q, int nq, const void* Xh, const float* stats, int64_t N_local,
                                  int64_t N_total, int D, int K, float* topr, void* workspace, size_t workspace_bytes,
                                  void* stream, const LabelArgs& lab) {
  TT_CHECK_ARG(q && Xh && stats && topr && workspace, "null pointer");
  TT_CHECK_ARG(nq >= 1 && N_local >= 1 && N_local < (1LL << 31) && N_total >= N_local && D >= 1 && K >= 1, "bad sizes");
  TT_CHECK_ARG((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "workspace must be 256-byte aligned");
  bool ok = false;
  const ScanPlan pl = make_shard_plan(N_local, N_total, D, nq, K, &ok);
  if (!ok) { set_error("tt_flat_shard_sample: no global-threshold plan for these sizes (use tt_flat_search_shard)"); return TT_ERR_UNSUPPORTED; }
  const SearchWs w = search_ws_layout(pl, D, nq);
  if (workspace_bytes < w.total) { set_error("tt_flat_shard_sample: workspace too small"); return TT_ERR_WORKSPACE; }
  cudaStream_t st = (cudaStream_t)stream;
  unsigned char* ws = reinterpret_cast<unsigned char*>(workspace);
  if (int e = launch_prep_queries(q, nq, pl.nq_pad, D, pl.Dp, stats, reinterpret_cast<float*>(ws + w.qn), ws + w.qh,
                                  reinterpret_cast<float*>(ws + w.eps), nullptr, st)) return e;
  return launch_sample(pl, ws + w.qh, Xh, N_local, nq, nullptr, topr, reinterpret_cast<float*>(ws + w.sample), st,
                       false, lab);
}

extern "C" __attribute__((visibility("default"))) int tt_flat_shard_sample(const float* q, int nq, const void* Xh, const float* stats, int64_t N_local,
                                    int64_t N_total, int D, int K, float* topr, void* workspace,
                                    size_t workspace_bytes, void* stream) {
  return flat_shard_sample_impl(q, nq, Xh, stats, N_local, N_total, D, K, topr, workspace, workspace_bytes, stream,
                                LabelArgs{});
}

extern "C" __attribute__((visibility("default"))) int tt_flat_shard_sample_filtered(const float* q, int nq, const void* Xh, const float* stats,
                                             int64_t N_local, int64_t N_total, int D, int K, const uint32_t* labels,
                                             const uint32_t* require, float* topr, void* workspace,
                                             size_t workspace_bytes, void* stream) {
  LabelArgs lab;
  const char* bad = label_args(labels, require, &lab);
  TT_CHECK_ARG(bad == nullptr, bad);
  return flat_shard_sample_impl(q, nq, Xh, stats, N_local, N_total, D, K, topr, workspace, workspace_bytes, stream, lab);
}

static int flat_shard_search_impl(int nq, const float* Xn, const void* Xh, int64_t N_local, int64_t N_total, int D,
                                  int K, int64_t id_offset, const float* topr_g, int G, float* scores, int64_t* ids,
                                  int32_t* flags, int32_t* n_uncertified, float* bound, const int64_t* excl, int E,
                                  void* workspace, size_t workspace_bytes, void* stream,
                                  const LabelArgs& lab = LabelArgs{}) {
  TT_CHECK_ARG(E >= 0 && E <= TT_FLAT_MAX_EXCLUDE, "need 0 <= E <= TT_FLAT_MAX_EXCLUDE (1024) exclusions per query");
  TT_CHECK_ARG(excl != nullptr || E == 0, "null exclusion list with E > 0");
  TT_CHECK_ARG(Xn && Xh && topr_g && scores && ids && flags && n_uncertified && bound && workspace, "null pointer");
  TT_CHECK_ARG(nq >= 1 && G >= 1 && G <= 64 && N_local >= 1 && N_local < (1LL << 31) && N_total >= N_local, "bad sizes");
  TT_CHECK_ARG(K >= 1 && K <= N_local && K <= TT_FLAT_MAX_K, "need 1 <= K <= min(N_local, TT_FLAT_MAX_K)");
  bool ok = false;
  // the sample pass and the plan checks were called with K_plan = min(K + E, N_total, TT_FLAT_MAX_K)
  const ScanPlan pl = make_shard_plan(N_local, N_total, D, nq, plan_k(N_total, K, E), &ok);
  if (!ok) { set_error("tt_flat_shard_search: no global-threshold plan for these sizes"); return TT_ERR_UNSUPPORTED; }
  const SearchWs w = search_ws_layout(pl, D, nq);
  if (workspace_bytes < w.total) { set_error("tt_flat_shard_search: workspace too small"); return TT_ERR_WORKSPACE; }
  cudaStream_t st = (cudaStream_t)stream;
  unsigned char* ws = reinterpret_cast<unsigned char*>(workspace);
  float* qn = reinterpret_cast<float*>(ws + w.qn);
  float* eps = reinterpret_cast<float*>(ws + w.eps);
  float* thr = reinterpret_cast<float*>(ws + w.thr);
  unsigned int* cnt = reinterpret_cast<unsigned int*>(ws + w.cnt);
  if (int e = launch_select_gathered(topr_g, G, nq, pl.sample_rank, thr, n_uncertified, st)) return e;
  if (int e = launch_main_scan(pl, ws + w.qh, Xh, N_local, nq, thr, cnt, ws + w.cand, st, nullptr, lab)) return e;
  return launch_finalize(pl, qn, Xn, N_local, D, nq, K, id_offset, thr, eps, cnt, ws + w.cand, scores,
                         reinterpret_cast<long long*>(ids), flags, n_uncertified, bound, st,
                         reinterpret_cast<const long long*>(excl), E);
}

extern "C" __attribute__((visibility("default"))) int tt_flat_shard_search(int nq, const float* Xn, const void* Xh, int64_t N_local, int64_t N_total, int D,
                                    int K, int64_t id_offset, const float* topr_g, int G, float* scores, int64_t* ids,
                                    int32_t* flags, int32_t* n_uncertified, float* bound, void* workspace,
                                    size_t workspace_bytes, void* stream) {
  return flat_shard_search_impl(nq, Xn, Xh, N_local, N_total, D, K, id_offset, topr_g, G, scores, ids, flags,
                                n_uncertified, bound, nullptr, 0, workspace, workspace_bytes, stream);
}

extern "C" __attribute__((visibility("default"))) int tt_flat_shard_search_excl(int nq, const float* Xn, const void* Xh, int64_t N_local, int64_t N_total,
                                         int D, int K, int64_t id_offset, const float* topr_g, int G, float* scores,
                                         int64_t* ids, int32_t* flags, int32_t* n_uncertified, float* bound,
                                         const int64_t* excl, int E, void* workspace, size_t workspace_bytes,
                                         void* stream) {
  return flat_shard_search_impl(nq, Xn, Xh, N_local, N_total, D, K, id_offset, topr_g, G, scores, ids, flags,
                                n_uncertified, bound, excl, E, workspace, workspace_bytes, stream);
}

extern "C" __attribute__((visibility("default"))) int tt_flat_shard_search_filtered(int nq, const float* Xn, const void* Xh, int64_t N_local,
                                             int64_t N_total, int D, int K, int64_t id_offset, const float* topr_g,
                                             int G, float* scores, int64_t* ids, int32_t* flags,
                                             int32_t* n_uncertified, float* bound, const uint32_t* labels,
                                             const uint32_t* require, const int64_t* excl, int E, void* workspace,
                                             size_t workspace_bytes, void* stream) {
  LabelArgs lab;
  const char* bad = label_args(labels, require, &lab);
  TT_CHECK_ARG(bad == nullptr, bad);
  return flat_shard_search_impl(nq, Xn, Xh, N_local, N_total, D, K, id_offset, topr_g, G, scores, ids, flags,
                                n_uncertified, bound, excl, E, workspace, workspace_bytes, stream, lab);
}

// ------------------------------------------------------------------------------------------
// Diagnostic: dense bf16 tensor-core scores of a small catalog (parity tests of the scan itself).
namespace tt {
__global__ void scatter_scores_kernel(const unsigned int* __restrict__ seg_cnt, const uint2* __restrict__ cand,
                                      int nslices, int seg_cap, long long N, float* __restrict__ out) {
  const int q = blockIdx.y;
  for (int sl = blockIdx.x; sl < nslices; sl += gridDim.x) {
    const unsigned int n = min(seg_cnt[(size_t)q * nslices + sl], (unsigned int)seg_cap);
    const uint2* seg = cand + ((size_t)q * nslices + sl) * seg_cap;
    for (unsigned int i = threadIdx.x; i < n; i += blockDim.x) {
      const uint2 c = seg[i];
      if ((long long)c.y < N) out[(long long)q * N + c.y] = __uint_as_float(c.x);
    }
  }
}
}  // namespace tt

extern "C" __attribute__((visibility("default"))) size_t tt_flat_scan_scores_workspace_bytes(int64_t N, int D, int nq) {
  if (N < 1 || D < 1 || nq < 1) return 0;
  ScanPlan pl = make_scan_plan(N, D, nq, 1);
  pl.use_threshold = false;
  pl.route_exact = false;
  pl.seg_cap = (pl.num_tiles + pl.main_slices - 1) / pl.main_slices * 256;
  return search_ws_layout(pl, D, nq).total;
}

extern "C" __attribute__((visibility("default"))) int tt_flat_scan_scores(const float* q, int nq, const void* Xh, const float* stats, int64_t N, int D,
                                   float* out, void* workspace, size_t workspace_bytes, void* stream) {
  TT_CHECK_ARG(q && Xh && stats && out && workspace, "null pointer");
  TT_CHECK_ARG(nq >= 1 && N >= 1 && N <= (1 << 22) && D >= 1, "need nq >= 1, 1 <= N <= 2^22, D >= 1");
  cudaStream_t st = (cudaStream_t)stream;
  ScanPlan pl = make_scan_plan(N, D, nq, 1);
  if (!pl.supported) { set_error("tt_flat_scan_scores: D too large"); return TT_ERR_UNSUPPORTED; }
  pl.use_threshold = false;
  pl.route_exact = false;
  pl.seg_cap = (pl.num_tiles + pl.main_slices - 1) / pl.main_slices * 256;
  const SearchWs w = search_ws_layout(pl, D, nq);
  if (workspace_bytes < w.total) { set_error("tt_flat_scan_scores: workspace too small"); return TT_ERR_WORKSPACE; }
  unsigned char* ws = reinterpret_cast<unsigned char*>(workspace);
  float* qn = reinterpret_cast<float*>(ws + w.qn);
  void* qh = ws + w.qh;
  float* eps = reinterpret_cast<float*>(ws + w.eps);
  float* thr = reinterpret_cast<float*>(ws + w.thr);
  unsigned int* cnt = reinterpret_cast<unsigned int*>(ws + w.cnt);
  void* cand = ws + w.cand;
  float* sample = reinterpret_cast<float*>(ws + w.sample);
  TT_CHECK_CUDA(cudaMemsetAsync(out, 0xFF, (size_t)nq * N * sizeof(float), st));   // NaN = "row never reported"
  if (int e = launch_prep_queries(q, nq, pl.nq_pad, D, pl.Dp, stats, qn, qh, eps, nullptr, st)) return e;
  if (int e = launch_scan(pl, qh, Xh, N, nq, thr, cnt, cand, sample, st)) return e;
  scatter_scores_kernel<<<dim3(64, nq), 256, 0, st>>>(cnt, reinterpret_cast<const uint2*>(cand), pl.main_slices, pl.seg_cap, N, out);
  TT_CHECK_LAUNCH();
  return TT_OK;
}

// Host-only: the decisions tt_flat_search would take for (N, D, nq, K); lets CPU tests check the planner.
extern "C" __attribute__((visibility("default"))) int tt_flat_plan_describe(int64_t N, int D, int nq, int K, int32_t* out16) {
  TT_CHECK_ARG(out16 != nullptr && N >= 1 && D >= 1 && nq >= 1 && K >= 1, "bad argument");
  const ScanPlan pl = make_scan_plan(N, D, nq, K);
  const int32_t v[16] = {pl.supported, pl.pair ? 2 * pl.block_m : pl.block_m, pl.num_kb, pl.num_stages, pl.nqu, pl.num_tiles,
                         pl.use_threshold, pl.route_exact, pl.target, pl.cand_cap, pl.sample_stride, pl.sample_slots,
                         pl.sample_rank, pl.main_slices, pl.seg_cap, (int32_t)pl.smem_bytes};
  for (int i = 0; i < 16; ++i) out16[i] = v[i];
  return TT_OK;
}

// Diagnostic: after tt_flat_search on `workspace`, copy out each query's scan threshold and its total
// number of candidates (sum over slices, before capacity clamping).  Device pointers.
namespace tt {
__global__ void debug_read_kernel(const float* thr, const unsigned int* seg_cnt, int nslices, int nq,
                                  float* thr_out, int* cnt_out) {
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= nq) return;
  unsigned int t = 0;
  for (int s = 0; s < nslices; ++s) t += seg_cnt[(size_t)q * nslices + s];
  thr_out[q] = thr[q];
  cnt_out[q] = (int)t;
}
}  // namespace tt

extern "C" __attribute__((visibility("default"))) int tt_flat_debug_read(const void* workspace, int64_t N, int D, int nq, int K,
                                                        float* thr_out, int32_t* cnt_out, void* stream) {
  TT_CHECK_ARG(workspace && thr_out && cnt_out && N >= 1 && D >= 1 && nq >= 1 && K >= 1, "bad argument");
  const ScanPlan pl = make_scan_plan(N, D, nq, K);
  TT_CHECK_ARG(!pl.route_exact, "this (N, K) is served by the exact path: no thresholds");
  const SearchWs w = search_ws_layout(pl, D, nq);
  const unsigned char* ws = reinterpret_cast<const unsigned char*>(workspace);
  debug_read_kernel<<<(nq + 127) / 128, 128, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const float*>(ws + w.thr), reinterpret_cast<const unsigned int*>(ws + w.cnt), pl.main_slices, nq,
      thr_out, cnt_out);
  TT_CHECK_LAUNCH();
  return TT_OK;
}
