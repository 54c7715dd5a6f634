// Range search (tt_flat_range_search): every catalog row whose fp32 score is strictly above a per-query radius, its
// exact count and the best L of them, certified per query like the top-K search.
//
//   1. thr[q] = radius[q] - eps[q] rounded toward -inf, hi[q] = radius[q] + eps[q] rounded toward +inf.  A row's bf16
//      tensor-core score is within eps of its fp32 score, so every row scoring above the radius has a bf16 score
//      >= thr (it is a candidate), and every candidate whose bf16 score is > hi scores above the radius in fp32.
//   2. The main scan of the top-K search (flat_scan.cu, FILTER instances for label filters) with that threshold: no
//      sample pass and no threshold selection.  Its per-(query, slice) counters keep counting past a full segment, so a
//      query whose candidates did not fit reports exactly how much room a re-run needs.
//   3. flat_range_finalize_kernel, one CTA per query, streaming the candidate segments from global memory (a low
//      radius can give millions of candidates): count the certain ones, rescore the band [thr, hi] in fp32 and count
//      those above the radius; b_L = L-th largest bf16 score (radix select); rescore the candidates >= b_L -
//      PRUNE_MARGIN * eps, keep those above the radius, sort, emit the best L.
#include <float.h>
#include <algorithm>
#include "tt_common.cuh"
#include "flat_internal.cuh"
#include "flat_scan_common.cuh"
#include "flat_select_common.cuh"

namespace tt {

constexpr int RANGE_KEY_CAP = 24576;    // candidates one CTA ranks in shared memory (192 KiB of keys)
constexpr int RANGE_SORT_MAX = 16384;   // keys the bitonic sort takes (a power of two <= RANGE_KEY_CAP)

__global__ void range_threshold_kernel(const float* __restrict__ radius, const float* __restrict__ eps, int nq,
                                       float* __restrict__ thr, float* __restrict__ hi) {
  pdl_trigger();
  pdl_wait();
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q < nq) {
    thr[q] = __fsub_rd(radius[q], eps[q]);
    hi[q] = __fadd_ru(radius[q], eps[q]);
  }
}

// Keys to rank in shared memory for at most L results: room for the L best and the rows within the pruning margin of
// the L-th.  A power of two up to the sort's limit, so that the sort of every list that fits needs no extra room.
static int range_key_cap(int L) {
  if (L > RANGE_SORT_MAX / 2) return RANGE_KEY_CAP;
  int c = 4096;
  while (c < 2 * L) c <<= 1;
  return c;
}

// flags: 1 = certified; otherwise -(reason bits): 1 a candidate segment overflowed (need[q] = the largest segment
// count: re-run with room for it), 2 more candidates within reach of the L-th than one CTA ranks, 4 tensor-core / fp32
// score mismatch beyond eps, 8 the L-th result does not clear the bound of the rows that were not rescored.
// EXCL: candidates the query excludes are dropped at every step (never counted, never ranked).
// The 256-thread instances get up to 128 registers (ptxas spills them at its own choice of 64); the 1024-thread one
// is held to 64 by its size.
template <int NT, bool EXCL>
__global__ void __launch_bounds__(NT, NT > 512 ? 0 : 2)
flat_range_finalize_kernel(const float* __restrict__ qn, const float* __restrict__ Xn, long long N, int D, int L,
                           long long id_offset, const float* __restrict__ radius, const float* __restrict__ thr,
                           const float* __restrict__ hi, const float* __restrict__ eps,
                           const unsigned int* __restrict__ seg_cnt, const uint2* __restrict__ cand, int nslices,
                           int seg_cap, int key_cap, long long* __restrict__ counts, float* __restrict__ scores,
                           long long* __restrict__ ids, int* __restrict__ flags, int* __restrict__ need,
                           int* __restrict__ n_uncertified, const long long* __restrict__ excl, int E) {
  pdl_trigger();
  pdl_wait();
  extern __shared__ __align__(16) unsigned char fsm[];
  unsigned long long* key = reinterpret_cast<unsigned long long*>(fsm);   // [key_cap]
  float* qs = reinterpret_cast<float*>(key + key_cap);
  unsigned int* ex = reinterpret_cast<unsigned int*>(qs + D);           // EXCL: the query's sorted exclusion list
  __shared__ int s_off[FINALIZE_MAX_SLICES + 1];
  __shared__ unsigned int s_hist[256];
  __shared__ int s_wsum[NT / 32];
  __shared__ int s_digit, s_kk, s_any_ex, s_bad, s_m;
  __shared__ unsigned int s_need, s_count, s_valid;
  __shared__ float s_fl;
  constexpr int NWARPS = NT / 32;
  constexpr int RANGE_U = 2;   // rows a warp rescores at once
  const int q = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int EP = EXCL ? next_pow2(E) : 0;

  // ---- 1. segment sizes -> offsets, the largest segment count, the query, the exclusion list ---------------
  if (tid == 0) { s_bad = 0; s_m = 0; s_count = 0u; s_valid = 0u; s_fl = -INFINITY; }
  stage_query<NT, EXCL>(q, seg_cnt, nslices, seg_cap, qn, D, excl, E, id_offset, N, s_off, &s_need, qs, ex, EP, &s_any_ex);
  const bool overflow = s_need > (unsigned int)seg_cap;
  const int n = s_off[nslices];
  const float my_eps = eps[q], t = thr[q], h = hi[q], rad = radius[q];
  const bool any_ex = EXCL && s_any_ex;
  const bool vec = (D % 4 == 0) && ((reinterpret_cast<uintptr_t>(Xn) & 15) == 0);
  auto cand_at = [&](int i) { return segment_entry(cand, s_off, nslices, seg_cap, q, i); };
  auto allowed = [&](uint32_t row) { return !(any_ex && is_excluded(ex, EP, row)); };

  // ---- 2. exact count: candidates above hi are certainly above the radius; the band [thr, hi] is rescored ------
  // Each warp takes 32 consecutive candidates per step; the band rows among them are rescored RANGE_U at a time.
  {
    unsigned int cnt = 0, nvalid = 0;
    int bad = 0;
    for (int base = warp * 32; base < n; base += NT) {
      const int i = base + lane;
      const uint2 e = (i < n) ? cand_at(i) : make_uint2(NEG_INF_BITS, 0u);
      const bool valid = i < n && allowed(e.y);
      const float v = __uint_as_float(e.x);
      nvalid += valid ? 1u : 0u;
      if (valid && v > h) ++cnt;
      unsigned int band = __ballot_sync(0xffffffffu, valid && !(v > h));
      while (band) {
        uint32_t row[RANGE_U];
        bool ok[RANGE_U];
        float bsc[RANGE_U], sc[RANGE_U];
        int src[RANGE_U];
#pragma unroll
        for (int u = 0; u < RANGE_U; ++u) {
          src[u] = band ? __ffs(band) - 1 : -1;
          if (band) band &= band - 1;
          row[u] = __shfl_sync(0xffffffffu, e.y, src[u] < 0 ? 0 : src[u]);
          bsc[u] = __shfl_sync(0xffffffffu, v, src[u] < 0 ? 0 : src[u]);
          ok[u] = src[u] >= 0 && (long long)row[u] < N;   // row >= N cannot happen unless the scan is broken
        }
        rescore_rows<RANGE_U>(qs, Xn, D, vec, row, ok, sc, lane);
#pragma unroll
        for (int u = 0; u < RANGE_U; ++u) {
          if (lane == src[u]) {
            if (!ok[u] || !(fabsf(bsc[u] - sc[u]) <= my_eps)) bad = 1;
            if (ok[u] && sc[u] > rad) ++cnt;
          }
        }
      }
    }
    cnt = __reduce_add_sync(0xffffffffu, cnt);
    nvalid = __reduce_add_sync(0xffffffffu, nvalid);
    if (lane == 0) { atomicAdd(&s_count, cnt); atomicAdd(&s_valid, nvalid); }
    if (bad) s_bad = 1;
  }
  __syncthreads();
  const unsigned int count = s_count, nvalid = s_valid;

  // ---- 3. b_L = L-th largest bf16 score of the allowed candidates, streamed from global memory ---------------
  float cutoff = -INFINITY;
  if (nvalid > (unsigned int)L) {
    const uint32_t b = radix_select_desc<NT>(n, L, s_hist, &s_digit, &s_kk, [&](int i) -> uint32_t {
      const uint2 e = cand_at(i);
      return allowed(e.y) ? float_to_ordered(__uint_as_float(e.x)) : 0u;
    });
    cutoff = ordered_to_float(b) - PRUNE_MARGIN * my_eps;
  }

  // ---- 4. the candidates within reach of the L-th -> shared memory, rescored in fp32, kept if above the radius --
  for (int i = tid; i < n; i += NT) {
    const uint2 e = cand_at(i);
    const float v = __uint_as_float(e.x);
    if (v >= cutoff && allowed(e.y)) {
      const int pos = atomicAdd(&s_m, 1);
      if (pos < key_cap) key[pos] = make_key(v, e.y);
    }
  }
  __syncthreads();
  const int m_all = s_m;
  const bool rank_overflow = m_all > key_cap;
  const int m = rank_overflow ? 0 : m_all;
  {
    int bad = 0;
    for (int i0 = warp * RANGE_U; i0 < m; i0 += NWARPS * RANGE_U) {
      uint32_t row[RANGE_U];
      bool ok[RANGE_U];
      float bsc[RANGE_U], sc[RANGE_U];
#pragma unroll
      for (int u = 0; u < RANGE_U; ++u) {
        const unsigned long long k = (i0 + u < m) ? key[i0 + u] : 0ull;
        row[u] = key_row(k);
        bsc[u] = key_score(k);
        ok[u] = (i0 + u < m) && (long long)row[u] < N;
      }
      rescore_rows<RANGE_U>(qs, Xn, D, vec, row, ok, sc, lane);
      __syncwarp();
      if (lane == 0) {
#pragma unroll
        for (int u = 0; u < RANGE_U; ++u) {
          if (i0 + u >= m) continue;
          if (!ok[u] || !(fabsf(bsc[u] - sc[u]) <= my_eps)) bad = 1;
          key[i0 + u] = (ok[u] && sc[u] > rad) ? make_key(sc[u], row[u]) : 0ull;
        }
      }
    }
    if (bad) s_bad = 1;
  }
  __syncthreads();
  // key 0 marks a rescored row at or below the radius
  const int m2 = compact_keys<NT>(key, m, s_wsum, [](unsigned long long k) { return k != 0ull; });

  // ---- 5. more than the sort takes (only with L > RANGE_SORT_MAX / 2): keep the keys >= the L-th fp32 score -----
  int m3 = m2;
  bool tie_overflow = false;
  if (m2 > RANGE_SORT_MAX) {
    const uint32_t s = radix_select_desc<NT>(m2, L, s_hist, &s_digit, &s_kk, [&](int i) { return (uint32_t)(key[i] >> 32); });
    m3 = compact_keys<NT>(key, m2, s_wsum, [&](unsigned long long k) { return (uint32_t)(k >> 32) >= s; });
    tie_overflow = m3 > RANGE_SORT_MAX;     // more than RANGE_SORT_MAX - L rows tie with the L-th fp32 score
    if (tie_overflow) m3 = 0;
  }

  // ---- 6. order by (score desc, row asc) and emit the best min(m3, L) ---------------------------------------
  const int P2 = next_pow2(m3 < 1 ? 1 : m3);
  for (int i = m3 + tid; i < P2; i += NT) key[i] = 0ull;
  __syncthreads();
  bitonic_sort_desc(key, P2);
  const int nout = m3 < L ? m3 : L;
  for (int i = tid; i < L; i += NT) {
    if (i < nout) {
      scores[(long long)q * L + i] = key_score(key[i]);
      ids[(long long)q * L + i] = (long long)key_row(key[i]) + id_offset;
      if (i == L - 1) s_fl = key_score(key[i]);
    } else {
      scores[(long long)q * L + i] = -INFINITY;
      ids[(long long)q * L + i] = -1;
    }
  }
  __syncthreads();
  if (tid == 0) {
    // Every allowed candidate above the radius was ranked when the count equals the rows kept in step 4 (then the
    // output is all of them, or the best L).  Otherwise the rows that were not rescored have bf16 scores below
    // c = max(thr, cutoff), hence fp32 scores below c + eps, and the L-th result must clear that.
    int why = 0;
    if (overflow) why |= 1;
    if (rank_overflow || tie_overflow) why |= 2;
    if (s_bad) why |= 4;
    const float c = fmaxf(t, cutoff);
    if (!(why & 2) && (unsigned int)m2 != count && !(nout == L && s_fl >= c + my_eps)) why |= 8;
    flags[q] = why == 0 ? 1 : -why;
    if (why) atomicAdd(n_uncertified, 1);
    counts[q] = (long long)count;
    need[q] = (int)s_need;
  }
}

static int launch_range_finalize(const ScanPlan& pl, const float* qn, const float* Xn, long long N, int D, int nq, int L,
                                 long long id_offset, const float* radius, const float* thr, const float* hi,
                                 const float* eps, const unsigned int* seg_cnt, const void* cand, long long* counts,
                                 float* scores, long long* ids, int* flags, int* need, int* n_uncertified,
                                 const long long* excl, int E, cudaStream_t st) {
  TT_CHECK_ARG(pl.main_slices <= FINALIZE_MAX_SLICES, "too many catalog slices");
  const bool with_excl = excl != nullptr && E > 0;
  const int key_cap = range_key_cap(L);
  const size_t smem = finalize_smem_bytes(key_cap, D, with_excl ? E : 0);
  count_launch();
  return launch_finalize_instance(nq, with_excl, [&](auto nt, auto ex) {
    auto kern = flat_range_finalize_kernel<decltype(nt)::value, decltype(ex)::value>;
    TT_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    TT_CHECK_CUDA(launch_pdl(kern, dim3(nq), dim3(nt), smem, st, qn, Xn, N, D, L, id_offset, radius, thr, hi, eps, seg_cnt,
                             reinterpret_cast<const uint2*>(cand), pl.main_slices, pl.seg_cap, key_cap, counts, scores, ids,
                             flags, need, n_uncertified, ex ? excl : nullptr, ex ? E : 0));
    return TT_OK;
  });
}

ScanPlan make_range_plan(long long N, int D, int nq, long long cand_budget) {
  ScanPlan pl = make_scan_plan(N, D, nq, 1);      // tiling, stages and slices; the sampling decisions are not used
  pl.use_threshold = true;
  pl.route_exact = false;
  pl.sample_stride = 1; pl.sample_slots = 1; pl.sample_rank = 1; pl.sample_tile_max = false; pl.sample_slices = 1;
  pl.target = (int)std::min<long long>(cand_budget, 1LL << 30);
  pl.cand_cap = 0;
  const long long slice_rows = ((long long)(pl.num_tiles + pl.main_slices - 1) / pl.main_slices) * BLOCK_N;
  long long seg = (2 * cand_budget + pl.main_slices - 1) / pl.main_slices;
  if (seg < 64) seg = 64;
  if (seg > slice_rows) seg = slice_rows;
  pl.seg_cap = (int)((seg + 63) / 64 * 64);
  return pl;
}

struct RangeWs {
  size_t qn, qh, eps, thr, hi, cnt, cand, total;
};

// the candidate segments come last: the search sizes them from the bytes it is given
static RangeWs range_ws_layout(const ScanPlan& pl, int D, int nq) {
  RangeWs w{};
  size_t o = 0;
  w.qn = o;   o += align_up((size_t)nq * D * sizeof(float), 256);
  w.qh = o;   o += align_up((size_t)pl.nq_pad * pl.Dp * 2, 256);
  w.eps = o;  o += align_up((size_t)nq * sizeof(float), 256);
  w.thr = o;  o += align_up((size_t)nq * sizeof(float), 256);
  w.hi = o;   o += align_up((size_t)nq * sizeof(float), 256);
  w.cnt = o;  o += align_up((size_t)nq * pl.main_slices * sizeof(unsigned int), 256);
  w.cand = o; o += (size_t)nq * pl.main_slices * pl.seg_cap * 8;
  w.total = o;
  return w;
}

// ------------------------------------------------------------------------------------------
// exact path: the exact path of the top-K search (launch_exact_group) for the best min(L, N) rows of every query slot,
// plus a count of the rows above the radius
__global__ void __launch_bounds__(256)
range_exact_count_kernel(const float* __restrict__ scores_ws, long long N, const float* __restrict__ radius,
                         const int* __restrict__ qsel, int slot0, unsigned int* __restrict__ cnt) {
  const int s = blockIdx.y;
  const int qi = qsel ? qsel[slot0 + s] : (slot0 + s);
  const float r = radius[qi];
  const float* sc = scores_ws + (long long)s * N;
  unsigned int c = 0;
  // an excluded or disallowed row holds a NaN sentinel: never above the radius
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += (long long)gridDim.x * blockDim.x)
    c += (sc[i] > r) ? 1u : 0u;
  c = __reduce_add_sync(0xffffffffu, c);
  if ((threadIdx.x & 31) == 0 && c) atomicAdd(cnt + s, c);
}

__global__ void __launch_bounds__(256)
range_exact_emit_kernel(const float* __restrict__ ts, const long long* __restrict__ ti, int K,
                        const unsigned int* __restrict__ cnt, const int* __restrict__ qsel, int slot0, int L,
                        long long* __restrict__ counts, float* __restrict__ scores, long long* __restrict__ ids) {
  const int s = blockIdx.x;
  const int qi = qsel ? qsel[slot0 + s] : (slot0 + s);
  const unsigned int c = cnt[s];
  const int nout = (int)min(c, (unsigned int)K);
  if (threadIdx.x == 0) counts[qi] = (long long)c;
  for (int i = threadIdx.x; i < L; i += blockDim.x) {
    scores[(long long)qi * L + i] = (i < nout) ? ts[(long long)s * K + i] : -INFINITY;
    ids[(long long)qi * L + i] = (i < nout) ? ti[(long long)s * K + i] : -1;
  }
}

struct RangeExactWs {
  size_t sel, ts, ti, cnt, total;
};
static RangeExactWs range_exact_ws_layout(int64_t N, int D, int K) {
  RangeExactWs w{};
  size_t o = 0;
  w.sel = o; o += align_up(tt_flat_search_exact_workspace_bytes(N, D, EX_QB, K), 256);
  w.ts = o;  o += align_up((size_t)EX_QB * K * sizeof(float), 256);
  w.ti = o;  o += align_up((size_t)EX_QB * K * sizeof(long long), 256);
  w.cnt = o; o += align_up(EX_QB * sizeof(unsigned int), 256);
  w.total = o;
  return w;
}

}  // namespace tt

using namespace tt;

// The filter arguments: both NULL, or both non-NULL and aligned; nullptr when valid, else the error message.
static const char* range_label_args(const uint32_t* labels, const uint32_t* require) {
  if ((labels == nullptr) != (require == nullptr)) return "labels and require must be both NULL or both non-NULL";
  if ((reinterpret_cast<uintptr_t>(labels) & 15) != 0) return "labels must be 16-byte aligned";
  if ((reinterpret_cast<uintptr_t>(require) & 7) != 0) return "require must be 8-byte aligned";
  return nullptr;
}

extern "C" __attribute__((visibility("default"))) size_t tt_flat_range_exact_workspace_bytes(int64_t N, int D, int nsel, int L) {
  (void)nsel;
  if (N < 1 || D < 1 || L < 1) return 0;
  return range_exact_ws_layout(N, D, (int)std::min<int64_t>(L, N)).total;
}

static int flat_range_exact_impl(const float* q, int nq, const int32_t* qsel, int nsel, const float* Xn, int64_t N, int D,
                                 const float* radius, int L, int64_t id_offset, int64_t* counts, float* scores,
                                 int64_t* ids, const uint32_t* labels, const uint32_t* require, const int64_t* excl,
                                 int E, void* workspace, size_t workspace_bytes, cudaStream_t st) {
  if (nsel == 0) return TT_OK;
  const int K = (int)std::min<int64_t>(L, N);
  const RangeExactWs w = range_exact_ws_layout(N, D, K);
  if (workspace_bytes < w.total) { set_error("tt_flat_range_search_exact: workspace too small"); return TT_ERR_WORKSPACE; }
  unsigned char* ws = reinterpret_cast<unsigned char*>(workspace);
  float* ts = reinterpret_cast<float*>(ws + w.ts);
  long long* ti = reinterpret_cast<long long*>(ws + w.ti);
  unsigned int* cnt = reinterpret_cast<unsigned int*>(ws + w.cnt);
  const float* scores_ws = reinterpret_cast<const float*>(ws + w.sel);
  long long gs = (N + 255) / 256;
  if (gs > (long long)num_sms() * 8) gs = (long long)num_sms() * 8;
  for (int slot0 = 0; slot0 < nsel; slot0 += EX_QB) {
    const int nslot = (nsel - slot0 < EX_QB) ? (nsel - slot0) : EX_QB;
    if (int e = launch_exact_group(q, qsel, slot0, nslot, Xn, N, D, K, id_offset, ts, reinterpret_cast<int64_t*>(ti), false,
                                   excl, E, labels, require, ws + w.sel, st)) return e;
    TT_CHECK_CUDA(cudaMemsetAsync(cnt, 0, EX_QB * sizeof(unsigned int), st));
    range_exact_count_kernel<<<dim3((unsigned)gs, nslot), 256, 0, st>>>(scores_ws, N, radius, qsel, slot0, cnt);
    TT_CHECK_LAUNCH();
    range_exact_emit_kernel<<<nslot, 256, 0, st>>>(ts, ti, K, cnt, qsel, slot0, L, reinterpret_cast<long long*>(counts),
                                                   scores, reinterpret_cast<long long*>(ids));
    TT_CHECK_LAUNCH();
  }
  return TT_OK;
}

extern "C" __attribute__((visibility("default"))) int tt_flat_range_search_exact(
    const float* q, int nq, const int32_t* qsel, int nsel, const float* Xn, int64_t N, int D, const float* radius, int L,
    int64_t id_offset, int64_t* counts, float* scores, int64_t* ids, const uint32_t* labels, const uint32_t* require,
    const int64_t* excl, int E, void* workspace, size_t workspace_bytes, void* stream) {
  const char* bad = range_label_args(labels, require);
  TT_CHECK_ARG(bad == nullptr, bad);
  TT_CHECK_ARG(E >= 0 && E <= TT_FLAT_MAX_EXCLUDE, "need 0 <= E <= TT_FLAT_MAX_EXCLUDE (1024) exclusions per query");
  TT_CHECK_ARG(excl != nullptr || E == 0, "null exclusion list with E > 0");
  TT_CHECK_ARG(q && Xn && radius && counts && scores && ids && workspace, "null pointer");
  TT_CHECK_ARG(N >= 1 && N < (1LL << 31) && D >= 1, "need 1 <= N < 2^31 rows, D >= 1");
  TT_CHECK_ARG(L >= 1 && L <= TT_FLAT_RANGE_MAX_RESULTS, "need 1 <= L <= TT_FLAT_RANGE_MAX_RESULTS (16384)");
  TT_CHECK_ARG(nq >= 0 && nsel >= 0 && (qsel != nullptr || nsel == nq), "qsel == NULL requires nsel == nq");
  TT_CHECK_ARG((size_t)EX_QB * D * sizeof(float) <= 160 * 1024, "D too large");
  return flat_range_exact_impl(q, nq, qsel, nsel, Xn, N, D, radius, L, id_offset, counts, scores, ids, labels, require, excl,
                               E, workspace, workspace_bytes, (cudaStream_t)stream);
}

extern "C" __attribute__((visibility("default"))) size_t tt_flat_range_workspace_bytes(int64_t N, int D, int nq, int64_t cand_budget) {
  if (N < 1 || D < 1 || nq < 1 || cand_budget < 1) return 0;
  const ScanPlan pl = make_range_plan(N, D, nq, cand_budget);
  if (!pl.supported) return tt_flat_range_exact_workspace_bytes(N, D, nq, TT_FLAT_RANGE_MAX_RESULTS);
  return range_ws_layout(pl, D, nq).total;
}

namespace tt {
__global__ void range_candidates_kernel(const unsigned int* __restrict__ seg_cnt, int nslices, int nq, int* __restrict__ out) {
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= nq) return;
  unsigned int t = 0;
  for (int s = 0; s < nslices; ++s) t += seg_cnt[(size_t)q * nslices + s];
  out[q] = (int)t;
}
}  // namespace tt

extern "C" __attribute__((visibility("default"))) int tt_flat_range_debug_read(const void* workspace, int64_t N, int D, int nq,
                                                                              int32_t* cnt_out, void* stream) {
  TT_CHECK_ARG(workspace && cnt_out && N >= 1 && D >= 1 && nq >= 1, "bad argument");
  const ScanPlan pl = make_range_plan(N, D, nq, 1);
  TT_CHECK_ARG(pl.supported, "this width is served by the exact path: no candidates");
  const RangeWs w = range_ws_layout(pl, D, nq);     // the counters precede the segments, whatever their capacity
  range_candidates_kernel<<<(nq + 127) / 128, 128, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const unsigned int*>(reinterpret_cast<const unsigned char*>(workspace) + w.cnt), pl.main_slices, nq,
      cnt_out);
  TT_CHECK_LAUNCH();
  return TT_OK;
}

extern "C" __attribute__((visibility("default"))) int tt_flat_range_search(
    const float* q, int nq, const float* Xn, const void* Xh, const float* stats, int64_t N, int D, const float* radius,
    int L, int64_t id_offset, int64_t* counts, float* scores, int64_t* ids, int32_t* flags, int32_t* need,
    int32_t* n_uncertified, const uint32_t* labels, const uint32_t* require, const int64_t* excl, int E, void* workspace,
    size_t workspace_bytes, void* stream) {
  const char* bad = range_label_args(labels, require);
  TT_CHECK_ARG(bad == nullptr, bad);
  TT_CHECK_ARG(E >= 0 && E <= TT_FLAT_MAX_EXCLUDE, "need 0 <= E <= TT_FLAT_MAX_EXCLUDE (1024) exclusions per query");
  TT_CHECK_ARG(excl != nullptr || E == 0, "null exclusion list with E > 0");
  TT_CHECK_ARG(q && Xn && Xh && stats && radius && counts && scores && ids && flags && need && n_uncertified, "null pointer");
  TT_CHECK_ARG(nq >= 0, "nq < 0");
  TT_CHECK_ARG(N >= 1 && N < (1LL << 31), "need 1 <= N < 2^31 rows per shard");
  TT_CHECK_ARG(D >= 1, "D < 1");
  TT_CHECK_ARG(L >= 1 && L <= TT_FLAT_RANGE_MAX_RESULTS, "need 1 <= L <= TT_FLAT_RANGE_MAX_RESULTS (16384)");
  TT_CHECK_ARG((reinterpret_cast<uintptr_t>(Xh) & 15) == 0, "Xh must be 16-byte aligned");
  TT_CHECK_ARG(workspace != nullptr, "null workspace");
  TT_CHECK_ARG((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "workspace must be 256-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  if (nq == 0) { TT_CHECK_CUDA(cudaMemsetAsync(n_uncertified, 0, sizeof(int32_t), st)); return TT_OK; }

  ScanPlan pl = make_range_plan(N, D, nq, 1);
  if (!pl.supported) {
    // rows too wide for the resident-query scan (D > 1024): the fp32 exact path serves the batch
    TT_CHECK_CUDA(cudaMemsetAsync(n_uncertified, 0, sizeof(int32_t), st));
    TT_CHECK_CUDA(cudaMemsetAsync(need, 0, (size_t)nq * sizeof(int32_t), st));
    fill_int_kernel<<<(nq + 255) / 256, 256, 0, st>>>(flags, nq, 1);
    TT_CHECK_LAUNCH();
    TT_CHECK_ARG((size_t)EX_QB * D * sizeof(float) <= 160 * 1024, "D too large");
    return flat_range_exact_impl(q, nq, nullptr, nq, Xn, N, D, radius, L, id_offset, counts, scores, ids, labels, require,
                                 excl, E, workspace, workspace_bytes, st);
  }
  // the segments take whatever room the workspace has beyond the fixed part (tt_flat_range_workspace_bytes)
  const size_t fixed = range_ws_layout(pl, D, nq).cand;
  const size_t per_row = (size_t)nq * pl.main_slices * 8;
  const long long slice_rows = ((long long)(pl.num_tiles + pl.main_slices - 1) / pl.main_slices) * BLOCK_N;
  long long seg = workspace_bytes > fixed ? (long long)((workspace_bytes - fixed) / per_row) / 64 * 64 : 0;
  if (seg > slice_rows) seg = slice_rows;     // a slice can report every one of its rows
  if (seg < 64) { set_error("tt_flat_range_search: workspace too small"); return TT_ERR_WORKSPACE; }
  pl.seg_cap = (int)seg;
  const RangeWs w = range_ws_layout(pl, D, nq);
  unsigned char* ws = reinterpret_cast<unsigned char*>(workspace);
  float* qn = reinterpret_cast<float*>(ws + w.qn);
  void* qh = ws + w.qh;
  float* eps = reinterpret_cast<float*>(ws + w.eps);
  float* thr = reinterpret_cast<float*>(ws + w.thr);
  float* hi = reinterpret_cast<float*>(ws + w.hi);
  unsigned int* cnt = reinterpret_cast<unsigned int*>(ws + w.cnt);
  void* cand = ws + w.cand;
  LabelArgs lab;
  lab.labels = labels;
  lab.require = require;

  if (int e = launch_prep_queries(q, nq, pl.nq_pad, D, pl.Dp, stats, qn, qh, eps, n_uncertified, st)) return e;
  count_launch();
  TT_CHECK_CUDA(launch_pdl(range_threshold_kernel, dim3((nq + 255) / 256), dim3(256), 0, st, radius, (const float*)eps, nq, thr, hi));
  if (int e = launch_main_scan(pl, qh, Xh, N, nq, thr, cnt, cand, st, nullptr, lab)) return e;
  return launch_range_finalize(pl, qn, Xn, N, D, nq, L, id_offset, radius, thr, hi, eps, cnt, cand,
                               reinterpret_cast<long long*>(counts), scores, reinterpret_cast<long long*>(ids), flags, need,
                               n_uncertified, reinterpret_cast<const long long*>(excl), E, st);
}
