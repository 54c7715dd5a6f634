// Merge of per-rank range-search records (tt_range_merge), the range counterpart of tt_shard_merge.
//
// Each rank's record holds, per query, the exact count of its qualifying rows and the best min(count, L) of them,
// sorted by (score desc, id asc) - when the rank certified the query (flag 1).  An uncertified rank's count and list
// may disagree (its list can be empty or short while its count is exact or larger), so such a run is merged with
// length 0: the merged query is uncertified anyway and is replaced after the rank's re-run.  The global count is the sum
// of the counts, and the global best min(count, L) lie in the union of the per-rank lists, so the merge needs no
// certificate of its own: a query is exact iff every rank certified it.  One CTA per query:
//   1. With at most L listed keys in all, every key goes out.  Otherwise the L-th largest key of the union is found by
//      bisection over the 64-bit key space; each step counts the keys >= the probe in every run with a warp-wide
//      32-ary search in global memory (3 dependent loads for a run of 16384).  The probe's counts are the prefix
//      lengths p_g of the runs, with sum L (keys are unique: ids are global rows).
//   2. The <= L selected keys are staged in dynamic shared memory (L * 8 bytes, at most 128 KiB).
//   3. A key's output position is its index in its run plus, for every other run, the number of larger keys found by
//      binary search in shared memory (as in shard_merge_kernel); no sort.
#include "tt_common.cuh"

namespace tt {

constexpr int RM_THREADS = 256;
constexpr int RM_WARPS = RM_THREADS / 32;
constexpr int RM_MAX_G = 64;

struct RangeRun {
  const float* scores;
  const long long* ids;
};

__device__ __forceinline__ RangeRun range_run(const unsigned char* gathered, size_t rank_stride, size_t off_scores,
                                              size_t off_ids, int g, int q, int L) {
  const unsigned char* rec = gathered + (size_t)g * rank_stride;
  return {reinterpret_cast<const float*>(rec + off_scores) + (size_t)q * L,
          reinterpret_cast<const long long*>(rec + off_ids) + (size_t)q * L};
}

__device__ __forceinline__ unsigned long long run_key(const RangeRun& r, int j) {
  return make_key(r.scores[j], (uint32_t)r.ids[j]);
}

// Number of keys >= t in a run of n keys sorted descending; the whole warp calls it and gets the answer.  Invariant:
// positions < lo hold keys >= t, positions >= hi keys < t.  Each round 32 lanes probe evenly spaced positions.
__device__ int warp_count_ge(const RangeRun& r, int n, unsigned long long t, int lane) {
  int lo = 0, hi = n;
  while (hi > lo) {
    const int step = (hi - lo + 31) >> 5;
    const int p = lo + (lane + 1) * step - 1;
    const bool ge = p < hi && run_key(r, p) >= t;
    const int c = __popc(__ballot_sync(0xffffffffu, ge));
    const int p_fail = lo + (c + 1) * step - 1;        // the first probe that failed, if it was in range
    if (p_fail < hi) hi = p_fail;
    lo += c * step;
    if (lo > hi) lo = hi;
  }
  return lo;
}

__global__ void __launch_bounds__(RM_THREADS)
range_merge_kernel(const unsigned char* __restrict__ gathered, size_t rank_stride, size_t off_counts, size_t off_scores,
                   size_t off_ids, size_t off_flags, int G, int L, long long* __restrict__ counts,
                   float* __restrict__ scores, long long* __restrict__ ids, int* __restrict__ flags,
                   int* __restrict__ n_uncertified) {
  extern __shared__ __align__(16) unsigned char msm[];
  unsigned long long* key = reinterpret_cast<unsigned long long*>(msm);     // [<= L] selected keys, run after run
  __shared__ int s_n[RM_MAX_G];        // run lengths min(counts_g, L); 0 for a rank that did not certify the query
  __shared__ int s_p[RM_MAX_G];        // keys taken from each run
  __shared__ int s_off[RM_MAX_G + 1];
  __shared__ unsigned long long s_lo, s_hi;
  const int q = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid < G) {
    const unsigned char* rec = gathered + (size_t)tid * rank_stride;
    const long long c = reinterpret_cast<const long long*>(rec + off_counts)[q];
    const int f = reinterpret_cast<const int*>(rec + off_flags)[q];
    s_n[tid] = (f != 1 || c < 0) ? 0 : (int)(c > L ? L : c);
  }
  __syncthreads();
  if (tid == 0) {
    long long cnt = 0;
    int why = 0, total = 0;
    bool ok = true;
    unsigned long long lo = ~0ull, hi = 0ull;
    for (int g = 0; g < G; ++g) {
      const unsigned char* rec = gathered + (size_t)g * rank_stride;
      cnt += reinterpret_cast<const long long*>(rec + off_counts)[q];
      const int f = reinterpret_cast<const int*>(rec + off_flags)[q];
      if (f != 1) {
        ok = false;
        if (f < 0) why |= -f;
      }
      total += s_n[g];
      if (s_n[g] > 0) {
        const RangeRun r = range_run(gathered, rank_stride, off_scores, off_ids, g, q, L);
        lo = min(lo, run_key(r, s_n[g] - 1));
        hi = max(hi, run_key(r, 0));
      }
    }
    counts[q] = cnt;
    flags[q] = ok ? 1 : -why;
    if (!ok) atomicAdd(n_uncertified, 1);
    // bisection bounds: every key is >= lo (total > L of them), no key is >= hi + 1
    s_lo = lo;
    s_hi = hi + 1;
    s_off[RM_MAX_G] = total;
  }
  __syncthreads();
  const int total = s_off[RM_MAX_G];
  if (total <= L) {
    if (tid < G) s_p[tid] = s_n[tid];
  } else {
    for (;;) {
      const unsigned long long lo = s_lo, hi = s_hi;
      if (hi - lo <= 1) break;
      const unsigned long long mid = lo + (hi - lo) / 2;
      for (int g = warp; g < G; g += RM_WARPS) {
        const int c = warp_count_ge(range_run(gathered, rank_stride, off_scores, off_ids, g, q, L), s_n[g], mid, lane);
        if (lane == 0) s_p[g] = c;
      }
      __syncthreads();
      if (tid == 0) {
        int c = 0;
        for (int g = 0; g < G; ++g) c += s_p[g];
        if (c >= L) {
          s_lo = mid;
          if (c == L) s_hi = mid + 1;     // mid selects exactly L keys: done
        } else {
          s_hi = mid;
        }
      }
      __syncthreads();
    }
    // the L-th largest key is s_lo: the runs' prefixes of keys >= it hold exactly L keys
    const unsigned long long t = s_lo;
    for (int g = warp; g < G; g += RM_WARPS) {
      const int c = warp_count_ge(range_run(gathered, rank_stride, off_scores, off_ids, g, q, L), s_n[g], t, lane);
      if (lane == 0) s_p[g] = c;
    }
  }
  __syncthreads();
  if (tid == 0) {
    // Unique keys give sum(p_g) <= L.  Equal keys (ids repeated across runs, which a valid record never has) could make
    // the prefixes hold more: cut them to L so that no staged key and no output position reaches L.
    int o = 0;
    for (int g = 0; g < G; ++g) {
      s_p[g] = min(s_p[g], L - o);
      s_off[g] = o;
      o += s_p[g];
    }
    s_off[G] = o;
  }
  __syncthreads();
  const int m = s_off[G];
  for (int g = 0; g < G; ++g) {
    const RangeRun r = range_run(gathered, rank_stride, off_scores, off_ids, g, q, L);
    for (int j = tid; j < s_p[g]; j += RM_THREADS) key[s_off[g] + j] = run_key(r, j);
  }
  __syncthreads();
  float* out_s = scores + (size_t)q * L;
  long long* out_i = ids + (size_t)q * L;
  for (int i = tid; i < m; i += RM_THREADS) {
    int g = 0;
    while (i >= s_off[g + 1]) ++g;
    const unsigned long long ki = key[i];
    int rank = i - s_off[g];
    for (int h = 0; h < G; ++h) {
      if (h == g) continue;
      const unsigned long long* lst = key + s_off[h];
      int lo = 0, hi = s_p[h];
      while (lo < hi) { const int mid = (lo + hi) >> 1; if (lst[mid] > ki) lo = mid + 1; else hi = mid; }
      rank += lo;
    }
    if (rank < L) {
      out_s[rank] = key_score(ki);
      out_i[rank] = (long long)key_row(ki);
    }
  }
  for (int i = m + tid; i < L; i += RM_THREADS) {
    out_s[i] = -INFINITY;
    out_i[i] = -1;
  }
}

}  // namespace tt

using namespace tt;

extern "C" __attribute__((visibility("default"))) int tt_range_merge(const void* gathered, size_t rank_stride, size_t off_counts,
                              size_t off_scores, size_t off_ids, size_t off_flags, int G, int nq, int L, int64_t* counts,
                              float* scores, int64_t* ids, int32_t* flags, int32_t* n_uncertified, void* stream) {
  TT_CHECK_ARG(gathered && counts && scores && ids && flags && n_uncertified, "null pointer");
  TT_CHECK_ARG(G >= 1 && G <= RM_MAX_G, "need 1 <= G <= 64");
  TT_CHECK_ARG(nq >= 0, "need nq >= 0");
  TT_CHECK_ARG(L >= 1 && L <= TT_FLAT_RANGE_MAX_RESULTS, "need 1 <= L <= TT_FLAT_RANGE_MAX_RESULTS");
  TT_CHECK_ARG(reinterpret_cast<uintptr_t>(gathered) % 8 == 0 && off_counts % 8 == 0 && off_scores % 4 == 0 &&
               off_ids % 8 == 0 && off_flags % 4 == 0 && rank_stride % 8 == 0, "misaligned record layout");
  cudaStream_t st = (cudaStream_t)stream;
  TT_CHECK_CUDA(cudaMemsetAsync(n_uncertified, 0, sizeof(int32_t), st));
  if (nq == 0) return TT_OK;
  const size_t smem = (size_t)L * 8;
  TT_CHECK_CUDA(cudaFuncSetAttribute(range_merge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  range_merge_kernel<<<nq, RM_THREADS, smem, st>>>(reinterpret_cast<const unsigned char*>(gathered), rank_stride,
                                                   off_counts, off_scores, off_ids, off_flags, G, L,
                                                   reinterpret_cast<long long*>(counts), scores,
                                                   reinterpret_cast<long long*>(ids), flags, n_uncertified);
  TT_CHECK_LAUNCH();
  return TT_OK;
}
