// Grouped top-K (tt_flat_search_grouped): the exact top-K with at most m rows per group (a brand, a seller).
//
// Contract: rows carry a group id (groups[r] in [0, n_groups), anything else = ungrouped).  Walk the rows the query
// may return (allowed by its label filter, not on its exclusion list) in (fp32 score desc, row asc) order and TAKE a
// row if it is ungrouped or fewer than m rows of its group were taken before it; stop after K takes.  The result is the
// taken rows in walk order, (-inf, -1) padded.
//
// Tensor path, flat_group_finalize_kernel (one CTA per query; the scan, its plan and its FILTER instances are the
// top-K search's, planned for K_plan = min(K + E, N, TT_FLAT_MAX_K)):
//   1. gather the candidates and drop the excluded ones (as flat_finalize_kernel);
//   2. sort them by bf16 key (n <= cand_cap, a power of two) and walk them: b* = bf16 score of the K-th taken
//      candidate, -inf when fewer than K are taken;
//   3. rescore the candidates with bf16 >= cutoff = b* - PRUNE_MARGIN * eps in fp32 (rescore_rows: the same score every
//      other path gives a row), with the same self-check as the top-K finalize;
//   4. sort the rescored rows by fp32 key, walk them again and emit the first K taken rows; f_K = K-th taken score;
//   5. certificate, the same a-posteriori check as flat_finalize_kernel: c = max(scan threshold, cutoff) and every
//      allowed row that was not rescored has a bf16 score below c, hence an fp32 score below c + eps.  If f_K >= c + eps,
//      every row the global walk visits before its K-th take ranks at or above the K-th taken rescored row, so it has
//      fp32 >= c + eps and was rescored.  The walk over the rescored rows therefore visits the same rows in the same
//      order up to its K-th take and takes the same decisions, which depend only on the rows visited before: the result
//      is exact.  b* only decides how much is rescored; the walk over any superset of the bf16 walk's rows takes at
//      least as many rows (a group's takes are min(m, its rows)), so step 4 takes K whenever step 2 did.
//      flags: bit 1 candidate list overflow, 2 fewer than K rows could be taken (only when c > -inf: with c = -inf
//      every allowed row was rescored and a short answer is the answer), 4 self-check, 8 f_K below c + eps.
//
// The walk: one warp, 32 sorted keys at a time.  __match_any_sync on the group id gives each lane its rank among the
// lanes of its group in the chunk; a shared-memory open-addressing table maps a group id to the rows taken so far.
// A group enters the table only with a take, so it never holds more than K groups: 2 * next_pow2(K) slots (at most
// 32 KiB) keep it at most half full whatever n or the group layout.
//
// Exact path (launch_exact_group with groups): after the exclusion and filter sentinels, m rounds over each slot's
// scores find, per group, the m-th best (score, row) key of its remaining rows; every grouped row below it gets the
// exclusion sentinel, and the unchanged select / collect / sort follow.  Each round is one pass over the N scores, so
// m <= TT_FLAT_MAX_PER_GROUP (64) bounds the cost at 64 passes.
#include "tt_common.cuh"
#include "flat_internal.cuh"
#include "flat_select_common.cuh"

namespace tt {

constexpr int GROUP_SLOT_FREE = -1;

// group of a row for the walk; -1 = ungrouped (a negative id, an id >= n_groups, or not a row of the table)
__device__ __forceinline__ int row_group(const int* __restrict__ groups, int n_groups, long long N, uint32_t row) {
  if ((long long)row >= N) return -1;
  const int g = __ldg(groups + row);
  return (g >= 0 && g < n_groups) ? g : -1;
}

__device__ __forceinline__ int group_slot(int g, int tab_bits) {
  return (int)(((uint32_t)g * 0x9E3779B1u) >> (32 - tab_bits));
}

// The group walk over key[0, n) (sorted descending; key 0 = not a row), run by warp 0 of the CTA; the table
// tab_g / tab_c [1 << tab_bits] must be free on entry.  take(pos, k) is called by the lane that takes key k as the
// pos-th taken row.  Returns the number of rows taken (at most K) in every lane of warp 0.
template <typename Take>
__device__ __forceinline__ int group_walk(const unsigned long long* key, int n, int K, int m,
                                          const int* __restrict__ groups, int n_groups, long long N, int* tab_g,
                                          int* tab_c, int tab_bits, Take take) {
  const int lane = threadIdx.x & 31;
  const unsigned int lt = (1u << lane) - 1u;
  const int tmask = (1 << tab_bits) - 1;
  int taken = 0;
  for (int base = 0; base < n && taken < K; base += 32) {
    const int i = base + lane;
    const unsigned long long k = (i < n) ? key[i] : 0ull;
    const bool valid = k != 0ull;
    const int g = valid ? row_group(groups, n_groups, N, key_row(k)) : -1;
    const unsigned int peers = __match_any_sync(0xffffffffu, g);
    const int leader = __ffs(peers) - 1;
    const bool lead = g >= 0 && lane == leader;
    int slot = -1, prior = 0;
    if (lead) {
      for (int h = group_slot(g, tab_bits);; h = (h + 1) & tmask) {
        const int t = tab_g[h];
        if (t == g) { slot = h; prior = tab_c[h]; break; }
        if (t == GROUP_SLOT_FREE) break;
      }
    }
    prior = __shfl_sync(0xffffffffu, prior, leader);
    const bool want = valid && (g < 0 || prior + __popc(peers & lt) < m);
    const int pos = taken + __popc(__ballot_sync(0xffffffffu, want) & lt);
    const bool tk = want && pos < K;
    const unsigned int tb = __ballot_sync(0xffffffffu, tk);
    if (tk) take(pos, k);
    if (lead) {
      const int t = __popc(tb & peers);
      if (t > 0) {
        if (slot >= 0) {
          tab_c[slot] = prior + t;
        } else {
          int h = group_slot(g, tab_bits);
          while (atomicCAS(&tab_g[h], GROUP_SLOT_FREE, g) != GROUP_SLOT_FREE) h = (h + 1) & tmask;
          tab_c[h] = t;
        }
      }
    }
    __syncwarp();
    taken += __popc(tb);
  }
  return taken;
}

template <int NT>
__device__ __forceinline__ void free_table(int* tab_g, int slots) {
  for (int i = threadIdx.x; i < slots; i += NT) tab_g[i] = GROUP_SLOT_FREE;
}

// 1 + log2 of the table size for K (2 * next_pow2(K) slots)
__host__ __device__ __forceinline__ int group_tab_bits(int K) {
  int b = 1;
  while ((1 << (b - 1)) < K) ++b;
  return b;
}

// The 256-thread instances may use more than 128 registers: ptxas spills them at 64 and at 128 (the 1024-thread ones
// are held to 64 by their size and do not spill).
template <int FIN_THREADS, bool EXCL>
__global__ void __launch_bounds__(FIN_THREADS, FIN_THREADS > 512 ? 0 : 1)
flat_group_finalize_kernel(const float* __restrict__ qn, const float* __restrict__ Xn, long long N, int D, int K,
                           long long id_offset, const float* __restrict__ thr, const float* __restrict__ eps,
                           const unsigned int* __restrict__ seg_cnt, const uint2* __restrict__ cand, int nslices,
                           int seg_cap, int cand_cap, float* __restrict__ scores, long long* __restrict__ ids,
                           int* __restrict__ flags, int* __restrict__ n_uncertified, const int* __restrict__ groups,
                           int n_groups, int max_per_group, const long long* __restrict__ excl, int E) {
  pdl_trigger();
  pdl_wait();
  extern __shared__ __align__(16) unsigned char fsm[];
  unsigned long long* key = reinterpret_cast<unsigned long long*>(fsm);
  float* qs = reinterpret_cast<float*>(key + cand_cap);
  unsigned int* ex = reinterpret_cast<unsigned int*>(qs + D);   // EXCL: the query's sorted exclusion list
  const int EP = EXCL ? next_pow2(E) : 0;
  const int tab_bits = group_tab_bits(K);
  const int tab_slots = 1 << tab_bits;
  int* tab_g = reinterpret_cast<int*>(ex + EP);
  int* tab_c = tab_g + tab_slots;
  __shared__ int s_off[FINALIZE_MAX_SLICES + 1];
  __shared__ int s_wsum[FIN_THREADS / 32];
  __shared__ int s_bad, s_any_ex, s_taken;
  __shared__ unsigned int s_need;
  __shared__ float s_bk, s_fk;
  const int q = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int NWARPS = FIN_THREADS / 32;

  // ---- 1. segment sizes -> offsets, the query, the exclusion list; gather --------------------------
  if (tid == 0) { s_bad = 0; s_bk = -INFINITY; s_fk = -INFINITY; s_taken = 0; }
  stage_query<FIN_THREADS, EXCL>(q, seg_cnt, nslices, seg_cap, qn, D, excl, E, id_offset, N, s_off, &s_need, qs, ex, EP,
                                 &s_any_ex);
  const int total = s_off[nslices];
  const bool overflow = s_need > (unsigned int)seg_cap || total > cand_cap;
  int n = min(total, cand_cap);
  const float my_eps = eps[q];
  const float t = thr[q];
  for (int i = tid; i < n; i += FIN_THREADS) {
    const uint2 e = segment_entry(cand, s_off, nslices, seg_cap, q, i);
    key[i] = make_key(__uint_as_float(e.x), e.y);
  }
  __syncthreads();
  if constexpr (EXCL) {
    if (s_any_ex)
      n = compact_keys<FIN_THREADS>(key, n, s_wsum,
                                    [&](unsigned long long k) { return !is_excluded(ex, EP, key_row(k)); });
  }

  // ---- 2. sort by bf16 key, walk: b* = bf16 score of the K-th taken candidate --------------------------
  {
    const int P = next_pow2(n < 1 ? 1 : n);
    for (int i = n + tid; i < P; i += FIN_THREADS) key[i] = 0ull;
    free_table<FIN_THREADS>(tab_g, tab_slots);
    __syncthreads();
    bitonic_sort_desc(key, P);   // ends with a barrier
    if (warp == 0) {
      const int taken = group_walk(key, n, K, max_per_group, groups, n_groups, N, tab_g, tab_c, tab_bits,
                                   [=](int pos, unsigned long long k) { if (pos == K - 1) s_bk = key_score(k); });
      (void)taken;
    }
    __syncthreads();
  }
  const float cutoff = (s_bk == -INFINITY) ? -INFINITY : s_bk - PRUNE_MARGIN * my_eps;

  // ---- 3. prune (the sorted survivors stay a prefix) and rescore in fp32 --------------------------------
  int m = n;
  if (cutoff > -INFINITY)
    m = compact_keys<FIN_THREADS>(key, n, s_wsum, [&](unsigned long long k) { return key_score(k) >= cutoff; });
  const bool vec = (D % 4 == 0) && ((reinterpret_cast<uintptr_t>(Xn) & 15) == 0);
  int bad = 0;
  constexpr bool WIDE = FIN_THREADS > 512;   // the rescoring schedule of flat_finalize_kernel
  constexpr int U = WIDE ? 2 : 4;
  for (int i0 = warp * U; i0 < m; i0 += NWARPS * U) {
    uint32_t row[U];
    float bsc[U], sc[U];
    bool ok[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int i = i0 + u;
      const unsigned long long kk64 = (i < m) ? key[i] : 0ull;
      row[u] = key_row(kk64);
      bsc[u] = key_score(kk64);
      ok[u] = (i < m) && ((long long)row[u] < N);
    }
    rescore_rows<U, WIDE>(qs, Xn, D, vec, row, ok, sc, lane);
    __syncwarp();
    if (lane == 0) {
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int i = i0 + u;
        if (i >= m) continue;
        if (ok[u]) {
          key[i] = make_key(sc[u], row[u]);
          if (!(fabsf(bsc[u] - sc[u]) <= my_eps)) bad = 1;
        } else {
          key[i] = 0ull;
          bad = 1;
        }
      }
    }
  }
  if (bad) s_bad = 1;

  // ---- 4. sort by fp32 key, walk again, emit the first K taken rows ------------------------------------
  {
    const int P = next_pow2(m < 1 ? 1 : m);
    for (int i = m + tid; i < P; i += FIN_THREADS) key[i] = 0ull;
    free_table<FIN_THREADS>(tab_g, tab_slots);
    __syncthreads();
    bitonic_sort_desc(key, P);
    if (warp == 0) {
      const int taken = group_walk(key, m, K, max_per_group, groups, n_groups, N, tab_g, tab_c, tab_bits,
                                   [=](int pos, unsigned long long k) {
                                     scores[(long long)q * K + pos] = key_score(k);
                                     ids[(long long)q * K + pos] = (long long)key_row(k) + id_offset;
                                     if (pos == K - 1) s_fk = key_score(k);
                                   });
      if (lane == 0) s_taken = taken;
    }
    __syncthreads();
    for (int i = s_taken + tid; i < K; i += FIN_THREADS) {
      scores[(long long)q * K + i] = -INFINITY;
      ids[(long long)q * K + i] = -1;
    }
  }

  // ---- 5. certificate -----------------------------------------------------------------------------------
  if (tid == 0) {
    const float c = fmaxf(t, cutoff);   // every allowed row not rescored has a bf16 score < c
    const bool unbounded = (c == -INFINITY);
    int why = 0;
    if (overflow) why |= 1;
    if (s_taken < K && !unbounded) why |= 2;
    if (s_bad) why |= 4;
    if (s_taken >= K && !unbounded && !(s_fk >= c + my_eps)) why |= 8;
    flags[q] = why == 0 ? 1 : -why;
    if (why) atomicAdd(n_uncertified, 1);
  }
}

int launch_group_finalize(const ScanPlan& pl, const float* qn, const float* Xn, long long N, int D, int nq, int K,
                          long long id_offset, const float* thr, const float* eps, const unsigned int* seg_cnt,
                          const void* cand, float* scores, long long* ids, int* flags, int* n_uncertified,
                          const GroupArgs& grp, cudaStream_t st, const long long* excl, int E) {
  TT_CHECK_ARG(pl.main_slices <= FINALIZE_MAX_SLICES, "too many catalog slices");
  const bool with_excl = excl != nullptr && E > 0;
  const size_t smem = finalize_smem_bytes(pl.cand_cap, D, with_excl ? E : 0) + ((size_t)8 << group_tab_bits(K));
  count_launch();
  return launch_finalize_instance(nq, with_excl, [&](auto nt, auto ex) {
    auto kern = flat_group_finalize_kernel<decltype(nt)::value, decltype(ex)::value>;
    TT_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    TT_CHECK_CUDA(launch_pdl(kern, dim3(nq), dim3(nt), smem, st, qn, Xn, N, D, K, id_offset, thr, eps, seg_cnt,
                             reinterpret_cast<const uint2*>(cand), pl.main_slices, pl.seg_cap, pl.cand_cap, scores, ids,
                             flags, n_uncertified, grp.groups, grp.n_groups, grp.max_per_group, ex ? excl : nullptr,
                             ex ? E : 0));
    return TT_OK;
  });
}

// ------------------------------------------------------------------------------------------
// exact path: per (slot, group) u64 state last[g] (the key of the group's last kept row; rows below it are dropped)
// and best[g] (this round's best key below last[g]).
constexpr unsigned int GROUP_SENTINEL_HI = 0u;   // high word of the key of a row holding the exclusion sentinel

__global__ void __launch_bounds__(256)
exact_group_init_kernel(unsigned long long* __restrict__ last, unsigned long long* __restrict__ best, long long n) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    last[i] = ~0ull;
    best[i] = 0ull;
  }
}

__global__ void __launch_bounds__(256)
exact_group_round_kernel(const float* __restrict__ scores_ws, long long N, const int* __restrict__ groups, int n_groups,
                         const unsigned long long* __restrict__ last, unsigned long long* __restrict__ best) {
  const int s = blockIdx.y;
  const float* sc = scores_ws + (long long)s * N;
  const unsigned long long* ls = last + (long long)s * n_groups;
  unsigned long long* bs = best + (long long)s * n_groups;
  for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < N; r += (long long)gridDim.x * blockDim.x) {
    const int g = groups[r];
    if (g < 0 || g >= n_groups) continue;
    const unsigned long long k = make_key(sc[r], (uint32_t)r);
    if ((uint32_t)(k >> 32) == GROUP_SENTINEL_HI || k >= ls[g]) continue;
    if (k > *(volatile const unsigned long long*)(bs + g)) atomicMax(bs + g, k);   // the read skips most atomics
  }
}

__global__ void __launch_bounds__(256)
exact_group_advance_kernel(unsigned long long* __restrict__ last, unsigned long long* __restrict__ best, long long n) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    last[i] = best[i];   // 0 when the group has no row left: then it keeps all its rows
    best[i] = 0ull;
  }
}

__global__ void __launch_bounds__(256)
exact_group_drop_kernel(float* __restrict__ scores_ws, long long N, const int* __restrict__ groups, int n_groups,
                        const unsigned long long* __restrict__ last, unsigned int sentinel_bits) {
  const int s = blockIdx.y;
  float* sc = scores_ws + (long long)s * N;
  const unsigned long long* ls = last + (long long)s * n_groups;
  for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < N; r += (long long)gridDim.x * blockDim.x) {
    const int g = groups[r];
    if (g < 0 || g >= n_groups) continue;
    if (make_key(sc[r], (uint32_t)r) < ls[g]) sc[r] = __uint_as_float(sentinel_bits);
  }
}

size_t exact_group_ws_bytes(int n_groups) {
  return align_up((size_t)EX_QB * (size_t)n_groups * 16, 256);
}

int launch_exact_group_cap(float* scores_ws, long long N, int nslot, const GroupArgs& grp, void* group_ws,
                           unsigned int sentinel_bits, cudaStream_t st) {
  unsigned long long* last = reinterpret_cast<unsigned long long*>(group_ws);
  unsigned long long* best = last + (size_t)EX_QB * grp.n_groups;
  const long long ns = (long long)nslot * grp.n_groups;
  const int sms = num_sms();
  long long gi = (ns + 255) / 256;
  if (gi > (long long)sms * 8) gi = (long long)sms * 8;
  if (gi < 1) gi = 1;
  long long gs = (N + 255) / 256;
  if (gs > (long long)sms * 8) gs = (long long)sms * 8;
  exact_group_init_kernel<<<(unsigned)gi, 256, 0, st>>>(last, best, ns);
  TT_CHECK_LAUNCH();
  for (int round = 0; round < grp.max_per_group; ++round) {
    exact_group_round_kernel<<<dim3((unsigned)gs, nslot), 256, 0, st>>>(scores_ws, N, grp.groups, grp.n_groups, last, best);
    TT_CHECK_LAUNCH();
    exact_group_advance_kernel<<<(unsigned)gi, 256, 0, st>>>(last, best, ns);
    TT_CHECK_LAUNCH();
  }
  exact_group_drop_kernel<<<dim3((unsigned)gs, nslot), 256, 0, st>>>(scores_ws, N, grp.groups, grp.n_groups, last,
                                                                      sentinel_bits);
  TT_CHECK_LAUNCH();
  return TT_OK;
}

}  // namespace tt
