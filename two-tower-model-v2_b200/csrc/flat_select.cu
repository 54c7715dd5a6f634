// Selection side of the exact inner-product search:
//   finalize : fp32 rescoring of the candidate lists the tensor-core scan produced, exact sort by
//              (score desc, row asc), and the per-query exactness certificate
//   merge    : G sorted per-shard top-K lists -> one top-K (multi-GPU path)
//   exact    : always-exact fp32 path (CUDA-core scoring, 64-bit radix select), used for queries
//              the certificate rejects and as an on-device cross-check
// Semantics follow faiss.IndexFlatIP.search as used at src/inference/vector_db.py:160,197:
// fp32 inner products, k largest, sorted descending, int64 labels.
#include "tt_common.cuh"
#include "flat_internal.cuh"

namespace tt {

// In-place bitonic sort of P (power of two) keys in shared memory, descending.
template <typename T>
__device__ __forceinline__ void bitonic_sort_desc(T* key, int P) {
  for (int k = 2; k <= P; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = threadIdx.x; i < P; i += blockDim.x) {
        const int ixj = i ^ j;
        if (ixj > i) {
          const T a = key[i], b = key[ixj];
          const bool up = (i & k) == 0;          // "up" blocks are sorted descending
          if (up ? (a < b) : (a > b)) { key[i] = b; key[ixj] = a; }
        }
      }
      __syncthreads();
    }
  }
}

__device__ __forceinline__ int next_pow2(int n) {
  int p = 1;
  while (p < n) p <<= 1;
  return p;
}

// fp32 dot of a shared-memory query with a global row, warp-cooperative.
__device__ __forceinline__ float warp_dot(const float* __restrict__ qs, const float* __restrict__ row, int D,
                                          int lane, bool vec) {
  float a = 0.f;
  if (vec) {
    const float4* r4 = reinterpret_cast<const float4*>(row);
    const float4* q4 = reinterpret_cast<const float4*>(qs);
    for (int c = lane; c < (D >> 2); c += 32) {
      const float4 x = __ldg(r4 + c);
      const float4 y = q4[c];
      a = fmaf(x.x, y.x, a); a = fmaf(x.y, y.y, a); a = fmaf(x.z, y.z, a); a = fmaf(x.w, y.w, a);
    }
  } else {
    for (int d = lane; d < D; d += 32) a = fmaf(__ldg(row + d), qs[d], a);
  }
  return warp_sum(a);
}

// ------------------------------------------------------------------------------------------
// Per-query exclusion lists (tt_flat_search_excl & co.): excl i64 [nq, E], entry = local row + id_offset; entries
// below 0 are padding, ids outside [id_offset, id_offset + N) are ignored, duplicates are harmless.  A CTA stages
// its query's list in shared memory as local rows sorted descending; EXCL_NONE fills the unused slots (rows are
// < 2^31, so it never matches one).  Membership is then a binary search.
constexpr unsigned int EXCL_NONE = 0xffffffffu;

// ex[j] for j < P (P = next_pow2(E)); returns true if the query excludes a row of this shard.  No barrier.
__device__ __forceinline__ bool stage_exclusions(const long long* __restrict__ excl, int E, int q, long long id_offset,
                                                 long long N, unsigned int* ex, int P) {
  bool any = false;
  for (int j = threadIdx.x; j < P; j += blockDim.x) {
    unsigned int v = EXCL_NONE;
    if (j < E) {
      const long long id = excl[(long long)q * E + j];
      const long long r = id - id_offset;
      if (id >= 0 && r >= 0 && r < N) { v = (unsigned int)r; any = true; }
    }
    ex[j] = v;
  }
  return any;
}

__device__ __forceinline__ bool is_excluded(const unsigned int* ex, int P, unsigned int row) {
  int lo = 0, hi = P;   // first position whose entry is <= row (the list is descending)
  while (lo < hi) { const int mid = (lo + hi) >> 1; if (ex[mid] > row) lo = mid + 1; else hi = mid; }
  return lo < P && ex[lo] == row;
}

// In-place, order-keeping compaction of key[0, n) to the keys `keep(key)` accepts; returns the new count.  Chunks of
// NT keys move left only, so a chunk never overwrites keys not yet read.  n must be the same in every thread.
template <int NT, typename Keep>
__device__ __forceinline__ int compact_keys(unsigned long long* key, int n, int* s_wsum, Keep keep_fn) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int out = 0;
  for (int base = 0; base < n; base += NT) {
    const int i = base + (int)threadIdx.x;
    const unsigned long long kk64 = (i < n) ? key[i] : 0ull;
    const bool keep = (i < n) && keep_fn(kk64);
    const unsigned int bal = __ballot_sync(0xffffffffu, keep);
    if (lane == 0) s_wsum[warp] = __popc(bal);
    __syncthreads();                       // also orders every read of this chunk before the writes below
    int wbase = 0, tot = 0;
#pragma unroll
    for (int w = 0; w < NT / 32; ++w) { const int c = s_wsum[w]; if (w < warp) wbase += c; tot += c; }
    if (keep) key[out + wbase + __popc(bal & ((1u << lane) - 1u))] = kk64;
    out += tot;
    __syncthreads();
  }
  return out;
}

// ------------------------------------------------------------------------------------------
// finalize: one CTA per query.
//   1. gather the query's per-slice candidate segments (bf16 tensor-core score, row);
//   2. b_K = K-th largest bf16 score by a 4-pass radix select (no sort of the over-fetched list);
//   3. prune: only rows with bf16 score >= cutoff = b_K - PRUNE_MARGIN*eps are rescored (a row of the
//      fp32 top-K scores within eps of its bf16 score, so it sits well inside that band);
//   4. rescore the survivors in fp32 against the fp32 table; rank them by (score desc, row asc); emit K;
//   5. certificate (a posteriori, rigorous): every row that was NOT rescored has a bf16 score below
//      c = max(scan threshold, cutoff), hence an fp32 score below c + eps.  If the K-th best rescored
//      fp32 score f_K >= c + eps, no such row can enter the top-K: the result is exact.  Otherwise the
//      query is flagged and the host re-runs it through the exact path.
// EXCL (exclusion lists): right after the gather, candidates whose row the query excludes are dropped, so n, b_K,
// the cutoff and m all count allowed rows only, and the certificate reads "every ALLOWED row not rescored has a
// bf16 score < c".  Excluded rows are typically a query's best ones: the caller plans the scan for
// K_plan = min(K + E, N, TT_FLAT_MAX_K) so that the candidate budget covers them.
constexpr int FIN_THREADS = 256;          // large batches: one 256-thread CTA per query, several CTAs per SM
constexpr int FIN_THREADS_WIDE = 1024;    // small batches (fewer queries than SMs): the latency-bound phases of the
                                          // single query (gather, fp32 rescoring of ~200 scattered rows) get 4x the warps
constexpr float PRUNE_MARGIN = 1.5f;       // in units of eps; typical |bf16 - fp32| is ~eps/25
constexpr int RANK_BY_COUNT_MAX = 1024;    // survivors up to this many are ranked by counting, else bitonic sort

template <int FIN_THREADS, bool EXCL>
__global__ void __launch_bounds__(FIN_THREADS)
flat_finalize_kernel(const float* __restrict__ qn, const float* __restrict__ Xn, long long N, int D, int K,
                     long long id_offset, const float* __restrict__ thr, const float* __restrict__ eps,
                     const unsigned int* __restrict__ seg_cnt, const uint2* __restrict__ cand, int nslices,
                     int seg_cap, int cand_cap,
                     float* __restrict__ scores, long long* __restrict__ ids, int* __restrict__ flags,
                     int* __restrict__ n_uncertified, float* __restrict__ bound_out,
                     const long long* __restrict__ excl, int E) {
  pdl_trigger();
  pdl_wait();
  extern __shared__ __align__(16) unsigned char fsm[];
  unsigned long long* key = reinterpret_cast<unsigned long long*>(fsm);
  float* qs = reinterpret_cast<float*>(key + cand_cap);
  unsigned int* ex = reinterpret_cast<unsigned int*>(qs + D);   // EXCL: the query's sorted exclusion list
  __shared__ int s_off[FINALIZE_MAX_SLICES + 1];
  __shared__ unsigned int s_hist[256];
  __shared__ int s_wsum[FIN_THREADS / 32];
  __shared__ int s_over, s_bad, s_digit, s_kk, s_any_ex;
  __shared__ float s_fk;
  const int q = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int NWARPS = FIN_THREADS / 32;
  const int EP = EXCL ? next_pow2(E) : 0;

  // ---- 1. segment sizes -> offsets (parallel loads, warp-0 scan) --------------------------------
  if (tid == 0) { s_over = 0; s_bad = 0; s_fk = -INFINITY; s_off[0] = 0; s_any_ex = 0; }
  __syncthreads();
  for (int sl = tid; sl < nslices; sl += FIN_THREADS) {
    unsigned int c = seg_cnt[(size_t)q * nslices + sl];
    if (c > (unsigned int)seg_cap) { c = (unsigned int)seg_cap; s_over = 1; }
    s_off[sl + 1] = (int)c;
  }
  for (int d = tid; d < D; d += FIN_THREADS) qs[d] = qn[(long long)q * D + d];
  if constexpr (EXCL) {
    if (stage_exclusions(excl, E, q, id_offset, N, ex, EP)) s_any_ex = 1;
  }
  __syncthreads();
  if constexpr (EXCL) {
    if (s_any_ex) bitonic_sort_desc(ex, EP);   // ends with a barrier
  }
  if (warp == 0) {
    int carry = 0;
    for (int base = 0; base < nslices; base += 32) {
      const int sl = base + lane;
      int v = (sl < nslices) ? s_off[sl + 1] : 0;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, v, o); if (lane >= o) v += t; }
      int incl = carry + v;
      if (incl > cand_cap) { incl = cand_cap; s_over = 1; }
      if (sl < nslices) s_off[sl + 1] = incl;
      carry = __shfl_sync(0xffffffffu, incl, 31);
    }
  }
  __syncthreads();
  const bool overflow = s_over != 0;
  int n = s_off[nslices];
  const float my_eps = eps[q];
  const float t = thr[q];

  // ---- gather: one candidate per thread step, slice found by binary search over the offsets ------
  for (int i = tid; i < n; i += FIN_THREADS) {
    int lo = 0, hi = nslices;           // largest sl with s_off[sl] <= i
    while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (s_off[mid] <= i) lo = mid; else hi = mid; }
    const uint2 e = cand[((size_t)q * nslices + lo) * seg_cap + (i - s_off[lo])];
    key[i] = make_key(__uint_as_float(e.x), e.y);
  }
  __syncthreads();
  if constexpr (EXCL) {
    if (s_any_ex)   // from here on: allowed rows only
      n = compact_keys<FIN_THREADS>(key, n, s_wsum,
                                    [&](unsigned long long k) { return !is_excluded(ex, EP, key_row(k)); });
  }

  // ---- 2. b_K by radix select on the ordered score bits (8 bits per pass, MSB first) --------------
  float cutoff = -INFINITY;
  if (n > K) {   // n == K: everything is rescored anyway
    uint32_t prefix = 0u, mask = 0u;
    int kk = K;
    for (int shift = 24; shift >= 0; shift -= 8) {
      if (tid < 256) s_hist[tid] = 0u;
      __syncthreads();
      for (int i = tid; i < n; i += FIN_THREADS) {
        const uint32_t u = (uint32_t)(key[i] >> 32);
        if ((u & mask) == prefix) atomicAdd(&s_hist[(u >> shift) & 255u], 1u);
      }
      __syncthreads();
      if (warp == 0) {
        // lane l owns bins 255-8l .. 248-8l (descending)
        unsigned int loc[8];
        unsigned int sum = 0;
#pragma unroll
        for (int j = 0; j < 8; ++j) { loc[j] = s_hist[255 - 8 * lane - j]; sum += loc[j]; }
        unsigned int incl = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const unsigned int v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
        const unsigned int excl = incl - sum;
        if (excl < (unsigned int)kk && incl >= (unsigned int)kk) {   // exactly one lane
          unsigned int above = excl;
          int d = 255 - 8 * lane - 7;
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            if (above + loc[j] >= (unsigned int)kk) { d = 255 - 8 * lane - j; break; }
            above += loc[j];
          }
          s_digit = d;
          s_kk = kk - (int)above;
        }
      }
      __syncthreads();
      prefix |= (uint32_t)s_digit << shift;
      mask |= 255u << shift;
      kk = s_kk;
    }
    cutoff = ordered_to_float(prefix) - PRUNE_MARGIN * my_eps;
  }

  // ---- 3. prune: in-place compaction of the survivors (chunks of FIN_THREADS, left-moving) ---------
  int m = n;
  if (cutoff > -INFINITY)
    m = compact_keys<FIN_THREADS>(key, n, s_wsum, [&](unsigned long long k) { return key_score(k) >= cutoff; });

  // ---- 4. fp32 rescoring of the m survivors (in place) --------------------------------------------
  const bool vec = (D % 4 == 0) && ((reinterpret_cast<uintptr_t>(Xn) & 15) == 0);
  int bad = 0;   // self-check: a candidate's tensor-core score must match its fp32 rescoring within eps
  // candidates rescored concurrently per warp.  The wide CTA of a small batch is latency-bound: 2 rows with every
  // 16-byte piece in flight at once (18.6 vs 21.4 us at nq = 1); the 256-thread CTAs of large batches are
  // throughput-bound and keep 4 rows x one piece (the wide scheme there: 45 vs 35 us at nq = 128, 294 vs 261 us at 4096)
  constexpr bool WIDE = FIN_THREADS > 512;
  constexpr int U = WIDE ? 2 : 4;
  for (int i0 = warp * U; i0 < m; i0 += NWARPS * U) {
    uint32_t row[U];
    float bsc[U];
    bool ok[U];
    float a[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int i = i0 + u;
      const unsigned long long kk64 = (i < m) ? key[i] : 0ull;
      row[u] = key_row(kk64);
      bsc[u] = key_score(kk64);
      ok[u] = (i < m) && ((long long)row[u] < N);   // row >= N cannot happen unless the scan is broken
      a[u] = 0.f;
    }
    if (WIDE && vec && D <= 512) {
      // every 16-byte piece of the U rows is requested before the first one is used: one memory latency per round
      // instead of one per 128 columns (the rows are scattered over the table: DRAM or, after the prefetch, L2)
      constexpr int NVX = 4;
      const float4* q4 = reinterpret_cast<const float4*>(qs);
      const int nvec = D >> 2;
      float4 x[U][NVX];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const float4* rp = reinterpret_cast<const float4*>(Xn + (long long)row[u] * D);
#pragma unroll
        for (int v = 0; v < NVX; ++v) {
          const int cc = v * 32 + lane;
          x[u][v] = (ok[u] && cc < nvec) ? __ldg(rp + cc) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
      }
#pragma unroll
      for (int v = 0; v < NVX; ++v) {
        const int cc = v * 32 + lane;
        const float4 y = (cc < nvec) ? q4[cc] : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int u = 0; u < U; ++u) {
          a[u] = fmaf(x[u][v].x, y.x, a[u]); a[u] = fmaf(x[u][v].y, y.y, a[u]);
          a[u] = fmaf(x[u][v].z, y.z, a[u]); a[u] = fmaf(x[u][v].w, y.w, a[u]);
        }
      }
    } else if (vec) {
      const float4* q4 = reinterpret_cast<const float4*>(qs);
      for (int cc = lane; cc < (D >> 2); cc += 32) {
        const float4 y = q4[cc];
        float4 x[U];
#pragma unroll
        for (int u = 0; u < U; ++u)
          x[u] = ok[u] ? __ldg(reinterpret_cast<const float4*>(Xn + (long long)row[u] * D) + cc)
                       : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int u = 0; u < U; ++u) {
          a[u] = fmaf(x[u].x, y.x, a[u]); a[u] = fmaf(x[u].y, y.y, a[u]);
          a[u] = fmaf(x[u].z, y.z, a[u]); a[u] = fmaf(x[u].w, y.w, a[u]);
        }
      }
    } else {
      for (int d = lane; d < D; d += 32) {
        const float y = qs[d];
#pragma unroll
        for (int u = 0; u < U; ++u)
          if (ok[u]) a[u] = fmaf(__ldg(Xn + (long long)row[u] * D + d), y, a[u]);
      }
    }
    __syncwarp();
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const float sc = warp_sum(a[u]);
      const int i = i0 + u;
      if (lane == 0 && i < m) {
        if (ok[u]) {
          key[i] = make_key(sc, row[u]);
          if (!(fabsf(bsc[u] - sc) <= my_eps)) bad = 1;
        } else {
          key[i] = 0ull;
          bad = 1;
        }
      }
    }
  }
  if (bad) s_bad = 1;
  __syncthreads();

  // ---- 5. order the survivors by (score desc, row asc) and emit K ---------------------------------
  if (m <= RANK_BY_COUNT_MAX) {
    // keys are distinct (the row is part of the key): rank = number of larger keys
    for (int i = tid; i < m; i += FIN_THREADS) {
      const unsigned long long ki = key[i];
      int rank = 0;
      for (int j = 0; j < m; ++j) rank += (key[j] > ki) ? 1 : 0;
      if (rank < K) {
        scores[(long long)q * K + rank] = key_score(ki);
        ids[(long long)q * K + rank] = (ki == 0ull) ? -1 : (long long)key_row(ki) + id_offset;
        if (rank == K - 1) s_fk = key_score(ki);
      }
    }
    for (int i = m + tid; i < K; i += FIN_THREADS) {
      scores[(long long)q * K + i] = -INFINITY;
      ids[(long long)q * K + i] = -1;
    }
  } else {
    const int P2 = next_pow2(m);
    for (int i = m + tid; i < P2; i += FIN_THREADS) key[i] = 0ull;
    __syncthreads();
    bitonic_sort_desc(key, P2);
    for (int i = tid; i < K; i += FIN_THREADS) {
      if (i < m) {
        scores[(long long)q * K + i] = key_score(key[i]);
        ids[(long long)q * K + i] = (long long)key_row(key[i]) + id_offset;
        if (i == K - 1) s_fk = key_score(key[i]);
      } else {
        scores[(long long)q * K + i] = -INFINITY;
        ids[(long long)q * K + i] = -1;
      }
    }
  }
  __syncthreads();
  if (tid == 0) {
    // flags: 1 = certified; otherwise -(reason bits): 1 list overflow, 2 fewer than K candidates,
    // 4 tensor-core/fp32 score mismatch beyond eps, 8 f_K does not clear the bound of the rows not rescored.
    const float c = fmaxf(t, cutoff);                 // every row not rescored has a bf16 score < c
    const bool unbounded = (c == -INFINITY);          // every row of the shard was rescored
    int why = 0;
    if (overflow) why |= 1;
    if (m < K) why |= 2;
    if (s_bad) why |= 4;
    if (m >= K && !unbounded && !(s_fk >= c + my_eps)) why |= 8;
    const bool ok = why == 0;
    flags[q] = ok ? 1 : -why;
    if (!ok) atomicAdd(n_uncertified, 1);
    // shard mode: fp32 upper bound of every row of this shard that was not rescored (global certificate)
    if (bound_out) bound_out[q] = unbounded ? -INFINITY : c + my_eps;
  }
}

template <int NT, bool EXCL>
static int launch_finalize_t(const ScanPlan& pl, const float* qn, const float* Xn, long long N, int D, int nq, int K,
                             long long id_offset, const float* thr, const float* eps, const unsigned int* seg_cnt,
                             const void* cand, float* scores, long long* ids, int* flags, int* n_uncertified,
                             float* bound_out, const long long* excl, int E, size_t smem, cudaStream_t st) {
  TT_CHECK_CUDA(cudaFuncSetAttribute(flat_finalize_kernel<NT, EXCL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  TT_CHECK_CUDA(launch_pdl(flat_finalize_kernel<NT, EXCL>, dim3(nq), dim3(NT), smem, st, qn, Xn, N, D, K, id_offset, thr, eps,
                           seg_cnt, reinterpret_cast<const uint2*>(cand), pl.main_slices, pl.seg_cap, pl.cand_cap, scores,
                           ids, flags, n_uncertified, bound_out, excl, E));
  return TT_OK;
}

int launch_finalize(const ScanPlan& pl, const float* qn, const float* Xn, long long N, int D, int nq, int K,
                    long long id_offset, const float* thr, const float* eps, const unsigned int* seg_cnt,
                    const void* cand, float* scores, long long* ids, int* flags, int* n_uncertified,
                    float* bound_out, cudaStream_t st, const long long* excl, int E) {
  TT_CHECK_ARG(pl.main_slices <= FINALIZE_MAX_SLICES, "too many catalog slices");
  const bool with_excl = excl != nullptr && E > 0;
  size_t smem = (size_t)pl.cand_cap * 8 + (size_t)D * 4 + 16;
  if (with_excl) {
    int P = 1;
    while (P < E) P <<= 1;
    smem += (size_t)P * 4;
  }
  count_launch();
  // wide CTAs for small batches, measured (1M x 384): nq = 1 wide 20 us vs 31 us; nq = 128 wide 57 us vs 23 us
  if (nq <= 16)
    return with_excl ? launch_finalize_t<FIN_THREADS_WIDE, true>(pl, qn, Xn, N, D, nq, K, id_offset, thr, eps, seg_cnt, cand,
                                                                scores, ids, flags, n_uncertified, bound_out, excl, E, smem, st)
                     : launch_finalize_t<FIN_THREADS_WIDE, false>(pl, qn, Xn, N, D, nq, K, id_offset, thr, eps, seg_cnt, cand,
                                                                 scores, ids, flags, n_uncertified, bound_out, nullptr, 0, smem, st);
  return with_excl ? launch_finalize_t<FIN_THREADS, true>(pl, qn, Xn, N, D, nq, K, id_offset, thr, eps, seg_cnt, cand, scores,
                                                         ids, flags, n_uncertified, bound_out, excl, E, smem, st)
                   : launch_finalize_t<FIN_THREADS, false>(pl, qn, Xn, N, D, nq, K, id_offset, thr, eps, seg_cnt, cand, scores,
                                                          ids, flags, n_uncertified, bound_out, nullptr, 0, smem, st);
}

// ------------------------------------------------------------------------------------------
// merge: one CTA per query, G*K <= 16384 keys
__global__ void __launch_bounds__(128)
topk_merge_kernel(const float* __restrict__ sg, const long long* __restrict__ ig, int G, int nq, int K,
                  float* __restrict__ scores, long long* __restrict__ ids) {
  extern __shared__ __align__(16) unsigned char msm[];
  unsigned long long* key = reinterpret_cast<unsigned long long*>(msm);
  const int q = blockIdx.x;
  const int n = G * K;
  const int P = next_pow2(n);
  for (int i = threadIdx.x; i < P; i += blockDim.x) {
    unsigned long long kk = 0ull;
    if (i < n) {
      const int g = i / K, j = i % K;
      const long long id = ig[((long long)g * nq + q) * K + j];
      const float s = sg[((long long)g * nq + q) * K + j];
      if (id >= 0) kk = make_key(s, (uint32_t)id);
    }
    key[i] = kk;
  }
  __syncthreads();
  bitonic_sort_desc(key, P);
  for (int i = threadIdx.x; i < K; i += blockDim.x) {
    const unsigned long long kk = key[i];
    scores[(long long)q * K + i] = (kk == 0ull) ? -INFINITY : key_score(kk);
    ids[(long long)q * K + i] = (kk == 0ull) ? -1 : (long long)key_row(kk);
  }
}

// ------------------------------------------------------------------------------------------
// shard merge with the global exactness certificate: one CTA per query.
// Every rank contributed a record {scores f32[nq,K] | ids i64[nq,K] | bound f32[nq] | flags i32[nq]} (the
// layout ONE all-gather of the per-rank byte buffers produces).  The G lists are sorted (score desc, id
// asc) and padded with (-inf, -1); an element's position in the merged order is its own index plus, for
// every other list, the number of larger keys found by binary search - no sort.
// Certificate: on shard g every row that was not rescored in fp32 scores strictly below bound_g[q]; the
// merged top-K is exact iff its K-th score f_K >= max_g bound_g[q] (and no shard reported a candidate-list
// overflow or a tensor-core/fp32 self-check failure).
__global__ void __launch_bounds__(128)
shard_merge_kernel(const unsigned char* __restrict__ gathered, size_t rank_stride, size_t off_scores, size_t off_ids,
                   size_t off_bound, size_t off_flags, int G, int nq, int K, float* __restrict__ scores,
                   long long* __restrict__ ids, int* __restrict__ flags, int* __restrict__ n_uncertified) {
  extern __shared__ __align__(16) unsigned char msm[];
  unsigned long long* key = reinterpret_cast<unsigned long long*>(msm);   // [G][K]
  __shared__ int s_valid[64];
  __shared__ int s_flag[64];
  __shared__ float s_bound[64];
  __shared__ float s_fk;
  const int q = blockIdx.x;
  const int n = G * K;
  if (threadIdx.x == 0) s_fk = -INFINITY;
  if (threadIdx.x < G) {
    const unsigned char* rec = gathered + (size_t)threadIdx.x * rank_stride;
    s_flag[threadIdx.x] = reinterpret_cast<const int*>(rec + off_flags)[q];
    s_bound[threadIdx.x] = reinterpret_cast<const float*>(rec + off_bound)[q];
    s_valid[threadIdx.x] = 0;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const int g = i / K, j = i % K;
    const unsigned char* rec = gathered + (size_t)g * rank_stride;
    const long long* idp = reinterpret_cast<const long long*>(rec + off_ids) + (long long)q * K;
    const long long id = idp[j];
    const float sc = reinterpret_cast<const float*>(rec + off_scores)[(long long)q * K + j];
    key[i] = (id >= 0) ? make_key(sc, (uint32_t)id) : 0ull;
    // lists are padded at the tail: the last valid position marks the list's length (no atomics)
    if (id >= 0 && (j == K - 1 || idp[j + 1] < 0)) s_valid[g] = j + 1;
  }
  __syncthreads();
  int total = 0;
  for (int g = 0; g < G; ++g) total += s_valid[g];
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const unsigned long long ki = key[i];
    if (ki == 0ull) continue;
    const int g = i / K;
    int rank = i % K;
    // binary search every other list for the number of larger keys; stop once the element is out of the top K
    for (int h = 0; h < G && rank < K; ++h) {
      if (h == g) continue;
      const unsigned long long* lst = key + h * K;
      int lo = 0, hi = s_valid[h];
      while (lo < hi) { const int mid = (lo + hi) >> 1; if (lst[mid] > ki) lo = mid + 1; else hi = mid; }
      rank += lo;
    }
    if (rank < K) {
      scores[(long long)q * K + rank] = key_score(ki);
      ids[(long long)q * K + rank] = (long long)key_row(ki);
      if (rank == K - 1) s_fk = key_score(ki);
    }
  }
  for (int i = total + threadIdx.x; i < K; i += blockDim.x) {
    scores[(long long)q * K + i] = -INFINITY;
    ids[(long long)q * K + i] = -1;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    int why = 0;
    float bmax = -INFINITY;
    for (int g = 0; g < G; ++g) {
      const int f = s_flag[g];
      if (f <= 0) why |= (-f) & (1 | 4);     // local "fewer than K" / local f_K checks are superseded by the global one
      bmax = fmaxf(bmax, s_bound[g]);
    }
    if (total < K) why |= 2;
    if (total >= K && !(bmax == -INFINITY) && !(s_fk >= bmax)) why |= 8;
    flags[q] = why == 0 ? 1 : -why;
    if (why) atomicAdd(n_uncertified, 1);
  }
}

// ------------------------------------------------------------------------------------------
// exact path
constexpr int EX_QB = 8;   // queries scored per pass over the fp32 table

struct SelState {
  unsigned long long prefix;   // bits of the K-th key decided so far
  int kremain;                 // rank still to resolve inside the current prefix bucket
  unsigned int count;          // collect cursor
};

// scores_ws[slot, r] = <q_slot / (||q_slot|| + 1e-8), Xn[r]>
__global__ void __launch_bounds__(256)
exact_scores_kernel(const float* __restrict__ q, const int* __restrict__ qsel, int slot0, int nslot,
                    const float* __restrict__ Xn, long long N, int D, float* __restrict__ scores_ws) {
  extern __shared__ __align__(16) float qs[];   // [nslot][D]
  __shared__ float inv[EX_QB];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  for (int s = warp; s < nslot; s += nwarps) {
    const int qi = qsel ? qsel[slot0 + s] : (slot0 + s);
    float ss = 0.f;
    for (int d = lane; d < D; d += 32) { const float v = q[(long long)qi * D + d]; ss += v * v; }
    ss = warp_sum(ss);
    if (lane == 0) inv[s] = sqrtf(ss) + 1e-8f;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < nslot * D; i += blockDim.x) {
    const int s = i / D, d = i % D;
    const int qi = qsel ? qsel[slot0 + s] : (slot0 + s);
    qs[i] = q[(long long)qi * D + d] / inv[s];
  }
  __syncthreads();
  const bool vec = (D % 4 == 0) && ((reinterpret_cast<uintptr_t>(Xn) & 15) == 0);
  const long long gw = (long long)blockIdx.x * nwarps + warp;
  const long long tw = (long long)gridDim.x * nwarps;
  for (long long r = gw; r < N; r += tw) {
    float acc[EX_QB];
#pragma unroll
    for (int s = 0; s < EX_QB; ++s) acc[s] = 0.f;
    const float* row = Xn + r * D;
    if (vec) {
      const float4* r4 = reinterpret_cast<const float4*>(row);
      for (int c = lane; c < (D >> 2); c += 32) {
        const float4 x = ldg_stream(r4 + c);
#pragma unroll
        for (int s = 0; s < EX_QB; ++s) {
          if (s < nslot) {
            const float4 y = reinterpret_cast<const float4*>(qs + s * D)[c];
            acc[s] = fmaf(x.x, y.x, acc[s]); acc[s] = fmaf(x.y, y.y, acc[s]);
            acc[s] = fmaf(x.z, y.z, acc[s]); acc[s] = fmaf(x.w, y.w, acc[s]);
          }
        }
      }
    } else {
      for (int d = lane; d < D; d += 32) {
        const float x = __ldg(row + d);
#pragma unroll
        for (int s = 0; s < EX_QB; ++s) if (s < nslot) acc[s] = fmaf(x, qs[s * D + d], acc[s]);
      }
    }
#pragma unroll
    for (int s = 0; s < EX_QB; ++s) {
      if (s < nslot) {
        const float v = warp_sum(acc[s]);
        if (lane == 0) scores_ws[(long long)s * N + r] = v;
      }
    }
  }
}

// Exclusion lists on the exact path: the score of every excluded row becomes EXCL_SCORE_BITS, whose ordered key has
// zero high bits, below the key of any real score (-inf included).  O(E) per query; select, collect and sort then
// see these rows as the smallest keys and the sort writes them as (-inf, -1).  The list row is the QUERY row qsel[i].
constexpr unsigned int EXCL_SCORE_BITS = 0xffffffffu;   // a negative NaN: float_to_ordered() maps it to 0

__global__ void __launch_bounds__(256)
exact_exclude_kernel(const long long* __restrict__ excl, int E, const int* __restrict__ qsel, int slot0,
                     long long id_offset, long long N, float* __restrict__ scores_ws) {
  const int s = blockIdx.x;
  const int qi = qsel ? qsel[slot0 + s] : (slot0 + s);
  for (int j = threadIdx.x; j < E; j += blockDim.x) {
    const long long id = excl[(long long)qi * E + j];
    const long long r = id - id_offset;
    if (id >= 0 && r >= 0 && r < N) scores_ws[(long long)s * N + r] = __uint_as_float(EXCL_SCORE_BITS);
  }
}

__global__ void exact_init_kernel(SelState* st, unsigned int* hist, int nslot, int K) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < nslot) { st[i].prefix = 0ull; st[i].kremain = K; st[i].count = 0u; }
  if (i < nslot * 256) hist[i] = 0u;
}

// histogram of the digit at `shift` over keys whose higher bits equal the prefix
__global__ void __launch_bounds__(256)
exact_hist_kernel(const float* __restrict__ scores_ws, long long N, const SelState* __restrict__ st,
                  unsigned int* __restrict__ hist, int shift) {
  __shared__ unsigned int h[256];
  const int s = blockIdx.y;
  h[threadIdx.x] = 0u;
  __syncthreads();
  const unsigned long long prefix = st[s].prefix;
  const float* sc = scores_ws + (long long)s * N;
  for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < N; r += (long long)gridDim.x * blockDim.x) {
    const unsigned long long k = make_key(sc[r], (uint32_t)r);
    const bool match = (shift == 56) ? true : ((k >> (shift + 8)) == (prefix >> (shift + 8)));
    if (match) atomicAdd(&h[(unsigned int)(k >> shift) & 255u], 1u);
  }
  __syncthreads();
  if (h[threadIdx.x]) atomicAdd(&hist[s * 256 + threadIdx.x], h[threadIdx.x]);
}

// choose the digit containing the kremain-th largest key, then clear the histogram
__global__ void exact_pick_kernel(SelState* st, unsigned int* hist, int shift) {
  const int s = blockIdx.x;
  if (threadIdx.x == 0) {
    int krem = st[s].kremain;
    int d = 255;
    unsigned int above = 0;
    for (; d > 0; --d) {
      const unsigned int c = hist[s * 256 + d];
      if (above + c >= (unsigned int)krem) break;
      above += c;
    }
    st[s].prefix |= ((unsigned long long)d) << shift;
    st[s].kremain = krem - (int)above;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 256; i += blockDim.x) hist[s * 256 + i] = 0u;
}

__global__ void __launch_bounds__(256)
exact_collect_kernel(const float* __restrict__ scores_ws, long long N, SelState* st, unsigned long long* keys_out, int K) {
  const int s = blockIdx.y;
  const unsigned long long kth = st[s].prefix;
  const float* sc = scores_ws + (long long)s * N;
  for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < N; r += (long long)gridDim.x * blockDim.x) {
    const unsigned long long k = make_key(sc[r], (uint32_t)r);
    if (k >= kth) {
      const unsigned int pos = atomicAdd(&st[s].count, 1u);
      if (pos < (unsigned int)K) keys_out[(long long)s * K + pos] = k;
    }
  }
}

__global__ void __launch_bounds__(256)
exact_sort_kernel(const unsigned long long* __restrict__ keys_in, const int* __restrict__ qsel, int slot0, int K,
                  long long id_offset, float* __restrict__ scores, long long* __restrict__ ids, bool excl) {
  extern __shared__ __align__(16) unsigned char ssm[];
  unsigned long long* key = reinterpret_cast<unsigned long long*>(ssm);
  const int s = blockIdx.x;
  const int qi = qsel ? qsel[slot0 + s] : (slot0 + s);
  const int P = next_pow2(K);
  for (int i = threadIdx.x; i < P; i += blockDim.x) key[i] = (i < K) ? keys_in[(long long)s * K + i] : 0ull;
  __syncthreads();
  bitonic_sort_desc(key, P);
  for (int i = threadIdx.x; i < K; i += blockDim.x) {
    if (excl && (key[i] >> 32) == 0ull) {   // an excluded row (fewer than K allowed rows): the tail is padding
      scores[(long long)qi * K + i] = -INFINITY;
      ids[(long long)qi * K + i] = -1;
    } else {
      scores[(long long)qi * K + i] = key_score(key[i]);
      ids[(long long)qi * K + i] = (long long)key_row(key[i]) + id_offset;
    }
  }
}

}  // namespace tt

using namespace tt;

extern "C" __attribute__((visibility("default"))) int tt_topk_merge(const float* scores_g, const int64_t* ids_g, int G, int nq, int K,
                             float* scores, int64_t* ids, void* stream) {
  TT_CHECK_ARG(scores_g && ids_g && scores && ids, "null pointer");
  TT_CHECK_ARG(G >= 1 && nq >= 0 && K >= 1, "need G >= 1, nq >= 0, K >= 1");
  TT_CHECK_ARG((long long)G * K <= FINALIZE_MAX_CAND, "G*K exceeds 16384");
  if (nq == 0) return TT_OK;
  int P = 1;
  while (P < G * K) P <<= 1;
  const size_t smem = (size_t)P * 8;
  TT_CHECK_CUDA(cudaFuncSetAttribute(topk_merge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  topk_merge_kernel<<<nq, 128, smem, (cudaStream_t)stream>>>(scores_g, reinterpret_cast<const long long*>(ids_g), G,
                                                            nq, K, scores, reinterpret_cast<long long*>(ids));
  TT_CHECK_LAUNCH();
  return TT_OK;
}

extern "C" __attribute__((visibility("default"))) int tt_shard_merge(const void* gathered, size_t rank_stride, size_t off_scores, size_t off_ids,
                              size_t off_bound, size_t off_flags, int G, int nq, int K, float* scores, int64_t* ids,
                              int32_t* flags, int32_t* n_uncertified, void* stream) {
  TT_CHECK_ARG(gathered && scores && ids && flags && n_uncertified, "null pointer");
  TT_CHECK_ARG(G >= 1 && G <= 64 && nq >= 0 && K >= 1, "need 1 <= G <= 64, nq >= 0, K >= 1");
  TT_CHECK_ARG((long long)G * K <= FINALIZE_MAX_CAND, "G*K exceeds 16384");
  TT_CHECK_ARG(off_scores % 4 == 0 && off_ids % 8 == 0 && off_bound % 4 == 0 && off_flags % 4 == 0 && rank_stride % 8 == 0,
               "misaligned record layout");
  cudaStream_t st = (cudaStream_t)stream;
  TT_CHECK_CUDA(cudaMemsetAsync(n_uncertified, 0, sizeof(int32_t), st));
  if (nq == 0) return TT_OK;
  const size_t smem = (size_t)G * K * 8;
  TT_CHECK_CUDA(cudaFuncSetAttribute(shard_merge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  shard_merge_kernel<<<nq, 128, smem, st>>>(reinterpret_cast<const unsigned char*>(gathered), rank_stride, off_scores,
                                            off_ids, off_bound, off_flags, G, nq, K, scores,
                                            reinterpret_cast<long long*>(ids), flags, n_uncertified);
  TT_CHECK_LAUNCH();
  return TT_OK;
}

static size_t exact_ws_layout(int64_t N, int K, size_t* off_state, size_t* off_hist, size_t* off_keys) {
  size_t o = 0;
  o += align_up((size_t)EX_QB * (size_t)N * sizeof(float), 256);
  *off_state = o; o += align_up(EX_QB * sizeof(SelState), 256);
  *off_hist = o;  o += align_up(EX_QB * 256 * sizeof(unsigned int), 256);
  *off_keys = o;  o += align_up((size_t)EX_QB * K * sizeof(unsigned long long), 256);
  return o;
}

extern "C" __attribute__((visibility("default"))) size_t tt_flat_search_exact_workspace_bytes(int64_t N, int D, int nsel, int K) {
  (void)D; (void)nsel;
  size_t a, b, c;
  return exact_ws_layout(N, K, &a, &b, &c);
}

static int flat_search_exact_impl(const float* q, int nq, const int32_t* qsel, int nsel, const float* Xn, int64_t N,
                                  int D, int K, int64_t id_offset, float* scores, int64_t* ids, const int64_t* excl,
                                  int E, void* workspace, size_t workspace_bytes, void* stream) {
  TT_CHECK_ARG(q && Xn && scores && ids && workspace, "null pointer");
  TT_CHECK_ARG(N >= 1 && N < (1LL << 32) && D >= 1, "need 1 <= N < 2^32, D >= 1");
  TT_CHECK_ARG(K >= 1 && K <= N && K <= TT_FLAT_MAX_K, "need 1 <= K <= min(N, TT_FLAT_MAX_K)");
  TT_CHECK_ARG(nq >= 0 && nsel >= 0 && (qsel != nullptr || nsel == nq), "qsel == NULL requires nsel == nq");
  TT_CHECK_ARG((size_t)EX_QB * D * sizeof(float) <= 160 * 1024, "D too large");
  if (nsel == 0) return TT_OK;
  size_t o_state, o_hist, o_keys;
  const size_t need = exact_ws_layout(N, K, &o_state, &o_hist, &o_keys);
  if (workspace_bytes < need) { set_error("tt_flat_search_exact: workspace too small"); return TT_ERR_WORKSPACE; }
  cudaStream_t st = (cudaStream_t)stream;
  unsigned char* ws = reinterpret_cast<unsigned char*>(workspace);
  float* scores_ws = reinterpret_cast<float*>(ws);
  SelState* state = reinterpret_cast<SelState*>(ws + o_state);
  unsigned int* hist = reinterpret_cast<unsigned int*>(ws + o_hist);
  unsigned long long* keys = reinterpret_cast<unsigned long long*>(ws + o_keys);

  const int sms = num_sms();
  const size_t smem_q = (size_t)EX_QB * D * sizeof(float);
  TT_CHECK_CUDA(cudaFuncSetAttribute(exact_scores_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_q));
  int P = 1;
  while (P < K) P <<= 1;
  long long gs = (N + 255) / 256;
  if (gs > (long long)sms * 8) gs = (long long)sms * 8;
  for (int slot0 = 0; slot0 < nsel; slot0 += EX_QB) {
    const int nslot = (nsel - slot0 < EX_QB) ? (nsel - slot0) : EX_QB;
    long long gw = (N + 7) / 8;
    if (gw > (long long)sms * 4) gw = (long long)sms * 4;
    exact_scores_kernel<<<(unsigned)gw, 256, smem_q, st>>>(q, qsel, slot0, nslot, Xn, N, D, scores_ws);
    TT_CHECK_LAUNCH();
    if (E > 0) {
      exact_exclude_kernel<<<nslot, 256, 0, st>>>(reinterpret_cast<const long long*>(excl), E, qsel, slot0, id_offset, N,
                                                  scores_ws);
      TT_CHECK_LAUNCH();
    }
    exact_init_kernel<<<(nslot * 256 + 255) / 256, 256, 0, st>>>(state, hist, nslot, K);
    TT_CHECK_LAUNCH();
    for (int shift = 56; shift >= 0; shift -= 8) {
      exact_hist_kernel<<<dim3((unsigned)gs, nslot), 256, 0, st>>>(scores_ws, N, state, hist, shift);
      TT_CHECK_LAUNCH();
      exact_pick_kernel<<<nslot, 256, 0, st>>>(state, hist, shift);
      TT_CHECK_LAUNCH();
    }
    exact_collect_kernel<<<dim3((unsigned)gs, nslot), 256, 0, st>>>(scores_ws, N, state, keys, K);
    TT_CHECK_LAUNCH();
    exact_sort_kernel<<<nslot, 256, (size_t)P * 8, st>>>(keys, qsel, slot0, K, id_offset, scores,
                                                         reinterpret_cast<long long*>(ids), E > 0);
    TT_CHECK_LAUNCH();
  }
  return TT_OK;
}

extern "C" __attribute__((visibility("default"))) int tt_flat_search_exact(const float* q, int nq, const int32_t* qsel, int nsel,
                                    const float* Xn, int64_t N, int D, int K, int64_t id_offset,
                                    float* scores, int64_t* ids, void* workspace, size_t workspace_bytes,
                                    void* stream) {
  return flat_search_exact_impl(q, nq, qsel, nsel, Xn, N, D, K, id_offset, scores, ids, nullptr, 0, workspace,
                                workspace_bytes, stream);
}

extern "C" __attribute__((visibility("default"))) int tt_flat_search_exact_excl(const float* q, int nq, const int32_t* qsel, int nsel,
                                         const float* Xn, int64_t N, int D, int K, int64_t id_offset,
                                         float* scores, int64_t* ids, const int64_t* excl, int E,
                                         void* workspace, size_t workspace_bytes, void* stream) {
  TT_CHECK_ARG(E >= 0 && E <= TT_FLAT_MAX_EXCLUDE, "need 0 <= E <= TT_FLAT_MAX_EXCLUDE (1024) exclusions per query");
  TT_CHECK_ARG(excl != nullptr || E == 0, "null exclusion list with E > 0");
  return flat_search_exact_impl(q, nq, qsel, nsel, Xn, N, D, K, id_offset, scores, ids, excl, E, workspace,
                                workspace_bytes, stream);
}
