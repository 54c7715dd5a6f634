// Helpers shared by the top-K finalize (flat_select.cu) and the range finalize (flat_range.cu): sorting, exclusion
// lists, the prologue and candidate lookup, in-place compaction, radix select, fp32 rescoring, and the launch rule.
// Both kernels give a row the same fp32 score because both call rescore_rows.
#pragma once
#include <type_traits>
#include "tt_common.cuh"
#include "flat_internal.cuh"

namespace tt {

constexpr float PRUNE_MARGIN = 1.5f;       // in units of eps; typical |bf16 - fp32| is ~eps/25

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

__host__ __device__ __forceinline__ int next_pow2(int n) {
  int p = 1;
  while (p < n) p <<= 1;
  return p;
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

// ------------------------------------------------------------------------------------------
// Prologue of both finalize kernels (one CTA of NT threads per query q).  The scan left the query's candidates in
// per-slice segments cand[q, sl, 0 .. seg_cnt[q, sl]), each holding at most seg_cap of them.  Lays them end to end:
// s_off[sl] = where slice sl starts, s_off[nslices] = the number of candidates; *s_need = the largest count before
// clamping (a segment overflowed iff it exceeds seg_cap).  Stages the query in qs[0, D) and, under EXCL, its exclusion
// list in ex[0, EP) sorted descending, *s_any_ex = 1 if it names a row of this shard.  Ends with a barrier, so shared
// state the caller's thread 0 sets before the call is visible to every thread after it.
template <int NT, bool EXCL>
__device__ __forceinline__ void stage_query(int q, const unsigned int* __restrict__ seg_cnt, int nslices, int seg_cap,
                                            const float* __restrict__ qn, int D, const long long* __restrict__ excl, int E,
                                            long long id_offset, long long N, int* s_off, unsigned int* s_need, float* qs,
                                            unsigned int* ex, int EP, int* s_any_ex) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) { s_off[0] = 0; *s_need = 0u; *s_any_ex = 0; }
  __syncthreads();
  for (int sl = tid; sl < nslices; sl += NT) {
    const unsigned int c = seg_cnt[(size_t)q * nslices + sl];
    if (c) atomicMax(s_need, c);
    s_off[sl + 1] = (int)min(c, (unsigned int)seg_cap);
  }
  for (int d = tid; d < D; d += NT) qs[d] = qn[(long long)q * D + d];
  if constexpr (EXCL) {
    if (stage_exclusions(excl, E, q, id_offset, N, ex, EP)) *s_any_ex = 1;
  }
  __syncthreads();
  if constexpr (EXCL) {
    if (*s_any_ex) bitonic_sort_desc(ex, EP);   // ends with a barrier
  }
  if (warp == 0) {
    int carry = 0;
    for (int base = 0; base < nslices; base += 32) {
      const int sl = base + lane;
      int v = (sl < nslices) ? s_off[sl + 1] : 0;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, v, o); if (lane >= o) v += t; }
      const int incl = carry + v;
      if (sl < nslices) s_off[sl + 1] = incl;
      carry = __shfl_sync(0xffffffffu, incl, 31);
    }
  }
  __syncthreads();
}

// Candidate i of query q (bf16 score bits, row) in the list stage_query laid out: slice lo is the largest with
// s_off[lo] <= i, found by binary search.
__device__ __forceinline__ uint2 segment_entry(const uint2* __restrict__ cand, const int* s_off, int nslices, int seg_cap,
                                               int q, int i) {
  int lo = 0, hi = nslices;
  while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (s_off[mid] <= i) lo = mid; else hi = mid; }
  return cand[((size_t)q * nslices + lo) * seg_cap + (i - s_off[lo])];
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

// The kk-th largest (1 <= kk <= number of valid keys) of the ordered 32-bit keys key_at(i), i < n, found by a CTA of NT
// threads: four 8-bit passes, MSB first, over a 256-bin shared-memory histogram (s_hist), warp 0 scanning the bins
// from the top; s_digit / s_kk are shared scratch.  key_at may read shared or global memory.  An invalid entry returns
// key 0: it falls in the lowest bin, which the walk never reaches while kk is at most the number of valid keys and
// every valid key has a non-zero top byte (the key of every score with |score| < 2^127).
template <int NT, typename KeyAt>
__device__ __forceinline__ uint32_t radix_select_desc(int n, int kk, unsigned int* s_hist, int* s_digit, int* s_kk,
                                                      KeyAt key_at) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  uint32_t prefix = 0u, mask = 0u;
  for (int shift = 24; shift >= 0; shift -= 8) {
    if (tid < 256) s_hist[tid] = 0u;
    __syncthreads();
    for (int i = tid; i < n; i += NT) {
      const uint32_t u = key_at(i);
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
        *s_digit = d;
        *s_kk = kk - (int)above;
      }
    }
    __syncthreads();
    prefix |= (uint32_t)*s_digit << shift;
    mask |= 255u << shift;
    kk = *s_kk;
  }
  return prefix;
}

// The fp32 score of a row, as both finalize kernels compute it: fp32 scores of U catalog rows against the shared-memory
// query qs, warp-cooperative.  Per row: float4 pieces lane, lane + 32, ..., fmaf in x, y, z, w order, then warp_sum;
// scalar columns when !vec.  Rows with ok[u] false score 0.  Every lane returns the sums.
// WIDE (latency-bound CTAs of a small batch): with D <= 512, every 16-byte piece of the U rows is requested before the
// first one is used, one memory latency per call instead of one per 128 columns (the rows are scattered over the
// table: DRAM or, after the prefetch, L2).  The summation order is the same, so the score is too.
template <int U, bool WIDE = false>
__device__ __forceinline__ void rescore_rows(const float* __restrict__ qs, const float* __restrict__ Xn, int D, bool vec,
                                             const uint32_t (&row)[U], const bool (&ok)[U], float (&sc)[U], int lane) {
  float a[U];
#pragma unroll
  for (int u = 0; u < U; ++u) a[u] = 0.f;
  if (WIDE && vec && D <= 512) {
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
        x[u] = ok[u] ? __ldg(reinterpret_cast<const float4*>(Xn + (long long)row[u] * D) + cc) : make_float4(0.f, 0.f, 0.f, 0.f);
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
#pragma unroll
  for (int u = 0; u < U; ++u) sc[u] = warp_sum(a[u]);
}

// ------------------------------------------------------------------------------------------
// Launch rule of both finalize kernels, one CTA per query.  Large batches get one 256-thread CTA per query, several CTAs
// per SM.  Small batches (fewer queries than SMs) get 1024-thread CTAs: the latency-bound phases of the single query
// (gather or streaming, fp32 rescoring of scattered rows) get 4x the warps.  Measured on the top-K finalize
// (1M x 384): nq = 1 wide 20 us vs 31 us; nq = 128 wide 57 us vs 23 us.
constexpr int FIN_THREADS = 256;
constexpr int FIN_THREADS_WIDE = 1024;
constexpr int FIN_WIDE_MAX_NQ = 16;   // batches up to this many queries get the wide CTA

// Calls launch(nt, excl) for the finalize instance of a batch of nq queries, with the CTA size nt and whether the
// queries carry exclusion lists as std::integral_constant, so that they can be the kernel's template arguments.
template <typename Launch>
int launch_finalize_instance(int nq, bool with_excl, Launch&& launch) {
  using Wide = std::integral_constant<int, FIN_THREADS_WIDE>;
  using Narrow = std::integral_constant<int, FIN_THREADS>;
  if (nq <= FIN_WIDE_MAX_NQ) return with_excl ? launch(Wide{}, std::true_type{}) : launch(Wide{}, std::false_type{});
  return with_excl ? launch(Narrow{}, std::true_type{}) : launch(Narrow{}, std::false_type{});
}

// Dynamic shared memory of a finalize CTA: `keys` 8-byte keys, the query (D floats) and, for E > 0 exclusions, the
// staged list of next_pow2(E) rows.
inline size_t finalize_smem_bytes(int keys, int D, int E) {
  return (size_t)keys * 8 + (size_t)D * 4 + 16 + (E > 0 ? (size_t)next_pow2(E) * 4 : 0);
}

}  // namespace tt
