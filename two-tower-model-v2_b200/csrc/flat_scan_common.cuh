// Device helpers shared by the scan kernels (flat_scan.cu: A operand in shared memory; flat_scan_ts.cu: A operand
// in tensor memory).
#pragma once
#include <cuda.h>
#include <math.h>
#include <type_traits>
#include "tt_common.cuh"
#include "sm100_ptx.cuh"
#include "flat_internal.cuh"

namespace tt {

using namespace ptx;

constexpr int SCAN_THREADS = 256;
constexpr int BLOCK_N = 256;                    // catalog rows per tile
constexpr int BLOCK_K = 64;                     // bf16 per K-block = one 128-byte swizzle row
constexpr int UMMA_K = 16;
constexpr int MAX_STAGES = 8;
constexpr int TMEM_COLS = 512;                  // 2 accumulator buffers x 256 fp32 columns
constexpr int CHUNKS = BLOCK_N / 32;
constexpr int BAR_BYTES = 256;                  // mbarriers + TMEM base pointer
constexpr int SCRATCH_BYTES = 4 * 256;          // one 64-value row per epilogue warp (candidate extraction)

struct ScanParams {
  long long N;            // catalog rows
  int nq;                 // valid queries
  int num_kb;             // K-blocks per row (Dp / 64)
  int num_kb_res;         // leading K-blocks of the query block that stay resident in shared memory; the
                          // rest (D > 640 in pair mode) is streamed with the catalog, once per tile, from L2
  int stage_bytes;        // ring stride: the catalog K-block, plus room for a query K-block when streaming
  int num_stages;         // ring depth
  int nqu;                // query units (query blocks, or query-block pairs)
  int nslices;            // catalog slices
  int num_slots;          // tiles to visit in total (main: all tiles; sample: sampled tiles)
  int tile_stride;        // tile index = slot * tile_stride
  // MAIN
  const float* thr;       // [nq]
  unsigned int* seg_cnt;  // [nq, nslices]
  uint2* cand;            // [nq, nslices, seg_cap]  (score bits, row)
  int seg_cap;
  // MAIN with the threshold selection folded into the prologue (a batch of one query): thr[q] = the sel_rank-th
  // largest of the query's sel_n sampled maxima, computed by the epilogue warps while the first tile streams in
  const float* sel_sample;
  float* thr_out;         // [nq] written by CTA 0 for the finalize kernel
  int sel_n, sel_ld, sel_rank, sel_query_major;
  // SAMPLE
  float* sample_out;      // chunk mode: [nq_pad, num_slots, 8] maxima of the 32-row chunks of every sampled tile
                          // tile mode : [num_slots, sample_ld] maximum of every sampled tile (query fastest)
  int sample_tile_max;    // 1 = tile mode
  int sample_ld;          // tile mode: leading dimension (nq_pad)
};

// Parameters of the FILTER instances (both passes): row r is allowed for query q iff
// make_label_filter(require[q]).allows(labels[r]).  A separate type, so that the unfiltered instances keep theirs.
struct FilterScanParams : ScanParams {
  const uint32_t* labels;   // [N], 16-byte aligned
  const uint2* require;     // [nq] {all, any}
};

// The label filter of one query: (label & all) == all, and (label & any) != 0 unless any == 0.  any_free = 1 when
// any == 0, so that the second test passes for every label, 0 included.
struct LabelFilter {
  uint32_t all, any, any_free;
  __device__ __forceinline__ bool allows(uint32_t label) const {
    return ((label & all) == all) && (((label & any) | any_free) != 0u);
  }
};
__device__ __forceinline__ LabelFilter make_label_filter(uint2 req) {
  return LabelFilter{req.x, req.y, req.y == 0u ? 1u : 0u};
}
constexpr uint32_t NEG_INF_BITS = 0xff800000u;

// 32 accumulator columns of rows lab[0..31] (16-byte aligned): every disallowed column becomes -inf.  All lanes of a
// warp read the same words (broadcast loads).
__device__ __forceinline__ void mask_columns32(uint32_t (&v)[32], const uint32_t* __restrict__ lab, const LabelFilter& f) {
#pragma unroll
  for (int j = 0; j < 32; j += 4) {
    const uint4 l = __ldg(reinterpret_cast<const uint4*>(lab + j));
    if (!f.allows(l.x)) v[j] = NEG_INF_BITS;
    if (!f.allows(l.y)) v[j + 1] = NEG_INF_BITS;
    if (!f.allows(l.z)) v[j + 2] = NEG_INF_BITS;
    if (!f.allows(l.w)) v[j + 3] = NEG_INF_BITS;
  }
}

__device__ __forceinline__ float max3(float a, float b, float c) {
  float r;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));   // FMNMX3 (sm_100)
  return r;
}
__device__ __forceinline__ float max_tree(const uint32_t (&v)[32]) {
  float m[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) m[i] = max3(__uint_as_float(v[i]), __uint_as_float(v[i + 4]), __uint_as_float(v[i + 8]));
#pragma unroll
  for (int j = 12; j < 28; j += 8)
#pragma unroll
    for (int i = 0; i < 4; ++i) m[i] = max3(m[i], __uint_as_float(v[j + i]), __uint_as_float(v[j + i + 4]));
#pragma unroll
  for (int i = 0; i < 4; ++i) m[i] = fmaxf(m[i], __uint_as_float(v[28 + i]));
  return max3(fmaxf(m[0], m[1]), m[2], m[3]);
}

// Slow paths of the epilogue (warp-collective: every lane of the warp must call them).  They read
// `ncols` consecutive accumulator columns starting at `taddr`, 8 at a time, in a rolled loop.
static __device__ __noinline__ void append_columns(uint32_t taddr, int ncols, float thr, uint32_t row_base, uint2* seg,
                                            unsigned int& cnt, unsigned int seg_cap) {
#pragma unroll 1
  for (int c = 0; c < ncols; c += 8) {
    uint32_t v[8];
    __syncwarp();
    tmem_ld_32x8(taddr + (uint32_t)c, v);
    tmem_ld_wait();
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      if (c + j < ncols && __uint_as_float(v[j]) >= thr) {
        if (cnt < seg_cap) seg[cnt] = make_uint2(v[j], row_base + (uint32_t)(c + j));
        ++cnt;
      }
    }
  }
}
// r-th largest of the n <= 4096 sampled maxima of query q, by the 128 epilogue threads of a CTA (et = 0..127): the
// values sit in registers as order-preserving keys, four 8-bit radix passes over a 256-bin shared-memory histogram
// (`hist`, 1 KB) fix the key byte by byte; `tmp` = two words of shared memory.  Named barrier 1 (128 threads).
// One copy per FILTER value: ptxas fits a callee's registers to all its callers, and the unfiltered scan kernels keep
// the code they had without the FILTER instances.
template <bool FILTER>
static __device__ __noinline__ float epilogue_select(const float* __restrict__ sample, int n, int ld, int q, int query_major,
                                                     int r, uint32_t* hist, uint32_t* tmp, int et) {
  constexpr int VPT = 32;
  uint32_t key[VPT];
#pragma unroll
  for (int i = 0; i < VPT; ++i) {
    const int idx = et + i * 128;
    // padding key 0 sorts below every value, -inf included: it can never be among the r <= n largest
    key[i] = (idx < n) ? float_to_ordered(query_major ? __ldg(sample + (size_t)q * n + idx) : __ldg(sample + (size_t)idx * ld + q)) : 0u;
  }
  if (n < r) return -INFINITY;
  uint32_t prefix = 0u, mask = 0u;
  unsigned int kk = (unsigned int)r;
  const int lane = et & 31;
  for (int shift = 24; shift >= 0; shift -= 8) {
    hist[et] = 0u;
    hist[et + 128] = 0u;
    asm volatile("bar.sync 1, 128;" ::: "memory");
#pragma unroll
    for (int i = 0; i < VPT; ++i)
      if ((key[i] & mask) == prefix) atomicAdd(&hist[(key[i] >> shift) & 255u], 1u);
    asm volatile("bar.sync 1, 128;" ::: "memory");
    if (et < 32) {
      // lane l owns bins 255-8l .. 248-8l (descending)
      unsigned int loc[8], sum = 0;
#pragma unroll
      for (int j = 0; j < 8; ++j) { loc[j] = hist[255 - 8 * lane - j]; sum += loc[j]; }
      unsigned int incl = sum;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { const unsigned int v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
      const unsigned int excl = incl - sum;
      if (excl < kk && incl >= kk) {           // exactly one lane
        unsigned int above = excl;
        int d = 255 - 8 * lane - 7;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          if (above + loc[j] >= kk) { d = 255 - 8 * lane - j; break; }
          above += loc[j];
        }
        tmp[0] = (uint32_t)d;
        tmp[1] = kk - above;
      }
    }
    asm volatile("bar.sync 1, 128;" ::: "memory");
    prefix |= tmp[0] << shift;
    mask |= 255u << shift;
    kk = tmp[1];
  }
  return ordered_to_float(prefix);
}
static __device__ __noinline__ float max_columns(uint32_t taddr, int ncols) {
  float m = -INFINITY;
#pragma unroll 1
  for (int c = 0; c < ncols; c += 8) {
    uint32_t v[8];
    __syncwarp();
    tmem_ld_32x8(taddr + (uint32_t)c, v);
    tmem_ld_wait();
#pragma unroll
    for (int j = 0; j < 8; ++j) if (c + j < ncols) m = fmaxf(m, __uint_as_float(v[j]));
  }
  return m;
}
// The same two slow paths over allowed rows only (FILTER instances); column c is row row_base + c.  thr must not be
// -inf here (the caller clamps it to -FLT_MAX), so a masked column can never qualify.
static __device__ __noinline__ void append_columns_filtered(uint32_t taddr, int ncols, float thr, uint32_t row_base,
                                                            uint2* seg, unsigned int& cnt, unsigned int seg_cap,
                                                            const uint32_t* __restrict__ labels, LabelFilter f) {
#pragma unroll 1
  for (int c = 0; c < ncols; c += 8) {
    uint32_t v[8];
    __syncwarp();
    tmem_ld_32x8(taddr + (uint32_t)c, v);
    tmem_ld_wait();
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      if (c + j < ncols && __uint_as_float(v[j]) >= thr && f.allows(__ldg(labels + row_base + (uint32_t)(c + j)))) {
        if (cnt < seg_cap) seg[cnt] = make_uint2(v[j], row_base + (uint32_t)(c + j));
        ++cnt;
      }
    }
  }
}
static __device__ __noinline__ float max_columns_filtered(uint32_t taddr, int ncols, uint32_t row_base,
                                                          const uint32_t* __restrict__ labels, LabelFilter f) {
  float m = -INFINITY;
#pragma unroll 1
  for (int c = 0; c < ncols; c += 8) {
    uint32_t v[8];
    __syncwarp();
    tmem_ld_32x8(taddr + (uint32_t)c, v);
    tmem_ld_wait();
#pragma unroll
    for (int j = 0; j < 8; ++j)
      if (c + j < ncols && f.allows(__ldg(labels + row_base + (uint32_t)(c + j)))) m = fmaxf(m, __uint_as_float(v[j]));
  }
  return m;
}


}  // namespace tt
