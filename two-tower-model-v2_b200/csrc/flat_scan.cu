// Tensor-core catalog scan with a fused candidate filter (the hot loop of
// faiss.IndexFlatIP.search as called at src/inference/vector_db.py:160,197).
//
// scores[q, r] = <qh[q,:], Xh[r,:]>  (bf16 operands, fp32 accumulation in TMEM) for one block of
// queries against a stream of 256-row catalog tiles.  The score matrix never reaches shared or
// global memory: epilogue warps read the accumulator straight out of TMEM and keep only rows whose
// score reaches the query's threshold, appending (score, row) to a small candidate segment that
// belongs to this (query, catalog slice) alone - a register counter, no atomics.
//
// CTA anatomy (256 threads, 1 CTA / SM):
//   warp 0  lane 0 : TMA producer   - query block once (resident A operand, 128B swizzle), then
//                                     catalog K-blocks [rows x 64 bf16] through an mbarrier ring
//   warp 1  lane 0 : MMA issuer     - tcgen05.mma kind::f16, N = 256, K = 16; accumulators
//                                     double-buffered in TMEM (2 x 256 fp32 columns)
//   warp 2         : TMEM allocator
//   warps 4-7      : epilogue       - tcgen05.ld 32x32b, one query per thread, threshold in a
//                                     register; overlaps the next tile's MMAs
//
// Two tilings:
//   single (nq <= 128, or D > 512): cta_group::1, M = BLOCK_M queries (128, or 64 when D > 512).
//       HBM-bound regime: every CTA streams its own slice of the catalog once.
//   pair   (nq > 128): a cluster of two CTAs runs cta_group::2 MMAs with M = 256 queries (128 per
//       CTA, each resident in its own shared memory) and each CTA loads only HALF of every catalog
//       tile (128 rows): per-SM shared-memory traffic (operand reads + TMA writes) drops from
//       ~160 to ~96 bytes/cycle, which is what lets the tensor pipe run near its rate, and L2->SM
//       traffic halves.
//
// Work decomposition: unit = (query block [pair], catalog slice); slices interleave tiles
// (tile = slice + t * nslices) so that contiguous clusters of similar catalog rows spread over all
// slices, and units that share a slice run next to each other and share catalog tiles through L2.
//
// Two epilogue modes:
//   SAMPLE : scan every `tile_stride`-th tile and write only the maximum score of each 32-row
//            chunk (or of the whole tile) per query; the r-th largest of those maxima becomes the
//            query's threshold (select_threshold_radix_kernel / select_threshold_tile_kernel, or -
//            for a batch of one - the main scan's own prologue, epilogue_select).  The maxima are
//            scores of distinct rows, so the threshold is a guaranteed lower bound of the r-th best
//            bf16 score of the whole catalog.
//   MAIN   : scan every tile, append scores >= threshold.
//
// FILTER instances (per-row label words, per-query masks; tt_flat_search_filtered) turn every accumulator column whose
// row the query does not allow into -inf before the maximum and the threshold test, in both passes.  The sampled
// maxima are then maxima of allowed rows, so the threshold is a lower bound of the r-th best ALLOWED score and the
// certificate of the finalize kernel holds over allowed rows unchanged.  The threshold these instances compare against
// is max(thr, -FLT_MAX): it is -inf on the every-row-a-candidate route and for a query whose sample holds fewer allowed
// maxima than the rank, and -inf >= -inf would append masked columns.
#include <cuda.h>
#include <float.h>
#include <math.h>
#include "tt_common.cuh"
#include "sm100_ptx.cuh"
#include "flat_internal.cuh"
#include "flat_scan_common.cuh"

namespace tt {

using namespace ptx;

template <int BLOCK_M, bool SAMPLE, bool PAIR, bool FILTER>
__global__ void __launch_bounds__(SCAN_THREADS, 1)
flat_scan_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_x,
                 const std::conditional_t<FILTER, FilterScanParams, ScanParams> p) {
  constexpr int A_KB_BYTES = BLOCK_M * BLOCK_K * 2;
  constexpr int B_ROWS = PAIR ? BLOCK_N / 2 : BLOCK_N;            // rows of a tile this CTA loads
  constexpr int B_STAGE_BYTES = B_ROWS * BLOCK_K * 2;
  constexpr int UMMA_M = PAIR ? 2 * BLOCK_M : BLOCK_M;
  extern __shared__ uint8_t smem_raw[];
  // 128B-swizzled operand tiles need 1024-byte alignment (identical offsets in both CTAs of a pair)
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem_a + (size_t)p.num_kb_res * A_KB_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_b + (size_t)p.num_stages * p.stage_bytes);
  uint64_t* full_bar = bars;                       // [MAX_STAGES]
  uint64_t* empty_bar = bars + MAX_STAGES;         // [MAX_STAGES]
  uint64_t* a_full_bar = bars + 2 * MAX_STAGES;    // [1]
  uint64_t* tmem_full_bar = a_full_bar + 1;        // [2]
  uint64_t* tmem_empty_bar = tmem_full_bar + 2;    // [2]
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(tmem_empty_bar + 2);
  uint32_t* scratch_base = reinterpret_cast<uint32_t*>(reinterpret_cast<uint8_t*>(bars) + BAR_BYTES);   // 4 x 256 B

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t cta_rank = PAIR ? cluster_ctarank() : 0u;
  const bool leader = cta_rank == 0;
  pdl_trigger();      // the next kernel of the search may be scheduled once every CTA of this grid has started

  // ---- work assignment ----------------------------------------------------------------------
  const int unit = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  const int qu = unit % p.nqu;
  const int slice = unit / p.nqu;
  const int qb = PAIR ? (2 * qu + (int)cta_rank) : qu;           // 128- (or 64-) query block of this CTA
  const int ntiles = (p.num_slots > slice) ? (p.num_slots - slice + p.nslices - 1) / p.nslices : 0;

  // ---- one-time setup -----------------------------------------------------------------------
  if (warp == 0 && lane == 0) {
    prefetch_tensormap(&tmap_q);
    prefetch_tensormap(&tmap_x);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < p.num_stages; ++i) {
      mbar_init(smem_u32(full_bar + i), PAIR ? 2 : 1);     // pair: both producers arrive on the leader's barrier
      mbar_init(smem_u32(empty_bar + i), 1);
    }
    mbar_init(smem_u32(a_full_bar), PAIR ? 2 : 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(smem_u32(tmem_full_bar + i), 1);
      mbar_init(smem_u32(tmem_empty_bar + i), PAIR ? 8 : 4);   // one arrival per epilogue warp (of both CTAs)
    }
    fence_barrier_init();
  }
  if (PAIR) cluster_sync();        // peer barriers must be initialised before any remote arrive / 2-SM alloc
  if (warp == 2) {
    if (PAIR) { tmem_alloc_2cta(smem_u32(tmem_ptr_smem), TMEM_COLS); tmem_relinquish_2cta(); }
    else      { tmem_alloc(smem_u32(tmem_ptr_smem), TMEM_COLS); tmem_relinquish(); }
  }
  tc_fence_before();
  if (PAIR) cluster_sync(); else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  pdl_wait();         // barriers, TMEM and descriptors were set up under the previous kernel's tail; its outputs
                      // (query block, thresholds) are visible from here on

  if (warp == 0) {
    // =========================== TMA producer ===============================================
    if (lane == 0) {
      // In pair mode every TMA of either CTA signals the LEADER's barrier (the MMA issuer waits there).
      const uint32_t a_bar = smem_u32(a_full_bar);
      if (leader) mbar_arrive_expect_tx(a_bar, (uint32_t)(p.num_kb_res * A_KB_BYTES) * (PAIR ? 2u : 1u));
      for (int kb = 0; kb < p.num_kb_res; ++kb) {
        if (PAIR) tma_load_2d_2cta(smem_u32(smem_a + (size_t)kb * A_KB_BYTES), &tmap_q, a_bar, kb * BLOCK_K, qb * BLOCK_M);
        else      tma_load_2d(smem_u32(smem_a + (size_t)kb * A_KB_BYTES), &tmap_q, a_bar, kb * BLOCK_K, qb * BLOCK_M);
      }
      if (PAIR && !leader) mbar_arrive_remote(a_bar, 0);
      int stage = 0;
      uint32_t phase = 0;
      for (int t = 0; t < ntiles; ++t) {
        const long long tile = (long long)(slice + t * p.nslices) * p.tile_stride;
        const int row0 = (int)(tile * BLOCK_N) + (PAIR ? (int)cta_rank * B_ROWS : 0);
        for (int kb = 0; kb < p.num_kb; ++kb) {
          mbar_wait(smem_u32(empty_bar + stage), phase ^ 1, 100 + stage);
          const uint32_t fb = smem_u32(full_bar + stage);
          const bool stream_a = kb >= p.num_kb_res;
          const uint32_t dst = smem_u32(smem_b + (size_t)stage * p.stage_bytes);
          if (leader) mbar_arrive_expect_tx(fb, (uint32_t)(B_STAGE_BYTES + (stream_a ? A_KB_BYTES : 0)) * (PAIR ? 2u : 1u));
          if (PAIR) tma_load_2d_2cta(dst, &tmap_x, fb, kb * BLOCK_K, row0);
          else      tma_load_2d(dst, &tmap_x, fb, kb * BLOCK_K, row0);
          if (stream_a) {   // this K-block of the query block rides along (L2-resident after the first tile)
            if (PAIR) tma_load_2d_2cta(dst + B_STAGE_BYTES, &tmap_q, fb, kb * BLOCK_K, qb * BLOCK_M);
            else      tma_load_2d(dst + B_STAGE_BYTES, &tmap_q, fb, kb * BLOCK_K, qb * BLOCK_M);
          }
          if (PAIR && !leader) mbar_arrive_remote(fb, 0);
          if (++stage == p.num_stages) { stage = 0; phase ^= 1; }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // =========================== MMA issuer (leader CTA only in pair mode) ====================
    if (lane == 0 && leader) {
      constexpr uint32_t idesc = make_idesc_bf16_f32(UMMA_M, BLOCK_N);
      const uint64_t a_desc0 = make_smem_desc_sw128(smem_u32(smem_a));
      const uint64_t b_desc0 = make_smem_desc_sw128(smem_u32(smem_b));
      mbar_wait(smem_u32(a_full_bar), 0, 200);
      tc_fence_after();
      int stage = 0;
      uint32_t phase = 0;
      for (int t = 0; t < ntiles; ++t) {
        const int buf = t & 1;
        const uint32_t use_phase = (uint32_t)(t >> 1) & 1u;
        mbar_wait(smem_u32(tmem_empty_bar + buf), use_phase ^ 1, 210 + buf);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(buf * BLOCK_N);
        for (int kb = 0; kb < p.num_kb; ++kb) {
          mbar_wait(smem_u32(full_bar + stage), phase, 220 + stage);
          tc_fence_after();
          // descriptor start-address field is in 16-byte units
          const uint64_t b_desc = b_desc0 + (uint64_t)((stage * p.stage_bytes) >> 4);
          const uint64_t a_desc = (kb < p.num_kb_res) ? a_desc0 + (uint64_t)((kb * A_KB_BYTES) >> 4)
                                                      : b_desc + (uint64_t)(B_STAGE_BYTES >> 4);
#pragma unroll
          for (int k = 0; k < BLOCK_K / UMMA_K; ++k) {
            const uint64_t koff = (uint64_t)((k * UMMA_K * 2) >> 4);   // 32 bytes per K=16 step
            if (PAIR) mma_bf16_ss_2cta(d_tmem, a_desc + koff, b_desc + koff, idesc, (uint32_t)((kb | k) != 0));
            else      mma_bf16_ss(d_tmem, a_desc + koff, b_desc + koff, idesc, (uint32_t)((kb | k) != 0));
          }
          // smem slot free (in both CTAs) once these MMAs retire; accumulator ready after the last K-block
          if (PAIR) {
            mma_commit_2cta(smem_u32(empty_bar + stage));
            if (kb == p.num_kb - 1) mma_commit_2cta(smem_u32(tmem_full_bar + buf));
          } else {
            mma_commit(smem_u32(empty_bar + stage));
            if (kb == p.num_kb - 1) mma_commit(smem_u32(tmem_full_bar + buf));
          }
          if (++stage == p.num_stages) { stage = 0; phase ^= 1; }
        }
      }
    }
    __syncwarp();
  } else if (warp >= 4) {
    // =========================== epilogue ====================================================
    const int quad = warp & 3;                         // TMEM lane quadrant this warp may read
    int q_local;
    if (BLOCK_M == 128) q_local = quad * 32 + lane;    // accumulator row m lives in TMEM lane m
    else q_local = (lane < 16) ? quad * 16 + lane : -1;   // M=64: rows 16g..16g+15 -> lanes 32g..32g+15
    const int q = qb * BLOCK_M + q_local;
    const bool valid = (q_local >= 0) && (q < p.nq);

    float thr = INFINITY;
    LabelFilter flt{0u, 0u, 1u};                       // FILTER: this query's masks (padding lanes allow every row)
    if constexpr (FILTER) { if (valid) flt = make_label_filter(__ldg(p.require + q)); }
    if (!SAMPLE) {
      if (p.sel_n > 0) {
        // batch of one: no separate selection kernel - the 128 epilogue threads pick the threshold from the sampled
        // maxima while the producer and the MMA warp already stream the first tile
        uint32_t* sel_tmp = reinterpret_cast<uint32_t*>(bars) + 48;      // two free words of the barrier block
        for (int qq = 0; qq < p.nq; ++qq) {
          const float t = epilogue_select<FILTER>(p.sel_sample, p.sel_n, p.sel_ld, qq, p.sel_query_major, p.sel_rank, scratch_base,
                                          sel_tmp, (int)threadIdx.x - 128);
          if (q == qq) thr = t;
        }
        asm volatile("bar.sync 1, 128;" ::: "memory");      // the histogram doubles as the warps' scratch rows
        if (blockIdx.x == 0 && valid) p.thr_out[q] = thr;
      } else if (valid) {
        thr = __ldg(p.thr + q);
      }
      if (FILTER) thr = fmaxf(thr, -FLT_MAX);
    }
    uint2* my_cand = SAMPLE ? nullptr : (p.cand + ((size_t)(valid ? q : 0) * p.nslices + slice) * p.seg_cap);
    unsigned int my_cnt = 0;
    uint32_t* scratch = scratch_base + (warp - 4) * 64;

    for (int t = 0; t < ntiles; ++t) {
      const int buf = t & 1;
      const uint32_t use_phase = (uint32_t)(t >> 1) & 1u;
      const int slot = slice + t * p.nslices;
      const long long row0 = (long long)slot * p.tile_stride * BLOCK_N;
      const int ncols = (int)min((long long)BLOCK_N, p.N - row0);   // last tile may be partial
      if constexpr (FILTER) {   // the tile's label words into L1 while the MMAs run
        if (lane < CHUNKS && lane * 32 < ncols) asm volatile("prefetch.global.L1 [%0];" :: "l"(p.labels + row0 + lane * 32));
      }
      mbar_wait(smem_u32(tmem_full_bar + buf), use_phase, 300 + buf);
      tc_fence_after();
      const uint32_t taddr0 = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(buf * BLOCK_N);
      float* sample_row = SAMPLE ? (p.sample_out + ((size_t)(valid ? q : 0) * p.num_slots + slot) * CHUNKS) : nullptr;

      if (ncols == BLOCK_N) {
        // ---- full tile.  64 accumulator columns per step, software-pipelined over two register sets:
        // the tcgen05.ld of the next 64 columns is in flight while the current 64 are reduced (3-input
        // max tree) and compared once against the threshold.  The loop stays rolled (a fully unrolled
        // 256-way compare/append thrashed the instruction cache).
        uint32_t a0[32], a1[32], b0[32], b1[32];
        float tile_max = -INFINITY;
        auto consume = [&](const uint32_t (&v0)[32], const uint32_t (&v1)[32], int c) {
          const float m0 = max_tree(v0);
          const float m1 = max_tree(v1);
          if (SAMPLE) {
            if (p.sample_tile_max) tile_max = fmaxf(tile_max, fmaxf(m0, m1));
            else if (valid) *reinterpret_cast<float2*>(sample_row + c) = make_float2(m0, m1);
          } else {
            // Lanes (queries) with a qualifying column among these 64.  Hits are sparse - a handful per
            // tile for the whole warp - so they are extracted cooperatively: the hit lane spills its 64
            // values to a 256-byte scratch row, the warp re-reads them one column per lane, and the
            // qualifying (score, row) pairs are appended to that query's segment with ballot-prefix
            // positions (coalesced 8-byte stores).  Cost is per hit, not per column.
            unsigned int hitmask = __ballot_sync(0xffffffffu, fmaxf(m0, m1) >= thr);
            while (hitmask) {
              const int src = __ffs(hitmask) - 1;
              hitmask &= hitmask - 1;
              // which 32-column halves of the hit lane qualify (usually one): only those are spilled and re-read
              const unsigned int halves = __shfl_sync(0xffffffffu, (m0 >= thr ? 1u : 0u) | (m1 >= thr ? 2u : 0u), src);
              if (lane == src) {
                if (halves & 1u) {
#pragma unroll
                  for (int j = 0; j < 32; j += 4)
                    *reinterpret_cast<uint4*>(scratch + j) = make_uint4(v0[j], v0[j + 1], v0[j + 2], v0[j + 3]);
                }
                if (halves & 2u) {
#pragma unroll
                  for (int j = 0; j < 32; j += 4)
                    *reinterpret_cast<uint4*>(scratch + 32 + j) = make_uint4(v1[j], v1[j + 1], v1[j + 2], v1[j + 3]);
                }
              }
              __syncwarp();
              const float thr_s = __shfl_sync(0xffffffffu, thr, src);
              const unsigned int cnt_s = __shfl_sync(0xffffffffu, my_cnt, src);
              const int q_s = __shfl_sync(0xffffffffu, q, src);
              const uint32_t x0 = (halves & 1u) ? scratch[lane] : 0xff800000u;          // -inf: never qualifies
              const uint32_t x1 = (halves & 2u) ? scratch[32 + lane] : 0xff800000u;
              const bool h0 = __uint_as_float(x0) >= thr_s, h1 = __uint_as_float(x1) >= thr_s;
              const unsigned int b0 = __ballot_sync(0xffffffffu, h0), b1 = __ballot_sync(0xffffffffu, h1);
              const unsigned int lt = (1u << lane) - 1u;
              const unsigned int p0 = cnt_s + __popc(b0 & lt), p1 = cnt_s + __popc(b0) + __popc(b1 & lt);
              uint2* seg = p.cand + ((size_t)q_s * p.nslices + slice) * p.seg_cap;
              const uint32_t rbase = (uint32_t)row0 + (uint32_t)(c * 32 + lane);
              if (h0 && p0 < (unsigned int)p.seg_cap) seg[p0] = make_uint2(x0, rbase);
              if (h1 && p1 < (unsigned int)p.seg_cap) seg[p1] = make_uint2(x1, rbase + 32u);
              if (lane == src) my_cnt += __popc(b0) + __popc(b1);
              __syncwarp();
            }
          }
        };
        __syncwarp();
        tmem_ld_32x32(taddr0, a0);
        tmem_ld_32x32(taddr0 + 32u, a1);
#pragma unroll 1
        for (int c = 0; c < CHUNKS; c += 4) {
          tmem_ld_wait();
          __syncwarp();
          tmem_ld_32x32(taddr0 + (uint32_t)(c * 32 + 64), b0);
          tmem_ld_32x32(taddr0 + (uint32_t)(c * 32 + 96), b1);
          if constexpr (FILTER) { mask_columns32(a0, p.labels + row0 + c * 32, flt); mask_columns32(a1, p.labels + row0 + c * 32 + 32, flt); }
          consume(a0, a1, c);
          tmem_ld_wait();
          if (c + 4 < CHUNKS) {
            __syncwarp();
            tmem_ld_32x32(taddr0 + (uint32_t)(c * 32 + 128), a0);
            tmem_ld_32x32(taddr0 + (uint32_t)(c * 32 + 160), a1);
          }
          if constexpr (FILTER) { mask_columns32(b0, p.labels + row0 + c * 32 + 64, flt); mask_columns32(b1, p.labels + row0 + c * 32 + 96, flt); }
          consume(b0, b1, c + 2);
        }
        if (SAMPLE && p.sample_tile_max && q_local >= 0)
          p.sample_out[(size_t)slot * p.sample_ld + (size_t)(qb * BLOCK_M + q_local)] = tile_max;
      } else {
        // ---- partial last tile: columns >= ncols are zero-filled padding rows ----------------------
        if (SAMPLE) {
          float tile_max = -INFINITY;
          for (int c = 0; c < CHUNKS; ++c) {
            const int limit = min(32, ncols - c * 32);
            float m;
            if constexpr (FILTER)
              m = (limit > 0) ? max_columns_filtered(taddr0 + (uint32_t)(c * 32), limit, (uint32_t)row0 + (uint32_t)(c * 32), p.labels, flt)
                              : -INFINITY;
            else
              m = (limit > 0) ? max_columns(taddr0 + (uint32_t)(c * 32), limit) : -INFINITY;
            if (p.sample_tile_max) tile_max = fmaxf(tile_max, m);
            else if (valid) sample_row[c] = m;
          }
          if (p.sample_tile_max && q_local >= 0)
            p.sample_out[(size_t)slot * p.sample_ld + (size_t)(qb * BLOCK_M + q_local)] = tile_max;
        } else {
          if constexpr (FILTER) append_columns_filtered(taddr0, ncols, thr, (uint32_t)row0, my_cand, my_cnt, (unsigned int)p.seg_cap, p.labels, flt);
          else append_columns(taddr0, ncols, thr, (uint32_t)row0, my_cand, my_cnt, (unsigned int)p.seg_cap);
        }
      }
      // release this accumulator buffer to the MMA issuer (on the leader CTA)
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (PAIR && !leader) mbar_arrive_remote(smem_u32(tmem_empty_bar + buf), 0);
        else mbar_arrive(smem_u32(tmem_empty_bar + buf));
      }
    }
    if (!SAMPLE && valid) p.seg_cnt[(size_t)q * p.nslices + slice] = my_cnt;
  }

  // ---- teardown ---------------------------------------------------------------------------
  tc_fence_before();
  if (PAIR) cluster_sync(); else __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    if (PAIR) tmem_dealloc_2cta(tmem_base, TMEM_COLS);
    else tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

// ------------------------------------------------------------------------------------------
// thr[q] = r-th largest of the sampled chunk maxima of query q; -inf if there are fewer than r.
// One CTA per query, values staged in shared memory.  Small r: r rounds of block-wide arg-max where
// every thread caches the best of its own strided values and only the winner rescans; large r: a
// bitonic sort.
__global__ void __launch_bounds__(256)
select_threshold_kernel(const float* __restrict__ sample, int n, int npad, int r, float* thr) {
  pdl_trigger();
  pdl_wait();
  extern __shared__ float vals[];
  __shared__ float wmax[8];
  __shared__ int widx[8];
  const int q = blockIdx.x;
  for (int i = threadIdx.x; i < npad; i += blockDim.x) vals[i] = (i < n) ? sample[(size_t)q * n + i] : -INFINITY;
  __syncthreads();
  if (r > 64) {
    for (int k = 2; k <= npad; k <<= 1) {
      for (int j = k >> 1; j > 0; j >>= 1) {
        for (int i = threadIdx.x; i < npad; i += blockDim.x) {
          const int ixj = i ^ j;
          if (ixj > i) {
            const float a = vals[i], b = vals[ixj];
            const bool up = (i & k) == 0;
            if (up ? (a < b) : (a > b)) { vals[i] = b; vals[ixj] = a; }
          }
        }
        __syncthreads();
      }
    }
    if (threadIdx.x == 0) thr[q] = (r <= n) ? vals[r - 1] : -INFINITY;
    return;
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float best = -INFINITY;   // best of this thread's own values (indices tid, tid+256, ...)
  int bi = -1;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const float v = vals[i];
    if (v > best) { best = v; bi = i; }
  }
  float result = -INFINITY;
  for (int round = 0; round < r; ++round) {
    float wb = best;
    int wi = bi;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ob = __shfl_xor_sync(0xffffffffu, wb, o);
      const int oi = __shfl_xor_sync(0xffffffffu, wi, o);
      if (ob > wb || (ob == wb && oi > wi)) { wb = ob; wi = oi; }
    }
    if (lane == 0) { wmax[warp] = wb; widx[warp] = wi; }
    __syncthreads();
    float b = wmax[0];
    int idx = widx[0];
#pragma unroll
    for (int w = 1; w < 8; ++w) if (wmax[w] > b || (wmax[w] == b && widx[w] > idx)) { b = wmax[w]; idx = widx[w]; }
    result = (idx >= 0) ? b : -INFINITY;
    if (idx >= 0 && idx == bi) {             // this thread owns the winner: drop it and rescan its values
      vals[idx] = -INFINITY;
      best = -INFINITY; bi = -1;
      for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const float v = vals[i];
        if (v > best) { best = v; bi = i; }
      }
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) thr[q] = result;
}

// Tile mode: thr[q] = r-th largest of the sampled tile maxima sample[slot][q] (query fastest), one warp
// per query.  The CTA stages a [slots x WQ] panel through shared memory with sector-sized reads, then
// every warp runs r rounds of arg-max over its own column (each lane caches the best of its strided
// values; only the winning lane rescans).  No block-wide barrier inside the rounds.
// r rounds of "take the largest remaining value" over one warp's values v[0..n) (shared memory; lane l caches the best
// of v[l], v[l+32], ... in best/bi).  A round is ONE redux.sync (warp max of the order-preserving uint32 image of the
// lanes' bests) + one ballot to elect the owning lane, which drops its value and rescans its own stripe - instead of
// a 5-step shuffle arg-max of (value, index) pairs.  Returns the r-th largest (-inf if fewer than r values); the
// largest `out_n` are also written to out[] when given.
__device__ __forceinline__ float warp_select_rounds(float* v, int n, int r, float best, int bi, int lane, float* out, int out_n) {
  uint32_t kbest = (bi >= 0) ? float_to_ordered(best) : 0u;
  float result = -INFINITY;
  for (int round = 0; round < r; ++round) {
    const uint32_t kmax = __reduce_max_sync(0xffffffffu, kbest);
    const unsigned int owners = __ballot_sync(0xffffffffu, bi >= 0 && kbest == kmax);
    result = owners ? ordered_to_float(kmax) : -INFINITY;
    if (out && lane == 0 && round < out_n) out[round] = result;
    if (owners && lane == __ffs(owners) - 1) {        // this lane owns the winner: drop it and rescan its own values
      v[bi] = -INFINITY;
      float nb = -INFINITY;
      int ni = -1;
      for (int i = lane; i < n; i += 32) {
        const float x = v[i];
        if (x > nb) { nb = x; ni = i; }
      }
      best = nb; bi = ni;
      kbest = (bi >= 0) ? float_to_ordered(best) : 0u;
    }
    __syncwarp();
  }
  return result;
}

constexpr int SEL_WQ = 8;   // queries (warps) per CTA
__global__ void __launch_bounds__(SEL_WQ * 32)
select_threshold_tile_kernel(const float* __restrict__ sample, int slots, int ld, int nq, int r, float* __restrict__ thr,
                             float* __restrict__ topr, int topr_ld) {
  pdl_trigger();
  pdl_wait();
  extern __shared__ float sv[];   // [SEL_WQ][slots]
  const int q0 = blockIdx.x * SEL_WQ;
  for (int e = threadIdx.x; e < slots * SEL_WQ; e += blockDim.x) {      // tile maxima: sample[slot][ld] (query fastest)
    const int i = e / SEL_WQ, qq = e % SEL_WQ;
    sv[qq * slots + i] = (q0 + qq < ld) ? sample[(size_t)i * ld + q0 + qq] : -INFINITY;
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int q = q0 + warp;
  if (q >= nq) return;
  float* v = sv + warp * slots;
  float best = -INFINITY;
  int bi = -1;
  for (int i = lane; i < slots; i += 32) {
    const float x = v[i];
    if (x > best) { best = x; bi = i; }
  }
  const float result = warp_select_rounds(v, slots, r, best, bi, lane, topr ? topr + (size_t)q * topr_ld : nullptr, topr_ld);
  if (thr && lane == 0) thr[q] = result;
  if (topr) for (int i = r + lane; i < topr_ld; i += 32) topr[(size_t)q * topr_ld + i] = -INFINITY;
}

// thr[q] = r-th largest of the n <= 4096 sampled maxima of query q by a CTA-wide radix select: the values sit in
// registers (16 per thread) as order-preserving 32-bit keys and four 8-bit passes (shared-memory histogram, one warp
// scans it from the top) fix the key byte by byte.  ~1.5 us whatever r is; the warp-per-query rounds above cost
// ~130 ns per rank (8.9 us at r = 66, the small-batch plan of a 1M-row catalog).
constexpr int SELR_THREADS = 256, SELR_VPT = 16;
__global__ void __launch_bounds__(SELR_THREADS)
select_threshold_radix_kernel(const float* __restrict__ sample, int n, int ld, int r, float* __restrict__ thr, int query_major) {
  pdl_trigger();
  pdl_wait();
  __shared__ unsigned int hist[256];
  __shared__ unsigned int s_digit, s_kk;
  const int q = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  uint32_t key[SELR_VPT];
#pragma unroll
  for (int i = 0; i < SELR_VPT; ++i) {
    const int idx = tid + i * SELR_THREADS;
    // padding key 0 sorts below every finite value, -inf included: it can never be among the r <= n largest
    key[i] = (idx < n) ? float_to_ordered(query_major ? sample[(size_t)q * n + idx] : sample[(size_t)idx * ld + q]) : 0u;
  }
  if (n < r) {
    if (tid == 0) thr[q] = -INFINITY;
    return;
  }
  uint32_t prefix = 0u, mask = 0u;
  unsigned int kk = (unsigned int)r;
  for (int shift = 24; shift >= 0; shift -= 8) {
    hist[tid] = 0u;
    __syncthreads();
#pragma unroll
    for (int i = 0; i < SELR_VPT; ++i)
      if ((key[i] & mask) == prefix) atomicAdd(&hist[(key[i] >> shift) & 255u], 1u);
    __syncthreads();
    if (warp == 0) {
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
        s_digit = (unsigned int)d;
        s_kk = kk - above;
      }
    }
    __syncthreads();
    prefix |= s_digit << shift;
    mask |= 255u << shift;
    kk = s_kk;
  }
  if (tid == 0) thr[q] = ordered_to_float(prefix);
}

// Sharded catalogs: thr[q] = r-th largest of the union of every rank's top-r sampled tile maxima
// (gathered f32 [G, nq, SHARD_TOPR], the layout an all-gather of the per-rank lists produces): the same
// threshold on every rank, estimated from a sample of the WHOLE catalog.  One warp per query.
__global__ void __launch_bounds__(SEL_WQ * 32)
select_threshold_gathered_kernel(const float* __restrict__ gathered, int G, int nq, int r, float* __restrict__ thr,
                                 int* zero_me) {
  pdl_trigger();
  pdl_wait();
  extern __shared__ float sv[];   // [SEL_WQ][G * SHARD_TOPR]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (zero_me && blockIdx.x == 0 && threadIdx.x == 0) *zero_me = 0;     // n_uncertified of this call
  const int q = blockIdx.x * SEL_WQ + warp;
  if (q >= nq) return;
  const int n = G * SHARD_TOPR;
  float* v = sv + warp * n;
  float best = -INFINITY;
  int bi = -1;
  for (int i = lane; i < n; i += 32) {
    const int g = i / SHARD_TOPR, j = i % SHARD_TOPR;
    const float x = gathered[((size_t)g * nq + q) * SHARD_TOPR + j];
    v[i] = x;
    if (x > best) { best = x; bi = i; }
  }
  __syncwarp();
  const float result = warp_select_rounds(v, n, r, best, bi, lane, nullptr, 0);
  if (lane == 0) thr[q] = result;
}

__global__ void fill_kernel(float* p, int n, float v) {
  pdl_trigger();
  pdl_wait();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}

// ------------------------------------------------------------------------------------------
// host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// bf16 [rows, pitch] row-major, box = [box_rows, 64 columns], 128-byte swizzle, OOB rows read as 0.
static int encode_tmap_bf16(CUtensorMap* m, const void* base, long long rows, int pitch, int box_rows);


// A search call encodes four descriptors (query block + catalog, sample + main pass) that only depend on
// (base, rows, pitch, box): a small per-thread cache saves the driver calls on the small-batch path, where the
// host enqueue time is comparable to the device time.
static int make_tmap_bf16(CUtensorMap* m, const void* base, long long rows, int pitch, int box_rows) {
  struct Entry { const void* base; long long rows; int pitch, box_rows; unsigned long long stamp; CUtensorMap map; };
  constexpr int NE = 16;
  static thread_local Entry cache[NE] = {};
  static thread_local unsigned long long clock_ = 0;
  int victim = 0;
  for (int i = 0; i < NE; ++i) {
    Entry& e = cache[i];
    if (e.stamp && e.base == base && e.rows == rows && e.pitch == pitch && e.box_rows == box_rows) {
      e.stamp = ++clock_;
      *m = e.map;
      return TT_OK;
    }
    if (e.stamp < cache[victim].stamp) victim = i;
  }
  if (int err = encode_tmap_bf16(m, base, rows, pitch, box_rows)) return err;
  cache[victim] = Entry{base, rows, pitch, box_rows, ++clock_, *m};
  return TT_OK;
}

static int encode_tmap_bf16(CUtensorMap* m, const void* base, long long rows, int pitch, int box_rows) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) { set_error("cuTensorMapEncodeTiled entry point not available"); return TT_ERR_CUDA; }
  cuuint64_t dims[2] = {(cuuint64_t)pitch, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)pitch * 2};
  cuuint32_t box[2] = {(cuuint32_t)BLOCK_K, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed with CUresult " + std::to_string((int)r));
    return TT_ERR_CUDA;
  }
  return TT_OK;
}

// fp32 [rows, cols] row-major (row pitch = cols*4 bytes, a multiple of 16), box = [box_rows, box_cols <= 32],
// 128-byte swizzle, out-of-range rows/columns read as 0.
int make_tmap_f32(void* tensor_map, const void* base, long long rows, int cols, int box_rows, int box_cols) {
  CUtensorMap* m = reinterpret_cast<CUtensorMap*>(tensor_map);
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) { set_error("cuTensorMapEncodeTiled entry point not available"); return TT_ERR_CUDA; }
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)cols * 4};
  cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled (f32) failed with CUresult " + std::to_string((int)r));
    return TT_ERR_CUDA;
  }
  return TT_OK;
}

// Number of catalog slices for `nqu` query units on `cap` concurrent units (SMs, or SM pairs):
// the count that wastes the fewest unit slots over whole waves.
static int pick_slices(int nqu, int cap, int max_slices) {
  if (max_slices < 1) max_slices = 1;
  if (nqu >= cap) return 1;
  int best = 1;
  double best_eff = 0.0;
  const int hi = max_slices < 4 * cap ? max_slices : 4 * cap;
  for (int ns = 1; ns <= hi; ++ns) {
    const long long total = (long long)nqu * ns;
    const long long waves = (total + cap - 1) / cap;
    const double eff = (double)total / (double)(waves * cap);
    if (eff > best_eff + 1e-9) { best_eff = eff; best = ns; }
    if (total >= cap && eff > 0.97) break;     // good enough; more slices only add prologues
  }
  return best;
}

ScanPlan make_scan_plan(long long N, int D, int nq, int K) {
  ScanPlan pl{};
  pl.Dp = (int)tt_flat_pitch(D);
  pl.num_kb = pl.Dp / BLOCK_K;
  const int sms = num_sms();
  const int budget = 227 * 1024 - 1024 /*align*/ - BAR_BYTES - SCRATCH_BYTES;
  const int kb_bytes_m128 = 128 * BLOCK_K * 2;                 // one K-block of a 128-query block: 16 KB
  const int b_full = BLOCK_N * BLOCK_K * 2, b_half = b_full / 2;
  pl.block_m = 128;
  pl.num_kb_res = pl.num_kb;
  // CTA pairs for nq > 128, and already for nq > 64 when the rows are too wide for a resident 128-query block
  // (D > 512): two 64-query single-CTA units would read every catalog tile twice and run M = 64 MMAs at half rate
  // (10M x 768, nq = 128: 0.81 of the HBM peak), the pair keeps one pass over the catalog.
  const bool wide = budget - pl.num_kb * kb_bytes_m128 < 3 * b_full;
  pl.pair = (nq > 128 || (wide && nq > 64)) && (sms >= 2);
  if (pl.pair) {
    // 2-CTA tiling, 128 queries per CTA.  The query block stays resident while it leaves room for 4 half-tile
    // stages (D <= 640); wider rows keep the leading K-blocks resident and stream the rest with the catalog.
    if (pl.num_kb * kb_bytes_m128 + 4 * b_half <= budget) {
      pl.stage_bytes = b_half;
    } else {
      pl.stage_bytes = b_half + kb_bytes_m128;
      pl.num_kb_res = (budget - 4 * pl.stage_bytes) / kb_bytes_m128;
      if (pl.num_kb_res < 0) pl.num_kb_res = 0;
      if (pl.num_kb_res > pl.num_kb) pl.num_kb_res = pl.num_kb;
    }
  } else {
    // single-CTA tiling (HBM-bound batches): resident query block of 128 rows while it leaves room for >= 3
    // full-tile stages, else 64 rows.
    if (budget - pl.num_kb * kb_bytes_m128 < 3 * b_full) pl.block_m = 64;
    pl.stage_bytes = b_full;
  }
  const int a_bytes = pl.num_kb_res * pl.block_m * BLOCK_K * 2;
  pl.num_stages = (budget - a_bytes) / pl.stage_bytes;
  if (pl.num_stages > MAX_STAGES) pl.num_stages = MAX_STAGES;
  pl.supported = pl.num_stages >= 2;
  pl.smem_bytes = (size_t)a_bytes + (size_t)pl.num_stages * pl.stage_bytes + 1024 /*align*/ + BAR_BYTES + SCRATCH_BYTES;
  pl.nqb = (nq + pl.block_m - 1) / pl.block_m;
  if (pl.pair) pl.nqb = (pl.nqb + 1) / 2 * 2;
  pl.nq_pad = pl.nqb * pl.block_m;
  pl.nqu = pl.pair ? pl.nqb / 2 : pl.nqb;
  pl.num_tiles = (int)((N + BLOCK_N - 1) / BLOCK_N);
  const int cap_units = pl.pair ? sms / 2 : sms;
  pl.main_slices = pick_slices(pl.nqu, cap_units, pl.num_tiles);

  // Candidate budget and sampling plan.  We aim at ~T candidates per query: the threshold is read
  // among the 32-row chunk maxima of every `stride`-th tile at the rank r' = T * n_s / N (n_s =
  // sampled rows) corrected for chunk collisions.  r' >= 12 keeps the sampling noise of the
  // candidate count near +-30%.
  auto try_plan = [&](int T, int stride) -> bool {
    if (stride < 1) stride = 1;
    long long slots = (pl.num_tiles + stride - 1) / stride;
    if (slots > SAMPLE_MAX_SLOTS) return false;
    const long long last_slot = slots - 1;
    long long rem = N - last_slot * (long long)stride * BLOCK_N;
    if (rem > BLOCK_N) rem = BLOCK_N;
    const long long ns_rows = last_slot * BLOCK_N + rem;
    // r' = rank (within the sample) of the score that ~T rows of the whole catalog reach
    const double rp = (double)T * (double)ns_rows / (double)N;
    // One maximum per sampled tile is enough (and 8x less data to write, read and select from) when the
    // top-r' sampled rows rarely share a tile; otherwise keep one maximum per 32-row chunk.
    const bool tile_mode = slots >= 128 && rp <= (double)slots / 4.0 && rp <= 64.0;
    const double nvals = tile_mode ? (double)slots : (double)(slots * CHUNKS);
    if (rp < 11.5 || rp > 1.5 * nvals) return false;
    if (nvals < 128.0 && stride > 1) return false;   // too few chunk maxima for a stable quantile: sample denser
    // The top-r' sampled rows occupy about nvals*(1-exp(-r'/nvals)) distinct 32-row chunks, so that is
    // the rank to read among the chunk maxima (a smaller rank would only over-fetch; never unsafe).
    const double r = nvals * (1.0 - exp(-rp / nvals));
    pl.target = T;
    pl.sample_stride = stride;
    pl.sample_slots = (int)slots;
    pl.sample_rank = (int)(r + 0.5) < 1 ? 1 : (int)(r + 0.5);
    pl.sample_tile_max = tile_mode;
    return true;
  };
  bool reliable = false;
  const int Tmax = FINALIZE_MAX_CAND / 4;
  {
    // ~10K candidates: with r' ~ 16 the count is ~Gamma(16)-distributed around T, and the certificate
    // needs about K + 2*eps*density (~2.2K at N = 1e7, K = 100) of them: P(fail) ~ 1e-6 per query.
    // Extra candidates are cheap (8-byte append; finalize prunes before rescoring).
    int T = 10 * K < 256 ? 256 : 10 * K;
    if (T > Tmax) T = Tmax;
    // (a) r' ~ 16 from a sparse sample; small catalogs / large K fall through to denser samples
    for (int stride = T / 16; !reliable && stride >= 1; stride /= 2) reliable = try_plan(T, stride);
    // (b) huge catalogs: the slot cap forces a sparser sample; raise T so that r' stays >= 12
    if (!reliable && (pl.num_tiles + T / 16 - 1) / (T / 16) > SAMPLE_MAX_SLOTS) {
      const int stride = (pl.num_tiles + SAMPLE_MAX_SLOTS - 1) / SAMPLE_MAX_SLOTS;
      for (int T2 = T; T2 <= Tmax && !reliable; T2 += T2 / 4 + 1) reliable = try_plan(T2, stride);
    }
    // (c) K is a large fraction of N: a leaner budget
    const int T_lean = (3 * K + 64 < 128) ? 128 : 3 * K + 64;
    if (!reliable && T_lean < T && T_lean <= Tmax)
      for (int stride = T_lean / 16; !reliable && stride >= 1; stride /= 2) reliable = try_plan(T_lean, stride);
  }
  int C = 4096;
  if (reliable) while (C < 4 * pl.target) C <<= 1;
  if (C > FINALIZE_MAX_CAND) C = FINALIZE_MAX_CAND;

  // Routing: threshold path when the estimate is trustworthy; otherwise every row is a candidate
  // if the catalog fits a candidate list, else the always-exact fp32 path.
  pl.route_exact = false;
  pl.use_threshold = reliable;
  const long long slice_rows = ((long long)(pl.num_tiles + pl.main_slices - 1) / pl.main_slices) * BLOCK_N;
  if (!reliable) {
    pl.sample_stride = 1; pl.sample_slots = 1; pl.sample_rank = 1; pl.target = 0; pl.sample_tile_max = false;
    if (N <= FINALIZE_MAX_CAND) {
      C = 2048;
      while (C < N) C <<= 1;
      pl.seg_cap = (int)slice_rows;                   // a slice can report every one of its rows
    } else {
      pl.route_exact = true;
      pl.seg_cap = 64;
    }
  } else {
    // Segment of one (query, slice): 4x its fair share of the target, at least 512 (bursts of
    // near-duplicate rows land in few slices), never more than the slice has rows.
    long long seg = 4LL * pl.target / pl.main_slices;
    if (seg < 512) seg = 512;
    if (seg > C) seg = C;
    if (seg > slice_rows) seg = slice_rows;
    pl.seg_cap = (int)((seg + 63) / 64 * 64);
  }
  pl.sample_slices = pick_slices(pl.nqu, cap_units, pl.sample_slots);
  pl.cand_cap = C;
  return pl;
}

template <int BLOCK_M, bool SAMPLE, bool PAIR, bool FILTER>
static int launch_scan_t(const CUtensorMap& tq, const CUtensorMap& tx, const FilterScanParams& fsp, int units, size_t smem,
                         cudaStream_t st) {
  const std::conditional_t<FILTER, FilterScanParams, ScanParams>& sp = fsp;
  auto kern = flat_scan_kernel<BLOCK_M, SAMPLE, PAIR, FILTER>;
  TT_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)(PAIR ? 2 * units : units));
  cfg.blockDim = dim3(SCAN_THREADS);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = PAIR ? 2 : 1;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 2;
  count_launch();
  TT_CHECK_CUDA(cudaLaunchKernelEx(&cfg, kern, tq, tx, sp));
  return TT_OK;
}

template <bool SAMPLE, bool FILTER>
static int launch_scan_tiling(const ScanPlan& pl, const CUtensorMap& tq, const CUtensorMap& tx, const FilterScanParams& sp,
                              int units, cudaStream_t st) {
  if (pl.pair) return launch_scan_t<128, SAMPLE, true, FILTER>(tq, tx, sp, units, pl.smem_bytes, st);
  if (pl.block_m == 128) return launch_scan_t<128, SAMPLE, false, FILTER>(tq, tx, sp, units, pl.smem_bytes, st);
  return launch_scan_t<64, SAMPLE, false, FILTER>(tq, tx, sp, units, pl.smem_bytes, st);
}

// the FILTER instances run when the call has label words
template <bool SAMPLE>
static int launch_scan_mode(const ScanPlan& pl, const CUtensorMap& tq, const CUtensorMap& tx, const FilterScanParams& sp,
                            int units, cudaStream_t st) {
  return sp.labels ? launch_scan_tiling<SAMPLE, true>(pl, tq, tx, sp, units, st)
                   : launch_scan_tiling<SAMPLE, false>(pl, tq, tx, sp, units, st);
}

static int make_scan_params(const ScanPlan& pl, const void* qh, const void* Xh, long long N, int nq, float* thr,
                            unsigned int* seg_cnt, void* cand, float* sample_buf, const LabelArgs& lab, CUtensorMap* tq,
                            CUtensorMap* tx, FilterScanParams* sp) {
  if (int e = make_tmap_bf16(tq, qh, pl.nq_pad, pl.Dp, pl.block_m)) return e;
  if (int e = make_tmap_bf16(tx, Xh, N, pl.Dp, pl.pair ? BLOCK_N / 2 : BLOCK_N)) return e;
  *sp = FilterScanParams{};
  sp->N = N; sp->nq = nq; sp->num_kb = pl.num_kb; sp->num_stages = pl.num_stages; sp->nqu = pl.nqu;
  sp->num_kb_res = pl.num_kb_res; sp->stage_bytes = pl.stage_bytes;
  sp->thr = thr; sp->seg_cnt = seg_cnt; sp->cand = reinterpret_cast<uint2*>(cand); sp->seg_cap = pl.seg_cap;
  sp->sample_out = sample_buf;
  sp->sample_tile_max = pl.sample_tile_max ? 1 : 0;
  sp->sample_ld = pl.nq_pad;
  sp->labels = lab.labels;
  sp->require = reinterpret_cast<const uint2*>(lab.require);
  return TT_OK;
}

// Sample pass + selection.  thr != NULL: the query's threshold; topr != NULL (tile mode only): its
// SHARD_TOPR largest sampled tile maxima, descending (sharded catalogs exchange these lists).
// A single query (the batch-1 serving call): the main scan selects the threshold itself (epilogue_select).  Measured at
// 1M x 384: 150.4 vs 155.2 us per step at nq = 1; at nq = 4 the four selections in a row delay the first epilogue
// enough to stall the MMAs (174.9 vs 158.3 us), so larger batches keep the separate kernel.
static bool fold_select(const ScanPlan& pl, int nq) {
  const int nvals = pl.sample_tile_max ? pl.sample_slots : pl.sample_slots * CHUNKS;
  return nq == 1 && !pl.pair && pl.nqu == 1 && nvals <= 4096;
}

int launch_sample(const ScanPlan& pl, const void* qh, const void* Xh, long long N, int nq, float* thr, float* topr,
                  float* sample_buf, cudaStream_t st, bool skip_select, const LabelArgs& lab) {
  CUtensorMap tq, tx;
  FilterScanParams sp;
  if (int e = make_scan_params(pl, qh, Xh, N, nq, thr, nullptr, nullptr, sample_buf, lab, &tq, &tx, &sp)) return e;
  sp.num_slots = pl.sample_slots; sp.tile_stride = pl.sample_stride; sp.nslices = pl.sample_slices;
  if (int e = launch_scan_mode<true>(pl, tq, tx, sp, pl.sample_slices * pl.nqu, st)) return e;
  if (skip_select) return TT_OK;
  {
    // few values per query: CTA-wide radix select (query-minor tile maxima only for small batches: a CTA reads one
    // 4-byte value per sampled tile row there)
    const int nvals = pl.sample_tile_max ? pl.sample_slots : pl.sample_slots * CHUNKS;
    if (!topr && nvals <= SELR_THREADS * SELR_VPT && (!pl.sample_tile_max || nq <= 256)) {
      TT_CHECK_CUDA(launch_pdl(select_threshold_radix_kernel, dim3(nq), dim3(SELR_THREADS), 0, st, (const float*)sample_buf, nvals,
                               pl.nq_pad, pl.sample_rank, thr, pl.sample_tile_max ? 0 : 1));
      TT_CHECK_LAUNCH();
      return TT_OK;
    }
  }
  if (pl.sample_tile_max) {
    const size_t sm = (size_t)pl.sample_slots * SEL_WQ * sizeof(float);
    TT_CHECK_CUDA(cudaFuncSetAttribute(select_threshold_tile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
    TT_CHECK_CUDA(launch_pdl(select_threshold_tile_kernel, dim3((nq + SEL_WQ - 1) / SEL_WQ), dim3(SEL_WQ * 32), sm, st,
                             (const float*)sample_buf, pl.sample_slots, pl.nq_pad, nq,
                             topr ? min(pl.sample_rank, SHARD_TOPR) : pl.sample_rank, thr, topr, (int)SHARD_TOPR));
  } else {
    // chunk maxima: more than 4096 values per query (up to 4096 took the radix select above)
    TT_CHECK_ARG(topr == nullptr, "top-r lists need the tile sampling mode");
    const int nvals = pl.sample_slots * CHUNKS;
    int npad = 1;
    while (npad < nvals) npad <<= 1;
    const size_t sm = (size_t)npad * sizeof(float);
    TT_CHECK_CUDA(cudaFuncSetAttribute(select_threshold_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
    TT_CHECK_CUDA(launch_pdl(select_threshold_kernel, dim3(nq), dim3(256), sm, st, (const float*)sample_buf, nvals, npad,
                             pl.sample_rank, thr));
  }
  TT_CHECK_LAUNCH();
  return TT_OK;
}

int launch_select_gathered(const float* topr_g, int G, int nq, int r, float* thr, int* zero_me, cudaStream_t st) {
  const size_t sm = (size_t)SEL_WQ * G * SHARD_TOPR * sizeof(float);
  TT_CHECK_CUDA(cudaFuncSetAttribute(select_threshold_gathered_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
  select_threshold_gathered_kernel<<<(nq + SEL_WQ - 1) / SEL_WQ, SEL_WQ * 32, sm, st>>>(topr_g, G, nq, r, thr, zero_me);
  TT_CHECK_LAUNCH();
  return TT_OK;
}

int launch_main_scan(const ScanPlan& pl, const void* qh, const void* Xh, long long N, int nq, float* thr,
                     unsigned int* seg_cnt, void* cand, cudaStream_t st, const float* sel_sample, const LabelArgs& lab) {
  CUtensorMap tq, tx;
  FilterScanParams sp;
  if (int e = make_scan_params(pl, qh, Xh, N, nq, thr, seg_cnt, cand, nullptr, lab, &tq, &tx, &sp)) return e;
  sp.num_slots = pl.num_tiles; sp.tile_stride = 1; sp.nslices = pl.main_slices;
  if (sel_sample) {       // thresholds selected in the kernel's prologue from the sample pass's maxima
    sp.sel_sample = sel_sample; sp.thr_out = thr;
    sp.sel_n = pl.sample_tile_max ? pl.sample_slots : pl.sample_slots * CHUNKS;
    sp.sel_ld = pl.nq_pad; sp.sel_rank = pl.sample_rank; sp.sel_query_major = pl.sample_tile_max ? 0 : 1;
  }
  profile_scan_begin(st);
  const int e = launch_scan_mode<false>(pl, tq, tx, sp, pl.main_slices * pl.nqu, st);
  profile_scan_end(st);
  return e;
}

int launch_scan(const ScanPlan& pl, const void* qh, const void* Xh, long long N, int nq,
                float* thr, unsigned int* seg_cnt, void* cand, float* sample_buf, cudaStream_t st, const LabelArgs& lab) {
  bool fold = false;
  if (pl.use_threshold) {
    fold = fold_select(pl, nq);
    if (int e = launch_sample(pl, qh, Xh, N, nq, thr, nullptr, sample_buf, st, fold, lab)) return e;
  } else {
    count_launch();
    TT_CHECK_CUDA(launch_pdl(fill_kernel, dim3((nq + 255) / 256), dim3(256), 0, st, thr, nq, -INFINITY));
  }
  return launch_main_scan(pl, qh, Xh, N, nq, thr, seg_cnt, cand, st, fold ? sample_buf : nullptr, lab);
}

// Plan of one shard of a catalog of N_total rows: tiling and slicing follow the shard, the sampling
// decisions (stride, rank, candidate target) follow the WHOLE catalog so that every rank samples the
// same fraction of its rows and the gathered sample is the sample a single device would have drawn.
ScanPlan make_shard_plan(long long N_local, long long N_total, int D, int nq, int K, bool* global_ok) {
  ScanPlan pl = make_scan_plan(N_local, D, nq, K);
  const ScanPlan gp = make_scan_plan(N_total, D, nq, K);
  *global_ok = pl.supported && gp.use_threshold && !gp.route_exact && gp.sample_tile_max &&
               gp.sample_rank <= SHARD_TOPR && N_local >= K;
  if (!*global_ok) return pl;
  pl.use_threshold = true;
  pl.route_exact = false;
  pl.target = gp.target;
  pl.sample_stride = gp.sample_stride;
  pl.sample_slots = (pl.num_tiles + gp.sample_stride - 1) / gp.sample_stride;
  pl.sample_rank = gp.sample_rank;
  pl.sample_tile_max = true;
  pl.cand_cap = gp.cand_cap;
  const int cap_units = pl.pair ? num_sms() / 2 : num_sms();
  pl.sample_slices = pick_slices(pl.nqu, cap_units, pl.sample_slots);
  // a shard may hold every candidate of a query (clustered catalogs): size its segments for the whole target
  const long long slice_rows = ((long long)(pl.num_tiles + pl.main_slices - 1) / pl.main_slices) * BLOCK_N;
  long long seg = 4LL * pl.target / pl.main_slices;
  if (seg < 512) seg = 512;
  if (seg > pl.cand_cap) seg = pl.cand_cap;
  if (seg > slice_rows) seg = slice_rows;
  pl.seg_cap = (int)((seg + 63) / 64 * 64);
  return pl;
}

}  // namespace tt
