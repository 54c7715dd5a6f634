// Fused attention pooling of the buyer tower (reference: src/models/buyer_tower.py:70-101):
//     logit_s = W2 . relu(W1 x_s + b1) + b2 ;  a = softmax_s(logit * w) ;  out = normalize(sum_s a_s x_s)
// ONE kernel, ONE pass over x in HBM: the score MLP runs on the tensor cores while the rows stream in, and
// the softmax-weighted sum re-reads the same rows a few microseconds later, when they are still in L2.
//
// Arithmetic of the hidden layer (fp32-accurate, like the 3xTF32 kernel it replaces, at twice the tensor
// rate and half the operand bytes): every fp32 operand is split into two fp16 pieces, v*2^e = hi + lo with
// hi = rn_f16(v*2^e), lo = rn_f16(v*2^e - hi)  (22 significant bits; 2^e is a power of two chosen so that
// `lo` stays a normal fp16: 16 for x, from max|W1| for the weights), and
//     x.w ~= hi_x.hi_w + hi_x.lo_w + lo_x.hi_w          (dropped lo.lo term ~2^-22 relative)
// is accumulated in fp32 in TMEM by three tcgen05.mma kind::f16 per K step; the epilogue undoes 2^e.
// The tensor core TRUNCATES (round toward zero) when it adds into the accumulator: 72 updates of one accumulator
// bias the hidden pre-activations by ~6e-6 relative, which the event weight (up to 10) turns into 1.2e-5 element-wise
// on the pooled output (measured; reproduced by a numpy model of truncating accumulation).  So the large hi.hi
// products go to one accumulator (24 updates) and the two cross terms, 2^-11 smaller, to a second one; the epilogue
// adds the two in fp32.  Measured/modelled error of the pooled output: 4e-6 element-wise, 1e-6 norm-wise - the level
// of an fp32 sgemm.
// A value outside the fp16 range after scaling (|x| > 4094, or a non-finite input) raises a device flag and a
// predicated fp32 CUDA-core kernel recomputes the call: no host synchronisation, always the fp32 answer.
//
// Orientation: D[hidden(128) x rows(64)] = W1 . x^T.  The A operand W1 (hi and lo, 2 x 192 TMEM columns for
// D = 384) is written ONCE per CTA into tensor memory (tcgen05.st) and never touches shared memory again;
// the B operand (64 rows of x, hi and lo fp16 tiles) is the only MMA operand read from shared memory
// (64 B/cycle while the tensor pipe is busy).  L2->SM traffic is x twice (TMA + pooling re-read), nothing else.
//
// Persistent CTAs (one per SM, 20 warps); CTA c owns a contiguous range of buyers and walks its rows in 64-row tiles:
//   warp 0 lane 0   : TMA producer  - raw fp32 [64 rows x 64 cols] (two 128B-swizzled boxes) per K-block, 6-stage ring;
//                                     with the L2 evict_last hint when pooling (the pooling warps re-read the rows)
//   warps 8-11      : splitters     - raw fp32 -> scaled fp16 hi/lo tiles in the UMMA K-major 128B-swizzle layout
//                                     (3-stage ring), fence.proxy.async, arrive
//   warp 1 lane 0   : MMA issuer    - per K-block 4 K-steps x 3 MMAs (M = 128 hidden, N = 64 rows, K = 16) into the main
//                                     and the cross-term accumulator (2 x 64 TMEM columns; the kernel is HBM-bound, the
//                                     tensor pipe may idle while the epilogue reads them)
//   warps 4-7       : epilogue      - lane = hidden unit: relu(acc*2^-e + b1)*W2, butterfly transpose-reduce over
//                                     the 128 hidden units -> one logit per row into a shared-memory array
//   warps 12-19     : pooling       - one warp per buyer, as soon as the tile holding the buyer's last row is done:
//                                     softmax of logit*weight, weighted row sum (128-bit loads, L2 hits), L2 normalise
//   warp 2          : TMEM allocator
// Rooflines: HBM (x once: B*S*D*4 bytes); tensor pipe 3 x 2*D*128 flop per row at the fp16 rate; shared memory
// ~6.9 KB per row (TMA write, splitter read + write, MMA B reads).
#include <cuda.h>
#include <cuda_fp16.h>
#include <math.h>
#include "tt_common.cuh"
#include "sm100_ptx.cuh"
#include "flat_internal.cuh"

namespace tt {

using namespace ptx;

constexpr int AF_TILE = 64;                          // rows of x per MMA tile (UMMA N)
constexpr int AF_M = 128;                            // hidden units (UMMA M); H <= 128
constexpr int AF_RAW_STAGE = 2 * AF_TILE * 128;      // two fp32 boxes [64 rows x 32 cols] = 16 KB
constexpr int AF_B_STAGE = 2 * AF_TILE * 128;        // fp16 hi tile + lo tile [64 rows x 64 cols] = 16 KB
constexpr int AF_RAW_STAGES = 6;
constexpr int AF_B_STAGES = 3;
constexpr int AF_RMAX = 8192;                        // rows (logits) one CTA may own per launch
constexpr int AF_MAX_KB = 6;                         // D <= 384: W hi + lo = 2 * 6 * 32 = 384 TMEM columns
constexpr int AF_SPLIT_WARPS = 4;
constexpr int AF_POOL_WARPS = 8;                     // the re-read must keep pace with the stream or it falls out of L2
constexpr int AF_POOL_WARP0 = 8 + AF_SPLIT_WARPS;
constexpr int AF_WARPS = 20;
constexpr int AF_THREADS = AF_WARPS * 32;
constexpr int AF_ACC_COLS = 128;                     // main + cross-term accumulator (64 columns each), then W hi, W lo
constexpr float AF_X_SCALE = 16.0f;
constexpr float AF_F16_MAX = 65504.0f;

struct AttnFusedParams {
  const float* x;          // [R, D]
  const float* w;          // [B, S]       (pool mode)
  float* out;              // [B, D]       (pool mode)
  float* logits_out;       // [R]          (logits-only mode)
  const uint4* Wp;         // [2][nkb][8][128] uint4: fp16 pieces of W1 * 2^kw, 8 K elements per uint4, by hidden unit
  const float* b1;
  const float* W2;
  const float* b2;
  const float* inv_scale;  // 2^-(kw + 4), written by the weight-preparation kernel
  int* flag;               // raised when a value leaves the fp16 range
  long long R;
  int B, S, D, H, nkb;
};

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ unsigned int ld_acquire_cta_shared(const unsigned int* p) {
  unsigned int v;
  asm volatile("ld.acquire.cta.shared::cta.u32 %0, [%1];" : "=r"(v) : "r"(smem_u32(p)) : "memory");
  return v;
}
__device__ __forceinline__ void red_release_cta_shared_add(unsigned int* p, unsigned int v) {
  asm volatile("red.release.cta.shared::cta.add.u32 [%0], %1;" ::"r"(smem_u32(p)), "r"(v) : "memory");
}
__device__ __forceinline__ void fence_proxy_async_shared() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// 8 consecutive fp32 (already scaled) -> 8 fp16 `hi` + 8 fp16 `lo`
__device__ __forceinline__ void split8(const float4 a, const float4 b, uint4& hi, uint4& lo, float& mabs) {
  const float v[8] = {a.x * AF_X_SCALE, a.y * AF_X_SCALE, a.z * AF_X_SCALE, a.w * AF_X_SCALE,
                      b.x * AF_X_SCALE, b.y * AF_X_SCALE, b.z * AF_X_SCALE, b.w * AF_X_SCALE};
  uint32_t h[4], l[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const __half2 hh = __floats2half2_rn(v[2 * i], v[2 * i + 1]);
    const float2 back = __half22float2(hh);
    const __half2 ll = __floats2half2_rn(v[2 * i] - back.x, v[2 * i + 1] - back.y);
    h[i] = *reinterpret_cast<const uint32_t*>(&hh);
    l[i] = *reinterpret_cast<const uint32_t*>(&ll);
    mabs = fmaxf(mabs, fmaxf(fabsf(v[2 * i]), fabsf(v[2 * i + 1])));
    if (!(fabsf(v[2 * i]) <= AF_F16_MAX) || !(fabsf(v[2 * i + 1]) <= AF_F16_MAX)) mabs = INFINITY;   // NaN too
  }
  hi = make_uint4(h[0], h[1], h[2], h[3]);
  lo = make_uint4(l[0], l[1], l[2], l[3]);
}

template <bool POOL>
__global__ void __launch_bounds__(AF_THREADS, 1)
attn_pool_fused_kernel(const __grid_constant__ CUtensorMap tmap_x, const AttnFusedParams p) {
  extern __shared__ uint8_t smem_raw_[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw_) + 1023) & ~(uintptr_t)1023);
  uint8_t* raw_ring = smem;
  uint8_t* b_ring = raw_ring + AF_RAW_STAGES * AF_RAW_STAGE;
  float* logits_s = reinterpret_cast<float*>(b_ring + AF_B_STAGES * AF_B_STAGE);      // [AF_RMAX]
  float* partial = logits_s + AF_RMAX;                                                 // [2][4][64]
  uint64_t* bars = reinterpret_cast<uint64_t*>(partial + 2 * 4 * AF_TILE);
  uint64_t* full_raw = bars;                              // [AF_RAW_STAGES]  TMA landed
  uint64_t* empty_raw = full_raw + AF_RAW_STAGES;         // [AF_RAW_STAGES]  one arrival per splitter warp
  uint64_t* full_b = empty_raw + AF_RAW_STAGES;           // [AF_B_STAGES]    one arrival per splitter warp
  uint64_t* empty_b = full_b + AF_B_STAGES;               // [AF_B_STAGES]    tcgen05.commit
  uint64_t* tmem_full = empty_b + AF_B_STAGES;            // [2]
  uint64_t* tmem_empty = tmem_full + 2;                   // [2]  one arrival per epilogue warp
  uint64_t* w_bar = tmem_empty + 2;                       // [1]  W1 pieces are in TMEM (one arrival per epilogue warp)
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(w_bar + 1);
  unsigned int* done_cnt = tmem_ptr_smem + 1;             // += 1 per logits-writing warp per finished tile

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  // ---- this CTA's buyers / rows -------------------------------------------------------------------
  const int b0 = (int)((long long)blockIdx.x * p.B / gridDim.x);
  const int b1 = (int)((long long)(blockIdx.x + 1) * p.B / gridDim.x);
  const long long r0 = (long long)b0 * p.S;
  const int nrows = (b1 - b0) * p.S;
  const int ntiles = (nrows + AF_TILE - 1) / AF_TILE;
  const int nkb = p.nkb;

  if (warp == 0 && lane == 0) prefetch_tensormap(&tmap_x);
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < AF_RAW_STAGES; ++i) { mbar_init(smem_u32(full_raw + i), 1); mbar_init(smem_u32(empty_raw + i), AF_SPLIT_WARPS); }
    for (int i = 0; i < AF_B_STAGES; ++i) { mbar_init(smem_u32(full_b + i), AF_SPLIT_WARPS); mbar_init(smem_u32(empty_b + i), 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(smem_u32(tmem_full + i), 1); mbar_init(smem_u32(tmem_empty + i), 4); }
    mbar_init(smem_u32(w_bar), 4);
    *done_cnt = 0u;
    fence_barrier_init();
  }
  if (warp == 2) { tmem_alloc(smem_u32(tmem_ptr_smem), 512); tmem_relinquish(); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  const uint32_t w_hi_col = AF_ACC_COLS, w_lo_col = AF_ACC_COLS + (uint32_t)nkb * 32u;

  if (warp == 0) {
    // =========================== TMA producer =====================================================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int t = 0; t < ntiles; ++t) {
        const int row = (int)(r0 + (long long)t * AF_TILE);
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(smem_u32(empty_raw + stage), phase ^ 1, 500 + stage);
          const uint32_t fb = smem_u32(full_raw + stage);
          const uint32_t dst = smem_u32(raw_ring + (size_t)stage * AF_RAW_STAGE);
          mbar_arrive_expect_tx(fb, (uint32_t)AF_RAW_STAGE);
          if (POOL) {         // the rows are read again by the pooling warps: ask L2 to keep them (evict_last)
            tma_load_2d_hint(dst, &tmap_x, fb, kb * 64, row, kEvictLast);
            tma_load_2d_hint(dst + AF_RAW_STAGE / 2, &tmap_x, fb, kb * 64 + 32, row, kEvictLast);
          } else {
            tma_load_2d(dst, &tmap_x, fb, kb * 64, row);
            tma_load_2d(dst + AF_RAW_STAGE / 2, &tmap_x, fb, kb * 64 + 32, row);
          }
          if (++stage == AF_RAW_STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // =========================== MMA issuer =======================================================
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc_f16_f32(AF_M, AF_TILE);
      mbar_wait(smem_u32(w_bar), 0, 510);
      tc_fence_after();
      int stage = 0;
      uint32_t phase = 0;
      for (int t = 0; t < ntiles; ++t) {
        mbar_wait(smem_u32(tmem_empty), ((uint32_t)t & 1u) ^ 1u, 520);
        tc_fence_after();
        const uint32_t d_main = tmem_base, d_cross = tmem_base + (uint32_t)AF_TILE;
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(smem_u32(full_b + stage), phase, 530 + stage);
          tc_fence_after();
          const uint64_t xh = make_smem_desc_sw128(smem_u32(b_ring + (size_t)stage * AF_B_STAGE));
          const uint64_t xl = make_smem_desc_sw128(smem_u32(b_ring + (size_t)stage * AF_B_STAGE + AF_B_STAGE / 2));
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const uint64_t koff = (uint64_t)((k * 16 * 2) >> 4);               // 32 bytes per K = 16 step
            const uint32_t a_hi = tmem_base + w_hi_col + (uint32_t)((kb * 4 + k) * 8);
            const uint32_t a_lo = tmem_base + w_lo_col + (uint32_t)((kb * 4 + k) * 8);
            const uint32_t first = (uint32_t)((kb | k) != 0);
            mma_f16_ts(d_main, a_hi, xh + koff, idesc, first);                 // hi.hi   -> main accumulator
            mma_f16_ts(d_cross, a_lo, xh + koff, idesc, first);                // lo_w.hi_x
            mma_f16_ts(d_cross, a_hi, xl + koff, idesc, 1u);                   // hi_w.lo_x -> cross accumulator
          }
          mma_commit(smem_u32(empty_b + stage));
          if (kb == nkb - 1) mma_commit(smem_u32(tmem_full));
          if (++stage == AF_B_STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
    __syncwarp();
  } else if (warp >= 4 && warp < 8) {
    // =========================== epilogue: lane = hidden unit ========================================
    const int e = warp - 4;                      // TMEM lane quadrant
    const int h = e * 32 + lane;
    const uint32_t lane_base = tmem_base + ((uint32_t)(e * 32) << 16);
    pdl_wait();      // the weight-preparation kernel (previous launch) has written Wp / inv_scale / flag
    // one-time: this CTA's copy of the W1 pieces into tensor memory (A operand of every MMA)
    for (int j = 0; j < 2 * nkb; ++j) {
      const uint4* src = p.Wp + (size_t)j * 8 * AF_M + h;
      uint32_t r[32];
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        const uint4 v = __ldg(src + q * AF_M);
        r[4 * q] = v.x; r[4 * q + 1] = v.y; r[4 * q + 2] = v.z; r[4 * q + 3] = v.w;
      }
      __syncwarp();
      tmem_st_32x32(lane_base + w_hi_col + (uint32_t)(j * 32), r);
    }
    tmem_st_wait();
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(smem_u32(w_bar));

    const float b1h = (h < p.H) ? __ldg(p.b1 + h) : 0.f;
    const float w2h = (h < p.H) ? __ldg(p.W2 + h) : 0.f;
    const float sc = __ldg(p.inv_scale);
    const float b2v = __ldg(p.b2);
    for (int t = 0; t < ntiles; ++t) {
      mbar_wait(smem_u32(tmem_full), (uint32_t)t & 1u, 540);
      tc_fence_after();
      float* part = partial + (size_t)(t & 1) * 4 * AF_TILE + e * AF_TILE;
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        uint32_t v[32], c[32];
        __syncwarp();
        tmem_ld_32x32(lane_base + (uint32_t)(half * 32), v);                     // main accumulator
        tmem_ld_32x32(lane_base + (uint32_t)(AF_TILE + half * 32), c);           // cross terms
        tmem_ld_wait();
        if (half == 1) {                          // everything is in registers: hand the accumulators back
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(smem_u32(tmem_empty));
        }
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] = __float_as_uint(__uint_as_float(v[i]) + __uint_as_float(c[i]));
        float tv[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) tv[i] = w2h * fmaxf(fmaf(__uint_as_float(v[i]), sc, b1h), 0.f);
        // butterfly transpose-reduce: afterwards lane l holds the sum over the warp's 32 hidden units of column l
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) {
          const bool upper = (lane & off) != 0;
#pragma unroll
          for (int i = 0; i < off; ++i) {
            const float send = upper ? tv[i] : tv[i + off];
            const float keep = upper ? tv[i + off] : tv[i];
            tv[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
          }
        }
        part[half * 32 + lane] = tv[0];
      }
      named_bar_sync(1, 128);                     // the four partial sums of every column are in shared memory
      if (e < 2) {
        const int n = e * 32 + lane;
        const float* pp = partial + (size_t)(t & 1) * 4 * AF_TILE + n;
        const float logit = ((pp[0] + pp[AF_TILE]) + pp[2 * AF_TILE]) + pp[3 * AF_TILE] + b2v;
        const int rl = t * AF_TILE + n;
        if (rl < nrows) {
          if (POOL) logits_s[rl] = logit;
          else p.logits_out[r0 + rl] = logit;
        }
        if (POOL) {
          __syncwarp();
          if (lane == 0) red_release_cta_shared_add(done_cnt, 1u);
        }
      }
    }
  } else if (warp >= 8 && warp < 8 + AF_SPLIT_WARPS) {
    // =========================== splitters ==========================================================
    const int tid = (warp - 8) * 32 + lane;                    // 0..127
    int rstage = 0, bstage = 0;
    uint32_t rphase = 0, bphase = 0;
    float mabs = 0.f;
    const int nsteps = ntiles * nkb;
    for (int n = 0; n < nsteps; ++n) {
      mbar_wait(smem_u32(full_raw + rstage), rphase, 550 + rstage);
      const uint8_t* raw = raw_ring + (size_t)rstage * AF_RAW_STAGE;
      constexpr int UPT = 512 / (AF_SPLIT_WARPS * 32);           // 32-byte units per thread per stage
      float4 fa[UPT], fb[UPT];
      int row[UPT], cpos[UPT];
#pragma unroll
      for (int i = 0; i < UPT; ++i) {
        const int u = tid + AF_SPLIT_WARPS * 32 * i;
        row[i] = u >> 3;
        const int sub = u & 7, box = sub >> 2, j = sub & 3;
        const int x7 = row[i] & 7;
        const int p0 = (2 * j) ^ x7, p1 = p0 ^ 1;                  // swizzled slots of raw chunks 2j and 2j+1
        const uint8_t* a0 = raw + box * (AF_RAW_STAGE / 2) + row[i] * 128;
        // box-1 lanes read the odd chunk first: the 8 lanes of a quarter-warp then touch 8 distinct 16-byte slots
        const float4 first = *reinterpret_cast<const float4*>(a0 + (box ? p1 : p0) * 16);
        const float4 second = *reinterpret_cast<const float4*>(a0 + (box ? p0 : p1) * 16);
        fa[i] = box ? second : first;                              // raw chunk 2j   (columns 8j .. 8j+3 of the box)
        fb[i] = box ? first : second;                              // raw chunk 2j+1 (columns 8j+4 .. 8j+7)
        cpos[i] = ((4 * box + j) ^ x7) * 16;                       // slot of fp16 chunk c = 4*box + j in its row
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(empty_raw + rstage));    // values are in registers: the raw stage is free
      if (++rstage == AF_RAW_STAGES) { rstage = 0; rphase ^= 1; }
      mbar_wait(smem_u32(empty_b + bstage), bphase ^ 1, 560 + bstage);
      uint8_t* hi_tile = b_ring + (size_t)bstage * AF_B_STAGE;
      uint8_t* lo_tile = hi_tile + AF_B_STAGE / 2;
#pragma unroll
      for (int i = 0; i < UPT; ++i) {
        uint4 hi, lo;
        split8(fa[i], fb[i], hi, lo, mabs);
        *reinterpret_cast<uint4*>(hi_tile + row[i] * 128 + cpos[i]) = hi;
        *reinterpret_cast<uint4*>(lo_tile + row[i] * 128 + cpos[i]) = lo;
      }
      fence_proxy_async_shared();        // generic-proxy writes -> visible to the tensor core's async-proxy reads
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(full_b + bstage));
      if (++bstage == AF_B_STAGES) { bstage = 0; bphase ^= 1; }
    }
    pdl_wait();      // ... and cleared the flag
    if (!(mabs <= AF_F16_MAX)) atomicOr(p.flag, 1);
  } else if (POOL && warp >= AF_POOL_WARP0) {
    // =========================== pooling: one warp per buyer ==========================================
    const int pw = warp - AF_POOL_WARP0;
    const int S = p.S, D = p.D;
    const int nvalid4 = D >> 2;
    constexpr int NV = 3, U = 4;
    for (int b = b0 + pw; b < b1; b += AF_POOL_WARPS) {
      const int rl0 = (b - b0) * S;
      const unsigned int need = 2u * (unsigned int)((rl0 + S - 1) / AF_TILE + 1);
      if (lane == 0) {
        while (ld_acquire_cta_shared(done_cnt) < need) __nanosleep(100);
      }
      __syncwarp();
      const float* lg = logits_s + rl0;
      const float* wb = p.w + (long long)b * S;
      // ---- softmax normaliser (buyer_tower.py:89-92) -----------------------------------------------
      float m = -INFINITY, tot = 0.f;
      for (int s = lane; s < S; s += 32) m = fmaxf(m, lg[s] * __ldg(wb + s));
      m = warp_max(m);
      for (int s = lane; s < S; s += 32) tot += expf(lg[s] * __ldg(wb + s) - m);
      tot = warp_sum(tot);
      // ---- weighted row sum (buyer_tower.py:96) ----------------------------------------------------
      float4 acc[NV];
#pragma unroll
      for (int v = 0; v < NV; ++v) acc[v] = make_float4(0.f, 0.f, 0.f, 0.f);
      const float4* xb = reinterpret_cast<const float4*>(p.x + ((long long)b * S) * D);
      for (int s0 = 0; s0 < S; s0 += 32) {
        const int s = s0 + lane;
        const float coef = (s < S) ? expf(lg[s] * __ldg(wb + s) - m) / tot : 0.f;
        const int nrow = min(32, S - s0);
        for (int j0 = 0; j0 < nrow; j0 += U) {
          float4 buf[U][NV];
          float cf[U];
#pragma unroll
          for (int u = 0; u < U; ++u) {
            const int j = j0 + u;
            const bool ok = j < nrow;
            cf[u] = ok ? __shfl_sync(0xffffffffu, coef, ok ? j : 0) : 0.f;
            const float4* rp = xb + (long long)(s0 + (ok ? j : 0)) * nvalid4;
#pragma unroll
            for (int v = 0; v < NV; ++v) {
              const int c4 = v * 32 + lane;
              buf[u][v] = (ok && c4 < nvalid4) ? ldg_stream(rp + c4) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
          }
#pragma unroll
          for (int u = 0; u < U; ++u) {
#pragma unroll
            for (int v = 0; v < NV; ++v) {
              acc[v].x = fmaf(buf[u][v].x, cf[u], acc[v].x);
              acc[v].y = fmaf(buf[u][v].y, cf[u], acc[v].y);
              acc[v].z = fmaf(buf[u][v].z, cf[u], acc[v].z);
              acc[v].w = fmaf(buf[u][v].w, cf[u], acc[v].w);
            }
          }
        }
      }
      // ---- F.normalize(p=2, dim=1, eps=1e-12) (buyer_tower.py:99) ------------------------------------
      float ss = 0.f;
#pragma unroll
      for (int v = 0; v < NV; ++v)
        ss += acc[v].x * acc[v].x + acc[v].y * acc[v].y + acc[v].z * acc[v].z + acc[v].w * acc[v].w;
      ss = warp_sum(ss);
      const float denom = fmaxf(sqrtf(ss), 1e-12f);
      float4* op = reinterpret_cast<float4*>(p.out + (long long)b * D);
#pragma unroll
      for (int v = 0; v < NV; ++v) {
        const int c4 = v * 32 + lane;
        if (c4 < nvalid4) op[c4] = make_float4(acc[v].x / denom, acc[v].y / denom, acc[v].z / denom, acc[v].w / denom);
      }
    }
  }

  // ---- teardown -----------------------------------------------------------------------------------
  tc_fence_before();
  __syncthreads();
  if (warp == 2) { tc_fence_after(); tmem_dealloc(tmem_base, 512); }
}

// W1 f32 [H, D] -> fp16 pieces of W1 * 2^kw laid out for the epilogue threads' coalesced loads:
//   Wp[part][kb][q][m] (uint4 = 8 consecutive K elements k = kb*64 + q*8 .. +7 of hidden unit m; part 0 = hi, 1 = lo)
// kw puts max|W1| * 2^kw into [8192, 16384), so that `lo` (2^-11 of `hi`) stays a normal fp16.  Every block reduces
// max|W1| over the whole (L2-resident, 196 KB) matrix itself - cheaper than a second launch - and then converts its
// share: one thread per (hidden unit, 8 consecutive k), i.e. 32-byte coalesced reads.
constexpr int AF_PREP_THREADS = 256;
__global__ void __launch_bounds__(AF_PREP_THREADS)
attn_fused_prep_w_kernel(const float* __restrict__ W1, int H, int D, int nkb, uint4* __restrict__ Wp,
                         float* __restrict__ inv_scale, int* __restrict__ flag) {
  __shared__ float red[AF_PREP_THREADS / 32];
  __shared__ float s_scale;
  float m = 0.f;
  bool bad = false;
  const int n = H * D;
  if ((n & 3) == 0 && (reinterpret_cast<uintptr_t>(W1) & 15) == 0) {
    const float4* w4 = reinterpret_cast<const float4*>(W1);
    for (int i = threadIdx.x; i < (n >> 2); i += blockDim.x) {
      const float4 v = __ldg(w4 + i);
      const float a = fmaxf(fmaxf(fabsf(v.x), fabsf(v.y)), fmaxf(fabsf(v.z), fabsf(v.w)));
      if (!(fabsf(v.x) <= 3.0e38f) || !(fabsf(v.y) <= 3.0e38f) || !(fabsf(v.z) <= 3.0e38f) || !(fabsf(v.w) <= 3.0e38f)) bad = true;
      m = fmaxf(m, a);
    }
  } else {
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
      const float a = fabsf(__ldg(W1 + i));
      if (!(a <= 3.0e38f)) bad = true;
      m = fmaxf(m, a);
    }
  }
  m = warp_max(m);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
  const int anybad = __syncthreads_or(bad ? 1 : 0);
  if (threadIdx.x == 0) {
    float mm = 0.f;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) mm = fmaxf(mm, red[i]);
    int e = 0;
    float scale = 1.f;
    if (mm > 0.f && !anybad) { (void)frexpf(mm, &e); scale = ldexpf(1.f, 14 - e); }     // mm = f * 2^e, f in [0.5, 1)
    s_scale = scale;
    if (blockIdx.x == 0) {
      *inv_scale = 1.0f / (scale * AF_X_SCALE);
      *flag = anybad ? 1 : 0;             // also clears the flag for this call
    }
  }
  __syncthreads();
  const float scale = s_scale;
  const int k8n = nkb * 8;                                  // groups of 8 consecutive k per hidden unit
  const int units = AF_M * k8n;
  for (int u = blockIdx.x * blockDim.x + threadIdx.x; u < units; u += gridDim.x * blockDim.x) {
    const int mrow = u / k8n, k8 = u % k8n;
    const int kb = k8 >> 3, q = k8 & 7;
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int k = k8 * 8 + j;
      v[j] = (mrow < H && k < D) ? __ldg(W1 + (size_t)mrow * D + k) * scale : 0.f;
    }
    uint32_t hi[4], lo[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const __half2 hh = __floats2half2_rn(v[2 * j], v[2 * j + 1]);
      const float2 back = __half22float2(hh);
      const __half2 ll = __floats2half2_rn(v[2 * j] - back.x, v[2 * j + 1] - back.y);
      hi[j] = *reinterpret_cast<const uint32_t*>(&hh);
      lo[j] = *reinterpret_cast<const uint32_t*>(&ll);
    }
    Wp[((size_t)(0 * nkb + kb) * 8 + q) * AF_M + mrow] = make_uint4(hi[0], hi[1], hi[2], hi[3]);
    Wp[((size_t)(1 * nkb + kb) * 8 + q) * AF_M + mrow] = make_uint4(lo[0], lo[1], lo[2], lo[3]);
  }
}

// Predicated fp32 recomputation (CUDA cores, one CTA per buyer): runs only when the fused kernel found a value
// outside the fp16 range.  Plain fp32 FMA arithmetic of buyer_tower.py:85-99; speed is irrelevant here.
__global__ void __launch_bounds__(256)
attn_pool_fallback_kernel(const float* __restrict__ x, const float* __restrict__ w, const float* __restrict__ W1,
                          const float* __restrict__ b1, const float* __restrict__ W2, const float* __restrict__ b2,
                          int H, float* __restrict__ out, int B, int S, int D, const int* __restrict__ flag) {
  pdl_wait();
  if (*flag == 0) return;
  extern __shared__ float fsm[];
  float* lg = fsm;                 // [S]
  float* hsum = fsm + S;           // [8] per-warp partial logits
  __shared__ float bc[2];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int b = blockIdx.x; b < B; b += gridDim.x) {
  const float* xb = x + (long long)b * S * D;
  for (int s = 0; s < S; ++s) {
    const float* row = xb + (long long)s * D;
    float part = 0.f;
    for (int h = warp; h < H; h += 8) {
      float a = 0.f;
      for (int d = lane; d < D; d += 32) a = fmaf(__ldg(row + d), __ldg(W1 + (long long)h * D + d), a);
      a = warp_sum(a);
      part = fmaf(fmaxf(a + __ldg(b1 + h), 0.f), __ldg(W2 + h), part);
    }
    if (lane == 0) hsum[warp] = part;
    __syncthreads();
    if (tid == 0) {
      float t = 0.f;
      for (int i = 0; i < 8; ++i) t += hsum[i];
      lg[s] = (t + __ldg(b2)) * __ldg(w + (long long)b * S + s);
    }
    __syncthreads();
  }
  if (tid == 0) {
    float m = -INFINITY, tot = 0.f;
    for (int s = 0; s < S; ++s) m = fmaxf(m, lg[s]);
    for (int s = 0; s < S; ++s) tot += expf(lg[s] - m);
    bc[0] = m; bc[1] = tot;
  }
  __syncthreads();
  const float m = bc[0], tot = bc[1];
  float ss = 0.f;
  for (int d = tid; d < D; d += blockDim.x) {
    float a = 0.f;
    for (int s = 0; s < S; ++s) a = fmaf(__ldg(xb + (long long)s * D + d), expf(lg[s] - m) / tot, a);
    out[(long long)b * D + d] = a;
    ss += a * a;
  }
  ss = warp_sum(ss);
  __syncthreads();
  if (lane == 0) hsum[warp] = ss;
  __syncthreads();
  if (tid == 0) { float t = 0.f; for (int i = 0; i < 8; ++i) t += hsum[i]; bc[0] = fmaxf(sqrtf(t), 1e-12f); }
  __syncthreads();
  const float denom = bc[0];
  for (int d = tid; d < D; d += blockDim.x) out[(long long)b * D + d] /= denom;
  __syncthreads();
  }
}

struct FusedWs { size_t wp, meta, total; };
static FusedWs fused_ws_layout(int nkb) {
  FusedWs w{};
  w.wp = 0;
  w.meta = align_up((size_t)2 * nkb * 8 * AF_M * sizeof(uint4), 256);
  w.total = w.meta + 256;
  return w;
}

static bool fused_shape_ok(const float* x, const float* out, long long B, long long S, int D, int H) {
  return D % 64 == 0 && D <= 64 * AF_MAX_KB && H >= 1 && H <= AF_M && S >= 1 && S <= AF_RMAX && B * S >= 64 &&
         B * S < (1LL << 31) && ((reinterpret_cast<uintptr_t>(x) & 15) == 0) && ((reinterpret_cast<uintptr_t>(out) & 15) == 0);
}

// Logits-only mode (tt_attention_logits; e.g. once over the whole catalog for the gather path): the same kernel without
// the pooling warps, logits written to global memory; the weight pieces live in a stream-ordered scratch block.  Nothing
// re-reads the rows, so the TMA loads carry no L2 evict_last hint.
int launch_attn_logits_fused(const float* x, long long R, int D, const float* W1, const float* b1, const float* W2,
                             const float* b2, int H, float* logits, cudaStream_t st) {
  if (!(D % 64 == 0 && D <= 64 * AF_MAX_KB && H >= 1 && H <= AF_M && R >= 64 && R < (1LL << 31) &&
        (reinterpret_cast<uintptr_t>(x) & 15) == 0))
    return TT_ERR_UNSUPPORTED;
  int dev = 0;
  TT_CHECK_CUDA(cudaGetDevice(&dev));
  cudaMemPool_t pool = scratch_pool(dev);
  if (!pool) return TT_ERR_UNSUPPORTED;
  const int nkb = D / 64;
  const FusedWs lay = fused_ws_layout(nkb);
  unsigned char* ws = nullptr;
  TT_CHECK_CUDA(cudaMallocFromPoolAsync(reinterpret_cast<void**>(&ws), lay.total, pool, st));
  uint4* Wp = reinterpret_cast<uint4*>(ws + lay.wp);
  float* inv_scale = reinterpret_cast<float*>(ws + lay.meta);
  int* flag = reinterpret_cast<int*>(ws + lay.meta + 16);
  attn_fused_prep_w_kernel<<<(AF_M * nkb * 8 + AF_PREP_THREADS - 1) / AF_PREP_THREADS, AF_PREP_THREADS, 0, st>>>(W1, H, D, nkb, Wp, inv_scale, flag);
  count_launch();
  int rc = TT_OK;
  CUtensorMap tx;
  if ((rc = make_tmap_f32(&tx, x, R, D, AF_TILE, 32)) == TT_OK) {
    AttnFusedParams p{};
    p.x = x; p.logits_out = logits; p.Wp = Wp; p.b1 = b1; p.W2 = W2; p.b2 = b2; p.inv_scale = inv_scale; p.flag = flag;
    p.R = R; p.B = (int)R; p.S = 1; p.D = D; p.H = H; p.nkb = nkb;
    const size_t smem = (size_t)AF_RAW_STAGES * AF_RAW_STAGE + (size_t)AF_B_STAGES * AF_B_STAGE + AF_RMAX * sizeof(float) +
                        2 * 4 * AF_TILE * sizeof(float) + 512 + 1024;
    const long long tiles = (R + AF_TILE - 1) / AF_TILE;
    const int grid = (int)(tiles < num_sms() ? tiles : num_sms());
    cudaError_t ce = cudaFuncSetAttribute(attn_pool_fused_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (ce == cudaSuccess) { count_launch(); ce = launch_pdl(attn_pool_fused_kernel<false>, dim3(grid), dim3(AF_THREADS), smem, st, tx, p); }
    if (ce != cudaSuccess) { set_error(std::string("launch_attn_logits_fused: ") + cudaGetErrorString(ce)); rc = TT_ERR_CUDA; }
    if (rc == TT_OK) rc = launch_attn_logits_generic_if(x, R, D, W1, b1, W2, b2, H, logits, flag, st);
  }
  const cudaError_t fe = cudaFreeAsync(ws, st);
  if (rc == TT_OK && fe != cudaSuccess) { set_error("launch_attn_logits_fused: cudaFreeAsync failed"); rc = TT_ERR_CUDA; }
  return rc;
}

}  // namespace tt

using namespace tt;

extern "C" __attribute__((visibility("default"))) size_t tt_pool_attention_fused_workspace_bytes(int B, int S, int D, int H) {
  if (B < 1 || S < 1 || D < 1 || H < 1) return 0;
  const int nkb = (D + 63) / 64;
  // the fused path needs the fp16 weight pieces + a flag; other shapes run logits + pooling and need [B,S] logits
  return fused_ws_layout(nkb < 1 ? 1 : nkb).total + align_up((size_t)B * S * sizeof(float), 256);
}

extern "C" __attribute__((visibility("default"))) int tt_pool_attention_fused(const float* x, const float* w, const float* W1, const float* b1,
                                                                 const float* W2, const float* b2, int H, float* out, int B, int S,
                                                                 int D, void* workspace, size_t workspace_bytes, void* stream) {
  TT_CHECK_ARG(x && w && W1 && b1 && W2 && b2 && out && workspace, "null pointer");
  TT_CHECK_ARG(B >= 0 && S >= 1 && D >= 1 && H >= 1, "need B >= 0, S >= 1, D >= 1, H >= 1");
  TT_CHECK_ARG((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "workspace must be 256-byte aligned");
  if (B == 0) return TT_OK;
  if (workspace_bytes < tt_pool_attention_fused_workspace_bytes(B, S, D, H)) {
    set_error("tt_pool_attention_fused: workspace too small");
    return TT_ERR_WORKSPACE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  const int nkb = (D + 63) / 64;
  const FusedWs lay = fused_ws_layout(nkb);
  unsigned char* ws = reinterpret_cast<unsigned char*>(workspace);
  if (!fused_shape_ok(x, out, B, S, D, H)) {
    // shapes outside the fused kernel: logits (tensor cores when aligned, else CUDA cores) + softmax pooling
    float* logits = reinterpret_cast<float*>(ws + lay.total);
    if (int e = tt_attention_logits(x, (int64_t)B * S, D, W1, b1, W2, b2, H, logits, stream)) return e;
    return tt_pool_attention(x, logits, w, out, B, S, D, stream);
  }
  uint4* Wp = reinterpret_cast<uint4*>(ws + lay.wp);
  float* inv_scale = reinterpret_cast<float*>(ws + lay.meta);
  int* flag = reinterpret_cast<int*>(ws + lay.meta + 16);
  attn_fused_prep_w_kernel<<<(AF_M * nkb * 8 + AF_PREP_THREADS - 1) / AF_PREP_THREADS, AF_PREP_THREADS, 0, st>>>(W1, H, D, nkb, Wp, inv_scale, flag);
  TT_CHECK_LAUNCH();
  const size_t smem = (size_t)AF_RAW_STAGES * AF_RAW_STAGE + (size_t)AF_B_STAGES * AF_B_STAGE + AF_RMAX * sizeof(float) +
                      2 * 4 * AF_TILE * sizeof(float) + 512 + 1024;
  TT_CHECK_CUDA(cudaFuncSetAttribute(attn_pool_fused_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  // every launch covers at most grid * floor(AF_RMAX / S) buyers (a CTA keeps its rows' logits in shared memory)
  const int sms = num_sms();
  const long long per_cta = AF_RMAX / S;
  for (long long bdone = 0; bdone < B;) {
    const long long nb = (B - bdone < per_cta * sms) ? (B - bdone) : per_cta * sms;
    CUtensorMap tx;
    if (int e = make_tmap_f32(&tx, x + bdone * S * D, nb * S, D, AF_TILE, 32)) return e;
    AttnFusedParams p{};
    p.x = x + bdone * S * D; p.w = w + bdone * S; p.out = out + bdone * D; p.Wp = Wp;
    p.b1 = b1; p.W2 = W2; p.b2 = b2; p.inv_scale = inv_scale; p.flag = flag;
    p.R = nb * S; p.B = (int)nb; p.S = S; p.D = D; p.H = H; p.nkb = nkb;
    const int grid = (int)(nb < sms ? nb : sms);
    // programmatic dependent launch: the x stream (TMA, splitters) starts under the weight-preparation kernel's tail;
    // only the epilogue warps (W1 pieces, scale) and the flag wait for it.  The preparation kernel itself is a plain
    // launch, so everything that produced x has completed before either kernel starts.
    count_launch();
    TT_CHECK_CUDA(launch_pdl(attn_pool_fused_kernel<true>, dim3(grid), dim3(AF_THREADS), smem, st, tx, p));
    bdone += nb;
  }
  const size_t fsm = (size_t)(S + 8) * sizeof(float);
  if (fsm > 48 * 1024)
    TT_CHECK_CUDA(cudaFuncSetAttribute(attn_pool_fallback_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fsm));
  count_launch();
  const int fgrid = B < num_sms() * 8 ? B : num_sms() * 8;      // grid-stride: an all-exit launch stays a few microseconds
  TT_CHECK_CUDA(launch_pdl(attn_pool_fallback_kernel, dim3(fgrid), dim3(256), fsm, st, x, w, W1, b1, W2, b2, H, out, B, S, D,
                           (const int*)flag));
  return TT_OK;
}
