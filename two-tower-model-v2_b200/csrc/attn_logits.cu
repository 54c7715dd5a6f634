// Attention-score MLP of the buyer tower (reference: src/models/buyer_tower.py:32-36,85-86):
//     logit[r] = W2 . relu(W1 x_r + b1) + b2
// fp32 FMA arithmetic end to end.  A bf16 tensor-core MLP does NOT meet the 1e-5 tolerance of
// the pooled output (the event weight, up to 10, multiplies the logit inside exp; measured
// 4e-4), so this is a register-tiled CUDA-core SGEMM with the ReLU / W2 dot / bias fused into
// the epilogue: the [R,H] hidden activations never leave registers.
// Roofline: fp32 FMA pipe, 2*D*H + 2*H flop per row.  The inner product runs on packed FFMA2
// (fma.rn.f32x2, two k-partial sums per 64-bit accumulator): half the issue slots per FMA, which is
// what the unpacked version was short of (ncu: 70 % issue utilisation, 24 % dispatch stalls at 52 % of
// the FMA peak).
#include "tt_common.cuh"
#include "flat_internal.cuh"

namespace tt {

constexpr int AL_BM = 64;      // rows per CTA tile (4 per thread)
constexpr int AL_BN = 128;     // hidden units per chunk
constexpr int AL_BK = 32;      // k-slab
constexpr int AL_LD = AL_BK + 4;   // padded smem row (floats): conflict-free 128-bit LDS/STS
constexpr int AL_THREADS = 256;
constexpr int AL_STAGE_FLOATS = (AL_BM + AL_BN) * AL_LD;

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem, int src_bytes) {
  const uint32_t s = (uint32_t)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(s), "l"(gmem), "r"(src_bytes));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N)); }

// Loads one k-slab of the X tile and of the W1 chunk into a stage (zero-filling out-of-range
// rows / hidden units / k).
__device__ __forceinline__ void al_load_stage(float* stage, const float* __restrict__ x, long long R, int D,
                                              const float* __restrict__ W1, int H,
                                              long long row0, int h0, int k0, int tid) {
  float* Xs = stage;
  float* Ws = stage + AL_BM * AL_LD;
#pragma unroll
  for (int i = 0; i < (AL_BM * AL_BK / 4) / AL_THREADS; ++i) {
    const int f = tid + i * AL_THREADS;
    const int r = f >> 3, c4 = f & 7;
    const long long gr = row0 + r;
    const int k = k0 + c4 * 4;
    const bool ok = (gr < R) && (k < D);
    cp_async16(Xs + r * AL_LD + c4 * 4, ok ? (x + gr * D + k) : x, ok ? 16 : 0);
  }
#pragma unroll
  for (int i = 0; i < (AL_BN * AL_BK / 4) / AL_THREADS; ++i) {
    const int f = tid + i * AL_THREADS;
    const int r = f >> 3, c4 = f & 7;
    const int gh = h0 + r;
    const int k = k0 + c4 * 4;
    const bool ok = (gh < H) && (k < D);
    cp_async16(Ws + r * AL_LD + c4 * 4, ok ? (W1 + (long long)gh * D + k) : W1, ok ? 16 : 0);
  }
}

// d.{x,y} += a.{x,y} * b.{x,y}  (one FFMA2)
__device__ __forceinline__ void ffma2(float2& d, const float2 a, const float2 b) {
  unsigned long long dd = *reinterpret_cast<unsigned long long*>(&d);
  const unsigned long long aa = *reinterpret_cast<const unsigned long long*>(&a);
  const unsigned long long bb = *reinterpret_cast<const unsigned long long*>(&b);
  asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(dd) : "l"(aa), "l"(bb));
  d = *reinterpret_cast<float2*>(&dd);
}

__global__ void __launch_bounds__(AL_THREADS, 2)
attn_logits_kernel(const float* __restrict__ x, long long R, int D,
                   const float* __restrict__ W1, const float* __restrict__ b1,
                   const float* __restrict__ W2, const float* __restrict__ b2, int H,
                   float* __restrict__ logits) {
  extern __shared__ __align__(16) float smem[];
  const int tid = threadIdx.x;
  const int tx = tid & 15;    // hidden sub-index: hidden = h0 + tx + 16*j
  const int ty = tid >> 4;    // row sub-index:    row    = row0 + ty + 16*i
  const long long row0 = (long long)blockIdx.x * AL_BM;
  const int nk = (D + AL_BK - 1) / AL_BK;

  constexpr int TI = AL_BM / 16;   // rows per thread (4)
  float logit[TI];
#pragma unroll
  for (int i = 0; i < TI; ++i) logit[i] = 0.f;

  for (int h0 = 0; h0 < H; h0 += AL_BN) {
    float2 acc[TI][8];               // {even-k partial, odd-k partial}
#pragma unroll
    for (int i = 0; i < TI; ++i)
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[i][j] = make_float2(0.f, 0.f);

    al_load_stage(smem, x, R, D, W1, H, row0, h0, 0, tid);
    cp_async_commit();
    for (int kt = 0; kt < nk; ++kt) {
      float* cur = smem + (kt & 1) * AL_STAGE_FLOATS;
      if (kt + 1 < nk) {
        al_load_stage(smem + ((kt + 1) & 1) * AL_STAGE_FLOATS, x, R, D, W1, H, row0, h0, (kt + 1) * AL_BK, tid);
        cp_async_commit();
        cp_async_wait<1>();
      } else {
        cp_async_wait<0>();
      }
      __syncthreads();
      const float* Xs = cur;
      const float* Ws = cur + AL_BM * AL_LD;
#pragma unroll
      for (int kk4 = 0; kk4 < AL_BK / 4; ++kk4) {
        float4 xa[TI];
#pragma unroll
        for (int i = 0; i < TI; ++i)
          xa[i] = *reinterpret_cast<const float4*>(Xs + (ty + 16 * i) * AL_LD + kk4 * 4);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float4 wb = *reinterpret_cast<const float4*>(Ws + (tx + 16 * j) * AL_LD + kk4 * 4);
#pragma unroll
          for (int i = 0; i < TI; ++i) {
            ffma2(acc[i][j], make_float2(xa[i].x, xa[i].y), make_float2(wb.x, wb.y));
            ffma2(acc[i][j], make_float2(xa[i].z, xa[i].w), make_float2(wb.z, wb.w));
          }
        }
      }
      __syncthreads();
    }
    // fused epilogue for this hidden chunk: relu(acc + b1) . W2
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int h = h0 + tx + 16 * j;
      const float bj = (h < H) ? __ldg(b1 + h) : 0.f;
      const float wj = (h < H) ? __ldg(W2 + h) : 0.f;
#pragma unroll
      for (int i = 0; i < TI; ++i) logit[i] = fmaf(fmaxf((acc[i][j].x + acc[i][j].y) + bj, 0.f), wj, logit[i]);
    }
  }
  const float bias2 = __ldg(b2);
#pragma unroll
  for (int i = 0; i < TI; ++i) {
    float v = logit[i];
    v += __shfl_xor_sync(0xffffffffu, v, 8);
    v += __shfl_xor_sync(0xffffffffu, v, 4);
    v += __shfl_xor_sync(0xffffffffu, v, 2);
    v += __shfl_xor_sync(0xffffffffu, v, 1);
    const long long r = row0 + ty + 16 * i;
    if (tx == 0 && r < R) logits[r] = v + bias2;
  }
}

// Shapes the tiled kernel does not take (D % 4 != 0 or unaligned pointers): one CTA per row.
__global__ void __launch_bounds__(128)
attn_logits_generic_kernel(const float* __restrict__ x, long long R, int D,
                           const float* __restrict__ W1, const float* __restrict__ b1,
                           const float* __restrict__ W2, const float* __restrict__ b2, int H,
                           float* __restrict__ logits, const int* __restrict__ run_if) {
  pdl_wait();
  if (run_if && *run_if == 0) return;       // predicated fp32 recomputation behind the tensor-core kernel
  extern __shared__ float xs[];
  __shared__ float red[4];
  for (long long r = blockIdx.x; r < R; r += gridDim.x) {
    for (int d = threadIdx.x; d < D; d += blockDim.x) xs[d] = x[r * D + d];
    __syncthreads();
    float part = 0.f;
    for (int h = threadIdx.x; h < H; h += blockDim.x) {
      float a = 0.f;
      const float* wr = W1 + (long long)h * D;
      for (int d = 0; d < D; ++d) a = fmaf(xs[d], __ldg(wr + d), a);
      part = fmaf(fmaxf(a + __ldg(b1 + h), 0.f), __ldg(W2 + h), part);
    }
    part = warp_sum(part);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = part;
    __syncthreads();
    if (threadIdx.x == 0) logits[r] = red[0] + red[1] + red[2] + red[3] + __ldg(b2);
    __syncthreads();
  }
}

// predicated launch for attn_pool_fused.cu (logits-only mode): recompute every row in fp32 when *run_if != 0
int launch_attn_logits_generic_if(const float* x, long long R, int D, const float* W1, const float* b1, const float* W2,
                                  const float* b2, int H, float* logits, const int* run_if, cudaStream_t st) {
  TT_CHECK_ARG(R <= 0x7fffffffLL && (size_t)D * sizeof(float) <= 48 * 1024, "shape too large for the generic logits kernel");
  count_launch();
  const long long cap = (long long)num_sms() * 16;       // grid-stride: an all-exit launch stays a few microseconds
  TT_CHECK_CUDA(launch_pdl(attn_logits_generic_kernel, dim3((unsigned)(R < cap ? R : cap)), dim3(128), (size_t)D * sizeof(float),
                           st, x, R, D, W1, b1, W2, b2, H, logits, run_if));
  return TT_OK;
}

}  // namespace tt

using namespace tt;

extern "C" __attribute__((visibility("default"))) int tt_attention_logits(const float* x, int64_t R, int D,
                                   const float* W1, const float* b1, const float* W2, const float* b2,
                                   int H, float* logits, void* stream) {
  TT_CHECK_ARG(x && W1 && b1 && W2 && b2 && logits, "null pointer");
  TT_CHECK_ARG(R >= 0 && D >= 1 && H >= 1, "need R >= 0, D >= 1, H >= 1");
  if (R == 0) return TT_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const bool fast = (D % 4 == 0) && ((reinterpret_cast<uintptr_t>(x) & 15) == 0) &&
                    ((reinterpret_cast<uintptr_t>(W1) & 15) == 0);
  // Tensor-core paths (fp32-accurate) for aligned shapes; the rest runs on the CUDA cores (FFMA2 tiled, else generic).
  if (fast && R >= 64 && R < (1LL << 31)) {
    // D % 64 == 0, D <= 384, H <= 128: the fp16 two-piece kernel of the fused pooling in its logits-only mode
    int e = launch_attn_logits_fused(x, R, D, W1, b1, W2, b2, H, logits, st);
    if (e != TT_ERR_UNSUPPORTED) return e;
    if (R >= 128) {
      e = launch_attn_logits_tc(x, R, D, W1, b1, W2, b2, H, logits, st);
      if (e != TT_ERR_UNSUPPORTED) return e;
    }
  }
  if (fast) {
    const size_t smem = 2 * AL_STAGE_FLOATS * sizeof(float);
    TT_CHECK_CUDA(cudaFuncSetAttribute(attn_logits_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const long long grid = (R + AL_BM - 1) / AL_BM;
    TT_CHECK_ARG(grid <= 0x7fffffffLL, "too many rows");
    attn_logits_kernel<<<(unsigned)grid, AL_THREADS, smem, st>>>(x, R, D, W1, b1, W2, b2, H, logits);
  } else {
    TT_CHECK_ARG(R <= 0x7fffffffLL, "too many rows");
    TT_CHECK_ARG((size_t)D * sizeof(float) <= 48 * 1024, "D too large for the generic logits kernel");
    attn_logits_generic_kernel<<<(unsigned)R, 128, (size_t)D * sizeof(float), st>>>(x, R, D, W1, b1, W2, b2, H, logits, nullptr);
  }
  TT_CHECK_LAUNCH();
  return TT_OK;
}
