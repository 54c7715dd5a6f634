// Internal interfaces between the translation units of the exact inner-product search.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

namespace tt {

constexpr int SAMPLE_MAX_SLOTS = 4096;      // sampled tiles per query (8 chunk maxima each are staged in smem)
constexpr int SHARD_TOPR = 32;              // sampled maxima per query a shard contributes to the global threshold
constexpr int FINALIZE_MAX_SLICES = 1024;   // catalog slices per query the finalize kernel gathers
constexpr int FINALIZE_MAX_CAND = 16384;   // candidates per query the finalize kernel can sort (128 KiB smem)

// Everything the host decides about one search call (pure function of N, D, nq, K and the SM count).
struct ScanPlan {
  int Dp, num_kb, block_m, num_stages;
  int num_kb_res, stage_bytes;   // resident query K-blocks; ring stride (see ScanParams)
  bool supported;
  bool pair;           // 2-CTA clusters running cta_group::2 MMAs (nq > 128)
  size_t smem_bytes;
  int nqb, nq_pad, num_tiles;
  int nqu;             // query units the grid is built from: query blocks, or pairs of them
  int target;          // expected candidates per query
  int cand_cap;        // candidates of one query the finalize kernel sorts (sum over slices)
  int seg_cap;         // capacity of one (query, slice) candidate segment
  bool use_threshold;  // false: every row is a candidate (small catalogs)
  bool route_exact;    // true: K is too large a fraction of N for a sampled threshold -> fp32 exact path
  int main_slices;
  int sample_stride, sample_slots, sample_slices, sample_rank;
  bool sample_tile_max;  // sample pass records one maximum per sampled tile (else one per 32-row chunk)
};

ScanPlan make_scan_plan(long long N, int D, int nq, int K);

// zero_me (may be NULL): an int the kernel sets to 0 (the call's n_uncertified counter)
int launch_prep_queries(const float* q, int nq, int nq_pad, int D, int Dp, const float* stats,
                        float* qn, void* qh, float* eps, int* zero_me, cudaStream_t st);

// sample pass (if plan.use_threshold) + threshold selection + main scan
int launch_scan(const ScanPlan& pl, const void* qh, const void* Xh, long long N, int nq,
                float* thr, unsigned int* seg_cnt, void* cand, float* sample_buf, cudaStream_t st);

// the pieces launch_scan is made of (the sharded path runs them with an exchange in between)
ScanPlan make_shard_plan(long long N_local, long long N_total, int D, int nq, int K, bool* global_ok);
int launch_sample(const ScanPlan& pl, const void* qh, const void* Xh, long long N, int nq, float* thr, float* topr,
                  float* sample_buf, cudaStream_t st, bool skip_select = false);
int launch_select_gathered(const float* topr_g, int G, int nq, int r, float* thr, int* zero_me, cudaStream_t st);
int launch_main_scan(const ScanPlan& pl, const void* qh, const void* Xh, long long N, int nq, float* thr,
                     unsigned int* seg_cnt, void* cand, cudaStream_t st, const float* sel_sample = nullptr);

// fp32 rescoring of every candidate, exact sort, certificate; excl i64 [nq, E] (E > 0) drops the listed rows
int launch_finalize(const ScanPlan& pl, const float* qn, const float* Xn, long long N, int D, int nq, int K,
                    long long id_offset, const float* thr, const float* eps, const unsigned int* seg_cnt,
                    const void* cand, float* scores, long long* ids, int* flags, int* n_uncertified,
                    float* bound_out, cudaStream_t st, const long long* excl = nullptr, int E = 0);

// shared TMA descriptor helper (flat_scan.cu) and the tensor-core attention-logits launcher (attn_logits_tc.cu)
int make_tmap_f32(void* tensor_map /* CUtensorMap* */, const void* base, long long rows, int cols, int box_rows, int box_cols);
int launch_attn_logits_tc(const float* x, long long R, int D, const float* W1, const float* b1, const float* W2,
                          const float* b2, int H, float* logits, cudaStream_t st);

// attn_pool_fused.cu in logits-only mode (TT_ERR_UNSUPPORTED without an error message when the shape does not fit),
// its predicated fp32 recomputation (attn_logits.cu) and the library-private stream-ordered scratch pool
int launch_attn_logits_fused(const float* x, long long R, int D, const float* W1, const float* b1, const float* W2,
                             const float* b2, int H, float* logits, cudaStream_t st);
int launch_attn_logits_generic_if(const float* x, long long R, int D, const float* W1, const float* b1, const float* W2,
                                  const float* b2, int H, float* logits, const int* run_if, cudaStream_t st);
cudaMemPool_t scratch_pool(int dev);

// Optional device-side timing of the main scan kernel (bench.py roofline): when armed, launch_scan
// brackets the main scan launch with a pair of CUDA events on the launching stream.
void profile_scan_begin(cudaStream_t st);
void profile_scan_end(cudaStream_t st);

}  // namespace tt
