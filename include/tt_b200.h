/*
 * tt_b200.h — C-ABI of the B200-native serving hot path of the two-tower recommender.
 *
 * This is the drop-in boundary: every entry point takes plain device pointers, sizes and a
 * CUDA stream (passed as void* so that no CUDA header is needed by the binder).  No torch
 * types, no ownership transfer: the caller allocates every output and the workspace.
 * All functions return 0 on success and a non-zero TT_ERR_* code otherwise;
 * tt_last_error() returns a thread-local, human-readable message for the last failure.
 *
 * The reference (HeikalPro/two-tower-model-v2) has no FFI for this path; its boundary is
 * the Python class API of two modules.  Each entry point cites the reference lines whose
 * arithmetic it replaces:
 *
 *   src/models/buyer_tower.py:43-68    weighted_average        -> tt_pool_weighted[_gather]
 *   src/training/losses.py:36-79       InfoNCELoss.forward     -> tt_infonce_forward / tt_infonce_backward
 *   src/models/buyer_tower.py:70-101   attention_aggregation   -> tt_pool_attention_fused (dense), tt_attention_logits + tt_pool_attention[_gather]
 *   src/inference/vector_db.py:44-54   build_index (normalise + IndexFlatIP.add) -> tt_flat_build
 *   src/inference/vector_db.py:152-160 retrieve  (renormalise + IndexFlatIP.search) -> tt_flat_search
 *   src/inference/vector_db.py:189-197 retrieve_batch (same, nq > 1)            -> tt_flat_search
 *   (absent in the reference)          cross-GPU merge of per-shard top-K       -> tt_topk_merge
 *
 * There is no CPU implementation behind any of these symbols: without a CUDA device they
 * return TT_ERR_CUDA.
 */
#ifndef TT_B200_H_
#define TT_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TT_B200_ABI_VERSION 1

enum {
  TT_OK = 0,
  TT_ERR_INVALID = 1,   /* bad argument (null pointer, size, alignment, unsupported shape) */
  TT_ERR_CUDA = 2,      /* a CUDA runtime/driver call failed (message has the CUDA error)    */
  TT_ERR_WORKSPACE = 3, /* workspace too small                                               */
  TT_ERR_UNSUPPORTED = 4
};

/* ABI version of the loaded library (== TT_B200_ABI_VERSION of the header it was built from). */
int tt_abi_version(void);

/* Thread-local message describing the last non-zero return on this thread ("" if none). */
const char* tt_last_error(void);

/* ------------------------------------------------------------------------------------------
 * Buyer tower pooling  (reference: src/models/buyer_tower.py)
 * ------------------------------------------------------------------------------------------
 * x      f32 [B,S,D] row-major, D fastest          (dense variant)
 * table  f32 [N,D], idx i64 [B,S]                  (gather variant: row s of buyer b is
 *                                                   table[idx[b,s]]; idx < 0 or >= N reads as
 *                                                   an all-zero row, i.e. the reference's
 *                                                   zero-padded history, trainer.py:144-151)
 * w      f32 [B,S]   event weights (arbitrary floats; zeros allowed)
 * out    f32 [B,D]   L2-normalised buyer embeddings
 *
 * weighted_avg (buyer_tower.py:58-66):
 *     nw = w / (sum_s w + 1e-8);  y = sum_s x_s * nw_s;  out = y / max(||y||_2, 1e-12)
 * attention (buyer_tower.py:85-99), given logit_s = W2 . relu(W1 x_s + b1) + b2:
 *     c = logit * w;  a = softmax_s(c);  y = sum_s x_s * a_s;  out = y / max(||y||_2, 1e-12)
 *     (no masking: a zero-weight position keeps softmax mass e^0, exactly as the reference)
 */
int tt_pool_weighted(const float* x, const float* w, float* out,
                     int B, int S, int D, void* stream);

int tt_pool_weighted_gather(const float* table, int64_t N, const int64_t* idx, const float* w,
                            float* out, int B, int S, int D, void* stream);

/* logits[r] = W2 . relu(W1 x_r + b1) + b2 for R rows of x at fp32 accuracy: the hidden layer runs on the tensor
 * cores as a 3xTF32 split (tcgen05 kind::tf32, error ~1e-7 absolute on O(0.1) logits) when D % 4 == 0, H <= 256,
 * R >= 128 and the pointers are 16-byte aligned, otherwise (or with TT_B200_ATTN_LOGITS=fma in the environment)
 * as fp32 FMA arithmetic on the CUDA cores.
 * x f32 [R,D], W1 f32 [H,D], b1 f32 [H], W2 f32 [H], b2 f32 [1], logits f32 [R].
 * (buyer_tower.py:32-36 and :85-86).  For the gather path call it once over the item table
 * (R = N) and keep the result: the logit depends on the item row only. */
int tt_attention_logits(const float* x, int64_t R, int D,
                        const float* W1, const float* b1, const float* W2, const float* b2,
                        int H, float* logits, void* stream);

/* Softmax-weighted pooling with precomputed logits.  logits f32 [B,S] (dense) or f32 [N]
 * indexed through idx (gather; an out-of-range idx has logit b2-less 0 row semantics: the
 * caller passes zero_row_logit = W2.relu(b1)+b2, the logit of an all-zero row). */
int tt_pool_attention(const float* x, const float* logits, const float* w, float* out,
                      int B, int S, int D, void* stream);

int tt_pool_attention_gather(const float* table, int64_t N, const float* row_logits,
                             float zero_row_logit, const int64_t* idx, const float* w,
                             float* out, int B, int S, int D, void* stream);

/* Backward of the pooling op for training callers (src/models/two_tower.py:212, src/training/trainer.py:216-236): given
 * g = dL/dout f32 [B,D] it recomputes y = sum_s coef_s x_s and writes
 *   dx  f32 [B,S,D] (may be NULL) = coef_s * dy         - the pooling part of dL/dx
 *   dw  f32 [B,S]                 = dL/dw
 *   dlogit f32 [B,S] (attention: logits != NULL)        = dL/dlogit, which the caller feeds to the score MLP's own
 *                                   backward (two plain GEMMs: dx += ..., dW1, db1, dW2, db2)
 * with dy = (g - out (out.g)) / ||y|| (F.normalize), coefficients as in the forward.  D % 4 == 0, D <= 1024. */
int tt_pool_backward(const float* x, const float* w, const float* logits, const float* g,
                     float* dx, float* dw, float* dlogit, int B, int S, int D, void* stream);

/* InfoNCE loss of the training callers (src/training/losses.py:36-79; trainer.py:216-236): for buyer embeddings
 * b f32 [B,D], positive product embeddings p f32 [B,D] and sampled negatives n f32 [B,M,D] (M may be 0, then n may be
 * NULL) the logits of row i are [ b_i.p_i | b_i.n_ij (j < M) | b_i.p_k (k != i, the masked in-batch block) ] / T and
 *   loss[0] = mean_i row_loss[i],  row_loss[i] = lse[i] - b_i.p_i / T,  lse[i] = logsumexp(logits_i)
 * (F.cross_entropy with label 0).  Neither the [B,B,D] expansion nor the logits matrix is materialised.  D <= 1024.
 * tt_infonce_backward: grad_loss = device pointer to dL/dloss (one float); writes d_buyer [B,D], d_pos [B,D] and
 * d_neg [B,M,D] (NULL when M == 0).  workspace: tt_infonce_workspace_bytes(B) bytes of device memory. */
size_t tt_infonce_workspace_bytes(int B);
int tt_infonce_forward(const float* buyer, const float* pos, const float* neg, int B, int M, int D, float temperature,
                       float* loss, float* row_loss, float* lse, void* stream);
int tt_infonce_backward(const float* buyer, const float* pos, const float* neg, const float* lse, const float* grad_loss,
                        int B, int M, int D, float temperature, float* d_buyer, float* d_pos, float* d_neg,
                        void* workspace, size_t workspace_bytes, void* stream);

/* Pooling out of a row-SHARDED item table (BASELINE config C5: the catalog, which is the item table of the
 * /retrieve path - src/inference/encoder.py:276-303 pools the item embeddings of the history - is split over the
 * GPUs).  Owner computes: idx holds GLOBAL row ids; this rank reduces the positions whose row it owns
 * ([row_lo, row_lo + N_local), read from `table` = its local rows) into partial f32 [B, D+4] = {acc[D], m, l, 0, 0}
 * (D % 4 == 0: every record row stays 16-byte aligned):
 *   weighted_avg (row_logits == NULL): acc = sum w_s x_s, l = sum w_s, m = 0
 *   attention (row_logits f32 [N_local]): c_s = logit_s * w_s, m = max c_s, l = sum e^(c_s-m), acc = sum e^(c_s-m) x_s
 * A position with idx outside [0, N_total) is an all-zero row: nothing for acc, but its weight / softmax mass
 * (logit = zero_row_logit) is kept by the rank called with owns_invalid = 1 (exactly one rank).
 * tt_pool_partial_merge: the all-gathered partials f32 [G, B, D+4] -> out f32 [B, D], L2-normalised; same result as
 * tt_pool_*_gather on an unsharded table up to fp32 summation order. */
int tt_pool_partial_gather(const float* table, int64_t N_local, int64_t row_lo, int64_t N_total, int owns_invalid,
                           const float* row_logits, float zero_row_logit, const int64_t* idx, const float* w,
                           float* partial, int B, int S, int D, void* stream);
int tt_pool_partial_merge(const float* partials_g, int G, int attention, float* out, int B, int D, void* stream);

/* attention_aggregation in ONE kernel and one pass over x in HBM (buyer_tower.py:70-101): the score MLP runs on
 * the tensor cores (fp16 two-piece split of both operands, fp32 accumulation in TMEM: fp32-accurate) while the rows
 * stream in through TMA, and the softmax-weighted row sum + L2 normalisation re-read the rows while they are still in
 * L2.  Fused for D % 64 == 0, D <= 384, H <= 128, S <= 8192, B*S >= 64; any other shape runs tt_attention_logits +
 * tt_pool_attention behind the same entry point.  Inputs outside the fp16 range after scaling (|x| > 4094, inf, nan)
 * are detected on the device and recomputed by a predicated fp32 CUDA-core kernel (no host synchronisation).
 * workspace: tt_pool_attention_fused_workspace_bytes(B,S,D,H) bytes of device memory, 256-byte aligned. */
size_t tt_pool_attention_fused_workspace_bytes(int B, int S, int D, int H);
int tt_pool_attention_fused(const float* x, const float* w,
                            const float* W1, const float* b1, const float* W2, const float* b2, int H,
                            float* out, int B, int S, int D,
                            void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * Exact inner-product index  (reference: src/inference/vector_db.py over faiss.IndexFlatIP)
 * ------------------------------------------------------------------------------------------
 * The index is two device arrays owned by the caller:
 *   Xn  f32  [N, D]            rows x / (||x||_2 + 1e-8)              (vector_db.py:44-45,51)
 *   Xh  bf16 [N, Dp]           round-to-nearest-even of Xn, row pitch Dp = tt_flat_pitch(D),
 *                              zero padded; the copy the tensor-core scan streams
 * plus stats f32 [4] = { max_row ||bf16(xn)||, max_row ||bf16(xn) - xn||, 0, 0 }, which bound
 * the bf16 scoring error so that the search can certify exactness per query.
 */
int64_t tt_flat_pitch(int D); /* D rounded up to a multiple of 64 (one 128-byte TMA box) */

/* Add `rows` rows of X to the index arrays starting at row `row0` and fold their norms into
 * stats (call once per chunk; zero `stats` before the first chunk).
 *   normalize = 1 : Xn = x / (||x|| + 1e-8)          (build_index, vector_db.py:44-45)
 *   normalize = 0 : Xn = x verbatim                   (load_index of rows faiss already stored,
 *                                                      vector_db.py:77)
 * Xn + row0*D may alias X (in-place). */
int tt_flat_build(const float* X, int64_t rows, int D, int normalize,
                  float* Xn, void* Xh, int64_t row0, float* stats, void* stream);

/* Bytes of device workspace tt_flat_search needs for (N, D, nq, K). */
size_t tt_flat_search_workspace_bytes(int64_t N, int D, int nq, int K);

/* Exact top-K inner-product search of nq queries against the index.
 *   q       f32 [nq, D]   un-normalised; the op renormalises with q / (||q|| + 1e-8)
 *                         (vector_db.py:152-153 / :189-190)
 *   K       1 <= K <= min(N, TT_FLAT_MAX_K)   (the caller clamps k = min(k, ntotal),
 *                         vector_db.py:159)
 *   scores  f32 [nq, K]   fp32 inner products, descending
 *   ids     i64 [nq, K]   row index + id_offset; ties ordered by ascending id
 *   flags   i32 [nq]      1 = top-K certified exact; <= 0 = this query must be re-run through
 *                         tt_flat_search_exact (value = -(reason bits): 1 candidate list overflow, 2 fewer
 *                         than K candidates, 4 score self-check failed, 8 the K-th rescored score does not clear the
 *                         bound of the rows that were not rescored)
 *   n_uncertified i32 [1] number of flags != 1
 * Scores come from a bf16 tensor-core scan (tcgen05) that over-fetches a candidate set, followed
 * by fp32 rescoring of the candidates whose bf16 score is within reach of the K-th; the certificate
 * proves no row that was not rescored can belong to the fp32 top-K.  Asynchronous on `stream`. */
#define TT_FLAT_MAX_K 2048
int tt_flat_search(const float* q, int nq,
                   const float* Xn, const void* Xh, const float* stats, int64_t N, int D,
                   int K, int64_t id_offset,
                   float* scores, int64_t* ids, int32_t* flags, int32_t* n_uncertified,
                   void* workspace, size_t workspace_bytes, void* stream);

/* Always-exact fp32 path (CUDA-core scoring + radix select), used for uncertified queries and
 * as an independent on-device cross-check.  qsel i32 [nsel] lists the query rows to process
 * (NULL = all nq queries, nsel = nq); results are written to the same rows of scores/ids. */
size_t tt_flat_search_exact_workspace_bytes(int64_t N, int D, int nsel, int K);
int tt_flat_search_exact(const float* q, int nq, const int32_t* qsel, int nsel,
                         const float* Xn, int64_t N, int D, int K, int64_t id_offset,
                         float* scores, int64_t* ids,
                         void* workspace, size_t workspace_bytes, void* stream);

/* Exclusion lists: the exact top-K over the rows a query does NOT exclude (e.g. a buyer's own history).
 *   excl    i64 [nq, E]   row-major; excl[q, j] is an id in the result id space (row + id_offset, a global id
 *                         on a shard).  Entries below 0 are padding, ids outside the index (or this shard) are
 *                         ignored, duplicates are allowed: the padded history idx of the pooling calls fits as is.
 *   E       0 <= E <= TT_FLAT_MAX_EXCLUDE; excl may be NULL only when E == 0.  E == 0 is the plain call.
 * Results are ordered as above; with fewer than K allowed rows the tail is score -inf / id -1.  An excluded row
 * never appears in an output.  The certificate is read over the allowed rows: "every allowed row not rescored
 * scores below the bound"; flags, bound and the merge keep their meaning.
 * Excluded rows are typically a query's best ones, so the scan is planned for
 *     K_plan = min(K + E, N, TT_FLAT_MAX_K)          (N = rows of this index, N_total on the global-threshold path)
 * while K results are emitted and the K-th ALLOWED score is certified.  tt_flat_search_excl_workspace_bytes sizes the
 * workspace for it.  The global-threshold calls that never see the list - tt_flat_shard_plan_ok,
 * tt_flat_shard_workspace_bytes and tt_flat_shard_sample - are called with K_plan as their K (N = N_total), and
 * tt_flat_shard_search_excl with K.  tt_flat_search_exact_excl reads the list row of the QUERY row qsel[i] (not of
 * the slot i); an uncertified query is re-run there with the same list. */
#define TT_FLAT_MAX_EXCLUDE 1024
size_t tt_flat_search_excl_workspace_bytes(int64_t N, int D, int nq, int K, int E);
int tt_flat_search_excl(const float* q, int nq,
                        const float* Xn, const void* Xh, const float* stats, int64_t N, int D,
                        int K, int64_t id_offset,
                        float* scores, int64_t* ids, int32_t* flags, int32_t* n_uncertified,
                        const int64_t* excl, int E,
                        void* workspace, size_t workspace_bytes, void* stream);
int tt_flat_search_exact_excl(const float* q, int nq, const int32_t* qsel, int nsel,
                              const float* Xn, int64_t N, int D, int K, int64_t id_offset,
                              float* scores, int64_t* ids, const int64_t* excl, int E,
                              void* workspace, size_t workspace_bytes, void* stream);

/* Merge G per-shard sorted top-K lists into one: scores_g f32 [G, nq, K], ids_g i64 [G, nq, K]
 * (the layout an all-gather of per-rank [nq,K] results produces) -> [nq, K], same ordering
 * (score descending, id ascending). */
int tt_topk_merge(const float* scores_g, const int64_t* ids_g, int G, int nq, int K,
                  float* scores, int64_t* ids, void* stream);

/* Catalog sharded over G devices (north_star (3); the reference has no multi-device path).
 * tt_flat_search_shard = tt_flat_search over this shard's rows (ids = local row + id_offset), plus
 *   bound f32 [nq]: every row of this shard that was NOT rescored in fp32 scores strictly below bound[q]
 *                   (-inf when every row was rescored).  The per-shard flags keep their meaning, but bits 2
 *                   and 8 (local K-th score checks) are superseded by the global certificate below.
 * Each rank packs {scores f32[nq,K] | ids i64[nq,K] | bound f32[nq] | flags i32[nq]} into one byte record
 * (lists shorter than K padded with score -inf / id -1); ONE all-gather of the records gives `gathered`
 * (G records, rank_stride bytes apart, fields at the given byte offsets).
 * tt_shard_merge merges the G sorted lists (score descending, id ascending) into scores/ids [nq,K] and
 * certifies each query: exact iff the merged K-th score >= max over shards of bound[q] and no shard
 * reported a candidate overflow (1) or a score self-check failure (4); flags/n_uncertified as in
 * tt_flat_search - an uncertified query is re-run through tt_flat_search_exact on every shard. */
int tt_flat_search_shard(const float* q, int nq,
                         const float* Xn, const void* Xh, const float* stats, int64_t N, int D,
                         int K, int64_t id_offset,
                         float* scores, int64_t* ids, int32_t* flags, int32_t* n_uncertified, float* bound,
                         void* workspace, size_t workspace_bytes, void* stream);
/* One threshold for the whole sharded catalog (the fast sharded path; both calls use the SAME workspace):
 *   tt_flat_shard_plan_ok   host-only, 1 if this path applies to (N_local, N_total, D, nq, K) - a function of
 *                           N_total, D, nq, K and of N_local >= K only, so every rank decides alike when
 *                           called with its smallest shard; otherwise use tt_flat_search_shard.
 *   tt_flat_shard_sample    renormalises the queries, samples this shard's tiles at the stride a single device
 *                           would use for N_total rows and writes each query's TT_SHARD_TOPR largest sampled
 *                           scores, descending, -inf padded: topr f32 [nq, TT_SHARD_TOPR].
 *   (all-gather the lists: topr_g f32 [G, nq, TT_SHARD_TOPR])
 *   tt_flat_shard_search    threshold = planned rank among the union of the G lists (identical on every rank),
 *                           main scan, finalize; outputs as tt_flat_search_shard.  The threshold only decides
 *                           how many candidates are rescored; exactness rests on the certificate of
 *                           tt_shard_merge. */
#define TT_SHARD_TOPR 32
int tt_flat_shard_plan_ok(int64_t N_local, int64_t N_total, int D, int nq, int K);
size_t tt_flat_shard_workspace_bytes(int64_t N_local, int64_t N_total, int D, int nq, int K);
int tt_flat_shard_sample(const float* q, int nq, const void* Xh, const float* stats,
                         int64_t N_local, int64_t N_total, int D, int K, float* topr,
                         void* workspace, size_t workspace_bytes, void* stream);
int tt_flat_shard_search(int nq, const float* Xn, const void* Xh, int64_t N_local, int64_t N_total, int D,
                         int K, int64_t id_offset, const float* topr_g, int G,
                         float* scores, int64_t* ids, int32_t* flags, int32_t* n_uncertified, float* bound,
                         void* workspace, size_t workspace_bytes, void* stream);
/* The same two shard searches with per-query exclusion lists (see tt_flat_search_excl; ids are global).  On the
 * global-threshold path call tt_flat_shard_plan_ok / tt_flat_shard_workspace_bytes / tt_flat_shard_sample with
 * K_plan = min(K + E, N_total, TT_FLAT_MAX_K) and tt_flat_shard_search_excl with K.  A shard whose allowed rows
 * are fewer than K pads its record with -inf / -1; its bound keeps its meaning over the allowed rows. */
int tt_flat_search_shard_excl(const float* q, int nq,
                              const float* Xn, const void* Xh, const float* stats, int64_t N, int D,
                              int K, int64_t id_offset,
                              float* scores, int64_t* ids, int32_t* flags, int32_t* n_uncertified, float* bound,
                              const int64_t* excl, int E,
                              void* workspace, size_t workspace_bytes, void* stream);
int tt_flat_shard_search_excl(int nq, const float* Xn, const void* Xh, int64_t N_local, int64_t N_total, int D,
                              int K, int64_t id_offset, const float* topr_g, int G,
                              float* scores, int64_t* ids, int32_t* flags, int32_t* n_uncertified, float* bound,
                              const int64_t* excl, int E,
                              void* workspace, size_t workspace_bytes, void* stream);
int tt_shard_merge(const void* gathered, size_t rank_stride, size_t off_scores, size_t off_ids,
                   size_t off_bound, size_t off_flags, int G, int nq, int K,
                   float* scores, int64_t* ids, int32_t* flags, int32_t* n_uncertified, void* stream);

/* All-gather of per-rank records over NVLink peer memory by our own kernels (the exchange of the sharded
 * search; NCCL stays available as the alternative).  The caller owns, on every rank, a receive buffer and
 * an int32 flag array [G] that are mapped into every peer (CUDA IPC) and double-buffered by sequence parity.
 *   tt_p2p_push  copies `src` (nbytes, multiple of 16) into peer_dst[g] for every g (host arrays of G device
 *                pointers: my slot in rank g's receive buffer / my flag cell in rank g's flag array), then
 *                publishes `seq` in the flags with system-scope release stores.  done_counter: u32 device
 *                scalar, zero-initialised, private to this stream.
 *   tt_p2p_wait  one-warp kernel: returns when flags[g] >= seq for every g (acquire loads); after
 *                timeout_seconds it gives up and writes seq to *timed_out (device i32, 0 = fine) instead of
 *                hanging the device.  Kernels enqueued after it may read the receive buffer. */
int tt_p2p_enable_peer(int peer_device);   /* cudaDeviceEnablePeerAccess from the current device (idempotent) */
/* Receive-buffer plumbing: tt_p2p_alloc = cudaMalloc (zero-filled) + its 64-byte CUDA IPC handle; tt_p2p_open maps
 * another rank's handle into the CURRENT device's address space with peer access; close / free undo them. */
int tt_p2p_alloc(size_t bytes, void** dev_ptr, void* handle64);
int tt_p2p_open(const void* handle64, void** dev_ptr);
int tt_p2p_close(void* dev_ptr);
int tt_p2p_free(void* dev_ptr);
int tt_p2p_push(const void* src, size_t nbytes, void* const* peer_dst, int32_t* const* peer_flag, int G,
                int32_t seq, uint32_t* done_counter, void* stream);
int tt_p2p_wait(const int32_t* flags, int G, int32_t seq, double timeout_seconds, int32_t* timed_out,
                void* stream);

/* Measurement hooks (bench.py).  tt_kernel_launch_count: kernels this library has launched in this
 * process.  tt_profile_scan_arm(n): the next n main-scan launches of tt_flat_search are bracketed by
 * CUDA events on their stream; tt_profile_scan_read: waits for them, writes their durations in ms,
 * returns how many were recorded (-1 on a CUDA error) and disarms. */
int64_t tt_kernel_launch_count(void);
int tt_profile_scan_arm(int max_records);
int tt_profile_scan_read(float* ms_out, int max_out);

/* Host-only: the planner's decisions for (N, D, nq, K) as 16 ints: supported, queries per unit (64 /
 * 128 single CTA, 256 CTA pair), k_blocks, stages, query_units, tiles, use_threshold, route_exact,
 * target_candidates, candidate_capacity, sample_stride, sample_slots, sample_rank, main_slices,
 * segment_capacity, smem_bytes. */
int tt_flat_plan_describe(int64_t N, int D, int nq, int K, int32_t* out16);

/* Diagnostic: after a tt_flat_search call that used `workspace`, copy out every query's scan threshold
 * (bf16-score domain) and its candidate count (device pointers thr_out f32[nq], cnt_out i32[nq]). */
int tt_flat_debug_read(const void* workspace, int64_t N, int D, int nq, int K,
                       float* thr_out, int32_t* cnt_out, void* stream);

/* Diagnostic / parity-test entry: the raw bf16 tensor-core scores of EVERY row of a small catalog
 * (N <= 2^22), out f32 [nq, N] = <bf16(qn), Xh[r]> with fp32 accumulation, as the scan kernel's
 * epilogue sees them.  Runs the same kernel as tt_flat_search with the threshold at -inf. */
size_t tt_flat_scan_scores_workspace_bytes(int64_t N, int D, int nq);
int tt_flat_scan_scores(const float* q, int nq, const void* Xh, const float* stats, int64_t N, int D,
                        float* out, void* workspace, size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* TT_B200_H_ */
