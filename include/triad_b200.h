/*
 * triad_b200 — C ABI of the B200-native max-mean similarity + symmetric InfoNCE path.
 *
 * The reference (SajayR/TRIAD) is pure Python and has NO FFI of its own: the boundary it
 * exposes for this path is the set of methods in src/model.py / src/retrieval.py listed in
 * SURVEY.md §8(b).  The entry points below are what a ctypes binding behind those methods
 * calls (INTEGRATION.md shows the stub); each one cites the reference lines it replaces.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer into caller-owned memory (torch storage); the library
 *     never allocates device memory — scratch is passed in (`ws`, sized by *_workspace_bytes);
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*; 0 = default);
 *   - return value: 0 on success, a negative TRIAD_ERR_* otherwise; nothing throws;
 *   - tensors are contiguous row-major; q/v need 16-byte aligned base pointers and D % 8 == 0;
 *   - `temperature` is a device pointer to one fp32 (the nn.Parameter at model.py:348), so no
 *     host synchronisation is needed to read it; it must be > 0;
 *   - M = Bq*Nq is the number of query-token rows ("rows" below).
 *
 * Layouts the library defines (the reference never materialises them on this path):
 *   idx   : [Bv][Bq][nq_pad]  uint8 when Nv <= 256 else uint16, nq_pad = Nq rounded up to 16 —
 *           idx[j][i][a] = argmax_p S[i,j,a,p], first index among ties (torch.max, model.py:389);
 *           entries a >= Nq are never written or read.  Image-major so that the dV pass reads one
 *           image's winners contiguously; the per-query padding keeps every query's run 16-byte
 *           aligned for the vector loads of the dQ pass.
 *   row_scale : [M] fp32 — weight of token row r in its query's (masked) mean:
 *           1/Nq (model.py:391) or mask/clamp(sum mask,1e-7) (model.py:509-512).
 */
#ifndef TRIAD_B200_H
#define TRIAD_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TRIAD_OK                 0
#define TRIAD_ERR_BAD_ARG       (-1)  /* null pointer / negative size / unknown enum          */
#define TRIAD_ERR_BAD_SHAPE     (-2)  /* D % 8 != 0, Nv > 65535, B == 0, ...                  */
#define TRIAD_ERR_ALIGNMENT     (-3)  /* q / v / ws not 16-byte aligned                       */
#define TRIAD_ERR_WORKSPACE     (-4)  /* ws_bytes smaller than *_workspace_bytes()            */
#define TRIAD_ERR_CUDA          (-5)  /* a CUDA runtime/driver call failed (see last_error)   */
#define TRIAD_ERR_ARCH          (-6)  /* device is not sm_100 (the kernels are sm_100a only)  */
#define TRIAD_ERR_UNSUPPORTED   (-7)  /* shape outside what this build implements             */
#define TRIAD_ERR_TIMEOUT       (-8)  /* a kernel watchdog fired (pipeline deadlock guard)    */

#define TRIAD_DTYPE_F32   0
#define TRIAD_DTYPE_BF16  1

/* flags for triad_maxmean_fwd */
#define TRIAD_FWD_DEFAULT      0
#define TRIAD_FWD_FORCE_SIMT   1   /* fp32-accumulate CUDA-core kernel (always used for fp32 inputs) */
#define TRIAD_FWD_FORCE_1CTA   2   /* tcgen05 kernel with cta_group::1 (debug / small shapes)        */
#define TRIAD_FWD_DIVIDE_BY_T  4   /* S = <q,v> / T (retrieval.py:108) instead of <q,v> * T          */
#define TRIAD_FWD_SYNC_CHUNKS  8   /* test aid: chunk-synchronous tile order (the V > 48 MB path) with 3-image chunks */
#define TRIAD_FWD_PACK_ROWS   16   /* bf16 tensor-core path: rows whose row_scale is 0 (padded text tokens,
                                      model.py:509-512) are dropped before the GEMM; their idx entries read 0 */

#define TRIAD_FWD_TEST_TRIP_WATCHDOG 32 /* test aid: raise the pipeline-watchdog flag after the kernel, as a timed-out
                                         barrier wait would: clip must come back NaN (never a silent garbage matrix) */

int         triad_abi_version(void);
const char* triad_status_string(int status);
/* Text of the last CUDA error seen by the calling thread ("" if none). */
const char* triad_last_error(void);
/* Number of CUDA kernels this library has launched in this process so far (all threads); lets a
 * caller state exactly how many of the library's kernels ran inside a timed region. */
long long   triad_launch_count(void);
/* 0 if `device` can run the kernels (compute capability 10.x), TRIAD_ERR_ARCH otherwise. */
int         triad_device_check(int device);

/* ---- row weights ------------------------------------------------------------------- */
/* row_scale[i*Nq+t] = mask ? mask[i,t]/clamp(sum_t mask[i,t],1e-7) : 1/Nq.
 * Replaces model.py:391 (mean) and model.py:509-512 (mask.float(), sum, clamp, divide).
 * `mask` is the tokenizer's int64 attention mask [Bq,Nq] (model.py:118) or NULL. */
int triad_row_scale(const int64_t* mask, int Bq, int Nq, float* row_scale, void* stream);

/* ---- forward: token similarity -> max over patches -> weighted mean over tokens ------ */
/* Replaces compute_all_similarities_av (model.py:370-392) and _tv (model.py:490-514):
 *   S[i,j,a,p] = round(T * <q[i,a,:], v[j,p,:]>)   (rounded like the reference: see triad_round.h)
 *   clip[i,j]  = sum_a row_scale[i*Nq+a] * max_p S[i,j,a,p]
 * q [Bq,Nq,D], v [Bv,Nv,D] in `dtype`; clip fp32 [Bq,Bv]; idx as described above or NULL
 * (forward-only).  The Bq x Bv x Nq x Nv tensor is never written to memory. */
size_t triad_maxmean_fwd_workspace_bytes(int Bq, int Bv, int Nq, int Nv, int D, int dtype);
/* the same, for a call that passes `flags` (TRIAD_FWD_PACK_ROWS needs room for the packed copy of q) */
size_t triad_maxmean_fwd_workspace_bytes_ex(int Bq, int Bv, int Nq, int Nv, int D, int dtype, int flags);
int triad_maxmean_fwd(const void* q, const void* v, const float* row_scale,
                      const float* temperature,
                      int Bq, int Bv, int Nq, int Nv, int D, int dtype,
                      float* clip, void* idx,
                      void* ws, size_t ws_bytes, int flags, void* stream);

/* Debug/test aid: synchronises `stream` and returns TRIAD_ERR_TIMEOUT if the forward kernel
 * that last used `ws` tripped its pipeline-deadlock watchdog, TRIAD_OK otherwise. */
int triad_maxmean_fwd_status(const void* ws, void* stream);

/* ---- symmetric InfoNCE on a row block of the clip matrix ---------------------------- */
/* Replaces model.py:453-459 / :572-578 (two log_softmax + gathers) and the statistics block
 * model.py:435-450 / :553-568, for rows [row0,row0+rows) of a B x B matrix (rows == B and
 * row0 == 0 on one GPU; one block per rank when the batch is row-sharded).
 *
 * Step 1 (per rank): row log-sum-exp and this block's per-column (max, sum exp) partials.
 *   row_lse  fp32 [rows];  col_part fp32 [2][B]  (col_part[0]=running max, [1]=sum exp(x-max))
 *   ws: triad_infonce_workspace_bytes(rows,B) (shared with step 2). */
int triad_infonce_partial(const float* clip_rows, int rows, int B, int row0,
                          float* row_lse, float* col_part,
                          void* ws, size_t ws_bytes, void* stream);
/* Step 2: given the column partials of all `nparts` row blocks (concatenated [nparts][2][B];
 * an all-gather of step 1's col_part), produce
 *   g     fp32 [rows,B] : dLoss/dclip = (softmax_row + softmax_col - 2 I)/(2B) * grad_scale
 *   sums  fp64 [8]      : {sum_i(row_lse-diag) + sum_{j in block}(col_lse-diag),  sum diag,
 *                          sum diag^2, sum offdiag, sum offdiag^2, max offdiag,
 *                          sum g*clip (unscaled), 0}   — block-local, to be summed (max for [5])
 *                          across ranks; loss = sums[0]/(2B).
 * ws: triad_infonce_workspace_bytes(rows,B). */
size_t triad_infonce_workspace_bytes(int rows, int B);
int triad_infonce_finish(const float* clip_rows, int rows, int B, int row0,
                         const float* row_lse, const float* col_parts, int nparts,
                         float grad_scale, float* g, double* sums,
                         void* ws, size_t ws_bytes, void* stream);

/* Fused single-device head: the whole B x B matrix is on this GPU (row0 = 0, rows = B).  Two launches produce
 * g and sums as triad_infonce_partial + triad_infonce_finish do (bit-identical), plus the scalars
 *   out4[0] = contrastive loss = sums[0]/(2B)                       (model.py:453-459 / :572-578)
 *   out4[1] = 20*relu(-log T)^2, the temperature-calibration term   (model.py:420-427); 0 when temperature == NULL
 *   out4[2] = out4[0] + out4[1]
 *   out4[3] = d out4[1] / dT
 * so the loss needs no further arithmetic on the host side.  B <= 2048 (TRIAD_ERR_UNSUPPORTED beyond: use the
 * partial/finish pair).  ws: triad_contrastive_head_workspace_bytes(B). */
size_t triad_contrastive_head_workspace_bytes(int B);
int triad_contrastive_head(const float* clip, int B, const float* temperature,
                           float* g, double* sums, float* out4,
                           void* ws, size_t ws_bytes, void* stream);

/* ---- backward through max-mean ------------------------------------------------------- */
/* Replaces autograd's backward of model.py:387-391 (SURVEY.md §8 a5):
 *   dq[i,a,:] = T*row_scale[r] * sum_j g[i,j] * v[j, idx[j][r], :]
 *   dv[j,p,:] = sum_{r: idx[j][r]==p} T*row_scale[r]*g[i(r),j] * q[r,:]
 *   dT        = sum_ij g[i,j]*clip[i,j] / T
 * g fp32 [Bq,Bv] is dLoss/dclip.  dq is written in `dtype` ([Bq,Nq,D]); dv is written as
 * fp32 [Bv,Nv,D] when dv_f32 != 0 (partial to be reduce-scattered across ranks) else in
 * `dtype`; dT fp32 [1].  Any of dq / dv / dT may be NULL to skip it.  dv needs Nv <= 3072: beyond,
 * the call fails with TRIAD_ERR_UNSUPPORTED before queueing any work.  `flags` is an OR of the
 * TRIAD_BWD_* bits below; any other bit (4, 8 and 64 are retired) fails with TRIAD_ERR_BAD_ARG. */
#define TRIAD_BWD_DEFAULT      0
#define TRIAD_BWD_GENERIC_DQ   1   /* L2-served gather kernel for dq (always used for fp32 / D % 64 != 0) */
#define TRIAD_BWD_GENERIC_DV   2   /* per-segment L2-served gather for dv                                 */
#define TRIAD_BWD_SMALL_BLOCKS 16   /* dv: 64 KB query blocks instead of 64 MB (test aid: multi-block path) */
#define TRIAD_BWD_PACK_ROWS   32   /* dq sweeps only the rows whose row_scale is non-zero (masked text tokens
                                      get an exact zero gradient without being gathered for)                */
#define TRIAD_BWD_UNIFORM_SCALE 128  /* the caller guarantees row_scale has no zeros (no attention mask): the dv sort then
                                      does not read it per row to decide which rows to list                            */
#define TRIAD_BWD_TEST_TRIP_WATCHDOG 256 /* test aid: raise the watchdog flag before the kernels run: dq must come back NaN */
#define TRIAD_BWD_ACCUMULATE_DV 1024 /* dv += the gradient instead of dv = (every query block adds to the caller's
                                        values, the first one included), so a row-sharded step can land one rank's
                                        contrastive dv on its dense-regulariser dV in one fp32 buffer; needs fp32 dv
                                        (dv_f32 != 0 or fp32 inputs), TRIAD_ERR_BAD_ARG otherwise */
size_t triad_maxmean_bwd_workspace_bytes(int Bq, int Bv, int Nq, int Nv, int D, int dtype);
int triad_maxmean_bwd(const void* q, const void* v, const void* idx, const float* g,
                      const float* clip, const float* row_scale, const float* temperature,
                      int Bq, int Bv, int Nq, int Nv, int D, int dtype,
                      void* dq, void* dv, int dv_f32, float* dT,
                      void* ws, size_t ws_bytes, int flags, void* stream);

/* ---- dense regulariser (SURVEY.md §8 f1) ----------------------------------------------- */
/* Elementwise stage of the "non-negative pressure" term, model.py:411-412 (lo = -60) and :525-526
 * (lo = -20):  l_nonneg = mean(clamp(S, lo, 0)^2) over ALL Bq*Bv*Nq*Nv token pairs, S = T*<q,v>.
 * `S` holds one chunk of RAW dot products <q,v> ([n] contiguous, `dtype`: the output of a
 * library GEMM of q rows against a block of patches).  The call
 *   sums[0] += sum clamp(round(T*raw), lo, 0)^2
 *   sums[1] += sum coef*clamp'(.)*raw            (this chunk's share of dL/dT)
 * and, when write_grad != 0, overwrites every element with dL/d(raw) =
 * coef * clamp(S,lo,0) * [S >= lo] * T in `dtype` (coef = 2*weight/numel chosen by the caller),
 * which the caller feeds to the two backward GEMMs (dQ += N V, dV = N^T Q).  Deterministic. */
size_t triad_nonneg_workspace_bytes(void);
int triad_nonneg_chunk(void* S, size_t n, int dtype, const float* temperature, float lo, float coef,
                       int write_grad, double* sums, void* ws, size_t ws_bytes, void* stream);

/* The same for bf16 embeddings straight from q and a block of images (D % 64 == 0, D <= 512, Nv <= 256,
 * Nv % 8 == 0): the tcgen05 forward kernel computes the similarities and its epilogue writes
 * n_out[r][j*Nv + p] = dL/d<q_r, v_jp> (bf16, row pitch ldn >= Bv*Nv elements, ldn % 8 == 0) when write_grad != 0,
 * accumulating sums[0..1] as above — no S chunk is materialised and there is no separate elementwise pass. */
size_t triad_nonneg_fused_workspace_bytes(void);
int triad_nonneg_fused_chunk(const void* q, const void* v, const float* temperature,
                             int Bq, int Bv, int Nq, int Nv, int D, float lo, float coef,
                             void* n_out, long long ldn, int write_grad, double* sums,
                             void* ws, size_t ws_bytes, void* stream);

/* The max-mean forward (triad_maxmean_fwd: clip, idx) AND the dense regulariser's N = dL/d<q,v> (as
 * triad_nonneg_fused_chunk with write_grad = 1, all Bv images in one call; sums[0..1] accumulated) from ONE pass over
 * the similarities: the training step with the reference's full loss (model.py:430-472 calls both on the same
 * token_sims) needs both of every tile.  bf16, D % 64 == 0, D <= 512, Nv <= 256, Nv % 8 == 0, all rows (padded text
 * tokens take part in the regulariser, model.py:525, so rows are not packed).  flags: TRIAD_FWD_FORCE_1CTA,
 * TRIAD_FWD_SYNC_CHUNKS. */
size_t triad_maxmean_fwd_nonneg_workspace_bytes(int Bq, int Bv, int Nq, int Nv, int D);
int triad_maxmean_fwd_nonneg(const void* q, const void* v, const float* row_scale, const float* temperature,
                             int Bq, int Bv, int Nq, int Nv, int D, float* clip, void* idx,
                             float lo, float coef, void* n_out, long long ldn, double* sums,
                             void* ws, size_t ws_bytes, int flags, void* stream);

/* The two backward GEMMs of the dense regulariser, hand-written (tcgen05, cta_group::2, MN-major operands: no
 * transposed copies).  n_mat = N = dL/d<q,v> as written by triad_maxmean_fwd_nonneg / triad_nonneg_fused_chunk
 * ([M][ldn] bf16, Kc = Bv*Nv valid columns).  mode 0: out[M][D] = N . x with x = the patches [Kc][D] (dQ, autograd of
 * model.py:384-387 w.r.t. the query embeddings); mode 1: out[Kc][D] = N^T . x with x = the tokens [M][D] (dV).
 * bf16 in, fp32 accumulation, bf16 out; D % 8 == 0, D <= 512.  Deterministic (K splits are added in order). */
size_t triad_dense_grad_gemm_workspace_bytes(int M, int Kc, int D, int mode);
int triad_dense_grad_gemm(const void* n_mat, long long ldn, int M, int Kc, const void* x, int D, int mode,
                          void* out, void* ws, size_t ws_bytes, void* stream);
/* The same product with an fp32 output (same workspace query).  accumulate = 0: out = sum of the K splits in order
 * (bf16(out) is bit for bit what triad_dense_grad_gemm writes); accumulate = 1: out = out + (sum of the splits in
 * order), added once per element, so a zero `out` ends up equal to accumulate = 0.  Deterministic, no atomics.  Lets a
 * caller carry dQ across image chunks in fp32, or write a chunk's dV straight into its rows of a larger fp32 buffer.
 * Any other `accumulate` fails with TRIAD_ERR_BAD_ARG. */
int triad_dense_grad_gemm_f32(const void* n_mat, long long ldn, int M, int Kc, const void* x, int D, int mode,
                              float* out, int accumulate, void* ws, size_t ws_bytes, void* stream);

/* Regularisers on the B POSITIVE pairs only (token_sims[i,i]): temporal smoothness (mode 0, model.py:394-408:
 * mean over (i, a < Nq-1, p) of (S[i,a+1,p] - S[i,a,p])^2) and patch-usage sparsity (mode 1, model.py:528-541:
 * softmax over patches, usage fraction per patch over ALL Nq token rows, mean of relu(frac - threshold)^2).
 * `raw` [B,Nq,Nv] (`dtype`) holds the raw dot products <q[i,a], v[i,p]> of the diagonal blocks (one small batched
 * library GEMM); S = round(T*raw) as in model.py:387.  One pass writes G = d value / d raw (same shape and dtype; the
 * operand of the two small backward GEMMs dq_i = G_i v_i, dv_i = G_i^T q_i) and sums[0] = value,
 * sums[1] = d value / dT.  Replaces ~40 ATen kernels of the reference's autograd graph.  Deterministic. */
size_t triad_pospair_workspace_bytes(int B);
int triad_pospair_terms(const void* raw, int dtype, const float* temperature, int mode, float threshold,
                        int B, int Nq, int Nv, void* G, double* sums, void* ws, size_t ws_bytes, void* stream);

/* y[k] = x[k] * (*scale) for n elements of `dtype`; `scale` is an fp32 scalar in DEVICE memory (the upstream
 * gradient of a loss term inside autograd's backward: no host synchronisation).  x == y is allowed. */
int triad_scale(const void* x, void* y, size_t n, int dtype, const float* scale, void* stream);

/* ---- retrieval: one query against a gallery, top-k ---------------------------------- */
/* Replaces the per-pair aggregators retrieval.py:106-110 / :190-193 (direction 0:
 * mean_q max_p) and :112-115 / :195-198 (direction 1: mean_p max_q) and the python double
 * loops at :161-175 / :265-279: scores[n] for n in [0,n_img), each image Nv patches.
 * The retrieval path DIVIDES by the temperature (retrieval.py:108); `divide_by_T` selects
 * that (1) or the training-time multiply (0).  scores fp32 [n_img]. */
size_t triad_retrieve_workspace_bytes(int Nq, int n_img, int Nv, int D, int dtype);
int triad_retrieve_scores(const void* q, int Nq, const void* gallery, int n_img, int Nv, int D,
                          int dtype, const float* temperature, int divide_by_T, int direction,
                          float* scores, void* ws, size_t ws_bytes, void* stream);
/* ---- retrieval on an e4m3 gallery (opt-in compressed storage; direction 0 only) ------- */
/* Per-row quantization: for each row x[0..D) of `x` ([rows][D], `dtype` fp32 or bf16)
 *   s = fp32(max_k |x_k| / 448),  codes[k] = e4m3_rn_satfinite(fp32(x_k / s)) if s > 0, else 0;
 * a row holding an inf or a NaN gets s = NaN.  codes [rows][D] (one e4m3 byte each), scales fp32 [rows].
 * D % 16 == 0, D <= 512; x and codes 16-byte aligned. */
int triad_quantize_e4m3(const void* x, int dtype, long long rows, int D, void* codes, float* scales, void* stream);
/* scores[n] = sum_a fp32(m_a * t_a), m_a = max_p fp32(g_scales[n][p] * acc_ap), acc_ap = sum_k q_codes[a][k] *
 * g_codes[n][p][k] (tensor cores, fp32 accumulation), t_a = fp32(fp32(q_scales[a] * (1/Nq)) * fp32(1/T)): the
 * direction-0 retrieval score (mean over query tokens of max over patches, divided by T) of the quantized operands.
 * q_codes [Nq][D], g_codes [n_img][Nv][D] as written by triad_quantize_e4m3; D in {128, 256, 384, 512}
 * (TRIAD_ERR_UNSUPPORTED otherwise).  Deterministic; a watchdog timeout gives NaN scores. */
size_t triad_retrieve_e4m3_workspace_bytes(int Nq, int n_img, int Nv, int D);
int triad_retrieve_scores_e4m3(const void* q_codes, const float* q_scales, int Nq, const void* g_codes,
                               const float* g_scales, int n_img, int Nv, int D, const float* temperature,
                               float* scores, void* ws, size_t ws_bytes, void* stream);
/* ---- retrieval on a ragged caption gallery (bf16, items of 1..256 tokens) ------------------------------------
 * Layout: the captions' token rows in 256-row slots, slots [n_slots * 256][D] bf16.  Captions are placed greedily
 * in order; one that does not fit in the rest of the current slot starts a new slot (no caption straddles a slot);
 * the rows after a slot's last caption are zero.
 * triad_ragged_plan (host only, no CUDA call): from lengths[n_cap] (host, each 1..256, else TRIAD_ERR_BAD_SHAPE)
 * writes the host arrays slot_meta [n_slots][20] int32 = {first caption id, caption count, used rows, 0,
 * caption-start mask [8] (bit r%32 of word r/32: a caption starts at row r), caption-end mask [8] (its last row)}
 * and cap_info [n_cap][2] int32 = {first row (slot * 256 + offset), length}, and *n_slots.  slot_meta needs room
 * for n_cap slots (the most there can be). */
int triad_ragged_plan(const int32_t* lengths, int n_cap, int32_t* slot_meta, int32_t* cap_info, int* n_slots);
/* dst[r] = bf16(src[rowmap[r]]) for r < dst_rows (a multiple of 256), a zero row where rowmap[r] < 0 or
 * rowmap[r] >= src_rows; src [src_rows][D] fp32 or bf16 (dtype), D % 8 == 0, src and dst 16-byte aligned. */
int triad_ragged_pack(const void* src, int dtype, long long src_rows, int D, const int32_t* rowmap, long long dst_rows,
                      void* dst, void* stream);
/* scores[c] for one query q [Nq][D] bf16 against the n_cap captions of a ragged gallery (slot_meta and cap_info as
 * triad_ragged_plan wrote them, on the device), divided by T:
 *   direction 0: mean over the query's tokens of the max over caption c's tokens (the V->T ranking, the
 *                reference's aggregator_tv_v2t with the image as query);
 *   direction 1: mean over caption c's tokens of the max over the query's tokens (aggregator_tv_t2v).
 * Each similarity is rounded as the dense retrieval forward rounds it, bf16(bf16(acc) * (1/T)).  The sums are
 * deterministic (fixed-order partials, no float atomics) and do not depend on where a caption sits in the slots.  D in {64, ..., 512} (multiple of 64,
 * TRIAD_ERR_UNSUPPORTED otherwise), 1 <= Nq <= 65535; q, slots and ws 16-byte aligned.  No host synchronisation;
 * a watchdog timeout gives NaN scores. */
size_t triad_retrieve_ragged_workspace_bytes(int Nq, int n_slots, int n_cap, int direction);
int triad_retrieve_scores_ragged(const void* q, int Nq, const void* slots, const int32_t* slot_meta,
                                 const int32_t* cap_info, int n_slots, int n_cap, int D, const float* temperature,
                                 int direction, float* scores, void* ws, size_t ws_bytes, void* stream);
/* ---- the ragged caption gallery stored as e4m3 codes with one fp32 scale per slot row --------------------------
 * triad_ragged_pack_e4m3: codes[r], scales[r] = triad_quantize_e4m3 of src[rowmap[r]] for r < dst_rows (a multiple
 * of 256), bit for bit; a zero row (scale 0, codes 0) where rowmap[r] < 0 or rowmap[r] >= src_rows.  fp32 input is
 * quantized as it is (not rounded to bf16 first).  src [src_rows][D] fp32 or bf16 (dtype), D in {128, 256, 384, 512}
 * (TRIAD_ERR_UNSUPPORTED otherwise); src and codes 16-byte, rowmap and scales 4-byte aligned. */
int triad_ragged_pack_e4m3(const void* src, int dtype, long long src_rows, int D, const int32_t* rowmap,
                           long long dst_rows, void* codes, float* scales, void* stream);
/* scores[c] for one query, quantized per token by triad_quantize_e4m3 (q_codes [Nq][D], q_scales [Nq]), against the
 * captions of an e4m3 ragged gallery (codes [n_slots * 256][D], scales [n_slots * 256] from triad_ragged_pack_e4m3;
 * slot_meta and cap_info as for triad_retrieve_scores_ragged).  acc = the tensor-core dot product of the codes (fp32
 * accumulation), s_t the scale of slot row t, sq_a the scale of query token a:
 *   direction 0: sum_a fp32(m_ac * t_a), m_ac = max_{t in c} fp32(s_t * acc_at),
 *                t_a = fp32(fp32(sq_a * (1/Nq)) * (1/T)), the sum in the dense forward's 32-row-group order;
 *   direction 1: sum_{t in c, token order} fp32(m_t * w_t), m_t = max_a fp32(sq_a * acc_ta),
 *                w_t = fp32(fp32(s_t * (1/length_c)) * (1/T)).
 * The maxima propagate NaN: a caption row holding an inf or a NaN makes that caption's score NaN, a non-finite
 * query token every score.  D in {128, 256, 384, 512}; the workspace is triad_retrieve_ragged_workspace_bytes;
 * q_codes, codes and ws 16-byte, metadata 8-byte, scales and scores 4-byte aligned.  Deterministic, position
 * independent, no host synchronisation; a watchdog timeout gives NaN scores. */
int triad_retrieve_scores_ragged_e4m3(const void* q_codes, const float* q_scales, int Nq, const void* codes,
                                      const float* scales, const int32_t* slot_meta, const int32_t* cap_info,
                                      int n_slots, int n_cap, int D, const float* temperature, int direction,
                                      float* scores, void* ws, size_t ws_bytes, void* stream);
/* top-k of scores (descending, ties -> lower id first, like a stable argsort of -scores;
 * -0.0 and +0.0 are equal scores): out_scores fp32 [k] = scores[out_ids], bit for bit,
 * out_ids int32 [k].  NaN scores have no defined place.  ws: triad_topk_workspace_bytes(n). */
size_t triad_topk_workspace_bytes(int n, int k);
int triad_topk(const float* scores, int n, int k, float* out_scores, int32_t* out_ids,
               void* ws, size_t ws_bytes, void* stream);
/* rank of the diagonal in each row of an N x N similarity matrix (retrieval.py:125-133):
 * ranks int32 [N] = #{j : sim[i,j] > sim[i,i]} + #{j < i : sim[i,j] == sim[i,i]}, the position
 * of i in a stable argsort of -sim[i].  NaN sorts last: a NaN entry ranks below every number, and
 * a NaN diagonal gets #{j : sim[i,j] is not NaN} + #{j < i : sim[i,j] is NaN}. */
int triad_diag_ranks(const float* sim, int N, int32_t* ranks, void* stream);

/* ---- per-pair normalised similarity (viz / forward()) -------------------------------- */
/* Replaces compute_similarity_matrix (model.py:355-368): out[b,n1,n2] =
 * T * <f1[b,n1]/|f1[b,n1]|, f2[b,n2]/|f2[b,n2]|>, fp32 in/out. */
int triad_similarity_matrix(const float* f1, const float* f2, const float* temperature,
                            int B, int N1, int N2, int D, float* out, void* stream);

/* ---- producers of the hot path's inputs (SURVEY.md §8 f3) -------------------------------- */
/* The projection head of the audio / text / visual embedders, fused: replaces
 *   projection2(layer_norm(projection1(x)))     model.py:32-34,68 / :81-83,116 / :253-255,326
 * and, with l2_normalize != 0, the F.normalize(feats, dim=-1) of retrieval.py:93-94.
 * x bf16 [M, Din] (token rows of the encoder output, flattened over the batch), w1 bf16 [512, Din] and w2 bf16
 * [Dout, 512] in nn.Linear's own [out, in] layout, b1 / ln_g / ln_b fp32 [512], b2 fp32 [Dout]; out bf16 [M, Dout],
 * i.e. [B, N, D] with D innermost — the layout triad_maxmean_fwd reads.  Arithmetic follows the reference under
 * autocast: bf16 GEMMs with fp32 accumulation, Linear outputs rounded to bf16, LayerNorm in fp32.
 * Din % 64 == 0, Dout % 16 == 0, Dout <= 512.  ws: triad_project_workspace_bytes(). */
size_t triad_project_workspace_bytes(void);
int triad_project_tokens(const void* x, const void* w1, const float* b1, const float* ln_g, const float* ln_b,
                         float ln_eps, const void* w2, const float* b2, int M, int Din, int Dout, int l2_normalize,
                         void* out, void* ws, size_t ws_bytes, void* stream);
/* Patch dropout's compaction (model.py:283-307 without the per-image loop): for every image the patches with
 * keep[b][n] != 0 are copied, in order, to the front of out[b] ([B, max_len, D], same element type as x) and the
 * remaining rows are zero-filled.  max_len >= the largest kept count (the caller sizes the output, as the
 * reference's max(...) does).  D*elt_bytes % 16 == 0. */
int triad_patch_compact(const void* x, const uint8_t* keep, int B, int N, int D, int elt_bytes, int max_len,
                        void* out, void* stream);

/* Backward of triad_project_tokens (l2_normalize = 0) for gy = dLoss/dout, bf16 [M, Dout] (e.g. the dq / dv that
 * triad_maxmean_bwd writes).  x, w1, b1, ln_g, ln_b, ln_eps and w2 are the forward's arguments (b2 is not needed).
 * The hidden activations are recomputed from x with the forward's arithmetic (bit-identical LayerNorm statistics).
 * Outputs, each optional (NULL skips it; dx / dw1 / dw2 skip their GEMM):
 *   dx  bf16 [M, Din]      dw1 fp32 [512, Din]     db1 fp32 [512]
 *   dln_g, dln_b fp32 [512]                        dw2 fp32 [Dout, 512]    db2 fp32 [Dout]
 * Weight gradients are fp32 sums of fp32 products of bf16 operands (not rounded to bf16).  Deterministic: every
 * reduction over tokens adds fixed partial sums in a fixed order, no float atomics.  Shapes as the forward:
 * Din % 64 == 0, Dout % 16 == 0, Dout <= 512, any M >= 1.  x, w1, w2, gy, dx, dw1, dw2 and ws 16-byte aligned, the
 * fp32 vectors 4-byte aligned.  ws: triad_project_tokens_bwd_workspace_bytes(M, Din, Dout) (it holds the bf16
 * [M, 512] hidden gradient and LayerNorm output, about 2 KB per token). */
size_t triad_project_tokens_bwd_workspace_bytes(int M, int Din, int Dout);
int triad_project_tokens_bwd(const void* x, const void* w1, const float* b1, const float* ln_g, const float* ln_b,
                             float ln_eps, const void* w2, const void* gy, int M, int Din, int Dout,
                             void* dx, float* dw1, float* db1, float* dln_g, float* dln_b, float* dw2, float* db2,
                             void* ws, size_t ws_bytes, void* stream);
/* Backward of triad_patch_compact (same keep, B, N, D, elt_bytes, max_len): gx[b][n] = keep[b][n] ? gy[b][slot] : 0,
 * where slot is patch n's position among image b's kept patches; gy [B, max_len, D], gx [B, N, D], one launch, no
 * host synchronisation.  A pure copy: bit-identical to indexing gy. */
int triad_patch_expand(const void* gy, const uint8_t* keep, int B, int N, int D, int elt_bytes, int max_len,
                       void* gx, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* TRIAD_B200_H */
