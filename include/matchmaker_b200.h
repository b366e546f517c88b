/*
 * matchmaker_b200 -- C ABI of the B200-native interaction-scoring library.
 *
 * This is the drop-in boundary for the query-document interaction hot path of
 * sebastian-hofstaetter/matchmaker.  The reference is pure Python/PyTorch and has no FFI of
 * its own; each entry point below replaces the *inline arithmetic* of one reference method
 * (cited as path:line relative to the reference repository root) and is what a binding for
 * that method calls.  The Python host layer (matchmaker_b200/) binds these symbols with
 * ctypes; INTEGRATION.md shows the stub a maintainer of the reference would add.
 *
 * Conventions
 *   - plain pointers and sizes only; no torch / C++ types cross this boundary;
 *   - every function returns 0 (MMB200_OK) or a negative MMB200_ERR_* code;
 *     mmb200_last_error() returns a thread-local human-readable message for the last failure;
 *   - pointers whose name does not end in `_host` are DEVICE pointers valid on the CURRENT
 *     CUDA device of the calling thread; `stream` is a cudaStream_t (0 = legacy default);
 *     launches are asynchronous with respect to the host and ordered on `stream`;
 *   - tensors are dense row-major ("contiguous" in PyTorch terms) unless a stride is given;
 *   - the library never falls back to a CPU implementation: on a device that is not
 *     compute capability 10.x every compute entry point fails with MMB200_ERR_UNSUPPORTED.
 */
#ifndef MATCHMAKER_B200_H_
#define MATCHMAKER_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MMB200_VERSION 100 /* 0.1.0 */

#if defined(__GNUC__)
#define MMB200_API __attribute__((visibility("default")))
#else
#define MMB200_API
#endif

/* error codes */
#define MMB200_OK 0
#define MMB200_ERR_INVALID (-1)     /* bad argument (shape, dtype, alignment, null pointer) */
#define MMB200_ERR_CUDA (-2)        /* a CUDA runtime / driver call failed */
#define MMB200_ERR_UNSUPPORTED (-3) /* device is not sm_100, or shape outside kernel limits */

/* element types of embedding / vector tensors */
#define MMB200_F16 0
#define MMB200_BF16 1
#define MMB200_F32 2
#define MMB200_F32_SPLIT16 3 /* mmb200_flat_ip_topk only: fp32 vectors held as fp16 hi / lo halves (see there) */

/* element types of mask tensors (nonzero = real token, zero = padding) */
#define MMB200_MASK_NONE 0
#define MMB200_MASK_U8 1  /* torch.bool / uint8 */
#define MMB200_MASK_I32 2
#define MMB200_MASK_I64 3 /* HF attention_mask */
#define MMB200_MASK_F32 4 /* matchmaker `(tokens > 0).float()` masks */

/* kernel selection for entry points that have more than one device implementation */
#define MMB200_IMPL_AUTO 0
#define MMB200_IMPL_SIMT 1    /* CUDA-core kernel, any shape/dtype */
#define MMB200_IMPL_TCGEN05 2 /* TMA + tcgen05 tensor-core kernel (fails if shape unsupported) */
#define MMB200_IMPL_TCGEN05_DOCM 3 /* max-sim only: the first-generation "documents on M" tcgen05 kernel */
#define MMB200_IMPL_TCGEN05_RAGGED 4 /* max-sim only: tcgen05 kernel that fetches each document only up to its
                                        last unmasked row (padding rows never leave HBM / host memory) */

MMB200_API int mmb200_version(void);
MMB200_API const char* mmb200_last_error(void);

/* Properties of CUDA device `device` (-1 = current). Any out pointer may be NULL. */
MMB200_API int mmb200_device_info(int device, int* sm_count, int* cc_major, int* cc_minor);

/* ------------------------------------------------------------------------------------------
 * ColBERT late-interaction max-sim
 *
 *   score[p] = sum_{i < Lq, q_mask[qi][i]} max_{j < Ld} ( d_mask[di][j] ? <q[qi][i], d[di][j]> : -1000 )
 *
 * Replaces: ColBERT.forward scoring            matchmaker/models/colbert.py:68-75   (masks given)
 *           ColBERT.forward_aggregation        matchmaker/models/colbert.py:100-112 (masks NULL)
 *           ColBERT.forward_inbatch_aggregation matchmaker/models/colbert.py:154-162
 *               (all pairs: n_pairs = n_q * n_d, pair_q[p] = p / n_d, pair_d[p] = p % n_d, or
 *                mmb200_maxsim_allpairs_fwd below)
 *
 * q      [n_q, Lq, dim]  dtype `dtype`
 * d      [n_d, Ld, dim]  dtype `dtype`
 * q_mask [n_q, Lq] or NULL, d_mask [n_d, Ld] or NULL, element type `mask_dtype`
 * pair_q / pair_d [n_pairs] int32 or NULL.  With NULL: qi = p / docs_per_query, di = p
 *        (docs_per_query = 1 is the training/re-ranking case "pair p = query p x doc p";
 *         docs_per_query = 1000 is BASELINE config 3 "1 query x 1000 docs").
 * pair_dmask [n_pairs] int32 or NULL: row of d_mask applied to pair p (default di).  Exists only
 *        to reproduce colbert.py:158, which indexes the document mask by the QUERY position.
 * out    [n_pairs] float32
 * argmax [n_pairs, Lq] int32 or NULL: index j* of the first max per query token (-1 when the
 *        query token is masked or the -1000 fill is the max) -- what backward needs.
 * Envelope: 1 <= Lq <= 128, 1 <= dim <= 1024, Ld >= 1 (else MMB200_ERR_INVALID); IMPL_AUTO serves
 *        all of it, a forced impl returns MMB200_ERR_UNSUPPORTED where its kernel does not apply.
 * ------------------------------------------------------------------------------------------ */
MMB200_API int mmb200_maxsim_fwd(const void* q, const void* d, const void* q_mask, const void* d_mask,
                      const int32_t* pair_q, const int32_t* pair_d, const int32_t* pair_dmask,
                      float* out, int32_t* argmax,
                      int64_t n_q, int64_t n_d, int64_t n_pairs, int32_t docs_per_query, int32_t Lq,
                      int32_t Ld, int32_t dim, int32_t dtype, int32_t mask_dtype, int32_t impl,
                      void* stream);

/* Backward of mmb200_maxsim_fwd (pairs mode with pair_q = pair_d = NULL, docs_per_query >= 1).
 * grad_out [n_pairs] f32; argmax from the forward; grad_q [n_q, Lq, dim] f32 and
 * grad_d [n_d, Ld, dim] f32 are OVERWRITTEN (zero-filled then accumulated).
 * Mirrors what autograd derives from colbert.py:68-75 (gradient flows only through the max
 * element; masked query tokens and fully masked documents get none). */
MMB200_API int mmb200_maxsim_bwd(const void* q, const void* d, const float* grad_out, const int32_t* argmax,
                      float* grad_q, float* grad_d, int64_t n_q, int64_t n_d, int64_t n_pairs,
                      int32_t docs_per_query, int32_t Lq, int32_t Ld, int32_t dim, int32_t dtype,
                      void* stream);

/* Host-buffer variant (the end-to-end call): all pointers are HOST pointers (pinned memory
 * gives full PCIe bandwidth, pageable works).  Documents are streamed to the device in chunks
 * on internal streams, overlapped with the kernel; scores are copied back before returning.
 * Synchronous.  Same semantics as mmb200_maxsim_fwd with pair_q = pair_d = NULL.
 * When d_host is pinned (device-mapped) memory and the shape fits the queries-on-M kernel, the
 * documents are not staged at all: the kernel's TMA reads them directly over PCIe, 16 rows at a time, and
 * only up to each document's last unmasked row.  chunk_pairs: 0 = default slab size, -1 = force the
 * staged (slab) pipeline. */
MMB200_API int mmb200_maxsim_fwd_host(const void* q_host, const void* d_host, const void* q_mask_host,
                           const void* d_mask_host, float* out_host, int64_t n_q, int64_t n_d,
                           int32_t docs_per_query, int32_t Lq, int32_t Ld, int32_t dim, int32_t dtype,
                           int32_t mask_dtype, int64_t chunk_pairs);

/* ------------------------------------------------------------------------------------------
 * Cosine match matrix + RBF kernel pooling (KNRM / TK)
 *
 *   c_ij  = <q_i/(|q_i|+1e-13), d_j/(|d_j|+1e-13)>
 *   S_ik  = sum_j d_mask[j] * exp(-(c_ij - mu_k)^2 / (2 sigma_k^2))
 *   P_k   = sum_i q_mask[i] * log_scale * log(max(alpha_k * S_ik, 1e-10))
 *   score = sum_k weight_k * P_k
 *
 * Replaces: KNRM.forward        matchmaker/models/knrm.py:52-84        (alpha = NULL, log_scale = 0.01)
 *           ECAI20_TK.forward   matchmaker/models/published/ecai20_tk.py:105-124 (log_scale = 1)
 *           CosineMatrixAttention (allennlp 2.5.1, third party) at knrm.py:60, ecai20_tk.py:105
 *
 * q [B,Lq,D] f32, d [B,Ld,D] f32 (D % 4 == 0, 16-byte aligned); q_mask [B,Lq], d_mask [B,Ld] of
 * `mask_dtype` (matchmaker passes float masks: MMB200_MASK_F32); mu, sigma, weight [K] f32 device
 * arrays, alpha [K] or NULL (= 1); K <= 32.
 * Outputs (any of per_kernel / per_kernel_query / cosine may be NULL):
 *   score [B]; per_kernel [B,K] (= P); per_kernel_query [B,Lq,K] (= S, what backward needs);
 *   cosine [B,Lq,Ld] = c_ij * q_mask[i] * d_mask[j] (the reference's secondary output).
 * impl: MMB200_IMPL_AUTO / _TCGEN05 take the tensor-core kernel for K <= 32, Lq <= 128, cosine == NULL (queries longer
 * than 32 terms: one pass per block of 32 query rows), _SIMT the FFMA kernel (any Lq).
 * ------------------------------------------------------------------------------------------ */
MMB200_API int mmb200_kernel_pool_fwd(const float* q, const float* d, const void* q_mask, const void* d_mask,
                                      const float* mu, const float* sigma, const float* alpha,
                                      const float* weight, float* score, float* per_kernel,
                                      float* per_kernel_query, float* cosine, int64_t B, int32_t Lq,
                                      int32_t Ld, int32_t D, int32_t K, float log_scale, int32_t mask_dtype,
                                      int32_t impl, void* stream);

/* Backward of mmb200_kernel_pool_fwd for d(loss)/d(score) = grad_score [B]:
 *   grad_q [B,Lq,D], grad_d [B,Ld,D] (overwritten), grad_alpha [K] or NULL, grad_weight [K]
 *   (overwritten; summed over the batch deterministically via `workspace` [2*B*K] f32).
 * per_kernel_query is S from the forward.  Matches autograd of the reference expression
 * (clamp passes gradient when alpha*S >= 1e-10; rows with |x| = 0 get no normalisation term). */
MMB200_API int mmb200_kernel_pool_bwd(const float* q, const float* d, const void* q_mask, const void* d_mask,
                                      const float* mu, const float* sigma, const float* alpha,
                                      const float* weight, const float* per_kernel_query,
                                      const float* grad_score, float* grad_q, float* grad_d,
                                      float* grad_alpha, float* grad_weight, float* workspace, int64_t B,
                                      int32_t Lq, int32_t Ld, int32_t D, int32_t K, float log_scale,
                                      int32_t mask_dtype, void* stream);

/* Variants of the same pooling (SURVEY 8(f) row 3) -- mmb200_kernel_pool_fwd / _bwd are these with doc_gate = NULL,
 * clamp_min = 1e-10, score_bias = 0:
 *   doc_gate [B, Ld] f32 or NULL: multiplier of every activation of document term j (negative values count as 0),
 *            S_ik = sum_j d_mask[j] * doc_gate[j] * exp(...).  Replaces the `* document_stop_words` of
 *            CIKM20_TK_Sparse.forward, matchmaker/models/published/cikm20_tk_sparse.py:135.
 *   clamp_min: floor of alpha_k * S_ik before the log.  IDCM's ESM patch scorer uses 1e-4
 *            (matchmaker/models/published/sigir21_idcm.py:185).
 *   score_bias: added to the score (the bias of IDCM's `sampling_binweights` Linear(11, 1), sigir21_idcm.py:100,186).
 *   Conv-KNRM's n x n cross matches (matchmaker/models/conv_knrm.py:125-135) are n*n calls with log_scale = 0.01, each
 *   taking its K-slice of dense.weight (Linear over a concatenation = sum of per-block Linears).
 * Backward additionally returns grad_gate [B, Ld] (or NULL): d(loss)/d(doc_gate). */
MMB200_API int mmb200_kernel_pool_fwd_ex(const float* q, const float* d, const void* q_mask, const void* d_mask,
                                         const float* doc_gate, const float* mu, const float* sigma, const float* alpha,
                                         const float* weight, float* score, float* per_kernel, float* per_kernel_query,
                                         float* cosine, int64_t B, int32_t Lq, int32_t Ld, int32_t D, int32_t K,
                                         float log_scale, float clamp_min, float score_bias, int32_t mask_dtype,
                                         int32_t impl, void* stream);
MMB200_API int mmb200_kernel_pool_bwd_ex(const float* q, const float* d, const void* q_mask, const void* d_mask,
                                         const float* doc_gate, const float* mu, const float* sigma, const float* alpha,
                                         const float* weight, const float* per_kernel_query, const float* grad_score,
                                         float* grad_q, float* grad_d, float* grad_gate, float* grad_alpha,
                                         float* grad_weight, float* workspace, int64_t B, int32_t Lq, int32_t Ld,
                                         int32_t D, int32_t K, float log_scale, float clamp_min, int32_t mask_dtype,
                                         void* stream);

/* Training pair on the tensor cores (the step of train.py:330-360 for KNRM / TK: forward, loss, backward).
 *   mmb200_kernel_pool_fwd_train = mmb200_kernel_pool_fwd_ex (tcgen05 kernel; doc_gate as there, or NULL) that additionally leaves
 *   `saved` for the backward: mmb200_kernel_pool_saved_floats(B, Ld) = B * (33 * Ld + 32) floats, 16-byte aligned
 *   (cosines document-row-major [B][Ld][32], then 1 / (|d_j| + eps) [B][Ld], then 1 / (|q_i| + eps) [B][32]); the
 *   layout is private to the pair of calls.
 *   mmb200_kernel_pool_bwd_saved = mmb200_kernel_pool_bwd_ex (doc_gate / grad_gate as there, or NULL) computed from `saved` with both contractions
 *   (G q^ and G^T d^) as kind::tf32 UMMAs on the raw fp32 tiles; gradients agree with the fp32 expression to a few
 *   1e-4 relative (tf32 operands; the reference trains under fp16 autocast).  grad_q / grad_d must be 16-byte aligned.
 *   Envelope: mmb200_kernel_pool_train_tc_supported(Lq, Ld, D, K) != 0  (Lq <= 32, K <= 32, D % 4 == 0, D <= 320);
 *   outside it both calls return MMB200_ERR_UNSUPPORTED and the caller uses _fwd_ex / _bwd_ex. */
MMB200_API int32_t mmb200_kernel_pool_train_tc_supported(int32_t Lq, int32_t Ld, int32_t D, int32_t K);
MMB200_API int64_t mmb200_kernel_pool_saved_floats(int64_t B, int32_t Ld);
MMB200_API int mmb200_kernel_pool_fwd_train(const float* q, const float* d, const void* q_mask, const void* d_mask,
                                            const float* doc_gate, const float* mu, const float* sigma, const float* alpha,
                                            const float* weight, float* score, float* per_kernel, float* per_kernel_query, float* saved,
                                            int64_t B, int32_t Lq, int32_t Ld, int32_t D, int32_t K, float log_scale,
                                            float clamp_min, float score_bias, int32_t mask_dtype, void* stream);
MMB200_API int mmb200_kernel_pool_bwd_saved(const float* q, const float* d, const void* q_mask, const void* d_mask,
                                            const float* doc_gate, const float* mu, const float* sigma, const float* alpha,
                                            const float* weight, const float* per_kernel_query, const float* saved,
                                            const float* grad_score, float* grad_q, float* grad_d, float* grad_gate,
                                            float* grad_alpha, float* grad_weight,
                                            float* workspace, int64_t B, int32_t Lq, int32_t Ld, int32_t D, int32_t K,
                                            float log_scale, float clamp_min, int32_t mask_dtype, void* stream);

/* ------------------------------------------------------------------------------------------
 * BERT_DOT pair scoring: out[b] = <q[b], d[b]>, fp32 accumulate.
 * Replaces: BERT_Dot.forward   matchmaker/models/bert_dot.py:62  (bmm([B,1,dim],[B,dim,1]))
 * q, d [B, dim] of `dtype`; out [B] f32.
 * ------------------------------------------------------------------------------------------ */
MMB200_API int mmb200_dot_pairs(const void* q, const void* d, float* out, int64_t B, int32_t dim,
                                int32_t dtype, void* stream);

/* ------------------------------------------------------------------------------------------
 * TKL (long documents): per-chunk cosine + RBF kernels, sliding-window kernel pooling with learned
 * saturation, window scores; then the greedy top-3 window selection.
 *
 * Replaces: TKL_sigir20.forward   matchmaker/models/published/sigir20_tkl.py:180-252 (window scores)
 *                                 matchmaker/models/published/sigir20_tkl.py:254-286 (top hills)
 * Chunking / packing / contextualisation (:136-175) stay in PyTorch, as in the reference.
 *
 * q             [B, Lq, D] f32  contextualised, masked query embeddings (Lq <= 40)
 * q_mask        [B, Lq] (`mask_dtype`)
 * chunks        [Nc, 40, D] f32 contextualised packed chunks, overlap removed (:174)
 * chunk_mask    [Nc, 40]
 * slot_to_packed [B*C] int32: packed index of chunk slot (b, c), -1 where the reference's
 *               `packed_indices` (:159) dropped the chunk
 * mu, sigma, dense_w [K] (K <= 16)
 * saturation 0 ("embedding", :222-234): sat_red_w [D] = sat_emb_reduce1.weight, sat_params[13] =
 *               {sat_normer.weight[2], sat_normer.bias[2], saturation_linear.weight[2], .bias,
 *                saturation_linear2.weight[2], .bias, saturation_linear3.weight[2], .bias}
 * saturation 1 ("log", :245-246): sat_params[K] = kernel_mult[0]
 * window_score  [B, W] f32 out, W = (C*40 - 30)/2 + 1  (raw dense output, sentinel not yet applied)
 * n_chunks      Nc (rows of `chunks` / `chunk_mask`)
 * impl          MMB200_IMPL_AUTO: the TMA + tcgen05 kernel (Lq * K <= 512) when the kernel set activates on every cosine
 *               in [-1, 1] -- decided on the device, no host sync -- else the FFMA kernel; _TCGEN05 / _SIMT force one.
 * ------------------------------------------------------------------------------------------ */
MMB200_API int mmb200_tkl_window_scores(const float* q, const void* q_mask, const float* chunks,
                                        const void* chunk_mask, const int32_t* slot_to_packed,
                                        const float* mu, const float* sigma, const float* dense_w,
                                        const float* sat_red_w, const float* sat_params,
                                        float* window_score, int64_t B, int64_t n_chunks, int32_t Lq, int32_t D,
                                        int32_t C, int32_t K, int32_t saturation, int32_t mask_dtype, int32_t impl,
                                        void* stream);

/* window_score [B,W] in; orig_score [B,W] out (may be the same buffer): the reference's "orig_score" (exact zeros ->
 * -9900 sentinel during selection, written back as 0).  chunk_scoring [15]; top_idx [B,3] int64;
 * top15 [B,15] ("top_k_non_overlapping"); score [B]. */
MMB200_API int mmb200_tkl_top_hills(const float* window_score, float* orig_score, const float* chunk_scoring,
                                    int64_t* top_idx, float* top15, float* score, int64_t B, int32_t W, void* stream);

/* slot_to_packed [n_slots] int32 from the reference's chunk packing mask `packed_indices` (sigir20_tkl.py:159, one
 * byte per chunk slot, n_slots = B*C): the packed index of the slot, -1 where the chunk was dropped. */
MMB200_API int mmb200_tkl_slot_map(const void* packed_mask, int32_t* slot_to_packed, int64_t n_slots, void* stream);

/* Backward of the TKL interaction stage (mmb200_tkl_window_scores + mmb200_tkl_top_hills) for
 * d(loss)/d(score) = grad_score [B]: what autograd derives from sigir20_tkl.py:180-286.  Only the <= 15
 * gathered windows per document carry gradient.
 * top_idx [B,3], orig_score [B,W]: outputs of mmb200_tkl_top_hills.
 * grad_q [B,Lq,D] and grad_chunks [n_chunks,40,D] are overwritten.
 * grad_params [K + 15 + (saturation == 0 ? 13 + D : K)]: d dense_w | d chunk_scoring | d sat_params |
 *   d sat_emb_reduce1.weight (embedding saturation only); summed over the batch in a fixed order.
 * workspace: B * (that length) floats. */
MMB200_API int mmb200_tkl_bwd(const float* q, const void* q_mask, const float* chunks, const void* chunk_mask,
                              const int32_t* slot_to_packed, const float* mu, const float* sigma,
                              const float* dense_w, const float* sat_red_w, const float* sat_params,
                              const float* chunk_scoring, const int64_t* top_idx, const float* orig_score,
                              const float* grad_score, float* grad_q, float* grad_chunks, float* grad_params,
                              float* workspace, int64_t B, int64_t n_chunks, int32_t Lq, int32_t D, int32_t C,
                              int32_t K, int32_t saturation, int32_t mask_dtype, void* stream);

/* ------------------------------------------------------------------------------------------
 * Exact maximum-inner-product search with fused per-query top-k (BERT_DOT dense retrieval scoring)
 *
 * Replaces: FaissIdIndexer / FaissBaseIndexer.search   matchmaker/retrieval/faiss_indices.py:27,34,49-74
 *           (faiss.IndexIDMap(IndexFlatIP), GPU-sharded, useFloat16), called from
 *           matchmaker/dense_retrieval.py:328 (index) and :391 (search).
 *
 * queries  [nq, dim], passages [n_pass, dim]: fp16 or bf16 (`dtype`), dim % 64 == 0, row-major,
 *          resident on the current device (one shard per GPU); fp32 accumulate on the tensor cores.
 *          dtype MMB200_F32_SPLIT16 (faiss without useFloat16, faiss_indices.py:65,72: fp32 storage): every fp32
 *          value x (pre-scaled by a power of two so that |x| < 2^15) is held as hi = fp16(x), lo = fp16(x - hi);
 *          passages [n_pass, 2*dim] = [hi | lo], queries [nq, 3*dim] = [hi | lo | hi]; the kernel runs 3*dim/64
 *          k-blocks pairing q_hi.p_hi + q_lo.p_hi + q_hi.p_lo (22 mantissa bits per operand, fp32 accumulate) and
 *          returns scores in the scaled domain (the caller multiplies by 2^-(sq+sp), exact).
 * ids      [n_pass] int64 user ids (add_with_ids) or NULL: id = id_base + row.
 * out_scores [nq, k] f32 descending; out_ids [nq, k] int64; ties ordered by id ascending (faiss leaves
 *          tie order unspecified); when n_pass < k the tail is (-3.4028235e38, -1) as in faiss.
 * workspace: device scratch of at least mmb200_flat_ip_workspace_bytes(nq, n_pass, k) bytes.
 * 1 <= k <= 1024 (k <= 256: 1024-entry candidate lists per query row; larger k: 2048-entry lists).
 * ------------------------------------------------------------------------------------------ */
MMB200_API int64_t mmb200_flat_ip_workspace_bytes(int64_t nq, int64_t n_pass, int32_t k);
/* The work decomposition mmb200_flat_ip_topk uses on a device with `sm_count` SMs (pure host arithmetic, no device
 * needed): out[0] query blocks of 128, out[1] passage tiles of 256, out[2] passage ranges, out[3] tiles per range,
 * out[4] grid (CTAs, a multiple of the cluster size), out[5] cluster size, out[6..7] workspace bytes (low, high 32
 * bits).  Returns 0, or MMB200_ERR_INVALID for sizes mmb200_flat_ip_topk would reject. */
MMB200_API int mmb200_flat_ip_plan(int64_t nq, int64_t n_pass, int32_t k, int32_t sm_count, int32_t out[8]);
MMB200_API int mmb200_flat_ip_topk(const void* queries, const void* passages, const int64_t* ids,
                                   float* out_scores, int64_t* out_ids, void* workspace,
                                   int64_t workspace_bytes, int64_t nq, int64_t n_pass, int32_t dim, int32_t k,
                                   int32_t dtype, int64_t id_base, void* stream);

/* Merge candidate lists: cand_scores / cand_ids [nq, n_candidates] -> the k best per query under (score desc,
 * id asc).  A candidate is void when its SCORE is NaN, -inf or -FLT_MAX (faiss's "no result"); ids may be any int64,
 * negative user ids included (faiss IndexIDMap allows them).  Any n_candidates: more than 8192 per query are merged
 * in passes.  Used after the NCCL all-gather of per-rank top-k lists (the reference merges faiss IndexShards results on
 * the host). */
MMB200_API int mmb200_topk_merge(const float* cand_scores, const int64_t* cand_ids, float* out_scores,
                                 int64_t* out_ids, int64_t nq, int32_t n_candidates, int32_t k, void* stream);

/* ------------------------------------------------------------------------------------------
 * Storage block loader: byte ranges of files -> one contiguous DEVICE buffer.
 *
 * Replaces: the host path of the encoded collection between matchmaker/dense_retrieval.py:291-302
 *           (np.memmap of token_reps_<n>.npy cut to storage_filled_to_index) and :328
 *           (indexer.index(id_mapping, storage) -> faiss add_with_ids from host arrays).
 * Segment s = nbytes[s] bytes of file paths[s] starting at file_offsets[s]; segments land back to back at
 * dst_device.  pread() into two pinned staging buffers of staging_bytes (0 = 32 MiB) each, cudaMemcpyAsync on
 * `stream`, read of the next piece overlapped with the transfer of the previous one.  Returns after the last
 * piece has left the staging buffers (the device copies are complete on `stream` by then).
 * ------------------------------------------------------------------------------------------ */
MMB200_API int mmb200_storage_load(const char* const* paths, const int64_t* file_offsets, const int64_t* nbytes,
                                   int32_t n_segments, void* dst_device, int64_t staging_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MATCHMAKER_B200_H_ */
