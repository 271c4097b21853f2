/*
 * lr_b200.h — C ABI of liblr_b200.so, the B200 (sm_100a) retrieval hot path.
 *
 * The reference (caskcsg/lightretriever) has no FFI of its own: the seams are
 * Python duck-typed protocols.  Every entry point below names the reference
 * interface (file:line under /root/reference) whose arithmetic it replaces.
 * A maintainer binds these with ctypes (see INTEGRATION.md); torch is only the
 * allocator — every argument is a plain device pointer, a size, or a stream.
 *
 * Conventions
 *   - all pointers are DEVICE pointers unless the name ends in _host;
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream);
 *   - every function returns LR_OK (0) or a negative LR_E* code; the message is
 *     available from lr_last_error() (thread-local);
 *   - nothing is allocated by the library: the caller owns outputs and the
 *     workspace (size it with the *_workspace_bytes functions);
 *   - there is no CPU fallback: without a CUDA device every compute entry point
 *     returns LR_ECUDA.
 */
#ifndef LR_B200_H
#define LR_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LR_OK        0
#define LR_EINVAL   -1   /* bad shape / dtype / alignment  -> Python ValueError   */
#define LR_ECUDA    -2   /* CUDA runtime / driver failure  -> Python RuntimeError */
#define LR_EWORKSPACE -3 /* workspace too small            -> Python ValueError   */

/* dtype tags */
#define LR_F32  0
#define LR_BF16 1

/* score kinds carried in the high word of a 64-bit candidate key */
#define LR_SCORE_F32 0   /* order-preserving map of an IEEE float (dense path) */
#define LR_SCORE_U32 1   /* non-negative integer impact score (sparse path)     */

const char* lr_last_error(void);
int         lr_version(void);
/* Number of SMs of the current device (148 on B200); <0 on error. */
int         lr_device_sm_count(void);
/* The LR_* experiment knobs (DESIGN.md appendix) are read from the environment once per thread and the search plans are
 * cached per shape; call this after changing a knob inside a running process (tests, A/B tools).  No reference
 * counterpart: the reference re-reads nothing either (its Faiss options are fixed at index build, faiss_index.py:60-70). */
int         lr_reload_env(void);

/* ---------------------------------------------------------------------------
 * K1  EmbeddingBag query encoder (mean, padding_idx) + MRL truncate + L2 norm
 *   replaces  emb_bag.forward(input, offsets)   finetune/modeling_hybrid.py:474
 *             emb_reps[..., :dense_shrink_dim]  finetune/modeling_hybrid.py:487-488
 *             F.normalize(emb_reps, p=2, dim=-1) finetune/modeling_hybrid.py:489-490
 *   ids      [n_ids]  int64, flattened token ids (nonctx_emb_utils.py:197-219)
 *   offsets  [n_bags] int64, bag starts; last bag runs to n_ids
 *            (torch include_last_offset=False)
 *   table    [V, d] row-major, table_dtype LR_BF16 | LR_F32, rows 16-byte aligned
 *   padding_idx  id excluded from sum and from the mean's denominator; -1 = none
 *   out_dim  m <= d, m % 8 == 0 : only the first m columns are read and written
 *   normalize != 0 : x / max(||x||_2, 1e-12)
 *   out      [n_bags, out_dim] out_dtype LR_BF16 | LR_F32
 * Empty bag (or all-padding bag) -> zero vector (torch semantics).
 * An id outside [0, V) is an error in torch; here it sets the row to NaN and the
 * call returns LR_EINVAL after the kernel (checked through a device flag).
 * ------------------------------------------------------------------------- */
int lr_embbag_encode(const int64_t* ids, const int64_t* offsets, int64_t n_ids, int64_t n_bags,
                     const void* table, int table_dtype, int64_t V, int64_t d, int64_t padding_idx,
                     int64_t out_dim, int normalize, void* out, int out_dtype,
                     int32_t* err_flag /* device int32, may be NULL */, void* stream);

/* ---------------------------------------------------------------------------
 * K1b  document dense head: last-token pooling + truncate + normalise
 *   replaces pooling(last_hidden, attention_mask, 'lasttoken')  finetune/dense_pooling.py:48-55
 *            + shrink / normalize                               finetune/modeling_hybrid.py:266-278
 *   hidden [B, S, d] (dtype LR_BF16 | LR_F32); mask [B, S] int64 (HF attention mask)
 *   If every row's last column is valid (left padding) row S-1 is taken for all
 *   rows, else row sum(mask)-1 (negative index wraps like torch: -1 -> S-1).
 *   scratch: device int32[B + 1].
 * ------------------------------------------------------------------------- */
int lr_lasttoken_head(const void* hidden, int hidden_dtype, const int64_t* mask,
                      int64_t B, int64_t S, int64_t d, int64_t out_dim, int normalize,
                      void* out, int out_dtype, int32_t* scratch, void* stream);

/* ---------------------------------------------------------------------------
 * K2  exact flat inner-product top-k   (TMA -> tcgen05.mma -> TMEM -> top-k epilogue)
 *   replaces FaissIndex.search(q, k) -> (scores f32 [Q,k] desc, ids i64 [Q,k])
 *            retriever/faiss_index.py:27-40 (faiss.IndexFlatIP.search), and the
 *            per-chunk heap merge retriever/hybrid_search.py:182-205.
 *   q       [Q, ldq]  bf16, row-major, ldq*2 % 16 == 0, base 16-byte aligned
 *   corpus  [N, ldc]  bf16, row-major, ldc*2 % 16 == 0, base 16-byte aligned
 *   d_used  inner-product length (MRL prefix m <= ldq, ldc); % 8 == 0
 *   q_scale [Q] / c_scale [N] f32 or NULL: score = dot * q_scale[q] * c_scale[n]
 *           (MRL on full-width stored vectors: reciprocal prefix norms)
 *   id_offset  added to the local row index (row-sharded corpus); ids must stay < 2^32
 *   k       1 <= k <= 2048
 *   out_scores [Q,k] f32 descending; out_ids [Q,k] i64; when N < k the tail is
 *   (-inf, -1) (Faiss convention for missing results).
 *   out_keys   optional [Q,k] u64 sorted candidate keys (for the cross-GPU merge), may be NULL
 *   Ties: equal scores are ordered by ascending id (Faiss leaves this undefined).
 *   workspace: >= lr_flatip_workspace_bytes_for(Q, N, k, d_used) bytes, 256-byte aligned.
 *              lr_flatip_workspace_bytes(Q, N, k) is the bound over every d_used (short rows, d_used <= 768,
 *              keep two candidate lists per corpus split and need about twice the space of full-width rows).
 * ------------------------------------------------------------------------- */
size_t lr_flatip_workspace_bytes(int64_t Q, int64_t N, int k);
size_t lr_flatip_workspace_bytes_for(int64_t Q, int64_t N, int k, int64_t d_used);
int lr_flatip_topk(const void* q, int64_t ldq, const void* corpus, int64_t ldc,
                   int64_t Q, int64_t N, int64_t d_used,
                   const float* q_scale, const float* c_scale, int64_t id_offset, int k,
                   float* out_scores, int64_t* out_ids, uint64_t* out_keys,
                   void* workspace, size_t ws_bytes, void* stream);

/* Row-sharded search, one shard per GPU (Faiss GpuMultipleClonerOptions.shard = True, retriever/faiss_index.py:60-70):
 * the warm start is shared between the shards.  lr_flatip_topk_begin scores this shard's 1/n_shards share of the
 * warm-start prefix and writes its top-k there as sorted keys out_prefix_keys [Q, k] (local ids; zeros when the plan of
 * this shape has no warm-start pass).  The caller exchanges them (NCCL all-gather), merges them per query with
 * lr_topk_merge and hands the merged [Q, k] keys to lr_flatip_topk_finish as seed_keys: the k-th best score of the whole
 * prefix is a lower bound of the global k-th score, so every shard runs its remaining passes with the thresholds of the
 * unsharded search at 1/n_shards of its warm-start cost.  The per-shard result then holds only documents that can
 * still reach the GLOBAL top-k: it may have fewer than k entries (tail (-inf, -1), key 0).  seed_keys NULL = no exchange.
 * Both calls take the same arguments, workspace (>= lr_flatip_workspace_bytes_sharded) and stream; the workspace
 * carries the state from one to the other and must not be used in between. */
size_t lr_flatip_workspace_bytes_sharded(int64_t Q, int64_t N, int k, int64_t d_used, int n_shards);
int lr_flatip_topk_begin(const void* q, int64_t ldq, const void* corpus, int64_t ldc,
                         int64_t Q, int64_t N, int64_t d_used, const float* q_scale, const float* c_scale,
                         int k, int n_shards, uint64_t* out_prefix_keys /*[Q,k]*/,
                         void* workspace, size_t ws_bytes, void* stream);
int lr_flatip_topk_finish(const void* q, int64_t ldq, const void* corpus, int64_t ldc,
                          int64_t Q, int64_t N, int64_t d_used, const float* q_scale, const float* c_scale,
                          int64_t id_offset, int k, int n_shards, const uint64_t* seed_keys /*[Q,k] or NULL*/,
                          float* out_scores, int64_t* out_ids, uint64_t* out_keys,
                          void* workspace, size_t ws_bytes, void* stream);

/* ---------------------------------------------------------------------------
 * Document filters and deletions inside the exact top-k (K2 above, K4 below).  No reference counterpart: the reference
 * can neither delete from a Faiss IndexFlatIP / Lucene index without rebuilding it nor restrict one search to a subset
 * of documents (Faiss offers SearchParameters(sel=IDSelectorBitmap), Lucene filter queries; the reference uses neither).
 *   Bitmaps are u32 words indexed by GLOBAL document id (local row + id_offset, the id a search returns): document i is
 *   allowed when bit (i & 31) of word (i >> 5) is set.  On a little-endian machine these are the same bytes Faiss's
 *   IDSelectorBitmap reads (bit i & 7 of byte i >> 3).  ld_words >= ceil((id_offset + N) / 32) words per bitmap, so the
 *   shards of a row-sharded index all read one replicated bitmap; nothing past ld_words is read.
 *   live      [ld_words] or NULL: deleted documents have their bit cleared (index state).
 *   allow     [n_filters][ld_words] or NULL: per-request filters; n_filters >= 1 when allow is set.
 *   q_filter  [Q] int32 or NULL (needs allow): the row of `allow` query q uses; -1 = unrestricted; any other value
 *             outside [0, n_filters) allows NOTHING (fail closed).  NULL with allow set = row 0 for every query.
 * A query's candidates are live AND its allow row.  The filter is applied before a document can enter a candidate list,
 * so every threshold (list cuts, warm-start prefix, refresh passes, the exchanged seed of a sharded search) comes from
 * allowed documents only and the result is the exact top-k of the allowed set.  Fewer than k allowed documents: the
 * result ends in a (-inf, -1) tail.  The filtered calls take the same workspace as the unfiltered ones
 * (lr_flatip_workspace_bytes*, lr_sparse_score_workspace_bytes); every pointer argument is a device pointer.
 * ------------------------------------------------------------------------- */
/* lr_flatip_topk with filters. */
int lr_flatip_topk_filtered(const void* q, int64_t ldq, const void* corpus, int64_t ldc,
                            int64_t Q, int64_t N, int64_t d_used,
                            const float* q_scale, const float* c_scale, int64_t id_offset, int k,
                            float* out_scores, int64_t* out_ids, uint64_t* out_keys,
                            const uint32_t* live, const uint32_t* allow, int64_t ld_words, int n_filters,
                            const int32_t* q_filter, void* workspace, size_t ws_bytes, void* stream);
/* lr_flatip_topk_begin / _finish with filters; begin also takes the shard's id_offset (it indexes the bitmaps).  The
 * prefix keys it writes hold allowed documents only, so the exchanged seed is a bound of the filtered global k-th score. */
int lr_flatip_topk_begin_filtered(const void* q, int64_t ldq, const void* corpus, int64_t ldc,
                                  int64_t Q, int64_t N, int64_t d_used, const float* q_scale, const float* c_scale,
                                  int64_t id_offset, int k, int n_shards, uint64_t* out_prefix_keys /*[Q,k]*/,
                                  const uint32_t* live, const uint32_t* allow, int64_t ld_words, int n_filters,
                                  const int32_t* q_filter, void* workspace, size_t ws_bytes, void* stream);
int lr_flatip_topk_finish_filtered(const void* q, int64_t ldq, const void* corpus, int64_t ldc,
                                   int64_t Q, int64_t N, int64_t d_used, const float* q_scale, const float* c_scale,
                                   int64_t id_offset, int k, int n_shards, const uint64_t* seed_keys /*[Q,k] or NULL*/,
                                   float* out_scores, int64_t* out_ids, uint64_t* out_keys,
                                   const uint32_t* live, const uint32_t* allow, int64_t ld_words, int n_filters,
                                   const int32_t* q_filter, void* workspace, size_t ws_bytes, void* stream);
/* Sets (set = 1) or clears (set = 0) the bits of ids [n] (int64, device) in words [ld_words] with atomicOr / atomicAnd;
 * ids outside [0, 32 * ld_words) are ignored.  One launch, no host synchronisation, no allocation: it may be captured in a
 * CUDA graph or enqueued between replays of one that reads `words`. */
int lr_doc_bitmap_update(uint32_t* words, int64_t ld_words, const int64_t* ids, int64_t n, int set, void* stream);

/* Debug / parity helper: the same TMA+tcgen05 main loop with a plain store
 * epilogue, scores [Q, N] f32 (small shapes only). Definition of the score:
 * torch.matmul(q, p.T)  finetune/modeling_encoder.py:414-427. */
int lr_flatip_scores(const void* q, int64_t ldq, const void* corpus, int64_t ldc,
                     int64_t Q, int64_t N, int64_t d_used, float* out_scores /*[Q,N]*/, void* stream);

/* Measurement hook (bench.py): when both are non-NULL cudaEvent_t handles, every following lr_flatip_topk /
 * lr_sparse_head_max call on this thread records ev_begin / ev_end on its stream immediately around the main
 * (tcgen05) kernel launch, so the caller can read that kernel's device time without a profiler.  NULL, NULL disables. */
int lr_set_profile_events(void* ev_begin, void* ev_end);

/* Plan of a (Q, N, k) search without running it (needs no CUDA device; 148 SMs are assumed when none is present):
 * out[0]=CTAs per cluster out[1]=cta_group::2 pair (0|1) out[2]=query tiles out[3]=corpus tiles out[4]=list capacity
 * out[5]=prefix tiles (0 = single phase) out[6]=prefix splits out[7]=prefix units out[8]=main first tile
 * out[9]=main splits out[10]=main units out[11]=main grid (CTAs) out[12]=band (query tiles) out[13]=workspace bytes
 * out[14]=main rounds out[15]=concurrent clusters */
int lr_flatip_plan(int64_t Q, int64_t N, int k, int64_t* out16);
/* The sequence of scoring passes of a (Q, N, k, d_used) search: warm-start prefix, threshold-refresh passes (short rows
 * only), main pass.  Writes up to max_passes rows of 4 values {first tile, end tile, splits, team schedule (0|1)} and
 * returns the number of passes (negative on error).  out_flags[0] = two epilogue warp sets (0|1),
 * out_flags[1] = candidate lists per split. */
int lr_flatip_plan_passes(int64_t Q, int64_t N, int k, int64_t d_used, int64_t* out_rows, int max_passes,
                          int64_t* out_flags2);
/* Same for one shard of a row-sharded search (lr_flatip_topk_begin / _finish): the warm-start prefix is 1/n_shards long. */
int lr_flatip_plan_passes_sharded(int64_t Q, int64_t N, int k, int64_t d_used, int n_shards, int64_t* out_rows,
                                  int max_passes, int64_t* out_flags2);

/* Plan of the last lr_flatip_topk call on this thread (for bench / DESIGN):
 * out[0]=m_tiles out[1]=n_tiles out[2]=splits out[3]=band out[4]=cap out[5]=grid out[6]=units out[7]=warm-start prefix tiles (0 = single phase) */
int lr_flatip_last_plan(int64_t* out8);
/* The scoring passes of the last lr_flatip_topk / _begin / _finish call on this thread, rows as in lr_flatip_plan_passes
 * (the last row is the main pass, the one lr_set_profile_events brackets); returns the number of passes. */
int lr_flatip_last_plan_passes(int64_t* out_rows, int max_passes);
/* Number of kernels this library has launched in this process (bench.py's gpu_launches is a difference of two reads). */
unsigned long long lr_kernel_launches(void);

/* ---------------------------------------------------------------------------
 * Merge of candidate lists (per-split partials, per-shard top-k after the
 * NCCL all-gather, per-chunk results):  exact top-k of the union.
 *   replaces HybridSearch._add_to_heap  retriever/hybrid_search.py:182-205
 *            (and Faiss IndexShards' host-side merge, retriever/faiss_index.py:65-68)
 *   keys    L lists per query; list l of query q starts at keys[(l*q_stride + q)*cap]
 *   counts  [L*q_stride] int32 valid entries per list, or NULL = every list holds `cap`
 *   key     = (score_key << 32) | (0xFFFFFFFF - id32); keys equal to 0 are ignored
 *   outputs any of out_scores/out_ids/out_keys may be NULL; sorted (score desc, id asc)
 * ------------------------------------------------------------------------- */
int lr_topk_merge(const uint64_t* keys, const int32_t* counts, int L, int64_t Q, int64_t q_stride,
                  int cap, int k, int score_kind, int64_t id_offset,
                  float* out_scores, int64_t* out_ids, uint64_t* out_keys, void* stream);

/* (scores f32, ids i64) [n] -> candidate keys u64 [n]; id < 0 -> key 0 (ignored). */
int lr_encode_keys(const float* scores, const int64_t* ids, int64_t n, uint64_t* keys, void* stream);

/* ---------------------------------------------------------------------------
 * K3  document sparse head
 *   replaces aggregate()/max_linear_mapping  finetune/sparse_pooling.py:244-278,
 *            utils/max_linear_map.py:10-90  (max over valid tokens of h_t.W + b)
 *            relu_/log1p_                   finetune/modeling_hybrid.py:183-187
 *   hidden [B*S, d] bf16 (tokens of doc b are rows b*S .. b*S+S-1), W [V, d] bf16
 *   (= lm_head.weight), bias [V] f32 or NULL, mask [B*S] uint8 (1 = valid token;
 *   get_sparse_attention_mask, finetune/sparse_pooling.py:23-41)
 *   out [B, V] f32:  max_t(h_t.W_v + b_v) over valid t, then optional relu, log1p.
 *   A doc without valid token gives finfo(bf16).min before relu (max_linear_map.py:27).
 * ------------------------------------------------------------------------- */
int lr_sparse_head_max(const void* hidden, const void* W, const float* bias, const uint8_t* mask,
                       int64_t B, int64_t S, int64_t d, int64_t V, int relu, int log1p,
                       float* out /*[B,V]*/, void* stream);

/* Packed form of the same operator: `hidden` holds ONLY the valid tokens, document after document ([T, d] bf16), and
 * cu_seqlens [B+1] int32 (device) gives document b the rows [cu_seqlens[b], cu_seqlens[b+1]); T = cu_seqlens[B] is passed
 * by the host (it knows the attention mask before the backbone runs).  Padding is never multiplied: the work is
 * 2*T*d*V instead of 2*B*S*d*V.  The tokens are cut into balanced runs of whole 256-token tiles; a document that
 * crosses a cut is finished by a small second kernel from the pieces the GEMM epilogue left in the workspace
 * (device, 256-byte aligned, >= lr_sparse_head_packed_workspace_bytes(T, V)).  A document without a token gives
 * finfo(bf16).min before relu, as above. */
size_t lr_sparse_head_packed_workspace_bytes(int64_t T, int64_t V);
/* planner introspection (host only): out[4] = 256-token tiles, splits, edge-buffer offset, workspace bytes */
int lr_sparse_head_packed_plan(int64_t T, int64_t V, int64_t* out);
int lr_sparse_head_max_packed(const void* hidden, const void* W, const float* bias, const int32_t* cu_seqlens,
                              int64_t B, int64_t T, int64_t d, int64_t V, int relu, int log1p,
                              float* out /*[B,V]*/, void* workspace, size_t ws_bytes, void* stream);
/* hidden [B*S, d] bf16 + mask [B*S] uint8 -> packed [<= cap, d] (valid rows in order) and cu_seqlens [B+1] int32. */
int lr_pack_tokens(const void* hidden, const uint8_t* mask, int64_t B, int64_t S, int64_t d, void* packed,
                   int64_t cap, int32_t* cu_seqlens, void* stream);

/* top_p_sampling (finetune/sparse_pooling.py:64-87, called at modeling_hybrid.py:189-195 with sparse_top_p_qry/_psg):
 * in ascending order of value, entries are set to 0 while the cumulative softmax probability up to and including them
 * is <= 1 - top_p; the min_keep largest always stay; top_p outside (0, 1) is a no-op.  reps [B, V] f32, in place.
 * min_keep = 0 keeps every entry (the reference's remove[..., -0:] = False selects all columns); min_keep < 0 -> LR_EINVAL.
 * The reference's float32 cumsum has no defined rounding: entries whose cumulative probability is within ~1e-6 of the
 * bound may differ (tests state the band). */
int lr_top_p_filter(float* reps, int64_t B, int64_t V, float top_p, int min_keep, void* stream);

/* top_k_sampling (finetune/sparse_pooling.py:89-106: keep every entry >= the k_eff-th
 * largest, k_eff = min(max(top_k, min_keep), V), top_k <= 0 disables) followed by the
 * quantiser of convert_sparse_reps_to_json_pt (finetune/sparse_converter_mixin.py:103-160):
 * clamp(min=0), round-half-even(x*quant) -> int, zeros dropped.
 *   reps [B, V] f32 ; indptr [B+1] int32 ; tok/impact [cap] ; returns LR_EWORKSPACE
 *   if nnz > cap (indptr is still fully written so the caller can re-size).
 *   scratch: device, >= lr_sparsify_scratch_bytes(B, V). */
size_t lr_sparsify_scratch_bytes(int64_t B, int64_t V);
int lr_sparsify_quantize(const float* reps, int64_t B, int64_t V, int top_k, int min_keep, float quant,
                         int32_t* indptr, int32_t* tok, uint16_t* impact, int64_t cap,
                         void* scratch, void* stream);

/* ---------------------------------------------------------------------------
 * K4  sparse impact scoring + top-k over an inverted index (CSC by token)
 *   replaces Anserini impact search  retriever/anserini_search.py:143-216
 *   score(q,d) = sum_t count_q(t) * impact_d(t)   scripts/asymmetric_sparse_infer.ipynb:207-228
 *   q_indptr [Q+1] i32, q_tok [nnz_q] i32, q_cnt [nnz_q] i32   (Counter(ids), exact_search_base.py:371-435)
 *   post_indptr [V+1] i64, post_doc [nnz] i32 ascending inside a token, post_imp [nnz] u16
 *   Only documents with score > 0 are returned (Lucene returns matching docs only);
 *   missing tail = (-inf, -1). Scores are exact integers (returned as f32; exact < 2^24).
 * ------------------------------------------------------------------------- */
/* Documents are scored in blocks of lr_sparse_block_docs() (4096) consecutive ids whose int32 accumulators
 * live in shared memory, one block per warp.  blockptr[t*(nblk+1) + b] = number of postings of token t with
 * doc < b*block_docs (nblk = ceil(N / block_docs)); built once per index (index time, not on the query path).
 * Query terms with a count <= 0 contribute nothing. */
int    lr_sparse_block_docs(void);
int    lr_sparse_build_blockptr(const int64_t* post_indptr, const int32_t* post_doc, int64_t V, int64_t N,
                                uint32_t* blockptr /* [V*(nblk+1)] */, void* stream);
size_t lr_sparse_score_workspace_bytes(int64_t Q, int64_t N, int k);
/* planner introspection (host only): out[16] = block_docs, index blocks, list capacity, flat kernel launched, row
 * kernel launched, splits (flat), splits (rows), lists per query, workers per CTA of the four launches (flat 16-bit,
 * flat int32, rows 16-bit, rows 32-bit), dynamic shared memory of the flat / row 16-bit launches, workspace bytes,
 * documents per step of the row kernel */
int lr_sparse_score_plan(int64_t Q, int64_t N, int k, int64_t* out);
/* k <= 1024 */
int lr_sparse_score_topk(const int32_t* q_indptr, const int32_t* q_tok, const int32_t* q_cnt, int64_t Q,
                         const int64_t* post_indptr, const int32_t* post_doc, const uint16_t* post_imp,
                         const uint32_t* blockptr, int64_t V, int64_t N, int64_t id_offset, int k,
                         float* out_scores, int64_t* out_ids, uint64_t* out_keys,
                         void* workspace, size_t ws_bytes, void* stream);

/* lr_sparse_score_topk with the document filters described above K2's filtered entry points. */
int lr_sparse_score_topk_filtered(const int32_t* q_indptr, const int32_t* q_tok, const int32_t* q_cnt, int64_t Q,
                                  const int64_t* post_indptr, const int32_t* post_doc, const uint16_t* post_imp,
                                  const uint32_t* blockptr, int64_t V, int64_t N, int64_t id_offset, int k,
                                  float* out_scores, int64_t* out_ids, uint64_t* out_keys,
                                  const uint32_t* live, const uint32_t* allow, int64_t ld_words, int n_filters,
                                  const int32_t* q_filter, void* workspace, size_t ws_bytes, void* stream);

/* ---------------------------------------------------------------------------
 * Query token counts: the sparse query of K4, built on the device
 *   replaces Counter(ids) / {t: 1 for t in set(ids)}  inference/exact_search_base.py:371-435
 *            (the query token ids of scripts/asymmetric_sparse_infer.ipynb:50; sparse_search.parse_queries on the host)
 *   ids      [n_ids]  int64, flattened token ids; an id outside [0, V) contributes nothing (a caller may pad with -1)
 *   offsets  [n_bags] int64, bag starts; last bag runs to n_ids (as lr_embbag_encode reads them)
 *   bow      0 = count of each token ("sum"), 1 = count 1 per distinct token ("bow")
 *   q_indptr [n_bags+1] i32, q_tok [n_ids] i32, q_cnt [n_ids] i32: compact CSR, the q_* input of lr_sparse_score_topk.
 *            A bag gets one term per distinct in-range token, tokens ascending, counts >= 1; rows past
 *            q_indptr[n_bags] are zero.
 *   max_bag  host bound on the in-range ids of any bag, 0 <= max_bag <= LR_QUERY_MAX_BAG (it sizes shared memory).
 *            A bag with more, a bag outside [0, n_ids] or one that ends before it starts (descending offsets) sets
 *            *err_flag = 1 (device int32, may be NULL) and gets no terms.
 *   scratch  device, >= lr_query_token_counts_scratch_bytes(n_ids, n_bags) bytes (0 when n_bags < 1; needs no device).
 * Two launches, no host synchronisation and no allocation: may be captured in a CUDA graph.
 * ------------------------------------------------------------------------- */
#define LR_QUERY_MAX_BAG 8192
size_t lr_query_token_counts_scratch_bytes(int64_t n_ids, int64_t n_bags);
int lr_query_token_counts(const int64_t* ids, const int64_t* offsets, int64_t n_ids, int64_t n_bags, int64_t V,
                          int64_t max_bag, int bow, int32_t* q_indptr /*[n_bags+1]*/, int32_t* q_tok /*[n_ids]*/,
                          int32_t* q_cnt /*[n_ids]*/, int32_t* err_flag, void* scratch, size_t scratch_bytes,
                          void* stream);

/* ---------------------------------------------------------------------------
 * Hybrid score fusion of two top-k lists per query (dense + sparse), on device
 *   replaces fuse_scores_linear / fuse_scores_rrf  retriever/score_fuse_utils.py:48-90, 3-46
 *            (HybridSearch._fuse_results           retriever/hybrid_search.py:207-232)
 *   scores0/ids0 [Q,k0], scores1/ids1 [Q,k1]: sorted lists as returned by lr_flatip_topk / lr_sparse_score_topk
 *   (id -1 = padding).  method 0 = linear: sum_s w_s * (x - min_s) / (max_s - min_s + eps) over the union of ids;
 *   method 1 = rrf: sum_s 1 / (k_rrf + rank_s).  float64 arithmetic in the reference's operation order.
 *   out_ids [Q, k0+k1] int64 (-1 padded), out_scores [Q, k0+k1] float64 (-inf padded), sorted by (fused desc, id asc);
 *   out_counts [Q] int32 (size of the union), may be NULL.   k0 + k1 <= 4096.
 * ------------------------------------------------------------------------- */
int lr_fuse_topk(const float* scores0, const int64_t* ids0, int k0, const float* scores1, const int64_t* ids1, int k1,
                 int64_t Q, int method, double w0, double w1, double eps, double k_rrf,
                 int64_t* out_ids, double* out_scores, int32_t* out_counts, void* stream);
/* Same with float64 input scores: the dict-shaped callers (fuse_scores_linear / fuse_scores_rrf over
 * dict[qid -> dict[pid -> float]], score_fuse_utils.py:3-90) hold Python floats, i.e. float64. */
int lr_fuse_topk_f64(const double* scores0, const int64_t* ids0, int k0, const double* scores1, const int64_t* ids1, int k1,
                     int64_t Q, int method, double w0, double w1, double eps, double k_rrf,
                     int64_t* out_ids, double* out_scores, int32_t* out_counts, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* LR_B200_H */
