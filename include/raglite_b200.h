/* raglite_b200 -- C-ABI of the B200-native RAGLite retrieval hot path.
 *
 * Every entry point takes plain device/host pointers, sizes and a CUDA stream handle
 * (`void* stream` == cudaStream_t); there are no torch / C++ types in any signature.
 * Return value: 0 on success, a negative RL_E* code on failure; rl_last_error() gives the
 * message of the last failure on the calling thread.  No entry point allocates device memory:
 * the caller passes a workspace sized by the matching *_workspace_bytes() query.  All calls are
 * asynchronous on `stream` and re-entrant (no global mutable state), so several host threads may
 * drive different streams concurrently (reference callers use thread pools: _rag.py:317,
 * _eval.py:178).
 *
 * The reference (superlinear-ai/raglite @ 2069f8d) is pure Python and has no FFI; each entry point
 * cites the Python code whose arithmetic it replaces.  INTEGRATION.md shows the ctypes binding a
 * RAGLite maintainer would add.
 */
#ifndef RAGLITE_B200_H_
#define RAGLITE_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RL_OK 0
#define RL_EINVAL (-1)    /* bad argument (null pointer, unsupported size/metric, misalignment) */
#define RL_ECUDA (-2)     /* a CUDA runtime call failed */
#define RL_ENOSPACE (-3)  /* workspace too small */
#define RL_EUNSUPPORTED (-4)

/* Distance metric: RAGLiteConfig.vector_search_distance_metric (_config.py:69), rendered per
 * dialect at _typing.py:110-134.  sim = 1 - dist (_search.py:72). */
#define RL_METRIC_COSINE 0 /* dist = 1 - <e,q>/sqrt(|e|^2 |q|^2)  (array_cosine_distance)        */
#define RL_METRIC_DOT 1    /* dist = -<e,q>                        (array_negative_inner_product) */
#define RL_METRIC_L2 2     /* dist = |e - q|_2                     (array_distance)               */

/* Scan kernel selection. */
#define RL_ALGO_AUTO 0
#define RL_ALGO_FP32 1    /* exact fp32 CUDA-core scan (any d) */
#define RL_ALGO_TCGEN05 2 /* fp16-input tcgen05/TMEM coarse scan + exact rescoring (d % 4 == 0) */

/* rl_maxsim_topk flags. */
#define RL_FLAG_REUSE_THRESHOLDS 1u /* skip the sample pass; use thresholds left in the workspace */
#define RL_FLAG_TIME_KERNELS 2u     /* record CUDA events around each stage (see rl_maxsim_kernel_times) */
#define RL_FLAG_COUNT_UNFILTERED 4u /* also count, per query, the rows that pass the emission threshold but are masked
                                       out by row_allowed (and alive per row_alive): rl_maxsim_unfiltered_bound */

/* Per-query status bits written by rl_maxsim_topk. */
#define RL_STATUS_CAND_OVERFLOW 1 /* candidate list overflowed: call again with REUSE_THRESHOLDS */
#define RL_STATUS_TIE_OVERFLOW 2  /* reserved (never set since v101: more than RL_MAX_SURVIVORS rows inside the error
                                     band of the cut are rescored by a streaming pass over the candidate list) */

#define RL_MAX_SURVIVORS 4096

int rl_version(void);
const char* rl_last_error(void);

/* Number of SMs etc. of the current device (diagnostics for bench.py). */
int rl_device_info(int* sm_count, int* cc_major, int* cc_minor, size_t* l2_bytes);

/* ---- Index build -------------------------------------------------------------------------
 * Per-row statistics of the embedding matrix E[n_rows, d] (row stride ld floats): inv_norm[j] =
 * 1/|e_j| (0 for a zero row), sq_norm[j] = |e_j|^2, and four global statistics used to scale rows for
 * the fp16 scan (stats[4], device floats, zeroed by the caller once -- the kernel folds maxima in, so
 * appended rows (insert_documents flushes, _insert.py:247-255) only need a call over the new rows): [0] max row norm, [1] max
 * |element|, [2] max 1/|e_j| over non-zero rows, [3] 1 if any row is all-zero.  Replaces nothing in the reference (DuckDB recomputes norms per query inside
 * array_cosine_distance); it is the device-side part of building the resident index from the
 * chunk_embedding table (_database.py:403-430). */
int rl_row_stats(const float* E, int64_t n_rows, int d, int64_t ld, float* inv_norm, float* sq_norm,
                 float* stats, void* stream);
/* Same for an embedding matrix stored as float16 (rl_scan_params.e_dtype == 1). */
int rl_row_stats_f16(const void* E, int64_t n_rows, int d, int64_t ld, float* inv_norm, float* sq_norm,
                     float* stats, void* stream);

/* row_chunk[j] = c for chunk_off[c] <= j < chunk_off[c+1]  (CSR -> per-row owner; the
 * chunk_embedding.chunk_id column, _database.py:421). */
int rl_chunk_row_map(const int64_t* chunk_off, int64_t n_chunks, int32_t* row_chunk, void* stream);

/* Per-row byte mask for rl_scan_params.row_allowed: out[j] = chunk_ok[row_chunk[j]] AND alive[j].
 * chunk_ok (uint8 [n_chunks], or NULL = every chunk) is the metadata filter resolved per chunk (the JSON
 * containment tests of _search.py:82-95), alive (uint8 [n_rows], or NULL) the tombstones of deleted
 * chunks (_delete.py:146-152).  row_chunk, alive and out must be 16-byte aligned. */
int rl_row_mask(const uint8_t* chunk_ok, const int32_t* row_chunk, const uint8_t* alive, int64_t n_rows,
                uint8_t* out, void* stream);

/* ---- Query adapter apply: _search.py:58-62 -------------------------------------------------
 * Q_out[b,:] = round_to(A @ Q_in[b,:]) with A[d,d] float64 row-major exactly as the reference
 * stores it (_query_adapter.py:211), accumulated in float64; round_mode 0 = keep float32,
 * 1 = round through float16 (the reference casts back to the query dtype, fp16 for string
 * queries, _embed.py:140). */
int rl_adapter_apply(const double* A, const float* Q_in, float* Q_out, int B, int d, int round_mode,
                     void* stream);

/* ---- MaxSim scan + top-k: _search.py:65-79, 143-153 -----------------------------------------
 * One shard of the corpus, a batch of B queries.
 *   E[n_rows,d] float32 row-major (ld = row stride in floats), inv_norm/sq_norm from
 *   rl_row_stats, row_chunk from rl_chunk_row_map, chunk_base = global index of this shard's
 *   first chunk, max_vecs_per_chunk = max CSR segment length, row_stats = stats from rl_row_stats.
 *   row_allowed: optional uint8[n_rows], or NULL: rows with a zero byte do not take part -- the metadata
 *     filter (_search.py:82-121) and the tombstones of deleted chunks (_delete.py:146-152), ANDed by the caller.
 *   Q[B,d] float32 (already adapter-applied).
 *   num_hits > 0: reference SQL semantics -- the num_hits vectors with smallest distance
 *     (_search.py:75-79); hits are those vectors, ascending distance.
 *   num_hits == 0: exact per-chunk MaxSim -- hits are the best k chunks.
 * Outputs (H = num_hits ? num_hits : k):
 *   hit_sim[B,H] float32 (sim = 1 - dist), hit_chunk[B,H] int64 global chunk index,
 *   hit_count[B] int32, status[B] int32 (RL_STATUS_* bits).
 * Feed the hit lists of all shards to rl_topk_merge for the GROUP BY / ORDER BY / LIMIT. */
typedef struct rl_scan_params {
  const float* E;
  const float* inv_norm;
  const float* sq_norm;
  const int32_t* row_chunk;
  const float* row_stats;
  const uint8_t* row_allowed;
  int64_t n_rows;
  int64_t ld;
  int64_t chunk_base;
  int32_t d;
  int32_t max_vecs_per_chunk;
  const float* Q;
  int32_t B;
  int32_t metric;
  int32_t k;
  int32_t num_hits;
  int32_t algo;
  uint32_t flags;
  int32_t sample_stride; /* 0 = auto */
  int32_t cand_cap;      /* 0 = auto */
  int32_t e_dtype;       /* storage of E: 0 = float32, 1 = float16 (E then points to IEEE binary16; needs
                            RL_ALGO_TCGEN05, d % 8 == 0 and rows that need no per-row scaling) */
  int32_t rows_unit_scale; /* 1: the caller guarantees (from the rl_row_stats statistics: max 1/|e| <= 2, max |e_ij| <= 1024,
                            no all-zero row -- true for normalised embeddings) that rows can enter the fp16 scan unscaled,
                            which lets the cosine scan use the two-tiles-per-query-slice kernel.  0: unknown (always valid) */
  const uint8_t* row_alive; /* optional uint8[n_rows] (NULL = all): rows that exist at all -- the tombstone mask without
                            the metadata filter (only read with RL_FLAG_COUNT_UNFILTERED) */
} rl_scan_params;

size_t rl_maxsim_workspace_bytes(const rl_scan_params* p);
int rl_maxsim_topk(const rl_scan_params* p, float* hit_sim, int64_t* hit_chunk, int32_t* hit_count,
                   int32_t* status, void* workspace, size_t workspace_bytes, void* stream);

/* Counters of the last rl_maxsim_topk call on this workspace (device->host copy, synchronises the
 * stream): kernel launches issued, and per-call totals of emitted candidates / survivors. */
typedef struct rl_scan_stats {
  int32_t launches;
  int32_t sample_stride;
  int32_t cand_cap;
  int32_t algo;
  int64_t n_sample_rows;
  int64_t cand_total;
  int64_t cand_max;
  int64_t survivors_total;
  int64_t survivors_max; /* largest per-query survivor count (> RL_MAX_SURVIVORS: that query took the streaming path) */
} rl_scan_stats;
int rl_maxsim_stats(const rl_scan_params* p, const void* workspace, rl_scan_stats* out, void* stream);

/* Fused bound for the rank-then-filter metadata branch (_search.py:122-143).  After an rl_maxsim_topk call made
 * with RL_FLAG_COUNT_UNFILTERED on a FILTERED scan (row_allowed set), bound[b] (device int64 [B]) is an UPPER bound
 * of the number of live rows of the shard -- filtered or not -- that are at least as near to query b as the worst
 * of its num_hits filtered hits: every emission threshold the scan ever used lies at or below that hit's key, so
 * the rows counted against the thresholds (allowed ones = the candidate count, masked ones = the extra counter)
 * plus the whole sample are a superset.  bound <= 1 000 000 proves that the filter-first answer is also the
 * rank-then-filter answer, without the second pass over the corpus rl_maxsim_count_at_least needs.  Returns
 * RL_EUNSUPPORTED when the last call did not count (fp32 scan, flag not set). */
int rl_maxsim_unfiltered_bound(const rl_scan_params* p, const void* workspace, int64_t* bound, void* stream);

/* Rank probe for the reference's rank-then-filter metadata branch (_search.py:122-143, which keeps the
 * 1 000 000 nearest vectors before it applies the filter): counts[b] = number of rows of the shard
 * (p->row_allowed honoured, normally the tombstone mask only) whose similarity to query b is at least
 * sim_floor[b] (device float32 [B], in the units vector_search returns: 1 - dist).  The scan compares
 * approximate keys, so `bound` picks the side of the bracket: +1 counts every row whose exact
 * similarity can reach the floor (upper bound), -1 only rows that certainly do (lower bound), 0 the raw
 * key comparison.  One pass over the corpus, nothing stored; p is the same struct rl_maxsim_topk takes
 * and the workspace the same size.  counts is device int32 [B]. */
int rl_maxsim_count_at_least(const rl_scan_params* p, const float* sim_floor, int bound, int32_t* counts,
                             void* workspace, size_t workspace_bytes, void* stream);

/* Device time in ms of the stages of the rl_maxsim_topk calls made with RL_FLAG_TIME_KERNELS on this
 * workspace since the previous read (average over up to 32 calls): ms[0] = prep, ms[1] = sample scan (dump), ms[2] = select, ms[3] = main scan (emit),
 * ms[4] = finalize.  CUDA events are recorded on the launching stream; the call synchronises on the
 * last one.  Diagnostics for bench.py's roofline figure. */
int rl_maxsim_kernel_times(const void* workspace, float* ms);

/* Releases the timing events tied to a workspace pointer (created on the first RL_FLAG_TIME_KERNELS call);
 * call before freeing the workspace.  No-op for a workspace that was never timed. */
int rl_maxsim_release(const void* workspace);

/* Debug/test hook: copy the sampled approximate keys of the last call (float32 [B, n_sample_rows],
 * sample position p <-> row (p / 128) * sample_stride * 128 + p % 128) into dst (device memory);
 * *n_sample_rows receives the row count.  dst may be NULL to query the size only. */
int rl_maxsim_copy_dump(const rl_scan_params* p, const void* workspace, float* dst, int64_t* n_sample_rows,
                        void* stream);

/* ---- Shard merge + GROUP BY chunk + top-k: _search.py:143-150 --------------------------------
 * hit_*[R,B,H] are the per-shard outputs of rl_maxsim_topk (all-gathered).  num_hits > 0: keep
 * the num_hits best vectors overall, group by chunk (max sim), order desc, limit k.  num_hits == 0:
 * merge the per-shard chunk lists, limit k.  Outputs out_sim[B,k], out_chunk[B,k] (-1 padded),
 * out_count[B]. */
int rl_topk_merge(const float* hit_sim, const int64_t* hit_chunk, const int32_t* hit_count, int R,
                  int B, int H, int num_hits, int k, float* out_sim, int64_t* out_chunk,
                  int32_t* out_count, void* stream);

/* Packed per-shard hit list, the unit the single all-gather of the sharded path moves (NCCL over NVLink):
 *   chunk int64 [B, H] | sim float32 [B, H] | count int32 [B] | (status int32 [B])   -- padded to 16 bytes.
 * rl_maxsim_topk can write straight into such a buffer (its four output pointers are the four sections),
 * so nothing is re-packed before the collective, and rl_topk_merge_packed reads the R gathered buffers in
 * place (rank_stride_bytes apart), so nothing is unpacked after it. */
size_t rl_hits_packed_bytes(int B, int H, int with_status);
int rl_topk_merge_packed(const void* packed, int64_t rank_stride_bytes, int R, int B, int H, int num_hits, int k,
                         float* out_sim, int64_t* out_chunk, int32_t* out_count, void* stream);

/* ---- Query-adapter fit: _query_adapter.py:21-38, 172-183 ---------------------------------------------------
 * rl_best_vectors: for every eval e and retrieved chunk chunks[e, slot] (shard-local chunk index, -1 = unused), the
 * vector of that chunk with the largest inner product with the eval's query Q[e, :] -- argmax(embedding_matrix @ q),
 * first maximum on ties -- written to best[e, slot, :] (float32; zeros for unused slots) and its row to best_row.
 * E: the corpus (e_dtype 0 = float32, 1 = float16), chunk_off the CSR offsets (device int64 [n_chunks + 1]). */
int rl_best_vectors(const void* E, int e_dtype, int64_t ld, int d, const int64_t* chunk_off, const int64_t* chunks,
                    int n_evals, int n_slots, const float* Q, float* best, int64_t* best_row, void* stream);
/* rl_adapter_targets: _optimize_query_target for every eval at once.  kind[e, slot] = 1 for a relevant chunk's vector
 * (P), 0 for an irrelevant one (N), anything else = unused.  T[e, :] (float64) = q + D^T mu* with
 * D = {p_i - (1 + alpha) n_j} and mu* = argmin_{mu >= 0} |q + D^T mu|^2 (active-set NNLS in float64 on the Gram
 * form, see csrc/adapter_fit.cu); ok[e] = 0 when the eval has no relevant or no irrelevant chunk (T = q then, the
 * reference skips such evals), iters[e] = outer iterations.  n_slots <= 64, |P| |N| <= 1024. */
int rl_adapter_targets(const float* best, const uint8_t* kind, int n_evals, int n_slots, int d, const float* Q, double alpha,
                       double* T, int32_t* ok, int32_t* iters, void* stream);

/* ---- Fusion and span collation on device chunk indices: _search.py:233-280, 323-360 ------------------------
 * rl_rrf_fuse: Reciprocal Rank Fusion of R rankings per query.  ids[B, R, L] int64 chunk indices (-1 padded at
 * the tail of a ranking), weights[R] float64 (device), k the RRF constant (60 in the reference).
 * score(c) = sum_r weights[r] / (k + position of c in ranking r), float64 summed ranking by ranking exactly as the
 * reference's dict does; output ordered by descending score, ties in first-appearance order (ranking 0 first) --
 * Python's stable sort.  out_ids[B, K] (-1 padded), out_score[B, K] float64, out_count[B].  R * L <= 4096. */
int rl_rrf_fuse(const int64_t* ids, const double* weights, int B, int R, int L, double k, int K, int64_t* out_ids,
                double* out_score, int32_t* out_count, void* stream);

/* rl_span_collate: the ranking half of retrieve_chunk_spans (_search.py:323-360) for B lists of M retrieved chunk
 * indices (ranked[B, M], -1 padded).  Index tables (device): chunk_doc[c] = ordinal of the chunk's document in
 * ascending document_id order, chunk_pos[c] = Chunk.index, chunk_alive[c] (or NULL), and the lookup
 * (doc << 32 | pos) -> chunk as two arrays sorted by key.  Every retrieved chunk is joined by its neighbours at
 * the given position offsets inside its document (neighbors[n_neighbors], e.g. {-1, +1}), duplicates are dropped,
 * members are ordered by (document, position) and cut into runs of consecutive positions; a run's score is the
 * sum of 1 / (rank + 1) over its retrieved members (float64), runs are ordered by descending score (stable).
 * Outputs, cap = M * (1 + n_neighbors) per query: out_member[B, cap] chunk indices in document order (-1 padded),
 * out_span_start / out_span_len[B, cap] (offsets into the member row, in final span order), out_span_score[B, cap],
 * out_n_span[B], out_n_member[B].  cap <= 4096. */
int rl_span_collate(const int64_t* ranked, int B, int M, const int32_t* chunk_doc, const int32_t* chunk_pos,
                    const uint8_t* chunk_alive, const uint64_t* sorted_key, const int64_t* sorted_chunk, int64_t n_chunks,
                    const int32_t* neighbors, int n_neighbors, int64_t* out_member, int32_t* out_span_start,
                    int32_t* out_span_len, double* out_span_score, int32_t* out_n_span, int32_t* out_n_member, void* stream);

/* ---- Late-chunking pool: _embed.py:129-140 (and the simple pool :154-164) ---------------------
 * X[T,d] token embeddings (float32, row stride ld); sentence s averages rows
 * [row_begin[s], row_end[s]) (host computes them with the largest-remainder rule, _embed.py:122-128;
 * preamble sentences are simply not listed), then optional L2 normalisation (normalize: 0 = off,
 * 1 = divide by the norm as _embed.py:139, 2 = eps-guarded as _embed.py:161-163) and a cast to
 * float16 (out[S,d], IEEE binary16 bit patterns).  Accumulation is float64 like NumPy's. */
int rl_segment_mean_pool(const float* X, int64_t ld, int d, const int32_t* row_begin,
                         const int32_t* row_end, int S, int normalize, uint16_t* out, void* stream);

/* ---- Cross-encoder scoring: _search.py:364-397 (reranker.rank -> FlashRank -> onnxruntime) --------
 * BERT cross-encoder forward (ms-marco-MiniLM-L-12-v2 architecture: LayerNorm(word+pos+type) ->
 * n_layers x [self-attention, dense+residual+LN, dense+GELU(erf), dense+residual+LN] -> pooler
 * (dense+tanh on [CLS]) -> classifier (1 logit)), fp16 storage / fp32 accumulate.  Linear layers are
 * pre-packed once with rl_xenc_pack_linear into the swizzled fp16 image the tensor-core kernel
 * bulk-copies.  All pointers are device pointers except `layers` (host array). */
typedef struct rl_xenc_layer {
  const void* qkv_img;   /* packed [3H, H]  (Q | K | V rows) */
  const float* qkv_bias; /* [3H] */
  const void* o_img;     /* packed [H, H] */
  const float* o_bias;
  const float* ln1_g;
  const float* ln1_b;
  const void* up_img;    /* packed [F, H] */
  const float* up_bias;
  const void* down_img;  /* packed [H, F] */
  const float* down_bias;
  const float* ln2_g;
  const float* ln2_b;
} rl_xenc_layer;

typedef struct rl_xenc_weights {
  int32_t n_layers, hidden, n_heads, ffn, vocab, max_pos, type_vocab;
  float ln_eps;
  const void* word_emb; /* fp16 [vocab, H] */
  const void* pos_emb;  /* fp16 [max_pos, H] */
  const void* type_emb; /* fp16 [type_vocab, H] */
  const float* emb_ln_g;
  const float* emb_ln_b;
  const rl_xenc_layer* layers; /* HOST array of n_layers entries */
  const float* pooler_w; /* fp32 [H, H] */
  const float* pooler_b;
  const float* cls_w;    /* fp32 [H]: the classifier row whose sigmoid is the score (row 1 of a two-label head) */
  const float* cls_b;    /* fp32 [1]: that row's bias */
} rl_xenc_weights;

size_t rl_xenc_linear_image_bytes(int N, int K);
/* W[N, K] float32 row-major (torch nn.Linear.weight) -> packed fp16 image. */
int rl_xenc_pack_linear(const float* W, int N, int K, void* image, void* stream);
/* Y[T, N] (fp16) = act(X[T, K] (fp16) W^T + bias); act 0 = identity, 1 = GELU(erf).  N % 32 == 0,
 * K % 8 == 0, bias 16-byte aligned. */
int rl_xenc_linear(const void* X, const void* image, const float* bias, void* Y, int T, int N, int K, int act,
                   void* stream);
size_t rl_xenc_workspace_bytes(const rl_xenc_weights* w, int T);
/* Packed variable-length batch: input_ids/type_ids/pos_ids [T], cu_seqlens [P+1]; max_len = longest
 * sequence.  out_logit[P], out_score[P] = sigmoid(logit) (FlashRank's score).  head_dim (hidden / n_heads)
 * must be 32 or 64 and hidden a multiple of 32 up to 768; anything else returns RL_EUNSUPPORTED. */
int rl_xenc_score(const rl_xenc_weights* w, const int32_t* input_ids, const int32_t* type_ids, const int32_t* pos_ids,
                  const int32_t* cu_seqlens, int P, int T, int max_len, float* out_logit, float* out_score,
                  void* workspace, size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* RAGLITE_B200_H_ */
