/* mse_b200.h — C ABI of the B200-native retrieval hot path.
 *
 * The reference (StephenTaf/Modern-Search-Engines-Project) is pure Python and has no FFI; each
 * entry point below replaces the inside of one reference function and is what a ctypes binding
 * in the reference would call (see INTEGRATION.md for the stubs):
 *
 *   mse_bm25_load           <- what BM25.__init__ opens: the four bm25_* tables
 *                              (indexer/bm25_indexer.py:57-80, DDL :82-128)
 *   mse_bm25_search_batch   <- BM25.search steps 5-8: candidate SQL, grouping, float64 scoring
 *                              loop, sort, slice (indexer/bm25_indexer.py:435-485)
 *   mse_dense_load          <- chunks_optimized + embeddings tables (indexer/embedder.py:31-52)
 *   mse_rerank_batch        <- rerank(): candidate fetch, cosine, min-max, fusion, positional
 *                              weighting, per-doc max, sort (reranker/reranker_api.py:27-63,273-372)
 *   mse_hybrid_search_batch <- the per-query body of the batch path: bm_25.search(top_k=1000) followed by
 *                              POST /rerank (search_api.py:252-274, single query :88-102), both stages on the device
 *   mse_diversify_batch     <- hybrid_diversification (reranker_api.py:196-236) of fused lists the caller holds
 *   mse_hybrid_search_diversified <- the same batch path with the reranker's final diversification step (on by
 *                              default, reranker/config.yaml:29), all three stages on the device
 *   mse_dense_scan_batch    <- the removed Retriever.quick_search (call sites search_api.py:60,87)
 *   mse_topk_merge          <- (new) merge of per-shard top-k lists after an NCCL all-gather
 *   mse_comm_* / *_sharded  <- (new) the same calls over a corpus sharded by document range across the GPUs of
 *                              one box, with the NCCL exchange inside the call (SURVEY.md 8b / 8e)
 *
 * Conventions: every function returns 0 on success or an MSE_ERR_* code and sets a thread-local
 * message readable through mse_last_error(); no exception crosses the boundary.  An mse_index
 * owns all device memory it allocates; callers own every buffer they pass in.  The index is
 * immutable after load, and search calls may be issued concurrently from several host threads and
 * streams: every call takes its own workspace from a small pool owned by the index.  There is no CPU
 * fallback: without a CUDA device every compute entry point fails with MSE_ERR_CUDA.
 *
 * Document numbering: all kernels work on the dense document index 0..n_docs-1 (ascending
 * urlsDB id, so "tie -> lower doc id" == "tie -> lower index"); outputs are doc_base + local
 * index, where doc_base is the first dense index of this shard.
 *
 * Buffer location (`where`) and synchronisation:
 *   MSE_HOST        host buffers (pageable or pinned).  The call copies, runs and returns when the
 *                   outputs are filled (it synchronises `stream`).  Results are always exact.
 *   MSE_DEVICE      device buffers.  The call ENQUEUES its work on `stream` and returns; it never blocks
 *                   the host, allocates nothing once its workspace has grown to the batch size, and can be
 *                   captured in a CUDA graph.  The plain (non-_async) BM25 and dense-scan calls additionally
 *                   read one status word back before returning, because they re-run queries whose candidate
 *                   list overflowed; the *_async / hybrid / sharded calls report that in `status` instead.
 *   MSE_HOST_ASYNC  PINNED host buffers.  H2D copies, kernels and D2H copies are enqueued on `stream`
 *                   and the call returns; outputs (and `status`) are valid once the caller has synchronised
 *                   the stream.  Two streams used alternately overlap the copies of one batch with the
 *                   kernels of the next.
 * `status` (may be NULL) is an int32[MSE_STATUS_WORDS] record in the same memory space as the outputs:
 *   [0] MSE_ST_* error flags (malformed query CSR: the offending queries return no result)
 *   [1] number of queries whose candidate list overflowed its workspace; their out_count is -1 (hybrid: 0 results)
 *       and they must be repeated through an MSE_HOST call (which handles it internally).  Does not
 *       happen unless a large share of a corpus ties at the k-th score.
 *   [2] sharded calls: 1 when a shard list cut to m entries could hide a result of the exact top-k —
 *       repeat the call with `shard_list_len` = top_k (always exact)
 *   [3] diversifying calls: number of queries whose diversified list was cut to max_out (the reference's list can be
 *       longer than its top_k, see mse_diversify_batch)
 */
#ifndef MSE_B200_H
#define MSE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MSE_ABI_VERSION 2

#define MSE_OK 0
#define MSE_ERR_INVALID 1      /* bad argument / malformed index (unsorted postings, ...) */
#define MSE_ERR_CUDA 2         /* CUDA runtime error, or no device */
#define MSE_ERR_NOMEM 3
#define MSE_ERR_STATE 4        /* e.g. search before load */
#define MSE_ERR_UNSUPPORTED 5  /* e.g. top_k above MSE_MAX_TOPK */
#define MSE_ERR_COMM 6         /* NCCL missing or a collective failed */

#define MSE_MAX_TOPK 4096      /* the reference uses 1000 (config.py:13) and 100 (reranker/config.yaml:30) */
#define MSE_EMB_DIM 768        /* config.py:2 */
#define MSE_MAX_QUERY_TERMS 32 /* distinct valid terms per query */
#define MSE_MAX_RERANK_CAND 1024   /* candidates per query of the rerank stage (reference: 1000) */

#define MSE_HOST 0
#define MSE_DEVICE 1
#define MSE_DEVICE_BORROW 2    /* mse_dense_load only: `emb` is bf16 device memory that the index uses IN PLACE
                                  (no copy; the caller keeps it alive and unchanged until the next load/destroy) */
#define MSE_HOST_ASYNC 3

#define MSE_STATUS_WORDS 4
#define MSE_ST_BAD_CSR 1       /* q_off not monotone / not ending at n_slots, or a query with more than MSE_MAX_QUERY_TERMS terms */
#define MSE_ST_BAD_LIST 2      /* diversify: an input list that is not non-increasing, in_count outside [0, in_stride] or a doc
                                  outside the domain table */

typedef struct mse_index mse_index;

const char* mse_last_error(void);
int mse_abi_version(void);
int mse_device_count(int* n_devices);

int mse_index_create(int device, mse_index** out);
int mse_index_destroy(mse_index* idx);

/* Tuning knobs (all optional; 0 restores the automatic choice unless stated):
 *   "bm25_range_docs"        docs per shared-memory accumulator range of the fp32 score kernel (rounded up to a multiple of
 *                            128, default 1536); asking for a size selects that kernel
 *   "bm25_accum"             0 (default) = the two-phase score kernel (16-bit upper-bound accumulators over 3072-doc ranges, exact
 *                            fp32 rescoring of the documents that reach the bound: the same scores bit for bit) whenever
 *                            min_score >= 0, the shard holds at least top_k such ranges and the batch is large enough for a bound
 *                            to form while it runs (>= 64 tasks per resident warp: ~100 queries at 10 M docs), the fp32 kernel
 *                            otherwise — also for the 64 calls that follow an exact call in which > 45 % of the tasks needed exact mode;
 *                            16 = the two-phase kernel wherever min_score >= 0; 32 = always the fp32 kernel
 *   "bm25_queries_per_item"  queries a warp scores per scheduled work item (<= 8, default 8; 6 in the two-phase kernel)
 *   "bm25_cand_cap"          per-query capacity of the candidate list between scoring and selection
 *   "bm25_use_tau"           1 (default) = running k-th-score bound filters candidates, 0 = emit all
 *   "bm25_tau_init"          1 (default) = seed the bound from the per-term impact table built at load time, 0 = off
 *   "bm25_readout"           1 (default) = candidates are found while the postings are applied, 0 = by a scan of the
 *                            accumulators (identical results)
 *   "bm25_neg_lookup"        1 (default) = with min_score >= 0 the postings of negative-idf terms are not streamed; their
 *                            contribution is read from a dense per-term impact row for the documents that reach the
 *                            bound on their other terms.  0 = stream every posting list (identical results up to the
 *                            order of the float32 additions)
 *   "bm25_class_term"        term id (idf < 0) whose per-document impact class is kept in every posting, so that a document that
 *                            cannot reach the running bound once this term is charged is never looked up: set it to the term the
 *                            caller appends to every query ("tübingen", search_api.py:160-165).  Default: the negative-idf term
 *                            with the most postings.  Takes effect on the loaded index (rewrites 4 bits per posting); results
 *                            never depend on it
 *   "dense_scan_ctas_per_sm" persistent CTAs per SM of the scan kernel
 *   "dense_gemm_min_batch"   smallest batch routed to the tcgen05 GEMM kernel (default 8; faster from 3 on, but queries are rounded to bf16 there)
 *   "dense_gemm_pair_mode"   batches of 129..256 queries run as clusters of two CTAs: 1 (default) = every E tile TMA-multicast into
 *                            both CTAs, cta_group::1 MMAs; 2 = cta_group::2 MMAs issued by the leader CTA, E stages split
 *   "timers"                 1 (default) = bracket the kernels with CUDA events (mse_kernel_time), 0 = off
 *   "reset_timers"           any value: zero the accumulated kernel timers
 * Environment: MSE_DEBUG_SYNC=1 synchronises after every BM25 kernel so that a device fault names its kernel. */
int mse_index_set_option(mse_index* idx, const char* name, int64_t value);

/* ---- BM25 (Stage 1) -------------------------------------------------------------------- */

/* Loads the inverted index of one shard.
 *   term_off[n_terms+1]  CSR offsets into the posting arrays (bm25_term_freq ORDER BY term, doc_id)
 *   post_doc[P]          LOCAL dense doc index (0..n_docs-1), strictly ascending inside a term
 *   post_tf[P]           bm25_term_freq.freq
 *   doc_len[n_docs]      bm25_doc_stats.doc_length
 *   idf[n_terms]         bm25_term_stats.idf_score verbatim (float32 log10, may be <= 0; :140)
 *   avgdl                bm25_corpus_stats 'avg_doc_length' (float32; GLOBAL, never per shard)
 *   k1, b                BM25.__init__ parameters (:57)
 * `where` tells whether the five arrays are host (MSE_HOST) or device (MSE_DEVICE) memory.
 * The arrays are only read during the call.  The library keeps the postings as one {doc, fp32 impact} array with
 * impact = tf / (tf + k1*(1 - b + b*doc_len/avgdl)) (the tf factor of bm25_indexer.py:470-476, formed in float64 and
 * rounded once), so k1, b and avgdl are fixed per loaded index: load again after the corpus statistics change.
 * Terms with idf < 0 additionally get a dense per-document impact row (see "bm25_neg_lookup"). */
int mse_bm25_load(mse_index* idx, int64_t n_terms, int64_t n_docs, int64_t doc_base,
                  const int64_t* term_off, const int32_t* post_doc, const int32_t* post_tf,
                  const int32_t* doc_len, const float* idf, float avgdl, float k1, float b, int where);

/* Index aggregation on the device (replaces the aggregation half of BM25.build_index,
 * indexer/bm25_indexer.py:181-211 and :283-343; tokenisation and the term dictionary stay with the caller).
 *   doc_tok_off[n_docs+1], tok_term[T]   documents as a CSR of term ids, T = doc_tok_off[n_docs] < 2^31
 *   term_off[n_terms+1]                  out: CSR offsets of the posting arrays (term-major, doc ascending)
 *   post_doc[>=T], post_tf[>=T]          out: postings (dense doc index, term frequency); *n_postings entries are written
 *   total_freq[n_terms]                  out: bm25_term_stats.total_freq; doc_freq is term_off[t+1] - term_off[t]
 * The float32 corpus statistics and the float32 log10 IDF (:130-147, :346-369) are V- / N-sized: the caller forms
 * them from these outputs exactly as the reference does.  Needs no mse_index; `device` selects the GPU. */
int mse_bm25_aggregate(int device, int64_t n_docs, int64_t n_terms, const int64_t* doc_tok_off, const int32_t* tok_term,
                       int64_t* term_off, int32_t* post_doc, int32_t* post_tf, int64_t* total_freq, int64_t* n_postings,
                       int where, void* stream);

/* Scores a batch of tokenised queries and returns, per query, the top_k documents with
 * score >= min_score among documents holding at least one posting of a valid query term
 * (:436-456, :480), ordered by score descending, ties by ascending doc (:484).
 *   q_off[n_queries+1], q_term[], q_tf[]   CSR of DISTINCT term indices per query with their
 *       query frequency (:405-409); indices < 0 or >= n_terms or with df == 0 are ignored (:430)
 *   out_doc[n_queries*top_k], out_score[n_queries*top_k], out_count[n_queries]
 * Scores are computed in float32 (reference: float64 on float32 idf/avgdl).
 * `where` = MSE_HOST or MSE_DEVICE; always exact and complete on return (see "Buffer location"). */
int mse_bm25_search_batch(mse_index* idx, int32_t n_queries, const int32_t* q_off, const int32_t* q_term,
                          const int32_t* q_tf, int32_t top_k, float min_score,
                          int32_t* out_doc, float* out_score, int32_t* out_count, int where, void* stream);

/* The same, enqueue-only: `where` = MSE_DEVICE or MSE_HOST_ASYNC, n_slots = q_off[n_queries] (the caller built the
 * CSR and knows it), `status` as described above. */
int mse_bm25_search_batch_async(mse_index* idx, int32_t n_queries, int32_t n_slots, const int32_t* q_off,
                                const int32_t* q_term, const int32_t* q_tf, int32_t top_k, float min_score,
                                int32_t* out_doc, float* out_score, int32_t* out_count, int32_t* status,
                                int where, void* stream);

/* Counters of the last BM25 call on this index (for the roofline report); synchronises the device.
 * stats[0] = postings traversed (sum of df over the streamed query terms), stats[1] = candidates
 * emitted to the selection stage, stats[2] = queries re-run through the unbounded-capacity path,
 * stats[3] = doc ranges, stats[4] = score-kernel CTAs launched, stats[5] = postings of looked-up
 * (negative-idf) terms that were NOT streamed, stats[6] = (sub-range, query) tasks the two-phase score
 * kernel rescored in its exact fp32 mode (0 when the fp32 kernel ran). */
int mse_bm25_last_stats(mse_index* idx, int64_t stats[8]);

/* Timing hooks: every call brackets its kernels with CUDA events on the launching stream (not while the stream is
 * being captured).  Returns the accumulated device time (ms) and the number of launches since the last
 * "reset_timers"; waits for the launches still in flight.  kernel: 0 = bm25 score, 1 = top-k select,
 * 2 = dense scan, 3 = rerank, 4 = bm25 prepare, 5 = shard exchange (collectives + merges), 6 = diversify. */
int mse_kernel_time(mse_index* idx, int kernel, double* total_ms, int64_t* launches);

/* ---- dense (Stage 2) ------------------------------------------------------------------- */

/* Loads one shard of chunk embeddings, doc-contiguous in ascending chunk id.
 *   emb            n_chunks x 768, float32 (emb_is_bf16 = 0; converted to bf16 on load) or bf16
 *   doc_chunk_off  [n_docs+1] chunk range of every local doc (chunks_optimized ORDER BY doc_id, chunk_id)
 *   chunk_base     global row number of the first local chunk (chunk ids are sequential, indexer.py:108-111) */
int mse_dense_load(mse_index* idx, int64_t n_chunks, int64_t n_docs, int64_t doc_base, int64_t chunk_base,
                   const void* emb, int emb_is_bf16, const int64_t* doc_chunk_off, int where);

/* Stores the url-up-to-'?' group id of every document of the WHOLE corpus (GLOBAL dense index, n entries;
 * reranker_api.py:44-47) in the index; the rerank / hybrid calls use it when their url_group argument is NULL.
 * n == 0 clears it. */
int mse_dense_set_url_groups(mse_index* idx, const int32_t* url_group, int64_t n, int where);

/* Stores the domain id (urlparse(url).netloc.lower(), reranker_api.py:170-176, mapped to int32 by the caller; a missing
 * URL counts as "") of every document of the WHOLE corpus (GLOBAL dense index, n entries) in the index; the diversifying
 * calls use it.  n == 0 clears it.  With a dense shard loaded, n must cover it: n >= doc_base + n_docs. */
int mse_dense_set_domains(mse_index* idx, const int32_t* domain, int64_t n, int where);

/* Exhaustive scan: inner product of each query with every stored chunk, max over the chunks of
 * a document, top_k documents per query (ties -> lower doc).  q is float32 [n_queries*768].
 * MSE_HOST or MSE_DEVICE; exact and complete on return. */
int mse_dense_scan_batch(mse_index* idx, int32_t n_queries, const float* q, int32_t top_k,
                         int32_t* out_doc, float* out_score, int32_t* out_count, int where, void* stream);
/* Enqueue-only form (MSE_DEVICE or MSE_HOST_ASYNC). */
int mse_dense_scan_batch_async(mse_index* idx, int32_t n_queries, const float* q, int32_t top_k,
                               int32_t* out_doc, float* out_score, int32_t* out_count, int32_t* status,
                               int where, void* stream);

/* Gathered rerank of BM25 candidates (reranker_api.py:336-372).
 *   cand_off[n_queries+1], cand_doc[], cand_bm25[]   candidates per query in BM25 order (GLOBAL dense index)
 *   url_group[n_docs] or NULL   id of the url-up-to-'?' group of each local doc (:44-47); among
 *       candidates of one group only the lowest doc survives; NULL = the groups stored by mse_dense_set_url_groups, if any
 *   q            float32 [n_queries*768], NOT normalised (:355); a device pointer must be 16-byte aligned
 *   out_*        [n_queries*max_out]: docs sorted by fused score descending; out_orig = min-max'd BM25
 *                score, out_chunk = global row (== chunk id) of the representative chunk,
 *                out_rows[n_queries] = fetched chunk rows (`total_documents` of the reference response).
 * MSE_HOST, MSE_DEVICE (enqueue-only: nothing here depends on a read-back) or MSE_HOST_ASYNC. */
int mse_rerank_batch(mse_index* idx, int32_t n_queries, const int32_t* cand_off, const int32_t* cand_doc,
                     const float* cand_bm25, const int32_t* url_group, const float* q,
                     float smoothing, int32_t max_chunks, int32_t max_out,
                     int32_t* out_doc, float* out_score, float* out_orig, int64_t* out_chunk,
                     int32_t* out_count, int32_t* out_rows, int where, void* stream);

/* One hybrid query batch: BM25 top_k candidates (:252 `bm_25.search(query, top_k=1000)`) handed on the device to the
 * rerank stage (:259-274) -> max_out results per query.  Inputs as mse_bm25_search_batch_async (q_off / q_term / q_tf,
 * n_slots) plus q_vec float32 [n_queries*768] (16-byte aligned on the device); outputs as mse_rerank_batch.
 * top_k <= MSE_MAX_RERANK_CAND.
 * `where` = MSE_HOST (exact, complete on return), MSE_DEVICE or MSE_HOST_ASYNC (enqueue-only, see `status`). */
int mse_hybrid_search_batch(mse_index* idx, int32_t n_queries, int32_t n_slots, const int32_t* q_off,
                            const int32_t* q_term, const int32_t* q_tf, const float* q_vec,
                            int32_t top_k, float min_score, float smoothing, int32_t max_chunks, int32_t max_out,
                            int32_t* out_doc, float* out_score, float* out_orig, int64_t* out_chunk,
                            int32_t* out_count, int32_t* out_rows, int32_t* status, int where, void* stream);

/* Domain diversification (reranker_api.py:196-236) of n_queries fused lists, each sorted by score descending (ties in
 * any order: the rule is applied to the list as given).
 *   in_count[n_queries], in_doc / in_score / in_orig / in_chunk [n_queries * in_stride]: lists shaped like the outputs
 *       of mse_rerank_batch (in_stride <= MSE_MAX_RERANK_CAND); in_doc is a GLOBAL dense doc index
 *   domain       int32 per GLOBAL dense doc index, covering the documents of this index (doc_base + n_docs entries),
 *                or NULL = the table stored by mse_dense_set_domains
 *   relevance_threshold   a domain is hot if one of its documents has score >= it (compared in double; 0.8 in the reference)
 *   top_k        the reference's top_k (100).  Kept documents keep their score; back-filled ones get
 *                float(max(0, s - delta)).  The list can be longer than top_k (a reference quirk: more than top_k hot
 *                domains); it is cut to max_out and status[3] counts the cut lists.  1 <= top_k <= max_out <= 1024.
 *   out_*        [n_queries * max_out] (-1 / 0 padded), out_count[n_queries]; out_orig and out_chunk carry the inputs'.
 * A bad list sets MSE_ST_BAD_LIST in status[0] and returns no result.
 * MSE_HOST, MSE_DEVICE (enqueue-only, graph-capturable) or MSE_HOST_ASYNC. */
int mse_diversify_batch(mse_index* idx, int32_t n_queries, int32_t in_stride, const int32_t* in_count, const int32_t* in_doc,
                        const float* in_score, const float* in_orig, const int64_t* in_chunk, const int32_t* domain,
                        double relevance_threshold, int32_t top_k, int32_t max_out,
                        int32_t* out_doc, float* out_score, float* out_orig, int64_t* out_chunk, int32_t* out_count,
                        int32_t* status, int where, void* stream);

/* mse_hybrid_search_batch followed on the device by mse_diversify_batch(top_k = div_top_k) with the stored domain table:
 * the rerank stage keeps the whole fused list of every query (up to MSE_MAX_RERANK_CAND documents), which the
 * diversification needs (it back-fills from far down the list), and only the max_out diversified results are written.
 * Arguments, outputs and `status` as mse_hybrid_search_batch, plus status[0] / [3] as mse_diversify_batch.
 * MSE_ERR_STATE without a domain table covering the index. */
int mse_hybrid_search_diversified(mse_index* idx, int32_t n_queries, int32_t n_slots, const int32_t* q_off,
                                  const int32_t* q_term, const int32_t* q_tf, const float* q_vec,
                                  int32_t top_k, float min_score, float smoothing, int32_t max_chunks, int32_t max_out,
                                  int32_t* out_doc, float* out_score, float* out_orig, int64_t* out_chunk,
                                  int32_t* out_count, int32_t* out_rows, int32_t* status, int where, void* stream,
                                  double relevance_threshold, int32_t div_top_k);

/* Sharded form of mse_rerank_batch, host-driven variant (chunk table sharded by doc range over several GPUs);
 * device buffers only (q 16-byte aligned).  Step 1, every rank: same replicated candidates; dedupes, then fills the cosines of the
 * candidates whose documents THIS shard owns into cos[B][1024][10] / rows[B][1024] / chunk0[B][1024] (zeroed here
 * first) and the replicated survivor description surv_*.  url_group is indexed by the GLOBAL dense doc index.
 * The caller then sums cos / rows / chunk0 over the ranks and calls step 2 on any rank.  (mse_hybrid_search_sharded
 * below does the whole exchange inside one call with far less traffic.) */
int mse_rerank_shard_cos(mse_index* idx, int32_t n_queries, const int32_t* cand_off, const int32_t* cand_doc,
                         const float* cand_bm25, const int32_t* url_group, int64_t n_docs_global, const float* q,
                         int32_t max_chunks, float* cos, int32_t* rows, int64_t* chunk0,
                         int32_t* surv_doc, float* surv_bm25, int32_t* surv_count, void* stream);
/* Step 2: pool-wide min-max, fusion, positional weighting, per-doc max, sort (reranker_api.py:289-372) from the
 * gathered arrays; outputs as mse_rerank_batch. */
int mse_rerank_shard_fuse(mse_index* idx, int32_t n_queries, const float* cos, const int32_t* rows, const int64_t* chunk0,
                          const int32_t* surv_doc, const float* surv_bm25, const int32_t* surv_count,
                          float smoothing, int32_t max_out, int32_t* out_doc, float* out_score, float* out_orig,
                          int64_t* out_chunk, int32_t* out_count, int32_t* out_rows, void* stream);

/* ---- shard merge (multi-GPU) ------------------------------------------------------------ */

/* Merges n_lists sorted top-k lists per query (the all-gathered per-rank results, laid out
 * [n_lists][n_queries][list_k]) into one top_k list per query with the same ordering rule. */
int mse_topk_merge(mse_index* idx, int32_t n_queries, int32_t n_lists, int32_t list_k,
                   const int32_t* in_doc, const float* in_score, const int32_t* in_count, int32_t top_k,
                   int32_t* out_doc, float* out_score, int32_t* out_count, int where, void* stream);

/* ---- corpus sharded by document range over the GPUs of one box (one process per GPU) ---------------------
 * Every rank loads its contiguous doc range (mse_bm25_load / mse_dense_load with doc_base / chunk_base, GLOBAL
 * idf and avgdl) and attaches a communicator.  A sharded call takes the WHOLE replicated batch of n_queries =
 * world * queries_per_rank queries on every rank and returns, on rank r, the results of ITS block of the batch
 * (queries r*queries_per_rank .. (r+1)*queries_per_rank - 1).  All collectives are NCCL calls enqueued on `stream`
 * (NVLink / NVSwitch); the calls are enqueue-only (MSE_DEVICE buffers) and report through `status`.
 * NCCL is loaded at run time (libnccl.so.2 — the copy the process has already loaded, e.g. PyTorch's, is used). */
#define MSE_COMM_ID_BYTES 128
int mse_comm_unique_id(void* id_bytes /* out: MSE_COMM_ID_BYTES, create on rank 0 and hand to every rank */);
int mse_comm_init(mse_index* idx, const void* id_bytes, int32_t rank, int32_t world);   /* ncclCommInitRank, owned by the index */
int mse_comm_attach(mse_index* idx, void* nccl_comm /* ncclComm_t owned by the caller */, int32_t rank, int32_t world);
int mse_comm_destroy(mse_index* idx);

/* BM25 over the sharded corpus.  Every rank scores all n_queries against its shard and keeps shard_list_len
 * entries per query (0 = automatic: mean + 6 sigma + 16 of Binomial(top_k, 1/world); a shard owns ~top_k/world of a global top-k); block w of the
 * lists travels to rank w (one grouped send/receive per peer), which merges the `world` lists of its queries to the
 * exact top_k.  status[2] reports a cut that could have hidden a result.  Outputs: [queries_per_rank * top_k]. */
int mse_bm25_search_sharded(mse_index* idx, int32_t n_queries, int32_t n_slots, const int32_t* q_off,
                            const int32_t* q_term, const int32_t* q_tf, int32_t top_k, float min_score,
                            int32_t shard_list_len, int32_t* out_doc, float* out_score, int32_t* out_count,
                            int32_t* status, void* stream);

/* Hybrid query over the sharded corpus (postings AND chunks of a document live on its rank):
 *   1. sharded BM25 as above -> exact global top_k candidates on the query-owning rank, which also applies the
 *      URL-group dedupe (reranker_api.py:38-47; needs mse_dense_set_url_groups with the GLOBAL groups, if any)
 *   2. all-gather of the surviving candidates (8 B each)
 *   3. every rank: cosines of the candidates whose chunks it owns (<= max_chunks rows per doc), local min / max
 *   4. all-reduce(min, max) of 4 floats per query: the pool-wide normalisation bounds of :289-296
 *   5. every rank: fusion + positional weighting + per-doc max of ITS documents (:299-372), local top max_out
 *   6. the local lists travel to the query owner, which merges them: scores are formed exactly as on one GPU.
 * q_vec float32 [n_queries*768], 16-byte aligned.  Outputs as mse_rerank_batch for the queries_per_rank owned queries. */
int mse_hybrid_search_sharded(mse_index* idx, int32_t n_queries, int32_t n_slots, const int32_t* q_off,
                              const int32_t* q_term, const int32_t* q_tf, const float* q_vec,
                              int32_t top_k, float min_score, int32_t shard_list_len,
                              float smoothing, int32_t max_chunks, int32_t max_out,
                              int32_t* out_doc, float* out_score, float* out_orig, int64_t* out_chunk,
                              int32_t* out_count, int32_t* out_rows, int32_t* status, void* stream);
/* Diversified results: call it with max_out = MSE_MAX_RERANK_CAND (the whole fused list) and pass its outputs to
 * mse_diversify_batch on the same rank (domain table: the GLOBAL ids, mse_dense_set_domains). */

/* Exhaustive dense scan over the sharded chunk table: local top_k per query, NCCL all-gather of the lists,
 * merge on every rank (replicated result: out_* are [n_queries * top_k] on every rank). */
int mse_dense_scan_sharded(mse_index* idx, int32_t n_queries, const float* q, int32_t top_k,
                           int32_t* out_doc, float* out_score, int32_t* out_count, int32_t* status, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MSE_B200_H */
