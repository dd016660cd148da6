/*
 * flmr_maxsim.h — C ABI of the B200-native FLMR / ColBERT late-interaction MaxSim + top-k path.
 *
 * This is the drop-in boundary for the ONE hot path this repository accelerates
 * (SURVEY.md §8b).  The reference has no FFI registry for this path: it binds four pybind11
 * torch extensions and calls Python scoring functions.  Each entry point below names the
 * reference interface it replaces (paths relative to the reference checkout, `CB/` =
 * third_party/ColBERT/colbert/):
 *
 *   flmr_corpus_create / _destroy / _info
 *       replaces the PLAID index residency built by IndexScorer.__init__ / IndexLoader
 *       (CB/search/index_storage.py:21-66, CB/search/index_loader.py:13-86) and the packed
 *       `D_packed [sum(doclens), dim]` + `D_lengths` operand pair of colbert_score_packed
 *       (CB/modeling/colbert.py:289-311).
 *   flmr_maxsim_scores
 *       replaces colbert_score / colbert_score_reduce / colbert_score_packed
 *       (CB/modeling/colbert.py:235-311) and the native segmented_maxsim_cpp
 *       (CB/modeling/segmented_maxsim.cpp:49-93): all-passage MaxSim scores of each query.
 *   flmr_maxsim_topk
 *       replaces IndexScorer.rank (CB/search/index_storage.py:86-98: retrieve -> score_pids ->
 *       sort) as called per query from Searcher.dense_search (CB/searcher.py:91-132); exhaustive
 *       instead of PLAID-pruned, batched over queries, top-k fused into the scoring kernel.
 *   flmr_topk_merge
 *       the only exchange step of the sharded path (SURVEY.md §8e): merges per-shard top-k lists
 *       (gathered by the host with one NCCL all-gather) into the global top-k.
 *   flmr_debug_maxsim_scores_simt
 *       test infrastructure: an independent plain-SIMT fp32 device kernel used by tests to
 *       cross-check the tensor-core kernel at sizes where the CPU oracle is too slow.
 *
 * Conventions (cf. SURVEY.md §8b "ownership / errors / threading"):
 *   - plain pointers and sizes only; no torch / C++ types cross this boundary;
 *   - every function returns an int status (0 = FLMR_OK); no exceptions, aborts or asserts
 *     cross the boundary; flmr_last_error() returns a thread-local message for the last failure;
 *   - the caller owns every input and output buffer; "d_" parameters are DEVICE pointers on the
 *     corpus' device, "h_" parameters are HOST pointers;
 *   - compute entry points are asynchronous on the supplied CUDA stream (passed as void* so the
 *     header needs no CUDA include; NULL = default stream);
 *   - a corpus handle is immutable after creation and may be shared by threads; concurrent
 *     searches on one handle must use distinct flmr_workspace handles.
 */
#ifndef FLMR_MAXSIM_H_
#define FLMR_MAXSIM_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FLMR_ABI_VERSION 2

/* status codes */
#define FLMR_OK 0
#define FLMR_ERR_INVALID_ARG 1
#define FLMR_ERR_CUDA 2
#define FLMR_ERR_UNSUPPORTED 3
#define FLMR_ERR_OOM 4
#define FLMR_ERR_KERNEL 5 /* device-side watchdog / self-check tripped */

/* flags for flmr_maxsim_scores / flmr_maxsim_topk */
#define FLMR_FLAG_RELU 1u /* reproduce the reference CPU packed path: sum_i max(0, max_j s_ij)   \
                             (CB/modeling/segmented_maxsim.cpp:58-59 zero-initialises the max) */

/* flags for flmr_corpus_create */
#define FLMR_CORPUS_COPY 0u  /* always copy the token matrix into library-owned HBM            */
#define FLMR_CORPUS_ADOPT 1u /* tokens is a device pointer; keep it (zero-copy) when every     \
                                doclen is a multiple of FLMR_TOKEN_GROUP, else copy+repack     */

#define FLMR_DIM 128        /* embedding dim of FLMR / ColBERT (CB/infra/config/settings.py:101) */
#define FLMR_TOKEN_GROUP 4  /* passages are stored padded to a multiple of this many tokens     */
#define FLMR_MAX_K 128      /* largest k of the fused top-k                                     */
#define FLMR_TILE_TOKENS 96 /* passage tokens per streamed tile of the scan kernel              */

typedef struct flmr_corpus flmr_corpus_t;       /* resident passage-token shard            */
typedef struct flmr_workspace flmr_workspace_t; /* per-caller scratch (candidates, Q pad)  */
typedef struct flmr_comm flmr_comm_t;           /* this rank's end of the shard exchange   */
typedef struct flmr_corpus_builder flmr_corpus_builder_t; /* streaming index load          */
typedef struct flmr_corpus_plaid_builder flmr_corpus_plaid_builder_t; /* chunked compressed load */

typedef struct flmr_corpus_info {
  int64_t n_passages;     /* passages in this shard                                           */
  int64_t n_tokens;       /* real tokens (sum of doclens)                                     */
  int64_t n_rows;         /* stored rows (tokens incl. group padding)                         */
  int64_t pid_base;       /* global id of passage 0 of this shard                             */
  int32_t dim;            /* = FLMR_DIM                                                       */
  int32_t device;         /* CUDA device ordinal                                              */
  int32_t n_ctas;         /* persistent CTAs the scan kernel launches (= SMs of the device)   */
  int32_t adopted;        /* 1 if the token matrix is the caller's buffer (zero-copy)         */
  int64_t n_tiles;        /* passage-token tiles streamed per corpus pass                     */
  int64_t hbm_bytes;      /* bytes of HBM held by the handle (excluding an adopted matrix)    */
                          /* (flmr_corpus_create_plaid: the compressed arrays + centroids)    */
} flmr_corpus_info_t;

/* Thread-local description of the last error returned on this thread ("" if none). */
const char* flmr_last_error(void);

/* ABI version of the loaded library (== FLMR_ABI_VERSION it was built with). */
int flmr_abi_version(void);

/*
 * Create a resident corpus shard from a packed token matrix.
 *   tokens      bf16 [sum(h_doclens), dim] row-major, passage after passage.  Host or device
 *               pointer (detected); with FLMR_CORPUS_ADOPT it must be a device pointer on `device`
 *               that outlives the handle.
 *   h_doclens   int32 [n_passages], every entry >= 1 (a zero-length passage has no defined score
 *               on the reference's two paths, SURVEY.md §8a, and is rejected).
 *   pid_base    added to local passage indices in every returned id (shard offset, §8e).
 */
int flmr_corpus_create(const void* tokens, const int32_t* h_doclens, int64_t n_passages, int dim,
                       int device, int64_t pid_base, unsigned flags, flmr_corpus_t** out);
/*
 * Create a resident corpus shard that stays COMPRESSED in HBM: the PLAID (ColBERTv2 residual) arrays of an index
 * written by the reference's Indexer, decoded inside the scan kernel instead of once into bf16 (flmr_plaid_decode).
 * Searches return exactly what a corpus created from the decoded tokens returns; the shard takes
 * 4 (code) + 16 * nbits (residual) + 4 (inverse norm) bytes per stored row instead of 256.
 *   d_codes          int32 [sum(h_doclens)]                    (<c>.codes.pt, passage after passage)
 *   d_residuals      uint8 [sum(h_doclens), dim * nbits / 8]   (<c>.residuals.pt)
 *   d_centroids      fp32  [n_centroids, dim]                  (centroids.pt, upcast; copied)
 *   d_bucket_weights fp32  [2^nbits]                            (buckets.pt[1]; copied)
 *   nbits            1, 2, 4 or 8;  h_doclens / pid_base as flmr_corpus_create
 * All d_ arrays are device pointers on `device` and may be freed when the call returns.  Every code is checked
 * against [0, n_centroids) here (FLMR_ERR_INVALID_ARG otherwise), never during a search.  Every entry point taking
 * a corpus accepts the handle; flmr_debug_maxsim_scores_simt returns FLMR_ERR_UNSUPPORTED for it.  Synchronous.
 */
int flmr_corpus_create_plaid(const int32_t* d_codes, const uint8_t* d_residuals, const float* d_centroids,
                             int64_t n_centroids, const float* d_bucket_weights, int nbits, const int32_t* h_doclens,
                             int64_t n_passages, int dim, int device, int64_t pid_base, flmr_corpus_t** out);
/*
 * The same, chunk by chunk — the load path of a large index: builder_create allocates the handle's arrays from the
 * doclens (and copies the centroids and bucket weights), every append packs the next chunk of WHOLE passages
 * (d_codes int32 [n_tokens], d_residuals uint8 [n_tokens, dim * nbits / 8], device pointers, passage after passage
 * in order; synchronous, the chunk may be freed on return), finish checks the codes of every chunk and hands over
 * the corpus (the builder is destroyed).  Peak device memory of a load = the resident arrays + one chunk.
 * A shard holds fewer than 2^31 - FLMR_TILE_TOKENS stored rows (as every corpus handle).
 */
int flmr_corpus_plaid_builder_create(const float* d_centroids, int64_t n_centroids, const float* d_bucket_weights,
                                     int nbits, const int32_t* h_doclens, int64_t n_passages, int dim, int device,
                                     int64_t pid_base, flmr_corpus_plaid_builder_t** out);
int flmr_corpus_plaid_builder_append(flmr_corpus_plaid_builder_t* b, const int32_t* d_codes,
                                     const uint8_t* d_residuals, int64_t n_tokens);
int flmr_corpus_plaid_builder_finish(flmr_corpus_plaid_builder_t* b, flmr_corpus_t** out);
int flmr_corpus_plaid_builder_destroy(flmr_corpus_plaid_builder_t* b);
int flmr_corpus_destroy(flmr_corpus_t* corpus);
int flmr_corpus_info(const flmr_corpus_t* corpus, flmr_corpus_info_t* out);

/*
 * Streaming construction of a corpus shard — the index LOAD path (replaces IndexLoader / ResidualEmbeddings.load_chunks,
 * CB/search/index_loader.py:24-62, CB/indexing/codecs/residual_embeddings.py:24-69): the padded token matrix is
 * allocated once from the doclens, then packed bf16 rows arrive IN ORDER, in chunks of any size, from host memory
 * or straight from a file, through two pinned staging buffers (the host fill of one overlaps the DMA of the
 * other; the file variant preads into pinned memory with 8 threads — no intermediate host copy).  If every
 * doclen is a multiple of FLMR_TOKEN_GROUP the rows are copied straight into place, else a scatter kernel puts
 * them into the padded layout.  finish() synchronises, builds the partition metadata and hands over the corpus
 * (the builder is destroyed); *host_fill_seconds (may be NULL) = host time spent reading / copying into the
 * staging buffers.  destroy() abandons a build.
 */
int flmr_corpus_builder_create(const int32_t* h_doclens, int64_t n_passages, int dim, int device,
                               int64_t pid_base, flmr_corpus_builder_t** out);
int flmr_corpus_builder_append(flmr_corpus_builder_t* b, const void* h_tokens_bf16, int64_t n_rows);
int flmr_corpus_builder_append_file(flmr_corpus_builder_t* b, const char* path, int64_t byte_offset, int64_t n_rows);
int flmr_corpus_builder_finish(flmr_corpus_builder_t* b, flmr_corpus_t** out, double* host_fill_seconds);
int flmr_corpus_builder_destroy(flmr_corpus_builder_t* b);

/* Scratch for searches on `corpus`.  max_queries (>= 1) sizes the per-CTA candidate buffer: a call with more
 * queries is processed in chunks of max_queries (each chunk: its scan passes + ONE merge launch).  max_nq
 * (>= 1) is the longest query expected: if it exceeds the 640 rows one pass holds, the partial-score rows of
 * row-sliced queries are allocated here instead of inside the first such search (longer queries still work,
 * the buffer then grows on demand). */
int flmr_workspace_create(const flmr_corpus_t* corpus, int max_queries, int max_nq,
                          flmr_workspace_t** out);
int flmr_workspace_destroy(flmr_workspace_t* ws);
/* Device-side watchdog code of the last scan on this workspace (0 = none; 101 producer, 102 MMA
 * issuer, 103 epilogue starved).  Readable even after the launch trapped. */
int flmr_workspace_status(const flmr_workspace_t* ws, int* out);

/*
 * MaxSim scores of every passage for each of n_queries queries.
 *   d_q          bf16 [n_queries, nq, dim] (rows L2-normalised by the encoder; all-zero rows allowed
 *                and contribute exactly 0, as in the reference)
 *   d_out_scores fp32 [n_queries, n_passages]:  out[b][p] = sum_i max_{j<len_p} <Q_b,i , D_p,j>
 */
int flmr_maxsim_scores(const flmr_corpus_t* corpus, flmr_workspace_t* ws, const void* d_q,
                       int n_queries, int nq, unsigned flags, float* d_out_scores, void* stream);

/*
 * Fused MaxSim + top-k: the k best passages of each query, sorted by descending score
 * (ties: ascending id).  No score matrix is written to HBM when nq fits one resident query tile.
 *   d_out_scores fp32  [n_queries, k]
 *   d_out_pids   int64 [n_queries, k]  (pid_base + local index; -1 / -inf fill if n_passages < k)
 */
int flmr_maxsim_topk(const flmr_corpus_t* corpus, flmr_workspace_t* ws, const void* d_q,
                     int n_queries, int nq, int k, unsigned flags, float* d_out_scores,
                     int64_t* d_out_pids, void* stream);

/*
 * Merge n_lists candidate lists per query into one top-k (the post-all-gather step of the
 * sharded path).  Entries with pid < 0 are ignored.
 *   d_in_scores fp32  [n_lists, n_queries, k_in]     d_in_pids int64 [n_lists, n_queries, k_in]
 *   d_out_*           [n_queries, k_out], k_out <= FLMR_MAX_K, n_lists * k_in <= 20480
 */
int flmr_topk_merge(const float* d_in_scores, const int64_t* d_in_pids, int n_lists, int n_queries,
                    int k_in, int k_out, float* d_out_scores, int64_t* d_out_pids, int device,
                    void* stream);

/*
 * The sharded search at the C boundary (SURVEY.md 8e; the reference has no counterpart: under DDP every rank
 * repeats the whole CPU search, src/executors/FLMR_executor.py:778-781).  Each rank holds a contiguous passage
 * shard (flmr_corpus_create with its pid_base); ONE exchange step — an NCCL all-gather of every rank's [B, k]
 * (score, pid) lists — then the merge kernel, all asynchronous on `stream`, no host synchronisation, so a
 * non-Python host can run the multi-GPU path.  NCCL is dlopen'ed at run time (the process's own copy if it has
 * loaded one); without it these calls return FLMR_ERR_UNSUPPORTED.
 *
 *   flmr_comm_unique_id   rank 0 obtains the 128-byte NCCL id and hands it to the other ranks (any host channel)
 *   flmr_comm_create      collective: ncclCommInitRank on `device`
 *   flmr_comm_adopt       wrap an existing ncclComm_t (not destroyed with the handle)
 *   flmr_topk_exchange    all-gather + merge of lists the caller already has (d_scores / d_pids [n_queries, k_in],
 *                         entries with pid < 0 ignored) -> [n_queries, k_out] on EVERY rank
 *   flmr_maxsim_topk_sharded   flmr_maxsim_topk on this rank's shard + flmr_topk_exchange, one call
 */
int flmr_comm_unique_id(void* out_id_128_bytes);
int flmr_comm_create(const void* id_128_bytes, int rank, int world_size, int device, flmr_comm_t** out);
int flmr_comm_adopt(void* nccl_comm, int device, flmr_comm_t** out);
int flmr_comm_destroy(flmr_comm_t* comm);
int flmr_comm_info(const flmr_comm_t* comm, int* rank, int* world_size);
int flmr_topk_exchange(flmr_comm_t* comm, const float* d_scores, const int64_t* d_pids, int n_queries, int k_in,
                       int k_out, float* d_out_scores, int64_t* d_out_pids, void* stream);
int flmr_maxsim_topk_sharded(const flmr_corpus_t* corpus, flmr_workspace_t* ws, flmr_comm_t* comm, const void* d_q,
                             int n_queries, int nq, int k, unsigned flags, float* d_out_scores,
                             int64_t* d_out_pids, void* stream);

/*
 * Top-k of dense score rows for k beyond FLMR_MAX_K (Searcher.dense_search accepts any k,
 * CB/searcher.py:91-132; replaces the `scores.sort(descending=True)[:k]` of IndexScorer.rank):
 * radix select + order-preserving compaction + bitonic sort, one block per query.
 *   d_scores fp32 [n_queries, n] (e.g. from flmr_maxsim_scores), k <= 2048, ties -> lower id first;
 *   outputs as flmr_maxsim_topk (pid = pid_base + column; -inf / -1 fill when n < k).
 */
int flmr_topk_select(const float* d_scores, int n_queries, int64_t n, int k, int64_t pid_base,
                     float* d_out_scores, int64_t* d_out_pids, int device, void* stream);

/*
 * Decode a chunk of a PLAID (ColBERTv2 residual-compressed) index into bf16 token embeddings,
 * so existing reference indexes can be scanned without re-encoding.  Replaces
 * decompress_residuals_cpp (CB/search/decompress_residuals.cpp:80-155), its CUDA twin
 * (CB/indexing/codecs/decompress_residuals.cu:8-75) and the F.normalize that follows
 * (CB/search/index_storage.py:173).  Synchronous on `stream` (validates the centroid codes).
 *   d_codes      int32 [n_tokens]            nearest-centroid id per token   (<c>.codes.pt)
 *   d_residuals  uint8 [n_tokens, dim*nbits/8] packed bucket indices         (<c>.residuals.pt)
 *   d_centroids  fp32  [n_centroids, dim]    (centroids.pt, upcast)
 *   d_bucket_weights fp32 [2^nbits]          (buckets.pt[1])
 *   d_out_bf16   bf16  [n_tokens, dim]       = normalize(centroids[code] + weights[idx]) if normalize
 */
int flmr_plaid_decode(const int32_t* d_codes, const uint8_t* d_residuals, int64_t n_tokens,
                      const float* d_centroids, int64_t n_centroids, const float* d_bucket_weights,
                      int nbits, int dim, int normalize, void* d_out_bf16, int device, void* stream);

/*
 * Gather retrieved passages out of the resident corpus into a padded batch — the operand of the RAG
 * re-score (src/models/rag/rag_model_blip.py:414-435 looks the embeddings up in a host dictionary, stacks
 * them and copies them to the device for every query; here they never leave HBM).
 *   d_pids   int64 [n_pids] GLOBAL passage ids (pid_base-relative ids are derived inside); ids outside
 *            this shard (e.g. the -1 fill of a short result list) produce an all-masked, zero row.
 *   d_out    bf16  [n_pids, nd_max, FLMR_DIM]  tokens, zero-padded; passages longer than nd_max are cut
 *   d_mask   uint8 [n_pids, nd_max]            1 for real tokens (may be NULL)
 * Asynchronous on `stream`.
 */
int flmr_corpus_gather(const flmr_corpus_t* corpus, const int64_t* d_pids, int64_t n_pids, int nd_max,
                       void* d_out_bf16, uint8_t* d_mask, void* stream);

/*
 * Backward of the all-pairs MaxSim used in training and RAG re-scoring (SURVEY.md 8f-2).  The
 * reference differentiates colbert_score through torch autograd (CB/modeling/colbert.py:235-286,
 * callers colbert.py:64-113 and src/models/rag/rag_model_blip.py:430-437), keeping the [n, Nd, Nq]
 * score tensor alive; here nothing is kept by the forward and the winners are recomputed:
 *
 * flmr_maxsim_argmax:   d_argmax[b, p, i] = argmax_{j : d_mask[p, j] != 0} <Q[b, i], D[p, j]>
 *                       (index into the PADDED document, lowest j on ties, -1 if p is fully masked);
 *                       d_rowmax (optional, fp32, same shape) receives the maximum itself: summed over i it
 *                       is score[b, p], so for a training-sized batch this one launch is the forward AND
 *                       saves what the backward needs (4 B per pair instead of the Nd scores).
 *                       Two kernels behind it: a warp-MMA one for small batches (a RAG re-score of 5 passages) and,
 *                       from 16M (query row, token) pairs up, a tcgen05 one (documents compacted to their unmasked
 *                       tokens, then a TMA / TMEM pipeline with the query tile stationary).
 * flmr_maxsim_backward: given d_grad[b, p] = dLoss/dScore[b, p],
 *                         d_dq[b, i, :]                  = sum_p grad[b, p] * D[p, argmax[b, p, i], :]
 *                         d_dd[p, argmax[b, p, i], :]   += grad[b, p] * Q[b, i, :]      (d_dd zeroed first)
 *                       either output may be NULL.  d_dd is accumulated with fp32 atomics.
 *   d_q     bf16 [n_queries, nq, FLMR_DIM]        d_docs bf16 [n_docs, nd, FLMR_DIM] (padded, contiguous)
 *   d_mask  uint8 [n_docs, nd] (any pattern, e.g. the punctuation mask of ColBERT.doc)
 *   d_argmax int32 [n_queries, n_docs, nq]        d_dq fp32 [n_queries, nq, FLMR_DIM]
 *   d_dd    fp32 [n_docs, nd, FLMR_DIM]
 * Asynchronous on `stream`; all pointers are device pointers on `device`.
 */
int flmr_maxsim_argmax(const void* d_q, int n_queries, int nq, const void* d_docs,
                       const uint8_t* d_mask, int n_docs, int nd, int32_t* d_argmax, float* d_rowmax,
                       int device, void* stream);
int flmr_maxsim_backward(const void* d_q, int n_queries, int nq, const void* d_docs, int n_docs, int nd,
                         const int32_t* d_argmax, const float* d_grad, float* d_dq, float* d_dd,
                         int device, void* stream);

/*
 * The loss head of ColBERT.compute_ib_loss_new (CB/modeling/colbert.py:82-113) on top of flmr_maxsim_argmax's
 * d_rowmax: scores[b, p] = sum_i rowmax[b, p, i]; cross-entropy of row b against the positive at column
 * label0 + b * nway (colbert.py:103-111; label0 = rank * B * nway with cross-rank negatives); and its gradient,
 * one launch instead of torch's sum + log_softmax + nll_loss and their backward kernels:
 *   d_scores fp32 [n_queries, n_docs]     d_loss_per_query fp32 [n_queries] (the loss is their mean)
 *   d_dscores fp32 [n_queries, n_docs] = d mean-loss / d scores — the d_grad operand of flmr_maxsim_backward
 */
int flmr_ib_loss(const float* d_rowmax, int n_queries, int n_docs, int nq, int nway, int label0,
                 float* d_scores, float* d_loss_per_query, float* d_dscores, int device, void* stream);

/*
 * Block-diagonal ("aligned") form of the two calls above: query b meets only ITS docs_per_query documents,
 * d_docs[b * docs_per_query .. (b + 1) * docs_per_query).  This is ColBERT.score(Q.repeat_interleave(nway), D,
 * D_mask) (CB/modeling/colbert.py:71-73, 217-224; src/models/rag/rag_model_blip.py:430-435;
 * src/executors/FLMR_executor.py:828-833) without materialising the repeated queries and without scoring the
 * off-diagonal pairs.
 *   d_docs  bf16 [n_queries * docs_per_query, nd, FLMR_DIM]    d_mask uint8 [n_queries * docs_per_query, nd]
 *   d_argmax / d_rowmax [n_queries, docs_per_query, nq]        d_grad fp32 [n_queries, docs_per_query]
 *   d_dq fp32 [n_queries, nq, FLMR_DIM]                        d_dd fp32 [n_queries * docs_per_query, nd, FLMR_DIM]
 */
int flmr_maxsim_argmax_grouped(const void* d_q, int n_queries, int nq, const void* d_docs,
                               const uint8_t* d_mask, int docs_per_query, int nd, int32_t* d_argmax,
                               float* d_rowmax, int device, void* stream);
int flmr_maxsim_backward_grouped(const void* d_q, int n_queries, int nq, const void* d_docs,
                                 int docs_per_query, int nd, const int32_t* d_argmax, const float* d_grad,
                                 float* d_dq, float* d_dd, int device, void* stream);

/* Test infrastructure: plain SIMT fp32 MaxSim of every passage (same contract as
 * flmr_maxsim_scores), independent of the tensor-core kernel. */
int flmr_debug_maxsim_scores_simt(const flmr_corpus_t* corpus, const void* d_q, int n_queries,
                                  int nq, unsigned flags, float* d_out_scores, void* stream);

/* Test infrastructure: which scan kernel searches on the calling thread launch — 0 = chosen per call and pass (the
 * product behaviour: CTA-pair passes for as many queries as fill them when the shard spans every SM, else normal
 * passes, those with three resident query tiles on the three-warpgroup kernel),
 * 2 = flmr_scan_kernel (two epilogue warpgroups), normal passes only, 3 = flmr_scan3_kernel (three warpgroups,
 * static query-tile assignment), normal passes only, 4 = CTA-pair passes (clusters of two CTAs stream one token
 * range, each D tile fetched once and TMA-multicast to both) whenever a call has enough queries, on any shard —
 * so the parity suite can run against any of them at any shape. */
int flmr_debug_set_scan_variant(int variant);

/* Test infrastructure: which kernel flmr_maxsim_argmax(_grouped) runs on the calling thread — 0 = chosen by size
 * (the product behaviour), 1 = the warp-MMA kernel, 2 = the tcgen05 kernel — so tests can hold either against
 * the other and the oracle at any shape. */
int flmr_debug_set_argmax_path(int path);

/* Test infrastructure, host-only (no GPU needed): the token-balanced CTA partition + per-tile
 * passage-end metadata the scan kernel consumes, for `n_ctas` persistent CTAs and
 * FLMR_TILE_TOKENS-token tiles (bit g of a tile's mask: a passage ends with 4-token group g).
 * cta_row_begin / cta_tile_base hold min(n_ctas, n_passages) + 1 entries; tile arrays may be NULL
 * to query *n_tiles_out only. */
int flmr_debug_build_partition(const int32_t* h_doclens, int64_t n_passages, int n_ctas,
                               int32_t* cta_row_begin, int64_t* cta_tile_base,
                               uint32_t* tile_end_mask, int32_t* tile_first_pid,
                               int64_t tile_capacity, int64_t* n_tiles_out);

/* Test infrastructure, host-only: the corpus passes flmr_maxsim_scores / flmr_maxsim_topk run for a batch of
 * `n_queries` queries of `nq` tokens (a pass = one scan-kernel launch with up to 640 query rows resident per CTA);
 * allow_pair != 0 plans CTA-pair passes (clusters of two CTAs share a token range, each with its own queries) for
 * the query prefix that fills them, as the library does on shards that span every SM.
 * out_plan (may be NULL to query *n_passes_out) receives 8 int32 per pass: first query, queries resident PER CTA (a
 * pair pass covers twice as many: CTA r the r-th half), first row, rows, 32-row blocks per query, 128-row tiles per
 * CTA, flags (1 = adds earlier partial scores, 2 = stores partial scores, 4 = final: scores complete, top-k taken,
 * 8 = pair pass), row of the pass's first query in the partial-score buffer. */
int flmr_debug_plan_passes(int n_queries, int nq, int allow_pair, int32_t* out_plan, int capacity, int* n_passes_out);

/* Kernels launched by this library on the calling thread since the last reset (bench evidence). */
int64_t flmr_launch_count(int reset);

/* Average device time (ms) of the scan kernel launches recorded since the last reset, measured
 * with CUDA events on the launching stream; requires flmr_set_profiling(1). */
int flmr_set_profiling(int enable);
int flmr_scan_kernel_stats(double* total_ms, int64_t* launches, int reset);

#ifdef __cplusplus
}
#endif
#endif /* FLMR_MAXSIM_H_ */
