/*
 * kirag_b200.h — C ABI of the B200-native (sm_100a) exact inner-product top-k
 * search and the mean-pool + L2-normalise embedding epilogue.
 *
 * This is the drop-in boundary for the one native dependency on KiRAG's
 * dense-retrieval hot path: the `faiss` module object as seen by
 * /root/reference/retriever/index.py:6.  Every entry point below names the
 * reference call site it replaces.  All signatures are plain C: pointers,
 * sizes, ints.  No torch / numpy types cross this boundary.
 *
 * Conventions
 *   - every function returning `int` returns 0 on success, non-zero on
 *     failure; the message is in kirag_last_error() (thread-local).  The
 *     library never calls abort()/exit().
 *   - `stream` is a cudaStream_t passed as void* (NULL = the legacy default
 *     stream).  Host-pointer entry points are synchronous (results are ready
 *     on return, like FAISS).  Device-pointer entry points are stream-ordered
 *     except where noted.
 *   - inputs are borrowed for the duration of the call; outputs are
 *     caller-owned buffers.  The index owns its copy of the corpus (FAISS
 *     copies on add(), reference call site retriever/index.py:32).
 *   - threading: calls on DIFFERENT index handles may run concurrently from different host threads;
 *     calls on the SAME handle must be serialised by the caller (search workspaces belong to the
 *     handle).  KiRAG's callers are single-threaded Python (retriever/retrievers.py:250-275).
 *   - there is NO CPU fallback.  If no CUDA device is usable every call fails
 *     with a non-zero status.
 */
#ifndef KIRAG_B200_H
#define KIRAG_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KIRAG_ABI_VERSION 7

/* metric ids; only inner product is implemented, as only inner product is
 * ever constructed by the reference (retrieve.py:112, faiss_index_corpus.py:29) */
#define KIRAG_METRIC_INNER_PRODUCT 0
#define KIRAG_METRIC_L2 1

/* search path selectors for kirag_index_search_ex() */
#define KIRAG_PATH_AUTO 0   /* tcgen05 bf16 filter scan + fp32 rescoring, certified; exact fp32 scan for uncertified queries */
#define KIRAG_PATH_EXACT 1  /* fp32 CUDA-core scan of the fp32 master only */
#define KIRAG_PATH_FAST 2   /* bf16 filter scan + rescoring, certificate evaluated and reported but not acted on */

/* hidden-state dtypes for kirag_pool_normalize() */
#define KIRAG_DTYPE_F32 0
#define KIRAG_DTYPE_BF16 1
#define KIRAG_DTYPE_F16 2

/* mask dtypes */
#define KIRAG_MASK_I64 0
#define KIRAG_MASK_I32 1
#define KIRAG_MASK_U8 2

/* pooling modes */
#define KIRAG_POOL_MEAN 0 /* E5Encoder.forward tail: retriever/encoders.py:56-58,75-76 */
#define KIRAG_POOL_CLS 1  /* BGEEncoder.forward tail: retriever/encoders.py:115-117 */

typedef struct kirag_index kirag_index_t;

/* per-call search statistics (all counts are queries unless noted) */
typedef struct kirag_search_stats {
    int64_t nq;              /* queries in the call */
    int64_t n_fast;          /* answered by the tcgen05 filter path with a passing certificate (first attempt) */
    int64_t n_exact;         /* answered by the exact fp32 scan (forced, ineligible shape, or escalated) */
    int64_t n_cert_fail;     /* certificate failures observed on the filter path */
    int64_t n_overflow;      /* candidate-buffer overflows observed on the filter path */
    int32_t levels;          /* filter launches (geometric levels) of the last query chunk */
    int32_t path;            /* path actually taken for the bulk of the call (KIRAG_PATH_*) */
    int64_t kernel_launches; /* kernels launched by this library during the call */
    int64_t n_rescan;        /* certificate failures answered by the second bf16 pass (threshold s_k - eps) */
    int64_t n_retry;         /* buffer overflows answered by re-running the filter path with the gentle level schedule */
} kirag_search_stats_t;

/* ---- library ---------------------------------------------------------- */

/* ABI version of the loaded library (== KIRAG_ABI_VERSION it was built with). */
int kirag_abi_version(void);

/* Thread-local message of the last failing call on this thread ("" if none). */
const char* kirag_last_error(void);

/* Number of usable CUDA devices (0 if none / no driver).  Never fails. */
int kirag_device_count(void);

/* Per-kernel timing of the dominant kernel (the tcgen05 filter scan) with CUDA
 * events recorded on the launching stream; used by bench.py for the roofline
 * line.  enable(1) clears and starts recording, read() returns the summed
 * duration (ms), the number of launches and the corpus rows they streamed,
 * then clears. */
int kirag_profile_enable(int on);
int kirag_profile_read(double* scan_ms, int64_t* scan_launches, double* scan_rows);
/* Per-launch durations (ms) and corpus rows of the recorded scan launches, up to max_n entries;
 * does not clear (call before kirag_profile_read). */
int kirag_profile_read_launches(double* ms_out, double* rows_out, int64_t max_n);
/* Timeline of the recorded search phases: tag 0 start, 1 queries converted, 10+l scan of level l
 * done, 30+l select of level l done, 50 rescored, 51 final written; ms relative to the first mark.
 * Returns the number of entries written; does not clear. */
int kirag_profile_read_timeline(int* tags_out, double* ms_since_first, int64_t max_n);

/* ---- flat inner-product index  (replaces faiss.IndexFlatIP) ------------ */

/* faiss.IndexFlatIP(d)                      retriever/index.py:13,23 */
int kirag_index_create(int d, int metric, int device, kirag_index_t** out);

/* destructor of the faiss index object */
int kirag_index_destroy(kirag_index_t* h);

/* Pre-size device storage for n_total rows (optional; add() grows as needed). */
int kirag_index_reserve(kirag_index_t* h, int64_t n_total);

/* index.add(x)                              retriever/index.py:32
 * x: row-major float32 [n, d]; host pointer (x_is_device == 0) or device
 * pointer on the index's device.  Rows get implicit ids ntotal .. ntotal+n-1. */
int kirag_index_add(kirag_index_t* h, const float* x, int64_t n, int x_is_device, void* stream);

/* index.ntotal                              retriever/index.py:74,79 */
int64_t kirag_index_ntotal(const kirag_index_t* h);

/* index.d */
int kirag_index_dim(const kirag_index_t* h);

/* index.search(x, k)                        retriever/index.py:47
 * q: float32 [nq, d]; D: float32 [nq, k]; I: int64 [nq, k].
 * Rows of D/I are ordered by (score descending, id ascending); unfilled slots
 * (k > ntotal) hold D = -FLT_MAX (numeric_limits<float>::lowest()), I = -1,
 * which is FAISS's heap neutral element.  `id_offset` is added to every
 * returned id (row-sharded multi-GPU search: global id = local row + offset).
 * k <= 2048; the over-fetch of the filter path is k' = min(4k, 2048).
 * ptrs_are_device: 0 = q/D/I are host pointers.  The call is synchronous like FAISS; results and the
 *                      per-query certificate flags come back together, ONE stream synchronisation
 *                      per 16384 queries (a second one only if a query had to be re-answered).
 *                  1 = device pointers on the index's device.  The work is enqueued on `stream`, then
 *                      the call synchronises ONCE (per 16384 queries) to read the certificate flags and
 *                      re-answers flagged queries before returning: on return D/I are final, but the
 *                      call is NOT purely stream-ordered.  Use kirag_index_search_async +
 *                      kirag_index_search_finish where the synchronisation has to move (e.g. behind a
 *                      collective) or where the call is captured into a CUDA graph. */
int kirag_index_search(kirag_index_t* h, const float* q, int64_t nq, int k,
                       float* D, int64_t* I, int ptrs_are_device, int64_t id_offset, void* stream);

/* Same, with an explicit path selector and optional statistics. */
int kirag_index_search_ex(kirag_index_t* h, const float* q, int64_t nq, int k,
                          float* D, int64_t* I, int ptrs_are_device, int64_t id_offset,
                          int path, kirag_search_stats_t* stats, void* stream);

/* index.range_search(x, radius)             (faiss IndexFlatIP::range_search; no reference call site)
 * Every row j with canonical fp32 score s_qj > radius (strict, FAISS's rule for inner product).  NaN scores are never
 * returned; a NaN or +inf radius gives empty lists, -inf every row whose score is a number above -inf.  Scores are
 * bit-identical to what kirag_index_search returns for the same (query, row); each query's list is ordered by
 * (score descending, id ascending) (FAISS leaves the order unspecified); `id_offset` is added to every id.
 * Layout is FAISS's: query i owns entries [lims[i], lims[i+1]) of D (float32) / I (int64), lims[nq] in all.
 * q: float32 [nq, d], host or device (q_is_device).  lims_out: HOST int64 [nq + 1].  Synchronous.
 * path: KIRAG_PATH_AUTO / KIRAG_PATH_FAST one bf16 filter pass with the threshold radius - eps(q) (complete by
 *       construction) + fp32 rescoring, a second pass for queries with more survivors than the candidate buffer
 *       holds (stats: n_fast / n_overflow, levels 1 or 2); the exact fp32 scan for shapes the filter cannot take
 *       (d % 64 != 0, more than 0x7fffff00 rows); KIRAG_PATH_EXACT the fp32 scan.  AUTO and EXACT agree bit for bit.
 * The D/I entries stay in the handle (grow-only workspaces, no allocation once warm) until kirag_index_range_fetch;
 * the next search, add or range search on the handle drops them.  A call that fails (e.g. a result that does not fit
 * in device memory) holds nothing. */
int kirag_index_range_search(kirag_index_t* h, const float* q, int64_t nq, float radius, int q_is_device,
                             int64_t id_offset, int path, int64_t* lims_out, kirag_search_stats_t* stats,
                             void* stream);
/* Copies the lims_out[nq] entries of the last range search into D (float32) / I (int64), host or device
 * (ptrs_are_device), and releases the held result (a second fetch is an error).  Synchronous.  An error if nothing is
 * held. */
int kirag_index_range_fetch(kirag_index_t* h, float* D, int64_t* I, int ptrs_are_device, void* stream);

/* Stream-ordered half of a device-pointer search (KIRAG_PATH_AUTO, nq <= 16384): enqueues every kernel of the
 * first attempt (filter levels, fp32 rescoring, final sort, certificate) and the copy of the certificate flags to
 * pinned host memory on `stream` and returns WITHOUT synchronising.  D/I then hold the answer of every query whose
 * certificate passed (all of them on well-spread data); the caller may enqueue further work that consumes them.
 * No cudaMalloc / pageable copy happens once the workspaces are warm (one earlier call with the same nq and k), so
 * the call can be captured into a CUDA graph.  The search is completed by kirag_index_search_finish; any other
 * call on the handle completes it implicitly first.  q/D/I must stay valid until then. */
int kirag_index_search_async(kirag_index_t* h, const float* q, int64_t nq, int k,
                             float* D, int64_t* I, int64_t id_offset, void* stream);

/* Second half: waits for the asynchronous search (the event recorded on its stream; after a graph replay the
 * stream it was captured on is synchronised instead), examines the certificate flags and re-answers flagged
 * queries in place (second bf16 pass with the provable threshold, exact fp32 scan as the last resort).
 * n_changed (optional) = number of queries whose rows of D/I were rewritten: consumers that already read D/I
 * (e.g. an exchange between GPUs) must run again when it is non-zero.  Returns with the stream idle. */
int kirag_index_search_finish(kirag_index_t* h, kirag_search_stats_t* stats, int64_t* n_changed);

/* Device pointer to the per-query certificate flags of the pending asynchronous search (int32 [nq]: 0 certified,
 * 1 certificate failed, 2 candidate buffer overflowed), NULL if nothing is pending or the exact path answered.
 * Lets a following kernel (the multi-GPU exchange) carry the flags along without a host round trip. */
int kirag_index_search_flags(const kirag_index_t* h, const int** flags_dev);

/* CUDA-graph replay of a captured kirag_index_search_async (KiRAG's own call shape is 1-2 queries per retrieval,
 * knowledge_graph/models.py:1645: a dozen launches per search are then what a call costs on the host).  After the
 * graph that contains the captured call has been launched on `stream`, this marks that search pending again, so that
 * kirag_index_search_finish examines the certificate flags of the REPLAY and re-answers flagged queries in the
 * captured D/I buffers.  Any other call on the handle completes a pending search first, as always. */
int kirag_index_search_rearm(kirag_index_t* h, void* stream);

/* A captured search has the index storage, the workspaces and the certificate constants baked into its kernel
 * arguments.  The token changes whenever one of them does (rows added, a workspace grown by a larger call):
 * replay a graph only while the token equals the one read right after the capture. */
int kirag_index_state_token(const kirag_index_t* h, uint64_t* token);

/* index.reconstruct_n(i0, n): copy rows [i0, i0+n) of the fp32 master out. */
int kirag_index_reconstruct(const kirag_index_t* h, int64_t i0, int64_t n, float* out,
                            int out_is_device, void* stream);

/* faiss.write_index(index, path)            retriever/index.py:62
 * Writes the FAISS "IxFI" flat-index container (see DESIGN.md). */
int kirag_index_save(const kirag_index_t* h, const char* path);

/* faiss.read_index(path, flags)             retriever/index.py:73 */
int kirag_index_load(const char* path, int device, kirag_index_t** out);

/* Raw device pointers of the index storage (for zero-copy integration and
 * for the benchmark's synthetic-corpus generator).  fp32 master is row-major
 * [ntotal, d]. */
int kirag_index_device_ptrs(const kirag_index_t* h, const float** master_f32, const void** shadow_bf16);

/* Test hook (host only, no device needed): the level schedule of the filter path for a search of nq queries
 * over n_rows rows: rows_hi_out[l] = number of corpus rows covered after level l (the last entry is n_rows).
 * Returns the number of levels (> 0), -1 if the shape is not eligible for the filter path (exact scan),
 * -2 (kirag_last_error() set) on a bad argument.  cap_out: candidate-buffer entries per query;
 * kprime_out: the over-fetch k' = max(4k, 32). */
int kirag_debug_level_schedule(int64_t n_rows, int64_t nq, int k, int d, int64_t* rows_hi_out, int max_levels,
                               int* cap_out, int* kprime_out);

/* Test hook: dense approximate scores of the bf16 tcgen05 scan, written to a
 * host buffer laid out [ntotal, nq].  Used by the parity tests to check the
 * tensor-core contraction in isolation from the top-k logic. */
int kirag_index_debug_scores(kirag_index_t* h, const float* q_host, int64_t nq, float* out_host);

/* Merge G per-shard results into the global top-k, (score desc, id asc).
 * D_all: float32 [G, nq, k]; I_all: int64 [G, nq, k] (entries with id < 0 are
 * padding).  Used after the NCCL all-gather of the row-sharded search. */
int kirag_merge_topk(const float* D_all, const int64_t* I_all, int G, int64_t nq, int k,
                     float* D_out, int64_t* I_out, int ptrs_are_device, int device, void* stream);

/* ---- peer-memory exchange of the row-sharded search (one process per GPU) ---
 * Replaces "NCCL all-gather of the per-shard [nq,k] results + kirag_merge_topk" by ONE kernel per
 * rank that stores its result rows into every rank's exchange buffer over NVLink (buffers mapped
 * with CUDA IPC), waits per query range for the other ranks' rows and merges them.  No counterpart
 * in the reference (FAISS search is single-process CPU, retriever/index.py:47).
 * SPMD contract: every rank makes the same sequence of kirag_exchange_merge_topk calls with the
 * same nq and k.  The 64-byte IPC handles are exchanged by the host (torch.distributed). */
typedef struct kirag_exchange kirag_exchange_t;

/* Allocate this rank's exchange buffer: capacity max_nq*max_k result entries per rank and parity. */
int kirag_exchange_create(int device, int rank, int world, int64_t max_nq, int max_k, kirag_exchange_t** out);
int kirag_exchange_destroy(kirag_exchange_t* x);
/* sizeof(cudaIpcMemHandle_t) (64) */
int kirag_exchange_handle_bytes(void);
/* Write this rank's IPC handle (kirag_exchange_handle_bytes() bytes) to handle_out. */
int kirag_exchange_export(kirag_exchange_t* x, void* handle_out);
/* handles_all: world * kirag_exchange_handle_bytes() bytes, rank-major; maps every peer's buffer. */
int kirag_exchange_connect(kirag_exchange_t* x, const void* handles_all);
/* Same with raw device pointers (ranks living in one process: peer_buffers[g] = kirag_exchange_buffer
 * of rank g; entry [rank] is ignored). */
int kirag_exchange_connect_ptrs(kirag_exchange_t* x, void* const* peer_buffers);
void* kirag_exchange_buffer(kirag_exchange_t* x);
/* D_loc/I_loc: this rank's per-shard result [nq,k] (device, rows sorted by (score desc, id asc), global
 * ids, padding id -1); D_out/I_out: the global top-k [nq,k] (device), identical on every rank.
 * Stream-ordered; the kernel spins (bounded, ~20 s) until every peer's call has delivered.  The buffers are
 * double-buffered by call parity, which is only safe if a rank's exchanges EXECUTE in call order: calls on one
 * stream are ordered by it, a call on another stream first waits (cudaStreamWaitEvent) for the previous exchange.
 * The call parity (epoch) lives on the device, so a captured call can be replayed from a CUDA graph; whoever
 * replays it orders the replays against the rank's other exchanges (e.g. by synchronising the replay stream). */
int kirag_exchange_merge_topk(kirag_exchange_t* x, const float* D_loc, const int64_t* I_loc, int64_t nq, int k,
                              float* D_out, int64_t* I_out, void* stream);

/* Same, and every rank's per-query certificate flags (int32 [nq], device: kirag_index_search_flags of the pending
 * asynchronous search) travel with its rows; the kernel ORs them over all ranks and queries.  The result — read
 * with kirag_exchange_last_any_flag once the stream has been synchronised — is IDENTICAL on every rank, so all
 * ranks decide together, without a host collective, whether some rank has to re-answer queries
 * (kirag_index_search_finish) and the exchange has to run again.  nq <= the max_nq given at creation. */
int kirag_exchange_merge_topk_flags(kirag_exchange_t* x, const float* D_loc, const int64_t* I_loc, const int* flags_loc,
                                    int64_t nq, int k, float* D_out, int64_t* I_out, void* stream);
/* OR of the flags carried by the last kirag_exchange_merge_topk_flags call (valid after its stream was synchronised);
 * -2 (kirag_last_error() set) if an exchange timed out waiting for a peer. */
int kirag_exchange_last_any_flag(kirag_exchange_t* x);

/* torch.topk(torch.matmul(Q, T.T), k, dim=1)   knowledge_graph/models.py:1532-1538
 * One-shot search over a transient candidate matrix T [nt, d] (device or host
 * pointers).  T is indexed in a per-(device, d) scratch index owned by the library whose device
 * buffers are kept between calls (no allocation once warm); calls are serialised by a mutex.
 * Synchronises like kirag_index_search. */
int kirag_topk_ip(const float* q, int64_t nq, const float* t, int64_t nt, int d, int k,
                  float* D, int64_t* I, int ptrs_are_device, int device, void* stream);
/* Frees the scratch indexes of kirag_topk_ip (optional; e.g. before a process gives a GPU back). */
int kirag_topk_ip_release(void);

/* ---- embedding epilogue (replaces average_pool + F.normalize) ---------- */

/* out[b,:] = normalize(pool(hidden[b], mask[b]))   retriever/encoders.py:56-58,75-76 (mean)
 *                                                   retriever/encoders.py:115-117    (cls)
 *                                                   retriever/e5.py:46-48,59-60      (mean, duplicate)
 * hidden: device [B, S, H] with element strides (sb, ss, 1); mask: device
 * [B, S] with element strides (mb, 1); out: device float32 [B, H] contiguous.
 * normalize = x / max(||x||_2, 1e-12) (torch F.normalize eps).  If
 * `normalize` == 0 only the pooling is applied (ContrieverEncoder tail,
 * encoders.py:94-95).  An all-zero mask row divides by zero exactly like the
 * reference does (nan/inf), it is not "fixed".  Stream-ordered. */
int kirag_pool_normalize(const void* hidden, const void* mask, float* out,
                         int64_t B, int64_t S, int64_t H, int64_t sb, int64_t ss, int64_t mb,
                         int hidden_dtype, int mask_dtype, int mode, int normalize,
                         int device, void* stream);

/* Backward of kirag_pool_normalize (mean or cls mode, normalize on or off):
 * grad_hidden [B,S,H] contiguous, same dtype as `hidden_dtype`; `out` is the
 * forward output, grad_out float32 [B,H].  `pooled_norm` float32 [B] is the
 * pre-normalisation L2 norm saved by the forward (see kirag_pool_normalize_fwd_saved). */
int kirag_pool_normalize_backward(const float* grad_out, const float* out, const float* pooled_norm,
                                  const void* mask, void* grad_hidden,
                                  int64_t B, int64_t S, int64_t H, int64_t mb,
                                  int hidden_dtype, int mask_dtype, int mode, int normalize,
                                  int device, void* stream);

/* Forward that additionally writes the pre-normalisation norms (float32 [B]). */
int kirag_pool_normalize_fwd_saved(const void* hidden, const void* mask, float* out, float* pooled_norm,
                                   int64_t B, int64_t S, int64_t H, int64_t sb, int64_t ss, int64_t mb,
                                   int hidden_dtype, int mask_dtype, int mode, int normalize,
                                   int device, void* stream);

/* Forward that also writes the result in the dtype of the hidden states (out_typed: device [B, H] of hidden_dtype —
 * what the reference's ops return for bf16 / fp16 hidden states under autocast, base_trainer.py:498-499), in the same
 * kernel instead of a separate cast.  out (float32) is still written: the backward needs it; pooled_norm may be NULL. */
int kirag_pool_normalize_typed(const void* hidden, const void* mask, float* out, void* out_typed, float* pooled_norm,
                               int64_t B, int64_t S, int64_t H, int64_t sb, int64_t ss, int64_t mb,
                               int hidden_dtype, int mask_dtype, int mode, int normalize,
                               int device, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* KIRAG_B200_H */
