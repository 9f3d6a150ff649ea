/*
 * vidmem.h -- C ABI of libvidmem.so, the B200 (sm_100a) embedding-similarity engine.
 *
 * The reference (RaphaelHaddad/Real-Time-Brain-Inspired-Video-Memory, "VidGraph") is pure
 * Python and has NO FFI/plugin interface for this path (SURVEY.md 8b): the seams it exposes
 * are Python methods.  Each entry point below therefore cites the reference method whose
 * arithmetic it replaces; the Python adapters that keep those method signatures live in
 * real-time-brain-inspired-video-memory_b200/adapters.py and the binding a maintainer would
 * add to the reference is shown in INTEGRATION.md.
 *
 * Conventions
 *  - C linkage, plain pointers and sizes, no torch / C++ types.
 *  - Every function returns int: VM_OK (0) or a negative vm_status; vm_last_error() returns a
 *    thread-local message for the last failure on the calling thread.
 *  - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).  Work is
 *    enqueued on it.  Calls whose outputs live in HOST memory synchronise the stream before
 *    returning; calls whose inputs and outputs are all DEVICE memory and that pass
 *    VM_FLAG_ASYNC return as soon as the work is enqueued (outputs valid after the stream
 *    reaches that point).
 *  - The library owns only opaque handles (vm_store, vm_comm) and its workspaces; every
 *    input/output buffer is owned by the caller.
 *  - One caller thread per store (the reference calls this path from a single asyncio
 *    thread, SURVEY.md 8b); handles are not re-entrant.
 *  - There is no CPU fallback: without a CUDA device of compute capability 10.x every compute
 *    entry point fails with VM_ERR_CUDA / VM_ERR_UNSUPPORTED.
 *
 * Row identity: the engine works on dense row indices (append order == store order of the
 * reference's dict, SURVEY.md 9.2); the adapters keep the row <-> chunk-id table on the host.
 */
#ifndef VIDMEM_H_
#define VIDMEM_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VM_ABI_VERSION 1

typedef enum vm_status {
    VM_OK = 0,
    VM_ERR_BADARG = -1,
    VM_ERR_OOM = -2,
    VM_ERR_CUDA = -3,
    VM_ERR_NCCL = -4,
    VM_ERR_OVERFLOW = -5,    /* a caller-provided output capacity was exceeded (count is still returned) */
    VM_ERR_UNSUPPORTED = -6, /* wrong GPU architecture / shape outside the supported envelope */
    VM_ERR_STATE = -7
} vm_status;

typedef enum vm_dtype { VM_F32 = 0, VM_BF16 = 1, VM_F64 = 2 } vm_dtype;
typedef enum vm_mem { VM_MEM_HOST = 0, VM_MEM_DEVICE = 1 } vm_mem;

/* Score convention of the returned `score` field.
 *   VM_SCORE_RAW   : cosine, as PreLLMInjector._cosine_similarity returns it
 *                    (src/components/pre_llm_injector.py:374-388).
 *   VM_SCORE_NEO4J : (1 + cosine) / 2, the normalised value Neo4j's vector.similarity.cosine
 *                    yields in the Cypher of _vector_search_chunks
 *                    (src/pipeline/retriever_hybrid.py:295-301; SURVEY.md 9.3, parity unpinned).
 * `min_score` (strict `>`) is applied to the value in the selected convention. */
typedef enum vm_score_mode { VM_SCORE_RAW = 0, VM_SCORE_NEO4J = 1 } vm_score_mode;

/* Summation order of the reference's Python `sum()` over binary64 products:
 * plain left-to-right on CPython < 3.12, Neumaier-compensated on CPython >= 3.12. */
typedef enum vm_sum_mode { VM_SUM_NAIVE = 0, VM_SUM_NEUMAIER = 1 } vm_sum_mode;

enum {
    VM_FLAG_ASYNC = 1,       /* do not synchronise (device outputs only) */
    VM_FLAG_FORCE_EXACT = 2, /* skip the fast scan: binary64 scan of every row (slow, always exact) */
    VM_FLAG_FORCE_SIMT = 4,  /* use the CUDA-core scan kernel even where the tcgen05 kernel applies */
    VM_FLAG_FORCE_TC = 8,    /* accepted and ignored: the tcgen05/TMA scan kernel is the default wherever it applies */
    VM_FLAG_TIMING = 16,     /* bracket the scan kernel with CUDA events on `stream` (see vm_store_last_scan_ms);
                                also launches the call's kernels without programmatic overlap */
    VM_FLAG_NO_SPLIT = 32,   /* bf16 store: feed the query as ONE bf16 term (scan error bound 2^-8) */
    VM_FLAG_SPLIT = 64       /* bf16 store: feed the query as hi + lo bf16 terms, two MMAs per K slice (scan error bound
                                ~2^-16 + (D+16) 2^-23 < 1e-4 at 384-d).  Default: split for batches of <= 48 queries,
                                where it is free; single term above (the complete near-tie band is rescored either way). */
};

typedef struct vm_store vm_store; /* a row-major embedding store resident in HBM (one shard) */
typedef struct vm_comm vm_comm;   /* an NCCL communicator wrapper (one rank) */

/* Filled by vm_topk* when `stats` is non-NULL (all values for the last call). */
typedef struct vm_topk_stats {
    int32_t scan_kernel;      /* 0 = exact only, 1 = SIMT scan, 2 = tcgen05 scan */
    int32_t scan_launches;    /* kernels launched by the call (all kinds) */
    int32_t uncertified;      /* queries left for a fallback pass after the rescoring kernel (it settles near-tie bands itself):
                                 settled by the collect pass or the binary64 scan of every row */
    int32_t candidates;       /* candidate list length per query (KP) */
    int32_t scan_ctas;
    int32_t scan_stages;      /* shared-memory pipeline depth of the tcgen05 scan (0 otherwise) */
    int32_t full_rescans;     /* of the uncertified queries, how many the collect pass could not settle and the
                                 binary64 scan of every row re-did (-1: not read back, e.g. graph replay) */
    int32_t scan_variant;     /* tcgen05 scan: 1 = dump mode (small store: every row's key is ranked), 2 = band mode (lock-free
                                 per-CTA slabs + spill buffer, cooperative bounds); 0 = not a tcgen05 scan */
} vm_topk_stats;

/* ---- library ----------------------------------------------------------------------- */
int vm_version(void);                  /* VM_ABI_VERSION */
const char *vm_last_error(void);       /* thread-local, never NULL */
/* sm count / compute capability / HBM bytes of `device`; any out pointer may be NULL */
int vm_device_info(int device, int *sm_count, int *cc_major, int *cc_minor, size_t *total_mem);

/* ---- embedding store (one shard = rows resident on one GPU) --------------------------
 * Replaces the per-call store fetch of PreLLMInjector._get_chunk_embeddings
 * (src/components/pre_llm_injector.py:390-412: the whole store crosses Bolt every batch) with
 * rows that stay resident in HBM.  dtype is VM_F32 or VM_BF16; `dim` is the logical embedding
 * length; rows are stored with a leading dimension of vm_store_ld() elements (dim rounded up
 * to 8, zero padded). */
int vm_store_create(vm_store **out, int device, int dim, int dtype, int64_t capacity);
/* Same, over caller-owned device buffers (e.g. torch tensors): rows_dev holds
 * capacity * vm_ld(dim) elements of `dtype`, inv_norms_dev holds capacity floats. */
int vm_store_attach(vm_store **out, int device, int dim, int dtype, int64_t capacity, void *rows_dev,
                    float *inv_norms_dev);
/* BINARY64 store: the rows are kept exactly as given (the reference scores Python float lists, i.e. binary64:
 * pre_llm_injector.py:382-388), [capacity][ld] doubles, next to a rounded SHADOW copy in `shadow_dtype` (VM_F32 or
 * VM_BF16) that only the streaming scan reads.  Candidate selection runs on the shadow with an error bound widened
 * by the shadow's rounding (2^-24 / 2^-8 in cosine units, with margin); every exact step -- rescoring, near-tie band,
 * collect pass, binary64 scan -- reads the binary64 rows.  Returned scores and order are therefore those of the reference formula on
 * the ORIGINAL values, whatever their representability in fp32 / bf16.  HBM per row: ld * (8 + sizeof(shadow)) + 4
 * bytes; scan traffic is that of the shadow alone.  vm_store_attach_exact: rows_exact_dev holds capacity * vm_ld(dim)
 * doubles (16-byte aligned).  Rows whose elements overflow the shadow type, or that vanish in it, stay scorable: they
 * are counted as out of range and every query then also takes the binary64 pass (exact, slower). */
int vm_store_create_exact(vm_store **out, int device, int dim, int shadow_dtype, int64_t capacity);
int vm_store_attach_exact(vm_store **out, int device, int dim, int shadow_dtype, int64_t capacity, void *rows_dev,
                          float *inv_norms_dev, double *rows_exact_dev);
/* GROWABLE store (SURVEY.md H6: the reference's store only ever grows, one SET c.embedding per new chunk,
 * neo4j_handler.py:221-253).  The library reserves a VIRTUAL address range for max_capacity rows and backs it with
 * physical HBM from its start as rows arrive (CUDA virtual memory management): vm_store_append grows the backed part on
 * demand (what the append needs + 256 MB of slack, capped at max_capacity), vm_store_reserve grows it explicitly.  Base addresses never change and
 * resident rows are never copied -- no second allocation, no device-to-device copy, HBM in use = the backed rows.
 * exact != 0: a binary64 store as vm_store_create_exact (dtype = the shadow type). */
int vm_store_create_growable(vm_store **out, int device, int dim, int dtype, int exact, int64_t initial_capacity,
                             int64_t max_capacity);
int vm_store_reserve(vm_store *s, int64_t capacity);    /* no-op when capacity <= vm_store_capacity(s) */
int64_t vm_store_max_capacity(const vm_store *s);       /* == capacity for a store over fixed buffers */
size_t vm_store_resident_bytes(const vm_store *s);      /* physical HBM behind rows + inverse norms (+ binary64 rows) */
/* device addresses of the store's buffers (valid for the store's lifetime; rows beyond vm_store_capacity() of a
 * growable store are not backed) */
void *vm_store_rows_ptr(const vm_store *s);
float *vm_store_inv_norms_ptr(const vm_store *s);
double *vm_store_rows_exact_ptr(const vm_store *s);     /* NULL unless a binary64 store */
int vm_store_destroy(vm_store *s);
int64_t vm_store_size(const vm_store *s);
int64_t vm_store_capacity(const vm_store *s);
int vm_store_dim(const vm_store *s);
int vm_store_ld(const vm_store *s);
int vm_ld(int dim); /* leading dimension used for a given dim */

/* Append n rows ([n][dim], row-major, src_dtype VM_F32/VM_BF16/VM_F64, host or device).
 * Replaces the per-row `SET c.embedding = $embedding` round trip of
 * Neo4jHandler._create_chunks_with_embeddings (src/components/neo4j_handler.py:221-253) as the
 * insert hook; values are rounded to the store dtype once, and 1/||row|| of the STORED values
 * is cached (binary64 accumulate) -- this is the "fused normalisation" the scan kernels use.
 * first_row (may be NULL) receives the index of the first appended row.  A later vm_topk on
 * the same stream sees every row appended before it. */
int vm_store_append(vm_store *s, const void *rows, int src_dtype, int src_mem, int64_t n, int64_t *first_row,
                    void *stream);
/* Overwrite rows [row0, row0+n) in place (idempotent upsert by id, neo4j_handler.py:229 MERGE). */
int vm_store_update(vm_store *s, int64_t row0, const void *rows, int src_dtype, int src_mem, int64_t n,
                    void *stream);
/* Mark rows as skipped: they are never returned, like a falsy `existing_emb`
 * (src/components/pre_llm_injector.py:363) or `c.embedding IS NULL` (retriever_hybrid.py:296). */
int vm_store_invalidate(vm_store *s, const int64_t *rows_host, int64_t n, void *stream);
/* Tell an attached store that rows [0, n) are already filled (e.g. generated on device);
 * recomputes the cached inverse norms for [row0, n). */
int vm_store_set_size(vm_store *s, int64_t n, int64_t recompute_from_row, void *stream);
int vm_store_clear(vm_store *s);
/* Device time (ms) of the scan kernel(s) of the last vm_topk* call made with VM_FLAG_TIMING,
 * measured with CUDA events recorded on that call's stream; synchronises on the end event. */
int vm_store_last_scan_ms(vm_store *s, float *ms);
/* Average scan-kernel time (ms) over the VM_FLAG_TIMING calls made since the previous read (the most
 * recent 64 at most), each bracketed by its own event pair on its stream -- nothing is synchronised
 * until this call, so a back-to-back timed loop is measured as it ran.  *calls (optional) = how many. */
int vm_store_avg_scan_ms(vm_store *s, float *ms, int *calls);

/* Certification counters over the store's lifetime (or since the last reset), kept on the device by the
 * rescoring kernels so that they also cover VM_FLAG_ASYNC calls and graph replays, whose per-call stats
 * cannot report them.  queries = uncertified + (queries certified by the first pass); every uncertified query
 * is settled exactly by one of the three fallbacks.  Synchronises with the device. */
typedef struct vm_store_counters {
    int64_t batches;          /* scan passes (<= 64 queries each) */
    int64_t queries;          /* queries scored */
    int64_t uncertified;      /* queries whose first candidate list could not be certified */
    int64_t band_settled;     /* ... settled inside the same pass from the complete near-tie band (no second scan) */
    int64_t collect_settled;  /* ... settled by the collect pass (one more streaming scan) */
    int64_t full_rescans;     /* ... redone by the binary64 scan of every row */
    int64_t bound_violations; /* queries in which a rescored candidate's approximate score was further from its exact
                                 score than the scan's error bound (audited on every candidate; such a query is always
                                 redone by the binary64 scan).  Expected: 0. */
} vm_store_counters;
int vm_store_read_counters(vm_store *s, vm_store_counters *out, int reset);

/* Diagnostics of the last tcgen05 scan of this store: per query, how many keys the scan kept in the near-tie band
 * (appended to the per-CTA slabs, including those that went on to the spill buffer) and how many were spilled --
 * a measure of how tight the cooperative bounds were.  nq_cap = room in the two arrays (>= queries of that scan).
 * Synchronises with the device. */
int vm_store_band_keys(vm_store *s, int nq_cap, int64_t *kept_per_query, int64_t *spilled_per_query, int *nq_out);

/* ---- top-k scorer ---------------------------------------------------------------------
 * Replaces the hot loop of PreLLMInjector._calculate_batch_similarities
 * (src/components/pre_llm_injector.py:356-370: every query x every stored row through
 * _cosine_similarity, stable sort descending, slice [:k]) and the exhaustive Cypher scan of
 * HybridRetriever._vector_search_chunks (src/pipeline/retriever_hybrid.py:293-306).
 *
 *  queries    [nq][dim] row-major, q_dtype VM_F32/VM_BF16/VM_F64, q_mem host or device
 *  k          entries wanted per query, 1 <= k <= 64
 *  min_score  strict lower bound on the returned score (use -INFINITY for none)
 *  out_idx    [nq][k] int64 row indices, best first; ties -> lowest row (SURVEY.md 9.2)
 *  out_score  [nq][k] binary64 scores, BIT-IDENTICAL to the reference formula evaluated on the
 *             stored row values (fp32 / bf16 store: rounded once at append; binary64 store: the
 *             original values) and the given query values
 *  out_count  [nq] number of valid entries (rows may be fewer than k: no padding, :370)
 *  out_mem    where the three outputs live
 *
 * How: a fast scan (the tcgen05/TMA tensor-core kernel; the CUDA-core kernel only for shapes it
 * does not fit) streams the store once and keeps, per query, EVERY row whose approximate fp32 score
 * lies within the scan's error band of the k-th best (the complete near-tie band); an exact binary64
 * pass rescores the best candidates in the reference's summation order, sorts them and CERTIFIES
 * that no other row can reach the k-th score; when more near-ties exist than it rescored at first
 * (near-duplicate chunks) it rescores the whole band in the same launch.  Only thousands of
 * near-ties per query fall back to a second scan that collects the band, or a binary64 scan of all
 * rows.  Results are therefore exact, not approximate; vm_store_read_counters reports how each
 * query was settled. */
int vm_topk(vm_store *s, const void *queries, int q_dtype, int q_mem, int nq, int k, double min_score,
            int score_mode, int sum_mode, int flags, int64_t *out_idx, double *out_score, int32_t *out_count,
            int out_mem, vm_topk_stats *stats, void *stream);

/* Row-sharded variant: every rank holds one shard whose first row has global index
 * row_offset.  Local scan + exact rescoring, then ONE ncclAllGather of the per-rank
 * (score, global row)[nq][k] lists over NVLink and a device-side merge (ties -> lowest global
 * row); every rank receives identical outputs (global row indices). */
int vm_topk_sharded(vm_store *s, vm_comm *comm, int64_t row_offset, const void *queries, int q_dtype, int q_mem,
                    int nq, int k, double min_score, int score_mode, int sum_mode, int flags, int64_t *out_idx,
                    double *out_score, int32_t *out_count, int out_mem, vm_topk_stats *stats, void *stream);

/* The device-side merge alone (exposed for tests and for callers that gather themselves):
 * lists [nlists][nq][k] (idx, score, count per list) -> best k per query. */
int vm_merge_topk_lists(int device, const int64_t *idx_dev, const double *score_dev, const int32_t *count_dev,
                        int nlists, int nq, int k, int64_t *out_idx_dev, double *out_score_dev,
                        int32_t *out_count_dev, void *stream);

/* The same merge over the PACKED exchange layout vm_topk_sharded all-gathers: `nlists` consecutive blocks of
 * vm_topk_packed_bytes(nq, k) bytes, each [idx nq*k int64 | score nq*k double | count nq int32, padded to 8 bytes]
 * (one block per rank, global row indices).  For callers that move the blocks with their own transport, and for
 * checking the exchange format on a single GPU. */
size_t vm_topk_packed_bytes(int nq, int k);
int vm_merge_topk_packed(int device, const void *packed_dev, int nlists, int nq, int k, int64_t *out_idx_dev,
                         double *out_score_dev, int32_t *out_count_dev, void *stream);

/* Cross-query merge of _parallel_chunk_extraction_with_similarity
 * (src/components/pre_llm_injector.py:235-249): max score per row id over all queries' lists
 * (strict `>` replace), stable sort descending (first-seen order on ties), first k2.
 * Device buffers in, device buffers out; out_count is a single int32. */
int vm_merge_max_by_id(int device, const int64_t *idx_dev, const double *score_dev, const int32_t *count_dev,
                       int nq, int k, int k2, int64_t *out_idx_dev, double *out_score_dev,
                       int32_t *out_count_dev, void *stream);

/* ---- scalar cosine seams ---------------------------------------------------------------
 * n independent pairs a[i], b[i] of length dim (row-major [n][dim], VM_F32/VM_F64, host or
 * device) -> out[i] binary64, bit-identical to PreLLMInjector._cosine_similarity
 * (pre_llm_injector.py:374-388) / HybridRetriever._cosine_similarity
 * (retriever_hybrid.py:655-664; used by _post_compress_chunks :492-504).
 * zero_rule 0: norm1 == 0 or norm2 == 0 -> 0.0 ; zero_rule 1: mag1 * mag2 == 0 -> 0.0 ;
 * zero_rule 2: EmbeddingUtils.cosine_similarity (src/utils/embedding_utils.py:29-39): zero test as
 * rule 0, magnitudes through `** 0.5` (pow instead of sqrt: agrees with CPython's libm pow to a
 * few ulp, not bit-pinned -- the only entry point of this header whose scores carry a tolerance). */
int vm_cosine_pairs(int device, const void *a, const void *b, int dtype, int mem, int64_t n, int dim, int zero_rule,
                    int sum_mode, double *out, int out_mem, void *stream);

/* ---- all-pairs threshold scorer (entity / relation dedup) ------------------------------
 * Replaces Graph._are_same_context (src/pipeline/prune.py:67-79): S = cosine_similarity(E);
 * fill_diagonal(S, 0); S > threshold -- generalised from `any()` to the pair set.
 * x_dev [n][ld] bf16 or fp32 device rows (ld = vm_ld(dim)); emits every (i, j, S_ij) with
 * i < j and S_ij > threshold (strict) into out_* (device, capacity cap, unordered);
 * *out_count_dev (int64, device) receives the TOTAL number of hits, which may exceed cap, in
 * which case the call reports VM_ERR_OVERFLOW on sync paths and only the first cap hits are
 * written.  part/nparts split the upper-triangular tile grid across ranks (0/1 = all).
 * Scores are fp32 (bf16 x bf16 products accumulated in fp32 on the tensor cores), rows
 * normalised by cached fp32 inverse norms; pairs whose fp32 score lies within the kernel's own
 * error bound of the threshold ((dim + 32) * 2^-23 for bf16 rows, + 2^-8 for tf32-truncated fp32
 * rows; not a parameter) are re-decided in binary64, so the pair SET is exact for the stored
 * values.  Re-entrant: scratch is kept per (device, stream). */
int vm_pairs_above(int device, const void *x_dev, int dtype, int64_t n, int dim, float threshold, int64_t cap,
                   int64_t *out_i_dev, int64_t *out_j_dev, float *out_score_dev, int64_t *out_count_dev, int part,
                   int nparts, int flags, void *stream);

/* Multi-GPU form of vm_pairs_above (SURVEY.md 8e row 2), collective over `comm` (every rank calls it with the
 * same n / dim / threshold / cap on its own stream):
 *   1. the operand x_dev [n][ld] is replicated with ONE ncclBroadcast from rank `root` (root = -1: every
 *      rank already holds the rows);
 *   2. the upper-triangular tile grid is dealt cyclically to the ranks (part = rank of vm_pairs_above);
 *   3. one ncclAllGather of the per-rank hit counts and one ncclAllGather of the hit lists, concatenated in
 *      rank order on the device -- every rank ends with the same, complete (i, j, score) list in out_* and the
 *      total in *out_count_dev.  Nothing but the 8-byte counts passes through the host; with VM_FLAG_ASYNC not
 *      even those (the lists are then gathered at full capacity `cap` per rank).
 * More than `cap` pairs (in total, or on one rank) -> VM_ERR_OVERFLOW with the total in *out_count_dev. */
int vm_pairs_above_sharded(vm_comm *comm, void *x_dev, int dtype, int64_t n, int dim, float threshold, int64_t cap,
                           int64_t *out_i_dev, int64_t *out_j_dev, float *out_score_dev, int64_t *out_count_dev,
                           int root, int flags, void *stream);

/* ---- multi-GPU plumbing -----------------------------------------------------------------
 * One process per GPU; the 128-byte NCCL unique id is created on rank 0 and shipped to the
 * other ranks by the host (torch.distributed / any out-of-band channel). */
int vm_comm_unique_id(void *out128);
int vm_comm_init_rank(vm_comm **out, int device, int nranks, int rank, const void *id128);
int vm_comm_destroy(vm_comm *c);
/* Optional peer-memory exchange (NVLink loads instead of the NCCL all-gather): bufs[r] is rank r's
 * exchange buffer as mapped into THIS process (e.g. torch symmetric memory `buffer_ptrs`), each
 * vm_comm_exchange_bytes() long and zero-filled before first use on every rank.  Once attached,
 * vm_topk_sharded writes each batch's exact local lists into its own buffer, publishes a generation
 * flag with system scope, and ONE kernel per batch waits for every peer's flag, pulls the peers' lists
 * over NVLink and merges them (ties -> lowest global row).  Every rank must make the same sequence of
 * vm_topk_sharded calls. */
size_t vm_comm_exchange_bytes(void);
int vm_comm_attach_peer_buffers(vm_comm *c, void *const *bufs, int nranks);
int vm_comm_nranks(const vm_comm *c);
int vm_comm_rank(const vm_comm *c);

/* ---- synthetic data (bench / tests) ------------------------------------------------------
 * Fills rows [row0, row0+n) of a device buffer ([n][ld]) with the counter-based generator of
 * SURVEY.md 8d (same definition as oracle/synth.py). */
int vm_synth_fill(int device, void *rows_dev, int dtype, uint64_t seed, int64_t row0, int64_t n, int dim,
                  uint64_t dup_period, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* VIDMEM_H_ */
