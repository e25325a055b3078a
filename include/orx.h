/* orx -- B200-native exact cosine top-k retrieval engine: the C-ABI boundary.
 *
 * The reference (Molyleaf/Outline-RAG) has no FFI; its seam for this path is the
 * LangChain VectorStore object bound to `rag.vector_store`
 * (reference app/rag.py:28, created at app/rag.py:69-79).  Every entry point below
 * names the reference call it stands in for; INTEGRATION.md shows the ctypes
 * binding and the drop-in class that replaces `AsyncPGVectorStore` at rag.py:69.
 *
 * Conventions: return 0 = OK, negative = error (message via orx_last_error(),
 * thread-local).  The caller owns every buffer it passes; the library owns all
 * device memory.  Pointer arguments documented "host or device" are classified
 * with cudaPointerGetAttributes.  An orx_index lives on ONE GPU (orx_create) or is
 * a row-sharded table over several GPUs driven by one process (orx_create_multi);
 * both kinds answer the same calls.  One process PER GPU (torchrun ranks,
 * outline_rag_b200/sharded.py) uses orx_shard_* / orx_search_sharded instead.
 * Calls on one index are serialised internally (stream order = call order, so a
 * search issued after an upsert sees it: at least as consistent as the
 * reference's separate delete / insert transactions, app/rag.py:231-235).
 */
#ifndef ORX_H
#define ORX_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ORX_DIM 1024            /* VECTOR_DIM, reference app/config.py:8 */
#define ORX_MAX_K 128           /* TOP_K is 12 (reference app/config.py:253); up to 128 for a wider
                                   reranker feed (SURVEY.md 8f-4).  Batches with k <= 64 run the tcgen05 scan
                                   (64-key candidate lists up to k = 16, 160-key lists beyond); k > 64 runs
                                   one GEMV scan per query (over the bf16 image of a large fp32 table, see
                                   ORX_OPT_IMAGE_MIN_ROWS). */

#define ORX_DTYPE_F32 0         /* rows stored verbatim (fp32) + per-row 1/norm;
                                   + a bf16 image of the rows when the device has room
                                   (see ORX_OPT_IMAGE_MIN_ROWS)                    */
#define ORX_DTYPE_BF16 1        /* rows stored as RNE-bf16 of the normalised row  */

#define ORX_OK 0
#define ORX_ERR_INVALID (-1)    /* bad argument (k, nq, null pointer, ...)        */
#define ORX_ERR_DIM (-2)        /* "expected 1024 dimensions" (pgvector CheckDim) */
#define ORX_ERR_NONFINITE (-3)  /* "NaN/infinite value not allowed in vector"     */
#define ORX_ERR_CUDA (-4)       /* CUDA runtime error / out of device memory      */
#define ORX_ERR_CAPACITY (-5)   /* table cannot grow further                      */

typedef struct orx_index orx_index;

/* 128-bit chunk id = `langchain_id UUID` (reference app/database.py:119).
 * Ordered as the big-endian integer (hi, lo): the order Postgres gives uuid and
 * the tie-break of this build's ordering contract (distance ASC, id ASC). */
typedef struct orx_id { uint64_t hi, lo; } orx_id;

/* Counters for bench.py / tests (cumulative since create unless noted). */
typedef struct orx_stats {
    uint64_t kernel_launches;     /* kernels this library launched                */
    uint64_t searches;            /* orx_search* calls                             */
    uint64_t queries;             /* queries answered                              */
    uint64_t fallback_gemv;       /* queries re-run on the fp32 scan (coarse pass unproven) */
    uint64_t fallback_exhaustive; /* queries answered by the threshold-collect pass */
    uint64_t rows_moved;          /* rows relocated by delete compaction           */
    float    last_scan_ms;        /* device time of the last search's scan kernel(s) */
    float    last_search_ms;      /* host wall time of the last orx_search call     */
    int      last_path;           /* 0 none, 1 gemv scan, 2 tcgen05 scan,
                                     3 gemv scan over the bf16 image of an fp32 table,
                                     4 gemv scan over the 8-bit image of an fp32 table */
    int      reserved;
    uint64_t scan_launches;       /* scan kernel launches (gemv or tcgen05)        */
    double   scan_ms_total;       /* sum of their device times (CUDA events around each launch) */
} orx_stats;

/* Replaces `AsyncPGVectorStore.create(engine, embedding_service,
 * table_name="langchain_pg_embedding", ...)` (reference app/rag.py:69-79) and the
 * DDL `embedding vector(1024)` (app/database.py:118-131).  dim must be ORX_DIM. */
int orx_create(orx_index **out, int dim, int dtype, uint64_t capacity_rows, int device);
void orx_destroy(orx_index *idx);

/* The same table ROW-SHARDED over the GPUs `devices[0..n_devices)` of one NVSwitch box, owned by ONE process -- what
 * a uvicorn worker of the reference (app/entrypoint.sh:16, one `rag.vector_store` per process, app/rag.py:28) needs
 * to put a table larger than one GPU, or the bandwidth of eight, behind the same object (SURVEY.md 8b / 8e).
 * Rows are placed by mix64(id) mod n_devices.  Every call of this header works on the returned handle: upsert /
 * delete route rows to their shards; orx_search runs all shards concurrently (one launcher thread per GPU), every
 * GPU's finalize kernel pushes its k candidates per query into the first GPU's gather buffer with peer stores over
 * NVLink and that GPU merges them -- no collective library, no host round trip before the merged answer.  capacity_rows
 * is the total.  A device may be listed more than once (several shards on one GPU: tests).  Device-resident query
 * or output buffers must live on devices[0].  Not available on a multi-GPU handle: orx_set_stream, orx_filter_*
 * handles (orx_search_filtered works), orx_shard_*. */
int orx_create_multi(orx_index **out, int dim, int dtype, uint64_t capacity_rows,
                     const int *devices, int n_devices);
int orx_shard_count(const orx_index *idx);      /* 1 for orx_create, n_devices for orx_create_multi */

/* Kernels are launched on this CUDA stream (a cudaStream_t; NULL = legacy default
 * stream).  Python hands over torch's current stream so torch.cuda.Event sees them. */
int orx_set_stream(orx_index *idx, void *cuda_stream);

/* Options.  ORX_OPT_SCAN_TIMING (default 1): record a CUDA event pair around every scan launch so that orx_get_stats
 * can report the scan kernel's own device time (bench.py's roofline); 0 saves the two event records per search.
 * ORX_OPT_IMAGE_MIN_ROWS (default 1048576 = 2^20): live rows from which an fp32 table's GEMV scans (one query, batches
 * with k > 64, filtered bitmap scans) read the table's bf16 IMAGE instead of its fp32 rows.  The image holds RNE-bf16 of
 * every stored element (not normalised: 2 bytes per element, +50 % device memory, e.g. +20.5 GB at 10M rows) and is kept
 * in step by upsert, delete, import and growth.  It is allocated only for a capacity of at least this many rows -- when
 * the table is created or grows, or by the first search that would read it (after the option was lowered) -- so small
 * tables pay nothing for it; an fp32 table for which the device has no room simply has none (scans read the fp32 rows).
 * The image takes device memory other allocations (search scratch, the caller's tensors) might want; only growth of
 * the table itself takes it back.  The re-scan of queries the tcgen05 batch pass could not prove always reads the fp32
 * rows.  The image scan halves
 * the bytes a query streams; its candidates are still rescored canonically from the fp32 rows and the completeness proof
 * uses the image's error bound, so the answers are the same ids and distance bits (last_path reports 3).  0 = always
 * (when an image exists), a negative value = never.  bf16 tables have no image.  A multi-GPU handle sets every shard. */
/* ORX_OPT_IMAGE8_MIN_ROWS (default 4194304 = 2^22): capacities from which an fp32 table's image is an 8-bit one INSTEAD of
 * the bf16 one (a table holds at most one image; the kind is chosen when the image is allocated -- create, growth or the
 * first search that needs it -- and growth past this capacity replaces a bf16 image by an 8-bit one).  Each row is kept
 * as 1024 int8 X_i = rint(x_i / d), d = max|x_i| / 127, plus one fp32 d / |x|: 1 byte per element + 4 per row (10.3 GB
 * at 10M rows instead of 20.5 GB for the bf16 image).  The single-query and filtered bitmap scans with k <= 12 read it
 * (last_path 4) once ORX_OPT_IMAGE_MIN_ROWS live rows are reached, scoring each row by an exact integer dot with a
 * 15-bit quantisation of the query: a quarter of the fp32 rows' bytes.  The candidates are rescored canonically from
 * the fp32 rows, so ids and distance bits are those of the fp32 scan.  A row whose quantisation residual exceeds 2^-6
 * of its norm is always a candidate; a table with more than 16 such rows, batches of GEMV queries (k > 64) and k > 12
 * read the fp32 rows (last_path 1).  0 = every fp32 table that gets an image, a negative value = never. */
#define ORX_OPT_SCAN_TIMING 1
#define ORX_OPT_IMAGE_MIN_ROWS 2
#define ORX_OPT_IMAGE8_MIN_ROWS 3
int orx_set_option(orx_index *idx, int option, int value);

uint64_t orx_size(const orx_index *idx);       /* live rows */
uint64_t orx_capacity(const orx_index *idx);
int orx_dtype(const orx_index *idx);
/* Changes with every successful write (upsert, delete, import).  A snapshot taken in several orx_export_rows calls is
 * consistent iff this value is the same before the first and after the last call (Index.save checks it). */
uint64_t orx_mutation_count(const orx_index *idx);
int orx_get_stats(const orx_index *idx, orx_stats *out);

/* Replaces `vector_store.aadd_documents(chunks)` -> per-row
 * `INSERT ... ON CONFLICT (langchain_id) DO UPDATE` (reference app/rag.py:235).
 * ids [n]; vecs [n, dim] fp32, host or device.  An id already present is replaced
 * in place; an id repeated inside the batch keeps its last occurrence.  The whole
 * batch is rejected (table unchanged) on a NaN/Inf element (ORX_ERR_NONFINITE). */
int orx_upsert(orx_index *idx, const orx_id *ids, const float *vecs, uint64_t n, int dim);

/* Replaces `vector_store.adelete(ids=[...])` -> `DELETE ... WHERE langchain_id IN (...)`
 * (reference app/rag.py:231, :371).  Unknown ids are ignored, like the SQL. */
int orx_delete(orx_index *idx, const orx_id *ids, uint64_t n, uint64_t *n_removed);

/* 1 if the id is live, 0 if not. */
int orx_contains(const orx_index *idx, orx_id id);

/* Replaces the SQL of `asimilarity_search_with_score_by_vector(embedding, k)`:
 *   SELECT ..., cosine_distance("embedding", :q) AS distance
 *   FROM langchain_pg_embedding ORDER BY "embedding" <=> :q LIMIT :k
 * (langchain-postgres 0.0.16 [UPSTREAM]; reached from reference app/rag.py:85-87,
 * called at app/blueprints/api.py:122) with EXACT sequential-scan semantics.
 * queries [nq, dim] fp32, host or device.  Outputs (host or device, same kind for
 * all three): out_ids [nq, k], out_dist [nq, k] = cosine distance as float8,
 * out_counts [nq] = min(k, live rows).  Order: distance ASC, NaN last, id ASC.
 * Unused tail slots are filled with id (0,0) / NaN. */
int orx_search(orx_index *idx, const float *queries, int nq, int dim, int k,
               orx_id *out_ids, double *out_dist, int *out_counts);

/* The same search in two halves, so that a caller can keep TWO searches in flight per index (the host side of the next
 * query -- staging, launches -- and its first kernels overlap the tail of the previous one: finalize, exchange, merge,
 * the completion hand-shake).  orx_search_submit launches the whole chain and returns at once with a ticket;
 * orx_search_wait(ticket) blocks until that search is complete, settles whatever the fast path could not prove, and
 * fills the output buffers given at submit (they and, for host queries, nothing else must stay valid until then;
 * the queries are copied at submit).  At most two tickets may be outstanding; wait for them in submission order.
 * orx_search == submit + wait.  orx_search_sharded_submit is the same for the collective row-sharded search (every
 * rank submits and waits in the same order; its tickets are waited for with orx_search_wait too). */
int orx_search_submit(orx_index *idx, const float *queries, int nq, int dim, int k,
                      orx_id *out_ids, double *out_dist, int *out_counts, int *ticket);
int orx_search_wait(orx_index *idx, int ticket);
int orx_search_sharded_submit(orx_index *idx, const float *queries, int nq, int dim, int k,
                              orx_id *out_ids, double *out_dist, int *out_counts, int *ticket);

/* The same query restricted to a set of chunk ids -- the SQL with a WHERE clause, i.e. what the
 * upstream store's `filter=` argument compiles to after the metadata predicate has been resolved to
 * `langchain_id`s (e.g. `source_id = ANY(...)`, reference app/rag.py:216-224 shows that look-up).
 * allow_ids [n_allow] host; unknown ids are ignored, duplicates count once.  Up to 4095 eligible rows
 * are each rescored canonically (no scan; O(n_allow) row reads per query).  From 4096 eligible rows on
 * the predicate becomes a row bitmap and the sequential scan skips the rows whose bit is clear (HBM
 * traffic = eligible rows only), with the same candidate proof as orx_search; an unproven query falls
 * back to the rescoring path.  A BATCH with nq x eligible rows >= rows runs ONE tcgen05 pass over the
 * table instead of nq bitmap scans: the predicate is folded into the per-row scale the epilogue
 * multiplies with (an excluded row can never be a candidate).  Exact either way.  Same outputs and
 * ordering as orx_search. */
int orx_search_filtered(orx_index *idx, const float *queries, int nq, int dim, int k,
                        const orx_id *allow_ids, uint64_t n_allow,
                        orx_id *out_ids, double *out_dist, int *out_counts);

/* A reusable predicate: resolving every allowed id to its row costs one hash look-up per id, which for
 * large allow-lists is far more than the scan itself (measured: 115 ms vs 1.2 ms for 2M ids).  A filter
 * keeps the resolved rows (list + bitmap) on the device between searches; it is re-resolved
 * automatically when the id -> row map has changed (upsert of new ids, delete, import), so it always
 * denotes "the live rows whose id is in the set".  orx_search_with_filter == orx_search_filtered with the
 * ids the filter was created from.  Destroy filters before their index. */
typedef struct orx_filter orx_filter;
int orx_filter_create(orx_index *idx, const orx_id *allow_ids, uint64_t n_allow, orx_filter **out);
void orx_filter_destroy(orx_filter *flt);
int orx_search_with_filter(orx_index *idx, orx_filter *flt, const float *queries, int nq, int dim, int k,
                           orx_id *out_ids, double *out_dist, int *out_counts);

/* Maximal marginal relevance over the exact candidates -- what langchain's `VectorStoreRetriever(search_type="mmr")`
 * gets from `max_marginal_relevance_search(query, k, fetch_k, lambda_mult)`, which langchain-postgres answers by
 * fetching fetch_k rows with their embeddings and running `maximal_marginal_relevance` on the host.  Here both halves
 * stay on the GPU and the result is defined bit for bit (DESIGN.md section 2, "MMR"):
 *   candidates  C = the exact top-fetch_k of orx_search / orx_search_filtered / orx_search_with_filter, in contract
 *               order; position p in C is the tie-break below;
 *   s_q[p]      = 1 - distance[p] (binary64);
 *   s_dd(p, r)  = clamp(canonical dot / sqrt(n2_p * n2_r), -1, 1) of the rows AS STORED (the halving tree of the
 *               canonical distance, IEEE div / sqrt / mul);
 *   greedy      first pick = position 0; then argmax of lambda*s_q[p] - (1-lambda)*max over picked r of s_dd(p, r),
 *               evaluated without contraction; ties -> lowest position; NaN scores (zero-norm rows, zero query) only
 *               once no finite score is left, in position order.
 * Outputs as orx_search (host buffers only): out_ids [nq, k] and out_dist [nq, k] in SELECTION order, each with the
 * canonical query distance orx_search reports for that row; out_counts [nq] = min(k, candidates); unused slots (0,0) /
 * NaN.  1 <= k <= fetch_k <= ORX_MAX_K and 0 <= lambda_mult <= 1 (lambda 0 = pure diversity), else ORX_ERR_INVALID.
 * The candidate search and the gather of their rows run under the index lock: no write lands in between.  Queries are
 * processed in chunks of 256 (candidate matrix <= 256 x 128 x 4 KB = 128 MB of device scratch).  Rejected while
 * orx_search_submit tickets are in flight (ORX_ERR_INVALID).  A multi-GPU handle gathers each shard's candidates on its own GPU and runs
 * the selection on devices[0]; orx_search_mmr_with_filter is per GPU.  Not available: the row-sharded
 * one-process-per-GPU search (orx_search_sharded), asynchronous submit / wait, device-resident buffers. */
int orx_search_mmr(orx_index *idx, const float *queries, int nq, int dim, int k, int fetch_k, double lambda_mult,
                   orx_id *out_ids, double *out_dist, int *out_counts);
int orx_search_mmr_filtered(orx_index *idx, const float *queries, int nq, int dim, int k, int fetch_k,
                            double lambda_mult, const orx_id *allow_ids, uint64_t n_allow,
                            orx_id *out_ids, double *out_dist, int *out_counts);
int orx_search_mmr_with_filter(orx_index *idx, orx_filter *flt, const float *queries, int nq, int dim, int k,
                               int fetch_k, double lambda_mult, orx_id *out_ids, double *out_dist, int *out_counts);

/* Merge `n_lists` per-shard results (each [nq, k] as written by orx_search, all on
 * this index's device or all on the host) into the global top-k with the same
 * ordering.  The on-device step after the NCCL allgather of the row-sharded path. */
int orx_merge_topk(orx_index *idx, int n_lists, int nq, int k,
                   const orx_id *ids, const double *dist, const int *counts,
                   orx_id *out_ids, double *out_dist, int *out_counts);

/* Same merge, reading the lists where an allgather left them: every rank contributes ONE block
 * holding its ids, distances and counts, rank l's block starts l*list_stride_bytes after rank 0's.
 * ids0 / dist0 / counts0 point at rank 0's arrays inside the gathered buffer.  Device pointers
 * only; asynchronous on the index's stream (outline_rag_b200/sharded.py). */
int orx_merge_topk_strided(orx_index *idx, int n_lists, int nq, int k,
                           const orx_id *ids0, const double *dist0, const int *counts0,
                           uint64_t list_stride_bytes,
                           orx_id *out_ids, double *out_dist, int *out_counts);

/* ---- row-sharded search over NVLink peer memory (one process per GPU; SURVEY.md 8e) ----------
 * Setup, once: every rank calls orx_shard_export (allocates its gather buffer, returns a CUDA IPC
 * handle of ORX_IPC_HANDLE_BYTES bytes), the handles are exchanged out of band (torch.distributed
 * all_gather in outline_rag_b200/sharded.py), then every rank calls orx_shard_connect with all
 * `world` handles in rank order.
 * orx_search_sharded is COLLECTIVE: every rank calls it with the same queries, nq and k.  Each GPU
 * scans its shard, pushes its k candidates per query into every peer's gather buffer with P2P
 * stores, and merges what arrives; every rank receives the global top-k (same layout and ordering
 * as orx_search).  Replaces the same SQL as orx_search, for a table partitioned by row. */
#define ORX_IPC_HANDLE_BYTES 64
int orx_shard_export(orx_index *idx, int world, int rank, void *handle_out);
int orx_shard_connect(orx_index *idx, const void *handles, int n_handles);
int orx_search_sharded(orx_index *idx, const float *queries, int nq, int dim, int k,
                       orx_id *out_ids, double *out_dist, int *out_counts);

/* Diagnostic for the exactness argument (DESIGN.md section 2): the COARSE scores of the tcgen05 batch scan -- the
 * tf32 (fp32 table) or bf16 (bf16 table) tensor-core dot of every live row with every normalised query, times the
 * row's 1/|x| -- computed by the same TMA / tcgen05.mma / TMEM pipeline as orx_search (only the epilogue writes
 * instead of selecting; use_pairs picks the cta_group::2 kernel).  out_device [live rows, nq] fp32 in table row order
 * (row order = orx_export_rows).  A test measures max |coarse - cosine| with it and checks it against the epsilon
 * the completeness proof assumes.  1 <= nq <= 2048. */
int orx_debug_coarse_scores(orx_index *idx, const float *queries, int nq, int use_pairs, float *out_device);

/* Diagnostic for the same argument, GEMV side: the FAST scores of the GEMV scans (orx_search of one query, batches the
 * tensor pass does not take, filtered bitmap scans) -- the fp32 FMA-chain dot of every live row with every normalised
 * query, times the row's 1/|x|, exactly the value the scans key their candidates on (same load / FMA / shuffle
 * sequence).  Irregular rows (norm outside [2^-40, 2^40]) come out +-inf or NaN, zero-norm rows NaN.  out_device
 * [live rows, nq] fp32 in table row order.  1 <= nq <= 65535. */
int orx_debug_fast_scores(orx_index *idx, const float *queries, int nq, float *out_device);

/* The same diagnostic for the scans over the bf16 image of an fp32 table (ORX_OPT_IMAGE_MIN_ROWS): the fp32 FMA-chain dot
 * of every live row's IMAGE with every normalised query, times the fp32 row's 1/|x| -- the value the image scans key
 * their candidates on.  ORX_ERR_INVALID when the index has no image (bf16 table, or no device memory for it).
 * out_device [live rows, nq] fp32 in table row order.  1 <= nq <= 65535. */
int orx_debug_image_scores(orx_index *idx, const float *queries, int nq, float *out_device);

/* The same for the 8-bit image (ORX_OPT_IMAGE8_MIN_ROWS): (float(D) * dq) * scale8 of every live row, D the exact integer
 * dot of the row's int8 image with the query's 15-bit quantisation -- the value the 8-bit scans key their candidates on.
 * ORX_ERR_INVALID when the index has no 8-bit image (bf16 table, a bf16 image, or no device memory for it). */
int orx_debug_image8_scores(orx_index *idx, const float *queries, int nq, float *out_device);

/* Read back stored rows (as fp32) by id -- snapshot / debugging / tests.
 * out_vecs [n, dim] host; out_found [n] host (1/0). */
int orx_fetch(orx_index *idx, const orx_id *ids, uint64_t n, float *out_vecs, int *out_found);

/* Snapshot / cold start (SURVEY.md 8f-2; the device table is a cache of
 * `langchain_pg_embedding.embedding`, reference app/database.py:118-131).
 * orx_export_rows copies live rows [row_start, row_start+n) VERBATIM in the table dtype (fp32: 4096 B,
 * bf16: 2048 B per row) with their ids to host buffers; orx_import_rows appends such rows (ids must be
 * new) without re-normalising, so a bf16 table round-trips bit for bit.  rows_raw may be host or device. */
int orx_export_rows(orx_index *idx, uint64_t row_start, uint64_t n, orx_id *ids_out, void *rows_out);
int orx_import_rows(orx_index *idx, const orx_id *ids, const void *rows_raw, uint64_t n);

/* ---- pgvector wire formats on either side of the path (SURVEY.md 8f-1, 8a3) ------------------
 * Cold start: the device table is rebuilt from
 *   COPY (SELECT langchain_id, embedding FROM langchain_pg_embedding) TO STDOUT (FORMAT binary)
 * (table: reference app/database.py:118-131; the reference's driver, psycopg 3 -- requirements.txt:5 --
 * yields that stream chunk by chunk from `cursor.copy(...)`).  orx_pgcopy_feed accepts the stream in
 * chunks of ANY size; complete tuples are staged in pinned memory, decoded on the GPU (big-endian float4
 * image of pgvector's vector_send [UPSTREAM src/vector.c]) and upserted 16384 rows at a time.  Checks
 * and messages follow Postgres' CopyFrom and pgvector's vector_recv: signature / flags, 2 columns,
 * 16-byte uuid, dim == 1024 (ORX_ERR_DIM), unused == 0, NaN / infinite element (ORX_ERR_NONFINITE; the
 * batch holding it is rejected).  Rows whose embedding is NULL (the column is nullable) are skipped and
 * counted.  An id seen before -- in the table or earlier in the stream -- is replaced (upsert).
 * A full batch is copied, decoded and committed by a helper thread of the loader while the caller feeds
 * the next one (two staging buffer sets, the loader's own stream), so the error of a batch is reported by
 * the NEXT feed or by orx_pgcopy_close.  After an error every later feed fails; batches flushed before it
 * stay loaded.  orx_pgcopy_close flushes the tail, waits for the batch in flight, reports the totals and
 * frees the loader, also after an error (its return code repeats it).  Several loaders may feed one index
 * concurrently (one thread each); a loader must be closed before its index is destroyed.
 * idx == NULL opens a DRY RUN: framing and element checks on the host, nothing loaded, no GPU needed. */
typedef struct orx_pgcopy orx_pgcopy;
int orx_pgcopy_open(orx_index *idx, orx_pgcopy **out);
/* Row-sharded cold start (SURVEY.md 8e): every rank feeds the SAME stream to its own loader, which keeps
 * only the rows with mix64(id) mod world == rank (the shard function of outline_rag_b200/sharded.py) --
 * no data-path collective, like the sharded upsert.  rows_loaded then counts this rank's rows. */
int orx_pgcopy_open_sharded(orx_index *idx, int world, int rank, orx_pgcopy **out);
int orx_pgcopy_feed(orx_pgcopy *ld, const void *bytes, uint64_t n);
int orx_pgcopy_close(orx_pgcopy *ld, uint64_t *rows_loaded, uint64_t *rows_null);

/* pgvector's text input `vector_in` [UPSTREAM src/vector.c]: '[0.1, 0.2, ...]' -> fp32.  This is the
 * format the reference sends the query vector (:q of the SQL above) and the stored embeddings in
 * (langchain-postgres formats the Python float list with str(); pgvector parses each element with strtof,
 * i.e. ONE rounding decimal -> fp32).  text need not be NUL-terminated; out [dim]; the vector must have
 * exactly dim elements.  Host-only (no GPU).  Errors as pgvector: syntax / out of range -> ORX_ERR_INVALID,
 * dimension -> ORX_ERR_DIM, NaN / infinity -> ORX_ERR_NONFINITE. */
int orx_parse_vector_text(const char *text, uint64_t len, float *out, int dim);

const char *orx_last_error(void);
const char *orx_version(void);

#ifdef __cplusplus
}
#endif
#endif /* ORX_H */
