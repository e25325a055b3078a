// pgvector wire formats on either side of the hot path (SURVEY.md 8f-1: cold-start bulk load
// `SELECT langchain_id, embedding FROM langchain_pg_embedding`; 8a3: ":q sent as text '[f,...]'").
//
//   * orx_pgcopy_*: streaming loader for a PostgreSQL `COPY (SELECT langchain_id, embedding FROM
//     langchain_pg_embedding) TO STDOUT (FORMAT binary)` byte stream (reference table:
//     app/database.py:118-131; psycopg3 `cursor.copy()` hands the stream over in arbitrary chunks,
//     requirements.txt:5).  The host walks the framing (19-byte header, per tuple: int16 field count,
//     int32 length + 16-byte uuid, int32 length + pgvector `vector_send` image = int16 dim, int16
//     unused, dim big-endian float4 [UPSTREAM pgvector src/vector.c vector_recv]) inside a pinned
//     staging buffer; the raw bytes go to HBM as they are and decode_pgvector_kernel turns the
//     2-byte-aligned big-endian payloads into fp32 rows, which then take the normal upsert path
//     (element check, canonical norms, id map).  HBM-bound byte work: 4096 B read + 4096 B written
//     per row, one warp per row, aligned 128-byte warp loads + one PRMT per element.
//   * orx_parse_vector_text: pgvector's text input (`vector_in`), the format the reference sends
//     both the query and the stored embeddings in (langchain-postgres 0.0.16 formats the Python
//     float list with str() [UPSTREAM]); strtof in the C locale, same checks, same messages.
#include <cuda_runtime.h>

#include <algorithm>
#include <cerrno>
#include <clocale>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <locale.h>
#include <string>

#include <string>
#include <thread>

#include "internal.h"

namespace orx {

// one warp per row; off[i] = byte offset of row i's first float inside raw (any alignment).
__global__ void __launch_bounds__(256)
decode_pgvector_kernel(const uint8_t *__restrict__ raw, const uint64_t *__restrict__ off, uint32_t n,
                       float *__restrict__ out) {
    const int lane = threadIdx.x & 31;
    const uint32_t gw = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const uint32_t n_gw = gridDim.x * (blockDim.x >> 5);
    for (uint32_t i = gw; i < n; i += n_gw) {
        const uint64_t o = off[i];
        const uint32_t sh = (uint32_t)(o & 3);                       // raw is 256-byte aligned (cudaMalloc)
        const uint32_t *w = reinterpret_cast<const uint32_t *>(raw + (o - sh));
        // element bytes b[sh..sh+3] of the word pair (lo, hi), most significant first -> little-endian word
        const uint32_t sel = (sh + 3) | ((sh + 2) << 4) | ((sh + 1) << 8) | (sh << 12);
        float *dst = out + (size_t)i * ORX_DIM;
#pragma unroll 8
        for (int j = 0; j < ORX_DIM / 32; ++j) {
            const int e = lane + 32 * j;
            const uint32_t lo = w[e];
            const uint32_t hi = sh ? w[e + 1] : 0u;                  // neighbour lane's word: an L1 hit
            dst[e] = __uint_as_float(__byte_perm(lo, hi, sel));
        }
    }
}

void launch_decode_pgvector(const uint8_t *raw, const uint64_t *off, uint32_t n, float *out, cudaStream_t st) {
    if (n == 0) return;
    uint32_t blocks = (n + 7) / 8;
    blocks = cap_grid(blocks, 8);
    decode_pgvector_kernel<<<blocks, 256, 0, st>>>(raw, off, n, out);
}

}  // namespace orx

namespace {

constexpr uint32_t PG_BATCH_ROWS = 16384;                  // rows per flush: 64 MB of fp32 rows in HBM
constexpr size_t PG_TUPLE_HEAD = 2 + 4 + 16 + 4;           // field count, uuid length + uuid, vector length
constexpr size_t PG_VEC_BYTES = 4 + 4 * (size_t)ORX_DIM;   // dim, unused, floats
constexpr size_t PG_TUPLE_MAX = PG_TUPLE_HEAD + PG_VEC_BYTES;
constexpr size_t PG_RAW_CAP = (size_t)PG_BATCH_ROWS * PG_TUPLE_MAX + 4096;
const unsigned char PG_SIGNATURE[11] = {'P', 'G', 'C', 'O', 'P', 'Y', '\n', 0xFF, '\r', '\n', 0};

inline uint32_t be32(const uint8_t *p) { return ((uint32_t)p[0] << 24) | ((uint32_t)p[1] << 16) | ((uint32_t)p[2] << 8) | p[3]; }
inline uint16_t be16(const uint8_t *p) { return (uint16_t)(((uint16_t)p[0] << 8) | p[1]); }
inline uint64_t be64(const uint8_t *p) { return ((uint64_t)be32(p) << 32) | be32(p + 4); }

}  // namespace

struct orx_pgcopy {
    orx_index *ix = nullptr;          // null: dry run (framing + element check on the host, nothing loaded)
    int device = 0;                   // the index's GPU (kept here: freeing the loader must not touch the index)
    uint32_t world = 1, rank = 0;     // row-sharded load: keep only the ids this rank owns (sharded.py shard_of)
    enum State { HEADER, EXTENSION, TUPLES, DONE, FAILED } state = HEADER;
    // TWO batch buffer sets: while the GPU side of a full batch (H2D copy, decode, validate, commit, id map) runs on a
    // helper thread, the caller's thread keeps copying and parsing the stream into the other set
    struct Batch {
        uint8_t *raw = nullptr;       // staging (pinned when loading)
        orx_id *ids = nullptr;        // rows parsed inside raw[0, pos): id and payload offset
        uint64_t *offs = nullptr;
        uint8_t *d_raw = nullptr;
        uint64_t *d_offs = nullptr;
        float *d_vecs = nullptr;
    } batch[2];
    int cur = 0;
    uint8_t *raw = nullptr;           // = batch[cur].raw: the bytes not yet flushed
    size_t fill = 0, pos = 0;         // bytes held / parsed
    uint64_t skip = 0;                // header extension bytes still to drop
    orx_id *ids = nullptr;            // = batch[cur].ids / offs
    uint64_t *offs = nullptr;
    uint32_t n_batch = 0;
    cudaStream_t st = nullptr;        // the loader's own stream (copy + decode): several loaders may feed one index
    std::thread job;                  // the batch in flight on the GPU side
    bool job_running = false;
    int job_rc = ORX_OK;
    uint32_t job_rows = 0;
    std::string job_err;
    uint64_t rows = 0, nulls = 0, foreign = 0, bytes = 0;
    int err = ORX_OK;
    std::string err_text;
};

namespace {

int pg_fail(orx_pgcopy *ld, int code) {       // the caller has just recorded the message (orx::set_error)
    ld->state = orx_pgcopy::FAILED;
    ld->err = code;
    ld->err_text = orx_last_error();           // kept: the close may come from another thread (asyncio.to_thread)
    return code;
}

void pg_free(orx_pgcopy *ld) {
    if (ld->job.joinable()) ld->job.join();
    if (ld->ix) {
        int prev = -1;
        cudaGetDevice(&prev);
        cudaSetDevice(ld->device);
        for (orx_pgcopy::Batch &b : ld->batch) {
            if (b.raw) cudaFreeHost(b.raw);
            if (b.ids) cudaFreeHost(b.ids);
            if (b.offs) cudaFreeHost(b.offs);
            if (b.d_raw) cudaFree(b.d_raw);
            if (b.d_offs) cudaFree(b.d_offs);
            if (b.d_vecs) cudaFree(b.d_vecs);
        }
        if (ld->st) cudaStreamDestroy(ld->st);
        cudaGetLastError();
        if (prev >= 0) cudaSetDevice(prev);
    } else {
        free(ld->batch[0].raw);
        free(ld->batch[0].ids);
        free(ld->batch[0].offs);
    }
    delete ld;
}

// vector_recv's element check on the host (dry run only; the loading path checks on the GPU)
int pg_check_elements_host(orx_pgcopy *ld, const uint8_t *payload) {
    for (int e = 0; e < ORX_DIM; ++e) {
        const uint32_t u = be32(payload + 4 * (size_t)e);
        if ((u & 0x7F800000u) == 0x7F800000u) {
            orx::set_error(ORX_ERR_NONFINITE, "%s not allowed in vector (COPY row %llu)",
                           (u & 0x007FFFFFu) ? "NaN" : "infinite value", (unsigned long long)(ld->rows + ld->nulls + ld->n_batch));
            return pg_fail(ld, ORX_ERR_NONFINITE);
        }
    }
    return ORX_OK;
}

// the GPU side of one full batch (runs on the helper thread): raw bytes -> HBM, decode, upsert
void pg_job(orx_pgcopy *ld, orx_pgcopy::Batch *b, uint32_t n, size_t bytes) {
    cudaSetDevice(ld->device);
    cudaStream_t st = ld->st;
    cudaError_t e = cudaMemcpyAsync(b->d_raw, b->raw, bytes, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(b->d_offs, b->offs, n * sizeof(uint64_t), cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) {
        orx::launch_decode_pgvector(b->d_raw, b->d_offs, n, b->d_vecs, st);
        orx::index_count_launches(ld->ix, 1);
        e = cudaGetLastError();
    }
    // the rows are decoded on the loader's stream and committed on the index's: only this helper thread waits in between
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) {
        ld->job_rc = ORX_ERR_CUDA;
        ld->job_err = std::string("COPY decode failed: ") + cudaGetErrorString(e);
        return;
    }
    const int rc = orx_upsert(ld->ix, b->ids, b->d_vecs, n, ORX_DIM);
    ld->job_rc = rc;
    if (rc != ORX_OK) ld->job_err = orx_last_error();
}

// wait for the batch in flight (if any) and account for it
int pg_join(orx_pgcopy *ld) {
    if (!ld->job_running) return ORX_OK;
    ld->job.join();
    ld->job_running = false;
    if (ld->job_rc != ORX_OK) {
        orx::set_error(ld->job_rc, "%s", ld->job_err.c_str());
        return pg_fail(ld, ld->job_rc);
    }
    ld->rows += ld->job_rows;
    return ORX_OK;
}

// hand the rows parsed so far to the table; afterwards raw[0, pos) is dead.  The batch is loaded by the helper thread
// while the caller goes on parsing into the other buffer set; its outcome is collected by the NEXT flush (or the close).
int pg_flush(orx_pgcopy *ld) {
    const uint32_t n = ld->n_batch;
    if (ld->ix) {
        int rc = pg_join(ld);                       // at most one batch in flight: the other buffer set is free now
        if (rc != ORX_OK) return rc;
        orx_pgcopy::Batch *b = &ld->batch[ld->cur];
        const size_t done = ld->pos, left = ld->fill - ld->pos;
        ld->cur ^= 1;
        orx_pgcopy::Batch *nb = &ld->batch[ld->cur];
        memcpy(nb->raw, b->raw + done, left);       // the unparsed tail moves to the other set
        ld->raw = nb->raw;
        ld->ids = nb->ids;
        ld->offs = nb->offs;
        ld->fill = left;
        ld->pos = 0;
        ld->n_batch = 0;
        if (n) {
            ld->job_rc = ORX_OK;
            ld->job_rows = n;
            ld->job_running = true;
            ld->job = std::thread(pg_job, ld, b, n, done);
        }
        return ORX_OK;
    }
    ld->rows += n;
    ld->n_batch = 0;
    memmove(ld->raw, ld->raw + ld->pos, ld->fill - ld->pos);
    ld->fill -= ld->pos;
    ld->pos = 0;
    return ORX_OK;
}

// advance over every complete item in raw[pos, fill); returns ORX_OK when more bytes are needed
int pg_parse(orx_pgcopy *ld) {
    for (;;) {
        const uint8_t *p = ld->raw + ld->pos;
        const size_t have = ld->fill - ld->pos;
        switch (ld->state) {
            case orx_pgcopy::HEADER: {
                if (have < 19) return ORX_OK;
                if (memcmp(p, PG_SIGNATURE, 11) != 0) {
                    orx::set_error(ORX_ERR_INVALID, "COPY file signature not recognized");
                    return pg_fail(ld, ORX_ERR_INVALID);
                }
                const uint32_t flags = be32(p + 11);
                if (flags & (1u << 16)) {
                    orx::set_error(ORX_ERR_INVALID, "invalid COPY file header (WITH OIDS)");
                    return pg_fail(ld, ORX_ERR_INVALID);
                }
                if (flags >> 17) {
                    orx::set_error(ORX_ERR_INVALID, "unrecognized critical flags in COPY file header");
                    return pg_fail(ld, ORX_ERR_INVALID);
                }
                ld->skip = be32(p + 15);
                if ((int32_t)ld->skip < 0) {
                    orx::set_error(ORX_ERR_INVALID, "invalid COPY file header (missing length)");
                    return pg_fail(ld, ORX_ERR_INVALID);
                }
                ld->pos += 19;
                ld->state = orx_pgcopy::EXTENSION;
                break;
            }
            case orx_pgcopy::EXTENSION: {
                const size_t drop = (size_t)std::min<uint64_t>(ld->skip, have);
                ld->pos += drop;
                ld->skip -= drop;
                if (ld->skip) return ORX_OK;
                ld->state = orx_pgcopy::TUPLES;
                break;
            }
            case orx_pgcopy::TUPLES: {
                if (ld->n_batch == PG_BATCH_ROWS) return ORX_OK;          // flush first
                if (have < 2) return ORX_OK;
                const int16_t nf = (int16_t)be16(p);
                if (nf == -1) {
                    ld->pos += 2;
                    ld->state = orx_pgcopy::DONE;
                    break;
                }
                if (nf != 2) {
                    orx::set_error(ORX_ERR_INVALID, "COPY row has %d columns, expected 2 (langchain_id, embedding)", (int)nf);
                    return pg_fail(ld, ORX_ERR_INVALID);
                }
                if (have < 6) return ORX_OK;
                const int32_t l1 = (int32_t)be32(p + 2);
                if (l1 != 16) {
                    orx::set_error(ORX_ERR_INVALID, l1 < 0 ? "null value in column \"langchain_id\""
                                                           : "incorrect binary data format: uuid of %d bytes", l1);
                    return pg_fail(ld, ORX_ERR_INVALID);
                }
                if (have < PG_TUPLE_HEAD) return ORX_OK;
                const int32_t l2 = (int32_t)be32(p + 22);
                if (l2 == -1) {                                           // `embedding` is nullable (database.py:121)
                    ld->nulls += 1;
                    ld->pos += PG_TUPLE_HEAD;
                    break;
                }
                if (l2 < 4) {
                    orx::set_error(ORX_ERR_INVALID, "incorrect binary data format: vector of %d bytes", l2);
                    return pg_fail(ld, ORX_ERR_INVALID);
                }
                if (have < PG_TUPLE_HEAD + 4) return ORX_OK;
                const int dim = (int16_t)be16(p + 26), unused = (int16_t)be16(p + 28);
                if (dim != ORX_DIM) {                                     // CheckDim / CheckExpectedDim
                    orx::set_error(ORX_ERR_DIM, "expected %d dimensions, not %d", ORX_DIM, dim);
                    return pg_fail(ld, ORX_ERR_DIM);
                }
                if (unused != 0) {
                    orx::set_error(ORX_ERR_INVALID, "expected unused to be 0, not %d", unused);
                    return pg_fail(ld, ORX_ERR_INVALID);
                }
                if ((size_t)l2 != PG_VEC_BYTES) {
                    orx::set_error(ORX_ERR_INVALID, "incorrect binary data format: vector of %d bytes for %d dimensions", l2, dim);
                    return pg_fail(ld, ORX_ERR_INVALID);
                }
                if (have < PG_TUPLE_MAX) return ORX_OK;
                const orx_id id{be64(p + 6), be64(p + 14)};
                if (ld->world > 1 && orx::shard_of_id(id, ld->world) != ld->rank) {
                    ld->foreign += 1;                                     // another rank's row: not staged
                    ld->pos += PG_TUPLE_MAX;
                    break;
                }
                if (!ld->ix) {
                    const int rc = pg_check_elements_host(ld, p + PG_TUPLE_HEAD + 4);
                    if (rc != ORX_OK) return rc;
                }
                ld->ids[ld->n_batch] = id;
                ld->offs[ld->n_batch] = ld->pos + PG_TUPLE_HEAD + 4;
                ld->n_batch += 1;
                ld->pos += PG_TUPLE_MAX;
                break;
            }
            case orx_pgcopy::DONE:
                if (have) {
                    orx::set_error(ORX_ERR_INVALID, "received copy data after EOF marker");
                    return pg_fail(ld, ORX_ERR_INVALID);
                }
                return ORX_OK;
            case orx_pgcopy::FAILED:
                return ld->err;
        }
    }
}

// parse what is buffered; flush whenever a batch is full or the buffer cannot take more bytes
int pg_drain(orx_pgcopy *ld, bool final) {
    for (;;) {
        int rc = pg_parse(ld);
        if (rc != ORX_OK) return rc;
        const bool batch_full = ld->n_batch == PG_BATCH_ROWS;
        const bool no_room = ld->fill == PG_RAW_CAP;
        if (!(batch_full || no_room || final)) return ORX_OK;
        if (!batch_full && ld->pos == 0 && !final) {       // cannot happen: one item is at most PG_TUPLE_MAX bytes
            orx::set_error(ORX_ERR_INVALID, "COPY item larger than the staging buffer");
            return pg_fail(ld, ORX_ERR_INVALID);
        }
        rc = pg_flush(ld);
        if (rc != ORX_OK) return rc;
        if (!batch_full) return ORX_OK;                    // nothing complete is left in the buffer
    }
}

locale_t c_locale() {
    static locale_t loc = newlocale(LC_ALL_MASK, "C", (locale_t)0);
    return loc;
}
inline bool vector_isspace(char c) { return c == ' ' || c == '\t' || c == '\n' || c == '\r' || c == '\v' || c == '\f'; }

}  // namespace

extern "C" {

int orx_pgcopy_open(orx_index *ix, orx_pgcopy **out) { return orx_pgcopy_open_sharded(ix, 1, 0, out); }

int orx_pgcopy_open_sharded(orx_index *ix, int world, int rank, orx_pgcopy **out) {
    if (!out) return orx::set_error(ORX_ERR_INVALID, "out is null");
    *out = nullptr;
    if (world < 1 || rank < 0 || rank >= world) return orx::set_error(ORX_ERR_INVALID, "bad world/rank %d/%d", rank, world);
    orx_pgcopy *ld = new orx_pgcopy();
    ld->ix = ix;
    ld->world = (uint32_t)world;
    ld->rank = (uint32_t)rank;
    if (ix) {
        int prev = -1;
        cudaGetDevice(&prev);
        ld->device = orx::index_device(ix);
        cudaSetDevice(ld->device);
        cudaError_t e = cudaStreamCreateWithFlags(&ld->st, cudaStreamNonBlocking);
        for (orx_pgcopy::Batch &b : ld->batch) {
            if (e == cudaSuccess) e = cudaHostAlloc(reinterpret_cast<void **>(&b.raw), PG_RAW_CAP, cudaHostAllocPortable);
            if (e == cudaSuccess) e = cudaHostAlloc(reinterpret_cast<void **>(&b.ids), PG_BATCH_ROWS * sizeof(orx_id), cudaHostAllocPortable);
            if (e == cudaSuccess) e = cudaHostAlloc(reinterpret_cast<void **>(&b.offs), PG_BATCH_ROWS * sizeof(uint64_t), cudaHostAllocPortable);
            if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void **>(&b.d_raw), PG_RAW_CAP + 16);
            if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void **>(&b.d_offs), PG_BATCH_ROWS * sizeof(uint64_t));
            if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void **>(&b.d_vecs), (size_t)PG_BATCH_ROWS * ORX_DIM * sizeof(float));
        }
        ld->raw = ld->batch[0].raw;
        ld->ids = ld->batch[0].ids;
        ld->offs = ld->batch[0].offs;
        if (prev >= 0) cudaSetDevice(prev);
        if (e != cudaSuccess) {
            cudaGetLastError();
            pg_free(ld);
            return orx::set_error(ORX_ERR_CUDA, "COPY loader buffers: %s", cudaGetErrorString(e));
        }
    } else {
        ld->raw = ld->batch[0].raw = static_cast<uint8_t *>(malloc(PG_RAW_CAP));
        ld->ids = ld->batch[0].ids = static_cast<orx_id *>(malloc(PG_BATCH_ROWS * sizeof(orx_id)));
        ld->offs = ld->batch[0].offs = static_cast<uint64_t *>(malloc(PG_BATCH_ROWS * sizeof(uint64_t)));
        if (!ld->raw || !ld->ids || !ld->offs) {
            pg_free(ld);
            return orx::set_error(ORX_ERR_INVALID, "COPY loader buffers: out of host memory");
        }
    }
    *out = ld;
    return ORX_OK;
}

int orx_pgcopy_feed(orx_pgcopy *ld, const void *bytes, uint64_t n) {
    if (!ld) return orx::set_error(ORX_ERR_INVALID, "loader is null");
    if (ld->state == orx_pgcopy::FAILED) return orx::set_error(ld->err, "COPY loader already failed");
    if (n && !bytes) return orx::set_error(ORX_ERR_INVALID, "null bytes");
    const uint8_t *src = static_cast<const uint8_t *>(bytes);
    ld->bytes += n;
    while (n) {
        const size_t take = (size_t)std::min<uint64_t>(n, PG_RAW_CAP - ld->fill);
        memcpy(ld->raw + ld->fill, src, take);
        ld->fill += take;
        src += take;
        n -= take;
        const int rc = pg_drain(ld, false);
        if (rc != ORX_OK) return rc;
    }
    return ORX_OK;
}

int orx_pgcopy_close(orx_pgcopy *ld, uint64_t *rows_loaded, uint64_t *rows_null) {
    if (rows_loaded) *rows_loaded = 0;
    if (rows_null) *rows_null = 0;
    if (!ld) return orx::set_error(ORX_ERR_INVALID, "loader is null");
    int rc = ld->err;
    if (ld->state == orx_pgcopy::FAILED) {
        // a batch may still be in flight (the failure was found while parsing behind it): it counts if it lands
        if (ld->job_running) {
            ld->job.join();
            ld->job_running = false;
            if (ld->job_rc == ORX_OK) ld->rows += ld->job_rows;
        }
        orx::set_error(rc, "%s", ld->err_text.c_str());
    } else {
        rc = pg_drain(ld, true);
        if (rc == ORX_OK) rc = pg_join(ld);          // the last batch has landed (or failed)
        // EOF at a tuple boundary ends the data like the -1 marker does (Postgres' CopyFrom treats it so);
        // anything else is a truncated stream.  Rows of batches flushed earlier stay loaded, like the
        // batches a COPY consumer already committed.
        if (rc == ORX_OK && ld->state != orx_pgcopy::DONE && !(ld->state == orx_pgcopy::TUPLES && ld->fill == 0))
            rc = orx::set_error(ORX_ERR_INVALID, ld->state == orx_pgcopy::TUPLES ? "unexpected EOF in COPY data"
                                                                                 : "invalid COPY file header (missing length)");
    }
    if (rows_loaded) *rows_loaded = ld->rows;
    if (rows_null) *rows_null = ld->nulls;
    pg_free(ld);
    return rc;
}

int orx_parse_vector_text(const char *text, uint64_t len, float *out, int dim) {
    if (!text || !out) return orx::set_error(ORX_ERR_INVALID, "null argument");
    if (dim < 1 || dim > 16000) return orx::set_error(ORX_ERR_DIM, "dimensions for type vector must be between 1 and 16000");
    const std::string lit(text, (size_t)len);            // NUL-terminated copy, as a cstring argument is
    const char *pt = lit.c_str();
    auto syntax = [&](const char *detail) {
        return orx::set_error(ORX_ERR_INVALID, "invalid input syntax for type vector: \"%.64s\"%s%s", lit.c_str(),
                              detail ? " -- " : "", detail ? detail : "");
    };
    while (vector_isspace(*pt)) ++pt;
    if (*pt != '[') return syntax("Vector contents must start with \"[\".");
    ++pt;
    while (vector_isspace(*pt)) ++pt;
    if (*pt == ']') return orx::set_error(ORX_ERR_DIM, "vector must have at least 1 dimension");
    int n = 0;
    for (;;) {
        if (n == 16000) return orx::set_error(ORX_ERR_DIM, "vector cannot have more than 16000 dimensions");
        while (vector_isspace(*pt)) ++pt;
        if (*pt == '\0') return syntax(nullptr);
        errno = 0;
        char *end = nullptr;
        const float val = strtof_l(pt, &end, c_locale());    // like float4in: no double rounding
        if (end == pt) return syntax(nullptr);
        if (errno == ERANGE && std::isinf(val))
            return orx::set_error(ORX_ERR_INVALID, "\"%.*s\" is out of range for type vector", (int)(end - pt), pt);
        if (std::isnan(val)) return orx::set_error(ORX_ERR_NONFINITE, "NaN not allowed in vector");
        if (std::isinf(val)) return orx::set_error(ORX_ERR_NONFINITE, "infinite value not allowed in vector");
        if (n < dim) out[n] = val;
        ++n;
        pt = end;
        while (vector_isspace(*pt)) ++pt;
        if (*pt == ',') ++pt;
        else if (*pt == ']') {
            ++pt;
            break;
        } else return syntax(nullptr);
    }
    while (vector_isspace(*pt)) ++pt;
    if (*pt != '\0') return syntax("Junk after closing right brace.");
    if (n != dim) return orx::set_error(ORX_ERR_DIM, "expected %d dimensions, not %d", dim, n);
    return ORX_OK;
}

}  // extern "C"
