// Host-side declarations of the kernel launchers (one .cu per kernel family).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/orx.h"

namespace orx {

// Rigorous bounds on |fast score - canonical cosine| per scan path (DESIGN.md, "Exactness").
constexpr double EPS_GEMV_F32 = 3.0e-6;   // fp32 FMA chain of depth 32 + 5 shuffle adds
constexpr double EPS_GEMV_BF16 = 3.0e-6;  // same arithmetic on exactly-converted bf16 rows
// the same scans over the bf16 image of an fp32 table (RNE of every element, not normalised, scored with the fp32 row's
// 1/|x|): |img_i - x_i| <= 2^-8 |x_i| (+ 2^-134 for subnormals) -> |q^.(img - x)| * scale <= 2^-8 (1 + 2^-20), plus the
// fp32 arithmetic of the bf16 dot (EPS_GEMV_BF16); 3.9093e-3 rounded up (DESIGN.md section 2)
constexpr double EPS_GEMV_IMAGE = 3.92e-3;
// live rows from which an fp32 table's single-query / k > 64 batch / bitmap scans read the image (ORX_OPT_IMAGE_MIN_ROWS)
constexpr uint64_t IMAGE_MIN_ROWS = 1ull << 20;
// the 8-bit image of a large fp32 table (ORX_OPT_IMAGE8_MIN_ROWS; DESIGN.md section 2): X_i = rint(x_i / d) with
// d = max|x_i| / 127, scored as the exact integer dot with the query's 15-bit quantisation Q (step dq, residual
// r_q <= 16 dq <= 9.7662e-4) times scale8 = d / |x| and dq.  A row whose relative residual |x - d X| / |x| exceeds
// R8_CAP is an always-candidate (+inf marker), so with r_x <= R8_CAP:
//   |s - cos| <= R8_CAP + (1 + R8_CAP) (r_q + 6e-8) + 2.5e-7 = 1.66172e-2, rounded up
constexpr double R8_CAP = 1.0 / 64;
constexpr double EPS_GEMV_IMAGE8 = 1.662e-2;
// capacities from which an fp32 table's image is the 8-bit one instead of the bf16 one (ORX_OPT_IMAGE8_MIN_ROWS)
constexpr uint64_t IMAGE8_MIN_ROWS = 1ull << 22;
// rows over R8_CAP a table may hold before its searches read the fp32 rows again: every such row takes a slot of every
// candidate list it reaches, and the 8-bit scan's lists keep at least this many keys beyond k
constexpr uint64_t IMAGE8_MAX_CAPPED = 16;
// the 8-bit scan's candidate lists: 160 keys (slots 5) for k <= IMAGE8_MAX_K.  Its eps puts ~200 rows of a 10M-row
// table within 2 eps of the 12th best; a 160-key list proves every query of a 10M-row CPU emulation at k = 12 (least
// margin 1.1e-3), a 128-key one leaves 4 of 32 unproven, and at k = 16 even 160 keys leave 1 of 32 (DESIGN.md section
// 4).  Searches with a wider k read the fp32 rows.
constexpr int IMAGE8_MAX_K = 12;
constexpr int IMAGE8_SLOTS = 5;
// kind::tf32 truncates both operands to 10 mantissa bits (measured on sm_100a, tests/test_epsilon_adversarial_gpu.py):
// worst case (1+2^-10)^2-1 = 1.96e-3; a worst-case query against its own row measures 1.927e-3 (DESIGN.md section 2)
constexpr double EPS_UMMA_TF32 = 2.5e-3;
// RNE bf16 query: 2^-9 = 1.96e-3 (rows are exact bf16); the worst-case construction measures 1.929e-3
constexpr double EPS_UMMA_BF16 = 2.5e-3;

// candidate list = 32 * slots keys per query: k <= 16 -> 32 candidates, k <= 32 -> 64
// candidate list = 32 * slots keys per query: k <= 16 -> 32, k <= 32 -> 64, k <= 128 -> 32 more than k at least
inline int slots_for_k(int k) { return k <= 16 ? 1 : k <= 32 ? 2 : k <= 96 ? 4 : 5; }
// the scans over an fp32 table's bf16 image: one width up.  Their eps is ~1300x the fp32 scan's, so more rows have fast
// scores within eps of the k-th (measured at 10M rows, k = 12: 21-49 rows within 2 eps); finalize's proof needs the
// list's K-th fast score to lie eps below the k-th cosine, and a list of 32 keys left ~6 % of queries unproven
inline int image_slots_for_k(int k) { return k <= 16 ? 2 : k <= 32 ? 4 : 5; }
constexpr int SCAN_THREADS = 256;
constexpr int SCAN_WARPS = SCAN_THREADS / 32;

struct QueryPrep {            // per query, written by prep_queries
    double n2q;               // canonical |q|^2
    int nonfinite;            // 1 if any element is NaN/Inf
    int zero;                 // 1 if |q| == 0 (every distance is NaN)
    float dq8;                // step of the 15-bit quantisation of qhat the 8-bit scan reads (max|qhat_i| / 16383)
};

// the 8-bit image of an fp32 table, as the kernels that write or move rows see it; rows == nullptr: none
struct Image8 {
    int8_t *rows;             // [cap, ORX_DIM] X_i = rint(x_i / d)
    float *scale8;            // [cap] d / |x|, or the row's scale marker (NaN zero row, +inf irregular or over R8_CAP)
};

// ---- where a search's results go and how its completion is signalled (finalize.cu, exchange.cu)
// Result arrays of the WHOLE search, indexed by the query's position in the search (a launch that covers queries
// [q_base, q_base + nq) of it is told q_base).  Device memory, mapped host memory or peer memory alike.
struct ResultOut {
    orx_id *ids;        // [nq_total, k]
    double *dist;       // [nq_total, k]
    int *counts;        // [nq_total]
    int *flags;         // [nq_total]  bit 0 unproven, bit 1 non-finite query, bit 2 zero query, bit 3 rank error
};
// Row-sharded search: finalize pushes this rank's block straight into the gather buffers of its targets (every
// rank, or only the root of a one-process group) with peer stores, and the LAST finalize CTA of the search raises
// this rank's arrival word on each target.  n_targets == 0: not sharded, results go to `ResultOut`.
struct PublishArgs {
    char *const *slot;          // device array [n_targets]: MY slot inside target t's gather buffer (current set)
    uint32_t *const *flag;      // device array [n_targets]: MY arrival word on target t (current set)
    int n_targets;
    uint32_t seq;               // value the arrival words take
    uint64_t dist_off, counts_off, flags_off;      // layout of a slot for (nq_total, k)
};
// Completion of a search made of several launches: every CTA (= query) counts itself on `counter`; the one that
// brings it to `total` resets it and signals -- arrival words (sharded finalize) or `done_host` (a mapped host word the
// host polls instead of synchronising the stream).
struct DoneArgs {
    unsigned int *counter;      // device word, 0 between searches
    unsigned int total;         // queries of the whole search
    uint32_t *done_host;        // mapped host word <- token (nullptr: nothing to signal here)
    uint32_t token;
};

// ---- finalize.cu
// qhat8 (nullptr: none): [nq, 2 * ORX_DIM] int8, the 15-bit quantisation Q of qhat split into Q >> 7 (elements 0..1023)
// and Q & 127 (elements 1024..2047), for the 8-bit scan; its step goes to prep->dq8
void launch_prep_queries(const float *q, int nq, float *q_copy, float *qhat, void *qhat_bf16, int8_t *qhat8,
                         QueryPrep *prep, cudaStream_t st);
// q / prep / partial / floor are launch-relative (query 0 of this launch); results are written at q_base + query
void launch_finalize(int dtype, const void *table, const double *n2, const orx_id *row_ids,
                     const float *q, const QueryPrep *prep, const uint64_t *partial, int nparts,
                     int slots, int nq, int k, uint32_t n_rows, double eps,
                     const ResultOut &out, int q_base, const PublishArgs &pub, const DoneArgs &done,
                     cudaStream_t st, const float *floor = nullptr, const uint32_t *covered = nullptr);
// covered (nq == 1): rows the scan offered for the query (LapState::covered); a count other than n_rows leaves the query
// unproven, so the exhaustive pass answers it
// list_stride_bytes == 0: three dense [n_lists][...] arrays; otherwise list l of each array is at +l*stride
void launch_merge_topk(int n_lists, int nq, int k, const orx_id *ids, const double *dist,
                       const int *counts, size_t list_stride_bytes, orx_id *out_ids, double *out_dist,
                       int *out_counts, cudaStream_t st);
// exhaustive fallback: collect rows whose fast score may reach `cos_floor`, rescore, select
void launch_collect(int dtype, const void *table, const float *scale, uint32_t n_rows,
                    const float *qhat, float fast_floor, int collect_all,
                    uint32_t *list, uint32_t *count, cudaStream_t st);
// diagnostic: fast scores of every row for nq staged queries, out [n_rows, nq] (orx_debug_fast_scores)
void launch_dump_fast_scores(int dtype, const void *table, const float *scale, uint32_t n_rows, const float *qhat,
                             int nq, float *out, cudaStream_t st);
// the same diagnostic for the 8-bit scan (orx_debug_image8_scores)
void launch_dump_image8_scores(const int8_t *image, const float *scale8, uint32_t n_rows, const int8_t *qhat8,
                               const QueryPrep *prep, int nq, float *out, cudaStream_t st);
void launch_rescore_list(int dtype, const void *table, const double *n2, const orx_id *row_ids,
                         const float *q, const QueryPrep *prep, const uint32_t *list,
                         const uint32_t *count, double *dist_out, cudaStream_t st);
void launch_select_list(const orx_id *row_ids, const uint32_t *list, const uint32_t *count,
                        const double *dist, int k, orx_id *out_ids, double *out_dist,
                        int *out_count, cudaStream_t st);

void launch_flags_from_prep(const QueryPrep *prep, int nq, int *flags, cudaStream_t st);
void launch_fill_flags(int *flags, int nq, int value, cudaStream_t st);

// ---- exchange.cu (row-sharded search over NVLink peer memory)
void launch_publish(const void *my_slot, void *const *peer_slot, uint32_t *const *peer_flag, int world,
                    size_t bytes, uint32_t seq, cudaStream_t st);
// err_host: mapped host word <- 1 when a rank never arrived within the bounded wait (the kernel then gives up
// WITHOUT trapping: the CUDA context and the resident table survive, the host reports ORX_ERR_CUDA)
void launch_merge_wait(int world, int rank, int nq, int k, const void *set_base, size_t slot_stride,
                       size_t dist_off, size_t counts_off, size_t flags_off, const uint32_t *arrival,
                       int arrival_stride_words, uint32_t seq, orx_id *out_ids, double *out_dist,
                       int *out_counts, int *flags_any, int *flags_mine, int *redo, uint32_t *err_host,
                       const DoneArgs &done, cudaStream_t st);
void launch_signal_done(const DoneArgs &done, cudaStream_t st);      // 1 thread: *done_host = token (paths without a last CTA)

// ---- scan_gemv.cu
int scan_gemv_grid(int device, uint32_t n_rows);
void launch_scan_gemv(int dtype, const void *table, const float *scale, uint32_t n_rows,
                      const float *qhat, int nq, int slots, uint64_t *partial, int grid,
                      cudaStream_t st);

// the same scan over the rows whose bit is set in allow_bits [(n_rows+31)/32 words; bits >= n_rows are 0]
int scan_gemv_batch_parts(int device, uint32_t n_rows, int nq);
void launch_scan_gemv_batch(int dtype, const void *table, const float *scale, uint32_t n_rows, const float *qhat, int nq,
                            int slots, uint64_t *partial, int parts, cudaStream_t st);
void launch_scan_gemv_filtered(int dtype, const void *table, const float *scale, uint32_t n_rows,
                               const uint32_t *allow_bits, const float *qhat, int nq, int slots,
                               uint64_t *partial, int grid, cudaStream_t st);
// the single-query and bitmap scans over the 8-bit image (IMAGE8_SLOTS lists); allow_bits == nullptr: every row
void launch_scan_gemv8(const int8_t *image, const float *scale8, uint32_t n_rows, const uint32_t *allow_bits,
                       const int8_t *qhat8, const QueryPrep *prep, int nq, uint64_t *partial, int grid, cudaStream_t st);

// The single-query scan over the 8-bit image of a search submitted with orx_search_submit is a LAP (DESIGN.md section
// 4, "two searches in flight"; orx_search, which no other search can join, keeps scan_gemv8_kernel): the table is cut
// into LAP_SEGS segments, warps claim LAP_CHUNK rows at a time from a device-side counter, front to back, and the first
// claim in a segment SEALS the segment's query-set word.  Until then a second search may JOIN the segment (atomicCAS
// 0 -> SEG_JOINED, join kernel): every claimer of the segment then scores its rows against both queries.  A sealed word
// never changes, so all claimers see the same set.  The joiner's CATCH-UP is a lap of its own over the segments it did
// not get (itself joinable), merged into the lists the joined lap left.  Every lap counts the rows it offered per query
// into that query's `covered`; finalize marks a query unproven unless covered == n_rows.
constexpr int LAP_SEGS = 64;
constexpr uint32_t LAP_CHUNK = 64;
constexpr uint32_t SEG_SEALED = 1u << 31, SEG_JOINED = 1u;
struct LapJoiner {               // written by the join kernel before its first atomicCAS
    const int8_t *q8;            // the joiner's qhat8 (h | l slices) and prep
    const QueryPrep *prep;
    uint64_t *partial;           // its per-CTA lists for this lap's grid, zeroed before the join
    uint32_t *covered;
};
struct LapState {                // one per search slot, device memory
    uint32_t next;               // work queue: chunks claimed so far
    uint32_t covered;            // rows offered for this slot's query, by its own lap and by a lap it joined
    uint32_t n_list;             // catch-up: segments to scan, list[0, n_list)
    uint32_t pad;
    uint32_t seg[LAP_SEGS];      // query-set word of each segment: SEG_SEALED | SEG_JOINED
    uint32_t list[LAP_SEGS];
    LapJoiner joiner;
};
// rows per segment (a multiple of LAP_CHUNK, so a chunk never straddles two segments)
inline uint32_t lap_seg_rows(uint32_t n_rows) {
    const uint32_t per = (n_rows + LAP_SEGS - 1) / LAP_SEGS;
    return (per + LAP_CHUNK - 1) / LAP_CHUNK * LAP_CHUNK;
}
// the lap of one query (q8 / prep / partial of query 0).  catch_up == 0: every segment, lap->seg all 0 (the caller
// clears next / covered / seg); catch_up == 1: the segments in lap->list (join kernel), each CTA's list merged with
// the one partial already holds
void launch_scan_lap8(const int8_t *image, const float *scale8, uint32_t n_rows, const int8_t *qhat8,
                      const QueryPrep *prep, uint64_t *partial, LapState *lap, int catch_up, int grid, cudaStream_t st);
// one CTA: publish `me` on `host`, try to join every segment of host's lap that is still open, and set up `mine` (the
// joiner's own lap state; next / covered already cleared) for the catch-up over the others.  rows_joined: mapped host
// word <- rows of the joined segments
void launch_join_lap8(LapState *host, LapState *mine, const LapJoiner &me, uint32_t n_rows, uint32_t *rows_joined,
                      cudaStream_t st);

// ---- table_ops.cu
void launch_validate_rows(const float *src, uint64_t n, int *flag, cudaStream_t st);
// image: the bf16 image of an fp32 table ([cap, ORX_DIM] __nv_bfloat16), kept in step with the rows; nullptr = none
//        image8: the 8-bit image (Image8::rows == nullptr: none); a table has at most one of the two
void launch_commit_rows(int dtype, const float *src, const uint32_t *src_idx, const uint32_t *dst_row,
                        const orx_id *ids, uint32_t n, void *table, float *scale, double *n2,
                        orx_id *row_ids, const int *abort_flag, void *image, const Image8 &image8, cudaStream_t st);
void launch_adopt_rows(int dtype, const void *table, uint32_t row0, uint32_t n, const orx_id *ids, float *scale,
                       double *n2, orx_id *row_ids, int *flag, void *image, const Image8 &image8, cudaStream_t st);
void launch_move_rows(int dtype, const uint32_t *src_row, const uint32_t *dst_row, uint32_t n,
                      void *table, float *scale, double *n2, orx_id *row_ids, void *image, const Image8 &image8,
                      cudaStream_t st);
void launch_image_rows(const float *table, uint64_t n, void *image, cudaStream_t st);     // image of rows [0, n)
void launch_image8_rows(const float *table, const double *n2, const float *scale, uint64_t n, const Image8 &image8,
                        cudaStream_t st);                                                 // 8-bit image of rows [0, n)
// *count <- live rows [0, n) over R8_CAP (scale8 +inf while scale is regular)
void launch_count_capped8(const float *scale, const float *scale8, uint64_t n, uint32_t *count, cudaStream_t st);
void launch_gather_rows(int dtype, const void *table, const uint32_t *rows, uint32_t n, float *out,
                        cudaStream_t st);

// ---- pgwire.cu (pgvector wire formats: COPY BINARY bulk load, text input)
void launch_mask_scale(const float *scale, const uint32_t *allow_bits, uint32_t n_rows, float *out, cudaStream_t st);
void launch_decode_pgvector(const uint8_t *raw, const uint64_t *payload_off, uint32_t n, float *out,
                            cudaStream_t st);

// ---- mmr.cu (orx_search_mmr*): rows [nq, fetch_k, ORX_DIM] = each query's candidates in contract order, gathered
//      as fp32; dist [nq, fetch_k] their canonical distances; counts [nq].  sel [nq, k] <- picked positions in selection
//      order, -1 past min(k, count)
void launch_mmr_select(const float *rows, const double *dist, const int *counts, int nq, int fetch_k, int k,
                       double lam, int *sel, cudaStream_t st);

// launch `kernel` on `st` with the programmatic-stream-serialization attribute (common.cuh: PDL)
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// SM count of the CURRENT device (cached per device): launch geometry is sized from it, never from a literal
int device_sms();
template <typename T> inline T cap_grid(T blocks, int ctas_per_sm) {     // persistent-style grids: <= ctas_per_sm x SMs
    const T cap = (T)device_sms() * (T)ctas_per_sm;
    return blocks > cap ? cap : blocks;
}

// mix64(hi * GOLD ^ lo): the hash of the host's id -> row map and, mod the shard count, the row-shard function
// (== outline_rag_b200/sharded.py shard_of, SURVEY.md 8e)
inline uint64_t id_hash(const orx_id &id) {
    uint64_t z = id.hi * 0x9E3779B97F4A7C15ull ^ id.lo;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
inline uint32_t shard_of_id(const orx_id &id, uint32_t world) { return (uint32_t)(id_hash(id) % world); }

// ---- orx_api.cu: what the other translation units need from an index
int set_error(int code, const char *fmt, ...);     // records the thread-local message, returns code
int index_device(const orx_index *ix);
void index_count_launches(orx_index *ix, uint64_t n);

}  // namespace orx
