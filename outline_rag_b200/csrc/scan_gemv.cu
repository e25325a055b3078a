// scan_gemv: the single-query sequential scan -- HBM-bound GEMV with a fused top-K select.
//
// Stands in for the per-row `cosine_distance(row.embedding, q)` + top-N heapsort that the
// Postgres executor runs for `ORDER BY embedding <=> :q LIMIT :k`
// (pgvector src/vector.c [UPSTREAM]; SQL reached from reference app/rag.py:85-87).
//
// Layout / schedule (DESIGN.md "scan_gemv"):
//   * persistent grid: 2 CTAs x 8 warps per SM, one warp per row, ROWS_PER_ITER rows per
//     warp in flight; a warp's rows are consecutive so each warp streams 8 KB contiguous,
//     and the whole grid walks the table front to back (DRAM page locality);
//   * 128-bit ld.global.nc.L1::no_allocate loads, lane l owns elements 4*(l+32j)..+3
//     (fp32) or 8*(l+32j)..+7 (bf16) and keeps the matching slice of the normalised query
//     in 32 registers;
//   * fp32 FMA chain per lane + xor-butterfly -> every lane has the dot; score = dot*scale[row];
//   * one compare per row against the warp's running K-th best; the rare insert shifts a
//     register-resident sorted list spread over the 32 lanes (common.cuh WarpTopK);
//   * per-CTA merge in shared memory -> partial[query][cta][KC] (sorted keys).
// Algorithmic bytes per launch: n_rows * 1024 * sizeof(elem) (+4 B/row scale, <0.1%).
#include "scan_common.cuh"
#include "internal.h"

namespace orx {

// per-CTA merge by counting, shared by the scan kernels: the 8 warp lists hold 8*K distinct keys (0 = empty), each sorted
// descending; a key's rank is the number of larger keys (a binary search per list), ranks < K are the CTA's sorted
// top-K -> partial[0..K)
template <int S>
__device__ __forceinline__ void cta_merge_store(const WarpTopK<S> &top, uint64_t (&s_keys)[SCAN_WARPS][32 * S],
                                                uint64_t *__restrict__ partial, int lane, int warp) {
    constexpr int K = 32 * S;
    top.store(s_keys[warp], lane);
    __syncthreads();
    const uint64_t *all = &s_keys[0][0];
    constexpr int TOTAL = SCAN_WARPS * K;
    int nonzero = 0;
#pragma unroll
    for (int h = 0; h < TOTAL / SCAN_THREADS; ++h) {
        const uint64_t mine = all[threadIdx.x + h * SCAN_THREADS];
        nonzero += (mine != 0ull);
        if (mine == 0ull) continue;
        int rank = 0;
#pragma unroll
        for (int w = 0; w < SCAN_WARPS; ++w) {
            int lo = 0, hi = K;                         // keys of list w above `mine`: the first position not above it
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if (s_keys[w][mid] > mine) lo = mid + 1;
                else hi = mid;
            }
            rank += lo;
        }
        if (rank < K) partial[rank] = mine;
    }
    int nnz = 0;
#pragma unroll
    for (int j = 1; j <= TOTAL / SCAN_THREADS; ++j) nnz += __syncthreads_count(nonzero >= j);
    if ((int)threadIdx.x < K && (int)threadIdx.x >= nnz) partial[threadIdx.x] = 0ull;
}

template <typename T> struct RowsPerIter { static constexpr int value = sizeof(T) == 4 ? 2 : 4; };   // 8 KB per warp in flight

template <typename T, int S>
__global__ void __launch_bounds__(SCAN_THREADS, 2)
scan_gemv_kernel(const T *__restrict__ table, const float *__restrict__ scale, uint32_t n_rows,
                 const float *__restrict__ qhat_all, uint64_t *__restrict__ partial_all) {
    constexpr int NV = RowVec<T>::NV;
    constexpr int ROWS_PER_ITER = RowsPerIter<T>::value;
    constexpr int K = 32 * S;
    __shared__ uint64_t s_keys[SCAN_WARPS][K];

    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int query = blockIdx.y;
    const float *qhat = qhat_all + (size_t)query * ORX_DIM;
    uint64_t *partial = partial_all + ((size_t)query * gridDim.x + blockIdx.x) * K;

    pdl_launch_dependents();          // finalize may be scheduled as soon as an SM has room; it parks at its own wait
    pdl_wait();                       // prep_queries (qhat) and the previous reader of `partial` are done
    float4 qv[8];
    load_q_slice<T>(qhat, lane, qv);

    WarpTopK<S> top;
    top.init();

    const uint4 *tab = reinterpret_cast<const uint4 *>(table);
    const uint32_t gw = blockIdx.x * SCAN_WARPS + warp;
    const uint32_t n_gw = gridDim.x * SCAN_WARPS;
    const uint32_t n_chunks = (n_rows + ROWS_PER_ITER - 1) / ROWS_PER_ITER;

    for (uint32_t c = gw; c < n_chunks; c += n_gw) {
        uint4 v[ROWS_PER_ITER][NV];
        float sc[ROWS_PER_ITER];
        const uint32_t row0 = c * ROWS_PER_ITER;
#pragma unroll
        for (int r = 0; r < ROWS_PER_ITER; ++r) {
            const uint32_t rr = min(row0 + r, n_rows - 1);   // tail rows re-read the last row
            load_row_vecs<T>(tab, rr, lane, v[r]);
            sc[r] = __ldg(scale + rr);
        }
#pragma unroll
        for (int r = 0; r < ROWS_PER_ITER; ++r) {
            const float acc = warp_row_dot<T>(v[r], qv);
            const uint32_t row = row0 + r;
            if (row < n_rows) top.offer(make_key(score_ord(acc, sc[r]), row), lane);
        }
    }

    cta_merge_store<S>(top, s_keys, partial, lane, warp);
}

// ------------------------------------------------------------------ batched exact scan
// The same fp32 scan for a BATCH the tensor-core pass cannot take (k beyond its candidate lists): the 8 warps of a CTA
// serve 8 DIFFERENT queries and share every row through shared memory, so a row is fetched once per 8 queries instead
// of once per query (cp.async 16-byte copies, double-buffered tiles of 16 KB).  Each warp keeps its query slice in
// registers and scores a row with the SAME instruction sequence as the single-query scan (warp_row_dot on the same
// lane / vector assignment), so fast scores, error bound and completeness proof are those of scan_gemv_kernel; a warp's
// sorted top-K is the (query, CTA) list itself.  grid = (row partitions, ceil(nq / 8)); CTAs that differ only in their
// query group walk the same tiles at the same time, so the extra passes are served by L2.
template <typename T> struct BatchTile { static constexpr int ROWS = sizeof(T) == 4 ? 4 : 8; };     // 16 KB of rows

__device__ __forceinline__ void cp_async_16(void *smem_dst, const void *gmem_src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gmem_src)
                 : "memory");
}

template <typename T, int S>
__global__ void __launch_bounds__(SCAN_THREADS, 2)
scan_gemv_batch_kernel(const T *__restrict__ table, const float *__restrict__ scale, uint32_t n_rows,
                       const float *__restrict__ qhat_all, int nq, uint64_t *__restrict__ partial_all) {
    constexpr int NV = RowVec<T>::NV;
    constexpr int VPR = RowVec<T>::VEC_PER_ROW;
    constexpr int ROWS = BatchTile<T>::ROWS;
    constexpr int TILE_VECS = ROWS * VPR;                      // 1024 16-byte vectors
    constexpr int K = 32 * S;
    __shared__ uint4 s_rows[2][TILE_VECS];

    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int query = blockIdx.y * SCAN_WARPS + warp;
    const bool active = query < nq;

    pdl_launch_dependents();
    pdl_wait();
    float4 qv[8];
    load_q_slice<T>(qhat_all + (size_t)(active ? query : 0) * ORX_DIM, lane, qv);

    WarpTopK<S> top;
    top.init();

    const uint4 *tab = reinterpret_cast<const uint4 *>(table);
    const uint32_t n_tiles = (n_rows + ROWS - 1) / ROWS;
    auto fetch = [&](uint32_t t, int buf) {
#pragma unroll
        for (int i = 0; i < TILE_VECS / SCAN_THREADS; ++i) {
            const int idx = threadIdx.x + i * SCAN_THREADS;
            const uint32_t row = min(t * ROWS + (uint32_t)(idx / VPR), n_rows - 1);      // tail rows re-read the last row
            cp_async_16(&s_rows[buf][idx], tab + (size_t)row * VPR + (idx % VPR));
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    uint32_t t = blockIdx.x;
    int buf = 0;
    if (t < n_tiles) fetch(t, 0);
    for (; t < n_tiles; t += gridDim.x, buf ^= 1) {
        const uint32_t t_next = t + gridDim.x;
        if (t_next < n_tiles) {
            fetch(t_next, buf ^ 1);
            asm volatile("cp.async.wait_group 1;" ::: "memory");
        } else {
            asm volatile("cp.async.wait_group 0;" ::: "memory");
        }
        __syncthreads();                                       // every thread's copies of this tile have landed
#pragma unroll
        for (int r = 0; r < ROWS; ++r) {
            uint4 v[NV];
#pragma unroll
            for (int j = 0; j < NV; ++j) v[j] = s_rows[buf][r * VPR + lane + 32 * j];
            const float acc = warp_row_dot<T>(v, qv);
            const uint32_t row = t * ROWS + r;
            if (active && row < n_rows) top.offer(make_key(score_ord(acc, __ldg(scale + row)), row), lane);
        }
        __syncthreads();                                       // the buffer may be refilled by the next iteration
    }
    if (active) top.store(partial_all + ((size_t)query * gridDim.x + blockIdx.x) * K, lane);
}

// ------------------------------------------------------------------ filtered scan
// The same scan restricted to the rows whose bit is set in `allow_bits` (bit r%32 of word r/32; bits at
// or beyond n_rows are 0): the SQL with a WHERE clause once the predicate is resolved to rows
// (orx_search_filtered, SURVEY.md 8f-4 "bitmap AND pushed into the scan").  Work unit = one bitmap word
// = 32 consecutive rows per warp; rows whose bit is clear are never loaded, so HBM traffic is
// eligible_rows * row_bytes.  Scores come from the same instruction sequence as the unfiltered scan
// (scan_common.cuh), so the same error bound and the same completeness proof apply.
template <typename T, int S>
__global__ void __launch_bounds__(SCAN_THREADS, 2)
scan_gemv_filtered_kernel(const T *__restrict__ table, const float *__restrict__ scale, uint32_t n_rows,
                          const uint32_t *__restrict__ allow_bits, const float *__restrict__ qhat_all,
                          uint64_t *__restrict__ partial_all) {
    constexpr int NV = RowVec<T>::NV;
    constexpr int ROWS_PER_ITER = RowsPerIter<T>::value;
    constexpr int K = 32 * S;
    __shared__ uint64_t s_keys[SCAN_WARPS][K];

    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int query = blockIdx.y;
    const float *qhat = qhat_all + (size_t)query * ORX_DIM;
    uint64_t *partial = partial_all + ((size_t)query * gridDim.x + blockIdx.x) * K;

    float4 qv[8];
    load_q_slice<T>(qhat, lane, qv);

    WarpTopK<S> top;
    top.init();

    const uint4 *tab = reinterpret_cast<const uint4 *>(table);
    const uint32_t gw = blockIdx.x * SCAN_WARPS + warp;
    const uint32_t n_gw = gridDim.x * SCAN_WARPS;
    const uint32_t n_groups = (n_rows + 31) / 32;

    uint32_t w_next = gw < n_groups ? __ldg(allow_bits + gw) : 0u;
    for (uint32_t g = gw; g < n_groups; g += n_gw) {
        uint32_t w = w_next;                                        // warp-uniform
        w_next = g + n_gw < n_groups ? __ldg(allow_bits + g + n_gw) : 0u;   // in flight while this group streams
        while (w) {
            uint4 v[ROWS_PER_ITER][NV];
            float sc[ROWS_PER_ITER];
            uint32_t row[ROWS_PER_ITER];
            bool ok[ROWS_PER_ITER];
#pragma unroll
            for (int r = 0; r < ROWS_PER_ITER; ++r) {
                ok[r] = w != 0u;
                row[r] = g * 32u + (ok[r] ? (uint32_t)(__ffs(w) - 1) : 0u);
                w &= w - 1u;                                        // 0 stays 0
                if (ok[r]) {
                    load_row_vecs<T>(tab, row[r], lane, v[r]);
                    sc[r] = __ldg(scale + row[r]);
                }
            }
#pragma unroll
            for (int r = 0; r < ROWS_PER_ITER; ++r) {
                if (ok[r] && row[r] < n_rows) {
                    const float acc = warp_row_dot<T>(v[r], qv);
                    top.offer(make_key(score_ord(acc, sc[r]), row[r]), lane);
                }
            }
        }
    }
    cta_merge_store<S>(top, s_keys, partial, lane, warp);
}

// ------------------------------------------------------------------ 8-bit image scan
// The single-query and bitmap scans over the 8-bit image of an fp32 table (DESIGN.md section 2): a row is 1024 int8
// X_i = rint(x_i / d), scored as the EXACT integer dot D = sum X_i Q_i with the query's 15-bit quantisation, then
// s = (float(D) * dq) * scale8[row], scale8 = d / |x|.  Q = 128 h + l is held as two int8 slices (h = Q >> 7 in
// [-128, 127], l = Q & 127), so D = 128 sum X h + sum X l comes from 16 __dp4a per lane and row; |D| <= 1024 * 128 *
// 16383 < 2^31, so every partial sum is exact and the order of the sums does not matter.  Schedule as scan_gemv_kernel:
// persistent grid, one warp per row, lane l owns the 16-byte vectors l and l + 32 of a 1 KB row, ROWS8 rows (8 KB) per
// warp in flight.  The 8 rows' lane partials are reduced together (9 shuffles for 8 rows instead of 40); afterwards lane
// group l / 4 holds row l / 4, scores it, and the warp offers the 8 keys through the usual WarpTopK.
constexpr int ROWS8 = 8;
constexpr int SLOTS8 = IMAGE8_SLOTS;

__device__ __forceinline__ int lane_dot8(const uint4 (&v)[2], const uint4 (&qh)[2], const uint4 (&ql)[2]) {
    int h = 0, l = 0;
#pragma unroll
    for (int j = 0; j < 2; ++j) {
        h = __dp4a((int)v[j].x, (int)qh[j].x, h);
        h = __dp4a((int)v[j].y, (int)qh[j].y, h);
        h = __dp4a((int)v[j].z, (int)qh[j].z, h);
        h = __dp4a((int)v[j].w, (int)qh[j].w, h);
        l = __dp4a((int)v[j].x, (int)ql[j].x, l);
        l = __dp4a((int)v[j].y, (int)ql[j].y, l);
        l = __dp4a((int)v[j].z, (int)ql[j].z, l);
        l = __dp4a((int)v[j].w, (int)ql[j].w, l);
    }
    return 128 * h + l;
}

// p[r]: this lane's partial dot of row r -> the full dot of row lane / 4 (in all four lanes of the group)
__device__ __forceinline__ int warp_reduce8(const int (&p)[ROWS8], int lane) {
    const bool b4 = lane & 16, b3 = lane & 8, b2 = lane & 4;
    int a[4], b[2];
#pragma unroll
    for (int i = 0; i < 4; ++i)          // rows 4 * b4 + i
        a[i] = (b4 ? p[i + 4] : p[i]) + __shfl_xor_sync(FULL_MASK, b4 ? p[i] : p[i + 4], 16);
#pragma unroll
    for (int i = 0; i < 2; ++i)          // rows 4 * b4 + 2 * b3 + i
        b[i] = (b3 ? a[i + 2] : a[i]) + __shfl_xor_sync(FULL_MASK, b3 ? a[i] : a[i + 2], 8);
    int c = (b2 ? b[1] : b[0]) + __shfl_xor_sync(FULL_MASK, b2 ? b[0] : b[1], 4);     // row lane / 4
    c += __shfl_xor_sync(FULL_MASK, c, 2);
    c += __shfl_xor_sync(FULL_MASK, c, 1);
    return c;
}

// the score every 8-bit path keys on (scan and orx_debug_image8_scores): D and dq -> float(D) * dq, then * scale8
__device__ __forceinline__ float image8_dot(int D, float dq) { return __fmul_rn(__int2float_rn(D), dq); }

__device__ __forceinline__ void load_q8_slice(const int8_t *q8, int lane, uint4 (&qh)[2], uint4 (&ql)[2]) {
    const uint4 *p = reinterpret_cast<const uint4 *>(q8);
#pragma unroll
    for (int j = 0; j < 2; ++j) {
        qh[j] = p[lane + 32 * j];
        ql[j] = p[64 + lane + 32 * j];
    }
}

// allow_bits == nullptr: rows in chunks of ROWS8 consecutive rows; otherwise one bitmap word (32 rows) per work unit and
// only the rows whose bit is set are loaded
template <bool FILTERED>
__global__ void __launch_bounds__(SCAN_THREADS, 2)
scan_gemv8_kernel(const int8_t *__restrict__ table, const float *__restrict__ scale8, uint32_t n_rows,
                  const uint32_t *__restrict__ allow_bits, const int8_t *__restrict__ q8_all,
                  const QueryPrep *__restrict__ prep, uint64_t *__restrict__ partial_all) {
    constexpr int K = 32 * SLOTS8;
    __shared__ uint64_t s_keys[SCAN_WARPS][K];

    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int query = blockIdx.y;
    uint64_t *partial = partial_all + ((size_t)query * gridDim.x + blockIdx.x) * K;

    if (!FILTERED) {
        pdl_launch_dependents();
        pdl_wait();
    }
    uint4 qh[2], ql[2];
    load_q8_slice(q8_all + (size_t)query * 2 * ORX_DIM, lane, qh, ql);
    const float dq = prep[query].dq8;

    WarpTopK<SLOTS8> top;
    top.init();

    const uint4 *tab = reinterpret_cast<const uint4 *>(table);
    const uint32_t gw = blockIdx.x * SCAN_WARPS + warp;
    const uint32_t n_gw = gridDim.x * SCAN_WARPS;
    const int my = lane >> 2;                                  // the row of the group this lane scores

    // score ROWS8 loaded rows (row[r] valid where ok[r]) and offer them
    auto score = [&](const uint4 (&v)[ROWS8][2], uint32_t my_row, bool my_ok, float my_sc) {
        int p[ROWS8];
#pragma unroll
        for (int r = 0; r < ROWS8; ++r) p[r] = lane_dot8(v[r], qh, ql);
        const int D = warp_reduce8(p, lane);
        const uint64_t key = my_ok ? make_key(score_ord(image8_dot(D, dq), my_sc), my_row) : 0ull;
        top.offer_lanes((lane & 3) == 0 ? key : 0ull, lane);
    };

    if (!FILTERED) {
        const uint32_t n_chunks = (n_rows + ROWS8 - 1) / ROWS8;
        for (uint32_t c = gw; c < n_chunks; c += n_gw) {
            uint4 v[ROWS8][2];
            const uint32_t row0 = c * ROWS8;
            const uint32_t my_row = row0 + my;
            const float my_sc = __ldg(scale8 + min(my_row, n_rows - 1));
#pragma unroll
            for (int r = 0; r < ROWS8; ++r) {
                const uint4 *p = tab + (size_t)min(row0 + r, n_rows - 1) * 64 + lane;   // tail rows re-read the last
                v[r][0] = ldg_stream_u4(p);
                v[r][1] = ldg_stream_u4(p + 32);
            }
            score(v, my_row, my_row < n_rows, my_sc);
        }
    } else {
        const uint32_t n_groups = (n_rows + 31) / 32;
        uint32_t w_next = gw < n_groups ? __ldg(allow_bits + gw) : 0u;
        for (uint32_t g = gw; g < n_groups; g += n_gw) {
            uint32_t w = w_next;                                        // warp-uniform
            w_next = g + n_gw < n_groups ? __ldg(allow_bits + g + n_gw) : 0u;
            while (w) {
                uint4 v[ROWS8][2];
                uint32_t my_row = 0;
                bool my_ok = false;
#pragma unroll
                for (int r = 0; r < ROWS8; ++r) {
                    const bool ok = w != 0u;
                    const uint32_t row = g * 32u + (ok ? (uint32_t)(__ffs(w) - 1) : 0u);
                    w &= w - 1u;                                        // 0 stays 0
                    if (r == my) {
                        my_row = row;
                        my_ok = ok && row < n_rows;
                    }
                    if (ok) {
                        const uint4 *p = tab + (size_t)row * 64 + lane;
                        v[r][0] = ldg_stream_u4(p);
                        v[r][1] = ldg_stream_u4(p + 32);
                    } else {
                        v[r][0] = v[r][1] = make_uint4(0u, 0u, 0u, 0u);
                    }
                }
                const float my_sc = my_ok ? __ldg(scale8 + my_row) : 0.f;
                score(v, my_row, my_ok, my_sc);
            }
        }
    }
    cta_merge_store<SLOTS8>(top, s_keys, partial, lane, warp);
}

void launch_scan_gemv8(const int8_t *image, const float *scale8, uint32_t n_rows, const uint32_t *allow_bits,
                       const int8_t *qhat8, const QueryPrep *prep, int nq, uint64_t *partial, int grid, cudaStream_t st) {
    dim3 g(grid, nq);
    if (allow_bits)
        scan_gemv8_kernel<true><<<g, SCAN_THREADS, 0, st>>>(image, scale8, n_rows, allow_bits, qhat8, prep, partial);
    else
        launch_pdl(scan_gemv8_kernel<false>, g, dim3(SCAN_THREADS), 0, st, image, scale8, n_rows, allow_bits, qhat8, prep,
                   partial);
}

// orx_debug_image8_scores: every row's 8-bit score (the value score_ord keys on) for nq queries, out[row * nq + query]
__global__ void __launch_bounds__(256)
dump_image8_kernel(const int8_t *__restrict__ table, const float *__restrict__ scale8, uint32_t n_rows,
                   const int8_t *__restrict__ q8_all, const QueryPrep *__restrict__ prep, float *__restrict__ out) {
    const int lane = threadIdx.x & 31;
    const uint32_t gw = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const uint32_t n_gw = gridDim.x * (blockDim.x >> 5);
    uint4 qh[2], ql[2];
    load_q8_slice(q8_all + (size_t)blockIdx.y * 2 * ORX_DIM, lane, qh, ql);
    const float dq = prep[blockIdx.y].dq8;
    const uint4 *tab = reinterpret_cast<const uint4 *>(table);
    for (uint32_t row = gw; row < n_rows; row += n_gw) {
        const uint4 v[2] = {tab[(size_t)row * 64 + lane], tab[(size_t)row * 64 + lane + 32]};
        int D = lane_dot8(v, qh, ql);
#pragma unroll
        for (int d = 16; d >= 1; d >>= 1) D += __shfl_xor_sync(FULL_MASK, D, d);
        if (lane == 0) out[(size_t)row * gridDim.y + blockIdx.y] = image8_dot(D, dq) * __ldg(scale8 + row);
    }
}

void launch_dump_image8_scores(const int8_t *image, const float *scale8, uint32_t n_rows, const int8_t *qhat8,
                               const QueryPrep *prep, int nq, float *out, cudaStream_t st) {
    if (n_rows == 0 || nq <= 0) return;
    dump_image8_kernel<<<dim3(device_sms() * 4, nq), 256, 0, st>>>(image, scale8, n_rows, qhat8, prep, out);
}

int scan_gemv_grid(int device, uint32_t n_rows) {
    int sms = 0;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || sms <= 0) sms = 1;
    constexpr int ROWS_PER_ITER = 2;      // grid sizing only: enough chunks for every warp of the persistent grid
    uint32_t chunks = (n_rows + ROWS_PER_ITER - 1) / ROWS_PER_ITER;
    uint32_t want = (chunks + SCAN_WARPS - 1) / SCAN_WARPS;
    uint32_t full = (uint32_t)sms * 2u;
    uint32_t g = want < full ? want : full;
    return g < 1 ? 1 : (int)g;
}

template <typename T>
static void launch_scan_gemv_t(const void *table, const float *scale, uint32_t n_rows, const float *qhat,
                               int nq, int slots, uint64_t *partial, int grid, cudaStream_t st) {
    dim3 g(grid, nq);
    const T *tab = static_cast<const T *>(table);
    switch (slots) {
        case 1: launch_pdl(scan_gemv_kernel<T, 1>, g, dim3(SCAN_THREADS), 0, st, tab, scale, n_rows, qhat, partial); break;
        case 2: launch_pdl(scan_gemv_kernel<T, 2>, g, dim3(SCAN_THREADS), 0, st, tab, scale, n_rows, qhat, partial); break;
        case 4: launch_pdl(scan_gemv_kernel<T, 4>, g, dim3(SCAN_THREADS), 0, st, tab, scale, n_rows, qhat, partial); break;
        default: launch_pdl(scan_gemv_kernel<T, 5>, g, dim3(SCAN_THREADS), 0, st, tab, scale, n_rows, qhat, partial); break;
    }
}

void launch_scan_gemv(int dtype, const void *table, const float *scale, uint32_t n_rows,
                      const float *qhat, int nq, int slots, uint64_t *partial, int grid,
                      cudaStream_t st) {
    if (dtype == ORX_DTYPE_F32)
        launch_scan_gemv_t<float>(table, scale, n_rows, qhat, nq, slots, partial, grid, st);
    else
        launch_scan_gemv_t<__nv_bfloat16>(table, scale, n_rows, qhat, nq, slots, partial, grid, st);
}

// partitions of the batched scan: two resident CTAs per SM over all query groups, at least one tile each
int scan_gemv_batch_parts(int device, uint32_t n_rows, int nq) {
    int sms = 0;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || sms <= 0) sms = 1;
    const int groups = (nq + SCAN_WARPS - 1) / SCAN_WARPS;
    int parts = (2 * sms + groups - 1) / groups;
    const uint32_t tiles = (n_rows + 3) / 4;
    if ((uint32_t)parts > tiles) parts = (int)tiles;
    return parts < 1 ? 1 : parts;
}

template <typename T>
static void launch_scan_gemv_batch_t(const void *table, const float *scale, uint32_t n_rows, const float *qhat, int nq,
                                     int slots, uint64_t *partial, int parts, cudaStream_t st) {
    dim3 g(parts, (nq + SCAN_WARPS - 1) / SCAN_WARPS);
    const T *tab = static_cast<const T *>(table);
    switch (slots) {
        case 1: launch_pdl(scan_gemv_batch_kernel<T, 1>, g, dim3(SCAN_THREADS), 0, st, tab, scale, n_rows, qhat, nq, partial); break;
        case 2: launch_pdl(scan_gemv_batch_kernel<T, 2>, g, dim3(SCAN_THREADS), 0, st, tab, scale, n_rows, qhat, nq, partial); break;
        case 4: launch_pdl(scan_gemv_batch_kernel<T, 4>, g, dim3(SCAN_THREADS), 0, st, tab, scale, n_rows, qhat, nq, partial); break;
        default: launch_pdl(scan_gemv_batch_kernel<T, 5>, g, dim3(SCAN_THREADS), 0, st, tab, scale, n_rows, qhat, nq, partial); break;
    }
}

void launch_scan_gemv_batch(int dtype, const void *table, const float *scale, uint32_t n_rows, const float *qhat, int nq,
                            int slots, uint64_t *partial, int parts, cudaStream_t st) {
    if (dtype == ORX_DTYPE_F32)
        launch_scan_gemv_batch_t<float>(table, scale, n_rows, qhat, nq, slots, partial, parts, st);
    else
        launch_scan_gemv_batch_t<__nv_bfloat16>(table, scale, n_rows, qhat, nq, slots, partial, parts, st);
}

template <typename T>
static void launch_scan_gemv_filtered_t(const void *table, const float *scale, uint32_t n_rows,
                                        const uint32_t *allow_bits, const float *qhat, int nq, int slots,
                                        uint64_t *partial, int grid, cudaStream_t st) {
    dim3 g(grid, nq);
    const T *tab = static_cast<const T *>(table);
    switch (slots) {
        case 1: scan_gemv_filtered_kernel<T, 1><<<g, SCAN_THREADS, 0, st>>>(tab, scale, n_rows, allow_bits, qhat, partial); break;
        case 2: scan_gemv_filtered_kernel<T, 2><<<g, SCAN_THREADS, 0, st>>>(tab, scale, n_rows, allow_bits, qhat, partial); break;
        case 4: scan_gemv_filtered_kernel<T, 4><<<g, SCAN_THREADS, 0, st>>>(tab, scale, n_rows, allow_bits, qhat, partial); break;
        default: scan_gemv_filtered_kernel<T, 5><<<g, SCAN_THREADS, 0, st>>>(tab, scale, n_rows, allow_bits, qhat, partial); break;
    }
}

void launch_scan_gemv_filtered(int dtype, const void *table, const float *scale, uint32_t n_rows,
                               const uint32_t *allow_bits, const float *qhat, int nq, int slots,
                               uint64_t *partial, int grid, cudaStream_t st) {
    if (dtype == ORX_DTYPE_F32)
        launch_scan_gemv_filtered_t<float>(table, scale, n_rows, allow_bits, qhat, nq, slots, partial, grid, st);
    else
        launch_scan_gemv_filtered_t<__nv_bfloat16>(table, scale, n_rows, allow_bits, qhat, nq, slots, partial, grid, st);
}

}  // namespace orx
