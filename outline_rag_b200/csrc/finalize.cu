// Query preparation, candidate finalisation (merge + canonical rescore + ordering + proof),
// shard merge, and the exhaustive threshold-collect fallback.
//
// The rescore is what makes the answer bit-exact and independent of scan order: every
// candidate's cosine distance is recomputed in binary64 in the fixed halving-tree order of
// oracle/cosine_topk.py:canon_distance, then candidates are ordered by the SQL contract
// (distance ASC, NaN last, id ASC) of `ORDER BY embedding <=> :q LIMIT :k`
// (reference app/rag.py:85-87 -> langchain-postgres [UPSTREAM]).
#include "scan_common.cuh"
#include "internal.h"

namespace orx {

// --------------------------------------------------------------- prep_queries
// One warp per query: pgvector's input check (NaN/Inf -> error), canonical |q|^2,
// normalised fp32 copy qhat (and its RNE bf16 image for the tcgen05 bf16 scan, and its 15-bit quantisation for the
// scan over an 8-bit image: Q_i = rint(qhat_i / dq), dq = max|qhat_i| / 16383, so |Q_i| <= 16383 and
// |qhat_i - dq Q_i| <= dq / 2 (the division is binary64), i.e. |qhat - dq Q| <= 16 dq <= 9.7662e-4; DESIGN.md section 2).
__global__ void __launch_bounds__(128)
prep_queries_kernel(const float *__restrict__ q_all, int nq, float *__restrict__ q_copy,
                    float *__restrict__ qhat_all, __nv_bfloat16 *__restrict__ qhat16_all,
                    int8_t *__restrict__ qhat8_all, QueryPrep *__restrict__ prep) {
    const int lane = threadIdx.x & 31;
    const int qi = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    pdl_launch_dependents();            // the scan's CTAs may take their SMs now; they wait for this grid before reading qhat
    if (qi >= nq) return;
    const float *q = q_all + (size_t)qi * ORX_DIM;
    float x[32];
    double p[32];
    bool bad = false;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
        x[j] = q[lane + 32 * j];            // may be mapped host memory (zero-copy upload of small batches)
        if (q_copy) q_copy[(size_t)qi * ORX_DIM + lane + 32 * j] = x[j];
        bad |= !isfinite(x[j]);
        p[j] = __dmul_rn((double)x[j], (double)x[j]);
    }
    const double n2q = bcast_lane0(canon_tree_1024(p));
    const bool any_bad = __any_sync(FULL_MASK, bad);
    const bool zero = !(n2q > 0.0);
    const double inv = (any_bad || zero) ? 0.0 : __ddiv_rn(1.0, __dsqrt_rn(n2q));
    float amax = 0.f;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
        const float h = (any_bad || zero) ? 0.f : __double2float_rn(__dmul_rn((double)x[j], inv));
        x[j] = h;
        amax = fmaxf(amax, fabsf(h));
        qhat_all[(size_t)qi * ORX_DIM + lane + 32 * j] = h;
        if (qhat16_all) qhat16_all[(size_t)qi * ORX_DIM + lane + 32 * j] = __float2bfloat16_rn(h);
    }
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) amax = fmaxf(amax, __shfl_xor_sync(FULL_MASK, amax, d));
    const float dq = __fdiv_rn(amax, 16383.f);
    if (qhat8_all) {
        int8_t *q8 = qhat8_all + (size_t)qi * 2 * ORX_DIM;
#pragma unroll
        for (int j = 0; j < 32; ++j) {
            const int Q = dq > 0.f ? __double2int_rn(__ddiv_rn((double)x[j], (double)dq)) : 0;
            q8[lane + 32 * j] = (int8_t)(Q >> 7);                  // arithmetic shift: floor(Q / 128) in [-128, 127]
            q8[ORX_DIM + lane + 32 * j] = (int8_t)(Q & 127);       // Q - 128 (Q >> 7) in [0, 127]
        }
    }
    if (lane == 0) {
        prep[qi].n2q = n2q;
        prep[qi].nonfinite = any_bad ? 1 : 0;
        prep[qi].zero = zero ? 1 : 0;
        prep[qi].dq8 = dq;
    }
}

void launch_prep_queries(const float *q, int nq, float *q_copy, float *qhat, void *qhat_bf16, int8_t *qhat8,
                         QueryPrep *prep, cudaStream_t st) {
    if (nq <= 0) return;
    prep_queries_kernel<<<(nq + 3) / 4, 128, 0, st>>>(q, nq, q_copy, qhat,
                                                      static_cast<__nv_bfloat16 *>(qhat_bf16), qhat8, prep);
}

__global__ void flags_from_prep_kernel(const QueryPrep *__restrict__ prep, int nq, int *__restrict__ flags) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < nq) flags[j] = (prep[j].nonfinite ? 2 : 0) | (prep[j].zero ? 4 : 0);
}
__global__ void fill_flags_kernel(int *__restrict__ flags, int nq, int value) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < nq) flags[j] = value;
}
void launch_fill_flags(int *flags, int nq, int value, cudaStream_t st) {
    if (nq > 0) fill_flags_kernel<<<(nq + 127) / 128, 128, 0, st>>>(flags, nq, value);
}
void launch_flags_from_prep(const QueryPrep *prep, int nq, int *flags, cudaStream_t st) {
    if (nq > 0) flags_from_prep_kernel<<<(nq + 127) / 128, 128, 0, st>>>(prep, nq, flags);
}

// ------------------------------------------------------------------- finalize
// One CTA of 16 warps per query (512 threads: the binary64 rescore needs ~100 registers).
//   1. the query's top-K candidates by fast score (K = 32*S) out of the scan's per-CTA lists:
//      1a sorted lists (GEMV scan): the K-th largest list HEAD is a lower bound of the global K-th best key and only
//         the K lists whose head reaches it can hold keys above it -- K coalesced list reads, one round of loads;
//      1c unsorted lists that fit shared memory (tcgen05 scan): bitonic sort;  1b generic: warp top-K + tree merge;
//   2. canonical binary64 rescore, one warp per candidate, the query staged in shared memory, the next round's rows
//      prefetched into L2 while this round's are summed;
//   3. rank by (distance ASC, NaN last, id ASC) by counting;
//   4. completeness proof -> flag (bit 0: unproven, bit 1: non-finite query, bit 2: zero query);
//   5. results go where the search wants them -- caller / mapped host arrays, or (row-sharded search) straight into
//      the gather buffers of the peer GPUs with P2P stores; the search's last CTA raises the arrival words / the
//      host's completion word (internal.h PublishArgs / DoneArgs), so no publish kernel and no stream sync follow.
constexpr int FIN_THREADS = 512;
constexpr int FIN_WARPS = FIN_THREADS / 32;
constexpr int FIN_SURV = 256;          // survivors of the head-threshold filter (fast path)
constexpr int FIN_SORT_MAX = 2048;     // keys the shared-memory bitonic sort takes (unsorted-list path)

__device__ __forceinline__ void prefetch_l2(const void *p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

// canonical binary64 dot of a stored row with the query held in shared memory (same tree as warp_canon_dot)
template <typename T>
__device__ __forceinline__ double warp_canon_dot_sq(const T *row, const float *s_q, int lane) {
    double p[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) {
        const int e = lane + 32 * j;
        p[j] = __dmul_rn((double)row_elem<T>(row, e), (double)s_q[e]);
    }
    return bcast_lane0(canon_tree_1024(p));
}

template <typename T, int S>
__global__ void __launch_bounds__(FIN_THREADS)
finalize_kernel(const T *__restrict__ table, const double *__restrict__ n2,
                const orx_id *__restrict__ row_ids, const float *__restrict__ q_all,
                const QueryPrep *__restrict__ prep, const uint64_t *__restrict__ partial_all,
                int nparts, int k, uint32_t n_rows, double eps, const ResultOut out, int q_base,
                const PublishArgs pub, const DoneArgs done, const float *__restrict__ floor_all,
                int sorted_lists, const uint32_t *__restrict__ covered) {
    constexpr int K = 32 * S;
    __shared__ uint64_t s_keys[FIN_WARPS][K];
    __shared__ double s_dist[K];
    __shared__ uint64_t s_hi[K], s_lo[K];
    __shared__ double s_kth;
    __shared__ int s_valid;

    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int qi = blockIdx.x;
    const uint64_t *partial = partial_all + (size_t)qi * nparts * K;
    if (threadIdx.x == 0) {
        s_kth = __longlong_as_double(0x7ff8000000000000ll);
        s_valid = 0;
    }
    pdl_wait();                         // the scan that filled `partial` has completed (no-op for a plain launch)
    pdl_launch_dependents();            // a merge_wait launched behind this grid may take its SM now and start polling

    // 1. the query's top-K candidates by fast score.
    __shared__ uint64_t s_surv[FIN_SURV];
    __shared__ uint64_t s_thresh;
    __shared__ int s_nsurv;
    __shared__ int s_sel[K];
    uint64_t *s_flat = &s_keys[0][0];                   // FIN_WARPS*K >= 512 words of scratch
    bool fast = sorted_lists && nparts >= K && nparts <= FIN_THREADS;
    if (fast) {
        if (threadIdx.x == 0) {
            s_nsurv = 0;
            s_thresh = 0ull;
        }
        const uint64_t head = threadIdx.x < nparts ? partial[(size_t)threadIdx.x * K] : 0ull;
        s_flat[threadIdx.x] = head;
        __syncthreads();
        if (threadIdx.x < nparts && head != 0ull) {
            int rank = 0;
            for (int i = 0; i < nparts; ++i) rank += (s_flat[i] > head);
            if (rank < K) s_sel[rank] = threadIdx.x;    // heads are distinct rows: ranks 0..K-1 are taken exactly once
            if (rank == K - 1) s_thresh = head;
        }
        __syncthreads();
        const uint64_t T = s_thresh;
        if (T == 0ull) fast = false;                    // fewer than K non-empty lists
        else {
            // every key >= T lives in one of the K selected lists; each warp reads whole lists, coalesced
            constexpr int LISTS_PER_WARP = (K + FIN_WARPS - 1) / FIN_WARPS;
#pragma unroll 2
            for (int u = 0; u < LISTS_PER_WARP; ++u) {
                const int li = warp + u * FIN_WARPS;
                const uint64_t *src = partial + (size_t)s_sel[li < K ? li : 0] * K;
                uint64_t mine[S];
#pragma unroll
                for (int sl = 0; sl < S; ++sl) mine[sl] = li < K ? src[sl * 32 + lane] : 0ull;
#pragma unroll
                for (int sl = 0; sl < S; ++sl) {
                    const bool keep = mine[sl] >= T && mine[sl] != 0ull;
                    const unsigned m = __ballot_sync(FULL_MASK, keep);
                    if (m == 0u) continue;
                    int base = 0;
                    if (lane == 0) base = atomicAdd(&s_nsurv, __popc(m));
                    base = __shfl_sync(FULL_MASK, base, 0);
                    const int pos = base + __popc(m & ((1u << lane) - 1u));
                    if (keep && pos < FIN_SURV) s_surv[pos] = mine[sl];
                }
            }
            __syncthreads();
            const int ns = s_nsurv;
            if (ns > FIN_SURV) fast = false;            // a flood of ties
            else {
                __syncthreads();
                if (threadIdx.x < K) s_flat[threadIdx.x] = 0ull;
                __syncthreads();
                if (threadIdx.x < ns) {
                    const uint64_t me = s_surv[threadIdx.x];
                    int rank = 0;
                    for (int i = 0; i < ns; ++i) rank += (s_surv[i] > me);
                    if (rank < K) s_flat[rank] = me;
                }
                __syncthreads();
            }
        }
    }
    __shared__ uint64_t s_all[FIN_SORT_MAX];
    const int total_keys = nparts * K;
    if (!fast && total_keys <= FIN_SORT_MAX) {
        // 1c (unsorted lists that fit shared memory, i.e. the tcgen05 scan at large batches): the lists are mostly
        //     EMPTY slots (a list holds only the rows that passed its CTA's running threshold), so the non-empty keys
        //     are compacted first and the bitonic sort runs over the next power of two of THEIR number (typically 256-512
        //     instead of 2048 slots); descending; the first K are the query's candidates.
        __shared__ int s_nkeys;
        if (threadIdx.x == 0) s_nkeys = 0;
        __syncthreads();
        for (int i0 = 0; i0 < total_keys; i0 += FIN_THREADS) {
            const int i = i0 + threadIdx.x;
            const uint64_t key = i < total_keys ? partial[i] : 0ull;
            const unsigned m = __ballot_sync(FULL_MASK, key != 0ull);
            int base = 0;
            if (lane == 0 && m) base = atomicAdd(&s_nkeys, __popc(m));
            base = __shfl_sync(FULL_MASK, base, 0);
            if (key != 0ull) s_all[base + __popc(m & ((1u << lane) - 1u))] = key;
        }
        __syncthreads();
        const int nkeys = s_nkeys;
        int n = 64;
        while (n < nkeys || n < K) n <<= 1;               // the first K sorted entries are read below
        for (int i = nkeys + threadIdx.x; i < n; i += FIN_THREADS) s_all[i] = 0ull;
        __syncthreads();
        for (int size = 2; size <= n; size <<= 1) {
            for (int stride = size >> 1; stride > 0; stride >>= 1) {
                for (int i = threadIdx.x; i < (n >> 1); i += FIN_THREADS) {
                    const int lo = 2 * i - (i & (stride - 1));          // index with bit `stride` clear
                    const int hi = lo + stride;
                    const uint64_t a = s_all[lo], b = s_all[hi];
                    const bool desc = (lo & size) == 0;                // descending overall
                    if ((a < b) == desc) {
                        s_all[lo] = b;
                        s_all[hi] = a;
                    }
                }
                __syncthreads();
            }
        }
        if (threadIdx.x < K) s_keys[0][threadIdx.x] = s_all[threadIdx.x];
        __syncthreads();
        fast = true;
    }
    if (!fast) {
        // 1b (generic): each warp folds lists warp, warp+16, ... into a register-resident sorted
        //     top-K (offer_lanes takes unsorted input), then a tree merge through shared memory.
        __syncthreads();
        WarpTopK<S> top;
        top.init();
        for (int p = warp; p < nparts; p += FIN_WARPS) {
#pragma unroll
            for (int s = 0; s < S; ++s) top.offer_lanes(partial[(size_t)p * K + s * 32 + lane], lane);
        }
        top.store(s_keys[warp], lane);
        __syncthreads();
#pragma unroll 1
        for (int half = FIN_WARPS / 2; half >= 1; half >>= 1) {
            if (warp < half) {
#pragma unroll
                for (int s = 0; s < S; ++s) top.offer_lanes(s_keys[warp + half][s * 32 + lane], lane);
                top.store(s_keys[warp], lane);
            }
            __syncthreads();
        }
    }
    const uint64_t *s_cand = s_keys[0];

    // 2. canonical rescore, one warp per candidate.  A candidate whose fast score is more than 2*eps (+ slack) below
    //    the k-th best FAST score cannot reach the top-k (|fast - cosine| <= eps for both), so it is not rescored; the
    //    proof below accounts for the ones left out through `cut`.  With k = 12 of K = 32 candidates that is one
    //    round of 16 warps instead of two.
    __shared__ unsigned char s_ok[K];
    float *s_q = reinterpret_cast<float *>(s_all);          // the bitonic scratch is free now: stage the query (4 KB)
    const float *q = q_all + (size_t)qi * ORX_DIM;
    __syncthreads();
    for (int e = threadIdx.x; e < ORX_DIM; e += FIN_THREADS) s_q[e] = q[e];
    const double n2q = prep[qi].n2q;
    float cut = __int_as_float(0xff800000);               // -inf: nothing is cut
    {
        // s_cand is sorted by key, descending: untrusted (ORD_ALWAYS) rows first, then by fast score;
        // the cut hangs on the k-th best REGULAR candidate
        int n_always = 0;
        for (int c = 0; c < K; ++c) n_always += (key_ord(s_cand[c]) == ORD_ALWAYS);
        const int kth = n_always + k - 1;
        const uint32_t ok_ord = kth < K ? key_ord(s_cand[kth]) : 0u;
        if (ok_ord != 0u) cut = ord_to_float(ok_ord) - (float)(2.0 * eps + 1e-6);
    }
    auto skipped = [&](uint64_t key) {
        return key == 0ull || (key_ord(key) != ORD_ALWAYS && ord_to_float(key_ord(key)) <= cut);
    };
    __syncthreads();
    // candidates are sorted by fast score, so the ones to rescore are a prefix (plus nothing after the first cut one)
    for (int c = warp; c < K; c += FIN_WARPS) {
        const uint64_t key = s_cand[c];
        // the row this warp takes in the NEXT round: pull its 32 lines towards L2 now (one line per lane)
        if (c + FIN_WARPS < K) {
            const uint64_t nk = s_cand[c + FIN_WARPS];
            if (!skipped(nk))
                prefetch_l2(reinterpret_cast<const char *>(table + (size_t)key_row(nk) * ORX_DIM) + lane * (ORX_DIM * sizeof(T) / 32));
        }
        if (skipped(key)) {                   // empty or cut: sorts after everything, never output
            if (lane == 0) {
                s_ok[c] = 0;
                s_dist[c] = __longlong_as_double(0x7ff8000000000000ll);
                s_hi[c] = ~0ull;
                s_lo[c] = ~0ull;
            }
            continue;
        }
        const uint32_t row = key_row(key);
        const double n2x = n2[row];                       // issued before the row itself: one DRAM round trip
        const orx_id id = row_ids[row];
        const double dot = warp_canon_dot_sq<T>(table + (size_t)row * ORX_DIM, s_q, lane);
        if (lane == 0) {
            s_ok[c] = 1;
            s_dist[c] = canon_dist(dot, n2x, n2q);
            s_hi[c] = id.hi;
            s_lo[c] = id.lo;
            atomicAdd(&s_valid, 1);
        }
    }
    __syncthreads();

    // 3. order by (distance ASC, NaN last, id ASC): rank by counting; 5. write where the search wants the results
    const int t = threadIdx.x;
    const size_t qo = (size_t)(q_base + qi);
    const int n_out = pub.n_targets > 0 ? pub.n_targets : 1;
    const int count = min(k, s_valid);
    if (t < K && s_ok[t]) {
        int rank = 0;
        const double d = s_dist[t];
        const uint64_t hi = s_hi[t], lo = s_lo[t];
        for (int c = 0; c < K; ++c)
            rank += (c != t && s_ok[c] && sorts_before(s_dist[c], s_hi[c], s_lo[c], d, hi, lo));
        if (rank < k) {
            for (int o = 0; o < n_out; ++o) {
                char *b = pub.n_targets > 0 ? pub.slot[o] : nullptr;
                orx_id *oi = b ? reinterpret_cast<orx_id *>(b) : out.ids;
                double *od = b ? reinterpret_cast<double *>(b + pub.dist_off) : out.dist;
                oi[qo * k + rank].hi = hi;
                oi[qo * k + rank].lo = lo;
                od[qo * k + rank] = d;
            }
        }
        if (rank == count - 1) s_kth = d;
    }
    if (t >= count && t < k) {
        for (int o = 0; o < n_out; ++o) {
            char *b = pub.n_targets > 0 ? pub.slot[o] : nullptr;
            orx_id *oi = b ? reinterpret_cast<orx_id *>(b) : out.ids;
            double *od = b ? reinterpret_cast<double *>(b + pub.dist_off) : out.dist;
            oi[qo * k + t].hi = 0ull;
            oi[qo * k + t].lo = 0ull;
            od[qo * k + t] = __longlong_as_double(0x7ff8000000000000ll);
        }
    }
    __syncthreads();

    // 4. completeness proof: no row outside the candidate list can sort before the k-th.
    //    GEMV scan: the lists are each CTA's true top-K, so every outside row has fast score
    //    <= the merged list's K-th.  tcgen05 scan (floor_all != null): the lists hold every row
    //    above the CTA's running threshold; outside rows are <= max(final thresholds, merged K-th).
    if (t == 0) {
        int flag = 1;
        const bool coarse = floor_all != nullptr;
        if (!coarse && n_rows <= (uint32_t)K) {
            flag = 0;                                  // every live row is a candidate
        } else if (!prep[qi].zero && !prep[qi].nonfinite) {
            const uint32_t ord_last = key_ord(s_cand[K - 1]);   // K-th best fast score
            const double dk = s_kth;
            if (ord_last == ORD_ALWAYS) flag = 1;      // list flooded by untrusted rows
            else if (dk != dk) flag = 1;               // k-th is NaN: id order among NaN rows unknown
            else if (coarse) {
                // zero-norm rows are never collected by the coarse pass: too few finite rows -> exact scan
                if (count == k) {
                    double bound = ord_last == ORD_NAN ? -1.0e30 : (double)ord_to_float(ord_last);
                    if ((double)cut > bound) bound = (double)cut;      // candidates that were not rescored
                    for (int p = 0; p < nparts; ++p) {
                        const double f = (double)floor_all[(size_t)qi * nparts + p];
                        if (!(f <= bound)) bound = f;  // also catches NaN / +inf (overflowed list)
                    }
                    bound += eps;
                    flag = ((1.0 - dk) > bound && dk < 2.0) ? 0 : 1;
                }
            } else if (ord_last == ORD_NAN && !((double)cut > -1.0e30)) flag = 0;  // everything outside is a NaN row
            else {
                // rows outside the list have fast score <= the list's K-th; listed rows that were not rescored have
                // fast score <= cut
                double bound = ord_last == ORD_NAN ? -1.0e30 : (double)ord_to_float(ord_last);
                if ((double)cut > bound) bound = (double)cut;
                bound += eps;
                flag = ((1.0 - dk) > bound && dk < 2.0) ? 0 : 1;
            }
        }
        if (covered != nullptr && covered[qi] != n_rows) flag |= 1;     // a lap missed or repeated rows: prove nothing
        flag |= (prep[qi].nonfinite ? 2 : 0) | (prep[qi].zero ? 4 : 0);
        for (int o = 0; o < n_out; ++o) {
            char *b = pub.n_targets > 0 ? pub.slot[o] : nullptr;
            int *oc = b ? reinterpret_cast<int *>(b + pub.counts_off) : out.counts;
            int *of = b ? reinterpret_cast<int *>(b + pub.flags_off) : out.flags;
            oc[qo] = count;
            of[qo] = flag;
        }
    }

    // 5. completion: every thread's result stores are performed system-wide before this CTA counts itself; the
    //    search's last CTA raises the arrival words on the targets / the host's completion word.
    if (done.counter != nullptr) {
        __threadfence_system();
        __syncthreads();
        if (t == 0) {
            bool last = done.total == 1u;                  // a single-query search has one CTA: nothing to count
            if (!last) {
                const unsigned int old = atomicAdd(done.counter, 1u);
                if (old + 1u == done.total) {
                    *done.counter = 0u;
                    __threadfence_system();
                    last = true;
                }
            }
            if (last) {
                for (int o = 0; o < pub.n_targets; ++o) *reinterpret_cast<volatile uint32_t *>(pub.flag[o]) = pub.seq;
                if (done.done_host != nullptr) *reinterpret_cast<volatile uint32_t *>(done.done_host) = done.token;
            }
        }
    }
}

template <typename T>
static void launch_finalize_t(const void *table, const double *n2, const orx_id *row_ids, const float *q,
                              const QueryPrep *prep, const uint64_t *partial, int nparts, int slots, int nq,
                              int k, uint32_t n_rows, double eps, const ResultOut &out, int q_base,
                              const PublishArgs &pub, const DoneArgs &done, cudaStream_t st, const float *floor,
                              const uint32_t *covered) {
    const T *tab = static_cast<const T *>(table);
#define ORX_FIN(S_)                                                                                          \
    launch_pdl(finalize_kernel<T, S_>, dim3(nq), dim3(FIN_THREADS), 0, st, tab, n2, row_ids, q, prep, partial, nparts, k, \
               n_rows, eps, out, q_base, pub, done, floor, (int)(floor == nullptr), covered)
    switch (slots) {
        case 1: ORX_FIN(1); break;
        case 2: ORX_FIN(2); break;
        case 4: ORX_FIN(4); break;
        default: ORX_FIN(5); break;
    }
#undef ORX_FIN
}

void launch_finalize(int dtype, const void *table, const double *n2, const orx_id *row_ids,
                     const float *q, const QueryPrep *prep, const uint64_t *partial, int nparts,
                     int slots, int nq, int k, uint32_t n_rows, double eps, const ResultOut &out, int q_base,
                     const PublishArgs &pub, const DoneArgs &done, cudaStream_t st, const float *floor,
                     const uint32_t *covered) {
    if (nq <= 0) return;
    if (dtype == ORX_DTYPE_F32)
        launch_finalize_t<float>(table, n2, row_ids, q, prep, partial, nparts, slots, nq, k, n_rows, eps,
                                 out, q_base, pub, done, st, floor, covered);
    else
        launch_finalize_t<__nv_bfloat16>(table, n2, row_ids, q, prep, partial, nparts, slots, nq, k, n_rows,
                                         eps, out, q_base, pub, done, st, floor, covered);
}

__global__ void signal_done_kernel(DoneArgs done) {
    __threadfence_system();
    if (done.done_host != nullptr) *reinterpret_cast<volatile uint32_t *>(done.done_host) = done.token;
}
void launch_signal_done(const DoneArgs &done, cudaStream_t st) { signal_done_kernel<<<1, 1, 0, st>>>(done); }

// ----------------------------------------------------------------- merge_topk
// The on-device step after the allgather of the row-sharded path: n_lists shard results
// [n_lists][nq][k] -> global top-k per query, same ordering contract.
constexpr int MERGE_MAX = 1024;

__global__ void __launch_bounds__(256)
merge_topk_kernel(int n_lists, int nq, int k, const char *__restrict__ ids_base,
                  const char *__restrict__ dist_base, const char *__restrict__ counts_base,
                  size_t ids_stride, size_t dist_stride, size_t counts_stride,
                  orx_id *__restrict__ out_ids, double *__restrict__ out_dist,
                  int *__restrict__ out_counts) {
    __shared__ double s_d[MERGE_MAX];
    __shared__ uint64_t s_hi[MERGE_MAX], s_lo[MERGE_MAX];
    __shared__ unsigned char s_ok[MERGE_MAX];
    __shared__ int s_valid;
    const int qi = blockIdx.x;
    const int total = n_lists * k;
    if (threadIdx.x == 0) s_valid = 0;
    __syncthreads();
    int mine = 0;
    for (int e = threadIdx.x; e < total; e += blockDim.x) {
        const int l = e / k, r = e % k;
        // list l lives at base + l * stride (bytes): separate arrays or one gathered block per rank
        const orx_id *ids = reinterpret_cast<const orx_id *>(ids_base + (size_t)l * ids_stride);
        const double *dist = reinterpret_cast<const double *>(dist_base + (size_t)l * dist_stride);
        const int *counts = reinterpret_cast<const int *>(counts_base + (size_t)l * counts_stride);
        const size_t src = (size_t)qi * k + r;
        const bool ok = r < counts[qi];
        s_ok[e] = ok;
        s_d[e] = dist[src];
        s_hi[e] = ids[src].hi;
        s_lo[e] = ids[src].lo;
        mine += ok;
    }
    atomicAdd(&s_valid, mine);
    __syncthreads();
    const int count = min(k, s_valid);
    for (int e = threadIdx.x; e < total; e += blockDim.x) {
        if (!s_ok[e]) continue;
        int rank = 0;
        for (int c = 0; c < total; ++c)
            rank += (c != e && s_ok[c] &&
                     (sorts_before(s_d[c], s_hi[c], s_lo[c], s_d[e], s_hi[e], s_lo[e]) ||
                      // identical (distance, id) in two lists (cannot happen with disjoint
                      // shards): keep a strict total order by list position
                      (c < e && s_d[c] == s_d[e] && s_hi[c] == s_hi[e] && s_lo[c] == s_lo[e])));
        if (rank < k) {
            out_ids[(size_t)qi * k + rank].hi = s_hi[e];
            out_ids[(size_t)qi * k + rank].lo = s_lo[e];
            out_dist[(size_t)qi * k + rank] = s_d[e];
        }
    }
    for (int r = count + threadIdx.x; r < k; r += blockDim.x) {
        out_ids[(size_t)qi * k + r].hi = 0ull;
        out_ids[(size_t)qi * k + r].lo = 0ull;
        out_dist[(size_t)qi * k + r] = __longlong_as_double(0x7ff8000000000000ll);
    }
    if (threadIdx.x == 0) out_counts[qi] = count;
}

void launch_merge_topk(int n_lists, int nq, int k, const orx_id *ids, const double *dist,
                       const int *counts, size_t list_stride_bytes, orx_id *out_ids, double *out_dist,
                       int *out_counts, cudaStream_t st) {
    if (nq <= 0) return;
    const size_t si = list_stride_bytes ? list_stride_bytes : (size_t)nq * k * sizeof(orx_id);
    const size_t sd = list_stride_bytes ? list_stride_bytes : (size_t)nq * k * sizeof(double);
    const size_t sc = list_stride_bytes ? list_stride_bytes : (size_t)nq * sizeof(int);
    merge_topk_kernel<<<nq, 256, 0, st>>>(n_lists, nq, k, reinterpret_cast<const char *>(ids),
                                          reinterpret_cast<const char *>(dist),
                                          reinterpret_cast<const char *>(counts), si, sd, sc, out_ids,
                                          out_dist, out_counts);
}

// -------------------------------------------------- exhaustive fallback (rare path)
// collect: every row whose fast score could still reach `fast_floor` (or every row).
// DUMP (diagnostic instantiation behind orx_debug_fast_scores): query blockIdx.y of a batch, and instead of collecting,
// every row's fast score -- the `dot * scale` that score_ord keys on -- is written to dump[row * nq + query], so that a
// test can MEASURE max |fast - cosine| against the eps of the GEMV scans (same load / FMA / butterfly sequence).
template <typename T, bool DUMP = false>
__global__ void __launch_bounds__(256)
collect_kernel(const T *__restrict__ table, const float *__restrict__ scale, uint32_t n_rows,
               const float *__restrict__ qhat, float fast_floor, int collect_all,
               uint32_t *__restrict__ list, uint32_t *__restrict__ count, float *__restrict__ dump = nullptr) {
    const int lane = threadIdx.x & 31;
    const uint32_t gw = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const uint32_t n_gw = gridDim.x * (blockDim.x >> 5);
    float4 qv[8];
    load_q_slice<T>(qhat + (DUMP ? (size_t)blockIdx.y * ORX_DIM : 0), lane, qv);
    const uint4 *tab = reinterpret_cast<const uint4 *>(table);
    for (uint32_t row = gw; row < n_rows; row += n_gw) {
        if constexpr (DUMP) {
            uint4 v[RowVec<T>::NV];
            load_row_vecs<T>(tab, row, lane, v);
            const float acc = warp_row_dot<T>(v, qv);
            if (lane == 0) dump[(size_t)row * gridDim.y + blockIdx.y] = acc * __ldg(scale + row);
            continue;
        }
        bool take = collect_all != 0;
        if (!take) {
            uint4 v[RowVec<T>::NV];
            load_row_vecs<T>(tab, row, lane, v);
            const float acc = warp_row_dot<T>(v, qv);
            const uint32_t ord = score_ord(acc, __ldg(scale + row));
            // NaN rows can only matter when fewer than k finite rows exist; the caller
            // passes collect_all in that case.
            take = (ord == ORD_ALWAYS) || (ord != ORD_NAN && ord_to_float(ord) >= fast_floor);
        }
        if (take && lane == 0) list[atomicAdd(count, 1u)] = row;
    }
}

void launch_collect(int dtype, const void *table, const float *scale, uint32_t n_rows,
                    const float *qhat, float fast_floor, int collect_all, uint32_t *list,
                    uint32_t *count, cudaStream_t st) {
    if (n_rows == 0) return;
    const int grid = device_sms() * 4;
    if (dtype == ORX_DTYPE_F32)
        collect_kernel<float><<<grid, 256, 0, st>>>(static_cast<const float *>(table), scale, n_rows,
                                                    qhat, fast_floor, collect_all, list, count);
    else
        collect_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>(
            static_cast<const __nv_bfloat16 *>(table), scale, n_rows, qhat, fast_floor, collect_all,
            list, count);
}

void launch_dump_fast_scores(int dtype, const void *table, const float *scale, uint32_t n_rows, const float *qhat,
                             int nq, float *out, cudaStream_t st) {
    if (n_rows == 0 || nq <= 0) return;
    const dim3 grid(device_sms() * 4, nq);
    if (dtype == ORX_DTYPE_F32)
        collect_kernel<float, true><<<grid, 256, 0, st>>>(static_cast<const float *>(table), scale, n_rows, qhat, 0.f, 0,
                                                          nullptr, nullptr, out);
    else
        collect_kernel<__nv_bfloat16, true><<<grid, 256, 0, st>>>(static_cast<const __nv_bfloat16 *>(table), scale,
                                                                  n_rows, qhat, 0.f, 0, nullptr, nullptr, out);
}

template <typename T>
__global__ void __launch_bounds__(256)
rescore_list_kernel(const T *__restrict__ table, const double *__restrict__ n2,
                    const float *__restrict__ q, const QueryPrep *__restrict__ prep,
                    const uint32_t *__restrict__ list, const uint32_t *__restrict__ count,
                    double *__restrict__ dist_out) {
    const int lane = threadIdx.x & 31;
    const uint32_t gw = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const uint32_t n_gw = gridDim.x * (blockDim.x >> 5);
    const uint32_t m = *count;
    const double n2q = prep->n2q;
    for (uint32_t i = gw; i < m; i += n_gw) {
        const uint32_t row = list[i];
        const double dot = warp_canon_dot<T>(table + (size_t)row * ORX_DIM, q, lane);
        if (lane == 0) dist_out[i] = canon_dist(dot, n2[row], n2q);
    }
}

void launch_rescore_list(int dtype, const void *table, const double *n2, const orx_id *,
                         const float *q, const QueryPrep *prep, const uint32_t *list,
                         const uint32_t *count, double *dist_out, cudaStream_t st) {
    const int grid = device_sms() * 2;
    if (dtype == ORX_DTYPE_F32)
        rescore_list_kernel<float><<<grid, 256, 0, st>>>(static_cast<const float *>(table), n2, q,
                                                         prep, list, count, dist_out);
    else
        rescore_list_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>(
            static_cast<const __nv_bfloat16 *>(table), n2, q, prep, list, count, dist_out);
}

// select: k rounds of "smallest entry that sorts strictly after the previous winner".
__global__ void __launch_bounds__(1024)
select_list_kernel(const orx_id *__restrict__ row_ids, const uint32_t *__restrict__ list,
                   const uint32_t *__restrict__ count, const double *__restrict__ dist, int k,
                   orx_id *__restrict__ out_ids, double *__restrict__ out_dist,
                   int *__restrict__ out_count) {
    __shared__ double s_d[1024];
    __shared__ uint64_t s_hi[1024], s_lo[1024];
    __shared__ int s_has[1024];
    const uint32_t m = *count;
    const int t = threadIdx.x;
    double pd = 0.0;
    uint64_t phi = 0, plo = 0;
    bool have_prev = false;
    int found = 0;
    for (int r = 0; r < k; ++r) {
        double bd = 0.0;
        uint64_t bhi = 0, blo = 0;
        bool has = false;
        for (uint32_t i = t; i < m; i += blockDim.x) {
            const double d = dist[i];
            const orx_id id = row_ids[list[i]];
            if (have_prev && !sorts_before(pd, phi, plo, d, id.hi, id.lo)) continue;
            if (!has || sorts_before(d, id.hi, id.lo, bd, bhi, blo)) {
                has = true; bd = d; bhi = id.hi; blo = id.lo;
            }
        }
        s_d[t] = bd; s_hi[t] = bhi; s_lo[t] = blo; s_has[t] = has;
        __syncthreads();
        for (int off = 512; off >= 1; off >>= 1) {
            if (t < off && s_has[t + off] &&
                (!s_has[t] || sorts_before(s_d[t + off], s_hi[t + off], s_lo[t + off], s_d[t], s_hi[t], s_lo[t]))) {
                s_d[t] = s_d[t + off]; s_hi[t] = s_hi[t + off]; s_lo[t] = s_lo[t + off]; s_has[t] = 1;
            }
            __syncthreads();
        }
        const bool any = s_has[0];
        pd = s_d[0]; phi = s_hi[0]; plo = s_lo[0];
        __syncthreads();
        if (!any) break;
        have_prev = true;
        if (t == 0) {
            out_ids[r].hi = phi; out_ids[r].lo = plo; out_dist[r] = pd;
        }
        ++found;
    }
    if (t == 0) {
        for (int r = found; r < k; ++r) {
            out_ids[r].hi = 0; out_ids[r].lo = 0;
            out_dist[r] = __longlong_as_double(0x7ff8000000000000ll);
        }
        *out_count = found;
    }
}

void launch_select_list(const orx_id *row_ids, const uint32_t *list, const uint32_t *count,
                        const double *dist, int k, orx_id *out_ids, double *out_dist, int *out_count,
                        cudaStream_t st) {
    select_list_kernel<<<1, 1024, 0, st>>>(row_ids, list, count, dist, k, out_ids, out_dist, out_count);
}

}  // namespace orx
