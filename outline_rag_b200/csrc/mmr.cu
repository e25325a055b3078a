// Exact maximal-marginal-relevance selection (orx_search_mmr*, DESIGN.md section 2 "MMR").
//
// One CTA per query.  Input: the query's exact top-fetch_k candidates in contract order (distance ASC, NaN last,
// id ASC) as a gathered fp32 matrix [fetch_k, 1024] (the rows AS STORED: verbatim fp32, or the exact fp32 image of a
// bf16 row), their canonical query distances and their count m.  Output: the positions of the min(k, m) picks in
// selection order.
//
//   s_q[p]     = 1 - d[p]                                            (binary64)
//   s_dd(p, r) = clamp(canon_dot(x_p, x_r) / sqrt(n2_p * n2_r), -1, 1)  (halving tree, IEEE div / sqrt / mul)
//   red[p]     = max over picked r of s_dd(p, r)                     (NaN propagates)
//   score[p]   = lambda * s_q[p] - (1 - lambda) * red[p]             (no contraction: __dmul_rn / __dsub_rn)
// Pick 0 first; then the largest score, the lowest position on ties; a NaN score (zero-norm row, zero query) only
// when no finite score is left, in position order.  Each step computes s_dd between the row just picked and every
// row still available -- (k-1)*m canonical dots per query, never the Gram matrix.
#include "scan_common.cuh"
#include "internal.h"

namespace orx {

constexpr int MMR_THREADS = 256;
constexpr int MMR_WARPS = MMR_THREADS / 32;

// (score, position) a is a better pick than b: larger score; NaN below every number; lowest position on ties
__device__ __forceinline__ bool mmr_better(double sa, int pa, double sb, int pb) {
    if (pb < 0) return pa >= 0;
    if (pa < 0) return false;
    const bool na = sa != sa, nb = sb != sb;
    if (na != nb) return nb;
    if (!na && sa != sb) return sa > sb;
    return pa < pb;
}

__global__ void __launch_bounds__(MMR_THREADS)
mmr_select_kernel(const float *__restrict__ rows, const double *__restrict__ dist, const int *__restrict__ counts,
                  int fetch_k, int k, double lam, int *__restrict__ sel) {
    __shared__ float s_x[ORX_DIM];                 // the row picked last
    __shared__ double s_n2[ORX_MAX_K], s_sq[ORX_MAX_K], s_red[ORX_MAX_K];
    __shared__ int s_avail[ORX_MAX_K];
    __shared__ double s_best[MMR_WARPS];
    __shared__ int s_bestp[MMR_WARPS];
    __shared__ int s_pick;

    const int qi = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int m = min(counts[qi], fetch_k);
    const int n_out = min(k, m);
    const float *X = rows + (size_t)qi * fetch_k * ORX_DIM;
    int *out = sel + (size_t)qi * k;
    for (int t = n_out + tid; t < k; t += MMR_THREADS) out[t] = -1;
    if (n_out == 0) return;

    // canonical |x|^2 of every candidate as stored (bit-identical to the table's n2 column: same tree, exact products)
    for (int p = warp; p < m; p += MMR_WARPS) {
        const double n2 = warp_canon_dot<float>(X + (size_t)p * ORX_DIM, X + (size_t)p * ORX_DIM, lane);
        if (lane == 0) {
            s_n2[p] = n2;
            s_sq[p] = __dsub_rn(1.0, dist[(size_t)qi * fetch_k + p]);
            s_red[p] = -INFINITY;
            s_avail[p] = p != 0;
        }
    }
    if (tid == 0) {
        out[0] = 0;
        s_pick = 0;
    }
    const double one_minus_lam = __dsub_rn(1.0, lam);
    for (int t = 1; t < n_out; ++t) {
        __syncthreads();                            // s_pick, s_avail, s_n2 of the previous step are visible
        const int r = s_pick;
        const float4 *src = reinterpret_cast<const float4 *>(X + (size_t)r * ORX_DIM);
        for (int e = tid; e < ORX_DIM / 4; e += MMR_THREADS) reinterpret_cast<float4 *>(s_x)[e] = src[e];
        __syncthreads();
        const double n2r = s_n2[r];
        for (int p = warp; p < m; p += MMR_WARPS) {
            if (!s_avail[p]) continue;              // warp-uniform
            const double dot = warp_canon_dot<float>(X + (size_t)p * ORX_DIM, s_x, lane);
            if (lane == 0) {
                double s = __ddiv_rn(dot, __dsqrt_rn(__dmul_rn(s_n2[p], n2r)));
                if (s > 1.0) s = 1.0;
                else if (s < -1.0) s = -1.0;
                const double red = s_red[p];
                if (red == red && (s != s || s > red)) s_red[p] = s;     // max with NaN propagating
            }
        }
        __syncthreads();
        // block argmax over the available positions (p < m <= ORX_MAX_K <= MMR_THREADS: one position per thread)
        double best = 0.0;
        int bestp = -1;
        if (tid < m && s_avail[tid]) {
            best = __dsub_rn(__dmul_rn(lam, s_sq[tid]), __dmul_rn(one_minus_lam, s_red[tid]));
            bestp = tid;
        }
#pragma unroll
        for (int d = 16; d >= 1; d >>= 1) {
            const double ob = __shfl_down_sync(FULL_MASK, best, d);
            const int op = __shfl_down_sync(FULL_MASK, bestp, d);
            if (mmr_better(ob, op, best, bestp)) {
                best = ob;
                bestp = op;
            }
        }
        if (lane == 0) {
            s_best[warp] = best;
            s_bestp[warp] = bestp;
        }
        __syncthreads();
        if (tid == 0) {
            double b = s_best[0];
            int bp = s_bestp[0];
            for (int w = 1; w < MMR_WARPS; ++w)
                if (mmr_better(s_best[w], s_bestp[w], b, bp)) {
                    b = s_best[w];
                    bp = s_bestp[w];
                }
            s_pick = bp;
            s_avail[bp] = 0;
            out[t] = bp;
        }
    }
}

void launch_mmr_select(const float *rows, const double *dist, const int *counts, int nq, int fetch_k, int k,
                       double lam, int *sel, cudaStream_t st) {
    if (nq <= 0) return;
    mmr_select_kernel<<<nq, MMR_THREADS, 0, st>>>(rows, dist, counts, fetch_k, k, lam, sel);
}

}  // namespace orx
