// tcgen05 / TMEM batched scan (scan_umma.cu): host-side interface.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include "internal.h"

namespace orx {

struct UmmaPlan;

UmmaPlan *umma_plan_create(int device);
void umma_plan_destroy(UmmaPlan *p);
constexpr int UMMA_MAX_K = 64;                   // largest k the coarse pass can prove (candidate lists of 160 keys)
bool umma_should_use(const UmmaPlan *p, int nq, int k, uint32_t n_rows);
const char *umma_last_error();

// Coarse tensor-core scan + finalize for nq queries; writes results and per-query proof flags.
// `scale` may be a MASKED copy (launch_mask_scale: NaN for the rows a filter excludes -- never candidates, like zero-norm rows).
int umma_search(UmmaPlan *p, int dtype, const void *table, const float *scale, const double *n2,
                const orx_id *row_ids, uint32_t n_rows, const float *q_dev, const float *qhat,
                const __nv_bfloat16 *qhat16, const QueryPrep *prep, int nq, int k, const ResultOut &out,
                const PublishArgs &pub, const DoneArgs &done, cudaStream_t st,
                uint64_t *launch_counter, cudaEvent_t ev_begin, cudaEvent_t ev_end);

// diagnostic: every scaled coarse score of the tcgen05 pass, out[row * nq + query] (device), same MMA path as the search
int umma_dump_scores(UmmaPlan *p, int dtype, const void *table, const float *scale, uint32_t n_rows, const float *qhat,
                     const __nv_bfloat16 *qhat16, int nq, bool pairs, float *out, cudaStream_t st);

}  // namespace orx
