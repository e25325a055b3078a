// Table maintenance kernels: the device side of upsert / delete.
//
// upsert  = `vector_store.aadd_documents` -> INSERT ... ON CONFLICT DO UPDATE (reference
//           app/rag.py:235); "pre-normalised on upsert": the per-row 1/|x| (fp32 `scale`) and the
//           canonical binary64 |x|^2 (`n2`) are computed HERE, once, so a query never touches norms.
//           fp32 tables keep the row bits verbatim (so the canonical rescore sees exactly what the
//           caller stored); bf16 tables store RNE_bf16(x/|x|) and the norm of that rounded row.
//           An fp32 table may also keep a bf16 IMAGE: RNE_bf16(x) of every element, not normalised (the
//           row's fp32 `scale` applies to it unchanged).  The large-table GEMV scans read it instead of the
//           fp32 rows (half the bytes); every kernel here that writes or moves rows keeps it in step.
//           A large fp32 table keeps an 8-bit image instead (quantise8_row): a quarter of the bytes.
// delete  = `vector_store.adelete` -> DELETE ... WHERE langchain_id IN (...) (app/rag.py:231, :371);
//           the host plans disjoint (last live row -> hole) moves, so the table stays dense and the
//           scan needs no tombstone test.
#include "common.cuh"
#include "internal.h"

namespace orx {

__global__ void __launch_bounds__(256)
validate_rows_kernel(const float4 *__restrict__ src, uint64_t n_vec4, int *__restrict__ flag) {
    bool bad = false;
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n_vec4;
         i += (uint64_t)gridDim.x * blockDim.x) {
        const float4 v = src[i];
        bad |= !(isfinite(v.x) && isfinite(v.y) && isfinite(v.z) && isfinite(v.w));
    }
    if (__any_sync(FULL_MASK, bad) && (threadIdx.x & 31) == 0) atomicOr(flag, 1);
}

void launch_validate_rows(const float *src, uint64_t n, int *flag, cudaStream_t st) {
    if (n == 0) return;
    const uint64_t n4 = n * (ORX_DIM / 4);
    uint64_t blocks = (n4 + 255) / 256;
    blocks = cap_grid(blocks, 16);
    validate_rows_kernel<<<(unsigned)blocks, 256, 0, st>>>(reinterpret_cast<const float4 *>(src), n4, flag);
}

// scale markers (see common.cuh score_ord): NaN = zero-norm row, +inf = irregular magnitude
__device__ __forceinline__ float scale_from_n2(double n2) {
    if (!(n2 > 0.0)) return __int_as_float(0x7fc00000);
    // |x| in [2^-40, 2^40]  <=>  n2 in [2^-80, 2^80]; outside, fp32 products may under/overflow
    if (n2 < 8.271806125530277e-25 || n2 > 1.2089258196146292e24) return __int_as_float(0x7f800000);
    return __double2float_rn(__ddiv_rn(1.0, __dsqrt_rn(n2)));
}

// The 8-bit image of one fp32 row (warp-wide, lane l holds elements l + 32 j in v[j]): d = max|x_i| / 127,
// X_i = rint(x_i / d) in [-127, 127], scale8 = d / |x| (binary64, rounded once).  The relative residual
// |x - d X| / |x| is computed in binary64 from the stored X_i; a row over R8_CAP (with a 2^-30 margin for the binary64
// sums) gets the +inf marker, so it is an always-candidate that only the canonical rescore settles.  Zero rows and rows
// of irregular magnitude keep the marker of their fp32 `scale` (sc).  No fp32 operation here sees a subnormal result
// that matters: the residual is measured, whatever rounding produced X.
__device__ __forceinline__ void quantise8_row(const float (&v)[32], double n2, float sc, int lane,
                                              int8_t *__restrict__ xrow, float *__restrict__ scale8_out) {
    float m = 0.f;
#pragma unroll
    for (int j = 0; j < 32; ++j) m = fmaxf(m, fabsf(v[j]));
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) m = fmaxf(m, __shfl_xor_sync(FULL_MASK, m, d));
    const bool regular = isfinite(sc);                 // not a marker
    const float d = __fdiv_rn(m, 127.f);
    double e2 = 0.0;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
        const int8_t X = regular ? (int8_t)__float2int_rn(__fdiv_rn(v[j], d)) : (int8_t)0;
        xrow[lane + 32 * j] = X;
        const double e = __dsub_rn((double)v[j], (double)d * (double)X);    // d * X is exact in binary64
        e2 = __fma_rn(e, e, e2);
    }
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) e2 += __shfl_xor_sync(FULL_MASK, e2, o);
    if (lane == 0) {
        float s8 = sc;
        if (regular)
            s8 = e2 * (1.0 + 0x1p-30) <= R8_CAP * R8_CAP * n2 ? __double2float_rn(__ddiv_rn((double)d, __dsqrt_rn(n2)))
                                                               : __int_as_float(0x7f800000);
        *scale8_out = s8;
    }
}

template <typename T>
__global__ void __launch_bounds__(256)
commit_rows_kernel(const float *__restrict__ src, const uint32_t *__restrict__ src_idx,
                   const uint32_t *__restrict__ dst_row, const orx_id *__restrict__ ids, uint32_t n,
                   T *__restrict__ table, float *__restrict__ scale, double *__restrict__ n2_out,
                   orx_id *__restrict__ row_ids, const int *__restrict__ abort_flag,
                   __nv_bfloat16 *__restrict__ image, Image8 image8) {
    // the batch's element check (validate_rows, earlier on this stream) found a NaN / Inf: nothing is written --
    // the whole batch is rejected and the table stays as it was, without a host round trip in between
    if (abort_flag != nullptr && *abort_flag != 0) return;
    const int lane = threadIdx.x & 31;
    const uint32_t gw = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const uint32_t n_gw = gridDim.x * (blockDim.x >> 5);
    for (uint32_t i = gw; i < n; i += n_gw) {
        const uint32_t si = src_idx[i];
        const uint32_t dst = dst_row[i];
        const float *x = src + (size_t)si * ORX_DIM;
        float v[32];
        double p[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) {
            v[j] = x[lane + 32 * j];
            p[j] = __dmul_rn((double)v[j], (double)v[j]);
        }
        double n2 = bcast_lane0(canon_tree_1024(p));
        T *row = table + (size_t)dst * ORX_DIM;
        if constexpr (sizeof(T) == 4) {
#pragma unroll
            for (int j = 0; j < 32; ++j) row[lane + 32 * j] = v[j];
            if (image != nullptr) {
                __nv_bfloat16 *img = image + (size_t)dst * ORX_DIM;
#pragma unroll
                for (int j = 0; j < 32; ++j) img[lane + 32 * j] = __float2bfloat16_rn(v[j]);
            }
            if (image8.rows != nullptr)
                quantise8_row(v, n2, scale_from_n2(n2), lane, image8.rows + (size_t)dst * ORX_DIM, image8.scale8 + dst);
        } else {
            const double inv = (n2 > 0.0) ? __ddiv_rn(1.0, __dsqrt_rn(n2)) : 0.0;
#pragma unroll
            for (int j = 0; j < 32; ++j) {
                const __nv_bfloat16 b = __float2bfloat16_rn(__double2float_rn(__dmul_rn((double)v[j], inv)));
                row[lane + 32 * j] = b;
                const double bd = (double)__bfloat162float(b);
                p[j] = __dmul_rn(bd, bd);
            }
            n2 = bcast_lane0(canon_tree_1024(p));     // norm of the row AS STORED
        }
        if (lane == 0) {
            scale[dst] = scale_from_n2(n2);
            n2_out[dst] = n2;
            row_ids[dst] = ids[si];
        }
    }
}

void launch_commit_rows(int dtype, const float *src, const uint32_t *src_idx, const uint32_t *dst_row,
                        const orx_id *ids, uint32_t n, void *table, float *scale, double *n2,
                        orx_id *row_ids, const int *abort_flag, void *image, const Image8 &image8, cudaStream_t st) {
    if (n == 0) return;
    uint32_t blocks = (n + 7) / 8;
    blocks = cap_grid(blocks, 8);
    if (dtype == ORX_DTYPE_F32)
        commit_rows_kernel<float><<<blocks, 256, 0, st>>>(src, src_idx, dst_row, ids, n,
                                                          static_cast<float *>(table), scale, n2, row_ids, abort_flag,
                                                          static_cast<__nv_bfloat16 *>(image), image8);
    else
        commit_rows_kernel<__nv_bfloat16><<<blocks, 256, 0, st>>>(
            src, src_idx, dst_row, ids, n, static_cast<__nv_bfloat16 *>(table), scale, n2, row_ids, abort_flag, nullptr,
            Image8{nullptr, nullptr});
}

// Bulk load (snapshot restore / cold start): the rows were copied VERBATIM (table dtype) to the
// table tail [row0, row0+n); this computes what upsert would have: finite check, canonical |x|^2 of
// the row as stored, 1/|x|, the id column.  Nothing is visible to searches until the host bumps
// the live row count, so a NaN/Inf batch is rejected without side effects.  An fp32 table's image rows are
// built from the verbatim rows here (snapshots do not store the image).
template <typename T>
__global__ void __launch_bounds__(256)
adopt_rows_kernel(const T *__restrict__ table, uint32_t row0, uint32_t n, const orx_id *__restrict__ ids,
                  float *__restrict__ scale, double *__restrict__ n2_out, orx_id *__restrict__ row_ids,
                  int *__restrict__ flag, __nv_bfloat16 *__restrict__ image, Image8 image8) {
    const int lane = threadIdx.x & 31;
    const uint32_t gw = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const uint32_t n_gw = gridDim.x * (blockDim.x >> 5);
    for (uint32_t i = gw; i < n; i += n_gw) {
        const uint32_t r = row0 + i;
        const T *row = table + (size_t)r * ORX_DIM;
        __nv_bfloat16 *img = image != nullptr ? image + (size_t)r * ORX_DIM : nullptr;
        float v[32];
        double p[32];
        bool bad = false;
#pragma unroll
        for (int j = 0; j < 32; ++j) {
            v[j] = row_elem<T>(row, lane + 32 * j);
            bad |= !isfinite(v[j]);
            p[j] = __dmul_rn((double)v[j], (double)v[j]);
            if (img != nullptr) img[lane + 32 * j] = __float2bfloat16_rn(v[j]);
        }
        const double n2 = bcast_lane0(canon_tree_1024(p));
        if (__any_sync(FULL_MASK, bad) && lane == 0) atomicOr(flag, 1);
        if (image8.rows != nullptr)             // a rejected batch is never published: its image rows do not matter
            quantise8_row(v, n2, scale_from_n2(n2), lane, image8.rows + (size_t)r * ORX_DIM, image8.scale8 + r);
        if (lane == 0) {
            scale[r] = scale_from_n2(n2);
            n2_out[r] = n2;
            row_ids[r] = ids[i];
        }
    }
}

void launch_adopt_rows(int dtype, const void *table, uint32_t row0, uint32_t n, const orx_id *ids, float *scale,
                       double *n2, orx_id *row_ids, int *flag, void *image, const Image8 &image8, cudaStream_t st) {
    if (n == 0) return;
    uint32_t blocks = (n + 7) / 8;
    blocks = cap_grid(blocks, 8);
    if (dtype == ORX_DTYPE_F32)
        adopt_rows_kernel<float><<<blocks, 256, 0, st>>>(static_cast<const float *>(table), row0, n, ids, scale, n2,
                                                         row_ids, flag, static_cast<__nv_bfloat16 *>(image), image8);
    else
        adopt_rows_kernel<__nv_bfloat16><<<blocks, 256, 0, st>>>(static_cast<const __nv_bfloat16 *>(table), row0, n,
                                                                 ids, scale, n2, row_ids, flag, nullptr,
                                                                 Image8{nullptr, nullptr});
}

// the image of fp32 rows [0, n) that are already in the table (a grown table whose earlier allocation had no image)
__global__ void __launch_bounds__(256)
image_rows_kernel(const float4 *__restrict__ table, uint64_t n_vec4, uint2 *__restrict__ image) {
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n_vec4; i += (uint64_t)gridDim.x * blockDim.x) {
        const float4 v = table[i];
        const __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
        image[i] = make_uint2(*reinterpret_cast<const uint32_t *>(&lo), *reinterpret_cast<const uint32_t *>(&hi));
    }
}

void launch_image_rows(const float *table, uint64_t n, void *image, cudaStream_t st) {
    if (n == 0) return;
    const uint64_t n4 = n * (ORX_DIM / 4);
    const uint64_t blocks = cap_grid((n4 + 255) / 256, 16);
    image_rows_kernel<<<(unsigned)blocks, 256, 0, st>>>(reinterpret_cast<const float4 *>(table), n4,
                                                       static_cast<uint2 *>(image));
}

// the 8-bit image of fp32 rows [0, n) that are already in the table, from their stored n2 and scale
__global__ void __launch_bounds__(256)
image8_rows_kernel(const float *__restrict__ table, const double *__restrict__ n2, const float *__restrict__ scale,
                   uint64_t n, Image8 image8) {
    const int lane = threadIdx.x & 31;
    const uint64_t gw = blockIdx.x * (uint64_t)(blockDim.x >> 5) + (threadIdx.x >> 5);
    const uint64_t n_gw = (uint64_t)gridDim.x * (blockDim.x >> 5);
    for (uint64_t r = gw; r < n; r += n_gw) {
        const float *row = table + r * ORX_DIM;
        float v[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = row[lane + 32 * j];
        quantise8_row(v, n2[r], scale[r], lane, image8.rows + r * ORX_DIM, image8.scale8 + r);
    }
}

void launch_image8_rows(const float *table, const double *n2, const float *scale, uint64_t n, const Image8 &image8,
                        cudaStream_t st) {
    if (n == 0) return;
    const uint64_t blocks = cap_grid((n + 7) / 8, 8);
    image8_rows_kernel<<<(unsigned)blocks, 256, 0, st>>>(table, n2, scale, n, image8);
}

__global__ void __launch_bounds__(256)
count_capped8_kernel(const float *__restrict__ scale, const float *__restrict__ scale8, uint64_t n,
                     uint32_t *__restrict__ count) {
    uint32_t mine = 0;
    for (uint64_t r = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; r < n; r += (uint64_t)gridDim.x * blockDim.x)
        mine += (scale8[r] == __int_as_float(0x7f800000) && isfinite(scale[r])) ? 1u : 0u;
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) mine += __shfl_xor_sync(FULL_MASK, mine, d);
    if ((threadIdx.x & 31) == 0 && mine) atomicAdd(count, mine);
}

void launch_count_capped8(const float *scale, const float *scale8, uint64_t n, uint32_t *count, cudaStream_t st) {
    cudaMemsetAsync(count, 0, sizeof(uint32_t), st);
    if (n == 0) return;
    const uint64_t blocks = cap_grid((n + 255) / 256, 8);
    count_capped8_kernel<<<(unsigned)blocks, 256, 0, st>>>(scale, scale8, n, count);
}

// one warp per relocated row; sources (>= new live count) and destinations (< new live count)
// are disjoint sets, so all moves run in parallel.
__global__ void __launch_bounds__(256)
move_rows_kernel(const uint32_t *__restrict__ src_row, const uint32_t *__restrict__ dst_row, uint32_t n,
                 uint4 *__restrict__ table, int vec_per_row, float *__restrict__ scale,
                 double *__restrict__ n2, orx_id *__restrict__ row_ids, uint4 *__restrict__ image, Image8 image8) {
    const int lane = threadIdx.x & 31;
    const uint32_t gw = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const uint32_t n_gw = gridDim.x * (blockDim.x >> 5);
    for (uint32_t i = gw; i < n; i += n_gw) {
        const uint32_t s = src_row[i], d = dst_row[i];
        const uint4 *sp = table + (size_t)s * vec_per_row;
        uint4 *dp = table + (size_t)d * vec_per_row;
        for (int j = lane; j < vec_per_row; j += 32) dp[j] = sp[j];
        if (image != nullptr) {                  // 2048 B of image per row = 128 x 16 B
            const uint4 *si = image + (size_t)s * 128;
            uint4 *di = image + (size_t)d * 128;
#pragma unroll
            for (int j = 0; j < 4; ++j) di[lane + 32 * j] = si[lane + 32 * j];
        }
        if (image8.rows != nullptr) {            // 1024 B = 64 x 16 B
            const uint4 *si = reinterpret_cast<const uint4 *>(image8.rows) + (size_t)s * 64;
            uint4 *di = reinterpret_cast<uint4 *>(image8.rows) + (size_t)d * 64;
            di[lane] = si[lane];
            di[lane + 32] = si[lane + 32];
            if (lane == 0) image8.scale8[d] = image8.scale8[s];
        }
        if (lane == 0) {
            scale[d] = scale[s];
            n2[d] = n2[s];
            row_ids[d] = row_ids[s];
        }
    }
}

void launch_move_rows(int dtype, const uint32_t *src_row, const uint32_t *dst_row, uint32_t n,
                      void *table, float *scale, double *n2, orx_id *row_ids, void *image, const Image8 &image8,
                      cudaStream_t st) {
    if (n == 0) return;
    uint32_t blocks = (n + 7) / 8;
    blocks = cap_grid(blocks, 8);
    const int vpr = dtype == ORX_DTYPE_F32 ? 256 : 128;
    move_rows_kernel<<<blocks, 256, 0, st>>>(src_row, dst_row, n, static_cast<uint4 *>(table), vpr,
                                             scale, n2, row_ids, static_cast<uint4 *>(image), image8);
}

template <typename T>
__global__ void __launch_bounds__(256)
gather_rows_kernel(const T *__restrict__ table, const uint32_t *__restrict__ rows, uint32_t n,
                   float *__restrict__ out) {
    const int lane = threadIdx.x & 31;
    const uint32_t gw = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const uint32_t n_gw = gridDim.x * (blockDim.x >> 5);
    for (uint32_t i = gw; i < n; i += n_gw) {
        const uint32_t r = rows[i];
        if (r == ROW_INVALID) {
            for (int e = lane; e < ORX_DIM; e += 32) out[(size_t)i * ORX_DIM + e] = 0.f;
            continue;
        }
        const T *row = table + (size_t)r * ORX_DIM;
        for (int e = lane; e < ORX_DIM; e += 32) out[(size_t)i * ORX_DIM + e] = row_elem<T>(row, e);
    }
}

void launch_gather_rows(int dtype, const void *table, const uint32_t *rows, uint32_t n, float *out,
                        cudaStream_t st) {
    if (n == 0) return;
    uint32_t blocks = (n + 7) / 8;
    blocks = cap_grid(blocks, 8);
    if (dtype == ORX_DTYPE_F32)
        gather_rows_kernel<float><<<blocks, 256, 0, st>>>(static_cast<const float *>(table), rows, n, out);
    else
        gather_rows_kernel<__nv_bfloat16><<<blocks, 256, 0, st>>>(
            static_cast<const __nv_bfloat16 *>(table), rows, n, out);
}

// ---- filtered tcgen05 scan: the row predicate enters the scan through the per-row scale -- a row whose bit is clear gets
//      the "never a candidate" marker (NaN, the same as a zero-norm row), so the tensor-core epilogue needs no bitmap
__global__ void mask_scale_kernel(const float *__restrict__ scale, const uint32_t *__restrict__ allow_bits, uint32_t n_rows,
                                  float *__restrict__ out) {
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t r = blockIdx.x * blockDim.x + threadIdx.x; r < n_rows; r += stride) {
        const uint32_t w = __ldg(allow_bits + (r >> 5));
        out[r] = (w >> (r & 31)) & 1u ? scale[r] : __int_as_float(0x7fc00000);
    }
}
void launch_mask_scale(const float *scale, const uint32_t *allow_bits, uint32_t n_rows, float *out, cudaStream_t st) {
    if (n_rows == 0) return;
    const uint32_t blocks = cap_grid((n_rows + 255u) / 256u, 8);
    mask_scale_kernel<<<blocks, 256, 0, st>>>(scale, allow_bits, n_rows, out);
}

}  // namespace orx
