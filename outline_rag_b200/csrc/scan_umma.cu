// scan_umma: the batched scan -- a tcgen05 / TMEM GEMM fed by TMA with the top-k selection
// fused into the epilogue, so the [queries x rows] score matrix never reaches HBM.
//
// Stands in for `ORDER BY embedding <=> :q LIMIT :k` issued for MANY queries at once (the
// micro-batched form of reference app/rag.py:85-87 -> langchain-postgres SQL; SURVEY.md 8f-3).
//
// Orientation: queries on M (TMEM lanes), table rows on N (TMEM columns):
//     D[128 queries x 256 rows] += Qhat[128 x Kc] . X[256 x Kc]^T      (both operands K-major)
// bf16 tables run kind::f16 (bf16 x bf16 -> fp32), fp32 tables run kind::tf32 on the fp32 bits.
// Each epilogue thread owns ONE query (one TMEM lane): it reads its accumulator row with
// tcgen05.ld and tests every column against a private running threshold
//     thr = (k-th best coarse score seen for this query) - margin,   margin = 2*eps + 1e-6
// appending survivors (score key | ~row) to a small per-(query, CTA) list in global memory.
// Every row a thread drops has coarse score <= thr, and k kept rows have coarse >= thr + margin,
// so with |coarse - cos| <= eps no dropped row can belong to the top-k: the candidate set is
// COMPLETE by construction; finalize_kernel rescoring makes it exact and re-proves it
// (floor = the largest final thr of the query's CTAs).  Thresholds are shared between CTAs
// through an atomicMax'd per-query word, so the bootstrap flood is paid about once.
//
// Warp roles (256 threads, 1 CTA / SM, persistent): warps 0..3 = epilogue (TMEM lane quarter =
// warp % 4), warp 4 = TMA producer, warp 5 = MMA issuer (one lane), warp 6 = TMEM allocator.
// Pipelines: smem full/empty ring (4 stages x 48 KB) and a 2 x 256-column TMEM accumulator
// ring, so the epilogue of tile i overlaps the MMAs of tile i+1.
// CTA c works on query tile m = c % m_tiles and row tiles slot, slot + n_slots, ... with
// slot = c / m_tiles: the m_tiles CTAs of a slot stream the same table tile at the same time,
// so it is read from HBM once and served from L2 to the others.
// Algorithmic work per launch: bytes = rows*1024*sizeof(elem); flops = 2*rows*1024*queries.
#include <cuda.h>

#include <cstdlib>
#include <mutex>
#include <string>

#include "common.cuh"
#include "scan_umma.h"

namespace orx {

namespace {

constexpr int UM_THREADS = 256;
// Warp roles.  The SM's warp arbiter prefers the HIGHEST warp id among the eligible warps of a scheduler
// (B300_MICROARCH.md), so the two single-lane control warps sit above the epilogue warp they share a
// scheduler with: a busy epilogue must not delay TMA or MMA issue (same-box A/B at 6Mx1024 bf16, B=1024:
// 10.03 -> 9.65 ms).  Epilogue = warps 0..3 (TMEM lane quarter = warp % 4).
constexpr int WARP_TMA = 4, WARP_MMA = 5, WARP_ALLOC = 6;
constexpr int TILE_M = 128;            // queries per CTA tile (UMMA M)
constexpr int TILE_N = 256;            // table rows per tile (UMMA N)
constexpr int STAGES = 4;
constexpr int A_BYTES = TILE_M * 128;  // 16 KB: 128 rows x one 128-byte swizzle row of K
constexpr int B_BYTES = TILE_N * 128;  // 32 KB
constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
// Candidate slots per (query, CTA).  A list must hold the CTA's k best coarse scores AND every row within the margin
// (2 eps + 1e-6 = 5e-3) below the k-th of them; measured on the synthetic corpus (tools/bench_wide_k.py) that is ~2.2-2.5 k
// rows, so: 64 keys (finalize S=2) up to k = 16, 160 keys (S=5) up to k = 64.  Beyond that even finalize's 160 rescored
// candidates cannot prove a tf32 / bf16 coarse ranking, and the caller keeps the exact fp32 scan (UMMA_MAX_K, scan_umma.h).
constexpr int CAND = 64;
constexpr int CAND_WIDE = 160;
constexpr int CAND_NARROW_MAX_K = 16;
constexpr int SMEM_MAIN = STAGES * STAGE_BYTES;
constexpr int SMEM_SCALE = 2 * TILE_N * 4;
constexpr int SMEM_TOTAL = SMEM_MAIN + SMEM_SCALE + 256 + 1024;   // + barriers + alignment slack

// CTA-pair kernel: each CTA stages its 128 queries + HALF of the 256-row table tile per K chunk
constexpr int STAGES2 = 6;
constexpr int B2_BYTES = (TILE_N / 2) * 128;                 // 16 KB
constexpr int STAGE2_BYTES = A_BYTES + B2_BYTES;             // 32 KB
constexpr int SMEM2_MAIN = STAGES2 * STAGE2_BYTES;
constexpr int SMEM2_TOTAL = SMEM2_MAIN + SMEM_SCALE + 256 + 1024;

constexpr uint64_t HINT_EVICT_NORMAL = 0x1000000000000000ull;
constexpr uint64_t HINT_EVICT_FIRST = 0x12F0000000000000ull;
constexpr uint64_t HINT_EVICT_LAST = 0x14F0000000000000ull;

// Two data-movement variants of the pair kernel were built, parity-checked and A/B-measured in round 2 (DESIGN.md 4.1);
// neither beats it, so they are compiled only into variant builds (make variant NAME=... DEFS=-DORX_UMMA_QUADS=1):
#ifndef ORX_UMMA_QUADS
#define ORX_UMMA_QUADS 0             // 1: batches with an even number of 256-query tiles run on clusters of 4 (table tile multicast)
#endif
#ifndef ORX_UMMA_ARES
#define ORX_UMMA_ARES 0              // 1: bf16 batches on CTA pairs keep half of the query tile resident in shared memory
#endif

// ------------------------------------------------------------------------- PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// Bounded wait: a pipeline bug traps (launch failure) after ~4 s instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t done = 0;
    uint64_t t0 = 0;
    for (uint32_t it = 0;; ++it) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done) : "r"(bar), "r"(parity) : "memory");
        if (done) return;
        if ((it & 1023u) == 1023u) {
            uint64_t now;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
            if (t0 == 0) t0 = now;
            else if (now - t0 > 4000000000ull) __trap();
        }
    }
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap *map, uint32_t bar, int c0, int c1,
                                            uint64_t hint) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
        " [%0], [%1, {%3, %4}], [%2], %5;"
        ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "l"(hint) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
template <bool TF32>
__device__ __forceinline__ void tc_mma(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
    if constexpr (TF32)
        asm volatile(
            "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
            ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc) : "memory");
    else
        asm volatile(
            "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
            ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
          "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
          "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// the staged 1/|x| values go through explicit shared-space instructions (a generic pointer derived from the
// aligned dynamic-smem base compiles to LD.E / ST.E, which take the slower generic path)
__device__ __forceinline__ float4 lds_f4(uint32_t addr) {
    float4 r;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "r"(addr) : "memory");
    return r;
}
__device__ __forceinline__ float lds_f32(uint32_t addr) {
    float r;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(r) : "r"(addr) : "memory");
    return r;
}
__device__ __forceinline__ void sts_f32(uint32_t addr, float v) {
    asm volatile("st.shared.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory");
}

// Timing experiments (skip the column scan / the query loads / the table loads: results are garbage) exist ONLY in
// builds made with -DORX_DEBUG_VARIANTS (`make variant NAME=dbg DEFS=-DORX_DEBUG_VARIANTS`); the product library
// contains neither the code paths nor the ORX_UMMA_DEBUG / ORX_UMMA_PAIRS environment look-ups.
#ifdef ORX_DEBUG_VARIANTS
#define ORX_DBG_PARAM , int dbg
#define ORX_DBG_ARG(p) , (p)->dbg
#define ORX_DBG_FWD , dbg
#define ORX_DBG(bit) (dbg & (bit))
#else
#define ORX_DBG_PARAM
#define ORX_DBG_ARG(p)
#define ORX_DBG_FWD
#define ORX_DBG(bit) 0
#endif

// ---- CTA-pair (cta_group::2) variants
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of `local_addr` in CTA `rank` of this cluster
__device__ __forceinline__ uint32_t map_to_cta(uint32_t local_addr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(rank));
    return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// each CTA of the pair loads into ITS OWN smem; the bytes are counted on the LEADER's barrier
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst, const CUtensorMap *map, uint32_t leader_bar, int c0,
                                                 int c1, uint64_t hint) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
        " [%0], [%1, {%3, %4}], [%2], %5;"
        ::"r"(dst), "l"(map), "r"(leader_bar), "r"(c0), "r"(c1), "l"(hint) : "memory");
}
__device__ __forceinline__ void tc_commit_pair(uint32_t bar) {      // arrives on `bar` in BOTH CTAs of the pair
    asm volatile(
        "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
        ::"r"(bar), "h"((uint16_t)3) : "memory");
}
#if ORX_UMMA_QUADS
// cta_group::2 + multicast: the box lands at the same smem offset in every CTA of `cta_mask`; its bytes are counted on the
// barrier at `bar`'s offset in the EVEN CTA (the MMA leader) of each destination's pair (`bar` carries an even CTA rank)
__device__ __forceinline__ void tma_load_2d_pair_mc(uint32_t dst, const CUtensorMap *map, uint32_t bar, int c0, int c1,
                                                    uint16_t cta_mask, uint64_t hint) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster.L2::cache_hint"
        " [%0], [%1, {%4, %5}], [%2], %3, %6;"
        ::"r"(dst), "l"(map), "r"(bar), "h"(cta_mask), "r"(c0), "r"(c1), "l"(hint) : "memory");
}
__device__ __forceinline__ void tc_commit_mc(uint32_t bar, uint16_t cta_mask) {      // arrives on `bar` in every CTA of the mask
    asm volatile(
        "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
        ::"r"(bar), "h"(cta_mask) : "memory");
}
#endif
template <bool TF32>
__device__ __forceinline__ void tc_mma_pair(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
    if constexpr (TF32)
        asm volatile(
            "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
            ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc) : "memory");
    else
        asm volatile(
            "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
            ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc) : "memory");
}

// K-major, 128-byte swizzle shared-memory matrix descriptor (sm_100 "version 1"):
// start>>4 | LBO(=1, unused for swizzled K-major)<<16 | SBO(= 8 rows x 128 B = 1024 B)>>4 <<32 | layout SWIZZLE_128B.
__device__ __forceinline__ uint64_t make_desc_sw128(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)(1024 >> 4) << 32;
    d |= (uint64_t)1 << 46;           // descriptor version (Blackwell)
    d |= (uint64_t)2 << 61;           // SWIZZLE_128B
    return d;
}
// instruction descriptor: D fp32, A/B bf16 (1) or tf32 (2), both K-major, N>>3 at [17,23), M>>4 at [24,29)
__host__ __device__ constexpr uint32_t make_idesc(bool tf32, int m = TILE_M) {
    return (1u << 4) | ((tf32 ? 2u : 1u) << 7) | ((tf32 ? 2u : 1u) << 10) | ((uint32_t)(TILE_N >> 3) << 17) |
           ((uint32_t)(m >> 4) << 24);
}

// ------------------------------------------------------------------ candidate list upkeep
// Warp-cooperative compaction of lane L's candidate list (<= 32 x CPL keys, CPL per lane): raise L's
// threshold to (k-th best REGULAR coarse score) - margin, keep what is still above it (and every
// ORD_ALWAYS key), publish the threshold.  All 32 lanes call this with the same L.
template <int CPL>
__device__ __forceinline__ void coop_compact(uint64_t *list, int L, int lane, int &cnt, float &thr, int k,
                                             float margin, uint32_t *gthr_L) {
    __syncwarp();                                    // lane L's appends are visible to the warp
    const int n = __shfl_sync(FULL_MASK, cnt, L);
    const float thr_L = __shfl_sync(FULL_MASK, thr, L);
    uint64_t key[CPL], reg[CPL];                     // reg: regular keys only take part in the ranking
    bool alw[CPL];
    int rank[CPL];
#pragma unroll
    for (int i = 0; i < CPL; ++i) {
        key[i] = lane + 32 * i < n ? list[lane + 32 * i] : 0ull;
        alw[i] = key_ord(key[i]) == ORD_ALWAYS;
        reg[i] = alw[i] ? 0ull : key[i];
        rank[i] = 0;
    }
#pragma unroll 4
    for (int s = 0; s < 32; ++s) {
#pragma unroll
        for (int j = 0; j < CPL; ++j) {
            const uint64_t x = shfl_u64(reg[j], s);
#pragma unroll
            for (int i = 0; i < CPL; ++i) rank[i] += (x > reg[i]);
        }
    }
    // keys are unique (distinct rows), so exactly one regular key has rank k-1 when >= k exist
    uint32_t mine = 0u;
#pragma unroll
    for (int i = 0; i < CPL; ++i)
        if (reg[i] != 0ull && rank[i] == k - 1) mine = key_ord(reg[i]);
    const uint32_t kth = __reduce_max_sync(FULL_MASK, mine);
    float new_thr = thr_L;
    if (kth != 0u) new_thr = fmaxf(thr_L, ord_to_float(kth) - margin);
    const unsigned lt = (1u << lane) - 1u;
    bool keep[CPL];
    int pos[CPL];
    int total = 0;
#pragma unroll
    for (int i = 0; i < CPL; ++i) {
        keep[i] = key[i] != 0ull && (alw[i] || ord_to_float(key_ord(key[i])) > new_thr);
        const unsigned b = __ballot_sync(FULL_MASK, keep[i]);
        pos[i] = total + __popc(b & lt);
        total += __popc(b);
    }
    __syncwarp();
#pragma unroll
    for (int i = 0; i < CPL; ++i)
        if (keep[i]) list[pos[i]] = key[i];
    __syncwarp();
    if (lane == L) {
        cnt = total;
        thr = new_thr;
        if (kth != 0u) atomicMax(gthr_L, float_to_ord(new_thr));
    }
}

// ------------------------------------------------------------------------------- epilogue
// Shared by the 1-CTA and the 2-CTA kernels: 4 warps, thread = one query (TMEM lane), see the file
// header.  `arrive_empty(buf)` hands accumulator buffer `buf` back to the MMA issuer.
// DUMP (diagnostic instantiation behind orx_debug_coarse_scores): instead of selecting, every scaled coarse score is
// written to dump[row * dump_ld + query], so that a test can MEASURE max |coarse - cosine| against eps.
template <bool DUMP, int C, class ArriveEmpty>
__device__ __forceinline__ void epilogue_loop(int q_base, int nq, int slot, int n_slots, uint32_t n_tiles,
                                              const float *__restrict__ scale, uint32_t n_rows, int k, float margin,
                                              uint64_t *__restrict__ partial, float *__restrict__ floor_out,
                                              uint32_t *__restrict__ gthr_all, float *s_scale, uint32_t bar_tfull,
                                              uint32_t tmem_base, int ew, int lane, ArriveEmpty arrive_empty,
                                              float *__restrict__ dump, uint32_t dump_ld
                                              ORX_DBG_PARAM) {
    const int et = ew * 32 + lane;                          // 0..127
    const int q = q_base + ew * 32 + lane;
    const bool active = q < nq;
    uint64_t *buf_keys = partial + ((size_t)(active ? q : 0) * n_slots + slot) * C;
    uint32_t *gthr = gthr_all + (active ? q : 0);
    float thr = __int_as_float(0xff800000);                 // -inf
    int cnt = 0;
    bool overflow = false;
    uint32_t buf = 0, tphase = 0;
    // 1/|x| of the NEXT tile is fetched while the current one is scanned (the loads miss to HBM)
    float sc_next[2];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const uint32_t r = (uint32_t)slot * TILE_N + et + 128 * h;
        sc_next[h] = ((uint32_t)slot < n_tiles && r < n_rows) ? __ldg(scale + r) : __int_as_float(0x7fc00000);
    }
    for (uint32_t t = slot; t < n_tiles; t += n_slots) {
        const uint32_t n0 = t * TILE_N;
        // stage this tile's 1/|x| (NaN beyond the table end: never a candidate)
        const uint32_t sc = smem_u32(s_scale) + buf * TILE_N * 4;
        bool special = false;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const float s = sc_next[h];
            // +inf (irregular magnitude: always a candidate) needs the slow path; NaN (zero-norm row, row beyond the end, row
            // excluded by a filter) needs nothing: its score is NaN, which fmaxf ignores and `> thr` rejects
            special |= fabsf(s) == __int_as_float(0x7f800000);
            sts_f32(sc + 4 * (et + 128 * h), s);
            const uint32_t rn = n0 + (uint32_t)n_slots * TILE_N + et + 128 * h;
            sc_next[h] = (t + n_slots < n_tiles && rn < n_rows) ? __ldg(scale + rn) : __int_as_float(0x7fc00000);
        }
        uint32_t tile_special;
        asm volatile(
            "{\n\t.reg .pred p, q;\n\tsetp.ne.u32 q, %1, 0;\n\t"
            "bar.red.or.pred p, 1, 128, q;\n\tselp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(tile_special) : "r"((uint32_t)special) : "memory");
        if (active) {
            const uint32_t g = *reinterpret_cast<volatile uint32_t *>(gthr);
            if (g) thr = fmaxf(thr, ord_to_float(g));
        }
        mbar_wait(bar_tfull + 8 * buf, tphase);
        tc_fence_after();
        const uint32_t taddr = tmem_base + ((uint32_t)(ew * 32) << 16) + buf * TILE_N;
#pragma unroll 1
        for (int c = 0; c < (ORX_DBG(1) ? 0 : TILE_N / 32); ++c) {
            uint32_t v[32];
            tmem_ld32(taddr + c * 32, v);
            tmem_ld_wait();
            float s[32];
            float mx = __int_as_float(0xff800000);
#pragma unroll
            for (int j4 = 0; j4 < 8; ++j4) {
                const float4 f = lds_f4(sc + 4 * (c * 32 + 4 * j4));
                s[4 * j4 + 0] = __uint_as_float(v[4 * j4 + 0]) * f.x;
                s[4 * j4 + 1] = __uint_as_float(v[4 * j4 + 1]) * f.y;
                s[4 * j4 + 2] = __uint_as_float(v[4 * j4 + 2]) * f.z;
                s[4 * j4 + 3] = __uint_as_float(v[4 * j4 + 3]) * f.w;
                mx = fmaxf(fmaxf(mx, fmaxf(s[4 * j4 + 0], s[4 * j4 + 1])), fmaxf(s[4 * j4 + 2], s[4 * j4 + 3]));
            }
            if constexpr (DUMP) {
                if (active) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const uint32_t row = n0 + c * 32 + j;
                        if (row < n_rows) dump[(size_t)row * dump_ld + q] = s[j];      // a warp writes 32 consecutive queries
                    }
                }
                continue;
            }
            // fmaxf ignores NaN (zero-norm rows, rows beyond the end); irregular rows need the slow path
            const bool hit = active && ((mx > thr) || tile_special);
            if (!__any_sync(FULL_MASK, hit)) continue;
            // ---- slow path (warp-uniform): some lane has survivors in these 32 columns
            uint32_t always = 0;
            if (tile_special) {
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    const float sj = lds_f32(sc + 4 * (c * 32 + j));
                    if (sj == __int_as_float(0x7f800000)) always |= 1u << j;      // irregular magnitude
                    else if (sj != sj) s[j] = __int_as_float(0xff800000);         // zero-norm / beyond the end
                }
            }
            uint32_t mask = 0;
            for (int round = 0;; ++round) {
                mask = 0;
                if (active) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) mask |= (s[j] > thr) ? (1u << j) : 0u;
                    mask = (mask & ~always) | (overflow ? 0u : always);
                }
                const unsigned need = __ballot_sync(FULL_MASK, active && cnt + __popc(mask) > C);
                if (!need) break;
                if (round == 1) {
                    // near-ties wider than the list: the query is re-answered by the fp32 scan
                    if (need & (1u << lane)) {
                        overflow = true;
                        thr = __int_as_float(0x7f800000);
                        atomicMax(gthr, float_to_ord(thr));
                    }
                    continue;
                }
                unsigned todo = need;
                while (todo) {
                    const int L = __ffs(todo) - 1;
                    todo &= todo - 1;
                    uint64_t *list_L = partial + ((size_t)(q - lane + L) * n_slots + slot) * C;
                    coop_compact<C / 32>(list_L, L, lane, cnt, thr, k, margin, gthr_all + (q - lane + L));
                }
            }
            if (mask) {
                const uint32_t row0 = n0 + c * 32;
#pragma unroll
                for (int j = 0; j < 32; ++j)
                    if (mask & (1u << j))
                        buf_keys[cnt++] = make_key((always >> j) & 1u ? ORD_ALWAYS : float_to_ord(s[j]), row0 + j);
            }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) arrive_empty(buf);
        if (++buf == 2) { buf = 0; tphase ^= 1; }
    }
    if (active && !DUMP) {
        for (int i = cnt; i < C; ++i) buf_keys[i] = 0ull;
        floor_out[(size_t)q * n_slots + slot] = overflow ? __int_as_float(0x7f800000) : thr;
    }
}

template <bool TF32, bool DUMP = false, int C = CAND>
__global__ void __launch_bounds__(UM_THREADS, 1)
scan_umma_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_x,
                 const float *__restrict__ scale, uint32_t n_rows, int nq, int m_tiles, int n_slots, int k,
                 float margin, uint64_t *__restrict__ partial, float *__restrict__ floor_out,
                 uint32_t *__restrict__ gthr_all, float *__restrict__ dump, uint32_t dump_ld ORX_DBG_PARAM) {
    constexpr int ES = TF32 ? 4 : 2;                // operand element size
    constexpr int BLOCK_K = 128 / ES;               // elements per 128-byte swizzle row
    constexpr int K_CHUNKS = ORX_DIM / BLOCK_K;     // 16 (bf16) / 32 (tf32)
    constexpr uint32_t IDESC = make_idesc(TF32);

    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    float *s_scale = reinterpret_cast<float *>(smem + SMEM_MAIN);               // [2][TILE_N]
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem + SMEM_MAIN + SMEM_SCALE);
    uint32_t *s_tmem = reinterpret_cast<uint32_t *>(bars + 16);
    const uint32_t smem_base = smem_u32(smem);
    const uint32_t bar_full = smem_u32(bars);            // [STAGES]
    const uint32_t bar_empty = bar_full + 8 * STAGES;    // [STAGES]
    const uint32_t bar_tfull = bar_empty + 8 * STAGES;   // [2]
    const uint32_t bar_tempty = bar_tfull + 16;          // [2]

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int m_tile = blockIdx.x % m_tiles;
    const int slot = blockIdx.x / m_tiles;
    const uint32_t n_tiles = (n_rows + TILE_N - 1) / TILE_N;

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(bar_full + 8 * s, 1);
            mbar_init(bar_empty + 8 * s, 1);
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(bar_tfull + 8 * b, 1);
            mbar_init(bar_tempty + 8 * b, 4);            // one arrival per epilogue warp
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == WARP_ALLOC) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(s_tmem)),
                     "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *s_tmem;

    if (warp == WARP_TMA) {
        // ===================================================================== TMA producer
        if (lane == 0) {
            asm volatile("prefetch.tensormap [%0];" ::"l"(&map_q) : "memory");
            asm volatile("prefetch.tensormap [%0];" ::"l"(&map_x) : "memory");
            const uint64_t hint_x = (m_tiles > 1) ? HINT_EVICT_NORMAL : HINT_EVICT_FIRST;
            uint32_t stage = 0, phase = 0;
            for (uint32_t t = slot; t < n_tiles; t += n_slots) {
                for (int kc = 0; kc < K_CHUNKS; ++kc) {
                    mbar_wait(bar_empty + 8 * stage, phase ^ 1);
                    const uint32_t sa = smem_base + stage * STAGE_BYTES;
                    mbar_expect_tx(bar_full + 8 * stage, (ORX_DBG(2) ? 0 : A_BYTES) + (ORX_DBG(4) ? 0 : B_BYTES));
                    if (!ORX_DBG(2))
                        tma_load_2d(sa, &map_q, bar_full + 8 * stage, kc * BLOCK_K, m_tile * TILE_M, HINT_EVICT_LAST);
                    if (!ORX_DBG(4))
                        tma_load_2d(sa + A_BYTES, &map_x, bar_full + 8 * stage, kc * BLOCK_K, (int)(t * TILE_N), hint_x);
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == WARP_MMA) {
        // ======================================================================= MMA issuer
        if (lane == 0) {
            uint32_t stage = 0, phase = 0, buf = 0, tphase = 0;
            for (uint32_t t = slot; t < n_tiles; t += n_slots) {
                mbar_wait(bar_tempty + 8 * buf, tphase ^ 1);       // epilogue drained this accumulator
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + buf * TILE_N;
                for (int kc = 0; kc < K_CHUNKS; ++kc) {
                    mbar_wait(bar_full + 8 * stage, phase);
                    tc_fence_after();
                    const uint32_t sa = smem_base + stage * STAGE_BYTES;
                    const uint64_t adesc = make_desc_sw128(sa);
                    const uint64_t bdesc = make_desc_sw128(sa + A_BYTES);
#pragma unroll
                    for (int k4 = 0; k4 < 4; ++k4)             // 4 x (32 bytes of K) per swizzle row
                        tc_mma<TF32>(d_tmem, adesc + 2 * k4, bdesc + 2 * k4, IDESC, (kc | k4) != 0 ? 1u : 0u);
                    tc_commit(bar_empty + 8 * stage);           // frees the smem stage when the MMAs retire
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
                tc_commit(bar_tfull + 8 * buf);                 // accumulator ready for the epilogue
                if (++buf == 2) { buf = 0; tphase ^= 1; }
            }
        }
    } else if (warp < 4) {
        // ========================================================================= epilogue
        epilogue_loop<DUMP, C>(m_tile * TILE_M, nq, slot, n_slots, n_tiles, scale, n_rows, k, margin, partial, floor_out,
                            gthr_all, s_scale, bar_tfull, tmem_base, warp, lane,
                            [&](uint32_t b) { mbar_arrive(bar_tempty + 8 * b); }, dump, dump_ld ORX_DBG_FWD);
    }

    tc_fence_before();
    __syncthreads();
    if (warp == WARP_ALLOC) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

// ------------------------------------------------------------------ CTA-pair kernel (cta_group::2)
// For batches of more than 128 queries.  A cluster of two CTAs (one TPC) computes
//     D[256 queries x 256 rows] : UMMA M=256, each CTA holds its 128 queries (A) and HALF of the
// table tile (B, 128 rows); the hardware shares the B halves, so per CTA and K chunk only 32 KB are
// staged instead of 48 KB.  That halves the L2->smem traffic of the table operand and buys a 6-stage
// ring (3072 MMA cycles of prefetch instead of 2048).  Only the leader CTA issues MMAs; commits are
// multicast to both CTAs' barriers; both CTAs' TMA bytes are counted on the leader's full barrier;
// both CTAs' epilogues hand accumulators back by arriving on the leader's tmem-empty barrier.
template <bool TF32, bool DUMP = false, int C = CAND>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(UM_THREADS, 1)
scan_umma2_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_x,
                  const float *__restrict__ scale, uint32_t n_rows, int nq, int m_pairs, int n_slots, int k,
                  float margin, uint64_t *__restrict__ partial, float *__restrict__ floor_out,
                  uint32_t *__restrict__ gthr_all, float *__restrict__ dump, uint32_t dump_ld ORX_DBG_PARAM) {
    constexpr int ES = TF32 ? 4 : 2;
    constexpr int BLOCK_K = 128 / ES;
    constexpr int K_CHUNKS = ORX_DIM / BLOCK_K;
    constexpr uint32_t IDESC = make_idesc(TF32, 2 * TILE_M);

    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    float *s_scale = reinterpret_cast<float *>(smem + SMEM2_MAIN);
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem + SMEM2_MAIN + SMEM_SCALE);
    uint32_t *s_tmem = reinterpret_cast<uint32_t *>(bars + 20);
    const uint32_t smem_base = smem_u32(smem);
    const uint32_t bar_full = smem_u32(bars);              // [STAGES2]   (the leader's are used)
    const uint32_t bar_empty = bar_full + 8 * STAGES2;     // [STAGES2]   per CTA
    const uint32_t bar_tfull = bar_empty + 8 * STAGES2;    // [2]         per CTA
    const uint32_t bar_tempty = bar_tfull + 16;            // [2]         (the leader's are used)

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const uint32_t cta_rank = cluster_ctarank();
    const bool leader = cta_rank == 0;
    const int pair = blockIdx.x >> 1;
    const int m_pair = pair % m_pairs;
    const int slot = pair / m_pairs;
    const uint32_t n_tiles = (n_rows + TILE_N - 1) / TILE_N;

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES2; ++s) {
            mbar_init(bar_full + 8 * s, 1);
            mbar_init(bar_empty + 8 * s, 1);
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(bar_tfull + 8 * b, 1);
            mbar_init(bar_tempty + 8 * b, 8);             // 4 epilogue warps x 2 CTAs
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == WARP_ALLOC) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(s_tmem)),
                     "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    cluster_sync_all();                                    // barriers of BOTH CTAs are initialised
    tc_fence_after();
    const uint32_t tmem_base = *s_tmem;

    if (warp == WARP_TMA) {
        // ============================================== TMA producer (one per CTA, own smem)
        if (lane == 0) {
            asm volatile("prefetch.tensormap [%0];" ::"l"(&map_q) : "memory");
            asm volatile("prefetch.tensormap [%0];" ::"l"(&map_x) : "memory");
            const uint64_t hint_x = (m_pairs > 1) ? HINT_EVICT_NORMAL : HINT_EVICT_FIRST;
            uint32_t stage = 0, phase = 0;
            for (uint32_t t = slot; t < n_tiles; t += n_slots) {
                for (int kc = 0; kc < K_CHUNKS; ++kc) {
                    mbar_wait(bar_empty + 8 * stage, phase ^ 1);
                    const uint32_t sa = smem_base + stage * STAGE2_BYTES;
                    const uint32_t full_leader = map_to_cta(bar_full + 8 * stage, 0);
                    if (leader)
                        mbar_expect_tx(bar_full + 8 * stage, 2 * ((ORX_DBG(2) ? 0 : A_BYTES) + (ORX_DBG(4) ? 0 : B2_BYTES)));
                    if (!ORX_DBG(2))
                        tma_load_2d_pair(sa, &map_q, full_leader, kc * BLOCK_K,
                                         m_pair * 2 * TILE_M + (int)cta_rank * TILE_M, HINT_EVICT_LAST);
                    if (!ORX_DBG(4))
                        tma_load_2d_pair(sa + A_BYTES, &map_x, full_leader, kc * BLOCK_K,
                                         (int)(t * TILE_N) + (int)cta_rank * (TILE_N / 2), hint_x);
                    if (++stage == STAGES2) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == WARP_MMA) {
        // ============================================== MMA issuer (leader CTA, one lane)
        if (leader && lane == 0) {
            uint32_t stage = 0, phase = 0, buf = 0, tphase = 0;
            for (uint32_t t = slot; t < n_tiles; t += n_slots) {
                mbar_wait(bar_tempty + 8 * buf, tphase ^ 1);       // both CTAs drained this accumulator
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + buf * TILE_N;
                for (int kc = 0; kc < K_CHUNKS; ++kc) {
                    mbar_wait(bar_full + 8 * stage, phase);        // both CTAs' bytes have landed
                    tc_fence_after();
                    const uint32_t sa = smem_base + stage * STAGE2_BYTES;
                    const uint64_t adesc = make_desc_sw128(sa);
                    const uint64_t bdesc = make_desc_sw128(sa + A_BYTES);
#pragma unroll
                    for (int k4 = 0; k4 < 4; ++k4)
                        tc_mma_pair<TF32>(d_tmem, adesc + 2 * k4, bdesc + 2 * k4, IDESC, (kc | k4) != 0 ? 1u : 0u);
                    tc_commit_pair(bar_empty + 8 * stage);          // frees the stage in both CTAs
                    if (++stage == STAGES2) { stage = 0; phase ^= 1; }
                }
                tc_commit_pair(bar_tfull + 8 * buf);                // accumulators ready in both CTAs
                if (++buf == 2) { buf = 0; tphase ^= 1; }
            }
        }
    } else if (warp < 4) {
        // ============================================== epilogue (each CTA: its own 128 queries)
        const uint32_t tempty_leader = map_to_cta(bar_tempty, 0);
        epilogue_loop<DUMP, C>(m_pair * 2 * TILE_M + (int)cta_rank * TILE_M, nq, slot, n_slots, n_tiles, scale, n_rows, k, margin,
                            partial, floor_out, gthr_all, s_scale, bar_tfull, tmem_base, warp, lane,
                            [&](uint32_t b) { mbar_arrive_cluster(tempty_leader + 8 * b); }, dump, dump_ld ORX_DBG_FWD);
    }

    tc_fence_before();
    cluster_sync_all();                                    // nobody exits while the peer may still touch its smem / barriers
    if (warp == WARP_ALLOC) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

#if ORX_UMMA_ARES
// ------------------------------------------------------------------ CTA pairs with HALF of the query tile resident
// What bounds the pair kernel is the operand bytes each SM has to take in per flop (ncu: 40 B/clk/SM of TMA reads at 61 %
// tensor-pipe activity; multicasting the table tile across pairs changes the L2 reads but not this, and changes nothing --
// DESIGN.md 4.1).  Per CTA and table tile the pair kernel ingests its 256 KB query tile (again and again: it does not fit
// beside the ring) plus its 256 KB half of the table tile.  Here the EVEN K chunks of the query tile (128 KB) are loaded once
// and stay in shared memory for the life of the CTA; only the odd chunks are re-streamed: 384 KB instead of 512 KB per
// tile (-25 % ingest per flop).  Layout: 8 resident A chunks | 2-slot A ring | 4-stage B ring.  bf16 tables only (a tf32
// tile's resident share would be a quarter and its ring too shallow).
constexpr int R_STAGES = 4;
constexpr int R_ARES_CHUNKS = 8;
constexpr int R_OFF_ARING = R_ARES_CHUNKS * A_BYTES;                       // 128 KB
constexpr int R_OFF_BRING = R_OFF_ARING + 2 * A_BYTES;                     // 160 KB
constexpr int R_OFF_SCALE = R_OFF_BRING + R_STAGES * B2_BYTES;             // 224 KB
constexpr int SMEM2R_TOTAL = R_OFF_SCALE + SMEM_SCALE + 256;               // 231,680 B (the base must be 1 KB aligned)

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(UM_THREADS, 1)
scan_umma2r_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_x,
                   const float *__restrict__ scale, uint32_t n_rows, int nq, int m_pairs, int n_slots, int k,
                   float margin, uint64_t *__restrict__ partial, float *__restrict__ floor_out,
                   uint32_t *__restrict__ gthr_all) {
    constexpr int BLOCK_K = 64;                     // bf16 elements per 128-byte swizzle row
    constexpr int K_CHUNKS = ORX_DIM / BLOCK_K;     // 16
    constexpr uint32_t IDESC = make_idesc(false, 2 * TILE_M);
    static_assert(K_CHUNKS == 2 * R_ARES_CHUNKS && K_CHUNKS % R_STAGES == 0, "even chunks resident, ring divides the tile");

    extern __shared__ __align__(1024) uint8_t smem_al[];
    uint8_t *smem = smem_al;
    float *s_scale = reinterpret_cast<float *>(smem + R_OFF_SCALE);
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem + R_OFF_SCALE + SMEM_SCALE);
    uint32_t *s_tmem = reinterpret_cast<uint32_t *>(bars + 20);
    const uint32_t smem_base = smem_u32(smem);
    if ((smem_base & 1023u) != 0u) __trap();               // SWIZZLE_128B tiles need a 1 KB aligned base (no slack to align up)
    const uint32_t bar_full = smem_u32(bars);              // [R_STAGES]  (the leader's are used)
    const uint32_t bar_empty = bar_full + 8 * R_STAGES;    // [R_STAGES]  per CTA
    const uint32_t bar_tfull = bar_empty + 8 * R_STAGES;   // [2]         per CTA
    const uint32_t bar_tempty = bar_tfull + 16;            // [2]         (the leader's are used)
    const uint32_t bar_ares = bar_tempty + 16;             // [1]         resident chunks of both CTAs have landed (leader's)

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const uint32_t cta_rank = cluster_ctarank();
    const bool leader = cta_rank == 0;
    const int pair = blockIdx.x >> 1;
    const int m_pair = pair % m_pairs;
    const int slot = pair / m_pairs;
    const uint32_t n_tiles = (n_rows + TILE_N - 1) / TILE_N;

    if (threadIdx.x == 0) {
        for (int s = 0; s < R_STAGES; ++s) {
            mbar_init(bar_full + 8 * s, 1);
            mbar_init(bar_empty + 8 * s, 1);
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(bar_tfull + 8 * b, 1);
            mbar_init(bar_tempty + 8 * b, 8);             // 4 epilogue warps x 2 CTAs
        }
        mbar_init(bar_ares, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == WARP_ALLOC) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(s_tmem)),
                     "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = *s_tmem;
    const int q_row = m_pair * 2 * TILE_M + (int)cta_rank * TILE_M;

    if (warp == WARP_TMA) {
        // ============================================== TMA producer (one per CTA, own smem)
        if (lane == 0) {
            asm volatile("prefetch.tensormap [%0];" ::"l"(&map_q) : "memory");
            asm volatile("prefetch.tensormap [%0];" ::"l"(&map_x) : "memory");
            const uint64_t hint_x = (m_pairs > 1) ? HINT_EVICT_NORMAL : HINT_EVICT_FIRST;
            // the resident half of the query tile: even K chunks, once
            const uint32_t ares_leader = map_to_cta(bar_ares, 0);
            if (leader) mbar_expect_tx(bar_ares, 2 * R_ARES_CHUNKS * A_BYTES);
            for (int i = 0; i < R_ARES_CHUNKS; ++i)
                tma_load_2d_pair(smem_base + i * A_BYTES, &map_q, ares_leader, (2 * i) * BLOCK_K, q_row, HINT_EVICT_LAST);
            uint32_t phase = 0;
            for (uint32_t t = slot; t < n_tiles; t += n_slots) {
                for (int kc = 0; kc < K_CHUNKS; ++kc) {
                    const uint32_t stage = kc & (R_STAGES - 1);
                    const bool streamed = (kc & 1) != 0;
                    mbar_wait(bar_empty + 8 * stage, phase ^ 1);   // chunk kc-4 is consumed: its B stage AND its A slot are free
                    const uint32_t full_leader = map_to_cta(bar_full + 8 * stage, 0);
                    if (leader) mbar_expect_tx(bar_full + 8 * stage, 2 * (B2_BYTES + (streamed ? A_BYTES : 0)));
                    if (streamed)
                        tma_load_2d_pair(smem_base + R_OFF_ARING + ((kc >> 1) & 1) * A_BYTES, &map_q, full_leader, kc * BLOCK_K,
                                         q_row, HINT_EVICT_LAST);
                    tma_load_2d_pair(smem_base + R_OFF_BRING + stage * B2_BYTES, &map_x, full_leader, kc * BLOCK_K,
                                     (int)(t * TILE_N) + (int)cta_rank * (TILE_N / 2), hint_x);
                    if (stage == R_STAGES - 1) phase ^= 1;
                }
            }
        }
    } else if (warp == WARP_MMA) {
        // ============================================== MMA issuer (leader CTA, one lane)
        if (leader && lane == 0) {
            mbar_wait(bar_ares, 0);                                // both CTAs' resident chunks are in shared memory
            uint32_t phase = 0, buf = 0, tphase = 0;
            for (uint32_t t = slot; t < n_tiles; t += n_slots) {
                mbar_wait(bar_tempty + 8 * buf, tphase ^ 1);       // both CTAs drained this accumulator
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + buf * TILE_N;
                for (int kc = 0; kc < K_CHUNKS; ++kc) {
                    const uint32_t stage = kc & (R_STAGES - 1);
                    mbar_wait(bar_full + 8 * stage, phase);        // both CTAs' bytes of this chunk have landed
                    tc_fence_after();
                    const uint32_t a_addr = (kc & 1) ? smem_base + R_OFF_ARING + ((kc >> 1) & 1) * A_BYTES
                                                     : smem_base + (kc >> 1) * A_BYTES;
                    const uint64_t adesc = make_desc_sw128(a_addr);
                    const uint64_t bdesc = make_desc_sw128(smem_base + R_OFF_BRING + stage * B2_BYTES);
#pragma unroll
                    for (int k4 = 0; k4 < 4; ++k4)
                        tc_mma_pair<false>(d_tmem, adesc + 2 * k4, bdesc + 2 * k4, IDESC, (kc | k4) != 0 ? 1u : 0u);
                    tc_commit_pair(bar_empty + 8 * stage);          // frees the B stage (and the A slot) in both CTAs
                    if (stage == R_STAGES - 1) phase ^= 1;
                }
                tc_commit_pair(bar_tfull + 8 * buf);                // accumulators ready in both CTAs
                if (++buf == 2) { buf = 0; tphase ^= 1; }
            }
        }
    } else if (warp < 4) {
        // ============================================== epilogue (each CTA: its own 128 queries)
        const uint32_t tempty_leader = map_to_cta(bar_tempty, 0);
        epilogue_loop<false, CAND>(q_row, nq, slot, n_slots, n_tiles, scale, n_rows, k, margin,
                             partial, floor_out, gthr_all, s_scale, bar_tfull, tmem_base, warp, lane,
                             [&](uint32_t b) { mbar_arrive_cluster(tempty_leader + 8 * b); }, nullptr, 0u
#ifdef ORX_DEBUG_VARIANTS
                             , 0
#endif
        );
    }

    tc_fence_before();
    cluster_sync_all();
    if (warp == WARP_ALLOC) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

#endif  // ORX_UMMA_ARES

#if ORX_UMMA_QUADS
// ------------------------------------------------------------------ two CTA pairs per cluster (cluster of 4)
// The pair kernel's L2 -> SM traffic is what bounds it (ncu: 9.7 TB/s of TMA reads at 61 % tensor-pipe activity; B300_MICROARCH.md puts
// the L2 slice throughput cap near 6300 B/cycle): every pair streams its own copy of the table tile although the pairs
// of a slot read the SAME tile.  Here two pairs (512 queries) form ONE cluster and share the tile through TMA multicast:
// CTA r of the cluster (pair p = r >> 1, parity h = r & 1) fetches one QUARTER of the tile -- rows [128 h + 64 p, +64) --
// and multicasts it into the two CTAs of parity h, so each table byte leaves L2 once per cluster instead of once per
// pair (-25 % L2 -> SM bytes per flop).  Both pairs consume a stage before anyone refills it (the stage's empty barrier
// counts both leaders' commits, multicast to all four CTAs), so the pairs advance in lock step.
template <bool TF32>
__global__ void __cluster_dims__(4, 1, 1) __launch_bounds__(UM_THREADS, 1)
scan_umma4_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_x,
                  const float *__restrict__ scale, uint32_t n_rows, int nq, int m_quads, int n_slots, int k,
                  float margin, uint64_t *__restrict__ partial, float *__restrict__ floor_out,
                  uint32_t *__restrict__ gthr_all) {
    constexpr int ES = TF32 ? 4 : 2;
    constexpr int BLOCK_K = 128 / ES;
    constexpr int K_CHUNKS = ORX_DIM / BLOCK_K;
    constexpr uint32_t IDESC = make_idesc(TF32, 2 * TILE_M);
    constexpr int BQ_BYTES = (TILE_N / 4) * 128;          // one quarter of the table tile per K chunk: 8 KB

    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    float *s_scale = reinterpret_cast<float *>(smem + SMEM2_MAIN);
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem + SMEM2_MAIN + SMEM_SCALE);
    uint32_t *s_tmem = reinterpret_cast<uint32_t *>(bars + 20);
    const uint32_t smem_base = smem_u32(smem);
    const uint32_t bar_full = smem_u32(bars);              // [STAGES2]   (each pair leader's are used)
    const uint32_t bar_empty = bar_full + 8 * STAGES2;     // [STAGES2]   per CTA, 2 arrivals: both pairs consumed the stage
    const uint32_t bar_tfull = bar_empty + 8 * STAGES2;    // [2]         per CTA
    const uint32_t bar_tempty = bar_tfull + 16;            // [2]         (each pair leader's are used)

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const uint32_t cta_rank = cluster_ctarank();           // 0..3
    const uint32_t pair_in_cluster = cta_rank >> 1, parity = cta_rank & 1u, leader_rank = cta_rank & ~1u;
    const bool leader = parity == 0;
    const int quad = blockIdx.x >> 2;
    const int m_pair = 2 * (quad % m_quads) + (int)pair_in_cluster;
    const int slot = quad / m_quads;
    const uint32_t n_tiles = (n_rows + TILE_N - 1) / TILE_N;

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES2; ++s) {
            mbar_init(bar_full + 8 * s, 1);
            mbar_init(bar_empty + 8 * s, 2);
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(bar_tfull + 8 * b, 1);
            mbar_init(bar_tempty + 8 * b, 8);             // 4 epilogue warps x 2 CTAs of the pair
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == WARP_ALLOC) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(s_tmem)),
                     "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    cluster_sync_all();                                    // barriers of all four CTAs are initialised
    tc_fence_after();
    const uint32_t tmem_base = *s_tmem;

    if (warp == WARP_TMA) {
        // ============================================== TMA producer (one per CTA)
        if (lane == 0) {
            asm volatile("prefetch.tensormap [%0];" ::"l"(&map_q) : "memory");
            asm volatile("prefetch.tensormap [%0];" ::"l"(&map_x) : "memory");
            const uint16_t mc_mask = (uint16_t)((1u << parity) | (1u << (parity + 2)));       // the two CTAs holding this half
            uint32_t stage = 0, phase = 0;
            for (uint32_t t = slot; t < n_tiles; t += n_slots) {
                for (int kc = 0; kc < K_CHUNKS; ++kc) {
                    mbar_wait(bar_empty + 8 * stage, phase ^ 1);          // BOTH pairs are done with this stage
                    const uint32_t sa = smem_base + stage * STAGE2_BYTES;
                    const uint32_t full_leader = map_to_cta(bar_full + 8 * stage, leader_rank);
                    if (leader) mbar_expect_tx(bar_full + 8 * stage, 2 * (A_BYTES + B2_BYTES));
                    tma_load_2d_pair(sa, &map_q, full_leader, kc * BLOCK_K, m_pair * 2 * TILE_M + (int)parity * TILE_M,
                                     HINT_EVICT_LAST);
                    // my quarter of the table tile, into both CTAs of my parity (offset: quarter `pair_in_cluster` of the half)
                    tma_load_2d_pair_mc(sa + A_BYTES + pair_in_cluster * BQ_BYTES, &map_x, full_leader, kc * BLOCK_K,
                                        (int)(t * TILE_N) + (int)parity * (TILE_N / 2) + (int)pair_in_cluster * (TILE_N / 4),
                                        mc_mask, HINT_EVICT_NORMAL);
                    if (++stage == STAGES2) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == WARP_MMA) {
        // ============================================== MMA issuer (each pair's leader CTA, one lane)
        if (leader && lane == 0) {
            const uint16_t pair_mask = (uint16_t)(3u << (2 * pair_in_cluster));
            uint32_t stage = 0, phase = 0, buf = 0, tphase = 0;
            for (uint32_t t = slot; t < n_tiles; t += n_slots) {
                mbar_wait(bar_tempty + 8 * buf, tphase ^ 1);       // both CTAs of the pair drained this accumulator
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + buf * TILE_N;
                for (int kc = 0; kc < K_CHUNKS; ++kc) {
                    mbar_wait(bar_full + 8 * stage, phase);        // the pair's A and both halves of the tile have landed
                    tc_fence_after();
                    const uint32_t sa = smem_base + stage * STAGE2_BYTES;
                    const uint64_t adesc = make_desc_sw128(sa);
                    const uint64_t bdesc = make_desc_sw128(sa + A_BYTES);
#pragma unroll
                    for (int k4 = 0; k4 < 4; ++k4)
                        tc_mma_pair<TF32>(d_tmem, adesc + 2 * k4, bdesc + 2 * k4, IDESC, (kc | k4) != 0 ? 1u : 0u);
                    tc_commit_mc(bar_empty + 8 * stage, (uint16_t)0xF);      // one of the two arrivals every CTA waits for
                    if (++stage == STAGES2) { stage = 0; phase ^= 1; }
                }
                tc_commit_mc(bar_tfull + 8 * buf, pair_mask);       // accumulators ready in both CTAs of this pair
                if (++buf == 2) { buf = 0; tphase ^= 1; }
            }
        }
    } else if (warp < 4) {
        // ============================================== epilogue (each CTA: its own 128 queries)
        const uint32_t tempty_leader = map_to_cta(bar_tempty, leader_rank);
        epilogue_loop<false, CAND>(m_pair * 2 * TILE_M + (int)parity * TILE_M, nq, slot, n_slots, n_tiles, scale, n_rows, k, margin,
                             partial, floor_out, gthr_all, s_scale, bar_tfull, tmem_base, warp, lane,
                             [&](uint32_t b) { mbar_arrive_cluster(tempty_leader + 8 * b); }, nullptr, 0u
#ifdef ORX_DEBUG_VARIANTS
                             , 0
#endif
        );
    }

    tc_fence_before();
    cluster_sync_all();                                    // nobody exits while a peer may still write its smem / barriers
    if (warp == WARP_ALLOC) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

#endif  // ORX_UMMA_QUADS

// ------------------------------------------------------------------------------ host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

thread_local std::string g_umma_err;

EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
        cudaGetLastError();
    });
    return fn;
}

// [rows, 1024] K-major matrix, box = one 128-byte swizzle row of K x box_rows rows
bool encode_map(CUtensorMap *map, const void *base, uint64_t rows, bool fp32, uint32_t box_rows) {
    EncodeTiledFn fn = encode_fn();
    if (!fn) { g_umma_err = "cuTensorMapEncodeTiled entry point not found"; return false; }
    const cuuint64_t dims[2] = {ORX_DIM, rows};
    const cuuint64_t strides[1] = {(cuuint64_t)ORX_DIM * (fp32 ? 4 : 2)};
    const cuuint32_t box[2] = {(cuuint32_t)(fp32 ? 32 : 64), box_rows};
    const cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(map, fp32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2,
                    const_cast<void *>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        g_umma_err = "cuTensorMapEncodeTiled failed with CUresult " + std::to_string((int)r);
        return false;
    }
    return true;
}

}  // namespace

struct UmmaPlan {
    int device = 0;
    int sms = 1;
    bool attr_set = false;
#ifdef ORX_DEBUG_VARIANTS
    int dbg = 0;                     // ORX_UMMA_DEBUG: timing experiments (results are garbage when set)
#endif
    bool use_pairs = true;           // variant builds: ORX_UMMA_PAIRS=0 keeps every batch on the 1-CTA kernel
    bool use_quads = ORX_UMMA_QUADS != 0;
    bool use_ares = ORX_UMMA_ARES != 0;
    int max_quads[2] = {-1, -1};     // co-resident clusters of 4 (tf32 / bf16 kernel), queried once
    uint64_t *partial = nullptr;
    size_t partial_n = 0;
    float *floor = nullptr;
    size_t floor_n = 0;
    uint32_t *gthr = nullptr;
    size_t gthr_n = 0;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
};

UmmaPlan *umma_plan_create(int device) {
    UmmaPlan *p = new UmmaPlan();
    p->device = device;
    cudaDeviceGetAttribute(&p->sms, cudaDevAttrMultiProcessorCount, device);
#ifdef ORX_DEBUG_VARIANTS
    const char *env = getenv("ORX_UMMA_PAIRS");
    if (env && env[0] == '0') p->use_pairs = false;
    env = getenv("ORX_UMMA_DEBUG");
    if (env) p->dbg = atoi(env);
#endif
    return p;
}
void umma_plan_destroy(UmmaPlan *p) {
    if (!p) return;
    cudaFree(p->partial);
    cudaFree(p->floor);
    cudaFree(p->gthr);
    delete p;
}
const char *umma_last_error() { return g_umma_err.c_str(); }

bool umma_should_use(const UmmaPlan *p, int nq, int k, uint32_t n_rows) {
    // one table pass for the whole batch beats nq GEMV passes as soon as nq >= 2
    return p != nullptr && nq >= 2 && k <= UMMA_MAX_K && n_rows >= 4096;
}

static bool ensure_attrs(UmmaPlan *p) {
    if (p->attr_set) return true;
    cudaError_t e = cudaSuccess;
    auto set = [&](const void *fn, int bytes) {
        if (e == cudaSuccess) e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    };
    set((const void *)scan_umma_kernel<true, false>, SMEM_TOTAL);
    set((const void *)scan_umma_kernel<false, false>, SMEM_TOTAL);
    set((const void *)scan_umma_kernel<true, true>, SMEM_TOTAL);
    set((const void *)scan_umma_kernel<false, true>, SMEM_TOTAL);
    set((const void *)scan_umma2_kernel<true, false>, SMEM2_TOTAL);
    set((const void *)scan_umma2_kernel<false, false>, SMEM2_TOTAL);
    set((const void *)scan_umma2_kernel<true, true>, SMEM2_TOTAL);
    set((const void *)scan_umma2_kernel<false, true>, SMEM2_TOTAL);
    set((const void *)scan_umma_kernel<true, false, CAND_WIDE>, SMEM_TOTAL);
    set((const void *)scan_umma_kernel<false, false, CAND_WIDE>, SMEM_TOTAL);
    set((const void *)scan_umma2_kernel<true, false, CAND_WIDE>, SMEM2_TOTAL);
    set((const void *)scan_umma2_kernel<false, false, CAND_WIDE>, SMEM2_TOTAL);
#if ORX_UMMA_ARES
    set((const void *)scan_umma2r_kernel, SMEM2R_TOTAL);
#endif
#if ORX_UMMA_QUADS
    set((const void *)scan_umma4_kernel<true>, SMEM2_TOTAL);
    set((const void *)scan_umma4_kernel<false>, SMEM2_TOTAL);
#endif
    if (e != cudaSuccess) {
        g_umma_err = cudaGetErrorString(e);
        return false;
    }
    p->attr_set = true;
    return true;
}

#if ORX_UMMA_QUADS
// how many clusters of 4 CTAs of the quad kernel the device can hold at once (0: do not use it)
static int max_active_quads(UmmaPlan *p, bool tf32) {
    int &cached = p->max_quads[tf32 ? 0 : 1];
    if (cached >= 0) return cached;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(p->sms / 4 * 4));
    cfg.blockDim = dim3(UM_THREADS);
    cfg.dynamicSmemBytes = SMEM2_TOTAL;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 4;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    int n = 0;
    cudaError_t e = tf32 ? cudaOccupancyMaxActiveClusters(&n, scan_umma4_kernel<true>, &cfg)
                         : cudaOccupancyMaxActiveClusters(&n, scan_umma4_kernel<false>, &cfg);
    if (e != cudaSuccess) {
        cudaGetLastError();
        n = 0;
    }
    cached = n;
    return n;
}
#endif

template <typename T>
static cudaError_t ensure_buf(T *&ptr, size_t &have, size_t want) {
    if (want <= have) return cudaSuccess;
    if (ptr) cudaFree(ptr);
    ptr = nullptr;
    have = 0;
    cudaError_t e = cudaMalloc(&ptr, want * sizeof(T));
    if (e == cudaSuccess) have = want;
    return e;
}

int umma_search(UmmaPlan *p, int dtype, const void *table, const float *scale, const double *n2,
                const orx_id *row_ids, uint32_t n_rows, const float *q_dev, const float *qhat,
                const __nv_bfloat16 *qhat16, const QueryPrep *prep, int nq, int k, const ResultOut &out,
                const PublishArgs &pub, const DoneArgs &done, cudaStream_t st, uint64_t *launch_counter,
                cudaEvent_t ev_begin, cudaEvent_t ev_end) {
    const bool tf32 = dtype == ORX_DTYPE_F32;
    const double eps = tf32 ? EPS_UMMA_TF32 : EPS_UMMA_BF16;
    const float margin = (float)(2.0 * eps + 1e-6);
    if (!ensure_attrs(p)) return ORX_ERR_CUDA;
    if (k > UMMA_MAX_K) { g_umma_err = "k beyond the candidate lists"; return ORX_ERR_INVALID; }
    const bool wide = k > CAND_NARROW_MAX_K;   // lists of 160 instead of 64 keys per (query, CTA)
    const int cand = wide ? CAND_WIDE : CAND;
    constexpr int MAX_Q = 2048;              // 16 query tiles -> 9 row slots -> 144 CTAs
    for (int q0 = 0; q0 < nq; q0 += MAX_Q) {
        const int m = nq - q0 < MAX_Q ? nq - q0 : MAX_Q;
        // batches beyond one query tile run on CTA pairs (cta_group::2, 256 queries per pair)
        const bool pairs = m > TILE_M && p->use_pairs;
        const int m_tiles = pairs ? (m + 2 * TILE_M - 1) / (2 * TILE_M) : (m + TILE_M - 1) / TILE_M;
        const uint32_t n_tiles = (n_rows + TILE_N - 1) / TILE_N;
        // clusters of 4 (two pairs sharing the table tile by multicast) when the batch has an even number of pair tiles
        int quads_fit = 0;
#if ORX_UMMA_QUADS
        if (pairs && p->use_quads && !wide && m_tiles % 2 == 0) quads_fit = max_active_quads(p, tf32) / (m_tiles / 2);
#endif
        const bool quads = quads_fit >= 1;
        int n_slots = quads ? quads_fit : (pairs ? p->sms / 2 : p->sms) / m_tiles;
        if (n_slots < 1) n_slots = 1;
        if ((uint32_t)n_slots > n_tiles) n_slots = (int)n_tiles;
        cudaError_t e = ensure_buf(p->partial, p->partial_n, (size_t)m * n_slots * cand);
        if (e == cudaSuccess) e = ensure_buf(p->floor, p->floor_n, (size_t)m * n_slots);
        if (e == cudaSuccess) e = ensure_buf(p->gthr, p->gthr_n, (size_t)m);
        if (e != cudaSuccess) { g_umma_err = cudaGetErrorString(e); return ORX_ERR_CUDA; }
        CUtensorMap map_q, map_x;
        const void *qbase = tf32 ? (const void *)(qhat + (size_t)q0 * ORX_DIM) : (const void *)(qhat16 + (size_t)q0 * ORX_DIM);
        // qhat / qhat16 are padded with zero rows to a multiple of 256 by the caller (stage_queries)
        if (!encode_map(&map_q, qbase, (uint64_t)((m + 255) / 256 * 256), tf32, TILE_M)) return ORX_ERR_CUDA;
        if (!encode_map(&map_x, table, (uint64_t)n_rows, tf32, quads ? TILE_N / 4 : (pairs ? TILE_N / 2 : TILE_N))) return ORX_ERR_CUDA;
        cudaMemsetAsync(p->gthr, 0, (size_t)m * sizeof(uint32_t), st);
        if (ev_begin && q0 == 0) cudaEventRecord(ev_begin, st);
        if (false) {
#if ORX_UMMA_QUADS
        } else if (quads) {
            const int grid = 4 * (m_tiles / 2) * n_slots;
            if (tf32)
                scan_umma4_kernel<true><<<grid, UM_THREADS, SMEM2_TOTAL, st>>>(map_q, map_x, scale, n_rows, m, m_tiles / 2, n_slots,
                                                                               k, margin, p->partial, p->floor, p->gthr);
            else
                scan_umma4_kernel<false><<<grid, UM_THREADS, SMEM2_TOTAL, st>>>(map_q, map_x, scale, n_rows, m, m_tiles / 2, n_slots,
                                                                                k, margin, p->partial, p->floor, p->gthr);
#endif
#if ORX_UMMA_ARES
        } else if (pairs && !tf32 && p->use_ares && !wide) {
            const int grid = 2 * m_tiles * n_slots;
            scan_umma2r_kernel<<<grid, UM_THREADS, SMEM2R_TOTAL, st>>>(map_q, map_x, scale, n_rows, m, m_tiles, n_slots, k, margin,
                                                                       p->partial, p->floor, p->gthr);
#endif
        } else if (pairs) {
            const int grid = 2 * m_tiles * n_slots;
#define ORX_LAUNCH_UMMA2(TF, C)                                                                                           \
    scan_umma2_kernel<TF, false, C><<<grid, UM_THREADS, SMEM2_TOTAL, st>>>(map_q, map_x, scale, n_rows, m, m_tiles, n_slots, k, \
                                                                           margin, p->partial, p->floor, p->gthr, nullptr, 0u ORX_DBG_ARG(p))
            if (tf32 && wide) ORX_LAUNCH_UMMA2(true, CAND_WIDE);
            else if (tf32) ORX_LAUNCH_UMMA2(true, CAND);
            else if (wide) ORX_LAUNCH_UMMA2(false, CAND_WIDE);
            else ORX_LAUNCH_UMMA2(false, CAND);
#undef ORX_LAUNCH_UMMA2
        } else {
            const int grid = m_tiles * n_slots;
#define ORX_LAUNCH_UMMA1(TF, C)                                                                                          \
    scan_umma_kernel<TF, false, C><<<grid, UM_THREADS, SMEM_TOTAL, st>>>(map_q, map_x, scale, n_rows, m, m_tiles, n_slots, k,  \
                                                                         margin, p->partial, p->floor, p->gthr, nullptr, 0u ORX_DBG_ARG(p))
            if (tf32 && wide) ORX_LAUNCH_UMMA1(true, CAND_WIDE);
            else if (tf32) ORX_LAUNCH_UMMA1(true, CAND);
            else if (wide) ORX_LAUNCH_UMMA1(false, CAND_WIDE);
            else ORX_LAUNCH_UMMA1(false, CAND);
#undef ORX_LAUNCH_UMMA1
        }
        if (ev_end && q0 + MAX_Q >= nq) cudaEventRecord(ev_end, st);
        launch_finalize(dtype, table, n2, row_ids, q_dev + (size_t)q0 * ORX_DIM, prep + q0, p->partial, n_slots, cand / 32, m,
                        k, n_rows, eps, out, q0, pub, done, st, p->floor);
#ifdef ORX_DEBUG_VARIANTS
        if (p->dbg && out.flags) launch_flags_from_prep(prep + q0, m, out.flags + q0, st);   // timing experiments: no fallbacks
#endif
        *launch_counter += 2;
        e = cudaGetLastError();
        if (e != cudaSuccess) { g_umma_err = cudaGetErrorString(e); return ORX_ERR_CUDA; }
    }
    return ORX_OK;
}

// Diagnostic: the scaled coarse scores of the tcgen05 pass, out[row * nq + query] (device memory, [n_rows, nq] fp32), through
// the SAME TMA / UMMA / TMEM path as the search (only the epilogue differs: it writes instead of selecting).
int umma_dump_scores(UmmaPlan *p, int dtype, const void *table, const float *scale, uint32_t n_rows, const float *qhat,
                     const __nv_bfloat16 *qhat16, int nq, bool pairs, float *out, cudaStream_t st) {
    const bool tf32 = dtype == ORX_DTYPE_F32;
    if (!ensure_attrs(p)) return ORX_ERR_CUDA;
    if (nq < 1 || nq > 2048) { g_umma_err = "1..2048 queries"; return ORX_ERR_INVALID; }
    const int m_tiles = pairs ? (nq + 2 * TILE_M - 1) / (2 * TILE_M) : (nq + TILE_M - 1) / TILE_M;
    const uint32_t n_tiles = (n_rows + TILE_N - 1) / TILE_N;
    int n_slots = (pairs ? p->sms / 2 : p->sms) / m_tiles;
    if (n_slots < 1) n_slots = 1;
    if ((uint32_t)n_slots > n_tiles) n_slots = (int)n_tiles;
    CUtensorMap map_q, map_x;
    const void *qbase = tf32 ? (const void *)qhat : (const void *)qhat16;
    if (!encode_map(&map_q, qbase, (uint64_t)((nq + 255) / 256 * 256), tf32, TILE_M)) return ORX_ERR_CUDA;
    if (!encode_map(&map_x, table, (uint64_t)n_rows, tf32, pairs ? TILE_N / 2 : TILE_N)) return ORX_ERR_CUDA;
    // the selection state is unused in DUMP mode but the kernel signature wants valid pointers
    cudaError_t e = ensure_buf(p->partial, p->partial_n, (size_t)nq * n_slots * CAND);
    if (e == cudaSuccess) e = ensure_buf(p->floor, p->floor_n, (size_t)nq * n_slots);
    if (e == cudaSuccess) e = ensure_buf(p->gthr, p->gthr_n, (size_t)nq);
    if (e != cudaSuccess) { g_umma_err = cudaGetErrorString(e); return ORX_ERR_CUDA; }
    cudaMemsetAsync(p->gthr, 0, (size_t)nq * sizeof(uint32_t), st);
    if (pairs) {
        const int grid = 2 * m_tiles * n_slots;
        if (tf32) scan_umma2_kernel<true, true><<<grid, UM_THREADS, SMEM2_TOTAL, st>>>(map_q, map_x, scale, n_rows, nq, m_tiles, n_slots, 12, 0.f, p->partial, p->floor, p->gthr, out, (uint32_t)nq ORX_DBG_ARG(p));
        else scan_umma2_kernel<false, true><<<grid, UM_THREADS, SMEM2_TOTAL, st>>>(map_q, map_x, scale, n_rows, nq, m_tiles, n_slots, 12, 0.f, p->partial, p->floor, p->gthr, out, (uint32_t)nq ORX_DBG_ARG(p));
    } else {
        const int grid = m_tiles * n_slots;
        if (tf32) scan_umma_kernel<true, true><<<grid, UM_THREADS, SMEM_TOTAL, st>>>(map_q, map_x, scale, n_rows, nq, m_tiles, n_slots, 12, 0.f, p->partial, p->floor, p->gthr, out, (uint32_t)nq ORX_DBG_ARG(p));
        else scan_umma_kernel<false, true><<<grid, UM_THREADS, SMEM_TOTAL, st>>>(map_q, map_x, scale, n_rows, nq, m_tiles, n_slots, 12, 0.f, p->partial, p->floor, p->gthr, out, (uint32_t)nq ORX_DBG_ARG(p));
    }
    e = cudaGetLastError();
    if (e != cudaSuccess) { g_umma_err = cudaGetErrorString(e); return ORX_ERR_CUDA; }
    return ORX_OK;
}

}  // namespace orx
