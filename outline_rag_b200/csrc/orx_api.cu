// orx C-ABI (include/orx.h) and the host side of the engine: the device-resident table,
// the chunk-id -> row map, search orchestration (scan -> finalize -> proof -> fallbacks),
// upsert / delete planning.  One orx_index = one GPU; sharding lives above (sharded.py).
#include <cuda_runtime.h>
#include <cuda_bf16.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <functional>
#include <memory>
#include <thread>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <string>
#include <unordered_map>
#include <vector>

#include "internal.h"
#include "scan_umma.h"

namespace {

thread_local std::string g_err;

int fail(int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

#define CK(call)                                                                          \
    do {                                                                                  \
        cudaError_t e_ = (call);                                                          \
        if (e_ != cudaSuccess)                                                            \
            return fail(ORX_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), \
                        __FILE__, __LINE__);                                              \
    } while (0)

struct IdHash {
    size_t operator()(const orx_id &a) const { return (size_t)orx::id_hash(a); }
};
struct IdEq {
    bool operator()(const orx_id &a, const orx_id &b) const { return a.hi == b.hi && a.lo == b.lo; }
};

// chunk id -> row: open addressing with linear probing over a power-of-two table kept at most half full (one cache line
// per look-up in the common case; std::unordered_map's node-per-entry layout cost ~150 ns per operation, which was the
// largest host term of an upsert / delete / filter resolution / cold-start batch).  Deletions leave tombstones that the
// next rehash drops.
class IdMap {
    struct Entry {
        orx_id id;
        uint32_t row;
        uint32_t state;          // 0 empty, 1 used, 2 tombstone
    };
    std::vector<Entry> tab_;
    size_t used_ = 0, filled_ = 0;   // live entries / live + tombstones
    static size_t hash(const orx_id &a) { return IdHash()(a); }
    void rehash(size_t want_entries) {
        size_t cap = 64;
        while (cap < want_entries * 2) cap <<= 1;
        std::vector<Entry> old;
        old.swap(tab_);
        tab_.assign(cap, Entry{{0, 0}, 0, 0});
        used_ = filled_ = 0;
        for (const Entry &e : old)
            if (e.state == 1) set(e.id, e.row);
    }

public:
    void reserve(size_t n) {
        if (tab_.size() < n * 2) rehash(n);
    }
    void clear() {
        for (Entry &e : tab_) e.state = 0;
        used_ = filled_ = 0;
    }
    const uint32_t *find(const orx_id &id) const {
        if (tab_.empty()) return nullptr;
        const size_t mask = tab_.size() - 1;
        for (size_t i = hash(id) & mask;; i = (i + 1) & mask) {
            const Entry &e = tab_[i];
            if (e.state == 0) return nullptr;
            if (e.state == 1 && e.id.hi == id.hi && e.id.lo == id.lo) return &e.row;
        }
    }
    void set(const orx_id &id, uint32_t row) {          // insert or assign
        if ((filled_ + 1) * 2 > tab_.size()) rehash(std::max<size_t>(used_ + 1, 32) * 2);
        const size_t mask = tab_.size() - 1;
        size_t grave = (size_t)-1;
        for (size_t i = hash(id) & mask;; i = (i + 1) & mask) {
            Entry &e = tab_[i];
            if (e.state == 1) {
                if (e.id.hi == id.hi && e.id.lo == id.lo) {
                    e.row = row;
                    return;
                }
            } else if (e.state == 2) {
                if (grave == (size_t)-1) grave = i;
            } else {
                Entry &dst = grave != (size_t)-1 ? tab_[grave] : e;
                if (grave == (size_t)-1) ++filled_;
                dst.id = id;
                dst.row = row;
                dst.state = 1;
                ++used_;
                return;
            }
        }
    }
    bool erase(const orx_id &id) {
        if (tab_.empty()) return false;
        const size_t mask = tab_.size() - 1;
        for (size_t i = hash(id) & mask;; i = (i + 1) & mask) {
            Entry &e = tab_[i];
            if (e.state == 0) return false;
            if (e.state == 1 && e.id.hi == id.hi && e.id.lo == id.lo) {
                e.state = 2;
                --used_;
                return true;
            }
        }
    }
};

bool is_device_ptr(const void *p) {
    if (!p) return false;
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged;
}
// the device a device pointer lives on, or -1 for host memory
int ptr_device(const void *p) {
    if (!p) return -1;
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
        cudaGetLastError();
        return -1;
    }
    return (at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged) ? at.device : -1;
}

size_t elem_size(int dtype) { return dtype == ORX_DTYPE_F32 ? 4 : 2; }

constexpr uint64_t STAGE_ROWS = 65536;   // 256 MB fp32 staging chunk for host uploads
constexpr int GEMV_QCHUNK = 64;          // queries per gemv launch (partial-list scratch bound)

// Scratch buffers grow geometrically (and never below 64 KB): re-allocating device or pinned memory
// synchronises the device and costs up to tens of ms, which showed up as latency spikes in the
// interleaved upsert / search workload when a refresh batch was a few rows larger than any before.
template <typename T>
size_t grown(size_t have, size_t want) {
    size_t n = std::max(want, have * 2);
    const size_t floor_elems = (64 * 1024 + sizeof(T) - 1) / sizeof(T);
    return std::max(n, floor_elems);
}

template <typename T>
struct DevBuf {
    T *p = nullptr;
    size_t n = 0;
    cudaError_t ensure(size_t want) {
        if (want <= n) return cudaSuccess;
        want = grown<T>(n, want);
        if (p) cudaFree(p);
        p = nullptr;
        n = 0;
        cudaError_t e = cudaMalloc(&p, want * sizeof(T));
        if (e == cudaSuccess) n = want;
        return e;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        n = 0;
    }
};
template <typename T>
struct PinBuf {
    T *p = nullptr;
    size_t n = 0;
    cudaError_t ensure(size_t want) {
        if (want <= n) return cudaSuccess;
        want = grown<T>(n, want);
        if (p) cudaFreeHost(p);
        p = nullptr;
        n = 0;
        // mapped: kernels write results / read small query batches directly over PCIe (no memcpy calls)
        cudaError_t e = cudaHostAlloc(&p, want * sizeof(T), cudaHostAllocMapped | cudaHostAllocPortable);
        if (e == cudaSuccess) n = want;
        return e;
    }
    void release() {
        if (p) cudaFreeHost(p);
        p = nullptr;
        n = 0;
    }
};

// Layout of one rank's result block for (nq, k): ids | dist | counts | flags (16-byte padded).
struct SlotLayout {
    size_t dist_off = 0, counts_off = 0, flags_off = 0, bytes = 0;
};
SlotLayout slot_layout(int nq, int k) {
    SlotLayout L;
    L.dist_off = (size_t)nq * k * sizeof(orx_id);
    L.counts_off = L.dist_off + (size_t)nq * k * sizeof(double);
    L.flags_off = L.counts_off + (size_t)nq * sizeof(int);
    L.bytes = (L.flags_off + (size_t)nq * sizeof(int) + 15) & ~(size_t)15;
    return L;
}

}  // namespace

constexpr int XQ_MAX = 1024;                         // queries per exchange round (larger batches are chunked)
constexpr size_t XFLAG_STRIDE = 128;                 // one arrival word per 128 bytes

struct Exchange {   // peer-memory exchange state of one rank (orx_shard_*) or of one shard of a one-process group
    int world = 0, rank = 0;
    int n_targets = 0;                               // gather buffers my block is pushed into: every rank's, or the group root's
    size_t slot_bytes = 0;                           // capacity of one slot
    size_t set_bytes = 0;                            // world slots
    size_t flags_off = 0;                            // offset of the arrival words (2 sets x world x 128 B)
    char *base = nullptr;                            // my buffer
    std::vector<char *> peer_base;                   // every rank's buffer as mapped in this process
    void **d_peer_slot[2] = {nullptr, nullptr};      // device arrays [world]: MY slot inside peer g's set s
    uint32_t **d_peer_flag[2] = {nullptr, nullptr};  // device arrays [world]: MY arrival word on peer g, set s
    uint32_t seq = 0;
    bool connected = false;
};

struct SearchSlot {         // everything ONE search in flight owns
    DevBuf<float> q_dev, qhat;
    DevBuf<__nv_bfloat16> qhat16;
    DevBuf<int8_t> qhat8;               // fp32 tables: the 15-bit quantised queries of the 8-bit scan [nq, 2 * ORX_DIM]
    DevBuf<orx::QueryPrep> prep;
    DevBuf<uint64_t> partial;
    DevBuf<double> blk;                 // scratch result block (empty shard / error block of the row-sharded search)
    PinBuf<float> h_q;
    PinBuf<orx::QueryPrep> h_prep;
    PinBuf<orx_id> h_ids;
    PinBuf<double> h_dist;
    PinBuf<int> h_counts, h_flags, h_myflags, h_redo;
    PinBuf<uint32_t> h_done;            // [0] completion word the last CTA of a search writes (host polls it), [1] error word
    DevBuf<unsigned int> d_counters;    // [0] finalize CTAs, [1] merge CTAs of the search in flight (0 between searches)
    std::vector<cudaEvent_t> scan_ev;   // pairs bracketing each scan launch of the search
    size_t scan_ev_used = 0;
    orx::UmmaPlan *umma = nullptr;
    // single-query 8-bit scans (lap_search): they run on this slot's own stream, so that the other slot's search can
    // join a lap while it runs (internal.h LapState).  ev_entry: the index stream at submit; ev_ready: this slot's lap
    // state is set up (and its join attempt, if any, is over); ev_lap: after its lap; ev_done: after its finalize
    DevBuf<orx::LapState> lap;
    cudaStream_t lap_stream = nullptr;
    cudaEvent_t ev_entry = nullptr, ev_ready = nullptr, ev_lap = nullptr, ev_done = nullptr;
    // the search in flight in this slot (orx_search_submit ... orx_search_wait)
    struct Pending {
        bool active = false, complete = false, sharded = false, out_on_dev = false;
        bool settled = false;               // completed early by a write that had to wait for it; `settled_rc` is its verdict
        int settled_rc = ORX_OK;
        std::string settled_err;
        int nq = 0, k = 0, path = 1;
        orx_id *out_ids = nullptr;          // the caller's arrays
        double *out_dist = nullptr;
        int *out_counts = nullptr;
        orx::ResultOut out{};               // where the kernels write (prepare_results)
        const float *q_src = nullptr;
        bool lap = false;                   // ran on lap_stream (lap_search)
        SearchSlot *join_host = nullptr;    // the other slot, whose lap this search tries to join
        uint32_t lap_rows = 0;              // live rows its lap scans
        uint32_t token = 0, seq = 0, ticket = 0;
        SlotLayout L;
        std::chrono::steady_clock::time_point t_begin;
    } pend;
    void release() {
        q_dev.release(); qhat.release(); qhat16.release(); qhat8.release(); prep.release(); partial.release(); blk.release();
        h_q.release(); h_prep.release(); h_ids.release(); h_dist.release(); h_counts.release(); h_flags.release();
        h_myflags.release(); h_redo.release(); h_done.release(); d_counters.release();
        for (auto &e : scan_ev) cudaEventDestroy(e);
        scan_ev.clear();
        lap.release();
        for (cudaEvent_t *e : {&ev_entry, &ev_ready, &ev_lap, &ev_done}) {
            if (*e) cudaEventDestroy(*e);
            *e = nullptr;
        }
        if (lap_stream) cudaStreamDestroy(lap_stream);
        lap_stream = nullptr;
    }
};

struct orx_index {
    int device = 0;
    int dtype = ORX_DTYPE_F32;
    cudaStream_t stream = nullptr;
    uint64_t capacity = 0;
    uint64_t n_live = 0;
    uint64_t generation = 0;            // bumped whenever the id -> row map changes (orx_filter re-resolves then)
    std::atomic<uint64_t> mutations{0}; // bumped by EVERY successful write (upsert incl. in-place, delete, import): snapshots check it

    // the table (device)
    void *table = nullptr;
    float *scale = nullptr;
    double *n2 = nullptr;
    orx_id *row_ids = nullptr;
    // fp32 tables: the bf16 image of the rows ([capacity, ORX_DIM], RNE of every element) that the GEMV scans read from
    // image_min_rows live rows on -- half the bytes of the fp32 rows; finalize still rescores the fp32 rows.  Allocated
    // only for a capacity of image_min_rows rows or more (at create / growth, or by the first search that needs it),
    // and best effort: null when the device has no room (the scans then read the fp32 rows; bf16 tables never have one)
    __nv_bfloat16 *image = nullptr;
    // ... or, for a capacity of image8_min_rows rows or more, the 8-bit image instead (never both): a quarter of the
    // fp32 rows' bytes.  capped8 = live rows over R8_CAP, recounted by every write; more than IMAGE8_MAX_CAPPED of them
    // and the scans read the fp32 rows again
    orx::Image8 image8{nullptr, nullptr};
    uint64_t image_min_rows = orx::IMAGE_MIN_ROWS;    // ORX_OPT_IMAGE_MIN_ROWS
    uint64_t image8_min_rows = orx::IMAGE8_MIN_ROWS;  // ORX_OPT_IMAGE8_MIN_ROWS
    uint64_t image_failed_cap = 0;                    // capacity at which allocating the image failed (no retry until it changes)
    uint64_t capped8 = 0;
    DevBuf<uint32_t> d_capped8;
    PinBuf<uint32_t> h_capped8;

    // host mirror of the id column + id -> row map
    std::vector<orx_id> host_row_ids;
    IdMap map;

    // search scratch: TWO complete sets, so that one search can be launched while the previous one is still in flight
    // (orx_search_submit / orx_search_wait); `cur` = the set the search being submitted / completed works on
    SearchSlot slot[2];
    SearchSlot *cur = &slot[0];
    uint32_t tickets = 0;               // searches submitted so far; ticket t lives in slot[t & 1]
    uint32_t token = 0;                 // last completion token handed out (never 0)
    bool scan_timing = true;            // ORX_OPT_SCAN_TIMING
    struct Exchange *xchg = nullptr;     // peer-memory exchange of the row-sharded search (orx_shard_*)
    struct Group *group = nullptr;       // non-null: this handle is a multi-GPU group (orx_create_multi); shard fields unused
    // filtered search: eligibility bitmap (one bit per row) for the filtered scan
    DevBuf<uint32_t> allow_bits;
    DevBuf<float> scale_masked;          // the per-row scale with the filter folded in (filtered tcgen05 scan)
    PinBuf<uint32_t> h_allow_bits;
    // exhaustive fallback scratch
    DevBuf<uint32_t> fb_list, fb_count;
    DevBuf<double> fb_dist;
    // maximal-marginal-relevance scratch (orx_search_mmr*)
    DevBuf<float> mmr_rows;              // [queries of a chunk, fetch_k, ORX_DIM] candidate matrix the kernel reads
    DevBuf<float> mmr_stage;             // multi-GPU: this shard's candidates, gathered before the copy to the root
    DevBuf<uint32_t> mmr_idx;
    DevBuf<double> mmr_dist;
    DevBuf<int> mmr_cnt, mmr_sel;
    // upsert / delete scratch
    DevBuf<float> stage;
    DevBuf<uint32_t> d_src_idx, d_dst_row;
    DevBuf<orx_id> d_ids;
    DevBuf<int> d_flag;
    PinBuf<uint32_t> h_u32a, h_u32b;
    PinBuf<int> h_flag;

    mutable std::mutex mu;
    orx_stats stats{};
    uint64_t shared_rows = 0;           // orx_shared_rows
};

struct FilterOnDevice {          // a resolved predicate: the eligible rows, as a sorted list and (when large) a bitmap
    uint32_t m;
    const uint32_t *list;        // [m] device
    const uint32_t *count;       // device word holding m
    const uint32_t *bits;        // [(n_live+31)/32] device, or null: rescore the list, no scan
};

struct orx_filter {     // a reusable resolved predicate (orx_filter_create / orx_search_with_filter)
    orx_index *ix = nullptr;
    int device = 0;
    std::vector<orx_id> ids;              // the id set as given
    DevBuf<uint32_t> d_list, d_count, d_bits;
    FilterOnDevice dev{};                 // the eligible live rows at `generation`, in d_list / d_count / d_bits
    uint64_t generation = 0;
    bool resolved = false;
};

#define ORX_GROUP_TYPES
#include "group.inl"
#undef ORX_GROUP_TYPES

namespace {

struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev) {
        cudaGetDevice(&prev);
        if (prev != dev) cudaSetDevice(dev);
    }
    ~DeviceGuard() {
        int cur = -1;
        cudaGetDevice(&cur);
        if (prev >= 0 && cur != prev) cudaSetDevice(prev);
    }
};

// the image a capacity gets: 2 the 8-bit one (from image8_min_rows rows), 1 the bf16 one (from image_min_rows rows), 0
// none (bf16 tables, small capacities: small tables pay no memory for it)
int image_kind_for(const orx_index *ix, uint64_t cap) {
    if (ix->dtype != ORX_DTYPE_F32) return 0;
    return cap >= ix->image8_min_rows ? 2 : cap >= ix->image_min_rows ? 1 : 0;
}
int image_kind(const orx_index *ix) { return ix->image8.rows ? 2 : ix->image ? 1 : 0; }

struct ImageAlloc {
    __nv_bfloat16 *bf16 = nullptr;
    orx::Image8 i8{nullptr, nullptr};
    bool ok() const { return bf16 || i8.rows; }
    void release() {
        if (bf16) cudaFree(bf16);
        if (i8.rows) cudaFree(i8.rows);
        if (i8.scale8) cudaFree(i8.scale8);
        *this = ImageAlloc{};
    }
};
// an image of `kind` with room for `cap` rows; best effort: none when the device has no room
ImageAlloc alloc_image(orx_index *ix, uint64_t cap, int kind) {
    ImageAlloc a;
    if (kind == 0) return a;
    cudaError_t e = kind == 1 ? cudaMalloc(&a.bf16, cap * ORX_DIM * sizeof(__nv_bfloat16))
                              : cudaMalloc(&a.i8.rows, cap * ORX_DIM * sizeof(int8_t));
    if (e == cudaSuccess && kind == 2) e = cudaMalloc(&a.i8.scale8, cap * sizeof(float));
    if (e != cudaSuccess) {
        cudaGetLastError();
        a.release();
        ix->image_failed_cap = cap;
    }
    return a;
}
void free_image(orx_index *ix) {
    ImageAlloc{ix->image, ix->image8}.release();
    ix->image = nullptr;
    ix->image8 = orx::Image8{nullptr, nullptr};
}
// build image a of the first n rows from a table's fp32 rows (and their n2 / scale)
void build_image(const ImageAlloc &a, const void *table, const double *n2, const float *scale, uint64_t n,
                 cudaStream_t st) {
    if (a.bf16) orx::launch_image_rows(static_cast<const float *>(table), n, a.bf16, st);
    else orx::launch_image8_rows(static_cast<const float *>(table), n2, scale, n, a.i8, st);
}
// the 8-bit image's over-cap count of rows [0, n) into h_capped8, stream-ordered (read it after the next sync)
cudaError_t launch_recount8(orx_index *ix, uint64_t n) {
    cudaError_t e = ix->d_capped8.ensure(1);
    if (e == cudaSuccess) e = ix->h_capped8.ensure(1);
    if (e != cudaSuccess) return e;
    orx::launch_count_capped8(ix->scale, ix->image8.scale8, n, ix->d_capped8.p, ix->stream);
    ix->stats.kernel_launches += 1;
    return cudaMemcpyAsync(ix->h_capped8.p, ix->d_capped8.p, sizeof(uint32_t), cudaMemcpyDeviceToHost, ix->stream);
}

// rows a GEMV launch of m queries reads: 4 the 8-bit image (one query or a bitmap scan, k <= IMAGE8_MAX_K, few rows
// over R8_CAP), 3 the bf16 image, 1 the table's own rows (also below image_min_rows live rows)
int gemv_source(const orx_index *ix, int m, int k, bool filtered) {
    if (ix->n_live < ix->image_min_rows) return 1;
    if (ix->image) return 3;
    if (ix->image8.rows && (filtered || m == 1) && k <= orx::IMAGE8_MAX_K && ix->capped8 <= orx::IMAGE8_MAX_CAPPED)
        return 4;
    return 1;
}

// an fp32 table that has reached image_min_rows live rows (or whose options were changed) without the image its capacity
// gets: allocate that one and build it from the live rows, once per capacity (an image of the other kind is dropped
// first).  Best effort: without it the scans read the fp32 rows.  force_kind: the diagnostic hooks, which want an image
// whatever the thresholds (and keep one of either kind).
void ensure_image(orx_index *ix, int force_kind = 0) {
    if (ix->dtype != ORX_DTYPE_F32 || ix->n_live == 0) return;
    if (!force_kind && ix->n_live < ix->image_min_rows) return;
    const int kind = force_kind ? force_kind : ix->capacity >= ix->image8_min_rows ? 2 : 1;
    if (image_kind(ix) == kind || (force_kind && image_kind(ix)) || ix->image_failed_cap == ix->capacity) return;
    free_image(ix);
    ImageAlloc a = alloc_image(ix, ix->capacity, kind);
    if (!a.ok()) return;
    build_image(a, ix->table, ix->n2, ix->scale, ix->n_live, ix->stream);
    ix->stats.kernel_launches += 1;
    ix->image = a.bf16;
    ix->image8 = a.i8;
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess && kind == 2) e = launch_recount8(ix, ix->n_live);
    if (e == cudaSuccess && kind == 2) e = cudaStreamSynchronize(ix->stream);
    if (e != cudaSuccess) {                       // stay without an image
        cudaGetLastError();
        cudaStreamSynchronize(ix->stream);
        free_image(ix);
        ix->image_failed_cap = ix->capacity;
        return;
    }
    if (kind == 2) ix->capped8 = *ix->h_capped8.p;  // stream order: every later scan sees the built rows
}

int alloc_table(orx_index *ix, uint64_t cap) {
    CK(cudaMalloc(&ix->table, cap * ORX_DIM * elem_size(ix->dtype)));
    CK(cudaMalloc(&ix->scale, cap * sizeof(float)));
    CK(cudaMalloc(&ix->n2, cap * sizeof(double)));
    CK(cudaMalloc(&ix->row_ids, cap * sizeof(orx_id)));
    const ImageAlloc a = alloc_image(ix, cap, image_kind_for(ix, cap));   // after the table: never takes the table's room
    ix->image = a.bf16;
    ix->image8 = a.i8;
    ix->capacity = cap;
    return ORX_OK;
}

int grow_table(orx_index *ix, uint64_t need) {
    if (need <= ix->capacity) return ORX_OK;
    if (need >= 0xFFFFFFFFull) return fail(ORX_ERR_CAPACITY, "table limited to 2^32-2 rows per GPU");
    uint64_t cap = std::max<uint64_t>(need, ix->capacity + ix->capacity / 2 + 1024);
    cap = std::min<uint64_t>(cap, 0xFFFFFFFEull);
    void *t = nullptr;
    float *s = nullptr;
    double *n = nullptr;
    orx_id *r = nullptr;
    const size_t rb = ORX_DIM * elem_size(ix->dtype);
    cudaError_t e = cudaSuccess;
    for (int attempt = 0; attempt < 2; ++attempt) {
        e = cudaMalloc(&t, cap * rb);
        if (e == cudaSuccess) e = cudaMalloc(&s, cap * sizeof(float));
        if (e == cudaSuccess) e = cudaMalloc(&n, cap * sizeof(double));
        if (e == cudaSuccess) e = cudaMalloc(&r, cap * sizeof(orx_id));
        if (e == cudaSuccess) break;
        cudaGetLastError();
        if (t) cudaFree(t);
        if (s) cudaFree(s);
        if (n) cudaFree(n);
        if (r) cudaFree(r);
        t = nullptr, s = nullptr, n = nullptr, r = nullptr;
        if (!image_kind(ix)) break;
        free_image(ix);                     // the image is best effort: it gives its room to the table's growth
    }
    if (e != cudaSuccess)
        return fail(ORX_ERR_CAPACITY, "cannot grow table to %llu rows: %s", (unsigned long long)cap,
                    cudaGetErrorString(e));
    const int kind_was = image_kind(ix);
    int kind = image_kind_for(ix, cap);
    if (kind == 0) kind = kind_was;         // an image that exists is carried over whatever the thresholds
    ImageAlloc im = alloc_image(ix, cap, kind);
    e = cudaMemcpyAsync(t, ix->table, ix->n_live * rb, cudaMemcpyDeviceToDevice, ix->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(s, ix->scale, ix->n_live * sizeof(float), cudaMemcpyDeviceToDevice, ix->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(n, ix->n2, ix->n_live * sizeof(double), cudaMemcpyDeviceToDevice, ix->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(r, ix->row_ids, ix->n_live * sizeof(orx_id), cudaMemcpyDeviceToDevice, ix->stream);
    if (e == cudaSuccess && im.ok()) {
        if (kind == kind_was && im.bf16)
            e = cudaMemcpyAsync(im.bf16, ix->image, ix->n_live * ORX_DIM * sizeof(__nv_bfloat16), cudaMemcpyDeviceToDevice,
                                ix->stream);
        else if (kind == kind_was) {
            e = cudaMemcpyAsync(im.i8.rows, ix->image8.rows, ix->n_live * ORX_DIM, cudaMemcpyDeviceToDevice, ix->stream);
            if (e == cudaSuccess)
                e = cudaMemcpyAsync(im.i8.scale8, ix->image8.scale8, ix->n_live * sizeof(float), cudaMemcpyDeviceToDevice,
                                    ix->stream);
        } else {                            // none yet, or bf16 -> 8-bit at image8_min_rows
            build_image(im, ix->table, ix->n2, ix->scale, ix->n_live, ix->stream);
            ix->stats.kernel_launches += 1;
        }
        if (e == cudaSuccess) e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(ix->stream);
    if (e != cudaSuccess) {                 // the old table stays in place and valid
        cudaGetLastError();
        cudaFree(t);
        cudaFree(s);
        cudaFree(n);
        cudaFree(r);
        im.release();
        return fail(ORX_ERR_CUDA, "copying the table to its grown allocation failed: %s", cudaGetErrorString(e));
    }
    cudaFree(ix->table);
    cudaFree(ix->scale);
    cudaFree(ix->n2);
    cudaFree(ix->row_ids);
    free_image(ix);
    ix->table = t;
    ix->scale = s;
    ix->n2 = n;
    ix->row_ids = r;
    ix->image = im.bf16;
    ix->image8 = im.i8;
    ix->capacity = cap;
    if (kind == 2 && kind_was != 2) {       // a rebuilt 8-bit image: count its rows over R8_CAP
        CK(launch_recount8(ix, ix->n_live));
        CK(cudaStreamSynchronize(ix->stream));
        ix->capped8 = *ix->h_capped8.p;
    }
    return ORX_OK;
}

int group_upsert(Group *g, const orx_id *ids, const float *vecs, uint64_t n);

// ---------------------------------------------------------------- upsert
int validate_locked(orx_index *ix, const float *vecs, uint64_t n) {      // pgvector's element check, whole batch
    cudaStream_t st = ix->stream;
    const bool on_dev = is_device_ptr(vecs);
    const uint64_t chunk = std::min<uint64_t>(n, STAGE_ROWS);
    CK(ix->d_flag.ensure(1));
    CK(ix->h_flag.ensure(1));
    if (!on_dev) CK(ix->stage.ensure(chunk * ORX_DIM));
    CK(cudaMemsetAsync(ix->d_flag.p, 0, sizeof(int), st));
    for (uint64_t s = 0; s < n; s += chunk) {
        const uint64_t m = std::min(chunk, n - s);
        const float *src = vecs + s * ORX_DIM;
        if (!on_dev) {
            CK(cudaMemcpyAsync(ix->stage.p, src, m * ORX_DIM * sizeof(float), cudaMemcpyHostToDevice, st));
            src = ix->stage.p;
        }
        orx::launch_validate_rows(src, m, ix->d_flag.p, st);
        ix->stats.kernel_launches += 1;
    }
    CK(cudaMemcpyAsync(ix->h_flag.p, ix->d_flag.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    CK(cudaGetLastError());
    if (*ix->h_flag.p) return fail(ORX_ERR_NONFINITE, "NaN or infinite value not allowed in vector");
    return ORX_OK;
}

// validate (pgvector's element check over the WHOLE batch) -> commit, stream-ordered: the commit kernels read the
// validation flag on the device and write nothing when it is set, so a batch of up to STAGE_ROWS rows needs ONE host
// synchronisation.  Host state (id -> row map, live row count) is published only after the device work of a chunk
// has succeeded: an error in between leaves ids mapped to nothing new and the live rows untouched.
int upsert_locked(orx_index *ix, const orx_id *ids, const float *vecs, uint64_t n, bool validate) {
    cudaStream_t st = ix->stream;
    const bool on_dev = is_device_ptr(vecs);
    const uint64_t chunk = std::min<uint64_t>(n, STAGE_ROWS);
    const bool single = n <= chunk;           // one chunk: staged once, validated and committed back to back
    if (validate && !single) {
        // several chunks: the whole batch is checked before anything is written
        int rc = validate_locked(ix, vecs, n);
        if (rc != ORX_OK) return rc;
    }
    CK(ix->d_flag.ensure(1));
    CK(ix->h_flag.ensure(1));
    if (!on_dev) CK(ix->stage.ensure(chunk * ORX_DIM));
    CK(cudaMemsetAsync(ix->d_flag.p, 0, sizeof(int), st));

    CK(ix->d_src_idx.ensure(chunk));
    CK(ix->d_dst_row.ensure(chunk));
    CK(ix->d_ids.ensure(chunk));
    CK(ix->h_u32a.ensure(chunk));
    CK(ix->h_u32b.ensure(chunk));
    IdMap pending;                                                   // ids new in this chunk -> row (published after the sync)
    std::vector<std::pair<orx_id, uint32_t>> pending_list;
    std::unordered_map<uint32_t, uint32_t> slot_of_row;              // dst row -> plan slot
    for (uint64_t s = 0; s < n; s += chunk) {
        const uint64_t m = std::min(chunk, n - s);
        // plan: existing id -> its row, new id -> append; an id repeated inside the chunk keeps the later source row
        pending.clear();
        pending.reserve(m);
        pending_list.clear();
        slot_of_row.clear();
        uint32_t np = 0;
        uint64_t next_row = ix->n_live;
        bool repeats = false;
        for (uint64_t i = 0; i < m; ++i) {
            const orx_id id = ids[s + i];
            uint32_t row;
            bool fresh = false;
            if (const uint32_t *r = ix->map.find(id)) row = *r;
            else if (const uint32_t *r2 = pending.find(id)) row = *r2;
            else {
                row = (uint32_t)next_row++;
                pending.set(id, row);
                pending_list.emplace_back(id, row);
                fresh = true;
            }
            if (!fresh) {
                // a row written before: by an earlier element of this chunk (the later source row wins) or not at all yet
                if (!repeats) {                                       // build the row -> slot index lazily: rare path
                    for (uint32_t p = 0; p < np; ++p) slot_of_row.emplace(ix->h_u32b.p[p], p);
                    repeats = true;
                }
                auto ps = slot_of_row.find(row);
                if (ps != slot_of_row.end()) {
                    ix->h_u32a.p[ps->second] = (uint32_t)i;
                    continue;
                }
            }
            if (repeats) slot_of_row.emplace(row, np);
            ix->h_u32a.p[np] = (uint32_t)i;
            ix->h_u32b.p[np] = row;
            ++np;
        }
        int rc = grow_table(ix, next_row);                            // room for the ids that are new
        if (rc != ORX_OK) return rc;
        const float *src = vecs + s * ORX_DIM;
        if (!on_dev) {
            CK(cudaMemcpyAsync(ix->stage.p, src, m * ORX_DIM * sizeof(float), cudaMemcpyHostToDevice, st));
            src = ix->stage.p;
        }
        if (validate && single) {
            orx::launch_validate_rows(src, m, ix->d_flag.p, st);
            ix->stats.kernel_launches += 1;
        }
        CK(cudaMemcpyAsync(ix->d_src_idx.p, ix->h_u32a.p, np * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(ix->d_dst_row.p, ix->h_u32b.p, np * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(ix->d_ids.p, ids + s, m * sizeof(orx_id), cudaMemcpyHostToDevice, st));
        orx::launch_commit_rows(ix->dtype, src, ix->d_src_idx.p, ix->d_dst_row.p, ix->d_ids.p, np, ix->table,
                                ix->scale, ix->n2, ix->row_ids, ix->d_flag.p, ix->image, ix->image8, st);
        ix->stats.kernel_launches += 1;
        if (ix->image8.rows) CK(launch_recount8(ix, next_row));
        CK(cudaMemcpyAsync(ix->h_flag.p, ix->d_flag.p, sizeof(int), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));     // the ONE sync of a chunk: scratch + the caller's buffers are reusable after it
        CK(cudaGetLastError());
        if (*ix->h_flag.p) return fail(ORX_ERR_NONFINITE, "NaN or infinite value not allowed in vector");
        if (ix->image8.rows) ix->capped8 = *ix->h_capped8.p;
        // ---- the device holds the rows: publish them
        if (!pending_list.empty()) {
            if (ix->host_row_ids.size() < next_row) ix->host_row_ids.resize(next_row);
            for (const auto &kv : pending_list) {
                ix->map.set(kv.first, kv.second);
                ix->host_row_ids[kv.second] = kv.first;
            }
            ix->n_live = next_row;
            ix->generation += 1;
        }
        ix->mutations.fetch_add(1);
    }
    return ORX_OK;
}

// ---------------------------------------------------------------- search core
// a fresh event from the per-search pool (pairs: before / after one scan launch)
cudaEvent_t scan_event(orx_index *ix) {
    if (!ix->scan_timing) return nullptr;
    if (ix->cur->scan_ev_used == ix->cur->scan_ev.size()) {
        cudaEvent_t e = nullptr;
        if (cudaEventCreate(&e) != cudaSuccess) return nullptr;
        ix->cur->scan_ev.push_back(e);
    }
    return ix->cur->scan_ev[ix->cur->scan_ev_used++];
}
void harvest_scan_events(orx_index *ix) {       // stream is synchronised
    float last = 0.f;
    for (size_t i = 0; i + 1 < ix->cur->scan_ev_used; i += 2) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, ix->cur->scan_ev[i], ix->cur->scan_ev[i + 1]) == cudaSuccess) {
            ix->stats.scan_ms_total += ms;
            ix->stats.scan_launches += 1;
            last += ms;
        }
    }
    if (ix->cur->scan_ev_used) ix->stats.last_scan_ms = last;
    ix->cur->scan_ev_used = 0;
    cudaGetLastError();
}

struct SearchCtx {          // where a search's results go and how its completion is signalled (internal.h)
    orx::ResultOut out;
    orx::PublishArgs pub;
    orx::DoneArgs done;
    bool lap = false;                   // a single-query 8-bit scan runs as a lap (lap_search)
    SearchSlot *join_host = nullptr;    // ... that joins this slot's lap
};
SearchCtx plain_ctx(const orx::ResultOut &out) {      // no publish, no completion word
    SearchCtx c{};
    c.out = out;
    return c;
}

int exhaustive_query(orx_index *ix, const float *q_src, int qi, int k, double dk, bool force_all,
                     const orx::ResultOut &out) {
    // Collect every row that could sort at or before the current k-th candidate, rescore all of
    // them canonically, select the k best.  Always exact; cost grows with the number of near-ties.
    const uint32_t n_rows = (uint32_t)ix->n_live;
    CK(ix->fb_list.ensure(ix->capacity));
    CK(ix->fb_dist.ensure(ix->capacity));
    CK(ix->fb_count.ensure(1));
    const double eps = ix->dtype == ORX_DTYPE_F32 ? orx::EPS_GEMV_F32 : orx::EPS_GEMV_BF16;
    bool all = force_all || !(dk == dk) || dk >= 2.0;
    float floor_f = 0.f;
    if (!all) {
        floor_f = (float)((1.0 - dk) - eps);
        floor_f = nextafterf(floor_f, -INFINITY);     // conversion may have rounded up
    }
    CK(cudaMemsetAsync(ix->fb_count.p, 0, sizeof(uint32_t), ix->stream));
    orx::launch_collect(ix->dtype, ix->table, ix->scale, n_rows, ix->cur->qhat.p + (size_t)qi * ORX_DIM, floor_f,
                        all ? 1 : 0, ix->fb_list.p, ix->fb_count.p, ix->stream);
    orx::launch_rescore_list(ix->dtype, ix->table, ix->n2, ix->row_ids, q_src + (size_t)qi * ORX_DIM,
                             ix->cur->prep.p + qi, ix->fb_list.p, ix->fb_count.p, ix->fb_dist.p, ix->stream);
    orx::launch_select_list(ix->row_ids, ix->fb_list.p, ix->fb_count.p, ix->fb_dist.p, k,
                            out.ids + (size_t)qi * k, out.dist + (size_t)qi * k, out.counts + qi, ix->stream);
    ix->stats.kernel_launches += 3;
    ix->stats.fallback_exhaustive += 1;
    CK(cudaGetLastError());
    return ORX_OK;
}

// ---- the lap of a single-query 8-bit scan on ix->stream (internal.h LapState): set up the slot's lap state, and for a
//      search that joins the other slot's lap (host) run the join, then wait for that lap before the catch-up
int ensure_lap(SearchSlot *sl) {
    CK(sl->lap.ensure(1));
    if (!sl->lap_stream) CK(cudaStreamCreateWithFlags(&sl->lap_stream, cudaStreamNonBlocking));
    for (cudaEvent_t *e : {&sl->ev_entry, &sl->ev_ready, &sl->ev_lap, &sl->ev_done})
        if (!*e) CK(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
    return ORX_OK;
}
int lap_setup(orx_index *ix, int qa, uint32_t n_rows, int grid, SearchSlot *host) {
    SearchSlot *sl = ix->cur;
    SearchSlot *other = &ix->slot[sl == &ix->slot[0] ? 1 : 0];
    cudaStream_t st = ix->stream;
    const int rc = ensure_lap(sl);
    if (rc != ORX_OK) return rc;
    // the other slot's join kernel may have worked on this slot's state (it joined this slot's previous lap)
    if (other->ev_ready) CK(cudaStreamWaitEvent(st, other->ev_ready, 0));
    if (!host) {
        CK(cudaMemsetAsync(sl->lap.p, 0, offsetof(orx::LapState, list), st));
        CK(cudaEventRecord(sl->ev_ready, st));
        return ORX_OK;
    }
    // the joined lap writes this query's lists of its grid (same rows, same grid) only in the CTAs that met the join
    CK(cudaMemsetAsync(sl->partial.p, 0, (size_t)grid * 32 * orx::IMAGE8_SLOTS * sizeof(uint64_t), st));
    CK(cudaMemsetAsync(sl->lap.p, 0, 2 * sizeof(uint32_t), st));             // next, covered
    const orx::LapJoiner me{sl->qhat8.p + (size_t)qa * 2 * ORX_DIM, sl->prep.p + qa, sl->partial.p, &sl->lap.p->covered};
    orx::launch_join_lap8(host->lap.p, sl->lap.p, me, n_rows, sl->h_done.p + 2, st);
    CK(cudaEventRecord(sl->ev_ready, st));
    CK(cudaStreamWaitEvent(st, host->ev_lap, 0));                           // the catch-up merges into its lists
    ix->stats.kernel_launches += 1;
    return ORX_OK;
}
// a submitted search whose scan is a lap: one query over the 8-bit image
bool lap_search(orx_index *ix, int nq, int k) {
    if (nq != 1 || ix->n_live == 0) return false;
    ensure_image(ix);
    return gemv_source(ix, 1, k, false) == 4;
}

// f: a filter with a bitmap -- the sequential scan skips the rows whose bit is clear (HBM traffic = eligible rows only).
// allow_image: a large fp32 table with an image is scanned over the image (the bf16 instantiation of the same kernels,
// the fp32 row's 1/|x|, EPS_GEMV_IMAGE; or the 8-bit scan, EPS_GEMV_IMAGE8, see gemv_source); finalize rescores the fp32
// rows either way, so the answer is the same.  The
// re-scan of queries the tcgen05 pass could not prove passes false: it reads the fp32 rows with EPS_GEMV_F32, whose
// bound is ~800x tighter than the tensor pass's, and so settles them; the image's bound would be looser than it.
int gemv_pass(orx_index *ix, const float *q_src, int q0, int nq, int k, const SearchCtx &ctx,
              const FilterOnDevice *f = nullptr, bool allow_image = true) {
    const uint32_t n_rows = (uint32_t)ix->n_live;
    const int grid = orx::scan_gemv_grid(ix->device, n_rows);
    for (int s = 0; s < nq; s += GEMV_QCHUNK) {
        const int m = std::min(GEMV_QCHUNK, nq - s);
        const int qa = q0 + s;
        const int src = allow_image ? gemv_source(ix, m, k, f != nullptr) : 1;
        const bool img = src == 3;
        const int scan_dtype = img ? ORX_DTYPE_BF16 : ix->dtype;      // the element type the scan reads
        const void *scan_rows = img ? static_cast<const void *>(ix->image) : ix->table;
        const double eps = src == 4 ? orx::EPS_GEMV_IMAGE8 : img ? orx::EPS_GEMV_IMAGE
                           : ix->dtype == ORX_DTYPE_F32 ? orx::EPS_GEMV_F32 : orx::EPS_GEMV_BF16;
        const int slots = src == 4 ? orx::IMAGE8_SLOTS : img ? orx::image_slots_for_k(k) : orx::slots_for_k(k);
        const bool lap = src == 4 && !f && ctx.lap;                     // (m == 1: gemv_source)
        // several queries: the batched kernel (8 queries share every row through shared memory); one: the streaming
        // kernel.  A lap leaves two CTA slots of the GPU free (2 CTAs of it fill an SM's registers), so that the other
        // slot's prep, memsets and join kernel -- and the tail of its catch-up or finalize -- find room while it runs; with
        // every slot taken, none of 20 pairs submitted back to back joined.  Its work queue gives the two half-used SMs
        // their share of the rows
        const int parts = lap ? std::max(1, std::min(grid, 2 * orx::device_sms() - 2))
                          : !f && m >= 2 ? orx::scan_gemv_batch_parts(ix->device, n_rows, m) : grid;
        CK(ix->cur->partial.ensure((size_t)m * parts * 32 * slots));
        if (lap) {
            const int rc = lap_setup(ix, qa, n_rows, parts, ctx.join_host);
            if (rc != ORX_OK) return rc;
        }
        cudaEvent_t e0 = scan_event(ix), e1 = scan_event(ix);
        if (e0 && e1) CK(cudaEventRecord(e0, ix->stream));
        if (lap)
            orx::launch_scan_lap8(ix->image8.rows, ix->image8.scale8, n_rows, ix->cur->qhat8.p + (size_t)qa * 2 * ORX_DIM,
                                  ix->cur->prep.p + qa, ix->cur->partial.p, ix->cur->lap.p, ctx.join_host != nullptr,
                                  parts, ix->stream);
        else if (src == 4)
            orx::launch_scan_gemv8(ix->image8.rows, ix->image8.scale8, n_rows, f ? f->bits : nullptr,
                                   ix->cur->qhat8.p + (size_t)qa * 2 * ORX_DIM, ix->cur->prep.p + qa, m,
                                   ix->cur->partial.p, grid, ix->stream);
        else if (f)
            orx::launch_scan_gemv_filtered(scan_dtype, scan_rows, ix->scale, n_rows, f->bits,
                                           ix->cur->qhat.p + (size_t)qa * ORX_DIM, m, slots, ix->cur->partial.p, grid,
                                           ix->stream);
        else if (m >= 2)
            orx::launch_scan_gemv_batch(scan_dtype, scan_rows, ix->scale, n_rows, ix->cur->qhat.p + (size_t)qa * ORX_DIM, m,
                                        slots, ix->cur->partial.p, parts, ix->stream);
        else
            orx::launch_scan_gemv(scan_dtype, scan_rows, ix->scale, n_rows, ix->cur->qhat.p + (size_t)qa * ORX_DIM, m,
                                  slots, ix->cur->partial.p, grid, ix->stream);
        if (e0 && e1) CK(cudaEventRecord(e1, ix->stream));
        if (lap) CK(cudaEventRecord(ix->cur->ev_lap, ix->stream));
        // a filter's row bound is the eligible count: "every eligible row is a candidate" when it fits the list
        orx::launch_finalize(ix->dtype, ix->table, ix->n2, ix->row_ids, q_src + (size_t)qa * ORX_DIM,
                             ix->cur->prep.p + qa, ix->cur->partial.p, parts, slots, m, k, f ? f->m : n_rows, eps, ctx.out,
                             qa, ctx.pub, ctx.done, ix->stream, nullptr, lap ? &ix->cur->lap.p->covered : nullptr);
        ix->stats.kernel_launches += 2;
    }
    CK(cudaGetLastError());
    return ORX_OK;
}

constexpr uint32_t FILTER_SCAN_MIN_ROWS = 4096;   // eligible rows from which the bitmap scan replaces rescoring them all
constexpr int ZERO_COPY_MAX_Q = 16;     // query batches up to this size are read by the prep kernel over PCIe

// ---- query staging: *q_src is what the rescoring kernels read (device memory); launches prep
//      src_pinned: `queries` is mapped pinned host memory every device can read (a group stages the batch once)
int stage_queries(orx_index *ix, const float *queries, int nq, const float **q_src, bool src_pinned = false) {
    cudaStream_t st = ix->stream;
    // the tcgen05 scan reads query tiles of 128 rows (256 per CTA pair): keep the buffers padded (and the pad zeroed) so
    // its TMA never touches an out-of-range row (measured: mostly-out-of-range query boxes cost ~40 %)
    const size_t nq_pad = ((size_t)nq + 255) / 256 * 256;
    CK(ix->cur->qhat.ensure(nq_pad * ORX_DIM));
    CK(ix->cur->qhat16.ensure(nq_pad * ORX_DIM));
    CK(ix->cur->prep.ensure(nq));
    int8_t *q8 = nullptr;                 // quantised for the 8-bit scan (fp32 tables: a search may build the image)
    if (ix->dtype == ORX_DTYPE_F32) {
        CK(ix->cur->qhat8.ensure((size_t)nq * 2 * ORX_DIM));
        q8 = ix->cur->qhat8.p;
    }
    if (nq_pad != (size_t)nq && nq > 1) {
        CK(cudaMemsetAsync(ix->cur->qhat.p + (size_t)nq * ORX_DIM, 0, (nq_pad - nq) * ORX_DIM * sizeof(float), st));
        CK(cudaMemsetAsync(ix->cur->qhat16.p + (size_t)nq * ORX_DIM, 0, (nq_pad - nq) * ORX_DIM * sizeof(__nv_bfloat16), st));
    }
    const int qdev = ptr_device(queries);
    if (qdev == ix->device) {
        *q_src = queries;
        orx::launch_prep_queries(queries, nq, nullptr, ix->cur->qhat.p, ix->cur->qhat16.p, q8, ix->cur->prep.p, st);
    } else if (qdev >= 0) {
        // the batch lives on ANOTHER GPU (a group's shards all receive the root's pointer): the prep kernel reads it
        // over NVLink once and leaves a local copy for the rescoring kernels
        CK(ix->cur->q_dev.ensure((size_t)nq * ORX_DIM));
        *q_src = ix->cur->q_dev.p;
        orx::launch_prep_queries(queries, nq, ix->cur->q_dev.p, ix->cur->qhat.p, ix->cur->qhat16.p, q8, ix->cur->prep.p, st);
    } else {
        CK(ix->cur->q_dev.ensure((size_t)nq * ORX_DIM));
        const float *pinned = queries;
        if (!src_pinned) {
            CK(ix->cur->h_q.ensure((size_t)nq * ORX_DIM));
            memcpy(ix->cur->h_q.p, queries, (size_t)nq * ORX_DIM * sizeof(float));
            pinned = ix->cur->h_q.p;
        }
        *q_src = ix->cur->q_dev.p;
        if (nq <= ZERO_COPY_MAX_Q) {
            orx::launch_prep_queries(pinned, nq, ix->cur->q_dev.p, ix->cur->qhat.p, ix->cur->qhat16.p, q8, ix->cur->prep.p, st);
        } else {
            CK(cudaMemcpyAsync(ix->cur->q_dev.p, pinned, (size_t)nq * ORX_DIM * sizeof(float), cudaMemcpyHostToDevice, st));
            orx::launch_prep_queries(ix->cur->q_dev.p, nq, nullptr, ix->cur->qhat.p, ix->cur->qhat16.p, q8, ix->cur->prep.p, st);
        }
    }
    ix->stats.kernel_launches += 1;
    return ORX_OK;
}

// ---- the scan + finalize of all nq queries (tcgen05 for batches, GEMV otherwise); *path = 1 / 2 / 3 (GEMV over the bf16
//      image) / 4 (GEMV over the 8-bit image)
//      f: a filter with a bitmap.  A BATCH of filtered queries whose bitmap scans together would read more than the
//      whole table takes ONE tcgen05 pass over all rows instead: the predicate enters through the per-row scale (a
//      cleared bit -> the "never a candidate" marker), so the kernel and its candidate proof are those of orx_search.
int scan_pass(orx_index *ix, const float *q_src, int nq, int k, const SearchCtx &ctx, int *path,
              const FilterOnDevice *f = nullptr) {
    const uint32_t n_rows = (uint32_t)ix->n_live;
    if (ix->cur->umma && orx::umma_should_use(ix->cur->umma, nq, k, n_rows) && (!f || (uint64_t)nq * f->m >= n_rows)) {
        const float *scale = ix->scale;
        if (f) {
            CK(ix->scale_masked.ensure(n_rows));
            orx::launch_mask_scale(ix->scale, f->bits, n_rows, ix->scale_masked.p, ix->stream);
            ix->stats.kernel_launches += 1;
            scale = ix->scale_masked.p;
        }
        *path = 2;
        cudaEvent_t e0 = scan_event(ix), e1 = scan_event(ix);
        int rc = orx::umma_search(ix->cur->umma, ix->dtype, ix->table, scale, ix->n2, ix->row_ids, n_rows,
                                  q_src, ix->cur->qhat.p, ix->cur->qhat16.p, ix->cur->prep.p, nq, k, ctx.out, ctx.pub, ctx.done,
                                  ix->stream, &ix->stats.kernel_launches, e0, e1);
        if (rc != ORX_OK) return fail(rc, "tcgen05 scan failed: %s", orx::umma_last_error());
        return ORX_OK;
    }
    ensure_image(ix);
    *path = gemv_source(ix, f ? 1 : std::min(nq, GEMV_QCHUNK), k, f != nullptr);
    return gemv_pass(ix, q_src, 0, nq, k, ctx, f);
}

// ---- completion of the search whose last kernel writes `token` into the mapped completion word: the host polls the
//      word (a few ns per poll, visible ~1 us after the store) instead of cudaStreamSynchronize; the stream is queried
//      now and then so that a failed launch or a dead kernel surfaces as an error instead of an endless spin.
uint32_t next_token(orx_index *ix) {
    if (++ix->token == 0) ++ix->token;
    return ix->token;
}
int wait_done(orx_index *ix, uint32_t token) {
    volatile uint32_t *w = ix->cur->h_done.p;
    cudaStream_t st = ix->cur->pend.lap ? ix->cur->lap_stream : ix->stream;
    for (uint64_t it = 0;; ++it) {
        if (*w == token) return ORX_OK;
        if ((it & 0x3FFu) == 0x3FFu) {
            cudaError_t e = cudaStreamQuery(st);
            if (e == cudaSuccess) {
                if (*w == token) return ORX_OK;
                return fail(ORX_ERR_CUDA, "search finished without signalling completion");
            }
            if (e != cudaErrorNotReady) return fail(ORX_ERR_CUDA, "search failed: %s", cudaGetErrorString(e));
        }
#if defined(__x86_64__)
        __builtin_ia32_pause();
#endif
    }
}
int ensure_signalling(orx_index *ix) {
    if (!ix->cur->h_done.p) {
        CK(ix->cur->h_done.ensure(3));
        ix->cur->h_done.p[0] = 0;
        ix->cur->h_done.p[1] = 0;
        ix->cur->h_done.p[2] = 0;
    }
    if (!ix->cur->d_counters.p) {
        CK(ix->cur->d_counters.ensure(2));
        CK(cudaMemsetAsync(ix->cur->d_counters.p, 0, ix->cur->d_counters.n * sizeof(unsigned int), ix->stream));
    }
    return ORX_OK;
}

// ---- where a search's results land: the caller's device arrays, or the slot's mapped pinned staging (the kernels write
//      it over PCIe) that deliver_results copies into the caller's host arrays after the wait.  Flags always go to the
//      staging.
int prepare_results(SearchSlot *sl, int nq, int k, bool on_dev, orx_id *ids, double *dist, int *counts,
                    orx::ResultOut *out) {
    const size_t nk = (size_t)nq * k;
    CK(sl->h_flags.ensure(nq));
    if (!on_dev) {
        CK(sl->h_ids.ensure(nk));
        CK(sl->h_dist.ensure(nk));
        CK(sl->h_counts.ensure(nq));
    }
    *out = on_dev ? orx::ResultOut{ids, dist, counts, sl->h_flags.p}
                  : orx::ResultOut{sl->h_ids.p, sl->h_dist.p, sl->h_counts.p, sl->h_flags.p};
    return ORX_OK;
}
void deliver_results(const SearchSlot *sl, int nq, int k, bool on_dev, orx_id *ids, double *dist, int *counts) {
    if (on_dev) return;
    const size_t nk = (size_t)nq * k;
    memcpy(ids, sl->h_ids.p, nk * sizeof(orx_id));
    memcpy(dist, sl->h_dist.p, nk * sizeof(double));
    memcpy(counts, sl->h_counts.p, nq * sizeof(int));
}
int outputs_on_device(const orx_id *ids, const double *dist, const int *counts, bool *on_dev) {
    *on_dev = is_device_ptr(ids);
    if (*on_dev != is_device_ptr(dist) || *on_dev != is_device_ptr(counts))
        return fail(ORX_ERR_INVALID, "out_ids, out_dist and out_counts must all be host or all be device");
    return ORX_OK;
}

// ---- the verdict of a finished search from the flags on the host (bit 1: non-finite query; bit 3: a peer failed) and,
//      when `peer` names the other parties of a sharded search, the merge's timeout word.  *unproven: a query has bit 0.
int search_verdict(const SearchSlot *sl, int nq, const char *peer, bool *unproven) {
    if (peer && sl->h_done.p[1]) return fail(ORX_ERR_CUDA, "%s did not publish its candidates within 10 s", peer);
    bool any = false;
    for (int j = 0; j < nq; ++j) {
        const int f = sl->h_flags.p[j];
        if (peer && (f & 8)) return fail(ORX_ERR_CUDA, "%s failed (query %d)", peer, j);
        if (f & 2) return fail(ORX_ERR_NONFINITE, "NaN or infinite value not allowed in vector (query %d)", j);
        any |= (f & 1) != 0;
    }
    *unproven = any;
    return ORX_OK;
}

// ---- re-answer the queries whose flag bit 0 (unproven) is set.  `flags` is where the kernels
//      write (device or mapped host); hflags is a host-readable copy, refreshed here as needed.
int resolve_unproven(orx_index *ix, const float *q_src, int nq, int k, const orx::ResultOut &out,
                     int *hflags, int path, bool host_readable) {
    int *flags = out.flags;
    const SearchCtx ctx = plain_ctx(out);
    cudaStream_t st = ix->stream;
    // level 1: coarse tensor-core pass unproven -> exact fp32 scan for those queries
    if (path == 2) {
        for (int j = 0; j < nq;) {
            if (!(hflags[j] & 1)) { ++j; continue; }
            int j1 = j + 1;                                    // a run of flagged neighbours shares its table passes
            while (j1 < nq && (hflags[j1] & 1)) ++j1;
            ix->stats.fallback_gemv += (uint64_t)(j1 - j);
            int rc = gemv_pass(ix, q_src, j, j1 - j, k, ctx, nullptr, /*allow_image=*/false);
            if (rc != ORX_OK) return rc;
            j = j1;
        }
        if (!host_readable) CK(cudaMemcpyAsync(hflags, flags, nq * sizeof(int), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
    }
    // level 2: still unproven (dense near-ties, NaN rows, zero query) -> exhaustive collect
    for (int j = 0; j < nq; ++j) {
        if (!(hflags[j] & 1)) continue;
        int cnt = 0;
        double dk = NAN;
        if (!host_readable) {
            CK(cudaMemcpyAsync(&cnt, out.counts + j, sizeof(int), cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
            if (cnt > 0) {
                CK(cudaMemcpyAsync(&dk, out.dist + (size_t)j * k + cnt - 1, sizeof(double), cudaMemcpyDeviceToHost, st));
                CK(cudaStreamSynchronize(st));
            }
        } else {
            cnt = out.counts[j];
            if (cnt > 0) dk = out.dist[(size_t)j * k + cnt - 1];
        }
        const bool force_all = (hflags[j] & 4) != 0 || cnt < k;
        int rc = exhaustive_query(ix, q_src, j, k, dk, force_all, out);
        if (rc != ORX_OK) return rc;
        hflags[j] &= ~1;
        if (!host_readable) CK(cudaMemsetAsync(flags + j, 0, sizeof(int), st));   // proven now (exhaustive is exact)
    }
    CK(cudaStreamSynchronize(st));
    return ORX_OK;
}

// ---- a search = submit (launch the whole chain on the slot `ix->cur`, no waiting) + wait (poll the completion word,
//      settle unproven queries, hand the results over).  orx_search is the two back to back; orx_search_submit /
//      orx_search_wait let a caller keep two searches in flight.
// joinable: orx_search_submit -- a single-query 8-bit scan runs as a lap another submit can join (orx_search holds the
// index mutex until its search is complete, so nothing can join it: it keeps the plain scan on the index stream)
int search_submit_locked(orx_index *ix, const float *queries, int nq, int k, orx_id *out_ids, double *out_dist,
                         int *out_counts, bool joinable) {
    SearchSlot::Pending &pd = ix->cur->pend;
    pd = SearchSlot::Pending{};
    pd.t_begin = std::chrono::steady_clock::now();
    pd.out_on_dev = is_device_ptr(out_ids);        // (out_dist / out_counts are documented to be of the same kind)
    pd.nq = nq;
    pd.k = k;
    pd.out_ids = out_ids;
    pd.out_dist = out_dist;
    pd.out_counts = out_counts;
    const bool out_on_dev = pd.out_on_dev;
    // a lap search runs on the slot's own stream behind everything the index stream holds now; it joins the other
    // slot's lap when that one is still running over the same rows (no write can have come between: a write settles
    // every search in flight)
    pd.lap = joinable && lap_search(ix, nq, k);
    cudaStream_t index_stream = ix->stream;
    if (pd.lap) {
        int rc = ensure_lap(ix->cur);
        if (rc != ORX_OK) return rc;
        CK(cudaEventRecord(ix->cur->ev_entry, index_stream));
        CK(cudaStreamWaitEvent(ix->cur->lap_stream, ix->cur->ev_entry, 0));
        SearchSlot *other = &ix->slot[ix->cur == &ix->slot[0] ? 1 : 0];
        const SearchSlot::Pending &op = other->pend;
        pd.lap_rows = (uint32_t)ix->n_live;
        if (op.active && op.lap && !op.complete && !op.settled && op.lap_rows == pd.lap_rows &&
            cudaEventQuery(other->ev_lap) == cudaErrorNotReady)
            pd.join_host = other;
        ix->stream = ix->cur->lap_stream;
    }
    struct RestoreStream {
        orx_index *ix;
        cudaStream_t st;
        ~RestoreStream() { ix->stream = st; }
    } restore{ix, index_stream};
    cudaStream_t st = ix->stream;
    const size_t nk = (size_t)nq * k;
    ix->cur->scan_ev_used = 0;

    int rc = prepare_results(ix->cur, nq, k, out_on_dev, out_ids, out_dist, out_counts, &pd.out);
    if (rc != ORX_OK) return rc;
    rc = ensure_signalling(ix);
    if (rc != ORX_OK) return rc;

    rc = stage_queries(ix, queries, nq, &pd.q_src);
    if (rc != ORX_OK) return rc;

    const uint32_t n_rows = (uint32_t)ix->n_live;
    if (n_rows == 0) {
        // nothing to scan: only the pgvector input check matters (settled here; the wait has nothing left to do)
        CK(ix->cur->h_prep.ensure(nq));
        CK(cudaMemcpyAsync(ix->cur->h_prep.p, ix->cur->prep.p, nq * sizeof(orx::QueryPrep), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        for (int j = 0; j < nq; ++j)
            if (ix->cur->h_prep.p[j].nonfinite)
                return fail(ORX_ERR_NONFINITE, "NaN or infinite value not allowed in vector (query %d)", j);
        if (out_on_dev) {
            CK(cudaMemsetAsync(out_ids, 0, nk * sizeof(orx_id), st));
            CK(cudaMemsetAsync(out_dist, 0xFF, nk * sizeof(double), st));   // all-ones = NaN
            CK(cudaMemsetAsync(out_counts, 0, nq * sizeof(int), st));
            CK(cudaStreamSynchronize(st));
        } else {
            memset(out_ids, 0, nk * sizeof(orx_id));
            memset(out_dist, 0xFF, nk * sizeof(double));
            memset(out_counts, 0, nq * sizeof(int));
        }
        pd.active = true;
        pd.complete = true;
        return ORX_OK;
    }
    SearchCtx ctx = plain_ctx(pd.out);
    ctx.lap = pd.lap;
    ctx.join_host = pd.join_host;
    pd.token = next_token(ix);
    ctx.done = orx::DoneArgs{ix->cur->d_counters.p, (unsigned int)nq, ix->cur->h_done.p, pd.token};
    if (pd.join_host) ix->cur->h_done.p[2] = 0;
    rc = scan_pass(ix, pd.q_src, nq, k, ctx, &pd.path);
    if (rc != ORX_OK) {
        cudaStreamSynchronize(st);          // part of the chain may be in flight: drain it, forget its count
        cudaMemsetAsync(ix->cur->d_counters.p, 0, 2 * sizeof(unsigned int), st);
        cudaGetLastError();
        return rc;
    }
    if (pd.lap) CK(cudaEventRecord(ix->cur->ev_done, st));
    pd.active = true;
    return ORX_OK;
}

// the slot of a new search: slots alternate with the ticket number; at most two searches are in flight
int claim_slot(orx_index *ix, int *ticket) {
    SearchSlot *sl = &ix->slot[ix->tickets & 1u];
    if (sl->pend.active)
        return fail(ORX_ERR_INVALID, "two searches are in flight already: wait for ticket %u first", ix->tickets - 2u);
    ix->cur = sl;
    if (ticket) *ticket = (int)(ix->tickets & 0x7FFFFFFFu);
    return ORX_OK;
}
bool any_in_flight(const orx_index *ix) { return ix->slot[0].pend.active || ix->slot[1].pend.active; }

// =========================================================================== filtered search
// the arguments every search form checks (an empty batch is valid: nothing to do)
int check_query_args(orx_index *ix, const float *queries, int nq, int dim, int k, orx_id *out_ids, double *out_dist,
                     int *out_counts) {
    if (!ix) return fail(ORX_ERR_INVALID, "index is null");
    if (dim != ORX_DIM) return fail(ORX_ERR_DIM, "different vector dimensions %d and %d", ORX_DIM, dim);
    if (k < 1 || k > ORX_MAX_K) return fail(ORX_ERR_INVALID, "k must be in [1, %d], got %d", ORX_MAX_K, k);
    if (nq < 0) return fail(ORX_ERR_INVALID, "nq must be >= 0");
    if (nq == 0) return ORX_OK;
    if (!queries || !out_ids || !out_dist || !out_counts) return fail(ORX_ERR_INVALID, "null argument");
    return ORX_OK;
}

int upload_filter(orx_index *ix, const std::vector<uint32_t> &rows, DevBuf<uint32_t> &list, DevBuf<uint32_t> &count,
                  DevBuf<uint32_t> &bits) {
    cudaStream_t st = ix->stream;
    const uint32_t m = (uint32_t)rows.size();
    CK(list.ensure(std::max<size_t>(m, 1)));
    CK(count.ensure(1));
    CK(ix->h_u32a.ensure(1));
    *ix->h_u32a.p = m;
    if (m) CK(cudaMemcpyAsync(list.p, rows.data(), m * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(count.p, ix->h_u32a.p, sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    if (m >= FILTER_SCAN_MIN_ROWS) {
        const size_t n_words = ((size_t)ix->n_live + 31) / 32;
        CK(ix->h_allow_bits.ensure(n_words));
        CK(bits.ensure(n_words));
        memset(ix->h_allow_bits.p, 0, n_words * sizeof(uint32_t));
        for (uint32_t r : rows) ix->h_allow_bits.p[r >> 5] |= 1u << (r & 31);
        CK(cudaMemcpyAsync(bits.p, ix->h_allow_bits.p, n_words * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    }
    CK(cudaStreamSynchronize(st));          // `rows` and the pinned scratch may be reused by the caller
    return ORX_OK;
}

// the eligible rows of `ids` -- ids that are live, each row once (the WHERE clause of the SQL), ascending -- uploaded
// into list / count / bits
int resolve_filter(orx_index *ix, const orx_id *ids, uint64_t n, DevBuf<uint32_t> &list, DevBuf<uint32_t> &count,
                   DevBuf<uint32_t> &bits, FilterOnDevice *out) {
    std::vector<uint32_t> rows;
    rows.reserve(n);
    for (uint64_t i = 0; i < n; ++i) {
        if (const uint32_t *r = ix->map.find(ids[i])) rows.push_back(*r);
    }
    std::sort(rows.begin(), rows.end());
    rows.erase(std::unique(rows.begin(), rows.end()), rows.end());
    int rc = upload_filter(ix, rows, list, count, bits);
    if (rc != ORX_OK) return rc;
    const uint32_t m = (uint32_t)rows.size();
    *out = FilterOnDevice{m, list.p, count.p, m >= FILTER_SCAN_MIN_ROWS ? bits.p : nullptr};
    return ORX_OK;
}

int filtered_search_locked(orx_index *ix, const FilterOnDevice &f, const float *queries, int nq, int k, orx_id *out_ids,
                           double *out_dist, int *out_counts) {
    cudaStream_t st = ix->stream;
    bool out_on_dev = false;
    int rc = outputs_on_device(out_ids, out_dist, out_counts, &out_on_dev);
    if (rc != ORX_OK) return rc;
    const uint32_t m = f.m;

    const float *q_src = nullptr;
    rc = stage_queries(ix, queries, nq, &q_src);
    if (rc != ORX_OK) return rc;
    CK(ix->cur->h_prep.ensure(nq));
    CK(cudaMemcpyAsync(ix->cur->h_prep.p, ix->cur->prep.p, nq * sizeof(orx::QueryPrep), cudaMemcpyDeviceToHost, st));
    orx::ResultOut out;
    rc = prepare_results(ix->cur, nq, k, out_on_dev, out_ids, out_dist, out_counts, &out);
    if (rc != ORX_OK) return rc;
    CK(ix->fb_dist.ensure(std::max<size_t>(m, 1)));
    // exact by construction: every eligible row is rescored canonically and the k best are selected
    auto list_query = [&](int j) {
        if (m)
            orx::launch_rescore_list(ix->dtype, ix->table, ix->n2, ix->row_ids, q_src + (size_t)j * ORX_DIM, ix->cur->prep.p + j,
                                     f.list, f.count, ix->fb_dist.p, st);
        orx::launch_select_list(ix->row_ids, f.list, f.count, ix->fb_dist.p, k, out.ids + (size_t)j * k,
                                out.dist + (size_t)j * k, out.counts + j, st);
        ix->stats.kernel_launches += m ? 2 : 1;
    };
    if (f.bits != nullptr && m > 32u * (uint32_t)orx::slots_for_k(k)) {
        // many eligible rows: a scan restricted to them, with the candidate proof of orx_search; the rare unproven
        // query is re-answered by the exact list path
        ix->cur->scan_ev_used = 0;
        int path = 1;
        rc = scan_pass(ix, q_src, nq, k, plain_ctx(out), &path, &f);
        if (rc != ORX_OK) return rc;
        CK(cudaStreamSynchronize(st));
        CK(cudaGetLastError());
        harvest_scan_events(ix);
        ix->stats.last_path = path;
        for (int j = 0; j < nq; ++j) {
            if (!(ix->cur->h_flags.p[j] & 1) || (ix->cur->h_flags.p[j] & 2)) continue;
            ix->stats.fallback_exhaustive += 1;
            list_query(j);
        }
    } else {
        // few rows: no scan at all
        for (int j = 0; j < nq; ++j) list_query(j);
    }
    CK(cudaStreamSynchronize(st));
    CK(cudaGetLastError());
    for (int j = 0; j < nq; ++j)
        if (ix->cur->h_prep.p[j].nonfinite)
            return fail(ORX_ERR_NONFINITE, "NaN or infinite value not allowed in vector (query %d)", j);
    deliver_results(ix->cur, nq, k, out_on_dev, out_ids, out_dist, out_counts);
    ix->stats.searches += 1;
    ix->stats.queries += nq;
    return ORX_OK;
}

// the live rows of a filter handle, re-resolved when the id -> row map has changed since (upsert of new ids, delete,
// import)
int filter_on_device(orx_index *ix, orx_filter *f, FilterOnDevice *out) {
    if (!f->resolved || f->generation != ix->generation) {
        int rc = resolve_filter(ix, f->ids.data(), f->ids.size(), f->d_list, f->d_count, f->d_bits, &f->dev);
        if (rc != ORX_OK) return rc;
        f->generation = ix->generation;
        f->resolved = true;
    }
    *out = f->dev;
    return ORX_OK;
}

// =========================================================================== maximal marginal relevance
// Two phases per chunk of queries, under the caller's lock: `fetch` = the exact top-fetch_k (any search path) into host
// arrays; `gather` = the candidates' stored rows as the fp32 matrix [m, fetch_k, ORX_DIM] on `kx`'s device (zero rows
// past a query's count); then mmr_select_kernel on `kx`'s stream picks positions, and the host maps them back to the
// candidates' ids and distances.
constexpr int MMR_QCHUNK = 256;          // queries per chunk: candidate matrix <= 256 x 128 x 4 KB = 128 MB

using MmrFetch = std::function<int(const float *q, int m, orx_id *ids, double *dist, int *cnt)>;
using MmrGather = std::function<int(const orx_id *ids, const int *cnt, int m, const float **rows)>;

int check_mmr_args(orx_index *ix, const float *queries, int nq, int dim, int k, int fetch_k, double lam,
                   orx_id *out_ids, double *out_dist, int *out_counts) {
    if (k < 1 || fetch_k < k || fetch_k > ORX_MAX_K)
        return fail(ORX_ERR_INVALID, "need 1 <= k <= fetch_k <= %d, got k = %d, fetch_k = %d", ORX_MAX_K, k, fetch_k);
    if (!(lam >= 0.0 && lam <= 1.0)) return fail(ORX_ERR_INVALID, "lambda_mult must be a number in [0, 1], got %g", lam);
    int rc = check_query_args(ix, queries, nq, dim, k, out_ids, out_dist, out_counts);
    if (rc != ORX_OK || nq == 0) return rc;
    if (is_device_ptr(queries) || is_device_ptr(out_ids) || is_device_ptr(out_dist) || is_device_ptr(out_counts))
        return fail(ORX_ERR_INVALID, "MMR search takes host queries and host outputs");
    return ORX_OK;
}

int mmr_run(orx_index *kx, const float *queries, int nq, int k, int fetch_k, double lam, orx_id *out_ids,
            double *out_dist, int *out_counts, const MmrFetch &fetch, const MmrGather &gather) {
    std::vector<orx_id> ids;
    std::vector<double> dist;
    std::vector<int> cnt, sel;
    for (int q0 = 0; q0 < nq; q0 += MMR_QCHUNK) {
        const int m = std::min(MMR_QCHUNK, nq - q0);
        const size_t nc = (size_t)m * fetch_k;
        ids.assign(nc, orx_id{0, 0});
        dist.assign(nc, NAN);
        cnt.assign(m, 0);
        sel.assign((size_t)m * k, -1);
        int rc = fetch(queries + (size_t)q0 * ORX_DIM, m, ids.data(), dist.data(), cnt.data());
        if (rc != ORX_OK) return rc;
        const float *rows = nullptr;
        rc = gather(ids.data(), cnt.data(), m, &rows);
        if (rc != ORX_OK) return rc;
        {
            DeviceGuard g(kx->device);
            cudaStream_t st = kx->stream;
            CK(kx->mmr_dist.ensure(nc));
            CK(kx->mmr_cnt.ensure(m));
            CK(kx->mmr_sel.ensure((size_t)m * k));
            CK(cudaMemcpyAsync(kx->mmr_dist.p, dist.data(), nc * sizeof(double), cudaMemcpyHostToDevice, st));
            CK(cudaMemcpyAsync(kx->mmr_cnt.p, cnt.data(), m * sizeof(int), cudaMemcpyHostToDevice, st));
            orx::launch_mmr_select(rows, kx->mmr_dist.p, kx->mmr_cnt.p, m, fetch_k, k, lam, kx->mmr_sel.p, st);
            kx->stats.kernel_launches += 1;
            CK(cudaGetLastError());
            CK(cudaMemcpyAsync(sel.data(), kx->mmr_sel.p, (size_t)m * k * sizeof(int), cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
        }
        for (int j = 0; j < m; ++j) {
            const int n = std::min(k, cnt[j]);
            const size_t o = (size_t)(q0 + j) * k;
            out_counts[q0 + j] = n;
            for (int t = 0; t < k; ++t) {
                const int p = t < n ? sel[(size_t)j * k + t] : -1;
                if (t < n && (p < 0 || p >= cnt[j]))
                    return fail(ORX_ERR_CUDA, "MMR selection returned position %d of %d (query %d)", p, cnt[j], q0 + j);
                out_ids[o + t] = p >= 0 ? ids[(size_t)j * fetch_k + p] : orx_id{0, 0};
                out_dist[o + t] = p >= 0 ? dist[(size_t)j * fetch_k + p] : NAN;
            }
        }
    }
    return ORX_OK;
}

// candidates of a one-GPU index -> their table rows (the map is stable: the caller holds ix->mu since the fetch)
int mmr_gather_local(orx_index *ix, const orx_id *ids, const int *cnt, int m, int fetch_k, const float **rows) {
    const size_t nc = (size_t)m * fetch_k;
    std::vector<uint32_t> idx(nc, 0xFFFFFFFFu);
    for (int j = 0; j < m; ++j)
        for (int p = 0; p < cnt[j]; ++p) {
            const uint32_t *r = ix->map.find(ids[(size_t)j * fetch_k + p]);
            if (!r) return fail(ORX_ERR_CUDA, "MMR candidate of query %d is not in the table", j);
            idx[(size_t)j * fetch_k + p] = *r;
        }
    CK(ix->mmr_idx.ensure(nc));
    CK(ix->mmr_rows.ensure(nc * ORX_DIM));
    CK(cudaMemcpyAsync(ix->mmr_idx.p, idx.data(), nc * sizeof(uint32_t), cudaMemcpyHostToDevice, ix->stream));
    orx::launch_gather_rows(ix->dtype, ix->table, ix->mmr_idx.p, (uint32_t)nc, ix->mmr_rows.p, ix->stream);
    ix->stats.kernel_launches += 1;
    CK(cudaStreamSynchronize(ix->stream));      // `idx` is host memory of this frame
    *rows = ix->mmr_rows.p;
    return ORX_OK;
}

int mmr_local(orx_index *ix, const float *queries, int nq, int k, int fetch_k, double lam, orx_id *out_ids,
              double *out_dist, int *out_counts, const MmrFetch &fetch) {
    return mmr_run(ix, queries, nq, k, fetch_k, lam, out_ids, out_dist, out_counts, fetch,
                   [&](const orx_id *ids, const int *cnt, int m, const float **rows) {
                       return mmr_gather_local(ix, ids, cnt, m, fetch_k, rows);
                   });
}

// =========================================================================== sharded search
// The gather buffer of `world` ranks: two sets of `world` slots (one slot = a rank's block of up to XQ_MAX x 32
// results), then 2 x world arrival words.  Returns its size.
size_t exchange_layout(Exchange *x, int world, int rank) {
    x->world = world;
    x->rank = rank;
    x->slot_bytes = slot_layout(XQ_MAX, 32).bytes;          // nq * k <= XQ_MAX * 32 per exchange round
    x->set_bytes = x->slot_bytes * world;
    x->flags_off = 2 * x->set_bytes;
    return x->flags_off + 2 * (size_t)world * XFLAG_STRIDE;
}
// d_peer_slot / d_peer_flag of both sets: my slot and my arrival word inside each target's gather buffer (every rank's,
// or the group root's), allocated on the current device
cudaError_t upload_peer_tables(Exchange *x, const std::vector<char *> &targets) {
    const int n = (int)targets.size();
    x->n_targets = n;
    std::vector<void *> slots(n);
    std::vector<uint32_t *> flags(n);
    for (int s = 0; s < 2; ++s) {
        for (int t = 0; t < n; ++t) {
            slots[t] = targets[t] + (size_t)s * x->set_bytes + (size_t)x->rank * x->slot_bytes;
            flags[t] = reinterpret_cast<uint32_t *>(targets[t] + x->flags_off + ((size_t)s * x->world + x->rank) * XFLAG_STRIDE);
        }
        cudaError_t e = cudaMalloc(&x->d_peer_slot[s], n * sizeof(void *));
        if (e == cudaSuccess) e = cudaMalloc(&x->d_peer_flag[s], n * sizeof(uint32_t *));
        if (e == cudaSuccess) e = cudaMemcpy(x->d_peer_slot[s], slots.data(), n * sizeof(void *), cudaMemcpyHostToDevice);
        if (e == cudaSuccess) e = cudaMemcpy(x->d_peer_flag[s], flags.data(), n * sizeof(uint32_t *), cudaMemcpyHostToDevice);
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}
// Queries per exchange round at this k (a slot holds XQ_MAX of them at k <= 32), or 0 when one round cannot hold
// world x k candidates per query.
int exchange_queries(size_t world, int k) {
    if (world * k > 1024) return 0;
    return k <= 32 ? XQ_MAX : XQ_MAX * 32 / k;
}

// merge what every rank published under `seq` into the caller's result arrays; the last merge CTA writes `token`
int launch_shard_merge(orx_index *ix, Exchange *x, int nq, int k, const orx::ResultOut &final_out, const SlotLayout &L,
                       uint32_t seq, uint32_t token) {
    const int set = seq & 1;
    const uint32_t *arrival = reinterpret_cast<const uint32_t *>(x->base + x->flags_off + (size_t)set * x->world * XFLAG_STRIDE);
    orx::launch_merge_wait(x->world, x->rank, nq, k, x->base + (size_t)set * x->set_bytes, x->slot_bytes, L.dist_off,
                           L.counts_off, L.flags_off, arrival, (int)(XFLAG_STRIDE / 4), seq, final_out.ids,
                           final_out.dist, final_out.counts, ix->cur->h_flags.p, ix->cur->h_myflags.p, ix->cur->h_redo.p,
                           ix->cur->h_done.p + 1, orx::DoneArgs{ix->cur->d_counters.p + 1, (unsigned int)nq, ix->cur->h_done.p, token},
                           ix->stream);
    ix->stats.kernel_launches += 1;
    CK(cudaGetLastError());
    return ORX_OK;
}
// stand-alone push of the block that sits in my local slot of set (seq & 1) (paths that do not end in finalize)
int launch_shard_publish(orx_index *ix, Exchange *x, const SlotLayout &L, uint32_t seq) {
    const int set = seq & 1;
    char *my_slot = x->base + (size_t)set * x->set_bytes + (size_t)x->rank * x->slot_bytes;
    orx::launch_publish(my_slot, x->d_peer_slot[set], x->d_peer_flag[set], x->n_targets, L.bytes, seq, ix->stream);
    ix->stats.kernel_launches += 1;
    CK(cudaGetLastError());
    return ORX_OK;
}

// Publish a zeroed block from the slot's scratch (the shard may own no local slot) in place of this shard's results
// under `seq`.  Its flags carry the query check (`prep`: an empty shard) or, with prep null, bit 3 (this shard failed:
// whoever merges fails fast instead of waiting for it).
cudaError_t publish_substitute(orx_index *ix, Exchange *x, const SlotLayout &L, int nq, uint32_t seq,
                               const orx::QueryPrep *prep) {
    cudaStream_t st = ix->stream;
    cudaError_t e = ix->cur->blk.ensure((L.bytes + 7) / 8);
    if (e != cudaSuccess) return e;
    char *blk = reinterpret_cast<char *>(ix->cur->blk.p);
    int *flags = reinterpret_cast<int *>(blk + L.flags_off);
    cudaMemsetAsync(blk, 0, L.bytes, st);
    if (prep) orx::launch_flags_from_prep(prep, nq, flags, st);
    else orx::launch_fill_flags(flags, nq, 8, st);
    orx::launch_publish(blk, x->d_peer_slot[seq & 1], x->d_peer_flag[seq & 1], x->n_targets, L.bytes, seq, st);
    return cudaGetLastError();
}

// Round 1 of a row-sharded search on ONE shard, launches only (no wait): stage the batch, scan, finalize pushes the
// shard's block into its targets' gather buffers under `seq`.  On failure the shard still publishes a block whose flags
// carry bit 3, so that whoever merges fails fast instead of waiting for it.
int shard_round1(orx_index *ix, Exchange *x, const float *queries, bool src_pinned, int nq, int k, const SlotLayout &L,
                 uint32_t seq, const float **q_src, int *path) {
    cudaStream_t st = ix->stream;
    ix->cur->scan_ev_used = 0;
    const int set = seq & 1;
    int rc = ensure_signalling(ix);
    if (rc == ORX_OK) rc = stage_queries(ix, queries, nq, q_src, src_pinned);
    if (rc == ORX_OK) {
        if (ix->n_live == 0) {
            // an empty shard contributes nothing (its peers may still hold rows); flags carry the query check
            if (publish_substitute(ix, x, L, nq, seq, ix->cur->prep.p) != cudaSuccess)
                rc = fail(ORX_ERR_CUDA, "publishing an empty shard's block failed");
            ix->stats.kernel_launches += 2;
        } else {
            SearchCtx ctx{};
            ctx.pub = orx::PublishArgs{reinterpret_cast<char *const *>(x->d_peer_slot[set]), x->d_peer_flag[set],
                                       x->n_targets, seq, L.dist_off, L.counts_off, L.flags_off};
            ctx.done = orx::DoneArgs{ix->cur->d_counters.p, (unsigned int)nq, nullptr, 0u};
            rc = scan_pass(ix, *q_src, nq, k, ctx, path);
        }
    }
    if (rc != ORX_OK) {
        const std::string why = g_err;
        cudaStreamSynchronize(st);
        if (ix->cur->d_counters.p) cudaMemsetAsync(ix->cur->d_counters.p, 0, 2 * sizeof(unsigned int), st);
        publish_substitute(ix, x, L, nq, seq, nullptr);
        cudaStreamSynchronize(st);
        cudaGetLastError();
        g_err = why;
    }
    return rc;
}

int sharded_submit_locked(orx_index *ix, Exchange *x, const float *queries, int nq, int k, orx_id *out_ids,
                          double *out_dist, int *out_counts) {
    SearchSlot::Pending &pd = ix->cur->pend;
    pd = SearchSlot::Pending{};
    pd.t_begin = std::chrono::steady_clock::now();
    pd.sharded = true;
    pd.nq = nq;
    pd.k = k;
    pd.out_ids = out_ids;
    pd.out_dist = out_dist;
    pd.out_counts = out_counts;
    int rc = outputs_on_device(out_ids, out_dist, out_counts, &pd.out_on_dev);
    if (rc != ORX_OK) return rc;
    pd.L = slot_layout(nq, k);
    if (pd.L.bytes > x->slot_bytes) return fail(ORX_ERR_INVALID, "sharded search limited to %d queries per call", XQ_MAX);

    CK(ix->cur->h_myflags.ensure(nq));
    CK(ix->cur->h_redo.ensure(1));
    rc = prepare_results(ix->cur, nq, k, pd.out_on_dev, out_ids, out_dist, out_counts, &pd.out);
    if (rc != ORX_OK) return rc;
    rc = ensure_signalling(ix);
    if (rc != ORX_OK) return rc;
    *ix->cur->h_redo.p = 0;
    ix->cur->h_done.p[1] = 0;

    // ---- round 1: scan, finalize pushes my block into every rank's gather buffer, merge what arrives
    pd.seq = ++x->seq;
    rc = shard_round1(ix, x, queries, false, nq, k, pd.L, pd.seq, &pd.q_src, &pd.path);
    if (rc != ORX_OK) return rc;
    pd.token = next_token(ix);
    rc = launch_shard_merge(ix, x, nq, k, pd.out, pd.L, pd.seq, pd.token);
    if (rc != ORX_OK) return rc;
    pd.active = true;
    return ORX_OK;
}

// ---- the wait of a search submitted on `ix->cur` (one GPU, or one rank of the row-sharded search): poll the completion
//      word, check the flags, settle unproven queries, hand the results over
int search_wait_locked(orx_index *ix) {
    SearchSlot::Pending &pd = ix->cur->pend;
    if (!pd.active) return fail(ORX_ERR_INVALID, "no search in flight under this ticket");
    pd.active = false;
    if (pd.settled) {
        if (pd.settled_rc != ORX_OK) g_err = pd.settled_err;
        return pd.settled_rc;
    }
    const int nq = pd.nq, k = pd.k;
    if (!pd.complete) {
        const char *peer = pd.sharded ? "sharded search: a peer rank" : nullptr;
        int rc = wait_done(ix, pd.token);       // the last kernel wrote the completion word; flags are on the host
        if (rc != ORX_OK) return rc;
        if (pd.lap) {                           // the index stream (the caller's) is ordered after the search
            CK(cudaStreamWaitEvent(ix->stream, ix->cur->ev_done, 0));
            if (pd.join_host && ix->cur->h_done.p[2] != 0) {
                ix->stats.shared_scans += 1;
                ix->shared_rows += ix->cur->h_done.p[2];
            }
        }
        bool unproven = false;
        rc = search_verdict(ix->cur, nq, peer, &unproven);
        if (rc != ORX_OK) return rc;
        if (!pd.sharded && unproven) {
            rc = resolve_unproven(ix, pd.q_src, nq, k, pd.out, ix->cur->h_flags.p, pd.path, /*host_readable=*/!pd.out_on_dev);
            if (rc != ORX_OK) return rc;
        }
        if (pd.sharded && *ix->cur->h_redo.p) {
            // ---- round 2 (every rank sees the same redo word): ranks with unproven queries re-answer them
            //      exactly, everybody republishes and merges again under the next sequence number.  (With another search in
            //      flight that number selects the same buffer set as round 1 did; it is free again by then: this round is
            //      stream-ordered behind the other search's merge, which needed every peer's publish, which every peer
            //      issued after finishing ITS merge of round 1.)
            Exchange *x = ix->xchg;
            cudaStream_t st = ix->stream;
            const SlotLayout &L = pd.L;
            char *slot = x->base + (size_t)(pd.seq & 1) * x->set_bytes + (size_t)x->rank * x->slot_bytes;  // my block, local copy
            const uint32_t seq2 = ++x->seq;
            char *slot2 = x->base + (size_t)(seq2 & 1) * x->set_bytes + (size_t)x->rank * x->slot_bytes;
            if (slot2 != slot) CK(cudaMemcpyAsync(slot2, slot, L.bytes, cudaMemcpyDeviceToDevice, st));
            const orx::ResultOut mine2{reinterpret_cast<orx_id *>(slot2), reinterpret_cast<double *>(slot2 + L.dist_off),
                                       reinterpret_cast<int *>(slot2 + L.counts_off), reinterpret_cast<int *>(slot2 + L.flags_off)};
            bool mine_unproven = false;
            for (int j = 0; j < nq; ++j) mine_unproven |= (ix->cur->h_myflags.p[j] & 1) != 0;
            if (mine_unproven && ix->n_live > 0)
                rc = resolve_unproven(ix, pd.q_src, nq, k, mine2, ix->cur->h_myflags.p, pd.path, /*host_readable=*/false);
            if (rc != ORX_OK) {
                const std::string why = g_err;
                publish_substitute(ix, x, L, nq, seq2, nullptr);
                ix->stats.kernel_launches += 1;
                cudaStreamSynchronize(st);
                cudaGetLastError();
                g_err = why;
                return rc;
            }
            *ix->cur->h_redo.p = 0;
            rc = launch_shard_publish(ix, x, L, seq2);
            if (rc != ORX_OK) return rc;
            const uint32_t token = next_token(ix);
            rc = launch_shard_merge(ix, x, nq, k, pd.out, L, seq2, token);
            if (rc != ORX_OK) return rc;
            rc = wait_done(ix, token);
            if (rc != ORX_OK) return rc;
            rc = search_verdict(ix->cur, nq, peer, &unproven);
            if (rc != ORX_OK) return rc;
            if (*ix->cur->h_redo.p) return fail(ORX_ERR_CUDA, "sharded search: a rank could not prove its candidates");
        }
        deliver_results(ix->cur, nq, k, pd.out_on_dev, pd.out_ids, pd.out_dist, pd.out_counts);
        harvest_scan_events(ix);
        ix->stats.last_path = pd.path;
    }
    ix->stats.last_search_ms =
        std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - pd.t_begin).count();
    ix->stats.searches += 1;
    ix->stats.queries += nq;
    return ORX_OK;
}

// one search on a fresh slot, submitted and waited for; x: the row-sharded search over that exchange
int search_locked(orx_index *ix, Exchange *x, const float *queries, int nq, int k, orx_id *out_ids, double *out_dist,
                  int *out_counts) {
    int rc = claim_slot(ix, nullptr);
    if (rc != ORX_OK) return rc;
    rc = x ? sharded_submit_locked(ix, x, queries, nq, k, out_ids, out_dist, out_counts)
           : search_submit_locked(ix, queries, nq, k, out_ids, out_dist, out_counts, /*joinable=*/false);
    if (rc != ORX_OK) return rc;
    ix->tickets += 1;
    return search_wait_locked(ix);
}

// A write (upsert / delete / import) is ordered AFTER every search submitted before it: the searches in flight are
// completed here -- including the exact re-answer of queries the fast path could not prove, which must see the table as
// it was -- in ticket order, their verdicts kept for the caller's orx_search_wait.  (Output buffers given at submit are
// filled now; they have to stay valid until the wait anyway.)
void settle_in_flight(orx_index *ix) {
    SearchSlot *order[2] = {&ix->slot[ix->tickets & 1u], &ix->slot[(ix->tickets + 1u) & 1u]};     // older ticket first
    for (SearchSlot *sl : order) {
        SearchSlot::Pending &pd = sl->pend;
        if (!pd.active || pd.settled) continue;
        ix->cur = sl;
        const std::string keep = g_err;
        const int rc = search_wait_locked(ix);
        pd.settled = true;
        pd.settled_rc = rc;
        pd.settled_err = g_err;
        pd.active = true;                   // still owed to the caller
        g_err = keep;
    }
}

#include "group.inl"

}  // namespace

namespace orx {
int device_sms() {
    static int cache[64] = {0};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 1;
    int v = cache[dev];
    if (v == 0) {
        if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0) v = 1;
        cache[dev] = v;
    }
    return v;
}
int set_error(int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}
int index_device(const orx_index *ix) {
    if (ix->group) ix = ix->group->shards[0];          // a multi-GPU index stages on its first device
    return ix->device;
}
void index_count_launches(orx_index *ix, uint64_t n) {
    if (ix->group) ix = ix->group->shards[0];
    std::lock_guard<std::mutex> lk(ix->mu);
    ix->stats.kernel_launches += n;
}
}  // namespace orx

// =============================================================================== C-ABI
extern "C" {

const char *orx_last_error(void) { return g_err.c_str(); }
const char *orx_version(void) { return "orx 0.1 (sm_100a)"; }

int orx_create(orx_index **out, int dim, int dtype, uint64_t capacity_rows, int device) {
    if (!out) return fail(ORX_ERR_INVALID, "out is null");
    *out = nullptr;
    if (dim != ORX_DIM) return fail(ORX_ERR_DIM, "expected %d dimensions, not %d", ORX_DIM, dim);
    if (dtype != ORX_DTYPE_F32 && dtype != ORX_DTYPE_BF16) return fail(ORX_ERR_INVALID, "unknown dtype %d", dtype);
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(ORX_ERR_CUDA, "no CUDA device: this engine has no CPU fallback");
    }
    if (device < 0 || device >= ndev) return fail(ORX_ERR_INVALID, "device %d out of range (%d present)", device, ndev);
    DeviceGuard g(device);
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
        return fail(ORX_ERR_CUDA, "device %d is sm_%d%d; this library is built for sm_100a (B200) only", device,
                    prop.major, prop.minor);
    orx_index *ix = new orx_index();
    ix->device = device;
    ix->dtype = dtype;
    uint64_t cap = std::max<uint64_t>(capacity_rows, 1024);
    if (cap >= 0xFFFFFFFFull) {
        delete ix;
        return fail(ORX_ERR_CAPACITY, "table limited to 2^32-2 rows per GPU");
    }
    int rc = alloc_table(ix, cap);
    if (rc != ORX_OK) {
        orx_destroy(ix);
        return rc;
    }
    ix->slot[0].umma = orx::umma_plan_create(device);
    ix->slot[1].umma = orx::umma_plan_create(device);
    ix->host_row_ids.reserve(cap);
    ix->map.reserve(cap);
    *out = ix;
    return ORX_OK;
}

int orx_create_multi(orx_index **out, int dim, int dtype, uint64_t capacity_rows, const int *devices, int n_devices) {
    if (!out) return fail(ORX_ERR_INVALID, "out is null");
    *out = nullptr;
    if (dim != ORX_DIM) return fail(ORX_ERR_DIM, "expected %d dimensions, not %d", ORX_DIM, dim);
    if (dtype != ORX_DTYPE_F32 && dtype != ORX_DTYPE_BF16) return fail(ORX_ERR_INVALID, "unknown dtype %d", dtype);
    if (!devices || n_devices < 1 || n_devices > 64) return fail(ORX_ERR_INVALID, "n_devices must be in [1, 64]");
    return group_create(out, dtype, capacity_rows, devices, n_devices);
}

int orx_shard_count(const orx_index *ix) {
    if (!ix) return 0;
    return ix->group ? (int)ix->group->shards.size() : 1;
}

void orx_destroy(orx_index *ix) {
    if (!ix) return;
    if (ix->group) {
        group_destroy(ix);
        return;
    }
    DeviceGuard g(ix->device);
    cudaDeviceSynchronize();
    for (SearchSlot &sl : ix->slot) {
        if (sl.umma) orx::umma_plan_destroy(sl.umma);
        sl.release();
    }
    cudaFree(ix->table);
    cudaFree(ix->scale);
    cudaFree(ix->n2);
    cudaFree(ix->row_ids);
    free_image(ix);
    ix->fb_list.release(); ix->fb_count.release(); ix->fb_dist.release();
    ix->mmr_rows.release(); ix->mmr_stage.release(); ix->mmr_idx.release(); ix->mmr_dist.release();
    ix->mmr_cnt.release(); ix->mmr_sel.release();
    ix->allow_bits.release(); ix->h_allow_bits.release(); ix->scale_masked.release();
    ix->stage.release(); ix->d_src_idx.release(); ix->d_dst_row.release(); ix->d_ids.release();
    ix->d_flag.release(); ix->h_u32a.release(); ix->h_u32b.release(); ix->h_flag.release();
    if (ix->xchg) {
        Exchange *x = ix->xchg;
        for (int r = 0; r < (int)x->peer_base.size(); ++r)
            if (r != x->rank && x->peer_base[r]) cudaIpcCloseMemHandle(x->peer_base[r]);
        for (int s = 0; s < 2; ++s) {
            cudaFree(x->d_peer_slot[s]);
            cudaFree(x->d_peer_flag[s]);
        }
        cudaFree(x->base);
        delete x;
    }
    cudaGetLastError();
    delete ix;
}

int orx_set_stream(orx_index *ix, void *cuda_stream) {
    if (!ix) return fail(ORX_ERR_INVALID, "index is null");
    if (ix->group) return fail(ORX_ERR_INVALID, "a multi-GPU index runs on its own per-device streams");
    std::lock_guard<std::mutex> lk(ix->mu);
    DeviceGuard g(ix->device);
    cudaStreamSynchronize(ix->stream);
    ix->stream = static_cast<cudaStream_t>(cuda_stream);
    return ORX_OK;
}

int orx_set_option(orx_index *ix, int option, int value) {
    if (!ix) return fail(ORX_ERR_INVALID, "index is null");
    if (option != ORX_OPT_SCAN_TIMING && option != ORX_OPT_IMAGE_MIN_ROWS && option != ORX_OPT_IMAGE8_MIN_ROWS)
        return fail(ORX_ERR_INVALID, "unknown option %d", option);
    if (ix->group) {
        for (orx_index *s : ix->group->shards) orx_set_option(s, option, value);
        return ORX_OK;
    }
    std::lock_guard<std::mutex> lk(ix->mu);
    if (option == ORX_OPT_SCAN_TIMING) ix->scan_timing = value != 0;
    else if (option == ORX_OPT_IMAGE_MIN_ROWS) ix->image_min_rows = value < 0 ? UINT64_MAX : (uint64_t)value;
    else ix->image8_min_rows = value < 0 ? UINT64_MAX : (uint64_t)value;
    return ORX_OK;
}

uint64_t orx_size(const orx_index *ix) {
    if (!ix) return 0;
    if (ix->group) return group_size(ix->group);
    std::lock_guard<std::mutex> lk(ix->mu);
    return ix->n_live;
}
uint64_t orx_capacity(const orx_index *ix) {
    if (!ix) return 0;
    if (ix->group) {
        uint64_t c = 0;
        for (orx_index *s : ix->group->shards) c += orx_capacity(s);
        return c;
    }
    std::lock_guard<std::mutex> lk(ix->mu);
    return ix->capacity;
}
int orx_dtype(const orx_index *ix) { return ix ? ix->dtype : -1; }

uint64_t orx_mutation_count(const orx_index *ix) {
    if (!ix) return 0;
    if (ix->group) {
        uint64_t m = 0;
        for (orx_index *s : ix->group->shards) m += s->mutations.load();
        return m;
    }
    return ix->mutations.load();
}

int orx_get_stats(const orx_index *ix, orx_stats *out) {
    if (!ix || !out) return fail(ORX_ERR_INVALID, "null argument");
    if (ix->group) return group_stats(ix->group, out);
    std::lock_guard<std::mutex> lk(ix->mu);
    *out = ix->stats;
    return ORX_OK;
}

uint64_t orx_shared_rows(const orx_index *ix) {
    if (!ix || ix->group) return 0;
    std::lock_guard<std::mutex> lk(ix->mu);
    return ix->shared_rows;
}

int orx_contains(const orx_index *ix, orx_id id) {
    if (!ix) return 0;
    if (ix->group) return orx_contains(ix->group->shards[orx::shard_of_id(id, (uint32_t)ix->group->shards.size())], id);
    std::lock_guard<std::mutex> lk(ix->mu);
    return ix->map.find(id) != nullptr ? 1 : 0;
}

int orx_upsert(orx_index *ix, const orx_id *ids, const float *vecs, uint64_t n, int dim) {
    if (!ix) return fail(ORX_ERR_INVALID, "index is null");
    if (dim != ORX_DIM) return fail(ORX_ERR_DIM, "expected %d dimensions, not %d", ORX_DIM, dim);
    if (n == 0) return ORX_OK;
    if (!ids || !vecs) return fail(ORX_ERR_INVALID, "null ids/vecs");
    if (is_device_ptr(ids)) return fail(ORX_ERR_INVALID, "ids must be a host pointer");
    if (ix->group) return group_upsert(ix->group, ids, vecs, n);
    std::lock_guard<std::mutex> lk(ix->mu);
    DeviceGuard g(ix->device);
    settle_in_flight(ix);
    return upsert_locked(ix, ids, vecs, n, /*validate=*/true);
}

int orx_delete(orx_index *ix, const orx_id *ids, uint64_t n, uint64_t *n_removed) {
    if (n_removed) *n_removed = 0;
    if (!ix) return fail(ORX_ERR_INVALID, "index is null");
    if (n == 0) return ORX_OK;
    if (!ids) return fail(ORX_ERR_INVALID, "null ids");
    if (ix->group) return group_delete(ix->group, ids, n, n_removed);
    std::lock_guard<std::mutex> lk(ix->mu);
    DeviceGuard g(ix->device);
    settle_in_flight(ix);
    cudaStream_t st = ix->stream;

    std::vector<uint32_t> doomed;
    doomed.reserve(n);
    for (uint64_t i = 0; i < n; ++i) {
        const uint32_t *r = ix->map.find(ids[i]);
        if (!r) continue;                         // unknown id: ignored, like the SQL DELETE
        doomed.push_back(*r);
        ix->map.erase(ids[i]);                    // also drops a repeated id in the same call
    }
    const uint64_t d = doomed.size();
    if (d == 0) return ORX_OK;
    const uint64_t new_live = ix->n_live - d;
    // holes below the new end are filled by the surviving rows above it
    std::vector<char> dead_tail(d, 0);            // rows in [new_live, n_live) that are deleted
    std::vector<uint32_t> holes;
    for (uint32_t r : doomed) {
        if (r >= new_live) dead_tail[r - new_live] = 1;
        else holes.push_back(r);
    }
    CK(ix->h_u32a.ensure(std::max<size_t>(holes.size(), 1)));
    CK(ix->h_u32b.ensure(std::max<size_t>(holes.size(), 1)));
    size_t hmv = 0;
    for (uint64_t r = new_live; r < ix->n_live && hmv < holes.size(); ++r) {
        if (dead_tail[r - new_live]) continue;
        const uint32_t dst = holes[hmv];
        ix->h_u32a.p[hmv] = (uint32_t)r;
        ix->h_u32b.p[hmv] = dst;
        const orx_id moved = ix->host_row_ids[r];
        ix->host_row_ids[dst] = moved;
        ix->map.set(moved, dst);
        ++hmv;
    }
    ix->host_row_ids.resize(new_live);
    ix->n_live = new_live;
    ix->generation += 1;
    ix->mutations.fetch_add(1);
    if (hmv > 0) {
        CK(ix->d_src_idx.ensure(hmv));
        CK(ix->d_dst_row.ensure(hmv));
        CK(cudaMemcpyAsync(ix->d_src_idx.p, ix->h_u32a.p, hmv * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(ix->d_dst_row.p, ix->h_u32b.p, hmv * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
        orx::launch_move_rows(ix->dtype, ix->d_src_idx.p, ix->d_dst_row.p, (uint32_t)hmv, ix->table, ix->scale,
                              ix->n2, ix->row_ids, ix->image, ix->image8, st);
        ix->stats.kernel_launches += 1;
        ix->stats.rows_moved += hmv;
    }
    if (ix->image8.rows) CK(launch_recount8(ix, new_live));
    if (hmv > 0 || ix->image8.rows) {
        CK(cudaStreamSynchronize(st));
        CK(cudaGetLastError());
        if (ix->image8.rows) ix->capped8 = *ix->h_capped8.p;
    }
    if (n_removed) *n_removed = d;
    return ORX_OK;
}

int orx_search(orx_index *ix, const float *queries, int nq, int dim, int k, orx_id *out_ids, double *out_dist,
               int *out_counts) {
    int rc = check_query_args(ix, queries, nq, dim, k, out_ids, out_dist, out_counts);
    if (rc != ORX_OK || nq == 0) return rc;
    if (ix->group) return group_search(ix->group, queries, nq, k, out_ids, out_dist, out_counts);
    std::lock_guard<std::mutex> lk(ix->mu);
    DeviceGuard g(ix->device);
    return search_locked(ix, nullptr, queries, nq, k, out_ids, out_dist, out_counts);
}

namespace {
int check_search_args(orx_index *ix, const float *queries, int nq, int dim, int k, orx_id *out_ids, double *out_dist,
                      int *out_counts) {
    if (nq < 1) return fail(ORX_ERR_INVALID, "nq must be >= 1");
    int rc = check_query_args(ix, queries, nq, dim, k, out_ids, out_dist, out_counts);
    if (rc != ORX_OK) return rc;
    if (ix->group) return fail(ORX_ERR_INVALID, "asynchronous searches are per GPU: a multi-GPU index answers orx_search");
    return ORX_OK;
}
}  // namespace

int orx_search_submit(orx_index *ix, const float *queries, int nq, int dim, int k, orx_id *out_ids, double *out_dist,
                      int *out_counts, int *ticket) {
    int rc = check_search_args(ix, queries, nq, dim, k, out_ids, out_dist, out_counts);
    if (rc != ORX_OK) return rc;
    if (!ticket) return fail(ORX_ERR_INVALID, "ticket is null");
    std::lock_guard<std::mutex> lk(ix->mu);
    DeviceGuard g(ix->device);
    rc = claim_slot(ix, ticket);
    if (rc != ORX_OK) return rc;
    rc = search_submit_locked(ix, queries, nq, k, out_ids, out_dist, out_counts, /*joinable=*/true);
    if (rc != ORX_OK) return rc;
    ix->cur->pend.ticket = ix->tickets;
    ix->tickets += 1;
    return ORX_OK;
}

int orx_search_wait(orx_index *ix, int ticket) {
    if (!ix) return fail(ORX_ERR_INVALID, "index is null");
    if (ix->group) return fail(ORX_ERR_INVALID, "asynchronous searches are per GPU");
    std::lock_guard<std::mutex> lk(ix->mu);
    DeviceGuard g(ix->device);
    SearchSlot *sl = &ix->slot[(uint32_t)ticket & 1u];
    if (!sl->pend.active || (sl->pend.ticket & 0x7FFFFFFFu) != (uint32_t)ticket)
        return fail(ORX_ERR_INVALID, "ticket %d is not in flight", ticket);
    ix->cur = sl;
    return search_wait_locked(ix);
}

int orx_search_sharded_submit(orx_index *ix, const float *queries, int nq, int dim, int k, orx_id *out_ids,
                              double *out_dist, int *out_counts, int *ticket) {
    int rc = check_search_args(ix, queries, nq, dim, k, out_ids, out_dist, out_counts);
    if (rc != ORX_OK) return rc;
    if (!ticket) return fail(ORX_ERR_INVALID, "ticket is null");
    std::lock_guard<std::mutex> lk(ix->mu);
    DeviceGuard g(ix->device);
    if (!ix->xchg || !ix->xchg->connected) return fail(ORX_ERR_INVALID, "shard exchange not connected (orx_shard_export / orx_shard_connect)");
    const int qchunk = exchange_queries(ix->xchg->world, k);
    if (!qchunk) return fail(ORX_ERR_INVALID, "sharded search: world * k must be <= 1024");
    if (nq > qchunk) return fail(ORX_ERR_INVALID, "an asynchronous sharded search takes at most %d queries at k = %d", qchunk, k);
    rc = claim_slot(ix, ticket);
    if (rc != ORX_OK) return rc;
    rc = sharded_submit_locked(ix, ix->xchg, queries, nq, k, out_ids, out_dist, out_counts);
    if (rc != ORX_OK) return rc;
    ix->cur->pend.ticket = ix->tickets;
    ix->tickets += 1;
    return ORX_OK;
}

int orx_search_filtered(orx_index *ix, const float *queries, int nq, int dim, int k, const orx_id *allow_ids,
                        uint64_t n_allow, orx_id *out_ids, double *out_dist, int *out_counts) {
    int rc = check_query_args(ix, queries, nq, dim, k, out_ids, out_dist, out_counts);
    if (rc != ORX_OK || nq == 0) return rc;
    if (n_allow && !allow_ids) return fail(ORX_ERR_INVALID, "null argument");
    if (is_device_ptr(allow_ids)) return fail(ORX_ERR_INVALID, "allow_ids must be a host pointer");
    if (ix->group) return group_search_filtered(ix->group, queries, nq, k, allow_ids, n_allow, out_ids, out_dist, out_counts);
    std::lock_guard<std::mutex> lk(ix->mu);
    DeviceGuard g(ix->device);
    if (any_in_flight(ix)) return fail(ORX_ERR_INVALID, "wait for the searches in flight (orx_search_wait) first");
    FilterOnDevice f;
    rc = resolve_filter(ix, allow_ids, n_allow, ix->fb_list, ix->fb_count, ix->allow_bits, &f);
    if (rc != ORX_OK) return rc;
    return filtered_search_locked(ix, f, queries, nq, k, out_ids, out_dist, out_counts);
}

int orx_filter_create(orx_index *ix, const orx_id *allow_ids, uint64_t n_allow, orx_filter **out) {
    if (!out) return fail(ORX_ERR_INVALID, "out is null");
    *out = nullptr;
    if (!ix) return fail(ORX_ERR_INVALID, "index is null");
    if (ix->group) return fail(ORX_ERR_INVALID, "filter handles are per GPU: use orx_search_filtered on a multi-GPU index");
    if (n_allow && !allow_ids) return fail(ORX_ERR_INVALID, "null argument");
    if (is_device_ptr(allow_ids)) return fail(ORX_ERR_INVALID, "allow_ids must be a host pointer");
    orx_filter *f = new orx_filter();
    f->ix = ix;
    f->device = ix->device;
    f->ids.assign(allow_ids, allow_ids + n_allow);
    *out = f;
    return ORX_OK;
}

void orx_filter_destroy(orx_filter *f) {
    if (!f) return;
    DeviceGuard g(f->device);
    f->d_list.release();
    f->d_count.release();
    f->d_bits.release();
    cudaGetLastError();
    delete f;
}

int orx_search_with_filter(orx_index *ix, orx_filter *f, const float *queries, int nq, int dim, int k,
                           orx_id *out_ids, double *out_dist, int *out_counts) {
    int rc = check_query_args(ix, queries, nq, dim, k, out_ids, out_dist, out_counts);
    if (rc != ORX_OK || nq == 0) return rc;
    if (!f || f->ix != ix) return fail(ORX_ERR_INVALID, "filter does not belong to this index");
    std::lock_guard<std::mutex> lk(ix->mu);
    DeviceGuard g(ix->device);
    if (any_in_flight(ix)) return fail(ORX_ERR_INVALID, "wait for the searches in flight (orx_search_wait) first");
    FilterOnDevice fd;
    rc = filter_on_device(ix, f, &fd);
    if (rc != ORX_OK) return rc;
    return filtered_search_locked(ix, fd, queries, nq, k, out_ids, out_dist, out_counts);
}

int orx_search_mmr(orx_index *ix, const float *queries, int nq, int dim, int k, int fetch_k, double lambda_mult,
                   orx_id *out_ids, double *out_dist, int *out_counts) {
    int rc = check_mmr_args(ix, queries, nq, dim, k, fetch_k, lambda_mult, out_ids, out_dist, out_counts);
    if (rc != ORX_OK || nq == 0) return rc;
    if (ix->group)
        return group_search_mmr(ix->group, queries, nq, k, fetch_k, lambda_mult, nullptr, 0, false, out_ids, out_dist,
                                out_counts);
    std::lock_guard<std::mutex> lk(ix->mu);
    DeviceGuard g(ix->device);
    if (any_in_flight(ix)) return fail(ORX_ERR_INVALID, "wait for the searches in flight (orx_search_wait) first");
    return mmr_local(ix, queries, nq, k, fetch_k, lambda_mult, out_ids, out_dist, out_counts,
                     [&](const float *q, int m, orx_id *ids, double *dist, int *cnt) {
                         return search_locked(ix, nullptr, q, m, fetch_k, ids, dist, cnt);
                     });
}

int orx_search_mmr_filtered(orx_index *ix, const float *queries, int nq, int dim, int k, int fetch_k,
                            double lambda_mult, const orx_id *allow_ids, uint64_t n_allow, orx_id *out_ids,
                            double *out_dist, int *out_counts) {
    int rc = check_mmr_args(ix, queries, nq, dim, k, fetch_k, lambda_mult, out_ids, out_dist, out_counts);
    if (rc != ORX_OK || nq == 0) return rc;
    if (n_allow && !allow_ids) return fail(ORX_ERR_INVALID, "null argument");
    if (is_device_ptr(allow_ids)) return fail(ORX_ERR_INVALID, "allow_ids must be a host pointer");
    if (ix->group)
        return group_search_mmr(ix->group, queries, nq, k, fetch_k, lambda_mult, allow_ids, n_allow, true, out_ids,
                                out_dist, out_counts);
    std::lock_guard<std::mutex> lk(ix->mu);
    DeviceGuard g(ix->device);
    if (any_in_flight(ix)) return fail(ORX_ERR_INVALID, "wait for the searches in flight (orx_search_wait) first");
    FilterOnDevice f;
    rc = resolve_filter(ix, allow_ids, n_allow, ix->fb_list, ix->fb_count, ix->allow_bits, &f);
    if (rc != ORX_OK) return rc;
    return mmr_local(ix, queries, nq, k, fetch_k, lambda_mult, out_ids, out_dist, out_counts,
                     [&](const float *q, int m, orx_id *ids, double *dist, int *cnt) {
                         return filtered_search_locked(ix, f, q, m, fetch_k, ids, dist, cnt);
                     });
}

int orx_search_mmr_with_filter(orx_index *ix, orx_filter *f, const float *queries, int nq, int dim, int k,
                               int fetch_k, double lambda_mult, orx_id *out_ids, double *out_dist, int *out_counts) {
    int rc = check_mmr_args(ix, queries, nq, dim, k, fetch_k, lambda_mult, out_ids, out_dist, out_counts);
    if (rc != ORX_OK || nq == 0) return rc;
    if (ix->group) return fail(ORX_ERR_INVALID, "filter handles are per GPU: use orx_search_mmr_filtered on a multi-GPU index");
    if (!f || f->ix != ix) return fail(ORX_ERR_INVALID, "filter does not belong to this index");
    std::lock_guard<std::mutex> lk(ix->mu);
    DeviceGuard g(ix->device);
    if (any_in_flight(ix)) return fail(ORX_ERR_INVALID, "wait for the searches in flight (orx_search_wait) first");
    FilterOnDevice fd;
    rc = filter_on_device(ix, f, &fd);
    if (rc != ORX_OK) return rc;
    return mmr_local(ix, queries, nq, k, fetch_k, lambda_mult, out_ids, out_dist, out_counts,
                     [&](const float *q, int m, orx_id *ids, double *dist, int *cnt) {
                         return filtered_search_locked(ix, fd, q, m, fetch_k, ids, dist, cnt);
                     });
}

int orx_merge_topk(orx_index *ix, int n_lists, int nq, int k, const orx_id *ids, const double *dist,
                   const int *counts, orx_id *out_ids, double *out_dist, int *out_counts) {
    if (!ix) return fail(ORX_ERR_INVALID, "index is null");
    if (n_lists < 1 || nq < 0 || k < 1 || k > ORX_MAX_K || (size_t)n_lists * k > 1024)
        return fail(ORX_ERR_INVALID, "bad merge shape (n_lists=%d, nq=%d, k=%d)", n_lists, nq, k);
    if (nq == 0) return ORX_OK;
    if (!ids || !dist || !counts || !out_ids || !out_dist || !out_counts) return fail(ORX_ERR_INVALID, "null argument");
    if (ix->group) ix = ix->group->shards[0];
    std::lock_guard<std::mutex> lk(ix->mu);
    DeviceGuard g(ix->device);
    cudaStream_t st = ix->stream;
    const bool in_dev = is_device_ptr(ids), out_dev = is_device_ptr(out_ids);
    const size_t nin = (size_t)n_lists * nq * k, nout = (size_t)nq * k;
    if (in_dev && out_dev) {
        orx::launch_merge_topk(n_lists, nq, k, ids, dist, counts, 0, out_ids, out_dist, out_counts, st);
        ix->stats.kernel_launches += 1;
        CK(cudaGetLastError());
        return ORX_OK;
    }
    if (in_dev || out_dev) return fail(ORX_ERR_INVALID, "merge inputs and outputs must live on the same side");
    // host buffers: stage through device scratch (the merge itself always runs on the GPU)
    struct Scratch {                       // one allocation, released on every exit path
        char *p = nullptr;
        ~Scratch() { if (p) cudaFree(p); }
    } scratch;
    auto up16 = [](size_t b) { return (b + 15) & ~(size_t)15; };
    const size_t b_ids = nin * sizeof(orx_id), b_dist = up16(nin * sizeof(double));
    const size_t b_cnt = up16((size_t)n_lists * nq * sizeof(int));
    const size_t b_oids = nout * sizeof(orx_id), b_odist = up16(nout * sizeof(double)), b_ocnt = up16(nq * sizeof(int));
    CK(cudaMalloc(reinterpret_cast<void **>(&scratch.p), b_ids + b_dist + b_cnt + b_oids + b_odist + b_ocnt));
    orx_id *d_ids = reinterpret_cast<orx_id *>(scratch.p);
    double *d_dist = reinterpret_cast<double *>(scratch.p + b_ids);
    int *d_cnt = reinterpret_cast<int *>(scratch.p + b_ids + b_dist);
    orx_id *d_oids = reinterpret_cast<orx_id *>(scratch.p + b_ids + b_dist + b_cnt);
    double *d_odist = reinterpret_cast<double *>(scratch.p + b_ids + b_dist + b_cnt + b_oids);
    int *d_ocnt = reinterpret_cast<int *>(scratch.p + b_ids + b_dist + b_cnt + b_oids + b_odist);
    CK(cudaMemcpyAsync(d_ids, ids, nin * sizeof(orx_id), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_dist, dist, nin * sizeof(double), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_cnt, counts, (size_t)n_lists * nq * sizeof(int), cudaMemcpyHostToDevice, st));
    orx::launch_merge_topk(n_lists, nq, k, d_ids, d_dist, d_cnt, 0, d_oids, d_odist, d_ocnt, st);
    ix->stats.kernel_launches += 1;
    CK(cudaMemcpyAsync(out_ids, d_oids, nout * sizeof(orx_id), cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(out_dist, d_odist, nout * sizeof(double), cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(out_counts, d_ocnt, nq * sizeof(int), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    CK(cudaGetLastError());
    return ORX_OK;
}

int orx_merge_topk_strided(orx_index *ix, int n_lists, int nq, int k, const orx_id *ids0, const double *dist0,
                           const int *counts0, uint64_t list_stride_bytes, orx_id *out_ids, double *out_dist,
                           int *out_counts) {
    if (!ix) return fail(ORX_ERR_INVALID, "index is null");
    if (n_lists < 1 || nq < 0 || k < 1 || k > ORX_MAX_K || (size_t)n_lists * k > 1024 || list_stride_bytes == 0)
        return fail(ORX_ERR_INVALID, "bad merge shape (n_lists=%d, nq=%d, k=%d)", n_lists, nq, k);
    if (nq == 0) return ORX_OK;
    if (!ids0 || !dist0 || !counts0 || !out_ids || !out_dist || !out_counts) return fail(ORX_ERR_INVALID, "null argument");
    if (ix->group) ix = ix->group->shards[0];
    std::lock_guard<std::mutex> lk(ix->mu);
    DeviceGuard g(ix->device);
    orx::launch_merge_topk(n_lists, nq, k, ids0, dist0, counts0, (size_t)list_stride_bytes, out_ids, out_dist,
                           out_counts, ix->stream);
    ix->stats.kernel_launches += 1;
    CK(cudaGetLastError());
    return ORX_OK;
}

int orx_export_rows(orx_index *ix, uint64_t row_start, uint64_t n, orx_id *ids_out, void *rows_out) {
    if (!ix) return fail(ORX_ERR_INVALID, "index is null");
    if (n == 0) return ORX_OK;
    if (!ids_out || !rows_out) return fail(ORX_ERR_INVALID, "null argument");
    if (ix->group) return group_export_rows(ix->group, row_start, n, ids_out, rows_out);
    std::lock_guard<std::mutex> lk(ix->mu);
    DeviceGuard g(ix->device);
    if (row_start + n > ix->n_live) return fail(ORX_ERR_INVALID, "rows [%llu, %llu) exceed the %llu live rows",
                                                (unsigned long long)row_start, (unsigned long long)(row_start + n),
                                                (unsigned long long)ix->n_live);
    const size_t rb = ORX_DIM * elem_size(ix->dtype);
    memcpy(ids_out, ix->host_row_ids.data() + row_start, n * sizeof(orx_id));
    CK(cudaMemcpyAsync(rows_out, static_cast<const char *>(ix->table) + row_start * rb, n * rb, cudaMemcpyDeviceToHost,
                       ix->stream));
    CK(cudaStreamSynchronize(ix->stream));
    return ORX_OK;
}

int orx_import_rows(orx_index *ix, const orx_id *ids, const void *rows_raw, uint64_t n) {
    if (!ix) return fail(ORX_ERR_INVALID, "index is null");
    if (n == 0) return ORX_OK;
    if (!ids || !rows_raw) return fail(ORX_ERR_INVALID, "null argument");
    if (ix->group) return group_import_rows(ix->group, ids, rows_raw, n);
    std::lock_guard<std::mutex> lk(ix->mu);
    DeviceGuard g(ix->device);
    settle_in_flight(ix);
    cudaStream_t st = ix->stream;
    {   // every id must be new: this is an append, not an upsert
        std::unordered_map<orx_id, int, IdHash, IdEq> seen;
        seen.reserve(n);
        for (uint64_t i = 0; i < n; ++i)
            if (ix->map.find(ids[i]) != nullptr || !seen.emplace(ids[i], 1).second)
                return fail(ORX_ERR_INVALID, "orx_import_rows: id %llu of the batch is already present", (unsigned long long)i);
    }
    int rc = grow_table(ix, ix->n_live + n);
    if (rc != ORX_OK) return rc;
    const size_t rb = ORX_DIM * elem_size(ix->dtype);
    const uint64_t row0 = ix->n_live;
    CK(ix->d_ids.ensure(n));
    CK(ix->d_flag.ensure(1));
    CK(ix->h_flag.ensure(1));
    CK(cudaMemsetAsync(ix->d_flag.p, 0, sizeof(int), st));
    // straight into the table tail: invisible to searches until n_live moves
    CK(cudaMemcpyAsync(static_cast<char *>(ix->table) + row0 * rb, rows_raw, n * rb,
                       is_device_ptr(rows_raw) ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(ix->d_ids.p, ids, n * sizeof(orx_id), cudaMemcpyHostToDevice, st));
    orx::launch_adopt_rows(ix->dtype, ix->table, (uint32_t)row0, (uint32_t)n, ix->d_ids.p, ix->scale, ix->n2,
                           ix->row_ids, ix->d_flag.p, ix->image, ix->image8, st);
    ix->stats.kernel_launches += 1;
    if (ix->image8.rows) CK(launch_recount8(ix, row0 + n));
    CK(cudaMemcpyAsync(ix->h_flag.p, ix->d_flag.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    CK(cudaGetLastError());
    if (*ix->h_flag.p) return fail(ORX_ERR_NONFINITE, "NaN or infinite value not allowed in vector");
    if (ix->image8.rows) ix->capped8 = *ix->h_capped8.p;
    ix->host_row_ids.resize(row0 + n);
    for (uint64_t i = 0; i < n; ++i) {
        ix->host_row_ids[row0 + i] = ids[i];
        ix->map.set(ids[i], (uint32_t)(row0 + i));
    }
    ix->n_live = row0 + n;
    ix->generation += 1;
    ix->mutations.fetch_add(1);
    return ORX_OK;
}

int orx_shard_export(orx_index *ix, int world, int rank, void *handle_out) {
    if (!ix || !handle_out) return fail(ORX_ERR_INVALID, "null argument");
    if (world < 1 || world > 64 || rank < 0 || rank >= world) return fail(ORX_ERR_INVALID, "bad world/rank %d/%d", rank, world);
    if (ix->group) return fail(ORX_ERR_INVALID, "a multi-GPU index is not a rank of a process group");
    std::lock_guard<std::mutex> lk(ix->mu);
    DeviceGuard g(ix->device);
    if (ix->xchg) return fail(ORX_ERR_INVALID, "shard exchange already initialised");
    Exchange *x = new Exchange();
    const size_t bytes = exchange_layout(x, world, rank);
    cudaError_t e = cudaMalloc(&x->base, bytes);
    if (e == cudaSuccess) e = cudaMemset(x->base, 0, bytes);
    cudaIpcMemHandle_t h;
    if (e == cudaSuccess) e = cudaIpcGetMemHandle(&h, x->base);
    if (e != cudaSuccess) {
        if (x->base) cudaFree(x->base);
        delete x;
        cudaGetLastError();
        return fail(ORX_ERR_CUDA, "shard exchange buffer: %s", cudaGetErrorString(e));
    }
    static_assert(sizeof(cudaIpcMemHandle_t) == ORX_IPC_HANDLE_BYTES, "IPC handle size");
    memcpy(handle_out, &h, sizeof h);
    ix->xchg = x;
    return ORX_OK;
}

int orx_shard_connect(orx_index *ix, const void *handles, int n_handles) {
    if (!ix || !handles) return fail(ORX_ERR_INVALID, "null argument");
    if (ix->group) return fail(ORX_ERR_INVALID, "a multi-GPU index is not a rank of a process group");
    std::lock_guard<std::mutex> lk(ix->mu);
    DeviceGuard g(ix->device);
    Exchange *x = ix->xchg;
    if (!x) return fail(ORX_ERR_INVALID, "call orx_shard_export first");
    if (x->connected) return fail(ORX_ERR_INVALID, "shard exchange already connected");
    if (n_handles != x->world) return fail(ORX_ERR_INVALID, "expected %d handles, got %d", x->world, n_handles);
    x->peer_base.assign(x->world, nullptr);
    for (int r = 0; r < x->world; ++r) {
        if (r == x->rank) {
            x->peer_base[r] = x->base;
            continue;
        }
        cudaIpcMemHandle_t h;
        memcpy(&h, static_cast<const char *>(handles) + (size_t)r * sizeof h, sizeof h);
        void *p = nullptr;
        cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) {
            cudaGetLastError();
            return fail(ORX_ERR_CUDA, "cannot map rank %d's exchange buffer (NVLink/P2P peer access): %s", r,
                        cudaGetErrorString(e));
        }
        x->peer_base[r] = static_cast<char *>(p);
    }
    CK(upload_peer_tables(x, x->peer_base));
    x->connected = true;
    return ORX_OK;
}

int orx_search_sharded(orx_index *ix, const float *queries, int nq, int dim, int k, orx_id *out_ids,
                       double *out_dist, int *out_counts) {
    int rc = check_query_args(ix, queries, nq, dim, k, out_ids, out_dist, out_counts);
    if (rc != ORX_OK || nq == 0) return rc;
    if (ix->group) return fail(ORX_ERR_INVALID, "a multi-GPU index is not a rank of a process group: use orx_search");
    std::lock_guard<std::mutex> lk(ix->mu);
    DeviceGuard g(ix->device);
    if (!ix->xchg || !ix->xchg->connected) return fail(ORX_ERR_INVALID, "shard exchange not connected (orx_shard_export / orx_shard_connect)");
    const int qchunk = exchange_queries(ix->xchg->world, k);
    if (!qchunk) return fail(ORX_ERR_INVALID, "sharded search: world * k must be <= 1024");
    for (int q0 = 0; q0 < nq; q0 += qchunk) {       // every rank chunks identically
        const int m = std::min(qchunk, nq - q0);
        rc = search_locked(ix, ix->xchg, queries + (size_t)q0 * ORX_DIM, m, k, out_ids + (size_t)q0 * k,
                           out_dist + (size_t)q0 * k, out_counts + q0);
        if (rc != ORX_OK) return rc;
    }
    return ORX_OK;
}

int orx_debug_coarse_scores(orx_index *ix, const float *queries, int nq, int use_pairs, float *out_device) {
    if (!ix || !queries || !out_device) return fail(ORX_ERR_INVALID, "null argument");
    if (ix->group) return fail(ORX_ERR_INVALID, "per-GPU diagnostic: call it on a single-GPU index");
    if (!is_device_ptr(out_device)) return fail(ORX_ERR_INVALID, "out must be device memory");
    std::lock_guard<std::mutex> lk(ix->mu);
    DeviceGuard g(ix->device);
    if (any_in_flight(ix)) return fail(ORX_ERR_INVALID, "wait for the searches in flight (orx_search_wait) first");
    if (!ix->cur->umma || ix->n_live == 0) return fail(ORX_ERR_INVALID, "empty table");
    const float *q_src = nullptr;
    int rc = stage_queries(ix, queries, nq, &q_src);
    if (rc != ORX_OK) return rc;
    rc = orx::umma_dump_scores(ix->cur->umma, ix->dtype, ix->table, ix->scale, (uint32_t)ix->n_live, ix->cur->qhat.p, ix->cur->qhat16.p, nq,
                               use_pairs != 0, out_device, ix->stream);
    if (rc != ORX_OK) return fail(rc, "tcgen05 dump failed: %s", orx::umma_last_error());
    ix->stats.kernel_launches += 2;
    CK(cudaStreamSynchronize(ix->stream));
    CK(cudaGetLastError());
    return ORX_OK;
}

int orx_debug_fast_scores(orx_index *ix, const float *queries, int nq, float *out_device) {
    if (!ix || !queries || !out_device) return fail(ORX_ERR_INVALID, "null argument");
    if (ix->group) return fail(ORX_ERR_INVALID, "per-GPU diagnostic: call it on a single-GPU index");
    if (!is_device_ptr(out_device)) return fail(ORX_ERR_INVALID, "out must be device memory");
    if (nq < 1 || nq > 65535) return fail(ORX_ERR_INVALID, "1 <= nq <= 65535, got %d", nq);
    std::lock_guard<std::mutex> lk(ix->mu);
    DeviceGuard g(ix->device);
    if (any_in_flight(ix)) return fail(ORX_ERR_INVALID, "wait for the searches in flight (orx_search_wait) first");
    if (ix->n_live == 0) return fail(ORX_ERR_INVALID, "empty table");
    const float *q_src = nullptr;
    int rc = stage_queries(ix, queries, nq, &q_src);
    if (rc != ORX_OK) return rc;
    orx::launch_dump_fast_scores(ix->dtype, ix->table, ix->scale, (uint32_t)ix->n_live, ix->cur->qhat.p, nq, out_device,
                                 ix->stream);
    ix->stats.kernel_launches += 1;
    CK(cudaStreamSynchronize(ix->stream));
    CK(cudaGetLastError());
    return ORX_OK;
}

// kind 1: the bf16 image's scores, 2: the 8-bit image's
int debug_image_scores(orx_index *ix, const float *queries, int nq, float *out_device, int kind) {
    if (!ix || !queries || !out_device) return fail(ORX_ERR_INVALID, "null argument");
    if (ix->group) return fail(ORX_ERR_INVALID, "per-GPU diagnostic: call it on a single-GPU index");
    if (!is_device_ptr(out_device)) return fail(ORX_ERR_INVALID, "out must be device memory");
    if (nq < 1 || nq > 65535) return fail(ORX_ERR_INVALID, "1 <= nq <= 65535, got %d", nq);
    std::lock_guard<std::mutex> lk(ix->mu);
    DeviceGuard g(ix->device);
    if (any_in_flight(ix)) return fail(ORX_ERR_INVALID, "wait for the searches in flight (orx_search_wait) first");
    if (ix->n_live == 0) return fail(ORX_ERR_INVALID, "empty table");
    ensure_image(ix, kind);
    if (image_kind(ix) != kind)
        return fail(ORX_ERR_INVALID, "this index has no %s image (bf16 table, an image of the other kind, or no device "
                    "memory for it)", kind == 1 ? "bf16" : "8-bit");
    const float *q_src = nullptr;
    int rc = stage_queries(ix, queries, nq, &q_src);
    if (rc != ORX_OK) return rc;
    if (kind == 1)
        orx::launch_dump_fast_scores(ORX_DTYPE_BF16, ix->image, ix->scale, (uint32_t)ix->n_live, ix->cur->qhat.p, nq,
                                     out_device, ix->stream);
    else
        orx::launch_dump_image8_scores(ix->image8.rows, ix->image8.scale8, (uint32_t)ix->n_live, ix->cur->qhat8.p,
                                       ix->cur->prep.p, nq, out_device, ix->stream);
    ix->stats.kernel_launches += 1;
    CK(cudaStreamSynchronize(ix->stream));
    CK(cudaGetLastError());
    return ORX_OK;
}
int orx_debug_image_scores(orx_index *ix, const float *queries, int nq, float *out_device) {
    return debug_image_scores(ix, queries, nq, out_device, 1);
}
int orx_debug_image8_scores(orx_index *ix, const float *queries, int nq, float *out_device) {
    return debug_image_scores(ix, queries, nq, out_device, 2);
}

int orx_fetch(orx_index *ix, const orx_id *ids, uint64_t n, float *out_vecs, int *out_found) {
    if (!ix) return fail(ORX_ERR_INVALID, "index is null");
    if (n == 0) return ORX_OK;
    if (!ids || !out_vecs || !out_found) return fail(ORX_ERR_INVALID, "null argument");
    if (ix->group) return group_fetch(ix->group, ids, n, out_vecs, out_found);
    std::lock_guard<std::mutex> lk(ix->mu);
    DeviceGuard g(ix->device);
    cudaStream_t st = ix->stream;
    const uint64_t chunk = std::min<uint64_t>(n, STAGE_ROWS);
    CK(ix->stage.ensure(chunk * ORX_DIM));
    CK(ix->d_src_idx.ensure(chunk));
    CK(ix->h_u32a.ensure(chunk));
    for (uint64_t s = 0; s < n; s += chunk) {
        const uint64_t m = std::min(chunk, n - s);
        for (uint64_t i = 0; i < m; ++i) {
            const uint32_t *r = ix->map.find(ids[s + i]);
            out_found[s + i] = r != nullptr;
            ix->h_u32a.p[i] = r ? *r : 0xFFFFFFFFu;
        }
        CK(cudaMemcpyAsync(ix->d_src_idx.p, ix->h_u32a.p, m * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
        orx::launch_gather_rows(ix->dtype, ix->table, ix->d_src_idx.p, (uint32_t)m, ix->stage.p, st);
        ix->stats.kernel_launches += 1;
        CK(cudaMemcpyAsync(out_vecs + s * ORX_DIM, ix->stage.p, m * ORX_DIM * sizeof(float), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
    }
    CK(cudaGetLastError());
    return ORX_OK;
}

}  // extern "C"
