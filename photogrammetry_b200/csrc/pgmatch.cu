// pgmatch.cu -- C ABI (include/pgmatch.h) and host-side engine of libpgmatch.so.
//
// Replaces ImageProcessing.KeypointMatching.MatchKeypoints
// (dotnet_src/ImageProcessing/KeypointMatching.cs:14-69) behind a P/Invoke-able
// boundary.  There is deliberately no CPU implementation in this file: if no
// sm_100 device is usable every entry point fails with PGM_E_NO_DEVICE.
#include "../../include/pgmatch.h"
#include "pgm_kernels.cuh"
#include "pgm_l2.cuh"
#include "pgm_detect.cuh"
#include "pgm_ransac.cuh"

#include <cub/device/device_radix_sort.cuh>

#include <algorithm>
#include <chrono>
#include <cstddef>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

using namespace pgm;

// ---------------------------------------------------------------------------
// handle
// ---------------------------------------------------------------------------
struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
};
struct HostBuf {
    void *p = nullptr;
    size_t cap = 0;
};

struct pgm_handle {
    int device = 0;
    int num_sms = 0;
    cudaStream_t own_stream = nullptr;
    cudaStream_t stream = nullptr;
    std::mutex mu;
    std::string err;
    DevBuf state;     // per-chunk matcher state (carved by carve())
    DevBuf desc;      // descriptors uploaded by the host-buffer entry points
    DevBuf out;       // device staging of outputs for the host-buffer entry points
    DevBuf out2;      // second output buffer: the batch entry point overlaps D2H of chunk k with chunk k+1
    HostBuf pin_out2;
    cudaStream_t copy_stream = nullptr;            // D2H of finished chunks (batch entry point)
    cudaEvent_t ev_done[2] = {nullptr, nullptr};   // chunk's kernels finished (main stream)
    cudaEvent_t ev_copied[2] = {nullptr, nullptr}; // chunk's triples sit in pinned memory (copy stream)
    DevBuf misc;      // knn2 partials etc.
    DevBuf shard_pool_state, shard_pool_est;   // a destroyed pgm_shard parks its device buffers here: the next one reuses them
    void *shard_pool_hctl = nullptr;           // (cudaMalloc / cudaMallocHost / cudaFree cost ~1.5 ms per train-sharded call)
    DevBuf l2_state;  // float path, fp16 ranking: [max |x| bits, flagged rows, fallback ticket, batch call's flagged rows];
                      // zeroed on allocation, words 0-2 self-cleaning
    HostBuf pin_in;   // pinned staging, host -> device
    HostBuf pin_out;  // pinned staging, device -> host
    HostBuf pin_meta; // pinned PairDesc array + PlanInfo readback
    pgm_stats stats{};
    int rounds_hint = 4;      // grid rounds to enqueue before the first completion check
    int ctas_per_sm[5] = {0, 0, 0, 0, 0};   // round-kernel occupancy per descriptor width (words / 4)
    bool order_attr_set = false;
    bool tail_attr_set[5] = {false, false, false, false, false};
    bool l2_attr_set = false;         // cudaFuncSetAttribute is per device, hence per handle
    int l2_max_clusters = 1;          // co-resident CTA pairs of the float pair kernel (persistent grid)
    unsigned *l2_hdr = nullptr;       // fp16 ranking mode of the last float call: [max |x| bits, rows recomputed exhaustively]
    int l2_fallback_word = 1;         // the word of l2_hdr that counts them: 1 (one pair), 3 (the batch entry points' call total)
    DevBuf lat_state;             // LatState of latency mode (pgm_kernels.cuh): zeroed before its first use, left clean by every call
    bool lat_dirty = false;       // a latency-mode call was cut short between its launches: zero lat_state before the next
    bool stats_pending = false;   // rounds / evals of the last latency-mode call still sit in lat_state (device) ...
    bool stats_copied = false;    // ... or, once a read-back has been enqueued, in the pinned slot pending_plan points at
    void *pending_plan = nullptr;
    bool tail_timeline = false;      // PGM_TAIL_TIMELINE=1: dump the tail kernel's phase timeline to stderr (debug)
    DevBuf timeline;
    bool fin_attr_set[5] = {false, false, false, false, false};
    bool sparse_attr_set = false;
    // profiling mode (pgm_set_profiling): events around every round-kernel launch
    bool profiling = false;
    std::vector<cudaEvent_t> prof_events;   // 2 per round
    HostBuf pin_prof;                       // PlanInfo snapshot per round
    int prof_rounds = 0;
};
constexpr int PROF_MAX_ROUNDS = 256;
constexpr int LATENCY_MODE_MAX_PAIRS = PACK_PAIRS;

#define CU_CHECK(h, call)                                                                      \
    do {                                                                                       \
        cudaError_t e__ = (call);                                                              \
        if (e__ != cudaSuccess) {                                                              \
            char b__[512];                                                                     \
            snprintf(b__, sizeof b__, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), \
                     __FILE__, __LINE__);                                                      \
            (h)->err = b__;                                                                    \
            return PGM_E_CUDA;                                                                 \
        }                                                                                      \
    } while (0)

static int fail(pgm_handle *h, int code, const char *msg) {
    if (h) h->err = msg;
    return code;
}

static int ensure_dev(pgm_handle *h, DevBuf &b, size_t bytes) {
    if (bytes <= b.cap) return PGM_OK;
    size_t want = std::max(bytes, b.cap + b.cap / 2);
    want = (want + 255) & ~(size_t)255;
    if (b.p) {
        CU_CHECK(h, cudaStreamSynchronize(h->stream));
        CU_CHECK(h, cudaFree(b.p));
        b.p = nullptr; b.cap = 0;
    }
    cudaError_t e = cudaMalloc(&b.p, want);
    if (e != cudaSuccess) {
        h->err = std::string("cudaMalloc failed: ") + cudaGetErrorString(e);
        b.p = nullptr;
        return e == cudaErrorMemoryAllocation ? PGM_E_NOMEM : PGM_E_CUDA;
    }
    b.cap = want;
    return PGM_OK;
}

static int ensure_host(pgm_handle *h, HostBuf &b, size_t bytes) {
    if (bytes <= b.cap) return PGM_OK;
    size_t want = std::max(bytes, b.cap + b.cap / 2);
    if (b.p) {
        CU_CHECK(h, cudaStreamSynchronize(h->stream));
        CU_CHECK(h, cudaFreeHost(b.p));
        b.p = nullptr; b.cap = 0;
    }
    CU_CHECK(h, cudaMallocHost(&b.p, want));
    b.cap = want;
    return PGM_OK;
}

static void resolve_pending_stats(pgm_handle *h);
static void enqueue_stats_readback(pgm_handle *h);

// Page-locked host memory (cudaHostAlloc / cudaHostRegister) can be the source or target of an asynchronous
// copy directly; pageable memory is staged through the handle's pinned buffers.
static bool is_pinned_host(const void *p) {
    if (!p) return false;
    cudaPointerAttributes a{};
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost;
}

extern "C" int pgm_host_alloc(size_t bytes, void **out) {
    if (!out) return PGM_E_INVALID_ARG;
    *out = nullptr;
    if (bytes == 0) return PGM_OK;
    cudaError_t e = cudaHostAlloc(out, bytes, cudaHostAllocPortable);
    if (e != cudaSuccess) { cudaGetLastError(); *out = nullptr; return e == cudaErrorMemoryAllocation ? PGM_E_NOMEM : PGM_E_CUDA; }
    return PGM_OK;
}

extern "C" int pgm_host_free(void *p) {
    if (!p) return PGM_OK;
    return cudaFreeHost(p) == cudaSuccess ? PGM_OK : PGM_E_CUDA;
}

extern "C" int pgm_version(void) { return PGM_VERSION; }

extern "C" const char *pgm_status_string(int s) {
    switch (s) {
        case PGM_OK: return "ok";
        case PGM_E_INVALID_ARG: return "invalid argument";
        case PGM_E_CAPACITY: return "output capacity too small";
        case PGM_E_CUDA: return "CUDA error";
        case PGM_E_NCCL: return "NCCL error";
        case PGM_E_EMPTY_TRAIN: return "train set is empty (reference throws ArgumentOutOfRangeException)";
        case PGM_E_NOMEM: return "out of memory";
        case PGM_E_NO_DEVICE: return "no usable sm_100 CUDA device (there is no CPU fallback)";
        default: return "unknown status";
    }
}

extern "C" int pgm_create(int device_ordinal, pgm_handle **out) {
    if (!out) return PGM_E_INVALID_ARG;
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0 || device_ordinal < 0 || device_ordinal >= count) {
        cudaGetLastError();
        return PGM_E_NO_DEVICE;
    }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device_ordinal) != cudaSuccess) return PGM_E_NO_DEVICE;
    if (prop.major != 10) return PGM_E_NO_DEVICE;   // the .so carries sm_100a SASS only
    if (cudaSetDevice(device_ordinal) != cudaSuccess) return PGM_E_NO_DEVICE;
    pgm_handle *h = new pgm_handle();
    h->device = device_ordinal;
    h->num_sms = prop.multiProcessorCount;
    if (cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking) != cudaSuccess) {
        delete h;
        return PGM_E_CUDA;
    }
    h->stream = h->own_stream;
    const char *tl = getenv("PGM_TAIL_TIMELINE");
    h->tail_timeline = tl && tl[0] == '1';
    *out = h;
    return PGM_OK;
}

extern "C" int pgm_destroy(pgm_handle *h) {
    if (!h) return PGM_E_INVALID_ARG;
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->stream);
    if (h->copy_stream) { cudaStreamSynchronize(h->copy_stream); cudaStreamDestroy(h->copy_stream); }
    for (cudaEvent_t e : {h->ev_done[0], h->ev_done[1], h->ev_copied[0], h->ev_copied[1]})
        if (e) cudaEventDestroy(e);
    if (h->shard_pool_hctl) cudaFreeHost(h->shard_pool_hctl);
    for (DevBuf *b : {&h->state, &h->desc, &h->out, &h->out2, &h->misc, &h->l2_state, &h->lat_state, &h->shard_pool_state, &h->shard_pool_est})
        if (b->p) cudaFree(b->p);
    for (HostBuf *b : {&h->pin_in, &h->pin_out, &h->pin_out2, &h->pin_meta, &h->pin_prof})
        if (b->p) cudaFreeHost(b->p);
    for (cudaEvent_t e : h->prof_events) cudaEventDestroy(e);
    if (h->own_stream) cudaStreamDestroy(h->own_stream);
    delete h;
    return PGM_OK;
}

extern "C" const char *pgm_last_error(pgm_handle *h) { return h ? h->err.c_str() : "null handle"; }

extern "C" int pgm_set_stream(pgm_handle *h, void *cuda_stream) {
    if (!h) return PGM_E_INVALID_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    h->stream = cuda_stream ? (cudaStream_t)cuda_stream : h->own_stream;
    return PGM_OK;
}

extern "C" int pgm_synchronize(pgm_handle *h) {
    if (!h) return PGM_E_INVALID_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    CU_CHECK(h, cudaSetDevice(h->device));
    CU_CHECK(h, cudaStreamSynchronize(h->stream));
    return PGM_OK;
}

extern "C" int pgm_get_stats(pgm_handle *h, pgm_stats *out) {
    if (!h || !out) return PGM_E_INVALID_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    if (h->stats_pending) {
        CU_CHECK(h, cudaSetDevice(h->device));
        CU_CHECK(h, cudaStreamSynchronize(h->stream));
        resolve_pending_stats(h);
    }
    *out = h->stats;
    return PGM_OK;
}

// ---------------------------------------------------------------------------
// kernel dispatch on descriptor width
// ---------------------------------------------------------------------------
constexpr int RQ_DEFAULT = RQ_LARGE;

template <int WORDS>
static void launch_round(const Chunk &c, int r, int grid, cudaStream_t s) {
    hamming_round_kernel<WORDS><<<grid, ROUND_THREADS, 0, s>>>(c, r);
}
static void dispatch_round(int words, const Chunk &c, int r, int grid, cudaStream_t s) {
    switch (words) {
        case 4: launch_round<4>(c, r, grid, s); break;
        case 8: launch_round<8>(c, r, grid, s); break;
        case 12: launch_round<12>(c, r, grid, s); break;
        default: launch_round<16>(c, r, grid, s); break;
    }
}
template <int WORDS>
static cudaError_t launch_fin(pgm_handle *h, const Chunk &c, cudaStream_t s) {
    const size_t smem = finisher_smem_bytes(WORDS);
    if (!h->fin_attr_set[WORDS / 4]) {
        cudaError_t e = cudaFuncSetAttribute(finisher_kernel<WORDS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        h->fin_attr_set[WORDS / 4] = true;
    }
    finisher_kernel<WORDS><<<c.n_pairs, FIN_THREADS, smem, s>>>(c);
    return cudaSuccess;
}
static cudaError_t dispatch_fin(pgm_handle *h, int words, const Chunk &c, cudaStream_t s) {
    switch (words) {
        case 4: return launch_fin<4>(h, c, s);
        case 8: return launch_fin<8>(h, c, s);
        case 12: return launch_fin<12>(h, c, s);
        default: return launch_fin<16>(h, c, s);
    }
}
template <int WORDS>
static cudaError_t launch_tail(pgm_handle *h, Chunk c, int r_start, int nbins, uint32_t flags, int32_t *oq, int32_t *ot,
                               int32_t *od, cudaStream_t s) {
    const size_t smem = tail_smem_bytes<WORDS>(513);
    if (!h->tail_attr_set[WORDS / 4]) {
        cudaError_t e = cudaFuncSetAttribute(tail_kernel<WORDS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        h->tail_attr_set[WORDS / 4] = true;
    }
    void *args[] = {&c, &r_start, &nbins, &flags, &oq, &ot, &od};
    return cudaLaunchCooperativeKernel((void *)tail_kernel<WORDS>, dim3(h->num_sms), dim3(TAIL_THREADS), args, smem, s);
}
static cudaError_t dispatch_tail(pgm_handle *h, int words, const Chunk &c, int r_start, int nbins, uint32_t flags,
                                 int32_t *oq, int32_t *ot, int32_t *od, cudaStream_t s) {
    switch (words) {
        case 4: return launch_tail<4>(h, c, r_start, nbins, flags, oq, ot, od, s);
        case 8: return launch_tail<8>(h, c, r_start, nbins, flags, oq, ot, od, s);
        case 12: return launch_tail<12>(h, c, r_start, nbins, flags, oq, ot, od, s);
        default: return launch_tail<16>(h, c, r_start, nbins, flags, oq, ot, od, s);
    }
}
template <int WORDS>
static int round_occupancy() {
    int nb = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, hamming_round_kernel<WORDS>, ROUND_THREADS, 0);
    return nb;
}
static int dispatch_occupancy(int words) {
    switch (words) {
        case 4: return round_occupancy<4>();
        case 8: return round_occupancy<8>();
        case 12: return round_occupancy<12>();
        default: return round_occupancy<16>();
    }
}
template <int WORDS>
static void launch_knn2(const uint32_t *q, int n1, const uint32_t *t, int n2, int cps, int splits, uint32_t *part,
                        cudaStream_t s) {
    const int tile_rows = ROUND_THREADS * RQ_DEFAULT;
    dim3 grid((n1 + tile_rows - 1) / tile_rows, splits);
    knn2_kernel<WORDS, RQ_DEFAULT><<<grid, ROUND_THREADS, 0, s>>>(q, n1, t, n2, cps, part);
}
static void dispatch_knn2(int words, const uint32_t *q, int n1, const uint32_t *t, int n2, int cps, int splits,
                          uint32_t *part, cudaStream_t s) {
    switch (words) {
        case 4: launch_knn2<4>(q, n1, t, n2, cps, splits, part, s); break;
        case 8: launch_knn2<8>(q, n1, t, n2, cps, splits, part, s); break;
        case 12: launch_knn2<12>(q, n1, t, n2, cps, splits, part, s); break;
        default: launch_knn2<16>(q, n1, t, n2, cps, splits, part, s); break;
    }
}

// ---------------------------------------------------------------------------
// argument checks shared by every entry point
// ---------------------------------------------------------------------------
static int check_format(pgm_handle *h, int32_t desc_bits, int32_t stride_bytes) {
    if (desc_bits < 1 || desc_bits > 512) return fail(h, PGM_E_INVALID_ARG, "desc_bits must be in 1..512");
    if (stride_bytes < 16 || stride_bytes > 64 || stride_bytes % 16 != 0)
        return fail(h, PGM_E_INVALID_ARG, "stride_bytes must be 16, 32, 48 or 64");
    if (8 * stride_bytes < desc_bits) return fail(h, PGM_E_INVALID_ARG, "stride_bytes too small for desc_bits");
    return PGM_OK;
}

// ---------------------------------------------------------------------------
// the engine: greedy assignment of one chunk of pairs, everything on device
// ---------------------------------------------------------------------------
struct HostPair {
    const uint8_t *d_q, *d_t;   // device pointers
    int32_t n1, n2;
    int64_t out_base;           // in rows, relative to the chunk's output arrays
};

static size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// Rounds with at least this many live cells use the large (512-row, RQ = 4) tiles: two such tiles per SM.
static long long large_tile_min_evals(const pgm_handle *h) {
    return 2ll * h->num_sms * ROUND_THREADS * RQ_LARGE * STAGE_LARGE;
}

static int run_chunk(pgm_handle *h, const HostPair *pairs, int n_pairs, int desc_bits, int stride_bytes,
                     uint32_t flags, int32_t *d_out_qi, int32_t *d_out_tj, int32_t *d_out_dist) {
    const int words = stride_bytes / 4;
    cudaStream_t s = h->stream;

    int64_t rows = 0, cols = 0;
    int max_n = 1;
    for (int p = 0; p < n_pairs; p++) {
        rows += pairs[p].n1; cols += pairs[p].n2;
        max_n = std::max(max_n, std::max(pairs[p].n1, pairs[p].n2));
    }
    // carve the state arena
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return o; };
    const size_t o_pairs = take(sizeof(PairDesc) * n_pairs);
    const size_t o_rb0 = take(4 * rows), o_rb1 = take(4 * rows), o_cb0 = take(4 * cols), o_cb1 = take(4 * cols);
    const size_t o_lr0 = take(4 * rows), o_lr1 = take(4 * rows), o_lc0 = take(4 * cols), o_lc1 = take(4 * cols);
    const size_t o_cnt = take(sizeof(int32_t) * 6 * n_pairs);
    const size_t o_mk = take(4 * rows);
    const size_t o_tb = take(4 * (n_pairs + 1)), o_ab = take(4 * (n_pairs + 1));
    const size_t o_st = take(n_pairs);
    const size_t o_small = take(sizeof(SmallInfo) * n_pairs);
    const size_t o_plan = take(sizeof(PlanInfo));
    const bool latency_mode = n_pairs <= LATENCY_MODE_MAX_PAIRS;
    // latency mode: global scratch for the finisher's matrices / first-round minima (finisher_prepare)
    const size_t o_find = latency_mode ? take((size_t)n_pairs * FIN_D_STRIDE * 2) : 0;
    const size_t o_finr = latency_mode ? take((size_t)n_pairs * FIN_PARTS * FIN_MAX_DIM * 4) : 0;
    const size_t o_finc = latency_mode ? take((size_t)n_pairs * FIN_PARTS * FIN_MAX_DIM * 4) : 0;
    const size_t o_fini = latency_mode ? take((size_t)n_pairs * 2 * FIN_MAX_DIM * 4) : 0;
    const size_t o_ocnt = latency_mode ? take((size_t)n_pairs * ORDER_MAX_SLICES * ORDER_BIN_PITCH * 4) : 0;
    // candidate edges (pgm_kernels.cuh): per pair a raw list of about 2 x CAND_TARGET entries per row and a list of the
    // edges that survive the accept, sized for the sparse phase's shared memory
    // a few pairs (latency mode): the single-CTA sparse phase is on the critical path, keep its edge list short; batches:
    // the sparse phases of different pairs run side by side, a longer list saves more recomputation than it costs
    const float cand_target = n_pairs <= LATENCY_MODE_MAX_PAIRS ? CAND_TARGET : CAND_TARGET_BATCH;
    std::vector<int64_t> cand_off(n_pairs + 1, 0), ledge_off(n_pairs + 1, 0);
    for (int p = 0; p < n_pairs; p++) {
        const int64_t cells = (int64_t)pairs[p].n1 * pairs[p].n2;
        const int64_t cap = std::min<int64_t>(cells, (int64_t)(2.0f * cand_target + 1.0f) * std::max(pairs[p].n1, pairs[p].n2) + 1024);
        cand_off[p + 1] = cand_off[p] + cap;
        ledge_off[p + 1] = ledge_off[p] + std::min<int64_t>(cap, SP_LCAP_MAX);
    }
    const size_t o_cand = take(16 * (size_t)cand_off[n_pairs]);   // two words per record
    const size_t o_ledge = take(8 * (size_t)ledge_off[n_pairs]);
    const size_t o_ccnt = take(4 * (size_t)n_pairs), o_lcnt = take(4 * (size_t)n_pairs);
    const size_t o_thr = take(4 * (size_t)n_pairs), o_pstat = take(sizeof(PairStat) * (size_t)n_pairs);
    const size_t o_rpos = take(4 * rows), o_cpos = take(4 * cols);
    int rc = ensure_dev(h, h->state, off);
    if (rc) return rc;
    rc = ensure_host(h, h->pin_meta, sizeof(PairDesc) * n_pairs + 512);
    if (rc) return rc;
    char *base = (char *)h->state.p;

    if (h->ctas_per_sm[words / 4] == 0) h->ctas_per_sm[words / 4] = std::max(1, dispatch_occupancy(words));
    const int ctas_per_sm = h->ctas_per_sm[words / 4];
    const int round_grid = h->num_sms * ctas_per_sm;

    Chunk c{};
    c.pairs = (PairDesc *)(base + o_pairs);
    c.n_pairs = n_pairs;
    c.num_sms = h->num_sms;
    c.ctas_per_sm = latency_mode ? TAIL_THREADS / ROUND_THREADS : ctas_per_sm;
    c.ctas_per_sm0 = latency_mode ? ctas_per_sm : 0;    // round 0 of latency mode is a standalone launch at full occupancy
    c.fin_max_evals = latency_mode ? FIN_MAX_EVALS_TAIL : FIN_MAX_EVALS;
    c.large_min_evals = large_tile_min_evals(h);
    if (latency_mode) {
        c.fin_d = (uint16_t *)(base + o_find);
        c.fin_rb = (uint32_t *)(base + o_finr);
        c.fin_cb = (uint32_t *)(base + o_finc);
        c.fin_ids = (int32_t *)(base + o_fini);
        c.order_cnt = (int32_t *)(base + o_ocnt);
    }
    c.rowbest[0] = (uint32_t *)(base + o_rb0); c.rowbest[1] = (uint32_t *)(base + o_rb1);
    c.colbest[0] = (uint32_t *)(base + o_cb0); c.colbest[1] = (uint32_t *)(base + o_cb1);
    c.live_rows[0] = (int32_t *)(base + o_lr0); c.live_rows[1] = (int32_t *)(base + o_lr1);
    c.live_cols[0] = (int32_t *)(base + o_lc0); c.live_cols[1] = (int32_t *)(base + o_lc1);
    c.counts = (int32_t *)(base + o_cnt);
    c.match_key = (uint32_t *)(base + o_mk);
    c.tile_base = (int32_t *)(base + o_tb);
    c.ablock_base = (int32_t *)(base + o_ab);
    c.status = (uint8_t *)(base + o_st);
    c.small = (SmallInfo *)(base + o_small);
    c.plan = (PlanInfo *)(base + o_plan);
    c.lat = nullptr;
    if (latency_mode) {           // the plan lives in the handle's self-cleaning block: no memset, no read-back per call
        if (!h->lat_state.p) {
            if ((rc = ensure_dev(h, h->lat_state, sizeof(LatState)))) return rc;
            h->lat_dirty = true;
        }
        c.lat = (LatState *)h->lat_state.p;
        c.plan = &c.lat->plan;
    }
    c.words = words;
    c.cand_target = cand_target;
    c.sp_slots_max = SP_EPT;
    if (const char *e = getenv("PGM_SP_SLOTS_MAX")) c.sp_slots_max = std::min(SP_EPT, std::max(1, atoi(e)));   // tests: force the truncation path
    // a few pairs: later passes list at most 16 candidates per row (the sparse phase of a pass runs on ONE SM and sits on
    // the call's critical path; measured best at 4096^2 ... 16384^2); batches: the list budget alone decides
    c.cand_row_max = latency_mode ? 16.0f : 1e9f;
    c.cand = (unsigned long long *)(base + o_cand); c.ledge = (unsigned long long *)(base + o_ledge);
    c.cand_cnt = (int32_t *)(base + o_ccnt); c.ledge_cnt = (int32_t *)(base + o_lcnt);
    c.thr = (uint32_t *)(base + o_thr); c.pstat = (PairStat *)(base + o_pstat);
    c.row_pos = (int32_t *)(base + o_rpos); c.col_pos = (int32_t *)(base + o_cpos);
    c.timeline = nullptr;
    if (h->tail_timeline) {
        if ((rc = ensure_dev(h, h->timeline, 1000 * 8))) return rc;
        CU_CHECK(h, cudaMemsetAsync(h->timeline.p, 0, 1000 * 8, s));
        c.timeline = (unsigned long long *)h->timeline.p;
    }

    PairDesc *hp = (PairDesc *)h->pin_meta.p;
    char *meta_tail = (char *)h->pin_meta.p + align_up(sizeof(PairDesc) * n_pairs, 64);
    PlanInfo *h_plan = (PlanInfo *)meta_tail;             // readback slot
    int64_t rb = 0, cb = 0, ablocks = 0;
    for (int p = 0; p < n_pairs; p++) {
        hp[p].q = (const uint32_t *)pairs[p].d_q;
        hp[p].t = (const uint32_t *)pairs[p].d_t;
        hp[p].n1 = pairs[p].n1; hp[p].n2 = pairs[p].n2;
        hp[p].row_base = rb; hp[p].col_base = cb; hp[p].out_base = pairs[p].out_base;
        hp[p].col_id_offset = 0; hp[p].flags = 0;
        hp[p].cand_off = cand_off[p]; hp[p].ledge_off = ledge_off[p];
        hp[p].cand_cap = (int32_t)(cand_off[p + 1] - cand_off[p]); hp[p].ledge_cap = (int32_t)(ledge_off[p + 1] - ledge_off[p]);
        rb += pairs[p].n1; cb += pairs[p].n2;
        ablocks += (pairs[p].n1 + ACCEPT_THREADS - 1) / ACCEPT_THREADS + (pairs[p].n2 + ACCEPT_THREADS - 1) / ACCEPT_THREADS;
        h->stats.distance_evals += (int64_t)pairs[p].n1 * pairs[p].n2;
        h->stats.matched += std::min(pairs[p].n1, pairs[p].n2);
    }
    h->stats.pairs += n_pairs;
    // live sets only shrink, so the initial block count bounds every later accept launch
    const int accept_grid = (int)std::max<int64_t>(1, std::min<int64_t>(ablocks, (int64_t)h->num_sms * 8));
    // PGM_LAT_SPLIT=1 (debug): events between the launches of a latency-mode call, printed after a synchronisation
    static const bool lat_split_env = getenv("PGM_LAT_SPLIT") != nullptr;
    const bool lat_split = lat_split_env && latency_mode;
    cudaEvent_t sev[4] = {};
    if (lat_split) { for (auto &e : sev) cudaEventCreate(&e); cudaEventRecord(sev[0], s); }
    if (!latency_mode) CU_CHECK(h, cudaMemsetAsync(c.plan, 0, sizeof(PlanInfo), s));
    else if (h->lat_dirty) CU_CHECK(h, cudaMemsetAsync(c.lat, 0, sizeof(LatState), s));
    if (latency_mode) h->lat_dirty = true;      // until the tail kernel is enqueued
    dim3 igrid(std::max(1, std::min((max_n + ACCEPT_THREADS - 1) / ACCEPT_THREADS, 64)), n_pairs);
    if (latency_mode) {
        PairPack pack{};
        for (int p = 0; p < n_pairs; p++) pack.p[p] = hp[p];
        init_kernel<true><<<igrid, ACCEPT_THREADS, 0, s>>>(c, pack);     // also plans round 0 in its last block
    } else {
        CU_CHECK(h, cudaMemcpyAsync(c.pairs, hp, sizeof(PairDesc) * n_pairs, cudaMemcpyHostToDevice, s));
        init_kernel<false><<<igrid, ACCEPT_THREADS, 0, s>>>(c, PairPack{});
    }
    h->stats.kernel_launches += 1;

    // Histogram bins of the ordering pass.  Sized by the padded row width, not by desc_bits: nothing checks that the
    // caller zeroed the bits at positions >= desc_bits, and a distance above desc_bits must not leave its histogram.
    (void)desc_bits;
    const int nbins = 8 * stride_bytes + 1;
    const bool prof = h->profiling;
    // ---- latency mode: a few pairs.  init, one full round, then the persistent tail kernel runs
    // every remaining round, the finisher and the ordering without coming back to the host.
    if (latency_mode) {
        bool any_big = false;
        for (int p = 0; p < n_pairs; p++) {
            const int64_t a = pairs[p].n1, b = pairs[p].n2;
            if (a > 0 && b > 0 && !(a <= FIN_MAX_DIM && b <= FIN_MAX_DIM && a * b <= FIN_MAX_EVALS_TAIL)) any_big = true;
        }
        int r_start = 0;
        h->prof_rounds = 0;
        if (any_big) {
            PlanInfo *pp = (PlanInfo *)h->pin_prof.p;
            if (prof) {   // events around the one standalone launch of the dominant kernel
                CU_CHECK(h, cudaMemcpyAsync(&pp[0], c.plan, sizeof(PlanInfo), cudaMemcpyDeviceToHost, s));
                CU_CHECK(h, cudaEventRecord(h->prof_events[0], s));
            }
            if (lat_split) cudaEventRecord(sev[1], s);
            dispatch_round(words, c, 0, round_grid, s);
            if (lat_split) cudaEventRecord(sev[2], s);
            if (prof) CU_CHECK(h, cudaEventRecord(h->prof_events[1], s));
            if (prof) h->prof_rounds = 1;
            h->stats.kernel_launches += 1;
            r_start = 1;                  // the tail kernel begins with round 0's accept phase
        }
        CU_CHECK(h, dispatch_tail(h, words, c, r_start, nbins, (flags & ~TAIL_FLAG_ACCEPT_FIRST) | (any_big ? TAIL_FLAG_ACCEPT_FIRST : 0u), d_out_qi,
                                  d_out_tj, d_out_dist, s));
        h->stats.kernel_launches += 1;
        h->lat_dirty = false;
        if (lat_split) {
            cudaEventRecord(sev[3], s);
            cudaStreamSynchronize(s);
            float d[3] = {};
            for (int k = 0; k < 3; k++) cudaEventElapsedTime(&d[k], sev[k], sev[k + 1]);
            fprintf(stderr, "[pgm lat split, us] init %.1f  round0 %.1f  tail %.1f\n", d[0] * 1e3, d[1] * 1e3, d[2] * 1e3);
            for (auto &e : sev) cudaEventDestroy(e);
        }
        h->stats_pending = true;          // resolved by pgm_get_stats / the host-buffer entry points (with their own read-back)
        h->stats_copied = false;
        h->pending_plan = h_plan;
        CU_CHECK(h, cudaGetLastError());
        if (h->tail_timeline) {
            std::vector<unsigned long long> tl(1000);
            CU_CHECK(h, cudaMemcpyAsync(tl.data(), h->timeline.p, 1000 * 8, cudaMemcpyDeviceToHost, s));
            CU_CHECK(h, cudaStreamSynchronize(s));
            fprintf(stderr, "[pgm tail timeline, us since kernel start]");
            for (int k = 1; k < 1000 && tl[k]; k++) fprintf(stderr, " %.1f", (tl[k] - tl[0]) * 1e-3);
            fprintf(stderr, "\n[tile stamps code:us]");
            for (int k = 500; k < 980 && tl[k]; k++) fprintf(stderr, " %d:%.1f", (int)(tl[k] & 0xFF), (double)(((tl[k] >> 8) - (tl[0] & 0x00FFFFFFFFFFFFFFull)) & 0xFFFFFFFFFFull) * 1e-3);
            fprintf(stderr, "\n");
        }
        return PGM_OK;
    }

    PlanInfo *prof_plan = (PlanInfo *)h->pin_prof.p;
    h->prof_rounds = 0;
    if (prof) CU_CHECK(h, cudaMemcpyAsync(&prof_plan[0], c.plan, sizeof(PlanInfo), cudaMemcpyDeviceToHost, s));
    int r = 0;
    int batch = std::max(0, h->rounds_hint);
    for (;;) {
        for (int k = 0; k < batch; k++, r++) {
            const bool pr = prof && r < PROF_MAX_ROUNDS;
            if (pr) CU_CHECK(h, cudaEventRecord(h->prof_events[2 * r], s));
            dispatch_round(words, c, r, round_grid, s);
            if (pr) CU_CHECK(h, cudaEventRecord(h->prof_events[2 * r + 1], s));
            accept_kernel<<<accept_grid, ACCEPT_THREADS, 0, s>>>(c, r);        // + candidate-edge filter
            if (!h->sparse_attr_set) {                                          // sparse sub-rounds, then the plan of r + 1
                CU_CHECK(h, cudaFuncSetAttribute(sparse_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SP_SMEM_BYTES));
                h->sparse_attr_set = true;
            }
            sparse_kernel<<<std::min(n_pairs, h->num_sms * 4), SP_THREADS, SP_SMEM_BYTES, s>>>(c, r);
            if (pr) {
                CU_CHECK(h, cudaMemcpyAsync(&prof_plan[r + 1], c.plan, sizeof(PlanInfo), cudaMemcpyDeviceToHost, s));
                h->prof_rounds = r + 1;
            }
            h->stats.kernel_launches += 3;
        }
        // pairs that became small wait in place (SmallInfo) until this launch
        CU_CHECK(h, dispatch_fin(h, words, c, s));
        h->stats.kernel_launches += 1;
        CU_CHECK(h, cudaMemcpyAsync(h_plan, c.plan, sizeof(PlanInfo), cudaMemcpyDeviceToHost, s));
        CU_CHECK(h, cudaStreamSynchronize(s));
        h->stats.host_syncs++;
        if (h_plan->n_big == 0) break;
        batch = 2;
        if (r > 4 * MAX_N) return fail(h, PGM_E_CUDA, "matcher failed to converge (internal error)");
    }
    // grid rounds actually needed = first round whose plan had no big pair; the next call on this
    // handle enqueues that many before its first completion check
    const int needed = h_plan->done_round_p1 > 0 ? h_plan->done_round_p1 - 1 : r;
    h->stats.rounds += needed;
    h->stats.evals_computed += (int64_t)h_plan->evals;
    h->rounds_hint = std::max(0, std::min(needed, 64));

    const size_t osmem = order_smem_bytes(nbins, ORDER_THREADS_STANDALONE);
    if (!h->order_attr_set) {
        CU_CHECK(h, cudaFuncSetAttribute(order_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)order_smem_bytes(513, ORDER_THREADS_STANDALONE)));
        h->order_attr_set = true;
    }
    order_kernel<<<n_pairs, ORDER_THREADS_STANDALONE, osmem, s>>>(c, nbins, flags, d_out_qi, d_out_tj, d_out_dist);
    h->stats.kernel_launches += 1;
    CU_CHECK(h, cudaGetLastError());
    return PGM_OK;
}

// Statistics of the last latency-mode call: the tail kernel left them in lat_state.  enqueue_stats_readback adds the
// 16-byte copy to the stream (host-buffer entry points: ahead of the synchronisation they do anyway);
// resolve_pending_stats folds the values into the stats, fetching them first if nobody has.
static void enqueue_stats_readback(pgm_handle *h) {
    if (!h->stats_pending || h->stats_copied || !h->lat_state.p) return;
    const LatState *ls = (const LatState *)h->lat_state.p;
    if (cudaMemcpyAsync(h->pending_plan, &ls->last_rounds, 16, cudaMemcpyDeviceToHost, h->stream) == cudaSuccess) h->stats_copied = true;
}
static void resolve_pending_stats(pgm_handle *h) {
    if (!h->stats_pending) return;
    if (!h->stats_copied) {
        enqueue_stats_readback(h);
        if (!h->stats_copied || cudaStreamSynchronize(h->stream) != cudaSuccess) { h->stats_pending = false; return; }
    }
    const unsigned long long *v = (const unsigned long long *)h->pending_plan;
    h->stats.rounds += (int64_t)v[0];
    h->stats.evals_computed += (int64_t)v[1];
    h->stats_pending = false;
}

static int32_t out_count_for(int32_t n1, int32_t n2, uint32_t flags) {
    return (flags & PGM_FLAG_REFERENCE_COMPAT_TAIL) ? n1 : std::min(n1, n2);
}

static int check_pair(pgm_handle *h, int32_t n1, int32_t n2) {
    if (n1 < 0 || n2 < 0) return fail(h, PGM_E_INVALID_ARG, "negative size");
    if (n1 >= MAX_N || n2 >= MAX_N) return fail(h, PGM_E_INVALID_ARG, "n1 and n2 must be < 2^20");
    if (n1 > 0 && n2 == 0)
        return fail(h, PGM_E_EMPTY_TRAIN, "keypoints2 is empty (KeypointMatching.cs:61 throws)");
    return PGM_OK;
}

extern "C" int pgm_match_hamming_greedy_dev(pgm_handle *h, const uint8_t *d_q, int32_t n1, const uint8_t *d_t,
                                            int32_t n2, int32_t desc_bits, int32_t stride_bytes, int32_t *d_out_qi,
                                            int32_t *d_out_tj, int32_t *d_out_dist, int32_t capacity,
                                            int32_t *out_count, uint32_t flags) {
    if (!h) return PGM_E_INVALID_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    int rc = check_format(h, desc_bits, stride_bytes);
    if (rc) return rc;
    rc = check_pair(h, n1, n2);
    if (rc) return rc;
    h->stats = pgm_stats{};
    h->stats_pending = false;
    const int32_t cnt = out_count_for(n1, n2, flags);
    if (out_count) *out_count = cnt;
    if (n1 == 0) return PGM_OK;
    if (!d_q || !d_t || !d_out_qi || !d_out_tj || !d_out_dist) return fail(h, PGM_E_INVALID_ARG, "null pointer");
    if (capacity < cnt) return fail(h, PGM_E_CAPACITY, "capacity < number of triples");
    CU_CHECK(h, cudaSetDevice(h->device));
    HostPair hp{d_q, d_t, n1, n2, 0};
    return run_chunk(h, &hp, 1, desc_bits, stride_bytes, flags, d_out_qi, d_out_tj, d_out_dist);
}

extern "C" int pgm_match_hamming_greedy(pgm_handle *h, const uint8_t *q, int32_t n1, const uint8_t *t, int32_t n2,
                                        int32_t desc_bits, int32_t stride_bytes, int32_t *out_qi, int32_t *out_tj,
                                        int32_t *out_dist, int32_t capacity, int32_t *out_count, uint32_t flags) {
    if (!h) return PGM_E_INVALID_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    int rc = check_format(h, desc_bits, stride_bytes);
    if (rc) return rc;
    rc = check_pair(h, n1, n2);
    if (rc) return rc;
    h->stats = pgm_stats{};
    h->stats_pending = false;
    const int32_t cnt = out_count_for(n1, n2, flags);
    if (out_count) *out_count = cnt;
    if (n1 == 0) return PGM_OK;
    if (!q || !t || !out_qi || !out_tj || !out_dist) return fail(h, PGM_E_INVALID_ARG, "null pointer");
    if (capacity < cnt) return fail(h, PGM_E_CAPACITY, "capacity < number of triples");
    CU_CHECK(h, cudaSetDevice(h->device));
    cudaStream_t s = h->stream;

    const size_t qb = (size_t)n1 * stride_bytes, tb = (size_t)n2 * stride_bytes;
    const size_t q_off = 0, t_off = align_up(qb, 256);
    const bool in_pinned = is_pinned_host(q) && is_pinned_host(t);
    const bool out_pinned = is_pinned_host(out_qi) && is_pinned_host(out_tj) && is_pinned_host(out_dist);
    if ((rc = ensure_dev(h, h->desc, t_off + tb))) return rc;
    if ((rc = ensure_dev(h, h->out, (size_t)3 * n1 * 4))) return rc;
    if (in_pinned) {
        // the caller's buffers are page-locked: DMA straight out of them
        CU_CHECK(h, cudaMemcpyAsync((char *)h->desc.p + q_off, q, qb, cudaMemcpyHostToDevice, s));
        CU_CHECK(h, cudaMemcpyAsync((char *)h->desc.p + t_off, t, tb, cudaMemcpyHostToDevice, s));
    } else {
        if ((rc = ensure_host(h, h->pin_in, t_off + tb))) return rc;
        memcpy((char *)h->pin_in.p + q_off, q, qb);
        memcpy((char *)h->pin_in.p + t_off, t, tb);
        CU_CHECK(h, cudaMemcpyAsync(h->desc.p, h->pin_in.p, t_off + tb, cudaMemcpyHostToDevice, s));
    }
    int32_t *d_qi = (int32_t *)h->out.p, *d_tj = d_qi + n1, *d_dd = d_tj + n1;
    HostPair hp{(const uint8_t *)h->desc.p + q_off, (const uint8_t *)h->desc.p + t_off, n1, n2, 0};
    rc = run_chunk(h, &hp, 1, desc_bits, stride_bytes, flags, d_qi, d_tj, d_dd);
    if (rc) return rc;
    if (out_pinned) {
        CU_CHECK(h, cudaMemcpyAsync(out_qi, d_qi, (size_t)cnt * 4, cudaMemcpyDeviceToHost, s));
        CU_CHECK(h, cudaMemcpyAsync(out_tj, d_tj, (size_t)cnt * 4, cudaMemcpyDeviceToHost, s));
        CU_CHECK(h, cudaMemcpyAsync(out_dist, d_dd, (size_t)cnt * 4, cudaMemcpyDeviceToHost, s));
        enqueue_stats_readback(h);
        CU_CHECK(h, cudaStreamSynchronize(s));
        h->stats.host_syncs++;
        resolve_pending_stats(h);
    } else {
        if ((rc = ensure_host(h, h->pin_out, (size_t)3 * n1 * 4))) return rc;
        CU_CHECK(h, cudaMemcpyAsync(h->pin_out.p, h->out.p, (size_t)3 * n1 * 4, cudaMemcpyDeviceToHost, s));
        enqueue_stats_readback(h);
        CU_CHECK(h, cudaStreamSynchronize(s));
        h->stats.host_syncs++;
        resolve_pending_stats(h);
        const int32_t *po = (const int32_t *)h->pin_out.p;
        memcpy(out_qi, po, (size_t)cnt * 4);
        memcpy(out_tj, po + n1, (size_t)cnt * 4);
        memcpy(out_dist, po + 2 * (size_t)n1, (size_t)cnt * 4);
    }
    h->stats.h2d_bytes += (int64_t)(qb + tb);
    h->stats.d2h_bytes += (int64_t)3 * (out_pinned ? cnt : n1) * 4;
    return PGM_OK;
}

// ---------------------------------------------------------------------------
// many pairs
// ---------------------------------------------------------------------------
constexpr int MAX_CHUNK_PAIRS = 4096;
constexpr int64_t MAX_CHUNK_SLOTS = 24ll << 20;   // rows + cols per chunk

static int batch_impl(pgm_handle *h, const uint8_t *d_all_desc, const int64_t *image_offsets, int32_t n_images,
                      const int32_t *pair_list, int32_t n_pairs, int32_t desc_bits, int32_t stride_bytes,
                      int32_t *out_qi, int32_t *out_tj, int32_t *out_dist, bool out_on_host, int64_t capacity,
                      int32_t *out_counts, uint32_t flags) {
    cudaStream_t s = h->stream;
    // validate + total size
    int64_t total = 0;
    for (int p = 0; p < n_pairs; p++) {
        const int a = pair_list[2 * p], b = pair_list[2 * p + 1];
        if (a < 0 || a >= n_images || b < 0 || b >= n_images) return fail(h, PGM_E_INVALID_ARG, "pair index out of range");
        const int64_t n1 = image_offsets[a + 1] - image_offsets[a], n2 = image_offsets[b + 1] - image_offsets[b];
        if (n1 < 0 || n2 < 0) return fail(h, PGM_E_INVALID_ARG, "image_offsets must be non-decreasing");
        int rc = check_pair(h, (int32_t)std::min<int64_t>(n1, MAX_N), (int32_t)std::min<int64_t>(n2, MAX_N));
        if (rc) return rc;
        total += n1;
        if (out_counts) out_counts[p] = out_count_for((int32_t)n1, (int32_t)n2, flags);
    }
    if (capacity < total) return fail(h, PGM_E_CAPACITY, "capacity < sum of query sizes");

    // Host outputs: chunk k's triples leave over a second stream (device buffer -> pinned staging) and a
    // helper thread moves them into the caller's (pageable) arrays while chunk k+1 computes.
    struct Joiner {
        std::thread th[2];
        ~Joiner() { for (auto &t : th) if (t.joinable()) t.join(); }
    } jobs;
    if (out_on_host && !h->copy_stream) {
        CU_CHECK(h, cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
        for (int k = 0; k < 2; k++) {
            CU_CHECK(h, cudaEventCreateWithFlags(&h->ev_done[k], cudaEventDisableTiming));
            CU_CHECK(h, cudaEventCreateWithFlags(&h->ev_copied[k], cudaEventDisableTiming));
        }
    }
    // page-locked caller arrays (pgm_host_alloc): the copy stream writes the triples straight into them -- no
    // staging buffer, no helper thread, a third of the host-memory traffic
    const bool out_pinned = out_on_host && is_pinned_host(out_qi) && is_pinned_host(out_tj) && is_pinned_host(out_dist);
    bool slot_used[2] = {false, false};
    std::vector<HostPair> chunk;
    int64_t done_rows = 0;
    int p = 0, chunk_no = 0;
    while (p < n_pairs) {
        chunk.clear();
        int64_t slots = 0, rows = 0;
        while (p < n_pairs && (int)chunk.size() < MAX_CHUNK_PAIRS) {
            const int a = pair_list[2 * p], b = pair_list[2 * p + 1];
            const int32_t n1 = (int32_t)(image_offsets[a + 1] - image_offsets[a]);
            const int32_t n2 = (int32_t)(image_offsets[b + 1] - image_offsets[b]);
            if (!chunk.empty() && slots + n1 + n2 > MAX_CHUNK_SLOTS) break;
            if (n1 > 0)
                chunk.push_back(HostPair{d_all_desc + (size_t)image_offsets[a] * stride_bytes,
                                         d_all_desc + (size_t)image_offsets[b] * stride_bytes, n1, n2, rows});
            slots += n1 + n2; rows += n1;
            p++;
        }
        if (rows == 0) continue;
        const int slot = chunk_no & 1;
        chunk_no++;
        int32_t *d_qi, *d_tj, *d_dd;
        DevBuf &dout = slot ? h->out2 : h->out;
        HostBuf &pin = slot ? h->pin_out2 : h->pin_out;
        if (out_on_host) {
            // this slot's previous user (chunk k-2) must have left both the device buffer and the staging
            if (jobs.th[slot].joinable()) jobs.th[slot].join();
            int rc;
            if (out_pinned && slot_used[slot]) {
                if (dout.cap < (size_t)3 * rows * 4) CU_CHECK(h, cudaEventSynchronize(h->ev_copied[slot]));   // about to reallocate
                else CU_CHECK(h, cudaStreamWaitEvent(s, h->ev_copied[slot], 0));
            }
            if ((rc = ensure_dev(h, dout, (size_t)3 * rows * 4))) return rc;
            if (!out_pinned && (rc = ensure_host(h, pin, (size_t)3 * rows * 4))) return rc;
            d_qi = (int32_t *)dout.p; d_tj = d_qi + rows; d_dd = d_tj + rows;
        } else {
            d_qi = out_qi + done_rows; d_tj = out_tj + done_rows; d_dd = out_dist + done_rows;
        }
        if (!(flags & PGM_FLAG_REFERENCE_COMPAT_TAIL)) {
            // rows beyond min(n1,n2) of a pair are not written without the tail flag: define them
            CU_CHECK(h, cudaMemsetAsync(d_qi, 0xFF, (size_t)rows * 4, s));
            CU_CHECK(h, cudaMemsetAsync(d_tj, 0xFF, (size_t)rows * 4, s));
            CU_CHECK(h, cudaMemsetAsync(d_dd, 0xFF, (size_t)rows * 4, s));
        }
        int rc = run_chunk(h, chunk.data(), (int)chunk.size(), desc_bits, stride_bytes, flags, d_qi, d_tj, d_dd);
        if (rc) return rc;
        if (h->stats_pending) {       // latency-mode chunk: its statistics slot is shared with the next chunk
            enqueue_stats_readback(h);
            CU_CHECK(h, cudaStreamSynchronize(s));
            h->stats.host_syncs++;
            resolve_pending_stats(h);
        }
        if (out_on_host) {
            CU_CHECK(h, cudaEventRecord(h->ev_done[slot], s));
            CU_CHECK(h, cudaStreamWaitEvent(h->copy_stream, h->ev_done[slot], 0));
            if (out_pinned) {
                const size_t nb = (size_t)rows * 4;
                CU_CHECK(h, cudaMemcpyAsync(out_qi + done_rows, d_qi, nb, cudaMemcpyDeviceToHost, h->copy_stream));
                CU_CHECK(h, cudaMemcpyAsync(out_tj + done_rows, d_tj, nb, cudaMemcpyDeviceToHost, h->copy_stream));
                CU_CHECK(h, cudaMemcpyAsync(out_dist + done_rows, d_dd, nb, cudaMemcpyDeviceToHost, h->copy_stream));
                CU_CHECK(h, cudaEventRecord(h->ev_copied[slot], h->copy_stream));
                slot_used[slot] = true;
                h->stats.d2h_bytes += (int64_t)3 * rows * 4;
                done_rows += rows;
                continue;
            }
            CU_CHECK(h, cudaMemcpyAsync(pin.p, dout.p, (size_t)3 * rows * 4, cudaMemcpyDeviceToHost, h->copy_stream));
            CU_CHECK(h, cudaEventRecord(h->ev_copied[slot], h->copy_stream));
            const int32_t *src = (const int32_t *)pin.p;
            int32_t *dq = out_qi + done_rows, *dt = out_tj + done_rows, *dd = out_dist + done_rows;
            cudaEvent_t evc = h->ev_copied[slot];
            const int dev = h->device;
            const size_t nb = (size_t)rows * 4;
            const int64_t nrows = rows;
            jobs.th[slot] = std::thread([=]() {
                cudaSetDevice(dev);
                cudaEventSynchronize(evc);
                memcpy(dq, src, nb);
                memcpy(dt, src + nrows, nb);
                memcpy(dd, src + 2 * nrows, nb);
            });
            h->stats.d2h_bytes += (int64_t)3 * rows * 4;
        }
        done_rows += rows;
    }
    if (out_on_host) {
        for (auto &t : jobs.th) if (t.joinable()) t.join();
        CU_CHECK(h, cudaStreamSynchronize(h->copy_stream));
        CU_CHECK(h, cudaStreamSynchronize(s));
        h->stats.host_syncs++;
        CU_CHECK(h, cudaGetLastError());
    }
    return PGM_OK;
}

extern "C" int pgm_match_pairs_batch_dev(pgm_handle *h, const uint8_t *d_all_desc, const int64_t *image_offsets,
                                         int32_t n_images, const int32_t *pair_list, int32_t n_pairs,
                                         int32_t desc_bits, int32_t stride_bytes, int32_t *d_out_qi,
                                         int32_t *d_out_tj, int32_t *d_out_dist, int64_t capacity,
                                         int32_t *out_counts, uint32_t flags) {
    if (!h) return PGM_E_INVALID_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    int rc = check_format(h, desc_bits, stride_bytes);
    if (rc) return rc;
    if (n_images < 0 || n_pairs < 0 || !image_offsets || (n_pairs > 0 && !pair_list))
        return fail(h, PGM_E_INVALID_ARG, "bad image/pair arguments");
    h->stats = pgm_stats{};
    h->stats_pending = false;
    if (n_pairs == 0) return PGM_OK;
    CU_CHECK(h, cudaSetDevice(h->device));
    return batch_impl(h, d_all_desc, image_offsets, n_images, pair_list, n_pairs, desc_bits, stride_bytes, d_out_qi,
                      d_out_tj, d_out_dist, false, capacity, out_counts, flags);
}

extern "C" int pgm_match_pairs_batch(pgm_handle *h, const uint8_t *all_desc, const int64_t *image_offsets,
                                     int32_t n_images, const int32_t *pair_list, int32_t n_pairs, int32_t desc_bits,
                                     int32_t stride_bytes, int32_t *out_qi, int32_t *out_tj, int32_t *out_dist,
                                     int64_t capacity, int32_t *out_counts, uint32_t flags) {
    if (!h) return PGM_E_INVALID_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    int rc = check_format(h, desc_bits, stride_bytes);
    if (rc) return rc;
    if (n_images < 0 || n_pairs < 0 || !image_offsets || (n_pairs > 0 && !pair_list))
        return fail(h, PGM_E_INVALID_ARG, "bad image/pair arguments");
    h->stats = pgm_stats{};
    h->stats_pending = false;
    if (n_pairs == 0) return PGM_OK;
    CU_CHECK(h, cudaSetDevice(h->device));
    const size_t bytes = (size_t)image_offsets[n_images] * stride_bytes;
    if ((rc = ensure_dev(h, h->desc, std::max<size_t>(bytes, 16)))) return rc;
    if (bytes) {
        // one bulk upload of every image's descriptors; pairs then index into it
        CU_CHECK(h, cudaMemcpyAsync(h->desc.p, all_desc, bytes, cudaMemcpyHostToDevice, h->stream));
        h->stats.h2d_bytes += (int64_t)bytes;
    }
    return batch_impl(h, (const uint8_t *)h->desc.p, image_offsets, n_images, pair_list, n_pairs, desc_bits,
                      stride_bytes, out_qi, out_tj, out_dist, true, capacity, out_counts, flags);
}

// ---------------------------------------------------------------------------
// nearest / second nearest, ratio test, cross-check
// ---------------------------------------------------------------------------
static int knn2_dev_impl(pgm_handle *h, const uint8_t *d_q, int32_t n1, const uint8_t *d_t, int32_t n2,
                         int32_t stride_bytes, int32_t *d_bj, int32_t *d_bd, int32_t *d_sj, int32_t *d_sd,
                         size_t misc_off) {
    const int words = stride_bytes / 4;
    cudaStream_t s = h->stream;
    const int tile_rows = ROUND_THREADS * RQ_DEFAULT;
    const int row_tiles = (n1 + tile_rows - 1) / tile_rows;
    // enough column splits to fill the machine ~2x, each a multiple of STAGE_COLS columns
    int splits = std::max(1, (2 * h->num_sms * 8 + row_tiles - 1) / row_tiles);
    int cps = (n2 + splits - 1) / splits;
    cps = std::max(STAGE_COLS, (cps + STAGE_COLS - 1) / STAGE_COLS * STAGE_COLS);
    splits = std::max(1, (n2 + cps - 1) / cps);
    int rc = ensure_dev(h, h->misc, misc_off + (size_t)splits * n1 * 8);
    if (rc) return rc;
    uint32_t *part = (uint32_t *)((char *)h->misc.p + misc_off);
    dispatch_knn2(words, (const uint32_t *)d_q, n1, (const uint32_t *)d_t, n2, cps, splits, part, s);
    knn2_merge_kernel<<<(n1 + 255) / 256, 256, 0, s>>>(part, n1, splits, d_bj, d_bd, d_sj, d_sd);
    h->stats.kernel_launches += 2;
    h->stats.distance_evals += (int64_t)n1 * n2;
    h->stats.evals_computed += (int64_t)n1 * n2;
    CU_CHECK(h, cudaGetLastError());
    return PGM_OK;
}

extern "C" int pgm_knn2_hamming_dev(pgm_handle *h, const uint8_t *d_q, int32_t n1, const uint8_t *d_t, int32_t n2,
                                    int32_t desc_bits, int32_t stride_bytes, int32_t *d_best_j, int32_t *d_best_d,
                                    int32_t *d_second_j, int32_t *d_second_d) {
    if (!h) return PGM_E_INVALID_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    int rc = check_format(h, desc_bits, stride_bytes);
    if (rc) return rc;
    if (n1 < 0 || n2 < 0 || n1 >= MAX_N || n2 >= MAX_N) return fail(h, PGM_E_INVALID_ARG, "bad sizes");
    h->stats = pgm_stats{};
    h->stats_pending = false;
    if (n1 == 0) return PGM_OK;
    CU_CHECK(h, cudaSetDevice(h->device));
    if (n2 == 0) {
        for (int32_t *o : {d_best_j, d_best_d, d_second_j, d_second_d})
            CU_CHECK(h, cudaMemsetAsync(o, 0xFF, (size_t)n1 * 4, h->stream));
        return PGM_OK;
    }
    return knn2_dev_impl(h, d_q, n1, d_t, n2, stride_bytes, d_best_j, d_best_d, d_second_j, d_second_d, 0);
}

static int upload_pair(pgm_handle *h, const uint8_t *q, int32_t n1, const uint8_t *t, int32_t n2, int stride_bytes,
                       const uint8_t **d_q, const uint8_t **d_t) {
    const size_t qb = (size_t)n1 * stride_bytes, tb = (size_t)n2 * stride_bytes;
    const size_t t_off = align_up(std::max<size_t>(qb, 1), 256);
    int rc;
    if ((rc = ensure_host(h, h->pin_in, t_off + tb + 16))) return rc;
    if ((rc = ensure_dev(h, h->desc, t_off + tb + 16))) return rc;
    if (qb) memcpy(h->pin_in.p, q, qb);
    if (tb) memcpy((char *)h->pin_in.p + t_off, t, tb);
    CU_CHECK(h, cudaMemcpyAsync(h->desc.p, h->pin_in.p, t_off + tb, cudaMemcpyHostToDevice, h->stream));
    *d_q = (const uint8_t *)h->desc.p;
    *d_t = (const uint8_t *)h->desc.p + t_off;
    h->stats.h2d_bytes += (int64_t)(qb + tb);
    return PGM_OK;
}

extern "C" int pgm_knn2_hamming(pgm_handle *h, const uint8_t *q, int32_t n1, const uint8_t *t, int32_t n2,
                                int32_t desc_bits, int32_t stride_bytes, int32_t *best_j, int32_t *best_d,
                                int32_t *second_j, int32_t *second_d) {
    if (!h) return PGM_E_INVALID_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    int rc = check_format(h, desc_bits, stride_bytes);
    if (rc) return rc;
    if (n1 < 0 || n2 < 0 || n1 >= MAX_N || n2 >= MAX_N) return fail(h, PGM_E_INVALID_ARG, "bad sizes");
    h->stats = pgm_stats{};
    h->stats_pending = false;
    if (n1 == 0) return PGM_OK;
    if (n2 == 0) {
        for (int32_t *o : {best_j, best_d, second_j, second_d}) std::fill(o, o + n1, -1);
        return PGM_OK;
    }
    CU_CHECK(h, cudaSetDevice(h->device));
    const uint8_t *d_q, *d_t;
    if ((rc = upload_pair(h, q, n1, t, n2, stride_bytes, &d_q, &d_t))) return rc;
    if ((rc = ensure_dev(h, h->out, (size_t)4 * n1 * 4))) return rc;
    if ((rc = ensure_host(h, h->pin_out, (size_t)4 * n1 * 4))) return rc;
    int32_t *o = (int32_t *)h->out.p;
    if ((rc = knn2_dev_impl(h, d_q, n1, d_t, n2, stride_bytes, o, o + n1, o + 2 * (size_t)n1, o + 3 * (size_t)n1, 0)))
        return rc;
    CU_CHECK(h, cudaMemcpyAsync(h->pin_out.p, o, (size_t)4 * n1 * 4, cudaMemcpyDeviceToHost, h->stream));
    CU_CHECK(h, cudaStreamSynchronize(h->stream));
    h->stats.host_syncs++;
    h->stats.d2h_bytes += (int64_t)4 * n1 * 4;
    const int32_t *po = (const int32_t *)h->pin_out.p;
    memcpy(best_j, po, (size_t)n1 * 4);
    memcpy(best_d, po + n1, (size_t)n1 * 4);
    memcpy(second_j, po + 2 * (size_t)n1, (size_t)n1 * 4);
    memcpy(second_d, po + 3 * (size_t)n1, (size_t)n1 * 4);
    return PGM_OK;
}

extern "C" int pgm_match_ratio_crosscheck(pgm_handle *h, const uint8_t *q, int32_t n1, const uint8_t *t, int32_t n2,
                                          int32_t desc_bits, int32_t stride_bytes, float ratio, int32_t cross_check,
                                          int32_t max_dist, int32_t *out_qi, int32_t *out_tj, int32_t *out_dist,
                                          int32_t capacity, int32_t *out_count) {
    if (!h || !out_count) return PGM_E_INVALID_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    int rc = check_format(h, desc_bits, stride_bytes);
    if (rc) return rc;
    if (n1 < 0 || n2 < 0 || n1 >= MAX_N || n2 >= MAX_N) return fail(h, PGM_E_INVALID_ARG, "bad sizes");
    h->stats = pgm_stats{};
    h->stats_pending = false;
    *out_count = 0;
    if (n1 == 0 || n2 == 0) return PGM_OK;
    CU_CHECK(h, cudaSetDevice(h->device));
    cudaStream_t s = h->stream;
    const uint8_t *d_q, *d_t;
    if ((rc = upload_pair(h, q, n1, t, n2, stride_bytes, &d_q, &d_t))) return rc;
    // layout of h->out: row side 4*n1 | column side 4*n2 | keep n1 bytes
    const size_t o_col = (size_t)4 * n1 * 4, o_keep = o_col + (size_t)4 * n2 * 4, o_end = o_keep + align_up(n1, 16);
    if ((rc = ensure_dev(h, h->out, o_end))) return rc;
    if ((rc = ensure_host(h, h->pin_out, o_end))) return rc;
    int32_t *rj = (int32_t *)h->out.p, *rd = rj + n1, *sj = rd + n1, *sd = sj + n1;
    int32_t *ci = (int32_t *)((char *)h->out.p + o_col), *cd = ci + n2, *c2 = cd + n2, *c3 = c2 + n2;
    uint8_t *keep = (uint8_t *)h->out.p + o_keep;
    if ((rc = knn2_dev_impl(h, d_q, n1, d_t, n2, stride_bytes, rj, rd, sj, sd, 0))) return rc;
    if (cross_check) {
        // column side = the same kernel with the roles swapped: best query per train under (d, i)
        if ((rc = knn2_dev_impl(h, d_t, n2, d_q, n1, stride_bytes, ci, cd, c2, c3, 0))) return rc;
    }
    ratio_crosscheck_kernel<<<(n1 + 255) / 256, 256, 0, s>>>(n1, n2, rj, rd, sd, ci, ratio, cross_check, max_dist, keep);
    h->stats.kernel_launches += 1;
    CU_CHECK(h, cudaMemcpyAsync(h->pin_out.p, h->out.p, o_end, cudaMemcpyDeviceToHost, s));
    CU_CHECK(h, cudaStreamSynchronize(s));
    h->stats.host_syncs++;
    h->stats.d2h_bytes += (int64_t)o_end;
    const int32_t *pj = (const int32_t *)h->pin_out.p, *pd = pj + n1;
    const uint8_t *pk = (const uint8_t *)h->pin_out.p + o_keep;
    int cnt = 0;
    for (int i = 0; i < n1; i++) {
        if (!pk[i]) continue;
        if (cnt >= capacity) return fail(h, PGM_E_CAPACITY, "capacity too small");
        out_qi[cnt] = i; out_tj[cnt] = pj[i]; out_dist[cnt] = pd[i]; cnt++;
    }
    *out_count = cnt;
    h->stats.matched = cnt;
    return PGM_OK;
}

// ---------------------------------------------------------------------------
// many small pairs: nearest neighbour + ratio test + cross-check in ONE launch (BASELINE configs[2]: the consecutive
// frames of a sequence).  Pair p's kept triples (ascending query index) start at sum of n1 over the pairs before it.
// ---------------------------------------------------------------------------
constexpr size_t RCB_SMEM_MAX = 200 * 1024;
template <int WORDS>
static cudaError_t launch_rcb(pgm_handle *h, const RcbPair *d_pairs, int n_pairs, size_t smem, float ratio, int cross_check,
                              int max_dist, int32_t *oq, int32_t *ot, int32_t *od, int32_t *d_counts, cudaStream_t s) {
    cudaError_t e = cudaFuncSetAttribute(ratio_crosscheck_batch_kernel<WORDS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RCB_SMEM_MAX);
    if (e != cudaSuccess) return e;
    (void)h;
    ratio_crosscheck_batch_kernel<WORDS><<<n_pairs, RCB_THREADS, smem, s>>>(d_pairs, ratio, cross_check, max_dist, oq, ot, od, d_counts);
    return cudaGetLastError();
}

extern "C" int pgm_match_ratio_crosscheck_batch_dev(pgm_handle *h, const uint8_t *d_all_desc, const int64_t *image_offsets,
                                                    int32_t n_images, const int32_t *pair_list, int32_t n_pairs,
                                                    int32_t desc_bits, int32_t stride_bytes, float ratio, int32_t cross_check,
                                                    int32_t max_dist, int32_t *d_out_qi, int32_t *d_out_tj,
                                                    int32_t *d_out_dist, int64_t capacity, int32_t *out_counts) {
    if (!h || !out_counts || n_pairs < 0 || n_images < 0 || (n_pairs > 0 && (!image_offsets || !pair_list))) return PGM_E_INVALID_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    int rc = check_format(h, desc_bits, stride_bytes);
    if (rc) return rc;
    h->stats = pgm_stats{};
    h->stats_pending = false;
    if (n_pairs == 0) return PGM_OK;
    if (!d_all_desc || !d_out_qi || !d_out_tj || !d_out_dist) return fail(h, PGM_E_INVALID_ARG, "null pointer");
    CU_CHECK(h, cudaSetDevice(h->device));
    cudaStream_t s = h->stream;
    std::vector<RcbPair> hp(n_pairs);
    int64_t total = 0;
    size_t smem = 0;
    for (int p = 0; p < n_pairs; p++) {
        const int a = pair_list[2 * p], b = pair_list[2 * p + 1];
        if (a < 0 || a >= n_images || b < 0 || b >= n_images) return fail(h, PGM_E_INVALID_ARG, "pair index out of range");
        const int64_t n1 = image_offsets[a + 1] - image_offsets[a], n2 = image_offsets[b + 1] - image_offsets[b];
        if (n1 < 0 || n2 < 0 || n1 >= MAX_N || n2 >= MAX_N) return fail(h, PGM_E_INVALID_ARG, "bad image sizes");
        hp[p] = RcbPair{(const uint32_t *)(d_all_desc + (size_t)image_offsets[a] * stride_bytes),
                        (const uint32_t *)(d_all_desc + (size_t)image_offsets[b] * stride_bytes), (int32_t)n1, (int32_t)n2, total};
        total += n1;
        smem = std::max(smem, (size_t)(n1 + n2) * stride_bytes + (size_t)n2 * 4 + 16);
    }
    if (capacity < total) return fail(h, PGM_E_CAPACITY, "capacity < sum of query sizes");
    if (smem > RCB_SMEM_MAX)
        return fail(h, PGM_E_INVALID_ARG, "a pair is too large for the small-pair batch kernel (use pgm_match_ratio_crosscheck_pairs_batch_dev)");
    const size_t pb = align_up(sizeof(RcbPair) * n_pairs, 256);
    if ((rc = ensure_dev(h, h->misc, pb + (size_t)n_pairs * 4))) return rc;
    if ((rc = ensure_host(h, h->pin_in, pb + (size_t)n_pairs * 4))) return rc;
    CU_CHECK(h, cudaStreamSynchronize(s));                 // the staging buffer may still feed an earlier call's copy
    memcpy(h->pin_in.p, hp.data(), sizeof(RcbPair) * n_pairs);
    CU_CHECK(h, cudaMemcpyAsync(h->misc.p, h->pin_in.p, sizeof(RcbPair) * n_pairs, cudaMemcpyHostToDevice, s));
    const RcbPair *d_pairs = (const RcbPair *)h->misc.p;
    int32_t *d_counts = (int32_t *)((char *)h->misc.p + pb);
    cudaError_t e;
    switch (stride_bytes / 4) {
        case 4: e = launch_rcb<4>(h, d_pairs, n_pairs, smem, ratio, cross_check, max_dist, d_out_qi, d_out_tj, d_out_dist, d_counts, s); break;
        case 8: e = launch_rcb<8>(h, d_pairs, n_pairs, smem, ratio, cross_check, max_dist, d_out_qi, d_out_tj, d_out_dist, d_counts, s); break;
        case 12: e = launch_rcb<12>(h, d_pairs, n_pairs, smem, ratio, cross_check, max_dist, d_out_qi, d_out_tj, d_out_dist, d_counts, s); break;
        default: e = launch_rcb<16>(h, d_pairs, n_pairs, smem, ratio, cross_check, max_dist, d_out_qi, d_out_tj, d_out_dist, d_counts, s); break;
    }
    CU_CHECK(h, e);
    CU_CHECK(h, cudaMemcpyAsync((char *)h->pin_in.p + pb, d_counts, (size_t)n_pairs * 4, cudaMemcpyDeviceToHost, s));
    CU_CHECK(h, cudaStreamSynchronize(s));
    memcpy(out_counts, (char *)h->pin_in.p + pb, (size_t)n_pairs * 4);
    h->stats.kernel_launches += 1; h->stats.host_syncs += 2; h->stats.pairs = n_pairs;
    for (int p = 0; p < n_pairs; p++) { h->stats.distance_evals += (int64_t)hp[p].n1 * hp[p].n2; h->stats.matched += out_counts[p]; }
    h->stats.evals_computed = h->stats.distance_evals * (cross_check ? 2 : 1);
    return PGM_OK;
}

// ---------------------------------------------------------------------------
// many pairs of any size: the same result through one fused distance pass per chunk (pgm_kernels.cuh, RcpPair).
// The host plans every chunk first, uploads the whole plan in one copy and then only enqueues: three kernels per
// chunk, no read-back until the counts at the end.
// ---------------------------------------------------------------------------
template <int WORDS, bool CROSS>
static int rcp_occupancy() {
    int nb = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, knn2_cols_pairs_kernel<WORDS, CROSS>, ROUND_THREADS, 0);
    return std::max(nb, 1);
}
template <int WORDS>
static void launch_rcp_dist(bool cross, int grid, const RcpPair *pairs, const int32_t *tile_base, int n, uint2 *part,
                            int64_t part_cap, uint32_t *colbest, int64_t col_cap, cudaStream_t s) {
    if (cross) knn2_cols_pairs_kernel<WORDS, true><<<grid, ROUND_THREADS, 0, s>>>(pairs, tile_base, n, part, part_cap, colbest, col_cap);
    else knn2_cols_pairs_kernel<WORDS, false><<<grid, ROUND_THREADS, 0, s>>>(pairs, tile_base, n, part, part_cap, colbest, col_cap);
}

struct RcpChunk {
    int first, n;              // its pairs: plan[first, first + n)
    int base_off;              // tile_base at bases[base_off], fblk_base at bases[base_off + n + 1]
    int32_t items, fblocks;    // distance-kernel CTAs, filter / scatter CTAs
    int64_t part_slots, cols, rows;
};

extern "C" int pgm_match_ratio_crosscheck_pairs_batch_dev(pgm_handle *h, const uint8_t *d_all_desc, const int64_t *image_offsets,
                                                          int32_t n_images, const int32_t *pair_list, int32_t n_pairs,
                                                          int32_t desc_bits, int32_t stride_bytes, float ratio, int32_t cross_check,
                                                          int32_t max_dist, int32_t *d_out_qi, int32_t *d_out_tj,
                                                          int32_t *d_out_dist, int64_t capacity, int32_t *out_counts) {
    if (!h || !out_counts || n_pairs < 0 || n_images < 0 || (n_pairs > 0 && (!image_offsets || !pair_list))) return PGM_E_INVALID_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    int rc = check_format(h, desc_bits, stride_bytes);
    if (rc) return rc;
    h->stats = pgm_stats{};
    h->stats_pending = false;
    if (n_pairs == 0) return PGM_OK;
    if (!d_all_desc || !d_out_qi || !d_out_tj || !d_out_dist) return fail(h, PGM_E_INVALID_ARG, "null pointer");
    int64_t total = 0, evals = 0;
    for (int p = 0; p < n_pairs; p++) {
        const int a = pair_list[2 * p], b = pair_list[2 * p + 1];
        if (a < 0 || a >= n_images || b < 0 || b >= n_images) return fail(h, PGM_E_INVALID_ARG, "pair index out of range");
        const int64_t n1 = image_offsets[a + 1] - image_offsets[a], n2 = image_offsets[b + 1] - image_offsets[b];
        if (n1 < 0 || n2 < 0 || n1 >= MAX_N || n2 >= MAX_N) return fail(h, PGM_E_INVALID_ARG, "bad image sizes");
        total += n1;
        evals += n1 * n2;
    }
    if (capacity < total) return fail(h, PGM_E_CAPACITY, "capacity < sum of query sizes");
    CU_CHECK(h, cudaSetDevice(h->device));
    cudaStream_t s = h->stream;
    const int words = stride_bytes / 4;
    const bool cross = cross_check != 0;
    int ctas_per_sm;
    switch (words) {
        case 4: ctas_per_sm = cross ? rcp_occupancy<4, true>() : rcp_occupancy<4, false>(); break;
        case 8: ctas_per_sm = cross ? rcp_occupancy<8, true>() : rcp_occupancy<8, false>(); break;
        case 12: ctas_per_sm = cross ? rcp_occupancy<12, true>() : rcp_occupancy<12, false>(); break;
        default: ctas_per_sm = cross ? rcp_occupancy<16, true>() : rcp_occupancy<16, false>(); break;
    }
    // few row tiles (one big pair): split the columns until the distance kernel has about two waves of CTAs
    const int64_t target_items = 2ll * h->num_sms * ctas_per_sm;
    constexpr int tile_rows = ROUND_THREADS * RQ_LARGE;

    // plan: chunks of <= MAX_CHUNK_PAIRS pairs and <= MAX_CHUNK_SLOTS rows + columns (as batch_impl); a pair without
    // query or train rows keeps no triple and is not launched
    std::vector<RcpPair> plan;
    std::vector<int32_t> bases;
    std::vector<RcpChunk> chunks;
    int64_t out_base = 0, max_part = 0, max_cols = 0, max_rows = 0, max_fblocks = 0;
    for (int p = 0; p < n_pairs;) {
        RcpChunk c{(int)plan.size(), 0, (int)bases.size(), 0, 0, 0, 0, 0};
        int64_t row_tiles = 0;
        for (; p < n_pairs && c.n < MAX_CHUNK_PAIRS; p++) {
            const int a = pair_list[2 * p], b = pair_list[2 * p + 1];
            const int32_t n1 = (int32_t)(image_offsets[a + 1] - image_offsets[a]), n2 = (int32_t)(image_offsets[b + 1] - image_offsets[b]);
            if (n1 > 0 && n2 > 0) {
                if (c.n > 0 && c.rows + c.cols + n1 + n2 > MAX_CHUNK_SLOTS) break;
                RcpPair r{};
                r.q = (const uint32_t *)(d_all_desc + (size_t)image_offsets[a] * stride_bytes);
                r.t = (const uint32_t *)(d_all_desc + (size_t)image_offsets[b] * stride_bytes);
                r.n1 = n1; r.n2 = n2; r.out_base = out_base; r.col_base = c.cols; r.row_base = c.rows; r.pair_id = p;
                plan.push_back(r);
                c.n++; c.cols += n2; c.rows += n1;
                row_tiles += (n1 + tile_rows - 1) / tile_rows;
            }
            out_base += n1;
        }
        if (c.n == 0) continue;
        const int64_t want = row_tiles >= target_items ? 1 : (target_items + row_tiles - 1) / row_tiles;
        bases.resize(bases.size() + 2 * (size_t)(c.n + 1));
        int32_t *tb = bases.data() + c.base_off, *fb = tb + c.n + 1;
        for (int k = 0; k < c.n; k++) {
            RcpPair &r = plan[c.first + k];
            const int64_t col_stages = (r.n2 + STAGE_LARGE - 1) / STAGE_LARGE;
            const int64_t splits = std::min(want, col_stages);
            r.cols_per_split = (int32_t)((col_stages + splits - 1) / splits * STAGE_LARGE);
            r.splits = (r.n2 + r.cols_per_split - 1) / r.cols_per_split;
            r.part_base = c.part_slots;
            c.part_slots += (int64_t)r.n1 * r.splits;
            tb[k] = c.items; fb[k] = c.fblocks;
            c.items += (r.n1 + tile_rows - 1) / tile_rows * r.splits;
            c.fblocks += (r.n1 + RCF_THREADS - 1) / RCF_THREADS;
        }
        tb[c.n] = c.items; fb[c.n] = c.fblocks;
        max_part = std::max(max_part, c.part_slots); max_cols = std::max(max_cols, c.cols);
        max_rows = std::max(max_rows, c.rows); max_fblocks = std::max<int64_t>(max_fblocks, c.fblocks);
        chunks.push_back(c);
    }

    // h->misc: plan | bases | counts | partials | column minima | per-row results | block counts (reused by every chunk)
    const size_t o_bases = align_up(sizeof(RcpPair) * std::max<size_t>(plan.size(), 1), 256);
    const size_t o_counts = o_bases + align_up(4 * std::max<size_t>(bases.size(), 1), 256);
    const size_t o_part = o_counts + align_up(4 * (size_t)n_pairs, 256);
    const size_t o_col = o_part + align_up(8 * (size_t)std::max<int64_t>(max_part, 1), 256);
    const size_t o_res = o_col + align_up(4 * (size_t)std::max<int64_t>(max_cols, 1), 256);
    const size_t o_bcnt = o_res + align_up(4 * (size_t)std::max<int64_t>(max_rows, 1), 256);
    const size_t o_end = o_bcnt + align_up(4 * (size_t)std::max<int64_t>(max_fblocks, 1), 256);
    if ((rc = ensure_dev(h, h->misc, o_end))) return rc;
    if ((rc = ensure_host(h, h->pin_in, o_part))) return rc;
    CU_CHECK(h, cudaStreamSynchronize(s));                 // the staging buffer may still feed an earlier call's copy
    char *pin = (char *)h->pin_in.p, *dev = (char *)h->misc.p;
    memcpy(pin, plan.data(), sizeof(RcpPair) * plan.size());
    memcpy(pin + o_bases, bases.data(), 4 * bases.size());
    CU_CHECK(h, cudaMemcpyAsync(dev, pin, o_counts, cudaMemcpyHostToDevice, s));
    CU_CHECK(h, cudaMemsetAsync(dev + o_counts, 0, 4 * (size_t)n_pairs, s));
    const RcpPair *d_plan = (const RcpPair *)dev;
    const int32_t *d_bases = (const int32_t *)(dev + o_bases);
    int32_t *d_counts = (int32_t *)(dev + o_counts), *d_bcnt = (int32_t *)(dev + o_bcnt);
    uint2 *d_part = (uint2 *)(dev + o_part);
    uint32_t *d_col = (uint32_t *)(dev + o_col), *d_res = (uint32_t *)(dev + o_res);
    for (const RcpChunk &c : chunks) {
        const RcpPair *cp = d_plan + c.first;
        const int32_t *tb = d_bases + c.base_off, *fb = tb + c.n + 1;
        if (cross) CU_CHECK(h, cudaMemsetAsync(d_col, 0xFF, 4 * (size_t)c.cols, s));     // KEY_NONE
        switch (words) {
            case 4: launch_rcp_dist<4>(cross, c.items, cp, tb, c.n, d_part, c.part_slots, d_col, c.cols, s); break;
            case 8: launch_rcp_dist<8>(cross, c.items, cp, tb, c.n, d_part, c.part_slots, d_col, c.cols, s); break;
            case 12: launch_rcp_dist<12>(cross, c.items, cp, tb, c.n, d_part, c.part_slots, d_col, c.cols, s); break;
            default: launch_rcp_dist<16>(cross, c.items, cp, tb, c.n, d_part, c.part_slots, d_col, c.cols, s); break;
        }
        rcp_filter_kernel<<<c.fblocks, RCF_THREADS, 0, s>>>(cp, fb, c.n, d_part, c.part_slots, d_col, c.cols, ratio,
                                                            cross ? 1 : 0, max_dist, d_res, d_bcnt);
        rcp_scatter_kernel<<<c.fblocks, RCF_THREADS, 0, s>>>(cp, fb, c.n, d_res, d_bcnt, capacity, d_out_qi, d_out_tj,
                                                             d_out_dist, d_counts);
        CU_CHECK(h, cudaGetLastError());
        h->stats.kernel_launches += 3;
    }
    CU_CHECK(h, cudaMemcpyAsync(pin + o_counts, d_counts, 4 * (size_t)n_pairs, cudaMemcpyDeviceToHost, s));
    CU_CHECK(h, cudaStreamSynchronize(s));
    memcpy(out_counts, pin + o_counts, 4 * (size_t)n_pairs);
    h->stats.host_syncs += 2; h->stats.pairs = n_pairs;
    h->stats.distance_evals = evals;
    h->stats.evals_computed = evals;                       // one fused pass, cross-check or not
    for (int p = 0; p < n_pairs; p++) h->stats.matched += out_counts[p];
    return PGM_OK;
}

// ---------------------------------------------------------------------------
// train-sharded nearest neighbours: key exchange format, top-2 merge, device-side filter
// ---------------------------------------------------------------------------
extern "C" int pgm_pack_top2_keys_dev(pgm_handle *h, const int32_t *d_best_j, const int32_t *d_best_d,
                                      const int32_t *d_second_j, const int32_t *d_second_d, int32_t n,
                                      int32_t index_offset, int32_t *d_keys) {
    if (!h) return PGM_E_INVALID_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    if (n < 0 || index_offset < 0 || index_offset >= MAX_N ||
        (n > 0 && (!d_best_j || !d_best_d || !d_second_j || !d_second_d || !d_keys)))
        return fail(h, PGM_E_INVALID_ARG, "bad arguments");
    if (n == 0) return PGM_OK;
    CU_CHECK(h, cudaSetDevice(h->device));
    pack_top2_kernel<<<(n + 255) / 256, 256, 0, h->stream>>>(d_best_j, d_best_d, d_second_j, d_second_d, n, index_offset,
                                                             (uint32_t *)d_keys);
    h->stats.kernel_launches += 1;
    CU_CHECK(h, cudaGetLastError());
    return PGM_OK;
}

extern "C" int pgm_merge_top2_dev(pgm_handle *h, const int32_t *d_keys, int32_t n_shards, int32_t n, int32_t *d_best_j,
                                  int32_t *d_best_d, int32_t *d_second_j, int32_t *d_second_d) {
    if (!h) return PGM_E_INVALID_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    if (n < 0 || n_shards < 1 || (n > 0 && (!d_keys || !d_best_j || !d_best_d || !d_second_j || !d_second_d)))
        return fail(h, PGM_E_INVALID_ARG, "bad arguments");
    if (n == 0) return PGM_OK;
    CU_CHECK(h, cudaSetDevice(h->device));
    merge_top2_kernel<<<(n + 255) / 256, 256, 0, h->stream>>>((const uint32_t *)d_keys, n_shards, n, d_best_j, d_best_d,
                                                              d_second_j, d_second_d);
    h->stats.kernel_launches += 1;
    CU_CHECK(h, cudaGetLastError());
    return PGM_OK;
}

extern "C" int pgm_ratio_crosscheck_filter_dev(pgm_handle *h, int32_t n1, int32_t n2, const int32_t *d_best_j,
                                               const int32_t *d_best_d, const int32_t *d_second_d,
                                               const int32_t *d_col_best_i, float ratio, int32_t cross_check,
                                               int32_t max_dist, int32_t *d_out_qi, int32_t *d_out_tj,
                                               int32_t *d_out_dist, int32_t *out_count) {
    if (!h || !out_count) return PGM_E_INVALID_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    *out_count = 0;
    if (n1 < 0 || n2 < 0 || n1 >= MAX_N || (cross_check && n1 > 0 && n2 > 0 && !d_col_best_i) ||
        (n1 > 0 && (!d_best_j || !d_best_d || !d_second_d || !d_out_qi || !d_out_tj || !d_out_dist)))
        return fail(h, PGM_E_INVALID_ARG, "bad arguments");
    if (n1 == 0 || n2 == 0) return PGM_OK;
    CU_CHECK(h, cudaSetDevice(h->device));
    cudaStream_t s = h->stream;
    int rc = ensure_dev(h, h->out, align_up(n1, 16) + 16);
    if (rc) return rc;
    if ((rc = ensure_host(h, h->pin_out, 64))) return rc;
    uint8_t *keep = (uint8_t *)h->out.p;
    int32_t *d_cnt = (int32_t *)((char *)h->out.p + align_up(n1, 16));
    ratio_crosscheck_kernel<<<(n1 + 255) / 256, 256, 0, s>>>(n1, n2, d_best_j, d_best_d, d_second_d, d_col_best_i, ratio,
                                                             cross_check, max_dist, keep);
    compact_matches_kernel<<<1, 1024, 0, s>>>(keep, d_best_j, d_best_d, n1, d_out_qi, d_out_tj, d_out_dist, d_cnt);
    CU_CHECK(h, cudaMemcpyAsync(h->pin_out.p, d_cnt, 4, cudaMemcpyDeviceToHost, s));
    CU_CHECK(h, cudaStreamSynchronize(s));
    *out_count = *(const int32_t *)h->pin_out.p;
    h->stats.kernel_launches += 2; h->stats.host_syncs++; h->stats.matched = *out_count;
    CU_CHECK(h, cudaGetLastError());
    return PGM_OK;
}

// ---------------------------------------------------------------------------
// match_keypoints of the Python generation: every row ranked (keypoint_matching.py:7-33)
// ---------------------------------------------------------------------------
template <int WORDS>
static void launch_sorted_rows(const uint32_t *q, int n1, const uint32_t *t, int n2, int nbins, long long *out,
                               cudaStream_t s) {
    sorted_rows_kernel<WORDS><<<n1, TWIN_THREADS, sizeof(int32_t) * TWIN_WARPS * (nbins + 1), s>>>(q, n1, t, n2, nbins, out);
}
static int sorted_rows_dev_impl(pgm_handle *h, const uint8_t *d_q, int32_t n1, const uint8_t *d_t, int32_t n2,
                                int32_t desc_bits, int32_t stride_bytes, int64_t *d_out) {
    (void)desc_bits;
    const int nbins = 8 * stride_bytes + 1;   // by padded width: set padding bits must not index outside the histogram
    const uint32_t *q = (const uint32_t *)d_q, *t = (const uint32_t *)d_t;
    switch (stride_bytes / 4) {
        case 4: launch_sorted_rows<4>(q, n1, t, n2, nbins, (long long *)d_out, h->stream); break;
        case 8: launch_sorted_rows<8>(q, n1, t, n2, nbins, (long long *)d_out, h->stream); break;
        case 12: launch_sorted_rows<12>(q, n1, t, n2, nbins, (long long *)d_out, h->stream); break;
        default: launch_sorted_rows<16>(q, n1, t, n2, nbins, (long long *)d_out, h->stream); break;
    }
    h->stats.kernel_launches += 1;
    h->stats.distance_evals += (int64_t)n1 * n2;
    h->stats.evals_computed += 2 * (int64_t)n1 * n2;
    CU_CHECK(h, cudaGetLastError());
    return PGM_OK;
}

extern "C" int pgm_match_keypoints_sorted_dev(pgm_handle *h, const uint8_t *d_q, int32_t n1, const uint8_t *d_t,
                                              int32_t n2, int32_t desc_bits, int32_t stride_bytes, int64_t *d_out) {
    if (!h) return PGM_E_INVALID_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    int rc = check_format(h, desc_bits, stride_bytes);
    if (rc) return rc;
    if (n1 < 0 || n2 < 0 || n1 >= MAX_N || n2 >= MAX_N) return fail(h, PGM_E_INVALID_ARG, "bad sizes");
    h->stats = pgm_stats{};
    h->stats_pending = false;
    if (n1 == 0 || n2 == 0) return PGM_OK;
    CU_CHECK(h, cudaSetDevice(h->device));
    return sorted_rows_dev_impl(h, d_q, n1, d_t, n2, desc_bits, stride_bytes, d_out);
}

extern "C" int pgm_match_keypoints_sorted(pgm_handle *h, const uint8_t *q, int32_t n1, const uint8_t *t, int32_t n2,
                                          int32_t desc_bits, int32_t stride_bytes, int64_t *out) {
    if (!h) return PGM_E_INVALID_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    int rc = check_format(h, desc_bits, stride_bytes);
    if (rc) return rc;
    if (n1 < 0 || n2 < 0 || n1 >= MAX_N || n2 >= MAX_N) return fail(h, PGM_E_INVALID_ARG, "bad sizes");
    h->stats = pgm_stats{};
    h->stats_pending = false;
    if (n1 == 0 || n2 == 0) return PGM_OK;
    CU_CHECK(h, cudaSetDevice(h->device));
    const uint8_t *d_q, *d_t;
    if ((rc = upload_pair(h, q, n1, t, n2, stride_bytes, &d_q, &d_t))) return rc;
    const size_t bytes = (size_t)n1 * n2 * 16;
    if ((rc = ensure_dev(h, h->out, bytes))) return rc;
    if ((rc = sorted_rows_dev_impl(h, d_q, n1, d_t, n2, desc_bits, stride_bytes, (int64_t *)h->out.p))) return rc;
    CU_CHECK(h, cudaMemcpyAsync(out, h->out.p, bytes, cudaMemcpyDeviceToHost, h->stream));
    CU_CHECK(h, cudaStreamSynchronize(h->stream));
    h->stats.host_syncs++;
    h->stats.d2h_bytes += (int64_t)bytes;
    return PGM_OK;
}

// ---------------------------------------------------------------------------
// float descriptors: squared-L2 nearest / second nearest on tcgen05 (pgm_l2.cuh)
// ---------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                    const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode_tiled() {
    static PFN_encodeTiled fn = nullptr;
    if (!fn) {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = (PFN_encodeTiled)p;
    }
    return fn;
}

// rows x kprime bf16, row-major; box = 64 (K, 128 bytes) x 128 rows, 128-byte swizzle
static int make_operand_map(pgm_handle *h, CUtensorMap *map, void *base, int rows, int kprime, int box_rows = pgm_l2::TILE_N) {
    PFN_encodeTiled enc = get_encode_tiled();
    if (!enc) return fail(h, PGM_E_CUDA, "cuTensorMapEncodeTiled entry point not available");
    cuuint64_t gdim[2] = {(cuuint64_t)kprime, (cuuint64_t)rows};
    cuuint64_t gstr[1] = {(cuuint64_t)kprime * 2};
    cuuint32_t box[2] = {(cuuint32_t)pgm_l2::CHUNK_K, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, base, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(h, PGM_E_CUDA, "cuTensorMapEncodeTiled failed");
    return PGM_OK;
}

// kernel attributes and the co-resident cluster count of the CTA-pair kernel, once per handle
static int l2_setup(pgm_handle *h) {
    using namespace pgm_l2;
    if (h->l2_attr_set) return PGM_OK;
    CU_CHECK(h, cudaFuncSetAttribute(l2_topk_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)l2_smem_bytes()));
    CU_CHECK(h, cudaFuncSetAttribute(l2_topk_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)l2_smem_bytes()));
    CU_CHECK(h, cudaFuncSetAttribute(l2_topk_pair_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)l2_pair_smem_bytes()));
    CU_CHECK(h, cudaFuncSetAttribute(l2_topk_pair_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)l2_pair_smem_bytes()));
    CU_CHECK(h, cudaFuncSetAttribute(l2_topk_pair_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)l2_pair_smem_bytes()));
    // how many CTA pairs are co-resident: the pair kernel is persistent, one segment of the work per cluster
    cudaLaunchAttribute ca{};
    ca.id = cudaLaunchAttributeClusterDimension;
    ca.val.clusterDim.x = 2; ca.val.clusterDim.y = 1; ca.val.clusterDim.z = 1;
    cudaLaunchConfig_t qc{};
    qc.gridDim = dim3(2 * (unsigned)h->num_sms); qc.blockDim = dim3(THREADS);
    qc.dynamicSmemBytes = l2_pair_smem_bytes(); qc.attrs = &ca; qc.numAttrs = 1;
    int nc = 0;
    if (cudaOccupancyMaxActiveClusters(&nc, l2_topk_pair_kernel<false, false>, &qc) != cudaSuccess || nc < 1) {
        (void)cudaGetLastError();
        nc = std::max(1, h->num_sms / 2);
    }
    h->l2_max_clusters = std::min(nc, std::max(1, h->num_sms / 2));
    h->l2_attr_set = true;
    return PGM_OK;
}

static int l2_dev_impl(pgm_handle *h, const float *d_q, int32_t n1, const float *d_t, int32_t n2, int32_t dim,
                       int32_t *d_bj, float *d_bd, int32_t *d_sj, float *d_sd, float *d_dbg) {
    using namespace pgm_l2;
    cudaStream_t s = h->stream;
    const int dp = (dim + CHUNK_K - 1) / CHUNK_K * CHUNK_K, dpc = dp / CHUNK_K;
    const int row_tiles = (n1 + TILE_M - 1) / TILE_M;
    // CTA pairs (cta_group::2, M = 256 x N = 256) whenever there are at least two row tiles.  Ranking precision: one
    // fp16 term + certified band + exhaustive fallback (pair kernel), or the three-term bf16 split (single-CTA kernel)
    const bool pair = row_tiles >= 2, fp16 = pair;
    const int kprime = fp16 ? dp + CHUNK_K : 2 * dp + CHUNK_K;   // rows = [x16 | norm] or [hi | lo | norm]
    int rc = l2_setup(h);
    if (rc) return rc;
    int splits = 1, tps = 0, items = 0, clusters = 0;
    const int row_pairs = (row_tiles + 1) / 2;
    const int col_tiles = (n2 + (pair ? TILE_N2 : TILE_N) - 1) / (pair ? TILE_N2 : TILE_N);
    if (pair) {
        // equal contiguous segments of the row-major (row pair, column tile) list, one per resident cluster: no wave
        // quantisation (DESIGN.md section 4.2)
        const long long total = (long long)row_pairs * col_tiles;
        if (total > 0x7FFFFFFFll) return fail(h, PGM_E_INVALID_ARG, "problem too large for the float path");
        items = (int)total;
        clusters = std::min(h->l2_max_clusters, items);
        // a row pair's candidates come from every segment that touches it: slots = the most any row pair sees
        for (int rp = 0; rp < row_pairs; rp++) {
            const long long x0 = (long long)rp * col_tiles, x1 = x0 + col_tiles - 1;
            const int k0 = (int)(((x0 + 1) * clusters - 1) / items), k1 = (int)(((x1 + 1) * clusters - 1) / items);
            splits = std::max(splits, k1 - k0 + 1);
        }
    } else {
        // column splits: the run time is (waves) x (tiles per split); pick the split count that minimises it
        // (half a tile of fixed cost per unit for the resident A' load)
        tps = col_tiles;
        double best_cost = 1e300;
        for (int sp = 1; sp <= std::min(col_tiles, 32); sp++) {
            const int t = (col_tiles + sp - 1) / sp, se = (col_tiles + t - 1) / t;
            const double cost = (double)(((long long)row_tiles * se + h->num_sms - 1) / h->num_sms) * (t + 0.5);
            if (cost < best_cost - 1e-9) { best_cost = cost; splits = se; tps = t; }
        }
    }
    // scratch: A' | B' | cand_j | cand_d
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 1024); return o; };
    const size_t o_a = take((size_t)n1 * kprime * 2), o_b = take((size_t)n2 * kprime * 2);
    const size_t o_cj = take((size_t)splits * n1 * CAND * 4), o_cd = take((size_t)splits * n1 * CAND * 4);
    // fp16 mode: [max |x| bits, flagged-row count | ticket per flagged row] (one memset), flagged rows, slice partials
    const size_t o_ovf = take(fp16 ? (size_t)n1 * 4 : 0);
    const size_t o_part = take(fp16 ? (size_t)n1 * EX_MAX_SLICES_PER_ROW * 16 : 0);
    const size_t o_qn = take((size_t)n1 * 4), o_drop = take((size_t)splits * n1 * EPI_GROUPS * 4);
    if ((rc = ensure_dev(h, h->misc, off))) return rc;
    if (fp16 && h->l2_state.cap < 16) {
        if ((rc = ensure_dev(h, h->l2_state, 16))) return rc;
        CU_CHECK(h, cudaMemsetAsync(h->l2_state.p, 0, h->l2_state.cap, s));
    }
    char *base = (char *)h->misc.p;
    __nv_bfloat16 *a = (__nv_bfloat16 *)(base + o_a), *b = (__nv_bfloat16 *)(base + o_b);
    L2Params p{};
    p.n1 = n1; p.n2 = n2; p.dpc = dpc; p.tiles_per_split = tps; p.col_tiles = col_tiles; p.items = items;
    p.key_mask = 0x7FFFFFE0u;
    unsigned *hdr = fp16 ? (unsigned *)h->l2_state.p : nullptr;
    int32_t *ovf_rows = fp16 ? (int32_t *)(base + o_ovf) : nullptr;
    float *qnorm = (float *)(base + o_qn);
    p.qnorm = qnorm; p.cand_drop = (float *)(base + o_drop);
    // band of the ranking (d-domain, two approximations compared): 2^-12 (3|q|^2 + 2d) covers the three-term bf16 split
    // 2.8 times over; one fp16 term needs 2 x 2^-10, taken with 25 % to spare.  The accumulator holds -d s^2 / 2, hence
    // half of it there; the absolute terms (fp16 subnormals under the global scale, the norm chunk's last term) are
    // expressed in scaled units, where max |x| < 2^10.
    const float slack_rel = fp16 ? 0.00244140625f : 0.000244140625f;
    p.band_rel = 0.5f * slack_rel;
    p.band_abs_sqrt = fp16 ? 4.8828125e-7f * sqrtf((float)dp) : 0.f;     // 2^-21 sqrt(D) sqrt(3|q|^2 + 4|a|)
    p.band_abs_const = fp16 ? 2.44140625e-4f : 0.f;                        // 2^-12
    p.absmax_bits = hdr;
    h->l2_hdr = hdr;
    h->l2_fallback_word = 1;
    p.cand_j = (int32_t *)(base + o_cj); p.cand_d = (float *)(base + o_cd); p.dbg_dist = d_dbg;
    const bool tl = getenv("PGM_L2_TIMELINE") != nullptr;
    if (tl) {
        if ((rc = ensure_dev(h, h->timeline, 1000 * 8))) return rc;
        CU_CHECK(h, cudaMemsetAsync(h->timeline.p, 0, 1000 * 8, s));
        p.timeline = (unsigned long long *)h->timeline.p;
    }
    // the GEMM kernel and the refinement are programmatic dependents of their predecessors (griddepcontrol)
    cudaLaunchAttribute pdl{};
    pdl.id = cudaLaunchAttributeProgrammaticStreamSerialization;
    pdl.val.programmaticStreamSerializationAllowed = 1;
    cudaLaunchConfig_t cfg{};
    cfg.stream = s; cfg.attrs = &pdl; cfg.numAttrs = 1;
    const int split_blocks = (int)(((size_t)(n1 + n2) * 32 + 255) / 256);
    if (fp16) {
        const size_t nq = (size_t)n1 * dim, nt = (size_t)n2 * dim;
        const int ab = (int)std::min<size_t>((size_t)h->num_sms * 8, (nq + nt + 4095) / 4096 + 1);
        absmax_kernel<<<ab, 256, 0, s>>>(d_q, nq, d_t, nt, hdr);
        cfg.gridDim = dim3((unsigned)split_blocks); cfg.blockDim = dim3(256); cfg.dynamicSmemBytes = 0;
        CU_CHECK(h, cudaLaunchKernelEx(&cfg, split16_kernel, d_q, (int)n1, d_t, (int)n2, (int)dim, dp, (__half *)a, (__half *)b,
                                       p.cand_j, splits, (const unsigned *)hdr, qnorm, p.cand_drop));
    } else {
        split_kernel<<<split_blocks, 256, 0, s>>>(d_q, n1, d_t, n2, dim, dp, a, b, p.cand_j, splits, qnorm, p.cand_drop);
    }
    CUtensorMap map_a, map_b;
    if ((rc = make_operand_map(h, &map_a, a, n1, kprime))) return rc;
    if ((rc = make_operand_map(h, &map_b, b, n2, kprime, pair ? B_ROWS2 : TILE_N))) return rc;
    cfg.blockDim = dim3(THREADS);
    if (pair) {
        cfg.gridDim = dim3(2 * (unsigned)clusters);
        cfg.dynamicSmemBytes = l2_pair_smem_bytes();
        if (d_dbg) CU_CHECK(h, cudaLaunchKernelEx(&cfg, l2_topk_pair_kernel<true, false>, map_a, map_b, p));
        else CU_CHECK(h, cudaLaunchKernelEx(&cfg, l2_topk_pair_kernel<false, false>, map_a, map_b, p));
    } else {
        cfg.gridDim = dim3(row_tiles, splits); cfg.dynamicSmemBytes = l2_smem_bytes();
        if (d_dbg) CU_CHECK(h, cudaLaunchKernelEx(&cfg, l2_topk_kernel<true>, map_a, map_b, p));
        else CU_CHECK(h, cudaLaunchKernelEx(&cfg, l2_topk_kernel<false>, map_a, map_b, p));
    }
    cfg.gridDim = dim3((unsigned)(((size_t)n1 * 32 + 255) / 256)); cfg.blockDim = dim3(256); cfg.dynamicSmemBytes = 0;
    CU_CHECK(h, cudaLaunchKernelEx(&cfg, l2_refine_kernel, d_q, n1, d_t, n2, dim, (const int32_t *)p.cand_j,
                                   (const float *)p.cand_d, (const float *)p.cand_drop, splits, d_bj, d_bd, d_sj, d_sd,
                                   slack_rel, hdr, ovf_rows));
    if (fp16) {
        cfg.gridDim = dim3((unsigned)h->num_sms * 4); cfg.blockDim = dim3(EX_THREADS);
        CU_CHECK(h, cudaLaunchKernelEx(&cfg, l2_exact_rows_kernel, d_q, (int)n1, d_t, (int)n2, (int)dim, hdr,
                                       (const int32_t *)ovf_rows, (float4 *)(base + o_part), d_bj, d_bd, d_sj, d_sd));
    }
    if (tl) {                                        // debug: phase timeline of cluster 0's leader CTA, us since kernel start
        std::vector<unsigned long long> v(256);
        CU_CHECK(h, cudaMemcpyAsync(v.data(), h->timeline.p, 256 * 8, cudaMemcpyDeviceToHost, s));
        CU_CHECK(h, cudaStreamSynchronize(s));
        fprintf(stderr, "[pgm l2 plan] pair %d max_clusters %d clusters %d row_pairs %d col_tiles %d splits %d tps %d\n", (int)pair,
                h->l2_max_clusters, clusters, row_pairs, col_tiles, splits, tps);
        fprintf(stderr, "[pgm l2 timeline us] sync %.2f pdl %.2f a_ready %.2f |", (v[1] - v[0]) * 1e-3, (v[2] - v[0]) * 1e-3,
                (v[3] - v[0]) * 1e-3);
        for (int t = 0; t < 36 && v[4 + t]; t++)
            fprintf(stderr, " t%d mma %.2f full %.2f epi %.2f |", t, (v[4 + t] - v[0]) * 1e-3, (v[40 + t] - v[0]) * 1e-3,
                    (v[80 + t] - v[0]) * 1e-3);
        fprintf(stderr, " flushed %.2f end %.2f\n", (v[120] - v[0]) * 1e-3, (v[121] - v[0]) * 1e-3);
        // SM cycles (clock64 of the stamping warps; all on one SM): tile-to-tile MMA completion intervals
        fprintf(stderr, "[pgm l2 timeline cycles] whole %llu (%.0f MHz) | full-to-full:", v[128 + 121] - v[128 + 0],
                (double)(v[128 + 121] - v[128 + 0]) / ((v[121] - v[0]) * 1e-3));
        for (int t = 1; t < 36 && v[40 + t]; t++) fprintf(stderr, " %llu", v[128 + 40 + t] - v[128 + 40 + t - 1]);
        fprintf(stderr, "\n");
    }
    h->stats.kernel_launches += fp16 ? 5 : 3;
    h->stats.distance_evals += (int64_t)n1 * n2;
    h->stats.evals_computed += (int64_t)n1 * n2;
    CU_CHECK(h, cudaGetLastError());
    return PGM_OK;
}

__global__ void fill_f32_kernel(float *p, int n, float v) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}

static int l2_check(pgm_handle *h, int32_t n1, int32_t n2, int32_t dim) {
    if (n1 < 0 || n2 < 0 || n1 >= MAX_N || n2 >= MAX_N) return fail(h, PGM_E_INVALID_ARG, "bad sizes");
    if (dim < 1 || dim > 128) return fail(h, PGM_E_INVALID_ARG, "dim must be in 1..128");
    return PGM_OK;
}

extern "C" int pgm_knn2_l2_dev(pgm_handle *h, const float *d_q, int32_t n1, const float *d_t, int32_t n2, int32_t dim,
                               int32_t *d_best_j, float *d_best_d, int32_t *d_second_j, float *d_second_d,
                               float *d_debug_dist) {
    if (!h) return PGM_E_INVALID_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    int rc = l2_check(h, n1, n2, dim);
    if (rc) return rc;
    h->stats = pgm_stats{};
    h->stats_pending = false;
    if (n1 == 0) return PGM_OK;
    CU_CHECK(h, cudaSetDevice(h->device));
    if (n2 == 0) {    // "-1 where absent" for all four arrays, like the host-buffer variant
        if (!d_best_j || !d_best_d || !d_second_j || !d_second_d) return fail(h, PGM_E_INVALID_ARG, "null pointer");
        for (void *o : {(void *)d_best_j, (void *)d_second_j}) CU_CHECK(h, cudaMemsetAsync(o, 0xFF, (size_t)n1 * 4, h->stream));
        const int fg = (n1 + 255) / 256;
        fill_f32_kernel<<<fg, 256, 0, h->stream>>>(d_best_d, n1, -1.0f);
        fill_f32_kernel<<<fg, 256, 0, h->stream>>>(d_second_d, n1, -1.0f);
        CU_CHECK(h, cudaGetLastError());
        return PGM_OK;
    }
    return l2_dev_impl(h, d_q, n1, d_t, n2, dim, d_best_j, d_best_d, d_second_j, d_second_d, d_debug_dist);
}

extern "C" int pgm_l2_last_fallback_rows(pgm_handle *h) {
    if (!h) return -1;
    std::lock_guard<std::mutex> lk(h->mu);
    if (!h->l2_hdr) return -1;
    unsigned v[4] = {0, 0, 0, 0};
    if (cudaSetDevice(h->device) != cudaSuccess) return -1;
    if (cudaMemcpyAsync(v, h->l2_hdr, 16, cudaMemcpyDeviceToHost, h->stream) != cudaSuccess) return -1;
    if (cudaStreamSynchronize(h->stream) != cudaSuccess) return -1;
    return (int)v[h->l2_fallback_word];
}

extern "C" int pgm_knn2_l2(pgm_handle *h, const float *q, int32_t n1, const float *t, int32_t n2, int32_t dim,
                           int32_t *best_j, float *best_d, int32_t *second_j, float *second_d) {
    if (!h) return PGM_E_INVALID_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    int rc = l2_check(h, n1, n2, dim);
    if (rc) return rc;
    h->stats = pgm_stats{};
    h->stats_pending = false;
    if (n1 == 0) return PGM_OK;
    if (n2 == 0) {
        std::fill(best_j, best_j + n1, -1); std::fill(second_j, second_j + n1, -1);
        std::fill(best_d, best_d + n1, -1.f); std::fill(second_d, second_d + n1, -1.f);
        return PGM_OK;
    }
    CU_CHECK(h, cudaSetDevice(h->device));
    cudaStream_t s = h->stream;
    const size_t qb = (size_t)n1 * dim * 4, tb = (size_t)n2 * dim * 4, t_off = align_up(qb, 256);
    if ((rc = ensure_dev(h, h->desc, t_off + tb))) return rc;
    if ((rc = ensure_dev(h, h->out, (size_t)4 * n1 * 4))) return rc;
    if ((rc = ensure_host(h, h->pin_out, (size_t)4 * n1 * 4))) return rc;
    CU_CHECK(h, cudaMemcpyAsync(h->desc.p, q, qb, cudaMemcpyHostToDevice, s));
    CU_CHECK(h, cudaMemcpyAsync((char *)h->desc.p + t_off, t, tb, cudaMemcpyHostToDevice, s));
    h->stats.h2d_bytes += (int64_t)(qb + tb);
    int32_t *o = (int32_t *)h->out.p;
    rc = l2_dev_impl(h, (const float *)h->desc.p, n1, (const float *)((char *)h->desc.p + t_off), n2, dim, o,
                     (float *)(o + n1), o + 2 * (size_t)n1, (float *)(o + 3 * (size_t)n1), nullptr);
    if (rc) return rc;
    CU_CHECK(h, cudaMemcpyAsync(h->pin_out.p, o, (size_t)4 * n1 * 4, cudaMemcpyDeviceToHost, s));
    CU_CHECK(h, cudaStreamSynchronize(s));
    h->stats.host_syncs++;
    h->stats.d2h_bytes += (int64_t)4 * n1 * 4;
    const int32_t *po = (const int32_t *)h->pin_out.p;
    memcpy(best_j, po, (size_t)n1 * 4);
    memcpy(best_d, po + n1, (size_t)n1 * 4);
    memcpy(second_j, po + 2 * (size_t)n1, (size_t)n1 * 4);
    memcpy(second_d, po + 3 * (size_t)n1, (size_t)n1 * 4);
    return PGM_OK;
}

// ---------------------------------------------------------------------------
// float descriptors, many pairs per call (pgm_l2.cuh, "many pairs per launch").  The host plans every chunk first,
// uploads the whole plan in one copy and then only enqueues: five kernels per chunk (seven with the ratio filter).
// ---------------------------------------------------------------------------
constexpr int64_t L2B_MAX_ROWS = 1ll << 22;            // query rows per chunk (with cross-check: both directions)
constexpr int64_t L2B_MAX_CONV_ROWS = 1ll << 22;       // fp16 operand rows per chunk (A' + B')
constexpr int64_t L2B_MAX_CAND_BYTES = 1ll << 30;      // candidate lists: slots x rows x (CAND 8 + EPI_GROUPS 4) bytes

struct L2BChunk {
    int first, n;                  // GEMM pairs: plan[first, first + n)
    int img_first, n_img;          // converted images: imgs[img_first, img_first + n_img)
    int rfirst, rn;                // ratio entry point: filter pairs rplan[rfirst, rfirst + rn)
    int base_off;                  // bases[base_off]: item_base (n + 1), row_base (n + 1), img_base (n_img + 1), fblk_base (rn + 1)
    int32_t items, rows, a_rows, b_rows, clusters, splits, fblocks;
};

struct L2BPlan {
    std::vector<pgm_l2::L2BPair> plan;
    std::vector<pgm_l2::L2BImage> imgs;
    std::vector<pgm_l2::L2RPair> rplan;
    std::vector<int32_t> bases;
    std::vector<L2BChunk> chunks;
};

// Chunks of at most MAX_CHUNK_PAIRS caller pairs, L2B_MAX_ROWS query rows, L2B_MAX_CONV_ROWS operand rows and
// L2B_MAX_CAND_BYTES of candidate lists.  ratio: the filter's pairs too; with cross_check every pair (a, b) brings its
// reversed pair (b, a), whose row best is the column best of (a, b) (the refinement's distances are symmetric).
static void l2b_plan(pgm_handle *h, const int64_t *offs, int32_t n_images, const int32_t *pair_list, int32_t n_pairs,
                     bool ratio, bool cross, L2BPlan &P) {
    using namespace pgm_l2;
    std::vector<int32_t> qpos(n_images), tpos(n_images), stamp_q(n_images, -1), stamp_t(n_images, -1);
    int attempt = 0;
    int64_t out_base = 0;
    for (int p = 0; p < n_pairs;) {
        int cap = MAX_CHUNK_PAIRS;
        for (;;) {
            attempt++;
            L2BChunk c{(int)P.plan.size(), 0, (int)P.imgs.size(), 0, (int)P.rplan.size(), 0, (int)P.bases.size(), 0, 0, 0, 0, 0, 0, 0};
            int64_t conv = 0, ob = out_base;
            int q = p, taken = 0;
            auto image = [&](int im, bool train) {                 // operand row of image im in its role (added once)
                std::vector<int32_t> &pos = train ? tpos : qpos, &st = train ? stamp_t : stamp_q;
                if (st[im] != attempt) {
                    st[im] = attempt;
                    const int32_t n = (int32_t)(offs[im + 1] - offs[im]);
                    int32_t &rows = train ? c.b_rows : c.a_rows;
                    pos[im] = rows;
                    P.imgs.push_back(L2BImage{offs[im], rows, n, train ? 1 : 0, 0});
                    rows += n; conv += n;
                }
                return pos[im];
            };
            auto gemm_pair = [&](int a, int b, int64_t out_row) {
                L2BPair r{};
                r.q_row = offs[a]; r.t_row = offs[b];
                r.n1 = (int32_t)(offs[a + 1] - offs[a]); r.n2 = (int32_t)(offs[b + 1] - offs[b]);
                r.a_row = image(a, false);
                r.b_row = r.n2 > 0 ? image(b, true) : 0;
                r.row0 = c.rows; r.out_row = ratio ? c.rows : out_row;
                r.item0 = c.items; r.col_tiles = (r.n2 + TILE_N2 - 1) / TILE_N2;
                c.items += (r.n1 + 2 * TILE_M - 1) / (2 * TILE_M) * r.col_tiles;
                c.rows += r.n1;
                P.plan.push_back(r);
                c.n++;
                return r.row0;
            };
            for (; q < n_pairs && taken < cap; q++) {
                const int a = pair_list[2 * q], b = pair_list[2 * q + 1];
                const int64_t n1 = offs[a + 1] - offs[a], n2 = offs[b + 1] - offs[b];
                const bool run = n1 > 0 && (!ratio || n2 > 0);       // the ratio filter keeps nothing without train rows
                if (run) {
                    const bool rev = ratio && cross;
                    const int64_t rows = n1 + (rev ? n2 : 0);
                    const int64_t cv = (stamp_q[a] == attempt ? 0 : n1) + (stamp_t[b] == attempt ? 0 : n2) +
                                       (rev ? (stamp_q[b] == attempt || a == b ? 0 : n2) + (stamp_t[a] == attempt || a == b ? 0 : n1) : 0);
                    if (taken > 0 && (c.rows + rows > L2B_MAX_ROWS || conv + cv > L2B_MAX_CONV_ROWS)) break;
                    const int32_t row0 = gemm_pair(a, b, ob);
                    const int32_t rrow0 = rev ? gemm_pair(b, a, 0) : 0;
                    if (ratio) {
                        P.rplan.push_back(L2RPair{ob, row0, rrow0, (int32_t)n1, (int32_t)n2, q, 0});
                        c.rn++;
                    }
                    taken++;
                }
                ob += n1;
            }
            // candidate slots: the most segments any row pair is cut into (as in l2_dev_impl)
            c.clusters = std::max(1, std::min(h->l2_max_clusters, c.items));
            c.splits = 1;
            for (int k = c.first; k < c.first + c.n; k++) {
                const L2BPair &r = P.plan[k];
                if (r.col_tiles == 0) continue;
                for (int32_t x0 = r.item0; x0 < r.item0 + (r.n1 + 2 * TILE_M - 1) / (2 * TILE_M) * r.col_tiles; x0 += r.col_tiles) {
                    const int64_t x1 = x0 + r.col_tiles - 1;
                    const int k0 = (int)(((int64_t)(x0 + 1) * c.clusters - 1) / c.items), k1 = (int)(((x1 + 1) * c.clusters - 1) / c.items);
                    c.splits = std::max(c.splits, k1 - k0 + 1);
                }
            }
            if (taken > 1 && (int64_t)c.splits * c.rows * (CAND * 8 + EPI_GROUPS * 4) > L2B_MAX_CAND_BYTES) {
                P.plan.resize(c.first); P.imgs.resize(c.img_first); P.rplan.resize(c.rfirst);
                cap = taken / 2;
                continue;
            }
            c.n_img = (int)P.imgs.size() - c.img_first;
            P.bases.resize(P.bases.size() + 2 * (size_t)(c.n + 1) + (size_t)(c.n_img + 1) + (size_t)(c.rn + 1));
            int32_t *ib = P.bases.data() + c.base_off, *rb = ib + c.n + 1, *gb = rb + c.n + 1, *fb = gb + c.n_img + 1;
            for (int k = 0; k < c.n; k++) { ib[k] = P.plan[c.first + k].item0; rb[k] = P.plan[c.first + k].row0; }
            ib[c.n] = c.items; rb[c.n] = c.rows;
            int32_t g = 0;
            for (int k = 0; k < c.n_img; k++) { gb[k] = g; g += P.imgs[c.img_first + k].n; }
            gb[c.n_img] = g;
            for (int k = 0; k < c.rn; k++) { fb[k] = c.fblocks; c.fblocks += (P.rplan[c.rfirst + k].n1 + L2F_THREADS - 1) / L2F_THREADS; }
            fb[c.rn] = c.fblocks;
            if (c.n > 0) P.chunks.push_back(c);
            p = q;
            out_base = ob;
            break;
        }
    }
}

// Enqueues the chunks of a plan.  d_bj.. : knn2 results (the caller's arrays, or the per-chunk scratch with the ratio
// filter, which then writes the triples).
static int l2b_run(pgm_handle *h, const float *d_all, int32_t dim, int32_t n_pairs, const L2BPlan &P, bool ratio_mode,
                   float ratio, bool cross, float max_sq_dist, int32_t *d_bj, float *d_bd, int32_t *d_sj, float *d_sd,
                   int32_t *d_out_qi, int32_t *d_out_tj, float *d_out_dist, int64_t capacity, int32_t *out_counts) {
    using namespace pgm_l2;
    cudaStream_t s = h->stream;
    const int dp = (dim + CHUNK_K - 1) / CHUNK_K * CHUNK_K, dpc = dp / CHUNK_K, kprime = dp + CHUNK_K;
    int64_t max_rows = 1, max_a = 1, max_b = 1, max_cand = 1, max_fb = 1;
    for (const L2BChunk &c : P.chunks) {
        max_rows = std::max<int64_t>(max_rows, c.rows); max_a = std::max<int64_t>(max_a, c.a_rows);
        max_b = std::max<int64_t>(max_b, c.b_rows); max_cand = std::max<int64_t>(max_cand, (int64_t)c.splits * c.rows);
        max_fb = std::max<int64_t>(max_fb, c.fblocks);
    }
    // h->misc: plan | images | filter pairs | bases | counts || A' | B' | |q|^2 | cand_j | cand_d | cand_drop | flagged rows |
    // fallback partials | knn2 scratch (ratio) | kept-row flags | block counts
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + std::max<size_t>(bytes, 1), 1024); return o; };
    const size_t o_plan = take(sizeof(L2BPair) * P.plan.size()), o_img = take(sizeof(L2BImage) * P.imgs.size());
    const size_t o_rplan = take(sizeof(L2RPair) * P.rplan.size()), o_bases = take(4 * P.bases.size());
    const size_t o_counts = take(4 * (size_t)n_pairs), upload = o_counts;
    const size_t o_a = take((size_t)max_a * kprime * 2), o_b = take((size_t)max_b * kprime * 2), o_qn = take((size_t)max_a * 4);
    const size_t o_cj = take((size_t)max_cand * CAND * 4), o_cd = take((size_t)max_cand * CAND * 4);
    const size_t o_drop = take((size_t)max_cand * EPI_GROUPS * 4), o_ovf = take((size_t)max_rows * 4);
    const size_t o_part = take((size_t)max_rows * EX_MAX_SLICES_PER_ROW * 16);
    const size_t o_knn = take(ratio_mode ? (size_t)max_rows * 16 : 0), o_keep = take(ratio_mode ? (size_t)max_rows * 4 : 0);
    const size_t o_bcnt = take(ratio_mode ? (size_t)max_fb * 4 : 0);
    int rc = ensure_dev(h, h->misc, off);
    if (rc) return rc;
    if ((rc = ensure_host(h, h->pin_in, upload + 4 * (size_t)n_pairs))) return rc;      // the plan, then the counts read-back
    if (h->l2_state.cap < 16) {
        if ((rc = ensure_dev(h, h->l2_state, 16))) return rc;
        CU_CHECK(h, cudaMemsetAsync(h->l2_state.p, 0, h->l2_state.cap, s));
    }
    unsigned *hdr = (unsigned *)h->l2_state.p;
    CU_CHECK(h, cudaStreamSynchronize(s));                 // the staging buffer may still feed an earlier call's copy
    char *pin = (char *)h->pin_in.p, *dev = (char *)h->misc.p;
    memcpy(pin + o_plan, P.plan.data(), sizeof(L2BPair) * P.plan.size());
    memcpy(pin + o_img, P.imgs.data(), sizeof(L2BImage) * P.imgs.size());
    memcpy(pin + o_rplan, P.rplan.data(), sizeof(L2RPair) * P.rplan.size());
    memcpy(pin + o_bases, P.bases.data(), 4 * P.bases.size());
    CU_CHECK(h, cudaMemcpyAsync(dev, pin, upload, cudaMemcpyHostToDevice, s));
    CU_CHECK(h, cudaMemsetAsync(hdr + 3, 0, 4, s));       // flagged rows of this call, over all chunks
    h->l2_hdr = hdr;
    h->l2_fallback_word = 3;
    if (ratio_mode) CU_CHECK(h, cudaMemsetAsync(dev + o_counts, 0, 4 * (size_t)n_pairs, s));
    const L2BPair *d_plan = (const L2BPair *)(dev + o_plan);
    const L2BImage *d_img = (const L2BImage *)(dev + o_img);
    const L2RPair *d_rplan = (const L2RPair *)(dev + o_rplan);
    const int32_t *d_bases = (const int32_t *)(dev + o_bases);
    __half *a = (__half *)(dev + o_a), *b = (__half *)(dev + o_b);
    float *qnorm = (float *)(dev + o_qn);
    int32_t *cand_j = (int32_t *)(dev + o_cj), *ovf = (int32_t *)(dev + o_ovf);
    float *cand_d = (float *)(dev + o_cd), *cand_drop = (float *)(dev + o_drop);
    if (ratio_mode) {
        d_bj = (int32_t *)(dev + o_knn); d_bd = (float *)(d_bj + max_rows);
        d_sj = (int32_t *)(d_bd + max_rows); d_sd = (float *)(d_sj + max_rows);
    }
    // the band of l2_dev_impl's fp16 ranking
    const float slack_rel = 0.00244140625f;
    L2Params p{};
    p.dpc = dpc; p.key_mask = 0x7FFFFFE0u;
    p.band_rel = 0.5f * slack_rel;
    p.band_abs_sqrt = 4.8828125e-7f * sqrtf((float)dp);
    p.band_abs_const = 2.44140625e-4f;
    p.absmax_bits = hdr; p.qnorm = qnorm; p.cand_j = cand_j; p.cand_d = cand_d; p.cand_drop = cand_drop;
    cudaLaunchAttribute pdl{};
    pdl.id = cudaLaunchAttributeProgrammaticStreamSerialization;
    pdl.val.programmaticStreamSerializationAllowed = 1;
    const float rr = ratio * ratio;                        // Lowe's ratio on Euclidean distances, on squared ones
    for (const L2BChunk &c : P.chunks) {
        const int32_t *ib = d_bases + c.base_off, *rb = ib + c.n + 1, *gb = rb + c.n + 1, *fb = gb + c.n_img + 1;
        const L2BPair *cp = d_plan + c.first;
        const size_t n_cand = (size_t)c.splits * c.rows;
        int64_t conv_floats = 0;
        for (int k = 0; k < c.n_img; k++) conv_floats += (int64_t)P.imgs[c.img_first + k].n * dim;
        const int pb = (int)std::min<int64_t>((int64_t)h->num_sms * 8, (conv_floats + (int64_t)n_cand * CAND + 4095) / 4096 + 1);
        l2b_prep_kernel<<<pb, 256, 0, s>>>(d_all, dim, d_img + c.img_first, c.n_img, hdr, cand_j, n_cand * CAND, cand_drop,
                                           n_cand * EPI_GROUPS);
        cudaLaunchConfig_t cfg{};
        cfg.stream = s; cfg.attrs = &pdl; cfg.numAttrs = 1;
        cfg.gridDim = dim3((unsigned)(((int64_t)(c.a_rows + c.b_rows) * 32 + 255) / 256)); cfg.blockDim = dim3(256);
        CU_CHECK(h, cudaLaunchKernelEx(&cfg, l2b_split16_kernel, d_all, (int)dim, dp, d_img + c.img_first, gb, c.n_img, a, b,
                                       (const unsigned *)hdr, qnorm));
        int launches = 4;
        if (c.items > 0) {
            CUtensorMap map_a, map_b;
            if ((rc = make_operand_map(h, &map_a, a, std::max(c.a_rows, 1), kprime))) return rc;
            if ((rc = make_operand_map(h, &map_b, b, std::max(c.b_rows, 1), kprime, B_ROWS2))) return rc;
            p.items = c.items; p.bpairs = cp; p.item_base = ib; p.n_pairs = c.n; p.rows = c.rows;
            cfg.gridDim = dim3(2 * (unsigned)c.clusters); cfg.blockDim = dim3(THREADS);
            cfg.dynamicSmemBytes = l2_pair_smem_bytes();
            CU_CHECK(h, cudaLaunchKernelEx(&cfg, l2_topk_pair_kernel<false, true>, map_a, map_b, p));
            launches++;
        }
        cfg.gridDim = dim3((unsigned)(((int64_t)c.rows * 32 + 255) / 256)); cfg.blockDim = dim3(256); cfg.dynamicSmemBytes = 0;
        CU_CHECK(h, cudaLaunchKernelEx(&cfg, l2b_refine_kernel, d_all, (int)dim, cp, rb, c.n, (int)c.rows, (const int32_t *)cand_j,
                                       (const float *)cand_d, (const float *)cand_drop, (int)c.splits, d_bj, d_bd, d_sj, d_sd,
                                       slack_rel, hdr, ovf));
        cfg.gridDim = dim3((unsigned)h->num_sms * 4); cfg.blockDim = dim3(EX_THREADS);
        CU_CHECK(h, cudaLaunchKernelEx(&cfg, l2b_exact_rows_kernel, d_all, (int)dim, cp, rb, c.n, (int)c.rows, hdr,
                                       (const int32_t *)ovf, (float4 *)(dev + o_part), d_bj, d_bd, d_sj, d_sd));
        if (ratio_mode && c.rn > 0) {
            int32_t *keep = (int32_t *)(dev + o_keep), *bcnt = (int32_t *)(dev + o_bcnt);
            l2b_filter_kernel<<<c.fblocks, L2F_THREADS, 0, s>>>(d_rplan + c.rfirst, fb, c.rn, c.rows, d_bj, d_bd, d_sd, ratio, rr,
                                                                cross ? 1 : 0, max_sq_dist, keep, bcnt);
            l2b_scatter_kernel<<<c.fblocks, L2F_THREADS, 0, s>>>(d_rplan + c.rfirst, fb, c.rn, keep, d_bj, d_bd, bcnt, capacity,
                                                                 d_out_qi, d_out_tj, d_out_dist, (int32_t *)(dev + o_counts));
            launches += 2;
        }
        CU_CHECK(h, cudaGetLastError());
        h->stats.kernel_launches += launches;
    }
    h->stats.host_syncs += 1;
    if (ratio_mode) {
        CU_CHECK(h, cudaMemcpyAsync(pin + o_counts, dev + o_counts, 4 * (size_t)n_pairs, cudaMemcpyDeviceToHost, s));
        CU_CHECK(h, cudaStreamSynchronize(s));
        memcpy(out_counts, pin + o_counts, 4 * (size_t)n_pairs);
        h->stats.host_syncs += 1;
        for (int q = 0; q < n_pairs; q++) h->stats.matched += out_counts[q];
    }
    return PGM_OK;
}

// argument checks shared by both batch entry points; *evals = sum of n1 n2, *rows = sum of n1
static int l2b_check(pgm_handle *h, const int64_t *image_offsets, int32_t n_images, const int32_t *pair_list, int32_t n_pairs,
                     int32_t dim, int64_t *evals, int64_t *rows) {
    if (dim < 1 || dim > 128) return fail(h, PGM_E_INVALID_ARG, "dim must be in 1..128");
    *evals = 0; *rows = 0;
    for (int p = 0; p < n_pairs; p++) {
        const int a = pair_list[2 * p], b = pair_list[2 * p + 1];
        if (a < 0 || a >= n_images || b < 0 || b >= n_images) return fail(h, PGM_E_INVALID_ARG, "pair index out of range");
        const int64_t n1 = image_offsets[a + 1] - image_offsets[a], n2 = image_offsets[b + 1] - image_offsets[b];
        if (n1 < 0 || n2 < 0 || n1 >= MAX_N || n2 >= MAX_N || image_offsets[a] < 0 || image_offsets[b] < 0)
            return fail(h, PGM_E_INVALID_ARG, "bad image sizes");
        *rows += n1;
        *evals += n1 * n2;
    }
    return PGM_OK;
}

extern "C" int pgm_knn2_l2_pairs_batch_dev(pgm_handle *h, const float *d_all_desc, const int64_t *image_offsets, int32_t n_images,
                                           const int32_t *pair_list, int32_t n_pairs, int32_t dim, int32_t *d_best_j,
                                           float *d_best_d, int32_t *d_second_j, float *d_second_d, int64_t capacity) {
    if (!h || n_pairs < 0 || n_images < 0 || (n_pairs > 0 && (!image_offsets || !pair_list))) return PGM_E_INVALID_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    h->stats = pgm_stats{};
    h->stats_pending = false;
    int64_t evals, rows;
    int rc = l2b_check(h, image_offsets, n_images, pair_list, n_pairs, dim, &evals, &rows);
    if (rc) return rc;
    if (capacity < rows) return fail(h, PGM_E_CAPACITY, "capacity < sum of query sizes");
    if (n_pairs == 0 || rows == 0) return PGM_OK;
    if (!d_all_desc || !d_best_j || !d_best_d || !d_second_j || !d_second_d) return fail(h, PGM_E_INVALID_ARG, "null pointer");
    CU_CHECK(h, cudaSetDevice(h->device));
    if ((rc = l2_setup(h))) return rc;
    L2BPlan P;
    l2b_plan(h, image_offsets, n_images, pair_list, n_pairs, false, false, P);
    if ((rc = l2b_run(h, d_all_desc, dim, n_pairs, P, false, 0.f, false, -1.f, d_best_j, d_best_d, d_second_j, d_second_d,
                      nullptr, nullptr, nullptr, capacity, nullptr)))
        return rc;
    h->stats.pairs = n_pairs;
    h->stats.distance_evals = evals;
    h->stats.evals_computed = evals;
    return PGM_OK;
}

extern "C" int pgm_match_l2_ratio_crosscheck_pairs_batch_dev(pgm_handle *h, const float *d_all_desc, const int64_t *image_offsets,
                                                             int32_t n_images, const int32_t *pair_list, int32_t n_pairs,
                                                             int32_t dim, float ratio, int32_t cross_check, float max_sq_dist,
                                                             int32_t *d_out_qi, int32_t *d_out_tj, float *d_out_dist,
                                                             int64_t capacity, int32_t *out_counts) {
    if (!h || !out_counts || n_pairs < 0 || n_images < 0 || (n_pairs > 0 && (!image_offsets || !pair_list))) return PGM_E_INVALID_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    h->stats = pgm_stats{};
    h->stats_pending = false;
    int64_t evals, rows;
    int rc = l2b_check(h, image_offsets, n_images, pair_list, n_pairs, dim, &evals, &rows);
    if (rc) return rc;
    if (capacity < rows) return fail(h, PGM_E_CAPACITY, "capacity < sum of query sizes");
    if (n_pairs == 0) return PGM_OK;
    if (!d_all_desc || !d_out_qi || !d_out_tj || !d_out_dist) return fail(h, PGM_E_INVALID_ARG, "null pointer");
    CU_CHECK(h, cudaSetDevice(h->device));
    if ((rc = l2_setup(h))) return rc;
    const bool cross = cross_check != 0;
    L2BPlan P;
    l2b_plan(h, image_offsets, n_images, pair_list, n_pairs, true, cross, P);
    if ((rc = l2b_run(h, d_all_desc, dim, n_pairs, P, true, ratio, cross, max_sq_dist, nullptr, nullptr, nullptr, nullptr,
                      d_out_qi, d_out_tj, d_out_dist, capacity, out_counts)))
        return rc;
    h->stats.pairs = n_pairs;
    h->stats.distance_evals = evals;
    h->stats.evals_computed = cross ? 2 * evals : evals;    // the reversed pairs' top-2 pass gives the column best
    return PGM_OK;
}

// ---------------------------------------------------------------------------
// keypoint producer: FAST-12, BRIEF, NMS (pgm_detect.cuh)
// ---------------------------------------------------------------------------
extern "C" int pgm_fast_detect(pgm_handle *h, const float *gray, int32_t width, int32_t height, float threshold,
                               uint32_t flags, int32_t *out_xy, int32_t *out_score, int32_t capacity,
                               int32_t *out_count) {
    using namespace pgm_det;
    if (!h || !out_count) return PGM_E_INVALID_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    if (!gray || width < 1 || height < 1 || width > 65535 || height > 65535)
        return fail(h, PGM_E_INVALID_ARG, "bad image");     // MatrixDimensions are ushort upstream
    h->stats = pgm_stats{};
    h->stats_pending = false;
    CU_CHECK(h, cudaSetDevice(h->device));
    cudaStream_t s = h->stream;
    const size_t npx = (size_t)width * height;
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return o; };
    const size_t o_img = take(npx * 4), o_sc = take(npx), o_cnt = take((size_t)height * 4), o_off = take((size_t)(height + 1) * 4);
    int rc = ensure_dev(h, h->misc, off);
    if (rc) return rc;
    char *base = (char *)h->misc.p;
    float *d_img = (float *)(base + o_img);
    uint8_t *d_sc = (uint8_t *)(base + o_sc);
    int32_t *d_cnt = (int32_t *)(base + o_cnt), *d_off = (int32_t *)(base + o_off);
    CU_CHECK(h, cudaMemcpyAsync(d_img, gray, npx * 4, cudaMemcpyHostToDevice, s));
    dim3 blk(32, 8), grd((width + 31) / 32, (height + 7) / 8);
    if (flags & PGM_FLAG_PYTHON_GENERATION) fast_score_kernel<1><<<grd, blk, 0, s>>>(d_img, width, height, threshold, d_sc);
    else fast_score_kernel<0><<<grd, blk, 0, s>>>(d_img, width, height, threshold, d_sc);
    row_count_kernel<<<height, 128, 0, s>>>(d_sc, width, d_cnt);
    scan_kernel<<<1, 1024, 0, s>>>(d_cnt, height, d_off);
    if ((rc = ensure_host(h, h->pin_out, 64))) return rc;
    CU_CHECK(h, cudaMemcpyAsync(h->pin_out.p, d_off + height, 4, cudaMemcpyDeviceToHost, s));
    CU_CHECK(h, cudaStreamSynchronize(s));
    const int32_t total = *(int32_t *)h->pin_out.p;
    *out_count = total;
    h->stats.kernel_launches += 3; h->stats.host_syncs++; h->stats.h2d_bytes += (int64_t)npx * 4;
    if (total > capacity) return fail(h, PGM_E_CAPACITY, "more keypoints than capacity (out_count holds the number found)");
    if (total == 0) return PGM_OK;
    if ((rc = ensure_dev(h, h->out, (size_t)total * 12))) return rc;
    if ((rc = ensure_host(h, h->pin_out, (size_t)total * 12))) return rc;
    int32_t *d_xy = (int32_t *)h->out.p, *d_s = d_xy + 2 * (size_t)total;
    emit_kernel<<<(height + 3) / 4, 128, 0, s>>>(d_sc, width, height, d_off, total, d_xy, d_s);
    CU_CHECK(h, cudaMemcpyAsync(h->pin_out.p, h->out.p, (size_t)total * 12, cudaMemcpyDeviceToHost, s));
    CU_CHECK(h, cudaStreamSynchronize(s));
    memcpy(out_xy, h->pin_out.p, (size_t)total * 8);
    memcpy(out_score, (char *)h->pin_out.p + (size_t)total * 8, (size_t)total * 4);
    h->stats.kernel_launches += 1; h->stats.host_syncs++; h->stats.d2h_bytes += (int64_t)total * 12;
    CU_CHECK(h, cudaGetLastError());
    return PGM_OK;
}

extern "C" int pgm_brief_describe(pgm_handle *h, const float *gray, int32_t width, int32_t height, const int32_t *xy,
                                  int32_t n, const int32_t *pairs, int32_t n_pairs, int32_t stride_bytes,
                                  uint32_t flags, uint8_t *out_desc) {
    using namespace pgm_det;
    if (!h) return PGM_E_INVALID_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    int rc = check_format(h, n_pairs, stride_bytes);       // desc_bits == NumGaussianPairs
    if (rc) return rc;
    if (!gray || width < 1 || height < 1 || n < 0 || !pairs) return fail(h, PGM_E_INVALID_ARG, "bad arguments");
    h->stats = pgm_stats{};
    h->stats_pending = false;
    if (n == 0) return PGM_OK;
    CU_CHECK(h, cudaSetDevice(h->device));
    cudaStream_t s = h->stream;
    const size_t npx = (size_t)width * height;
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return o; };
    const size_t o_img = take(npx * 4), o_xy = take((size_t)n * 8), o_pr = take((size_t)n_pairs * 16), o_d = take((size_t)n * stride_bytes);
    if ((rc = ensure_dev(h, h->misc, off))) return rc;
    char *base = (char *)h->misc.p;
    CU_CHECK(h, cudaMemcpyAsync(base + o_img, gray, npx * 4, cudaMemcpyHostToDevice, s));
    CU_CHECK(h, cudaMemcpyAsync(base + o_xy, xy, (size_t)n * 8, cudaMemcpyHostToDevice, s));
    CU_CHECK(h, cudaMemcpyAsync(base + o_pr, pairs, (size_t)n_pairs * 16, cudaMemcpyHostToDevice, s));
    const int warps = 4, sw = stride_bytes / 4;
    brief_kernel<<<(n + warps - 1) / warps, warps * 32, warps * sw * 4, s>>>((const float *)(base + o_img), width, height,
                                                                         (const int32_t *)(base + o_xy), n,
                                                                         (const int32_t *)(base + o_pr), n_pairs, sw,
                                                                         (flags & PGM_FLAG_PYTHON_GENERATION) ? 1 : 0,
                                                                         (uint32_t *)(base + o_d));
    CU_CHECK(h, cudaMemcpyAsync(out_desc, base + o_d, (size_t)n * stride_bytes, cudaMemcpyDeviceToHost, s));
    CU_CHECK(h, cudaStreamSynchronize(s));
    h->stats.kernel_launches += 1; h->stats.host_syncs++;
    h->stats.h2d_bytes += (int64_t)(npx * 4 + (size_t)n * 8); h->stats.d2h_bytes += (int64_t)n * stride_bytes;
    CU_CHECK(h, cudaGetLastError());
    return PGM_OK;
}

// NMS on device-resident keypoints (d_xy int32[n][2], d_sc int32[n]); `hxy` = the same coordinates on the host
// (bounding box for the cell grid).  Scratch comes from h->misc (and h->out2 for the radix sorts), so the inputs
// must live elsewhere.  On return *d_kept_out points into h->misc (valid until its next use) and *count is set.
static int nms_core(pgm_handle *h, const int32_t *d_xy, const int32_t *d_sc, const int32_t *hxy, int32_t n, int32_t radius,
                    int32_t **d_kept_out, int32_t *count) {
    using namespace pgm_det;
    cudaStream_t s = h->stream;
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return o; };
    const size_t o_rk = take((size_t)n * 4), o_or = take((size_t)n * 4);
    const size_t o_s0 = take(n), o_s1 = take(n), o_kept = take((size_t)n * 4), o_cnt = take(16);
    const size_t o_k0 = take((size_t)n * 8), o_k1 = take((size_t)n * 8), o_v0 = take((size_t)n * 4), o_v1 = take((size_t)n * 4);
    int rc = ensure_dev(h, h->misc, off);
    if (rc) return rc;
    if ((rc = ensure_host(h, h->pin_meta, 64))) return rc;
    char *base = (char *)h->misc.p;
    int32_t *d_rk = (int32_t *)(base + o_rk);
    int32_t *d_or = (int32_t *)(base + o_or), *d_kept = (int32_t *)(base + o_kept), *d_cnt = (int32_t *)(base + o_cnt);
    uint8_t *st[2] = {(uint8_t *)(base + o_s0), (uint8_t *)(base + o_s1)};
    CU_CHECK(h, cudaMemsetAsync(st[0], 0, n, s));
    const int blocks = (n + 255) / 256;
    int32_t *h_cnt = (int32_t *)h->pin_meta.p;
    const long long r2 = (long long)radius * radius;

    // Spatial binning pays once the all-pairs scans (n^2 per round) outweigh two radix sorts.  PGM_NMS_MODE=dense
    // or =binned forces one form (tests run both); the answers are identical.
    const int cs = std::max(radius, 1);
    long long minx = hxy[0], miny = hxy[1], maxx = hxy[0], maxy = hxy[1];
    for (int i = 1; i < n; i++) {
        minx = std::min<long long>(minx, hxy[2 * i]); maxx = std::max<long long>(maxx, hxy[2 * i]);
        miny = std::min<long long>(miny, hxy[2 * i + 1]); maxy = std::max<long long>(maxy, hxy[2 * i + 1]);
    }
    const long long ncx = (maxx - minx) / cs + 1, ncy = (maxy - miny) / cs + 1;   // each <= 2^32
    bool binned = n >= 1024 && (ncx >= 8 || ncy >= 8) && ncx * (double)ncy >= 64.0;  // else 3 x 3 cells hold most keypoints
    if (const char *mode = getenv("PGM_NMS_MODE")) {
        if (!strcmp(mode, "dense")) binned = false;
        else if (!strcmp(mode, "binned")) binned = true;
    }
    if (!binned) {
        nms_rank_kernel<<<blocks, 256, 0, s>>>(d_sc, n, d_rk, d_or);
        h->stats.kernel_launches += 1;
        for (int round = 0;; round++) {
            CU_CHECK(h, cudaMemsetAsync(d_cnt, 0, 4, s));
            nms_round_kernel<<<blocks, 256, 0, s>>>(d_xy, d_rk, n, r2, st[round & 1], st[(round + 1) & 1], d_cnt);
            CU_CHECK(h, cudaMemcpyAsync(h_cnt, d_cnt, 4, cudaMemcpyDeviceToHost, s));
            CU_CHECK(h, cudaStreamSynchronize(s));
            h->stats.kernel_launches += 1; h->stats.host_syncs++; h->stats.rounds++;
            if (*h_cnt == 0) {
                nms_emit_kernel<<<1, 1024, 0, s>>>(d_or, st[(round + 1) & 1], n, d_kept, d_cnt);
                break;
            }
            if (round > n + 2) return fail(h, PGM_E_CUDA, "NMS failed to converge (internal error)");
        }
    } else {
        // order: ascending sort of (inverted score << 32 | index) = stable order by score descending
        unsigned long long *k_in = (unsigned long long *)(base + o_k0), *k_out = (unsigned long long *)(base + o_k1);
        int32_t *v_in = (int32_t *)(base + o_v0), *d_cidx = (int32_t *)(base + o_v1);
        size_t tmp_bytes = 0, tmp2 = 0;
        CU_CHECK(h, cub::DeviceRadixSort::SortKeys(nullptr, tmp_bytes, k_in, k_out, n, 0, 64, s));
        CU_CHECK(h, cub::DeviceRadixSort::SortPairs(nullptr, tmp2, k_in, k_out, v_in, d_cidx, n, 0, 64, s));
        tmp_bytes = std::max(tmp_bytes, tmp2);
        if ((rc = ensure_dev(h, h->out2, tmp_bytes))) return rc;
        nms_score_key_kernel<<<blocks, 256, 0, s>>>(d_sc, n, k_in);
        CU_CHECK(h, cub::DeviceRadixSort::SortKeys(h->out2.p, tmp_bytes, k_in, k_out, n, 0, 64, s));
        nms_order_from_keys_kernel<<<blocks, 256, 0, s>>>(k_out, n, d_or, d_rk);
        // cells: keypoints sorted by cell id
        nms_cell_kernel<<<blocks, 256, 0, s>>>(d_xy, n, cs, (int)minx, (int)miny, ncx, k_in, v_in);
        int cell_bits = 1;
        while (cell_bits < 64 && ((unsigned long long)ncx * (unsigned long long)ncy - 1) >> cell_bits) cell_bits++;
        CU_CHECK(h, cub::DeviceRadixSort::SortPairs(h->out2.p, tmp_bytes, k_in, k_out, v_in, d_cidx, n, 0, cell_bits, s));
        h->stats.kernel_launches += 3;
        for (int round = 0;; round++) {
            CU_CHECK(h, cudaMemsetAsync(d_cnt, 0, 4, s));
            nms_round_binned_kernel<<<blocks, 256, 0, s>>>(d_xy, d_rk, n, r2, cs, (int)minx, (int)miny, ncx, ncy, k_out,
                                                           d_cidx, st[round & 1], st[(round + 1) & 1], d_cnt);
            CU_CHECK(h, cudaMemcpyAsync(h_cnt, d_cnt, 4, cudaMemcpyDeviceToHost, s));
            CU_CHECK(h, cudaStreamSynchronize(s));
            h->stats.kernel_launches += 1; h->stats.host_syncs++; h->stats.rounds++;
            if (*h_cnt == 0) {
                nms_emit_kernel<<<1, 1024, 0, s>>>(d_or, st[(round + 1) & 1], n, d_kept, d_cnt);
                break;
            }
            if (round > n + 2) return fail(h, PGM_E_CUDA, "NMS failed to converge (internal error)");
        }
    }
    CU_CHECK(h, cudaMemcpyAsync(h_cnt, d_cnt, 4, cudaMemcpyDeviceToHost, s));
    CU_CHECK(h, cudaStreamSynchronize(s));
    *count = h_cnt[0];
    *d_kept_out = d_kept;
    h->stats.kernel_launches += 1; h->stats.host_syncs++;
    CU_CHECK(h, cudaGetLastError());
    return PGM_OK;
}

extern "C" int pgm_nms(pgm_handle *h, const int32_t *xy, const int32_t *score, int32_t n, int32_t radius,
                       int32_t *out_kept, int32_t *out_count) {
    if (!h || !out_count) return PGM_E_INVALID_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    if (n < 0 || radius < 0 || (n > 0 && (!xy || !score || !out_kept))) return fail(h, PGM_E_INVALID_ARG, "bad arguments");
    h->stats = pgm_stats{};
    h->stats_pending = false;
    *out_count = 0;
    if (n == 0) return PGM_OK;
    CU_CHECK(h, cudaSetDevice(h->device));
    cudaStream_t s = h->stream;
    int rc = ensure_dev(h, h->desc, (size_t)n * 12);
    if (rc) return rc;
    int32_t *d_xy = (int32_t *)h->desc.p, *d_sc = d_xy + 2 * (size_t)n;
    CU_CHECK(h, cudaMemcpyAsync(d_xy, xy, (size_t)n * 8, cudaMemcpyHostToDevice, s));
    CU_CHECK(h, cudaMemcpyAsync(d_sc, score, (size_t)n * 4, cudaMemcpyHostToDevice, s));
    int32_t *d_kept = nullptr, cnt = 0;
    if ((rc = nms_core(h, d_xy, d_sc, xy, n, radius, &d_kept, &cnt))) return rc;
    if ((rc = ensure_host(h, h->pin_out, (size_t)n * 4 + 64))) return rc;
    CU_CHECK(h, cudaMemcpyAsync(h->pin_out.p, d_kept, (size_t)cnt * 4, cudaMemcpyDeviceToHost, s));
    CU_CHECK(h, cudaStreamSynchronize(s));
    memcpy(out_kept, h->pin_out.p, (size_t)cnt * 4);
    *out_count = cnt;
    h->stats.host_syncs++;
    return PGM_OK;
}

// ---------------------------------------------------------------------------
// the producer chain on a device-resident image: FAST-12 -> (NMS) -> BRIEF, descriptors never leave the GPU
// ---------------------------------------------------------------------------
extern "C" int pgm_detect_describe_dev(pgm_handle *h, const float *d_gray, int32_t width, int32_t height, float threshold,
                                       int32_t nms_radius, const int32_t *pairs, int32_t n_pairs, int32_t stride_bytes,
                                       uint32_t flags, int32_t *d_out_xy, int32_t *d_out_score, uint8_t *d_out_desc,
                                       int32_t capacity, int32_t *out_count) {
    using namespace pgm_det;
    if (!h || !out_count) return PGM_E_INVALID_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    int rc = check_format(h, n_pairs, stride_bytes);       // desc_bits == NumGaussianPairs
    if (rc) return rc;
    if (!d_gray || width < 1 || height < 1 || width > 65535 || height > 65535 || !pairs || capacity < 0 ||
        (capacity > 0 && (!d_out_xy || !d_out_score || !d_out_desc)))
        return fail(h, PGM_E_INVALID_ARG, "bad arguments");
    h->stats = pgm_stats{};
    h->stats_pending = false;
    *out_count = 0;
    CU_CHECK(h, cudaSetDevice(h->device));
    cudaStream_t s = h->stream;
    // 1. FAST-12: score map, ordered compaction into (xy | score) in h->out
    const size_t npx = (size_t)width * height;
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return o; };
    const size_t o_sc = take(npx), o_cnt = take((size_t)height * 4), o_off = take((size_t)(height + 1) * 4);
    if ((rc = ensure_dev(h, h->misc, off))) return rc;
    if ((rc = ensure_host(h, h->pin_meta, 64))) return rc;
    char *base = (char *)h->misc.p;
    uint8_t *d_sc = (uint8_t *)(base + o_sc);
    int32_t *d_cnt = (int32_t *)(base + o_cnt), *d_off = (int32_t *)(base + o_off);
    dim3 blk(32, 8), grd((width + 31) / 32, (height + 7) / 8);
    if (flags & PGM_FLAG_PYTHON_GENERATION) fast_score_kernel<1><<<grd, blk, 0, s>>>(d_gray, width, height, threshold, d_sc);
    else fast_score_kernel<0><<<grd, blk, 0, s>>>(d_gray, width, height, threshold, d_sc);
    row_count_kernel<<<height, 128, 0, s>>>(d_sc, width, d_cnt);
    scan_kernel<<<1, 1024, 0, s>>>(d_cnt, height, d_off);
    CU_CHECK(h, cudaMemcpyAsync(h->pin_meta.p, d_off + height, 4, cudaMemcpyDeviceToHost, s));
    CU_CHECK(h, cudaStreamSynchronize(s));
    const int32_t total = *(int32_t *)h->pin_meta.p;
    h->stats.kernel_launches += 3; h->stats.host_syncs++;
    *out_count = total;
    if (total == 0) return PGM_OK;
    if (nms_radius < 0 && total > capacity) return fail(h, PGM_E_CAPACITY, "more keypoints than capacity (out_count holds the number found)");
    if ((rc = ensure_dev(h, h->out, (size_t)total * 12))) return rc;
    int32_t *d_xy = (int32_t *)h->out.p, *d_s = d_xy + 2 * (size_t)total;
    emit_kernel<<<(height + 3) / 4, 128, 0, s>>>(d_sc, width, height, d_off, total, d_xy, d_s);
    h->stats.kernel_launches += 1;
    // 2. NMS (optional): survivors in the reference's output order, gathered into the caller's arrays
    int32_t n = total;
    if (nms_radius >= 0) {
        if ((rc = ensure_host(h, h->pin_out, (size_t)total * 8))) return rc;
        CU_CHECK(h, cudaMemcpyAsync(h->pin_out.p, d_xy, (size_t)total * 8, cudaMemcpyDeviceToHost, s));   // bounding box
        CU_CHECK(h, cudaStreamSynchronize(s));
        h->stats.host_syncs++; h->stats.d2h_bytes += (int64_t)total * 8;
        int32_t *d_kept = nullptr;
        if ((rc = nms_core(h, d_xy, d_s, (const int32_t *)h->pin_out.p, total, nms_radius, &d_kept, &n))) return rc;
        *out_count = n;
        if (n > capacity) return fail(h, PGM_E_CAPACITY, "more keypoints than capacity (out_count holds the number found)");
        gather_kept_kernel<<<(n + 255) / 256, 256, 0, s>>>(d_xy, d_s, d_kept, n, d_out_xy, d_out_score);
        h->stats.kernel_launches += 1;
    } else {
        CU_CHECK(h, cudaMemcpyAsync(d_out_xy, d_xy, (size_t)n * 8, cudaMemcpyDeviceToDevice, s));
        CU_CHECK(h, cudaMemcpyAsync(d_out_score, d_s, (size_t)n * 4, cudaMemcpyDeviceToDevice, s));
    }
    // 3. BRIEF on the survivors, straight into the matcher's row layout
    if ((rc = ensure_dev(h, h->out2, (size_t)n_pairs * 16))) return rc;     // (h->misc still holds d_kept for the gather)
    CU_CHECK(h, cudaMemcpyAsync(h->out2.p, pairs, (size_t)n_pairs * 16, cudaMemcpyHostToDevice, s));
    const int warps = 4, sw = stride_bytes / 4;
    brief_kernel<<<(n + warps - 1) / warps, warps * 32, warps * sw * 4, s>>>(d_gray, width, height, d_out_xy, n,
                                                                         (const int32_t *)h->out2.p, n_pairs, sw,
                                                                         (flags & PGM_FLAG_PYTHON_GENERATION) ? 1 : 0,
                                                                         (uint32_t *)d_out_desc);
    CU_CHECK(h, cudaStreamSynchronize(s));        // `pairs` is a pageable host buffer: do not return before it is consumed
    h->stats.kernel_launches += 1; h->stats.host_syncs++;
    CU_CHECK(h, cudaGetLastError());
    return PGM_OK;
}

// Batched detection: many images in one call, every image at its own size (pgm_detect.cuh's ImageGeom table).
// counts[z] = the FAST total behind image z's row offsets (slot h of its rows)
__global__ void batch_counts_kernel(const int32_t *__restrict__ rowoff, const pgm_det::ImageGeom *__restrict__ geo,
                                    int n_images, int32_t *__restrict__ counts) {
    const int z = blockIdx.x * blockDim.x + threadIdx.x;
    if (z < n_images) counts[z] = rowoff[geo[z].row + geo[z].h];
}

// resident grid of a flat kernel (pgm_detect.cuh): `ctas_per_sm` per SM, at most one CTA per `per_cta` items
static unsigned flat_grid(const pgm_handle *h, long long items, int ctas_per_sm, int per_cta) {
    return (unsigned)std::max<long long>(std::min<long long>((long long)h->num_sms * ctas_per_sm, (items + per_cta - 1) / per_cta), 1);
}

// The three batch entry points' common body.  Image k is widths[k] x heights[k] at d_gray + pixel_offsets[k]; the
// caller holds h->mu, has checked every argument and reset the statistics, and n_images >= 1.
//   no NMS (nms_radius < 0): FAST-12 -> ordered keypoint list -> BRIEF for image k into its own `capacity` output
//     slots; the counts stay on the device (d_out_counts), nothing is read back.  6 kernel launches.
//   NMS: FAST-12 -> RedundantKeypointEliminator -> BRIEF, equal per image to pgm_detect_describe_dev(nms_radius).  One
//     read-back (the per-image FAST totals, which size the flat keypoint list); the NMS rounds of all images run in one
//     cooperative kernel that decides by itself when they are over.  11 kernel launches.
// Either way the counts are copied to `out_counts` at the end if the caller wants them (one more synchronisation).
static int detect_batch(pgm_handle *h, const float *d_gray, const int64_t *pixel_offsets, const int32_t *widths,
                        const int32_t *heights, int32_t n_images, float threshold, int32_t nms_radius,
                        const int32_t *pairs, int32_t n_pairs, int32_t stride_bytes, uint32_t flags, int32_t *d_out_xy,
                        int32_t *d_out_score, uint8_t *d_out_desc, int32_t capacity, int32_t *d_out_counts,
                        int32_t *out_counts) {
    using namespace pgm_det;
    CU_CHECK(h, cudaSetDevice(h->device));
    cudaStream_t s = h->stream;
    const bool py = (flags & PGM_FLAG_PYTHON_GENERATION) != 0, nms = nms_radius >= 0;
    const int cs = std::max(nms_radius, 1);

    // the geometry table and the pair table, staged together
    const size_t geo_bytes = align_up((size_t)(n_images + 1) * sizeof(ImageGeom), 256), pair_bytes = (size_t)n_pairs * 16;
    int rc = ensure_host(h, h->pin_in, geo_bytes + pair_bytes);
    if (rc) return rc;
    CU_CHECK(h, cudaStreamSynchronize(s));                 // the staging buffer may still feed an earlier call's copy
    ImageGeom *hg = (ImageGeom *)h->pin_in.p, acc{};
    for (int z = 0; z < n_images; z++) {
        const int w = widths[z], hh = heights[z];
        acc.px = pixel_offsets[z]; acc.w = w; acc.h = hh;
        acc.ncx = nms ? (w - 1) / cs + 1 : 0; acc.ncy = nms ? (hh - 1) / cs + 1 : 0;
        hg[z] = acc;
        acc.sc += (long long)w * hh; acc.row += hh + 1;
        acc.tile += (long long)((w + FAST_TILE_W - 1) / FAST_TILE_W) * ((hh + FAST_TILE_H - 1) / FAST_TILE_H);
        acc.cell += (long long)acc.ncx * acc.ncy;
    }
    acc.px = 0; acc.w = acc.h = acc.ncx = acc.ncy = 0;
    hg[n_images] = acc;                                    // totals
    memcpy((char *)h->pin_in.p + geo_bytes, pairs, pair_bytes);

    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return o; };
    const size_t o_geo = take(geo_bytes + pair_bytes), o_sc = take((size_t)acc.sc), o_cnt = take((size_t)acc.row * 4);
    const size_t o_off = take((size_t)acc.row * 4), o_tot = take((size_t)n_images * 4), o_base = take((size_t)(n_images + 1) * 4);
    if ((rc = ensure_dev(h, h->misc, off))) return rc;
    if ((rc = ensure_host(h, h->pin_out, (size_t)n_images * 4))) return rc;
    char *mb = (char *)h->misc.p;
    const ImageGeom *d_geo = (const ImageGeom *)(mb + o_geo);
    const int32_t *d_pairs = (const int32_t *)(mb + o_geo + geo_bytes);
    uint8_t *d_sc = (uint8_t *)(mb + o_sc);
    int32_t *d_cnt = (int32_t *)(mb + o_cnt), *d_off = (int32_t *)(mb + o_off), *d_tot = (int32_t *)(mb + o_tot);
    int32_t *d_base = (int32_t *)(mb + o_base);
    CU_CHECK(h, cudaMemcpyAsync(mb + o_geo, h->pin_in.p, geo_bytes + pair_bytes, cudaMemcpyHostToDevice, s));
    h->stats.h2d_bytes += (int64_t)(geo_bytes + pair_bytes);

    // 1. FAST-12 of every image: score maps, row counts, row offsets (slot h = the image's total)
    const dim3 tile(FAST_TILE_W, FAST_TILE_H);
    // one size packed back to back: the kernels' table-free grids (pgm_detect.cuh); else flat work over all images
    bool one_size = true;
    for (int z = 1; z < n_images && one_size; z++)
        one_size = widths[z] == widths[0] && heights[z] == heights[0] &&
                   pixel_offsets[z] == pixel_offsets[0] + (int64_t)z * widths[0] * heights[0];
    const int uw = one_size ? widths[0] : 0, uh = one_size ? heights[0] : 0;
    const float *d_img = one_size ? d_gray + pixel_offsets[0] : d_gray;
    const dim3 fast_grid = one_size ? dim3((uw + FAST_TILE_W - 1) / FAST_TILE_W, (uh + FAST_TILE_H - 1) / FAST_TILE_H, n_images)
                                    : dim3(flat_grid(h, acc.tile, FLAT_CTAS_PER_SM_256, 1));
    const dim3 row_grid = one_size ? dim3(uh, n_images) : dim3(flat_grid(h, acc.row, FLAT_CTAS_PER_SM_128, 1));
    const dim3 warp_grid = one_size ? dim3((uh + 3) / 4, n_images) : dim3(flat_grid(h, acc.row, FLAT_CTAS_PER_SM_128, 4));
    if (py) fast_score_kernel<1><<<fast_grid, tile, 0, s>>>(d_img, d_geo, n_images, uw, uh, threshold, d_sc);
    else fast_score_kernel<0><<<fast_grid, tile, 0, s>>>(d_img, d_geo, n_images, uw, uh, threshold, d_sc);
    row_count_kernel<<<row_grid, 128, 0, s>>>(d_sc, d_geo, n_images, uw, uh, d_cnt);
    scan_kernel<<<n_images, 1024, 0, s>>>(d_cnt, 0, d_off, d_geo);
    const int warps = 4, sw = stride_bytes / 4;
    if (!nms) {
        batch_counts_kernel<<<(n_images + 255) / 256, 256, 0, s>>>(d_off, d_geo, n_images, d_out_counts);
        emit_kernel<<<warp_grid, 128, 0, s>>>(d_sc, d_geo, n_images, uw, uh, d_off, capacity, d_out_xy, d_out_score);
        brief_kernel<<<dim3((capacity + warps - 1) / warps, n_images), warps * 32, warps * sw * 4, s>>>(
            d_gray, 0, 0, d_out_xy, capacity, d_pairs, n_pairs, sw, py ? 1 : 0, (uint32_t *)d_out_desc, d_geo, d_out_counts);
        h->stats.kernel_launches += 6;
    } else {
        batch_counts_kernel<<<(n_images + 255) / 256, 256, 0, s>>>(d_off, d_geo, n_images, d_tot);
        CU_CHECK(h, cudaMemcpyAsync(h->pin_out.p, d_tot, (size_t)n_images * 4, cudaMemcpyDeviceToHost, s));
        CU_CHECK(h, cudaStreamSynchronize(s));
        h->stats.kernel_launches += 4; h->stats.host_syncs++; h->stats.d2h_bytes += (int64_t)n_images * 4;

        // image bases of the flat keypoint list (the sync above freed pin_in); every index below is an int32
        const int32_t *h_tot = (const int32_t *)h->pin_out.p;
        int64_t total = 0;
        for (int z = 0; z < n_images; z++) total += h_tot[z];
        if (total > INT32_MAX) return fail(h, PGM_E_CAPACITY, "the batch has more than 2^31 - 1 FAST keypoints: split it");
        const int32_t n = (int32_t)total;
        const size_t base_bytes = (size_t)(n_images + 1) * 4;
        if ((rc = ensure_host(h, h->pin_in, base_bytes))) return rc;
        int32_t *h_base = (int32_t *)h->pin_in.p;
        h_base[0] = 0;
        for (int z = 0; z < n_images; z++) h_base[z + 1] = h_base[z] + h_tot[z];
        CU_CHECK(h, cudaMemcpyAsync(d_base, h->pin_in.p, base_bytes, cudaMemcpyHostToDevice, s));
        h->stats.h2d_bytes += (int64_t)base_bytes;
        if (n == 0) {
            CU_CHECK(h, cudaMemsetAsync(d_out_counts, 0, (size_t)n_images * 4, s));
        } else {
            // scratch of the flat list: h->out; radix-sort temporaries: h->out2
            const long long r2 = (long long)nms_radius * nms_radius;
            size_t o2 = 0;
            auto take2 = [&](size_t bytes) { size_t o = o2; o2 = align_up(o2 + bytes, 256); return o; };
            const size_t o_xy = take2((size_t)n * 8), o_s = take2((size_t)n * 4), o_rk = take2((size_t)n * 4), o_or = take2((size_t)n * 4);
            const size_t o_k0 = take2((size_t)n * 8), o_k1 = take2((size_t)n * 8), o_c0 = take2((size_t)n * 8), o_c1 = take2((size_t)n * 8);
            const size_t o_v0 = take2((size_t)n * 4), o_v1 = take2((size_t)n * 4), o_st0 = take2(n), o_st1 = take2(n);
            const size_t o_ctl = take2(sizeof(NmsBatchCtl));
            if ((rc = ensure_dev(h, h->out, o2))) return rc;
            char *ob = (char *)h->out.p;
            int32_t *d_xy = (int32_t *)(ob + o_xy), *d_s = (int32_t *)(ob + o_s), *d_rk = (int32_t *)(ob + o_rk);
            int32_t *d_or = (int32_t *)(ob + o_or), *d_v0 = (int32_t *)(ob + o_v0), *d_v1 = (int32_t *)(ob + o_v1);
            unsigned long long *d_k0 = (unsigned long long *)(ob + o_k0), *d_k1 = (unsigned long long *)(ob + o_k1);
            unsigned long long *d_c0 = (unsigned long long *)(ob + o_c0), *d_c1 = (unsigned long long *)(ob + o_c1);
            uint8_t *d_st0 = (uint8_t *)(ob + o_st0), *d_st1 = (uint8_t *)(ob + o_st1);
            NmsBatchCtl *d_ctl = (NmsBatchCtl *)(ob + o_ctl);
            int img_bits = 0, cell_bits = 1;
            while ((n_images - 1) >> img_bits) img_bits++;
            const unsigned long long n_cells = (unsigned long long)acc.cell;      // sum over the images of ncx * ncy
            while (cell_bits < 64 && (n_cells - 1) >> cell_bits) cell_bits++;
            const int rank_bits = NMS_RANK_IMAGE_SHIFT + img_bits;
            size_t tmp_bytes = 0, tmp2 = 0;
            CU_CHECK(h, cub::DeviceRadixSort::SortKeys(nullptr, tmp_bytes, d_k0, d_k1, n, 0, rank_bits, s));
            CU_CHECK(h, cub::DeviceRadixSort::SortPairs(nullptr, tmp2, d_c0, d_c1, d_v0, d_v1, n, 0, cell_bits, s));
            tmp_bytes = std::max(tmp_bytes, tmp2);
            if ((rc = ensure_dev(h, h->out2, tmp_bytes))) return rc;
            int nb = 0;
            CU_CHECK(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, nms_rounds_batch_kernel, NMS_BATCH_THREADS, 0));
            const int rounds_grid = (int)std::min<int64_t>((int64_t)std::max(nb, 1) * h->num_sms,
                                                           ((int64_t)n + NMS_BATCH_THREADS - 1) / NMS_BATCH_THREADS);

            // 2. flat list with rank keys and cell ids; 3. rank order; 4. cell order
            nms_batch_emit_kernel<<<warp_grid, 128, 0, s>>>(d_sc, d_geo, n_images, uw, uh, d_off, d_base, cs, d_xy,
                                                                         d_s, d_k0, d_c0, d_v0);
            CU_CHECK(h, cub::DeviceRadixSort::SortKeys(h->out2.p, tmp_bytes, d_k0, d_k1, n, 0, rank_bits, s));
            nms_batch_order_kernel<<<(n + 255) / 256, 256, 0, s>>>(d_k1, n, d_base, n_images, d_or, d_rk);
            CU_CHECK(h, cub::DeviceRadixSort::SortPairs(h->out2.p, tmp_bytes, d_c0, d_c1, d_v0, d_v1, n, 0, cell_bits, s));
            // 5. every round of every image; 6. survivors in output order into the caller's slots
            CU_CHECK(h, cudaMemsetAsync(d_st0, 0, n, s));
            CU_CHECK(h, cudaMemsetAsync(d_ctl, 0, sizeof(NmsBatchCtl), s));
            int n_arg = n, cs_arg = cs, ni_arg = n_images;
            long long r2_arg = r2;
            const int32_t *a_xy = d_xy, *a_rk = d_rk, *a_v1 = d_v1;
            const unsigned long long *a_k0 = d_k0, *a_c0 = d_c0, *a_c1 = d_c1;
            void *args[] = {&a_xy, &a_rk, &n_arg, &r2_arg, &cs_arg, &d_geo, &ni_arg, &a_k0, &a_c0, &a_c1, &a_v1,
                            &d_st0, &d_st1, &d_ctl};
            CU_CHECK(h, cudaLaunchCooperativeKernel((void *)nms_rounds_batch_kernel, dim3(rounds_grid),
                                                    dim3(NMS_BATCH_THREADS), args, 0, s));
            nms_batch_gather_kernel<<<n_images, NMS_EMIT_THREADS, 0, s>>>(d_or, d_base, d_st0, d_st1, d_ctl, d_xy, d_s,
                                                                          capacity, d_out_xy, d_out_score, d_out_counts);
            // 7. BRIEF of the survivors
            brief_kernel<<<dim3((capacity + warps - 1) / warps, n_images), warps * 32, warps * sw * 4, s>>>(
                d_gray, 0, 0, d_out_xy, capacity, d_pairs, n_pairs, sw, py ? 1 : 0, (uint32_t *)d_out_desc, d_geo,
                d_out_counts);
            // emit, rank sort, order, cell sort, rounds, gather, BRIEF (a radix sort counts once)
            h->stats.kernel_launches += 7;
        }
    }
    CU_CHECK(h, cudaGetLastError());
    if (out_counts) {
        CU_CHECK(h, cudaMemcpyAsync(h->pin_out.p, d_out_counts, (size_t)n_images * 4, cudaMemcpyDeviceToHost, s));
        CU_CHECK(h, cudaStreamSynchronize(s));
        memcpy(out_counts, h->pin_out.p, (size_t)n_images * 4);
        h->stats.host_syncs++; h->stats.d2h_bytes += (int64_t)n_images * 4;
    }
    return PGM_OK;
}

// the uniform forms: image k at d_gray + k * width * height
static int detect_batch_uniform(pgm_handle *h, const float *d_gray, int32_t n_images, int32_t width, int32_t height,
                                float threshold, int32_t nms_radius, const int32_t *pairs, int32_t n_pairs,
                                int32_t stride_bytes, uint32_t flags, int32_t *d_out_xy, int32_t *d_out_score,
                                uint8_t *d_out_desc, int32_t capacity, int32_t *d_out_counts, int32_t *out_counts) {
    std::vector<int64_t> offsets(n_images);
    for (int z = 0; z < n_images; z++) offsets[z] = (int64_t)z * width * height;
    const std::vector<int32_t> widths(n_images, width), heights(n_images, height);
    return detect_batch(h, d_gray, offsets.data(), widths.data(), heights.data(), n_images, threshold, nms_radius, pairs,
                        n_pairs, stride_bytes, flags, d_out_xy, d_out_score, d_out_desc, capacity, d_out_counts,
                        out_counts);
}

// Many equally sized images in one call, nothing read back in between.  A count above `capacity` means the image's
// list was truncated.  No NMS in this form (pgm_detect_nms_describe_batch_dev has it).
extern "C" int pgm_detect_describe_batch_dev(pgm_handle *h, const float *d_gray, int32_t n_images, int32_t width,
                                             int32_t height, float threshold, const int32_t *pairs, int32_t n_pairs,
                                             int32_t stride_bytes, uint32_t flags, int32_t *d_out_xy,
                                             int32_t *d_out_score, uint8_t *d_out_desc, int32_t capacity,
                                             int32_t *d_out_counts, int32_t *out_counts) {
    if (!h) return PGM_E_INVALID_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    int rc = check_format(h, n_pairs, stride_bytes);       // desc_bits == NumGaussianPairs
    if (rc) return rc;
    if (!d_gray || n_images < 0 || n_images > 65535 || width < 1 || height < 1 || width > 65535 || height > 65535 ||
        !pairs || capacity < 1 || !d_out_xy || !d_out_score || !d_out_desc || !d_out_counts)
        return fail(h, PGM_E_INVALID_ARG, "bad arguments");
    h->stats = pgm_stats{};
    h->stats_pending = false;
    if (n_images == 0) return PGM_OK;
    return detect_batch_uniform(h, d_gray, n_images, width, height, threshold, -1, pairs, n_pairs, stride_bytes, flags,
                                d_out_xy, d_out_score, d_out_desc, capacity, d_out_counts, out_counts);
}

// The batched chain with NMS, equal per image to pgm_detect_describe_dev(nms_radius).
extern "C" int pgm_detect_nms_describe_batch_dev(pgm_handle *h, const float *d_gray, int32_t n_images, int32_t width,
                                                 int32_t height, float threshold, int32_t nms_radius, const int32_t *pairs,
                                                 int32_t n_pairs, int32_t stride_bytes, uint32_t flags, int32_t *d_out_xy,
                                                 int32_t *d_out_score, uint8_t *d_out_desc, int32_t capacity,
                                                 int32_t *d_out_counts, int32_t *out_counts) {
    if (!h) return PGM_E_INVALID_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    int rc = check_format(h, n_pairs, stride_bytes);       // desc_bits == NumGaussianPairs
    if (rc) return rc;
    if (!d_gray || n_images < 0 || n_images > 65535 || width < 1 || height < 1 || width > 65535 || height > 65535 ||
        nms_radius < 0 || !pairs || capacity < 1 || !d_out_xy || !d_out_score || !d_out_desc || !d_out_counts)
        return fail(h, PGM_E_INVALID_ARG, "bad arguments");
    h->stats = pgm_stats{};
    h->stats_pending = false;
    if (n_images == 0) return PGM_OK;
    return detect_batch_uniform(h, d_gray, n_images, width, height, threshold, nms_radius, pairs, n_pairs, stride_bytes,
                                flags, d_out_xy, d_out_score, d_out_desc, capacity, d_out_counts, out_counts);
}

// Images of any sizes in one call: image k is widths[k] x heights[k] at d_gray + pixel_offsets[k].
extern "C" int pgm_detect_describe_images_batch_dev(pgm_handle *h, const float *d_gray, const int64_t *pixel_offsets,
                                                    const int32_t *widths, const int32_t *heights, int32_t n_images,
                                                    float threshold, int32_t nms_radius, const int32_t *pairs,
                                                    int32_t n_pairs, int32_t stride_bytes, uint32_t flags,
                                                    int32_t *d_out_xy, int32_t *d_out_score, uint8_t *d_out_desc,
                                                    int32_t capacity, int32_t *d_out_counts, int32_t *out_counts) {
    if (!h) return PGM_E_INVALID_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    int rc = check_format(h, n_pairs, stride_bytes);       // desc_bits == NumGaussianPairs
    if (rc) return rc;
    if (!d_gray || !pixel_offsets || !widths || !heights || n_images < 0 || n_images > 65535 || !pairs ||
        capacity < 1 || !d_out_xy || !d_out_score || !d_out_desc || !d_out_counts)
        return fail(h, PGM_E_INVALID_ARG, "bad arguments");
    if (pixel_offsets[0] < 0) return fail(h, PGM_E_INVALID_ARG, "pixel_offsets[0] < 0");
    for (int z = 0; z < n_images; z++) {
        if (widths[z] < 1 || heights[z] < 1 || widths[z] > 65535 || heights[z] > 65535)
            return fail(h, PGM_E_INVALID_ARG, "an image size is outside 1..65535");   // MatrixDimensions are ushort upstream
        if (pixel_offsets[z + 1] < pixel_offsets[z] + (int64_t)widths[z] * heights[z])
            return fail(h, PGM_E_INVALID_ARG, "pixel_offsets[k + 1] < pixel_offsets[k] + widths[k] * heights[k]");
    }
    h->stats = pgm_stats{};
    h->stats_pending = false;
    if (n_images == 0) return PGM_OK;
    return detect_batch(h, d_gray, pixel_offsets, widths, heights, n_images, threshold, nms_radius, pairs, n_pairs,
                        stride_bytes, flags, d_out_xy, d_out_score, d_out_desc, capacity, d_out_counts, out_counts);
}

// ---------------------------------------------------------------------------
// the consumer of the match list: RANSAC hypothesis scoring (pgm_ransac.cuh)
// ---------------------------------------------------------------------------
extern "C" int pgm_ransac_score(pgm_handle *h, const float *F, const uint8_t *valid, int32_t n_hyp, const int32_t *xy1,
                                const int32_t *xy2, int32_t n, float threshold, int32_t *out_counts, int32_t *out_best,
                                uint8_t *out_best_mask) {
    using namespace pgm_ransac;
    if (!h) return PGM_E_INVALID_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    if (n_hyp < 0 || n < 0 || (n_hyp > 0 && !F) || (n > 0 && (!xy1 || !xy2))) return fail(h, PGM_E_INVALID_ARG, "bad arguments");
    h->stats = pgm_stats{};
    h->stats_pending = false;
    if (out_best) *out_best = -1;
    if (n_hyp == 0) return PGM_OK;
    CU_CHECK(h, cudaSetDevice(h->device));
    cudaStream_t s = h->stream;
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return o; };
    const size_t o_f = take((size_t)n_hyp * 36), o_v = take(n_hyp), o_1 = take((size_t)std::max(n, 1) * 8), o_2 = take((size_t)std::max(n, 1) * 8);
    const size_t o_c = take((size_t)n_hyp * 4), o_b = take(16), o_m = take(std::max(n, 1));
    int rc = ensure_dev(h, h->misc, off);
    if (rc) return rc;
    if ((rc = ensure_host(h, h->pin_out, (size_t)n_hyp * 4 + 64 + (size_t)n))) return rc;
    char *base = (char *)h->misc.p;
    CU_CHECK(h, cudaMemcpyAsync(base + o_f, F, (size_t)n_hyp * 36, cudaMemcpyHostToDevice, s));
    if (valid) CU_CHECK(h, cudaMemcpyAsync(base + o_v, valid, n_hyp, cudaMemcpyHostToDevice, s));
    if (n) {
        CU_CHECK(h, cudaMemcpyAsync(base + o_1, xy1, (size_t)n * 8, cudaMemcpyHostToDevice, s));
        CU_CHECK(h, cudaMemcpyAsync(base + o_2, xy2, (size_t)n * 8, cudaMemcpyHostToDevice, s));
    }
    score_kernel<<<n_hyp, 256, 0, s>>>((const float *)(base + o_f), valid ? (const uint8_t *)(base + o_v) : nullptr, n_hyp,
                                       (const int32_t *)(base + o_1), (const int32_t *)(base + o_2), n, threshold,
                                       (int32_t *)(base + o_c));
    best_kernel<<<1, 1024, 0, s>>>((const float *)(base + o_f), (const int32_t *)(base + o_c), n_hyp, (const int32_t *)(base + o_1),
                                   (const int32_t *)(base + o_2), n, threshold, (int32_t *)(base + o_b),
                                   out_best_mask ? (uint8_t *)(base + o_m) : nullptr);
    char *ph = (char *)h->pin_out.p;
    CU_CHECK(h, cudaMemcpyAsync(ph, base + o_c, (size_t)n_hyp * 4, cudaMemcpyDeviceToHost, s));
    CU_CHECK(h, cudaMemcpyAsync(ph + (size_t)n_hyp * 4, base + o_b, 4, cudaMemcpyDeviceToHost, s));
    if (out_best_mask && n) CU_CHECK(h, cudaMemcpyAsync(ph + (size_t)n_hyp * 4 + 64, base + o_m, n, cudaMemcpyDeviceToHost, s));
    CU_CHECK(h, cudaStreamSynchronize(s));
    if (out_counts) memcpy(out_counts, ph, (size_t)n_hyp * 4);
    if (out_best) *out_best = *(int32_t *)(ph + (size_t)n_hyp * 4);
    if (out_best_mask && n) memcpy(out_best_mask, ph + (size_t)n_hyp * 4 + 64, n);
    h->stats.kernel_launches += 2; h->stats.host_syncs++;
    h->stats.h2d_bytes += (int64_t)n_hyp * 36 + (int64_t)n * 16; h->stats.d2h_bytes += (int64_t)n_hyp * 4 + n;
    CU_CHECK(h, cudaGetLastError());
    return PGM_OK;
}

// Many match lists in one call: the hypotheses of the pairs with count >= P form one flattened space g = k S + s
// (k = the k-th such pair), cut into chunks of RB_CHUNK_HYPS whose F and rank flags reuse one scratch area.  The host
// plans every chunk from host arrays and uploads the plan in one copy; nothing is read back.
constexpr int64_t RB_CHUNK_HYPS = 1ll << 20;

extern "C" int pgm_ransac_fundamental_pairs_batch_dev(pgm_handle *h, const int32_t *d_all_xy, const int64_t *image_offsets,
        int32_t n_images, const int32_t *pair_list, int32_t n_pairs, const int32_t *d_match_qi, const int32_t *d_match_tj,
        const int64_t *match_starts, const int32_t *match_counts, int32_t n_samples, int32_t pairs_per_sample,
        float threshold, uint64_t seed, uint32_t flags, int32_t *d_out_best, int32_t *d_out_inliers, float *d_out_F,
        uint8_t *d_out_mask, int64_t capacity, float *d_hyp_F, int32_t *d_hyp_counts) {
    using namespace pgm_ransac;
    if (!h) return PGM_E_INVALID_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    h->stats = pgm_stats{};
    h->stats_pending = false;
    const int P = pairs_per_sample;
    const int64_t S = n_samples;
    if (P < 8 || P > RB_MAX_P || S < 1 || n_pairs < 0 || n_images < 0 || capacity < 0 || (flags & ~PGM_FLAG_RANSAC_RANK_TEST))
        return fail(h, PGM_E_INVALID_ARG, "bad n_samples, pairs_per_sample, sizes or flags");
    if (n_pairs == 0) return PGM_OK;
    if (!image_offsets || !pair_list || !match_starts || !match_counts || !d_all_xy || !d_match_qi || !d_match_tj ||
        !d_out_best || !d_out_inliers || !d_out_F || !d_out_mask)
        return fail(h, PGM_E_INVALID_ARG, "null pointer");
    std::vector<RbPair> plan(n_pairs);
    std::vector<int32_t> act;
    for (int p = 0; p < n_pairs; p++) {
        const int a = pair_list[2 * p], b = pair_list[2 * p + 1];
        if (a < 0 || a >= n_images || b < 0 || b >= n_images) return fail(h, PGM_E_INVALID_ARG, "pair index out of range");
        const int64_t oa = image_offsets[a], ob = image_offsets[b];
        const int64_t na = image_offsets[a + 1] - oa, nb = image_offsets[b + 1] - ob;
        if (oa < 0 || ob < 0 || na < 0 || nb < 0 || na > INT32_MAX || nb > INT32_MAX) return fail(h, PGM_E_INVALID_ARG, "bad image offsets");
        const int64_t st = match_starts[p];
        const int32_t cnt = match_counts[p];
        if (cnt < 0 || st < 0 || st + cnt > capacity) return fail(h, PGM_E_INVALID_ARG, "match slots outside [0, capacity)");
        if (cnt > 0 && (na == 0 || nb == 0)) return fail(h, PGM_E_INVALID_ARG, "matches of an empty image");
        plan[p] = RbPair{st, oa, ob, cnt, a, b, (int32_t)na, (int32_t)nb, 0};
        if (cnt >= P) act.push_back(p);
    }
    // chunks of the flattened hypothesis space; item_base: per chunk, the score items' prefix over its pairs
    struct Chunk { int64_t g0, g1, k0; int n_local, base_off, items; };
    std::vector<Chunk> chunks;
    std::vector<int32_t> bases;
    const int64_t total = (int64_t)act.size() * S;
    for (int64_t g0 = 0; g0 < total; g0 += RB_CHUNK_HYPS) {
        const int64_t g1 = std::min(total, g0 + RB_CHUNK_HYPS);
        Chunk c{g0, g1, g0 / S, 0, (int)bases.size(), 0};
        for (int64_t k = c.k0; k * S < g1; k++) {
            const int64_t len = std::min(g1, (k + 1) * S) - std::max(g0, k * S);
            bases.push_back(c.items);
            c.items += (int)((len + RB_SCORE_THREADS - 1) / RB_SCORE_THREADS);
            c.n_local++;
        }
        bases.push_back(c.items);
        chunks.push_back(c);
    }
    const int64_t hyps = std::min<int64_t>(std::max<int64_t>(total, 1), RB_CHUNK_HYPS);
    // h->misc: plan | active pairs | item bases | keys | chunk F | chunk rank flags
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + std::max<size_t>(bytes, 1), 256); return o; };
    const size_t o_plan = take(sizeof(RbPair) * plan.size()), o_act = take(4 * act.size()), o_bases = take(4 * bases.size());
    const size_t upload = off;
    const size_t o_keys = take(8 * (size_t)n_pairs), o_F = take((size_t)hyps * 36), o_v = take((size_t)hyps);
    int rc = ensure_dev(h, h->misc, off);
    if (rc) return rc;
    CU_CHECK(h, cudaSetDevice(h->device));
    cudaStream_t s = h->stream;
    std::vector<char> host(upload);
    memcpy(host.data() + o_plan, plan.data(), sizeof(RbPair) * plan.size());
    if (!act.empty()) memcpy(host.data() + o_act, act.data(), 4 * act.size());
    memcpy(host.data() + o_bases, bases.data(), 4 * bases.size());
    char *dev = (char *)h->misc.p;
    // pageable source: the runtime stages it before returning, so the vector may go; no stream synchronisation
    CU_CHECK(h, cudaMemcpyAsync(dev, host.data(), upload, cudaMemcpyHostToDevice, s));
    CU_CHECK(h, cudaMemsetAsync(dev + o_keys, 0, 8 * (size_t)n_pairs, s));
    const RbPair *d_plan = (const RbPair *)(dev + o_plan);
    const int32_t *d_act = (const int32_t *)(dev + o_act), *d_bases = (const int32_t *)(dev + o_bases);
    unsigned long long *d_keys = (unsigned long long *)(dev + o_keys);
    float *d_F = (float *)(dev + o_F);
    uint8_t *d_v = (uint8_t *)(dev + o_v);
    const int rank_test = (flags & PGM_FLAG_RANSAC_RANK_TEST) ? 1 : 0;
    for (const Chunk &c : chunks) {
        const unsigned grid = (unsigned)((c.g1 - c.g0 + RB_EST_THREADS - 1) / RB_EST_THREADS);
        estimate_kernel<<<grid, RB_EST_THREADS, RB_EST_THREADS * RB_SM_DOUBLES * sizeof(double), s>>>(
            d_plan, d_act, S, c.g0, c.g1, d_all_xy, d_match_qi, d_match_tj, P, seed, rank_test, d_F, d_v, d_hyp_F);
        pairs_score_kernel<<<c.items, RB_SCORE_THREADS, 0, s>>>(d_plan, d_act, d_bases + c.base_off, c.n_local, c.k0, S,
                                                                 c.g0, c.g1, d_F, d_v, d_all_xy, d_match_qi, d_match_tj,
                                                                 threshold, d_keys, d_hyp_counts);
        CU_CHECK(h, cudaGetLastError());
        h->stats.kernel_launches += 2;
    }
    winner_kernel<<<n_pairs, RB_WIN_THREADS, 0, s>>>(d_plan, P, seed, d_keys, d_all_xy, d_match_qi, d_match_tj, threshold,
                                                     d_out_best, d_out_inliers, d_out_F, d_out_mask);
    CU_CHECK(h, cudaGetLastError());
    h->stats.kernel_launches += 1;
    h->stats.pairs = n_pairs;
    h->stats.h2d_bytes = (int64_t)upload;
    return PGM_OK;
}

// ---------------------------------------------------------------------------
// train-sharded single pair (BASELINE configs[3]).  Two surfaces over the same kernels:
//   pgm_shard_*   stepwise: the ONE exchange per round (element-wise min of X over the ranks) belongs to the caller
//                 (torch.distributed, MPI, or -- in the tests -- several emulated ranks on one GPU)
//   pgm_multi_*   the library owns an NCCL communicator (one rank per handle) and runs the whole match with no host
//                 synchronisation per round: rounds are enqueued in batches and an 8-byte status read-back per batch,
//                 checked two batches late, stops the loop and shrinks the exchange
// ---------------------------------------------------------------------------
struct ShardDev {                  // small device-resident control block of a shard (zeroed before every round)
    unsigned bar;                  // grid-barrier counter of the cooperative sparse kernel
    int32_t edge_cnt;              // filtered candidate edges of the round
    int32_t alive[2];
    unsigned ticket;               // last-block-done counter of the edge filter
};

struct pgm_shard {
    pgm_handle *h = nullptr;
    DevBuf state, est;
    Chunk c{};
    int words = 8, desc_bits = 256, n1 = 0, n2_local = 0, n2_total = 0, col_offset = 0;
    int round = 0;
    int round_grid = 0;
    const uint32_t *q_host_ptr = nullptr, *t_host_ptr = nullptr;   // the pair's descriptors (device pointers)
    int raw_cap = 0;               // candidate records this rank may emit per pass
    uint8_t *coldead = nullptr;    // [n2_total] by GLOBAL column id
    uint32_t *rbest_g = nullptr, *cbest_g = nullptr;   // [n1], [n2_total]: min slots of the grid-wide sparse phase
    int32_t *blockcnt = nullptr;
    ShardDev *dev = nullptr;
    ShardCtl *ctl = nullptr;       // device
    ShardCtl *h_ctl = nullptr;     // pinned: [8] status read-backs (ring)
};

constexpr float CAND_TARGET_SHARD = 4.0f;
// edges a rank may contribute per pass (identical on every rank for given sizes: the gathered layout is [ranks][1 + cap])
static int shard_edge_capacity(int n1, int n2_total, int world) {
    const int64_t m = std::max(n1, n2_total);
    return (int)std::min<int64_t>((int64_t)(2.0f * CAND_TARGET_SHARD + 1.0f) * m * 5 / (4 * std::max(world, 1)) + 4096, (int64_t)1 << 28);
}

extern "C" int pgm_shard_create(pgm_handle *h, const uint8_t *d_q, int32_t n1, const uint8_t *d_t_local,
                                int32_t n2_local, int32_t col_offset, int32_t n2_total, int32_t desc_bits,
                                int32_t stride_bytes, pgm_shard **out) {
    if (!h || !out) return PGM_E_INVALID_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    *out = nullptr;
    int rc = check_format(h, desc_bits, stride_bytes);
    if (rc) return rc;
    if (n1 <= 0 || n2_local < 0 || n2_total <= 0 || col_offset < 0 || col_offset + n2_local > n2_total ||
        n1 >= MAX_N || n2_total >= MAX_N || !d_q || (n2_local > 0 && !d_t_local))
        return fail(h, PGM_E_INVALID_ARG, "bad shard geometry");
    CU_CHECK(h, cudaSetDevice(h->device));
    cudaStream_t s = h->stream;
    pgm_shard *sh = new pgm_shard();
    sh->h = h; sh->words = stride_bytes / 4; sh->desc_bits = desc_bits;
    sh->n1 = n1; sh->n2_local = n2_local; sh->n2_total = n2_total; sh->col_offset = col_offset;
    sh->q_host_ptr = (const uint32_t *)d_q; sh->t_host_ptr = (const uint32_t *)d_t_local;
    const int64_t rows = n1, cols = std::max(n2_local, 1);
    const int n_blocks = (n1 + SHARD_BLOCK - 1) / SHARD_BLOCK;
    // this rank's share of the pass's candidate records (x 1.25 slack), by its share of the columns
    sh->raw_cap = (int)std::min<int64_t>(
        (int64_t)((2.0f * CAND_TARGET_SHARD + 1.0f) * 1.25f * (float)std::max(n1, n2_total) * ((float)cols / (float)n2_total)) + 4096,
        (int64_t)n1 * cols);
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return o; };
    const size_t o_pairs = take(sizeof(PairDesc));
    const size_t o_rb0 = take(4 * rows), o_rb1 = take(4 * rows), o_cb0 = take(4 * cols), o_cb1 = take(4 * cols);
    const size_t o_lr0 = take(4 * rows), o_lr1 = take(4 * rows), o_lc0 = take(4 * cols), o_lc1 = take(4 * cols);
    const size_t o_cnt = take(sizeof(int32_t) * 6), o_mk = take(4 * rows), o_tb = take(8), o_ab = take(8);
    const size_t o_st = take(1), o_small = take(sizeof(SmallInfo)), o_plan = take(sizeof(PlanInfo));
    const size_t o_dead = take((size_t)n2_total);
    const size_t o_rpos = take(4 * rows), o_bcnt = take(4 * (size_t)n_blocks), o_ctl = take(sizeof(ShardCtl));
    const size_t o_dev = take(sizeof(ShardDev));
    const size_t o_rbg = take(4 * rows), o_cbg = take(4 * (size_t)n2_total);
    const size_t o_cand = take(16 * (size_t)sh->raw_cap), o_ccnt = take(4), o_thr = take(4), o_pstat = take(sizeof(PairStat));
    std::swap(sh->state, h->shard_pool_state);      // buffers parked by the previous shard of this handle, if any
    std::swap(sh->est, h->shard_pool_est);
    if ((rc = ensure_dev(h, sh->state, off))) { if (sh->est.p) cudaFree(sh->est.p); delete sh; return rc; }
    if (h->shard_pool_hctl) { sh->h_ctl = (ShardCtl *)h->shard_pool_hctl; h->shard_pool_hctl = nullptr; }
    else if (cudaMallocHost((void **)&sh->h_ctl, sizeof(ShardCtl) * 8) != cudaSuccess) {
        cudaFree(sh->state.p); if (sh->est.p) cudaFree(sh->est.p); delete sh; return PGM_E_CUDA;
    }
    char *base = (char *)sh->state.p;
    if (h->ctas_per_sm[sh->words / 4] == 0) h->ctas_per_sm[sh->words / 4] = std::max(1, dispatch_occupancy(sh->words));
    sh->round_grid = h->num_sms * h->ctas_per_sm[sh->words / 4];
    Chunk &c = sh->c;
    c.pairs = (PairDesc *)(base + o_pairs); c.n_pairs = 1; c.num_sms = h->num_sms;
    c.ctas_per_sm = h->ctas_per_sm[sh->words / 4];
    c.fin_max_evals = FIN_MAX_EVALS;
    c.large_min_evals = large_tile_min_evals(h);
    c.words = sh->words;
    c.shard_n2_total = n2_total;
    c.cand_target = CAND_TARGET_SHARD;
    c.cand_row_max = 1e9f;
    c.sp_slots_max = SP_EPT;
    c.rowbest[0] = (uint32_t *)(base + o_rb0); c.rowbest[1] = (uint32_t *)(base + o_rb1);
    c.colbest[0] = (uint32_t *)(base + o_cb0); c.colbest[1] = (uint32_t *)(base + o_cb1);
    c.live_rows[0] = (int32_t *)(base + o_lr0); c.live_rows[1] = (int32_t *)(base + o_lr1);
    c.live_cols[0] = (int32_t *)(base + o_lc0); c.live_cols[1] = (int32_t *)(base + o_lc1);
    c.counts = (int32_t *)(base + o_cnt); c.match_key = (uint32_t *)(base + o_mk);
    c.tile_base = (int32_t *)(base + o_tb); c.ablock_base = (int32_t *)(base + o_ab);
    c.status = (uint8_t *)(base + o_st); c.small = (SmallInfo *)(base + o_small); c.plan = (PlanInfo *)(base + o_plan);
    c.row_pos = (int32_t *)(base + o_rpos);
    // candidate records of the pass; the edges themselves live in the caller's exchange buffer
    c.cand = (unsigned long long *)(base + o_cand);
    c.cand_cnt = (int32_t *)(base + o_ccnt); c.ledge_cnt = c.cand_cnt;   // (ledge_cnt is only reset by the planner here)
    c.thr = (uint32_t *)(base + o_thr); c.pstat = (PairStat *)(base + o_pstat);
    c.timeline = nullptr;
    sh->coldead = (uint8_t *)(base + o_dead);
    sh->blockcnt = (int32_t *)(base + o_bcnt);
    sh->ctl = (ShardCtl *)(base + o_ctl);
    sh->dev = (ShardDev *)(base + o_dev);
    sh->rbest_g = (uint32_t *)(base + o_rbg); sh->cbest_g = (uint32_t *)(base + o_cbg);
    PairPack pack{};
    pack.p[0].q = (const uint32_t *)d_q; pack.p[0].t = (const uint32_t *)d_t_local;
    pack.p[0].n1 = n1; pack.p[0].n2 = n2_local; pack.p[0].row_base = 0; pack.p[0].col_base = 0; pack.p[0].out_base = 0;
    pack.p[0].col_id_offset = col_offset; pack.p[0].flags = PAIR_FLAG_NO_FINISHER | PAIR_FLAG_SHARD;
    pack.p[0].cand_off = 0; pack.p[0].cand_cap = sh->raw_cap;
    CU_CHECK(h, cudaMemsetAsync(c.plan, 0, sizeof(PlanInfo), s));
    CU_CHECK(h, cudaMemsetAsync(sh->coldead, 0, (size_t)n2_total, s));
    CU_CHECK(h, cudaMemsetAsync(sh->ctl, 0, sizeof(ShardCtl), s));
    CU_CHECK(h, cudaMemsetAsync(sh->rbest_g, 0xFF, 4 * rows, s));
    CU_CHECK(h, cudaMemsetAsync(sh->cbest_g, 0xFF, 4 * (size_t)n2_total, s));
    dim3 igrid(std::max(1, std::min((std::max(n1, n2_local) + ACCEPT_THREADS - 1) / ACCEPT_THREADS, 64)), 1);
    init_kernel<true><<<igrid, ACCEPT_THREADS, 0, s>>>(c, pack);
    CU_CHECK(h, cudaGetLastError());
    *out = sh;
    return PGM_OK;
}

extern "C" int pgm_shard_edge_capacity(int32_t n1, int32_t n2_total, int32_t n_ranks, int32_t *out_cap) {
    if (!out_cap || n1 < 1 || n2_total < 1 || n_ranks < 1) return PGM_E_INVALID_ARG;
    *out_cap = shard_edge_capacity(n1, n2_total, n_ranks);
    return PGM_OK;
}

// enqueue: local round r, then this rank's contribution to the exchange into d_x[2 * bound] (bound >= live rows)
static int shard_enqueue_round(pgm_shard *sh, uint32_t *d_x, int bound, cudaStream_t s) {
    pgm_handle *h = sh->h;
    CU_CHECK(h, cudaMemsetAsync(sh->dev, 0, sizeof(ShardDev), s));
    dispatch_round(sh->words, sh->c, sh->round, sh->round_grid, s);
    const int g = std::max(1, std::min((bound + 255) / 256, h->num_sms * 8));
    shard_export_rows_kernel<<<g, 256, 0, s>>>(sh->c, sh->round, d_x, bound);
    const int gc = std::max(1, std::min((sh->n2_local + 255) / 256, h->num_sms * 8));
    shard_propose_cols_kernel<<<gc, 256, 0, s>>>(sh->c, sh->round, d_x, bound);
    h->stats.kernel_launches += 3;
    return PGM_OK;
}

// enqueue: commit step 1 + 2 from the reduced exchange buffer: matches, dead flags, this rank's filtered candidate edges
// into d_edges[1 + edge_cap] (d_edges[0] = count, or the overflow marker)
static int shard_enqueue_commit(pgm_shard *sh, const uint32_t *d_x, int bound, unsigned long long *d_edges, int edge_cap,
                                cudaStream_t s) {
    pgm_handle *h = sh->h;
    const int r = sh->round;
    const int nb = std::max(1, (std::min(bound, sh->n1) + SHARD_BLOCK - 1) / SHARD_BLOCK);
    shard_commit_mark_kernel<<<nb, SHARD_BLOCK, 0, s>>>(sh->c, r, d_x, bound, sh->coldead);
    h->stats.kernel_launches += 1;
    if (d_edges) {
        shard_filter_kernel<<<h->num_sms * 4, ACCEPT_THREADS, 0, s>>>(sh->c, r, sh->coldead, d_edges, edge_cap, &sh->dev->edge_cnt,
                                                                     &sh->dev->ticket);
        h->stats.kernel_launches += 1;
    }
    return PGM_OK;
}

// enqueue: commit steps 3-6: grid-wide sparse sub-rounds over every rank's edges, stable row compaction, columns, plan
static int shard_enqueue_finish_round(pgm_shard *sh, const unsigned long long *d_edges_all, int n_ranks, int edge_cap,
                                      cudaStream_t s) {
    pgm_handle *h = sh->h;
    const int r = sh->round;
    if (d_edges_all && n_ranks >= 1) {
        int rc = ensure_dev(h, sh->est, (size_t)n_ranks * edge_cap);
        if (rc) return rc;
        Chunk c = sh->c;
        uint32_t *rb = sh->rbest_g, *cb = sh->cbest_g;
        uint8_t *cd = sh->coldead, *est = (uint8_t *)sh->est.p;
        unsigned *bar = &sh->dev->bar;
        int32_t *alive = sh->dev->alive;
        void *args[] = {&c, &d_edges_all, &n_ranks, &edge_cap, &rb, &cb, &cd, &est, &bar, &alive};
        CU_CHECK(h, cudaLaunchCooperativeKernel((void *)shard_sparse_kernel, dim3(h->num_sms), dim3(TAIL_THREADS), args, 0, s));
        h->stats.kernel_launches += 1;
    }
    const int nb = (sh->n1 + SHARD_BLOCK - 1) / SHARD_BLOCK;
    shard_count_kernel<<<nb, SHARD_BLOCK, 0, s>>>(sh->c, r, sh->blockcnt);
    shard_commit_scatter_kernel<<<nb, SHARD_BLOCK, 0, s>>>(sh->c, r, sh->blockcnt, nb, sh->ctl, sh->n1, sh->n2_total);
    const int g2 = std::max(1, std::min((sh->n2_local + ACCEPT_THREADS - 1) / ACCEPT_THREADS, h->num_sms * 8));
    shard_commit_cols_kernel<<<g2, ACCEPT_THREADS, 0, s>>>(sh->c, r, sh->coldead, sh->ctl);
    h->stats.kernel_launches += 3;
    sh->round = r + 1;
    return PGM_OK;
}

// Step 1: local round; d_x (device, uint32[2 * bound], bound >= the live rows, e.g. n1) receives this rank's [R | P].
extern "C" int pgm_shard_round(pgm_shard *sh, uint32_t *d_x, int32_t bound) {
    if (!sh || !d_x || bound < 1) return PGM_E_INVALID_ARG;
    pgm_handle *h = sh->h;
    std::lock_guard<std::mutex> lk(h->mu);
    CU_CHECK(h, cudaSetDevice(h->device));
    int rc = shard_enqueue_round(sh, d_x, bound, h->stream);
    if (rc) return rc;
    CU_CHECK(h, cudaGetLastError());
    return PGM_OK;
}

// Step 2 (d_x now min-reduced over the ranks): matches of the round; this rank's surviving candidate edges go to
// d_edges[1 + edge_cap] (count first).  d_edges may be NULL (no candidate edges: plain one-accept-per-round behaviour).
extern "C" int pgm_shard_commit(pgm_shard *sh, const uint32_t *d_x, int32_t bound, uint64_t *d_edges, int32_t edge_cap) {
    if (!sh || !d_x || bound < 1 || (d_edges && edge_cap < 1)) return PGM_E_INVALID_ARG;
    pgm_handle *h = sh->h;
    std::lock_guard<std::mutex> lk(h->mu);
    CU_CHECK(h, cudaSetDevice(h->device));
    int rc = shard_enqueue_commit(sh, d_x, bound, (unsigned long long *)d_edges, edge_cap, h->stream);
    if (rc) return rc;
    CU_CHECK(h, cudaGetLastError());
    return PGM_OK;
}

// Step 3 (d_edges_all[n_ranks][1 + edge_cap] = every rank's edges, gathered; NULL skips the sparse phase): sparse
// sub-rounds, compaction, plan of the next round.  Returns the live rows (identical on all ranks) and whether the pair is
// finished.  Synchronises the stream (16 bytes read back).
extern "C" int pgm_shard_finish_round(pgm_shard *sh, const uint64_t *d_edges_all, int32_t n_ranks, int32_t edge_cap,
                                      int32_t *live_rows, int32_t *done) {
    if (!sh || (d_edges_all && (n_ranks < 1 || n_ranks > 64 || edge_cap < 1))) return PGM_E_INVALID_ARG;
    pgm_handle *h = sh->h;
    std::lock_guard<std::mutex> lk(h->mu);
    CU_CHECK(h, cudaSetDevice(h->device));
    cudaStream_t s = h->stream;
    int rc = shard_enqueue_finish_round(sh, (const unsigned long long *)d_edges_all, n_ranks, edge_cap, s);
    if (rc) return rc;
    CU_CHECK(h, cudaMemcpyAsync(sh->h_ctl, sh->ctl, sizeof(ShardCtl), cudaMemcpyDeviceToHost, s));
    CU_CHECK(h, cudaStreamSynchronize(s));
    if (live_rows) *live_rows = sh->h_ctl[0].live_rows;
    if (done) *done = sh->h_ctl[0].done;
    return PGM_OK;
}

static int shard_finish_locked(pgm_shard *sh, int32_t *d_out_qi, int32_t *d_out_tj, int32_t *d_out_dist, uint32_t flags,
                               cudaStream_t s) {
    pgm_handle *h = sh->h;
    // the order kernel derives the tail from min(n1, n2): it needs the TOTAL train size
    CU_CHECK(h, cudaMemcpyAsync((char *)sh->c.pairs + offsetof(PairDesc, n2), &sh->n2_total, 4, cudaMemcpyHostToDevice, s));
    const int nbins = 32 * sh->words + 1;     // padded width (see run_chunk)
    if (!h->order_attr_set) {
        CU_CHECK(h, cudaFuncSetAttribute(order_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)order_smem_bytes(513, ORDER_THREADS_STANDALONE)));
        h->order_attr_set = true;
    }
    if (!(flags & PGM_FLAG_REFERENCE_COMPAT_TAIL)) {
        CU_CHECK(h, cudaMemsetAsync(d_out_qi, 0xFF, (size_t)sh->n1 * 4, s));
        CU_CHECK(h, cudaMemsetAsync(d_out_tj, 0xFF, (size_t)sh->n1 * 4, s));
        CU_CHECK(h, cudaMemsetAsync(d_out_dist, 0xFF, (size_t)sh->n1 * 4, s));
    }
    order_kernel<<<1, ORDER_THREADS_STANDALONE, order_smem_bytes(nbins, ORDER_THREADS_STANDALONE), s>>>(
        sh->c, nbins, flags, d_out_qi, d_out_tj, d_out_dist);
    h->stats.kernel_launches += 1;
    CU_CHECK(h, cudaGetLastError());
    return PGM_OK;
}

// Final step: every rank holds every accepted (row -> global column, distance); emit them in the
// reference's order into device arrays of n1 triples (tail included with PGM_FLAG_REFERENCE_COMPAT_TAIL).
extern "C" int pgm_shard_finish(pgm_shard *sh, int32_t *d_out_qi, int32_t *d_out_tj, int32_t *d_out_dist, uint32_t flags,
                                int32_t *out_count, int32_t *out_rounds) {
    if (!sh || !d_out_qi || !d_out_tj || !d_out_dist) return PGM_E_INVALID_ARG;
    pgm_handle *h = sh->h;
    std::lock_guard<std::mutex> lk(h->mu);
    CU_CHECK(h, cudaSetDevice(h->device));
    cudaStream_t s = h->stream;
    int rc = shard_finish_locked(sh, d_out_qi, d_out_tj, d_out_dist, flags, s);
    if (rc) return rc;
    CU_CHECK(h, cudaMemcpyAsync(sh->h_ctl, sh->ctl, sizeof(ShardCtl), cudaMemcpyDeviceToHost, s));
    CU_CHECK(h, cudaStreamSynchronize(s));
    if (out_count) *out_count = out_count_for(sh->n1, sh->n2_total, flags);
    if (out_rounds) *out_rounds = sh->h_ctl[0].rounds;
    return PGM_OK;
}

extern "C" int pgm_shard_destroy(pgm_shard *sh) {
    if (!sh) return PGM_E_INVALID_ARG;
    pgm_handle *h = sh->h;
    std::lock_guard<std::mutex> lk(h->mu);
    cudaSetDevice(h->device);
    // park the buffers in the handle for the next shard (stream order protects them: every later use is enqueued on
    // the same stream); free only what the pool already holds
    if (sh->state.p && !h->shard_pool_state.p) { h->shard_pool_state = sh->state; sh->state = DevBuf{}; }
    if (sh->est.p && !h->shard_pool_est.p) { h->shard_pool_est = sh->est; sh->est = DevBuf{}; }
    if (sh->h_ctl && !h->shard_pool_hctl) { h->shard_pool_hctl = sh->h_ctl; sh->h_ctl = nullptr; }
    if (sh->state.p || sh->est.p || sh->h_ctl) {
        cudaStreamSynchronize(h->stream);
        if (sh->state.p) cudaFree(sh->state.p);
        if (sh->est.p) cudaFree(sh->est.p);
        if (sh->h_ctl) cudaFreeHost(sh->h_ctl);
    }
    delete sh;
    return PGM_OK;
}

// ---------------------------------------------------------------------------
// pgm_multi: one rank of a multi-GPU job, the library owning the NCCL communicator (SURVEY.md section 8b, threading
// row).  NCCL is resolved at run time (dlopen): the single-GPU entry points carry no dependency on it, and a process
// that already loaded NCCL (torch's bundled copy) shares that copy instead of loading a second one.
// ---------------------------------------------------------------------------
#include <dlfcn.h>
namespace {
struct NcclUniqueIdBlob { char internal[128]; };          // == ncclUniqueId (NCCL_UNIQUE_ID_BYTES = 128, stable across 2.x)
struct NcclApi {
    void *lib = nullptr;
    int (*GetUniqueId)(NcclUniqueIdBlob *) = nullptr;
    int (*CommInitRank)(void **, int, NcclUniqueIdBlob, int) = nullptr;
    int (*CommDestroy)(void *) = nullptr;
    int (*AllReduce)(const void *, void *, size_t, int, int, void *, cudaStream_t) = nullptr;
    int (*AllGather)(const void *, void *, size_t, int, void *, cudaStream_t) = nullptr;
    const char *(*GetErrorString)(int) = nullptr;
    std::string why;
};
constexpr int kNcclInt32 = 2, kNcclUint32 = 3, kNcclUint64 = 5, kNcclMin = 3;   // ncclDataType_t / ncclRedOp_t values (nccl.h, 2.x)
NcclApi *nccl_api() {
    static NcclApi api;
    static std::once_flag once;
    std::call_once(once, [] {
        const char *names[] = {"libnccl.so.2", "libnccl.so"};
        for (const char *n : names) { api.lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL); if (api.lib) break; }
        if (!api.lib) { api.why = std::string("cannot load libnccl.so.2: ") + (dlerror() ? dlerror() : "?"); return; }
        auto sym = [&](const char *n) { void *p = dlsym(api.lib, n); if (!p && api.why.empty()) api.why = std::string("missing NCCL symbol ") + n; return p; };
        api.GetUniqueId = (decltype(api.GetUniqueId))sym("ncclGetUniqueId");
        api.CommInitRank = (decltype(api.CommInitRank))sym("ncclCommInitRank");
        api.CommDestroy = (decltype(api.CommDestroy))sym("ncclCommDestroy");
        api.AllReduce = (decltype(api.AllReduce))sym("ncclAllReduce");
        api.AllGather = (decltype(api.AllGather))sym("ncclAllGather");
        api.GetErrorString = (decltype(api.GetErrorString))sym("ncclGetErrorString");
    });
    return &api;
}
}  // namespace

struct pgm_multi {
    pgm_handle *h = nullptr;
    void *comm = nullptr;
    int rank = 0, world = 1;
    DevBuf xbuf;                 // exchange buffer [2 * n1] / gathered keys
    DevBuf fin;                  // replicated finish: gathered rows / columns, sub-problem output
    int64_t exchange_bytes = 0;  // payload this rank contributed to collectives in the last call
    int32_t collectives = 0;
};

#define NCCL_CHECK(h, call)                                                                     \
    do {                                                                                        \
        int r__ = (call);                                                                       \
        if (r__ != 0) {                                                                         \
            (h)->err = std::string(#call " failed: ") + (nccl_api()->GetErrorString ? nccl_api()->GetErrorString(r__) : "?"); \
            return PGM_E_NCCL;                                                                  \
        }                                                                                       \
    } while (0)

extern "C" int pgm_multi_unique_id(uint8_t *out_id128) {
    if (!out_id128) return PGM_E_INVALID_ARG;
    NcclApi *a = nccl_api();
    if (!a->lib || !a->why.empty()) return PGM_E_NCCL;
    NcclUniqueIdBlob id;
    if (a->GetUniqueId(&id) != 0) return PGM_E_NCCL;
    memcpy(out_id128, id.internal, 128);
    return PGM_OK;
}

extern "C" int pgm_multi_create(pgm_handle *h, const uint8_t *id128, int32_t rank, int32_t world, pgm_multi **out) {
    if (!h || !out || world < 1 || rank < 0 || rank >= world || (world > 1 && !id128)) return PGM_E_INVALID_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    *out = nullptr;
    pgm_multi *mh = new pgm_multi();
    mh->h = h; mh->rank = rank; mh->world = world;
    if (world > 1) {
        NcclApi *a = nccl_api();
        if (!a->lib || !a->why.empty()) { h->err = a->why.empty() ? "NCCL unavailable" : a->why; delete mh; return PGM_E_NCCL; }
        if (cudaSetDevice(h->device) != cudaSuccess) { delete mh; return PGM_E_CUDA; }
        NcclUniqueIdBlob id;
        memcpy(id.internal, id128, 128);
        const int r = a->CommInitRank(&mh->comm, world, id, rank);
        if (r != 0) { h->err = std::string("ncclCommInitRank failed: ") + a->GetErrorString(r); delete mh; return PGM_E_NCCL; }
    }
    *out = mh;
    return PGM_OK;
}

extern "C" int pgm_multi_destroy(pgm_multi *mh) {
    if (!mh) return PGM_E_INVALID_ARG;
    pgm_handle *h = mh->h;
    {
        std::lock_guard<std::mutex> lk(h->mu);
        cudaSetDevice(h->device);
        cudaStreamSynchronize(h->stream);
        if (mh->comm) nccl_api()->CommDestroy(mh->comm);
        if (mh->xbuf.p) cudaFree(mh->xbuf.p);
        if (mh->fin.p) cudaFree(mh->fin.p);
    }
    delete mh;
    return PGM_OK;
}

extern "C" int pgm_multi_get_exchange(pgm_multi *mh, int64_t *bytes, int32_t *collectives) {
    if (!mh) return PGM_E_INVALID_ARG;
    if (bytes) *bytes = mh->exchange_bytes;
    if (collectives) *collectives = mh->collectives;
    return PGM_OK;
}

// Once at most SHARD_FINISH_MAX rows and columns are left, the remaining rounds would be a few microseconds of work each
// behind two collectives and a dozen launches.  Instead every rank gathers the descriptors of ALL surviving rows (it holds
// every query) and columns (one all-gather of the ranks' surviving train rows, ascending) and finishes the remaining small
// problem itself with the single-GPU engine -- identical input on every rank, hence identical matches.  The gathered
// indices are order-preserving (the row list is compacted stably, the columns are packed ascending), so the engine's
// (distance, i, j) tie-break in sub-problem indices is the reference's tie-break in original indices.
constexpr int SHARD_FINISH_MAX = 12288;
static int shard_replicated_finish(pgm_multi *mh, pgm_shard *sh, int live_rows, cudaStream_t s) {
    pgm_handle *h = sh->h;
    const int words = sh->words, stride = words * 4;
    const int Lr = live_rows, Lc = sh->n2_total - (sh->n1 - live_rows);
    if (Lr <= 0 || Lc <= 0) return PGM_OK;
    const int r = sh->round;                                   // the lists of the NEXT round hold the survivors
    const size_t blk_bytes = align_up(16 + align_up((size_t)Lc * 4, 16) + (size_t)Lc * stride, 256);
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return o; };
    const size_t o_q = take((size_t)Lr * stride), o_t = take((size_t)Lc * stride), o_gid = take((size_t)Lc * 4);
    const size_t o_out = take((size_t)3 * Lr * 4), o_flag = take(4), o_all = take(blk_bytes * mh->world);
    int rc = ensure_dev(h, mh->fin, off);
    if (rc) return rc;
    char *base = (char *)mh->fin.p;
    uint32_t *q_sub = (uint32_t *)(base + o_q), *t_sub = (uint32_t *)(base + o_t);
    int32_t *gid = (int32_t *)(base + o_gid), *oq = (int32_t *)(base + o_out), *ot = oq + Lr, *od = ot + Lr;
    int32_t *d_flag = (int32_t *)(base + o_flag);
    unsigned long long *all = (unsigned long long *)(base + o_all);
    unsigned long long *mine = (unsigned long long *)((char *)all + blk_bytes * mh->rank);
    CU_CHECK(h, cudaMemsetAsync(d_flag, 0, 4, s));
    const uint32_t *qd = sh->q_host_ptr, *td = sh->t_host_ptr;
    shard_gather_rows_kernel<<<std::min((Lr * (words / 4) + 255) / 256, h->num_sms * 8), 256, 0, s>>>(
        qd, sh->c.live_rows[r & 1], Lr, words, q_sub);
    shard_pack_cols_kernel<<<1, 1024, 0, s>>>(td, sh->n2_local, sh->col_offset, words, sh->coldead, Lc, mine);
    if (mh->world > 1) {
        NCCL_CHECK(h, nccl_api()->AllGather(mine, all, blk_bytes / 8, kNcclUint64, mh->comm, s));
        mh->exchange_bytes += (int64_t)blk_bytes; mh->collectives++;
    }
    shard_merge_cols_kernel<<<std::min((Lc + 255) / 256, h->num_sms * 8), 256, 0, s>>>(all, blk_bytes / 8, mh->world, Lc, words,
                                                                                   t_sub, gid, Lc, d_flag);
    h->stats.kernel_launches += 3;
    HostPair hp{(const uint8_t *)q_sub, (const uint8_t *)t_sub, Lr, Lc, 0};
    const pgm_stats keep = h->stats;
    rc = run_chunk(h, &hp, 1, sh->desc_bits, stride, 0u, oq, ot, od);
    if (rc) return rc;
    const int launches = h->stats.kernel_launches;
    h->stats = keep; h->stats.kernel_launches = launches; h->stats_pending = false;
    const int nm = std::min(Lr, Lc);
    shard_map_matches_kernel<<<std::min((nm + 255) / 256, h->num_sms * 8), 256, 0, s>>>(oq, ot, od, nm, sh->c.live_rows[r & 1], gid,
                                                                                    sh->c.match_key);
    h->stats.kernel_launches += 1;
    int32_t flag = 0;
    CU_CHECK(h, cudaMemcpyAsync(&flag, d_flag, 4, cudaMemcpyDeviceToHost, s));
    CU_CHECK(h, cudaStreamSynchronize(s));
    if (flag) return fail(h, PGM_E_CUDA, "train-sharded finish: the ranks' surviving columns do not add up (internal error)");
    return PGM_OK;
}

// MatchKeypoints on ONE pair whose train set is sharded over the ranks: d_q = all queries, d_t_local = train rows
// [col_offset, col_offset + n2_local).  Collective: every rank of the communicator must call it with the same n1,
// n2_total, format and flags.  Writes the n1 (or min) triples, identical on every rank.
extern "C" int pgm_multi_match_train_sharded_dev(pgm_multi *mh, const uint8_t *d_q, int32_t n1, const uint8_t *d_t_local,
                                                 int32_t n2_local, int32_t col_offset, int32_t n2_total, int32_t desc_bits,
                                                 int32_t stride_bytes, int32_t *d_out_qi, int32_t *d_out_tj,
                                                 int32_t *d_out_dist, int32_t capacity, int32_t *out_count, uint32_t flags,
                                                 int32_t *out_rounds) {
    if (!mh || !d_out_qi || !d_out_tj || !d_out_dist) return PGM_E_INVALID_ARG;
    pgm_handle *h = mh->h;
    const int32_t cnt = out_count_for(n1, n2_total, flags);
    if (out_count) *out_count = cnt;
    if (capacity < cnt) return fail(h, PGM_E_CAPACITY, "capacity < number of triples");
    pgm_shard *sh = nullptr;
    int rc = pgm_shard_create(h, d_q, n1, d_t_local, n2_local, col_offset, n2_total, desc_bits, stride_bytes, &sh);
    if (rc) return rc;
    {
        std::lock_guard<std::mutex> lk(h->mu);
        h->stats = pgm_stats{};
        mh->exchange_bytes = 0; mh->collectives = 0;
        if (cudaSetDevice(h->device) != cudaSuccess) { rc = PGM_E_CUDA; }
        cudaStream_t s = h->stream;
        const int edge_cap = shard_edge_capacity(n1, n2_total, mh->world);
        const bool edges_on = mh->world <= 64;
        const size_t x_bytes = align_up((size_t)2 * n1 * 4, 256);
        if (!rc) rc = ensure_dev(h, mh->xbuf, x_bytes + (edges_on ? (size_t)mh->world * (1 + (size_t)edge_cap) * 8 : 0));
        uint32_t *X = (uint32_t *)mh->xbuf.p;
        unsigned long long *E_all = edges_on ? (unsigned long long *)((char *)mh->xbuf.p + x_bytes) : nullptr;
        // Rounds while many rows are live (each is milliseconds of work: one 16-byte status read-back per round costs
        // nothing), then the replicated finish.  Every rank reads the same status, so all ranks take the same path.
        int bound = n1;
        bool done = false;
        const bool timing = getenv("PGM_SHARD_TIMING") != nullptr;      // debug: host wall time of every round (stream is idle at each mark)
        auto t_prev = std::chrono::steady_clock::now();
        auto mark = [&](const char *what, int a) {
            if (!timing) return;
            const auto now = std::chrono::steady_clock::now();
            fprintf(stderr, "[pgm shard rank %d] %s %d: %.3f ms\n", mh->rank, what, a, std::chrono::duration<double, std::milli>(now - t_prev).count());
            t_prev = now;
        };
        if (timing) { cudaStreamSynchronize(s); mark("create", 0); }
        while (!rc && !done) {
            if ((rc = shard_enqueue_round(sh, X, bound, s))) break;
            if (mh->world > 1) {
                const int r = nccl_api()->AllReduce(X, X, (size_t)2 * bound, kNcclUint32, kNcclMin, mh->comm, s);
                if (r != 0) { h->err = std::string("ncclAllReduce failed: ") + nccl_api()->GetErrorString(r); rc = PGM_E_NCCL; break; }
                mh->exchange_bytes += (int64_t)2 * bound * 4; mh->collectives++;
            }
            // the pass cannot list more than p_max x live rows x live columns edges (plan_pair_emit's density clamp,
            // <= 0.05): late rounds exchange small edge blocks.  `bound` is the same on every rank, hence so is the block size.
            const double live_cols_max = (double)bound + (double)std::max(0, n2_total - n1);     // live columns = total - matched rows
            const int cap_r = (int)std::min<int64_t>(edge_cap, (int64_t)(0.06 * (double)bound * live_cols_max) + 4096);
            unsigned long long *E_mine_r = edges_on ? E_all + (size_t)mh->rank * (1 + (size_t)cap_r) : nullptr;
            if ((rc = shard_enqueue_commit(sh, X, bound, E_mine_r, cap_r, s))) break;
            if (edges_on && mh->world > 1) {      // in place: this rank's block already sits at its slot of the gathered buffer
                const int r = nccl_api()->AllGather(E_mine_r, E_all, (size_t)(1 + cap_r), kNcclUint64, mh->comm, s);
                if (r != 0) { h->err = std::string("ncclAllGather failed: ") + nccl_api()->GetErrorString(r); rc = PGM_E_NCCL; break; }
                mh->exchange_bytes += (int64_t)(1 + cap_r) * 8; mh->collectives++;
            }
            if ((rc = shard_enqueue_finish_round(sh, E_all, mh->world, cap_r, s))) break;
            if (cudaMemcpyAsync(&sh->h_ctl[0], sh->ctl, sizeof(ShardCtl), cudaMemcpyDeviceToHost, s) != cudaSuccess ||
                cudaStreamSynchronize(s) != cudaSuccess) { rc = PGM_E_CUDA; break; }
            h->stats.host_syncs++;
            const int live = sh->h_ctl[0].live_rows;
            done = sh->h_ctl[0].done != 0;
            mark("round, live rows after", live);
            bound = std::min(bound, std::max(SHARD_BLOCK, (live + SHARD_BLOCK - 1) / SHARD_BLOCK * SHARD_BLOCK));
            if (!done && live <= SHARD_FINISH_MAX && (int64_t)n2_total - (n1 - live) <= SHARD_FINISH_MAX) {
                rc = shard_replicated_finish(mh, sh, live, s);
                done = true;
                mark("replicated finish of rows", live);
            }
            if (sh->round > 4 * MAX_N) { h->err = "train-sharded matcher failed to converge (internal error)"; rc = PGM_E_CUDA; }
        }
        if (!rc) rc = shard_finish_locked(sh, d_out_qi, d_out_tj, d_out_dist, flags, s);
        if (!rc && cudaMemcpyAsync(&sh->h_ctl[0], sh->ctl, sizeof(ShardCtl), cudaMemcpyDeviceToHost, s) != cudaSuccess) rc = PGM_E_CUDA;
        if (!rc && cudaStreamSynchronize(s) != cudaSuccess) rc = PGM_E_CUDA;
        if (!rc) {
            h->stats.host_syncs++;
            h->stats.rounds = sh->h_ctl[0].rounds;
            h->stats.distance_evals = (int64_t)n1 * n2_local;
            h->stats.matched = std::min(n1, n2_total);
            h->stats.pairs = 1;
            if (out_rounds) *out_rounds = sh->h_ctl[0].rounds;
        } else if (rc == PGM_E_CUDA && h->err.empty()) {
            h->err = std::string("CUDA error in the train-sharded matcher: ") + cudaGetErrorString(cudaGetLastError());
        }
    }
    pgm_shard_destroy(sh);
    return rc;
}

// Nearest / second-nearest neighbour of every query over a train set sharded across the ranks: local search, packed
// (distance << 20 | GLOBAL train index) keys, ONE all-gather of [2][n1] keys per rank, top-2 merge (north_star:
// "train-set shard with a top-2 merge").  Identical results on every rank.
extern "C" int pgm_multi_knn2_train_sharded_dev(pgm_multi *mh, const uint8_t *d_q, int32_t n1, const uint8_t *d_t_local,
                                                int32_t n2_local, int32_t col_offset, int32_t desc_bits,
                                                int32_t stride_bytes, int32_t *d_best_j, int32_t *d_best_d,
                                                int32_t *d_second_j, int32_t *d_second_d) {
    if (!mh || !d_best_j || !d_best_d || !d_second_j || !d_second_d) return PGM_E_INVALID_ARG;
    pgm_handle *h = mh->h;
    int rc = pgm_knn2_hamming_dev(h, d_q, n1, d_t_local, n2_local, desc_bits, stride_bytes, d_best_j, d_best_d, d_second_j, d_second_d);
    if (rc) return rc;
    if (n1 == 0) return PGM_OK;
    {
        std::lock_guard<std::mutex> lk(h->mu);
        CU_CHECK(h, cudaSetDevice(h->device));
        if ((rc = ensure_dev(h, mh->xbuf, (size_t)(mh->world + 1) * 2 * n1 * 4))) return rc;
        mh->exchange_bytes = 0; mh->collectives = 0;
    }
    uint32_t *mine = (uint32_t *)mh->xbuf.p, *all = mine + (size_t)2 * n1;
    if ((rc = pgm_pack_top2_keys_dev(h, d_best_j, d_best_d, d_second_j, d_second_d, n1, col_offset, (int32_t *)mine))) return rc;
    if (mh->world > 1) {
        std::lock_guard<std::mutex> lk(h->mu);
        NCCL_CHECK(h, nccl_api()->AllGather(mine, all, (size_t)2 * n1, kNcclInt32, mh->comm, h->stream));
        mh->exchange_bytes = (int64_t)2 * n1 * 4; mh->collectives = 1;
    } else {
        all = mine;
    }
    return pgm_merge_top2_dev(h, (const int32_t *)all, mh->world, n1, d_best_j, d_best_d, d_second_j, d_second_d);
}

// ---------------------------------------------------------------------------
// profiling mode
// ---------------------------------------------------------------------------
extern "C" int pgm_set_profiling(pgm_handle *h, int32_t enabled) {
    if (!h) return PGM_E_INVALID_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    CU_CHECK(h, cudaSetDevice(h->device));
    if (enabled && h->prof_events.empty()) {
        h->prof_events.resize(2 * PROF_MAX_ROUNDS);
        for (auto &e : h->prof_events) CU_CHECK(h, cudaEventCreate(&e));
        int rc = ensure_host(h, h->pin_prof, sizeof(PlanInfo) * (PROF_MAX_ROUNDS + 2));
        if (rc) return rc;
    }
    h->profiling = enabled != 0;
    h->prof_rounds = 0;
    return PGM_OK;
}

extern "C" int pgm_get_round_profile(pgm_handle *h, float *ms, int64_t *evals, int32_t capacity, int32_t *out_n) {
    if (!h || !out_n) return PGM_E_INVALID_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    CU_CHECK(h, cudaSetDevice(h->device));
    CU_CHECK(h, cudaStreamSynchronize(h->stream));
    const PlanInfo *pp = (const PlanInfo *)h->pin_prof.p;
    int n = 0;
    for (int r = 0; r < h->prof_rounds && n < capacity; r++) {
        const int64_t e = (int64_t)pp[r].evals - (r > 0 ? (int64_t)pp[r - 1].evals : 0);
        if (e <= 0) continue;                       // idle round (pair already small/done)
        float t = 0.f;
        CU_CHECK(h, cudaEventElapsedTime(&t, h->prof_events[2 * r], h->prof_events[2 * r + 1]));
        if (ms) ms[n] = t;
        if (evals) evals[n] = e;
        n++;
    }
    *out_n = n;
    return PGM_OK;
}

// ---------------------------------------------------------------------------
// roofline denominators
// ---------------------------------------------------------------------------
extern "C" int pgm_measure_popc_peak(pgm_handle *h, int32_t millis, double *popc32_per_s, double *lop3_per_s) {
    if (!h) return PGM_E_INVALID_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    CU_CHECK(h, cudaSetDevice(h->device));
    cudaStream_t s = h->stream;
    const int threads = 256, blocks = h->num_sms * 8, iters = 4096;
    int rc = ensure_dev(h, h->misc, (size_t)threads * blocks * 4);
    if (rc) return rc;
    cudaEvent_t e0, e1;
    CU_CHECK(h, cudaEventCreate(&e0));
    CU_CHECK(h, cudaEventCreate(&e1));
    const double ops_per_launch = (double)threads * blocks * iters * 32.0;   // 4 x 8 per iteration
    for (int which = 0; which < 2; which++) {
        double best = 0.0;
        auto t0 = std::chrono::steady_clock::now();
        int reps = 0;
        do {
            CU_CHECK(h, cudaEventRecord(e0, s));
            if (which == 0) popc_peak_kernel<<<blocks, threads, 0, s>>>((uint32_t *)h->misc.p, iters, 12345u + reps);
            else lop3_peak_kernel<<<blocks, threads, 0, s>>>((uint32_t *)h->misc.p, iters, 12345u + reps);
            CU_CHECK(h, cudaEventRecord(e1, s));
            CU_CHECK(h, cudaEventSynchronize(e1));
            float ms = 0.f;
            CU_CHECK(h, cudaEventElapsedTime(&ms, e0, e1));
            if (reps >= 2) best = std::max(best, ops_per_launch / (ms * 1e-3));
            reps++;
        } while (reps < 4 || std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count() <
                                 millis / 2.0);
        if (which == 0 && popc32_per_s) *popc32_per_s = best;
        if (which == 1 && lop3_per_s) *lop3_per_s = best;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    return PGM_OK;
}
