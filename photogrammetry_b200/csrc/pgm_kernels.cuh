// pgm_kernels.cuh -- sm_100a kernels of the descriptor-matching path.
//
// Reference path: ImageProcessing.KeypointMatching.MatchKeypoints
//   dotnet_src/ImageProcessing/KeypointMatching.cs:14-69 (+ CountOnes :71-82).
// The reference builds the full N1 x N2 Hamming matrix and then removes the
// global (distance, i, j)-minimum N1 times.  Here the same assignment is
// computed as iterated mutual-nearest-neighbour rounds (DESIGN.md section 3):
//
//   round kernel   distances of live rows x live columns, fused with the
//                  per-row argmin (registers) and per-column argmin (REDUX +
//                  shared/global atomicMin) over packed (distance<<20 | index)
//                  keys, so an integer min IS the reference tie-break
//                  (KeypointMatching.cs:44-54: ascending i, ascending j, strict <)
//   accept kernel  rows/columns that chose each other are matched and retired,
//                  survivors are compacted
//   candidate edges  every distance pass also keeps EVERY edge with distance <= T (T from a
//                  Gaussian fit of sampled distances, so a row sees a handful).  That edge set is
//                  complete up to T on both sides, hence the greedy matching restricted to it is a
//                  prefix of the reference's matching: one CTA per pair runs mutual-best
//                  "sub-rounds" on the sparse list out of shared memory (no distance is
//                  recomputed), then re-compacts the survivors and plans the next pass.  Uniform
//                  8192 x 8192: live rows per distance pass 8192 -> 1236 -> 172 instead of
//                  8192 -> 4155 -> 2352 -> 1362 -> 782 -> 454 -> 255 (tools/sim_threshold_rounds.py)
//   finisher       once a pair is small, one CTA runs all remaining rounds out
//                  of a distance matrix held in shared memory
//   order kernel   stable counting sort of the matches by distance -> the
//                  reference's output order, plus the n1>n2 tail (:38-42)
//
// Nothing here is translated from the reference (it has no native code).
#pragma once

#include <algorithm>
#include <cstdint>
#include <cuda_runtime.h>

#include <cstdio>

// Checked build (make checked -> libpgmatch_checked.so, loaded with PGM_LIB=...): every index a kernel derives from
// data another kernel or CTA produced -- packed keys, candidate records, list positions, output slots -- is range
// checked on the device and a violation traps.  compute-sanitizer is closed on this pool (it left GPUs needing a reset),
// so this build, run on the small cases of tools/sanitize_cases.py, is the memory-safety evidence (profiles/r02_checked_build.log).
#ifdef PGM_CHECKED
#define PGM_ASSERT(cond)                                                                                          \
    do {                                                                                                          \
        if (!(cond)) {                                                                                            \
            printf("PGM_ASSERT failed: %s  (%s:%d, block %d thread %d)\n", #cond, __FILE__, __LINE__, (int)blockIdx.x, \
                   (int)threadIdx.x);                                                                             \
            __trap();                                                                                             \
        }                                                                                                         \
    } while (0)
#else
#define PGM_ASSERT(cond) ((void)0)
#endif

namespace pgm {

constexpr uint32_t KEY_IDX_BITS = 20;
constexpr uint32_t KEY_IDX_MASK = (1u << KEY_IDX_BITS) - 1u;
constexpr uint32_t KEY_NONE = 0xFFFFFFFFu;
// Index part of a padded (non-existent) row/column slot: with distance <= 512,
// (d << 20) + KEY_INVALID never overflows and always exceeds every real key.
constexpr uint32_t KEY_INVALID = 0xDFFFFFFFu;
constexpr int MAX_N = 1 << KEY_IDX_BITS;

constexpr int ROUND_THREADS = 128;    // 4 warps per CTA
constexpr int RQ_LARGE = 4;           // query rows per thread, large tiles
constexpr int STAGE_LARGE = 64;       // train descriptors staged in smem per step, large tiles
constexpr int RQ_SMALL = 1;           // small tiles: late rounds, where the machine would otherwise idle
constexpr int STAGE_SMALL = 32;
constexpr int STAGE_COLS = STAGE_LARGE;
constexpr int ACCEPT_THREADS = 256;
constexpr int FIN_THREADS = 512;
constexpr int FIN_MAX_DIM = 512;      // (== FIN_THREADS) finisher takes a pair once nlr, nlc <= this ...
constexpr int FIN_MAX_EVALS = 49152;  // ... and nlr * nlc <= this (u16 distance matrix in smem)
// Latency mode (persistent tail kernel): the matrix and the first round's minima of a small pair are computed by
// ALL CTAs into global memory, so the single-CTA finisher can afford to start earlier (one grid round less).
constexpr int FIN_MAX_EVALS_TAIL = 65536;
constexpr int FIN_D_STRIDE = FIN_MAX_EVALS_TAIL + 4 * FIN_MAX_DIM;   // u16 cells per pair incl. row-pitch padding
constexpr uint32_t TAIL_FLAG_ACCEPT_FIRST = 0x80000000u;            // tail_kernel flags bit: run accept(r_start - 1) first
constexpr int FIN_PREP_MIN_EVALS = 8192;                            // below this the finisher CTA computes its matrix itself
constexpr int FIN_SEG = 128;                                        // entries of a row / column one warp handles
constexpr int FIN_PARTS = FIN_MAX_DIM / FIN_SEG;                    // partial minima per row / column
constexpr int ORDER_THREADS_STANDALONE = 1024;
constexpr int TAIL_THREADS = 512;     // persistent tail kernel: 1 CTA per SM, four 128-thread groups
constexpr int ORDER_KEY_CACHE = 16384;  // match keys cached in smem by the order kernel
static_assert(TAIL_THREADS == 512, "the sparse phase and the ordering slices assume 512-thread CTAs");
// candidate edges / sparse sub-rounds
constexpr int SCAND = 512;              // candidate records a tile stages in shared memory between two global appends
constexpr int SP_THREADS = 512;         // threads of the CTA that runs a pair's sparse sub-rounds
constexpr int SP_EPT = 32;              // live edges a thread of the sparse phase holds at most (its private column of shared memory)
constexpr int SP_B = 4;                 // edges are processed in batches of SP_B: loads of a batch first, then its stores
constexpr int SP_LB = 8;                // edges a thread loads from the global list at a time
constexpr int SP_IPT = 8;               // ids a thread re-compacts at a time
constexpr int SP_SMEM_BYTES = 224 * 1024;   // shared memory of a sparse phase: the edges (8 or 12 bytes each)
                                            // and one min slot per live row and live column
constexpr int SP_LCAP_MAX = SP_THREADS * SP_EPT;   // live edges per pair the global list is sized for
constexpr int SP_MAX_SUB = 64;          // sub-rounds per sparse phase (each accepts >= 1 pair; the rest waits for the next pass)
constexpr float CAND_TARGET = 6.0f;     // expected candidate edges per row of the larger side and pass: a few pairs ...
constexpr float CAND_TARGET_BATCH = 6.0f;   // ... and batches of pairs
constexpr uint32_t KEY_DEAD = 0xFFFFFFFEu;  // sparse phase: row / column matched in an earlier sub-round

enum PairStatus : uint8_t { PAIR_DONE = 0, PAIR_BIG = 1, PAIR_SMALL = 2 };

struct PairDesc {
    const uint32_t *q;   // query descriptors (row-major, `words` u32 per row)
    const uint32_t *t;   // train descriptors
    int32_t n1, n2;
    int64_t row_base;    // first slot of this pair in the per-row state arrays
    int64_t col_base;    // first slot in the per-column state arrays
    int64_t out_base;    // where this pair's triples start in the output arrays
    int32_t col_id_offset;   // added to train indices inside keys (train-sharded mode: global column ids)
    int32_t flags;           // PAIR_FLAG_*
    int64_t cand_off;        // this pair's region of Chunk::cand (raw candidate edges of the current pass)
    int64_t ledge_off;       // this pair's region of Chunk::ledge (candidate edges whose endpoints survived the accept)
    int32_t cand_cap, ledge_cap;
};
constexpr int PAIR_FLAG_NO_FINISHER = 1;   // never hand this pair to the single-CTA finisher
constexpr int PAIR_FLAG_SHARD = 4;         // one rank's slice of a train-sharded pair (keys carry global column ids)

struct PairStat {            // per pair, written by the init kernel
    float mu, sd;            // mean / standard deviation of a sample of this pair's distances
    float cscale;            // multiplies CAND_TARGET; quartered whenever a pass overflowed the candidate list
    int32_t pad;
};

struct SmallInfo {       // written when the planner hands a pair to the finisher
    int32_t nlr, nlc, parity, pad;
};

struct PlanInfo {                 // device resident, rewritten every round
    int32_t total_tiles;          // round-kernel work items
    int32_t cols_per_tile;        // column extent of one tile (multiple of the stage size)
    int32_t total_ablocks;        // accept-kernel work items
    int32_t n_big;                // pairs still on grid rounds
    int32_t n_small;              // pairs waiting for the finisher
    int32_t round;
    uint32_t ticket;              // last-block-done counter (init and accept kernels)
    int32_t done_round_p1;        // 1 + first round whose plan found no PAIR_BIG pair (0: not yet)
    int32_t rq;                   // rows per thread this round (RQ_LARGE or RQ_SMALL)
    uint32_t grid_bar;            // grid-barrier counter of the persistent tail kernel
    unsigned long long evals;     // XOR+popcount evaluations planned so far (grid rounds)
};

// Latency mode keeps its PlanInfo in a per-handle allocation that the tail kernel leaves CLEAN (all zero) for the next
// call and reports the call's statistics through: a cudaMemsetAsync before and a 48-byte cudaMemcpyAsync after the
// three launches cost 5-8 us and 9-14 us of a 0.24 ms call.
struct LatState {
    PlanInfo plan;
    unsigned exit_cnt;                // CTAs of the tail kernel that have finished
    unsigned pad;
    unsigned long long last_rounds;   // statistics of the last call (read back on demand: pgm_get_stats)
    unsigned long long last_evals;
};

struct Chunk {
    PairDesc *pairs;
    int32_t n_pairs;
    int32_t num_sms;
    int32_t ctas_per_sm;          // resident round-kernel CTAs per SM
    int32_t ctas_per_sm0;         // the same for round 0 when it runs as a standalone launch before the tail kernel (0: n/a)
    int32_t fin_max_evals;        // a pair goes to the finisher once nlr * nlc <= this (FIN_MAX_EVALS or _TAIL)
    uint32_t *rowbest[2];
    uint32_t *colbest[2];
    int32_t *live_rows[2];
    int32_t *live_cols[2];
    int32_t *counts;              // [3][n_pairs][2] live rows / live cols
    uint32_t *match_key;          // per row: accepted (d<<20 | j) or KEY_NONE
    int32_t *tile_base;           // [n_pairs + 1]
    int32_t *ablock_base;         // [n_pairs + 1]
    uint8_t *status;              // PairStatus per pair
    SmallInfo *small;             // per pair
    PlanInfo *plan;
    unsigned long long *timeline; // optional (PGM_TAIL_TIMELINE=1): globaltimer stamps of the tail kernel's phases
    uint16_t *fin_d;              // latency mode: [n_pairs][FIN_D_STRIDE] distance matrices written by finisher_prepare
    uint32_t *fin_rb, *fin_cb;    // latency mode: [n_pairs][FIN_PARTS][FIN_MAX_DIM] first-round row / column minima (partial)
    int32_t *fin_ids;             // latency mode: [n_pairs][2][FIN_MAX_DIM] rank-sorted row / column ids
    long long large_min_evals;    // a round with at least this many live cells uses the large (RQ = 4) tiles
    // candidate edges
    unsigned long long *cand;     // raw candidate records of the current pass, per pair region, two words each:
                                  // (d << 40 | i << 20 | j) with d <= T, and (RQ << 20 | first live-list slot of the emitting thread)
    unsigned long long *ledge;    // the raw edges whose row and column both survived the pass's accept
    int32_t *cand_cnt;            // [n_pairs] raw edges appended this pass (> cand_cap: overflow, list unusable)
    int32_t *ledge_cnt;           // [n_pairs]
    uint32_t *thr;                // [n_pairs] emission bound of the current pass as a key: (T + 1) << 20; 0 = none
    PairStat *pstat;              // [n_pairs]
    int32_t *row_pos, *col_pos;   // position of a surviving row / column in the next live list (written by accept)
    int32_t words;                // descriptor words (runtime copy of the kernels' template parameter)
    int32_t *order_cnt;           // latency mode: [n_pairs][ORDER_MAX_SLICES][ORDER_BIN_PITCH] per-slice distance histograms
    int32_t shard_n2_total;       // train-sharded pair: columns of the whole pair
    float cand_target;            // expected candidate edges per row of the smaller side (CAND_TARGET, _BATCH or _SHARD)
    float cand_row_max;           // upper bound of the per-row target of a pass (later passes: few live rows share the list budget)
    LatState *lat;                // latency mode: the self-cleaning plan + statistics block (plan == &lat->plan), else nullptr
    int32_t sp_slots_max;         // edge slots per thread a sparse phase may use (SP_EPT; smaller values force its truncation path in tests)
};

__device__ __forceinline__ int32_t *cnt_ptr(const Chunk &c, int buf3, int p) {
    return c.counts + ((size_t)buf3 * c.n_pairs + p) * 2;
}

// Largest p with base[p] <= g (base is an exclusive prefix, base[n] = total).
__device__ __forceinline__ int find_pair(const int32_t *__restrict__ base, int n, int g) {
    int lo = 0, hi = n;
    while (hi - lo > 1) {
        int mid = (lo + hi) >> 1;
        if (__ldcg(base + mid) <= g) lo = mid; else hi = mid;
    }
    return lo;
}

// A barrier over a warp-aligned group of threads of the CTA (PTX named barrier).
// id 0 with the whole block is __syncthreads().  Lets one 512-thread CTA of the
// persistent tail kernel run four independent 128-thread "virtual CTAs".
struct GroupBar {
    int id, nthreads;
    __device__ __forceinline__ void sync() const {
        asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
    }
};

// ---------------------------------------------------------------------------
// planner: one CTA (any multiple of 32 threads).  Classifies every pair from
// counts[r % 3], picks the tile shape so the round kernel gets enough work
// items to cover the machine, and writes the per-pair exclusive prefixes the
// round/accept kernels search.
// ---------------------------------------------------------------------------
__device__ __forceinline__ int tiles_of(int nlr, int nlc, int tile_rows, int cpt) {
    return ((nlr + tile_rows - 1) / tile_rows) * ((nlc + cpt - 1) / cpt);
}
__device__ __forceinline__ int ablocks_of(int nlr, int nlc) {
    return (nlr + ACCEPT_THREADS - 1) / ACCEPT_THREADS + (nlc + ACCEPT_THREADS - 1) / ACCEPT_THREADS;
}

// z with P(N(0,1) < -z) = p (Abramowitz-Stegun 26.2.23, |error| < 4.5e-4; any value is CORRECT, it only sizes lists)
__device__ __forceinline__ float inv_norm_tail(float p) {
    p = fminf(fmaxf(p, 1e-12f), 0.5f);
    const float t = sqrtf(-2.0f * __logf(p));
    return t - (2.515517f + t * (0.802853f + t * 0.010328f)) / (1.0f + t * (1.432788f + t * (0.189269f + t * 0.001308f)));
}

// Per pair and pass: the candidate-edge bound T such that the pass emits about CAND_TARGET x max(nlr, nlc)
// edges (distances taken as N(mu, sd) from the init kernel's sample).  Also resets the pair's edge counters and
// reacts to an overflow of the previous pass.  Called by the planner thread that owns pair p.
__device__ __forceinline__ void plan_pair_emit(const Chunk &c, int p, uint8_t st, int nlr, int nlc, int rq) {   // (nlr, nlc by value)
    // a tile stages at most SCAND records between two flushes (one stage of columns): keep the expected number per stage
    // below half of that, whatever the list budget would allow
    const float p_max = 0.4f * (float)SCAND / (float)(ROUND_THREADS * rq * (rq == RQ_LARGE ? STAGE_LARGE : STAGE_SMALL));
    uint32_t thr = 0u;
    const PairDesc &pd = c.pairs[p];
    if (!(pd.flags & PAIR_FLAG_SHARD) && __ldcg(c.cand_cnt + p) > pd.cand_cap) c.pstat[p].cscale *= 0.25f;   // the last pass overflowed
    if (pd.flags & PAIR_FLAG_SHARD) {
        // one rank of a train-sharded pair: every rank must arrive at the SAME bound, so it is computed from quantities
        // all ranks share -- the live rows, the live columns of the whole pair (columns = total - matched rows) and a
        // distance sample that does not involve the rank's train slice (init: queries against queries); no feedback
        nlc = c.shard_n2_total - (pd.n1 - nlr);
        if (nlr > 0 && nlc > 0 && pd.cand_cap > 0) {
            const PairStat ps = c.pstat[p];
            const float target = c.cand_target * (float)max(pd.n1, c.shard_n2_total) / (float)max(nlr, nlc);
            const float z = inv_norm_tail(fminf(target / (float)min(nlr, nlc), p_max));
            const float T = floorf(ps.mu - z * ps.sd - 0.5f);
            if (T >= 0.0f) thr = ((uint32_t)fminf(T, 1022.0f) + 1u) << KEY_IDX_BITS;
        }
    } else if (st == PAIR_BIG && pd.cand_cap > 0) {
        const PairStat ps = c.pstat[p];
        // about cand_target x max(n1, n2) raw edges in EVERY pass: later passes have fewer live rows, so each row may
        // list more candidates for the same list size (8192 x 8192: 6 per row in pass 0, ~36 per row of the 1236 left
        // in pass 1, after which ~30 rows remain -- tools/sim_threshold_rounds.py)
        const float target = fminf(c.cand_target * ps.cscale * (float)max(pd.n1, pd.n2) / (float)max(nlr, nlc), c.cand_row_max);
        if (target >= 0.09f) {
            const float z = inv_norm_tail(fminf(target / (float)min(nlr, nlc), p_max));
            const float T = floorf(ps.mu - z * ps.sd - 0.5f);                  // P(d <= T) ~ Phi((T + 0.5 - mu) / sd)
            if (T >= 0.0f) thr = ((uint32_t)fminf(T, 1022.0f) + 1u) << KEY_IDX_BITS;
        }
    }
    c.thr[p] = thr;
    c.cand_cnt[p] = 0;
    c.ledge_cnt[p] = 0;
}

// Mean and standard deviation of 1024 sampled distances of pair p, by one CTA of ACCEPT_THREADS threads (four samples
// per thread, all their descriptor loads in flight together: after an L2 flush each is an HBM round trip, and a serial
// loop of them was 30 us on the critical path of the call).  Only the SIZE of the candidate lists depends on the
// result, never a match.
__device__ __forceinline__ void sample_pair_stats(const Chunk &c, int p, const PairDesc &pd) {
    __shared__ unsigned s_sum, s_sum2;
    const int tid = threadIdx.x;
    if (tid == 0) { s_sum = 0u; s_sum2 = 0u; }
    __syncthreads();
    unsigned sum = 0, sum2 = 0;
    if (pd.n1 > 0 && pd.n2 > 0) {
        constexpr int SPT = 1024 / ACCEPT_THREADS;
        const int v4 = c.words >> 2;
        uint4 a[SPT][4], b[SPT][4];
#pragma unroll
        for (int u = 0; u < SPT; u++) {
            const unsigned sidx = (unsigned)(tid * SPT + u);
            const int i = (int)(((unsigned long long)(sidx * 2654435761u) * (unsigned)pd.n1) >> 32);     // spread over the pair
            const int j = (int)(((unsigned long long)(sidx * 2246822519u + 374761393u) * (unsigned)pd.n2) >> 32);
            const uint4 *qa = reinterpret_cast<const uint4 *>(pd.q + (size_t)i * c.words);
            const uint4 *tb = reinterpret_cast<const uint4 *>(pd.t + (size_t)j * c.words);
#pragma unroll
            for (int v = 0; v < 4; v++) {
                a[u][v] = v < v4 ? __ldg(qa + v) : make_uint4(0u, 0u, 0u, 0u);
                b[u][v] = v < v4 ? __ldg(tb + v) : make_uint4(0u, 0u, 0u, 0u);
            }
        }
#pragma unroll
        for (int u = 0; u < SPT; u++) {
            unsigned d = 0;
#pragma unroll
            for (int v = 0; v < 4; v++)
                d += __popc(a[u][v].x ^ b[u][v].x) + __popc(a[u][v].y ^ b[u][v].y) + __popc(a[u][v].z ^ b[u][v].z) + __popc(a[u][v].w ^ b[u][v].w);
            sum += d; sum2 += d * d;
        }
    }
    sum = __reduce_add_sync(0xffffffffu, sum); sum2 = __reduce_add_sync(0xffffffffu, sum2);
    if ((tid & 31) == 0) { atomicAdd(&s_sum, sum); atomicAdd(&s_sum2, sum2); }
    __syncthreads();
    if (tid == 0) {
        float mu = 0.0f, sd = 1.0f;
        if (pd.n1 > 0 && pd.n2 > 0) {
            mu = (float)s_sum * (1.0f / 1024.0f);
            sd = sqrtf(fmaxf((float)s_sum2 * (1.0f / 1024.0f) - mu * mu, 1.0f));
        }
        c.pstat[p] = PairStat{mu, sd, 1.0f, 0};
    }
}

// The same plan for at most 32 pairs, by ONE warp with everything in registers (no shared memory, no block
// barriers): in latency mode the planner sits on the critical path of every round between two grid barriers, and
// the block-wide form costs ~5 us of dependent L2 round trips and barriers there.
__device__ __forceinline__ void plan_warp(const Chunk &c, int r) {
    const int lane = threadIdx.x & 31, buf = r % 3, p = lane;
    unsigned long long ev = 0; int nbig = 0, nsmall = 0, nlr = 0, nlc = 0;
    uint8_t st = PAIR_DONE;
    if (p < c.n_pairs) {
        st = c.status[p];
        if (st == PAIR_SMALL) { nsmall = 1; }
        else {
            const int32_t *cp = cnt_ptr(c, buf, p);
            nlr = __ldcg(cp); nlc = __ldcg(cp + 1);
            st = PAIR_DONE;
            if (nlr > 0 && nlc > 0) {
                const bool small = nlr <= FIN_MAX_DIM && nlc <= FIN_MAX_DIM && nlr * nlc <= c.fin_max_evals &&
                                   !(__ldg(&c.pairs[p].flags) & PAIR_FLAG_NO_FINISHER);
                if (small) { st = PAIR_SMALL; nsmall = 1; c.small[p] = SmallInfo{nlr, nlc, r & 1, 0}; }
                else { st = PAIR_BIG; nbig = 1; ev = (unsigned long long)nlr * (unsigned long long)nlc; }
            }
            c.status[p] = st;
        }
        int32_t *nx = cnt_ptr(c, (r + 1) % 3, p);   // accept(r) appends here
        nx[0] = 0; nx[1] = 0;
    }
    for (int o = 16; o; o >>= 1) {
        ev += __shfl_xor_sync(0xffffffffu, ev, o);
        nbig += __shfl_xor_sync(0xffffffffu, nbig, o);
        nsmall += __shfl_xor_sync(0xffffffffu, nsmall, o);
    }
    // tile shape: identical arithmetic to plan_device (every lane computes it)
    const unsigned slots = (unsigned)(c.num_sms * (r == 0 && c.ctas_per_sm0 ? c.ctas_per_sm0 : c.ctas_per_sm));
    int rq, stage;
    if (ev >= (unsigned long long)c.large_min_evals) { rq = RQ_LARGE; stage = STAGE_LARGE; }
    else { rq = RQ_SMALL; stage = STAGE_SMALL; }
    const int tile_rows = ROUND_THREADS * rq;
    if (p < c.n_pairs) plan_pair_emit(c, p, st, nlr, nlc, rq);
    float per_tile = (float)ev / (2.0f * (float)slots);
    const float min_tile = (float)(tile_rows * stage);
    if (per_tile < min_tile) per_tile = min_tile;
    unsigned cpt = (unsigned)(per_tile / (float)tile_rows);
    if (cpt < 1u) cpt = 1u;
    cpt = ((cpt + stage - 1) / stage) * stage;
    if (cpt > (unsigned)MAX_N) cpt = MAX_N;
    // wave-aware refinement: a round takes ~ceil(tiles / slots) x cpt; a slightly wider tile often saves a whole,
    // mostly empty, second wave (2301 x 2301 live: 648 tiles of 64 columns on 592 slots -> 432 tiles of 96)
    if (c.n_pairs == 1) {
        // one pair: 32 candidate tilings at once, one per lane.  Under the cost model below (waves x (width + 16)) the best
        // tiling for a given number of waves is the NARROWEST one that still fits them, so lane l tries the tiling with
        // floor((l + 1) x slots / row tiles) column tiles; a tile's column extent only has to be a multiple of 8.
        // 8192 x 8192 on 888 slots: 55 -> 54 column tiles of 152 columns = 864 tiles, one wave; 1817 x 1817 (small tiles,
        // 592 slots): 38 column tiles of 48 = 570 tiles, one wave (a search around the heuristic width found two waves of
        // 40-column tiles: 14 us instead of 9); 200 000 x 25 000: 9 column tiles -> 3519 tiles = 3.96 waves.
        const int nlr0 = __shfl_sync(0xffffffffu, nlr, 0), nlc0 = __shfl_sync(0xffffffffu, nlc, 0);
        const int big0 = __shfl_sync(0xffffffffu, (int)(st == PAIR_BIG), 0);
        const int row_tiles = max(1, (nlr0 + tile_rows - 1) / tile_rows);
        const int nct = max(1, (int)(((unsigned)(lane + 1) * slots) / (unsigned)row_tiles));
        unsigned cand = (unsigned)((nlc0 + nct - 1) / nct);
        cand = min(max((cand + 7u) & ~7u, 8u), (unsigned)MAX_N);
        const unsigned t = big0 ? (unsigned)tiles_of(nlr0, nlc0, tile_rows, (int)cand) : 0u;
        unsigned long long key = ((unsigned long long)(((t + slots - 1) / slots)) * (cand + 16u) << 8) | (unsigned)lane;
        unsigned long long best = key;
        for (int o = 16; o; o >>= 1) {
            const unsigned long long other = __shfl_xor_sync(0xffffffffu, best, o);
            best = other < best ? other : best;
        }
        cpt = __shfl_sync(0xffffffffu, cand, (int)(best & 0xFFu));
    } else {
        unsigned best_cpt = cpt, best_cost = 0xFFFFFFFFu;
        for (unsigned k = 0; k < 4; k++) {
            const unsigned cand = min(cpt + k * (unsigned)stage, (unsigned)MAX_N);
            int tsum = st == PAIR_BIG ? tiles_of(nlr, nlc, tile_rows, (int)cand) : 0;
            for (int o = 16; o; o >>= 1) tsum += __shfl_xor_sync(0xffffffffu, tsum, o);
            const unsigned cost = (((unsigned)tsum + slots - 1) / slots) * cand;
            if (cost < best_cost) { best_cost = cost; best_cpt = cand; }
        }
        cpt = best_cpt;
    }
    const int tiles = st == PAIR_BIG ? tiles_of(nlr, nlc, tile_rows, (int)cpt) : 0;
    const int ablocks = st == PAIR_BIG ? ablocks_of(nlr, nlc) : 0;
    int tinc = tiles, ainc = ablocks;                // warp inclusive scans
    for (int o = 1; o < 32; o <<= 1) {
        const int a = __shfl_up_sync(0xffffffffu, tinc, o), b = __shfl_up_sync(0xffffffffu, ainc, o);
        if (lane >= o) { tinc += a; ainc += b; }
    }
    const int ttot = __shfl_sync(0xffffffffu, tinc, 31), atot = __shfl_sync(0xffffffffu, ainc, 31);
    if (p < c.n_pairs) { c.tile_base[p] = tinc - tiles; c.ablock_base[p] = ainc - ablocks; }
    if (lane == 0) {
        PlanInfo *pl = c.plan;
        pl->cols_per_tile = (int)cpt; pl->rq = rq;
        pl->n_big = nbig; pl->n_small = nsmall; pl->round = r;
        pl->ticket = 0u;
        pl->evals += ev;
        if (nbig == 0 && pl->done_round_p1 == 0) pl->done_round_p1 = r + 1;
        pl->total_tiles = ttot; pl->total_ablocks = atot;
        c.tile_base[c.n_pairs] = ttot; c.ablock_base[c.n_pairs] = atot;
    }
}

__device__ void plan_device(const Chunk &c, int r) {
    __shared__ unsigned long long s_evals[32];
    __shared__ int s_w[4][32];
    __shared__ int s_cpt, s_tile_rows;
    const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, wid = tid >> 5;
    const int NW = nt >> 5;
    const int buf = r % 3;

    unsigned long long ev = 0; int nbig = 0, nsmall = 0;
    for (int p = tid; p < c.n_pairs; p += nt) {
        uint8_t st = c.status[p];
        int nlr = 0, nlc = 0;
        if (st == PAIR_SMALL) { nsmall++; }
        else {
            const int32_t *cp = cnt_ptr(c, buf, p);
            nlr = __ldcg(cp); nlc = __ldcg(cp + 1);
            st = PAIR_DONE;
            if (nlr > 0 && nlc > 0) {
                const bool small = nlr <= FIN_MAX_DIM && nlc <= FIN_MAX_DIM && nlr * nlc <= c.fin_max_evals &&
                                   !(__ldg(&c.pairs[p].flags) & PAIR_FLAG_NO_FINISHER);
                if (small) {
                    st = PAIR_SMALL; nsmall++;
                    c.small[p] = SmallInfo{nlr, nlc, r & 1, 0};
                } else {
                    st = PAIR_BIG; nbig++;
                    ev += (unsigned long long)nlr * (unsigned long long)nlc;
                }
            }
            c.status[p] = st;
        }
        int32_t *nx = cnt_ptr(c, (r + 1) % 3, p);   // accept(r) appends here
        nx[0] = 0; nx[1] = 0;
    }
    for (int o = 16; o; o >>= 1) {
        ev += __shfl_xor_sync(0xffffffffu, ev, o);
        nbig += __shfl_xor_sync(0xffffffffu, nbig, o);
        nsmall += __shfl_xor_sync(0xffffffffu, nsmall, o);
    }
    if (lane == 0) { s_evals[wid] = ev; s_w[0][wid] = nbig; s_w[1][wid] = nsmall; }
    __syncthreads();
    if (tid == 0) {
        unsigned long long e = 0; int b = 0, s = 0;
        for (int w = 0; w < NW; w++) { e += s_evals[w]; b += s_w[0][w]; s += s_w[1][w]; }
        // tile shape: large tiles while they still cover the machine ~2x over, else small ones
        const unsigned slots = (unsigned)(c.num_sms * c.ctas_per_sm);
        int rq, stage;
        if (e >= (unsigned long long)c.large_min_evals) { rq = RQ_LARGE; stage = STAGE_LARGE; }
        else { rq = RQ_SMALL; stage = STAGE_SMALL; }
        const int tile_rows = ROUND_THREADS * rq;
        // heuristic sizing in fp32 (64-bit integer division is ~100 instructions on the GPU)
        float per_tile = (float)e / (2.0f * (float)slots);
        const float min_tile = (float)(tile_rows * stage);
        if (per_tile < min_tile) per_tile = min_tile;
        unsigned cpt = (unsigned)(per_tile / (float)tile_rows);
        if (cpt < 1u) cpt = 1u;
        cpt = ((cpt + stage - 1) / stage) * stage;
        if (cpt > (unsigned)MAX_N) cpt = MAX_N;
        s_cpt = (int)cpt; s_tile_rows = tile_rows;
        PlanInfo *pl = c.plan;
        pl->cols_per_tile = (int)cpt; pl->rq = rq;
        pl->n_big = b; pl->n_small = s; pl->round = r;
        pl->ticket = 0u;
        pl->evals += e;
        if (b == 0 && pl->done_round_p1 == 0) pl->done_round_p1 = r + 1;
    }
    __syncthreads();
    const int cpt = s_cpt, tile_rows = s_tile_rows;
    for (int p = tid; p < c.n_pairs; p += nt) {           // the pass's candidate bound of every pair (needs the tile shape)
        const uint8_t st = c.status[p];
        const int32_t *cp = cnt_ptr(c, buf, p);
        plan_pair_emit(c, p, st, st == PAIR_BIG ? __ldcg(cp) : 0, st == PAIR_BIG ? __ldcg(cp + 1) : 0, tile_rows / ROUND_THREADS);
    }
    // exclusive scan over pairs: each thread owns a contiguous slice
    const int per = (c.n_pairs + nt - 1) / nt;
    const int p0 = min(tid * per, c.n_pairs), p1 = min(p0 + per, c.n_pairs);
    int tsum = 0, asum = 0;
    for (int p = p0; p < p1; p++) {
        if (c.status[p] == PAIR_BIG) {
            const int32_t *cp = cnt_ptr(c, buf, p);
            const int nlr = __ldcg(cp), nlc = __ldcg(cp + 1);
            tsum += tiles_of(nlr, nlc, tile_rows, cpt);
            asum += ablocks_of(nlr, nlc);
        }
    }
    int tinc = tsum, ainc = asum;                    // warp inclusive scans
    for (int o = 1; o < 32; o <<= 1) {
        const int a = __shfl_up_sync(0xffffffffu, tinc, o), b = __shfl_up_sync(0xffffffffu, ainc, o);
        if (lane >= o) { tinc += a; ainc += b; }
    }
    if (lane == 31) { s_w[2][wid] = tinc; s_w[3][wid] = ainc; }
    __syncthreads();
    int toff = 0, aoff = 0, ttot = 0, atot = 0;
    for (int w = 0; w < NW; w++) {
        if (w < wid) { toff += s_w[2][w]; aoff += s_w[3][w]; }
        ttot += s_w[2][w]; atot += s_w[3][w];
    }
    int tb = toff + tinc - tsum, ab = aoff + ainc - asum;
    for (int p = p0; p < p1; p++) {
        c.tile_base[p] = tb; c.ablock_base[p] = ab;
        if (c.status[p] == PAIR_BIG) {
            const int32_t *cp = cnt_ptr(c, buf, p);
            const int nlr = __ldcg(cp), nlc = __ldcg(cp + 1);
            tb += tiles_of(nlr, nlc, tile_rows, cpt);
            ab += ablocks_of(nlr, nlc);
        }
    }
    if (tid == 0) {
        c.plan->total_tiles = ttot; c.plan->total_ablocks = atot;
        c.tile_base[c.n_pairs] = ttot; c.ablock_base[c.n_pairs] = atot;
    }
}

// Runs `plan_device(c, r)` in the last block of the calling grid to finish.
__device__ __forceinline__ void plan_in_last_block(const Chunk &c, int r, unsigned total_blocks) {
    __shared__ bool s_last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = (atomicAdd(&c.plan->ticket, 1u) == total_blocks - 1);
    __syncthreads();
    if (s_last) {
        __threadfence();
        if (c.n_pairs <= 32) { if (threadIdx.x < 32) plan_warp(c, r); }
        else plan_device(c, r);
    }
}

// ---------------------------------------------------------------------------
// init: live lists = identity, keys = none, counts[0] = (n1, n2); the last
// block plans round 0.  The host zeroes PlanInfo (memset) before the launch.
// In latency mode the few pair descriptors travel as a kernel argument (no
// pinned staging buffer to race on between back-to-back asynchronous calls).
// ---------------------------------------------------------------------------
constexpr int PACK_PAIRS = 16;
struct PairPack { PairDesc p[PACK_PAIRS]; };

template <bool PACKED>
__global__ void __launch_bounds__(ACCEPT_THREADS) init_kernel(Chunk c, PairPack pack) {
    const int p = blockIdx.y;
    const PairDesc pd = PACKED ? pack.p[p] : c.pairs[p];
    if (PACKED && blockIdx.x == 0 && threadIdx.x == 0) c.pairs[p] = pd;
    const int n = max(pd.n1, pd.n2);
    for (int x = blockIdx.x * blockDim.x + threadIdx.x; x < n; x += gridDim.x * blockDim.x) {
        if (x < pd.n1) {
            c.live_rows[0][pd.row_base + x] = x;
            c.rowbest[0][pd.row_base + x] = KEY_NONE;
            c.rowbest[1][pd.row_base + x] = KEY_NONE;
            c.match_key[pd.row_base + x] = KEY_NONE;
        }
        if (x < pd.n2) {
            c.live_cols[0][pd.col_base + x] = x;
            c.colbest[0][pd.col_base + x] = KEY_NONE;
            c.colbest[1][pd.col_base + x] = KEY_NONE;
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        int32_t *c0 = cnt_ptr(c, 0, p);
        c0[0] = pd.n1; c0[1] = pd.n2;
        int32_t *c1 = cnt_ptr(c, 1, p), *c2 = cnt_ptr(c, 2, p);
        c1[0] = c1[1] = 0; c2[0] = c2[1] = 0;
        c.status[p] = PAIR_BIG;                      // classified by plan(0)
        c.cand_cnt[p] = 0; c.ledge_cnt[p] = 0; c.thr[p] = 0u;
    }
    if (blockIdx.x == 0) {                                 // (block-uniform)
        PairDesc sp = pd;
        if (pd.flags & PAIR_FLAG_SHARD) { sp.t = pd.q; sp.n2 = pd.n1; }      // rank-invariant sample (see plan_pair_emit)
        sample_pair_stats(c, p, sp);
    }
    plan_in_last_block(c, 0, gridDim.x * gridDim.y);
}

// ---------------------------------------------------------------------------
// distance of one query (registers) against one train descriptor (registers)
// ---------------------------------------------------------------------------
// Plain form: WORDS x (LOP3 xor + POPC).  POPC.32 issues at 16 lanes/clk/SM (a
// quarter of the LOP3/IADD3 rate), so it is the bottleneck of this form.
template <int WORDS>
__device__ __forceinline__ uint32_t hamming_words_plain(const uint32_t (&q)[WORDS], const uint32_t (&t)[WORDS]) {
    uint32_t d = 0;
#pragma unroll
    for (int w = 0; w < WORDS; w++) d += __popc(q[w] ^ t[w]);
    return d;
}

// Carry-save form: three full adders (2 LOP3 each: xor3 = 0x96, majority = 0xE8)
// compress 7 of every 8 xor words into one "ones" word and three "twos" words, so
// 8 words cost 5 POPC + 14 LOP3 instead of 8 POPC + 8 LOP3.  That moves work from
// the quarter-rate POPC pipe to the ALU pipe until the two are about balanced
// (5 x 8 = 40 vs ~19 x 2 = 38 issue cycles per warp and distance).  Same value.
// (inline PTX keeps the front end from re-associating the adders into longer LOP3 chains)
__device__ __forceinline__ uint32_t xor3(uint32_t a, uint32_t b, uint32_t c) {
    uint32_t r;
    asm("lop3.b32 %0, %1, %2, %3, 0x96;" : "=r"(r) : "r"(a), "r"(b), "r"(c));
    return r;
}
__device__ __forceinline__ uint32_t maj3(uint32_t a, uint32_t b, uint32_t c) {
    uint32_t r;
    asm("lop3.b32 %0, %1, %2, %3, 0xE8;" : "=r"(r) : "r"(a), "r"(b), "r"(c));
    return r;
}

template <int WORDS>
__device__ __forceinline__ uint32_t hamming_words(const uint32_t (&q)[WORDS], const uint32_t (&t)[WORDS]) {
    uint32_t x[WORDS];
#pragma unroll
    for (int w = 0; w < WORDS; w++) x[w] = q[w] ^ t[w];
    uint32_t ones = 0, twos = 0;
#pragma unroll
    for (int g = 0; g + 8 <= WORDS; g += 8) {
        const uint32_t s1 = xor3(x[g], x[g + 1], x[g + 2]), c1 = maj3(x[g], x[g + 1], x[g + 2]);
        const uint32_t s2 = xor3(x[g + 3], x[g + 4], x[g + 5]), c2 = maj3(x[g + 3], x[g + 4], x[g + 5]);
        const uint32_t s3 = xor3(s1, s2, x[g + 6]), c3 = maj3(s1, s2, x[g + 6]);
        ones += __popc(s3) + __popc(x[g + 7]);
        twos += __popc(c1) + __popc(c2) + __popc(c3);
    }
    if (WORDS % 8 == 4) {
        constexpr int g = WORDS - 4;
        const uint32_t s1 = xor3(x[g], x[g + 1], x[g + 2]), c1 = maj3(x[g], x[g + 1], x[g + 2]);
        ones += __popc(s1) + __popc(x[g + 3]);
        twos += __popc(c1);
    }
    return ones + 2u * twos;
}

// One compression level more: the three "twos" words go through a fourth full adder, leaving 4 POPC + 16 LOP3 per 8
// words (popc(s3) + popc(x7) + 2 popc(t) + 4 popc(f)).  Alone it would make the ALU pipe the bottleneck (ptxas already
// puts the additions on the FMA pipe as IMAD); alternated with the 5-POPC form over a thread's rows the two pipes come
// out even: per distance 4.5 POPC x 8 = 36 cycles on the XU pipe vs ~17.7 ALU instructions x 2 = 35 cycles.
template <int WORDS>
__device__ __forceinline__ uint32_t hamming_words_deep(const uint32_t (&q)[WORDS], const uint32_t (&t)[WORDS]) {
    if constexpr (WORDS % 8 != 0) {
        return hamming_words<WORDS>(q, t);
    } else {
        uint32_t x[WORDS];
#pragma unroll
        for (int w = 0; w < WORDS; w++) x[w] = q[w] ^ t[w];
        uint32_t ones = 0, twos = 0, fours = 0;
#pragma unroll
        for (int g = 0; g + 8 <= WORDS; g += 8) {
            const uint32_t s1 = xor3(x[g], x[g + 1], x[g + 2]), c1 = maj3(x[g], x[g + 1], x[g + 2]);
            const uint32_t s2 = xor3(x[g + 3], x[g + 4], x[g + 5]), c2 = maj3(x[g + 3], x[g + 4], x[g + 5]);
            const uint32_t s3 = xor3(s1, s2, x[g + 6]), c3 = maj3(s1, s2, x[g + 6]);
            const uint32_t tw = xor3(c1, c2, c3), fo = maj3(c1, c2, c3);
            ones += __popc(s3) + __popc(x[g + 7]);
            twos += __popc(tw);
            fours += __popc(fo);
        }
        return ones + 2u * twos + 4u * fours;
    }
}

// ---------------------------------------------------------------------------
// round kernel: live rows x live columns of every PAIR_BIG pair.
// One thread owns RQ query descriptors in registers; the CTA streams train
// descriptors through shared memory in stages of STAGE (128-bit loads,
// 128-bit broadcast LDS).  Row argmin stays in registers for the whole tile;
// the column argmin is a warp REDUX.MIN of the packed keys followed by one
// shared-memory atomicMin per (warp, column).
// ---------------------------------------------------------------------------
__device__ __forceinline__ void tstamp(const Chunk &c, int vb, int tid, int code) {
    if (c.timeline && vb == 0 && tid == 0) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        const unsigned k = atomicAdd(reinterpret_cast<unsigned *>(c.timeline + 999), 1u);
        if (k < 480) { c.timeline[500 + k] = (t << 8) | (unsigned)code; }
    }
}

// Slow path of the distance loop (~0.1 % of the cells): a column minimum of this thread's RQ rows lies below the
// candidate bound.  cm = (distance << 20 | row id) of the best of the thread's rows IS a candidate edge; the
// thread's other rows in that column might be candidates too (rarely), which the edge filter verifies later from
// `aux` = (RQ << 20 | live-list slot of the thread's first row) -- so the hot loop recomputes nothing.
__device__ __forceinline__ void emit_record(uint32_t cm, uint32_t jk, uint32_t aux, uint32_t &thr,
                                            unsigned long long *s_cand, int *s_cctl) {
    if (cm >= thr || jk == KEY_INVALID) return;
    const int slot = atomicAdd(&s_cctl[0], 1);
    if (slot < SCAND) {
        s_cand[2 * slot] = ((unsigned long long)(cm >> KEY_IDX_BITS) << 40) | ((unsigned long long)(cm & KEY_IDX_MASK) << 20) | jk;
        s_cand[2 * slot + 1] = aux;
    } else {
        thr = 0u;                            // staging full: the flush marks the list unusable; stop trying
    }
}

template <int WORDS, int RQ, int STAGE>
__device__ __forceinline__ void round_tiles(const Chunk &c, int r, int total, int cpt,
                                            int vb, int vgrid, int tid, GroupBar bar,
                                            uint4 *s_t, uint32_t *s_jkey, uint32_t *s_col,
                                            unsigned long long *s_cand, int *s_cctl) {
    constexpr int V4 = WORDS / 4;
    constexpr int tile_rows = ROUND_THREADS * RQ;
    const int cur = r & 1, buf = r % 3, lane = tid & 31;

    tstamp(c, vb, tid, 1);
    for (int g = vb; g < total; g += vgrid) {
        const int p = find_pair(c.tile_base, c.n_pairs, g);
        const PairDesc pd = c.pairs[p];
        const int32_t *cp = cnt_ptr(c, buf, p);
        const int nlr = __ldcg(cp), nlc = __ldcg(cp + 1);
        const int nct = (nlc + cpt - 1) / cpt;
        const int local = g - __ldcg(c.tile_base + p);
        const int rt = local / nct, ct = local - rt * nct;
        const int32_t *live_rows = c.live_rows[cur] + pd.row_base;
        const int32_t *live_cols = c.live_cols[cur] + pd.col_base;
        // candidate edges: every (i, j) of this tile with distance <= T goes to the pair's list (staged in shared
        // memory, one global append per tile).  thr = (T + 1) << 20 as a key bound; 0 = this pass emits nothing.
        uint32_t thr = __ldcg(c.thr + p);
        if (thr && __ldcg(c.cand_cnt + p) > pd.cand_cap) thr = 0u;     // the list already overflowed: stop feeding it
        if (tid == 0) s_cctl[0] = 0;                                   // (ordered by the stage loop's first barrier)
        const uint32_t aux = ((uint32_t)RQ << KEY_IDX_BITS) | (uint32_t)(rt * tile_rows + tid);
        // Append the staged records to the pair's list once at least `at_least` (+1) are waiting.  Called by every thread
        // of the group right after a group barrier (the count is uniform); leaves the staging buffer empty.
        auto flush_cands = [&](int at_least) {
            const int n = s_cctl[0];
            if (n <= at_least) return;
            if (n > SCAND) {                 // the staging buffer overflowed: the pair's list is incomplete, mark it unusable
                if (tid == 0) atomicMax(c.cand_cnt + p, 0x40000000);
            } else {
                if (tid == 0) s_cctl[1] = atomicAdd(c.cand_cnt + p, n);
                bar.sync();
                const int base = s_cctl[1];
                for (int k = tid; k < 2 * n; k += ROUND_THREADS)
                    if (base + (k >> 1) < pd.cand_cap) c.cand[2 * (pd.cand_off + base) + k] = s_cand[k];
            }
            bar.sync();                      // every record is out before the counter restarts
            if (tid == 0) s_cctl[0] = 0;     // (ordered before the next records by the next stage's / tile's barriers)
        };

        uint32_t q[RQ][WORDS], ikey[RQ], rowkey[RQ];
#pragma unroll
        for (int k = 0; k < RQ; k++) {
            const int slot = rt * tile_rows + k * ROUND_THREADS + tid;
            rowkey[k] = KEY_NONE;
            if (slot < nlr) {
                const int i = __ldcg(live_rows + slot);
                PGM_ASSERT(i >= 0 && i < pd.n1);
                ikey[k] = (uint32_t)i;
                const uint4 *src = reinterpret_cast<const uint4 *>(pd.q + (size_t)i * WORDS);
#pragma unroll
                for (int v = 0; v < V4; v++) {
                    const uint4 x = __ldg(src + v);
                    q[k][4 * v + 0] = x.x; q[k][4 * v + 1] = x.y; q[k][4 * v + 2] = x.z; q[k][4 * v + 3] = x.w;
                }
            } else {
                ikey[k] = KEY_INVALID;
#pragma unroll
                for (int w = 0; w < WORDS; w++) q[k][w] = 0u;
            }
        }

        tstamp(c, vb, tid, 2);
        const int c0 = ct * cpt, c1 = min(nlc, c0 + cpt);
        for (int s0 = c0; s0 < c1; s0 += STAGE) {
            bar.sync();                       // previous stage fully consumed
            for (int k = tid; k < STAGE * V4; k += ROUND_THREADS) {
                const int col = k / V4, part = k - col * V4, y = s0 + col;
                uint4 x = make_uint4(0u, 0u, 0u, 0u);
                uint32_t jk = KEY_INVALID;
                if (y < c1) {
                    const int j = __ldcg(live_cols + y);
                    PGM_ASSERT(j >= 0 && j < pd.n2);
                    x = __ldg(reinterpret_cast<const uint4 *>(pd.t + (size_t)j * WORDS) + part);
                    jk = (uint32_t)(j + pd.col_id_offset);
                }
                s_t[k] = x;
                if (part == 0) s_jkey[col] = jk;
            }
            if (tid < STAGE) s_col[tid] = KEY_NONE;
            bar.sync();
            tstamp(c, vb, tid, 3);

            const int ncs = min(STAGE, (c1 - s0 + 7) & ~7);
            // No store, atomic or branch sits between the columns of a block, so their shared-memory loads and
            // popcount chains overlap (with the column atomics inline, ptxas serialised column after column behind
            // each ATOMS).  Candidate edges are rare (~0.1 % of the cells): a block that saw one recomputes it.
            if (RQ >= 4) {
                // large tiles: one warp-aggregated shared atomicMin per (warp, column); ptxas turns the
                // 32 same-address lanes into CREDUX.MIN + one elected ATOMS.MIN
                for (int jj0 = 0; jj0 < ncs; jj0 += 4) {
                    uint32_t cm[4];
#pragma unroll
                    for (int u = 0; u < 4; u++) {
                        const int jj = jj0 + u;
                        uint32_t t[WORDS];
#pragma unroll
                        for (int v = 0; v < V4; v++) {
                            const uint4 x = s_t[jj * V4 + v];
                            t[4 * v + 0] = x.x; t[4 * v + 1] = x.y; t[4 * v + 2] = x.z; t[4 * v + 3] = x.w;
                        }
                        const uint32_t jk = s_jkey[jj];
                        uint32_t cmin = KEY_NONE;
#pragma unroll
                        for (int k = 0; k < RQ; k++) {
                            // (rows alternate between the 5-POPC and the 4-POPC popcount so that the XU and ALU pipes balance)
                            const uint32_t d = ((k & 1) ? hamming_words_deep<WORDS>(q[k], t) : hamming_words<WORDS>(q[k], t)) << KEY_IDX_BITS;
                            rowkey[k] = min(rowkey[k], d + jk);
                            cmin = min(cmin, d + ikey[k]);
                        }
                        cm[u] = cmin;
                    }
#pragma unroll
                    for (int u = 0; u < 4; u++) atomicMin(&s_col[jj0 + u], cm[u]);
                    if (__builtin_expect(min(min(cm[0], cm[1]), min(cm[2], cm[3])) < thr, 0)) {
#pragma unroll
                        for (int u = 0; u < 4; u++) emit_record(cm[u], s_jkey[jj0 + u], aux, thr, s_cand, s_cctl);
                    }
                }
            } else {
                // small tiles (latency-bound late rounds): 32 columns at a time, the column minimum of
                // each (warp, column) is one CREDUX.MIN whose result lane (jj & 31) keeps; a single
                // conflict-free ATOMS.MIN per warp then publishes 32 columns.
                for (int jb = 0; jb < ncs; jb += 32) {
                    uint32_t mycol = KEY_NONE;
                    const int jend = min(ncs, jb + 32);
                    for (int jj0 = jb; jj0 < jend; jj0 += 8) {
                        uint32_t bmin = KEY_NONE, cm[8];
#pragma unroll
                        for (int u = 0; u < 8; u++) {
                            const int jj = jj0 + u;
                            uint32_t t[WORDS];
#pragma unroll
                            for (int v = 0; v < V4; v++) {
                                const uint4 x = s_t[jj * V4 + v];
                                t[4 * v + 0] = x.x; t[4 * v + 1] = x.y; t[4 * v + 2] = x.z; t[4 * v + 3] = x.w;
                            }
                            const uint32_t jk = s_jkey[jj];
                            uint32_t cmin = KEY_NONE;
#pragma unroll
                            for (int k = 0; k < RQ; k++) {
                                const uint32_t d = hamming_words<WORDS>(q[k], t) << KEY_IDX_BITS;
                                rowkey[k] = min(rowkey[k], d + jk);
                                cmin = min(cmin, d + ikey[k]);
                            }
                            const uint32_t wmin = __reduce_min_sync(0xffffffffu, cmin);
                            if (lane == (jj & 31)) mycol = wmin;
                            bmin = min(bmin, cmin);
                            cm[u] = cmin;
                        }
                        if (__builtin_expect(bmin < thr, 0)) {
#pragma unroll
                            for (int u = 0; u < 8; u++) emit_record(cm[u], s_jkey[jj0 + u], aux, thr, s_cand, s_cctl);
                        }
                    }
                    atomicMin(&s_col[jb + lane], mycol);
                }
            }
            bar.sync();
            tstamp(c, vb, tid, 4);
            if (tid < STAGE) {
                const uint32_t jk = s_jkey[tid], v = s_col[tid];
                if (jk != KEY_INVALID && v < KEY_INVALID)      // jk carries the global id; the state arrays are local
                    atomicMin(c.colbest[cur] + pd.col_base + (jk - (uint32_t)pd.col_id_offset), v);
            }
            flush_cands(SCAND / 2);                          // wide tiles (batches of pairs) see more records than one staging buffer holds
        }
#pragma unroll
        for (int k = 0; k < RQ; k++)
            if (ikey[k] != KEY_INVALID && rowkey[k] < KEY_INVALID)
                atomicMin(c.rowbest[cur] + pd.row_base + ikey[k], rowkey[k]);
        bar.sync(); flush_cands(0);                     // the tile's remaining staged candidate records
        tstamp(c, vb, tid, 5);
    }
}

template <int WORDS>
__global__ void __launch_bounds__(ROUND_THREADS, WORDS <= 8 ? 6 : (WORDS == 12 ? 5 : 4)) hamming_round_kernel(Chunk c, int r) {
    __shared__ uint4 s_t[STAGE_LARGE * (WORDS / 4)];
    __shared__ uint32_t s_jkey[STAGE_LARGE];
    __shared__ uint32_t s_col[STAGE_LARGE];
    __shared__ unsigned long long s_cand[2 * SCAND];
    __shared__ int s_cctl[2];
    const int total = __ldcg(&c.plan->total_tiles);
    if ((int)blockIdx.x >= total) return;
    const int cpt = __ldcg(&c.plan->cols_per_tile);
    const int rq = __ldcg(&c.plan->rq);
    const GroupBar bar{0, ROUND_THREADS};
    if (rq == RQ_LARGE)
        round_tiles<WORDS, RQ_LARGE, STAGE_LARGE>(c, r, total, cpt, blockIdx.x, gridDim.x, threadIdx.x, bar, s_t, s_jkey, s_col, s_cand, s_cctl);
    else
        round_tiles<WORDS, RQ_SMALL, STAGE_SMALL>(c, r, total, cpt, blockIdx.x, gridDim.x, threadIdx.x, bar, s_t, s_jkey, s_col, s_cand, s_cctl);
}

// ---------------------------------------------------------------------------
// accept kernel: a row and a column that chose each other are the minimum of
// every edge touching either of them, i.e. the pair the reference's next
// applicable argmin scan would emit (KeypointMatching.cs:44-65).  Survivors
// are appended to the next live lists; their key slots in the other buffer
// are reset.  The last block to finish plans round r+1.
// ---------------------------------------------------------------------------
__device__ __forceinline__ void accept_blocks(const Chunk &c, int r, int vb, int vgrid, int tid) {
    const int lane = tid & 31;
    const int cur = r & 1, nxt = cur ^ 1, buf = r % 3, nbuf = (r + 1) % 3;
    const int total = __ldcg(&c.plan->total_ablocks);

    for (int b = vb; b < total; b += vgrid) {
        const int p = find_pair(c.ablock_base, c.n_pairs, b);
        const PairDesc pd = c.pairs[p];
        const int32_t *cp = cnt_ptr(c, buf, p);
        const int nlr = __ldcg(cp), nlc = __ldcg(cp + 1);
        const int nrb = (nlr + ACCEPT_THREADS - 1) / ACCEPT_THREADS;
        const int local = b - __ldcg(c.ablock_base + p);
        const uint32_t *rowbest = c.rowbest[cur] + pd.row_base;
        const uint32_t *colbest = c.colbest[cur] + pd.col_base;
        const bool is_row = local < nrb;
        const int x = (is_row ? local : local - nrb) * ACCEPT_THREADS + tid;
        bool survive = false;
        int id = 0;
        if (is_row) {
            if (x < nlr) {
                id = __ldcg(c.live_rows[cur] + pd.row_base + x);
                PGM_ASSERT(id >= 0 && id < pd.n1);
                const uint32_t rk = __ldcg(rowbest + id);
                PGM_ASSERT(rk != KEY_NONE && (int)(rk & KEY_IDX_MASK) - pd.col_id_offset >= 0 && (int)(rk & KEY_IDX_MASK) - pd.col_id_offset < pd.n2);
                const uint32_t ck = __ldcg(colbest + (rk & KEY_IDX_MASK));
                if ((ck & KEY_IDX_MASK) == (uint32_t)id) c.match_key[pd.row_base + id] = rk;
                else { survive = true; c.rowbest[nxt][pd.row_base + id] = KEY_NONE; }
            }
        } else {
            if (x < nlc) {
                id = __ldcg(c.live_cols[cur] + pd.col_base + x);
                PGM_ASSERT(id >= 0 && id < pd.n2);
                const uint32_t ck = __ldcg(colbest + id);
                PGM_ASSERT(ck != KEY_NONE && (int)(ck & KEY_IDX_MASK) < pd.n1);
                const uint32_t rk = __ldcg(rowbest + (ck & KEY_IDX_MASK));
                if ((rk & KEY_IDX_MASK) != (uint32_t)id) { survive = true; c.colbest[nxt][pd.col_base + id] = KEY_NONE; }
            }
        }
        const unsigned m = __ballot_sync(0xffffffffu, survive);
        if (m) {
            int base = 0;
            if (lane == (__ffs(m) - 1)) base = atomicAdd(cnt_ptr(c, nbuf, p) + (is_row ? 0 : 1), __popc(m));
            base = __shfl_sync(0xffffffffu, base, __ffs(m) - 1);
            if (survive) {
                const int pos = base + __popc(m & ((1u << lane) - 1u));
                PGM_ASSERT(pos >= 0 && pos < (is_row ? nlr : nlc));
                if (is_row) { c.live_rows[nxt][pd.row_base + pos] = id; c.row_pos[pd.row_base + id] = pos; }
                else { c.live_cols[nxt][pd.col_base + pos] = id; c.col_pos[pd.col_base + id] = pos; }
            }
        }
    }
}

// ---------------------------------------------------------------------------
// candidate edges, step 2 (same phase as the accept: both only READ the pass's row / column minima): keep the raw
// edges of pair p whose row and column both survive the accept of round r -- a row is matched by that accept iff
// the column it chose chose it back, which any thread can evaluate from rowbest / colbest without waiting for the
// accept to finish.  Warps walk the list from edge `start` in steps of `step` (both multiples of 32).
// ---------------------------------------------------------------------------
__device__ __forceinline__ void filter_edges(const Chunk &c, int r, int p, int start, int step) {
    const int n = __ldcg(c.cand_cnt + p);
    if (n <= 0) return;
    const PairDesc &pd = c.pairs[p];
    const int cap = __ldg(&pd.cand_cap), lcap = __ldg(&pd.ledge_cap);
    if (n > cap) return;                                   // overflowed: no sparse phase for this pair this pass
    const int lane = threadIdx.x & 31, cur = r & 1, words = c.words;
    const int64_t row_base = __ldg(&pd.row_base), col_base = __ldg(&pd.col_base);
    const uint32_t *rowbest = c.rowbest[cur] + row_base, *colbest = c.colbest[cur] + col_base;
    const int32_t *live_rows = c.live_rows[cur] + row_base;
    const int nlr = __ldcg(cnt_ptr(c, r % 3, p));
    const uint32_t thr = __ldcg(c.thr + p);
    const uint32_t *qd = pd.q, *td = pd.t;
    const unsigned long long *raw = c.cand + 2 * __ldg(&pd.cand_off);
    unsigned long long *out = c.ledge + __ldg(&pd.ledge_off);
    for (int e0 = start; e0 < n; e0 += step) {
        const int e = e0 + lane;
        unsigned long long ed[RQ_LARGE];                   // the record's edge and its verified siblings (~0: none)
#pragma unroll
        for (int k = 0; k < RQ_LARGE; k++) ed[k] = ~0ull;
        if (e < n) {
            const unsigned long long key = __ldcg(raw + 2 * e);
            const uint32_t aux = (uint32_t)__ldcg(raw + 2 * e + 1);
            PGM_ASSERT((int)((key >> KEY_IDX_BITS) & KEY_IDX_MASK) < pd.n1 && (int)(key & KEY_IDX_MASK) < pd.n2 && (key >> 40) <= 512);
            PGM_ASSERT((aux >> KEY_IDX_BITS) == 1 || (aux >> KEY_IDX_BITS) == RQ_LARGE);
            const uint32_t i0 = (uint32_t)(key >> KEY_IDX_BITS) & KEY_IDX_MASK, j = (uint32_t)key & KEY_IDX_MASK;
            // the column first: it is shared by the record's edge and its siblings, and about half of the columns are
            // matched by this very accept -- those records cost two sectors instead of a dozen
            const uint32_t ck = __ldcg(colbest + j);
            PGM_ASSERT((int)(ck & KEY_IDX_MASK) < pd.n1);
            const uint32_t rk_of_ck = __ldcg(rowbest + (ck & KEY_IDX_MASK));
            const int rqn = (int)(aux >> KEY_IDX_BITS), slot0 = (int)(aux & KEY_IDX_MASK);
            if ((rk_of_ck & KEY_IDX_MASK) != j) {
              ed[0] = key;
              if (rqn > 1) {
                // the emitting thread held rqn rows (live-list slots slot0 + k * ROUND_THREADS) and reported the best
                // of them in this column: check the others against the bound
                uint32_t tw[16];
#pragma unroll
                for (int v = 0; v < 4; v++) {            // rows are 16-byte aligned: 128-bit loads
                    const uint4 x = 4 * v < words ? __ldg(reinterpret_cast<const uint4 *>(td + (size_t)j * words) + v) : make_uint4(0u, 0u, 0u, 0u);
                    tw[4 * v] = x.x; tw[4 * v + 1] = x.y; tw[4 * v + 2] = x.z; tw[4 * v + 3] = x.w;
                }
                int used = 1;
                for (int k = 0; k < rqn && k < RQ_LARGE; k++) {
                    const int slot = slot0 + k * ROUND_THREADS;
                    if (slot >= nlr) break;
                    const uint32_t i2 = r == 0 ? (uint32_t)slot : (uint32_t)__ldcg(live_rows + slot);   // (pass 0: the live list is the identity)
                    if (i2 == i0) continue;
                    uint32_t d = 0;
#pragma unroll
                    for (int v = 0; v < 4; v++) {
                        if (4 * v < words) {
                            const uint4 x = __ldg(reinterpret_cast<const uint4 *>(qd + (size_t)i2 * words) + v);
                            d += __popc(x.x ^ tw[4 * v]) + __popc(x.y ^ tw[4 * v + 1]) + __popc(x.z ^ tw[4 * v + 2]) + __popc(x.w ^ tw[4 * v + 3]);
                        }
                    }
                    if ((d << KEY_IDX_BITS) < thr) {
                        const unsigned long long k2 = ((unsigned long long)d << 40) | ((unsigned long long)i2 << 20) | j;
                        if (used == 1) ed[1] = k2; else if (used == 2) ed[2] = k2; else ed[3] = k2;
                        used++;
                    }
                }
              }
            }
        }
#pragma unroll
        for (int x = 0; x < RQ_LARGE; x++) {
            bool keep = false;
            if (ed[x] != ~0ull) {                              // (the column survives: checked above)
                const uint32_t i = (uint32_t)(ed[x] >> KEY_IDX_BITS) & KEY_IDX_MASK;
                const uint32_t rk = __ldcg(rowbest + i);
                PGM_ASSERT((int)(rk & KEY_IDX_MASK) < pd.n2);
                const uint32_t ck_of_rk = __ldcg(colbest + (rk & KEY_IDX_MASK));
                keep = (ck_of_rk & KEY_IDX_MASK) != i;
            }
            const unsigned m = __ballot_sync(0xffffffffu, keep);
            if (m) {
                int base = 0;
                if (lane == (__ffs(m) - 1)) base = atomicAdd(c.ledge_cnt + p, __popc(m));
                base = __shfl_sync(0xffffffffu, base, __ffs(m) - 1);
                const int pos = base + __popc(m & ((1u << lane) - 1u));
                if (keep && pos < lcap) out[pos] = ed[x];   // (ledge_cnt > ledge_cap: the sparse phase skips the pair)
            }
        }
    }
}

// ---------------------------------------------------------------------------
// candidate edges, step 3: the sparse sub-rounds of pair p, by ONE CTA.
// The pass computed every distance of live rows x live columns and listed every edge with distance <= T, so for a
// row (column) that still has a live listed edge, its smallest live listed edge IS its best live column (row) under
// the reference's (distance, j) / (distance, i) order; an edge that is the minimum of both its row and its column is
// locally dominant, i.e. the pair the reference's argmin scan (KeypointMatching.cs:44-65) emits before any other
// edge touching either endpoint.  Sub-round: atomicMin the live edges into per-row / per-column slots, accept the
// mutual ones, drop the edges that lost an endpoint; repeat until no edge is left.  Rows whose listed edges all died
// simply stay live for the next distance pass.  Afterwards the pair's live lists (already compacted by the accept)
// are re-compacted in place and its counts updated.
// Shared memory holds the edges and one min slot per row and column (layout: sparse_body).
// ---------------------------------------------------------------------------
template <int NT>
__device__ __forceinline__ void sparse_body(const Chunk &c, int r, int p, unsigned char *smem) {
    if (__ldcg(c.status + p) != PAIR_BIG) return;
    const int tid = threadIdx.x, lane = tid & 31;
    const PairDesc &pdr = c.pairs[p];
    const int nL = __ldcg(c.ledge_cnt + p);
    const int nxt = (r & 1) ^ 1, nbuf = (r + 1) % 3;
    int32_t *cnt = cnt_ptr(c, nbuf, p);
    const int nlr = __ldcg(cnt), nlc = __ldcg(cnt + 1);
    const int n1 = __ldg(&pdr.n1), n2 = __ldg(&pdr.n2);
    if (nL <= 0 || nL > __ldg(&pdr.ledge_cap) || nL > NT * SP_EPT || nlr <= 0 || nlc <= 0) return;
    // Edges live in SHARED memory, `slots` per thread in the thread's private column E[k * NT] (conflict-free), kept
    // compact: a thread's live edges are E[0 .. ne).  Every loop below is a real loop over the live edges -- the phase
    // runs once per pass on one SM, its code is fetched cold, and the register-resident, fully unrolled form it replaces
    // (138 KB of SASS) was bound by instruction fetch, not by the edges.
    // Min slots are addressed by the ORIGINAL row / column id when the pair is small enough (no position look-ups: they
    // are 2 random 32-byte sectors per edge, and one SM's L2 bandwidth is what bounds the loading of the edges), else by
    // the position the accept gave the survivor in the next live list (one more word per edge).
    // When the pass listed more edges than shared memory holds, the phase keeps the edges with distance <= T' for the
    // largest T' that fits: a set that is complete up to T' is as valid as one complete up to T (it is what a smaller
    // candidate bound would have produced), the rows it does not resolve wait for the next distance pass.
    static_assert(NT == 512, "the distance histogram of the truncation gives one bin to every thread");
    const int need = (nL + NT - 1) / NT;
    const int slots_id = (int)min((long long)c.sp_slots_max, max(0ll, ((long long)SP_SMEM_BYTES - 4ll * (n1 + n2)) / (8 * NT)));
    const int slots_pos = nlr <= 65535 && nlc <= 65535 ? (int)min((long long)c.sp_slots_max, max(0ll, ((long long)SP_SMEM_BYTES - 4ll * (nlr + nlc)) / (12 * NT))) : 0;
    // (positions cost two random L2 sectors per edge when the list is loaded -- ~20 us for 13 000 edges on one SM -- so
    //  ids are preferred even when they leave room for somewhat fewer edges)
    const bool by_id = slots_id >= need || 2 * slots_id >= slots_pos;
    const int slots = min(need, by_id ? slots_id : slots_pos);
    if (slots <= 0) return;
    const bool truncated = slots < need;
    const int nr = by_id ? n1 : nlr, nc = by_id ? n2 : nlc;
    const int64_t row_base = __ldg(&pdr.row_base), col_base = __ldg(&pdr.col_base);
    uint2 *E = reinterpret_cast<uint2 *>(smem);                             // .x = (d << 20 | j), .y = i; thread t owns E[t + k * NT]
    uint32_t *P = reinterpret_cast<uint32_t *>(smem + 8 * (size_t)slots * NT);   // !by_id: (row slot << 16 | column slot)
    uint32_t *rbest = reinterpret_cast<uint32_t *>(smem + (by_id ? 8 : 12) * (size_t)slots * NT);
    uint32_t *cbest = rbest + nr;
    __shared__ int s_cnt[2], s_alive[3], s_fill, s_nsel, s_wsum[NT / 32];
    const unsigned long long *edges = c.ledge + __ldg(&pdr.ledge_off);

    tstamp(c, p, tid, 20);
    uint32_t dmax = 0xFFFFFFFFu;                                            // edges with distance <= dmax take part
    int n_sel = nL;
    if (truncated) {                                                        // (block-uniform)
        int *hist = reinterpret_cast<int *>(smem);                          // (the edge arrays are written after this block)
        for (int k = tid; k < NT + 1; k += NT) hist[k] = 0;
        if (tid == 0) s_fill = 0;
        __syncthreads();
        for (int e0 = 0; e0 < nL; e0 += NT * SP_LB) {
            unsigned long long key[SP_LB];
#pragma unroll
            for (int u = 0; u < SP_LB; u++) { const int e = e0 + u * NT + tid; key[u] = e < nL ? __ldcg(edges + e) : ~0ull; }
#pragma unroll
            for (int u = 0; u < SP_LB; u++) {
                // (the list holds a handful of distinct distances: one atomic per warp and distance, not per edge)
                const uint32_t d = min((uint32_t)(key[u] >> 40), (uint32_t)NT + 1u);       // NT + 1: no edge
                const unsigned peers = __match_any_sync(0xffffffffu, d);
                if (d <= (uint32_t)NT && lane == __ffs(peers) - 1) atomicAdd(&hist[d], __popc(peers));
            }
        }
        __syncthreads();
        int cum = hist[tid];                                                // thread t: edges with distance <= t
        for (int o = 1; o < 32; o <<= 1) { const int a = __shfl_up_sync(0xffffffffu, cum, o); if (lane >= o) cum += a; }
        if (lane == 31) s_wsum[tid >> 5] = cum;
        __syncthreads();
        for (int w = 0; w < (tid >> 5); w++) cum += s_wsum[w];
        const int keep = __syncthreads_count(cum <= slots * NT);            // cum never decreases: the kept distances are a prefix
        if (keep == 0) return;
        if (tid == keep - 1) s_nsel = cum;
        __syncthreads();
        dmax = (uint32_t)(keep - 1);
        n_sel = s_nsel;
        if (n_sel <= 0) return;
    }
    for (int k = tid; k < nr + nc; k += NT) rbest[k] = KEY_NONE;        // (rbest and cbest are contiguous)
    if (tid == 0) { s_alive[0] = 0; s_alive[1] = 0; s_alive[2] = 0; }
    {
        const int32_t *row_pos = c.row_pos + row_base, *col_pos = c.col_pos + col_base;
        for (int k0 = 0; k0 < need; k0 += SP_LB) {                      // SP_LB independent L2 loads in flight per thread
            unsigned long long key[SP_LB];
#pragma unroll
            for (int u = 0; u < SP_LB; u++) {
                const int e = tid + (k0 + u) * NT;
                key[u] = e < nL ? __ldcg(edges + e) : ~0ull;
                if ((uint32_t)(key[u] >> 40) > dmax) key[u] = ~0ull;        // (~0 >> 40 exceeds every distance)
            }
            uint32_t pp[SP_LB];
#pragma unroll
            for (int u = 0; u < SP_LB; u++) {
                pp[u] = 0u;
                if (!by_id && key[u] != ~0ull) {
                    const uint32_t i = (uint32_t)(key[u] >> KEY_IDX_BITS) & KEY_IDX_MASK, j = (uint32_t)key[u] & KEY_IDX_MASK;
                    PGM_ASSERT((int)i < n1 && (int)j < n2);
                    pp[u] = ((uint32_t)__ldcg(row_pos + i) << 16) | (uint32_t)__ldcg(col_pos + j);
                }
            }
#pragma unroll
            for (int u = 0; u < SP_LB; u++) {
                const bool sel = key[u] != ~0ull;
                int pos = tid + (k0 + u) * NT;                              // nothing cut: list position = layout position
                if (truncated) {                                            // (uniform; the loop bound is uniform too)
                    const unsigned m = __ballot_sync(0xffffffffu, sel);
                    int base = 0;
                    if (m && lane == (__ffs(m) - 1)) base = atomicAdd(&s_fill, __popc(m));
                    base = __shfl_sync(0xffffffffu, base, m ? __ffs(m) - 1 : 0);
                    pos = base + __popc(m & ((1u << lane) - 1u));
                }
                if (sel) {
                    const uint32_t i = (uint32_t)(key[u] >> KEY_IDX_BITS) & KEY_IDX_MASK, j = (uint32_t)key[u] & KEY_IDX_MASK;
                    PGM_ASSERT((int)i < n1 && (int)j < n2 && pos < slots * NT && (by_id || ((int)(pp[u] >> 16) < nr && (int)(pp[u] & 0xFFFFu) < nc)));
                    E[pos] = make_uint2(((uint32_t)(key[u] >> 40) << KEY_IDX_BITS) | j, i);
                    if (!by_id) P[pos] = pp[u];
                }
            }
        }
    }
    E += tid; P += tid;                                                     // from here on: the thread's own column
    int ne = n_sel > tid ? (n_sel - tid + NT - 1) / NT : 0;                 // its live edges are E[0 .. ne) (x NT)
    __syncthreads();
    tstamp(c, p, tid, 21);
    uint32_t *match_key = c.match_key + row_base;
    // slot indices of an edge
#define PGM_SP_RS(e, q) (by_id ? (e).y : (q) >> 16)
#define PGM_SP_CS(e, q) (by_id ? ((e).x & KEY_IDX_MASK) : ((q) & 0xFFFFu))
#define PGM_SP_CKEY(e) (((e).x & ~KEY_IDX_MASK) | (e).y)
    for (int sub = 0; sub < SP_MAX_SUB; sub++) {
        // (three counters: the one reset here was last read two barriers ago -- with two, a warp late to read the
        //  previous sub-round's total could see the reset)
        if (tid == 0) s_alive[(sub + 1) % 3] = 0;
        // A. every live edge goes to the min slot of its row (key d, j) and of its column (key d, i)
        for (int k0 = 0; k0 < ne; k0 += SP_B) {
            uint2 e[SP_B]; uint32_t q[SP_B];
#pragma unroll
            for (int u = 0; u < SP_B; u++) {
                const int k = min(k0 + u, ne - 1);
                e[u] = E[k * NT]; q[u] = by_id ? 0u : P[k * NT];
            }
#pragma unroll
            for (int u = 0; u < SP_B; u++)
                if (k0 + u < ne) { atomicMin(&rbest[PGM_SP_RS(e[u], q[u])], e[u].x); atomicMin(&cbest[PGM_SP_CS(e[u], q[u])], PGM_SP_CKEY(e[u])); }
        }
        __syncthreads();
        // B. an edge that is the minimum of both its row and its column is accepted.  Loads first, stores after, in
        // batches: a shared-memory store between two loads makes ptxas order them (possible alias)
        for (int k0 = 0; k0 < ne; k0 += SP_B) {
            uint2 e[SP_B]; uint32_t q[SP_B], rv[SP_B], cv[SP_B];
#pragma unroll
            for (int u = 0; u < SP_B; u++) {
                const int k = min(k0 + u, ne - 1);
                e[u] = E[k * NT]; q[u] = by_id ? 0u : P[k * NT];
            }
#pragma unroll
            for (int u = 0; u < SP_B; u++) { rv[u] = rbest[PGM_SP_RS(e[u], q[u])]; cv[u] = cbest[PGM_SP_CS(e[u], q[u])]; }
#pragma unroll
            for (int u = 0; u < SP_B; u++) {
                // (a concurrent KEY_DEAD store by the accepting thread of another edge of this row / column can only
                //  turn a mismatch into a mismatch: keys within a row, and within a column, are distinct)
                if (k0 + u < ne && rv[u] == e[u].x && cv[u] == PGM_SP_CKEY(e[u])) {
                    PGM_ASSERT(__ldcg(match_key + e[u].y) == KEY_NONE);      // a row is matched once
                    match_key[e[u].y] = e[u].x;
                    rbest[PGM_SP_RS(e[u], q[u])] = KEY_DEAD; cbest[PGM_SP_CS(e[u], q[u])] = KEY_DEAD;
                }
            }
        }
        __syncthreads();
        // C. edges that lost an endpoint leave the thread's list (survivors move to the front: a batch is read before any
        // of it is written, and the write position never passes the read position); live slots are reset for the next
        // sub-round (never overwrites KEY_DEAD: a dead slot has no live edge)
        int w = 0;
        for (int k0 = 0; k0 < ne; k0 += SP_B) {
            uint2 e[SP_B]; uint32_t q[SP_B], rv[SP_B], cv[SP_B];
#pragma unroll
            for (int u = 0; u < SP_B; u++) {
                const int k = min(k0 + u, ne - 1);
                e[u] = E[k * NT]; q[u] = by_id ? 0u : P[k * NT];
            }
#pragma unroll
            for (int u = 0; u < SP_B; u++) { rv[u] = rbest[PGM_SP_RS(e[u], q[u])]; cv[u] = cbest[PGM_SP_CS(e[u], q[u])]; }
#pragma unroll
            for (int u = 0; u < SP_B; u++) {
                if (k0 + u < ne && rv[u] != KEY_DEAD && cv[u] != KEY_DEAD) {
                    rbest[PGM_SP_RS(e[u], q[u])] = KEY_NONE; cbest[PGM_SP_CS(e[u], q[u])] = KEY_NONE;
                    if (w != k0 + u) { E[w * NT] = e[u]; if (!by_id) P[w * NT] = q[u]; }
                    w++;
                }
            }
        }
        ne = w;
        const int alive = __reduce_add_sync(0xffffffffu, ne);
        if (lane == 0 && alive) atomicAdd(&s_alive[sub % 3], alive);
        tstamp(c, p, tid, 22);
        __syncthreads();
        if (s_alive[sub % 3] == 0) break;
    }
#undef PGM_SP_RS
#undef PGM_SP_CS
#undef PGM_SP_CKEY
    // re-compact the live lists in place, SP_IPT ids per thread and side at a time (order is arbitrary).  A chunk's ids
    // are all read before any of them is written back, and the kept ones land below the chunk's end: no unread slot is
    // hit.  Rows and columns share the loop so that their loads are in flight together.
    {
        int32_t *live_r = c.live_rows[nxt] + row_base, *live_c = c.live_cols[nxt] + col_base;
        if (tid == 0) { s_cnt[0] = 0; s_cnt[1] = 0; }
        const int nmax = nlr > nlc ? nlr : nlc;
        for (int k0 = 0; k0 < nmax; k0 += NT * SP_IPT) {
            int32_t idr[SP_IPT], idc[SP_IPT];
            bool kr[SP_IPT], kc[SP_IPT];
#pragma unroll
            for (int u = 0; u < SP_IPT; u++) {
                const int k = k0 + u * NT + tid;
                idr[u] = k < nlr ? __ldcg(live_r + k) : 0;
                idc[u] = k < nlc ? __ldcg(live_c + k) : 0;
            }
#pragma unroll
            for (int u = 0; u < SP_IPT; u++) {
                const int k = k0 + u * NT + tid;
                kr[u] = k < nlr && rbest[by_id ? idr[u] : k] != KEY_DEAD;
                kc[u] = k < nlc && cbest[by_id ? idc[u] : k] != KEY_DEAD;
            }
            __syncthreads();
            // one shared-memory atomic per warp, side and chunk (not per 32 ids: 16 warps queueing on two counters was
            // most of this step's time)
#pragma unroll
            for (int side = 0; side < 2; side++) {
                unsigned m[SP_IPT];
                int tot = 0;
#pragma unroll
                for (int u = 0; u < SP_IPT; u++) { m[u] = __ballot_sync(0xffffffffu, side ? kc[u] : kr[u]); tot += __popc(m[u]); }
                int at = 0;
                if (lane == 0 && tot) at = atomicAdd(&s_cnt[side], tot);
                at = __shfl_sync(0xffffffffu, at, 0);
#pragma unroll
                for (int u = 0; u < SP_IPT; u++) {
                    if (side ? kc[u] : kr[u]) {
                        const int o = at + __popc(m[u] & ((1u << lane) - 1u));
                        PGM_ASSERT(o < (side ? nlc : nlr));
                        (side ? live_c : live_r)[o] = side ? idc[u] : idr[u];
                    }
                    at += __popc(m[u]);
                }
            }
        }
    }
    __syncthreads();
    if (tid == 0) { cnt[0] = s_cnt[0]; cnt[1] = s_cnt[1]; }
    tstamp(c, p, tid, 23);
}

// standalone forms (throughput mode): accept + edge filter, then one sparse CTA per pair whose last block plans
// (5 CTAs per SM: the kernel is a chain of dependent L2 / HBM accesses per record, more resident warps is what it needs)
__global__ void __launch_bounds__(ACCEPT_THREADS, 5) accept_kernel(Chunk c, int r) {
    accept_blocks(c, r, blockIdx.x, gridDim.x, threadIdx.x);
    // a pair's raw list is dealt out in FILTER_SEGS interleaved segments: with one CTA per pair a grid of ~1200
    // CTAs walked 2016 lists as two unequal waves of ~100 dependent iterations each
    constexpr int FILTER_SEGS = 8;
    for (int item = blockIdx.x; item < c.n_pairs * FILTER_SEGS; item += gridDim.x) {
        const int p = item / FILTER_SEGS, seg = item - p * FILTER_SEGS;
        filter_edges(c, r, p, seg * ACCEPT_THREADS + (int)(threadIdx.x & ~31u), ACCEPT_THREADS * FILTER_SEGS);
    }
}

__global__ void __launch_bounds__(SP_THREADS) sparse_kernel(Chunk c, int r) {
    extern __shared__ __align__(16) unsigned char dyn_smem[];
    for (int p = blockIdx.x; p < c.n_pairs; p += gridDim.x) { sparse_body<SP_THREADS>(c, r, p, dyn_smem); __syncthreads(); }
    plan_in_last_block(c, r + 1, gridDim.x);
}

// ---------------------------------------------------------------------------
// finisher: one CTA per PAIR_SMALL pair runs every remaining round out of a
// u16 distance matrix in shared memory.  Live lists arrive in arbitrary order
// (atomic append), so they are rank-sorted first: local positions then order
// like the original indices and keys can carry positions.  After the first
// round a row (column) is rescanned only if the column (row) it had chosen
// was matched to someone else -- otherwise its argmin is still valid.
// ---------------------------------------------------------------------------
// live lists of pair p -> rank-sorted original ids (ids are distinct) in rowid[] / colid[]
__device__ __forceinline__ void finisher_sorted_ids(const Chunk &c, const PairDesc &pd, int nr, int nc, int cur, int32_t *rowid,
                                                    int32_t *colid, int32_t *tmp) {
    const int tid = threadIdx.x, nt = FIN_THREADS;
    for (int k = tid; k < nr + nc; k += nt)
        tmp[k < nr ? k : FIN_MAX_DIM + (k - nr)] =
            k < nr ? __ldcg(c.live_rows[cur] + pd.row_base + k) : __ldcg(c.live_cols[cur] + pd.col_base + (k - nr));
    __syncthreads();
    for (int k = tid; k < nr + nc; k += nt) {
        const bool is_row = k < nr;
        const int32_t *src = is_row ? tmp : tmp + FIN_MAX_DIM;
        const int n = is_row ? nr : nc, me = src[is_row ? k : k - nr];
        int rank = 0;
#pragma unroll 8
        for (int m = 0; m < n; m++) rank += (src[m] < me);
        if (is_row) rowid[rank] = me; else colid[rank] = me;
    }
    __syncthreads();
}

__device__ __forceinline__ int finisher_pitch(int nc) {
    int S = (nc + 1) & ~1;            // row pitch in u16; S/2 odd -> row scans hit 32 distinct banks
    if (((S >> 1) & 1) == 0) S += 2;
    return S;
}

// Latency mode, run by EVERY CTA of the tail kernel for every small pair: one warp per row (then per column) of
// the live x live matrix computes its distances straight from global memory, writes the row's cells and the
// row's (column's) first-round minimum to global memory.  A single SM would need ~8 us for a 145 x 145 matrix and
// ~6 us for the first round of scans; spread over the machine both cost one grid barrier.
// The CTAs working on pair p are numbered sub_rank = 0 .. sub_count - 1 (the tail kernel splits its grid among
// the small pairs).
template <int WORDS>
__device__ __forceinline__ void finisher_prepare(const Chunk &c, int p, unsigned char *fin_smem, int sub_rank, int sub_count) {
    const int tid = threadIdx.x, lane = tid & 31, nw = FIN_THREADS >> 5;
    const PairDesc pd = c.pairs[p];
    const int4 si_raw = __ldcg(reinterpret_cast<const int4 *>(c.small + p));
    const int nr = si_raw.x, nc = si_raw.y, cur = si_raw.z;
    const int S = finisher_pitch(nc);
    int32_t *rowid = reinterpret_cast<int32_t *>(fin_smem);
    int32_t *colid = rowid + FIN_MAX_DIM;
    int32_t *tmp = colid + FIN_MAX_DIM;                                   // 2 * FIN_MAX_DIM
    finisher_sorted_ids(c, pd, nr, nc, cur, rowid, colid, tmp);
    uint16_t *Dg = c.fin_d + (size_t)p * FIN_D_STRIDE;
    uint32_t *rb = c.fin_rb + (size_t)p * FIN_PARTS * FIN_MAX_DIM, *cb = c.fin_cb + (size_t)p * FIN_PARTS * FIN_MAX_DIM;
    if (sub_rank == 0) {                                                 // the finisher CTA does not sort again
        int32_t *gi = c.fin_ids + (size_t)p * 2 * FIN_MAX_DIM;
        for (int k = tid; k < nr + nc; k += FIN_THREADS) gi[k < nr ? k : FIN_MAX_DIM + (k - nr)] = k < nr ? rowid[k] : colid[k - nr];
    }
    constexpr int V4 = WORDS / 4;
    // work item = (row or column, segment of FIN_SEG entries of the other side): four entries per lane, whose
    // descriptor gathers are all in flight together; one item per warp at the sizes the finisher takes
    const int segs_r = (nc + FIN_SEG - 1) / FIN_SEG, segs_c = (nr + FIN_SEG - 1) / FIN_SEG;
    const int n_items = nr * segs_r + nc * segs_c;
    const int gw = sub_rank * nw + (tid >> 5), GW = sub_count * nw;
    for (int item = gw; item < n_items; item += GW) {
        const bool is_row = item < nr * segs_r;
        const int it = is_row ? item : item - nr * segs_r, segs = is_row ? segs_r : segs_c;
        const int me = it / segs, seg = it - me * segs, n_other = is_row ? nc : nr;
        const uint32_t *mine = (is_row ? pd.q + (size_t)rowid[me] * WORDS : pd.t + (size_t)colid[me] * WORDS);
        uint32_t a[WORDS];
#pragma unroll
        for (int v = 0; v < V4; v++) {
            const uint4 u = __ldg(reinterpret_cast<const uint4 *>(mine) + v);
            a[4 * v] = u.x; a[4 * v + 1] = u.y; a[4 * v + 2] = u.z; a[4 * v + 3] = u.w;
        }
        uint4 bv[FIN_SEG / 32][V4];
#pragma unroll
        for (int e = 0; e < FIN_SEG / 32; e++) {
            const int o = seg * FIN_SEG + e * 32 + lane;
            const int oid = o < n_other ? (is_row ? colid[o] : rowid[o]) : 0;
            const uint32_t *oth = (is_row ? pd.t : pd.q) + (size_t)oid * WORDS;
#pragma unroll
            for (int v = 0; v < V4; v++) bv[e][v] = __ldg(reinterpret_cast<const uint4 *>(oth) + v);
        }
        uint32_t best = KEY_NONE;
#pragma unroll
        for (int e = 0; e < FIN_SEG / 32; e++) {
            const int o = seg * FIN_SEG + e * 32 + lane;
            uint32_t b[WORDS];
#pragma unroll
            for (int v = 0; v < V4; v++) { b[4 * v] = bv[e][v].x; b[4 * v + 1] = bv[e][v].y; b[4 * v + 2] = bv[e][v].z; b[4 * v + 3] = bv[e][v].w; }
            const uint32_t d = hamming_words<WORDS>(a, b);
            if (o < n_other) {
                if (is_row) Dg[me * S + o] = (uint16_t)d;
                best = min(best, (d << KEY_IDX_BITS) + (uint32_t)o);
            }
        }
        best = __reduce_min_sync(0xffffffffu, best);
        if (lane == 0) (is_row ? rb : cb)[seg * FIN_MAX_DIM + me] = best;
    }
}

// PRE: the matrix and the first-round minima were left in global memory by finisher_prepare (latency mode).
template <int WORDS, bool PRE>
__device__ __forceinline__ void finisher_body(const Chunk &c, int p, unsigned char *fin_smem) {
    const int tid = threadIdx.x, nt = FIN_THREADS;
    const PairDesc pd = c.pairs[p];
    const int4 si_raw = __ldcg(reinterpret_cast<const int4 *>(c.small + p));
    const SmallInfo si{si_raw.x, si_raw.y, si_raw.z, si_raw.w};
    const int nr = si.nlr, nc = si.nlc, cur = si.parity;
    const int S = finisher_pitch(nc);

    int32_t *rowid = reinterpret_cast<int32_t *>(fin_smem);
    int32_t *colid = rowid + FIN_MAX_DIM;
    int32_t *tmp = colid + FIN_MAX_DIM;                                   // 2 * FIN_MAX_DIM
    uint32_t *rkoff = reinterpret_cast<uint32_t *>(tmp + 2 * FIN_MAX_DIM);
    uint32_t *ckoff = rkoff + FIN_MAX_DIM;
    uint32_t *rbest = ckoff + FIN_MAX_DIM;
    uint32_t *cbest = rbest + FIN_MAX_DIM;
    uint16_t *D = reinterpret_cast<uint16_t *>(cbest + FIN_MAX_DIM);

    if (!PRE) finisher_sorted_ids(c, pd, nr, nc, cur, rowid, colid, tmp);
    for (int k = tid; k < nr + nc; k += nt) {
        const bool is_row = k < nr;
        const int me = is_row ? k : k - nr;
        uint32_t first = KEY_NONE;
        if (PRE) {
            const int32_t *gi = c.fin_ids + (size_t)p * 2 * FIN_MAX_DIM;
            (is_row ? rowid : colid)[me] = __ldcg(gi + (is_row ? me : FIN_MAX_DIM + me));
            const uint32_t *part = (is_row ? c.fin_rb : c.fin_cb) + (size_t)p * FIN_PARTS * FIN_MAX_DIM + me;
            const int segs = ((is_row ? nc : nr) + FIN_SEG - 1) / FIN_SEG;
            for (int sg = 0; sg < segs; sg++) first = min(first, __ldcg(part + sg * FIN_MAX_DIM));
        }
        if (is_row) { rkoff[me] = (uint32_t)me; rbest[me] = first; }
        else { ckoff[me] = (uint32_t)me; cbest[me] = first; }
    }
    if (PRE) {
        const uint4 *src = reinterpret_cast<const uint4 *>(c.fin_d + (size_t)p * FIN_D_STRIDE);
        uint4 *dst = reinterpret_cast<uint4 *>(D);
        for (int k = tid; k < (nr * S * 2 + 15) / 16; k += nt) dst[k] = __ldcg(src + k);
    }
    __syncthreads();
    tstamp(c, blockIdx.x, tid, 10);

  if (!PRE) {
    // stage both descriptor sets in shared memory (coalesced 128-bit loads), then every thread
    // computes its share of the nr x nc matrix from smem
    constexpr int V4 = WORDS / 4;
    uint4 *sq = reinterpret_cast<uint4 *>(D + (((size_t)nr * S + 7) & ~(size_t)7));
    uint4 *st = sq + (size_t)nr * V4;
    for (int k = tid; k < (nr + nc) * V4; k += nt) {
        const int row = k / V4, part = k - row * V4;
        sq[k] = row < nr ? __ldg(reinterpret_cast<const uint4 *>(pd.q + (size_t)rowid[row] * WORDS) + part)
                         : __ldg(reinterpret_cast<const uint4 *>(pd.t + (size_t)colid[row - nr] * WORDS) + part);
    }
    __syncthreads();
    tstamp(c, blockIdx.x, tid, 11);
    for (int e = tid; e < nr * nc; e += nt) {
        const int x = e / nc, y = e - x * nc;
        uint32_t q[WORDS], t[WORDS];
#pragma unroll
        for (int v = 0; v < V4; v++) {
            const uint4 a = sq[x * V4 + v], b = st[y * V4 + v];
            q[4 * v] = a.x; q[4 * v + 1] = a.y; q[4 * v + 2] = a.z; q[4 * v + 3] = a.w;
            t[4 * v] = b.x; t[4 * v + 1] = b.y; t[4 * v + 2] = b.z; t[4 * v + 3] = b.w;
        }
        D[x * S + y] = (uint16_t)hamming_words<WORDS>(q, t);
    }
    __syncthreads();
  }
    tstamp(c, blockIdx.x, tid, 12);

    int live_r = nr, live_c = nc;
    int32_t *todo = tmp;                             // the rank-sort scratch is free now: rows / columns to rescan
    __shared__ int s_todo;
    const int lane = tid & 31, wid = tid >> 5, nw = nt >> 5;
    while (live_r > 0 && live_c > 0) {
        // 1. which rows / columns lost their choice (or never had one)?  Usually a minority after the first round.
        if (tid == 0) s_todo = 0;
        __syncthreads();
        for (int k = tid; k < nr + nc; k += nt) {
            bool need;
            if (k < nr) {
                const uint32_t old = rbest[k];
                need = rkoff[k] != KEY_INVALID && (old == KEY_NONE || ckoff[old & KEY_IDX_MASK] == KEY_INVALID);
            } else {
                const uint32_t old = cbest[k - nr];
                need = ckoff[k - nr] != KEY_INVALID && (old == KEY_NONE || rkoff[old & KEY_IDX_MASK] == KEY_INVALID);
            }
            if (need) todo[atomicAdd(&s_todo, 1)] = k;
        }
        __syncthreads();
        // 2. one warp per rescan: lanes stride over the row (consecutive u16) or the column (odd word pitch:
        //    conflict-free), then a warp minimum -- the latency of a rescan is ~nc/32 steps instead of nc
        const int n_todo = s_todo;
        for (int w = wid; w < n_todo; w += nw) {
            const int k = todo[w];
            uint32_t bmin = KEY_NONE;
            if (k < nr) {
                const uint16_t *row = D + k * S;
                for (int y = lane; y < nc; y += 32) bmin = min(bmin, ((uint32_t)row[y] << KEY_IDX_BITS) + ckoff[y]);
            } else {
                const uint16_t *col = D + (k - nr);
                for (int x = lane; x < nr; x += 32) bmin = min(bmin, ((uint32_t)col[x * S] << KEY_IDX_BITS) + rkoff[x]);
            }
            bmin = __reduce_min_sync(0xffffffffu, bmin);
            if (lane == 0) { if (k < nr) rbest[k] = bmin; else cbest[k - nr] = bmin; }
        }
        __syncthreads();
        // FIN_MAX_DIM == FIN_THREADS: a thread owns at most one row
        int accepted = 0;
        if (tid < nr && rkoff[tid] != KEY_INVALID) {
            const uint32_t rk = rbest[tid];
            const uint32_t y = rk & KEY_IDX_MASK;
            if ((cbest[y] & KEY_IDX_MASK) == (uint32_t)tid) {
                c.match_key[pd.row_base + rowid[tid]] = (rk & ~KEY_IDX_MASK) | (uint32_t)colid[y];
                accepted = 1;
            }
        }
        const int n_acc = __syncthreads_count(accepted);   // everyone has read rkoff/ckoff/cbest
        if (accepted) {
            ckoff[rbest[tid] & KEY_IDX_MASK] = KEY_INVALID;  // column claimed by exactly this row
            rkoff[tid] = KEY_INVALID;
        }
        live_r -= n_acc; live_c -= n_acc;
        __syncthreads();
        tstamp(c, blockIdx.x, tid, 13);
    }
    if (tid == 0) c.status[p] = PAIR_DONE;
}

template <int WORDS>
__global__ void __launch_bounds__(FIN_THREADS) finisher_kernel(Chunk c) {
    extern __shared__ __align__(16) unsigned char dyn_smem[];
    const int p = blockIdx.x;
    if (c.status[p] != PAIR_SMALL) return;
    finisher_body<WORDS, false>(c, p, dyn_smem);
}

inline size_t finisher_smem_bytes(int words, int max_evals = FIN_MAX_EVALS) {
    // ids/keys: 8 arrays of FIN_MAX_DIM words; D: worst case rows * (pitch <= nc + 3);
    // staged descriptors: nr + nc <= FIN_MAX_DIM + max_evals / FIN_MAX_DIM rows
    return (size_t)8 * FIN_MAX_DIM * 4 + ((size_t)max_evals + 3 * FIN_MAX_DIM) * 2 + 64 +
           (size_t)(FIN_MAX_DIM + max_evals / FIN_MAX_DIM + 2) * words * 4;
}

// ---------------------------------------------------------------------------
// order kernel: one CTA per pair.  Stable counting sort of the matched rows by
// distance (rows are visited in ascending i, and a row has one j), which is
// the (distance, i, j) order the reference emits; then the degenerate tail.
// Keys of the first ORDER_KEY_CACHE rows are cached in shared memory so the
// ranking pass does not wait on global loads.
// ---------------------------------------------------------------------------
// Sliced form: the rows of pair p are cut into n_slices contiguous slices, one CTA each.  order_count histograms a
// slice (per warp, kept in shared memory) and publishes the slice's per-distance totals; after a grid-wide barrier
// order_emit turns them into output offsets -- rows with a smaller distance first, then the same distance in earlier
// slices, earlier warps, earlier lanes -- and writes the triples.  n_slices == 1 needs no global scratch / barrier.
constexpr int ORDER_MAX_SLICES = 32;
constexpr int ORDER_BIN_PITCH = 520;            // >= 513 + 1 bins
struct OrderSlice { int x_begin, x_end, seg; };

template <int ORDER_THREADS>
__device__ __forceinline__ OrderSlice order_slice_of(int n1, int slice, int n_slices) {
    constexpr int ORDER_WARPS = ORDER_THREADS / 32;
    int seg = (n1 + n_slices * ORDER_WARPS - 1) / (n_slices * ORDER_WARPS);   // rows per warp, a multiple of 32
    seg = (seg + 31) & ~31;
    const int b = min(n1, slice * seg * ORDER_WARPS);
    return OrderSlice{b, min(n1, b + seg * ORDER_WARPS), seg};
}

template <int ORDER_THREADS>
__device__ __forceinline__ void order_count(const Chunk &c, int p, int slice, int n_slices, int nbins, int32_t *s_order,
                                            int32_t *g_cnt /* [pairs][ORDER_MAX_SLICES][ORDER_BIN_PITCH] or nullptr */) {
    constexpr int ORDER_WARPS = ORDER_THREADS / 32;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const PairDesc &pd = c.pairs[p];
    const int n1 = __ldg(&pd.n1);
    const int hb = nbins + 1;                    // last bin: unmatched rows (never written out)
    int32_t *s_hist = s_order;                   // s_order: [ORDER_WARPS][nbins + 1] hist | key cache
    uint32_t *s_keys = reinterpret_cast<uint32_t *>(s_order + ORDER_WARPS * hb);
    const uint32_t *mk = c.match_key + __ldg(&pd.row_base);
    const OrderSlice sl = order_slice_of<ORDER_THREADS>(n1, slice, n_slices);
    for (int k = tid; k < ORDER_WARPS * hb; k += ORDER_THREADS) s_hist[k] = 0;
    const int x0 = min(sl.x_end, sl.x_begin + wid * sl.seg), x1 = min(sl.x_end, x0 + sl.seg);
    __syncthreads();
    for (int xb = x0; xb < x1; xb += 128) {      // 4 independent loads in flight per lane
        uint32_t k4[4];
#pragma unroll
        for (int u = 0; u < 4; u++) {
            const int x = xb + 32 * u + lane;
            k4[u] = x < x1 ? __ldcg(mk + x) : KEY_NONE;
        }
#pragma unroll
        for (int u = 0; u < 4; u++) {
            const int x = xb + 32 * u + lane;
            if (x < x1) {
                if (x - sl.x_begin < ORDER_KEY_CACHE) s_keys[x - sl.x_begin] = k4[u];
                if (k4[u] != KEY_NONE) atomicAdd(&s_hist[wid * hb + (k4[u] >> KEY_IDX_BITS)], 1);
            }
        }
    }
    __syncthreads();
    if (g_cnt && n_slices > 1) {
        int32_t *mine = g_cnt + ((size_t)p * ORDER_MAX_SLICES + slice) * ORDER_BIN_PITCH;
        for (int b = tid; b < nbins; b += ORDER_THREADS) {
            int t = 0;
            for (int w = 0; w < ORDER_WARPS; w++) t += s_hist[w * hb + b];
            mine[b] = t;
        }
    }
}

template <int ORDER_THREADS>
__device__ __forceinline__ void order_emit(const Chunk &c, int p, int slice, int n_slices, int nbins, uint32_t flags,
                                           int32_t *out_qi, int32_t *out_tj, int32_t *out_dist, int32_t *s_order,
                                           const int32_t *g_cnt) {
    constexpr int ORDER_WARPS = ORDER_THREADS / 32;
    __shared__ int32_t s_wsum[ORDER_WARPS];
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const PairDesc &pd = c.pairs[p];
    const int n1 = __ldg(&pd.n1), n2 = __ldg(&pd.n2);
    const int64_t out_base = __ldg(&pd.out_base);
    const int hb = nbins + 1;
    int32_t *s_hist = s_order;
    const uint32_t *s_keys = reinterpret_cast<const uint32_t *>(s_order + ORDER_WARPS * hb);
    const uint32_t *mk = c.match_key + __ldg(&pd.row_base);
    const OrderSlice sl = order_slice_of<ORDER_THREADS>(n1, slice, n_slices);
    const int x0 = min(sl.x_end, sl.x_begin + wid * sl.seg), x1 = min(sl.x_end, x0 + sl.seg);
    // thread t owns bins 2t and 2t+1 (nbins <= 513 <= 2 * ORDER_THREADS): totals over all slices and over the earlier
    // slices, block-wide exclusive scan over distances, then per-warp bases
    const int b0 = 2 * tid, b1 = 2 * tid + 1;
    int ta = 0, tb = 0, pa = 0, pb = 0;          // totals of the bin over every slice; over the slices before this one
    if (n_slices > 1) {
        const int32_t *pc = g_cnt + (size_t)p * ORDER_MAX_SLICES * ORDER_BIN_PITCH;
        for (int sidx = 0; sidx < n_slices; sidx++) {
            const int va = b0 < nbins ? __ldcg(pc + (size_t)sidx * ORDER_BIN_PITCH + b0) : 0;
            const int vb = b1 < nbins ? __ldcg(pc + (size_t)sidx * ORDER_BIN_PITCH + b1) : 0;
            ta += va; tb += vb;
            if (sidx < slice) { pa += va; pb += vb; }
        }
    } else {
        if (b0 < nbins) for (int w = 0; w < ORDER_WARPS; w++) ta += s_hist[w * hb + b0];
        if (b1 < nbins) for (int w = 0; w < ORDER_WARPS; w++) tb += s_hist[w * hb + b1];
    }
    int inc = ta + tb;
    for (int o = 1; o < 32; o <<= 1) { const int a = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += a; }
    if (lane == 31) s_wsum[wid] = inc;
    __syncthreads();
    int woff = 0;
    for (int w = 0; w < wid; w++) woff += s_wsum[w];
    const int start = woff + inc - (ta + tb);    // first output slot of distance b0
    int a = start + pa;
    if (b0 < nbins) for (int w = 0; w < ORDER_WARPS; w++) { const int t = s_hist[w * hb + b0]; s_hist[w * hb + b0] = a; a += t; }
    a = start + ta + pb;
    if (b1 < nbins) for (int w = 0; w < ORDER_WARPS; w++) { const int t = s_hist[w * hb + b1]; s_hist[w * hb + b1] = a; a += t; }
    __syncthreads();
    for (int xb = x0; xb < x1; xb += 32) {
        const int x = xb + lane;
        uint32_t key = KEY_NONE;
        if (x < x1) key = x - sl.x_begin < ORDER_KEY_CACHE ? s_keys[x - sl.x_begin] : __ldcg(mk + x);
        const int d = key != KEY_NONE ? (int)(key >> KEY_IDX_BITS) : nbins;
        const unsigned peers = __match_any_sync(0xffffffffu, d);
        const int rank = __popc(peers & ((1u << lane) - 1u));
        const int base = s_hist[wid * hb + d];
        __syncwarp();
        if (rank == 0) s_hist[wid * hb + d] = base + __popc(peers);
        __syncwarp();
        if (key != KEY_NONE) {
            const int64_t o = out_base + base + rank;
            PGM_ASSERT(base + rank >= 0 && base + rank < min(n1, n2) && d < nbins);
            out_qi[o] = x; out_tj[o] = (int32_t)(key & KEY_IDX_MASK); out_dist[o] = d;
        }
    }
    if (flags & 1u) {                            // PGM_FLAG_REFERENCE_COMPAT_TAIL (KeypointMatching.cs:38-42)
        const int matched = min(n1, n2);         // every pair ends with exactly min(n1,n2) real matches
        for (int k = matched + slice * ORDER_THREADS + tid; k < n1; k += n_slices * ORDER_THREADS) {
            const int64_t o = out_base + k;
            out_qi[o] = 0; out_tj[o] = 0; out_dist[o] = 2147483647;
        }
    }
}

template <int ORDER_THREADS>
__device__ __forceinline__ void order_body(const Chunk &c, int p, int nbins, uint32_t flags,
                                           int32_t *out_qi, int32_t *out_tj, int32_t *out_dist, int32_t *s_order) {
    order_count<ORDER_THREADS>(c, p, 0, 1, nbins, s_order, nullptr);
    order_emit<ORDER_THREADS>(c, p, 0, 1, nbins, flags, out_qi, out_tj, out_dist, s_order, nullptr);
}

__global__ void __launch_bounds__(ORDER_THREADS_STANDALONE) order_kernel(Chunk c, int nbins, uint32_t flags,
                                                                        int32_t *out_qi, int32_t *out_tj, int32_t *out_dist) {
    extern __shared__ __align__(16) unsigned char dyn_smem[];
    order_body<ORDER_THREADS_STANDALONE>(c, blockIdx.x, nbins, flags, out_qi, out_tj, out_dist,
                                        reinterpret_cast<int32_t *>(dyn_smem));
}

inline size_t order_smem_bytes(int nbins, int threads) {
    return sizeof(int32_t) * ((size_t)(threads / 32) * (nbins + 1) + ORDER_KEY_CACHE);
}

// ---------------------------------------------------------------------------
// persistent tail kernel (latency mode: one or a few pairs).  After the first
// full round, what remains is a chain of short rounds whose cost is dominated
// by kernel boundaries.  This kernel is launched cooperatively with one
// 512-thread CTA per SM and runs every remaining round (round phase -> grid
// barrier -> accept phase + planner in the last CTA -> grid barrier), then the
// finisher and the ordering of each pair, with no host involvement.
// ---------------------------------------------------------------------------
__device__ __forceinline__ void stamp(const Chunk &c, int &slot) {
    if (c.timeline && blockIdx.x == 0 && threadIdx.x == 0 && slot < 1000) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        c.timeline[slot] = t;
    }
    slot++;
}

__device__ __forceinline__ unsigned ld_acquire_u32(const unsigned *p) {
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

// All CTAs are co-resident (cooperative launch), so a counting barrier in global memory is safe.
__device__ __forceinline__ void grid_barrier(unsigned *counter, unsigned nblocks, unsigned &epoch) {
    epoch += nblocks;                 // the counter only grows: the k-th barrier completes at k * nblocks
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        atomicAdd(counter, 1u);
        while (ld_acquire_u32(counter) < epoch) {}
        __threadfence();
    }
    __syncthreads();
}

template <int WORDS>
__host__ __device__ constexpr size_t tail_group_bytes() {   // one 128-thread group of the round phase: staged train tile, keys, column minima, edges
    return (size_t)STAGE_LARGE * (WORDS / 4) * 16 + (size_t)STAGE_LARGE * 8 + (size_t)SCAND * 16 + 16;
}
template <int WORDS>
inline size_t tail_smem_bytes(int nbins) {
    const size_t round_bytes = 4 * tail_group_bytes<WORDS>();
    return std::max(std::max(round_bytes, (size_t)SP_SMEM_BYTES),
                    std::max(finisher_smem_bytes(WORDS, FIN_MAX_EVALS_TAIL), order_smem_bytes(nbins, TAIL_THREADS)));
}

template <int WORDS>
__global__ void __launch_bounds__(TAIL_THREADS, 1) tail_kernel(Chunk c, int r_start, int nbins, uint32_t flags,
                                                              int32_t *out_qi, int32_t *out_tj, int32_t *out_dist) {
    extern __shared__ __align__(16) unsigned char dyn_smem[];
    constexpr int V4 = WORDS / 4;
    constexpr size_t GROUP_BYTES = tail_group_bytes<WORDS>();
    const int tid = threadIdx.x, grp = tid >> 7, gtid = tid & 127;
    unsigned char *gb = dyn_smem + grp * GROUP_BYTES;
    uint4 *s_t = reinterpret_cast<uint4 *>(gb);
    uint32_t *s_jkey = reinterpret_cast<uint32_t *>(gb + (size_t)STAGE_LARGE * V4 * 16);
    uint32_t *s_col = s_jkey + STAGE_LARGE;
    unsigned long long *s_cand = reinterpret_cast<unsigned long long *>(s_col + STAGE_LARGE);
    int *s_cctl = reinterpret_cast<int *>(s_cand + 2 * SCAND);
    unsigned epoch = 0;
    unsigned *bar_counter = &c.plan->grid_bar;
    int slot = 0;
    stamp(c, slot);

    // what follows every distance pass r: accept + candidate-edge filter (all CTAs) | barrier | sparse sub-rounds of
    // pair p in CTA p, the last of them plans pass r + 1 | barrier
    auto after_pass = [&](int r) {
        accept_blocks(c, r, (tid >> 8) * gridDim.x + blockIdx.x, gridDim.x * 2, tid & (ACCEPT_THREADS - 1));
        const int gw32 = (int)((blockIdx.x * TAIL_THREADS + tid) & ~31u);
        for (int p = 0; p < c.n_pairs; p++) filter_edges(c, r, p, gw32, (int)gridDim.x * TAIL_THREADS);
        stamp(c, slot);
        grid_barrier(bar_counter, gridDim.x, epoch);
        stamp(c, slot);
        if ((int)blockIdx.x < c.n_pairs) {
            sparse_body<TAIL_THREADS>(c, r, blockIdx.x, dyn_smem);
            if (c.n_pairs == 1) { __syncthreads(); if (tid < 32) plan_warp(c, r + 1); }   // (no ticket to take)
            else plan_in_last_block(c, r + 1, (unsigned)c.n_pairs);
        }
        stamp(c, slot);
        grid_barrier(bar_counter, gridDim.x, epoch);
        stamp(c, slot);
    };
    // (one copy of the pass body: the kernel's code size is what its short phases pay for in instruction-cache misses)
    bool have_pass = (flags & TAIL_FLAG_ACCEPT_FIRST) != 0;         // round r_start - 1 ran as a standalone launch
    for (int r = have_pass ? r_start - 1 : r_start;; r++) {
        if (!have_pass) {
            // plan(r) was published before the previous barrier (or by the preceding kernel)
            if (__ldcg(&c.plan->n_big) == 0) break;
            const int total = __ldcg(&c.plan->total_tiles);
            const int cpt = __ldcg(&c.plan->cols_per_tile);
            const int rq = __ldcg(&c.plan->rq);
            const GroupBar bar{1 + grp, ROUND_THREADS};
            if (rq == RQ_LARGE)
                round_tiles<WORDS, RQ_LARGE, STAGE_LARGE>(c, r, total, cpt, grp * gridDim.x + blockIdx.x, gridDim.x * 4, gtid, bar, s_t, s_jkey, s_col, s_cand, s_cctl);
            else
                round_tiles<WORDS, RQ_SMALL, STAGE_SMALL>(c, r, total, cpt, grp * gridDim.x + blockIdx.x, gridDim.x * 4, gtid, bar, s_t, s_jkey, s_col, s_cand, s_cctl);
            stamp(c, slot);
            grid_barrier(bar_counter, gridDim.x, epoch);
            stamp(c, slot);
        }
        have_pass = false;
        after_pass(r);
    }
    // every small pair's distance matrix and first-round minima, computed by all CTAs (finisher_prepare)
    // (the grid is split among the small pairs: CTA b works on the (b mod n_small)-th of them)
    // (a small pair whose matrix has at most FIN_PREP_MIN_EVALS cells is not worth the extra grid phase: its finisher
    //  CTA computes the few distances itself -- after the sparse sub-rounds a pair usually arrives here with ~30 rows)
    int n_small = 0, n_prep = 0, my_pair = -1;
    stamp(c, slot);
    for (int p = 0; p < c.n_pairs; p++)
        if (__ldcg(c.status + p) == PAIR_SMALL) {
            n_small++;
            const int4 si = __ldcg(reinterpret_cast<const int4 *>(c.small + p));
            if (si.x * si.y > FIN_PREP_MIN_EVALS) n_prep++;
        }
    stamp(c, slot);
    if (n_prep) {                                     // uniform: every CTA reads the same statuses
        const int mine = (int)blockIdx.x % n_prep;
        for (int p = 0, k = 0; p < c.n_pairs; p++)
            if (__ldcg(c.status + p) == PAIR_SMALL) {
                const int4 si = __ldcg(reinterpret_cast<const int4 *>(c.small + p));
                if (si.x * si.y > FIN_PREP_MIN_EVALS && k++ == mine) my_pair = p;
            }
        finisher_prepare<WORDS>(c, my_pair, dyn_smem, (int)blockIdx.x / n_prep,
                                ((int)gridDim.x - mine + n_prep - 1) / n_prep);
        __threadfence();
        grid_barrier(bar_counter, gridDim.x, epoch);
    }
    for (int p = blockIdx.x; p < c.n_pairs; p += gridDim.x) {
        stamp(c, slot);
        if (__ldcg(c.status + p) == PAIR_SMALL) {
            const int4 si = __ldcg(reinterpret_cast<const int4 *>(c.small + p));
            if (si.x * si.y > FIN_PREP_MIN_EVALS) finisher_body<WORDS, true>(c, p, dyn_smem);
            else finisher_body<WORDS, false>(c, p, dyn_smem);
        }
    }
    if (n_small) {                                    // the finishers' matches must be visible to every ordering CTA
        __threadfence();
        grid_barrier(bar_counter, gridDim.x, epoch);
    }
    stamp(c, slot);
    // ordering, sliced over the grid: S CTAs per pair (count | barrier | emit)
    const int S = max(1, min(ORDER_MAX_SLICES, (int)gridDim.x / c.n_pairs));
    const bool ordering = (int)blockIdx.x < c.n_pairs * S;
    const int op = (int)blockIdx.x / S, oslice = (int)blockIdx.x - op * S;
    __syncthreads();                                  // the finisher's shared memory is reused
    if (ordering) order_count<TAIL_THREADS>(c, op, oslice, S, nbins, reinterpret_cast<int32_t *>(dyn_smem), c.order_cnt);
    if (S > 1) grid_barrier(bar_counter, gridDim.x, epoch);
    stamp(c, slot);
    if (ordering) order_emit<TAIL_THREADS>(c, op, oslice, S, nbins, flags, out_qi, out_tj, out_dist,
                                           reinterpret_cast<int32_t *>(dyn_smem), c.order_cnt);
    stamp(c, slot);
    // the last CTA out publishes the call's statistics and zeroes the plan for the next call (every CTA is past its last
    // grid barrier once it counts itself out, so the barrier counter can be reset)
    if (c.lat && tid == 0) {
        if (atomicAdd(&c.lat->exit_cnt, 1u) == gridDim.x - 1) {
            PlanInfo *pl = &c.lat->plan;
            const int done = __ldcg(&pl->done_round_p1), rnd = __ldcg(&pl->round);
            c.lat->last_rounds = (unsigned long long)(done > 0 ? done - 1 : rnd);
            c.lat->last_evals = __ldcg(&pl->evals);
            pl->total_tiles = 0; pl->cols_per_tile = 0; pl->total_ablocks = 0; pl->n_big = 0; pl->n_small = 0; pl->round = 0;
            pl->ticket = 0u; pl->done_round_p1 = 0; pl->rq = 0; pl->grid_bar = 0u; pl->evals = 0ull;
            c.lat->exit_cnt = 0u;
        }
    }
}

// ---------------------------------------------------------------------------
// train-sharded single pair (SURVEY.md section 8e): every rank holds all N1 queries and a contiguous slice of the
// train set.  Per round each rank runs the ordinary round kernel on (live rows x live LOCAL columns) with global column
// ids in the row keys, then ONE exchange decides the round: X = [R | P], both indexed by the row's position in the live
// list (identical on every rank: the row compaction below is stable),
//     R[pos] = the row's best key over the rank's columns          (d << 20 | global j)
//     P[pos] = the best key among the rank's columns that CHOSE this row as their best row (each rank sees every
//              row, so a local column's choice is final without any exchange)
// and after an element-wise `min` over the ranks (NCCL all-reduce, or any other transport) row `pos` is matched iff
// R[pos] == P[pos]: P >= R always (P ranges over a subset of the row's columns), with equality exactly when the row's
// best column chose it back -- the locally dominant edge the reference's argmin scan emits next
// (KeypointMatching.cs:44-65).  Every rank commits identically.  Exchange buffers use 0x7F7F7F7F for "none" so that a
// signed 32-bit min (what some transports offer) orders them like the unsigned keys.
// ---------------------------------------------------------------------------
constexpr uint32_t XKEY_NONE = 0x7F7F7F7Fu;   // memset-able, above every real key, positive as int32
constexpr int SHARD_BLOCK = 1024;             // rows per block of the stable row compaction

struct ShardCtl {                 // device resident, one per sharded pair
    int32_t done;                 // sticky: no live row or no live column is left anywhere
    int32_t live_rows;            // after the last commit (identical on every rank)
    int32_t live_cols_local;
    int32_t rounds;               // commits that found the pair not yet done
};

// X[0, bound) = R (padded with none), X[bound, 2 bound) = none (the proposals are min-ed in by the next kernel)
__global__ void shard_export_rows_kernel(Chunk c, int r, uint32_t *__restrict__ X, int bound) {
    const int nlr = __ldcg(cnt_ptr(c, r % 3, 0));
    const int32_t *live = c.live_rows[r & 1];
    const uint32_t *rowbest = c.rowbest[r & 1];
    for (int pos = blockIdx.x * blockDim.x + threadIdx.x; pos < bound; pos += gridDim.x * blockDim.x) {
        uint32_t k = XKEY_NONE;
        if (pos < nlr) { const uint32_t v = __ldcg(rowbest + __ldcg(live + pos)); if (v != KEY_NONE) k = v; }
        X[pos] = k;
        X[bound + pos] = XKEY_NONE;
    }
}

// every live local column proposes (distance, its GLOBAL id) to the row it chose
__global__ void shard_propose_cols_kernel(Chunk c, int r, uint32_t *__restrict__ X, int bound) {
    const PairDesc &pd = c.pairs[0];
    const int nlc = __ldcg(cnt_ptr(c, r % 3, 0) + 1);
    const int32_t *live = c.live_cols[r & 1];
    const uint32_t *colbest = c.colbest[r & 1];
    const int off = __ldg(&pd.col_id_offset);
    for (int y = blockIdx.x * blockDim.x + threadIdx.x; y < nlc; y += gridDim.x * blockDim.x) {
        const int j = __ldcg(live + y);
        const uint32_t ck = __ldcg(colbest + j);
        if (ck == KEY_NONE) continue;
        const int pos = r == 0 ? (int)(ck & KEY_IDX_MASK) : __ldcg(c.row_pos + (ck & KEY_IDX_MASK));   // round 0: identity list
        PGM_ASSERT((int)(ck & KEY_IDX_MASK) < pd.n1 && pos >= 0 && pos < bound);
        if (pos < bound) atomicMin(X + bound + pos, (ck & ~KEY_IDX_MASK) | (uint32_t)(j + off));
    }
}

// X: reduced over the ranks.  Commit, step 1: record the matches and flag their columns dead (every rank sees every
// match, so every rank keeps the dead flags of ALL columns: coldead[global j]).
__global__ void __launch_bounds__(SHARD_BLOCK) shard_commit_mark_kernel(Chunk c, int r, const uint32_t *__restrict__ X, int bound,
                                                                        uint8_t *__restrict__ coldead) {
    const int nlr = __ldcg(cnt_ptr(c, r % 3, 0));
    const int pos = blockIdx.x * SHARD_BLOCK + threadIdx.x;
    if (pos < nlr && pos < bound) {
        const uint32_t R = __ldcg(X + pos), P = __ldcg(X + bound + pos);
        if (R != XKEY_NONE && R == P) {
            const int i = __ldcg(c.live_rows[r & 1] + pos);
            c.match_key[i] = R;
            coldead[R & KEY_IDX_MASK] = 1;
        }
    }
}

// Commit, step 2 (candidate edges, SURVEY-free extension of section 3.1 to the sharded pair): this rank's candidate
// records of the pass -> the edges whose row and column are both still unmatched, with the emitting thread's sibling
// rows verified.  out[0] = number of edges (SHARD_EDGE_OVERFLOW if this rank's lists cannot be trusted), out[1 + k] =
// (d << 40 | i << 20 | GLOBAL j).
constexpr unsigned long long SHARD_EDGE_OVERFLOW = 0x7FFFFFFFull;
__global__ void __launch_bounds__(ACCEPT_THREADS) shard_filter_kernel(Chunk c, int r, const uint8_t *__restrict__ coldead,
                                                                      unsigned long long *__restrict__ out, int out_cap,
                                                                      int32_t *__restrict__ out_cnt, unsigned *__restrict__ ticket) {
    const PairDesc &pd = c.pairs[0];
    const int n = __ldcg(c.cand_cnt), cap = __ldg(&pd.cand_cap);
    if (n > cap) { if (blockIdx.x == 0 && threadIdx.x == 0) out[0] = SHARD_EDGE_OVERFLOW; return; }     // (uniform)
    const int lane = threadIdx.x & 31, words = c.words, off = __ldg(&pd.col_id_offset);
    const int32_t *live_rows = c.live_rows[r & 1];
    const int nlr = __ldcg(cnt_ptr(c, r % 3, 0));
    const uint32_t thr = __ldcg(c.thr);
    const uint32_t *qd = pd.q, *td = pd.t;
    const unsigned long long *raw = c.cand + 2 * __ldg(&pd.cand_off);
    const int start = (int)((blockIdx.x * ACCEPT_THREADS + threadIdx.x) & ~31u), step = (int)gridDim.x * ACCEPT_THREADS;
    for (int e0 = start; e0 < n; e0 += step) {
        const int e = e0 + lane;
        unsigned long long ed[RQ_LARGE];
#pragma unroll
        for (int k = 0; k < RQ_LARGE; k++) ed[k] = ~0ull;
        if (e < n) {
            const unsigned long long key = __ldcg(raw + 2 * e);
            const uint32_t aux = (uint32_t)__ldcg(raw + 2 * e + 1);
            ed[0] = key;
            const int rqn = (int)(aux >> KEY_IDX_BITS), slot0 = (int)(aux & KEY_IDX_MASK);
            if (rqn > 1) {
                const uint32_t i0 = (uint32_t)(key >> KEY_IDX_BITS) & KEY_IDX_MASK, j = (uint32_t)key & KEY_IDX_MASK;
                PGM_ASSERT((int)j - off >= 0 && (int)j - off < pd.n2);
                uint32_t tw[16];
#pragma unroll
                for (int v = 0; v < 4; v++) {
                    const uint4 x = 4 * v < words ? __ldg(reinterpret_cast<const uint4 *>(td + (size_t)(j - off) * words) + v) : make_uint4(0u, 0u, 0u, 0u);
                    tw[4 * v] = x.x; tw[4 * v + 1] = x.y; tw[4 * v + 2] = x.z; tw[4 * v + 3] = x.w;
                }
                int used = 1;
                for (int k = 0; k < rqn && k < RQ_LARGE; k++) {
                    const int slot = slot0 + k * ROUND_THREADS;
                    if (slot >= nlr) break;
                    const uint32_t i2 = (uint32_t)__ldcg(live_rows + slot);
                    if (i2 == i0) continue;
                    uint32_t d = 0;
#pragma unroll
                    for (int v = 0; v < 4; v++) {
                        if (4 * v < words) {
                            const uint4 x = __ldg(reinterpret_cast<const uint4 *>(qd + (size_t)i2 * words) + v);
                            d += __popc(x.x ^ tw[4 * v]) + __popc(x.y ^ tw[4 * v + 1]) + __popc(x.z ^ tw[4 * v + 2]) + __popc(x.w ^ tw[4 * v + 3]);
                        }
                    }
                    if ((d << KEY_IDX_BITS) < thr) {
                        const unsigned long long k2 = ((unsigned long long)d << 40) | ((unsigned long long)i2 << 20) | j;
                        if (used == 1) ed[1] = k2; else if (used == 2) ed[2] = k2; else ed[3] = k2;
                        used++;
                    }
                }
            }
        }
#pragma unroll
        for (int x = 0; x < RQ_LARGE; x++) {
            bool keep = false;
            if (ed[x] != ~0ull) {
                const uint32_t i = (uint32_t)(ed[x] >> KEY_IDX_BITS) & KEY_IDX_MASK, j = (uint32_t)ed[x] & KEY_IDX_MASK;
                keep = __ldcg(c.match_key + i) == KEY_NONE && !coldead[j];
            }
            const unsigned m = __ballot_sync(0xffffffffu, keep);
            if (m) {
                int base = 0;
                if (lane == (__ffs(m) - 1)) base = atomicAdd(out_cnt, __popc(m));
                base = __shfl_sync(0xffffffffu, base, __ffs(m) - 1);
                const int pos = base + __popc(m & ((1u << lane) - 1u));
                if (keep && pos < out_cap) out[1 + pos] = ed[x];
            }
        }
    }
    // the last block to finish publishes the edge count next to the edges
    __shared__ bool s_last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = atomicAdd(ticket, 1u) == gridDim.x - 1;
    __syncthreads();
    if (s_last && threadIdx.x == 0) {
        __threadfence();
        const int total = __ldcg(out_cnt);
        out[0] = total > out_cap ? SHARD_EDGE_OVERFLOW : (unsigned long long)total;
    }
}

// Commit, step 3: the sparse sub-rounds of section 3.1 over the edges of ALL ranks (gathered: all[g][1 + cap]), by the
// whole grid (cooperative launch), every rank redundantly and identically.  One min slot per row and per GLOBAL column
// in global memory, addressed by original id (a pair of this size does not fit one CTA's shared memory).  est[] holds
// one live bit per edge slot.  Skipped altogether (uniformly on every rank) if any rank reported an overflow.
__global__ void __launch_bounds__(TAIL_THREADS, 1) shard_sparse_kernel(Chunk c, const unsigned long long *__restrict__ all,
                                                                       int n_ranks, int cap, uint32_t *__restrict__ rbest,
                                                                       uint32_t *__restrict__ cbest, uint8_t *__restrict__ coldead,
                                                                       uint8_t *__restrict__ est, unsigned *bar_counter,
                                                                       int32_t *alive_cnt /*[2]*/) {
    __shared__ int s_cnt[64], s_pre[65];
    const int tid = threadIdx.x;
    unsigned epoch = 0;
    for (int g = tid; g < n_ranks && g < 64; g += TAIL_THREADS) {
        const unsigned long long v = __ldcg(all + (size_t)g * (1 + cap));
        s_cnt[g] = v >= SHARD_EDGE_OVERFLOW ? -1 : (int)v;
    }
    __syncthreads();
    for (int g = 0; g < n_ranks; g++) if (s_cnt[g] < 0) return;              // uniform: every CTA reads the same counts
    if (tid == 0) { int a = 0; for (int g = 0; g < n_ranks; g++) { s_pre[g] = a; a += s_cnt[g]; } s_pre[n_ranks] = a; }
    __syncthreads();
    const int E = s_pre[n_ranks];                                            // edges of all ranks, addressed 0 .. E-1
    if (E == 0) return;
    const int gt = (int)blockIdx.x * TAIL_THREADS + tid, gs = (int)gridDim.x * TAIL_THREADS;
    uint32_t *match_key = c.match_key;
    auto edge_at = [&](int e) -> unsigned long long {
        int g = 0;
        while (g + 1 < n_ranks && s_pre[g + 1] <= e) g++;
        return __ldcg(all + (size_t)g * (1 + cap) + 1 + (e - s_pre[g]));
    };
    for (int e = gt; e < E; e += gs) est[e] = 1;
    if (blockIdx.x == 0 && tid == 0) { alive_cnt[0] = 0; alive_cnt[1] = 0; }
    grid_barrier(bar_counter, gridDim.x, epoch);
    for (int sub = 0; sub < SP_MAX_SUB; sub++) {
        for (int e = gt; e < E; e += gs) {
            if (!est[e]) continue;
            const unsigned long long key = edge_at(e);
            const uint32_t d = (uint32_t)(key >> 40), i = (uint32_t)(key >> KEY_IDX_BITS) & KEY_IDX_MASK, j = (uint32_t)key & KEY_IDX_MASK;
            atomicMin(rbest + i, (d << KEY_IDX_BITS) | j);
            atomicMin(cbest + j, (d << KEY_IDX_BITS) | i);
        }
        grid_barrier(bar_counter, gridDim.x, epoch);
        for (int e = gt; e < E; e += gs) {
            if (!est[e]) continue;
            const unsigned long long key = edge_at(e);
            const uint32_t d = (uint32_t)(key >> 40), i = (uint32_t)(key >> KEY_IDX_BITS) & KEY_IDX_MASK, j = (uint32_t)key & KEY_IDX_MASK;
            // (only the threads of THE mutual edge of a row / column pass this test, so nobody races on these stores)
            if (__ldcg(rbest + i) == ((d << KEY_IDX_BITS) | j) && __ldcg(cbest + j) == ((d << KEY_IDX_BITS) | i)) {
                match_key[i] = (d << KEY_IDX_BITS) | j;
                coldead[j] = 1;
            }
        }
        if (blockIdx.x == 0 && tid == 0) alive_cnt[(sub + 1) & 1] = 0;
        grid_barrier(bar_counter, gridDim.x, epoch);
        int alive = 0;
        for (int e = gt; e < E; e += gs) {
            if (!est[e]) continue;
            const unsigned long long key = edge_at(e);
            const uint32_t i = (uint32_t)(key >> KEY_IDX_BITS) & KEY_IDX_MASK, j = (uint32_t)key & KEY_IDX_MASK;
            // every slot touched in this sub-round goes back to "none": a live row whose listed edges all died must not
            // carry a stale minimum into the next pass
            rbest[i] = KEY_NONE; cbest[j] = KEY_NONE;
            if (__ldcg(match_key + i) != KEY_NONE || __ldcg(coldead + j)) est[e] = 0; else alive++;
        }
        alive = __reduce_add_sync(0xffffffffu, alive);
        if ((tid & 31) == 0 && alive) atomicAdd(&alive_cnt[sub & 1], alive);
        grid_barrier(bar_counter, gridDim.x, epoch);
        if (__ldcg(&alive_cnt[sub & 1]) == 0) break;                         // uniform
    }
}

// Commit, step 4: survivors of each block of SHARD_BLOCK live-list positions (a row survives iff it is still unmatched)
__global__ void __launch_bounds__(SHARD_BLOCK) shard_count_kernel(Chunk c, int r, int32_t *__restrict__ blockcnt) {
    const int nlr = __ldcg(cnt_ptr(c, r % 3, 0));
    const int pos = blockIdx.x * SHARD_BLOCK + threadIdx.x;
    const bool survive = pos < nlr && __ldcg(c.match_key + __ldcg(c.live_rows[r & 1] + pos)) == KEY_NONE;
    const int n = __syncthreads_count(survive);
    if (threadIdx.x == 0) blockcnt[blockIdx.x] = n;
}

// Commit, step 5: stable compaction of the surviving rows (block b starts behind the survivors of blocks 0 .. b-1), so
// every rank ends up with the same list in the same order.  Also keeps row_pos and resets the survivors' keys.
__global__ void __launch_bounds__(SHARD_BLOCK) shard_commit_scatter_kernel(Chunk c, int r, const int32_t *__restrict__ blockcnt,
                                                                           int n_blocks, ShardCtl *__restrict__ ctl, int n1,
                                                                           int n2_total) {
    __shared__ int s_w[SHARD_BLOCK / 32], s_base, s_total;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int cur = r & 1, nxt = cur ^ 1;
    const int nlr = __ldcg(cnt_ptr(c, r % 3, 0));
    int before = 0, total = 0;
    for (int b = tid; b < n_blocks; b += SHARD_BLOCK) {
        const int v = (b * SHARD_BLOCK < nlr) ? __ldcg(blockcnt + b) : 0;
        total += v;
        if (b < (int)blockIdx.x) before += v;
    }
    before = __reduce_add_sync(0xffffffffu, before); total = __reduce_add_sync(0xffffffffu, total);
    if (tid == 0) { s_base = 0; s_total = 0; }
    __syncthreads();
    if (lane == 0) { atomicAdd(&s_base, before); atomicAdd(&s_total, total); }
    __syncthreads();
    const int pos = blockIdx.x * SHARD_BLOCK + tid;
    bool survive = false;
    int i = 0;
    if (pos < nlr) {
        i = __ldcg(c.live_rows[cur] + pos);
        survive = __ldcg(c.match_key + i) == KEY_NONE;
    }
    const unsigned m = __ballot_sync(0xffffffffu, survive);
    if (lane == 0) s_w[wid] = __popc(m);
    __syncthreads();
    int woff = s_base;
    for (int w = 0; w < wid; w++) woff += s_w[w];
    if (survive) {
        const int np = woff + __popc(m & ((1u << lane) - 1u));
        PGM_ASSERT(np >= 0 && np <= pos && i >= 0 && i < n1);
        c.live_rows[nxt][np] = i;
        c.row_pos[i] = np;
        c.rowbest[nxt][i] = KEY_NONE;
    }
    if (blockIdx.x == 0 && tid == 0) {
        const int left = s_total;
        cnt_ptr(c, (r + 1) % 3, 0)[0] = left;
        const bool was_done = ctl->done != 0;
        ctl->live_rows = left;
        if (!was_done) ctl->rounds = r + 1;
        if (left == 0 || n2_total - (n1 - left) <= 0) ctl->done = 1;
    }
}

// Commit, step 6: the rank's own columns (coldead is indexed by GLOBAL column id); the last block plans the next pass
__global__ void __launch_bounds__(ACCEPT_THREADS) shard_commit_cols_kernel(Chunk c, int r, const uint8_t *coldead, ShardCtl *ctl) {
    const int cur = r & 1, nxt = cur ^ 1, lane = threadIdx.x & 31;
    const int nlc = __ldcg(cnt_ptr(c, r % 3, 0) + 1);
    const int off = __ldg(&c.pairs[0].col_id_offset);
    const int nrounded = (nlc + 31) & ~31;
    for (int y = blockIdx.x * blockDim.x + threadIdx.x; y < nrounded; y += gridDim.x * blockDim.x) {
        bool survive = false;
        int j = 0;
        if (y < nlc) {
            j = __ldcg(c.live_cols[cur] + y);
            if (!coldead[j + off]) { survive = true; c.colbest[nxt][j] = KEY_NONE; }
        }
        const unsigned m = __ballot_sync(0xffffffffu, survive);
        if (m) {
            int base = 0;
            if (lane == (__ffs(m) - 1)) base = atomicAdd(cnt_ptr(c, (r + 1) % 3, 0) + 1, __popc(m));
            base = __shfl_sync(0xffffffffu, base, __ffs(m) - 1);
            if (survive) c.live_cols[nxt][base + __popc(m & ((1u << lane) - 1u))] = j;
        }
    }
    plan_in_last_block(c, r + 1, gridDim.x);
    (void)ctl;
}

// ---- replicated finish of a train-sharded pair (pgm_multi): once few rows are left, every rank collects the descriptors
// of all surviving rows and columns and finishes the remaining (small) problem itself with the single-GPU engine ----
__global__ void shard_gather_rows_kernel(const uint32_t *__restrict__ q, const int32_t *__restrict__ live, int n, int words,
                                         uint32_t *__restrict__ out) {
    const int v4 = words >> 2;
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n * v4; k += gridDim.x * blockDim.x) {
        const int row = k / v4, part = k - row * v4;
        reinterpret_cast<uint4 *>(out)[k] = __ldg(reinterpret_cast<const uint4 *>(q + (size_t)__ldcg(live + row) * words) + part);
    }
}

// this rank's surviving columns in ASCENDING order (one block, ordered compaction over the dead flags):
// block[0] = count (16-byte header), then ids (global) int32[cap], then descriptors uint32[cap][words] (16-byte aligned)
__global__ void __launch_bounds__(1024) shard_pack_cols_kernel(const uint32_t *__restrict__ t, int n2_local, int off, int words,
                                                               const uint8_t *__restrict__ coldead, int cap,
                                                               unsigned long long *__restrict__ block) {
    __shared__ int s_w[32], s_base;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, v4 = words >> 2;
    int32_t *ids = reinterpret_cast<int32_t *>(block + 2);
    uint4 *desc = reinterpret_cast<uint4 *>(reinterpret_cast<char *>(block + 2) + (((size_t)cap * 4 + 15) & ~(size_t)15));
    if (tid == 0) s_base = 0;
    __syncthreads();
    for (int j0 = 0; j0 < n2_local; j0 += 1024) {
        const int j = j0 + tid;
        const bool alive = j < n2_local && !coldead[j + off];
        const unsigned m = __ballot_sync(0xffffffffu, alive);
        if (lane == 0) s_w[wid] = __popc(m);
        __syncthreads();
        int o = s_base;
        for (int w = 0; w < wid; w++) o += s_w[w];
        if (alive) {
            const int at = o + __popc(m & ((1u << lane) - 1u));
            if (at < cap) {
                ids[at] = j + off;
                for (int v = 0; v < v4; v++) desc[(size_t)at * v4 + v] = __ldg(reinterpret_cast<const uint4 *>(t + (size_t)j * words) + v);
            }
        }
        __syncthreads();
        if (tid == 0) { int tot = 0; for (int w = 0; w < 32; w++) tot += s_w[w]; s_base += tot; }
        __syncthreads();
    }
    if (tid == 0) block[0] = (unsigned long long)s_base;
}

// the ranks' column blocks (rank order = ascending global id) -> one dense train set + its global ids
__global__ void shard_merge_cols_kernel(const unsigned long long *__restrict__ all, size_t block_words64, int n_ranks, int cap,
                                        int words, uint32_t *__restrict__ t_sub, int32_t *__restrict__ gid, int total_expected,
                                        int32_t *__restrict__ mismatch) {
    __shared__ int s_pre[65];
    const int v4 = words >> 2;
    if (threadIdx.x == 0) {
        int a = 0;
        for (int g = 0; g < n_ranks; g++) { s_pre[g] = a; a += (int)min((unsigned long long)cap, __ldcg(all + (size_t)g * block_words64)); }
        s_pre[n_ranks] = a;
        if (blockIdx.x == 0 && a != total_expected) *mismatch = 1;
    }
    __syncthreads();
    const int total = min(s_pre[n_ranks], total_expected);
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < total; k += gridDim.x * blockDim.x) {
        int g = 0;
        while (g + 1 < n_ranks && s_pre[g + 1] <= k) g++;
        const unsigned long long *blk = all + (size_t)g * block_words64;
        const int32_t *ids = reinterpret_cast<const int32_t *>(blk + 2);
        const uint4 *desc = reinterpret_cast<const uint4 *>(reinterpret_cast<const char *>(blk + 2) + (((size_t)cap * 4 + 15) & ~(size_t)15));
        const int e = k - s_pre[g];
        gid[k] = __ldcg(ids + e);
        for (int v = 0; v < v4; v++) reinterpret_cast<uint4 *>(t_sub)[(size_t)k * v4 + v] = __ldcg(desc + (size_t)e * v4 + v);
    }
}

// triples of the sub-problem (indices into the gathered rows / columns) -> match keys of the original rows
__global__ void shard_map_matches_kernel(const int32_t *__restrict__ sq, const int32_t *__restrict__ st, const int32_t *__restrict__ sd,
                                         int n, const int32_t *__restrict__ live_rows, const int32_t *__restrict__ gid,
                                         uint32_t *__restrict__ match_key) {
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x)
        match_key[__ldcg(live_rows + sq[k])] = ((uint32_t)sd[k] << KEY_IDX_BITS) | (uint32_t)__ldcg(gid + st[k]);
}

// ---------------------------------------------------------------------------
// nearest / second nearest (no masks): same tiling, two keys per row in
// registers; column splits write partial top-2 that a merge kernel combines.
// ---------------------------------------------------------------------------
template <int WORDS, int RQ>
__global__ void __launch_bounds__(ROUND_THREADS) knn2_kernel(const uint32_t *__restrict__ qd, int n1,
                                                            const uint32_t *__restrict__ td, int n2,
                                                            int cols_per_split, uint32_t *__restrict__ part /*[splits][n1][2]*/) {
    constexpr int V4 = WORDS / 4;
    __shared__ uint4 s_t[STAGE_COLS * V4];
    const int tid = threadIdx.x;
    const int tile_rows = ROUND_THREADS * RQ;
    const int rt = blockIdx.x, sp = blockIdx.y;
    uint32_t q[RQ][WORDS], best[RQ], second[RQ];
#pragma unroll
    for (int k = 0; k < RQ; k++) {
        const int i = rt * tile_rows + k * ROUND_THREADS + tid;
        best[k] = KEY_NONE; second[k] = KEY_NONE;
        const uint4 *src = reinterpret_cast<const uint4 *>(qd + (size_t)min(i, n1 - 1) * WORDS);
#pragma unroll
        for (int v = 0; v < V4; v++) {
            const uint4 x = __ldg(src + v);
            q[k][4 * v + 0] = x.x; q[k][4 * v + 1] = x.y; q[k][4 * v + 2] = x.z; q[k][4 * v + 3] = x.w;
        }
    }
    const int c0 = sp * cols_per_split, c1 = min(n2, c0 + cols_per_split);
    for (int s0 = c0; s0 < c1; s0 += STAGE_COLS) {
        __syncthreads();
        for (int k = tid; k < STAGE_COLS * V4; k += ROUND_THREADS) {
            const int col = k / V4, part_i = k - col * V4, j = s0 + col;
            s_t[k] = j < c1 ? __ldg(reinterpret_cast<const uint4 *>(td + (size_t)j * WORDS) + part_i)
                            : make_uint4(0u, 0u, 0u, 0u);
        }
        __syncthreads();
        const int ncs = min(STAGE_COLS, c1 - s0);
        for (int jj = 0; jj < ncs; jj++) {
            uint32_t t[WORDS];
#pragma unroll
            for (int v = 0; v < V4; v++) {
                const uint4 x = s_t[jj * V4 + v];
                t[4 * v + 0] = x.x; t[4 * v + 1] = x.y; t[4 * v + 2] = x.z; t[4 * v + 3] = x.w;
            }
            const uint32_t jk = (uint32_t)(s0 + jj);
#pragma unroll
            for (int k = 0; k < RQ; k++) {
                const uint32_t key = (hamming_words<WORDS>(q[k], t) << KEY_IDX_BITS) + jk;
                second[k] = min(second[k], max(best[k], key));
                best[k] = min(best[k], key);
            }
        }
    }
#pragma unroll
    for (int k = 0; k < RQ; k++) {
        const int i = rt * tile_rows + k * ROUND_THREADS + tid;
        if (i < n1) {
            part[((size_t)sp * n1 + i) * 2 + 0] = best[k];
            part[((size_t)sp * n1 + i) * 2 + 1] = second[k];
        }
    }
}

__global__ void knn2_merge_kernel(const uint32_t *__restrict__ part, int n1, int splits,
                                  int32_t *best_j, int32_t *best_d, int32_t *second_j, int32_t *second_d) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n1) return;
    uint32_t b = KEY_NONE, s = KEY_NONE;
    for (int sp = 0; sp < splits; sp++) {
        const uint32_t pb = part[((size_t)sp * n1 + i) * 2 + 0], ps = part[((size_t)sp * n1 + i) * 2 + 1];
        s = min(min(s, ps), max(b, pb));
        b = min(b, pb);
    }
    best_j[i] = b == KEY_NONE ? -1 : (int32_t)(b & KEY_IDX_MASK);
    best_d[i] = b == KEY_NONE ? -1 : (int32_t)(b >> KEY_IDX_BITS);
    second_j[i] = s == KEY_NONE ? -1 : (int32_t)(s & KEY_IDX_MASK);
    second_d[i] = s == KEY_NONE ? -1 : (int32_t)(s >> KEY_IDX_BITS);
}

// per-train best query under (d, i): the cross-check side.  Same kernel with
// the roles swapped gives best only; reuse knn2 by calling it with (t, q).

// ---------------------------------------------------------------------------
// Python generation's match_keypoints (python_src/photogrammetry/image_processing/
// keypoint_matching.py:7-33): for every keypoint of image 1 ALL keypoints of image 2
// ranked by distance, as int64 (idx2, dist) pairs.  One CTA per query row: a stable
// counting sort over the <= 513 possible distances (per-warp histograms over
// contiguous column segments, MATCH.ANY ranks) -- the (dist, idx2) order, which is one
// of the orders numpy's unstable argsort may return upstream.  Write-bound: 16 B/cell.
// ---------------------------------------------------------------------------
constexpr int TWIN_THREADS = 256;
constexpr int TWIN_WARPS = TWIN_THREADS / 32;

template <int WORDS>
__global__ void __launch_bounds__(TWIN_THREADS) sorted_rows_kernel(const uint32_t *__restrict__ qd, int n1,
                                                                  const uint32_t *__restrict__ td, int n2,
                                                                  int nbins, long long *__restrict__ out) {
    extern __shared__ int32_t s_twin[];          // [TWIN_WARPS][nbins + 1]
    __shared__ int32_t s_wsum[TWIN_WARPS];
    const int i = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int hb = nbins + 1;
    uint32_t q[WORDS];
#pragma unroll
    for (int v = 0; v < WORDS / 4; v++) {
        const uint4 a = __ldg(reinterpret_cast<const uint4 *>(qd + (size_t)i * WORDS) + v);
        q[4 * v] = a.x; q[4 * v + 1] = a.y; q[4 * v + 2] = a.z; q[4 * v + 3] = a.w;
    }
    for (int k = tid; k < TWIN_WARPS * hb; k += TWIN_THREADS) s_twin[k] = 0;
    int seg = (n2 + TWIN_WARPS - 1) / TWIN_WARPS;
    seg = (seg + 31) & ~31;
    const int y0 = min(n2, wid * seg), y1 = min(n2, y0 + seg);
    __syncthreads();
    auto dist_of = [&](int j) -> int {
        uint32_t t[WORDS];
#pragma unroll
        for (int v = 0; v < WORDS / 4; v++) {
            const uint4 a = __ldg(reinterpret_cast<const uint4 *>(td + (size_t)j * WORDS) + v);
            t[4 * v] = a.x; t[4 * v + 1] = a.y; t[4 * v + 2] = a.z; t[4 * v + 3] = a.w;
        }
        return (int)hamming_words<WORDS>(q, t);
    };
    for (int j = y0 + lane; j < y1; j += 32) atomicAdd(&s_twin[wid * hb + dist_of(j)], 1);
    __syncthreads();
    // thread t owns bins 4t..4t+3 (nbins <= 513 <= 4 * 256): exclusive scan over distances, then per-warp bases
    int tot[4] = {0, 0, 0, 0};
#pragma unroll
    for (int u = 0; u < 4; u++) {
        const int b = 4 * tid + u;
        if (b < nbins) for (int w = 0; w < TWIN_WARPS; w++) tot[u] += s_twin[w * hb + b];
    }
    const int mine = tot[0] + tot[1] + tot[2] + tot[3];
    int inc = mine;
    for (int o = 1; o < 32; o <<= 1) { const int a = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += a; }
    if (lane == 31) s_wsum[wid] = inc;
    __syncthreads();
    int a = inc - mine;
    for (int w = 0; w < wid; w++) a += s_wsum[w];
#pragma unroll
    for (int u = 0; u < 4; u++) {
        const int b = 4 * tid + u;
        if (b < nbins) for (int w = 0; w < TWIN_WARPS; w++) { const int t = s_twin[w * hb + b]; s_twin[w * hb + b] = a; a += t; }
    }
    __syncthreads();
    long long *row = out + (size_t)i * n2 * 2;
    for (int jb = y0; jb < y1; jb += 32) {
        const int j = jb + lane;
        const int d = j < y1 ? dist_of(j) : nbins;
        const unsigned peers = __match_any_sync(0xffffffffu, d);
        const int rank = __popc(peers & ((1u << lane) - 1u));
        const int base = s_twin[wid * hb + d];
        __syncwarp();
        if (rank == 0) s_twin[wid * hb + d] = base + __popc(peers);
        __syncwarp();
        if (j < y1) {
            const size_t o = (size_t)(base + rank) * 2;
            row[o] = j; row[o + 1] = d;            // key1_to_key2_dist[idx1, rank] = [idx2, dist]
        }
    }
}

// ratio + cross-check filter over knn2 results, compacted in ascending i.
__global__ void ratio_crosscheck_kernel(int n1, int n2, const int32_t *best_j, const int32_t *best_d,
                                        const int32_t *second_d, const int32_t *col_best_i,
                                        float ratio, int cross_check, int max_dist, uint8_t *keep) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n1) return;
    bool k = best_j[i] >= 0;
    if (k && ratio > 0.0f && n2 >= 2 && !((float)best_d[i] < ratio * (float)second_d[i])) k = false;
    if (k && cross_check && col_best_i[best_j[i]] != i) k = false;
    if (k && max_dist >= 0 && best_d[i] > max_dist) k = false;
    keep[i] = k ? 1 : 0;
}

// ---------------------------------------------------------------------------
// Many small pairs at once (a frame sequence, BASELINE configs[2]): nearest / second nearest of every query, best query
// of every train descriptor, ratio test, cross-check and max-distance filter, ordered compaction -- one CTA per pair,
// both descriptor sets in shared memory (read as broadcasts), a thread's own descriptor in registers.  Same keys,
// same tie-break and the same filter expression as knn2_kernel + ratio_crosscheck_kernel.
// ---------------------------------------------------------------------------
constexpr int RCB_THREADS = 512;
struct RcbPair { const uint32_t *q, *t; int32_t n1, n2; int64_t out_base; };

template <int WORDS>
__global__ void __launch_bounds__(RCB_THREADS) ratio_crosscheck_batch_kernel(const RcbPair *__restrict__ pairs, float ratio,
                                                                             int cross_check, int max_dist,
                                                                             int32_t *__restrict__ out_qi, int32_t *__restrict__ out_tj,
                                                                             int32_t *__restrict__ out_dist, int32_t *__restrict__ counts) {
    extern __shared__ __align__(16) unsigned char dyn_smem[];
    constexpr int V4 = WORDS / 4;
    __shared__ int s_w[RCB_THREADS / 32], s_base;
    const RcbPair pr = pairs[blockIdx.x];
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, n1 = pr.n1, n2 = pr.n2;
    uint4 *sq = reinterpret_cast<uint4 *>(dyn_smem), *st = sq + (size_t)n1 * V4;
    uint32_t *colbest = reinterpret_cast<uint32_t *>(st + (size_t)n2 * V4);          // [n2] (d << 20 | i)
    for (int k = tid; k < n1 * V4; k += RCB_THREADS) sq[k] = __ldg(reinterpret_cast<const uint4 *>(pr.q) + k);
    for (int k = tid; k < n2 * V4; k += RCB_THREADS) st[k] = __ldg(reinterpret_cast<const uint4 *>(pr.t) + k);
    if (tid == 0) s_base = 0;
    __syncthreads();
    auto load = [&](const uint4 *base, int idx, uint32_t (&x)[WORDS]) {
#pragma unroll
        for (int v = 0; v < V4; v++) { const uint4 a = base[idx * V4 + v]; x[4 * v] = a.x; x[4 * v + 1] = a.y; x[4 * v + 2] = a.z; x[4 * v + 3] = a.w; }
    };
    if (cross_check) {
        for (int j = tid; j < n2; j += RCB_THREADS) {
            uint32_t mine[WORDS], other[WORDS], best = KEY_NONE;
            load(st, j, mine);
            for (int i = 0; i < n1; i++) { load(sq, i, other); best = min(best, (hamming_words<WORDS>(mine, other) << KEY_IDX_BITS) + (uint32_t)i); }
            colbest[j] = best;
        }
    }
    __syncthreads();
    for (int i0 = 0; i0 < n1; i0 += RCB_THREADS) {
        const int i = i0 + tid;
        bool keep = false;
        uint32_t best = KEY_NONE, second = KEY_NONE;
        if (i < n1) {
            uint32_t mine[WORDS], other[WORDS];
            load(sq, i, mine);
            for (int j = 0; j < n2; j++) {
                load(st, j, other);
                const uint32_t key = (hamming_words<WORDS>(mine, other) << KEY_IDX_BITS) + (uint32_t)j;
                second = min(second, max(best, key));
                best = min(best, key);
            }
            const int bj = (int)(best & KEY_IDX_MASK), bd = (int)(best >> KEY_IDX_BITS), sd = second == KEY_NONE ? -1 : (int)(second >> KEY_IDX_BITS);
            keep = n2 > 0;
            if (keep && ratio > 0.0f && n2 >= 2 && !((float)bd < ratio * (float)sd)) keep = false;
            if (keep && cross_check && (int)(colbest[bj] & KEY_IDX_MASK) != i) keep = false;
            if (keep && max_dist >= 0 && bd > max_dist) keep = false;
        }
        const unsigned m = __ballot_sync(0xffffffffu, keep);
        if (lane == 0) s_w[wid] = __popc(m);
        __syncthreads();
        int off = s_base;
        for (int w = 0; w < wid; w++) off += s_w[w];
        if (keep) {
            const int64_t o = pr.out_base + off + __popc(m & ((1u << lane) - 1u));
            out_qi[o] = i; out_tj[o] = (int32_t)(best & KEY_IDX_MASK); out_dist[o] = (int32_t)(best >> KEY_IDX_BITS);
        }
        __syncthreads();
        if (tid == 0) { int t = 0; for (int w = 0; w < RCB_THREADS / 32; w++) t += s_w[w]; s_base += t; }
        __syncthreads();
    }
    if (tid == 0) counts[blockIdx.x] = s_base;
}

// ---------------------------------------------------------------------------
// Many pairs of any size (BASELINE configs[4]): nearest / second nearest, best query of every train descriptor, ratio
// test, cross-check and max-distance filter.  Three launches per chunk of pairs:
//   knn2_cols_pairs_kernel    one fused distance pass over flattened (pair, row tile, column split) items: the round
//                             kernel's inner loop with top-2 row keys (d << 20 | j) in registers and, with CROSS, the
//                             column minimum (d << 20 | i) through shared and global atomicMin -- the second distance
//                             pass of pgm_match_ratio_crosscheck is not needed
//   rcp_filter_kernel         merges a row's split partials as knn2_merge_kernel does, applies the filter expression of
//                             ratio_crosscheck_kernel and counts the kept rows of each block of RCF_THREADS rows
//   rcp_scatter_kernel        prefix of the block counts of the block's pair, ordered write of the kept triples
// A large pair's ordered compaction is spread over ceil(n1 / RCF_THREADS) CTAs rather than walked by one.
// ---------------------------------------------------------------------------
struct RcpPair {
    const uint32_t *q, *t;
    int32_t n1, n2;
    int64_t out_base;      // first slot of this pair's triples in the caller's output arrays
    int64_t part_base;     // row i, split s: partial (best, second) at part[part_base + i * splits + s]
    int64_t col_base;      // this pair's column minima in the chunk's colbest
    int64_t row_base;      // this pair's rows in the chunk's per-row filter results
    int32_t splits, cols_per_split;
    int32_t pair_id;       // index in the caller's pair list (out_counts)
    int32_t pad;
};
constexpr int RCF_THREADS = 1024;   // rows per filter / scatter block (n1 < 2^20: at most 1024 blocks per pair)

template <int WORDS, bool CROSS>
__global__ void __launch_bounds__(ROUND_THREADS, WORDS <= 8 ? 6 : (WORDS == 12 ? 5 : 4))
knn2_cols_pairs_kernel(const RcpPair *__restrict__ pairs, const int32_t *__restrict__ tile_base, int n_pairs,
                       uint2 *__restrict__ part, int64_t part_cap, uint32_t *__restrict__ colbest, int64_t col_cap) {
    constexpr int V4 = WORDS / 4, RQ = RQ_LARGE, STAGE = STAGE_LARGE, tile_rows = ROUND_THREADS * RQ;
    __shared__ uint4 s_t[STAGE * V4];
    __shared__ uint32_t s_jkey[STAGE];
    __shared__ uint32_t s_col[CROSS ? STAGE : 1];
    const int tid = threadIdx.x, g = blockIdx.x;
    const int p = find_pair(tile_base, n_pairs, g);
    const RcpPair pr = pairs[p];
    const int local = g - __ldg(tile_base + p);
    const int rt = local / pr.splits, sp = local - rt * pr.splits;

    uint32_t q[RQ][WORDS], ikey[RQ], best[RQ], second[RQ];
#pragma unroll
    for (int k = 0; k < RQ; k++) {
        const int i = rt * tile_rows + k * ROUND_THREADS + tid;
        best[k] = KEY_NONE; second[k] = KEY_NONE;
        if (i < pr.n1) {
            ikey[k] = (uint32_t)i;
            const uint4 *src = reinterpret_cast<const uint4 *>(pr.q + (size_t)i * WORDS);
#pragma unroll
            for (int v = 0; v < V4; v++) {
                const uint4 x = __ldg(src + v);
                q[k][4 * v + 0] = x.x; q[k][4 * v + 1] = x.y; q[k][4 * v + 2] = x.z; q[k][4 * v + 3] = x.w;
            }
        } else {
            ikey[k] = KEY_INVALID;             // a padded row never wins a column
#pragma unroll
            for (int w = 0; w < WORDS; w++) q[k][w] = 0u;
        }
    }

    const int c0 = sp * pr.cols_per_split, c1 = min(pr.n2, c0 + pr.cols_per_split);
    for (int s0 = c0; s0 < c1; s0 += STAGE) {
        __syncthreads();                       // previous stage fully consumed
        for (int k = tid; k < STAGE * V4; k += ROUND_THREADS) {
            const int col = k / V4, part_i = k - col * V4, j = s0 + col;
            uint4 x = make_uint4(0u, 0u, 0u, 0u);
            uint32_t jk = KEY_INVALID;         // a padded column's keys exceed every real key: it never becomes a best
            if (j < c1) {
                x = __ldg(reinterpret_cast<const uint4 *>(pr.t + (size_t)j * WORDS) + part_i);
                jk = (uint32_t)j;
            }
            s_t[k] = x;
            if (part_i == 0) s_jkey[col] = jk;
        }
        if (CROSS && tid < STAGE) s_col[tid] = KEY_NONE;
        __syncthreads();

        const int ncs = min(STAGE, (c1 - s0 + 3) & ~3);
        // as in round_tiles: no store, atomic or branch between the columns of a 4-column block
        for (int jj0 = 0; jj0 < ncs; jj0 += 4) {
            uint32_t cm[4];
#pragma unroll
            for (int u = 0; u < 4; u++) {
                const int jj = jj0 + u;
                uint32_t t[WORDS];
#pragma unroll
                for (int v = 0; v < V4; v++) {
                    const uint4 x = s_t[jj * V4 + v];
                    t[4 * v + 0] = x.x; t[4 * v + 1] = x.y; t[4 * v + 2] = x.z; t[4 * v + 3] = x.w;
                }
                const uint32_t jk = s_jkey[jj];
                uint32_t cmin = KEY_NONE;
#pragma unroll
                for (int k = 0; k < RQ; k++) {
                    // (rows alternate between the 5-POPC and the 4-POPC popcount so that the XU and ALU pipes balance)
                    const uint32_t d = ((k & 1) ? hamming_words_deep<WORDS>(q[k], t) : hamming_words<WORDS>(q[k], t)) << KEY_IDX_BITS;
                    const uint32_t key = d + jk;
                    second[k] = min(second[k], max(best[k], key));
                    best[k] = min(best[k], key);
                    if (CROSS) cmin = min(cmin, d + ikey[k]);
                }
                cm[u] = cmin;
            }
            if (CROSS) {
                // one warp-aggregated shared atomicMin per (warp, column)
#pragma unroll
                for (int u = 0; u < 4; u++) atomicMin(&s_col[jj0 + u], cm[u]);
            }
        }
        if (CROSS) {
            __syncthreads();
            if (tid < STAGE) {
                const uint32_t jk = s_jkey[tid], v = s_col[tid];
                if (jk != KEY_INVALID && v < KEY_INVALID) {
                    PGM_ASSERT((int)jk < pr.n2 && pr.col_base + (int64_t)jk < col_cap);
                    atomicMin(colbest + pr.col_base + jk, v);
                }
            }
        }
    }
#pragma unroll
    for (int k = 0; k < RQ; k++) {
        const int i = rt * tile_rows + k * ROUND_THREADS + tid;
        if (i < pr.n1) {
            const int64_t slot = pr.part_base + (int64_t)i * pr.splits + sp;
            PGM_ASSERT(slot >= 0 && slot < part_cap);
            part[slot] = make_uint2(best[k], second[k]);
        }
    }
}

// res[row] = the row's best key if it passes the filter, else KEY_NONE; bcnt[block] = kept rows of the block
__global__ void __launch_bounds__(RCF_THREADS) rcp_filter_kernel(const RcpPair *__restrict__ pairs,
                                                                 const int32_t *__restrict__ fblk_base, int n_pairs,
                                                                 const uint2 *__restrict__ part, int64_t part_cap,
                                                                 const uint32_t *__restrict__ colbest, int64_t col_cap,
                                                                 float ratio, int cross_check, int max_dist,
                                                                 uint32_t *__restrict__ res, int32_t *__restrict__ bcnt) {
    const int g = blockIdx.x, tid = threadIdx.x;
    const int p = find_pair(fblk_base, n_pairs, g);
    const RcpPair pr = pairs[p];
    const int i = (g - __ldg(fblk_base + p)) * RCF_THREADS + tid;
    bool keep = false;
    if (i < pr.n1) {
        uint32_t b = KEY_NONE, s = KEY_NONE;
        for (int sp = 0; sp < pr.splits; sp++) {
            const int64_t slot = pr.part_base + (int64_t)i * pr.splits + sp;
            PGM_ASSERT(slot >= 0 && slot < part_cap);
            const uint2 x = part[slot];
            s = min(min(s, x.y), max(b, x.x));
            b = min(b, x.x);
        }
        const int bj = (int)(b & KEY_IDX_MASK), bd = (int)(b >> KEY_IDX_BITS), sd = (int)(s >> KEY_IDX_BITS);
        PGM_ASSERT(b < KEY_INVALID && bj < pr.n2);
        // the expression of ratio_crosscheck_kernel (n2 >= 1 here: a pair without train rows is never launched)
        keep = true;
        if (keep && ratio > 0.0f && pr.n2 >= 2 && !((float)bd < ratio * (float)sd)) keep = false;
        if (keep && cross_check) {
            PGM_ASSERT(pr.col_base + bj < col_cap);
            if ((int)(colbest[pr.col_base + bj] & KEY_IDX_MASK) != i) keep = false;
        }
        if (keep && max_dist >= 0 && bd > max_dist) keep = false;
        res[pr.row_base + i] = keep ? b : KEY_NONE;
    }
    const int n = __syncthreads_count(keep);
    if (tid == 0) bcnt[g] = n;
}

// kept triples of one block, in ascending i, at the pair's output offset + the kept rows of the pair's earlier blocks
__global__ void __launch_bounds__(RCF_THREADS) rcp_scatter_kernel(const RcpPair *__restrict__ pairs,
                                                                  const int32_t *__restrict__ fblk_base, int n_pairs,
                                                                  const uint32_t *__restrict__ res,
                                                                  const int32_t *__restrict__ bcnt, int64_t capacity,
                                                                  int32_t *__restrict__ out_qi, int32_t *__restrict__ out_tj,
                                                                  int32_t *__restrict__ out_dist, int32_t *__restrict__ counts) {
    __shared__ int s_before[RCF_THREADS / 32], s_total[RCF_THREADS / 32], s_w[RCF_THREADS / 32];
    const int g = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int p = find_pair(fblk_base, n_pairs, g);
    const RcpPair pr = pairs[p];
    const int first = __ldg(fblk_base + p), nb = __ldg(fblk_base + p + 1) - first, b = g - first;
    // kept rows of the pair's blocks before this one, and of all of them (nb <= RCF_THREADS)
    const int c = tid < nb ? __ldg(bcnt + first + tid) : 0;
    int before = tid < b ? c : 0, total = c;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        before += __shfl_xor_sync(0xffffffffu, before, o);
        total += __shfl_xor_sync(0xffffffffu, total, o);
    }
    const int i = b * RCF_THREADS + tid;
    const uint32_t key = i < pr.n1 ? __ldg(res + pr.row_base + i) : KEY_NONE;
    const bool keep = key != KEY_NONE;
    const unsigned m = __ballot_sync(0xffffffffu, keep);
    if (lane == 0) { s_before[wid] = before; s_total[wid] = total; s_w[wid] = __popc(m); }
    __syncthreads();
    int off = 0;
    before = 0; total = 0;
#pragma unroll 4
    for (int w = 0; w < RCF_THREADS / 32; w++) {
        before += s_before[w]; total += s_total[w];
        if (w < wid) off += s_w[w];
    }
    if (keep) {
        const int64_t o = pr.out_base + before + off + __popc(m & ((1u << lane) - 1u));
        PGM_ASSERT(o >= pr.out_base && o < pr.out_base + pr.n1 && o < capacity);
        out_qi[o] = i; out_tj[o] = (int32_t)(key & KEY_IDX_MASK); out_dist[o] = (int32_t)(key >> KEY_IDX_BITS);
    }
    if (b == nb - 1 && tid == 0) counts[pr.pair_id] = total;
}

// ---------------------------------------------------------------------------
// train-sharded nearest / second-nearest neighbour (SURVEY.md section 8e, "top-2 merge"):
// every rank searches its slice of the train set, the (best, second) pairs travel as packed keys
// (distance << 20 | GLOBAL train index, XKEY_NONE where absent -- integer order == the (distance, j)
// order) through one all-gather, and every rank picks the two smallest of the 2G keys of each query.
// ---------------------------------------------------------------------------
__global__ void pack_top2_kernel(const int32_t *__restrict__ bj, const int32_t *__restrict__ bd,
                                 const int32_t *__restrict__ sj, const int32_t *__restrict__ sd, int n, int offset,
                                 uint32_t *__restrict__ keys) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    keys[i] = bj[i] >= 0 ? ((uint32_t)bd[i] << KEY_IDX_BITS) | (uint32_t)(bj[i] + offset) : XKEY_NONE;
    keys[(size_t)n + i] = sj[i] >= 0 ? ((uint32_t)sd[i] << KEY_IDX_BITS) | (uint32_t)(sj[i] + offset) : XKEY_NONE;
}

__global__ void merge_top2_kernel(const uint32_t *__restrict__ keys, int n_shards, int n, int32_t *__restrict__ bj,
                                  int32_t *__restrict__ bd, int32_t *__restrict__ sj, int32_t *__restrict__ sd) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t k1 = XKEY_NONE, k2 = XKEY_NONE;                  // the two smallest keys (train slices are disjoint: no duplicates)
    for (int g = 0; g < 2 * n_shards; g++) {
        const uint32_t k = keys[(size_t)g * n + i];
        k2 = min(k2, max(k1, k));
        k1 = min(k1, k);
    }
    bj[i] = k1 != XKEY_NONE ? (int32_t)(k1 & KEY_IDX_MASK) : -1;
    bd[i] = k1 != XKEY_NONE ? (int32_t)(k1 >> KEY_IDX_BITS) : -1;
    sj[i] = k2 != XKEY_NONE ? (int32_t)(k2 & KEY_IDX_MASK) : -1;
    sd[i] = k2 != XKEY_NONE ? (int32_t)(k2 >> KEY_IDX_BITS) : -1;
}

// kept rows (ascending i) -> (i, best_j, best_d) triples; single block, ordered compaction
__global__ void __launch_bounds__(1024) compact_matches_kernel(const uint8_t *__restrict__ keep, const int32_t *__restrict__ best_j,
                                                               const int32_t *__restrict__ best_d, int n1,
                                                               int32_t *__restrict__ qi, int32_t *__restrict__ tj,
                                                               int32_t *__restrict__ dist, int32_t *__restrict__ count) {
    __shared__ int s_w[32];
    __shared__ int s_base;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    if (tid == 0) s_base = 0;
    __syncthreads();
    for (int i0 = 0; i0 < n1; i0 += 1024) {
        const int i = i0 + tid;
        const bool hit = i < n1 && keep[i];
        const unsigned m = __ballot_sync(0xffffffffu, hit);
        if (lane == 0) s_w[wid] = __popc(m);
        __syncthreads();
        int off = s_base;
        for (int k = 0; k < wid; k++) off += s_w[k];
        if (hit) {
            const int o = off + __popc(m & ((1u << lane) - 1u));
            qi[o] = i; tj[o] = best_j[i]; dist[o] = best_d[i];
        }
        __syncthreads();
        if (tid == 0) { int t = 0; for (int k = 0; k < 32; k++) t += s_w[k]; s_base += t; }
        __syncthreads();
    }
    if (tid == 0) *count = s_base;
}

// ---------------------------------------------------------------------------
// integer-pipe micro-benchmarks (roofline denominators, SURVEY.md section 8d)
// ---------------------------------------------------------------------------
__global__ void popc_peak_kernel(uint32_t *out, int iters, uint32_t seed) {
    uint32_t a[8], acc[8];
#pragma unroll
    for (int k = 0; k < 8; k++) { a[k] = seed * (threadIdx.x + 1) + k * 0x9E3779B9u; acc[k] = 0; }
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int u = 0; u < 4; u++) {
#pragma unroll
            for (int k = 0; k < 8; k++) acc[k] = __popc(acc[k] ^ a[k]);   // dependent chain per k, 8 chains
        }
    }
    uint32_t s = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) s += acc[k];
    out[blockIdx.x * blockDim.x + threadIdx.x] = s;   // keeps the chains alive
}

__global__ void lop3_peak_kernel(uint32_t *out, int iters, uint32_t seed) {
    uint32_t a[8], acc[8];
#pragma unroll
    for (int k = 0; k < 8; k++) { a[k] = seed * (threadIdx.x + 1) + k * 0x9E3779B9u; acc[k] = k; }
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int u = 0; u < 4; u++) {
#pragma unroll
            for (int k = 0; k < 8; k++) acc[k] = (acc[k] & a[(k + u) & 7]) ^ acc[(k + 1 + u) & 7];   // one LOP3 each
        }
    }
    uint32_t s = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) s += acc[k];
    out[blockIdx.x * blockDim.x + threadIdx.x] = s;   // keeps the chains alive
}

}  // namespace pgm
