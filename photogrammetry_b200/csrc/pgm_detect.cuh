// pgm_detect.cuh -- the producer of the matcher's inputs on the GPU (SURVEY.md section 8, rows f1/f2):
//
//   FAST-12 corner test      dotnet_src/ImageProcessing/KeypointDetection.cs:42-138
//   BRIEF descriptor         dotnet_src/ImageProcessing.Abstractions/Keypoint.cs:29-57
//   non-maximum suppression  dotnet_src/ImageProcessing/RedundantKeypointEliminator.cs:16-39
//
// Images are float32 [H][W] arrays of Grayscale.K (Grayscale.cs:19-23), pixel (x, y) at img[y*W + x].
// All three stages reproduce the reference bit for bit, quirks included (the ring table's last entry
// repeats {-3, 1}; a fifth in-threshold ring pixel rejects the candidate; out-of-image BRIEF pairs give
// a 0 bit; NMS drops distance <= radius).  These kernels are HBM/latency-bound byte work: coalesced
// loads, no tensor cores.
#pragma once

#include <cstdint>
#include <cuda_runtime.h>

#include "pgm_kernels.cuh"   // PGM_ASSERT, grid_barrier

namespace pgm_det {

// Ring tables as (dx, dy).  [0] = KeypointDetection.cs:15-19; entry 15 is upstream's typo ({-3, 1} twice), kept.
// [1] = the Python generation's BRESENHAM_CIRCLE_3 (python_src/.../keypoint_detection.py:12-29), whose entries
// are (height_offset, width_offset) = (dy, dx) and whose entry 15 is the correct {-3, -1}.
__constant__ int c_ring[2][16][2] = {
    {{-3, 0}, {-3, 1}, {-2, 2}, {-1, 3}, {0, 3}, {1, 3}, {2, 2}, {3, 1},
     {3, 0}, {3, -1}, {2, -2}, {1, -3}, {0, -3}, {-1, -3}, {-2, -2}, {-3, 1}},
    {{0, -3}, {1, -3}, {2, -2}, {3, -1}, {3, 0}, {3, 1}, {2, 2}, {1, 3},
     {0, 3}, {-1, 3}, {-2, 2}, {-3, 1}, {-3, 0}, {-3, -1}, {-2, -2}, {-1, -3}}};

// ---- batch geometry ------------------------------------------------------------------------------------------------
// Image k of a batch, as the batch kernels see it.  Every image owns a run of each flat index space, at a prefix of
// the sizes of the images before it; the table has n_images + 1 entries, the last holding the totals.  Work items are
// flat over all images (FAST tiles, rows) unless every image has one size (see fast_score_kernel).
constexpr int FAST_TILE_W = 32, FAST_TILE_H = 8;   // fast_score_kernel's block
struct ImageGeom {
    long long px;     // first pixel in the caller's image buffer
    long long sc;     // first byte of the score map (sum of w * h)
    long long row;    // first of h + 1 row slots: row counts, row offsets (slot h = the image's total), row work items
    long long tile;   // first FAST tile (FAST_TILE_W x FAST_TILE_H pixels)
    long long cell;   // first NMS cell id (cells of side max(radius, 1) over [0, w) x [0, h)); 0 without NMS
    int w, h;
    int ncx, ncy;     // NMS cells per row / column; 0 without NMS
};

// The flat kernels run a resident grid (FLAT_CTAS_PER_SM_* CTAs per SM) in which every CTA (or warp) takes one
// contiguous, balanced range of the work items: the image lookup, a dependent chain of table loads, is paid once per
// range.  Paid once per short-lived CTA it adds its latency to every FAST tile and row (about 10 % on 4000 x 3000 frames).
constexpr int FLAT_CTAS_PER_SM_256 = 8, FLAT_CTAS_PER_SM_128 = 16;   // full occupancy at <= 32 registers

// [*b, *e): the items of work unit u out of n_units
__device__ __forceinline__ void unit_range(long long n_items, long long u, long long n_units, long long *b, long long *e) {
    const long long per = (n_items + n_units - 1) / n_units;
    *b = min(u * per, n_items); *e = min(*b + per, n_items);
}

// image owning flat item t of the index space F (the last k with geo[k].*F <= t; every image owns at least one item)
template <long long ImageGeom::*F>
__device__ __forceinline__ int image_of(const ImageGeom *__restrict__ geo, int n_images, long long t) {
    int lo = 0, hi = n_images - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (geo[mid].*F <= t) lo = mid; else hi = mid - 1;
    }
    return lo;
}

// score of pixel (x, y): 0 = no keypoint, else the longest circular run (12..16) = Keypoint.FastScore
template <int RING>
__device__ __forceinline__ uint8_t fast_score_at(const float *__restrict__ img, int w, int h, int x, int y,
                                                 float threshold) {
    uint8_t out = 0;
    if (x >= 3 && x < w - 3 && y >= 3 && y < h - 3) {                 // Detect's loop bounds, :45-47
        const float *p = img + (size_t)y * w + x;
        const float c = __ldg(p);
        const float lo = c - threshold, hi = c + threshold;            // InThreshold, :135-138
        unsigned inside = 0;                                           // bit k: ring pixel k is inside the threshold
        // IsPotentialKeypoint (:116-133): the compass points are ring entries 0, 4, 8, 12; at most one may be
        // inside.  Most pixels of a natural image fail here and never touch the other twelve taps.
#pragma unroll
        for (int k = 0; k < 16; k += 4) {
            const float t = __ldg(p + c_ring[RING][k][1] * w + c_ring[RING][k][0]);
            inside |= (unsigned)(t > lo && t < hi) << k;
        }
        if (__popc(inside) <= 1) {
#pragma unroll
            for (int k = 0; k < 16; k++) {
                if ((k & 3) == 0) continue;
                const float t = __ldg(p + c_ring[RING][k][1] * w + c_ring[RING][k][0]);
                inside |= (unsigned)(t > lo && t < hi) << k;
            }
            // GetIntensityValueIfKeypoint (:65-114): longest circular run of ring pixels OUTSIDE the threshold,
            // accepted from 12 up.  (Its early exit on a fifth inside pixel cannot change the outcome: five
            // inside pixels leave at most eleven outside.)  On the doubled ring a circular run is a linear run;
            // bit i of `r` survives the shifts iff bits i .. i+11 are all set.
            const unsigned o16 = ~inside & 0xFFFFu;
            if (o16 == 0xFFFFu) out = 16;
            else {
                unsigned r = o16 | (o16 << 16);
                r &= r >> 1; r &= r >> 2; r &= r >> 4; r &= r >> 4;
                if (r) {
                    int len = 12;
                    while ((r &= r >> 1) != 0u) len++;
                    out = (uint8_t)len;
                }
            }
        }
    }
    return out;
}

// score map of one image, block (FAST_TILE_W, FAST_TILE_H)
template <int RING>
__global__ void fast_score_kernel(const float *__restrict__ img, int w, int h, float threshold,
                                  uint8_t *__restrict__ score) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= w || y >= h) return;
    score[(size_t)y * w + x] = fast_score_at<RING>(img, w, h, x, y, threshold);
}

// batched form, image k's map at score + geo[k].sc.  A set of one size uw x uh packed back to back (uw > 0) runs on the
// grid (tiles x, tiles y, images) and reads no table: these CTAs are short and latency-bound, and a table read before
// the pixel loads would add its latency to each.  Any other set: one contiguous range of the flat FAST tile space
// (geo[].tile) per CTA.
template <int RING>
__global__ void __launch_bounds__(FAST_TILE_W * FAST_TILE_H, FLAT_CTAS_PER_SM_256) fast_score_kernel(
        const float *__restrict__ img, const ImageGeom *__restrict__ geo, int n_images, int uw, int uh,
        float threshold, uint8_t *__restrict__ score) {
    if (uw) {
        const int x = blockIdx.x * FAST_TILE_W + threadIdx.x, y = blockIdx.y * FAST_TILE_H + threadIdx.y;
        if (x >= uw || y >= uh) return;
        const long long off = (long long)blockIdx.z * uw * uh;
        score[off + (long long)y * uw + x] = fast_score_at<RING>(img + off, uw, uh, x, y, threshold);
        return;
    }
    long long t0, t1;
    unit_range(geo[n_images].tile, blockIdx.x, gridDim.x, &t0, &t1);
    if (t0 >= t1) return;
    // the image's pointers and sizes and the tile's coordinates stay in registers while the range is inside the image
    int z = image_of<&ImageGeom::tile>(geo, n_images, t0), w = 0, h = 0, ntx = 1, left = 0;
    const float *im = nullptr;
    uint8_t *sm = nullptr;
    auto enter = [&]() {
        im = img + geo[z].px; sm = score + geo[z].sc; w = geo[z].w; h = geo[z].h;
        ntx = (w + FAST_TILE_W - 1) / FAST_TILE_W; left = (int)(geo[z + 1].tile - geo[z].tile);   // < 2^24 tiles
    };
    enter();
    const int lt = (int)(t0 - geo[z].tile);
    int ty = lt / ntx, tx = lt - ty * ntx;
    left -= lt;
    for (int n = (int)(t1 - t0); n > 0; n--) {                           // per <= 2^31 tiles
        if (left == 0) { z++; enter(); tx = ty = 0; }                      // every image owns a tile: none is skipped
        PGM_ASSERT(z < n_images && left > 0);
        const int x = tx * FAST_TILE_W + threadIdx.x, y = ty * FAST_TILE_H + threadIdx.y;
        if (x < w && y < h) sm[(long long)y * w + x] = fast_score_at<RING>(im, w, h, x, y, threshold);
        if (++tx == ntx) { tx = 0; ty++; }
        left--;
    }
}

// keypoints in one row of a score map, summed over the block (every thread gets the sum; safe to call in a loop)
__device__ __forceinline__ int row_count_block(const uint8_t *__restrict__ row, int w) {
    __shared__ int s;
    int c = 0;
    for (int x = threadIdx.x; x < w; x += blockDim.x) c += row[x] != 0;
    c = __reduce_add_sync(0xffffffffu, c);
    if (threadIdx.x == 0) s = 0;
    __syncthreads();
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(&s, c);
    __syncthreads();
    const int total = s;
    __syncthreads();
    return total;
}

// per-row keypoint counts (one block per row)
__global__ void row_count_kernel(const uint8_t *__restrict__ score, int w, int32_t *__restrict__ rowcnt) {
    const int y = blockIdx.x;
    const int c = row_count_block(score + (size_t)y * w, w);
    if (threadIdx.x == 0) rowcnt[y] = c;
}

// batched form; rowcnt has the row slots' layout.  One size uw x uh (uw > 0): grid (rows, images), no table read.  Any
// other set: one contiguous range of the flat row-slot space (geo[].row) per block.
__global__ void __launch_bounds__(128, FLAT_CTAS_PER_SM_128) row_count_kernel(
        const uint8_t *__restrict__ score, const ImageGeom *__restrict__ geo, int n_images, int uw, int uh,
        int32_t *__restrict__ rowcnt) {
    if (uw) {
        const int y = blockIdx.x, z = blockIdx.y;
        const int c = row_count_block(score + ((long long)z * uh + y) * uw, uw);
        if (threadIdx.x == 0) rowcnt[(long long)z * (uh + 1) + y] = c;
        return;
    }
    long long g0, g1;
    unit_range(geo[n_images].row, blockIdx.x, gridDim.x, &g0, &g1);
    if (g0 >= g1) return;
    int z = image_of<&ImageGeom::row>(geo, n_images, g0);
    long long row0 = geo[z].row;
    int w = geo[z].w, h = geo[z].h;
    for (long long g = g0; g < g1; g++) {
        if (g > row0 + h) { z++; row0 = geo[z].row; w = geo[z].w; h = geo[z].h; }   // past the total's slot
        const int y = (int)(g - row0);
        PGM_ASSERT(z < n_images && y >= 0 && y <= h);
        if (y == h) continue;                                               // the total's slot
        const int c = row_count_block(score + geo[z].sc + (long long)y * w, w);
        if (threadIdx.x == 0) rowcnt[g] = c;
    }
}

// exclusive scan of n <= 65536 ints by one block of 1024 threads; total written to out[n].  Batched form (geo given):
// blockIdx.x = image, n = its height, in / out at its row slots.
__global__ void scan_kernel(const int32_t *__restrict__ in, int n, int32_t *__restrict__ out,
                            const ImageGeom *__restrict__ geo = nullptr) {
    __shared__ int s_w[32];
    if (geo) { n = geo[blockIdx.x].h; in += geo[blockIdx.x].row; out += geo[blockIdx.x].row; }
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int per = (n + 1023) / 1024, p0 = min(tid * per, n), p1 = min(p0 + per, n);
    int sum = 0;
    for (int k = p0; k < p1; k++) sum += in[k];
    int inc = sum;
    for (int o = 1; o < 32; o <<= 1) { const int a = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += a; }
    if (lane == 31) s_w[wid] = inc;
    __syncthreads();
    int off = inc - sum, tot = 0;
    for (int k = 0; k < 32; k++) { if (k < wid) off += s_w[k]; tot += s_w[k]; }
    for (int k = p0; k < p1; k++) { out[k] = off; off += in[k]; }
    if (tid == 0) out[n] = tot;
}

// ordered emission of row y of one score map by one warp (ballot prefix): Detect's row-major list order, from list
// position `base`, into slots below `capacity`
__device__ __forceinline__ void emit_row(const uint8_t *__restrict__ row, int w, int y, int base, int capacity,
                                         int32_t *__restrict__ xy, int32_t *__restrict__ sc) {
    const int lane = threadIdx.x & 31;
    for (int x0 = 0; x0 < w; x0 += 32) {
        const int x = x0 + lane;
        const uint8_t v = x < w ? row[x] : 0;
        const unsigned m = __ballot_sync(0xffffffffu, v != 0);
        if (v) {
            const int pos = base + __popc(m & ((1u << lane) - 1u));
            if (pos < capacity) { xy[2 * pos] = x; xy[2 * pos + 1] = y; sc[pos] = v; }
        }
        base += __popc(m);
    }
}

// one warp per row
__global__ void emit_kernel(const uint8_t *__restrict__ score, int w, int h, const int32_t *__restrict__ rowoff,
                            int capacity, int32_t *__restrict__ xy, int32_t *__restrict__ sc) {
    const int y = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (y >= h) return;
    emit_row(score + (size_t)y * w, w, y, rowoff[y], capacity, xy, sc);
}

// batched form; every image owns `capacity` output slots.  One size uw x uh (uw > 0): grid (rows / 4, images), one warp
// per row, no table read.  Any other set: one contiguous range of the flat row-slot space per warp.
__global__ void __launch_bounds__(128, FLAT_CTAS_PER_SM_128) emit_kernel(
        const uint8_t *__restrict__ score, const ImageGeom *__restrict__ geo, int n_images, int uw, int uh,
        const int32_t *__restrict__ rowoff, int capacity, int32_t *__restrict__ xy, int32_t *__restrict__ sc) {
    if (uw) {
        const int y = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), z = blockIdx.y;
        if (y >= uh) return;
        emit_row(score + ((long long)z * uh + y) * uw, uw, y, rowoff[(long long)z * (uh + 1) + y], capacity,
                 xy + (size_t)z * capacity * 2, sc + (size_t)z * capacity);
        return;
    }
    long long g0, g1;
    unit_range(geo[n_images].row, (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5),
               (long long)gridDim.x * (blockDim.x >> 5), &g0, &g1);
    if (g0 >= g1) return;
    int z = image_of<&ImageGeom::row>(geo, n_images, g0);
    long long row0 = geo[z].row;
    int h = geo[z].h;
    for (long long g = g0; g < g1; g++) {
        if (g > row0 + h) { z++; row0 = geo[z].row; h = geo[z].h; }
        const int w = geo[z].w, y = (int)(g - row0);
        PGM_ASSERT(z < n_images && y >= 0 && y <= h);
        if (y == h) continue;
        emit_row(score + geo[z].sc + (long long)y * w, w, y, rowoff[g], capacity, xy + (size_t)z * capacity * 2,
                 sc + (size_t)z * capacity);
    }
}

// BRIEF: one warp per keypoint.  pair p sets bit (n_pairs - 1 - p) of the descriptor integer
// (`descriptor <<= 1` per pair, first pair = MSB), stored little-endian in `stride` bytes.
__global__ void brief_kernel(const float *__restrict__ img, int w, int h, const int32_t *__restrict__ xy, int n,
                             const int32_t *__restrict__ pairs /*[n_pairs][4]*/, int n_pairs, int stride_words,
                             int lsb_first, uint32_t *__restrict__ desc, const ImageGeom *__restrict__ geo = nullptr,
                             const int32_t *__restrict__ counts = nullptr) {
    extern __shared__ uint32_t s_desc[];           // [warps][stride_words]
    const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int i = blockIdx.x * (blockDim.x >> 5) + wid;
    if (geo) {                                     // batched form: blockIdx.y = image, its geometry in geo, n = capacity
        const int z = blockIdx.y;                  // per image, and the image's keypoint count in counts[z] on the device
        w = geo[z].w; h = geo[z].h;
        img += geo[z].px; xy += (size_t)z * n * 2; desc += (size_t)z * n * stride_words;
        n = min(n, __ldg(counts + z));
    }
    uint32_t *mine = s_desc + wid * stride_words;
    for (int k = lane; k < stride_words; k += 32) mine[k] = 0u;
    __syncwarp();
    if (i < n) {
        const int x = xy[2 * i], y = xy[2 * i + 1];
        for (int p = lane; p < n_pairs; p += 32) {
            const int4 pr = __ldg(reinterpret_cast<const int4 *>(pairs) + p);
            const int x1 = x + pr.x, y1 = y + pr.y, x2 = x + pr.z, y2 = y + pr.w;
            bool bit = false;
            if (x1 >= 0 && x1 < w && y1 >= 0 && y1 < h && x2 >= 0 && x2 < w && y2 >= 0 && y2 < h)   // Keypoint.cs:39-45
                bit = __ldg(img + (size_t)y1 * w + x1) < __ldg(img + (size_t)y2 * w + x2);          // :47-53
            const int pos = lsb_first ? p : n_pairs - 1 - p;   // models/keypoint.py:49 `des += 2**idx` vs Keypoint.cs:36 `<<= 1`
            if (bit) atomicOr(&mine[pos >> 5], 1u << (pos & 31));
        }
        __syncwarp();
        for (int k = lane; k < stride_words; k += 32) desc[(size_t)i * stride_words + k] = mine[k];
    }
}

// ---- NMS ------------------------------------------------------------------------------------
// rank[i] = position of keypoint i in the stable order by score descending (LINQ OrderByDescending is
// stable, :20): the number of keypoints with a larger score plus the earlier ones with the same score.
__global__ void nms_rank_kernel(const int32_t *__restrict__ sc, int n, int32_t *__restrict__ rank,
                                int32_t *__restrict__ order) {
    __shared__ int s_s[256];
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int mine = i < n ? sc[i] : 0;
    int r = 0;
    for (int j0 = 0; j0 < n; j0 += 256) {
        __syncthreads();
        if (j0 + (int)threadIdx.x < n) s_s[threadIdx.x] = sc[j0 + threadIdx.x];
        __syncthreads();
        const int lim = min(256, n - j0);
        for (int k = 0; k < lim; k++) r += (s_s[k] > mine) || (s_s[k] == mine && j0 + k < i);
    }
    if (i < n) { rank[i] = r; order[r] = i; }
}

// One round of the parallel form of the sequential suppression loop (:23-32).  In rank order, a keypoint
// is kept iff no KEPT keypoint of smaller rank lies within the radius.  state: 0 undecided, 1 kept, 2 dropped.
// An undecided keypoint is dropped as soon as a kept higher-priority neighbour exists, kept once every
// higher-priority neighbour is dropped; repeating to a fixed point gives exactly the sequential answer.
__global__ void nms_round_kernel(const int32_t *__restrict__ xy, const int32_t *__restrict__ rank, int n,
                                 long long radius2, const uint8_t *__restrict__ state_in, uint8_t *__restrict__ state_out,
                                 int32_t *__restrict__ n_undecided) {
    __shared__ int s_x[256], s_y[256], s_r[256];
    __shared__ uint8_t s_s[256];
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    int x = 0, y = 0, r = 0;
    uint8_t st = 2;
    if (i < n) { x = xy[2 * i]; y = xy[2 * i + 1]; r = rank[i]; st = state_in[i]; }
    bool any_kept = false, any_undecided = false;
    for (int j0 = 0; j0 < n; j0 += 256) {
        const int j = j0 + threadIdx.x;
        __syncthreads();
        if (j < n) { s_x[threadIdx.x] = xy[2 * j]; s_y[threadIdx.x] = xy[2 * j + 1]; s_r[threadIdx.x] = rank[j]; s_s[threadIdx.x] = state_in[j]; }
        __syncthreads();
        if (st == 0) {
            const int lim = min(256, n - j0);
            for (int k = 0; k < lim; k++) {
                if (s_r[k] >= r || s_s[k] == 2) continue;
                const long long dx = s_x[k] - x, dy = s_y[k] - y;
                if (dx * dx + dy * dy > radius2) continue;          // IsAcceptableDistance: distance > radius survives
                if (s_s[k] == 1) any_kept = true; else any_undecided = true;
            }
        }
    }
    if (i < n) {
        uint8_t ns = st;
        if (st == 0) {
            if (any_kept) ns = 2;
            else if (!any_undecided) ns = 1;
            if (ns == 0) atomicAdd(n_undecided, 1);
        }
        state_out[i] = ns;
    }
}

// ---- spatially binned form of the same rounds -------------------------------------------------------
// Cells of side max(radius, 1): every keypoint within `radius` of (x, y) lies in the 3 x 3 cells around it.
// Keypoints are sorted by cell id (64-bit radix sort); a round then visits only the 9 neighbouring runs
// instead of all n keypoints, so the cost is O(n . neighbours) per round instead of O(n^2).
__global__ void nms_cell_kernel(const int32_t *__restrict__ xy, int n, int cs, int minx, int miny, long long ncx,
                                unsigned long long *__restrict__ cell, int32_t *__restrict__ idx) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const long long cx = ((long long)xy[2 * i] - minx) / cs, cy = ((long long)xy[2 * i + 1] - miny) / cs;
    cell[i] = (unsigned long long)(cy * ncx + cx);
    idx[i] = i;
}

// key[i] = (inverted score << 32) | i: an ascending sort of the keys is the stable order by score descending
__global__ void nms_score_key_kernel(const int32_t *__restrict__ sc, int n, unsigned long long *__restrict__ key) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) key[i] = ((unsigned long long)(~((unsigned)sc[i] ^ 0x80000000u)) << 32) | (unsigned)i;
}

// order[r] = keypoint of rank r, rank[order[r]] = r
__global__ void nms_order_from_keys_kernel(const unsigned long long *__restrict__ sorted_key, int n,
                                           int32_t *__restrict__ order, int32_t *__restrict__ rank) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    const int i = (int)(unsigned)sorted_key[r];
    order[r] = i; rank[i] = r;
}

__device__ __forceinline__ int lower_bound_u64(const unsigned long long *__restrict__ a, int n, unsigned long long key) {
    int lo = 0, hi = n;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (a[mid] < key) lo = mid + 1; else hi = mid;
    }
    return lo;
}

__global__ void nms_round_binned_kernel(const int32_t *__restrict__ xy, const int32_t *__restrict__ rank, int n,
                                        long long radius2, int cs, int minx, int miny, long long ncx, long long ncy,
                                        const unsigned long long *__restrict__ sorted_cell,
                                        const int32_t *__restrict__ sorted_idx, const uint8_t *__restrict__ state_in,
                                        uint8_t *__restrict__ state_out, int32_t *__restrict__ n_undecided) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint8_t st = state_in[i];
    if (st != 0) { state_out[i] = st; return; }
    const int x = xy[2 * i], y = xy[2 * i + 1], r = rank[i];
    const long long cx = ((long long)x - minx) / cs, cy = ((long long)y - miny) / cs;
    bool any_kept = false, any_undecided = false;
    for (int dy = -1; dy <= 1 && !any_kept; dy++) {
        const long long yy = cy + dy;
        if (yy < 0 || yy >= ncy) continue;
        // the three cells (cx-1 .. cx+1) of one cell row are consecutive ids: one search, one run
        const long long x0 = cx > 0 ? cx - 1 : 0, x1 = cx + 1 < ncx ? cx + 1 : ncx - 1;
        const unsigned long long c0 = (unsigned long long)(yy * ncx + x0), c1 = (unsigned long long)(yy * ncx + x1);
        for (int k = lower_bound_u64(sorted_cell, n, c0); k < n && sorted_cell[k] <= c1; k++) {
            const int j = sorted_idx[k];
            if (rank[j] >= r) continue;
            const uint8_t sj = state_in[j];
            if (sj == 2) continue;
            const long long ddx = (long long)xy[2 * j] - x, ddy = (long long)xy[2 * j + 1] - y;
            if (ddx * ddx + ddy * ddy > radius2) continue;       // IsAcceptableDistance: distance > radius survives
            if (sj == 1) { any_kept = true; break; }
            any_undecided = true;
        }
    }
    uint8_t ns = 0;
    if (any_kept) ns = 2;
    else if (!any_undecided) ns = 1;
    if (ns == 0) atomicAdd(n_undecided, 1);
    state_out[i] = ns;
}

// gathers (xy, score) of the kept keypoints, in output order
__global__ void gather_kept_kernel(const int32_t *__restrict__ xy, const int32_t *__restrict__ sc,
                                   const int32_t *__restrict__ kept, int n_kept, int32_t *__restrict__ oxy,
                                   int32_t *__restrict__ osc) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_kept) return;
    const int i = kept[k];
    oxy[2 * k] = xy[2 * i]; oxy[2 * k + 1] = xy[2 * i + 1]; osc[k] = sc[i];
}

// kept keypoints in rank order = the reference's output order (acceptableList, :21-26)
__global__ void nms_emit_kernel(const int32_t *__restrict__ order, const uint8_t *__restrict__ state, int n,
                                int32_t *__restrict__ kept, int32_t *__restrict__ n_kept) {
    // single block, ordered compaction
    __shared__ int s_w[32];
    __shared__ int s_base;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, nt = blockDim.x;
    if (tid == 0) s_base = 0;
    __syncthreads();
    for (int r0 = 0; r0 < n; r0 += nt) {
        const int r = r0 + tid;
        const int i = r < n ? order[r] : 0;
        const bool hit = r < n && state[i] == 1;
        const unsigned m = __ballot_sync(0xffffffffu, hit);
        if (lane == 0) s_w[wid] = __popc(m);
        __syncthreads();
        int off = s_base;
        for (int k = 0; k < wid; k++) off += s_w[k];
        if (hit) kept[off + __popc(m & ((1u << lane) - 1u))] = i;
        __syncthreads();
        if (tid == 0) { int t = 0; for (int k = 0; k < (nt >> 5); k++) t += s_w[k]; s_base += t; }
        __syncthreads();
    }
    if (tid == 0) *n_kept = s_base;
}

// ---- batched NMS: many images, every round on the device (pgm_detect_nms_describe_batch_dev) ---------------
// All images' FAST lists sit in one flat list, image z's at base[z] .. base[z + 1].  The rounds are those of
// nms_round_binned_kernel, run for every image at once by one persistent kernel; nothing is read back per round.
constexpr int NMS_BATCH_THREADS = 256;
constexpr int NMS_EMIT_THREADS = 1024;
constexpr int NMS_RANK_IMAGE_SHIFT = 40;   // rank key: image << 40 | (255 - score) << 32 | index within the image

// Control words of the rounds kernel, zeroed before its launch.
struct NmsBatchCtl {
    int32_t undecided[3];   // round r counts into [r % 3]; see nms_rounds_batch_kernel
    uint32_t grid_bar;      // grid_barrier counter
    int32_t final_buf;      // which state buffer holds the final states (written at exit)
};

// Detect's row-major list of every image (one warp per row slot, ballot prefix, as emit_kernel) into the flat list at
// the image's base, with each keypoint's rank key, its cell id (geo[z].cell + cy * ncx + cx, cells of side cs over
// [0, w) x [0, h)) and its own flat index (the values of the cell sort).
// One size uw x uh (uw > 0): grid (rows / 4, images), no table read; any other set: a range of row slots per warp
// (as emit_kernel).
__global__ void __launch_bounds__(128, FLAT_CTAS_PER_SM_128) nms_batch_emit_kernel(
        const uint8_t *__restrict__ score, const ImageGeom *__restrict__ geo, int n_images, int uw, int uh,
        const int32_t *__restrict__ rowoff, const int32_t *__restrict__ base, int cs, int32_t *__restrict__ xy,
        int32_t *__restrict__ sc, unsigned long long *__restrict__ rank_key, unsigned long long *__restrict__ cell,
        int32_t *__restrict__ idx) {
    const int lane = threadIdx.x & 31;
    long long g0, g1;
    int z = 0;
    if (uw) {
        const int y = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
        if (y >= uh) return;
        z = blockIdx.y; g0 = (long long)z * (uh + 1) + y; g1 = g0 + 1;
    } else {                                                               // one range of row slots per warp
        unit_range(geo[n_images].row, (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5),
                   (long long)gridDim.x * (blockDim.x >> 5), &g0, &g1);
        if (g0 >= g1) return;
        z = image_of<&ImageGeom::row>(geo, n_images, g0);
    }
    for (long long g = g0; g < g1; g++) {
        int w, h, y, ncx;
        long long sc0, cell0;
        if (uw) {
            w = uw; h = uh; y = (int)(g - (long long)z * (uh + 1));
            ncx = (uw - 1) / cs + 1;
            sc0 = (long long)z * uw * uh; cell0 = (long long)z * ncx * ((uh - 1) / cs + 1);
        } else {
            if (g > geo[z].row + geo[z].h) z++;
            w = geo[z].w; h = geo[z].h; y = (int)(g - geo[z].row); ncx = geo[z].ncx;
            sc0 = geo[z].sc; cell0 = geo[z].cell;
        }
        PGM_ASSERT(z < n_images && y >= 0 && y <= h);
        if (y == h) continue;
        const uint8_t *row = score + sc0 + (long long)y * w;
        const int b0 = __ldg(base + z), n_img = __ldg(base + z + 1) - b0;
        const unsigned long long row_cell = (unsigned long long)cell0 + (unsigned long long)(y / cs) * ncx;
        PGM_ASSERT(row_cell + ncx <= (unsigned long long)geo[n_images].cell);
        int local = rowoff[g];
        for (int x0 = 0; x0 < w; x0 += 32) {
            const int x = x0 + lane;
            const uint8_t v = x < w ? row[x] : 0;
            const unsigned m = __ballot_sync(0xffffffffu, v != 0);
            if (v) {
                const int li = local + __popc(m & ((1u << lane) - 1u));
                PGM_ASSERT(li >= 0 && li < n_img);
                const int i = b0 + li;
                xy[2 * (size_t)i] = x; xy[2 * (size_t)i + 1] = y; sc[i] = v;
                rank_key[i] = ((unsigned long long)z << NMS_RANK_IMAGE_SHIFT) | ((unsigned long long)(255u - v) << 32) | (unsigned)li;
                cell[i] = row_cell + (unsigned)(x / cs);
                idx[i] = i;
            }
            local += __popc(m);
        }
    }
}

// order[r] = flat index of rank r, rank[order[r]] = r.  The key sorts by image first, so image z's ranks are exactly
// base[z] .. base[z + 1] - 1, in LINQ's stable order by score descending.
__global__ void nms_batch_order_kernel(const unsigned long long *__restrict__ sorted_key, int n, const int32_t *__restrict__ base,
                                       int n_images, int32_t *__restrict__ order, int32_t *__restrict__ rank) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    const unsigned long long key = sorted_key[r];
    const int z = (int)(key >> NMS_RANK_IMAGE_SHIFT), li = (int)(unsigned)key;
    PGM_ASSERT(z >= 0 && z < n_images && li >= 0 && li < base[z + 1] - base[z]);
    const int i = base[z] + li;
    PGM_ASSERT(r >= base[z] && r < base[z + 1]);
    order[r] = i; rank[i] = r;
}

// Every round of every image in one cooperative launch.  Round r applies nms_round_binned_kernel's rule to every
// undecided keypoint (state: 0 undecided, 1 kept, 2 dropped; read from st[r & 1], written to st[(r + 1) & 1]) and
// counts the keypoints it leaves undecided into ctl->undecided[r % 3].  Thread 0 zeroes the next round's counter
// during round r; three counters, because with two the zeroing in round r + 1 would race with a late warp still
// reading round r's count after the barrier.  Each round decides at least the best-ranked undecided keypoint of every
// image that has one, so the rounds end after at most n of them.
__global__ void __launch_bounds__(NMS_BATCH_THREADS) nms_rounds_batch_kernel(
        const int32_t *__restrict__ xy, const int32_t *__restrict__ rank, int n, long long radius2, int cs,
        const ImageGeom *__restrict__ geo, int n_images, const unsigned long long *__restrict__ rank_key,
        const unsigned long long *__restrict__ cell, const unsigned long long *__restrict__ sorted_cell,
        const int32_t *__restrict__ sorted_idx, uint8_t *st0, uint8_t *st1, NmsBatchCtl *ctl) {
    const int gt = blockIdx.x * blockDim.x + threadIdx.x, gs = gridDim.x * blockDim.x;
    unsigned epoch = 0;
    for (int round = 0; round < n; round++) {      // (the bound is never reached, see above)
        const uint8_t *st_in = (round & 1) ? st1 : st0;
        uint8_t *st_out = (round & 1) ? st0 : st1;
        int undecided = 0;
        for (int i = gt; i < n; i += gs) {
            const uint8_t st = __ldcg(st_in + i);
            if (st != 0) { st_out[i] = st; continue; }
            const int x = __ldg(xy + 2 * i), y = __ldg(xy + 2 * i + 1), r = __ldg(rank + i);
            const int z = (int)(__ldg(rank_key + i) >> NMS_RANK_IMAGE_SHIFT);   // the image's cell grid
            PGM_ASSERT(z >= 0 && z < n_images);
            const int ncx = geo[z].ncx, ncy = geo[z].ncy, cx = x / cs, cy = y / cs;
            const long long c = (long long)__ldg(cell + i);
            PGM_ASSERT(cx < ncx && cy < ncy && c == geo[z].cell + (long long)cy * ncx + cx);
            bool any_kept = false, any_undecided = false;
            for (int dy = -1; dy <= 1 && !any_kept; dy++) {
                if (cy + dy < 0 || cy + dy >= ncy) continue;
                // the three cells (cx-1 .. cx+1) of one cell row of this image are consecutive ids: one search, one run
                const long long row = c - cx + (long long)dy * ncx;
                const unsigned long long c0 = (unsigned long long)(row + max(cx - 1, 0));
                const unsigned long long c1 = (unsigned long long)(row + min(cx + 1, ncx - 1));
                for (int k = lower_bound_u64(sorted_cell, n, c0); k < n && __ldg(sorted_cell + k) <= c1; k++) {
                    const int j = __ldg(sorted_idx + k);
                    PGM_ASSERT(j >= 0 && j < n);
                    if (__ldg(rank + j) >= r) continue;
                    const uint8_t sj = __ldcg(st_in + j);
                    if (sj == 2) continue;
                    const long long ddx = (long long)__ldg(xy + 2 * j) - x, ddy = (long long)__ldg(xy + 2 * j + 1) - y;
                    if (ddx * ddx + ddy * ddy > radius2) continue;       // IsAcceptableDistance: distance > radius survives
                    if (sj == 1) { any_kept = true; break; }
                    any_undecided = true;
                }
            }
            const uint8_t ns = any_kept ? 2 : (any_undecided ? 0 : 1);
            st_out[i] = ns;
            undecided += ns == 0;
        }
        undecided = __reduce_add_sync(0xffffffffu, undecided);
        if ((threadIdx.x & 31) == 0 && undecided) atomicAdd(&ctl->undecided[round % 3], undecided);
        if (gt == 0) ctl->undecided[(round + 1) % 3] = 0;
        pgm::grid_barrier(&ctl->grid_bar, gridDim.x, epoch);
        if (__ldcg(&ctl->undecided[round % 3]) == 0) {                        // uniform over the grid
            if (gt == 0) ctl->final_buf = (round + 1) & 1;
            return;
        }
    }
    PGM_ASSERT(false);
}

// One CTA per image: the kept keypoints of its rank-ordered run (ballot prefixes, as nms_emit_kernel) into the image's
// `capacity` output slots, in the reference's output order; counts[z] = all survivors, also those beyond capacity.
__global__ void __launch_bounds__(NMS_EMIT_THREADS) nms_batch_gather_kernel(
        const int32_t *__restrict__ order, const int32_t *__restrict__ base, const uint8_t *__restrict__ st0,
        const uint8_t *__restrict__ st1, const NmsBatchCtl *__restrict__ ctl, const int32_t *__restrict__ xy,
        const int32_t *__restrict__ sc, int capacity, int32_t *__restrict__ out_xy, int32_t *__restrict__ out_sc,
        int32_t *__restrict__ counts) {
    __shared__ int s_w[NMS_EMIT_THREADS / 32];
    __shared__ int s_base;
    const int z = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const uint8_t *state = ctl->final_buf ? st1 : st0;
    const int r0 = base[z], r1 = base[z + 1];
    out_xy += (size_t)z * capacity * 2; out_sc += (size_t)z * capacity;
    if (tid == 0) s_base = 0;
    __syncthreads();
    for (int rb = r0; rb < r1; rb += NMS_EMIT_THREADS) {
        const int r = rb + tid;
        const int i = r < r1 ? order[r] : 0;
        PGM_ASSERT(r >= r1 || (i >= r0 && i < r1));
        const bool hit = r < r1 && state[i] == 1;
        const unsigned m = __ballot_sync(0xffffffffu, hit);
        if (lane == 0) s_w[wid] = __popc(m);
        __syncthreads();
        int off = s_base;
        for (int k = 0; k < wid; k++) off += s_w[k];
        const int pos = off + __popc(m & ((1u << lane) - 1u));
        if (hit && pos < capacity) {
            out_xy[2 * (size_t)pos] = xy[2 * (size_t)i]; out_xy[2 * (size_t)pos + 1] = xy[2 * (size_t)i + 1];
            out_sc[pos] = sc[i];
        }
        __syncthreads();
        if (tid == 0) { int t = 0; for (int k = 0; k < NMS_EMIT_THREADS / 32; k++) t += s_w[k]; s_base += t; }
        __syncthreads();
    }
    if (tid == 0) counts[z] = s_base;
}

}  // namespace pgm_det
