// pgm_ransac.cuh -- hypothesis scoring of the fundamental-matrix RANSAC, the consumer of the match list
// (SURVEY.md section 8 row f3): the inner loops of CameraPoseEstimation.GetFundamentalMatrix
// (dotnet_src/ImageProcessing/CameraPoseEstimation.cs:41-88).
//
// For every hypothesis F (row-major 3x3 float) and every pair (Keypoint1 = (x1, y1), Keypoint2 = (x2, y2)):
//     result = (F . (x2, y2, 1)) . (x1, y1, 1)              :66-71
//     inlier  <=>  result <= threshold                      :73 (signed, as upstream -- no absolute value)
// and the winner is the first hypothesis whose inlier count exceeds every earlier one (:79-84); a hypothesis
// flagged invalid (upstream: rank != 2, :46-51) is skipped.  Arithmetic is float32 in MathNet.Numerics'
// (5.0.0) managed order -- each 3-term sum accumulated left to right, no fused multiply-add.
// Trivially parallel integer/float work: one CTA per hypothesis, coordinates streamed from L2.
#pragma once

#include <cstdint>
#include <cuda_runtime.h>

#include "pgm_kernels.cuh"   // PGM_ASSERT

namespace pgm_ransac {

__device__ __forceinline__ float residual(const float (&f)[9], float x1, float y1, float x2, float y2) {
    // F.Multiply(kp1Mat): r_i = (f[i][0]*x2 + f[i][1]*y2) + f[i][2]*1   -- __f*_rn forbids FMA contraction
    const float r0 = __fadd_rn(__fadd_rn(__fmul_rn(f[0], x2), __fmul_rn(f[1], y2)), f[2]);
    const float r1 = __fadd_rn(__fadd_rn(__fmul_rn(f[3], x2), __fmul_rn(f[4], y2)), f[5]);
    const float r2 = __fadd_rn(__fadd_rn(__fmul_rn(f[6], x2), __fmul_rn(f[7], y2)), f[8]);
    // .DotProduct(kp2Mat)
    return __fadd_rn(__fadd_rn(__fmul_rn(r0, x1), __fmul_rn(r1, y1)), r2);
}

__global__ void score_kernel(const float *__restrict__ F, const uint8_t *__restrict__ valid, int n_hyp,
                             const int32_t *__restrict__ xy1, const int32_t *__restrict__ xy2, int n, float threshold,
                             int32_t *__restrict__ counts) {
    const int hyp = blockIdx.x;
    if (hyp >= n_hyp) return;
    __shared__ int s_cnt;
    if (threadIdx.x == 0) s_cnt = 0;
    __syncthreads();
    int c = 0;
    if (!valid || valid[hyp]) {
        float f[9];
#pragma unroll
        for (int k = 0; k < 9; k++) f[k] = __ldg(F + (size_t)hyp * 9 + k);
        for (int p = threadIdx.x; p < n; p += blockDim.x) {
            const int2 a = __ldg(reinterpret_cast<const int2 *>(xy1) + p), b = __ldg(reinterpret_cast<const int2 *>(xy2) + p);
            c += residual(f, (float)a.x, (float)a.y, (float)b.x, (float)b.y) <= threshold;
        }
    }
    for (int o = 16; o; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(&s_cnt, c);
    __syncthreads();
    if (threadIdx.x == 0) counts[hyp] = (!valid || valid[hyp]) ? s_cnt : -1;
}

// first index attaining the maximum count (> 0), else -1; then the winner's inlier mask
__global__ void best_kernel(const float *__restrict__ F, const int32_t *__restrict__ counts, int n_hyp,
                            const int32_t *__restrict__ xy1, const int32_t *__restrict__ xy2, int n, float threshold,
                            int32_t *__restrict__ best, uint8_t *__restrict__ mask) {
    __shared__ unsigned long long s_key;
    if (threadIdx.x == 0) s_key = 0ull;
    __syncthreads();
    unsigned long long k = 0ull;
    for (int hI = threadIdx.x; hI < n_hyp; hI += blockDim.x) {
        const int c = counts[hI];
        if (c > 0) {   // larger count wins, then the smaller index
            const unsigned long long key = ((unsigned long long)c << 32) | (unsigned)(0x7FFFFFFF - hI);
            k = key > k ? key : k;
        }
    }
    atomicMax(&s_key, k);
    __syncthreads();
    const int b = s_key ? 0x7FFFFFFF - (int)(s_key & 0xFFFFFFFFull) : -1;
    if (threadIdx.x == 0) *best = b;
    if (mask) {
        float f[9];
#pragma unroll
        for (int q = 0; q < 9; q++) f[q] = b >= 0 ? F[(size_t)b * 9 + q] : 0.f;
        for (int p = threadIdx.x; p < n; p += blockDim.x)
            mask[p] = b >= 0 && residual(f, (float)xy1[2 * p], (float)xy1[2 * p + 1], (float)xy2[2 * p], (float)xy2[2 * p + 1]) <= threshold;
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// Many match lists in one call (pgm_ransac_fundamental_pairs_batch_dev): the whole of GetFundamentalMatrix per pair --
// sampler, 8-point estimate (:204-250), rank gate (:46-51), scoring, winner and inlier mask -- with no host round trip.
//
//   estimate_kernel  one thread per hypothesis of a chunk; R and V of its 9x9 fp64 solve live in shared memory
//   pairs_score_kernel  (pair, block of RB_SCORE_THREADS hypotheses) items; the pair's matches are staged through
//                    shared memory as float (x1, y1, x2, y2) tiles; one 64-bit atomicMax of (count << 32 | ~s) per CTA
//   winner_kernel    one CTA per pair: decodes the key, recomputes the winner's F from (seed, a, b, s) with the same
//                    device function, writes F, its inlier count and the mask at the pair's match slots
// The estimate is one deterministic device function (no atomics, no cross-thread reduction), so the winner's F is
// recomputed bit-identically instead of being kept for every hypothesis: scratch is O(pairs + chunk), not O(S).
// ---------------------------------------------------------------------------------------------------------------------
constexpr int RB_MAX_P = 64;
constexpr int RB_EST_THREADS = 32;                // shared memory: 162 doubles per thread
constexpr int RB_SCORE_THREADS = 128;
constexpr int RB_TILE = 2048;                     // matches per shared-memory tile of the score kernel (32 KB)
constexpr int RB_WIN_THREADS = 256;
constexpr int RB_SM_DOUBLES = 162;                // R[81] | V[81] (the sample indices live in V until the QR is done)

struct RbPair {                 // one pair of the caller's list
    int64_t start;              // its first match slot
    int64_t off_a, off_b;       // first rows of images a and b in d_all_xy
    int32_t count, a, b;        // matches; the image indices (sampler key)
    int32_t n_a, n_b;           // image sizes (checked build)
    int32_t pad;
};

__host__ __device__ __forceinline__ uint64_t splitmix64(uint64_t z) {
    z += 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
// the sampler's key of an image pair, and the 32-bit draw t of hypothesis s (include/pgmatch.h states both)
__host__ __device__ __forceinline__ uint64_t pair_key(uint64_t seed, int32_t a, int32_t b) {
    return splitmix64(seed ^ splitmix64(((uint64_t)(uint32_t)a << 32) | (uint32_t)b));
}
__device__ __forceinline__ uint32_t draw_u32(uint64_t key, uint32_t s, uint32_t t) {
    return (uint32_t)(splitmix64(key ^ (((uint64_t)s << 32) | t)) >> 32);
}

// One-sided (Hestenes) Jacobi rotation of columns p < q of the 9x9 matrices M and V (element (i, j) at [(9 i + j) ld]).
__device__ __forceinline__ bool jacobi_rotate9(double *M, double *V, int ld, int p, int q) {
    double al = 0.0, be = 0.0, ga = 0.0;
#pragma unroll
    for (int i = 0; i < 9; i++) {
        const double x = M[(9 * i + p) * ld], y = M[(9 * i + q) * ld];
        al += x * x; be += y * y; ga += x * y;
    }
    if (!(fabs(ga) > 1e-15 * sqrt(al * be))) return false;
    const double ze = (be - al) / (2.0 * ga);
    const double t = copysign(1.0, ze) / (fabs(ze) + sqrt(1.0 + ze * ze));
    const double c = 1.0 / sqrt(1.0 + t * t), s = c * t;
#pragma unroll
    for (int i = 0; i < 9; i++) {
        const double x = M[(9 * i + p) * ld], y = M[(9 * i + q) * ld];
        M[(9 * i + p) * ld] = c * x - s * y;
        M[(9 * i + q) * ld] = s * x + c * y;
        const double u = V[(9 * i + p) * ld], w = V[(9 * i + q) * ld];
        V[(9 * i + p) * ld] = c * u - s * w;
        V[(9 * i + q) * ld] = s * u + c * w;
    }
    return true;
}

// Singular values of a 3x3 (one-sided Jacobi in registers, fp64), descending.
__device__ __forceinline__ void svd3_values(const double (&f)[9], double (&sv)[3]) {
    double m[9];
#pragma unroll
    for (int k = 0; k < 9; k++) m[k] = f[k];
    for (int sweep = 0; sweep < 40; sweep++) {
        bool rot = false;
#pragma unroll
        for (int pq = 0; pq < 3; pq++) {
            const int p = pq == 2 ? 1 : 0, q = pq == 0 ? 1 : 2;
            double al = 0.0, be = 0.0, ga = 0.0;
#pragma unroll
            for (int i = 0; i < 3; i++) { al += m[3 * i + p] * m[3 * i + p]; be += m[3 * i + q] * m[3 * i + q]; ga += m[3 * i + p] * m[3 * i + q]; }
            if (!(fabs(ga) > 1e-15 * sqrt(al * be))) continue;
            const double ze = (be - al) / (2.0 * ga);
            const double t = copysign(1.0, ze) / (fabs(ze) + sqrt(1.0 + ze * ze));
            const double c = 1.0 / sqrt(1.0 + t * t), s = c * t;
#pragma unroll
            for (int i = 0; i < 3; i++) {
                const double x = m[3 * i + p], y = m[3 * i + q];
                m[3 * i + p] = c * x - s * y; m[3 * i + q] = s * x + c * y;
            }
            rot = true;
        }
        if (!rot) break;
    }
#pragma unroll
    for (int j = 0; j < 3; j++) sv[j] = sqrt(m[j] * m[j] + m[3 + j] * m[3 + j] + m[6 + j] * m[6 + j]);
    if (sv[0] < sv[1]) { const double x = sv[0]; sv[0] = sv[1]; sv[1] = x; }
    if (sv[1] < sv[2]) { const double x = sv[1]; sv[1] = sv[2]; sv[2] = x; }
    if (sv[0] < sv[1]) { const double x = sv[0]; sv[0] = sv[1]; sv[1] = x; }
}

// Upstream's rank gate (Svd.Rank of the float32 F): rank = #{sigma_k > 3 ulp_f32(sigma_0)}, sigma in fp64.
__device__ __forceinline__ bool rank_is_2(const float (&F)[9]) {
    double f[9], sv[3];
#pragma unroll
    for (int k = 0; k < 9; k++) f[k] = (double)F[k];
    svd3_values(f, sv);
    const float s0 = (float)sv[0];
    const double tol = (double)((nextafterf(s0, __int_as_float(0x7f800000)) - s0) * 3.0f);
    return (int)(sv[0] > tol) + (int)(sv[1] > tol) + (int)(sv[2] > tol) == 2;
}

__device__ __forceinline__ void load_match(const RbPair &pp, int64_t slot, const int32_t *__restrict__ xy,
                                           const int32_t *__restrict__ qi, const int32_t *__restrict__ tj,
                                           int32_t &x1, int32_t &y1, int32_t &x2, int32_t &y2) {
    const int32_t q = qi[slot], t = tj[slot];
    PGM_ASSERT(q >= 0 && q < pp.n_a && t >= 0 && t < pp.n_b);
    const int2 u = reinterpret_cast<const int2 *>(xy)[pp.off_a + q], v = reinterpret_cast<const int2 *>(xy)[pp.off_b + t];
    x1 = u.x; y1 = u.y; x2 = v.x; y2 = v.y;
}

// Hypothesis s of pair pp: Floyd's sample of P distinct match indices (ascending), the translation-only normalised
// 8-point estimate of the host mirror (camera_pose_estimation.py) with the null vector of A from Givens QR + one-sided
// Jacobi in fp64, and F = T2^T F0 T1 rounded once to float32.  sm: this thread's RB_SM_DOUBLES doubles at stride ld.
__device__ void estimate_hypothesis(const RbPair &pp, uint64_t key, uint32_t s, int P, const int32_t *__restrict__ xy,
                                    const int32_t *__restrict__ qi, const int32_t *__restrict__ tj, double *sm, int ld,
                                    float (&F)[9]) {
    double *R = sm, *V = sm + 81 * ld;
    // sampler: Floyd's algorithm; V[k] holds the sorted sample (indices < 2^31 are exact doubles)
    const int count = pp.count;
    int n = 0;
    for (int t = 0; t < P; t++) {
        const uint32_t j = (uint32_t)(count - P + t);
        const uint32_t r = (uint32_t)(((uint64_t)draw_u32(key, s, (uint32_t)t) * ((uint64_t)j + 1)) >> 32);
        int pos = n;
        bool present = false;
        for (int k = 0; k < n; k++) {
            const double v = V[k * ld];
            if (v == (double)r) { present = true; break; }
            if (v > (double)r) { pos = k; break; }
        }
        if (present) {
            V[n * ld] = (double)j;           // every element is < j
        } else {
            for (int k = n; k > pos; k--) V[k * ld] = V[(k - 1) * ld];
            V[pos * ld] = (double)r;
        }
        n++;
    }
    // CalculateTransformationMatrix: centroid in double, rounded to float32; Pow(x, 0) == 1, so no scaling
    int64_t sx1 = 0, sy1 = 0, sx2 = 0, sy2 = 0;
    for (int k = 0; k < P; k++) {
        int32_t x1, y1, x2, y2;
        load_match(pp, pp.start + (int64_t)V[k * ld], xy, qi, tj, x1, y1, x2, y2);
        sx1 += x1; sy1 += y1; sx2 += x2; sy2 += y2;
    }
    const float c1x = (float)((double)sx1 / P), c1y = (float)((double)sy1 / P);
    const float c2x = (float)((double)sx2 / P), c2y = (float)((double)sy2 / P);
    // A (P x 9) row by row into R by Givens rotations: backward-stable QR without storing A
    for (int k = 0; k < 81; k++) R[k * ld] = 0.0;
    for (int k = 0; k < P; k++) {
        int32_t x1, y1, x2, y2;
        load_match(pp, pp.start + (int64_t)V[k * ld], xy, qi, tj, x1, y1, x2, y2);
        const float a1 = __fsub_rn((float)x1, c1x), b1 = __fsub_rn((float)y1, c1y);
        const float a2 = __fsub_rn((float)x2, c2x), b2 = __fsub_rn((float)y2, c2y);
        double row[9] = {(double)__fmul_rn(a1, a2), (double)__fmul_rn(a1, b2), (double)a1,
                         (double)__fmul_rn(b1, a2), (double)__fmul_rn(b1, b2), (double)b1,
                         (double)a2, (double)b2, 1.0};
#pragma unroll
        for (int i = 0; i < 9; i++) {
            const double rii = R[(9 * i + i) * ld];
            const double r = sqrt(rii * rii + row[i] * row[i]);
            const bool z = row[i] == 0.0;                      // nothing to eliminate: identity rotation
            const double c = z ? 1.0 : rii / r, sn = z ? 0.0 : row[i] / r;
            R[(9 * i + i) * ld] = z ? rii : r;
#pragma unroll
            for (int j = i + 1; j < 9; j++) {
                const double x = R[(9 * i + j) * ld];
                R[(9 * i + j) * ld] = c * x + sn * row[j];
                row[j] = c * row[j] - sn * x;
            }
        }
    }
    // one-sided Jacobi on R: R V = U Sigma; the null vector of A is the column of V with the smallest column norm
    for (int k = 0; k < 81; k++) V[k * ld] = (k % 10 == 0) ? 1.0 : 0.0;
    for (int sweep = 0; sweep < 40; sweep++) {
        bool rot = false;
        for (int p = 0; p < 8; p++)
            for (int q = p + 1; q < 9; q++) rot |= jacobi_rotate9(R, V, ld, p, q);
        if (!rot) break;
    }
    int jmin = 0;
    double nmin = 0.0;
    for (int j = 0; j < 9; j++) {
        double nn = 0.0;
#pragma unroll
        for (int i = 0; i < 9; i++) nn += R[(9 * i + j) * ld] * R[(9 * i + j) * ld];
        if (j == 0 || nn < nmin) { nmin = nn; jmin = j; }
    }
    double v[9], vmax = 0.0;
#pragma unroll
    for (int i = 0; i < 9; i++) {
        v[i] = V[(9 * i + jmin) * ld];
        if (i == 0 || fabs(v[i]) > fabs(vmax)) vmax = v[i];
    }
    const double sg = vmax < 0.0 ? -1.0 : 1.0;             // largest component positive (lowest index on ties)
    // F0 = DenseOfColumnMajor(3, 3, v): F0[i][j] = v[3 j + i];  F = T2^T F0 T1
    const double t1[9] = {1.0, 0.0, -(double)c1x, 0.0, 1.0, -(double)c1y, 0.0, 0.0, 1.0};
    const double t2t[9] = {1.0, 0.0, 0.0, 0.0, 1.0, 0.0, -(double)c2x, -(double)c2y, 1.0};
    double m[9];
#pragma unroll
    for (int i = 0; i < 3; i++)
#pragma unroll
        for (int j = 0; j < 3; j++)
            m[3 * i + j] = (sg * v[i]) * t1[j] + (sg * v[3 + i]) * t1[3 + j] + (sg * v[6 + i]) * t1[6 + j];
#pragma unroll
    for (int i = 0; i < 3; i++)
#pragma unroll
        for (int j = 0; j < 3; j++)
            F[3 * i + j] = (float)(t2t[3 * i] * m[j] + t2t[3 * i + 1] * m[3 + j] + t2t[3 * i + 2] * m[6 + j]);
}

// Hypotheses [g0, g1) of the flattened (active pair k, sample s) space, g = k S + s.
__global__ void __launch_bounds__(RB_EST_THREADS) estimate_kernel(const RbPair *__restrict__ plan, const int32_t *__restrict__ act,
        int64_t S, int64_t g0, int64_t g1, const int32_t *__restrict__ xy, const int32_t *__restrict__ qi,
        const int32_t *__restrict__ tj, int P, uint64_t seed, int rank_test, float *__restrict__ hF,
        uint8_t *__restrict__ hvalid, float *__restrict__ out_hyp_F) {
    extern __shared__ double rb_sm[];
    const int64_t g = g0 + (int64_t)blockIdx.x * RB_EST_THREADS + threadIdx.x;
    if (g >= g1) return;
    const int64_t k = g / S;
    const uint32_t s = (uint32_t)(g - k * S);
    const int32_t pid = act[k];
    const RbPair pp = plan[pid];
    float F[9];
    estimate_hypothesis(pp, pair_key(seed, pp.a, pp.b), s, P, xy, qi, tj, rb_sm + threadIdx.x, RB_EST_THREADS, F);
    const bool ok = !rank_test || rank_is_2(F);
#pragma unroll
    for (int i = 0; i < 9; i++) hF[(g - g0) * 9 + i] = F[i];
    hvalid[g - g0] = ok;
    if (out_hyp_F) {
#pragma unroll
        for (int i = 0; i < 9; i++) out_hyp_F[((int64_t)pid * S + s) * 9 + i] = F[i];
    }
}

// item -> (pair of the chunk, block of hypotheses): item_base[0..n] is the chunk's prefix of items per pair
__global__ void __launch_bounds__(RB_SCORE_THREADS) pairs_score_kernel(const RbPair *__restrict__ plan,
        const int32_t *__restrict__ act, const int32_t *__restrict__ item_base, int n_local, int64_t k_first, int64_t S,
        int64_t g0, int64_t g1, const float *__restrict__ hF, const uint8_t *__restrict__ hvalid,
        const int32_t *__restrict__ xy, const int32_t *__restrict__ qi, const int32_t *__restrict__ tj, float threshold,
        unsigned long long *__restrict__ keys, int32_t *__restrict__ out_hyp_counts) {
    __shared__ float4 s_m[RB_TILE];
    __shared__ unsigned long long s_key[RB_SCORE_THREADS / 32];
    const int item = blockIdx.x;
    int lo = 0, hi = n_local;                                  // last j with item_base[j] <= item
    while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (item_base[mid] <= item) lo = mid; else hi = mid; }
    const int64_t k = k_first + lo;
    PGM_ASSERT(lo >= 0 && lo < n_local && item >= item_base[lo] && item < item_base[lo + 1]);
    const int32_t pid = act[k];
    const RbPair pp = plan[pid];
    const int64_t hs = (g0 > k * S ? g0 : k * S) + (int64_t)(item - item_base[lo]) * RB_SCORE_THREADS;
    const int64_t he = g1 < (k + 1) * S ? g1 : (k + 1) * S;
    const int64_t g = hs + threadIdx.x;
    const bool live = g < he;
    bool valid = false;
    float f[9];
#pragma unroll
    for (int i = 0; i < 9; i++) f[i] = 0.f;
    if (live) {
        valid = hvalid[g - g0] != 0;
#pragma unroll
        for (int i = 0; i < 9; i++) f[i] = hF[(g - g0) * 9 + i];
    }
    int c = 0;
    for (int base = 0; base < pp.count; base += RB_TILE) {
        const int n = pp.count - base < RB_TILE ? pp.count - base : RB_TILE;
        __syncthreads();
        for (int m = threadIdx.x; m < n; m += RB_SCORE_THREADS) {
            int32_t x1, y1, x2, y2;
            load_match(pp, pp.start + base + m, xy, qi, tj, x1, y1, x2, y2);
            s_m[m] = make_float4((float)x1, (float)y1, (float)x2, (float)y2);
        }
        __syncthreads();
        if (valid) {
#pragma unroll 4
            for (int m = 0; m < n; m++) {
                const float4 u = s_m[m];
                c += residual(f, u.x, u.y, u.z, u.w) <= threshold;
            }
        }
    }
    const uint32_t s = (uint32_t)(g - k * S);
    if (live && out_hyp_counts) out_hyp_counts[(int64_t)pid * S + s] = valid ? c : -1;
    unsigned long long key = (live && valid && c > 0) ? (((unsigned long long)c << 32) | (uint32_t)~s) : 0ull;
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        const unsigned long long x = __shfl_xor_sync(0xffffffffu, key, o);
        key = x > key ? x : key;
    }
    if ((threadIdx.x & 31) == 0) s_key[threadIdx.x >> 5] = key;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long b = 0ull;
#pragma unroll
        for (int w = 0; w < RB_SCORE_THREADS / 32; w++) b = s_key[w] > b ? s_key[w] : b;
        if (b) atomicMax(keys + pid, b);
    }
}

// One CTA per pair of the caller's list.  best: -2 below P matches, -1 without a positive count.
__global__ void __launch_bounds__(RB_WIN_THREADS) winner_kernel(const RbPair *__restrict__ plan, int P, uint64_t seed,
        const unsigned long long *__restrict__ keys, const int32_t *__restrict__ xy, const int32_t *__restrict__ qi,
        const int32_t *__restrict__ tj, float threshold, int32_t *__restrict__ out_best, int32_t *__restrict__ out_inliers,
        float *__restrict__ out_F, uint8_t *__restrict__ out_mask) {
    __shared__ double s_sm[RB_SM_DOUBLES];
    __shared__ float s_F[9];
    __shared__ int s_cnt;
    const int pid = blockIdx.x;
    const RbPair pp = plan[pid];
    const unsigned long long key = pp.count >= P ? keys[pid] : 0ull;
    const uint32_t s = ~(uint32_t)key;
    if (threadIdx.x == 0) {
        float F[9];
        if (key) estimate_hypothesis(pp, pair_key(seed, pp.a, pp.b), s, P, xy, qi, tj, s_sm, 1, F);
#pragma unroll
        for (int i = 0; i < 9; i++) s_F[i] = key ? F[i] : 0.f;
        s_cnt = 0;
    }
    __syncthreads();
    float f[9];
#pragma unroll
    for (int i = 0; i < 9; i++) f[i] = s_F[i];
    int c = 0;
    for (int m = threadIdx.x; m < pp.count; m += RB_WIN_THREADS) {
        bool in = false;
        if (key) {
            int32_t x1, y1, x2, y2;
            load_match(pp, pp.start + m, xy, qi, tj, x1, y1, x2, y2);
            in = residual(f, (float)x1, (float)y1, (float)x2, (float)y2) <= threshold;
        }
        out_mask[pp.start + m] = in;
        c += in;
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(&s_cnt, c);
    __syncthreads();
    if (threadIdx.x == 0) {
        PGM_ASSERT(s_cnt == (int)(key >> 32));
        out_best[pid] = pp.count < P ? -2 : key ? (int32_t)s : -1;
        out_inliers[pid] = s_cnt;
    }
    if (threadIdx.x < 9) out_F[(int64_t)pid * 9 + threadIdx.x] = f[threadIdx.x];
}

}  // namespace pgm_ransac
