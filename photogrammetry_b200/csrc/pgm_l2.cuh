// pgm_l2.cuh -- float-descriptor nearest/second-nearest neighbour on the 5th-gen tensor cores.
//
// north_star extension (SURVEY.md section 8 row a8): the reference has no float descriptor, so
// the semantics are fixed by the test oracle (orc_l2_knn2: exact squared L2, ties by
// smaller train index).  This is the one place where the path is a dense contraction:
//
//     ||q - t||^2 = ||q||^2 + ||t||^2 - 2 q.t          (N1 x N2 x D GEMM)
//
// The GEMM only RANKS.  CTA-pair kernel (n1 > 128): every component becomes ONE fp16 value under a global power-of-two
// scale (absmax_kernel + split16_kernel), one GEMM pass of K = Dp.  Single-CTA kernel (n1 <= 128): bf16 hi + lo split,
// q.t ~ hi.hi + lo.hi + hi.lo as three passes into the same fp32 TMEM accumulator.  Operand rows are stored once as
// [x16 | norm] (resp. [x_hi | x_lo | norm]).  The norm chunk folds ||q||^2 and ||t||^2 into the SAME accumulator: the
// query row carries -||q||^2/2 as three 16-bit terms against constants on the train side and vice versa, so one extra
// K = 16 MMA per tile leaves q.t - (||q||^2 + ||t||^2)/2 = -d/2 in TMEM and the epilogue needs no arithmetic at all: a
// distance's rank is its bit pattern.  The epilogue keeps, per query and column group, the columns within the
// ranking's error band of the second best one (RowTop below); l2_refine_kernel recomputes those few distances exactly
// in fp32 (sum of squared differences), picks best/second and certifies that the lists cannot have hidden a better
// column; rows it cannot certify are recomputed exhaustively by l2_exact_rows_kernel.  Reported distances are exact to
// fp32 rounding; indices can differ from the oracle only where exact fp32 distances tie up to summation order.
//
// Kernel anatomy (sm_100a, hand-written PTX; layouts follow the canonical K-major
// SWIZZLE_128B UMMA atoms):
//   warp 0   TMA producer: A' tile (128 queries x K', resident) once, then B' tiles
//            (128 train rows x 64) through a ring of mbarrier-guarded stages
//   warp 1   one thread issues tcgen05.mma.kind::f16 (K = 16) into one of two TMEM accumulators,
//            tcgen05.commit frees stages / publishes the accumulator
//   warp 2   TMEM alloc / dealloc
//   warps 4-11 epilogue (two warpgroups, half the columns each): tcgen05.ld (32 lanes x 32
//            columns per instruction), float max tree + one compare per 32 columns, slow path only for
//            chunks that can still matter
#pragma once

#include <cstdint>
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

namespace pgm_l2 {

constexpr int TILE_M = 128;        // queries per CTA (TMEM lanes)
constexpr int TILE_N = 128;        // train rows per accumulator
constexpr int CHUNK_K = 64;        // bf16 elements per 128-byte swizzle row
constexpr int UMMA_K = 16;         // K of one tcgen05.mma for 16-bit inputs
constexpr int MAX_CHUNKS = 5;      // resident A' chunks: [hi | lo | norm], Dp <= 128
constexpr int STAGES = 8;          // B' ring of chunk slots: two whole tiles deep at Dp = 128
constexpr int EPI_GROUPS = 2;      // each epilogue warpgroup reduces an equal share of the accumulator's columns
constexpr int THREADS = 128 + 128 * EPI_GROUPS; // warps 0-3: TMA / MMA / TMEM alloc / spare; then the epilogue warpgroups
constexpr int TOPK = 8;            // candidates kept per (query, column split, epilogue warpgroup)
constexpr int CAND = TOPK * EPI_GROUPS;
constexpr uint32_t CHUNK_BYTES = TILE_N * CHUNK_K * 2;   // 16 KB (A' and B' chunks have the same shape)
constexpr uint32_t TMEM_COLS = 256;                      // two fp32 accumulators of 128 columns

// ---- PTX helpers ------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"     // suspend-time hint: the thread sleeps in
        "selp.u32 %0, 1, 0, p;\n\t}"                                         // hardware, no issue slots (a pure spin measured 4-8 % slower)
        : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity), "r"(20000u) : "memory");
    return ok != 0;
}
// Bounded wait: a protocol bug traps (kernel error) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    uint32_t spins = 0;
    while (!mbar_try_wait(bar, parity)) {
        if (++spins > 2000000u) __trap();
    }
}
__device__ __forceinline__ void tma_load_2d(void *smem_dst, const CUtensorMap *map, uint64_t *bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t *bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_mma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tc_ld_32x32b_x32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
          "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
          "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr) : "memory");
}
// Programmatic dependent launch: a kernel launched with the programmatic-stream-serialization attribute may
// start (prologue: barriers, TMEM allocation) while its predecessor drains; pdl_wait() blocks until the
// predecessor grid has completed and its memory is visible.  pdl_trigger() lets the successor start early.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major, SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor):
// start>>4 | LBO(=1)<<16 | SBO(=1024 B >> 4)<<32 | version 1 <<46 | layout SWIZZLE_128B(2) <<61
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
    return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | (1ull << 16) | ((uint64_t)(1024 >> 4) << 32) | (1ull << 46) |
           (2ull << 61);
}
// Instruction descriptor (cute::UMMA::InstrDescriptor): D=F32, A=B=BF16, both K-major, N>>3, M>>4.
constexpr uint32_t IDESC_BF16_M128_N128 =
    (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(TILE_N >> 3) << 17) | ((uint32_t)(TILE_M >> 4) << 24);

// ---- preprocessing: fp32 rows -> split bf16 operand rows (one launch for both operands) --------
// Row layout: [hi (Dp) | lo (Dp) | norm chunk (64)], zero padded.  Norm chunk of a query row:
// (h0, h1, h2, 1, 1, 1, 0...) with h0 + h1 + h2 = -||q||^2 / 2 exactly (three bf16 terms carry 24 bits);
// of a train row: (1, 1, 1, h0, h1, h2, 0...).  Their dot product is -(||q||^2 + ||t||^2) / 2.
// One warp per row: rows [0, n1) are queries, rows [n1, n1 + n2) train descriptors.
__global__ void __launch_bounds__(256) split_kernel(const float *__restrict__ q, int n1, const float *__restrict__ t, int n2,
                                                    int dim, int dp, __nv_bfloat16 *__restrict__ a,
                                                    __nv_bfloat16 *__restrict__ b, int32_t *__restrict__ cand_j,
                                                    int slots, float *__restrict__ qnorm, float *__restrict__ cand_drop) {
    const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    pdl_trigger();                                   // the GEMM kernel's prologue may overlap this kernel
    if (w >= n1 + n2) return;
    const bool train = w >= n1;
    const int row = train ? w - n1 : w;
    if (!train)                                      // candidate slots no segment of the GEMM kernel fills stay "absent"
    {
        for (int e = lane; e < slots * CAND; e += 32) cand_j[((size_t)(e / CAND) * n1 + row) * CAND + (e % CAND)] = -1;
        for (int e = lane; e < slots * EPI_GROUPS; e += 32)
            cand_drop[((size_t)(e / EPI_GROUPS) * n1 + row) * EPI_GROUPS + (e % EPI_GROUPS)] = 3.4e38f;
    }
    const float *x = (train ? t : q) + (size_t)row * dim;
    __nv_bfloat16 *o = (train ? b : a) + (size_t)row * (2 * dp + CHUNK_K);
    float acc = 0.f;
    const bool vec = (dim & 3) == 0 && ((reinterpret_cast<uintptr_t>(x) & 15) == 0);   // rows are 16-byte aligned
    for (int k = 4 * lane; k < dp; k += 128) {       // four components per lane: one 128-bit load, two 64-bit stores
        float v[4];
        if (vec && k + 3 < dim) {
            const float4 f = __ldg(reinterpret_cast<const float4 *>(x + k));
            v[0] = f.x; v[1] = f.y; v[2] = f.z; v[3] = f.w;
        } else {
#pragma unroll
            for (int e = 0; e < 4; e++) v[e] = k + e < dim ? __ldg(x + k + e) : 0.f;
        }
        __nv_bfloat162 hi[2], lo[2];
#pragma unroll
        for (int e = 0; e < 2; e++) {
            const __nv_bfloat16 h0 = __float2bfloat16_rn(v[2 * e]), h1 = __float2bfloat16_rn(v[2 * e + 1]);
            hi[e].x = h0; hi[e].y = h1;
            lo[e].x = __float2bfloat16_rn(v[2 * e] - __bfloat162float(h0));
            lo[e].y = __float2bfloat16_rn(v[2 * e + 1] - __bfloat162float(h1));
        }
        *reinterpret_cast<uint2 *>(o + k) = make_uint2(*reinterpret_cast<uint32_t *>(&hi[0]), *reinterpret_cast<uint32_t *>(&hi[1]));
        *reinterpret_cast<uint2 *>(o + dp + k) = make_uint2(*reinterpret_cast<uint32_t *>(&lo[0]), *reinterpret_cast<uint32_t *>(&lo[1]));
#pragma unroll
        for (int e = 0; e < 4; e++) acc = fmaf(v[e], v[e], acc);
    }
    for (int sh = 16; sh; sh >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, sh);
    if (!train && lane == 0) qnorm[row] = acc;
    const float hn = -0.5f * acc;
    const __nv_bfloat16 e0 = __float2bfloat16_rn(hn);
    const float r1 = hn - __bfloat162float(e0);
    const __nv_bfloat16 e1 = __float2bfloat16_rn(r1);
    const __nv_bfloat16 e2 = __float2bfloat16_rn(r1 - __bfloat162float(e1));
    const __nv_bfloat16 one = __float2bfloat16_rn(1.f), zero = __float2bfloat16_rn(0.f);
    // columns 0..2 and 3..5 of the norm chunk; lane l writes columns 2l and 2l + 1
    const __nv_bfloat16 n0 = train ? one : e0, n1v = train ? one : e1, n2v = train ? one : e2;
    const __nv_bfloat16 n3 = train ? e0 : one, n4 = train ? e1 : one, n5 = train ? e2 : one;
    __nv_bfloat162 ext;
    ext.x = lane == 0 ? n0 : lane == 1 ? n2v : lane == 2 ? n4 : zero;
    ext.y = lane == 0 ? n1v : lane == 1 ? n3 : lane == 2 ? n5 : zero;
    *reinterpret_cast<__nv_bfloat162 *>(o + 2 * dp + 2 * lane) = ext;
}


// ---- single-term fp16 ranking (round 2) ---------------------------------------------------------
// The three-term bf16 split costs three GEMM passes for a ranking that the refinement kernel re-derives
// exactly anyway.  One fp16 term ranks as well as needed: fp16 rounds to 2^-11 relative, so
//     |h_q.h_t - q.t| <= (2 * 2^-11 + 2^-22) sum |q_i t_i| <= 2^-10 |q| |t|,   i.e.  |d_approx - d| <= 2^-10 (|q|^2 + |t|^2)
// and the refinement keeps every candidate within that band of the second-best approximation (typically
// one extra train row per query).  A query whose band could hide a train row the epilogue's top-4 lists
// dropped is recomputed exhaustively (l2_exact_rows_kernel), so the result does not depend on the data
// being well spread.  fp16 has a narrow exponent range, hence a global power-of-two scale s (exact in
// fp32) that maps max |x| over both sets into [2^9, 2^10): squared norms stay below 2^27 and components down
// to 2^-24 of the maximum keep their full relative precision.  The norm chunk carries -|x s|^2 / 2 as
// 4096 * (h0 + h1 + h2) -- three fp16 terms, 33 bits -- against (4096, 4096, 4096) on the other side.
constexpr float NORM_C = 4096.f;
__device__ __forceinline__ void l2_scale_from_bits(unsigned bits, float &s, float &inv_s2, float &mprime) {
    int eb = (int)(bits >> 23);                      // biased exponent of max |x| (sign bit is clear)
    if (bits == 0u) { s = 1.f; inv_s2 = 1.f; mprime = 0.f; return; }
    eb = max(eb, 1);
    const int sb = min(max(263 - eb, 127 - 60), 127 + 60);   // s = 2^(136 - eb), clamped to 2^+-60 so that 1/s^2 stays finite
    s = __uint_as_float((unsigned)sb << 23);
    const float is = __uint_as_float((unsigned)(254 - sb) << 23);
    inv_s2 = is * is;
    mprime = __uint_as_float((unsigned)min(eb + 1, 254) << 23);
}

// hdr[0] = max |x| bits, one atomicMax per block.  hdr lives in a buffer of its own that is zeroed when allocated; every
// call leaves hdr[0] = 0 behind (l2_exact_rows_kernel, the last kernel of the chain) and its ticket hdr[2] self-cleans, so no
// memset sits in front of the chain.
__device__ __forceinline__ unsigned absmax_span(const float *__restrict__ x, size_t n, size_t tid, size_t stride, unsigned m) {
    if ((reinterpret_cast<uintptr_t>(x) & 15) == 0) {
        const size_t n4 = n >> 2;
        const uint4 *x4 = reinterpret_cast<const uint4 *>(x);
        for (size_t i = tid; i < n4; i += stride) {
            const uint4 v = __ldg(x4 + i);
            m = max(max(m, v.x & 0x7FFFFFFFu), max(max(v.y & 0x7FFFFFFFu, v.z & 0x7FFFFFFFu), v.w & 0x7FFFFFFFu));
        }
        for (size_t i = (n4 << 2) + tid; i < n; i += stride) m = max(m, __float_as_uint(__ldg(x + i)) & 0x7FFFFFFFu);
    } else {
        for (size_t i = tid; i < n; i += stride) m = max(m, __float_as_uint(__ldg(x + i)) & 0x7FFFFFFFu);
    }
    return m;
}
// block maximum, one atomicMax into hdr[0] (blockDim.x <= 256)
__device__ __forceinline__ void absmax_commit(unsigned m, unsigned *__restrict__ hdr) {
    m = __reduce_max_sync(0xffffffffu, m);
    __shared__ unsigned sm[8];
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < (int)(blockDim.x >> 5); w++) m = max(m, sm[w]);
        if (m) atomicMax(hdr, m);
    }
}
__global__ void __launch_bounds__(256) absmax_kernel(const float *__restrict__ q, size_t nq, const float *__restrict__ t, size_t nt,
                                                     unsigned *__restrict__ hdr) {
    pdl_trigger();
    if (blockIdx.x == 0 && threadIdx.x == 0) hdr[1] = 0;      // flagged-row count of this call (the refinement fills it)
    const size_t stride = (size_t)gridDim.x * blockDim.x, tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    absmax_commit(absmax_span(t, nt, tid, stride, absmax_span(q, nq, tid, stride, 0u)), hdr);
}

// One fp16 operand row: lane l holds components 4l .. 4l + 3 (Dp <= 128).  split16_load reads them (before the scale is
// known), split16_store writes [x16 (Dp) | norm chunk (64)] and returns the scaled |x|^2.
__device__ __forceinline__ void split16_load(const float *__restrict__ x, int dim, int dp, int lane, float (&v)[4]) {
    const bool vec = (dim & 3) == 0 && ((reinterpret_cast<uintptr_t>(x) & 15) == 0);
    v[0] = v[1] = v[2] = v[3] = 0.f;
    const int k = 4 * lane;
    if (k < dp) {
        if (vec && k + 3 < dim) {
            const float4 f = __ldg(reinterpret_cast<const float4 *>(x + k));
            v[0] = f.x; v[1] = f.y; v[2] = f.z; v[3] = f.w;
        } else {
#pragma unroll
            for (int e = 0; e < 4; e++) v[e] = k + e < dim ? __ldg(x + k + e) : 0.f;
        }
    }
}
__device__ __forceinline__ float split16_store(float (&v)[4], float s, int dp, int lane, bool train, __half *__restrict__ o) {
    const int k = 4 * lane;
    float acc = 0.f;
    if (k < dp) {
        __half2 h[2];
#pragma unroll
        for (int e = 0; e < 4; e++) v[e] *= s;
        h[0] = __floats2half2_rn(v[0], v[1]);
        h[1] = __floats2half2_rn(v[2], v[3]);
        *reinterpret_cast<uint2 *>(o + k) = make_uint2(*reinterpret_cast<uint32_t *>(&h[0]), *reinterpret_cast<uint32_t *>(&h[1]));
#pragma unroll
        for (int e = 0; e < 4; e++) acc = fmaf(v[e], v[e], acc);
    }
    for (int sh = 16; sh; sh >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, sh);
    const float hn = -0.5f * acc * (1.f / NORM_C);
    const __half e0 = __float2half_rn(hn);
    const float r1 = hn - __half2float(e0);
    const __half e1 = __float2half_rn(r1);
    const __half e2 = __float2half_rn(r1 - __half2float(e1));
    const __half cc = __float2half_rn(NORM_C), zero = __float2half_rn(0.f);
    const __half n0 = train ? cc : e0, n1v = train ? cc : e1, n2v = train ? cc : e2;
    const __half n3 = train ? e0 : cc, n4 = train ? e1 : cc, n5 = train ? e2 : cc;
    __half2 ext;
    ext.x = lane == 0 ? n0 : lane == 1 ? n2v : lane == 2 ? n4 : zero;
    ext.y = lane == 0 ? n1v : lane == 1 ? n3 : lane == 2 ? n5 : zero;
    *reinterpret_cast<__half2 *>(o + dp + 2 * lane) = ext;
    return acc;
}

// Row layout in fp16 mode: [x16 (Dp) | norm chunk (64)].  One warp per row, as split_kernel.
__global__ void __launch_bounds__(256) split16_kernel(const float *__restrict__ q, int n1, const float *__restrict__ t, int n2,
                                                      int dim, int dp, __half *__restrict__ a, __half *__restrict__ b,
                                                      int32_t *__restrict__ cand_j, int slots, const unsigned *__restrict__ hdr,
                                                      float *__restrict__ qnorm, float *__restrict__ cand_drop) {
    const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    pdl_trigger();
    if (w >= n1 + n2) return;
    const bool train = w >= n1;
    const int row = train ? w - n1 : w;
    if (!train)
    {
        for (int e = lane; e < slots * CAND; e += 32) cand_j[((size_t)(e / CAND) * n1 + row) * CAND + (e % CAND)] = -1;
        for (int e = lane; e < slots * EPI_GROUPS; e += 32)
            cand_drop[((size_t)(e / EPI_GROUPS) * n1 + row) * EPI_GROUPS + (e % EPI_GROUPS)] = 3.4e38f;
    }
    const float *x = (train ? t : q) + (size_t)row * dim;
    __half *o = (train ? b : a) + (size_t)row * (dp + CHUNK_K);
    float v[4];
    split16_load(x, dim, dp, lane, v);
    pdl_wait();                                      // the scale comes from absmax_kernel
    float s, inv_s2, mprime;
    l2_scale_from_bits(__ldcg(hdr), s, inv_s2, mprime);
    const float acc = split16_store(v, s, dp, lane, train, o);
    if (!train && lane == 0) qnorm[row] = acc;       // scaled, like the accumulator
}

// ---- the GEMM + top-8 kernel ----------------------------------------------------------------
struct L2BPair;
struct L2Params {
    int n1, n2, dpc;               // dpc = Dp / 64: chunks per operand part (hi or lo)
    int tiles_per_split;           // single-CTA kernel: column tiles handled by one blockIdx.y
    int col_tiles, items;          // pair kernel: column tiles per row pair, row pairs x column tiles
    uint32_t key_mask;             // 0x7FFFFFE0, passed as data so that (acc & mask) | column is ONE LOP3
    const unsigned *absmax_bits;   // pair kernel (fp16): bit pattern of max |x| over both operand sets (the scale derives from it)
    float band_rel, band_abs_sqrt, band_abs_const;   // error band of one accumulator comparison (see RowTop)
    const float *qnorm;            // [n1] |q|^2 in the accumulator's units (written by the split kernel)
    float *cand_drop;              // [splits][n1][EPI_GROUPS] approximate distance of a FULL list's last entry (3.4e38: list not full)
    int32_t *cand_j;               // [splits][n1][CAND]
    float *cand_d;                 // [splits][n1][CAND] approximate distances (diagnostic)
    float *dbg_dist;               // optional [n1][n2] approximate distance matrix (tests)
    unsigned long long *timeline;  // optional (PGM_L2_TIMELINE=1): %globaltimer stamps of cluster 0's leader CTA
    // many pairs (l2_topk_pair_kernel<DBG, true>): the items of pair k are [item_base[k], item_base[k + 1]), the
    // candidate lists have `rows` (the chunk's query rows) rows per slot
    const L2BPair *bpairs;
    const int32_t *item_base;
    int n_pairs, rows;
};
// One pair of a batched chunk (pgm_knn2_l2_pairs_batch_dev).  Pairs without query rows are not in the plan.
struct L2BPair {
    int64_t q_row, t_row;          // first row of the query / train image in the caller's descriptor array
    int64_t out_row;               // first result row: the caller's output arrays (knn2) or the chunk's knn2 scratch
    int32_t a_row, b_row;          // first row of the query / train image in the chunk's A' / B' operands
    int32_t n1, n2;
    int32_t row0;                  // first query row of the chunk: candidate lists, flagged-row ids
    int32_t item0, col_tiles;      // first GEMM item; column tiles (0 when n2 = 0: such a pair has no GEMM item)
    int32_t pad;
};
// One image of a chunk converted into fp16 operand rows: once per role (query form into A', train form into B').
struct L2BImage {
    int64_t src_row;               // first row in the caller's descriptor array
    int32_t dst_row, n;            // first operand row, rows
    int32_t train, pad;
};
// Largest k with base[k] <= g (base is an exclusive prefix over n entries, base[n] = total).
__device__ __forceinline__ int l2_find(const int32_t *__restrict__ base, int n, int g) {
    int lo = 0, hi = n;
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (__ldg(base + mid) <= g) lo = mid; else hi = mid;
    }
    return lo;
}
__device__ __forceinline__ void l2_stamp(const L2Params &p, int slot) {
    if (p.timeline && blockIdx.x == 0 && blockIdx.y == 0) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        p.timeline[slot] = t;
        p.timeline[128 + slot] = (unsigned long long)clock64();
    }
}

// Epilogue reducer shared by both kernels.  The accumulator holds -d/2 (see the header); one query row per thread.
//
// Hot path, per 32 accumulator columns: a float max tree (3-input FMNMX, half an instruction per element) and ONE
// compare against the row's trigger level -- nothing else.  Only a chunk holding a column that can still matter takes
// the slow path, which rebuilds tagged integer keys (|acc| bits with the column-in-chunk in the 5 low mantissa bits,
// one LOP3 per element; the 2^-18 relative perturbation only affects ranking) and inserts into the row's sorted
// top-K list.
//
// "Can still matter": the refinement only ever needs the columns whose approximate distance lies within the ranking's
// error band of the SECOND best one (pgm_l2.cuh header).  The band of the current second best only shrinks as the
// stream goes on, so a column outside it now is outside it at the end: trigger level = min(K-th best key, second best
// + band).  That makes the slow path rare (about 3 ln n visits per row instead of K ln n) without weakening what the
// lists certify.  A column that a FULL list turned away or evicted has a key >= the list's final last entry, which is
// what the refinement's certificate looks at (cand_drop).
//
// Rows that do not exist never trigger (trigger level +inf); columns >= n2 (zero rows from the TMA's out-of-bounds
// fill) are skipped on insertion.
struct RowTop {
    uint32_t bk[TOPK];     // ascending keys, index bits cleared; 0xFFFFFFFF = empty
    int bj[TOPK];
    uint32_t thr_key;      // slow-path insertion bound (tagged keys below it are inserted)
    float thr_acc;         // hot-path trigger: some accumulator of the chunk > thr_acc
    float qn3;             // 3 |q|^2 in the accumulator's units (scaled in fp16 mode)
};
struct BandParams { float rel, abs_sqrt, abs_const; };   // band of an accumulator a: rel (3|q|^2 + 4|a|) + abs_sqrt sqrt(.) + abs_const

__device__ __forceinline__ void rowtop_reset(RowTop &r, bool exists, float qn) {
#pragma unroll
    for (int k = 0; k < TOPK; k++) { r.bk[k] = 0xFFFFFFFFu; r.bj[k] = -1; }
    r.thr_key = exists ? 0xFFFFFFFFu : 0u;
    r.thr_acc = exists ? -__int_as_float(0x7F800000) : __int_as_float(0x7F800000);
    r.qn3 = 3.f * qn;
}
__device__ __forceinline__ void rowtop_update_trigger(RowTop &r, const BandParams &bp) {
    uint32_t tk = r.bk[TOPK - 1];
    if (r.bk[1] != 0xFFFFFFFFu) {
        const float a2 = __uint_as_float(r.bk[1]);
        const float span = r.qn3 + 4.f * a2;
        const float lim = a2 + bp.rel * span + bp.abs_sqrt * sqrtf(span) + bp.abs_const;
        tk = min(tk, (__float_as_uint(lim) + 64u) & 0xFFFFFFE0u);
        r.thr_key = tk;
        r.thr_acc = -__uint_as_float(tk);
    }
}
__device__ __forceinline__ float fmax3(float a, float b, float c) {
    float d;
    asm("max.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
    return d;
}
template <int NCOLS, bool DBG>
__device__ __forceinline__ void epilogue_reduce(uint32_t taddr, int jbase, int n2, uint32_t mask, RowTop &r, const BandParams &bp,
                                                float *dbg_row, float dbg_scale) {
    uint32_t va[32], vb[32];
    constexpr int GROUPS = NCOLS / 32;
    tc_ld_32x32b_x32(taddr, va);
#pragma unroll
    for (int g = 0; g < GROUPS; g++) {
        uint32_t (&v)[32] = (g & 1) ? vb : va;
        tc_wait_ld();
        if (g + 1 < GROUPS) tc_ld_32x32b_x32(taddr + (uint32_t)((g + 1) * 32), (g & 1) ? va : vb);
        const int jg = jbase + g * 32;
        if (DBG && dbg_row) {
#pragma unroll
            for (int c = 0; c < 32; c++)
                if (jg + c < n2) dbg_row[jg + c] = dbg_scale * __uint_as_float(v[c] & 0x7FFFFFE0u);
        }
        float m0 = fmax3(__uint_as_float(v[0]), __uint_as_float(v[1]), __uint_as_float(v[2]));
        float m1 = fmax3(__uint_as_float(v[3]), __uint_as_float(v[4]), __uint_as_float(v[5]));
        float m2 = fmax3(__uint_as_float(v[6]), __uint_as_float(v[7]), __uint_as_float(v[8]));
        float m3 = fmax3(__uint_as_float(v[9]), __uint_as_float(v[10]), __uint_as_float(v[11]));
#pragma unroll
        for (int c = 12; c < 28; c += 8) {
            m0 = fmax3(m0, __uint_as_float(v[c]), __uint_as_float(v[c + 1]));
            m1 = fmax3(m1, __uint_as_float(v[c + 2]), __uint_as_float(v[c + 3]));
            m2 = fmax3(m2, __uint_as_float(v[c + 4]), __uint_as_float(v[c + 5]));
            m3 = fmax3(m3, __uint_as_float(v[c + 6]), __uint_as_float(v[c + 7]));
        }
        m0 = fmax3(m0, __uint_as_float(v[28]), __uint_as_float(v[29]));
        m1 = fmax3(m1, __uint_as_float(v[30]), __uint_as_float(v[31]));
        const float mx = fmaxf(fmax3(m0, m1, m2), m3);
        if (mx > r.thr_acc) {
            // tagged keys of the chunk, then the sorted insertion (usually one iteration)
            uint32_t key[32];
#pragma unroll
            for (int c = 0; c < 32; c++) key[c] = (v[c] & mask) | (uint32_t)c;
            uint32_t k0 = key[0], k1 = key[1], k2 = key[2], k3 = key[3];
#pragma unroll
            for (int c = 4; c < 32; c += 4) {
                k0 = min(k0, key[c]); k1 = min(k1, key[c + 1]); k2 = min(k2, key[c + 2]); k3 = min(k3, key[c + 3]);
            }
            uint32_t kmin = min(min(k0, k1), min(k2, k3));
            while (kmin < r.thr_key) {
                const int j = jg + (int)(kmin & 31u);
                if (j < n2) {
                    r.bk[TOPK - 1] = kmin & 0xFFFFFFE0u; r.bj[TOPK - 1] = j;
#pragma unroll
                    for (int k = TOPK - 1; k > 0; k--)
                        if (r.bk[k] < r.bk[k - 1]) {
                            const uint32_t tk = r.bk[k]; r.bk[k] = r.bk[k - 1]; r.bk[k - 1] = tk;
                            const int tj = r.bj[k]; r.bj[k] = r.bj[k - 1]; r.bj[k - 1] = tj;
                        }
                    rowtop_update_trigger(r, bp);
                }
                // next key strictly above the one just taken: keys at or below it wrap to >= 2^31 under the
                // unsigned subtraction (all keys are < 2^31), so one add+min per element finds it
                const uint32_t k1p = kmin + 1u;
                uint32_t d0 = 0xFFFFFFFFu, d1 = 0xFFFFFFFFu, d2 = 0xFFFFFFFFu, d3 = 0xFFFFFFFFu;
#pragma unroll
                for (int c = 0; c < 32; c += 4) {
                    d0 = min(d0, key[c] - k1p); d1 = min(d1, key[c + 1] - k1p); d2 = min(d2, key[c + 2] - k1p); d3 = min(d3, key[c + 3] - k1p);
                }
                const uint32_t dlt = min(min(d0, d1), min(d2, d3));
                if (dlt >= 0x80000000u) break;
                kmin = k1p + dlt;
            }
        }
    }
}

template <bool DBG>
__global__ void __launch_bounds__(THREADS, 1)
l2_topk_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b, L2Params p) {
    extern __shared__ unsigned char smem_raw[];
    // SWIZZLE_128B atoms need 1024-byte alignment: align the dynamic window by hand (1 KB of slack is allocated)
    unsigned char *smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    // layout: A' chunks | B' stages | barriers
    unsigned char *sa = smem;
    unsigned char *sb = smem + (size_t)MAX_CHUNKS * CHUNK_BYTES;
    uint64_t *bars = reinterpret_cast<uint64_t *>(sb + (size_t)STAGES * CHUNK_BYTES);
    uint64_t *full = bars, *empty = bars + STAGES, *a_bar = bars + 2 * STAGES;
    uint64_t *tfull = bars + 2 * STAGES + 1, *tempty = bars + 2 * STAGES + 3;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 2 * STAGES + 5);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int m0 = blockIdx.x * TILE_M;
    const int n_col_tiles = (p.n2 + TILE_N - 1) / TILE_N;
    const int ct0 = blockIdx.y * p.tiles_per_split, ct1 = min(n_col_tiles, ct0 + p.tiles_per_split);
    const int ntiles = max(ct1 - ct0, 0);

    if (warp == 1 && lane == 0) {
        for (int s = 0; s < STAGES; s++) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        mbar_init(a_bar, 1);
        for (int a = 0; a < 2; a++) { mbar_init(&tfull[a], 1); mbar_init(&tempty[a], 4 * EPI_GROUPS); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    pdl_wait();                                      // operands are written by split_kernel

    if (warp == 0 && lane == 0) {
        // ===== TMA producer =====
        const int nch = 2 * p.dpc + 1;                    // hi chunks, lo chunks, norm chunk
        mbar_expect_tx(a_bar, (uint32_t)nch * CHUNK_BYTES);
        for (int kc = 0; kc < nch; kc++) tma_load_2d(sa + (size_t)kc * CHUNK_BYTES, &map_a, a_bar, kc * CHUNK_K, m0);
        int s = 0; uint32_t ph = 0;
        for (int t = 0; t < ntiles; t++) {
            for (int kc = 0; kc < nch; kc++) {               // t_hi chunks, t_lo chunks, norm chunk
                mbar_wait(&empty[s], ph ^ 1);
                mbar_expect_tx(&full[s], CHUNK_BYTES);
                tma_load_2d(sb + (size_t)s * CHUNK_BYTES, &map_b, &full[s], kc * CHUNK_K, (ct0 + t) * TILE_N);
                if (++s == STAGES) { s = 0; ph ^= 1; }
            }
        }
    } else if (warp == 1 && lane == 0) {
        // ===== MMA issuer =====
        mbar_wait(a_bar, 0);
        const int dpc = p.dpc;
        uint32_t g = 0;                                         // running chunk-slot counter of the B' ring
        for (int t = 0; t < ntiles; t++) {
            const int acc = t & 1;
            mbar_wait(&tempty[acc], ((t >> 1) & 1) ^ 1);       // epilogue drained this accumulator
            tc_fence_after();
            const uint32_t d_tmem = tmem_base + (uint32_t)acc * TILE_N;
            // pass 0: q_hi . t_hi (waits for the hi slots), pass 1: q_lo . t_hi (frees them), pass 2: q_hi . t_lo
            for (int pass = 0; pass < 3; pass++) {
                for (int c = 0; c < dpc; c++) {
                    const uint32_t i = g + (uint32_t)(pass == 2 ? dpc + c : c), s = i % STAGES, ph = (i / STAGES) & 1u;
                    if (pass != 1) { mbar_wait(&full[s], ph); tc_fence_after(); }
                    const int ac = pass == 1 ? dpc + c : c;
                    const uint64_t adesc = umma_desc_sw128(smem_u32(sa + (size_t)ac * CHUNK_BYTES));
                    const uint64_t bdesc = umma_desc_sw128(smem_u32(sb + (size_t)s * CHUNK_BYTES));
#pragma unroll
                    for (int k = 0; k < CHUNK_K / UMMA_K; k++)     // +32 B per K step inside the 128-B swizzle row
                        tc_mma_bf16(d_tmem, adesc + (uint64_t)(k * 2), bdesc + (uint64_t)(k * 2), IDESC_BF16_M128_N128,
                                    (uint32_t)((pass | c | k) != 0));
                    if (pass != 0) tc_commit(&empty[s]);            // slot reusable once these MMAs retire
                }
            }
            {   // norm chunk: one K = 16 step adds -(||q||^2 + ||t||^2) / 2
                const uint32_t i = g + 2u * (uint32_t)dpc, s = i % STAGES, ph = (i / STAGES) & 1u;
                mbar_wait(&full[s], ph); tc_fence_after();
                tc_mma_bf16(d_tmem, umma_desc_sw128(smem_u32(sa + (size_t)(2 * dpc) * CHUNK_BYTES)),
                            umma_desc_sw128(smem_u32(sb + (size_t)s * CHUNK_BYTES)), IDESC_BF16_M128_N128, 1u);
                tc_commit(&empty[s]);
            }
            g += 2u * (uint32_t)dpc + 1u;
            tc_commit(&tfull[acc]);                             // accumulator complete
        }
    } else if (warp >= 4) {
        // ===== epilogue: one query row per thread =====
        const int ew = warp & 3;                                // the TMEM lane quarter this warp may read (warp % 4)
        const int eg = (warp - 4) >> 2;                         // which half of the accumulator's columns
        const int row = m0 + ew * 32 + lane;
        RowTop rt;
        const BandParams bp{p.band_rel, p.band_abs_sqrt, p.band_abs_const};
        rowtop_reset(rt, row < p.n1, row < p.n1 ? __ldcg(p.qnorm + row) : 0.f);
        constexpr int NCOLS = TILE_N / EPI_GROUPS;
        for (int t = 0; t < ntiles; t++) {
            const int acc = t & 1;
            mbar_wait(&tfull[acc], (t >> 1) & 1);
            tc_fence_after();
            const int jbase = (ct0 + t) * TILE_N + eg * NCOLS;
            const uint32_t taddr = tmem_base + ((uint32_t)(ew * 32) << 16) + (uint32_t)(acc * TILE_N + eg * NCOLS);
            epilogue_reduce<NCOLS, DBG>(taddr, jbase, p.n2, p.key_mask, rt, bp,
                                        DBG && p.dbg_dist && row < p.n1 ? p.dbg_dist + (size_t)row * p.n2 : nullptr, 2.f);
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tempty[acc]);
        }
        if (row < p.n1) {
            const size_t o = ((size_t)blockIdx.y * p.n1 + row) * CAND + (size_t)eg * TOPK;
#pragma unroll
            for (int k = 0; k < TOPK; k++) {
                p.cand_j[o + k] = rt.bk[k] != 0xFFFFFFFFu ? rt.bj[k] : -1;
                p.cand_d[o + k] = rt.bk[k] != 0xFFFFFFFFu ? 2.f * __uint_as_float(rt.bk[k]) : 3.4e38f;
            }
            p.cand_drop[((size_t)blockIdx.y * p.n1 + row) * EPI_GROUPS + eg] =
                rt.bk[TOPK - 1] != 0xFFFFFFFFu ? 2.f * __uint_as_float(rt.bk[TOPK - 1]) : 3.4e38f;
        }
    }
    pdl_trigger();                                   // the refinement kernel may be scheduled
    tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
    }
}

// ---- the same contraction on CTA pairs (cta_group::2) --------------------------------------------
// Why: with M = 128 per CTA every byte of the streamed B' tile is written to shared memory once (TMA)
// and read once per MMA while A' is re-read by every MMA -- 192 B/clk of shared-memory traffic per SM
// against 128 B/clk available, so the single-CTA kernel saturates shared memory at ~0.55 of the tensor
// peak.  A CTA pair (two SMs of one TPC, cluster 2x1x1) runs ONE tcgen05.mma.cta_group::2 of
// M = 256 (128 query rows per CTA) x N = 256: each CTA stages only HALF of every B' tile (128 train
// rows), the tensor cores of both SMs read both halves, and the per-SM shared-memory traffic drops to
// ~96 B/clk.  TMEM: two accumulators of 256 fp32 columns (all 512 columns).
//
//   both CTAs   warp 0: TMA producer for its own A' rows and its half of each B' tile; completions are
//               counted on the LEADER's (rank 0) full barriers
//   leader      warp 1: issues the MMAs; tcgen05.commit.multicast arrives on both CTAs' barriers
//   both CTAs   warps 4-11: epilogue over the CTA's own 128 rows x 256 columns (TMEM is per SM);
//               accumulator release arrives on the leader's tempty barrier (remote arrive for rank 1)
constexpr int TILE_N2 = 256;                  // train rows per accumulator in pair mode (half per CTA)
constexpr uint32_t TMEM_COLS2 = 512;
constexpr int NACC2 = 512 / TILE_N2;          // accumulators in flight: all 512 TMEM columns
constexpr int B_ROWS2 = TILE_N2 / 2;          // train rows each CTA stages per tile
constexpr uint32_t B_CHUNK_BYTES2 = B_ROWS2 * CHUNK_K * 2;
constexpr int STAGES2 = (int)((size_t)STAGES * CHUNK_BYTES / B_CHUNK_BYTES2);   // same 128 KB ring
static_assert(TILE_N2 == 256, "pair tile width");
// f32 accumulator (bit 4), A and B format F16 (0 in bits 7-9 and 10-12), N = TILE_N2, M = 256
constexpr uint32_t IDESC_F16_M256_N2 = (1u << 4) | ((uint32_t)(TILE_N2 >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);
constexpr uint32_t PEER_BIT_MASK = 0xFEFFFFFFu;   // shared::cluster address of the same offset in the pair's even CTA

__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// TMA load whose completion bytes are accounted on the leader CTA's barrier (issued by both CTAs)
__device__ __forceinline__ void tma_load_2d_pair(void *smem_dst, const CUtensorMap *map, uint64_t *bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(map), "r"(smem_u32(bar) & PEER_BIT_MASK), "r"(c0), "r"(c1) : "memory");
}
// arrive on the barrier at the same offset in CTA `rank` of the cluster
__device__ __forceinline__ void mbar_arrive_remote(uint64_t *bar, uint32_t rank) {
    asm volatile(
        "{\n\t.reg .b32 ra;\n\t"
        "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
        "mbarrier.arrive.shared::cluster.b64 _, [ra];\n\t}"
        ::"r"(smem_u32(bar)), "r"(rank) : "memory");
}
__device__ __forceinline__ void tc_commit_pair(uint64_t *bar) {      // arrives on both CTAs' barrier at this offset
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(smem_u32(bar)), "h"((uint16_t)3) : "memory");
}
__device__ __forceinline__ void tc_mma_bf16_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}

// Work distribution: the (row pair, column tile) items are flattened row-major and cut into gridDim.x / 2
// contiguous, equally long segments, one per cluster (persistent: as many clusters as are co-resident) -- no wave
// quantisation.  A segment that crosses into the next row pair reloads A' (after the MMAs of the old rows have
// retired) and its epilogue flushes the finished rows' candidates; a row pair's candidates therefore arrive
// from several segments, each writing its own slot (segment index minus the index of the first segment that
// touches the row pair).  Unused slots keep the -1 the split kernel wrote.
__device__ __forceinline__ int l2_segment_start(int k, int items, int clusters) {
    return (int)(((long long)k * items) / clusters);
}
__device__ __forceinline__ int l2_segment_of_item(int x, int items, int clusters) {      // max k with start(k) <= x
    return (int)((((long long)x + 1) * clusters - 1) / items);
}

// One work item decoded: its row pair (identified by the item that starts it), column tile and pair.  With BATCH the
// items of the chunk's pairs are concatenated (pair-major, then row pair, then column tile); the cursor `pp` only moves
// forward, as the roles walk their segment in order.
struct L2Item {
    int first, ct, col_tiles;      // first item of the row pair, column tile, column tiles of the pair
    int m0;                        // the row pair's first query row (pair-local)
    int n1, n2, a_row, b_row, row0;
};
template <bool BATCH>
__device__ __forceinline__ void l2_item(const L2Params &p, int it, int &pp, L2Item &x) {
    if constexpr (BATCH) {
        while (it >= __ldg(p.item_base + pp + 1)) pp++;
        PGM_ASSERT(pp >= 0 && pp < p.n_pairs);
        const L2BPair *b = p.bpairs + pp;
        const int i0 = __ldg(&b->item0), ct_n = __ldg(&b->col_tiles);
        PGM_ASSERT(ct_n > 0 && it >= i0);
        const int rp = (it - i0) / ct_n;
        x.ct = it - i0 - rp * ct_n; x.first = i0 + rp * ct_n; x.col_tiles = ct_n; x.m0 = 2 * rp * TILE_M;
        x.n1 = __ldg(&b->n1); x.n2 = __ldg(&b->n2); x.a_row = __ldg(&b->a_row); x.b_row = __ldg(&b->b_row);
        x.row0 = __ldg(&b->row0);
    } else {
        const int rp = it / p.col_tiles;
        x.ct = it - rp * p.col_tiles; x.first = rp * p.col_tiles; x.col_tiles = p.col_tiles; x.m0 = 2 * rp * TILE_M;
        x.n1 = p.n1; x.n2 = p.n2; x.a_row = 0; x.b_row = 0; x.row0 = 0;
    }
}

// BATCH: many pairs in one launch (pgm_knn2_l2_pairs_batch_dev).  A' / B' hold every image of the chunk once; a tile's
// TMA rows are the pair's first operand row plus the tile offset, so rows past the end of an image are the NEXT image's
// rows, not zeros: query rows >= n1 do not exist (never trigger, never flushed) and columns >= n2 are masked by
// epilogue_reduce.  Candidate lists are indexed by the chunk's query row (row0 + local row), `rows` of them per slot.
template <bool DBG, bool BATCH>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(THREADS, 1)
l2_topk_pair_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b, L2Params p) {
    extern __shared__ unsigned char smem_raw[];
    unsigned char *smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    unsigned char *sa = smem;                                              // A' chunks of this CTA's 128 rows
    unsigned char *sb = smem + (size_t)MAX_CHUNKS * CHUNK_BYTES;           // this CTA's half of the B' stages
    uint64_t *bars = reinterpret_cast<uint64_t *>(sb + (size_t)STAGES2 * B_CHUNK_BYTES2);
    uint64_t *full = bars, *empty = bars + STAGES2, *a_bar = bars + 2 * STAGES2;
    uint64_t *tfull = bars + 2 * STAGES2 + 1, *tempty = tfull + NACC2;
    uint64_t *a_empty = tempty + NACC2;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(a_empty + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();
    const bool leader = rank == 0;
    const int clusters = (int)(gridDim.x >> 1), cid = (int)(blockIdx.x >> 1);
    const int items = p.items;
    const int it0 = l2_segment_start(cid, items, clusters), it1 = l2_segment_start(cid + 1, items, clusters);
    const int cand_rows = BATCH ? p.rows : p.n1;
    int pp = BATCH && it0 < it1 ? l2_find(p.item_base, p.n_pairs, it0) : 0;     // pair cursor of this thread's role
    if (threadIdx.x == 0) l2_stamp(p, 0);

    if (warp == 1 && lane == 0) {
        for (int s = 0; s < STAGES2; s++) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        mbar_init(a_bar, 1);
        mbar_init(a_empty, 1);
        for (int a = 0; a < NACC2; a++) { mbar_init(&tfull[a], 1); mbar_init(&tempty[a], 2 * 4 * EPI_GROUPS); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(TMEM_COLS2) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    cluster_sync_all();                       // barriers of both CTAs initialised before any remote arrive / TMA
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    if (threadIdx.x == 0) l2_stamp(p, 1);
    pdl_wait();                                      // operands are written by split_kernel
    if (threadIdx.x == 0) l2_stamp(p, 2);

    if (warp == 0 && lane == 0) {
        // ===== TMA producer (both CTAs): own A' rows, own half of every B' tile =====
        const int nch = p.dpc + 1;                        // x16 chunks, norm chunk
        int s = 0; uint32_t ph = 0;
        int cur_rp = -1; uint32_t n_a = 0;
        for (int it = it0; it < it1; it++) {
            L2Item x;
            l2_item<BATCH>(p, it, pp, x);
            const int m0 = x.a_row + x.m0 + (int)rank * TILE_M;
            if (x.first != cur_rp && cur_rp < 0) {             // first rows of the segment: A' first
                if (leader) mbar_expect_tx(a_bar, 2u * (uint32_t)nch * CHUNK_BYTES);
                for (int kc = 0; kc < nch; kc++) tma_load_2d_pair(sa + (size_t)kc * CHUNK_BYTES, &map_a, a_bar, kc * CHUNK_K, m0);
                cur_rp = x.first; n_a++;
            }
            for (int kc = 0; kc < nch; kc++) {                 // t16 chunks, norm chunk
                mbar_wait(&empty[s], ph ^ 1);                  // the pair's MMAs no longer read this stage (multicast commit)
                if (leader) mbar_expect_tx(&full[s], 2u * B_CHUNK_BYTES2);
                tma_load_2d_pair(sb + (size_t)s * B_CHUNK_BYTES2, &map_b, &full[s], kc * CHUNK_K,
                                 x.b_row + x.ct * TILE_N2 + (int)rank * B_ROWS2);
                if (++s == STAGES2) { s = 0; ph ^= 1; }
            }
            if (x.first != cur_rp) {
                // next row pair: its first B' tile is already on its way into the ring (the slots free up while the
                // old rows' last MMAs run); A' can only be replaced once those MMAs have retired
                mbar_wait(a_empty, (n_a - 1u) & 1u);
                if (leader) mbar_expect_tx(a_bar, 2u * (uint32_t)nch * CHUNK_BYTES);
                for (int kc = 0; kc < nch; kc++) tma_load_2d_pair(sa + (size_t)kc * CHUNK_BYTES, &map_a, a_bar, kc * CHUNK_K, m0);
                cur_rp = x.first; n_a++;
            }
        }
    } else if (warp == 1 && lane == 0 && leader) {
        // ===== MMA issuer (leader only) =====
        const int dpc = p.dpc;
        uint32_t g = 0;                                         // running chunk-slot counter of the B' ring
        int cur_rp = -1; uint32_t n_a = 0;
        for (int it = it0; it < it1; it++) {
            L2Item x;
            l2_item<BATCH>(p, it, pp, x);
            const int t = it - it0;
            if (x.first != cur_rp) { mbar_wait(a_bar, n_a & 1u); tc_fence_after(); cur_rp = x.first; n_a++; l2_stamp(p, 3); }
            const int acc = t % NACC2;
            mbar_wait(&tempty[acc], ((t / NACC2) & 1) ^ 1);    // both CTAs' epilogues drained this accumulator
            tc_fence_after();
            if (t < 36) l2_stamp(p, 4 + t);
            const uint32_t d_tmem = tmem_base + (uint32_t)acc * TILE_N2;
            for (int c = 0; c < dpc; c++) {
                const uint32_t i = g + (uint32_t)c, s = i % STAGES2, ph = (i / STAGES2) & 1u;
                mbar_wait(&full[s], ph); tc_fence_after();
                const uint64_t adesc = umma_desc_sw128(smem_u32(sa + (size_t)c * CHUNK_BYTES));
                const uint64_t bdesc = umma_desc_sw128(smem_u32(sb + (size_t)s * B_CHUNK_BYTES2));
#pragma unroll
                for (int k = 0; k < CHUNK_K / UMMA_K; k++)
                    tc_mma_bf16_pair(d_tmem, adesc + (uint64_t)(k * 2), bdesc + (uint64_t)(k * 2), IDESC_F16_M256_N2,
                                     (uint32_t)((c | k) != 0));
                tc_commit_pair(&empty[s]);
            }
            {   // norm chunk: one K = 16 step adds -(||q||^2 + ||t||^2) / 2
                const uint32_t i = g + (uint32_t)dpc, s = i % STAGES2, ph = (i / STAGES2) & 1u;
                mbar_wait(&full[s], ph); tc_fence_after();
                tc_mma_bf16_pair(d_tmem, umma_desc_sw128(smem_u32(sa + (size_t)dpc * CHUNK_BYTES)),
                                 umma_desc_sw128(smem_u32(sb + (size_t)s * B_CHUNK_BYTES2)), IDESC_F16_M256_N2, 1u);
                tc_commit_pair(&empty[s]);
            }
            g += (uint32_t)dpc + 1u;
            tc_commit_pair(&tfull[acc]);
            if (it + 1 < it1 && it + 1 - x.first >= x.col_tiles) tc_commit_pair(a_empty);   // A' may be overwritten once these retire
        }
    } else if (warp >= 4) {
        // ===== epilogue: one query row per thread, this CTA's 128 rows x 256 columns =====
        const int ew = warp & 3;
        const int eg = (warp - 4) >> 2;
        RowTop rt;
        const BandParams bp{p.band_rel, p.band_abs_sqrt, p.band_abs_const};
        constexpr int NCOLS = TILE_N2 / EPI_GROUPS;
        int cur_rp = -1, row = 0, n1 = 0, crow = 0;             // crow: the row's candidate-list row
        float s_, is2, mp;                                      // accumulator -> distance: -2 / s^2
        l2_scale_from_bits(__ldcg(p.absmax_bits), s_, is2, mp);
        const float out_scale = 2.f * is2;
        auto flush = [&]() {
            if (cur_rp < 0 || row >= n1) return;
            const int slot = cid - l2_segment_of_item(cur_rp, items, clusters);
            const size_t o = ((size_t)slot * cand_rows + crow) * CAND + (size_t)eg * TOPK;
#pragma unroll
            for (int k = 0; k < TOPK; k++) {
                p.cand_j[o + k] = rt.bk[k] != 0xFFFFFFFFu ? rt.bj[k] : -1;
                p.cand_d[o + k] = rt.bk[k] != 0xFFFFFFFFu ? out_scale * __uint_as_float(rt.bk[k]) : 3.4e38f;
            }
            p.cand_drop[((size_t)slot * cand_rows + crow) * EPI_GROUPS + eg] =
                rt.bk[TOPK - 1] != 0xFFFFFFFFu ? out_scale * __uint_as_float(rt.bk[TOPK - 1]) : 3.4e38f;
        };
        for (int it = it0; it < it1; it++) {
            L2Item x;
            l2_item<BATCH>(p, it, pp, x);
            const int t = it - it0;
            if (x.first != cur_rp) {
                flush();
                cur_rp = x.first; n1 = x.n1;
                row = x.m0 + (int)rank * TILE_M + ew * 32 + lane;
                crow = x.row0 + row;
                rowtop_reset(rt, row < n1, row < n1 ? __ldcg(p.qnorm + x.a_row + row) : 0.f);
            }
            const int acc = t % NACC2;
            mbar_wait(&tfull[acc], (t / NACC2) & 1);
            tc_fence_after();
            if (warp == 4 && lane == 0 && t < 36) l2_stamp(p, 40 + t);
            const int jbase = x.ct * TILE_N2 + eg * NCOLS;
            const uint32_t taddr = tmem_base + ((uint32_t)(ew * 32) << 16) + (uint32_t)(acc * TILE_N2 + eg * NCOLS);
            epilogue_reduce<NCOLS, DBG>(taddr, jbase, x.n2, p.key_mask, rt, bp,
                                        DBG && p.dbg_dist && row < n1 ? p.dbg_dist + (size_t)row * p.n2 : nullptr, out_scale);
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_remote(&tempty[acc], 0);      // the leader's barrier counts both CTAs' warps
            if (warp == 4 && lane == 0 && t < 36) l2_stamp(p, 80 + t);
        }
        flush();
        if (warp == 4 && lane == 0) l2_stamp(p, 120);
    }
    pdl_trigger();                                   // the refinement kernel may be scheduled
    __syncwarp();
    tc_fence_before();
    cluster_sync_all();                       // neither CTA leaves (or frees TMEM) while its partner may still use it
    if (threadIdx.x == 0) l2_stamp(p, 121);
    if (warp == 2) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS2) : "memory");
    }
}

inline size_t l2_pair_smem_bytes() {
    return (size_t)MAX_CHUNKS * CHUNK_BYTES + (size_t)STAGES2 * B_CHUNK_BYTES2 + (2 * STAGES2 + 2 * NACC2 + 4) * 8 + 1024;
}

inline size_t l2_smem_bytes() {
    return (size_t)(MAX_CHUNKS + STAGES) * CHUNK_BYTES + (2 * STAGES + 7) * 8 + 1024;
}

// ---- refinement: exact fp32 distances of the candidates, best / second by (distance, index) ----
// One warp per query.  Step 1 prunes with the approximate distances the GEMM kernel left in cand_d: a
// candidate whose approximate distance exceeds the second-smallest one by more than the error bound of
// the two approximations cannot be among the exact top two, so its train row is never read (typically 2-4
// of the 8 x splits candidates survive; the gather of 512-byte train rows is what this kernel costs).
// Error bound: |approx - exact| <= 2^-14.5 (|q|^2 + |t|^2) worst case (bf16 hi/lo residuals 2^-15.7 |q||t|,
// fp32 accumulation over K' = 272, the key's 5 dropped mantissa bits); |t|^2 <= 2|q|^2 + 2d, hence the slack
// 2^-12 (3|q|^2 + 2 d_approx) covers both approximations with a factor 2.8 to spare.
// Step 2: the survivors four at a time, so sixteen independent train-row loads are in flight per lane.
// Summation order per distance: each lane's strided partial sum, then a butterfly.
// One warp refines candidate-list row i (n1 rows per slot) of the query q (one row); the results go to element o of the
// output arrays, an uncertified row is flagged as i.
__device__ __forceinline__ void l2_refine_row(const float *__restrict__ q, const float *__restrict__ t, int n2, int dim,
                                              const int32_t *__restrict__ cand_j, const float *__restrict__ cand_d,
                                              const float *__restrict__ cand_drop, int splits, int n1, int i, size_t o_out,
                                              int32_t *best_j, float *best_d, int32_t *second_j, float *second_d,
                                              float slack_rel, unsigned *hdr, int32_t *ovf_rows) {
    const int lane = threadIdx.x & 31;
    float qv[4], qn = 0.f;
#pragma unroll
    for (int k = 0; k < 4; k++) {
        qv[k] = lane + 32 * k < dim ? __ldg(q + lane + 32 * k) : 0.f;
        qn = fmaf(qv[k], qv[k], qn);
    }
    for (int o = 16; o; o >>= 1) qn += __shfl_xor_sync(0xffffffffu, qn, o);
    pdl_wait();                                      // candidates are written by the GEMM kernel
    const int ncand = splits * CAND;
    // fp16 mode (hdr != null): absolute terms of the band -- fp16 subnormals (components below 2^-24 of the scaled
    // maximum round to 2^-25 absolute) and the norm chunk's last term
    float slack_abs = 0.f, slack_const = 0.f;
    if (hdr) {
        float s_, is2, mp;
        l2_scale_from_bits(__ldcg(hdr), s_, is2, mp);
        slack_abs = 4.656612873e-10f * mp * sqrtf((float)dim);     // 2^-31 M' sqrt(D), times sqrt(3|q|^2 + 2d) below
        slack_const = 4.8828125e-4f * is2;                          // 2^-11 / s^2
    }
    bool overflow = false;
    // second-smallest approximate distance over all candidates (two warp minima per 32 candidates)
    float m1 = 3.4e38f, m2 = 3.4e38f;
    for (int c0 = 0; c0 < ncand; c0 += 32) {
        const int c = c0 + lane, sp = c / CAND, k = c - sp * CAND;
        const size_t o = ((size_t)sp * n1 + i) * CAND + k;
        const int j = c < ncand ? __ldg(cand_j + o) : -1;
        float d = (j >= 0 && j < n2) ? __ldg(cand_d + o) : 3.4e38f;
        float a = d;
        for (int sh = 16; sh; sh >>= 1) a = fminf(a, __shfl_xor_sync(0xffffffffu, a, sh));
        const unsigned holders = __ballot_sync(0xffffffffu, d == a);
        if (lane == __ffs(holders) - 1) d = 3.4e38f;                 // drop ONE instance of the minimum
        float b2 = d;
        for (int sh = 16; sh; sh >>= 1) b2 = fminf(b2, __shfl_xor_sync(0xffffffffu, b2, sh));
        // merge (a <= b2) into (m1 <= m2)
        const float n1m = fminf(m1, a), n2m = fminf(fmaxf(m1, a), fminf(m2, b2));
        m1 = n1m; m2 = n2m;
    }
    float b = 0.f, s = 0.f; int bj = -1, sj = -1;
    for (int c0 = 0; c0 < ncand; c0 += 32) {
        const int c = c0 + lane, sp = c / CAND, k = c - sp * CAND;
        const size_t o = ((size_t)sp * n1 + i) * CAND + k;
        const int jc = c < ncand ? __ldg(cand_j + o) : -1;
        const float dc = (jc >= 0 && jc < n2) ? __ldg(cand_d + o) : 3.4e38f;
        const float span = 3.f * qn + 2.f * dc;
        const bool keep = jc >= 0 && jc < n2 && dc <= m2 + slack_rel * span + slack_abs * sqrtf(span) + slack_const;
        unsigned todo = __ballot_sync(0xffffffffu, keep);

        while (todo) {                                               // ascending candidate order, four per batch
            int j[4]; float acc[4];
#pragma unroll
            for (int u = 0; u < 4; u++) {
                const int src = todo ? __ffs(todo) - 1 : 0;
                const int ju = __shfl_sync(0xffffffffu, jc, src);
                j[u] = todo ? ju : -1;
                todo &= todo - 1;
            }
            float tv[4][4];
#pragma unroll
            for (int u = 0; u < 4; u++)
#pragma unroll
                for (int k2 = 0; k2 < 4; k2++)
                    tv[u][k2] = (j[u] >= 0 && lane + 32 * k2 < dim) ? __ldg(t + (size_t)j[u] * dim + lane + 32 * k2) : 0.f;
#pragma unroll
            for (int u = 0; u < 4; u++) {
                acc[u] = 0.f;
#pragma unroll
                for (int k2 = 0; k2 < 4; k2++) {
                    const float df = qv[k2] - tv[u][k2];
                    if (lane + 32 * k2 < dim) acc[u] = fmaf(df, df, acc[u]);
                }
            }
#pragma unroll
            for (int sh = 16; sh; sh >>= 1)
#pragma unroll
                for (int u = 0; u < 4; u++) acc[u] += __shfl_xor_sync(0xffffffffu, acc[u], sh);
#pragma unroll
            for (int u = 0; u < 4; u++) {
                if (j[u] < 0) continue;
                const bool lt_b = bj < 0 || acc[u] < b || (acc[u] == b && j[u] < bj);
                const bool lt_s = sj < 0 || acc[u] < s || (acc[u] == s && j[u] < sj);
                if (lt_b) { s = b; sj = bj; b = acc[u]; bj = j[u]; }
                else if (lt_s) { s = acc[u]; sj = j[u]; }
            }
        }
    }
    if (lane == 0) {
        best_j[o_out] = bj; best_d[o_out] = bj < 0 ? -1.f : b;
        second_j[o_out] = sj; second_d[o_out] = sj < 0 ? -1.f : s;
    }
    // Certificate.  A train row x that the GEMM kernel's lists do not hold either lay outside the band of the second
    // best approximation when it was seen (and the band only shrinks), or was turned away / evicted by a full list --
    // then approx(x) >= that list's last entry (cand_drop).  If x belonged to the exact top two, exact(x) <= s (the
    // exact second best of the kept candidates) and |t_x|^2 <= 2|q|^2 + 2 exact(x), so approx(x) <= s + err (3|q|^2 + 2 s).
    // A full list whose last entry lies above that hid nothing; otherwise the row is recomputed exhaustively.
    if (ovf_rows && sj >= 0) {
        const float span = 3.f * qn + 2.f * s;
        const float lim = s + 0.5f * slack_rel * span + slack_abs * sqrtf(span) + slack_const;
        const int nlists = splits * EPI_GROUPS;
        for (int c = lane; c < nlists; c += 32) {
            const int sp = c / EPI_GROUPS, g = c - sp * EPI_GROUPS;
            overflow |= __ldg(cand_drop + ((size_t)sp * n1 + i) * EPI_GROUPS + g) <= lim;
        }
        if (__any_sync(0xffffffffu, overflow) && lane == 0) ovf_rows[atomicAdd(hdr + 1, 1u)] = i;
    }
}
__global__ void __launch_bounds__(256, 7) l2_refine_kernel(const float *__restrict__ q, int n1, const float *__restrict__ t, int n2,
                                                        int dim, const int32_t *__restrict__ cand_j,
                                                        const float *__restrict__ cand_d, const float *__restrict__ cand_drop, int splits,
                                                        int32_t *best_j, float *best_d, int32_t *second_j, float *second_d,
                                                        float slack_rel, unsigned *hdr, int32_t *ovf_rows) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (warp >= n1) return;
    l2_refine_row(q + (size_t)warp * dim, t, n2, dim, cand_j, cand_d, cand_drop, splits, n1, warp, (size_t)warp, best_j, best_d,
                  second_j, second_d, slack_rel, hdr, ovf_rows);
}

// ---- exhaustive fallback for the rows the refinement could not certify ----------------------------
// Every CTA owns slices of the train set and evaluates ALL flagged queries against them, EX_R queries at a time
// (queries in shared memory, a train row is loaded once per EX_R queries): exact fp32 distances with the
// refinement's summation order (so a distance has the same bits whichever kernel computed it), top-2 by
// (distance, index) per warp, merged per CTA into part[row][slice]; the CTA that finishes last (one ticket,
// returned to zero) merges the slices of every flagged row.  A handful of flagged rows -- the usual case when there
// are any -- costs one pass over the train set (16 MB at 32k x 128: ~5 us); with nothing flagged every CTA reads
// the count and leaves.  slices = min(grid, n2 / 64, EX_MAX_SLICES_PER_ROW * n1 / rows), the last term being the
// capacity of `part`.
constexpr int EX_MAX_SLICES_PER_ROW = 16;   // capacity of `part`: n1 * this many float4
constexpr int EX_THREADS = 256;
constexpr int EX_R = 8;                     // flagged queries evaluated per pass over a slice
struct Top2 { float b, s; int bj, sj; };
__device__ __forceinline__ void top2_insert(Top2 &x, float d, int j) {
    if (j < 0) return;
    const bool lt_b = x.bj < 0 || d < x.b || (d == x.b && j < x.bj);
    const bool lt_s = x.sj < 0 || d < x.s || (d == x.s && j < x.sj);
    if (lt_b) { x.s = x.b; x.sj = x.bj; x.b = d; x.bj = j; }
    else if (lt_s) { x.s = d; x.sj = j; }
}
__device__ __forceinline__ Top2 top2_warp_merge(Top2 x) {
#pragma unroll
    for (int sh = 16; sh; sh >>= 1) {
        const float ob = __shfl_xor_sync(0xffffffffu, x.b, sh), os = __shfl_xor_sync(0xffffffffu, x.s, sh);
        const int obj = __shfl_xor_sync(0xffffffffu, x.bj, sh), osj = __shfl_xor_sync(0xffffffffu, x.sj, sh);
        top2_insert(x, ob, obj);
        top2_insert(x, os, osj);
    }
    return x;
}
__global__ void __launch_bounds__(EX_THREADS) l2_exact_rows_kernel(const float *__restrict__ q, int n1, const float *__restrict__ t,
                                                                   int n2, int dim, unsigned *__restrict__ hdr,
                                                                   const int32_t *__restrict__ ovf_rows,
                                                                   float4 *__restrict__ part, int32_t *best_j, float *best_d,
                                                                   int32_t *second_j, float *second_d) {
    pdl_wait();
    const int count = (int)__ldcg(hdr + 1);
    if (blockIdx.x == 0 && threadIdx.x == 0) hdr[0] = 0;       // every reader of the scale has finished: reset for the next call
    if (count == 0) return;
    long long want = min((long long)gridDim.x, (long long)EX_MAX_SLICES_PER_ROW * n1 / count);
    want = max(1ll, min(want, (long long)(n2 + 63) / 64));
    const int slice = (int)(((n2 + want - 1) / want + 31) / 32 * 32);
    const int n_slices = (n2 + slice - 1) / slice;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    __shared__ float s_q[EX_R][128];
    __shared__ Top2 s_top[EX_THREADS / 32][EX_R];
    __shared__ unsigned s_ticket;
    for (int sl = blockIdx.x; sl < n_slices; sl += gridDim.x) {
        const int j0 = sl * slice, j1 = min(n2, j0 + slice);
        for (int r0 = 0; r0 < count; r0 += EX_R) {
            const int nr = min(EX_R, count - r0);
            for (int e = threadIdx.x; e < EX_R * 128; e += EX_THREADS) {
                const int r = e >> 7, k = e & 127;
                s_q[r][k] = (r < nr && k < dim) ? __ldg(q + (size_t)__ldcg(ovf_rows + r0 + r) * dim + k) : 0.f;
            }
            __syncthreads();
            Top2 x[EX_R];
#pragma unroll
            for (int r = 0; r < EX_R; r++) x[r] = Top2{0.f, 0.f, -1, -1};
            for (int jb = j0 + 4 * warp; jb < j1; jb += 4 * (EX_THREADS / 32)) {      // four train rows per warp step
                float tv[4][4];
#pragma unroll
                for (int u = 0; u < 4; u++)
#pragma unroll
                    for (int k2 = 0; k2 < 4; k2++)
                        tv[u][k2] = (jb + u < j1 && lane + 32 * k2 < dim) ? __ldg(t + (size_t)(jb + u) * dim + lane + 32 * k2) : 0.f;
#pragma unroll
                for (int r = 0; r < EX_R; r++) {
                    if (r >= nr) break;                                                   // uniform
                    float acc[4];
#pragma unroll
                    for (int u = 0; u < 4; u++) {
                        acc[u] = 0.f;
#pragma unroll
                        for (int k2 = 0; k2 < 4; k2++) {
                            const float df = s_q[r][lane + 32 * k2] - tv[u][k2];
                            if (lane + 32 * k2 < dim) acc[u] = fmaf(df, df, acc[u]);
                        }
                    }
#pragma unroll
                    for (int sh = 16; sh; sh >>= 1)
#pragma unroll
                        for (int u = 0; u < 4; u++) acc[u] += __shfl_xor_sync(0xffffffffu, acc[u], sh);
#pragma unroll
                    for (int u = 0; u < 4; u++) top2_insert(x[r], acc[u], jb + u < j1 ? jb + u : -1);
                }
            }
            if (lane == 0) {
#pragma unroll
                for (int r = 0; r < EX_R; r++) s_top[warp][r] = x[r];
            }
            __syncthreads();
            if ((int)threadIdx.x < nr) {
                const int r = threadIdx.x;
                Top2 m = s_top[0][r];
                for (int w = 1; w < EX_THREADS / 32; w++) { top2_insert(m, s_top[w][r].b, s_top[w][r].bj); top2_insert(m, s_top[w][r].s, s_top[w][r].sj); }
                part[(size_t)(r0 + r) * n_slices + sl] = make_float4(m.b, __int_as_float(m.bj), m.s, __int_as_float(m.sj));
            }
            __syncthreads();
        }
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_ticket = atomicAdd(hdr + 2, 1u);
    __syncthreads();
    if (s_ticket != gridDim.x - 1) return;
    __threadfence();                                                               // last CTA: merge the slices of every flagged row
    for (int r = warp; r < count; r += EX_THREADS / 32) {
        Top2 m{0.f, 0.f, -1, -1};
        for (int k = lane; k < n_slices; k += 32) {
            const float4 v = __ldcg(part + (size_t)r * n_slices + k);
            top2_insert(m, v.x, __float_as_int(v.y));
            top2_insert(m, v.z, __float_as_int(v.w));
        }
        m = top2_warp_merge(m);
        if (lane == 0) {
            const int i = __ldcg(ovf_rows + r);
            best_j[i] = m.bj; best_d[i] = m.bj < 0 ? -1.f : m.b;
            second_j[i] = m.sj; second_d[i] = m.sj < 0 ? -1.f : m.s;
        }
    }
    if (threadIdx.x == 0) hdr[2] = 0;                                              // ticket ready for the next call
}


// ---- many pairs per launch (pgm_knn2_l2_pairs_batch_dev, pgm_match_l2_ratio_crosscheck_pairs_batch_dev) ----------
// A chunk of pairs runs the single-pair chain of the CTA-pair path -- scale, fp16 operands, GEMM + top-8, refinement,
// exhaustive fallback -- once over all its pairs:
//   l2b_prep_kernel          max |x| over every image the chunk converts (one power-of-two scale per chunk), resets the
//                            flagged-row count, fills the candidate lists with "absent"
//   l2b_split16_kernel       each image once per role: query form into A', train form into B' (one warp per row)
//   l2_topk_pair_kernel<DBG, true>  flattened (pair, row pair, column tile) items
//   l2b_refine_kernel        one warp per query row of the chunk; every row knows its pair
//   l2b_exact_rows_kernel    the flagged rows of all pairs, (flagged row, train slice) work, merged by the last CTA
// The ratio entry point adds l2b_filter_kernel + l2b_scatter_kernel.  Distances are computed by the code of the single-
// pair kernels (l2_refine_row; the fallback sums in the same order), so a pair's result is bit-identical to its
// pgm_knn2_l2_dev result whatever scale the chunk uses: the band is certified, the scale only decides how many rows
// need the fallback.
__global__ void __launch_bounds__(256) l2b_prep_kernel(const float *__restrict__ all, int dim, const L2BImage *__restrict__ img,
                                                       int n_img, unsigned *__restrict__ hdr, int32_t *__restrict__ cand_j,
                                                       size_t n_cand, float *__restrict__ cand_drop, size_t n_drop) {
    pdl_trigger();
    if (blockIdx.x == 0 && threadIdx.x == 0) hdr[1] = 0;
    const size_t stride = (size_t)gridDim.x * blockDim.x, tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (size_t e = tid; e < n_cand; e += stride) cand_j[e] = -1;
    for (size_t e = tid; e < n_drop; e += stride) cand_drop[e] = 3.4e38f;
    unsigned m = 0;
    for (int k = 0; k < n_img; k++) m = absmax_span(all + (size_t)img[k].src_row * dim, (size_t)img[k].n * dim, tid, stride, m);
    absmax_commit(m, hdr);
}

// img_base[k] = first conversion row of image entry k (exclusive prefix over n_img entries)
__global__ void __launch_bounds__(256) l2b_split16_kernel(const float *__restrict__ all, int dim, int dp, const L2BImage *__restrict__ img,
                                                          const int32_t *__restrict__ img_base, int n_img, __half *__restrict__ a,
                                                          __half *__restrict__ b, const unsigned *__restrict__ hdr,
                                                          float *__restrict__ qnorm) {
    const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    pdl_trigger();
    if (w >= __ldg(img_base + n_img)) return;
    const int e = l2_find(img_base, n_img, w);
    const int r = w - __ldg(img_base + e);
    PGM_ASSERT(e >= 0 && e < n_img && r >= 0 && r < img[e].n);
    const bool train = img[e].train != 0;
    const int row = img[e].dst_row + r;
    __half *o = (train ? b : a) + (size_t)row * (dp + CHUNK_K);
    float v[4];
    split16_load(all + (size_t)(img[e].src_row + r) * dim, dim, dp, lane, v);
    pdl_wait();                                      // the scale comes from l2b_prep_kernel
    float s, inv_s2, mprime;
    l2_scale_from_bits(__ldcg(hdr), s, inv_s2, mprime);
    const float acc = split16_store(v, s, dp, lane, train, o);
    if (!train && lane == 0) qnorm[row] = acc;
}

// row_base[k] = pairs[k].row0 (exclusive prefix over the chunk's pairs, row_base[n_pairs] = rows)
__global__ void __launch_bounds__(256, 7) l2b_refine_kernel(const float *__restrict__ all, int dim, const L2BPair *__restrict__ pairs,
                                                         const int32_t *__restrict__ row_base, int n_pairs, int rows,
                                                         const int32_t *__restrict__ cand_j, const float *__restrict__ cand_d,
                                                         const float *__restrict__ cand_drop, int splits, int32_t *best_j,
                                                         float *best_d, int32_t *second_j, float *second_d, float slack_rel,
                                                         unsigned *hdr, int32_t *ovf_rows) {
    const int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (r >= rows) return;
    const int k = l2_find(row_base, n_pairs, r);
    const L2BPair &pr = pairs[k];
    const int i = r - pr.row0;
    PGM_ASSERT(k >= 0 && k < n_pairs && i >= 0 && i < pr.n1);
    l2_refine_row(all + (size_t)(pr.q_row + i) * dim, all + (size_t)pr.t_row * dim, pr.n2, dim, cand_j, cand_d, cand_drop,
                  splits, rows, r, (size_t)(pr.out_row + i), best_j, best_d, second_j, second_d, slack_rel, hdr, ovf_rows);
}

// Flagged rows of all pairs of the chunk: work item = (flagged row, one of S slices of its pair's train image), S chosen
// from the flagged count so that the grid has work (at most EX_MAX_SLICES_PER_ROW: `part` holds rows x that many).  Each
// CTA's warps take four train rows per step; a distance is summed exactly as l2_refine_row sums it.  The CTA that
// finishes last merges every flagged row's slices, adds the count to hdr[3] (the call's total) and returns the ticket
// to zero.
__global__ void __launch_bounds__(EX_THREADS) l2b_exact_rows_kernel(const float *__restrict__ all, int dim,
                                                                    const L2BPair *__restrict__ pairs,
                                                                    const int32_t *__restrict__ row_base, int n_pairs, int rows,
                                                                    unsigned *__restrict__ hdr, const int32_t *__restrict__ ovf_rows,
                                                                    float4 *__restrict__ part, int32_t *best_j, float *best_d,
                                                                    int32_t *second_j, float *second_d) {
    pdl_wait();
    const int count = (int)__ldcg(hdr + 1);
    if (blockIdx.x == 0 && threadIdx.x == 0) hdr[0] = 0;       // every reader of the scale has finished: reset for the next chunk
    if (count == 0) return;
    PGM_ASSERT(count <= rows);
    const int S = (int)min((long long)EX_MAX_SLICES_PER_ROW, max(1ll, (2ll * gridDim.x + count - 1) / count));
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    __shared__ Top2 s_top[EX_THREADS / 32];
    __shared__ unsigned s_ticket;
    for (long long w = blockIdx.x; w < (long long)count * S; w += gridDim.x) {
        const int f = (int)(w / S), sl = (int)(w - (long long)f * S);
        const int r = __ldcg(ovf_rows + f);
        PGM_ASSERT(r >= 0 && r < rows);
        const int k = l2_find(row_base, n_pairs, r);
        PGM_ASSERT(k >= 0 && k < n_pairs && r - pairs[k].row0 < pairs[k].n1);
        const int n2 = pairs[k].n2;
        const float *q = all + (size_t)(pairs[k].q_row + (r - pairs[k].row0)) * dim;
        const float *t = all + (size_t)pairs[k].t_row * dim;
        const int len = ((n2 + S - 1) / S + 3) & ~3;
        const int j0 = min(n2, sl * len), j1 = min(n2, j0 + len);
        float qv[4];
#pragma unroll
        for (int k2 = 0; k2 < 4; k2++) qv[k2] = lane + 32 * k2 < dim ? __ldg(q + lane + 32 * k2) : 0.f;
        Top2 x{0.f, 0.f, -1, -1};
        for (int jb = j0 + 4 * warp; jb < j1; jb += 4 * (EX_THREADS / 32)) {
            float tv[4][4], acc[4];
#pragma unroll
            for (int u = 0; u < 4; u++)
#pragma unroll
                for (int k2 = 0; k2 < 4; k2++)
                    tv[u][k2] = (jb + u < j1 && lane + 32 * k2 < dim) ? __ldg(t + (size_t)(jb + u) * dim + lane + 32 * k2) : 0.f;
#pragma unroll
            for (int u = 0; u < 4; u++) {
                acc[u] = 0.f;
#pragma unroll
                for (int k2 = 0; k2 < 4; k2++) {
                    const float df = qv[k2] - tv[u][k2];
                    if (lane + 32 * k2 < dim) acc[u] = fmaf(df, df, acc[u]);
                }
            }
#pragma unroll
            for (int sh = 16; sh; sh >>= 1)
#pragma unroll
                for (int u = 0; u < 4; u++) acc[u] += __shfl_xor_sync(0xffffffffu, acc[u], sh);
#pragma unroll
            for (int u = 0; u < 4; u++) top2_insert(x, acc[u], jb + u < j1 ? jb + u : -1);
        }
        if (lane == 0) s_top[warp] = x;
        __syncthreads();
        if (threadIdx.x == 0) {
            Top2 m = s_top[0];
            for (int v = 1; v < EX_THREADS / 32; v++) { top2_insert(m, s_top[v].b, s_top[v].bj); top2_insert(m, s_top[v].s, s_top[v].sj); }
            part[(size_t)f * S + sl] = make_float4(m.b, __int_as_float(m.bj), m.s, __int_as_float(m.sj));
        }
        __syncthreads();
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_ticket = atomicAdd(hdr + 2, 1u);
    __syncthreads();
    if (s_ticket != gridDim.x - 1) return;
    __threadfence();                                                               // last CTA: merge the slices of every flagged row
    for (int f = warp; f < count; f += EX_THREADS / 32) {
        Top2 m{0.f, 0.f, -1, -1};
        if (lane < S) {
            const float4 v = __ldcg(part + (size_t)f * S + lane);
            top2_insert(m, v.x, __float_as_int(v.y));
            top2_insert(m, v.z, __float_as_int(v.w));
        }
        m = top2_warp_merge(m);
        if (lane == 0) {
            const int r = __ldcg(ovf_rows + f);
            const int k = l2_find(row_base, n_pairs, r);
            PGM_ASSERT(k >= 0 && k < n_pairs && r - pairs[k].row0 >= 0 && r - pairs[k].row0 < pairs[k].n1);
            const size_t o = (size_t)(pairs[k].out_row + (r - pairs[k].row0));
            best_j[o] = m.bj; best_d[o] = m.bj < 0 ? -1.f : m.b;
            second_j[o] = m.sj; second_d[o] = m.sj < 0 ? -1.f : m.s;
        }
    }
    if (threadIdx.x == 0) { hdr[3] += (unsigned)count; hdr[2] = 0; }              // call total; ticket ready for the next chunk
}

// Ratio test + cross-check + distance bound on the chunk's knn2 results, then the ordered compaction, as
// rcp_filter_kernel / rcp_scatter_kernel do for Hamming keys (L2 distances are floats, so the keys do not carry them).
struct L2RPair {
    int64_t out_base;          // first slot of this pair's triples in the caller's output arrays
    int32_t row0, rrow0;       // knn2 rows of the pair and, with cross-check, of the reversed pair (train image as query)
    int32_t n1, n2, pair_id, pad;
};
constexpr int L2F_THREADS = 1024;    // rows per filter / scatter block (n1 < 2^20: at most 1024 blocks per pair)
__global__ void __launch_bounds__(L2F_THREADS) l2b_filter_kernel(const L2RPair *__restrict__ pairs, const int32_t *__restrict__ fblk_base,
                                                                 int n_pairs, int rows, const int32_t *__restrict__ bj,
                                                                 const float *__restrict__ bd, const float *__restrict__ sd,
                                                                 float ratio, float rr, int cross_check, float max_sq_dist,
                                                                 int32_t *__restrict__ keep_row, int32_t *__restrict__ bcnt) {
    const int g = blockIdx.x;
    const int k = l2_find(fblk_base, n_pairs, g);
    const L2RPair pr = pairs[k];
    const int i = (g - __ldg(fblk_base + k)) * L2F_THREADS + threadIdx.x;
    bool keep = false;
    if (i < pr.n1) {
        const int r = pr.row0 + i;
        PGM_ASSERT(r >= 0 && r < rows);
        const int j = bj[r];
        const float d1 = bd[r], d2 = sd[r];
        PGM_ASSERT(j < pr.n2);
        keep = j >= 0;
        keep = keep && (pr.n2 < 2 || ratio <= 0.f || d1 < rr * d2);
        if (keep && cross_check) {
            PGM_ASSERT(pr.rrow0 + j >= 0 && pr.rrow0 + j < rows);
            keep = bj[pr.rrow0 + j] == i;
        }
        keep = keep && (max_sq_dist < 0.f || d1 <= max_sq_dist);
        keep_row[r] = keep ? 1 : 0;
    }
    const int n = __syncthreads_count(keep);
    if (threadIdx.x == 0) bcnt[g] = n;
}

__global__ void __launch_bounds__(L2F_THREADS) l2b_scatter_kernel(const L2RPair *__restrict__ pairs, const int32_t *__restrict__ fblk_base,
                                                                  int n_pairs, const int32_t *__restrict__ keep_row,
                                                                  const int32_t *__restrict__ bj, const float *__restrict__ bd,
                                                                  const int32_t *__restrict__ bcnt, int64_t capacity,
                                                                  int32_t *__restrict__ out_qi, int32_t *__restrict__ out_tj,
                                                                  float *__restrict__ out_dist, int32_t *__restrict__ counts) {
    __shared__ int s_before[L2F_THREADS / 32], s_total[L2F_THREADS / 32], s_w[L2F_THREADS / 32];
    const int g = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int k = l2_find(fblk_base, n_pairs, g);
    const L2RPair pr = pairs[k];
    const int first = __ldg(fblk_base + k), nb = __ldg(fblk_base + k + 1) - first, b = g - first;
    // kept rows of the pair's blocks before this one, and of all of them (nb <= L2F_THREADS)
    const int c = tid < nb ? __ldg(bcnt + first + tid) : 0;
    int before = tid < b ? c : 0, total = c;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        before += __shfl_xor_sync(0xffffffffu, before, o);
        total += __shfl_xor_sync(0xffffffffu, total, o);
    }
    const int i = b * L2F_THREADS + tid;
    const bool keep = i < pr.n1 && __ldg(keep_row + pr.row0 + i) != 0;
    const unsigned m = __ballot_sync(0xffffffffu, keep);
    if (lane == 0) { s_before[wid] = before; s_total[wid] = total; s_w[wid] = __popc(m); }
    __syncthreads();
    int off = 0;
    before = 0; total = 0;
#pragma unroll 4
    for (int w = 0; w < L2F_THREADS / 32; w++) {
        before += s_before[w]; total += s_total[w];
        if (w < wid) off += s_w[w];
    }
    if (keep) {
        const int64_t o = pr.out_base + before + off + __popc(m & ((1u << lane) - 1u));
        PGM_ASSERT(o >= pr.out_base && o < pr.out_base + pr.n1 && o < capacity);
        out_qi[o] = i; out_tj[o] = __ldg(bj + pr.row0 + i); out_dist[o] = __ldg(bd + pr.row0 + i);
    }
    if (b == nb - 1 && tid == 0) counts[pr.pair_id] = total;
}

}  // namespace pgm_l2
