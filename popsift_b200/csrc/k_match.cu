// Brute-force 2-nearest-neighbour descriptor matcher, hand-written for sm_100a (tcgen05 + TMEM + TMA).
//
// Replaces FeaturesDev::match -> compute_distance (reference src/popsift/features.cu:165-227,282-304): for every
// left descriptor the best and second-best right descriptor by squared L2 distance and the ratio test
// best / second < 0.8.  The reference runs one 32-thread block per left descriptor and walks all right
// descriptors one by one (n_left x n_right x 128 scalar flops on CUDA cores, every right descriptor re-read
// n_left times).  This is the one dense contraction of the library:
//     |a - b|^2 = |a|^2 + |b|^2 - 2 a.b        ->   S = A . B^T  on the tensor cores.
//
// Pipeline (ps_match):
//   1. match_split_kernel     a = hi + lo with hi = tf32(a) (round to nearest), lo = a - hi; |b|^2 per right
//                             descriptor.  Three tf32 products hi.hi + hi.lo + lo.hi give a.b to ~2^-21 relative.
//   2. match_tc_kernel        one CTA per 128 left descriptors.  The A tile (hi and lo, 128 x 128 floats each) is
//                             loaded once with TMA (SWIZZLE_128B, K-major) and stays in shared memory; the right
//                             descriptors stream in order through a 2-stage TMA ring of [128 descriptors x 32 floats]
//                             tiles (hi and lo); ONE thread issues tcgen05.mma.kind::tf32 (M = 128, N = 128, K = 8) into
//                             a double-buffered fp32 accumulator in TMEM; four epilogue warps read the accumulator with tcgen05.ld
//                             (thread = one left descriptor = one TMEM lane) and keep that descriptor's four best
//                             candidates |b|^2 - 2 a.b in registers.  The n_left x n_right distance matrix never
//                             touches HBM.  Warp roles: 0 = TMA producer, 1 = MMA issuer + TMEM owner, 2..5 = epilogue.
//   3. match_rerank_kernel    one warp per left descriptor recomputes the exact float32 distance of its four
//                             candidates in the reference's own evaluation order (per lane x*x, fma, fma, fma over its
//                             float4, shuffle-down tree 16, 8, 4, 2, 1) and applies the reference's scan rule
//                             (strict <, ties keep the lower index) and ratio test.
// The result equals the reference's except when three or more right descriptors lie within ~4e-6 (relative) of the second
// best (the candidate pass could then miss the reference's pick among exact near-ties).
// match_exact_kernel is the same computation on CUDA cores (one warp per left descriptor over all right ones): used
// for small problems and as the in-library cross-check (PS_MATCH_EXACT).
#include "ps_internal.h"
#include "tma_util.h"

#include <cstdint>
#include <mutex>

namespace psb {

namespace {

// ------------------------------------------------------------------------------------------------ exact (CUDA cores)

// squared distance of the warp's left descriptor (lane holds l4) to right descriptor r, reference order
// (features.cu:165-185: per lane x*x + y*y + z*z + w*w -- SASS FMUL, FFMA, FFMA, FFMA -- then shuffle_down 16..1)
__device__ __forceinline__ float warp_sq_dist(const float4 l4, const float4* __restrict__ r, int lane)
{
    const float4 r4 = __ldg(r + lane);
    const float dx = __fsub_rn(l4.x, r4.x), dy = __fsub_rn(l4.y, r4.y), dz = __fsub_rn(l4.z, r4.z), dw = __fsub_rn(l4.w, r4.w);
    float res = __fmul_rn(dx, dx);
    res = __fmaf_rn(dy, dy, res);
    res = __fmaf_rn(dz, dz, res);
    res = __fmaf_rn(dw, dw, res);
    res = __fadd_rn(res, __shfl_down_sync(0xffffffffu, res, 16));
    res = __fadd_rn(res, __shfl_down_sync(0xffffffffu, res, 8));
    res = __fadd_rn(res, __shfl_down_sync(0xffffffffu, res, 4));
    res = __fadd_rn(res, __shfl_down_sync(0xffffffffu, res, 2));
    res = __fadd_rn(res, __shfl_down_sync(0xffffffffu, res, 1));
    return __shfl_sync(0xffffffffu, res, 0);
}

struct Best2 {
    float v1, v2; int i1, i2;
    __device__ __forceinline__ void init() { v1 = v2 = INFINITY; i1 = i2 = 0; }
    // the reference's scan step (features.cu:205-217); candidates must arrive in increasing index order
    __device__ __forceinline__ void step(float res, int i)
    {
        if (res < v1) { v2 = v1; i2 = i1; v1 = res; i1 = i; }
        else if (res < v2) { v2 = res; i2 = i; }
    }
    __device__ __forceinline__ void store(int32_t* out) const
    {
        out[0] = i1; out[1] = i2; out[2] = (__fdiv_rn(v1, v2) < 0.8f) ? 1 : 0;
    }
};

__global__ void __launch_bounds__(128)
match_exact_kernel(const ps_descriptor* __restrict__ l, int nl, const ps_descriptor* __restrict__ r, int nr, int32_t* __restrict__ out)
{
    const int lane = threadIdx.x & 31;
    const int row = blockIdx.x * 4 + (threadIdx.x >> 5);
    if (row >= nl) return;
    const float4 l4 = __ldg(reinterpret_cast<const float4*>(l + row) + lane);
    Best2 b; b.init();
    for (int i = 0; i < nr; ++i) b.step(warp_sq_dist(l4, reinterpret_cast<const float4*>(r + i), lane), i);
    if (lane == 0) b.store(out + 3 * (size_t)row);
}

// ------------------------------------------------------------------------------------------------ split / norms

__device__ __forceinline__ float to_tf32(float v)
{
    unsigned u;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(v));
    return __uint_as_float(u);
}

// one warp per descriptor: hi / lo planes (rows padded with zero descriptors up to n_pad) and, for the right set,
// |b|^2 (+inf for the padding rows so that they never become candidates)
__global__ void __launch_bounds__(128)
match_split_kernel(const ps_descriptor* __restrict__ d, int n, int n_pad, float* __restrict__ hi, float* __restrict__ lo, float* __restrict__ norm)
{
    const int lane = threadIdx.x & 31;
    const int row = blockIdx.x * 4 + (threadIdx.x >> 5);
    if (row >= n_pad) return;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (row < n) v = __ldg(reinterpret_cast<const float4*>(d + row) + lane);
    const float4 h = make_float4(to_tf32(v.x), to_tf32(v.y), to_tf32(v.z), to_tf32(v.w));
    const float4 lw = make_float4(v.x - h.x, v.y - h.y, v.z - h.z, v.w - h.w);
    reinterpret_cast<float4*>(hi + (size_t)row * 128)[lane] = h;
    reinterpret_cast<float4*>(lo + (size_t)row * 128)[lane] = lw;
    if (norm) {
        float s = fmaf(v.x, v.x, fmaf(v.y, v.y, fmaf(v.z, v.z, v.w * v.w)));
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) norm[row] = row < n ? s : INFINITY;
    }
}

// ------------------------------------------------------------------------------------------------ tensor-core pass

constexpr int BM = 128, BN = 128;            // left descriptors per CTA, right descriptors per accumulator tile
constexpr int KB = 32;                       // floats per K-block = one 128-byte swizzle span
constexpr int NKB = 128 / KB;                // K-blocks per descriptor
constexpr int UMMA_K = 8;                    // tf32: 32 bytes per instruction
constexpr int TILE_BYTES = BM * KB * 4;      // 16 KB: one [128 rows x 128 bytes] operand tile of the left set
constexpr int BTILE_BYTES = BN * KB * 4;     // 16 KB: one [128 rows x 128 bytes] operand tile of the right set
constexpr int STAGES = 2;                    // B ring: stages of [hi, lo] tiles
constexpr int TC_THREADS = 192;              // 6 warps
constexpr int kCand = 4;                     // candidates kept per left descriptor
constexpr size_t TC_SMEM = (size_t)2 * NKB * TILE_BYTES + (size_t)STAGES * 2 * BTILE_BYTES;   // A hi/lo resident + 64 KB B ring = 192 KB
constexpr int TMEM_COLS = 2 * BN;            // two fp32 accumulators of 128 columns

__device__ __forceinline__ unsigned s32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mb_init(uint64_t* b, unsigned n) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(s32(b)), "r"(n) : "memory"); }
__device__ __forceinline__ void mb_expect(uint64_t* b, unsigned bytes) { asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(s32(b)), "r"(bytes) : "memory"); }
__device__ __forceinline__ void mb_arrive(uint64_t* b) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(s32(b)) : "memory"); }
__device__ __forceinline__ void mb_wait(uint64_t* b, unsigned parity)
{
    unsigned ok, spins = 0;
    for (;;) {
        asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
                     : "=r"(ok) : "r"(s32(b)), "r"(parity) : "memory");
        if (ok) break;
        if (++spins > (1u << 24)) __trap();          // abort instead of hanging the device
    }
}
__device__ __forceinline__ void tma_tile(void* dst, const CUtensorMap* map, int k0, int row0, uint64_t* bar)
{
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 :: "r"(s32(dst)), "l"(reinterpret_cast<unsigned long long>(map)), "r"(k0), "r"(row0), "r"(s32(bar)) : "memory");
}
// K-major operand tile, SWIZZLE_128B, rows 128 bytes wide, 8-row groups 1024 bytes apart (cute::UMMA::SmemDescriptor:
// start >> 4 in [0,14), LBO = 1 in [16,30), SBO = 1024 >> 4 in [32,46), version 1 in [46,48), layout SWIZZLE_128B = 2 in [61,64))
__device__ __forceinline__ uint64_t umma_desc(const void* tile)
{
    return (uint64_t)((s32(tile) >> 4) & 0x3fffu) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
// cute::UMMA::InstrDescriptor: D = F32 (1 << 4), A = B = TF32 (2 << 7, 2 << 10), both K-major, N >> 3 at [17,23), M >> 4 at [24,29)
constexpr unsigned kIdesc = (1u << 4) | (2u << 7) | (2u << 10) | ((unsigned)(BN >> 3) << 17) | ((unsigned)(BM >> 4) << 24);

__device__ __forceinline__ void umma_tf32(unsigned d_tmem, uint64_t a_desc, uint64_t b_desc, unsigned accumulate, unsigned kIdesc)
{
    asm volatile("{\n .reg .pred p;\n setp.ne.b32 p, %4, 0;\n tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n}"
                 :: "r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(kIdesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(s32(bar)) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// 32 consecutive fp32 columns of this thread's TMEM lane: issue (the registers are valid after tmem_ld_wait)
__device__ __forceinline__ void tmem_ld32_issue(unsigned taddr, unsigned (&r)[32])
{
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                 "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                 "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                   "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
                   "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
                   "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
                 : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// Candidate bookkeeping of one left descriptor (one epilogue thread): the four smallest keys seen so far and where they
// came from.  A key is the approximate distance |b|^2 - 2 a.b with its 5 low mantissa bits replaced by the column's index
// inside its group of 32 (relative 2^-18: far below what separates candidates that matter, the exact re-rank follows), so
// that the group's minimum -- a branch-free FMNMX tree -- carries its own position.
struct Top4 {
    float t0 = INFINITY, t1 = INFINITY, t2 = INFINITY, t3 = INFINITY;
    int i0 = -1, i1 = -1, i2 = -1, i3 = -1;
    __device__ __forceinline__ void insert(float key, int idx)           // key < t3
    {
        t3 = key; i3 = idx;
        if (t3 < t2) { float tf = t2; t2 = t3; t3 = tf; int ti = i2; i2 = i3; i3 = ti;
            if (t2 < t1) { tf = t1; t1 = t2; t2 = tf; ti = i1; i1 = i2; i2 = ti;
                if (t1 < t0) { tf = t0; t0 = t1; t1 = tf; ti = i0; i0 = i1; i1 = ti; } } }
    }
};

// one group of 32 columns: r = raw accumulator bits (a.b), rn = |b|^2 of the 32 columns, nb = index of the group's first column
__device__ __forceinline__ void top4_group(Top4& T, const unsigned (&r)[32], const float4 (&rn)[8], int nb)
{
    float k[32];
#pragma unroll
    for (int i4 = 0; i4 < 8; ++i4) {
        const float rr[4] = {rn[i4].x, rn[i4].y, rn[i4].z, rn[i4].w};
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int i = i4 * 4 + u;
            const float val = fmaf(-2.0f, __uint_as_float(r[i]), rr[u]);          // |b|^2 - 2 a.b  (+inf for padding)
            k[i] = __uint_as_float((__float_as_uint(val) & 0xffffffe0u) | (unsigned)i);   // padding: inf -> inf (i = 0) or NaN
        }
    }
    float m[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) m[i] = fminf(k[i], k[i + 16]);                  // fminf drops NaNs
#pragma unroll
    for (int w = 8; w >= 1; w >>= 1)
#pragma unroll
        for (int i = 0; i < w; ++i) m[i] = fminf(m[i], m[i + w]);
    float best = m[0];
    // rare after the first tiles: the k-th best of n random items improves about 4 / n of the time
    while (best < T.t3) {
        T.insert(best, nb + (int)(__float_as_uint(best) & 31u));
        float nxt = INFINITY;                                                  // the group's next key above `best`
#pragma unroll
        for (int i = 0; i < 32; ++i) nxt = (k[i] > best) ? fminf(nxt, k[i]) : nxt;
        best = nxt;
    }
}

__global__ void __launch_bounds__(TC_THREADS, 1)
match_tc_kernel(const __grid_constant__ CUtensorMap tm_lhi, const __grid_constant__ CUtensorMap tm_llo,
                const __grid_constant__ CUtensorMap tm_rhi, const __grid_constant__ CUtensorMap tm_rlo,
                const float* __restrict__ rnorm, int nl, int n_tiles, int32_t* __restrict__ cand)
{
    extern __shared__ __align__(1024) uint8_t smem[];          // SWIZZLE_128B tiles: 1024-byte aligned
    __shared__ __align__(8) uint64_t a_full, b_full[STAGES], b_empty[STAGES], acc_full[2], acc_empty[2];
    __shared__ unsigned tmem_base_s;
    uint8_t* A_hi = smem;                                       // NKB tiles
    uint8_t* A_lo = smem + NKB * TILE_BYTES;
    uint8_t* B_st = smem + 2 * NKB * TILE_BYTES;                // [STAGES][hi, lo]
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int m0 = blockIdx.x * BM;

    if (threadIdx.x == 0) {
        mb_init(&a_full, 1);
        for (int s = 0; s < STAGES; ++s) { mb_init(&b_full[s], 1); mb_init(&b_empty[s], 1); }
        for (int b = 0; b < 2; ++b) { mb_init(&acc_full[b], 1); mb_init(&acc_empty[b], 4); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {                                            // TMEM: allocated and freed by the same warp
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(s32(&tmem_base_s)), "n"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const unsigned tmem_base = tmem_base_s;

    if (warp == 0) {
        // ===== TMA producer (one thread) =====
        if (lane == 0) {
            mb_expect(&a_full, 2 * NKB * TILE_BYTES);
            for (int kb = 0; kb < NKB; ++kb) {
                tma_tile(A_hi + kb * TILE_BYTES, &tm_lhi, kb * KB, m0, &a_full);
                tma_tile(A_lo + kb * TILE_BYTES, &tm_llo, kb * KB, m0, &a_full);
            }
            int s = 0; unsigned ph = 0;
            for (int j = 0; j < n_tiles; ++j)
                for (int kb = 0; kb < NKB; ++kb) {
                    mb_wait(&b_empty[s], ph ^ 1u);               // the MMAs that read this slot have completed
                    mb_expect(&b_full[s], 2 * BTILE_BYTES);
                    tma_tile(B_st + (s * 2 + 0) * BTILE_BYTES, &tm_rhi, kb * KB, j * BN, &b_full[s]);
                    tma_tile(B_st + (s * 2 + 1) * BTILE_BYTES, &tm_rlo, kb * KB, j * BN, &b_full[s]);
                    if (++s == STAGES) { s = 0; ph ^= 1u; }
                }
        }
    } else if (warp == 1) {
        // ===== MMA issuer (one thread issues; the warp stays converged on the barriers) =====
        mb_wait(&a_full, 0);
        tc_fence_after();
        int s = 0; unsigned ph = 0;
        for (int j = 0; j < n_tiles; ++j) {
            const int buf = j & 1;
            mb_wait(&acc_empty[buf], ((unsigned)(j >> 1) & 1u) ^ 1u);   // the epilogue has drained this accumulator
            tc_fence_after();
            const unsigned d_tmem = tmem_base + (unsigned)(buf * BN);
            for (int kb = 0; kb < NKB; ++kb) {
                mb_wait(&b_full[s], ph);
                tc_fence_after();
                if (lane == 0) {
                    const uint64_t a_hi = umma_desc(A_hi + kb * TILE_BYTES), a_lo = umma_desc(A_lo + kb * TILE_BYTES);
                    const uint64_t b_hi = umma_desc(B_st + (s * 2 + 0) * BTILE_BYTES), b_lo = umma_desc(B_st + (s * 2 + 1) * BTILE_BYTES);
#pragma unroll
                    for (int k8 = 0; k8 < KB / UMMA_K; ++k8) {
                        const uint64_t adv = (uint64_t)(k8 * UMMA_K * 4 / 16);      // +32 bytes inside the swizzle span
                        umma_tf32(d_tmem, a_hi + adv, b_hi + adv, (kb | k8) != 0 ? 1u : 0u, kIdesc);
                        umma_tf32(d_tmem, a_hi + adv, b_lo + adv, 1u, kIdesc);
                        umma_tf32(d_tmem, a_lo + adv, b_hi + adv, 1u, kIdesc);
                    }
                    umma_commit(&b_empty[s]);                    // slot free once these MMAs have read it
                    if (kb == NKB - 1) umma_commit(&acc_full[buf]);
                }
                __syncwarp();
                if (++s == STAGES) { s = 0; ph ^= 1u; }
            }
        }
    } else {
        // ===== epilogue: thread = one left descriptor = one TMEM lane =====
        const int q = warp & 3;                                  // TMEM lanes 32q .. 32q+31 belong to warps with warp % 4 == q
        const int row = m0 + q * 32 + lane;
        Top4 T;
        const unsigned lane_base = tmem_base + ((unsigned)(q * 32) << 16);
        for (int j = 0; j < n_tiles; ++j) {
            const int buf = j & 1;
            const int nb0 = j * BN;
            const float4* rn4 = reinterpret_cast<const float4*>(rnorm + nb0);
            // |b|^2 of the first group is on its way while the accumulator is still being written
            float4 rnA[8], rnB[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) rnA[i] = __ldg(rn4 + i);
            mb_wait(&acc_full[buf], (unsigned)(j >> 1) & 1u);
            tc_fence_after();
            // four groups of 32 columns, two register sets: group g+1 is loaded from TMEM while group g is processed
            unsigned ra[32], rb[32];
            tmem_ld32_issue(lane_base + (unsigned)(buf * BN), ra);
            tmem_ld_wait();
            tmem_ld32_issue(lane_base + (unsigned)(buf * BN + 32), rb);
#pragma unroll
            for (int i = 0; i < 8; ++i) rnB[i] = __ldg(rn4 + 8 + i);
            top4_group(T, ra, rnA, nb0);
            tmem_ld_wait();
            tmem_ld32_issue(lane_base + (unsigned)(buf * BN + 64), ra);
#pragma unroll
            for (int i = 0; i < 8; ++i) rnA[i] = __ldg(rn4 + 16 + i);
            top4_group(T, rb, rnB, nb0 + 32);
            tmem_ld_wait();
            tmem_ld32_issue(lane_base + (unsigned)(buf * BN + 96), rb);
#pragma unroll
            for (int i = 0; i < 8; ++i) rnB[i] = __ldg(rn4 + 24 + i);
            top4_group(T, ra, rnA, nb0 + 64);
            tmem_ld_wait();
            // the accumulator has been read completely: hand it back before the last group is processed
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mb_arrive(&acc_empty[buf]);
            top4_group(T, rb, rnB, nb0 + 96);
        }
        if (row < nl) *reinterpret_cast<int4*>(cand + (size_t)row * kCand) = make_int4(T.i0, T.i1, T.i2, T.i3);
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem_base), "n"(TMEM_COLS) : "memory");
}

// exact distances of the candidates, in increasing index order, through the reference's scan
__global__ void __launch_bounds__(128)
match_rerank_kernel(const ps_descriptor* __restrict__ l, int nl, const ps_descriptor* __restrict__ r, int nr,
                    const int32_t* __restrict__ cand, int32_t* __restrict__ out)
{
    const int lane = threadIdx.x & 31;
    const int row = blockIdx.x * 4 + (threadIdx.x >> 5);
    if (row >= nl) return;
    const float4 l4 = __ldg(reinterpret_cast<const float4*>(l + row) + lane);
    int c[kCand];
#pragma unroll
    for (int k = 0; k < kCand; ++k) { c[k] = cand[(size_t)row * kCand + k]; if (c[k] < 0 || c[k] >= nr) c[k] = 0x7fffffff; }
    // sort the four indices ascending (the scan rule depends on arrival order)
#pragma unroll
    for (int a = 0; a < kCand; ++a)
#pragma unroll
        for (int b = a + 1; b < kCand; ++b)
            if (c[b] < c[a]) { const int t = c[a]; c[a] = c[b]; c[b] = t; }
    Best2 best; best.init();
#pragma unroll
    for (int k = 0; k < kCand; ++k) {
        if (c[k] == 0x7fffffff) continue;                         // warp-uniform
        if (k > 0 && c[k] == c[k - 1]) continue;
        best.step(warp_sq_dist(l4, reinterpret_cast<const float4*>(r + c[k]), lane), c[k]);
    }
    if (lane == 0) best.store(out + 3 * (size_t)row);
}

} // namespace

int run_match(const ps_descriptor* l, int nl, const ps_descriptor* r, int nr, int32_t* out, int flags, cudaStream_t st,
              const char** err)
{
    *err = nullptr;
    if (nl <= 0) return 0;
    // the tensor-core pass pays off from a few thousand pairs per left descriptor; below that (and for nr < 2, where
    // the reference's scan has its own corner cases) the CUDA-core kernel is the whole job
    const bool tensor = flags == PS_MATCH_TENSOR ? nr >= 1 : (flags == PS_MATCH_EXACT ? false : (nr >= 256 && (long long)nl * nr >= (1LL << 20)));
    if (!tensor) {
        match_exact_kernel<<<(nl + 3) / 4, 128, 0, st>>>(l, nl, r, nr, out);
        return 1;
    }
    const int nl_pad = (nl + BM - 1) / BM * BM, n_tiles = (nr + BN - 1) / BN, nr_pad = n_tiles * BN;
    float *lhi = nullptr, *llo = nullptr, *rhi = nullptr, *rlo = nullptr, *rnorm = nullptr;
    int32_t* cand = nullptr;
    const size_t lb = (size_t)nl_pad * 512, rb = (size_t)nr_pad * 512;
    // one workspace allocation per call, stream-ordered so nothing blocks, from the library's own pool per device: a pool
    // gives freed memory back to the OS at the next synchronisation unless told to keep it, and mapping 50 MB again on
    // every call costs more than the matching itself (the application's default pool is left alone)
    cudaMemPool_t pool = nullptr;
    {
        static std::mutex mu;
        static cudaMemPool_t pools[64] = {};
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) { cudaGetLastError(); *err = "cudaGetDevice failed (matcher)"; return -1; }
        std::lock_guard<std::mutex> g(mu);
        if (!pools[dev]) {
            cudaMemPoolProps props = {};
            props.allocType = cudaMemAllocationTypePinned;
            props.handleTypes = cudaMemHandleTypeNone;
            props.location.type = cudaMemLocationTypeDevice;
            props.location.id = dev;
            if (cudaMemPoolCreate(&pools[dev], &props) != cudaSuccess) { cudaGetLastError(); pools[dev] = nullptr; *err = "cudaMemPoolCreate failed (matcher)"; return -1; }
            unsigned long long keep = 1ull << 30;                          // up to 1 GB of freed workspace stays mapped
            cudaMemPoolSetAttribute(pools[dev], cudaMemPoolAttrReleaseThreshold, &keep);
        }
        pool = pools[dev];
    }
    uint8_t* ws = nullptr;
    const size_t total = 2 * lb + 2 * rb + (size_t)nr_pad * 4 + (size_t)nl_pad * kCand * 4;
    if (cudaMallocFromPoolAsync(&ws, total, pool, st) != cudaSuccess) { *err = "cudaMallocFromPoolAsync failed (matcher workspace)"; cudaGetLastError(); return -1; }
    lhi = reinterpret_cast<float*>(ws); llo = reinterpret_cast<float*>(ws + lb);
    rhi = reinterpret_cast<float*>(ws + 2 * lb); rlo = reinterpret_cast<float*>(ws + 2 * lb + rb);
    rnorm = reinterpret_cast<float*>(ws + 2 * lb + 2 * rb);
    cand = reinterpret_cast<int32_t*>(ws + 2 * lb + 2 * rb + (size_t)nr_pad * 4);
    CUtensorMap m_lhi, m_llo, m_rhi, m_rlo;
    const bool ok = make_tmap_2d(&m_lhi, lhi, 128, nl_pad, 512, KB, BM, true) && make_tmap_2d(&m_llo, llo, 128, nl_pad, 512, KB, BM, true) &&
                    make_tmap_2d(&m_rhi, rhi, 128, nr_pad, 512, KB, BN, true) && make_tmap_2d(&m_rlo, rlo, 128, nr_pad, 512, KB, BN, true);
    if (!ok) { cudaFreeAsync(ws, st); *err = "cuTensorMapEncodeTiled failed (matcher)"; return -1; }
    static_assert(TC_SMEM + 2048 <= 227 * 1024, "matcher shared memory");
    match_split_kernel<<<(nl_pad + 3) / 4, 128, 0, st>>>(l, nl, nl_pad, lhi, llo, nullptr);
    match_split_kernel<<<(nr_pad + 3) / 4, 128, 0, st>>>(r, nr, nr_pad, rhi, rlo, rnorm);
    cudaFuncSetAttribute(match_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TC_SMEM);
    match_tc_kernel<<<nl_pad / BM, TC_THREADS, TC_SMEM, st>>>(m_lhi, m_llo, m_rhi, m_rlo, rnorm, nl, n_tiles, cand);
    match_rerank_kernel<<<(nl + 3) / 4, 128, 0, st>>>(l, nl, r, nr, cand, out);
    cudaFreeAsync(ws, st);
    return 4;
}

} // namespace psb
