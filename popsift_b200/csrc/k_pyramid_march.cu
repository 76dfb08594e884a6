// Stage 1, fast path -- "column-marching" fused Gaussian level kernel for sm_100a.
//
// One CTA (128 threads) owns a strip of TW=128 output columns and marches down a segment of rows in
// chunks of Q=16 rows.  Per chunk:
//   1. the Q new source rows (+ horizontal halo) are staged in shared memory by the TMA unit: ONE elected
//      thread issues one cp.async.bulk.tensor.2d (box = padded strip width x 16 rows, SASS UTMALDG) per
//      chunk, NBUF-2 chunks ahead, completion on an mbarrier per staging buffer.  No thread computes copy
//      addresses or issues per-piece copies.  The tensor map's out-of-bounds zero fill covers the left /
//      right image border (the halo columns are then patched to clamp-to-edge in shared memory); the few
//      chunks that touch the top / bottom border are staged row by row with 1-D bulk copies from the
//      clamped row addresses (UBLKCP), on the same mbarrier;
//   2. row pass: thread = (row, 16-column group); a 16+2R wide register window is loaded with
//      conflict-free LDS.128 (row stride with an odd number of float4 -- the TMA box is that wide) and
//      produces 16 outputs -> ring buffer HB of row-filtered lines (Q+2R lines);
//   3. column pass: thread = (pair of adjacent columns, 8 rows); the 8+2R ring lines are loaded once and every
//      tap is one packed FFMA2; the outputs lag the input by R rows: level l, DoG[l-1] (= out - centre
//      source, still in the staging buffers) and, for level L, the 2:1 decimated level 0 of the next octave.
// Every source row is read from HBM once (+2R warm-up rows per segment), every output written once;
// the row-filtered intermediate never leaves shared memory.
//
// The floating-point evaluation order is exactly the one documented in k_pyramid.cu (taken from the
// reference's sm_100 SASS); results are bit-identical to the tile kernels and to the reference.
#include "ps_internal.h"
#include "k_pyramid.h"
#include "k_texture.h"
#include "k_partition.h"

#include "tma_util.h"

#include <cstdint>
#include <mutex>
#include <set>
#include <utility>

namespace psb {

namespace {

constexpr int TW = 128;     // output columns per CTA
constexpr int Q = 16;       // rows per chunk
constexpr int NT = 128;     // threads per CTA
constexpr int HBW = TW + 4; // ring-buffer row stride (== 4 mod 32: conflict-free 128-bit row-wise stores)

// smallest stride >= v whose float4 count is odd: rows j = 0..7 of a quarter-warp then start in eight
// different 4-bank groups, which is all a conflict-free row-wise LDS.128 / STS.128 needs
constexpr int pad_odd4(int v) { return v + ((4 - (v % 8)) + 8) % 8; }

template <int R>
struct Geo {
    static constexpr int RP = (R + 3) / 4 * 4;          // halo rounded to float4
    static constexpr int SW = TW + 2 * RP;              // staged columns per row
    static constexpr int SWP = pad_odd4(SW);            // stage row stride
    // staging buffers: chunk k, chunk k-1 (DoG centre rows) and NBUF-2 chunks in flight.  Two chunks
    // ahead where four buffers still leave room for 4 CTAs per SM (R <= 8).
    static constexpr int NBUF = (R <= 8) ? 4 : 3;
    static constexpr int AHEAD = NBUF - 2;
    // lines in the ring buffer: Q + 2R rounded up to a multiple of 8, so that every window of the column pass starts on
    // a multiple of 8 and wraps between two blocks of 8 lines (col_pass)
    static constexpr int RING = (Q + 2 * R + 7) / 8 * 8;
    static constexpr size_t smem = sizeof(float) * (NBUF * Q * SWP + RING * HBW);   // staging buffers + ring
    static_assert(R <= Q, "centre rows must still be in the two staging buffers");
    static_assert((Q * SWP * sizeof(float)) % 128 == 0, "staging buffers stay 128-byte aligned (TMA destination)");
    static_assert(SWP <= 256, "TMA box dimension");
};

__device__ __forceinline__ int clampi(int v, int lo, int hi) { return min(max(v, lo), hi); }

// ---- staging: source rows -> shared (TMA) ----------------------------------------------------------

__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, unsigned count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, unsigned bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, unsigned parity)
{
    unsigned ok, spins = 0;
    for (;;) {
        asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
                     : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
        if (ok) break;
        if (++spins > (1u << 24)) __trap();      // a copy that never lands must abort the launch, not hang the device
    }
}
// one box of the source plane -> shared; coordinates may lie outside the tensor (zero fill)
__device__ __forceinline__ void tma_load_2d(float* dst, const CUtensorMap* map, int x, int y, uint64_t* bar)
{
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 :: "r"(smem_u32(dst)), "l"(reinterpret_cast<unsigned long long>(map)), "r"(x), "r"(y), "r"(smem_u32(bar)) : "memory");
}
// one contiguous piece (16-byte aligned, multiple of 16 bytes) -> shared
__device__ __forceinline__ void bulk_load_1d(float* dst, const float* src, unsigned bytes, uint64_t* bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

// Stage chunk rows [iy, iy+Q) x columns [x0-RP, x0-RP+SWP) of `src` into S (row stride SWP); called by ONE thread.
// Interior chunks: one tensor copy (the box is SWP wide so that the shared-memory row stride is the conflict-free one;
// columns outside [0, W) arrive as zeros).  Chunks that cross the top / bottom border: Q row copies from the
// clamped rows, clipped to the row's storage (columns >= W hold padding; both cases are patched by patch_halo).
template <int R, bool EDGE>
__device__ __forceinline__ void stage_tma(const CUtensorMap* map, const float* __restrict__ src, int H, int pitch, int x0, int iy,
                                          float* __restrict__ S, uint64_t* bar)
{
    using G = Geo<R>;
    if (iy >= 0 && iy + Q <= H) {
        mbar_expect_tx(bar, (unsigned)(Q * G::SWP * sizeof(float)));
        tma_load_2d(S, map, x0 - G::RP, iy, bar);
    } else {
        const int gx0 = EDGE ? max(x0 - G::RP, 0) : x0 - G::RP;
        const int gx1 = EDGE ? min(x0 - G::RP + G::SW, pitch) : x0 - G::RP + G::SW;
        const unsigned bytes = (unsigned)(gx1 - gx0) * (unsigned)sizeof(float);
        mbar_expect_tx(bar, (unsigned)Q * bytes);
#pragma unroll 1
        for (int j = 0; j < Q; ++j) {
            const int gy = clampi(iy + j, 0, H - 1);
            bulk_load_1d(S + j * G::SWP + (gx0 - (x0 - G::RP)), src + (long long)gy * pitch + gx0, bytes, bar);
        }
    }
}

// EDGE strips: replicate the border column into the halo columns the copy skipped.  Outputs right of
// the image are never stored, so only R columns past the last image column have to be valid.
template <int R>
__device__ __forceinline__ void patch_halo(float* __restrict__ S, int x0, int W)
{
    using G = Geo<R>;
    const int j = threadIdx.x & (Q - 1);
    const int u = threadIdx.x >> 4;                      // 0..NT/Q-1
    float* row = S + j * G::SWP;
    if (x0 < G::RP) {                                    // left border: stage column RP - x0 is x = 0
        const int c0 = G::RP - x0;
        const float v = row[c0];
        for (int c = u; c < c0; c += NT / Q) row[c] = v;
    }
    const int cl = W - 1 - (x0 - G::RP);                 // stage column of x = W-1
    if (cl + 1 < G::SW) {
        const float v = row[cl];
        const int ce = min(cl + R, G::SW - 1);
        for (int c = cl + 1 + u; c <= ce; c += NT / Q) row[c] = v;
    }
    // these generic-proxy writes precede a later TMA write into the same buffer
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// ---- row pass: stage -> ring ------------------------------------------------------------------

template <int R, bool LEVEL0>
__device__ __forceinline__ void row_pass(const float* __restrict__ S, float* __restrict__ HB, int slot0, const Taps& t)
{
    using G = Geo<R>;
    const int j = threadIdx.x & (Q - 1);        // row of the chunk
    const int g = threadIdx.x >> 4;             // 16-column group (0..7)
    constexpr int WIN = 16 + 2 * G::RP;
    float w[WIN];
    const float* p = S + j * G::SWP + 16 * g;
#pragma unroll
    for (int m = 0; m < WIN / 4; ++m) {
        const float4 v = *reinterpret_cast<const float4*>(p + 4 * m);
        w[4 * m] = v.x; w[4 * m + 1] = v.y; w[4 * m + 2] = v.z; w[4 * m + 3] = v.w;
    }
    int slot = slot0 + j;
    if (slot >= G::RING) slot -= G::RING;
    float* o = HB + slot * HBW + 16 * g;
#pragma unroll
    for (int q4 = 0; q4 < 4; ++q4) {
        float r[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int c = 4 * q4 + u + G::RP;       // centre index in the window
            float acc;
            if (LEVEL0) {
                acc = 0.0f;
#pragma unroll
                for (int off = R; off > 0; --off) acc = __fmaf_rn(__fadd_rn(w[c - off], w[c + off]), t.g[off], acc);
                acc = __fmaf_rn(w[c], t.g[0], acc);
                acc = __fmul_rn(acc, 255.0f);
            } else {
                acc = __fmaf_rn(w[c], t.g[0], 0.0f);
#pragma unroll
                for (int off = R; off > 0; --off) acc = __fmaf_rn(__fadd_rn(w[c - off], w[c + off]), t.g[off], acc);
            }
            r[u] = acc;
        }
        *reinterpret_cast<float4*>(o + 4 * q4) = make_float4(r[0], r[1], r[2], r[3]);
    }
}

// ---- column pass: ring -> outputs ------------------------------------------------------------
//
// Thread = (pair of adjacent columns, half of the chunk's rows).  Both columns ride in one 64-bit
// register pair, so every tap is ONE packed FFMA2 (fma.rn.f32x2; the tap weight is a scalar
// uniform-register operand): half the FP32 issue slots of the scalar form, identical IEEE results.

typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pack2(float lo, float hi) { f32x2 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ void unpack2(f32x2 v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) { f32x2 d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d; }

constexpr int QH = Q / 2;   // output rows per thread in the column pass

// Candidates (CandSink): a lane notes the rows in which one of its two DoG samples passes the peak
// threshold -- one compare pair and one predicated OR per row in the hot loop -- and afterwards, if it
// has any, reserves entries of the block's list region with ONE shared-memory atomic and stores them.
template <int R, bool WRITE_DOG, bool NEXT, bool GUARD, bool CAND>
__device__ __forceinline__ void col_emit(const f32x2 (&win)[QH + 2 * R], const float* __restrict__ Scur,
                                         const float* __restrict__ Sprev, int jbase, int y_first, int ys, int ye,
                                         float* __restrict__ pd, float* __restrict__ pg, float* __restrict__ pn,
                                         int pitch, int next_pitch, const Taps& t, const CandSink& sink, int* cand_n, int x, int W)
{
    using G = Geo<R>;
    const int c2 = 2 * (threadIdx.x & 63);
    const int par = y_first & 1;
    const bool col_in = !GUARD || x < W;            // GUARD: the pair may start right of the image
    unsigned pm = 0;
#pragma unroll
    for (int jj = 0; jj < QH; ++jj) {
        f32x2 acc = pack2(0.0f, 0.0f);
#pragma unroll
        for (int off = R; off > 0; --off) {
            const f32x2 g2 = pack2(t.g[off], t.g[off]);
            acc = fma2(win[jj + R - off], g2, acc);
            acc = fma2(win[jj + R + off], g2, acc);
        }
        acc = fma2(win[jj + R], pack2(t.g[0], t.g[0]), acc);
        const int j = jbase + jj;                       // row of the chunk's output block (0..Q-1)
        const bool ok = !GUARD || (col_in && y_first + j >= ys && y_first + j < ye);
        if (ok) {
            *reinterpret_cast<f32x2*>(pd) = acc;
            float a0, a1;
            unpack2(acc, a0, a1);
            if (WRITE_DOG) {
                // centre source row: chunk-relative row j-R lives in the current (j >= R) or previous buffer
                const float* cp = (j >= R) ? Scur + (j - R) * G::SWP : Sprev + (j - R + Q) * G::SWP;
                const float2 cs = *reinterpret_cast<const float2*>(cp + G::RP + c2);
                const float g0 = __fsub_rn(a0, cs.x), g1 = __fsub_rn(a1, cs.y);
                *reinterpret_cast<float2*>(pg) = make_float2(g0, g1);
                if (CAND) {
                    // (a pair that straddles the right border may report garbage in its second sample: the
                    // extrema stage re-tests every sample and ignores border columns)
                    if (fabsf(g0) >= sink.thr || fabsf(g1) >= sink.thr) pm |= 1u << jj;
                }
            }
            if (NEXT && ((j & 1) == par)) pn[(size_t)((y_first + j) >> 1) * next_pitch] = a0;
        }
        pd += pitch;
        if (WRITE_DOG) pg += pitch;
    }
    if (CAND) {
        if (pm != 0u) {
            const int idx = atomicAdd(cand_n, __popc(pm));
            unsigned* out = sink.list + (size_t)blockIdx.x * sink.region + idx;
            const int y0 = y_first + jbase;
            do {
                const int b = __ffs(pm) - 1;
                pm &= pm - 1;
                *out++ = (unsigned)x | ((unsigned)(y0 + b) << 16);
            } while (pm);
        }
    }
}

template <int R, bool WRITE_DOG, bool NEXT, bool CAND = false>
__device__ __forceinline__ void col_pass(const float* __restrict__ HB, const float* __restrict__ Scur,
                                         const float* __restrict__ Sprev, int slot_oldest, int y_first,
                                         int ys, int ye, int x0, int W, float* __restrict__ dst, float* __restrict__ dog,
                                         float* __restrict__ next0, int pitch, int next_pitch, const Taps& t,
                                         const CandSink& sink = CandSink(), int* cand_n = nullptr)
{
    using G = Geo<R>;
    const int c2 = 2 * (threadIdx.x & 63);
    const int jbase = (threadIdx.x >> 6) * QH;          // 0 or Q/2 (warp-uniform)
    f32x2 win[QH + 2 * R];
    int first = slot_oldest + jbase;                    // ring slot of the first window line (warp-uniform, a multiple of 8)
    if (first >= G::RING) first -= G::RING;
    // `first` is the line Q + 2R' lines before the newest (R' = R rounded so that the ring is a multiple of 8); the window
    // proper starts PAD lines later.  It wraps around the ring at most once, and only between two blocks of 8 lines (RING,
    // the chunk height and the half-chunk offset are multiples of 8): one base-pointer select per block, every line at a
    // compile-time offset from it.
    constexpr int PAD = G::RING - Q - 2 * R;
    const int nb = (G::RING - first) >> 3;              // blocks before the wrap
    const float* a0 = HB + first * HBW + c2;
    const float* a1 = a0 - G::RING * HBW;
#pragma unroll
    for (int b = 0; b < (PAD + QH + 2 * R + 7) / 8; ++b) {
        const float* base = (b < nb) ? a0 : a1;
#pragma unroll
        for (int p = (8 * b > PAD ? 8 * b : PAD); p < 8 * b + 8 && p < PAD + QH + 2 * R; ++p)
            win[p - PAD] = *reinterpret_cast<const f32x2*>(base + p * HBW);
    }
    const int x = x0 + c2;
    const int yb = y_first + jbase;
    if (yb + QH <= ys || yb >= ye) return;                     // nothing of this half-block is inside the segment (warp-uniform)
    const long long o = (long long)yb * pitch + x;             // may point outside for guarded samples (never dereferenced)
    float* pd = dst + o;
    float* pg = WRITE_DOG ? dog + o : nullptr;
    float* pn = NEXT ? next0 + (x >> 1) : nullptr;
    if (yb >= ys && yb + QH <= ye && x0 + TW <= W)
        col_emit<R, WRITE_DOG, NEXT, false, CAND>(win, Scur, Sprev, jbase, y_first, ys, ye, pd, pg, pn, pitch, next_pitch, t, sink, cand_n, x, W);
    else
        col_emit<R, WRITE_DOG, NEXT, true, CAND>(win, Scur, Sprev, jbase, y_first, ys, ye, pd, pg, pn, pitch, next_pitch, t, sink, cand_n, x, W);
}

template <int R, bool EDGE, bool NEXT, bool CAND>
__device__ __forceinline__ void march_body(float* __restrict__ smem, uint64_t* __restrict__ full, const CUtensorMap* map,
                                           const float* __restrict__ src, float* __restrict__ dst,
                                           float* __restrict__ dog, float* __restrict__ next0, int W, int H, int pitch,
                                           int next_pitch, int x0, int ys, int ye, const Taps& taps, const CandSink& sink,
                                           int* cand_n)
{
    using G = Geo<R>;
    constexpr int SB = Q * G::SWP;         // floats per staging buffer (buffer b starts at smem + b*SB)
    constexpr int AHEAD = G::AHEAD;        // chunks in flight
    float* HB = smem + G::NBUF * SB;
    const int nchunks = (ye - ys + 2 * R + Q - 1) / Q;

    // staging of chunks k+1 .. k+AHEAD overlaps the computation of chunk k; thread 0 is the producer
    auto issue = [&](int k) {
        stage_tma<R, EDGE>(map, src, H, pitch, x0, ys - R + k * Q, smem + (k % G::NBUF) * SB, full + (k % G::NBUF));
    };
    if (threadIdx.x == 0) {
#pragma unroll
        for (int k = 0; k < AHEAD; ++k)
            if (k < nchunks) issue(k);
    }
    int slot_in = 0;                     // ring slot of the chunk's first input row
    int cur = 0;                         // staging buffer of chunk k
    unsigned parity = 0;                 // phase of full[cur]: flips every time cur wraps
    for (int k = 0; k < nchunks; ++k) {
        float* Scur = smem + cur * SB;
        float* Sprev = smem + (cur == 0 ? G::NBUF - 1 : cur - 1) * SB;
        mbar_wait(full + cur, parity);    // chunk k has landed
        __syncthreads();                  // column pass k-1 finished (ring + buffer of chunk k-2 are free)
        if (threadIdx.x == 0 && k + AHEAD < nchunks) issue(k + AHEAD);
        if (EDGE) {
            patch_halo<R>(Scur, x0, W);
            __syncthreads();
        }
        row_pass<R, false>(Scur, HB, slot_in, taps);
        __syncthreads();
        int slot_old = slot_in + Q;       // oldest line = the one after the newest
        if (slot_old >= G::RING) slot_old -= G::RING;
        col_pass<R, true, NEXT, CAND>(HB, Scur, Sprev, slot_old, ys - 2 * R + k * Q, ys, ye, x0, W, dst, dog, next0, pitch,
                                      next_pitch, taps, sink, cand_n);
        slot_in = slot_old;
        if (cur == G::NBUF - 1) { cur = 0; parity ^= 1u; } else ++cur;
    }
    __syncthreads();                      // last column pass finished
    if (CAND && threadIdx.x == 0) sink.counts[blockIdx.x] = *cand_n;
}

template <int R, bool NEXT, bool CAND>
__global__ void __launch_bounds__(NT, 4)
march_level_kernel(const __grid_constant__ CUtensorMap tmap, const float* __restrict__ src, float* __restrict__ dst,
                   float* __restrict__ dog, float* __restrict__ next0, int W, int H, int pitch, int next_pitch, Partition part,
                   Taps taps, CandSink sink)
{
    using G = Geo<R>;
    extern __shared__ __align__(128) float smem[];   // TMA destinations: 128-byte aligned (every staging buffer is)
    __shared__ __align__(8) uint64_t full[G::NBUF];  // one mbarrier per staging buffer
    __shared__ int s_cand_n;                         // candidates of this block so far
    int strip, ys, ye;
    if (!locate(part, blockIdx.x, H, Q, strip, ys, ye)) return;
    const int x0 = strip * TW;
    const bool edge = (x0 - G::RP < 0) || (x0 + TW + G::RP > W);
    if (threadIdx.x == 0) {
#pragma unroll
        for (int b = 0; b < G::NBUF; ++b) mbar_init(full + b, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        if (CAND) s_cand_n = 0;
    }
    __syncthreads();
    if (!edge) march_body<R, false, NEXT, CAND>(smem, full, &tmap, src, dst, dog, next0, W, H, pitch, next_pitch, x0, ys, ye, taps, sink, &s_cand_n);
    else       march_body<R, true, NEXT, CAND>(smem, full, &tmap, src, dst, dog, next0, W, H, pitch, next_pitch, x0, ys, ye, taps, sink, &s_cand_n);
}

// ---- octave 0, level 0 from the input image -----------------------------------------------------

using AxisTap = TexAxis;

// the coordinate the reference hands to tex2D for virtual sample X (s_pyramid_build.cu:108-131): (X + shift) / N0
__device__ __forceinline__ AxisTap virt_axis(int X, float shift, int N0, int n)
{
    return tex_axis(__fdiv_rn(__fadd_rn((float)X, shift), (float)N0), n);
}

// unorm16 -> float exactly as the texture unit: (float)r16 / 65535.0f, correctly rounded.
// int->float through the 2^23 trick and a 3-instruction division (q = x*c; q += c*fma(-q, 65535, x))
// that is exact for every r16 in [0, 65535] (exhaustively checked, tests/test_host_cpu.py).
__device__ __forceinline__ float unorm16_to_float(unsigned r16)
{
    const float x = __fsub_rn(__uint_as_float(0x4B000000u | r16), 8388608.0f);
    const float c = __uint_as_float(0x37800080u);      // RN(1/65535)
    const float q = __fmul_rn(x, c);
    const float rem = __fmaf_rn(-q, 65535.0f, x);
    return __fmaf_rn(rem, c, q);
}

// General path (any scale factor, 8-bit or float input): every staged sample is one emulated
// bilinear texture fetch.
template <int R, typename PIX, bool EXACT>
__device__ __forceinline__ void level0_body(float* __restrict__ smem, AxisTap* __restrict__ ax, AxisTap* __restrict__ ay,
                                            const PIX* __restrict__ img, size_t img_pitch, int w, int h, float shift,
                                            float* __restrict__ dst, int W, int H, int pitch, int x0, int ys, int ye,
                                            const Taps& dd, const Taps& inc0)
{
    using G = Geo<R>;
    float* S0 = smem;
    float* S1 = smem + Q * G::SWP;
    float* HB = smem + G::NBUF * Q * G::SWP;
    const int nchunks = (ye - ys + 2 * R + Q - 1) / Q;

    if (!EXACT) {
        for (int i = threadIdx.x; i < G::SW; i += NT) ax[i] = virt_axis(x0 - G::RP + i, shift, W, w);
        __syncthreads();
    }

    int slot_in = 0;
    for (int k = 0; k < nchunks; ++k) {
        float* Scur = (k & 1) ? S1 : S0;
        const int iy = ys - R + k * Q;
        // rows outside the octave clamp to the border row of the row-filtered plane
        if (threadIdx.x < Q) ay[threadIdx.x] = virt_axis(clampi(iy + threadIdx.x, 0, H - 1), shift, H, h);
        __syncthreads();
        if (EXACT) {
            // every tap at the reference's own coordinate: thread = column, one chunk row after the other
            static_assert(NT == TW, "one thread per output column");
            const int X = min(x0 + (int)threadIdx.x, W - 1);
            for (int j = 0; j < Q; ++j) {
                int slot = slot_in + j;
                if (slot >= G::RING) slot -= G::RING;
                HB[slot * HBW + threadIdx.x] = level0_row_sample<R, PIX>(img, img_pitch, w, ay[j], X, shift, W, dd);
            }
            __syncthreads();
        } else {
            for (int e = threadIdx.x; e < Q * G::SW; e += NT) {
                const int j = e / G::SW;
                const int i = e - j * G::SW;
                Scur[j * G::SWP + i] = tex_fetch(img, img_pitch, ax[i], ay[j]);
            }
            __syncthreads();
            row_pass<R, true>(Scur, HB, slot_in, dd);
            __syncthreads();
        }
        int slot_old = slot_in + Q;
        if (slot_old >= G::RING) slot_old -= G::RING;
        col_pass<R, false, false>(HB, Scur, Scur, slot_old, ys - 2 * R + k * Q, ys, ye, x0, W, dst, nullptr, nullptr, pitch, 0, inc0);
        slot_in = slot_old;
        __syncthreads();
    }
}

template <int R, typename PIX, bool EXACT>
__global__ void __launch_bounds__(NT)
march_level0_kernel(const PIX* __restrict__ img, size_t img_pitch, int w, int h, float shift,
                    float* __restrict__ dst, int W, int H, int pitch, Partition part, Taps dd, Taps inc0)
{
    using G = Geo<R>;
    extern __shared__ __align__(128) float smem[];
    __shared__ AxisTap ax[G::SW];
    __shared__ AxisTap ay[Q];
    int strip, ys, ye;
    if (!locate(part, blockIdx.x, H, Q, strip, ys, ye)) return;
    level0_body<R, PIX, EXACT>(smem, ax, ay, img, img_pitch, w, h, shift, dst, W, H, pitch, strip * TW, ys, ye, dd, inc0);
}

// ---- octave 0, level 0, the default case: 8-bit input, exactly 2x up-scaled -------------------------
//
// W == 2w, H == 2h, shift == 1.  Virtual sample (X, Y) then only depends on the SUM s4 of the 2x2 source
// texels {Y>>1, (Y+1)>>1} x {X>>1, (X+1)>>1} (indices repeat when a fraction is 0):
// r16 = (257*s4 + 2) >> 2, value = r16/65535.  Per chunk the CTA needs 9 source rows x (SW/2 + 1) bytes:
// they are staged as raw bytes with 4-byte cp.async two chunks ahead (the tile is < 1 KB), then
// "expanded" into the float staging buffer: thread = virtual column, the column's 9 row sums live in
// registers and the row pairing is static because the chunk's first row has the parity of R.
template <int R>
struct Geo0 {
    using G = Geo<R>;
    static constexpr int TROWS = Q / 2 + 2;             // source rows per tile (9 used away from the border)
    static constexpr int TSW = G::SW / 2 + 4;           // bytes per tile row (multiple of 4)
    static constexpr int PIECES = TROWS * (TSW / 4);    // 4-byte pieces per tile
    static constexpr int NP = (PIECES + NT - 1) / NT;
    static constexpr int AHEAD = 2, NRAW = AHEAD + 2;
    static constexpr int TAIL = G::SW - NT;             // staged columns beyond the first NT (= 2*RP)
    // float staging buffer, ring, raw tiles
    static constexpr size_t smem = sizeof(float) * (Q * G::SWP + G::RING * HBW) + (size_t)NRAW * TROWS * TSW;
    static_assert(TAIL >= 0 && TAIL <= NT, "one extra expand pass covers the halo columns");
};

__device__ __forceinline__ float s4_to_float(unsigned s4) { return unorm16_to_float((257u * s4 + 2u) >> 2); }

template <int R>
__global__ void __launch_bounds__(NT, 6)
march_level0x2_kernel(const uint8_t* __restrict__ img, size_t img_pitch, int w, int h,
                      float* __restrict__ dst, int W, int H, int pitch, Partition part, Taps dd, Taps inc0)
{
    using G = Geo<R>;
    using G0 = Geo0<R>;
    extern __shared__ __align__(128) float smem[];
    int strip, ys, ye;
    if (!locate(part, blockIdx.x, H, Q, strip, ys, ye)) return;
    const int x0 = strip * TW;
    float* S = smem;
    float* HB = smem + Q * G::SWP;
    uint8_t* T = reinterpret_cast<uint8_t*>(HB + G::RING * HBW);
    const int nchunks = (ye - ys + 2 * R + Q - 1) / Q;
    const int sx0 = ((x0 - G::RP) >> 1) & ~3;           // source column of tile byte 0 (may be negative)

    // tile offsets of the two source columns of this thread's virtual columns (main + halo tail)
    auto col_offsets = [&](int i, int& o0, int& o1) {
        const int X = x0 - G::RP + i;
        o0 = clampi(X >> 1, 0, w - 1) - sx0;
        o1 = clampi((X + 1) >> 1, 0, w - 1) - sx0;
    };
    int m0, m1, t0 = 0, t1 = 0;
    col_offsets(threadIdx.x, m0, m1);
    const bool has_tail = threadIdx.x < G0::TAIL;
    if (has_tail) col_offsets(NT + threadIdx.x, t0, t1);

    auto issue = [&](int k) {
        const int rbase = (ys - R + k * Q) >> 1;         // floor: tile row r holds source row clamp(rbase + r)
        uint8_t* Tk = T + (k % G0::NRAW) * (G0::TROWS * G0::TSW);
#pragma unroll
        for (int q = 0; q < G0::NP; ++q) {
            const int e = threadIdx.x + q * NT;
            const int r = e / (G0::TSW / 4);
            const int c4 = 4 * (e - r * (G0::TSW / 4));
            const int sc = sx0 + c4;
            if (e < G0::PIECES && sc >= 0 && sc < w) {
                const uint8_t* g = img + (size_t)clampi(rbase + r, 0, h - 1) * img_pitch + sc;
                const unsigned sa = (unsigned)__cvta_generic_to_shared(Tk + r * G0::TSW + c4);
                asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" :: "r"(sa), "l"(g) : "memory");
            }
        }
    };
    // expand one virtual column of chunk k: 16 staged samples
    auto expand = [&](int k, int i, int o0, int o1) {
        const int iy = ys - R + k * Q;
        const uint8_t* Tk = T + (k % G0::NRAW) * (G0::TROWS * G0::TSW);
        float* out = S + i;
        if (iy >= 0 && iy + Q < H && (iy & 1) == (R & 1)) {
            constexpr int P = R & 1;
            unsigned hs[Q / 2 + 1];
#pragma unroll
            for (int r = 0; r < Q / 2 + 1; ++r) hs[r] = (unsigned)Tk[r * G0::TSW + o0] + (unsigned)Tk[r * G0::TSW + o1];
#pragma unroll
            for (int j = 0; j < Q; ++j) out[j * G::SWP] = s4_to_float(hs[(P + j) >> 1] + hs[(P + j + 1) >> 1]);
        } else {
            const int rbase = iy >> 1;
            for (int j = 0; j < Q; ++j) {
                const int vy = clampi(iy + j, 0, H - 1);
                const int ra = clampi((vy >> 1) - rbase, 0, G0::TROWS - 1);
                const int rb = clampi(min((vy + 1) >> 1, h - 1) - rbase, 0, G0::TROWS - 1);
                const unsigned s4 = (unsigned)Tk[ra * G0::TSW + o0] + (unsigned)Tk[ra * G0::TSW + o1] +
                                    (unsigned)Tk[rb * G0::TSW + o0] + (unsigned)Tk[rb * G0::TSW + o1];
                out[j * G::SWP] = s4_to_float(s4);
            }
        }
    };

#pragma unroll
    for (int k = 0; k < G0::AHEAD; ++k) {
        if (k < nchunks) issue(k);
        asm volatile("cp.async.commit_group;" ::: "memory");
    }
    asm volatile("cp.async.wait_group %0;" :: "n"(G0::AHEAD - 1) : "memory");
    __syncthreads();                                      // tile 0 visible
    int slot_in = 0;
    for (int k = 0; k < nchunks; ++k) {
        // S was last read by row pass k-1 (before the barrier that ended iteration k-1's row pass)
        expand(k, threadIdx.x, m0, m1);
        if (has_tail) expand(k, NT + threadIdx.x, t0, t1);
        if (k + G0::AHEAD < nchunks) issue(k + G0::AHEAD);
        asm volatile("cp.async.commit_group;" ::: "memory");
        __syncthreads();                                  // chunk k expanded; column pass k-1 finished (ring free)
        row_pass<R, true>(S, HB, slot_in, dd);
        asm volatile("cp.async.wait_group %0;" :: "n"(G0::AHEAD - 1) : "memory");
        __syncthreads();                                  // ring lines of chunk k written; tile k+1 visible
        int slot_old = slot_in + Q;
        if (slot_old >= G::RING) slot_old -= G::RING;
        col_pass<R, false, false>(HB, S, S, slot_old, ys - 2 * R + k * Q, ys, ye, x0, W, dst, nullptr, nullptr, pitch, 0, inc0);
        slot_in = slot_old;
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
}

// ---- launch helpers ---------------------------------------------------------------------------

Partition make_partition(int W, int H, int slots = 0)     // one wave: SMs x 4 resident CTAs (592 on B200)
{
    return psb::make_partition(W, H, TW, Q, slots > 0 ? slots : 4 * sm_count());
}

template <int R, bool NEXT, bool CAND>
int launch_march(const Partition& part, const float* src, float* dst, float* dog, float* next0, const OctaveView& o,
                 int next_pitch, const Taps& t, const CandSink& sink, cudaStream_t st)
{
    ensure_smem(march_level_kernel<R, NEXT, CAND>, Geo<R>::smem, true);
    CUtensorMap map;
    if (!make_tmap_2d(&map, src, o.w, o.h, (size_t)o.pitch * sizeof(float), Geo<R>::SWP, Q, false)) return -2;
    march_level_kernel<R, NEXT, CAND><<<part.B, NT, Geo<R>::smem, st>>>(map, src, dst, dog, next0, o.w, o.h, o.pitch, next_pitch,
                                                                        part, t, sink);
    return 1;
}

template <int R>
int run_march(const OctaveView& o, int level, const Taps& t, float* next0, int next_pitch, const CandSink* sink, cudaStream_t st)
{
    const Partition part = make_partition(o.w, o.h);
    const float* src = o.gauss + o.plane * (level - 1);
    float* dst = o.gauss + o.plane * level;
    float* dog = o.dog + o.plane * (level - 1);
    const bool cand = sink && sink->list && o.w <= 65535 && o.h <= 65535 && sink->region == cand_region_cap(part, TW, Q);
    const CandSink cs = cand ? *sink : CandSink();
    if (next0) return cand ? launch_march<R, true, true>(part, src, dst, dog, next0, o, next_pitch, t, cs, st)
                           : launch_march<R, true, false>(part, src, dst, dog, next0, o, next_pitch, t, cs, st);
    return cand ? launch_march<R, false, true>(part, src, dst, dog, next0, o, next_pitch, t, cs, st)
                : launch_march<R, false, false>(part, src, dst, dog, next0, o, next_pitch, t, cs, st);
}

template <int R, typename PIX>
int run_march0(const PIX* img, size_t img_pitch, int w, int h, float shift, const OctaveView& o0, const Taps& dd,
               const Taps& inc0, int plan, cudaStream_t st)
{
    if constexpr (sizeof(PIX) == 1) {
        const bool x2 = plan == LEVEL0_IDEAL_X2 && shift == 1.0f && o0.w == 2 * w && o0.h == 2 * h && (img_pitch & 3) == 0 &&
                        (reinterpret_cast<uintptr_t>(img) & 3) == 0;
        if (x2) {
            // one wave: 26 KB of shared memory per CTA allows 6 resident CTAs per SM
            const Partition part = make_partition(o0.w, o0.h, 6 * sm_count());
            ensure_smem(march_level0x2_kernel<R>, Geo0<R>::smem, true);
            march_level0x2_kernel<R><<<part.B, NT, Geo0<R>::smem, st>>>(img, img_pitch, w, h, o0.gauss, o0.w, o0.h, o0.pitch,
                                                                        part, dd, inc0);
            return 1;
        }
    }
    const Partition part = make_partition(o0.w, o0.h);
    if (plan == LEVEL0_PER_TAP) {
        ensure_smem(march_level0_kernel<R, PIX, true>, Geo<R>::smem, true);
        march_level0_kernel<R, PIX, true><<<part.B, NT, Geo<R>::smem, st>>>(img, img_pitch, w, h, shift, o0.gauss, o0.w, o0.h,
                                                                            o0.pitch, part, dd, inc0);
    } else {
        ensure_smem(march_level0_kernel<R, PIX, false>, Geo<R>::smem, true);
        march_level0_kernel<R, PIX, false><<<part.B, NT, Geo<R>::smem, st>>>(img, img_pitch, w, h, shift, o0.gauss, o0.w, o0.h,
                                                                             o0.pitch, part, dd, inc0);
    }
    return 1;
}

} // namespace

bool march_supports(int R) { return R >= 3 && R <= 16; }
int march_cand_blocks(int w, int h) { return make_partition(w, h).B; }
int march_cand_region(int w, int h) { return cand_region_cap(make_partition(w, h), TW, Q); }
long long march_cand_entry_bound(int w, int h) { return cand_entry_bound(w, h, TW, Q, 4 * sm_count()); }

int march_blur_level(const OctaveView& o, int level, const Taps& t, int R, float* next0, int next_pitch,
                     const CandSink* sink, cudaStream_t st)
{
    switch (R) {
#define PSB_CASE(N) case N: return run_march<N>(o, level, t, next0, next_pitch, sink, st);
        PSB_CASE(3) PSB_CASE(4) PSB_CASE(5) PSB_CASE(6) PSB_CASE(7) PSB_CASE(8) PSB_CASE(9) PSB_CASE(10)
        PSB_CASE(11) PSB_CASE(12) PSB_CASE(13) PSB_CASE(14) PSB_CASE(15) PSB_CASE(16)
#undef PSB_CASE
        default: return -1;
    }
}

int march_level0_u8(const uint8_t* img, size_t img_pitch, int w, int h, float shift, const OctaveView& o0,
                    const Taps& dd, const Taps& inc0, int R, int plan, cudaStream_t st)
{
    switch (R) {
#define PSB_CASE(N) case N: return run_march0<N, uint8_t>(img, img_pitch, w, h, shift, o0, dd, inc0, plan, st);
        PSB_CASE(3) PSB_CASE(4) PSB_CASE(5) PSB_CASE(6) PSB_CASE(7) PSB_CASE(8) PSB_CASE(9)
#undef PSB_CASE
        default: return -1;
    }
}

int march_level0_f32(const float* img, size_t img_pitch, int w, int h, float shift, const OctaveView& o0,
                     const Taps& dd, const Taps& inc0, int R, int plan, cudaStream_t st)
{
    switch (R) {
#define PSB_CASE(N) case N: return run_march0<N, float>(img, img_pitch, w, h, shift, o0, dd, inc0, plan, st);
        PSB_CASE(3) PSB_CASE(4) PSB_CASE(5) PSB_CASE(6) PSB_CASE(7) PSB_CASE(8) PSB_CASE(9)
#undef PSB_CASE
        default: return -1;
    }
}

} // namespace psb
