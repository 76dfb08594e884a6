// Stage 1 -- Gaussian scale-space pyramid + DoG, hand-written for sm_100a.
//
// What the reference does with 13 launches per octave through textures and surfaces
// (normalizedSource::horiz, absoluteSource::horiz/vert, get_by_2_pick_every_second, make_dog;
// reference src/popsift/s_pyramid_build_ra.cu:17-55, s_pyramid_build_aa.cu:17-86,
// s_pyramid_build.cu:50-92,547-586) is done here with ONE kernel per level on linear HBM planes:
//   source tile (+halo, clamp-to-edge) -> shared memory -> row pass -> shared memory ->
//   column pass in registers -> level l, DoG[l-1] = G[l] - G[l-1] and (for level L) the
//   2:1 decimated level 0 of the next octave, all written from the same registers.
//
// Parity contract (tests/test_gpu_parity.py): every plane is BIT-IDENTICAL to the reference's.
// That fixes the floating-point evaluation order, taken from the reference's sm_100 SASS:
//   rows    (levels >= 1): acc = fma(C, g0, 0); for off = span-1..1: acc = fma(v(-off)+v(+off), g[off], acc)
//   rows    (level 0)    : acc = 0; for off = span-1..1: acc = fma(v(-off)+v(+off), g[off], acc);
//                          acc = fma(C, g0, acc); out = acc*255
//   columns (all levels) : acc = 0; for off = span-1..1: acc = fma(v(-off), g[off], acc);
//                          acc = fma(v(+off), g[off], acc); then acc = fma(C, g0, acc)
// (the reference also adds the +/-span taps, whose weight is exactly 0).
// All intrinsics are explicit (__fmaf_rn/__fadd_rn/__fmul_rn) so nvcc cannot re-associate.
#include "ps_internal.h"
#include "k_pyramid.h"
#include "k_texture.h"

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <tuple>

namespace psb {

namespace {

constexpr int TW = 64;          // output tile width
constexpr int TH = 32;          // output tile height
constexpr int NT = 256;         // threads per CTA

__device__ __forceinline__ int clampi(int v, int lo, int hi) { return min(max(v, lo), hi); }

// ---- row pass / column pass over shared-memory tiles ---------------------------------------

// s  : source tile, (TH+2R) rows x SW floats, column c <-> image x = x0 - R + c
// m  : row-filtered tile, (TH+2R) rows x TW floats
template <int R, bool LEVEL0>
__device__ __forceinline__ void row_pass(const float* __restrict__ s, float* __restrict__ m, int SW,
                                         const Taps& t)
{
    constexpr int ROWS = TH + 2 * R;
    for (int idx = threadIdx.x; idx < ROWS * TW; idx += NT) {
        const int j = idx / TW;
        const int i = idx - j * TW;
        const float* p = s + j * SW + i + R;     // centre
        float acc;
        if (LEVEL0) {
            acc = 0.0f;
#pragma unroll
            for (int off = R; off > 0; --off)
                acc = __fmaf_rn(__fadd_rn(p[-off], p[off]), t.g[off], acc);
            acc = __fmaf_rn(p[0], t.g[0], acc);
            acc = __fmul_rn(acc, 255.0f);
        } else {
            acc = __fmaf_rn(p[0], t.g[0], 0.0f);
#pragma unroll
            for (int off = R; off > 0; --off)
                acc = __fmaf_rn(__fadd_rn(p[-off], p[off]), t.g[off], acc);
        }
        m[j * TW + i] = acc;
    }
}

template <int R>
__device__ __forceinline__ float col_at(const float* __restrict__ m, int y, int x, const Taps& t)
{
    const float* p = m + (y + R) * TW + x;
    float acc = 0.0f;
#pragma unroll
    for (int off = R; off > 0; --off) {
        acc = __fmaf_rn(p[-off * TW], t.g[off], acc);
        acc = __fmaf_rn(p[off * TW], t.g[off], acc);
    }
    return __fmaf_rn(p[0], t.g[0], acc);
}

// ---- level l >= 1 ---------------------------------------------------------------------------

template <int R>
__global__ void __launch_bounds__(NT)
blur_level_kernel(const float* __restrict__ src, float* __restrict__ dst, float* __restrict__ dog,
                  float* __restrict__ next0, int W, int H, int pitch, int next_pitch, Taps taps)
{
    extern __shared__ float smem[];
    constexpr int SW = TW + 2 * R;
    constexpr int ROWS = TH + 2 * R;
    float* s = smem;                 // ROWS x SW
    float* m = smem + ROWS * SW;     // ROWS x TW

    const int x0 = blockIdx.x * TW;
    const int y0 = blockIdx.y * TH;

    for (int idx = threadIdx.x; idx < ROWS * SW; idx += NT) {
        const int j = idx / SW;
        const int i = idx - j * SW;
        const int gx = clampi(x0 - R + i, 0, W - 1);
        const int gy = clampi(y0 - R + j, 0, H - 1);
        s[idx] = __ldg(src + (size_t)gy * pitch + gx);
    }
    __syncthreads();
    row_pass<R, false>(s, m, SW, taps);
    __syncthreads();
    for (int idx = threadIdx.x; idx < TH * TW; idx += NT) {
        const int y = idx / TW;
        const int x = idx - y * TW;
        const int gx = x0 + x, gy = y0 + y;
        if (gx >= W || gy >= H) continue;
        const float v = col_at<R>(m, y, x, taps);
        const size_t o = (size_t)gy * pitch + gx;
        dst[o] = v;
        dog[o] = __fsub_rn(v, s[(y + R) * SW + x + R]);
        if (next0 != nullptr && !((gx | gy) & 1))
            next0[(size_t)(gy >> 1) * next_pitch + (gx >> 1)] = v;
    }
}

// generic-radius fallback (any span up to 31): same arithmetic, run-time loops
__global__ void __launch_bounds__(NT)
blur_level_generic_kernel(const float* __restrict__ src, float* __restrict__ dst, float* __restrict__ dog,
                          float* __restrict__ next0, int W, int H, int pitch, int next_pitch, Taps taps, int R)
{
    extern __shared__ float smem[];
    const int SW = TW + 2 * R;
    const int ROWS = TH + 2 * R;
    float* s = smem;
    float* m = smem + ROWS * SW;
    const int x0 = blockIdx.x * TW;
    const int y0 = blockIdx.y * TH;
    for (int idx = threadIdx.x; idx < ROWS * SW; idx += NT) {
        const int j = idx / SW;
        const int i = idx - j * SW;
        const int gx = clampi(x0 - R + i, 0, W - 1);
        const int gy = clampi(y0 - R + j, 0, H - 1);
        s[idx] = __ldg(src + (size_t)gy * pitch + gx);
    }
    __syncthreads();
    for (int idx = threadIdx.x; idx < ROWS * TW; idx += NT) {
        const int j = idx / TW;
        const int i = idx - j * TW;
        const float* p = s + j * SW + i + R;
        float acc = __fmaf_rn(p[0], taps.g[0], 0.0f);
        for (int off = R; off > 0; --off)
            acc = __fmaf_rn(__fadd_rn(p[-off], p[off]), taps.g[off], acc);
        m[j * TW + i] = acc;
    }
    __syncthreads();
    for (int idx = threadIdx.x; idx < TH * TW; idx += NT) {
        const int y = idx / TW;
        const int x = idx - y * TW;
        const int gx = x0 + x, gy = y0 + y;
        if (gx >= W || gy >= H) continue;
        const float* p = m + (y + R) * TW + x;
        float acc = 0.0f;
        for (int off = R; off > 0; --off) {
            acc = __fmaf_rn(p[-off * TW], taps.g[off], acc);
            acc = __fmaf_rn(p[off * TW], taps.g[off], acc);
        }
        const float v = __fmaf_rn(p[0], taps.g[0], acc);
        const size_t o = (size_t)gy * pitch + gx;
        dst[o] = v;
        dog[o] = __fsub_rn(v, s[(y + R) * SW + x + R]);
        if (next0 != nullptr && !((gx | gy) & 1))
            next0[(size_t)(gy >> 1) * next_pitch + (gx >> 1)] = v;
    }
}

// ---- octave 0, level 0: straight from the input image ----------------------------------------
//
// The reference samples a normalized-coordinate, bilinear, clamp, u8->unorm-float texture at
// ((X+shift)/W0 -/+ off/W0, (Y+shift)/H0).  What the B200 texture unit returns for that was
// measured (oracle/texprobe.cu, tests/golden/texture_pairs.npz): texel coordinate rx*w-0.5 with the
// fraction rounded to 1/256, texels widened to unorm16 (x257), integer 2x2 blend rounded half-up
// to 16 bits, result (float)r16/65535.  virt_axis() + sample below restate exactly that.

using AxisTap = TexAxis;

// the coordinate the reference hands to tex2D for virtual sample X (s_pyramid_build.cu:108-131): (X + shift) / N0
__device__ __forceinline__ AxisTap virt_axis(int X, float shift, int N0, int n)
{
    return tex_axis(__fdiv_rn(__fadd_rn((float)X, shift), (float)N0), n);
}

template <int R, typename PIX, bool EXACT>
__global__ void __launch_bounds__(NT)
level0_kernel(const PIX* __restrict__ img, size_t img_pitch, int w, int h, float shift,
              float* __restrict__ dst, int W, int H, int pitch, Taps dd, Taps inc0)
{
    extern __shared__ float smem[];
    constexpr int SW = TW + 2 * R;
    constexpr int ROWS = TH + 2 * R;
    float* s = smem;                 // ROWS x SW : virtual up-scaled image (normalised floats)
    float* m = smem + ROWS * SW;     // ROWS x TW
    __shared__ AxisTap ax[SW];
    __shared__ AxisTap ay[ROWS];

    const int x0 = blockIdx.x * TW;
    const int y0 = blockIdx.y * TH;
    // rows/columns outside the octave clamp to the border pixel of the *virtual* image first
    // (intermediate-plane clamp for rows; for columns the texture clamp is equivalent).
    if (!EXACT) for (int i = threadIdx.x; i < SW; i += NT) ax[i] = virt_axis(x0 - R + i, shift, W, w);
    for (int j = threadIdx.x; j < ROWS; j += NT) ay[j] = virt_axis(clampi(y0 - R + j, 0, H - 1), shift, H, h);
    __syncthreads();
    if (EXACT) {
        // LEVEL0_PER_TAP: every tap at the reference's own coordinate
        for (int idx = threadIdx.x; idx < ROWS * TW; idx += NT) {
            const int j = idx / TW;
            const int x = idx - j * TW;
            m[idx] = level0_row_sample<R, PIX>(img, img_pitch, w, ay[j], min(x0 + x, W - 1), shift, W, dd);
        }
    } else {
        for (int idx = threadIdx.x; idx < ROWS * SW; idx += NT) {
            const int j = idx / SW;
            const int i = idx - j * SW;
            s[idx] = tex_fetch(img, img_pitch, ax[i], ay[j]);
        }
        __syncthreads();
        row_pass<R, true>(s, m, SW, dd);
    }
    __syncthreads();
    for (int idx = threadIdx.x; idx < TH * TW; idx += NT) {
        const int y = idx / TW;
        const int x = idx - y * TW;
        const int gx = x0 + x, gy = y0 + y;
        if (gx >= W || gy >= H) continue;
        dst[(size_t)gy * pitch + gx] = col_at<R>(m, y, x, inc0);
    }
}

// Generic form of the level-0 kernel (run-time radii, any span up to 31): rows with `dd` (radius Rr), columns with `inc0`
// (radius Rc).  Used by --gauss-mode vlfeat-direct (VLFeat_Relative_All, reference s_pyramid_build_ra.cu:90-129 +
// s_pyramid_build_aa.cu:124-167), whose rows reach 21 taps a side.  exact != 0: every tap at the reference's own coordinate.
template <typename PIX>
__global__ void __launch_bounds__(NT)
level0_generic_kernel(const PIX* __restrict__ img, size_t img_pitch, int w, int h, float shift,
                      float* __restrict__ dst, int W, int H, int pitch, Taps dd, Taps inc0, int Rr, int Rc, int exact)
{
    extern __shared__ float smem[];
    const int SW = TW + 2 * Rr;
    const int ROWS = TH + 2 * Rc;
    float* s = smem;                 // ROWS x SW staged virtual samples (fetch-sharing form only)
    float* m = smem + ROWS * SW;     // ROWS x TW row-filtered
    const int x0 = blockIdx.x * TW;
    const int y0 = blockIdx.y * TH;
    if (exact) {
        for (int idx = threadIdx.x; idx < ROWS * TW; idx += NT) {
            const int j = idx / TW;
            const int x = idx - j * TW;
            const TexAxis ty = virt_axis(clampi(y0 - Rc + j, 0, H - 1), shift, H, h);
            const int X = min(x0 + x, W - 1);
            const float cx = tex_coord_centre(X, shift, W);
            float acc = 0.0f;
            for (int off = Rr; off > 0; --off) {
                const float v1 = tex_fetch(img, img_pitch, tex_axis(tex_coord_tap(cx, -off, W), w), ty);
                const float v2 = tex_fetch(img, img_pitch, tex_axis(tex_coord_tap(cx, off, W), w), ty);
                acc = __fmaf_rn(__fadd_rn(v1, v2), dd.g[off], acc);
            }
            acc = __fmaf_rn(tex_fetch(img, img_pitch, tex_axis(cx, w), ty), dd.g[0], acc);
            m[idx] = __fmul_rn(acc, 255.0f);
        }
    } else {
        for (int idx = threadIdx.x; idx < ROWS * SW; idx += NT) {
            const int j = idx / SW;
            const int i = idx - j * SW;
            s[idx] = tex_fetch(img, img_pitch, virt_axis(x0 - Rr + i, shift, W, w), virt_axis(clampi(y0 - Rc + j, 0, H - 1), shift, H, h));
        }
        __syncthreads();
        for (int idx = threadIdx.x; idx < ROWS * TW; idx += NT) {
            const int j = idx / TW;
            const int i = idx - j * TW;
            const float* p = s + j * SW + i + Rr;
            float acc = 0.0f;
            for (int off = Rr; off > 0; --off) acc = __fmaf_rn(__fadd_rn(p[-off], p[off]), dd.g[off], acc);
            acc = __fmaf_rn(p[0], dd.g[0], acc);
            m[idx] = __fmul_rn(acc, 255.0f);
        }
    }
    __syncthreads();
    for (int idx = threadIdx.x; idx < TH * TW; idx += NT) {
        const int y = idx / TW;
        const int x = idx - y * TW;
        const int gx = x0 + x, gy = y0 + y;
        if (gx >= W || gy >= H) continue;
        const float* p = m + (y + Rc) * TW + x;
        float acc = 0.0f;
        for (int off = Rc; off > 0; --off) {
            acc = __fmaf_rn(p[-off * TW], inc0.g[off], acc);
            acc = __fmaf_rn(p[off * TW], inc0.g[off], acc);
        }
        dst[(size_t)gy * pitch + gx] = __fmaf_rn(p[0], inc0.g[0], acc);
    }
}

// DoG planes of an octave whose levels were not produced by the fused blur + DoG kernels (reference make_dog,
// s_pyramid_build.cu:74-92): dog[l] = gauss[l + 1] - gauss[l]
__global__ void dog_planes_kernel(const float* __restrict__ gauss, float* __restrict__ dog, size_t plane, int nplanes, int W, int H, int pitch)
{
    const size_t n = (size_t)H * pitch;
    for (int l = 0; l < nplanes; ++l) {
        const float* a = gauss + plane * l;
        const float* b = a + plane;
        float* d = dog + plane * l;
        for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
            if ((int)(i % (size_t)pitch) < W) d[i] = __fsub_rn(b[i], a[i]);
    }
}

// level 0 of the next octave: every second pixel of level L (reference get_by_2_pick_every_second, s_pyramid_build.cu:50-71)
__global__ void decimate_kernel(const float* __restrict__ src, int Wp, int Hp, int pitch_p, float* __restrict__ dst, int W, int H, int pitch)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (x >= W || y >= H) return;
    dst[(size_t)y * pitch + x] = src[(size_t)clampi(2 * y, 0, Hp - 1) * pitch_p + clampi(2 * x, 0, Wp - 1)];
}

template <int R>
constexpr size_t tile_smem() { return sizeof(float) * ((TH + 2 * R) * (TW + 2 * R) + (TH + 2 * R) * TW); }

template <int R>
int run_blur(const OctaveView& o, int level, const Taps& t, float* next0, int next_pitch, cudaStream_t st)
{
    ensure_smem(blur_level_kernel<R>, tile_smem<R>());
    dim3 grid((o.w + TW - 1) / TW, (o.h + TH - 1) / TH);
    blur_level_kernel<R><<<grid, NT, tile_smem<R>(), st>>>(
        o.gauss + o.plane * (level - 1), o.gauss + o.plane * level, o.dog + o.plane * (level - 1),
        next0, o.w, o.h, o.pitch, next_pitch, t);
    return 1;
}

template <int R, typename PIX>
int run_level0(const PIX* img, size_t img_pitch, int w, int h, float shift, const OctaveView& o0,
               const Taps& dd, const Taps& inc0, int plan, cudaStream_t st)
{
    dim3 grid((o0.w + TW - 1) / TW, (o0.h + TH - 1) / TH);
    if (plan == LEVEL0_PER_TAP) {
        ensure_smem(level0_kernel<R, PIX, true>, tile_smem<R>());
        level0_kernel<R, PIX, true><<<grid, NT, tile_smem<R>(), st>>>(img, img_pitch, w, h, shift, o0.gauss, o0.w, o0.h,
                                                                      o0.pitch, dd, inc0);
    } else {
        ensure_smem(level0_kernel<R, PIX, false>, tile_smem<R>());
        level0_kernel<R, PIX, false><<<grid, NT, tile_smem<R>(), st>>>(img, img_pitch, w, h, shift, o0.gauss, o0.w, o0.h,
                                                                       o0.pitch, dd, inc0);
    }
    return 1;
}

// Which evaluation of level 0 is exact for this geometry: run the texture unit's coordinate arithmetic (k_texture.h,
// the same code the kernels use) over every output column and tap.  Sharing fetches between neighbouring outputs is
// exact when tap `off` of column X lands on the texels and fraction of column X+off's centre; the byte-tile kernel
// additionally needs the ideal 2x pattern on both axes.  Power-of-two scale factors of images up to a few thousand
// pixels pass; other scale factors and very wide images (the unit truncates the normalized coordinate to 21 bits)
// do not.  One evaluation per geometry, cached.
struct Level0Key { int w, h, W, H, R; unsigned shift; bool operator<(const Level0Key& o) const {
    return std::tie(w, h, W, H, R, shift) < std::tie(o.w, o.h, o.W, o.H, o.R, o.shift); } };

TexAxis canonical(TexAxis t)
{
    if (t.i0 == t.i1) t.a = 0;
    if (t.a == 0) t.i1 = t.i0;
    return t;
}
bool same_fetch(TexAxis a, TexAxis b)
{
    a = canonical(a); b = canonical(b);
    return a.i0 == b.i0 && a.i1 == b.i1 && a.a == b.a;
}

int level0_plan(int w, int h, int W, int H, float shift, int R)
{
    static std::mutex mu;
    static std::map<Level0Key, int> cache;
    Level0Key key{w, h, W, H, R, 0};
    memcpy(&key.shift, &shift, sizeof(shift));
    std::lock_guard<std::mutex> lk(mu);
    auto it = cache.find(key);
    if (it != cache.end()) return it->second;
    bool shared = true;
    for (int X = 0; X < W && shared; ++X) {
        const float cx = tex_coord_centre(X, shift, W);
        for (int off = -R; off <= R; ++off)
            if (!same_fetch(tex_axis(tex_coord_tap(cx, off, W), w), tex_axis(tex_coord_centre(X + off, shift, W), w))) { shared = false; break; }
    }
    bool ideal = shared && shift == 1.0f && W == 2 * w && H == 2 * h;
    auto ideal_axis = [](int X, int n) {
        TexAxis t;
        t.i0 = std::min(std::max(X >> 1, 0), n - 1);
        t.i1 = std::min(std::max((X + 1) >> 1, 0), n - 1);
        t.a = (X & 1) ? 128 : 0;
        return t;
    };
    for (int X = -R - 4; X < W + R + 4 && ideal; ++X) ideal = same_fetch(tex_axis(tex_coord_centre(X, shift, W), w), ideal_axis(X, w));
    for (int Y = 0; Y < H && ideal; ++Y) ideal = same_fetch(tex_axis(tex_coord_centre(Y, shift, H), h), ideal_axis(Y, h));
    return cache[key] = ideal ? LEVEL0_IDEAL_X2 : shared ? LEVEL0_SHARED : LEVEL0_PER_TAP;
}

// POPSIFT_B200_TILE_KERNELS=1 forces the simple tile kernels (debugging / A-B timing)
bool use_march()
{
    static const bool on = [] { const char* e = getenv("POPSIFT_B200_TILE_KERNELS"); return !(e && e[0] == '1'); }();
    return on;
}

Taps make_taps(const GaussRow& g)
{
    Taps t;
    for (int i = 0; i < PS_GAUSS_ALIGN; ++i) t.g[i] = g.tap[i];
    return t;
}

template <typename PIX>
int launch_level0_any(const PIX* img, size_t img_pitch, int w, int h, float upscale, int sift_mode,
                      const OctaveView& o0, const GaussRow& dd, const GaussRow& inc0, cudaStream_t st, int octave)
{
    // reference s_pyramid_build.cu:108-114
    float shift = 0.5f;
    if (octave == 0 && (sift_mode == PS_MODE_POPSIFT || sift_mode == PS_MODE_VLFEAT)) shift = 0.5f * powf(2.0f, upscale);
    // both passes use sigma_inc[0]; the two tables have the same span by construction
    const int R = (dd.span > inc0.span ? dd.span : inc0.span) - 1;
    const Taps a = make_taps(dd), b = make_taps(inc0);
    const int plan = level0_plan(w, h, o0.w, o0.h, shift, R);
    if (use_march()) {
        const int r = sizeof(PIX) == 1
            ? march_level0_u8(reinterpret_cast<const uint8_t*>(img), img_pitch, w, h, shift, o0, a, b, R, plan, st)
            : march_level0_f32(reinterpret_cast<const float*>(img), img_pitch, w, h, shift, o0, a, b, R, plan, st);
        if (r >= 0) return r;
    }
    switch (R) {
#define PSB_CASE(N) case N: return run_level0<N, PIX>(img, img_pitch, w, h, shift, o0, a, b, plan, st);
        PSB_CASE(1) PSB_CASE(2) PSB_CASE(3) PSB_CASE(4) PSB_CASE(5) PSB_CASE(6) PSB_CASE(7) PSB_CASE(8)
        PSB_CASE(9) PSB_CASE(10)
#undef PSB_CASE
        default: return -1;   // sigma0 <= 2.0 bounds the level-0 span at 10 (R <= 9) for any initial blur
    }
}

} // namespace

int level0_plan_for(int w, int h, int W, int H, float shift, int R) { return level0_plan(w, h, W, H, shift, R); }

int launch_level0_u8(const uint8_t* img, size_t img_pitch, int w, int h, float upscale, int sift_mode,
                     const OctaveView& o0, const GaussRow& dd, const GaussRow& inc0, cudaStream_t st, int octave)
{
    return launch_level0_any<uint8_t>(img, img_pitch, w, h, upscale, sift_mode, o0, dd, inc0, st, octave);
}

int launch_level0_f32(const float* img, size_t img_pitch_floats, int w, int h, float upscale, int sift_mode,
                      const OctaveView& o0, const GaussRow& dd, const GaussRow& inc0, cudaStream_t st, int octave)
{
    return launch_level0_any<float>(img, img_pitch_floats, w, h, upscale, sift_mode, o0, dd, inc0, st, octave);
}

bool blur_level_collects(const GaussRow& g) { return use_march() && march_supports(g.span - 1); }
int cand_blocks_for(int w, int h) { return march_cand_blocks(w, h); }
int cand_region_for(int w, int h) { return march_cand_region(w, h); }
long long cand_entry_bound_for(int w, int h) { return march_cand_entry_bound(w, h); }

int launch_blur_level(const OctaveView& o, int level, const GaussRow& g, const OctaveView* next, const CandSink* sink,
                      cudaStream_t st)
{
    const int R = g.span - 1;
    const Taps t = make_taps(g);
    float* next0 = next ? next->gauss : nullptr;
    const int next_pitch = next ? next->pitch : 0;
    if (use_march()) {
        const int r = march_blur_level(o, level, t, R, next0, next_pitch, sink, st);
        if (r >= 0) return r;
    }
    switch (R) {
        case 5:  return run_blur<5>(o, level, t, next0, next_pitch, st);
        case 7:  return run_blur<7>(o, level, t, next0, next_pitch, st);
        case 8:  return run_blur<8>(o, level, t, next0, next_pitch, st);
        case 10: return run_blur<10>(o, level, t, next0, next_pitch, st);
        case 13: return run_blur<13>(o, level, t, next0, next_pitch, st);
        default: break;
    }
    {
        const int Rm = PS_GAUSS_ALIGN - 2;
        ensure_smem(blur_level_generic_kernel, sizeof(float) * ((TH + 2 * Rm) * (TW + 2 * Rm) + (TH + 2 * Rm) * TW));
    }
    const size_t sm = sizeof(float) * ((TH + 2 * R) * (TW + 2 * R) + (TH + 2 * R) * TW);
    dim3 grid((o.w + TW - 1) / TW, (o.h + TH - 1) / TH);
    blur_level_generic_kernel<<<grid, NT, sm, st>>>(o.gauss + o.plane * (level - 1), o.gauss + o.plane * level,
                                                    o.dog + o.plane * (level - 1), next0, o.w, o.h, o.pitch,
                                                    next_pitch, t, R);
    return 1;
}

// --gauss-mode relative / vlfeat-hw-interpolated (VLFeat_Relative; reference absoluteSourceInterpolated::horiz / vert,
// s_pyramid_build_ai.cu:17-66): pairs of taps are merged into ONE linearly interpolated fetch of the unnormalized float
// texture at distance off = offset + (1 - u).  The texture unit's arithmetic there, measured with `texprobe lcoords`
// (tests/golden/texture_lcoords.npz, oracle orc_tex_lin1d): texel position c - 0.5 rounded half-up to 1/256 and clamped
// to [0, n-1], then the 8-bit-weight blend of every float texture (tex_blend_f32).  Order from the reference's SASS:
// off = offset + (1 - u); coordinate (x -/+ off) + 0.5; val = tex(-) + tex(+); out = fma(val, v, out); centre last.
__device__ __forceinline__ float tex_lin1d(const float* __restrict__ base, long long stride, int n, float c)
{
    double I = floor(__fma_rn(__dsub_rn((double)c, 0.5), 256.0, 0.5));
    I = fmin(fmax(I, 0.0), (double)(n - 1) * 256.0);
    const long long Ii = (long long)I;
    const int i = (int)(Ii >> 8), a = (int)(Ii & 255);
    const int i1 = min(i + 1, n - 1);
    return tex_blend_f32(__ldg(base + i * stride), __ldg(base + i1 * stride), 0.0f, 0.0f, a, 0);
}

template <bool ALONG_X>
__global__ void __launch_bounds__(256)
interp_pass_kernel(const float* __restrict__ src, float* __restrict__ dst, int W, int H, int pitch, Taps f, int span)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (x >= W || y >= H) return;
    const float* base = ALONG_X ? src + (size_t)y * pitch : src + x;
    const long long stride = ALONG_X ? 1 : pitch;
    const int n = ALONG_X ? W : H;
    const float pos = (float)(ALONG_X ? x : y);
    float out = 0.0f;
    for (int offset = 1; offset <= span; offset += 2) {
        const float u = f.g[offset];
        const float off = __fadd_rn((float)offset, __fsub_rn(1.0f, u));
        const float t0 = tex_lin1d(base, stride, n, __fadd_rn(__fsub_rn(pos, off), 0.5f));
        const float t1 = tex_lin1d(base, stride, n, __fadd_rn(__fadd_rn(pos, off), 0.5f));
        out = __fmaf_rn(__fadd_rn(t0, t1), f.g[offset + 1], out);
    }
    dst[(size_t)y * pitch + x] = __fmaf_rn(__ldg(src + (size_t)y * pitch + x), f.g[0], out);
}

// --gauss-mode fixed9 / fixed15 (reference s_pyramid_fixed.cu): every level is filtered VERTICALLY first, then horizontally,
// with a fixed half width S = 4 / 7.  Accumulation order from the reference's SASS (all four octave_fixed kernels):
// acc = pair_1 * f[1]; acc = fma(centre, f[0], acc); acc = fma(pair_i, f[i], acc) for i = 2..S.
__device__ __forceinline__ float fixed_acc(const float* v /* 2S+1 values, centre at v[S] */, int stride, const Taps& f, int S)
{
    float acc = __fmul_rn(__fadd_rn(v[(S - 1) * stride], v[(S + 1) * stride]), f.g[1]);
    acc = __fmaf_rn(v[S * stride], f.g[0], acc);
    for (int i = 2; i <= S; ++i) acc = __fmaf_rn(__fadd_rn(v[(S - i) * stride], v[(S + i) * stride]), f.g[i], acc);
    return acc;
}

// vertical pass of octave 0 (relativeTexAddress::octave_fixed_vert, s_pyramid_fixed.cu:127-146) for the virtual columns
// -S .. W-1+S: fetches of the input texture at ((col + tshift) * rcp(W), fma(-/+i, rcp(H), (row + tshift) * rcp(H)))
template <typename PIX>
__global__ void __launch_bounds__(256)
fixed_vert0_kernel(const PIX* __restrict__ img, size_t img_pitch, int w, int h, float tshift, float* __restrict__ V, int vpitch,
                   int W, int H, Taps f, int S)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (k >= W + 2 * S || y >= H) return;
    const float mul_w = __frcp_rn((float)W), mul_h = __frcp_rn((float)H);
    const float xpos = __fmul_rn(__fadd_rn((float)(k - S), tshift), mul_w);
    const float ypos = __fmul_rn(__fadd_rn((float)y, tshift), mul_h);
    const TexAxis tx = tex_axis(xpos, w);
    float v[2 * 7 + 1];
    for (int i = -S; i <= S; ++i) v[S + i] = tex_fetch(img, img_pitch, tx, tex_axis(__fmaf_rn((float)i, mul_h, ypos), h));
    V[(size_t)y * vpitch + k] = fixed_acc(v, 1, f, S);
}

// vertical pass of octaves >= 1 (absoluteTexAddress::octave_fixed_vert, s_pyramid_fixed.cu:46-66): from level 0 of the octave,
// clamp addressing; also for the virtual columns -S .. W-1+S (= the clamped columns)
__global__ void __launch_bounds__(256)
fixed_vertN_kernel(const float* __restrict__ src, int pitch, float* __restrict__ V, int vpitch, int W, int H, Taps f, int S)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (k >= W + 2 * S || y >= H) return;
    const int x = clampi(k - S, 0, W - 1);
    float v[2 * 7 + 1];
    for (int i = -S; i <= S; ++i) v[S + i] = __ldg(src + (size_t)clampi(y + i, 0, H - 1) * pitch + x);
    V[(size_t)y * vpitch + k] = fixed_acc(v, 1, f, S);
}

// horizontal pass (octave_fixed_horiz, s_pyramid_fixed.cu:24-44: shuffles there, the row of vertical results here)
__global__ void __launch_bounds__(256)
fixed_horiz_kernel(const float* __restrict__ V, int vpitch, float* __restrict__ dst, int pitch, int W, int H, Taps f, int S, int times255)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (x >= W || y >= H) return;
    const float out = fixed_acc(V + (size_t)y * vpitch + x, 1, f, S);
    dst[(size_t)y * pitch + x] = times255 ? __fmul_rn(out, 255.0f) : out;
}

// --gauss-mode vlfeat-direct: level `level` of octave 0 straight from the input image with `taps` in both directions
template <typename PIX>
static int launch_level0_abs_any(const PIX* img, size_t img_pitch, int w, int h, float upscale, int sift_mode,
                                 const OctaveView& o0, int level, const GaussRow& taps, cudaStream_t st)
{
    float shift = 0.5f;
    if (sift_mode == PS_MODE_POPSIFT || sift_mode == PS_MODE_VLFEAT) shift = 0.5f * powf(2.0f, upscale);
    const int R = taps.span - 1;
    if (R < 0 || R >= PS_GAUSS_ALIGN) return -1;
    const Taps t = make_taps(taps);
    const int plan = level0_plan(w, h, o0.w, o0.h, shift, R);
    const size_t sm = sizeof(float) * ((size_t)(TH + 2 * R) * (TW + 2 * R) + (size_t)(TH + 2 * R) * TW);
    constexpr int RMAX = PS_GAUSS_ALIGN - 1;      // the opt-in is made once per kernel: ask for the largest radius
    ensure_smem(level0_generic_kernel<PIX>, sizeof(float) * ((size_t)(TH + 2 * RMAX) * (TW + 2 * RMAX) + (size_t)(TH + 2 * RMAX) * TW));
    dim3 grid((o0.w + TW - 1) / TW, (o0.h + TH - 1) / TH);
    level0_generic_kernel<PIX><<<grid, NT, sm, st>>>(img, img_pitch, w, h, shift, o0.gauss + o0.plane * level, o0.w, o0.h, o0.pitch,
                                                     t, t, R, R, plan == LEVEL0_PER_TAP ? 1 : 0);
    return 1;
}
int launch_level0_abs_u8(const uint8_t* img, size_t img_pitch, int w, int h, float upscale, int sift_mode,
                         const OctaveView& o0, int level, const GaussRow& taps, cudaStream_t st)
{
    return launch_level0_abs_any<uint8_t>(img, img_pitch, w, h, upscale, sift_mode, o0, level, taps, st);
}
int launch_level0_abs_f32(const float* img, size_t img_pitch_floats, int w, int h, float upscale, int sift_mode,
                          const OctaveView& o0, int level, const GaussRow& taps, cudaStream_t st)
{
    return launch_level0_abs_any<float>(img, img_pitch_floats, w, h, upscale, sift_mode, o0, level, taps, st);
}
int launch_dog_planes(const OctaveView& o, int nplanes, cudaStream_t st)
{
    dog_planes_kernel<<<sm_count() * 8, 256, 0, st>>>(o.gauss, o.dog, o.plane, nplanes, o.w, o.h, o.pitch);
    return 1;
}
int launch_decimate(const OctaveView& prev, int level, const OctaveView& next, cudaStream_t st)
{
    dim3 grid((next.w + 127) / 128, next.h);
    decimate_kernel<<<grid, 128, 0, st>>>(prev.gauss + prev.plane * level, prev.w, prev.h, prev.pitch, next.gauss, next.w, next.h, next.pitch);
    return 1;
}

// one interpolated pass (rows: along_x != 0) over a plane; `f` = the transformed row (gauss_filter.cu:372-405), span its i_span
int launch_interp_pass(const float* src, float* dst, int W, int H, int pitch, const GaussRow& f, int ispan, int along_x, cudaStream_t st)
{
    if (ispan < 1 || ispan >= PS_GAUSS_ALIGN) return -1;
    const Taps t = make_taps(f);
    dim3 grid((W + 255) / 256, H);
    if (along_x) interp_pass_kernel<true><<<grid, 256, 0, st>>>(src, dst, W, H, pitch, t, ispan);
    else         interp_pass_kernel<false><<<grid, 256, 0, st>>>(src, dst, W, H, pitch, t, ispan);
    return 1;
}
// rows of octave 0 straight from the input image (the first horizontal pass alone) into `dst` (pitch of the octave)
template <typename PIX>
static int launch_level0_rows_any(const PIX* img, size_t img_pitch, int w, int h, float upscale, int sift_mode,
                                  const OctaveView& o0, float* dst, const GaussRow& dd, cudaStream_t st, int octave)
{
    float shift = 0.5f;
    if (octave == 0 && (sift_mode == PS_MODE_POPSIFT || sift_mode == PS_MODE_VLFEAT)) shift = 0.5f * powf(2.0f, upscale);
    const int R = dd.span - 1;
    if (R < 0 || R >= PS_GAUSS_ALIGN) return -1;
    const Taps t = make_taps(dd);
    Taps ident;
    for (int i = 0; i < PS_GAUSS_ALIGN; ++i) ident.g[i] = 0.0f;
    ident.g[0] = 1.0f;                            // column pass of radius 0 with weight 1: fma(v, 1, 0) == v
    const int plan = level0_plan(w, h, o0.w, o0.h, shift, R);
    const size_t sm = sizeof(float) * ((size_t)TH * (TW + 2 * R) + (size_t)TH * TW);
    constexpr int RMAX = PS_GAUSS_ALIGN - 1;
    ensure_smem(level0_generic_kernel<PIX>, sizeof(float) * ((size_t)(TH + 2 * RMAX) * (TW + 2 * RMAX) + (size_t)(TH + 2 * RMAX) * TW));
    dim3 grid((o0.w + TW - 1) / TW, (o0.h + TH - 1) / TH);
    level0_generic_kernel<PIX><<<grid, NT, sm, st>>>(img, img_pitch, w, h, shift, dst, o0.w, o0.h, o0.pitch, t, ident, R, 0,
                                                     plan == LEVEL0_PER_TAP ? 1 : 0);
    return 1;
}
int launch_level0_rows_u8(const uint8_t* img, size_t img_pitch, int w, int h, float upscale, int sift_mode,
                          const OctaveView& o0, float* dst, const GaussRow& dd, cudaStream_t st, int octave)
{
    return launch_level0_rows_any<uint8_t>(img, img_pitch, w, h, upscale, sift_mode, o0, dst, dd, st, octave);
}
int launch_level0_rows_f32(const float* img, size_t img_pitch_floats, int w, int h, float upscale, int sift_mode,
                           const OctaveView& o0, float* dst, const GaussRow& dd, cudaStream_t st, int octave)
{
    return launch_level0_rows_any<float>(img, img_pitch_floats, w, h, upscale, sift_mode, o0, dst, dd, st, octave);
}

// --gauss-mode fixed9 / fixed15: one level of an octave; `scratch` holds (W + 2S rounded up to 32) x H floats
int launch_fixed_level0_u8(const uint8_t* img, size_t img_pitch, int w, int h, float upscale, const OctaveView& o0, int level,
                           const GaussRow& taps, int S, float* scratch, cudaStream_t st)
{
    const Taps t = make_taps(taps);
    const int vpitch = (o0.w + 2 * S + 31) / 32 * 32;
    dim3 gv((o0.w + 2 * S + 255) / 256, o0.h), gh((o0.w + 255) / 256, o0.h);
    fixed_vert0_kernel<uint8_t><<<gv, 256, 0, st>>>(img, img_pitch, w, h, 0.5f * powf(2.0f, upscale), scratch, vpitch, o0.w, o0.h, t, S);
    fixed_horiz_kernel<<<gh, 256, 0, st>>>(scratch, vpitch, o0.gauss + o0.plane * level, o0.pitch, o0.w, o0.h, t, S, 1);
    return 2;
}
int launch_fixed_level0_f32(const float* img, size_t img_pitch_floats, int w, int h, float upscale, const OctaveView& o0, int level,
                            const GaussRow& taps, int S, float* scratch, cudaStream_t st)
{
    const Taps t = make_taps(taps);
    const int vpitch = (o0.w + 2 * S + 31) / 32 * 32;
    dim3 gv((o0.w + 2 * S + 255) / 256, o0.h), gh((o0.w + 255) / 256, o0.h);
    fixed_vert0_kernel<float><<<gv, 256, 0, st>>>(img, img_pitch_floats, w, h, 0.5f * powf(2.0f, upscale), scratch, vpitch, o0.w, o0.h, t, S);
    fixed_horiz_kernel<<<gh, 256, 0, st>>>(scratch, vpitch, o0.gauss + o0.plane * level, o0.pitch, o0.w, o0.h, t, S, 1);
    return 2;
}
int launch_fixed_levelN(const OctaveView& o, int level, const GaussRow& taps, int S, float* scratch, cudaStream_t st)
{
    const Taps t = make_taps(taps);
    const int vpitch = (o.w + 2 * S + 31) / 32 * 32;
    dim3 gv((o.w + 2 * S + 255) / 256, o.h), gh((o.w + 255) / 256, o.h);
    fixed_vertN_kernel<<<gv, 256, 0, st>>>(o.gauss, o.pitch, scratch, vpitch, o.w, o.h, t, S);
    fixed_horiz_kernel<<<gh, 256, 0, st>>>(scratch, vpitch, o.gauss + o.plane * level, o.pitch, o.w, o.h, t, S, 0);
    return 2;
}

} // namespace psb
