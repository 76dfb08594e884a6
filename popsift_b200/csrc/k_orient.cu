// Stage 3a -- dominant orientations, hand-written for sm_100a.
//
// Replaces ori_par + ori_prefix_sum (reference src/popsift/s_orientation.cu:75-362,
// s_gradiant.h:55-69, common/warp_bitonic_sort.h, common/excl_blk_prefix_sum.h).
// Differences in structure (not in arithmetic):
//   * no host round trip: the reference reads the extrema counters back to size its grid
//     (s_orientation.cu:364-441); here a fixed grid of warps walks the device-side counters;
//   * all octaves in one launch, 4 keypoints (warps) per CTA instead of 1;
//   * the histogram is accumulated exactly like the reference's: one warp per keypoint, lane i takes samples
//     i, i+32, ... and adds its weight with a shared-memory float atomicAdd (ATOMS.CAST.SPIN loop), all
//     in-circle lanes of an iteration together.  The order in which the hardware serialises lanes that hit
//     the same bin is fixed for a converged warp (the reference reproduces its own output bit for bit on
//     the 32 benchmark frames, tests/golden/bench32_parity.json), so the same instruction on the same
//     lane <-> sample assignment gives the same float sums, hence the same peaks, the same number of
//     orientations and the same angles.  (Round 1 summed lane-private bins in lane order: 925 of 453 753
//     keypoints of the benchmark frames then differed in the last bits of an angle, and 7 in the NUMBER of
//     orientations -- 522 535 vs 522 542 descriptors.);
//   * top-4 selection by four warp arg-max rounds instead of a 64-wide bitonic sort.
// Per-sample math is the reference's: hypotf/atan2f gradients of the data plane lpos,
// weight = grad*expf(int(sq_dist)*__fdividef(-0.5, sigw^2)), bin = round(36*(theta+pi)/2pi),
// 3x(box3, box3) smoothing, parabola refinement, peaks >= 0.8*best, theta = fma(2pi*bin, 1/36, -pi).
#include "ps_internal.h"

namespace psb {

namespace {

constexpr int kWarps = 4;        // keypoints (warps) per CTA
constexpr int kBatch = 4;        // window iterations evaluated together
constexpr int kSlice = PS_ORI_SLICE;   // extrema per slice of the descriptor-index scan (ori_scatter_kernel)
__device__ const float kPi  = 3.14159265358979323846f;
__device__ const float kPi2 = 2.0f * 3.14159265358979323846f;

// total number of extrema and the octave prefix, from the raw per-octave counters
__device__ __forceinline__ int octave_prefix(const Counters* ct, const Consts& k, int num_octaves, int* ps /*[kMaxOctaves+1]*/)
{
    int total = 0;
    const int* counts = ct->filtered ? ct->ext_ct_f : ct->ext_ct;      // after the grid filter: the survivors
    for (int o = 0; o < num_octaves; ++o) {
        ps[o] = total;
        int c = min(counts[o], k.max_extrema);
        if (total + c > k.ext_capacity) c = k.ext_capacity - total;
        total += c;
    }
    ps[num_octaves] = total;
    return total;
}

__global__ void __launch_bounds__(kWarps * 32)
orientation_kernel(PyramidView pyr, Consts k, const InitialExtremum* __restrict__ iext_all, const InitialExtremum* __restrict__ iext_f,
                   ps_extremum* __restrict__ ext, int* __restrict__ slice_sum, Counters* ct)
{
    const InitialExtremum* __restrict__ iext = ct->filtered ? iext_f : iext_all;
    __shared__ float sm_a[kWarps][kOriBins];
    __shared__ float sm_b[kWarps][kOriBins];
    __shared__ int   ps[kMaxOctaves + 1];

    if (threadIdx.x == 0) octave_prefix(ct, k, pyr.num_octaves, ps);
    __syncthreads();
    const int total = ps[pyr.num_octaves];
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    float* A = sm_a[warp];
    float* B = sm_b[warp];

    // Keypoints cost between ~150 and ~1100 samples and a resident warp only gets about three of them, so a static
    // assignment leaves the SMs 72 % busy on average; every warp instead draws its next keypoint from a device-side
    // cursor (zeroed with the frame's counters), one draw ahead so that the atomic's latency hides behind the current one.
    int pend = 0;
    if (lane == 0) pend = atomicAdd(&ct->work_ori, 1);
    for (;;) {
        const int item = __shfl_sync(0xffffffffu, pend, 0);
        if (item >= total) break;
        if (lane == 0) pend = atomicAdd(&ct->work_ori, 1);
        int o = 0;
        while (o + 1 < pyr.num_octaves && item >= ps[o + 1]) ++o;
        const InitialExtremum ie = iext[(size_t)o * k.max_extrema + (item - ps[o])];
        const OctaveView& ov = pyr.oct[o];
        const int w = ov.w, h = ov.h;
        const int lvl = min(max(ie.lpos, 0), pyr.levels + 2);
        const float* pl = ov.gauss + (size_t)lvl * ov.plane;

        for (int b = lane; b < kOriBins; b += 32) A[b] = 0.0f;
        __syncwarp();

        const float x = ie.xpos, y = ie.ypos, sig = ie.sigma;
        const float sigw = __fmul_rn(1.5f, sig);
        const int rad = (int)roundf(__fmul_rn(3.0f, sigw));
        const float factor = __fdividef(-0.5f, __fmul_rn(sigw, sigw));
        const int sq_thres = rad * rad;
        const int xmin = max(1, (int)roundf(x) - rad);
        const int xmax = min(w - 2, (int)roundf(x) + rad);
        const int ymin = max(1, (int)roundf(y) - rad);
        const int ymax = min(h - 2, (int)roundf(y) + rad);
        const int wx = xmax - xmin + 1;
        const int hy = ymax - ymin + 1;
        const int loops = (wx > 0 && hy > 0) ? wx * hy : 0;

        // Sample i of the window is row i / wx, column i % wx, and belongs to lane i % 32, iteration i / 32
        // (reference s_orientation.cu:117-163).  The lane walks its samples with a running (row, column)
        // instead of a division per sample; the window lies inside [1, w-2] x [1, h-2], so the four
        // neighbours need no clamping; hypotf / atan2f / expf only run for samples inside the circle.
        // All lanes of an iteration reconverge before the atomic, like the reference's warp does.
        int xx = xmin + lane, yy = ymin;
        while (xx > xmax && wx > 0) { xx -= wx; ++yy; }
        // kBatch iterations are evaluated together -- positions first, then all gradient loads (samples outside the window
        // or the circle read the window's first pixel and are dropped afterwards), then the hypotf / atan2f / expf chains side
        // by side -- and their atomics issued in iteration order: per bin, the adds still arrive iteration by iteration, the
        // lanes of one iteration together.
        const float* safe = pl + (max(ymin, 1) * ov.pitch + max(xmin, 1));
        for (int i0 = 0; i0 < loops; i0 += 32 * kBatch) {
            int bidx[kBatch], sq[kBatch];
            float weight[kBatch];
            const float* p[kBatch];
#pragma unroll
            for (int u = 0; u < kBatch; ++u) {
                sq[u] = -1; p[u] = safe;
                if (i0 + 32 * u + lane < loops) {
                    const float ddx = __fsub_rn((float)xx, x), ddy = __fsub_rn((float)yy, y);
                    // reference SASS (ori_par): FMUL dx*dx, then FFMA dy*dy + that, F2I.TRUNC -- the contraction nvcc chose;
                    // the other operand order differs in the last bit often enough to move int(sq_dist) for about one
                    // keypoint in a thousand (a 1 % change of one sample's weight, angles off by ~1e-5 rad)
                    const int sq_dist = (int)__fmaf_rn(ddy, ddy, __fmul_rn(ddx, ddx));
                    if (sq_dist <= sq_thres) { sq[u] = sq_dist; p[u] = pl + (yy * ov.pitch + xx); }   // a plane holds < 2^31 floats
                    xx += 32;
                    while (xx > xmax) { xx -= wx; ++yy; }
                }
            }
            float gdx[kBatch], gdy[kBatch];
#pragma unroll
            for (int u = 0; u < kBatch; ++u) {
                gdx[u] = __fsub_rn(__ldg(p[u] + 1), __ldg(p[u] - 1));
                gdy[u] = __fsub_rn(__ldg(p[u] + ov.pitch), __ldg(p[u] - ov.pitch));
            }
#pragma unroll
            for (int u = 0; u < kBatch; ++u) {
                const float grad = hypotf(gdx[u], gdy[u]);
                const float theta = atan2f(gdy[u], gdx[u]);
                weight[u] = __fmul_rn(grad, expf(__fmul_rn((float)sq[u], factor)));
                // reference SASS (ori_par): (theta + pi) * 36 * 0.15915494 -- the division by the constant 2 pi of
                // __fdividef(36 * (theta + pi), M_PI2) is folded into a multiplication by RN(1 / 2pi)
                int b = (int)roundf(__fmul_rn(__fmul_rn(__fadd_rn(theta, kPi), (float)kOriBins), 0.15915493667125701904f));
                if (b == kOriBins) b = 0;
                bidx[u] = (sq[u] < 0 || b > kOriBins) ? -1 : b;
            }
#pragma unroll
            for (int u = 0; u < kBatch; ++u) {
                __syncwarp();
                if (bidx[u] >= 0) atomicAdd(&A[bidx[u]], weight[u]);
            }
        }
        __syncwarp();
        // 3 x (box3 ; box3), circular over 36 bins (reference s_orientation.cu:58-68,166-174)
        for (int it = 0; it < 3; ++it) {
            for (int b = lane; b < kOriBins; b += 32) {
                const int pv = b == 0 ? kOriBins - 1 : b - 1, nx = b == kOriBins - 1 ? 0 : b + 1;
                B[b] = __fdiv_rn(__fadd_rn(__fadd_rn(A[pv], A[b]), A[nx]), 3.0f);
            }
            __syncwarp();
            for (int b = lane; b < kOriBins; b += 32) {
                const int pv = b == 0 ? kOriBins - 1 : b - 1, nx = b == kOriBins - 1 ? 0 : b + 1;
                A[b] = __fdiv_rn(__fadd_rn(__fadd_rn(B[pv], B[b]), B[nx]), 3.0f);
            }
            __syncwarp();
        }
        // peaks + parabola refinement; lane holds bins `lane` and `lane+32`
        float yv[2], ra[2];
#pragma unroll
        for (int s = 0; s < 2; ++s) {
            const int b = lane + 32 * s;
            yv[s] = -INFINITY; ra[s] = -1.0f;
            if (b < kOriBins) {
                const int pv = b == 0 ? kOriBins - 1 : b - 1, nx = b == kOriBins - 1 ? 0 : b + 1;
                const float hp = A[pv], hc = A[b], hn = A[nx];
                bool pred = hc > fmaxf(hp, hn);
                // the reference's SASS evaluates 3*hp - 4*hc + 1*hn as  hn + fma(hp, 3, hc * -4)  (nvcc contracts the first
                // two products; cuobjdump of ori_par: FMUL R6 = hc*-4; FFMA R6 = hp*3 + R6; FADD R0 = hn + R6)
                const float num = pred ? __fadd_rn(hn, __fmaf_rn(hp, 3.0f, __fmul_rn(hc, -4.0f))) : 0.0f;
                const float den = pred ? 2.0f * (hp - 2.0f * hc + hn) : 1.0f;
                const float newbin = __fdividef(num, den);
                pred = pred && newbin >= 0.0f && newbin <= 2.0f;
                if (pred) { ra[s] = (float)pv + newbin; yv[s] = -(num * num) / (4.0f * den) + hp; }
            }
        }
        // four arg-max rounds (descending yval; ties -> lower bin)
        float best_y[PS_MAX_ORI], best_r[PS_MAX_ORI];
#pragma unroll
        for (int r = 0; r < PS_MAX_ORI; ++r) {
            float cy; int cb;
            if (yv[0] >= yv[1] || !(yv[1] == yv[1])) { cy = yv[0]; cb = lane; } else { cy = yv[1]; cb = lane + 32; }
            float wy = cy; int wb = cb;
#pragma unroll
            for (int d = 16; d >= 1; d >>= 1) {
                const float oy = __shfl_xor_sync(0xffffffffu, wy, d);
                const int ob = __shfl_xor_sync(0xffffffffu, wb, d);
                if (oy > wy || (oy == wy && ob < wb)) { wy = oy; wb = ob; }
            }
            // owner publishes its refined angle and retires the bin
            const int owner = wb & 31, slot = wb >> 5;
            const float rr = __shfl_sync(0xffffffffu, slot ? ra[1] : ra[0], owner);
            best_y[r] = wy; best_r[r] = rr;
            if (lane == owner) { if (slot) yv[1] = -INFINITY; else yv[0] = -INFINITY; }
        }
        const float yref = __fmul_rn(0.8f, best_y[0]);
        if (lane == 0) {
            ps_extremum e;
            e.xpos = ie.xpos; e.ypos = ie.ypos; e.lpos = ie.lpos; e.sigma = ie.sigma;
            e.octave = o; e.idx_ori = 0;
            int n = 0;
#pragma unroll
            for (int r = 0; r < PS_MAX_ORI; ++r) {
                e.orientation[r] = 0.0f;
            }
#pragma unroll
            for (int r = 0; r < PS_MAX_ORI; ++r) {
                // best_y[0] == -inf (no peak at all): -inf >= -inf holds for all four (reference quirk)
                if (best_y[r] >= yref) {
                    float chosen = best_r[r];
                    if (chosen >= (float)kOriBins) chosen -= (float)kOriBins;
                    e.orientation[n++] = __fmaf_rn(__fmul_rn(kPi2, chosen), 1.0f / kOriBins, -kPi);
                }
            }
            e.num_ori = n;
            ext[item] = e;
            if (n > 0) atomicAdd(&slice_sum[item / kSlice], n);
        }
        __syncwarp();
    }
}

// Exclusive prefix sum of num_ori over all extrema, reverse map, totals.  The orientation kernel has
// already added every extremum's num_ori to the sum of its slice of kSlice extrema, so one block per slice
// only needs the sums of the slices before it: the scan runs on as many SMs as there are slices instead
// of on one (a single block spent 30 us at 4K on its one SM's memory bandwidth).
__global__ void __launch_bounds__(kSlice)
ori_scatter_kernel(int num_octaves, Consts k, ps_extremum* __restrict__ ext, int* __restrict__ feat_to_ext,
                   const int* __restrict__ slice_sum, Counters* ct)
{
    __shared__ int warp_sums[kSlice / 32];
    __shared__ int base_s;
    __shared__ int ps[kMaxOctaves + 1];
    if (threadIdx.x == 0) octave_prefix(ct, k, num_octaves, ps);
    __syncthreads();
    const int total = ps[num_octaves];
    const int b = blockIdx.x;
    const int first = b * kSlice;
    if (first >= total && b != 0) return;                       // block-uniform
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;

    // descriptors before this slice
    int part = 0;
    for (int j = threadIdx.x; j < b; j += kSlice) part += slice_sum[j];
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) part += __shfl_down_sync(0xffffffffu, part, d);
    if (lane == 0) warp_sums[warp] = part;
    __syncthreads();
    if (threadIdx.x == 0) {
        int s = 0;
        for (int w = 0; w < kSlice / 32; ++w) s += warp_sums[w];
        base_s = s;
    }
    __syncthreads();
    const int base = base_s;
    __syncthreads();                                            // warp_sums is reused below

    const int i = first + threadIdx.x;
    const int n = i < total ? ext[i].num_ori : 0;
    int v = n;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, v, d);
        if (lane >= d) v += t;
    }
    if (lane == 31) warp_sums[warp] = v;
    __syncthreads();
    int before = 0, block_total = 0;
#pragma unroll
    for (int w = 0; w < kSlice / 32; ++w) {
        const int ws = warp_sums[w];
        if (w < warp) before += ws;
        block_total += ws;
    }
    const int excl = base + before + v - n;
    if (i < total) {
        int nn = n;
        if (excl + nn > k.desc_capacity) {
            nn = max(0, k.desc_capacity - excl);
            ext[i].num_ori = nn;
            atomicOr(&ct->overflow, 2);
        }
        ext[i].idx_ori = min(excl, k.desc_capacity);
        for (int r = 0; r < nn; ++r) feat_to_ext[excl + r] = i;
    }
    const int last = total > 0 ? (total - 1) / kSlice : 0;
    if (b == last && threadIdx.x == 0) {
        ct->ext_total = total;
        ct->ori_total = min(base + block_total, k.desc_capacity);
        ct->ori_needed = base + block_total;
        int raw = 0;
        const int* counts = ct->filtered ? ct->ext_ct_f : ct->ext_ct;
        for (int o = 0; o < num_octaves; ++o) raw += min(counts[o], k.max_extrema);
        if (raw > total) atomicOr(&ct->overflow, 1);
    }
}

} // namespace

int launch_orientation(const PyramidView& pyr, const Consts& k, const InitialExtremum* iext, const InitialExtremum* iext_f, ps_extremum* ext,
                       int* feat_to_ext, int* slice_sum, Counters* ct, cudaStream_t st)
{
    // fixed grid: SMs x 8 resident CTAs of 4 warps; warps stride over the device-side count
    orientation_kernel<<<sm_count() * 8, kWarps * 32, 0, st>>>(pyr, k, iext, iext_f, ext, slice_sum, ct);
    ori_scatter_kernel<<<k.ext_capacity / kSlice + 1, kSlice, 0, st>>>(pyr.num_octaves, k, ext, feat_to_ext, slice_sum, ct);
    return 2;
}

} // namespace psb
