// Stage 2 -- DoG extrema scan + sub-pixel refinement, hand-written for sm_100a.
//
// Replaces find_extrema_in_dog / is_extremum / ModeFunctions / solve
// (reference src/popsift/s_extrema.cu:22-558, s_solve.h:25-86).  One launch covers every
// octave and all levels of an image (the reference launches once per octave with one CTA layer per
// level): see the scan kernel below.  Survivors of the 26-neighbour test are refined in registers
// and appended with one warp-ballot + one atomicAdd per warp.
//
// Parity contract: with bit-identical DoG planes, the accepted set and (x, y, lpos) of every
// extremum are bit-identical to the reference's.  The floating-point pattern below is the one in
// the reference's sm_100 SASS (cuobjdump of oracle/_ref/libpopsift_ref.so):
//   detK = fma(a1,a2, -(b1*b2));  det = fma(i02,det2, fma(i00,det0, i01*det1));  rsd = __frcp_rn(det)
//   d    = rows of (adj*rsd) . b as fma chains starting from fma(.,b.x,0)
//   contr= v + 0.5*fma(dz,Dz, fma(dy,Dy, dx*Dx));  det2 = fma(DDx,DDy, -(DXx*DXx))
#include "ps_internal.h"

#include <cstdlib>

namespace psb {

namespace {

struct DogView {
    const float* base;
    int w, h, pitch, nplanes;
    size_t plane;
    __device__ __forceinline__ float at(int x, int y, int z) const
    {   // clamp addressing in x, y and layer, like the reference's clamp textures
        x = min(max(x, 0), w - 1);
        y = min(max(y, 0), h - 1);
        z = min(max(z, 0), nplanes - 1);
        return __ldg(base + z * plane + (size_t)y * pitch + x);
    }
};

__device__ __forceinline__ bool solve3(float i00, float i01, float i02, float i11, float i12, float i22,
                                       float& bx, float& by, float& bz)
{
    const float det0 = __fmaf_rn(i11, i22, -__fmul_rn(i12, i12));
    const float det1 = __fmaf_rn(i12, i02, -__fmul_rn(i01, i22));
    const float det2 = __fmaf_rn(i01, i12, -__fmul_rn(i11, i02));
    const float det3 = __fmaf_rn(i00, i22, -__fmul_rn(i02, i02));
    const float det4 = __fmaf_rn(i01, i02, -__fmul_rn(i00, i12));
    const float det5 = __fmaf_rn(i00, i11, -__fmul_rn(i01, i01));
    float det = __fmul_rn(i01, det1);
    det = __fmaf_rn(i00, det0, det);
    det = __fmaf_rn(i02, det2, det);
    if (det == 0.0f) return false;
    const float rsd = __frcp_rn(det);
    const float a00 = __fmul_rn(det0, rsd), a10 = __fmul_rn(det1, rsd), a20 = __fmul_rn(det2, rsd);
    const float a11 = __fmul_rn(det3, rsd), a12 = __fmul_rn(det4, rsd), a22 = __fmul_rn(det5, rsd);
    const float X = bx, Y = by, Z = bz;
    bx = __fmaf_rn(a20, Z, __fmaf_rn(a10, Y, __fmaf_rn(a00, X, 0.0f)));
    by = __fmaf_rn(a12, Z, __fmaf_rn(a11, Y, __fmaf_rn(a10, X, 0.0f)));
    bz = __fmaf_rn(a22, Z, __fmaf_rn(a12, Y, __fmaf_rn(a20, X, 0.0f)));
    return true;
}

template <int MODE>
__device__ __noinline__ bool refine(const DogView& dv, const Consts& k, int x, int y, int level, int maxlevel, float val,
                       InitialExtremum& out)
{
    const int width = dv.w, height = dv.h;
    float Dx = 0.f, Dy = 0.f, Dz = 0.f, DDx = 0.f, DDy = 0.f, DXx = 0.f;
    float dx = 0.f, dy = 0.f, dz = 0.f;
    int nx = x, ny = y, nz = level;
    int iter = 0;
    do {
        ++iter;
        const float x2y1z1 = dv.at(nx + 1, ny, nz), x0y1z1 = dv.at(nx - 1, ny, nz);
        const float x1y2z1 = dv.at(nx, ny + 1, nz), x1y0z1 = dv.at(nx, ny - 1, nz);
        const float x1y1z2 = dv.at(nx, ny, nz + 1), x1y1z0 = dv.at(nx, ny, nz - 1);
        Dx = __fmul_rn(__fsub_rn(x2y1z1, x0y1z1), 0.5f);
        Dy = __fmul_rn(__fsub_rn(x1y2z1, x1y0z1), 0.5f);
        Dz = __fmul_rn(__fsub_rn(x1y1z2, x1y1z0), 0.5f);
        const float c2 = __fmul_rn(dv.at(nx, ny, nz), 2.0f);
        DDx = __fsub_rn(__fadd_rn(x2y1z1, x0y1z1), c2);
        DDy = __fsub_rn(__fadd_rn(x1y2z1, x1y0z1), c2);
        const float DDz = __fsub_rn(__fadd_rn(x1y1z2, x1y1z0), c2);
        const float x0y0z1 = dv.at(nx - 1, ny - 1, nz), x0y1z0 = dv.at(nx - 1, ny, nz - 1);
        const float x0y1z2 = dv.at(nx - 1, ny, nz + 1), x0y2z1 = dv.at(nx - 1, ny + 1, nz);
        const float x1y0z0 = dv.at(nx, ny - 1, nz - 1), x1y0z2 = dv.at(nx, ny - 1, nz + 1);
        const float x1y2z0 = dv.at(nx, ny + 1, nz - 1), x1y2z2 = dv.at(nx, ny + 1, nz + 1);
        const float x2y0z1 = dv.at(nx + 1, ny - 1, nz), x2y1z0 = dv.at(nx + 1, ny, nz - 1);
        const float x2y1z2 = dv.at(nx + 1, ny, nz + 1), x2y2z1 = dv.at(nx + 1, ny + 1, nz);
        DXx = __fmul_rn(__fsub_rn(__fsub_rn(__fadd_rn(x2y2z1, x0y0z1), x0y2z1), x2y0z1), 0.25f);
        const float DXy = __fmul_rn(__fsub_rn(__fsub_rn(__fadd_rn(x2y1z2, x0y1z0), x0y1z2), x2y1z0), 0.25f);
        const float DXz = __fmul_rn(__fsub_rn(__fsub_rn(__fadd_rn(x1y2z2, x1y0z0), x1y2z0), x1y0z2), 0.25f);

        float bx = -Dx, by = -Dy, bz = -Dz;
        if (!solve3(DDx, DXx, DXy, DDy, DXz, DDz, bx, by, bz)) { dx = dy = dz = 0.0f; break; }
        dx = bx; dy = by; dz = bz;

        int retval;
        if (MODE == PS_MODE_OPENCV) {
            if (fabsf(dx) < 0.5f && fabsf(dy) < 0.5f && fabsf(dz) < 0.5f) retval = 1;
            else {
                nx += (int)roundf(dx); ny += (int)roundf(dy); nz += (int)roundf(dz);
                retval = (nx < 5 || nx >= width - 5 || ny < 5 || ny >= height - 5 || nz < 1 || nz > maxlevel - 2) ? -1 : 0;
            }
        } else if (iter == 5) {
            retval = 0;
        } else {
            const int tx = ((dx >= 0.6f && nx < width - 2) ? 1 : 0) + ((dx <= -0.6f && nx > 1) ? -1 : 0);
            const int ty = ((dy >= 0.6f && ny < height - 2) ? 1 : 0) + ((dy <= -0.6f && ny > 1) ? -1 : 0);
            int tz = 0;
            if (MODE == PS_MODE_POPSIFT)
                tz = ((dz >= 0.6f && nz < maxlevel - 1) ? 1 : 0) + ((dz <= -0.6f && nz > 1) ? -1 : 0);
            if (tx == 0 && ty == 0 && tz == 0) retval = 1;
            else { nx += tx; ny += ty; nz += tz; retval = 0; }
        }
        if (retval == -1) return false;
        if (retval == 1) break;
    } while (iter < 5);

    if (MODE == PS_MODE_OPENCV) { if (iter >= 5) return false; }
    else if (dx >= 1.5f || dy >= 1.5f || dz >= 1.5f) return false;

    const float xn = __fadd_rn((float)nx, dx), yn = __fadd_rn((float)ny, dy), sn = __fadd_rn((float)nz, dz);
    if (MODE != PS_MODE_OPENCV)
        if (xn < 0.0f || xn > (float)width - 1.0f || yn < 0.0f || yn > (float)height - 1.0f ||
            sn < 0.0f || sn > (float)maxlevel) return false;

    const float t = __fmaf_rn(dz, Dz, __fmaf_rn(dy, Dy, __fmul_rn(dx, Dx)));
    const float contr = __fadd_rn(val, __fmul_rn(t, 0.5f));
    const float tr = __fadd_rn(DDx, DDy);
    const float det = __fmaf_rn(DDx, DDy, -__fmul_rn(DXx, DXx));
    const float edgeval = __fdiv_rn(__fmul_rn(tr, tr), det);
    if (!(det > 0.0f)) return false;
    if (fabsf(contr) < __fmul_rn(k.threshold, 2.0f)) return false;
    const float el1 = __fadd_rn(k.edge_limit, 1.0f);
    if (edgeval >= __fdiv_rn(__fmul_rn(el1, el1), k.edge_limit)) return false;

    out.xpos = xn;
    out.ypos = yn;
    out.lpos = (int)roundf(sn);
    out.sigma = __fmul_rn(k.sigma0, powf(k.sigma_k, sn));
    return true;
}

// ---- scan kernel -------------------------------------------------------------------------------
//
// A warp owns 30 output columns (lanes 1..30; lanes 0 and 31 only carry the x-halo) and walks down
// SCAN_ROWS rows.  For every row it loads one value per DoG plane (coalesced 128-byte reads), forms the
// horizontal 3-max / 3-min of each plane with two shuffles, and keeps the last three rows in registers.
// The 26-neighbour test of a voxel is then a handful of max/min over those registers:
//     strict maximum  <=>  v > max( 3x3 of plane l-1, 3x3 of plane l+1, 8 neighbours in plane l )
// All NLEV levels of the octave are evaluated in the same pass, so each DoG value is loaded from HBM
// once (the reference re-reads 27 texels per candidate, s_extrema.cu:56-120).  The verdict is identical:
// a voxel survives iff it is strictly greater, or strictly smaller, than all 26 neighbours.
constexpr int SCAN_COLS = 30;      // output columns per warp
constexpr int SCAN_WARPS = 8;      // warps side by side in x
constexpr int SCAN_ROWS = 32;      // rows walked by a CTA

struct ScanParams {
    int tile_begin[kMaxOctaves + 1];   // first CTA index of each octave
    int tiles_x[kMaxOctaves];
    int first_level;                   // first level evaluated (1-based DoG level)
};

template <int MODE, int NLEV>
__global__ void __launch_bounds__(SCAN_WARPS * 32, 2)
find_extrema_kernel(PyramidView pyr, Consts k, ScanParams sp, InitialExtremum* __restrict__ iext, Counters* ct)
{
    const int tile = blockIdx.x;
    int o = 0;
    while (o + 1 < pyr.num_octaves && tile >= sp.tile_begin[o + 1]) ++o;
    const OctaveView& ov = pyr.oct[o];
    const int local = tile - sp.tile_begin[o];
    const int ty = local / sp.tiles_x[o];
    const int tx = local - ty * sp.tiles_x[o];
    const int maxlevel = pyr.levels + 2;      // reference passes _levels-1 (s_extrema.cu:597)
    const int lvl0 = sp.first_level;          // planes lvl0-1 .. lvl0+NLEV are read

    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int W = ov.w, H = ov.h;
    const int x = tx * (SCAN_WARPS * SCAN_COLS) + warp * SCAN_COLS + lane;   // lane 0 is the left halo column
    const int xc = min(x, W - 1);
    const int y0 = ty * SCAN_ROWS + 1;                                        // first output row
    if (y0 > H - 2) return;
    bool xout = (lane >= 1 && lane <= SCAN_COLS) && (x >= 1) && (x <= W - 2);
    if (MODE == PS_MODE_OPENCV) xout = xout && !(x < 5 || x >= W - 5);

    DogView dv;
    dv.base = ov.dog; dv.w = W; dv.h = H; dv.pitch = ov.pitch; dv.plane = ov.plane;
    dv.nplanes = pyr.levels + 2;

    float thr;
    if (MODE == PS_MODE_OPENCV) thr = floorf(k.threshold);
    else if (MODE == PS_MODE_VLFEAT) thr = __fmul_rn(__fmul_rn(0.8f, 2.0f), k.threshold);
    else thr = __fmul_rn(1.6f, k.threshold);

    constexpr int NP = NLEV + 2;
    const float* colp = ov.dog + (size_t)(lvl0 - 1) * ov.plane + xc;
    // ring of three rows: value, horizontal 3-max, horizontal 3-min
    float v[3][NP], hx[3][NP], hn[3][NP];

    // rows y+1, y+2, y+3: three rows of loads stay in flight per warp (~46 KB per SM, enough to cover
    // the HBM latency at full bandwidth) while row y is evaluated
    float pend[3][NP];
    const unsigned plane_u = (unsigned)ov.plane;     // a whole octave (<= 15 planes) stays below 2^32 floats
    auto issue_row = [&](int slot, int y) {
        const int yc = min(max(y, 0), H - 1);
        const float* rowp = colp + (size_t)yc * ov.pitch;
#pragma unroll
        for (int p = 0; p < NP; ++p) pend[slot][p] = __ldg(rowp + p * plane_u);
    };
    auto finish_row = [&](int slot, int ps) {
#pragma unroll
        for (int p = 0; p < NP; ++p) {
            const float c = pend[ps][p];
            const float l = __shfl_up_sync(0xffffffffu, c, 1);
            const float r = __shfl_down_sync(0xffffffffu, c, 1);
            v[slot][p] = c;
            hx[slot][p] = fmaxf(fmaxf(l, r), c);
            hn[slot][p] = fminf(fminf(l, r), c);
        }
    };
    issue_row(0, y0 - 1); issue_row(1, y0);
    finish_row(0, 0); finish_row(1, 1);
    issue_row(0, y0 + 1); issue_row(1, y0 + 2); issue_row(2, y0 + 3);

#pragma unroll 1
    for (int rr = 0; rr < SCAN_ROWS; rr += 3) {
        // three rows per trip so that the ring slots are compile-time constants
#pragma unroll
        for (int u = 0; u < 3; ++u) {
            const int y = y0 + rr + u;
            if (rr + u >= SCAN_ROWS || y > H - 2) break;           // warp-uniform
            const int sa = u % 3, sb = (u + 1) % 3, sc = (u + 2) % 3;    // above, centre, below
            finish_row(sc, u);              // row y+1 has landed (pending slot u)
            issue_row(u, y + 4);            // refill the slot: rows y+2 .. y+4 are now in flight
            bool yok = true;
            if (MODE == PS_MODE_OPENCV) yok = !(y < 5 || y >= H - 5);
            unsigned candbits = 0u;
#pragma unroll
            for (int q = 0; q < NLEV; ++q) {
                const int p = q + 1;                              // centre plane index in the register ring
                const float c = v[sb][p];
                // left / right neighbours in the own plane, own row
                const float l = __shfl_up_sync(0xffffffffu, c, 1);
                const float r = __shfl_down_sync(0xffffffffu, c, 1);
                float mx = fmaxf(fmaxf(hx[sa][p], hx[sc][p]), fmaxf(l, r));
                float mn = fminf(fminf(hn[sa][p], hn[sc][p]), fminf(l, r));
                mx = fmaxf(mx, fmaxf(fmaxf(hx[sa][p - 1], hx[sb][p - 1]), hx[sc][p - 1]));
                mn = fminf(mn, fminf(fminf(hn[sa][p - 1], hn[sb][p - 1]), hn[sc][p - 1]));
                mx = fmaxf(mx, fmaxf(fmaxf(hx[sa][p + 1], hx[sb][p + 1]), hx[sc][p + 1]));
                mn = fminf(mn, fminf(fminf(hn[sa][p + 1], hn[sb][p + 1]), hn[sc][p + 1]));
                if ((fabsf(c) >= thr) && ((c > mx) || (c < mn))) candbits |= 1u << q;
            }
            if (!(xout && yok)) candbits = 0u;
            if (__any_sync(0xffffffffu, candbits != 0u)) {
                // rare path (a few voxels per thousand): refine and append, level by level
                for (int q = 0; q < NLEV; ++q) {
                    const bool cand = (candbits >> q) & 1u;
                    if (!__any_sync(0xffffffffu, cand)) continue;
                    bool found = false;
                    InitialExtremum e;
                    e.xpos = e.ypos = e.sigma = 0.f; e.lpos = 0;
                    float cval = v[sb][1];
                    if (q == 1 && NLEV > 1) cval = v[sb][2];
                    if (q == 2 && NLEV > 2) cval = v[sb][3];
                    if (cand) found = refine<MODE>(dv, k, x, y, lvl0 + q, maxlevel, cval, e);
                    const unsigned mask = __ballot_sync(0xffffffffu, found);
                    if (mask != 0) {
                        int base = 0;
                        if (lane == 0) base = atomicAdd(&ct->ext_ct[o], __popc(mask));
                        base = __shfl_sync(0xffffffffu, base, 0);
                        const int idx = base + __popc(mask & ((1u << lane) - 1u));
                        if (found && idx < k.max_extrema) iext[(size_t)o * k.max_extrema + idx] = e;
                    }
                }
            }
        }
    }
}

// ---- candidate-driven scan ---------------------------------------------------------------------
//
// The pyramid kernels report every DoG pixel pair in which a sample has |value| >= threshold into the
// list region of the block that produced it (CandSink) while they write the plane.  On real and
// synthetic images that is a few samples per thousand, so testing only those against their 26
// neighbours replaces the dense scan's read of every DoG plane.  Accepted set and refinement are those of the dense
// kernel: same comparisons, same refine<MODE>.
constexpr int kScanThreads = 256;

// one octave's DoG planes, by value (a reference to the kernel's PyramidView parameter would make every
// thread copy the whole structure to local memory)
struct DogOct { const float* dog; int w, h, pitch, nplanes; size_t plane; };

// Region-driven form (default).  A list region = the candidates one block of one level kernel reported; block b of this
// kernel takes regions b, b + gridDim.x, ... (no prefix sum, no search: a region's octave, level and list follow from
// its index), its 8 warps take the region's samples 32 at a time.  The three tests of a sample have very different
// survival rates, so each is run on full warps of survivors:
//   stage 1  (every sample)   threshold re-test + the 8 in-plane neighbours           ~10 % survive
//   stage 2  (per-warp queue) the 18 neighbours of the planes below and above         ~0.6 % survive
//   stage 3  (per-block queue) refine<MODE> + append
// Survivors are compacted with a warp ballot into shared-memory queues; a queue is served when it holds a full warp
// (stage 2) or when the block has run out of regions (stage 3 and the stage-2 remainders).
constexpr int kQ2 = 64;            // stage-2 queue entries per warp (< 32 pending + <= 32 new)
constexpr int kQ3 = 1024;          // stage-3 queue entries per block; overflowing survivors are refined at once

struct Q2Entry { unsigned xy; unsigned ol; };      // x | y << 16 ;  octave | level << 8 | is_max << 16

// Stage 1 on a reported PAIR (x even, x + 1): the two samples share their rows and most of their neighbours, so one
// thread tests both from three aligned float4 loads + three scalars (columns x-1 .. x+2 of rows y-1, y, y+1) instead of
// nine scalar loads per sample.  The candidates of a warp are scattered (a few per thousand pixels), every load
// instruction touches 32 different cache lines: the number of load instructions, not their width, sets the time
// (9 per sample: 74 us of L1 wavefronts at 4K; 3 per sample now).  Returns bit 0 / bit 1 = sample x / x + 1 survives;
// bits 2 / 3 = it is a maximum.
template <int MODE>
__device__ __forceinline__ unsigned stage1_pair(const DogOct& ov, int level, float thr, int x, int y)
{
    const int W = ov.w, H = ov.h;
    bool iny = y >= 1 && y <= H - 2;
    if (MODE == PS_MODE_OPENCV) iny = iny && !(y < 5 || y >= H - 5);
    if (!iny) return 0u;
    const float* row = ov.dog + (size_t)level * ov.plane + (size_t)y * ov.pitch;
    const int xa = x & ~3;                                 // aligned group holding x and x + 1 (x is even)
    const bool lowhalf = (x & 2) == 0;                     // x, x+1 are the group's first two floats: x-1 is outside
    const int xs = lowhalf ? max(x - 1, 0) : x + 2;        // the one column outside the group
    float a[3], b[3], c[3], d[3];                          // columns x-1, x, x+1, x+2 of rows y-1, y, y+1
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        const float* p = row + (long long)(r - 1) * ov.pitch;
        const float4 g = __ldg(reinterpret_cast<const float4*>(p + xa));
        const float e = __ldg(p + xs);
        if (lowhalf) { a[r] = e; b[r] = g.x; c[r] = g.y; d[r] = g.z; }
        else         { a[r] = g.y; b[r] = g.z; c[r] = g.w; d[r] = e; }
    }
    unsigned out = 0u;
    {   // sample x: centre b[1]
        bool inx = x >= 1 && x <= W - 2;
        if (MODE == PS_MODE_OPENCV) inx = inx && !(x < 5 || x >= W - 5);
        const float v = b[1];
        const float mx = fmaxf(fmaxf(fmaxf(a[0], b[0]), fmaxf(c[0], a[1])), fmaxf(fmaxf(c[1], a[2]), fmaxf(b[2], c[2])));
        const float mn = fminf(fminf(fminf(a[0], b[0]), fminf(c[0], a[1])), fminf(fminf(c[1], a[2]), fminf(b[2], c[2])));
        if (inx && fabsf(v) >= thr) { if (v > mx) out |= 1u | 4u; else if (v < mn) out |= 1u; }
    }
    {   // sample x + 1: centre c[1]
        const int x1 = x + 1;
        bool inx = x1 >= 1 && x1 <= W - 2;
        if (MODE == PS_MODE_OPENCV) inx = inx && !(x1 < 5 || x1 >= W - 5);
        const float v = c[1];
        const float mx = fmaxf(fmaxf(fmaxf(b[0], c[0]), fmaxf(d[0], b[1])), fmaxf(fmaxf(d[1], b[2]), fmaxf(c[2], d[2])));
        const float mn = fminf(fminf(fminf(b[0], c[0]), fminf(d[0], b[1])), fminf(fminf(d[1], b[2]), fminf(c[2], d[2])));
        if (inx && fabsf(v) >= thr) { if (v > mx) out |= 2u | 8u; else if (v < mn) out |= 2u; }
    }
    return out;
}

__device__ __forceinline__ bool stage2(const DogOct& ov, int level, int x, int y, bool is_max, float& cval)
{
    const float* pc = ov.dog + (size_t)level * ov.plane + (size_t)y * ov.pitch + x;
    const float c = __ldg(pc);
    cval = c;
    float mx = -INFINITY, mn = INFINITY;
#pragma unroll
    for (int dz = -1; dz <= 1; dz += 2) {
        const float* p = dz < 0 ? pc - ov.plane : pc + ov.plane;
        const float* ra = p - ov.pitch;
        const float* rb = p + ov.pitch;
        const float n0 = __ldg(p - 1), n1 = __ldg(p), n2 = __ldg(p + 1);
        const float n3 = __ldg(ra - 1), n4 = __ldg(ra), n5 = __ldg(ra + 1);
        const float n6 = __ldg(rb - 1), n7 = __ldg(rb), n8 = __ldg(rb + 1);
        mx = fmaxf(mx, fmaxf(fmaxf(fmaxf(n0, n1), fmaxf(n2, n3)), fmaxf(fmaxf(n4, n5), fmaxf(fmaxf(n6, n7), n8))));
        mn = fminf(mn, fminf(fminf(fminf(n0, n1), fminf(n2, n3)), fminf(fminf(n4, n5), fminf(fminf(n6, n7), n8))));
    }
    return is_max ? c > mx : c < mn;
}

template <int MODE>
__device__ __forceinline__ void stage3(const PyramidView& pyr, const Consts& k, const Q2Entry q, float cval,
                                       InitialExtremum* __restrict__ iext, Counters* ct)
{
    const int o = (int)(q.ol & 0xffu), level = (int)((q.ol >> 8) & 0xffu);
    const OctaveView& ov = pyr.oct[o];
    DogView dv;
    dv.base = ov.dog; dv.w = ov.w; dv.h = ov.h; dv.pitch = ov.pitch; dv.plane = ov.plane;
    dv.nplanes = pyr.levels + 2;
    InitialExtremum e;
    e.xpos = e.ypos = e.sigma = 0.f; e.lpos = 0;
    if (refine<MODE>(dv, k, (int)(q.xy & 0xffffu), (int)(q.xy >> 16), level, dv.nplanes, cval, e)) {
        const int idx = atomicAdd(&ct->ext_ct[o], 1);
        if (idx < k.max_extrema) iext[(size_t)o * k.max_extrema + idx] = e;
    }
}

// 3 resident CTAs per SM: 80 registers, 77.7 us per 4K frame; 4 CTAs force 64 registers, which spill in the
// candidate loop (84.4 us)
template <int MODE>
__global__ void __launch_bounds__(kScanThreads, 3)
cand_extrema_kernel(PyramidView pyr, Consts k, InitialExtremum* __restrict__ iext, Counters* ct)
{
    __shared__ Q2Entry q2[kScanThreads / 32][kQ2];
    __shared__ Q2Entry q3[kQ3];
    __shared__ float q3c[kQ3];
    __shared__ int q3n;
    const int L = pyr.levels;
    const float thr = extrema_threshold(k);
    const int nreg = pyr.cand_regions;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned lt = (1u << lane) - 1u;
    if (threadIdx.x == 0) q3n = 0;
    __syncthreads();
    int q2n = 0;                                               // warp-uniform

    auto octave_view = [&](int o) {
        DogOct d;
        const OctaveView& ov = pyr.oct[o];
        d.dog = ov.dog; d.w = ov.w; d.h = ov.h; d.pitch = ov.pitch; d.plane = ov.plane; d.nplanes = L + 2;
        return d;
    };
    // stage 2 on one warp-full (or the remainder) of this warp's queue, survivors -> the block's stage-3 queue
    auto serve_q2 = [&](int first, int n) {
        Q2Entry q; q.xy = 0u; q.ol = 0u;
        bool ok = false;
        float cval = 0.0f;
        if (lane < n) {
            q = q2[warp][first + lane];
            const DogOct ov = octave_view((int)(q.ol & 0xffu));
            ok = stage2(ov, (int)((q.ol >> 8) & 0xffu), (int)(q.xy & 0xffffu), (int)(q.xy >> 16), (q.ol >> 16) & 1u, cval);
        }
        const unsigned m = __ballot_sync(0xffffffffu, ok);
        if (m == 0u) return;
        int base = 0;
        if (lane == 0) base = atomicAdd(&q3n, __popc(m));
        base = __shfl_sync(0xffffffffu, base, 0);
        if (ok) {
            const int pos = base + __popc(m & lt);
            if (pos < kQ3) { q3[pos] = q; q3c[pos] = cval; }
            else stage3<MODE>(pyr, k, q, cval, iext, ct);      // queue full (never on real images): refine at once
        }
    };

    // Region g = (octave, level, pyramid CTA).  A plain block-strided walk would hand block b the SAME image area in every
    // level (the level kernels have as many CTAs as this grid has blocks), so a block that draws a textured area would
    // draw it fifteen times; rotating the assignment by a stride coprime to the grid from one pass to the next spreads
    // the areas over the blocks (cycles active: average / maximum 0.78 -> see profiles).
    // The count and the first candidates of the NEXT region are requested before the current region is processed (the list
    // address does not depend on the count, entries beyond it are simply ignored), so a region costs one memory round trip
    // -- its plane samples -- instead of three in a row.
    const int G = (int)gridDim.x;
    struct Region { const unsigned* list; int o, level, cap; bool valid; };
    auto prepare = [&](int pass, Region& r, int& cnt, unsigned& first) -> bool {
        const int g0 = pass * G;
        if (g0 >= nreg) return false;
        const int g = g0 + (int)(((unsigned)blockIdx.x + (unsigned)pass * 197u) % (unsigned)G);
        r.valid = g < nreg;
        cnt = 0; first = 0u;
        if (r.valid) {
            int o = 0, local = g;                                // region -> octave, (level - 1) * cand_blocks + block
            while (local >= pyr.oct[o].cand_blocks * L) { local -= pyr.oct[o].cand_blocks * L; ++o; }
            const OctaveView& ovv = pyr.oct[o];
            r.o = o;
            r.level = local / ovv.cand_blocks + 1;               // DoG plane of the region's samples
            r.cap = ovv.cand_region;
            r.list = ovv.cand + (size_t)local * ovv.cand_region;
            cnt = __ldg(pyr.cand_cnt_all + g);                   // block-uniform
            if ((int)threadIdx.x < r.cap) first = __ldg(r.list + threadIdx.x);
        }
        return true;
    };
    Region nx; int cnt_nx = 0; unsigned first_nx = 0u;
    int pass = 0;
    bool more = prepare(pass, nx, cnt_nx, first_nx);
    while (more) {
        const Region cur = nx;
        const int cnt = cnt_nx;
        const unsigned first = first_nx;
        more = prepare(++pass, nx, cnt_nx, first_nx);
        if (!cur.valid || cnt <= 0) continue;
        const int o = cur.o, level = cur.level;
        const int n = min(cnt, cur.cap);                         // reported pairs
        const unsigned* __restrict__ list = cur.list;
        const DogOct ov = octave_view(o);
        for (int t0 = warp * 32; t0 < n; t0 += kScanThreads) {
            const int t = t0 + lane;
            unsigned packed = 0u, res = 0u;
            if (t < n) {
                packed = t0 == warp * 32 ? first : __ldg(list + t);
                res = stage1_pair<MODE>(ov, level, thr, (int)(packed & 0xffffu), (int)(packed >> 16));
            }
#pragma unroll
            for (int sidx = 0; sidx < 2; ++sidx) {                // the pair's two samples, one ballot each
                const bool ok = (res >> sidx) & 1u;
                const unsigned m = __ballot_sync(0xffffffffu, ok);
                if (m == 0u) continue;
                if (ok) {
                    Q2Entry q;
                    q.xy = packed + (unsigned)sidx;                // x + 1 for the second sample (x is even: no carry)
                    q.ol = (unsigned)o | ((unsigned)level << 8) | (((res >> (2 + sidx)) & 1u) << 16);
                    q2[warp][q2n + __popc(m & lt)] = q;
                }
                q2n += __popc(m);
                __syncwarp();
                if (q2n >= 32) { q2n -= 32; serve_q2(q2n, 32); __syncwarp(); }
            }
        }
    }
    if (q2n > 0) serve_q2(0, q2n);
    __syncthreads();
    const int n3 = min(q3n, kQ3);
    for (int i = threadIdx.x; i < n3; i += kScanThreads) stage3<MODE>(pyr, k, q3[i], q3c[i], iext, ct);
}

// POPSIFT_B200_DENSE_SCAN=1 forces the dense scan kernels (A/B timing and cross-check)
static bool dense_choice()
{
    static const bool v = [] { const char* e = getenv("POPSIFT_B200_DENSE_SCAN"); return e && e[0] == '1'; }();
    return v;
}

template <int MODE>
int launch_scan(const PyramidView& pyr, const Consts& k, InitialExtremum* iext, Counters* ct, cudaStream_t st)
{
    if (pyr.cands_filled && !dense_choice()) {
        cand_extrema_kernel<MODE><<<sm_count() * 3, kScanThreads, 0, st>>>(pyr, k, iext, ct);
        return 1;
    }
    int launches = 0;
    // levels are evaluated in groups of up to 3 (all of them at once for the default levels = 3)
    for (int first = 1; first <= pyr.levels; first += 3) {
        const int nlev = pyr.levels - first + 1 < 3 ? pyr.levels - first + 1 : 3;
        ScanParams sp;
        sp.first_level = first;
        int total = 0;
        for (int o = 0; o < kMaxOctaves; ++o) {
            sp.tile_begin[o] = total;
            sp.tiles_x[o] = 1;
            if (o < pyr.num_octaves && pyr.oct[o].w >= 3 && pyr.oct[o].h >= 3) {
                const int tx = (pyr.oct[o].w - 2 + SCAN_WARPS * SCAN_COLS - 1) / (SCAN_WARPS * SCAN_COLS);
                const int ty = (pyr.oct[o].h - 2 + SCAN_ROWS - 1) / SCAN_ROWS;
                sp.tiles_x[o] = tx;
                total += tx * ty;
            }
        }
        sp.tile_begin[kMaxOctaves] = total;
        if (total == 0) continue;
        if (nlev == 3)      find_extrema_kernel<MODE, 3><<<total, SCAN_WARPS * 32, 0, st>>>(pyr, k, sp, iext, ct);
        else if (nlev == 2) find_extrema_kernel<MODE, 2><<<total, SCAN_WARPS * 32, 0, st>>>(pyr, k, sp, iext, ct);
        else                find_extrema_kernel<MODE, 1><<<total, SCAN_WARPS * 32, 0, st>>>(pyr, k, sp, iext, ct);
        ++launches;
    }
    return launches;
}

} // namespace

int launch_find_extrema(const PyramidView& pyr, const Consts& k, InitialExtremum* iext, Counters* ct, cudaStream_t st)
{
    switch (k.sift_mode) {
        case PS_MODE_OPENCV: return launch_scan<PS_MODE_OPENCV>(pyr, k, iext, ct, st);
        case PS_MODE_VLFEAT: return launch_scan<PS_MODE_VLFEAT>(pyr, k, iext, ct, st);
        default:             return launch_scan<PS_MODE_POPSIFT>(pyr, k, iext, ct, st);
    }
}

} // namespace psb
