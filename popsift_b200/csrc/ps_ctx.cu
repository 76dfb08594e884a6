// C-ABI layer: contexts, slots (one CUDA stream + one set of HBM buffers per in-flight image),
// kernel choreography.  See include/popsift_b200.h for the contract and the reference interfaces
// each entry point replaces.
//
// HBM layout of a slot (all float32, linear, row pitch = multiple of 32 floats):
//   for each octave o: [ (L+3) Gaussian planes | (L+2) DoG planes ], octaves back to back;
//   InitialExtremum[octaves][max_extrema], ps_extremum[ext_cap], ps_feature[ext_cap],
//   ps_descriptor[desc_cap], int feat_to_ext[desc_cap], Counters.
// There is no intermediate (row-filtered) plane in HBM: the row pass lives in shared memory.
#include "ps_internal.h"

#include <algorithm>
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

using namespace psb;

namespace {

thread_local std::string g_create_error;
constexpr bool kGridFilterBuilt = true;

struct Slot {
    cudaStream_t stream = nullptr;
    // levels L+1, L+2 of octave o run on side[o % kSides], beside the next octaves
    static constexpr int kSides = 1;     // (two side streams measured 3 % slower at 4K: the big launches fight for the SMs)
    cudaStream_t side[kSides] = {};
    cudaEvent_t  ev_fork[kMaxOctaves] = {};
    cudaEvent_t  ev_join[kSides] = {};
    // input
    uint8_t* d_img = nullptr;      // max_w*max_h*4 bytes (u8 or f32 images)
    uint8_t* h_img = nullptr;      // pinned staging, same size
    // pyramid
    float*  d_planes = nullptr;
    float*  d_interm = nullptr;    // one octave-0 plane of row-filtered values (--gauss-mode relative only)
    size_t  planes_floats = 0;
    int*    cand_cnt = nullptr;    // candidate counts of all octaves, levels and blocks (inside d_planes)
    size_t  cand_cnt_bytes = 0;
    PyramidView view{};
    // detections
    InitialExtremum* d_iext = nullptr;
    InitialExtremum* d_iext_f = nullptr;      // grid filter: survivors, keep flags, plan (allocated only when the filter is configured)
    unsigned char*   d_keep = nullptr;
    FilterPlan*      d_plan = nullptr;
    ps_extremum*     d_ext = nullptr;
    ps_feature*      d_feat = nullptr;
    ps_descriptor*   d_desc = nullptr;
    int*             d_f2e = nullptr;
    Counters*        d_ct = nullptr;
    int*             d_ori_slice = nullptr;   // num_ori sums per PS_ORI_SLICE extrema (k_orient.cu)
    Counters*        h_ct = nullptr;   // pinned
    // pinned result staging (grown on demand)
    ps_feature*    h_feat = nullptr;  size_t h_feat_cap = 0;
    ps_descriptor* h_desc = nullptr;  size_t h_desc_cap = 0;
    cudaEvent_t ev[PS_NUM_STAGES + 1] = {};
    cudaEvent_t done = nullptr;
    cudaEvent_t in_done = nullptr;   // recorded after the copy of the slot's input image (host or device source)
    bool in_pending = false;         // in_done has been recorded at least once
    int ext_cap = 0, desc_cap = 0;   // capacity of d_ext / d_feat and of d_desc / d_f2e; grown on demand (regrow_slot)
    // the slot's per-frame work as a CUDA graph (submit_common)
    cudaGraphExec_t graph_exec = nullptr;
    bool graph_ok = false, graph_float = false, warm_float = false;
    int graph_w = 0, graph_h = 0, warm_w = 0, warm_h = 0, graph_launches = 0;
    bool submitted = false;
    bool is_float = false;
    int w = 0, h = 0;
    int32_t W[kMaxOctaves] = {}, H[kMaxOctaves] = {};
    int num_octaves = 0;
};

} // namespace

struct ps_ctx {
    int device = 0;
    ps_config cfg{};
    ps_gauss_tables tab{};
    GaussRow rows[PS_GAUSS_LEVELS];
    GaussRow dd0;                         // first horizontal pass over the input image, octave 0
    GaussRow dd[kMaxOctaves];             // ... of every octave (Config::ScaleDirect)
    GaussRow abs0[PS_GAUSS_LEVELS];       // octave 0 from the input image, every level (--gauss-mode vlfeat-direct)
    GaussRow absn[PS_GAUSS_LEVELS];       // levels >= 1 of an octave from its level 0 (--gauss-mode fixed9 / fixed15, octaves >= 1)
    GaussRow irows[PS_GAUSS_LEVELS];      // incremental rows transformed for interpolated fetches (--gauss-mode relative); span = i_span
    Consts k{};
    int max_w = 0, max_h = 0;
    int max_octaves = 0;
    int levels = 3;
    bool timing = false;
    bool graph_broken = false;       // a stream capture failed once: direct launches from then on
    std::vector<Slot> slots;
    std::atomic<int64_t> launches{0};
    mutable std::mutex err_mu;
    std::string err;

    int fail(int code, const char* fmt, ...)
    {
        char buf[512];
        va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof(buf), fmt, ap); va_end(ap);
        std::lock_guard<std::mutex> g(err_mu);
        err = buf;
        return code;
    }
};

#define PS_CUDA(ctx, call)                                                                   \
    do {                                                                                     \
        cudaError_t e_ = (call);                                                             \
        if (e_ != cudaSuccess)                                                               \
            return (ctx)->fail(PS_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

namespace {

size_t round_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// floats needed for the planes of a w x h image
size_t plane_budget(const ps_config& cfg, int w, int h, int levels)
{
    int32_t W[kMaxOctaves], H[kMaxOctaves];
    const int n = ps_geometry(&cfg, w, h, W, H);
    size_t total = 0;
    for (int o = 0; o < n; ++o) {
        total += round_up(W[o], 32) * (size_t)H[o] * (size_t)(2 * levels + 5);
        // candidate lists of the `levels` scanned DoG planes + one count per block (<= 4096 blocks... generous)
        total += ((size_t)cand_entry_bound_for(W[o], H[o]) + 16384) * (size_t)levels + 16;
    }
    return total;
}

int build_view(ps_ctx* ctx, Slot& s, int w, int h)
{
    s.num_octaves = ps_geometry(&ctx->cfg, w, h, s.W, s.H);
    if (s.num_octaves < 1) return ctx->fail(PS_ERR_ARG, "bad geometry for %dx%d", w, h);
    if (s.num_octaves > ctx->max_octaves)
        return ctx->fail(PS_ERR_TOO_LARGE, "%dx%d needs %d octaves, context has %d", w, h, s.num_octaves, ctx->max_octaves);
    const int L = ctx->levels;
    size_t off = 0;
    std::memset(&s.view, 0, sizeof(s.view));
    for (int o = 0; o < s.num_octaves; ++o) {
        OctaveView& v = s.view.oct[o];
        v.w = s.W[o]; v.h = s.H[o];
        v.pitch = (int)round_up(v.w, 32);
        v.plane = (size_t)v.pitch * v.h;
        v.gauss = s.d_planes + off;  off += v.plane * (L + 3);
        v.dog = s.d_planes + off;    off += v.plane * (L + 2);
        v.cand_blocks = cand_blocks_for(v.w, v.h);
        v.cand_region = cand_region_for(v.w, v.h);
        v.cand = reinterpret_cast<uint32_t*>(s.d_planes + off);  off += (size_t)v.cand_blocks * v.cand_region * L;
    }
    // all block counts in one piece: zeroed with one memset per image
    s.cand_cnt = reinterpret_cast<int*>(s.d_planes + off);
    for (int o = 0; o < s.num_octaves; ++o) {
        OctaveView& v = s.view.oct[o];
        v.cand_cnt = reinterpret_cast<int*>(s.d_planes + off);  off += (size_t)v.cand_blocks * L;
    }
    s.cand_cnt_bytes = (size_t)(reinterpret_cast<int*>(s.d_planes + off) - s.cand_cnt) * sizeof(int);
    s.view.cand_cnt_all = s.cand_cnt;
    s.view.cand_regions = (int)(s.cand_cnt_bytes / sizeof(int));
    s.view.cand_prefix = reinterpret_cast<int*>(s.d_planes + off);  off += (size_t)s.view.cand_regions + 1;
    if (off > s.planes_floats) return ctx->fail(PS_ERR_TOO_LARGE, "%dx%d exceeds the slot's plane memory", w, h);
    s.view.num_octaves = s.num_octaves;
    s.view.levels = L;
    s.w = w; s.h = h;
    return PS_OK;
}

// device pitch of the 8-bit input image: rows start 4-byte aligned (the level-0 kernel stages them with
// 4-byte cp.async)
static inline size_t u8_pitch(int w) { return ((size_t)w + 3) & ~(size_t)3; }

// The sink of Gaussian level l of octave o: DoG plane l-1 is scanned for extrema when 1 <= l-1 <= L.
static bool level_sink(ps_ctx* ctx, Slot& s, int o, int l, CandSink& cs)
{
    const int L = ctx->levels;
    if (!s.view.cands_filled || l < 2 || l > L + 1) return false;
    const OctaveView& v = s.view.oct[o];
    cs.list = v.cand + (size_t)(l - 2) * v.cand_blocks * v.cand_region;
    cs.counts = v.cand_cnt + (size_t)(l - 2) * v.cand_blocks;
    cs.thr = extrema_threshold(ctx->k);
    cs.region = v.cand_region;
    return true;
}

// Dependency graph of the pyramid: within an octave level l needs level l-1; octave o+1 needs only level L
// of octave o.  Levels L+1 and L+2 of octave o are therefore issued on the slot's side stream and overlap
// the (much smaller) next octaves, which would otherwise run alone at a fraction of the GPU.
int run_pyramid(ps_ctx* ctx, Slot& s)
{
    const int L = ctx->levels;
    const bool fork = s.num_octaves > 1;
    const bool direct = ctx->cfg.scaling_mode == PS_SCALE_DIRECT;
    int n = 0, r;
    // the pyramid kernels report the threshold-passing DoG samples when every scanned level runs on the
    // marching kernels (16-bit coordinates in the lists)
    // --gauss-mode fixed9 / fixed15 (Fixed9 / Fixed15, s_pyramid_build.cu:487-498 + s_pyramid_fixed.cu): every level straight from
    // the input image (octave 0) or from level 0 of its octave, vertical pass first, fixed half width 4 / 7
    if (ctx->cfg.gauss_mode == PS_GAUSS_FIXED9 || ctx->cfg.gauss_mode == PS_GAUSS_FIXED15) {
        const int S = ctx->cfg.gauss_mode == PS_GAUSS_FIXED9 ? 4 : 7;
        if (L != 3) return ctx->fail(PS_ERR_ARG, "unsupported configuration: --gauss-mode fixed9 / fixed15 needs levels == 3 (reference s_pyramid_fixed.cu:271-289)");
        s.view.cands_filled = 0;
        for (int o = 0; o < s.num_octaves; ++o) {
            const OctaveView& ov = s.view.oct[o];
            if (o == 0) {
                for (int l = 0; l < L + 3; ++l)
                    n += s.is_float ? launch_fixed_level0_f32(reinterpret_cast<const float*>(s.d_img), (size_t)s.w, s.w, s.h, ctx->cfg.upscale, ov, l,
                                                              ctx->abs0[l], S, s.d_interm, s.stream)
                                    : launch_fixed_level0_u8(s.d_img, u8_pitch(s.w), s.w, s.h, ctx->cfg.upscale, ov, l, ctx->abs0[l], S,
                                                             s.d_interm, s.stream);
            } else {
                if (direct) {
                    // ScaleDirect (s_pyramid_build.cu:478-486): level 0 straight from the input image (rows dd[o], columns inc[0])
                    r = s.is_float ? launch_level0_f32(reinterpret_cast<const float*>(s.d_img), (size_t)s.w, s.w, s.h, ctx->cfg.upscale,
                                                       ctx->cfg.sift_mode, ov, ctx->dd[o], ctx->rows[0], s.stream, o)
                                   : launch_level0_u8(s.d_img, u8_pitch(s.w), s.w, s.h, ctx->cfg.upscale, ctx->cfg.sift_mode, ov,
                                                      ctx->dd[o], ctx->rows[0], s.stream, o);
                    if (r < 0) return ctx->fail(PS_ERR_ARG, "unsupported level-0 filter span %d (octave %d)", ctx->dd[o].span, o);
                    n += r;
                } else {
                    n += launch_decimate(s.view.oct[o - 1], L, ov, s.stream);
                }
                for (int l = 1; l < L + 3; ++l) n += launch_fixed_levelN(ov, l, ctx->absn[l], S, s.d_interm, s.stream);
            }
            n += launch_dog_planes(ov, L + 2, s.stream);
        }
        ctx->launches += n;
        PS_CUDA(ctx, cudaGetLastError());
        return PS_OK;
    }
    // --gauss-mode relative / vlfeat-hw-interpolated (VLFeat_Relative, s_pyramid_build.cu:515-542): every pass merges pairs of
    // taps into interpolated fetches; simple per-pixel kernels (k_pyramid.cu), DoG and decimation by their own kernels, dense
    // extrema scan.
    if (ctx->cfg.gauss_mode == PS_GAUSS_VLFEAT_RELATIVE) {
        s.view.cands_filled = 0;
        for (int o = 0; o < s.num_octaves; ++o) {
            const OctaveView& ov = s.view.oct[o];
            if (o == 0 || direct) {
                // (ScaleDirect, s_pyramid_build.cu:499-508: level 0 of every octave from the input image, dd row of the octave)
                if (s.is_float)
                    r = launch_level0_rows_f32(reinterpret_cast<const float*>(s.d_img), (size_t)s.w, s.w, s.h, ctx->cfg.upscale,
                                               ctx->cfg.sift_mode, ov, s.d_interm, ctx->dd[o], s.stream, o);
                else
                    r = launch_level0_rows_u8(s.d_img, u8_pitch(s.w), s.w, s.h, ctx->cfg.upscale, ctx->cfg.sift_mode, ov, s.d_interm,
                                              ctx->dd[o], s.stream, o);
                if (r < 0) return ctx->fail(PS_ERR_ARG, "unsupported level-0 filter span %d (octave %d)", ctx->dd[o].span, o);
                n += r;
                n += launch_interp_pass(s.d_interm, ov.gauss, ov.w, ov.h, ov.pitch, ctx->irows[0], ctx->irows[0].span, 0, s.stream);
            } else {
                n += launch_decimate(s.view.oct[o - 1], L, ov, s.stream);
            }
            for (int l = 1; l < L + 3; ++l) {
                n += launch_interp_pass(ov.gauss + ov.plane * (l - 1), s.d_interm, ov.w, ov.h, ov.pitch, ctx->irows[l], ctx->irows[l].span, 1, s.stream);
                n += launch_interp_pass(s.d_interm, ov.gauss + ov.plane * l, ov.w, ov.h, ov.pitch, ctx->irows[l], ctx->irows[l].span, 0, s.stream);
            }
            n += launch_dog_planes(ov, L + 2, s.stream);
        }
        ctx->launches += n;
        PS_CUDA(ctx, cudaGetLastError());
        return PS_OK;
    }
    // --gauss-mode vlfeat-direct (VLFeat_Relative_All, s_pyramid_build.cu:543-546; under ScaleDirect the direct-scaling
    // arm comes first, :499): every level of octave 0 straight from the input image
    const bool abs_o0 = ctx->cfg.gauss_mode == PS_GAUSS_VLFEAT_RELATIVE_ALL && !direct;
    bool collects = L <= kMaxLevels && !abs_o0;
    for (int l = 2; l <= L + 1 && collects; ++l) collects = blur_level_collects(ctx->rows[l]);
    for (int o = 0; o < s.num_octaves && collects; ++o) collects = s.view.oct[o].w <= 65535 && s.view.oct[o].h <= 65535;
    s.view.cands_filled = collects ? 1 : 0;
    if (abs_o0) {
        for (int l = 0; l < L + 3; ++l) {
            if (s.is_float)
                r = launch_level0_abs_f32(reinterpret_cast<const float*>(s.d_img), (size_t)s.w, s.w, s.h, ctx->cfg.upscale,
                                          ctx->cfg.sift_mode, s.view.oct[0], l, ctx->abs0[l], s.stream);
            else
                r = launch_level0_abs_u8(s.d_img, u8_pitch(s.w), s.w, s.h, ctx->cfg.upscale, ctx->cfg.sift_mode, s.view.oct[0], l,
                                         ctx->abs0[l], s.stream);
            if (r < 0) return ctx->fail(PS_ERR_ARG, "unsupported filter span %d (octave 0, level %d)", ctx->abs0[l].span, l);
            n += r;
        }
        n += launch_dog_planes(s.view.oct[0], L + 2, s.stream);
        if (s.num_octaves > 1) n += launch_decimate(s.view.oct[0], L, s.view.oct[1], s.stream);
    } else {
    if (s.is_float)
        r = launch_level0_f32(reinterpret_cast<const float*>(s.d_img), (size_t)s.w, s.w, s.h, ctx->cfg.upscale,
                              ctx->cfg.sift_mode, s.view.oct[0], ctx->dd0, ctx->rows[0], s.stream);
    else
        r = launch_level0_u8(s.d_img, u8_pitch(s.w), s.w, s.h, ctx->cfg.upscale, ctx->cfg.sift_mode, s.view.oct[0],
                             ctx->dd0, ctx->rows[0], s.stream);
    if (r < 0) return ctx->fail(PS_ERR_ARG, "unsupported level-0 filter span %d", ctx->dd0.span);
    n += r;
    }
    bool forked[Slot::kSides] = {};
    for (int o = 0; o < s.num_octaves; ++o) {
        const bool last = (o + 1 == s.num_octaves);
        if (direct && o > 0) {
            if (s.is_float)
                r = launch_level0_f32(reinterpret_cast<const float*>(s.d_img), (size_t)s.w, s.w, s.h, ctx->cfg.upscale,
                                      ctx->cfg.sift_mode, s.view.oct[o], ctx->dd[o], ctx->rows[0], s.stream, o);
            else
                r = launch_level0_u8(s.d_img, u8_pitch(s.w), s.w, s.h, ctx->cfg.upscale, ctx->cfg.sift_mode, s.view.oct[o],
                                     ctx->dd[o], ctx->rows[0], s.stream, o);
            if (r < 0) return ctx->fail(PS_ERR_ARG, "unsupported level-0 filter span %d (octave %d)", ctx->dd[o].span, o);
            n += r;
        }
        for (int l = 1; l < L + 3 && !(abs_o0 && o == 0); ++l) {
            // Config::ScaleDirect (s_pyramid_build.cu:499-514): level 0 of EVERY octave comes straight from the input image
            // (rows: the dd table of the octave, columns: the level-0 table), nothing is decimated from the octave above
            const OctaveView* next = (l == L && !last && !direct) ? &s.view.oct[o + 1] : nullptr;
            cudaStream_t st = s.stream;
            if (fork && !last && l > L) {
                const int sd = o % Slot::kSides;
                if (l == L + 1) {
                    PS_CUDA(ctx, cudaEventRecord(s.ev_fork[o], s.stream));
                    PS_CUDA(ctx, cudaStreamWaitEvent(s.side[sd], s.ev_fork[o], 0));
                    forked[sd] = true;
                }
                st = s.side[sd];
            }
            CandSink cs;
            const bool has_sink = level_sink(ctx, s, o, l, cs);
            r = launch_blur_level(s.view.oct[o], l, ctx->rows[l], next, has_sink ? &cs : nullptr, st);
            if (r < 0) return ctx->fail(PS_ERR_ARG, "unsupported filter span %d", ctx->rows[l].span);
            n += r;
        }
    }
    for (int sd = 0; sd < Slot::kSides; ++sd)
        if (forked[sd]) {
            PS_CUDA(ctx, cudaEventRecord(s.ev_join[sd], s.side[sd]));
            PS_CUDA(ctx, cudaStreamWaitEvent(s.stream, s.ev_join[sd], 0));
        }
    ctx->launches += n;
    PS_CUDA(ctx, cudaGetLastError());
    return PS_OK;
}

} // namespace

int psb::sm_count()
{
    static std::mutex mu;
    static int cached[64] = {};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) { cudaGetLastError(); return 148; }
    std::lock_guard<std::mutex> g(mu);
    if (cached[dev] == 0) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n < 1) { cudaGetLastError(); n = 148; }
        cached[dev] = n;
    }
    return cached[dev];
}

// the slot's view of the constants: its own (growable) capacities
static Consts slot_consts(const ps_ctx* ctx, const Slot& s)
{
    Consts k = ctx->k;
    k.ext_capacity = s.ext_cap;
    k.desc_capacity = s.desc_cap;
    return k;
}

// orientation -> descriptors -> Feature records -> counters to the host; everything after the (optional) grid filter
static int run_tail(ps_ctx* ctx, Slot& s, bool tm)
{
    const Consts k = slot_consts(ctx, s);
    PS_CUDA(ctx, cudaMemsetAsync(s.d_ori_slice, 0, sizeof(int) * ((size_t)s.ext_cap / PS_ORI_SLICE + 1), s.stream));
    int n = launch_orientation(s.view, k, s.d_iext, s.d_iext_f, s.d_ext, s.d_f2e, s.d_ori_slice, s.d_ct, s.stream);
    if (tm) PS_CUDA(ctx, cudaEventRecord(s.ev[4], s.stream));
    if (ctx->cfg.desc_mode == PS_DESC_LOOP) n += launch_descriptors(s.view, k, s.d_ext, s.d_f2e, s.d_desc, s.d_ct, s.stream);
    else n += launch_descriptors_mode(ctx->cfg.desc_mode, s.view, k, s.d_ext, s.d_f2e, s.d_desc, s.d_ct, s.stream);
    n += launch_prep_features(k, s.d_ext, s.d_feat, s.d_ct, s.stream);
    if (tm) PS_CUDA(ctx, cudaEventRecord(s.ev[5], s.stream));
    ctx->launches += n;
    PS_CUDA(ctx, cudaGetLastError());
    PS_CUDA(ctx, cudaMemcpyAsync(s.h_ct, s.d_ct, sizeof(Counters), cudaMemcpyDeviceToHost, s.stream));
    return PS_OK;
}

// More extrema or descriptors than the slot's buffers hold: grow them and run the tail of the pipeline again on the
// planes and initial extrema that are still in the slot (reference: Pyramid::reallocExtrema, sift_pyramid.cu:179-209,
// called from the orientation / descriptor stages).  Rare: the buffers start at 2 x max_extrema records.
static int regrow_slot(ps_ctx* ctx, Slot& s)
{
    for (int round = 0; round < 3 && s.h_ct->overflow; ++round) {
        const Counters& c = *s.h_ct;
        const int* counts = c.filtered ? c.ext_ct_f : c.ext_ct;
        long long need_ext = 0;
        for (int o = 0; o < s.num_octaves; ++o) need_ext += std::min(counts[o], ctx->k.max_extrema);
        const long long need_desc = c.ori_needed;
        if (need_ext > s.ext_cap) {
            const int cap = (int)std::min<long long>(need_ext + need_ext / 8 + 1024, 0x7ffffff0);
            cudaFree(s.d_ext); cudaFree(s.d_feat); cudaFree(s.d_ori_slice);
            s.d_ext = nullptr; s.d_feat = nullptr; s.d_ori_slice = nullptr; s.ext_cap = 0;
            PS_CUDA(ctx, cudaMalloc(&s.d_ext, sizeof(ps_extremum) * (size_t)cap));
            PS_CUDA(ctx, cudaMalloc(&s.d_feat, sizeof(ps_feature) * (size_t)cap));
            PS_CUDA(ctx, cudaMalloc(&s.d_ori_slice, sizeof(int) * ((size_t)cap / PS_ORI_SLICE + 1)));
            s.ext_cap = cap;
        }
        const long long want_desc = std::max<long long>(need_desc, (c.overflow & 1) ? need_ext * 5 / 4 : 0);
        if (want_desc > s.desc_cap) {
            const int cap = (int)std::min<long long>(want_desc + want_desc / 8 + 1024, 0x3ffffff0);
            cudaFree(s.d_desc); cudaFree(s.d_f2e);
            s.d_desc = nullptr; s.d_f2e = nullptr; s.desc_cap = 0;
            PS_CUDA(ctx, cudaMalloc(&s.d_desc, sizeof(ps_descriptor) * (size_t)cap));
            PS_CUDA(ctx, cudaMalloc(&s.d_f2e, sizeof(int) * (size_t)cap));
            s.desc_cap = cap;
        }
        // reset what the tail writes (the per-octave extremum counts and the filter's verdict stay)
        Counters reset = c;
        reset.ext_total = reset.ori_total = reset.ori_needed = reset.overflow = reset.work_ori = reset.work_desc = 0;
        PS_CUDA(ctx, cudaMemcpyAsync(s.d_ct, &reset, sizeof(Counters), cudaMemcpyHostToDevice, s.stream));
        PS_CUDA(ctx, cudaStreamSynchronize(s.stream));          // `reset` lives on this stack frame
        int rc = run_tail(ctx, s, false);
        if (rc != PS_OK) return rc;
        PS_CUDA(ctx, cudaEventRecord(s.done, s.stream));
        PS_CUDA(ctx, cudaEventSynchronize(s.done));
        s.graph_ok = false;                  // the captured graph holds the old buffer addresses
    }
    return PS_OK;
}

// everything between the input copy and the `done` event: memsets, pyramid, extrema, (grid filter), orientation,
// descriptors, Feature records, counters to the host.  Issued directly, or once under stream capture (below).
static int enqueue_pipeline(ps_ctx* ctx, Slot& s, bool tm, int* launched)
{
    int rc;
    const long long before = ctx->launches.load();
    PS_CUDA(ctx, cudaMemsetAsync(s.d_ct, 0, sizeof(Counters), s.stream));
    PS_CUDA(ctx, cudaMemsetAsync(s.cand_cnt, 0, s.cand_cnt_bytes, s.stream));
    if (tm) PS_CUDA(ctx, cudaEventRecord(s.ev[1], s.stream));
    if ((rc = run_pyramid(ctx, s)) != PS_OK) return rc;
    if (tm) PS_CUDA(ctx, cudaEventRecord(s.ev[2], s.stream));
    int n = launch_find_extrema(s.view, ctx->k, s.d_iext, s.d_ct, s.stream);
    if (tm) PS_CUDA(ctx, cudaEventRecord(s.ev[3], s.stream));
    {
        // grid filter (off by default): between extrema and orientation, like the reference (s_orientation.cu:380-383)
        const FilterCfg fc = {ctx->cfg.filter_max_extrema, ctx->cfg.filter_grid_size, ctx->cfg.filter_sort};
        n += launch_grid_filter(s.view, ctx->k, fc, s.d_iext, s.d_iext_f, s.d_keep, (size_t)s.num_octaves * ctx->k.max_extrema,
                                s.d_plan, s.d_ct, s.stream);
    }
    ctx->launches += n;
    if ((rc = run_tail(ctx, s, tm)) != PS_OK) return rc;
    if (launched) *launched = (int)(ctx->launches.load() - before);
    return PS_OK;
}

// POPSIFT_B200_GRAPH=0 issues every launch of every frame individually (A/B switch)
static bool graph_choice()
{
    static const bool v = [] { const char* e = getenv("POPSIFT_B200_GRAPH"); return !(e && e[0] == '0'); }();
    return v;
}

// The per-frame work of a slot is the same ~35 launches, memsets and stream forks for every image of one geometry, on
// buffers that do not move: from the second image of a geometry on it is replayed as ONE CUDA graph launch (captured
// from the slot's own stream, side stream included).  The submitting thread then makes 3 driver calls per frame
// instead of ~45 -- on a busy host (this path is driven from one thread per GPU) that is the difference between a
// GPU-bound and a launch-bound pipeline.  The first image of a geometry runs un-captured so that every lazy
// initialisation (shared-memory opt-ins, tensor-map encoder lookup, constant tables) happens outside a capture.
static int submit_common(ps_ctx* ctx, Slot& s)
{
    const bool tm = ctx->timing;
    int rc;
    const bool want_graph = graph_choice() && !tm && !ctx->graph_broken;
    if (want_graph && s.graph_ok && s.graph_w == s.w && s.graph_h == s.h && s.graph_float == s.is_float) {
        PS_CUDA(ctx, cudaGraphLaunch(s.graph_exec, s.stream));
        ctx->launches += s.graph_launches;
    } else if (want_graph && s.warm_w == s.w && s.warm_h == s.h && s.warm_float == s.is_float) {
        // second image of this geometry: capture while issuing
        if (s.graph_exec) { cudaGraphExecDestroy(s.graph_exec); s.graph_exec = nullptr; }
        s.graph_ok = false;
        cudaGraph_t g = nullptr;
        int launched = 0;
        cudaError_t e = cudaStreamBeginCapture(s.stream, cudaStreamCaptureModeRelaxed);
        if (e == cudaSuccess) {
            rc = enqueue_pipeline(ctx, s, false, &launched);
            e = cudaStreamEndCapture(s.stream, &g);
            if (rc == PS_OK && e == cudaSuccess && g) e = cudaGraphInstantiate(&s.graph_exec, g, 0);
            else if (e == cudaSuccess) e = cudaErrorUnknown;
            if (g) cudaGraphDestroy(g);
        }
        if (e != cudaSuccess || !s.graph_exec) {
            // capture is an optimisation: fall back to direct launches for this context and say so once
            cudaGetLastError();
            ctx->graph_broken = true;
            fprintf(stderr, "popsift_b200: CUDA graph capture failed (%s); launching directly\n", cudaGetErrorString(e));
            if ((rc = enqueue_pipeline(ctx, s, tm, nullptr)) != PS_OK) return rc;
        } else {
            s.graph_ok = true; s.graph_w = s.w; s.graph_h = s.h; s.graph_float = s.is_float; s.graph_launches = launched;
            PS_CUDA(ctx, cudaGraphLaunch(s.graph_exec, s.stream));       // the capture recorded the work, it did not run it
        }
    } else {
        if ((rc = enqueue_pipeline(ctx, s, tm, nullptr)) != PS_OK) return rc;
        s.warm_w = s.w; s.warm_h = s.h; s.warm_float = s.is_float;
    }
    PS_CUDA(ctx, cudaEventRecord(s.done, s.stream));
    s.submitted = true;
    return PS_OK;
}

static Slot* get_slot(ps_ctx* ctx, int slot)
{
    if (!ctx || slot < 0 || slot >= (int)ctx->slots.size()) return nullptr;
    return &ctx->slots[slot];
}

extern "C" const char* ps_last_error(const ps_ctx* ctx)
{
    if (!ctx) return g_create_error.c_str();
    std::lock_guard<std::mutex> g(ctx->err_mu);
    return ctx->err.c_str();
}

extern "C" void ps_destroy(ps_ctx* ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    for (Slot& s : ctx->slots) {
        if (s.stream) cudaStreamSynchronize(s.stream);
        cudaFree(s.d_img); cudaFreeHost(s.h_img); cudaFree(s.d_planes); cudaFree(s.d_interm); cudaFree(s.d_iext); cudaFree(s.d_iext_f); cudaFree(s.d_keep); cudaFree(s.d_plan); cudaFree(s.d_ext); cudaFree(s.d_ori_slice);
        cudaFree(s.d_feat); cudaFree(s.d_desc); cudaFree(s.d_f2e); cudaFree(s.d_ct); cudaFreeHost(s.h_ct);
        cudaFreeHost(s.h_feat); cudaFreeHost(s.h_desc);
        for (auto& e : s.ev) if (e) cudaEventDestroy(e);
        if (s.done) cudaEventDestroy(s.done);
        if (s.graph_exec) cudaGraphExecDestroy(s.graph_exec);
        if (s.in_done) cudaEventDestroy(s.in_done);
        for (auto& e : s.ev_fork) if (e) cudaEventDestroy(e);
        for (auto& e : s.ev_join) if (e) cudaEventDestroy(e);
        for (auto& st : s.side) if (st) cudaStreamDestroy(st);
        if (s.stream) cudaStreamDestroy(s.stream);
    }
    delete ctx;
}

extern "C" ps_ctx* ps_create(int device, const ps_config* cfg, int max_w, int max_h, int n_slots)
{
    auto bail = [&](const char* msg, cudaError_t e) -> ps_ctx* {
        g_create_error = std::string(msg) + (e != cudaSuccess ? std::string(": ") + cudaGetErrorString(e) : std::string());
        return nullptr;
    };
    if (!cfg || max_w < 1 || max_h < 1 || n_slots < 1 || n_slots > 64) return bail("ps_create: bad argument", cudaSuccess);
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) return bail("ps_create: no CUDA device (this library has no CPU fallback)", e);
    if (device < 0 || device >= ndev) return bail("ps_create: bad device index", cudaSuccess);
    if ((e = cudaSetDevice(device)) != cudaSuccess) return bail("cudaSetDevice", e);

    ps_ctx* ctx = new ps_ctx;
    ctx->device = device;
    ctx->cfg = *cfg;
    ctx->cfg.levels = std::max(2, cfg->levels);       // reference popsift.cpp:86
    ctx->levels = ctx->cfg.levels;
    if (ctx->cfg.max_extrema < 1) ctx->cfg.max_extrema = 100000;
    // Options whose numerics are not implemented are refused, never silently replaced by the default path.
    {
        const char* why = nullptr;
        if (ctx->cfg.desc_mode < PS_DESC_LOOP || ctx->cfg.desc_mode > PS_DESC_NOTILE)
            why = "ps_create: bad descriptor mode";
        else if (ctx->cfg.scaling_mode != PS_SCALE_DEFAULT && ctx->cfg.scaling_mode != PS_SCALE_DIRECT)
            why = "ps_create: bad scaling mode";
        else if ((ctx->cfg.gauss_mode == PS_GAUSS_FIXED9 || ctx->cfg.gauss_mode == PS_GAUSS_FIXED15) && std::max(2, ctx->cfg.levels) != 3)
            why = "ps_create: unsupported configuration: --gauss-mode fixed9 / fixed15 needs levels == 3 (reference s_pyramid_fixed.cu:271-289)";
        else if (ctx->cfg.sift_mode != PS_MODE_POPSIFT && ctx->cfg.sift_mode != PS_MODE_OPENCV && ctx->cfg.sift_mode != PS_MODE_VLFEAT)
            why = "ps_create: bad sift mode";
        else if (ctx->cfg.filter_max_extrema > 0 && !kGridFilterBuilt)
            why = "ps_create: unsupported configuration: the grid filter (--filter-max-extrema) is not implemented";
        else if (ctx->cfg.filter_max_extrema > 0 && (ctx->cfg.filter_grid_size < 1 || ctx->cfg.filter_grid_size > PS_MAX_FILTER_GRID))
            why = "ps_create: unsupported configuration: filter grid size out of range";
        if (why) { delete ctx; return bail(why, cudaSuccess); }
    }
    if (ps_gauss_tables_compute(&ctx->cfg, &ctx->tab) != PS_OK) {
        delete ctx;
        return bail("ps_create: unsupported configuration (sigma > 2.0 or levels > 12)", cudaSuccess);
    }
    for (int l = 0; l < PS_GAUSS_LEVELS; ++l) {
        std::memcpy(ctx->rows[l].tap, &ctx->tab.inc_filter[l * PS_GAUSS_ALIGN], sizeof(float) * PS_GAUSS_ALIGN);
        ctx->rows[l].span = ctx->tab.inc_span[l];
    }
    std::memcpy(ctx->dd0.tap, ctx->tab.dd_filter0, sizeof(float) * PS_GAUSS_ALIGN);
    ctx->dd0.span = ctx->tab.dd_span0;
    for (int o = 0; o < kMaxOctaves && o < PS_MAX_OCTAVES; ++o) {
        std::memcpy(ctx->dd[o].tap, &ctx->tab.dd_filter[o * PS_GAUSS_ALIGN], sizeof(float) * PS_GAUSS_ALIGN);
        ctx->dd[o].span = ctx->tab.dd_span[o];
    }
    for (int l = 0; l < PS_GAUSS_LEVELS; ++l) {
        std::memcpy(ctx->abs0[l].tap, &ctx->tab.abs_filter[l * PS_GAUSS_ALIGN], sizeof(float) * PS_GAUSS_ALIGN);
        ctx->abs0[l].span = ctx->tab.abs_span[l];
        std::memcpy(ctx->irows[l].tap, &ctx->tab.inc_ifilter[l * PS_GAUSS_ALIGN], sizeof(float) * PS_GAUSS_ALIGN);
        ctx->irows[l].span = ctx->tab.inc_ispan[l];
        std::memcpy(ctx->absn[l].tap, &ctx->tab.absn_filter[l * PS_GAUSS_ALIGN], sizeof(float) * PS_GAUSS_ALIGN);
        ctx->absn[l].span = ctx->tab.absn_span[l];
    }
    ctx->max_w = max_w; ctx->max_h = max_h;
    int32_t W[kMaxOctaves], H[kMaxOctaves];
    ctx->max_octaves = ps_geometry(&ctx->cfg, max_w, max_h, W, H);
    if (ctx->max_octaves < 1) { delete ctx; return bail("ps_create: bad geometry", cudaSuccess); }

    Consts& k = ctx->k;
    k.sigma0 = ctx->cfg.sigma;
    k.sigma_k = ctx->tab.sigma_k;
    k.edge_limit = ctx->cfg.edge_limit;
    k.threshold = ctx->tab.peak_threshold;
    k.max_extrema = ctx->cfg.max_extrema;
    // initial capacity of one slot: like the reference (max_extrema Extremum records and max(2, 1.25) * max_extrema
    // descriptors, sift_pyramid.cu:136-159) it grows on demand -- ps_counts re-runs orientation and descriptors
    // with larger buffers when a frame overflows them (regrow_slot).  POPSIFT_B200_INIT_CAP overrides (tests).
    k.ext_capacity = 2 * k.max_extrema;
    k.desc_capacity = 2 * k.max_extrema;
    if (const char* e = getenv("POPSIFT_B200_INIT_CAP")) { const int c = atoi(e); if (c > 0) k.ext_capacity = k.desc_capacity = c; }
    k.norm_multi = ctx->cfg.norm_multi;
    k.norm_mode = ctx->cfg.norm_mode;
    k.sift_mode = ctx->cfg.sift_mode;
    k.up_fac = (int)ctx->cfg.upscale;

    const size_t planes = plane_budget(ctx->cfg, max_w, max_h, ctx->levels);
    ctx->slots.resize(n_slots);
    for (Slot& s : ctx->slots) {
#define PS_TRY(call) if ((e = (call)) != cudaSuccess) { std::string m = #call; ps_destroy(ctx); return bail(m.c_str(), e); }
        PS_TRY(cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking));
        for (auto& st : s.side) PS_TRY(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
        for (auto& ev : s.ev_fork) PS_TRY(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        for (auto& ev : s.ev_join) PS_TRY(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        PS_TRY(cudaMalloc(&s.d_img, (size_t)max_w * max_h * 4));
        // the padding bytes between an image row and its pitch are read (never used) by the level-0 kernel's 4-byte copies
        PS_TRY(cudaMemset(s.d_img, 0, (size_t)max_w * max_h * 4));
        PS_TRY(cudaHostAlloc(&s.h_img, (size_t)max_w * max_h * 4, cudaHostAllocDefault));
        PS_TRY(cudaMalloc(&s.d_planes, planes * sizeof(float)));
        // once, so that the extrema kernel's speculative read of a candidate list beyond its count (k_extrema.cu, `prepare`)
        // and the padding columns of the planes are defined memory
        PS_TRY(cudaMemset(s.d_planes, 0, planes * sizeof(float)));
        s.planes_floats = planes;
        if (ctx->cfg.gauss_mode == PS_GAUSS_VLFEAT_RELATIVE || ctx->cfg.gauss_mode == PS_GAUSS_FIXED9 || ctx->cfg.gauss_mode == PS_GAUSS_FIXED15) {
            int32_t W0[kMaxOctaves], H0[kMaxOctaves];
            ps_geometry(&ctx->cfg, max_w, max_h, W0, H0);
            PS_TRY(cudaMalloc(&s.d_interm, sizeof(float) * (size_t)((W0[0] + 31) / 32 * 32 + 32) * (size_t)H0[0]));
        }
        PS_TRY(cudaMalloc(&s.d_iext, sizeof(InitialExtremum) * (size_t)ctx->max_octaves * k.max_extrema));
        if (ctx->cfg.filter_max_extrema > 0) {
            PS_TRY(cudaMalloc(&s.d_iext_f, sizeof(InitialExtremum) * (size_t)ctx->max_octaves * k.max_extrema));
            PS_TRY(cudaMalloc(&s.d_keep, (size_t)ctx->max_octaves * k.max_extrema));
            PS_TRY(cudaMalloc(&s.d_plan, sizeof(FilterPlan)));
        }
        s.ext_cap = k.ext_capacity; s.desc_cap = k.desc_capacity;
        PS_TRY(cudaMalloc(&s.d_ext, sizeof(ps_extremum) * (size_t)k.ext_capacity));
        PS_TRY(cudaMalloc(&s.d_feat, sizeof(ps_feature) * (size_t)k.ext_capacity));
        PS_TRY(cudaMalloc(&s.d_desc, sizeof(ps_descriptor) * (size_t)k.desc_capacity));
        PS_TRY(cudaMalloc(&s.d_f2e, sizeof(int) * (size_t)k.desc_capacity));
        PS_TRY(cudaMalloc(&s.d_ct, sizeof(Counters)));
        PS_TRY(cudaMalloc(&s.d_ori_slice, sizeof(int) * ((size_t)k.ext_capacity / PS_ORI_SLICE + 1)));
        PS_TRY(cudaHostAlloc(&s.h_ct, sizeof(Counters), cudaHostAllocDefault));
        for (auto& ev : s.ev) PS_TRY(cudaEventCreate(&ev));
        PS_TRY(cudaEventCreateWithFlags(&s.done, cudaEventDisableTiming));
        PS_TRY(cudaEventCreateWithFlags(&s.in_done, cudaEventDisableTiming));
#undef PS_TRY
    }
    return ctx;
}

static bool is_pinned(const void* p);

static int stage_input(ps_ctx* ctx, Slot& s, const void* host_img, size_t bytes)
{
    // Pinned caller memory goes straight to the device (the caller keeps it valid until ps_wait_input /
    // ps_counts / ps_sync returns for this slot); pageable memory is staged through the slot's pinned
    // buffer (the reference always stages: popsift.cpp:392-395 + s_image.cu:75) and may be reused as soon
    // as the call returns.
    const bool pinned = is_pinned(host_img);
    const void* src = host_img;
    if (!pinned) {
        // the staging buffer is free once the PREVIOUS image's copy has left it -- the submitting thread
        // never waits for the previous image's kernels
        if (s.in_pending) PS_CUDA(ctx, cudaEventSynchronize(s.in_done));
        std::memcpy(s.h_img, host_img, bytes);
        src = s.h_img;
    }
    if (!s.is_float && u8_pitch(s.w) != (size_t)s.w)
        PS_CUDA(ctx, cudaMemcpy2DAsync(s.d_img, u8_pitch(s.w), src, (size_t)s.w, (size_t)s.w, (size_t)s.h,
                                       cudaMemcpyHostToDevice, s.stream));
    else
        PS_CUDA(ctx, cudaMemcpyAsync(s.d_img, src, bytes, cudaMemcpyHostToDevice, s.stream));
    PS_CUDA(ctx, cudaEventRecord(s.in_done, s.stream));
    s.in_pending = true;
    return PS_OK;
}

extern "C" int ps_submit_u8(ps_ctx* ctx, int slot, const uint8_t* host_img, int w, int h)
{
    Slot* s = get_slot(ctx, slot);
    if (!s || !host_img) return ctx ? ctx->fail(PS_ERR_ARG, "ps_submit_u8: bad argument") : PS_ERR_ARG;
    if (w < 1 || h < 1 || w > ctx->max_w || h > ctx->max_h)
        return ctx->fail(PS_ERR_TOO_LARGE, "image %dx%d exceeds context maximum %dx%d", w, h, ctx->max_w, ctx->max_h);
    PS_CUDA(ctx, cudaSetDevice(ctx->device));
    int rc = build_view(ctx, *s, w, h);
    if (rc != PS_OK) return rc;
    s->is_float = false;
    if (ctx->timing) PS_CUDA(ctx, cudaEventRecord(s->ev[0], s->stream));
    if ((rc = stage_input(ctx, *s, host_img, (size_t)w * h)) != PS_OK) return rc;
    return submit_common(ctx, *s);
}

extern "C" int ps_submit_f32(ps_ctx* ctx, int slot, const float* host_img, int w, int h)
{
    Slot* s = get_slot(ctx, slot);
    if (!s || !host_img) return ctx ? ctx->fail(PS_ERR_ARG, "ps_submit_f32: bad argument") : PS_ERR_ARG;
    if (w < 1 || h < 1 || w > ctx->max_w || h > ctx->max_h)
        return ctx->fail(PS_ERR_TOO_LARGE, "image %dx%d exceeds context maximum %dx%d", w, h, ctx->max_w, ctx->max_h);
    PS_CUDA(ctx, cudaSetDevice(ctx->device));
    int rc = build_view(ctx, *s, w, h);
    if (rc != PS_OK) return rc;
    s->is_float = true;
    if (ctx->timing) PS_CUDA(ctx, cudaEventRecord(s->ev[0], s->stream));
    if ((rc = stage_input(ctx, *s, host_img, (size_t)w * h * sizeof(float))) != PS_OK) return rc;
    return submit_common(ctx, *s);
}

extern "C" int ps_submit_dev_u8(ps_ctx* ctx, int slot, const uint8_t* dev_img, size_t pitch, int w, int h)
{
    Slot* s = get_slot(ctx, slot);
    if (!s || !dev_img) return ctx ? ctx->fail(PS_ERR_ARG, "ps_submit_dev_u8: bad argument") : PS_ERR_ARG;
    if (w < 1 || h < 1 || w > ctx->max_w || h > ctx->max_h)
        return ctx->fail(PS_ERR_TOO_LARGE, "image %dx%d exceeds context maximum %dx%d", w, h, ctx->max_w, ctx->max_h);
    if (pitch < (size_t)w)
        return ctx->fail(PS_ERR_ARG, "ps_submit_dev_u8: pitch %zu is smaller than the image width %d", pitch, w);
    PS_CUDA(ctx, cudaSetDevice(ctx->device));
    int rc = build_view(ctx, *s, w, h);
    if (rc != PS_OK) return rc;
    s->is_float = false;
    if (ctx->timing) PS_CUDA(ctx, cudaEventRecord(s->ev[0], s->stream));
    PS_CUDA(ctx, cudaMemcpy2DAsync(s->d_img, u8_pitch(w), dev_img, pitch, (size_t)w, (size_t)h, cudaMemcpyDeviceToDevice, s->stream));
    // ps_wait_input: the caller may overwrite dev_img once this copy has left it
    PS_CUDA(ctx, cudaEventRecord(s->in_done, s->stream));
    s->in_pending = true;
    return submit_common(ctx, *s);
}

extern "C" int ps_wait_input(ps_ctx* ctx, int slot)
{
    Slot* s = get_slot(ctx, slot);
    if (!s) return PS_ERR_ARG;
    PS_CUDA(ctx, cudaSetDevice(ctx->device));
    if (s->in_pending) PS_CUDA(ctx, cudaEventSynchronize(s->in_done));
    return PS_OK;
}

extern "C" int ps_sync(ps_ctx* ctx, int slot)
{
    Slot* s = get_slot(ctx, slot);
    if (!s) return PS_ERR_ARG;
    PS_CUDA(ctx, cudaSetDevice(ctx->device));
    PS_CUDA(ctx, cudaStreamSynchronize(s->stream));
    return PS_OK;
}

extern "C" int ps_counts(ps_ctx* ctx, int slot, int32_t* n_feat, int32_t* n_desc)
{
    Slot* s = get_slot(ctx, slot);
    if (!s) return PS_ERR_ARG;
    if (!s->submitted) return ctx->fail(PS_ERR_STATE, "ps_counts: nothing submitted to slot %d", slot);
    PS_CUDA(ctx, cudaSetDevice(ctx->device));
    PS_CUDA(ctx, cudaEventSynchronize(s->done));
    if (s->h_ct->overflow) {
        // more extrema / descriptors than the slot's buffers hold: grow them and redo orientation + descriptors
        const int rc = regrow_slot(ctx, *s);
        if (rc != PS_OK) return rc;
    }
    if (n_feat) *n_feat = s->h_ct->ext_total;
    if (n_desc) *n_desc = s->h_ct->ori_total;
    if (s->h_ct->overflow)
        return ctx->fail(PS_ERR_OVERFLOW, "slot %d: capacity exceeded (flags %d); results truncated", slot, s->h_ct->overflow);
    return PS_OK;
}

static int grow_pinned(ps_ctx* ctx, void** p, size_t* cap, size_t need, size_t elem)
{
    if (need <= *cap) return PS_OK;
    size_t ncap = std::max(need, *cap * 2);
    ncap = std::max<size_t>(ncap, 4096);
    if (*p) PS_CUDA(ctx, cudaFreeHost(*p));
    *p = nullptr; *cap = 0;
    PS_CUDA(ctx, cudaHostAlloc(p, ncap * elem, cudaHostAllocDefault));
    *cap = ncap;
    return PS_OK;
}

static bool is_pinned(const void* p)
{
    cudaPointerAttributes at{};
    const bool yes = cudaPointerGetAttributes(&at, p) == cudaSuccess && at.type == cudaMemoryTypeHost;
    cudaGetLastError();
    return yes;
}

extern "C" void* ps_host_alloc(size_t bytes)
{
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}

extern "C" void ps_host_free(void* p)
{
    if (p) cudaFreeHost(p);
}

extern "C" int ps_download(ps_ctx* ctx, int slot, ps_feature* feat, ps_descriptor* desc)
{
    Slot* s = get_slot(ctx, slot);
    if (!s) return PS_ERR_ARG;
    if (!s->submitted) return ctx->fail(PS_ERR_STATE, "ps_download: nothing submitted to slot %d", slot);
    PS_CUDA(ctx, cudaSetDevice(ctx->device));
    PS_CUDA(ctx, cudaEventSynchronize(s->done));
    const size_t nf = (size_t)s->h_ct->ext_total, nd = (size_t)s->h_ct->ori_total;
    if (nf == 0) return PS_OK;
    if (!feat || (nd && !desc)) return ctx->fail(PS_ERR_ARG, "ps_download: null output array");
    int rc;
    // page-locked destinations receive the DMA directly; pageable ones go through the slot's staging
    const bool direct = is_pinned(feat) && (nd == 0 || is_pinned(desc));
    ps_feature* hf = feat;
    if (direct) {
        PS_CUDA(ctx, cudaMemcpyAsync(feat, s->d_feat, nf * sizeof(ps_feature), cudaMemcpyDeviceToHost, s->stream));
        if (nd) PS_CUDA(ctx, cudaMemcpyAsync(desc, s->d_desc, nd * sizeof(ps_descriptor), cudaMemcpyDeviceToHost, s->stream));
        PS_CUDA(ctx, cudaStreamSynchronize(s->stream));
    } else {
        if ((rc = grow_pinned(ctx, (void**)&s->h_feat, &s->h_feat_cap, nf, sizeof(ps_feature))) != PS_OK) return rc;
        if ((rc = grow_pinned(ctx, (void**)&s->h_desc, &s->h_desc_cap, nd, sizeof(ps_descriptor))) != PS_OK) return rc;
        PS_CUDA(ctx, cudaMemcpyAsync(s->h_feat, s->d_feat, nf * sizeof(ps_feature), cudaMemcpyDeviceToHost, s->stream));
        if (nd) PS_CUDA(ctx, cudaMemcpyAsync(s->h_desc, s->d_desc, nd * sizeof(ps_descriptor), cudaMemcpyDeviceToHost, s->stream));
        PS_CUDA(ctx, cudaStreamSynchronize(s->stream));
        if (nd) std::memcpy(desc, s->h_desc, nd * sizeof(ps_descriptor));
        hf = s->h_feat;
    }
    for (size_t i = 0; i < nf; ++i) {
        ps_feature f = hf[i];
        const int first = f.pad_;
        f.pad_ = 0;
        for (int r = 0; r < PS_MAX_ORI; ++r) f.desc[r] = (r < f.num_ori) ? desc + first + r : nullptr;
        feat[i] = f;
    }
    return PS_OK;
}

extern "C" int ps_download_dev(ps_ctx* ctx, int slot, ps_feature* d_feat, ps_descriptor* d_desc, int32_t* d_rev)
{
    Slot* s = get_slot(ctx, slot);
    if (!s) return PS_ERR_ARG;
    if (!s->submitted) return ctx->fail(PS_ERR_STATE, "ps_download_dev: nothing submitted to slot %d", slot);
    PS_CUDA(ctx, cudaSetDevice(ctx->device));
    PS_CUDA(ctx, cudaEventSynchronize(s->done));
    const size_t nf = (size_t)s->h_ct->ext_total, nd = (size_t)s->h_ct->ori_total;
    if (nf == 0) return PS_OK;
    if (!d_feat || (nd && (!d_desc || !d_rev))) return ctx->fail(PS_ERR_ARG, "ps_download_dev: null output array");
    PS_CUDA(ctx, cudaMemcpyAsync(d_feat, s->d_feat, nf * sizeof(ps_feature), cudaMemcpyDeviceToDevice, s->stream));
    if (nd) {
        PS_CUDA(ctx, cudaMemcpyAsync(d_desc, s->d_desc, nd * sizeof(ps_descriptor), cudaMemcpyDeviceToDevice, s->stream));
        PS_CUDA(ctx, cudaMemcpyAsync(d_rev, s->d_f2e, nd * sizeof(int32_t), cudaMemcpyDeviceToDevice, s->stream));
    }
    ctx->launches += launch_fix_feature_pointers(d_feat, d_desc, (int)nf, s->stream);
    PS_CUDA(ctx, cudaGetLastError());
    PS_CUDA(ctx, cudaStreamSynchronize(s->stream));
    return PS_OK;
}

extern "C" void* ps_dev_alloc(size_t bytes)
{
    void* p = nullptr;
    if (cudaMalloc(&p, bytes ? bytes : 1) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}

extern "C" void ps_dev_free(void* p)
{
    if (p) cudaFree(p);
}

extern "C" int ps_host_to_dev(void* dst_dev, const void* src_host, size_t bytes)
{
    if (bytes == 0) return PS_OK;
    if (!dst_dev || !src_host) return PS_ERR_ARG;
    if (cudaMemcpy(dst_dev, src_host, bytes, cudaMemcpyHostToDevice) != cudaSuccess) { cudaGetLastError(); return PS_ERR_CUDA; }
    return PS_OK;
}

extern "C" int ps_pointer_device(const void* dev_ptr)
{
    cudaPointerAttributes at{};
    if (!dev_ptr || cudaPointerGetAttributes(&at, dev_ptr) != cudaSuccess || at.type != cudaMemoryTypeDevice) { cudaGetLastError(); return -1; }
    return at.device;
}

extern "C" int ps_match(int device, const ps_descriptor* d_left, int n_left, const ps_descriptor* d_right, int n_right,
                        int32_t* d_out, int flags)
{
    if (n_left < 0 || n_right < 0 || (n_left > 0 && (!d_left || !d_out)) || (n_right > 0 && !d_right)) return PS_ERR_ARG;
    if (n_left == 0) return PS_OK;
    if (cudaSetDevice(device) != cudaSuccess) { cudaGetLastError(); return PS_ERR_CUDA; }
    const char* err = nullptr;
    const int n = run_match(d_left, n_left, d_right, n_right, d_out, flags, nullptr, &err);
    if (n < 0) { g_create_error = err ? err : "ps_match failed"; return PS_ERR_CUDA; }
    const cudaError_t e = cudaStreamSynchronize(nullptr);
    if (e != cudaSuccess) { g_create_error = std::string("ps_match: ") + cudaGetErrorString(e); cudaGetLastError(); return PS_ERR_CUDA; }
    return PS_OK;
}

extern "C" int ps_dev_to_host(void* dst_host, const void* src_dev, size_t bytes)
{
    if (bytes == 0) return PS_OK;
    if (!dst_host || !src_dev) return PS_ERR_ARG;
    if (cudaMemcpy(dst_host, src_dev, bytes, cudaMemcpyDeviceToHost) != cudaSuccess) { cudaGetLastError(); return PS_ERR_CUDA; }
    return PS_OK;
}

extern "C" int ps_debug_plane(ps_ctx* ctx, int slot, int octave, int level, int which, float* out)
{
    Slot* s = get_slot(ctx, slot);
    if (!s || !out) return PS_ERR_ARG;
    if (!s->submitted) return ctx->fail(PS_ERR_STATE, "ps_debug_plane: nothing submitted");
    if (octave < 0 || octave >= s->num_octaves) return ctx->fail(PS_ERR_ARG, "bad octave %d", octave);
    const int L = ctx->levels;
    const int nl = which == PS_PLANE_DOG ? L + 2 : L + 3;
    if (level < 0 || level >= nl) return ctx->fail(PS_ERR_ARG, "bad level %d", level);
    PS_CUDA(ctx, cudaSetDevice(ctx->device));
    PS_CUDA(ctx, cudaStreamSynchronize(s->stream));
    const OctaveView& v = s->view.oct[octave];
    const float* src = (which == PS_PLANE_DOG ? v.dog : v.gauss) + v.plane * level;
    PS_CUDA(ctx, cudaMemcpy2D(out, (size_t)v.w * sizeof(float), src, (size_t)v.pitch * sizeof(float),
                              (size_t)v.w * sizeof(float), v.h, cudaMemcpyDeviceToHost));
    return PS_OK;
}

extern "C" int ps_debug_level0_plan(int w, int h, int W, int H, float shift, int R)
{
    if (w < 1 || h < 1 || W < 1 || H < 1 || R < 0 || R >= PS_GAUSS_ALIGN) return PS_ERR_ARG;
    return psb::level0_plan_for(w, h, W, H, shift, R);
}

extern "C" int ps_debug_extrema(ps_ctx* ctx, int slot, ps_extremum* out, int cap)
{
    Slot* s = get_slot(ctx, slot);
    if (!s) return PS_ERR_ARG;
    if (!s->submitted) return ctx->fail(PS_ERR_STATE, "ps_debug_extrema: nothing submitted");
    PS_CUDA(ctx, cudaSetDevice(ctx->device));
    PS_CUDA(ctx, cudaEventSynchronize(s->done));
    const int n = s->h_ct->ext_total;
    const int m = std::min(n, cap);
    if (m > 0 && out) PS_CUDA(ctx, cudaMemcpy(out, s->d_ext, sizeof(ps_extremum) * (size_t)m, cudaMemcpyDeviceToHost));
    return n;
}

extern "C" int ps_slot_geometry(ps_ctx* ctx, int slot, int32_t* n_octaves, int32_t* W, int32_t* H)
{
    Slot* s = get_slot(ctx, slot);
    if (!s) return PS_ERR_ARG;
    if (n_octaves) *n_octaves = s->num_octaves;
    for (int o = 0; o < s->num_octaves; ++o) { if (W) W[o] = s->W[o]; if (H) H[o] = s->H[o]; }
    return PS_OK;
}

extern "C" int ps_set_timing(ps_ctx* ctx, int enable)
{
    if (!ctx) return PS_ERR_ARG;
    ctx->timing = enable != 0;
    return PS_OK;
}

extern "C" int ps_stage_ms(ps_ctx* ctx, int slot, float ms[PS_NUM_STAGES])
{
    Slot* s = get_slot(ctx, slot);
    if (!s || !ms) return PS_ERR_ARG;
    if (!ctx->timing || !s->submitted) return ctx->fail(PS_ERR_STATE, "ps_stage_ms: timing not enabled or nothing submitted");
    PS_CUDA(ctx, cudaSetDevice(ctx->device));
    PS_CUDA(ctx, cudaEventSynchronize(s->done));
    PS_CUDA(ctx, cudaEventSynchronize(s->ev[5]));
    for (int i = 0; i < 5; ++i) PS_CUDA(ctx, cudaEventElapsedTime(&ms[i], s->ev[i], s->ev[i + 1]));
    PS_CUDA(ctx, cudaEventElapsedTime(&ms[PS_STAGE_TOTAL], s->ev[0], s->ev[5]));
    return PS_OK;
}

extern "C" int64_t ps_launch_count(const ps_ctx* ctx) { return ctx ? ctx->launches.load() : 0; }

extern "C" void* ps_slot_stream(ps_ctx* ctx, int slot)
{
    Slot* s = get_slot(ctx, slot);
    return s ? (void*)s->stream : nullptr;
}

extern "C" int ps_run_pyramid_only(ps_ctx* ctx, int slot)
{
    Slot* s = get_slot(ctx, slot);
    if (!s) return PS_ERR_ARG;
    if (!s->submitted) return ctx->fail(PS_ERR_STATE, "ps_run_pyramid_only: nothing submitted");
    PS_CUDA(ctx, cudaSetDevice(ctx->device));
    // start from empty candidate tiles like a submit does
    PS_CUDA(ctx, cudaMemsetAsync(s->cand_cnt, 0, s->cand_cnt_bytes, s->stream));
    return run_pyramid(ctx, *s);
}

extern "C" int ps_run_level_only(ps_ctx* ctx, int slot, int octave, int level)
{
    Slot* s = get_slot(ctx, slot);
    if (!s) return PS_ERR_ARG;
    if (!s->submitted) return ctx->fail(PS_ERR_STATE, "ps_run_level_only: nothing submitted");
    const int L = ctx->levels;
    if (octave < 0 || octave >= s->num_octaves || level < 0 || level >= L + 3 || (level == 0 && octave != 0))
        return ctx->fail(PS_ERR_ARG, "ps_run_level_only: bad octave/level %d/%d", octave, level);
    PS_CUDA(ctx, cudaSetDevice(ctx->device));
    int r;
    if (level == 0) {
        r = s->is_float ? launch_level0_f32(reinterpret_cast<const float*>(s->d_img), (size_t)s->w, s->w, s->h, ctx->cfg.upscale,
                                            ctx->cfg.sift_mode, s->view.oct[0], ctx->dd0, ctx->rows[0], s->stream)
                        : launch_level0_u8(s->d_img, u8_pitch(s->w), s->w, s->h, ctx->cfg.upscale, ctx->cfg.sift_mode,
                                           s->view.oct[0], ctx->dd0, ctx->rows[0], s->stream);
    } else {
        const OctaveView* next = (level == L && octave + 1 < s->num_octaves) ? &s->view.oct[octave + 1] : nullptr;
        CandSink cs;
        const bool has_sink = level_sink(ctx, *s, octave, level, cs);
        if (has_sink)
            PS_CUDA(ctx, cudaMemsetAsync(cs.counts, 0, sizeof(int) * (size_t)s->view.oct[octave].cand_blocks, s->stream));
        r = launch_blur_level(s->view.oct[octave], level, ctx->rows[level], next, has_sink ? &cs : nullptr, s->stream);
    }
    if (r < 0) return ctx->fail(PS_ERR_ARG, "unsupported filter span");
    ctx->launches += r;
    PS_CUDA(ctx, cudaGetLastError());
    return PS_OK;
}
