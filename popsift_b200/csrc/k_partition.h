// Work partition of the marching pyramid kernels (k_pyramid_march.cu).  Plain C++ so that the host
// logic can be checked without a GPU (csrc/app/partition_check.cpp, tests/test_host_cpu.py).
#pragma once
#ifdef __CUDACC__
#define PSB_HD __host__ __device__ __forceinline__
#else
#define PSB_HD inline
#endif

namespace psb {

// Work partition: strips of TW columns x segments of whole chunk-rows (Q rows), ONE wave of CTAs
// (148 SMs x 4 resident CTAs).  CTAs of one segment index handle neighbouring strips, so CTAs that run
// side by side touch the same image rows and every DRAM page of a row is streamed by neighbouring CTAs
// at about the same time (a strip-major split of the same work measured ~30 % slower).
//
// S strips seldom divide the 592 slots: with nh segments of uh chunk-rows per strip, S*nh CTAs leave
// slots (and whole SMs' worth of issue bandwidth) idle.  The spare slots go to `light` strips, spread
// evenly over the image, that are cut into nl > nh shorter segments (ul chunk-rows).  Block b < S*nh is
// (strip b % S, segment b / S); the remaining blocks are the extra segments of the light strips.
struct Partition {
    int strips;         // S
    int nh, uh;         // segments per heavy strip, chunk-rows per segment
    int nl, ul;         // the same for light strips
    int heavy;          // number of heavy strips (== S: uniform partition)
    int B, pad;         // CTAs
};

// number of heavy strips with index <= s; heavy strip i sits at floor((i + 0.5) * S / heavy)
PSB_HD int heavy_upto(const Partition& p, int s)
{
    if (p.heavy >= p.strips) return s + 1;
    const int num = 2 * p.heavy * (s + 1) - p.strips;
    if (num <= 0) return 0;
    const int c = (num + 2 * p.strips - 1) / (2 * p.strips);
    return c < p.heavy ? c : p.heavy;
}

// block -> (strip, first row, end row); false when the block has no rows
PSB_HD bool locate(const Partition& p, int b, int H, int Q, int& strip, int& ys, int& ye)
{
    int seg, units;
    if (b < p.strips * p.nh) {
        strip = b % p.strips;
        seg = b / p.strips;
        const bool is_heavy = heavy_upto(p, strip) != heavy_upto(p, strip - 1);
        units = is_heavy ? p.uh : p.ul;
    } else {
        const int light = p.strips - p.heavy;
        const int e2 = b - p.strips * p.nh;
        const int e = e2 % light;                 // rank among the light strips
        seg = p.nh + e2 / light;
        int s = e;                                // smallest s with s == e + heavy_upto(s): the e-th light strip
        for (int it = 0; it <= p.heavy; ++it) {
            const int s2 = e + heavy_upto(p, s);
            if (s2 == s) break;
            s = s2;
        }
        strip = s;
        units = p.ul;
    }
    ys = seg * units * Q;
    ye = ys + units * Q;
    if (ye > H) ye = H;
    return ys < H;
}

inline Partition make_partition(int W, int H, int TW, int Q, int slots)
{
    Partition p;
    const int S = (W + TW - 1) / TW;
    const int C = (H + Q - 1) / Q;
    int n = slots / S;
    if (n < 1) n = 1;
    int u = (C + n - 1) / n;
    // Small planes (fewer chunk-rows than slots per strip) are latency-bound, not work-bound: a CTA that marches 4
    // chunk-rows plus its 2R warm-up rows takes 6 serial chunks where one chunk-row per CTA takes 3, and the extra
    // warm-up work runs on SMs that would otherwise idle.  (Round 1 kept u >= 4: octaves 2..4 of the 4K pyramid then
    // ran 10-20 us per launch at 6-11 % of the warps.)
    if (u < 1) u = 1;
    p.strips = S;
    p.uh = u;
    p.nh = (C + u - 1) / u;
    p.nl = p.nh; p.ul = u; p.heavy = S; p.pad = 0;
    if (u - 1 >= 4 && S * p.nh < slots) {
        const int nl = (C + u - 2) / (u - 1);
        if (nl > p.nh) {
            int x = (slots - S * p.nh) / (nl - p.nh);      // light strips that fit in the spare slots
            if (x > S) x = S;
            if (x > 0) {
                p.nl = nl;
                p.ul = (C + nl - 1) / nl;
                p.heavy = S - x;
            }
        }
    }
    p.B = S * p.nh + (S - p.heavy) * (p.nl - p.nh);
    return p;
}

// ---- candidate regions -----------------------------------------------------------------------
// Every block of a level kernel owns a private region of the level's candidate list, large enough for
// every pixel pair of its segment (units * Q rows x TW/2 pairs), and a count: reporting a candidate needs
// a shared-memory counter only, never a global atomic.
inline int cand_region_cap(const Partition& p, int TW, int Q) { return (p.uh > p.ul ? p.uh : p.ul) * Q * (TW / 2); }

inline long long cand_entries(const Partition& p, int TW, int Q) { return (long long)p.B * cand_region_cap(p, TW, Q); }

// upper bound of cand_entries(make_partition(W, H, ...)) that is monotonic in W and H (memory budget)
inline long long cand_entry_bound(int W, int H, int TW, int Q, int slots)
{
    const long long S = (W + TW - 1) / TW, C = (H + Q - 1) / Q;
    long long n = slots / S;
    if (n < 1) n = 1;
    return (S * (C + C / n + 5) + 4LL * slots + 3 * S) * Q * (TW / 2);
}

} // namespace psb
