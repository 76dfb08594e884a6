// Host check of the marching kernels' work partition (popsift_b200/csrc/k_partition.h): for a sweep of
// plane sizes every (strip, row) must be covered by exactly one block, no block may be empty beyond
// the ones `locate` rejects, and the grid must fit the slots whenever a single wave is possible.  Checked at
// the two slot counts the library partitions for on a B200 (148 SMs): 4 x 148 resident CTAs of the level
// kernels and 6 x 148 of the exact-2x level-0 kernel.
#include "k_partition.h"
#include <cstdio>
#include <vector>

int main()
{
    const int TW = 128, Q = 16;
    long checked = 0;
    for (const int slots : {592, 888})
        for (int W = 1; W <= 16384; W += (W < 300 ? 7 : 97))
            for (int H = 1; H <= 9000; H += (H < 200 ? 5 : 131)) {
                const psb::Partition p = psb::make_partition(W, H, TW, Q, slots);
                const int S = (W + TW - 1) / TW;
                if (p.strips != S || p.B < 1) { std::printf("FAIL strips/B slots=%d W=%d H=%d\n", slots, W, H); return 1; }
                if (S <= slots && p.uh > 4 && p.B > slots) { std::printf("FAIL wave slots=%d W=%d H=%d B=%d\n", slots, W, H, p.B); return 1; }
                if (psb::cand_entries(p, TW, Q) > psb::cand_entry_bound(W, H, TW, Q, slots)) {
                    std::printf("FAIL candidate bound slots=%d W=%d H=%d entries=%lld bound=%lld\n", slots, W, H, psb::cand_entries(p, TW, Q),
                                psb::cand_entry_bound(W, H, TW, Q, slots));
                    return 1;
                }
                std::vector<int> cover((size_t)S * H, 0);
                for (int b = 0; b < p.B; ++b) {
                    int strip = -1, ys = 0, ye = 0;
                    if (!psb::locate(p, b, H, Q, strip, ys, ye)) continue;
                    if (strip < 0 || strip >= S || ys < 0 || ye > H || ys >= ye || (ys % Q) != 0) {
                        std::printf("FAIL range slots=%d W=%d H=%d b=%d strip=%d ys=%d ye=%d\n", slots, W, H, b, strip, ys, ye);
                        return 1;
                    }
                    // a block's candidate region holds every pixel pair of its segment
                    if ((long long)(ye - ys) * (TW / 2) > psb::cand_region_cap(p, TW, Q)) {
                        std::printf("FAIL region slots=%d W=%d H=%d b=%d\n", slots, W, H, b);
                        return 1;
                    }
                    for (int y = ys; y < ye; ++y) ++cover[(size_t)strip * H + y];
                }
                for (size_t i = 0; i < cover.size(); ++i)
                    if (cover[i] != 1) {
                        std::printf("FAIL cover slots=%d W=%d H=%d strip=%zu y=%zu count=%d (S=%d nh=%d uh=%d nl=%d ul=%d heavy=%d B=%d)\n",
                                    slots, W, H, i / H, i % H, cover[i], p.strips, p.nh, p.uh, p.nl, p.ul, p.heavy, p.B);
                        return 1;
                    }
                ++checked;
            }
    const psb::Partition p4k = psb::make_partition(7680, 4320, TW, Q, 592);
    std::printf("OK %ld partitions; 7680x4320: S=%d nh=%d uh=%d nl=%d ul=%d heavy=%d B=%d\n", checked, p4k.strips, p4k.nh,
                p4k.uh, p4k.nl, p4k.ul, p4k.heavy, p4k.B);
    return 0;
}
