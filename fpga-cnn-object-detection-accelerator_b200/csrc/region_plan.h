// region_plan.h -- checks of a region array and the staging plan of a host-pointer region call (cnnacc_detect_regions /
// cnnacc_preprocess_regions; cnnacc_detect_frames / cnnacc_preprocess_bgr are the case of one centre region per frame).  Pure
// host arithmetic, no CUDA; tests/test_regions_cpu.py replays it through cnnacc_region_plan_host.
//
// A chunk stages the frames [f0, f1) with one copy and runs the regions [r0, r1) on them.  Its frames are a run of
// consecutive frames that regions reference, at most about 16 MiB of them, so a frame that no region references never
// crosses the link, and every referenced frame crosses it once per chunk that needs it: once, unless a chunk boundary falls
// inside its regions (only at the prediction-block edges, every kPredSuper regions).  However many regions a frame has, they
// stay in its chunk; the call splits them over several launches on the staged copy.
// The price of never staging an unreferenced frame: with regions on every other frame each referenced frame is a chunk of
// its own (one copy, one event hand-off and its own launches).  tools/regions_throughput.py measures that case beside the
// dense grid ("grid_every_other_frame", DESIGN.md section 5).
#pragma once
#include <algorithm>
#include <cstddef>
#include <cstdint>
#include <vector>

namespace cnnacc {

constexpr int kRegionMinSide = 128, kRegionMaxSide = 8192;
constexpr size_t kRegionChunkBytes = (size_t)16 << 20;     // frames staged per chunk, as the centre-crop path always did

// nullptr when regions [n][4] = (frame, x, y, side) are valid for n_frames frames of fh x fw, else why not; *bad = the index
// of the first offending region.
inline const char* region_error(const int32_t* rg, int64_t n, int64_t n_frames, int fh, int fw, int64_t* bad) {
    *bad = -1;
    for (int64_t r = 0; r < n; r++) {
        const int64_t f = rg[4 * r], x = rg[4 * r + 1], y = rg[4 * r + 2], s = rg[4 * r + 3];
        *bad = r;
        if (f < 0 || f >= n_frames) return "frame index outside [0, n_frames)";
        if (s < kRegionMinSide || s > kRegionMaxSide) return "side outside 128..8192";
        if (x < 0 || y < 0 || x + s > fw || y + s > fh) return "region outside its frame";
        if (r > 0 && f < rg[4 * (r - 1)]) return "frame indices decrease (group the regions by frame, in non-decreasing order)";
    }
    *bad = -1;
    return nullptr;
}

struct RegionChunk { int64_t f0, f1, r0, r1; };

// frame_of(r): the frame of region r, non-decreasing in r.  `super`: chunks never straddle a multiple of it (the call brings
// the predictions of up to `super` regions back in one block).
template <class FrameOf>
std::vector<RegionChunk> make_region_plan(FrameOf frame_of, int64_t n, size_t frame_bytes, int64_t super) {
    const int64_t per_chunk = frame_bytes >= kRegionChunkBytes ? 1 : (int64_t)(kRegionChunkBytes / frame_bytes);
    std::vector<RegionChunk> plan;
    for (int64_t r = 0; r < n;) {
        RegionChunk c;
        c.r0 = r;
        c.f0 = frame_of(r);
        int64_t last = c.f0;
        const int64_t end = std::min<int64_t>(n, (r / super + 1) * super);
        for (; r < end; r++) {
            const int64_t f = frame_of(r);
            if (f != last && (f != last + 1 || f - c.f0 >= per_chunk)) break;
            last = f;
        }
        c.r1 = r;
        c.f1 = last + 1;
        plan.push_back(c);
    }
    return plan;
}

}  // namespace cnnacc
