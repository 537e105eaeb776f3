// region_plan.h -- checks of a region array and the staging plan of a host-pointer region call (cnnacc_detect_regions /
// cnnacc_preprocess_regions; cnnacc_detect_frames / cnnacc_preprocess_bgr are the case of one centre region per frame).  Host
// arithmetic, plus the decoders of the descriptor's size field that the kernels share; tests/test_regions_cpu.py and tests/test_rect_regions_cpu.py replay it through
// cnnacc_region_plan_host and cnnacc_rect_plan_host.
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

#if defined(__CUDACC__)
#define CNNACC_REGION_HD __host__ __device__ __forceinline__
#else
#define CNNACC_REGION_HD inline
#endif

// The caller's region records, the one place that knows their two formats: [n][4] squares (frame, x, y, side), or with
// CNNACC_FLAG_RECTS [n][5] rectangles (frame, x, y, w, h).  A square is the rectangle w = h = side, so everything past this
// reads (frame, x, y, w, h).  The device descriptor of every region is the int4 (frame, x, y, wh) with wh = w | h << 16
// (w, h <= 8192 fit 14 bits), where h = 0 stands for h = w: a square's record is its descriptor as it is, so square calls
// copy their records as before instead of re-packing them.
CNNACC_REGION_HD int desc_w(int wh) { return wh & 0xffff; }
CNNACC_REGION_HD int desc_h(int wh) { return (wh >> 16) ? (wh >> 16) : (wh & 0xffff); }

struct RegionRecords {
    const int32_t* p;
    int stride;                                            // 4 (squares) or 5 (rectangles)
    RegionRecords(const int32_t* p_, bool rects) : p(p_), stride(rects ? 5 : 4) {}
    int64_t frame(int64_t r) const { return p[stride * r]; }
    int32_t x(int64_t r) const { return p[stride * r + 1]; }
    int32_t y(int64_t r) const { return p[stride * r + 2]; }
    int32_t w(int64_t r) const { return p[stride * r + 3]; }
    int32_t h(int64_t r) const { return p[stride * r + stride - 1]; }
    int32_t wh(int64_t r) const { return stride == 4 ? w(r) : w(r) | h(r) << 16; }   // the descriptor's, for checked records
};

// nullptr when the regions' frame, position and sizes are valid for n_frames frames and, when `sized` (the merging calls have
// no frame size), they lie inside frames of fh x fw (in int64: x + w cannot wrap), else why not; *bad = the index of the
// first offending region.
inline const char* region_error(const RegionRecords& rg, int64_t n, int64_t n_frames, bool sized, int fh, int fw, int64_t* bad) {
    *bad = -1;
    for (int64_t r = 0; r < n; r++) {
        const int64_t f = rg.frame(r), x = rg.x(r), y = rg.y(r), w = rg.w(r), h = rg.h(r);
        *bad = r;
        if (f < 0 || f >= n_frames) return "frame index outside [0, n_frames)";
        if (w < kRegionMinSide || w > kRegionMaxSide || h < kRegionMinSide || h > kRegionMaxSide)
            return rg.stride == 4 ? "side outside 128..8192" : "width or height outside 128..8192";
        if (x < 0 || y < 0) return sized ? "region outside its frame" : "negative position";
        if (sized && (x + w > fw || y + h > fh)) return "region outside its frame";
        if (r > 0 && f < rg.frame(r - 1)) return "frame indices decrease (group the regions by frame, in non-decreasing order)";
    }
    *bad = -1;
    return nullptr;
}

struct RegionChunk { int64_t f0, f1, r0, r1; };

// frame_of(r): the frame of region r, non-decreasing in r.  block_end(r) > r: the end of the prediction block that holds
// region r; chunks never straddle a block edge (the call brings the predictions of a block back, or merges them, at once).
template <class FrameOf, class BlockEnd>
std::vector<RegionChunk> make_region_plan_blocks(FrameOf frame_of, int64_t n, size_t frame_bytes, BlockEnd block_end) {
    const int64_t per_chunk = frame_bytes >= kRegionChunkBytes ? 1 : (int64_t)(kRegionChunkBytes / frame_bytes);
    std::vector<RegionChunk> plan;
    for (int64_t r = 0; r < n;) {
        RegionChunk c;
        c.r0 = r;
        c.f0 = frame_of(r);
        int64_t last = c.f0;
        const int64_t end = std::min<int64_t>(n, block_end(r));
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

// The plan of cnnacc_detect_regions / cnnacc_detect_frames: prediction blocks of `super` regions each.
template <class FrameOf>
std::vector<RegionChunk> make_region_plan(FrameOf frame_of, int64_t n, size_t frame_bytes, int64_t super) {
    return make_region_plan_blocks(frame_of, n, frame_bytes, [super](int64_t r) { return (r / super + 1) * super; });
}

// Prediction blocks of at most `super` regions that end at frame edges (cnnacc_detect_objects merges a block once all of its
// frames are predicted): bounds[0] = 0 < bounds[1] < ... = n.  Always possible while a frame has fewer than `super` regions.
template <class FrameOf>
std::vector<int64_t> frame_aligned_blocks(FrameOf frame_of, int64_t n, int64_t super) {
    std::vector<int64_t> bounds{0};
    while (bounds.back() < n) {
        const int64_t b0 = bounds.back();
        int64_t e = b0 + super;
        if (e >= n) {
            e = n;
        } else {
            while (e > b0 && frame_of(e) == frame_of(e - 1)) e--;   // back to the first region of the frame that holds e
            if (e == b0) e = b0 + super;                          // a frame of super regions or more: cut inside it
        }
        bounds.push_back(e);
    }
    return bounds;
}

}  // namespace cnnacc
