// region_merge.h -- the merge rule of cnnacc_detect_objects / cnnacc_merge_regions, written once for the kernel
// (region_merge.cuh) and the CPU replay (merge_frame_host, cnnacc_merge_regions_host).
//
// Per frame, independently: clamp every box coordinate to [0, 127]; map it to the frame exactly, in 1/128 pixel as int64
// (X = 128 x + bx w, Y = 128 y + by h for the region (x, y, w, h); w = h = side for a square); candidates are the regions with score >= score_min (never a NaN score); order them by score
// descending, then region index ascending (-0.0 and +0.0 are equal); walk them in that order and keep a candidate unless an
// already-kept box of the same class (any class with CNNACC_FLAG_CLASS_AGNOSTIC) has IoU > iou_max with it; stop at max_det.
// IoU = (double)inter / (double)union from exact int64 areas (0 when union == 0).  With w, h <= 8192 a box spans at most
// 127 * 8192 < 2^20 units a side, so inter and union are below 2^40, both exact doubles: one IEEE division gives the same
// bits on the device and on the host (the build has no fast-math).
#pragma once
#include <algorithm>
#include <cstdint>
#include <cstring>
#include <vector>
#include "region_plan.h"

#if defined(__CUDACC__)
#define CNNACC_MERGE_HD __host__ __device__ __forceinline__
#else
#define CNNACC_MERGE_HD inline
#endif

namespace cnnacc {

constexpr int kMergeMaxDet = 1024;          // CNNACC_MERGE_MAX_DET
constexpr int kMergeMaxPerFrame = 16384;    // CNNACC_MERGE_MAX_PER_FRAME

// a box in 1/128 frame pixels
struct MergeBox { long long x1, y1, x2, y2; };

CNNACC_MERGE_HD int merge_clamp(int v) { return v < 0 ? 0 : (v > 127 ? 127 : v); }

// box (x1, y1, x2, y2) on the 128 grid of the region (x, y, w, h), clamped, in 1/128 frame pixels
CNNACC_MERGE_HD MergeBox merge_box(int x, int y, int w, int h, int bx1, int by1, int bx2, int by2) {
    MergeBox m;
    m.x1 = 128LL * x + (long long)merge_clamp(bx1) * w;
    m.y1 = 128LL * y + (long long)merge_clamp(by1) * h;
    m.x2 = 128LL * x + (long long)merge_clamp(bx2) * w;
    m.y2 = 128LL * y + (long long)merge_clamp(by2) * h;
    return m;
}

CNNACC_MERGE_HD long long merge_area(const MergeBox& b) {
    const long long w = b.x2 - b.x1, h = b.y2 - b.y1;
    return (w > 0 ? w : 0) * (h > 0 ? h : 0);
}

// a NaN score is never a candidate
CNNACC_MERGE_HD bool merge_candidate(float score, float score_min) { return score >= score_min; }

CNNACC_MERGE_HD uint32_t merge_float_bits(float f) {
#if defined(__CUDA_ARCH__)
    return __float_as_uint(f);
#else
    uint32_t u;
    std::memcpy(&u, &f, sizeof(u));
    return u;
#endif
}

// Sort key of a candidate: ascending keys are descending scores, ties by ascending index (the region's index within its frame).
CNNACC_MERGE_HD unsigned long long merge_key(float score, uint32_t idx) {
    if (score == 0.f) score = 0.f;                                    // -0.0 -> +0.0
    const uint32_t u = merge_float_bits(score);
    const uint32_t ord = (u & 0x80000000u) ? ~u : (u | 0x80000000u);  // ascending with the score
    return ((unsigned long long)(~ord) << 32) | idx;
}
CNNACC_MERGE_HD uint32_t merge_key_index(unsigned long long key) { return (uint32_t)(key & 0xffffffffu); }

// Does a kept box `a` suppress the candidate `b`: IoU(a, b) > iou_max?
CNNACC_MERGE_HD bool merge_suppresses(const MergeBox& a, long long area_a, const MergeBox& b, long long area_b, double iou_max) {
    const long long iw = (a.x2 < b.x2 ? a.x2 : b.x2) - (a.x1 > b.x1 ? a.x1 : b.x1);
    const long long ih = (a.y2 < b.y2 ? a.y2 : b.y2) - (a.y1 > b.y1 ? a.y1 : b.y1);
    const long long inter = (iw > 0 ? iw : 0) * (ih > 0 ? ih : 0);
    const long long uni = area_a + area_b - inter;
    const double iou = uni == 0 ? 0.0 : (double)inter / (double)uni;
    return iou > iou_max;
}

// A box coordinate in frame pixels: the correctly rounded float of X / 128.
CNNACC_MERGE_HD float merge_px(long long X) { return (float)((double)X / 128.0); }

// nullptr when the merge's own arguments are valid, else why not
inline const char* merge_limits_error(float iou_max, int max_det) {
    if (max_det < 1 || max_det > kMergeMaxDet) return "max_det outside 1..1024";
    if (!(iou_max >= 0.f && iou_max <= 1.f)) return "iou_max NaN or outside [0, 1]";
    return nullptr;
}

// first[f] .. first[f + 1] = the regions of frame f (n_frames + 1 entries) from frame indices that do not decrease; nullptr, or
// why not when a frame has more than kMergeMaxPerFrame regions (*bad = that frame).  *max_count = the most regions of a frame.
template <class FrameOf>
const char* merge_frame_ranges(FrameOf frame_of, int64_t n, int64_t n_frames, std::vector<int64_t>& first, int64_t* max_count,
                               int64_t* bad) {
    first.assign((size_t)n_frames + 1, n);
    *max_count = 0;
    *bad = -1;
    int64_t r = 0;
    for (int64_t f = 0; f < n_frames; f++) {
        first[f] = r;
        while (r < n && frame_of(r) == f) r++;
        *max_count = std::max(*max_count, r - first[f]);
        if (r - first[f] > kMergeMaxPerFrame) {
            *bad = f;
            return "more than 16384 regions in one frame";
        }
    }
    return nullptr;
}

// The merge rule on the CPU for one frame: regions r0 .. r0 + cnt - 1 of `rg`, score[r], cls[r], bbox[r][4].  Outputs hold
// max_det rows; returns n_det.
inline int merge_frame_host(const RegionRecords& rg, const float* score, const int32_t* cls, const int32_t* bbox, int64_t r0,
                            int64_t cnt, float score_min, float iou_max, int max_det, bool agnostic, int32_t* det_region,
                            int32_t* det_cls, float* det_score, float* det_box) {
    std::vector<unsigned long long> keys;
    for (int64_t i = 0; i < cnt; i++)
        if (merge_candidate(score[r0 + i], score_min)) keys.push_back(merge_key(score[r0 + i], (uint32_t)i));
    std::sort(keys.begin(), keys.end());
    std::vector<MergeBox> kept;
    std::vector<long long> kept_area;
    std::vector<int> kept_cls;
    std::vector<int64_t> kept_r;
    for (unsigned long long k : keys) {
        if ((int)kept.size() >= max_det) break;
        const int64_t r = r0 + merge_key_index(k);
        const int32_t* b = bbox + 4 * r;
        const MergeBox m = merge_box(rg.x(r), rg.y(r), rg.w(r), rg.h(r), b[0], b[1], b[2], b[3]);
        const long long area = merge_area(m);
        bool sup = false;
        for (size_t j = 0; j < kept.size() && !sup; j++)
            sup = (agnostic || kept_cls[j] == cls[r]) && merge_suppresses(kept[j], kept_area[j], m, area, (double)iou_max);
        if (sup) continue;
        kept.push_back(m); kept_area.push_back(area); kept_cls.push_back(cls[r]); kept_r.push_back(r);
    }
    for (int k = 0; k < max_det; k++) {
        const bool on = k < (int)kept.size();
        if (det_region) det_region[k] = on ? (int32_t)kept_r[k] : -1;
        if (det_cls) det_cls[k] = on ? kept_cls[k] : -1;
        if (det_score) det_score[k] = on ? score[kept_r[k]] : 0.f;
        if (det_box) {
            det_box[4 * k + 0] = on ? merge_px(kept[k].x1) : 0.f;
            det_box[4 * k + 1] = on ? merge_px(kept[k].y1) : 0.f;
            det_box[4 * k + 2] = on ? merge_px(kept[k].x2) : 0.f;
            det_box[4 * k + 3] = on ? merge_px(kept[k].y2) : 0.f;
        }
    }
    return (int)kept.size();
}

}  // namespace cnnacc
