// region_merge.cuh -- per-frame greedy NMS of region detections (the rule of region_merge.h) on the GPU.
//
// One CTA per frame.  The frame's regions are first[f] .. first[f+1]-1 (computed on the host from the host region array; the
// descriptors' frame fields are not read, since host-pointer calls store them relative to a staging buffer).  The CTA loads
// every candidate as a 64-bit key (orderable score, index in the frame) into shared memory, bitonic-sorts the keys, and walks
// them in order against the kept list in shared memory: each thread tests its share of the kept boxes, one barrier vote
// decides.  The boxes of the next kMergeThreads candidates are mapped to frame coordinates in parallel before the walk reaches
// them, so the serial part reads shared memory only.
#pragma once
#include "common.cuh"
#include "region_merge.h"

namespace cnnacc {

constexpr int kMergeThreads = 256;

struct MergeArgs {
    const int4* desc;               // [r] (frame, x, y, wh) as in regions.cuh, indexed by region r of the call
    const long long* first;         // [F + 1] region ranges of this launch's F frames (absolute region indices)
    long long r_pred0;              // region index of element 0 of score / cls / bbox
    const float* score;             // score of region r: score[(r - r_pred0) * score_stride + (score_by_cls ? cls : 0)]
    int score_stride, score_by_cls;
    const int32_t* cls;             // [r - r_pred0]
    const int32_t* bbox;            // [r - r_pred0][4] (x1, y1, x2, y2) on the region's 128 grid (4-byte aligned)
    float score_min, iou_max;
    int max_det, agnostic;
    int key_cap;                    // power of two >= the largest per-frame region count of the launch
    int kept_cap;                   // min(max_det, key_cap)
    int32_t* n_det;                 // [F]; the others [F][max_det](x4), any may be null but n_det
    int32_t* det_region;
    int32_t* det_cls;
    float* det_score;
    float4* det_box;
};

struct MergeCand { MergeBox b; long long area; int cls, idx; };

inline size_t merge_smem_bytes(int key_cap, int kept_cap) {
    return (size_t)key_cap * 8 + (size_t)(kMergeThreads + kept_cap) * sizeof(MergeCand);
}

__device__ __forceinline__ float merge_score_of(const MergeArgs& A, long long r) {
    const long long u = r - A.r_pred0;
    return A.score[u * A.score_stride + (A.score_by_cls ? A.cls[u] : 0)];
}

__global__ void __launch_bounds__(kMergeThreads)
merge_regions_kernel(const MergeArgs A)
{
    extern __shared__ __align__(16) unsigned char merge_smem[];
    unsigned long long* key = reinterpret_cast<unsigned long long*>(merge_smem);
    MergeCand* cand = reinterpret_cast<MergeCand*>(key + A.key_cap);   // [kMergeThreads]: the next candidates, mapped
    MergeCand* kept = cand + kMergeThreads;                             // [kept_cap]
    __shared__ int s_ncand;
    const int tid = threadIdx.x, f = blockIdx.x;
    const long long r0 = A.first[f];
    const int cnt = (int)(A.first[f + 1] - r0);
    int n2 = 1;
    while (n2 < cnt) n2 <<= 1;
    if (tid == 0) s_ncand = 0;
    for (int i = tid; i < n2; i += kMergeThreads) {
        unsigned long long k = ~0ull;
        if (i < cnt) {
            const float s = merge_score_of(A, r0 + i);
            if (merge_candidate(s, A.score_min)) k = merge_key(s, (uint32_t)i);
        }
        key[i] = k;
    }
    __syncthreads();
    for (int k = 2; k <= n2; k <<= 1) {                 // bitonic sort, ascending
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = tid; i < n2; i += kMergeThreads) {
                const int p = i ^ j;
                if (p > i) {
                    const unsigned long long a = key[i], b = key[p];
                    if ((a > b) == ((i & k) == 0)) { key[i] = b; key[p] = a; }
                }
            }
            __syncthreads();
        }
    }
    for (int i = tid; i < n2; i += kMergeThreads)       // candidates are the keys before the first ~0
        if (key[i] != ~0ull && (i + 1 == n2 || key[i + 1] == ~0ull)) s_ncand = i + 1;
    __syncthreads();
    const int ncand = s_ncand;
    const double iou_max = (double)A.iou_max;
    int n_kept = 0;
    for (int c0 = 0; c0 < ncand && n_kept < A.max_det; c0 += kMergeThreads) {
        if (c0 + tid < ncand) {
            const int idx = (int)merge_key_index(key[c0 + tid]);
            const long long r = r0 + idx;
            const int4 d = __ldg(A.desc + r);
            const int32_t* b = A.bbox + 4 * (r - A.r_pred0);
            MergeCand m;
            m.b = merge_box(d.y, d.z, desc_w(d.w), desc_h(d.w), __ldg(b), __ldg(b + 1), __ldg(b + 2), __ldg(b + 3));
            m.area = merge_area(m.b);
            m.cls = __ldg(A.cls + (r - A.r_pred0));
            m.idx = idx;
            cand[tid] = m;
        }
        __syncthreads();
        const int c1 = min(ncand, c0 + kMergeThreads);
        for (int c = c0; c < c1 && n_kept < A.max_det; c++) {
            const MergeCand& m = cand[c - c0];
            bool sup = false;
            for (int j = tid; j < n_kept && !sup; j += kMergeThreads)
                sup = (A.agnostic || kept[j].cls == m.cls) && merge_suppresses(kept[j].b, kept[j].area, m.b, m.area, iou_max);
            if (!__syncthreads_or(sup)) {
                if (tid == 0) kept[n_kept] = m;
                n_kept++;
                __syncthreads();
            }
        }
        __syncthreads();                                 // cand[] is refilled next
    }
    const size_t row = (size_t)f * A.max_det;
    if (tid == 0) A.n_det[f] = n_kept;
    for (int k = tid; k < A.max_det; k += kMergeThreads) {
        const bool on = k < n_kept;
        const long long r = on ? r0 + kept[k].idx : -1;
        if (A.det_region) A.det_region[row + k] = on ? (int32_t)r : -1;
        if (A.det_cls) A.det_cls[row + k] = on ? kept[k].cls : -1;
        if (A.det_score) A.det_score[row + k] = on ? merge_score_of(A, r) : 0.f;
        if (A.det_box)
            A.det_box[row + k] = on ? make_float4(merge_px(kept[k].b.x1), merge_px(kept[k].b.y1), merge_px(kept[k].b.x2),
                                                  merge_px(kept[k].b.y2))
                                    : make_float4(0.f, 0.f, 0.f, 0.f);
    }
}

}  // namespace cnnacc
