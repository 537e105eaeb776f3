// regions.cuh -- the pre-processing of preprocess.cuh on caller-chosen regions of BGR frames, many sizes in one launch.
//
// Region r is the rectangle frames[frame][y:y+h, x:x+w, :] with w and h 128..8192 (a square region is w == h); its output is
// exactly cv2.resize(cv2.cvtColor(rect, COLOR_BGR2GRAY), (128, 128), INTER_AREA): BGR2GRAY in OpenCV's 15-bit fixed point,
// then INTER_AREA on the path OpenCV picks from both scales w/128 and h/128 (resize.cpp):
//   * w and h both multiples of 128 (kx = w/128, ky = h/128): the integer box sum of kx x ky pixels, then
//       kx = ky = 1 : copy;   kx = ky = 2 : (sum + 2) >> 2;   otherwise : saturate_cast<uchar>(float(sum) * (1.f / (kx*ky)))
//   * otherwise: ResizeArea's float accumulation with x taps from computeResizeAreaTab(w) and y taps from
//     computeResizeAreaTab(h); an axis that is an integer multiple takes the table too (kx taps of (float)(1.0/kx)).
// For a square this is what the centre-crop path gives for the square cut out as a frame of its own.  The INTER_AREA taps are
// computed in the kernel from the sizes (area_taps, preprocess.cuh), so one launch mixes any sizes and nothing is uploaded
// per size.
//
// Work split as preprocess_bgr_kernel: one CTA of 128 threads per (output row, region), thread = output column.
#pragma once
#include "preprocess.cuh"
#include "region_plan.h"

namespace cnnacc {

struct RegionPrep {
    const uint8_t* frames;        // [..][fh][fw][3] BGR
    uint8_t* out;                 // [n][128][128]
    const int4* desc;             // [n] (frame, x, y, wh), frame relative to `frames` (wh: desc_w / desc_h, region_plan.h)
    int fh, fw;
};

__global__ void __launch_bounds__(kPrepOut)
preprocess_regions_kernel(const RegionPrep P)
{
    const int dx = threadIdx.x, dy = blockIdx.x;
    const int r = blockIdx.y;
    const int4 d = __ldg(P.desc + r);
    const int frame = d.x, x0 = d.y, y0 = d.z, W = desc_w(d.w), H = desc_h(d.w);
    const bool box = W % kPrepOut == 0 && H % kPrepOut == 0;
    const AreaTaps tx = area_taps(W, kPrepOut, dx, box), ty = area_taps(H, kPrepOut, dy, box);
    const uint8_t* src = P.frames + (size_t)frame * P.fh * P.fw * 3 + ((size_t)(y0 + ty.first) * P.fw + (x0 + tx.first)) * 3;
    const size_t pitch = (size_t)P.fw * 3;
    int v;
    if (!box) {
        float sum = 0.f;
        for (int j = 0; j < ty.n; j++) {
            const uint8_t* row = src + j * pitch;
            float buf = 0.f;
            for (int i = 0; i < tx.n; i++) buf = __fadd_rn(buf, __fmul_rn((float)bgr2gray(row + 3 * i), area_tap_weight(tx, i)));
            const float term = __fmul_rn(area_tap_weight(ty, j), buf);
            sum = j == 0 ? term : __fadd_rn(sum, term);
        }
        v = min(max(__float2int_rn(sum), 0), 255);
    } else {
        const int kx = W / kPrepOut, ky = H / kPrepOut;
        int tot = 0;
        for (int j = 0; j < ky; j++) {
            const uint8_t* row = src + j * pitch;
            for (int i = 0; i < kx; i++) tot += bgr2gray(row + 3 * i);
        }
        if (kx * ky == 1)           v = tot;
        else if (kx == 2 && ky == 2) v = (tot + 2) >> 2;
        else                         v = min(max(__float2int_rn(__fmul_rn((float)tot, 1.f / (float)(kx * ky))), 0), 255);
    }
    P.out[((size_t)r * kPrepOut + dy) * kPrepOut + dx] = (uint8_t)v;
}

}  // namespace cnnacc
