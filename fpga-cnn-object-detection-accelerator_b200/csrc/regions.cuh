// regions.cuh -- the pre-processing of preprocess.cuh on caller-chosen square regions of BGR frames, many sides in one launch.
//
// Region r is the square frames[frame][y:y+side, x:x+side, :] with side 128..8192; its output is exactly what the centre-crop
// path gives for that square cut out as a frame of its own (a square is its own centre crop): BGR2GRAY in OpenCV's 15-bit
// fixed point, then INTER_AREA to 128x128 on whichever of the four paths the side selects (copy, 2x2, k x k, fractional).
// The INTER_AREA taps are computed in the kernel from the side (area_taps, preprocess.cuh), so one launch mixes any sides and
// nothing is uploaded per side.
//
// Work split as preprocess_bgr_kernel: one CTA of 128 threads per (output row, region), thread = output column.
#pragma once
#include "preprocess.cuh"

namespace cnnacc {

struct RegionPrep {
    const uint8_t* frames;        // [..][fh][fw][3] BGR
    uint8_t* out;                 // [n][128][128]
    const int4* desc;             // [n] (frame, x, y, side), frame relative to `frames`
    int fh, fw;
};

__global__ void __launch_bounds__(kPrepOut)
preprocess_regions_kernel(const RegionPrep P)
{
    const int dx = threadIdx.x, dy = blockIdx.x;
    const int r = blockIdx.y;
    const int4 d = __ldg(P.desc + r);
    const int frame = d.x, x0 = d.y, y0 = d.z, S = d.w;
    const AreaTaps tx = area_taps(S, dx), ty = area_taps(S, dy);
    const uint8_t* src = P.frames + (size_t)frame * P.fh * P.fw * 3 + ((size_t)(y0 + ty.first) * P.fw + (x0 + tx.first)) * 3;
    const size_t pitch = (size_t)P.fw * 3;
    int v;
    if (S % kPrepOut != 0) {
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
        const int k = S / kPrepOut;
        int tot = 0;
        for (int j = 0; j < k; j++) {
            const uint8_t* row = src + j * pitch;
            for (int i = 0; i < k; i++) tot += bgr2gray(row + 3 * i);
        }
        if (k == 1)      v = tot;
        else if (k == 2) v = (tot + 2) >> 2;
        else             v = min(max(__float2int_rn(__fmul_rn((float)tot, 1.f / (float)(k * k))), 0), 255);
    }
    P.out[((size_t)r * kPrepOut + dy) * kPrepOut + dx] = (uint8_t)v;
}

}  // namespace cnnacc
