// pyramid.cuh -- the levels of an image pyramid from full-resolution gray frames (cnnacc_preprocess_pyramid /
// cnnacc_scan_pyramid / cnnacc_scan_pyramid_objects), every level of a piece of frames in one launch.
//
// Level l of frame f is exactly cv2.resize(gray[f], (w, h), interpolation=INTER_AREA) for a downscale of the fh x fw gray
// frame to w x h, on the path OpenCV picks from both scales fw/w and fh/h (resize.cpp), as regions.cuh does for D = 128:
//   * both scales integers by OpenCV's own test (area_fast_axis; kx = fw/w, ky = fh/h): the integer box sum of kx x ky
//     pixels, then
//       kx = ky = 1 : copy;   kx = ky = 2 : (sum + 2) >> 2;   otherwise : saturate_cast<uchar>(float(sum) * (1.f / (kx*ky)))
//   * otherwise: ResizeArea's float accumulation with x taps from computeResizeAreaTab(fw -> w) and y taps from
//     computeResizeAreaTab(fh -> h) (area_taps, preprocess.cuh); an integer axis takes the table too.
// The gray frames come from gray_full_kernel, so each source pixel is converted once per frame, not once per level.
//
// Work split: one CTA of 128 threads per (output row of any level, frame); a thread walks the row's columns 128 apart.
#pragma once
#include <cfloat>
#include <cmath>
#include "preprocess.cuh"

namespace cnnacc {

constexpr int kPyramidMaxLevels = 16;

// OpenCV's test for the integer (ResizeAreaFast) path on one axis of a downscale S -> D (resize.cpp): scale = 1 / (D / S)
// in double lies within DBL_EPSILON of an integer.  That is S % D == 0, except for S = 49 D: 1.0 / (1.0 / 49) is not 49 in
// double, so OpenCV resizes a 49x axis with the table (49 taps of (float)(1.0 / 49)).  A level takes the integer path when
// both axes pass.
inline bool area_fast_axis(int S, int D) {
    const double scale = 1.0 / ((double)D / S);
    return std::fabs(scale - std::rint(scale)) < DBL_EPSILON;
}

struct PyramidLevel {
    int w, h, row0;               // level size; its first row among the launch's rows
    int box;                      // both axes take the integer path (area_fast_axis)
    size_t off, fstride;          // level l of frame f is written at out + off + f * fstride, [h][w]
};

struct PyramidPrep {
    const uint8_t* gray;          // [n][fh][fw]
    uint8_t* out;
    int fh, fw, n_levels;
    PyramidLevel lv[kPyramidMaxLevels];
};

__global__ void __launch_bounds__(kPrepOut)
pyramid_levels_kernel(const __grid_constant__ PyramidPrep P)
{
    int l = 0;
    while (l + 1 < P.n_levels && (int)blockIdx.x >= P.lv[l + 1].row0) l++;
    const PyramidLevel& L = P.lv[l];
    const int dy = blockIdx.x - L.row0, f = blockIdx.y;
    const bool box = L.box != 0;
    const AreaTaps ty = area_taps(P.fh, L.h, dy, box);
    const uint8_t* frame = P.gray + (size_t)f * P.fh * P.fw + (size_t)ty.first * P.fw;
    uint8_t* out = P.out + L.off + (size_t)f * L.fstride + (size_t)dy * L.w;
    for (int dx = threadIdx.x; dx < L.w; dx += kPrepOut) {
        const AreaTaps tx = area_taps(P.fw, L.w, dx, box);
        const uint8_t* src = frame + tx.first;
        int v;
        if (!box) {
            float sum = 0.f;
            for (int j = 0; j < ty.n; j++) {
                const uint8_t* row = src + (size_t)j * P.fw;
                float buf = 0.f;
                for (int i = 0; i < tx.n; i++) buf = __fadd_rn(buf, __fmul_rn((float)__ldg(row + i), area_tap_weight(tx, i)));
                const float term = __fmul_rn(area_tap_weight(ty, j), buf);
                sum = j == 0 ? term : __fadd_rn(sum, term);
            }
            v = min(max(__float2int_rn(sum), 0), 255);
        } else {
            const int kx = tx.n, ky = ty.n;
            int tot = 0;
            for (int j = 0; j < ky; j++) {
                const uint8_t* row = src + (size_t)j * P.fw;
                for (int i = 0; i < kx; i++) tot += __ldg(row + i);
            }
            if (kx * ky == 1)            v = tot;
            else if (kx == 2 && ky == 2) v = (tot + 2) >> 2;
            else                         v = min(max(__float2int_rn(__fmul_rn((float)tot, 1.f / (float)(kx * ky))), 0), 255);
        }
        out[dx] = (uint8_t)v;
    }
}

}  // namespace cnnacc
