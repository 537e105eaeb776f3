// pil_resize.cuh -- the image-loading step of pynq_inference.py on the GPU: load_image_any
// (/root/reference/software/pynq_inference.py:414-425) for a decoded image,
//     Image.open(path).convert('L').resize((128, 128))  ->  (128,128) u8.
//
// Third-party arithmetic, restated from Pillow's sources and pinned against Pillow 12.2.0 through tests/golden/pil_cases.npz
// (made by running the reference's own load_image_any on PNG files, tests/golden/make_pil_golden.py):
//   * convert('L') of RGB / RGBA (src/libImaging/Convert.c rgb2l): L = (R*19595 + G*38470 + B*7471 + 0x8000) >> 16;
//   * resize() of a mode "L" image defaults to BICUBIC (a = -0.5, support 2); when shrinking, the support and the filter
//     argument scale with the ratio (antialiasing).  8-bit images are resampled in integers (src/libImaging/Resample.c):
//     per output index a window [xmin, xmin + xmax) and coefficients normalised in double precision, rounded to 22
//     fractional bits; out = clip8((2^21 + sum in * k) >> 22); one pass rounded to u8, then the other; a pass is skipped
//     when that side is already 128;
//   * pass order (PIL/Image.py Image.resize): horizontal first, except that an image more than 100 times taller than wide
//     (H > 100 W, H > 128) is first resized to (W, 128) and then to (128, 128), i.e. the vertical pass runs first.
// The coefficient tables depend on the input size, so they are built on the host exactly as precompute_coeffs /
// normalize_coeffs_8bpc do and cached per (H, W) in the handle.
#pragma once
#include <cmath>
#include <vector>
#include "common.cuh"

namespace cnnacc {

constexpr int kPilOut = 128, kPilCoefBits = 22;

struct PilTabHost {
    int ksize = 0;
    std::vector<int32_t> k;          // [128][ksize]
    std::vector<int32_t> bounds;     // [128][2]: xmin, count
};

inline double pil_bicubic(double x) {
    const double a = -0.5;
    if (x < 0.0) x = -x;
    if (x < 1.0) return ((a + 2.0) * x - (a + 3.0)) * x * x + 1;
    if (x < 2.0) return (((x - 5) * x + 8) * x - 4) * a;
    return 0.0;
}

// Pillow: precompute_coeffs(inSize, 0, inSize, 128, BICUBIC) + normalize_coeffs_8bpc
inline PilTabHost make_pil_tab(int in_size) {
    PilTabHost t;
    const double scale = (double)in_size / kPilOut;
    const double filterscale = scale < 1.0 ? 1.0 : scale;
    const double support = 2.0 * filterscale;
    t.ksize = (int)std::ceil(support) * 2 + 1;
    t.k.assign((size_t)kPilOut * t.ksize, 0);
    t.bounds.assign(2 * kPilOut, 0);
    std::vector<double> w(t.ksize);
    for (int xx = 0; xx < kPilOut; xx++) {
        const double center = (xx + 0.5) * scale, ss = 1.0 / filterscale;
        int xmin = (int)(center - support + 0.5);
        if (xmin < 0) xmin = 0;
        int xmax = (int)(center + support + 0.5);
        if (xmax > in_size) xmax = in_size;
        xmax -= xmin;
        double ww = 0.0;
        for (int x = 0; x < xmax; x++) { w[x] = pil_bicubic((x + xmin - center + 0.5) * ss); ww += w[x]; }
        for (int x = 0; x < xmax; x++)
            if (ww != 0.0) w[x] /= ww;
        for (int x = xmax; x < t.ksize; x++) w[x] = 0.0;
        for (int x = 0; x < t.ksize; x++)
            t.k[(size_t)xx * t.ksize + x] = w[x] < 0 ? (int)(-0.5 + w[x] * (1 << kPilCoefBits)) : (int)(0.5 + w[x] * (1 << kPilCoefBits));
        t.bounds[2 * xx] = xmin; t.bounds[2 * xx + 1] = xmax;
    }
    return t;
}

__device__ __forceinline__ uint32_t pil_gray(const uint8_t* px, int C) {
    if (C == 1) return px[0];
    return (px[0] * 19595u + px[1] * 38470u + px[2] * 7471u + 0x8000u) >> 16;
}
__device__ __forceinline__ uint8_t pil_clip8_acc(int acc) { return (uint8_t)min(max(acc >> kPilCoefBits, 0), 255); }

// Horizontal pass (and the gray conversion): one CTA per (row, image), thread = output column.  in [n][H][W][C] -> tmp [n][H][128].
// With `copy` (W == 128) it only converts.
__global__ void __launch_bounds__(kPilOut)
pil_horizontal_kernel(const uint8_t* __restrict__ in, uint8_t* __restrict__ tmp, const int32_t* __restrict__ k,
                      const int32_t* __restrict__ bounds, int ksize, int H, int W, int C, int copy)
{
    const int xx = threadIdx.x, row = blockIdx.x;
    const size_t img = blockIdx.y;
    const uint8_t* src = in + ((img * H + row) * (size_t)W) * C;
    uint8_t* dst = tmp + (img * H + row) * kPilOut;
    if (copy) { dst[xx] = (uint8_t)pil_gray(src + (size_t)xx * C, C); return; }
    const int xmin = bounds[2 * xx], cnt = bounds[2 * xx + 1];
    const int32_t* kk = k + (size_t)xx * ksize;
    int acc = 1 << (kPilCoefBits - 1);
    for (int x = 0; x < cnt; x++) acc += (int)pil_gray(src + (size_t)(xmin + x) * C, C) * kk[x];
    dst[xx] = pil_clip8_acc(acc);
}

// Vertical pass (and the gray conversion): one CTA per (output row, image), thread = column, looping over the W columns.
// in [n][H][W][C] -> out [n][128][W].  Horizontal-first runs it on the [n][H][128] u8 result of the horizontal pass (W = 128,
// C = 1); vertical-first on the source image, and the horizontal pass then reads its [n][128][W] output (H = 128, C = 1).
__global__ void __launch_bounds__(kPilOut)
pil_vertical_kernel(const uint8_t* __restrict__ in, uint8_t* __restrict__ out, const int32_t* __restrict__ k,
                    const int32_t* __restrict__ bounds, int ksize, int H, int W, int C)
{
    const int yy = blockIdx.x;
    const size_t img = blockIdx.y;
    const int ymin = bounds[2 * yy], cnt = bounds[2 * yy + 1];
    const int32_t* kk = k + (size_t)yy * ksize;
    const size_t row = (size_t)W * C;
    for (int x = threadIdx.x; x < W; x += blockDim.x) {
        const uint8_t* src = in + (img * H + ymin) * row + (size_t)x * C;
        int acc = 1 << (kPilCoefBits - 1);
        for (int y = 0; y < cnt; y++) acc += (int)pil_gray(src + (size_t)y * row, C) * kk[y];
        out[(img * kPilOut + yy) * W + x] = pil_clip8_acc(acc);
    }
}

}  // namespace cnnacc
