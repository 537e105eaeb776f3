// preprocess.cuh -- the step in front of the hot path in the real-time loop
// (/root/reference/software/realtime_detect.py:582-591), batched and fused into one kernel:
//
//     centre-crop the (h,w,3) BGR frame to a square of side S = min(h,w)
//  -> cv2.cvtColor(COLOR_BGR2GRAY)      gray = (3735 B + 19235 G + 9798 R + 2^14) >> 15   (OpenCV's 15-bit fixed point)
//  -> cv2.resize((128,128), INTER_AREA)
//
// OpenCV's INTER_AREA has three arithmetic paths, all reproduced bit for bit (pinned against cv2 4.13.0,
// tests/golden/prep_cases.npz):
//   * S == 128           : copy
//   * S == 256           : ResizeAreaFastVec, (a + b + c + d + 2) >> 2
//   * S == 128 k, k >= 3 : ResizeAreaFast, saturate_cast<uchar>(float(box sum) * (1.f / (k*k)))  (round half to even)
//   * otherwise          : ResizeArea, float accumulation: per source row buf = sum_k S[sx_k] * alpha_k (left to right),
//                          then out = beta_0 * buf_0 + beta_1 * buf_1 + ... (top to bottom), every product and sum rounded
//                          to fp32 on its own (no FMA), weights from computeResizeAreaTab in double -> float.
// The weight table (same for x and y: the crop is square) is built on the host by make_area_tab below.
//
// Work split: one CTA of 128 threads per (output row, frame); thread = output column.  A VGA frame is 900 KiB in and
// 16 KiB out, so the kernel is bound by HBM reads of the frames (and, end to end, by PCIe bringing them in).
#pragma once
#include <cmath>
#include <vector>
#include "common.cuh"

namespace cnnacc {

constexpr int kPrepOut = 128, kPrepRowsPerCta = 1, kPrepMaxSide = 8192;

enum PrepMode : int { kPrepCopy = 0, kPrepBox2 = 1, kPrepBoxK = 2, kPrepFrac = 3 };

struct AreaTabHost {
    int mode = kPrepCopy, k = 1, taps = 1;     // taps = table row length
    float inv = 1.f;                           // 1.f / (k*k) for kPrepBoxK
    std::vector<int> start, cnt;               // [128] first source index and number of taps per output index
    std::vector<float> alpha;                  // [128][taps]
};

// The INTER_AREA taps of output index d for a square side S (128..8192): OpenCV's computeResizeAreaTab(ssize = S, dsize = 128,
// scale = S/128.) for one d, in its order (double arithmetic, then float).  The taps are the consecutive source indices
// first .. first+n-1; tap i weighs area_tap_weight(t, i).  Integer scales (S = 128 k) give k taps of weight 1 (their kernels
// sum integers instead).  Host (make_area_tab, cnnacc_area_tab_host) and device (regions.cuh) get the same bits: scale = S/128
// is exact, so are d * scale, fsx1 + scale and S - fsx1 for S <= 8192 (at most 20 significant bits) -- an FMA the compiler
// forms from them rounds nothing -- ceil / floor / min are exact, and the three divisions are correctly rounded in IEEE double
// on both sides.  Up to 65 taps per output at S = 8191: the weights stay three scalars (first partial, 1/cell, last partial)
// instead of a table in registers.
struct AreaTaps {
    int first, n;
    bool head, tail;                 // tap 0 / tap n-1 is a partial cell
    float a_head, a_mid, a_tail;
};

__host__ __device__ __forceinline__ AreaTaps area_taps(int S, int d) {
    AreaTaps t;
    if (S % kPrepOut == 0) {
        const int k = S / kPrepOut;
        t.first = d * k; t.n = k; t.head = t.tail = false; t.a_head = t.a_mid = t.a_tail = 1.f;
        return t;
    }
    const double scale = (double)S / kPrepOut;
    const double fsx1 = d * scale, fsx2 = fsx1 + scale;
    const double cell = scale < S - fsx1 ? scale : S - fsx1;
    int sx1 = (int)ceil(fsx1), sx2 = (int)floor(fsx2);
    sx2 = sx2 < S - 1 ? sx2 : S - 1;
    sx1 = sx1 < sx2 ? sx1 : sx2;
    t.head = sx1 - fsx1 > 1e-3;
    t.tail = fsx2 - sx2 > 1e-3;
    t.first = t.head ? sx1 - 1 : sx1;
    t.n = (int)t.head + (sx2 - sx1) + (int)t.tail;
    double last = fsx2 - sx2;
    last = last < 1. ? last : 1.;
    last = last < cell ? last : cell;
    t.a_head = (float)((sx1 - fsx1) / cell);
    t.a_mid = (float)(1.0 / cell);
    t.a_tail = (float)(last / cell);
    return t;
}

__host__ __device__ __forceinline__ float area_tap_weight(const AreaTaps& t, int i) {
    return (t.head && i == 0) ? t.a_head : (t.tail && i == t.n - 1) ? t.a_tail : t.a_mid;
}

// The whole table of one side (the same for x and y: the crop is square)
inline AreaTabHost make_area_tab(int S) {
    AreaTabHost t;
    t.start.assign(kPrepOut, 0); t.cnt.assign(kPrepOut, 1);
    if (S % kPrepOut == 0) {
        t.k = S / kPrepOut; t.mode = t.k == 1 ? kPrepCopy : t.k == 2 ? kPrepBox2 : kPrepBoxK; t.inv = 1.f / (float)(t.k * t.k);
    } else {
        t.mode = kPrepFrac;
        t.taps = (int)std::ceil((double)S / kPrepOut) + 2;
    }
    t.alpha.assign((size_t)kPrepOut * t.taps, 1.f);
    for (int d = 0; d < kPrepOut; d++) {
        const AreaTaps a = area_taps(S, d);
        t.start[d] = a.first; t.cnt[d] = a.n;
        if (t.mode == kPrepFrac)
            for (int i = 0; i < t.taps; i++) t.alpha[(size_t)d * t.taps + i] = i < a.n ? area_tap_weight(a, i) : 0.f;
    }
    return t;
}

struct PrepParams {
    const uint8_t* frames;        // [n][fh][fw][3] BGR
    uint8_t* out;                 // [n][128][128]
    const int* start;             // device copies of the table
    const int* cnt;
    const float* alpha;
    int fh, fw, x0, y0;           // frame size and crop origin
    int mode, k, taps;
    float inv;
};

__device__ __forceinline__ int bgr2gray(const uint8_t* p) {
    return (3735 * (int)__ldg(p) + 19235 * (int)__ldg(p + 1) + 9798 * (int)__ldg(p + 2) + (1 << 14)) >> 15;
}

__global__ void __launch_bounds__(kPrepOut)
preprocess_bgr_kernel(const PrepParams P)
{
    const int dx = threadIdx.x;
    const uint8_t* frame = P.frames + (size_t)blockIdx.y * P.fh * P.fw * 3;
    uint8_t* out = P.out + (size_t)blockIdx.y * kPrepOut * kPrepOut;
    const int sx0 = P.start[dx], nx = P.cnt[dx];
    const float* ax = P.alpha + (size_t)dx * P.taps;

#pragma unroll 1
    for (int r = 0; r < kPrepRowsPerCta; r++) {
        const int dy = blockIdx.x * kPrepRowsPerCta + r;
        const int sy0 = P.start[dy], ny = P.cnt[dy];
        const uint8_t* src = frame + ((size_t)(P.y0 + sy0) * P.fw + (P.x0 + sx0)) * 3;
        int v;
        if (P.mode == kPrepFrac) {
            const float* ay = P.alpha + (size_t)dy * P.taps;
            float sum = 0.f;
            for (int j = 0; j < ny; j++) {
                const uint8_t* row = src + (size_t)j * P.fw * 3;
                float buf = 0.f;
                for (int i = 0; i < nx; i++) buf = __fadd_rn(buf, __fmul_rn((float)bgr2gray(row + 3 * i), ax[i]));
                const float term = __fmul_rn(ay[j], buf);
                sum = j == 0 ? term : __fadd_rn(sum, term);
            }
            v = min(max(__float2int_rn(sum), 0), 255);
        } else {
            int tot = 0;
            for (int j = 0; j < ny; j++) {
                const uint8_t* row = src + (size_t)j * P.fw * 3;
                for (int i = 0; i < nx; i++) tot += bgr2gray(row + 3 * i);
            }
            if (P.mode == kPrepBox2)      v = (tot + 2) >> 2;
            else if (P.mode == kPrepBoxK) v = min(max(__float2int_rn(__fmul_rn((float)tot, P.inv)), 0), 255);
            else                          v = tot;
        }
        out[dy * kPrepOut + dx] = (uint8_t)v;
    }
}

}  // namespace cnnacc
