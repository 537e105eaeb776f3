// tail.cuh -- follow-on stage: 4x4 spatial-bin pool -> linear -> softmax -> argmax -> CAM bbox.
//
// tail_image(): 128 threads (four warps) take one 64x16x16 u8 feature map that sits in SHARED memory (CHW, 16 KiB) to its
// 44 bytes of predictions.  It has two callers:
//   * conv_fused.cuh: four extra warps of the conv-stack kernel run it on the layer-2 staging buffer while the tensor
//     core and the epilogue warps are already busy with the next image -- the features never leave the SM and, when the
//     caller passes no feature pointer, HBM sees 44 B per image instead of 16 KiB out + 16 KiB back in;
//   * classify_bbox_kernel below (features-in entry point, cnnacc_classify_batch and, on windows of a frame's map,
//     cnnacc_scan_frames): eight such groups per CTA.
// Both produce bit-identical predictions because they are the same code on the same bytes.
//
// Reference (all /root/reference/software/realtime_detect.py):
//   classify_vec :68-82   pooled[ch*16 + r*4 + c] = mean of the 4x4 bin of (feat/255); logits = W.pooled + b;
//                         softmax; argmax
//   bbox_vec     :85-116  channels with mean > 250 masked; cam = sum_ch w[cls][ch,bin] * fm (fp32, channel
//                         order); ReLU; /max; thr = max(percentile70, 0.25); bbox of cam > thr, x8 scaling
// Numerics:
//   * bin sums are exact integers; pooled = S / 4080 in one rounding (identical to Classifier.classify's
//     mean-then-/255, pynq_inference.py:325-334; within 1 ulp of classify_vec's /255-then-mean);
//   * logits: fp32, fixed summation tree (4 bins per task, 2 tasks per thread in order, warp shuffle tree, four warp
//     partials pairwise, bias last);
//   * CAM: products and sums rounded separately (no FMA) in channel order 0..63, as numpy's reduction over
//     the outer axis does, so the bbox integers match bit for bit given the same class;
//   * percentile(70) of 256 values = index 178.5 -> hi - (hi-lo)*0.5 in fp32 (numpy _lerp with t = 0.5).
#pragma once
#include "common.cuh"

namespace cnnacc {

constexpr int kMaxClasses = 16;
constexpr int kTailThreads = 128;               // front stage: four warps (bin sums, logits, softmax, CAM) on one image
constexpr int kTailBackThreads = 64;            // back stage: two warps (CAM maximum, percentile, box), one image behind

struct TailArgs {
    const float* fc_w;                          // [n_cls][1024] row-major
    const float* fc_b;                          // [n_cls]
    int n_cls;
    int want_logits;                            // probs receives the raw logits instead of the softmax (CNNACC_FLAG_LOGITS)
    float* probs;                               // [n][n_cls] or null
    int32_t* cls_out;                           // [n] or null
    int32_t* bbox_out;                          // [n][4] or null (null: the CAM stage is skipped)
    const int32_t* cls_in;                      // [n] or null: bbox_vec's cls_idx argument (CNNACC_FLAG_CLS_GIVEN)
};

struct __align__(16) TailScratch {              // per group
    float cam[256];                             // front -> back: the ReLU-ed, not yet normalised CAM of one image
    float sort[256];                            // back: the one cross-warp exchange of its bitonic sort
    float part[4][kMaxClasses];                 // front: per-warp logit partials
    unsigned long long valid[4];                // front, per warp: bit ch = channel ch is not saturated (mean <= 250) and not all zero
    float red[2];                               // back
    float thr;
    int pad;
    int box[2][4];
};
constexpr int kTailScratchBytes = 2560;
static_assert(sizeof(TailScratch) <= kTailScratchBytes, "tail scratch");

__device__ __forceinline__ void tail_bar(int id) { asm volatile("bar.sync %0, %1;" :: "r"(id), "n"(kTailThreads) : "memory"); }
__device__ __forceinline__ void tail_back_bar(int id) { asm volatile("bar.sync %0, %1;" :: "r"(id), "n"(kTailBackThreads) : "memory"); }

// Classifier rows the tail keeps in shared memory.  The rows do not depend on the image, but from global memory every image
// pays L2 latency for them: next to 217 KB of shared memory the SM's L1 is 28 KB and held only 69 % of the 24 KiB (ncu,
// profiles/r2_fusedtail_v1_*).  Rows that do not fit stay on the __ldg path.
struct TailWeights {
    uint32_t smem;                              // shared-space address of [rows][1024] floats (explicit ld.shared: a pointer that
                                                // may be shared or global turns every load into a slow generic LD)
    int rows;
    float bias;                                 // fc_b[lane] for lane < n_cls, read once per kernel
};
__device__ __forceinline__ float lds_f32(uint32_t a) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ float4 lds_f32x4(uint32_t a) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
    return v;
}

// Copies min(n_cls, max_rows) classifier rows into shared memory; call with all threads of the group, then tail_bar.
__device__ __forceinline__ TailWeights tail_stage_weights(float* dst, int max_rows, const TailArgs& A, const int T) {
    TailWeights W;
    W.rows = min(A.n_cls, max_rows);
    W.smem = (uint32_t)__cvta_generic_to_shared(dst);
    for (int i = T; i < W.rows * 256; i += kTailThreads)
        reinterpret_cast<float4*>(dst)[i] = __ldg(reinterpret_cast<const float4*>(A.fc_w) + i);
    W.bias = (T & 31) < A.n_cls ? __ldg(A.fc_b + (T & 31)) : 0.f;
    return W;
}

struct TailNoTrace { __device__ __forceinline__ void operator()(int) const {} };
struct TailTrue { static constexpr bool value = true; };
struct TailFalse { static constexpr bool value = false; };

// The tail is a two-stage pipeline.  tail_front (128 threads) needs the feature map: bin sums, logits, softmax / argmax and
// the class activation map, whose two pixels per thread it returns after ReLU.  tail_back (64 threads) needs only those 256
// floats: maximum, normalisation, 70th percentile, box.  In the fused kernel the two stages run on different warps, one image
// apart, so the serial chain that holds the staging buffer ends with the CAM.
//
// tail_front: T = 0..127 within the group; bar_id = a named barrier reserved for these 128 threads; release() is called by
// every thread after its last read of `stg` (the fused kernel hands the staging buffer back to the epilogue warps there).
// Returns false when no box is wanted (cam0 / cam1 are then not written).
template <typename Release, typename Trace = TailNoTrace>
__device__ __forceinline__ bool tail_front(const uint8_t* __restrict__ stg, TailScratch* sc, const int T, const int bar_id,
                                           const TailArgs& A, const TailWeights& W, const size_t img, float& cam0, float& cam1,
                                           Release release, Trace trace = Trace())
{
    trace(1);
    const int lane = T & 31, w = T >> 5;
    const unsigned full = 0xffffffffu;

    // ---- bin sums: task q = T + 128 i owns channel q/4, bin-row q%4 = four 16-byte map rows (64 contiguous bytes, read in a
    // per-lane rotated order so that the eight lanes of a 128-bit wavefront hit eight different 16-byte bank groups) ----
    int S[2][4];
    unsigned long long vbits = 0;
#pragma unroll
    for (int i = 0; i < 2; i++) {
        const uint4* p = reinterpret_cast<const uint4*>(stg + (T + 128 * i) * 64);
        S[i][0] = S[i][1] = S[i][2] = S[i][3] = 0;
#pragma unroll
        for (int r = 0; r < 4; r++) {
            const uint4 v = p[(r + (T >> 1)) & 3];
            S[i][0] = __dp4a(v.x, 0x01010101u, (unsigned)S[i][0]);
            S[i][1] = __dp4a(v.y, 0x01010101u, (unsigned)S[i][1]);
            S[i][2] = __dp4a(v.z, 0x01010101u, (unsigned)S[i][2]);
            S[i][3] = __dp4a(v.w, 0x01010101u, (unsigned)S[i][3]);
        }
        // channel mean <= 250  <=>  channel sum <= 64000 (bbox_vec: valid = ch_means <= 250)
        int cs = S[i][0] + S[i][1] + S[i][2] + S[i][3];
        cs += __shfl_xor_sync(full, cs, 1);
        cs += __shfl_xor_sync(full, cs, 2);
        // lanes 4q..4q+3 of warp w hold channel 32 i + 8 w + q: squeeze ballot bits 0,4,..,28 into one byte.  A channel that is
        // zero everywhere adds (+-)0 to every CAM pixel, exactly like a masked one, so it is dropped from the CAM as well.
        uint32_t b = __ballot_sync(full, cs <= 250 * 256 && cs > 0) & 0x11111111u;
        b = (b | (b >> 3)) & 0x03030303u;
        b = (b | (b >> 6)) & 0x000F000Fu;
        b = (b | (b >> 12)) & 0xFFu;
        vbits |= (unsigned long long)b << (32 * i + 8 * w);
    }
    if (lane == 0) sc->valid[w] = vbits;                  // each warp knows a quarter of the channels
    trace(2);

    // ---- logits: W row-major [n_cls][1024]; task q covers bins 4q .. 4q+3 ----
    float pooled[2][4];
#pragma unroll
    for (int i = 0; i < 2; i++)
#pragma unroll
        for (int c = 0; c < 4; c++) pooled[i][c] = div_rn_zero_ok((float)S[i][c], 4080.0f);
    // three classes at a time: their shuffle trees are independent and interleave (one tree is ~150 clk of pure latency)
    for (int k0 = 0; k0 < A.n_cls; k0 += 3) {
        float acc[3];
#pragma unroll
        for (int c = 0; c < 3; c++) {
            const int k = min(k0 + c, A.n_cls - 1);       // the padding classes of the last group recompute the last one
            const bool in_smem = k < W.rows;              // uniform
            const float4* wr = reinterpret_cast<const float4*>(A.fc_w + (size_t)k * 1024) + T;
            const uint32_t ws = W.smem + (uint32_t)(k * 4096 + T * 16);
#pragma unroll
            for (int i = 0; i < 2; i++) {
                float4 wv;
                if (in_smem) wv = lds_f32x4(ws + 2048 * i); else wv = __ldg(wr + 128 * i);
                float p = pooled[i][0] * wv.x;
                p = fmaf(pooled[i][1], wv.y, p);
                p = fmaf(pooled[i][2], wv.z, p);
                p = fmaf(pooled[i][3], wv.w, p);
                acc[c] = i ? acc[c] + p : p;
            }
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
#pragma unroll
            for (int c = 0; c < 3; c++) acc[c] += __shfl_xor_sync(full, acc[c], off);
        }
        if (lane == 0) {
#pragma unroll
            for (int c = 0; c < 3; c++)
                if (k0 + c < A.n_cls) sc->part[w][k0 + c] = acc[c];
        }
    }
    trace(3);
    tail_bar(bar_id);                                     // #1: partials and the valid mask are visible

    // ---- softmax / argmax: every warp computes it (no second barrier), warp 0 writes ----
    float logit = -INFINITY;
    if (lane < A.n_cls) logit = ((sc->part[0][lane] + sc->part[1][lane]) + (sc->part[2][lane] + sc->part[3][lane])) + W.bias;
    float mx = logit;
    int arg = lane < A.n_cls ? lane : 0x7fffffff;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        const float om = __shfl_xor_sync(full, mx, off);
        const int   oa = __shfl_xor_sync(full, arg, off);
        if (om > mx || (om == mx && oa < arg)) { mx = om; arg = oa; }   // first maximum, like np.argmax
    }
    if (w == 0) {
        if (A.probs) {
            const float e = lane < A.n_cls ? expf(logit - mx) : 0.f;
            float sum = e;
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) sum += __shfl_xor_sync(full, sum, off);
            if (lane < A.n_cls) A.probs[img * A.n_cls + lane] = A.want_logits ? logit : div_rn_zero_ok(e, sum);
        }
        if (lane == 0 && A.cls_out && !A.cls_in) A.cls_out[img] = arg;
    }
    if (!A.bbox_out) {                                    // uniform: a kernel argument
        release();
        tail_bar(bar_id);                                 // everyone has read sc->part before the next image overwrites it
        return false;
    }
    trace(4);
    // bbox_vec takes the class as an argument (realtime_detect.py:85); cls_in carries it when given
    const int cls = A.cls_in ? min(max(A.cls_in[img], 0), A.n_cls - 1) : arg;

    // ---- CAM: thread T owns pixels 2T, 2T+1 = row T/8, columns 2(T%8), +1, both in bin (T/32, (T%8)/2), so one class weight and
    // one 16-bit feature load per channel serve two pixels.  Saturated channels contribute w = 0 (bbox_vec zeroes their weights),
    // all-zero channels +-0: neither can change a sum that starts at +0, so with few active channels (this network saturates: 21
    // of 64 on random images at the default shifts) only those are visited, in ascending order.  u8 -> f32 and the product in
    // ONE rounding: x = 0x4B0000bb is the float 2^23 + b, and fma(w, x, -w * 2^23) rounds the exact w * b -- the same value as
    // fmul_rn(w, float(b)) -- so a pixel-channel costs one PRMT, one FFMA and the separately rounded FADD numpy's reduction does.
    const unsigned long long valid = (sc->valid[0] | sc->valid[1]) | (sc->valid[2] | sc->valid[3]);
    const bool cam_smem = cls < W.rows;                   // uniform: every thread has the same class
    const int woff = cls * 1024 + (T >> 5) * 4 + ((T & 7) >> 1);
    const float* wc = A.fc_w + woff;
    const uint32_t wcs = W.smem + 4u * (uint32_t)woff;
    const uint16_t* fwp = reinterpret_cast<const uint16_t*>(stg) + T;
    float cam[2] = {0.f, 0.f};
    auto cam_pass = [&](auto from_smem) {
        if (__popcll(valid) <= 40) {                      // sparse: walk the set bits, the next channel's operands one step ahead
            uint32_t m_lo = (uint32_t)valid, m_hi = (uint32_t)(valid >> 32);
            auto next = [&]() -> int {
                if (m_lo) { const int c = __ffs(m_lo) - 1; m_lo &= m_lo - 1; return c; }
                if (m_hi) { const int c = __ffs(m_hi) - 1; m_hi &= m_hi - 1; return c + 32; }
                return -1;
            };
            auto load = [&](int ch, float& wv, uint32_t& word) {
                wv = decltype(from_smem)::value ? lds_f32(wcs + 64u * (uint32_t)ch) : __ldg(wc + ch * 16);
                word = fwp[ch * 128];
            };
            int ch = next();
            float wv_n = 0.f;
            uint32_t word_n = 0;
            if (ch >= 0) load(ch, wv_n, word_n);
            while (ch >= 0) {
                const float wv = wv_n;
                const uint32_t word = word_n;
                ch = next();
                if (ch >= 0) load(ch, wv_n, word_n);
                const float cc = __fmul_rn(wv, -8388608.0f);
                cam[0] = __fadd_rn(cam[0], __fmaf_rn(wv, __uint_as_float(__byte_perm(word, 0x4B000000u, 0x7440)), cc));
                cam[1] = __fadd_rn(cam[1], __fmaf_rn(wv, __uint_as_float(__byte_perm(word, 0x4B000000u, 0x7441)), cc));
            }
            return;
        }
        // dense: 4 x 16 channels, constant offsets inside, one mask word per block
#pragma unroll 1
        for (int o = 0; o < 4; o++) {
            const uint32_t vm = (uint32_t)(valid >> (16 * o));
#pragma unroll
            for (int c = 0; c < 16; c++) {
                const int ch = 16 * o + c;
                float wv = decltype(from_smem)::value ? lds_f32(wcs + 64u * (uint32_t)ch) : __ldg(wc + ch * 16);
                wv = ((vm >> c) & 1u) ? wv : 0.f;
                const float cc = __fmul_rn(wv, -8388608.0f);   // exact
                const uint32_t word = fwp[ch * 128];
                cam[0] = __fadd_rn(cam[0], __fmaf_rn(wv, __uint_as_float(__byte_perm(word, 0x4B000000u, 0x7440)), cc));
                cam[1] = __fadd_rn(cam[1], __fmaf_rn(wv, __uint_as_float(__byte_perm(word, 0x4B000000u, 0x7441)), cc));
            }
        }
    };
    if (cam_smem) cam_pass(TailTrue()); else cam_pass(TailFalse());
    release();                                            // last read of the feature map
    trace(5);
    cam0 = fmaxf(cam[0], 0.f);
    cam1 = fmaxf(cam[1], 0.f);
    tail_bar(bar_id);                                     // #2: everyone has read sc->part / sc->valid of this image
    return true;
}

// tail_back: T = 0..63; v[b] = ReLU-ed CAM of pixel 4T + b (row T/4, columns 4(T%4) + b); bar_id = a named barrier reserved for
// these 64 threads.  Maximum -> normalise -> 70th percentile of the 256 values (index 178.5: sorted[178], sorted[179]) ->
// threshold -> box.  Bitonic sort of element e = 4T + b: strides 1, 2 stay inside the thread, 4..64 are warp shuffles
// (lane ^ stride/4), 128 is one exchange through shared memory.
template <typename Trace = TailNoTrace>
__device__ __forceinline__ void tail_back(float (&cam)[4], TailScratch* sc, const int T, const int bar_id, const TailArgs& A,
                                          const size_t img, Trace trace = Trace())
{
    const int lane = T & 31, w = T >> 5;
    const unsigned full = 0xffffffffu;
    float m = fmaxf(fmaxf(cam[0], cam[1]), fmaxf(cam[2], cam[3]));
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) m = fmaxf(m, __shfl_xor_sync(full, m, off));
    if (lane == 0) sc->red[w] = m;
    tail_back_bar(bar_id);
    m = fmaxf(sc->red[0], sc->red[1]);
    if (m > 0.f) {
#pragma unroll
        for (int b = 0; b < 4; b++) cam[b] = div_rn_zero_ok(cam[b], m);
    }
    trace(6);
    float v[4] = {cam[0], cam[1], cam[2], cam[3]};
#pragma unroll
    for (int k = 2; k <= 256; k <<= 1) {
        const bool up = (k == 256) ? true : ((T & (k >> 2)) == 0);       // k == 2: decided per pair below
#pragma unroll
        for (int j = k >> 1; j > 0; j >>= 1) {
            if (j == 128) {
                reinterpret_cast<float4*>(sc->sort)[T] = make_float4(v[0], v[1], v[2], v[3]);
                tail_back_bar(bar_id);
                const float4 o = reinterpret_cast<const float4*>(sc->sort)[T ^ 32];
                const bool lower = (T & 32) == 0;         // k = 256: every block ascends
                v[0] = lower ? fminf(v[0], o.x) : fmaxf(v[0], o.x);
                v[1] = lower ? fminf(v[1], o.y) : fmaxf(v[1], o.y);
                v[2] = lower ? fminf(v[2], o.z) : fmaxf(v[2], o.z);
                v[3] = lower ? fminf(v[3], o.w) : fmaxf(v[3], o.w);
            } else if (j >= 4) {
                const bool keep_min = (((T & (j >> 2)) == 0) == up);
#pragma unroll
                for (int b = 0; b < 4; b++) {
                    const float o = __shfl_xor_sync(full, v[b], j >> 2);
                    v[b] = keep_min ? fminf(v[b], o) : fmaxf(v[b], o);
                }
            } else {
#pragma unroll
                for (int a = 0; a < 4; a++) {
                    if (a & j) continue;
                    const bool asc = (k == 2) ? ((a & 2) == 0) : up;
                    const float lo = fminf(v[a], v[a | j]), hi = fmaxf(v[a], v[a | j]);
                    v[a] = asc ? lo : hi;
                    v[a | j] = asc ? hi : lo;
                }
            }
        }
    }
    trace(7);
    if (T == 44) {                                        // elements 178, 179 = thread 44, b = 2, 3
        const float lo = v[2], hi = v[3];
        float thr = __fsub_rn(hi, __fmul_rn(__fsub_rn(hi, lo), 0.5f));
        sc->thr = (0.25f > thr) ? 0.25f : thr;            // python max(p, 0.25)
    }
    tail_back_bar(bar_id);
    const float thr = sc->thr;
    const int x0 = 4 * (T & 3), y = T >> 2;
    int xmin = 16, xmax = -1;
#pragma unroll
    for (int b = 0; b < 4; b++)
        if (cam[b] > thr) { xmin = min(xmin, x0 + b); xmax = x0 + b; }
    int ymin = xmax >= 0 ? y : 16, ymax = xmax >= 0 ? y : -1;
    xmin = __reduce_min_sync(full, xmin); ymin = __reduce_min_sync(full, ymin);
    xmax = __reduce_max_sync(full, xmax); ymax = __reduce_max_sync(full, ymax);
    if (lane == 0) { sc->box[w][0] = xmin; sc->box[w][1] = ymin; sc->box[w][2] = xmax; sc->box[w][3] = ymax; }
    tail_back_bar(bar_id);
    if (T == 0) {
        xmin = min(sc->box[0][0], sc->box[1][0]); ymin = min(sc->box[0][1], sc->box[1][1]);
        xmax = max(sc->box[0][2], sc->box[1][2]); ymax = max(sc->box[0][3], sc->box[1][3]);
        int4 bx;
        if (xmax >= 0) bx = make_int4(xmin * 8, ymin * 8, min(127, (xmax + 1) * 8), min(127, (ymax + 1) * 8));
        else bx = make_int4(0, 0, 127, 127);
        reinterpret_cast<int4*>(A.bbox_out)[img] = bx;
    }
    trace(8);
}

// Features-in entry point: persistent CTAs of seven 128-thread groups; a group copies its item's 16 KiB map into its own
// shared-memory slot (8 independent 128-bit loads per thread), runs tail_front on it, and its first two warps then run
// tail_back while the other two already fetch the next item.  Where an item's map comes from is the one thing that varies:
//   CompactMaps  cnnacc_classify_batch: item img is the 16 KiB map feats[img];
//   ScanWindows  cnnacc_scan_frames / cnnacc_scan_pyramid: item img is a 16 x 16 window of a frame's [64][ho][wo] map
//                (of one of its pyramid levels), gathered in place.
// Both hand the same slot layout to the same tail_front / tail_back, so a window's predictions are classify_batch's on the
// window's map, bit for bit.  load(img, T, v): thread T's eight 16-byte rows, row T + 128 r = channel (T >> 4) + 8 r, map row
// T & 15.
struct CompactMaps {
    const uint8_t* feats;
    __device__ __forceinline__ void load(long long img, int T, uint4 (&v)[8]) const {
        const uint4* src = reinterpret_cast<const uint4*>(feats + (size_t)img * 16384);
#pragma unroll
        for (int r = 0; r < 8; r++) v[r] = __ldcs(src + T + kTailThreads * r);       // read once: streaming
    }
};

// The 16 bytes at byte offset sh (0..15) of the 32 bytes a:b.
__device__ __forceinline__ uint4 bytes_at(const uint4 a, const uint4 b, int sh) {
    uint32_t w0 = a.x, w1 = a.y, w2 = a.z, w3 = a.w, w4 = b.x, w5 = b.y, w6 = b.z, w7 = b.w;
    if (sh & 8) { w0 = w2; w1 = w3; w2 = w4; w3 = w5; w4 = w6; w5 = w7; }
    if (sh & 4) { w0 = w1; w1 = w2; w2 = w3; w3 = w4; w4 = w5; }
    const uint32_t s = 8u * (sh & 3);
    return make_uint4(__funnelshift_r(w0, w1, s), __funnelshift_r(w1, w2, s), __funnelshift_r(w2, w3, s), __funnelshift_r(w3, w4, s));
}

// Window (ix, iy) of a level of frame f is the level map's cells [v, v + 16) x [u, u + 16), u = min(ix step, umax),
// v = min(iy step, vmax): the 128 x 128 level pixels at (8u, 8v).  Windows are numbered frame-major, then level, then row,
// then column, so the seven groups of a CTA take horizontally adjacent windows, which share 15/16 of their bytes: L1 serves
// most of the gather.  A row of a window starts at any byte (u may be odd): it is read as the two aligned 16-byte blocks
// around it and shifted into place.  With ho and wo even, a channel plane is a multiple of 4 bytes, so the shift is the same
// for all eight rows of a thread.  The second block of a row that starts aligned lies past the row: the workspace has 16
// bytes of slack after the last map.  cnnacc_scan_frames is the one-level case (the frame's own map).
constexpr int kScanMaxLevels = 16;
struct ScanLevel {
    const uint8_t* feats;                       // [k][64][ho][wo], 16-byte aligned
    int ho, wo, nx, umax, vmax, first;          // map size, windows per row, last origins in cells, first window in a frame
};
// kOneLevel: the instance of one-level calls (cnnacc_scan_frames), which looks up no level; the other walks the table.
template <bool kOneLevel>
struct ScanWindows {
    int per, step, n_levels;                    // windows per frame, stride / 8, levels
    ScanLevel lv[kOneLevel ? 1 : kScanMaxLevels];
    __device__ __forceinline__ void load(long long img, int T, uint4 (&v)[8]) const {
        const long long f = img / per;
        const int rem = (int)(img - f * per);
        if constexpr (kOneLevel) {
            gather(lv[0], f, rem, T, v);
        } else {
            int l = 0;
            while (l + 1 < n_levels && rem >= lv[l + 1].first) l++;
            gather(lv[l], f, rem - lv[l].first, T, v);
        }
    }
    // window rem of level L of frame f
    __device__ __forceinline__ void gather(const ScanLevel& L, long long f, int rem, int T, uint4 (&v)[8]) const {
        const int iy = rem / L.nx, ix = rem - iy * L.nx;
        const size_t plane = (size_t)L.ho * L.wo;
        const uint8_t* p = L.feats + (size_t)f * 64 * plane + (size_t)(min(iy * step, L.vmax) + (T & 15)) * L.wo +
                           min(ix * step, L.umax) + (size_t)(T >> 4) * plane;
        const int sh = (int)(reinterpret_cast<uintptr_t>(p) & 15);
        const uint4* a = reinterpret_cast<const uint4*>(p - sh);
        const size_t step8 = 8 * plane / 16;                // channel c -> c + 8, in 16-byte blocks
#pragma unroll
        for (int r = 0; r < 8; r++) v[r] = bytes_at(__ldg(a + r * step8), __ldg(a + r * step8 + 1), sh);
    }
};

constexpr int kTailGroups = 7;                          // 7 x (one 128-thread + one 64-thread named barrier) = 14 of the 15 ids
constexpr int kTailSmemW = kMaxClasses * 4096;          // every classifier row, shared by the groups
constexpr int kTailSmem = kTailGroups * (16384 + kTailScratchBytes) + kTailSmemW;

template <class Maps>
__global__ void __launch_bounds__(kTailGroups * kTailThreads, 1)
classify_bbox_kernel(const __grid_constant__ Maps maps, long long n, const TailArgs A)
{
    extern __shared__ __align__(16) uint8_t tail_smem[];
    const int g = threadIdx.x / kTailThreads, T = threadIdx.x % kTailThreads;
    const int bar_front = 1 + g, bar_back = 1 + kTailGroups + g;
    uint8_t* stg = tail_smem + g * 16384;
    TailScratch* sc = reinterpret_cast<TailScratch*>(tail_smem + kTailGroups * 16384 + g * kTailScratchBytes);
    float* wsm = reinterpret_cast<float*>(tail_smem + kTailGroups * (16384 + kTailScratchBytes));
    // all threads stage the n_cls classifier rows once per CTA
    for (int i = threadIdx.x; i < A.n_cls * 256; i += kTailGroups * kTailThreads)
        reinterpret_cast<float4*>(wsm)[i] = __ldg(reinterpret_cast<const float4*>(A.fc_w) + i);
    TailWeights W;
    W.smem = (uint32_t)__cvta_generic_to_shared(wsm); W.rows = A.n_cls;
    W.bias = (T & 31) < A.n_cls ? __ldg(A.fc_b + (T & 31)) : 0.f;
    __syncthreads();
    for (long long img = (long long)blockIdx.x * kTailGroups + g; img < n; img += (long long)gridDim.x * kTailGroups) {
        uint4 v[8];
        maps.load(img, T, v);
        // (the previous image's tail_front ended with a group barrier after its last read of stg, and its tail_back
        // threads have read sc->cam before they come back here: both buffers are free)
#pragma unroll
        for (int r = 0; r < 8; r++) reinterpret_cast<uint4*>(stg)[T + kTailThreads * r] = v[r];
        tail_bar(bar_front);
        float c0, c1;
        const bool want_box = tail_front(stg, sc, T, bar_front, A, W, (size_t)img, c0, c1, [] {});
        if (want_box) {
            reinterpret_cast<float2*>(sc->cam)[T] = make_float2(c0, c1);
            tail_bar(bar_front);
            if (T < kTailBackThreads) {
                const float4 q = reinterpret_cast<const float4*>(sc->cam)[T];
                float cam[4] = {q.x, q.y, q.z, q.w};
                tail_back(cam, sc, T, bar_back, A, (size_t)img);
            }
        }
    }
}

// Spatial-bin pooled features alone: (64,256) u8 -> (1024,) f32, pooled[ch*16 + r*4 + c] = mean(4x4 bin) / 255 -- the
// classifier's input, which the reference's trainer builds from a feature dump (retrain_classifier.py:188-205) and
// Classifier.classify builds per image (pynq_inference.py:325-334).  Bin sums are exact integers and sum/16 is exact,
// so one correctly rounded division S/4080 equals the reference's mean-then-/255.
__global__ void __launch_bounds__(256)
pool_features_kernel(const uint8_t* __restrict__ feats, float* __restrict__ pooled)
{
    const int t = threadIdx.x;
    const size_t img = blockIdx.x;
    const uint4* src = reinterpret_cast<const uint4*>(feats + img * 16384);
    int S[4] = {0, 0, 0, 0};                     // thread t: channel t/4, bin-row t%4 -> bins 4t .. 4t+3
#pragma unroll
    for (int r = 0; r < 4; r++) {
        const uint4 v = __ldg(src + t * 4 + r);
        S[0] = __dp4a(v.x, 0x01010101u, (unsigned)S[0]);
        S[1] = __dp4a(v.y, 0x01010101u, (unsigned)S[1]);
        S[2] = __dp4a(v.z, 0x01010101u, (unsigned)S[2]);
        S[3] = __dp4a(v.w, 0x01010101u, (unsigned)S[3]);
    }
    reinterpret_cast<float4*>(pooled + img * 1024)[t] =
        make_float4(div_rn_zero_ok((float)S[0], 4080.0f), div_rn_zero_ok((float)S[1], 4080.0f),
                    div_rn_zero_ok((float)S[2], 4080.0f), div_rn_zero_ok((float)S[3], 4080.0f));
}

}  // namespace cnnacc
