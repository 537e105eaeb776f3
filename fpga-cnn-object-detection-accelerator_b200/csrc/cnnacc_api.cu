// cnnacc_api.cu -- the C ABI of include/cnnacc.h: handle, host logic, launches.  No CPU compute path.
#include "../../include/cnnacc.h"

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <memory>
#include <mutex>
#include <string>
#include <system_error>
#include <thread>
#include <utility>
#include <vector>

#include "conv_direct.cuh"
#include "conv_fused.cuh"
#include "tail.cuh"
#include "int8_peak_probe.cuh"
#include "cam_upsampled.cuh"
#include "preprocess.cuh"
#include "regions.cuh"
#include "pyramid.cuh"
#include "region_plan.h"
#include "region_merge.cuh"
#include "pil_resize.cuh"
#include "host_chunks.h"
#include "pdl_chain.h"
#include "shard_plan.h"
#include "tiling.cuh"
#include "weights_pack.h"

using namespace cnnacc;

namespace {

constexpr int kSlots = 4;                       // staging buffers in flight for host-pointer batches
constexpr int kSmallN = 64;                     // calls up to this many units skip the staging ring (latency path)
constexpr size_t kPredBytesPerImage = 16 + kMaxClasses * 4 + 4;   // bbox | probs | cls, sized for the most classes
constexpr int64_t kPredSuper = 1 << 20;         // host-pointer calls bring predictions back in blocks of up to this many images
constexpr size_t kBramBytes = 16 * 4096 + 32 * 1024 + 64 * 256;   // 112-channel feature-BRAM mirror
constexpr int64_t kRegionLaunch = 1024;         // host-pointer region calls: regions per launch (16 MiB of gray per slot)
constexpr int kDescRing = 4;                    // region-descriptor buffers in flight

// ---- owners of the handle's CUDA resources: move-only, the destructor frees what they hold ------------------------------

enum class Mem { kDevice, kPinned, kMapped };   // cudaMalloc / cudaHostAlloc default / cudaHostAlloc mapped

// cap elements of T at p, or nothing; grow() (below) is the one place that allocates one.
template <class T, Mem K = Mem::kDevice>
struct Buf {
    T* p = nullptr;
    size_t cap = 0;
    Buf() = default;
    Buf(Buf&& o) noexcept : p(std::exchange(o.p, nullptr)), cap(std::exchange(o.cap, 0)) {}
    Buf& operator=(Buf&& o) noexcept { std::swap(p, o.p); std::swap(cap, o.cap); return *this; }
    ~Buf() { release(); }
    // frees the allocation; the buffer is empty afterwards whatever the free returned
    cudaError_t release() {
        const cudaError_t e = !p ? cudaSuccess : K == Mem::kDevice ? cudaFree(p) : cudaFreeHost(p);
        p = nullptr; cap = 0;
        return e;
    }
};

// A CUDA event or stream, created by create(flags).
template <class T, cudaError_t (*Create)(T*, unsigned), cudaError_t (*Destroy)(T)>
struct Owned {
    T raw = nullptr;
    Owned() = default;
    Owned(Owned&& o) noexcept : raw(std::exchange(o.raw, nullptr)) {}
    Owned& operator=(Owned&& o) noexcept { std::swap(raw, o.raw); return *this; }
    ~Owned() { if (raw) Destroy(raw); }
    cudaError_t create(unsigned flags) { return Create(&raw, flags); }
    operator T() const { return raw; }
};
using Event = Owned<cudaEvent_t, cudaEventCreateWithFlags, cudaEventDestroy>;
using Stream = Owned<cudaStream_t, cudaStreamCreateWithFlags, cudaStreamDestroy>;

// Pinned host and device copies of one call's region descriptors (and, for the merging calls, of its per-frame region
// ranges); ev is recorded after the call's last launch that reads them.
struct DescBuf {
    Buf<int4, Mem::kPinned> host;
    Buf<int4> dev;
    Buf<long long, Mem::kPinned> first_host;
    Buf<long long> first_dev;
    Event ev;
};

struct Slot {
    Event ev_in, ev_k, ev_out;                  // H2D landed / kernels done / D2H drained
    Buf<uint8_t> d_in, d_out;
    Buf<int32_t> d_cls, d_bbox;                 // cnnacc_cam_bbox_batch's classes in and boxes out
};

std::string g_create_error;
std::atomic<int64_t> g_pdl_seq{0};              // programmatic conv-stack launches of ALL handles (see conv_stack_device)

}  // namespace

// No user-provided default constructor: `new cnnacc_handle()` zero-initialises the members without an initialiser
// (fused's weight arrays, one_map).
struct cnnacc_handle {
    int device = 0;
    Stream own_stream;
    cudaStream_t stream = nullptr;                  // own_stream or the caller's (cnnacc_set_stream)
    Stream st_h2d, st_k, st_d2h;                    // one stream per engine for host-pointer batches
    Event ev_t0, ev_t1, ev_a, ev_b, ev_done;
    int sm_count = 0;
    bool weights_loaded = false, fc_loaded = false, tail_attr_set = false, scan_attr_set = false, pyramid_attr_set = false;
    int shifts[3] = {2, 4, 6};                  // SHIFT_L0..2 defaults, pynq_inference.py:83-85
    bool acc24 = false;                         // accumulator width: false = int32 (arm_cnn.c:31), true = 24-bit wrap (accumulator.v:15)
    uint8_t wbin[CNNACC_WEIGHT_BYTES];
    // device-side weights
    Buf<uint32_t> d_wdirect; size_t wdirect_off[3] = {0, 0, 0};
    FusedWeights fused;                         // packed operands of the fused kernel (conv_fused.cuh)
    Buf<float> d_fcw, d_fcb; int n_cls = 0;
    float fcw_host[kMaxClasses * 1024], fcb_host[kMaxClasses];   // what d_fcw / d_fcb hold: sharded calls compare members
    // workspaces (grown on demand) for the per-layer path and for infer_batch
    Buf<uint8_t> d_l0, d_l1, d_feat;
    Slot slots[kSlots];
    // pre-processing (preprocess.cuh): INTER_AREA weight table of the last crop side seen
    int prep_side = 0; AreaTabHost prep_tab;
    Buf<int> d_prep_start, d_prep_cnt; Buf<float> d_prep_alpha;
    Buf<uint8_t> d_gray;
    // scanning calls (cnnacc_scan_frames / cnnacc_scan_objects): full-resolution gray frames and their feature maps
    Buf<uint8_t> d_scan_gray, d_scan_feat;
    DescBuf rdesc[kDescRing]; int rdesc_next = 0;   // region calls (regions_impl)
    // merging calls (region_merge.cuh): device predictions of detect_objects' device-pointer path, and the detections of
    // host-pointer merges on the device and in pinned memory
    Buf<uint8_t> d_mpred;
    Buf<uint8_t> d_det; Buf<uint8_t, Mem::kPinned> h_det;
    bool merge_attr_set = false;
    // load_image_any (pil_resize.cuh): Pillow coefficient tables of the last (H, W) seen, on the device
    int pil_h = 0, pil_w = 0, pil_kh = 0, pil_kw = 0;
    Buf<int32_t> d_pil_kx, d_pil_bx, d_pil_ky, d_pil_by;
    Buf<uint8_t> d_pil_tmp, d_pil_in, d_pil_out;
    // the prediction block of host-pointer calls (PredBlock): device block the kernels write, pinned block it is copied to
    Buf<uint8_t> d_pred; Buf<uint8_t, Mem::kPinned> h_pred;
    // single-image protocol state
    Buf<uint8_t, Mem::kMapped> h_img, h_bram;       // the batch-1 path runs zero-copy on them
    Buf<int, Mem::kMapped> h_done;                  // completion word of the batch-1 path
    int* h_done_dev = nullptr;                      // its device address
    int done_seq = 0;
    uint8_t *h_img_dev = nullptr, *h_bram_dev = nullptr;   // their device addresses
    CUtensorMap one_map;                            // tensor map over h_img (1 image), encoded once
    bool one_map_ok = false;
    Buf<uint8_t> d_img1, d_bram;
    bool image_loaded = false, started = false;
    int64_t launches = 0;
    PdlChain pdl;                                   // overlapped back-to-back conv-stack launches (pdl_chain.h)
    // cnnacc_run_batch_async: completion events of the last kMaxPending submitted calls, and the ring position the staging
    // slots continue from (asynchronous calls share one continuous ring across calls)
    Event ev_ticket[CNNACC_MAX_PENDING];
    int64_t next_ticket = 0, ring_ci = 0;
    std::string err;

    ~cnnacc_handle() { fused_free(fused); }
};

namespace {

int fail(cnnacc_handle* h, int code, const std::string& msg) {
    if (h) h->err = msg; else g_create_error = msg;
    return code;
}
#define CU(h, call)                                                                              \
    do {                                                                                         \
        cudaError_t e_ = (call);                                                                 \
        if (e_ != cudaSuccess)                                                                   \
            return fail((h), CNNACC_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); \
    } while (0)

// Makes b hold at least n elements: nothing when it does already, otherwise free, then allocate exactly n -- never both at
// once, which would double the peak of the 512 MiB per-layer workspaces.  Contents are not kept.  On failure b is empty.
template <class T, Mem K>
int grow(cnnacc_handle* h, Buf<T, K>& b, size_t n) {
    if (n <= b.cap) return 0;
    const size_t bytes = n * sizeof(T);
    void* p = nullptr;
    cudaError_t e = b.release();
    if (e == cudaSuccess)
        e = K == Mem::kDevice ? cudaMalloc(&p, bytes)
                              : cudaHostAlloc(&p, bytes, K == Mem::kMapped ? cudaHostAllocMapped : cudaHostAllocDefault);
    if (e != cudaSuccess)
        return fail(h, CNNACC_ERR_CUDA, "growing a buffer to " + std::to_string(bytes) + " bytes: " + cudaGetErrorString(e));
    b.p = static_cast<T*>(p);
    b.cap = n;
    return 0;
}

// Device pointers go straight into TMA descriptors, bulk stores and 128-bit loads / stores: a misaligned one would fault the
// whole context, so it is refused here.  (Host pointers are copied into the library's own aligned staging buffers.)
bool aligned(const void* p, uintptr_t a) { return (reinterpret_cast<uintptr_t>(p) & (a - 1)) == 0; }
#define REQUIRE_ALIGNED(h, p, a, what)                                                                           \
    do {                                                                                                         \
        if ((p) && !aligned((p), (a)))                                                                           \
            return fail((h), CNNACC_ERR_ARG, std::string(what) + " device pointer must be " #a "-byte aligned"); \
    } while (0)

bool valid_hw(int H, int W) { return H >= 16 && W >= 16 && H % 16 == 0 && W % 16 == 0 && H <= 8192 && W <= 8192; }

// An integer environment setting (CNNACC_PDL, INTEGRATION.md): the variable's value, or dflt when it is unset.  Read once,
// into a function-local static where it is used.
int env_int(const char* name, int dflt) { const char* e = getenv(name); return e ? atoi(e) : dflt; }

// Which kernels run the conv stack of an H x W call.  128x128 is one fused launch (its maps can also be kept); larger sizes
// run as overlapping 128x128 windows through the fused kernel; everything else, and DIRECT, takes the per-layer kernels.
enum class ConvPath { kFused128, kFusedWindows, kPerLayer };
ConvPath conv_path(int H, int W, uint32_t flags) {
    if (flags & CNNACC_FLAG_DIRECT) return ConvPath::kPerLayer;
    if (H == CNNACC_IMG && W == CNNACC_IMG) return ConvPath::kFused128;
    if (H >= CNNACC_IMG && W >= CNNACC_IMG && !(flags & CNNACC_FLAG_KEEP_MAPS)) return ConvPath::kFusedWindows;
    return ConvPath::kPerLayer;
}

// Does the classifier tail of a 128x128 call run inside the fused conv kernel, on the feature map still in shared memory?
bool tail_in_conv(uint32_t flags) {
    return conv_path(CNNACC_IMG, CNNACC_IMG, flags) == ConvPath::kFused128 &&
           !(flags & (CNNACC_FLAG_KEEP_MAPS | CNNACC_FLAG_TWO_KERNELS));
}

// One layer of the generic per-layer path on `stream`.
int launch_direct_layer(cnnacc_handle* h, cudaStream_t stream, int layer, const uint8_t* in, uint8_t* out,
                        int64_t n, int H, int W) {
    const int tiles_x = (W + kDirTile - 1) / kDirTile, tiles_y = (H + kDirTile - 1) / kDirTile;
    // image and tile share gridDim.x (2^31-1); gridDim.y (65535) would overflow at 8192x8192 (256 x 256 layer-0 tiles)
    if (n * tiles_x * tiles_y > 0x7fffffffLL) return fail(h, CNNACC_ERR_ARG, "too many tiles in one launch");
    dim3 grid((unsigned)(n * tiles_x * tiles_y), 1u, (unsigned)(kLayers[layer].oc / kDirOcb));
    conv3x3_pool_direct_kernel<<<grid, 256, 0, stream>>>(in, out, h->d_wdirect.p + h->wdirect_off[layer],
                                                         kLayers[layer].ic, kLayers[layer].oc, H, W,
                                                         h->shifts[layer], tiles_x, tiles_x * tiles_y, h->acc24 ? 1 : 0);
    h->launches++;
    CU(h, cudaGetLastError());
    return 0;
}

// Conv stack for n device-resident images on `stream`.  l0/l1 are workspaces for the per-layer path.
int conv_stack_device(cnnacc_handle* h, cudaStream_t stream, const uint8_t* d_imgs, int64_t n, int H, int W,
                      uint8_t* d_feats, uint32_t flags, uint8_t* d_l0, uint8_t* d_l1) {
    const ConvPath path = conv_path(H, W, flags);
    if (path == ConvPath::kFused128) {
        // May this launch overlap the previous conv-stack launch (no griddepcontrol.wait)?  Only if that one is the last thing
        // this handle launched, on the same stream, and none of the launches since the last full wait shares memory with it.
        static const bool pdl_on = env_int("CNNACC_PDL", 1) != 0;
        // Why a waiting launch is enough of a fence: every launch in such a chain fills all SMs with one CTA each, so a CTA of
        // launch B only starts on an SM after the CTAs of A, A-1, ... there have exited -- "A complete" implies the whole chain
        // is.  Launches smaller than the SM count therefore always wait and break the chain, and so does any other kernel of
        // this handle (launch counter) or a conv-stack launch of ANOTHER handle (global sequence number).
        int pdl_wait = -1;                               // -1: plain launch
        if (pdl_on && !(flags & CNNACC_FLAG_KEEP_MAPS)) {
            const uintptr_t in = reinterpret_cast<uintptr_t>(d_imgs), out = reinterpret_cast<uintptr_t>(d_feats);
            const PdlRange r = {in, in + (size_t)n * CNNACC_FEAT_BYTES, out, out + (size_t)n * CNNACC_FEAT_BYTES};
            const int64_t seq_now = g_pdl_seq.load(), seq_mine = ++g_pdl_seq;
            pdl_wait = h->pdl.decide(r, n, h->sm_count, reinterpret_cast<uintptr_t>(stream), h->launches, seq_now, seq_mine);
        } else {
            h->pdl.reset();
        }
        int rc = launch_fused(h->fused, stream, d_imgs, n, d_feats, h->shifts, h->sm_count,
                              (flags & CNNACC_FLAG_KEEP_MAPS) ? d_l0 : nullptr,
                              (flags & CNNACC_FLAG_KEEP_MAPS) ? d_l1 : nullptr, nullptr, pdl_wait);
        h->launches++;
        if (rc != 0) return fail(h, CNNACC_ERR_CUDA, std::string("fused launch: ") + cudaGetErrorString((cudaError_t)rc));
        return 0;
    }
    if (path == ConvPath::kFusedWindows) {
        // larger images: overlapping 128x128 windows through the fused kernel (tiling.cuh)
        const TilePlan py = make_tile_plan(H / 8), px = make_tile_plan(W / 8);
        const int64_t n_t = n * py.n * px.n;
        if (n_t > 0x7fffffff) return fail(h, CNNACC_ERR_ARG, "too many tiles in one chunk");
        // the fused kernel reads each window straight out of the big image (TMA box at the window origin, zero fill beyond
        // the image border) and its epilogue stores the outputs the window computes exactly straight into d_feats
        CUtensorMap map;
        int rc = fused_encode_map(d_imgs, n, &map, H, W);
        if (rc == 0) {
            FusedWindows win;
            win.ntx = px.n; win.nty = py.n; win.ho = H / 8; win.wo = W / 8; win.gx = px.g; win.gy = py.g;
            rc = launch_fused_map(h->fused, stream, map, n_t, d_feats, h->shifts, h->sm_count, nullptr, nullptr, &win);
        }
        if (rc != 0) return fail(h, CNNACC_ERR_CUDA, std::string("fused launch (windows): ") + cudaGetErrorString((cudaError_t)rc));
        h->launches += 1;
        return 0;
    }
    int rc;
    if ((rc = launch_direct_layer(h, stream, 0, d_imgs, d_l0, n, H, W))) return rc;
    if ((rc = launch_direct_layer(h, stream, 1, d_l0, d_l1, n, H / 2, W / 2))) return rc;
    if ((rc = launch_direct_layer(h, stream, 2, d_l1, d_feats, n, H / 4, W / 4))) return rc;
    return 0;
}

bool needs_maps(int H, int W, uint32_t flags) {   // only the per-layer path has intermediate maps in HBM
    return conv_path(H, W, flags) == ConvPath::kPerLayer || (flags & CNNACC_FLAG_KEEP_MAPS);
}

// images per chunk so that the per-layer workspaces stay around 512 MiB
int64_t chunk_images(int H, int W) {
    const size_t per = (size_t)H * W * 8;
    return (int64_t)std::max<size_t>(1, ((size_t)512 << 20) / per);
}

int ensure_maps(cnnacc_handle* h, int64_t n, int H, int W) {
    int rc;
    // per-layer path: the two intermediate maps
    if ((rc = grow(h, h->d_l0, (size_t)n * 16 * (H / 2) * (W / 2)))) return rc;
    if ((rc = grow(h, h->d_l1, (size_t)n * 32 * (H / 4) * (W / 4)))) return rc;
    return 0;
}

TailArgs make_tail(const cnnacc_handle* h, float* d_probs, int32_t* d_cls, int32_t* d_bbox, bool cls_given, uint32_t flags) {
    TailArgs A;
    A.fc_w = h->d_fcw.p; A.fc_b = h->d_fcb.p; A.n_cls = h->n_cls;
    A.want_logits = (flags & CNNACC_FLAG_LOGITS) ? 1 : 0;
    A.probs = d_probs; A.bbox_out = d_bbox;
    A.cls_out = cls_given ? nullptr : d_cls;
    A.cls_in = cls_given ? d_cls : nullptr;
    return A;
}

// classify_vec + bbox_vec on n device-resident feature maps that `maps` fetches (tail.cuh); attr_set: the handle's flag of
// this kernel instance's shared-memory attribute
template <class Maps>
int launch_tail_kernel(cnnacc_handle* h, cudaStream_t stream, const Maps& maps, int64_t n, const TailArgs& A, bool& attr_set) {
    if (n == 0) return 0;
    if (!attr_set) {
        CU(h, cudaFuncSetAttribute(classify_bbox_kernel<Maps>, cudaFuncAttributeMaxDynamicSharedMemorySize, kTailSmem));
        attr_set = true;
    }
    const unsigned grid = (unsigned)std::min<int64_t>((n + kTailGroups - 1) / kTailGroups, h->sm_count);
    classify_bbox_kernel<Maps><<<grid, kTailGroups * kTailThreads, kTailSmem, stream>>>(maps, (long long)n, A);
    h->launches++;
    CU(h, cudaGetLastError());
    return 0;
}
// ... on n compact 16 KiB maps
int launch_tail(cnnacc_handle* h, cudaStream_t stream, const uint8_t* d_feats, int64_t n, const TailArgs& A) {
    return launch_tail_kernel(h, stream, CompactMaps{d_feats}, n, A, h->tail_attr_set);
}

// Conv stack + tail for m device-resident 128x128 images on `stream`.  The fused kernel's tail warps produce the
// predictions while the features are still in shared memory; d_feat_ws (m x 16 KiB) is written only when the caller needs
// the features afterwards (want_feats) or the per-layer kernels are in use.
int infer_device(cnnacc_handle* h, cudaStream_t stream, const uint8_t* d_imgs, int64_t m, uint8_t* d_feat_ws, bool want_feats,
                 const TailArgs& A, uint32_t flags) {
    if (tail_in_conv(flags)) {
        int rc = launch_fused(h->fused, stream, d_imgs, m, want_feats ? d_feat_ws : nullptr, h->shifts, h->sm_count, nullptr, nullptr, &A);
        h->launches++;
        if (rc != 0) return fail(h, CNNACC_ERR_CUDA, std::string("fused launch: ") + cudaGetErrorString((cudaError_t)rc));
        return 0;
    }
    int rc;
    if ((rc = conv_stack_device(h, stream, d_imgs, m, CNNACC_IMG, CNNACC_IMG, d_feat_ws, flags, h->d_l0.p, h->d_l1.p))) return rc;
    return launch_tail(h, stream, d_feat_ws, m, A);
}
bool infer_needs_feat_ws(bool want_feats, uint32_t flags) {
    return want_feats || !tail_in_conv(flags);
}

// Classifier.get_cam_bbox per image (cam_upsampled.cuh); d_cam may be null
int launch_cam_upsampled(cnnacc_handle* h, cudaStream_t stream, const uint8_t* d_feats, int64_t n, const int32_t* d_cls,
                         int32_t* d_bbox, uint8_t* d_cam) {
    if (n == 0) return 0;
    static const ResampleTab tab = make_resample_tab();
    cam_bbox_upsampled_kernel<<<(unsigned)n, 256, 0, stream>>>(d_feats, h->d_fcw.p, h->n_cls, d_cls, d_bbox, d_cam, tab);
    h->launches++;
    CU(h, cudaGetLastError());
    return 0;
}

// realtime_detect.py:582-591 for n frames already on the device (preprocess.cuh)
int launch_preprocess(cnnacc_handle* h, cudaStream_t stream, const uint8_t* d_frames, int64_t n, int fh, int fw, uint8_t* d_gray) {
    if (n == 0) return 0;
    const int S = std::min(fh, fw);
    if (S != h->prep_side) {
        CU(h, cudaDeviceSynchronize());                  // nothing in flight may still be reading the old table
        h->prep_tab = make_area_tab(S);
        const size_t na = h->prep_tab.alpha.size();
        int rc;
        if ((rc = grow(h, h->d_prep_start, kPrepOut)) || (rc = grow(h, h->d_prep_cnt, kPrepOut)) || (rc = grow(h, h->d_prep_alpha, na)))
            return rc;
        CU(h, cudaMemcpy(h->d_prep_start.p, h->prep_tab.start.data(), kPrepOut * sizeof(int), cudaMemcpyHostToDevice));
        CU(h, cudaMemcpy(h->d_prep_cnt.p, h->prep_tab.cnt.data(), kPrepOut * sizeof(int), cudaMemcpyHostToDevice));
        CU(h, cudaMemcpy(h->d_prep_alpha.p, h->prep_tab.alpha.data(), na * sizeof(float), cudaMemcpyHostToDevice));
        h->prep_side = S;
    }
    PrepParams P;
    P.frames = d_frames; P.out = d_gray;
    P.start = h->d_prep_start.p; P.cnt = h->d_prep_cnt.p; P.alpha = h->d_prep_alpha.p;
    P.fh = fh; P.fw = fw;
    P.x0 = fw > fh ? (fw - fh) / 2 : 0;                  // realtime_detect.py:583-589
    P.y0 = fh > fw ? (fh - fw) / 2 : 0;
    P.mode = h->prep_tab.mode; P.k = h->prep_tab.k; P.taps = h->prep_tab.taps; P.inv = h->prep_tab.inv;
    for (int64_t i0 = 0; i0 < n; i0 += 65535) {          // gridDim.y limit
        const int64_t m = std::min<int64_t>(65535, n - i0);
        P.frames = d_frames + (size_t)i0 * fh * fw * 3; P.out = d_gray + (size_t)i0 * kPrepOut * kPrepOut;
        preprocess_bgr_kernel<<<dim3(kPrepOut / kPrepRowsPerCta, (unsigned)m), kPrepOut, 0, stream>>>(P);
        h->launches++;
    }
    CU(h, cudaGetLastError());
    return 0;
}

// A fused launch whose internal waits timed out reports it through a device status word.
int check_fused_status(cnnacc_handle* h) {
    int bits = 0;
    int e = fused_poll_status(h->fused, &bits);
    if (e) return fail(h, CNNACC_ERR_CUDA, std::string("status readback: ") + cudaGetErrorString((cudaError_t)e));
    if (bits) return fail(h, CNNACC_ERR_CUDA, "fused kernel pipeline timeout, status bits " + std::to_string(bits));
    return 0;
}

int check_ready(cnnacc_handle* h) {
    if (!h) return CNNACC_ERR_ARG;
    if (!h->weights_loaded) return fail(h, CNNACC_ERR_STATE, "weights not loaded (call cnnacc_load_weights)");
    return 0;
}

// Waits for the handle's stream and the three ring streams.
int sync_all(cnnacc_handle* h) {
    CU(h, cudaStreamSynchronize(h->stream));
    for (const Stream* st : {&h->st_h2d, &h->st_k, &h->st_d2h}) CU(h, cudaStreamSynchronize(*st));
    return 0;
}

// One host-pointer call on the staging ring, the one place the ring's protocol is written.  kSlots slots are driven through
// one stream per engine (st_h2d copies in, st_k runs the kernels, st_d2h copies out) so that copies in both directions and
// kernels of different chunks overlap.  Each chunk takes its slot through
//   acquire   reserve the buffers; st_h2d waits for ev_out, i.e. until the slot's previous chunk is done with it
//   staged    after the copies in: ev_in on st_h2d, st_k waits for it
//   computed  after the kernels: ev_k on st_k, st_d2h waits for it (calls that copy nothing out per slot skip it)
//   released  ev_out on the stream of the last operation that reads or writes the slot
// The call queues copies that read and write the CALLER's buffers: until finish() or done() ends it, the destructor drains
// the ring's streams, so a call that returns early with an error leaves none of those copies in flight.
struct HostCall {
    cnnacc_handle* const h;
    const bool pipelined;       // cnnacc_run_batch_async: the call continues the ring where the previous one left it, and
    const int64_t ring0;        // a slot's last user may be an earlier call still in flight
    int64_t ci = 0;             // chunks acquired so far
    bool armed = true;

    explicit HostCall(cnnacc_handle* h_, bool pipelined_ = false)
        : h(h_), pipelined(pipelined_), ring0(pipelined_ ? h_->ring_ci : 0) {}
    ~HostCall() { if (armed) for (const Stream* st : {&h->st_h2d, &h->st_k, &h->st_d2h}) cudaStreamSynchronize(*st); }
    // a synchronous call starts on an idle handle (the ring is idle already unless asynchronous calls are pending)
    int begin() { return sync_all(h); }
    // the call's last operation is queued on `st`: wait for it and end the call; `fused`: the call ran the conv stack
    int finish(cudaStream_t st, bool fused) { CU(h, cudaStreamSynchronize(st)); return done(fused); }
    // end a call that has waited for its last operation already, or leaves it in flight on purpose (asynchronous calls)
    int done(bool fused) { armed = false; return fused ? check_fused_status(h) : 0; }

    // the call's next slot, with room for in_bytes / out_bytes and for the classes and boxes of n_pred units
    int acquire(Slot*& out, size_t in_bytes, size_t out_bytes, size_t n_pred = 0) {
        Slot& s = h->slots[(ring0 + ci) % kSlots];
        int rc;
        if ((rc = grow(h, s.d_in, in_bytes)) || (rc = grow(h, s.d_out, out_bytes)) || (rc = grow(h, s.d_cls, n_pred)) ||
            (rc = grow(h, s.d_bbox, n_pred * 4)))
            return rc;
        if ((ci >= kSlots || pipelined) && (rc = wait_released(s, h->st_h2d))) return rc;   // an unrecorded event is complete
        ci++;
        if (pipelined) h->ring_ci = (ring0 + ci) % kSlots;
        out = &s;
        return 0;
    }
    int wait_released(const Slot& s, cudaStream_t st) { CU(h, cudaStreamWaitEvent(st, s.ev_out, 0)); return 0; }
    int staged(const Slot& s) { CU(h, cudaEventRecord(s.ev_in, h->st_h2d)); CU(h, cudaStreamWaitEvent(h->st_k, s.ev_in, 0)); return 0; }
    int computed(const Slot& s) { CU(h, cudaEventRecord(s.ev_k, h->st_k)); CU(h, cudaStreamWaitEvent(h->st_d2h, s.ev_k, 0)); return 0; }
    int released(const Slot& s, cudaStream_t st) { CU(h, cudaEventRecord(s.ev_out, st)); return 0; }
};

// The predictions of a host-pointer call come back in blocks of up to kPredSuper units.  The kernels write the block of units
// [s0, s0 + m) into h->d_pred as [bbox m x 4 i32 | probs m x nc f32 | cls m i32]; flush() brings it with one D2H into the
// pinned h->h_pred, then with plain memcpy into the caller's (usually pageable) arrays.  Copying straight into pageable
// memory would make every cudaMemcpyAsync synchronous and stall the H2D ring behind each chunk's kernels
// (tools/host_fed_probe.py).
struct PredBlock {
    cnnacc_handle* const h;
    int64_t s0 = 0, m = 0;

    explicit PredBlock(cnnacc_handle* h_) : h(h_) {}
    // lay the block out for units [first, first + count), growing the handle's two buffers when they are too small
    int start(int64_t first, int64_t count) {
        const size_t bytes = (size_t)count * kPredBytesPerImage;
        if (bytes > h->d_pred.cap || bytes > h->h_pred.cap) {
            CU(h, cudaStreamSynchronize(h->st_d2h));
            int rc;
            if ((rc = grow(h, h->d_pred, bytes)) || (rc = grow(h, h->h_pred, bytes))) return rc;
        }
        s0 = first; m = count;
        return 0;
    }
    int64_t end() const { return s0 + m; }
    size_t off_probs() const { return (size_t)m * 16; }
    size_t off_cls() const { return off_probs() + (size_t)m * h->n_cls * 4; }
    // where the kernels write the predictions of unit u, s0 <= u < end()
    int32_t* bbox(int64_t u) const { return reinterpret_cast<int32_t*>(h->d_pred.p) + (u - s0) * 4; }
    float* probs(int64_t u) const { return reinterpret_cast<float*>(h->d_pred.p + off_probs()) + (u - s0) * h->n_cls; }
    int32_t* cls(int64_t u) const { return reinterpret_cast<int32_t*>(h->d_pred.p + off_cls()) + (u - s0); }
    // the block, after the kernels queued on `st`, into the caller's arrays (indexed from unit 0); waits for st
    int flush(cudaStream_t st, float* probs_out, int32_t* cls_out, int32_t* bbox_out, bool cls_given) {
        CU(h, cudaMemcpyAsync(h->h_pred.p, h->d_pred.p, off_cls() + (size_t)m * 4, cudaMemcpyDeviceToHost, st));
        CU(h, cudaStreamSynchronize(st));
        if (bbox_out) std::memcpy(bbox_out + s0 * 4, h->h_pred.p, (size_t)m * 16);
        if (probs_out) std::memcpy(probs_out + s0 * h->n_cls, h->h_pred.p + off_probs(), (size_t)m * h->n_cls * 4);
        if (cls_out && !cls_given) std::memcpy(cls_out + s0, h->h_pred.p + off_cls(), (size_t)m * 4);
        return 0;
    }
};

// The host-pointer conv stack: queue the staged copies and kernels of one call on the ring; does not wait for anything.  A
// pipelined call has no ramped chunk sizes: the neighbouring calls keep both copy directions busy at its edges.
int enqueue_host_batch(HostCall& call, const uint8_t* imgs, int64_t n, int H, int W, uint8_t* feats, uint32_t flags) {
    cnnacc_handle* h = call.h;
    int rc;
    const size_t in_sz = (size_t)H * W, out_sz = (size_t)64 * (H / 8) * (W / 8);
    const HostChunkPlan plan = make_host_chunk_plan(n, in_sz, chunk_images(H, W), call.pipelined);
    const int64_t hchunk = plan.full;
    if (needs_maps(H, W, flags) && (rc = ensure_maps(h, hchunk, H, W))) return rc;
    if (call.pipelined) {
        // earlier calls may still be using the slots: growing one (free + malloc) waits for the device first
        bool grows = false;
        for (const Slot& s : h->slots) grows |= s.d_in.cap < hchunk * in_sz || s.d_out.cap < hchunk * out_sz;
        if (grows) CU(h, cudaDeviceSynchronize());
    }
    int64_t m = 0;
    for (int64_t i0 = 0, ci = 0; i0 < n; i0 += m, ci++) {
        m = plan.next(i0, ci);
        Slot* s;
        if ((rc = call.acquire(s, hchunk * in_sz, hchunk * out_sz))) return rc;
        CU(h, cudaMemcpyAsync(s->d_in.p, imgs + i0 * in_sz, m * in_sz, cudaMemcpyHostToDevice, h->st_h2d));
        if ((rc = call.staged(*s)) || (rc = conv_stack_device(h, h->st_k, s->d_in.p, m, H, W, s->d_out.p, flags, h->d_l0.p, h->d_l1.p)) ||
            (rc = call.computed(*s)))
            return rc;
        CU(h, cudaMemcpyAsync(feats + i0 * out_sz, s->d_out.p, m * out_sz, cudaMemcpyDeviceToHost, h->st_d2h));
        if ((rc = call.released(*s, h->st_d2h))) return rc;
    }
    return 0;
}

// ---- sharded host-batch calls (cnnacc_*_sharded, shard_plan.h) ----------------------------------------------------------

// Checked on the calling thread before any member starts work: the member array, the flags, and that every member computes the
// same function as member 0 (members that silently disagreed would make a prediction depend on which shard its image fell
// in).  Returns 0 or a code; *bad = the index of the member concerned (its cnnacc_last_error holds the text), -1 for none.
int check_members(cnnacc_handle* const* hs, int n_handles, uint32_t flags, bool predictions, int* bad) {
    *bad = -1;
    if (!hs || n_handles < 1) return CNNACC_ERR_ARG;
    for (int i = 0; i < n_handles; i++) {
        *bad = i;
        if (!hs[i]) return CNNACC_ERR_ARG;
        for (int j = 0; j < i; j++)
            if (hs[j] == hs[i])
                return fail(hs[i], CNNACC_ERR_ARG, "sharded call: members " + std::to_string(j) + " and " + std::to_string(i) +
                                                       " are the same handle (one handle is used by one thread only)");
    }
    *bad = 0;
    if (flags & (CNNACC_FLAG_DEVICE_PTRS | CNNACC_FLAG_KEEP_MAPS))
        return fail(hs[0], CNNACC_ERR_ARG, "sharded call: CNNACC_FLAG_DEVICE_PTRS / CNNACC_FLAG_KEEP_MAPS have no sharded form");
    const cnnacc_handle* h0 = hs[0];
    for (int i = 0; i < n_handles; i++) {
        cnnacc_handle* h = hs[i];
        const std::string who = "sharded call: member " + std::to_string(i);
        *bad = i;
        if (!h->weights_loaded) return fail(h, CNNACC_ERR_STATE, who + ": weights not loaded (call cnnacc_load_weights)");
        if (predictions && !h->fc_loaded) return fail(h, CNNACC_ERR_STATE, who + ": classifier not loaded (call cnnacc_load_classifier)");
        if (std::memcmp(h->wbin, h0->wbin, CNNACC_WEIGHT_BYTES) != 0) return fail(h, CNNACC_ERR_ARG, who + ": weights differ from member 0's");
        if (std::memcmp(h->shifts, h0->shifts, sizeof(h->shifts)) != 0) return fail(h, CNNACC_ERR_ARG, who + ": shifts differ from member 0's");
        if (h->acc24 != h0->acc24) return fail(h, CNNACC_ERR_ARG, who + ": accumulator bits differ from member 0's");
        if (predictions && (h->n_cls != h0->n_cls || std::memcmp(h->fcw_host, h0->fcw_host, (size_t)h->n_cls * 1024 * sizeof(float)) != 0 ||
                            std::memcmp(h->fcb_host, h0->fcb_host, (size_t)h->n_cls * sizeof(float)) != 0))
            return fail(h, CNNACC_ERR_ARG, who + ": classifier differs from member 0's");
    }
    *bad = -1;
    return 0;
}

// One sharded call: checks, then run(h, lo, hi) -- the member's own single-handle call on units [lo, hi) -- for every shard of
// the plan: shard 0 on the calling thread, shards 1 .. m-1 on a thread each, joined before it returns, so every started
// shard runs to completion and each member handle is used by exactly one thread.  `args_ok`: the pointers are usable and
// `unit_bytes` means something (otherwise member 0 alone runs the call, which reports the bad argument).  Returns the code
// of the lowest-index failing member and stores its index in *failed (-1: success, or no member to blame).
template <class Run>
int run_sharded(cnnacc_handle* const* hs, int n_handles, int64_t n, int64_t unit_bytes, bool args_ok, uint32_t flags,
                bool predictions, int* failed, Run run) {
    int bad = -1;
    int rc = check_members(hs, n_handles, flags, predictions, &bad);
    if (!rc && n < 0) { bad = 0; rc = fail(hs[0], CNNACC_ERR_ARG, "sharded call: negative n"); }
    if (!rc && n > 0 && !args_ok) { bad = 0; rc = fail(hs[0], CNNACC_ERR_ARG, "sharded call: bad size or NULL input / output pointer"); }
    if (!rc) {
        const ShardPlan plan = make_shard_plan(n, n_handles, unit_bytes);
        std::vector<int> rcs(plan.m, CNNACC_OK);
        std::vector<std::thread> workers;
        workers.reserve(plan.m);
        for (int i = 1; i < plan.m; i++) {
            try {
                workers.emplace_back([&, i] { rcs[i] = run(hs[i], plan.begin(i), plan.begin(i + 1)); });
            } catch (const std::system_error& e) {
                rcs[i] = fail(hs[i], CNNACC_ERR_CUDA, std::string("sharded call: could not start the member's thread: ") + e.what());
            }
        }
        rcs[0] = run(hs[0], plan.begin(0), plan.begin(1));
        for (auto& t : workers) t.join();
        for (int i = plan.m - 1; i >= 0; i--)
            if (rcs[i]) { rc = rcs[i]; bad = i; }
    }
    if (failed) *failed = rc ? bad : -1;
    return rc;
}

}  // namespace

extern "C" {

int cnnacc_create(int device_id, cnnacc_handle** out) {
    if (!out) return fail(nullptr, CNNACC_ERR_ARG, "out is NULL");
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return fail(nullptr, CNNACC_ERR_CUDA, std::string("no CUDA device: ") + cudaGetErrorString(e) +
                                                  " (this library has no CPU fallback)");
    if (device_id < 0 || device_id >= count) return fail(nullptr, CNNACC_ERR_ARG, "device_id out of range");
    // on a failed step the handle is deleted with whatever it holds so far, device_id being current
    std::unique_ptr<cnnacc_handle> h(new cnnacc_handle());
    h->device = device_id;
    auto bail = [&](const char* what, cudaError_t err) {
        g_create_error = std::string(what) + ": " + cudaGetErrorString(err);
        return CNNACC_ERR_CUDA;
    };
    if ((e = cudaSetDevice(device_id)) != cudaSuccess) return bail("cudaSetDevice", e);
    cudaDeviceProp prop;
    if ((e = cudaGetDeviceProperties(&prop, device_id)) != cudaSuccess) return bail("cudaGetDeviceProperties", e);
    if (prop.major != 10) {
        g_create_error = "device is sm_" + std::to_string(prop.major * 10 + prop.minor) +
                         "; this library is built for sm_100a (B200) only";
        return CNNACC_ERR_CUDA;
    }
    h->sm_count = prop.multiProcessorCount;
    if ((e = h->own_stream.create(cudaStreamNonBlocking)) != cudaSuccess) return bail("cudaStreamCreate", e);
    h->stream = h->own_stream;
    for (Event* ev : {&h->ev_t0, &h->ev_t1, &h->ev_a, &h->ev_b, &h->ev_done})
        if ((e = ev->create(cudaEventDefault)) != cudaSuccess) return bail("cudaEventCreate", e);
    for (auto& s : h->slots) {
        for (Event* ev : {&s.ev_in, &s.ev_k, &s.ev_out})
            if ((e = ev->create(cudaEventDisableTiming)) != cudaSuccess) return bail("cudaEventCreate", e);
    }
    for (auto& ev : h->ev_ticket)
        if ((e = ev.create(cudaEventDisableTiming)) != cudaSuccess) return bail("cudaEventCreate", e);
    for (auto& b : h->rdesc)
        if ((e = b.ev.create(cudaEventDisableTiming)) != cudaSuccess) return bail("cudaEventCreate", e);
    for (Stream* st : {&h->st_h2d, &h->st_k, &h->st_d2h})
        if ((e = st->create(cudaStreamNonBlocking)) != cudaSuccess) return bail("cudaStreamCreate", e);
    int rc;
    if ((rc = grow(nullptr, h->h_img, CNNACC_IMG * CNNACC_IMG)) || (rc = grow(nullptr, h->h_bram, kBramBytes)) ||
        (rc = grow(nullptr, h->h_done, 64 / sizeof(int))) || (rc = grow(nullptr, h->h_pred, kSmallN * kPredBytesPerImage)) ||
        (rc = grow(nullptr, h->d_pred, kSmallN * kPredBytesPerImage)) || (rc = grow(nullptr, h->d_img1, CNNACC_IMG * CNNACC_IMG)) ||
        (rc = grow(nullptr, h->d_bram, kBramBytes)))
        return rc;
    if ((e = cudaHostGetDevicePointer(&h->h_img_dev, h->h_img.p, 0)) != cudaSuccess) return bail("cudaHostGetDevicePointer", e);
    if ((e = cudaHostGetDevicePointer(&h->h_bram_dev, h->h_bram.p, 0)) != cudaSuccess) return bail("cudaHostGetDevicePointer", e);
    *h->h_done.p = 0;
    if ((e = cudaHostGetDevicePointer(&h->h_done_dev, h->h_done.p, 0)) != cudaSuccess) return bail("cudaHostGetDevicePointer", e);
    *out = h.release();
    return CNNACC_OK;
}

int cnnacc_destroy(cnnacc_handle* h) {
    if (!h) return CNNACC_ERR_ARG;
    cudaSetDevice(h->device);
    cudaDeviceSynchronize();
    delete h;
    return CNNACC_OK;
}

int cnnacc_set_stream(cnnacc_handle* h, void* cuda_stream) {
    if (!h) return CNNACC_ERR_ARG;
    h->stream = cuda_stream ? (cudaStream_t)cuda_stream : h->own_stream;
    return CNNACC_OK;
}

const char* cnnacc_last_error(const cnnacc_handle* h) { return h ? h->err.c_str() : g_create_error.c_str(); }
int64_t cnnacc_launch_count(const cnnacc_handle* h) { return h ? h->launches : 0; }

int cnnacc_load_weights(cnnacc_handle* h, const uint8_t* weights_bin, size_t n) {
    if (!h || !weights_bin) return fail(h, CNNACC_ERR_ARG, "NULL argument");
    if (n != CNNACC_WEIGHT_BYTES)
        return fail(h, CNNACC_ERR_ARG, "Expected 23184 weights, got " + std::to_string(n));   // pynq_inference.py:189
    h->weights_loaded = false;           // a reload that fails partway leaves a handle that refuses calls
    CU(h, cudaSetDevice(h->device));
    CU(h, cudaDeviceSynchronize());      // weights may be in use by queued launches
    std::memcpy(h->wbin, weights_bin, n);
    std::vector<uint32_t> packed;
    pack_direct_weights(h->wbin, packed, h->wdirect_off);
    int rc;
    if ((rc = grow(h, h->d_wdirect, packed.size()))) return rc;
    CU(h, cudaMemcpy(h->d_wdirect.p, packed.data(), packed.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
    rc = fused_load_weights(h->fused, h->wbin);
    if (rc != 0) return fail(h, CNNACC_ERR_CUDA, std::string("fused_load_weights: ") + cudaGetErrorString((cudaError_t)rc));
    h->weights_loaded = true;
    return CNNACC_OK;
}

int cnnacc_set_shifts(cnnacc_handle* h, int s0, int s1, int s2) {
    if (!h) return CNNACC_ERR_ARG;
    const int s[3] = {s0, s1, s2};
    for (int v : s)
        if (v < 0 || v > 31) return fail(h, CNNACC_ERR_ARG, "shift outside 0..31: " + std::to_string(v));
    std::memcpy(h->shifts, s, sizeof(s));
    return CNNACC_OK;
}

int cnnacc_set_accumulator_bits(cnnacc_handle* h, int bits) {
    if (!h) return CNNACC_ERR_ARG;
    if (bits != 24 && bits != 32) return fail(h, CNNACC_ERR_ARG, "accumulator width must be 32 (arm_cnn.c) or 24 (RTL / train_cnn.py)");
    h->acc24 = h->fused.acc24 = (bits == 24);
    return CNNACC_OK;
}

int cnnacc_get_accumulator_bits(const cnnacc_handle* h) { return h ? (h->acc24 ? 24 : 32) : CNNACC_ERR_ARG; }

int cnnacc_pack_weights_host(const uint8_t* weights_bin, size_t n, uint32_t* w0, uint8_t* b1, uint8_t* b2) {
    if (!weights_bin || !w0 || !b1 || !b2 || n != CNNACC_WEIGHT_BYTES) return CNNACC_ERR_ARG;
    static_assert(CNNACC_PACK_B1_BYTES == kB1Bytes && CNNACC_PACK_B2_BYTES == kB2Bytes, "header out of date");
    fused_pack_weights(weights_bin, reinterpret_cast<uint32_t(*)[6]>(w0), reinterpret_cast<uint32_t(*)[32]>(w0 + 96), b1, b2);
    return CNNACC_OK;
}

int cnnacc_pdl_chain_host(int n_launches, const uint64_t* ranges, const int64_t* n_images, const int32_t* stream_id,
                          const int32_t* foreign_before, int sm_count, int32_t* wait_out) {
    if (n_launches < 0 || !ranges || !n_images || !stream_id || !foreign_before || !wait_out || sm_count < 1) return CNNACC_ERR_ARG;
    PdlChain chain;
    int64_t launches = 0, seq = 0;
    for (int i = 0; i < n_launches; i++) {
        if (foreign_before[i] & 1) launches++;          // another kernel of the same handle in between
        if (foreign_before[i] & 2) seq++;               // a conv-stack launch of another handle in between
        const PdlRange r = {(uintptr_t)ranges[4 * i], (uintptr_t)ranges[4 * i + 1], (uintptr_t)ranges[4 * i + 2], (uintptr_t)ranges[4 * i + 3]};
        const int64_t seq_now = seq, seq_mine = ++seq;
        wait_out[i] = chain.decide(r, n_images[i], sm_count, (uintptr_t)stream_id[i], launches, seq_now, seq_mine);
        launches++;
    }
    return CNNACC_OK;
}

int cnnacc_chunk_plan_host(int64_t n, int H, int W, int pipelined, int64_t* sizes, int cap) {
    if (n < 1 || !valid_hw(H, W) || !sizes || cap < 1) return CNNACC_ERR_ARG;
    const HostChunkPlan plan = make_host_chunk_plan(n, (size_t)H * W, chunk_images(H, W), pipelined != 0);
    int count = 0;
    for (int64_t i0 = 0; i0 < n; count++) {
        const int64_t m = plan.next(i0, count);
        if (count >= cap) return CNNACC_ERR_ARG;
        sizes[count] = m;
        i0 += m;
    }
    return count;
}

int cnnacc_tile_plan_host(int n_out, int* origin, int* first, int* end, int cap) {
    if (n_out < 16 || n_out > 1024 || !origin || !first || !end) return CNNACC_ERR_ARG;
    const TilePlan p = make_tile_plan(n_out);
    if (p.n > cap) return CNNACC_ERR_ARG;
    for (int i = 0; i < p.n; i++) { origin[i] = p.g[i]; first[i] = p.s[i]; end[i] = p.e[i]; }
    return p.n;
}

int cnnacc_get_shifts(const cnnacc_handle* h, int* s3) {
    if (!h || !s3) return CNNACC_ERR_ARG;
    std::memcpy(s3, h->shifts, sizeof(h->shifts));
    return CNNACC_OK;
}

int cnnacc_run_batch(cnnacc_handle* h, const uint8_t* imgs, int64_t n, int H, int W, uint8_t* feats, uint32_t flags) {
    int rc;
    if ((rc = check_ready(h))) return rc;
    if (n < 0 || !valid_hw(H, W)) return fail(h, CNNACC_ERR_ARG, "bad n / H / W (H, W must be multiples of 16)");
    if (n == 0) return CNNACC_OK;
    if (!imgs || !feats) return fail(h, CNNACC_ERR_ARG, "NULL image / feature pointer");
    CU(h, cudaSetDevice(h->device));
    const size_t in_sz = (size_t)H * W, out_sz = (size_t)64 * (H / 8) * (W / 8);
    const bool maps = needs_maps(H, W, flags);
    const int64_t chunk = maps ? std::min<int64_t>(n, chunk_images(H, W)) : n;

    if (flags & CNNACC_FLAG_DEVICE_PTRS) {
        REQUIRE_ALIGNED(h, imgs, 16, "image");
        REQUIRE_ALIGNED(h, feats, 16, "feature");
        if (maps && (rc = ensure_maps(h, chunk, H, W))) return rc;
        for (int64_t i0 = 0; i0 < n; i0 += chunk) {
            const int64_t m = std::min(chunk, n - i0);
            if ((rc = conv_stack_device(h, h->stream, imgs + i0 * in_sz, m, H, W, feats + i0 * out_sz, flags, h->d_l0.p, h->d_l1.p)))
                return rc;
        }
        return CNNACC_OK;
    }

    // host pointers: returns when feats is complete
    HostCall call(h);
    if ((rc = call.begin()) || (rc = enqueue_host_batch(call, imgs, n, H, W, feats, flags))) return rc;
    return call.finish(h->st_d2h, true);                // the last D2H is the last operation of the whole chain
}

int cnnacc_run_batch_async(cnnacc_handle* h, const uint8_t* imgs, int64_t n, int H, int W, uint8_t* feats, uint32_t flags,
                           int64_t* ticket) {
    int rc;
    if ((rc = check_ready(h))) return rc;
    if (!ticket) return fail(h, CNNACC_ERR_ARG, "ticket is NULL");
    if (n < 0 || !valid_hw(H, W)) return fail(h, CNNACC_ERR_ARG, "bad n / H / W (H, W must be multiples of 16)");
    if (flags & CNNACC_FLAG_DEVICE_PTRS) return fail(h, CNNACC_ERR_ARG, "device-pointer calls are asynchronous already (cnnacc_run_batch)");
    if (n > 0 && (!imgs || !feats)) return fail(h, CNNACC_ERR_ARG, "NULL image / feature pointer");
    // the per-layer kernels share two workspaces between chunks; only the paths without them can overlap calls
    if (needs_maps(H, W, flags)) return fail(h, CNNACC_ERR_ARG, "this size / flag combination has no asynchronous form: use cnnacc_run_batch");
    CU(h, cudaSetDevice(h->device));
    // the event of the call submitted CNNACC_MAX_PENDING calls ago is about to be reused: that call must have completed
    cudaEvent_t ev = h->ev_ticket[h->next_ticket % CNNACC_MAX_PENDING];
    if (h->next_ticket >= CNNACC_MAX_PENDING) CU(h, cudaEventSynchronize(ev));
    HostCall call(h, /*pipelined=*/true);
    if (n > 0 && (rc = enqueue_host_batch(call, imgs, n, H, W, feats, flags))) return rc;
    CU(h, cudaEventRecord(ev, h->st_d2h));
    *ticket = h->next_ticket++;
    return call.done(false);
}

int cnnacc_wait_batch(cnnacc_handle* h, int64_t ticket) {
    if (!h) return CNNACC_ERR_ARG;
    if (ticket < 0 || ticket >= h->next_ticket) return fail(h, CNNACC_ERR_ARG, "unknown ticket");
    CU(h, cudaSetDevice(h->device));
    // calls complete in submission order and an event is reused only after its call has completed
    if (ticket + CNNACC_MAX_PENDING >= h->next_ticket)         // older tickets: their event has been reused, i.e. they are complete
        CU(h, cudaEventSynchronize(h->ev_ticket[ticket % CNNACC_MAX_PENDING]));
    return check_fused_status(h);
}

int cnnacc_load_image(cnnacc_handle* h, const uint8_t* img, size_t n) {
    if (!h || !img) return fail(h, CNNACC_ERR_ARG, "NULL argument");
    if (n != (size_t)CNNACC_IMG * CNNACC_IMG)
        return fail(h, CNNACC_ERR_ARG, "Expected 16384 pixels, got " + std::to_string(n));     // pynq_inference.py:214
    CU(h, cudaSetDevice(h->device));
    if (h->started) CU(h, cudaEventSynchronize(h->ev_done));   // s_axis_tready = !busy (…S00_AXI.v:390)
    std::memcpy(h->h_img.p, img, n);
    h->image_loaded = true;
    return CNNACC_OK;
}

int cnnacc_start(cnnacc_handle* h) {
    int rc;
    if ((rc = check_ready(h))) return rc;
    if (!h->image_loaded) return fail(h, CNNACC_ERR_STATE, "no image loaded (call cnnacc_load_image)");
    CU(h, cudaSetDevice(h->device));
    uint8_t *l0 = h->d_bram.p, *l1 = h->d_bram.p + 16 * 4096, *l2 = l1 + 32 * 1024;
    CU(h, cudaMemcpyAsync(h->d_img1.p, h->h_img.p, CNNACC_IMG * CNNACC_IMG, cudaMemcpyHostToDevice, h->stream));
    if ((rc = conv_stack_device(h, h->stream, h->d_img1.p, 1, CNNACC_IMG, CNNACC_IMG, l2, CNNACC_FLAG_KEEP_MAPS, l0, l1))) return rc;
    CU(h, cudaMemcpyAsync(h->h_bram.p, h->d_bram.p, kBramBytes, cudaMemcpyDeviceToHost, h->stream));
    CU(h, cudaEventRecord(h->ev_done, h->stream));
    h->started = true;
    return CNNACC_OK;
}

int cnnacc_status(cnnacc_handle* h) {
    if (!h) return CNNACC_ERR_ARG;
    if (!h->started) return 0;                               // idle: busy=0 done=0
    cudaError_t e = cudaEventQuery(h->ev_done);
    if (e == cudaSuccess) return 0x2 | (2 << 2);             // done, current_layer = 2
    if (e == cudaErrorNotReady) return 0x1;                  // busy
    return fail(h, CNNACC_ERR_CUDA, std::string("cudaEventQuery: ") + cudaGetErrorString(e));
}

int cnnacc_wait(cnnacc_handle* h, int timeout_us) {
    if (!h) return CNNACC_ERR_ARG;
    if (!h->started) return fail(h, CNNACC_ERR_STATE, "wait without start");
    const auto t0 = std::chrono::steady_clock::now();
    for (;;) {
        cudaError_t e = cudaEventQuery(h->ev_done);
        if (e == cudaSuccess) return CNNACC_OK;
        if (e != cudaErrorNotReady) return fail(h, CNNACC_ERR_CUDA, std::string("cudaEventQuery: ") + cudaGetErrorString(e));
        const auto us = std::chrono::duration_cast<std::chrono::microseconds>(std::chrono::steady_clock::now() - t0).count();
        if (us > timeout_us) return fail(h, CNNACC_ERR_TIMEOUT, "timed out waiting for done");   // fast_readout.c:91
    }
}

int cnnacc_read_feature_map(cnnacc_handle* h, int channel, int num_values, uint8_t* out) {
    if (!h || !out) return fail(h, CNNACC_ERR_ARG, "NULL argument");
    if (!h->started) return fail(h, CNNACC_ERR_STATE, "no inference has been started");
    if (channel < 0 || channel >= CNNACC_BRAM_CHANNELS) return fail(h, CNNACC_ERR_ARG, "channel outside 0..111");
    CU(h, cudaEventSynchronize(h->ev_done));
    size_t off, depth;
    if (channel < 16)      { off = (size_t)channel * 4096;                       depth = 4096; }
    else if (channel < 48) { off = 16 * 4096 + (size_t)(channel - 16) * 1024;    depth = 1024; }
    else                   { off = 16 * 4096 + 32 * 1024 + (size_t)(channel - 48) * 256; depth = 256; }
    if (num_values < 0 || (size_t)num_values > depth) return fail(h, CNNACC_ERR_ARG, "num_values exceeds the channel's BRAM depth");
    { int rc = check_fused_status(h); if (rc) return rc; }
    std::memcpy(out, h->h_bram.p + off, (size_t)num_values);
    return CNNACC_OK;
}

int cnnacc_read_features(cnnacc_handle* h, uint8_t* out, int n_ch, int ch_off) {
    if (!h || !out) return fail(h, CNNACC_ERR_ARG, "NULL argument");
    if (n_ch < 0 || ch_off < 0 || ch_off + n_ch > CNNACC_BRAM_CHANNELS) return fail(h, CNNACC_ERR_ARG, "channel range outside 0..111");
    for (int c = 0; c < n_ch; c++) {                        // read_features_full reads 256 values per channel
        int rc = cnnacc_read_feature_map(h, ch_off + c, 256, out + (size_t)c * 256);
        if (rc) return rc;
    }
    return CNNACC_OK;
}

int cnnacc_infer_one(cnnacc_handle* h, const uint8_t* img, uint8_t* feat, float* conv_ms, float* read_ms) {
    int rc;
    if ((rc = check_ready(h))) return rc;
    if (!img || !feat) return fail(h, CNNACC_ERR_ARG, "NULL argument");
    CU(h, cudaSetDevice(h->device));
    if (h->started) CU(h, cudaEventSynchronize(h->ev_done));
    uint8_t* h_l2 = h->h_bram.p + 16 * 4096 + 32 * 1024;
    const auto t0 = std::chrono::steady_clock::now();
    std::memcpy(h->h_img.p, img, CNNACC_FEAT_BYTES);
    // Zero-copy: the kernel TMA-loads the image straight from mapped pinned host memory and its 16 KiB bulk
    // store lands in mapped pinned host memory -- one launch, one stream sync, no copy-engine round trips.
    if (!h->one_map_ok) {
        if (fused_encode_map(h->h_img_dev, 1, &h->one_map)) return fail(h, CNNACC_ERR_CUDA, "tensor map over the pinned image buffer");
        h->one_map_ok = true;
    }
    uint8_t* l2_dev = h->h_bram_dev + 16 * 4096 + 32 * 1024;
    const int seq = ++h->done_seq;
    rc = launch_fused_map(h->fused, h->stream, h->one_map, 1, l2_dev, h->shifts, h->sm_count, nullptr, nullptr, nullptr, nullptr,
                          h->h_done_dev, seq);
    h->launches++;
    if (rc != 0) return fail(h, CNNACC_ERR_CUDA, std::string("fused launch: ") + cudaGetErrorString((cudaError_t)rc));
    // The kernel stores `seq` into a mapped host word after its feature store has landed: spinning on that word skips the
    // driver's wake-up path of a stream synchronise (~8 us of the ~36).  Bounded: after 2 s fall back to the synchronise.
    {
        const volatile int* flag = h->h_done.p;
        const auto spin0 = std::chrono::steady_clock::now();
        for (unsigned it = 0; *flag != seq; it++) {
#if defined(__x86_64__)
            __builtin_ia32_pause();
#endif
            if ((it & 0xFFFF) == 0xFFFF && std::chrono::steady_clock::now() - spin0 > std::chrono::seconds(2)) {
                CU(h, cudaStreamSynchronize(h->stream));
                break;
            }
        }
    }
    const auto t1 = std::chrono::steady_clock::now();
    std::memcpy(feat, h_l2, CNNACC_FEAT_BYTES);
    if (conv_ms) *conv_ms = std::chrono::duration<float, std::milli>(t1 - t0).count();
    if (read_ms) *read_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t1).count();
    return check_fused_status(h);
}

int cnnacc_load_classifier(cnnacc_handle* h, const float* fc_w, const float* fc_b, int n_cls) {
    if (!h || !fc_w || !fc_b) return fail(h, CNNACC_ERR_ARG, "NULL argument");
    if (n_cls < 1 || n_cls > kMaxClasses) return fail(h, CNNACC_ERR_ARG, "n_cls outside 1..16");
    // The CAM forms w * float(byte) as fma(w, 2^23 + byte, -w * 2^23) (tail.cuh), which is exact as long as w * 2^23 is finite;
    // weights beyond 2^100 (or not finite) make every logit meaningless anyway and are rejected here.
    for (size_t i = 0; i < (size_t)n_cls * 1024; i++)
        if (!(std::fabs(fc_w[i]) < 1.2676506002282294e30f)) return fail(h, CNNACC_ERR_ARG, "classifier weight not finite or |w| >= 2^100");
    CU(h, cudaSetDevice(h->device));
    CU(h, cudaDeviceSynchronize());
    int rc;
    if ((rc = grow(h, h->d_fcw, (size_t)kMaxClasses * 1024)) || (rc = grow(h, h->d_fcb, kMaxClasses))) return rc;
    CU(h, cudaMemcpy(h->d_fcw.p, fc_w, (size_t)n_cls * 1024 * sizeof(float), cudaMemcpyHostToDevice));
    CU(h, cudaMemcpy(h->d_fcb.p, fc_b, n_cls * sizeof(float), cudaMemcpyHostToDevice));
    std::memcpy(h->fcw_host, fc_w, (size_t)n_cls * 1024 * sizeof(float));
    std::memcpy(h->fcb_host, fc_b, n_cls * sizeof(float));
    h->n_cls = n_cls;
    h->fc_loaded = true;
    return CNNACC_OK;
}

// shared body of classify_batch / infer_batch
static int predict_impl(cnnacc_handle* h, const uint8_t* src, int64_t n, bool src_is_images,
                        float* probs, int32_t* cls, int32_t* bbox, uint32_t flags) {
    int rc;
    if (!h) return CNNACC_ERR_ARG;
    if (src_is_images && (rc = check_ready(h))) return rc;
    if (!h->fc_loaded) return fail(h, CNNACC_ERR_STATE, "classifier not loaded (call cnnacc_load_classifier)");
    if (n < 0 || n > 0x7fffffffLL) return fail(h, CNNACC_ERR_ARG, "n outside 0..2^31-1");
    if (n == 0) return CNNACC_OK;
    if (!src) return fail(h, CNNACC_ERR_ARG, "NULL input pointer");
    CU(h, cudaSetDevice(h->device));
    const size_t img_sz = CNNACC_FEAT_BYTES;        // 128*128 image and 64*256 feature map are both 16 KiB
    const int nc = h->n_cls;
    const bool maps = src_is_images && needs_maps(CNNACC_IMG, CNNACC_IMG, flags);
    const bool cls_given = (flags & CNNACC_FLAG_CLS_GIVEN) != 0;
    if (cls_given && !cls) return fail(h, CNNACC_ERR_ARG, "CNNACC_FLAG_CLS_GIVEN without a cls array");
    const bool upsampled = (flags & CNNACC_FLAG_BBOX_UPSAMPLED) != 0 && bbox;
    if (upsampled && !cls && (flags & CNNACC_FLAG_DEVICE_PTRS))
        return fail(h, CNNACC_ERR_ARG, "CNNACC_FLAG_BBOX_UPSAMPLED with device pointers needs a cls array");
    // images in: does anything after the conv stack need the feature maps in HBM?
    const bool feat_ws = src_is_images && infer_needs_feat_ws(upsampled, flags);

    if (flags & CNNACC_FLAG_DEVICE_PTRS) {
        REQUIRE_ALIGNED(h, src, 16, "image / feature");
        REQUIRE_ALIGNED(h, bbox, 16, "bbox");
        REQUIRE_ALIGNED(h, probs, 4, "probs");
        REQUIRE_ALIGNED(h, cls, 4, "cls");
        // one fused launch covers the whole call unless a workspace bounds the chunk
        const int64_t chunk = feat_ws ? std::min<int64_t>(n, 16384) : n;
        if (feat_ws) {
            if ((rc = grow(h, h->d_feat, (size_t)chunk * img_sz))) return rc;
            if (maps && (rc = ensure_maps(h, chunk, CNNACC_IMG, CNNACC_IMG))) return rc;
        }
        for (int64_t i0 = 0; i0 < n; i0 += chunk) {
            const int64_t m = std::min(chunk, n - i0);
            const TailArgs A = make_tail(h, probs ? probs + i0 * nc : nullptr, cls ? cls + i0 : nullptr,
                                         (bbox && !upsampled) ? bbox + i0 * 4 : nullptr, cls_given, flags);
            const uint8_t* f = src + i0 * img_sz;
            if (src_is_images) {
                if ((rc = infer_device(h, h->stream, f, m, h->d_feat.p, upsampled, A, flags))) return rc;
                f = h->d_feat.p;
            } else if ((rc = launch_tail(h, h->stream, f, m, A))) return rc;
            if (upsampled && (rc = launch_cam_upsampled(h, h->stream, f, m, cls + i0, bbox + i0 * 4, nullptr))) return rc;
        }
        return CNNACC_OK;
    }

    HostCall call(h);
    if ((rc = call.begin())) return rc;
    PredBlock pred(h);
    auto kernels = [&](cudaStream_t st, const Slot& s, int64_t i0, int64_t m) -> int {   // units [i0, i0 + m), staged in s
        const TailArgs A = make_tail(h, pred.probs(i0), pred.cls(i0), upsampled ? nullptr : pred.bbox(i0), cls_given, flags);
        const uint8_t* f = s.d_in.p;
        int r;
        if (src_is_images) {
            if ((r = infer_device(h, st, s.d_in.p, m, s.d_out.p, upsampled, A, flags))) return r;
            f = s.d_out.p;
        } else if ((r = launch_tail(h, st, f, m, A))) return r;
        return upsampled ? launch_cam_upsampled(h, st, f, m, pred.cls(i0), pred.bbox(i0), nullptr) : 0;
    };
    Slot* s;
    if (n <= kSmallN) {                                      // latency path: one stream, one result copy
        cudaStream_t st = h->st_k;
        if ((rc = call.acquire(s, n * img_sz, feat_ws ? n * img_sz : 0))) return rc;
        if (maps && (rc = ensure_maps(h, n, CNNACC_IMG, CNNACC_IMG))) return rc;
        if ((rc = pred.start(0, n))) return rc;
        CU(h, cudaMemcpyAsync(s->d_in.p, src, n * img_sz, cudaMemcpyHostToDevice, st));
        if (cls_given) CU(h, cudaMemcpyAsync(pred.cls(0), cls, n * sizeof(int32_t), cudaMemcpyHostToDevice, st));
        if ((rc = kernels(st, *s, 0, n)) || (rc = pred.flush(st, probs, cls, bbox, cls_given))) return rc;
        return call.done(src_is_images);
    }
    // Only the predictions (44 B per image) come back, so the link carries H2D traffic alone: no ramp, and no cap beyond the
    // call's own size.  Nothing is copied out per slot, so a slot is released once its kernels have ended.
    const int64_t hchunk = make_host_chunk_plan(n, img_sz, INT64_MAX, false).full;
    if (maps && (rc = ensure_maps(h, hchunk, CNNACC_IMG, CNNACC_IMG))) return rc;
    for (int64_t s0 = 0; s0 < n; s0 += kPredSuper) {
        if ((rc = pred.start(s0, std::min<int64_t>(kPredSuper, n - s0)))) return rc;
        for (int64_t i0 = s0; i0 < pred.end(); i0 += hchunk) {
            const int64_t m = std::min(hchunk, pred.end() - i0);
            if ((rc = call.acquire(s, hchunk * img_sz, feat_ws ? hchunk * img_sz : 0))) return rc;
            CU(h, cudaMemcpyAsync(s->d_in.p, src + i0 * img_sz, m * img_sz, cudaMemcpyHostToDevice, h->st_h2d));
            if (cls_given) CU(h, cudaMemcpyAsync(pred.cls(i0), cls + i0, m * sizeof(int32_t), cudaMemcpyHostToDevice, h->st_h2d));
            if ((rc = call.staged(*s)) || (rc = kernels(h->st_k, *s, i0, m)) || (rc = call.released(*s, h->st_k))) return rc;
        }
        if ((rc = pred.flush(h->st_k, probs, cls, bbox, cls_given))) return rc;
    }
    return call.done(src_is_images);
}

int cnnacc_classify_batch(cnnacc_handle* h, const uint8_t* feats, int64_t n, float* probs, int32_t* cls, int32_t* bbox, uint32_t flags) {
    return predict_impl(h, feats, n, false, probs, cls, bbox, flags);
}

int cnnacc_infer_batch(cnnacc_handle* h, const uint8_t* imgs, int64_t n, float* probs, int32_t* cls, int32_t* bbox, uint32_t flags) {
    return predict_impl(h, imgs, n, true, probs, cls, bbox, flags);
}

int cnnacc_pool_features(cnnacc_handle* h, const uint8_t* feats, int64_t n, float* pooled, uint32_t flags) {
    int rc;
    if (!h) return CNNACC_ERR_ARG;
    if (n < 0) return fail(h, CNNACC_ERR_ARG, "negative n");
    if (n == 0) return CNNACC_OK;
    if (!feats || !pooled) return fail(h, CNNACC_ERR_ARG, "NULL feature / output pointer");
    CU(h, cudaSetDevice(h->device));
    const size_t feat_sz = CNNACC_FEAT_BYTES, out_sz = 1024 * sizeof(float);
    if (flags & CNNACC_FLAG_DEVICE_PTRS) {
        REQUIRE_ALIGNED(h, feats, 16, "feature");
        REQUIRE_ALIGNED(h, pooled, 16, "pooled");
        pool_features_kernel<<<(unsigned)n, 256, 0, h->stream>>>(feats, pooled);
        h->launches++;
        CU(h, cudaGetLastError());
        return CNNACC_OK;
    }
    HostCall call(h);
    if ((rc = call.begin())) return rc;
    const int64_t hchunk = std::min<int64_t>(n, 2048);
    for (int64_t i0 = 0; i0 < n; i0 += hchunk) {
        const int64_t m = std::min(hchunk, n - i0);
        Slot* s;
        if ((rc = call.acquire(s, hchunk * feat_sz, hchunk * out_sz))) return rc;
        CU(h, cudaMemcpyAsync(s->d_in.p, feats + i0 * feat_sz, m * feat_sz, cudaMemcpyHostToDevice, h->st_h2d));
        if ((rc = call.staged(*s))) return rc;
        pool_features_kernel<<<(unsigned)m, 256, 0, h->st_k>>>(s->d_in.p, reinterpret_cast<float*>(s->d_out.p));
        h->launches++;
        CU(h, cudaGetLastError());
        if ((rc = call.computed(*s))) return rc;
        CU(h, cudaMemcpyAsync(pooled + i0 * 1024, s->d_out.p, m * out_sz, cudaMemcpyDeviceToHost, h->st_d2h));
        if ((rc = call.released(*s, h->st_d2h))) return rc;
    }
    return call.finish(h->st_d2h, false);
}

int cnnacc_cam_bbox_batch(cnnacc_handle* h, const uint8_t* feats, int64_t n, const int32_t* cls, int32_t* bbox, uint8_t* cam,
                          uint32_t flags) {
    int rc;
    if (!h) return CNNACC_ERR_ARG;
    if (!h->fc_loaded) return fail(h, CNNACC_ERR_STATE, "classifier not loaded (call cnnacc_load_classifier)");
    if (n < 0) return fail(h, CNNACC_ERR_ARG, "negative n");
    if (n == 0) return CNNACC_OK;
    if (!feats || !cls || (!bbox && !cam)) return fail(h, CNNACC_ERR_ARG, "NULL feature / class pointer, or nothing to write");
    CU(h, cudaSetDevice(h->device));
    const size_t feat_sz = CNNACC_FEAT_BYTES, cam_sz = (size_t)kCamOut * kCamOut;
    if (flags & CNNACC_FLAG_DEVICE_PTRS) {
        REQUIRE_ALIGNED(h, feats, 16, "feature");
        REQUIRE_ALIGNED(h, bbox, 16, "bbox");
        REQUIRE_ALIGNED(h, cam, 4, "cam");
        REQUIRE_ALIGNED(h, cls, 4, "cls");
        return launch_cam_upsampled(h, h->stream, feats, n, cls, bbox, cam);
    }

    HostCall call(h);
    if ((rc = call.begin())) return rc;
    const int64_t hchunk = std::min<int64_t>(n, 4096);
    for (int64_t i0 = 0; i0 < n; i0 += hchunk) {
        const int64_t m = std::min(hchunk, n - i0);
        Slot* s;
        if ((rc = call.acquire(s, hchunk * feat_sz, cam ? hchunk * cam_sz : 0, hchunk))) return rc;
        CU(h, cudaMemcpyAsync(s->d_in.p, feats + i0 * feat_sz, m * feat_sz, cudaMemcpyHostToDevice, h->st_h2d));
        CU(h, cudaMemcpyAsync(s->d_cls.p, cls + i0, m * sizeof(int32_t), cudaMemcpyHostToDevice, h->st_h2d));
        if ((rc = call.staged(*s)) ||
            (rc = launch_cam_upsampled(h, h->st_k, s->d_in.p, m, s->d_cls.p, bbox ? s->d_bbox.p : nullptr, cam ? s->d_out.p : nullptr)) ||
            (rc = call.computed(*s)))
            return rc;
        if (bbox) CU(h, cudaMemcpyAsync(bbox + i0 * 4, s->d_bbox.p, m * 4 * sizeof(int32_t), cudaMemcpyDeviceToHost, h->st_d2h));
        if (cam)  CU(h, cudaMemcpyAsync(cam + i0 * cam_sz, s->d_out.p, m * cam_sz, cudaMemcpyDeviceToHost, h->st_d2h));
        if ((rc = call.released(*s, h->st_d2h))) return rc;
    }
    return call.finish(h->st_d2h, false);
}

// Pre-processing of m square regions of frames already on the device into d_gray: base.desc = their descriptors (frame
// relative to base.frames, regions.cuh), or nullptr for the centre crops of m consecutive frames (preprocess.cuh).  The
// centre crops keep the table kernel: it pre-processes device-resident VGA frames 1.3x faster than the region kernel
// (2.50 M against 1.89-1.94 M frames/s on a B200 at 1000 W, DESIGN.md section 5).
static int launch_regions(cnnacc_handle* h, cudaStream_t st, RegionPrep base, int64_t m) {
    if (!base.desc) return launch_preprocess(h, st, base.frames, m, base.fh, base.fw, base.out);
    for (int64_t i0 = 0; i0 < m; i0 += 65535) {          // gridDim.y limit
        const int64_t k = std::min<int64_t>(65535, m - i0);
        RegionPrep P = base;
        P.desc += i0;
        P.out += i0 * CNNACC_FEAT_BYTES;
        preprocess_regions_kernel<<<dim3(kPrepOut, (unsigned)k), kPrepOut, 0, st>>>(P);
        h->launches++;
    }
    CU(h, cudaGetLastError());
    return 0;
}

// The loop body of realtime_detect.py:582-598 once the frames are on the device: pre-process m regions into d_gray, then --
// for detect -- conv stack, classify_vec and bbox_vec (or get_cam_bbox) into the device prediction pointers.
static int prep_then_tail(cnnacc_handle* h, cudaStream_t st, const RegionPrep& base, int64_t m, bool detect,
                          float* d_probs, int32_t* d_cls, int32_t* d_bbox, uint32_t flags) {
    int rc;
    if ((rc = launch_regions(h, st, base, m))) return rc;
    if (!detect) return 0;
    const size_t img_sz = CNNACC_FEAT_BYTES;
    const bool ups = (flags & CNNACC_FLAG_BBOX_UPSAMPLED) && d_bbox;
    if (infer_needs_feat_ws(ups, 0) && (rc = grow(h, h->d_feat, (size_t)m * img_sz))) return rc;
    const TailArgs A = make_tail(h, d_probs, d_cls, ups ? nullptr : d_bbox, false, flags);
    if ((rc = infer_device(h, st, base.out, m, h->d_feat.p, ups, A, 0))) return rc;
    if (ups && (rc = launch_cam_upsampled(h, st, h->d_feat.p, m, d_cls, d_bbox, nullptr))) return rc;
    return 0;
}

// The next entry of the descriptor ring, with room for n descriptors and n_first frame-range entries.  Its previous user --
// kDescRing calls ago, possibly an asynchronous device-pointer call on any stream -- recorded the entry's event after its last
// launch that reads it.
static int desc_acquire(cnnacc_handle* h, int64_t n, DescBuf** out, int64_t n_first = 0) {
    DescBuf& b = h->rdesc[h->rdesc_next];
    h->rdesc_next = (h->rdesc_next + 1) % kDescRing;
    CU(h, cudaEventSynchronize(b.ev));                   // an event never recorded counts as complete
    int rc;
    if ((rc = grow(h, b.host, (size_t)n)) || (rc = grow(h, b.dev, (size_t)n)) || (rc = grow(h, b.first_host, (size_t)n_first)) ||
        (rc = grow(h, b.first_dev, (size_t)n_first)))
        return rc;
    *out = &b;
    return 0;
}

// ---- merging region detections into per-frame detections (region_merge.h / region_merge.cuh) -----------------------------

// The merge of one call: its arguments, the caller's five outputs (rows of frame 0) and the per-frame region ranges.
struct MergeSpec {
    float score_min = 0.f, iou_max = 0.f;
    int max_det = 1;
    bool agnostic = false;
    int32_t *n_det = nullptr, *det_region = nullptr, *det_cls = nullptr;
    float *det_score = nullptr, *det_box = nullptr;
    std::vector<int64_t> first;                 // [n_frames + 1]: frame f holds regions first[f] .. first[f+1]-1
};

// Checks shared by cnnacc_detect_objects and the cnnacc_merge_regions calls once the regions themselves passed their checks:
// the merge limits, n_det, and at most kMergeMaxPerFrame regions per frame.  Fills M.first.  "" or why not.
static std::string merge_error(const RegionRecords& rg, int64_t n, int64_t n_frames, MergeSpec& M) {
    if (!M.n_det) return "NULL n_det";
    if (const char* why = merge_limits_error(M.iou_max, M.max_det)) return why;
    if (n > 0x7fffffffLL) return "more than 2^31-1 regions in one merging call";
    int64_t most, bad;
    if (const char* why = merge_frame_ranges([&](int64_t r) { return rg.frame(r); }, n, n_frames, M.first, &most, &bad))
        return "frame " + std::to_string(bad) + ": " + why;
    return "";
}
static int merge_check(cnnacc_handle* h, const RegionRecords& rg, int64_t n, int64_t n_frames, MergeSpec& M) {
    const std::string why = merge_error(rg, n, n_frames, M);
    return why.empty() ? 0 : fail(h, CNNACC_ERR_ARG, why);
}

// The arguments of cnnacc_merge_regions / cnnacc_merge_regions_host: "" or why not.  There is no frame size, so a region's
// frame, position and sizes are checked, not that it lies inside its frame.
static std::string merge_call_error(const RegionRecords& rg, int64_t n, int64_t n_frames, const float* scores, const int32_t* cls,
                                    const int32_t* bbox, MergeSpec& M) {
    if (n < 0 || n_frames < 0) return "negative n_frames / n_regions";
    if (n > 0 && (!rg.p || !scores || !cls || !bbox)) return "NULL region / score / class / box pointer";
    int64_t bad;
    if (const char* why = region_error(rg, n, n_frames, false, 0, 0, &bad)) return "region " + std::to_string(bad) + ": " + why;
    return merge_error(rg, n, n_frames, M);
}

// The device descriptors (regions.cuh, region_merge.cuh) of regions [0, n), frame indices as the caller gave them
static void fill_desc(int4* d, const RegionRecords& rg, int64_t n) {
    if (rg.stride == 4) {
        if (n) std::memcpy(d, rg.p, (size_t)n * sizeof(int4));          // a square's record is its descriptor
        return;
    }
    for (int64_t r = 0; r < n; r++) d[r] = make_int4((int)rg.frame(r), rg.x(r), rg.y(r), rg.wh(r));
}

static MergeSpec make_merge_spec(float score_min, float iou_max, int max_det, int32_t* n_det, int32_t* det_region, int32_t* det_cls,
                          float* det_score, float* det_box, uint32_t flags) {
    MergeSpec M;
    M.score_min = score_min; M.iou_max = iou_max; M.max_det = max_det;
    M.agnostic = (flags & CNNACC_FLAG_CLASS_AGNOSTIC) != 0;
    M.n_det = n_det; M.det_region = det_region; M.det_cls = det_cls; M.det_score = det_score; M.det_box = det_box;
    return M;
}

// Merge frames [fa, fb) on `st`: A carries the region data (desc, predictions) and the outputs of frame fa; d_first is the
// device copy of M.first.  The shared memory follows the largest frame of the launch.
static int launch_merge(cnnacc_handle* h, cudaStream_t st, MergeArgs A, const MergeSpec& M, const long long* d_first,
                        int64_t fa, int64_t fb) {
    if (!h->merge_attr_set) {
        CU(h, cudaFuncSetAttribute(merge_regions_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   (int)merge_smem_bytes(kMergeMaxPerFrame, kMergeMaxDet)));
        h->merge_attr_set = true;
    }
    A.score_min = M.score_min; A.iou_max = M.iou_max; A.max_det = M.max_det; A.agnostic = M.agnostic ? 1 : 0;
    constexpr int64_t kFramesPerLaunch = 1 << 20;
    for (int64_t g0 = fa; g0 < fb; g0 += kFramesPerLaunch) {
        const int64_t g1 = std::min(fb, g0 + kFramesPerLaunch);
        int64_t most = 0;
        for (int64_t f = g0; f < g1; f++) most = std::max(most, M.first[f + 1] - M.first[f]);
        int cap = 1;
        while (cap < most) cap <<= 1;
        MergeArgs L = A;
        const size_t o = (size_t)(g0 - fa) * M.max_det;
        L.first = d_first + g0;
        L.key_cap = cap; L.kept_cap = std::min(M.max_det, cap);
        L.n_det = A.n_det + (g0 - fa);
        L.det_region = A.det_region ? A.det_region + o : nullptr;
        L.det_cls = A.det_cls ? A.det_cls + o : nullptr;
        L.det_score = A.det_score ? A.det_score + o : nullptr;
        L.det_box = A.det_box ? A.det_box + o : nullptr;
        merge_regions_kernel<<<(unsigned)(g1 - g0), kMergeThreads, merge_smem_bytes(L.key_cap, L.kept_cap), st>>>(L);
        h->launches++;
        CU(h, cudaGetLastError());
    }
    return 0;
}

// Merge frames [fa, fb) of a host-pointer call into the caller's host arrays: the kernel writes a group of frames into h->d_det
// as [box | region | cls | score | n_det], one D2H brings it to the pinned h->h_det, memcpy to the caller.  Waits for st.
static int merge_to_host(cnnacc_handle* h, cudaStream_t st, MergeArgs A, const MergeSpec& M, const long long* d_first,
                         int64_t fa, int64_t fb) {
    const size_t D = (size_t)M.max_det, per_frame = 4 + D * 28;
    const int64_t step = std::max<int64_t>(1, std::min<int64_t>(fb - fa, ((size_t)8 << 20) / per_frame));
    const size_t need = (size_t)step * per_frame;
    int rc;
    if ((rc = grow(h, h->d_det, need)) || (rc = grow(h, h->h_det, need))) return rc;
    for (int64_t g0 = fa; g0 < fb; g0 += step) {
        const int64_t m = std::min(step, fb - g0);
        const size_t md = (size_t)m * D, o_reg = md * 16, o_cls = o_reg + md * 4, o_score = o_cls + md * 4, o_n = o_score + md * 4;
        uint8_t *d = h->d_det.p, *hd = h->h_det.p;
        A.det_box = reinterpret_cast<float4*>(d);
        A.det_region = reinterpret_cast<int32_t*>(d + o_reg);
        A.det_cls = reinterpret_cast<int32_t*>(d + o_cls);
        A.det_score = reinterpret_cast<float*>(d + o_score);
        A.n_det = reinterpret_cast<int32_t*>(d + o_n);
        if ((rc = launch_merge(h, st, A, M, d_first, g0, g0 + m))) return rc;
        CU(h, cudaMemcpyAsync(hd, d, o_n + (size_t)m * 4, cudaMemcpyDeviceToHost, st));
        CU(h, cudaStreamSynchronize(st));
        const size_t at = (size_t)g0 * D;
        std::memcpy(M.n_det + g0, hd + o_n, (size_t)m * 4);
        if (M.det_box) std::memcpy(M.det_box + at * 4, hd, md * 16);
        if (M.det_region) std::memcpy(M.det_region + at, hd + o_reg, md * 4);
        if (M.det_cls) std::memcpy(M.det_cls + at, hd + o_cls, md * 4);
        if (M.det_score) std::memcpy(M.det_score + at, hd + o_score, md * 4);
    }
    return 0;
}

// The region data of a merge over predictions laid out as PredBlock's [bbox | probs | cls] for regions r_pred0 ..: the score
// of a region is its probability (or logit) of its own class.
static MergeArgs merge_args_of_predictions(const int4* d_desc, int64_t r_pred0, const int32_t* bbox, const float* probs,
                                           const int32_t* cls, int n_cls, const MergeSpec& M) {
    MergeArgs A = {};
    A.desc = d_desc; A.r_pred0 = r_pred0;
    A.score = probs; A.score_stride = n_cls; A.score_by_cls = 1;
    A.cls = cls; A.bbox = bbox;
    A.n_det = M.n_det; A.det_region = M.det_region; A.det_cls = M.det_cls; A.det_score = M.det_score;
    A.det_box = reinterpret_cast<float4*>(M.det_box);
    return A;
}

// Shared body of preprocess_bgr / detect_frames (centre: n frames, one centre crop each) and of
// preprocess_regions / detect_regions (n regions over n_frames frames).  gray128 out, predictions out, or both.  With `mg`
// (detect_objects, n > 0) the predictions stay on the device and are merged into mg's per-frame detections instead; pieces of
// the call then end at frame edges, so no frame is merged before all of its regions are predicted.
static int regions_impl(cnnacc_handle* h, const uint8_t* frames, int64_t n_frames, int fh, int fw, bool centre,
                        const int32_t* regions, int64_t n, uint8_t* gray128, float* probs, int32_t* cls, int32_t* bbox,
                        bool detect, uint32_t flags, MergeSpec* mg = nullptr) {
    int rc;
    const RegionRecords rg(regions, (flags & CNNACC_FLAG_RECTS) != 0);
    if (!h) return CNNACC_ERR_ARG;
    if (detect) {
        if ((rc = check_ready(h))) return rc;
        if (!h->fc_loaded) return fail(h, CNNACC_ERR_STATE, "classifier not loaded (call cnnacc_load_classifier)");
    }
    if (centre && (n < 0 || fh < kPrepOut || fw < kPrepOut || std::min(fh, fw) > kPrepMaxSide))
        return fail(h, CNNACC_ERR_ARG, "bad n / frame size (the square crop must be 128..8192 pixels a side)");
    if (!centre && (n < 0 || n_frames < 0)) return fail(h, CNNACC_ERR_ARG, "negative n_frames / n_regions");
    if (n == 0) return CNNACC_OK;
    if (!frames || (!centre && !regions) || (!detect && !gray128)) return fail(h, CNNACC_ERR_ARG, "NULL frame / region / output pointer");
    if (!centre) {
        int64_t bad;
        if (const char* why = region_error(rg, n, n_frames, true, fh, fw, &bad))
            return fail(h, CNNACC_ERR_ARG, "region " + std::to_string(bad) + ": " + why);
        if (mg && (rc = merge_check(h, rg, n, n_frames, *mg))) return rc;
    }
    CU(h, cudaSetDevice(h->device));
    const size_t frame_sz = (size_t)fh * fw * 3, img_sz = CNNACC_FEAT_BYTES;
    const int nc = h->n_cls;
    RegionPrep base;
    base.fh = fh; base.fw = fw; base.desc = nullptr;

    if (flags & CNNACC_FLAG_DEVICE_PTRS) {
        if (detect && (flags & CNNACC_FLAG_BBOX_UPSAMPLED) && bbox && !cls)
            return fail(h, CNNACC_ERR_ARG, "CNNACC_FLAG_BBOX_UPSAMPLED with device pointers needs a cls array");
        REQUIRE_ALIGNED(h, gray128, 16, "gray128");
        REQUIRE_ALIGNED(h, bbox, 16, "bbox");
        REQUIRE_ALIGNED(h, probs, 4, "probs");
        REQUIRE_ALIGNED(h, cls, 4, "cls");
        if (mg) {
            REQUIRE_ALIGNED(h, mg->det_box, 16, "det_box");
            REQUIRE_ALIGNED(h, mg->n_det, 4, "n_det");
            REQUIRE_ALIGNED(h, mg->det_region, 4, "det_region");
            REQUIRE_ALIGNED(h, mg->det_cls, 4, "det_cls");
            REQUIRE_ALIGNED(h, mg->det_score, 4, "det_score");
        }
        DescBuf* db = nullptr;
        if (!centre) {
            if ((rc = desc_acquire(h, n, &db, mg ? n_frames + 1 : 0))) return rc;
            fill_desc(db->host.p, rg, n);
            CU(h, cudaMemcpyAsync(db->dev.p, db->host.p, (size_t)n * sizeof(int4), cudaMemcpyHostToDevice, h->stream));
            if (mg) {
                std::memcpy(db->first_host.p, mg->first.data(), (size_t)(n_frames + 1) * sizeof(long long));
                CU(h, cudaMemcpyAsync(db->first_dev.p, db->first_host.p, (size_t)(n_frames + 1) * sizeof(long long),
                                      cudaMemcpyHostToDevice, h->stream));
            }
        }
        auto run = [&]() -> int {
            const int64_t chunk = std::min<int64_t>(n, 16384);
            uint8_t* g = gray128;
            int r;
            if (!g && (r = grow(h, h->d_gray, (size_t)chunk * img_sz))) return r;
            // detect_objects: the predictions of a piece go to a workspace laid out as PredBlock's, then the piece's frames
            // are merged; a piece is the whole frames that fit `chunk` regions (a frame has at most kMergeMaxPerFrame)
            const size_t w_probs = (size_t)chunk * 16, w_cls = w_probs + (size_t)chunk * nc * 4;
            if (mg && (r = grow(h, h->d_mpred, (size_t)chunk * kPredBytesPerImage))) return r;
            int64_t m = 0;
            for (int64_t i0 = 0, fa = 0; i0 < n; i0 += m) {
                m = std::min(chunk, n - i0);
                if (mg && i0 + m < n) m = mg->first[rg.frame(i0 + m)] - i0;
                RegionPrep P = base;
                P.frames = centre ? frames + i0 * frame_sz : frames;
                P.desc = centre ? nullptr : db->dev.p + i0;
                P.out = g ? g + i0 * img_sz : h->d_gray.p;
                if (mg) {
                    int32_t* wb = reinterpret_cast<int32_t*>(h->d_mpred.p);
                    float* wp = reinterpret_cast<float*>(h->d_mpred.p + w_probs);
                    int32_t* wc = reinterpret_cast<int32_t*>(h->d_mpred.p + w_cls);
                    const int64_t fb = i0 + m == n ? n_frames : rg.frame(i0 + m);
                    MergeArgs A = merge_args_of_predictions(db->dev.p, i0, wb, wp, wc, nc, *mg);
                    A.n_det += fa;
                    const size_t o = (size_t)fa * mg->max_det;
                    if (A.det_region) A.det_region += o;
                    if (A.det_cls) A.det_cls += o;
                    if (A.det_score) A.det_score += o;
                    if (A.det_box) A.det_box += o;
                    if ((r = prep_then_tail(h, h->stream, P, m, detect, wp, wc, wb, flags)) ||
                        (r = launch_merge(h, h->stream, A, *mg, db->first_dev.p, fa, fb)))
                        return r;
                    fa = fb;
                } else if ((r = prep_then_tail(h, h->stream, P, m, detect, probs ? probs + i0 * nc : nullptr, cls ? cls + i0 : nullptr,
                                               bbox ? bbox + i0 * 4 : nullptr, flags))) {
                    return r;
                }
            }
            return 0;
        };
        rc = run();
        if (db) CU(h, cudaEventRecord(db->ev, h->stream));   // also after a failed launch: earlier ones may still read it
        return rc;
    }

    HostCall call(h);
    if ((rc = call.begin())) return rc;
    // prediction blocks: kPredSuper regions each, or for detect_objects the whole frames that fit in kPredSuper
    auto frame_of = [&](int64_t r) -> int64_t { return centre ? r : rg.frame(r); };
    std::vector<int64_t> blocks;
    if (mg) {
        blocks = frame_aligned_blocks(frame_of, n, kPredSuper);
    } else {
        for (int64_t b = 0; b < n; b += kPredSuper) blocks.push_back(b);
        blocks.push_back(n);
    }
    auto block_end = [&](int64_t r) { return *std::upper_bound(blocks.begin(), blocks.end(), r); };
    const std::vector<RegionChunk> plan = make_region_plan_blocks(frame_of, n, frame_sz, block_end);
    size_t staged = 0, max_stage = 0;
    int64_t max_regions = 0;
    for (const RegionChunk& c : plan) {
        staged += (size_t)(c.f1 - c.f0) * frame_sz;
        max_stage = std::max(max_stage, (size_t)(c.f1 - c.f0) * frame_sz);
        max_regions = std::max(max_regions, c.r1 - c.r0);
    }
    const bool small = n <= kSmallN && staged <= ((size_t)64 << 20);   // latency path: one stream, one result copy
    // descriptors with the frame index relative to the staging buffer of the region's chunk
    DescBuf* db = nullptr;
    if (!centre) {
        if ((rc = desc_acquire(h, n, &db, mg ? n_frames + 1 : 0))) return rc;
        int64_t below = 0;                               // small: frames staged ahead of the chunk in the one buffer
        for (const RegionChunk& c : plan) {
            for (int64_t r = c.r0; r < c.r1; r++)
                db->host.p[r] = make_int4((int)(rg.frame(r) - c.f0 + (small ? below : 0)), rg.x(r), rg.y(r), rg.wh(r));
            below += c.f1 - c.f0;
        }
        CU(h, cudaMemcpyAsync(db->dev.p, db->host.p, (size_t)n * sizeof(int4), cudaMemcpyHostToDevice, small ? h->st_k : h->st_h2d));
        if (mg) {
            std::memcpy(db->first_host.p, mg->first.data(), (size_t)(n_frames + 1) * sizeof(long long));
            CU(h, cudaMemcpyAsync(db->first_dev.p, db->first_host.p, (size_t)(n_frames + 1) * sizeof(long long), cudaMemcpyHostToDevice,
                                  small ? h->st_k : h->st_h2d));
        }
    }
    // detect_objects: merge the block of predictions [pred.s0, pred.end()) -- whole frames -- into the caller's arrays, up to
    // the frame of the next block (frames without regions in between belong to this block)
    int64_t det_f = 0;
    auto merge_block = [&](const PredBlock& pred, cudaStream_t st) -> int {
        const int64_t fb = pred.end() == n ? n_frames : rg.frame(pred.end());
        const MergeArgs A = merge_args_of_predictions(db->dev.p, pred.s0, pred.bbox(pred.s0), pred.probs(pred.s0), pred.cls(pred.s0), nc, *mg);
        const int r = merge_to_host(h, st, A, *mg, db->first_dev.p, det_f, fb);
        det_f = fb;
        return r;
    };
    auto region_base = [&](const uint8_t* d_frames, int64_t r, int64_t r_frame0, uint8_t* d_gray) {
        RegionPrep P = base;
        P.frames = centre ? d_frames + (r - r_frame0) * frame_sz : d_frames;
        P.desc = centre ? nullptr : db->dev.p + r;
        P.out = d_gray;
        return P;
    };

    PredBlock pred(h);
    Slot* s;
    if (small) {
        cudaStream_t st = h->st_k;
        if ((rc = call.acquire(s, staged, n * img_sz)) || (rc = pred.start(0, n))) return rc;
        // one copy per run of consecutive staged frames (the chunks of one run are adjacent in the buffer)
        size_t off = 0;
        for (size_t k = 0; k < plan.size();) {
            size_t j = k + 1;
            while (j < plan.size() && plan[j].f0 == plan[j - 1].f1) j++;
            const size_t bytes = (size_t)(plan[j - 1].f1 - plan[k].f0) * frame_sz;
            CU(h, cudaMemcpyAsync(s->d_in.p + off, frames + plan[k].f0 * frame_sz, bytes, cudaMemcpyHostToDevice, st));
            off += bytes;
            k = j;
        }
        if ((rc = prep_then_tail(h, st, region_base(s->d_in.p, 0, 0, s->d_out.p), n, detect, pred.probs(0), pred.cls(0), pred.bbox(0), flags)))
            return rc;
        if (gray128) CU(h, cudaMemcpyAsync(gray128, s->d_out.p, n * img_sz, cudaMemcpyDeviceToHost, st));
        if (mg) rc = merge_block(pred, st);
        else if (detect) rc = pred.flush(st, probs, cls, bbox, false);
        if (db) CU(h, cudaEventRecord(db->ev, st));
        if (rc) return rc;
        return detect ? call.done(true) : call.finish(st, false);
    }
    // Staged chunks of about 16 MiB of frames through the ring (HostCall).  A chunk's regions run in launches of up to
    // kRegionLaunch: their gray images fill the slot's output buffer, so a launch after the first waits for the gray copy of
    // the launch before.
    const int64_t per_launch = std::min<int64_t>(max_regions, kRegionLaunch);
    size_t bi = 1;                                       // pred holds block [blocks[bi - 1], blocks[bi])
    if (detect && (rc = pred.start(0, blocks[1]))) return rc;
    for (const RegionChunk& c : plan) {
        if (detect && c.r0 >= pred.end()) {              // the plan never lets a chunk straddle a block edge
            if ((rc = mg ? merge_block(pred, h->st_k) : pred.flush(h->st_k, probs, cls, bbox, false)) ||
                (rc = pred.start(pred.end(), blocks[bi + 1] - blocks[bi])))
                return rc;
            bi++;
        }
        if ((rc = call.acquire(s, max_stage, per_launch * img_sz))) return rc;
        CU(h, cudaMemcpyAsync(s->d_in.p, frames + c.f0 * frame_sz, (size_t)(c.f1 - c.f0) * frame_sz, cudaMemcpyHostToDevice, h->st_h2d));
        if ((rc = call.staged(*s))) return rc;
        for (int64_t r = c.r0; r < c.r1; r += per_launch) {
            const int64_t m = std::min(per_launch, c.r1 - r);
            if (r > c.r0 && gray128 && (rc = call.wait_released(*s, h->st_k))) return rc;
            if ((rc = prep_then_tail(h, h->st_k, region_base(s->d_in.p, r, c.r0, s->d_out.p), m, detect, detect ? pred.probs(r) : nullptr,
                                     detect ? pred.cls(r) : nullptr, detect ? pred.bbox(r) : nullptr, flags)) ||
                (rc = call.computed(*s)))
                return rc;
            if (gray128) CU(h, cudaMemcpyAsync(gray128 + r * img_sz, s->d_out.p, m * img_sz, cudaMemcpyDeviceToHost, h->st_d2h));
            if ((rc = call.released(*s, h->st_d2h))) return rc;
        }
    }
    if (mg) rc = merge_block(pred, h->st_k);
    else if (detect) rc = pred.flush(h->st_k, probs, cls, bbox, false);
    if (db) CU(h, cudaEventRecord(db->ev, h->st_k));
    if (rc) return rc;
    return call.finish(h->st_d2h, detect);
}

int cnnacc_preprocess_bgr(cnnacc_handle* h, const uint8_t* frames, int64_t n, int fh, int fw, uint8_t* gray128, uint32_t flags) {
    return regions_impl(h, frames, n, fh, fw, true, nullptr, n, gray128, nullptr, nullptr, nullptr, false, flags);
}

int cnnacc_detect_frames(cnnacc_handle* h, const uint8_t* frames, int64_t n, int fh, int fw, uint8_t* gray128,
                         float* probs, int32_t* cls, int32_t* bbox, uint32_t flags) {
    return regions_impl(h, frames, n, fh, fw, true, nullptr, n, gray128, probs, cls, bbox, true, flags);
}

int cnnacc_preprocess_regions(cnnacc_handle* h, const uint8_t* frames, int64_t n_frames, int fh, int fw,
                              const int32_t* regions, int64_t n_regions, uint8_t* gray128, uint32_t flags) {
    return regions_impl(h, frames, n_frames, fh, fw, false, regions, n_regions, gray128, nullptr, nullptr, nullptr, false, flags);
}

int cnnacc_detect_regions(cnnacc_handle* h, const uint8_t* frames, int64_t n_frames, int fh, int fw,
                          const int32_t* regions, int64_t n_regions, uint8_t* gray128,
                          float* probs, int32_t* cls, int32_t* bbox, uint32_t flags) {
    return regions_impl(h, frames, n_frames, fh, fw, false, regions, n_regions, gray128, probs, cls, bbox, true, flags);
}

// cnnacc_merge_regions: the merge alone on predictions the caller has (n may be 0: every frame gets no detections)
static int merge_impl(cnnacc_handle* h, const int32_t* regions, int64_t n, int64_t n_frames, const float* scores, const int32_t* cls,
                      const int32_t* bbox, MergeSpec& M, uint32_t flags) {
    int rc;
    const RegionRecords rg(regions, (flags & CNNACC_FLAG_RECTS) != 0);
    const std::string why = merge_call_error(rg, n, n_frames, scores, cls, bbox, M);
    if (!why.empty()) return fail(h, CNNACC_ERR_ARG, why);
    if (n_frames == 0) return CNNACC_OK;
    CU(h, cudaSetDevice(h->device));
    const size_t first_bytes = (size_t)(n_frames + 1) * sizeof(long long);
    MergeArgs A = {};
    A.score_stride = 1; A.score_by_cls = 0;
    if (flags & CNNACC_FLAG_DEVICE_PTRS) {
        REQUIRE_ALIGNED(h, scores, 4, "scores");
        REQUIRE_ALIGNED(h, cls, 4, "cls");
        REQUIRE_ALIGNED(h, bbox, 4, "bbox");
        REQUIRE_ALIGNED(h, M.det_box, 16, "det_box");
        REQUIRE_ALIGNED(h, M.n_det, 4, "n_det");
        REQUIRE_ALIGNED(h, M.det_region, 4, "det_region");
        REQUIRE_ALIGNED(h, M.det_cls, 4, "det_cls");
        REQUIRE_ALIGNED(h, M.det_score, 4, "det_score");
        DescBuf* db = nullptr;
        if ((rc = desc_acquire(h, n, &db, n_frames + 1))) return rc;
        fill_desc(db->host.p, rg, n);
        std::memcpy(db->first_host.p, M.first.data(), first_bytes);
        if (n) CU(h, cudaMemcpyAsync(db->dev.p, db->host.p, (size_t)n * sizeof(int4), cudaMemcpyHostToDevice, h->stream));
        CU(h, cudaMemcpyAsync(db->first_dev.p, db->first_host.p, first_bytes, cudaMemcpyHostToDevice, h->stream));
        A.desc = db->dev.p; A.r_pred0 = 0; A.score = scores; A.cls = cls; A.bbox = bbox;
        A.n_det = M.n_det; A.det_region = M.det_region; A.det_cls = M.det_cls; A.det_score = M.det_score;
        A.det_box = reinterpret_cast<float4*>(M.det_box);
        rc = launch_merge(h, h->stream, A, M, db->first_dev.p, 0, n_frames);
        CU(h, cudaEventRecord(db->ev, h->stream));     // also after a failed launch: earlier ones may still read it
        return rc;
    }
    // Host pointers: blocks of whole frames (at most kPredSuper regions) go in, are merged, and their detections come out.
    HostCall call(h);
    if ((rc = call.begin())) return rc;
    cudaStream_t st = h->st_k;
    DescBuf* db = nullptr;
    if ((rc = desc_acquire(h, n, &db, n_frames + 1))) return rc;
    fill_desc(db->host.p, rg, n);
    std::memcpy(db->first_host.p, M.first.data(), first_bytes);
    if (n) CU(h, cudaMemcpyAsync(db->dev.p, db->host.p, (size_t)n * sizeof(int4), cudaMemcpyHostToDevice, st));
    CU(h, cudaMemcpyAsync(db->first_dev.p, db->first_host.p, first_bytes, cudaMemcpyHostToDevice, st));
    const std::vector<int64_t> blocks = frame_aligned_blocks([&](int64_t r) { return rg.frame(r); }, n, kPredSuper);
    int64_t most = 0;
    for (size_t k = 1; k < blocks.size(); k++) most = std::max(most, blocks[k] - blocks[k - 1]);
    if (most && (rc = grow(h, h->d_mpred, (size_t)most * 24))) return rc;
    A.desc = db->dev.p;
    int64_t fa = 0;
    for (size_t k = 0; k < std::max<size_t>(1, blocks.size() - 1); k++) {
        const int64_t b0 = blocks[k], m = blocks.size() > 1 ? blocks[k + 1] - b0 : 0;
        const int64_t fb = b0 + m == n ? n_frames : rg.frame(b0 + m);
        if (m) {
            CU(h, cudaMemcpyAsync(h->d_mpred.p, bbox + 4 * b0, (size_t)m * 16, cudaMemcpyHostToDevice, st));
            CU(h, cudaMemcpyAsync(h->d_mpred.p + (size_t)m * 16, scores + b0, (size_t)m * 4, cudaMemcpyHostToDevice, st));
            CU(h, cudaMemcpyAsync(h->d_mpred.p + (size_t)m * 20, cls + b0, (size_t)m * 4, cudaMemcpyHostToDevice, st));
        }
        A.r_pred0 = b0;
        A.bbox = reinterpret_cast<const int32_t*>(h->d_mpred.p);
        A.score = reinterpret_cast<const float*>(h->d_mpred.p + (size_t)m * 16);
        A.cls = reinterpret_cast<const int32_t*>(h->d_mpred.p + (size_t)m * 20);
        rc = merge_to_host(h, st, A, M, db->first_dev.p, fa, fb);
        if (rc) break;
        fa = fb;
    }
    CU(h, cudaEventRecord(db->ev, st));
    if (rc) return rc;
    return call.done(false);
}

int cnnacc_detect_objects(cnnacc_handle* h, const uint8_t* frames, int64_t n_frames, int fh, int fw, const int32_t* regions,
                          int64_t n_regions, float score_min, float iou_max, int max_det, int32_t* n_det, int32_t* det_region,
                          int32_t* det_cls, float* det_score, float* det_box, uint32_t flags) {
    int rc;
    if (!h) return CNNACC_ERR_ARG;
    MergeSpec M = make_merge_spec(score_min, iou_max, max_det, n_det, det_region, det_cls, det_score, det_box, flags);
    if (n_regions != 0)
        return regions_impl(h, frames, n_frames, fh, fw, false, regions, n_regions, nullptr, nullptr, nullptr, nullptr, true, flags, &M);
    // no regions: detect_regions' state checks, then every frame gets no detections
    if ((rc = check_ready(h))) return rc;
    if (!h->fc_loaded) return fail(h, CNNACC_ERR_STATE, "classifier not loaded (call cnnacc_load_classifier)");
    return merge_impl(h, nullptr, 0, n_frames, nullptr, nullptr, nullptr, M, flags);
}

int cnnacc_merge_regions(cnnacc_handle* h, const int32_t* regions, int64_t n_regions, int64_t n_frames, const float* scores,
                         const int32_t* cls, const int32_t* bbox, float score_min, float iou_max, int max_det, int32_t* n_det,
                         int32_t* det_region, int32_t* det_cls, float* det_score, float* det_box, uint32_t flags) {
    if (!h) return CNNACC_ERR_ARG;
    MergeSpec M = make_merge_spec(score_min, iou_max, max_det, n_det, det_region, det_cls, det_score, det_box, flags);
    return merge_impl(h, regions, n_regions, n_frames, scores, cls, bbox, M, flags);
}

int cnnacc_merge_regions_host(const int32_t* regions, int64_t n_regions, int64_t n_frames, const float* scores, const int32_t* cls,
                              const int32_t* bbox, float score_min, float iou_max, int max_det, int32_t* n_det, int32_t* det_region,
                              int32_t* det_cls, float* det_score, float* det_box, uint32_t flags) {
    if (flags & CNNACC_FLAG_DEVICE_PTRS) return CNNACC_ERR_ARG;
    MergeSpec M = make_merge_spec(score_min, iou_max, max_det, n_det, det_region, det_cls, det_score, det_box, flags);
    const RegionRecords rg(regions, (flags & CNNACC_FLAG_RECTS) != 0);
    if (!merge_call_error(rg, n_regions, n_frames, scores, cls, bbox, M).empty()) return CNNACC_ERR_ARG;
    const size_t D = (size_t)max_det;
    for (int64_t f = 0; f < n_frames; f++)
        n_det[f] = merge_frame_host(rg, scores, cls, bbox, M.first[f], M.first[f + 1] - M.first[f], score_min, iou_max, max_det,
                                    M.agnostic, det_region ? det_region + f * D : nullptr, det_cls ? det_cls + f * D : nullptr,
                                    det_score ? det_score + f * D : nullptr, det_box ? det_box + f * D * 4 : nullptr);
    return CNNACC_OK;
}

// ---- scanning whole frames and image pyramids (cnnacc_scan_frames / cnnacc_scan_objects, cnnacc_preprocess_pyramid /
// cnnacc_scan_pyramid / cnnacc_scan_pyramid_objects) ---------------------------------------------------------------------

// Scan windows along a side of `side` pixels: 0, stride, 2 stride, ... plus one flush with the far edge when that is missing.
static int scan_count(int side, int stride) {
    const int last = side - CNNACC_IMG;
    return last / stride + 1 + (last % stride != 0);
}

// The checked levels of a pyramid call (include/cnnacc.h); cnnacc_scan_frames is the one level (fw, fh).  Level l of a frame
// holds its windows first[l] .. first[l + 1] - 1 and w[l] * h[l] gray pixels (and map bytes) at px[l] of the frame's total.
static_assert(kPyramidMaxLevels == CNNACC_PYRAMID_MAX_LEVELS && kScanMaxLevels == CNNACC_PYRAMID_MAX_LEVELS, "level limits");

struct PyramidPlan {
    int fh = 0, fw = 0, n_levels = 0, stride = 0;
    int w[kPyramidMaxLevels] = {}, h[kPyramidMaxLevels] = {}, nx[kPyramidMaxLevels] = {}, ny[kPyramidMaxLevels] = {};
    int64_t first[kPyramidMaxLevels + 1] = {};
    size_t px[kPyramidMaxLevels + 1] = {};
    bool identity(int l) const { return w[l] == fw && h[l] == fh; }   // the gray frame itself: no resize, no copy
    int box(int l) const { return area_fast_axis(fw, w[l]) && area_fast_axis(fh, h[l]); }   // OpenCV's integer path
    int64_t per() const { return first[n_levels]; }                 // windows per frame
    size_t level_px() const { return px[n_levels]; }
    // the frame rectangle (x, y, w, h) of window (ix, iy) of level l
    int4 rect(int l, int ix, int iy) const {
        const int64_t x = std::min(ix * stride, w[l] - CNNACC_IMG), y = std::min(iy * stride, h[l] - CNNACC_IMG);
        return make_int4((int)(x * fw / w[l]), (int)(y * fh / h[l]), CNNACC_IMG * fw / w[l], CNNACC_IMG * fh / h[l]);
    }
};

// Do the windows of a level of side D land on whole pixels of the frame's side S: 128 S / D and o S / D an integer for every
// window origin o (the actual origins, flush one included, not just the stride)?
static bool whole_pixels(int S, int D, int stride) {
    if ((int64_t)CNNACC_IMG * S % D) return false;
    for (int ix = 0, n = scan_count(D, stride); ix < n; ix++)
        if ((int64_t)std::min(ix * stride, D - CNNACC_IMG) * S % D) return false;
    return true;
}

// nullptr with *P filled when frames of fh x fw, levels [L][2] (w, h) and stride (0: no windows, cnnacc_preprocess_pyramid)
// make a pyramid call, else why not.
static const char* pyramid_error(int fh, int fw, const int32_t* levels, int L, int stride, PyramidPlan* P) {
    if (fh < kRegionMinSide || fh > kRegionMaxSide || fw < kRegionMinSide || fw > kRegionMaxSide) return "frame sides must be in 128..8192";
    if (L < 1 || L > kPyramidMaxLevels) return "1..16 levels";
    if (!levels) return "NULL levels";
    if (stride && (stride < 8 || stride % 8)) return "stride must be a positive multiple of 8";
    P->fh = fh; P->fw = fw; P->n_levels = L; P->stride = stride;
    for (int l = 0; l < L; l++) {
        const int w = levels[2 * l], hl = levels[2 * l + 1];
        if (w % 16 || hl % 16 || w < CNNACC_IMG || hl < CNNACC_IMG || w > fw || hl > fh)
            return "level sides must be multiples of 16 with 128 <= w <= fw and 128 <= h <= fh";
        P->w[l] = w; P->h[l] = hl;
        P->px[l + 1] = P->px[l] + (size_t)w * hl;
        if (stride) {
            if (!whole_pixels(fw, w, stride) || !whole_pixels(fh, hl, stride))
                return "a window's frame rectangle (x fw / w, y fh / h, 128 fw / w, 128 fh / h) is not in whole pixels";
            P->nx[l] = scan_count(w, stride); P->ny[l] = scan_count(hl, stride);
        }
        P->first[l + 1] = P->first[l] + (int64_t)P->nx[l] * P->ny[l];
    }
    return nullptr;
}

// gray_full_kernel over k frames of `plane` pixels
static int launch_gray(cnnacc_handle* h, cudaStream_t st, const uint8_t* d_frames, int64_t k, size_t plane, uint8_t* d_gray) {
    const long long pixels = (long long)(k * plane), quads = pixels / 4;
    gray_full_kernel<<<(unsigned)std::max<long long>(1, std::min<long long>((quads + 255) / 256, 16LL * h->sm_count)), 256, 0, st>>>(
        d_frames, d_gray, pixels);
    h->launches++;
    CU(h, cudaGetLastError());
    return 0;
}

// pyramid_levels_kernel on k gray frames: R's levels, `rows` rows in all
static int launch_levels(cnnacc_handle* h, cudaStream_t st, PyramidPrep R, int rows, int64_t k) {
    const size_t plane = (size_t)R.fh * R.fw;
    for (int64_t g0 = 0; g0 < k; g0 += 65535) {          // gridDim.y limit
        PyramidPrep P = R;
        P.gray += g0 * plane;
        for (int l = 0; l < P.n_levels; l++) P.lv[l].off += g0 * P.lv[l].fstride;
        pyramid_levels_kernel<<<dim3((unsigned)rows, (unsigned)std::min<int64_t>(65535, k - g0)), kPrepOut, 0, st>>>(P);
        h->launches++;
    }
    CU(h, cudaGetLastError());
    return 0;
}

static constexpr uint32_t kNoScanForm = CNNACC_FLAG_BBOX_UPSAMPLED | CNNACC_FLAG_RECTS | CNNACC_FLAG_DIRECT | CNNACC_FLAG_KEEP_MAPS |
                                        CNNACC_FLAG_TWO_KERNELS;

// Gray once per frame, the pyramid's levels, the conv stack once per level, then every window's predictions read straight
// out of its level's feature map; with `mg` (the _objects calls) the predictions stay on the device and are merged per frame
// with the windows' frame rectangles as the regions.  levels == nullptr: cnnacc_scan_frames (the one level fw x fh).
static int scan_impl(cnnacc_handle* h, const uint8_t* frames, int64_t n, int fh, int fw, const int32_t* levels, int n_levels,
                     int stride, float* probs, int32_t* cls, int32_t* bbox, uint32_t flags, MergeSpec* mg) {
    int rc;
    if (!h) return CNNACC_ERR_ARG;
    if ((rc = check_ready(h))) return rc;
    if (!h->fc_loaded) return fail(h, CNNACC_ERR_STATE, "classifier not loaded (call cnnacc_load_classifier)");
    if (n < 0) return fail(h, CNNACC_ERR_ARG, "negative n");
    PyramidPlan P;
    if (!levels) {
        if (!valid_hw(fh, fw) || fh < CNNACC_IMG || fw < CNNACC_IMG)
            return fail(h, CNNACC_ERR_ARG, "frame sides must be multiples of 16 in 128..8192");
        if (stride < 8 || stride % 8) return fail(h, CNNACC_ERR_ARG, "stride must be a positive multiple of 8");
        const int32_t one[2] = {fw, fh};
        pyramid_error(fh, fw, one, 1, stride, &P);        // passes: the identity level of a valid frame
    } else {
        if (stride < 1) return fail(h, CNNACC_ERR_ARG, "stride must be a positive multiple of 8");
        if (const char* why = pyramid_error(fh, fw, levels, n_levels, stride, &P)) return fail(h, CNNACC_ERR_ARG, why);
    }
    if (flags & kNoScanForm)
        return fail(h, CNNACC_ERR_ARG, "BBOX_UPSAMPLED / RECTS / DIRECT / KEEP_MAPS / TWO_KERNELS have no scanning form");
    const int64_t per = P.per();
    if (n > 0x7fffffffLL / per) return fail(h, CNNACC_ERR_ARG, "more than 2^31-1 windows in one call");
    if (mg) {
        if (!mg->n_det) return fail(h, CNNACC_ERR_ARG, "NULL n_det");
        if (const char* why = merge_limits_error(mg->iou_max, mg->max_det)) return fail(h, CNNACC_ERR_ARG, why);
        if (per > kMergeMaxPerFrame) return fail(h, CNNACC_ERR_ARG, "more than 16384 windows per frame in a merging call");
    }
    if (n == 0) return CNNACC_OK;
    if (!frames) return fail(h, CNNACC_ERR_ARG, "NULL frame pointer");
    CU(h, cudaSetDevice(h->device));
    const int L = P.n_levels;
    const size_t frame_sz = (size_t)fh * fw * 3, plane = (size_t)fh * fw;
    size_t resized = 0;                                   // gray pixels per frame of the levels that are resized
    for (int l = 0; l < L; l++) resized += P.identity(l) ? 0 : (size_t)P.w[l] * P.h[l];
    const int nc = h->n_cls;
    // Workspaces for k frames: d_scan_gray holds the gray frames, then (from a 256-byte boundary) each resized level as
    // [k][h][w]; d_scan_feat holds each level's maps as [k][64][h/8][w/8].  w * h is a multiple of 256, so every level
    // starts 16-byte aligned.  The window gather may read 16 bytes past the last map.
    auto gray_base = [&](int64_t k) { return (k * plane + 255) / 256 * 256; };
    auto grow_ws = [&](int64_t k) -> int {
        int r;
        if ((r = grow(h, h->d_scan_gray, gray_base(k) + k * resized)) || (r = grow(h, h->d_scan_feat, k * P.level_px() + 16))) return r;
        return 0;
    };
    // gray -> levels -> conv stack per level -> window tail for k frames staged at d_frames; p / c / b: the predictions of
    // their first window
    auto kernels = [&](cudaStream_t st, const uint8_t* d_frames, int64_t k, float* p, int32_t* c, int32_t* b) -> int {
        int r;
        if ((r = launch_gray(h, st, d_frames, k, plane, h->d_scan_gray.p))) return r;
        PyramidPrep R;
        R.gray = h->d_scan_gray.p; R.out = h->d_scan_gray.p; R.fh = fh; R.fw = fw; R.n_levels = 0;
        const uint8_t* in[kPyramidMaxLevels];
        size_t o = gray_base(k);
        int rows = 0;
        for (int l = 0; l < L; l++) {
            if (P.identity(l)) { in[l] = h->d_scan_gray.p; continue; }
            R.lv[R.n_levels++] = PyramidLevel{P.w[l], P.h[l], rows, P.box(l), o, (size_t)P.w[l] * P.h[l]};
            in[l] = h->d_scan_gray.p + o;
            rows += P.h[l];
            o += k * P.w[l] * P.h[l];
        }
        if (R.n_levels && (r = launch_levels(h, st, R, rows, k))) return r;
        ScanLevel lv[kScanMaxLevels];
        for (int l = 0; l < L; l++) {
            uint8_t* maps = h->d_scan_feat.p + k * P.px[l];
            if ((r = conv_stack_device(h, st, in[l], k, P.h[l], P.w[l], maps, 0, nullptr, nullptr))) return r;
            lv[l] = ScanLevel{maps, P.h[l] / 8, P.w[l] / 8, P.nx[l], (P.w[l] - CNNACC_IMG) / 8, (P.h[l] - CNNACC_IMG) / 8,
                              (int)P.first[l]};
        }
        const TailArgs A = make_tail(h, p, c, b, false, flags);
        if (L == 1) {
            ScanWindows<true> win{(int)per, stride / 8, 1, {lv[0]}};
            return launch_tail_kernel(h, st, win, k * per, A, h->scan_attr_set);
        }
        ScanWindows<false> win{(int)per, stride / 8, L, {}};
        std::copy(lv, lv + L, win.lv);
        return launch_tail_kernel(h, st, win, k * per, A, h->pyramid_attr_set);
    };
    // the merge's region descriptors (f, x, y, w | h << 16) -- the windows' frame rectangles -- and per-frame ranges, uploaded on st
    DescBuf* db = nullptr;
    auto upload_desc = [&](cudaStream_t st) -> int {
        int r;
        if ((r = desc_acquire(h, n * per, &db, n + 1))) return r;
        mg->first.resize((size_t)n + 1);
        for (int64_t f = 0; f <= n; f++) mg->first[f] = f * per;
        int4* d = db->host.p;
        for (int64_t f = 0; f < n; f++)
            for (int l = 0; l < L; l++)
                for (int iy = 0; iy < P.ny[l]; iy++)
                    for (int ix = 0; ix < P.nx[l]; ix++) {
                        const int4 q = P.rect(l, ix, iy);
                        *d++ = make_int4((int)f, q.x, q.y, q.z | q.w << 16);
                    }
        std::memcpy(db->first_host.p, mg->first.data(), (size_t)(n + 1) * sizeof(long long));
        CU(h, cudaMemcpyAsync(db->dev.p, db->host.p, (size_t)(n * per) * sizeof(int4), cudaMemcpyHostToDevice, st));
        CU(h, cudaMemcpyAsync(db->first_dev.p, db->first_host.p, (size_t)(n + 1) * sizeof(long long), cudaMemcpyHostToDevice, st));
        return 0;
    };

    if (flags & CNNACC_FLAG_DEVICE_PTRS) {
        REQUIRE_ALIGNED(h, bbox, 16, "bbox");
        REQUIRE_ALIGNED(h, probs, 4, "probs");
        REQUIRE_ALIGNED(h, cls, 4, "cls");
        if (mg) {
            REQUIRE_ALIGNED(h, mg->det_box, 16, "det_box");
            REQUIRE_ALIGNED(h, mg->n_det, 4, "n_det");
            REQUIRE_ALIGNED(h, mg->det_region, 4, "det_region");
            REQUIRE_ALIGNED(h, mg->det_cls, 4, "det_cls");
            REQUIRE_ALIGNED(h, mg->det_score, 4, "det_score");
        }
        // pieces of whole frames: gray and feature workspaces of at most 256 MiB each, at most kPredSuper windows
        const size_t ws_frame = std::max(plane + resized, P.level_px());
        const int64_t chunk = std::min<int64_t>(n, std::max<int64_t>(1, std::min<int64_t>(((size_t)256 << 20) / ws_frame, kPredSuper / per)));
        if ((rc = grow_ws(chunk))) return rc;
        const size_t cw = (size_t)(chunk * per), w_probs = cw * 16, w_cls = w_probs + cw * nc * 4;   // PredBlock's layout
        if (mg && ((rc = grow(h, h->d_mpred, cw * kPredBytesPerImage)) || (rc = upload_desc(h->stream)))) return rc;
        auto run = [&]() -> int {
            int r;
            for (int64_t f0 = 0; f0 < n; f0 += chunk) {
                const int64_t k = std::min(chunk, n - f0), w0 = f0 * per;
                if (!mg) {
                    if ((r = kernels(h->stream, frames + f0 * frame_sz, k, probs ? probs + w0 * nc : nullptr, cls ? cls + w0 : nullptr,
                                     bbox ? bbox + w0 * 4 : nullptr)))
                        return r;
                    continue;
                }
                int32_t* wb = reinterpret_cast<int32_t*>(h->d_mpred.p);
                float* wp = reinterpret_cast<float*>(h->d_mpred.p + w_probs);
                int32_t* wc = reinterpret_cast<int32_t*>(h->d_mpred.p + w_cls);
                MergeArgs A = merge_args_of_predictions(db->dev.p, w0, wb, wp, wc, nc, *mg);
                A.n_det += f0;
                const size_t o = (size_t)f0 * mg->max_det;
                if (A.det_region) A.det_region += o;
                if (A.det_cls) A.det_cls += o;
                if (A.det_score) A.det_score += o;
                if (A.det_box) A.det_box += o;
                if ((r = kernels(h->stream, frames + f0 * frame_sz, k, wp, wc, wb)) ||
                    (r = launch_merge(h, h->stream, A, *mg, db->first_dev.p, f0, f0 + k)))
                    return r;
            }
            return 0;
        };
        rc = run();
        if (db) CU(h, cudaEventRecord(db->ev, h->stream));   // also after a failed launch: earlier ones may still read it
        return rc;
    }

    // Host pointers: prediction blocks of whole frames, staged in chunks of about 16 MiB of frames (a larger frame alone)
    // through the ring.  A block holds up to kPredSuper windows, or one frame when a frame has more (a pyramid of an 8192 x
    // 8192 frame at stride 8 has 1.34 M): a block never ends inside a frame, since every frame's kernels write its block.
    HostCall call(h);
    if ((rc = call.begin())) return rc;
    const std::vector<int64_t> blocks =
        frame_aligned_blocks([per](int64_t r) { return r / per; }, n * per, std::max<int64_t>(kPredSuper, per));
    const int64_t fpc = std::min<int64_t>(n, std::max<int64_t>(1, (int64_t)(kRegionChunkBytes / frame_sz)));
    const bool small = blocks.size() == 2 && n <= fpc;    // latency path: one chunk, one stream, one result copy
    cudaStream_t st = small ? h->st_k : h->st_h2d;
    if ((rc = grow_ws(fpc)) || (mg && (rc = upload_desc(st)))) return rc;
    PredBlock pred(h);
    auto finish_block = [&](cudaStream_t s, int64_t fa, int64_t fb) -> int {
        if (!mg) return pred.flush(s, probs, cls, bbox, false);
        const MergeArgs A = merge_args_of_predictions(db->dev.p, pred.s0, pred.bbox(pred.s0), pred.probs(pred.s0), pred.cls(pred.s0), nc, *mg);
        return merge_to_host(h, s, A, *mg, db->first_dev.p, fa, fb);
    };
    Slot* s;
    if (small) {
        if ((rc = call.acquire(s, n * frame_sz, 0)) || (rc = pred.start(0, n * per))) return rc;
        CU(h, cudaMemcpyAsync(s->d_in.p, frames, n * frame_sz, cudaMemcpyHostToDevice, st));
        if (!(rc = kernels(st, s->d_in.p, n, pred.probs(0), pred.cls(0), pred.bbox(0)))) rc = finish_block(st, 0, n);
    } else {
        for (size_t bi = 0; !rc && bi + 1 < blocks.size(); bi++) {
            const int64_t fa = blocks[bi] / per, fb = blocks[bi + 1] / per;
            if ((rc = pred.start(blocks[bi], blocks[bi + 1] - blocks[bi]))) break;
            for (int64_t f0 = fa; !rc && f0 < fb; f0 += fpc) {
                const int64_t k = std::min(fpc, fb - f0);
                if ((rc = call.acquire(s, fpc * frame_sz, 0))) break;
                CU(h, cudaMemcpyAsync(s->d_in.p, frames + f0 * frame_sz, k * frame_sz, cudaMemcpyHostToDevice, h->st_h2d));
                if (!(rc = call.staged(*s)) && !(rc = kernels(h->st_k, s->d_in.p, k, pred.probs(f0 * per), pred.cls(f0 * per),
                                                               pred.bbox(f0 * per))))
                    rc = call.released(*s, h->st_k);
            }
            if (!rc) rc = finish_block(h->st_k, fa, fb);
        }
        st = h->st_k;
    }
    if (db) CU(h, cudaEventRecord(db->ev, st));
    if (rc) return rc;
    return call.done(true);                               // finish_block waited for st
}

int cnnacc_scan_frames(cnnacc_handle* h, const uint8_t* frames, int64_t n, int fh, int fw, int stride, float* probs, int32_t* cls,
                       int32_t* bbox, uint32_t flags) {
    return scan_impl(h, frames, n, fh, fw, nullptr, 1, stride, probs, cls, bbox, flags, nullptr);
}

int cnnacc_scan_objects(cnnacc_handle* h, const uint8_t* frames, int64_t n, int fh, int fw, int stride, float score_min, float iou_max,
                        int max_det, int32_t* n_det, int32_t* det_region, int32_t* det_cls, float* det_score, float* det_box,
                        uint32_t flags) {
    if (!h) return CNNACC_ERR_ARG;
    MergeSpec M = make_merge_spec(score_min, iou_max, max_det, n_det, det_region, det_cls, det_score, det_box, flags);
    return scan_impl(h, frames, n, fh, fw, nullptr, 1, stride, nullptr, nullptr, nullptr, flags, &M);
}

int cnnacc_scan_pyramid(cnnacc_handle* h, const uint8_t* frames, int64_t n, int fh, int fw, const int32_t* levels, int n_levels,
                        int stride, float* probs, int32_t* cls, int32_t* bbox, uint32_t flags) {
    if (!h) return CNNACC_ERR_ARG;
    if (!levels) return fail(h, CNNACC_ERR_ARG, "NULL levels");
    return scan_impl(h, frames, n, fh, fw, levels, n_levels, stride, probs, cls, bbox, flags, nullptr);
}

int cnnacc_scan_pyramid_objects(cnnacc_handle* h, const uint8_t* frames, int64_t n, int fh, int fw, const int32_t* levels,
                                int n_levels, int stride, float score_min, float iou_max, int max_det, int32_t* n_det,
                                int32_t* det_region, int32_t* det_cls, float* det_score, float* det_box, uint32_t flags) {
    if (!h) return CNNACC_ERR_ARG;
    if (!levels) return fail(h, CNNACC_ERR_ARG, "NULL levels");
    MergeSpec M = make_merge_spec(score_min, iou_max, max_det, n_det, det_region, det_cls, det_score, det_box, flags);
    return scan_impl(h, frames, n, fh, fw, levels, n_levels, stride, nullptr, nullptr, nullptr, flags, &M);
}

// The pyramid's gray levels alone, [n][sum of h * w] frame-major, then level: gray once per frame, then every level (an
// identity level is copied) in one launch per piece.
int cnnacc_preprocess_pyramid(cnnacc_handle* h, const uint8_t* frames, int64_t n, int fh, int fw, const int32_t* levels,
                              int n_levels, uint8_t* gray, uint32_t flags) {
    int rc;
    if (!h) return CNNACC_ERR_ARG;
    if (n < 0) return fail(h, CNNACC_ERR_ARG, "negative n");
    PyramidPlan P;
    if (const char* why = pyramid_error(fh, fw, levels, n_levels, 0, &P)) return fail(h, CNNACC_ERR_ARG, why);
    if (flags & kNoScanForm)
        return fail(h, CNNACC_ERR_ARG, "BBOX_UPSAMPLED / RECTS / DIRECT / KEEP_MAPS / TWO_KERNELS have no pyramid form");
    if (n == 0) return CNNACC_OK;
    if (!frames || !gray) return fail(h, CNNACC_ERR_ARG, "NULL frame / output pointer");
    CU(h, cudaSetDevice(h->device));
    const size_t frame_sz = (size_t)fh * fw * 3, plane = (size_t)fh * fw, out_sz = P.level_px();
    PyramidPrep R;
    R.fh = fh; R.fw = fw; R.n_levels = P.n_levels;
    int rows = 0;
    for (int l = 0; l < P.n_levels; l++) {
        R.lv[l] = PyramidLevel{P.w[l], P.h[l], rows, P.box(l), P.px[l], out_sz};
        rows += P.h[l];
    }
    // gray of k frames at d_frames, then their levels into out
    auto kernels = [&](cudaStream_t st, const uint8_t* d_frames, int64_t k, uint8_t* out) -> int {
        int r;
        if ((r = launch_gray(h, st, d_frames, k, plane, h->d_scan_gray.p))) return r;
        R.gray = h->d_scan_gray.p; R.out = out;
        return launch_levels(h, st, R, rows, k);
    };
    if (flags & CNNACC_FLAG_DEVICE_PTRS) {
        const int64_t chunk = std::min<int64_t>(n, std::max<int64_t>(1, ((size_t)256 << 20) / plane));   // gray workspace <= 256 MiB
        if ((rc = grow(h, h->d_scan_gray, chunk * plane))) return rc;
        for (int64_t f0 = 0; f0 < n; f0 += chunk)
            if ((rc = kernels(h->stream, frames + f0 * frame_sz, std::min(chunk, n - f0), gray + f0 * out_sz))) return rc;
        return CNNACC_OK;
    }
    // Host pointers: chunks of about 16 MiB of frames (a larger frame alone) through the ring, levels copied out per chunk
    HostCall call(h);
    if ((rc = call.begin())) return rc;
    const int64_t fpc = std::min<int64_t>(n, std::max<int64_t>(1, (int64_t)(kRegionChunkBytes / frame_sz)));
    if ((rc = grow(h, h->d_scan_gray, fpc * plane))) return rc;
    Slot* s;
    for (int64_t f0 = 0; f0 < n; f0 += fpc) {
        const int64_t k = std::min(fpc, n - f0);
        if ((rc = call.acquire(s, fpc * frame_sz, fpc * out_sz))) return rc;
        CU(h, cudaMemcpyAsync(s->d_in.p, frames + f0 * frame_sz, k * frame_sz, cudaMemcpyHostToDevice, h->st_h2d));
        if ((rc = call.staged(*s)) || (rc = kernels(h->st_k, s->d_in.p, k, s->d_out.p)) || (rc = call.computed(*s))) return rc;
        CU(h, cudaMemcpyAsync(gray + f0 * out_sz, s->d_out.p, k * out_sz, cudaMemcpyDeviceToHost, h->st_d2h));
        if ((rc = call.released(*s, h->st_d2h))) return rc;
    }
    return call.finish(h->st_d2h, false);
}

int cnnacc_pyramid_windows_host(int fh, int fw, const int32_t* levels, int n_levels, int stride, int32_t* rects, int64_t cap) {
    PyramidPlan P;
    if (stride < 1 || pyramid_error(fh, fw, levels, n_levels, stride, &P)) return CNNACC_ERR_ARG;
    if (rects) {
        if (cap < P.per()) return CNNACC_ERR_ARG;
        for (int l = 0; l < P.n_levels; l++)
            for (int iy = 0; iy < P.ny[l]; iy++)
                for (int ix = 0; ix < P.nx[l]; ix++) {
                    const int4 q = P.rect(l, ix, iy);
                    *rects++ = 0; *rects++ = q.x; *rects++ = q.y; *rects++ = q.z; *rects++ = q.w;
                }
    }
    return (int)P.per();
}

static int region_plan_host(const RegionRecords& rg, int64_t n_regions, int64_t n_frames, int fh, int fw, int64_t* chunks, int cap) {
    if (n_regions < 0 || n_frames < 0 || (n_regions > 0 && !rg.p) || !chunks || cap < 0) return CNNACC_ERR_ARG;
    int64_t bad;
    if (region_error(rg, n_regions, n_frames, true, fh, fw, &bad)) return CNNACC_ERR_ARG;
    const std::vector<RegionChunk> plan =
        make_region_plan([&](int64_t r) { return rg.frame(r); }, n_regions, (size_t)fh * fw * 3, kPredSuper);
    if ((int64_t)plan.size() > cap) return CNNACC_ERR_ARG;
    for (size_t i = 0; i < plan.size(); i++) {
        chunks[4 * i] = plan[i].f0; chunks[4 * i + 1] = plan[i].f1; chunks[4 * i + 2] = plan[i].r0; chunks[4 * i + 3] = plan[i].r1;
    }
    return (int)plan.size();
}

int cnnacc_region_plan_host(const int32_t* regions, int64_t n_regions, int64_t n_frames, int fh, int fw, int64_t* chunks, int cap) {
    return region_plan_host(RegionRecords(regions, false), n_regions, n_frames, fh, fw, chunks, cap);
}

int cnnacc_rect_plan_host(const int32_t* regions, int64_t n_regions, int64_t n_frames, int fh, int fw, int64_t* chunks, int cap) {
    return region_plan_host(RegionRecords(regions, true), n_regions, n_frames, fh, fw, chunks, cap);
}

int cnnacc_area_tab_host(int side, int* start, int* cnt, float* alpha, int taps_cap) {
    if (side < kRegionMinSide || side > kRegionMaxSide || !start || !cnt || !alpha || taps_cap < 1) return CNNACC_ERR_ARG;
    int taps = 0;
    for (int d = 0; d < kPrepOut; d++) {
        const AreaTaps a = area_taps(side, kPrepOut, d, side % kPrepOut == 0);
        if (a.n > taps_cap) return CNNACC_ERR_ARG;
        taps = std::max(taps, a.n);
        start[d] = a.first; cnt[d] = a.n;
        for (int i = 0; i < taps_cap; i++) alpha[(size_t)d * taps_cap + i] = i < a.n ? area_tap_weight(a, i) : 0.f;
    }
    return taps;
}

int cnnacc_shard_plan_host(int64_t n, int n_handles, int64_t unit_bytes, int64_t* begin, int cap) {
    if (n < 0 || n_handles < 1 || unit_bytes < 1 || !begin) return CNNACC_ERR_ARG;
    const ShardPlan plan = make_shard_plan(n, n_handles, unit_bytes);
    if (cap < plan.m + 1) return CNNACC_ERR_ARG;
    for (int i = 0; i <= plan.m; i++) begin[i] = plan.begin(i);
    return plan.m;
}

int cnnacc_run_batch_sharded(cnnacc_handle* const* hs, int n_handles, const uint8_t* imgs, int64_t n, int H, int W,
                             uint8_t* feats, uint32_t flags, int* failed) {
    const bool ok = valid_hw(H, W) && imgs && feats;
    const size_t in_sz = ok ? (size_t)H * W : 0, out_sz = ok ? (size_t)64 * (H / 8) * (W / 8) : 0;
    return run_sharded(hs, n_handles, n, (int64_t)in_sz, ok, flags, false, failed, [=](cnnacc_handle* h, int64_t lo, int64_t hi) {
        return cnnacc_run_batch(h, imgs + lo * in_sz, hi - lo, H, W, feats + lo * out_sz, flags);
    });
}

int cnnacc_infer_batch_sharded(cnnacc_handle* const* hs, int n_handles, const uint8_t* imgs, int64_t n,
                               float* probs, int32_t* cls, int32_t* bbox, uint32_t flags, int* failed) {
    const size_t img_sz = CNNACC_FEAT_BYTES;
    return run_sharded(hs, n_handles, n, (int64_t)img_sz, imgs != nullptr, flags, true, failed, [=](cnnacc_handle* h, int64_t lo, int64_t hi) {
        const int nc = h->n_cls;                                    // the same on every member (check_members)
        return cnnacc_infer_batch(h, imgs + lo * img_sz, hi - lo, probs ? probs + lo * nc : nullptr, cls ? cls + lo : nullptr,
                                  bbox ? bbox + lo * 4 : nullptr, flags);
    });
}

int cnnacc_detect_frames_sharded(cnnacc_handle* const* hs, int n_handles, const uint8_t* frames, int64_t n, int fh, int fw,
                                 uint8_t* gray128, float* probs, int32_t* cls, int32_t* bbox, uint32_t flags, int* failed) {
    const bool ok = fh > 0 && fw > 0 && (int64_t)fh * fw <= ((int64_t)1 << 40) && frames;
    const size_t frame_sz = ok ? (size_t)fh * fw * 3 : 0, img_sz = CNNACC_FEAT_BYTES;
    return run_sharded(hs, n_handles, n, (int64_t)frame_sz, ok, flags, true, failed, [=](cnnacc_handle* h, int64_t lo, int64_t hi) {
        const int nc = h->n_cls;
        return cnnacc_detect_frames(h, frames + lo * frame_sz, hi - lo, fh, fw, gray128 ? gray128 + lo * img_sz : nullptr,
                                    probs ? probs + lo * nc : nullptr, cls ? cls + lo : nullptr, bbox ? bbox + lo * 4 : nullptr, flags);
    });
}

int cnnacc_probe_int8_peak(cnnacc_handle* h, double target_ms, double* tops, double* ms_out) {
    if (!h || !tops) return fail(h, CNNACC_ERR_ARG, "NULL argument");
    if (!(target_ms > 0.0) || target_ms > 2000.0) return fail(h, CNNACC_ERR_ARG, "target_ms outside (0, 2000]");
    CU(h, cudaSetDevice(h->device));
    int rc;
    Buf<int> d_status;
    if ((rc = grow(h, d_status, 1))) return rc;
    CU(h, cudaMemset(d_status.p, 0, sizeof(int)));
    auto run = [&](int iters, float* ms) -> int {
        CU(h, cudaEventRecord(h->ev_a, h->stream));
        int8_peak_probe_kernel<<<h->sm_count, 32, kProbeSmem, h->stream>>>(iters, d_status.p);
        h->launches++;
        CU(h, cudaGetLastError());
        CU(h, cudaEventRecord(h->ev_b, h->stream));
        CU(h, cudaEventSynchronize(h->ev_b));
        CU(h, cudaEventElapsedTime(ms, h->ev_a, h->ev_b));
        return 0;
    };
    float ms = 0.f;
    const int iters0 = 1 << 15;                                          // calibration: ~2 ms
    if ((rc = run(iters0, &ms)) || (rc = run(iters0, &ms))) return rc;
    double want = (double)iters0 * target_ms / std::max(ms, 1e-3f);
    const int iters = (int)std::min<double>(1 << 30, std::max<double>(iters0, want)) & ~7;
    if ((rc = run(iters, &ms))) return rc;
    int st = 0;
    CU(h, cudaMemcpy(&st, d_status.p, sizeof(int), cudaMemcpyDeviceToHost));
    if (st) return fail(h, CNNACC_ERR_CUDA, "int8 peak probe timed out");
    *tops = (double)h->sm_count * iters * kProbeOpsPerMma / (ms * 1e-3) / 1e12;
    if (ms_out) *ms_out = ms;
    return CNNACC_OK;
}

int cnnacc_register_host(void* p, size_t bytes) {
    if (!p || bytes == 0) return CNNACC_ERR_ARG;
    cudaError_t e = cudaHostRegister(p, bytes, cudaHostRegisterPortable);
    if (e != cudaSuccess) { g_create_error = std::string("cudaHostRegister: ") + cudaGetErrorString(e); return CNNACC_ERR_CUDA; }
    return CNNACC_OK;
}

int cnnacc_unregister_host(void* p) {
    if (!p) return CNNACC_ERR_ARG;
    return cudaHostUnregister(p) == cudaSuccess ? CNNACC_OK : CNNACC_ERR_CUDA;
}

int cnnacc_image_to_gray128(cnnacc_handle* h, const uint8_t* img, int64_t n, int H, int W, int C, uint8_t* gray128, uint32_t flags) {
    int rc;
    if (!h) return CNNACC_ERR_ARG;
    if (n < 0 || H < 1 || W < 1 || H > 32768 || W > 32768 || (C != 1 && C != 3 && C != 4) || n > 65535)
        return fail(h, CNNACC_ERR_ARG, "bad n / size / channels (channels: 1 = L, 3 = RGB, 4 = RGBA; sides up to 32768)");
    if (n == 0) return CNNACC_OK;
    if (!img || !gray128) return fail(h, CNNACC_ERR_ARG, "NULL image / output pointer");
    CU(h, cudaSetDevice(h->device));
    if (H != h->pil_h || W != h->pil_w) {                // Pillow's coefficient tables depend on the input size
        CU(h, cudaDeviceSynchronize());
        const PilTabHost tx = make_pil_tab(W), ty = make_pil_tab(H);
        h->pil_h = h->pil_w = 0;
        if ((rc = grow(h, h->d_pil_kx, tx.k.size())) || (rc = grow(h, h->d_pil_bx, tx.bounds.size())) ||
            (rc = grow(h, h->d_pil_ky, ty.k.size())) || (rc = grow(h, h->d_pil_by, ty.bounds.size())))
            return rc;
        CU(h, cudaMemcpy(h->d_pil_kx.p, tx.k.data(), tx.k.size() * 4, cudaMemcpyHostToDevice));
        CU(h, cudaMemcpy(h->d_pil_bx.p, tx.bounds.data(), tx.bounds.size() * 4, cudaMemcpyHostToDevice));
        CU(h, cudaMemcpy(h->d_pil_ky.p, ty.k.data(), ty.k.size() * 4, cudaMemcpyHostToDevice));
        CU(h, cudaMemcpy(h->d_pil_by.p, ty.bounds.data(), ty.bounds.size() * 4, cudaMemcpyHostToDevice));
        h->pil_kw = tx.ksize; h->pil_kh = ty.ksize; h->pil_h = H; h->pil_w = W;
    }
    const size_t in_bytes = (size_t)n * H * W * C, out_bytes = (size_t)n * kPilOut * kPilOut;
    const bool dev = (flags & CNNACC_FLAG_DEVICE_PTRS) != 0;
    cudaStream_t st = h->stream;
    const uint8_t* d_in = img;
    uint8_t* d_out = gray128;
    if (!dev) {
        if ((rc = grow(h, h->d_pil_in, in_bytes))) return rc;
        if ((rc = grow(h, h->d_pil_out, out_bytes))) return rc;
        CU(h, cudaMemcpyAsync(h->d_pil_in.p, img, in_bytes, cudaMemcpyHostToDevice, st));
        d_in = h->d_pil_in.p; d_out = h->d_pil_out.p;
    }
    const unsigned nu = (unsigned)n;
    if (H > 100 * W && H > kPilOut) {
        // Pillow's order for a very tall image (H > 100 W, so W <= 327): the vertical pass over the source, gray conversion
        // folded in, writes [n][128][W] -- the result itself when W == 128 -- and the horizontal pass reads that
        uint8_t* d_tmp = d_out;
        if (W != kPilOut) {
            if ((rc = grow(h, h->d_pil_tmp, (size_t)n * kPilOut * W))) return rc;
            d_tmp = h->d_pil_tmp.p;
        }
        pil_vertical_kernel<<<dim3(kPilOut, nu), kPilOut, 0, st>>>(d_in, d_tmp, h->d_pil_ky.p, h->d_pil_by.p, h->pil_kh, H, W, C);
        h->launches++;
        if (W != kPilOut) {
            pil_horizontal_kernel<<<dim3(kPilOut, nu), kPilOut, 0, st>>>(d_tmp, d_out, h->d_pil_kx.p, h->d_pil_bx.p, h->pil_kw, kPilOut, W, 1, 0);
            h->launches++;
        }
    } else {
        const bool need_v = H != kPilOut;
        // the horizontal pass (or, at W == 128, the plain gray conversion) writes [n][H][128]: the result itself when H == 128
        uint8_t* d_tmp = d_out;
        if (need_v) {
            if ((rc = grow(h, h->d_pil_tmp, (size_t)n * H * kPilOut))) return rc;
            d_tmp = h->d_pil_tmp.p;
        }
        pil_horizontal_kernel<<<dim3((unsigned)H, nu), kPilOut, 0, st>>>(d_in, d_tmp, h->d_pil_kx.p, h->d_pil_bx.p, h->pil_kw, H, W, C, W == kPilOut);
        h->launches++;
        if (need_v) {
            pil_vertical_kernel<<<dim3(kPilOut, nu), kPilOut, 0, st>>>(d_tmp, d_out, h->d_pil_ky.p, h->d_pil_by.p, h->pil_kh, H, kPilOut, 1);
            h->launches++;
        }
    }
    CU(h, cudaGetLastError());
    if (!dev) {
        CU(h, cudaMemcpyAsync(gray128, d_out, out_bytes, cudaMemcpyDeviceToHost, st));
        CU(h, cudaStreamSynchronize(st));
    }
    return CNNACC_OK;
}

int cnnacc_alloc_host(size_t bytes, void** out) {
    if (!out || bytes == 0) return CNNACC_ERR_ARG;
    *out = nullptr;
    cudaError_t e = cudaHostAlloc(out, bytes, cudaHostAllocPortable);
    if (e != cudaSuccess) { g_create_error = std::string("cudaHostAlloc: ") + cudaGetErrorString(e); return CNNACC_ERR_CUDA; }
    return CNNACC_OK;
}

int cnnacc_free_host(void* p) {
    if (!p) return CNNACC_ERR_ARG;
    return cudaFreeHost(p) == cudaSuccess ? CNNACC_OK : CNNACC_ERR_CUDA;
}

int cnnacc_timer_start(cnnacc_handle* h) {
    if (!h) return CNNACC_ERR_ARG;
    CU(h, cudaSetDevice(h->device));
    CU(h, cudaEventRecord(h->ev_t0, h->stream));
    return CNNACC_OK;
}

int cnnacc_timer_stop(cnnacc_handle* h, float* ms) {
    if (!h || !ms) return CNNACC_ERR_ARG;
    CU(h, cudaEventRecord(h->ev_t1, h->stream));
    CU(h, cudaEventSynchronize(h->ev_t1));
    CU(h, cudaEventElapsedTime(ms, h->ev_t0, h->ev_t1));
    return check_fused_status(h);
}

int cnnacc_synchronize(cnnacc_handle* h) {
    if (!h) return CNNACC_ERR_ARG;
    CU(h, cudaSetDevice(h->device));
    int rc = sync_all(h);
    return rc ? rc : check_fused_status(h);
}

// ---- drop-in for arm_cnn.c:159-162 -------------------------------------------------------------
static std::mutex g_compat_mutex;
static cnnacc_handle* g_compat = nullptr;

int cnn_infer(const uint8_t* input_img, const uint8_t* weights_bin, const int* shifts, uint8_t* output) {
    if (!input_img || !weights_bin || !shifts || !output) return CNNACC_ERR_ARG;
    std::lock_guard<std::mutex> lock(g_compat_mutex);
    int rc;
    if (!g_compat && (rc = cnnacc_create(0, &g_compat))) return rc;
    if (!g_compat->weights_loaded || std::memcmp(g_compat->wbin, weights_bin, CNNACC_WEIGHT_BYTES) != 0)
        if ((rc = cnnacc_load_weights(g_compat, weights_bin, CNNACC_WEIGHT_BYTES))) return rc;
    if ((rc = cnnacc_set_shifts(g_compat, shifts[0], shifts[1], shifts[2]))) return rc;
    return cnnacc_infer_one(g_compat, input_img, output, nullptr, nullptr);
}

}  // extern "C"
