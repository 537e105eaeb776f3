// cnnacc_api.cu -- the C ABI of include/cnnacc.h: handle, host logic, launches.  No CPU compute path.
#include "../../include/cnnacc.h"

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <string>
#include <system_error>
#include <thread>
#include <vector>

#include "conv_direct.cuh"
#include "conv_fused.cuh"
#include "tail.cuh"
#include "int8_peak_probe.cuh"
#include "cam_upsampled.cuh"
#include "preprocess.cuh"
#include "regions.cuh"
#include "region_plan.h"
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

// Pinned host and device copies of one call's region descriptors; ev is recorded after the call's last launch that reads them.
struct DescBuf {
    int4 *host = nullptr, *dev = nullptr;
    size_t cap = 0;
    cudaEvent_t ev = nullptr;
};

struct Slot {
    cudaEvent_t ev_in = nullptr, ev_k = nullptr, ev_out = nullptr;   // H2D landed / kernels done / D2H drained
    uint8_t *d_in = nullptr, *d_out = nullptr;
    int32_t *d_cls = nullptr, *d_bbox = nullptr;            // cnnacc_cam_bbox_batch's classes in and boxes out
    size_t cap_in = 0, cap_out = 0, cap_pred = 0;
};

std::string g_create_error;
std::atomic<int64_t> g_pdl_seq{0};              // programmatic conv-stack launches of ALL handles (see conv_stack_device)

}  // namespace

struct cnnacc_handle {
    int device = 0;
    cudaStream_t own_stream = nullptr, stream = nullptr;
    cudaStream_t st_h2d = nullptr, st_k = nullptr, st_d2h = nullptr;   // one stream per engine for host-pointer batches
    cudaEvent_t ev_t0 = nullptr, ev_t1 = nullptr, ev_a = nullptr, ev_b = nullptr, ev_c = nullptr, ev_done = nullptr;
    int sm_count = 0;
    bool weights_loaded = false, fc_loaded = false, tail_attr_set = false;
    int shifts[3] = {2, 4, 6};                  // SHIFT_L0..2 defaults, pynq_inference.py:83-85
    bool acc24 = false;                         // accumulator width: false = int32 (arm_cnn.c:31), true = 24-bit wrap (accumulator.v:15)
    uint8_t wbin[CNNACC_WEIGHT_BYTES];
    // device-side weights
    uint32_t* d_wdirect = nullptr; size_t wdirect_off[3] = {0, 0, 0};
    FusedWeights fused;                         // packed operands of the fused kernel (conv_fused.cuh)
    float *d_fcw = nullptr, *d_fcb = nullptr; int n_cls = 0;
    float fcw_host[kMaxClasses * 1024], fcb_host[kMaxClasses];   // what d_fcw / d_fcb hold: sharded calls compare members
    // workspaces (grown on demand) for the per-layer path and for infer_batch
    uint8_t *d_l0 = nullptr, *d_l1 = nullptr, *d_feat = nullptr;
    size_t cap_l0 = 0, cap_l1 = 0, cap_feat = 0;
    Slot slots[kSlots];
    // pre-processing (preprocess.cuh): INTER_AREA weight table of the last crop side seen
    int prep_side = 0; AreaTabHost prep_tab;
    int *d_prep_start = nullptr, *d_prep_cnt = nullptr; float* d_prep_alpha = nullptr; size_t cap_prep_alpha = 0;
    uint8_t* d_gray = nullptr; size_t cap_gray = 0;
    DescBuf rdesc[kDescRing]; int rdesc_next = 0;   // region calls (regions_impl)
    // load_image_any (pil_resize.cuh): Pillow coefficient tables of the last (H, W) seen, on the device
    int pil_h = 0, pil_w = 0, pil_kh = 0, pil_kw = 0;
    int32_t *d_pil_kx = nullptr, *d_pil_bx = nullptr, *d_pil_ky = nullptr, *d_pil_by = nullptr;
    uint8_t *d_pil_tmp = nullptr, *d_pil_in = nullptr, *d_pil_out = nullptr; size_t cap_pil_tmp = 0, cap_pil_in = 0, cap_pil_out = 0;
    // the prediction block of host-pointer calls (PredBlock): device block the kernels write, pinned block it is copied to
    uint8_t *d_pred = nullptr, *h_pred = nullptr;
    size_t cap_pred = 0;                            // images the two blocks hold
    // single-image protocol state
    uint8_t *h_img = nullptr, *h_bram = nullptr;    // pinned + mapped: the batch-1 path runs zero-copy on them
    int *h_done = nullptr, *h_done_dev = nullptr;   // mapped completion word of the batch-1 path and its device address
    int done_seq = 0;
    uint8_t *h_img_dev = nullptr, *h_bram_dev = nullptr;   // their device addresses
    CUtensorMap one_map;                            // tensor map over h_img (1 image), encoded once
    bool one_map_ok = false;
    uint8_t *d_img1 = nullptr, *d_bram = nullptr;
    bool image_loaded = false, started = false;
    int64_t launches = 0;
    PdlChain pdl;                                   // overlapped back-to-back conv-stack launches (pdl_chain.h)
    // cnnacc_run_batch_async: completion events of the last kMaxPending submitted calls, and the ring position the staging
    // slots continue from (asynchronous calls share one continuous ring across calls)
    cudaEvent_t ev_ticket[CNNACC_MAX_PENDING] = {};
    int64_t next_ticket = 0, ring_ci = 0;
    std::string err;
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

int grow(cnnacc_handle* h, uint8_t** p, size_t* cap, size_t need) {
    if (*cap >= need) return 0;
    if (*p) CU(h, cudaFree(*p));
    *p = nullptr; *cap = 0;
    CU(h, cudaMalloc(p, need));
    *cap = need;
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

// The tuning overrides the sweeps in tools/ set (CNNACC_PDL, CNNACC_HOST_CHUNK_MB, CNNACC_HOST_RAMP, CNNACC_WS_CHUNK): the
// variable's integer value, or dflt when it is unset.  Each is read once, into a function-local static where it is used.
int env_int(const char* name, int dflt) { const char* e = getenv(name); return e ? atoi(e) : dflt; }

// Which kernels run the conv stack of an H x W call.  128x128 is one fused launch (its maps can also be kept); larger sizes
// run as overlapping 128x128 windows through the fused kernel; everything else, and DIRECT, takes the per-layer kernels.
enum class ConvPath { kFused128, kFusedWindows, kPerLayer };
ConvPath conv_path(const cnnacc_handle* h, int H, int W, uint32_t flags) {
    if (!h->fused.ready || (flags & CNNACC_FLAG_DIRECT)) return ConvPath::kPerLayer;
    if (H == CNNACC_IMG && W == CNNACC_IMG) return ConvPath::kFused128;
    if (H >= CNNACC_IMG && W >= CNNACC_IMG && !(flags & CNNACC_FLAG_KEEP_MAPS)) return ConvPath::kFusedWindows;
    return ConvPath::kPerLayer;
}

// Does the classifier tail of a 128x128 call run inside the fused conv kernel, on the feature map still in shared memory?
bool tail_in_conv(const cnnacc_handle* h, uint32_t flags) {
    return conv_path(h, CNNACC_IMG, CNNACC_IMG, flags) == ConvPath::kFused128 &&
           !(flags & (CNNACC_FLAG_KEEP_MAPS | CNNACC_FLAG_TWO_KERNELS));
}

// One layer of the generic per-layer path on `stream`.
int launch_direct_layer(cnnacc_handle* h, cudaStream_t stream, int layer, const uint8_t* in, uint8_t* out,
                        int64_t n, int H, int W) {
    const int tiles_x = (W + kDirTile - 1) / kDirTile, tiles_y = (H + kDirTile - 1) / kDirTile;
    // image and tile share gridDim.x (2^31-1); gridDim.y (65535) would overflow at 8192x8192 (256 x 256 layer-0 tiles)
    if (n * tiles_x * tiles_y > 0x7fffffffLL) return fail(h, CNNACC_ERR_ARG, "too many tiles in one launch");
    dim3 grid((unsigned)(n * tiles_x * tiles_y), 1u, (unsigned)(kLayers[layer].oc / kDirOcb));
    conv3x3_pool_direct_kernel<<<grid, 256, 0, stream>>>(in, out, h->d_wdirect + h->wdirect_off[layer],
                                                         kLayers[layer].ic, kLayers[layer].oc, H, W,
                                                         h->shifts[layer], tiles_x, tiles_x * tiles_y, h->acc24 ? 1 : 0);
    h->launches++;
    CU(h, cudaGetLastError());
    return 0;
}

// Conv stack for n device-resident images on `stream`.  l0/l1 are workspaces for the per-layer path.
int conv_stack_device(cnnacc_handle* h, cudaStream_t stream, const uint8_t* d_imgs, int64_t n, int H, int W,
                      uint8_t* d_feats, uint32_t flags, uint8_t* d_l0, uint8_t* d_l1) {
    const ConvPath path = conv_path(h, H, W, flags);
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

bool needs_maps(const cnnacc_handle* h, int H, int W, uint32_t flags) {   // only the per-layer path has intermediate maps in HBM
    return conv_path(h, H, W, flags) == ConvPath::kPerLayer || (flags & CNNACC_FLAG_KEEP_MAPS);
}

// images per chunk so that the per-layer workspaces stay around 512 MiB
int64_t chunk_images(int H, int W) {
    const size_t per = (size_t)H * W * 8;
    return (int64_t)std::max<size_t>(1, ((size_t)512 << 20) / per);
}

int ensure_maps(cnnacc_handle* h, int64_t n, int H, int W) {
    int rc;
    // per-layer path: the two intermediate maps
    if ((rc = grow(h, &h->d_l0, &h->cap_l0, (size_t)n * 16 * (H / 2) * (W / 2)))) return rc;
    if ((rc = grow(h, &h->d_l1, &h->cap_l1, (size_t)n * 32 * (H / 4) * (W / 4)))) return rc;
    return 0;
}

TailArgs make_tail(const cnnacc_handle* h, float* d_probs, int32_t* d_cls, int32_t* d_bbox, bool cls_given, uint32_t flags) {
    TailArgs A;
    A.fc_w = h->d_fcw; A.fc_b = h->d_fcb; A.n_cls = h->n_cls;
    A.want_logits = (flags & CNNACC_FLAG_LOGITS) ? 1 : 0;
    A.probs = d_probs; A.bbox_out = d_bbox;
    A.cls_out = cls_given ? nullptr : d_cls;
    A.cls_in = cls_given ? d_cls : nullptr;
    return A;
}

// classify_vec + bbox_vec on n device-resident feature maps (tail.cuh)
int launch_tail(cnnacc_handle* h, cudaStream_t stream, const uint8_t* d_feats, int64_t n, const TailArgs& A) {
    if (n == 0) return 0;
    if (!h->tail_attr_set) {
        CU(h, cudaFuncSetAttribute(classify_bbox_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kTailSmem));
        h->tail_attr_set = true;
    }
    const unsigned grid = (unsigned)std::min<int64_t>((n + kTailGroups - 1) / kTailGroups, h->sm_count);
    classify_bbox_kernel<<<grid, kTailGroups * kTailThreads, kTailSmem, stream>>>(d_feats, (long long)n, A);
    h->launches++;
    CU(h, cudaGetLastError());
    return 0;
}

// Conv stack + tail for m device-resident 128x128 images on `stream`.  The fused kernel's tail warps produce the
// predictions while the features are still in shared memory; d_feat_ws (m x 16 KiB) is written only when the caller needs
// the features afterwards (want_feats) or the per-layer kernels are in use.
int infer_device(cnnacc_handle* h, cudaStream_t stream, const uint8_t* d_imgs, int64_t m, uint8_t* d_feat_ws, bool want_feats,
                 const TailArgs& A, uint32_t flags) {
    if (tail_in_conv(h, flags)) {
        int rc = launch_fused(h->fused, stream, d_imgs, m, want_feats ? d_feat_ws : nullptr, h->shifts, h->sm_count, nullptr, nullptr, &A);
        h->launches++;
        if (rc != 0) return fail(h, CNNACC_ERR_CUDA, std::string("fused launch: ") + cudaGetErrorString((cudaError_t)rc));
        return 0;
    }
    int rc;
    if ((rc = conv_stack_device(h, stream, d_imgs, m, CNNACC_IMG, CNNACC_IMG, d_feat_ws, flags, h->d_l0, h->d_l1))) return rc;
    return launch_tail(h, stream, d_feat_ws, m, A);
}
bool infer_needs_feat_ws(const cnnacc_handle* h, bool want_feats, uint32_t flags) {
    return want_feats || !tail_in_conv(h, flags);
}

// Classifier.get_cam_bbox per image (cam_upsampled.cuh); d_cam may be null
int launch_cam_upsampled(cnnacc_handle* h, cudaStream_t stream, const uint8_t* d_feats, int64_t n, const int32_t* d_cls,
                         int32_t* d_bbox, uint8_t* d_cam) {
    if (n == 0) return 0;
    static const ResampleTab tab = make_resample_tab();
    cam_bbox_upsampled_kernel<<<(unsigned)n, 256, 0, stream>>>(d_feats, h->d_fcw, h->n_cls, d_cls, d_bbox, d_cam, tab);
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
        if (!h->d_prep_start) CU(h, cudaMalloc(&h->d_prep_start, kPrepOut * sizeof(int)));
        if (!h->d_prep_cnt) CU(h, cudaMalloc(&h->d_prep_cnt, kPrepOut * sizeof(int)));
        const size_t ab = h->prep_tab.alpha.size() * sizeof(float);
        if (ab > h->cap_prep_alpha) {
            cudaFree(h->d_prep_alpha); h->d_prep_alpha = nullptr; h->cap_prep_alpha = 0;
            CU(h, cudaMalloc(&h->d_prep_alpha, ab));
            h->cap_prep_alpha = ab;
        }
        CU(h, cudaMemcpy(h->d_prep_start, h->prep_tab.start.data(), kPrepOut * sizeof(int), cudaMemcpyHostToDevice));
        CU(h, cudaMemcpy(h->d_prep_cnt, h->prep_tab.cnt.data(), kPrepOut * sizeof(int), cudaMemcpyHostToDevice));
        CU(h, cudaMemcpy(h->d_prep_alpha, h->prep_tab.alpha.data(), ab, cudaMemcpyHostToDevice));
        h->prep_side = S;
    }
    PrepParams P;
    P.frames = d_frames; P.out = d_gray;
    P.start = h->d_prep_start; P.cnt = h->d_prep_cnt; P.alpha = h->d_prep_alpha;
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
    for (auto st : {h->st_h2d, h->st_k, h->st_d2h}) CU(h, cudaStreamSynchronize(st));
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
    ~HostCall() { if (armed) for (auto st : {h->st_h2d, h->st_k, h->st_d2h}) cudaStreamSynchronize(st); }
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
        if ((rc = grow(h, &s.d_in, &s.cap_in, in_bytes)) || (rc = grow(h, &s.d_out, &s.cap_out, out_bytes))) return rc;
        if (n_pred > s.cap_pred) {
            cudaFree(s.d_cls); cudaFree(s.d_bbox);
            s.d_cls = s.d_bbox = nullptr; s.cap_pred = 0;
            CU(h, cudaMalloc(&s.d_cls, n_pred * sizeof(int32_t)));
            CU(h, cudaMalloc(&s.d_bbox, n_pred * 4 * sizeof(int32_t)));
            s.cap_pred = n_pred;
        }
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
        if ((size_t)count > h->cap_pred) {
            CU(h, cudaStreamSynchronize(h->st_d2h));
            cudaFree(h->d_pred); cudaFreeHost(h->h_pred);
            h->d_pred = h->h_pred = nullptr; h->cap_pred = 0;
            CU(h, cudaMalloc(&h->d_pred, (size_t)count * kPredBytesPerImage));
            CU(h, cudaHostAlloc(&h->h_pred, (size_t)count * kPredBytesPerImage, cudaHostAllocDefault));
            h->cap_pred = (size_t)count;
        }
        s0 = first; m = count;
        return 0;
    }
    int64_t end() const { return s0 + m; }
    size_t off_probs() const { return (size_t)m * 16; }
    size_t off_cls() const { return off_probs() + (size_t)m * h->n_cls * 4; }
    // where the kernels write the predictions of unit u, s0 <= u < end()
    int32_t* bbox(int64_t u) const { return reinterpret_cast<int32_t*>(h->d_pred) + (u - s0) * 4; }
    float* probs(int64_t u) const { return reinterpret_cast<float*>(h->d_pred + off_probs()) + (u - s0) * h->n_cls; }
    int32_t* cls(int64_t u) const { return reinterpret_cast<int32_t*>(h->d_pred + off_cls()) + (u - s0); }
    // the block, after the kernels queued on `st`, into the caller's arrays (indexed from unit 0); waits for st
    int flush(cudaStream_t st, float* probs_out, int32_t* cls_out, int32_t* bbox_out, bool cls_given) {
        CU(h, cudaMemcpyAsync(h->h_pred, h->d_pred, off_cls() + (size_t)m * 4, cudaMemcpyDeviceToHost, st));
        CU(h, cudaStreamSynchronize(st));
        if (bbox_out) std::memcpy(bbox_out + s0 * 4, h->h_pred, (size_t)m * 16);
        if (probs_out) std::memcpy(probs_out + s0 * h->n_cls, h->h_pred + off_probs(), (size_t)m * h->n_cls * 4);
        if (cls_out && !cls_given) std::memcpy(cls_out + s0, h->h_pred + off_cls(), (size_t)m * 4);
        return 0;
    }
};

// The cut of a host-pointer call into staging chunks (host_chunks.h) under the CNNACC_HOST_CHUNK_MB / CNNACC_HOST_RAMP
// overrides.  `ramp`: the call may ramp its chunk sizes up and down at its edges.
HostChunkPlan host_chunk_plan(int64_t n, size_t in_sz, int64_t cap_images, bool pipelined, bool ramp) {
    static const size_t chunk_mb = (size_t)std::max(0, env_int("CNNACC_HOST_CHUNK_MB", 0));
    static const int depth = std::clamp(env_int("CNNACC_HOST_RAMP", 2), 0, 4);
    return make_host_chunk_plan(n, in_sz, cap_images, pipelined, chunk_mb, ramp ? depth : 0);
}

// The host-pointer conv stack: queue the staged copies and kernels of one call on the ring; does not wait for anything.  A
// pipelined call has no ramped chunk sizes: the neighbouring calls keep both copy directions busy at its edges.
int enqueue_host_batch(HostCall& call, const uint8_t* imgs, int64_t n, int H, int W, uint8_t* feats, uint32_t flags) {
    cnnacc_handle* h = call.h;
    int rc;
    const size_t in_sz = (size_t)H * W, out_sz = (size_t)64 * (H / 8) * (W / 8);
    const HostChunkPlan plan = host_chunk_plan(n, in_sz, chunk_images(H, W), call.pipelined, true);
    const int64_t hchunk = plan.full;
    if (needs_maps(h, H, W, flags) && (rc = ensure_maps(h, hchunk, H, W))) return rc;
    if (call.pipelined) {
        // earlier calls may still be using the slots: growing one (free + malloc) waits for the device first
        bool grows = false;
        for (const Slot& s : h->slots) grows |= s.cap_in < hchunk * in_sz || s.cap_out < hchunk * out_sz;
        if (grows) CU(h, cudaDeviceSynchronize());
    }
    int64_t m = 0;
    for (int64_t i0 = 0, ci = 0; i0 < n; i0 += m, ci++) {
        m = plan.next(i0, ci);
        Slot* s;
        if ((rc = call.acquire(s, hchunk * in_sz, hchunk * out_sz))) return rc;
        CU(h, cudaMemcpyAsync(s->d_in, imgs + i0 * in_sz, m * in_sz, cudaMemcpyHostToDevice, h->st_h2d));
        if ((rc = call.staged(*s)) || (rc = conv_stack_device(h, h->st_k, s->d_in, m, H, W, s->d_out, flags, h->d_l0, h->d_l1)) ||
            (rc = call.computed(*s)))
            return rc;
        CU(h, cudaMemcpyAsync(feats + i0 * out_sz, s->d_out, m * out_sz, cudaMemcpyDeviceToHost, h->st_d2h));
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
    cnnacc_handle* h = new cnnacc_handle();
    h->device = device_id;
    auto bail = [&](const char* what, cudaError_t err) {
        g_create_error = std::string(what) + ": " + cudaGetErrorString(err);
        cnnacc_destroy(h);                               // releases whatever was created so far (null members are skipped)
        return CNNACC_ERR_CUDA;
    };
    if ((e = cudaSetDevice(device_id)) != cudaSuccess) return bail("cudaSetDevice", e);
    cudaDeviceProp prop;
    if ((e = cudaGetDeviceProperties(&prop, device_id)) != cudaSuccess) return bail("cudaGetDeviceProperties", e);
    if (prop.major != 10) {
        g_create_error = "device is sm_" + std::to_string(prop.major * 10 + prop.minor) +
                         "; this library is built for sm_100a (B200) only";
        cnnacc_destroy(h);
        return CNNACC_ERR_CUDA;
    }
    h->sm_count = prop.multiProcessorCount;
    if ((e = cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking)) != cudaSuccess) return bail("cudaStreamCreate", e);
    h->stream = h->own_stream;
    cudaEvent_t* evs[] = {&h->ev_t0, &h->ev_t1, &h->ev_a, &h->ev_b, &h->ev_c, &h->ev_done};
    for (auto ev : evs)
        if ((e = cudaEventCreate(ev)) != cudaSuccess) return bail("cudaEventCreate", e);
    for (auto& s : h->slots) {
        for (auto ev : {&s.ev_in, &s.ev_k, &s.ev_out})
            if ((e = cudaEventCreateWithFlags(ev, cudaEventDisableTiming)) != cudaSuccess) return bail("cudaEventCreate", e);
    }
    for (auto& ev : h->ev_ticket)
        if ((e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming)) != cudaSuccess) return bail("cudaEventCreate", e);
    for (auto& b : h->rdesc)
        if ((e = cudaEventCreateWithFlags(&b.ev, cudaEventDisableTiming)) != cudaSuccess) return bail("cudaEventCreate", e);
    for (auto st : {&h->st_h2d, &h->st_k, &h->st_d2h})
        if ((e = cudaStreamCreateWithFlags(st, cudaStreamNonBlocking)) != cudaSuccess) return bail("cudaStreamCreate", e);
    if ((e = cudaHostAlloc(&h->h_img, CNNACC_IMG * CNNACC_IMG, cudaHostAllocMapped)) != cudaSuccess) return bail("cudaHostAlloc", e);
    if ((e = cudaHostAlloc(&h->h_bram, kBramBytes, cudaHostAllocMapped)) != cudaSuccess) return bail("cudaHostAlloc", e);
    if ((e = cudaHostGetDevicePointer(&h->h_img_dev, h->h_img, 0)) != cudaSuccess) return bail("cudaHostGetDevicePointer", e);
    if ((e = cudaHostGetDevicePointer(&h->h_bram_dev, h->h_bram, 0)) != cudaSuccess) return bail("cudaHostGetDevicePointer", e);
    if ((e = cudaHostAlloc(&h->h_done, 64, cudaHostAllocMapped)) != cudaSuccess) return bail("cudaHostAlloc", e);
    *h->h_done = 0;
    if ((e = cudaHostGetDevicePointer(&h->h_done_dev, h->h_done, 0)) != cudaSuccess) return bail("cudaHostGetDevicePointer", e);
    if ((e = cudaHostAlloc(&h->h_pred, kSmallN * kPredBytesPerImage, cudaHostAllocDefault)) != cudaSuccess) return bail("cudaHostAlloc", e);
    if ((e = cudaMalloc(&h->d_pred, kSmallN * kPredBytesPerImage)) != cudaSuccess) return bail("cudaMalloc", e);
    h->cap_pred = kSmallN;
    if ((e = cudaMalloc(&h->d_img1, CNNACC_IMG * CNNACC_IMG)) != cudaSuccess) return bail("cudaMalloc", e);
    if ((e = cudaMalloc(&h->d_bram, kBramBytes)) != cudaSuccess) return bail("cudaMalloc", e);
    *out = h;
    return CNNACC_OK;
}

int cnnacc_destroy(cnnacc_handle* h) {
    if (!h) return CNNACC_ERR_ARG;
    cudaSetDevice(h->device);
    cudaDeviceSynchronize();
    for (auto& s : h->slots) {
        cudaFree(s.d_in); cudaFree(s.d_out); cudaFree(s.d_cls); cudaFree(s.d_bbox);
        for (auto ev : {s.ev_in, s.ev_k, s.ev_out}) if (ev) cudaEventDestroy(ev);
    }
    for (auto st : {h->st_h2d, h->st_k, h->st_d2h}) if (st) cudaStreamDestroy(st);
    for (auto ev : h->ev_ticket) if (ev) cudaEventDestroy(ev);
    for (auto& b : h->rdesc) {
        cudaFreeHost(b.host); cudaFree(b.dev);
        if (b.ev) cudaEventDestroy(b.ev);
    }
    cudaFree(h->d_prep_start); cudaFree(h->d_prep_cnt); cudaFree(h->d_prep_alpha); cudaFree(h->d_gray);
    cudaFree(h->d_pil_kx); cudaFree(h->d_pil_bx); cudaFree(h->d_pil_ky); cudaFree(h->d_pil_by);
    cudaFree(h->d_pil_tmp); cudaFree(h->d_pil_in); cudaFree(h->d_pil_out);
    cudaFree(h->d_wdirect); cudaFree(h->d_fcw); cudaFree(h->d_fcb);
    cudaFree(h->d_l0); cudaFree(h->d_l1); cudaFree(h->d_feat); cudaFree(h->d_img1); cudaFree(h->d_bram);
    fused_free(h->fused);
    cudaFreeHost(h->h_img); cudaFreeHost(h->h_bram); cudaFreeHost(h->h_done); cudaFreeHost(h->h_pred); cudaFree(h->d_pred);
    cudaEvent_t evs[] = {h->ev_t0, h->ev_t1, h->ev_a, h->ev_b, h->ev_c, h->ev_done};
    for (auto ev : evs) if (ev) cudaEventDestroy(ev);
    if (h->own_stream) cudaStreamDestroy(h->own_stream);
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
    CU(h, cudaSetDevice(h->device));
    CU(h, cudaDeviceSynchronize());      // weights may be in use by queued launches
    std::memcpy(h->wbin, weights_bin, n);
    std::vector<uint32_t> packed;
    pack_direct_weights(h->wbin, packed, h->wdirect_off);
    if (!h->d_wdirect) CU(h, cudaMalloc(&h->d_wdirect, packed.size() * sizeof(uint32_t)));
    CU(h, cudaMemcpy(h->d_wdirect, packed.data(), packed.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
    int rc = fused_load_weights(h->fused, h->wbin);
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
    const HostChunkPlan plan = make_host_chunk_plan(n, (size_t)H * W, chunk_images(H, W), pipelined != 0, 0, 2);
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
    const bool maps = needs_maps(h, H, W, flags);
    const int64_t chunk = maps ? std::min<int64_t>(n, chunk_images(H, W)) : n;

    if (flags & CNNACC_FLAG_DEVICE_PTRS) {
        REQUIRE_ALIGNED(h, imgs, 16, "image");
        REQUIRE_ALIGNED(h, feats, 16, "feature");
        if (maps && (rc = ensure_maps(h, chunk, H, W))) return rc;
        for (int64_t i0 = 0; i0 < n; i0 += chunk) {
            const int64_t m = std::min(chunk, n - i0);
            if ((rc = conv_stack_device(h, h->stream, imgs + i0 * in_sz, m, H, W, feats + i0 * out_sz, flags, h->d_l0, h->d_l1)))
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
    if (needs_maps(h, H, W, flags)) return fail(h, CNNACC_ERR_ARG, "this size / flag combination has no asynchronous form: use cnnacc_run_batch");
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
    std::memcpy(h->h_img, img, n);
    h->image_loaded = true;
    return CNNACC_OK;
}

int cnnacc_start(cnnacc_handle* h) {
    int rc;
    if ((rc = check_ready(h))) return rc;
    if (!h->image_loaded) return fail(h, CNNACC_ERR_STATE, "no image loaded (call cnnacc_load_image)");
    CU(h, cudaSetDevice(h->device));
    uint8_t *l0 = h->d_bram, *l1 = h->d_bram + 16 * 4096, *l2 = l1 + 32 * 1024;
    CU(h, cudaMemcpyAsync(h->d_img1, h->h_img, CNNACC_IMG * CNNACC_IMG, cudaMemcpyHostToDevice, h->stream));
    if ((rc = conv_stack_device(h, h->stream, h->d_img1, 1, CNNACC_IMG, CNNACC_IMG, l2, CNNACC_FLAG_KEEP_MAPS, l0, l1))) return rc;
    CU(h, cudaMemcpyAsync(h->h_bram, h->d_bram, kBramBytes, cudaMemcpyDeviceToHost, h->stream));
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
    std::memcpy(out, h->h_bram + off, (size_t)num_values);
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
    uint8_t* h_l2 = h->h_bram + 16 * 4096 + 32 * 1024;
    const auto t0 = std::chrono::steady_clock::now();
    std::memcpy(h->h_img, img, CNNACC_FEAT_BYTES);
    if (h->fused.ready) {
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
            const volatile int* flag = h->h_done;
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
    // generic path (no fused kernel): staged copies around the per-layer kernels
    uint8_t *l0 = h->d_bram, *l1 = h->d_bram + 16 * 4096, *l2 = l1 + 32 * 1024;
    CU(h, cudaMemcpyAsync(h->d_img1, h->h_img, CNNACC_IMG * CNNACC_IMG, cudaMemcpyHostToDevice, h->stream));
    CU(h, cudaEventRecord(h->ev_a, h->stream));
    if ((rc = conv_stack_device(h, h->stream, h->d_img1, 1, CNNACC_IMG, CNNACC_IMG, l2, 0, l0, l1))) return rc;
    CU(h, cudaEventRecord(h->ev_b, h->stream));
    CU(h, cudaMemcpyAsync(h_l2, l2, CNNACC_FEAT_BYTES, cudaMemcpyDeviceToHost, h->stream));
    CU(h, cudaEventRecord(h->ev_c, h->stream));
    CU(h, cudaStreamSynchronize(h->stream));
    std::memcpy(feat, h_l2, CNNACC_FEAT_BYTES);
    if (conv_ms) CU(h, cudaEventElapsedTime(conv_ms, h->ev_a, h->ev_b));
    if (read_ms) CU(h, cudaEventElapsedTime(read_ms, h->ev_b, h->ev_c));
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
    if (!h->d_fcw) CU(h, cudaMalloc(&h->d_fcw, (size_t)kMaxClasses * 1024 * sizeof(float)));
    if (!h->d_fcb) CU(h, cudaMalloc(&h->d_fcb, kMaxClasses * sizeof(float)));
    CU(h, cudaMemcpy(h->d_fcw, fc_w, (size_t)n_cls * 1024 * sizeof(float), cudaMemcpyHostToDevice));
    CU(h, cudaMemcpy(h->d_fcb, fc_b, n_cls * sizeof(float), cudaMemcpyHostToDevice));
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
    const bool maps = src_is_images && needs_maps(h, CNNACC_IMG, CNNACC_IMG, flags);
    const bool cls_given = (flags & CNNACC_FLAG_CLS_GIVEN) != 0;
    if (cls_given && !cls) return fail(h, CNNACC_ERR_ARG, "CNNACC_FLAG_CLS_GIVEN without a cls array");
    const bool upsampled = (flags & CNNACC_FLAG_BBOX_UPSAMPLED) != 0 && bbox;
    if (upsampled && !cls && (flags & CNNACC_FLAG_DEVICE_PTRS))
        return fail(h, CNNACC_ERR_ARG, "CNNACC_FLAG_BBOX_UPSAMPLED with device pointers needs a cls array");
    // images in: does anything after the conv stack need the feature maps in HBM?
    const bool feat_ws = src_is_images && infer_needs_feat_ws(h, upsampled, flags);

    if (flags & CNNACC_FLAG_DEVICE_PTRS) {
        REQUIRE_ALIGNED(h, src, 16, "image / feature");
        REQUIRE_ALIGNED(h, bbox, 16, "bbox");
        REQUIRE_ALIGNED(h, probs, 4, "probs");
        REQUIRE_ALIGNED(h, cls, 4, "cls");
        // one fused launch covers the whole call unless a workspace bounds the chunk
        static const int ws_chunk = env_int("CNNACC_WS_CHUNK", 0);
        const int64_t chunk = feat_ws ? std::min<int64_t>(n, ws_chunk > 0 ? ws_chunk : 16384) : n;
        if (feat_ws) {
            if ((rc = grow(h, &h->d_feat, &h->cap_feat, (size_t)chunk * img_sz))) return rc;
            if (maps && (rc = ensure_maps(h, chunk, CNNACC_IMG, CNNACC_IMG))) return rc;
        }
        for (int64_t i0 = 0; i0 < n; i0 += chunk) {
            const int64_t m = std::min(chunk, n - i0);
            const TailArgs A = make_tail(h, probs ? probs + i0 * nc : nullptr, cls ? cls + i0 : nullptr,
                                         (bbox && !upsampled) ? bbox + i0 * 4 : nullptr, cls_given, flags);
            const uint8_t* f = src + i0 * img_sz;
            if (src_is_images) {
                if ((rc = infer_device(h, h->stream, f, m, h->d_feat, upsampled, A, flags))) return rc;
                f = h->d_feat;
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
        const uint8_t* f = s.d_in;
        int r;
        if (src_is_images) {
            if ((r = infer_device(h, st, s.d_in, m, s.d_out, upsampled, A, flags))) return r;
            f = s.d_out;
        } else if ((r = launch_tail(h, st, f, m, A))) return r;
        return upsampled ? launch_cam_upsampled(h, st, f, m, pred.cls(i0), pred.bbox(i0), nullptr) : 0;
    };
    Slot* s;
    if (n <= kSmallN) {                                      // latency path: one stream, one result copy
        cudaStream_t st = h->st_k;
        if ((rc = call.acquire(s, n * img_sz, feat_ws ? n * img_sz : 0))) return rc;
        if (maps && (rc = ensure_maps(h, n, CNNACC_IMG, CNNACC_IMG))) return rc;
        if ((rc = pred.start(0, n))) return rc;
        CU(h, cudaMemcpyAsync(s->d_in, src, n * img_sz, cudaMemcpyHostToDevice, st));
        if (cls_given) CU(h, cudaMemcpyAsync(pred.cls(0), cls, n * sizeof(int32_t), cudaMemcpyHostToDevice, st));
        if ((rc = kernels(st, *s, 0, n)) || (rc = pred.flush(st, probs, cls, bbox, cls_given))) return rc;
        return call.done(src_is_images);
    }
    // Only the predictions (44 B per image) come back, so the link carries H2D traffic alone: no ramp, and no cap beyond the
    // call's own size.  Nothing is copied out per slot, so a slot is released once its kernels have ended.
    const int64_t hchunk = host_chunk_plan(n, img_sz, INT64_MAX, false, false).full;
    if (maps && (rc = ensure_maps(h, hchunk, CNNACC_IMG, CNNACC_IMG))) return rc;
    for (int64_t s0 = 0; s0 < n; s0 += kPredSuper) {
        if ((rc = pred.start(s0, std::min<int64_t>(kPredSuper, n - s0)))) return rc;
        for (int64_t i0 = s0; i0 < pred.end(); i0 += hchunk) {
            const int64_t m = std::min(hchunk, pred.end() - i0);
            if ((rc = call.acquire(s, hchunk * img_sz, feat_ws ? hchunk * img_sz : 0))) return rc;
            CU(h, cudaMemcpyAsync(s->d_in, src + i0 * img_sz, m * img_sz, cudaMemcpyHostToDevice, h->st_h2d));
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
        CU(h, cudaMemcpyAsync(s->d_in, feats + i0 * feat_sz, m * feat_sz, cudaMemcpyHostToDevice, h->st_h2d));
        if ((rc = call.staged(*s))) return rc;
        pool_features_kernel<<<(unsigned)m, 256, 0, h->st_k>>>(s->d_in, reinterpret_cast<float*>(s->d_out));
        h->launches++;
        CU(h, cudaGetLastError());
        if ((rc = call.computed(*s))) return rc;
        CU(h, cudaMemcpyAsync(pooled + i0 * 1024, s->d_out, m * out_sz, cudaMemcpyDeviceToHost, h->st_d2h));
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
        CU(h, cudaMemcpyAsync(s->d_in, feats + i0 * feat_sz, m * feat_sz, cudaMemcpyHostToDevice, h->st_h2d));
        CU(h, cudaMemcpyAsync(s->d_cls, cls + i0, m * sizeof(int32_t), cudaMemcpyHostToDevice, h->st_h2d));
        if ((rc = call.staged(*s)) ||
            (rc = launch_cam_upsampled(h, h->st_k, s->d_in, m, s->d_cls, bbox ? s->d_bbox : nullptr, cam ? s->d_out : nullptr)) ||
            (rc = call.computed(*s)))
            return rc;
        if (bbox) CU(h, cudaMemcpyAsync(bbox + i0 * 4, s->d_bbox, m * 4 * sizeof(int32_t), cudaMemcpyDeviceToHost, h->st_d2h));
        if (cam)  CU(h, cudaMemcpyAsync(cam + i0 * cam_sz, s->d_out, m * cam_sz, cudaMemcpyDeviceToHost, h->st_d2h));
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
    if (infer_needs_feat_ws(h, ups, 0) && (rc = grow(h, &h->d_feat, &h->cap_feat, (size_t)m * img_sz))) return rc;
    const TailArgs A = make_tail(h, d_probs, d_cls, ups ? nullptr : d_bbox, false, flags);
    if ((rc = infer_device(h, st, base.out, m, h->d_feat, ups, A, 0))) return rc;
    if (ups && (rc = launch_cam_upsampled(h, st, h->d_feat, m, d_cls, d_bbox, nullptr))) return rc;
    return 0;
}

// The next entry of the descriptor ring, with room for n descriptors.  Its previous user -- kDescRing calls ago, possibly an
// asynchronous device-pointer call on any stream -- recorded the entry's event after its last launch that reads it.
static int desc_acquire(cnnacc_handle* h, int64_t n, DescBuf** out) {
    DescBuf& b = h->rdesc[h->rdesc_next];
    h->rdesc_next = (h->rdesc_next + 1) % kDescRing;
    CU(h, cudaEventSynchronize(b.ev));                   // an event never recorded counts as complete
    if ((int64_t)b.cap < n) {
        cudaFreeHost(b.host); cudaFree(b.dev);
        b.host = nullptr; b.dev = nullptr; b.cap = 0;
        CU(h, cudaHostAlloc(&b.host, (size_t)n * sizeof(int4), cudaHostAllocDefault));
        CU(h, cudaMalloc(&b.dev, (size_t)n * sizeof(int4)));
        b.cap = (size_t)n;
    }
    *out = &b;
    return 0;
}

// Shared body of preprocess_bgr / detect_frames (centre: n frames, one centre crop each) and of
// preprocess_regions / detect_regions (n regions over n_frames frames).  gray128 out, predictions out, or both.
static int regions_impl(cnnacc_handle* h, const uint8_t* frames, int64_t n_frames, int fh, int fw, bool centre,
                        const int32_t* regions, int64_t n, uint8_t* gray128, float* probs, int32_t* cls, int32_t* bbox,
                        bool detect, uint32_t flags) {
    int rc;
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
        if (const char* why = region_error(regions, n, n_frames, fh, fw, &bad))
            return fail(h, CNNACC_ERR_ARG, "region " + std::to_string(bad) + ": " + why);
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
        DescBuf* db = nullptr;
        if (!centre) {
            if ((rc = desc_acquire(h, n, &db))) return rc;
            std::memcpy(db->host, regions, (size_t)n * sizeof(int4));
            CU(h, cudaMemcpyAsync(db->dev, db->host, (size_t)n * sizeof(int4), cudaMemcpyHostToDevice, h->stream));
        }
        auto run = [&]() -> int {
            const int64_t chunk = std::min<int64_t>(n, 16384);
            uint8_t* g = gray128;
            int r;
            if (!g && (r = grow(h, &h->d_gray, &h->cap_gray, (size_t)chunk * img_sz))) return r;
            for (int64_t i0 = 0; i0 < n; i0 += chunk) {
                const int64_t m = std::min(chunk, n - i0);
                RegionPrep P = base;
                P.frames = centre ? frames + i0 * frame_sz : frames;
                P.desc = centre ? nullptr : db->dev + i0;
                P.out = g ? g + i0 * img_sz : h->d_gray;
                if ((r = prep_then_tail(h, h->stream, P, m, detect, probs ? probs + i0 * nc : nullptr, cls ? cls + i0 : nullptr,
                                        bbox ? bbox + i0 * 4 : nullptr, flags))) return r;
            }
            return 0;
        };
        rc = run();
        if (db) CU(h, cudaEventRecord(db->ev, h->stream));   // also after a failed launch: earlier ones may still read it
        return rc;
    }

    HostCall call(h);
    if ((rc = call.begin())) return rc;
    const std::vector<RegionChunk> plan =
        make_region_plan([&](int64_t r) -> int64_t { return centre ? r : regions[4 * r]; }, n, frame_sz, kPredSuper);
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
        if ((rc = desc_acquire(h, n, &db))) return rc;
        int64_t below = 0;                               // small: frames staged ahead of the chunk in the one buffer
        for (const RegionChunk& c : plan) {
            for (int64_t r = c.r0; r < c.r1; r++) {
                const int32_t* g = regions + 4 * r;
                db->host[r] = make_int4((int)(g[0] - c.f0 + (small ? below : 0)), g[1], g[2], g[3]);
            }
            below += c.f1 - c.f0;
        }
        CU(h, cudaMemcpyAsync(db->dev, db->host, (size_t)n * sizeof(int4), cudaMemcpyHostToDevice, small ? h->st_k : h->st_h2d));
    }
    auto region_base = [&](const uint8_t* d_frames, int64_t r, int64_t r_frame0, uint8_t* d_gray) {
        RegionPrep P = base;
        P.frames = centre ? d_frames + (r - r_frame0) * frame_sz : d_frames;
        P.desc = centre ? nullptr : db->dev + r;
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
            CU(h, cudaMemcpyAsync(s->d_in + off, frames + plan[k].f0 * frame_sz, bytes, cudaMemcpyHostToDevice, st));
            off += bytes;
            k = j;
        }
        if ((rc = prep_then_tail(h, st, region_base(s->d_in, 0, 0, s->d_out), n, detect, pred.probs(0), pred.cls(0), pred.bbox(0), flags)))
            return rc;
        if (db) CU(h, cudaEventRecord(db->ev, st));
        if (gray128) CU(h, cudaMemcpyAsync(gray128, s->d_out, n * img_sz, cudaMemcpyDeviceToHost, st));
        if (detect && (rc = pred.flush(st, probs, cls, bbox, false))) return rc;
        return detect ? call.done(true) : call.finish(st, false);
    }
    // Staged chunks of about 16 MiB of frames through the ring (HostCall).  A chunk's regions run in launches of up to
    // kRegionLaunch: their gray images fill the slot's output buffer, so a launch after the first waits for the gray copy of
    // the launch before.
    const int64_t per_launch = std::min<int64_t>(max_regions, kRegionLaunch);
    if (detect && (rc = pred.start(0, std::min<int64_t>(kPredSuper, n)))) return rc;
    for (const RegionChunk& c : plan) {
        if (detect && c.r0 >= pred.end()) {              // the plan never lets a chunk straddle a block edge
            if ((rc = pred.flush(h->st_k, probs, cls, bbox, false)) ||
                (rc = pred.start(pred.end(), std::min<int64_t>(kPredSuper, n - pred.end()))))
                return rc;
        }
        if ((rc = call.acquire(s, max_stage, per_launch * img_sz))) return rc;
        CU(h, cudaMemcpyAsync(s->d_in, frames + c.f0 * frame_sz, (size_t)(c.f1 - c.f0) * frame_sz, cudaMemcpyHostToDevice, h->st_h2d));
        if ((rc = call.staged(*s))) return rc;
        for (int64_t r = c.r0; r < c.r1; r += per_launch) {
            const int64_t m = std::min(per_launch, c.r1 - r);
            if (r > c.r0 && gray128 && (rc = call.wait_released(*s, h->st_k))) return rc;
            if ((rc = prep_then_tail(h, h->st_k, region_base(s->d_in, r, c.r0, s->d_out), m, detect, detect ? pred.probs(r) : nullptr,
                                     detect ? pred.cls(r) : nullptr, detect ? pred.bbox(r) : nullptr, flags)) ||
                (rc = call.computed(*s)))
                return rc;
            if (gray128) CU(h, cudaMemcpyAsync(gray128 + r * img_sz, s->d_out, m * img_sz, cudaMemcpyDeviceToHost, h->st_d2h));
            if ((rc = call.released(*s, h->st_d2h))) return rc;
        }
    }
    if (db) CU(h, cudaEventRecord(db->ev, h->st_k));
    if (detect && (rc = pred.flush(h->st_k, probs, cls, bbox, false))) return rc;
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

int cnnacc_region_plan_host(const int32_t* regions, int64_t n_regions, int64_t n_frames, int fh, int fw, int64_t* chunks, int cap) {
    if (n_regions < 0 || n_frames < 0 || (n_regions > 0 && !regions) || !chunks || cap < 0) return CNNACC_ERR_ARG;
    int64_t bad;
    if (region_error(regions, n_regions, n_frames, fh, fw, &bad)) return CNNACC_ERR_ARG;
    const std::vector<RegionChunk> plan =
        make_region_plan([&](int64_t r) -> int64_t { return regions[4 * r]; }, n_regions, (size_t)fh * fw * 3, kPredSuper);
    if ((int64_t)plan.size() > cap) return CNNACC_ERR_ARG;
    for (size_t i = 0; i < plan.size(); i++) {
        chunks[4 * i] = plan[i].f0; chunks[4 * i + 1] = plan[i].f1; chunks[4 * i + 2] = plan[i].r0; chunks[4 * i + 3] = plan[i].r1;
    }
    return (int)plan.size();
}

int cnnacc_area_tab_host(int side, int* start, int* cnt, float* alpha, int taps_cap) {
    if (side < kRegionMinSide || side > kRegionMaxSide || !start || !cnt || !alpha || taps_cap < 1) return CNNACC_ERR_ARG;
    int taps = 0;
    for (int d = 0; d < kPrepOut; d++) {
        const AreaTaps a = area_taps(side, d);
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
    int* d_status = nullptr;
    CU(h, cudaMalloc(&d_status, sizeof(int)));
    CU(h, cudaMemset(d_status, 0, sizeof(int)));
    auto run = [&](int iters, float* ms) -> int {
        CU(h, cudaEventRecord(h->ev_a, h->stream));
        int8_peak_probe_kernel<<<h->sm_count, 32, kProbeSmem, h->stream>>>(iters, d_status);
        h->launches++;
        CU(h, cudaGetLastError());
        CU(h, cudaEventRecord(h->ev_b, h->stream));
        CU(h, cudaEventSynchronize(h->ev_b));
        CU(h, cudaEventElapsedTime(ms, h->ev_a, h->ev_b));
        return 0;
    };
    int rc; float ms = 0.f;
    const int iters0 = 1 << 15;                                          // calibration: ~2 ms
    if ((rc = run(iters0, &ms)) || (rc = run(iters0, &ms))) { cudaFree(d_status); return rc; }
    double want = (double)iters0 * target_ms / std::max(ms, 1e-3f);
    const int iters = (int)std::min<double>(1 << 30, std::max<double>(iters0, want)) & ~7;
    if ((rc = run(iters, &ms))) { cudaFree(d_status); return rc; }
    int st = 0;
    const cudaError_t e_st = cudaMemcpy(&st, d_status, sizeof(int), cudaMemcpyDeviceToHost);
    cudaFree(d_status);
    CU(h, e_st);
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
        for (int32_t** p : {&h->d_pil_kx, &h->d_pil_bx, &h->d_pil_ky, &h->d_pil_by}) { cudaFree(*p); *p = nullptr; }
        h->pil_h = h->pil_w = 0;
        CU(h, cudaMalloc(&h->d_pil_kx, tx.k.size() * 4)); CU(h, cudaMalloc(&h->d_pil_bx, tx.bounds.size() * 4));
        CU(h, cudaMalloc(&h->d_pil_ky, ty.k.size() * 4)); CU(h, cudaMalloc(&h->d_pil_by, ty.bounds.size() * 4));
        CU(h, cudaMemcpy(h->d_pil_kx, tx.k.data(), tx.k.size() * 4, cudaMemcpyHostToDevice));
        CU(h, cudaMemcpy(h->d_pil_bx, tx.bounds.data(), tx.bounds.size() * 4, cudaMemcpyHostToDevice));
        CU(h, cudaMemcpy(h->d_pil_ky, ty.k.data(), ty.k.size() * 4, cudaMemcpyHostToDevice));
        CU(h, cudaMemcpy(h->d_pil_by, ty.bounds.data(), ty.bounds.size() * 4, cudaMemcpyHostToDevice));
        h->pil_kw = tx.ksize; h->pil_kh = ty.ksize; h->pil_h = H; h->pil_w = W;
    }
    const size_t in_bytes = (size_t)n * H * W * C, out_bytes = (size_t)n * kPilOut * kPilOut;
    const bool dev = (flags & CNNACC_FLAG_DEVICE_PTRS) != 0;
    cudaStream_t st = h->stream;
    const uint8_t* d_in = img;
    uint8_t* d_out = gray128;
    if (!dev) {
        if ((rc = grow(h, &h->d_pil_in, &h->cap_pil_in, in_bytes))) return rc;
        if ((rc = grow(h, &h->d_pil_out, &h->cap_pil_out, out_bytes))) return rc;
        CU(h, cudaMemcpyAsync(h->d_pil_in, img, in_bytes, cudaMemcpyHostToDevice, st));
        d_in = h->d_pil_in; d_out = h->d_pil_out;
    }
    const unsigned nu = (unsigned)n;
    if (H > 100 * W && H > kPilOut) {
        // Pillow's order for a very tall image (H > 100 W, so W <= 327): the vertical pass over the source, gray conversion
        // folded in, writes [n][128][W] -- the result itself when W == 128 -- and the horizontal pass reads that
        uint8_t* d_tmp = d_out;
        if (W != kPilOut) {
            if ((rc = grow(h, &h->d_pil_tmp, &h->cap_pil_tmp, (size_t)n * kPilOut * W))) return rc;
            d_tmp = h->d_pil_tmp;
        }
        pil_vertical_kernel<<<dim3(kPilOut, nu), kPilOut, 0, st>>>(d_in, d_tmp, h->d_pil_ky, h->d_pil_by, h->pil_kh, H, W, C);
        h->launches++;
        if (W != kPilOut) {
            pil_horizontal_kernel<<<dim3(kPilOut, nu), kPilOut, 0, st>>>(d_tmp, d_out, h->d_pil_kx, h->d_pil_bx, h->pil_kw, kPilOut, W, 1, 0);
            h->launches++;
        }
    } else {
        const bool need_v = H != kPilOut;
        // the horizontal pass (or, at W == 128, the plain gray conversion) writes [n][H][128]: the result itself when H == 128
        uint8_t* d_tmp = d_out;
        if (need_v) {
            if ((rc = grow(h, &h->d_pil_tmp, &h->cap_pil_tmp, (size_t)n * H * kPilOut))) return rc;
            d_tmp = h->d_pil_tmp;
        }
        pil_horizontal_kernel<<<dim3((unsigned)H, nu), kPilOut, 0, st>>>(d_in, d_tmp, h->d_pil_kx, h->d_pil_bx, h->pil_kw, H, W, C, W == kPilOut);
        h->launches++;
        if (need_v) {
            pil_vertical_kernel<<<dim3(kPilOut, nu), kPilOut, 0, st>>>(d_tmp, d_out, h->d_pil_ky, h->d_pil_by, h->pil_kh, H, kPilOut, 1);
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
