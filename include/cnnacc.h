/*
 * cnnacc.h -- C ABI of the B200 conv-stack accelerator (libcnnacc.so).
 *
 * This is the drop-in boundary for the reference's hot path.  Every entry point is extern "C",
 * takes plain pointers and sizes, returns an int status, and never lets a C++ exception or a
 * torch type cross.  Each one names the reference interface it replaces (file:line under
 * /root/reference/).  INTEGRATION.md shows the ctypes stubs a maintainer of the reference adds.
 *
 * Status codes (SURVEY.md 8b "Error conventions"):
 *    0  success
 *   -1  timeout                       (fast_readout.c:91 start_and_wait -> -1; Python: TimeoutError)
 *   -2  bad argument / size / state   (pynq_inference.py:189,214 asserts;      Python: ValueError)
 *   -3  CUDA error                    (pynq_inference.py:128 RuntimeError;     Python: RuntimeError)
 *   -4  not initialised: no weights / no classifier / no image loaded          (Python: RuntimeError)
 * There is no CPU fallback: without a CUDA device every call that computes returns -3.
 *
 * Pointers: host pointers may have any alignment (they are copied through the library's own staging buffers).  With
 * CNNACC_FLAG_DEVICE_PTRS the image / feature / gray128 / bbox / pooled pointers must be 16-byte aligned and the probs / cls /
 * cam pointers 4-byte aligned (they feed TMA descriptors, bulk stores and 128-bit accesses); anything else returns -2.
 *
 * Threading: one handle = one device + one stream.  A handle is not thread-safe (neither is the
 * reference: arm_cnn.c:30-32 static scratch); distinct handles are independent.  The cnnacc_*_sharded calls spread one host
 * batch over several handles, one thread per handle.
 */
#ifndef CNNACC_H
#define CNNACC_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CNNACC_OK            0
#define CNNACC_ERR_TIMEOUT  (-1)
#define CNNACC_ERR_ARG      (-2)
#define CNNACC_ERR_CUDA     (-3)
#define CNNACC_ERR_STATE    (-4)

#define CNNACC_WEIGHT_BYTES  23184   /* 144 + 4608 + 18432          arm_cnn.c:169-173 */
#define CNNACC_IMG           128     /* native image side            arm_cnn.c:165     */
#define CNNACC_FEAT_CH       64      /* final channels               arm_cnn.c:167     */
#define CNNACC_FEAT_BYTES    16384   /* 64 x 16 x 16                 arm_cnn.c:155     */
#define CNNACC_BRAM_CHANNELS 112     /* 16 + 32 + 64 feature BRAMs   cnn_acc_top.v:48-54 */
#define CNNACC_L2_CH_OFFSET  48      /* CH_OFF                       realtime_detect.py:33 */

/* flags for the batch calls */
#define CNNACC_FLAG_DEVICE_PTRS   0x1u  /* image / feature / result pointers are device memory of the handle's GPU */
#define CNNACC_FLAG_DIRECT        0x2u  /* use the generic per-layer kernels even for 128x128 (cross-check path) */
#define CNNACC_FLAG_KEEP_MAPS     0x4u  /* keep image 0's layer-0/1 maps for cnnacc_read_feature_map (BRAM ch 0-47) */
#define CNNACC_FLAG_CLS_GIVEN     0x8u  /* classify_batch: cls[] is an INPUT (bbox_vec's cls_idx argument), not written */
#define CNNACC_FLAG_BBOX_UPSAMPLED 0x10u /* classify_batch / infer_batch: bbox = Classifier.get_cam_bbox (pynq_inference.py:349-408:
                                            u8 CAM -> PIL bilinear 16->128 -> percentile / 0.2 floor -> pad 3) instead of bbox_vec */
#define CNNACC_FLAG_TWO_KERNELS   0x40u /* infer_batch / detect_frames: write the features to a workspace and run the features-in
                                            tail kernel on them instead of the tail warps inside the conv-stack kernel (A/B path) */
#define CNNACC_FLAG_LOGITS        0x20u /* classify_batch / infer_batch / detect_frames: probs[] receives the raw fp32 logits
                                            W.pooled + b (realtime_detect.py:79) instead of their softmax -- the quantity the
                                            1e-5-relative parity bar is stated on */

typedef struct cnnacc_handle cnnacc_handle;

/* ---- lifetime ------------------------------------------------------------------------------
 * Replaces Overlay(bitstream) + IP/DMA discovery (pynq_inference.py:98-155, realtime_detect.py:247-286)
 * and open_devmem (fast_readout.c:99-113; NULL on failure -> here *out = NULL and a negative code). */
int cnnacc_create(int device_id, cnnacc_handle **out);
int cnnacc_destroy(cnnacc_handle *h);
/* Run later launches on a caller-owned CUDA stream (cudaStream_t as void*); NULL -> the handle's own. */
int cnnacc_set_stream(cnnacc_handle *h, void *cuda_stream);
/* Last error text of this handle (or of create when h == NULL).  Never NULL. */
const char *cnnacc_last_error(const cnnacc_handle *h);
/* Number of kernels this handle has launched since creation (bench.py's gpu_launches). */
int64_t cnnacc_launch_count(const cnnacc_handle *h);

/* ---- configuration -------------------------------------------------------------------------
 * load_weights: the one-off DMA of weights.bin into weight BRAM (pynq_inference.py:186-207,
 * realtime_detect.py:288-296); n must be 23184.  parse_kernels (arm_cnn.c:43-59) runs here once,
 * not per image (arm_cnn.c:186).  A load that fails after its argument checks leaves the handle
 * without weights: calls that need them return -4 until a load succeeds. */
int cnnacc_load_weights(cnnacc_handle *h, const uint8_t *weights_bin, size_t n);
/* set_shifts: AXI reg 10 write, s0 | s1<<5 | s2<<10 (pynq_inference.py:226-229).  The hardware
 * masks with 0x1F; here values outside 0..31 are rejected with -2 (C >> by >=32 is undefined). */
int cnnacc_set_shifts(cnnacc_handle *h, int s0, int s1, int s2);
int cnnacc_get_shifts(const cnnacc_handle *h, int *s3);
/* Accumulator width of the conv stack.  32 (default) = arm_cnn.c:31,106 (int32, never wraps: the parity target).
 * 24 = the PL accumulator (rtl/core/accumulator.v:15 `reg signed [23:0]`) and the trainer's bit-accurate model
 * (training/train_cnn.py:101-116 fpga_conv_layer: ((out + 2^23) mod 2^24) - 2^23 before the shift): every finished sum is
 * wrapped to 24-bit two's complement BEFORE the 2x2 pool.  Only layer 2 can reach 2^23 (32*9*255*128 = 9.4 M); the shipped
 * weights never do.  The RTL's spatial quirks (bottom-right window anchor, no left/right padding) are NOT modelled. */
int cnnacc_set_accumulator_bits(cnnacc_handle *h, int bits);
int cnnacc_get_accumulator_bits(const cnnacc_handle *h);
/* Host-only view of the one-off weight permutation (parse_kernels, arm_cnn.c:43-59, hoisted out of the
 * per-image path): weights.bin -> the fused kernel's operand images.  No GPU needed; tests/ re-derive the conv
 * from these buffers to pin the packed layouts.  w0: 96 dp4a words
 * [oc][lo0..2,hi0..2] followed by 256 layer-0 mma.sync B-fragment words [block][lane]; b1: 24576 B; b2: 18432 B. */
#define CNNACC_PACK_W0_WORDS 352
#define CNNACC_PACK_B1_BYTES 24576
#define CNNACC_PACK_B2_BYTES 18432
int cnnacc_pack_weights_host(const uint8_t *weights_bin, size_t n, uint32_t *w0, uint8_t *b1, uint8_t *b2);

/* Host-only replay of the bookkeeping behind the overlapped conv-stack launches (csrc/pdl_chain.h; DESIGN.md section 4): for
 * a sequence of device-pointer cnnacc_run_batch launches i -- ranges[4i..4i+3] = input begin / end, output begin / end
 * addresses, n_images[i], stream_id[i], foreign_before[i] bit 0 = another kernel of the handle was launched in between, bit 1 =
 * another handle launched a conv stack in between -- wait_out[i] = 1 when launch i must wait for its predecessor before touching
 * memory, 0 when it may overlap it.  No GPU needed; tests/ check the dependency rules with it. */
int cnnacc_pdl_chain_host(int n_launches, const uint64_t *ranges, const int64_t *n_images, const int32_t *stream_id,
                          const int32_t *foreign_before, int sm_count, int32_t *wait_out);

/* Host-only view of the window plan used for images larger than 128x128 (csrc/tiling.cuh): along one dimension with
 * n_out = size/8 outputs, window i starts at output origin[i] (pixel 8*origin[i]) and owns outputs [first[i], end[i]).
 * Returns the number of windows (<= cap) or a negative code.  The FPGA's analogue is the 4-tile drain of layer 0
 * (layer_fsm.v:66-75,205-213); tests/ check that the plan owns every output exactly once and only where it is valid. */
int cnnacc_tile_plan_host(int n_out, int *origin, int *first, int *end, int cap);

/* Host-only view of how a host-pointer cnnacc_run_batch (pipelined = 0) or cnnacc_run_batch_async (pipelined = 1) call of n
 * H x W images is cut into staging chunks (csrc/host_chunks.h): sizes[i] = images in chunk i.  Returns the number of chunks
 * (<= cap) or a negative code.  No GPU needed; tests/ check that every plan covers the call exactly once. */
int cnnacc_chunk_plan_host(int64_t n, int H, int W, int pipelined, int64_t *sizes, int cap);

/* ---- the hot path: batched conv stack ------------------------------------------------------
 * Replaces cnn_infer (arm_cnn.c:159-198) / FPGAEngine.run (realtime_detect.py:313-363) for n images.
 *   imgs  : [n][H][W] u8          feats : [n][64][H/8][W/8] u8   (CHW per image, arm_cnn.c:64-65)
 * H, W multiples of 16.  128x128 runs the fused sm_100a kernel; larger sizes run as overlapping 128x128 windows through
 * the same kernel (halo recompute, csrc/tiling.cuh); smaller ones (and CNNACC_FLAG_DIRECT) the generic per-layer kernels.
 * Host pointers: the call stages through pinned buffers, overlapping H2D / compute / D2H, and
 * returns when feats is complete.  Device pointers: asynchronous on the handle's stream. */
int cnnacc_run_batch(cnnacc_handle *h, const uint8_t *imgs, int64_t n, int H, int W,
                     uint8_t *feats, uint32_t flags);

/* The same call for a STREAM of host batches (the camera loop of realtime_detect.py:575-598 turned into a pipeline):
 * cnnacc_run_batch_async queues the staged copies and kernels of one batch of HOST buffers and returns a ticket at once;
 * cnnacc_wait_batch(ticket) returns when that batch's features are in `feats`.  Batches complete in submission order and share
 * one staging ring, so the H2D of batch k+1 overlaps the kernels and the D2H of batch k (a synchronous call leaves the link idle
 * in one direction during its first H2D and its last D2H).  imgs / feats should be page-locked (cnnacc_alloc_host /
 * cnnacc_register_host; pageable memory makes the copies synchronous) and must stay untouched until the ticket was waited for.
 * At most CNNACC_MAX_PENDING batches are outstanding: submitting one more first waits for the oldest.  Any synchronous
 * host-pointer call, cnnacc_synchronize and cnnacc_destroy wait for everything pending.  Sizes / flags that need the per-layer
 * workspaces (sides below 128, CNNACC_FLAG_DIRECT, CNNACC_FLAG_KEEP_MAPS) have no asynchronous form (CNNACC_ERR_ARG). */
#define CNNACC_MAX_PENDING 8
int cnnacc_run_batch_async(cnnacc_handle *h, const uint8_t *imgs, int64_t n, int H, int W,
                           uint8_t *feats, uint32_t flags, int64_t *ticket);
int cnnacc_wait_batch(cnnacc_handle *h, int64_t ticket);

/* ---- single-image register-style protocol (CNNAccelerator / fast_readout.c) ----------------
 * load_image   : DMA of one 128x128 image into input BRAM        (pynq_inference.py:209-224)
 * start        : control reg bit 0                                (pynq_inference.py:231-234)
 * status       : status reg: bit0 busy, bit1 done, bits3:2 layer (pynq_inference.py:65, :240-246)
 * wait         : start_and_wait's poll loop, 0 or -1 on timeout  (fast_readout.c:77-92)
 * read_features: read_features_full, n_ch x 256 bytes from BRAM channel ch_off (fast_readout.c:33-45)
 * read_feature_map: read_feature_map(channel, n) over the 112-channel map: 0-15 layer 0 (4096 B each),
 *                16-47 layer 1 (1024 B), 48-111 layer 2 (256 B)   (pynq_inference.py:253-265, cnn_acc_top.v:48-54) */
int cnnacc_load_image(cnnacc_handle *h, const uint8_t *img, size_t n);
int cnnacc_start(cnnacc_handle *h);
int cnnacc_status(cnnacc_handle *h);
int cnnacc_wait(cnnacc_handle *h, int timeout_us);
int cnnacc_read_features(cnnacc_handle *h, uint8_t *out, int n_ch, int ch_off);
int cnnacc_read_feature_map(cnnacc_handle *h, int channel, int num_values, uint8_t *out);
/* One image in, features out, lowest latency (FPGAEngine.run / ARMEngine.run shape,
 * realtime_detect.py:313-363,422-436).  128x128 runs zero-copy: the kernel reads the image from and writes the
 * features to mapped pinned host memory (one launch + one sync).  conv_ms = wall time from the call to "done"
 * (the reference times the same span with time.time(), realtime_detect.py:325-335); read_ms = the copy into feat. */
int cnnacc_infer_one(cnnacc_handle *h, const uint8_t *img, uint8_t *feat, float *conv_ms, float *read_ms);

/* ---- follow-on kernels: spatial-bin pool + linear + softmax + CAM bbox ---------------------
 * load_classifier: fc_w [n_cls][1024] f32 row-major, fc_b [n_cls] (realtime_detect.py:533-545), n_cls <= 16.
 *                  Weights must be finite with |w| < 2^100 (else -2).
 * classify_batch : classify_vec + bbox_vec (realtime_detect.py:68-116) on feats [n][64][256] u8.
 *                  probs [n][n_cls] f32, cls [n] i32, bbox [n][4] i32 (x1,y1,x2,y2); any output may be NULL.
 * infer_batch    : run_batch (128x128) followed by classify_batch without the features leaving the GPU. */
int cnnacc_load_classifier(cnnacc_handle *h, const float *fc_w, const float *fc_b, int n_cls);
int cnnacc_classify_batch(cnnacc_handle *h, const uint8_t *feats, int64_t n,
                          float *probs, int32_t *cls, int32_t *bbox, uint32_t flags);
int cnnacc_infer_batch(cnnacc_handle *h, const uint8_t *imgs, int64_t n,
                       float *probs, int32_t *cls, int32_t *bbox, uint32_t flags);
/* pool_features  : feats [n][64][256] u8 -> pooled [n][1024] f32, pooled[ch*16 + r*4 + c] = mean(4x4 bin) / 255: the classifier
 *                  input the trainer builds from a feature dump (retrain_classifier.py:188-205; pynq_inference.py:325-334).
 *                  Exact: equal to the numpy result bit for bit.  Needs no weights or classifier. */
int cnnacc_pool_features(cnnacc_handle *h, const uint8_t *feats, int64_t n, float *pooled, uint32_t flags);
/* cam_bbox_batch : Classifier.get_cam_bbox(features, class_idx, img_size=128) (pynq_inference.py:349-408) per image:
 *                  feats [n][64][256] u8, cls [n] i32 (the class_idx argument) -> bbox [n][4] i32 (x1,y1,x2,y2) and,
 *                  when cam != NULL, cam [n][128][128] u8 = the upsampled map (the reference's cam_full is cam/255 as f32).
 *                  Pillow's BILINEAR resize of an 8-bit image is integer arithmetic and is reproduced bit for bit. */
int cnnacc_cam_bbox_batch(cnnacc_handle *h, const uint8_t *feats, int64_t n, const int32_t *cls,
                          int32_t *bbox, uint8_t *cam, uint32_t flags);

/* ---- the step in front of the hot path in the real-time loop (realtime_detect.py:582-591) ------------------
 * preprocess_bgr: frames [n][fh][fw][3] u8 BGR (cv2 frames) -> gray128 [n][128][128] u8 =
 *                 centre-crop to the square of side min(fh,fw), cv2.cvtColor(BGR2GRAY), cv2.resize((128,128), INTER_AREA);
 *                 OpenCV's fixed-point gray and all three INTER_AREA arithmetic paths are reproduced bit for bit
 *                 (pinned against cv2 4.13.0).  The crop side must be 128..8192.
 * detect_frames : one iteration of the loop body (:582-598) per frame: preprocess -> conv stack -> classify_vec -> bbox_vec
 *                 (or get_cam_bbox with CNNACC_FLAG_BBOX_UPSAMPLED) without anything but the predictions leaving the GPU;
 *                 gray128 may be NULL; probs / cls / bbox as in classify_batch. */
int cnnacc_preprocess_bgr(cnnacc_handle *h, const uint8_t *frames, int64_t n, int fh, int fw,
                          uint8_t *gray128, uint32_t flags);
int cnnacc_detect_frames(cnnacc_handle *h, const uint8_t *frames, int64_t n, int fh, int fw, uint8_t *gray128,
                         float *probs, int32_t *cls, int32_t *bbox, uint32_t flags);

/* ---- the same loop body on caller-chosen square regions of each frame -------------------------------------------------
 * A region is four int32 (frame, x, y, side): the square frames[frame][y:y+side, x:x+side, :] of the BGR frames
 * [n_frames][fh][fw][3] u8.  For every region the calls produce exactly what preprocess_bgr / detect_frames produce for that
 * square cut out as a frame of its own (a square is its own centre crop): gray128 / cls / bbox byte for byte, probs bit for
 * bit.  Boxes stay in the region's own 128x128 coordinates.  One call mixes any sides: the INTER_AREA taps are computed in the
 * kernel from each region's side.  Outputs are indexed by region, in the order of `regions`.
 *   regions : [n_regions][4] int32 in HOST memory in both modes, read only during the call (reusable once it returns).  The
 *             frame indices must not decrease (group the regions by frame).  frames / gray128 / probs / cls / bbox are host or
 *             device memory as for detect_frames, with the same flags, alignment rules and NULL conventions (gray128 may be
 *             NULL in detect_regions; any prediction array may be NULL).
 *   -2, nothing launched: n_regions > 0 with regions or frames NULL, a frame index outside [0, n_frames), a side outside
 *             128..8192, x < 0, y < 0, x + side > fw, y + side > fh, or frame indices that decrease.  n_regions == 0 returns 0.
 *   detect_regions returns -4 without weights or without a classifier.
 * Host pointers: the call copies each run of consecutive referenced frames once (about 16 MiB per staged chunk; unreferenced
 * frames never cross the link) and runs all regions of a frame on that copy.  Device pointers: asynchronous on the handle's
 * stream; the library keeps its own device copy of the descriptors alive until the call's kernels are done. */
int cnnacc_preprocess_regions(cnnacc_handle *h, const uint8_t *frames, int64_t n_frames, int fh, int fw,
                              const int32_t *regions, int64_t n_regions, uint8_t *gray128, uint32_t flags);
int cnnacc_detect_regions(cnnacc_handle *h, const uint8_t *frames, int64_t n_frames, int fh, int fw,
                          const int32_t *regions, int64_t n_regions, uint8_t *gray128,
                          float *probs, int32_t *cls, int32_t *bbox, uint32_t flags);
/* ---- rectangles: CNNACC_FLAG_RECTS -----------------------------------------------------------------------------------
 * With CNNACC_FLAG_RECTS, `regions` of preprocess_regions, detect_regions, detect_objects, merge_regions and
 * merge_regions_host is [n_regions][5] int32 (frame, x, y, w, h): the rectangle frames[frame][y:y+h, x:x+w, :], w and h each
 * 128..8192 (a square is w == h).  Everything else is as for squares.  Its gray128 is, byte for byte,
 *     cv2.resize(cv2.cvtColor(rect, COLOR_BGR2GRAY), (128, 128), interpolation=INTER_AREA)
 * with OpenCV's INTER_AREA arithmetic picked from both scales, kx = w/128 and ky = h/128 (csrc/regions.cuh):
 *   w == h == 128                          copy
 *   w, h multiples of 128, kx = ky = 2     (sum of 4 + 2) >> 2
 *   w, h multiples of 128, other kx, ky    rint(float(kx x ky box sum) * (1.f / float(kx*ky))), clamped to 0..255
 *   otherwise (an axis is fractional)      ResizeArea's float accumulation, x taps from computeResizeAreaTab(w) and y taps
 *                                          from computeResizeAreaTab(h); an integer axis takes that table too (kx taps of
 *                                          (float)(1.0/kx) each)
 * One exception: a side of exactly 6272 = 49 x 128 pixels counts as an integer axis here, while OpenCV (whose test is
 * 1 / (128 / side) within DBL_EPSILON of an integer, and 1.0 / (1.0 / 49) != 49 in double) takes the table for it; single
 * outputs can then differ from cv2.resize by 1.  The pyramid calls below follow OpenCV's test.
 * cls / probs / bbox are what infer_batch gives for that gray128; boxes stay on the rectangle's 128 grid.  The merge maps
 * them with X = 128 x + clamp(bx) w and Y = 128 y + clamp(by) h.
 *   -2, nothing launched: as for squares with w and h in place of side -- w or h outside 128..8192, x < 0, y < 0,
 *       x + w > fw or y + h > fh (in 64-bit arithmetic), a frame index outside [0, n_frames), frame indices that decrease;
 *       for the merging calls (no frame size): a frame outside [0, n_frames), x < 0, y < 0, w or h outside 128..8192.
 * Regions below 128 on an axis (OpenCV upsamples them) are refused, as for squares.  One call takes squares or rectangles,
 * not both: a square can be written as the rectangle w == h. */
#define CNNACC_FLAG_RECTS           0x100u /* region calls: regions are [n][5] (frame, x, y, w, h) */
/* ---- merging region detections into per-frame detections --------------------------------------------------------------
 * The rule (csrc/region_merge.h), per frame, independently: clamp every box coordinate to [0, 127]; map the box to the frame
 * exactly, in 1/128 pixel (X = 128 x + bx * side, the same for y); candidates are the regions with score >= score_min (a NaN
 * score never is; -0.0 equals +0.0); walk them by score descending, ties by region index ascending, and keep a candidate
 * unless an already-kept box of the same class (of any class with CNNACC_FLAG_CLASS_AGNOSTIC) has IoU > iou_max with it, where
 * IoU = (double)inter / (double)union of the exact integer areas (0 when union == 0); stop after max_det kept boxes.
 * Outputs per frame f, in kept order: n_det [F] i32, det_region [F][max_det] i32 (index into `regions`), det_cls [F][max_det]
 * i32, det_score [F][max_det] f32, det_box [F][max_det][4] f32 frame pixels (x1, y1, x2, y2) = the float nearest X / 128.
 * Rows k >= n_det[f] hold region -1, class -1, score 0 and box 0.  n_det is required; the other four may be NULL.
 *   -2, nothing launched: max_det outside 1..CNNACC_MERGE_MAX_DET, iou_max NaN or outside [0, 1], a frame with more than
 *       CNNACC_MERGE_MAX_PER_FRAME regions, n_det NULL, more than 2^31-1 regions; device pointers with det_box not 16-byte
 *       aligned or another array not 4-byte aligned.
 * detect_objects: detect_regions followed by the merge with score[r] = probs[r][cls[r]] (the logit with CNNACC_FLAG_LOGITS); the
 *       per-region predictions never leave the GPU.  Same flags, regions and refusals as detect_regions (-2, -4), plus the
 *       merge's.  n_regions == 0 gives every frame no detections.
 * merge_regions: the merge alone on predictions the caller has, scores [R] f32, cls [R] i32, bbox [R][4] i32, host or device
 *       memory (CNNACC_FLAG_DEVICE_PTRS); needs no weights or classifier.  Regions as above, in host memory; checked: a frame
 *       in [0, n_frames), frame indices that do not decrease, x, y >= 0, side 128..8192 (there is no frame size to check them
 *       against).  Device pointers: asynchronous on the handle's stream.
 * merge_regions_host: the same rule on the CPU (host arrays only), for tests. */
#define CNNACC_FLAG_CLASS_AGNOSTIC  0x80u  /* detect_objects / merge_regions: suppression across classes */
#define CNNACC_MERGE_MAX_DET        1024
#define CNNACC_MERGE_MAX_PER_FRAME  16384
int cnnacc_detect_objects(cnnacc_handle *h, const uint8_t *frames, int64_t n_frames, int fh, int fw,
                          const int32_t *regions, int64_t n_regions, float score_min, float iou_max, int max_det,
                          int32_t *n_det, int32_t *det_region, int32_t *det_cls, float *det_score, float *det_box, uint32_t flags);
int cnnacc_merge_regions(cnnacc_handle *h, const int32_t *regions, int64_t n_regions, int64_t n_frames,
                         const float *scores, const int32_t *cls, const int32_t *bbox, float score_min, float iou_max, int max_det,
                         int32_t *n_det, int32_t *det_region, int32_t *det_cls, float *det_score, float *det_box, uint32_t flags);
int cnnacc_merge_regions_host(const int32_t *regions, int64_t n_regions, int64_t n_frames,
                              const float *scores, const int32_t *cls, const int32_t *bbox, float score_min, float iou_max,
                              int max_det, int32_t *n_det, int32_t *det_region, int32_t *det_cls, float *det_score,
                              float *det_box, uint32_t flags);
/* ---- scanning whole frames: every 128x128 window at a multiple-of-8 stride from one conv pass per frame -----------------
 * frames [n][fh][fw][3] u8 BGR, fh and fw multiples of 16 in 128..8192 (so 1920x1080 frames are refused: 1080 is not a
 * multiple of 16, exactly as cnnacc_run_batch refuses them), stride a positive multiple of 8.
 * Windows: x = 0, stride, 2 stride, ... plus one window flush with the right edge (x = fw - 128) when that position is
 * missing, so nx = (fw - 128) / stride + 1 + ((fw - 128) % stride != 0); the same for y and ny.  Window r of the call is
 * (f, x, y) with r = (f * ny + iy) * nx + ix: frame-major, then y, then x -- the order of grid_regions(n, fh, fw, 128, stride)
 * in the Python package.  Outputs are indexed by window in that order.
 * What a window computes:
 *   gray[f] = cvtColor(frames[f], COLOR_BGR2GRAY) at full resolution (OpenCV's 15-bit fixed point, as preprocess_bgr)
 *   feat[f] = cnnacc_run_batch(gray[f]) at fh x fw: [64][fh/8][fw/8], with the handle's shifts and accumulator width
 *   window (f, x, y) -> cls / probs (logits with CNNACC_FLAG_LOGITS) / bbox = cnnacc_classify_batch of the 64x16x16 map
 *                       feat[f][:, y/8 : y/8+16, x/8 : x/8+16], bit for bit; the box is on the window's 128 grid
 * This is NOT detect_regions on the same squares.  A region is pre-processed as an image of its own, so its conv stack pads
 * with zeros at the region's border; a scan window sees the frame's real pixels beyond its border.  Their maps agree on the
 * inner 14x14 cells, and on the outer ring only on the sides where the window's edge is the frame's edge; on a 128x128 frame
 * the two are the same computation.  The gain: each pixel goes through the conv stack once per frame, not once per window.
 * scan_frames : probs [R][n_cls] f32, cls [R] i32, bbox [R][4] i32 for R = n * nx * ny windows; any output may be NULL.
 * scan_objects: scan_frames followed by the merge above, the windows being the regions (f, x, y, 128), score[r] =
 *               probs[r][cls[r]] (the logit with CNNACC_FLAG_LOGITS); det_region indexes the window order.  The result is
 *               exactly merge_regions on those regions and scan_frames' outputs.  Per-window predictions never leave the GPU.
 * Host pointers: frames are staged in chunks of about 16 MiB (a larger frame alone).  Device pointers
 * (CNNACC_FLAG_DEVICE_PTRS): asynchronous on the handle's stream, with detect_regions' alignment rules.  CNNACC_FLAG_LOGITS
 * and, for scan_objects, CNNACC_FLAG_CLASS_AGNOSTIC are honoured.
 *   -2, nothing launched: n < 0, fh or fw not a multiple of 16 or outside 128..8192, stride not a positive multiple of 8,
 *       more than 2^31-1 windows in the call, CNNACC_FLAG_BBOX_UPSAMPLED / _RECTS / _DIRECT / _KEEP_MAPS / _TWO_KERNELS,
 *       frames NULL with n > 0; for scan_objects also more than CNNACC_MERGE_MAX_PER_FRAME windows per frame and the
 *       merge's own refusals.  -4 without weights or without a classifier.  n == 0 returns 0. */
int cnnacc_scan_frames(cnnacc_handle *h, const uint8_t *frames, int64_t n, int fh, int fw, int stride,
                       float *probs, int32_t *cls, int32_t *bbox, uint32_t flags);
int cnnacc_scan_objects(cnnacc_handle *h, const uint8_t *frames, int64_t n, int fh, int fw, int stride,
                        float score_min, float iou_max, int max_det, int32_t *n_det, int32_t *det_region,
                        int32_t *det_cls, float *det_score, float *det_box, uint32_t flags);
/* ---- scanning image pyramids: the windows of several downscaled levels of each frame, one conv pass per level ------------
 * frames [n][fh][fw][3] u8 BGR, fh and fw any integers in 128..8192.  levels [L][2] int32 (w, h) in host memory,
 * 1 <= L <= CNNACC_PYRAMID_MAX_LEVELS: each level has w and h multiples of 16 with 128 <= w <= fw and 128 <= h <= fh
 * (downscales only; a level may be anisotropic).  stride: a positive multiple of 8, in level pixels, the same at every level.
 * Level gray (byte for byte):
 *   gray_l[f] = cv2.resize(cv2.cvtColor(frames[f], COLOR_BGR2GRAY), (w, h), interpolation=INTER_AREA)
 * with OpenCV's choice of arithmetic from both scales, as for the rectangle regions with 128 replaced by w / h: a copy when the
 * level is the frame size; (sum + 2) >> 2 at 2x2; rint(float(sum) * (1.f / (kx * ky))) for other integer pairs; otherwise
 * ResizeArea with x taps from computeResizeAreaTab(fw -> w) and y taps from (fh -> h).  An axis counts as integer as OpenCV
 * decides it: 1 / (w / fw) in double within DBL_EPSILON of an integer, so a 49x axis (1.0 / (1.0 / 49) != 49) takes the table.
 * Windows of a level: x in the origins of cnnacc_scan_frames along w (0, stride, 2 stride, ... plus the one flush with the far
 * edge), y likewise along h.  Window r of the call is numbered frame-major, then level in the given order, then y, then x.
 * What a window computes: cnnacc_classify_batch of the 64x16x16 cells at (x/8, y/8) of cnnacc_run_batch(gray_l[f]), bit for
 * bit; its box is on the window's 128 grid.  Its frame rectangle is (f, x fw / w, y fh / h, 128 fw / w, 128 fh / h): the call
 * is refused unless all four are integers for every window of every level (the actual origins are checked, so a level with
 * one window position is never refused for its stride), so the rectangle merge maps every box exactly.  A single level
 * (fw, fh) gives exactly cnnacc_scan_frames' outputs.
 * This is NOT detect_regions on the same rectangles: a region is cropped and then resized, a pyramid window is resized with
 * the whole frame and sees the frame beyond its border (see cnnacc_scan_frames).
 * preprocess_pyramid  : gray [n][sum of h * w] u8, frame-major, then level (the weights are not needed).
 * scan_pyramid        : probs [R][n_cls] f32, cls [R] i32, bbox [R][4] i32 for R = n * (windows per frame); any may be NULL.
 * scan_pyramid_objects: scan_pyramid followed by the merge above with CNNACC_FLAG_RECTS, the windows' frame rectangles being
 *                       the regions and score[r] = probs[r][cls[r]] (the logit with CNNACC_FLAG_LOGITS): exactly
 *                       merge_regions on those rectangles and scan_pyramid's outputs.  Predictions never leave the GPU.
 * Host and device pointers, alignment, CNNACC_FLAG_LOGITS and CNNACC_FLAG_CLASS_AGNOSTIC as for the scan_frames calls.
 *   -2, nothing launched: n < 0, a frame side outside 128..8192, L outside 1..16 or levels NULL, a level that breaks the
 *       rules above, a window rectangle not in whole frame pixels, stride not a positive multiple of 8, more than 2^31-1
 *       windows in the call, the flags cnnacc_scan_frames refuses, frames (or gray) NULL with n > 0; for the _objects call
 *       also more than CNNACC_MERGE_MAX_PER_FRAME windows per frame and the merge's own refusals.  preprocess_pyramid takes
 *       no stride and has no windows to check.  -4 without weights or without a classifier (scan calls).  n == 0 returns 0. */
#define CNNACC_PYRAMID_MAX_LEVELS 16
int cnnacc_preprocess_pyramid(cnnacc_handle *h, const uint8_t *frames, int64_t n, int fh, int fw, const int32_t *levels,
                              int n_levels, uint8_t *gray, uint32_t flags);
int cnnacc_scan_pyramid(cnnacc_handle *h, const uint8_t *frames, int64_t n, int fh, int fw, const int32_t *levels,
                        int n_levels, int stride, float *probs, int32_t *cls, int32_t *bbox, uint32_t flags);
int cnnacc_scan_pyramid_objects(cnnacc_handle *h, const uint8_t *frames, int64_t n, int fh, int fw, const int32_t *levels,
                                int n_levels, int stride, float score_min, float iou_max, int max_det, int32_t *n_det,
                                int32_t *det_region, int32_t *det_cls, float *det_score, float *det_box, uint32_t flags);
/* Host-only: the windows per frame of a pyramid call with these frame sides, levels and stride, or -2 where the call refuses
 * them (the same checks).  With rects, also writes their frame rectangles [R][5] (0, x, y, w, h) in window order (cap >= R,
 * else -2).  No GPU needed. */
int cnnacc_pyramid_windows_host(int fh, int fw, const int32_t *levels, int n_levels, int stride, int32_t *rects, int64_t cap);
/* Host-only view of the staging plan of a host-pointer region call (csrc/region_plan.h): chunk i stages frames
 * [chunks[4i], chunks[4i+1]) with one copy and runs regions [chunks[4i+2], chunks[4i+3]) on them.  Returns the number of chunks
 * (<= cap), or -2 for a region array the real call refuses, or when cap is too small.  No GPU needed. */
int cnnacc_region_plan_host(const int32_t *regions, int64_t n_regions, int64_t n_frames, int fh, int fw, int64_t *chunks, int cap);
/* The same for [n_regions][5] rectangles (frame, x, y, w, h), with the refusals of CNNACC_FLAG_RECTS. */
int cnnacc_rect_plan_host(const int32_t *regions, int64_t n_regions, int64_t n_frames, int fh, int fw, int64_t *chunks, int cap);
/* Host-only view of the INTER_AREA taps the kernels use for one crop side (128..8192): output index d reads source indices
 * start[d] .. start[d]+cnt[d]-1 with weights alpha[d*taps_cap + i] (zero beyond cnt[d]; weight 1 at integer scales, whose
 * kernels sum integers).  Returns the largest cnt, or -2 when it exceeds taps_cap.  No GPU needed. */
int cnnacc_area_tab_host(int side, int *start, int *cnt, float *alpha, int taps_cap);

/* image_to_gray128: the image-loading step of pynq_inference.py, load_image_any (:414-425), for n decoded images of one size:
 *                 img [n][H][W][C] u8 with C = 1 (mode L), 3 (RGB) or 4 (RGBA) -> gray128 [n][128][128] u8 =
 *                 Image.convert('L').resize((128, 128)): Pillow's ITU-R 601 integer luma and its default BICUBIC resampler
 *                 (22-bit fixed point, horizontal pass then vertical pass, or vertical first when H > 100 W as Image.resize
 *                 does), reproduced bit for bit (pinned against Pillow 12.2.0).  File decoding itself stays on the host. */
int cnnacc_image_to_gray128(cnnacc_handle *h, const uint8_t *img, int64_t n, int H, int W, int C,
                            uint8_t *gray128, uint32_t flags);

/* ---- one host batch over several GPUs ------------------------------------------------------------------------------------
 * The sharded forms of cnnacc_run_batch / cnnacc_infer_batch / cnnacc_detect_frames for HOST pointers take an array of
 * n_handles member handles the caller created and configured (usually one per GPU; two handles on one GPU are allowed) and
 * cut the n images / frames into contiguous shards: shard i = [begin[i], begin[i+1]) runs through member i's own
 * single-handle host path with every pointer offset to that slice, so the outputs are those of one handle, byte for byte.
 * The calling thread runs shard 0; shards 1 .. m-1 run on a thread each that the call starts and joins before it returns (a
 * call small enough for one member starts none), so every member handle is used by one thread only.
 *   Plan (csrc/shard_plan.h): m = min(n_handles, max(1, n * unit_bytes / kMinShardBytes)) members, begin[i] = n*i/m, where
 *   unit_bytes is the input size of one image (H*W) or frame (fh*fw*3).
 *   Checked before any member starts (nothing is launched; -2 or -4): hs / an entry NULL, n_handles < 1, a handle listed
 *   twice, CNNACC_FLAG_DEVICE_PTRS or CNNACC_FLAG_KEEP_MAPS set, a member without weights (-4) or -- for the prediction
 *   calls -- without a classifier (-4), and members configured unlike member 0: weights, shifts, accumulator bits and, for
 *   the prediction calls, the classifier (-2).  The other flags pass through to every member unchanged.
 *   Errors: every started shard runs to completion; the call returns the code of the lowest-index failing member and, when
 *   failed != NULL, stores that index there (-1 on success, or when no member is at fault: hs NULL / n_handles < 1).  The text
 *   stays in that member's cnnacc_last_error.  After a failure the outputs of the whole call are undefined.
 *   Host buffers should be page-locked (cnnacc_alloc_host / cnnacc_register_host pin memory for every GPU at once); pageable
 *   memory works but makes each member's copies synchronous and slow. */
int cnnacc_run_batch_sharded(cnnacc_handle *const *hs, int n_handles, const uint8_t *imgs, int64_t n, int H, int W,
                             uint8_t *feats, uint32_t flags, int *failed);
int cnnacc_infer_batch_sharded(cnnacc_handle *const *hs, int n_handles, const uint8_t *imgs, int64_t n,
                               float *probs, int32_t *cls, int32_t *bbox, uint32_t flags, int *failed);
int cnnacc_detect_frames_sharded(cnnacc_handle *const *hs, int n_handles, const uint8_t *frames, int64_t n, int fh, int fw,
                                 uint8_t *gray128, float *probs, int32_t *cls, int32_t *bbox, uint32_t flags, int *failed);
/* Host-only view of the shard plan: begin[0 .. m] (m + 1 entries, begin[m] = n).  Returns m, or a negative code when n < 0,
 * n_handles < 1, unit_bytes < 1 or cap < m + 1.  No GPU needed; tests/ check that every plan covers the call exactly once. */
int cnnacc_shard_plan_host(int64_t n, int n_handles, int64_t unit_bytes, int64_t *begin, int cap);

/* ---- host memory the DMA engines can stream from (pynq.allocate, realtime_detect.py:293,301) */
int cnnacc_alloc_host(size_t bytes, void **out);
int cnnacc_free_host(void *p);
/* Page-lock memory the caller already owns (e.g. a shared-memory mapping that several per-GPU processes write their slice of
 * the prediction array into: SURVEY.md 8e "per-GPU D2H into one pinned host array"). */
int cnnacc_register_host(void *p, size_t bytes);
int cnnacc_unregister_host(void *p);

/* ---- timing on the handle's stream (CUDA events; bench.py) ---------------------------------- */
int cnnacc_timer_start(cnnacc_handle *h);
int cnnacc_timer_stop(cnnacc_handle *h, float *ms);   /* synchronises the stream */
int cnnacc_synchronize(cnnacc_handle *h);
/* Dense int8 tensor-core ceiling of this GPU, measured now: back-to-back tcgen05.mma kind::i8 M=128 N=256 K=32 on every SM
 * for about target_ms milliseconds (csrc/int8_peak_probe.cuh).  *tops = 10^12 integer ops per second (2 per MAC). */
int cnnacc_probe_int8_peak(cnnacc_handle *h, double target_ms, double *tops, double *ms);

/* ---- drop-in for the reference symbol ------------------------------------------------------
 * Same name and signature as arm_cnn.c:159-162, so ARMEngine's ctypes call
 * (realtime_detect.py:389-391,427-431) works unchanged against libcnnacc.so.  Uses a lazily
 * created process-global handle on device 0 guarded by a mutex; weights are re-packed only when
 * the 23184 bytes change.  Returns 0, or a negative code above. */
int cnn_infer(const uint8_t *input_img, const uint8_t *weights_bin, const int *shifts, uint8_t *output);

#ifdef __cplusplus
}
#endif
#endif /* CNNACC_H */
