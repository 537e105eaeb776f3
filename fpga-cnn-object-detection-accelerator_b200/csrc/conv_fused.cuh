// conv_fused.cuh -- the hot path: one persistent, warp-specialised sm_100a kernel for the whole 128x128 conv stack.
//
// What it replaces: cnn_infer (/root/reference/software/arm_cnn.c:159-198) == the PL datapath
// layer_fsm + conv_core + accumulator + ReLU + max_pooling_engine over feature/weight BRAM
// (rtl/core/cnn_acc_top.v).  Like the FPGA design, every intermediate map stays on chip: one CTA per SM
// keeps an image's maps in shared memory and HBM sees 16 KiB of pixels in and 16 KiB of features out.
//
//   layer 0  (1->16, 128x128, K=9)    half the rows on the dp4a pipe (dp4a.u32.s32), half on warp-level int8 MMA
//                                     (mma.sync m16n8k16); 2x2 pool in registers, -> act1 (smem)
//   layer 1  (16->32, 64x64, K=144)   tcgen05.mma kind::i8 (A = u8 activations, B = s8 weights, D = s32 in TMEM)
//   layer 2  (32->64, 32x32, K=288)   tcgen05.mma kind::i8
//   each followed by >>shift, ReLU/saturate (arm_cnn.c:127-135) and 2x2 max-pool (arm_cnn.c:115-143),
//   pooled on the raw s32 first (monotone activation, SURVEY.md 2.3-4).
//
// Implicit GEMM without im2col.  Activation maps are stored as [y+1][x-parity][(x+1)/2][16 ch] bytes with a
// zero halo, so a no-swizzle K-major UMMA core matrix (8 rows x 16 B) is "8 same-parity pixels x 16 channels",
// a conv tap is a 16-byte-granular start-address offset, and SBO = 2 row pitches makes the 128 rows of an MMA
// a block of 16 row-pairs x 8 column-pairs.
//   layer 1: one MMA row = one 2x2 POOLING WINDOW.  N = 128 = 4 window members x 32 out-channels, and the B
//            operand is the 3x3 kernel Toeplitz-expanded over the window's 4x4 input patch: 8 K-slabs of
//            (2 adjacent pixels x 16 ch), LBO = parity-plane stride.  An M=128, K=32 i8 MMA from shared memory
//            costs max(N/2, 32 + N/4) clk (profiles/r1_probe_umma_rate.txt: N=32 -> 40, N=64 -> 48, N=128 -> 64),
//            which beats the 160 x 40 = 6.4 k clk of one N=32 MMA per tap pair.  Patch row 0 only reaches the
//            window's upper members and patch row 3 only its lower ones, so those four slabs are N = 64 MMAs
//            into the matching half of the accumulator columns: 8 tiles x (4 x 64 + 4 x 48) = 3.6 k clk per
//            image, 64 % of the MAC slots useful, and the operand is 24 KiB instead of 32.
//            All four members of a window land in one TMEM lane: the pool is thread-local.
//   layer 2: one MMA row = one output pixel of ONE parity (y%2, x%2); K=32 = one tap over both 16-channel
//            planes (LBO = plane stride), 9 MMAs, N = 64; the four parities go to four TMEM column groups.
// These descriptor forms were verified on a B200 by tools/probe_umma.cu (profiles/r1_probe_umma_dp4a_tmem.txt).
//
// Warp roles (21 warps, 1 CTA/SM).  Layer 0 and the tcgen05 layers run concurrently on DIFFERENT images: while the
// tensor core and the epilogue warps finish image k, the layer-0 warps already produce image k+1 into the half of
// act1 the MMAs have released.
//   warps 0-7    layer 0 on the dp4a pipe : input slot -> act1   (rows w, w+16, w+32, w+48)
//   warps 8-15   layer 0 on mma.sync      : input slot -> act1
//   warps 16-19  epilogues : TMEM -> pool -> shift/ReLU/saturate -> act2 (layer 1) / staging -> TMA store (layer 2)
//   warp 20      tcgen05 MMA issue (whole warp walks the schedule, one elected lane issues), TMEM allocation,
//                TMA loads (weights once, then images two ahead)
//   warps 24-27  (kTail instantiation only) front stage of the classifier / CAM-box tail of tail.cuh on the layer-2
//                staging buffer of the image the epilogue warps have just finished (bin sums, logits, softmax, CAM);
//   warps 22-23  (kTail; warp 21 idle) its back stage, one image behind (CAM maximum, percentile, box): predictions leave
//                the SM, the feature map need not.  28 warps only fit because the two light warpgroups (20-23, 24-27) hand
//                registers to the five heavy ones with setmaxnreg: the kernel launches at 72 registers per thread (7 warps
//                x 72 x 32 = 16 128 of a sub-partition's 16 384), then warps 0-19 grow to 80 and warps 20-27 shrink to 48.
#pragma once
#include <cuda.h>
#include <cstdlib>

#include "common.cuh"
#include "tail.cuh"
#include "weights_pack.h"

namespace cnnacc {

// ---- shared-memory plan (bytes) ---------------------------------------------------------------------
constexpr int kInPitch   = 160;                       // x = -16 .. 143 (TMA box, OOB zero-filled; the innermost
                                                      // box coordinate must be 16-byte aligned: tools/probe_tma.cu)
constexpr int kInRows    = 130;                       // y = -1 .. 128
constexpr int kInBytes   = kInPitch * kInRows;        // 20800, one TMA transaction
constexpr int kInStride  = 20864;                     // 128-byte aligned slot size
constexpr int kA1Q       = 33 * 16;                   // act1 parity-plane stride   (528)
constexpr int kA1P       = 2 * kA1Q;                  // act1 row pitch             (1056)
constexpr int kA1Bytes   = 66 * kA1P;                 // 69696
constexpr int kA1Alloc   = 69760;                     // rounded up to 128
constexpr int kA2Q       = 17 * 16;                   // act2 parity-plane stride   (272)
constexpr int kA2P       = 2 * kA2Q;                  // act2 row pitch             (544)
constexpr int kA2C       = 34 * kA2P;                 // act2 channel-block plane   (18496)
constexpr int kA2Bytes   = 2 * kA2C;                  // 36992
constexpr int kB1Slab    = 4096;                      // layer-1 B: one K=32 slab x N=128 (patch rows 1, 2)
constexpr int kB1Half    = 2048;                      // ... x N=64 (patch row 0: upper window members; row 3: lower)
constexpr int kB1Bytes   = 4 * kB1Slab + 4 * kB1Half; // 24576: [r1s0][r1s1][r2s0][r2s1] [r0s0][r0s1][r3s0][r3s1]
constexpr int kB2Bytes   = 9 * 2048;                  // layer-2 B: 9 taps x (2 K-halves x 8 row groups x 128 B)
constexpr int kStageBytes = 16384;                    // one image's features, CHW, for the TMA store

constexpr int kOffIn0   = 0;
constexpr int kOffIn1   = kInStride;
constexpr int kOffA1    = 2 * kInStride;              // 41728
constexpr int kOffA2    = kOffA1 + kA1Alloc;          // 111488
constexpr int kOffB1    = kOffA2 + kA2Bytes;          // 148480
constexpr int kOffB2    = kOffB1 + kB1Bytes;          // 181248
constexpr int kOffStage = kOffB2 + kB2Bytes;          // 199680
constexpr int kOffBar   = kOffStage + kStageBytes;    // 216064
constexpr int kOffTail  = kOffBar + 256;              // scratch of the two tail warps (tail.cuh)
#ifdef CNNACC_TRACE
constexpr int kTailWRows = 4;                         // the trace build's static buffers take 4 KiB
#else
constexpr int kTailWRows = 5;                         // classifier rows kept in shared memory (the rest: __ldg through L1)
#endif
constexpr int kOffTailW = kOffTail + kTailScratchBytes;
constexpr int kFusedSmem = kOffTailW + kTailWRows * 4096;   // 229888 <= 232448
static_assert(kFusedSmem <= 232448, "shared memory plan exceeds 227 KB");

// Optional schedule trace (tools only, -DCNNACC_TRACE): CTA 0 records clock() at pipeline events in shared memory and
// prints them at exit (tools/trace_run.py).
#ifdef CNNACC_TRACE
#include <cstdio>
constexpr int kTraceMax = 90, kTraceRoles = 6;
#define TRACE(role, code)                                                                                          \
    do {                                                                                                           \
        if (blockIdx.x == 0 && lane == 0 && trace_n < kTraceMax) {                                                 \
            trace_buf[(role) * kTraceMax + trace_n] = ((unsigned)(code) << 24) | ((unsigned)clock64() & 0xFFFFFFu);   \
            trace_n++;                                                                                             \
        }                                                                                                          \
    } while (0)
#define TRACE_END(role) do { if (blockIdx.x == 0 && lane == 0) trace_cnt[role] = trace_n; } while (0)
#if CNNACC_TRACE >= 2
#define TRACE2(role, code) TRACE(role, code)             // per-tile detail (perturbs the MMA warp noticeably)
#else
#define TRACE2(role, code) do { } while (0)
#endif
#else
#define TRACE(role, code) do { } while (0)
#define TRACE2(role, code) do { } while (0)
#define TRACE_END(role) do { } while (0)
#endif

constexpr int kL0Warps = 16;                          // layer 0 (a multiple of 4: TMEM lane quarter == warp % 4)
constexpr int kL0Dp4aWarps = 8;                       // ... of which these use dp4a, the rest mma.sync
constexpr int kEpiWarps = 4;                          // one per TMEM lane quarter
constexpr int kWarpMma = kL0Warps + kEpiWarps;       // the last warp: MMA issue and TMA loads
constexpr int kFusedThreads = (kWarpMma + 1) * 32;    // 21 warps = 672
constexpr int kTailWarps = kTailThreads / 32;         // 4 tail warps = warpgroup 6 of the kTail instantiation
constexpr int kWarpTail0 = 24;                        // first tail warp (warpgroup aligned: setmaxnreg acts on warpgroups)
constexpr int kTailKernelThreads = (kWarpTail0 + kTailWarps) * 32;   // 896
constexpr uint32_t kTmemCols = 512;
#ifndef CNNACC_WAIT_BUDGET_CLK
#define CNNACC_WAIT_BUDGET_CLK 8000000000LL            // bounded pipeline waits: ~4 s of SM clocks
#endif
constexpr long long kWaitBudgetClk = CNNACC_WAIT_BUDGET_CLK;

// mbarrier slots (8 bytes each) at kOffBar
enum : uint32_t {
    kBarInFull0 = 0, kBarInFull1, kBarInFree0, kBarInFree1,        // TMA -> layer 0 ; layer 0 -> TMA
    kBarA1TopReady, kBarA1BotReady,                                 // layer 0 -> MMA  (act1 rows 0-33 / all rows written)
    kBarA1TopFree, kBarA1BotFree,                                   // MMA (tcgen05.commit) -> layer 0
    kBarTmFull0, kBarTmFull1, kBarTmEmpty0, kBarTmEmpty1,           // MMA -> epilogue ; epilogue -> MMA (TMEM halves)
    kBarA2ReadyA, kBarA2ReadyB,                                     // epilogue -> MMA: act2 written by tiles 0-6 (all block 0 needs) / by all 8
    kBarW,                                                          // weights landed
    kBarStageFull, kBarStageFree,                                   // epilogue -> tail warps (features staged) ; tail -> epilogue
    kNumBars
};

// error bits reported through the status word
constexpr int kErrInputTimeout = 1, kErrMmaTimeout = 2, kErrEmptyTimeout = 4, kErrWeightTimeout = 8,
              kErrAct1Timeout = 16, kErrAct2Timeout = 32, kErrSlotTimeout = 64, kErrStageTimeout = 128;

struct FusedParams {
    uint32_t w0[16][6];          // layer-0 dp4a words per out-channel: lo[dy], hi[dy]  (constant bank)
    uint32_t w0f[8][32];         // layer-0 mma.sync B fragments: [block = py*4 + ol][lane]
    int shift0, shift1, shift2;
    int acc24;                   // layer-2 accumulators wrap at 24 bits before the pool (RTL / trainer width, accumulator.v:15,
                                 // train_cnn.py:110-111); layers 0/1 cannot reach 2^23 (9*255*128, 16*9*255*128 = 4.7 M)
    int n_images;
    const uint8_t* b1;           // packed layer-1 B operand (kB1Bytes)
    const uint8_t* b2;           // packed layer-2 B operand (kB2Bytes)
    uint8_t* out;                // [n][64][16][16]; may be null in the kTail instantiation (predictions only)
    TailArgs tail;               // kTail instantiation: classifier + outputs (tail.cuh)
    uint8_t* dump_l0;            // optional [n][16][64][64]
    uint8_t* dump_l1;            // optional [n][32][32][32]
    int* status;                 // device int, OR-ed error bits
    int* status_host;            // the same in mapped pinned host memory: polled without a CUDA call
    int pdl_wait;                // conv-only instantiation, launched with programmatic stream serialisation: 1 = execute
                                 // griddepcontrol.wait before touching global memory (the launch may depend on the previous one)
    int* done_flag;              // optional (single-CTA latency path): mapped pinned host word that receives done_seq once the
    int done_seq;                // last feature store has landed, so the host can spin on it instead of a stream synchronise
    // window mode (images larger than 128x128, tiling.cuh): unit u = window (u % win_ntx, (u / win_ntx) % win_nty) of image
    // u / (win_ntx * win_nty); the TMA box is read straight from the big image at pixel origin 8 * win_g{x,y}[..] (origins are
    // even, so x stays 16-byte aligned).  win_ntx == 0: unit u = image u of an [n][128][128] array.
    // In window mode the features go straight to out[img][64][win_ho][win_wo]: every window stores the outputs it computes
    // exactly (local rows/columns 1..14, plus 0 / 15 where the window touches the image border); neighbouring windows write
    // identical bytes where those regions overlap.
    int win_ntx, win_nty, win_ho, win_wo;
    short win_gx[80], win_gy[80];
};

// ---- PTX wrappers ---------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(bar), "r"(bytes) : "memory");
}
// Plain SYNCS.TRYWAIT: the hardware holds the warp until this barrier's phase completes or its own time limit passes.
// With a suspend-time hint every failed try_wait cost a NANOSLEEP.SYNCS that woke on ANY barrier event of the CTA (ncu:
// ~100 wake-ups per image per waiting warp, 16.8 k polling instructions per image in the round-1 kernel); without it the
// kernel ran 2.5-4 % more images/s (profiles/r2_trywait_hint_sweep.txt).
__device__ __forceinline__ uint32_t mbar_try(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}\n"
                 : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    return ok;
}
// Bounded wait: a broken pipeline must never hang the GPU.  Returns false on timeout.  Every try_wait parks the warp in
// hardware for a while, and the clock is only consulted every 32 unsuccessful polls.
__device__ __forceinline__ bool mbar_wait(uint32_t bar, uint32_t parity, long long budget) {
    const long long t0 = clock64();
    for (;;) {
#pragma unroll 1
        for (int i = 0; i < 32; i++)
            if (mbar_try(bar, parity)) return true;
        if (clock64() - t0 > budget) return false;
    }
}
// One lane of a converged warp.  With warp-uniform operands around it the compiler keeps descriptors and addresses
// in uniform registers, so tcgen05.mma / TMA issue back to back instead of through a per-instruction R2UR loop.
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n .reg .pred P;\n elect.sync _|P, 0xffffffff;\n selp.u32 %0, 1, 0, P;\n}\n" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// K-major, no-swizzle shared-memory matrix descriptor (version 1 = sm_100).  Offsets in bytes, multiples of 16.
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
    return (uint64_t)((saddr >> 4) & 0x3FFF) | (uint64_t)((lbo >> 4) & 0x3FFF) << 16 |
           (uint64_t)((sbo >> 4) & 0x3FFF) << 32 | (uint64_t)1 << 46;
}
// kind::i8 instruction descriptor: D = s32, A = unsigned 8-bit, B = signed 8-bit, both K-major, M = 128.
__device__ __forceinline__ constexpr uint32_t umma_idesc_i8(int n) {
    return (2u << 4) | (0u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
}
__device__ __forceinline__ void umma_i8(uint32_t d_tmem, uint64_t a, uint64_t b, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n .reg .pred p;\n setp.ne.b32 p, %4, 0;\n tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n}\n"
                 :: "r"(d_tmem), "l"(a), "l"(b), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, int* v) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                   "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
                 : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// 3D tiled TMA load (x, y, image) -> smem, completion on an mbarrier.
__device__ __forceinline__ void tma_load_box(uint32_t dst, const CUtensorMap* map, uint32_t bar, int x, int y, int img) {
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
                 :: "r"(dst), "l"(map), "r"(x), "r"(y), "r"(img), "r"(bar) : "memory");
}
// 1D bulk copy global -> smem (pre-packed weights).
__device__ __forceinline__ void bulk_load(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
// 1D bulk copy smem -> global (one image's features), tracked by the issuing thread's bulk group.
__device__ __forceinline__ void bulk_store(void* dst, uint32_t src, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" :: "l"(dst), "r"(src), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void bulk_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void epi_bar_sync() { asm volatile("bar.sync 1, %0;" :: "n"(kEpiWarps * 32) : "memory"); }
// Staging-buffer hand-over between the epilogue warps and the tail warps (kTail): hardware named barriers, so the waiting
// side costs no issue slots at all (an mbarrier wait polls, and NANOSLEEP.SYNCS wakes on every barrier event of the CTA:
// ncu counted ~100 wake-ups per image per waiting warp).  The two barriers strictly alternate -- full(k), free(k),
// full(k+1) ... -- and both sides run the same n_local iterations, so arrivals can never run a phase ahead.
constexpr int kNamedL0Bot = 9;                        // kTail: the sixteen layer-0 warps behind one poller (see the layer-0 loop)
__device__ __forceinline__ void l0_bar_sync(int id) { asm volatile("bar.sync %0, %1;" :: "r"(id), "n"(kL0Warps * 32) : "memory"); }
constexpr int kNamedStageFull = 3, kNamedStageFree = 4;
// ... and the same between the tail's front warps (24-27) and back warps (22-23) for the 1 KiB CAM buffer; 2 and 5 are the
// front's and the back's own barriers.
constexpr int kNamedTailFront = 2, kNamedTailBack = 5, kNamedCamFull = 6, kNamedCamFree = 7;
constexpr int kWarpTailBack0 = 22;
__device__ __forceinline__ void cam_bar_sync(int id) {
    asm volatile("bar.sync %0, %1;" :: "r"(id), "n"(kTailThreads + kTailBackThreads) : "memory");
}
__device__ __forceinline__ void cam_bar_arrive(int id) {
    asm volatile("bar.arrive %0, %1;" :: "r"(id), "n"(kTailThreads + kTailBackThreads) : "memory");
}
__device__ __forceinline__ void stage_bar_sync(int id) {
    asm volatile("bar.sync %0, %1;" :: "r"(id), "n"(kEpiWarps * 32 + kTailThreads) : "memory");
}
__device__ __forceinline__ void stage_bar_arrive(int id) {
    asm volatile("bar.arrive %0, %1;" :: "r"(id), "n"(kEpiWarps * 32 + kTailThreads) : "memory");
}

// Warp-level int8 MMA for layer 0 (K = 9 is too thin for a 128-row tcgen05 tile without a re-layout pass):
// D(16x8,s32) += A(16x16,u8) * B(16x8,s8).  Fragments (lane = 4*g + t): a0/a1 = rows g / g+8, k = 4t..4t+3;
// b0 = k 4t..4t+3 of column g; c0,c1 = row g cols 2t,2t+1; c2,c3 = row g+8.  SASS: IMMA.16816.U8.S8.
__device__ __forceinline__ void imma_16816(int (&c)[4], uint32_t a0, uint32_t a1, uint32_t b0) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.s32.u8.s8.s32 {%0,%1,%2,%3}, {%4,%5}, {%6}, {%0,%1,%2,%3};"
                 : "+r"(c[0]), "+r"(c[1]), "+r"(c[2]), "+r"(c[3]) : "r"(a0), "r"(a1), "r"(b0));
}

// arm_cnn.c:127-135 for one accumulator: shift, then saturate to [0,255] (negatives stay negative under >>).
__device__ __forceinline__ uint32_t act_u8(int v, int shift) {
    uint32_t d;
    asm("cvt.sat.u8.s32 %0, %1;" : "=r"(d) : "r"(v >> shift));
    return d;
}

// 24-bit two's-complement wrap of a finished sum (accumulator.v:15 `reg signed [23:0]`; train_cnn.py:110-111
// ((out + M) % 2M) - M): wrapping once at the end equals wrapping after every add.
__device__ __forceinline__ int wrap24(int v) { return (int)((unsigned)v << 8) >> 8; }

// ---- the kernel ---------------------------------------------------------------------------------------------
// Register budget: each SM sub-partition has 16 384 registers and 21 warps put 6 on one of them, so 80 per thread
// (6 x 80 x 32 = 15 360) is the most that launches; 96 would need <= 20 warps.
// kWin = window mode (FusedParams::win_*): a separate instantiation, so the 128x128 path carries none of its code.
// kTail = two more warps run the classifier / CAM-box tail on each image's staged features (tail.cuh).
template <bool kWin, bool kTail>
__global__ void __launch_bounds__(kTail ? kTailKernelThreads : kFusedThreads, 1)
conv_stack_fused_kernel(const __grid_constant__ CUtensorMap in_map, const __grid_constant__ FusedParams P)
{
    static_assert(!(kWin && kTail), "the tail needs a whole 16x16 map in the staging buffer");
    constexpr int kThreads = kTail ? kTailKernelThreads : kFusedThreads;
    extern __shared__ __align__(1024) uint8_t smem[];
    const uint32_t s_base = smem_u32(smem);
    const uint32_t bars = s_base + kOffBar;
    auto bar = [&](uint32_t i) { return bars + 8u * i; };
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + kOffBar + 8 * kNumBars);
    int* s_err = reinterpret_cast<int*>(smem + kOffBar + 8 * kNumBars + 8);

    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);          // warp-uniform in the compiler's eyes
    const int n_local = (P.n_images - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;   // images of this CTA
#ifdef CNNACC_TRACE
    __shared__ unsigned trace_buf[kTraceRoles * kTraceMax];
    __shared__ int trace_cnt[kTraceRoles];
    int trace_n = 0;
    if (tid < kTraceRoles) trace_cnt[tid] = 0;
#endif

    // ---- one-time setup ---------------------------------------------------------------------------------
    for (int i = tid; i < (kA1Alloc + kA2Bytes) / 16; i += kThreads)                            // zero halos (and interiors)
        reinterpret_cast<uint4*>(smem + kOffA1)[i] = make_uint4(0, 0, 0, 0);
    if (tid == 0) {
        mbar_init(bar(kBarInFull0), 1); mbar_init(bar(kBarInFull1), 1);
        mbar_init(bar(kBarInFree0), kL0Warps); mbar_init(bar(kBarInFree1), kL0Warps);
        mbar_init(bar(kBarA1TopReady), kL0Warps); mbar_init(bar(kBarA1BotReady), kL0Warps);
        mbar_init(bar(kBarA1TopFree), 1); mbar_init(bar(kBarA1BotFree), 1);
        mbar_init(bar(kBarTmFull0), 1); mbar_init(bar(kBarTmFull1), 1);
        mbar_init(bar(kBarTmEmpty0), kEpiWarps); mbar_init(bar(kBarTmEmpty1), kEpiWarps);
        mbar_init(bar(kBarA2ReadyA), kEpiWarps); mbar_init(bar(kBarA2ReadyB), kEpiWarps);
        mbar_init(bar(kBarW), 1);
        mbar_init(bar(kBarStageFull), kEpiWarps); mbar_init(bar(kBarStageFree), kTailWarps);
        *s_err = 0;
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == kWarpMma) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smem_u32(tmem_slot)), "r"(kTmemCols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tm = __shfl_sync(0xffffffffu, *tmem_slot, 0);
    if constexpr (!kWin && !kTail) {
        // Programmatic dependent launch (launch_fused_map): the NEXT conv-stack launch of this stream may be scheduled as soon
        // as every CTA of this one has got here, so its CTAs start on each SM the moment this grid's CTA there exits -- no
        // launch gap, and SMs that got one image fewer do not idle until the slowest is done.  This grid in turn must not
        // touch global memory before its predecessor has completed, unless the host has shown the two to be independent.
        asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
        if (P.pdl_wait) asm volatile("griddepcontrol.wait;" ::: "memory");
    }
    if constexpr (kTail) {
        // register hand-over (see the warp-role table): the light warpgroups release first, the heavy ones then grow.
        // The two dec branches stay separate: merged into one `warp >= kWarpMma` branch they compile to one
        // USETMAXREG.DEALLOC instead of two, i.e. to a kernel other than the measured one.
        if (warp >= kWarpTail0)    asm volatile("setmaxnreg.dec.sync.aligned.u32 48;");
        else if (warp >= kWarpMma) asm volatile("setmaxnreg.dec.sync.aligned.u32 48;");
        else                       asm volatile("setmaxnreg.inc.sync.aligned.u32 80;");
    }

    auto wait_or_flag = [&](uint32_t b, uint32_t parity, int code) {
        if (mbar_try(b, parity)) return;                 // fast path: already complete
        // ~4 s budget (a wait this long means a broken pipeline, not time-slicing or a debugger); once any wait has timed
        // out every later wait gives up quickly so the CTA drains.  A reported timeout invalidates the whole launch.
        if (!mbar_wait(b, parity, *reinterpret_cast<volatile int*>(s_err) ? 2000LL : kWaitBudgetClk)) atomicOr(s_err, code);
    };

    // TMA load of unit u (an image, or a window of a larger image) into an input slot; the box starts one pixel row above
    // and 16 bytes left of the unit's first pixel, out-of-bounds bytes arrive as zeros = the conv padding at image borders.
    auto tma_load_unit = [&](uint32_t dst, uint32_t b, int u) {
        int x = -16, y = -1, img = u;
        if constexpr (kWin) {
            const int per = P.win_ntx * P.win_nty, w = u % per;
            img = u / per;
            x += 8 * P.win_gx[w % P.win_ntx];
            y += 8 * P.win_gy[w / P.win_ntx];
        }
        tma_load_box(dst, &in_map, b, x, y, img);
    };

    if (warp < kL0Warps) {
        // =============== layer 0 (1->16, K=9): two instruction mixes on two different pipes ========================
        // One warp-iteration = one pooled row (64 pooling windows x 16 out-channels), 2x2 pool + shift/saturate in
        // registers, 16-channel vectors stored straight into act1.  Warps 0..kL0Dp4aWarps-1 compute their rows with
        // dp4a (IDP pipe: 64 lanes/clk/SM, 3 useful MACs per lane-op), the others with warp-level int8 MMA
        // (mma.sync m16n8k16 on the tensor pipe: 2 clk/SM per instruction, shared with the tcgen05 MMAs of layers
        // 1-2).  Neither pipe alone is fast enough (profiles/: dp4a-only 16.4 M img/s with the IDP pipe saturated,
        // mma.sync-only 17.9 M with the tensor pipe saturated); split between them both have headroom.
        const bool use_dp4a = warp < kL0Dp4aWarps;
        // mma.sync operands: lane (g,t); B fragments stay in registers for the whole kernel
        const int g = lane >> 2, t = lane & 3;
        uint32_t bfr[8];
#pragma unroll
        for (int blk = 0; blk < 8; blk++) bfr[blk] = P.w0f[blk][lane];
        for (int k = 0; k < n_local; k++) {
            const int img = (int)blockIdx.x + k * (int)gridDim.x;
            const int slot = k & 1;
            wait_or_flag(bar(kBarInFull0 + slot), (uint32_t)(k >> 1) & 1, kErrInputTimeout);
            const uint32_t* in_w = reinterpret_cast<const uint32_t*>(smem + (slot ? kOffIn1 : kOffIn0));
#pragma unroll 1
            for (int yp = warp; yp < 64; yp += kL0Warps) {
                // act1 rows still being read by image k-1's layer-1 MMAs: rows 0-33 by the top tiles, 32-65 by the bottom
                // ones.  This unit writes row yp+1.
                // Sixteen warps polling one mbarrier are costly (ncu, profiles/r2a_conv_*: 2 166 try_waits per image at
                // A1TopFree -- four pollers per sub-partition next to the one epilogue warp whose progress they wait for).  The
                // alternative is a rendezvous: warp 0 polls and the others park on a hardware named barrier, which costs no
                // issue slots but moves the warps in lockstep behind the slowest.  Measured (tools/pipe_timing_short.py, M img/s
                // conv-only / infer_batch with the same choice in both instantiations): no rendezvous 19.73 / 15.67, at both
                // points 17.88 / 16.09, per sub-partition groups of four 18.82 / 15.62, top point only 19.29 / 16.02, bottom
                // point only 19.08 / 16.23.  So the conv-only and window kernels have every warp poll, and the kTail kernel
                // (+3.5 %) meets at the bottom point only.  Every layer-0 warp reaches each point exactly once per image, so the
                // named barrier stays in step.
                if (k > 0 && yp == warp) wait_or_flag(bar(kBarA1TopFree), (uint32_t)(k - 1) & 1, kErrAct1Timeout);
                if (k > 0 && yp >= 31 && yp - kL0Warps < 31) {
                    if (!kTail || warp == 0) wait_or_flag(bar(kBarA1BotFree), (uint32_t)(k - 1) & 1, kErrAct1Timeout);
                    if constexpr (kTail) l0_bar_sync(kNamedL0Bot);
                }
                if (warp == 0) TRACE(2, 1); else if (warp == kL0Warps - 1) TRACE(3, 1);
                if (use_dp4a) {
                    // ---- dp4a: two adjacent windows per lane (xp = 2*lane, 2*lane+1) so the weight words (uniform
                    // registers) and the input words are fetched once for 384 dp4a.  Pixel columns 4*lane-1 .. 4*lane+4
                    // = slot bytes 4*lane+15 .. 4*lane+20 ----
                    const uint32_t* rp = in_w + (2 * yp) * (kInPitch / 4) + lane + 3;
                    uint32_t A[4], B[4];
#pragma unroll
                    for (int r = 0; r < 4; r++) {
                        const uint32_t w0 = rp[r * (kInPitch / 4)], w1 = rp[r * (kInPitch / 4) + 1], w2 = rp[r * (kInPitch / 4) + 2];
                        A[r] = __funnelshift_r(w0, w1, 24);
                        B[r] = __funnelshift_r(w1, w2, 8);
                    }
                    uint32_t va[4], vb[4];
#pragma unroll
                    for (int o4 = 0; o4 < 4; o4++) {
                        int pa[4], pb[4];
#pragma unroll
                        for (int oo = 0; oo < 4; oo++) {
                            const int o = o4 * 4 + oo;
                            const uint32_t l0 = P.w0[o][0], l1 = P.w0[o][1], l2 = P.w0[o][2];
                            const uint32_t h0 = P.w0[o][3], h1 = P.w0[o][4], h2 = P.w0[o][5];
                            int a00 = dp4a_u8s8(A[0], l0, dp4a_u8s8(A[1], l1, dp4a_u8s8(A[2], l2, 0)));
                            int a01 = dp4a_u8s8(A[0], h0, dp4a_u8s8(A[1], h1, dp4a_u8s8(A[2], h2, 0)));
                            int a10 = dp4a_u8s8(A[1], l0, dp4a_u8s8(A[2], l1, dp4a_u8s8(A[3], l2, 0)));
                            int a11 = dp4a_u8s8(A[1], h0, dp4a_u8s8(A[2], h1, dp4a_u8s8(A[3], h2, 0)));
                            int b00 = dp4a_u8s8(B[0], l0, dp4a_u8s8(B[1], l1, dp4a_u8s8(B[2], l2, 0)));
                            int b01 = dp4a_u8s8(B[0], h0, dp4a_u8s8(B[1], h1, dp4a_u8s8(B[2], h2, 0)));
                            int b10 = dp4a_u8s8(B[1], l0, dp4a_u8s8(B[2], l1, dp4a_u8s8(B[3], l2, 0)));
                            int b11 = dp4a_u8s8(B[1], h0, dp4a_u8s8(B[2], h1, dp4a_u8s8(B[3], h2, 0)));
                            pa[oo] = max4(a00, a01, a10, a11);
                            pb[oo] = max4(b00, b01, b10, b11);
                        }
                        va[o4] = act_pack4(pa[0], pa[1], pa[2], pa[3], P.shift0);
                        vb[o4] = act_pack4(pb[0], pb[1], pb[2], pb[3], P.shift0);
                    }
                    // window 2*lane -> halo column 2*lane+1 (odd plane, index lane); window 2*lane+1 -> column 2*lane+2
                    // (even plane, index lane+1): both 16-byte stores are contiguous across the warp
                    uint8_t* row = smem + kOffA1 + (yp + 1) * kA1P;
                    *reinterpret_cast<uint4*>(row + kA1Q + lane * 16) = make_uint4(va[0], va[1], va[2], va[3]);
                    *reinterpret_cast<uint4*>(row + (lane + 1) * 16) = make_uint4(vb[0], vb[1], vb[2], vb[3]);
                    if (P.dump_l0) {                     // debug / register-protocol path: BRAM channels 0-15
                        uint8_t* d = P.dump_l0 + (size_t)img * 65536 + yp * 64 + 2 * lane;
#pragma unroll
                        for (int c = 0; c < 16; c++) {
                            d[c * 4096] = (uint8_t)(va[c >> 2] >> (8 * (c & 3)));
                            d[c * 4096 + 1] = (uint8_t)(vb[c >> 2] >> (8 * (c & 3)));
                        }
                    }
                } else {
                    // ---- mma.sync m16n8k16: A row = one 2x2 pooling window, K = its 4x4 input patch (k = 4*patch row +
                    // patch column), N = 8 columns = (4 out-channels) x (horizontal member px); 8 column blocks = (vertical
                    // member py) x (oc%4).  Lane (g,t) ends up with all four members of window g (and g+8) for out-channels
                    // 4t..4t+3: thread-local pool, one packed word of the act1 vector.  4 fragments of 16 windows per row
                    // (even windows in rows 0-7, odd ones in rows 8-15: both 128-byte stores are contiguous in their plane).
                    // Patch row t of windows 2g+16f (a0) and 2g+16f+1 (a1): image row 2yp-1+t, columns 4g+32f-1 .. +4 ----
                    const uint32_t* rp = in_w + (2 * yp + t) * (kInPitch / 4) + g + 3;
                    uint8_t* row = smem + kOffA1 + (yp + 1) * kA1P + g * 16 + t * 4;
#pragma unroll
                    for (int f = 0; f < 4; f++) {
                        const uint32_t w0 = rp[8 * f], w1 = rp[8 * f + 1], w2 = rp[8 * f + 2];
                        const uint32_t a0 = __funnelshift_r(w0, w1, 24), a1 = __funnelshift_r(w1, w2, 8);
                        int c[8][4];
#pragma unroll
                        for (int blk = 0; blk < 8; blk++) {
                            c[blk][0] = c[blk][1] = c[blk][2] = c[blk][3] = 0;
                            imma_16816(c[blk], a0, a1, bfr[blk]);
                        }
                        int pe[4], po[4];
#pragma unroll
                        for (int ol = 0; ol < 4; ol++) {
                            pe[ol] = max4(c[ol][0], c[ol][1], c[4 + ol][0], c[4 + ol][1]);
                            po[ol] = max4(c[ol][2], c[ol][3], c[4 + ol][2], c[4 + ol][3]);
                        }
                        const uint32_t we = act_pack4(pe[0], pe[1], pe[2], pe[3], P.shift0);
                        const uint32_t wo = act_pack4(po[0], po[1], po[2], po[3], P.shift0);
                        // window 2g+16f -> halo column odd (plane 1, index g+8f); window +1 -> even plane, index g+8f+1
                        *reinterpret_cast<uint32_t*>(row + kA1Q + f * 128) = we;
                        *reinterpret_cast<uint32_t*>(row + 16 + f * 128) = wo;
                        if (P.dump_l0) {                 // debug / register-protocol path: BRAM channels 0-15
                            uint8_t* d = P.dump_l0 + (size_t)img * 65536 + (size_t)(4 * t) * 4096 + yp * 64 + 2 * g + 16 * f;
#pragma unroll
                            for (int ol = 0; ol < 4; ol++) {
                                d[ol * 4096] = (uint8_t)(we >> (8 * ol));
                                d[ol * 4096 + 1] = (uint8_t)(wo >> (8 * ol));
                            }
                        }
                    }
                }
                if (warp == 0) TRACE(2, 2); else if (warp == kL0Warps - 1) TRACE(3, 2);
                if (yp <= 32 && yp + kL0Warps > 32) {    // this warp's share of pooled rows 0-32 (act1 rows 0-33) is written
                    fence_async_smem();                  // generic-proxy writes -> visible to the MMA (async proxy)
                    __syncwarp();
                    if (lane == 0) mbar_arrive(bar(kBarA1TopReady));
                }
            }
            fence_async_smem();
            __syncwarp();
            if (lane == 0) { mbar_arrive(bar(kBarA1BotReady)); mbar_arrive(bar(kBarInFree0 + slot)); }
        }
        if (warp == 0) TRACE_END(2); else if (warp == kL0Warps - 1) TRACE_END(3);
    } else if (warp < kWarpMma) {
        // =============== epilogue warps ==========================================================================
        const int e = warp - kL0Warps;
        const int q = e & 3;                             // TMEM lane quarter (== warp % 4)
        const int L = q * 32 + lane;
        const uint32_t t_lane = tm + ((uint32_t)(q * 32) << 16);
        uint32_t use0 = 0, use1 = 0;                     // completed uses of each TMEM half (scalars: an array indexed by the
                                                         // half would live in local memory on the critical path)
        for (int k = 0; k < n_local; k++) {
            const int img = (int)blockIdx.x + k * (int)gridDim.x;
            // ---- layer 1: 8 tiles of 128 pooling windows; TMEM -> pool -> shift/ReLU/saturate -> act2 (smem) ----
#pragma unroll 1
            for (int t = 0; t < 8; t++) {
                const int h = t & 1, i0 = (t >> 2) * 16, j0 = (t & 3) * 8;
                if (e == 0) TRACE2(1, 10 + t);
                wait_or_flag(bar(kBarTmFull0 + h), (h ? use1 : use0) & 1, kErrMmaTimeout);
                if (h) use1++; else use0++;
                if (e == 0) TRACE2(1, 20 + t);
                tc_fence_after();
                const int i = i0 + (L >> 3), j = j0 + (L & 7);
                // channel half: 16 of the 32 output channels.  e >> 2 is always 0, but a literal 0 here schedules the window
                // instantiation differently; this start keeps the measured code.
#pragma unroll
                for (int g = e >> 2; g < 2; g++) {
                    const uint32_t taddr = t_lane + h * 256 + g * 16;
                    int mx[16];
                    {
                        int v0[16], v1[16];
                        tmem_ld16(taddr, v0);
                        tmem_ld16(taddr + 32, v1);
                        tmem_ld_wait();
#pragma unroll
                        for (int c = 0; c < 16; c++) mx[c] = max(v0[c], v1[c]);
                        tmem_ld16(taddr + 64, v0);
                        tmem_ld16(taddr + 96, v1);
                        tmem_ld_wait();
#pragma unroll
                        for (int c = 0; c < 16; c++) mx[c] = max(mx[c], max(v0[c], v1[c]));
                    }
                    if (g == 1) {                        // last read of this TMEM half by this warp
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(bar(kBarTmEmpty0 + h));
                    }
                    uint4 w;
                    w.x = act_pack4(mx[0], mx[1], mx[2], mx[3], P.shift1);
                    w.y = act_pack4(mx[4], mx[5], mx[6], mx[7], P.shift1);
                    w.z = act_pack4(mx[8], mx[9], mx[10], mx[11], P.shift1);
                    w.w = act_pack4(mx[12], mx[13], mx[14], mx[15], P.shift1);
                    *reinterpret_cast<uint4*>(smem + kOffA2 + g * kA2C + (i + 1) * kA2P + ((j + 1) & 1) * kA2Q + ((j + 1) >> 1) * 16) = w;
                    if (P.dump_l1) {                     // BRAM channels 16-47
                        uint8_t* d = P.dump_l1 + (size_t)img * 32768 + (size_t)(g * 16) * 1024 + i * 32 + j;
                        const uint32_t ww[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
                        for (int c = 0; c < 16; c++) d[c * 1024] = (uint8_t)(ww[c >> 2] >> (8 * (c & 3)));
                    }
                }
                if (t >= 6) {
                    // layer-2 block 0 reads act2 columns 0-16 only: everything but tile 7 (rows 16-31, columns 24-31),
                    // so it can start while tile 7 is still being drained
                    fence_async_smem();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(bar(t == 6 ? kBarA2ReadyA : kBarA2ReadyB));
                }
            }

            // ---- layer 2: 2 blocks of 128 pooling windows x 4 parities; -> staging (CHW) -> one 16 KiB TMA store ----
            constexpr bool win = kWin;
            uint8_t* wbase = nullptr;                    // window mode: this lane's pixel in channel 0 of the big feature map
            size_t wcs = 0;                              // ... and the channel stride
            bool wrow = false;
            int wgx = 0, wlo = 0, whi = 0;
            if (win) {
                const int per = P.win_ntx * P.win_nty, w = img % per, gy = P.win_gy[w / P.win_ntx], i = L >> 3;
                wgx = P.win_gx[w % P.win_ntx];
                wlo = wgx == 0 ? 0 : 1; whi = wgx == P.win_wo - 16 ? 15 : 14;
                wrow = i >= (gy == 0 ? 0 : 1) && i <= (gy == P.win_ho - 16 ? 15 : 14);
                wcs = (size_t)P.win_ho * P.win_wo;
                wbase = P.out + ((size_t)(img / per) * 64 * P.win_ho + gy + i) * P.win_wo + wgx;
            } else if (k > 0) {                          // the previous image's store and its tail must be done with staging
                if (P.out && e == 0 && lane == 0) bulk_store_wait_read();
                if (e == 0) TRACE(1, 70);
                if constexpr (kTail) stage_bar_sync(kNamedStageFree);        // the tail has released the previous image's map
                else epi_bar_sync();
                if (e == 0) TRACE(1, 71);
            }
#pragma unroll 1
            for (int s = 0; s < 2; s++) {
                const int h = s, j0 = s * 8;
                if (e == 0) TRACE2(1, 40 + s);
                wait_or_flag(bar(kBarTmFull0 + h), (h ? use1 : use0) & 1, kErrMmaTimeout);
                if (h) use1++; else use0++;
                if (e == 0) TRACE2(1, 50 + s);
                tc_fence_after();
                const int i = L >> 3, j = j0 + (L & 7);
#pragma unroll
                for (int cg = 0; cg < 4; cg++) {         // group of 16 output channels
                    const uint32_t taddr = t_lane + h * 256 + cg * 16;
                    int m[16];
                    {
                        int v0[16], v1[16];
                        tmem_ld16(taddr, v0);
                        tmem_ld16(taddr + 64, v1);
                        tmem_ld_wait();
                        if (P.acc24) {
#pragma unroll
                            for (int c = 0; c < 16; c++) { v0[c] = wrap24(v0[c]); v1[c] = wrap24(v1[c]); }
                        }
#pragma unroll
                        for (int c = 0; c < 16; c++) m[c] = max(v0[c], v1[c]);
                        tmem_ld16(taddr + 128, v0);
                        tmem_ld16(taddr + 192, v1);
                        tmem_ld_wait();
                        if (P.acc24) {
#pragma unroll
                            for (int c = 0; c < 16; c++) { v0[c] = wrap24(v0[c]); v1[c] = wrap24(v1[c]); }
                        }
#pragma unroll
                        for (int c = 0; c < 16; c++) m[c] = max(m[c], max(v0[c], v1[c]));
                    }
                    if (cg == 3) {                       // last read of this TMEM half by this warp
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(bar(kBarTmEmpty0 + h));
                    }
                    if (win) {
                        if (wrow && j >= wlo && j <= whi) {
                            uint8_t* o = wbase + (size_t)(cg * 16) * wcs + j;
#pragma unroll
                            for (int c = 0; c < 16; c++) o[c * wcs] = (uint8_t)act_u8(m[c], P.shift2);
                        }
                    } else {
                        uint8_t* o = smem + kOffStage + (cg * 16) * 256 + i * 16 + j;
#pragma unroll
                        for (int c = 0; c < 16; c++) o[c * 256] = (uint8_t)act_u8(m[c], P.shift2);
                    }
                }
            }
            if (!win) {
                if constexpr (kTail) {                   // hand the staged map to the tail warps
                    stage_bar_arrive(kNamedStageFull);
                    if (e == 0) TRACE(1, 72);
                }
                if (P.out) {
                    fence_async_smem();
                    epi_bar_sync();
                    if (e == 0 && lane == 0) bulk_store(P.out + (size_t)img * 16384, s_base + kOffStage, kStageBytes);
                }
            }
        }
        if (e == 0 && lane == 0) {
            bulk_store_wait_all();
            if (P.done_flag) {                           // cnnacc_infer_one: one CTA, features in mapped host memory
                if (*reinterpret_cast<volatile int*>(s_err)) *reinterpret_cast<volatile int*>(P.status_host) = *s_err;
                __threadfence_system();                  // the feature bytes (and the status) before the flag
                *reinterpret_cast<volatile int*>(P.done_flag) = P.done_seq;
            }
        }
        if (e == 0) TRACE_END(1);
    } else if (warp == kWarpMma) {
        // =============== MMA issue + TMA loads: the whole warp walks the schedule, one elected lane issues ========
        // TMA: weights once, then every image two ahead of its consumer (the prefetch of image k+2 is issued when
        // layer 0 has released image k's slot, which this warp learns while waiting for image k's bottom rows anyway).
        if (elect_one()) {
            mbar_expect_tx(bar(kBarW), kB1Bytes + kB2Bytes);
            bulk_load(s_base + kOffB1, P.b1, kB1Bytes, bar(kBarW));
            bulk_load(s_base + kOffB2, P.b2, kB2Bytes, bar(kBarW));
            for (int k = 0; k < 2 && k < n_local; k++) {
                mbar_expect_tx(bar(kBarInFull0 + k), kInBytes);
                tma_load_unit(s_base + (k ? kOffIn1 : kOffIn0), bar(kBarInFull0 + k), (int)blockIdx.x + k * (int)gridDim.x);
            }
        }
        __syncwarp();
        wait_or_flag(bar(kBarW), 0, kErrWeightTimeout);
        constexpr uint32_t idesc1 = umma_idesc_i8(128), idesc2 = umma_idesc_i8(64);
        uint32_t use0 = 0, use1 = 0;                     // uses of each TMEM half issued so far
        for (int k = 0; k < n_local; k++) {
            // ---- layer 1: 8 tiles (2 row halves x 4 column blocks) x 8 K-slabs, N = 128 ----
#pragma unroll 1
            for (int t = 0; t < 8; t++) {
                const int h = t & 1, ty = t >> 2, tx = t & 3;
                TRACE2(0, 10 + t);
                if (t == 0) { TRACE(0, 1); wait_or_flag(bar(kBarA1TopReady), (uint32_t)k & 1, kErrAct1Timeout); TRACE(0, 2); }
                if (t == 4) {
                    TRACE(0, 3);
                    wait_or_flag(bar(kBarA1BotReady), (uint32_t)k & 1, kErrAct1Timeout);
                    if (k + 2 < n_local) {               // layer 0 is done with image k: refill its slot with image k+2
                        const int slot = k & 1;
                        wait_or_flag(bar(kBarInFree0 + slot), (uint32_t)(k >> 1) & 1, kErrSlotTimeout);
                        if (elect_one()) {
                            mbar_expect_tx(bar(kBarInFull0 + slot), kInBytes);
                            tma_load_unit(s_base + (slot ? kOffIn1 : kOffIn0), bar(kBarInFull0 + slot),
                                          (int)blockIdx.x + (k + 2) * (int)gridDim.x);
                        }
                        __syncwarp();
                    }
                    TRACE(0, 4);
                }
                TRACE2(0, 20 + t);
                wait_or_flag(bar(kBarTmEmpty0 + h), ((h ? use1 : use0) & 1) ^ 1, kErrEmptyTimeout);   // previous use drained
                if (h) use1++; else use0++;
                TRACE2(0, 30 + t);
                tc_fence_after();
                if (elect_one()) {
                    const uint32_t d = tm + h * 256;
                    const uint64_t a0 = umma_desc(s_base + kOffA1 + (32 * ty) * kA1P + (8 * tx) * 16, kA1Q, 2 * kA1P);
                    const uint64_t bw = umma_desc(s_base + kOffB1, 2048, 128);                 // N = 128 slabs
                    const uint64_t bn = umma_desc(s_base + kOffB1 + 4 * kB1Slab, 1024, 128);   // N = 64 slabs
#pragma unroll
                    for (int q = 0; q < 4; q++) {        // patch rows 1, 2 reach all four window members; the first overwrites
                        const int r = 1 + (q >> 1), sx = q & 1;
                        umma_i8(d, a0 + (uint64_t)((r * kA1P + sx * 16) >> 4), bw + (uint64_t)((q * kB1Slab) >> 4), idesc1, q > 0);
                    }
#pragma unroll
                    for (int q = 0; q < 4; q++) {        // patch row 0 -> upper members (columns 0-63), row 3 -> lower (64-127)
                        const int r = (q >> 1) ? 3 : 0, sx = q & 1;
                        umma_i8(d + (uint32_t)(q >> 1) * 64u, a0 + (uint64_t)((r * kA1P + sx * 16) >> 4),
                                bn + (uint64_t)((q * kB1Half) >> 4), idesc2, 1);
                    }
                    umma_commit(bar(kBarTmFull0 + h));
                    if (t == 3) umma_commit(bar(kBarA1TopFree));
                    if (t == 7) umma_commit(bar(kBarA1BotFree));
                }
                __syncwarp();
            }
            // ---- layer 2: 2 blocks x 4 parities x 9 taps, N = 64 ----
#pragma unroll 1
            for (int s = 0; s < 2; s++) {
                const int h = s, j0 = s * 8;
                TRACE(0, 40 + s);
                wait_or_flag(bar(s ? kBarA2ReadyB : kBarA2ReadyA), (uint32_t)k & 1, kErrAct2Timeout);
                wait_or_flag(bar(kBarTmEmpty0 + h), ((h ? use1 : use0) & 1) ^ 1, kErrEmptyTimeout);
                if (h) use1++; else use0++;
                TRACE(0, 50 + s);
                tc_fence_after();
                if (elect_one()) {
                    const uint64_t a0 = umma_desc(s_base + kOffA2 + j0 * 16, kA2C, 2 * kA2P);
                    const uint64_t b0 = umma_desc(s_base + kOffB2, 1024, 128);
#pragma unroll
                    for (int p = 0; p < 4; p++) {
                        const int a = p >> 1, b = p & 1;
                        const uint32_t d = tm + h * 256 + p * 64;
#pragma unroll
                        for (int t = 0; t < 9; t++) {
                            const int dy = t / 3, dx = t % 3;
                            const int aoff = (a + dy) * kA2P + ((b + dx) & 1) * kA2Q + ((b + dx) >> 1) * 16;
                            umma_i8(d, a0 + (uint64_t)(aoff >> 4), b0 + (uint64_t)((t * 2048) >> 4), idesc2, t > 0);
                        }
                    }
                    umma_commit(bar(kBarTmFull0 + h));
                }
                __syncwarp();
                TRACE(0, 60 + s);
            }
        }
        TRACE_END(0);
    } else if (kTail && warp >= kWarpTail0) {
        // =============== tail warps: staged features -> class / probabilities / CAM box (tail.cuh) =================
        const int T = (warp - kWarpTail0) * 32 + lane;
        TailScratch* sc = reinterpret_cast<TailScratch*>(smem + kOffTail);
        const TailWeights W = tail_stage_weights(reinterpret_cast<float*>(smem + kOffTailW), kTailWRows, P.tail, T);
        tail_bar(kNamedTailFront);
        for (int k = 0; k < n_local; k++) {
            const int img = (int)blockIdx.x + k * (int)gridDim.x;
            stage_bar_sync(kNamedStageFull);
            float c0, c1;
            const bool want_box = tail_front(smem + kOffStage, sc, T, kNamedTailFront, P.tail, W, (size_t)img, c0, c1, [&] {
                if (k + 1 < n_local) stage_bar_arrive(kNamedStageFree);    // the epilogue only waits for it before the next image
            }, [&](int code) { if (T == 0) TRACE(4, code); (void)code; });
            if (want_box) {                              // hand the CAM to the back warps (single 1 KiB buffer)
                if (k > 0) cam_bar_sync(kNamedCamFree);
                reinterpret_cast<float2*>(sc->cam)[T] = make_float2(c0, c1);
                cam_bar_arrive(kNamedCamFull);
            }
        }
        if (T == 0) TRACE_END(4);
    } else if (kTail && warp >= kWarpTailBack0 && warp < kWarpTail0) {
        // =============== tail back warps: CAM -> maximum, 70th percentile, box; one image behind the front warps =========
        if (P.tail.bbox_out) {
            const int T = (warp - kWarpTailBack0) * 32 + lane;
            TailScratch* sc = reinterpret_cast<TailScratch*>(smem + kOffTail);
            for (int k = 0; k < n_local; k++) {
                const int img = (int)blockIdx.x + k * (int)gridDim.x;
                cam_bar_sync(kNamedCamFull);
                const float4 q = reinterpret_cast<const float4*>(sc->cam)[T];
                float cam[4] = {q.x, q.y, q.z, q.w};
                if (k + 1 < n_local) cam_bar_arrive(kNamedCamFree);
                tail_back(cam, sc, T, kNamedTailBack, P.tail, (size_t)img, [&](int code) { if (T == 0) TRACE(5, code); (void)code; });
            }
            if (T == 0) TRACE_END(5);
        }
    }

    // ---- teardown ---------------------------------------------------------------------------------------------
    tc_fence_before();
    __syncthreads();
#ifdef CNNACC_TRACE
    if (blockIdx.x == 0 && tid == 0)
        for (int r = 0; r < kTraceRoles; r++)
            for (int i = 0; i < trace_cnt[r]; i++)
                printf("TRACE %d %d %u\n", r, (int)(trace_buf[r * kTraceMax + i] >> 24), trace_buf[r * kTraceMax + i] & 0xFFFFFFu);
#endif
    if (tid == 0 && *s_err) {
        atomicOr(P.status, *s_err);
        *reinterpret_cast<volatile int*>(P.status_host) = *s_err;
        __threadfence_system();
    }
    if (warp == kWarpMma) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tm), "r"(kTmemCols) : "memory");
}

// ---- host side ------------------------------------------------------------------------------------------------
struct FusedWeights {
    uint32_t w0[16][6];
    uint32_t w0f[8][32];
    uint8_t* d_b1 = nullptr;
    uint8_t* d_b2 = nullptr;
    int* d_status = nullptr;
    int* h_status = nullptr;      // mapped pinned mirror of the status word
    int* h_status_dev = nullptr;  // its device address
    bool attr_set = false;
    bool acc24 = false;           // cnnacc_set_accumulator_bits(24)
};

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                    const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// Looked up once per process; the initialisation of a function-local static is thread-safe (handles of a sharded call encode
// tensor maps from several threads at once).
inline PFN_encodeTiled get_encode_tiled() {
    static const PFN_encodeTiled fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        return (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
                qres == cudaDriverEntryPointSuccess) ? (PFN_encodeTiled)p : nullptr;
    }();
    return fn;
}

// Pure host permutation of weights.bin (parse_kernels, arm_cnn.c:43-59, done once) into the three operand layouts.
inline void fused_pack_weights(const uint8_t* wbin, uint32_t w0[16][6], uint32_t w0f[8][32], uint8_t* b1, uint8_t* b2) {
    // layer 0, mma.sync B fragments: lane (g,t) of block (py, ol) holds patch row r = t, columns c = 0..3 of
    // output column n = g -> out-channel 4*(g>>1) + ol, horizontal member px = g&1:  w0[oc][r - py][c - px]
    for (int blk = 0; blk < 8; blk++)
        for (int lane = 0; lane < 32; lane++) {
            const int py = blk >> 2, ol = blk & 3, g = lane >> 2, t = lane & 3, oc = 4 * (g >> 1) + ol, px = g & 1;
            uint32_t word = 0;
            for (int c = 0; c < 4; c++) {
                const int dy = t - py, dx = c - px;
                if (dy >= 0 && dy <= 2 && dx >= 0 && dx <= 2) word |= (uint32_t)weight_byte(wbin, 0, oc, 0, dy * 3 + dx) << (8 * c);
            }
            w0f[blk][lane] = word;
        }
    std::memset(b1, 0, kB1Bytes);
    std::memset(b2, 0, kB2Bytes);
    for (int o = 0; o < 16; o++)
        for (int dy = 0; dy < 3; dy++) {
            uint32_t lo = (uint32_t)weight_byte(wbin, 0, o, 0, dy * 3) | (uint32_t)weight_byte(wbin, 0, o, 0, dy * 3 + 1) << 8 |
                          (uint32_t)weight_byte(wbin, 0, o, 0, dy * 3 + 2) << 16;
            w0[o][dy] = lo;
            w0[o][3 + dy] = lo << 8;
        }
    // layer 1 (Toeplitz over a 2x2 pooling window): slab (patch row r, column pair sx), K byte k = jx*16 + ic is patch
    // pixel (r, 2*sx + jx) channel ic, N row n = (py*2 + px)*32 + oc is window member (py,px):
    //   B[n][k] = w1[oc][ic][r - py][2*sx + jx - px]   when both tap indices are in 0..2, else 0
    // Patch rows 1, 2 reach both window rows: N = 128 slabs, K-major, at ((r-1)*2 + sx)*4096 + (k/16)*2048 + (n/8)*128 +
    // (n%8)*16 + k%16.  Patch row 0 only reaches py = 0 and patch row 3 only py = 1 (the other half would be all zero):
    // N = 64 slabs over n' = n % 64 at 16384 + ((r==3)*2 + sx)*2048 + (k/16)*1024 + (n'/8)*128 + (n'%8)*16 + k%16.
    for (int sl = 0; sl < 8; sl++)
        for (int n = 0; n < 128; n++)
            for (int kk = 0; kk < 32; kk++) {
                const int r = sl >> 1, sx = sl & 1, py = n >> 6, px = (n >> 5) & 1, oc = n & 31, jx = kk >> 4, ic = kk & 15;
                const int dy = r - py, dx = 2 * sx + jx - px;
                if (dy < 0 || dy > 2 || dx < 0 || dx > 2) continue;
                const uint8_t wv = weight_byte(wbin, 1, oc, ic, dy * 3 + dx);
                if (r == 1 || r == 2) {
                    b1[((r - 1) * 2 + sx) * kB1Slab + jx * 2048 + (n / 8) * 128 + (n % 8) * 16 + ic] = wv;
                } else {
                    const int nn = n & 63;               // r == 0 -> py == 0, r == 3 -> py == 1
                    b1[4 * kB1Slab + ((r == 3 ? 2 : 0) + sx) * kB1Half + jx * 1024 + (nn / 8) * 128 + (nn % 8) * 16 + ic] = wv;
                }
            }
    // layer 2: tap t, K = input channel; B[n][k] at t*2048 + (k/16)*1024 + (n/8)*128 + (n%8)*16 + k%16
    for (int t = 0; t < 9; t++)
        for (int n = 0; n < 64; n++)
            for (int ic = 0; ic < 32; ic++)
                b2[t * 2048 + (ic / 16) * 1024 + (n / 8) * 128 + (n % 8) * 16 + (ic % 16)] = weight_byte(wbin, 2, n, ic, t);
}

// Pack and upload.  Returns a cudaError_t as int.
inline int fused_load_weights(FusedWeights& fw, const uint8_t* wbin) {
    std::vector<uint8_t> b1(kB1Bytes), b2(kB2Bytes);
    fused_pack_weights(wbin, fw.w0, fw.w0f, b1.data(), b2.data());
    cudaError_t e;
    if (!fw.d_b1 && (e = cudaMalloc(&fw.d_b1, kB1Bytes)) != cudaSuccess) return (int)e;
    if (!fw.d_b2 && (e = cudaMalloc(&fw.d_b2, kB2Bytes)) != cudaSuccess) return (int)e;
    if (!fw.d_status) {
        if ((e = cudaMalloc(&fw.d_status, sizeof(int))) != cudaSuccess) return (int)e;
        if ((e = cudaMemset(fw.d_status, 0, sizeof(int))) != cudaSuccess) return (int)e;
        if ((e = cudaHostAlloc(&fw.h_status, sizeof(int), cudaHostAllocMapped)) != cudaSuccess) return (int)e;
        *fw.h_status = 0;
        if ((e = cudaHostGetDevicePointer(&fw.h_status_dev, fw.h_status, 0)) != cudaSuccess) return (int)e;
    }
    if ((e = cudaMemcpy(fw.d_b1, b1.data(), kB1Bytes, cudaMemcpyHostToDevice)) != cudaSuccess) return (int)e;
    if ((e = cudaMemcpy(fw.d_b2, b2.data(), kB2Bytes, cudaMemcpyHostToDevice)) != cudaSuccess) return (int)e;
    if (!fw.attr_set) {
        if ((e = cudaFuncSetAttribute(conv_stack_fused_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kFusedSmem)) != cudaSuccess) return (int)e;
        if ((e = cudaFuncSetAttribute(conv_stack_fused_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kFusedSmem)) != cudaSuccess) return (int)e;
        if ((e = cudaFuncSetAttribute(conv_stack_fused_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kFusedSmem)) != cudaSuccess) return (int)e;
        fw.attr_set = true;
    }
    if (!get_encode_tiled()) return (int)cudaErrorNotSupported;
    return 0;
}

inline void fused_free(FusedWeights& fw) {
    cudaFree(fw.d_b1); cudaFree(fw.d_b2); cudaFree(fw.d_status);
    if (fw.h_status) cudaFreeHost(fw.h_status);
    fw.d_b1 = fw.d_b2 = nullptr; fw.d_status = nullptr; fw.h_status = fw.h_status_dev = nullptr;
}

// Tensor map over n images [n][H][W] u8 (W a multiple of 16) at a device-accessible address (device memory or mapped
// pinned host memory); the box is always the kernel's 160 x 130 input slot.
inline int fused_encode_map(const uint8_t* d_imgs, int64_t n, CUtensorMap* map, int H = 128, int W = 128) {
    if (n <= 0 || n > 0x7fffffff || (reinterpret_cast<uintptr_t>(d_imgs) & 15) || (W & 15) || !get_encode_tiled()) return (int)cudaErrorInvalidValue;
    const cuuint64_t gdim[3] = {(cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)n};
    const cuuint64_t gstride[2] = {(cuuint64_t)W, (cuuint64_t)W * H};
    const cuuint32_t box[3] = {(cuuint32_t)kInPitch, (cuuint32_t)kInRows, 1};
    const cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = get_encode_tiled()(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, const_cast<uint8_t*>(d_imgs), gdim, gstride, box, estr,
                                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? 0 : (int)cudaErrorInvalidValue;
}

// One launch for the n images described by `map`.  Returns a cudaError_t as int (0 = launched).
struct FusedWindows {             // window mode: see FusedParams
    int ntx = 0, nty = 0, ho = 0, wo = 0;     // windows per row / column, feature-map size of the big image
    const short *gx = nullptr, *gy = nullptr;
};
inline int launch_fused_map(const FusedWeights& fw, cudaStream_t stream, const CUtensorMap& map, int64_t n, uint8_t* d_feats,
                            const int* shifts, int sm_count, uint8_t* dump_l0, uint8_t* dump_l1, const FusedWindows* win = nullptr,
                            const TailArgs* tail = nullptr, int* done_flag = nullptr, int done_seq = 0, int pdl_wait = -1) {
    FusedParams P;
    P.pdl_wait = pdl_wait != 0;
    P.done_flag = (n == 1 && !win && !tail) ? done_flag : nullptr;
    P.done_seq = done_seq;
    if (win && tail) return (int)cudaErrorInvalidValue;
    if (!tail && !d_feats) return (int)cudaErrorInvalidValue;
    std::memset(&P.tail, 0, sizeof(P.tail));
    if (tail) P.tail = *tail;
    P.win_ntx = P.win_nty = P.win_ho = P.win_wo = 0;
    if (win) {
        if (win->ntx < 1 || win->nty < 1 || win->ntx > 80 || win->nty > 80) return (int)cudaErrorInvalidValue;
        P.win_ntx = win->ntx; P.win_nty = win->nty; P.win_ho = win->ho; P.win_wo = win->wo;
        std::memcpy(P.win_gx, win->gx, win->ntx * sizeof(short));
        std::memcpy(P.win_gy, win->gy, win->nty * sizeof(short));
    }
    std::memcpy(P.w0, fw.w0, sizeof(P.w0));
    std::memcpy(P.w0f, fw.w0f, sizeof(P.w0f));
    P.shift0 = shifts[0]; P.shift1 = shifts[1]; P.shift2 = shifts[2];
    P.acc24 = fw.acc24 ? 1 : 0;
    P.n_images = (int)n;
    P.b1 = fw.d_b1; P.b2 = fw.d_b2;
    P.out = d_feats; P.dump_l0 = dump_l0; P.dump_l1 = dump_l1;
    P.status = fw.d_status; P.status_host = fw.h_status_dev;
    const int grid = (int)std::min<int64_t>(n, sm_count);
    if (win)       conv_stack_fused_kernel<true, false><<<grid, kFusedThreads, kFusedSmem, stream>>>(map, P);
    else if (tail) conv_stack_fused_kernel<false, true><<<grid, kTailKernelThreads, kFusedSmem, stream>>>(map, P);
    else if (pdl_wait < 0) conv_stack_fused_kernel<false, false><<<grid, kFusedThreads, kFusedSmem, stream>>>(map, P);
    else {
        // programmatic stream serialisation: this launch may begin while the previous kernel of the stream is still
        // running; pdl_wait (above) says whether the kernel must then wait for it before its first global access
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)grid); cfg.blockDim = dim3(kFusedThreads); cfg.dynamicSmemBytes = kFusedSmem; cfg.stream = stream;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr; cfg.numAttrs = 1;
        return (int)cudaLaunchKernelEx(&cfg, conv_stack_fused_kernel<false, false>, map, P);
    }
    return (int)cudaGetLastError();
}

// One launch for n device-resident images.
inline int launch_fused(const FusedWeights& fw, cudaStream_t stream, const uint8_t* d_imgs, int64_t n, uint8_t* d_feats,
                        const int* shifts, int sm_count, uint8_t* dump_l0, uint8_t* dump_l1, const TailArgs* tail = nullptr,
                        int pdl_wait = -1) {
    if (n <= 0) return 0;
    CUtensorMap map;
    int rc = fused_encode_map(d_imgs, n, &map);
    if (rc) return rc;
    return launch_fused_map(fw, stream, map, n, d_feats, shifts, sm_count, dump_l0, dump_l1, nullptr, tail, nullptr, 0, pdl_wait);
}

// Reads (and clears) the status word; non-zero = a pipeline wait timed out inside some launch.  The caller has
// synchronised the stream, so the host-mapped mirror is current and no CUDA call is needed on the good path.
inline int fused_poll_status(const FusedWeights& fw, int* bits) {
    *bits = 0;
    if (!fw.h_status) return 0;
    *bits = *reinterpret_cast<volatile int*>(fw.h_status);
    if (!*bits) return 0;
    *fw.h_status = 0;
    return (int)cudaMemset(fw.d_status, 0, sizeof(int));
}

}  // namespace cnnacc
