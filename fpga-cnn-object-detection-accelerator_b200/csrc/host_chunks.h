// host_chunks.h -- how a host-pointer conv-stack call is cut into staging chunks (pure host arithmetic, no CUDA).
//
// A ring of staging buffers is driven through one stream per engine (H2D copies, kernels, D2H copies), chained by per-slot
// events, so copies in both directions and the kernels overlap.  chunk = what one slot stages.
//  * Synchronous call: the first H2D and the last D2H cannot overlap anything, so a call wants at least ~4 chunks; each chunk
//    costs ~20-40 us of cross-engine hand-offs on top of its copies (tools/probe_pipeline.cu shows the same for any
//    H2D -> kernel -> D2H chain), so they should not be small either: a quarter of the call, clamped to 4..32 MiB
//    (profiles/r1_e2e_chunk_sweep.txt).  Chunk sizes ramp up at the start and down at the end (1/4, 1/2, 1, ..., 1, 1/2, 1/4 of
//    the full chunk for depth 2): the shorter the lone first H2D and last D2H are, the sooner both directions are busy together.
//  * Streamed call (cnnacc_run_batch_async): the neighbouring calls cover a call's edges, so only the hand-off cost counts: one
//    chunk per call up to 64 MiB, no ramp (profiles/r2_e2e_stream_sweep.txt: 2.85 M img/s at 64 MiB, 2.77 M at 32, 2.60 M at 16,
//    batch 4096, 3 in flight).
// tests/test_boundary_cpu.py replays the plans through cnnacc_chunk_plan_host.
#pragma once
#include <algorithm>
#include <cstddef>
#include <cstdint>

namespace cnnacc {

struct HostChunkPlan {
    int64_t n = 0;            // images in the call
    int64_t full = 1;         // images of a full-size chunk (what every slot must hold)
    int depth = 0;            // ramp steps at each end (0: all chunks full-size, the last one takes the remainder)
    int64_t tail_total = 0;   // images in the ramp-down pieces: full/2 + full/4 + ... + full/2^depth

    // size of chunk number `ci` that starts at image `i0` (1 <= size <= min(full, n - i0))
    int64_t next(int64_t i0, int64_t ci) const {
        int64_t m = full;
        if (depth) {
            const int64_t left = n - i0;
            if (ci < depth) m = full >> (depth - ci);                                  // ramp up
            else if (left <= tail_total) {                                             // ramp down: largest full/2^j that fits, remainder first
                int64_t piece = full >> 1, rest = tail_total;
                while (piece > 1 && left <= rest - piece) { rest -= piece; piece >>= 1; }
                m = left - (rest - piece);
            } else if (left < full + tail_total) m = left - tail_total;                // the last full-size piece takes the remainder
            m = std::max<int64_t>(m, 1);
        }
        return std::min(m, n - i0);
    }
};

constexpr int kHostRampDepth = 2;   // ramp steps at each end of a synchronous call (see above)

// in_sz: bytes per image; cap_images: most images a chunk may hold (workspace bound of the per-layer path)
inline HostChunkPlan make_host_chunk_plan(int64_t n, size_t in_sz, int64_t cap_images, bool pipelined) {
    HostChunkPlan p;
    p.n = n;
    const size_t call_bytes = (size_t)n * in_sz;
    size_t chunk_bytes = std::min<size_t>((size_t)32 << 20, std::max<size_t>((size_t)4 << 20, call_bytes / 4));
    if (pipelined) chunk_bytes = std::min<size_t>((size_t)64 << 20, std::max<size_t>((size_t)4 << 20, call_bytes));
    p.full = std::min<int64_t>(n, std::max<int64_t>(1, std::min<int64_t>(cap_images, (int64_t)(chunk_bytes / in_sz))));
    p.depth = (!pipelined && n >= 4 * p.full && (p.full >> kHostRampDepth) >= 1) ? kHostRampDepth : 0;
    p.tail_total = p.full - (p.full >> p.depth);
    return p;
}

}  // namespace cnnacc
