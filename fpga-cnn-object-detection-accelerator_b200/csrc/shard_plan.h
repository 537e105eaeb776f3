// shard_plan.h -- how a sharded host-batch call (cnnacc_*_sharded) cuts one batch over its member handles (pure host
// arithmetic, no CUDA).
//
// Shard i is the contiguous range [begin(i), begin(i+1)) with begin(i) = n*i/m: near-equal pieces (sizes differ by at most
// one unit), the same cut as bench.py's shard_range.  A call only spreads over as many members as keep every shard at
// about kMinShardBytes of input or more: below that a second member's thread start, per-call synchronisation and its own
// ramped first H2D / last D2H cost more than the copies it takes over.
// tests/test_shard_plan_cpu.py replays the plans through cnnacc_shard_plan_host.
#pragma once
#include <algorithm>
#include <cstdint>

namespace cnnacc {

// Smallest input per shard worth a member of its own: 2 MiB (128 images of 128x128).  From tools/sharded_scaling.py's sweep
// on a one-GPU B200 box (1000 W limit, profiles/r3_sharded_sweep_1gpu.jsonl): one member's host call takes 57-63 us up to 8
// images, then 76 / 71 / 85 / 105 / 151 / 235 us for 16 ... 512 images (infer_batch; run_batch 65 / 74 / 88 / 134 / 216 /
// 325 us), and spreading a call over a second member adds 25-30 us (its thread, its own synchronisation).  Two GPUs with
// links of their own therefore win once t(n) - t(n/2) exceeds that: from 256 images (4 MiB, 2 MiB a shard) for infer_batch,
// 128 for run_batch.  Two devices against one were not measured (the box has one GPU).
constexpr int64_t kMinShardBytes = (int64_t)2 << 20;

struct ShardPlan {
    int64_t n = 0;            // units (images / frames) in the call
    int m = 1;                // members used: shards 0 .. m-1
    int64_t begin(int i) const { return (int64_t)((__int128)n * i / m); }
};

// n >= 0, n_handles >= 1, unit_bytes >= 1: m = min(n_handles, max(1, n*unit_bytes / kMinShardBytes))
inline ShardPlan make_shard_plan(int64_t n, int n_handles, int64_t unit_bytes) {
    ShardPlan p;
    p.n = n;
    const __int128 wanted = (__int128)n * unit_bytes / kMinShardBytes;
    p.m = (int)std::max<__int128>(1, std::min<__int128>(n_handles, wanted));
    return p;
}

}  // namespace cnnacc
