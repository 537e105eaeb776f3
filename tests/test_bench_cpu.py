"""Host-side logic of bench.py: sharding and the max-over-ranks reduction, exercised with gloo, world_size 2."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def test_shard_range_partitions_exactly():
    for n in (0, 1, 7, 65536, 1_000_000):
        for world in (1, 2, 4, 8):
            spans = [bench.shard_range(n, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(spans[i][1] == spans[i + 1][0] for i in range(world - 1))
            sizes = [hi - lo for lo, hi in spans]
            assert max(sizes) - min(sizes) <= 1


def _worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    lo, hi = bench.shard_range(1001, rank, world)
    mx = bench.reduce_max(10.0 + rank, dist)            # rank 1 is "slower"
    counts = bench.gather_counts(hi - lo, dist)
    q.put((rank, mx, counts))
    dist.destroy_process_group()


def test_two_rank_gloo_reduction():
    import torch.multiprocessing as tmp
    ctx = tmp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + os.getpid() % 2000
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=120) for _ in procs)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for rank, mx, counts in res:
        assert mx == 11.0                               # max over ranks, seen by every rank
        assert counts == [500, 501] and sum(counts) == 1001


def test_reference_arm_prints_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "images/s" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] in ("reference", "port") and line["cpu_baseline"]["cores"] >= 1
    assert line["cpu_baseline"]["sample"].startswith(bench.CPU_PROGRAMS[line["cpu_baseline"]["kind"]])   # names what was timed
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["gpu_launches"] == 0


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=120, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_both_arms_describe_the_same_config():
    """The driver compares the two arms' `config`: the reference arm must print exactly what our arm prints."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=300)
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["config"] == bench.ours_config(4096, 1, False, 16)
    assert "sample" not in line["config"] and "sample" in line["cpu_baseline"]


def test_dump_outputs_writes_a_fixed_float32_sample(tmp_path):
    import numpy as np
    import torch
    feats = torch.randint(0, 256, (3000, 64, 16, 16), dtype=torch.uint8, generator=torch.Generator().manual_seed(5))
    idx = bench.dump_outputs(str(tmp_path / "a"), feats)
    got = np.load(tmp_path / "a" / "features.npy")
    assert got.dtype == np.float32 and got.shape == (bench.DUMP_IMAGES, 64, 16, 16) and got.nbytes <= 64 << 20
    assert np.all(np.diff(idx) > 0) and np.array_equal(got, feats.numpy()[idx])
    assert np.array_equal(bench.dump_outputs(str(tmp_path / "b"), feats), idx)           # the same images on every run
    bench.dump_outputs(str(tmp_path / "c"), feats[:100])                                  # a small batch is written whole
    assert np.array_equal(np.load(tmp_path / "c" / "features.npy"), feats[:100].numpy())


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]])
def test_bad_arguments_are_refused(argv):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + argv, capture_output=True, text=True, timeout=120)
    assert r.returncode == 2 and r.stdout == "" and argv[-2] in r.stderr


def test_roofline_traffic_comes_from_the_newest_committed_capture():
    per_image, name = bench.ncu_dram_bytes_per_image()
    assert name and name.endswith("_ncu_summary.txt") and os.path.exists(os.path.join(ROOT, "profiles", name))
    assert 16384 <= per_image <= 40000            # one image in, (up to) one feature map out
    rounds = [int(f[1:f.index("_")]) for f in os.listdir(os.path.join(ROOT, "profiles")) if f.endswith("_ncu_summary.txt") and f[1].isdigit()]
    assert name.startswith(f"r{max(rounds)}_") or per_image                        # newest round preferred


def _shared_worker(rank, world, port, path, n, q):
    import numpy as np
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    if rank == 0:
        bench.create_shared_predictions(path, n)
    dist.barrier()
    shm, cls, probs, bbox = bench.map_shared_predictions(path, n)
    lo, hi = bench.shard_range(n, rank, world)
    idx = np.arange(lo, hi)
    cls[lo:hi] = idx % 6                                   # what this rank's GPU would copy into its slice
    probs[lo:hi] = (idx[:, None] * 6 + np.arange(6)).astype(np.float32)
    bbox[lo:hi] = idx[:, None] * 4 + np.arange(4)
    shm.flush()
    dist.barrier()
    ok = None
    if rank == 0:                                          # rank 0 holds the gathered result without a collective
        all_idx = np.arange(n)
        ok = bool(np.array_equal(cls, all_idx % 6) and np.array_equal(bbox, all_idx[:, None] * 4 + np.arange(4)) and
                  np.array_equal(probs, (all_idx[:, None] * 6 + np.arange(6)).astype(np.float32)))
    q.put((rank, ok))
    dist.barrier()
    dist.destroy_process_group()


def test_two_ranks_fill_one_shared_prediction_array():
    """The gather of bench.py's stream_1m: every rank maps the same /dev/shm file and writes rows shard_range(...) of each
    prediction array; rank 0 then reads the whole job's predictions.  (On the GPU box the writes are the GPUs' D2H copies.)"""
    import torch.multiprocessing as tmp
    ctx = tmp.get_context("spawn")
    q = ctx.Queue()
    port = 31500 + os.getpid() % 2000
    n = 100_001
    path = f"/dev/shm/cnnacc_test_shared_{os.getpid()}.bin"
    procs = [ctx.Process(target=_shared_worker, args=(r, 2, port, path, n, q)) for r in range(2)]
    try:
        for p in procs:
            p.start()
        res = dict(q.get(timeout=120) for _ in procs)
        for p in procs:
            p.join(timeout=60)
            assert p.exitcode == 0
        assert res[0] is True and res[1] is None
        assert os.path.getsize(path) == n * bench.PRED_BYTES
    finally:
        if os.path.exists(path):
            os.unlink(path)
