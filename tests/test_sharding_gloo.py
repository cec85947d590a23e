"""CPU tier, world_size 2 over gloo: the N > 1 host logic (block sharding of independent streams + the optional
edge gather of packets).  Per-rank compute is the CPU oracle here; on GPUs it is the Context of that rank."""
import os
import sys

import numpy as np
import torch.multiprocessing as mp

from conftest import MODEL_DIR, ROOT
from lyra_b200 import sharding


def test_shard_ranges_cover_everything():
    for n, w in ((32768, 8), (4096, 1), (10, 4), (7, 8)):
        seen = []
        for r in range(w):
            first, cnt = sharding.shard_range(n, w, r)
            seen += list(range(first, first + cnt))
            for g in range(first, first + cnt):
                assert sharding.owner(g, n, w) == (r, g - first)
        assert seen == list(range(n))


def _worker(rank, world, port, n, out_path):
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    from oracle import oracle as O
    dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%d" % port, rank=rank, world_size=world)
    first, cnt = sharding.shard_range(n, world, rank)
    rng = np.random.default_rng(123)
    pcm = rng.integers(-8192, 8192, size=(2, n, 320), dtype=np.int16)      # same on every rank
    codecs = [O.Codec(MODEL_DIR) for _ in range(cnt)]
    gathered = []
    for f in range(2):
        local = np.stack([np.frombuffer(codecs[k].encode(pcm[f, first + k], 64)[0], dtype=np.uint8) for k in range(cnt)])
        gathered.append(sharding.gather_packets(local, n))
    if rank == 0:
        np.save(out_path, np.stack(gathered))
    dist.barrier()
    dist.destroy_process_group()


def test_two_rank_sharded_encode_matches_single_process(tmp_path, oracle):
    n, world, port = 5, 2, 29500 + (os.getpid() % 2000)
    out = str(tmp_path / "gathered.npy")
    mp.spawn(_worker, args=(world, port, n, out), nprocs=world, join=True)
    got = np.load(out)
    rng = np.random.default_rng(123)
    pcm = rng.integers(-8192, 8192, size=(2, n, 320), dtype=np.int16)
    codecs = [oracle.Codec(MODEL_DIR) for _ in range(n)]
    for f in range(2):
        for k in range(n):
            assert bytes(got[f, k]) == codecs[k].encode(pcm[f, k], 64)[0]


def test_bench_rank_core_slices_are_disjoint():
    # bench.py: under torchrun every rank keeps its host threads on its own slice of the allowed cores (host-buffer pass);
    # run in subprocesses because the call changes the process's affinity mask
    import json
    import subprocess
    code = ("import json, os, sys; sys.path.insert(0, %r); import bench; base = sorted(os.sched_getaffinity(0)); "
            "r = bench.pin_rank_cores(int(sys.argv[1]), int(sys.argv[2])); "
            "print(json.dumps({'ret': r, 'base': base, 'now': sorted(os.sched_getaffinity(0)), 'cores': bench.host_cores()}))" % ROOT)
    outs = [json.loads(subprocess.check_output([sys.executable, "-c", code, str(r), "2"]).decode().strip().splitlines()[-1]) for r in range(2)]
    base = outs[0]["base"]
    if len(base) < 4:
        assert outs[0]["ret"] is None and outs[0]["now"] == base      # too few cores to slice: left alone
        return
    a, b = set(outs[0]["now"]), set(outs[1]["now"])
    assert a and b and not (a & b) and (a | b) <= set(base)
    assert outs[0]["ret"] == len(a) == len(base) // 2 and outs[0]["cores"] <= len(a)
    single = json.loads(subprocess.check_output([sys.executable, "-c", code, "0", "1"]).decode().strip().splitlines()[-1])
    assert single["ret"] is None and single["now"] == single["base"]


def test_bench_host_pass_groups():
    """bench.py picks the host-buffer pass's worker groups from the workload and the host cores of the rank."""
    import sys
    sys.path.insert(0, ROOT)
    import bench
    assert bench.host_pass_groups(0, False, 1, 16, 4096) == 4        # one GPU, 16 logical cores: the measured configuration
    assert bench.host_pass_groups(0, False, 1, 12, 4096) == 2        # a 12-thread slice of an 8-GPU box: two groups
    assert bench.host_pass_groups(0, False, 1, 24, 4096) == 4        # a 24-thread slice (4 ranks on that box)
    assert bench.host_pass_groups(0, False, 2, 16, 4096) == 2        # two unpinned ranks sharing 16 cores
    assert bench.host_pass_groups(0, True, 1, 64, 4096) == 2         # decoder-only workloads: fewer, larger calls
    assert bench.host_pass_groups(3, False, 1, 64, 4096) == 2        # an explicit request is reduced to a divisor of the stream count
    assert bench.host_pass_groups(3, False, 1, 64, 3072) == 3
    assert bench.host_pass_priorities(4, 120, False) == (0, 0)       # four groups: equal priorities at every bit rate
    assert bench.host_pass_priorities(2, 64, False) == (0, 0)
    assert bench.host_pass_priorities(2, 120, False) == (-1, 0)      # two groups, long RVQ chains: encoder first
    assert bench.host_pass_priorities(2, 184, True) == (0, 0)        # decoder-only workload


def test_bench_dump_outputs(tmp_path, monkeypatch):
    """bench.py --dump-outputs: float32 .npy files, every stream while they fit the budget, else the same seeded rows of each."""
    sys.path.insert(0, ROOT)
    import bench
    n = 1000
    pcm = np.arange(n * 320, dtype=np.int64).reshape(n, 320).astype(np.int16)
    outputs = {"pcm": pcm, "packets": (np.arange(n * 8) % 256).astype(np.uint8).reshape(n, 8)}
    rows = bench.write_outputs(str(tmp_path / "all"), outputs)
    assert rows.tolist() == list(range(n))
    for name, a in outputs.items():
        got = np.load(str(tmp_path / "all" / (name + ".npy")))
        assert got.dtype == np.float32 and np.array_equal(got, a.astype(np.float32))
    monkeypatch.setattr(bench, "DUMP_MAX_BYTES", 100 * (320 + 8) * 4)
    rows = bench.write_outputs(str(tmp_path / "a"), outputs)
    assert len(rows) == 100 and (np.diff(rows) > 0).all()
    assert np.array_equal(rows, bench.write_outputs(str(tmp_path / "b"), outputs))
    total = 0
    for name, a in outputs.items():
        got = np.load(str(tmp_path / "a" / (name + ".npy")))
        assert np.array_equal(got, a[rows].astype(np.float32))
        assert np.array_equal(got, np.load(str(tmp_path / "b" / (name + ".npy"))))
        total += got.nbytes
    assert total <= bench.DUMP_MAX_BYTES
