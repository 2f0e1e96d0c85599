"""N > 1 host logic on CPU: the read-sharding rule against the reference's own thread split, and the sharded
E-step + allreduce + M-step flow over torch.distributed (gloo, world_size 2) against the single-process oracle.
The oracle stands in for the CUDA kernel here (tests only); the collective and the sharding are the real code."""
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import ref_golden
import rsem_files as rf
import synth
import rsem_b200


def shard_reads(row_ptr, n):
    """the library's rule (rsem_b200_shard_reads, host arithmetic: no GPU needed) - the one rsem-run-em and bench.py use"""
    return rsem_b200.load_library().shard_reads(row_ptr, n)


def slice_csr(row_ptr, first, last):
    row_ptr = np.asarray(row_ptr, dtype=np.uint64)
    h0, h1 = int(row_ptr[first]), int(row_ptr[last])
    return (row_ptr[first:last + 1] - np.uint64(h0)).astype(np.uint64), h0, h1


@pytest.mark.parametrize("threads", [2, 3, 7])
def test_shards_equal_reference_thread_split(tmp_path, built, threads):
    """the reference's rsem-run-em -p threads prints its split ("Thread t : N = .., NHit = .."): stored in
    tests/golden/ref_outputs.json.gz (tools/make_golden_ref.py)"""
    d = rf.gen_dataset(str(tmp_path / "d"), read_type=0, M=80, N1=900, N0=40, read_len=40, maxL=100, seed=threads)
    ref = [(int(a), int(b)) for a, b in ref_golden.Run(f"sharding/{threads}")["split"].reshape(-1, 2)]
    assert len(ref) == threads
    row_ptr, _, _, _ = rf.read_dat(f"{d}/s.temp/s.dat", False)
    mine = [(b - a, int(row_ptr[b] - row_ptr[a])) for a, b in shard_reads(row_ptr, threads)]
    assert mine == ref


def test_shards_edge_cases():
    rp = np.array([0, 3, 3, 10, 11], np.uint64)
    assert shard_reads(rp, 1) == [(0, 4)]
    parts = shard_reads(rp, 4)
    assert [b - a for a, b in parts] == [1, 1, 1, 1]
    parts = shard_reads(rp, 9)  # more shards than reads: the surplus shards are empty (the reference clamps, EM.cpp:640)
    assert parts[:4] == shard_reads(rp, 4) and all(p == (4, 4) for p in parts[4:])
    # a heavy first read: the first shard stops right after it, the middle shard takes reads until one is left for the last
    rp = np.array([0, 100, 101, 102, 103], np.uint64)
    assert shard_reads(rp, 3) == [(0, 1), (1, 3), (3, 4)]


def _worker(rank, world, port, tmp):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import oracle_binding
    orc = oracle_binding.Oracle()
    N, M = 6000, 400
    row_ptr, sid, conprb, ncpv = synth.random_matrix(N, M, 6, seed=77)
    n0 = 300.0
    theta = synth.init_theta(M, n0, N + n0)
    a, b = shard_reads(row_ptr, world)[rank]
    rp, h0, h1 = slice_csr(row_ptr, a, b)
    for _ in range(4):
        counts = orc.estep(rp, sid[h0:h1], conprb[h0:h1], ncpv[a:b], theta)       # local K2
        t = torch.from_numpy(counts)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)                                      # the one collective per round
        c = t.numpy().copy()
        c[0] += n0                                                                    # N0 added once, after the reduce
        theta = c / c.sum()                                                           # K4 on every rank
    np.save(os.path.join(tmp, f"theta{rank}.npy"), theta)
    dist.destroy_process_group()


def test_two_rank_em_equals_single_process(tmp_path, oracle):
    port = 29500 + (os.getpid() % 2000)
    mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    t0, t1 = np.load(tmp_path / "theta0.npy"), np.load(tmp_path / "theta1.npy")
    assert np.array_equal(t0, t1)  # every rank holds the same theta (no broadcast needed)
    row_ptr, sid, conprb, ncpv = synth.random_matrix(6000, 400, 6, seed=77)
    ref, _, _ = oracle.em_rounds(row_ptr, sid, conprb, ncpv, synth.init_theta(400, 300.0, 6300.0), 300.0, 1, 4, 20, 100)
    assert np.allclose(t0, ref, rtol=1e-12, atol=1e-18)
