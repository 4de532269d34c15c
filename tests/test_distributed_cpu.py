"""world_size-2 gloo tests (CPU) of the multi-GPU host logic: slab partition and
all-gather, convergence all-reduce, root-statistics merge."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from rl_agents_b200.distributed import shard_range, slab_sizes


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, fn, out):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        out[rank] = fn(rank, world)
    finally:
        dist.destroy_process_group()


def run_world(fn, world=2):
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_worker, args=(world, _free_port(), fn, out), nprocs=world, join=True)
    return [out[r] for r in range(world)]


def test_shard_range_is_a_partition():
    for n in (0, 1, 7, 100, 1001):
        for w in (1, 2, 3, 8):
            ranges = [shard_range(n, r, w) for r in range(w)]
            assert ranges[0][0] == 0 and ranges[-1][1] == n
            assert all(ranges[i][1] == ranges[i + 1][0] for i in range(w - 1))
            assert max(slab_sizes(n, w)) - min(slab_sizes(n, w)) <= 1


def _allgather_case(rank, world):
    from rl_agents_b200.distributed import allgather_slabs
    res = []
    for n in (10, 11):                      # equal and ragged slabs
        full = torch.full((n + 3,), -1.0, dtype=torch.float64)
        b, e = shard_range(n, rank, world)
        full[b:e] = torch.arange(b, e, dtype=torch.float64) * 10 + rank
        allgather_slabs(full, n)
        res.append(full.tolist())
    viol = torch.tensor([3 if rank == 0 else 0], dtype=torch.int32)
    dist.all_reduce(viol)
    res.append(int(viol.item()))
    return res


def test_allgather_slabs_and_violation_allreduce():
    out = run_world(_allgather_case)
    assert out[0] == out[1]
    for n, got in zip((10, 11), out[0][:2]):
        expect = []
        for r in range(2):
            b, e = shard_range(n, r, 2)
            expect += [i * 10.0 + r for i in range(b, e)]
        assert got[:n] == expect and got[n:] == [-1.0] * 3
    assert out[0][2] == 3


def _vi_slab_emulation(rank, world):
    """The DistributedVI loop with the sweep kernel replaced by the oracle's
    Bellman operator restricted to the rank's slab: the exchange logic is what is tested."""
    from oracle import envs as oenvs
    from oracle import planners
    from rl_agents_b200.distributed import allgather_slabs
    S, A, B, gamma, iters = 101, 3, 2, 0.9, 12
    P, N, R = oenvs.garnet(S, A, B, seed=3)
    term = np.zeros(S, bool)
    b, e = shard_range(S, rank, world)
    q = np.zeros((e - b, A))
    v = torch.zeros(S, dtype=torch.float64)
    for k in range(iters):
        nq = planners.bellman_expectation("sparse", P[b:e], R[b:e], term[b:e], v.numpy().copy(), gamma, nxt=N[b:e])
        viol = torch.tensor([int((~np.isclose(q, nq)).sum())], dtype=torch.int32)
        dist.all_reduce(viol)
        if int(viol.item()) == 0:
            break
        q = nq
        v[b:e] = torch.from_numpy(q.max(axis=-1))
        allgather_slabs(v, S)
    return q.tolist()


def test_slab_sharded_value_iteration_matches_single_process():
    from oracle import envs as oenvs
    from oracle import planners
    out = run_world(_vi_slab_emulation)
    P, N, R = oenvs.garnet(101, 3, 2, seed=3)
    q_ref, _ = planners.value_iteration("sparse", P, R, np.zeros(101, bool), 0.9, 12, nxt=N)
    assert np.array_equal(np.concatenate([np.array(o) for o in out]), q_ref)


def _too_few_states_case(rank, world):
    """n_states < world leaves the last rank an empty slab: every rank must raise before any allocation or
    collective, for both exchanges and for full or rank-local tables."""
    from oracle import envs as oenvs
    from rl_agents_b200.distributed import DistributedVI
    P, N, R = oenvs.garnet(1, 2, 2, seed=0)
    term = np.zeros(1, bool)
    b, e = shard_range(1, rank, world)
    out = []
    for exchange in ("nccl", "p2p"):
        for local in (False, True):
            tables = (P[b:e], R[b:e], term[b:e], N[b:e]) if local else (P, R, term, N)
            try:
                DistributedVI("sparse", *tables[:3], nxt=tables[3], gamma=0.9, device="cpu", exchange=exchange,
                              tables_are_local=local, n_states=1 if local else None)
                out.append(None)
            except ValueError as err:
                out.append(str(err))
    return out


def test_distributed_vi_rejects_fewer_states_than_ranks():
    out = run_world(_too_few_states_case)
    for msgs in out:
        assert len(msgs) == 4 and all(m is not None and "1 states cannot be split over 2 ranks" in m for m in msgs), msgs


def _merge_case(rank, world):
    from rl_agents_b200.distributed import merge_root_statistics
    counts = torch.tensor([[10, 0, 5], [2, 0, 13]][rank], dtype=torch.int32)
    values = torch.tensor([[1.0, 0.0, 2.0], [4.0, 0.0, 1.0]][rank], dtype=torch.float64)
    c, v = merge_root_statistics(counts, values)
    return c.tolist(), v.tolist()


def test_root_parallel_merge_and_recommendation():
    from rl_agents_b200.distributed import recommend
    out = run_world(_merge_case)
    assert out[0] == out[1]
    c, v = out[0]
    assert c == [12.0, 0.0, 18.0]
    assert v == pytest.approx([(10 * 1.0 + 2 * 4.0) / 12, 0.0, (5 * 2.0 + 13 * 1.0) / 18])
    assert recommend(c, v) == 2
    assert recommend([5, 5, 1], [0.1, 0.7, 9.0]) == 1


def _olop_merge_case(rank, world):
    from rl_agents_b200.distributed import merge_olop_root_statistics
    counts = torch.tensor([[4, 0, 6, 0], [5, 0, 3, 0]][rank], dtype=torch.int32)
    uppers = torch.tensor([[2.5, 9.0, 3.0, 9.0], [2.0, 9.0, 3.5, 9.0]][rank], dtype=torch.float64)
    c, u = merge_olop_root_statistics(counts, uppers)
    return c.tolist(), u.tolist()


def test_olop_root_parallel_merge_and_recommendation():
    from rl_agents_b200.distributed import recommend_olop
    out = run_world(_olop_merge_case)
    assert out[0] == out[1]
    c, u = out[0]
    assert c == [9.0, 0.0, 9.0, 0.0]
    assert u == [2.0, 9.0, 3.0, 9.0]          # tightest bound among the ranks that tried the action
    assert recommend_olop(c, u) == 2           # equal counts: larger value_upper (olop.py:126-130)
