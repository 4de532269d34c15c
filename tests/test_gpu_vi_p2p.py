"""The value-iteration sweep with the exchange step fused in (b2_vi_sweep_p2p) against numpy, on one GPU.

Several ranks are emulated in one process: every rank gets its own V ping-pong pair, arrival flags, violation table
and scratch as ordinary device tensors, and the b2_vi_p2p of every rank carries the same pointer tables to all of
them.  Sweep k of every rank is enqueued on one stream before any sweep k + 1, so every flag a kernel acquires was
published by a launch that has already retired: no kernel ever waits."""
import re

import numpy as np
import pytest

from oracle import envs as oenvs
from oracle import planners
from rl_agents_b200.distributed import shard_range

pytestmark = pytest.mark.gpu

SENTINEL = -1.0          # V >= 0 for the garnet rewards in [0, 1): no sweep can produce it


def make_mdp(mode, S, A, B, term, seed):
    """(transition, reward, terminal, nxt) of a seeded garnet MDP; `term` is 'none', 'some' or 'all'."""
    if mode == "sparse":
        P, N, R = oenvs.garnet(S, A, B, seed=seed)
    else:
        P, R = oenvs.garnet(S, A, 1, seed=seed, deterministic=True)
        N = None
    terminal = {"none": np.zeros(S, bool), "all": np.ones(S, bool),
                "some": np.random.default_rng(seed).uniform(size=S) < 0.1}[term]
    return P, R, terminal, N


def oracle_iterates(mode, P, R, terminal, N, gamma, T, bounds):
    """The fixed-point loop of planners.value_iteration without its early exit: Q_k and V_k = max_a Q_k for
    k = 0..T, and viol[k, j], the elements of slab j where np.isclose(Q_k, Q_{k+1}) fails."""
    qs, vs = [np.zeros(R.shape)], [np.zeros(R.shape[0])]
    viol = np.zeros((T, len(bounds)), np.int64)
    for k in range(T):
        nq = planners.bellman_expectation(mode, P, R, terminal, vs[k], gamma, nxt=N)
        bad = ~np.isclose(qs[k], nq)
        viol[k] = [bad[b:e].sum() for b, e in bounds]
        qs.append(nq)
        vs.append(nq.max(axis=-1))
    return qs, vs, viol


class EmulatedRanks(object):
    """`world` ranks of the peer-memory exchange on one device.  Rank r owns the rows shard_range(S, r, world)
    through its own VIEngine (tables, problem struct, Q ping-pong pair) and the device tensors a rank of
    DistributedVI keeps in its peer buffer: v [2, S], flags [world], parts [T, world], viol_local [T], done [T],
    status [1]."""

    def __init__(self, mode, P, R, terminal, N, gamma, world, T):
        import torch
        from rl_agents_b200 import _lib
        from rl_agents_b200.engine.vi import VIEngine
        self.torch, self._lib, self.lib = torch, _lib, _lib.load()
        S = R.shape[0]
        self.world, self.T = world, T
        self.bounds = [shard_range(S, r, world) for r in range(world)]
        self.engines = [VIEngine(mode, P[b:e], R[b:e], terminal[b:e], nxt=None if N is None else N[b:e], gamma=gamma,
                                 row_begin=b, row_end=e, n_states=S) for b, e in self.bounds]

        def zeros(shape, dtype=torch.int32):
            return [torch.zeros(shape, dtype=dtype, device="cuda") for _ in range(world)]
        self.v = zeros((2, S), torch.float64)
        self.flags, self.parts = zeros(world), zeros((T, world))
        self.viol, self.done, self.status = zeros(T), zeros(T), zeros(1)
        self.x = []
        for r in range(world):
            x = _lib.VIP2P()
            x.world, x.rank = world, r
            for j in range(world):
                x.v[0][j], x.v[1][j] = self.v[j][0].data_ptr(), self.v[j][1].data_ptr()
                x.flags[j], x.parts[j] = self.flags[j].data_ptr(), self.parts[j].data_ptr()
            x.viol_local, x.done, x.status = self.viol[r].data_ptr(), self.done[r].data_ptr(), self.status[r].data_ptr()
            self.x.append(x)

    def reset(self):
        for t in self.v + self.flags + self.parts + self.viol + self.done + self.status:
            t.zero_()
        for e in self.engines:
            for q in e.q:
                q.zero_()

    def sweep(self, r, k):
        e, _lib = self.engines[r], self._lib
        _lib.check(self.lib.b2_vi_sweep_p2p(e.problem, self.x[r], _lib.ptr(e.q[k & 1]), _lib.ptr(e.q[(k + 1) & 1]), k,
                                            _lib.current_stream()))

    def result(self, r):
        """Rank r's answer, selected as DistributedVI._solve_p2p does: the first sweep whose violation row sums to
        zero converged and its OLD iterate is returned."""
        zero = np.nonzero(self.parts[r].cpu().numpy().sum(axis=1) == 0)[0]
        k = int(zero[0]) if zero.size else None
        if k is None:
            return self.engines[r].q[self.T & 1], self.T
        return self.engines[r].q[k & 1], k + 1

    def grid(self, r):
        """The launch b2_vi_sweep_p2p makes: one CTA per 256 (s, a) elements, at most 8 CTAs per SM."""
        b, e = self.bounds[r]
        n_sa = (e - b) * self.engines[r].n_actions
        sms = self.torch.cuda.get_device_properties(self.torch.cuda.current_device()).multi_processor_count
        return min((n_sa + 255) // 256, 8 * sms)


def run_sweeps(em, rng, qs=None, vs=None, kc=None):
    """Enqueue T sweeps of every rank, all ranks' sweep k (in a random rank order) before any sweep k + 1.
    With the oracle's iterates: synchronise after every sweep, check every rank's Q slab and every rank's copy of
    the whole V, and once the converged sweep kc has run, fill V with SENTINEL, which later sweeps must not touch."""
    for k in range(em.T):
        for r in rng.permutation(em.world):
            em.sweep(int(r), k)
        if vs is None or (kc is not None and k > kc):
            continue
        for j, (b, e) in enumerate(em.bounds):
            assert np.array_equal(em.engines[j].q[(k + 1) & 1].cpu().numpy(), qs[k + 1][b:e]), (k, j)
            assert np.array_equal(em.v[j][(k + 1) & 1].cpu().numpy(), vs[k + 1]), (k, j)
        if k == kc:
            for v in em.v:
                v.fill_(SENTINEL)


def check_solve(em, qs, vs, viol, kc, synced):
    """Values, the protocol state and the V buffers after the T sweeps of run_sweeps."""
    T, world = em.T, em.world
    expect_q, expect_sweeps = (qs[T], T) if kc is None else (qs[kc], kc + 1)
    expect_parts = viol.copy()
    if kc is not None:
        expect_parts[kc + 1:] = 0              # converged launches publish 0 and compute nothing
    for r, (b, e) in enumerate(em.bounds):
        q, sweeps = em.result(r)
        assert sweeps == expect_sweeps, r
        assert np.array_equal(q.cpu().numpy(), expect_q[b:e]), r
        assert np.array_equal(em.parts[r].cpu().numpy(), expect_parts), r
        assert np.array_equal(em.viol[r].cpu().numpy(), expect_parts[:, r]), r
        assert (em.flags[r].cpu().numpy() == T).all(), r
        assert (em.done[r].cpu().numpy() == em.grid(r)).all(), r
        assert int(em.status[r].item()) == 0, r
        v = em.v[r].cpu().numpy()
        if synced and kc is not None:
            assert (v == SENTINEL).all(), r     # nothing stored V after the converged sweep
        else:
            K = T if kc is None else kc + 1     # last V computed; the converged launches leave both buffers alone
            assert np.array_equal(v[K & 1], vs[K]) and np.array_equal(v[(K - 1) & 1], vs[K - 1]), r


P2P_CASES = {
    # id: mode, S, A, B, world, gamma, sweeps (None: end exactly at the converged sweep), terminal, sync each sweep
    "sparse_ragged_w3": ("sparse", 1001, 8, 4, 3, 0.5, 40, "some", True),       # rows*A 2672 / 2664
    "det_w5": ("deterministic", 777, 4, 1, 5, 0.5, 40, "none", True),
    "sparse_tiny_slabs_w8": ("sparse", 13, 2, 2, 8, 0.99, 6, "some", True),     # 2-4 (s, a) elements per rank
    "sparse_b8_a16_w2_last": ("sparse", 300, 16, 8, 2, 0.5, None, "some", False),
    "det_a32_w3": ("deterministic", 50, 32, 1, 3, 0.99, 5, "some", False),
    "sparse_a1_b1_w5_all_terminal": ("sparse", 4099, 1, 1, 5, 0.5, 10, "all", False),
    "sparse_a32_w1": ("sparse", 2000, 32, 2, 1, 0.5, 50, "none", False),
    "det_w8_all_terminal": ("deterministic", 123, 2, 1, 8, 0.5, 30, "all", False),
    "sparse_b8_w2": ("sparse", 999, 4, 8, 2, 0.99, 8, "none", False),
    "det_a16_w2_last": ("deterministic", 4097, 16, 1, 2, 0.5, None, "some", True),
    # C4 shape: 125 000 rows x 8 actions per rank, more elements than one grid-stride pass of the capped grid
    "c4_w8": ("sparse", 1_000_000, 8, 4, 8, 0.95, 3, "none", True),
}


@pytest.mark.parametrize("key", list(P2P_CASES))
def test_p2p_sweep_emulated_ranks_vs_numpy(key):
    mode, S, A, B, world, gamma, T, term, sync = P2P_CASES[key]
    P, R, terminal, N = make_mdp(mode, S, A, B, term, seed=S)
    bounds = [shard_range(S, r, world) for r in range(world)]
    qs, vs, viol = oracle_iterates(mode, P, R, terminal, N, gamma, T or 60, bounds)
    zero = np.nonzero(viol.sum(axis=1) == 0)[0]
    kc = int(zero[0]) if zero.size else None
    if T is None:
        T = kc + 1                              # the converged sweep is the last one enqueued
        viol = viol[:T]
    elif kc is not None and kc >= T:
        kc = None
    assert (kc is None) == (gamma > 0.9), "gamma 0.5 converges early, 0.95 / 0.99 never within T sweeps"
    q_ref, sweeps_ref = planners.value_iteration(mode, P, R, terminal, gamma, T, nxt=N)
    assert sweeps_ref == (T if kc is None else kc + 1)
    assert np.array_equal(q_ref, qs[T] if kc is None else qs[kc])

    em = EmulatedRanks(mode, P, R, terminal, N, gamma, world, T)
    rng = np.random.default_rng(S)
    if sync:
        run_sweeps(em, rng, qs, vs, kc)
    else:
        run_sweeps(em, rng)
    check_solve(em, qs, vs, viol, kc, sync)
    # the same buffers, zeroed, solve again (with other rank orders)
    em.reset()
    run_sweeps(em, rng)
    check_solve(em, qs, vs, viol, kc, False)


def test_p2p_sweep_rejects_unsupported_arguments():
    """Every rejection returns an error code with a message and launches nothing (sweep 0 everywhere: a launch
    that slipped through would not wait on any flag, and would leave its mark in done / flags / V / Q)."""
    import torch
    from rl_agents_b200 import _lib
    from rl_agents_b200.engine.vi import VIEngine
    lib = _lib.load()
    S = 64
    P, R, terminal, N = make_mdp("sparse", S, 4, 4, "some", 1)
    em = EmulatedRanks("sparse", P, R, terminal, N, 0.9, 2, 1)
    e = em.engines[0]
    b, end = em.bounds[0]

    def engine(mode, A, B):
        if mode == "stochastic":
            rng = np.random.default_rng(A)
            Pd = rng.uniform(size=(S, A, S))
            return VIEngine(mode, Pd[b:end], rng.uniform(size=(S, A))[b:end], terminal[b:end], gamma=0.9,
                            row_begin=b, row_end=end, n_states=S)
        P2, R2, t2, N2 = make_mdp(mode, S, A, B, "some", 2)
        return VIEngine(mode, P2[b:end], R2[b:end], t2[b:end], nxt=None if N2 is None else N2[b:end], gamma=0.9,
                        row_begin=b, row_end=end, n_states=S)

    def rejected(match, eng=e, problem=None, x=None):
        rc = lib.b2_vi_sweep_p2p(eng.problem if problem is None else problem, em.x[0] if x is None else x,
                                 _lib.ptr(eng.q[0]), _lib.ptr(eng.q[1]), 0, _lib.current_stream())
        msg = lib.b2_last_error().decode()
        assert rc != 0 and re.search(match, msg), (match, rc, msg)

    for mode, A, B in [("deterministic", 3, 1), ("deterministic", 64, 1), ("sparse", 4, 3), ("sparse", 4, 16)]:
        rejected("A a power of two <= 32 and B in", engine(mode, A, B))
    rejected("sparse or deterministic mode", engine("stochastic", 4, S))
    p = _lib.VIProblem.from_buffer_copy(e.problem)
    p.next += 4
    rejected("A a power of two <= 32 and B in", problem=p)
    for world, rank in [(0, 0), (9, 0), (2, 2)]:
        x = _lib.VIP2P.from_buffer_copy(em.x[0])
        x.world, x.rank = world, rank
        rejected("bad world / rank", x=x)
    for field in ("v0", "v1", "flags", "parts"):
        x = _lib.VIP2P.from_buffer_copy(em.x[0])
        if field == "v0":
            x.v[0][1] = None
        elif field == "v1":
            x.v[1][1] = None
        else:
            getattr(x, field)[1] = None
        rejected("peer pointer missing", x=x)
    p = _lib.VIProblem.from_buffer_copy(e.problem)
    p.row_end = p.row_begin
    rejected("bad shape", problem=p)
    # the slab DistributedVI would give the last rank when n_states < world: empty tables, null pointers
    empty = VIEngine("sparse", P[S:], R[S:], terminal[S:], nxt=N[S:], gamma=0.9, row_begin=S, row_end=S, n_states=S)
    rejected("null pointer|tables missing|bad shape", empty)
    torch.cuda.synchronize()
    for t in em.v + em.flags + em.parts + em.viol + em.done + em.status + e.q:
        assert not bool(t.any())


@pytest.mark.parametrize("mode", ["sparse", "deterministic"])
def test_distributed_vi_p2p_on_a_single_rank_group(mode, tmp_path):
    """DistributedVI's p2p path end to end in a one-rank gloo group: the peer buffer, its offsets, the memset
    between solves, the status read and the result selection."""
    import torch.distributed as dist
    from rl_agents_b200.distributed import DistributedVI
    S, A, B, gamma, T = 3000, 8, 4, 0.6, 60
    P, R, terminal, N = make_mdp(mode, S, A, B, "some", 7)
    q_ref, sweeps_ref = planners.value_iteration(mode, P, R, terminal, gamma, T, nxt=N)
    assert sweeps_ref < T
    v_last = planners.bellman_expectation(mode, P, R, terminal, q_ref.max(axis=-1), gamma, nxt=N).max(axis=-1)
    assert not dist.is_initialized()
    dist.init_process_group("gloo", store=dist.FileStore(str(tmp_path / "store"), 1), rank=0, world_size=1)
    try:
        dvi = DistributedVI(mode, P, R, terminal, nxt=N, gamma=gamma, exchange="p2p", max_iterations=64)
        try:
            for _ in range(2):
                q, sweeps = dvi.solve(T)
                assert sweeps == sweeps_ref
                assert np.array_equal(q.cpu().numpy(), q_ref)
                assert np.array_equal(dvi.v_slab(sweeps), v_last)
        finally:
            dvi.close()
    finally:
        dist.destroy_process_group()
