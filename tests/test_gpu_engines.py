"""GPU parity tests: the CUDA engines (through the C ABI) against the oracle and
the golden vectors made by the unmodified reference.  Bit-exact: node order,
counts, fp64 bounds / values, fp32 env states."""
import numpy as np
import pytest

from oracle import envs as oenvs
from oracle import planners
from tests.util import assert_tree_matches, load_golden, load_mdps

pytestmark = pytest.mark.gpu

G = load_golden("golden_finite.json")
H = load_golden("golden_highway.json")
M = load_mdps()


def np_random(seed):
    return np.random.Generator(np.random.PCG64(np.random.SeedSequence(seed)))


def product_mdp(name="large1", terminal=None):
    from rl_agents_b200.envs.finite_mdp import FiniteMDP
    term = M[name + "_term"] if terminal is None else terminal
    return FiniteMDP("deterministic", M[name + "_T"], M[name + "_R"], term)


def terminal_variant():
    term = M["large1_term"].copy()
    term[[3, 17, 66, 91]] = True
    return term


# ------------------------------------------------------------------ env ----
def test_highway_step_matches_golden_traces():
    import torch
    from rl_agents_b200 import _lib
    lib = _lib.load()
    dev = torch.device("cuda")
    for seed, steps in H["traces"].items():
        st = torch.tensor(H["states"][seed] if seed in H["states"] else oenvs.make_highway_state(int(seed)).pack(),
                          dtype=torch.int32, device=dev).reshape(1, -1).contiguous()
        rew = torch.empty(1, dtype=torch.float32, device=dev)
        flg = torch.empty(1, dtype=torch.int32, device=dev)
        avail = torch.empty(1, dtype=torch.int32, device=dev)
        for k, s in enumerate(steps):
            act = torch.tensor([s["a"]], dtype=torch.int32, device=dev)
            _lib.check(lib.b2_highway_step(_lib.ptr(st), _lib.ptr(act), _lib.ptr(rew), _lib.ptr(flg), _lib.ptr(avail), 1,
                                           _lib.current_stream()))
            assert st.cpu().numpy().reshape(-1).tolist() == s["state"], (seed, k)
            assert float(rew.item()) == np.float32(s["r"])
            assert int(flg.item()) == (1 if s["term"] else 0) | (2 if s["trunc"] else 0)
            if k + 1 < len(steps):
                mask = int(avail.item())
                assert sorted(a for a in range(5) if mask >> a & 1) == sorted(steps[k + 1]["avail"])


def test_highway_step_batched_vs_oracle_random():
    import torch
    from rl_agents_b200 import _lib
    from rl_agents_b200.envs.highway_lite import make_scene
    lib = _lib.load()
    dev = torch.device("cuda")
    n = 37   # odd: exercises the idle half-warp
    scenes = [oenvs.HighwayLite(seed=100 + i) for i in range(n)]
    for i in range(n):   # product and oracle scene generators agree
        assert make_scene(100 + i).tolist() == scenes[i].state.pack().tolist()
    st = torch.tensor(np.stack([e.state.pack() for e in scenes]), dtype=torch.int32, device=dev)
    rng = np.random.default_rng(0)
    rew = torch.empty(n, dtype=torch.float32, device=dev)
    flg = torch.empty(n, dtype=torch.int32, device=dev)
    for step in range(6):
        acts = []
        for e in scenes:
            av = e.get_available_actions()
            acts.append(int(av[rng.integers(len(av))]))
        act = torch.tensor(acts, dtype=torch.int32, device=dev)
        _lib.check(lib.b2_highway_step(_lib.ptr(st), _lib.ptr(act), _lib.ptr(rew), _lib.ptr(flg), None, n,
                                       _lib.current_stream()))
        got = st.cpu().numpy()
        for i, e in enumerate(scenes):
            _, r, term, trunc, _ = e.step(acts[i])
            assert got[i].tolist() == e.state.pack().tolist(), (step, i)
            assert float(rew[i].item()) == np.float32(r)
            assert int(flg[i].item()) == (1 if term else 0) | (2 if trunc else 0)


def test_highway_step_exact_x_ties_take_the_scan_path():
    """Two (or more) vehicles with exactly equal x cannot be ordered by the rank structure: the kernel
    falls back to the literal scan of the spec (tie rules by slot index).  Also crashed and absent slots."""
    import torch
    from rl_agents_b200 import _lib
    lib = _lib.load()
    dev = torch.device("cuda")
    scenes = []
    for seed in range(60, 72):
        st = oenvs.make_highway_state(seed)
        st.x[5] = st.x[3]                      # exact tie, usually on different lanes
        st.x[9] = st.x[3]
        if seed % 3 == 0:
            st.y[5] = st.y[3]                  # same lane too: overlapping boxes -> crash at once
        if seed % 4 == 0:
            st.flags[11] = 0                   # an absent slot
            st.flags[12] = 3                   # a vehicle that is already crashed
        scenes.append(oenvs.HighwayLite(st))
    n = len(scenes)
    st = torch.tensor(np.stack([e.state.pack() for e in scenes]), dtype=torch.int32, device=dev)
    rew = torch.empty(n, dtype=torch.float32, device=dev)
    flg = torch.empty(n, dtype=torch.int32, device=dev)
    for step in range(5):
        acts = [int(e.get_available_actions()[step % len(e.get_available_actions())]) for e in scenes]
        _lib.check(lib.b2_highway_step(_lib.ptr(st), _lib.ptr(torch.tensor(acts, dtype=torch.int32, device=dev)),
                                       _lib.ptr(rew), _lib.ptr(flg), None, n, _lib.current_stream()))
        got = st.cpu().numpy()
        for i, e in enumerate(scenes):
            _, r, term, trunc, _ = e.step(acts[i])
            assert got[i].tolist() == e.state.pack().tolist(), (step, i)
            assert float(rew[i].item()) == np.float32(r) and int(flg[i].item()) == (1 if term else 0) | (2 if trunc else 0)


def test_highway_step_long_random_sweep_vs_oracle():
    """200 scenes x 10 random decisions (30 000 physics sub-steps per implementation), bit for bit."""
    import torch
    from rl_agents_b200 import _lib
    lib = _lib.load()
    dev = torch.device("cuda")
    n = 200
    scenes = [oenvs.HighwayLite(seed=1000 + i) for i in range(n)]
    st = torch.tensor(np.stack([e.state.pack() for e in scenes]), dtype=torch.int32, device=dev)
    rew = torch.empty(n, dtype=torch.float32, device=dev)
    flg = torch.empty(n, dtype=torch.int32, device=dev)
    rng = np.random.default_rng(5)
    for step in range(10):
        acts = [int(rng.choice(e.get_available_actions())) for e in scenes]
        _lib.check(lib.b2_highway_step(_lib.ptr(st), _lib.ptr(torch.tensor(acts, dtype=torch.int32, device=dev)),
                                       _lib.ptr(rew), _lib.ptr(flg), None, n, _lib.current_stream()))
        got, r_got, f_got = st.cpu().numpy(), rew.cpu().numpy(), flg.cpu().numpy()
        for i, e in enumerate(scenes):
            _, r, term, trunc, _ = e.step(acts[i])
            assert np.array_equal(got[i], e.state.pack()), (step, i)
            assert r_got[i] == np.float32(r) and f_got[i] == (1 if term else 0) | (2 if trunc else 0)


# ------------------------------------------------------------------- VI ----
def vi_cases():
    rng = np.random.default_rng(0)
    P = rng.uniform(size=(100, 4, 100))
    P /= P.sum(-1, keepdims=True)
    R = rng.uniform(size=(100, 4))
    Ps, Ns, Rs = oenvs.garnet(500, 4, 3, seed=1)
    term = np.zeros(500, bool)
    term[::37] = True
    return {
        "large1_g0.9_it100": ("deterministic", M["large1_T"], M["large1_R"], M["large1_term"], None),
        "large1_g1.0_it2": ("deterministic", M["large1_T"], M["large1_R"], M["large1_term"], None),
        "trap_g0.9_it100": ("deterministic", M["trap_T"], M["trap_R"], M["trap_term"], None),
        "loop_g0.9_it100": ("deterministic", M["loop_T"], M["loop_R"], M["loop_term"], None),
        "dense_c1_g0.95_it100": ("stochastic", P, R, np.zeros(100, bool), None),
        "sparse_garnet500_g0.95_it100": ("sparse", Ps, Rs, term, Ns),
    }


@pytest.mark.parametrize("key", sorted(vi_cases()))
def test_vi_golden(key):
    from rl_agents_b200.engine.vi import VIEngine
    mode, T, R, term, N = vi_cases()[key]
    g = G["vi"][key]
    eng = VIEngine(mode, T, R, term, nxt=N, gamma=g["gamma"])
    q, sweeps = eng.solve(g["iterations"])
    assert np.array_equal(q.cpu().numpy(), np.array(g["q"])), key
    _, ref_sweeps = planners.value_iteration(mode, T if mode != "deterministic" else np.asarray(T), R,
                                             term.astype(bool), g["gamma"], g["iterations"], nxt=N)
    assert sweeps == ref_sweeps


@pytest.mark.parametrize("S,A,B,seed", [(1000, 8, 1, 0), (777, 3, 2, 1), (5000, 8, 4, 2), (300, 5, 7, 3),
                                        (257, 2, 8, 4), (200, 4, 19, 5), (64, 3, 130, 6), (1, 1, 1, 7)])
def test_vi_sparse_random_vs_oracle(S, A, B, seed):
    from rl_agents_b200.engine.vi import VIEngine
    P, N, R = oenvs.garnet(S, A, B, seed=seed)
    term = np.random.default_rng(seed).uniform(size=S) < 0.05
    q_ref, sweeps_ref = planners.value_iteration("sparse", P, R, term, 0.93, 60, nxt=N)
    eng = VIEngine("sparse", P, R, term, nxt=N, gamma=0.93)
    q, sweeps = eng.solve(60)
    assert sweeps == sweeps_ref
    assert np.array_equal(q.cpu().numpy(), q_ref)


@pytest.mark.parametrize("mode,S,A,B,seed", [("sparse", 4096, 8, 4, 0), ("sparse", 1600, 8, 4, 1), ("sparse", 6400, 4, 2, 2),
                                             ("sparse", 2048, 3, 9, 3), ("deterministic", 2048, 4, 1, 4),
                                             ("deterministic", 5120, 8, 1, 5), ("sparse", 3200, 8, 8, 6)])
@pytest.mark.parametrize("kernel", [0, 1, 2])
def test_vi_kernel_variants_vs_oracle(mode, S, A, B, seed, kernel):
    """The three sweep kernels (0: register rows when the shape allows, 1: tiled, 2: TMA-staged
    tiles with a ragged last tile) all stay bit-identical with numpy."""
    from rl_agents_b200.engine.vi import VIEngine
    term = np.random.default_rng(seed).uniform(size=S) < 0.03
    if mode == "sparse":
        P, N, R = oenvs.garnet(S, A, B, seed=seed)
        q_ref, sweeps_ref = planners.value_iteration("sparse", P, R, term, 0.9, 25, nxt=N)
        eng = VIEngine("sparse", P, R, term, nxt=N, gamma=0.9)
    else:
        T, R = oenvs.garnet(S, A, 1, seed=seed, deterministic=True)
        q_ref, sweeps_ref = planners.value_iteration("deterministic", T, R, term, 0.9, 25)
        eng = VIEngine("deterministic", T, R, term, gamma=0.9)
    eng.problem.reserved = kernel
    q, sweeps = eng.solve(25)
    assert sweeps == sweeps_ref
    assert np.array_equal(q.cpu().numpy(), q_ref)


@pytest.mark.parametrize("S,A,seed", [(100, 4, 0), (5, 2, 1), (129, 3, 2), (300, 2, 3), (1000, 4, 4), (2051, 1, 5)])
@pytest.mark.parametrize("kernel", [0, 1])
def test_vi_dense_kernels_follow_numpy_pairwise_order(S, A, seed, kernel):
    """Dense (stochastic) mode: the 8-lanes-per-row kernel (default) and the thread-per-row kernel both
    reproduce numpy's pairwise summation bit for bit -- < 8, <= 128 and recursive-halving row lengths."""
    from rl_agents_b200.engine.vi import VIEngine
    rng = np.random.default_rng(seed)
    P = rng.uniform(size=(S, A, S))
    P /= P.sum(axis=-1, keepdims=True)
    R = rng.uniform(size=(S, A))
    term = rng.uniform(size=S) < 0.05
    q_ref, sweeps_ref = planners.value_iteration("stochastic", P, R, term, 0.9, 12)
    eng = VIEngine("stochastic", P, R, term, gamma=0.9)
    eng.problem.reserved = kernel
    q, sweeps = eng.solve(12)
    assert sweeps == sweeps_ref
    assert np.array_equal(q.cpu().numpy(), q_ref)


def test_vi_early_exit_returns_previous_iterate():
    from rl_agents_b200.engine.vi import VIEngine
    T, R = oenvs.garnet(400, 4, 1, seed=9, deterministic=True)
    term = np.zeros(400, bool)
    q_ref, sweeps_ref = planners.value_iteration("deterministic", T, R, term, 0.5, 100)
    assert sweeps_ref < 100     # converges early at gamma = 0.5
    eng = VIEngine("deterministic", T, R, term, gamma=0.5)
    q, sweeps = eng.solve(100)
    assert sweeps == sweeps_ref
    assert np.array_equal(q.cpu().numpy(), q_ref)


def test_vi_slabs_compose():
    """Two row slabs sharing V reproduce the single-slab sweep (the multi-GPU partition)."""
    import torch
    from rl_agents_b200.engine.vi import VIEngine
    S, A, B = 1001, 4, 3
    P, N, R = oenvs.garnet(S, A, B, seed=11)
    term = np.zeros(S, bool)
    full = VIEngine("sparse", P, R, term, nxt=N, gamma=0.9)
    q_full, _ = full.solve(7)
    cut = 400
    slabs = [VIEngine("sparse", P[:cut], R[:cut], term[:cut], nxt=N[:cut], gamma=0.9, row_begin=0, n_states=S),
             VIEngine("sparse", P[cut:], R[cut:], term[cut:], nxt=N[cut:], gamma=0.9, row_begin=cut, n_states=S)]
    for e in slabs:
        e.reset(7)
    for k in range(7):
        for e in slabs:
            e.sweep(k)
        torch.cuda.synchronize()
        v = slabs[0].v[(k + 1) & 1]
        v[cut:] = slabs[1].v[(k + 1) & 1][cut:]          # the all-gather step
        slabs[1].v[(k + 1) & 1].copy_(v)
        viol = slabs[0].viol + slabs[1].viol              # the all-reduce step
        slabs[0].viol.copy_(viol)
        slabs[1].viol.copy_(viol)
    q = torch.cat([slabs[0].q[7 & 1], slabs[1].q[7 & 1]]).cpu().numpy()
    assert np.array_equal(q, q_full.cpu().numpy())


# ------------------------------------------------------------ robust VI ----
def robust_models_random(mode, M, S, A, seed, shared_rows=0):
    """M seeded models: int successors [M, S, A] or dense rows [M, S, A, S], rewards [M, S, A].  The first
    `shared_rows` states of model 1 copy model 0, so both models give equal Q there."""
    rng = np.random.default_rng(seed)
    R = rng.uniform(size=(M, S, A))
    if mode == "deterministic":
        T = rng.integers(0, S, size=(M, S, A))
    else:
        T = rng.uniform(size=(M, S, A, S))
        T /= T.sum(axis=-1, keepdims=True)
    T[1:2, :shared_rows] = T[0, :shared_rows]
    R[1:2, :shared_rows] = R[0, :shared_rows]
    return T, R


def check_robust_vs_numpy(mode, T, R, gamma, iterations):
    from rl_agents_b200.engine.vi import RobustVIEngine
    q_ref, sweeps_ref = planners.robust_value_iteration(mode, T, R, gamma, iterations)
    q, sweeps = RobustVIEngine(mode, T, R, gamma=gamma).solve(iterations)
    assert sweeps == sweeps_ref
    assert np.array_equal(q.cpu().numpy(), q_ref)
    return sweeps


# gamma 0.5 converges (allclose) well before 200 sweeps; 0.95 never within 25
ROBUST_GAMMAS = [(0.5, 200), (0.95, 25)]


@pytest.mark.parametrize("gamma,iterations", ROBUST_GAMMAS)
@pytest.mark.parametrize("S", [1, 127, 1000, 5000])
@pytest.mark.parametrize("A", [1, 3, 5])
@pytest.mark.parametrize("M", [1, 2, 8])
def test_robust_vi_deterministic_vs_numpy(M, A, S, gamma, iterations):
    T, R = robust_models_random("deterministic", M, S, A, seed=1000 * M + 10 * A + S)
    sweeps = check_robust_vs_numpy("deterministic", T, R, gamma, iterations)
    assert (sweeps < iterations) == (gamma == 0.5)


@pytest.mark.parametrize("gamma,iterations", ROBUST_GAMMAS)
@pytest.mark.parametrize("S", [7, 128, 129, 300])
def test_robust_vi_dense_follows_numpy_pairwise_order(S, gamma, iterations):
    """Dense rows of < 8, exactly one 128-element pairwise block, and rows numpy splits by recursive halving."""
    T, R = robust_models_random("stochastic", 3, S, 2, seed=S)
    sweeps = check_robust_vs_numpy("stochastic", T, R, gamma, iterations)
    assert (sweeps < iterations) == (gamma == 0.5)


@pytest.mark.parametrize("mode,S", [("deterministic", 200), ("stochastic", 150)])
@pytest.mark.parametrize("iterations", [0, 1, 30])
def test_robust_vi_few_sweeps_and_tied_models(mode, S, iterations):
    """0 and 1 sweeps, and models that give equal Q on a third of the (s, a) pairs."""
    T, R = robust_models_random(mode, 3, S, 3, seed=iterations, shared_rows=S // 3)
    assert check_robust_vs_numpy(mode, T, R, 0.9, iterations) == iterations


@pytest.mark.parametrize("mode,S,A", [("deterministic", 1000, 4), ("stochastic", 129, 3)])
def test_robust_vi_with_one_model_equals_the_plain_sweep(mode, S, A):
    import torch
    from rl_agents_b200.engine.vi import RobustVIEngine, VIEngine
    T, R = robust_models_random(mode, 1, S, A, seed=3)
    q_robust, sweeps_robust = RobustVIEngine(mode, T, R, gamma=0.9).solve(40)
    q_plain, sweeps_plain = VIEngine(mode, T[0], R[0], np.zeros(S, bool), gamma=0.9).solve(40)
    assert sweeps_robust == sweeps_plain
    assert torch.equal(q_robust, q_plain)


def test_robust_vi_rejects_sparse_mode_and_zero_models():
    import torch
    from rl_agents_b200 import _lib
    from rl_agents_b200.engine.vi import RobustVIEngine
    T, R = robust_models_random("deterministic", 2, 50, 3, seed=0)
    with pytest.raises(ValueError):
        RobustVIEngine("sparse", T, R)
    eng = RobustVIEngine("deterministic", T, R, gamma=0.9)
    viol = torch.zeros(1, dtype=torch.int32, device="cuda")

    def rejected(problem, n_models, match):
        rc = eng.lib.b2_vi_robust_sweep(problem, n_models, _lib.ptr(eng.v[0]), _lib.ptr(eng.q[0]), _lib.ptr(eng.q[1]),
                                        _lib.ptr(eng.v[1]), _lib.ptr(viol), 0, _lib.current_stream())
        assert rc != 0 and match in eng.lib.b2_last_error().decode()

    sparse = _lib.VIProblem.from_buffer_copy(eng.problem)
    sparse.mode = _lib.VI_SPARSE
    rejected(sparse, 2, "deterministic or stochastic mode")
    rejected(eng.problem, 0, "bad shape")
    torch.cuda.synchronize()
    for t in eng.q + eng.v + [viol]:
        assert not bool(t.any())


# ------------------------------------------------------------------ OPD ----
def run_opd_finite(mdp, budget, gamma, roots, terminal_reward=0.0, keys_in_smem=False):
    import torch
    from rl_agents_b200 import _lib
    from rl_agents_b200.engine.opd import OPDEngine
    eng = OPDEngine(_lib.ENV_FINITE, len(roots), mdp.reward.shape[1], budget, gamma, terminal_reward, mdp=mdp,
                    keys_in_smem=keys_in_smem)
    eng.plan(torch.tensor(roots, dtype=torch.int32, device="cuda"))
    plans, res = eng.finish([np_random(0) for _ in roots])
    return eng, plans, res


@pytest.mark.parametrize("key,mdp,smem", [("large1_b500_g0.9", "large1", False), ("large1_b500_g0.9", "large1", True),
                                          ("large1_b75_g0.7", "large1", False),
                                          ("large1_b10000_g0.9", "large1", False),
                                          ("large1_b10000_g0.9", "large1", True),
                                          ("large2_b2000_g0.8", "large2", False)])
def test_opd_finite_golden(key, mdp, smem):
    g = G["opd"][key]
    eng, plans, res = run_opd_finite(product_mdp(mdp), g["budget"], g["gamma"], [0], keys_in_smem=smem)
    assert plans[0] == g["plan"]
    assert res[0, 1] == g["n_leaves"]
    assert_tree_matches(eng.tree_dict(0), g["tree"], ["reward", "lower", "upper"])


def test_opd_finite_terminal_golden():
    g = G["opd"]["large1_terminal_b300_g0.85"]
    eng, plans, res = run_opd_finite(product_mdp(terminal=terminal_variant()), 300, 0.85, [0])
    assert plans[0] == g["plan"]
    assert_tree_matches(eng.tree_dict(0), g["tree"], ["reward", "lower", "upper"])


def test_opd_finite_batch_vs_oracle():
    roots = [0, 5, 17, 42, 99, 63, 7]
    term = terminal_variant()
    eng, plans, res = run_opd_finite(product_mdp(terminal=term), 400, 0.8, roots, terminal_reward=0.25)
    for i, s0 in enumerate(roots):
        env = oenvs.FiniteMDPLite(M["large1_T"], M["large1_R"], term, state=s0)
        plan, t = planners.opd_plan(env, 400, 0.8, terminal_reward=0.25, np_random=np_random(0))
        d = eng.tree_dict(i)
        assert plans[i] == plan
        assert d["parent"].tolist() == t.parent and d["count"].tolist() == t.count
        assert d["action"].tolist() == t.action
        assert np.array_equal(d["lower"], np.array(t.lower)) and np.array_equal(d["upper"], np.array(t.upper))
        assert res[i, 3] == t.terminal_expansions


def test_opd_reward_out_of_range_raises():
    from rl_agents_b200.envs.finite_mdp import FiniteMDP
    for bad in (-0.5, 1.5):
        R = M["large1_R"].copy()
        R[24, 2] = bad           # state 24 = T[0,0]: reached at the second expansion
        mdp = FiniteMDP("deterministic", M["large1_T"], R, M["large1_term"])
        with pytest.raises(ValueError):      # deterministic.py:46-47
            run_opd_finite(mdp, 500, 0.9, [0])
        env = oenvs.FiniteMDPLite(M["large1_T"], R, M["large1_term"])
        with pytest.raises(ValueError):
            planners.opd_plan(env, 500, 0.9, np_random=np_random(0))


def test_opd_large_budget_invariants():
    """Budget 2e5 on a finite MDP (C5-sized trees are out of the oracle's reach: the reference is
    O(budget^2)): frontier keys and the first tournament level live in the global workspace here.
    Size-independent properties: every expansion creates A children; count(root) = #nodes;
    count(node) = 2 + #descendants; an internal node's bounds are the max of its children's;
    children bounds follow the update rule from the parent's creation-time lower bound."""
    import torch
    budget, gamma = 200000, 0.95
    eng, plans, res = run_opd_finite(product_mdp(), budget, gamma, [0, 13])
    n = 1 + (budget // 5) * 5
    assert res[:, 0].tolist() == [n, n] and res[:, 1].tolist() == [n - budget // 5] * 2
    for t in range(2):
        parent, fc, cnt = eng.parent[t, :n].long(), eng.first_child[t, :n].long(), eng.count[t, :n]
        lower, upper, meta = eng.lower[t, :n], eng.upper[t, :n], eng.meta[t, :n]
        internal = fc >= 0
        assert int(internal.sum()) == budget // 5 and int(cnt[0]) == n
        assert bool((((meta >> 8) & 0xff)[internal] == 5).all())
        kids = fc[internal].unsqueeze(1) + torch.arange(5, device=fc.device)
        assert bool((parent[kids] == torch.nonzero(internal)).all())
        assert bool((lower[internal] == lower[kids].max(dim=1).values).all())
        assert bool((upper[internal] == upper[kids].max(dim=1).values).all())
        sub = (cnt[kids] - 1).sum(dim=1)
        expect = sub + torch.where(torch.nonzero(internal).squeeze(1) == 0, 1, 2)
        assert bool((cnt[internal] == expect).all())
        assert bool((cnt[~internal] == 2).all())
        assert bool((upper >= lower).all()) and bool((upper[1:] <= upper[parent[1:]] + 1e-12).all())
    # the same search with the frontier in shared memory where it fits is identical (budget 10k)
    a, pa, _ = run_opd_finite(product_mdp(), 10000, 0.9, [5], keys_in_smem=True)
    b, pb, _ = run_opd_finite(product_mdp(), 10000, 0.9, [5], keys_in_smem=False)
    assert pa == pb and torch.equal(a.upper, b.upper) and torch.equal(a.count, b.count) and torch.equal(a.parent, b.parent)


def run_opd_highway(words_list, budget, gamma, keys_in_smem=False, kernel=0):
    import torch
    from rl_agents_b200 import _lib
    from rl_agents_b200.engine.opd import OPDEngine
    eng = OPDEngine(_lib.ENV_HIGHWAY, len(words_list), 5, budget, gamma, keys_in_smem=keys_in_smem, kernel=kernel)
    eng.plan(torch.tensor(np.stack(words_list), dtype=torch.int32, device="cuda"))
    plans, res = eng.finish([np_random(0) for _ in words_list])
    return eng, plans, res


@pytest.mark.parametrize("key,smem", [("s0_b75_g0.7", False), ("s1_b300_g0.8", False), ("s1_b300_g0.8", True),
                                      ("s2_b1000_g0.8", False), ("s0_b10000_g0.8", True), ("s0_b10000_g0.8", False)])
def test_opd_highway_golden(key, smem):
    g = H["opd"][key]
    words = np.array(H["states"][key[1]], dtype=np.int32)
    eng, plans, res = run_opd_highway([words], g["budget"], g["gamma"], keys_in_smem=smem)
    assert plans[0] == g["plan"]
    assert_tree_matches(eng.tree_dict(0), g["tree"], ["reward", "lower", "upper"])


def test_opd_highway_batch_vs_oracle():
    seeds = [10, 11, 12]
    words = [oenvs.make_highway_state(s).pack() for s in seeds]
    eng, plans, res = run_opd_highway(words, 120, 0.75)
    for i, s in enumerate(seeds):
        plan, t = planners.opd_plan(oenvs.HighwayLite(seed=s), 120, 0.75, np_random=np_random(0))
        d = eng.tree_dict(i)
        assert plans[i] == plan
        assert d["parent"].tolist() == t.parent and d["count"].tolist() == t.count and d["action"].tolist() == t.action
        assert np.array_equal(d["lower"], np.array(t.lower)) and np.array_equal(d["upper"], np.array(t.upper))


@pytest.mark.parametrize("kernel", [0, 1, 2])
def test_opd_highway_packed_batch_equals_single_tree_search(kernel):
    """>= 16 trees take a batch kernel (0: 8 trees per CTA, children of different trees share the
    simulation slots, block barriers between the phases; 1: one tree per warp; 2: 8 trees per CTA as a dataflow over
    a shared work ring, no block barriers); every tree must equal the one-tree-per-CTA search and the oracle."""
    seeds = list(range(40, 59))          # 19 trees: full CTAs + a partial one
    words = [oenvs.make_highway_state(s).pack() for s in seeds]
    eng, plans, res = run_opd_highway(words, 150, 0.8, kernel=kernel)
    for i in (0, 7, 8, 18):
        one, plans1, res1 = run_opd_highway([words[i]], 150, 0.8)
        a, b = eng.tree_dict(i), one.tree_dict(0)
        assert plans[i] == plans1[0] and res[i, :7].tolist() == res1[0, :7].tolist()
        for k in ("parent", "action", "count", "depth", "first_child", "done", "reward", "lower", "upper"):
            assert np.array_equal(a[k], b[k]), (i, k)
    for i in (3, 17):
        plan, t = planners.opd_plan(oenvs.HighwayLite(seed=seeds[i]), 150, 0.8, np_random=np_random(0))
        d = eng.tree_dict(i)
        assert plans[i] == plan and d["count"].tolist() == t.count and d["parent"].tolist() == t.parent
        assert np.array_equal(d["upper"], np.array(t.upper))


# ----------------------------------------------------------------- MCTS ----
def run_mcts(env_kind, roots, episodes, horizon, gamma, temperature, seeds, mdp=None):
    import torch
    from rl_agents_b200.engine.mcts import MCTSEngine, pcg64_words
    eng = MCTSEngine(env_kind, len(roots), 5, episodes, horizon, gamma, temperature, mdp=mdp)
    gens = [np_random(s) for s in seeds]
    eng.plan(torch.tensor(np.stack(roots), dtype=torch.int32, device="cuda").contiguous(),
             np.stack([pcg64_words(g) for g in gens]))
    plans, res, rng_words = eng.finish()
    return eng, plans, res, rng_words, gens


@pytest.mark.parametrize("key", sorted(G["mcts"]))
def test_mcts_finite_golden(key):
    from rl_agents_b200 import _lib
    from rl_agents_b200.engine.mcts import pcg64_words
    g = G["mcts"][key]
    mdp = product_mdp(terminal=terminal_variant() if "terminal" in key else None)
    eng, plans, res, rng_words, gens = run_mcts(_lib.ENV_FINITE, [np.int32(0)], g["episodes"], g["horizon"],
                                                g["config"]["gamma"], g["temperature"], [g["seed"]], mdp=mdp)
    assert plans[0] == g["plan"]
    assert_tree_matches(eng.tree_dict(0), g["tree"], ["value", "prior"])
    # the device consumed the stream exactly like the oracle (= the reference) does
    term = terminal_variant() if "terminal" in key else M["large1_term"]
    ref_rng = np_random(g["seed"])
    planners.mcts_plan(oenvs.FiniteMDPLite(M["large1_T"], M["large1_R"], term), g["episodes"], g["horizon"],
                       g["config"]["gamma"], g["temperature"], ref_rng)
    assert rng_words[0].tolist() == pcg64_words(ref_rng).tolist()


@pytest.mark.parametrize("key", sorted(H["mcts"]))
def test_mcts_highway_golden(key):
    from rl_agents_b200 import _lib
    g = H["mcts"][key]
    words = np.array(H["states"][key[1]], dtype=np.int32)
    eng, plans, res, _, _ = run_mcts(_lib.ENV_HIGHWAY, [words], g["episodes"], g["horizon"], g["config"]["gamma"],
                                     g["temperature"], [g["seed"]])
    assert plans[0] == g["plan"]
    assert_tree_matches(eng.tree_dict(0), g["tree"], ["value", "prior"])


def test_mcts_highway_batch_vs_oracle():
    from rl_agents_b200 import _lib
    seeds = [20, 21, 22]   # odd batch: one idle half-warp
    words = [oenvs.make_highway_state(s).pack() for s in seeds]
    eng, plans, res, _, _ = run_mcts(_lib.ENV_HIGHWAY, words, 40, 5, 0.85, 10.0, [1, 2, 3])
    for i, s in enumerate(seeds):
        plan, t = planners.mcts_plan(oenvs.HighwayLite(seed=s), 40, 5, 0.85, 10.0, np_random(i + 1))
        d = eng.tree_dict(i)
        assert plans[i] == plan
        assert d["parent"].tolist() == t.parent and d["count"].tolist() == t.count and d["action"].tolist() == t.action
        assert np.array_equal(d["value"], np.array(t.value))


# ----------------------------------------------------------------- OLOP ----
@pytest.mark.parametrize("key", sorted(G["olop"]))
def test_olop_finite_golden(key):
    """Node order / counts bit-exact; mu_ucb and value_upper within 1e-9 (the KL
    Newton solve uses log(): CUDA's and numpy's differ by at most an ulp)."""
    import torch
    from rl_agents_b200 import _lib
    from rl_agents_b200.agents.tree_search.mcts import allocation
    from rl_agents_b200.engine.mcts import pcg64_words
    from rl_agents_b200.engine.olop import OLOPEngine
    g = G["olop"][key]
    cfg = g["config"]
    episodes, horizon = allocation(max(5, cfg["budget"]), cfg["gamma"])
    assert (episodes, horizon) == (g["episodes"], g["horizon"])
    eng = OLOPEngine(_lib.ENV_FINITE, 1, 5, episodes, horizon, cfg["gamma"], cfg["upper_bound"],
                     cfg["continuation_type"], mdp=product_mdp())
    gen = np_random(g["seed"])
    eng.plan(torch.tensor([0], dtype=torch.int32, device="cuda"), pcg64_words(gen).reshape(1, -1))
    plans, res, rng_words = eng.finish()
    assert plans[0] == g["plan"]
    assert_tree_matches(eng.tree_dict(0), g["tree"], ["cumulative_reward", "mu_ucb", "upper"], exact=False,
                        rtol=1e-9, atol=1e-12)


def test_olop_highway_vs_oracle():
    import torch
    from oracle import ref_loader
    from rl_agents_b200 import _lib
    from rl_agents_b200.engine.mcts import pcg64_words
    from rl_agents_b200.engine.olop import OLOPEngine
    ub = {"type": "kullback-leibler", "time": "global", "threshold": "2*np.log(time)"}
    seeds = [30, 31, 32]
    words = [oenvs.make_highway_state(s).pack() for s in seeds]
    eng = OLOPEngine(_lib.ENV_HIGHWAY, len(seeds), 5, 12, 4, 0.8, ub, "uniform")
    eng.plan(torch.tensor(np.stack(words), dtype=torch.int32, device="cuda"),
             np.stack([pcg64_words(np_random(7 + i)) for i in range(len(seeds))]))
    plans, res, _ = eng.finish()
    for i, s in enumerate(seeds):
        rng, _ = ref_loader.legacy_np_random(7 + i)
        plan, t = planners.olop_plan(oenvs.LegacyStepEnv(oenvs.HighwayLite(seed=s)), 0, 0.8, rng, upper_bound=ub,
                                     continuation_type="uniform", episodes=12, horizon=4)
        d = eng.tree_dict(i)
        assert plans[i] == plan
        assert d["parent"].tolist() == t.parent and d["count"].tolist() == t.count and d["action"].tolist() == t.action
        np.testing.assert_allclose(d["upper"], np.array(t.upper), rtol=1e-9)
        np.testing.assert_allclose(d["cumulative_reward"], np.array(t.cumulative_reward, dtype=float), rtol=0, atol=0)


def test_olop_default_hoeffding_is_degenerate_like_the_reference():
    """The reference implements only the KL bound: with the DEFAULT config mu_ucb stays
    inf (olop.py:153-163) and the plan is all zeros."""
    import torch
    from rl_agents_b200 import _lib
    from rl_agents_b200.engine.mcts import pcg64_words
    from rl_agents_b200.engine.olop import OLOPEngine
    ub = {"type": "hoeffding", "time": "global", "threshold": "4*np.log(time)"}
    eng = OLOPEngine(_lib.ENV_FINITE, 1, 5, 14, 6, 0.8, ub, "zeros", mdp=product_mdp())
    eng.plan(torch.tensor([0], dtype=torch.int32, device="cuda"), pcg64_words(np_random(0)).reshape(1, -1))
    plans, res, _ = eng.finish()
    from oracle import ref_loader
    rng, _ = ref_loader.legacy_np_random(0)
    plan, t = planners.olop_plan(oenvs.LegacyStepEnv(oenvs.FiniteMDPLite(M["large1_T"], M["large1_R"], M["large1_term"])),
                                 100, 0.8, rng, upper_bound=ub, continuation_type="zeros")
    assert plans[0] == plan == [0] * 6
    assert eng.tree_dict(0)["count"].tolist() == t.count


# ------------------------------------------------- BASELINE full sizes ----
def test_vi_full_size_c4_vs_numpy():
    """C4 shape (S = 1e6, A = 8, B = 4 sparse): three sweeps against numpy, bit for bit, plus the
    fixed-point property V_{k+1} = max_a Q_{k+1} and the contraction |Q_{k+1} - Q_k| <= gamma^k max R."""
    import torch
    from rl_agents_b200.engine.vi import VIEngine
    S, A, B, gamma = 1_000_000, 8, 4, 0.95
    P, N, R = oenvs.garnet(S, A, B, seed=0)
    term = np.zeros(S, bool)
    eng = VIEngine("sparse", P, R, term, nxt=N, gamma=gamma)
    eng.reset(3)
    q_prev = np.zeros((S, A))
    v = np.zeros(S)
    for k in range(3):
        eng.sweep(k)
        q_ref = planners.bellman_expectation("sparse", P, R, term, v, gamma, nxt=N)
        q = eng.q[(k + 1) & 1].cpu().numpy()
        assert np.array_equal(q, q_ref), k
        v = q_ref.max(axis=-1)
        assert np.array_equal(eng.v[(k + 1) & 1].cpu().numpy(), v)
        assert np.abs(q - q_prev).max() <= gamma ** k * R.max() + 1e-12
        q_prev = q
    assert (eng.viol.cpu().numpy() > 0).all()


def test_mcts_full_size_c3_invariants():
    """C3 shape (4096 episodes x horizon 20 on HighwayLite) is beyond the Python oracle's reach
    (81 920 env steps per decision): size-independent properties instead."""
    from rl_agents_b200 import _lib
    seeds = [70, 71, 72, 73, 74]
    words = [oenvs.make_highway_state(s).pack() for s in seeds]
    eng, plans, res, rng_words, gens = run_mcts(_lib.ENV_HIGHWAY, words, 4096, 20, 0.8, 10.0, [1, 2, 3, 4, 5])
    vmax = (1 - 0.8 ** 20) / (1 - 0.8)
    for i in range(len(seeds)):
        d = eng.tree_dict(i)
        n = len(d["parent"])
        assert d["count"][0] == 4096                                   # every episode backs up through the root
        kids = d["first_child"] >= 0
        for p in np.nonzero(kids)[0][:2000]:
            c = slice(d["first_child"][p], d["first_child"][p] + d["n_children"][p])
            assert d["count"][c].sum() <= d["count"][p]                 # a visit of a child is a visit of its parent
            assert (d["parent"][c] == p).all()
        assert (d["value"] >= 0).all() and (d["value"] <= vmax + 1e-9).all()
        assert np.all(d["count"][1:] <= d["count"][d["parent"][1:]])
        assert 1 <= len(plans[i]) <= 20 and res[i, 2] <= 4096 * 20
        # the recommended first action is the most visited root child (mcts.py:212-218)
        c = slice(d["first_child"][0], d["first_child"][0] + d["n_children"][0])
        assert plans[i][0] == d["action"][c][np.argmax(d["count"][c])] or \
            (d["count"][c] == d["count"][c].max()).sum() > 1
    assert len({tuple(w) for w in rng_words.tolist()}) == len(seeds)   # independent streams advanced


# ------------------------------------------------------------ edge cases ----
def test_edge_cases_small_budgets_and_argument_validation():
    import torch
    from rl_agents_b200 import _lib
    from rl_agents_b200.engine.mcts import MCTSEngine, pcg64_words
    from rl_agents_b200.engine.opd import OPDEngine
    # budget < action_space.n: zero expansions, empty plan (the reference's get_plan returns [] too)
    eng, plans, res = run_opd_finite(product_mdp(), 3, 0.9, [0, 1, 2])
    assert plans == [[], [], []] and res[:, 0].tolist() == [1, 1, 1] and eng.tree_dict(0)["count"].tolist() == [1]
    plan, t = planners.opd_plan(oenvs.FiniteMDPLite(M["large1_T"], M["large1_R"], M["large1_term"]), 3, 0.9,
                                np_random=np_random(0))
    assert plan == [] and t.count == [1]
    # exactly one expansion
    eng, plans, res = run_opd_highway([oenvs.make_highway_state(0).pack()], 5, 0.8)
    plan, t = planners.opd_plan(oenvs.HighwayLite(seed=0), 5, 0.8, np_random=np_random(0))
    assert plans[0] == plan and eng.tree_dict(0)["count"].tolist() == t.count
    # a single MCTS episode: expands the root, one rollout, no child visited
    words = oenvs.make_highway_state(1).pack()
    eng, plans, res, _, _ = run_mcts(_lib.ENV_HIGHWAY, [words], 1, 3, 0.8, 10.0, [4])
    plan, t = planners.mcts_plan(oenvs.HighwayLite(seed=1), 1, 3, 0.8, 10.0, np_random(4))
    assert plans[0] == plan and eng.tree_dict(0)["count"].tolist() == t.count
    assert np.array_equal(eng.tree_dict(0)["value"], np.array(t.value))
    # argument validation comes back as an error code + message, not a crash
    bad = OPDEngine(_lib.ENV_FINITE, 1, 5, 100, 0.9, mdp=product_mdp())
    bad.cfg.node_capacity = 3
    with pytest.raises(_lib.B2Error, match="node_capacity"):
        bad.plan(torch.zeros(1, dtype=torch.int32, device="cuda"))
    m = MCTSEngine(_lib.ENV_FINITE, 1, 5, 4, 3, 0.9, 10.0, mdp=product_mdp())
    m.cfg.rollout_policy = 7
    with pytest.raises(_lib.B2Error, match="policy"):
        m.plan(torch.zeros(1, dtype=torch.int32, device="cuda"), pcg64_words(np_random(0)).reshape(1, -1))


@pytest.mark.parametrize("kernel", [0, 2])
def test_opd_highway_c2_full_size_batch_vs_c_oracle(kernel):
    """C2 at full size, many decisions: 24 scenes x budget 10 000 through the batch kernels (barrier and dataflow
    variants), every node array of every tree bit-identical with the C oracle (itself pinned to the reference's
    golden tree)."""
    from oracle import c_oracle
    seeds = list(range(500, 524))
    words = [oenvs.make_highway_state(s).pack() for s in seeds]
    eng, plans, res = run_opd_highway(words, 10000, 0.8, kernel=kernel)
    for i, w in enumerate(words):
        t = c_oracle.opd_plan(w, 10000, 0.8)
        d = eng.tree_dict(i)
        assert res[i, 0] == len(t["parent"]) and res[i, 1] == t["n_leaves"]
        for k in ("parent", "action", "count", "depth", "first_child", "n_children"):
            assert np.array_equal(np.asarray(d[k], dtype=np.int64), t[k].astype(np.int64)), (i, k)
        assert np.array_equal(d["done"], t["done"].astype(bool))
        for k in ("reward", "lower", "upper"):
            assert np.array_equal(d[k], t[k]), (i, k)


def test_mcts_highway_c3_full_size_vs_c_oracle():
    """C3 at full size (4096 episodes x horizon 20): every node statistic and the RNG stream position
    bit-identical with the C oracle (itself pinned to the reference's golden MCTS trees)."""
    from oracle import c_oracle
    from oracle.pcg64 import PCG64
    from rl_agents_b200 import _lib
    seeds = [70, 71, 72]
    words = [oenvs.make_highway_state(s).pack() for s in seeds]
    eng, plans, res, rng_words, gens = run_mcts(_lib.ENV_HIGHWAY, words, 4096, 20, 0.8, 10.0, [1, 2, 3])
    for i in range(len(seeds)):
        t, w = c_oracle.mcts_plan(words[i], 4096, 20, 0.8, 10.0, PCG64.from_numpy(np_random(i + 1)).words())
        d = eng.tree_dict(i)
        assert res[i, 0] == len(t["parent"])
        for k in ("parent", "action", "count", "first_child", "n_children"):
            assert np.array_equal(np.asarray(d[k], dtype=np.int64), t[k].astype(np.int64)), (i, k)
        assert np.array_equal(d["value"], t["value"]) and np.array_equal(d["prior"], t["prior"])
        assert rng_words[i].tolist() == w.tolist()


def test_constant_divisor_division_is_ieee_exact_exhaustively():
    """hw::div_const (3 instructions) against the IEEE division for the spec's two constant divisors: every
    mantissa, both signs, 41 exponents -- on the device itself."""
    import torch
    from rl_agents_b200 import _lib
    lib = _lib.load()
    out = torch.zeros(1, dtype=torch.int64, device="cuda")
    _lib.check(lib.b2_selftest_const_division(_lib.ptr(out), _lib.current_stream()))
    assert int(out.item()) == 0
