"""Shared helpers of the parity tests: golden loading and tree comparison."""
import json
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load_golden(name):
    with open(os.path.join(GOLDEN, name)) as f:
        return json.load(f)


def load_mdps():
    return np.load(os.path.join(GOLDEN, "finite_mdps.npz"))


def tree_summary(tree):
    """Same digest as tests/golden/make_golden.py::summarize (non-full)."""
    out = {"n_nodes": len(tree["parent"])}
    for k, v in tree.items():
        if k in ("lower", "upper", "value", "reward", "cumulative_reward", "mu_ucb"):
            out["sum_" + k] = float(np.sum(np.asarray(v, dtype=np.float64)))
        elif k in ("parent", "action", "count"):
            a = np.asarray(v, dtype=np.int64)
            out["sum_" + k] = int(a.sum())
            out["wsum_" + k] = int((a * (np.arange(len(a)) % 1009)).sum())
    return out


def assert_tree_matches(got, golden, float_fields, exact=True, rtol=0.0, atol=0.0):
    """`got`: dict of equal-length sequences; `golden`: a golden tree, either
    full or the digest form (first 64 nodes + sums)."""
    full = "n_nodes" not in golden
    n = len(golden["parent"]) if full else golden["n_nodes"]
    assert len(got["parent"]) == n
    k = n if full else 64
    for f in ("parent", "action", "count"):
        assert [int(x) for x in got[f][:k]] == [int(x) for x in golden[f][:k]], f
    for f in float_fields:
        a = np.asarray(got[f][:k], dtype=np.float64)
        b = np.asarray(golden[f][:k], dtype=np.float64)
        if exact:
            assert np.array_equal(a, b), (f, np.abs(a - b).max())
        else:
            np.testing.assert_allclose(a, b, rtol=rtol, atol=atol, err_msg=f)
    if "done" in golden and "done" in got:
        assert [bool(x) for x in got["done"][:k]] == [bool(x) for x in golden["done"][:k]]
    if not full:
        s = tree_summary({f: got[f] for f in list(float_fields) + ["parent", "action", "count"]})
        for key, val in s.items():
            if key.startswith("sum_") and key[4:] in float_fields:
                if exact:
                    assert val == golden[key], key
                else:
                    np.testing.assert_allclose(val, golden[key], rtol=max(rtol, 1e-12), err_msg=key)
            elif key != "n_nodes":
                assert val == golden[key], key


def canonical_tree(first_child, n_children, fields):
    """Breadth-first listing (children in stored order) of per-node tuples: an id-independent form
    for comparing trees whose node numbering differs (re-rooted sub-trees)."""
    order, head = [0], 0
    while head < len(order):
        n = order[head]
        order.extend(range(first_child[n], first_child[n] + n_children[n]) if n_children[n] > 0 else [])
        head += 1
    return [[int(n_children[i])] + [f[i] for f in fields] for i in order]


def receding_horizon_schedule(agent_cls, receding_horizon):
    """Drive a subclass of `agent_cls` (an AbstractTreeSearchAgent) by a scripted planner whose plans have fixed
    lengths, for 25 decisions with a reset() before the 14th: (plan() outputs, the planner's call log, the config).
    Lists only, so that the result compares equal to its JSON form in tests/golden/golden_host.json."""
    lengths = [4, 1, 3, 2, 6, 1, 1, 5, 3]

    class Scripted(object):
        def __init__(self, env, config):
            self.log, self.k = [], 0

        def plan(self, state, observation):
            n = lengths[self.k % len(lengths)]
            self.k += 1
            self.log.append(["plan", observation])
            return [10 * self.k + i for i in range(n)]

        def step_tree(self, actions):
            self.log.append(["step", list(actions)])

        def step_by_reset(self):
            self.log.append(["reset"])

        def seed(self, seed=None):
            return [seed]

    class Env(object):
        unwrapped = property(lambda self: self)

    class A(agent_cls):
        PLANNER_TYPE = Scripted
    a = A(Env(), {"receding_horizon": receding_horizon})
    outs = []
    for t in range(25):
        if t == 13:
            a.reset()
        outs.append(list(a.plan(t)))
    return outs, a.planner.log, a.config


def ttc_edge_scenes():
    """HighwayLite scenes that exercise the corners of the TTC-grid conversion (docs/HIGHWAY_LITE_SPEC.md section 9):
    absent slots, speeds equal to the grid speeds, integer times / zero distances, headings beyond the cosine clamp,
    negative speeds, vehicles off the road or between lanes, all ego cells, relative speeds inside the +-0.01 guard."""
    from oracle import envs as oenvs
    out = []
    rng = np.random.default_rng(7)
    for s in range(40):
        w = oenvs.make_highway_state(200 + s).pack()
        f = w[:96].view(np.float32)
        kind = s % 8
        if kind == 0:
            w[112 + rng.integers(1, 16, size=6)] = 0
        elif kind == 1:
            f[48 + 1:48 + 16] = np.float32(rng.choice([20.0, 25.0, 30.0], size=15))
        elif kind == 2:
            f[1:16] = f[0] + np.float32(rng.integers(-3, 4, size=15) * 5.0)
        elif kind == 3:
            f[32 + 1:32 + 16] = np.float32(rng.uniform(-2.0, 2.0, size=15))
        elif kind == 4:
            f[48 + 1:48 + 16] = np.float32(rng.uniform(-5.0, 45.0, size=15))
        elif kind == 5:
            f[16 + 1:16 + 16] = np.float32(rng.uniform(-6.0, 18.0, size=15))
        elif kind == 6:
            w[129] = int(rng.integers(0, 3))
            f[16] = np.float32(rng.choice([0.0, 4.0, 8.0, 12.0, 2.0, 6.0, 10.0]))
        else:
            f[1:16] = f[0] + np.float32(rng.uniform(-400, 400, size=15))
            f[48 + 1:48 + 16] = np.float32(f[48] + rng.uniform(-0.02, 0.02, size=15))
        out.append(w)
    return out
