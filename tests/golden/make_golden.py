"""Generate the golden vectors under tests/golden/ by running the UNMODIFIED
reference (/root/reference) on the oracle env models.

Build-container only (the reference tree does not travel to the GPU box);
the outputs are committed.  Usage:  python tests/golden/make_golden.py [--only-highway-vi | --only-host]
"""
import copy
import json
import os
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from oracle import ref_loader  # noqa: E402
from oracle import envs  # noqa: E402

ref_loader.load_reference()
from rl_agents.agents.tree_search import deterministic as ref_det  # noqa: E402
from rl_agents.agents.tree_search import mcts as ref_mcts  # noqa: E402
from rl_agents.agents.tree_search import olop as ref_olop  # noqa: E402
from rl_agents.agents.tree_search import abstract as ref_abs  # noqa: E402
from rl_agents.agents.dynamic_programming import value_iteration as ref_vi  # noqa: E402
from rl_agents import utils as ref_utils  # noqa: E402

CREATED = []


def _instrument(cls):
    """Record node creation order at run time (sources stay unmodified)."""
    orig = cls.__init__

    def init(self, *a, **k):
        orig(self, *a, **k)
        CREATED.append(self)
    cls.__init__ = init


for _cls in (ref_det.DeterministicNode, ref_mcts.MCTSNode, ref_olop.OLOPNode):
    _instrument(_cls)


def dump_tree(fields, root):
    # the planner builds a throw-away root in __init__ and again on
    # step_by_reset (abstract.py:113-114,189-193): keep the final tree only
    def top(n):
        while n.parent is not None:
            n = n.parent
        return n
    CREATED[:] = [n for n in CREATED if top(n) is root]
    assert CREATED[0] is root
    ids = {id(n): i for i, n in enumerate(CREATED)}
    out = {"parent": [], "action": [], "count": []}
    for f in fields:
        out[f] = []
    for n in CREATED:
        out["parent"].append(ids[id(n.parent)] if n.parent is not None else -1)
        act = -1
        if n.parent is not None:
            for a, c in n.parent.children.items():
                if c is n:
                    act = int(a)
        out["action"].append(act)
        out["count"].append(int(n.count))
        for f in fields:
            v = getattr(n, f)
            out[f].append(bool(v) if isinstance(v, (bool, np.bool_)) else float(v))
    return out


def summarize(tree, full):
    if full:
        return tree
    keep = {k: v[:64] for k, v in tree.items()}
    keep["n_nodes"] = len(tree["parent"])
    for k, v in tree.items():
        if k in ("lower", "upper", "value", "reward", "cumulative_reward", "mu_ucb"):
            keep["sum_" + k] = float(np.sum(np.asarray(v, dtype=np.float64)))
        elif k in ("parent", "action", "count"):
            keep["sum_" + k] = int(np.sum(np.asarray(v, dtype=np.int64)))
            keep["wsum_" + k] = int(np.sum(np.asarray(v, dtype=np.int64) * (np.arange(len(v)) % 1009)))
    return keep


def run_opd(env, budget, gamma, seed=0, full=True):
    del CREATED[:]
    agent = ref_det.DeterministicPlannerAgent(env, {"budget": budget, "gamma": gamma})
    agent.seed(seed)
    t0 = time.perf_counter()
    plan = agent.plan(None)
    dt = time.perf_counter() - t0
    for n in CREATED:
        n.lower, n.upper = n.value_lower, n.value_upper
    tree = dump_tree(["reward", "lower", "upper", "done"], agent.planner.root)
    return {"budget": budget, "gamma": gamma, "seed": seed, "plan": [int(a) for a in plan],
            "n_leaves": len(agent.planner.leaves), "seconds": dt,
            "tree": summarize(tree, full)}


def run_mcts(env, config, seed=0, full=True):
    del CREATED[:]
    agent = ref_mcts.MCTSAgent(env, dict(config))
    agent.seed(seed)
    t0 = time.perf_counter()
    plan = agent.plan(None)
    dt = time.perf_counter() - t0
    tree = dump_tree(["value", "prior"], agent.planner.root)
    return {"config": config, "seed": seed, "plan": [int(a) for a in plan],
            "episodes": int(agent.planner.config["episodes"]),
            "horizon": int(agent.planner.config["horizon"]),
            "temperature": float(agent.planner.config["temperature"]),
            "seconds": dt, "tree": summarize(tree, full)}


def run_olop(env, config, seed=0, full=True):
    del CREATED[:]
    agent = ref_olop.OLOPAgent(envs.LegacyStepEnv(env), dict(config))
    agent.planner.np_random, _ = ref_loader.legacy_np_random(seed)
    plan = agent.plan(None)
    for n in CREATED:
        n.upper = n.value_upper
    tree = dump_tree(["cumulative_reward", "mu_ucb", "upper", "done"], agent.planner.root)
    return {"config": config, "seed": seed, "plan": [int(a) for a in plan],
            "episodes": int(agent.planner.config["episodes"]),
            "horizon": int(agent.planner.config["horizon"]),
            "tree": summarize(tree, full)}


def run_vi(mdp_env, gamma, iterations):
    agent = ref_vi.ValueIterationAgent(mdp_env, {"gamma": gamma, "iterations": iterations})
    q = agent.state_action_value
    return {"gamma": gamma, "iterations": iterations, "q": q.tolist(),
            "act0": int(agent.act(0)) if True else None}


def load_json_mdp(path):
    with open(path) as f:
        cfg = json.load(f)
    return (np.array(cfg["transition"]), np.array(cfg["reward"], dtype=np.float64),
            np.array(cfg.get("terminal", [0] * len(cfg["reward"]))).astype(bool), cfg["mode"])


def main():
    cfg_dir = os.path.join(ref_loader.REFERENCE_ROOT, "scripts/configs/FiniteMDPEnv")
    out = {}

    # ---------------- finite MDP fixtures (inputs) ----------------
    T, R, term, mode = load_json_mdp(os.path.join(cfg_dir, "large/env_1.json"))
    T2, R2, term2, _ = load_json_mdp(os.path.join(cfg_dir, "large/env_2.json"))
    Tt, Rt, termt, _ = load_json_mdp(os.path.join(cfg_dir, "trap/env_1.json"))
    Tl, Rl, terml, _ = load_json_mdp(os.path.join(cfg_dir, "env_loop.json"))
    np.savez_compressed(os.path.join(HERE, "finite_mdps.npz"),
                        large1_T=T, large1_R=R, large1_term=term,
                        large2_T=T2, large2_R=R2, large2_term=term2,
                        trap_T=Tt, trap_R=Rt, trap_term=termt,
                        loop_T=Tl, loop_R=Rl, loop_term=terml)

    def finite(Tm=T, Rm=R, tm=term):
        return envs.FiniteMDPLite(Tm, Rm, tm, mode="deterministic", state=0)

    # ---------------- VI ----------------
    vi = {}
    vi["large1_g0.9_it100"] = run_vi(finite(), 0.9, 100)
    vi["large1_g1.0_it2"] = run_vi(finite(), 1.0, 2)
    vi["trap_g0.9_it100"] = run_vi(finite(Tt, Rt, termt), 0.9, 100)
    vi["loop_g0.9_it100"] = run_vi(finite(Tl, Rl, terml), 0.9, 100)
    # dense stochastic + sparse, C1-shaped (SURVEY 8d): seed 0, S=100, A=4
    rng = np.random.default_rng(0)
    P = rng.uniform(size=(100, 4, 100)); P /= P.sum(-1, keepdims=True)
    Rd = rng.uniform(size=(100, 4))
    env_d = envs.FiniteMDPLite(P, Rd, None, mode="stochastic")
    vi["dense_c1_g0.95_it100"] = run_vi(env_d, 0.95, 100)
    Ps, Ns, Rs = envs.garnet(500, 4, 3, seed=1)
    terms = np.zeros(500, bool); terms[::37] = True
    env_s = envs.FiniteMDPLite(Ps, Rs, terms, mode="sparse", nxt=Ns)
    vi["sparse_garnet500_g0.95_it100"] = run_vi(env_s, 0.95, 100)
    out["vi"] = vi

    # ---------------- robust VI (SURVEY 8f rank 1) ----------------
    from rl_agents.agents.dynamic_programming.robust_value_iteration import RobustValueIterationAgent
    rvi = {}
    models_det = []
    for m in range(3):
        Tm, Rm = envs.garnet(300, 4, 1, seed=20 + m, deterministic=True)
        models_det.append({"mode": "deterministic", "transition": Tm.tolist(), "reward": Rm.tolist()})
    agent = RobustValueIterationAgent(None, {"gamma": 0.9, "iterations": 60, "models": models_det})
    rvi["det_3x300x4_g0.9_it60"] = {"q": agent.get_state_action_value().tolist(), "act7": int(agent.act(7))}
    models_dense = []
    for m in range(2):
        rng_m = np.random.default_rng(30 + m)
        Pm = rng_m.uniform(size=(40, 3, 40)); Pm /= Pm.sum(-1, keepdims=True)
        models_dense.append({"mode": "stochastic", "transition": Pm.tolist(), "reward": rng_m.uniform(size=(40, 3)).tolist()})
    agent = RobustValueIterationAgent(None, {"gamma": 0.95, "iterations": 100, "models": models_dense})
    rvi["dense_2x40x3_g0.95_it100"] = {"q": agent.get_state_action_value().tolist(), "act7": int(agent.act(7))}
    out["robust_vi"] = rvi

    # ---------------- OPD on finite ----------------
    opd = {}
    opd["large1_b500_g0.9"] = run_opd(finite(), 500, 0.9)
    opd["large1_b75_g0.7"] = run_opd(finite(), 75, 0.7)
    opd["large1_b10000_g0.9"] = run_opd(finite(), 10000, 0.9, full=False)
    opd["large2_b2000_g0.8"] = run_opd(finite(T2, R2, term2), 2000, 0.8, full=False)
    # terminal states + terminal_reward path: mark a few states terminal
    termx = term.copy(); termx[[3, 17, 66, 91]] = True
    opd["large1_terminal_b300_g0.85"] = run_opd(finite(T, R, termx), 300, 0.85)
    out["opd"] = opd

    # ---------------- MCTS on finite ----------------
    mc = {}
    mc["large1_b10000_g0.9"] = run_mcts(finite(), {"budget": 10000, "gamma": 0.9}, full=False)
    mc["large1_b400_g0.8"] = run_mcts(finite(), {"budget": 400, "gamma": 0.8})
    mc["large1_ep200_h12_g0.95_T5"] = run_mcts(
        finite(), {"episodes": 200, "horizon": 12, "gamma": 0.95, "temperature": 5.0}, seed=3)
    mc["large1_terminal_b600_g0.9"] = run_mcts(finite(T, R, termx), {"budget": 600, "gamma": 0.9}, seed=1)
    out["mcts"] = mc

    # ---------------- DROP: DiscreteRobustPlanner on the joint env of M models (robust.py:9-47) ----------------
    # the reference's JointEnv.step returns the legacy 4-tuple while DeterministicNode.expand unpacks five values
    # (deterministic.py:41): the shim below only re-packs the tuple, like the OLOP legacy shim does the other way
    from rl_agents.agents.robust import robust as ref_robust

    class JointEnv5(ref_robust.JointEnv):
        def step(self, action):
            transitions = [state.step(action) for state in self.joint_state]
            observations, rewards, terminals, truncated, info = zip(*transitions)
            return observations, np.array(rewards), np.array(terminals), np.array(truncated), info

    drop = {}
    for key, (names, bud, gam, tr_) in {"large12_b300_g0.85": (("large1", "large2"), 300, 0.85, 0.0),
                                         "large1x3_terminal_b400_g0.8": (("large1", "large1t", "large2"), 400, 0.8, 0.3)}.items():
        def model(nm):
            if nm == "large1":
                return finite()
            if nm == "large1t":
                return finite(T, R, termx)
            return finite(T2, R2, term2)
        del CREATED[:]
        agent = ref_robust.DiscreteRobustPlannerAgent(finite(), {"budget": bud, "gamma": gam, "terminal_reward": tr_})
        agent.seed(0)
        agent.env = JointEnv5([model(nm) for nm in names])
        plan = ref_det.DeterministicPlannerAgent.plan(agent, None)       # skip robust.py:66-67 (env preprocessing)
        for n in CREATED:
            n.lower, n.upper = float(np.min(n.value_lower)), float(np.min(n.value_upper))
        tree = dump_tree(["lower", "upper"], agent.planner.root)
        drop[key] = {"models": list(names), "budget": bud, "gamma": gam, "terminal_reward": tr_,
                     "plan": [int(a) for a in plan], "tree": summarize(tree, True)}
    out["drop"] = drop

    # ---------------- MCTS policies other than random_available (mcts.py:34-97) ----------------
    pol = {}
    pref_cfg = {"budget": 400, "gamma": 0.8,
                "prior_policy": {"type": "preference", "action": 3, "ratio": 2},
                "rollout_policy": {"type": "preference", "action": 1, "ratio": 3}}
    pol["large1_preference_b400_g0.8"] = run_mcts(finite(), pref_cfg, seed=2)
    rand_cfg = {"budget": 300, "gamma": 0.85, "prior_policy": {"type": "random"}, "rollout_policy": {"type": "random"}}
    pol["large1_random_b300_g0.85"] = run_mcts(finite(), rand_cfg, seed=5)
    out["mcts_policies"] = pol

    # ---------------- closed-loop MCTS (mcts.py:125,147,267-273) on a deterministic env ----------------
    agent = ref_mcts.MCTSAgent(finite(), {"budget": 400, "gamma": 0.8, "closed_loop": True})
    agent.seed(3)
    plan = agent.plan(0)
    root = agent.planner.root
    out["mcts_closed_loop"] = {
        "config": {"budget": 400, "gamma": 0.8, "closed_loop": True}, "seed": 3,
        "plan_actions": [int(a) for a in plan[0::2]],          # the reference interleaves observation keys
        "plan_len": len(plan),
        "root": [[int(a), int(c.count), float(c.value)] for a, c in root.children.items()],
        "root_count": int(root.count), "root_value": float(root.value)}

    # ---------------- MCTS with step_strategy "subtree": two consecutive decisions ----------------
    def canonical(root):
        nodes, head = [root], 0
        rows = []
        while head < len(nodes):
            nd = nodes[head]
            rows.append([len(nd.children), int(nd.count), float(nd.value), float(nd.prior)])
            nodes.extend(nd.children.values())
            head += 1
        return rows
    env_s = finite()
    agent = ref_mcts.MCTSAgent(env_s, {"budget": 300, "gamma": 0.85, "step_strategy": "subtree"})
    agent.seed(4)
    sub = {"plans": [], "trees": [], "states": []}
    for _ in range(3):
        sub["states"].append(int(env_s.mdp.state))
        plan = agent.plan(None)
        sub["plans"].append([int(a) for a in plan])
        sub["trees"].append(canonical(agent.planner.root))
        env_s.step(plan[0])
    sub["episodes"], sub["horizon"] = int(agent.planner.config["episodes"]), int(agent.planner.config["horizon"])
    sub["temperature"] = float(agent.planner.config["temperature"])
    out["mcts_subtree"] = sub

    # ---------------- GBOP-T (state-aware OPD) on finite: oracle groundwork for SURVEY 8f rank 3 ----------------
    from rl_agents.agents.tree_search.state_aware import StateAwarePlannerAgent
    gb = {}
    for key, (bud, gam, seed_) in {"large1_b500_g0.9": (500, 0.9, 0), "large1_b2000_g0.8": (2000, 0.8, 1)}.items():
        del CREATED[:]
        _instrument_done = True
        agent = StateAwarePlannerAgent(finite(), {"budget": bud, "gamma": gam})
        agent.seed(seed_)
        plan = agent.plan(0)
        pl = agent.planner
        gb[key] = {"budget": bud, "gamma": gam, "seed": seed_, "plan": [int(a) for a in plan],
                   "state_values": {str(k): float(v) for k, v in pl.state_values.items()},
                   "n_leaves": len(pl.leaves), "n_states": len(pl.state_nodes),
                   "root_upper": float(pl.root.get_value_upper_bound()),
                   "leaf_depth_sum": int(sum(l.depth for l in pl.leaves)),
                   "leaf_lower_sum": float(sum(l.value_lower for l in pl.leaves))}
    out["gbopt"] = gb

    # ---------------- GBOP-D (graph-based OPD, graph_based.py): legacy 4-tuple step like OLOP ----------------
    from rl_agents.agents.tree_search.graph_based import GraphBasedPlannerAgent
    gd = {}
    for key, (bud, gam, acc, seed_) in {"large1_b500_g0.9_acc0": (500, 0.9, 0, 0), "large1_b1500_g0.8_acc0": (1500, 0.8, 0, 2),
                                        "large1_b500_g0.9_default": (500, 0.9, None, 0)}.items():
        cfg = {"budget": bud, "gamma": gam}
        if acc is not None:
            cfg["accuracy"] = acc
        agent = GraphBasedPlannerAgent(envs.LegacyStepEnv(finite()), cfg)
        agent.seed(seed_)
        plan = agent.plan(0)
        pl = agent.planner
        gd[key] = {"budget": bud, "gamma": gam, "accuracy": agent.config["accuracy"], "seed": seed_,
                   "sampling_timeout": agent.config["sampling_timeout"], "plan": [int(a) for a in plan],
                   "nodes": {str(k): [float(n.value_lower), float(n.value_upper), bool(n.children)]
                             for k, n in pl.nodes.items()}}
    # the default accuracy (1e-2) is NOT reproducible bit for bit, not even between two runs of this script
    gd["large1_b500_g0.9_default"]["note"] = (
        "run-dependent at the 1e-6 level: with accuracy > 0 the reference's partial value iteration pushes "
        "list(node.parents), a Python SET of node objects, i.e. an order that follows memory addresses "
        "(graph_based.py); plan, node set and expanded flags are reproducible, the bounds only within the accuracy "
        "-- tests compare them with that tolerance")
    out["gbopd"] = gd

    # ---------------- OLOP (KL) on finite ----------------
    ol = {}
    kl_cfg = {"budget": 200, "gamma": 0.9, "continuation_type": "uniform",
              "upper_bound": {"type": "kullback-leibler", "time": "global", "threshold": "2*np.log(time)"}}
    ol["large1_b200_g0.9_uniform"] = run_olop(finite(), kl_cfg)
    kl_cfg2 = {"budget": 500, "gamma": 0.7, "continuation_type": "zeros",
               "upper_bound": {"type": "kullback-leibler", "time": "local", "threshold": "1*np.log(time)"}}
    ol["large1_b500_g0.7_zeros_local"] = run_olop(finite(), kl_cfg2, seed=2)
    out["olop"] = ol
    out["allocation"] = {"%d_%g" % (b, g): list(ref_olop.OLOP.allocation(b, g))
                         for b, g in [(100, .8), (400, .8), (500, .7), (600, .8), (10000, .8),
                                      (10000, .9), (81920, .8)]}
    out["kl_upper_bound"] = [
        [s, c, th, float(ref_utils.kl_upper_bound(s, c, th, eps=1e-3))]
        for s, c, th in [(0.5, 1, float(np.log(10))), (5, 10, float(np.log(20))), (10, 20, float(np.log(40)))]]
    out["kl_upper_bound_eps1e-2"] = [
        [s, c, th, float(ref_utils.kl_upper_bound(s, c, th))]
        for s, c, th in [(0.5, 1, 2.0), (3.25, 7, 5.5), (0, 4, 3.0), (4, 4, 3.0), (17.5, 40, 9.2)]]
    with open(os.path.join(HERE, "golden_finite.json"), "w") as f:
        json.dump(out, f)
    print("finite done")

    # ---------------- HighwayLite ----------------
    hw = {"states": {}, "traces": {}, "opd": {}, "mcts": {}}
    for seed in range(6):
        hw["states"][str(seed)] = envs.make_highway_state(seed).pack().tolist()
    # env traces: random available actions, full state words after each step
    for seed in range(8):
        env = envs.HighwayLite(seed=seed)
        rng = np.random.default_rng(100 + seed)
        steps = []
        for _ in range(45):
            avail = env.get_available_actions()
            # mostly IDLE so that the trace survives long enough to exercise
            # IDM / MOBIL / truncation, with random lane/speed changes mixed in
            if seed < 4:
                a = 1 if rng.uniform() < 0.7 else int(avail[rng.integers(len(avail))])
            else:   # slow ego: traffic queues behind it, episode reaches truncation
                a = 4 if 4 in avail else 1
            _, r, term_, trunc, _ = env.step(a)
            steps.append({"a": a, "avail": [int(x) for x in avail], "r": float(r), "term": bool(term_),
                          "trunc": bool(trunc), "state": env.state.pack().tolist()})
            if term_:
                break
        hw["traces"][str(seed)] = steps
    hw["opd"]["s0_b75_g0.7"] = run_opd(envs.HighwayLite(seed=0), 75, 0.7)
    hw["opd"]["s1_b300_g0.8"] = run_opd(envs.HighwayLite(seed=1), 300, 0.8)
    hw["opd"]["s2_b1000_g0.8"] = run_opd(envs.HighwayLite(seed=2), 1000, 0.8, full=False)
    hw["mcts"]["s0_ep60_h6_g0.8"] = run_mcts(envs.HighwayLite(seed=0),
                                              {"episodes": 60, "horizon": 6, "gamma": 0.8}, seed=0)
    hw["mcts"]["s3_b200_g0.8"] = run_mcts(envs.HighwayLite(seed=3), {"budget": 200, "gamma": 0.8}, seed=5)
    if "--small" not in sys.argv:      # C2 full size: ~1 minute in the reference
        hw["opd"]["s0_b10000_g0.8"] = run_opd(envs.HighwayLite(seed=0), 10000, 0.8, full=False)
    with open(os.path.join(HERE, "golden_highway.json"), "w") as f:
        json.dump(hw, f)
    print("highway done")
    highway_vi()


def highway_vi():
    """ValueIterationAgent on HighwayLite scenes through `env.unwrapped.to_finite_mdp()` (value_iteration.py:17,32;
    shipped config scripts/configs/HighwayEnv/agents/ValueIterationAgent/baseline.json: iterations 10, gamma 1):
    the unmodified reference agent on the oracle's TTC-grid MDP of the scene -> tests/golden/golden_highway_vi.json."""
    out = {"cases": []}
    for seed in range(6):
        env = envs.HighwayLite(seed=seed)
        rng = np.random.default_rng(300 + seed)
        for step in range(0, 13):
            if step in (0, 3, 7, 12):
                for cfg in ({"iterations": 10}, {"gamma": 0.9, "iterations": 100}):
                    agent = ref_vi.ValueIterationAgent(env, dict(cfg))
                    mdp = agent.mdp
                    case = {"seed": seed, "step": step, "config": cfg, "words": env.state.pack().tolist(),
                            "state": int(mdp.state), "shape": list(mdp.original_shape),
                            "grid": envs.highway_ttc_grid(env.state).tolist(),
                            "q": agent.state_action_value.tolist(), "act": int(agent.act(None))}
                    if seed == 0 and step in (0, 7) and "gamma" not in cfg:
                        case["transition"] = mdp.transition.tolist()
                        case["reward"] = mdp.reward.tolist()
                        case["terminal"] = [bool(x) for x in mdp.terminal]
                    out["cases"].append(case)
            avail = env.get_available_actions()
            a = 1 if rng.uniform() < 0.5 else int(avail[rng.integers(len(avail))])
            _, _, term_, _, _ = env.step(a)
            if term_:
                break
    with open(os.path.join(HERE, "golden_highway_vi.json"), "w") as f:
        json.dump(out, f)
    print("highway VI done:", len(out["cases"]), "cases")


FACTORY_CASES = [("rl_agents_b200.agents.tree_search.deterministic.DeterministicPlannerAgent", ref_det.DeterministicPlannerAgent,
                  {"budget": 75}),
                 ("rl_agents_b200.agents.tree_search.mcts.MCTSAgent", ref_mcts.MCTSAgent, {"budget": 400, "gamma": 0.9})]


def host():
    """The agent shell: the completed configs of the reference agents that the drop-ins replace (built on the
    large/env_1 finite MDP), and the reference's AbstractTreeSearchAgent driven by the scripted planner of
    tests/util.py::receding_horizon_schedule -> tests/golden/golden_host.json."""
    from tests.util import load_mdps, receding_horizon_schedule
    m = load_mdps()
    env = envs.FiniteMDPLite(m["large1_T"], m["large1_R"], m["large1_term"])
    out = {"factory": [{"class": path, "config_in": cfg, "config": dict(ref_cls(env, dict(cfg)).config)}
                       for path, ref_cls, cfg in FACTORY_CASES],
           "receding_horizon": {}}
    for h in (1, 2, 3, 5):
        plans, log, config = receding_horizon_schedule(ref_abs.AbstractTreeSearchAgent, h)
        out["receding_horizon"][str(h)] = {"plans": plans, "log": log, "config": config}
    with open(os.path.join(HERE, "golden_host.json"), "w") as f:
        json.dump(out, f)
    print("host done")


if __name__ == "__main__":
    if "--only-highway-vi" in sys.argv:
        highway_vi()
    elif "--only-host" in sys.argv:
        host()
    else:
        main()
        host()
