"""CPU tests: the C ABI library exports what include/b2_planner.h declares, the
spec constants in the CUDA header equal the oracle's fp32 values, and the host
side of the plugin surface (config merge, defaults, allocation, env hand-off,
construction from a `__class__` string) behaves like the reference's."""
import importlib
import os
import re
import sys
import types
from abc import ABC

import numpy as np
import pytest

from oracle import envs as oenvs
from tests.util import load_golden, load_mdps, receding_horizon_schedule

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
M = load_mdps()


def test_library_exports_every_declared_symbol():
    from rl_agents_b200 import _lib, build
    build.build()
    header = open(os.path.join(ROOT, "include", "b2_planner.h")).read()
    declared = set(re.findall(r"\b(b2_[a-z0-9_]+)\s*\(", header))
    assert declared == set(_lib.EXPORTS), declared ^ set(_lib.EXPORTS)
    lib = _lib.load()          # resolves every symbol or raises
    assert lib.b2_version() >= 100
    assert lib.b2_last_error() is not None


def test_missing_library_fails_loudly(monkeypatch):
    from rl_agents_b200 import _lib
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", "/nonexistent/libb2planner.so")
    with pytest.raises(_lib.B2Error):
        _lib.load()


def test_highway_constants_match_the_spec():
    src = open(os.path.join(ROOT, "rl_agents_b200", "csrc", "highway_lite.cuh")).read()
    consts = dict(re.findall(r"HW_CONST\((\w+),\s*(-?0x[0-9a-fA-F.]+p[+-]?\d+)f\)", src))
    assert len(consts) >= 25
    for name, lit in consts.items():
        assert np.float32(float.fromhex(lit)) == getattr(oenvs, name), name
        assert float.fromhex(lit) == float(np.float32(float.fromhex(lit))), name   # exactly an fp32 value

    def poly(fn):
        body = src[src.index("float %s(" % fn):]
        body = body[:body.index("return")]
        return [np.float32(float.fromhex(x)) for x in re.findall(r"(-?0x[0-9a-fA-F.]+p[+-]?\d+)f", body)]
    assert poly("asin_p") == oenvs.ASIN_C[::-1]
    assert poly("sin_p") == oenvs.SIN_C[::-1]
    assert poly("cos_p") == oenvs.COS_C[::-1]


def test_configurable_merges_and_writes_back():
    from rl_agents_b200.configuration import Configurable

    class C(Configurable):
        @classmethod
        def default_config(cls):
            return {"a": 1, "nested": {"x": 1, "y": 2}}
    user = {"nested": {"y": 5}, "extra": "kept"}
    c = C(user)
    assert c.config == {"a": 1, "nested": {"x": 1, "y": 5}, "extra": "kept"}
    assert user == c.config        # configuration.py:12-18: the caller's dict is completed


def test_agent_defaults_match_reference_defaults():
    from rl_agents_b200.agents.tree_search.deterministic import DeterministicPlannerAgent
    from rl_agents_b200.agents.tree_search.mcts import MCTSAgent, allocation
    env = oenvs.FiniteMDPLite(M["large1_T"], M["large1_R"], M["large1_term"])
    a = DeterministicPlannerAgent(env, {})
    assert a.config == {"env_preprocessors": [], "display_tree": False, "receding_horizon": 1, "terminal_reward": 0,
                        "budget": 500, "gamma": 0.8, "step_strategy": "reset"}
    m = MCTSAgent(env, {"unknown_key": 3})
    assert m.config["budget"] == 100 and m.config["temperature"] == 2 / (1 - 0.8) and m.config["closed_loop"] is False
    assert (m.planner.config["episodes"], m.planner.config["horizon"]) == (14, 6) and m.config["unknown_key"] == 3
    for key, (ep, hz) in load_golden("golden_finite.json")["allocation"].items():
        b, g = key.split("_")
        assert allocation(int(b), float(g)) == (ep, hz)
    from rl_agents_b200.agents.tree_search.olop import OLOPAgent
    o = OLOPAgent(env, {"budget": 500, "gamma": 0.7})
    assert (o.planner.config["episodes"], o.planner.config["horizon"]) == (72, 6)
    assert o.config["upper_bound"] == {"type": "hoeffding", "time": "global", "threshold": "4*np.log(time)"}
    assert o.config["continuation_type"] == "zeros"
    assert a.save("x") is False and a.load("x") is False and a.seed(3) == [3]
    with pytest.raises(ValueError):
        MCTSAgent(env, {"rollout_policy": {"type": "nope"}})


def test_reference_defaults_and_factory_accept_the_drop_in(monkeypatch):
    """Our agents, built from a `__class__` string the way the reference's loader does it (factory.py:12-27: import
    the module, take the class, call it with (env, config)), complete their configs to what the reference agents
    complete them to (tests/golden/golden_host.json), and register as virtual subclasses of the reference's
    AbstractAgent (an ABC) when that package is loaded in the process."""
    class RefAbstractAgent(ABC):
        pass
    ref_abstract = types.ModuleType("rl_agents.agents.common.abstract")
    ref_abstract.AbstractAgent = RefAbstractAgent
    monkeypatch.setitem(sys.modules, "rl_agents.agents.common.abstract", ref_abstract)
    env = oenvs.FiniteMDPLite(M["large1_T"], M["large1_R"], M["large1_term"])
    for case in load_golden("golden_host.json")["factory"]:
        cfg = dict(case["config_in"], __class__="<class '%s'>" % case["class"])
        module, name = re.fullmatch(r"<class '(.+)\.(\w+)'>", cfg["__class__"]).groups()
        mine = getattr(importlib.import_module(module), name)(env, cfg)
        theirs = case["config"]
        ours = {k: v for k, v in mine.config.items() if k != "__class__"}
        assert ours == theirs
        assert isinstance(mine, RefAbstractAgent)
        assert mine.config.get("gamma", 1) == theirs["gamma"]     # evaluation.py:327 reads it


def test_env_adapters():
    from rl_agents_b200.envs import FiniteMDPEnv, HighwayLiteEnv
    from rl_agents_b200.envs.adapters import describe
    from rl_agents_b200.envs.highway_lite import available_actions, make_scene
    from rl_agents_b200 import _lib
    fe = FiniteMDPEnv(M["large1_T"], M["large1_R"], M["large1_term"], state=7)
    d = describe(fe)
    assert (d.kind, d.n_actions, d.root.tolist()) == (_lib.ENV_FINITE, 5, [7])
    d2 = describe(oenvs.FiniteMDPLite(M["large1_T"], M["large1_R"], M["large1_term"], state=3))   # duck-typed .mdp
    assert d2.root.tolist() == [3]
    he = HighwayLiteEnv(seed=4)
    d3 = describe(he.simplify())
    assert d3.kind == _lib.ENV_HIGHWAY and d3.root.tolist() == oenvs.make_highway_state(4).pack().tolist()
    for seed in range(20):
        assert available_actions(make_scene(seed)) == oenvs.highway_available_actions(oenvs.make_highway_state(seed))
    with pytest.raises(TypeError):
        class Weird(object):
            action_space = fe.action_space
            unwrapped = property(lambda self: self)
        describe(Weird())


def test_finite_env_steps_like_the_oracle_env():
    from rl_agents_b200.envs import FiniteMDPEnv
    a = FiniteMDPEnv(M["large1_T"], M["large1_R"], M["large1_term"])
    b = oenvs.FiniteMDPLite(M["large1_T"], M["large1_R"], M["large1_term"])
    rng = np.random.default_rng(0)
    for _ in range(50):
        act = int(rng.integers(5))
        assert a.step(act) == b.step(act)


@pytest.mark.parametrize("receding_horizon", [1, 2, 3, 5])
def test_receding_horizon_schedule_matches_the_reference_agent(receding_horizon):
    """The agent shell (own implementation) against the reference's AbstractTreeSearchAgent driven by the
    same scripted planner (tests/golden/golden_host.json): identical plan() outputs, planner calls and
    step_tree arguments."""
    from rl_agents_b200.agents.tree_search.abstract import AbstractTreeSearchAgent
    ours = receding_horizon_schedule(AbstractTreeSearchAgent, receding_horizon)
    ref = load_golden("golden_host.json")["receding_horizon"][str(receding_horizon)]
    assert ours[0] == ref["plans"] and ours[1] == ref["log"]
    assert ours[2] == ref["config"]


def test_preprocess_env_applies_methods_in_sequence():
    from rl_agents_b200.agents.common.factory import _apply, preprocess_env

    class E(object):
        def __init__(self, tag=""):
            self.tag = tag
        unwrapped = property(lambda self: self)

        def simplify(self):
            return E(self.tag + "s")

        def change(self, args):
            return E(self.tag + "c%d" % args)

    out = preprocess_env(E(), [{"method": "simplify"}, {"method": "change", "args": 3}, {"method": "missing"}, {"args": 1}])
    assert out.tag == "sc3"
    assert _apply(E("x"), {"method": "nope"}).tag == "x"


def _fake_highway_env(n_others=20, crashed_slot=None):
    """An object with the attribute names of upstream highway-env's HighwayEnv (the package itself is absent)."""
    class V(object):
        pass

    class Road(object):
        pass

    class Env(object):
        unwrapped = property(lambda self: self)
    rng = np.random.default_rng(1)
    env, road = Env(), Road()
    ego = V()
    ego.position, ego.heading, ego.speed, ego.crashed = np.array([103.5, 8.0]), 0.01, 25.0, False
    ego.lane_index, ego.target_lane_index = ("0", "1", 2), ("0", "1", 1)
    ego.target_speeds, ego.speed_index, ego.target_speed = np.array([20.0, 25.0, 30.0]), 1, 25.0
    vehicles = [ego]
    for k in range(n_others):
        v = V()
        lane = int(rng.integers(0, 4))
        v.position = np.array([103.5 + (k + 1) * 11.0 * (-1) ** k, 4.0 * lane])
        v.heading, v.speed, v.crashed = 0.0, 21.0 + k * 0.1, k == crashed_slot
        v.lane_index = v.target_lane_index = ("0", "1", lane)
        v.target_speed, v.timer = 22.0, 0.25
        vehicles.append(v)
    road.vehicles = vehicles[1:4] + [ego] + vehicles[4:]          # the ego is not first in the upstream list either
    env.road, env.vehicle = road, ego
    env.config = {"lanes_count": 4, "duration": 40, "policy_frequency": 1, "action": {"type": "DiscreteMetaAction"}}
    env.steps = 7

    class Space(object):
        n = 5
    env.action_space = Space()
    return env, vehicles


def test_live_highway_env_object_is_packed_into_a_highway_lite_scene():
    from rl_agents_b200 import _lib
    from rl_agents_b200.envs.adapters import describe
    env, vehicles = _fake_highway_env(n_others=20, crashed_slot=2)
    d = describe(env)
    assert d.kind == _lib.ENV_HIGHWAY and d.n_actions == 5 and d.root.shape == (136,) and d.root.dtype == np.int32
    f = d.root[:96].view(np.float32)
    # slot 0 is the ego; the 15 nearest others follow by |dx|
    assert f[0] == np.float32(103.5) and f[16] == np.float32(8.0) and f[32] == np.float32(0.01) and f[48] == 25.0
    assert d.root[96] == 1 and d.root[129] == 1 and d.root[128] == 7          # target lane, speed index, step
    order = sorted(vehicles[1:], key=lambda v: abs(v.position[0] - 103.5))[:15]
    assert [float(x) for x in f[1:16]] == [float(np.float32(v.position[0])) for v in order]
    assert [int(x) for x in d.root[112:128]] == [1] + [3 if v.crashed else 1 for v in order]
    assert all(np.float32(v.timer) == f[80 + 1 + i] for i, v in enumerate(order))
    # a scene with fewer vehicles leaves the remaining slots absent
    env2, _ = _fake_highway_env(n_others=6)
    assert describe(env2).root[112:128].tolist() == [1] * 7 + [0] * 9
    # unsupported variants are refused loudly, not approximated silently
    env2.config["lanes_count"] = 3
    with pytest.raises(TypeError):
        describe(env2)


def test_intersection_constants_match_the_spec():
    from oracle import intersection as oit
    src = open(os.path.join(ROOT, "rl_agents_b200", "csrc", "intersection_lite.cuh")).read()
    consts = dict(re.findall(r"IL_CONST\((\w+),\s*(-?0x[0-9a-fA-F.]+p[+-]?\d+)f\)", src))
    assert len(consts) >= 20
    expect = {"DT": oit.DT, "KP_A": oit.KP_A, "APPROACH": oit.APPROACH, "ARC_LEFT": oit.ARC_LEFT, "ARC_RIGHT": oit.ARC_RIGHT,
              "LEN_LEFT": oit.LEN[0], "LEN_STRAIGHT": oit.LEN[1], "LEN_RIGHT": oit.LEN[2],
              "PRIO_END_LEFT": (oit.APPROACH + oit.BOX[0]) + oit.PRIO_PAST,
              "PRIO_END_STRAIGHT": (oit.APPROACH + oit.BOX[1]) + oit.PRIO_PAST,
              "PRIO_END_RIGHT": (oit.APPROACH + oit.BOX[2]) + oit.PRIO_PAST, "LENGTH": oit.LENGTH, "HIT_D2": oit.HIT_D2,
              "ACC_MAX": oit.ACC_MAX, "OTHER_TS": oit.OTHER_TS, "STOP_LINE": oit.STOP_LINE, "YIELD_FROM": oit.YIELD_FROM,
              "PRIO_FROM": oit.PRIO_FROM, "ENTRY_CLEAR": oit.ENTRY_CLEAR, "SPAWN_SPEED": oit.SPAWN_SPEED,
              "SPEED_STEP": oit.SPEED_STEP}
    for name, lit in consts.items():
        assert np.float32(float.fromhex(lit)) == np.float32(expect[name]), name
