#!/usr/bin/env python
"""Headline benchmark: OPD leaf-expansions/sec on HighwayLite (highway-v0 stand-in).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA engine
    python bench.py --impl reference --gpus N --steps K ...  # CPU arm (oracle port of the reference)

Workload (BASELINE.json configs[1], C2): DeterministicPlannerAgent / OPD, budget
10 000 (=> 2 000 expand() calls per decision), gamma 0.8, on a batch of
`--trees` independent decisions (seeded scenes) per GPU -- eight search trees per
CTA, strict best-first order inside every tree (bit-exact with the reference).
A "step" is one plan() of the whole batch.  `value` = expand() calls per second
over all GPUs with the root scenes resident in HBM; `e2e` = the same through
the host-buffer path (pinned host scenes -> H2D -> search -> D2H of plans and
per-tree results) every step.  One JSON line on stdout (rank 0).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BUDGET = 10000
GAMMA = 0.8
C2_WORKLOAD = ("C2: DeterministicPlannerAgent (OPD) plan() on HighwayLite (highway-v0 stand-in, 16 vehicles, "
               "15 sub-steps/step), budget %d, gamma %g")
N_ACTIONS = 5
STATE_BYTES = 136 * 4
NODE_BYTES = 5 * 4 + 3 * 8          # parent, first_child, depth, count, meta + reward, lower, upper


def bench_config(a):
    """`config` of the JSON line: identical for the GPU arm and the --impl reference arm."""
    return {"workload": C2_WORKLOAD % (a.budget, a.gamma), "budget": a.budget, "gamma": a.gamma,
            "env": "HighwayLite", "n_actions": N_ACTIONS, "expansions_per_plan": a.budget // N_ACTIONS,
            "unit_of_work": "DeterministicNode.expand() calls (deterministic.py:28-43), strict best-first per tree",
            "l2": "GPU arm: thousands of independent decisions per step, tree arenas >> 126 MB L2 (no flush needed)"}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--trees", type=int, default=0, help="decisions per GPU per step (default 128 per SM, capped by free HBM)")
    ap.add_argument("--budget", type=int, default=BUDGET)
    ap.add_argument("--gamma", type=float, default=GAMMA)
    ap.add_argument("--keys-in-smem", type=int, default=0)
    ap.add_argument("--kernel", type=int, default=0, help="OPD batch kernel variant (b2_opd_config.reserved)")
    ap.add_argument("--cpu-box", type=float, default=20.0, help="time box (s) of the single-core CPU sample")
    ap.add_argument("--ref-plans", type=int, default=2, help="--impl reference: whole plan()s per process in the timed steps")
    ap.add_argument("--ref-time-box", type=float, default=420.0, help="--impl reference: stop after this many seconds")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--headline-only", action="store_true", help="skip the auxiliary paths (VI C4, MCTS C3, one-decision latency)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed as DIR/<name>.npy "
                                                          "(GPU arm, rank 0; see dump_outputs)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    return a


# ----------------------------------------------------------------------------
# clocks: sample nvidia-smi during the timed region
# ----------------------------------------------------------------------------
class ClockSampler(object):
    QUERY = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.samples, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.QUERY,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            parts = [p.strip() for p in s.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0]))
                mx = float(parts[1])
            except ValueError:
                continue
            for n, v in zip(names, parts[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ----------------------------------------------------------------------------
# CPU arm: the oracle port of the reference's plan() (reference/oracle is pure Python)
# ----------------------------------------------------------------------------
def usable_cores():
    """Host threads this process may really use: the affinity mask capped by the cgroup CPU quota
    (os.cpu_count() reports the machine, not the lease)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    quota = None
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:                       # cgroup v2
            q, period = f.read().split()[:2]
            if q != "max":
                quota = float(q) / float(period)
    except Exception:
        try:
            with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as f:      # cgroup v1
                q = float(f.read())
            with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f:
                period = float(f.read())
            if q > 0:
                quota = q / period
        except Exception:
            pass
    if quota is not None:
        n = min(n, max(1, int(quota + 0.5)))
    return max(1, n)


def _spin(seconds):
    """busy loop; returns iterations per second (probe of the cores that really run in parallel)."""
    t0 = time.perf_counter()
    n = 0
    x = 0
    while time.perf_counter() - t0 < seconds:
        for _ in range(20000):
            x += 1
        n += 1
    return n / (time.perf_counter() - t0)


def effective_workers(cores):
    """`cores` processes spinning together vs one alone: leases that advertise more threads than they
    schedule show up as a per-process slowdown; the pool is sized to what runs in parallel."""
    import multiprocessing as mp
    if cores <= 1:
        return 1
    solo = _spin(0.3)
    with mp.Pool(cores) as pool:
        pool.map(_spin, [0.05] * cores)
        rates = pool.map(_spin, [0.5] * cores)
    par = sum(rates) / solo
    return max(1, min(cores, int(par + 0.5)))


class _Stop(Exception):
    pass


def cpu_baseline(budget, gamma, box_s=20.0):
    """The oracle port's plan() (single core, as the reference planner is single-threaded Python) at the
    bench budget, time-boxed: expand() calls completed in `box_s` seconds of one plan()."""
    import numpy as np
    from oracle import envs as oenvs
    from oracle import planners
    st = {"n": 0, "t0": 0.0, "dt": 0.0}

    def tick():
        st["n"] += 1
        st["dt"] = time.perf_counter() - st["t0"]
        if st["dt"] > box_s:
            raise _Stop()

    env = oenvs.HighwayLite(seed=0)
    st["t0"] = time.perf_counter()
    try:
        planners.opd_plan(env, budget, gamma, np_random=np.random.Generator(np.random.PCG64(np.random.SeedSequence(0))),
                          on_expansion=tick)
        done = "whole plan()"
    except _Stop:
        done = "first %d of %d expansions (time box %.0f s; later expansions are slower: the frontier scan is O(n))" \
               % (st["n"], budget // N_ACTIONS, box_s)
    return {"value": st["n"] / st["dt"], "unit": "expansions/s", "cores": 1, "kind": "port",
            "sample": "oracle.planners.opd_plan on HighwayLite seed 0, budget %d: %s, %.1f s" % (budget, done, st["dt"])}


def cpu_port_c(budget, gamma, cores=None):
    """The C restatement (oracle/c: same spec, literal O(V^2) scans, heap frontier) on one core and on all
    usable host threads -- what an optimised CPU implementation of the same path does, next to the Python port."""
    from concurrent.futures import ThreadPoolExecutor
    from oracle import c_oracle
    from oracle import envs as oenvs
    cores = cores or usable_cores()
    scenes = [oenvs.make_highway_state(s).pack() for s in range(4 * cores)]
    c_oracle.opd_plan(scenes[0], 500, gamma)
    t0 = time.perf_counter()
    c_oracle.opd_plan(scenes[0], budget, gamma)
    single = (budget // N_ACTIONS) / (time.perf_counter() - t0)
    t0 = time.perf_counter()
    with ThreadPoolExecutor(cores) as ex:
        list(ex.map(lambda w: c_oracle.opd_plan(w, budget, gamma), scenes))
    multi = len(scenes) * (budget // N_ACTIONS) / (time.perf_counter() - t0)
    return {"value": multi, "unit": "expansions/s", "cores": cores, "os_cpu_count": os.cpu_count(),
            "single_core_value": single, "kind": "port",
            "sample": "oracle/c OPD, HighwayLite, budget %d (full C2 budget): 1 plan() on one core; %d plan()s on %d threads"
                      % (budget, len(scenes), cores)}


def _ref_worker(conn, rank, budget, gamma, bounds):
    """One reference-arm process: runs budget-`budget` plan()s of the oracle port back to back and stops at
    the cumulative expansion counts in `bounds` (a step boundary) until the parent says go."""
    import numpy as np
    from oracle import envs as oenvs
    from oracle import planners
    st = {"n": 0, "k": 0, "plans": [], "t_plan": 0.0}

    n_exp = budget // N_ACTIONS

    def tick():
        st["n"] += 1
        if st["n"] % n_exp == 0:            # a whole plan() is done (its greedy get_plan is negligible)
            now = time.perf_counter()
            st["plans"].append(now - st["t_plan"])
            st["t_plan"] = now
        if st["k"] < len(bounds) and st["n"] >= bounds[st["k"]]:
            st["k"] += 1
            conn.send(("step", st["n"], list(st["plans"])))
            if conn.recv() != "go":
                raise _Stop()

    try:
        if conn.recv() != "go":
            return
        seed = rank
        while st["k"] < len(bounds):
            st["t_plan"] = time.perf_counter()
            planners.opd_plan(oenvs.HighwayLite(seed=seed), budget, gamma,
                              np_random=np.random.Generator(np.random.PCG64(np.random.SeedSequence(0))),
                              on_expansion=tick)
            seed += 1000
    except _Stop:
        pass
    finally:
        conn.close()


def run_reference(a):
    """--impl reference: the oracle port of the reference's plan() (Python, like the reference) on every
    host core this lease really schedules, at the SAME budget / gamma / env as the GPU arm.  A step is a
    bounded slice of the workers' plan()s: the K timed steps cover exactly `plans_per_worker` whole
    plan()s per worker, the W warm-up steps the first part of a discarded plan()."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    os.environ.setdefault("OMP_NUM_THREADS", "1")
    cores = usable_cores()
    workers = effective_workers(cores)
    n_exp = a.budget // N_ACTIONS
    steps, warmup = max(a.steps, 1), max(a.warmup, 0)
    # size: the port does ~40-55 expand()/s per core at this budget => one plan() ~ 40-50 s
    plans_per_worker = max(1, int(a.ref_plans))
    timed = [int(round((k + 1) * plans_per_worker * n_exp / float(steps))) for k in range(steps)]
    warm_slice = max(1, min(n_exp // max(warmup, 1), 40))
    ctx = mp.get_context("fork")

    def launch(bounds):
        procs = []
        for w in range(workers):
            pc, cc = ctx.Pipe()
            p = ctx.Process(target=_ref_worker, args=(cc, w, a.budget, a.gamma, bounds), daemon=True)
            p.start()
            cc.close()
            procs.append((p, pc))
        return procs

    def stop(procs):
        for p, pc in procs:
            try:
                pc.send("stop")
            except Exception:
                pass
        for p, pc in procs:
            p.join(2.0)
            if p.is_alive():
                p.terminate()

    # warm-up: W short slices of a plan() that is then discarded (imports, allocator, caches)
    if warmup:
        procs = launch([warm_slice * (k + 1) for k in range(warmup)])
        for _ in range(warmup):
            for p, pc in procs:
                pc.send("go")
            for p, pc in procs:
                pc.recv()
        stop(procs)
    procs = launch(timed)
    t_box = float(a.ref_time_box)
    done_steps, plan_times, total = 0, [], 0
    t0 = time.perf_counter()
    for k in range(steps):
        for p, pc in procs:
            pc.send("go")
        counts = []
        for p, pc in procs:
            _, n, plans = pc.recv()
            counts.append(n)
            if k == steps - 1:
                plan_times.extend(plans)
        done_steps, total = k + 1, sum(counts)
        dt = time.perf_counter() - t0
        if dt > t_box and k + 1 < steps:
            for p, pc in procs:
                try:
                    pc.send("go")
                    _, _, plans = pc.recv()
                except Exception:
                    plans = []
            break
    dt = time.perf_counter() - t0
    stop(procs)
    value = total / dt
    plan_times.sort()
    med = plan_times[len(plan_times) // 2] if plan_times else None
    sample = ("%d processes (usable cores %d, os.cpu_count %d), each running whole plan()s of the oracle port "
              "(oracle.planners.opd_plan = the reference's algorithm in Python, HighwayLite) at budget %d (%d expand() "
              "each) back to back; %d of %d timed steps done = %d expansions in %.1f s; 1 step = 1/%d of %d plan()s per "
              "process" % (workers, cores, os.cpu_count() or 0, a.budget, n_exp, done_steps, steps, total, dt, steps,
                           plans_per_worker))
    emit({
        "impl": "reference", "metric": "OPD leaf-expansions/sec on highway-v0 (HighwayLite)", "value": value,
        "unit": "expansions/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "steps_done": done_steps,
        "ms_per_step": 1e3 * dt / max(done_steps, 1), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": bench_config(a),
        "cpu_baseline": {"value": value, "unit": "expansions/s", "cores": workers, "kind": "port", "sample": sample,
                         "single_process_median_plan_s": med,
                         "single_process_value": (n_exp / med) if med else None,
                         "plans_timed": len(plan_times)},
        "e2e": {"value": value, "unit": "expansions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0})


# ----------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------
def run_b200(a):
    import numpy as np
    import torch
    import torch.distributed as dist
    from rl_agents_b200 import _lib
    from rl_agents_b200.engine.opd import OPDEngine
    from rl_agents_b200.envs.highway_lite import make_scene

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    n_exp = a.budget // N_ACTIONS
    if a.trees:
        trees = a.trees
    else:
        # default batch: 128 decisions per SM (more work in flight = better overlap of the trees' phases),
        # capped so that the tree arena (scene + node record + frontier key per node) takes <= 65 % of the HBM;
        # of the whole HBM, not of what is free at the moment, so that the same arguments give the same inputs
        per_tree = (1 + n_exp * N_ACTIONS) * (STATE_BYTES + NODE_BYTES + 8) + 16 * 1024
        total = torch.cuda.get_device_properties(dev).total_memory
        trees = min(128 * sms, int(0.65 * total / per_tree))
        trees = max(8 * sms, trees // (8 * sms) * (8 * sms))

    eng = OPDEngine(_lib.ENV_HIGHWAY, trees, N_ACTIONS, a.budget, a.gamma, keys_in_smem=bool(a.keys_in_smem),
                    device=dev, kernel=a.kernel)
    # independent decisions: every (rank, tree) its own seeded scene; two alternating input sets
    host_scenes = [torch.from_numpy(np.stack([make_scene(1_000_000 * s + rank * trees + i) for i in range(trees)]))
                   .pin_memory() for s in range(2)]
    dev_scenes = [h.to(dev) for h in host_scenes]
    stream = torch.cuda.current_stream()

    per_rank_ms = []

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for k in range(steps):
            fn(k)
        e1.record(stream)
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            every = torch.empty(world, dtype=torch.float64, device=dev)
            dist.all_gather_into_tensor(every, ms)
            per_rank_ms[:] = every.cpu().tolist()
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        else:
            per_rank_ms[:] = [float(ms.item())]
        barrier()
        return float(ms.item())

    def device_step(k):
        eng.plan(dev_scenes[k & 1])

    for k in range(max(a.warmup, 3)):
        device_step(k)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms = timed(device_step, a.steps)
    clocks = sampler.stop() if rank == 0 else None
    headline_per_rank = {"min_ms": min(per_rank_ms) / a.steps, "mean_ms": sum(per_rank_ms) / len(per_rank_ms) / a.steps,
                         "max_ms": max(per_rank_ms) / a.steps, "per_rank_ms_per_step": [x / a.steps for x in per_rank_ms]}
    # sanity: the timed work really is the full search
    res = eng.result.cpu().numpy()
    assert (res[:, 0] > n_exp).all() and (res[:, 4] == 0).all()
    if a.dump_outputs and rank == 0:
        dump_outputs(eng, res, a.dump_outputs)
    mean_children = float((res[:, 0] - 1).mean() / n_exp)
    # ---- e2e: the host-buffer C ABI (b2_opd_create / b2_opd_plan_host): pinned host scenes -> H2D -> search
    #      -> D2H of plans and per-tree results, synchronous, every step ----
    import ctypes
    capacity, plan_capacity = eng.capacity, eng.plan_capacity
    del eng
    torch.cuda.empty_cache()
    hc = _lib.OPDHostConfig(_lib.ENV_HIGHWAY, trees, N_ACTIONS, a.budget, int(a.keys_in_smem), a.kernel, a.gamma, 0.0,
                            _lib.FiniteMDP())
    handle = ctypes.c_void_p()
    _lib.check(lib.b2_opd_create(ctypes.byref(hc), ctypes.byref(handle)))
    plan_host = torch.empty((trees, plan_capacity), dtype=torch.int8).pin_memory()
    res_host = torch.empty((trees, _lib.OPD_RESULT_WORDS), dtype=torch.int32).pin_memory()

    def e2e_step(k):
        _lib.check(lib.b2_opd_plan_host(handle, ctypes.c_void_p(host_scenes[k & 1].data_ptr()),
                                        ctypes.c_void_p(plan_host.data_ptr()), ctypes.c_void_p(res_host.data_ptr())))

    for k in range(2):
        e2e_step(k)
    barrier()
    t0 = time.perf_counter()
    for k in range(a.steps):
        e2e_step(k)
    t_e2e = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_e2e, op=dist.ReduceOp.MAX)
    ms_e2e = float(t_e2e.item()) * 1e3
    assert (res_host.numpy()[:, 0] > n_exp).all() and (res_host.numpy()[:, 4] == 0).all()
    lib.b2_opd_destroy(handle)
    total_exp = float(world) * trees * n_exp * a.steps
    value = total_exp / (ms * 1e-3)
    e2e_value = total_exp / (ms_e2e * 1e-3)
    # roofline of the dominant (only) kernel, opd_highway_kernel: algorithmic HBM bytes per expand()
    # = parent scene read + children scenes written + node records + keys + bottom-up pass (DESIGN.md section 4)
    bytes_per_exp = STATE_BYTES * (1.0 + mean_children) + mean_children * (NODE_BYTES + 8 + 20) + 24
    launch_ms = ms / a.steps
    achieved = trees * n_exp * bytes_per_exp / (launch_ms * 1e-3) / 1e9
    peak, peak_src = 6650.0, "fallback"
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peak, peak_src = float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        pass
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "opd_highway_traffic.json")) as f:
            tr = json.load(f)
        if tr.get("trees") == trees and tr.get("budget") == a.budget:
            traffic = tr["dram_bytes_per_launch"]
    except Exception:
        pass

    ncu = None      # static evidence from the committed ncu capture of this kernel (not measured in this run)
    for name in ("r02d_opd_multi_ncu_summary.json", "r02b_opd_multi_ncu_summary.json", "r01_opd_highway_multi_ncu_summary.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as f:
                summ = json.load(f)
            summ = summ.get("opd_highway_multi_kernel", summ)      # newer summaries are keyed by kernel name
            inst = float(summ["smsp__inst_executed.sum"][0]) if "smsp__inst_executed.sum" in summ else None
            ncu = {"source": "profiles/" + name,
                   "ipc_per_sm": float(summ["sm__inst_executed.avg.per_cycle_elapsed"][0]),
                   "issue_slots_busy_pct": float(summ["smsp__issue_active.avg.pct_of_peak_sustained_active"][0]),
                   "alu_pipe_pct": float(summ["sm__inst_executed_pipe_alu.avg.pct_of_peak_sustained_active"][0]),
                   "fma_pipe_pct": float(summ["sm__inst_executed_pipe_fma.avg.pct_of_peak_sustained_active"][0]),
                   "dram_pct": float(summ["gpu__dram_throughput.avg.pct_of_peak_sustained_elapsed"][0]),
                   "warp_instructions_in_capture": inst}
            break
        except Exception:
            continue
    out = {
        "metric": "OPD leaf-expansions/sec on highway-v0 (HighwayLite)", "value": value, "unit": "expansions/s",
        "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3), "ms_per_step": ms / a.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": bench_config(a),
        "run_config": {"trees_per_gpu": trees, "expansions_per_tree": n_exp,
                       "mean_children_per_expansion": mean_children, "child_nodes_per_s": value * mean_children,
                       "l2": "working set %.1f GB per step >> 126 MB L2 (no flush needed)"
                             % (trees * capacity * (STATE_BYTES + NODE_BYTES) / 1e9),
                       "parallelism": "trees sharded over %d GPU(s), no data-path collective" % world,
                       "keys_in_smem": bool(a.keys_in_smem)},
        "e2e": {"value": e2e_value, "unit": "expansions/s", "h2d_bytes_per_step": int(trees * STATE_BYTES),
                "d2h_bytes_per_step": int(plan_host.numel() + res_host.numel() * 4), "ms_per_step": ms_e2e / a.steps,
                "path": "b2_opd_plan_host (C ABI, host buffers, synchronous); wall clock over the steps, max over ranks"},
        "gpu_launches": a.steps,
        "per_rank": headline_per_rank,
        "clocks": clocks,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "peak_source": peak_src, "kernel": "opd_highway_multi_kernel",
                     "bytes_per_expansion": bytes_per_exp, "limiter": "instruction issue (see ncu)", "ncu": ncu,
                     "note": "latency/FP32-issue bound by construction (15 dependent sub-steps per child); "
                             "HBM fraction reported as the contract asks, see DESIGN.md section 4"},
    }
    if not a.headline_only:
        try:
            extra = other_paths(a, dev, world, rank)           # collective calls inside: every rank takes part
        except Exception as e:
            extra = {"error": repr(e)[:300]}
        out["other_paths"] = extra
    if rank == 0 and not a.headline_only:
        try:
            out["single_decision"] = single_decision_latency(a, dev)
        except Exception as e:          # an auxiliary measurement must never take the headline down
            out["single_decision"] = {"error": str(e)[:300]}
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        out["cpu_baseline"] = cpu_baseline(a.budget, a.gamma, a.cpu_box)
        try:
            out["cpu_port_c"] = cpu_port_c(a.budget, a.gamma)
        except Exception as e:      # the C oracle is optional test infrastructure
            out["cpu_port_c"] = {"unavailable": str(e)[:200]}
    if rank == 0:
        emit(out)
    if world > 1:
        dist.destroy_process_group()


DUMP_LIMIT_BYTES = 64 << 20
DUMP_TREES = 32         # seeded sample of the batch whose whole node arrays are written
DUMP_NODES = 64         # seeded sample of node ids whose scene words are written


def dump_outputs(eng, res, directory):
    """--dump-outputs: what the last timed b2_opd_plan() handed to its caller, one .npy file per array.

    Every tree: `result` [trees, 7] (n_nodes, n_leaves, max_depth, terminal_expansions, error, plan_len, tie_node)
    and `plan`, the trees' plans (plan_len actions each) one after the other.  A seeded sample of trees
    (`sample_trees`): their node arrays (n_nodes entries each, one tree after the other), and the scene words
    `state` [sample, nodes, 136] of a seeded sample of node ids (`sample_nodes`, all below n_expansions + 1, so
    present in every tree).  Entries past a tree's n_nodes or plan_len are left out: the search does not write
    them, they hold whatever the buffers held before.  Integer outputs are float32 (exact: all are below 2**24), scene words
    float64, reward / lower / upper float64 as computed."""
    import numpy as np
    import torch
    n_nodes, plan_len = res[:, 0], res[:, 5]
    out = {"result": res[:, :7].astype(np.float32)}
    plan = eng.plan_buf[:, :int(plan_len.max())].cpu().numpy()
    out["plan"] = plan[np.arange(plan.shape[1])[None, :] < plan_len[:, None]].astype(np.float32)   # row-major
    rng = np.random.default_rng(0)
    trees = np.sort(rng.choice(eng.n_trees, size=min(DUMP_TREES, eng.n_trees), replace=False))
    nodes = np.sort(rng.choice(eng.n_expansions + 1, size=min(DUMP_NODES, eng.n_expansions + 1), replace=False))
    out["sample_trees"], out["sample_nodes"] = trees.astype(np.float32), nodes.astype(np.float32)
    rows = torch.from_numpy(trees).to(eng.device)
    written = np.arange(eng.capacity)[None, :] < n_nodes[trees][:, None]
    for name in ("parent", "first_child", "depth", "count", "meta", "reward", "lower", "upper"):
        t = getattr(eng, name)
        x = t.index_select(0, rows).cpu().numpy()[written]
        out[name] = x.astype(np.float64 if t.dtype == torch.float64 else np.float32)
    cols = torch.from_numpy(nodes).to(eng.device)
    out["state"] = eng.state[rows[:, None], cols[None, :]].cpu().numpy().astype(np.float64)
    size = sum(x.nbytes for x in out.values())
    if size > DUMP_LIMIT_BYTES:
        raise SystemExit("--dump-outputs: %d bytes exceed the %d-byte limit (use fewer --trees)" % (size, DUMP_LIMIT_BYTES))
    os.makedirs(directory, exist_ok=True)
    for name, x in out.items():
        np.save(os.path.join(directory, name + ".npy"), x)


def other_paths(a, dev, world, rank):
    """The other BASELINE paths through the same launch (driver-visible evidence for SURVEY 8e): C4 value
    iteration slab-sharded over the ranks (the path's one exchange step timed next to the compute), C3 MCTS
    root-parallel with its single [2, A] all-reduce, and one budget-1e6 OPD decision sub-tree sharded.  Every
    time is CUDA events / device-synchronised wall clock, max over ranks."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from rl_agents_b200 import _lib
    from rl_agents_b200 import distributed as D
    from rl_agents_b200.engine.vi import VIEngine
    from rl_agents_b200.envs.finite_mdp import garnet_slab
    from rl_agents_b200.envs.highway_lite import make_scene
    out = {}

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def timed_ms(fn, reps=3):
        best = None
        for _ in range(reps):
            sync()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ms = max_over_ranks(e0.elapsed_time(e1))
            best = ms if best is None else min(best, ms)
        return best

    peak = 6650.0
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peak = float(json.load(f)["hbm_gbs"])
    except Exception:
        pass
    # ---- C4: value iteration, S = 1e6, A = 8, B = 4 sparse, 100 sweeps, early exit off (rtol 0, atol -1) ----
    try:
        S, A, B, sweeps = 1000000, 8, 4, 100
        b, e = D.shard_range(S, rank, world)
        P, N, R, term = garnet_slab(S, A, B, b, e, seed=0, device=dev)
        if world > 1:
            vi = D.DistributedVI("sparse", P, R, term, nxt=N, gamma=0.95, device=dev, tables_are_local=True,
                                 n_states=S, check_every=10, rtol=0.0, atol=-1.0)
            nccl_full = timed_ms(lambda: vi.solve(sweeps))
            comp = timed_ms(lambda: vi.solve(sweeps, exchange=False))
            eng = vi.engine
            p2p_full, p2p_err = None, None
            try:
                vi2 = D.DistributedVI("sparse", P, R, term, nxt=N, gamma=0.95, device=dev, tables_are_local=True,
                                      n_states=S, rtol=0.0, atol=-1.0, exchange="p2p", max_iterations=sweeps)
                p2p_full = timed_ms(lambda: vi2.solve(sweeps))
                vi2.close()
                del vi2
            except Exception as ex:
                p2p_err = repr(ex)[:200]
            full = nccl_full if p2p_full is None else min(nccl_full, p2p_full)
        else:
            eng = VIEngine("sparse", P, R, term, nxt=N, gamma=0.95, device=dev, rtol=0.0, atol=-1.0)
            full = timed_ms(lambda: eng.solve(sweeps))
            comp, nccl_full, p2p_full, p2p_err = full, None, None, None
        algo = float(S * A * B * 20 + S * A * 24 + S * 9)            # whole MDP, bytes per sweep (SURVEY 8d + Q_old)
        # cold-L2 variant on one GPU: alternate between two table sets (2 x 0.8 GB >> 126 MB L2)
        cold = None
        if world == 1:
            P2, N2, R2, term2 = garnet_slab(S, A, B, 0, S, seed=1, device=dev)
            eng2 = VIEngine("sparse", P2, R2, term2, nxt=N2, gamma=0.95, device=dev, rtol=0.0, atol=-1.0)
            eng.reset(sweeps)
            eng2.reset(sweeps)

            def alternate():
                for k in range(sweeps // 2):
                    eng.sweep(k)
                    eng2.sweep(k)
            cold = timed_ms(alternate)
            del eng2, P2, N2, R2
        out["vi_c4"] = {
            "workload": "C4: Bellman sweeps, garnet sparse MDP S=1e6 A=8 B=4 fp64/int32, gamma 0.95, %d sweeps, "
                        "early exit off, state slabs over %d GPU(s)" % (sweeps, world),
            "sweeps_per_s": sweeps / (full * 1e-3), "us_per_sweep": 1e3 * full / sweeps,
            "us_per_sweep_compute_only": 1e3 * comp / sweeps,
            "us_per_sweep_exchange": 1e3 * (full - comp) / sweeps,
            "exchange": None if world == 1 else {
                "nccl_us_per_sweep": 1e3 * nccl_full / sweeps,
                "nccl": "sweep kernel, then all_gather of the V slabs (%.1f MB per rank) every sweep + all_reduce of "
                        "10 violation counters every 10 sweeps" % (8.0 * S / world / 1e6),
                "p2p_us_per_sweep": None if p2p_full is None else 1e3 * p2p_full / sweeps,
                "p2p": "b2_vi_sweep_p2p: V' stored into every rank's copy over NVLink inside the sweep kernel, "
                       "violation counts + arrival flags published by the last CTA; no collective call, exact "
                       "per-sweep early-exit protocol" if p2p_err is None else "failed: " + p2p_err,
                "used_for_us_per_sweep": "p2p" if (p2p_full is not None and p2p_full <= nccl_full) else "nccl"},
            "roofline": {"bound": "hbm", "achieved": algo / (full * 1e-3 / sweeps) / 1e9, "peak": peak * world,
                         "unit": "GB/s", "frac": algo / (full * 1e-3 / sweeps) / 1e9 / (peak * world),
                         "algorithmic_bytes_per_sweep": algo, "kernel": "vi_sweep_row_kernel<4,true>"},
            "cold_l2_us_per_sweep": None if cold is None else 1e3 * cold / (2 * (sweeps // 2)),
            "cold_l2_frac": None if cold is None else algo / (cold * 1e-3 / (2 * (sweeps // 2))) / 1e9 / peak}
        del eng, P, N, R
        torch.cuda.empty_cache()
    except Exception as ex:
        out["vi_c4"] = {"error": repr(ex)[:300]}
    # ---- C1: dense stochastic VI, S = 100, A = 4 (the reference's CPU-runnable case): launch-latency bound ----
    try:
        g = torch.Generator(device=dev)
        g.manual_seed(0)
        P1 = torch.rand((100, 4, 100), dtype=torch.float64, device=dev, generator=g)
        P1 = P1 / P1.sum(dim=-1, keepdim=True)
        R1 = torch.rand((100, 4), dtype=torch.float64, device=dev, generator=g)
        e1 = VIEngine("stochastic", P1, R1, torch.zeros(100, dtype=torch.uint8, device=dev), gamma=0.95, device=dev,
                      rtol=0.0, atol=-1.0)
        ms = timed_ms(lambda: e1.solve(100))
        bytes1 = 100 * 4 * 100 * 8 + 100 * 4 * 24 + 100 * 9
        out["vi_c1"] = {"workload": "C1: dense VI S=100 A=4 fp64, 100 sweeps enqueued back to back (b2_vi_solve)",
                        "us_per_sweep": 1e3 * ms / 100,
                        "roofline": {"bound": "hbm", "achieved": bytes1 / (ms * 1e-3 / 100) / 1e9, "peak": peak, "unit": "GB/s",
                                     "frac": bytes1 / (ms * 1e-3 / 100) / 1e9 / peak, "algorithmic_bytes_per_sweep": bytes1,
                                     "note": "0.32 MB per sweep lives in L2; the sweep is bound by kernel launch latency"}}
    except Exception as ex:
        out["vi_c1"] = {"error": repr(ex)[:300]}
    # ---- C3: MCTS 4096 episodes x horizon 20, root-parallel: 64 trees of 64 episodes over all ranks ----
    try:
        from rl_agents_b200.engine.mcts import MCTSEngine, pcg64_words
        total_trees, episodes, horizon = 64, 64, 20
        mine = [t for t in range(total_trees) if t % world == rank]
        eng = MCTSEngine(_lib.ENV_HIGHWAY, len(mine), N_ACTIONS, episodes, horizon, 0.8, 10.0, device=dev)
        scene = torch.tensor(make_scene(0), dtype=torch.int32, device=dev)
        roots = scene.repeat(len(mine), 1).contiguous()
        gens = np.random.Generator(np.random.PCG64(np.random.SeedSequence(0))).spawn(total_trees)
        words = np.stack([pcg64_words(gens[t]) for t in mine])
        merged = {}

        def decide(collective=True):
            eng.plan(roots, words)
            fc = eng.first_child[:, 0]
            idx = fc.long().unsqueeze(1) + torch.arange(N_ACTIONS, device=dev).unsqueeze(0)
            nch = (eng.meta[:, 0] >> 8) & 0xff
            valid = torch.arange(N_ACTIONS, device=dev).unsqueeze(0) < nch.unsqueeze(1)
            idx = torch.where(valid, idx, torch.zeros_like(idx))
            acts = (torch.gather(eng.meta, 1, idx) & 0xff).long()
            cnt = torch.where(valid, torch.gather(eng.count, 1, idx), torch.zeros_like(idx, dtype=torch.int32)).double()
            val = torch.where(valid, torch.gather(eng.value, 1, idx), torch.zeros_like(cnt))
            acts = torch.where(valid, acts, torch.zeros_like(acts))
            counts = torch.zeros(N_ACTIONS, dtype=torch.float64, device=dev).scatter_add_(0, acts.reshape(-1), cnt.reshape(-1))
            sums = torch.zeros(N_ACTIONS, dtype=torch.float64, device=dev).scatter_add_(0, acts.reshape(-1), (cnt * val).reshape(-1))
            values = torch.where(counts > 0, sums / counts.clamp(min=1), torch.zeros_like(sums))
            if collective and world > 1:
                counts, values = D.merge_root_statistics(counts, values)
            merged["c"], merged["v"] = counts, values
        comp = timed_ms(lambda: decide(False))
        full = timed_ms(decide)
        c, v = merged["c"].cpu().numpy(), merged["v"].cpu().numpy()
        out["mcts_c3_root_parallel"] = {
            "workload": "C3: MCTS on HighwayLite, 4096 episodes x horizon 20 as 64 root-parallel trees of 64 episodes "
                        "(strict episode order inside each tree), trees dealt over %d GPU(s)" % world,
            "ms_per_decision": full, "ms_compute_only": comp, "ms_collective": full - comp,
            "collective": None if world == 1 else "one all_reduce of the root's [2, A] (count, count*value)",
            "episodes_per_s": 4096 / (full * 1e-3), "env_steps_upper_bound_per_s": 4096 * horizon / (full * 1e-3),
            "recommended_action": int(D.recommend(c, v)), "root_counts": c.tolist()}
        del eng
        torch.cuda.empty_cache()
    except Exception as ex:
        out["mcts_c3_root_parallel"] = {"error": repr(ex)[:300]}
    # ---- C3 as ONE decision searched by the whole GPU (rank 0's GPU; no collective): wavefront MCTS ----
    try:
        from rl_agents_b200.engine.mcts import MCTSWaveEngine
        rows = []
        scene = torch.tensor(make_scene(0), dtype=torch.int32, device=dev)
        for width in (256, 512, 1024):
            eng = MCTSWaveEngine(_lib.ENV_HIGHWAY, N_ACTIONS, 4096, 20, 0.8, 10.0, width, device=dev)
            ms = timed_ms(lambda: eng.plan(scene, 0), reps=5)
            eng.plan(scene, 0)
            plan, res = eng.finish()
            rows.append({"width": width, "ms_per_decision": ms, "episodes_per_s": 4096 / (ms * 1e-3),
                         "env_steps": int(res[2]), "env_steps_per_s": int(res[2]) / (ms * 1e-3), "waves": int(res[3]),
                         "recommended_action": plan[0] if plan else None})
            del eng
        out["mcts_c3_wavefront"] = {
            "workload": "C3: MCTS on HighwayLite, 4096 episodes x horizon 20, ONE tree, waves of `width` episodes "
                        "(b2_mcts_plan_wave; specification oracle/planners.py::mcts_plan_wavefront, bit-exact)",
            "strict_reference_order_ms": "2340 (one sequential chain of 81 920 env steps; profiles/r01_misc_measurements.json)",
            "rows": rows}
        torch.cuda.empty_cache()
    except Exception as ex:
        out["mcts_c3_wavefront"] = {"error": repr(ex)[:300]}
    # ---- C5: ONE OPD decision on IntersectionLite, budget 1e6 (333 333 expansions), gamma 0.9:
    #      the whole tree on one GPU in waves, and sub-tree sharded over the ranks (one all_reduce(MAX)) ----
    try:
        from rl_agents_b200.engine.opd import OPDWaveEngine
        from rl_agents_b200.envs.intersection_lite import make_scene as make_intersection
        rows = []
        sc = torch.tensor(make_intersection(0), dtype=torch.int32, device=dev)
        for width in (1024, 4096):
            eng = OPDWaveEngine(_lib.ENV_INTERSECTION, 3, 1000000, 0.9, width, device=dev)
            ms = timed_ms(lambda: eng.plan(sc), reps=3)
            res = eng.result.cpu().numpy()
            rows.append({"width": width, "ms_per_decision": ms, "expansions_per_s": 333333 / (ms * 1e-3),
                         "waves": int(res[0, 7]), "root_value_lower": float(eng.lower[0, 0].item())})
            del eng
        out["opd_c5_one_gpu_wavefront"] = {
            "workload": "C5: ONE OPD decision on IntersectionLite (the repo's model of intersection-v0), budget 1e6 = "
                        "333 333 expand() calls, gamma 0.9, the whole tree on ONE GPU in waves of `width` leaves "
                        "(every rank runs the same decision; rank 0's time)", "rows": rows}
        torch.cuda.empty_cache()
    except Exception as ex:
        out["opd_c5_one_gpu_wavefront"] = {"error": repr(ex)[:300]}
    try:
        sh = D.ShardedOPD(1000000, 0.9, device=dev, wave_width=1024, env="intersection")
        scene_np = make_intersection(0)
        sync()
        t0 = time.perf_counter()
        r = sh.decide(scene_np)
        torch.cuda.synchronize()
        dt = max_over_ranks(time.perf_counter() - t0)
        sync()
        t0 = time.perf_counter()
        r = sh.decide(scene_np)
        torch.cuda.synchronize()
        dt = min(dt, max_over_ranks(time.perf_counter() - t0))
        out["opd_c5_subtree_sharded"] = {
            "workload": "C5: ONE OPD decision on IntersectionLite, budget 1e6, gamma 0.9, tree-sharded: the root's depth-k "
                        "sub-trees (%d) dealt over %d GPU(s), each searched by its rank's whole GPU in waves of 1024 leaves"
                        % (r["n_subtrees"], world),
            "s_per_decision": dt, "expansions_per_s": 333333 / dt, "action": int(r["action"]),
            "root_lower": float(r["root_lower"]),
            "collective": None if world == 1 else "one all_reduce(MAX) of the [n_subtrees, 2] bounds"}
    except Exception as ex:
        out["opd_c5_subtree_sharded"] = {"error": repr(ex)[:300]}

    # ---- ValueIterationAgent on highway scenes (shipped config: iterations 10, gamma 1): conversion to the TTC-grid
    #      MDP + the agent's fixed point as ONE kernel over a batch of scenes resident in HBM (every rank the same batch;
    #      rank 0's time).  value_iteration.py:29-35 does both on the host at every act(). ----
    try:
        from rl_agents_b200.engine.ttc_vi import HighwayTTCVI
        n_sc = 1 << 18
        base = np.stack([make_scene(s) for s in range(256)])
        scenes = torch.from_numpy(np.tile(base, (n_sc // 256, 1))).to(dev)
        eng = HighwayTTCVI(1.0, 10, device=dev)
        res = {}

        def run_ttc():
            res["out"] = eng.solve(scenes, want_q=False)
        ms = timed_ms(run_ttc, reps=3)
        out["vi_highway_ttc"] = {
            "workload": "ValueIterationAgent.act() on %d HighwayLite scenes: to_finite_mdp() (TTC grid, 120 states x 5 "
                        "actions) + 10 sweeps of the fixed point per scene, fused (b2_highway_ttc_vi, one warp per scene)" % n_sc,
            "ms_per_launch": ms, "decisions_per_s": n_sc / (ms * 1e-3),
            "sweeps_mean": float(res["out"]["sweeps"].float().mean().item()),
            "parity": "Q bit-identical with the unmodified reference agent (tests/test_gpu_ttc_vi.py)"}
        del scenes
    except Exception as ex:
        out["vi_highway_ttc"] = {"error": repr(ex)[:300]}
    return out


def single_decision_latency(a, dev, reps=5):
    """ONE C2 decision (what agent.plan() does under scripts/experiments.py) at a time: the strict one-CTA
    kernel, the speculative strict kernel (b2_opd_plan_spec, same tree) and the wavefront kernel
    (b2_opd_plan_wave) at a few widths, plus one budget-1e6 decision.
    CUDA-event median over `reps` launches per scene; quality of each width against the strict tree
    (root action agreement, gap of the root value_lower) on the same scenes."""
    import numpy as np
    import torch
    from rl_agents_b200 import _lib
    from rl_agents_b200.engine.opd import OPDEngine, OPDSpeculativeEngine, OPDWaveEngine
    from rl_agents_b200.envs.highway_lite import make_scene
    scenes = [torch.tensor(make_scene(s), dtype=torch.int32, device=dev) for s in range(4)]
    n_exp = a.budget // N_ACTIONS

    def med_ms(fn):
        fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        return sorted(ts)[len(ts) // 2]

    rows = []
    eng = OPDEngine(_lib.ENV_HIGHWAY, 1, N_ACTIONS, a.budget, a.gamma, keys_in_smem=True, device=dev)
    ms = float(np.median([med_ms(lambda: eng.plan(s.reshape(1, -1))) for s in scenes]))
    strict = []
    for s in scenes:
        eng.plan(s.reshape(1, -1))
        plans, _ = eng.finish([np.random.default_rng(0)])
        strict.append((plans[0][0], float(eng.lower[0, 0].item())))
    rows.append({"mode": "strict (reference order, one CTA)", "ms": ms, "expansions_per_s": n_exp / (ms * 1e-3)})
    del eng
    # the same strict tree, bit for bit, searched by the whole GPU (b2_opd_plan_spec)
    for width in (64, 256):
        eng = OPDSpeculativeEngine(_lib.ENV_HIGHWAY, N_ACTIONS, a.budget, a.gamma, width, device=dev)
        ms = float(np.median([med_ms(lambda: eng.plan(s)) for s in scenes]))
        same, waves = 0, []
        for s, (act, low) in zip(scenes, strict):
            eng.plan(s)
            plans, res = eng.finish([np.random.default_rng(0)])
            same += int(plans[0][0] == act and float(eng.lower[0, 0].item()) == low)
            waves.append(int(res[0, 7]))
        rows.append({"mode": "speculative strict (reference order, whole GPU)", "candidates": width, "ms": ms,
                     "expansions_per_s": n_exp / (ms * 1e-3), "waves": float(np.mean(waves)),
                     "identical_root_action_and_value_vs_strict": same / float(len(scenes))})
        del eng
    for width in (16, 64, 128):
        eng = OPDWaveEngine(_lib.ENV_HIGHWAY, N_ACTIONS, a.budget, a.gamma, width, device=dev)
        ms = float(np.median([med_ms(lambda: eng.plan(s)) for s in scenes]))
        agree, gaps, waves = 0, [], []
        for s, (act, low) in zip(scenes, strict):
            eng.plan(s)
            plans, res = eng.finish([np.random.default_rng(0)])
            agree += int(plans[0][0] == act)
            gaps.append(low - float(eng.lower[0, 0].item()))
            waves.append(int(res[0, 7]))
        rows.append({"mode": "wavefront", "width": width, "ms": ms, "expansions_per_s": n_exp / (ms * 1e-3),
                     "waves": float(np.mean(waves)), "root_action_agreement_vs_strict": agree / float(len(scenes)),
                     "root_value_lower_gap_vs_strict_max": float(max(gaps)),
                     "root_value_lower_strict_mean": float(np.mean([l for _, l in strict]))})
        del eng
    big = []
    for width in (1024, 4096):
        try:
            eng = OPDWaveEngine(_lib.ENV_HIGHWAY, N_ACTIONS, 1000000, a.gamma, width, device=dev)
            ms = med_ms(lambda: eng.plan(scenes[0]))
            eng.plan(scenes[0])
            _, res = eng.finish([np.random.default_rng(0)])
            big.append({"budget": 1000000, "expansions": 200000, "width": width, "ms": float(ms), "waves": int(res[0, 7]),
                        "expansions_per_s": 200000 / (ms * 1e-3), "max_depth": int(res[0, 2]),
                        "root_value_lower": float(eng.lower[0, 0].item())})
            del eng
        except Exception as e:
            big.append({"width": width, "error": str(e)[:200]})
    return {"workload": "ONE C2 decision: OPD on HighwayLite, budget %d, gamma %g" % (a.budget, a.gamma),
            "specification": "oracle/planners.py::opd_plan_wavefront (bit-exact, tests/test_gpu_wave.py); width 1 = reference",
            "rows": rows, "budget_1e6_decision": big}


_JSON_OUT = None


def claim_stdout():
    """stdout carries ONE JSON line: libraries that write to fd 1 on their own (NCCL prints its version banner
    there under NCCL_DEBUG=VERSION) are pointed at stderr; emit() writes the line to the real stdout."""
    global _JSON_OUT
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def emit(obj):
    out = _JSON_OUT if _JSON_OUT is not None else sys.stdout
    out.write(json.dumps(obj) + "\n")
    out.flush()


def main():
    a = parse()
    claim_stdout()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)


if __name__ == "__main__":
    main()
