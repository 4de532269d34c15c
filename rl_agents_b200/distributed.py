"""Multi-GPU partitioning of the planning path: one process per GPU
(torch.distributed, NCCL on the GPU box / gloo in CPU tests).

  OPD / batched decisions   independent trees are sharded over ranks; no
                            data-path collective (results gathered at the end).
  OPD / one big decision    sub-tree sharding (ShardedOPD): every rank expands the
                            root identically to depth k, the depth-k sub-trees are
                            dealt round-robin, each rank searches its sub-trees
                            best-first, and ONE all-reduce(max) of the sub-trees'
                            (value_lower, value_upper) decides the action.
  MCTS root parallelism     every rank grows its own tree on episodes/world
                            episodes from the same root with an independent RNG
                            stream; ONE all-reduce of the root's per-action
                            (count, count*value) decides the action.
  Value iteration           state slabs: rank g owns rows [g*S/G, (g+1)*S/G) of
                            P/N/R/Q; after every sweep the V slabs are
                            all-gathered and the allclose violation counter is
                            all-reduced (the only exchange step of the path).
The helpers below work on CPU tensors too, which is how the gloo tests cover them.
"""
import numpy as np


def shard_range(n, rank, world):
    """Contiguous, balanced split of range(n): the first n % world ranks get one extra."""
    base, extra = divmod(int(n), int(world))
    begin = rank * base + min(rank, extra)
    return begin, begin + base + (1 if rank < extra else 0)


def slab_sizes(n, world):
    return [shard_range(n, r, world)[1] - shard_range(n, r, world)[0] for r in range(world)]


def allgather_slabs(full, n, group=None):
    """In place: every rank contributes full[begin:end] of its own slab and receives the rest."""
    import torch
    import torch.distributed as dist
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    if full.is_cuda and dist.get_backend(group) == "gloo":
        # gloo has no all_gather for device tensors: stage through the host (CPU-backend tests of the device
        # path, e.g. two ranks sharing one GPU; the production backend is NCCL or the fused peer-memory sweep)
        host = full[:n].cpu()
        allgather_slabs(host, n, group)
        full[:n].copy_(host)
        return full
    sizes = slab_sizes(n, world)
    if len(set(sizes)) == 1:
        b, e = shard_range(n, rank, world)
        dist.all_gather_into_tensor(full[:n], full[b:e].clone(), group=group)
        return full
    pad = max(sizes)
    b, e = shard_range(n, rank, world)
    mine = torch.zeros(pad, dtype=full.dtype, device=full.device)
    mine[:e - b] = full[b:e]
    out = torch.empty(pad * world, dtype=full.dtype, device=full.device)
    dist.all_gather_into_tensor(out, mine, group=group)
    for r in range(world):
        rb, re = shard_range(n, r, world)
        full[rb:re] = out[r * pad:r * pad + (re - rb)]
    return full


class PeerBuffer(object):
    """A device buffer of `nbytes` per rank that every rank of the group can address (CUDA IPC over
    NVLink / NVSwitch): `ptrs[r]` is the address of rank r's buffer in THIS process (ptrs[rank] is the
    local allocation).  One process per GPU on one node."""

    def __init__(self, nbytes, group=None):
        import ctypes
        import torch.distributed as dist
        from rl_agents_b200 import _lib
        self.lib = _lib.load()
        self.group = group
        self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        self.nbytes = int(nbytes)
        local = ctypes.c_void_p()
        _lib.check(self.lib.b2_p2p_alloc(self.nbytes, ctypes.byref(local)))
        self.local = local.value
        handle = ctypes.create_string_buffer(64)
        _lib.check(self.lib.b2_p2p_export(ctypes.c_void_p(self.local), handle))
        handles = [None] * self.world
        dist.all_gather_object(handles, handle.raw, group=group)
        self.ptrs, self._opened = [], []
        for r, h in enumerate(handles):
            if r == self.rank:
                self.ptrs.append(self.local)
                continue
            peer = ctypes.c_void_p()
            _lib.check(self.lib.b2_p2p_import(ctypes.create_string_buffer(h, 64), ctypes.byref(peer)))
            self.ptrs.append(peer.value)
            self._opened.append(peer.value)

    def close(self):
        import ctypes
        import torch
        import torch.distributed as dist
        torch.cuda.synchronize()
        dist.barrier(group=self.group)           # nobody still writes into a buffer that is about to go
        for p in self._opened:
            self.lib.b2_p2p_close(ctypes.c_void_p(p))
        self._opened = []
        if self.local:
            self.lib.b2_p2p_free(ctypes.c_void_p(self.local))
            self.local = None


class DistributedVI(object):
    """Slab-sharded value iteration (value_iteration.py:42-73 over G GPUs): rank g owns rows
    [g*S/G, (g+1)*S/G) of P / N / R / Q and needs the whole V for its gathers, so the path has ONE exchange
    step per sweep: the all-gather of the V slabs.  The allclose violation counters (one int per sweep) are
    all-reduced every `check_every` sweeps as a vector: 1 (default) keeps the reference's early exit exactly
    (the sweep after the converged one does nothing and the OLD iterate is returned); a larger value trades
    that for fewer collectives -- sweeps then continue up to the next check, and the result is the iterate
    at the first converged sweep only if it is still in the ping-pong buffers (otherwise the latest one,
    which differs from it by less than the allclose tolerance).

    tables_are_local=False: `transition/reward/terminal/nxt` are the FULL host tables and every rank slices its
    slab (small MDPs, tests).  tables_are_local=True: they are already this rank's slab (rows
    shard_range(n_states, rank, world)), host arrays or device tensors -- no rank ever materialises another
    rank's rows (C4: 640 MB of P/N per GPU instead of 5 GB each)."""

    def __init__(self, mode, transition, reward, terminal, nxt=None, gamma=1.0, device="cuda", group=None,
                 tables_are_local=False, n_states=None, check_every=1, rtol=1e-5, atol=1e-8, exchange="nccl",
                 max_iterations=1024):
        """exchange="nccl": all-gather / all-reduce collectives after each sweep kernel (also what the gloo CPU
        tests drive).  exchange="p2p": the exchange is fused into the sweep kernel over NVLink peer memory
        (b2_vi_sweep_p2p): no collective call inside the loop, exact per-sweep early exit."""
        import torch.distributed as dist
        from rl_agents_b200.engine.vi import VIEngine
        self.dist, self.group = dist, group
        self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        self.check_every = max(1, int(check_every))
        self.exchange = exchange
        self.max_iterations = int(max_iterations)
        self.peer = None
        if tables_are_local:
            if n_states is None:
                raise ValueError("tables_are_local needs n_states (the whole MDP's state count)")
            S = int(n_states)
            b, e = shard_range(S, self.rank, self.world)
            if int(reward.shape[0]) != e - b:
                raise ValueError("rank %d owns rows [%d, %d) but got %d rows" % (self.rank, b, e, reward.shape[0]))
            slab = (transition, reward, terminal, nxt)
        else:
            S = np.asarray(reward).shape[0]
            b, e = shard_range(S, self.rank, self.world)
            slab = (np.asarray(transition)[b:e], np.asarray(reward)[b:e], np.asarray(terminal)[b:e],
                    None if nxt is None else np.asarray(nxt)[b:e])
        if S < self.world:
            # some rank would own an empty slab (null device tables): its first sweep would fail while the other
            # ranks block in the exchange.  Every rank knows S and world, so every rank raises here.
            raise ValueError("%d states cannot be split over %d ranks: every rank needs at least one" % (S, self.world))
        self.n_states = S
        self.engine = VIEngine(mode, slab[0], slab[1], slab[2], nxt=slab[3], gamma=gamma, device=device,
                               row_begin=b, row_end=e, n_states=S, rtol=rtol, atol=atol)
        if exchange == "p2p":
            self._setup_p2p()
        elif exchange != "nccl":
            raise ValueError("exchange must be 'nccl' or 'p2p'")

    # ------------------------------------------------------------------ fused exchange over peer memory
    def _setup_p2p(self):
        from rl_agents_b200 import _lib
        if self.world > _lib.MAX_PEERS:
            raise ValueError("p2p exchange supports up to %d ranks" % _lib.MAX_PEERS)
        S, G, T = self.n_states, self.world, self.max_iterations
        al = lambda n: (n + 255) // 256 * 256
        self._off_v = [0, al(S * 8)]
        self._off_flags = self._off_v[1] + al(S * 8)
        self._off_parts = self._off_flags + al(G * 4)
        self._off_local = self._off_parts + al(T * G * 4)        # viol_local [T] + done [T]: never read by peers
        self._bytes = self._off_local + al(T * 4) + al(T * 4) + 256
        self.peer = PeerBuffer(self._bytes, self.group)
        x = _lib.VIP2P()
        x.world, x.rank = G, self.rank
        for r in range(G):
            base = self.peer.ptrs[r]
            x.v[0][r], x.v[1][r] = base + self._off_v[0], base + self._off_v[1]
            x.flags[r], x.parts[r] = base + self._off_flags, base + self._off_parts
        x.viol_local = self.peer.local + self._off_local
        x.done = self.peer.local + self._off_local + al(T * 4)
        x.status = self.peer.local + self._off_local + 2 * al(T * 4)
        self._x = x

    def _solve_p2p(self, iterations):
        import ctypes
        import torch
        from rl_agents_b200 import _lib
        if iterations > self.max_iterations:
            raise ValueError("iterations %d > max_iterations %d" % (iterations, self.max_iterations))
        eng, lib = self.engine, self.peer.lib
        stream = _lib.current_stream()
        for q in eng.q:
            q.zero_()
        _lib.check(lib.b2_p2p_memset(ctypes.c_void_p(self.peer.local), 0, self._bytes, stream))
        torch.cuda.synchronize()
        self.dist.barrier(group=self.group)      # every rank's flags are zero before anybody publishes
        for k in range(iterations):
            _lib.check(lib.b2_vi_sweep_p2p(eng.problem, self._x, _lib.ptr(eng.q[k & 1]), _lib.ptr(eng.q[(k + 1) & 1]),
                                           k, stream))
        parts = np.zeros((iterations, self.world), dtype=np.int32)
        _lib.check(lib.b2_p2p_read(parts.ctypes.data_as(ctypes.c_void_p),
                                   ctypes.c_void_p(self.peer.local + self._off_parts), parts.nbytes, stream))
        # a rank reads its own table only after ITS last kernel retired; peers publish their last entry
        # when THEIR last kernel retires: wait for everybody before trusting the last row
        self.dist.barrier(group=self.group)
        _lib.check(lib.b2_p2p_read(parts.ctypes.data_as(ctypes.c_void_p),
                                   ctypes.c_void_p(self.peer.local + self._off_parts), parts.nbytes, stream))
        status = np.zeros(1, dtype=np.int32)
        _lib.check(lib.b2_p2p_read(status.ctypes.data_as(ctypes.c_void_p), ctypes.c_void_p(self._x.status), 4, stream))
        if int(status[0]) != 0:
            raise _lib.B2Error("p2p value iteration: a peer's arrival flag timed out (rank %d)" % self.rank)
        viol = parts.sum(axis=1)
        zero = np.nonzero(viol == 0)[0]
        if zero.size:
            k = int(zero[0])
            return eng.q[k & 1], k + 1
        return eng.q[iterations & 1], int(iterations)

    def v_slab(self, iterations_done):
        """(p2p) this rank's copy of the full V after `iterations_done` sweeps, as a host array."""
        import ctypes
        from rl_agents_b200 import _lib
        out = np.zeros(self.n_states, dtype=np.float64)
        _lib.check(self.peer.lib.b2_p2p_read(out.ctypes.data_as(ctypes.c_void_p),
                                             ctypes.c_void_p(self.peer.local + self._off_v[iterations_done & 1]),
                                             out.nbytes, _lib.current_stream()))
        return out

    def close(self):
        if self.peer is not None:
            self.peer.close()
            self.peer = None

    def solve(self, iterations, exchange=True):
        """Returns (this rank's Q slab on device, sweeps).  No host sync inside the loop: the sweep kernels
        read the all-reduced violation counters from device memory.  exchange=False skips the collectives
        (timing of the compute alone; the values are then meaningless)."""
        if self.exchange == "p2p" and exchange:
            return self._solve_p2p(iterations)
        eng = self.engine
        eng.reset(iterations)
        m = self.check_every
        if m > 1 or not exchange:
            # a rank whose own slab shows 0 violations must keep sweeping until the GLOBAL count is known:
            # bias every local counter by one (removed again after the all-reduce)
            eng.viol.fill_(1)
        for k in range(iterations):
            eng.sweep(k)
            if not exchange:
                continue
            allgather_slabs(eng.v[(k + 1) & 1], self.n_states, self.group)
            if (k + 1) % m == 0 or k + 1 == iterations:
                k0 = (k // m) * m
                self.dist.all_reduce(eng.viol[k0:k + 1], group=self.group)
                if m > 1:
                    eng.viol[k0:k + 1] -= self.world
        return eng.result(iterations)


def merge_root_statistics(counts, values, group=None):
    """MCTS root parallelisation: counts/values are [A] tensors of THIS rank's root
    children (count, mean value).  One all-reduce of [2, A]; returns the merged
    (count, mean value) on every rank."""
    import torch
    import torch.distributed as dist
    packed = torch.stack([counts.to(torch.float64), counts.to(torch.float64) * values.to(torch.float64)])
    dist.all_reduce(packed, group=group)
    merged_counts = packed[0]
    merged_values = torch.where(merged_counts > 0, packed[1] / merged_counts.clamp(min=1), torch.zeros_like(packed[1]))
    return merged_counts, merged_values


def merge_olop_root_statistics(counts, uppers, group=None):
    """OLOP root parallelisation (SURVEY 8e row 3): every rank runs its share of the episodes on its own
    sequence tree from the same root; the recommendation (OLOPNode.selection_rule, olop.py:126-130: most
    visited child, ties -> largest value_upper) is taken on the merged root statistics -- counts summed,
    value_upper = the tightest bound any rank holds for that action (min over the ranks that tried it).
    ONE all-gather of [2, A]; returns (counts, uppers) on every rank."""
    import torch
    import torch.distributed as dist
    world = dist.get_world_size(group)
    mine = torch.stack([counts.to(torch.float64), uppers.to(torch.float64)]).contiguous()
    flat = torch.empty(world * mine.numel(), dtype=torch.float64, device=mine.device)
    dist.all_gather_into_tensor(flat, mine.reshape(-1), group=group)
    out = flat.reshape((world,) + tuple(mine.shape))
    merged_counts = out[:, 0].sum(dim=0)
    tried = out[:, 0] > 0
    inf = torch.full_like(out[:, 1], float("inf"))
    best_upper = torch.where(tried, out[:, 1], inf).min(dim=0).values
    merged_uppers = torch.where(merged_counts > 0, best_upper, out[:, 1].max(dim=0).values)
    return merged_counts, merged_uppers


def recommend_olop(counts, uppers):
    """OLOPNode.selection_rule (olop.py:126-130) on merged statistics."""
    counts, uppers = np.asarray(counts), np.asarray(uppers)
    ties = np.nonzero(counts == counts.max())[0]
    return int(max(ties, key=lambda i: uppers[i]))


def recommend(counts, values):
    """MCTSNode.selection_rule (mcts.py:212-218) on merged statistics: most visited,
    ties -> highest value (first)."""
    counts = np.asarray(counts)
    values = np.asarray(values)
    ties = np.nonzero(counts == counts.max())[0]
    return int(max(ties, key=lambda i: values[i]))


class ShardedOPD(object):
    """One OPD decision on HighwayLite sharded over the ranks of a process group (SURVEY 8e,
    BASELINE config C5's "tree-sharded"): best-first order is global in the reference, so an exact
    shard would need an arg-max exchange per expansion; instead the top of the tree is replicated.

      1. every rank expands the root to depth k (smallest k with #sub-trees >= world, k <= 3)
         with the batched transition kernel -- identical on all ranks;
      2. sub-tree j goes to rank j % world and gets an equal share of the remaining budget;
         each rank runs its sub-trees as one batch on the OPD engine (strict best-first inside
         each sub-tree);
      3. one all_reduce(MAX) of the [n_subtrees, 2] (lower, upper) table;
      4. every rank backs the replicated top levels up (max over children, deterministic.py:74-79)
         and returns the arg-max value_lower root action.

    The node set differs from a single best-first tree of the same budget (the budget is split
    evenly instead of greedily); with world == 1 the same decomposition runs on one GPU, which is
    what the parity test compares against."""

    def __init__(self, budget, gamma, terminal_reward=0.0, group=None, device="cuda", max_depth=3, wave_width=0,
                 env="highway"):
        """wave_width = 0: every sub-tree is searched in the reference's strict best-first order (one CTA per
        sub-tree, all of a rank's sub-trees in one launch).  wave_width = K > 0: every sub-tree is searched by
        the rank's whole GPU in waves of K leaves (b2_opd_plan_wave), one sub-tree after the other."""
        self.budget, self.gamma, self.terminal_reward = int(budget), float(gamma), float(terminal_reward)
        self.group, self.device, self.max_depth = group, device, max_depth
        self.wave_width = int(wave_width)
        if env not in ("highway", "intersection"):
            raise ValueError("env must be 'highway' or 'intersection'")
        self.env = env
        if env == "intersection" and self.wave_width <= 0:
            self.wave_width = 1            # IntersectionLite lives in the wavefront kernel (width 1 = strict order)

    def _world(self):
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            return dist.get_world_size(self.group), dist.get_rank(self.group)
        return 1, 0

    def _expand_level(self, words_list, actions_list):
        """Batched env transition of (scene, action) pairs on the device."""
        import torch
        from rl_agents_b200 import _lib
        lib = _lib.load()
        n = len(words_list)
        st = torch.tensor(np.stack(words_list), dtype=torch.int32, device=self.device)
        act = torch.tensor(actions_list, dtype=torch.int32, device=self.device)
        rew = torch.empty(n, dtype=torch.float32, device=self.device)
        flg = torch.empty(n, dtype=torch.int32, device=self.device)
        step = lib.b2_highway_step if self.env == "highway" else lib.b2_intersection_step
        _lib.check(step(_lib.ptr(st), _lib.ptr(act), _lib.ptr(rew), _lib.ptr(flg), None, n, _lib.current_stream()))
        return st.cpu().numpy(), rew.cpu().numpy().astype(np.float64), (flg.cpu().numpy() & 1).astype(bool)

    def decide(self, root_words):
        import torch
        from rl_agents_b200 import _lib
        from rl_agents_b200.engine.opd import OPDEngine
        if self.env == "highway":
            from rl_agents_b200.envs.highway_lite import available_actions
            kind, n_act = _lib.ENV_HIGHWAY, 5
        else:
            from rl_agents_b200.envs.intersection_lite import available_actions
            kind, n_act = _lib.ENV_INTERSECTION, 3
        world, rank = self._world()
        g = self.gamma
        # top of the tree, replicated: nodes = dicts in creation order
        top = [dict(parent=-1, action=-1, depth=0, words=np.asarray(root_words, dtype=np.int32), lower=0.0,
                    done=False, children=[])]
        frontier, spent, depth = [0], 0, 0
        while depth < self.max_depth and (depth == 0 or len(frontier) < world):
            pairs = [(i, a) for i in frontier if not top[i]["done"] for a in available_actions(top[i]["words"])]
            if not pairs:
                break
            words, rew, term = self._expand_level([top[i]["words"] for i, _ in pairs], [a for _, a in pairs])
            depth += 1
            new_frontier = []
            for (i, a), w, r, t in zip(pairs, words, rew, term):
                lower = top[i]["lower"] + (g ** (depth - 1)) * r           # deterministic.py:52
                if t:
                    lower = lower + self.terminal_reward * (g ** depth) / (1 - g)
                top.append(dict(parent=i, action=a, depth=depth, words=w, lower=lower, done=bool(t), children=[]))
                top[i]["children"].append(len(top) - 1)
                new_frontier.append(len(top) - 1)
            spent += len(pairs)
            frontier = new_frontier + [i for i in frontier if top[i]["done"]]
        subtrees = [i for i in frontier if not top[i]["done"] and not top[i]["children"]]
        table = torch.full((max(len(subtrees), 1), 2), -np.inf, dtype=torch.float64, device=self.device)
        mine = [j for j in range(len(subtrees)) if j % world == rank]
        per_tree = max((self.budget - spent) // max(len(subtrees), 1), n_act)
        if mine and self.wave_width > 0:
            from rl_agents_b200.engine.opd import OPDWaveEngine
            eng = OPDWaveEngine(kind, n_act, per_tree, g, self.wave_width, self.terminal_reward, device=self.device)
            for j in mine:
                node = top[subtrees[j]]
                eng.plan(torch.tensor(node["words"], dtype=torch.int32, device=self.device))
                eng.finish()
                scale = g ** node["depth"]
                table[j, 0] = node["lower"] + scale * float(eng.lower[0, 0].item())
                table[j, 1] = node["lower"] + scale * float(eng.upper[0, 0].item())
        elif mine:
            eng = OPDEngine(_lib.ENV_HIGHWAY, len(mine), 5, per_tree, g, self.terminal_reward, device=self.device,
                            keys_in_smem=True)
            eng.plan(torch.tensor(np.stack([top[subtrees[j]]["words"] for j in mine]), dtype=torch.int32,
                                  device=self.device))
            eng.finish()
            for slot, j in enumerate(mine):
                node = top[subtrees[j]]
                scale = g ** node["depth"]
                table[j, 0] = node["lower"] + scale * float(eng.lower[slot, 0].item())
                table[j, 1] = node["lower"] + scale * float(eng.upper[slot, 0].item())
        if world > 1:
            import torch.distributed as dist
            dist.all_reduce(table, op=dist.ReduceOp.MAX, group=self.group)      # the single exchange step
        table = table.cpu().numpy()
        # back the replicated levels up
        lo = {i: n["lower"] for i, n in enumerate(top)}
        up = {i: n["lower"] + (0.0 if n["done"] else (g ** n["depth"]) / (1 - g)) for i, n in enumerate(top)}
        for j, i in enumerate(subtrees):
            lo[i], up[i] = float(table[j, 0]), float(table[j, 1])
        for i in range(len(top) - 1, -1, -1):
            if top[i]["children"]:
                lo[i] = max(lo[c] for c in top[i]["children"])
                up[i] = max(up[c] for c in top[i]["children"])
        kids = top[0]["children"]
        best = max(kids, key=lambda c: lo[c])          # first max: ties resolved towards the earliest child
        return dict(action=top[best]["action"], root_lower=lo[0], root_upper=up[0],
                    children={top[c]["action"]: (lo[c], up[c]) for c in kids}, n_subtrees=len(subtrees),
                    budget_per_subtree=per_tree, table=table)
