"""Prioritized planner: the classical-planner baseline of the reference (``scripts/a-star.py``, ``scripts/cbs.py``) under
this env's own move rule, for every layout of a batch.

Agents plan in index order 0..N-1.  Agent i searches the earliest arrival at its goal by a space-time wavefront that
avoids the cells the agents before it hold, under the rule of the env's step (ENV:502-526): a move into a cell held by
a lower index at its new position, or by a higher index at its old position, fails.  With R_t the cells of the planned
agents at time t (R_{H+1} = R_H), agent i may stand on c at time t >= 1 iff

    c in W_t = free & ~R_t & ~R_{t+1} & (t == 1 ? ~(starts of the agents after i) : all)

Agents stay on their goal once there (the episode ends at the first step where every agent stands on its goal), so an
arrival at t needs the goal outside R_t' for every t' >= t, and the agent then holds its goal up to H.  Among the paths
with the earliest arrival the backtrack takes, at every step, the first predecessor in the action order NO_OP, UP,
RIGHT, DOWN, LEFT (:mod:`actions`): plans are deterministic.

An agent with no arrival within H (= ``steps_per_episode``) or an unreachable goal gets arrival -1 and NO_OP actions
and holds its start for every t; the later agents are still planned.  Such an env has status 0, and **only status-1
envs carry a guarantee**: their actions replay through the env with no failed move and end the episode (terminated,
not truncated) at step ``makespan`` = max(1, max arrival) with every agent on its goal.

:func:`plan_prioritized` runs the ``mapf_plan_prioritized`` kernel (one warp per env, one lane per map row) for a CUDA
env; :func:`plan_reference` is the PyTorch reference (any device, vectorised over envs), which is also the CPU path.
:class:`PlannedPolicy` plays plans through :func:`evaluate.evaluate`.  ``python -m dl_reference_models_b200.planner``
times the kernel (:func:`benchmark`).

**Windowed plans** (rolling-horizon planning, RHCR, Li et al. 2021; DESIGN.md §7 N4c): :func:`plan_windowed` plans from
the env's current positions to its current goals, lifelong envs included, with the rule above and H read as the window
W, and does not require arrival:

* the target is the goal if the distance table reaches it from the start (!= 255), else the agent's own start: an
  agent with an unreachable goal tries to stay put and gets out of the way when it must;
* an agent whose target is its goal arrives as above (the first t <= W with the goal in the wavefront and
  t >= max(d, last[goal] + 1)) and holds its goal to W; ``arrival`` = t;
* otherwise the search runs to t = W and the path ends on the cell of F_W with the smallest distance-table value
  d(target, cell), ties to the first cell in row-major order; the agent reserves that path (last[end] = W) and gets
  ``arrival`` -1;
* an agent whose wavefront empties before W, or whose start or goal lies off the map, fails as above (NO_OPs, start
  reserved for every t, env status 0); the later agents are still planned.

status[b] = 1 iff every agent of env b got a path; then the W actions replay through the env's step from the planned
state with no failed move and every agent on its planned cells -- in lifelong mode too, since goal reassignment never
moves an agent -- and an agent that arrived stands on its goal from its arrival on.  Makespan and sum of costs are as
above for envs where every agent arrived, -1 otherwise.  On an env where :func:`plan_prioritized` at H has status 1,
the windowed plan at W = H has the same actions and arrivals.  :class:`ReplanningPolicy` replans every h steps and
plays the first h actions of each plan through :func:`evaluate.evaluate`; ``python -m dl_reference_models_b200.planner
--windowed`` measures it (:func:`benchmark_windowed`).

**Conflict-based search** (CBS, Sharon et al. 2015; DESIGN.md §7 N4d): :func:`plan_cbs` finds, per env, a plan with the
least sum of arrivals within H that replays under the env's move rule, for small agent counts (2-8), with an
``outcome`` that says why there is none (0: no plan within H, 2: the ``max_nodes`` expansion budget ran out).  Two
conflicts exist under this rule: a vertex conflict (two agents on one cell at t + 1) and a following conflict (agent a
moves at t into the cell a higher index b holds at t); they split into the constraints (a, c, t+1) / (b, c, t+1) and
(a, c, t+1) / (b, c, t).  The low level is the wavefront above with the agent's constraints as the obstacles; the high
level pops the least (sum of arrivals, creation id), takes the first conflict (smallest t, vertex before following,
lowest a, then lowest b) and creates the child constraining a, then b.  :func:`cbs_reference` is the pure Python
reference and CPU path; ``PlannedPolicy("cbs")`` plays the plans through :func:`evaluate.evaluate`; ``python -m
dl_reference_models_b200.planner --cbs`` measures it (:func:`benchmark_cbs`).
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np
import torch

from . import _native as nat
from .batched_env import BatchedMapfEnv


@dataclass
class Plan:
    actions: torch.Tensor        # int8  [H,B,N]: action of agent n of env b at step t (NO_OP after arrival)
    arrival: torch.Tensor        # int16 [B,N]: arrival step (0 = starts on its goal), -1 = none within H
    status: torch.Tensor         # uint8 [B]: 1 = every agent arrived (windowed: got a path); the plan replays
    makespan: torch.Tensor       # int32 [B]: max(1, max arrival) = the step the episode terminates at; -1 for status 0
    sum_of_costs: torch.Tensor   # int32 [B]: sum of the arrivals; -1 for status 0 (windowed: or an agent not arrived)


@dataclass
class CbsPlan(Plan):
    outcome: torch.Tensor        # uint8 [B]: 1 = optimal plan found, 0 = no plan within H, 2 = max_nodes expansions hit
    expanded: torch.Tensor       # int32 [B]: high-level nodes popped


def _finish(actions, arrival, status) -> Plan:
    ok = status.bool() & (arrival >= 0).all(1)
    a = arrival.to(torch.int32)
    makespan = torch.where(ok, a.amax(1).clamp(min=1), torch.full_like(a[:, 0], -1))
    soc = torch.where(ok, a.sum(1), torch.full_like(a[:, 0], -1))
    return Plan(actions, arrival, status, makespan, soc)


def _finish_cbs(actions, arrival, outcome, expanded) -> CbsPlan:
    p = _finish(actions, arrival, (outcome == 1).to(torch.uint8))
    return CbsPlan(**vars(p), outcome=outcome, expanded=expanded)


def plan_prioritized(env: BatchedMapfEnv, starts=None, goals=None, horizon: int | None = None) -> Plan:
    """Plan every env of ``env`` on the device (``mapf_plan_prioritized``).  ``starts`` / ``goals``: int16 [B,N,2]
    (default: the env's current positions -- its starts right after a reset -- and its goals); ``horizon`` defaults to
    ``steps_per_episode``.  Lifelong envs are refused: their goals change during the episode."""
    if not isinstance(env, BatchedMapfEnv):
        raise TypeError(f"plan_prioritized plans a BatchedMapfEnv; use plan_reference on the CPU (got {type(env).__name__})")
    if env.lifelong:
        raise ValueError("a lifelong env assigns new goals during the episode: a plan to the first goals is not a plan")
    H = int(env.cfg.steps_per_episode if horizon is None else horizon)
    return _plan_native(env, starts, goals, H, "mapf_plan_prioritized")


def plan_windowed(env: BatchedMapfEnv, window: int, starts=None, goals=None) -> Plan:
    """Windowed plans of every env of ``env`` on the device (``mapf_plan_windowed``): W = ``window`` steps from
    ``starts`` to ``goals`` (int16 [B,N,2]; default: the env's current positions and current goals), lifelong or
    episodic.  ``actions`` is [W,B,N]; see the module docstring for what a windowed plan is."""
    if not isinstance(env, BatchedMapfEnv):
        raise TypeError(f"plan_windowed plans a BatchedMapfEnv; use plan_reference on the CPU (got {type(env).__name__})")
    return _plan_native(env, starts, goals, int(window), "mapf_plan_windowed")


def plan_cbs(env: BatchedMapfEnv, max_nodes: int = 1024, starts=None, goals=None,
             horizon: int | None = None) -> CbsPlan:
    """Conflict-based search of every env of ``env`` on the device (``mapf_plan_cbs``; DESIGN.md §7 N4d): plans with
    the least sum of arrivals within H under the env's own move rule, or the reason there is none.  ``outcome`` 1 =
    optimal plan (``status`` 1; it replays like a status-1 :func:`plan_prioritized` plan), 0 = no plan exists within
    H (an unreachable goal, a start or goal off the map, on an obstacle or repeated, or every split exhausted), 2 =
    ``max_nodes`` high-level expansions without an answer.  Envs with outcome 0 or 2 get NO_OPs and arrival -1.
    ``starts`` / ``goals`` / ``horizon`` as in :func:`plan_prioritized`; lifelong envs are refused.  CBS is for small
    agent counts (2-8): its search grows with the number of conflicts, so :func:`plan_prioritized` stays the
    large-N baseline."""
    if not isinstance(env, BatchedMapfEnv):
        raise TypeError(f"plan_cbs plans a BatchedMapfEnv; use cbs_reference on the CPU (got {type(env).__name__})")
    if env.lifelong:
        raise ValueError("a lifelong env assigns new goals during the episode: a plan to the first goals is not a plan")
    H = int(env.cfg.steps_per_episode if horizon is None else horizon)
    s, g = _layouts(env, starts, goals)
    B, N = int(s.shape[0]), int(s.shape[1])
    L = nat.lib()
    R, Cc = (int(x) for x in env.grid.shape[-2:])
    nbytes = nat.check(L.mapf_cbs_workspace_bytes(R, Cc, B, N, max(H, 1), int(max_nodes))) if B > 0 and N > 0 else 0
    dev = env.device
    ws = torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=dev)
    actions = torch.empty((H, B, N), dtype=torch.int8, device=dev)
    arrival = torch.empty((B, N), dtype=torch.int16, device=dev)
    outcome = torch.empty(B, dtype=torch.uint8, device=dev)
    expanded = torch.empty(B, dtype=torch.int32, device=dev)
    p = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
    args = nat.MapfCbsArgs(num_envs=B, num_agents=N, horizon=H, max_nodes=int(max_nodes), starts=p(s), goals=p(g),
                           distance_table=p(env.distance_table()), workspace=p(ws), workspace_bytes=ws.numel(),
                           actions=p(actions), arrival=p(arrival), status=p(outcome), expanded=p(expanded))
    nat.check(L.mapf_plan_cbs(env._h, C.byref(args), env._stream()))
    return _finish_cbs(actions, arrival, outcome, expanded)


def _layouts(env: BatchedMapfEnv, starts, goals):
    s = (env.state["positions"] if starts is None else torch.as_tensor(starts)).to(env.device, torch.int16).contiguous()
    g = (env.state["goals"] if goals is None else torch.as_tensor(goals)).to(env.device, torch.int16).contiguous()
    if s.ndim != 3 or s.shape[2] != 2 or s.shape != g.shape:
        raise ValueError(f"starts and goals must both be [B,N,2], got {tuple(s.shape)} and {tuple(g.shape)}")
    return s, g


def _plan_native(env: BatchedMapfEnv, starts, goals, H: int, entry: str) -> Plan:
    s, g = _layouts(env, starts, goals)
    B, N = int(s.shape[0]), int(s.shape[1])
    L = nat.lib()
    R, Cc = (int(x) for x in env.grid.shape[-2:])
    nbytes = nat.check(L.mapf_plan_workspace_bytes(R, Cc, B, max(H, 1))) if B > 0 else 0
    dev = env.device
    ws = torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=dev)
    actions = torch.empty((H, B, N), dtype=torch.int8, device=dev)
    arrival = torch.empty((B, N), dtype=torch.int16, device=dev)
    status = torch.empty(B, dtype=torch.uint8, device=dev)
    p = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
    args = nat.MapfPlanArgs(num_envs=B, num_agents=N, horizon=H, starts=p(s), goals=p(g),
                            distance_table=p(env.distance_table()), workspace=p(ws), workspace_bytes=ws.numel(),
                            actions=p(actions), arrival=p(arrival), status=p(status))
    nat.check(getattr(L, entry)(env._h, C.byref(args), env._stream()))
    return _finish(actions, arrival, status)


def _components(grid: np.ndarray) -> np.ndarray:
    """4-connected component label of every free cell (0 = obstacle)."""
    from scipy import ndimage

    lab, _ = ndimage.label(grid == 0, structure=[[0, 1, 0], [1, 1, 1], [0, 1, 0]])
    return lab


def _distances(grid: np.ndarray) -> np.ndarray:
    """Moves between any two cells around the obstacles, as the distance table stores them: int64 [R*C, R*C],
    255 = unreachable (an obstacle at either end) or more than 254 moves."""
    from scipy.sparse import coo_matrix
    from scipy.sparse.csgraph import shortest_path

    Rr, Cc = grid.shape
    free = (grid == 0).reshape(-1)
    idx = np.arange(Rr * Cc).reshape(Rr, Cc)
    right = np.stack([idx[:, :-1].reshape(-1), idx[:, 1:].reshape(-1)], 1)
    down = np.stack([idx[:-1].reshape(-1), idx[1:].reshape(-1)], 1)
    e = np.concatenate([right, down])
    e = e[free[e[:, 0]] & free[e[:, 1]]]
    adj = coo_matrix((np.ones(len(e)), (e[:, 0], e[:, 1])), shape=(Rr * Cc, Rr * Cc))
    d = shortest_path(adj, directed=False, unweighted=True)
    d[~free, :] = np.inf
    d[:, ~free] = np.inf
    return np.where(np.isfinite(d) & (d <= 254), d, 255).astype(np.int64)


@torch.no_grad()
def plan_reference(grid, starts, goals, horizon: int, device=None, window: bool = False) -> Plan:
    """The planner in PyTorch, vectorised over envs (``device``: default the starts' device, else the CPU): the same
    semantics and tie rule as the kernel, bit for bit, written from the rule itself: [B, H+1, rows] planes of int64 row
    words for R_t and F_t, and a reachability test by connected components instead of the distance table.
    ``window=True``: the windowed plan of ``mapf_plan_windowed`` with W = ``horizon`` (targets and end cells from a
    breadth-first distance table with the kernel's 255 cap)."""
    grid = np.ascontiguousarray(np.asarray(grid), dtype=np.uint8)
    if grid.ndim != 2 or grid.shape[0] > 32 or grid.shape[1] > 32:
        raise ValueError(f"the planner needs one map of at most 32x32 cells, got shape {grid.shape}")
    dev = torch.device(device) if device is not None else (starts.device if isinstance(starts, torch.Tensor) else torch.device("cpu"))
    st = torch.as_tensor(starts).to(dev, torch.int64)
    gl = torch.as_tensor(goals).to(dev, torch.int64)
    B, N = int(st.shape[0]), int(st.shape[1])
    H = int(horizon)
    if H < 1:
        raise ValueError("horizon must be >= 1")
    Rr, Cc = grid.shape
    free = torch.as_tensor((((grid == 0).astype(np.int64)) << np.arange(Cc, dtype=np.int64)).sum(1), device=dev)   # [R]
    comp = torch.as_tensor(_components(grid).reshape(-1), dtype=torch.int64, device=dev)
    dist = torch.as_tensor(_distances(grid), device=dev) if window else None
    cell_ix = torch.arange(Rr * Cc, device=dev)
    ar = torch.arange(B, device=dev)
    one = torch.ones((), dtype=torch.int64, device=dev)
    Res = torch.zeros((B, H + 1, Rr), dtype=torch.int64, device=dev)
    Fh = torch.zeros((B, H + 1, Rr), dtype=torch.int64, device=dev)
    last = torch.full((B, Rr * Cc), -1, dtype=torch.int64, device=dev)
    actions = torch.zeros((H, B, N), dtype=torch.int8, device=dev)
    arrival = torch.full((B, N), -1, dtype=torch.int16, device=dev)
    status = torch.ones(B, dtype=torch.uint8, device=dev)
    sr_all, sc_all, gr_all, gc_all = st[..., 0], st[..., 1], gl[..., 0], gl[..., 1]
    on_map = ((sr_all >= 0) & (sr_all < Rr) & (sc_all >= 0) & (sc_all < Cc) &
              (gr_all >= 0) & (gr_all < Rr) & (gc_all >= 0) & (gc_all < Cc))          # [B,N]
    hi = torch.zeros((B, Rr), dtype=torch.int64, device=dev)                          # starts of the unplanned agents
    for a in range(N):
        m = on_map[:, a]
        hi[ar[m], sr_all[m, a]] |= one << sc_all[m, a]
    tt = torch.arange(H + 1, device=dev)
    for i in range(N):
        m = on_map[:, i]
        sr, sc = sr_all[:, i].clamp(0, Rr - 1), sc_all[:, i].clamp(0, Cc - 1)
        gr, gc = gr_all[:, i].clamp(0, Rr - 1), gc_all[:, i].clamp(0, Cc - 1)
        sbit = one << sc
        hi[ar[m], sr[m]] &= ~sbit[m]
        s_cell, g_cell = sr * Cc + sc, gr * Cc + gc
        if window:   # the goal is the target where the table reaches it; the search runs for every agent on the map
            reach = m & (dist[g_cell, s_cell] != 255)
        else:
            reach = m & (comp[s_cell] > 0) & (comp[s_cell] == comp[g_cell])
        lo = last[ar, g_cell] + 1
        ta = torch.full((B,), -1, dtype=torch.int64, device=dev)
        ta[reach & (s_cell == g_cell) & (lo <= 0)] = 0
        search = (m if window else reach & (lo <= H)) & (ta < 0)
        F = torch.zeros((B, Rr), dtype=torch.int64, device=dev)
        F[ar[search], sr[search]] = sbit[search]
        Fh[:, 0] = F
        for t in range(1, H + 1):
            if not bool(search.any()):
                break
            nf = F | (F << 1) | (F >> 1)
            nf[:, :-1] |= F[:, 1:]
            nf[:, 1:] |= F[:, :-1]
            w = free & ~Res[:, t] & ~Res[:, min(t + 1, H)]
            if t == 1:
                w = w & ~hi
            F = torch.where(search[:, None], nf & w, torch.zeros_like(F))
            Fh[:, t] = F
            hit = search & reach & (t >= lo) & ((F[ar, gr] >> gc) & 1).bool()
            ta[hit] = t
            search = search & ~hit & (F != 0).any(1)
        arrival[:, i] = ta.to(torch.int16)
        if window and bool(search.any()):
            # still searching at t = W: the path ends on F_W's cell of least (d(target, cell), cell index)
            e = ar[search]
            target = torch.where(reach, g_cell, s_cell)[e]
            inF = ((F[e, :, None] >> torch.arange(Cc, device=dev)) & 1).bool().reshape(len(e), Rr * Cc)
            key = torch.where(inF, dist[target] * 1024 + cell_ix, 1 << 30)
            end = key.argmin(1)
            gr, gc = gr.clone(), gc.clone()
            gr[e], gc[e] = end // Cc, end % Cc
            g_cell = gr * Cc + gc
            ta[e] = H
        gbit = one << gc
        ok = ta >= 0
        status &= ok.to(torch.uint8)
        # failed agents on the map hold their start for every t
        bad = m & ~ok
        if bool(bad.any()):
            Res[ar[bad], :, sr[bad]] |= sbit[bad][:, None]
            last[ar[bad], s_cell[bad]] = H
        if not bool(ok.any()):
            continue
        # the goal from arrival + 1 on, then the path back from (goal, arrival)
        hold = ok[:, None] & (tt[None, :] > ta[:, None])                          # [B,H+1]
        Res[ar, :, gr] |= torch.where(hold, gbit[:, None], torch.zeros_like(hold, dtype=torch.int64))
        r, c = gr.clone(), gc.clone()
        for t in range(int(ta.max()), 0, -1):
            act = ok & (t <= ta)
            if not bool(act.any()):
                continue
            f = Fh[:, t - 1]
            f0 = f[ar, r]
            fp = torch.where(r + 1 < Rr, f[ar, (r + 1).clamp(max=Rr - 1)], torch.zeros_like(f0))
            fm = torch.where(r > 0, f[ar, (r - 1).clamp(min=0)], torch.zeros_like(f0))
            bit = lambda w, cc: ((w >> cc.clamp(0, 31)) & 1).bool() & (cc >= 0) & (cc < Cc)  # noqa: E731
            cand = torch.stack([bit(f0, c), bit(fp, c) & (r + 1 < Rr), bit(f0, c - 1), bit(fm, c) & (r > 0),
                                torch.ones_like(act)], 1)
            a = cand.to(torch.int64).argmax(1)                                     # first true in action order
            Res[ar[act], t, r[act]] |= (one << c)[act]
            cell = r * Cc + c
            last[ar[act], cell[act]] = torch.maximum(last[ar[act], cell[act]], torch.full_like(cell[act], t))
            actions[t - 1, act, i] = a[act].to(torch.int8)
            dr = torch.tensor([0, 1, 0, -1, 0], device=dev)[a]                    # predecessor = cell - move
            dc = torch.tensor([0, 0, -1, 0, 1], device=dev)[a]
            r = torch.where(act, r + dr, r)
            c = torch.where(act, c + dc, c)
        Res[ar[ok], 0, r[ok]] |= (one << c)[ok]
        cell = r * Cc + c
        last[ar[ok], cell[ok]] = torch.maximum(last[ar[ok], cell[ok]], torch.zeros_like(cell[ok]))
        last[ar[ok], g_cell[ok]] = H
    return _finish(actions, arrival, status)


_MOVES = ((0, 0), (-1, 0), (0, 1), (1, 0), (0, -1))     # (dr, dc) of NO_OP, UP, RIGHT, DOWN, LEFT


def _cbs_low_level(free, W, R, Cc, s, g, cons, H):
    """One agent's earliest arrival under its constraints ``cons`` ({t: forbidden cell bits}; cell (r, c) is bit
    r * W + c, W = C + 1 so that shifts never wrap into the next row): the path as the cells at t = 0..arrival, or
    None."""
    gb = 1 << (g[0] * W + g[1])
    L = 1 + max((t for t, m in cons.items() if m & gb), default=-1)
    f = 1 << (s[0] * W + s[1])
    if cons.get(0, 0) & f:
        return None
    F = [f]
    ta = 0 if s == g and L == 0 else -1
    if ta < 0:
        for t in range(1, H + 1):
            f = (f | (f << 1) | (f >> 1) | (f << W) | (f >> W)) & free & ~cons.get(t, 0)
            F.append(f)
            if t >= L and f & gb:
                ta = t
                break
            if not f:
                break
    if ta < 0:
        return None
    path = [g]
    r, c = g
    for t in range(ta, 0, -1):
        prev = F[t - 1]
        for dr, dc in _MOVES:                          # the first predecessor in action order
            pr, pc = r - dr, c - dc
            if 0 <= pr < R and 0 <= pc < Cc and prev >> (pr * W + pc) & 1:
                break
        r, c = pr, pc
        path.append((r, c))
    return path[::-1]


def _cbs_first_conflict(paths):
    """The first conflict of a joint plan in scan order, as its two vertex constraints (a, cell, t), (b, cell, t')."""
    N = len(paths)
    at = lambda p, t: p[t] if t < len(p) else p[-1]  # noqa: E731
    for t in range(max(len(p) for p in paths) - 1):
        cur = [at(p, t) for p in paths]
        nxt = [at(p, t + 1) for p in paths]
        for a in range(N):                             # vertex: lowest a, then lowest b
            for b in range(a + 1, N):
                if nxt[a] == nxt[b]:
                    return (a, nxt[a], t + 1), (b, nxt[a], t + 1)
        owner = {c: i for i, c in enumerate(cur)}
        for a in range(N):                             # following: a moves into the cell a higher index holds at t
            b = owner.get(nxt[a], -1)
            if nxt[a] != cur[a] and b > a:
                return (a, nxt[a], t + 1), (b, nxt[a], t)
    return None


def _cbs_one(grid, starts, goals, H, max_nodes):
    """CBS of one env: (paths or None, outcome, expanded)."""
    import heapq

    R, Cc = grid.shape
    W = Cc + 1
    free = sum(1 << (int(r) * W + int(c)) for r, c in np.argwhere(grid == 0))
    st = [(int(r), int(c)) for r, c in starts]
    gl = [(int(r), int(c)) for r, c in goals]
    inside = lambda p: 0 <= p[0] < R and 0 <= p[1] < Cc and grid[p] == 0  # noqa: E731
    if not all(inside(p) for p in st + gl) or len(set(st)) < len(st) or len(set(gl)) < len(gl):
        return None, 0, 0
    paths = [_cbs_low_level(free, W, R, Cc, s, g, {}, H) for s, g in zip(st, gl)]
    if any(p is None for p in paths):
        return None, 0, 0
    # a node: (SOC, id, per-agent constraint dicts, paths); a child shares its parent's lists but the replanned entry
    heap = [(sum(len(p) - 1 for p in paths), 0, [{} for _ in st], paths)]
    expanded, next_id = 0, 1
    while heap and expanded < max_nodes:
        soc, _, cons, paths = heapq.heappop(heap)
        expanded += 1
        conflict = _cbs_first_conflict(paths)
        if conflict is None:
            return paths, 1, expanded
        for agent, cell, t in conflict:
            c = dict(cons[agent])
            c[t] = c.get(t, 0) | 1 << (cell[0] * W + cell[1])
            p = _cbs_low_level(free, W, R, Cc, st[agent], gl[agent], c, H)
            if p is None:
                continue
            ncons, npaths = list(cons), list(paths)
            ncons[agent], npaths[agent] = c, p
            heapq.heappush(heap, (soc - (len(paths[agent]) - 1) + len(p) - 1, next_id, ncons, npaths))
            next_id += 1
    return None, (2 if heap else 0), expanded


def cbs_reference(grid, starts, goals, horizon: int, max_nodes: int = 1024) -> CbsPlan:
    """Conflict-based search in pure Python, env by env with integer bitboards (the CPU path, and what the
    ``mapf_plan_cbs`` kernel is tested against bit for bit: the same actions, arrivals, outcomes and expansion
    counts).  ``starts`` / ``goals``: [B,N,2] (row, col).  See DESIGN.md §7 N4d for the search it runs."""
    grid = np.ascontiguousarray(np.asarray(grid), dtype=np.uint8)
    if grid.ndim != 2 or grid.shape[0] > 32 or grid.shape[1] > 32:
        raise ValueError(f"the planner needs one map of at most 32x32 cells, got shape {grid.shape}")
    H, K = int(horizon), int(max_nodes)
    if H < 1 or not 1 <= K <= 65536:
        raise ValueError(f"horizon must be >= 1 and max_nodes in 1..65536, got {H} and {K}")
    st = np.asarray(torch.as_tensor(starts).cpu(), dtype=np.int64)
    gl = np.asarray(torch.as_tensor(goals).cpu(), dtype=np.int64)
    B, N = st.shape[:2]
    actions = np.zeros((H, B, N), np.int8)
    arrival = np.full((B, N), -1, np.int16)
    outcome = np.zeros(B, np.uint8)
    expanded = np.zeros(B, np.int32)
    for b in range(B):
        paths, outcome[b], expanded[b] = _cbs_one(grid, st[b], gl[b], H, K)
        for i, p in enumerate(paths or ()):
            arrival[b, i] = len(p) - 1
            for t in range(len(p) - 1):
                actions[t, b, i] = _MOVES.index((p[t + 1][0] - p[t][0], p[t + 1][1] - p[t][1]))
    return _finish_cbs(torch.from_numpy(actions), torch.from_numpy(arrival), torch.from_numpy(outcome),
                       torch.from_numpy(expanded))


class PlannedPolicy:
    """A callable policy for :func:`evaluate.evaluate`: on its first call with an env (right after the evaluator's
    reset) it plans every env's layout once with :func:`plan_prioritized` (``method="prioritized"``, the default) or
    :func:`plan_cbs` with ``max_nodes`` (``method="cbs"``), then returns action row t at the t-th call (NO_OP past the
    horizon).  The planner so gets the evaluator's CSV rows, heat-map and success rate on the very layouts a trained
    policy sees with the same ``env_config``.  Handed a different env it plans again."""

    def __init__(self, method: str = "prioritized", max_nodes: int = 1024):
        if method not in ("prioritized", "cbs"):
            raise ValueError(f"method must be 'prioritized' or 'cbs', got {method!r}")
        self.method, self.max_nodes = method, int(max_nodes)
        self.plan: Plan | None = None
        self._env = None
        self._t = 0

    def __call__(self, env, out):
        if not isinstance(env, BatchedMapfEnv):
            raise ValueError("PlannedPolicy plays the multi-agent view (BatchedMapfEnv), not the CTE view")
        if env is not self._env:
            plan = plan_cbs(env, self.max_nodes) if self.method == "cbs" else plan_prioritized(env)
            self.plan, self._env, self._t = plan, env, 0
        t, self._t = self._t, self._t + 1
        if t < self.plan.actions.shape[0]:
            return self.plan.actions[t]
        return torch.zeros((env.B, env.N), dtype=torch.int8, device=env.device)


class ReplanningPolicy:
    """Rolling-horizon replanning as a callable policy for :func:`evaluate.evaluate`, lifelong or episodic: on call k
    with k % ``replan_every`` == 0 it plans the env's current state with :func:`plan_windowed` at W = ``window``, and
    it returns action row k % ``replan_every`` of the last plan.  Handed a different env it starts again at k = 0.
    Only the multi-agent view (:class:`BatchedMapfEnv`) is planned; 1 <= ``replan_every`` <= ``window``."""

    def __init__(self, window: int, replan_every: int = 1):
        window, replan_every = int(window), int(replan_every)
        if replan_every < 1 or replan_every > window:
            raise ValueError(f"replan_every must be in 1..window, got {replan_every} with window {window}")
        self.window, self.replan_every = window, replan_every
        self.plan: Plan | None = None
        self._env = None
        self._k = 0

    def __call__(self, env, out):
        if not isinstance(env, BatchedMapfEnv):
            raise ValueError("ReplanningPolicy plays the multi-agent view (BatchedMapfEnv), not the CTE view")
        if env is not self._env:
            self._env, self._k = env, 0
        j = self._k % self.replan_every
        if j == 0:
            self.plan = plan_windowed(env, self.window)
        self._k += 1
        return self.plan.actions[j]


def _gpu_name(device) -> str:
    import subprocess

    try:
        gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader",
                              "-i", str(torch.device(device).index or 0)], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as exc:
        gpu = f"nvidia-smi not readable: {exc}"
    return gpu or torch.cuda.get_device_name(device)


def benchmark(num_envs: int = 65536, num_agents: int = 16, horizon: int = 256, rounds: int = 5,
              device: str = "cuda:0") -> dict:
    """Plans/s and agent-plans/s of the kernel for ``num_envs`` Philox layouts of ``num_agents`` agents on the 32x32
    benchmark map (the evaluator's and bench.py's map) at H = ``horizon``: best of ``rounds`` timed calls after one
    warm-up, CUDA events around the launch (workspace and outputs allocated once, outside the window).  Also the
    success rate, the mean makespan of the status-1 envs and, for the same envs, the mean makespan lower bound from
    ``mapf_goal_path_lengths`` (max over agents of the single-agent distance, at least 1)."""
    from . import maps

    cfg = {"num_agents": num_agents, "sensor_range": 2, "steps_per_episode": horizon, "lifelong_mapf": False,
           "seed": 999, "grid": maps.random_obstacle_grid(32, 32, 0.30, 2026, min_free=32)}
    env = BatchedMapfEnv(cfg, num_envs, device)
    env.reset()
    plan_prioritized(env)   # warm-up: module load, distance table
    times = []
    for _ in range(rounds):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(env.device)
        e0.record()
        plan = plan_prioritized(env)
        e1.record()
        e1.synchronize()
        times.append(e0.elapsed_time(e1) / 1e3)
    ok = plan.status.bool()
    lb = env.goal_path_lengths().to(torch.int32).amax(1).clamp(min=1)
    n_ok = int(ok.sum())
    t = min(times)
    res = {"gpu": _gpu_name(env.device), "envs": num_envs, "agents": num_agents,
           "horizon": horizon, "call_s": t, "rounds_s": times, "plans_per_s": num_envs / t,
           "agent_plans_per_s": num_envs * num_agents / t, "success_rate": n_ok / num_envs,
           "mean_makespan": float(plan.makespan[ok].float().mean()) if n_ok else None,
           "mean_makespan_lower_bound": float(lb[ok].float().mean()) if n_ok else None,
           "mean_sum_of_costs": float(plan.sum_of_costs[ok].float().mean()) if n_ok else None}
    env.close()
    return res


def benchmark_windowed(num_envs: int = 65536, num_agents: int = 16, windows=(8, 16, 32), rounds: int = 5,
                       device: str = "cuda:0") -> dict:
    """The windowed planner and rolling-horizon replanning on the 32x32 benchmark map, ``num_envs`` x ``num_agents``:

    * ``kernel``: per W in ``windows``, the :func:`plan_windowed` call on the mid-episode states of a lifelong env
      (C3 config, after 64 masked steps): best of ``rounds`` calls after one warm-up, CUDA events around the call, with
      the share of status-1 envs and of agents that arrived;
    * ``lifelong``: the evaluator's step loop (:func:`evaluate._play`) at the C3 shape (lifelong, 256 steps) for
      ``ReplanningPolicy(16, 1)``, ``ReplanningPolicy(16, 4)`` and ``"masked"``: episodes/s (host clock around the loop,
      which ends in a device synchronise, after a 4-step warm-up), and over the envs the mean throughput, completion
      ratio and goals reached, and the deadlock / livelock event totals summed over the batch;
    * ``episodic``: the success rate of ``ReplanningPolicy(32, 1)`` and of :class:`PlannedPolicy` on the layouts of
      :func:`benchmark` (episodic, 256 steps).

    The GPU's name, power limit and SM clocks are read in the same call."""
    import time

    from . import maps
    from .evaluate import _play

    grid = maps.random_obstacle_grid(32, 32, 0.30, 2026, min_free=32)
    base = {"num_agents": num_agents, "sensor_range": 2, "steps_per_episode": 256, "enable_lock_metrics": True,
            "seed": 999, "grid": grid}
    res = {"envs": num_envs, "agents": num_agents, "kernel": {}, "lifelong": {}, "episodic": {}}
    env = BatchedMapfEnv(dict(base, lifelong_mapf=True), num_envs, device)
    env.reset()
    for _ in range(64):
        env.step(env.sample_actions(masked=True), auto_reset=False)
    for W in windows:
        plan = plan_windowed(env, W)   # warm-up: module load, distance table, allocator
        times = []
        for _ in range(rounds):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize(env.device)
            e0.record()
            plan = plan_windowed(env, W)
            e1.record()
            e1.synchronize()
            times.append(e0.elapsed_time(e1) / 1e3)
        t = min(times)
        res["kernel"][f"W{W}"] = {"call_s": t, "rounds_s": times, "plans_per_s": num_envs / t,
                                  "agent_plans_per_s": num_envs * num_agents / t,
                                  "status1_rate": float(plan.status.float().mean()),
                                  "arrived_rate": float((plan.arrival >= 0).float().mean())}
    env.close()
    policies = {"replan_w16_h1": lambda: ReplanningPolicy(16, 1), "replan_w16_h4": lambda: ReplanningPolicy(16, 4),
                "masked": lambda: "masked"}
    env = BatchedMapfEnv(dict(base, lifelong_mapf=True), num_envs, device)
    for name, make in policies.items():
        _play(env, make(), 4)
        torch.cuda.synchronize(env.device)
        t0 = time.perf_counter()
        acc = _play(env, make())
        dt = time.perf_counter() - t0
        info = acc["last_info"].cpu().numpy().astype(np.float64)
        g_tot = info[:, nat.I_GOALS_REACHED_TOTAL]
        res["lifelong"][name] = {
            "loop_s": dt, "episodes_per_s": num_envs / dt,
            "throughput": float((g_tot / np.maximum(info[:, nat.I_STEP_COUNT], 1)).mean()),
            "completion_ratio": float((info[:, nat.I_COMPLETED_COUNT] / num_agents).mean()),
            "goals_reached_total": float(g_tot.mean()),
            "deadlock_events_total": float(info[:, nat.I_DEADLOCK_EVENTS_TOTAL].sum()),
            "livelock_events_total": float(info[:, nat.I_LIVELOCK_EVENTS_TOTAL].sum())}
    env.close()
    for name, pol in (("replan_w32_h1", ReplanningPolicy(32, 1)), ("planned", PlannedPolicy())):
        env = BatchedMapfEnv(dict(base, lifelong_mapf=False), num_envs, device)   # a fresh env: the first reset's layouts
        acc = _play(env, pol)
        ok = acc["success"].bool()
        res["episodic"][name] = {"success_rate": float(ok.float().mean()),
                                 "mean_timesteps_of_successes": float(acc["timesteps"][ok].float().mean()) if bool(ok.any()) else None}
        env.close()
    res["gpu"] = _gpu_name(device)
    return res


def benchmark_cbs(num_envs: int = 65536, rounds: int = 5, device: str = "cuda:0") -> dict:
    """:func:`plan_cbs` per shape: ``num_envs`` Philox layouts x 4 agents on maps 2-2 and 3-1 at H = 100 and x 8 agents on
    the 32x32 benchmark map at H = 256, at K = 1024 and (32x32) K = 256, and the seven deterministic tables as single
    envs at H = 254.  Per shape: best of ``rounds`` calls after one warm-up, CUDA events around the call (workspace
    included), plans/s, the outcome split, expansions p50 / p99 / max, and the mean sum of arrivals of CBS and of
    :func:`plan_prioritized` over the envs both solve.  The GPU's name, power limit and SM clocks are read in the same
    call."""
    from . import maps

    rand32 = maps.random_obstacle_grid(32, 32, 0.30, 2026, min_free=32)
    shapes = [("2-2", maps.get_grid("ReferenceModel-2-2"), 4, 100, 1024, num_envs),
              ("3-1", maps.get_grid("ReferenceModel-3-1"), 4, 100, 1024, num_envs),
              ("rand32", rand32, 8, 256, 1024, num_envs), ("rand32", rand32, 8, 256, 256, num_envs)]
    shapes += [(f"{m}-det", maps.get_grid(f"ReferenceModel-{m}"), 2 if m.startswith("1") else 4, 254, 1024, 1)
               for m in ("1-1", "1-2", "1-3", "1-4", "2-1", "2-2", "3-1")]
    res = {"shapes": []}
    for name, grid, N, H, K, B in shapes:
        cfg = {"num_agents": N, "sensor_range": 2, "steps_per_episode": H, "lifelong_mapf": False, "seed": 999,
               "grid": grid, "deterministic": name.endswith("-det"), "env_name": f"ReferenceModel-{name[:-4]}"}
        env = BatchedMapfEnv(cfg, B, device)
        env.reset()
        plan = plan_cbs(env, K)   # warm-up: module load, distance table, allocator
        times = []
        for _ in range(rounds):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize(env.device)
            e0.record()
            plan = plan_cbs(env, K)
            e1.record()
            e1.synchronize()
            times.append(e0.elapsed_time(e1) / 1e3)
        pr = plan_prioritized(env)
        both = (plan.status.bool() & pr.status.bool()).cpu()
        ex = plan.expanded.cpu().numpy()
        oc = plan.outcome.cpu().numpy()
        t = min(times)
        row = {"map": name, "envs": B, "agents": N, "horizon": H, "max_nodes": K, "call_s": t, "rounds_s": times,
               "plans_per_s": B / t, "outcome": {str(k): int((oc == k).sum()) for k in (0, 1, 2)},
               "expanded_p50_p99_max": [float(np.percentile(ex, 50)), float(np.percentile(ex, 99)), int(ex.max())],
               "prioritized_status1": int(pr.status.sum()), "both_solved": int(both.sum()),
               "mean_soc_cbs": float(plan.sum_of_costs.cpu()[both].float().mean()) if bool(both.any()) else None,
               "mean_soc_prioritized": float(pr.sum_of_costs.cpu()[both].float().mean()) if bool(both.any()) else None}
        if B == 1:
            row["arrival"] = plan.arrival[0].tolist()
            row["prioritized_arrival"] = pr.arrival[0].tolist()
        res["shapes"].append(row)
        env.close()
    res["gpu"] = _gpu_name(device)
    return res


if __name__ == "__main__":
    import json
    import sys

    flags = sys.argv[1:]
    print(json.dumps(benchmark_windowed() if "--windowed" in flags else benchmark_cbs() if "--cbs" in flags
                     else benchmark()))
