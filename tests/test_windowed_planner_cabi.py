"""CPU-side checks of the windowed planner (no GPU): the C ABI of mapf_plan_windowed (export, declaration, refusals
before any device work) and the PyTorch reference plan_reference(window=True), whose status-1 plans must replay through
the CPU oracle of a lifelong env for W steps -- every agent on its planned cells, no failed move, and an agent that
arrived on the cell of its goal at planning time from its arrival to W, whatever goal the oracle assigns it meanwhile --
and which must equal the one-shot plan of plan_reference at W = H on the envs where that plan has status 1."""
import ctypes as C
import re

import numpy as np
import pytest
import torch

import test_planner_cabi as pc
from dl_reference_models_b200 import _native as nat
from dl_reference_models_b200 import maps
from dl_reference_models_b200.planner import ReplanningPolicy, _components, _distances, plan_reference

RAND32 = maps.random_obstacle_grid(32, 32, 0.30, 2026, min_free=64)


def test_export_and_declaration():
    L = nat.lib()
    assert "mapf_plan_windowed" in nat.EXPORTS and hasattr(L, "mapf_plan_windowed")
    header = (pc.REPO / "include" / "mapf_b200.h").read_text()
    assert re.search(r"int mapf_plan_windowed\(mapf_handle \*h, const mapf_plan_args \*args, void \*stream\);", header)


@pytest.mark.parametrize("kw", pc.INVALID + [{"num_agents": 33}], ids=[str(k) for k in pc.INVALID + [{"num_agents": 33}]])
def test_windowed_refuses_before_any_device_work(kw):
    """The refusals of mapf_plan_prioritized, before the handle is read (FAKE is never dereferenced)."""
    want = nat.ERR_UNSUPPORTED if kw == {"num_agents": 33} else nat.ERR_INVALID_ARG
    assert nat.lib().mapf_plan_windowed(pc.FAKE, C.byref(pc._args(**kw)), None) == want


def test_windowed_refuses_null_handle_and_args():
    L = nat.lib()
    assert L.mapf_plan_windowed(None, C.byref(pc._args()), None) == nat.ERR_INVALID_ARG
    assert L.mapf_plan_windowed(pc.FAKE, None, None) == nat.ERR_INVALID_ARG


def test_replanning_policy_refusals():
    for w, h in ((4, 0), (4, 5), (1, 2), (0, 1)):
        with pytest.raises(ValueError):
            ReplanningPolicy(w, h)
    ReplanningPolicy(4, 4)
    with pytest.raises(ValueError):
        ReplanningPolicy(4, 1)(object(), None)          # not the multi-agent view (e.g. the CTE env)


def test_distances_match_a_breadth_first_search():
    grid = maps.get_grid("ReferenceModel-2-1")
    d = _distances(grid)
    Rr, Cc = grid.shape
    for src in (0, 7, Rr * Cc // 2, Rr * Cc - 1):
        want = np.full(Rr * Cc, 255)
        if grid.reshape(-1)[src] == 0:
            want[src], frontier, k = 0, [src], 0
            while frontier:
                k += 1
                nxt = []
                for c in frontier:
                    r, q = divmod(c, Cc)
                    for rr, qq in ((r - 1, q), (r + 1, q), (r, q - 1), (r, q + 1)):
                        if 0 <= rr < Rr and 0 <= qq < Cc and grid[rr, qq] == 0 and want[rr * Cc + qq] == 255:
                            want[rr * Cc + qq] = k
                            nxt.append(rr * Cc + qq)
                frontier = nxt
        assert np.array_equal(d[src], want)


# ------------------------------------------------------------------ the reference against the env's oracle
def layouts_with_unreachable_goals(grid, B, N, seed, every=4):
    """pc.random_layouts (start = goal for one agent of every 3rd env), and in every ``every``-th env agent 0's goal
    moved to a free cell of another connected component where the map has one (a goal the distance table cannot
    reach; the oracle takes any free cell as a goal, not an obstacle, so a walled-off pocket stands for it)."""
    st, gl = pc.random_layouts(grid, B, N, seed, same_cell_every=3)
    comp = _components(grid)
    rng = np.random.default_rng(seed + 1)
    for b in range(0, B, every):
        s = st[b, 0]
        taken = {tuple(x) for x in np.concatenate([st[b], gl[b]])}
        other = [c for c in np.argwhere((comp > 0) & (comp != comp[s[0], s[1]])) if tuple(c) not in taken]
        if other:
            gl[b, 0] = other[rng.integers(len(other))]
    return st, gl


def replay_window_on_lifelong_oracle(grid, starts, goals, plan, W):
    """Play W steps of every status-1 windowed plan on a lifelong oracle env; returns the number of envs replayed."""
    from oracle.oracle import OracleBatch

    idx = np.flatnonzero(plan.status.cpu().numpy() == 1)
    if len(idx) == 0:
        return 0
    acts = plan.actions.cpu().numpy()[:, idx]
    arr = plan.arrival.cpu().numpy()[idx].astype(int)
    N = starts.shape[1]
    cfg = {"num_agents": N, "sensor_range": 1, "steps_per_episode": W + 4, "lifelong_mapf": True}
    ob = OracleBatch(cfg, grid, len(idx))
    ob.reset(1, starts[idx], goals[idx])
    pos = starts[idx].astype(int)
    gl = goals[idx].astype(int)
    for t in range(W):
        a = acts[t].astype(int)
        buf = ob.step(acts[t])
        pos = pos + np.stack([pc.DR[a], pc.DC[a]], -1)
        assert np.array_equal(ob.state()["positions"].astype(int), pos), f"positions differ from the plan at step {t + 1}"
        assert not buf["failed_move"].any(), f"a planned move failed at step {t + 1}"
        held = (arr >= 0) & (arr <= t + 1)
        assert (pos == gl).all(-1)[held].all(), f"an agent left its goal after arriving, step {t + 1}"
        assert not buf["terminated"].any() and not buf["truncated"].any()
    return len(idx)


def _branches(grid, st, gl, plan):
    """Counts of (arrivals, end cells of agents whose goal is the target, end cells of agents whose start is the target
    (unreachable goal), status-0 envs)."""
    d = _distances(grid)
    Cc = grid.shape[1]
    s = st.astype(int)
    g = gl.astype(int)
    unreach = d[g[..., 0] * Cc + g[..., 1], s[..., 0] * Cc + s[..., 1]] == 255
    arr = plan.arrival.numpy()
    ok = (plan.status.numpy() == 1)[:, None]
    return (int((arr >= 0).sum()), int((ok & (arr < 0) & ~unreach).sum()), int((ok & unreach).sum()),
            int((plan.status.numpy() == 0).sum()))


@pytest.mark.parametrize("name", pc.MAPS)
@pytest.mark.parametrize("W", [1, 8, 32])
def test_windowed_plans_replay_on_the_lifelong_oracle_reference_maps(name, W):
    grid = maps.get_grid(name)
    n = 2 if name.startswith("ReferenceModel-1") else 4
    st, gl = layouts_with_unreachable_goals(grid, 48, n, seed=len(name) + W)
    plan = plan_reference(grid, st, gl, W, window=True)
    assert replay_window_on_lifelong_oracle(grid, st, gl, plan, W) == int(plan.status.sum())
    assert int(plan.status.sum()) >= 24
    arrived, ends, _, _ = _branches(grid, st, gl, plan)
    assert arrived > 0 and (ends > 0 or W == 32)


@pytest.mark.parametrize("N", [2, 4, 16, 32])
@pytest.mark.parametrize("W", [1, 8, 32])
def test_windowed_plans_replay_on_the_lifelong_oracle_random_32x32(N, W):
    st, gl = layouts_with_unreachable_goals(RAND32, 24, N, seed=N * 7 + W)
    plan = plan_reference(RAND32, st, gl, W, window=True)
    replayed = replay_window_on_lifelong_oracle(RAND32, st, gl, plan, W)
    assert replayed == int(plan.status.sum()) and replayed >= 2
    arrived, ends, unreach, _ = _branches(RAND32, st, gl, plan)
    assert arrived > 0 and ends > 0 and unreach > 0
    arr = plan.arrival.numpy()
    ok = plan.status.numpy() == 1
    # makespan and sum of costs only where every agent arrived
    full = ok & (arr >= 0).all(1)
    assert np.array_equal(plan.makespan.numpy() >= 0, full)
    assert np.array_equal(plan.makespan.numpy()[full], np.maximum(arr[full].max(1), 1))


def test_windowed_failures_and_edge_cases():
    grid = maps.get_grid("ReferenceModel-1-3")
    free = np.argwhere(grid == 0)
    a, b, c, d = free[:4]
    st = np.array([[a, b], [a, b], [a, b]], np.int16)
    gl = np.array([[a, d], [c, d], [a, b]], np.int16)
    st[2, 0] = (-1, 0)                                    # a start off the map: failure, status 0
    plan = plan_reference(grid, st, gl, 6, window=True)
    arr = plan.arrival.numpy()
    assert arr[0, 0] == 0 and arr[2, 0] == -1 and plan.status.numpy()[2] == 0 and arr[2, 1] == 0
    assert (plan.actions.numpy()[:, 2, 0] == 0).all()
    # a goal out of reach within W: the path ends at W on the wavefront's cell nearest the goal
    far = plan_reference(grid, np.array([[a]], np.int16), np.array([[free[-1]]], np.int16), 1, window=True)
    assert int(far.arrival[0, 0]) == -1 and int(far.status[0]) == 1 and int(far.makespan[0]) == -1
    dist = _distances(grid)
    Cc = grid.shape[1]
    end = a + np.array([pc.DR[int(far.actions[0, 0, 0])], pc.DC[int(far.actions[0, 0, 0])]])
    g = free[-1][0] * Cc + free[-1][1]
    g = g if dist[g, a[0] * Cc + a[1]] != 255 else a[0] * Cc + a[1]     # the target: the goal, or the start
    nbrs = [a + np.array([pc.DR[k], pc.DC[k]]) for k in range(5)]
    best = min((dist[g, r * Cc + q], r * Cc + q) for r, q in nbrs if 0 <= r < grid.shape[0] and 0 <= q < Cc and grid[r, q] == 0)
    assert (end[0] * Cc + end[1]) == best[1]
    # the agent ahead in a dead end: an agent boxed in by a lower index's path has an empty wavefront
    corridor = np.ones((3, 5), np.uint8)
    corridor[1, :] = 0
    st = np.array([[[1, 0], [1, 1]]], np.int16)
    gl = np.array([[[1, 4], [1, 0]]], np.int16)          # agent 0 passes through agent 1's cell; agent 1 cannot leave
    plan = plan_reference(corridor, st, gl, 8, window=True)
    assert int(plan.status[0]) == 0 and int(plan.arrival[0, 1]) == -1


@pytest.mark.parametrize("name", pc.MAPS + ("rand32",))
def test_episodic_equivalence_at_w_equal_h(name):
    """On the envs where the one-shot plan at H has status 1, the windowed plan at W = H is the same, bit for bit."""
    grid = RAND32 if name == "rand32" else maps.get_grid(name)
    N = 16 if name == "rand32" else (2 if name.startswith("ReferenceModel-1") else 4)
    H = 128 if name == "rand32" else 100
    st, gl = pc.random_layouts(grid, 32, N, seed=3, same_cell_every=4)
    one = plan_reference(grid, st, gl, H)
    win = plan_reference(grid, st, gl, H, window=True)
    ok = one.status.bool()
    assert int(ok.sum()) >= 2
    assert torch.equal(win.actions[:, ok], one.actions[:, ok]) and torch.equal(win.arrival[ok], one.arrival[ok])
    assert torch.equal(win.status[ok], one.status[ok]) and torch.equal(win.makespan[ok], one.makespan[ok])
    assert torch.equal(win.sum_of_costs[ok], one.sum_of_costs[ok])
