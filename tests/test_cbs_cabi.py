"""CPU-side checks of conflict-based search (no GPU): the C ABI of mapf_plan_cbs (struct layout against the header,
exports, the workspace formula, refusals before any device work) and the pure Python reference
(planner.cbs_reference): its plans replay through the CPU oracle of the env, its sums of arrivals are optimal against
an exhaustive joint search under the env's move rule, and it never does worse than prioritized planning."""
import ctypes as C
import itertools
import shutil
import subprocess
from pathlib import Path

import numpy as np
import pytest

from dl_reference_models_b200 import _native as nat
from dl_reference_models_b200 import maps
from dl_reference_models_b200.planner import PlannedPolicy, cbs_reference, plan_reference
from test_planner_cabi import GOLD, MAPS, _det_layout, random_layouts, replay_on_oracle

REPO = Path(__file__).resolve().parents[1]
DET_MAPS = [m for m in MAPS if m != "ReferenceModel-2-1-b"]   # the seven maps with a deterministic table


def _n(name):
    return 2 if name.startswith("ReferenceModel-1") else 4


@pytest.mark.skipif(shutil.which("gcc") is None, reason="needs gcc")
def test_ctypes_structure_matches_the_header_layout(tmp_path):
    name, cls = "mapf_cbs_args", nat.MapfCbsArgs
    fields = [f for f, _ in cls._fields_]
    src = tmp_path / "probe.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "mapf_b200.h"\nint main(void) {\n'
                   f'    printf("%zu\\n", sizeof({name}));\n'
                   + "".join(f'    printf("%zu\\n", offsetof({name}, {f}));\n' for f in fields)
                   + "    return 0;\n}\n")
    exe = tmp_path / "probe"
    subprocess.run(["gcc", "-std=c99", "-I", str(REPO / "include"), "-o", str(exe), str(src)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    assert got == [C.sizeof(cls)] + [getattr(cls, f).offset for f in fields]


def _ceil16(x):
    return -(-x // 16) * 16


def test_exports_and_workspace_bytes():
    L = nat.lib()
    for name in ("mapf_cbs_workspace_bytes", "mapf_plan_cbs"):
        assert name in nat.EXPORTS and hasattr(L, name)
    # 16-byte env counter; per env: node records + open-list keys (24 bytes a node), the root's arrivals (64), the
    # constraint and wavefront planes, one int8 action path per root agent and per child
    for rows, cols, B, N, H, K in ((32, 32, 65536, 8, 256, 1024), (10, 20, 3, 4, 7, 1), (5, 5, 1, 1, 1, 65536)):
        want = 16 + B * _ceil16(24 * (2 * K + 1) + 64 + 8 * (H + 1) * rows + (N + 2 * K) * _ceil16(H))
        assert L.mapf_cbs_workspace_bytes(rows, cols, B, N, H, K) == want
    assert L.mapf_cbs_workspace_bytes(32, 32, 65536, 8, 256, 1024) == 16 + 65536 * 641376   # 42 GB
    for bad in ((0, 5, 1, 1, 1, 1), (5, 0, 1, 1, 1, 1), (5, 5, 0, 1, 1, 1), (5, 5, 1, 0, 1, 1), (5, 5, 1, 1, 0, 1),
                (5, 5, 1, 1, 1, 0), (5, 5, 1, 1, 1, 65537), (5, 5, 1, 1, 32768, 1)):
        assert L.mapf_cbs_workspace_bytes(*bad) == nat.ERR_INVALID_ARG
    assert L.mapf_cbs_workspace_bytes(33, 5, 1, 1, 1, 1) == nat.ERR_UNSUPPORTED
    assert L.mapf_cbs_workspace_bytes(5, 33, 1, 1, 1, 1) == nat.ERR_UNSUPPORTED
    assert L.mapf_cbs_workspace_bytes(5, 5, 1, 33, 1, 1) == nat.ERR_UNSUPPORTED


FAKE = C.c_void_p(16)


def _args(**kw):
    a = nat.MapfCbsArgs(num_envs=4, num_agents=3, horizon=8, max_nodes=16, starts=FAKE, goals=FAKE,
                        distance_table=FAKE, workspace=FAKE, workspace_bytes=1 << 20, actions=FAKE, arrival=FAKE,
                        status=FAKE, expanded=FAKE)
    for k, v in kw.items():
        setattr(a, k, v)
    return a


INVALID = ([{k: None} for k in ("starts", "goals", "distance_table", "workspace", "actions", "arrival", "status",
                                "expanded")]
           + [{"num_envs": 0}, {"num_agents": 0}, {"horizon": 0}, {"horizon": -3}, {"horizon": 32768},
              {"reserved": 1}, {"max_nodes": 0}, {"max_nodes": -1}, {"max_nodes": 65537}])


@pytest.mark.parametrize("kw", INVALID + [{"num_agents": 33}], ids=[str(k) for k in INVALID + [{"num_agents": 33}]])
def test_cbs_refuses_before_any_device_work(kw):
    """Argument checks come before the handle is read (FAKE is never dereferenced)."""
    want = nat.ERR_UNSUPPORTED if kw == {"num_agents": 33} else nat.ERR_INVALID_ARG
    assert nat.lib().mapf_plan_cbs(FAKE, C.byref(_args(**kw)), None) == want


def test_cbs_refuses_null_handle_and_args():
    L = nat.lib()
    assert L.mapf_plan_cbs(None, C.byref(_args()), None) == nat.ERR_INVALID_ARG
    assert L.mapf_plan_cbs(FAKE, None, None) == nat.ERR_INVALID_ARG


# ------------------------------------------------------------------ the reference against the env's oracle
def _check_plan(plan):
    """Outcome 1 <=> status 1; other outcomes carry NO_OPs and arrival -1."""
    oc, st = plan.outcome.numpy(), plan.status.numpy()
    assert set(np.unique(oc)) <= {0, 1, 2} and np.array_equal(st == 1, oc == 1)
    arr, acts = plan.arrival.numpy(), plan.actions.numpy()
    assert (arr[oc != 1] == -1).all() and (acts[:, oc != 1] == 0).all() and (arr[oc == 1] >= 0).all()
    assert (plan.expanded.numpy()[oc == 1] >= 1).all()


@pytest.mark.parametrize("name", DET_MAPS)
def test_deterministic_tables_replay_on_the_oracle(name):
    grid = maps.get_grid(name)
    s0, g0 = _det_layout(name, _n(name))
    plan = cbs_reference(grid, s0[None], g0[None], 254)
    _check_plan(plan)
    assert int(plan.outcome[0]) == 1
    assert replay_on_oracle(grid, s0[None], g0[None], plan, 254) == 1


@pytest.mark.parametrize("name", MAPS)
def test_random_layouts_replay_on_the_oracle(name):
    grid = maps.get_grid(name)
    H = 100
    st, gl = random_layouts(grid, 32, _n(name), seed=7 * len(name), same_cell_every=5)
    plan = cbs_reference(grid, st, gl, H, max_nodes=256)
    _check_plan(plan)
    assert replay_on_oracle(grid, st, gl, plan, H) == int(plan.status.sum()) >= 8


@pytest.mark.parametrize("N", [2, 4, 8])
def test_random_32x32_layouts_replay_on_the_oracle(N):
    grid = maps.random_obstacle_grid(32, 32, 0.30, 2026, min_free=32)
    H = 256
    st, gl = random_layouts(grid, 16, N, seed=100 + N, same_cell_every=3)
    plan = cbs_reference(grid, st, gl, H, max_nodes=128)
    _check_plan(plan)
    assert replay_on_oracle(grid, st, gl, plan, H) == int(plan.status.sum()) >= 2
    # the map has walled-off pockets: an unreachable goal ends the search at the root
    pr = plan_reference(grid, st, gl, H)
    root0 = plan.expanded.numpy() == 0
    assert root0.any() and (plan.outcome.numpy()[root0] == 0).all()
    assert (pr.status.numpy()[root0] == 0).all()


def test_exact_numbers_on_the_deterministic_tables():
    def run(name, K=1024):
        grid = maps.get_grid(name)
        s0, g0 = _det_layout(name, _n(name))
        return cbs_reference(grid, s0[None], g0[None], 254, max_nodes=K)

    for name in ("ReferenceModel-1-1", "ReferenceModel-2-2"):   # prioritized planning fails both
        assert int(run(name).outcome[0]) == 1
        assert int(plan_reference(maps.get_grid(name), *(x[None] for x in _det_layout(name, _n(name))), 254).status[0]) == 0
    p = run("ReferenceModel-2-1")
    assert int(p.sum_of_costs[0]) == 45 and p.arrival.numpy()[0].tolist() == [11, 15, 5, 14]
    p = run("ReferenceModel-1-2")
    assert int(p.outcome[0]) == 1 and int(p.expanded[0]) == 511
    p = run("ReferenceModel-1-2", K=256)
    assert int(p.outcome[0]) == 2 and int(p.expanded[0]) == 256
    assert (p.actions.numpy() == 0).all() and (p.arrival.numpy() == -1).all()


# ------------------------------------------------------------------ optimality against an exhaustive search
DR = (0, -1, 0, 1, 0)
DC = (0, 0, 1, 0, -1)


def brute_force_soc(grid, starts, goals, H):
    """The least sum of arrivals of a plan within H under the env's move rule, or None: a search over joint states
    (positions, finished flags) by time layer.  An agent on its goal may finish and then stays for good; agents move in
    index order and a move fails off the map, into an obstacle, into a cell a lower index holds after its move, or into
    one a higher index holds before its move.  The value of a state is the sum of the finish times so far."""
    R, Cc = grid.shape
    N = len(starts)
    st = tuple(tuple(int(v) for v in p) for p in starts)
    gl = tuple(tuple(int(v) for v in p) for p in goals)

    def finishes(pos, done, t, cost, out):
        free = [i for i in range(N) if not done[i] and pos[i] == gl[i]]
        for k in range(len(free) + 1):
            for sub in itertools.combinations(free, k):
                d = list(done)
                for i in sub:
                    d[i] = True
                key = (pos, tuple(d))
                c = cost + t * len(sub)
                if c < out.get(key, 1 << 30):
                    out[key] = c

    layer = {}
    finishes(st, (False,) * N, 0, 0, layer)
    best = None
    for t in range(0, H + 1):
        for (pos, done), c in layer.items():
            if all(done):
                best = c if best is None else min(best, c)
        if t == H:
            break
        nxt = {}
        for (pos, done), c in layer.items():
            if all(done):
                continue
            choices = [range(1) if done[i] else range(5) for i in range(N)]
            for acts in itertools.product(*choices):
                new = list(pos)
                ok = True
                for i, a in enumerate(acts):
                    r, c2 = pos[i][0] + DR[a], pos[i][1] + DC[a]
                    if a and (not (0 <= r < R and 0 <= c2 < Cc) or grid[r, c2] or (r, c2) in new[:i]
                              or (r, c2) in pos[i + 1:]):
                        ok = False
                        break
                    new[i] = (r, c2)
                if ok:
                    finishes(tuple(new), done, t + 1, c, nxt)
        layer = nxt
    return best


def _small_instances():
    rng = np.random.default_rng(11)
    out = []
    for name in ("ReferenceModel-1-1", "ReferenceModel-1-2", "ReferenceModel-1-3"):
        grid = maps.get_grid(name)
        for N in (2, 3):
            st, gl = random_layouts(grid, 4, N, seed=N * 31 + len(out), same_cell_every=3)
            out += [(grid, st[b], gl[b], 14) for b in range(len(st))]
    for k in range(10):
        grid = (rng.random((5, 5)) < 0.25).astype(np.uint8)
        if (grid == 0).sum() < 8:
            continue
        N = 2 + k % 2
        st, gl = random_layouts(grid, 2, N, seed=k, same_cell_every=2)
        out += [(grid, st[b], gl[b], 10) for b in range(len(st))]
    return out


def test_optimal_against_an_exhaustive_joint_search():
    seen = {0: 0, 1: 0}
    for grid, s, g, H in _small_instances():
        plan = cbs_reference(grid, s[None], g[None], H, max_nodes=4096)
        oc = int(plan.outcome[0])
        if oc == 2:
            continue
        best = brute_force_soc(grid, s, g, H)
        seen[oc] += 1
        if oc == 1:
            assert int(plan.sum_of_costs[0]) == best, (grid.tolist(), s.tolist(), g.tolist())
        else:
            assert best is None, (grid.tolist(), s.tolist(), g.tolist())
    assert seen[0] >= 1 and seen[1] >= 10, seen


# ------------------------------------------------------------------ against prioritized planning and the golden A*
@pytest.mark.parametrize("name", MAPS)
def test_not_worse_than_prioritized_and_above_the_golden_astar(name):
    grid = maps.get_grid(name)
    H = 100
    st, gl = random_layouts(grid, 24, _n(name), seed=3 + len(name))
    cbs = cbs_reference(grid, st, gl, H, max_nodes=256)
    pr = plan_reference(grid, st, gl, H)
    both = (cbs.status.numpy() == 1) & (pr.status.numpy() == 1)
    assert both.any()
    assert (cbs.sum_of_costs.numpy()[both] <= pr.sum_of_costs.numpy()[both]).all()
    with np.load(GOLD) as z:
        fx = {k: z[k] for k in z.files}
    key = name.replace("ReferenceModel-", "m").replace("-", "_")
    if f"{key}_cbs_starts" in fx:
        p = cbs_reference(grid, fx[f"{key}_cbs_starts"][None], fx[f"{key}_cbs_goals"][None], 254, max_nodes=1024)
        if int(p.outcome[0]) == 1:
            assert (p.arrival.numpy()[0] >= fx[f"{key}_cbs_root_len"]).all()


# ------------------------------------------------------------------ edge cases
def test_refused_layouts_end_without_a_search():
    grid = maps.get_grid("ReferenceModel-1-3")
    free = np.argwhere(grid == 0)
    obstacle = np.argwhere(grid == 1)[0]
    a, b, c, d = free[:4]
    st = np.array([[a, b], [a, b], [a, b], [a, a], [a, b], [a, b]], np.int16)
    gl = np.array([[c, d], [c, d], [c, d], [c, d], [c, c], [obstacle, d]], np.int16)
    st[1, 0] = (-1, 0)                                     # off the map
    st[2, 1] = obstacle                                    # on an obstacle
    #   env 3: a repeated start; env 4: a repeated goal; env 5: a goal on an obstacle
    plan = cbs_reference(grid, st, gl, 30)
    _check_plan(plan)
    assert int(plan.outcome[0]) == 1 and int(plan.expanded[0]) >= 1
    assert (plan.outcome.numpy()[1:] == 0).all() and (plan.expanded.numpy()[1:] == 0).all()
    # a goal too far for the horizon: no path at the root
    far = cbs_reference(grid, np.array([[a]], np.int16), np.array([[free[-1]]], np.int16), 1)
    assert int(far.outcome[0]) == 0 and int(far.expanded[0]) == 0
    # everyone on its goal: the root is the answer with arrival 0
    home = cbs_reference(grid, np.array([[a, b]], np.int16), np.array([[a, b]], np.int16), 5)
    assert int(home.outcome[0]) == 1 and int(home.expanded[0]) == 1 and int(home.makespan[0]) == 1
    with pytest.raises(ValueError):
        cbs_reference(grid, st, gl, 10, max_nodes=0)
    with pytest.raises(ValueError):
        cbs_reference(np.zeros((33, 4), np.uint8), st, gl, 10)


def test_planned_policy_default_is_prioritized(monkeypatch):
    """PlannedPolicy() still plans with plan_prioritized; PlannedPolicy("cbs", K) with plan_cbs(env, K)."""
    import torch

    from dl_reference_models_b200 import planner
    from dl_reference_models_b200.batched_env import BatchedMapfEnv

    calls = []
    rows = torch.arange(6, dtype=torch.int8).reshape(3, 1, 2)
    fake = lambda kind: lambda env, *a: calls.append((kind, a)) or planner.Plan(rows, *[None] * 4)  # noqa: E731
    monkeypatch.setattr(planner, "plan_prioritized", fake("prioritized"))
    monkeypatch.setattr(planner, "plan_cbs", fake("cbs"))
    env = object.__new__(BatchedMapfEnv)
    assert torch.equal(PlannedPolicy()(env, None), rows[0]) and calls == [("prioritized", ())]
    pol = PlannedPolicy("cbs", max_nodes=64)
    assert torch.equal(pol(env, None), rows[0]) and torch.equal(pol(env, None), rows[1])
    assert calls[1:] == [("cbs", (64,))]
    with pytest.raises(ValueError):
        PlannedPolicy("astar")
