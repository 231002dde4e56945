"""The windowed planner kernel (mapf_plan_windowed) against the PyTorch reference bit for bit, on fresh layouts and on
mid-episode lifelong states, its episodic equivalence with mapf_plan_prioritized at W = H, its refusals on a real
handle, and ReplanningPolicy through the batched evaluator (lifelong against a hand loop, episodic against
PlannedPolicy)."""
import ctypes as C

import numpy as np
import pytest
import torch

from dl_reference_models_b200 import _native as nat
from dl_reference_models_b200 import maps
from dl_reference_models_b200.batched_env import BatchedMapfEnv
from dl_reference_models_b200.evaluate import _play, evaluate
from dl_reference_models_b200.planner import (PlannedPolicy, ReplanningPolicy, plan_prioritized, plan_reference,
                                              plan_windowed)
from test_gpu_planner import RAND32, _grid, layouts

pytestmark = pytest.mark.gpu

DR = torch.tensor([0, -1, 0, 1, 0])
DC = torch.tensor([0, 0, 1, 0, -1])


def lifelong_states(grid, B, N, seed, steps=24):
    """The positions and current goals of a lifelong env after ``steps`` masked steps, with the goal of the last agent
    of every 11th env moved onto an obstacle (a target the distance table cannot reach) and the start of agent 0 of
    every 13th env off the map (a failure); returns the env (its handle plans) and the [B,N,2] starts and goals."""
    env = BatchedMapfEnv({"grid": grid, "num_agents": N, "sensor_range": 1, "seed": seed, "lifelong_mapf": True,
                          "steps_per_episode": 1000}, B)
    env.reset()
    for _ in range(steps):
        env.step(env.sample_actions(masked=True), auto_reset=False)
    st, gl = env.state["positions"].clone(), env.state["goals"].clone()
    b = torch.arange(B, device="cuda")
    walls = np.argwhere(grid == 1)
    if len(walls):
        gl[b % 11 == 5, N - 1] = torch.as_tensor(walls[0], dtype=torch.int16, device="cuda")
    st[b % 13 == 6, 0] = torch.tensor([-1, 0], dtype=torch.int16, device="cuda")
    return env, st.contiguous(), gl.contiguous()


BRANCHES = {}
CASES = [("2-1", 1, 1003, 1, "fresh"), ("2-1", 4, 1003, 8, "mid"), ("2-1", 2, 65536, 32, "mid"),
         ("3-1", 2, 1003, 256, "fresh"), ("3-1", 16, 1003, 8, "mid"), ("3-1", 4, 65536, 32, "fresh"),
         ("rand32", 16, 1003, 256, "mid"), ("rand32", 32, 1003, 32, "mid"), ("rand32", 32, 1003, 1, "fresh"),
         ("rand32", 4, 65536, 8, "fresh"), ("rand32", 16, 65536, 32, "mid"), ("rand32", 16, 65536, 256, "fresh")]


@pytest.mark.parametrize("name,N,B,W,kind", CASES, ids=[f"{c[0]}-N{c[1]}-B{c[2]}-W{c[3]}-{c[4]}" for c in CASES])
def test_kernel_equals_the_reference(name, N, B, W, kind):
    grid = _grid(name)
    if kind == "mid":
        env, st, gl = lifelong_states(grid, B, N, seed=B + N + W)
    else:
        env = BatchedMapfEnv({"grid": grid, "num_agents": min(N, 8), "sensor_range": 1, "seed": 5}, 4)
        st, gl = layouts(grid, B, N, seed=B + N + W)
    got = plan_windowed(env, W, st, gl)
    ref = plan_reference(grid, st, gl, W, device="cuda", window=True)
    assert torch.equal(got.arrival, ref.arrival)
    assert torch.equal(got.status, ref.status)
    assert torch.equal(got.actions, ref.actions)
    assert torch.equal(got.makespan, ref.makespan) and torch.equal(got.sum_of_costs, ref.sum_of_costs)
    # the branches this case reached (test_every_branch_occurs checks that the cases reach all of them)
    Rr, Cc = grid.shape
    s, g = st.to(torch.int64), gl.to(torch.int64)
    inside = lambda p: (p[..., 0] >= 0) & (p[..., 0] < Rr) & (p[..., 1] >= 0) & (p[..., 1] < Cc)  # noqa: E731
    on_map = inside(s) & inside(g)
    table = env.distance_table().to(torch.int64)
    cell = lambda p: (p[..., 0] * Cc + p[..., 1]).clamp(0, Rr * Cc - 1)  # noqa: E731
    d = table[cell(g), cell(s)]
    ok = got.status.bool()[:, None]
    arr = got.arrival
    BRANCHES[(name, N, B, W, kind)] = {
        "arrival": int((arr >= 0).sum()),
        "end cell": int((ok & (arr < 0) & (d != 255)).sum()),
        "unreachable target": int((ok & (d == 255) & on_map).sum()),
        "failure": int(((got.status == 0) & on_map.all(1)).sum())}
    print(name, N, B, W, kind, BRANCHES[(name, N, B, W, kind)])
    # an agent arrives no earlier than its single-agent distance
    a = arr >= 0
    assert bool((arr[a].to(torch.int64) >= d[a]).all()) and bool((d[a] != 255).all())
    env.close()


def test_every_branch_occurs():
    """Arrivals, end cells towards a reachable goal, end cells of agents whose target is their start (unreachable
    goal), and failures of agents on the map (an emptied wavefront) all occur in the cases above."""
    if len(BRANCHES) < len(CASES):
        pytest.skip("needs every case of test_kernel_equals_the_reference in the same run")
    for k in ("arrival", "end cell", "unreachable target", "failure"):
        assert sum(v[k] for v in BRANCHES.values()) > 0, k


@pytest.mark.parametrize("name,N,B,H", [("2-1", 4, 1003, 64), ("3-1", 16, 1003, 256), ("rand32", 16, 65536, 256)])
def test_episodic_equivalence_with_the_one_shot_plan(name, N, B, H):
    grid = _grid(name)
    env = BatchedMapfEnv({"grid": grid, "num_agents": min(N, 8), "sensor_range": 1, "seed": 5, "steps_per_episode": H}, 4)
    st, gl = layouts(grid, B, N, seed=3 * B + N)
    one = plan_prioritized(env, st, gl, H)
    win = plan_windowed(env, H, st, gl)
    ok = one.status.bool()
    assert bool(ok.any())
    assert torch.equal(win.actions[:, ok], one.actions[:, ok]) and torch.equal(win.arrival[ok], one.arrival[ok])
    assert bool(win.status[ok].bool().all())
    env.close()


def test_refusals_on_a_handle():
    L = nat.lib()
    env = BatchedMapfEnv({"grid": np.zeros((8, 40), np.uint8), "num_agents": 2, "sensor_range": 1, "seed": 1}, 2)
    with pytest.raises(nat.MapfError) as e:
        plan_windowed(env, 8)
    assert e.value.code == nat.ERR_UNSUPPORTED
    env.close()
    grid = maps.get_grid("ReferenceModel-2-1")
    env = BatchedMapfEnv({"grid": grid, "num_agents": 2, "sensor_range": 1, "seed": 1, "lifelong_mapf": True}, 2)
    env.reset()
    need = L.mapf_plan_workspace_bytes(*grid.shape, 2, 16)
    ws = torch.zeros(need, dtype=torch.uint8, device="cuda")
    out = {"actions": torch.zeros((16, 2, 2), dtype=torch.int8, device="cuda"),
           "arrival": torch.zeros((2, 2), dtype=torch.int16, device="cuda"),
           "status": torch.full((2,), 7, dtype=torch.uint8, device="cuda")}
    p = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
    args = nat.MapfPlanArgs(num_envs=2, num_agents=2, horizon=16, starts=p(env.state["positions"]),
                            goals=p(env.state["goals"]), distance_table=p(env.distance_table()), workspace=p(ws),
                            workspace_bytes=need - 1, **{k: p(v) for k, v in out.items()})
    assert L.mapf_plan_windowed(env._h, C.byref(args), None) == nat.ERR_INVALID_ARG
    args.workspace_bytes, args.reserved = need, 1
    assert L.mapf_plan_windowed(env._h, C.byref(args), None) == nat.ERR_INVALID_ARG
    torch.cuda.synchronize()
    assert (out["status"] == 7).all()                           # nothing was launched
    args.reserved = 0
    assert L.mapf_plan_windowed(env._h, C.byref(args), None) == 0   # a lifelong env is planned
    torch.cuda.synchronize()
    assert bool((out["status"] <= 1).all())
    per_env = BatchedMapfEnv({"grid": np.stack([grid, grid]), "num_agents": 2, "sensor_range": 1, "seed": 1}, 2)
    with pytest.raises(nat.MapfError) as e:
        plan_windowed(per_env, 8)
    assert e.value.code == nat.ERR_UNSUPPORTED


LIFELONG = {"grid": RAND32, "num_agents": 16, "sensor_range": 2, "steps_per_episode": 64, "lifelong_mapf": True,
            "seed": 2468}


def hand_loop(cfg, B, window, h):
    """Rolling-horizon replanning written out: plan_windowed every h steps, env.step the plan's rows, and the
    evaluator's bookkeeping in torch.  Also checks that on status-1 envs the h steps after each plan have no failed
    move and follow the planned cells."""
    env = BatchedMapfEnv(cfg, B, "cuda:0")
    env.reset()
    N, T = env.N, int(env.cfg.steps_per_episode)
    Rr, Cc = env.grid.shape[-2:]
    starts, goals = env.state["starts"].cpu().numpy().copy(), env.state["goals"].cpu().numpy().copy()
    agent_reward = torch.zeros((B, N), dtype=torch.float64, device="cuda")
    occupancy = torch.zeros(Rr * Cc, dtype=torch.int64, device="cuda")
    dr, dc = DR.cuda(), DC.cuda()
    planned = None
    checked = 0
    for k in range(T):
        if k % h == 0:
            plan = plan_windowed(env, window)
            ok = plan.status.bool()
            planned = env.state["positions"].to(torch.int64).clone()
        a = plan.actions[k % h]
        out = env.step(a, auto_reset=False)
        planned = planned + torch.stack([dr[a.long()], dc[a.long()]], -1)
        pos = env.state["positions"].to(torch.int64)
        assert torch.equal(pos[ok], planned[ok]), f"step {k + 1}: positions differ from the plan"
        assert not bool((out.agent_step_flags[ok] & nat.ASF_FAILED_MOVE).any()), f"step {k + 1}: a planned move failed"
        checked += int(ok.sum())
        agent_reward += out.reward.to(torch.float64)
        occupancy += torch.bincount((pos[..., 0] * Cc + pos[..., 1]).reshape(-1), minlength=Rr * Cc)
    assert bool(out.truncated.bool().all()) and checked > 0
    info = out.info.cpu().numpy().astype(np.float64)
    env.close()
    return starts, goals, agent_reward.cpu().numpy(), occupancy.reshape(Rr, Cc).cpu().numpy(), info, T


@pytest.mark.parametrize("h", [1, 4])
@pytest.mark.parametrize("B", [1003, 65536])
def test_lifelong_evaluation_against_a_hand_loop(B, h):
    res = evaluate(LIFELONG, B, policy=ReplanningPolicy(16, h))
    starts, goals, agent_reward, occupancy, info, T = hand_loop(LIFELONG, B, 16, h)
    N = LIFELONG["num_agents"]
    g_tot = info[:, nat.I_GOALS_REACHED_TOTAL]
    thr = g_tot / np.maximum(info[:, nat.I_STEP_COUNT], 1)
    comp = info[:, nat.I_COMPLETED_COUNT] / N
    assert np.array_equal(res.occupancy_grid, occupancy)
    for e, row in enumerate(res.rows):
        assert row["timesteps"] == T
        assert (row["goals_reached_total"], row["throughput"], row["completion_ratio"]) == (g_tot[e], thr[e], comp[e])
        for i in range(N):
            assert row[f"agent_{i}_reward"] == agent_reward[e, i]
            assert (row[f"agent_{i}_start_x"], row[f"agent_{i}_start_y"]) == tuple(starts[e, i])
            assert (row[f"agent_{i}_goal_x"], row[f"agent_{i}_goal_y"]) == tuple(goals[e, i])
    # the evaluator sums an env's per-step reward over its agents by a shuffle tree: the same values in another order
    ep = np.array([r["total_reward"] for r in res.rows])
    assert np.allclose(ep, agent_reward.sum(1), rtol=1e-12, atol=1e-9)
    assert res.success_rate == pytest.approx(comp.mean())
    assert res.lifelong == pytest.approx({"goals_reached_total": g_tot.mean(), "throughput": thr.mean(),
                                          "completion_ratio": comp.mean()})
    assert res.average_timesteps == T
    masked = evaluate(LIFELONG, B, policy="masked")
    keys = [k for k in res.rows[0] if k.endswith(("_start_x", "_start_y", "_goal_x", "_goal_y"))]
    assert all(a[k] == b[k] for a, b in zip(res.rows, masked.rows) for k in keys)
    assert res.lifelong["goals_reached_total"] >= 2 * masked.lifelong["goals_reached_total"]


def test_episodic_evaluation_against_the_one_shot_plan():
    """ReplanningPolicy(H, H) plans once from the reset layouts like PlannedPolicy; where PlannedPolicy succeeds, it
    succeeds at the same step."""
    cfg = {"grid": RAND32, "num_agents": 8, "sensor_range": 2, "steps_per_episode": 256, "lifelong_mapf": False,
           "seed": 4242}
    env, env2 = BatchedMapfEnv(cfg, 16384, "cuda:0"), BatchedMapfEnv(cfg, 16384, "cuda:0")
    one = _play(env, PlannedPolicy())
    rep = _play(env2, ReplanningPolicy(256, 256))
    assert np.array_equal(one["starts"], rep["starts"]) and np.array_equal(one["goals"], rep["goals"])
    ok = one["success"].bool()
    assert bool(ok.any())
    assert torch.equal(rep["success"][ok], one["success"][ok])
    assert torch.equal(rep["timesteps"][ok], one["timesteps"][ok])
    env.close()
    env2.close()
