"""The conflict-based search kernel (mapf_plan_cbs) against the pure Python reference bit for bit (actions, arrivals,
outcomes, expansion counts), shards of a batch against the full launch, and PlannedPolicy("cbs") through the batched
evaluator (against a hand loop of plan_cbs and env.step, and against prioritized planning)."""
import numpy as np
import pytest
import torch

from dl_reference_models_b200 import maps
from dl_reference_models_b200.batched_env import BatchedMapfEnv
from dl_reference_models_b200.evaluate import _play, evaluate
from dl_reference_models_b200.planner import PlannedPolicy, cbs_reference, plan_cbs
from test_gpu_planner import _grid, layouts

pytestmark = pytest.mark.gpu

SEEN = {}
CASES = [("1-1", 2, 1003, 32, 16), ("1-2", 2, 1003, 100, 1024), ("2-1", 4, 1003, 100, 1024), ("2-2", 4, 1003, 256, 16),
         ("3-1", 1, 1003, 256, 1024), ("3-1", 8, 1003, 100, 1), ("rand32", 8, 1003, 256, 16),
         ("rand32", 4, 1003, 32, 1024), ("rand32", 2, 1003, 256, 1024), ("1-2", 2, 1003, 10, 1024),
         ("2-2", 4, 65536, 100, 1024)]


def _equal_rows(got, ref, rows):
    r = torch.as_tensor(rows, device=got.outcome.device)
    assert torch.equal(got.outcome[r].cpu(), ref.outcome)
    assert torch.equal(got.expanded[r].cpu(), ref.expanded)
    assert torch.equal(got.arrival[r].cpu(), ref.arrival)
    assert torch.equal(got.actions[:, r].cpu(), ref.actions)
    assert torch.equal(got.sum_of_costs[r].cpu(), ref.sum_of_costs)


@pytest.mark.parametrize("name,N,B,H,K", CASES, ids=[f"{c[0]}-N{c[1]}-B{c[2]}-H{c[3]}-K{c[4]}" for c in CASES])
def test_kernel_equals_the_reference(name, N, B, H, K):
    grid = _grid(name)
    env = BatchedMapfEnv({"grid": grid, "num_agents": min(N, 8), "sensor_range": 1, "seed": 5,
                          "steps_per_episode": H}, 4)
    st, gl = layouts(grid, B, N, seed=B + N + H + K)
    if B > 1003:
        st[B // 2, 1] = st[B // 2, 0]      # a repeated start
        gl[B // 2 + 1, 2] = gl[B // 2 + 1, 3]   # a repeated goal
    got = plan_cbs(env, K, st, gl, H)
    ex = got.expanded.cpu().numpy()
    if B <= 1003:
        rows = np.arange(B)
    else:   # a sample: 400 envs at random, the 100 longest searches and the repeated start and goal
        rng = np.random.default_rng(0)
        rows = np.unique(np.concatenate([rng.choice(B, 400, replace=False), np.argsort(-ex)[:100], [B // 2, B // 2 + 1]]))
    ref = cbs_reference(grid, st[rows].cpu(), gl[rows].cpu(), H, K)
    _equal_rows(got, ref, rows)
    oc = got.outcome.cpu().numpy()
    SEEN[(name, N, B, H, K)] = {"outcome0_root": int(((oc == 0) & (ex == 0)).sum()),
                                "outcome0_search": int(((oc == 0) & (ex > 0)).sum()),
                                "outcome1": int((oc == 1).sum()), "outcome2": int((oc == 2).sum()),
                                "max_expanded": int(ex.max()), "one_expansion": int((ex == 1).sum())}
    print(name, N, B, H, K, SEEN[(name, N, B, H, K)])
    assert (ex <= K).all() and ((oc == 2) <= (ex == K)).all()
    if B > 1003:
        assert (oc[B // 2:B // 2 + 2] == 0).all() and (ex[B // 2:B // 2 + 2] == 0).all()
    env.close()


def test_every_outcome_occurs():
    """Outcome 0 at the root and after a search, outcome 1 and outcome 2 all occur in the cases above, and one launch
    holds envs answered at the root next to envs that run to the budget of 1024 expansions."""
    if len(SEEN) < len(CASES):
        pytest.skip("needs every case of test_kernel_equals_the_reference in the same run")
    for k in ("outcome0_root", "outcome0_search", "outcome1", "outcome2"):
        assert sum(v[k] for v in SEEN.values()) > 0, k
    assert any(v["one_expansion"] > 0 and v["max_expanded"] >= 1024 for k, v in SEEN.items() if k[4] == 1024)


@pytest.mark.parametrize("name,N,H,K", [("2-1", 4, 100, 1024), ("rand32", 8, 256, 16)])
def test_a_shard_gives_the_rows_of_the_full_launch(name, N, H, K):
    grid = _grid(name)
    env = BatchedMapfEnv({"grid": grid, "num_agents": N, "sensor_range": 1, "seed": 5, "steps_per_episode": H}, 4)
    st, gl = layouts(grid, 3001, N, seed=77)
    full = plan_cbs(env, K, st, gl, H)
    for lo, hi in ((0, 1), (1000, 1777), (2900, 3001)):
        part = plan_cbs(env, K, st[lo:hi], gl[lo:hi], H)
        for f in ("actions", "arrival", "outcome", "expanded", "makespan", "sum_of_costs", "status"):
            a, b = getattr(full, f), getattr(part, f)
            assert torch.equal(a[:, lo:hi] if f == "actions" else a[lo:hi], b), f
    env.close()


EPISODIC = {"grid": maps.get_grid("ReferenceModel-2-1"), "num_agents": 4, "sensor_range": 2, "steps_per_episode": 100,
            "lifelong_mapf": False, "seed": 1357}


def hand_loop(cfg, B):
    """plan_cbs on the reset layouts, then env.step the plan's rows with the evaluator's bookkeeping written out in
    torch: per-agent rewards, timesteps and the heat-map over the envs still active before each step (an env is done
    at its first terminated or truncated step)."""
    env = BatchedMapfEnv(cfg, B, "cuda:0")
    env.reset()
    N, H = env.N, int(env.cfg.steps_per_episode)
    Rr, Cc = env.grid.shape[-2:]
    starts, goals = env.state["starts"].cpu().numpy().copy(), env.state["goals"].cpu().numpy().copy()
    plan = plan_cbs(env)
    active = torch.ones(B, dtype=torch.bool, device="cuda")
    agent_reward = torch.zeros((B, N), dtype=torch.float64, device="cuda")
    steps = torch.zeros(B, dtype=torch.int64, device="cuda")
    occupancy = torch.zeros(Rr * Cc, dtype=torch.int64, device="cuda")
    for t in range(H + 1):
        if not bool(active.any()):
            break
        a = plan.actions[t] if t < H else torch.zeros((B, N), dtype=torch.int8, device="cuda")
        out = env.step(a, auto_reset=False)
        pos = env.state["positions"].to(torch.int64)[active]
        occupancy += torch.bincount((pos[..., 0] * Cc + pos[..., 1]).reshape(-1), minlength=Rr * Cc)
        agent_reward[active] += out.reward.to(torch.float64)[active]
        steps[active] += 1
        done = out.terminated.bool() | out.truncated.bool()
        active &= ~done
    env.close()
    return plan, starts, goals, agent_reward.cpu().numpy(), steps.cpu().numpy(), occupancy.reshape(Rr, Cc).cpu().numpy()


@pytest.mark.parametrize("B", [1003, 65536])
def test_cbs_policy_through_the_evaluator(B):
    pol = PlannedPolicy("cbs")
    res = evaluate(EPISODIC, B, policy=pol)
    plan = pol.plan
    ok = plan.outcome.cpu().numpy() == 1
    ms = plan.makespan.cpu().numpy()
    steps = np.array([r["timesteps"] for r in res.rows])
    assert ok.any() and np.array_equal(steps[ok], ms[ok])
    assert res.success_rate == pytest.approx(ok.mean())
    # a hand loop of plan_cbs and env.step gives the same plan, rows, heat-map and summary
    hp, starts, goals, agent_reward, hsteps, occupancy = hand_loop(EPISODIC, B)
    for f in ("actions", "arrival", "outcome", "expanded"):
        assert torch.equal(getattr(hp, f), getattr(plan, f)), f
    assert np.array_equal(steps, hsteps)
    assert np.array_equal(res.occupancy_grid, occupancy)
    N = EPISODIC["num_agents"]
    for e, row in enumerate(res.rows):
        for i in range(N):
            assert row[f"agent_{i}_reward"] == agent_reward[e, i]
            assert (row[f"agent_{i}_start_x"], row[f"agent_{i}_start_y"]) == tuple(starts[e, i])
            assert (row[f"agent_{i}_goal_x"], row[f"agent_{i}_goal_y"]) == tuple(goals[e, i])
    assert res.average_timesteps == pytest.approx(hsteps.mean())
    # per env (the evaluator's own accumulators): success exactly on the outcome-1 envs
    env = BatchedMapfEnv(EPISODIC, B, "cuda:0")
    acc = _play(env, PlannedPolicy("cbs"))
    env.close()
    assert np.array_equal(acc["success"].cpu().numpy().astype(bool), ok)
    # where both planners succeed, CBS's sum of arrivals is at most prioritized planning's
    pp = PlannedPolicy()
    env = BatchedMapfEnv(EPISODIC, B, "cuda:0")
    acc = _play(env, pp)
    env.close()
    both = ok & acc["success"].cpu().numpy().astype(bool)
    assert both.any()
    assert (plan.sum_of_costs.cpu().numpy()[both] <= pp.plan.sum_of_costs.cpu().numpy()[both]).all()
