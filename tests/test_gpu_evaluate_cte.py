"""Evaluating trained CTE policies: the greedy mode of both centralised policy kernels (mapf_cte_policy_act,
mapf_cte_lstm_policy_act), the CTE bookkeeping entry point (mapf_cte_eval_accumulate) against a plain PyTorch loop,
and evaluate() on the single-agent view against an oracle replay and against the module paths played by hand."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

CASES = [("ReferenceModel-2-1", 1), ("ReferenceModel-2-1", 4), ("ReferenceModel-3-1", 16), ("ReferenceModel-3-1", 32),
         ("rand32", 1), ("rand32", 16), ("rand32", 32)]


def grid_of(name):
    from dl_reference_models_b200 import maps

    return maps.random_obstacle_grid(32, 32, 0.30, 2026, min_free=64) if name == "rand32" else maps.get_grid(name)


def make_env(name, n, B=1003, seed=5, scramble=3):
    import torch

    from dl_reference_models_b200.single_agent import BatchedCteEnv

    env = BatchedCteEnv({"grid": grid_of(name), "num_agents": n, "steps_per_episode": 64, "seed": seed}, B)
    env.reset()
    g = torch.Generator(device=env.device).manual_seed(seed)
    for _ in range(scramble):
        env.step(torch.randint(0, 5, (B, n), dtype=torch.int8, device=env.device, generator=g), auto_reset=True)
    return env


def scaled(module, scale=3.0):
    import torch

    with torch.no_grad():
        for p in module.parameters():
            p.mul_(scale)   # larger logits: a sharper test of the arithmetic
    return module


def r16(t):
    import torch

    return t.float().to(torch.bfloat16).double()


def mlp_bf16_reference(policy, grid, mask):
    """mapf_cte_policy_act's arithmetic in float64 with bf16 rounding at its points -> masked logits [B*N, 5]."""
    import torch

    h = grid.reshape(grid.shape[0], -1).double()
    for lin in [m for m in policy.trunk if isinstance(m, torch.nn.Linear)]:
        h = r16(torch.relu(h @ r16(lin.weight).T + lin.bias.double()))
    logits = h @ r16(policy.logits.weight).T + policy.logits.bias.double()
    return (logits + torch.where(mask != 0, 9.99999e-07, -13.815511).double()).reshape(-1, 5)


def lstm_bf16_reference(policy, grid, mask, pa, pr, h, c, start):
    """mapf_cte_lstm_policy_act's arithmetic in float64 with bf16 rounding at its points -> masked logits [B*N, 5]."""
    import torch

    B, N = mask.shape[0], policy.num_agents
    keep = (start == 0).double().unsqueeze(-1)
    h, c = h.double() * keep, c.double() * keep
    pa = pa.long() * (start == 0).long().unsqueeze(-1)
    pr = pr.float().double() * keep.squeeze(-1)
    y = grid.reshape(B, -1).double()
    for lin in [m for m in policy.trunk if isinstance(m, torch.nn.Linear)]:
        y = r16(torch.relu(y @ r16(lin.weight).T + lin.bias.double()))
    wih, whh = policy.lstm.weight_ih, policy.lstm.weight_hh
    onehot = torch.nn.functional.one_hot(pa, 5).reshape(B, 5 * N).double()
    gates = (y @ r16(wih[:, :64]).T + onehot @ r16(wih[:, 64:64 + 5 * N]).T + pr.unsqueeze(-1) * wih[:, 64 + 5 * N].double()
             + r16(h) @ r16(whh).T + (policy.lstm.bias_ih.float() + policy.lstm.bias_hh.float()).double())
    i, f, g, o = gates.chunk(4, -1)
    c2 = torch.sigmoid(f) * c + torch.sigmoid(i) * torch.tanh(g)
    h2 = torch.sigmoid(o) * torch.tanh(c2)
    logits = r16(h2) @ r16(policy.logits.weight).T + policy.logits.bias.double()
    return (logits + torch.where(mask != 0, 9.99999e-07, -13.815511).double()).reshape(-1, 5)


def check_greedy(acts, logp, logits, ref_logits):
    """acts = per agent the first argmax of the launch's own masked logits, logp the sum of their log-softmax in agent
    order (1e-4 per agent), and the bf16 reference's argmax wherever that reference's top-two margin exceeds 6e-2."""
    import torch

    B, N = acts.shape
    lg = logits.reshape(B * N, 5)
    a = acts.reshape(B * N).long()
    assert torch.equal(a, torch.argmax(lg, -1))
    per_agent = torch.log_softmax(lg.double(), -1).gather(-1, a.unsqueeze(-1)).reshape(B, N)
    assert float((logp.double() - per_agent.sum(-1)).abs().max()) <= 1e-4 * N
    top = torch.topk(ref_logits, 2, dim=-1).values
    sure = (top[:, 0] - top[:, 1]) > 6e-2
    assert float(sure.float().mean()) > 0.5
    assert torch.equal(a[sure], torch.argmax(ref_logits, -1)[sure])


@pytest.mark.parametrize("name,n", CASES)
def test_mlp_greedy_mode(name, n):
    import torch

    from dl_reference_models_b200.cte_rollout import CteActionMaskPolicy
    from dl_reference_models_b200.policy_kernels import FusedCtePolicy

    env = make_env(name, n)   # B = 1003: the last 32-env tile is partial
    torch.manual_seed(1)
    policy = scaled(CteActionMaskPolicy(env.R * env.C, n).to(env.device), 1.5)
    fused = FusedCtePolicy(policy, env)
    runs = {}
    for mode, greedy, seed, counter in (("draw", False, 5, 10), ("greedy", True, 5, 10), ("greedy2", True, 77, 12345)):
        fused.seed, fused.counter = seed, counter - 1
        logits = torch.full((env.B, n, 5), 7.0, device=env.device)
        acts, logp, value = fused.act(logits_out=logits, greedy=greedy)
        runs[mode] = (acts.clone(), logp.clone(), value.clone(), logits, fused.actions64.clone())
    acts, logp, value, logits, a64 = runs["greedy"]
    assert torch.equal(logits, runs["draw"][3]) and torch.equal(value, runs["draw"][2])
    for x, y in zip(runs["greedy"], runs["greedy2"]):   # nothing depends on seed or counter
        assert torch.equal(x, y)
    assert torch.equal(a64, acts.long())
    with torch.no_grad():
        ref = mlp_bf16_reference(policy, env.obs_grid, env.action_mask)
    check_greedy(acts, logp, logits, ref)


@pytest.mark.parametrize("name,n", CASES)
@pytest.mark.parametrize("starts", [False, True])
def test_lstm_greedy_mode(name, n, starts):
    import torch

    from dl_reference_models_b200.cte_rollout import CteRecurrentPolicy
    from dl_reference_models_b200.policy_kernels import FusedCteRecurrentPolicy

    env = make_env(name, n)
    torch.manual_seed(2)
    policy = scaled(CteRecurrentPolicy(env.R * env.C, n).to(env.device), 1.5)
    fused = FusedCteRecurrentPolicy(policy, env)
    B, dev = env.B, env.device
    g = torch.Generator(device=dev).manual_seed(n)
    h, c = torch.randn((B, 64), device=dev, generator=g) * 0.5, torch.randn((B, 64), device=dev, generator=g)
    pa = torch.randint(0, 5, (B, n), dtype=torch.int8, device=dev, generator=g)
    choices = torch.tensor([-0.2, -0.05, -0.25, 1.0, 0.0, 0.75], dtype=torch.float64, device=dev)
    pr = choices[torch.randint(0, len(choices), (B,), device=dev, generator=g)]
    start = ((torch.rand(B, device=dev, generator=g) < 0.2) if starts else torch.zeros(B, device=dev)).to(torch.uint8)
    runs = {}
    for mode, greedy, seed, counter in (("draw", False, 5, 10), ("greedy", True, 5, 10), ("greedy2", True, 77, 999)):
        fused.seed, fused.counter = seed, counter - 1
        ho, co = torch.full_like(h, 7.0), torch.full_like(c, 7.0)
        logits = torch.full((B, n, 5), 7.0, device=dev)
        acts, logp, value = fused.act((h, c), pa, pr, start if starts else None, None, state_out=(ho, co),
                                      logits_out=logits, greedy=greedy)
        runs[mode] = (acts.clone(), logp.clone(), value.clone(), logits, ho, co, fused.actions64.clone())
    acts, logp, value, logits, ho, co, a64 = runs["greedy"]
    for k in (2, 3, 4, 5):   # value, logits, h', c'
        assert torch.equal(runs["draw"][k], runs["greedy"][k]), k
    for x, y in zip(runs["greedy"], runs["greedy2"]):
        assert torch.equal(x, y)
    assert torch.equal(a64, acts.long())
    with torch.no_grad():
        ref = lstm_bf16_reference(policy, env.obs_grid, env.action_mask, pa, pr, h, c, start)
    check_greedy(acts, logp, logits, ref)


def goal_seeking_cte_policy(log, seed=0):
    """Seeded and logged: each agent mostly moves along its goal delta (a random axis when both differ), NO_OP on the
    goal, otherwise (blocked, or 15 % of the time) a uniform draw over its allowed actions."""
    import torch

    gen = {}

    def policy(env, out):
        grid, mask = out
        B, N, dev = env.B, env.N, env.device
        if not gen:
            gen["g"] = torch.Generator(device=dev).manual_seed(seed)
        g = gen["g"]
        d = (env.goals - env.positions).long()
        dr, dc = d[..., 0], d[..., 1]
        vertical = (dr != 0) & ((dc == 0) | (torch.rand((B, N), device=dev, generator=g) < 0.5))
        want = torch.where(vertical, torch.where(dr < 0, 1, 3), torch.where(dc > 0, 2, 4))   # UP, DOWN, RIGHT, LEFT
        want = torch.where((dr == 0) & (dc == 0), 0, want)
        m = mask.view(B, N, 5)
        ok = m.gather(-1, want.unsqueeze(-1)).squeeze(-1) != 0
        ok &= torch.rand((B, N), device=dev, generator=g) >= 0.15
        rnd = torch.argmax(torch.rand((B, N, 5), device=dev, generator=g) * m, -1)
        a = torch.where(ok, want, rnd).to(torch.int8).contiguous()
        log.append(a.cpu().numpy().copy())
        return a
    return policy


def replay_on_the_oracle(cfg, grid, res, log):
    """Every episode of an evaluate() result replayed on the CPU oracle with the logged joint actions: per episode
    the Python reward sum, steps, success, the last step's counters, and the heat-map of main.py:264-267."""
    from oracle.cte_oracle import CteOracleEnv

    R, C_ = grid.shape
    N = cfg["num_agents"]
    occ = np.zeros((R, C_), np.int64)
    eps = []
    for e, row in enumerate(res.rows):
        env = CteOracleEnv(cfg, grid)
        env.reset([[row[f"agent_{i}_start_x"], row[f"agent_{i}_start_y"]] for i in range(N)],
                  [[row[f"agent_{i}_goal_x"], row[f"agent_{i}_goal_y"]] for i in range(N)])
        total, steps, success, info = 0.0, 0, 0.0, np.zeros(4)
        for acts in log:
            _, reward, term, trunc, info = env.step(acts[e])
            total += reward
            steps += 1
            for r, c in env.positions:
                if 0 <= r < R and 0 <= c < C_:
                    occ[r, c] += 1
            if term or trunc:
                success = float(term and not trunc)
                break
        eps.append(dict(total=total, steps=steps, success=success, term=term, trunc=trunc, info=info.copy()))
    return eps, occ


def test_evaluate_on_the_cte_view_equals_an_oracle_replay():
    from dl_reference_models_b200 import maps
    from dl_reference_models_b200.evaluate import evaluate

    grid = maps.get_grid("ReferenceModel-2-1")
    cfg = {"grid": grid, "num_agents": 6, "steps_per_episode": 40, "seed": 13, "training_execution_mode": "CTE"}
    B, log = 301, []
    res = evaluate(cfg, B, policy=goal_seeking_cte_policy(log))
    eps, occ = replay_on_the_oracle(cfg, grid, res, log)
    assert any(e["term"] and not e["trunc"] for e in eps) and any(e["trunc"] for e in eps), \
        "the batch holds terminated and truncated episodes"
    assert len(log) == max(e["steps"] for e in eps)
    for e, (row, want) in enumerate(zip(res.rows, eps)):
        assert row["total_reward"] == want["total"], e
        assert row["timesteps"] == want["steps"], e
        assert row["goals_reached_total"] == want["info"][2] and row["blocking_count_total"] == want["info"][3], e
        assert list(row)[:7] == ["episode", "cpu_time", "seed", "total_reward", "timesteps", "goals_reached_total",
                                 "blocking_count_total"]
        assert row["episode"] == e + 1 and row["seed"] == 13 and len(row) == 7 + 4 * cfg["num_agents"]
    assert np.array_equal(res.occupancy_grid, occ)
    assert res.success_rate == float(np.mean([e["success"] for e in eps]))
    assert res.average_reward == float(np.sum([r["total_reward"] for r in res.rows]) / B)
    assert res.average_timesteps == float(np.sum([e["steps"] for e in eps]) / B)
    assert res.lifelong == {}


def reference_evaluate_cte(cfg, B, policy):
    """The CTE evaluator's loop with PyTorch bookkeeping (two host syncs per step) instead of mapf_cte_eval_accumulate."""
    import torch

    from dl_reference_models_b200.single_agent import BatchedCteEnv

    env = BatchedCteEnv(cfg, B)
    env.reset()
    dev, R, C_ = env.device, env.R, env.C
    starts, goals = env.starts.cpu().numpy().copy(), env.goals.cpu().numpy().copy()
    active = torch.ones(B, dtype=torch.bool, device=dev)
    ep_reward = torch.zeros(B, dtype=torch.float64, device=dev)
    steps = torch.zeros(B, dtype=torch.int64, device=dev)
    success = torch.zeros(B, dtype=torch.float64, device=dev)
    last_info = torch.zeros((B, 4), dtype=torch.float64, device=dev)
    occ = torch.zeros(R * C_, dtype=torch.int64, device=dev)
    for _ in range(env.steps_per_episode + 1):
        if not bool(active.any()):
            break
        env.step(policy(env, (env.obs_grid, env.action_mask)))
        ep_reward += torch.where(active, env.reward, torch.zeros_like(env.reward))
        steps += active.to(torch.int64)
        pos = env.positions[active].reshape(-1, 2).long()
        inside = (pos[:, 0] >= 0) & (pos[:, 0] < R) & (pos[:, 1] >= 0) & (pos[:, 1] < C_)
        occ += torch.bincount(pos[inside, 0] * C_ + pos[inside, 1], minlength=R * C_)
        last_info[active] = env.info[active]
        done = (env.terminated | env.truncated).bool() & active
        success[done] = ((env.terminated != 0) & (env.truncated == 0)).to(torch.float64)[done]
        active &= ~done
    return dict(starts=starts, goals=goals, ep_reward=ep_reward.cpu().numpy(), steps=steps.cpu().numpy(),
                success=success.cpu().numpy(), info=last_info.cpu().numpy(), occ=occ.reshape(R, C_).cpu().numpy())


@pytest.mark.parametrize("name,n,steps", [("ReferenceModel-2-1", 3, 60), ("rand32", 16, 48)])
def test_bookkeeping_kernel_equals_the_pytorch_loop(name, n, steps):
    from dl_reference_models_b200.evaluate import evaluate

    cfg = {"grid": grid_of(name), "num_agents": n, "steps_per_episode": steps, "seed": 11, "training_execution_mode": "CTE"}
    B = 517
    ref = reference_evaluate_cte(cfg, B, goal_seeking_cte_policy([], seed=4))
    res = evaluate(cfg, B, policy=goal_seeking_cte_policy([], seed=4))
    assert np.array_equal(res.occupancy_grid, ref["occ"])
    if name == "ReferenceModel-2-1":
        assert len(set(ref["steps"].tolist())) > 3 and 0 < ref["success"].mean() < 1
    for e, row in enumerate(res.rows):
        want = {"episode": e + 1, "cpu_time": 0.0, "seed": 11, "total_reward": float(ref["ep_reward"][e]),
                "timesteps": int(ref["steps"][e]), "goals_reached_total": float(ref["info"][e, 2]),
                "blocking_count_total": float(ref["info"][e, 3])}
        for i in range(n):
            want[f"agent_{i}_start_x"], want[f"agent_{i}_start_y"] = int(ref["starts"][e, i, 0]), int(ref["starts"][e, i, 1])
            want[f"agent_{i}_goal_x"], want[f"agent_{i}_goal_y"] = int(ref["goals"][e, i, 0]), int(ref["goals"][e, i, 1])
        assert row == want and list(row) == list(want), e
    assert res.success_rate == float(np.mean(ref["success"]))
    assert res.average_reward == float(ref["ep_reward"].sum() / B)
    assert res.average_timesteps == float(ref["steps"].sum() / B)


def same_results(a, b):
    assert a.rows == b.rows
    assert np.array_equal(a.occupancy_grid, b.occupancy_grid)
    assert (a.success_rate, a.average_reward, a.average_timesteps, a.lifelong) == \
        (b.success_rate, b.average_reward, b.average_timesteps, b.lifelong)


def eval_cfg(**kw):
    from dl_reference_models_b200 import maps

    return dict({"grid": maps.get_grid("ReferenceModel-2-1"), "num_agents": 4, "steps_per_episode": 40, "seed": 17}, **kw)


def test_evaluate_cte_mlp_module_on_the_fused_kernel():
    import torch

    from dl_reference_models_b200.cte_rollout import CteActionMaskPolicy
    from dl_reference_models_b200.evaluate import evaluate
    from dl_reference_models_b200.policy_kernels import FusedCtePolicy

    cfg = eval_cfg()
    torch.manual_seed(3)
    policy = scaled(CteActionMaskPolicy(200, 4).cuda(), 2.0)
    fused = {}

    def by_hand(env, out):
        if "f" not in fused:
            fused["f"] = FusedCtePolicy(policy, env)
        return fused["f"].act(greedy=True)[0]

    res = evaluate(cfg, 301, policy=policy)
    same_results(res, evaluate(dict(cfg, training_execution_mode="CTE"), 301, policy=by_hand))
    assert all(1 <= r["timesteps"] <= 40 for r in res.rows)


def test_evaluate_cte_lstm_module_on_the_fused_kernel():
    import torch

    from dl_reference_models_b200.cte_rollout import CteRecurrentPolicy
    from dl_reference_models_b200.evaluate import evaluate
    from dl_reference_models_b200.policy_kernels import FusedCteRecurrentPolicy

    cfg = eval_cfg(training_execution_mode="CTE")
    torch.manual_seed(4)
    policy = scaled(CteRecurrentPolicy(200, 4).cuda(), 2.0)
    carry = {}

    def by_hand(env, out):
        if not carry:
            carry.update(f=FusedCteRecurrentPolicy(policy, env), h=torch.zeros(env.B, 64, device=env.device),
                         c=torch.zeros(env.B, 64, device=env.device),
                         r=torch.zeros(env.B, dtype=torch.float64, device=env.device))
        else:
            carry["r"] = env.reward.clone()
        f = carry["f"]
        return f.act((carry["h"], carry["c"]), f.actions, carry["r"], greedy=True)[0]

    same_results(evaluate(cfg, 301, policy=policy), evaluate(cfg, 301, policy=by_hand))
    assert carry and not bool(carry["h"].eq(0).all())


@pytest.mark.parametrize("kind", ["mlp_32", "lstm_32"])
def test_evaluate_non_fused_cte_shapes_run_the_module_forward(kind):
    from types import SimpleNamespace

    import torch

    from dl_reference_models_b200.cte_rollout import CteActionMaskPolicy, CteRecurrentPolicy
    from dl_reference_models_b200.evaluate import evaluate
    from dl_reference_models_b200.policy_kernels import FusedCtePolicy, FusedCteRecurrentPolicy

    cfg = eval_cfg(training_execution_mode="CTE")
    torch.manual_seed(5)
    recurrent = kind.startswith("lstm")
    policy = (CteRecurrentPolicy if recurrent else CteActionMaskPolicy)(200, 4, hiddens=(32,)).cuda()
    assert not (FusedCteRecurrentPolicy if recurrent else FusedCtePolicy).matches(policy, SimpleNamespace(R=10, C=20, N=4))
    carry = {}

    @torch.no_grad()
    def by_hand(env, out):
        grid, mask = env.obs_grid.view(env.B, -1), env.action_mask
        if not recurrent:
            return torch.argmax(policy(grid, mask)[0], -1).to(torch.int8)
        if not carry:
            carry.update(s=policy.initial_state(env.B, env.device), a=torch.zeros((env.B, 4), dtype=torch.int64, device=env.device),
                         r=torch.zeros(env.B, dtype=torch.float64, device=env.device))
        else:
            carry["r"] = env.reward.clone()
        lg, _, carry["s"] = policy.step(grid, mask, carry["a"], carry["r"], carry["s"])
        carry["a"] = torch.argmax(lg, -1)
        return carry["a"].to(torch.int8)

    same_results(evaluate(cfg, 211, policy=policy), evaluate(cfg, 211, policy=by_hand))
    assert carry or not recurrent


@pytest.mark.parametrize("kind", ["mlp", "lstm", "mlp_32"])
def test_explore_draws_only_allowed_actions(kind):
    import torch

    from dl_reference_models_b200.cte_rollout import CteActionMaskPolicy, CteRecurrentPolicy
    from dl_reference_models_b200.evaluate import _cte_module_actor, evaluate
    from dl_reference_models_b200.single_agent import BatchedCteEnv

    cfg = eval_cfg()
    torch.manual_seed(6)
    policy = {"mlp": lambda: CteActionMaskPolicy(200, 4), "lstm": lambda: CteRecurrentPolicy(200, 4),
              "mlp_32": lambda: CteActionMaskPolicy(200, 4, hiddens=(32,))}[kind]().cuda()
    env = BatchedCteEnv(cfg, 1024)
    env.reset()
    act = _cte_module_actor(env, policy, explore=True)
    allowed, total = 0, 0
    for _ in range(10):
        a = act()
        allowed += int((env.action_mask.view(env.B, 4, 5).gather(-1, a.long().unsqueeze(-1)) == 1).sum())
        total += a.numel()
        env.step(a)
    assert allowed / total >= 0.9999
    res, greedy = evaluate(cfg, 256, policy=policy, explore=True), evaluate(cfg, 256, policy=policy)
    assert res.rows != greedy.rows and all(r["timesteps"] >= 1 for r in res.rows)


@pytest.mark.parametrize("policy", ["random", "masked"])
def test_builtin_policies_on_the_cte_view(policy):
    from dl_reference_models_b200.evaluate import evaluate

    res = evaluate(eval_cfg(training_execution_mode="CTE"), 300, policy=policy)
    assert len(res.rows) == 300 and all(1 <= r["timesteps"] <= 41 for r in res.rows)
    assert res.occupancy_grid.shape == (10, 20) and res.occupancy_grid.sum() >= 300 * 4
    assert 0.0 <= res.success_rate <= 1.0 and "agent_0_reward" not in res.rows[0]


def test_refusals():
    from dl_reference_models_b200.cte_rollout import CteActionMaskPolicy, CteRecurrentPolicy
    from dl_reference_models_b200.evaluate import evaluate
    from dl_reference_models_b200.rollout import ActionMaskPolicy

    cfg = eval_cfg()
    with pytest.raises(ValueError, match="centralised"):
        evaluate(dict(cfg, training_execution_mode="CTDE"), 8, policy=CteActionMaskPolicy(200, 4).cuda())
    with pytest.raises(ValueError, match="multi-agent view"):
        evaluate(dict(cfg, training_execution_mode="CTE"), 8, policy=ActionMaskPolicy(28).cuda())
    with pytest.raises(ValueError, match="grid cells"):
        evaluate(cfg, 8, policy=CteRecurrentPolicy(600, 4).cuda())
    with pytest.raises(ValueError, match="num_agents"):
        evaluate(cfg, 8, policy=CteActionMaskPolicy(200, 3).cuda())
    with pytest.raises(ValueError, match="cpu"):
        evaluate(cfg, 8, policy=CteRecurrentPolicy(200, 4, cell=32))
