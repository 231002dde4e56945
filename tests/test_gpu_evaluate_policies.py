"""Evaluating trained policies: the greedy (argmax) mode of both fused policy kernels, the evaluator's bookkeeping
kernel (mapf_eval_accumulate) against the PyTorch loop it replaces, and evaluate() with MLP / LSTM-64 modules on the
fused and on the PyTorch path."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def make_env(sr=2, B=2048, n=16):
    from dl_reference_models_b200 import maps
    from dl_reference_models_b200.batched_env import BatchedMapfEnv

    cfg = {"num_agents": n, "sensor_range": sr, "steps_per_episode": 64, "lifelong_mapf": True, "seed": 21,
           "grid": maps.random_obstacle_grid(32, 32, 0.3, 2026, min_free=2 * n)}
    env = BatchedMapfEnv(cfg, B, "cuda:0")
    out = env.reset()
    for _ in range(5):
        out = env.step(env.sample_actions(masked=True), auto_reset=True)
    return env, out


def scaled(module, env, scale=3.0, seed=0):
    import torch

    torch.manual_seed(seed)
    m = module(env.flat_obs_dim(include_action_mask=False)).to(env.device)
    with torch.no_grad():
        for p in m.parameters():
            p.mul_(scale)   # larger logits: a sharper test of the arithmetic
    return m


def r16(t):
    import torch

    return t.to(torch.bfloat16).to(torch.float32)


def masked(logits, mask):
    import torch

    return logits + torch.where(mask != 0, torch.full_like(logits, 9.99999e-07), torch.full_like(logits, -13.815511))


def mlp_bf16_reference(policy, feats, mask):
    """The MLP kernel's arithmetic in torch: bf16 rounding of inputs, weights and hidden activations, f32 accumulation."""
    import torch

    h = r16(feats)
    for lin in [m for m in policy.trunk if isinstance(m, torch.nn.Linear)]:
        h = r16(torch.relu(h @ r16(lin.weight).T + lin.bias))
    return masked(h @ r16(policy.logits.weight).T + policy.logits.bias, mask)


def lstm_bf16_reference(pol, feats, mask, pa, pr, h, c):
    """The LSTM kernel's arithmetic in torch (as tests/test_gpu_lstm_policy_kernel.py's bf16_reference)."""
    import torch

    x = r16(feats)
    for lin in [m for m in pol.trunk if isinstance(m, torch.nn.Linear)]:
        x = r16(torch.relu(x @ r16(lin.weight).T + lin.bias))
    xi = torch.cat([x, torch.nn.functional.one_hot(pa, 5).float(), r16(pr).unsqueeze(-1)], -1)
    lstm = pol.lstm
    gates = xi @ r16(lstm.weight_ih).T + r16(h) @ r16(lstm.weight_hh).T + (lstm.bias_ih + lstm.bias_hh)
    i, f, g, o = gates.chunk(4, -1)
    c1 = torch.sigmoid(f) * c + torch.sigmoid(i) * torch.tanh(g)
    h1 = torch.sigmoid(o) * torch.tanh(c1)
    return masked(r16(h1) @ r16(pol.logits.weight).T + pol.logits.bias, mask)


def check_greedy(acts, logp, logits, ref_logits):
    """acts = first argmax of the launch's own masked logits, logp its log-softmax, and the bf16 reference's argmax
    wherever that reference's top-two margin exceeds twice the kernels' 3e-2 worst-case logit error."""
    import torch

    M = logits.numel() // 5
    lg = logits.reshape(M, 5)
    a = acts.reshape(M).long()
    assert torch.equal(a, torch.argmax(lg, -1))
    want = torch.log_softmax(lg, -1).gather(-1, a.unsqueeze(-1)).squeeze(-1)
    assert float((logp.reshape(M) - want).abs().max()) <= 1e-4
    top = torch.topk(ref_logits, 2, dim=-1).values
    sure = (top[:, 0] - top[:, 1]) > 6e-2
    assert float(sure.float().mean()) > 0.5
    assert torch.equal(a[sure], torch.argmax(ref_logits, -1)[sure])


@pytest.mark.parametrize("sr", [1, 2, 3])
def test_mlp_greedy_mode(sr):
    import torch

    from dl_reference_models_b200.policy_kernels import FusedPolicy
    from dl_reference_models_b200.rollout import ActionMaskPolicy

    env, out = make_env(sr=sr, B=1003, n=7)   # B * N = 7021: the last tile is partial
    policy = scaled(ActionMaskPolicy, env)
    fused = FusedPolicy(policy, env)
    runs = {}
    for mode, greedy, seed, counter in (("draw", False, 5, 10), ("greedy", True, 5, 10), ("greedy2", True, 77, 12345)):
        fused.seed, fused.counter = seed, counter - 1
        logits = torch.full((env.B, env.N, 5), 7.0, device=env.device)
        acts, logp, value = fused.act(out, logits_out=logits, greedy=greedy)
        runs[mode] = (acts.clone(), logp.clone(), value.clone(), logits, fused.actions64.clone())
    acts, logp, value, logits, a64 = runs["greedy"]
    assert torch.equal(logits, runs["draw"][3]) and torch.equal(value, runs["draw"][2])
    for x, y in zip(runs["greedy"], runs["greedy2"]):   # nothing depends on seed or counter
        assert torch.equal(x, y)
    assert torch.equal(a64, acts.long())
    assert not torch.equal(acts, runs["draw"][0])
    with torch.no_grad():
        ref = mlp_bf16_reference(policy, env.flat_obs(include_action_mask=False).reshape(-1, env.flat_obs_dim(include_action_mask=False)),
                                 out.action_mask.reshape(-1, 5))
    check_greedy(acts, logp, logits, ref)


@pytest.mark.parametrize("sr", [1, 2, 3])
def test_lstm_greedy_mode(sr):
    import torch

    from dl_reference_models_b200.policy_kernels import FusedRecurrentPolicy
    from dl_reference_models_b200.recurrent import RecurrentActionMaskPolicy

    env, out = make_env(sr=sr, B=1003, n=7)
    pol = scaled(RecurrentActionMaskPolicy, env)
    fused = FusedRecurrentPolicy(pol, env)
    B, N, M, dev = env.B, env.N, env.B * env.N, env.device
    g = torch.Generator(device=dev).manual_seed(sr)
    h, c = torch.randn(M, 64, device=dev, generator=g) * 0.5, torch.randn(M, 64, device=dev, generator=g)
    pa = torch.randint(0, 5, (B, N), device=dev, generator=g).to(torch.int8)
    pr = torch.randint(-4, 3, (B, N), device=dev, generator=g).float() * 0.5
    runs = {}
    for mode, greedy, seed, counter in (("draw", False, 5, 10), ("greedy", True, 5, 10), ("greedy2", True, 77, 999)):
        fused.seed, fused.counter = seed, counter - 1
        ho, co = torch.full_like(h, 7.0), torch.full_like(c, 7.0)
        logits = torch.full((B, N, 5), 7.0, device=dev)
        acts, logp, value = fused.act(out, (h, c), pa, pr, state_out=(ho, co), logits_out=logits, greedy=greedy)
        runs[mode] = (acts.clone(), logp.clone(), value.clone(), logits, ho, co, fused.actions64.clone())
    acts, logp, value, logits, ho, co, a64 = runs["greedy"]
    for k in (2, 3, 4, 5):   # value, logits, h', c'
        assert torch.equal(runs["draw"][k], runs["greedy"][k]), k
    for x, y in zip(runs["greedy"], runs["greedy2"]):
        assert torch.equal(x, y)
    assert torch.equal(a64, acts.long())
    assert not torch.equal(acts, runs["draw"][0])
    # without advancing, greedy leaves the state and the previous-action buffer alone, like the draw mode
    before = fused.actions.clone()
    hh, cc = h.clone(), c.clone()
    fused.act(out, (hh, cc), pa, pr, advance=False, greedy=True)
    assert torch.equal(fused.actions, before) and torch.equal(hh, h) and torch.equal(cc, c)
    assert torch.equal(fused.actions64, a64)
    with torch.no_grad():
        feats = env.flat_obs(include_action_mask=False).reshape(M, -1)
        ref = lstm_bf16_reference(pol, feats, out.action_mask.reshape(M, 5), pa.long().reshape(-1), pr.reshape(-1), h, c)
    check_greedy(acts, logp, logits, ref)


def reference_evaluate(env_config, num_episodes, policy):
    """The evaluator's loop as it was before mapf_eval_accumulate: PyTorch bookkeeping, two host syncs per step."""
    import torch

    from dl_reference_models_b200 import _native as nat
    from dl_reference_models_b200.batched_env import BatchedMapfEnv

    env = BatchedMapfEnv(env_config, num_episodes, "cuda:0")
    B, N, dev = env.B, env.N, env.device
    out = env.reset()
    starts = env.state["starts"].cpu().numpy().copy()
    goals0 = env.state["goals"].cpu().numpy().copy()
    active = torch.ones(B, dtype=torch.bool, device=dev)
    ep_reward = torch.zeros(B, dtype=torch.float64, device=dev)
    agent_reward = torch.zeros((B, N), dtype=torch.float64, device=dev)
    steps = torch.zeros(B, dtype=torch.int64, device=dev)
    success = torch.zeros(B, dtype=torch.float64, device=dev)
    last_info = torch.zeros((B, nat.INFO_WORDS), dtype=torch.int32, device=dev)
    occupancy = torch.zeros(env.grid.shape[-2:], dtype=torch.int64, device=dev)
    calls = 0
    for _ in range(int(env.cfg.steps_per_episode) + 1):
        if not bool(active.any()):
            break
        actions = policy(env, out)
        calls += 1
        out = env.step(actions, auto_reset=False)
        act_f = active.to(torch.float64)
        r = out.reward.to(torch.float64)
        ep_reward += r.sum(dim=1) * act_f
        agent_reward += r * act_f[:, None]
        steps += active.to(torch.int64)
        env.accumulate_occupancy(occupancy, active.to(torch.uint8))
        done = (out.terminated | out.truncated).bool() & active
        last_info[active] = out.info[active]
        success[done] = ((out.terminated != 0) & (out.truncated == 0)).to(torch.float64)[done]
        active &= ~done
    res = dict(starts=starts, goals=goals0, ep_reward=ep_reward.cpu().numpy(), agent_reward=agent_reward.cpu().numpy(),
               steps=steps.cpu().numpy(), success=success.cpu().numpy(), info=last_info.cpu().numpy(),
               occupancy=occupancy.cpu().numpy(), calls=calls, lifelong=env.lifelong)
    env.close()
    return res


def goal_seeking_policy(counter, seed=0):
    """Seeded and replayable: mostly a move along the goal delta (a random axis when both differ), NO_OP on the goal,
    otherwise (blocked, or 10 % of the time) the env's uniform masked draw; episodes end at many different steps."""
    import torch

    gen = {}

    def policy(env, out):
        counter[0] += 1
        if not gen:
            gen["g"] = torch.Generator(device=env.device).manual_seed(seed)
        g, shape = gen["g"], (env.B, env.N)
        rnd = env.sample_actions(masked=True)   # Philox, keyed by the env's seed and call counter
        dr, dc = out.goal_delta[..., 0], out.goal_delta[..., 1]
        vertical = (dr != 0) & ((dc == 0) | (torch.rand(shape, device=env.device, generator=g) < 0.5))
        want = torch.where(vertical, torch.where(dr < 0, 1, 3), torch.where(dc > 0, 2, 4))   # UP, DOWN, RIGHT, LEFT
        want = torch.where((dr == 0) & (dc == 0), 0, want)
        ok = out.action_mask.gather(-1, want.long().unsqueeze(-1)).squeeze(-1) != 0
        ok &= torch.rand(shape, device=env.device, generator=g) >= 0.1
        return torch.where(ok, want.to(torch.int8), rnd).contiguous()
    return policy


@pytest.mark.parametrize("case", ["episodic_2_1", "lifelong_32x32"])
def test_bookkeeping_kernel_equals_the_pytorch_loop(case):
    from dl_reference_models_b200 import _native as nat
    from dl_reference_models_b200 import maps
    from dl_reference_models_b200.evaluate import evaluate

    if case == "episodic_2_1":
        cfg = {"env_name": "ReferenceModel-2-1", "num_agents": 3, "sensor_range": 2, "steps_per_episode": 60,
               "lifelong_mapf": False, "seed": 11}
        B = 333
    else:
        cfg = {"grid": maps.random_obstacle_grid(32, 32, 0.3, 2026, min_free=32), "num_agents": 16, "sensor_range": 2,
               "steps_per_episode": 48, "lifelong_mapf": True, "seed": 5}
        B = 517
    ref_calls, calls = [0], [0]
    ref = reference_evaluate(cfg, B, goal_seeking_policy(ref_calls))
    res = evaluate(cfg, B, policy=goal_seeking_policy(calls))
    assert calls == ref_calls
    N = cfg["num_agents"]
    if case == "episodic_2_1":
        assert len(set(ref["steps"].tolist())) > 3, "episodes end at different steps"
        assert 0 < ref["success"].mean() < 1
    assert np.array_equal(res.occupancy_grid, ref["occupancy"])
    info = ref["info"]
    g_tot = info[:, nat.I_GOALS_REACHED_TOTAL].astype(np.float64)
    thr = g_tot / np.maximum(info[:, nat.I_STEP_COUNT], 1)
    comp = info[:, nat.I_COMPLETED_COUNT].astype(np.float64) / float(N)
    for e, row in enumerate(res.rows):
        want = {"episode": e + 1, "cpu_time": 0.0, "seed": cfg["seed"], "total_reward": float(ref["ep_reward"][e]),
                "timesteps": int(ref["steps"][e])}
        if ref["lifelong"]:
            want.update(goals_reached_total=float(g_tot[e]), throughput=float(thr[e]), completion_ratio=float(comp[e]))
        for i in range(N):
            want[f"agent_{i}_reward"] = float(ref["agent_reward"][e, i])
            want[f"agent_{i}_start_x"], want[f"agent_{i}_start_y"] = int(ref["starts"][e, i, 0]), int(ref["starts"][e, i, 1])
            want[f"agent_{i}_goal_x"], want[f"agent_{i}_goal_y"] = int(ref["goals"][e, i, 0]), int(ref["goals"][e, i, 1])
        assert row == want, e
        assert list(row) == list(want), e
    assert res.success_rate == float(np.mean(comp if ref["lifelong"] else ref["success"]))
    assert res.average_reward == float(ref["ep_reward"].sum() / B)
    assert res.average_timesteps == float(ref["steps"].sum() / B)
    if ref["lifelong"]:
        assert res.lifelong == {"goals_reached_total": float(g_tot.mean()), "throughput": float(thr.mean()),
                                "completion_ratio": float(comp.mean())}


def same_results(a, b):
    assert a.rows == b.rows
    assert np.array_equal(a.occupancy_grid, b.occupancy_grid)
    assert (a.success_rate, a.average_reward, a.average_timesteps, a.lifelong) == \
        (b.success_rate, b.average_reward, b.average_timesteps, b.lifelong)


EVAL_CFG = {"num_agents": 8, "sensor_range": 2, "steps_per_episode": 40, "lifelong_mapf": False, "seed": 17}


def eval_cfg(**kw):
    from dl_reference_models_b200 import maps

    return dict(EVAL_CFG, grid=maps.random_obstacle_grid(16, 16, 0.2, 7, min_free=16), **kw)


def test_evaluate_mlp_module_on_the_fused_kernel():
    import torch

    from dl_reference_models_b200.evaluate import evaluate
    from dl_reference_models_b200.policy_kernels import FusedPolicy
    from dl_reference_models_b200.rollout import ActionMaskPolicy

    cfg = eval_cfg()
    torch.manual_seed(3)
    policy = ActionMaskPolicy(28).cuda()
    fused = {}

    def by_hand(env, out):
        if "f" not in fused:
            fused["f"] = FusedPolicy(policy, env)
        return fused["f"].act(out, greedy=True)[0]

    same_results(evaluate(cfg, 301, policy=policy), evaluate(cfg, 301, policy=by_hand))


def test_evaluate_lstm_module_on_the_fused_kernel():
    import torch

    from dl_reference_models_b200.evaluate import evaluate
    from dl_reference_models_b200.policy_kernels import FusedRecurrentPolicy
    from dl_reference_models_b200.recurrent import RecurrentActionMaskPolicy

    cfg = eval_cfg(lifelong_mapf=True)
    torch.manual_seed(4)
    policy = RecurrentActionMaskPolicy(28).cuda()
    carry = {}

    def by_hand(env, out):
        if not carry:
            M = env.B * env.N
            carry.update(f=FusedRecurrentPolicy(policy, env), h=torch.zeros(M, 64, device=env.device),
                         c=torch.zeros(M, 64, device=env.device), r=torch.zeros(env.B, env.N, device=env.device))
        else:
            carry["r"] = out.reward.clone()
        f = carry["f"]
        return f.act(out, (carry["h"], carry["c"]), f.actions, carry["r"], greedy=True)[0]

    res = evaluate(cfg, 301, policy=policy)
    same_results(res, evaluate(cfg, 301, policy=by_hand))
    assert carry and not bool(carry["h"].eq(0).all())


@pytest.mark.parametrize("kind", ["mlp_32_32", "lstm_cell_32"])
def test_evaluate_non_reference_shapes_run_the_module_forward(kind):
    from types import SimpleNamespace

    import torch

    from dl_reference_models_b200.evaluate import evaluate
    from dl_reference_models_b200.policy_kernels import FusedPolicy, FusedRecurrentPolicy
    from dl_reference_models_b200.recurrent import RecurrentActionMaskPolicy
    from dl_reference_models_b200.rollout import ActionMaskPolicy

    cfg = eval_cfg()
    torch.manual_seed(5)
    recurrent = kind.startswith("lstm")
    policy = (RecurrentActionMaskPolicy(28, cell=32) if recurrent else ActionMaskPolicy(28, hiddens=(32, 32))).cuda()
    carry = {}

    @torch.no_grad()
    def by_hand(env, out):
        M = env.B * env.N
        feats, mask = env.flat_obs(include_action_mask=False).reshape(M, -1), out.action_mask.reshape(M, 5)
        if not recurrent:
            return torch.argmax(policy(feats, mask)[0], -1).to(torch.int8).reshape(env.B, env.N)
        if not carry:
            carry.update(s=policy.initial_state(M, env.device), a=torch.zeros(M, dtype=torch.int64, device=env.device),
                         r=torch.zeros(M, device=env.device))
        else:
            carry["r"] = out.reward.reshape(M).clone()
        lg, _, carry["s"] = policy.step(feats, mask, carry["a"], carry["r"], carry["s"])
        carry["a"] = torch.argmax(lg, -1)
        return carry["a"].to(torch.int8).reshape(env.B, env.N)

    stub = SimpleNamespace(V=5, include_blocking_pressure=True)   # the test env's feature width, F = 28
    assert not (FusedRecurrentPolicy if recurrent else FusedPolicy).matches(policy, stub)
    res = evaluate(cfg, 211, policy=policy)
    same_results(res, evaluate(cfg, 211, policy=by_hand))
    assert carry or not recurrent


@pytest.mark.parametrize("kind", ["mlp", "lstm"])
def test_explore_draws_only_allowed_actions(kind):
    import torch

    from dl_reference_models_b200.batched_env import BatchedMapfEnv
    from dl_reference_models_b200.evaluate import _module_actor, evaluate
    from dl_reference_models_b200.recurrent import RecurrentActionMaskPolicy
    from dl_reference_models_b200.rollout import ActionMaskPolicy

    cfg = eval_cfg()
    torch.manual_seed(6)
    policy = (RecurrentActionMaskPolicy(28) if kind == "lstm" else ActionMaskPolicy(28)).cuda()
    env = BatchedMapfEnv(cfg, 1024, "cuda:0")
    out = env.reset()
    act = _module_actor(env, policy, explore=True)
    allowed, total = 0, 0
    for _ in range(10):
        a = act(out)
        allowed += int((out.action_mask.gather(-1, a.long().unsqueeze(-1)) == 1).sum())
        total += a.numel()
        out = env.step(a, auto_reset=False)
    assert allowed / total >= 0.9999
    env.close()
    res, greedy = evaluate(cfg, 256, policy=policy, explore=True), evaluate(cfg, 256, policy=policy)
    assert res.rows != greedy.rows and all(r["timesteps"] >= 1 for r in res.rows)


def test_refusals():
    from dl_reference_models_b200.evaluate import evaluate
    from dl_reference_models_b200.recurrent import RecurrentActionMaskPolicy
    from dl_reference_models_b200.rollout import ActionMaskPolicy

    cfg = eval_cfg()
    with pytest.raises(ValueError, match="27 features.*28"):
        evaluate(cfg, 8, policy=ActionMaskPolicy(27).cuda())
    with pytest.raises(ValueError, match="features"):
        evaluate(cfg, 8, policy=RecurrentActionMaskPolicy(30).cuda())
    with pytest.raises(ValueError, match="cpu"):
        evaluate(cfg, 8, policy=ActionMaskPolicy(28))
    with pytest.raises(ValueError, match="cpu"):
        evaluate(cfg, 8, policy=RecurrentActionMaskPolicy(28, cell=32))
