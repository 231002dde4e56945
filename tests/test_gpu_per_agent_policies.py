"""Per-agent (DTE) fused policies: mapf_policy_act_per_agent / mapf_lstm_policy_act_per_agent against the shared
entry points bit for bit (agent j's outputs = the shared launch with agent j's block, at agent j's rows), the
collectors against manual loops of per-agent launches, one PPO update, and the evaluator."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

CASES = [(sr, n) for sr in (1, 2, 3) for n in (3, 16, 32)]


def make_env(sr=2, n=16, B=37, steps_per_episode=64, seed=21):
    from dl_reference_models_b200 import maps
    from dl_reference_models_b200.batched_env import BatchedMapfEnv

    cfg = {"num_agents": n, "sensor_range": sr, "steps_per_episode": steps_per_episode, "lifelong_mapf": True,
           "seed": seed, "grid": maps.random_obstacle_grid(32, 32, 0.3, 2026, min_free=2 * n)}
    env = BatchedMapfEnv(cfg, B, "cuda:0")
    out = env.reset()
    for _ in range(5):
        out = env.step(env.sample_actions(masked=True), auto_reset=True)
    return env, out


def per_agent(kind, env, distinct=True, seed=0):
    import torch

    from dl_reference_models_b200.recurrent import PerAgentRecurrentPolicy, RecurrentActionMaskPolicy
    from dl_reference_models_b200.rollout import ActionMaskPolicy, PerAgentActionMaskPolicy

    F = env.flat_obs_dim(include_action_mask=False)
    torch.manual_seed(seed)
    cls, mod = (PerAgentActionMaskPolicy, ActionMaskPolicy) if kind == "mlp" else (PerAgentRecurrentPolicy,
                                                                                   RecurrentActionMaskPolicy)
    if distinct:
        return cls(env.N, F).to(env.device)
    one = mod(F)
    return cls.from_modules([one] * env.N).to(env.device), one.to(env.device)


def mlp_launch(fused, out, greedy, counter):
    import torch

    B, N, F, dev = fused.env.B, fused.env.N, fused.F, fused.env.device
    o = {"logits": torch.full((B, N, 5), 7.0, device=dev), "features": torch.full((B, N, F), 7.0, device=dev),
         "mask": torch.full((B, N, 5), 7, dtype=torch.int8, device=dev), "logp": torch.zeros(B, N, device=dev),
         "value": torch.zeros(B, N, device=dev), "actions64": torch.zeros(B, N, dtype=torch.int64, device=dev)}
    fused.counter = counter - 1
    fused.act(out, logits_out=o["logits"], features_out=o["features"], logp=o["logp"], value=o["value"],
              actions64=o["actions64"], mask_out=o["mask"], greedy=greedy)
    o["actions"] = fused.actions.clone()
    return o


@pytest.mark.parametrize("sr,n", CASES)
def test_mlp_per_agent_kernel_equals_the_shared_kernel_per_agent(sr, n):
    import torch

    from dl_reference_models_b200.policy_kernels import FusedPolicy

    env, out = make_env(sr, n)
    assert env.B % 32 != 0 and (n == 32 or (env.B * env.N) % 32 != 0)   # partial tiles in both tile layouts
    pa = per_agent("mlp", env)
    fp = FusedPolicy(pa, env, seed=11)
    assert fp.entry == "mapf_policy_act_per_agent"
    shared = [FusedPolicy(pa.module(j), env, seed=11) for j in range(n)]
    for greedy in (False, True):
        got = mlp_launch(fp, out, greedy, 3)
        for j in range(n):
            want = mlp_launch(shared[j], out, greedy, 3)
            for k in got:
                assert torch.equal(got[k][:, j], want[k][:, j]), (greedy, j, k)
    # all blocks equal: every output equals the shared launch's, bit for bit
    pa1, one = per_agent("mlp", env, distinct=False)
    f1, f0 = FusedPolicy(pa1, env, seed=11), FusedPolicy(one, env, seed=11)
    for greedy in (False, True):
        got, want = mlp_launch(f1, out, greedy, 5), mlp_launch(f0, out, greedy, 5)
        for k in got:
            assert torch.equal(got[k], want[k]), (greedy, k)
    assert env.poll_errors() == 0


def lstm_inputs(env, seed=0):
    import torch

    g = torch.Generator(device=env.device).manual_seed(seed)
    B, N, dev = env.B, env.N, env.device
    h = torch.randn(B * N, 64, device=dev, generator=g) * 0.5
    c = torch.randn(B * N, 64, device=dev, generator=g)
    pa = torch.randint(0, 5, (B, N), device=dev, generator=g).to(torch.int8)
    pr = torch.randint(-4, 3, (B, N), device=dev, generator=g).float() * 0.5
    term = (torch.rand(B, device=dev, generator=g) < 0.2).to(torch.uint8)
    trunc = (torch.rand(B, device=dev, generator=g) < 0.1).to(torch.uint8)
    assert bool(term.any()) and not bool(term.all())
    return h, c, pa, pr, term, trunc


def lstm_launch(fused, out, inputs, greedy, in_place, counter):
    import torch

    B, N, dev = fused.env.B, fused.env.N, fused.env.device
    h, c, pa, pr, term, trunc = (t.clone() for t in inputs)
    o = {"logits": torch.full((B, N, 5), 7.0, device=dev), "logp": torch.zeros(B, N, device=dev),
         "value": torch.zeros(B, N, device=dev), "actions64": torch.zeros(B, N, dtype=torch.int64, device=dev)}
    so = None if in_place else (torch.full_like(h, 7.0), torch.full_like(c, 7.0))
    fused.counter = counter - 1
    fused.actions.copy_(pa)
    fused.act(out, (h, c), fused.actions, pr, term, trunc, state_out=so, logits_out=o["logits"], logp=o["logp"],
              value=o["value"], actions64=o["actions64"], greedy=greedy)
    ho, co = (h, c) if in_place else so
    o.update(actions=fused.actions.clone(), h=ho.view(B, N, 64), c=co.view(B, N, 64))
    if not in_place:
        assert torch.equal(h, inputs[0]) and torch.equal(c, inputs[1])
    return o


@pytest.mark.parametrize("sr,n", CASES)
def test_lstm_per_agent_kernel_equals_the_shared_kernel_per_agent(sr, n):
    import torch

    from dl_reference_models_b200.policy_kernels import FusedRecurrentPolicy

    env, out = make_env(sr, n)
    pa = per_agent("lstm", env)
    fp = FusedRecurrentPolicy(pa, env, seed=13)
    assert fp.entry == "mapf_lstm_policy_act_per_agent"
    shared = [FusedRecurrentPolicy(pa.module(j), env, seed=13) for j in range(n)]
    inputs = lstm_inputs(env, seed=sr * 100 + n)
    for greedy in (False, True):
        for in_place in (True, False):
            got = lstm_launch(fp, out, inputs, greedy, in_place, 4)
            for j in range(n):
                want = lstm_launch(shared[j], out, inputs, greedy, in_place, 4)
                for k in got:
                    assert torch.equal(got[k][:, j], want[k][:, j]), (greedy, in_place, j, k)
    pa1, one = per_agent("lstm", env, distinct=False)
    f1, f0 = FusedRecurrentPolicy(pa1, env, seed=13), FusedRecurrentPolicy(one, env, seed=13)
    for greedy in (False, True):
        for in_place in (True, False):
            got, want = lstm_launch(f1, out, inputs, greedy, in_place, 6), lstm_launch(f0, out, inputs, greedy, in_place, 6)
            for k in got:
                assert torch.equal(got[k], want[k]), (greedy, in_place, k)
    assert env.poll_errors() == 0


def test_mlp_collector_equals_a_manual_loop_and_trains():
    import torch

    from dl_reference_models_b200.policy_kernels import FusedPolicy
    from dl_reference_models_b200.rollout import FusedCollector, ppo_update

    T = 24
    ea, _ = make_env(B=203, n=7, steps_per_episode=20)
    eb, out = make_env(B=203, n=7, steps_per_episode=20)
    pol = per_agent("mlp", ea)
    fa = FusedPolicy(pol, ea, seed=5)
    col = FusedCollector(ea, fa, T, compact=True)
    fb = FusedPolicy(pol, eb, seed=5)
    for rnd in range(2):
        batch = col.collect()
        rec = {k: [] for k in ("local_obs", "goal_delta", "blocking_prev", "masks", "actions", "logp", "values", "rewards",
                               "dones")}
        for t in range(T):
            rec["local_obs"].append(out.local_obs.clone())
            rec["goal_delta"].append(out.goal_delta.clone())
            rec["blocking_prev"].append(out.blocking_prev.clone())
            rec["masks"].append(out.action_mask.clone())
            a, lp, v = fb.act(out)
            rec["actions"].append(fb.actions64.clone())
            rec["logp"].append(lp.clone())
            rec["values"].append(v.clone())
            out = eb.step(a, auto_reset=True)
            rec["rewards"].append(out.reward.clone())
            rec["dones"].append((out.terminated | out.truncated).bool())
        _, _, lv = fb.act(out)
        for k, v in rec.items():
            got = getattr(batch, k)
            got = got[:T] if k in ("local_obs", "goal_delta", "blocking_prev") else got
            assert torch.equal(got, torch.stack(v)), f"round {rnd}: {k}"
        assert torch.equal(batch.local_obs[T], out.local_obs) and torch.equal(batch.last_value, lv), rnd
        assert bool(batch.dones.any())
    opt = torch.optim.Adam(pol.parameters(), lr=1e-3)
    st = ppo_update(pol, opt, batch, epochs=1, minibatch=256, max_minibatches=3)
    assert st and all(np.isfinite(v) for v in st.values())
    fa.refresh()
    _, logp, value = fa.act(ea._output())
    assert bool(torch.isfinite(logp).all()) and bool(torch.isfinite(value).all())
    assert ea.poll_errors() == 0 and eb.poll_errors() == 0


LSTM_FIELDS = ("local_obs", "goal_delta", "blocking_prev", "masks", "actions", "prev_actions", "prev_rewards", "resets",
               "logp", "values", "rewards", "dones", "last_value", "chunk_h", "chunk_c")


def test_recurrent_collector_equals_a_manual_loop_and_trains():
    import torch

    from dl_reference_models_b200.policy_kernels import FusedRecurrentPolicy
    from dl_reference_models_b200.recurrent import FusedRecurrentCollector, ppo_update_recurrent

    T, L = 64, 32
    ea, _ = make_env(B=203, n=7)
    eb, out = make_env(B=203, n=7)
    pol = per_agent("lstm", ea)
    fa = FusedRecurrentPolicy(pol, ea, seed=5)
    col = FusedRecurrentCollector(ea, fa, T, L)
    fb = FusedRecurrentPolicy(pol, eb, seed=5)
    B, N, dev = eb.B, eb.N, eb.device
    h, c = torch.zeros(B * N, 64, device=dev), torch.zeros(B * N, 64, device=dev)
    pr = torch.zeros(B, N, device=dev)
    pt, ptr = torch.ones(B, dtype=torch.uint8, device=dev), torch.zeros(B, dtype=torch.uint8, device=dev)
    for rnd in range(2):
        batch = col.collect()
        rec = {k: [] for k in LSTM_FIELDS}
        ch, cc = [], []
        for t in range(T):
            rs = (pt | ptr).bool()
            keep = (~rs).repeat_interleave(N).unsqueeze(-1).float()
            if t % L == 0:
                ch.append(h * keep)
                cc.append(c * keep)
            rec["local_obs"].append(out.local_obs.clone())
            rec["goal_delta"].append(out.goal_delta.clone())
            rec["blocking_prev"].append(out.blocking_prev.clone())
            rec["masks"].append(out.action_mask.clone())
            rec["resets"].append(rs)
            rec["prev_actions"].append(fb.actions.long() * (~rs).unsqueeze(-1))
            rec["prev_rewards"].append(pr * (~rs).unsqueeze(-1))
            a, lp, v = fb.act(out, (h, c), fb.actions, pr, pt, ptr)
            rec["actions"].append(a.long())
            rec["logp"].append(lp.clone())
            rec["values"].append(v.clone())
            out = eb.step(a, auto_reset=True)
            rec["rewards"].append(out.reward.clone())
            rec["dones"].append((out.terminated | out.truncated).bool())
            pr, pt, ptr = out.reward.clone(), out.terminated.clone(), out.truncated.clone()
        _, _, lv = fb.act(out, (h, c), fb.actions, pr, pt, ptr, advance=False)
        want = {k: torch.stack(v) for k, v in rec.items() if v}
        want.update(last_value=lv, chunk_h=torch.stack(ch), chunk_c=torch.stack(cc))
        for k in LSTM_FIELDS:
            got = getattr(batch, k)
            assert got.shape == want[k].shape and torch.equal(got, want[k]), f"round {rnd}: {k}"
        assert torch.equal(col.state[0], h) and torch.equal(col.state[1], c)
    opt = torch.optim.Adam(pol.parameters(), lr=1e-3)
    st = ppo_update_recurrent(pol, opt, batch, max_seq_len=L, epochs=1, minibatch=256, max_minibatches=3)
    assert st and all(np.isfinite(v) for v in st.values())
    fa.refresh()
    _, logp, value = fa.act(ea._output(), col.state, fa.actions, torch.zeros(B, N, device=dev), advance=False)
    assert bool(torch.isfinite(logp).all()) and bool(torch.isfinite(value).all())
    assert ea.poll_errors() == 0 and eb.poll_errors() == 0


EVAL_CFG = {"num_agents": 8, "sensor_range": 2, "steps_per_episode": 40, "lifelong_mapf": False, "seed": 17}


def eval_cfg(**kw):
    from dl_reference_models_b200 import maps

    return dict(EVAL_CFG, grid=maps.random_obstacle_grid(16, 16, 0.2, 7, min_free=16), **kw)


def same_results(a, b):
    assert a.rows == b.rows
    assert np.array_equal(a.occupancy_grid, b.occupancy_grid)
    assert (a.success_rate, a.average_reward, a.average_timesteps, a.lifelong) == \
        (b.success_rate, b.average_reward, b.average_timesteps, b.lifelong)


@pytest.mark.parametrize("kind", ["mlp", "lstm"])
def test_evaluate_per_agent_modules(kind):
    import torch

    from dl_reference_models_b200.evaluate import evaluate
    from dl_reference_models_b200.policy_kernels import FusedPolicy, FusedRecurrentPolicy
    from dl_reference_models_b200.recurrent import PerAgentRecurrentPolicy, RecurrentActionMaskPolicy
    from dl_reference_models_b200.rollout import ActionMaskPolicy, PerAgentActionMaskPolicy

    cfg = eval_cfg(lifelong_mapf=kind == "lstm")
    torch.manual_seed(5)
    cls, mod = (PerAgentActionMaskPolicy, ActionMaskPolicy) if kind == "mlp" else (PerAgentRecurrentPolicy,
                                                                                   RecurrentActionMaskPolicy)
    policy = cls(8, 28).cuda()
    carry = {}

    def by_hand(env, out):   # the same fused greedy launches, written out
        M = env.B * env.N
        if kind == "mlp":
            carry.setdefault("f", FusedPolicy(policy, env))
            return carry["f"].act(out, greedy=True)[0]
        if not carry:
            carry.update(f=FusedRecurrentPolicy(policy, env), h=torch.zeros(M, 64, device=env.device),
                         c=torch.zeros(M, 64, device=env.device), r=torch.zeros(env.B, env.N, device=env.device))
        else:
            carry["r"] = out.reward.clone()
        f = carry["f"]
        return f.act(out, (carry["h"], carry["c"]), f.actions, carry["r"], greedy=True)[0]

    res = evaluate(cfg, 301, policy=policy)
    same_results(res, evaluate(cfg, 301, policy=by_hand))
    assert carry["f"].per_agent
    # N copies of one module = that module shared
    one = mod(28).cuda()
    same_results(evaluate(cfg, 301, policy=cls.from_modules([one] * 8)), evaluate(cfg, 301, policy=one))
    # a non-reference per-agent shape runs its PyTorch forward
    small = cls(8, 28, hiddens=(32, 32)).cuda()
    assert not (FusedPolicy.matches(small, carry["f"].env) or FusedRecurrentPolicy.matches(small, carry["f"].env))
    r = evaluate(cfg, 97, policy=small)
    assert len(r.rows) == 97 and all(row["timesteps"] >= 1 for row in r.rows)
    with pytest.raises(ValueError, match="num_agents = 7.*num_agents = 8"):
        evaluate(cfg, 5, policy=cls(7, 28).cuda())
