"""The fused recurrent centralised CTE policy (mapf_cte_lstm_policy_act: trunk launch, then the LSTM step with the heads
and N masked draws), its collector and its learner, against plain PyTorch.  Maps 2-1 (10x20), 3-1 (20x30) and a random
32x32 one, N in {1, 4, 16, 32}, batches that are not a multiple of the kernels' 32-env tiles.  Tolerances: the kernels
round W1, W2, the trunk output, W_ih (except its reward column, kept in f32), W_hh, h, h' and the heads to bf16 and
accumulate in f32; against a torch step that rounds at the same points, logits, value, h' and c' agree to 2e-4 on
average and 3e-2 at worst."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

CASES = [("ReferenceModel-2-1", 1), ("ReferenceModel-2-1", 4), ("ReferenceModel-3-1", 16), ("ReferenceModel-3-1", 32),
         ("rand32", 1), ("rand32", 16), ("rand32", 32)]


def make_env(name, n, B=1003, steps_per_episode=64, seed=5, scramble=3):
    import torch

    from dl_reference_models_b200 import maps
    from dl_reference_models_b200.single_agent import BatchedCteEnv

    grid = maps.random_obstacle_grid(32, 32, 0.30, 2026, min_free=64) if name == "rand32" else maps.get_grid(name)
    env = BatchedCteEnv({"grid": grid, "num_agents": n, "steps_per_episode": steps_per_episode, "seed": seed}, B)
    env.reset()
    g = torch.Generator(device=env.device).manual_seed(seed)
    for _ in range(scramble):
        env.step(torch.randint(0, 5, (B, n), dtype=torch.int8, device=env.device, generator=g), auto_reset=True)
    return env


def make_policy(env, seed=0):
    import torch

    from dl_reference_models_b200.cte_rollout import CteRecurrentPolicy

    torch.manual_seed(seed)
    return CteRecurrentPolicy(env.R * env.C, env.N).to(env.device)


def random_inputs(env, seed=0, start_frac=0.2):
    """A random recurrent state, previous joint actions, rewards with the CTE penalties and episode-start flags."""
    import torch

    g = torch.Generator(device=env.device).manual_seed(seed)
    B, N, dev = env.B, env.N, env.device
    h = torch.randn((B, 64), device=dev, generator=g) * 0.5
    c = torch.randn((B, 64), device=dev, generator=g)
    pa = torch.randint(0, 5, (B, N), dtype=torch.int8, device=dev, generator=g)
    choices = torch.tensor([-0.2, -0.05, -0.25, 1.0, 0.0, 0.75], dtype=torch.float64, device=dev)
    pr = choices[torch.randint(0, len(choices), (B,), device=dev, generator=g)]
    start = (torch.rand(B, device=dev, generator=g) < start_frac).to(torch.uint8)
    return h, c, pa, pr, start


def bf16_reference(policy, grid, mask, pa, pr, h, c, start):
    """The kernels' arithmetic in float64 with bf16 rounding at their points -> (logits [B,N,5], value, h', c')."""
    import torch

    r = lambda t: t.float().to(torch.bfloat16).double()  # noqa: E731
    B, N = mask.shape[0], policy.num_agents
    keep = (start == 0).double().unsqueeze(-1)
    h, c = h.double() * keep, c.double() * keep
    pa = pa.long() * (start == 0).long().unsqueeze(-1)
    pr = pr.float().double() * keep.squeeze(-1)
    y = grid.reshape(B, -1).double()
    for l in [m for m in policy.trunk if isinstance(m, torch.nn.Linear)]:
        y = r(torch.relu(y @ r(l.weight).T + l.bias.double()))
    wih, whh = policy.lstm.weight_ih, policy.lstm.weight_hh
    onehot = torch.nn.functional.one_hot(pa, 5).reshape(B, 5 * N).double()
    gates = (y @ r(wih[:, :64]).T + onehot @ r(wih[:, 64:64 + 5 * N]).T + pr.unsqueeze(-1) * wih[:, 64 + 5 * N].double()
             + r(h) @ r(whh).T + (policy.lstm.bias_ih.float() + policy.lstm.bias_hh.float()).double())
    i, f, g, o = gates.chunk(4, -1)
    c2 = torch.sigmoid(f) * c + torch.sigmoid(i) * torch.tanh(g)
    h2 = torch.sigmoid(o) * torch.tanh(c2)
    hb = r(h2)
    logits = hb @ r(policy.logits.weight).T + policy.logits.bias.double()
    logits = logits + torch.where(mask != 0, 9.99999e-07, -13.815511).double()
    value = (hb @ r(policy.value.weight).T + policy.value.bias.double()).squeeze(-1)
    return logits.reshape(B, N, 5), value, h2, c2


def call(fused, inputs, *, advance=True, state_out=None, counter=1, **kw):
    import torch

    h, c, pa, pr, start = inputs
    env = fused.env
    logits = torch.zeros((env.B, env.N, 5), device=env.device)
    fused.counter = counter - 1
    a, lp, v = fused.act((h, c), pa, pr, start, None, advance=advance, state_out=state_out, logits_out=logits, **kw)
    return a.clone(), lp.clone(), v.clone(), logits


@pytest.mark.parametrize("name,n", CASES)
def test_one_call_matches_torch(name, n):
    import torch

    from dl_reference_models_b200.policy_kernels import FusedCteRecurrentPolicy

    env = make_env(name, n)
    policy = make_policy(env)
    fused = FusedCteRecurrentPolicy(policy, env, seed=7)
    h, c, pa, pr, start = random_inputs(env)
    ho, co = torch.zeros_like(h), torch.zeros_like(c)
    acts, logp, value, logits = call(fused, (h, c, pa, pr, start), state_out=(ho, co))
    with torch.no_grad():
        ref_l, ref_v, ref_h, ref_c = bf16_reference(policy, env.obs_grid, env.action_mask, pa, pr, h, c, start)
    for what, got, want in (("logits", logits, ref_l), ("value", value, ref_v), ("h", ho, ref_h), ("c", co, ref_c)):
        d = (got.double() - want).abs()
        assert float(d.max()) <= 3e-2 and float(d.mean()) <= 2e-4, (what, float(d.mean()), float(d.max()))
    ref_logp = torch.log_softmax(logits.double(), -1).gather(-1, acts.long().unsqueeze(-1)).squeeze(-1).sum(-1)
    assert float((logp.double() - ref_logp).abs().max()) <= 1e-4
    assert torch.equal(fused.actions64, acts.long())
    mask = env.action_mask.view(env.B, n, 5)
    assert bool((mask.gather(-1, acts.long().unsqueeze(-1)) == 1).all())


@pytest.mark.parametrize("name,n", [("ReferenceModel-2-1", 4), ("rand32", 32)])
def test_episode_start_flags_equal_explicitly_zeroed_inputs(name, n):
    import torch

    from dl_reference_models_b200.policy_kernels import FusedCteRecurrentPolicy

    env = make_env(name, n)
    fused = FusedCteRecurrentPolicy(make_policy(env), env, seed=5)
    h, c, pa, pr, start = random_inputs(env, seed=1, start_frac=0.3)
    ho1, co1 = torch.zeros_like(h), torch.zeros_like(c)
    got = call(fused, (h, c, pa, pr, start), state_out=(ho1, co1))
    keep = (start == 0)
    z = (h * keep.unsqueeze(-1), c * keep.unsqueeze(-1), pa * keep.unsqueeze(-1).to(pa.dtype), pr * keep, torch.zeros_like(start))
    ho2, co2 = torch.zeros_like(h), torch.zeros_like(c)
    want = call(fused, z, state_out=(ho2, co2))
    for x, y in zip(got + (ho1, co1), want + (ho2, co2)):
        assert torch.equal(x, y)


@pytest.mark.parametrize("name,n", [("ReferenceModel-3-1", 16), ("rand32", 32)])
def test_in_place_equals_out_of_place_and_no_state_out_leaves_the_state(name, n):
    import torch

    from dl_reference_models_b200.policy_kernels import FusedCteRecurrentPolicy

    env = make_env(name, n)
    fused = FusedCteRecurrentPolicy(make_policy(env), env, seed=2)
    h, c, pa, pr, start = random_inputs(env, seed=3)
    ho, co = torch.zeros_like(h), torch.zeros_like(c)
    out = call(fused, (h, c, pa, pr, start), state_out=(ho, co))
    # in place, with prev_action aliasing the launch's own action buffer
    fused.actions.copy_(pa)
    hi, ci = h.clone(), c.clone()
    inp = call(fused, (hi, ci, fused.actions, pr, start))
    for x, y in zip(out + (ho, co), inp + (hi, ci)):
        assert torch.equal(x, y)
    # no state out: state and the action buffer untouched, the outputs as before
    h2, c2 = h.clone(), c.clone()
    fused.actions.copy_(pa)
    a_before = fused.actions.clone()
    _, lp, v, lg = call(fused, (h2, c2, fused.actions, pr, start), advance=False)
    assert torch.equal(h2, h) and torch.equal(c2, c) and torch.equal(fused.actions, a_before)
    assert torch.equal(lp, out[1]) and torch.equal(v, out[2]) and torch.equal(lg, out[3])
    assert torch.equal(fused.actions64, out[0].long())


def test_draws_follow_the_softmax_of_the_launch_logits():
    """The same observation and state in every env, different Philox streams: per agent, the action frequencies
    follow the softmax of the launch's own logits."""
    import torch

    from dl_reference_models_b200.policy_kernels import FusedCteRecurrentPolicy

    env = make_env("ReferenceModel-2-1", 4, B=4096)
    env.obs_grid.copy_(env.obs_grid[:1].expand_as(env.obs_grid).clone())
    env.action_mask.copy_(env.action_mask[:1].expand_as(env.action_mask).clone())
    fused = FusedCteRecurrentPolicy(make_policy(env, seed=1), env)
    h, c, pa, pr, start = (x[:1].expand_as(x).contiguous() for x in random_inputs(env, seed=4))
    counts = torch.zeros((env.N, 5), device=env.device)
    draws = 0
    for k in range(20):
        _, _, _, logits = call(fused, (h, c, pa, pr, start), advance=False, counter=k + 1)
        counts += torch.nn.functional.one_hot(fused.actions64.long(), 5).sum(0)
        draws += env.B
    assert torch.equal(logits, logits[:1].expand_as(logits))
    exp = torch.softmax(logits[0], -1) * draws
    keep = exp > 5
    chi2 = (((counts - exp) ** 2 / exp.clamp_min(1e-9)) * keep).sum(-1)
    assert float(chi2.max()) < 40, (counts.tolist(), exp.tolist())   # <= 4 dof per agent, 4 agents


@pytest.mark.parametrize("name", ["ReferenceModel-2-1", "rand32"])
def test_a_shard_with_its_env_id_base_reproduces_the_full_launch(name):
    import torch

    from dl_reference_models_b200.policy_kernels import FusedCteRecurrentPolicy

    env = make_env(name, 16 if name == "rand32" else 4)
    policy = make_policy(env)
    h, c, pa, pr, start = random_inputs(env, seed=6)
    full = FusedCteRecurrentPolicy(policy, env, seed=3)
    hf, cf = h.clone(), c.clone()
    a, lp, v, lf = call(full, (hf, cf, pa, pr, start))
    off, n = 37, 500
    shard = FusedCteRecurrentPolicy(policy, env, seed=3, env_id_base=off)
    sl = slice(off, off + n)
    hs, cs = h[sl].clone(), c[sl].clone()
    ls = torch.zeros((n, env.N, 5), device=env.device)
    shard.counter = 0
    sa, slp, sv = shard.act((hs, cs), pa[sl].contiguous(), pr[sl].contiguous(), start[sl].contiguous(),
                            obs_grid=env.obs_grid[sl], action_mask=env.action_mask[sl], logits_out=ls, num_envs=n)
    assert torch.equal(sa[:n], a[sl]) and torch.equal(slp[:n], lp[sl]) and torch.equal(sv[:n], v[sl])
    assert torch.equal(ls, lf[sl]) and torch.equal(hs, hf[sl]) and torch.equal(cs, cf[sl])


def test_collector_equals_a_manual_loop_over_two_collects():
    import torch

    from dl_reference_models_b200.cte_rollout import FusedRecurrentCteCollector
    from dl_reference_models_b200.policy_kernels import FusedCteRecurrentPolicy

    n, B, T, L = 4, 203, 8, 4
    envs = [make_env("ReferenceModel-2-1", n, B=B, steps_per_episode=5, seed=9) for _ in range(2)]
    policy = make_policy(envs[0])
    fa, fb = FusedCteRecurrentPolicy(policy, envs[0], seed=4), FusedCteRecurrentPolicy(policy, envs[1], seed=4)
    collector = FusedRecurrentCteCollector(envs[0], fa, T, max_seq_len=L)
    env, dev = envs[1], envs[1].device
    cells = env.R * env.C
    h, c = torch.zeros((B, 64), device=dev), torch.zeros((B, 64), device=dev)
    prev_reward = torch.zeros(B, dtype=torch.float64, device=dev)
    pterm, ptrunc = torch.ones(B, dtype=torch.uint8, device=dev), torch.zeros(B, dtype=torch.uint8, device=dev)
    ended = 0
    for round_ in range(2):
        batch = collector.collect()
        want = {k: [] for k in ("grid", "masks", "actions", "logp", "values", "rewards", "dones", "prev_actions",
                                "prev_rewards", "resets", "chunk_h", "chunk_c")}
        for t in range(T):
            rs = (pterm | ptrunc).bool()
            keep = ~rs
            want["grid"].append(env.obs_grid.view(B, cells).clone())
            want["masks"].append(env.action_mask.clone())
            want["resets"].append(rs)
            want["prev_actions"].append(fb.actions.long() * keep.unsqueeze(-1))
            want["prev_rewards"].append(prev_reward.float() * keep)
            if t % L == 0:
                want["chunk_h"].append(h * keep.unsqueeze(-1))
                want["chunk_c"].append(c * keep.unsqueeze(-1))
            a, lp, v = fb.act((h, c), fb.actions, prev_reward, pterm, ptrunc)
            want["actions"].append(fb.actions64.clone())
            want["logp"].append(lp.clone())
            want["values"].append(v.clone())
            env.step(a, auto_reset=True)
            want["rewards"].append(env.reward.float())
            want["dones"].append((env.terminated | env.truncated).bool())
            prev_reward, pterm, ptrunc = env.reward.clone(), env.terminated.clone(), env.truncated.clone()
        want["grid"].append(env.obs_grid.view(B, cells).clone())
        want["masks"].append(env.action_mask.clone())
        _, _, last = fb.act((h, c), fb.actions, prev_reward, pterm, ptrunc, advance=False)
        for field, w in want.items():
            assert torch.equal(getattr(batch, field), torch.stack(w)), (round_, field)
        assert torch.equal(batch.last_value, last), round_
        assert torch.equal(collector.state[0], h) and torch.equal(collector.state[1], c), round_
        ended += int(batch.dones.sum())
        for k in ("positions", "goals", "starts", "reached_once", "step_count", "blocking_total", "obs_grid",
                  "action_mask", "flat_obs", "reward", "terminated", "truncated", "info"):
            assert torch.equal(getattr(envs[0], k), getattr(env, k)), (round_, k)
    assert ended > B   # episodes of 5 steps end and auto-reset inside the window


def test_fp32_module_rerun_over_a_fused_batch():
    """What PPO sees: the fp32 module re-run through its sequences over a fused batch at default init.  The
    differences and the importance ratios are printed (pytest -s) for the record."""
    import torch

    from dl_reference_models_b200.cte_rollout import FusedRecurrentCteCollector, joint_logp_entropy
    from dl_reference_models_b200.policy_kernels import FusedCteRecurrentPolicy

    env = make_env("rand32", 16, B=2051, steps_per_episode=32)
    policy = make_policy(env)
    batch = FusedRecurrentCteCollector(env, FusedCteRecurrentPolicy(policy, env), 32, max_seq_len=32).collect()
    T = batch.actions.shape[0]
    with torch.no_grad():
        lg, v, _ = policy.sequence(batch.grid[:T], batch.masks[:T], batch.prev_actions, batch.prev_rewards, batch.resets,
                                   (batch.chunk_h[0], batch.chunk_c[0]))
        lp, _ = joint_logp_entropy(lg, batch.actions)
    dlp, dv = (lp - batch.logp).abs(), (v - batch.values).abs()
    ratio = torch.exp(lp - batch.logp)
    print(f"\nfp32 re-run over a fused recurrent CTE batch (N=16, 32x32, T=32): |dlogp| mean {float(dlp.mean()):.3g} max "
          f"{float(dlp.max()):.3g}; |dvalue| mean {float(dv.mean()):.3g} max {float(dv.max()):.3g}; ratio "
          f"{float(ratio.min()):.6f} .. {float(ratio.max()):.6f}")
    assert float(ratio.min()) > 0.9 and float(ratio.max()) < 1.1


def test_a_ppo_update_then_refresh_changes_the_launch():
    import torch

    from dl_reference_models_b200.cte_rollout import FusedRecurrentCteCollector, ppo_update_cte_recurrent
    from dl_reference_models_b200.policy_kernels import FusedCteRecurrentPolicy

    env = make_env("ReferenceModel-3-1", 4, B=515, steps_per_episode=16)
    policy = make_policy(env)
    fused = FusedCteRecurrentPolicy(policy, env, seed=2)
    batch = FusedRecurrentCteCollector(env, fused, 8, max_seq_len=8).collect()
    inputs = random_inputs(env, seed=8)
    before = call(fused, inputs, advance=False)
    opt = torch.optim.Adam(policy.parameters(), lr=1e-3)
    stats = ppo_update_cte_recurrent(policy, opt, batch, max_seq_len=8, epochs=2, minibatch=512,
                                     generator=torch.Generator().manual_seed(0))
    assert all(np.isfinite(x) for x in stats.values()), stats
    fused.refresh()
    after = call(fused, inputs, advance=False)
    assert not torch.equal(after[1], before[1]) and not torch.equal(after[2], before[2])
