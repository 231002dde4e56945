"""Fused LSTM-64 policy kernel (mapf_lstm_policy_act) and FusedRecurrentCollector against the PyTorch module.

Tolerances: the kernel rounds features, weights, trunk activations and h to bf16 and accumulates in f32 (c and the cell
update stay f32); against a torch reference that rounds at the same points logits, value, h' and c' agree to 2e-4 on
average and 3e-2 at worst (the MLP kernel's bounds), against the pure fp32 module to 6e-2 (scaled with the logit
magnitude).  What PPO sees: the fp32 module re-run over the fused batch reproduces its log-probabilities to 5e-4 on
average and 5e-3 at worst, with at most 1e-4 of the importance ratios outside a 0.05 clip."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def make_env(sr=2, B=2048, n=16, steps_per_episode=64):
    from dl_reference_models_b200 import maps
    from dl_reference_models_b200.batched_env import BatchedMapfEnv

    cfg = {"num_agents": n, "sensor_range": sr, "steps_per_episode": steps_per_episode, "lifelong_mapf": True, "seed": 21,
           "grid": maps.random_obstacle_grid(32, 32, 0.3, 2026, min_free=2 * n)}
    env = BatchedMapfEnv(cfg, B, "cuda:0")
    out = env.reset()
    for _ in range(5):
        out = env.step(env.sample_actions(masked=True), auto_reset=True)
    return env, out


def make_policy(env, scale=1.0, seed=0):
    import torch

    from dl_reference_models_b200.recurrent import RecurrentActionMaskPolicy

    torch.manual_seed(seed)
    pol = RecurrentActionMaskPolicy(env.flat_obs_dim(include_action_mask=False)).to(env.device)
    with torch.no_grad():
        for p in pol.parameters():
            p.mul_(scale)
    return pol


def random_inputs(env, seed=0):
    """Nonzero state, previous actions, half-integer previous rewards, ~20 % of the envs starting an episode."""
    import torch

    g = torch.Generator(device=env.device).manual_seed(seed)
    B, N, dev = env.B, env.N, env.device
    h = torch.randn(B * N, 64, device=dev, generator=g) * 0.5
    c = torch.randn(B * N, 64, device=dev, generator=g)
    pa = torch.randint(0, 5, (B, N), device=dev, generator=g).to(torch.int8)
    pr = torch.randint(-4, 3, (B, N), device=dev, generator=g).float() * 0.5
    term = (torch.rand(B, device=dev, generator=g) < 0.1).to(torch.uint8)
    trunc = (torch.rand(B, device=dev, generator=g) < 0.1).to(torch.uint8)
    return h, c, pa, pr, term, trunc


def cut(env, h, c, pa, pr, term, trunc):
    """RecurrentCollector's episode-start rule: state, previous action and reward zero where a flag is set."""
    keep = ~(term | trunc).bool()
    ka = keep.repeat_interleave(env.N).unsqueeze(-1)
    return h * ka, c * ka, pa.long() * keep.unsqueeze(-1), pr * keep.unsqueeze(-1)


def bf16_reference(pol, feats, mask, pa, pr, h, c):
    import torch

    r = lambda t: t.to(torch.bfloat16).to(torch.float32)  # noqa: E731
    x = r(feats)
    for lin in [m for m in pol.trunk if isinstance(m, torch.nn.Linear)]:
        x = r(torch.relu(x @ r(lin.weight).T + lin.bias))
    xi = torch.cat([x, torch.nn.functional.one_hot(pa, 5).float(), r(pr).unsqueeze(-1)], -1)
    lstm = pol.lstm
    gates = xi @ r(lstm.weight_ih).T + r(h) @ r(lstm.weight_hh).T + (lstm.bias_ih + lstm.bias_hh)
    i, f, g, o = gates.chunk(4, -1)
    c1 = torch.sigmoid(f) * c + torch.sigmoid(i) * torch.tanh(g)
    h1 = torch.sigmoid(o) * torch.tanh(c1)
    hb = r(h1)
    logits = hb @ r(pol.logits.weight).T + pol.logits.bias
    value = (hb @ r(pol.value.weight).T + pol.value.bias).squeeze(-1)
    inf_mask = torch.where(mask != 0, torch.full_like(logits, 9.99999e-07), torch.full_like(logits, -13.815511))
    return logits + inf_mask, value, h1, c1


@pytest.mark.parametrize("sr", [1, 2, 3])
def test_one_step_matches_torch(sr):
    import torch

    from dl_reference_models_b200.policy_kernels import FusedRecurrentPolicy

    env, out = make_env(sr=sr, B=1003, n=7)   # B * N odd: the last tile is partial
    pol = make_policy(env, scale=3.0)          # larger logits and gates: a sharper test of the arithmetic
    fused = FusedRecurrentPolicy(pol, env)
    h, c, pa, pr, term, trunc = random_inputs(env, sr)
    h2, c2 = torch.empty_like(h), torch.empty_like(c)
    logits = torch.zeros((env.B, env.N, 5), device=env.device)
    acts, logp, value = fused.act(out, (h, c), pa, pr, term, trunc, state_out=(h2, c2), logits_out=logits)
    M = env.B * env.N
    feats = env.flat_obs(include_action_mask=False).reshape(M, -1)
    mask = out.action_mask.reshape(M, 5)
    h0, c0, pa0, pr0 = cut(env, h, c, pa, pr, term, trunc)
    with torch.no_grad():
        ref_l, ref_v, ref_h, ref_c = bf16_reference(pol, feats, mask, pa0.reshape(-1), pr0.reshape(-1), h0, c0)
        full_l, full_v, (full_h, _) = pol.step(feats, mask, pa0.reshape(-1), pr0.reshape(-1), (h0, c0))
    for name, got, want in (("logits", logits.reshape(M, 5), ref_l), ("value", value.reshape(M), ref_v), ("h", h2, ref_h),
                            ("c", c2, ref_c)):
        d = (got - want).abs()
        assert float(d.max()) <= 3e-2 and float(d.mean()) <= 2e-4, (name, float(d.max()), float(d.mean()))
    assert float((logits.reshape(M, 5) - full_l).abs().max()) <= 6e-2 * max(1.0, float(full_l.abs().max()) / 10)
    assert float((value.reshape(M) - full_v).abs().max()) <= 6e-2 * max(1.0, float(full_v.abs().max()) / 10)
    ref_logp = torch.log_softmax(logits, -1).gather(-1, acts.long().unsqueeze(-1)).squeeze(-1)
    assert float((logp - ref_logp).abs().max()) <= 1e-4
    assert torch.equal(fused.actions64, acts.long())
    assert (out.action_mask.gather(-1, acts.long().unsqueeze(-1)) == 1).float().mean() > 0.9999   # masked: p ~ 1e-6


def test_episode_start_flags_equal_explicitly_zeroed_inputs():
    import torch

    from dl_reference_models_b200.policy_kernels import FusedRecurrentPolicy

    env, out = make_env(B=611, n=5)
    fused = FusedRecurrentPolicy(make_policy(env, scale=2.0), env)
    h, c, pa, pr, term, trunc = random_inputs(env, 7)
    assert bool((term | trunc).any()) and not bool((term | trunc).all())
    runs = []
    for flagged in (True, False):
        if flagged:
            hh, cc, aa, rr, ft, fr = h.clone(), c.clone(), pa.clone(), pr.clone(), term, trunc
        else:
            hh, cc, aa, rr = cut(env, h, c, pa, pr, term, trunc)
            hh, cc, aa, rr, ft, fr = hh.contiguous(), cc.contiguous(), aa.to(torch.int8), rr.contiguous(), None, None
        fused.counter = 10   # the same Philox counter for both launches
        logits = torch.zeros((env.B, env.N, 5), device=env.device)
        acts, logp, value = fused.act(out, (hh, cc), aa, rr, ft, fr, logits_out=logits)
        runs.append((acts.clone(), logp.clone(), value.clone(), logits, hh, cc))
    for name, x, y in zip(("actions", "logp", "value", "logits", "h", "c"), *runs):
        assert torch.equal(x, y), name


def test_in_place_equals_out_of_place_and_null_state_out_leaves_the_state():
    import torch

    from dl_reference_models_b200.policy_kernels import FusedRecurrentPolicy

    env, out = make_env(B=517, n=9)
    fused = FusedRecurrentPolicy(make_policy(env), env)
    h, c, pa, pr, term, trunc = random_inputs(env, 3)
    h0, c0 = h.clone(), c.clone()
    res = []
    for mode in ("out_of_place", "in_place", "no_advance"):
        hh, cc = h0.clone(), c0.clone()
        ho, co = torch.full_like(h, 7.0), torch.full_like(c, 7.0)
        fused.counter = 4
        _, logp, value = fused.act(out, (hh, cc), pa, pr, term, trunc, advance=mode != "no_advance",
                                   state_out=(ho, co) if mode == "out_of_place" else None)
        torch.cuda.synchronize()
        res.append((fused.actions64.clone(), logp.clone(), value.clone(), ho if mode == "out_of_place" else hh,
                    co if mode == "out_of_place" else cc))
        if mode == "no_advance":
            assert torch.equal(hh, h0) and torch.equal(cc, c0)
    for k in range(3):
        assert torch.equal(res[0][k], res[1][k]) and torch.equal(res[0][k], res[2][k]), k
    assert torch.equal(res[0][3], res[1][3]) and torch.equal(res[0][4], res[1][4])
    assert not torch.equal(res[0][3], h0)


def test_sampling_distribution():
    """Same observation and state in every env, different Philox streams: action frequencies follow softmax(logits)."""
    import torch

    from dl_reference_models_b200.policy_kernels import FusedRecurrentPolicy

    env, out = make_env(B=4096, n=4)
    fused = FusedRecurrentPolicy(make_policy(env, seed=1), env)
    for t in (out.local_obs, out.goal_delta, out.blocking_prev, out.action_mask):
        t.copy_(t[:1].expand_as(t).clone())
    M = env.B * env.N
    h = (torch.arange(64, device=env.device).float() / 64 - 0.5).expand(M, 64).contiguous()
    c = h.clone()
    pa = torch.full((env.B, env.N), 2, dtype=torch.int8, device=env.device)
    pr = torch.full((env.B, env.N), -0.5, device=env.device)
    logits = torch.zeros((env.B, env.N, 5), device=env.device)
    counts = torch.zeros((env.N, 5), device=env.device)
    draws = 0
    for _ in range(20):
        acts, _, _ = fused.act(out, (h, c), pa, pr, advance=False, logits_out=logits)
        counts += torch.nn.functional.one_hot(fused.actions64, 5).sum(0)
        draws += env.B
    assert torch.equal(logits, logits[:1].expand_as(logits))
    probs = torch.softmax(logits[0], -1)
    exp = probs * draws
    keep = exp > 5
    chi2 = (((counts - exp) ** 2 / exp.clamp_min(1e-9)) * keep).sum(-1)
    assert float(chi2.max()) < 40, (counts.tolist(), exp.tolist())   # <= 4 dof, 4 agents


FIELDS = ("local_obs", "goal_delta", "blocking_prev", "masks", "actions", "prev_actions", "prev_rewards", "resets", "logp",
          "values", "rewards", "dones", "last_value", "chunk_h", "chunk_c")


def test_collector_equals_a_manual_loop():
    """FusedRecurrentCollector (two launches per step, compact rows) against FusedRecurrentPolicy.act + env.step with
    explicit copies on an identically seeded env, across an episode end and two consecutive collects."""
    import torch

    from dl_reference_models_b200.policy_kernels import FusedRecurrentPolicy
    from dl_reference_models_b200.recurrent import FusedRecurrentCollector

    T, L = 64, 32
    ea, _ = make_env(B=203, n=7)
    eb, out = make_env(B=203, n=7)
    pol = make_policy(ea)
    col = FusedRecurrentCollector(ea, FusedRecurrentPolicy(pol, ea, seed=5), T, L)
    fb = FusedRecurrentPolicy(pol, eb, seed=5)
    B, N, dev = eb.B, eb.N, eb.device
    h, c = torch.zeros(B * N, 64, device=dev), torch.zeros(B * N, 64, device=dev)
    pr = torch.zeros(B, N, device=dev)
    pt, ptr = torch.ones(B, dtype=torch.uint8, device=dev), torch.zeros(B, dtype=torch.uint8, device=dev)
    crossed = False
    for rnd in range(2):
        batch = col.collect()
        rec = {k: [] for k in FIELDS}
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
        for k in FIELDS:
            got = getattr(batch, k)
            assert got.shape == want[k].shape and got.dtype == want[k].dtype, (rnd, k, got.shape, want[k].shape)
            assert torch.equal(got, want[k]), f"round {rnd}: {k}"
        crossed = crossed or bool(batch.dones.any())
        for k in ea.state:
            assert torch.equal(ea.state[k], eb.state[k]), k
        for k in ("local_obs", "goal_delta", "blocking_prev", "action_mask"):
            assert torch.equal(ea.out[k], eb.out[k]), f"round {rnd}: env buffer {k}"
        assert torch.equal(col.state[0], h) and torch.equal(col.state[1], c)
    assert crossed, "the run crosses an episode end"
    assert ea.poll_errors() == 0 and eb.poll_errors() == 0


def test_what_ppo_sees_and_a_training_step():
    """The fp32 module re-run from each chunk's stored state over the batch's recorded inputs (what
    ppo_update_recurrent computes before its first step) reproduces the fused rollout's log-probabilities and values;
    then one PPO update on the fused batch, refresh() and one more launch."""
    import torch

    from dl_reference_models_b200.policy_kernels import FusedRecurrentPolicy
    from dl_reference_models_b200.recurrent import FusedRecurrentCollector, features_from_channels, ppo_update_recurrent

    T, L = 64, 32
    env, _ = make_env(B=512, n=16, steps_per_episode=40)
    pol = make_policy(env)
    fused = FusedRecurrentPolicy(pol, env)
    col = FusedRecurrentCollector(env, fused, T, L)
    col.collect()
    b = col.collect()   # starts from a carried, nonzero state
    assert bool(b.resets.any()) and not bool(b.chunk_h[0].eq(0).all())
    B, N, M = env.B, env.N, env.B * env.N
    dlp, dv = [], []
    with torch.no_grad():
        for k in range(T // L):
            s = slice(k * L, (k + 1) * L)
            feats = features_from_channels(b.local_obs[s], b.goal_delta[s], b.blocking_prev[s]).reshape(L, M, -1)
            rs = b.resets[s].unsqueeze(-1).expand(L, B, N).reshape(L, M)
            lg, v, _ = pol.sequence(feats, b.masks[s].reshape(L, M, 5), b.prev_actions[s].reshape(L, M),
                                    b.prev_rewards[s].reshape(L, M), rs, (b.chunk_h[k], b.chunk_c[k]))
            lp = torch.log_softmax(lg, -1).gather(-1, b.actions[s].reshape(L, M, 1)).squeeze(-1)
            dlp.append(lp - b.logp[s].reshape(L, M))
            dv.append(v - b.values[s].reshape(L, M))
    dlp, dv = torch.cat(dlp), torch.cat(dv)
    outside = float(((dlp.exp() - 1).abs() > 0.05).float().mean())
    stats = {"logp_mean": float(dlp.abs().mean()), "logp_max": float(dlp.abs().max()), "ratio_outside_clip": outside,
             "value_mean": float(dv.abs().mean()), "value_max": float(dv.abs().max())}
    print("fused vs fp32 module over the batch:", stats)
    assert outside <= 1e-4, stats
    assert stats["logp_mean"] <= 5e-4 and stats["logp_max"] <= 5e-3, stats
    assert stats["value_mean"] <= 5e-4 and stats["value_max"] <= 5e-3, stats
    opt = torch.optim.Adam(pol.parameters(), lr=1e-3)
    st = ppo_update_recurrent(pol, opt, b, max_seq_len=L, epochs=1, minibatch=1024, max_minibatches=4)
    assert st and all(np.isfinite(v) for v in st.values())
    fused.refresh()
    h = torch.zeros(M, 64, device=env.device)
    c = torch.zeros_like(h)
    _, logp, value = fused.act(env._output(), (h, c), fused.actions, torch.zeros(B, N, device=env.device))
    assert bool(torch.isfinite(logp).all()) and bool(torch.isfinite(value).all())
    assert env.poll_errors() == 0


def test_collector_refuses_the_fused_uniform_sampler():
    from dl_reference_models_b200.policy_kernels import FusedRecurrentPolicy
    from dl_reference_models_b200.recurrent import FusedRecurrentCollector

    env, _ = make_env(B=64, n=4)
    col = FusedRecurrentCollector(env, FusedRecurrentPolicy(make_policy(env), env), 32)
    env.fuse_sampler("masked")
    with pytest.raises(RuntimeError, match="fuse_sampler"):
        col.collect()
    env.fuse_sampler(None)
