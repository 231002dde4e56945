"""DQN on the device: mapf_q_act / mapf_q_act_per_agent against a bf16-rounding torch reference of the dueling Q and
their epsilon-greedy choice, the replay kernels against the CPU reference, DqnCollector against a manual loop of
launches, and dqn_update on a real collect against the loop written out by hand.  Tolerances as in
test_gpu_policy_kernels.py: the kernel rounds inputs, weights and hidden activations to bf16 and accumulates in f32."""
import copy
import ctypes as C
import sys
from pathlib import Path

import numpy as np
import pytest
import torch
from scipy import stats

pytestmark = pytest.mark.gpu
sys.path.insert(0, str(Path(__file__).resolve().parent))

FLOAT_MIN = -3.4e38


def make_env(sr=2, B=1003, n=16, seed=21, lifelong=True):
    from dl_reference_models_b200 import maps
    from dl_reference_models_b200.batched_env import BatchedMapfEnv

    cfg = {"num_agents": n, "sensor_range": sr, "steps_per_episode": 64, "lifelong_mapf": lifelong, "seed": seed,
           "grid": maps.random_obstacle_grid(32, 32, 0.3, 2026, min_free=2 * n)}
    env = BatchedMapfEnv(cfg, B, "cuda:0")
    out = env.reset()
    for _ in range(5):
        out = env.step(env.sample_actions(masked=True), auto_reset=True)
    return env, out


def bf16_q(policy, feats, mask):
    r = lambda t: t.to(torch.bfloat16).to(torch.float32)  # noqa: E731
    lin = [m for m in policy.trunk if isinstance(m, torch.nn.Linear)]
    h = r(feats)
    for l in lin:
        h = r(torch.relu(h @ r(l.weight).T + l.bias))
    adv = h @ r(policy.logits.weight).T + policy.logits.bias
    v = h @ r(policy.value.weight).T + policy.value.bias
    q = v + (adv - adv.mean(-1, keepdim=True))
    return torch.where(mask != 0, q, torch.full_like(q, FLOAT_MIN))


def first_argmax(q):
    return q.argmax(-1)   # torch.argmax: the first index of the largest value


@pytest.mark.parametrize("sr,n", [(1, 3), (2, 16), (3, 32)])
def test_q_act_matches_the_torch_reference_and_is_epsilon_greedy(sr, n):
    from dl_reference_models_b200.policy_kernels import FusedQPolicy
    from dl_reference_models_b200.rollout import ActionMaskPolicy

    torch.manual_seed(0)
    env, out = make_env(sr, 1003, n)
    F = env.flat_obs_dim(include_action_mask=False)
    pol = ActionMaskPolicy(F).to(env.device)
    fq = FusedQPolicy(pol, env, seed=5)
    q = torch.empty(env.B, env.N, 5, device=env.device)
    a0 = fq.act(out, 0.0, q_out=q).clone()
    with torch.no_grad():
        ref = bf16_q(pol, env.flat_obs(include_action_mask=False), out.action_mask)
    d = (q - ref).abs()
    assert float(d.max()) <= 3e-2 and float(d.mean()) <= 2e-4, (float(d.max()), float(d.mean()))
    assert torch.equal(a0.long(), first_argmax(q))
    fq.seed, fq.counter = 99, 1234
    assert torch.equal(fq.act(out, 0.0), a0)   # epsilon 0: no draw, independent of seed and counter
    legal = out.action_mask != 0
    n_legal = legal.sum(-1).double()
    # epsilon 1: uniform over the legal actions (chi^2 of the rank of the action among the legal ones, per n_legal)
    ranks = {k: [] for k in range(1, 6)}
    for _ in range(20):
        a = fq.act(out, 1.0).long()
        assert bool(legal.gather(-1, a.unsqueeze(-1)).all())
        rank = (legal.long().cumsum(-1).gather(-1, a.unsqueeze(-1)).squeeze(-1) - 1)
        for k in range(1, 6):
            ranks[k].append(rank[n_legal == k])
    for k, rs in ranks.items():   # one legal action leaves one category: its legality is checked above
        rs = torch.cat(rs)
        if k >= 2 and rs.numel() > 200 * k:
            counts = torch.bincount(rs, minlength=k).cpu().numpy()
            assert stats.chisquare(counts).pvalue > 1e-4, (k, counts)
    # epsilon 0.3: P(action != greedy) = eps (1 - 1 / n_legal)
    diff, expect = 0, 0.0
    for _ in range(10):
        a = fq.act(out, 0.3)
        assert bool(legal.gather(-1, a.long().unsqueeze(-1)).all())
        diff += int((a != a0).sum())
        expect += float((0.3 * (1 - 1 / n_legal)).sum())
    trials = 10 * env.B * env.N
    assert stats.binomtest(diff, trials, expect / trials).pvalue > 1e-4


def test_q_act_shards_and_per_agent_blocks():
    from dl_reference_models_b200 import _native as nat
    from dl_reference_models_b200.policy_kernels import FusedQPolicy
    from dl_reference_models_b200.rollout import PerAgentActionMaskPolicy

    torch.manual_seed(1)
    env, out = make_env(2, 1003, 16)
    F = env.flat_obs_dim(include_action_mask=False)
    pa = PerAgentActionMaskPolicy(16, F).to(env.device)
    fp = FusedQPolicy(pa, env, seed=3)
    assert fp.entry == "mapf_q_act_per_agent"
    q = torch.empty(env.B, env.N, 5, device=env.device)
    fp.counter = 6
    a = fp.act(out, 0.4, q_out=q).clone()
    ch = {k: getattr(out, k) for k in ("local_obs", "goal_delta", "blocking_prev", "action_mask")}
    for j in (0, 7, 15):   # agent j = the shared launch with block j
        fj = FusedQPolicy(pa.module(j), env, seed=3)
        qj = torch.empty_like(q)
        fj.counter = 6
        aj = fj.act(out, 0.4, q_out=qj)
        assert torch.equal(aj[:, j], a[:, j]) and torch.equal(qj[:, j], q[:, j])
    # a shard with its env_id_base equals the full launch
    lo = 500
    fs = FusedQPolicy(pa.module(0), env, seed=3)
    full = torch.empty(env.B, env.N, dtype=torch.int8, device=env.device)
    args = fs.args(ch, 0.5, full)
    args.counter = 17
    nat.check(nat.lib().mapf_q_act(C.byref(args), None))
    part = torch.zeros_like(full)
    sub = {k: v[lo:].contiguous() for k, v in ch.items()}
    a2 = fs.args(sub, 0.5, part[lo:])
    a2.num_envs, a2.env_id_base, a2.counter = env.B - lo, lo, 17
    nat.check(nat.lib().mapf_q_act(C.byref(a2), None))
    torch.cuda.synchronize()
    assert torch.equal(part[lo:], full[lo:])


def _cpu_twin(buf):
    """A CPU buffer with the same leaves and max priority."""
    from types import SimpleNamespace

    from dl_reference_models_b200 import dqn

    env = SimpleNamespace(B=buf.B, N=buf.N, V=buf.env.V, device="cpu", include_blocking_pressure=buf.with_bp,
                          out={k: v[0].cpu() for k, v in buf.rows.items()})
    c = dqn.ReplayBuffer(env, buf.K, alpha=buf.alpha, per_agent=buf.per_agent)
    c.leaves().copy_(buf.leaves().cpu())
    c.max_priority.copy_(buf.max_priority.cpu())
    c.filled = buf.filled
    return c


def _tree_reference(leaves_padded):
    """Sums (f64) and minimums (f32) of every internal node, level by level."""
    L = leaves_padded.numel()
    sums, mins = torch.zeros(L, dtype=torch.float64), torch.full((L,), float("inf"))
    s, m = leaves_padded.double(), torch.where(leaves_padded > 0, leaves_padded, torch.full_like(leaves_padded, float("inf")))
    n = L
    while n > 1:
        s, m = s.view(-1, 2).sum(1), m.view(-1, 2).min(1).values
        n //= 2
        sums[n:2 * n], mins[n:2 * n] = s, m
    return sums, mins


@pytest.mark.parametrize("per_agent", [False, True])
def test_tree_kernels_equal_the_cpu_reference(per_agent):
    from dl_reference_models_b200 import dqn

    env, _ = make_env(2, 1003, 3)
    buf = dqn.ReplayBuffer(env, 6, alpha=1.0, per_agent=per_agent)
    for t in range(9):   # across the wrap-around
        buf.max_priority.fill_(float(t % 4 + 1))
        buf.advance(t % 6, (t + 1) % 6)
    buf.filled = 5
    cpu = dqn.ReplayBuffer(_cpu_twin(buf).env, 6, alpha=1.0, per_agent=per_agent)
    cpu.max_priority.fill_(1.0)
    for t in range(9):
        cpu.max_priority.fill_(float(t % 4 + 1))
        cpu.advance(t % 6, (t + 1) % 6)
    cpu.filled = 5
    torch.testing.assert_close(buf.leaves().cpu(), cpu.leaves(), rtol=0, atol=0)
    # integer-valued priorities with duplicates and out-of-range indices
    g = torch.Generator().manual_seed(0)
    idx = torch.randint(-50, 6 * 1003 * 3 + 50, (3000,), generator=g)
    idx[1000:1100] = idx[:100]
    td = torch.randint(1, 20, (3000,), generator=g).float()
    td[1000:1100] = td[:100]
    buf.update_priorities(idx.cuda(), td.cuda())
    cpu.update_priorities(idx, td)
    torch.testing.assert_close(buf.leaves().cpu(), cpu.leaves(), rtol=0, atol=0)
    assert float(buf.max_priority) == float(cpu.max_priority)
    sums, mins = _tree_reference(buf._leaves.cpu())
    assert torch.equal(buf.sums.cpu()[1:], sums[1:]) and torch.equal(buf.mins.cpu()[1:], mins[1:])
    u = torch.empty(20000, dtype=torch.float64, device="cuda")
    idx_k, w_k = buf.sample(20000, 0.4, uniforms_out=u)
    idx_c, w_c = cpu.sample(20000, 0.4, uniforms=u.cpu())
    assert torch.equal(idx_k.cpu(), idx_c)
    np.testing.assert_allclose(w_k.cpu().numpy(), w_c.numpy(), rtol=1e-6)


def test_sampling_chi2_at_2_20_leaves():
    from dl_reference_models_b200 import dqn

    env, _ = make_env(1, 16384, 16)
    buf = dqn.ReplayBuffer(env, 4, alpha=1.0)
    assert buf._leaves.numel() == 1 << 20
    for t in range(3):
        buf.advance(t, t + 1)   # slot 3 stays empty: its leaves and the padding are 0
    buf.filled = 3
    n = 3 * 16384 * 16
    g = torch.Generator(device="cuda").manual_seed(0)
    p = torch.randint(1, 4, (n,), device="cuda", generator=g).float()
    buf.update_priorities(torch.arange(n, device="cuda"), p - 1e-6)
    idx, _ = buf.sample(1 << 22, 0.4)
    assert bool((idx >= 0).all() and (idx < n).all())   # never a slot without a transition
    counts = torch.bincount(idx, minlength=n).double()
    obs = torch.stack([counts[p == v].sum() for v in (1.0, 2.0, 3.0)]).cpu().numpy()
    exp = torch.stack([p[p == v].double().sum() for v in (1.0, 2.0, 3.0)]).cpu().numpy()
    assert stats.chisquare(obs, exp / exp.sum() * obs.sum()).pvalue > 1e-4
    per_cell = stats.chisquare(counts.cpu().numpy(), (p.double() / p.double().sum() * (1 << 22)).cpu().numpy())
    assert per_cell.pvalue > 1e-4


def test_collector_equals_a_manual_loop_and_the_learner_the_loop_by_hand():
    import test_dqn_cabi as cabi

    from dl_reference_models_b200 import _native as nat
    from dl_reference_models_b200 import dqn
    from dl_reference_models_b200.policy_kernels import FusedQPolicy
    from dl_reference_models_b200.rollout import ActionMaskPolicy

    torch.manual_seed(0)
    env, _ = make_env(2, 1003, 4, seed=5, lifelong=False)
    twin, _ = make_env(2, 1003, 4, seed=5, lifelong=False)
    F = env.flat_obs_dim(include_action_mask=False)
    pol = ActionMaskPolicy(F).to(env.device)
    K = 6
    buf = dqn.ReplayBuffer(env, K, alpha=0.6)
    dc = dqn.DqnCollector(env, FusedQPolicy(pol, env, seed=9), buf)
    dc.collect(4, 0.3)
    dc.collect(5, 0.3)   # 9 steps > K: the ring wraps
    # the manual loop: q_act on the env's own buffers, mapf_step, the tree advanced through the buffer
    ref = dqn.ReplayBuffer(twin, K, alpha=0.6)
    fq = FusedQPolicy(pol, twin, seed=9)
    obs = {k: [] for k in ("local_obs", "goal_delta", "blocking_prev", "action_mask")}
    acts, rews, dones = [], [], []
    for t in range(9):
        for k in obs:
            obs[k].append(twin.out[k].clone())
        a = fq.act(twin._output(), 0.3).clone()
        o = twin.step(a, auto_reset=True)
        acts.append(a)
        rews.append(o.reward.clone())
        dones.append(o.terminated.clone())
        ref.advance(t % K, (t + 1) % K)
    for k in obs:
        obs[k].append(twin.out[k].clone())
    torch.cuda.synchronize()
    for t in range(9 - K + 1, 10):   # the rows the ring still holds
        for k in obs:
            assert torch.equal(buf.rows[k][t % K], obs[k][t]), (k, t)
    for t in range(9 - K + 1, 9):
        assert torch.equal(buf.actions[t % K], acts[t]) and torch.equal(buf.rewards[t % K], rews[t])
        assert torch.equal(buf.dones[t % K], dones[t])
    assert torch.equal(buf.leaves(), ref.leaves())
    assert buf.head == 9 % K and buf.num_transitions == (K - 1) * 1003 * 4
    for k in ("local_obs", "goal_delta", "action_mask"):
        assert torch.equal(env.out[k], twin.out[k])
    assert torch.equal(env.state["positions"], twin.state["positions"])
    # the learner on this collect against the loop by hand, given the same draws
    target = copy.deepcopy(pol)
    ref_pol, ref_t = copy.deepcopy(pol), copy.deepcopy(pol)
    opt, ropt = torch.optim.Adam(pol.parameters(), lr=1e-3), torch.optim.Adam(ref_pol.parameters(), lr=1e-3)
    draws = cabi._recording(buf)
    dqn.dqn_update(pol, target, opt, buf, updates=2, minibatch=256, grad_clip=0.5)
    for idx, w in draws:   # the ring's rows are what they were: the learner writes priorities only
        _hand(ref_pol, ref_t, ropt, buf, idx, w)
    for p, q in zip(pol.parameters(), ref_pol.parameters()):
        torch.testing.assert_close(p, q, rtol=1e-4, atol=1e-4)
    dc.fused.refresh()
    dc.collect(3, 0.1)
    assert buf.head == 12 % K


def _hand(pol, target, opt, buf, idx, w):
    BN = buf.B * buf.N
    k, r = idx // BN, idx % BN
    kn = (k + 1) % buf.K
    V2 = buf.env.V ** 2

    def feats(kk):
        return torch.cat([buf.rows["local_obs"].view(buf.K, BN, V2)[kk, r].float(), buf.rows["goal_delta"].view(buf.K, BN, 2)[kk, r],
                          buf.rows["blocking_prev"].view(buf.K, BN)[kk, r].float().unsqueeze(-1)], -1)

    def q(m, kk):
        adv, v = m.heads(feats(kk))
        qq = v.unsqueeze(-1) + adv - adv.mean(-1, keepdim=True)
        return torch.where(buf.rows["action_mask"].view(buf.K, BN, 5)[kk, r] != 0, qq, torch.full_like(qq, FLOAT_MIN))

    q_sa = q(pol, k).gather(1, buf.actions.view(buf.K, BN)[k, r].long()[:, None])[:, 0]
    with torch.no_grad():
        nxt = q(target, kn).gather(1, q(pol, kn).argmax(1, keepdim=True))[:, 0]
        y = buf.rewards.view(buf.K, BN)[k, r] + 0.99 * (1 - buf.dones[k, r // buf.N].float()) * nxt
    x = q_sa - y
    loss = (w * torch.where(x.abs() < 1, 0.5 * x * x, x.abs() - 0.5)).mean()
    opt.zero_grad()
    loss.backward()
    torch.nn.utils.clip_grad_norm_(pol.parameters(), 0.5)
    opt.step()
    return x.detach().abs()
