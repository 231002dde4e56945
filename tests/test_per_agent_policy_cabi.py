"""CPU-side checks of the per-agent (DTE) policies (no GPU): the C entry points exist and validate their arguments like
the shared ones before any device work; the stacked PyTorch modules convert to / from ordinary modules and compute what
agent j's module computes on agent j's rows; the fused wrappers refuse what the kernels do not implement; and the
per-agent PPO learners equal N separate learners, each with its own Adam, on the same index draws."""
import ctypes as C
from types import SimpleNamespace

import pytest
import torch

from dl_reference_models_b200 import _native as nat
from dl_reference_models_b200.policy_kernels import FusedPolicy, FusedRecurrentPolicy
from dl_reference_models_b200.recurrent import (CompactRollout, PerAgentRecurrentPolicy, RecurrentActionMaskPolicy,
                                                features_from_channels, ppo_update_recurrent)
from dl_reference_models_b200.rollout import ActionMaskPolicy, Batch, PerAgentActionMaskPolicy, gae, ppo_update

ENTRIES = [("mapf_policy_act", "mapf_policy_act_per_agent", nat.MapfPolicyArgs),
           ("mapf_lstm_policy_act", "mapf_lstm_policy_act_per_agent", nat.MapfLstmPolicyArgs)]


def test_per_agent_entry_points_are_exported():
    L = nat.lib()
    for _, name, _ in ENTRIES:
        assert hasattr(L, name) and name in nat.EXPORTS


@pytest.mark.parametrize("shared,per_agent,Args", ENTRIES)
def test_per_agent_entry_points_validate_like_the_shared_ones(shared, per_agent, Args):
    L = nat.lib()
    fs, fp = getattr(L, shared), getattr(L, per_agent)
    assert fp(None, None) == fs(None, None) == nat.ERR_INVALID_ARG
    fake = C.c_void_p(16)
    a = Args(num_envs=4, num_agents=2, v2=25, feature_dim=28)   # 28 needs blocking_prev
    assert fp(C.byref(a), None) == fs(C.byref(a), None) == nat.ERR_UNSUPPORTED
    a.feature_dim = 27
    assert fp(C.byref(a), None) == fs(C.byref(a), None) == nat.ERR_INVALID_ARG   # no channels / weights
    for k in ("local_obs", "goal_delta", "weights") + (("prev_action", "prev_reward", "h_in", "c_in")
                                                       if Args is nat.MapfLstmPolicyArgs else ()):
        setattr(a, k, fake)
    a.greedy = 2
    assert fp(C.byref(a), None) == fs(C.byref(a), None) == nat.ERR_INVALID_ARG
    assert b"greedy" in L.mapf_last_error()
    a.greedy = 0
    a.num_agents = 33
    assert fp(C.byref(a), None) == nat.ERR_UNSUPPORTED
    assert b"num_agents 33" in L.mapf_last_error()


def _mlp_modules(N, F=28, **kw):
    torch.manual_seed(1)
    return [ActionMaskPolicy(F, **kw) for _ in range(N)]


def _lstm_modules(N, F=28, **kw):
    torch.manual_seed(2)
    return [RecurrentActionMaskPolicy(F, **kw) for _ in range(N)]


@pytest.mark.parametrize("cls,make", [(PerAgentActionMaskPolicy, _mlp_modules), (PerAgentRecurrentPolicy, _lstm_modules)])
def test_from_modules_and_module_round_trip(cls, make):
    mods = make(3)
    pa = cls.from_modules(mods)
    assert pa.num_agents == 3
    for j, m in enumerate(mods):
        back = pa.module(j)
        assert type(back) is type(m)
        want, got = dict(m.named_parameters()), dict(back.named_parameters())
        assert want.keys() == got.keys()
        for k in want:
            assert torch.equal(want[k], got[k]), (j, k)
    # default init: N independently initialised modules
    d = cls(4, 28)
    assert d.num_agents == 4 and not torch.equal(d.module(0).value.weight, d.module(1).value.weight)
    with pytest.raises(ValueError, match="one shape"):
        cls.from_modules([make(1)[0], make(1, hiddens=(32, 64))[0]])


def test_per_agent_mlp_forward_equals_each_agents_module():
    N, F = 3, 28
    pa = PerAgentActionMaskPolicy.from_modules(_mlp_modules(N, F))
    x = torch.randn(5, 7, N, F)   # [T, B, N, F]
    mask = (torch.rand(5, 7, N, 5) < 0.7).to(torch.int8)
    lg, v = pa(x, mask)
    flat_lg, flat_v = pa(x.reshape(-1, F), mask.reshape(-1, 5))
    assert lg.shape == (5, 7, N, 5) and v.shape == (5, 7, N)
    assert torch.equal(flat_lg, lg.reshape(-1, 5)) and torch.equal(flat_v, v.reshape(-1))
    for j in range(N):
        lj, vj = pa.module(j)(x[:, :, j], mask[:, :, j])
        torch.testing.assert_close(lg[:, :, j], lj, atol=1e-5, rtol=0)
        torch.testing.assert_close(v[:, :, j], vj, atol=1e-5, rtol=0)


def test_per_agent_lstm_step_and_sequence_equal_each_agents_module():
    N, F, B, T = 3, 28, 6, 5
    pa = PerAgentRecurrentPolicy.from_modules(_lstm_modules(N, F))
    M = B * N
    x = torch.randn(T, M, F)
    mask = (torch.rand(T, M, 5) < 0.7).to(torch.int8)
    pact = torch.randint(0, 5, (T, M))
    prew = torch.randn(T, M)
    resets = torch.rand(T, M) < 0.2
    h0, c0 = torch.randn(M, 64) * 0.3, torch.randn(M, 64) * 0.3
    lg, v, (h, c) = pa.step(x[0], mask[0], pact[0], prew[0], (h0, c0))
    slg, sv, (sh, sc) = pa.sequence(x, mask, pact, prew, resets, (h0, c0))
    for j in range(N):
        m, r = pa.module(j), slice(j, None, N)   # agent j's rows: j, j + N, ...
        lj, vj, (hj, cj) = m.step(x[0, r], mask[0, r], pact[0, r], prew[0, r], (h0[r], c0[r]))
        for got, want in ((lg[r], lj), (v[r], vj), (h[r], hj), (c[r], cj)):
            torch.testing.assert_close(got, want, atol=1e-5, rtol=0)
        lj, vj, (hj, cj) = m.sequence(x[:, r], mask[:, r], pact[:, r], prew[:, r], resets[:, r], (h0[r], c0[r]))
        for got, want in ((slg[:, r], lj), (sv[:, r], vj), (sh[r], hj), (sc[r], cj)):
            torch.testing.assert_close(got, want, atol=1e-5, rtol=0)


def _stub_env(N=4, V=5, bp=True):
    # enough of BatchedMapfEnv for the shape checks; device work would fail on the missing attributes
    F = V * V + 2 + (1 if bp else 0)
    return SimpleNamespace(V=V, N=N, include_blocking_pressure=bp, flat_obs_dim=lambda include_action_mask=False: F)


@pytest.mark.parametrize("kwargs", [dict(hiddens=(64,)), dict(hiddens=(64, 32)), dict(num_actions=4), dict(feature_dim=27),
                                    dict(num_agents=3)])
def test_fused_policy_refuses_non_reference_per_agent_modules(kwargs):
    kw = dict(num_agents=4, feature_dim=28)
    kw.update(kwargs)
    pa = PerAgentActionMaskPolicy(**kw)
    assert not FusedPolicy.matches(pa, _stub_env())
    with pytest.raises(ValueError, match="one module per env agent"):
        FusedPolicy(pa, _stub_env())


@pytest.mark.parametrize("kwargs", [dict(hiddens=(64,)), dict(cell=32), dict(use_prev_action=False),
                                    dict(use_prev_reward=False), dict(num_actions=4), dict(feature_dim=27),
                                    dict(num_agents=5)])
def test_fused_recurrent_policy_refuses_non_reference_per_agent_modules(kwargs):
    kw = dict(num_agents=4, feature_dim=28)
    kw.update(kwargs)
    pa = PerAgentRecurrentPolicy(**kw)
    assert not FusedRecurrentPolicy.matches(pa, _stub_env())
    with pytest.raises(ValueError, match="reference's policy"):
        FusedRecurrentPolicy(pa, _stub_env())


def test_reference_per_agent_modules_match():
    assert FusedPolicy.matches(PerAgentActionMaskPolicy(4, 28), _stub_env())
    assert FusedRecurrentPolicy.matches(PerAgentRecurrentPolicy(4, 28), _stub_env())
    # a per-agent module of the other kind never matches
    assert not FusedPolicy.matches(PerAgentRecurrentPolicy(4, 28), _stub_env())
    assert not FusedRecurrentPolicy.matches(PerAgentActionMaskPolicy(4, 28), _stub_env())


def _hand_loss(lg, v, acts, old_logp, adv, ret, clip=0.05, vf_coeff=0.5, entropy_coeff=0.001):
    dist = torch.distributions.Categorical(logits=lg)
    ratio = torch.exp(dist.log_prob(acts) - old_logp)
    surr = torch.min(ratio * adv, torch.clamp(ratio, 1 - clip, 1 + clip) * adv)
    return -surr.mean() + vf_coeff * (v - ret).pow(2).mean() - entropy_coeff * dist.entropy().mean()


def _norm(a):
    return (a - a.mean()) / (a.std() + 1e-8)


def test_per_agent_ppo_update_equals_separate_learners():
    torch.manual_seed(3)
    T, B, N, F, mb, steps = 4, 8, 3, 28, 8, 3
    mask = (torch.rand(T, B, N, 5) < 0.7).to(torch.int8)
    mask[..., 0] = 1
    acts = torch.multinomial(mask.reshape(-1, 5).float(), 1).reshape(T, B, N)
    batch = Batch(torch.randn(T, B, N, F), mask, acts, -torch.rand(T, B, N) * 2, torch.randn(T, B, N),
                  torch.randn(T, B, N), torch.rand(T, B) < 0.2, torch.randn(B, N))
    mods = _mlp_modules(N, F)
    pa = PerAgentActionMaskPolicy.from_modules(mods)
    ppo_update(pa, torch.optim.Adam(pa.parameters(), lr=1e-3), batch, epochs=1, minibatch=mb, max_minibatches=steps,
               generator=torch.Generator().manual_seed(7))
    # N separate learners on the same index draws: one permutation per agent, in agent order
    adv, ret = gae(batch.rewards, batch.values, batch.dones, batch.last_value)
    gen = torch.Generator().manual_seed(7)
    perms = [torch.randperm(T * B, generator=gen) for _ in range(N)]
    opts = [torch.optim.Adam(m.parameters(), lr=1e-3) for m in mods]
    for j, (m, opt) in enumerate(zip(mods, opts)):
        col = lambda x: x[:, :, j].reshape(T * B, *x.shape[3:])  # noqa: E731
        aj = _norm(col(adv))
        for i in range(steps):
            idx = perms[j][i * mb:(i + 1) * mb]
            lg, v = m(col(batch.features)[idx], col(batch.masks)[idx])
            loss = _hand_loss(lg, v, col(batch.actions)[idx], col(batch.logp)[idx], aj[idx], col(ret)[idx])
            opt.zero_grad()
            loss.backward()
            opt.step()
    for j, m in enumerate(mods):
        for (k, want), got in zip(m.named_parameters(), pa.module(j).parameters()):
            torch.testing.assert_close(got, want, atol=1e-5, rtol=0, msg=f"agent {j} {k}")
        assert not torch.equal(want, _mlp_modules(N, F)[j].value.bias)   # the learners did move


def test_per_agent_ppo_update_recurrent_equals_separate_learners():
    torch.manual_seed(4)
    T, L, B, N, V, steps = 8, 4, 4, 3, 5, 3
    mask = (torch.rand(T, B, N, 5) < 0.7).to(torch.int8)
    mask[..., 0] = 1
    z = lambda *s: torch.randn(*s)  # noqa: E731
    batch = CompactRollout(
        torch.randint(0, 4, (T, B, N, V, V), dtype=torch.uint8), z(T, B, N, 2), torch.randint(0, 2, (T, B, N), dtype=torch.uint8),
        mask, torch.multinomial(mask.reshape(-1, 5).float(), 1).reshape(T, B, N), torch.randint(0, 5, (T, B, N)),
        z(T, B, N), torch.rand(T, B) < 0.2, -torch.rand(T, B, N) * 2, z(T, B, N), z(T, B, N), torch.rand(T, B) < 0.2,
        z(B, N), z(T // L, B * N, 64) * 0.3, z(T // L, B * N, 64) * 0.3)
    mods = _lstm_modules(N, V * V + 3)
    pa = PerAgentRecurrentPolicy.from_modules(mods)
    per_mb = 2
    ppo_update_recurrent(pa, torch.optim.Adam(pa.parameters(), lr=1e-3), batch, max_seq_len=L, minibatch=per_mb * L,
                         epochs=1, max_minibatches=steps, generator=torch.Generator().manual_seed(9))
    adv, ret = gae(batch.rewards, batch.values, batch.dones, batch.last_value)
    gen = torch.Generator().manual_seed(9)
    perms = [torch.randperm(T // L * B, generator=gen) for _ in range(N)]
    M = B * N
    sv = lambda x: x.reshape(T // L, L, M, *x.shape[3:])  # noqa: E731
    rs = batch.resets.unsqueeze(-1).expand(T, B, N)
    for j, m in enumerate(mods):
        opt = torch.optim.Adam(m.parameters(), lr=1e-3)
        aj = adv.clone()
        aj[:, :, j] = _norm(adv[:, :, j])
        for i in range(steps):
            s = perms[j][i * per_mb:(i + 1) * per_mb]
            ck, row = s // B, (s % B) * N + j
            g = lambda x: sv(x)[ck, :, row].transpose(0, 1)  # noqa: E731
            feats = features_from_channels(g(batch.local_obs), g(batch.goal_delta), g(batch.blocking_prev))
            lg, v, _ = m.sequence(feats, g(batch.masks), g(batch.prev_actions), g(batch.prev_rewards), g(rs),
                                  (batch.chunk_h[ck, row], batch.chunk_c[ck, row]))
            loss = _hand_loss(lg, v, g(batch.actions), g(batch.logp), g(aj), g(ret))
            opt.zero_grad()
            loss.backward()
            opt.step()
    for j, m in enumerate(mods):
        for (k, want), got in zip(m.named_parameters(), pa.module(j).parameters()):
            torch.testing.assert_close(got, want, atol=1e-5, rtol=0, msg=f"agent {j} {k}")
