"""CPU-side checks of DQN (no GPU): the new structs' ctypes layouts against the header, the exports, every refusal
before any device work, q_values against a loop written out by hand, the modules' forward unchanged, the CPU replay
reference (distribution, zero leaves, weights, per-agent draws, priority updates), dqn_update against a loop written
out by hand, the per-agent learner against N separate modules, and two gloo ranks stepping with the mean gradient."""
import copy
import ctypes as C
import math
import os
import shutil
import socket
import subprocess
import sys
from pathlib import Path
from types import SimpleNamespace

import numpy as np
import pytest
import torch
from scipy import stats

from dl_reference_models_b200 import _native as nat
from dl_reference_models_b200 import dqn
from dl_reference_models_b200.rollout import FLOAT_MIN, ActionMaskPolicy, PerAgentActionMaskPolicy

REPO = Path(__file__).resolve().parents[1]
STRUCTS = {"mapf_q_act_args": nat.MapfQActArgs, "mapf_replay_tree": nat.MapfReplayTree,
           "mapf_replay_advance_args": nat.MapfReplayAdvanceArgs, "mapf_replay_sample_args": nat.MapfReplaySampleArgs,
           "mapf_replay_update_args": nat.MapfReplayUpdateArgs}


@pytest.mark.skipif(shutil.which("gcc") is None, reason="needs gcc")
@pytest.mark.parametrize("name", list(STRUCTS))
def test_ctypes_structure_matches_the_header_layout(tmp_path, name):
    cls = STRUCTS[name]
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


def test_exports():
    L = nat.lib()
    for name in ("mapf_q_act", "mapf_q_act_per_agent", "mapf_replay_tree_leaves", "mapf_replay_advance",
                 "mapf_replay_sample", "mapf_replay_update"):
        assert name in nat.EXPORTS and hasattr(L, name)
    assert L.mapf_replay_tree_leaves(65536, 16, 64) == 1 << 26
    assert L.mapf_replay_tree_leaves(1003, 3, 5) == 1024 * 4 * 8
    assert L.mapf_replay_tree_leaves(4, 2, 1) == nat.ERR_INVALID_ARG


FAKE = C.c_void_p(16)


def _q(**kw):
    a = nat.MapfQActArgs(num_envs=4, num_agents=3, v2=25, feature_dim=28, epsilon=0.1, local_obs=FAKE, goal_delta=FAKE,
                         blocking_prev=FAKE, action_mask=FAKE, weights=FAKE, actions=FAKE)
    for k, v in kw.items():
        setattr(a, k, v)
    return a


Q_INVALID = ([{k: None} for k in ("local_obs", "goal_delta", "action_mask", "weights", "actions")]
             + [{"num_envs": 0}, {"num_agents": 0}, {"epsilon": -0.01}, {"epsilon": 1.01}, {"epsilon": math.nan},
                {"reserved": 1}])
Q_UNSUPPORTED = [{"feature_dim": 27}, {"feature_dim": 70, "v2": 67}, {"blocking_prev": None}]


@pytest.mark.parametrize("per_agent", [False, True])
@pytest.mark.parametrize("kw", Q_INVALID + Q_UNSUPPORTED, ids=[str(k) for k in Q_INVALID + Q_UNSUPPORTED])
def test_q_act_refuses_before_any_device_work(kw, per_agent):
    L = nat.lib()
    fn = L.mapf_q_act_per_agent if per_agent else L.mapf_q_act
    want = nat.ERR_INVALID_ARG if kw in Q_INVALID else nat.ERR_UNSUPPORTED
    assert fn(C.byref(_q(**kw)), None) == want
    assert b"q_act" in L.mapf_last_error()
    assert fn(None, None) == nat.ERR_INVALID_ARG


def test_q_act_per_agent_refuses_more_than_32_agents():
    assert nat.lib().mapf_q_act_per_agent(C.byref(_q(num_agents=33)), None) == nat.ERR_UNSUPPORTED


def _tree(**kw):
    t = nat.MapfReplayTree(num_envs=5, num_agents=3, capacity=4, leaves=FAKE, sums=FAKE, mins=FAKE, max_priority=FAKE)
    for k, v in kw.items():
        setattr(t, k, v)
    return t


TREE_BAD = ([{k: None} for k in ("leaves", "sums", "mins", "max_priority")]
            + [{"num_envs": 0}, {"num_agents": 0}, {"capacity": 1}])
ADV_BAD = ([{"tree": t} for t in TREE_BAD] + [{"complete": 4}, {"complete": -1}, {"clear": 4}, {"complete": 2, "clear": 2},
           {"alpha": -0.1}, {"alpha": math.inf}, {"alpha": math.nan}, {"reserved": 1}])
SAMPLE_BAD = ([{"tree": t} for t in TREE_BAD] + [{"indices": None}, {"weights": None}, {"M": 0}, {"beta": -1.0},
              {"beta": math.nan}, {"per_agent": 2}, {"reserved": 1}])
UPDATE_BAD = ([{"tree": t} for t in TREE_BAD] + [{"indices": None}, {"td_abs": None}, {"M": 0}, {"M": -3},
              {"alpha": -1.0}, {"alpha": math.inf}, {"reserved": 1}])


def _with(a, kw):
    for k, v in kw.items():
        if k == "tree":
            v = _tree(**v)
        setattr(a, k, v)
    return a


@pytest.mark.parametrize("kw", ADV_BAD, ids=[str(k) for k in ADV_BAD])
def test_replay_advance_refuses(kw):
    L = nat.lib()
    a = _with(nat.MapfReplayAdvanceArgs(tree=_tree(), complete=1, clear=2, alpha=0.6), kw)
    assert L.mapf_replay_advance(C.byref(a), None) == nat.ERR_INVALID_ARG
    assert b"replay" in L.mapf_last_error()
    assert L.mapf_replay_advance(None, None) == nat.ERR_INVALID_ARG


@pytest.mark.parametrize("kw", SAMPLE_BAD, ids=[str(k) for k in SAMPLE_BAD])
def test_replay_sample_refuses(kw):
    L = nat.lib()
    a = _with(nat.MapfReplaySampleArgs(tree=_tree(), M=8, beta=0.4, indices=FAKE, weights=FAKE), kw)
    assert L.mapf_replay_sample(C.byref(a), None) == nat.ERR_INVALID_ARG
    assert b"replay" in L.mapf_last_error()
    assert L.mapf_replay_sample(None, None) == nat.ERR_INVALID_ARG


@pytest.mark.parametrize("kw", UPDATE_BAD, ids=[str(k) for k in UPDATE_BAD])
def test_replay_update_refuses(kw):
    L = nat.lib()
    a = _with(nat.MapfReplayUpdateArgs(tree=_tree(), M=8, indices=FAKE, td_abs=FAKE, alpha=0.6), kw)
    assert L.mapf_replay_update(C.byref(a), None) == nat.ERR_INVALID_ARG
    assert b"replay" in L.mapf_last_error()
    assert L.mapf_replay_update(None, None) == nat.ERR_INVALID_ARG


# ---- q_values and the modules ---------------------------------------------------------------------------------------

F_ = 12


def _q_loop(adv, v, mask, no_masking):
    out = torch.empty_like(adv)
    for r in range(adv.shape[0]):
        m = sum(float(adv[r, k]) for k in range(5)) / 5
        for k in range(5):
            q = float(v[r]) + (float(adv[r, k]) - m)
            out[r, k] = q if (no_masking or mask[r, k]) else FLOAT_MIN
    return out


@pytest.mark.parametrize("per_agent", [False, True])
@pytest.mark.parametrize("no_masking", [False, True])
def test_q_values_equals_a_loop_by_hand(per_agent, no_masking):
    torch.manual_seed(0)
    pol = PerAgentActionMaskPolicy(3, F_, no_masking=no_masking) if per_agent else ActionMaskPolicy(F_, no_masking=no_masking)
    x = torch.randn(12, F_)
    mask = (torch.rand(12, 5) < 0.6).to(torch.int8)
    mask[:, 0] = 1
    q = dqn.q_values(pol, x, mask)
    with torch.no_grad():
        if per_agent:
            adv = torch.empty(12, 5)
            v = torch.empty(12)
            for j in range(3):
                m = pol.module(j)
                z = m.trunk(x[j::3])
                adv[j::3], v[j::3] = m.logits(z), m.value(z).squeeze(-1)
        else:
            z = pol.trunk(x)
            adv, v = pol.logits(z), pol.value(z).squeeze(-1)
    torch.testing.assert_close(q.detach(), _q_loop(adv, v, mask, no_masking), rtol=1e-5, atol=1e-5)
    if not no_masking:
        assert bool((q[mask == 0] == FLOAT_MIN).all())


@pytest.mark.parametrize("per_agent", [False, True])
def test_forward_is_unchanged_bit_for_bit(per_agent):
    torch.manual_seed(1)
    pol = PerAgentActionMaskPolicy(4, F_) if per_agent else ActionMaskPolicy(F_)
    x = torch.randn(16, F_)
    mask = (torch.rand(16, 5) < 0.5).to(torch.int8)
    lg, v = pol(x, mask)
    # the forward as it was written before heads() existed
    if per_agent:
        from dl_reference_models_b200.rollout import agent_linear
        z = x.float().reshape(-1, 4, F_).transpose(0, 1)
        for w, b in zip(pol.trunk_w, pol.trunk_b):
            z = torch.relu(agent_linear(z, w, b))
        logits = agent_linear(z, pol.logits_w, pol.logits_b).transpose(0, 1).reshape(16, -1)
        value = agent_linear(z, pol.value_w, pol.value_b).transpose(0, 1).reshape(16)
    else:
        z = pol.trunk(x.float())
        logits, value = pol.logits(z), pol.value(z).squeeze(-1)
    logits = logits + torch.clamp(torch.log(mask.to(logits.dtype) + 1e-6), min=FLOAT_MIN)
    assert torch.equal(lg, logits) and torch.equal(v, value)


# ---- the CPU replay reference ---------------------------------------------------------------------------------------

V = 2


def fake_env(B, N, g):
    out = {"local_obs": torch.zeros(B, N, V, V, dtype=torch.uint8), "goal_delta": torch.zeros(B, N, 2),
           "blocking_prev": torch.zeros(B, N, dtype=torch.uint8), "action_mask": torch.zeros(B, N, 5, dtype=torch.int8)}
    return SimpleNamespace(B=B, N=N, V=V, device="cpu", include_blocking_pressure=True, out=out)


def filled_buffer(B, N, K, g, alpha=0.6, per_agent=False, slots=None):
    """A CPU buffer with every ring row filled at random and ``slots`` (default all but one) complete."""
    buf = dqn.ReplayBuffer(fake_env(B, N, g), K, alpha=alpha, per_agent=per_agent)
    r = buf.rows
    r["local_obs"].copy_(torch.randint(0, 3, r["local_obs"].shape, generator=g, dtype=torch.uint8))
    r["goal_delta"].copy_(torch.randn(r["goal_delta"].shape, generator=g))
    r["blocking_prev"].copy_(torch.randint(0, 2, r["blocking_prev"].shape, generator=g, dtype=torch.uint8))
    m = (torch.rand(r["action_mask"].shape, generator=g) < 0.7).to(torch.int8)
    m[..., 0] = 1
    buf.actions.copy_(torch.randint(0, 5, buf.actions.shape, generator=g, dtype=torch.int8))
    m.scatter_(-1, buf.actions.long().unsqueeze(-1), 1)   # the taken action is legal
    r["action_mask"].copy_(m)
    buf.rewards.copy_(torch.randn(buf.rewards.shape, generator=g))
    buf.dones.copy_((torch.rand(buf.dones.shape, generator=g) < 0.2).to(torch.uint8))
    slots = list(range(K - 1)) if slots is None else slots
    for k in slots:
        buf.advance(k, (k + 1) % K)
    buf.filled = len(slots)
    return buf


def test_sampling_distribution_chi2_and_zero_leaves_never_drawn():
    g = torch.Generator().manual_seed(0)
    buf = filled_buffer(5, 3, 4, g, alpha=1.0)
    leaves = buf.leaves()
    leaves[:, :3] = torch.randint(0, 5, (3, 3, 5), generator=g).float()   # zeros among them
    idx, w = buf.sample(200000, 0.4, generator=g)
    k, b, j = idx // 15, idx % 15 // 3, idx % 3
    assert bool((leaves[j, k, b] > 0).all())
    counts = torch.bincount(((j * 4 + k) * 5 + b), minlength=60).double()
    p = leaves.reshape(-1).double()
    nz = p > 0
    chi = stats.chisquare(counts[nz].numpy(), (p[nz] / p.sum() * 200000).numpy())
    assert chi.pvalue > 1e-4
    assert int(counts[~nz].sum()) == 0


def test_weights_follow_the_formula():
    g = torch.Generator().manual_seed(1)
    buf = filled_buffer(5, 3, 4, g, alpha=0.6)
    buf.update_priorities(torch.arange(45), torch.rand(45, generator=g) * 3)
    idx, w = buf.sample(500, 0.4, generator=g)
    leaves = buf.leaves().double()
    k, b, j = idx // 15, idx % 15 // 3, idx % 3
    p = leaves[j, k, b]
    total, n = leaves.sum(), int((leaves > 0).sum())
    p_min = leaves[leaves > 0].min()
    want = (p / total * n) ** -0.4 / ((p_min / total) * n) ** -0.4
    np.testing.assert_allclose(w.double().numpy(), want.numpy(), rtol=1e-6)


def test_per_agent_draws_come_from_agent_i_mod_n():
    g = torch.Generator().manual_seed(2)
    buf = filled_buffer(6, 4, 5, g, alpha=0.6, per_agent=True)
    buf.update_priorities(torch.arange(4 * 6 * 4), torch.rand(96, generator=g))
    idx, w = buf.sample(400, 0.5, generator=g)
    assert bool((idx % 4 == torch.arange(400) % 4).all())
    leaves = buf.leaves().double()
    k, b, j = idx // 24, idx % 24 // 4, idx % 4
    p_min = torch.stack([leaves[a][leaves[a] > 0].min() for a in range(4)])
    np.testing.assert_allclose(w.double().numpy(), ((leaves[j, k, b] / p_min[j]) ** -0.5).numpy(), rtol=1e-6)


def test_update_and_max_priority():
    g = torch.Generator().manual_seed(3)
    buf = filled_buffer(4, 2, 4, g, alpha=0.5, slots=[0, 1])
    BN = 8
    before = buf.leaves().clone()
    idx = torch.tensor([1, 1, 9, 2 * BN + 3, 4 * BN, -1, 5])   # a duplicate, a cleared slot, out of range
    td = torch.tensor([0.5, 2.0, 3.0, 7.0, 9.0, 9.0, 1.5])
    buf.update_priorities(idx, td)
    want = before.clone()
    want[1, 0, 0] = (2.0 + 1e-6) ** 0.5   # the larger duplicate
    want[1, 1, 0] = (3.0 + 1e-6) ** 0.5
    want[1, 0, 2] = (1.5 + 1e-6) ** 0.5
    torch.testing.assert_close(buf.leaves(), want)
    assert float(buf.max_priority) == pytest.approx(3.0 + 1e-6)
    buf.advance(2, 3)
    torch.testing.assert_close(buf.leaves()[:, 2], torch.full((2, 4), (3.0 + 1e-6) ** 0.5))


# ---- the learner ----------------------------------------------------------------------------------------------------

def _huber(x):
    return torch.where(x.abs() < 1, 0.5 * x * x, x.abs() - 0.5)


def hand_update(pol, target, opt, buf, idx, w, *, gamma, double_q, clip, per_agent, N):
    """One DQN step written out, on the given draws."""
    BN = buf.B * buf.N
    k, r = idx // BN, idx % BN
    kn = (k + 1) % buf.K
    V2 = V * V

    def feats(kk):
        return torch.cat([buf.rows["local_obs"].view(buf.K, BN, V2)[kk, r].float(), buf.rows["goal_delta"].view(buf.K, BN, 2)[kk, r],
                          buf.rows["blocking_prev"].view(buf.K, BN)[kk, r].float().unsqueeze(-1)], -1)

    def q(m, kk):
        adv, v = m.heads(feats(kk))
        qq = v.unsqueeze(-1) + adv - adv.mean(-1, keepdim=True)
        mask = buf.rows["action_mask"].view(buf.K, BN, 5)[kk, r]
        return torch.where(mask != 0, qq, torch.full_like(qq, FLOAT_MIN))

    a = buf.actions.view(buf.K, BN)[k, r].long()
    rew = buf.rewards.view(buf.K, BN)[k, r]
    d = buf.dones[k, r // buf.N].float()
    q_sa = q(pol, k).gather(1, a[:, None])[:, 0]
    with torch.no_grad():
        qt = q(target, kn)
        nxt = qt.gather(1, q(pol, kn).argmax(1, keepdim=True))[:, 0] if double_q else qt.max(1).values
        y = rew + gamma * (1 - d) * nxt
    loss_el = w * _huber(q_sa - y)
    loss = loss_el.reshape(-1, N).mean(0).sum() if per_agent else loss_el.mean()
    opt.zero_grad()
    loss.backward()
    torch.nn.utils.clip_grad_norm_(pol.parameters(), clip)
    opt.step()
    return (q_sa - y).detach().abs()


def _recording(buf):
    draws = []
    orig = buf.sample

    def rec(*a, **k):
        out = orig(*a, **k)
        draws.append(out)
        return out
    buf.sample = rec
    return draws


@pytest.mark.parametrize("double_q", [True, False])
def test_dqn_update_equals_the_loop_by_hand(double_q):
    g = torch.Generator().manual_seed(4)
    buf = filled_buffer(6, 3, 5, g)
    ref_buf = copy.deepcopy(buf)
    torch.manual_seed(0)
    F = V * V + 3
    pol, target = ActionMaskPolicy(F), ActionMaskPolicy(F)
    ref, ref_t = copy.deepcopy(pol), copy.deepcopy(target)
    opt, ropt = torch.optim.Adam(pol.parameters(), lr=1e-2), torch.optim.Adam(ref.parameters(), lr=1e-2)
    draws = _recording(buf)
    st = dqn.dqn_update(pol, target, opt, buf, updates=3, minibatch=16, gamma=0.9, beta=0.5, double_q=double_q,
                        grad_clip=0.3, generator=torch.Generator().manual_seed(8))
    assert set(st) == {"loss", "mean_q", "mean_td_abs"} and all(math.isfinite(x) for x in st.values())
    for idx, w in draws:
        td = hand_update(ref, ref_t, ropt, ref_buf, idx, w, gamma=0.9, double_q=double_q, clip=0.3, per_agent=False, N=3)
        ref_buf.update_priorities(idx, td)
    for p, q in zip(pol.parameters(), ref.parameters()):
        torch.testing.assert_close(p, q, rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(buf.leaves(), ref_buf.leaves(), rtol=1e-5, atol=1e-6)


def test_dqn_update_refusals():
    g = torch.Generator().manual_seed(5)
    F = V * V + 3
    empty = dqn.ReplayBuffer(fake_env(4, 2, g), 4)
    pol = ActionMaskPolicy(F)
    with pytest.raises(ValueError):
        dqn.dqn_update(pol, copy.deepcopy(pol), torch.optim.Adam(pol.parameters()), empty)
    buf = filled_buffer(4, 2, 4, g, per_agent=True)
    pa = PerAgentActionMaskPolicy(3, F)
    with pytest.raises(ValueError):
        dqn.dqn_update(pa, copy.deepcopy(pa), torch.optim.Adam(pa.parameters()), buf)
    buf.rewards[0, 0, 0] = math.nan
    buf.leaves().zero_()
    buf.leaves()[0, 0, 0] = 1.0   # every draw is the NaN-reward transition
    pol2 = PerAgentActionMaskPolicy(2, F)
    before = [p.detach().clone() for p in pol2.parameters()]
    with pytest.raises(FloatingPointError):
        dqn.dqn_update(pol2, copy.deepcopy(pol2), torch.optim.Adam(pol2.parameters()), buf, minibatch=4)
    assert all(torch.equal(p, q) for p, q in zip(pol2.parameters(), before))
    assert float(buf.leaves()[0, 0, 0]) == 1.0


def test_per_agent_learner_equals_n_separate_modules():
    N = 3
    g = torch.Generator().manual_seed(6)
    buf = filled_buffer(8, N, 5, g, per_agent=True)
    buf.rewards.mul_(torch.tensor([0.01, 1.0, 100.0]))   # agent 0 under the clip, agent 2 far over it
    ref_buf = copy.deepcopy(buf)
    F = V * V + 3
    torch.manual_seed(0)
    pol, target = PerAgentActionMaskPolicy(N, F), PerAgentActionMaskPolicy(N, F)
    mods, tmods = [pol.module(j) for j in range(N)], [target.module(j) for j in range(N)]
    opts = [torch.optim.Adam(m.parameters(), lr=1e-2) for m in mods]
    draws = _recording(buf)
    dqn.dqn_update(pol, target, torch.optim.Adam(pol.parameters(), lr=1e-2), buf, updates=2, minibatch=8, grad_clip=1.0,
                   generator=torch.Generator().manual_seed(2))
    norms = []
    for idx, w in draws:
        assert bool((idx % N == torch.arange(idx.numel()) % N).all())
        tds = torch.empty(idx.numel())
        for j in range(N):
            sel = torch.arange(j, idx.numel(), N)
            BN = buf.B * buf.N
            k, r = idx[sel] // BN, idx[sel] % BN
            kn = (k + 1) % buf.K

            def feats(kk):
                return torch.cat([ref_buf.rows["local_obs"].view(buf.K, BN, 4)[kk, r].float(),
                                  ref_buf.rows["goal_delta"].view(buf.K, BN, 2)[kk, r],
                                  ref_buf.rows["blocking_prev"].view(buf.K, BN)[kk, r].float().unsqueeze(-1)], -1)

            def masks(kk):
                return ref_buf.rows["action_mask"].view(buf.K, BN, 5)[kk, r]
            q_sa = dqn.q_values(mods[j], feats(k), masks(k)).gather(1, ref_buf.actions.view(buf.K, BN)[k, r].long()[:, None])[:, 0]
            with torch.no_grad():
                a2 = dqn.q_values(mods[j], feats(kn), masks(kn)).argmax(1, keepdim=True)
                y = (ref_buf.rewards.view(buf.K, BN)[k, r] + 0.99 * (1 - ref_buf.dones[k, r // N].float())
                     * dqn.q_values(tmods[j], feats(kn), masks(kn)).gather(1, a2)[:, 0])
            loss = (w[sel] * _huber(q_sa - y)).mean()
            opts[j].zero_grad()
            loss.backward()
            norms.append(float(torch.nn.utils.clip_grad_norm_(mods[j].parameters(), 1.0)))
            opts[j].step()
            tds[sel] = (q_sa - y).detach().abs()
        ref_buf.update_priorities(idx, tds)
    assert min(norms) < 1.0 < max(norms), norms
    for j, m in enumerate(mods):
        for p, q in zip(pol.module(j).parameters(), m.parameters()):
            torch.testing.assert_close(p, q, rtol=1e-5, atol=1e-5)


def _rank_worker(rank, world, port, q):
    import torch.distributed as dist

    sys.path.insert(0, str(REPO))
    sys.path.insert(0, str(REPO / "tests"))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from test_dqn_cabi import filled_buffer as fb
        torch.manual_seed(0)
        pol = ActionMaskPolicy(V * V + 3)
        buf = fb(6, 3, 5, torch.Generator().manual_seed(100 + rank))
        dqn.dqn_update(pol, copy.deepcopy(pol), torch.optim.Adam(pol.parameters(), lr=1e-2), buf, minibatch=16,
                       grad_clip=0.05, world_size=world, generator=torch.Generator().manual_seed(3 + rank))
        q.put((rank, [p.detach().numpy().copy() for p in pol.parameters()]))
    finally:
        dist.destroy_process_group()


def test_two_gloo_ranks_step_with_the_clipped_mean_gradient():
    import torch.multiprocessing as mp

    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_rank_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    try:
        res = dict(q.get(timeout=180) for _ in procs)
    finally:
        for p in procs:
            p.join(timeout=60)
            if p.is_alive():
                p.kill()
                p.join()
    assert [p.exitcode for p in procs] == [0, 0]
    torch.manual_seed(0)
    pol = ActionMaskPolicy(V * V + 3)
    grads = []
    for rank in range(2):
        m, t = copy.deepcopy(pol), copy.deepcopy(pol)
        buf = filled_buffer(6, 3, 5, torch.Generator().manual_seed(100 + rank))
        idx, w = buf.sample(16, 0.4, generator=torch.Generator().manual_seed(3 + rank))
        o = torch.optim.SGD(m.parameters(), lr=0.0)
        hand_update(m, t, o, buf, idx, w, gamma=0.99, double_q=True, clip=math.inf, per_agent=False, N=3)
        grads.append([p.grad for p in m.parameters()])
    for p, g0, g1 in zip(pol.parameters(), *grads):
        p.grad = (g0 + g1) / 2
    assert float(torch.nn.utils.clip_grad_norm_(pol.parameters(), 0.05)) > 0.05
    torch.optim.Adam(pol.parameters(), lr=1e-2).step()
    for rank in range(2):
        for p, q_ in zip(pol.parameters(), res[rank]):
            torch.testing.assert_close(torch.from_numpy(q_), p.detach(), rtol=1e-5, atol=1e-5)
