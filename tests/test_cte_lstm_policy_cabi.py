"""CPU-side checks of the recurrent centralised CTE policy (no GPU): the ctypes structure has the header's layout, the
entry points refuse unsupported shapes and bad arguments before any device work, FusedCteRecurrentPolicy refuses
modules it does not implement, the module's arithmetic equals a hand-written LSTM, and ppo_update_cte_recurrent equals
a hand-written PPO loop (also across two gloo ranks)."""
import ctypes as C
import os
import shutil
import subprocess
from pathlib import Path
from types import SimpleNamespace

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

from dl_reference_models_b200 import _native as nat

REPO = Path(__file__).resolve().parents[1]
FIELDS = [name for name, _ in nat.MapfCteLstmPolicyArgs._fields_]


@pytest.mark.skipif(shutil.which("gcc") is None, reason="needs gcc")
def test_ctypes_structure_matches_the_header_layout(tmp_path):
    src = tmp_path / "probe.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "mapf_b200.h"\nint main(void) {\n'
                   '    printf("%zu\\n", sizeof(mapf_cte_lstm_policy_args));\n'
                   + "".join(f'    printf("%zu\\n", offsetof(mapf_cte_lstm_policy_args, {f}));\n' for f in FIELDS)
                   + '    return 0;\n}\n')
    exe = tmp_path / "probe"
    subprocess.run(["gcc", "-std=c99", "-I", str(REPO / "include"), "-o", str(exe), str(src)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    want = [C.sizeof(nat.MapfCteLstmPolicyArgs)] + [getattr(nat.MapfCteLstmPolicyArgs, f).offset for f in FIELDS]
    assert got == want


def test_weight_block_size_refuses_unsupported_shapes():
    L = nat.lib()
    for cells, n in ((0, 4), (200, 0), (200, 33), (1025, 4), (-1, 4)):
        assert L.mapf_cte_lstm_policy_weights_nbytes(cells, n) == nat.ERR_UNSUPPORTED, (cells, n)
    for cells, n in ((1, 1), (200, 4), (600, 16), (1024, 32)):
        nb = L.mapf_cte_lstm_policy_weights_nbytes(cells, n)
        assert nb > 0 and nb % 16 == 0, (cells, n, nb)
    assert L.mapf_cte_lstm_policy_weights_nbytes(1024, 32) > L.mapf_cte_lstm_policy_weights_nbytes(1024, 1)


def test_pack_and_act_validate_their_arguments_before_any_device_work():
    L = nat.lib()
    assert L.mapf_cte_lstm_policy_pack_weights(200, 4, *([None] * 13)) == nat.ERR_INVALID_ARG
    assert L.mapf_cte_lstm_policy_pack_weights(1025, 4, *([None] * 13)) == nat.ERR_UNSUPPORTED
    assert L.mapf_cte_lstm_policy_pack_weights(200, 33, *([None] * 13)) == nat.ERR_UNSUPPORTED
    assert L.mapf_cte_lstm_policy_act(None, None) == nat.ERR_INVALID_ARG
    fake = C.c_void_p(16)
    required = ("obs_grid", "action_mask", "prev_action", "prev_reward", "h_in", "c_in", "trunk", "weights")
    a = nat.MapfCteLstmPolicyArgs(num_envs=4, num_agents=4, cells=1025, **{k: fake for k in required})
    assert L.mapf_cte_lstm_policy_act(C.byref(a), None) == nat.ERR_UNSUPPORTED
    a.cells, a.num_agents = 200, 33
    assert L.mapf_cte_lstm_policy_act(C.byref(a), None) == nat.ERR_UNSUPPORTED
    a.num_agents = 0
    assert L.mapf_cte_lstm_policy_act(C.byref(a), None) == nat.ERR_UNSUPPORTED
    a.num_agents = 4
    for k in required:
        setattr(a, k, None)
        assert L.mapf_cte_lstm_policy_act(C.byref(a), None) == nat.ERR_INVALID_ARG, k
        setattr(a, k, fake)
    a.num_envs = 0
    assert L.mapf_cte_lstm_policy_act(C.byref(a), None) == nat.ERR_INVALID_ARG
    a.num_envs = 4
    for ho, co in ((fake, None), (None, fake)):
        a.h_out, a.c_out = ho, co
        assert L.mapf_cte_lstm_policy_act(C.byref(a), None) == nat.ERR_INVALID_ARG
        assert b"together" in L.mapf_last_error()
    a.h_out = a.c_out = None
    a.reserved = 1
    assert L.mapf_cte_lstm_policy_act(C.byref(a), None) == nat.ERR_INVALID_ARG


def _stub_env(R=10, C_=20, N=4):
    # enough of BatchedCteEnv for the shape checks; device work would fail on the missing attributes
    return SimpleNamespace(R=R, C=C_, N=N)


@pytest.mark.parametrize("kwargs", [dict(hiddens=(64,)), dict(hiddens=(64, 32)), dict(cell=32), dict(use_prev_action=False),
                                    dict(use_prev_reward=False), dict(cells=199), dict(num_agents=5), None])
def test_fused_cte_recurrent_policy_refuses_modules_it_does_not_implement(kwargs):
    from dl_reference_models_b200.cte_rollout import CteActionMaskPolicy, CteRecurrentPolicy
    from dl_reference_models_b200.policy_kernels import FusedCteRecurrentPolicy

    if kwargs is None:   # the feed-forward CTE policy
        policy = CteActionMaskPolicy(200, 4)
    else:
        kw = dict(cells=200, num_agents=4)
        kw.update(kwargs)
        policy = CteRecurrentPolicy(**kw)
    with pytest.raises(ValueError, match="fused recurrent CTE kernel implements"):
        FusedCteRecurrentPolicy(policy, _stub_env())


def test_fused_cte_recurrent_policy_refuses_maps_beyond_the_supported_size():
    from dl_reference_models_b200.cte_rollout import CteRecurrentPolicy
    from dl_reference_models_b200.policy_kernels import FusedCteRecurrentPolicy

    with pytest.raises(ValueError, match="does not support"):
        FusedCteRecurrentPolicy(CteRecurrentPolicy(33 * 33, 4), _stub_env(33, 33, 4))


def test_step_equals_a_hand_written_lstm_with_the_concatenated_one_hots():
    from dl_reference_models_b200.cte_rollout import CteRecurrentPolicy
    from dl_reference_models_b200.rollout import FLOAT_MIN

    torch.manual_seed(0)
    M, R, C_, N = 6, 3, 4, 3
    pol = CteRecurrentPolicy(R * C_, N, hiddens=(16, 8), cell=5)
    assert pol.lstm.input_size == 8 + 5 * N + 1
    grid = torch.randint(0, 2 * N + 2, (M, R, C_), dtype=torch.uint8)
    mask = (torch.rand(M, 5 * N) < 0.6).to(torch.int8)
    pa = torch.randint(0, 5, (M, N))
    pr = torch.randn(M, dtype=torch.float64)
    h0, c0 = torch.randn(M, 5), torch.randn(M, 5)
    lg, v, (h, c) = pol.step(grid, mask, pa, pr, (h0, c0))
    assert lg.shape == (M, N, 5) and v.shape == (M,)
    lin = [m for m in pol.trunk if isinstance(m, torch.nn.Linear)]
    y = torch.relu(lin[1](torch.relu(lin[0](grid.reshape(M, -1).float()))))
    onehot = torch.zeros(M, 5 * N)
    for m in range(M):
        for j in range(N):   # agent j's five columns, agents in order
            onehot[m, 5 * j + int(pa[m, j])] = 1.0
    x = torch.cat([y, onehot, pr.float().unsqueeze(-1)], -1)
    gates = x @ pol.lstm.weight_ih.T + pol.lstm.bias_ih + h0 @ pol.lstm.weight_hh.T + pol.lstm.bias_hh
    i, f, g, o = gates.chunk(4, -1)
    want_c = torch.sigmoid(f) * c0 + torch.sigmoid(i) * torch.tanh(g)
    want_h = torch.sigmoid(o) * torch.tanh(want_c)
    want_l = pol.logits(want_h) + torch.clamp(torch.log(mask.float() + 1e-6), min=FLOAT_MIN)
    assert torch.allclose(h, want_h, atol=1e-6) and torch.allclose(c, want_c, atol=1e-6)
    assert torch.allclose(lg, want_l.reshape(M, N, 5), atol=1e-5)
    assert torch.allclose(v, pol.value(want_h).squeeze(-1), atol=1e-6)


def test_sequence_with_resets_equals_explicitly_zeroed_inputs():
    from dl_reference_models_b200.cte_rollout import CteRecurrentPolicy

    torch.manual_seed(1)
    T, M, cells, N = 5, 4, 12, 3
    pol = CteRecurrentPolicy(cells, N, hiddens=(8,), cell=6)
    grid = torch.randint(0, 8, (T, M, cells), dtype=torch.uint8)
    mask = torch.ones(T, M, 5 * N, dtype=torch.int8)
    pa = torch.randint(0, 5, (T, M, N))
    pr = torch.randn(T, M)
    resets = torch.rand(T, M) < 0.4
    resets[2, 1] = True
    state = (torch.randn(M, 6), torch.randn(M, 6))
    lg, v, (h, c) = pol.sequence(grid, mask, pa, pr, resets, state)
    hh, cc = state
    for t in range(T):
        l_t, v_t = [], []
        nh, nc = [], []
        for m in range(M):
            z = bool(resets[t, m])
            s = (torch.zeros(1, 6), torch.zeros(1, 6)) if z else (hh[m:m + 1], cc[m:m + 1])
            a = torch.zeros(1, N, dtype=torch.int64) if z else pa[t, m:m + 1]
            r = torch.zeros(1) if z else pr[t, m:m + 1]
            l1, v1, (h1, c1) = pol.step(grid[t, m:m + 1], mask[t, m:m + 1], a, r, s)
            l_t.append(l1); v_t.append(v1); nh.append(h1); nc.append(c1)
        assert torch.allclose(lg[t], torch.cat(l_t), atol=1e-6) and torch.allclose(v[t], torch.cat(v_t), atol=1e-6)
        hh, cc = torch.cat(nh), torch.cat(nc)
    assert torch.allclose(h, hh, atol=1e-6) and torch.allclose(c, cc, atol=1e-6)


def _synthetic_batch(T=8, B=6, cells=12, N=3, L=4, seed=0):
    from dl_reference_models_b200.cte_rollout import CteRecurrentBatch

    g = torch.Generator().manual_seed(seed)
    resets = torch.rand(T, B, generator=g) < 0.2
    keep = ~resets
    return CteRecurrentBatch(
        grid=torch.randint(0, 2 * N + 2, (T + 1, B, cells), dtype=torch.uint8, generator=g),
        masks=(torch.rand(T + 1, B, 5 * N, generator=g) < 0.7).to(torch.int8),
        actions=torch.randint(0, 5, (T, B, N), generator=g), logp=-torch.rand(T, B, generator=g) * 4,
        values=torch.randn(T, B, generator=g), rewards=torch.randn(T, B, generator=g),
        dones=torch.rand(T, B, generator=g) < 0.2, last_value=torch.randn(B, generator=g),
        prev_actions=torch.randint(0, 5, (T, B, N), generator=g) * keep.unsqueeze(-1),
        prev_rewards=torch.randn(T, B, generator=g) * keep, resets=resets,
        chunk_h=torch.randn(T // L, B, 64, generator=g), chunk_c=torch.randn(T // L, B, 64, generator=g))


KW = dict(max_seq_len=4, clip=0.05, vf_coeff=0.5, entropy_coeff=0.001, epochs=2, minibatch=8, gamma=0.99, lam=0.95)


def _reference_update(ref, ref_opt, batch, gen, L=4, epochs=2, per_mb=2, steps=None, on_grads=None):
    """The hand-written learner: scalar GAE, whole-batch normalisation, per_mb sequences of L steps from their chunk
    states, the joint multi-categorical PPO loss."""
    T, B = batch.rewards.shape
    N = batch.actions.shape[-1]
    adv = torch.zeros(T, B)
    running, next_value = torch.zeros(B), batch.last_value
    for t in range(T - 1, -1, -1):
        nd = (~batch.dones[t]).float()
        delta = batch.rewards[t] + 0.99 * next_value * nd - batch.values[t]
        running = delta + 0.99 * 0.95 * nd * running
        adv[t] = running
        next_value = batch.values[t]
    ret = adv + batch.values
    adv = (adv - adv.mean()) / (adv.std() + 1e-8)
    done, loss = 0, None
    for _ in range(epochs):
        perm = torch.randperm((T // L) * B, generator=gen)
        for i in range(0, len(perm), per_mb):
            lp_all, ent_all, v_all, old, a_, r_ = [], [], [], [], [], []
            for s in perm[i:i + per_mb].tolist():
                k, m = divmod(s, B)
                h, c = batch.chunk_h[k, m:m + 1], batch.chunk_c[k, m:m + 1]
                for t in range(k * L, k * L + L):
                    if batch.resets[t, m]:
                        h, c = torch.zeros_like(h), torch.zeros_like(c)
                    lg, v, (h, c) = ref.step(batch.grid[t, m:m + 1], batch.masks[t, m:m + 1],
                                             batch.prev_actions[t, m:m + 1], batch.prev_rewards[t, m:m + 1], (h, c))
                    lp, ent = torch.zeros(1), torch.zeros(1)
                    for j in range(N):
                        d = torch.distributions.Categorical(logits=lg[:, j])
                        lp = lp + d.log_prob(batch.actions[t, m, j].view(1))
                        ent = ent + d.entropy()
                    lp_all.append(lp); ent_all.append(ent); v_all.append(v)
                    old.append(batch.logp[t, m].view(1)); a_.append(adv[t, m].view(1)); r_.append(ret[t, m].view(1))
            lp, ent, v = torch.cat(lp_all), torch.cat(ent_all), torch.cat(v_all)
            old, a_, r_ = torch.cat(old), torch.cat(a_), torch.cat(r_)
            ratio = torch.exp(lp - old)
            surr = torch.min(ratio * a_, torch.clamp(ratio, 0.95, 1.05) * a_)
            loss = -surr.mean() + 0.5 * (v - r_).pow(2).mean() - 0.001 * ent.mean()
            ref_opt.zero_grad()
            loss.backward()
            if on_grads is not None:
                on_grads([p.grad.clone() for p in ref.parameters()])
            ref_opt.step()
            done += 1
            if steps is not None and done >= steps:
                return loss
    return loss


def test_ppo_update_cte_recurrent_equals_a_hand_written_loop():
    from dl_reference_models_b200.cte_rollout import CteRecurrentPolicy, ppo_update_cte_recurrent

    batch = _synthetic_batch()
    torch.manual_seed(3)
    pol = CteRecurrentPolicy(12, 3)
    ref = CteRecurrentPolicy(12, 3)
    ref.load_state_dict(pol.state_dict())
    opt, ref_opt = torch.optim.Adam(pol.parameters(), lr=1e-3), torch.optim.Adam(ref.parameters(), lr=1e-3)
    stats = ppo_update_cte_recurrent(pol, opt, batch, generator=torch.Generator().manual_seed(11), **KW)
    loss = _reference_update(ref, ref_opt, batch, torch.Generator().manual_seed(11))
    assert abs(stats["loss"] - float(loss.detach())) <= 1e-5
    for (name, p), q in zip(pol.named_parameters(), ref.parameters()):
        assert torch.allclose(p, q, atol=1e-5), name


def test_ppo_update_cte_recurrent_stops_after_max_minibatches():
    from dl_reference_models_b200.cte_rollout import CteRecurrentPolicy, ppo_update_cte_recurrent

    batch = _synthetic_batch()
    pol = CteRecurrentPolicy(12, 3)
    before = [p.detach().clone() for p in pol.parameters()]
    seen = []
    opt = torch.optim.SGD(pol.parameters(), lr=0.1)
    orig = opt.step
    opt.step = lambda *a, **k: (seen.append(1), orig(*a, **k))[1]
    stats = ppo_update_cte_recurrent(pol, opt, batch, max_seq_len=4, epochs=5, minibatch=8, max_minibatches=3)
    assert len(seen) == 3 and set(stats) == {"loss", "vf_loss", "entropy", "policy_loss"}
    assert any(not torch.equal(a, b) for a, b in zip(before, pol.parameters()))
    with pytest.raises(ValueError, match="multiple of max_seq_len"):
        ppo_update_cte_recurrent(pol, opt, batch, max_seq_len=3)


def _gloo_worker(rank, world, port, q):
    import torch.distributed as dist

    from dl_reference_models_b200.cte_rollout import CteRecurrentPolicy, ppo_update_cte_recurrent

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.manual_seed(0)
    pol = CteRecurrentPolicy(12, 3)
    opt = torch.optim.SGD(pol.parameters(), lr=0.0)
    grads = []
    orig = opt.step
    opt.step = lambda *a, **k: (grads.append([p.grad.detach().numpy().copy() for p in pol.parameters()]), orig(*a, **k))[1]
    ppo_update_cte_recurrent(pol, opt, _synthetic_batch(seed=100 + rank), world_size=world, max_minibatches=1,
                             generator=torch.Generator().manual_seed(5 + rank), **KW)
    q.put((rank, grads[0]))   # plain arrays: no shared-memory handles
    dist.barrier()
    dist.destroy_process_group()


def test_two_gloo_ranks_step_with_the_mean_of_their_gradients():
    from dl_reference_models_b200.cte_rollout import CteRecurrentPolicy

    import socket

    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = dict(q.get(timeout=120) for _ in procs)
    for p in procs:
        p.join(timeout=60)
    per_rank = []
    for r in range(2):   # reference: each rank's first minibatch in this process
        torch.manual_seed(0)
        ref = CteRecurrentPolicy(12, 3)
        seen = []
        _reference_update(ref, torch.optim.SGD(ref.parameters(), lr=0.0), _synthetic_batch(seed=100 + r),
                          torch.Generator().manual_seed(5 + r), steps=1, on_grads=seen.append)
        per_rank.append(seen[0])
    for i in range(len(per_rank[0])):
        want = ((per_rank[0][i] + per_rank[1][i]) / 2).numpy()
        assert np.allclose(got[0][i], want, atol=1e-6) and np.allclose(got[1][i], want, atol=1e-6), i
