"""CPU-side checks of the centralised CTE policy (no GPU): the ctypes structure has the header's layout, the entry
points refuse unsupported shapes and bad arguments before any device work, FusedCtePolicy refuses modules it does not
implement, the module's multi-categorical arithmetic equals a loop over N categoricals, and ppo_update_cte equals a
hand-written PPO loop."""
import ctypes as C
import shutil
import subprocess
from pathlib import Path
from types import SimpleNamespace

import pytest
import torch

from dl_reference_models_b200 import _native as nat

REPO = Path(__file__).resolve().parents[1]
FIELDS = [name for name, _ in nat.MapfCtePolicyArgs._fields_]


@pytest.mark.skipif(shutil.which("gcc") is None, reason="needs gcc")
def test_ctypes_structure_matches_the_header_layout(tmp_path):
    src = tmp_path / "probe.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "mapf_b200.h"\nint main(void) {\n'
                   '    printf("%zu\\n", sizeof(mapf_cte_policy_args));\n'
                   + "".join(f'    printf("%zu\\n", offsetof(mapf_cte_policy_args, {f}));\n' for f in FIELDS)
                   + '    printf("%d\\n", MAPF_CTE_POLICY_MAX_CELLS);\n    return 0;\n}\n')
    exe = tmp_path / "probe"
    subprocess.run(["gcc", "-std=c99", "-I", str(REPO / "include"), "-o", str(exe), str(src)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    want = [C.sizeof(nat.MapfCtePolicyArgs)] + [getattr(nat.MapfCtePolicyArgs, f).offset for f in FIELDS] + [1024]
    assert got == want


def test_weight_block_size_refuses_unsupported_shapes():
    L = nat.lib()
    for cells, n in ((0, 4), (200, 0), (200, 33), (1025, 4), (-1, 4)):
        assert L.mapf_cte_policy_weights_nbytes(cells, n) == nat.ERR_UNSUPPORTED, (cells, n)
    for cells, n in ((1, 1), (200, 4), (600, 16), (1024, 32)):
        nb = L.mapf_cte_policy_weights_nbytes(cells, n)
        assert nb > 0 and nb % 16 == 0, (cells, n, nb)
    assert L.mapf_cte_policy_weights_nbytes(1024, 32) > L.mapf_cte_policy_weights_nbytes(1024, 1)
    assert L.mapf_cte_policy_weights_nbytes(1024, 32) <= 227 * 1024 - 8 * 6144   # resident next to the staging


def test_pack_and_act_validate_their_arguments_before_any_device_work():
    L = nat.lib()
    assert L.mapf_cte_policy_pack_weights(200, 4, *([None] * 9)) == nat.ERR_INVALID_ARG
    assert L.mapf_cte_policy_pack_weights(1025, 4, *([None] * 9)) == nat.ERR_UNSUPPORTED
    assert L.mapf_cte_policy_pack_weights(200, 33, *([None] * 9)) == nat.ERR_UNSUPPORTED
    assert L.mapf_cte_policy_act(None, None) == nat.ERR_INVALID_ARG
    fake = C.c_void_p(16)
    a = nat.MapfCtePolicyArgs(num_envs=4, num_agents=4, cells=1025, obs_grid=fake, action_mask=fake, weights=fake)
    assert L.mapf_cte_policy_act(C.byref(a), None) == nat.ERR_UNSUPPORTED
    a.cells, a.num_agents = 200, 0
    assert L.mapf_cte_policy_act(C.byref(a), None) == nat.ERR_UNSUPPORTED
    a.num_agents = 33
    assert L.mapf_cte_policy_act(C.byref(a), None) == nat.ERR_UNSUPPORTED
    a.num_agents = 4
    for k in ("obs_grid", "action_mask", "weights"):
        setattr(a, k, None)
        assert L.mapf_cte_policy_act(C.byref(a), None) == nat.ERR_INVALID_ARG, k
        setattr(a, k, fake)
    a.num_envs = 0
    assert L.mapf_cte_policy_act(C.byref(a), None) == nat.ERR_INVALID_ARG
    a.num_envs, a.reserved = 4, 1
    assert L.mapf_cte_policy_act(C.byref(a), None) == nat.ERR_INVALID_ARG
    assert b"reserved" in L.mapf_last_error()


def _stub_env(R=10, C_=20, N=4):
    # enough of BatchedCteEnv for the shape checks; device work would fail on the missing attributes
    return SimpleNamespace(R=R, C=C_, N=N)


@pytest.mark.parametrize("kwargs", [dict(hiddens=(64,)), dict(hiddens=(64, 32)), dict(hiddens=(128, 64)),
                                    dict(no_masking=True), dict(cells=199), dict(num_agents=5), None])
def test_fused_cte_policy_refuses_modules_it_does_not_implement(kwargs):
    from dl_reference_models_b200.cte_rollout import CteActionMaskPolicy
    from dl_reference_models_b200.policy_kernels import FusedCtePolicy
    from dl_reference_models_b200.rollout import ActionMaskPolicy

    if kwargs is None:   # a multi-agent policy
        policy = ActionMaskPolicy(200)
    else:
        kw = dict(cells=200, num_agents=4)
        kw.update(kwargs)
        policy = CteActionMaskPolicy(**kw)
    with pytest.raises(ValueError, match="fused CTE kernel"):
        FusedCtePolicy(policy, _stub_env())


def test_fused_cte_policy_refuses_maps_beyond_the_supported_size():
    from dl_reference_models_b200.cte_rollout import CteActionMaskPolicy
    from dl_reference_models_b200.policy_kernels import FusedCtePolicy

    with pytest.raises(ValueError, match="does not support"):
        FusedCtePolicy(CteActionMaskPolicy(33 * 33, 4), _stub_env(33, 33, 4))


def test_module_masking_joint_logp_and_entropy_equal_a_loop_over_categoricals():
    from dl_reference_models_b200.cte_rollout import CteActionMaskPolicy, joint_logp_entropy
    from dl_reference_models_b200.rollout import FLOAT_MIN

    torch.manual_seed(0)
    B, R, C_, N = 7, 4, 5, 3
    pol = CteActionMaskPolicy(R * C_, N)
    grid = torch.randint(0, 2 * N + 2, (B, R, C_), dtype=torch.uint8)
    mask = (torch.rand(B, 5 * N) < 0.6).to(torch.int8)
    mask[:, 0::5] = 1
    lg, v = pol(grid, mask)
    assert lg.shape == (B, N, 5) and v.shape == (B,)
    z = pol.trunk(grid.reshape(B, -1).float())
    raw = pol.logits(z)
    assert torch.allclose(v, pol.value(z).squeeze(-1))
    acts = torch.randint(0, 5, (B, N))
    lp, ent = joint_logp_entropy(lg, acts)
    for b in range(B):
        want_lp, want_ent = 0.0, 0.0
        for j in range(N):
            l = raw[b, 5 * j:5 * j + 5] + torch.clamp(torch.log(mask[b, 5 * j:5 * j + 5].float() + 1e-6), min=FLOAT_MIN)
            assert torch.allclose(lg[b, j], l)
            d = torch.distributions.Categorical(logits=l)
            want_lp = want_lp + d.log_prob(acts[b, j])
            want_ent = want_ent + d.entropy()
        assert torch.allclose(lp[b], want_lp, atol=1e-6) and torch.allclose(ent[b], want_ent, atol=1e-6)
    unmasked, _ = CteActionMaskPolicy(R * C_, N, no_masking=True)(grid, mask)
    assert unmasked.shape == (B, N, 5)


def _synthetic_batch(T=6, B=10, R=3, C_=4, N=3, seed=0):
    from dl_reference_models_b200.cte_rollout import CteBatch

    g = torch.Generator().manual_seed(seed)
    masks = (torch.rand(T + 1, B, 5 * N, generator=g) < 0.7).to(torch.int8)
    return CteBatch(grid=torch.randint(0, 2 * N + 2, (T + 1, B, R * C_), dtype=torch.uint8, generator=g), masks=masks,
                    actions=torch.randint(0, 5, (T, B, N), generator=g), logp=-torch.rand(T, B, generator=g) * 4,
                    values=torch.randn(T, B, generator=g), rewards=torch.randn(T, B, generator=g),
                    dones=torch.rand(T, B, generator=g) < 0.2, last_value=torch.randn(B, generator=g))


def test_ppo_update_cte_equals_a_hand_written_loop():
    from dl_reference_models_b200.cte_rollout import CteActionMaskPolicy, ppo_update_cte

    T, B, R, C_, N = 6, 10, 3, 4, 3
    batch = _synthetic_batch(T, B, R, C_, N)
    torch.manual_seed(3)
    pol = CteActionMaskPolicy(R * C_, N)
    ref = CteActionMaskPolicy(R * C_, N)
    ref.load_state_dict(pol.state_dict())
    opt, ref_opt = torch.optim.Adam(pol.parameters(), lr=1e-3), torch.optim.Adam(ref.parameters(), lr=1e-3)
    kw = dict(clip=0.05, vf_coeff=0.5, entropy_coeff=0.001, epochs=3, minibatch=16, gamma=0.99, lam=0.95)
    stats = ppo_update_cte(pol, opt, batch, generator=torch.Generator().manual_seed(11), **kw)

    # the hand-written loop: scalar GAE, whole-batch normalisation, env-step minibatches, joint multi-categorical
    adv = torch.zeros(T, B)
    running, next_value = torch.zeros(B), batch.last_value
    for t in range(T - 1, -1, -1):
        nd = (~batch.dones[t]).float()
        delta = batch.rewards[t] + 0.99 * next_value * nd - batch.values[t]
        running = delta + 0.99 * 0.95 * nd * running
        adv[t] = running
        next_value = batch.values[t]
    ret = (adv + batch.values).reshape(-1)
    adv = ((adv - adv.mean()) / (adv.std() + 1e-8)).reshape(-1)
    grid, masks = batch.grid[:T].reshape(T * B, -1), batch.masks[:T].reshape(T * B, -1)
    acts, old = batch.actions.reshape(T * B, N), batch.logp.reshape(-1)
    gen = torch.Generator().manual_seed(11)
    for _ in range(3):
        perm = torch.randperm(T * B, generator=gen)
        for i in range(0, T * B, 16):
            idx = perm[i:i + 16]
            lg, v = ref(grid[idx], masks[idx])
            lp = torch.zeros(len(idx))
            ent = torch.zeros(len(idx))
            for j in range(N):
                d = torch.distributions.Categorical(logits=lg[:, j])
                lp = lp + d.log_prob(acts[idx, j])
                ent = ent + d.entropy()
            ratio = torch.exp(lp - old[idx])
            surr = torch.min(ratio * adv[idx], torch.clamp(ratio, 0.95, 1.05) * adv[idx])
            loss = -surr.mean() + 0.5 * (v - ret[idx]).pow(2).mean() - 0.001 * ent.mean()
            ref_opt.zero_grad()
            loss.backward()
            ref_opt.step()
    assert abs(stats["loss"] - float(loss.detach())) <= 1e-5
    for (name, p), q in zip(pol.named_parameters(), ref.parameters()):
        assert torch.allclose(p, q, atol=1e-5), name


def test_ppo_update_cte_stops_after_max_minibatches():
    from dl_reference_models_b200.cte_rollout import CteActionMaskPolicy, ppo_update_cte

    batch = _synthetic_batch()
    pol = CteActionMaskPolicy(12, 3)
    before = [p.detach().clone() for p in pol.parameters()]
    seen = []
    opt = torch.optim.SGD(pol.parameters(), lr=0.1)
    orig = opt.step
    opt.step = lambda *a, **k: (seen.append(1), orig(*a, **k))[1]
    stats = ppo_update_cte(pol, opt, batch, epochs=5, minibatch=8, max_minibatches=3)
    assert len(seen) == 3 and set(stats) == {"loss", "vf_loss", "entropy", "policy_loss"}
    assert any(not torch.equal(a, b) for a, b in zip(before, pol.parameters()))
