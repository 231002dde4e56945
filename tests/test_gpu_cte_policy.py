"""The fused centralised CTE policy (mapf_cte_policy_act: grid codes -> bf16 tensor-core MLP with a K = R*C first layer
-> N masked 5-way draws), its collector and its learner, against plain PyTorch.  Maps 2-1 (10x20), 3-1 (20x30) and a
random 32x32 one, N in {1, 4, 16, 32}, batches that are not a multiple of the kernel's 32-env tiles.  Tolerances: the
kernel rounds W1, W2, the heads and both hidden activations to bf16 (the grid codes are exact) and accumulates in f32;
against a torch reference that rounds at the same points the masked logits and the value agree to 2e-4 on average and
3e-2 at worst, as for the multi-agent MLP kernel (a hidden activation next to a bf16 rounding boundary may flip by one
ulp with the accumulation order)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

CASES = [("ReferenceModel-2-1", 1), ("ReferenceModel-2-1", 4), ("ReferenceModel-3-1", 16), ("ReferenceModel-3-1", 32),
         ("rand32", 1), ("rand32", 16), ("rand32", 32)]


def grid_of(name):
    from dl_reference_models_b200 import maps

    return maps.random_obstacle_grid(32, 32, 0.30, 2026, min_free=64) if name == "rand32" else maps.get_grid(name)


def make_env(name, n, B=1003, steps_per_episode=64, seed=5, scramble=3):
    import torch

    from dl_reference_models_b200.single_agent import BatchedCteEnv

    env = BatchedCteEnv({"grid": grid_of(name), "num_agents": n, "steps_per_episode": steps_per_episode, "seed": seed}, B)
    env.reset()
    g = torch.Generator(device=env.device).manual_seed(seed)
    for _ in range(scramble):
        env.step(torch.randint(0, 5, (B, n), dtype=torch.int8, device=env.device, generator=g), auto_reset=True)
    return env


def make_policy(env, seed=0):
    import torch

    from dl_reference_models_b200.cte_rollout import CteActionMaskPolicy

    torch.manual_seed(seed)
    return CteActionMaskPolicy(env.R * env.C, env.N).to(env.device)


def bf16_reference(policy, grid, mask):
    """The kernel's arithmetic in float64 with bf16 rounding at the kernel's points -> (masked logits [B,N,5], value)."""
    import torch

    r = lambda t: t.to(torch.bfloat16).double()  # noqa: E731
    lin = [m for m in policy.trunk if isinstance(m, torch.nn.Linear)]
    h = grid.reshape(grid.shape[0], -1).double()
    for l in lin:
        h = r(torch.relu(h @ r(l.weight).T + l.bias.double()))
    logits = h @ r(policy.logits.weight).T + policy.logits.bias.double()
    value = (h @ r(policy.value.weight).T + policy.value.bias.double()).squeeze(-1)
    logits = logits + torch.where(mask != 0, 9.99999e-07, -13.815511).double()
    return logits.reshape(grid.shape[0], -1, 5), value


@pytest.mark.parametrize("name,n", CASES)
def test_one_launch_matches_torch(name, n):
    import torch

    from dl_reference_models_b200.policy_kernels import FusedCtePolicy

    env = make_env(name, n)
    policy = make_policy(env)
    fused = FusedCtePolicy(policy, env, seed=7)
    logits = torch.zeros((env.B, n, 5), device=env.device)
    acts, logp, value = fused.act(logits_out=logits)
    with torch.no_grad():
        ref_l, ref_v = bf16_reference(policy, env.obs_grid, env.action_mask)
    dl, dv = (logits.double() - ref_l).abs(), (value.double() - ref_v).abs()
    assert float(dl.max()) <= 3e-2 and float(dv.max()) <= 3e-2, (float(dl.max()), float(dv.max()))
    assert float(dl.mean()) <= 2e-4 and float(dv.mean()) <= 2e-4, (float(dl.mean()), float(dv.mean()))
    ref_logp = torch.log_softmax(logits.double(), -1).gather(-1, acts.long().unsqueeze(-1)).squeeze(-1).sum(-1)
    assert float((logp.double() - ref_logp).abs().max()) <= 1e-4
    assert torch.equal(fused.actions64, acts.long())
    # masked actions carry a ~1e-6 probability; at these fixed seeds (a deterministic launch) none is drawn
    mask = env.action_mask.view(env.B, n, 5)
    assert bool((mask.gather(-1, acts.long().unsqueeze(-1)) == 1).all())
    # the same seed and counter draw the same actions
    again = FusedCtePolicy(policy, env, seed=7)
    assert torch.equal(again.act()[0], acts)


def test_draws_follow_the_softmax_of_the_launch_logits():
    """The same observation in every env, different Philox streams: per agent, the action frequencies follow the
    softmax of the launch's own logits."""
    import torch

    from dl_reference_models_b200.policy_kernels import FusedCtePolicy

    env = make_env("ReferenceModel-2-1", 4, B=4096)
    env.obs_grid.copy_(env.obs_grid[:1].expand_as(env.obs_grid).clone())
    env.action_mask.copy_(env.action_mask[:1].expand_as(env.action_mask).clone())
    fused = FusedCtePolicy(make_policy(env, seed=1), env)
    logits = torch.zeros((env.B, env.N, 5), device=env.device)
    counts = torch.zeros((env.N, 5), device=env.device)
    draws = 0
    for _ in range(20):
        acts, _, _ = fused.act(logits_out=logits)
        counts += torch.nn.functional.one_hot(acts.long(), 5).sum(0)
        draws += env.B
    assert torch.equal(logits, logits[:1].expand_as(logits))
    exp = torch.softmax(logits[0], -1) * draws
    keep = exp > 5
    chi2 = (((counts - exp) ** 2 / exp.clamp_min(1e-9)) * keep).sum(-1)
    assert float(chi2.max()) < 40, (counts.tolist(), exp.tolist())   # <= 4 dof per agent, 4 agents


@pytest.mark.parametrize("name", ["ReferenceModel-2-1", "rand32"])
def test_a_shard_with_its_env_id_base_reproduces_the_full_launch(name):
    import torch

    from dl_reference_models_b200.policy_kernels import FusedCtePolicy

    env = make_env(name, 16 if name == "rand32" else 4)
    policy = make_policy(env)
    full = FusedCtePolicy(policy, env, seed=3)
    lf = torch.zeros((env.B, env.N, 5), device=env.device)
    a, lp, v = (x.clone() for x in full.act(logits_out=lf))
    off, n = 37, 500
    shard = FusedCtePolicy(policy, env, seed=3, env_id_base=off)
    ls = torch.zeros((env.B, env.N, 5), device=env.device)
    sa, slp, sv = shard.act(env.obs_grid[off:off + n], env.action_mask[off:off + n], logits_out=ls, num_envs=n)
    assert torch.equal(sa[:n], a[off:off + n]) and torch.equal(slp[:n], lp[off:off + n])
    assert torch.equal(sv[:n], v[off:off + n]) and torch.equal(ls[:n], lf[off:off + n])


def test_collector_equals_a_manual_loop_over_two_collects():
    import torch

    from dl_reference_models_b200.cte_rollout import FusedCteCollector
    from dl_reference_models_b200.policy_kernels import FusedCtePolicy

    n, B, T = 4, 203, 8
    envs = [make_env("ReferenceModel-2-1", n, B=B, steps_per_episode=5, seed=9) for _ in range(2)]
    policy = make_policy(envs[0])
    fa, fb = FusedCtePolicy(policy, envs[0], seed=4), FusedCtePolicy(policy, envs[1], seed=4)
    collector = FusedCteCollector(envs[0], fa, T)
    env = envs[1]
    cells = env.R * env.C
    ended = 0
    for round_ in range(2):
        batch = collector.collect()
        grid, masks, acts, logp, vals, rew, dones = [], [], [], [], [], [], []
        for t in range(T):
            grid.append(env.obs_grid.view(B, cells).clone())
            masks.append(env.action_mask.clone())
            a, lp, v = fb.act()
            acts.append(fb.actions64.clone())
            logp.append(lp.clone())
            vals.append(v.clone())
            env.step(a, auto_reset=True)
            rew.append(env.reward.float())
            dones.append((env.terminated | env.truncated).bool())
        grid.append(env.obs_grid.view(B, cells).clone())
        masks.append(env.action_mask.clone())
        _, _, last = fb.act()
        for field, want in (("grid", grid), ("masks", masks), ("actions", acts), ("logp", logp), ("values", vals),
                            ("rewards", rew), ("dones", dones)):
            assert torch.equal(getattr(batch, field), torch.stack(want)), (round_, field)
        assert torch.equal(batch.last_value, last), round_
        ended += int(batch.dones.sum())
        for k in ("positions", "goals", "starts", "reached_once", "step_count", "blocking_total", "obs_grid",
                  "action_mask", "flat_obs", "reward", "terminated", "truncated", "info"):
            assert torch.equal(getattr(envs[0], k), getattr(env, k)), (round_, k)
    assert ended > B   # episodes of 5 steps end and auto-reset inside the window


def test_fp32_module_rerun_over_a_fused_batch():
    """What PPO sees: the fp32 module re-run over a fused batch at default init.  Every importance ratio stays inside
    the 0.05 clip; the differences are printed (pytest -s) for the record."""
    import torch

    from dl_reference_models_b200.cte_rollout import FusedCteCollector, joint_logp_entropy
    from dl_reference_models_b200.policy_kernels import FusedCtePolicy

    env = make_env("rand32", 16, B=2051, steps_per_episode=32)
    policy = make_policy(env)
    batch = FusedCteCollector(env, FusedCtePolicy(policy, env), 16).collect()
    T = batch.actions.shape[0]
    with torch.no_grad():
        lg, v = policy(batch.grid[:T], batch.masks[:T])
        lp, _ = joint_logp_entropy(lg, batch.actions)
    dlp, dv = (lp - batch.logp).abs(), (v - batch.values).abs()
    ratio = torch.exp(lp - batch.logp)
    print(f"\nfp32 re-run over a fused CTE batch (N=16, 32x32): |dlogp| mean {float(dlp.mean()):.3g} max "
          f"{float(dlp.max()):.3g}; |dvalue| mean {float(dv.mean()):.3g} max {float(dv.max()):.3g}; ratio "
          f"{float(ratio.min()):.6f} .. {float(ratio.max()):.6f}")
    assert float(ratio.min()) > 0.95 and float(ratio.max()) < 1.05


def test_a_ppo_update_then_refresh_changes_the_launch():
    import torch

    from dl_reference_models_b200.cte_rollout import FusedCteCollector, ppo_update_cte
    from dl_reference_models_b200.policy_kernels import FusedCtePolicy

    env = make_env("ReferenceModel-3-1", 4, B=515, steps_per_episode=16)
    policy = make_policy(env)
    fused = FusedCtePolicy(policy, env, seed=2)
    batch = FusedCteCollector(env, fused, 8).collect()
    fused.counter = 0
    before = [x.clone() for x in fused.act()]
    opt = torch.optim.Adam(policy.parameters(), lr=1e-3)
    stats = ppo_update_cte(policy, opt, batch, epochs=2, minibatch=512, generator=torch.Generator().manual_seed(0))
    assert all(np.isfinite(x) for x in stats.values()), stats
    fused.refresh()
    fused.counter = 0
    after = fused.act()
    assert not torch.equal(after[1], before[1]) and not torch.equal(after[2], before[2])


def test_unsupported_map_size_is_refused():
    import ctypes as C

    import torch

    from dl_reference_models_b200 import _native as nat
    from dl_reference_models_b200.cte_rollout import CteActionMaskPolicy
    from dl_reference_models_b200.policy_kernels import FusedCtePolicy
    from dl_reference_models_b200.single_agent import BatchedCteEnv

    env = BatchedCteEnv({"grid": np.zeros((40, 40), np.uint8), "num_agents": 4, "seed": 1}, 64)
    env.reset()
    with pytest.raises(ValueError, match="does not support"):
        FusedCtePolicy(CteActionMaskPolicy(1600, 4).to(env.device), env)
    w = torch.zeros(1 << 20, dtype=torch.uint8, device=env.device)
    out = torch.zeros(64, device=env.device)
    p = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
    a = nat.MapfCtePolicyArgs(num_envs=64, num_agents=4, cells=1600, obs_grid=p(env.obs_grid),
                              action_mask=p(env.action_mask), weights=p(w), value=p(out))
    assert nat.lib().mapf_cte_policy_act(C.byref(a), env._stream()) == nat.ERR_UNSUPPORTED
    torch.cuda.synchronize()
    assert not bool(out.any())
