"""IMPALA on the B200: the mapf_vtrace kernel against impala.vtrace (identity and gathered columns, out-of-range
column ids), and every learner on batches of the real fused collectors against the loop written out by hand
(tests/impala_loops.py) with impala.vtrace on the device, plus a collect / update / refresh / collect cycle per
family."""
import copy
import math
import sys
from pathlib import Path

import pytest
import torch

from dl_reference_models_b200 import impala, maps
from dl_reference_models_b200 import policy_kernels as pk

sys.path.insert(0, str(Path(__file__).resolve().parent))
import impala_loops  # noqa: E402

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _inputs(T, B, N, M, seed, log_rho_max=30.0):
    g = torch.Generator(device=DEV).manual_seed(seed)
    shape = (T, B, N) if N > 1 else (T, B)
    mu = torch.randn(shape, generator=g, device=DEV) - 1.5
    r = torch.randn(shape, generator=g, device=DEV)
    d = torch.rand((T, B), generator=g, device=DEV) < 0.1
    boot = torch.randn(shape[1:], generator=g, device=DEV)
    pi = torch.randn((T, M), generator=g, device=DEV) - 1.5
    pi += (torch.rand((T, M), generator=g, device=DEV) * 2 - 1) * log_rho_max * (torch.rand((T, M), generator=g, device=DEV) < 0.1)
    v = torch.randn((T, M), generator=g, device=DEV)
    return pi, mu, v, r, d, boot


@pytest.mark.parametrize("T", [1, 37, 64])
@pytest.mark.parametrize("N", [1, 7, 16])
@pytest.mark.parametrize("gathered", [False, True])
def test_kernel_equals_the_torch_recurrence(T, N, gathered):
    B = 13   # B * N = 13, 91, 208 columns: never a multiple of 32
    cols = None
    if gathered:   # repeated and unordered
        g = torch.Generator(device=DEV).manual_seed(T + N)
        cols = torch.randint(0, B * N, (45,), generator=g, device=DEV)
        cols[7] = cols[3]
    M = B * N if cols is None else cols.numel()
    args = _inputs(T, B, N, M, seed=T * 100 + N)
    kw = dict(columns=cols, gamma=0.97, clip_rho=1.5, clip_pg_rho=0.7)
    vs, pg = pk.vtrace(*args, **kw)
    rvs, rpg = impala.vtrace(*args, **kw)
    assert torch.isfinite(vs).all() and torch.isfinite(pg).all()
    torch.testing.assert_close(vs, rvs, rtol=1e-4, atol=1e-4)
    torch.testing.assert_close(pg, rpg, rtol=1e-4, atol=1e-4)
    # on-policy with the default clips: GAE with lambda 1
    if not gathered:
        _, mu, v, r, d, boot = args
        vs, pg = pk.vtrace(mu.reshape(T, -1), mu, v, r, d, boot)
        adv, ret = pk.gae(r.reshape(T, B, N), v.reshape(T, B, N), d, boot.reshape(B, N), 0.99, 1.0)
        torch.testing.assert_close(vs, ret.reshape(T, -1), rtol=1e-4, atol=1e-4)
        torch.testing.assert_close(pg, adv.reshape(T, -1), rtol=1e-4, atol=1e-4)


@pytest.mark.parametrize("N", [1, 16])
def test_gathered_columns_are_the_identity_launch_indexed_bit_for_bit(N):
    T, B = 64, 50
    g = torch.Generator(device=DEV).manual_seed(N)
    cols = torch.randint(0, B * N, (77,), generator=g, device=DEV)
    pi, mu, v, r, d, boot = _inputs(T, B, N, B * N, seed=5)
    vs, pg = pk.vtrace(pi, mu, v, r, d, boot)
    gvs, gpg = pk.vtrace(pi[:, cols], mu, v[:, cols], r, d, boot, columns=cols)
    assert torch.equal(gvs, vs[:, cols]) and torch.equal(gpg, pg[:, cols])


def test_an_out_of_range_column_writes_nan_to_its_own_column_only():
    T, B, N = 20, 10, 4
    cols = torch.tensor([3, -1, 39, 40, 0, 1 << 40], device=DEV)
    pi, mu, v, r, d, boot = _inputs(T, B, N, B * N, seed=9)
    vs, pg = pk.vtrace(pi, mu, v, r, d, boot)
    safe = cols.clamp(0, B * N - 1)
    gvs, gpg = pk.vtrace(pi[:, safe], mu, v[:, safe], r, d, boot, columns=cols)
    bad = torch.tensor([False, True, False, True, False, True], device=DEV)
    for out, ref in ((gvs, vs), (gpg, pg)):
        assert torch.isnan(out[:, bad]).all()
        assert torch.equal(out[:, ~bad], ref[:, safe[~bad]])
    torch.cuda.synchronize()


# ---- learners on real fused collects ---------------------------------------------------------------------------------

B, N, T, L = 64, 4, 32, 16
HP = dict(minibatch=128, grad_clip=1.0, gamma=0.99, clip_rho=1.0, clip_pg_rho=1.0, vf_coeff=0.5, entropy_coeff=0.01)


def _grid():
    return maps.random_obstacle_grid(16, 16, 0.2, 7, min_free=16)


def _mapf_env():
    from dl_reference_models_b200.batched_env import BatchedMapfEnv

    env = BatchedMapfEnv({"num_agents": N, "sensor_range": 2, "steps_per_episode": 24, "lifelong_mapf": True, "seed": 11,
                          "grid": _grid()}, B, DEV)
    env.reset()
    return env


def _cte_env():
    from dl_reference_models_b200.single_agent import BatchedCteEnv

    env = BatchedCteEnv({"grid": _grid(), "num_agents": N, "steps_per_episode": 24, "seed": 11}, B, DEV)
    env.reset()
    return env


def _family(name):
    """(policy, collector, learner, hand-loop kind, per_agent, learner keywords) of one module family."""
    from dl_reference_models_b200.cte_rollout import (CteActionMaskPolicy, CteRecurrentPolicy, FusedCteCollector,
                                                      FusedRecurrentCteCollector)
    from dl_reference_models_b200.recurrent import (FusedRecurrentCollector, PerAgentRecurrentPolicy,
                                                    RecurrentActionMaskPolicy)
    from dl_reference_models_b200.rollout import ActionMaskPolicy, FusedCollector, PerAgentActionMaskPolicy

    torch.manual_seed(0)
    if name.startswith("cte"):
        env = _cte_env()
        cells = env.R * env.C
        if name == "cte_mlp":
            pol = CteActionMaskPolicy(cells, N).to(DEV)
            return pol, FusedCteCollector(env, pk.FusedCtePolicy(pol, env), T), impala.impala_update_cte, "cte", False, {}
        pol = CteRecurrentPolicy(cells, N).to(DEV)
        return (pol, FusedRecurrentCteCollector(env, pk.FusedCteRecurrentPolicy(pol, env), T, max_seq_len=L),
                impala.impala_update_cte_recurrent, "cte_lstm", False, {"max_seq_len": L})
    env = _mapf_env()
    F = env.flat_obs_dim(include_action_mask=False)
    per_agent = name.startswith("per_agent")
    if name.endswith("mlp"):
        pol = (PerAgentActionMaskPolicy(N, F) if per_agent else ActionMaskPolicy(F)).to(DEV)
        return pol, FusedCollector(env, pk.FusedPolicy(pol, env), T, compact=True), impala.impala_update, "mlp", per_agent, {}
    pol = (PerAgentRecurrentPolicy(N, F) if per_agent else RecurrentActionMaskPolicy(F)).to(DEV)
    return (pol, FusedRecurrentCollector(env, pk.FusedRecurrentPolicy(pol, env), T, L), impala.impala_update_recurrent,
            "lstm", per_agent, {"max_seq_len": L})


FAMILIES = ["mlp", "per_agent_mlp", "lstm", "per_agent_lstm", "cte_mlp", "cte_lstm"]


@pytest.mark.parametrize("name", FAMILIES)
def test_learner_on_a_fused_collect_equals_the_loop_by_hand(name):
    pol, collector, update, kind, per_agent, kw = _family(name)
    batch = collector.collect()
    ref = copy.deepcopy(pol)
    # eps 1e-6: an Adam step of a gradient element at rounding-noise size stays far below the tolerance
    opt, ropt = (torch.optim.Adam(m.parameters(), lr=1e-3, eps=1e-6) for m in (pol, ref))
    stats = update(pol, opt, batch, max_minibatches=2, generator=torch.Generator(device=DEV).manual_seed(4), **HP, **kw)
    impala_loops.hand_update(kind, ref, ropt, batch, per_agent=per_agent, generator=torch.Generator(device=DEV).manual_seed(4),
                             max_minibatches=2, L=kw.get("max_seq_len", 32), **HP)
    assert all(math.isfinite(x) for x in stats.values())
    for (pname, p), q in zip(pol.named_parameters(), ref.parameters()):
        torch.testing.assert_close(p, q, rtol=1e-4, atol=1e-4, msg=pname)


@pytest.mark.parametrize("name", FAMILIES)
def test_collect_update_refresh_collect_cycle(name):
    pol, collector, update, _, _, kw = _family(name)
    opt = torch.optim.Adam(pol.parameters(), lr=5e-4)
    before = [p.detach().clone() for p in pol.parameters()]
    for _ in range(2):
        batch = collector.collect()
        stats = update(pol, opt, batch, **kw)   # the defaults: one epoch over every column
        assert stats and all(math.isfinite(x) for x in stats.values()), stats
        collector.fused.refresh()
    batch = collector.collect()
    assert torch.isfinite(batch.logp).all() and torch.isfinite(batch.values).all()
    assert any(not torch.equal(a, p) for a, p in zip(before, pol.parameters()))
