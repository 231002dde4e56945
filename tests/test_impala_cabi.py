"""CPU-side checks of IMPALA (no GPU): mapf_vtrace_args' ctypes layout against the header, mapf_vtrace's refusals
before any device work, impala.vtrace against a scalar float64 loop and against GAE with lambda 1 on-policy, the four
learners against the loops written out by hand (tests/impala_loops.py), per-agent learners against N separate modules
with their own optimizers and clips, and two gloo ranks stepping with the clipped mean of their gradients."""
import copy
import ctypes as C
import math
import os
import shutil
import socket
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

from dl_reference_models_b200 import _native as nat
from dl_reference_models_b200 import impala
from dl_reference_models_b200.cte_rollout import CteActionMaskPolicy, CteBatch, CteRecurrentBatch, CteRecurrentPolicy
from dl_reference_models_b200.recurrent import CompactRollout, PerAgentRecurrentPolicy, RecurrentActionMaskPolicy
from dl_reference_models_b200.rollout import ActionMaskPolicy, Batch, CompactBatch, PerAgentActionMaskPolicy, gae

REPO = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(REPO / "tests"))
import impala_loops  # noqa: E402


@pytest.mark.skipif(shutil.which("gcc") is None, reason="needs gcc")
def test_ctypes_structure_matches_the_header_layout(tmp_path):
    cls = nat.MapfVtraceArgs
    fields = [name for name, _ in cls._fields_]
    src = tmp_path / "probe.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "mapf_b200.h"\nint main(void) {\n'
                   '    printf("%zu\\n", sizeof(mapf_vtrace_args));\n'
                   + "".join(f'    printf("%zu\\n", offsetof(mapf_vtrace_args, {f}));\n' for f in fields)
                   + "    return 0;\n}\n")
    exe = tmp_path / "probe"
    subprocess.run(["gcc", "-std=c99", "-I", str(REPO / "include"), "-o", str(exe), str(src)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    assert got == [C.sizeof(cls)] + [getattr(cls, f).offset for f in fields]
    assert "mapf_vtrace" in nat.EXPORTS


def _args(**kw):
    fake = C.c_void_p(16)
    a = nat.MapfVtraceArgs(T=4, num_agents=2, num_columns=6, M=6, gamma=0.99, clip_rho=1.0, clip_pg_rho=1.0)
    for name, typ in a._fields_:
        if typ is C.c_void_p and name != "columns":
            setattr(a, name, fake)
    for k, v in kw.items():
        setattr(a, k, v)
    return a


REFUSALS = ([{k: None} for k in ("rewards", "behaviour_logp", "dones", "bootstrap_value", "target_logp", "values", "vs",
                                 "pg_advantages")]
            + [{"T": 0}, {"T": -1}, {"M": 0}, {"M": -5, "columns": 16}, {"num_agents": 0}, {"num_agents": -2},
               {"num_columns": 7, "M": 7}, {"num_columns": 0, "M": 0}, {"M": 5}, {"M": 7},
               {"gamma": -0.01}, {"gamma": 1.01}, {"gamma": math.nan}]
            + [{k: v} for k in ("clip_rho", "clip_pg_rho") for v in (0.0, -1.0, math.inf, math.nan)]
            + [{"reserved": 1}, {"reserved": -1}])


@pytest.mark.parametrize("kw", REFUSALS, ids=[str(k) for k in REFUSALS])
def test_mapf_vtrace_refuses_before_any_device_work(kw):
    L = nat.lib()
    assert L.mapf_vtrace(C.byref(_args(**kw)), None) == nat.ERR_INVALID_ARG
    assert b"vtrace" in L.mapf_last_error()
    assert L.mapf_vtrace(None, None) == nat.ERR_INVALID_ARG


def _vtrace_loop(pi, mu, v, r, d, boot, gamma, clip_rho, clip_pg_rho):
    """The recurrence for one column, scalar float64."""
    T = len(r)
    vs, pg = [0.0] * T, [0.0] * T
    acc, v_next, vs_next = 0.0, boot, boot
    for t in range(T - 1, -1, -1):
        rho = math.exp(pi[t] - mu[t])
        disc = gamma * (1.0 - d[t])
        delta = min(clip_rho, rho) * (r[t] + disc * v_next - v[t])
        acc = delta + disc * min(1.0, rho) * acc
        vs[t] = v[t] + acc
        pg[t] = min(clip_pg_rho, rho) * (r[t] + disc * vs_next - v[t])
        v_next, vs_next = v[t], vs[t]
    return vs, pg


def _vtrace_inputs(T, B, N, g, log_rho_max=30.0, dtype=torch.float64):
    mu = torch.randn(T, B, N, generator=g, dtype=dtype)
    r = torch.randn(T, B, N, generator=g, dtype=dtype)
    d = torch.rand(T, B, generator=g) < 0.2
    boot = torch.randn(B, N, generator=g, dtype=dtype)
    return mu, r, d, boot


@pytest.mark.parametrize("N", [1, 3])
@pytest.mark.parametrize("gathered", [False, True])
def test_vtrace_equals_a_scalar_float64_loop(N, gathered):
    g = torch.Generator().manual_seed(N + 10 * gathered)
    T, B = 13, 5
    mu, r, d, boot = _vtrace_inputs(T, B, N, g)
    cols = torch.tensor([3, 0, 3, B * N - 1, 1]) if gathered else None
    M = B * N if cols is None else cols.numel()
    ids = list(range(M)) if cols is None else cols.tolist()
    log_rho = (torch.rand(T, M, generator=g, dtype=torch.float64) * 2 - 1) * 30.0   # |log rho| up to 30, both signs
    pi = mu.reshape(T, -1)[:, ids] + log_rho
    v = torch.randn(T, M, generator=g, dtype=torch.float64)
    gamma, clip_rho, clip_pg_rho = 0.97, 1.3, 0.8
    vs, pg = impala.vtrace(pi, mu, v, r, d, boot, columns=cols, gamma=gamma, clip_rho=clip_rho, clip_pg_rho=clip_pg_rho)
    assert vs.dtype == torch.float64 and vs.shape == (T, M)
    for m, col in enumerate(ids):
        dd = d[:, col // N].double().tolist()
        evs, epg = _vtrace_loop(pi[:, m].tolist(), mu.reshape(T, -1)[:, col].tolist(), v[:, m].tolist(),
                                r.reshape(T, -1)[:, col].tolist(), dd, float(boot.reshape(-1)[col]), gamma, clip_rho,
                                clip_pg_rho)
        np.testing.assert_allclose(vs[:, m].numpy(), evs, rtol=1e-12, atol=1e-12)
        np.testing.assert_allclose(pg[:, m].numpy(), epg, rtol=1e-12, atol=1e-12)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_on_policy_vtrace_is_gae_with_lambda_one(dtype):
    g = torch.Generator().manual_seed(3)
    T, B, N = 17, 6, 4
    mu, r, d, boot = _vtrace_inputs(T, B, N, g, dtype=dtype)
    v = torch.randn(T, B, N, generator=g, dtype=dtype)
    vs, pg = impala.vtrace(mu.reshape(T, -1), mu, v.reshape(T, -1), r, d, boot, gamma=0.99)
    adv, ret = gae(r, v, d, boot, gamma=0.99, lam=1.0)
    np.testing.assert_allclose(vs.numpy(), ret.reshape(T, -1).numpy(), rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(pg.numpy(), adv.reshape(T, -1).numpy(), rtol=1e-5, atol=1e-5)


def test_impala_objective_is_rllibs_loss():
    g = torch.Generator().manual_seed(0)
    lp, ent, v, vs, pg = (torch.randn(8, 6, generator=g) for _ in range(5))
    loss, stats = impala.impala_objective(lp, ent, v, vs, pg, vf_coeff=0.5, entropy_coeff=0.01)
    want = -(lp * pg).mean() + 0.5 * 0.5 * ((v - vs) ** 2).mean() - 0.01 * ent.mean()
    assert float(loss) == pytest.approx(float(want), rel=1e-6)
    assert set(stats) == {"loss", "vf_loss", "entropy", "policy_loss"}
    loss3, _ = impala.impala_objective(lp, ent, v, vs, pg, vf_coeff=0.5, entropy_coeff=0.01, num_agents=3)
    per = [impala.impala_objective(x[:, j::3], e[:, j::3], w[:, j::3], s[:, j::3], p[:, j::3], vf_coeff=0.5,
                                   entropy_coeff=0.01)[0] for j in range(3) for x, e, w, s, p in [(lp, ent, v, vs, pg)]]
    assert float(loss3) == pytest.approx(float(sum(per)), rel=1e-6)


# ---- synthetic batches of every type (CPU) -------------------------------------------------------------------------

V, T_, L_ = 3, 8, 4


def _behaviour(g, shape, scale=0.3):
    return -1.6 + scale * torch.randn(*shape, generator=g)


def _masks(g, shape, actions):
    m = (torch.rand(*shape, 5, generator=g) < 0.8).to(torch.int8)
    m.scatter_(-1, actions.unsqueeze(-1), 1)   # the taken action is always allowed
    return m


def mlp_batch(B, N, g, compact, reward_scale=None):
    T = T_
    a = torch.randint(0, 5, (T, B, N), generator=g)
    lo = torch.randint(0, 3, (T + 1, B, N, V, V), generator=g, dtype=torch.uint8)
    gd = torch.randn(T + 1, B, N, 2, generator=g)
    bp = torch.randint(0, 2, (T + 1, B, N), generator=g, dtype=torch.uint8)
    r = torch.randn(T, B, N, generator=g) * (1 if reward_scale is None else reward_scale)
    rest = (_masks(g, (T, B, N), a), a, _behaviour(g, (T, B, N)), torch.randn(T, B, N, generator=g), r,
            torch.rand(T, B, generator=g) < 0.15, torch.randn(B, N, generator=g))
    cb = CompactBatch(lo, gd, bp, *rest)
    return cb if compact else Batch(cb.features, *rest)


def lstm_batch(B, N, g, reward_scale=None):
    T = T_
    a = torch.randint(0, 5, (T, B, N), generator=g)
    resets = torch.rand(T, B, generator=g) < 0.15
    r = torch.randn(T, B, N, generator=g) * (1 if reward_scale is None else reward_scale)
    return CompactRollout(torch.randint(0, 3, (T, B, N, V, V), generator=g, dtype=torch.uint8),
                          torch.randn(T, B, N, 2, generator=g), torch.randint(0, 2, (T, B, N), generator=g, dtype=torch.uint8),
                          _masks(g, (T, B, N), a), a, torch.randint(0, 5, (T, B, N), generator=g),
                          torch.randn(T, B, N, generator=g), resets, _behaviour(g, (T, B, N)),
                          torch.randn(T, B, N, generator=g), r, torch.rand(T, B, generator=g) < 0.15,
                          torch.randn(B, N, generator=g), 0.3 * torch.randn(T // L_, B * N, 64, generator=g),
                          0.3 * torch.randn(T // L_, B * N, 64, generator=g))


def cte_batch(B, N, cells, g, recurrent):
    T = T_
    a = torch.randint(0, 5, (T, B, N), generator=g)
    masks = torch.ones(T + 1, B, 5 * N, dtype=torch.int8)
    masks[:T] = _masks(g, (T, B, N), a).reshape(T, B, 5 * N)
    base = (torch.randint(0, 4, (T + 1, B, cells), generator=g, dtype=torch.uint8), masks, a,
            _behaviour(g, (T, B), 1.0) - 1.6 * (N - 1), torch.randn(T, B, generator=g), torch.randn(T, B, generator=g),
            torch.rand(T, B, generator=g) < 0.15, torch.randn(B, generator=g))
    if not recurrent:
        return CteBatch(*base)
    return CteRecurrentBatch(*base, torch.randint(0, 5, (T, B, N), generator=g), torch.randn(T, B, generator=g),
                             torch.rand(T, B, generator=g) < 0.15, 0.3 * torch.randn(T // L_, B, 64, generator=g),
                             0.3 * torch.randn(T // L_, B, 64, generator=g))


F_ = V * V + 3
FAMILIES = {
    "mlp": (lambda: ActionMaskPolicy(F_), lambda g: mlp_batch(6, 3, g, compact=True), impala.impala_update, {}),
    "mlp_full_batch": (lambda: ActionMaskPolicy(F_), lambda g: mlp_batch(6, 3, g, compact=False), impala.impala_update, {}),
    "per_agent_mlp": (lambda: PerAgentActionMaskPolicy(3, F_), lambda g: mlp_batch(6, 3, g, compact=True),
                      impala.impala_update, {}),
    "lstm": (lambda: RecurrentActionMaskPolicy(F_), lambda g: lstm_batch(6, 3, g), impala.impala_update_recurrent,
             {"max_seq_len": L_}),
    "per_agent_lstm": (lambda: PerAgentRecurrentPolicy(3, F_), lambda g: lstm_batch(6, 3, g),
                       impala.impala_update_recurrent, {"max_seq_len": L_}),
    "cte": (lambda: CteActionMaskPolicy(20, 3), lambda g: cte_batch(9, 3, 20, g, False), impala.impala_update_cte, {}),
    "cte_lstm": (lambda: CteRecurrentPolicy(20, 3), lambda g: cte_batch(9, 3, 20, g, True),
                 impala.impala_update_cte_recurrent, {"max_seq_len": L_}),
}
KIND = {"mlp": "mlp", "mlp_full_batch": "mlp", "per_agent_mlp": "mlp", "lstm": "lstm", "per_agent_lstm": "lstm",
        "cte": "cte", "cte_lstm": "cte_lstm"}


def _counting(opt):
    opt.count = 0
    step = opt.step

    def counted(*a, **k):
        opt.count += 1
        return step(*a, **k)
    opt.step = counted
    return opt


@pytest.mark.parametrize("family", list(FAMILIES))
def test_learner_equals_the_loop_by_hand(family):
    make, make_batch, update, kw = FAMILIES[family]
    torch.manual_seed(0)
    pol = make()
    ref = copy.deepcopy(pol)
    batch = make_batch(torch.Generator().manual_seed(1))
    opt = _counting(torch.optim.Adam(pol.parameters(), lr=1e-3))
    ropt = torch.optim.Adam(ref.parameters(), lr=1e-3)
    hp = dict(minibatch=2 * T_, grad_clip=0.5, gamma=0.95, clip_rho=1.2, clip_pg_rho=0.9, vf_coeff=0.4, entropy_coeff=0.05)
    stats = update(pol, opt, batch, max_minibatches=3, generator=torch.Generator().manual_seed(7), **hp, **kw)
    impala_loops.hand_update(KIND[family], ref, ropt, batch, per_agent=family.startswith("per_agent"),
                             generator=torch.Generator().manual_seed(7), max_minibatches=3, L=kw.get("max_seq_len", 32), **hp)
    assert opt.count == 3   # the batch has more than 3 minibatches: the learner stops at max_minibatches
    assert set(stats) == {"loss", "vf_loss", "entropy", "policy_loss"} and all(math.isfinite(x) for x in stats.values())
    for (name, p), q in zip(pol.named_parameters(), ref.parameters()):
        torch.testing.assert_close(p, q, rtol=1e-5, atol=1e-5, msg=name)


def test_every_epoch_takes_every_column_once(monkeypatch):
    make, make_batch, update, kw = FAMILIES["cte"]
    pol = make()
    batch = make_batch(torch.Generator().manual_seed(1))
    seen = []
    orig = impala.impala_objective

    def spy(lp, *a, **k):
        seen.append(tuple(lp.shape))
        return orig(lp, *a, **k)
    monkeypatch.setattr(impala, "impala_objective", spy)
    update(pol, torch.optim.Adam(pol.parameters()), batch, minibatch=2 * T_, epochs=2,
           generator=torch.Generator().manual_seed(0))
    assert seen == [(T_, 2)] * 4 + [(T_, 1)] + [(T_, 2)] * 4 + [(T_, 1)]   # 9 env columns, 2 per step, 2 epochs


@pytest.mark.parametrize("kind", ["mlp", "lstm"])
def test_per_agent_learner_equals_n_separate_modules(kind):
    N = 3
    scale = torch.tensor([0.01, 1.0, 100.0])   # agent 0 stays under the clip, agent 2 far over it
    g = torch.Generator().manual_seed(5)
    if kind == "mlp":
        batch = mlp_batch(6, N, g, compact=False, reward_scale=scale)
        torch.manual_seed(0)
        pol, update, kw = PerAgentActionMaskPolicy(N, F_), impala.impala_update, {}
    else:
        batch = lstm_batch(6, N, g, reward_scale=scale)
        torch.manual_seed(0)
        pol, update, kw = PerAgentRecurrentPolicy(N, F_), impala.impala_update_recurrent, {"max_seq_len": L_}
    mods = [pol.module(j) for j in range(N)]
    opts = [torch.optim.Adam(m.parameters(), lr=1e-3) for m in mods]
    clip = 1.0
    update(pol, torch.optim.Adam(pol.parameters(), lr=1e-3), batch, minibatch=2 * T_, grad_clip=clip, max_minibatches=2,
           generator=torch.Generator().manual_seed(9), **kw)
    draws = impala_loops.column_draws(batch, True, 2 * T_, torch.Generator().manual_seed(9))[:2]
    norms = []
    for idx in draws:
        for j, (m, o) in enumerate(zip(mods, opts)):
            cols = idx[j::N]   # agent j's columns
            assert bool((cols % N == j).all())
            lp, ent, v = impala_loops.forward(kind, m, batch, cols, L_)
            vs, pg = impala.vtrace(lp.detach(), batch.logp, v.detach(), batch.rewards, batch.dones, batch.last_value,
                                   columns=cols)
            loss = impala_loops.loss_of(lp, ent, v, vs, pg, vf_coeff=0.5, entropy_coeff=0.01)
            o.zero_grad()
            loss.backward()
            norms.append(float(torch.nn.utils.clip_grad_norm_(m.parameters(), clip)))
            o.step()
    assert min(norms) < clip < max(norms), norms   # the clip is active for some agents and not for others
    for j, m in enumerate(mods):
        got = pol.module(j)
        for (name, p), q in zip(got.named_parameters(), m.parameters()):
            torch.testing.assert_close(p, q, rtol=1e-5, atol=1e-5, msg=f"agent {j} {name}")


def _rank_worker(rank, world, port, q):
    import torch.distributed as dist

    sys.path.insert(0, str(REPO))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        torch.manual_seed(0)
        pol = CteActionMaskPolicy(20, 3)
        batch = cte_batch(9, 3, 20, torch.Generator().manual_seed(100 + rank), False)
        impala.impala_update_cte(pol, torch.optim.Adam(pol.parameters(), lr=1e-3), batch, minibatch=2 * T_,
                                 grad_clip=0.05, max_minibatches=1, world_size=world,
                                 generator=torch.Generator().manual_seed(3))
        q.put((rank, [p.detach().numpy().copy() for p in pol.parameters()]))   # numpy: no shared-memory handles
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
    # by hand: both ranks' gradients at the same start, averaged, clipped once, one Adam step
    torch.manual_seed(0)
    pol = CteActionMaskPolicy(20, 3)
    grads = []
    for rank in range(2):
        m = copy.deepcopy(pol)
        batch = cte_batch(9, 3, 20, torch.Generator().manual_seed(100 + rank), False)
        idx = impala_loops.column_draws(batch, False, 2 * T_, torch.Generator().manual_seed(3))[0]
        lp, ent, v = impala_loops.forward("cte", m, batch, idx)
        vs, pg = impala.vtrace(lp.detach(), batch.logp, v.detach(), batch.rewards, batch.dones, batch.last_value, columns=idx)
        impala_loops.loss_of(lp, ent, v, vs, pg, vf_coeff=0.5, entropy_coeff=0.01).backward()
        grads.append([p.grad for p in m.parameters()])
    for p, g0, g1 in zip(pol.parameters(), *grads):
        p.grad = (g0 + g1) / 2
    assert float(torch.nn.utils.clip_grad_norm_(pol.parameters(), 0.05)) > 0.05   # the clip is active
    opt = torch.optim.Adam(pol.parameters(), lr=1e-3)
    opt.step()
    for rank in range(2):
        for p, q_ in zip(pol.parameters(), res[rank]):
            torch.testing.assert_close(torch.from_numpy(q_), p.detach(), rtol=1e-5, atol=1e-5)
