"""IMPALA learners (V-trace off-policy correction) for every module type the PPO learners train, over the batches the
collectors already produce.

The reference trains with RLlib's PPO, IMPALA and DQN (SURVEY §2 row 6).  This module is the IMPALA side:

* :func:`vtrace` -- the V-trace targets (Espeholt et al. 2018; RLlib's ``vtrace_torch`` recurrence with c_bar fixed at
  1) in plain PyTorch, f32 or f64: the tests' reference and the learners' path for CPU batches.  CUDA batches go
  through the ``mapf_vtrace`` scan (:func:`policy_kernels.vtrace`), which gathers the batch-side inputs itself;
* :func:`impala_objective` -- RLlib's IMPALA loss: ``-mean(logp * pg_adv) + vf_coeff * 0.5 * mean((v - vs)^2) -
  entropy_coeff * mean(entropy)``, no advantage normalisation;
* four learners, one per PPO learner: :func:`impala_update` (:class:`rollout.ActionMaskPolicy` /
  :class:`rollout.PerAgentActionMaskPolicy` on a :class:`rollout.Batch` / :class:`rollout.CompactBatch`),
  :func:`impala_update_recurrent` (:class:`recurrent.RecurrentActionMaskPolicy` /
  :class:`recurrent.PerAgentRecurrentPolicy` on a :class:`recurrent.CompactRollout`), :func:`impala_update_cte`
  (:class:`cte_rollout.CteActionMaskPolicy` on a :class:`cte_rollout.CteBatch`) and
  :func:`impala_update_cte_recurrent` (:class:`cte_rollout.CteRecurrentPolicy` on a
  :class:`cte_rollout.CteRecurrentBatch`).

A minibatch is whole time columns: ``max(1, minibatch // T)`` series of all T steps, drawn from one permutation per
epoch.  Per SGD step the learner recomputes the logits and values of those columns with the current module, runs
V-trace on the detached target log-probabilities and values, with ``batch.last_value`` (the actor's value of the
observation after the last step) as the bootstrap, takes the loss's gradient, averages it over the ranks when
``world_size > 1``, clips it by global norm and steps the optimizer.

Defaults: gamma 0.99 is the reference's (``src/agents/ppo.py``).  The other defaults (clip_rho_threshold 1.0,
clip_pg_rho_threshold 1.0, vf_loss_coeff 0.5, entropy_coeff 0.01, grad_clip 40.0) are those of RLlib's
``IMPALAConfig``: the reference's own ``impala.py`` overrides are not recorded anywhere in this tree.

``python -m dl_reference_models_b200.impala`` prints the learners' minibatches/s and the V-trace time per minibatch
(kernel against :func:`vtrace`) as one JSON line.
"""
from __future__ import annotations

import torch

from .cte_rollout import joint_logp_entropy
from .recurrent import PerAgentRecurrentPolicy, allreduce_gradients, features_from_channels
from .rollout import CompactBatch, PerAgentActionMaskPolicy, draw_permutation, per_agent_minibatches


@torch.no_grad()
def vtrace(target_logp, behaviour_logp, values, rewards, dones, bootstrap_value, *, columns=None, gamma: float = 0.99,
           clip_rho: float = 1.0, clip_pg_rho: float = 1.0):
    """V-trace targets (vs, pg_advantages) [T,M] in PyTorch, with :func:`policy_kernels.vtrace`'s arguments:
    ``rewards`` / ``behaviour_logp`` [T,B,N] or [T,B], ``dones`` [T,B] (episode ended at the step: the bootstrap is
    cut), ``bootstrap_value`` [B,N] or [B], ``target_logp`` / ``values`` [T,M] of the batch columns ``columns`` (flat
    index b * N + n; None: all of them).  Computed in ``values``' dtype, in the order of the recurrence::

        rho_t = exp(pi_t - mu_t); rho_bar_t = min(clip_rho, rho_t); c_t = min(1, rho_t); rho_pg_t = min(clip_pg_rho, rho_t)
        disc_t = gamma * (1 - d_t); delta_t = rho_bar_t * (r_t + disc_t * V_{t+1} - V_t)       (V_T = bootstrap)
        acc_t = delta_t + disc_t * c_t * acc_{t+1} (acc_T = 0); vs_t = V_t + acc_t
        pg_adv_t = rho_pg_t * (r_t + disc_t * vs_{t+1} - V_t)                                   (vs_T = bootstrap)
    """
    T, B = rewards.shape[:2]
    dt = values.dtype
    r, mu, boot = rewards.reshape(T, -1).to(dt), behaviour_logp.reshape(T, -1).to(dt), bootstrap_value.reshape(-1).to(dt)
    d = dones.reshape(T, B).bool().repeat_interleave(r.shape[1] // B, dim=1)
    if columns is not None:
        r, mu, d, boot = r[:, columns], mu[:, columns], d[:, columns], boot[columns]
    rho = torch.exp(target_logp.to(dt) - mu)
    rho_bar, c, rho_pg = torch.clamp(rho, max=clip_rho), torch.clamp(rho, max=1.0), torch.clamp(rho, max=clip_pg_rho)
    disc = gamma * (1 - d.to(dt))
    vs, pg = torch.empty_like(values), torch.empty_like(values)
    acc, v_next, vs_next = torch.zeros_like(boot), boot, boot
    for t in range(T - 1, -1, -1):
        delta = rho_bar[t] * (r[t] + disc[t] * v_next - values[t])
        acc = delta + disc[t] * c[t] * acc
        vs[t] = values[t] + acc
        pg[t] = rho_pg[t] * (r[t] + disc[t] * vs_next - values[t])
        v_next, vs_next = values[t], vs[t]
    return vs, pg


def impala_objective(lp, entropy, v, vs, pg_adv, *, vf_coeff: float, entropy_coeff: float, num_agents: int | None = None):
    """RLlib's IMPALA loss of one minibatch and its stats (the keys of :func:`rollout.ppo_objective`): the policy
    gradient ``-mean(lp * pg_adv)``, plus ``vf_coeff`` times the value loss ``0.5 * mean((v - vs)^2)``, minus
    ``entropy_coeff`` times the mean entropy.  ``num_agents``: the rows are agent-fastest (last dimension, a multiple
    of num_agents) and every mean is taken per agent, then summed over the agents."""
    mean = (lambda x: x.mean()) if num_agents is None else (lambda x: x.reshape(-1, num_agents).mean(0).sum())  # noqa: E731
    policy_loss = -mean(lp * pg_adv)
    vf = 0.5 * mean((v - vs).pow(2))
    ent = mean(entropy)
    loss = policy_loss + vf_coeff * vf - entropy_coeff * ent
    return loss, {"loss": float(loss.detach()), "vf_loss": float(vf.detach()), "entropy": float(ent.detach()),
                  "policy_loss": float(policy_loss.detach())}


def clip_grad_norm_per_agent_(params, max_norm: float, num_agents: int):
    """``torch.nn.utils.clip_grad_norm_`` taken per agent over the agent-j slices of stacked parameters (leading
    dimension num_agents): N independent global-norm clips, one per agent's module."""
    grads = [p.grad for p in params if p.grad is not None]
    if not grads:
        return
    norms = torch.stack([g.reshape(num_agents, -1).norm(dim=1) for g in grads], dim=1).norm(dim=1)   # [N]
    coef = torch.clamp(max_norm / (norms + 1e-6), max=1.0)
    for g in grads:
        g.mul_(coef.view(num_agents, *([1] * (g.dim() - 1))))


def _columns(n_series: int, num_agents: int | None, per_step: int, device, generator):
    """One epoch of minibatch column ids: a permutation of the n_series batch columns in slices of per_step; per
    agent (``num_agents``), per_step of every agent's own columns per slice, agent-fastest (env ids drawn with
    :func:`rollout.per_agent_minibatches`, column = env * N + agent)."""
    if num_agents is None:
        perm = draw_permutation(n_series, device, generator)
        for i in range(0, n_series, per_step):
            yield perm[i:i + per_step]
    else:
        agents = torch.arange(num_agents, device=device)
        for s in per_agent_minibatches(n_series // num_agents, num_agents, per_step, device, generator):
            yield (s * num_agents + agents).reshape(-1)


def _learn(policy, optimizer, batch, evaluate, *, T: int, n_series: int, num_agents: int, per_agent: bool, gamma,
           clip_rho, clip_pg_rho, vf_coeff, entropy_coeff, grad_clip, epochs, minibatch, world_size, group,
           max_minibatches, generator) -> dict:
    """The SGD loop shared by the four learners.  ``evaluate(idx)`` -> (target logp, entropy, value), each [T,M], of
    the batch columns ``idx`` under the current parameters."""
    if batch.rewards.is_cuda:
        from .policy_kernels import vtrace as vtrace_fn
    else:
        vtrace_fn = vtrace
    params = list(policy.parameters())
    per_step = max(1, int(minibatch) // T)
    stats, done_mb = {}, 0
    for _ in range(epochs):
        for idx in _columns(n_series, num_agents if per_agent else None, per_step, batch.rewards.device, generator):
            lp, ent, v = evaluate(idx)
            vs, pg = vtrace_fn(lp.detach(), batch.logp, v.detach(), batch.rewards, batch.dones, batch.last_value,
                               columns=idx, gamma=gamma, clip_rho=clip_rho, clip_pg_rho=clip_pg_rho)
            loss, stats = impala_objective(lp, ent, v, vs, pg, vf_coeff=vf_coeff, entropy_coeff=entropy_coeff,
                                           num_agents=num_agents if per_agent else None)
            optimizer.zero_grad(set_to_none=True)
            loss.backward()
            allreduce_gradients(policy, world_size, group)
            if grad_clip is not None:
                if per_agent:
                    clip_grad_norm_per_agent_(params, grad_clip, num_agents)
                else:
                    torch.nn.utils.clip_grad_norm_(params, grad_clip)
            optimizer.step()
            done_mb += 1
            if max_minibatches is not None and done_mb >= max_minibatches:
                return stats
    return stats


def _check_agents(policy, per_agent: bool, N: int):
    if per_agent and policy.num_agents != N:
        raise ValueError(f"the policy has {policy.num_agents} agents, the batch {N}")


def impala_update(policy, optimizer, batch, *, gamma: float = 0.99, clip_rho: float = 1.0, clip_pg_rho: float = 1.0,
                  vf_coeff: float = 0.5, entropy_coeff: float = 0.01, grad_clip: float | None = 40.0, epochs: int = 1,
                  minibatch: int = 1024, world_size: int = 1, group=None, max_minibatches: int | None = None,
                  generator: torch.Generator | None = None) -> dict:
    """IMPALA epochs over a :class:`rollout.Batch` / :class:`rollout.CompactBatch` for an
    :class:`rollout.ActionMaskPolicy` or a :class:`rollout.PerAgentActionMaskPolicy`.  A column is one (env, agent)
    series of T steps; a per-agent module is N independent learners in lockstep: ``minibatch // T`` columns of every
    agent per step (agent-fastest), the loss the sum of the per-agent means, the global-norm clip per agent."""
    T, B, N = batch.actions.shape
    per_agent = isinstance(policy, PerAgentActionMaskPolicy)
    _check_agents(policy, per_agent, N)
    compact = isinstance(batch, CompactBatch)
    steps = torch.arange(T, device=batch.actions.device).unsqueeze(1)

    def evaluate(idx):
        b, n = idx // N, idx % N
        masks = batch.masks[steps, b, n]   # [T,M,5]; indexed, so a padded compact buffer is never copied whole
        feats = batch.features_of((steps * (B * N) + idx).reshape(-1)) if compact else batch.features[steps, b, n]
        lg, v = policy(feats.reshape(T * idx.numel(), -1), masks.reshape(T * idx.numel(), -1))
        dist = torch.distributions.Categorical(logits=lg.reshape(T, idx.numel(), -1))
        return dist.log_prob(batch.actions[steps, b, n]), dist.entropy(), v.reshape(T, -1)

    return _learn(policy, optimizer, batch, evaluate, T=T, n_series=B * N, num_agents=N, per_agent=per_agent,
                  gamma=gamma, clip_rho=clip_rho, clip_pg_rho=clip_pg_rho, vf_coeff=vf_coeff,
                  entropy_coeff=entropy_coeff, grad_clip=grad_clip, epochs=epochs, minibatch=minibatch,
                  world_size=world_size, group=group, max_minibatches=max_minibatches, generator=generator)


def _sequence_index(T: int, L: int, idx: torch.Tensor):
    """Step ids [L, K*M] of the K = T / L chunks of the columns ``idx`` (sequence s = chunk s // M of column s % M,
    so the sequences keep the columns' agent-fastest order) and the chunk ids [K*M]."""
    K, M = T // L, idx.numel()
    t = (torch.arange(K, device=idx.device).view(1, K, 1) * L + torch.arange(L, device=idx.device).view(L, 1, 1))
    return t.expand(L, K, M).reshape(L, K * M), torch.arange(K, device=idx.device).repeat_interleave(M)


def _unchunk(x: torch.Tensor, T: int, L: int, M: int) -> torch.Tensor:
    """[L, K*M, ...] outputs of the chunked sequences -> [T, M, ...]."""
    K = T // L
    return x.reshape(L, K, M, *x.shape[2:]).transpose(0, 1).reshape(T, M, *x.shape[2:])


def impala_update_recurrent(policy, optimizer, batch, *, max_seq_len: int = 32, gamma: float = 0.99,
                            clip_rho: float = 1.0, clip_pg_rho: float = 1.0, vf_coeff: float = 0.5,
                            entropy_coeff: float = 0.01, grad_clip: float | None = 40.0, epochs: int = 1,
                            minibatch: int = 1024, world_size: int = 1, group=None, max_minibatches: int | None = None,
                            generator: torch.Generator | None = None) -> dict:
    """IMPALA epochs over a :class:`recurrent.CompactRollout` for a :class:`recurrent.RecurrentActionMaskPolicy` or a
    :class:`recurrent.PerAgentRecurrentPolicy`: each column's T / ``max_seq_len`` chunks are re-run through
    ``sequence`` from their stored chunk states in one batched call (truncated back-propagation through time) and
    reassembled to [T, M]; per-agent modules as in :func:`impala_update`."""
    L = int(max_seq_len)
    T, B, N = batch.actions.shape
    if T % L:
        raise ValueError(f"the batch's {T} steps are not a multiple of max_seq_len ({L})")
    per_agent = isinstance(policy, PerAgentRecurrentPolicy)
    _check_agents(policy, per_agent, N)

    def evaluate(idx):
        M = idx.numel()
        t, ck = _sequence_index(T, L, idx)
        col = idx.repeat(T // L)   # [K*M]
        b, n = col // N, col % N
        g = lambda x: x[t, b, n]   # noqa: E731  [T,B,N,...] -> [L, K*M, ...]
        feats = features_from_channels(g(batch.local_obs), g(batch.goal_delta), g(batch.blocking_prev))
        lg, v, _ = policy.sequence(feats, g(batch.masks), g(batch.prev_actions), g(batch.prev_rewards),
                                   batch.resets[t, b], (batch.chunk_h[ck, col], batch.chunk_c[ck, col]))
        dist = torch.distributions.Categorical(logits=_unchunk(lg, T, L, M))
        acts = batch.actions[torch.arange(T, device=idx.device).unsqueeze(1), idx // N, idx % N]
        return dist.log_prob(acts), dist.entropy(), _unchunk(v, T, L, M)

    return _learn(policy, optimizer, batch, evaluate, T=T, n_series=B * N, num_agents=N, per_agent=per_agent,
                  gamma=gamma, clip_rho=clip_rho, clip_pg_rho=clip_pg_rho, vf_coeff=vf_coeff,
                  entropy_coeff=entropy_coeff, grad_clip=grad_clip, epochs=epochs, minibatch=minibatch,
                  world_size=world_size, group=group, max_minibatches=max_minibatches, generator=generator)


def impala_update_cte(policy, optimizer, batch, *, gamma: float = 0.99, clip_rho: float = 1.0,
                      clip_pg_rho: float = 1.0, vf_coeff: float = 0.5, entropy_coeff: float = 0.01,
                      grad_clip: float | None = 40.0, epochs: int = 1, minibatch: int = 1024, world_size: int = 1,
                      group=None, max_minibatches: int | None = None, generator: torch.Generator | None = None) -> dict:
    """IMPALA epochs over a :class:`cte_rollout.CteBatch` for a :class:`cte_rollout.CteActionMaskPolicy`: a column is
    one env's T steps; the target log-probability and entropy are the joint ones (:func:`cte_rollout.joint_logp_entropy`)."""
    T, B = batch.rewards.shape

    def evaluate(idx):
        lg, v = policy(batch.grid[:T, idx], batch.masks[:T, idx])
        lp, ent = joint_logp_entropy(lg, batch.actions[:, idx])
        return lp, ent, v

    return _learn(policy, optimizer, batch, evaluate, T=T, n_series=B, num_agents=1, per_agent=False, gamma=gamma,
                  clip_rho=clip_rho, clip_pg_rho=clip_pg_rho, vf_coeff=vf_coeff, entropy_coeff=entropy_coeff,
                  grad_clip=grad_clip, epochs=epochs, minibatch=minibatch, world_size=world_size, group=group,
                  max_minibatches=max_minibatches, generator=generator)


def impala_update_cte_recurrent(policy, optimizer, batch, *, max_seq_len: int = 32, gamma: float = 0.99,
                                clip_rho: float = 1.0, clip_pg_rho: float = 1.0, vf_coeff: float = 0.5,
                                entropy_coeff: float = 0.01, grad_clip: float | None = 40.0, epochs: int = 1,
                                minibatch: int = 1024, world_size: int = 1, group=None,
                                max_minibatches: int | None = None, generator: torch.Generator | None = None) -> dict:
    """IMPALA epochs over a :class:`cte_rollout.CteRecurrentBatch` for a :class:`cte_rollout.CteRecurrentPolicy`: each
    env column's chunks re-run from their stored states as in :func:`impala_update_recurrent`, joint log-probability
    and entropy as in :func:`impala_update_cte`."""
    L = int(max_seq_len)
    T, B = batch.rewards.shape
    if T % L:
        raise ValueError(f"the batch's {T} steps are not a multiple of max_seq_len ({L})")

    def evaluate(idx):
        M = idx.numel()
        t, ck = _sequence_index(T, L, idx)
        col = idx.repeat(T // L)
        g = lambda x: x[t, col]   # noqa: E731  [T,B,...] -> [L, K*M, ...]
        lg, v, _ = policy.sequence(g(batch.grid), g(batch.masks), g(batch.prev_actions), g(batch.prev_rewards),
                                   g(batch.resets), (batch.chunk_h[ck, col], batch.chunk_c[ck, col]))
        lp, ent = joint_logp_entropy(_unchunk(lg, T, L, M), batch.actions[:, idx])
        return lp, ent, _unchunk(v, T, L, M)

    return _learn(policy, optimizer, batch, evaluate, T=T, n_series=B, num_agents=1, per_agent=False, gamma=gamma,
                  clip_rho=clip_rho, clip_pg_rho=clip_pg_rho, vf_coeff=vf_coeff, entropy_coeff=entropy_coeff,
                  grad_clip=grad_clip, epochs=epochs, minibatch=minibatch, world_size=world_size, group=group,
                  max_minibatches=max_minibatches, generator=generator)


def benchmark(num_envs: int = 65536, num_agents: int = 16, steps: int = 64, minibatches: int = 50,
              device: str = "cuda:0") -> dict:
    """C3 (num_envs x 16 agents, 32x32 map with 30 % obstacles, 256 steps per episode), T = ``steps``: per learner
    family (shared MLP, shared LSTM-64, CTE MLP, CTE LSTM-64) one fused collect, then the learner's minibatches/s at
    the defaults (16 columns x 64 steps, Adam lr 5e-4) over ``minibatches`` SGD steps after a warm-up of 5 (host clock
    around work that ends in a device synchronise), and the V-trace time per minibatch on the first minibatch's inputs:
    the ``mapf_vtrace`` kernel against :func:`vtrace` on the device (CUDA events over 200 calls each)."""
    import time

    from . import maps
    from . import policy_kernels as pk
    from .batched_env import BatchedMapfEnv
    from .cte_rollout import CteActionMaskPolicy, CteRecurrentPolicy, FusedCteCollector, FusedRecurrentCteCollector
    from .recurrent import FusedRecurrentCollector, RecurrentActionMaskPolicy
    from .rollout import ActionMaskPolicy, FusedCollector
    from .single_agent import BatchedCteEnv

    grid = maps.random_obstacle_grid(32, 32, 0.30, 2026, min_free=32)

    def event_us(fn, n=200):
        for _ in range(10):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize(device)
        return e0.elapsed_time(e1) / n * 1e3

    def measure(policy, batch, update, **kw):
        opt = torch.optim.Adam(policy.parameters(), lr=5e-4)
        update(policy, opt, batch, max_minibatches=5, **kw)
        torch.cuda.synchronize(device)
        t0 = time.perf_counter()
        update(policy, opt, batch, max_minibatches=minibatches, **kw)
        torch.cuda.synchronize(device)
        mb_s = minibatches / (time.perf_counter() - t0)
        T = batch.rewards.shape[0]
        n_series = batch.rewards[0].numel()
        g = torch.Generator(device=device).manual_seed(0)
        idx = draw_permutation(n_series, device, g)[:max(1, 1024 // T)]
        lp, v = torch.randn(T, idx.numel(), device=device) * 0.1 + batch.logp.reshape(T, -1)[:, idx], batch.values.reshape(T, -1)[:, idx]
        args = (lp, batch.logp, v, batch.rewards, batch.dones, batch.last_value)
        k_vs, k_pg = pk.vtrace(*args, columns=idx)
        t_vs, t_pg = vtrace(*args, columns=idx)
        return {"minibatches_per_s": mb_s, "columns_per_minibatch": idx.numel(),
                "vtrace_kernel_us": event_us(lambda: pk.vtrace(*args, columns=idx)),
                "vtrace_torch_us": event_us(lambda: vtrace(*args, columns=idx), 50),
                "kernel_vs_torch_max_abs_diff": max(float((k_vs - t_vs).abs().max()), float((k_pg - t_pg).abs().max()))}

    res = {"envs": num_envs, "agents": num_agents, "steps": steps, "map": [32, 32]}
    cfg = {"num_agents": num_agents, "sensor_range": 2, "steps_per_episode": 256, "lifelong_mapf": True, "seed": 999,
           "grid": grid}
    env = BatchedMapfEnv(cfg, num_envs, device)
    env.reset()
    F = env.flat_obs_dim(include_action_mask=False)
    torch.manual_seed(0)
    pol = ActionMaskPolicy(F).to(env.device)
    col = FusedCollector(env, pk.FusedPolicy(pol, env), steps, compact=True)
    res["shared_mlp"] = measure(pol, col.collect(), impala_update)
    del col
    rpol = RecurrentActionMaskPolicy(F).to(env.device)
    rcol = FusedRecurrentCollector(env, pk.FusedRecurrentPolicy(rpol, env), steps, 32)
    res["shared_lstm"] = measure(rpol, rcol.collect(), impala_update_recurrent)
    del rcol
    env.close()
    del env
    torch.cuda.empty_cache()
    cenv = BatchedCteEnv({"grid": grid, "num_agents": num_agents, "steps_per_episode": 256, "seed": 999}, num_envs, device)
    cenv.reset()
    cells = cenv.R * cenv.C
    cpol = CteActionMaskPolicy(cells, num_agents).to(cenv.device)
    ccol = FusedCteCollector(cenv, pk.FusedCtePolicy(cpol, cenv), steps)
    res["cte_mlp"] = measure(cpol, ccol.collect(), impala_update_cte)
    del ccol
    crpol = CteRecurrentPolicy(cells, num_agents).to(cenv.device)
    crcol = FusedRecurrentCteCollector(cenv, pk.FusedCteRecurrentPolicy(crpol, cenv), steps, 32)
    res["cte_lstm"] = measure(crpol, crcol.collect(), impala_update_cte_recurrent)
    return res


if __name__ == "__main__":
    import json
    import subprocess

    from dl_reference_models_b200 import impala   # the package's functions, not this __main__ copy's

    r = impala.benchmark()
    try:
        r["gpu"] = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                                   "-i", "0"], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as exc:
        r["gpu"] = f"nvidia-smi not readable: {exc}"
    print(json.dumps(r))
