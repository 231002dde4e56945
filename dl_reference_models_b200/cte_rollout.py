"""CTE training: a centralised policy over the single-agent view (:class:`single_agent.BatchedCteEnv`), rolled out on
the device and trained with PPO.

The reference's third execution mode (``training_execution_mode == "CTE"`` in ``src/agents/ppo.py``) plays every agent
with ONE policy that sees the whole grid and emits the joint ``MultiDiscrete([5] * N)`` action:

* :class:`CteActionMaskPolicy` -- the model, a plain ``nn.Module``.  It restates ``models/action_mask_model_single.py``
  as SURVEY §2 row 7 records it (the flat observation split into the grid features and the trailing 5N mask); that
  source is not part of this tree, so the shape below is this restatement, not a copy: the R*C grid codes as float ->
  Linear(R*C, 64)-ReLU-Linear(64, 64)-ReLU -> Linear(64, 5N) logits and Linear(64, 1) value, masked with
  ``action_mask_model.py``'s ``logits + clamp(log(mask + 1e-6), FLOAT_MIN)`` element by element.  The action
  distribution is RLlib's multi-categorical: N independent 5-way categoricals, whose joint log-probability and entropy
  are the sums of the agents' (:func:`joint_logp_entropy`);
* :func:`collect_cte` -- the plain PyTorch rollout loop (the reference of the tests);
* :class:`FusedCteCollector` -- the same rollout as two launches per env step (``mapf_cte_policy_act`` +
  ``mapf_cte_step``) plus the env's masked auto-reset, into a compact :class:`CteBatch`;
* :func:`ppo_update_cte` -- PPO on the joint action with :func:`rollout.ppo_update`'s hyper-parameters.

``python -m dl_reference_models_b200.cte_rollout`` prints the env-only, :func:`collect_cte` and
:class:`FusedCteCollector` throughputs as one JSON line.
"""
from __future__ import annotations

import ctypes as C
import time
from dataclasses import dataclass

import torch
from torch import nn

from . import _native as nat
from .rollout import FLOAT_MIN, draw_permutation, gae, normalize_advantages, ppo_objective, sample_categorical


class CteActionMaskPolicy(nn.Module):
    """The centralised CTE policy: ``forward(grid, mask)`` takes the grid codes ([..., R*C] or [..., R, C], any dtype,
    e.g. the env's uint8 ``obs_grid`` rows) and the [..., 5N] action mask and returns the masked logits [..., N, 5] and
    the value [...]."""

    def __init__(self, cells: int, num_agents: int, hiddens=(64, 64), no_masking: bool = False):
        super().__init__()
        self.cells, self.num_agents = int(cells), int(num_agents)
        self.hiddens, self.no_masking = tuple(int(h) for h in hiddens), bool(no_masking)
        layers, last = [], self.cells
        for h in self.hiddens:
            layers += [nn.Linear(last, h), nn.ReLU()]
            last = h
        self.trunk = nn.Sequential(*layers) if layers else nn.Identity()
        self.logits = nn.Linear(last, 5 * self.num_agents)
        self.value = nn.Linear(last, 1)

    def forward(self, grid: torch.Tensor, action_mask: torch.Tensor):
        lead = action_mask.shape[:-1]
        z = self.trunk(grid.reshape(*lead, self.cells).float())
        logits = self.logits(z)
        value = self.value(z).squeeze(-1)
        if not self.no_masking:
            logits = logits + torch.clamp(torch.log(action_mask.to(logits.dtype) + 1e-6), min=FLOAT_MIN)
        return logits.reshape(*lead, self.num_agents, 5), value


def joint_logp_entropy(logits: torch.Tensor, actions: torch.Tensor):
    """Multi-categorical log-probability of the joint ``actions`` [..., N] and entropy under ``logits`` [..., N, 5]: the
    sums over the N independent categoricals."""
    dist = torch.distributions.Categorical(logits=logits)
    return dist.log_prob(actions).sum(-1), dist.entropy().sum(-1)


@dataclass
class CteBatch:
    """A CTE rollout kept the way the env emits it: R*C + 5N bytes of observation per env-step.  The observation
    tensors hold T + 1 rows (row T: the observation after the last step)."""
    grid: torch.Tensor        # [T+1,B,R*C] uint8 grid codes
    masks: torch.Tensor       # [T+1,B,5N] int8
    actions: torch.Tensor     # [T,B,N] int64 joint actions
    logp: torch.Tensor        # [T,B] joint log-probabilities
    values: torch.Tensor      # [T,B]
    rewards: torch.Tensor     # [T,B] float32
    dones: torch.Tensor       # [T,B] bool (episode ended at this step; the env auto-reset)
    last_value: torch.Tensor  # [B] bootstrap value of row T


@torch.no_grad()
def collect_cte(env, policy: CteActionMaskPolicy, steps: int) -> CteBatch:
    """T steps of ``policy -> one draw per agent -> BatchedCteEnv.step(auto_reset=True)`` in plain PyTorch, from the
    env's current observation."""
    B, N, T, cells, dev = env.B, env.N, int(steps), env.R * env.C, env.device
    grid = torch.empty((T + 1, B, cells), dtype=torch.uint8, device=dev)
    masks = torch.empty((T + 1, B, 5 * N), dtype=torch.int8, device=dev)
    actions = torch.empty((T, B, N), dtype=torch.int64, device=dev)
    logp, values, rewards = (torch.empty((T, B), device=dev) for _ in range(3))
    dones = torch.empty((T, B), dtype=torch.bool, device=dev)
    for t in range(T):
        grid[t].copy_(env.obs_grid.view(B, cells))
        masks[t].copy_(env.action_mask)
        lg, v = policy(grid[t], masks[t])
        a, lp = sample_categorical(lg)
        actions[t], logp[t], values[t] = a, lp.sum(-1), v
        env.step(a.to(torch.int8), auto_reset=True)
        rewards[t].copy_(env.reward)
        dones[t] = (env.terminated | env.truncated).bool()
    grid[T].copy_(env.obs_grid.view(B, cells))
    masks[T].copy_(env.action_mask)
    _, last_value = policy(grid[T], masks[T])
    return CteBatch(grid, masks, actions, logp, values, rewards, dones, last_value)


class FusedCteCollector:
    """T-step CTE rollouts with the policy kernel (:class:`policy_kernels.FusedCtePolicy`) and the env step as the
    only launches of a step, plus the env's masked auto-reset.  The env step of step t writes its grid codes and masks
    straight into row t + 1 of the [T+1, ...] buffers, from which the policy launch of step t + 1 reads; the float32
    ``flat_obs`` output is switched off during a collect and the rewards land in a float64 [T,B] buffer (the kernel's
    type), converted to float32 once per collect.  Argument blocks are built once here.  After :meth:`collect` the
    env's ``obs_grid``, ``action_mask``, ``flat_obs``, ``reward``, ``terminated`` and ``truncated`` show the last step
    again, as if it had been stepped by hand; its own argument block is not touched.  The buffers are reused: the
    :class:`CteBatch` of one collect is overwritten by the next."""

    def __init__(self, env, fused, steps: int):
        self.env, self.fused, self.T = env, fused, int(steps)
        B, N, T, cells, dev = env.B, env.N, self.T, env.R * env.C, env.device
        self._lib = nat.lib()
        self.grid = torch.empty((T + 1, B, cells), dtype=torch.uint8, device=dev)
        self.masks = torch.empty((T + 1, B, 5 * N), dtype=torch.int8, device=dev)
        self.actions = torch.empty((T, B, N), dtype=torch.int64, device=dev)
        self.logp, self.values, self.rewards = (torch.empty((T, B), device=dev) for _ in range(3))
        self.rewards64 = torch.empty((T, B), dtype=torch.float64, device=dev)
        self.term = torch.empty((T, B), dtype=torch.uint8, device=dev)
        self.trunc = torch.empty((T, B), dtype=torch.uint8, device=dev)
        self.last_value = torch.empty(B, device=dev)
        self._pargs = [fused.args(self.grid[t], self.masks[t], actions=fused.actions, actions64=self.actions[t],
                                  logp=self.logp[t], value=self.values[t]) for t in range(T)]
        self._pargs.append(fused.args(self.grid[T], self.masks[T], value=self.last_value))   # bootstrap value

        def step_args(t):   # the env's block with the outputs of step t redirected into the rollout's rows
            a = nat.MapfCteArgs.from_buffer_copy(env._args)
            a.actions, a.obs_grid, a.action_mask = fused.actions.data_ptr(), self.grid[t + 1].data_ptr(), self.masks[t + 1].data_ptr()
            a.flat_obs, a.reset_mask = None, None
            a.reward, a.terminated, a.truncated = self.rewards64[t].data_ptr(), self.term[t].data_ptr(), self.trunc[t].data_ptr()
            return a

        self._sargs = [step_args(t) for t in range(T)]

    @torch.no_grad()
    def collect(self) -> CteBatch:
        """Roll T steps from the env's current observation (its ``obs_grid`` / ``action_mask``)."""
        env, fused, lib, T = self.env, self.fused, self._lib, self.T
        B, cells = env.B, env.R * env.C
        stream = env._stream()
        self.grid[0].copy_(env.obs_grid.view(B, cells))
        self.masks[0].copy_(env.action_mask)
        for t in range(T):
            fused.counter += 1
            a = self._pargs[t]
            a.counter = fused.counter
            nat.check(lib.mapf_cte_policy_act(C.byref(a), stream))
            nat.check(lib.mapf_cte_step(C.byref(self._sargs[t]), stream))
            m = self.term[t] | self.trunc[t]   # BatchedCteEnv.step(auto_reset=True)'s reset, into row t + 1
            if not env.deterministic:
                env._draw(m)
            env._reset_launch(m, self._sargs[t])
        fused.counter += 1
        a = self._pargs[T]
        a.counter = fused.counter
        nat.check(lib.mapf_cte_policy_act(C.byref(a), stream))
        self.rewards.copy_(self.rewards64)
        env.obs_grid.view(B, cells).copy_(self.grid[T])
        env.action_mask.copy_(self.masks[T])
        env.flat_obs[:, :cells].copy_(self.grid[T])
        env.flat_obs[:, cells:].copy_(self.masks[T])
        env.reward.copy_(self.rewards64[T - 1])
        env.terminated.copy_(self.term[T - 1])
        env.truncated.copy_(self.trunc[T - 1])
        return CteBatch(self.grid, self.masks, self.actions, self.logp, self.values, self.rewards,
                        (self.term | self.trunc).bool(), self.last_value)


def ppo_update_cte(policy: CteActionMaskPolicy, optimizer, batch: CteBatch, *, clip: float = 0.05, vf_coeff: float = 0.5,
                   entropy_coeff: float = 0.001, epochs: int = 12, minibatch: int = 1024, gamma: float = 0.99,
                   lam: float = 0.95, max_minibatches: int | None = None, generator: torch.Generator | None = None) -> dict:
    """PPO epochs over a :class:`CteBatch` with :func:`rollout.ppo_update`'s hyper-parameters and keywords.  GAE runs
    over the scalar reward (the ``mapf_gae`` scan with N = 1 for a device batch; :func:`rollout.gae`, the same
    recurrence, for a CPU one); advantages are normalised over the whole batch; a minibatch is ``minibatch`` env-steps
    of one permutation per epoch (``generator`` draws it); the loss is :func:`rollout.ppo_objective` on the joint
    log-probability and the summed entropy."""
    T, B = batch.rewards.shape
    args = (batch.rewards.unsqueeze(-1), batch.values.unsqueeze(-1), batch.dones, batch.last_value.unsqueeze(-1), gamma, lam)
    if batch.rewards.is_cuda:
        from .policy_kernels import gae as gae_kernel

        adv, ret = gae_kernel(*args)
    else:
        adv, ret = gae(*args)
    adv = normalize_advantages(adv, False).reshape(-1)
    ret = ret.reshape(-1)
    grid = batch.grid[:T].reshape(T * B, -1)
    masks = batch.masks[:T].reshape(T * B, -1)
    acts, old_logp = batch.actions.reshape(T * B, -1), batch.logp.reshape(-1)
    n = T * B
    stats, done_mb = {}, 0
    for _ in range(epochs):
        perm = draw_permutation(n, acts.device, generator)
        for i in range(0, n, minibatch):
            idx = perm[i:i + minibatch]
            lg, v = policy(grid[idx], masks[idx])
            lp, ent = joint_logp_entropy(lg, acts[idx])
            loss, stats = ppo_objective(lp, ent, v, old_logp[idx], adv[idx], ret[idx], clip=clip, vf_coeff=vf_coeff,
                                        entropy_coeff=entropy_coeff)
            optimizer.zero_grad(set_to_none=True)
            loss.backward()
            optimizer.step()
            done_mb += 1
            if max_minibatches is not None and done_mb >= max_minibatches:
                return stats
    return stats


def benchmark(num_envs: int = 65536, num_agents: int = 16, steps: int = 64, device: str = "cuda:0") -> dict:
    """Env-steps/s and agent-steps/s of the CTE env alone (fixed random joint actions), :func:`collect_cte` and
    :class:`FusedCteCollector` on a 32x32 map with 30 % obstacles, 256 steps per episode, T = ``steps``."""
    from . import maps
    from .policy_kernels import FusedCtePolicy
    from .single_agent import BatchedCteEnv

    cfg = {"grid": maps.random_obstacle_grid(32, 32, 0.30, 2026, min_free=32), "num_agents": num_agents,
           "steps_per_episode": 256, "seed": 999}
    env = BatchedCteEnv(cfg, num_envs, device)
    env.reset()
    torch.manual_seed(0)
    policy = CteActionMaskPolicy(env.R * env.C, env.N).to(env.device)
    acts = torch.randint(0, 5, (env.B, env.N), dtype=torch.int8, device=env.device)

    def timed(fn):
        fn()   # warm-up
        torch.cuda.synchronize(env.device)
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize(env.device)
        return time.perf_counter() - t0

    def env_only():
        for _ in range(steps):
            env.step(acts, auto_reset=True)

    res = {"envs": num_envs, "agents": env.N, "steps": steps, "map": [env.R, env.C]}
    collector = FusedCteCollector(env, FusedCtePolicy(policy, env), steps)
    for name, fn in (("env_only", env_only), ("collect_cte", lambda: collect_cte(env, policy, steps)),
                     ("fused_cte_collector", collector.collect)):
        s = timed(fn)
        res[f"{name}_env_steps_per_s"] = num_envs * steps / s
        res[f"{name}_agent_steps_per_s"] = num_envs * env.N * steps / s
    return res


if __name__ == "__main__":
    import json
    import subprocess

    from dl_reference_models_b200 import cte_rollout   # the package's classes, not this __main__ copy's

    r = cte_rollout.benchmark()
    try:
        r["gpu"] = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                                  capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as exc:
        r["gpu"] = f"nvidia-smi not readable: {exc}"
    print(json.dumps(r))
