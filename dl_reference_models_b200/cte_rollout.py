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
* :func:`ppo_update_cte` -- PPO on the joint action with :func:`rollout.ppo_update`'s hyper-parameters;
* :class:`CteRecurrentPolicy` -- the same trunk followed by the reference's LSTM cell of 64 (``src/agents/ppo.py:67-75``:
  fed with the previous joint action and the previous reward, ``max_seq_len`` 32, shared value head), with its
  collectors (:class:`RecurrentCteCollector` in plain PyTorch, :class:`FusedRecurrentCteCollector` on the
  ``mapf_cte_lstm_policy_act`` kernels) and :func:`ppo_update_cte_recurrent` (PPO on sequence minibatches).

``python -m dl_reference_models_b200.cte_rollout`` prints the env-only, :func:`collect_cte`,
:class:`FusedCteCollector`, :class:`RecurrentCteCollector` and :class:`FusedRecurrentCteCollector` throughputs as one
JSON line.
"""
from __future__ import annotations

import ctypes as C
import time
from dataclasses import dataclass

import torch
from torch import nn

from . import _native as nat
from .recurrent import allreduce_gradients
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


class CteRecurrentPolicy(nn.Module):
    """The recurrent centralised CTE policy, the reference's PPO model (``src/agents/ppo.py:67-75``) on the
    single-agent view: the grid codes as float -> the ReLU trunk -> ``nn.LSTMCell(64 + 5N + 1, cell)`` fed with [trunk
    output | one-hot of the previous joint action | previous reward] -> 5N logits (masked as
    :class:`CteActionMaskPolicy`'s, returned as [..., N, 5]) and the value, both reading h.  The one-hot of a
    ``MultiDiscrete([5] * N)`` action is the N five-way one-hots concatenated in agent order (RLlib's ``one_hot``)."""

    def __init__(self, cells: int, num_agents: int, hiddens=(64, 64), cell: int = 64, use_prev_action: bool = True,
                 use_prev_reward: bool = True):
        super().__init__()
        self.cells, self.num_agents, self.cell = int(cells), int(num_agents), int(cell)
        self.hiddens = tuple(int(h) for h in hiddens)
        self.use_prev_action, self.use_prev_reward = bool(use_prev_action), bool(use_prev_reward)
        layers, last = [], self.cells
        for h in self.hiddens:
            layers += [nn.Linear(last, h), nn.ReLU()]
            last = h
        self.trunk = nn.Sequential(*layers) if layers else nn.Identity()
        extra = (5 * self.num_agents if self.use_prev_action else 0) + (1 if self.use_prev_reward else 0)
        self.lstm = nn.LSTMCell(last + extra, self.cell)
        self.logits = nn.Linear(self.cell, 5 * self.num_agents)
        self.value = nn.Linear(self.cell, 1)   # vf_share_layers: the value head reads the same LSTM output

    def initial_state(self, n: int, device=None):
        z = torch.zeros((n, self.cell), device=device)
        return z, z.clone()

    def step(self, grid, action_mask, prev_action, prev_reward, state):
        """One time step for a flat batch [M, ...]: ``grid`` [M, R*C] (or [M, R, C]), ``action_mask`` [M, 5N],
        ``prev_action`` [M, N], ``prev_reward`` [M] -> (masked logits [M, N, 5], value [M], new state)."""
        M = action_mask.shape[0]
        x = [self.trunk(grid.reshape(M, self.cells).float())]
        if self.use_prev_action:
            x.append(torch.nn.functional.one_hot(prev_action.long(), 5).reshape(M, 5 * self.num_agents).to(x[0].dtype))
        if self.use_prev_reward:
            x.append(prev_reward.to(x[0].dtype).unsqueeze(-1))
        h, c = self.lstm(torch.cat(x, dim=-1), state)
        logits = self.logits(h) + torch.clamp(torch.log(action_mask.to(h.dtype) + 1e-6), min=FLOAT_MIN)
        return logits.reshape(M, self.num_agents, 5), self.value(h).squeeze(-1), (h, c)

    def sequence(self, grid, action_mask, prev_action, prev_reward, resets, state):
        """[T, M, ...] inputs; ``resets`` [T, M] bool = the step starts a new episode (h, c, the previous action and
        the previous reward are zeroed in front of it).  Returns logits [T, M, N, 5], values [T, M], final state."""
        lg, vs = [], []
        h, c = state
        for t in range(grid.shape[0]):
            keep = ~resets[t]
            h, c = h * keep.to(h.dtype).unsqueeze(-1), c * keep.to(c.dtype).unsqueeze(-1)
            pa = prev_action[t] * keep.to(prev_action.dtype).unsqueeze(-1)
            pr = prev_reward[t] * keep.to(prev_reward.dtype)
            l, v, (h, c) = self.step(grid[t], action_mask[t], pa, pr, (h, c))
            lg.append(l)
            vs.append(v)
        return torch.stack(lg), torch.stack(vs), (h, c)


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


@dataclass
class CteRecurrentBatch(CteBatch):
    """A :class:`CteBatch` of a recurrent policy, plus what the learner needs to re-run its sequences."""
    prev_actions: torch.Tensor   # [T,B,N] int64 joint action of the step before (0 behind a reset)
    prev_rewards: torch.Tensor   # [T,B] float32 reward of the step before (0 behind a reset)
    resets: torch.Tensor         # [T,B] bool: step t is the first of an episode
    chunk_h: torch.Tensor        # [T/L,B,cell] LSTM state at the start of every max_seq_len chunk (after the cut)
    chunk_c: torch.Tensor


class RecurrentCteCollector:
    """T steps of ``CteRecurrentPolicy.step -> one draw per agent -> BatchedCteEnv.step(auto_reset=True)`` in plain
    PyTorch (the reference of the fused collector).  Carries the LSTM state, the previous action / reward and the
    episode-start flags across :meth:`collect` calls; the first collect starts every env's episode."""

    def __init__(self, env, policy: CteRecurrentPolicy, max_seq_len: int = 32):
        self.env, self.policy, self.L = env, policy, int(max_seq_len)
        dev = env.device
        self.state = policy.initial_state(env.B, dev)
        self.prev_action = torch.zeros((env.B, env.N), dtype=torch.int64, device=dev)
        self.prev_reward = torch.zeros(env.B, device=dev)
        self.reset_next = torch.ones(env.B, dtype=torch.bool, device=dev)

    @torch.no_grad()
    def collect(self, steps: int) -> CteRecurrentBatch:
        env, pol, L, T = self.env, self.policy, self.L, int(steps)
        if T % L:
            raise ValueError(f"steps ({T}) must be a multiple of max_seq_len ({L})")
        B, N, cells, dev = env.B, env.N, env.R * env.C, env.device
        z = lambda shape, dt=torch.float32: torch.empty(shape, dtype=dt, device=dev)  # noqa: E731
        r = CteRecurrentBatch(z((T + 1, B, cells), torch.uint8), z((T + 1, B, 5 * N), torch.int8), z((T, B, N), torch.int64),
                              z((T, B)), z((T, B)), z((T, B)), z((T, B), torch.bool), z(B),
                              z((T, B, N), torch.int64), z((T, B)), z((T, B), torch.bool),
                              z((T // L, B, pol.cell)), z((T // L, B, pol.cell)))
        h, c = self.state
        for t in range(T):
            keep = ~self.reset_next
            h, c = h * keep.unsqueeze(-1), c * keep.unsqueeze(-1)
            if t % L == 0:
                r.chunk_h[t // L], r.chunk_c[t // L] = h, c
            pa, pr = self.prev_action * keep.unsqueeze(-1), self.prev_reward * keep
            r.grid[t].copy_(env.obs_grid.view(B, cells))
            r.masks[t].copy_(env.action_mask)
            r.prev_actions[t], r.prev_rewards[t], r.resets[t] = pa, pr, self.reset_next
            lg, v, (h, c) = pol.step(r.grid[t], r.masks[t], pa, pr, (h, c))
            a, lp = sample_categorical(lg)
            r.actions[t], r.logp[t], r.values[t] = a, lp.sum(-1), v
            env.step(a.to(torch.int8), auto_reset=True)
            r.rewards[t].copy_(env.reward)
            r.dones[t] = (env.terminated | env.truncated).bool()
            self.prev_action, self.prev_reward, self.reset_next = a, env.reward.float(), r.dones[t].clone()
        r.grid[T].copy_(env.obs_grid.view(B, cells))
        r.masks[T].copy_(env.action_mask)
        keep = ~self.reset_next   # bootstrap value of row T; the state is not advanced
        _, lv, _ = pol.step(r.grid[T], r.masks[T], self.prev_action * keep.unsqueeze(-1), self.prev_reward * keep,
                            (h * keep.unsqueeze(-1), c * keep.unsqueeze(-1)))
        r.last_value.copy_(lv)
        self.state = (h, c)
        return r


class FusedRecurrentCteCollector:
    """:class:`RecurrentCteCollector` on the device: per step one policy call (:class:`policy_kernels.FusedCteRecurrentPolicy`,
    its two launches), the env step into row t + 1 and the env's masked auto-reset, as :class:`FusedCteCollector`
    does.  The policy call of step t reads the reward (float64, the env's type, no conversion) and the episode ends
    of step t - 1 (the carried ones at t = 0) and advances the LSTM state in place; its actions are the next step's
    previous actions.  Argument blocks are built once here.  The previous actions / rewards, the reset flags and the
    chunk-start states of the :class:`CteRecurrentBatch` are filled with a few vectorised ops per collect.  After
    :meth:`collect` the env's visible outputs show the last step, as :class:`FusedCteCollector` leaves them.  The
    buffers are reused: the batch of one collect is overwritten by the next."""

    def __init__(self, env, fused, steps: int, max_seq_len: int = 32):
        T, L = int(steps), int(max_seq_len)
        if T % L:
            raise ValueError(f"steps ({T}) must be a multiple of max_seq_len ({L})")
        self.env, self.fused, self.T, self.L = env, fused, T, L
        B, N, cells, dev = env.B, env.N, env.R * env.C, env.device
        self._lib = nat.lib()
        z = lambda shape, dt=torch.float32: torch.zeros(shape, dtype=dt, device=dev)  # noqa: E731
        self.grid, self.masks = z((T + 1, B, cells), torch.uint8), z((T + 1, B, 5 * N), torch.int8)
        self.actions, self.prev_actions = z((T, B, N), torch.int64), z((T, B, N), torch.int64)
        self.logp, self.values, self.rewards, self.prev_rewards = z((T, B)), z((T, B)), z((T, B)), z((T, B))
        self.rewards64 = z((T, B), torch.float64)
        self.term, self.trunc = z((T, B), torch.uint8), z((T, B), torch.uint8)
        self.resets = z((T, B), torch.bool)
        self.last_value = z(B)
        self.chunk_h, self.chunk_c = z((T // L, B, 64)), z((T // L, B, 64))
        # carried across collects: state, previous action / reward, episode-start flags (the first collect starts all)
        self.state = (z((B, 64)), z((B, 64)))
        self.act8 = z((B, N), torch.int8)   # this step's actions (to mapf_cte_step) = the next step's previous actions
        self.prev_reward = z(B, torch.float64)
        self.prev_term, self.prev_trunc = torch.ones(B, dtype=torch.uint8, device=dev), z(B, torch.uint8)

        def policy_args(t):
            last = t == T
            pr, pt, ptr = (self.prev_reward, self.prev_term, self.prev_trunc) if t == 0 else \
                (self.rewards64[t - 1], self.term[t - 1], self.trunc[t - 1])
            return fused.args(self.grid[t], self.masks[t], self.state, self.act8, pr, pt, ptr,
                              state_out=None if last else self.state, actions=None if last else self.act8,
                              actions64=None if last else self.actions[t], logp=None if last else self.logp[t],
                              value=self.last_value if last else self.values[t])

        self._pargs = [policy_args(t) for t in range(T + 1)]   # the last one: bootstrap value, state not advanced

        def step_args(t):   # the env's block with the outputs of step t redirected into the rollout's rows
            a = nat.MapfCteArgs.from_buffer_copy(env._args)
            a.actions, a.obs_grid, a.action_mask = self.act8.data_ptr(), self.grid[t + 1].data_ptr(), self.masks[t + 1].data_ptr()
            a.flat_obs, a.reset_mask = None, None
            a.reward, a.terminated, a.truncated = self.rewards64[t].data_ptr(), self.term[t].data_ptr(), self.trunc[t].data_ptr()
            return a

        self._sargs = [step_args(t) for t in range(T)]

    @torch.no_grad()
    def collect(self) -> CteRecurrentBatch:
        """Roll T steps from the env's current observation (its ``obs_grid`` / ``action_mask``)."""
        env, fused, lib, T, L = self.env, self.fused, self._lib, self.T, self.L
        B, cells = env.B, env.R * env.C
        stream = env._stream()
        h, c = self.state
        self.grid[0].copy_(env.obs_grid.view(B, cells))
        self.masks[0].copy_(env.action_mask)
        # step 0's previous action / reward / episode start are the carried ones (read before step 0 overwrites them)
        torch.logical_or(self.prev_term, self.prev_trunc, out=self.resets[0])
        self.prev_actions[0].copy_(self.act8)
        self.prev_rewards[0].copy_(self.prev_reward)
        for t in range(T):
            if t % L == 0:   # the chunk's start state after the episode-start cut
                keep = ~(self.resets[0] if t == 0 else (self.term[t - 1] | self.trunc[t - 1]).bool())
                torch.mul(h, keep.unsqueeze(-1), out=self.chunk_h[t // L])
                torch.mul(c, keep.unsqueeze(-1), out=self.chunk_c[t // L])
            fused.counter += 1
            a = self._pargs[t]
            a.counter = fused.counter
            nat.check(lib.mapf_cte_lstm_policy_act(C.byref(a), stream))
            nat.check(lib.mapf_cte_step(C.byref(self._sargs[t]), stream))
            m = self.term[t] | self.trunc[t]   # BatchedCteEnv.step(auto_reset=True)'s reset, into row t + 1
            if not env.deterministic:
                env._draw(m)
            env._reset_launch(m, self._sargs[t])
        fused.counter += 1
        a = self._pargs[T]
        a.counter = fused.counter
        nat.check(lib.mapf_cte_lstm_policy_act(C.byref(a), stream))
        self.rewards.copy_(self.rewards64)
        dones = (self.term | self.trunc).bool()
        self.resets[1:] = dones[:-1]
        self.prev_actions[1:] = self.actions[:-1]
        self.prev_rewards[1:] = self.rewards[:-1]
        keep = ~self.resets
        self.prev_actions.mul_(keep.unsqueeze(-1))
        self.prev_rewards.mul_(keep)
        # carried into the next collect; act8 already holds the last step's actions
        self.prev_reward.copy_(self.rewards64[T - 1])
        self.prev_term.copy_(self.term[T - 1])
        self.prev_trunc.copy_(self.trunc[T - 1])
        env.obs_grid.view(B, cells).copy_(self.grid[T])
        env.action_mask.copy_(self.masks[T])
        env.flat_obs[:, :cells].copy_(self.grid[T])
        env.flat_obs[:, cells:].copy_(self.masks[T])
        env.reward.copy_(self.rewards64[T - 1])
        env.terminated.copy_(self.term[T - 1])
        env.truncated.copy_(self.trunc[T - 1])
        return CteRecurrentBatch(self.grid, self.masks, self.actions, self.logp, self.values, self.rewards, dones,
                                 self.last_value, self.prev_actions, self.prev_rewards, self.resets, self.chunk_h,
                                 self.chunk_c)


def ppo_update_cte_recurrent(policy: CteRecurrentPolicy, optimizer, batch: CteRecurrentBatch, *, max_seq_len: int = 32,
                             clip: float = 0.05, vf_coeff: float = 0.5, entropy_coeff: float = 0.001, epochs: int = 12,
                             minibatch: int = 1024, gamma: float = 0.99, lam: float = 0.95, world_size: int = 1,
                             group=None, max_minibatches: int | None = None,
                             generator: torch.Generator | None = None) -> dict:
    """PPO over sequence minibatches of a :class:`CteRecurrentBatch`: GAE and whole-batch advantage normalisation as
    in :func:`ppo_update_cte`; a minibatch is ``minibatch // max_seq_len`` env sequences of one permutation per epoch
    (``generator`` draws it), each re-run through :meth:`CteRecurrentPolicy.sequence` from its stored chunk state
    (truncated back-propagation through time); the loss is :func:`rollout.ppo_objective` on the joint
    log-probability and the summed entropy.  With ``world_size > 1`` every rank trains on its own shard and the
    gradients are averaged over the ranks (:func:`recurrent.allreduce_gradients`) before each optimizer step."""
    L = int(max_seq_len)
    T, B = batch.rewards.shape
    if T % L:
        raise ValueError(f"the batch's {T} steps are not a multiple of max_seq_len ({L})")
    args = (batch.rewards.unsqueeze(-1), batch.values.unsqueeze(-1), batch.dones, batch.last_value.unsqueeze(-1), gamma, lam)
    if batch.rewards.is_cuda:
        from .policy_kernels import gae as gae_kernel

        adv, ret = gae_kernel(*args)
    else:
        adv, ret = gae(*args)
    adv, ret = normalize_advantages(adv, False).squeeze(-1), ret.squeeze(-1)
    nchunks, per_mb = T // L, max(1, minibatch // L)

    def seq_view(x):   # [T,B,...] -> [nchunks, L, B, ...]
        return x[:T].reshape(nchunks, L, B, *x.shape[2:])

    grid, masks, acts, pa, pr = (seq_view(x) for x in (batch.grid, batch.masks, batch.actions, batch.prev_actions,
                                                          batch.prev_rewards))
    rs, olp, av, rt = seq_view(batch.resets), seq_view(batch.logp), seq_view(adv), seq_view(ret)
    total = nchunks * B
    stats, done_mb = {}, 0
    for _ in range(epochs):
        perm = draw_permutation(total, acts.device, generator)
        for i in range(0, total, per_mb):
            idx = perm[i:i + per_mb]
            ck, m = idx // B, idx % B
            g = lambda x: x[ck, :, m].transpose(0, 1)   # noqa: E731  -> [L, S, ...]
            lg, v, _ = policy.sequence(g(grid), g(masks), g(pa), g(pr), g(rs), (batch.chunk_h[ck, m], batch.chunk_c[ck, m]))
            lp, ent = joint_logp_entropy(lg, g(acts))
            loss, stats = ppo_objective(lp, ent, v, g(olp), g(av), g(rt), clip=clip, vf_coeff=vf_coeff,
                                        entropy_coeff=entropy_coeff)
            optimizer.zero_grad(set_to_none=True)
            loss.backward()
            allreduce_gradients(policy, world_size, group)
            optimizer.step()
            done_mb += 1
            if max_minibatches is not None and done_mb >= max_minibatches:
                return stats
    return stats


def benchmark(num_envs: int = 65536, num_agents: int = 16, steps: int = 64, device: str = "cuda:0") -> dict:
    """Env-steps/s and agent-steps/s of the CTE env alone (fixed random joint actions), :func:`collect_cte`,
    :class:`FusedCteCollector`, :class:`RecurrentCteCollector` and :class:`FusedRecurrentCteCollector` (max_seq_len 32)
    on a 32x32 map with 30 % obstacles, 256 steps per episode, T = ``steps``."""
    from . import maps
    from .policy_kernels import FusedCtePolicy, FusedCteRecurrentPolicy
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
    rpolicy = CteRecurrentPolicy(env.R * env.C, env.N).to(env.device)
    rcollector = RecurrentCteCollector(env, rpolicy, 32)
    frcollector = FusedRecurrentCteCollector(env, FusedCteRecurrentPolicy(rpolicy, env), steps, 32)
    for name, fn in (("env_only", env_only), ("collect_cte", lambda: collect_cte(env, policy, steps)),
                     ("fused_cte_collector", collector.collect),
                     ("recurrent_cte_collector", lambda: rcollector.collect(steps)),
                     ("fused_recurrent_cte_collector", frcollector.collect)):
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
