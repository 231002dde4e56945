"""The recurrent policy of the reference's PPO configuration and a multi-GPU learner step around the batched env
(SURVEY 8f N1).  The module is plain PyTorch -- it is the user's model and the learner's; the rollout forward has a
fused CUDA path for the reference's shape (:class:`FusedRecurrentCollector`, ``mapf_lstm_policy_act``).

Reference: ``src/agents/ppo.py:67-75`` (``fcnet_hiddens [64, 64]``, ``use_lstm``, ``lstm_cell_size 64``,
``lstm_use_prev_action``, ``lstm_use_prev_reward``, ``max_seq_len 32``, ``vf_share_layers``) and ``:104-117``
(gamma 0.99, lambda 0.95, clip 0.05, lr 1e-3, entropy 1e-3, vf 0.5, minibatch 1024, 12 epochs).

* :class:`RecurrentActionMaskPolicy` -- MLP trunk -> LSTM(64) fed with the trunk output, the one-hot previous action
  and the previous reward -> logits (masked like ``models/action_mask_model.py:51-64``) and value heads.
* :class:`CompactRollout` / :func:`collect_recurrent` -- T env steps on the device; the batch keeps the env's
  *channels* (uint8 window 25 B + float32 goal delta 8 B + pressure flag 1 B = 34 B per agent-step at sensor range 2)
  instead of float32 feature rows (112 B), and expands them per minibatch (:func:`features_from_channels`), plus the
  LSTM state at the start of every ``max_seq_len`` chunk (truncated back-propagation through time, as RLlib does).
* :class:`FusedRecurrentCollector` -- the same :class:`CompactRollout` in two launches per step (fused LSTM policy +
  draw, env step); ``python -m dl_reference_models_b200.recurrent`` times it against :class:`RecurrentCollector`.
* :func:`ppo_update_recurrent` -- PPO on sequence minibatches; with ``world_size > 1`` every rank holds its own env
  shard and the gradients are all-reduced (mean) before each optimizer step: an N-GPU data-parallel learner whose
  only traffic is the ~50 k parameters' gradients (NCCL on GPUs, gloo in the CPU tests).
"""
from __future__ import annotations

from dataclasses import dataclass

import torch
from torch import nn

from .rollout import (FLOAT_MIN, agent_linear, draw_permutation, gae, normalize_advantages, observation_rows,
                      per_agent_minibatches, ppo_loss, sample_categorical, stack_parameters)


def features_from_channels(local_obs: torch.Tensor, goal_delta: torch.Tensor, blocking_prev: torch.Tensor | None) -> torch.Tensor:
    """ENV:306-328 without the mask: [..., V, V] uint8, [..., 2] float32, [...] uint8 -> [..., V*V + 2 (+ 1)] float32."""
    parts = [local_obs.flatten(-2).float(), goal_delta.float()]
    if blocking_prev is not None:
        parts.append(blocking_prev.float().unsqueeze(-1))
    return torch.cat(parts, dim=-1)


class RecurrentActionMaskPolicy(nn.Module):
    def __init__(self, feature_dim: int, num_actions: int = 5, hiddens=(64, 64), cell: int = 64,
                 use_prev_action: bool = True, use_prev_reward: bool = True):
        super().__init__()
        layers, last = [], int(feature_dim)
        for h in hiddens:
            layers += [nn.Linear(last, int(h)), nn.ReLU()]
            last = int(h)
        self.trunk = nn.Sequential(*layers)
        self.num_actions, self.cell = int(num_actions), int(cell)
        self.use_prev_action, self.use_prev_reward = bool(use_prev_action), bool(use_prev_reward)
        self.lstm = nn.LSTMCell(last + (num_actions if use_prev_action else 0) + (1 if use_prev_reward else 0), cell)
        self.logits = nn.Linear(cell, num_actions)
        self.value = nn.Linear(cell, 1)   # vf_share_layers: the value head reads the same LSTM output

    def initial_state(self, n: int, device=None):
        z = torch.zeros((n, self.cell), device=device)
        return z, z.clone()

    def step(self, features, action_mask, prev_action, prev_reward, state):
        """One time step for a flat batch [M, ...]: returns (masked logits [M, A], value [M], new state)."""
        x = [self.trunk(features.float())]
        if self.use_prev_action:
            x.append(torch.nn.functional.one_hot(prev_action.long(), self.num_actions).to(x[0].dtype))
        if self.use_prev_reward:
            x.append(prev_reward.to(x[0].dtype).unsqueeze(-1))
        h, c = self.lstm(torch.cat(x, dim=-1), state)
        logits = self.logits(h) + torch.clamp(torch.log(action_mask.to(h.dtype) + 1e-6), min=FLOAT_MIN)
        return logits, self.value(h).squeeze(-1), (h, c)

    def sequence(self, features, action_mask, prev_action, prev_reward, resets, state):
        """[T, M, ...] inputs; ``resets`` [T, M] bool = the step starts a new episode (state, previous action and
        previous reward are zeroed in front of it).  Returns logits [T, M, A], values [T, M], final state."""
        T = features.shape[0]
        lg, vs = [], []
        h, c = state
        for t in range(T):
            keep = (~resets[t]).to(h.dtype).unsqueeze(-1)
            h, c = h * keep, c * keep
            pa = prev_action[t] * (~resets[t]).to(prev_action.dtype)
            pr = prev_reward[t] * (~resets[t]).to(prev_reward.dtype)
            l, v, (h, c) = self.step(features[t], action_mask[t], pa, pr, (h, c))
            lg.append(l)
            vs.append(v)
        return torch.stack(lg), torch.stack(vs), (h, c)


class PerAgentRecurrentPolicy(nn.Module):
    """One :class:`RecurrentActionMaskPolicy` per agent (the reference's DTE mode), parameters stacked along a leading
    agent dimension (``trunk_w[k]`` / ``trunk_b[k]``, ``w_ih`` [N, 4 cell, in], ``w_hh``, ``b_ih``, ``b_hh``,
    ``logits_w`` / ``logits_b``, ``value_w`` / ``value_b``; torch LSTMCell's gate order [i; f; g; o]).  Inputs follow
    :class:`rollout.PerAgentActionMaskPolicy`'s convention: flat rows whose count is a multiple of ``num_agents``, row
    r of agent ``r % num_agents`` (the [B*N, ...] rows of :class:`RecurrentCollector`, the state's [B*N, cell] layout).
    :meth:`from_modules` / :meth:`module` convert from / to ordinary modules; the default initialisation is N
    independently initialised ones."""

    def __init__(self, num_agents: int, feature_dim: int, num_actions: int = 5, hiddens=(64, 64), cell: int = 64,
                 use_prev_action: bool = True, use_prev_reward: bool = True):
        super().__init__()
        self._stack([RecurrentActionMaskPolicy(feature_dim, num_actions, hiddens, cell, use_prev_action, use_prev_reward)
                     for _ in range(int(num_agents))])

    @classmethod
    def from_modules(cls, modules) -> "PerAgentRecurrentPolicy":
        """Agent j's parameters are copies of ``modules[j]``'s (N :class:`RecurrentActionMaskPolicy` of one shape)."""
        self = cls.__new__(cls)
        nn.Module.__init__(self)
        self._stack(list(modules))
        return self

    @staticmethod
    def _shape(m) -> tuple:
        lin = [x for x in m.trunk.modules() if isinstance(x, nn.Linear)]
        feature_dim = lin[0].in_features if lin else m.lstm.input_size - m.num_actions * m.use_prev_action - m.use_prev_reward
        return (int(feature_dim), tuple(x.out_features for x in lin), m.num_actions, m.cell, m.use_prev_action,
                m.use_prev_reward)

    def _stack(self, mods):
        if not mods or any(self._shape(m) != self._shape(mods[0]) for m in mods):
            raise ValueError(f"from_modules needs one or more modules of one shape, got {[self._shape(m) for m in mods]}")
        self.num_agents = len(mods)
        (self.feature_dim, self.hiddens, self.num_actions, self.cell, self.use_prev_action,
         self.use_prev_reward) = self._shape(mods[0])
        lins = [[x for x in m.trunk.modules() if isinstance(x, nn.Linear)] for m in mods]
        self.trunk_w = nn.ParameterList([stack_parameters(ls[k].weight for ls in lins) for k in range(len(self.hiddens))])
        self.trunk_b = nn.ParameterList([stack_parameters(ls[k].bias for ls in lins) for k in range(len(self.hiddens))])
        for name, get in (("w_ih", lambda m: m.lstm.weight_ih), ("w_hh", lambda m: m.lstm.weight_hh),
                          ("b_ih", lambda m: m.lstm.bias_ih), ("b_hh", lambda m: m.lstm.bias_hh),
                          ("logits_w", lambda m: m.logits.weight), ("logits_b", lambda m: m.logits.bias),
                          ("value_w", lambda m: m.value.weight), ("value_b", lambda m: m.value.bias)):
            setattr(self, name, stack_parameters(get(m) for m in mods))

    def module(self, j: int) -> RecurrentActionMaskPolicy:
        """Agent j's policy as an ordinary :class:`RecurrentActionMaskPolicy` (a copy, on this module's device)."""
        with torch.random.fork_rng(devices=[]):   # the throw-away default init must not move the caller's RNG
            m = RecurrentActionMaskPolicy(self.feature_dim, self.num_actions, self.hiddens, self.cell,
                                          self.use_prev_action, self.use_prev_reward)
        m = m.to(self.w_ih.device)
        with torch.no_grad():
            for lin, w, b in zip([x for x in m.trunk.modules() if isinstance(x, nn.Linear)], self.trunk_w, self.trunk_b):
                lin.weight.copy_(w[j])
                lin.bias.copy_(b[j])
            for t, name in ((m.lstm.weight_ih, "w_ih"), (m.lstm.weight_hh, "w_hh"), (m.lstm.bias_ih, "b_ih"),
                            (m.lstm.bias_hh, "b_hh"), (m.logits.weight, "logits_w"), (m.logits.bias, "logits_b"),
                            (m.value.weight, "value_w"), (m.value.bias, "value_b")):
                t.copy_(getattr(self, name)[j])
        return m

    initial_state = RecurrentActionMaskPolicy.initial_state
    sequence = RecurrentActionMaskPolicy.sequence   # steps through :meth:`step`

    def step(self, features, action_mask, prev_action, prev_reward, state):
        """One time step for flat rows [M, ...] (row r of agent r % N): (masked logits [M, A], value [M], new state)."""
        N = self.num_agents
        per = lambda x: x.reshape(-1, N, *x.shape[1:]).transpose(0, 1)   # noqa: E731  [M, ...] -> [N, M / N, ...]
        flat = lambda x: x.transpose(0, 1).reshape(-1, *x.shape[2:])    # noqa: E731  and back
        z = per(features.float())
        for w, b in zip(self.trunk_w, self.trunk_b):
            z = torch.relu(agent_linear(z, w, b))
        x = [z]
        if self.use_prev_action:
            x.append(torch.nn.functional.one_hot(per(prev_action).long(), self.num_actions).to(z.dtype))
        if self.use_prev_reward:
            x.append(per(prev_reward).to(z.dtype).unsqueeze(-1))
        gates = agent_linear(torch.cat(x, dim=-1), self.w_ih, self.b_ih) + agent_linear(per(state[0]), self.w_hh, self.b_hh)
        i, f, g, o = gates.chunk(4, dim=-1)
        c = torch.sigmoid(f) * per(state[1]) + torch.sigmoid(i) * torch.tanh(g)
        h = torch.sigmoid(o) * torch.tanh(c)
        logits = flat(agent_linear(h, self.logits_w, self.logits_b))
        logits = logits + torch.clamp(torch.log(action_mask.to(h.dtype) + 1e-6), min=FLOAT_MIN)
        return logits, flat(agent_linear(h, self.value_w, self.value_b)).squeeze(-1), (flat(h), flat(c))


@dataclass
class CompactRollout:
    local_obs: torch.Tensor      # [T,B,N,V,V] uint8
    goal_delta: torch.Tensor     # [T,B,N,2]  float32
    blocking_prev: torch.Tensor  # [T,B,N]    uint8
    masks: torch.Tensor          # [T,B,N,5]  int8
    actions: torch.Tensor        # [T,B,N]    int64
    prev_actions: torch.Tensor   # [T,B,N]    int64 (action of the step before, 0 behind a reset)
    prev_rewards: torch.Tensor   # [T,B,N]    float32
    resets: torch.Tensor         # [T,B]      bool: step t is the first of an episode
    logp: torch.Tensor           # [T,B,N]
    values: torch.Tensor         # [T,B,N]
    rewards: torch.Tensor        # [T,B,N]
    dones: torch.Tensor          # [T,B]      bool: the episode ended AT step t (the env auto-reset)
    last_value: torch.Tensor     # [B,N]
    chunk_h: torch.Tensor        # [T/L, B*N, cell] LSTM state at the start of every max_seq_len chunk
    chunk_c: torch.Tensor

    def bytes_per_agent_step(self) -> int:
        per = lambda t: t[0, 0, 0].numel() * t.element_size()  # noqa: E731
        return per(self.local_obs) + per(self.goal_delta) + per(self.blocking_prev) + per(self.masks)


class RecurrentCollector:
    """Carries env outputs, LSTM state, previous action / reward across :meth:`collect` calls."""

    def __init__(self, env, policy: RecurrentActionMaskPolicy, max_seq_len: int = 32):
        self.env, self.policy, self.L = env, policy, int(max_seq_len)
        M = env.B * env.N
        self.state = policy.initial_state(M, env.device)
        self.prev_action = torch.zeros((env.B, env.N), dtype=torch.int64, device=env.device)
        self.prev_reward = torch.zeros((env.B, env.N), device=env.device)
        self.reset_next = torch.ones((env.B,), dtype=torch.bool, device=env.device)
        self.out = env._output()

    @torch.no_grad()
    def collect(self, steps: int) -> CompactRollout:
        env, pol, L = self.env, self.policy, self.L
        if steps % L:
            raise ValueError(f"steps ({steps}) must be a multiple of max_seq_len ({L})")
        if getattr(env, "_fused", 0):
            raise RuntimeError("turn the env's fused uniform sampler off (fuse_sampler(None)) before a policy rollout")
        B, N, V, dev, T = env.B, env.N, env.V, env.device, int(steps)
        z = lambda shape, dt: torch.empty(shape, dtype=dt, device=dev)  # noqa: E731
        r = CompactRollout(z((T, B, N, V, V), torch.uint8), z((T, B, N, 2), torch.float32), z((T, B, N), torch.uint8),
                           z((T, B, N, 5), torch.int8), z((T, B, N), torch.int64), z((T, B, N), torch.int64),
                           z((T, B, N), torch.float32), z((T, B), torch.bool), z((T, B, N), torch.float32),
                           z((T, B, N), torch.float32), z((T, B, N), torch.float32), z((T, B), torch.bool),
                           z((B, N), torch.float32), z((T // L, B * N, pol.cell), torch.float32),
                           z((T // L, B * N, pol.cell), torch.float32))
        out = self.out
        h, c = self.state
        for t in range(T):
            rs = self.reset_next
            keep = (~rs).repeat_interleave(N).to(h.dtype).unsqueeze(-1)
            h, c = h * keep, c * keep
            if t % L == 0:
                r.chunk_h[t // L], r.chunk_c[t // L] = h, c
            pa = self.prev_action * (~rs).unsqueeze(-1)
            pr = self.prev_reward * (~rs).unsqueeze(-1)
            r.local_obs[t], r.goal_delta[t], r.blocking_prev[t], r.masks[t] = out.local_obs, out.goal_delta, out.blocking_prev, out.action_mask
            r.prev_actions[t], r.prev_rewards[t], r.resets[t] = pa, pr, rs
            feats = features_from_channels(out.local_obs, out.goal_delta, out.blocking_prev).reshape(B * N, -1)
            lg, v, (h, c) = pol.step(feats, out.action_mask.reshape(B * N, 5), pa.reshape(-1), pr.reshape(-1), (h, c))
            a, lp = sample_categorical(lg)
            r.actions[t], r.logp[t], r.values[t] = a.reshape(B, N), lp.reshape(B, N), v.reshape(B, N)
            out = env.step(a.reshape(B, N).to(torch.int8), auto_reset=True)
            r.rewards[t] = out.reward
            done = (out.terminated | out.truncated).bool()
            r.dones[t] = done
            self.prev_action, self.prev_reward, self.reset_next = a.reshape(B, N), out.reward.clone(), done
        # bootstrap value of the observation after the last step (state is not advanced)
        rs = self.reset_next
        keep = (~rs).repeat_interleave(N).to(h.dtype).unsqueeze(-1)
        feats = features_from_channels(out.local_obs, out.goal_delta, out.blocking_prev).reshape(B * N, -1)
        _, lv, _ = pol.step(feats, out.action_mask.reshape(B * N, 5), (self.prev_action * (~rs).unsqueeze(-1)).reshape(-1),
                            (self.prev_reward * (~rs).unsqueeze(-1)).reshape(-1), (h * keep, c * keep))
        r.last_value.copy_(lv.reshape(B, N))
        self.state, self.out = (h, c), out
        return r


class FusedRecurrentCollector:
    """:class:`RecurrentCollector` with the forward pass and the draw in one CUDA launch
    (:class:`policy_kernels.FusedRecurrentPolicy`): a step is exactly two launches, ``mapf_lstm_policy_act`` then
    ``mapf_step``, with argument blocks built once here.  The layout is ``FusedCollector(compact=True)``'s: env step t
    writes the observation channels into row t + 1 of [T + 1, ...] buffers and reward / terminated / truncated into row
    t; the policy launch of step t reads channel row t, the reward and episode ends of step t - 1 (the carried ones at
    t = 0), writes actions[t] / logp[t] / values[t] and advances the LSTM state in place.  The previous actions /
    rewards, reset flags and chunk-start states of the :class:`CompactRollout` are filled with a few vectorised ops per
    collect (one state snapshot per ``max_seq_len`` steps).  The returned batch's buffers are reused by the next
    :meth:`collect`."""

    def __init__(self, env, fused, steps: int, max_seq_len: int = 32):
        import ctypes as C

        from . import _native as nat

        T, L = int(steps), int(max_seq_len)
        if T % L:
            raise ValueError(f"steps ({T}) must be a multiple of max_seq_len ({L})")
        self.env, self.fused, self.T, self.L = env, fused, T, L
        B, N, dev, cell = env.B, env.N, env.device, 64
        o = env.out
        self.obs_rows = observation_rows(env, T + 1)
        z = lambda shape, dt=torch.float32: torch.zeros(shape, dtype=dt, device=dev)  # noqa: E731
        self.actions, self.prev_actions = z((T, B, N), torch.int64), z((T, B, N), torch.int64)
        self.logp, self.values, self.rewards = z((T, B, N)), z((T, B, N)), z((T, B, N))
        self.prev_rewards = z((T, B, N))
        self.term, self.trunc = z((T, B), torch.uint8), z((T, B), torch.uint8)
        self.last_value = z((B, N))
        self.chunk_h, self.chunk_c = z((T // L, B * N, cell)), z((T // L, B * N, cell))
        # carried across collects, as RecurrentCollector does: state, previous action / reward, episode-start flags
        self.state = (z((B * N, cell)), z((B * N, cell)))
        self.act8 = z((B, N), torch.int8)   # this step's actions (to mapf_step) = the next step's previous actions
        self.prev_reward = z((B, N))
        self.prev_term, self.prev_trunc = torch.ones((B,), dtype=torch.uint8, device=dev), z((B,), torch.uint8)
        self._C, self._nat, self._lib = C, nat, nat.lib()
        rows = self.obs_rows

        def policy_args(t):
            last = t == T
            ch = {k: r[t] for k, r in rows.items()}
            pr, pt, ptr = (self.prev_reward, self.prev_term, self.prev_trunc) if t == 0 else \
                (self.rewards[t - 1], self.term[t - 1], self.trunc[t - 1])
            return fused.args(ch, self.state, self.act8, pr, pt, ptr, state_out=None if last else self.state,
                              actions=None if last else self.act8, actions64=None if last else self.actions[t],
                              logp=None if last else self.logp[t], value=self.last_value if last else self.values[t])

        self._pargs = [policy_args(t) for t in range(T + 1)]   # the last one: bootstrap value, state not advanced

        def dst(k, t):   # where the env step t writes channel k
            if k == "reward":
                return self.rewards[t]
            if k == "terminated":
                return self.term[t]
            if k == "truncated":
                return self.trunc[t]
            if k in rows:
                return rows[k][t + 1]
            return o[k]

        self._couts = [nat.MapfOutputs(**{k: dst(k, t).data_ptr() for k in nat.OUTPUT_FIELDS}) for t in range(T)]
        self._actions_ptr = C.c_void_p(self.act8.data_ptr())
        self._act = getattr(self._lib, fused.entry)   # mapf_lstm_policy_act, or its per-agent variant

    @torch.no_grad()
    def collect(self) -> CompactRollout:
        """Roll T steps from the env's current observation (its output buffers, i.e. the last reset / step)."""
        C, lib, env, fused, T, L = self._C, self._lib, self.env, self.fused, self.T, self.L
        if getattr(env, "_fused", 0):
            raise RuntimeError("turn the env's fused uniform sampler off (fuse_sampler(None)) before a policy rollout")
        B, N = env.B, env.N
        stream, hnd, check = env._stream(), env._h, self._nat.check
        h, c = self.state
        for k, r in self.obs_rows.items():   # row 0 = the env's current observation
            r[0].copy_(env.out[k])
        # step 0's previous action / reward / episode start are the carried ones (read before step 0 overwrites them)
        resets = torch.empty((T, B), dtype=torch.bool, device=env.device)
        resets[0] = (self.prev_term | self.prev_trunc).bool()
        self.prev_actions[0].copy_(self.act8)
        self.prev_rewards[0].copy_(self.prev_reward)
        for t in range(T):
            if t % L == 0:   # the chunk's start state after the episode-start cut (RecurrentCollector's h * keep)
                keep = (~(resets[0] if t == 0 else (self.term[t - 1] | self.trunc[t - 1]).bool())).to(h.dtype).view(B, 1, 1)
                torch.mul(h.view(B, N, -1), keep, out=self.chunk_h[t // L].view(B, N, -1))
                torch.mul(c.view(B, N, -1), keep, out=self.chunk_c[t // L].view(B, N, -1))
            fused.counter += 1
            a = self._pargs[t]
            a.counter = fused.counter
            check(self._act(C.byref(a), stream))
            check(lib.mapf_step(hnd, self._actions_ptr, None, None, C.byref(self._couts[t]), 1, stream))
        fused.counter += 1
        a = self._pargs[T]
        a.counter = fused.counter
        check(self._act(C.byref(a), stream))
        dones = (self.term | self.trunc).bool()
        resets[1:] = dones[:-1]
        self.prev_actions[1:] = self.actions[:-1]
        self.prev_rewards[1:] = self.rewards[:-1]
        keep = (~resets).unsqueeze(-1)
        self.prev_actions.mul_(keep)
        self.prev_rewards.mul_(keep)
        # carried into the next collect; act8 already holds the last step's actions
        self.prev_reward.copy_(self.rewards[T - 1])
        self.prev_term.copy_(self.term[T - 1])
        self.prev_trunc.copy_(self.trunc[T - 1])
        for k, r in self.obs_rows.items():   # the env's own buffers show the latest observation again
            env.out[k].copy_(r[T])
        rows = self.obs_rows
        return CompactRollout(rows["local_obs"][:T], rows["goal_delta"][:T], rows["blocking_prev"][:T],
                              rows["action_mask"][:T], self.actions, self.prev_actions, self.prev_rewards, resets,
                              self.logp, self.values, self.rewards, dones, self.last_value, self.chunk_h, self.chunk_c)


def collect_recurrent(env, policy, steps: int, max_seq_len: int = 32) -> CompactRollout:
    return RecurrentCollector(env, policy, max_seq_len).collect(steps)


def allreduce_gradients(module: nn.Module, world_size: int, group=None):
    """Mean of the gradients over the ranks, one flat all-reduce (the learner's only collective)."""
    if world_size <= 1:
        return
    import torch.distributed as dist

    grads = [p.grad for p in module.parameters() if p.grad is not None]
    flat = torch.cat([g.reshape(-1) for g in grads])
    dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
    flat /= world_size
    at = 0
    for g in grads:
        n = g.numel()
        g.copy_(flat[at:at + n].view_as(g))
        at += n


def ppo_update_recurrent(policy: RecurrentActionMaskPolicy, optimizer, batch: CompactRollout, *, max_seq_len: int = 32,
                         clip: float = 0.05, vf_coeff: float = 0.5, entropy_coeff: float = 0.001, epochs: int = 12,
                         minibatch: int = 1024, gamma: float = 0.99, lam: float = 0.95, world_size: int = 1, group=None,
                         max_minibatches: int | None = None, generator: torch.Generator | None = None) -> dict:
    """PPO over sequence minibatches: ``minibatch`` time steps = ``minibatch / max_seq_len`` sequences of one agent,
    each re-run through the LSTM from its stored start state (truncated BPTT).  Every rank draws its own minibatches
    from its own shard; gradients are averaged over the ranks before each optimizer step.  A
    :class:`PerAgentRecurrentPolicy` is trained as N independent learners in lockstep (see :func:`rollout.ppo_update`):
    advantages normalised per agent, ``minibatch / max_seq_len`` of agent j's own sequences for every j per step
    (agent-fastest), the loss summed over the agents' mean losses."""
    L = int(max_seq_len)
    T, B, N = batch.actions.shape
    per_agent = isinstance(policy, PerAgentRecurrentPolicy)
    if per_agent and policy.num_agents != N:
        raise ValueError(f"the policy has {policy.num_agents} agents, the batch {N}")
    adv, ret = gae(batch.rewards, batch.values, batch.dones, batch.last_value, gamma, lam)
    adv = normalize_advantages(adv, per_agent)
    nchunks, M = T // L, B * N
    per_mb = max(1, minibatch // L)

    def seq_view(x):   # [T,B,N,...] -> [nchunks, L, M, ...]
        return x.reshape(nchunks, L, M, *x.shape[3:])

    lo, gd, bp, mk = seq_view(batch.local_obs), seq_view(batch.goal_delta), seq_view(batch.blocking_prev), seq_view(batch.masks)
    ac, pa, pr = seq_view(batch.actions), seq_view(batch.prev_actions), seq_view(batch.prev_rewards)
    olp, av, rt = seq_view(batch.logp), seq_view(adv), seq_view(ret)
    rs = batch.resets.unsqueeze(-1).expand(T, B, N).reshape(nchunks, L, M)
    stats, done_mb = {}, 0
    total = nchunks * M

    def minibatches():   # sequence numbers idx: chunk idx // M, row idx % M
        if per_agent:   # sequence s of agent j: chunk s // B, row (s % B) * N + j
            cols = torch.arange(N, device=ac.device)
            for s in per_agent_minibatches(nchunks * B, N, per_mb, ac.device, generator):
                yield ((s // B) * M + (s % B) * N + cols).reshape(-1)
        else:
            perm = draw_permutation(total, ac.device, generator)
            for i in range(0, total, per_mb):
                yield perm[i:i + per_mb]

    for _ in range(epochs):
        for idx in minibatches():
            ck, m = idx // M, idx % M
            g = lambda x: x[ck, :, m].transpose(0, 1)   # noqa: E731  -> [L, S, ...]
            feats = features_from_channels(g(lo), g(gd), g(bp))   # expanded here, per minibatch: 34 B -> 112 B per row
            lg, v, _ = policy.sequence(feats, g(mk), g(pa), g(pr), g(rs), (batch.chunk_h[ck, m], batch.chunk_c[ck, m]))
            loss, stats = ppo_loss(lg, v, g(ac), g(olp), g(av), g(rt), clip=clip, vf_coeff=vf_coeff,
                                   entropy_coeff=entropy_coeff, num_agents=N if per_agent else None)
            optimizer.zero_grad(set_to_none=True)
            loss.backward()
            allreduce_gradients(policy, world_size, group)
            optimizer.step()
            done_mb += 1
            if max_minibatches is not None and done_mb >= max_minibatches:
                return stats
    return stats


def benchmark(num_envs: int = 65536, steps: int = 64, max_seq_len: int = 32, rounds: int = 3, device: str = "cuda:0") -> dict:
    """C3 (num_envs x 16 agents, 32x32 map, lifelong): agent-steps/s of the env alone, of :class:`RecurrentCollector`
    (the PyTorch module's forward every step) and of :class:`FusedRecurrentCollector` (one policy launch + one env
    launch per step) with a shared policy and with a :class:`PerAgentRecurrentPolicy` (one LSTM per agent,
    ``mapf_lstm_policy_act_per_agent``), the three collectors alternated in the same process after a warm-up collect
    each.  Rates are the
    best of ``rounds`` timed collects (host clock around work that ends in a device synchronise)."""
    import subprocess
    import time

    from . import maps
    from .batched_env import BatchedMapfEnv
    from .policy_kernels import FusedRecurrentPolicy
    from .recurrent import PerAgentRecurrentPolicy   # the package's class (this file may run as __main__)

    cfg = {"num_agents": 16, "sensor_range": 2, "steps_per_episode": 256, "lifelong_mapf": True, "seed": 999,
           "grid": maps.random_obstacle_grid(32, 32, 0.30, 2026, min_free=32)}
    env = BatchedMapfEnv(cfg, num_envs, device)
    env.reset()
    n = num_envs * env.N * steps

    def timed(fn):
        torch.cuda.synchronize(env.device)
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize(env.device)
        return time.perf_counter() - t0

    a = env.sample_actions(masked=True)
    env.fuse_sampler("masked")
    for _ in range(8):
        env.step(a, auto_reset=True)
    env_s = min(timed(lambda: [env.step(a, auto_reset=True) for _ in range(steps)]) for _ in range(rounds))
    env.fuse_sampler(None)
    torch.manual_seed(0)
    pol = RecurrentActionMaskPolicy(env.flat_obs_dim(include_action_mask=False)).to(env.device)
    torch_col = RecurrentCollector(env, pol, max_seq_len)
    fused_col = FusedRecurrentCollector(env, FusedRecurrentPolicy(pol, env), steps, max_seq_len)
    per_agent = PerAgentRecurrentPolicy(env.N, env.flat_obs_dim(include_action_mask=False)).to(env.device)
    per_agent_col = FusedRecurrentCollector(env, FusedRecurrentPolicy(per_agent, env), steps, max_seq_len)
    torch_col.collect(steps)   # warm-up: allocator, cuBLAS / kernel selection, module load
    fused_col.collect()
    per_agent_col.collect()
    ts, fs, ps = [], [], []
    for _ in range(rounds):
        ts.append(timed(lambda: torch_col.collect(steps)))
        fs.append(timed(fused_col.collect))
        ps.append(timed(per_agent_col.collect))
    try:
        gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                              str(env.device.index)], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as exc:
        gpu = f"nvidia-smi not readable: {exc}"
    assert env.poll_errors() == 0
    return {"gpu": gpu or torch.cuda.get_device_name(env.device), "envs": num_envs, "agents": env.N, "steps": steps,
            "max_seq_len": max_seq_len, "env_only_agent_steps_per_s": n / env_s,
            "torch_recurrent_collector_agent_steps_per_s": n / min(ts),
            "fused_recurrent_collector_agent_steps_per_s": n / min(fs),
            "fused_per_agent_recurrent_collector_agent_steps_per_s": n / min(ps),
            "torch_collect_s": ts, "fused_collect_s": fs, "fused_per_agent_collect_s": ps}


if __name__ == "__main__":
    import json

    print(json.dumps(benchmark()))
