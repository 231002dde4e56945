"""On-device rollout loop around the batched env (BASELINE config 5).

The caller side of the hot path, restated without RLlib so that observations never leave HBM:

* :class:`ActionMaskPolicy` -- the reference's action-mask MLP (``models/action_mask_model.py:8-67``:
  shared ``Linear-ReLU`` trunk over the flat features, a logits head, a value head, and
  ``logits + clamp(log(mask + 1e-6), min=FLOAT_MIN)`` masking, ``:51-64``) as a plain ``nn.Module``
  that takes the feature block and the int8 mask as separate tensors (the batched env already
  emits them separately);
* :func:`collect` -- T steps of ``policy -> sample -> BatchedMapfEnv.step(auto_reset=True)``;
* :func:`gae` and :func:`ppo_update` -- the PPO arithmetic with the reference's hyper-parameters
  (``src/agents/ppo.py:104-117``: gamma 0.99, lambda 0.95, clip 0.05, lr 1e-3, entropy 1e-3,
  vf coeff 0.5, minibatch 1024, 12 epochs) so the loop is a complete, runnable learner.

This module is plain PyTorch by design (the policy is the user's model, not part of the env hot
path); the env transition inside the loop is the CUDA kernel.
"""
from __future__ import annotations

import time
from dataclasses import dataclass

import torch
from torch import nn

FLOAT_MIN = -3.4e38  # ray.rllib.utils.torch_utils.FLOAT_MIN


class ActionMaskPolicy(nn.Module):
    def __init__(self, feature_dim: int, num_actions: int = 5, hiddens=(64, 64), no_masking: bool = False):
        super().__init__()
        layers, last = [], int(feature_dim)
        for h in hiddens:
            layers += [nn.Linear(last, int(h)), nn.ReLU()]
            last = int(h)
        self.trunk = nn.Sequential(*layers) if layers else nn.Identity()
        self.logits = nn.Linear(last, num_actions)
        self.value = nn.Linear(last, 1)
        self.no_masking = no_masking

    def heads(self, features: torch.Tensor):
        """features [..., F] float -> (unmasked logits [..., A], value [...]): the two heads as they are (DQN reads them
        as a dueling network's advantage and value, :func:`dqn.q_values`)."""
        z = self.trunk(features.float())
        return self.logits(z), self.value(z).squeeze(-1)

    def forward(self, features: torch.Tensor, action_mask: torch.Tensor):
        """features [..., F] float, action_mask [..., A] (0/1 of any dtype) -> (masked logits, value)."""
        logits, value = self.heads(features)
        if self.no_masking:
            return logits, value
        inf_mask = torch.clamp(torch.log(action_mask.to(logits.dtype) + 1e-6), min=FLOAT_MIN)
        return logits + inf_mask, value


def agent_linear(x: torch.Tensor, w: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    """Per-agent ``Linear``: x [N, R, in], w [N, out, in], b [N, out] -> [N, R, out] (one batched matmul)."""
    return torch.baddbmm(b.unsqueeze(1), x, w.transpose(1, 2))


def stack_parameters(tensors) -> nn.Parameter:
    """One parameter stacked along a leading agent dimension from the same parameter of N modules."""
    return nn.Parameter(torch.stack([t.detach() for t in tensors]).clone())


class PerAgentActionMaskPolicy(nn.Module):
    """One :class:`ActionMaskPolicy` per agent: the reference's DTE mode, where agent j is played and trained by its own
    module.  The parameters are stacked along a leading agent dimension (``trunk_w[k]`` [N, out, in], ``trunk_b[k]``
    [N, out], ``logits_w`` / ``logits_b``, ``value_w`` / ``value_b``).  Inputs are flat rows whose count is a multiple of
    ``num_agents``, and row r belongs to agent ``r % num_agents``: the [..., B, N, ...] order of every buffer of this
    package, so a [T,B,N,F] block or its [T*B*N, F] view goes in as it is.  The forward is batched matmuls over the
    agent dimension.  Default initialisation: N independently initialised :class:`ActionMaskPolicy` modules;
    :meth:`from_modules` / :meth:`module` convert from / to those (RLlib's per-agent modules map to them one to one)."""

    def __init__(self, num_agents: int, feature_dim: int, num_actions: int = 5, hiddens=(64, 64), no_masking: bool = False):
        super().__init__()
        self._stack([ActionMaskPolicy(feature_dim, num_actions, hiddens, no_masking) for _ in range(int(num_agents))])

    @classmethod
    def from_modules(cls, modules) -> "PerAgentActionMaskPolicy":
        """Agent j's parameters are copies of ``modules[j]``'s (N :class:`ActionMaskPolicy` of one shape)."""
        self = cls.__new__(cls)
        nn.Module.__init__(self)
        self._stack(list(modules))
        return self

    def _stack(self, mods):
        shape = lambda m: (_in_features(m), tuple(x.out_features for x in _linears(m)), m.logits.out_features,  # noqa: E731
                           bool(m.no_masking))
        if not mods or any(shape(m) != shape(mods[0]) for m in mods):
            raise ValueError(f"from_modules needs one or more modules of one shape, got {[shape(m) for m in mods]}")
        self.num_agents = len(mods)
        self.feature_dim, self.hiddens, self.num_actions, self.no_masking = shape(mods[0])
        lins = [_linears(m) for m in mods]
        self.trunk_w = nn.ParameterList([stack_parameters(ls[k].weight for ls in lins) for k in range(len(self.hiddens))])
        self.trunk_b = nn.ParameterList([stack_parameters(ls[k].bias for ls in lins) for k in range(len(self.hiddens))])
        self.logits_w, self.logits_b = stack_parameters(m.logits.weight for m in mods), stack_parameters(m.logits.bias for m in mods)
        self.value_w, self.value_b = stack_parameters(m.value.weight for m in mods), stack_parameters(m.value.bias for m in mods)

    def module(self, j: int) -> ActionMaskPolicy:
        """Agent j's policy as an ordinary :class:`ActionMaskPolicy` (a copy, on this module's device)."""
        with torch.random.fork_rng(devices=[]):   # the throw-away default init must not move the caller's RNG
            m = ActionMaskPolicy(self.feature_dim, self.num_actions, self.hiddens, self.no_masking)
        m = m.to(self.logits_w.device)
        with torch.no_grad():
            for lin, w, b in zip(_linears(m), self.trunk_w, self.trunk_b):
                lin.weight.copy_(w[j])
                lin.bias.copy_(b[j])
            m.logits.weight.copy_(self.logits_w[j])
            m.logits.bias.copy_(self.logits_b[j])
            m.value.weight.copy_(self.value_w[j])
            m.value.bias.copy_(self.value_b[j])
        return m

    def heads(self, features: torch.Tensor):
        """features [..., F] float, flat row r of agent r % N -> (unmasked logits [..., A], value [...])."""
        lead, N = features.shape[:-1], self.num_agents
        z = features.float().reshape(-1, N, features.shape[-1]).transpose(0, 1)   # [N, rows / N, F]
        for w, b in zip(self.trunk_w, self.trunk_b):
            z = torch.relu(agent_linear(z, w, b))
        logits = agent_linear(z, self.logits_w, self.logits_b).transpose(0, 1).reshape(*lead, -1)
        value = agent_linear(z, self.value_w, self.value_b).transpose(0, 1).reshape(lead)
        return logits, value

    def forward(self, features: torch.Tensor, action_mask: torch.Tensor):
        """features [..., F] float, action_mask [..., A], flat row r of agent r % N -> (masked logits, value)."""
        logits, value = self.heads(features)
        if self.no_masking:
            return logits, value
        return logits + torch.clamp(torch.log(action_mask.to(logits.dtype) + 1e-6), min=FLOAT_MIN), value


def _linears(m) -> list:
    return [x for x in m.trunk.modules() if isinstance(x, nn.Linear)]


def _in_features(m) -> int:
    lin = _linears(m)
    return int(lin[0].in_features if lin else m.logits.in_features)


@dataclass
class Batch:
    features: torch.Tensor   # [T,B,N,F]
    masks: torch.Tensor      # [T,B,N,5] int8
    actions: torch.Tensor    # [T,B,N] int64
    logp: torch.Tensor       # [T,B,N]
    values: torch.Tensor     # [T,B,N]
    rewards: torch.Tensor    # [T,B,N]
    dones: torch.Tensor      # [T,B] bool (episode ended at this step; the env auto-reset)
    last_value: torch.Tensor  # [B,N] bootstrap value of the observation after the last step


@dataclass
class CompactBatch:
    """A rollout kept the way the env emits it -- uint8 window, float32 goal delta, uint8 pressure flag: V^2 + 9 bytes per
    agent-step instead of 4 (V^2 + 3) of float32 features -- and expanded per minibatch (:meth:`features_of`).  The other
    fields are those of :class:`Batch`; the observation tensors hold T + 1 rows (row T: the observation after the
    last step)."""
    local_obs: torch.Tensor      # [T+1,B,N,V,V] uint8
    goal_delta: torch.Tensor     # [T+1,B,N,2] float32
    blocking_prev: torch.Tensor  # [T+1,B,N] uint8 (None when the flat observation has no pressure flag)
    masks: torch.Tensor          # [T,B,N,5] int8 (a view of the first T rows of the collector's [T+1,...] buffer)
    actions: torch.Tensor
    logp: torch.Tensor
    values: torch.Tensor
    rewards: torch.Tensor
    dones: torch.Tensor
    last_value: torch.Tensor

    def features_of(self, idx: torch.Tensor) -> torch.Tensor:
        """Float32 feature rows (ENV:306-328 order: window, goal delta, pressure) of the flat agent-step indices ``idx``
        into the first T rows."""
        T1, B, N = self.local_obs.shape[:3]
        V2 = self.local_obs.shape[-1] * self.local_obs.shape[-2]
        t, r = idx // (B * N), idx % (B * N)   # the rows may be padded apart: index (step, agent), never reshape the block
        parts = [self.local_obs.view(T1, B * N, V2)[t, r].float(), self.goal_delta.view(T1, B * N, 2)[t, r]]
        if self.blocking_prev is not None:
            parts.append(self.blocking_prev.view(T1, B * N)[t, r].float().unsqueeze(-1))
        return torch.cat(parts, dim=-1)

    @property
    def features(self) -> torch.Tensor:
        """The whole [T,B,N,F] float32 block (what :class:`Batch` stores), materialised on demand."""
        T, B, N = self.actions.shape
        n = T * B * N
        return self.features_of(torch.arange(n, device=self.actions.device)).reshape(T, B, N, -1)


def sample_categorical(logits: torch.Tensor):
    """Gumbel-max draw from softmax(logits) and its log-probability (no multinomial kernel)."""
    logp_all = torch.log_softmax(logits, dim=-1)
    u = torch.rand_like(logits).clamp_(1e-20, 1.0)
    a = torch.argmax(logp_all - torch.log(-torch.log(u)), dim=-1)
    return a, torch.gather(logp_all, -1, a.unsqueeze(-1)).squeeze(-1)


def observation_rows(env, rows: int) -> dict:
    """[rows, *shape] buffers of the env's observation channels (local_obs, goal_delta, blocking_prev, action_mask) with
    every row 256-byte aligned (the kernels store 128-bit words): a compact rollout's per-step rows."""
    def rows_of(t):
        n, es = t.numel(), t.element_size()
        stride = -(-(n * es) // 256) * 256 // es
        buf = torch.empty((rows, stride), dtype=t.dtype, device=env.device)
        return buf[:, :n].view((rows,) + tuple(t.shape))

    return {k: rows_of(env.out[k]) for k in ("local_obs", "goal_delta", "blocking_prev", "action_mask")}


class FusedCollector:
    """T-step rollouts with two kernel launches per env step and nothing else: the policy kernel
    (:class:`policy_kernels.FusedPolicy`: bf16 tensor-core MLP straight from the env's output channels + masked draw)
    and the env step write every per-step row of the [T,...] batch themselves (features, masks, actions, logp, values /
    rewards, terminated, truncated), and the argument blocks of both launches are built once here, so the Python side
    of a step is two ctypes calls.  The buffers are reused: the :class:`Batch` of one :meth:`collect` is overwritten
    by the next."""

    def __init__(self, env, fused, steps: int, compact: bool = False):
        import ctypes as C

        from . import _native as nat

        self.env, self.fused, self.T, self.compact = env, fused, int(steps), bool(compact)
        B, N, T, dev = env.B, env.N, self.T, env.device
        F = env.flat_obs_dim(include_action_mask=False)
        if self.compact:
            # compact rollout: the env step writes the observation channels of step t straight into row t + 1 of
            # [T + 1, ...] buffers, the policy kernel reads row t and stores no feature block at all
            self.obs_rows = observation_rows(env, T + 1)
            self.feats = None
            self.masks = self.obs_rows["action_mask"][:T]
        else:
            self.feats = torch.empty((T, B, N, F), device=dev)
            self.masks = torch.empty((T, B, N, 5), dtype=torch.int8, device=dev)
        self.actions = torch.empty((T, B, N), dtype=torch.int64, device=dev)
        self.logp = torch.empty((T, B, N), device=dev)
        self.values = torch.empty((T, B, N), device=dev)
        self.rewards = torch.empty((T, B, N), device=dev)
        self.term = torch.empty((T, B), dtype=torch.uint8, device=dev)
        self.trunc = torch.empty((T, B), dtype=torch.uint8, device=dev)
        self.last_value = torch.empty((B, N), device=dev)
        self._C, self._nat, self._lib = C, nat, nat.lib()
        vp = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
        o = env.out

        rows = self.obs_rows if self.compact else None

        def src(k, t):   # where the policy kernel of step t reads channel k
            return vp(rows[k][t]) if rows is not None else vp(o[k])

        def policy_args(t):
            last = t == T
            return nat.MapfPolicyArgs(
                num_envs=B, num_agents=N, v2=env.V * env.V, feature_dim=fused.F,
                no_masking=int(bool(fused.policy.no_masking)), greedy=0, seed=fused.seed, counter=0,
                env_id_base=int(env.cfg.env_id_base), local_obs=src("local_obs", t), goal_delta=src("goal_delta", t),
                blocking_prev=src("blocking_prev", t) if fused.with_bp else None, action_mask=src("action_mask", t),
                weights=vp(fused._dev), actions=vp(fused.actions),
                actions64=vp(fused.actions64 if last else self.actions[t]), logp=vp(fused.logp if last else self.logp[t]),
                value=vp(self.last_value if last else self.values[t]), logits_out=None,
                features_out=None if (last or self.compact) else vp(self.feats[t]),
                action_mask_out=None if (last or self.compact) else vp(self.masks[t]))

        self._pargs = [policy_args(t) for t in range(T + 1)]   # the last one: bootstrap value of the final observation

        def dst(k, t):   # where the env step t writes channel k
            if k == "reward":
                return self.rewards[t]
            if k == "terminated":
                return self.term[t]
            if k == "truncated":
                return self.trunc[t]
            if rows is not None and k in rows:
                return rows[k][t + 1]
            return o[k]

        self._couts = [nat.MapfOutputs(**{k: dst(k, t).data_ptr() for k in nat.OUTPUT_FIELDS}) for t in range(T)]
        self._actions_ptr = vp(fused.actions)
        self._act = getattr(self._lib, fused.entry)   # mapf_policy_act, or its per-agent variant

    @torch.no_grad()
    def collect(self) -> Batch:
        """Roll T steps from the env's current observation (its output buffers, i.e. the last reset / step)."""
        C, lib, env, fused = self._C, self._lib, self.env, self.fused
        if getattr(env, "_fused", 0):
            raise RuntimeError("turn the env's fused uniform sampler off (fuse_sampler(None)) before a policy rollout")
        stream, h, check = env._stream(), env._h, self._nat.check
        if self.compact:   # row 0 = the env's current observation
            for k, r in self.obs_rows.items():
                r[0].copy_(env.out[k])
        for t in range(self.T):
            fused.counter += 1
            a = self._pargs[t]
            a.counter = fused.counter
            check(self._act(C.byref(a), stream))
            check(lib.mapf_step(h, self._actions_ptr, None, None, C.byref(self._couts[t]), 1, stream))
        fused.counter += 1
        a = self._pargs[self.T]
        a.counter = fused.counter
        check(self._act(C.byref(a), stream))
        dones = (self.term | self.trunc).bool()
        if self.compact:
            for k, r in self.obs_rows.items():   # the env's own buffers show the latest observation again
                env.out[k].copy_(r[self.T])
            return CompactBatch(self.obs_rows["local_obs"], self.obs_rows["goal_delta"],
                                self.obs_rows["blocking_prev"] if fused.with_bp else None, self.masks, self.actions,
                                self.logp, self.values, self.rewards, dones, self.last_value)
        return Batch(self.feats, self.masks, self.actions, self.logp, self.values, self.rewards, dones, self.last_value)


@torch.no_grad()
def collect_fused(env, fused, steps: int, out=None) -> Batch:
    """Like :func:`collect`, with policy forward + sampling in ONE CUDA launch per step: two launches per env step in
    total (fresh buffers per call; keep a :class:`FusedCollector` to reuse them).  ``out`` is accepted for symmetry
    with :func:`collect`: the rollout always starts from the env's current output buffers."""
    return FusedCollector(env, fused, steps).collect()


@torch.no_grad()
def collect(env, policy: ActionMaskPolicy, steps: int, out=None) -> Batch:
    """Roll the policy for ``steps`` env steps entirely on the env's device."""
    B, N = env.B, env.N
    dev = env.device
    F = env.flat_obs_dim(include_action_mask=False)
    T = int(steps)
    feats = torch.empty((T, B, N, F), device=dev)
    masks = torch.empty((T, B, N, 5), dtype=torch.int8, device=dev)
    actions = torch.empty((T, B, N), dtype=torch.int64, device=dev)
    logp = torch.empty((T, B, N), device=dev)
    values = torch.empty((T, B, N), device=dev)
    rewards = torch.empty((T, B, N), device=dev)
    dones = torch.empty((T, B), dtype=torch.bool, device=dev)
    if out is None:
        out = env._output()
    for t in range(T):
        env.flat_obs(include_action_mask=False, out=feats[t])
        masks[t].copy_(out.action_mask)
        lg, v = policy(feats[t], masks[t])
        a, lp = sample_categorical(lg)
        actions[t], logp[t], values[t] = a, lp, v
        out = env.step(a.to(torch.int8), auto_reset=True)
        rewards[t].copy_(out.reward)
        dones[t] = (out.terminated | out.truncated).bool()
    last_feats = env.flat_obs(include_action_mask=False)
    _, last_value = policy(last_feats, out.action_mask)
    return Batch(feats, masks, actions, logp, values, rewards, dones, last_value)


@torch.no_grad()
def gae(rewards, values, dones, last_value, gamma: float = 0.99, lam: float = 0.95):
    """Generalised advantage estimation over [T,B,N]; ``dones`` [T,B] cuts the bootstrap."""
    T = rewards.shape[0]
    adv = torch.zeros_like(rewards)
    running = torch.zeros_like(last_value)
    next_value = last_value
    for t in range(T - 1, -1, -1):
        nd = (~dones[t]).to(rewards.dtype).unsqueeze(-1)
        delta = rewards[t] + gamma * next_value * nd - values[t]
        running = delta + gamma * lam * nd * running
        adv[t] = running
        next_value = values[t]
    return adv, adv + values


def ppo_loss(lg, v, acts, old_logp, adv, ret, *, clip: float, vf_coeff: float, entropy_coeff: float,
             num_agents: int | None = None):
    """The clipped PPO loss of one minibatch (logits ``lg`` [..., A], values / actions / old log-probabilities /
    advantages / returns [...]) and its stats.  ``num_agents``: the rows are agent-fastest (flat row r of agent
    r % num_agents, the same number of rows per agent) and every mean is taken per agent, then summed over the agents:
    N independent learners, agent j's parameters getting agent j's mean loss's gradient."""
    dist = torch.distributions.Categorical(logits=lg)
    return ppo_objective(dist.log_prob(acts), dist.entropy(), v, old_logp, adv, ret, clip=clip, vf_coeff=vf_coeff,
                         entropy_coeff=entropy_coeff, num_agents=num_agents)


def ppo_objective(lp, entropy, v, old_logp, adv, ret, *, clip: float, vf_coeff: float, entropy_coeff: float,
                  num_agents: int | None = None):
    """:func:`ppo_loss` over precomputed log-probabilities ``lp`` and entropies ``entropy`` of the taken actions [...]:
    the clipped surrogate, plus ``vf_coeff`` times the value loss, minus ``entropy_coeff`` times the mean entropy (for
    a joint action, ``lp`` and ``entropy`` are the sums over its independent parts)."""
    ratio = torch.exp(lp - old_logp)
    surr = torch.min(ratio * adv, torch.clamp(ratio, 1 - clip, 1 + clip) * adv)
    mean = (lambda x: x.mean()) if num_agents is None else (lambda x: x.reshape(-1, num_agents).mean(0).sum())  # noqa: E731
    vf = mean((v - ret).pow(2))
    ent = mean(entropy)
    policy_loss = -mean(surr)
    loss = policy_loss + vf_coeff * vf - entropy_coeff * ent
    return loss, {"loss": float(loss.detach()), "vf_loss": float(vf.detach()), "entropy": float(ent.detach()),
                  "policy_loss": float(policy_loss.detach())}


def normalize_advantages(adv: torch.Tensor, per_agent: bool) -> torch.Tensor:
    """(adv - mean) / (std + 1e-8) over the whole [T,B,N] block, or per agent (over T and B) for per-agent policies."""
    if per_agent:
        return (adv - adv.mean((0, 1))) / (adv.std((0, 1)) + 1e-8)
    return (adv - adv.mean()) / (adv.std() + 1e-8)


def draw_permutation(n: int, device, generator: torch.Generator | None = None) -> torch.Tensor:
    """torch.randperm(n) on ``device`` from ``generator`` (the global RNG by default), drawn where the generator lives."""
    if generator is None or generator.device == torch.device(device):
        return torch.randperm(n, device=device, generator=generator)
    return torch.randperm(n, generator=generator).to(device)


def per_agent_minibatches(n_per_agent: int, N: int, size: int, device, generator: torch.Generator | None = None):
    """One epoch of a per-agent learner's minibatches: for every agent j (in order) a permutation of its
    ``n_per_agent`` samples, then per step ``size`` of each agent's samples.  Yields [size', N] sample numbers s of
    each agent (column j: agent j's), size' = size except for a shorter last step."""
    perm = torch.stack([draw_permutation(n_per_agent, device, generator) for _ in range(N)], dim=1)
    for i in range(0, n_per_agent, size):
        yield perm[i:i + size]


def ppo_update(policy, optimizer, batch: Batch, *, clip: float = 0.05, vf_coeff: float = 0.5,
               entropy_coeff: float = 0.001, epochs: int = 12, minibatch: int = 1024, gamma: float = 0.99,
               lam: float = 0.95, max_minibatches: int | None = None, generator: torch.Generator | None = None) -> dict:
    """PPO epochs over a :class:`Batch` / :class:`CompactBatch`.  ``generator`` (optional) draws the minibatch
    permutations.  A :class:`PerAgentActionMaskPolicy` is trained as N independent learners run in lockstep: each
    agent's advantages are normalised over its own samples; every step takes ``minibatch`` of agent j's samples for
    every j (one permutation per agent and epoch, drawn in agent order), laid out agent-fastest; the loss is the sum of
    the per-agent mean losses, so one element-wise optimizer over the stacked parameters is N independent ones."""
    adv, ret = gae(batch.rewards, batch.values, batch.dones, batch.last_value, gamma, lam)
    per_agent = isinstance(policy, PerAgentActionMaskPolicy)
    N = batch.actions.shape[-1]
    compact = isinstance(batch, CompactBatch)
    feats = None if compact else batch.features.reshape(-1, batch.features.shape[-1])
    masks = batch.masks.reshape(-1, batch.masks.shape[-1])
    acts, old_logp = batch.actions.reshape(-1), batch.logp.reshape(-1)
    adv = normalize_advantages(adv, per_agent).reshape(-1)
    ret = ret.reshape(-1)
    n = acts.shape[0]
    if per_agent and policy.num_agents != N:
        raise ValueError(f"the policy has {policy.num_agents} agents, the batch {N}")

    def minibatches():
        if per_agent:   # sample s of agent j is flat row s * N + j
            cols = torch.arange(N, device=acts.device)
            for s in per_agent_minibatches(n // N, N, minibatch, acts.device, generator):
                yield (s * N + cols).reshape(-1)
        else:
            perm = draw_permutation(n, acts.device, generator)
            for i in range(0, n, minibatch):
                yield perm[i:i + minibatch]

    stats, done_mb = {}, 0
    for _ in range(epochs):
        for idx in minibatches():
            lg, v = policy(batch.features_of(idx) if compact else feats[idx], masks[idx])
            loss, stats = ppo_loss(lg, v, acts[idx], old_logp[idx], adv[idx], ret[idx], clip=clip, vf_coeff=vf_coeff,
                                   entropy_coeff=entropy_coeff, num_agents=N if per_agent else None)
            optimizer.zero_grad(set_to_none=True)
            loss.backward()
            optimizer.step()
            done_mb += 1
            if max_minibatches is not None and done_mb >= max_minibatches:
                return stats
    return stats


def benchmark(num_envs: int = 65536, steps: int = 64, device: str = "cuda:0") -> dict:
    """BASELINE config 5: env-only vs policy+env loop throughput (agent-steps/s) on one GPU."""
    from . import maps
    from .batched_env import BatchedMapfEnv

    cfg = {"num_agents": 16, "sensor_range": 2, "steps_per_episode": 256, "lifelong_mapf": True, "seed": 999,
           "grid": maps.random_obstacle_grid(32, 32, 0.30, 2026, min_free=32)}
    env = BatchedMapfEnv(cfg, num_envs, device)
    env.reset()
    policy = ActionMaskPolicy(env.flat_obs_dim(include_action_mask=False)).to(env.device)
    collect(env, policy, 4)  # warm-up
    torch.cuda.synchronize(env.device)
    t0 = time.perf_counter()
    collect(env, policy, steps)
    torch.cuda.synchronize(env.device)
    loop_s = time.perf_counter() - t0
    a = env.sample_actions(masked=True)
    env.fuse_sampler("masked")
    for _ in range(4):
        env.step(a, auto_reset=True)
    torch.cuda.synchronize(env.device)
    t0 = time.perf_counter()
    for _ in range(steps):
        env.step(a, auto_reset=True)
    torch.cuda.synchronize(env.device)
    env_s = time.perf_counter() - t0
    from .policy_kernels import FusedPolicy

    env.fuse_sampler(None)
    fused = FusedPolicy(policy, env)
    res = {}
    for name, compact in (("fused_policy_loop", False), ("fused_policy_loop_compact", True)):
        collector = FusedCollector(env, fused, steps, compact=compact)
        collector.collect()
        torch.cuda.synchronize(env.device)
        t0 = time.perf_counter()
        collector.collect()
        torch.cuda.synchronize(env.device)
        res[name] = time.perf_counter() - t0
        del collector
    n = num_envs * env.N * steps
    return {"envs": num_envs, "agents": env.N, "steps": steps, "env_only_agent_steps_per_s": n / env_s,
            "policy_loop_agent_steps_per_s": n / loop_s, "fused_policy_loop_agent_steps_per_s": n / res["fused_policy_loop"],
            "fused_policy_loop_compact_agent_steps_per_s": n / res["fused_policy_loop_compact"]}


if __name__ == "__main__":
    import json

    print(json.dumps(benchmark()))
