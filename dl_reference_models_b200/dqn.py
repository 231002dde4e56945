"""DQN for the shared and per-agent MLP policies: device-resident prioritized replay, a fused epsilon-greedy collector and
a double-DQN learner.

The reference trains with RLlib's PPO, IMPALA and DQN (``src/agents/{ppo,impala,dqn}.py``, SURVEY §2 row 6).  This
module is the DQN side, for the two module types whose action space is RLlib's ``Discrete(5)``:
:class:`rollout.ActionMaskPolicy` (CTDE) and :class:`rollout.PerAgentActionMaskPolicy` (DTE, N learners in lockstep).

* The Q-network is the module read as a dueling network: the logits head is the advantage A[5], the value head V,
  Q = V + (A - mean(A)) with the mean over all 5 actions (RLlib's dueling combination), masked Q =
  ``where(mask, Q, FLOAT_MIN)`` (:func:`q_values`); ``no_masking`` modules use Q as it is.
* :class:`ReplayBuffer` -- a ring of K env steps holding the compact observation rows, int8 actions, f32 rewards and
  uint8 dones, with a prioritized sum tree over its transitions.  CUDA buffers run the ``mapf_replay_*`` kernels; CPU
  buffers a PyTorch reference (f64 ``cumsum`` + ``searchsorted``, direct leaf writes), the tests' reference.
* :class:`DqnCollector` -- three calls per env step and no host sync: ``mapf_q_act`` (epsilon-greedy, reads ring row
  t, writes the ring's action row t), ``mapf_step`` (writes the next observation into row t + 1, reward and done into
  row t) and ``mapf_replay_advance`` (slot t becomes drawable, slot t + 1 is cleared).
* :func:`dqn_update` -- double DQN with the Huber loss and importance weights, gradients averaged over the ranks, a
  global-norm clip, then new priorities |TD error| + 1e-6.  :func:`sync_target` is the caller's call.

Done = ``terminated``: in this env a time-limit truncation sets both flags (SURVEY F6), so no transition bootstraps from
an observation the auto-reset overwrote.

Defaults: gamma 0.99 is the reference's.  Double Q, dueling, the Huber loss (delta 1), grad clip 40, alpha 0.6, beta
0.4, priority |TD error| + 1e-6, new transitions at the largest priority seen so far (1.0 at first) and the hard target
update (tau 1) are RLlib's ``DQNConfig`` defaults: the reference's own ``dqn.py`` overrides, and ray, are not in this
tree.  The minibatch (1024 instead of RLlib's 32) and the capacity counted in env steps (64, instead of 50 000
transitions) are this project's: one env step here is up to a million agent transitions.  Uniform replay is
``alpha = 0``.

``python -m dl_reference_models_b200.dqn`` prints the collector and learner rates and a learning sanity figure as one
JSON line.
"""
from __future__ import annotations

import ctypes as C
import math

import torch
import torch.nn.functional as F_

from . import _native as nat
from .impala import clip_grad_norm_per_agent_
from .recurrent import allreduce_gradients
from .rollout import FLOAT_MIN, PerAgentActionMaskPolicy, observation_rows


def q_values(policy, features: torch.Tensor, mask: torch.Tensor) -> torch.Tensor:
    """The masked dueling Q [..., 5] of an :class:`rollout.ActionMaskPolicy` / :class:`rollout.PerAgentActionMaskPolicy`
    (per agent: flat row r of agent r % N): Q = V + (A - mean(A)), FLOAT_MIN where ``mask`` is 0 (not with
    ``no_masking``)."""
    adv, value = policy.heads(features)
    q = value.unsqueeze(-1) + (adv - adv.mean(-1, keepdim=True))
    if policy.no_masking:
        return q
    return torch.where(mask != 0, q, torch.full_like(q, FLOAT_MIN))


@torch.no_grad()
def sync_target(policy, target, tau: float = 1.0):
    """target <- tau * policy + (1 - tau) * target, parameter by parameter (tau = 1: a copy, RLlib's hard update)."""
    for p, q in zip(policy.parameters(), target.parameters()):
        if tau == 1.0:
            q.copy_(p)
        else:
            q.mul_(1.0 - tau).add_(p, alpha=tau)


class ReplayBuffer:
    """A ring of ``capacity_steps`` (K) env steps of ``env`` (B envs x N agents) and a prioritized sum tree over its
    transitions.  Transition (slot k, env b, agent j) has the flat index (k B + b) N + j, the row order of
    ``observation_rows(env, K)``: its observation is ring row k, its next observation row (k + 1) mod K, its action,
    reward and done (``terminated``) are row k of :attr:`actions` / :attr:`rewards` / :attr:`dones`.  At most K - 1
    slots hold a complete transition; the others' leaves are 0 and never drawn.  ``per_agent``: every draw i comes
    from agent i mod N's transitions, weighted by that agent's own minimum (a per-agent learner's minibatch).  On a
    CUDA env the tree lives on the device (``mapf_replay_*``); on a CPU env (an object with ``B``, ``N``, ``V``,
    ``device``, ``include_blocking_pressure`` and the observation channels in ``out``) a PyTorch reference keeps the
    leaves only."""

    def __init__(self, env, capacity_steps: int = 64, alpha: float = 0.6, per_agent: bool = False, seed: int = 0):
        K = int(capacity_steps)
        if K < 2:
            raise ValueError(f"capacity_steps {K} must be >= 2 (a transition needs its next observation's row)")
        if not (math.isfinite(alpha) and alpha >= 0):
            raise ValueError(f"alpha {alpha} must be finite and >= 0")
        self.env, self.K, self.B, self.N = env, K, int(env.B), int(env.N)
        self.alpha, self.per_agent = float(alpha), bool(per_agent)
        self.with_bp = bool(env.include_blocking_pressure)
        dev = self.device = torch.device(env.device)
        self.rows = observation_rows(env, K)
        self.actions = torch.zeros((K, self.B, self.N), dtype=torch.int8, device=dev)
        self.rewards = torch.zeros((K, self.B, self.N), dtype=torch.float32, device=dev)
        self.dones = torch.zeros((K, self.B), dtype=torch.uint8, device=dev)
        self.head = 0     # the ring row that holds the env's current observation
        self.filled = 0   # complete slots
        self.max_priority = torch.ones(1, dtype=torch.float32, device=dev)
        self.seed, self.counter = int(seed) & (2 ** 64 - 1), 0
        if dev.type == "cuda":
            self._lib = nat.lib()
            L = int(self._lib.mapf_replay_tree_leaves(self.B, self.N, K))
            if L < 0:
                raise nat.MapfError(L, self._lib.mapf_last_error().decode())
            self._leaves = torch.zeros(L, dtype=torch.float32, device=dev)
            self.sums = torch.zeros(L, dtype=torch.float64, device=dev)
            self.mins = torch.full((L,), math.inf, dtype=torch.float32, device=dev)
            p = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
            self._tree = nat.MapfReplayTree(num_envs=self.B, num_agents=self.N, capacity=K, leaves=p(self._leaves),
                                            sums=p(self.sums), mins=p(self.mins), max_priority=p(self.max_priority))
            self._pad = tuple(1 << (x - 1).bit_length() for x in (self.N, K, self.B))
        else:
            self._leaves = torch.zeros((self.N, K, self.B), dtype=torch.float32, device=dev)

    @property
    def is_cuda(self) -> bool:
        return self.device.type == "cuda"

    @property
    def num_transitions(self) -> int:
        return self.filled * self.B * self.N

    def leaves(self) -> torch.Tensor:
        """The tree's leaves p^alpha as [N, K, B] (agent, slot, env): a view."""
        if self.is_cuda:
            return self._leaves.view(self._pad)[:self.N, :self.K, :self.B]
        return self._leaves

    def advance_args(self, complete: int, clear: int) -> nat.MapfReplayAdvanceArgs:
        return nat.MapfReplayAdvanceArgs(tree=self._tree, complete=int(complete), clear=int(clear), alpha=self.alpha,
                                         reserved=0)

    def advance(self, complete: int, clear: int, stream=None):
        """Slot ``complete`` gets max_priority^alpha at every (env, agent), slot ``clear`` gets 0 (the collector's
        call, once per env step; this does not move :attr:`head`)."""
        if self.is_cuda:
            st = C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream) if stream is None else stream
            nat.check(self._lib.mapf_replay_advance(C.byref(self.advance_args(complete, clear)), st))
        else:
            self._leaves[:, complete] = self.max_priority.pow(self.alpha)
            self._leaves[:, clear] = 0.0

    def sample(self, M: int, beta: float = 0.4, *, generator: torch.Generator | None = None, counter: int | None = None,
               uniforms: torch.Tensor | None = None, uniforms_out: torch.Tensor | None = None):
        """M proportional draws (RLlib's ``_sample_proportional``) -> (int64 flat indices [M], float32 importance
        weights [M]), w = (p_i / p_min)^-beta (RLlib's (P(i) n)^-beta over its maximum; n and the total cancel).  CUDA:
        Philox keyed by (the buffer's seed, ``counter`` (default: the next of the buffer's), draw); ``uniforms_out``
        float64 [M] receives the uniforms.  CPU: the uniforms are ``uniforms`` or drawn from ``generator``."""
        M = int(M)
        if self.filled == 0:
            raise ValueError("the replay buffer holds no complete transition yet")
        if self.is_cuda:
            if counter is None:
                self.counter += 1
                counter = self.counter
            idx = torch.empty(M, dtype=torch.int64, device=self.device)
            w = torch.empty(M, dtype=torch.float32, device=self.device)
            p = lambda t: None if t is None else C.c_void_p(t.data_ptr())  # noqa: E731
            a = nat.MapfReplaySampleArgs(tree=self._tree, M=M, seed=self.seed, counter=int(counter), beta=float(beta),
                                         per_agent=int(self.per_agent), indices=p(idx), weights=p(w),
                                         uniforms=p(uniforms_out), reserved=0)
            nat.check(self._lib.mapf_replay_sample(C.byref(a), C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)))
            return idx, w
        u = torch.rand(M, generator=generator, dtype=torch.float64) if uniforms is None else uniforms.double()
        N, KB = self.N, self.K * self.B
        P = self._leaves.reshape(N, KB).double() if self.per_agent else self._leaves.reshape(1, -1).double()
        j = torch.arange(M) % N if self.per_agent else torch.zeros(M, dtype=torch.int64)
        cs = P.cumsum(1)
        total = cs[:, -1]
        last = torch.searchsorted(cs, total.unsqueeze(1).contiguous()).squeeze(1)   # each row's last nonzero leaf
        # one search per row over that row's draws: gathering cs[j] would copy a whole row per draw (M x K B N f64)
        pos = torch.empty(M, dtype=torch.int64)
        for r in range(cs.shape[0]):
            sel = j == r
            pos[sel] = torch.searchsorted(cs[r], u[sel] * total[r], right=True)
        pos = torch.minimum(pos, last[j])
        if self.per_agent:
            agent, k, b = j, pos // self.B, pos % self.B
        else:
            agent, k, b = pos // KB, pos % KB // self.B, pos % self.B
        p_min = torch.where(P > 0, P, torch.full_like(P, math.inf)).min(1).values
        w = (P[j, pos] / p_min[j]).pow(-float(beta)).float()
        return (k * self.B + b) * N + agent, w

    def update_priorities(self, indices: torch.Tensor, td_abs: torch.Tensor):
        """Leaf = (|delta| + 1e-6)^alpha for every in-range index whose slot holds a transition (the largest value among
        duplicates), max_priority = max(max_priority, |delta| + 1e-6) over them."""
        idx = indices.reshape(-1).to(device=self.device, dtype=torch.int64).contiguous()
        td = td_abs.reshape(-1).to(device=self.device, dtype=torch.float32).contiguous()
        if self.is_cuda:
            a = nat.MapfReplayUpdateArgs(tree=self._tree, M=int(idx.numel()), indices=C.c_void_p(idx.data_ptr()),
                                         td_abs=C.c_void_p(td.data_ptr()), alpha=self.alpha, reserved=0)
            nat.check(self._lib.mapf_replay_update(C.byref(a), C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)))
            return
        BN = self.B * self.N
        ok = (idx >= 0) & (idx < self.K * BN)
        i, t = idx[ok], td[ok]
        k, b, j = i // BN, i % BN // self.N, i % self.N
        flat = self._leaves.view(-1)
        lin = (j * self.K + k) * self.B + b
        held = flat[lin] > 0
        lin, p = lin[held], t[held] + 1e-6
        if lin.numel():
            flat[lin] = 0.0
            flat.scatter_reduce_(0, lin, p.pow(self.alpha), "amax")
            self.max_priority.copy_(torch.maximum(self.max_priority, p.max().reshape(1)))

    def _split(self, indices, next: bool):
        BN = self.B * self.N
        k, r = indices // BN, indices % BN
        return ((k + 1) % self.K if next else k), r

    def features_of(self, indices: torch.Tensor, next: bool = False) -> torch.Tensor:
        """Float32 feature rows (window, goal delta, pressure) of the transitions' observations (``next``: of their
        next observations)."""
        k, r = self._split(indices, next)
        K, BN = self.K, self.B * self.N
        lo = self.rows["local_obs"]
        parts = [lo.view(K, BN, lo.shape[-1] * lo.shape[-2])[k, r].float(), self.rows["goal_delta"].view(K, BN, 2)[k, r]]
        if self.with_bp:
            parts.append(self.rows["blocking_prev"].view(K, BN)[k, r].float().unsqueeze(-1))
        return torch.cat(parts, dim=-1)

    def masks_of(self, indices: torch.Tensor, next: bool = False) -> torch.Tensor:
        """int8 [M, 5] action masks of the transitions' observations (``next``: of their next observations)."""
        k, r = self._split(indices, next)
        return self.rows["action_mask"].view(self.K, self.B * self.N, 5)[k, r]

    def transitions_of(self, indices: torch.Tensor):
        """(int64 actions, float32 rewards, bool dones) [M] of the transitions."""
        k, r = self._split(indices, False)
        BN = self.B * self.N
        return (self.actions.view(self.K, BN)[k, r].long(), self.rewards.view(self.K, BN)[k, r],
                self.dones[k, r // self.N] != 0)


class DqnCollector:
    """Epsilon-greedy env steps into a CUDA :class:`ReplayBuffer`: per step ``mapf_q_act`` on ring row t (actions into
    the ring's action row t), ``mapf_step(auto_reset=1)`` with its observation channels written into row (t + 1) mod K
    and its reward and done into row t, and ``mapf_replay_advance(complete=t, clear=(t + 1) mod K)``; the argument
    blocks are built once.  The ring head carries over between collects: each collect starts by copying the env's
    current observation into the head row, and afterwards the env's buffers show the latest observation again (so do
    not step the env between collects of one buffer)."""

    def __init__(self, env, fused_q, buffer: ReplayBuffer):
        if not buffer.is_cuda or buffer.env is not env or fused_q.env is not env:
            raise ValueError("the collector needs a CUDA ReplayBuffer and a FusedQPolicy of this env")
        if fused_q.per_agent != buffer.per_agent:
            raise ValueError("a per-agent Q-network needs a per-agent buffer, a shared one a shared buffer")
        self.env, self.fused, self.buffer = env, fused_q, buffer
        K, rows = buffer.K, buffer.rows
        self._qargs = [fused_q.args({k: rows[k][t] for k in rows}, 0.0, buffer.actions[t]) for t in range(K)]
        self._trunc = torch.zeros(env.B, dtype=torch.uint8, device=env.device)   # truncation also sets terminated

        def dst(k, t):
            if k == "reward":
                return buffer.rewards[t]
            if k == "terminated":
                return buffer.dones[t]
            if k == "truncated":
                return self._trunc
            return rows[k][(t + 1) % K] if k in rows else env.out[k]

        self._couts = [nat.MapfOutputs(**{k: dst(k, t).data_ptr() for k in nat.OUTPUT_FIELDS}) for t in range(K)]
        self._adv = [buffer.advance_args(t, (t + 1) % K) for t in range(K)]
        self._actions = [C.c_void_p(buffer.actions[t].data_ptr()) for t in range(K)]
        self._lib = nat.lib()

    @torch.no_grad()
    def collect(self, steps: int, epsilon: float):
        """``steps`` env steps with exploration probability ``epsilon``."""
        env, fused, buf, lib = self.env, self.fused, self.buffer, self._lib
        if getattr(env, "_fused", 0):
            raise RuntimeError("turn the env's fused uniform sampler off (fuse_sampler(None)) before a policy rollout")
        if not (0.0 <= epsilon <= 1.0):
            raise ValueError(f"epsilon {epsilon} outside [0, 1]")
        stream, h, check = env._stream(), env._h, nat.check
        for k, r in buf.rows.items():
            r[buf.head].copy_(env.out[k])
        for _ in range(int(steps)):
            t = buf.head
            fused.counter += 1
            a = self._qargs[t]
            a.counter, a.epsilon = fused.counter, float(epsilon)
            check(fused._act(C.byref(a), stream))
            check(lib.mapf_step(h, self._actions[t], None, None, C.byref(self._couts[t]), 1, stream))
            check(lib.mapf_replay_advance(C.byref(self._adv[t]), stream))
            buf.head = (t + 1) % buf.K
            buf.filled = min(buf.filled + 1, buf.K - 1)
        for k, r in buf.rows.items():   # the env's own buffers show the latest observation again
            env.out[k].copy_(r[buf.head])


def dqn_update(policy, target, optimizer, buffer: ReplayBuffer, *, updates: int = 1, minibatch: int = 1024,
               gamma: float = 0.99, beta: float = 0.4, double_q: bool = True, grad_clip: float | None = 40.0,
               world_size: int = 1, group=None, generator: torch.Generator | None = None) -> dict:
    """``updates`` DQN steps on ``buffer``.  Each: sample ``minibatch`` transitions (per-agent modules: ``minibatch``
    of every agent's own, agent-fastest, from a ``per_agent`` buffer); Q(s, a) with ``policy``; under ``no_grad`` the
    target r + gamma (1 - done) Q_target(s', argmax over legal a' of Q_policy(s', a')) (``double_q=False``: the largest
    legal Q_target(s', a')); loss = mean(w huber(delta)) (per agent: the sum of the per-agent means); backward, the mean
    over ``world_size`` ranks, the global-norm clip (per agent for per-agent modules), the optimizer step, then the
    sampled transitions' priorities |delta| + 1e-6.  ``generator`` draws a CPU buffer's uniforms.  Raises
    ``ValueError`` on an empty buffer or an agent-count mismatch and ``FloatingPointError``, before any parameter or
    priority changes, when a TD error is not finite."""
    per_agent = isinstance(policy, PerAgentActionMaskPolicy)
    N = buffer.N
    if per_agent and (policy.num_agents != N or not buffer.per_agent):
        raise ValueError(f"the per-agent policy has {policy.num_agents} agents; it needs a per_agent buffer of as many "
                         f"(this one: {N} agents, per_agent={buffer.per_agent})")
    if buffer.num_transitions == 0:
        raise ValueError("the replay buffer holds no complete transition yet")
    params = list(policy.parameters())
    M = int(minibatch) * (N if per_agent else 1)
    mean = (lambda x: x.mean()) if not per_agent else (lambda x: x.reshape(-1, N).mean(0).sum())  # noqa: E731
    stats = {}
    for _ in range(int(updates)):
        idx, w = buffer.sample(M, beta, generator=generator)
        feats, masks = buffer.features_of(idx), buffer.masks_of(idx)
        acts, rew, done = buffer.transitions_of(idx)
        q_sa = q_values(policy, feats, masks).gather(-1, acts.unsqueeze(-1)).squeeze(-1)
        with torch.no_grad():
            nf, nm = buffer.features_of(idx, next=True), buffer.masks_of(idx, next=True)
            q_t = q_values(target, nf, nm)
            if double_q:
                q_next = q_t.gather(-1, q_values(policy, nf, nm).argmax(-1, keepdim=True)).squeeze(-1)
            else:
                q_next = q_t.max(-1).values
            y = rew + gamma * (~done).to(rew.dtype) * q_next
        td = q_sa - y
        if not bool(torch.isfinite(td).all()):
            raise FloatingPointError("non-finite TD error: the priorities and parameters are left as they are")
        loss = mean(w * F_.huber_loss(q_sa, y, reduction="none", delta=1.0))
        optimizer.zero_grad(set_to_none=True)
        loss.backward()
        allreduce_gradients(policy, world_size, group)
        if grad_clip is not None:
            if per_agent:
                clip_grad_norm_per_agent_(params, grad_clip, N)
            else:
                torch.nn.utils.clip_grad_norm_(params, grad_clip)
        optimizer.step()
        td_abs = td.detach().abs()
        buffer.update_priorities(idx, td_abs)
        stats = {"loss": float(loss.detach()), "mean_q": float(q_sa.detach().mean()), "mean_td_abs": float(td_abs.mean())}
    return stats


def _greedy_success(env_config: dict, policy, episodes: int, device) -> float:
    """Success rate of ``policy`` played greedily (epsilon 0) by the batched evaluator through a callable."""
    from .evaluate import evaluate
    from .policy_kernels import FusedQPolicy

    fused = {}

    def greedy(env, out):
        if id(env) not in fused:
            fused[id(env)] = FusedQPolicy(policy, env)
        return fused[id(env)].act(out, 0.0)

    return float(evaluate(env_config, episodes, policy=greedy, device=device).success_rate)


def benchmark(num_envs: int = 65536, num_agents: int = 16, capacity: int = 64, steps: int = 64, updates: int = 50,
              sanity_rounds: int = 150, device: str = "cuda:0") -> dict:
    """C3 (num_envs x 16 agents, 32x32 map with 30 % obstacles, seed 2026, sensor range 2, lifelong, K = ``capacity``):
    env-only, :class:`DqnCollector` and ``FusedCollector(compact=True)`` env-steps/s over ``steps`` steps (host clock
    around work that ends in a device synchronise, after a warm-up); :func:`dqn_update` updates/s at minibatch 1024,
    shared and per-agent; and a learning sanity figure: the greedy success rate on a small episodic map before and
    after ``sanity_rounds`` rounds of one collect step and one update."""
    import time

    from . import maps
    from .batched_env import BatchedMapfEnv
    from .policy_kernels import FusedPolicy, FusedQPolicy
    from .rollout import ActionMaskPolicy, FusedCollector

    def timed(fn, n):
        fn()
        torch.cuda.synchronize(device)
        t0 = time.perf_counter()
        for _ in range(n):
            fn()
        torch.cuda.synchronize(device)
        return (time.perf_counter() - t0) / n

    grid = maps.random_obstacle_grid(32, 32, 0.30, 2026, min_free=32)
    cfg = {"num_agents": num_agents, "sensor_range": 2, "steps_per_episode": 256, "lifelong_mapf": True, "seed": 999,
           "grid": grid}
    res = {"envs": num_envs, "agents": num_agents, "capacity_steps": capacity, "steps": steps, "map": [32, 32]}
    env = BatchedMapfEnv(cfg, num_envs, device)
    env.reset()
    F = env.flat_obs_dim(include_action_mask=False)
    torch.manual_seed(0)
    pol = ActionMaskPolicy(F).to(env.device)
    a = env.sample_actions(masked=True)
    env.fuse_sampler("masked")
    s = timed(lambda: [env.step(a, auto_reset=True) for _ in range(steps)], 1)
    res["env_only_env_steps_per_s"] = steps * num_envs / s
    env.fuse_sampler(None)
    col = FusedCollector(env, FusedPolicy(pol, env), steps, compact=True)
    s = timed(col.collect, 1)
    res["fused_collector_compact_env_steps_per_s"] = steps * num_envs / s
    del col
    for name, per_agent in (("shared", False), ("per_agent", True)):
        net = PerAgentActionMaskPolicy(num_agents, F).to(env.device) if per_agent else pol
        target = PerAgentActionMaskPolicy(num_agents, F).to(env.device) if per_agent else ActionMaskPolicy(F).to(env.device)
        sync_target(net, target)
        buf = ReplayBuffer(env, capacity, per_agent=per_agent)
        dc = DqnCollector(env, FusedQPolicy(net, env), buf)
        dc.collect(capacity, 0.1)   # fill the ring once
        s = timed(lambda: dc.collect(steps, 0.1), 1)
        res[f"dqn_collector_{name}_env_steps_per_s"] = steps * num_envs / s
        opt = torch.optim.Adam(net.parameters(), lr=5e-4)
        s = timed(lambda: dqn_update(net, target, opt, buf, updates=updates), 1)
        res[f"dqn_update_{name}_updates_per_s"] = updates / s
        del dc, buf
        torch.cuda.empty_cache()
    for k in list(res):
        if k.endswith("env_steps_per_s"):
            res[k.replace("env_steps", "agent_steps")] = res[k] * num_agents
    env.close()
    del env
    torch.cuda.empty_cache()
    res["learning_sanity"] = learning_sanity(sanity_rounds, device)
    return res


def learning_sanity(rounds: int = 150, device: str = "cuda:0") -> dict:
    """Greedy success rate on a small episodic map (12x12, 15 % obstacles, 2 agents, 32 steps per episode, 4096
    episodes) before and after ``rounds`` rounds of (one collect step of 4096 envs at epsilon 0.3, one update of
    minibatch 1024), target sync every 20 rounds, Adam lr 1e-3: reported, not asserted."""
    from . import maps
    from .batched_env import BatchedMapfEnv
    from .policy_kernels import FusedQPolicy
    from .rollout import ActionMaskPolicy

    cfg = {"num_agents": 2, "sensor_range": 2, "steps_per_episode": 32, "lifelong_mapf": False, "seed": 7,
           "grid": maps.random_obstacle_grid(12, 12, 0.15, 2026, min_free=8)}
    env = BatchedMapfEnv(cfg, 4096, device)
    env.reset()
    F = env.flat_obs_dim(include_action_mask=False)
    torch.manual_seed(0)
    net, target = ActionMaskPolicy(F).to(env.device), ActionMaskPolicy(F).to(env.device)
    sync_target(net, target)
    before = _greedy_success(dict(cfg, seed=11), net, 4096, device)
    buf = ReplayBuffer(env, 16)
    dc = DqnCollector(env, FusedQPolicy(net, env), buf)
    opt = torch.optim.Adam(net.parameters(), lr=1e-3)
    dc.collect(2, 0.3)
    for r in range(rounds):
        dc.collect(1, 0.3)
        dqn_update(net, target, opt, buf)
        dc.fused.refresh()
        if r % 20 == 19:
            sync_target(net, target)
    after = _greedy_success(dict(cfg, seed=11), net, 4096, device)
    return {"map": [12, 12], "agents": 2, "episodes": 4096, "rounds": rounds, "success_before": before,
            "success_after": after}


if __name__ == "__main__":
    import json
    import subprocess

    from dl_reference_models_b200 import dqn   # the package's functions, not this __main__ copy's

    r = dqn.benchmark()
    try:
        r["gpu"] = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                                   "-i", "0"], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as exc:
        r["gpu"] = f"nvidia-smi not readable: {exc}"
    print(json.dumps(r))
