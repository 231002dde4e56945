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

    def forward(self, features: torch.Tensor, action_mask: torch.Tensor):
        """features [..., F] float, action_mask [..., A] (0/1 of any dtype) -> (masked logits, value)."""
        z = self.trunk(features.float())
        logits = self.logits(z)
        value = self.value(z).squeeze(-1)
        if self.no_masking:
            return logits, value
        inf_mask = torch.clamp(torch.log(action_mask.to(logits.dtype) + 1e-6), min=FLOAT_MIN)
        return logits + inf_mask, value


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
            check(lib.mapf_policy_act(C.byref(a), stream))
            check(lib.mapf_step(h, self._actions_ptr, None, None, C.byref(self._couts[t]), 1, stream))
        fused.counter += 1
        a = self._pargs[self.T]
        a.counter = fused.counter
        check(lib.mapf_policy_act(C.byref(a), stream))
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


def ppo_update(policy, optimizer, batch: Batch, *, clip: float = 0.05, vf_coeff: float = 0.5,
               entropy_coeff: float = 0.001, epochs: int = 12, minibatch: int = 1024, gamma: float = 0.99,
               lam: float = 0.95, max_minibatches: int | None = None) -> dict:
    adv, ret = gae(batch.rewards, batch.values, batch.dones, batch.last_value, gamma, lam)
    compact = isinstance(batch, CompactBatch)
    feats = None if compact else batch.features.reshape(-1, batch.features.shape[-1])
    masks = batch.masks.reshape(-1, batch.masks.shape[-1])
    acts, old_logp = batch.actions.reshape(-1), batch.logp.reshape(-1)
    adv, ret = adv.reshape(-1), ret.reshape(-1)
    adv = (adv - adv.mean()) / (adv.std() + 1e-8)
    n = acts.shape[0]
    stats, done_mb = {}, 0
    for _ in range(epochs):
        perm = torch.randperm(n, device=acts.device)
        for i in range(0, n, minibatch):
            idx = perm[i:i + minibatch]
            lg, v = policy(batch.features_of(idx) if compact else feats[idx], masks[idx])
            dist = torch.distributions.Categorical(logits=lg)
            lp = dist.log_prob(acts[idx])
            ratio = torch.exp(lp - old_logp[idx])
            surr = torch.min(ratio * adv[idx], torch.clamp(ratio, 1 - clip, 1 + clip) * adv[idx])
            vf = (v - ret[idx]).pow(2).mean()
            ent = dist.entropy().mean()
            loss = -surr.mean() + vf_coeff * vf - entropy_coeff * ent
            optimizer.zero_grad(set_to_none=True)
            loss.backward()
            optimizer.step()
            stats = {"loss": float(loss), "vf_loss": float(vf), "entropy": float(ent),
                     "policy_loss": float(-surr.mean())}
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
