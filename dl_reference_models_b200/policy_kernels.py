"""Rollout-loop CUDA kernels around the env step (BASELINE config 5): the action-mask MLP evaluated straight from the
env's output channels and sampled in one launch (``mapf_policy_act``: bf16 tensor-core MLP with f32 accumulation), the
same for the LSTM-64 recurrent policy (``mapf_lstm_policy_act``), both with a greedy (argmax) mode for evaluation and a
per-agent variant (one weight set per agent: ``mapf_policy_act_per_agent`` / ``mapf_lstm_policy_act_per_agent``), the
centralised CTE policy over the single-agent view with one joint draw (``mapf_cte_policy_act``) and its recurrent
variant (``mapf_cte_lstm_policy_act``), GAE as a backwards
scan (``mapf_gae``), IMPALA's V-trace targets as another (``mapf_vtrace``) and DQN's epsilon-greedy dueling Q head
over the MLP (``mapf_q_act``).  Thin ctypes wrappers; torch is the allocator / stream provider.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _native as nat


def _per_agent_kind(policy) -> str | None:
    """"mlp" for a :class:`rollout.PerAgentActionMaskPolicy`, "lstm" for a :class:`recurrent.PerAgentRecurrentPolicy`,
    None for any other module."""
    from .recurrent import PerAgentRecurrentPolicy
    from .rollout import PerAgentActionMaskPolicy

    return "mlp" if isinstance(policy, PerAgentActionMaskPolicy) else "lstm" if isinstance(policy, PerAgentRecurrentPolicy) else None


def _per_agent_arrays(policy, names):
    """float32 numpy copies of a per-agent module's stacked parameters ``names``, then per agent j the list of their
    [j] slices (the pack function's arguments for agent j)."""
    f = lambda t: np.ascontiguousarray(t.detach().float().cpu().numpy())  # noqa: E731
    stacked = [f(getattr(policy, n)) if isinstance(n, str) else f(n) for n in names]
    return [[np.ascontiguousarray(a[j]) for a in stacked] for j in range(policy.num_agents)]


class FusedPolicy:
    """Inference view of an :class:`rollout.ActionMaskPolicy` (two 64-wide ReLU layers, 5 logits + value), or of a
    :class:`rollout.PerAgentActionMaskPolicy` of that shape with one module per env agent (launched through
    ``mapf_policy_act_per_agent``, :attr:`entry`): call :meth:`refresh` after every optimizer step, :meth:`act` once
    per env step."""

    def __init__(self, policy, env, seed: int | None = None):
        self.policy, self.env = policy, env
        self._lib = nat.lib()
        self.F = int(env.flat_obs_dim(include_action_mask=False))
        self.with_bp = bool(env.include_blocking_pressure)
        assert self.F == env.V * env.V + 2 + (1 if self.with_bp else 0)
        self.per_agent = _per_agent_kind(policy) is not None
        if self.per_agent:
            if not FusedPolicy.matches(policy, env):
                raise ValueError("the fused kernel implements the reference's 64-64 action-mask MLP only, one module per "
                                 f"env agent: the policy has {policy.num_agents} agents of feature_dim "
                                 f"{policy.feature_dim}, hiddens {policy.hiddens}, {policy.num_actions} actions; the env "
                                 f"has {env.N} agents and {self.F} features")
        else:
            assert FusedPolicy.matches(policy, env), "the fused kernel implements the reference's 64-64 action-mask MLP"
            self._lin = [m for m in policy.trunk if isinstance(m, torch.nn.Linear)]
        self.entry = "mapf_policy_act_per_agent" if self.per_agent else "mapf_policy_act"
        self._act = getattr(self._lib, self.entry)
        n = int(self._lib.mapf_policy_weights_nbytes(self.F))
        if n < 0:
            raise nat.MapfError(n, self._lib.mapf_last_error().decode())
        self._block = n
        n *= policy.num_agents if self.per_agent else 1   # per agent: block j at j * n
        self._host = np.zeros(n, np.uint8)
        self._dev = torch.zeros(n, dtype=torch.uint8, device=env.device)
        B, N = env.B, env.N
        dev = env.device
        self.actions = torch.zeros((B, N), dtype=torch.int8, device=dev)
        self.actions64 = torch.zeros((B, N), dtype=torch.int64, device=dev)
        self.logp = torch.zeros((B, N), dtype=torch.float32, device=dev)
        self.value = torch.zeros((B, N), dtype=torch.float32, device=dev)
        self.seed = int(env.cfg.seed if seed is None else seed) & (2 ** 64 - 1)
        self.counter = 0
        self.refresh()

    @staticmethod
    def matches(policy, env) -> bool:
        """Whether the fused kernel implements ``policy`` (an :class:`rollout.ActionMaskPolicy`) at ``env``'s feature
        width: trunk Linear(F, 64)-ReLU-Linear(64, 64)-ReLU over F = V*V + 2 (+1 pressure) features, 5 logits."""
        F = env.V * env.V + 2 + (1 if env.include_blocking_pressure else 0)
        kind = _per_agent_kind(policy)
        if kind is not None:   # a rollout.PerAgentActionMaskPolicy: every agent's module has the reference's shape
            return (kind == "mlp" and policy.num_agents == env.N and policy.feature_dim == F and tuple(policy.hiddens) == (64, 64)
                    and policy.num_actions == 5)
        lin = [m for m in policy.trunk.modules() if isinstance(m, torch.nn.Linear)]
        return (len(lin) == 2 and lin[0].in_features == F and lin[0].out_features == 64 and lin[1].in_features == 64
                and lin[1].out_features == 64 and policy.logits.out_features == 5)

    def refresh(self):
        """Re-pack the module's current float32 parameters (bf16, padded; per agent: one block per agent) and upload
        them."""
        f = lambda t: np.ascontiguousarray(t.detach().float().cpu().numpy())  # noqa: E731
        if self.per_agent:
            p = self.policy
            per = _per_agent_arrays(p, [p.trunk_w[0], p.trunk_b[0], p.trunk_w[1], p.trunk_b[1], "logits_w", "logits_b",
                                        "value_w", "value_b"])
        else:
            per = [[f(self._lin[0].weight), f(self._lin[0].bias), f(self._lin[1].weight), f(self._lin[1].bias),
                    f(self.policy.logits.weight), f(self.policy.logits.bias), f(self.policy.value.weight),
                    f(self.policy.value.bias)]]
        for j, arrs in enumerate(per):
            nat.check(self._lib.mapf_policy_pack_weights(self.F, *[a.ctypes.data_as(C.c_void_p) for a in arrs],
                                                         C.c_void_p(self._host.ctypes.data + j * self._block)))
        self._dev.copy_(torch.from_numpy(self._host))

    def act(self, out, logits_out: torch.Tensor | None = None, features_out: torch.Tensor | None = None,
            logp: torch.Tensor | None = None, value: torch.Tensor | None = None, actions64: torch.Tensor | None = None,
            mask_out: torch.Tensor | None = None, greedy: bool = False):
        """One launch: features from ``out`` (the env's StepOutput) -> MLP -> masked categorical draw (``greedy``: the
        first argmax of the masked logits instead, as RLlib's ``forward_inference``).
        Returns (actions int8 [B,N], logp, value); optional tensors receive the masked logits / the float feature
        block / a copy of the action masks (the rollout buffer's rows, so the loop needs no copy launches)."""
        env = self.env
        p = lambda t: None if t is None else C.c_void_p(t.data_ptr())  # noqa: E731
        logp = self.logp if logp is None else logp
        value = self.value if value is None else value
        actions64 = self.actions64 if actions64 is None else actions64
        self.counter += 1
        args = nat.MapfPolicyArgs(
            num_envs=env.B, num_agents=env.N, v2=env.V * env.V, feature_dim=self.F,
            no_masking=int(bool(self.policy.no_masking)), greedy=int(bool(greedy)), seed=self.seed, counter=self.counter,
            env_id_base=int(env.cfg.env_id_base), local_obs=p(out.local_obs), goal_delta=p(out.goal_delta),
            blocking_prev=p(out.blocking_prev) if self.with_bp else None, action_mask=p(out.action_mask),
            weights=p(self._dev), actions=p(self.actions), actions64=p(actions64), logp=p(logp), value=p(value),
            logits_out=p(logits_out), features_out=p(features_out), action_mask_out=p(mask_out))
        nat.check(self._act(C.byref(args), env._stream()))
        return self.actions, logp, value


class FusedQPolicy(FusedPolicy):
    """The same MLP read as a dueling Q network for DQN (``mapf_q_act`` / ``mapf_q_act_per_agent``, :attr:`entry`): the
    logits head is the advantage A, the value head V, Q = V + A - mean(A), masked to FLOAT_MIN where an action is
    illegal, then an epsilon-greedy choice (one Philox block per agent, keyed apart from the policy draws).  Packing,
    :meth:`refresh` and the accepted modules are :class:`FusedPolicy`'s."""

    def __init__(self, policy, env, seed: int | None = None):
        super().__init__(policy, env, seed)
        self.entry = "mapf_q_act_per_agent" if self.per_agent else "mapf_q_act"
        self._act = getattr(self._lib, self.entry)

    def args(self, channels: dict, epsilon: float, actions: torch.Tensor, q_out: torch.Tensor | None = None) -> nat.MapfQActArgs:
        """The argument block of one launch (counter 0; set ``.counter`` before launching): ``channels`` maps
        local_obs / goal_delta / blocking_prev / action_mask to device tensors, ``actions`` int8 [B,N] receives the
        choice, ``q_out`` (optional) float32 [B,N,5] the masked Q."""
        env = self.env
        p = lambda t: None if t is None else C.c_void_p(t.data_ptr())  # noqa: E731
        return nat.MapfQActArgs(
            num_envs=env.B, num_agents=env.N, v2=env.V * env.V, feature_dim=self.F,
            no_masking=int(bool(self.policy.no_masking)), epsilon=float(epsilon), seed=self.seed, counter=0,
            env_id_base=int(env.cfg.env_id_base), local_obs=p(channels["local_obs"]), goal_delta=p(channels["goal_delta"]),
            blocking_prev=p(channels["blocking_prev"]) if self.with_bp else None, action_mask=p(channels["action_mask"]),
            weights=p(self._dev), actions=p(actions), q_out=p(q_out), reserved=0)

    def act(self, out, epsilon: float, q_out: torch.Tensor | None = None, actions: torch.Tensor | None = None):
        """One launch on ``out`` (the env's StepOutput, or a dict of its observation channels): masked dueling Q, then
        with probability ``epsilon`` a uniform legal action, otherwise the first argmax of the masked Q.  Returns the
        int8 [B,N] actions (``actions``, default :attr:`actions`); ``q_out`` [B,N,5] receives the masked Q."""
        ch = out if isinstance(out, dict) else {k: getattr(out, k) for k in ("local_obs", "goal_delta", "blocking_prev",
                                                                             "action_mask")}
        actions = self.actions if actions is None else actions
        a = self.args(ch, epsilon, actions, q_out)
        self.counter += 1
        a.counter = self.counter
        nat.check(self._act(C.byref(a), self.env._stream()))
        return actions


class FusedRecurrentPolicy:
    """Inference view of a :class:`recurrent.RecurrentActionMaskPolicy` of the reference's shape (trunk 64-64, LSTM
    cell 64 fed with the previous action and reward): features -> trunk -> LSTM cell -> masked draw in ONE launch
    (``mapf_lstm_policy_act``); or of a :class:`recurrent.PerAgentRecurrentPolicy` of that shape with one module per
    env agent (``mapf_lstm_policy_act_per_agent``, :attr:`entry`).  The module stays the learner's model: call
    :meth:`refresh` after every optimizer step.  Other shapes are refused (``ValueError``); run those through the
    module itself."""

    def __init__(self, policy, env, seed: int | None = None):
        F = int(env.V * env.V + 2 + (1 if env.include_blocking_pressure else 0))
        self.per_agent = _per_agent_kind(policy) is not None
        if not FusedRecurrentPolicy.matches(policy, env):
            raise ValueError("the fused LSTM kernel implements the reference's policy only: trunk (64, 64) over "
                             f"F = V*V + 2 (+1) = {F} features, LSTM cell 64 with previous action and previous reward, "
                             "5 actions" + (f"; per agent, one module per env agent: the policy has {policy.num_agents} "
                                            f"agents, the env {env.N}" if self.per_agent else ""))
        lin = None if self.per_agent else [m for m in policy.trunk if isinstance(m, torch.nn.Linear)]
        self.policy, self.env, self.F, self._lin = policy, env, F, lin
        self.with_bp = bool(env.include_blocking_pressure)
        self._lib = nat.lib()
        self.entry = "mapf_lstm_policy_act_per_agent" if self.per_agent else "mapf_lstm_policy_act"
        self._act = getattr(self._lib, self.entry)
        n = int(self._lib.mapf_lstm_policy_weights_nbytes(self.F))
        if n < 0:
            raise nat.MapfError(n, self._lib.mapf_last_error().decode())
        self._block = n
        n *= policy.num_agents if self.per_agent else 1   # per agent: block j at j * n
        self._host = np.zeros(n, np.uint8)
        self._dev = torch.zeros(n, dtype=torch.uint8, device=env.device)
        B, N, dev = env.B, env.N, env.device
        self.actions = torch.zeros((B, N), dtype=torch.int8, device=dev)
        self.actions64 = torch.zeros((B, N), dtype=torch.int64, device=dev)
        self.logp = torch.zeros((B, N), dtype=torch.float32, device=dev)
        self.value = torch.zeros((B, N), dtype=torch.float32, device=dev)
        self.seed = int(env.cfg.seed if seed is None else seed) & (2 ** 64 - 1)
        self.counter = 0
        self.refresh()

    @staticmethod
    def matches(policy, env) -> bool:
        """Whether the fused kernel implements ``policy`` (a :class:`recurrent.RecurrentActionMaskPolicy`) at ``env``'s
        feature width: trunk (64, 64) over F = V*V + 2 (+1 pressure) features, LSTM cell 64 fed with the previous
        action and reward, 5 actions."""
        F = env.V * env.V + 2 + (1 if env.include_blocking_pressure else 0)
        kind = _per_agent_kind(policy)
        if kind is not None:   # a recurrent.PerAgentRecurrentPolicy: every agent's module has the reference's shape
            return (kind == "lstm" and policy.num_agents == env.N and policy.feature_dim == F and tuple(policy.hiddens) == (64, 64)
                    and policy.cell == 64 and policy.num_actions == 5 and policy.use_prev_action
                    and policy.use_prev_reward)
        lin = [m for m in policy.trunk.modules() if isinstance(m, torch.nn.Linear)]
        return (len(lin) == 2 and lin[0].in_features == F and lin[0].out_features == 64
                and lin[1].in_features == 64 and lin[1].out_features == 64 and policy.cell == 64
                and policy.num_actions == 5 and policy.use_prev_action and policy.use_prev_reward
                and policy.lstm.input_size == 64 + 5 + 1 and policy.lstm.hidden_size == 64)

    def refresh(self):
        """Re-pack the module's current float32 parameters (bf16, padded; b_ih + b_hh summed; per agent: one block per
        agent) and upload them."""
        f = lambda t: np.ascontiguousarray(t.detach().float().cpu().numpy())  # noqa: E731
        p = self.policy
        if self.per_agent:
            per = _per_agent_arrays(p, [p.trunk_w[0], p.trunk_b[0], p.trunk_w[1], p.trunk_b[1], "w_ih", "w_hh", "b_ih",
                                        "b_hh", "logits_w", "logits_b", "value_w", "value_b"])
        else:
            lstm = p.lstm
            per = [[f(self._lin[0].weight), f(self._lin[0].bias), f(self._lin[1].weight), f(self._lin[1].bias),
                    f(lstm.weight_ih), f(lstm.weight_hh), f(lstm.bias_ih), f(lstm.bias_hh),
                    f(p.logits.weight), f(p.logits.bias), f(p.value.weight), f(p.value.bias)]]
        for j, arrs in enumerate(per):
            nat.check(self._lib.mapf_lstm_policy_pack_weights(self.F, *[a.ctypes.data_as(C.c_void_p) for a in arrs],
                                                              C.c_void_p(self._host.ctypes.data + j * self._block)))
        self._dev.copy_(torch.from_numpy(self._host))

    def args(self, out_channels: dict, state, prev_action, prev_reward, prev_terminated=None, prev_truncated=None, *,
             state_out=None, actions=None, actions64=None, logp=None, value=None, logits_out=None,
             greedy: bool = False) -> nat.MapfLstmPolicyArgs:
        """The argument block of one launch (counter 0; set ``.counter`` before launching).  ``out_channels`` maps
        local_obs / goal_delta / blocking_prev / action_mask to device tensors; every other tensor argument may be None
        (``state_out=None``: the state is not advanced).  ``greedy``: first argmax of the masked logits, no draw."""
        env = self.env
        p = lambda t: None if t is None else C.c_void_p(t.data_ptr())  # noqa: E731
        h, c = state
        ho, co = (None, None) if state_out is None else state_out
        return nat.MapfLstmPolicyArgs(
            num_envs=env.B, num_agents=env.N, v2=env.V * env.V, feature_dim=self.F,
            no_masking=0, greedy=int(bool(greedy)), seed=self.seed, counter=0, env_id_base=int(env.cfg.env_id_base),
            local_obs=p(out_channels["local_obs"]), goal_delta=p(out_channels["goal_delta"]),
            blocking_prev=p(out_channels["blocking_prev"]) if self.with_bp else None,
            action_mask=p(out_channels["action_mask"]), prev_terminated=p(prev_terminated),
            prev_truncated=p(prev_truncated), prev_action=p(prev_action), prev_reward=p(prev_reward),
            h_in=p(h), c_in=p(c), h_out=p(ho), c_out=p(co), weights=p(self._dev), actions=p(actions),
            actions64=p(actions64), logp=p(logp), value=p(value), logits_out=p(logits_out))

    def act(self, out, state, prev_action, prev_reward, prev_terminated=None, prev_truncated=None, *, advance: bool = True,
            state_out=None, logits_out: torch.Tensor | None = None, logp: torch.Tensor | None = None,
            value: torch.Tensor | None = None, actions64: torch.Tensor | None = None, greedy: bool = False):
        """One launch for the env's StepOutput ``out``.  ``state`` = (h, c) float32 [B*N, 64]; ``prev_action`` int8
        [B,N] (may be :attr:`actions` itself), ``prev_reward`` float32 [B,N]; ``prev_terminated`` / ``prev_truncated``
        uint8 [B] flag the envs whose episode starts at this step (their state, previous action and reward count as
        zero).  With ``advance`` the new state goes to ``state_out`` (default: ``state``, in place) and the draw to
        :attr:`actions`; without it (a bootstrap value) the state and :attr:`actions` -- the next step's previous
        actions -- are left as they are and the draw goes to ``actions64`` only.  Returns (actions int8 [B,N], logp,
        value); ``logits_out`` [B,N,5] receives the masked logits.  ``greedy``: the action is the first argmax of the
        masked logits (RLlib's ``forward_inference``), every other output is what the draw mode writes."""
        for name, t, dt in (("h", state[0], torch.float32), ("c", state[1], torch.float32),
                            ("prev_action", prev_action, torch.int8), ("prev_reward", prev_reward, torch.float32)):
            if t.dtype != dt or not t.is_contiguous() or t.device != self.env.device:
                raise ValueError(f"{name} must be a contiguous {dt} tensor on {self.env.device}")
        logp = self.logp if logp is None else logp
        value = self.value if value is None else value
        actions64 = self.actions64 if actions64 is None else actions64
        ch = {"local_obs": out.local_obs, "goal_delta": out.goal_delta, "blocking_prev": out.blocking_prev,
              "action_mask": out.action_mask}
        a = self.args(ch, state, prev_action, prev_reward, prev_terminated, prev_truncated,
                      state_out=(state if state_out is None else state_out) if advance else None,
                      actions=self.actions if advance else None,
                      actions64=actions64, logp=logp, value=value, logits_out=logits_out, greedy=greedy)
        self.counter += 1
        a.counter = self.counter
        nat.check(self._act(C.byref(a), self.env._stream()))
        return self.actions, logp, value


class FusedCtePolicy:
    """Inference view of a :class:`cte_rollout.CteActionMaskPolicy` of the reference's shape (trunk 64-64 over the
    R*C grid codes, 5N logits + value) on a :class:`single_agent.BatchedCteEnv`: grid codes -> MLP -> N masked 5-way
    draws in ONE launch (``mapf_cte_policy_act``).  The module stays the learner's model: call :meth:`refresh` after
    every optimizer step.  Other shapes, and maps beyond ``MAPF_CTE_POLICY_MAX_CELLS`` cells, are refused
    (``ValueError``) before any device work.  ``env_id_base`` keys the draws of env e as global env
    ``env_id_base + e``: shards of one batch launched with their offsets draw what the whole batch draws."""

    def __init__(self, policy, env, seed: int | None = None, env_id_base: int = 0):
        from .cte_rollout import CteActionMaskPolicy

        cells, N = int(env.R * env.C), int(env.N)
        if not FusedCtePolicy.matches(policy, env):
            got = (f"a {type(policy).__name__}" if not isinstance(policy, CteActionMaskPolicy) else
                   f"cells {policy.cells}, {policy.num_agents} agents, hiddens {tuple(policy.hiddens)}, no_masking "
                   f"{bool(policy.no_masking)}")
            raise ValueError("the fused CTE kernel implements CteActionMaskPolicy with hiddens (64, 64) and masking at "
                             f"the env's shape (cells {cells}, {N} agents); got {got}")
        self._lib = nat.lib()
        n = int(self._lib.mapf_cte_policy_weights_nbytes(cells, N))
        if n < 0:
            raise ValueError(f"the fused CTE kernel does not support this env: {self._lib.mapf_last_error().decode()}")
        self.policy, self.env, self.cells = policy, env, cells
        self._host = np.zeros(n, np.uint8)
        self._dev = torch.zeros(n, dtype=torch.uint8, device=env.device)
        B, dev = env.B, env.device
        self.actions = torch.zeros((B, N), dtype=torch.int8, device=dev)
        self.actions64 = torch.zeros((B, N), dtype=torch.int64, device=dev)
        self.logp = torch.zeros(B, dtype=torch.float32, device=dev)
        self.value = torch.zeros(B, dtype=torch.float32, device=dev)
        self.seed = int((env.seed or 0) if seed is None else seed) & (2 ** 64 - 1)
        self.env_id_base = int(env_id_base)
        self.counter = 0
        self.refresh()

    @staticmethod
    def matches(policy, env) -> bool:
        """Whether the fused kernel implements ``policy`` at ``env``'s shape: a :class:`cte_rollout.CteActionMaskPolicy`
        over cells = R*C with num_agents = N, hiddens (64, 64), masking on."""
        from .cte_rollout import CteActionMaskPolicy

        return (isinstance(policy, CteActionMaskPolicy) and policy.cells == env.R * env.C and policy.num_agents == env.N
                and tuple(policy.hiddens) == (64, 64) and not policy.no_masking)

    def refresh(self):
        """Re-pack the module's current float32 parameters (bf16, padded) and upload them."""
        f = lambda t: np.ascontiguousarray(t.detach().float().cpu().numpy())  # noqa: E731
        p = self.policy
        lin = [m for m in p.trunk if isinstance(m, torch.nn.Linear)]
        arrs = [f(lin[0].weight), f(lin[0].bias), f(lin[1].weight), f(lin[1].bias), f(p.logits.weight), f(p.logits.bias),
                f(p.value.weight), f(p.value.bias)]
        nat.check(self._lib.mapf_cte_policy_pack_weights(self.cells, self.env.N, *[a.ctypes.data_as(C.c_void_p) for a in arrs],
                                                         C.c_void_p(self._host.ctypes.data)))
        self._dev.copy_(torch.from_numpy(self._host))

    def args(self, obs_grid, action_mask, *, actions=None, actions64=None, logp=None, value=None, logits_out=None,
             num_envs: int | None = None, greedy: bool = False) -> nat.MapfCtePolicyArgs:
        """The argument block of one launch (counter 0; set ``.counter`` before launching).  Tensor arguments may be
        None, except the inputs ``obs_grid`` (uint8 [B, R*C]) and ``action_mask`` (int8 [B, 5N]).  ``greedy``: each
        agent's first argmax of its masked logits instead of the draw."""
        p = lambda t: None if t is None else C.c_void_p(t.data_ptr())  # noqa: E731
        return nat.MapfCtePolicyArgs(
            num_envs=self.env.B if num_envs is None else int(num_envs), num_agents=self.env.N, cells=self.cells,
            reserved=0, seed=self.seed, counter=0, env_id_base=self.env_id_base,
            obs_grid=p(obs_grid), action_mask=p(action_mask), weights=p(self._dev), actions=p(actions),
            actions64=p(actions64), logp=p(logp), value=p(value), logits_out=p(logits_out), greedy=int(bool(greedy)))

    def act(self, obs_grid=None, action_mask=None, *, logits_out: torch.Tensor | None = None,
            logp: torch.Tensor | None = None, value: torch.Tensor | None = None, actions64: torch.Tensor | None = None,
            num_envs: int | None = None, greedy: bool = False):
        """One launch on ``obs_grid`` (uint8 [B, R, C] or [B, R*C]; default: the env's) and ``action_mask`` (int8
        [B, 5N]; default: the env's).  Returns (actions int8 [B, N], joint logp [B], value [B]); ``logits_out``
        [B, N, 5] receives the masked logits.  ``num_envs``: launch on the first ``num_envs`` rows of the given tensors
        (with the constructor's ``env_id_base``: one shard of a larger batch).  ``greedy``: every agent takes the first
        argmax of its masked logits (RLlib's deterministic MultiDiscrete sample), logp is the sum of their
        log-probabilities, the other outputs are what the draw mode writes."""
        env = self.env
        obs_grid = env.obs_grid if obs_grid is None else obs_grid
        action_mask = env.action_mask if action_mask is None else action_mask
        B = env.B if num_envs is None else int(num_envs)
        for name, t, dt, shape in (("obs_grid", obs_grid, torch.uint8, B * self.cells),
                                   ("action_mask", action_mask, torch.int8, B * 5 * env.N)):
            if t.dtype != dt or not t.is_contiguous() or t.device != env.device or t.numel() < shape:
                raise ValueError(f"{name} must be a contiguous {dt} tensor of at least {shape} elements on {env.device}")
        logp = self.logp if logp is None else logp
        value = self.value if value is None else value
        actions64 = self.actions64 if actions64 is None else actions64
        a = self.args(obs_grid, action_mask, actions=self.actions, actions64=actions64, logp=logp, value=value,
                      logits_out=logits_out, num_envs=B, greedy=greedy)
        self.counter += 1
        a.counter = self.counter
        nat.check(self._lib.mapf_cte_policy_act(C.byref(a), env._stream()))
        return self.actions, logp, value


class FusedCteRecurrentPolicy:
    """Inference view of a :class:`cte_rollout.CteRecurrentPolicy` of the reference's shape (trunk 64-64 over the R*C
    grid codes, LSTM cell 64 fed with the previous joint action and reward, 5N logits + value) on a
    :class:`single_agent.BatchedCteEnv`: ``mapf_cte_lstm_policy_act``, two launches per call (trunk, then the recurrent
    step with the heads and the N masked draws).  The module stays the learner's model: call :meth:`refresh` after
    every optimizer step.  Other shapes, and maps beyond ``MAPF_CTE_POLICY_MAX_CELLS`` cells, are refused
    (``ValueError``) before any device work.  ``env_id_base`` keys the draws of env e as global env ``env_id_base + e``."""

    def __init__(self, policy, env, seed: int | None = None, env_id_base: int = 0):
        from .cte_rollout import CteRecurrentPolicy

        cells, N = int(env.R * env.C), int(env.N)
        if not FusedCteRecurrentPolicy.matches(policy, env):
            got = (f"a {type(policy).__name__}" if not isinstance(policy, CteRecurrentPolicy) else
                   f"cells {policy.cells}, {policy.num_agents} agents, hiddens {tuple(policy.hiddens)}, cell "
                   f"{policy.cell}, previous action {policy.use_prev_action}, previous reward {policy.use_prev_reward}")
            raise ValueError("the fused recurrent CTE kernel implements CteRecurrentPolicy with hiddens (64, 64), cell 64 "
                             f"and the previous action and reward at the env's shape (cells {cells}, {N} agents); got {got}")
        self._lib = nat.lib()
        n = int(self._lib.mapf_cte_lstm_policy_weights_nbytes(cells, N))
        if n < 0:
            raise ValueError(f"the fused recurrent CTE kernel does not support this env: {self._lib.mapf_last_error().decode()}")
        self.policy, self.env, self.cells = policy, env, cells
        self._host = np.zeros(n, np.uint8)
        self._dev = torch.zeros(n, dtype=torch.uint8, device=env.device)
        B, dev = env.B, env.device
        self.trunk = torch.empty((B, 64), dtype=torch.bfloat16, device=dev)   # the first launch's output
        self.actions = torch.zeros((B, N), dtype=torch.int8, device=dev)
        self.actions64 = torch.zeros((B, N), dtype=torch.int64, device=dev)
        self.logp = torch.zeros(B, dtype=torch.float32, device=dev)
        self.value = torch.zeros(B, dtype=torch.float32, device=dev)
        self.seed = int((env.seed or 0) if seed is None else seed) & (2 ** 64 - 1)
        self.env_id_base = int(env_id_base)
        self.counter = 0
        self.refresh()

    @staticmethod
    def matches(policy, env) -> bool:
        """Whether the fused kernels implement ``policy`` at ``env``'s shape: a :class:`cte_rollout.CteRecurrentPolicy`
        over cells = R*C with num_agents = N, hiddens (64, 64), cell 64, previous action and reward on."""
        from .cte_rollout import CteRecurrentPolicy

        return (isinstance(policy, CteRecurrentPolicy) and policy.cells == env.R * env.C and policy.num_agents == env.N
                and tuple(policy.hiddens) == (64, 64) and policy.cell == 64 and policy.use_prev_action
                and policy.use_prev_reward)

    def refresh(self):
        """Re-pack the module's current float32 parameters (bf16, padded; the reward column and b_ih + b_hh in f32)
        and upload them."""
        f = lambda t: np.ascontiguousarray(t.detach().float().cpu().numpy())  # noqa: E731
        p = self.policy
        lin = [m for m in p.trunk if isinstance(m, torch.nn.Linear)]
        arrs = [f(lin[0].weight), f(lin[0].bias), f(lin[1].weight), f(lin[1].bias), f(p.lstm.weight_ih),
                f(p.lstm.weight_hh), f(p.lstm.bias_ih), f(p.lstm.bias_hh), f(p.logits.weight), f(p.logits.bias),
                f(p.value.weight), f(p.value.bias)]
        nat.check(self._lib.mapf_cte_lstm_policy_pack_weights(self.cells, self.env.N,
                                                              *[a.ctypes.data_as(C.c_void_p) for a in arrs],
                                                              C.c_void_p(self._host.ctypes.data)))
        self._dev.copy_(torch.from_numpy(self._host))

    def args(self, obs_grid, action_mask, state, prev_action, prev_reward, prev_terminated=None, prev_truncated=None, *,
             state_out=None, actions=None, actions64=None, logp=None, value=None, logits_out=None,
             num_envs: int | None = None, greedy: bool = False) -> nat.MapfCteLstmPolicyArgs:
        """The argument block of one call (counter 0; set ``.counter`` before launching).  ``state_out=None``: the
        state is not advanced; the outputs may be None.  ``greedy``: each agent's first argmax instead of the draw."""
        p = lambda t: None if t is None else C.c_void_p(t.data_ptr())  # noqa: E731
        h, c = state
        ho, co = (None, None) if state_out is None else state_out
        return nat.MapfCteLstmPolicyArgs(
            num_envs=self.env.B if num_envs is None else int(num_envs), num_agents=self.env.N, cells=self.cells,
            reserved=0, seed=self.seed, counter=0, env_id_base=self.env_id_base,
            obs_grid=p(obs_grid), action_mask=p(action_mask), prev_terminated=p(prev_terminated),
            prev_truncated=p(prev_truncated), prev_action=p(prev_action), prev_reward=p(prev_reward), h_in=p(h),
            c_in=p(c), h_out=p(ho), c_out=p(co), trunk=p(self.trunk), weights=p(self._dev), actions=p(actions),
            actions64=p(actions64), logp=p(logp), value=p(value), logits_out=p(logits_out), greedy=int(bool(greedy)))

    def act(self, state, prev_action, prev_reward, prev_terminated=None, prev_truncated=None, *, obs_grid=None,
            action_mask=None, advance: bool = True, state_out=None, logits_out: torch.Tensor | None = None,
            logp: torch.Tensor | None = None, value: torch.Tensor | None = None, actions64: torch.Tensor | None = None,
            num_envs: int | None = None, greedy: bool = False):
        """One call on ``obs_grid`` (uint8 [B, R*C]; default: the env's) and ``action_mask`` (int8 [B, 5N]; default:
        the env's).  ``state`` = (h, c) float32 [B, 64]; ``prev_action`` int8 [B, N] (may be :attr:`actions` itself);
        ``prev_reward`` float64 [B] (the env's ``reward``); ``prev_terminated`` / ``prev_truncated`` uint8 [B] flag the
        envs whose episode starts at this step (their state, previous action and reward count as zero).  With
        ``advance`` the new state goes to ``state_out`` (default: ``state``, in place) and the draw to :attr:`actions`;
        without it the state and :attr:`actions` are left as they are.  Returns (actions int8 [B, N], joint logp [B],
        value [B]); ``logits_out`` [B, N, 5] receives the masked logits.  ``num_envs``: the first ``num_envs`` rows of
        every tensor (with the constructor's ``env_id_base``: one shard of a larger batch).  ``greedy``: every agent
        takes the first argmax of its masked logits; the state, value, logp and logits are what the draw mode writes."""
        env = self.env
        obs_grid = env.obs_grid if obs_grid is None else obs_grid
        action_mask = env.action_mask if action_mask is None else action_mask
        B = env.B if num_envs is None else int(num_envs)
        for name, t, dt, n in (("obs_grid", obs_grid, torch.uint8, B * self.cells),
                               ("action_mask", action_mask, torch.int8, B * 5 * env.N),
                               ("h", state[0], torch.float32, B * 64), ("c", state[1], torch.float32, B * 64),
                               ("prev_action", prev_action, torch.int8, B * env.N),
                               ("prev_reward", prev_reward, torch.float64, B)):
            if t.dtype != dt or not t.is_contiguous() or t.device != env.device or t.numel() < n:
                raise ValueError(f"{name} must be a contiguous {dt} tensor of at least {n} elements on {env.device}")
        logp = self.logp if logp is None else logp
        value = self.value if value is None else value
        actions64 = self.actions64 if actions64 is None else actions64
        a = self.args(obs_grid, action_mask, state, prev_action, prev_reward, prev_terminated, prev_truncated,
                      state_out=(state if state_out is None else state_out) if advance else None,
                      actions=self.actions if advance else None, actions64=actions64, logp=logp, value=value,
                      logits_out=logits_out, num_envs=B, greedy=greedy)
        self.counter += 1
        a.counter = self.counter
        nat.check(self._lib.mapf_cte_lstm_policy_act(C.byref(a), env._stream()))
        return self.actions, logp, value


def gae(rewards, values, dones, last_value, gamma: float = 0.99, lam: float = 0.95):
    """GAE over [T,B,N] float32 CUDA tensors (``dones`` [T,B] bool / uint8) with the scan kernel."""
    T, B, N = rewards.shape
    adv, ret = torch.empty_like(rewards), torch.empty_like(rewards)
    d = dones.to(torch.uint8).contiguous()
    st = C.c_void_p(torch.cuda.current_stream(rewards.device).cuda_stream)
    p = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
    nat.check(nat.lib().mapf_gae(p(rewards.contiguous()), p(values.contiguous()), p(d), p(last_value.contiguous()), p(adv),
                                 p(ret), int(T), int(B), int(N), C.c_float(gamma), C.c_float(lam), st))
    return adv, ret


def vtrace(target_logp, behaviour_logp, values, rewards, dones, bootstrap_value, *, columns=None, gamma: float = 0.99,
           clip_rho: float = 1.0, clip_pg_rho: float = 1.0):
    """V-trace targets with the ``mapf_vtrace`` scan on the current stream: (vs, pg_advantages), float32 [T,M].
    ``rewards`` / ``behaviour_logp``: float32 [T,B,N] or [T,B] (the batch's own rows); ``dones``: [T,B] bool / uint8;
    ``bootstrap_value``: [B,N] or [B]; ``target_logp`` / ``values``: float32 [T,M], column m of batch column
    ``columns[m]`` (int64 [M], flat index b * N + n; None: all B*N columns in order).  :func:`impala.vtrace` is the
    same recurrence in PyTorch."""
    T, B = int(rewards.shape[0]), int(rewards.shape[1])
    N = int(rewards.shape[2]) if rewards.dim() == 3 else 1
    if rewards.dim() not in (2, 3) or tuple(behaviour_logp.shape) != tuple(rewards.shape):
        raise ValueError(f"rewards {tuple(rewards.shape)} and behaviour_logp {tuple(behaviour_logp.shape)} must be one "
                         "[T,B,N] or [T,B] shape")
    if tuple(dones.shape) != (T, B) or bootstrap_value.numel() != B * N:
        raise ValueError(f"dones {tuple(dones.shape)} must be [T,B] = [{T},{B}] and bootstrap_value "
                         f"{tuple(bootstrap_value.shape)} hold B*N = {B * N} values")
    M = B * N if columns is None else int(columns.numel())
    if tuple(target_logp.shape) != (T, M) or tuple(values.shape) != (T, M):
        raise ValueError(f"target_logp {tuple(target_logp.shape)} and values {tuple(values.shape)} must be [T,M] = [{T},{M}]")
    floats = [x.contiguous() for x in (target_logp, behaviour_logp, values, rewards, bootstrap_value)]
    dev = rewards.device
    if any(x.dtype != torch.float32 or x.device != dev or not x.is_cuda for x in floats):
        raise ValueError(f"the V-trace kernel takes float32 tensors on one CUDA device (got {[(x.dtype, x.device) for x in floats]})")
    tl, mu, v, r, boot = floats
    d = dones.contiguous()
    d = d.view(torch.uint8) if d.dtype == torch.bool else d if d.dtype == torch.uint8 else (d != 0).to(torch.uint8)
    cols = None if columns is None else columns.to(device=dev, dtype=torch.int64).contiguous()
    vs, pg = torch.empty((T, M), device=dev), torch.empty((T, M), device=dev)
    p = lambda t: None if t is None else C.c_void_p(t.data_ptr())  # noqa: E731
    a = nat.MapfVtraceArgs(T=T, num_agents=N, num_columns=B * N, M=M, columns=p(cols), rewards=p(r),
                           behaviour_logp=p(mu), dones=p(d), bootstrap_value=p(boot), target_logp=p(tl), values=p(v),
                           vs=p(vs), pg_advantages=p(pg), gamma=float(gamma), clip_rho=float(clip_rho),
                           clip_pg_rho=float(clip_pg_rho), reserved=0)
    nat.check(nat.lib().mapf_vtrace(C.byref(a), C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
    return vs, pg
