"""Batched evaluator: the reference's ``test_trained_model`` (main.py:93-387) with every episode running as one env
of a GPU batch.

The reference plays ``num_episodes`` episodes one after the other, sums the rewards, counts timesteps, tracks
per-agent returns, the start / goal layout, the lifelong metrics of the last ``info["__all__"]`` and an occupancy
heat-map (``occupancy_grid[y, x] += 1`` for every agent after every step), then writes one CSV row per episode.  Here
episode e is env e of a :class:`BatchedMapfEnv`; an env stops contributing at its first ``terminated | truncated``
(no auto-reset), the heat-map is accumulated by ``mapf_occupancy_accumulate`` over the still-active envs, the other
per-episode sums by ``mapf_eval_accumulate``, and they stay on the device until the end.  Policies: ``"random"`` (the
reference's ``ALGO_NAME == "RANDOM"`` branch: uniform actions, main.py:212-214), ``"masked"`` (uniform over the action
mask), any callable ``policy(env, out) -> int8 [B,N]``, or a trained :class:`rollout.ActionMaskPolicy` /
:class:`recurrent.RecurrentActionMaskPolicy` played like ``rl_module.forward_inference`` (main.py:209-223): argmax of the
masked logits, the LSTM state, previous action and previous reward carried from step to step.  Modules of the
reference's shape (and the per-agent variants :class:`rollout.PerAgentActionMaskPolicy` /
:class:`recurrent.PerAgentRecurrentPolicy`, one module per agent, of that shape) run as one fused kernel launch per step (``mapf_policy_act`` / ``mapf_lstm_policy_act`` in greedy
mode), any other shape through its PyTorch forward.

The reference's third execution mode, CTE (``env_config["training_execution_mode"] == "CTE"``, or a
:class:`cte_rollout.CteActionMaskPolicy` / :class:`cte_rollout.CteRecurrentPolicy`), plays the single-agent view
instead: episode e is env e of a :class:`single_agent.BatchedCteEnv`, one joint action and one scalar reward per step,
the heat-map and the per-episode sums accumulated by ``mapf_cte_eval_accumulate``.  Centralised modules of the fused
shape run ``mapf_cte_policy_act`` / ``mapf_cte_lstm_policy_act`` in greedy mode, other shapes their PyTorch forward.

``python -m dl_reference_models_b200.evaluate`` times the evaluator (:func:`benchmark`).
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field

import numpy as np
import torch

from . import _native as nat
from . import maps, rollout
from .batched_env import BatchedMapfEnv
from .cte_rollout import CteActionMaskPolicy, CteRecurrentPolicy
from .policy_kernels import FusedCtePolicy, FusedCteRecurrentPolicy, FusedPolicy, FusedRecurrentPolicy
from .recurrent import PerAgentRecurrentPolicy, RecurrentActionMaskPolicy
from .single_agent import BatchedCteEnv

MODULE_TYPES = (rollout.ActionMaskPolicy, RecurrentActionMaskPolicy, rollout.PerAgentActionMaskPolicy, PerAgentRecurrentPolicy)
RECURRENT_TYPES = (RecurrentActionMaskPolicy, PerAgentRecurrentPolicy)
CTE_MODULE_TYPES = (CteActionMaskPolicy, CteRecurrentPolicy)


@dataclass
class EvalResult:
    rows: list = field(default_factory=list)          # one dict per episode, the CSV schema of main.py:296-325
    occupancy_grid: np.ndarray | None = None          # int64 [R,C], main.py:153-155
    success_rate: float = 0.0                         # main.py:330
    average_reward: float = 0.0                       # main.py:327
    average_timesteps: float = 0.0                    # main.py:328
    lifelong: dict = field(default_factory=dict)      # main.py:332-338

    def to_dataframe(self):
        import pandas as pd

        return pd.DataFrame(self.rows)

    def save_csv(self, path):
        self.to_dataframe().to_csv(path, index=False)   # main.py:361
        return path


def _module_in_features(policy) -> int:
    if isinstance(policy, (rollout.PerAgentActionMaskPolicy, PerAgentRecurrentPolicy)):
        return int(policy.feature_dim)
    lin = [m for m in policy.trunk.modules() if isinstance(m, torch.nn.Linear)]
    if lin:
        return int(lin[0].in_features)
    if isinstance(policy, RecurrentActionMaskPolicy):
        return int(policy.lstm.input_size) - (policy.num_actions if policy.use_prev_action else 0) - int(policy.use_prev_reward)
    return int(policy.logits.in_features)


def _module_actor(env, policy, explore: bool):
    """``act(out) -> int8 [B,N]`` for a trained module: the fused kernel (one launch per step) where it implements the
    module's shape, its PyTorch forward otherwise.  Greedy unless ``explore``; the LSTM carries (h, c), the previous
    actions and the previous rewards from step to step, zero at reset (no episode starts: the evaluator never
    auto-resets)."""
    F = env.flat_obs_dim(include_action_mask=False)
    if _module_in_features(policy) != F:
        raise ValueError(f"the policy reads {_module_in_features(policy)} features, the env's observation has {F} "
                         "(flat_obs_dim without the action mask)")
    wrong = {str(p.device) for p in policy.parameters() if p.device != env.device}
    if wrong:
        raise ValueError(f"the policy's parameters are on {sorted(wrong)}, the evaluation runs on {env.device}")
    if isinstance(policy, (rollout.PerAgentActionMaskPolicy, PerAgentRecurrentPolicy)) and policy.num_agents != env.N:
        raise ValueError(f"the per-agent policy has num_agents = {policy.num_agents} modules, the env has "
                         f"num_agents = {env.N} agents")
    B, N, dev = env.B, env.N, env.device
    recurrent = isinstance(policy, RECURRENT_TYPES)
    if recurrent and FusedRecurrentPolicy.matches(policy, env):
        fused = FusedRecurrentPolicy(policy, env)
        state = (torch.zeros((B * N, 64), device=dev), torch.zeros((B * N, 64), device=dev))
        prev_reward = [torch.zeros((B, N), device=dev)]

        def act(out):
            a, _, _ = fused.act(out, state, fused.actions, prev_reward[0], greedy=not explore)
            prev_reward[0] = env.out["reward"]   # read by the next launch before the next step overwrites it
            return a
        return act
    if not recurrent and FusedPolicy.matches(policy, env):
        fused = FusedPolicy(policy, env)
        return lambda out: fused.act(out, greedy=not explore)[0]
    return _torch_actor(env, policy, explore)


def _torch_actor(env, policy, explore: bool):
    """The module's own forward (any shape), with the same carry as the fused path."""
    B, N, dev = env.B, env.N, env.device
    M = B * N
    recurrent = isinstance(policy, RECURRENT_TYPES)
    carry = {}
    if recurrent:
        carry.update(state=policy.initial_state(M, dev), prev_action=torch.zeros(M, dtype=torch.int64, device=dev),
                     prev_reward=torch.zeros(M, device=dev))

    @torch.no_grad()
    def act(out):
        feats = env.flat_obs(include_action_mask=False).reshape(M, -1)
        mask = out.action_mask.reshape(M, 5)
        if recurrent:
            logits, _, carry["state"] = policy.step(feats, mask, carry["prev_action"], carry["prev_reward"], carry["state"])
        else:
            logits, _ = policy(feats, mask)
        a = rollout.sample_categorical(logits)[0] if explore else torch.argmax(logits, dim=-1)
        if recurrent:
            carry["prev_action"] = a
            carry["prev_reward"] = env.out["reward"].reshape(M)   # read by the next forward before the next step
        return a.to(torch.int8).reshape(B, N)
    return act


def _play(env, policy="random", max_steps: int | None = None, explore: bool = False) -> dict:
    """Reset ``env`` and play every env's first episode to its end (or ``max_steps`` steps).  Per step: the policy,
    the env step, the heat-map (``mapf_occupancy_accumulate``, over the envs active before the step) and the rest of
    the bookkeeping (``mapf_eval_accumulate``); the loop's one host sync is the 4-byte read of the still-active
    count.  Returns the device accumulators."""
    B, N = env.B, env.N
    dev = env.device
    out = env.reset()
    if isinstance(policy, MODULE_TYPES):
        module_act = _module_actor(env, policy, explore)
        policy = lambda env, out: module_act(out)  # noqa: E731
    z = lambda shape, dt: torch.zeros(shape, dtype=dt, device=dev)  # noqa: E731
    acc = {"starts": env.state["starts"].cpu().numpy().copy(), "goals": env.state["goals"].cpu().numpy().copy(),
           "active": torch.ones(B, dtype=torch.uint8, device=dev), "episode_reward": z(B, torch.float64),
           "agent_reward": z((B, N), torch.float64), "timesteps": z(B, torch.int64), "success": z(B, torch.uint8),
           "last_info": z((B, nat.INFO_WORDS), torch.int32), "occupancy": z(env.grid.shape[-2:], torch.int64),
           "active_count": z(2, torch.int32)}
    # the argument block is built once: env.step writes its outputs to the env's own buffers every step
    p = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
    args = nat.MapfEvalArgs(
        num_envs=B, num_agents=N, reward=p(env.out["reward"]), terminated=p(env.out["terminated"]),
        truncated=p(env.out["truncated"]), info=p(env.out["info"]), active=p(acc["active"]),
        episode_reward=p(acc["episode_reward"]), agent_reward=p(acc["agent_reward"]), timesteps=p(acc["timesteps"]),
        success=p(acc["success"]), last_info=p(acc["last_info"]), active_count=p(acc["active_count"]))
    counts = (acc["active_count"][0], acc["active_count"][1])
    active, occupancy = p(acc["active"]), p(acc["occupancy"])
    lib, stream = nat.lib(), env._stream()
    limit = max_steps if max_steps is not None else int(env.cfg.steps_per_episode) + 1
    still = B
    for step in range(limit):
        if still == 0:
            break
        if callable(policy):
            actions = policy(env, out)
        else:
            actions = env.sample_actions(masked=(policy == "masked"))
        out = env.step(actions, auto_reset=False)
        # main.py:264-267, over the envs active before this step's done-clear
        nat.check(lib.mapf_occupancy_accumulate(env._h, active, occupancy, stream))
        args.step = step
        nat.check(lib.mapf_eval_accumulate(C.byref(args), stream))
        still = int(counts[step & 1])
    return acc


def _cte_view(env_config: dict, policy) -> bool:
    """Whether ``policy`` is evaluated on the single-agent (CTE) view: a centralised module, or, for the other
    policies, ``training_execution_mode == "CTE"`` (the reference's switch, main.py:71-77).  A module of one view with
    a config that names another mode is refused."""
    mode = env_config.get("training_execution_mode")
    if isinstance(policy, CTE_MODULE_TYPES):
        if mode is not None and mode != "CTE":
            raise ValueError(f"a {type(policy).__name__} is a centralised (CTE) policy; the env_config names "
                             f"training_execution_mode = {mode!r}")
        return True
    if isinstance(policy, MODULE_TYPES):
        if mode == "CTE":
            raise ValueError(f"a {type(policy).__name__} plays the multi-agent view; the env_config names "
                             "training_execution_mode = 'CTE' (use a CteActionMaskPolicy or CteRecurrentPolicy)")
        return False
    return mode == "CTE"


def _check_cte_module(policy, env_config: dict, device) -> None:
    """Refuse a centralised module whose cells, num_agents or device do not match the env, before any device work."""
    grid = env_config.get("grid")
    R, C_ = (np.asarray(grid) if grid is not None else maps.get_grid(env_config["env_name"])).shape
    N = int(env_config.get("num_agents", 2))
    if policy.cells != R * C_:
        raise ValueError(f"the policy reads {policy.cells} grid cells, the env's map has {R}x{C_} = {R * C_}")
    if policy.num_agents != N:
        raise ValueError(f"the policy has num_agents = {policy.num_agents}, the env has num_agents = {N} agents")
    dev = torch.device(device)
    if dev.type == "cuda" and dev.index is None:
        dev = torch.device("cuda", torch.cuda.current_device() if torch.cuda.is_available() else 0)
    wrong = {str(p.device) for p in policy.parameters() if p.device != dev}
    if wrong:
        raise ValueError(f"the policy's parameters are on {sorted(wrong)}, the evaluation runs on {dev}")


def _cte_module_actor(env, policy, explore: bool):
    """``act() -> int8 [B,N]`` for a centralised module on the CTE env's current ``obs_grid`` / ``action_mask``: one
    fused call (greedy unless ``explore``) where the kernels implement the module's shape, its PyTorch forward
    otherwise.  The LSTM carries (h, c), the previous joint action and the previous float64 reward, zero at reset."""
    B, dev = env.B, env.device
    if isinstance(policy, CteRecurrentPolicy) and FusedCteRecurrentPolicy.matches(policy, env):
        fused = FusedCteRecurrentPolicy(policy, env)
        state = (torch.zeros((B, 64), device=dev), torch.zeros((B, 64), device=dev))
        prev_reward = [torch.zeros(B, dtype=torch.float64, device=dev)]

        def act():
            a, _, _ = fused.act(state, fused.actions, prev_reward[0], greedy=not explore)
            prev_reward[0] = env.reward   # read by the next call before the next step overwrites it
            return a
        return act
    if isinstance(policy, CteActionMaskPolicy) and FusedCtePolicy.matches(policy, env):
        fused = FusedCtePolicy(policy, env)
        return lambda: fused.act(greedy=not explore)[0]
    return _cte_torch_actor(env, policy, explore)


def _cte_torch_actor(env, policy, explore: bool):
    """The centralised module's own forward / step (any shape), with the same carry as the fused path."""
    B, N, dev = env.B, env.N, env.device
    cells = env.R * env.C
    recurrent = isinstance(policy, CteRecurrentPolicy)
    carry = {}
    if recurrent:
        carry.update(state=policy.initial_state(B, dev), prev_action=torch.zeros((B, N), dtype=torch.int64, device=dev),
                     prev_reward=torch.zeros(B, dtype=torch.float64, device=dev))

    @torch.no_grad()
    def act():
        grid = env.obs_grid.view(B, cells)
        if recurrent:
            logits, _, carry["state"] = policy.step(grid, env.action_mask, carry["prev_action"], carry["prev_reward"],
                                                    carry["state"])
        else:
            logits, _ = policy(grid, env.action_mask)
        a = rollout.sample_categorical(logits)[0] if explore else torch.argmax(logits, dim=-1)
        if recurrent:
            carry["prev_action"] = a
            carry["prev_reward"] = env.reward   # read by the next step() before the next env step
        return a.to(torch.int8)
    return act


def _play_cte(env, policy="random", max_steps: int | None = None, explore: bool = False) -> dict:
    """:func:`_play` on the single-agent view: reset ``env`` (a :class:`single_agent.BatchedCteEnv`) once and play
    every env's first episode to its end (or ``max_steps`` steps).  Per step: the policy, the env step (without the
    float32 ``flat_obs`` output: the policies read ``obs_grid`` and ``action_mask``) and ``mapf_cte_eval_accumulate``
    (heat-map and bookkeeping); the loop's one host sync is the 4-byte read of the still-active count.  A callable
    policy is called as ``policy(env, (env.obs_grid, env.action_mask))``.  Returns the device accumulators."""
    B, N, dev = env.B, env.N, env.device
    env.reset()
    if isinstance(policy, CTE_MODULE_TYPES):
        module_act = _cte_module_actor(env, policy, explore)
        policy = lambda env, out: module_act()  # noqa: E731
    elif policy in ("random", "masked"):
        gen = torch.Generator(device=dev).manual_seed(int(env.seed or 0))
        masked = policy == "masked"

        def policy(env, out):
            if not masked:
                return torch.randint(0, 5, (B, N), dtype=torch.int8, device=dev, generator=gen)
            u = torch.rand((B, N, 5), device=dev, generator=gen)   # uniform over each agent's allowed actions
            return torch.argmax(u * env.action_mask.view(B, N, 5), dim=-1).to(torch.int8)
    elif not callable(policy):
        raise ValueError(f"policy must be 'random', 'masked', a callable or a centralised module, got {policy!r}")
    z = lambda shape, dt: torch.zeros(shape, dtype=dt, device=dev)  # noqa: E731
    acc = {"starts": env.starts.cpu().numpy().copy(), "goals": env.goals.cpu().numpy().copy(),
           "active": torch.ones(B, dtype=torch.uint8, device=dev), "episode_reward": z(B, torch.float64),
           "timesteps": z(B, torch.int64), "success": z(B, torch.uint8),
           "last_info": z((B, nat.CTE_INFO_WORDS), torch.float64), "occupancy": z((env.R, env.C), torch.int64),
           "active_count": z(2, torch.int32)}
    p = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
    sargs = nat.MapfCteArgs.from_buffer_copy(env._args)   # the env's own block, without the float32 observation
    sargs.flat_obs = None
    args = nat.MapfCteEvalArgs(
        num_envs=B, num_agents=N, rows=env.R, cols=env.C, positions=p(env.positions), reward=p(env.reward),
        terminated=p(env.terminated), truncated=p(env.truncated), info=p(env.info), active=p(acc["active"]),
        episode_reward=p(acc["episode_reward"]), timesteps=p(acc["timesteps"]), success=p(acc["success"]),
        last_info=p(acc["last_info"]), occupancy=p(acc["occupancy"]), active_count=p(acc["active_count"]))
    counts = (acc["active_count"][0], acc["active_count"][1])
    lib, stream = nat.lib(), env._stream()
    limit = max_steps if max_steps is not None else env.steps_per_episode + 1
    out = (env.obs_grid, env.action_mask)
    still = B
    for step in range(limit):
        if still == 0:
            break
        actions = policy(env, out)
        a = torch.as_tensor(actions).to(device=dev, dtype=torch.int8).reshape(B, N).contiguous()
        sargs.actions = a.data_ptr()
        nat.check(lib.mapf_cte_step(C.byref(sargs), stream))
        args.step = step
        nat.check(lib.mapf_cte_eval_accumulate(C.byref(args), stream))
        still = int(counts[step & 1])
    return acc


def _cte_result(env, acc) -> EvalResult:
    """The CSV rows and summary of the CTE view (DESIGN.md §7 N2b): the multi-agent schema without per-agent rewards
    (the view has one scalar reward), the two CTE counters of the episode's last step instead of the lifelong ones."""
    B, N = env.B, env.N
    starts, goals0 = acc["starts"], acc["goals"]
    info = acc["last_info"].cpu().numpy()
    ep_r, st = acc["episode_reward"].cpu().numpy(), acc["timesteps"].cpu().numpy()
    succ = acc["success"].cpu().numpy().astype(np.float64)
    res = EvalResult()
    for e in range(B):
        row = {"episode": e + 1, "cpu_time": 0.0, "seed": env.env_config.get("seed"), "total_reward": float(ep_r[e]),
               "timesteps": int(st[e]), "goals_reached_total": float(info[e, 2]), "blocking_count_total": float(info[e, 3])}
        for i in range(N):
            row[f"agent_{i}_start_x"], row[f"agent_{i}_start_y"] = int(starts[e, i, 0]), int(starts[e, i, 1])
            row[f"agent_{i}_goal_x"], row[f"agent_{i}_goal_y"] = int(goals0[e, i, 0]), int(goals0[e, i, 1])
        res.rows.append(row)
    res.occupancy_grid = acc["occupancy"].cpu().numpy()
    res.success_rate = float(np.mean(succ)) if B else 0.0
    res.average_reward = float(ep_r.sum() / max(B, 1))
    res.average_timesteps = float(st.sum() / max(B, 1))
    return res


def evaluate(env_config: dict, num_episodes: int, policy="random", device="cuda:0", max_steps: int | None = None,
             explore: bool = False) -> EvalResult:
    """Play ``num_episodes`` episodes, one per env of a batch.  ``policy``: ``"random"``, ``"masked"``, a callable
    ``policy(env, out) -> int8 [B,N]``, or a trained :class:`rollout.ActionMaskPolicy` /
    :class:`recurrent.RecurrentActionMaskPolicy` / :class:`rollout.PerAgentActionMaskPolicy` /
    :class:`recurrent.PerAgentRecurrentPolicy` (``num_agents`` = the env's) on ``device``, played as the reference's ``forward_inference`` (argmax
    of the masked logits; ``explore=True``: a draw from them).

    A :class:`cte_rollout.CteActionMaskPolicy` / :class:`cte_rollout.CteRecurrentPolicy`, or any other policy with
    ``env_config["training_execution_mode"] == "CTE"``, plays the single-agent view (:class:`single_agent.BatchedCteEnv`);
    there the callable receives the CTE env and ``(env.obs_grid, env.action_mask)``, and the rows carry the episode's
    scalar return and its last ``goals_reached_total`` / ``blocking_count_total`` instead of per-agent rewards."""
    if _cte_view(env_config, policy):
        if isinstance(policy, CTE_MODULE_TYPES):
            _check_cte_module(policy, env_config, device)
        env = BatchedCteEnv(env_config, num_episodes, device)
        return _cte_result(env, _play_cte(env, policy, max_steps, explore))
    env = BatchedMapfEnv(env_config, num_episodes, device)
    acc = _play(env, policy, max_steps, explore)
    B, N = env.B, env.N
    starts, goals0 = acc["starts"], acc["goals"]
    occupancy = acc["occupancy"]
    last_info, ep_reward, agent_reward, steps, success = (acc[k] for k in ("last_info", "episode_reward", "agent_reward",
                                                                            "timesteps", "success"))
    res = EvalResult()
    info = last_info.cpu().numpy()
    ep_r, ag_r, st = ep_reward.cpu().numpy(), agent_reward.cpu().numpy(), steps.cpu().numpy()
    lifelong = bool(env.lifelong)
    succ = success.cpu().numpy().astype(np.float64)
    g_tot = info[:, nat.I_GOALS_REACHED_TOTAL].astype(np.float64)
    thr = g_tot / np.maximum(info[:, nat.I_STEP_COUNT], 1)
    comp = info[:, nat.I_COMPLETED_COUNT].astype(np.float64) / float(N)
    for e in range(B):
        row = {"episode": e + 1, "cpu_time": 0.0, "seed": env.env_config.get("seed"), "total_reward": float(ep_r[e]),
               "timesteps": int(st[e])}
        if lifelong:   # main.py:305-315
            row.update(goals_reached_total=float(g_tot[e]), throughput=float(thr[e]), completion_ratio=float(comp[e]))
        for i in range(N):   # main.py:319-325 (x = row index, y = column index in the reference's naming)
            row[f"agent_{i}_reward"] = float(ag_r[e, i])
            row[f"agent_{i}_start_x"], row[f"agent_{i}_start_y"] = int(starts[e, i, 0]), int(starts[e, i, 1])
            row[f"agent_{i}_goal_x"], row[f"agent_{i}_goal_y"] = int(goals0[e, i, 0]), int(goals0[e, i, 1])
        res.rows.append(row)
    res.occupancy_grid = occupancy.cpu().numpy()
    res.success_rate = float(np.mean(comp if lifelong else succ)) if B else 0.0   # main.py:314,316,330
    res.average_reward = float(ep_r.sum() / max(B, 1))
    res.average_timesteps = float(st.sum() / max(B, 1))
    if lifelong:
        res.lifelong = {"goals_reached_total": float(g_tot.mean()), "throughput": float(thr.mean()),
                        "completion_ratio": float(comp.mean())}
    env.close()
    return res


def benchmark(num_episodes: int = 65536, rounds: int = 3, device: str = "cuda:0") -> dict:
    """``num_episodes`` episodes x 16 agents, 32x32 random map, episodic, 256 steps per episode: episodes/s and
    agent-steps/s of the evaluator's step loop (:func:`_play`: reset, then per step the policy, the env step, the
    heat-map and the bookkeeping kernel; the CSV rows are not built) for the uniform masked policy, the MLP and the
    LSTM-64 module greedy on their fused kernels, and the LSTM-64 module through its PyTorch forward (the path of
    non-reference shapes).  Agent-steps count every env at every loop step (finished envs are still stepped).  Best of
    ``rounds`` after a short warm-up each; host clock around work that ends in a device synchronise (the loop's last
    count read).  ``evaluate_masked_s`` is one whole :func:`evaluate` call, env construction and rows included.  The
    ``cte_*`` keys time :func:`_play_cte` the same way on the single-agent view of the same map and shape: the uniform
    masked policy, the centralised MLP and LSTM-64 modules greedy on their fused kernels, and the LSTM-64 module through
    its PyTorch forward."""
    import subprocess
    import time

    from . import maps

    cfg = {"num_agents": 16, "sensor_range": 2, "steps_per_episode": 256, "lifelong_mapf": False, "seed": 999,
           "grid": maps.random_obstacle_grid(32, 32, 0.30, 2026, min_free=32)}
    env = BatchedMapfEnv(cfg, num_episodes, device)
    F = env.flat_obs_dim(include_action_mask=False)
    torch.manual_seed(0)
    mlp = rollout.ActionMaskPolicy(F).to(env.device)
    lstm = RecurrentActionMaskPolicy(F).to(env.device)
    cases = {"masked": lambda: "masked", "mlp_greedy_fused": lambda: mlp, "lstm_greedy_fused": lambda: lstm,
             # the PyTorch path of a reference-shape module, called directly (a module alone gets the fused kernel);
             # a fresh actor per run: it carries the LSTM state
             "lstm_greedy_torch": lambda: (lambda e, o, act=_torch_actor(env, lstm, False): act(o))}
    res = {}
    for name, make in cases.items():
        def run(max_steps=None):
            return _play(env, make(), max_steps)

        run(8)   # warm-up: module load, weight upload, allocator
        times, steps = [], 0
        for _ in range(rounds):
            torch.cuda.synchronize(env.device)
            t0 = time.perf_counter()
            acc = run()
            times.append(time.perf_counter() - t0)
            steps = int(acc["timesteps"].max())
        n = num_episodes * env.N * steps
        res[name] = {"loop_s": min(times), "rounds_s": times, "loop_steps": steps,
                     "episodes_per_s": num_episodes / min(times), "agent_steps_per_s": n / min(times)}
    env.close()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    evaluate(cfg, num_episodes, "masked", device)
    res["evaluate_masked_s"] = time.perf_counter() - t0
    ccfg = {"num_agents": 16, "steps_per_episode": 256, "seed": 999, "grid": cfg["grid"]}
    cenv = BatchedCteEnv(ccfg, num_episodes, device)
    torch.manual_seed(0)
    cmlp = CteActionMaskPolicy(cenv.R * cenv.C, cenv.N).to(cenv.device)
    clstm = CteRecurrentPolicy(cenv.R * cenv.C, cenv.N).to(cenv.device)
    ccases = {"cte_masked": lambda: "masked", "cte_mlp_greedy_fused": lambda: cmlp, "cte_lstm_greedy_fused": lambda: clstm,
              "cte_lstm_greedy_torch": lambda: (lambda e, o, act=_cte_torch_actor(cenv, clstm, False): act())}
    for name, make in ccases.items():
        def crun(max_steps=None):
            return _play_cte(cenv, make(), max_steps)

        crun(8)
        times, steps = [], 0
        for _ in range(rounds):
            torch.cuda.synchronize(cenv.device)
            t0 = time.perf_counter()
            acc = crun()
            times.append(time.perf_counter() - t0)
            steps = int(acc["timesteps"].max())
        n = num_episodes * cenv.N * steps
        res[name] = {"loop_s": min(times), "rounds_s": times, "loop_steps": steps,
                     "episodes_per_s": num_episodes / min(times), "agent_steps_per_s": n / min(times)}
    del cenv
    try:
        gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                              str(torch.device(device).index or 0)], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as exc:
        gpu = f"nvidia-smi not readable: {exc}"
    return {"gpu": gpu or torch.cuda.get_device_name(device), "episodes": num_episodes, "agents": 16,
            "steps_per_episode": 256, **res}


if __name__ == "__main__":
    import json

    print(json.dumps(benchmark()))
