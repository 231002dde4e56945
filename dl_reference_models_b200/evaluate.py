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

``python -m dl_reference_models_b200.evaluate`` times the evaluator (:func:`benchmark`).
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field

import numpy as np
import torch

from . import _native as nat
from . import rollout
from .batched_env import BatchedMapfEnv
from .policy_kernels import FusedPolicy, FusedRecurrentPolicy
from .recurrent import PerAgentRecurrentPolicy, RecurrentActionMaskPolicy

MODULE_TYPES = (rollout.ActionMaskPolicy, RecurrentActionMaskPolicy, rollout.PerAgentActionMaskPolicy, PerAgentRecurrentPolicy)
RECURRENT_TYPES = (RecurrentActionMaskPolicy, PerAgentRecurrentPolicy)


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


def evaluate(env_config: dict, num_episodes: int, policy="random", device="cuda:0", max_steps: int | None = None,
             explore: bool = False) -> EvalResult:
    """Play ``num_episodes`` episodes, one per env of a batch.  ``policy``: ``"random"``, ``"masked"``, a callable
    ``policy(env, out) -> int8 [B,N]``, or a trained :class:`rollout.ActionMaskPolicy` /
    :class:`recurrent.RecurrentActionMaskPolicy` / :class:`rollout.PerAgentActionMaskPolicy` /
    :class:`recurrent.PerAgentRecurrentPolicy` (``num_agents`` = the env's) on ``device``, played as the reference's ``forward_inference`` (argmax
    of the masked logits; ``explore=True``: a draw from them)."""
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
    count read).  ``evaluate_masked_s`` is one whole :func:`evaluate` call, env construction and rows included."""
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
