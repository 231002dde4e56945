"""Single-agent ("CTE") view of the MAPF grid on the CUDA kernels.

Replaces ``src/environments/reference_model_single_agent.py`` of the reference (``CTE:line``): all agents are driven
by ONE joint ``MultiDiscrete([5] * N)`` action, the observation is the full grid (1 obstacle, ``2i+2`` agent i,
``2i+3`` goal of agent i) followed by the 5N action mask, flattened to float32, and the reward is one scalar with
the blocking / move-after-goal penalties (CTE:92-93).

* :class:`BatchedCteEnv` -- B envs stepped by one launch of ``mapf_cte_kernel`` (tensor API, device resident);
* :class:`ReferenceModel` -- the reference's ``gym.Env`` API as a B = 1 view: same ``reset()`` / ``step(action)``
  signatures and payloads (float32 flat obs, Python float reward, Python bools, ``info`` with ``action_mask`` and the
  four counters), same attributes (``positions`` / ``starts`` / ``goals`` dicts of arrays, ``step_count``,
  ``goal_reached_once``, ``grid``, ``seed``, ``rng``, ``_obs_slices`` ...).

Layout draws (CTE:155-185): ``rng_backend="numpy"`` (the default of a B = 1 env) keeps them on the host with a
``numpy.random.Generator`` exactly like the reference, so a seeded B = 1 env reproduces the reference's episodes bit
for bit; ``rng_backend="device"`` (the default for B > 1) draws them on the GPU -- the multi-agent reset kernel's Philox
layout draw, distributionally the same 2N distinct free cells -- so that resets, and ``step(..., auto_reset=True)``,
of a big batch never touch the host.  The transition always runs on the GPU (no CPU fallback).
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _native as nat
from . import maps
from .spaces import Box, MultiBinary, MultiDiscrete

INFO_KEYS = ("blocking_count_step", "goals_reached_step", "goals_reached_total", "blocking_count_total")


def draw_layout(rng: np.random.Generator, grid: np.ndarray, num_agents: int):
    """CTE:155-185, call for call: unique starts, then unique goals that are not a start."""
    available = np.argwhere(grid == 0)
    starts, goals = [], []
    for _ in range(num_agents):
        while True:
            pos = available[rng.choice(len(available))]
            if not any(np.array_equal(pos, q) for q in starts):
                starts.append(pos)
                break
    for _ in range(num_agents):
        while True:
            pos = available[rng.choice(len(available))]
            if not any(np.array_equal(pos, q) for q in goals) and not any(np.array_equal(pos, q) for q in starts):
                goals.append(pos)
                break
    return np.array(starts, np.int16), np.array(goals, np.int16)


class BatchedCteEnv:
    """B independent CTE envs on one GPU.  ``env_config``: the reference's keys (CTE:84-95) plus ``grid`` (inline map)."""

    def __init__(self, env_config: dict, num_envs: int, device="cuda:0"):
        if not torch.cuda.is_available():
            raise RuntimeError("no CUDA device available: dl_reference_models_b200 has no CPU fallback")
        self.env_config = dict(env_config)
        self.device = torch.device(device)
        self._lib = nat.lib()
        g = self.env_config.get
        self.grid = (np.ascontiguousarray(np.asarray(g("grid")), dtype=np.uint8) if g("grid") is not None
                     else maps.get_grid(self.env_config["env_name"]))
        self.R, self.C = (int(x) for x in self.grid.shape)
        self.B, self.N = int(num_envs), int(g("num_agents", 2))
        self.steps_per_episode = int(g("steps_per_episode", 100))
        self.deterministic = bool(g("deterministic", False))
        self.seed = g("seed", None)
        self.rng_backend = str(g("rng_backend", "numpy" if int(num_envs) == 1 else "device"))
        if self.rng_backend not in ("numpy", "device"):
            raise ValueError("rng_backend must be 'numpy' or 'device'")
        self._layout_env = None
        self.D = self.R * self.C + 5 * self.N
        dev = self.device
        z = lambda shape, dt: torch.zeros(shape, dtype=dt, device=dev)  # noqa: E731
        B, N = self.B, self.N
        self.grid_dev = torch.from_numpy(self.grid).to(dev)
        self.positions, self.goals, self.starts = z((B, N, 2), torch.int16), z((B, N, 2), torch.int16), z((B, N, 2), torch.int16)
        self.reached_once, self.step_count = z((B, N), torch.uint8), z((B,), torch.int32)
        self.blocking_total = z((B,), torch.float64)
        self.obs_grid, self.action_mask = z((B, self.R, self.C), torch.uint8), z((B, 5 * N), torch.int8)
        self.flat_obs, self.reward = z((B, self.D), torch.float32), z((B,), torch.float64)
        self.terminated, self.truncated = z((B,), torch.uint8), z((B,), torch.uint8)
        self.info, self._err = z((B, 4), torch.float64), z((1,), torch.int32)
        self._args = nat.MapfCteArgs(
            num_envs=B, num_agents=N, rows=self.R, cols=self.C, steps_per_episode=self.steps_per_episode, reserved=0,
            blocking_penalty=float(g("blocking_penalty", -0.2)), move_after_goal_penalty=float(g("move_after_goal_penalty", -0.05)),
            grid=self.grid_dev.data_ptr(), positions=self.positions.data_ptr(), goals=self.goals.data_ptr(),
            reached_once=self.reached_once.data_ptr(), step_count=self.step_count.data_ptr(),
            blocking_total=self.blocking_total.data_ptr(), actions=None, obs_grid=self.obs_grid.data_ptr(),
            action_mask=self.action_mask.data_ptr(), flat_obs=self.flat_obs.data_ptr(), reward=self.reward.data_ptr(),
            terminated=self.terminated.data_ptr(), truncated=self.truncated.data_ptr(), info=self.info.data_ptr(),
            err_bits=self._err.data_ptr(), reset_mask=None)
        # numpy backend: one Generator per env, env 0 seeded like the reference (default_rng(seed), CTE:97-101)
        nrng = B if self.rng_backend == "numpy" else 1
        self._rngs = [np.random.default_rng(None if self.seed is None else (self.seed if e == 0 else [int(self.seed), e]))
                      for e in range(nrng)]
        if self.rng_backend == "device" and not self.deterministic:
            # the layout source: a multi-agent handle of the same map / agent count whose masked reset draws 2N distinct
            # free cells per env with Philox (mapf_reset_kernel); only its starts / goals tensors are used
            from .batched_env import BatchedMapfEnv

            self._layout_env = BatchedMapfEnv({"grid": self.grid, "num_agents": N, "sensor_range": 1,
                                               "seed": 0 if self.seed is None else int(self.seed),
                                               "enable_lock_metrics": False}, B, dev)
        if self.deterministic:
            name = self.env_config["env_name"]
            sp, gp = maps.get_start_positions(name, N), maps.get_goal_positions(name, N)
            st = np.array([sp[f"agent_{i}"] for i in range(N)], np.int16)
            gl = np.array([gp[f"agent_{i}"] for i in range(N)], np.int16)
            self.starts.copy_(torch.from_numpy(np.broadcast_to(st, (B, N, 2)).copy()))
            self.goals.copy_(torch.from_numpy(np.broadcast_to(gl, (B, N, 2)).copy()))
        else:
            self._draw(None)   # the reference draws once in the constructor (CTE:112) ...
        self.positions.copy_(self.starts)

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _draw(self, mask):
        """New layouts for the envs of ``mask`` (uint8 [B] device tensor; None = all)."""
        if self._layout_env is not None:
            le = self._layout_env
            le.reset(mask=mask)
            if mask is None:
                self.starts.copy_(le.state["starts"])
                self.goals.copy_(le.state["goals"])
            else:
                m = mask.bool().view(self.B, 1, 1)
                torch.where(m, le.state["starts"], self.starts, out=self.starts)
                torch.where(m, le.state["goals"], self.goals, out=self.goals)
            return
        env_ids = np.arange(self.B) if mask is None else np.flatnonzero(mask.cpu().numpy())
        st = self.starts.cpu().numpy()
        gl = self.goals.cpu().numpy()
        for e in env_ids:
            st[e], gl[e] = draw_layout(self._rngs[int(e)], self.grid, self.N)
        self.starts.copy_(torch.from_numpy(st))
        self.goals.copy_(torch.from_numpy(gl))

    def reset(self, mask=None, starts=None, goals=None):
        """CTE:218-235 for the selected envs (uint8 [B] mask, None = all).  Deterministic envs go back to their
        starts, the others draw a fresh layout (... and again on every reset, CTE:227); ``starts`` / ``goals``
        (int16 [B,N,2]) install a given layout instead.  With the device RNG backend nothing here waits for the GPU."""
        m = (torch.ones(self.B, dtype=torch.uint8, device=self.device) if mask is None
             else torch.as_tensor(mask).to(device=self.device, dtype=torch.uint8).reshape(self.B).contiguous())
        if starts is not None:
            self.starts.copy_(torch.as_tensor(np.asarray(starts), dtype=torch.int16).reshape(self.B, self.N, 2))
            self.goals.copy_(torch.as_tensor(np.asarray(goals), dtype=torch.int16).reshape(self.B, self.N, 2))
        elif not self.deterministic:
            self._draw(None if mask is None else m)
        self._reset_launch(m, self._args)
        return self.flat_obs

    def _reset_launch(self, m, args):
        """Positions of the envs of ``m`` (uint8 [B] device tensor) back to their starts, then ``mapf_cte_reset`` with
        the output pointers of ``args`` (the env's own, or a rollout's rows)."""
        torch.where(m.bool().view(self.B, 1, 1), self.starts, self.positions, out=self.positions)
        self._reset_mask = m   # outlives the launch (replaced by the next reset, stream-ordered)
        args.reset_mask = m.data_ptr()
        nat.check(self._lib.mapf_cte_reset(C.byref(args), self._stream()))
        args.reset_mask = None

    def step(self, actions, auto_reset: bool = False):
        """CTE:237-346 for every env.  ``actions``: int8 [B,N] joint actions.  ``auto_reset`` (no reference counterpart,
        the vector-env convention of the multi-agent batch API): envs whose episode ended in this step are reset behind
        it -- ``flat_obs`` then holds the first observation of their next episode, ``reward`` / ``terminated`` /
        ``truncated`` / ``info`` still describe the step that ended the episode."""
        a = torch.as_tensor(actions).to(device=self.device, dtype=torch.int8).reshape(self.B, self.N).contiguous()
        self._actions = a
        self._args.actions = a.data_ptr()
        nat.check(self._lib.mapf_cte_step(C.byref(self._args), self._stream()))
        if auto_reset:
            self.reset(mask=self.terminated | self.truncated)
        return self.flat_obs, self.reward, self.terminated, self.truncated, self.info

    def poll_errors(self) -> int:
        bits = int(self._err.item())
        self._err.zero_()
        return bits


class ReferenceModel:
    """``gym.Env``-style B = 1 view with the reference's payloads (CTE:84-346)."""

    metadata: dict = {}

    def __init__(self, env_config):
        cfg = dict(env_config)
        self._env = BatchedCteEnv(cfg, 1, cfg.get("device", "cuda:0"))
        e = self._env
        self.step_count = 0
        self.steps_per_episode = e.steps_per_episode
        self.num_agents = e.N
        self.sensor_range = cfg.get("sensor_range", 1)
        self.deterministic = e.deterministic
        self._agent_ids = {f"agent_{i}" for i in range(e.N)}
        self.render_env = cfg.get("render_env", False)
        self.blocking_penalty = cfg.get("blocking_penalty", -0.2)
        self.move_after_goal_penalty = cfg.get("move_after_goal_penalty", -0.05)
        self._episode_blocking_count = 0.0
        self.validate_observation_space = bool(cfg.get("validate_observation_space", False))
        self.seed = cfg.get("seed", None)
        self.rng = e._rngs[0]
        self.grid = e.grid
        self._grid_obs_space = Box(low=0, high=2 * e.N + 1, shape=(e.R, e.C), dtype=np.uint8)
        self._action_mask_space = MultiBinary(5 * e.N)
        flat_grid_len, flat_mask_len = e.R * e.C, 5 * e.N
        low = np.zeros(flat_grid_len + flat_mask_len, np.float32)
        high = np.concatenate([np.full(flat_grid_len, 2 * e.N + 1, np.float32), np.ones(flat_mask_len, np.float32)])
        self._obs_slices = {"grid": slice(0, flat_grid_len), "action_mask": slice(flat_grid_len, flat_grid_len + flat_mask_len)}
        self.observation_space = Box(low=low, high=high, dtype=np.float32)
        self.action_space = MultiDiscrete([5] * e.N)
        self._sync()

    def _sync(self):
        e = self._env
        pos, st, gl = (t[0].cpu().numpy() for t in (e.positions, e.starts, e.goals))
        ids = [f"agent_{i}" for i in range(e.N)]
        self.positions = {a: pos[i].copy() for i, a in enumerate(ids)}
        self.starts = {a: st[i].copy() for i, a in enumerate(ids)}
        self.goals = {a: gl[i].copy() for i, a in enumerate(ids)}
        once = e.reached_once[0].cpu().numpy()
        self.goal_reached_once = {a: bool(once[i]) for i, a in enumerate(ids)}
        self.step_count = int(e.step_count[0])
        self._episode_blocking_count = float(e.blocking_total[0])

    def _checked(self, obs: np.ndarray, where: str) -> np.ndarray:
        if self.validate_observation_space and not self.observation_space.contains(obs):   # CTE:198-209
            raise ValueError(f"{where} produced observation outside observation_space "
                             f"(dtype={obs.dtype}, min={float(obs.min())}, max={float(obs.max())}).")
        return obs

    def split_flat_observation(self, flat_obs: np.ndarray):
        grid = flat_obs[self._obs_slices["grid"]].reshape(self._grid_obs_space.shape)
        return {"observations": grid, "action_mask": flat_obs[self._obs_slices["action_mask"]]}

    def reset(self, *, seed=None, options=None):
        e = self._env
        obs = e.reset()[0].cpu().numpy()
        self._sync()
        return self._checked(obs, "reset"), {"action_mask": e.action_mask[0].cpu().numpy().copy()}

    def step(self, action):
        e = self._env
        a = np.asarray(action).reshape(-1)
        if a.shape[0] != e.N or np.any(a < 0) or np.any(a > 4):
            raise ValueError("Invalid action")   # CTE:375-377
        e.step(a.astype(np.int8)[None])
        obs = e.flat_obs[0].cpu().numpy()
        self._sync()
        info_v = e.info[0].cpu().numpy()
        info = {"action_mask": e.action_mask[0].cpu().numpy().copy()}
        info.update({k: float(v) for k, v in zip(INFO_KEYS, info_v)})
        return (self._checked(obs, "step"), float(e.reward[0]), bool(e.terminated[0]), bool(e.truncated[0]), info)

    def get_obs(self):
        return self._env.obs_grid[0].cpu().numpy().copy()

    def get_action_mask(self, obs=None):
        return self._env.action_mask[0].cpu().numpy().copy()

    def render(self):  # the matplotlib view of the reference (CTE:491-590) is out of scope
        raise NotImplementedError("render() is not part of the GPU path")

    def close(self):
        pass
