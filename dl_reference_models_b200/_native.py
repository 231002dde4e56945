"""ctypes binding of ``libmapf_b200.so`` (C ABI declared in ``include/mapf_b200.h``).

The library is built in-tree by :func:`build` (``nvcc -gencode arch=compute_100a,code=sm_100a``)
and is the only compute path of this package: there is no CPU implementation to fall back to,
and every failure (missing library, no CUDA device, wrong architecture) raises.
"""
from __future__ import annotations

import ctypes as C
import os
import shutil
import subprocess
from pathlib import Path

PKG = Path(__file__).resolve().parent
REPO = PKG.parent
CSRC = PKG / "csrc"
LIB_PATH = Path(os.environ.get("MAPF_B200_LIB", PKG / "libmapf_b200.so"))
SOURCES = (CSRC / "mapf_b200.cu", CSRC / "mapf_kernels.cuh", CSRC / "mapf_env_kernel.cuh", CSRC / "mapf_pair_kernel.cuh", CSRC / "mapf_cte_kernel.cuh", CSRC / "mapf_policy_kernel.cuh",
           CSRC / "mapf_policy_lstm_kernel.cuh", CSRC / "mapf_eval_kernel.cuh", CSRC / "mapf_cte_policy_kernel.cuh",
           CSRC / "mapf_cte_lstm_policy_kernel.cuh", CSRC / "mapf_cte_trunk.inc",
           CSRC / "mapf_cte_heads.inc", CSRC / "mapf_vtrace_kernel.cuh", CSRC / "mapf_q_kernel.cuh",
           CSRC / "mapf_replay_kernel.cuh", CSRC / "mapf_pack_kernel.cuh", CSRC / "mapf_host_unpack.h", CSRC / "mapf_host_unpack.cpp",
           REPO / "include" / "mapf_b200.h")

MAX_AGENTS = 32
MAX_SENSOR_RANGE = 3
MAX_LOCK_WINDOW = 32
MAX_DIM = 255
ENV_WORDS = 16
METRIC_COUNT = 16
INFO_WORDS = 16
CTE_INFO_WORDS = 4

OK, ERR_INVALID_ARG, ERR_CUDA, ERR_UNSUPPORTED, ERR_STATE = 0, -1, -2, -3, -4
DEV_ERR_INVALID_ACTION, DEV_ERR_NO_GOAL_CELL, DEV_ERR_TOO_FEW_CELLS, DEV_ERR_DUPLICATE_LAYOUT = 1, 2, 4, 8

# env_words indices
(W_STEP_COUNT, W_LOCK_COUNT, W_LOCK_PREV, W_GOALS_TOTAL, W_BLOCKING_TOTAL, W_DEADLOCK_EVENTS,
 W_LIVELOCK_EVENTS, W_DEADLOCK_STEPS, W_LIVELOCK_STEPS, W_RNG_COUNTER, W_EPISODE_RETURN_X2,
 W_WFG_CYCLE_STEPS, W_EPISODES, W_LOCK_HEAD) = range(14)

AF_REACHED, AF_COMPLETED_ONCE, AF_BLOCKING_PREV, AF_NOT_OWNER = 1, 2, 4, 8

METRIC_NAMES = (
    "episodes", "return_sum", "length_sum", "success_sum", "goals_reached_sum",
    "blocking_count_sum", "deadlock_count_sum", "livelock_count_sum", "deadlock_steps_sum",
    "livelock_steps_sum", "throughput_sum", "completion_ratio_sum", "wfg_cycle_steps_sum",
    "reserved0", "reserved1", "reserved2",
)

SF_TERMINATED, SF_TRUNCATED, SF_DEADLOCK_STEP, SF_LIVELOCK_STEP = 1, 2, 4, 8
SF_DEADLOCK_EVENT, SF_LIVELOCK_EVENT, SF_GOAL_REASSIGNED, SF_WFG_CYCLE = 16, 32, 64, 128
ASF_MOVED, ASF_FAILED_MOVE, ASF_GOAL_REACHED, ASF_BLOCKING, ASF_WFG_CYCLE, ASF_ON_GOAL = 1, 2, 4, 8, 16, 32

(I_GOALS_REACHED_STEP, I_GOALS_REACHED_TOTAL, I_BLOCKING_COUNT_STEP, I_BLOCKING_COUNT_TOTAL,
 I_DEADLOCK_STEP, I_LIVELOCK_STEP, I_DEADLOCK_EVENT_STEP, I_LIVELOCK_EVENT_STEP,
 I_DEADLOCK_EVENTS_TOTAL, I_LIVELOCK_EVENTS_TOTAL, I_DEADLOCK_STEPS_TOTAL, I_LIVELOCK_STEPS_TOTAL,
 I_COMPLETED_COUNT, I_STEP_COUNT, I_REACHED_COUNT, I_WFG_CYCLE_STEPS) = range(16)


class MapfConfig(C.Structure):
    _fields_ = [
        ("num_envs", C.c_int32), ("num_agents", C.c_int32), ("rows", C.c_int32), ("cols", C.c_int32),
        ("sensor_range", C.c_int32), ("steps_per_episode", C.c_int32), ("lifelong_mapf", C.c_int32),
        ("enable_lock_metrics", C.c_int32), ("deadlock_window_steps", C.c_int32),
        ("livelock_window_steps", C.c_int32), ("lock_nearby_manhattan", C.c_int32),
        ("lock_min_neighbors", C.c_int32), ("lock_progress_epsilon_floor", C.c_int32),
        ("normalize_goal_delta", C.c_int32), ("deterministic", C.c_int32), ("per_env_maps", C.c_int32),
        ("env_id_base", C.c_int64), ("seed", C.c_uint64), ("device", C.c_int32), ("step_kernel", C.c_int32),
    ]


STATE_FIELDS = ("positions", "goals", "starts", "agent_flags", "lock_goal_progress", "lock_moved",
                "lock_failed_move", "lock_distance", "env_words", "env_metrics")
OUTPUT_FIELDS = ("local_obs", "action_mask", "goal_delta", "blocking_prev", "reward", "terminated",
                 "truncated", "step_flags", "agent_step_flags", "info")


class MapfState(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in STATE_FIELDS]


class MapfOutputs(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in OUTPUT_FIELDS]


class MapfCteArgs(C.Structure):
    """mapf_cte_args of include/mapf_b200.h (single-agent / CTE view)."""

    _fields_ = [
        ("num_envs", C.c_int32), ("num_agents", C.c_int32), ("rows", C.c_int32), ("cols", C.c_int32),
        ("steps_per_episode", C.c_int32), ("reserved", C.c_int32),
        ("blocking_penalty", C.c_double), ("move_after_goal_penalty", C.c_double),
    ] + [(k, C.c_void_p) for k in (
        "grid", "positions", "goals", "reached_once", "step_count", "blocking_total", "actions", "obs_grid",
        "action_mask", "flat_obs", "reward", "terminated", "truncated", "info", "err_bits", "reset_mask")]


class MapfPolicyArgs(C.Structure):
    """mapf_policy_args of include/mapf_b200.h (fused action-mask MLP + sampler)."""

    _fields_ = [
        ("num_envs", C.c_int32), ("num_agents", C.c_int32), ("v2", C.c_int32), ("feature_dim", C.c_int32),
        ("no_masking", C.c_int32), ("greedy", C.c_int32),
        ("seed", C.c_uint64), ("counter", C.c_uint64), ("env_id_base", C.c_int64),
    ] + [(k, C.c_void_p) for k in (
        "local_obs", "goal_delta", "blocking_prev", "action_mask", "weights", "actions", "actions64", "logp", "value",
        "logits_out", "features_out", "action_mask_out")]


class MapfLstmPolicyArgs(C.Structure):
    """mapf_lstm_policy_args of include/mapf_b200.h (fused LSTM-64 policy + sampler)."""

    _fields_ = [
        ("num_envs", C.c_int32), ("num_agents", C.c_int32), ("v2", C.c_int32), ("feature_dim", C.c_int32),
        ("no_masking", C.c_int32), ("greedy", C.c_int32),
        ("seed", C.c_uint64), ("counter", C.c_uint64), ("env_id_base", C.c_int64),
    ] + [(k, C.c_void_p) for k in (
        "local_obs", "goal_delta", "blocking_prev", "action_mask", "prev_terminated", "prev_truncated", "prev_action",
        "prev_reward", "h_in", "c_in", "h_out", "c_out", "weights", "actions", "actions64", "logp", "value", "logits_out")]


class MapfCtePolicyArgs(C.Structure):
    """mapf_cte_policy_args of include/mapf_b200.h (fused centralised CTE policy + per-agent draws)."""

    _fields_ = [
        ("num_envs", C.c_int32), ("num_agents", C.c_int32), ("cells", C.c_int32), ("reserved", C.c_int32),
        ("seed", C.c_uint64), ("counter", C.c_uint64), ("env_id_base", C.c_int64),
    ] + [(k, C.c_void_p) for k in (
        "obs_grid", "action_mask", "weights", "actions", "actions64", "logp", "value", "logits_out")] + [
        ("greedy", C.c_int32)]


class MapfCteLstmPolicyArgs(C.Structure):
    """mapf_cte_lstm_policy_args of include/mapf_b200.h (fused recurrent centralised CTE policy + per-agent draws)."""

    _fields_ = [
        ("num_envs", C.c_int32), ("num_agents", C.c_int32), ("cells", C.c_int32), ("reserved", C.c_int32),
        ("seed", C.c_uint64), ("counter", C.c_uint64), ("env_id_base", C.c_int64),
    ] + [(k, C.c_void_p) for k in (
        "obs_grid", "action_mask", "prev_terminated", "prev_truncated", "prev_action", "prev_reward", "h_in", "c_in",
        "h_out", "c_out", "trunk", "weights", "actions", "actions64", "logp", "value", "logits_out")] + [
        ("greedy", C.c_int32)]


class MapfEvalArgs(C.Structure):
    """mapf_eval_args of include/mapf_b200.h (the evaluator's per-step bookkeeping)."""

    _fields_ = [("num_envs", C.c_int32), ("num_agents", C.c_int32), ("step", C.c_int64)] + [(k, C.c_void_p) for k in (
        "reward", "terminated", "truncated", "info", "active", "episode_reward", "agent_reward", "timesteps", "success",
        "last_info", "active_count")]


class MapfCteEvalArgs(C.Structure):
    """mapf_cte_eval_args of include/mapf_b200.h (the evaluator's per-step bookkeeping over the single-agent view)."""

    _fields_ = [("num_envs", C.c_int32), ("num_agents", C.c_int32), ("rows", C.c_int32), ("cols", C.c_int32),
                ("step", C.c_int64)] + [(k, C.c_void_p) for k in (
        "positions", "reward", "terminated", "truncated", "info", "active", "episode_reward", "timesteps", "success",
        "last_info", "occupancy", "active_count")]


class MapfVtraceArgs(C.Structure):
    """mapf_vtrace_args of include/mapf_b200.h (V-trace targets over time columns of a rollout)."""

    _fields_ = [("T", C.c_int32), ("num_agents", C.c_int32), ("num_columns", C.c_int64), ("M", C.c_int64)] + [
        (k, C.c_void_p) for k in ("columns", "rewards", "behaviour_logp", "dones", "bootstrap_value", "target_logp",
                                  "values", "vs", "pg_advantages")] + [
        ("gamma", C.c_float), ("clip_rho", C.c_float), ("clip_pg_rho", C.c_float), ("reserved", C.c_int32)]


class MapfQActArgs(C.Structure):
    """mapf_q_act_args of include/mapf_b200.h (fused dueling Q MLP + epsilon-greedy choice)."""

    _fields_ = [
        ("num_envs", C.c_int32), ("num_agents", C.c_int32), ("v2", C.c_int32), ("feature_dim", C.c_int32),
        ("no_masking", C.c_int32), ("epsilon", C.c_float),
        ("seed", C.c_uint64), ("counter", C.c_uint64), ("env_id_base", C.c_int64),
    ] + [(k, C.c_void_p) for k in ("local_obs", "goal_delta", "blocking_prev", "action_mask", "weights", "actions",
                                   "q_out")] + [("reserved", C.c_int32)]


class MapfReplayTree(C.Structure):
    """mapf_replay_tree of include/mapf_b200.h (the prioritized replay sum tree's shape and device arrays)."""

    _fields_ = [("num_envs", C.c_int32), ("num_agents", C.c_int32), ("capacity", C.c_int32)] + [
        (k, C.c_void_p) for k in ("leaves", "sums", "mins", "max_priority")]


class MapfReplayAdvanceArgs(C.Structure):
    _fields_ = [("tree", MapfReplayTree), ("complete", C.c_int32), ("clear", C.c_int32), ("alpha", C.c_float),
                ("reserved", C.c_int32)]


class MapfReplaySampleArgs(C.Structure):
    _fields_ = [("tree", MapfReplayTree), ("M", C.c_int64), ("seed", C.c_uint64), ("counter", C.c_uint64),
                ("beta", C.c_float), ("per_agent", C.c_int32)] + [
        (k, C.c_void_p) for k in ("indices", "weights", "uniforms")] + [("reserved", C.c_int32)]


class MapfReplayUpdateArgs(C.Structure):
    _fields_ = [("tree", MapfReplayTree), ("M", C.c_int64), ("indices", C.c_void_p), ("td_abs", C.c_void_p),
                ("alpha", C.c_float), ("reserved", C.c_int32)]


class MapfError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"libmapf_b200 error {code}: {message}")
        self.code = code
        self.message = message


def nvcc_command(out: Path = LIB_PATH) -> list[str]:
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    return [
        nvcc, "-std=c++17", "-O3", "-shared", "-Xcompiler", "-fPIC",
        "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
        "-Xcompiler", "-pthread",
        "-o", str(out), str(CSRC / "mapf_b200.cu"), str(CSRC / "mapf_host_unpack.cpp"),
    ]


def needs_build() -> bool:
    if "MAPF_B200_LIB" in os.environ:  # explicit library (kernel A/B experiments): never rebuild over it
        return False
    if not LIB_PATH.exists():
        return True
    if not all(s.exists() for s in SOURCES):
        return False
    return LIB_PATH.stat().st_mtime < max(s.stat().st_mtime for s in SOURCES)


def build(force: bool = False) -> Path:
    """Compile the CUDA kernels + C ABI for sm_100a (cross-compiles without a GPU)."""
    if force or needs_build():
        tmp = LIB_PATH.with_suffix(".so.tmp%d" % os.getpid())
        subprocess.run(nvcc_command(tmp), check=True)
        os.replace(tmp, LIB_PATH)
    return LIB_PATH


_lib = None


def lib():
    """Load the shared library (building it first if the sources are newer)."""
    global _lib
    if _lib is not None:
        return _lib
    if needs_build():
        try:
            build()
        except (OSError, subprocess.CalledProcessError) as exc:
            raise ImportError(
                f"libmapf_b200.so is missing or stale and could not be built with nvcc: {exc}. "
                "This package has no CPU fallback."
            ) from exc
    L = C.CDLL(str(LIB_PATH))
    vp, i32, i64, u64 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint64
    L.mapf_version.restype = C.c_char_p
    L.mapf_last_error.restype = C.c_char_p
    L.mapf_create.argtypes = [C.POINTER(MapfConfig), C.POINTER(vp)]
    L.mapf_destroy.argtypes = [vp]
    L.mapf_set_map.argtypes = [vp, vp]
    L.mapf_state_nbytes.argtypes = [vp, C.POINTER(i64 * 10)]
    L.mapf_bind_state.argtypes = [vp, C.POINTER(MapfState)]
    L.mapf_alloc_state.argtypes = [vp]
    L.mapf_get_state_host.argtypes = [vp, C.POINTER(MapfState)]
    L.mapf_set_state_host.argtypes = [vp, C.POINTER(MapfState)]
    L.mapf_reset.argtypes = [vp, vp, vp, vp, C.POINTER(MapfOutputs), vp]
    L.mapf_step.argtypes = [vp, vp, vp, vp, C.POINTER(MapfOutputs), i32, vp]
    L.mapf_observe.argtypes = [vp, C.POINTER(MapfOutputs), vp]
    L.mapf_observe_host.argtypes = [vp, C.POINTER(MapfOutputs)]
    L.mapf_reset_host.argtypes = [vp, vp, vp, vp, C.POINTER(MapfOutputs)]
    L.mapf_step_host.argtypes = [vp, vp, vp, vp, C.POINTER(MapfOutputs), i32]
    L.mapf_step_many.argtypes = [vp, vp, C.POINTER(MapfOutputs), i32, C.c_int64, i32, vp]
    L.mapf_host_transfer_bytes.argtypes = [vp, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
    L.mapf_host_transfer_mode.argtypes = [vp]
    L.mapf_host_wait_stream.argtypes = [vp, vp]
    L.mapf_step_host_records.argtypes = [vp, vp, vp, C.POINTER(MapfOutputs), i32]
    L.mapf_host_memory_probe.argtypes = [vp, C.c_int64, C.POINTER(C.c_int32), C.POINTER(C.c_double), C.POINTER(C.c_double)]
    L.mapf_packed_record_bytes.argtypes = [i32]
    L.mapf_unpack_records.argtypes = [vp, C.c_int64, i32, i32, vp, vp, vp, vp, C.c_float, C.c_float]
    L.mapf_flat_obs_dim.argtypes = [vp, i32, i32, i32]
    L.mapf_pack_flat_obs.argtypes = [vp, C.POINTER(MapfOutputs), i32, i32, i32, vp, vp]
    L.mapf_sample_masked_actions.argtypes = [vp, vp, vp, u64, vp]
    L.mapf_sample_random_actions.argtypes = [vp, vp, u64, vp]
    L.mapf_metrics_reduce.argtypes = [vp, vp, vp]
    L.mapf_set_fused_sampler.argtypes = [vp, vp, i32, u64]
    L.mapf_poll_errors.argtypes = [vp, C.POINTER(C.c_uint32), vp]
    L.mapf_launch_count.argtypes = [vp]
    L.mapf_launch_count.restype = i64
    L.mapf_step_kernel_kind.argtypes = [vp]
    L.mapf_occupancy_accumulate.argtypes = [vp, vp, vp, vp]
    L.mapf_distance_table.argtypes = [vp, vp, vp]
    L.mapf_goal_path_lengths.argtypes = [vp, vp, vp, vp]
    L.mapf_policy_weights_nbytes.argtypes = [i32]
    L.mapf_policy_weights_nbytes.restype = i64
    L.mapf_policy_pack_weights.argtypes = [i32] + [vp] * 9
    L.mapf_policy_act.argtypes = [C.POINTER(MapfPolicyArgs), vp]
    L.mapf_lstm_policy_weights_nbytes.argtypes = [i32]
    L.mapf_lstm_policy_weights_nbytes.restype = i64
    L.mapf_lstm_policy_pack_weights.argtypes = [i32] + [vp] * 13
    L.mapf_lstm_policy_act.argtypes = [C.POINTER(MapfLstmPolicyArgs), vp]
    L.mapf_policy_act_per_agent.argtypes = [C.POINTER(MapfPolicyArgs), vp]
    L.mapf_lstm_policy_act_per_agent.argtypes = [C.POINTER(MapfLstmPolicyArgs), vp]
    L.mapf_cte_policy_weights_nbytes.argtypes = [i32, i32]
    L.mapf_cte_policy_weights_nbytes.restype = i64
    L.mapf_cte_policy_pack_weights.argtypes = [i32, i32] + [vp] * 9
    L.mapf_cte_policy_act.argtypes = [C.POINTER(MapfCtePolicyArgs), vp]
    L.mapf_cte_lstm_policy_weights_nbytes.argtypes = [i32, i32]
    L.mapf_cte_lstm_policy_weights_nbytes.restype = i64
    L.mapf_cte_lstm_policy_pack_weights.argtypes = [i32, i32] + [vp] * 13
    L.mapf_cte_lstm_policy_act.argtypes = [C.POINTER(MapfCteLstmPolicyArgs), vp]
    L.mapf_gae.argtypes = [vp, vp, vp, vp, vp, vp, i32, i64, i32, C.c_float, C.c_float, vp]
    L.mapf_eval_accumulate.argtypes = [C.POINTER(MapfEvalArgs), vp]
    L.mapf_vtrace.argtypes = [C.POINTER(MapfVtraceArgs), vp]
    L.mapf_cte_eval_accumulate.argtypes = [C.POINTER(MapfCteEvalArgs), vp]
    L.mapf_q_act.argtypes = [C.POINTER(MapfQActArgs), vp]
    L.mapf_q_act_per_agent.argtypes = [C.POINTER(MapfQActArgs), vp]
    L.mapf_replay_tree_leaves.argtypes = [i32, i32, i32]
    L.mapf_replay_tree_leaves.restype = i64
    L.mapf_replay_advance.argtypes = [C.POINTER(MapfReplayAdvanceArgs), vp]
    L.mapf_replay_sample.argtypes = [C.POINTER(MapfReplaySampleArgs), vp]
    L.mapf_replay_update.argtypes = [C.POINTER(MapfReplayUpdateArgs), vp]
    L.mapf_cte_step.argtypes = [C.POINTER(MapfCteArgs), vp]
    L.mapf_cte_reset.argtypes = [C.POINTER(MapfCteArgs), vp]
    for name in EXPORTS:
        if name not in ("mapf_version", "mapf_last_error", "mapf_launch_count", "mapf_policy_weights_nbytes",
                        "mapf_lstm_policy_weights_nbytes", "mapf_cte_policy_weights_nbytes",
                        "mapf_cte_lstm_policy_weights_nbytes", "mapf_replay_tree_leaves"):
            getattr(L, name).restype = C.c_int
    _lib = L
    return L


EXPORTS = (
    "mapf_version", "mapf_last_error", "mapf_create", "mapf_destroy", "mapf_set_map",
    "mapf_state_nbytes", "mapf_bind_state", "mapf_alloc_state", "mapf_get_state_host",
    "mapf_set_state_host", "mapf_reset", "mapf_step", "mapf_step_many", "mapf_reset_host", "mapf_step_host",
    "mapf_host_transfer_bytes", "mapf_host_transfer_mode", "mapf_host_wait_stream", "mapf_host_memory_probe", "mapf_step_host_records", "mapf_packed_record_bytes", "mapf_unpack_records",
    "mapf_observe", "mapf_observe_host",
    "mapf_flat_obs_dim", "mapf_pack_flat_obs", "mapf_sample_masked_actions",
    "mapf_sample_random_actions", "mapf_set_fused_sampler", "mapf_metrics_reduce", "mapf_poll_errors", "mapf_launch_count",
    "mapf_step_kernel_kind", "mapf_cte_step", "mapf_cte_reset", "mapf_occupancy_accumulate", "mapf_distance_table", "mapf_goal_path_lengths",
    "mapf_policy_weights_nbytes", "mapf_policy_pack_weights", "mapf_policy_act", "mapf_gae",
    "mapf_lstm_policy_weights_nbytes", "mapf_lstm_policy_pack_weights", "mapf_lstm_policy_act", "mapf_eval_accumulate",
    "mapf_policy_act_per_agent", "mapf_lstm_policy_act_per_agent",
    "mapf_cte_policy_weights_nbytes", "mapf_cte_policy_pack_weights", "mapf_cte_policy_act",
    "mapf_cte_lstm_policy_weights_nbytes", "mapf_cte_lstm_policy_pack_weights", "mapf_cte_lstm_policy_act",
    "mapf_cte_eval_accumulate", "mapf_vtrace",
    "mapf_q_act", "mapf_q_act_per_agent", "mapf_replay_tree_leaves", "mapf_replay_advance", "mapf_replay_sample",
    "mapf_replay_update",
)


def check(rc: int) -> int:
    if rc < 0:
        raise MapfError(rc, lib().mapf_last_error().decode(errors="replace"))
    return rc


def make_config(env_config: dict, rows: int, cols: int, num_envs: int, device: int = 0,
                env_id_base: int = 0, per_env_maps: bool = False) -> MapfConfig:
    """Translate the reference's ``env_config`` keys and defaults (ENV:38-61) into mapf_config."""
    import math

    g = env_config.get
    seed = g("seed", None)
    return MapfConfig(
        num_envs=int(num_envs),
        num_agents=int(g("num_agents", 2)),
        rows=int(rows), cols=int(cols),
        sensor_range=int(g("sensor_range", 1)),
        steps_per_episode=int(g("steps_per_episode", 100)),
        lifelong_mapf=int(bool(g("lifelong_mapf", False))),
        enable_lock_metrics=int(bool(g("enable_lock_metrics", True))),
        deadlock_window_steps=max(1, int(g("deadlock_window_steps", 8))),
        livelock_window_steps=max(1, int(g("livelock_window_steps", 16))),
        lock_nearby_manhattan=max(1, int(g("lock_nearby_manhattan", 2))),
        lock_min_neighbors=max(1, int(g("lock_min_neighbors", 1))),
        lock_progress_epsilon_floor=int(max(-(2 ** 30), min(2 ** 30, math.floor(float(g("lock_progress_epsilon", 1)))))),
        normalize_goal_delta=int(bool(g("normalize_goal_delta", True))),
        deterministic=int(bool(g("deterministic", False))),
        per_env_maps=int(bool(per_env_maps)),
        env_id_base=int(env_id_base),
        seed=(int(seed) if seed is not None else int.from_bytes(os.urandom(8), "little")) & (2 ** 64 - 1),
        device=int(device),
        step_kernel={'auto': 0, 'lane': 1, 'env': 2, 'pair': 3}[str(g('step_kernel', 'auto'))],
    )
