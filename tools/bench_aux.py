"""Timings of the kernels next to the hot path (CUDA events, warm-up, L2-sized working sets): the fused policy
kernels (MLP and LSTM-64, shared and per-agent; the CTE MLP and LSTM-64), the GAE scan, the V-trace scan, the single-agent (CTE) step, DQN's Q kernel and replay kernels.  Prints one JSON
object.  `python tools/bench_aux.py` (every entry), `python tools/bench_aux.py vtrace` (the V-trace entry alone) or
`python tools/bench_aux.py dqn` (the DQN entries alone)"""
import json
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))

from dl_reference_models_b200 import maps, policy_kernels  # noqa: E402
from dl_reference_models_b200.batched_env import BatchedMapfEnv  # noqa: E402
from dl_reference_models_b200.recurrent import RecurrentActionMaskPolicy  # noqa: E402
from dl_reference_models_b200.rollout import ActionMaskPolicy  # noqa: E402
from dl_reference_models_b200.single_agent import BatchedCteEnv  # noqa: E402


def timed(fn, n=50, warm=5):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n * 1e-3


def weight_reloads(B, N, warps, max_blocks):
    """Weight blocks the per-agent kernels load per launch: one per (CTA, agent) pair of the CTAs' contiguous tile
    ranges (the grid and the split of mapf_b200.cu / pol_per_agent_tiles)."""
    tpa = (B + 31) // 32
    ntiles = tpa * N
    G = min((ntiles + warps - 1) // warps, max_blocks)
    q, rm = divmod(ntiles, G)
    n = 0
    for b in range(G):
        k0 = b * q + min(b, rm)
        k1 = k0 + q + (1 if b < rm else 0)
        n += (k1 - 1) // tpa - k0 // tpa + 1 if k1 > k0 else 0
    return n, G


def per_agent_entry(shared_fn, per_agent_fn, one_agent_fn, agents, bytes_per_agent, block_bytes, reloads, blocks):
    """Shared and per-agent launches timed alternately (shared, per-agent, per-agent over the same channels viewed as
    B*N envs of one agent, twice) in one process.  The one-agent view runs the per-agent kernel's gather and tile loop
    over consecutive rows with one weight block per CTA: its gap to the shared launch is the per-agent code path, its gap
    to the per-agent launch the strided rows and the weight reloads."""
    sh, pa, one = [], [], []
    for _ in range(2):
        sh.append(timed(shared_fn, 200))
        pa.append(timed(per_agent_fn, 200))
        one.append(timed(one_agent_fn, 200))
    s = min(pa)
    nbytes = bytes_per_agent * agents + reloads * block_bytes
    return {"us_per_launch": s * 1e6, "rounds_us": [x * 1e6 for x in pa], "shared_rounds_us": [x * 1e6 for x in sh],
            "one_agent_view_rounds_us": [x * 1e6 for x in one],
            "ratio_to_shared": s / min(sh), "agents": agents, "weight_block_bytes": block_bytes, "ctas": blocks,
            "weight_reloads": reloads, "reload_bytes": reloads * block_bytes, "GBps": nbytes / s / 1e9,
            "agent_steps_per_s": agents / s}


def cte_policy_act_entry(B, N=16):
    """The fused centralised CTE policy (mapf_cte_policy_act) at 65 536 envs x 16 agents on the 32x32 benchmark map,
    over a rotation of 4 env batches (4 x 72 MB of grid codes and masks: more than L2)."""
    from dl_reference_models_b200.cte_rollout import CteActionMaskPolicy

    ccfg = {"grid": maps.random_obstacle_grid(32, 32, 0.30, 2026, min_free=32), "num_agents": N, "steps_per_episode": 256,
            "seed": 999}
    envs = [BatchedCteEnv(ccfg, B) for _ in range(4)]
    for e in envs:
        e.reset()
    cells = envs[0].R * envs[0].C
    policy = CteActionMaskPolicy(cells, N).cuda()
    fused = [policy_kernels.FusedCtePolicy(policy, e, env_id_base=k * B) for k, e in enumerate(envs)]
    i = [0]

    def act():
        fused[i[0] % 4].act()
        i[0] += 1

    s = timed(act, 200)
    # byte / FLOP model per env: grid codes R*C + mask 5N in; int8 + int64 actions, joint logp, value out.  GEMMs
    # without padding: R*C x 64, 64 x 64, 64 x (5N + 1)
    nbytes = (cells + 5 * N) + (N + 8 * N + 4 + 4)
    flops = 2 * (cells * 64 + 64 * 64 + 64 * (5 * N + 1))
    hbm_tbs, bf16_tflops = 6.45, 2250.0   # SURVEY 8d measured copy bandwidth; dense bf16 data-sheet rate (tcgen05)
    gbps, tflops = nbytes * B / s / 1e9, flops * B / s / 1e12
    return {"us_per_launch": s * 1e6, "envs": B, "agents": N, "cells": cells, "bytes_per_env": nbytes,
            "flops_per_env": flops, "GBps": gbps, "TFLOPs": tflops, "env_steps_per_s": B / s,
            "frac_of_hbm_6450GBps": gbps / (hbm_tbs * 1e3), "frac_of_bf16_2250TFLOPs": tflops / bf16_tflops,
            "hbm_floor_us": nbytes * B / (hbm_tbs * 1e12) * 1e6}


def cte_lstm_policy_act_entry(B, N=16):
    """The fused recurrent centralised CTE policy (mapf_cte_lstm_policy_act: trunk launch + recurrent step launch) at
    65 536 envs x 16 agents on the 32x32 benchmark map, state advanced in place, the env's episode-end flags as the
    episode-start flags, over the same rotation of 4 env batches as cte_policy_act.  The call is timed with CUDA
    events; each kernel's share comes from a separate torch.profiler run over the same rotation."""
    from dl_reference_models_b200.cte_rollout import CteRecurrentPolicy

    ccfg = {"grid": maps.random_obstacle_grid(32, 32, 0.30, 2026, min_free=32), "num_agents": N, "steps_per_episode": 256,
            "seed": 999}
    envs = [BatchedCteEnv(ccfg, B) for _ in range(4)]
    for e in envs:
        e.reset()
    cells = envs[0].R * envs[0].C
    policy = CteRecurrentPolicy(cells, N).cuda()
    fused = [policy_kernels.FusedCteRecurrentPolicy(policy, e, env_id_base=k * B) for k, e in enumerate(envs)]
    states = [(torch.zeros((B, 64), device="cuda"), torch.zeros((B, 64), device="cuda")) for _ in envs]
    i = [0]

    def act():
        k = i[0] % 4
        e = envs[k]
        fused[k].act(states[k], fused[k].actions, e.reward, e.terminated, e.truncated)
        i[0] += 1

    s = timed(act, 200)
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(40):
            act()
        torch.cuda.synchronize()
    dev_us = {}
    for ev in prof.key_averages():
        for kname in ("mapf_cte_lstm_trunk_kernel", "mapf_cte_lstm_step_kernel"):
            if kname in ev.key:
                dev_us[kname] = getattr(ev, "device_time_total", getattr(ev, "cuda_time_total", 0.0)) / 40
    # byte / FLOP models per env.  trunk: grid codes R*C in, bf16 y (128 B) out; GEMMs R*C x 64, 64 x 64.  step: y,
    # mask 5N, previous actions N, f64 reward, two flags, h / c in and out (4 x 256 B), int8 + int64 actions, joint
    # logp, value; GEMMs 256 x (64 + 5N + 1 + 64) gates and 64 x (5N + 1) heads, without padding
    b_trunk, b_step = cells + 128, 128 + 5 * N + N + 8 + 2 + 4 * 256 + N + 8 * N + 4 + 4
    f_trunk, f_step = 2 * (cells * 64 + 64 * 64), 2 * (256 * (64 + 5 * N + 1 + 64) + 64 * (5 * N + 1))
    hbm_tbs, bf16_tflops = 6.45, 2250.0   # SURVEY 8d measured copy bandwidth; dense bf16 data-sheet rate (tcgen05)
    gbps, tflops = (b_trunk + b_step) * B / s / 1e9, (f_trunk + f_step) * B / s / 1e12
    prof_total = sum(dev_us.values()) or float("nan")
    return {"us_per_call": s * 1e6, "envs": B, "agents": N, "cells": cells,
            "kernel_us_profiler": dev_us,
            "trunk_share": dev_us.get("mapf_cte_lstm_trunk_kernel", float("nan")) / prof_total,
            "step_share": dev_us.get("mapf_cte_lstm_step_kernel", float("nan")) / prof_total,
            "bytes_per_env": {"trunk": b_trunk, "step": b_step}, "flops_per_env": {"trunk": f_trunk, "step": f_step},
            "GBps": gbps, "TFLOPs": tflops, "env_steps_per_s": B / s,
            "frac_of_hbm_6450GBps": gbps / (hbm_tbs * 1e3), "frac_of_bf16_2250TFLOPs": tflops / bf16_tflops}


def vtrace_entry(T=64, B=65536, N=16):
    """The V-trace scan (mapf_vtrace) at C3: the identity launch over [T, B*N] (24 B per column-step -- rewards,
    behaviour and target logp, values in, vs and pg_advantages out -- plus T*B bytes of dones: 1.6 GB, more than L2),
    and the learner-shaped launch, 1024 // T = 16 gathered columns of the same batch."""
    from dl_reference_models_b200 import impala

    g = torch.Generator(device="cuda").manual_seed(0)
    mu, r = torch.randn(T, B, N, device="cuda", generator=g) - 1.5, torch.randn(T, B, N, device="cuda", generator=g)
    dones = torch.rand(T, B, device="cuda", generator=g) < 0.01
    boot = torch.randn(B, N, device="cuda", generator=g)
    pi, v = mu.reshape(T, -1) + 0.1 * torch.randn(T, B * N, device="cuda", generator=g), torch.randn(T, B * N, device="cuda", generator=g)
    s = timed(lambda: policy_kernels.vtrace(pi, mu, v, r, dones, boot), 20)
    nbytes = 24 * T * B * N + T * B
    hbm_tbs = 6.45   # SURVEY 8d measured copy bandwidth
    cols = torch.randperm(B * N, device="cuda", generator=g)[:1024 // T]
    pic, vc = pi[:, cols].contiguous(), v[:, cols].contiguous()
    sg = timed(lambda: policy_kernels.vtrace(pic, mu, vc, r, dones, boot, columns=cols), 500)
    st = timed(lambda: impala.vtrace(pic, mu, vc, r, dones, boot, columns=cols), 50)
    return {"identity": {"T": T, "columns": B * N, "us_per_launch": s * 1e6, "bytes": nbytes, "GBps": nbytes / s / 1e9,
                         "hbm_floor_us_at_6450GBps": nbytes / (hbm_tbs * 1e12) * 1e6,
                         "frac_of_hbm_6450GBps": nbytes / s / 1e9 / (hbm_tbs * 1e3)},
            "gathered": {"T": T, "columns": cols.numel(), "us_per_launch": sg * 1e6, "torch_vtrace_us": st * 1e6}}


def dqn_entries(B=65536, N=16, K=64):
    """DQN's kernels at C3: q_act and q_act_per_agent (epsilon 0.1) alternated with policy_act over the same 4-env
    rotation (working set > L2), and the replay kernels on a K-slot tree of 2^26 leaves (1 GiB: leaves f32, sums f64,
    minimums f32): advance (2 N B leaves written, plus their f64 / f32 subtree nodes), sample and update at the
    learner's sizes (1024 draws shared, 1024 x N per agent)."""
    from dl_reference_models_b200 import dqn
    from dl_reference_models_b200.rollout import PerAgentActionMaskPolicy

    cfg = {"num_agents": N, "sensor_range": 2, "steps_per_episode": 256, "lifelong_mapf": True, "seed": 999,
           "grid": maps.random_obstacle_grid(32, 32, 0.30, 2026, min_free=32)}
    envs = [BatchedMapfEnv(cfg, B, "cuda:0", env_id_base=r * B) for r in range(4)]
    outs = [e.reset() for e in envs]
    F = envs[0].flat_obs_dim(include_action_mask=False)
    policy = ActionMaskPolicy(F).cuda()
    fused = [policy_kernels.FusedPolicy(policy, e) for e in envs]
    qf = [policy_kernels.FusedQPolicy(policy, e) for e in envs]
    pq = [policy_kernels.FusedQPolicy(PerAgentActionMaskPolicy(N, F).cuda(), e) for e in envs]
    i = [0]

    def rot(fn):
        def run():
            k = i[0] % 4
            fn(k)
            i[0] += 1
        return run

    pol, q, qp = [], [], []
    for _ in range(2):
        pol.append(timed(rot(lambda k: fused[k].act(outs[k])), 200))
        q.append(timed(rot(lambda k: qf[k].act(outs[k], 0.1)), 200))
        qp.append(timed(rot(lambda k: pq[k].act(outs[k], 0.1)), 200))
    q_bytes = 25 + 8 + 1 + 5 + 1   # window, goal delta, pressure, mask in; int8 action out
    flops = 2 * (28 * 64 + 64 * 64 + 64 * 6)
    res = {"policy_act_same_run_us": min(pol) * 1e6,
           "q_act": {"us_per_launch": min(q) * 1e6, "rounds_us": [x * 1e6 for x in q], "bytes_per_agent": q_bytes,
                     "flops_per_agent": flops, "GBps": q_bytes * B * N / min(q) / 1e9,
                     "TFLOPs": flops * B * N / min(q) / 1e12},
           "q_act_per_agent": {"us_per_launch": min(qp) * 1e6, "rounds_us": [x * 1e6 for x in qp],
                               "bytes_per_agent": q_bytes, "GBps": q_bytes * B * N / min(qp) / 1e9}}
    for e in envs[1:]:
        e.close()
    buf = dqn.ReplayBuffer(envs[0], K)
    L = buf.sums.numel()
    t = [0]

    def advance():
        buf.advance(t[0] % K, (t[0] + 1) % K)
        t[0] += 1
    for _ in range(K):
        advance()
    buf.filled = K - 1
    s = timed(advance, 100)
    adv_bytes = 2 * N * B * 4 + 2 * N * B * (8 + 4)   # leaves written; about one node (f64 sum + f32 min) per leaf
    res["replay_advance"] = {"us_per_launch": s * 1e6, "leaves": L, "tree_bytes": 16 * L, "bytes": adv_bytes,
                             "GBps": adv_bytes / s / 1e9}
    for name, M, per_agent in (("replay_sample", 1024, False), ("replay_sample_per_agent", 1024 * N, True)):
        buf.per_agent = per_agent
        s = timed(lambda: buf.sample(M), 200)
        res[name] = {"us_per_launch": s * 1e6, "draws": M, "levels": L.bit_length() - 1,
                     "node_reads_per_draw": 2 * (L.bit_length() - 1)}
    buf.per_agent = False
    for name, M in (("replay_update", 1024), ("replay_update_per_agent", 1024 * N)):
        idx, _ = buf.sample(M)
        td = torch.rand(M, device="cuda")
        s = timed(lambda: buf.update_priorities(idx, td), 100)
        res[name] = {"us_per_launch": s * 1e6, "updates": M, "node_writes": M * (L.bit_length() - 1)}
    envs[0].close()
    return res


def gpu_name():
    import subprocess

    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                               "0"], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as exc:
        return f"nvidia-smi not readable: {exc}"


def main():
    if sys.argv[1:] == ["vtrace"]:
        print(json.dumps({"vtrace": vtrace_entry(), "gpu": gpu_name()}))
        return
    if sys.argv[1:] == ["dqn"]:
        print(json.dumps({"dqn": dqn_entries(), "gpu": gpu_name()}))
        return
    res = {}
    B, N = 65536, 16
    cfg = {"num_agents": N, "sensor_range": 2, "steps_per_episode": 256, "lifelong_mapf": True, "seed": 999,
           "grid": maps.random_obstacle_grid(32, 32, 0.30, 2026, min_free=32)}
    envs = [BatchedMapfEnv(cfg, B, "cuda:0", env_id_base=r * B) for r in range(4)]   # rotate: working set > L2
    outs = [e.reset() for e in envs]
    policy = ActionMaskPolicy(envs[0].flat_obs_dim(include_action_mask=False)).cuda()
    fused = [policy_kernels.FusedPolicy(policy, e) for e in envs]
    i = [0]

    def act():
        k = i[0] % 4
        fused[k].act(outs[k])
        i[0] += 1

    s = timed(act, 200)
    bytes_per_agent = 25 + 8 + 1 + 5 + 1 + 8 + 4 + 4   # window, goal delta, pressure, mask in; int8 + int64 action, logp, value out
    res["policy_act"] = {"us_per_launch": s * 1e6, "agents": B * N, "GBps": bytes_per_agent * B * N / s / 1e9,
                         "agent_steps_per_s": B * N / s, "flops": 2 * (28 * 64 + 64 * 64 + 64 * 6) * B * N,
                         "TFLOPs": 2 * (28 * 64 + 64 * 64 + 64 * 6) * B * N / s / 1e12}
    # the MLP runs on mma.sync (K <= 64 per layer, the channels it reads and writes bound it, not the tensor pipe):
    # reported against the measured dense bf16 peak so that nobody has to guess
    try:
        import json as _json
        from pathlib import Path as _Path

        _pk = _json.loads((_Path(__file__).resolve().parents[1] / "MEASURED_PEAKS.json").read_text())
        res["policy_act"]["bf16_peak_TFLOPs"] = float(_pk["bf16_tflops"])
        res["policy_act"]["frac_of_bf16_peak"] = res["policy_act"]["TFLOPs"] / float(_pk["bf16_tflops"])
        res["policy_act"]["frac_of_hbm_peak"] = res["policy_act"]["GBps"] / float(_pk["hbm_gbs"])
    except Exception as exc:   # no peaks file on this box
        res["policy_act"]["bf16_peak_TFLOPs"] = None
        res["policy_act"]["frac_note"] = f"MEASURED_PEAKS.json not readable: {exc}"
    # fused LSTM-64 policy (mapf_lstm_policy_act), same 4-env rotation; state advanced in place, episode starts off
    lstm = RecurrentActionMaskPolicy(envs[0].flat_obs_dim(include_action_mask=False)).cuda()
    lfused = [policy_kernels.FusedRecurrentPolicy(lstm, e) for e in envs]
    lstate = [(torch.randn(B * N, 64, device="cuda") * 0.1, torch.randn(B * N, 64, device="cuda") * 0.1) for _ in envs]
    lprev = [(torch.randint(0, 5, (B, N), dtype=torch.int8, device="cuda"), torch.zeros(B, N, device="cuda")) for _ in envs]

    def lstm_act():
        k = i[0] % 4
        lfused[k].act(outs[k], lstate[k], *lprev[k])
        i[0] += 1

    s = timed(lstm_act, 200)
    # byte / FLOP model per agent: channels 25 + 8 + 1 + 5, prev action 1, prev reward 4, h 256, c 256 in;
    # h 256, c 256, actions 1 + 8, logp 4, value 4 out.  GEMMs without padding: F x 64, 64 x 64, (70 + 64) x 256, 64 x 6
    lstm_bytes = (25 + 8 + 1 + 5 + 1 + 4 + 256 + 256) + (256 + 256 + 1 + 8 + 4 + 4)
    lstm_flops = 2 * (28 * 64 + 64 * 64 + (70 + 64) * 256 + 64 * 6)
    hbm_tbs, bf16_tflops = 6.45, 2250.0   # SURVEY 8d measured copy bandwidth; dense bf16 data-sheet rate (tcgen05)
    gbps, tflops = lstm_bytes * B * N / s / 1e9, lstm_flops * B * N / s / 1e12
    res["lstm_policy_act"] = {"us_per_launch": s * 1e6, "agents": B * N, "bytes_per_agent": lstm_bytes,
                              "flops_per_agent": lstm_flops, "GBps": gbps, "TFLOPs": tflops,
                              "agent_steps_per_s": B * N / s, "frac_of_hbm_6450GBps": gbps / (hbm_tbs * 1e3),
                              "frac_of_bf16_2250TFLOPs": tflops / bf16_tflops,
                              "hbm_floor_us": lstm_bytes * B * N / (hbm_tbs * 1e12) * 1e6}
    # per-agent variants (one weight block per agent, mapf_*_policy_act_per_agent): same shapes, same 4-env rotation,
    # alternated with the shared launches; GB/s = the byte models above plus the per-CTA weight reloads
    from dl_reference_models_b200.recurrent import PerAgentRecurrentPolicy  # noqa: E402
    from dl_reference_models_b200.rollout import PerAgentActionMaskPolicy  # noqa: E402

    F = envs[0].flat_obs_dim(include_action_mask=False)
    pfused = [policy_kernels.FusedPolicy(PerAgentActionMaskPolicy(N, F).cuda(), e) for e in envs]
    plfused = [policy_kernels.FusedRecurrentPolicy(PerAgentRecurrentPolicy(N, F).cuda(), e) for e in envs]

    def pa_act():
        k = i[0] % 4
        pfused[k].act(outs[k])
        i[0] += 1

    def pa_lstm_act():
        k = i[0] % 4
        plfused[k].act(outs[k], lstate[k], *lprev[k])
        i[0] += 1

    import ctypes as C

    from dl_reference_models_b200 import _native as nat  # noqa: E402

    def one_agent_view(k, lstm_kernel):   # env k's channels as B*N envs of one agent (agent 0's block)
        f = plfused[k] if lstm_kernel else pfused[k]
        a = f.args({c: getattr(outs[k], c) for c in ("local_obs", "goal_delta", "blocking_prev", "action_mask")},
                   lstate[k], *lprev[k], state_out=lstate[k], actions=f.actions, actions64=f.actions64, logp=f.logp,
                   value=f.value) if lstm_kernel else None
        if not lstm_kernel:
            p = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
            a = nat.MapfPolicyArgs(v2=f.env.V * f.env.V, feature_dim=f.F, seed=f.seed, local_obs=p(outs[k].local_obs),
                                   goal_delta=p(outs[k].goal_delta), blocking_prev=p(outs[k].blocking_prev),
                                   action_mask=p(outs[k].action_mask), weights=p(f._dev), actions=p(f.actions),
                                   actions64=p(f.actions64), logp=p(f.logp), value=p(f.value))
        a.num_envs, a.num_agents, a.counter = B * N, 1, 1
        return a

    ones = [[one_agent_view(k, False) for k in range(4)], [one_agent_view(k, True) for k in range(4)]]
    lib, stream = nat.lib(), [e._stream() for e in envs]

    def one_act(lstm_kernel):
        fn = lib.mapf_lstm_policy_act_per_agent if lstm_kernel else lib.mapf_policy_act_per_agent

        def run():
            k = i[0] % 4
            nat.check(fn(C.byref(ones[lstm_kernel][k]), stream[k]))
            i[0] += 1
        return run

    sms = torch.cuda.get_device_properties(0).multi_processor_count
    n, G = weight_reloads(B, N, 8, 148 * 8)
    res["policy_act_per_agent"] = per_agent_entry(act, pa_act, one_act(False), B * N, bytes_per_agent, pfused[0]._block, n, G)
    n, G = weight_reloads(B, N, 16, sms)
    res["lstm_policy_act_per_agent"] = per_agent_entry(lstm_act, pa_lstm_act, one_act(True), B * N, lstm_bytes,
                                                       plfused[0]._block, n, G)
    del lstate, lprev
    T = 64
    rewards, values = torch.randn(T, B, N, device="cuda"), torch.randn(T, B, N, device="cuda")
    dones = torch.rand(T, B, device="cuda") < 0.01
    last = torch.randn(B, N, device="cuda")
    s = timed(lambda: policy_kernels.gae(rewards, values, dones, last), 20)
    res["gae"] = {"us_per_launch": s * 1e6, "GBps": (4 * 4 * T * B * N + T * B) / s / 1e9}
    for e in envs:
        e.close()
    ccfg = {"env_name": "ReferenceModel-2-1", "num_agents": 4, "steps_per_episode": 100, "seed": 1, "deterministic": True}
    cte = BatchedCteEnv(ccfg, B)
    cte.reset()
    acts = torch.randint(0, 5, (B, 4), dtype=torch.int8, device="cuda")
    s = timed(lambda: cte.step(acts), 100)
    res["cte_step"] = {"us_per_launch": s * 1e6, "env_steps_per_s": B / s, "agent_steps_per_s": 4 * B / s,
                       "GBps": (cte.D * 4 + 200 + 20 + 40) * B / s / 1e9}
    del cte
    res["cte_policy_act"] = cte_policy_act_entry(B)
    res["cte_lstm_policy_act"] = cte_lstm_policy_act_entry(B)
    res["vtrace"] = vtrace_entry()
    res["dqn"] = dqn_entries()
    try:
        import subprocess

        res["gpu"] = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                                    capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as exc:
        res["gpu"] = f"nvidia-smi not readable: {exc}"
    print(json.dumps(res))


if __name__ == "__main__":
    main()
