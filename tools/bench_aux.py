"""Timings of the kernels next to the hot path (CUDA events, warm-up, L2-sized working sets): the fused policy
kernels (MLP and LSTM-64), the GAE scan, the single-agent (CTE) step.  Prints one JSON object.  `python tools/bench_aux.py`"""
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


def main():
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
    print(json.dumps(res))


if __name__ == "__main__":
    main()
