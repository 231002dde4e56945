"""The fused policy, Q, evaluator and replay kernels at the batch sizes training runs at, where every capped grid loops.

Each hot-path launch caps its grid and walks the rest of the batch in a loop: grid-stride loops over 32-row tiles or
envs, contiguous per-CTA tile ranges that reload an agent's weights at each agent change (pol_per_agent_tiles), the
replay tree's 1024-leaf chunks and its one-block top kernel.  The other test files check these kernels at sizes the
first trip covers.  Here every shape takes several trips (C3 = 65 536 envs x 16 agents, or just past one trip with a
partial last tile), and each launch faces three oracles:

* the bf16-rounding torch references of the sibling test files over every row (max 3e-2, mean 2e-4 on logits, Q, value
  and the LSTM state), and greedy actions equal to the first argmax of the launch's own logits / Q;
* launches over env slices [lo, hi) with env_id_base = lo, each one trip long and starting off a 32-row tile
  boundary, equal to the full launch bit for bit (so a row's result depends neither on its trip nor on its tile);
* outputs prefilled with a sentinel (NaN, 0x7F) in buffers with a guard tail: after the launch no row keeps the
  sentinel and the tail is untouched.

The evaluator kernels run on synthetic steps with half-integer rewards (exact f64 sums) against a torch loop of the
same bookkeeping, the replay kernels against the CPU ReplayBuffer and an exact per-node tree reference."""
import ctypes as C
import functools
from types import SimpleNamespace

import pytest
import torch

import test_gpu_cte_lstm_policy as ctel_t
import test_gpu_cte_policy as cte_t
import test_gpu_dqn as dqn_t
import test_gpu_lstm_policy_kernel as lstm_t
import test_gpu_policy_kernels as mlp_t

pytestmark = pytest.mark.gpu

GUARD = 257   # guard rows past the batch
SENTINEL = {torch.float32: float("nan"), torch.float64: float("nan"), torch.int8: 0x7F, torch.uint8: 0x7F,
            torch.int32: 0x7F7F7F7F, torch.int64: 0x7F7F7F7F7F7F7F7F}
CHANNELS = ("local_obs", "goal_delta", "blocking_prev", "action_mask")


def _p(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _nat():
    from dl_reference_models_b200 import _native as nat

    return nat


# ---------------------------------------------------------------------------------------------------------- helpers

def guarded(rows, shape, dtype):
    """A sentinel-filled [rows + GUARD, *shape] device buffer; the launch gets its first `rows` rows."""
    return torch.full((rows + GUARD,) + tuple(shape), SENTINEL[dtype], dtype=dtype, device="cuda")


def _is_sentinel(t):
    return torch.isnan(t) if t.is_floating_point() else t == SENTINEL[t.dtype]


def written_once(bufs, rows):
    """Every one of the first `rows` rows was written, the guard tail was not; returns the rows."""
    torch.cuda.synchronize()
    for name, full in bufs.items():
        assert not bool(_is_sentinel(full[:rows]).any()), f"{name}: a row keeps the sentinel"
        assert bool(_is_sentinel(full[rows:]).all()), f"{name}: written past the batch"
    return {k: v[:rows] for k, v in bufs.items()}


def slices(B, S):
    """Three env slices of at most S envs (one trip), at the start, the middle and the end of the batch, each starting
    at an odd env: off a 32-row tile boundary in the per-env-agent and the per-agent tile orders alike (N < 32)."""
    return [(lo, min(lo + S, B)) for lo in (17, (B // 2) | 1, (B - S) | 1)]


def assert_close(name, got, want):
    d = (got.double() - want.double()).abs()
    assert float(d.max()) <= 3e-2 and float(d.mean()) <= 2e-4, (name, float(d.max()), float(d.mean()))


def assert_same_rows(full, part, lo, hi, per_env):
    for k in part:
        assert torch.equal(part[k], full[k][lo * per_env:hi * per_env]), (k, lo, hi)


@functools.lru_cache(maxsize=4)
def mapf_env(sr, B, n):
    return dqn_t.make_env(sr, B, n)   # lifelong, five masked random steps after the reset


@functools.lru_cache(maxsize=2)
def cte_env(name, n, B):
    return cte_t.make_env(name, n, B)


# --------------------------------------------------------------------------------------- MLP and Q (shared, per agent)

def mlp_launch(fused, ch, lo, hi, counter, mode):
    """One launch of ``fused`` (a FusedPolicy: mode = greedy; a FusedQPolicy: mode = epsilon) over envs [lo, hi) with
    env_id_base lo, into fresh guarded outputs; returns the outputs' rows, flat per (env, agent)."""
    from dl_reference_models_b200.policy_kernels import FusedQPolicy

    nat, N = _nat(), fused.env.N
    rows = (hi - lo) * N
    sub = {k: ch[k][lo:hi] for k in CHANNELS}
    o = {"actions": guarded(rows, (), torch.int8)}
    if isinstance(fused, FusedQPolicy):
        o["q"] = guarded(rows, (5,), torch.float32)
        a = fused.args(sub, mode, o["actions"], o["q"])
    else:
        o.update(actions64=guarded(rows, (), torch.int64), logp=guarded(rows, (), torch.float32),
                 value=guarded(rows, (), torch.float32), logits=guarded(rows, (5,), torch.float32))
        a = nat.MapfPolicyArgs(
            num_envs=0, num_agents=N, v2=fused.env.V ** 2, feature_dim=fused.F, no_masking=0, greedy=int(mode), seed=fused.seed,
            counter=0, env_id_base=0, local_obs=_p(sub["local_obs"]), goal_delta=_p(sub["goal_delta"]),
            blocking_prev=_p(sub["blocking_prev"]) if fused.with_bp else None, action_mask=_p(sub["action_mask"]),
            weights=_p(fused._dev), actions=_p(o["actions"]), actions64=_p(o["actions64"]), logp=_p(o["logp"]),
            value=_p(o["value"]), logits_out=_p(o["logits"]), features_out=None, action_mask_out=None)
    a.num_envs, a.env_id_base, a.counter = hi - lo, lo, counter
    nat.check(fused._act(C.byref(a), None))
    return written_once(o, rows)


def check_mlp_outputs(got, ref_l, ref_v, mode, q):
    """Against the bf16 reference (Q: ref_l is the masked Q); greedy / epsilon 0: the first argmax of the launch's own
    logits / Q; a draw: logp is the log-softmax of the launch's logits at the drawn action."""
    if q:
        assert_close("q", got["q"], ref_l)
        if mode == 0.0:
            assert torch.equal(got["actions"].long(), got["q"].argmax(-1))
        return
    assert_close("logits", got["logits"], ref_l)
    assert_close("value", got["value"], ref_v)
    assert torch.equal(got["actions64"], got["actions"].long())
    if mode:
        assert torch.equal(got["actions"].long(), got["logits"].argmax(-1))
    else:
        ref_logp = torch.log_softmax(got["logits"], -1).gather(-1, got["actions"].long().unsqueeze(-1)).squeeze(-1)
        assert float((got["logp"] - ref_logp).abs().max()) <= 1e-4


# mapf_policy_act / mapf_q_act (policy_launch, q_act_launch): 148 * 8 blocks x 8 warps = 9 472 tiles = 303 104 agents
MLP_SHAPES = [
    (2, 65536, 16),   # C3, F = 28 (KC1 = 2): 32 768 tiles, 3.5 trips
    (3, 65536, 16),   # C3, F = 52 (KC1 = 4)
    (2, 18947, 16),   # 303 152 agents = 9 473.5 tiles: one trip, then a half-full last tile
]


@pytest.mark.parametrize("kind", ["mlp", "q"])
@pytest.mark.parametrize("sr,B,n", MLP_SHAPES)
def test_shared_mlp_and_q_kernels_past_the_first_trip(kind, sr, B, n):
    from dl_reference_models_b200.policy_kernels import FusedPolicy, FusedQPolicy
    from dl_reference_models_b200.rollout import ActionMaskPolicy

    env, out = mapf_env(sr, B, n)
    ch = {k: getattr(out, k) for k in CHANNELS}
    torch.manual_seed(0)
    pol = ActionMaskPolicy(env.flat_obs_dim(include_action_mask=False)).to(env.device)
    q = kind == "q"
    if not q:
        with torch.no_grad():
            for p in pol.parameters():
                p.mul_(3.0)   # larger logits, as test_gpu_policy_kernels
    fused = (FusedQPolicy if q else FusedPolicy)(pol, env, seed=5)
    feats = env.flat_obs(include_action_mask=False).reshape(B * n, -1)
    mask = out.action_mask.reshape(B * n, 5)
    with torch.no_grad():
        ref_l, ref_v = (dqn_t.bf16_q(pol, feats, mask), None) if q else mlp_t.bf16_reference(pol, feats, mask)
    for mode in ((0.0, 0.3) if q else (False, True)):
        full = mlp_launch(fused, ch, 0, B, 3, mode)
        check_mlp_outputs(full, ref_l, ref_v, mode, q)
        for lo, hi in slices(B, 5001):   # 80 016 agents: one trip
            assert_same_rows(full, mlp_launch(fused, ch, lo, hi, 3, mode), lo, hi, n)


# the per-agent launches: 148 * 8 CTAs, each a range of q or q + 1 agent-major tiles walked in rounds of 8
PER_AGENT_SHAPES = [
    (2, 65536, 16),   # C3: 2 048 tiles per agent, 32 768 tiles, q = 27: rounds of 8, ranges that start mid-agent
    (2, 40003, 13),   # 1 251 tiles per agent (the last holds 3 envs), 16 263 tiles, 13-14 per CTA across agent changes
]


@pytest.mark.parametrize("kind", ["mlp", "q"])
@pytest.mark.parametrize("sr,B,n", PER_AGENT_SHAPES)
def test_per_agent_mlp_and_q_kernels_past_the_first_trip(kind, sr, B, n):
    from dl_reference_models_b200.policy_kernels import FusedPolicy, FusedQPolicy
    from dl_reference_models_b200.rollout import PerAgentActionMaskPolicy

    env, out = mapf_env(sr, B, n)
    ch = {k: getattr(out, k) for k in CHANNELS}
    F = env.flat_obs_dim(include_action_mask=False)
    torch.manual_seed(1)
    pa = PerAgentActionMaskPolicy(n, F).to(env.device)
    q = kind == "q"
    cls = FusedQPolicy if q else FusedPolicy
    fused = cls(pa, env, seed=5)
    assert fused.entry.endswith("_per_agent")
    feats = env.flat_obs(include_action_mask=False).reshape(B, n, F)
    mask = out.action_mask.reshape(B, n, 5)
    refs = []
    with torch.no_grad():
        for j in range(n):
            m = pa.module(j)
            refs.append((dqn_t.bf16_q(m, feats[:, j], mask[:, j]), None) if q else mlp_t.bf16_reference(m, feats[:, j], mask[:, j]))
    ref_l = torch.stack([r[0] for r in refs], 1).reshape(B * n, 5)
    ref_v = None if q else torch.stack([r[1] for r in refs], 1).reshape(B * n)
    shared = [cls(pa.module(j), env, seed=5) for j in range(n)]
    for mode in ((0.0, 0.3) if q else (False, True)):
        full = mlp_launch(fused, ch, 0, B, 4, mode)
        check_mlp_outputs(full, ref_l, ref_v, mode, q)
        for j in range(n):   # agent j = the shared launch with block j
            want = mlp_launch(shared[j], ch, 0, B, 4, mode)
            for k in full:
                assert torch.equal(full[k].view(B, n, -1)[:, j], want[k].view(B, n, -1)[:, j]), (mode, j, k)
        for lo, hi in slices(B, 5001):   # 157 tiles per agent, at most 8 per CTA: one round
            assert_same_rows(full, mlp_launch(fused, ch, lo, hi, 4, mode), lo, hi, n)


# ------------------------------------------------------------------------------------------------ LSTM (shared, per agent)

def lstm_launch(fused, ch, inputs, lo, hi, counter, greedy):
    nat, N = _nat(), fused.env.N
    rows = (hi - lo) * N
    h, c, pa, pr, term, trunc = inputs
    o = {"actions": guarded(rows, (), torch.int8), "actions64": guarded(rows, (), torch.int64),
         "logp": guarded(rows, (), torch.float32), "value": guarded(rows, (), torch.float32),
         "logits": guarded(rows, (5,), torch.float32), "h": guarded(rows, (64,), torch.float32),
         "c": guarded(rows, (64,), torch.float32)}
    a = fused.args({k: ch[k][lo:hi] for k in CHANNELS}, (h[lo * N:hi * N], c[lo * N:hi * N]), pa[lo:hi], pr[lo:hi],
                   term[lo:hi], trunc[lo:hi], state_out=(o["h"], o["c"]), actions=o["actions"], actions64=o["actions64"],
                   logp=o["logp"], value=o["value"], logits_out=o["logits"], greedy=greedy)
    a.num_envs, a.env_id_base, a.counter = hi - lo, lo, counter
    nat.check(fused._act(C.byref(a), None))
    return written_once(o, rows)


@pytest.mark.parametrize("per_agent", [False, True])
@pytest.mark.parametrize("shape", ["C3", "one trip + 3 envs"])
def test_lstm_kernels_past_the_first_trip(shape, per_agent):
    from dl_reference_models_b200.policy_kernels import FusedRecurrentPolicy
    from dl_reference_models_b200.recurrent import PerAgentRecurrentPolicy

    sms = torch.cuda.get_device_properties(0).multi_processor_count
    n = 16
    # lstm_policy_launch: SM-count blocks x 16 warps x 32 rows = 512 * SMs agents (32 * SMs envs at N = 16) per trip;
    # per agent, 16 (SMs + 1) tiles over SMs CTAs.  C3: 13.8 trips, 221 tiles per CTA per agent.
    B = 65536 if shape == "C3" else 32 * sms + 3
    env, out = mapf_env(2, B, n)
    ch = {k: getattr(out, k) for k in CHANNELS}
    F = env.flat_obs_dim(include_action_mask=False)
    if per_agent:
        torch.manual_seed(2)
        pol = PerAgentRecurrentPolicy(n, F).to(env.device)
        mods = [pol.module(j) for j in range(n)]
    else:
        pol = lstm_t.make_policy(env, scale=3.0)
        mods = [pol]
    fused = FusedRecurrentPolicy(pol, env, seed=13)
    inputs = lstm_t.random_inputs(env, seed=3)
    h0, c0, pa0, pr0 = lstm_t.cut(env, *inputs)
    feats = env.flat_obs(include_action_mask=False).reshape(B, n, F)
    mask = out.action_mask.reshape(B, n, 5)
    with torch.no_grad():
        if per_agent:   # agent j's rows through module j, stacked back into the [B, N] row order
            refs = [lstm_t.bf16_reference(m, feats[:, j], mask[:, j], pa0[:, j], pr0[:, j], h0.view(B, n, 64)[:, j],
                                          c0.view(B, n, 64)[:, j]) for j, m in enumerate(mods)]
            ref = [torch.stack([r[i] for r in refs], 1).reshape((B * n,) + tuple(refs[0][i].shape[1:])) for i in range(4)]
            del refs
        else:
            ref = lstm_t.bf16_reference(pol, feats.reshape(B * n, F), mask.reshape(B * n, 5), pa0.reshape(-1),
                                        pr0.reshape(-1), h0, c0)
    shared = [FusedRecurrentPolicy(m, env, seed=13) for m in mods] if per_agent else []
    for greedy in (False, True):
        full = lstm_launch(fused, ch, inputs, 0, B, 5, greedy)
        for name, i in (("logits", 0), ("value", 1), ("h", 2), ("c", 3)):
            assert_close(name, full[name], ref[i])
        assert torch.equal(full["actions64"], full["actions"].long())
        if greedy:
            assert torch.equal(full["actions"].long(), full["logits"].argmax(-1))
        else:
            ref_logp = torch.log_softmax(full["logits"], -1).gather(-1, full["actions"].long().unsqueeze(-1)).squeeze(-1)
            assert float((full["logp"] - ref_logp).abs().max()) <= 1e-4
        for j, one in enumerate(shared):   # per agent: agent j = the shared launch with block j
            want = lstm_launch(one, ch, inputs, 0, B, 5, greedy)
            for k in full:
                assert torch.equal(full[k].view(B, n, -1)[:, j], want[k].view(B, n, -1)[:, j]), (greedy, j, k)
        for lo, hi in slices(B, 2001):   # 32 016 agents, 63 tiles per agent: one trip
            assert_same_rows(full, lstm_launch(fused, ch, inputs, lo, hi, 5, greedy), lo, hi, n)


# ---------------------------------------------------------------------------------------------- CTE MLP and CTE LSTM

# mapf_cte_policy_act / mapf_cte_lstm_policy_act: SMs x occupancy (<= 8) blocks x 8 warps <= 9 472 tiles = 303 104 envs
CTE_SHAPES = [
    ("ReferenceModel-2-1", 4, 310003),   # the 10 x 20 map, past the largest possible trip
    ("rand32", 16, 80003),   # 32 x 32: > 113 KB of shared memory per block in every kernel, one block per SM: 37 888 envs
]


def cte_launch(fused, inputs, lo, hi, counter, greedy):
    """One call of a FusedCtePolicy (inputs = None) or FusedCteRecurrentPolicy over envs [lo, hi) with env_id_base lo."""
    nat, N, env = _nat(), fused.env.N, fused.env
    rows = hi - lo
    o = {"actions": guarded(rows, (N,), torch.int8), "actions64": guarded(rows, (N,), torch.int64),
         "logp": guarded(rows, (), torch.float32), "value": guarded(rows, (), torch.float32),
         "logits": guarded(rows, (N, 5), torch.float32)}
    outs = dict(actions=o["actions"], actions64=o["actions64"], logp=o["logp"], value=o["value"], logits_out=o["logits"],
                num_envs=rows, greedy=greedy)
    if inputs is None:
        a = fused.args(env.obs_grid[lo:hi], env.action_mask[lo:hi], **outs)
        entry = nat.lib().mapf_cte_policy_act
    else:
        h, c, pa, pr, start = inputs
        o.update(h=guarded(rows, (64,), torch.float32), c=guarded(rows, (64,), torch.float32))
        a = fused.args(env.obs_grid[lo:hi], env.action_mask[lo:hi], (h[lo:hi], c[lo:hi]), pa[lo:hi], pr[lo:hi],
                       start[lo:hi], None, state_out=(o["h"], o["c"]), **outs)
        entry = nat.lib().mapf_cte_lstm_policy_act
    a.env_id_base, a.counter = lo, counter
    nat.check(entry(C.byref(a), None))
    return written_once(o, rows)


@pytest.mark.parametrize("kind", ["mlp", "lstm"])
@pytest.mark.parametrize("name,n,B", CTE_SHAPES)
def test_cte_kernels_past_the_first_trip(kind, name, n, B):
    from dl_reference_models_b200.policy_kernels import FusedCtePolicy, FusedCteRecurrentPolicy

    env = cte_env(name, n, B)
    if kind == "mlp":
        pol, inputs = cte_t.make_policy(env), None
        fused = FusedCtePolicy(pol, env, seed=7)
        with torch.no_grad():
            ref = cte_t.bf16_reference(pol, env.obs_grid, env.action_mask)
    else:
        pol, inputs = ctel_t.make_policy(env), ctel_t.random_inputs(env, seed=2)
        fused = FusedCteRecurrentPolicy(pol, env, seed=7)
        with torch.no_grad():
            h, c, pa, pr, start = inputs
            ref = ctel_t.bf16_reference(pol, env.obs_grid, env.action_mask, pa, pr, h, c, start)
    for greedy in (False, True):
        full = cte_launch(fused, inputs, 0, B, 9, greedy)
        for name_, i in (("logits", 0), ("value", 1), ("h", 2), ("c", 3))[:len(ref)]:
            assert_close(name_, full[name_], ref[i])
        assert torch.equal(full["actions64"], full["actions"].long())
        if greedy:
            assert torch.equal(full["actions"].long(), full["logits"].argmax(-1))
        ref_logp = torch.log_softmax(full["logits"].double(), -1).gather(-1, full["actions"].long().unsqueeze(-1)).squeeze(-1).sum(-1)
        assert float((full["logp"].double() - ref_logp).abs().max()) <= 1e-4
        for lo, hi in slices(B, 20001):   # 626 tiles: one trip at one block per SM
            assert_same_rows(full, cte_launch(fused, inputs, lo, hi, 9, greedy), lo, hi, 1)


# ---------------------------------------------------------------------------------------------------- evaluator kernels

def _episode_inputs(B, steps, g):
    """Staggered episode ends: env b ends at step end[b] (>= steps: it never ends), terminated, truncated or both."""
    end = torch.randint(0, steps + 2, (B,), generator=g, device="cuda")
    how = torch.randint(0, 3, (B,), generator=g, device="cuda")
    return [(((end == t) & (how != 1)).to(torch.uint8), ((end == t) & (how != 0)).to(torch.uint8)) for t in range(steps)]


def _state_buffers(B, per_env):
    """Guarded bookkeeping buffers (name -> (dtype, shape per env)) zeroed over the batch, the guard tail at its
    sentinel; `active` starts at 1 over the batch and its tail at 1 too, so a launch past the batch would act there."""
    bufs = {}
    for name, (dtype, shape) in per_env.items():
        t = guarded(B, shape, dtype)
        t[:B] = 0
        bufs[name] = t
    bufs["active"] = torch.ones(B + GUARD, dtype=torch.uint8, device="cuda")
    return bufs


def _tails_untouched(bufs, B):
    for name, t in bufs.items():
        tail = t[B:]
        assert bool((tail == 1).all()) if name == "active" else bool(_is_sentinel(tail).all()), f"{name}: written past the batch"


# mapf_eval_accumulate: 148 * 8 blocks x 8 warps x 32 / P envs, P = N rounded up to a power of two
EVAL_SHAPES = [
    (1, 700001),   # P = 1: 303 104 envs per trip; B % 32 = 1
    (3, 160003),   # P = 4: 75 776; B % 8 = 3
    (16, 40001),   # P = 16: 18 944; B odd
    (32, 20001),   # P = 32: 9 472
]


@pytest.mark.parametrize("n,B", EVAL_SHAPES)
def test_eval_accumulate_past_two_trips(n, B):
    nat = _nat()
    steps = 6
    g = torch.Generator(device="cuda").manual_seed(n)
    bufs = _state_buffers(B, {"episode_reward": (torch.float64, ()), "agent_reward": (torch.float64, (n,)),
                              "timesteps": (torch.int64, ()), "success": (torch.uint8, ()),
                              "last_info": (torch.int32, (16,))})
    # the word a step counts into was zeroed by the step before (the evaluator zeroes both first); the other one holds
    # a sentinel that step 0 must clear
    count = torch.tensor([0, 0xDEAD], dtype=torch.int32, device="cuda")
    ref = {k: v[:B].clone() for k, v in bufs.items()}
    ref["active"] = ref["active"].bool()
    for t, (term, trunc) in enumerate(_episode_inputs(B, steps, g)):
        reward = torch.randint(-6, 5, (B, n), generator=g, device="cuda").float() * 0.5
        info = torch.randint(-1000, 1000, (B, 16), generator=g, device="cuda", dtype=torch.int32)
        a = nat.MapfEvalArgs(num_envs=B, num_agents=n, step=t, reward=_p(reward), terminated=_p(term), truncated=_p(trunc),
                             info=_p(info), active=_p(bufs["active"]), episode_reward=_p(bufs["episode_reward"]),
                             agent_reward=_p(bufs["agent_reward"]), timesteps=_p(bufs["timesteps"]),
                             success=_p(bufs["success"]), last_info=_p(bufs["last_info"]), active_count=_p(count))
        nat.check(nat.lib().mapf_eval_accumulate(C.byref(a), None))
        act = ref["active"]
        ref["agent_reward"] += torch.where(act.unsqueeze(-1), reward.double(), 0.0)
        ref["episode_reward"] += torch.where(act, reward.double().sum(-1), 0.0)
        ref["timesteps"] += act.long()
        ref["last_info"][act] = info[act]
        done = (term | trunc).bool() & act
        ref["success"][done] = (term & (1 - trunc))[done]
        ref["active"] = act & ~done
        torch.cuda.synchronize()
        assert int(count[t & 1]) == int(ref["active"].sum()) and int(count[(t & 1) ^ 1]) == 0, t
    assert 0 < int(ref["active"].sum()) < B
    for k in ref:
        got = bufs[k][:B].bool() if k == "active" else bufs[k][:B]
        assert torch.equal(got, ref[k]), k
    _tails_untouched(bufs, B)


# mapf_cte_eval_accumulate: 148 * 8 blocks x 256 threads = 303 104 envs per trip, one thread per env; its heat-map
# launch (occupancy_launch) 1 184 blocks x 256 threads over the B * N agents
@pytest.mark.parametrize("n", [1, 3, 16, 32])
def test_cte_eval_accumulate_past_two_trips(n):
    nat = _nat()
    B, R, Cc, steps = 700001, 10, 20, 6
    g = torch.Generator(device="cuda").manual_seed(100 + n)
    bufs = _state_buffers(B, {"episode_reward": (torch.float64, ()), "timesteps": (torch.int64, ()),
                              "success": (torch.uint8, ()), "last_info": (torch.float64, (4,))})
    occ = torch.full((R * Cc + GUARD,), 0x7F7F7F7F7F7F7F7F, dtype=torch.int64, device="cuda")
    occ[:R * Cc] = 0
    # the word a step counts into was zeroed by the step before (the evaluator zeroes both first); the other one holds
    # a sentinel that step 0 must clear
    count = torch.tensor([0, 0xDEAD], dtype=torch.int32, device="cuda")
    ref = {k: v[:B].clone() for k, v in bufs.items()}
    ref["active"] = ref["active"].bool()
    ref_occ = torch.zeros(R * Cc, dtype=torch.int64, device="cuda")
    for t, (term, trunc) in enumerate(_episode_inputs(B, steps, g)):
        pos = torch.stack([torch.randint(-1, R + 1, (B, n), generator=g, device="cuda"),
                           torch.randint(-1, Cc + 1, (B, n), generator=g, device="cuda")], -1).to(torch.int16)
        reward = torch.randint(-6, 5, (B,), generator=g, device="cuda").double() * 0.5
        info = torch.randint(-1000, 1000, (B, 4), generator=g, device="cuda").double() * 0.5
        a = nat.MapfCteEvalArgs(num_envs=B, num_agents=n, rows=R, cols=Cc, step=t, positions=_p(pos), reward=_p(reward),
                                terminated=_p(term), truncated=_p(trunc), info=_p(info), active=_p(bufs["active"]),
                                episode_reward=_p(bufs["episode_reward"]), timesteps=_p(bufs["timesteps"]),
                                success=_p(bufs["success"]), last_info=_p(bufs["last_info"]), occupancy=_p(occ),
                                active_count=_p(count))
        nat.check(nat.lib().mapf_cte_eval_accumulate(C.byref(a), None))
        act = ref["active"]
        p = pos[act].reshape(-1, 2).long()
        inside = (p[:, 0] >= 0) & (p[:, 0] < R) & (p[:, 1] >= 0) & (p[:, 1] < Cc)
        ref_occ += torch.bincount(p[inside, 0] * Cc + p[inside, 1], minlength=R * Cc)
        ref["episode_reward"] += torch.where(act, reward, 0.0)
        ref["timesteps"] += act.long()
        ref["last_info"][act] = info[act]
        done = (term | trunc).bool() & act
        ref["success"][done] = (term & (1 - trunc))[done]
        ref["active"] = act & ~done
        torch.cuda.synchronize()
        assert int(count[t & 1]) == int(ref["active"].sum()) and int(count[(t & 1) ^ 1]) == 0, t
    assert 0 < int(ref["active"].sum()) < B
    for k in ref:
        got = bufs[k][:B].bool() if k == "active" else bufs[k][:B]
        assert torch.equal(got, ref[k]), k
    assert torch.equal(occ[:R * Cc], ref_occ) and bool((occ[R * Cc:] == 0x7F7F7F7F7F7F7F7F).all())
    _tails_untouched(bufs, B)


# ---------------------------------------------------------------------------------------------------------- replay tree

def ring(B, N, K, alpha, per_agent=False):
    """A CUDA ReplayBuffer of B envs x N agents x K slots on a stand-in env (the tree kernels read no observation)."""
    from dl_reference_models_b200 import dqn

    env = SimpleNamespace(B=B, N=N, V=1, device="cuda:0", include_blocking_pressure=False,
                          out={k: torch.zeros(1, dtype=torch.uint8, device="cuda") for k in CHANNELS})
    return dqn.ReplayBuffer(env, K, alpha=alpha, per_agent=per_agent)


def advance_both(buf, cpu, steps):
    """`steps` advances of the ring on the device and the CPU buffer, with a changing max priority."""
    for t in range(steps):
        for b in (buf, cpu):
            b.max_priority.fill_(float(t % 4 + 1))
            b.advance(t % buf.K, (t + 1) % buf.K)
    buf.filled = cpu.filled = min(steps, buf.K - 1)


def ulp_distance(a, b):
    """Largest distance in float32 ulps between two tensors of nonnegative floats."""
    return int((a.view(torch.int32).long() - b.view(torch.int32).long()).abs().max())


def check_leaves_and_tree(buf, cpu, alpha):
    """Leaves against the CPU buffer's, every internal node against _tree_reference of the device leaves; the
    comparisons run on the device (a 2^26-leaf tree is 1 GB)."""
    ulps = ulp_distance(buf.leaves(), cpu.leaves().to(buf.device))
    # alpha 0 and 1 are exact on both sides; otherwise device powf and torch pow may round differently
    assert ulps <= (0 if alpha in (0.0, 1.0) else 2), ulps
    assert int(torch.count_nonzero(buf._leaves)) == int(torch.count_nonzero(buf.leaves())), "a padding leaf is set"
    sums, mins = dqn_t._tree_reference(buf._leaves)
    assert torch.equal(buf.sums[1:], sums[1:].to(buf.device)), "an internal sum"
    assert torch.equal(buf.mins[1:], mins[1:].to(buf.device)), "an internal minimum"
    return ulps


# mapf_replay_advance: one block per (slot, agent, 1024-leaf chunk) of the B' = 2^ceil(log2 B) env leaves, then one
# block for the levels above min(B', 1024)
REPLAY_LAYOUTS = [   # (B, N, K, alpha, per_agent)
    (1, 1, 2, 1.0, False),
    (5, 3, 5, 0.6, True),
    (1, 16, 64, 0.0, False),
    (1024, 3, 2, 1.0, True),      # B' = 1 024: one chunk per (slot, agent)
    (1024, 16, 5, 0.6, False),
    (1025, 1, 64, 1.0, False),    # B' = 2 048: two chunks
    (1025, 3, 5, 0.0, True),
    (3000, 16, 2, 0.6, True),     # B' = 4 096: four chunks, 1 096 padding envs
    (3000, 3, 64, 1.0, False),
    (65536, 1, 5, 0.6, False),
    (65536, 3, 2, 0.0, True),
    (65536, 16, 64, 1.0, False),  # C3: 2^26 leaves, 64 chunks per (slot, agent)
]


@pytest.mark.parametrize("B,N,K,alpha,per_agent", REPLAY_LAYOUTS)
def test_replay_advance_across_the_wrap(B, N, K, alpha, per_agent):
    from dl_reference_models_b200 import dqn

    buf = ring(B, N, K, alpha, per_agent)
    cpu = dqn.ReplayBuffer(dqn_t._cpu_twin(buf).env, K, alpha=alpha, per_agent=per_agent)
    advance_both(buf, cpu, K + 3)
    ulps = check_leaves_and_tree(buf, cpu, alpha)
    print(f"advance B={B} N={N} K={K} alpha={alpha}: leaves within {ulps} ulp of the CPU buffer")
    # integer-valued leaves make every comparison of the descent exact; draws at 2^26 leaves are
    # test_replay_sample_at_c3_shared_and_per_agent's
    if alpha in (0.0, 1.0) and buf._leaves.numel() <= 1 << 22:
        u = torch.empty(4096, dtype=torch.float64, device="cuda")
        idx, w = buf.sample(4096, 0.4, uniforms_out=u)
        idx_c, w_c = cpu.sample(4096, 0.4, uniforms=u.cpu())
        assert torch.equal(idx.cpu(), idx_c)
        torch.testing.assert_close(w.cpu(), w_c, rtol=1e-6, atol=0)


# mapf_replay_update: one block of 1 024 threads striding over the M indices
UPDATE_RINGS = [   # (B, N, K, alpha, advances): the first leaves slots 11.. unfilled, the second wraps
    (3000, 3, 64, 0.6, 10),
    (1025, 16, 5, 1.0, 7),
]


@pytest.mark.parametrize("M", [1, 1023, 1024, 1025, 16384, 65536])
@pytest.mark.parametrize("B,N,K,alpha,advances", UPDATE_RINGS)
def test_replay_update_striding_over_the_indices(B, N, K, alpha, advances, M):
    from dl_reference_models_b200 import dqn

    buf = ring(B, N, K, alpha)
    cpu = dqn.ReplayBuffer(dqn_t._cpu_twin(buf).env, K, alpha=alpha)
    advance_both(buf, cpu, advances)
    BN, total = B * N, K * B * N
    clear = advances % K
    g = torch.Generator().manual_seed(M)
    idx = torch.randint(0, total, (M,), generator=g)
    td = torch.randint(1, 400, (M,), generator=g).float() * 0.125
    for d in (32, 1024):   # duplicates one stride of 32 and of 1 024 apart (one warp / one block trip), other TDs
        k = min(16, M - d)
        if k > 0:
            idx[d:d + k], td[d:d + k] = idx[:k], td[:k] + d / 64
    special = [-1, total, total - 1, clear * BN + 7, clear * BN + BN - 1]   # out of range, the last, the clear slot
    if advances < K - 1:
        special += [(K - 1) * BN + 5, (advances + 1) * BN]   # slots no advance has completed
    if M >= 64 + len(special):
        idx[64:64 + len(special)] = torch.tensor(special)
    buf.update_priorities(idx.cuda(), td.cuda())
    cpu.update_priorities(idx, td)
    ulps = check_leaves_and_tree(buf, cpu, alpha)
    print(f"update M={M} alpha={alpha}: leaves within {ulps} ulp of the CPU buffer")
    assert float(buf.max_priority) == float(cpu.max_priority)
    assert float(cpu.max_priority) > 4.0 or M == 1


def test_replay_sample_at_c3_shared_and_per_agent():
    """2^26 leaves with integer priorities written straight into the tree (one empty agent, the clear slot at 0), the
    device draws against the CPU buffer's f64 cumsum search given the kernel's own uniforms.  This caught the CPU
    buffer gathering one whole cumulative row per draw (2^20 x 2^26 f64 here); it now searches each row once."""
    B, N, K, empty = 65536, 16, 64, 5
    buf = ring(B, N, K, 1.0)
    g = torch.Generator(device="cuda").manual_seed(3)
    leaves = buf._leaves.view(N, K, B)   # no padding at C3
    leaves.copy_(torch.randint(1, 4, (N, K, B), generator=g, device="cuda"))
    leaves[:, 9] = 0.0        # the clear slot
    leaves[empty] = 0.0       # an agent whose subtree holds nothing
    sums, mins = dqn_t._tree_reference(buf._leaves)
    buf.sums.copy_(sums)
    buf.mins.copy_(mins)
    del sums, mins
    buf.filled = K - 1
    cpu = dqn_t._cpu_twin(buf)
    cpu.actions = cpu.rewards = None   # 335 MB of host memory the draws never read
    M = 1 << 20
    for per_agent in (False, True):
        buf.per_agent = cpu.per_agent = per_agent
        u = torch.empty(M, dtype=torch.float64, device="cuda")
        idx, w = buf.sample(M, 0.4, uniforms_out=u)
        idx, w = idx.cpu(), w.cpu()
        idx_c, w_c = cpu.sample(M, 0.4, uniforms=u.cpu())
        keep = torch.arange(M) % N != empty if per_agent else torch.ones(M, dtype=torch.bool)
        assert torch.equal(idx[keep], idx_c[keep])
        torch.testing.assert_close(w[keep], w_c[keep], rtol=1e-6, atol=0)
        assert not bool((idx[keep] % N == empty).any())
        if per_agent:   # the empty agent's draws: index -1, weight 0 (mapf_replay_sample's contract)
            assert bool((idx[~keep] == -1).all()) and bool((w[~keep] == 0).all())
