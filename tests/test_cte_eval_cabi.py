"""CPU-side checks of evaluating CTE policies (no GPU): the ctypes structures of both greedy-capable CTE policy entry
points and of mapf_cte_eval_accumulate have the header's layout (the fields the CTE policy structures had before
`greedy` was appended keep their offsets), the entry points refuse a greedy flag other than 0 / 1 and null or empty
bookkeeping arguments before any device work, and evaluate() refuses mismatched execution modes, modules and shapes
before it builds an env."""
import ctypes as C
import shutil
import subprocess
from pathlib import Path

import pytest

from dl_reference_models_b200 import _native as nat

REPO = Path(__file__).resolve().parents[1]
STRUCTS = [("mapf_cte_policy_args", nat.MapfCtePolicyArgs), ("mapf_cte_lstm_policy_args", nat.MapfCteLstmPolicyArgs),
           ("mapf_cte_eval_args", nat.MapfCteEvalArgs)]


@pytest.mark.skipif(shutil.which("gcc") is None, reason="needs gcc")
@pytest.mark.parametrize("cname, cls", STRUCTS)
def test_ctypes_structure_matches_the_header_layout(tmp_path, cname, cls):
    fields = [name for name, _ in cls._fields_]
    src = tmp_path / "probe.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "mapf_b200.h"\nint main(void) {\n'
                   f'    printf("%zu\\n", sizeof({cname}));\n'
                   + "".join(f'    printf("%zu\\n", offsetof({cname}, {f}));\n' for f in fields)
                   + "    return 0;\n}\n")
    exe = tmp_path / "probe"
    subprocess.run(["gcc", "-std=c99", "-I", str(REPO / "include"), "-o", str(exe), str(src)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    want = [C.sizeof(cls)] + [getattr(cls, f).offset for f in fields]
    assert got == want


def test_greedy_is_appended_and_the_existing_offsets_are_unchanged():
    # the layouts before `greedy`: four int32, three 64-bit words, then one pointer per field
    head = {"num_envs": 0, "num_agents": 4, "cells": 8, "reserved": 12, "seed": 16, "counter": 24, "env_id_base": 32}
    mlp = ("obs_grid", "action_mask", "weights", "actions", "actions64", "logp", "value", "logits_out")
    lstm = ("obs_grid", "action_mask", "prev_terminated", "prev_truncated", "prev_action", "prev_reward", "h_in", "c_in",
            "h_out", "c_out", "trunk", "weights", "actions", "actions64", "logp", "value", "logits_out")
    for cls, ptrs in ((nat.MapfCtePolicyArgs, mlp), (nat.MapfCteLstmPolicyArgs, lstm)):
        want = dict(head, **{k: 40 + 8 * i for i, k in enumerate(ptrs)})
        assert {k: getattr(cls, k).offset for k in want} == want, cls
        assert cls.greedy.offset == 40 + 8 * len(ptrs)
        assert [n for n, _ in cls._fields_][-1] == "greedy"
        assert cls().greedy == 0   # every caller that does not set it gets draw mode


def _filled(cls, **kw):
    a = cls(**kw)
    fake = C.c_void_p(16)
    for name, typ in cls._fields_:
        if typ is C.c_void_p:
            setattr(a, name, fake)
    return a


@pytest.mark.parametrize("greedy", [2, -1, 7])
def test_cte_policy_entry_points_refuse_other_greedy_values(greedy):
    L = nat.lib()
    a = _filled(nat.MapfCtePolicyArgs, num_envs=4, num_agents=2, cells=200, greedy=greedy)
    assert L.mapf_cte_policy_act(C.byref(a), None) == nat.ERR_INVALID_ARG
    assert b"greedy" in L.mapf_last_error()
    b = _filled(nat.MapfCteLstmPolicyArgs, num_envs=4, num_agents=2, cells=200, greedy=greedy)
    assert L.mapf_cte_lstm_policy_act(C.byref(b), None) == nat.ERR_INVALID_ARG
    assert b"greedy" in L.mapf_last_error()


def test_reserved_is_still_checked_with_greedy_set():
    L = nat.lib()
    a = _filled(nat.MapfCtePolicyArgs, num_envs=4, num_agents=2, cells=200, greedy=1, reserved=1)
    assert L.mapf_cte_policy_act(C.byref(a), None) == nat.ERR_INVALID_ARG
    assert b"reserved" in L.mapf_last_error()
    b = _filled(nat.MapfCteLstmPolicyArgs, num_envs=4, num_agents=2, cells=200, greedy=1, reserved=1)
    assert L.mapf_cte_lstm_policy_act(C.byref(b), None) == nat.ERR_INVALID_ARG
    assert b"reserved" in L.mapf_last_error()


def test_cte_eval_accumulate_refuses_null_or_empty_arguments():
    L = nat.lib()
    dims = dict(num_envs=8, num_agents=4, rows=10, cols=20)
    assert L.mapf_cte_eval_accumulate(None, None) == nat.ERR_INVALID_ARG
    for k in dims:
        for v in (0, -3):
            a = _filled(nat.MapfCteEvalArgs, **dict(dims, **{k: v}))
            assert L.mapf_cte_eval_accumulate(C.byref(a), None) == nat.ERR_INVALID_ARG, (k, v)
    for name, typ in nat.MapfCteEvalArgs._fields_:
        if typ is C.c_void_p:
            a = _filled(nat.MapfCteEvalArgs, **dims)
            setattr(a, name, None)
            assert L.mapf_cte_eval_accumulate(C.byref(a), None) == nat.ERR_INVALID_ARG, name
            assert b"cte eval" in L.mapf_last_error()
    a = _filled(nat.MapfCteEvalArgs, **dict(dims, num_agents=nat.MAX_AGENTS + 1))
    assert L.mapf_cte_eval_accumulate(C.byref(a), None) == nat.ERR_UNSUPPORTED


def _cfg(**kw):
    from dl_reference_models_b200 import maps

    return dict({"env_name": "ReferenceModel-2-1", "grid": maps.get_grid("ReferenceModel-2-1"), "num_agents": 4,
                 "steps_per_episode": 20, "seed": 3}, **kw)   # 10 x 20 = 200 cells


@pytest.mark.parametrize("mode", ["CTDE", "DTE", "ctde"])
@pytest.mark.parametrize("kind", ["mlp", "lstm"])
def test_a_centralised_module_with_another_execution_mode_is_refused(mode, kind):
    from dl_reference_models_b200.cte_rollout import CteActionMaskPolicy, CteRecurrentPolicy
    from dl_reference_models_b200.evaluate import evaluate

    policy = (CteActionMaskPolicy if kind == "mlp" else CteRecurrentPolicy)(200, 4)
    with pytest.raises(ValueError, match=f"centralised.*{mode}"):
        evaluate(_cfg(training_execution_mode=mode), 8, policy=policy)


@pytest.mark.parametrize("kind", ["mlp", "lstm", "per_agent_mlp", "per_agent_lstm"])
def test_a_multi_agent_module_with_the_cte_mode_is_refused(kind):
    from dl_reference_models_b200.evaluate import evaluate
    from dl_reference_models_b200.recurrent import PerAgentRecurrentPolicy, RecurrentActionMaskPolicy
    from dl_reference_models_b200.rollout import ActionMaskPolicy, PerAgentActionMaskPolicy

    policy = {"mlp": lambda: ActionMaskPolicy(11), "lstm": lambda: RecurrentActionMaskPolicy(11),
              "per_agent_mlp": lambda: PerAgentActionMaskPolicy(4, 11),
              "per_agent_lstm": lambda: PerAgentRecurrentPolicy(4, 11)}[kind]()
    with pytest.raises(ValueError, match="multi-agent view.*CTE"):
        evaluate(_cfg(training_execution_mode="CTE"), 8, policy=policy)


@pytest.mark.parametrize("kind", ["mlp", "lstm"])
def test_centralised_modules_of_another_shape_or_device_are_refused(kind):
    from dl_reference_models_b200.cte_rollout import CteActionMaskPolicy, CteRecurrentPolicy
    from dl_reference_models_b200.evaluate import evaluate

    cls = CteActionMaskPolicy if kind == "mlp" else CteRecurrentPolicy
    with pytest.raises(ValueError, match="199 grid cells.*10x20 = 200"):
        evaluate(_cfg(), 8, policy=cls(199, 4))
    with pytest.raises(ValueError, match="num_agents = 5.*num_agents = 4"):
        evaluate(_cfg(), 8, policy=cls(200, 5))
    with pytest.raises(ValueError, match="cpu"):   # the parameters stay on the CPU, the evaluation runs on cuda:0
        evaluate(_cfg(training_execution_mode="CTE"), 8, policy=cls(200, 4))
    with pytest.raises(ValueError, match="cells"):   # the map named by env_name when no grid is inline
        evaluate({"env_name": "ReferenceModel-3-1", "num_agents": 4}, 8, policy=cls(200, 4))


def test_view_selection():
    from dl_reference_models_b200.cte_rollout import CteActionMaskPolicy, CteRecurrentPolicy
    from dl_reference_models_b200.evaluate import _cte_view
    from dl_reference_models_b200.rollout import ActionMaskPolicy

    for pol in ("random", "masked", lambda env, out: None):
        assert _cte_view({"training_execution_mode": "CTE"}, pol)
        assert not _cte_view({"training_execution_mode": "CTDE"}, pol)
        assert not _cte_view({}, pol)
    for pol in (CteActionMaskPolicy(200, 4), CteRecurrentPolicy(200, 4)):
        assert _cte_view({}, pol) and _cte_view({"training_execution_mode": "CTE"}, pol)
    assert not _cte_view({}, ActionMaskPolicy(11)) and not _cte_view({"training_execution_mode": "DTE"}, ActionMaskPolicy(11))
