"""CPU-side checks of the evaluator's C ABI (no GPU): the ctypes structures of the greedy-capable MLP policy and of the
bookkeeping kernel have the header's layout, both policy entry points refuse a greedy flag other than 0 / 1, and
mapf_eval_accumulate refuses null or empty arguments before any device work."""
import ctypes as C
import shutil
import subprocess
from pathlib import Path

import pytest

from dl_reference_models_b200 import _native as nat

REPO = Path(__file__).resolve().parents[1]


@pytest.mark.skipif(shutil.which("gcc") is None, reason="needs gcc")
@pytest.mark.parametrize("cname, cls", [("mapf_policy_args", nat.MapfPolicyArgs), ("mapf_eval_args", nat.MapfEvalArgs)])
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


def test_greedy_sits_where_reserved_was():
    # the field that used to be `reserved`: same offset, same struct sizes
    assert nat.MapfPolicyArgs.greedy.offset == nat.MapfPolicyArgs.no_masking.offset + 4 == 20
    assert nat.MapfLstmPolicyArgs.greedy.offset == nat.MapfLstmPolicyArgs.no_masking.offset + 4 == 20
    assert nat.MapfPolicyArgs.seed.offset == nat.MapfLstmPolicyArgs.seed.offset == 24


def _filled(cls, **kw):
    a = cls(**kw)
    fake = C.c_void_p(16)
    for name, typ in cls._fields_:
        if typ is C.c_void_p:
            setattr(a, name, fake)
    return a


@pytest.mark.parametrize("greedy", [2, -1, 7])
def test_act_entry_points_refuse_other_greedy_values(greedy):
    L = nat.lib()
    a = _filled(nat.MapfPolicyArgs, num_envs=4, num_agents=2, v2=25, feature_dim=28, greedy=greedy)
    assert L.mapf_policy_act(C.byref(a), None) == nat.ERR_INVALID_ARG
    assert b"greedy" in L.mapf_last_error()
    b = _filled(nat.MapfLstmPolicyArgs, num_envs=4, num_agents=2, v2=25, feature_dim=28, greedy=greedy)
    assert L.mapf_lstm_policy_act(C.byref(b), None) == nat.ERR_INVALID_ARG
    assert b"greedy" in L.mapf_last_error()


def test_eval_accumulate_refuses_null_or_empty_arguments():
    L = nat.lib()
    assert L.mapf_eval_accumulate(None, None) == nat.ERR_INVALID_ARG
    for k in ("num_envs", "num_agents"):
        for v in (0, -3):
            a = _filled(nat.MapfEvalArgs, num_envs=8, num_agents=4)
            setattr(a, k, v)
            assert L.mapf_eval_accumulate(C.byref(a), None) == nat.ERR_INVALID_ARG, (k, v)
    for name, typ in nat.MapfEvalArgs._fields_:
        if typ is C.c_void_p:
            a = _filled(nat.MapfEvalArgs, num_envs=8, num_agents=4)
            setattr(a, name, None)
            assert L.mapf_eval_accumulate(C.byref(a), None) == nat.ERR_INVALID_ARG, name
    a = _filled(nat.MapfEvalArgs, num_envs=8, num_agents=nat.MAX_AGENTS + 1)
    assert L.mapf_eval_accumulate(C.byref(a), None) == nat.ERR_UNSUPPORTED


def test_policy_shape_predicates():
    from types import SimpleNamespace

    from dl_reference_models_b200.policy_kernels import FusedPolicy, FusedRecurrentPolicy
    from dl_reference_models_b200.recurrent import RecurrentActionMaskPolicy
    from dl_reference_models_b200.rollout import ActionMaskPolicy

    env = SimpleNamespace(V=5, include_blocking_pressure=True)   # F = 28
    assert FusedPolicy.matches(ActionMaskPolicy(28), env)
    assert FusedRecurrentPolicy.matches(RecurrentActionMaskPolicy(28), env)
    for kw in (dict(feature_dim=27), dict(hiddens=(32, 32)), dict(hiddens=(64,)), dict(hiddens=()), dict(num_actions=4)):
        kw = dict(dict(feature_dim=28), **kw)
        assert not FusedPolicy.matches(ActionMaskPolicy(**kw), env), kw
    for kw in (dict(cell=32), dict(hiddens=(64, 32)), dict(use_prev_reward=False)):
        assert not FusedRecurrentPolicy.matches(RecurrentActionMaskPolicy(28, **kw), env), kw
    assert not FusedPolicy.matches(ActionMaskPolicy(28), SimpleNamespace(V=5, include_blocking_pressure=False))
