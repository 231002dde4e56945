"""CPU-side checks of the fused LSTM-64 policy's C ABI (no GPU): the ctypes structure has the header's layout, the
weight-block size rejects unsupported feature widths, and the Python wrapper refuses non-reference modules before it
touches a device."""
import ctypes as C
import shutil
import subprocess
from pathlib import Path
from types import SimpleNamespace

import pytest

from dl_reference_models_b200 import _native as nat

REPO = Path(__file__).resolve().parents[1]
FIELDS = [name for name, _ in nat.MapfLstmPolicyArgs._fields_]


@pytest.mark.skipif(shutil.which("gcc") is None, reason="needs gcc")
def test_ctypes_structure_matches_the_header_layout(tmp_path):
    src = tmp_path / "probe.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "mapf_b200.h"\nint main(void) {\n'
                   '    printf("%zu\\n", sizeof(mapf_lstm_policy_args));\n'
                   + "".join(f'    printf("%zu\\n", offsetof(mapf_lstm_policy_args, {f}));\n' for f in FIELDS)
                   + "    return 0;\n}\n")
    exe = tmp_path / "probe"
    subprocess.run(["gcc", "-std=c99", "-I", str(REPO / "include"), "-o", str(exe), str(src)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    want = [C.sizeof(nat.MapfLstmPolicyArgs)] + [getattr(nat.MapfLstmPolicyArgs, f).offset for f in FIELDS]
    assert got == want


def test_weight_block_size_rejects_unsupported_feature_widths():
    L = nat.lib()
    for bad in (0, 65, -1):
        assert L.mapf_lstm_policy_weights_nbytes(bad) == nat.ERR_UNSUPPORTED, bad
    small, large = L.mapf_lstm_policy_weights_nbytes(28), L.mapf_lstm_policy_weights_nbytes(52)
    assert 0 < small < large and small % 16 == 0 and large % 16 == 0
    assert L.mapf_lstm_policy_weights_nbytes(32) == small and L.mapf_lstm_policy_weights_nbytes(64) == large


def test_pack_and_act_validate_their_arguments_before_any_device_work():
    L = nat.lib()
    assert L.mapf_lstm_policy_pack_weights(28, *([None] * 13)) == nat.ERR_INVALID_ARG
    assert L.mapf_lstm_policy_pack_weights(65, *([None] * 13)) == nat.ERR_UNSUPPORTED
    assert L.mapf_lstm_policy_act(None, None) == nat.ERR_INVALID_ARG
    a = nat.MapfLstmPolicyArgs(num_envs=4, num_agents=2, v2=25, feature_dim=28)   # 28 needs blocking_prev
    assert L.mapf_lstm_policy_act(C.byref(a), None) == nat.ERR_UNSUPPORTED
    a.feature_dim = 27
    assert L.mapf_lstm_policy_act(C.byref(a), None) == nat.ERR_INVALID_ARG       # no channels / weights
    fake = C.c_void_p(16)
    for k in ("local_obs", "goal_delta", "weights"):
        setattr(a, k, fake)
    assert L.mapf_lstm_policy_act(C.byref(a), None) == nat.ERR_INVALID_ARG       # no prev action / reward / state
    for k in ("prev_action", "prev_reward", "h_in", "c_in", "h_out"):
        setattr(a, k, fake)
    assert L.mapf_lstm_policy_act(C.byref(a), None) == nat.ERR_INVALID_ARG       # h_out without c_out
    assert b"h_out and c_out" in L.mapf_last_error()


def _stub_env(V=5, bp=True):
    # enough of BatchedMapfEnv for the shape checks; device work would fail on the missing attributes
    return SimpleNamespace(V=V, include_blocking_pressure=bp)


@pytest.mark.parametrize("kwargs", [dict(hiddens=(64,)), dict(hiddens=(64, 32)), dict(hiddens=(128, 64)), dict(cell=32),
                                    dict(use_prev_action=False), dict(use_prev_reward=False), dict(num_actions=4),
                                    dict(feature_dim=27)])
def test_fused_recurrent_policy_refuses_non_reference_modules(kwargs):
    from dl_reference_models_b200.policy_kernels import FusedRecurrentPolicy
    from dl_reference_models_b200.recurrent import RecurrentActionMaskPolicy

    kw = dict(feature_dim=28)
    kw.update(kwargs)
    with pytest.raises(ValueError, match="reference's policy"):
        FusedRecurrentPolicy(RecurrentActionMaskPolicy(**kw), _stub_env())
