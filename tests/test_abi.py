"""The C-ABI library loads on a CPU-only box and exports every symbol include/rr_b200.h declares."""
import ctypes
import os
import re

import pytest

from conftest import ROOT


def _declared_symbols():
    src = open(os.path.join(ROOT, "include", "rr_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(rr_[a-z0-9_]+)\s*\(", src)))


def test_header_declares_expected_surface():
    syms = _declared_symbols()
    for s in ("rr_create", "rr_destroy", "rr_reset", "rr_step", "rr_step_host", "rr_observe", "rr_get_state",
              "rr_set_state", "rr_get_stats", "rr_error_mask", "rr_last_error", "rr_default_config"):
        assert s in syms


def test_library_exports_every_declared_symbol():
    from roborugby_b200 import _lib
    assert os.path.exists(_lib.LIB_PATH), "build first: python -c 'import __graft_entry__ as g; g.build()'"
    lib = ctypes.CDLL(_lib.LIB_PATH)
    missing = [s for s in _declared_symbols() if not hasattr(lib, s)]
    assert not missing, missing
    # the ctypes table covers the whole header, nothing more
    assert sorted(_lib.SIGNATURES) == _declared_symbols()


def test_default_config_env_ids():
    from roborugby_b200 import _lib
    c = _lib.default_config(_lib.PRESET_GAME, "RoboRugbySimpleDuel-v2")
    assert (c.reward_mask, c.observer, c.discrete) == (7, _lib.OBS_BASIC_LIDAR, 1)
    c = _lib.default_config(_lib.PRESET_TRAIN, "RoboRugbySimpleDuel-v3")
    assert (c.reward_mask, c.observer, c.discrete) == (7, _lib.OBS_LIDAR6_V2, 1)
    c = _lib.default_config(_lib.PRESET_GAME, "RoboRugbySimple-v0")
    assert (c.reward_mask, c.observer) == (1, _lib.OBS_BASIC_LIDAR)
    c = _lib.default_config(_lib.PRESET_GAME, "RoboRugby-v0")
    assert (c.reward_mask, c.observer, c.discrete) == (0, _lib.OBS_NONE, 0)
    with pytest.raises(_lib.RRError):
        _lib.default_config(_lib.PRESET_GAME, "NoSuchEnv-v0")


def test_create_fails_loudly_without_gpu():
    """No CPU fallback: on a box without a CUDA device rr_create must fail, not degrade."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from roborugby_b200 import _lib
    cfg = _lib.default_config(_lib.PRESET_TRAIN, "RoboRugbySimpleDuel-v2")
    h = ctypes.c_void_p()
    rc = _lib.load().rr_create(ctypes.byref(cfg), 8, 0, ctypes.byref(h))
    assert rc != 0 and not h.value
    assert b"no usable CUDA device" in _lib.load().rr_last_error()
    import roborugby_b200
    with pytest.raises(RuntimeError):
        roborugby_b200.RoboRugbyVecEnv("RoboRugbySimpleDuel-v2", 8)


def test_reward_mixin_composition_to_config():
    """Host logic: class-definition order of RR_ScoreKeepers.py mixins -> (reward_mask, reward_order).  The bodies of
    on_step_end run in reverse MRO order and NaughtyBots ends the chain (it does not call super())."""
    from roborugby_b200.constants import reward_config_from_mixins as f
    # the registered ids' own composition (RR_Environments.py:11-37): Naughty, Chase, PushPos
    assert f(["PushPosBallsToGoal", "ChasePosBall", "NaughtyBots"]) == (7, 0x213)
    # mixins after NaughtyBots keep their mask bit (on_step_begin still runs) but never execute on_step_end
    assert f(["DontDriveInGoals", "ChasePosBall", "NaughtyBots", "KeepMovingGuys"]) == (8 | 1 | 4 | 16, 0x413)
    assert f(["KeepMovingGuys"]) == (16, 0x5)
    import pytest
    with pytest.raises(ValueError):
        f(["NoSuchMixin"])
    with pytest.raises(ValueError):   # "duplicate base class" in Python
        f(["ChasePosBall", "ChasePosBall"])


def test_bench_reference_arm_prints_the_contract_line():
    """bench.py --impl reference (the CPU arm the driver runs next to ours) needs no GPU: one JSON line with the
    contract's keys, timed on the C oracle port."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--preset", "TRAIN"], capture_output=True, text=True, timeout=300, check=True)
    d = json.loads(out.stdout.strip().splitlines()[-1])
    assert d["impl"] == "reference" and d["metric"] == "env_steps_per_sec" and d["unit"] == "env-steps/s"
    assert d["value"] > 0 and d["higher_is_better"] is True and d["gpu_launches"] == 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["env_id"] == "RoboRugbySimpleDuel-v2" and d["config"]["preset"] == "TRAIN"
