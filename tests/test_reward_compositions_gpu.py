"""GPU tier (B200): reward-mixin class compositions in k_step.

About two dozen compositions (the registered ids, each mixin alone, the full list in three orders, NaughtyBots first,
in the middle and last, DontDrive + KeepMoving) on both presets, goal scoring off and on, discrete and continuous
actions.  One K = 8 launch with auto-reset over N envs injected with the states of test_reward_compositions.py
(contact-rich golden states, robots on the goal triangles' edges and Div0 corners, zero and undone thrusts):
  * the first step of every env must equal the host build of the same source (tests/emul, GPU sin/cos routine) bit for
    bit: both are IEEE operations in the same order, compiled with --fmad=false;
  * all K rows of the first M envs must match the oracle replaying them, within the parity tolerance, up to the env's
    first done row; envs whose trajectories part after a last-bit contact difference are counted and bounded as in
    test_parity_gpu.py::test_gpu_fused_multistep_matches_oracle.
"""
import functools

import numpy as np
import pytest

from golden_util import STATE_KEYS
from parity_util import close
from roborugby_b200.constants import reward_config_from_mixins
from test_reward_compositions import BASEDESTR, CHASE, DONTDRIVE, KEEPMOVING, NAMES, NAUGHTY, PUSHNEG, PUSHPOS, _state_set

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

K = 8
N = 4096
ALL = [KEEPMOVING, DONTDRIVE, BASEDESTR, PUSHNEG, PUSHPOS, CHASE]
COMPS = ([[PUSHPOS, CHASE, NAUGHTY], [CHASE], []]                         # the registered ids' compositions
         + [[n] for n in NAMES]                                            # each mixin alone
         + [ALL + [NAUGHTY], [NAUGHTY] + ALL, ALL[::-1] + [NAUGHTY],       # the full list in three orders ...
            ALL[3:] + ALL[:3], ALL[::-1]]                                  # ... and without NaughtyBots
         + [[NAUGHTY, CHASE, PUSHPOS], [CHASE, NAUGHTY, PUSHPOS, DONTDRIVE], [KEEPMOVING, PUSHNEG, NAUGHTY]]
         + [[DONTDRIVE, KEEPMOVING], [KEEPMOVING, DONTDRIVE], [KEEPMOVING, DONTDRIVE, NAUGHTY, CHASE]])


@functools.lru_cache(maxsize=None)
def _pool(preset):
    """N states: the rich state set of the CPU tests, tiled; step counters kept small so no env ends by time."""
    recs = _state_set(preset, True)
    idx = np.arange(N) % len(recs)
    st = {k: np.stack([np.asarray(recs[i][0][k]) for i in idx]) for k in STATE_KEYS}
    st["step"] = np.minimum(st["step"], 100).astype(np.int32)
    return st


def _actions(preset, discrete, n, seed):
    R = 4 if preset == "GAME" else 1
    g = np.random.default_rng(seed)
    if discrete:
        return g.integers(0, 8, (K, n, R)).astype(np.uint8)
    return g.choice(np.array([-1.0, 0.0, 0.0, 0.0, 1.0], np.float32), (K, n, 2 * R))   # mostly standing still


def _run(oracle, preset, goals, discrete, mixins, n=N, m=32):
    from emul import emul
    from emul.emul import EmulBatch
    from roborugby_b200.vec_env import RoboRugbyVecEnv
    mask, order = reward_config_from_mixins(mixins)
    env_id = "RoboRugbySimpleDuel-v2" if discrete else "RoboRugby-v0"
    env = RoboRugbyVecEnv(env_id, n, preset=preset, device="cuda:0", time_limit=False, auto_reset=True,
                          out_dtype=torch.float64, reward_mask=mask, reward_order=order, goal_scoring=goals, seed=11)
    pool = _pool(preset) if n == N else {k: np.resize(v, (n,) + v.shape[1:]) for k, v in _pool(preset).items()}
    env.set_state(pool)
    acts = _actions(preset, discrete, n, seed=mask * 131 + order % 977 + 7 * goals)
    _, _, rew, done = env.step_k(torch.as_tensor(acts).cuda(), K)
    rew, done = rew.cpu().numpy(), done.cpu().numpy()

    # the host build, first row of every env, bit for bit
    emul.use_libm_sincos(False)
    hb = EmulBatch(env.cfg, n, env.num_robots, env.num_balls, env.obs_dim)
    for i in range(n):
        hb.set_state(i, {k: pool[k][i] for k in STATE_KEYS})
    h = hb.launch(acts[:1].astype(np.float64))
    diff = np.nonzero(np.any(h["rew"][0] != rew[0], axis=1) | (h["done"][0] != done[0]))[0]
    assert diff.size == 0, [(int(i), h["rew"][0, i].tolist(), rew[0, i].tolist()) for i in diff[:4]]

    # the oracle, every row of the first m envs
    ocfg = oracle.default_config(preset, env_id)
    ocfg.reward_mask, ocfg.reward_order, ocfg.goal_scoring = mask, order, int(goals)
    o = oracle.OracleEnv(cfg=ocfg)
    diverged = rows = 0
    for i in range(m):
        o.set_state({k: pool[k][i] for k in STATE_KEYS})
        for s in range(K):
            w = o.step(acts[s, i].astype(np.float64))
            if w["err"]:
                assert done[s, i] == 1, (i, s)
                break
            rows += 1
            if not close(rew[s, i], w["rew"]) or int(done[s, i]) != w["done"]:
                diverged += 1
                break
            if w["done"]:
                break
    return diverged, rows


@pytest.mark.parametrize("discrete", [True, False], ids=["discrete", "continuous"])
@pytest.mark.parametrize("goals", [False, True], ids=["head", "goals"])
@pytest.mark.parametrize("preset", ["GAME", "TRAIN"])
def test_gpu_compositions_match_host_build_and_oracle(oracle, preset, goals, discrete):
    oracle.scratch_mode(1)
    try:
        diverged = rows = 0
        for mixins in COMPS:
            d, r = _run(oracle, preset, goals, discrete, mixins)
            diverged += d; rows += r
        print(f"{preset} goals={goals} discrete={discrete}: {len(COMPS)} compositions x {N} envs bit-identical to the "
              f"host build; {rows} oracle rows compared, {diverged} trajectories diverged")
        assert diverged <= max(1, 32 * len(COMPS) // 200), diverged
    finally:
        oracle.scratch_mode(0)


@pytest.mark.parametrize("mixins", [ALL + [NAUGHTY], ALL[::-1], [DONTDRIVE, KEEPMOVING]], ids=["full", "reversed", "dd-km"])
def test_gpu_compositions_on_the_448_thread_kernel(oracle, mixins):
    """GAME with goal scoring and a batch above 384 threads x #SM selects the 448-thread k_step variant."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    oracle.scratch_mode(1)
    try:
        d, _ = _run(oracle, "GAME", True, False, mixins, n=384 * sms + 1, m=16)
        assert d <= 1
    finally:
        oracle.scratch_mode(0)
