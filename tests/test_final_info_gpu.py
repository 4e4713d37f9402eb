"""GPU tier (B200): rr_step_info, i.e. the terminal observation of every done row and the RR_ROW_* flags of every row
(k_step<L, OutT, true>).

* BASELINE configuration (65 536 GAME envs, K = 32, fp32, bench.py's phase desynchronisation, so resets fall inside the
  launch), through the sub-batch pipeline (384-thread kernel) and as one launch (448-thread kernel): sampled envs are
  replayed by the oracle; every done row's final observation must be within one fp32 ulp of the cast oracle value and
  every flag exact; diverged envs are counted and bounded as in test_parity_gpu.py.  The same batch stepped through
  rr_step from the same state must give bit-identical obs, rew, done and final state, and the same statistics counts.
* TRAIN over more than T steps with the time limit: truncated exactly at the rows where the step counter reaches T.
* Goal scoring (including the 448-thread goal-scoring kernel), fp64 outputs and an env without observations: done and
  flags of the first row of every env equal the host build's (tests/emul) bit for bit, final observations within the
  parity bar.
* Canaries in rows with done == 0; misaligned final buffers refused with nothing launched; the Python layer."""
import numpy as np
import pytest

from golden_util import STATE_KEYS
from parity_util import close

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

ROW_TRUNCATED, ROW_RAISED = 1, 2
V0, V2 = "RoboRugby-v0", "RoboRugbySimpleDuel-v2"
CANARY32 = -7777.25
FLAGS_CANARY = 0x55


def _venv(env_id, n, preset, **kw):
    from roborugby_b200.vec_env import RoboRugbyVecEnv
    kw.setdefault("time_limit", True)
    kw.setdefault("auto_reset", True)
    kw.setdefault("out_dtype", torch.float32)
    kw.setdefault("strict_reset", True)
    return RoboRugbyVecEnv(env_id, n, preset=preset, device="cuda:0", **kw)


def _step_info(env, acts, K, final=True, flags=True, canary=CANARY32):
    """One rr_step_info call with fresh buffers; final buffers and flags pre-filled with canaries."""
    from roborugby_b200 import _lib
    N, D = env.num_envs, max(env.obs_dim, 1)
    dt = env.out_dtype
    mk = lambda *s, d=dt: torch.empty(*s, dtype=d, device="cuda")
    oh, og, rew, done = mk(K, N, D), mk(K, N, D), mk(K, N, 2), mk(K, N, d=torch.uint8)
    fh = torch.full((K, N, D), canary, dtype=dt, device="cuda") if final else None
    fg = torch.full((K, N, D), canary, dtype=dt, device="cuda") if final else None
    fl = torch.full((K, N), FLAGS_CANARY, dtype=torch.uint8, device="cuda") if flags else None
    p = lambda t: None if t is None else t.data_ptr()
    has_obs = env.obs_dim > 0
    _lib.check(env.lib.rr_step_info(env._h, acts.data_ptr(), acts.shape[2], K, p(oh) if has_obs else None,
                                    p(og) if has_obs else None, p(rew), p(done), p(fh), p(fg), p(fl), env._stream()))
    env.join()
    torch.cuda.synchronize()
    c = lambda t: None if t is None else t.cpu().numpy()
    return dict(obs_h=c(oh)[..., :env.obs_dim], obs_g=c(og)[..., :env.obs_dim], rew=c(rew), done=c(done),
                final_h=None if fh is None else c(fh)[..., :env.obs_dim], final_g=None if fg is None else c(fg)[..., :env.obs_dim],
                flags=c(fl))


def _ulps32(got, want64):
    want = np.asarray(want64, np.float64).astype(np.float32)
    d = np.abs(np.asarray(got, np.float32).view(np.int32).astype(np.int64) - want.view(np.int32).astype(np.int64))
    return int(d.max()) if d.size else 0


@pytest.mark.parametrize("pipeline", [128, 1], ids=["pipeline128", "single_launch"])
def test_bench_configuration_final_info_matches_oracle(oracle, pipeline):
    N, K, seed = 65536, 32, 2026
    envs = [_venv(V2, N, "GAME", seed=seed, pipeline=pipeline) for _ in range(2)]
    T = envs[0].max_episode_steps
    st = envs[0].get_state()
    st["step"][:] = (np.arange(N) * 7919) % max(T - 1, 1)     # bench.py's desynchronisation
    for e in envs:
        e.set_state(st)
    g = torch.Generator(device="cuda").manual_seed(1)
    acts = torch.randint(0, 8, (K, N, envs[0].num_robots), generator=g, dtype=torch.uint8, device="cuda")

    # rr_step and rr_step_info from the same state: everything else bit-identical
    l0 = envs[0].launch_count
    obs_h, obs_g, rew, done = (x.cpu().numpy() for x in envs[0].step_k(acts, K))
    got = _step_info(envs[1], acts, K)
    assert envs[0].launch_count - l0 == (128 if pipeline > 1 else 1)
    for k, v in (("obs_h", obs_h), ("obs_g", obs_g), ("rew", rew), ("done", done)):
        assert np.array_equal(got[k], v, equal_nan=True), k
    fin = [e.get_state() for e in envs]
    for k in STATE_KEYS:
        assert np.array_equal(fin[0][k], fin[1][k]), k
    assert np.array_equal(envs[0].error_mask(), envs[1].error_mask())
    s0, s1 = envs[0].get_stats(), envs[1].get_stats()
    for k in ("episodes", "length", "naughty", "errors", "steps", "squeeze_replays"):
        assert s0[k] == s1[k], (k, s0[k], s1[k])
    for k in ("return_happy", "return_grumpy"):
        assert abs(s0[k] - s1[k]) <= 1e-9 * max(1.0, abs(s0[k])), (k, s0[k], s1[k])

    dn = got["done"] != 0
    assert (got["flags"][~dn] == 0).all() and set(np.unique(got["flags"])) <= {0, ROW_TRUNCATED, ROW_RAISED}
    assert (got["final_h"][~dn] == np.float32(CANARY32)).all() and (got["final_g"][~dn] == np.float32(CANARY32)).all()
    assert dn.sum() >= 256, dn.sum()

    stride = 67
    sample = np.unique(np.concatenate([np.arange(0, N, stride), np.nonzero(st["step"] >= T - K)[0][:256]]))
    oracle.scratch_mode(1)
    diverged, rows, exact, truncated = [], 0, 0, 0
    try:
        o = oracle.OracleEnv("GAME", V2, time_limit=True)
        a = acts[:, torch.as_tensor(sample, device="cuda")].cpu().numpy()
        for j, i in enumerate(sample):
            o.set_state({k: st[k][i] for k in STATE_KEYS})
            episode, bad = 0, None
            for s in range(K):
                out = o.step(a[s, j])
                finished = bool(out["done"]) or out["err"] != 0
                if int(finished) != int(got["done"][s, i]):
                    bad = (int(i), s, "done")
                    break
                if _ulps32(got["obs_h"][s, i], out["obs_h"]) > 1 and not finished:
                    bad = (int(i), s, "obs")
                    break
                if finished:
                    step = int(o.get_state()["step"])
                    flags = ROW_RAISED if out["err"] else (ROW_TRUNCATED if step == T else 0)   # no goals: game_is_done() is step > T
                    if got["flags"][s, i] != flags:
                        bad = (int(i), s, f"flags {got['flags'][s, i]} != {flags}")
                        break
                    truncated += flags == ROW_TRUNCATED
                    u = max(_ulps32(got["final_h"][s, i], o.observe(1)), _ulps32(got["final_g"][s, i], o.observe(-1)))
                    if out["err"] == 0:
                        if u > 1:
                            bad = (int(i), s, f"final obs {u} fp32 ulps")
                            break
                        rows += 1
                        exact += u == 0
                    episode += 1
                    o.reset_philox(seed, int(i), episode)
            if bad is not None:
                diverged.append(bad)
    finally:
        oracle.scratch_mode(0)
    print(f"final info, bench configuration, pipeline {pipeline}: {len(sample)} sampled envs, {rows} done rows compared "
          f"({exact} bit-equal in fp32, {truncated} truncated), {len(diverged)} diverged: {diverged[:4]}")
    assert rows >= 64 and truncated >= 64
    assert len(diverged) <= 2, diverged
    for e in envs:
        e.close()


def test_train_truncated_exactly_where_the_step_counter_reaches_T():
    """TRAIN, time limit and auto-reset from a fresh batch, 8 launches of 40 steps: every episode that does not raise
    ends by truncation on its T-th row, and the final observation is what rr_step_info with auto_reset = 0 reports as
    the observation of that row."""
    N, K = 1024, 40
    env = _venv(V2, N, "TRAIN", seed=5, out_dtype=torch.float64)
    twin = _venv(V2, N, "TRAIN", seed=5, out_dtype=torch.float64, auto_reset=False)
    T = env.max_episode_steps
    since = np.zeros(N, np.int64)
    seen = 0
    g = torch.Generator(device="cuda").manual_seed(2)
    for call in range(8):
        acts = torch.randint(0, 8, (K, N, 1), generator=g, dtype=torch.uint8, device="cuda")
        got = _step_info(env, acts, K, canary=np.nan)
        tw = _step_info(twin, acts, K, final=False, flags=False) if call * K < T else None
        for s in range(K):
            since += 1
            dn = got["done"][s] != 0
            raised = (got["flags"][s] & ROW_RAISED) != 0
            assert ((got["flags"][s] == ROW_TRUNCATED) == (dn & ~raised)).all()
            assert (since[dn & ~raised] == T).all() and (since[~dn] < T).all()
            if tw is not None and call * K + s == T - 1:             # the twin without auto-reset: the same rows
                ok = dn & ~raised
                assert np.array_equal(got["final_h"][s][ok], tw["obs_h"][s][ok], equal_nan=True)
                assert np.array_equal(got["final_g"][s][ok], tw["obs_g"][s][ok], equal_nan=True)
            assert np.isnan(got["final_h"][s][~dn]).all()
            seen += int((dn & ~raised).sum())
            since[dn] = 0
    assert seen >= N // 2, seen
    env.close(); twin.close()


# (env id, preset, goal scoring, out dtype, n envs): n > 384 x #SM selects the 448-thread GAME kernel for one launch
HOST_CASES = [("DuelGoals", "GAME", True, torch.float32, 60000), ("DuelGoals", "TRAIN", True, torch.float64, 4096),
              (V0, "GAME", True, torch.float64, 4096), (V2, "GAME", False, torch.float64, 4096),
              (V0, "GAME", False, torch.float32, 4096), ("DuelAllCoordsPrior", "TRAIN", False, torch.float64, 4096)]


@pytest.mark.parametrize("case", HOST_CASES, ids=[f"{c[0]}-{c[1]}-goals{int(c[2])}-{str(c[3])[6:]}-{c[4]}" for c in HOST_CASES])
def test_first_row_equals_the_host_build(case):
    """The handle's own placements with step counters spread around T (and past it), so that the first row ends by
    truncation, by the raw limit, by a refusal or not at all: done and flags of that row equal the host build's bit for
    bit, final observations within the parity bar (fp32: one ulp of the cast host value)."""
    from emul import emul_info
    from emul.emul import EmulBatch
    from golden_util import resolve_env, resolve_rewards
    env_id, preset, goals, dt, n = case
    base, observer = resolve_env(env_id)
    kw = dict(seed=3, out_dtype=dt, goal_scoring=goals)
    if observer is not None:
        kw["observer"] = observer
    if resolve_rewards(env_id) is not None:
        kw["reward_mask"], kw["reward_order"] = resolve_rewards(env_id)
    env = _venv(base, n, preset, **kw)
    T = env.max_episode_steps
    st = env.get_state()
    rng = np.random.default_rng(4)
    st["step"] = (T - rng.integers(-2, 4, n)).astype(np.int32)
    env.set_state(st)
    A = env.num_robots if env.discrete else 2 * env.num_robots
    a = (rng.integers(0, 8, (2, n, A)).astype(np.uint8) if env.discrete
         else rng.choice(np.array([-1.0, 0.0, 1.0, np.nan], np.float32), (2, n, A), p=[.33, .33, .33, .01]))
    got = _step_info(env, torch.as_tensor(a).cuda(), 2)
    emul_info.use_libm_sincos(False)
    hb = EmulBatch(env.cfg, n, env.num_robots, env.num_balls, env.obs_dim)
    for i in range(n):
        hb.set_state(i, {k: st[k][i] for k in STATE_KEYS})
    h = emul_info.launch(hb, a[:1].astype(np.float64), observe=True)
    assert np.array_equal(got["done"][0], h["done"][0]) and np.array_equal(got["flags"][0], h["flags"][0])
    print(f"{case}: first row flags {np.bincount(h['flags'][0], minlength=3).tolist()}")
    if env.obs_dim:
        # (the observers call atan, which CUDA's libm and the host's may round differently in the last bit)
        dn = h["done"][0] != 0
        for key in ("final_h", "final_g"):
            g_, w_ = got[key][0][dn], h[key][0][dn]
            if dt == torch.float32:
                assert _ulps32(g_, w_) <= 1, key
            else:
                assert close(g_, w_), key
            print(f"  {key}: {int(np.all((g_ == w_.astype(g_.dtype)) | np.isnan(g_), axis=1).sum())}/{int(dn.sum())} rows bit-equal")
        assert (h["flags"][0] == ROW_TRUNCATED).sum() > 0
    env.close()


def test_misaligned_final_buffers_are_refused_and_nothing_is_launched():
    from roborugby_b200 import _lib
    for dt, off in ((torch.float32, 2), (torch.float64, 4)):
        env = _venv(V2, 64, "TRAIN", out_dtype=dt)
        K, N, D = 2, 64, env.obs_dim
        acts = torch.zeros((K, N, 1), dtype=torch.uint8, device="cuda")
        raw = torch.zeros(K * N * D * 8 + 64, dtype=torch.uint8, device="cuda")
        for which in (0, 1):
            l0 = env.launch_count
            ptrs = [None, None]
            ptrs[which] = raw.data_ptr() + off
            rc = env.lib.rr_step_info(env._h, acts.data_ptr(), 1, K, None, None, None, None, ptrs[0], ptrs[1], None,
                                      env._stream())
            assert rc == -1 and b"aligned" in env.lib.rr_last_error() and env.launch_count == l0
        # the row flags need no alignment
        _lib.check(env.lib.rr_step_info(env._h, acts.data_ptr(), 1, K, None, None, None, None, None, None,
                                        raw.data_ptr() + 3, env._stream()))
        torch.cuda.synchronize()
        assert env.launch_count == l0 + 1
        env.close()


def test_python_layer_shapes_and_gym_truncation():
    """step_k(final_info=True) and step(final_info=True): shapes, dtypes and info keys; over one TRAIN episode the
    batched env's "TimeLimit.truncated" equals the single env's (gym_env.RoboRugbyEnv(time_limit=True))."""
    from roborugby_b200.gym_env import RoboRugbyEnv
    env = _venv(V2, 8, "TRAIN", seed=9, pipeline=1)
    K = 3
    out = env.step_k(torch.zeros((K, 8, 1), dtype=torch.uint8, device="cuda"), K, final_info=True)
    assert len(out) == 5
    f = out[4]
    assert f["final_obs"].shape == (K, 8, env.obs_dim) and f["final_obs"].dtype == torch.float32
    assert f["final_obs_grumpy"].shape == (K, 8, env.obs_dim)
    assert f["truncated"].shape == (K, 8) and f["truncated"].dtype == torch.bool and f["raised"].dtype == torch.bool
    assert len(env.step_k(torch.zeros((K, 8, 1), dtype=torch.uint8, device="cuda"), K)) == 4

    single = RoboRugbyEnv(V2, preset="TRAIN", device="cuda:0", seed=9, time_limit=True)
    single.reset()
    venv = _venv(V2, 1, "TRAIN", seed=9)
    venv.set_state(single._v.get_state())
    T = venv.max_episode_steps
    rng = np.random.default_rng(6)
    for t in range(T):
        a = int(rng.integers(0, 8))
        _, _, d1, info1 = single.step([a])
        _, _, d2, info2 = venv.step(torch.tensor([[a]], dtype=torch.uint8), final_info=True)
        assert set(info2) >= {"final_observation", "final_observation_grumpy", "TimeLimit.truncated", "raised"}
        assert info2["final_observation"].shape == (1, venv.obs_dim) and info2["raised"].shape == (1,)
        assert bool(d2[0]) == d1
        assert bool(info2["TimeLimit.truncated"][0]) == bool(info1.get("TimeLimit.truncated", False)), t
        if d1:
            assert t == T - 1 and info1["TimeLimit.truncated"]
            break
    else:
        pytest.fail("the episode did not end at the time limit")
    env.close(); venv.close(); single.close()
