"""GPU tier (B200): each row's episode result from the fused step kernel (rr_step_episodes, k_step<L, OutT, true> and
k_step<L, OutT, true, true> with their episode outputs).

* Kernel = host build, bit for bit (fp64 returns included): for a prefix of each case's envs, every row's episode
  return, length and goal words, and the launch's other rows and final state, equal tests/emul emul_episodes.launch
  under the rules of test_host_build_equivalence_gpu.  The cases follow test_reset_pool_gpu.CASES (GAME through 128
  groups, the 448-thread GAME launch with goals, AllCoords_WithPrior and fp64, TRAIN at 80 001 envs, TRAIN with goals
  through the pipeline), each without and with a reset pool.
* At full size the rows add up to the statistics: rows with ep_length >= 0 are the change in RR_STAT_EPISODES and their
  lengths the change in RR_STAT_LENGTH, exactly; the returns sum to the change in RR_STAT_RETURN_* within 1e-12 relative
  (the statistics add in atomic order).
* Setting the outputs changes nothing else: a second handle stepped through rr_step_info / rr_step_pool gives the same
  rows, state and statistics; with the three pointers NULL rr_step_episodes is rr_step_pool / rr_step_info bit for bit.
* One group and 128 groups give identical results; step(..., episode_info=True) agrees with step_k.
* Refusals: every RR_E_INVALID case of rr_step_episodes, with nothing launched, and the Python ValueErrors."""
import ctypes as C
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from test_host_build_equivalence_gpu import ATAN_COLS, Tally, _compare_rows, _compare_state, _sms, k_step_variant
from test_reset_pool_gpu import COUNTS, OBS_PRIOR, V2, _actions, _env, _eq, _np, _pool_rows

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

EPISODES, RET, LENGTH = 0, [1, 2], 3

# name -> (preset, N, K, pipeline, fp64, goal scoring, observer, envs checked against the host build)
CASES = {
    "game_pipeline128": ("GAME", 65536, 32, 128, False, False, None, 1536),
    "game_wide_goals_prior_f64": ("GAME", 65529, 16, 1, True, True, OBS_PRIOR, 1024),
    "train": ("TRAIN", 80001, 32, 1, False, False, None, 8192),
    "train_goals_pipeline8": ("TRAIN", 30001, 32, 8, False, True, None, 4096),
}


def _desync(env):
    """bench.py's episode phases: envs end one after another through the launches."""
    st = env.get_state()
    st["step"][:] = (np.arange(env.num_envs) * 7919) % max(env.max_episode_steps - 1, 1)
    env.set_state(st)


def _episode_rows(info):
    return dict(ep_return=_np(info["episode_return"]), ep_length=_np(info["episode_length"]),
                ep_goals=_np(info.get("episode_goals")))


def _check_sums(ga, stats, N):
    el, er = ga["ep_length"], ga["ep_return"]
    end = el >= 0
    assert (el >= -1).all() and (er[~end] == 0.0).all()
    if ga["ep_goals"] is not None:
        assert (ga["ep_goals"][~end] == 0).all()
    assert end.sum() == stats[EPISODES] and el[end].sum() == stats[LENGTH], (end.sum(), el[end].sum(), stats)
    # relative to the magnitudes summed: the statistics add the same values in atomic order
    tol = 1e-12 * np.abs(er).sum((0, 1))
    assert (np.abs(er.sum((0, 1)) - stats[RET]) <= tol).all(), (er.sum((0, 1)), stats[RET])
    return int(end.sum())


@pytest.mark.parametrize("pooled", [False, True], ids=["random_resets", "pool"])
@pytest.mark.parametrize("case", list(CASES))
def test_episode_rows_equal_the_host_build_and_add_up_to_the_statistics(case, pooled):
    from roborugby_b200.vec_env import ResetPool
    preset, N, K, pipeline, f64, goals, observer, n_host = CASES[case]
    rng = np.random.default_rng(N + pooled)
    A = _env(preset, N, pipeline, f64, goals, observer)
    B = _env(preset, N, pipeline, f64, goals, observer)
    _desync(A)
    pool = None
    if pooled:
        m = 256
        w = rng.random(m) * 3
        w[rng.random(m) < 0.2] = 0.0
        pool = ResetPool(_pool_rows(A, m, rng), torch.as_tensor(w), p=0.7)
    rows0 = A.save_states()
    B.load_states(rows0)
    rows0 = rows0.cpu().numpy()
    acts = _actions(A, K, rng)
    A.clear_stats(); B.clear_stats()
    n0 = A.launch_count
    oh, og, rew, done, info = A.step_k(torch.as_tensor(acts).cuda(), K, reset_pool=pool, episode_info=True)
    assert A.launch_count - n0 == k_step_variant(preset, goals, N, pipeline, _sms())[2]
    ga = dict(obs_h=_np(oh), obs_g=_np(og), rew=_np(rew), done=_np(done), final_h=_np(info["final_obs"]),
              final_g=_np(info["final_obs_grumpy"]), flags=_np(info["row_flags"]), **_episode_rows(info))
    ga["slot"] = _np(info["reset_slot"]) if pooled else np.full((K, N), -1, np.int32)
    assert (info["episode_end"].cpu().numpy() == (ga["ep_length"] >= 0)).all()
    assert (ga["ep_goals"] is not None) == goals
    ga["rows"] = A.save_states().cpu().numpy()
    stats = A.stats.cpu().numpy().copy()
    n_ep = _check_sums(ga, stats, N)
    print(f"{case} {'pool' if pooled else 'random resets'}: {N} envs x {K} steps, {n_ep} episodes counted, "
          f"{int((ga['done'] != 0).sum())} done rows, mean length {ga['ep_length'][ga['ep_length'] >= 0].mean():.1f}")
    assert n_ep >= (400 if case == "game_pipeline128" else 150 if preset == "GAME" else 1000)
    # the same launch without the episode outputs
    b = B.step_k(torch.as_tensor(acts).cuda(), K, final_info=True, reset_pool=pool)
    dn = ga["done"] != 0
    for key, got in (("obs_h", b[0]), ("obs_g", b[1]), ("rew", b[2]), ("done", b[3]), ("flags", b[4]["row_flags"])):
        assert _eq(ga[key], _np(got)), key
    if A.obs_dim:
        assert _eq(ga["final_h"][dn], _np(b[4]["final_obs"])[dn]) and _eq(ga["final_g"][dn], _np(b[4]["final_obs_grumpy"])[dn])
    if pooled:
        assert _eq(ga["slot"], _np(b[4]["reset_slot"]))
    assert np.array_equal(ga["rows"], B.save_states().cpu().numpy())
    sb = B.stats.cpu().numpy()
    assert np.array_equal(stats[COUNTS], sb[COUNTS]) and np.allclose(stats[RET], sb[RET], rtol=1e-12, atol=1e-9)
    _check_host_build(A, f"{case}/{'pool' if pooled else 'random'}", rows0, acts, ga, pool, n_host, f64)
    A.close(); B.close()


def _check_host_build(env, case, rows0, acts, ga, pool, n, f64):
    """Envs [0, n) of the launch against emul_episodes.launch, in chunks of their own EmulBatch (env_offset shifted, so
    that the draws and random resets are those of the GPU env)."""
    from emul import emul_episodes
    emul_episodes.use_libm_sincos(False)
    rows = None if pool is None else pool.rows.cpu().numpy()
    cdf = None if pool is None or pool.cdf is None else pool.cdf.cpu().numpy()
    p = 1.0 if pool is None else pool.p
    workers = max(1, os.cpu_count() or 1)
    bounds = [(n * j // (2 * workers), n * (j + 1) // (2 * workers)) for j in range(2 * workers)]
    f32, D = not f64, env.obs_dim
    atan = ATAN_COLS.get(env.cfg.observer, [])

    def chunk(bd):
        from emul import emul, emul_states
        from roborugby_b200._lib import Config
        c0, c1 = bd
        t = Tally()
        if c1 == c0:
            return t
        cfg = Config.from_buffer_copy(env.cfg)
        cfg.env_offset = env.cfg.env_offset + c0
        batch = emul.EmulBatch(cfg, c1 - c0, env.num_robots, env.num_balls, D)
        start = np.zeros((3 * env.num_robots + 2 * env.num_balls, c1 - c0))
        emul_states.load(batch, start, np.ascontiguousarray(rows0[c0:c1]))
        h = emul_episodes.launch(batch, acts[:, c0:c1].astype(np.float64), start, rows, cdf, p)
        g = {k: v[:, c0:c1] for k, v in ga.items() if k != "rows" and v is not None}
        for key in ("rew", "done", "flags", "slot"):
            _compare_rows(t, key, g[key], h[key], f32, c0)
        for key in ("ep_return", "ep_length", "ep_goals"):   # fp64 whatever out_f64 is
            if key in g:
                _compare_rows(t, key, g[key], h[key], False, c0)
        if D:
            _compare_rows(t, "obs_h", g["obs_h"], h["obs_h"], f32, c0, atan)
            _compare_rows(t, "obs_g", g["obs_g"], h["obs_g"], f32, c0, atan)
            dn = h["done"] != 0
            for key in ("final_h", "final_g"):
                _compare_rows(t, key, g[key][dn][None], h[key][dn][None], f32, c0, atan)
        _compare_state(t, "state", ga["rows"][c0:c1], emul_states.save(batch, start), c0)
        t.add("episodes", (h["ep_length"] >= 0).sum())
        return t

    t = Tally()
    with ThreadPoolExecutor(workers) as ex:   # ctypes releases the GIL
        for part in ex.map(chunk, bounds):
            t.merge(part)
    print(f"{case}: envs [0, {n}) against the host build: {t.n.get('ep_length.rows', 0)} episode rows, "
          f"{t.n.get('episodes', 0)} episodes, {t.n.get('state.bytes', 0)} state bytes; {t.n.get('differences', 0)} differing")
    for f in t.first:
        print("  ", f)
    assert not t.first, t.first
    assert t.n.get("episodes", 0) > 0


def _raw_launch(env, acts, K, pool, ep):
    """rr_step_episodes through ctypes into fresh buffers: (outputs dict, slot or None)."""
    from roborugby_b200 import _lib
    N = env.num_envs
    o = {k: torch.full_like(v, 0x7b) if v.dtype == torch.uint8 else torch.full_like(v, -3.25) for k, v in env._out(K).items()}
    f = {k: torch.full_like(v, 0x7b) if v.dtype == torch.uint8 else torch.full_like(v, -3.25)
         for k, v in env._final_out(K).items()}
    slot = torch.full((K, N), 7, dtype=torch.int32, device="cuda")
    e = dict(er=torch.full((K, N, 2), 9.5, dtype=torch.float64, device="cuda"),
             el=torch.full((K, N), 9, dtype=torch.int32, device="cuda"))
    if env.cfg.goal_scoring:
        e["eg"] = torch.full((K, N, 4), 9, dtype=torch.int32, device="cuda")
    ptr = (lambda k: e[k].data_ptr() if k in e else None) if ep else (lambda k: None)
    _lib.check(env.lib.rr_step_episodes(env._h, acts.data_ptr(), acts.shape[2], K, o["obs_h"].data_ptr(),
                                        o["obs_g"].data_ptr(), o["rew"].data_ptr(), o["done"].data_ptr(),
                                        f["final_obs_h"].data_ptr(), f["final_obs_g"].data_ptr(), f["row_flags"].data_ptr(),
                                        None if pool is None else C.byref(pool._c), slot.data_ptr(), ptr("er"), ptr("el"),
                                        ptr("eg"), env._stream()))
    env.join()
    return dict(o, **f, slot=slot, **e)


@pytest.mark.parametrize("pooled", [False, True], ids=["no_pool", "pool"])
def test_null_episode_pointers_equal_step_pool_and_step_info(pooled):
    """rr_step_episodes with the three pointers NULL is rr_step_pool (pool) / rr_step_info (no pool) bit for bit: every
    output, reset_slot, the saved rows and the statistics."""
    from roborugby_b200 import _lib
    from roborugby_b200.vec_env import ResetPool
    rng = np.random.default_rng(51)
    N, K = 65536, 32
    A = _env("GAME", N, 128, False, True, None)
    B = _env("GAME", N, 128, False, True, None)
    _desync(A)
    pool = ResetPool(_pool_rows(A, 128, rng), p=1.0) if pooled else None
    rows0 = A.save_states()
    B.load_states(rows0)
    A.clear_stats(); B.clear_stats()
    acts = torch.as_tensor(_actions(A, K, rng)).cuda()
    a = _raw_launch(A, acts, K, pool, ep=False)
    assert (a["er"] == 9.5).all() and (a["el"] == 9).all() and (a["eg"] == 9).all()   # NULL: nothing written
    o, f = B._out(K), B._final_out(K)
    args = (B._h, acts.data_ptr(), acts.shape[2], K, o["obs_h"].data_ptr(), o["obs_g"].data_ptr(), o["rew"].data_ptr(),
            o["done"].data_ptr(), f["final_obs_h"].data_ptr(), f["final_obs_g"].data_ptr(), f["row_flags"].data_ptr())
    slot = torch.full((K, N), 7, dtype=torch.int32, device="cuda")
    if pooled:
        _lib.check(B.lib.rr_step_pool(*args, C.byref(pool._c), slot.data_ptr(), B._stream()))
    else:
        _lib.check(B.lib.rr_step_info(*args, B._stream()))
        slot.fill_(-1)
    B.join()
    dn = o["done"].bool()
    assert dn.any()
    for key in ("obs_h", "obs_g", "rew", "done"):
        assert torch.equal(a[key], o[key]), key
    assert torch.equal(a["row_flags"], f["row_flags"]) and torch.equal(a["slot"], slot)
    assert torch.equal(a["final_obs_h"][dn], f["final_obs_h"][dn]) and torch.equal(a["final_obs_g"][dn], f["final_obs_g"][dn])
    assert torch.equal(A.save_states(), B.save_states())
    sa, sb = A.stats.cpu().numpy(), B.stats.cpu().numpy()
    assert np.array_equal(sa[COUNTS], sb[COUNTS]) and np.allclose(sa[RET], sb[RET], rtol=1e-12, atol=1e-9)
    A.close(); B.close()


def test_one_group_and_128_groups_give_identical_results():
    """GAME, 65 536 envs with goal scoring and a pool: one launch (448-thread blocks) and 128 sub-batch groups (384-thread
    blocks) give the same episode rows, the same other rows and the same final state."""
    from roborugby_b200.vec_env import ResetPool
    rng = np.random.default_rng(52)
    N, K = 65536, 32
    envs = {g: _env("GAME", N, g, False, True, None) for g in (1, 128)}
    _desync(envs[1])
    pool = ResetPool(_pool_rows(envs[1], 256, rng), p=0.5)
    rows0 = envs[1].save_states()
    envs[128].load_states(rows0)
    acts = torch.as_tensor(_actions(envs[1], K, rng)).cuda()
    out = {}
    for g, env in envs.items():
        oh, og, rew, done, info = env.step_k(acts, K, reset_pool=pool, episode_info=True)
        out[g] = dict(rew=_np(rew), done=_np(done), flags=_np(info["row_flags"]), slot=_np(info["reset_slot"]),
                      rows=env.save_states().cpu().numpy(), **_episode_rows(info))
    for key in out[1]:
        assert _eq(out[1][key], out[128][key]), key
    assert (out[1]["ep_length"] >= 0).sum() > 300
    for env in envs.values():
        env.close()


def test_step_agrees_with_step_k():
    """step(..., episode_info=True) K times equals one step_k(K, episode_info=True) from the same state: info["episode"]
    r / r_grumpy / l and info["_episode"] are the rows of episode_return, episode_length and episode_end; with goal
    scoring info["episode_goals"] those of episode_goals."""
    rng = np.random.default_rng(53)
    N, K = 4096, 12
    A = _env("TRAIN", N, 1, False, True, None)
    B = _env("TRAIN", N, 1, False, True, None)
    _desync(A)
    B.load_states(A.save_states())
    acts = torch.as_tensor(_actions(A, K, rng)).cuda()
    _, _, _, _, info = B.step_k(acts, K, episode_info=True)
    want = {k: _np(info[k]) for k in ("episode_return", "episode_length", "episode_end", "episode_goals")}
    for s in range(K):
        _, _, _, inf = A.step(acts[s], episode_info=True)
        ep = inf["episode"]
        assert inf["_episode"].dtype == torch.bool and ep["l"].dtype == torch.int32 and ep["r"].dtype == torch.float64
        assert _eq(_np(ep["r"]), want["episode_return"][s, :, 0]) and _eq(_np(ep["r_grumpy"]), want["episode_return"][s, :, 1])
        assert _eq(_np(ep["l"]), want["episode_length"][s]) and _eq(_np(inf["_episode"]), want["episode_end"][s])
        assert _eq(_np(inf["episode_goals"]), want["episode_goals"][s])
    assert want["episode_end"].sum() > 50
    A.close(); B.close()


def test_refusals_launch_nothing():
    from roborugby_b200 import _lib
    from roborugby_b200.vec_env import ResetPool
    N = 256
    env = _env("TRAIN", N, 1, False, False, None)
    goals = _env("TRAIN", N, 1, False, True, None)
    acts = torch.zeros(1, N, 1, dtype=torch.uint8, device="cuda")
    o = env._out(1)
    er = torch.empty(2, N, 2, dtype=torch.float64, device="cuda")
    ei = torch.empty(2, N, 4, dtype=torch.int32, device="cuda")
    rows = env.save_states()
    lib = env.lib

    def call(on=env, k=1, pool=None, ep_return=er.data_ptr(), ep_length=ei.data_ptr(), ep_goals=None, rew=o["rew"].data_ptr()):
        n0 = on.launch_count
        rc = lib.rr_step_episodes(on._h, acts.data_ptr(), 1, k, None, None, rew, o["done"].data_ptr(), None, None, None,
                                  None if pool is None else C.byref(pool), None, ep_return, ep_length, ep_goals,
                                  env._stream())
        assert on.launch_count == n0
        return rc, lib.rr_last_error().decode()

    for kw, msg in ((dict(ep_return=er.data_ptr() + 4), "ep_return"), (dict(ep_length=ei.data_ptr() + 2), "ep_length"),
                    (dict(on=goals, ep_goals=ei.data_ptr() + 2), "ep_goals"), (dict(ep_goals=ei.data_ptr()), "goal_scoring"),
                    (dict(k=0), "k_steps"), (dict(rew=o["rew"].data_ptr() + 2), "aligned"),
                    (dict(pool=_lib.ResetPoolC(rows.data_ptr(), N, None, float("nan"))), "p_pool"),
                    (dict(pool=_lib.ResetPoolC(None, N, None, 1.0)), "rows_dev")):
        rc, err = call(**kw)
        assert rc == -1 and msg in err, (kw, err)
    assert lib.rr_step_episodes(None, None, 0, 1, *([None] * 7), None, None, None, None, None, None) == -1
    # the same arguments, aligned, launch (goal words on the goal-scoring handle)
    n0 = goals.launch_count
    rc = lib.rr_step_episodes(goals._h, acts.data_ptr(), 1, 1, None, None, o["rew"].data_ptr(), o["done"].data_ptr(), None,
                              None, None, None, None, er.data_ptr(), ei.data_ptr(), ei.data_ptr(), goals._stream())
    assert rc == 0 and goals.launch_count == n0 + 1
    # Python: episode_info goes through the same checks of reset_pool
    with pytest.raises(ValueError):
        env.step_k(acts, 1, reset_pool=rows, episode_info=True)
    game = _env("GAME", 64, 1, False, False, None)
    with pytest.raises(ValueError, match="bytes wide"):
        game.step_k(torch.zeros(1, 64, 4, dtype=torch.uint8, device="cuda"), 1, reset_pool=ResetPool(rows),
                    episode_info=True)
    na = _env("TRAIN", N, 1, False, False, None, auto_reset=False)
    with pytest.raises(ValueError):
        na.step_k(acts, 1, reset_pool=ResetPool(rows), episode_info=True)
    _, _, _, info = na.step(acts[0], episode_info=True)   # without auto-reset the episode outputs still work
    assert "episode_goals" not in info and info["episode"]["l"].shape == (N,)
    for e in (env, goals, game, na):
        e.close()


def test_dqn_loop_returns_every_episode():
    """dqn.train(..., episode_returns=True): one entry per episode get_stats counts, whose sum is the statistics'
    return, and the reference's 100-episode average after each one."""
    from roborugby_b200.dqn import VecDQNAgent, train
    from roborugby_b200.vec_env import RoboRugbyVecEnv
    N, T = 256, 310
    env = RoboRugbyVecEnv(V2, N, preset="TRAIN", device="cuda:0", seed=5, n_actions=1)
    ag = VecDQNAgent(env.obs_dim, batch_size=512, max_mem_size=50000, device="cuda:0")
    out = train(env, ag, T, learn_every=10, episode_returns=True)
    r, avg = out["episode_returns"].numpy(), out["avg_return_100"].numpy()
    st = out["stats"]
    assert r.shape == (st["episodes"], 2) and st["episodes"] >= N
    assert np.allclose(r.sum(0), [st["return_happy"], st["return_grumpy"]], rtol=1e-12, atol=1e-9)
    want = [r[max(0, j - 99):j + 1, 0].mean() for j in range(len(r))]
    assert np.allclose(avg, want, rtol=1e-12) and avg.shape == out["avg_return_100_grumpy"].shape
    env.close()
