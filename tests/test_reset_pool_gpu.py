"""GPU tier (B200): auto-reset from a reset pool inside the fused step kernel (rr_step_pool, k_step<L, OutT, true, true>).

* Composition, bit for bit: handle A steps K env-steps in one launch with a pool (p = 1) and records reset_slot; handle B
  (same config, same starting rows) steps the same actions one env-step at a time through rr_step_info and, after each
  step, loads the rows A's resets drew (load_states).  Every rew, done, row_flags and terminal-observation row is equal;
  obs rows too, where a done row of A is compared with B's observe() after the load.  The final saved rows are
  byte-equal except the episode counter (A keeps its own, B took the row's), and the integer statistics are equal.  The
  pool is saved a few steps before the time limit, so most envs reset several times per launch.  The cases cover GAME
  and TRAIN, goal scoring, AllCoords_WithPrior, fp64 outputs, the sub-batch pipeline and one launch, and both GAME block
  variants (384 threads through the pipeline, 448 threads as one launch over more envs than 384 x #SM).
* Kernel = host build: for a prefix of each case's envs, the launch's rows, reset_slot, final rows and statistics equal
  tests/emul emul_pool.launch (the same rr_sim.cuh pool_reset) under the rules of test_host_build_equivalence_gpu.
* Draws on the device: reset_slot of a weighted pool passes a chi-square test against the weights and never names a
  zero-weight slot; p = 0.5 takes the pool half the time; p = 0 gives all -1 and exactly rr_step_info's outputs; a NULL
  pool through rr_step_pool is rr_step_info.
* Refusals: every RR_E_INVALID case of rr_step_pool and the Python ValueErrors, with nothing launched."""
import ctypes as C
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from test_host_build_equivalence_gpu import ATAN_COLS, Tally, _compare_rows, _compare_state, _same, k_step_variant, _sms

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

V2 = "RoboRugbySimpleDuel-v2"
OBS_PRIOR, OBS_L6V2 = 4, 2
COUNTS, RET = [0, 3, 4, 5, 6], [1, 2]   # statistics: episodes, length, naughty, errors, steps; returns

# name -> (preset, N, K, pipeline, fp64, goal scoring, observer, weighted, envs checked against the host build)
CASES = {
    "game_pipeline128": ("GAME", 65536, 32, 128, False, False, None, True, 1536),
    "game_wide_goals_prior_f64": ("GAME", 65529, 16, 1, True, True, OBS_PRIOR, False, 1024),
    "game_pipeline4_f64": ("GAME", 40000, 16, 4, True, False, OBS_L6V2, True, 1024),
    "train": ("TRAIN", 80001, 32, 1, False, False, None, False, 8192),
    "train_goals_prior_pipeline8_f64": ("TRAIN", 30001, 32, 8, True, True, OBS_PRIOR, True, 4096),
}


def _env(preset, N, pipeline, f64, goals, observer, **kw):
    from roborugby_b200.vec_env import RoboRugbyVecEnv
    return RoboRugbyVecEnv(V2, N, preset=preset, device="cuda:0", seed=4242, out_dtype=torch.float64 if f64 else
                           torch.float32, goal_scoring=goals, observer=observer, pipeline=pipeline, **kw)


def _pool_rows(env, m, rng):
    """m rows of envs a few steps before the time limit (saved from env, which is then loaded back as it was)."""
    keep = env.save_states()
    st = env.get_state()
    T = env.max_episode_steps
    st["step"][:] = T - 4 - (np.arange(env.num_envs) % 5)
    env.set_state(st)
    env.step_k(torch.as_tensor(_actions(env, 2, rng)).cuda(), 2)
    rows = env.save_states(torch.as_tensor(rng.choice(env.num_envs, m, replace=False)).cuda())
    env.load_states(keep)
    env.clear_stats()
    return rows


def _actions(env, K, rng):
    return rng.integers(0, 8, (K, env.num_envs, env.action_dim)).astype(np.uint8)


def _episode_bytes(env):
    """Byte range of the episode counter in a saved row: sf columns, the starting layout, then si (rr_sim.cuh RowLayout)."""
    from emul import emul
    dims = np.zeros(5, np.int32)
    emul.lib().emul_cols_dims(C.byref(env.cfg), dims.ctypes.data_as(C.c_void_p))
    off = 8 * (int(dims[0]) + 3 * env.num_robots + 2 * env.num_balls) + 4 * int(dims[2])
    return slice(off, off + 4)


def _np(x):
    return None if x is None else x.cpu().numpy().copy()


def _eq(a, b):
    """Bit-identical (floats: or both NaN)."""
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and (bool(_same(a, b).all()) if a.dtype.kind == "f" else np.array_equal(a, b))


@pytest.mark.parametrize("case", list(CASES))
def test_pool_launch_is_step_info_then_load_states(case):
    from roborugby_b200.vec_env import ResetPool
    preset, N, K, pipeline, f64, goals, observer, weighted, n_host = CASES[case]
    rng = np.random.default_rng(N)
    A = _env(preset, N, pipeline, f64, goals, observer)
    B = _env(preset, N, pipeline, f64, goals, observer)
    m = 256
    rows = _pool_rows(A, m, rng)
    w = None
    if weighted:
        w = rng.random(m) * 3
        w[rng.random(m) < 0.2] = 0.0
    pool = ResetPool(rows, None if w is None else torch.as_tensor(w), p=1.0)
    start = torch.as_tensor(rng.integers(0, m, N)).cuda()
    A.load_states(rows, slots=start)
    B.load_states(rows, slots=start)
    rows0 = A.save_states().cpu().numpy()
    acts = _actions(A, K, rng)
    A.clear_stats(); B.clear_stats()
    n0 = A.launch_count
    oh, og, rew, done, info = A.step_k(torch.as_tensor(acts).cuda(), K, reset_pool=pool)
    groups = k_step_variant(preset, goals, N, pipeline, _sms())[2]
    assert A.launch_count - n0 == groups
    ga = dict(obs_h=_np(oh), obs_g=_np(og), rew=_np(rew), done=_np(done), final_h=_np(info["final_obs"]),
              final_g=_np(info["final_obs_grumpy"]), flags=_np(info["row_flags"]), slot=_np(info["reset_slot"]))
    ga["rows"] = A.save_states().cpu().numpy()
    stats_a = A.stats.cpu().numpy().copy()
    slot = ga["slot"]
    dn_all = ga["done"] != 0
    assert ((slot >= 0) == dn_all).all() and (slot < m).all()
    if w is not None:
        assert (w[slot[dn_all]] > 0).all()
    D = A.obs_dim
    for s in range(K):
        b = B.step_k(torch.as_tensor(acts[s:s + 1]).cuda(), 1, final_info=True)
        dn = dn_all[s]
        for key, got in (("rew", b[2]), ("done", b[3]), ("flags", b[4]["row_flags"])):
            assert _eq(ga[key][s], got[0].cpu().numpy()), (case, s, key)
        if D:
            for key, got in (("final_h", b[4]["final_obs"]), ("final_g", b[4]["final_obs_grumpy"])):
                assert _eq(ga[key][s][dn], got[0].cpu().numpy()[dn]), (case, s, key)
            for key, got in (("obs_h", b[0]), ("obs_g", b[1])):
                assert _eq(ga[key][s][~dn], got[0].cpu().numpy()[~dn]), (case, s, key)
        B.load_states(rows, slots=torch.as_tensor(slot[s].astype(np.int64)).cuda())
        if D:
            loaded = B.observe()
            for key, got in zip(("obs_h", "obs_g"), loaded):
                assert _eq(ga[key][s][dn], got.cpu().numpy()[dn]), (case, s, key)
    rb = B.save_states().cpu().numpy()
    ep = _episode_bytes(A)
    keep = np.ones(rb.shape[1], bool)
    keep[ep] = False
    assert np.array_equal(ga["rows"][:, keep], rb[:, keep])
    ep_a = ga["rows"][:, ep].copy().view(np.uint32)[:, 0]
    assert (ep_a == rows0[:, ep].copy().view(np.uint32)[:, 0] + dn_all.sum(0)).all()   # one increment per reset
    stats_b = B.stats.cpu().numpy()
    assert np.array_equal(stats_a[COUNTS], stats_b[COUNTS]), (stats_a, stats_b)
    assert np.allclose(stats_a[RET], stats_b[RET], rtol=1e-12, atol=1e-9)
    resets = int(dn_all.sum())
    print(f"{case}: {N} envs x {K} steps, {resets} pool resets ({resets / N:.2f} per env), "
          f"{np.unique(slot[dn_all]).size} distinct slots")
    assert resets > 2 * N
    _check_host_build(A, case, rows0, acts, ga, pool, n_host, f64)
    A.close(); B.close()


def _check_host_build(env, case, rows0, acts, ga, pool, n, f64):
    """Envs [0, n) of the launch against emul_pool.launch, in chunks of their own EmulBatch (env_offset shifted, so the
    draws and random resets are those of the GPU env): every row (atan columns at the parity bar), reset_slot and the
    final rows byte for byte."""
    from emul import emul_pool
    emul_pool.use_libm_sincos(False)
    rows = pool.rows.cpu().numpy()
    cdf = None if pool.cdf is None else pool.cdf.cpu().numpy()
    workers = max(1, os.cpu_count() or 1)
    bounds = [(n * j // (2 * workers), n * (j + 1) // (2 * workers)) for j in range(2 * workers)]
    f32, D = not f64, env.obs_dim
    atan = ATAN_COLS.get(env.cfg.observer, [])

    def chunk(b):
        from emul import emul, emul_states
        from roborugby_b200._lib import Config
        c0, c1 = b
        t = Tally()
        if c1 == c0:
            return t
        cfg = Config.from_buffer_copy(env.cfg)
        cfg.env_offset = env.cfg.env_offset + c0
        batch = emul.EmulBatch(cfg, c1 - c0, env.num_robots, env.num_balls, D)
        start = np.zeros((3 * env.num_robots + 2 * env.num_balls, c1 - c0))
        emul_states.load(batch, start, np.ascontiguousarray(rows0[c0:c1]))
        h = emul_pool.launch(batch, start, acts[:, c0:c1].astype(np.float64), rows, cdf, pool.p)
        g = {k: v[:, c0:c1] for k, v in ga.items() if k != "rows"}
        for key in ("rew", "done", "flags", "slot"):
            _compare_rows(t, key, g[key], h[key], f32, c0)
        if D:
            _compare_rows(t, "obs_h", g["obs_h"], h["obs_h"], f32, c0, atan)
            _compare_rows(t, "obs_g", g["obs_g"], h["obs_g"], f32, c0, atan)
            dn = h["done"] != 0
            for key in ("final_h", "final_g"):
                _compare_rows(t, key, g[key][dn][None], h[key][dn][None], f32, c0, atan)
        _compare_state(t, "state", ga["rows"][c0:c1], emul_states.save(batch, start), c0)
        return t

    t = Tally()
    with ThreadPoolExecutor(workers) as ex:   # ctypes releases the GIL
        for part in ex.map(chunk, bounds):
            t.merge(part)
    print(f"{case}: envs [0, {n}) against the host build: {sum(v for k, v in t.n.items() if k.endswith('.rows'))} rows, "
          f"{t.n.get('state.bytes', 0)} state bytes; {t.n.get('differences', 0)} differing")
    for f in t.first:
        print("  ", f)
    assert not t.first, t.first


def test_device_draws_follow_the_weights_and_p():
    """TRAIN, 65 536 envs that end every few steps: the device's reset_slot over all resets of a weighted pool passes a
    chi-square test against the weights and never names a zero-weight slot; with p = 0.5 half of the resets are pool
    resets."""
    from scipy.stats import chisquare
    from roborugby_b200.vec_env import ResetPool
    rng = np.random.default_rng(31)
    env = _env("TRAIN", 65536, 1, False, False, None)
    m = 40
    rows = _pool_rows(env, m, rng)
    w = rng.random(m) + 0.1
    w[[0, 5, 6, m - 1]] = 0.0
    pool = ResetPool(rows, w, p=1.0)
    counts = np.zeros(m, np.int64)
    env.load_states(rows, slots=torch.as_tensor(rng.integers(0, m, env.num_envs)).cuda())
    for _ in range(4):
        out = env.step_k(torch.as_tensor(_actions(env, 64, rng)).cuda(), 64, reset_pool=pool)
        s = out[4]["reset_slot"].cpu().numpy()
        d = out[3].cpu().numpy() != 0
        assert ((s >= 0) == d).all()
        counts += np.bincount(s[d], minlength=m)
    nz = w > 0
    pval = chisquare(counts[nz], w[nz] / w.sum() * counts.sum()).pvalue
    print(f"{counts.sum()} device resets, chi-square p = {pval:.3g}")
    assert counts.sum() >= 1_000_000 and (counts[~nz] == 0).all() and pval > 1e-3
    half = ResetPool(rows, p=0.5)
    out = env.step_k(torch.as_tensor(_actions(env, 64, rng)).cuda(), 64, reset_pool=half)
    s = out[4]["reset_slot"].cpu().numpy()
    d = out[3].cpu().numpy() != 0
    frac = (s[d] >= 0).mean()
    assert abs(frac - 0.5) < 5 * np.sqrt(0.25 / d.sum()), frac
    env.close()


@pytest.mark.parametrize("pool_p", [0.0, None])
def test_p_zero_and_no_pool_equal_step_info(pool_p):
    """p = 0 through the pool kernel, and a NULL pool through rr_step_pool, give rr_step_info's outputs bit for bit and
    reset_slot all -1."""
    from roborugby_b200 import _lib
    from roborugby_b200.vec_env import ResetPool
    rng = np.random.default_rng(32)
    N, K = 65536, 32
    A = _env("GAME", N, 128, False, False, None)
    B = _env("GAME", N, 128, False, False, None)
    rows = _pool_rows(A, 64, rng)
    st = torch.as_tensor(rng.integers(0, 64, N)).cuda()
    A.load_states(rows, slots=st); B.load_states(rows, slots=st)
    acts = torch.as_tensor(_actions(A, K, rng)).cuda()
    b = B.step_k(acts, K, final_info=True)
    if pool_p is not None:
        a = A.step_k(acts, K, reset_pool=ResetPool(rows, p=pool_p))
        slot = a[4]["reset_slot"]
    else:
        o = A._out(K); f = A._final_out(K)
        slot = torch.full((K, N), 7, dtype=torch.int32, device="cuda")
        _lib.check(A.lib.rr_step_pool(A._h, acts.data_ptr(), acts.shape[2], K, o["obs_h"].data_ptr(), o["obs_g"].data_ptr(),
                                      o["rew"].data_ptr(), o["done"].data_ptr(), f["final_obs_h"].data_ptr(),
                                      f["final_obs_g"].data_ptr(), f["row_flags"].data_ptr(), None, slot.data_ptr(),
                                      A._stream()))
        A.join()
        a = (o["obs_h"], o["obs_g"], o["rew"], o["done"], dict(final_obs=f["final_obs_h"], final_obs_grumpy=f["final_obs_g"],
                                                                row_flags=f["row_flags"]))
    assert (slot == -1).all()
    dn = b[3].bool()
    assert dn.any()
    for x, y in zip(a[:4], b[:4]):
        assert torch.equal(x, y)
    assert torch.equal(a[4]["row_flags"], b[4]["row_flags"])
    assert torch.equal(a[4]["final_obs"][dn], b[4]["final_obs"][dn])
    assert torch.equal(A.save_states(), B.save_states())
    sa, sb = A.stats.cpu().numpy(), B.stats.cpu().numpy()
    assert np.array_equal(sa[COUNTS], sb[COUNTS]) and np.allclose(sa[RET], sb[RET], rtol=1e-12, atol=1e-9)
    A.close(); B.close()


def test_refusals_launch_nothing():
    from roborugby_b200 import _lib
    from roborugby_b200.vec_env import ResetPool
    N = 256
    env = _env("TRAIN", N, 1, False, False, None)
    rows = env.save_states()
    cdf = torch.ones(N, dtype=torch.float64, device="cuda").cumsum(0)
    acts = torch.zeros(1, N, 1, dtype=torch.uint8, device="cuda")
    o = env._out(1)
    slot = torch.empty(2, N, dtype=torch.int32, device="cuda")
    lib = env.lib

    def call(pool, reset_slot=slot[0].data_ptr(), k=1, rew=o["rew"].data_ptr(), on=env):
        n0 = on.launch_count
        rc = lib.rr_step_pool(on._h, acts.data_ptr(), 1, k, None, None, rew, o["done"].data_ptr(), None, None, None,
                              None if pool is None else C.byref(pool), reset_slot, env._stream())
        assert on.launch_count == n0
        return rc, lib.rr_last_error().decode()

    P = lambda rows_p=rows.data_ptr(), m=N, cdf_p=cdf.data_ptr(), p=1.0: _lib.ResetPoolC(rows_p, m, cdf_p, p)
    bad = [(P(rows_p=None), "rows_dev"), (P(m=0), "m must"), (P(m=2 ** 31), "m must"), (P(rows_p=rows.data_ptr() + 8), "16-byte"),
           (P(cdf_p=cdf.data_ptr() + 4), "8-byte"), (P(p=-0.5), "p_pool"), (P(p=1.0000001), "p_pool"),
           (P(p=float("nan")), "p_pool")]
    for pool, msg in bad:
        rc, err = call(pool)
        assert rc == -1 and msg in err, (msg, err)
    rc, err = call(P(), reset_slot=slot.data_ptr() + 2)
    assert rc == -1 and "reset_slot" in err
    rc, err = call(P(), k=0)                                   # rr_step_info's own checks
    assert rc == -1 and "k_steps" in err
    rc, err = call(P(), rew=o["rew"].data_ptr() + 2)
    assert rc == -1 and "aligned" in err
    rc, err = call(None, k=0)
    assert rc == -1
    na = _env("TRAIN", N, 1, False, False, None, auto_reset=False)
    rc, err = call(P(), on=na)
    assert rc == -1 and "auto_reset" in err
    # Python
    with pytest.raises(ValueError):
        na.step_k(acts, 1, reset_pool=ResetPool(rows))
    game = _env("GAME", 64, 1, False, False, None)
    with pytest.raises(ValueError, match="bytes wide"):
        game.step_k(torch.zeros(1, 64, 4, dtype=torch.uint8, device="cuda"), 1, reset_pool=ResetPool(rows))
    with pytest.raises(ValueError):
        env.step_k(acts, 1, reset_pool=rows)
    with pytest.raises(ValueError):
        ResetPool(rows, weights=torch.zeros(N, device="cuda"))
    with pytest.raises(ValueError):
        ResetPool(rows[:, 8:])                                   # not contiguous
    # step(): [N] reset_slot
    obs, r, d, info = env.step(acts[0], reset_pool=ResetPool(rows))
    assert info["reset_slot"].shape == (N,) and info["reset_slot"].dtype == torch.int32
    for e in (env, na, game):
        e.close()
