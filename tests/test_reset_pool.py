"""CPU tier: auto-reset from a reset pool (rr_step_pool, include/rr_b200.h) through the host build of the kernel source
(tests/emul emul_pool: rr_sim.cuh pool_draw / pool_reset on EmulBatch columns plus a start array).

The draw is restated here in numpy (Philox4x32-10, key = seed, counter = (global env, episode, 0xFFFFFFFF); u0 decides
pool or random, u1 picks the slot) and must agree with the host build's draw on every one of 10^6 pairs.  The drawn slots
follow the weights (chi-square), never hit a zero-weight slot, take the pool with probability p, and do not depend on
how a batch is split with env_offset.  A pool launch is the composition of the merged primitives: stepping one env-step
at a time with rr_step_info's launch and loading the drawn rows after each step (rr_load_states) gives the same rows,
statistics and final state, except the episode counter, which a pool reset keeps instead of taking the row's."""
import ctypes as C

import numpy as np
import pytest

from test_state_rows import _same, actions, batch, make_cfg

M32 = np.uint64(0xFFFFFFFF)


# ------------------------------------------------------------------------------------------ the draw, restated

def philox4x32_10(seed, c0, c1, c2, c3):
    """Philox4x32-10 (rr_sim.cuh Philox::block) over arrays of counters -> 4 uint64 arrays holding 32-bit words."""
    a, b, c, d = (np.asarray(x, np.uint64) & M32 for x in (c0, c1, c2, c3))
    k0, k1 = np.uint64(seed & 0xFFFFFFFF), np.uint64((seed >> 32) & 0xFFFFFFFF)
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * a
        p1 = np.uint64(0xCD9E8D57) * c
        a, b, c, d = (p1 >> np.uint64(32)) ^ b ^ k0, p1 & M32, (p0 >> np.uint64(32)) ^ d ^ k1, p0 & M32
        k0 = (k0 + np.uint64(0x9E3779B9)) & M32
        k1 = (k1 + np.uint64(0xBB67AE85)) & M32
    return a, b, c, d


def ref_draw(seed, env, episode, m, cdf=None, p=1.0):
    """include/rr_b200.h rr_step_pool step 2: the slot of each (global env, new episode counter), or -1 (random)."""
    env = np.asarray(env, np.uint64)
    w0, w1, w2, w3 = philox4x32_10(seed, env & M32, env >> np.uint64(32), episode, 0xFFFFFFFF)
    u = lambda hi, lo: ((hi << np.uint64(32) | lo) >> np.uint64(11)).astype(np.float64) * 2.0 ** -53
    u0, u1 = u(w0, w1), u(w2, w3)
    if cdf is None:
        slot = np.minimum(np.floor(u1 * m), m - 1).astype(np.int64)
    else:
        cdf = np.asarray(cdf, np.float64)
        slot = np.minimum(np.searchsorted(cdf, u1 * cdf[-1], side="right"), m - 1).astype(np.int64)
    return np.where(u0 < p, slot, -1)


def _pairs(n, rng):
    env = np.concatenate([rng.integers(0, 2 ** 40, n // 2, dtype=np.uint64), np.arange(n - n // 2, dtype=np.uint64)])
    ep = rng.integers(0, 2 ** 32, n, dtype=np.uint64).astype(np.uint32)
    return env, ep


def test_host_build_draw_equals_the_restated_draw():
    from emul import emul_pool
    rng = np.random.default_rng(1)
    env, ep = _pairs(1_000_000, rng)
    w = rng.random(37) * (rng.random(37) < 0.7)
    cdf = np.cumsum(w)
    for seed, m, c, p in ((2026, 37, cdf, 1.0), (7, 37, None, 0.3), (2 ** 63 + 5, 1, None, 1.0), (0, 1000, None, 0.999)):
        got = emul_pool.draw(seed, env, ep, m, c, p)
        assert np.array_equal(got, ref_draw(seed, env, ep, m, c, p)), (seed, m, p)


def test_weighted_draw_follows_the_weights_and_never_draws_a_zero_weight_slot():
    from scipy.stats import chisquare
    from emul import emul_pool
    rng = np.random.default_rng(2)
    m = 50
    w = rng.random(m) + 0.05
    w[[0, 7, 8, 31, m - 1]] = 0.0                          # zero weights at both ends and in a run
    n = 1_000_000
    env, ep = _pairs(n, rng)
    slot = emul_pool.draw(99, env, ep, m, np.cumsum(w), 1.0)
    assert (slot >= 0).all() and (slot < m).all()
    counts = np.bincount(slot, minlength=m)
    assert (counts[w == 0] == 0).all(), counts[w == 0]
    nz = w > 0
    pval = chisquare(counts[nz], w[nz] / w.sum() * n).pvalue
    print(f"chi-square over {nz.sum()} slots, {n} draws: p = {pval:.3g}")
    assert pval > 1e-3
    # uniform
    slot = emul_pool.draw(5, env, ep, m)
    assert chisquare(np.bincount(slot, minlength=m)).pvalue > 1e-3


def test_pool_fraction_matches_p():
    from emul import emul_pool
    rng = np.random.default_rng(3)
    n = 1_000_000
    env, ep = _pairs(n, rng)
    assert (emul_pool.draw(11, env, ep, 9, None, 0.0) == -1).all()
    assert (emul_pool.draw(11, env, ep, 9, None, 1.0) >= 0).all()
    for p in (0.05, 0.5, 0.9):
        frac = (emul_pool.draw(11, env, ep, 9, None, p) >= 0).mean()
        sigma = np.sqrt(p * (1 - p) / n)
        assert abs(frac - p) < 5 * sigma, (p, frac)


def test_malformed_cdf_never_leaves_the_pool():
    from emul import emul_pool
    rng = np.random.default_rng(4)
    env, ep = _pairs(20_000, rng)
    for cdf in (np.array([3.0, 1.0, 2.0, 0.5]), np.array([np.nan, 1.0, np.nan, 2.0]), np.array([0.0, 0.0, 0.0, -1.0]),
                np.array([np.inf, np.inf, np.inf, np.inf]), np.array([-np.inf, 5.0, 1.0, np.nan])):
        slot = emul_pool.draw(1, env, ep, 4, cdf, 1.0)
        assert ((slot >= 0) & (slot < 4)).all(), cdf


# ------------------------------------------------------------------------------------------ launches

def _pool_rows(cfg, R, B, rng, m, before_end=3):
    """m rows saved from envs a few steps before the time limit, so that envs reset from them end again soon."""
    from emul import emul_states
    src = batch(cfg, m)
    T = 4500 if cfg.preset == 0 else 300
    for i in range(m):
        st = src.get_state(i)
        st["step"] = np.int32(T - before_end - 2 - (i % 4))
        src.set_state(i, st)
    src.launch(actions(rng, src, 2))
    start = rng.normal(size=(3 * R + 2 * B, m)) * 100.0
    return emul_states.save(src, start)


def _setup(layout, M, m, seed):
    from emul import emul_states
    rng = np.random.default_rng(seed)
    cfg = make_cfg(*layout)
    a = batch(cfg, M)
    start = rng.normal(size=(3 * a.R + 2 * a.B, M)) * 100.0
    rows = _pool_rows(cfg, a.R, a.B, rng, m)
    # begin from pool rows too (so that most envs end within a few steps)
    emul_states.load(a, start, rows, rng.integers(0, m, M))
    return rng, cfg, a, start, rows


def _episode_bytes(b):
    """Byte range of the episode counter in a saved row (rr_sim.cuh RowLayout: sf, start, then si columns)."""
    off = 8 * (b.sf.shape[0] + 3 * b.R + 2 * b.B) + 4 * b._episode_row
    return slice(off, off + 4)


@pytest.mark.parametrize("layout", [("TRAIN", False, False), ("TRAIN", True, True), ("GAME", False, False),
                                    ("GAME", True, False)])
def test_pool_launch_is_step_info_then_load_states(layout):
    """A: one K-step pool launch (p = 1, weighted).  B: the same actions one env-step at a time through rr_step_info's
    launch, then the rows A's resets drew loaded (emul_states.load).  Every row is the same; done rows' obs are the
    loaded state's; final rows are byte-equal except the episode counter; the statistics agree."""
    from emul import emul, emul_info, emul_pool, emul_states
    M, m, K = (24, 5, 24) if layout[0] == "TRAIN" else (6, 3, 10)
    rng, cfg, a, start_a, rows = _setup(layout, M, m, 21)
    w = np.array([1.0, 0.0, 2.0, 0.5, 3.0][:m])
    b = batch(cfg, M)
    b.sf[...] = a.sf; b.si[...] = a.si
    start_b = start_a.copy()
    acts = actions(rng, a, K)
    ga = emul_pool.launch(a, start_a, acts, rows, np.cumsum(w), 1.0)
    resets = 0
    stats_b = np.zeros(8)
    for s in range(K):
        hb = emul_info.launch(b, acts[s:s + 1], observe=True)
        stats_b += hb["stats"].sum(0)
        for key in ("rew", "done", "err", "naughty", "flags"):
            assert _same(ga[key][s], hb[key][0]), (s, key)
        slots = ga["slot"][s]
        dn = hb["done"][0] != 0
        assert ((slots >= 0) == dn).all() and (w[slots[dn]] > 0).all()
        if a.obs_dim:
            assert _same(ga["final_h"][s][dn], hb["final_h"][0][dn]) and _same(ga["final_g"][s][dn], hb["final_g"][0][dn])
            assert _same(ga["obs_h"][s][~dn], hb["obs_h"][0][~dn]) and _same(ga["obs_g"][s][~dn], hb["obs_g"][0][~dn])
        emul_states.load(b, start_b, rows, slots.astype(np.int64))
        for i in np.nonzero(dn)[0]:     # the done row's observation is the loaded state's
            if a.obs_dim and cfg.observer == 1 and not cfg.goal_scoring:
                e = emul.EmulEnv(cfg, a.R, a.B, a.obs_dim)
                e.set_state(b.get_state(i))
                assert _same(ga["obs_h"][s][i], e.observe(1)), (s, i)
        resets += int(dn.sum())
    ra, rb = emul_states.save(a, start_a), emul_states.save(b, start_b)
    ep = _episode_bytes(a)
    keep = np.ones(ra.shape[1], bool); keep[ep] = False
    assert np.array_equal(ra[:, keep], rb[:, keep])
    counts = [0, 3, 4, 5, 6]
    sa = ga["stats"].sum(0)
    assert np.array_equal(sa[counts], stats_b[counts]) and np.allclose(sa[[1, 2]], stats_b[[1, 2]], rtol=1e-12, atol=1e-9)
    print(f"{layout}: {M} envs x {K} steps, {resets} pool resets")
    assert resets >= 2 * M                                  # most envs reset several times within the launch


@pytest.mark.parametrize("layout", [("TRAIN", False, False), ("GAME", True, True)])
def test_pool_with_p_zero_is_step_info(layout):
    from emul import emul_info, emul_pool
    M, m, K = (16, 4, 20) if layout[0] == "TRAIN" else (5, 3, 8)
    rng, cfg, a, start_a, rows = _setup(layout, M, m, 22)
    b = batch(cfg, M)
    b.sf[...] = a.sf; b.si[...] = a.si
    start_b = start_a.copy()
    acts = actions(rng, a, K)
    ga = emul_pool.launch(a, start_a, acts, rows, None, 0.0)
    hb = emul_info.launch(b, acts, observe=True)
    assert (ga["slot"] == -1).all() and ga["done"].any()
    for key in ("rew", "done", "err", "naughty", "flags", "obs_h", "obs_g", "final_h", "final_g", "stats"):
        assert _same(ga[key], hb[key]), key
    assert _same(a.sf, b.sf) and _same(a.si, b.si) and _same(start_a, start_b)


def test_slots_do_not_depend_on_how_the_batch_is_split():
    """The same envs as one batch (env_offset o) and as two (o, o + M1): the same slots, rows and final state."""
    from emul import emul_pool, emul_states
    from roborugby_b200._lib import Config
    rng, cfg, a, start_a, rows = _setup(("TRAIN", False, False), 20, 6, 23)
    rows0 = emul_states.save(a, start_a)
    acts = actions(rng, a, 30)
    w = np.arange(6, dtype=np.float64)
    whole = emul_pool.launch(a, start_a, acts, rows, np.cumsum(w), 0.7)
    M1 = 7
    for lo, hi in ((0, M1), (M1, 20)):
        c = Config.from_buffer_copy(cfg)
        c.env_offset = cfg.env_offset + lo
        part = batch(c, hi - lo)
        st = np.zeros((3 * part.R + 2 * part.B, hi - lo))
        emul_states.load(part, st, np.ascontiguousarray(rows0[lo:hi]))
        g = emul_pool.launch(part, st, np.ascontiguousarray(acts[:, lo:hi]), rows, np.cumsum(w), 0.7)
        for key in ("slot", "rew", "done", "obs_h", "flags"):
            assert _same(g[key], np.ascontiguousarray(whole[key][:, lo:hi])), (lo, key)
        assert np.array_equal(emul_states.save(part, st), rows_now(a, start_a)[lo:hi])
    assert (whole["slot"] >= 0).any() and ((whole["slot"] == -1) & (whole["done"] != 0)).any()
    assert not (whole["slot"] == 0).any()                  # weight 0


def rows_now(b, start):
    from emul import emul_states
    return emul_states.save(b, start)


# ------------------------------------------------------------------------------------------ argument checks

def test_reset_pool_refuses_bad_arguments():
    import torch
    from roborugby_b200.vec_env import ResetPool
    rows = torch.zeros(4, 224, dtype=torch.uint8)
    bad = [
        dict(rows=np.zeros((4, 224), np.uint8)),                 # not a tensor
        dict(rows=torch.zeros(4, 224, dtype=torch.int8)),        # dtype
        dict(rows=torch.zeros(4 * 224, dtype=torch.uint8)),      # not [m, S]
        dict(rows=torch.zeros(0, 224, dtype=torch.uint8)),       # m = 0
        dict(rows=rows, p=1.5), dict(rows=rows, p=-0.1), dict(rows=rows, p=float("nan")),
        dict(rows=rows, weights=[1.0, 2.0, 3.0]),                # shape
        dict(rows=rows, weights=torch.ones(4, 1)),
        dict(rows=rows, weights=[1.0, -1.0, 2.0, 0.0]),          # negative
        dict(rows=rows, weights=[1.0, float("nan"), 2.0, 0.0]),  # NaN
        dict(rows=rows, weights=[1.0, float("inf"), 2.0, 0.0]),  # infinite
        dict(rows=rows, weights=[0.0, 0.0, 0.0, 0.0]),           # zero sum
        dict(rows=rows, weights=torch.ones(4, dtype=torch.bool)),
        dict(rows=rows),                                         # not on a CUDA device
    ]
    for kw in bad:
        with pytest.raises(ValueError):
            ResetPool(**kw)


def test_rr_step_pool_refuses_a_null_handle():
    from roborugby_b200 import _lib
    lib = _lib.load()
    pool = _lib.ResetPoolC(None, 1, None, 1.0)
    assert lib.rr_step_pool(None, None, 0, 1, None, None, None, None, None, None, None, C.byref(pool), None, None) == -1
    assert b"null handle" in lib.rr_last_error()
