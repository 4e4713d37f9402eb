"""Every reward-mixin class composition (RR_ScoreKeepers.py), on the CPU.

* The (reward_mask, reward_order) rule of rr_sim.cuh (rr_reward_config_error) accepts exactly the pairs that a class
  `class Env(*mixins, Observer, GameEnv_Simple)` with distinct mixins produces, and rr_create refuses the rest with a
  message naming the field, before it looks for a device.
* The host build of the kernel source (tests/emul) against the oracle for every valid composition, one step from
  injected states: golden contact-rich states, robots whose corners sit exactly on a goal triangle's edges and on the
  hypotenuse corner where Div0(0, 0) raises, and the same states with zero or undone continuous thrusts.
* Goal scoring x composition: the goal golden files' action sequences replayed under other compositions.
"""
import ctypes as C
import itertools
import multiprocessing
import os

import numpy as np
import pytest

from conftest import golden_files
from golden_util import actions_at, parse_name, state_at
from parity_util import compare_record
from roborugby_b200 import _lib
from roborugby_b200.constants import REWARD_MIXINS, reward_config_from_mixins

NAMES = list(REWARD_MIXINS)
CHASE, PUSHPOS, NAUGHTY, DONTDRIVE, KEEPMOVING, BASEDESTR, PUSHNEG = NAMES
LISTS = [l for n in range(len(NAMES) + 1) for l in itertools.permutations(NAMES, n)]
VALID = sorted({reward_config_from_mixins(l) for l in LISTS})
VALID_KEYS = np.array([(m << 32) | o for m, o in VALID], np.uint64)
DIV0 = 128


def _expected_valid(mask, order):
    mask = np.asarray(mask, np.uint64); order = np.asarray(order, np.uint64)
    return ((order == 0) & (mask <= 127)) | np.isin((mask << np.uint64(32)) | order, VALID_KEYS)


# ------------------------------------------------------------------ the rule


def test_class_compositions_give_7253_pairs():
    assert len(LISTS) == 13700
    assert len(VALID) == 7253 and (0, 0) in VALID
    assert sum(o != 0 for _, o in VALID) == 7252


def test_rule_accepts_exactly_the_class_compositions():
    from emul import emul
    m = np.array([v[0] for v in VALID]); o = np.array([v[1] for v in VALID])
    assert emul.reward_config_valid(m, o).all()
    # every mask 0..255 with every order of up to 3 nibbles
    mm, oo = np.meshgrid(np.arange(256), np.arange(4096), indexing="ij")
    mm, oo = mm.ravel(), oo.ravel()
    got = emul.reward_config_valid(mm, oo)
    assert np.array_equal(got, _expected_valid(mm, oo))
    assert got[oo == 0].sum() == 128 and np.array_equal(np.nonzero(got[oo == 0])[0], np.arange(128))
    # seeded random full 32-bit orders, and the valid pairs with one nibble or one mask bit changed
    rng = np.random.default_rng(20261020)
    rm = rng.integers(0, 256, 200000); ro = rng.integers(0, 2 ** 32, 200000, dtype=np.uint64)
    k = rng.integers(0, len(VALID), 100000)
    sh = (4 * rng.integers(0, 8, k.size)).astype(np.uint64)
    mo = (o[k].astype(np.uint64) & ~(np.uint64(15) << sh)) | (rng.integers(0, 16, k.size).astype(np.uint64) << sh)
    mb = m[k] ^ (1 << rng.integers(0, 8, k.size))
    am = np.concatenate([rm, m[k], mb]); ao = np.concatenate([ro, mo, o[k].astype(np.uint64)])
    assert np.array_equal(emul.reward_config_valid(am, ao), _expected_valid(am, ao))
    # the C ABI's own check agrees on the valid pairs
    lib = _lib.load()
    cfg = _lib.default_config(_lib.PRESET_GAME, "RoboRugbySimpleDuel-v2")
    for mask, order in VALID:
        cfg.reward_mask, cfg.reward_order = mask, order
        assert lib.rr_check_config(C.byref(cfg)) == 0, (mask, order, lib.rr_last_error())


def test_repeated_mixin_is_refused():
    with pytest.raises(ValueError, match="twice"):
        reward_config_from_mixins([CHASE, CHASE])
    with pytest.raises(ValueError, match="twice"):
        reward_config_from_mixins([NAUGHTY, KEEPMOVING, CHASE, KEEPMOVING])


BAD_CONFIGS = [
    # (field overrides, substring of the message)
    (dict(reward_mask=1, reward_order=0x2), "reward_mask bit is clear"),      # PushPos body without its snapshot
    (dict(reward_mask=0, reward_order=0x5), "reward_mask bit is clear"),      # KeepMoving without its mask bit
    (dict(reward_mask=7, reward_order=0x8), "not an RR_MIX_* id"),
    (dict(reward_mask=7, reward_order=0x9213), "not an RR_MIX_* id"),
    (dict(reward_mask=7, reward_order=0x2213), "twice"),
    (dict(reward_mask=7, reward_order=0x2013), "after its terminating"),
    (dict(reward_mask=7, reward_order=0x10000003), "after its terminating"),
    (dict(reward_mask=7, reward_order=0x231), "must start with RR_MIX_NAUGHTY"),
    (dict(reward_mask=7, reward_order=0x21), "must start with RR_MIX_NAUGHTY"),
    (dict(reward_mask=3, reward_order=0x1), "every mixin of reward_mask"),
    (dict(reward_mask=0x80, reward_order=0), "bits above RR_REW_PUSHNEG"),
    (dict(reward_mask=0xFFFFFFFF, reward_order=0), "bits above RR_REW_PUSHNEG"),
] + [(dict(**{f: v}), f) for f in ("discrete", "time_limit", "auto_reset", "out_f64", "strict_reset", "goal_scoring")
     for v in (2, -1)] + [
    (dict(flags=2), "flags"), (dict(flags=0x80000000), "flags"), (dict(env_offset=-1), "env_offset"),
]


@pytest.mark.parametrize("over,why", BAD_CONFIGS, ids=[f"{i}-{w.split()[0]}" for i, (_, w) in enumerate(BAD_CONFIGS)])
def test_rr_create_refuses_bad_configs(over, why):
    """Refused with RR_E_INVALID and a message naming the field, before the device check (so on any box)."""
    lib = _lib.load()
    cfg = _lib.default_config(_lib.PRESET_GAME, "RoboRugbySimpleDuel-v2")
    for k, v in over.items():
        setattr(cfg, k, v)
    h = C.c_void_p()
    assert lib.rr_create(C.byref(cfg), 8, 0, C.byref(h)) == -1 and not h.value
    msg = lib.rr_last_error().decode()
    assert why in msg and "CUDA" not in msg, msg
    assert lib.rr_check_config(C.byref(cfg)) == -1 and why in lib.rr_last_error().decode()


@pytest.mark.parametrize("kw", [dict(reward_mask=1, reward_order=0x2), dict(reward_order=0x8), dict(reward_order=0x2213),
                                dict(reward_mask=0, reward_order=0x5), dict(reward_mixins=[CHASE, CHASE]),
                                dict(flags=2), dict(env_offset=-1)], ids=str)
def test_vec_env_refuses_bad_configs(kw):
    """RoboRugbyVecEnv raises ValueError before it needs a device."""
    import roborugby_b200
    with pytest.raises(ValueError):
        roborugby_b200.RoboRugbyVecEnv("RoboRugbySimpleDuel-v2", 8, **kw)


# ------------------------------------------------------------------ states

FIELD = {"GAME": 800.0, "TRAIN": 600.0}


def _robot(cx, cy, rot):
    hw, hh = (10.0, 20.0) if rot == 0 else (20.0, 10.0)   # ROBOT_LENGTH 20 x ROBOT_WIDTH 40
    return [cx, cy, cx - hw, cx + hw, cy - hh, cy + hh, float(rot)]


def _ball(cx, cy, vx=0.0, vy=0.0):
    return [cx, cy, cx - 7.0, cx + 7.0, cy - 7.0, cy + 7.0, vx, vy]


def _goal_features(W, rot):
    """Robot poses (integer centres) whose corners land exactly on the goal triangles' edges.  Happy goal: the
    bottom-right triangle with hypotenuse x + y = 2W - 240 and Div0 corner (W - 240, W); grumpy goal: the top-left one
    with hypotenuse x + y = 240 and Div0 corner (240, 0)."""
    if rot == 0:   # corners at (+-10, +-20)
        return dict(h_edge=(W - 10, W - 100), h_hyp=(W - 100, W - 110), h_div0=(W - 230, W - 20), h_miss=(W - 100, W - 111),
                    g_edge=(10, 100), g_hyp=(100, 110), g_div0=(230, 20), g_miss=(100, 109))
    return dict(h_edge=(W - 20, W - 100), h_hyp=(W - 100, W - 110), h_div0=(W - 220, W - 10), h_miss=(W - 101, W - 110),
                g_edge=(20, 100), g_hyp=(100, 110), g_div0=(220, 10), g_miss=(99, 110))


def _edge_states(preset):
    W = FIELD[preset]
    R, B = (4, 8) if preset == "GAME" else (1, 1)
    out = []
    for rot in (0, 90):
        f = _goal_features(W, rot)
        if R == 4:
            layouts = [("h_hyp", "h_edge", "g_hyp", "g_edge"), ("g_hyp", "g_edge", "h_hyp", "h_edge"),
                       ("h_div0", None, "g_miss", None), (None, "g_div0", None, "h_miss"), ("h_miss", "g_miss", None, None)]
        else:
            layouts = [(k,) for k in f]
        for lay in layouts:
            rob = [_robot(*(f[k] if k else (W / 2 - 150 + 100 * r, W / 2)), rot) for r, k in enumerate(lay)]
            ball = [_ball(W / 2 - 140 + 40 * b, W / 2 + 60, 0.0 if b % 2 else 0.75, 0.5 if b % 3 == 0 else 0.0) for b in range(B)]
            out.append(dict(rob=np.array(rob), rhist=np.zeros((R, 3)), rflag=np.zeros((R, 3), np.int32),
                            ball=np.array(ball), step=np.int32(10)))
    return out


def _golden_pool(preset, continuous):
    """(state, actions) records the reference completed, contact-rich ones (naughty robots, moving balls) first."""
    recs = []
    for p in golden_files(f"{preset}_*.npz"):
        _, env_id, kind = parse_name(p)
        if kind not in ("chase", "inject", "random", "partial", "sticky") or (env_id == "RoboRugby-v0") != continuous:
            continue
        d = dict(np.load(p))
        n, T = d["act"].shape[:2]
        for i in range(n):
            for t in range(0, T, max(1, T // 8)):
                if d["exc"][i, t]:
                    continue
                st = state_at(d, i, t)
                rank = 0 if d["naughty"][i, t] else (1 if np.any(st["ball"][:, 6:] != 0) else 2)
                recs.append((rank, len(recs), st, actions_at(d, i, t)))
    recs.sort(key=lambda r: r[:2])
    return [(r[2], r[3]) for r in recs]


def _state_set(preset, rich):
    """[(state, actions, discrete)]: rich = at least 256 records, else 8."""
    R = 4 if preset == "GAME" else 1
    rng = np.random.default_rng(5 if preset == "GAME" else 6)
    edges = _edge_states(preset)
    zero, fwd, back, turn = [0.0] * 2 * R, [1.0] * 2 * R, [-1.0] * 2 * R, [1.0, -1.0] * R
    disc, cont = _golden_pool(preset, False), _golden_pool(preset, True)
    if not rich:
        return [(disc[0][0], disc[0][1], True), (disc[1][0], disc[1][1], True), (disc[-1][0], disc[-1][1], True),
                (edges[0], rng.integers(0, 8, R).astype(float), True), (edges[0], zero, False),
                (edges[2], zero, False), (edges[-1], fwd, False), (cont[0][0], cont[0][1], False)]
    out = []
    for st in edges:
        out += [(st, rng.integers(0, 8, R).astype(float), True), (st, rng.integers(0, 8, R).astype(float), True),
                (st, zero, False), (st, fwd, False), (st, back, False), (st, turn, False)]
        gs = dict(st); gs["rflag"] = st["rflag"].copy(); gs["rflag"][:, :2] = 1   # a stored thrust no action replaces
        out.append((gs, [], True))
    for st, a in cont[:32]:
        out += [(st, a, False), (st, zero, False)]
    out += [(st, a, True) for st, a in disc[:max(0, 256 - len(out))]]
    assert len(out) >= 256
    return out


# ------------------------------------------------------------------ host build vs oracle, per composition

_STATES = {}


def _configs(oracle, preset, mask, order, discrete, goals=False):
    env_id = "RoboRugbySimpleDuel-v2" if discrete else "RoboRugby-v0"
    cfg = _lib.default_config(_lib.PRESET_GAME if preset == "GAME" else _lib.PRESET_TRAIN, env_id)
    cfg.time_limit = 0; cfg.auto_reset = 0; cfg.strict_reset = 1
    cfg.reward_mask, cfg.reward_order, cfg.goal_scoring = mask, order, int(goals)
    ocfg = oracle.default_config(preset, env_id)
    ocfg.reward_mask, ocfg.reward_order, ocfg.goal_scoring = mask, order, int(goals)
    return cfg, ocfg


def _sweep(args):
    """Host build (glibc and GPU sin/cos) vs oracle for compositions x states; returns counts and the first failures."""
    preset, states, comps = args
    from emul import emul
    from oracle import rr_oracle as oracle
    oracle.scratch_mode(1)
    res = dict(records=0, exact=dict(libm=0, dd=0), bad=[], nonzero=0, div0=0)
    for mask, order in comps:
        envs = {}
        for disc in (True, False):
            cfg, ocfg = _configs(oracle, preset, mask, order, disc)
            o = oracle.OracleEnv(cfg=ocfg)
            envs[disc] = (cfg, o, emul.EmulEnv(cfg, o.R, o.B, o.obs_dim))
        for j, (st, a, disc) in enumerate(states):
            cfg, o, e = envs[disc]
            o.set_state(st)
            want = o.step(a)
            ws = o.get_state()
            res["records"] += 1
            res["nonzero"] += bool(want["err"] == 0 and np.any(want["rew"] != 0))
            res["div0"] += bool(want["err"] & DIV0)
            for trig in ("libm", "dd"):
                emul.use_libm_sincos(trig == "libm")
                e.set_state(st)
                got = e.step(a)
                if got["err"] != want["err"]:
                    res["bad"].append((mask, order, j, trig, f"err {got['err']} != {want['err']}"))
                    continue
                if want["err"]:
                    res["exact"][trig] += 1
                    continue
                ok, ex, w, why = compare_record(e.get_state(), got, ws, want)
                res["exact"][trig] += ex
                if not ok:
                    res["bad"].append((mask, order, j, trig, why, w, got["rew"].tolist(), want["rew"].tolist()))
        res["bad"] = res["bad"][:5]
    emul.use_libm_sincos(False)
    oracle.scratch_mode(0)
    return res


def _run_sweep(oracle, preset, comps, rich):
    from emul import emul
    emul.lib()
    key = (preset, rich)
    if key not in _STATES:
        _STATES[key] = _state_set(preset, rich)
    states = _STATES[key]
    n = max(1, min(len(os.sched_getaffinity(0)), 16))
    chunks = [(preset, states, comps[i::n]) for i in range(n)]
    with multiprocessing.get_context("spawn").Pool(n) as pool:   # (spawn: the parent may run threads by now)
        parts = pool.map(_sweep, chunks)
    tot = dict(records=sum(p["records"] for p in parts), bad=[b for p in parts for b in p["bad"]],
               exact={t: sum(p["exact"][t] for p in parts) for t in ("libm", "dd")},
               nonzero=sum(p["nonzero"] for p in parts), div0=sum(p["div0"] for p in parts))
    print(f"{preset} {len(comps)} compositions x {len(states)} states: {tot['records']} records, bit-identical "
          f"{tot['exact']['libm']} (glibc sin/cos) / {tot['exact']['dd']} (GPU sin/cos); {tot['nonzero']} with a "
          f"non-zero reward, {tot['div0']} raising Div0")
    assert not tot["bad"], tot["bad"][:5]
    for t in ("libm", "dd"):
        assert tot["exact"][t] >= 0.6 * tot["records"], (t, tot["exact"][t], tot["records"])
    return tot


@pytest.mark.parametrize("preset", ["GAME", "TRAIN"])
def test_every_valid_composition_matches_oracle(oracle, preset):
    """All 7 253 (mask, order) pairs, 8 states each."""
    _run_sweep(oracle, preset, VALID, rich=False)


def _structured_compositions():
    comps = {(m, 0) for m in range(128)}                                              # every mask, canonical order
    six = [n for n in NAMES if n != NAUGHTY]
    comps |= {reward_config_from_mixins(p) for p in itertools.permutations(six)}      # 720 orders without NaughtyBots
    for i in range(7):                                                                # NaughtyBots at each position
        comps.add(reward_config_from_mixins(six[:i] + [NAUGHTY] + six[i:]))
    return sorted(comps)


@pytest.mark.parametrize("preset", ["GAME", "TRAIN"])
def test_structured_compositions_match_oracle_on_rich_states(oracle, preset):
    comps = _structured_compositions()
    assert len(comps) == 128 + 720 + 7
    _run_sweep(oracle, preset, comps, rich=True)


@pytest.mark.parametrize("preset", ["GAME", "TRAIN"])
def test_rich_states_make_every_term_non_zero(oracle, preset):
    """Each mixin alone pays something on some state of the rich set, and Div0(0, 0) of DontDriveInGoals raises on
    some state (in the host build too)."""
    from emul import emul
    states = _state_set(preset, True)
    oracle.scratch_mode(1)
    try:
        # (with one robot, TRAIN has no robot pair whose collision makes a robot naughty)
        for name in (CHASE, PUSHPOS, DONTDRIVE, KEEPMOVING, PUSHNEG) + ((NAUGHTY,) if preset == "GAME" else ()):
            mask, order = reward_config_from_mixins([name])
            nonzero = div0 = 0
            for disc in (True, False):
                cfg, ocfg = _configs(oracle, preset, mask, order, disc)
                o = oracle.OracleEnv(cfg=ocfg)
                e = emul.EmulEnv(cfg, o.R, o.B, o.obs_dim)
                for st, a, d in states:
                    if d != disc:
                        continue
                    o.set_state(st)
                    w = o.step(a)
                    nonzero += w["err"] == 0 and np.any(w["rew"] != 0)
                    if w["err"] & DIV0:
                        e.set_state(st)
                        div0 += bool(e.step(a)["err"] & DIV0)
            assert nonzero > 0, name
            if name == DONTDRIVE:
                assert div0 > 0
    finally:
        oracle.scratch_mode(0)


# ------------------------------------------------------------------ goal scoring x composition

GOAL_COMPS = [[], [NAUGHTY], [PUSHPOS, CHASE, NAUGHTY], [BASEDESTR, CHASE, NAUGHTY, PUSHPOS],
              [BASEDESTR], [BASEDESTR, PUSHPOS, CHASE], [PUSHPOS, BASEDESTR, CHASE], [CHASE, PUSHPOS, BASEDESTR],
              [KEEPMOVING, BASEDESTR, DONTDRIVE, PUSHNEG], [PUSHNEG, PUSHPOS, CHASE, BASEDESTR, KEEPMOVING, DONTDRIVE]]
GOALS = golden_files("*_goals_*.npz")


@pytest.mark.parametrize("mixins", GOAL_COMPS, ids=lambda m: "-".join(x[:6] for x in m) or "none")
@pytest.mark.parametrize("path", GOALS, ids=[p.split("/")[-1] for p in GOALS])
def test_goal_scoring_under_every_composition(oracle, path, mixins):
    """The goal files' action sequences with goal scoring on, host build (glibc sin/cos) vs oracle, step by step: every
    reward (the +-500 of a scored ball, BaseDestruction's 1.604 M points when a goal falls), done, the refused step
    after the end.  With NaughtyBots no ball may ever score."""
    from emul import emul
    from emul.emul import EmulEnv
    preset, env_id, _ = parse_name(path)
    d = dict(np.load(path))
    n, T = d["act"].shape[:2]
    mask, order = reward_config_from_mixins(mixins)
    cfg, ocfg = _configs(oracle, preset, mask, order, env_id != "RoboRugby-v0", goals=True)
    emul.use_libm_sincos(True)
    oracle.scratch_mode(1)
    dropped = destroyed = scored = 0
    try:
        for i in range(n):
            o = oracle.OracleEnv(cfg=ocfg)
            e = EmulEnv(cfg, o.R, o.B, o.obs_dim)
            o.set_state(state_at(d, i, 0)); e.set_state(state_at(d, i, 0))
            r = e.goal_rollout(d["act"][i])
            for t in range(T):
                w = o.step(actions_at(d, i, t))
                if w["err"]:   # the game was over: refused by both, with nothing paid
                    assert r["steps"] == t and r["err"] == w["err"] == 1, (i, t, r["err"], w["err"])
                    break
                assert t < r["steps"], (i, t, r["err"])
                if not np.allclose(r["rew"][t], w["rew"], rtol=1e-9, atol=1e-9):
                    dropped += 1   # a last-bit contact difference has grown (DESIGN.md §2): stop comparing it here
                    break
                assert int(r["done"][t]) == w["done"], (i, t)
                g = o.goal_state()
                assert r["alive"][t] == sum(int(v) << b for b, v in enumerate(g["alive"])), (i, t)
                destroyed += int(abs(w["rew"][0]) > 1e6)   # (500 + 200000) * 8 balls
                scored += int(g["delta"] != 0)
                if NAUGHTY in mixins:
                    assert g["alive"].all() and g["delta"] == 0, (i, t)
        print(f"{path.split('/')[-1]} {mixins}: {n} trajectories, {dropped} dropped, {scored} scoring steps, "
              f"{destroyed} goal-destruction payouts")
        assert dropped <= n // 2
        if BASEDESTR in mixins and NAUGHTY not in mixins and preset == "GAME" and "SimpleDuel" not in path:
            assert destroyed > 0
    finally:
        emul.use_libm_sincos(False)
        oracle.scratch_mode(0)
