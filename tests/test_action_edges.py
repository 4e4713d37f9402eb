"""CPU tier: the actions of an env-step as the kernels decode them (rr_sim.cuh decode_discrete / decode_continuous, which
k_step and the host build in tests/emul share) against the oracle, at the values where decoding can go wrong: rounding
ties, the ends of the 4-bit thrust field, values no int holds, signed zeros, subnormals, NaN, infinities and direction
ids above 7, in every robot slot and with every action count.

Where the oracle raises, the error bits must agree.  A finite thrust whose int(round(x)) falls outside [-8, 7] is
simulated by the reference (unbounded Python int) but refused by the kernels with RR_ERR_BAD_ACTION, env untouched
(include/rr_b200.h); everywhere else outputs, state and the stored thrusts must agree exactly."""
import numpy as np
import pytest

from conftest import golden_files
from golden_util import STATE_KEYS, state_at
from parity_util import FLOAT_KEYS, INT_KEYS, close, compare_record

BAD_ACTION = 512
V0, V2 = "RoboRugby-v0", "RoboRugbySimpleDuel-v2"


@pytest.fixture(params=["libm", "dd"])
def trig(request):
    """libm: glibc sin/cos in the host build (bit-identical trig to the oracle); dd: the routine the GPU runs."""
    from emul import emul
    emul.use_libm_sincos(request.param == "libm")
    yield request.param
    emul.use_libm_sincos(False)


@pytest.fixture
def fresh_scratch(oracle):
    oracle.scratch_mode(1)
    yield oracle
    oracle.scratch_mode(0)


def thrust_values():
    """Every multiple of 0.5 in [-10, 10], the float32 neighbours of the ties at the ends of the field, and values no
    4-bit field or int holds, as the ABI's float32 carries them (2^31 +- 1 round to 2^31 there)."""
    f = np.float32
    v = [0.5 * k for k in range(-20, 21)]
    v += [np.nextafter(f(x), f(d)) for x in (7.5, -7.5, -8.5) for d in (np.inf, -np.inf)]
    v += [-0.0, f(1e-45), -f(1e-45), f(1e-39), 2.0 ** 31 - 1, 2.0 ** 31 + 1, -2.0 ** 31 - 1, 1e10, -1e10,
          np.nan, np.inf, -np.inf]
    return np.array(v, np.float32).astype(np.float64)


def in_field(a):
    """The oracle's int(round(x)) (half to even) of every thrust lies in [-8, 7]."""
    with np.errstate(invalid="ignore"):
        r = np.rint(a)
        return bool(np.all((r >= -8) & (r <= 7)))


def _configs(oracle, preset, env_id):
    from roborugby_b200 import _lib
    cfg = _lib.default_config(_lib.PRESET_GAME if preset == "GAME" else _lib.PRESET_TRAIN, env_id)
    cfg.time_limit = 0
    cfg.auto_reset = 0
    cfg.strict_reset = 1
    return cfg, oracle.default_config(preset, env_id)


def start_states(oracle, preset, env_id, seed):
    """A Philox reset and a contact-rich state from the middle of a golden rollout.  The robots carry stored thrusts
    from the ends of the field, which robots without a command keep."""
    o = oracle.OracleEnv(preset, env_id)
    o.reset_philox(seed, 3, 0)
    states = [o.get_state()]
    kind = "random" if env_id == V0 else "chase"
    path = [p for p in golden_files(f"{preset}_{env_id}_{kind}_s*.npz")][0]
    d = np.load(path)
    i = int(np.nonzero(d["exc"].sum(1) == 0)[0][0])
    states.append(state_at(d, i, d["act"].shape[1] // 2))
    rng = np.random.default_rng(seed)
    for st in states:
        st["rflag"] = np.array(st["rflag"], np.int32)
        st["rflag"][:, :2] = rng.choice([-8, 7, -1, 1, 0, 3], size=(len(st["rflag"]), 2))
        st["step"] = np.int32(min(int(st["step"]), 100))
    return states


def same_state(a, b):
    return all(np.array_equal(np.asarray(a[k]), np.asarray(b[k])) for k in STATE_KEYS)


def check_step(env, o, st, a, why):
    """One step of `a` from `st` on both sides: "refused" (RR_ERR_BAD_ACTION, nothing changed), "raised" (the same
    error bits), "exact" (bit-identical) or "close" (integers exact, floats within the 1e-9 bar of parity_util)."""
    env.set_state(st)
    o.set_state(st)
    got, want = env.step(a), o.step(a)
    refused = got["err"] == BAD_ACTION
    if not env.cfg.discrete and not in_field(a[:2 * (len(a) // 2)]):
        assert refused, (why, got["err"])
        if not np.all(np.isfinite(a)):   # round() raises in the reference
            assert want["err"] & BAD_ACTION, (why, want["err"])
        assert same_state(env.get_state(), st), (why, "a refused step changed the state")
        return "refused"
    assert got["err"] == want["err"], (why, got["err"], want["err"])
    if refused:
        assert same_state(env.get_state(), st) and same_state(o.get_state(), st), (why, "state changed")
        return "refused"
    if want["err"]:
        return "raised"
    ok, exact, w, diff = compare_record(env.get_state(), got, o.get_state(), want)   # (rflag, step: exact)
    assert ok, (why, diff, w)
    return "exact" if exact else "close"


def check_counts(n, trig, refused):
    """Every refusal where expected; with glibc trig nearly every other step bit-identical (the rest differ in the
    last bits of the scratch rect or of atan / sqrt, parity_util)."""
    assert n["refused"] == refused, n
    if trig == "libm":
        assert n["exact"] >= 0.95 * (n["exact"] + n["close"]), n


@pytest.mark.parametrize("preset", ["GAME", "TRAIN"])
def test_continuous_thrust_edges_match_oracle(fresh_scratch, preset, trig):
    """Each edge value paired with itself, its negation, 0, 1 and -1 (robot_move branches on equality, sum and signs) in
    every robot slot; the commanded robots before the slot drive (1, -1), the action count runs from 2 to 2R so that
    robots beyond it keep their stored thrust."""
    from emul.emul import EmulEnv
    oracle = fresh_scratch
    cfg, ocfg = _configs(oracle, preset, V0)
    o = oracle.OracleEnv(cfg=ocfg)
    env = EmulEnv(cfg, o.R, o.B, o.obs_dim)
    R = o.R
    vals = thrust_values()
    n = dict(refused=0, raised=0, exact=0, close=0)
    want_refused = 0
    for st in start_states(oracle, preset, V0, 11):
        for r in range(R):
            j = 0
            for v in vals:
                for l, rt in ((v, v), (v, -v), (v, 0.0), (0.0, v), (v, 1.0), (-1.0, v)):
                    k = 2 * (r + 1 + j % (R - r))
                    j += 1
                    a = np.tile([1.0, -1.0], R)[:k]
                    a[2 * r], a[2 * r + 1] = l, rt
                    n[check_step(env, o, st, a, (r, k, l, rt))] += 1
                    want_refused += not in_field(np.array([l, rt]))
    print(f"{preset} ({trig}): {n}")
    check_counts(n, trig, want_refused)


@pytest.mark.parametrize("preset", ["GAME", "TRAIN"])
def test_discrete_ids_match_oracle(fresh_scratch, preset, trig):
    """Every uint8 id in every robot slot, with 1 to R actions: ids above 7 raise on both sides and change nothing."""
    from emul.emul import EmulEnv
    oracle = fresh_scratch
    cfg, ocfg = _configs(oracle, preset, V2)
    o = oracle.OracleEnv(cfg=ocfg)
    env = EmulEnv(cfg, o.R, o.B, o.obs_dim)
    R = o.R
    rng = np.random.default_rng(5)
    n = dict(refused=0, raised=0, exact=0, close=0)
    for st in start_states(oracle, preset, V2, 12):
        for r in range(R):
            for i in range(256):
                k = r + 1 + i % (R - r)
                a = rng.integers(0, 8, k).astype(np.float64)
                a[r] = i
                n[check_step(env, o, st, a, (r, k, i))] += 1
    print(f"{preset} ({trig}): {n}")
    check_counts(n, trig, 2 * R * 248)


def _probe_raises(oracle, ocfg, st, a):
    p = oracle.OracleEnv(cfg=ocfg)
    p.set_state(st)
    return p.step(a)["err"]


@pytest.mark.parametrize("bad", [np.nan, 8.0, -np.inf, -8.5000005])
@pytest.mark.parametrize("preset", ["GAME", "TRAIN"])
def test_continuous_multistep_carries_thrust_across_a_refused_step(fresh_scratch, preset, bad, trig):
    """Eight steps with a varying number of commands and one unusable thrust in the middle: the refused step changes
    nothing, and the stored thrusts of robots without a command carry across it."""
    from emul.emul import EmulEnv
    oracle = fresh_scratch
    cfg, ocfg = _configs(oracle, preset, V0)
    o = oracle.OracleEnv(cfg=ocfg)
    env = EmulEnv(cfg, o.R, o.B, o.obs_dim)
    R = o.R
    rng = np.random.default_rng(3)
    for st in start_states(oracle, preset, V0, 13):
        env.set_state(st)
        o.set_state(st)
        for s in range(8):
            n = 2 * (1 + s % R)
            a = rng.choice([-1.0, -0.5, 0.0, 0.5, 1.0, 1.5], n)
            if s == 4:
                a[n - 1] = bad
                before = env.get_state()
                if not np.isfinite(bad):
                    assert _probe_raises(oracle, ocfg, o.get_state(), a) & BAD_ACTION
                assert env.step(a)["err"] == BAD_ACTION and same_state(env.get_state(), before), s
                continue
            got, want = env.step(a), o.step(a)
            assert got["err"] == want["err"] == 0, (s, got["err"], want["err"])
            ok, exact, w, diff = compare_record(env.get_state(), got, o.get_state(), want)   # (rflag: every robot)
            assert ok and (exact or trig == "dd"), (s, diff, w)


@pytest.mark.parametrize("preset", ["GAME", "TRAIN"])
def test_discrete_fused_steps_go_on_after_a_refused_step(fresh_scratch, preset, trig):
    """emul_step_k (one Env object over K steps, like a fused launch) with an id above 7 in the middle: it raises
    RR_ERR_BAD_ACTION, moves nothing in that step, and the other steps equal the oracle's run without it."""
    from emul.emul import EmulEnv
    oracle = fresh_scratch
    cfg, ocfg = _configs(oracle, preset, V2)
    o = oracle.OracleEnv(cfg=ocfg)
    env = EmulEnv(cfg, o.R, o.B, o.obs_dim)
    R = o.R
    rng = np.random.default_rng(4)
    K = 9
    for st in start_states(oracle, preset, V2, 14):
        for A in range(1, R + 1):
            acts = rng.integers(0, 8, (K, A)).astype(np.float64)
            acts[K // 2, A - 1] = 8 + rng.integers(0, 248)
            env.set_state(st)
            err, rew, _ = env.step_k(acts)
            assert err == BAD_ACTION and np.all(rew[K // 2] == 0), (A, err)
            o.set_state(st)
            for s in range(K):
                if s == K // 2:
                    assert _probe_raises(oracle, ocfg, o.get_state(), acts[s]) == BAD_ACTION
                    continue
                out = o.step(acts[s])
                assert out["err"] == 0 and close(out["rew"], rew[s]), (A, s, out["err"])
            got, want = env.get_state(), o.get_state()
            assert all(np.array_equal(got[k], want[k]) for k in INT_KEYS), A
            assert all(close(got[k], want[k]) for k in FLOAT_KEYS), A
