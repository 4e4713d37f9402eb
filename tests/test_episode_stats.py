"""CPU tier: the episode statistics of k_step (RR_STAT_*, the rules of rr_get_stats in include/rr_b200.h) through the host
build of the kernel source (tests/emul emul_launch: one launch over M envs, the bookkeeping k_step shares through
rr_sim.cuh step_bookkeeping) against a plain restatement of those rules over the oracle.

The restatement (RefEnv) steps one oracle env per env, resets it from the env's own Philox stream, applies the refusal
order of the header and adds up, per env and launch: steps, errors, naughty events and, at the first done row since the
env's last reset or rr_set_state, one episode with its return and length.  Rows are compared as in parity_util; the
integer statistics must agree exactly; each return must equal bit for bit the step-order sum of the host build's own
reward rows, and the oracle's sum within the 1e-9 bar."""
import numpy as np
import pytest

from conftest import golden_files
from golden_util import apply_overrides, actions_at, parse_name, resolve_env, state_at
from parity_util import close

STEP_AFTER_DONE, BAD_ACTION = 1, 512
EPISODES, RET_H, RET_G, LENGTH, NAUGHTY, ERRORS, STEPS, REPLAYS = range(8)
INT_STATS = (EPISODES, LENGTH, NAUGHTY, ERRORS, STEPS)
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


def in_field(a):
    """Every thrust's int(round(x)) (half to even) lies in [-8, 7]."""
    with np.errstate(invalid="ignore"):
        r = np.rint(np.asarray(a, np.float32).astype(np.float64))
        return bool(np.all((r >= -8) & (r <= 7)))


def configs(oracle, preset, env_id, time_limit, auto_reset, goals=False, flags=0, seed=7, env_offset=40):
    """(C ABI config, oracle config) of one composition; strict placement, as the oracle's reset_philox draws it."""
    from roborugby_b200 import _lib
    base, _ = resolve_env(env_id)
    cfg = apply_overrides(_lib.default_config(_lib.PRESET_GAME if preset == "GAME" else _lib.PRESET_TRAIN, base), env_id)
    cfg.time_limit, cfg.auto_reset, cfg.strict_reset = int(time_limit), int(auto_reset), 1
    cfg.seed, cfg.env_offset, cfg.flags, cfg.goal_scoring = seed, env_offset, flags, int(goals)
    ocfg = apply_overrides(oracle.default_config(preset, base, time_limit=time_limit), env_id)
    ocfg.goal_scoring = int(goals)
    return cfg, ocfg


class RefEnv:
    """One env of the batch restated over the oracle: its rows as k_step reports them and its statistics."""

    def __init__(self, oracle, cfg, ocfg, i):
        self.o = oracle.OracleEnv(cfg=ocfg)
        self.cfg, self.gi = cfg, cfg.env_offset + i
        self.T = 4500 if ocfg.game_mode else 300
        self.episode = 0
        self.o.reset_philox(cfg.seed, self.gi, 0)
        self._fresh()
        self.st = np.zeros(8)

    def _fresh(self):
        self.ret = np.zeros(2)
        self.counted = False

    def set_state(self, st):
        self.o.set_state(st)
        self._fresh()

    def reset(self):
        self.episode += 1
        self.o.reset_philox(self.cfg.seed, self.gi, self.episode)
        self._fresh()

    def finished(self):
        """The reference's game_is_done() (RR_EnvBase.py:555-559): a step now raises "Game is over"."""
        if int(self.o.get_state()["step"]) > self.T:
            return True
        if self.cfg.goal_scoring:
            g = self.o.goal_state()
            return bool(g["destroyed"].any() or not g["alive"].any())
        return False

    def step(self, a):
        """One row: (err, done, rew[2], naughty, obs_h, obs_g), the rules table applied to self.st."""
        if not self.cfg.discrete and not self.finished() and not in_field(a):
            err, done, rew, ng = BAD_ACTION, 0, np.zeros(2), 0    # refused, env untouched (the header's deviation)
        else:
            out = self.o.step(a)
            err, done, rew, ng = out["err"], out["done"], out["rew"], out["naughty"]
        if err:                                                    # the reference has raised: the row is aborted
            done, rew, ng = 1, np.zeros(2), 0
        self.ret = self.ret + rew
        if not err & STEP_AFTER_DONE:
            self.st[STEPS] += 1
            self.st[NAUGHTY] += ng
            self.st[ERRORS] += err != 0
            if done and not self.counted:
                self.counted = True
                self.st[EPISODES] += 1
                self.st[[RET_H, RET_G]] += self.ret
                self.st[LENGTH] += int(self.o.get_state()["step"])
        if done and self.cfg.auto_reset:
            self.reset()
        return err, done, rew, ng, self.o.observe(1), self.o.observe(-1)


class Batch:
    """The host build's launch and the restatement side by side.  An env whose rows leave the 1e-9 bar (a last-bit
    contact flip, parity_util) is counted in `diverged` and no longer compared."""

    def __init__(self, oracle, cfg, ocfg, M):
        from emul.emul import EmulBatch
        self.refs = [RefEnv(oracle, cfg, ocfg, i) for i in range(M)]
        r = self.refs[0].o
        self.emul = EmulBatch(cfg, M, r.R, r.B, r.obs_dim)
        self.M = M
        self.ret = np.zeros((M, 2))          # step-order sum of the host build's own reward rows since the last reset
        self.counted = np.zeros(M, bool)
        self.diverged = set()
        self.totals = np.zeros(8)            # the host build's statistics summed over the launches
        self.ref_totals = np.zeros(8)

    def set_state(self, i, st):
        self.emul.set_state(i, st)
        self.refs[i].set_state(st)
        self.ret[i] = 0.0
        self.counted[i] = False

    def reset(self, mask):
        self.emul.reset(mask)
        for i in np.nonzero(mask)[0]:
            self.refs[i].reset()
            self.ret[i] = 0.0
            self.counted[i] = False

    def launch(self, acts):
        """One launch of acts [K, M, A]; returns the host build's output dict."""
        K = acts.shape[0]
        got = self.emul.launch(acts, observe=True)
        if got["obs_h"] is None:                        # an env without observations
            got["obs_h"] = got["obs_g"] = np.zeros(acts.shape[:2] + (0,))
        for r in self.refs:
            r.st[:] = 0.0
        for i in range(self.M):
            mine = np.zeros(8)
            for s in range(K):
                err, done, rew, ng, oh, og = self.refs[i].step(acts[s, i])
                if i in self.diverged:
                    continue
                assert got["err"][s, i] == err, (i, s, got["err"][s, i], err)
                assert got["done"][s, i] == done, (i, s, got["done"][s, i], done)
                # after a raise without a reset both envs hold what the abandoned step left: not compared
                left = err & ~(STEP_AFTER_DONE | BAD_ACTION) and not self.emul.cfg.auto_reset
                if not (close(got["rew"][s, i], rew) and got["naughty"][s, i] == ng and
                        (left or close(got["obs_h"][s, i], oh) and close(got["obs_g"][s, i], og))):
                    self.diverged.add(i)
                    continue
                # the host build's rows under the rules table, its own rewards summed in step order
                self.ret[i] += got["rew"][s, i]
                if not err & STEP_AFTER_DONE and done and not self.counted[i]:
                    self.counted[i] = True
                    mine[[RET_H, RET_G]] += self.ret[i]
                if done and self.emul.cfg.auto_reset:
                    self.ret[i] = 0.0
                    self.counted[i] = False
            if i in self.diverged:
                continue
            want, have = self.refs[i].st, got["stats"][i]
            assert np.array_equal(have[list(INT_STATS)], want[list(INT_STATS)]), (i, have, want)
            assert np.array_equal(have[[RET_H, RET_G]], mine[[RET_H, RET_G]]), (i, have, mine)
            assert close(have[[RET_H, RET_G]], want[[RET_H, RET_G]]), (i, have, want)
            self.totals += have
            self.ref_totals += want
        return got


def step_near_end(oracle, preset, env_id, cfg, steps, seed=3):
    """Philox reset states with their step counters set to `steps`."""
    o = oracle.OracleEnv(cfg=oracle.default_config(preset, resolve_env(env_id)[0]))
    out = []
    for j, s in enumerate(steps):
        o.reset_philox(seed, 500 + j, 0)
        st = o.get_state()
        st["step"] = np.int32(s)
        out.append(st)
    return out


def random_actions(rng, cfg, K, M, R):
    if cfg.discrete:
        return rng.integers(0, 8, (K, M, R)).astype(np.float64)
    return rng.choice([-1.0, -0.5, 0.0, 0.5, 1.0], (K, M, 2 * R))


@pytest.mark.parametrize("auto_reset", [0, 1])
@pytest.mark.parametrize("time_limit", [0, 1])
@pytest.mark.parametrize("preset", ["GAME", "TRAIN"])
def test_episode_counts_at_the_end_of_an_episode(fresh_scratch, preset, time_limit, auto_reset, trig):
    """Envs from T - 3 to T + 2 over three launches of 3 steps: episodes end inside a launch and across launches.
    Without auto-reset the rows at steps T, T + 1 and T + 2 report done on both sides, and only the first of them
    counts an episode (its return and length); the refused rows count nothing."""
    oracle = fresh_scratch
    cfg, ocfg = configs(oracle, preset, V2, time_limit, auto_reset)
    T = 4500 if preset == "GAME" else 300
    starts = [T - 3, T - 2, T - 1, T, T + 1, 0, T - 4, T - 1]
    b = Batch(oracle, cfg, ocfg, len(starts))
    for i, st in enumerate(step_near_end(oracle, preset, V2, cfg, starts)):
        b.set_state(i, st)
    rng = np.random.default_rng(1)
    for _ in range(3):
        b.launch(random_actions(rng, cfg, 3, b.M, b.refs[0].o.R))
    assert not b.diverged, b.diverged
    # one episode for every env that was not injected past its end (T + 1) and reaches it (not the one at step 0);
    # without auto-reset an env steps until its counter passes T and is refused from then on
    assert b.totals[EPISODES] == 6, b.totals
    assert b.totals[STEPS] == (9 * len(starts) - 1 if auto_reset else 4 + 3 + 2 + 1 + 0 + 9 + 5 + 2), b.totals
    assert b.totals[ERRORS] == 0


def test_time_limit_end_is_counted_once_without_auto_reset(oracle):
    """The rows at steps T, T + 1 and T + 2 report (done, err) = (1, 0), (1, 0), (1, STEP_AFTER_DONE): one episode of
    length T, two steps, no error."""
    for preset in ("GAME", "TRAIN"):
        cfg, ocfg = configs(oracle, preset, V2, 1, 0)
        T = 4500 if preset == "GAME" else 300
        b = Batch(oracle, cfg, ocfg, 1)
        b.set_state(0, step_near_end(oracle, preset, V2, cfg, [T - 1])[0])
        got = b.launch(np.zeros((3, 1, b.refs[0].o.R)))
        assert got["done"][:, 0].tolist() == [1, 1, 1] and got["err"][:, 0].tolist() == [0, 0, STEP_AFTER_DONE]
        st = got["stats"][0]
        assert (st[EPISODES], st[LENGTH], st[STEPS], st[ERRORS]) == (1, T, 2, 0), st


def bad_action_grid(cfg, R):
    """Per env a list of actions: unusable ones (ids above 7; NaN, infinite and out-of-field thrusts) among good ones."""
    if cfg.discrete:
        return [np.array([9.0] + [0.0] * (R - 1)), np.array([3.0] * (R - 1) + [255.0]), np.full(R, 8.0)]
    good = np.tile([1.0, -1.0], R)
    out = []
    for v in (np.nan, np.inf, -np.inf, 7.5, -8.5000005, 1e10):
        a = good.copy()
        a[2 * R - 1] = v
        out.append(a)
    return out


@pytest.mark.parametrize("auto_reset", [0, 1])
@pytest.mark.parametrize("env_id", [V2, V0])
@pytest.mark.parametrize("preset", ["GAME", "TRAIN"])
def test_unusable_actions_on_live_last_step_and_finished_envs(fresh_scratch, preset, env_id, auto_reset, trig):
    """Unusable actions on live envs, on envs at step T (time limit) and on finished envs.  The error bits are the
    oracle's: BAD_ACTION for a discrete id above 7 anywhere, STEP_AFTER_DONE for any continuous action on a finished env.
    A refused bad action on a finished env is a step and an error but not another episode."""
    oracle = fresh_scratch
    cfg, ocfg = configs(oracle, preset, env_id, 1, auto_reset)
    T = 4500 if preset == "GAME" else 300
    R = oracle.OracleEnv(cfg=ocfg).R
    grid = bad_action_grid(cfg, R)
    starts = [10, T - 1, T, T + 1, T + 3]
    M = len(starts) * len(grid)
    b = Batch(oracle, cfg, ocfg, M)
    states = step_near_end(oracle, preset, env_id, cfg, starts * len(grid))
    for i, st in enumerate(states):
        b.set_state(i, st)
    rng = np.random.default_rng(2)
    K = 4
    acts = random_actions(rng, cfg, K, M, R)
    for i in range(M):
        acts[1, i] = grid[i // len(starts)]          # the second row of every env
    got = b.launch(acts)
    assert not b.diverged, b.diverged
    for i in range(M):
        s0 = starts[i % len(starts)]
        finished_at_row1 = (s0 + 1 > T) and not auto_reset
        e = got["err"][1, i]
        if cfg.discrete or not finished_at_row1:
            assert e == BAD_ACTION, (i, s0, e)
        else:
            assert e == STEP_AFTER_DONE, (i, s0, e)


def test_unusable_actions_on_a_finished_env_count_as_steps_not_episodes(oracle):
    """After the counted time-limit end at step T: a discrete id above 7 adds a step and an error and no episode; a
    continuous NaN is refused as STEP_AFTER_DONE and adds nothing."""
    for preset in ("GAME", "TRAIN"):
        T = 4500 if preset == "GAME" else 300
        for env_id, bad, want in ((V2, 9.0, BAD_ACTION), (V0, np.nan, STEP_AFTER_DONE)):
            cfg, ocfg = configs(oracle, preset, env_id, 1, 0)
            b = Batch(oracle, cfg, ocfg, 1)
            R = b.refs[0].o.R
            b.set_state(0, step_near_end(oracle, preset, env_id, cfg, [T - 1])[0])
            a = np.zeros((4, 1, R if cfg.discrete else 2 * R))
            a[3, 0, -1] = bad
            got = b.launch(a)
            assert got["err"][:, 0].tolist() == [0, 0, STEP_AFTER_DONE, want], (preset, env_id, got["err"][:, 0])
            st = got["stats"][0]
            counted = want == BAD_ACTION
            assert (st[EPISODES], st[LENGTH], st[STEPS], st[ERRORS]) == (1, T, 2 + counted, counted), st


@pytest.mark.parametrize("env_id", [V2, V0])
@pytest.mark.parametrize("preset", ["GAME", "TRAIN"])
def test_env_injected_past_its_end_is_reset_by_auto_reset(fresh_scratch, preset, env_id, trig):
    """With auto-reset an env injected at a step beyond T reports done on a STEP_AFTER_DONE row that counts nothing,
    is reset on that row, and its next row is the first step of episode 1."""
    oracle = fresh_scratch
    for time_limit in (0, 1):
        cfg, ocfg = configs(oracle, preset, env_id, time_limit, 1)
        T = 4500 if preset == "GAME" else 300
        starts = [T + 1, T + 2, T + 1000, 2 ** 31 - 1]
        b = Batch(oracle, cfg, ocfg, len(starts))
        for i, st in enumerate(step_near_end(oracle, preset, env_id, cfg, starts)):
            b.set_state(i, st)
        rng = np.random.default_rng(4)
        got = b.launch(random_actions(rng, cfg, 3, b.M, b.refs[0].o.R))
        assert not b.diverged
        assert (got["err"][0] == STEP_AFTER_DONE).all() and (got["done"][0] == 1).all()
        assert (got["err"][1:] == 0).all() and (got["done"][1:] == 0).all()
        assert (b.emul.episode == 1).all()
        assert all(int(b.emul.get_state(i)["step"]) == 2 for i in range(b.M))
        st = got["stats"].sum(0)
        assert (st[EPISODES], st[STEPS], st[ERRORS]) == (0, 2 * b.M, 0), st


RAISED = [(f, int(i), int(t)) for f in golden_files("*.npz") if "exc" in np.load(f).files
          for i, t in np.argwhere(np.load(f)["exc"] == 1)]


@pytest.mark.parametrize("auto_reset", [0, 1])
@pytest.mark.parametrize("rec", RAISED, ids=[f"{r[0].split('/')[-1]}:{r[1]}:{r[2]}" for r in RAISED])
def test_rows_on_which_the_reference_raises(fresh_scratch, rec, auto_reset):
    """The golden records on which the reference raises, injected, and the same trajectory from two steps earlier: the
    aborted row adds no reward and counts a step, an error and an episode of its length.  With auto-reset the env
    restarts from its own Philox stream on that row and two more steps follow.  Without it the rows end at the raise:
    the reference's env is then in whatever state its exception left, which the kernels do not reproduce."""
    oracle = fresh_scratch
    from emul import emul
    emul.use_libm_sincos(True)
    try:
        path, i, t = rec
        preset, env_id, _ = parse_name(path)
        d = np.load(path)
        cfg, ocfg = configs(oracle, preset, env_id, 1, auto_reset)
        for back in sorted({0, min(t, 2)}):
            st = state_at(d, i, t - back)
            b = Batch(oracle, cfg, ocfg, 1)
            b.set_state(0, st)
            acts = np.stack([actions_at(d, i, t - q) for q in range(back, -1, -1)])
            if auto_reset:
                acts = np.concatenate([acts, acts[:2]])
            got = b.launch(acts[:, None])
            assert not b.diverged
            r = back
            assert got["err"][r, 0] != 0 and got["done"][r, 0] == 1 and (got["rew"][r, 0] == 0).all()
            s = got["stats"][0]
            assert (s[EPISODES], s[LENGTH], s[STEPS], s[ERRORS]) == (1, int(st["step"]) + r + 1, len(acts), 1), s
            assert b.emul.episode[0] == auto_reset
    finally:
        emul.use_libm_sincos(False)


@pytest.mark.parametrize("preset", ["GAME", "TRAIN"])
def test_set_state_and_reset_discard_the_partial_return(fresh_scratch, preset, trig):
    """rr_set_state and rr_reset in the middle of an episode start a new one: the return gathered before them is not
    counted.  Envs end at the time limit in the launch after the interruption."""
    oracle = fresh_scratch
    cfg, ocfg = configs(oracle, preset, V2, 1, 1)
    T = 4500 if preset == "GAME" else 300
    b = Batch(oracle, cfg, ocfg, 6)
    states = step_near_end(oracle, preset, V2, cfg, [T - 8] * 6)
    for i, st in enumerate(states):
        b.set_state(i, st)
    rng = np.random.default_rng(5)
    R = b.refs[0].o.R
    b.launch(random_actions(rng, cfg, 4, 6, R))
    for i in (0, 1):
        b.set_state(i, states[i])                       # back to step T - 8, return 0
    mask = np.zeros(6, bool); mask[[2, 3]] = True
    b.reset(mask)                                       # episode 1 from step 0
    for i in (2, 3):                                    # then step T - 3 of that episode
        st = b.emul.get_state(i); st["step"] = np.int32(T - 3)
        b.set_state(i, st)
    got = b.launch(random_actions(rng, cfg, 8, 6, R))
    assert not b.diverged
    assert (got["stats"][:, EPISODES] == 1).all() and (got["stats"][:, LENGTH] == T).all(), got["stats"]


GOALS = [f for f in golden_files("*_goals_*.npz") if "SimpleDuel" not in f]


@pytest.mark.parametrize("path", GOALS, ids=[p.split("/")[-1] for p in GOALS])
def test_goal_scoring_returns_and_goal_ended_episodes(fresh_scratch, path):
    """Goal scoring: the golden trajectories of the patched reference, several launches, without and with auto-reset.
    Returns carry the +-500 deltas and the BaseDestruction payout; episodes end on a destroyed goal or an empty field."""
    oracle = fresh_scratch
    from emul import emul
    emul.use_libm_sincos(True)
    try:
        preset, env_id, _ = parse_name(path)
        d = np.load(path)
        n, T = d["act"].shape[:2]
        ended = int((d["exc"] == 2).any(1).sum())
        for auto_reset in (0, 1):
            cfg, ocfg = configs(oracle, preset, env_id, 1, auto_reset, goals=True)
            b = Batch(oracle, cfg, ocfg, n)
            for i in range(n):
                b.set_state(i, state_at(d, i, 0))
            acts = np.nan_to_num(d["act"], nan=0.0).transpose(1, 0, 2)        # [T, n, A]
            for s0 in range(0, T, 55):
                b.launch(acts[s0:s0 + 55])
            print(f"{path.split('/')[-1]} auto_reset={auto_reset}: {b.ref_totals}, {len(b.diverged)} diverged")
            assert len(b.diverged) <= n // 2
            if not b.diverged:
                assert b.ref_totals[EPISODES] >= ended and ended > 0
                if "DuelGoals" in path:                     # (RoboRugby-v0 keeps no score)
                    assert np.abs(b.ref_totals[[RET_H, RET_G]]).max() >= 500
    finally:
        emul.use_libm_sincos(False)


@pytest.mark.parametrize("preset", ["GAME", "TRAIN"])
def test_squeeze_memo_changes_only_the_replay_count(fresh_scratch, preset):
    """RR_FLAG_NO_SQUEEZE_MEMO: replays are 0 and every other statistic is the same; with the memo on, replays are no
    more than the pinned-ball frames the oracle executed on the same trajectories."""
    oracle = fresh_scratch
    from emul import emul
    emul.use_libm_sincos(True)
    try:
        import squeeze_util
        rng = np.random.default_rng(9)
        states = [squeeze_util.oracle_env(oracle, preset, squeeze_util.scenario(rng, preset)).get_state() for _ in range(6)]
        acts = np.stack([squeeze_util.actions(rng, states[0]["rob"].shape[0], 6) for _ in states], 1).astype(np.float64)
        out = {}
        for flags in (0, 1):
            cfg, ocfg = configs(oracle, preset, V2, 1, 1, flags=flags)
            b = Batch(oracle, cfg, ocfg, len(states))
            for i, st in enumerate(states):
                b.set_state(i, st)
            oracle.failed_frames(clear=True)
            b.launch(acts[:3])
            b.launch(acts[3:])
            assert not b.diverged
            out[flags] = (b.totals.copy(), oracle.failed_frames())
        (memo, failed), (plain, _) = out[0], out[1]
        assert plain[REPLAYS] == 0 and np.array_equal(np.delete(memo, REPLAYS), np.delete(plain, REPLAYS))
        print(f"{preset}: {memo[REPLAYS]:.0f} replays, {failed} pinned-ball frames in the oracle")
        assert 0 < memo[REPLAYS] <= failed
    finally:
        emul.use_libm_sincos(False)
