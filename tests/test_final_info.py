"""CPU tier: rr_step_info's outputs, i.e. the terminal observation of every done row and the RR_ROW_* flags of every row,
through the host build of the kernel source (tests/emul emul_launch_info, which takes each row apart as k_step does:
step_accounting, step_row_flags, the terminal observation, step_auto_reset) against the oracle.

The restatement is test_episode_stats's RefEnv, which also observes the oracle env before each auto-reset.  A row is
TRUNCATED when it did not raise, the time limit is on, its step counter is >= T and game_is_done() is false (gym 0.17's
info['TimeLimit.truncated']); RAISED when its error bits are non-zero.  Every launch also runs on a twin batch without
these outputs (emul_launch, which ends each row with step_bookkeeping, the composition of the parts): every other
output and the state must be bit-identical.  Final observations of done rows must be within
the 1e-9 bar of the oracle's (bit-identical counts are printed); rows with done == 0 must keep a canary; with
auto_reset = 0 the final rows of done rows equal the obs rows bit for bit."""
import numpy as np
import pytest

from golden_util import actions_at, parse_name, state_at
from parity_util import close
from test_episode_stats import (GOALS, RAISED, V0, V2, Batch, RefEnv, bad_action_grid, configs,  # noqa: F401
                                fresh_scratch, random_actions, step_near_end)

ROW_TRUNCATED, ROW_RAISED = 1, 2
STEP_AFTER_DONE, BAD_ACTION = 1, 512
# registered ids and ad-hoc compositions covering every observer (RR_OBS_NONE .. RR_OBS_LIDAR6_V1)
OBSERVER_ENVS = [V0, V2, "RoboRugbySimpleDuel-v3", "DuelAllCoords", "DuelAllCoordsPrior", "DuelLidar6v1"]


class FinalRef(RefEnv):
    """RefEnv that records, per row, (done, terminal obs_h, terminal obs_g, RR_ROW_* flags): the oracle env observed
    after the row's step and before any auto-reset."""

    rows = ()

    def _capture(self):
        self.final = (self.o.observe(1), self.o.observe(-1), int(self.o.get_state()["step"]), self.finished())

    def reset(self):
        self._capture()
        super().reset()

    def step(self, a):
        self.final = None
        out = super().step(a)
        err, done = out[0], out[1]
        if self.final is None:
            self._capture()
        oh, og, step, finished = self.final
        trunc = not err and self.cfg.time_limit and step >= self.T and not finished
        self.rows.append((done, oh, og, (ROW_TRUNCATED if trunc else 0) | (ROW_RAISED if err else 0), err))
        return out


@pytest.fixture(params=["libm", "dd"])
def trig(request):
    """libm: glibc sin/cos in the host build (bit-identical trig to the oracle); dd: the routine the GPU runs."""
    from emul import emul_info
    emul_info.use_libm_sincos(request.param == "libm")
    yield request.param
    emul_info.use_libm_sincos(False)


class _WithInfo:
    """An EmulBatch whose launches also produce rr_step_info's outputs."""

    def __init__(self, emul):
        self._e = emul

    def __getattr__(self, name):
        return getattr(self._e, name)

    def launch(self, acts, observe=False):
        from emul import emul_info
        return emul_info.launch(self._e, acts, observe=observe)


class InfoBatch(Batch):
    """Batch with FinalRef restatements, launches with the final outputs, and a twin launched without them."""

    def __init__(self, oracle, cfg, ocfg, M):
        from emul.emul import EmulBatch
        super().__init__(oracle, cfg, ocfg, M)
        self.refs = [FinalRef(oracle, cfg, ocfg, i) for i in range(M)]
        self.plain = EmulBatch(cfg, M, self.emul.R, self.emul.B, self.emul.obs_dim)
        self.emul = _WithInfo(self.emul)
        self.seen = dict(done=0, exact=0, truncated=0, raised=0, terminated=0)

    def set_state(self, i, st):
        super().set_state(i, st)
        self.plain.set_state(i, st)

    def launch(self, acts):
        from emul.emul_info import FINAL_CANARY
        for r in self.refs:
            r.rows = []
        got = super().launch(acts)
        plain = self.plain.launch(acts, observe=True)
        for key in ("rew", "done", "err", "naughty", "stats"):
            assert np.array_equal(got[key], plain[key]), key
        if plain["obs_h"] is not None:
            for key in ("obs_h", "obs_g"):
                assert np.array_equal(got[key], plain[key], equal_nan=True), key
        assert np.array_equal(self.emul.sf, self.plain.sf, equal_nan=True) and np.array_equal(self.emul.si, self.plain.si)
        K, D = acts.shape[0], self.emul.obs_dim
        assert set(np.unique(got["flags"])) <= {0, ROW_TRUNCATED, ROW_RAISED}
        assert ((got["flags"] != 0) <= (got["done"] != 0)).all()
        if D:
            dn = got["done"] != 0
            assert (got["final_h"][~dn] == FINAL_CANARY).all() and (got["final_g"][~dn] == FINAL_CANARY).all()
            if not self.emul.cfg.auto_reset:
                assert np.array_equal(got["final_h"][dn], got["obs_h"][dn], equal_nan=True)
                assert np.array_equal(got["final_g"][dn], got["obs_g"][dn], equal_nan=True)
        for i in range(self.M):
            if i in self.diverged:
                continue
            for s in range(K):
                done, oh, og, flags, err = self.refs[i].rows[s]
                assert got["flags"][s, i] == flags, (i, s, got["flags"][s, i], flags)
                if not done:
                    continue
                self.seen["done"] += 1
                self.seen["truncated" if flags & ROW_TRUNCATED else "raised" if flags else "terminated"] += 1
                # after a raise inside the physics the reference's env holds whatever its exception left, which the
                # kernels do not reproduce (test_episode_stats): such rows are pinned by test_raised_rows_... below
                if D and not err & ~(STEP_AFTER_DONE | BAD_ACTION):
                    assert close(got["final_h"][s, i], oh) and close(got["final_g"][s, i], og), (i, s)
                    self.seen["exact"] += np.array_equal(got["final_h"][s, i], oh) and np.array_equal(got["final_g"][s, i], og)
        return got


@pytest.mark.parametrize("auto_reset", [0, 1])
@pytest.mark.parametrize("time_limit", [0, 1])
@pytest.mark.parametrize("preset", ["GAME", "TRAIN"])
def test_final_info_at_the_end_of_an_episode(fresh_scratch, preset, time_limit, auto_reset, trig):
    """Envs from T - 3 to T + 1 over three launches of 3 steps: episodes end inside and across launches.  With the time
    limit the row at step T is truncated; without it the raw row at T + 1 is a real end; without auto-reset the rows
    after the end are refused (RAISED, STEP_AFTER_DONE)."""
    oracle = fresh_scratch
    cfg, ocfg = configs(oracle, preset, V2, time_limit, auto_reset)
    T = 4500 if preset == "GAME" else 300
    starts = [T - 3, T - 2, T - 1, T, T + 1, 0, T - 4, T - 1]
    b = InfoBatch(oracle, cfg, ocfg, len(starts))
    for i, st in enumerate(step_near_end(oracle, preset, V2, cfg, starts)):
        b.set_state(i, st)
    rng = np.random.default_rng(1)
    for _ in range(3):
        b.launch(random_actions(rng, cfg, 3, b.M, b.refs[0].o.R))
    assert not b.diverged, b.diverged
    print(f"{preset} time_limit={time_limit} auto_reset={auto_reset}: {b.seen}")
    # truncated: the envs from T - 4 to T - 1 reach step T; the one injected at T ends raw at T + 1 (terminated)
    assert b.seen["truncated"] == (5 if time_limit else 0), b.seen
    assert b.seen["terminated"] >= (1 if time_limit else 6), b.seen


@pytest.mark.parametrize("env_id", OBSERVER_ENVS)
@pytest.mark.parametrize("preset", ["GAME", "TRAIN"])
def test_final_observation_of_every_observer(fresh_scratch, preset, env_id, trig):
    """Every observer, with and without auto-reset: envs at T - 2 and random steps with random actions.  For
    AllCoords_WithPrior the prior-step columns of the final observation are those of the terminal step, not the reset's."""
    oracle = fresh_scratch
    T = 4500 if preset == "GAME" else 300
    for auto_reset in (1, 0):
        cfg, ocfg = configs(oracle, preset, env_id, 1, auto_reset)
        starts = [T - 2, T - 1, T - 3, 17, T - 2, T - 5]
        b = InfoBatch(oracle, cfg, ocfg, len(starts))
        for i, st in enumerate(step_near_end(oracle, preset, env_id, cfg, starts, seed=11)):
            b.set_state(i, st)
        rng = np.random.default_rng(3)
        b.launch(random_actions(rng, cfg, 4, b.M, b.refs[0].o.R))
        assert not b.diverged, b.diverged
        assert b.seen["truncated"] == 4, b.seen           # the envs from T - 3 to T - 1
        print(f"{preset} {env_id} auto_reset={auto_reset}: {b.seen}")


@pytest.mark.parametrize("auto_reset", [0, 1])
@pytest.mark.parametrize("env_id", [V2, V0])
@pytest.mark.parametrize("preset", ["GAME", "TRAIN"])
def test_unusable_actions_and_refused_steps(fresh_scratch, preset, env_id, auto_reset, trig):
    """Bad discrete ids and bad thrusts on live, last-step and finished envs, steps refused with STEP_AFTER_DONE, and
    envs injected past their end: every such row is RAISED and never TRUNCATED, and its final observation is the state
    the refused step left untouched."""
    oracle = fresh_scratch
    cfg, ocfg = configs(oracle, preset, env_id, 1, auto_reset)
    T = 4500 if preset == "GAME" else 300
    R = oracle.OracleEnv(cfg=ocfg).R
    grid = bad_action_grid(cfg, R)
    starts = [10, T - 1, T, T + 1, T + 3]
    M = len(starts) * len(grid)
    b = InfoBatch(oracle, cfg, ocfg, M)
    for i, st in enumerate(step_near_end(oracle, preset, env_id, cfg, starts * len(grid))):
        b.set_state(i, st)
    rng = np.random.default_rng(2)
    acts = random_actions(rng, cfg, 4, M, R)
    for i in range(M):
        acts[1, i] = grid[i // len(starts)]
    got = b.launch(acts)
    assert not b.diverged, b.diverged
    assert ((got["flags"] == ROW_RAISED) == (got["err"] != 0)).all()
    assert (got["flags"][1] == ROW_RAISED).all()
    print(f"{preset} {env_id} auto_reset={auto_reset}: {b.seen}")


@pytest.mark.parametrize("path", GOALS, ids=[p.split("/")[-1] for p in GOALS])
def test_goal_ended_episodes_are_not_truncated(fresh_scratch, path):
    """Goal scoring (compositions without NaughtyBots): episodes that end on a destroyed goal or an empty field before T
    are terminated, and so are the same trajectories replayed with step counters shifted so that the goal falls at
    exactly step T, where the time limit would otherwise truncate."""
    oracle = fresh_scratch
    from emul import emul_info
    emul_info.use_libm_sincos(True)
    try:
        preset, env_id, _ = parse_name(path)
        T = 4500 if preset == "GAME" else 300
        d = np.load(path)
        n, L = d["act"].shape[:2]
        acts = np.nan_to_num(d["act"], nan=0.0).transpose(1, 0, 2)        # [L, n, A]
        states = [state_at(d, i, 0) for i in range(n)]
        cfg, ocfg = configs(oracle, preset, env_id, 1, 0, goals=True)
        b = InfoBatch(oracle, cfg, ocfg, n)
        for i in range(n):
            b.set_state(i, states[i])
        got = b.launch(acts)
        ends = (got["done"] == 1) & (got["flags"] == 0)                    # terminated rows
        ended = [i for i in range(n) if i not in b.diverged and ends[:, i].any()]
        assert ended and not b.seen["truncated"], b.seen
        first = {i: int(np.argmax(ends[:, i])) for i in ended}
        for auto_reset in (0, 1):
            cfg, ocfg = configs(oracle, preset, env_id, 1, auto_reset, goals=True)
            b = InfoBatch(oracle, cfg, ocfg, len(ended))
            for j, i in enumerate(ended):
                st = dict(states[i])
                st["step"] = np.int32(T - 1 - first[i])                 # the ending row lands on step T
                b.set_state(j, st)
            K = max(first.values()) + 1
            got = b.launch(acts[:K, ended])
            for j, i in enumerate(ended):
                if j not in b.diverged:
                    r = first[i]
                    assert got["done"][r, j] == 1 and got["flags"][r, j] == 0, (i, r, got["flags"][r, j])
            print(f"{path.split('/')[-1]} auto_reset={auto_reset}: {len(ended)} goal ends at T, {b.seen}, "
                  f"{len(b.diverged)} diverged")
            assert len(b.diverged) <= len(ended) // 2
    finally:
        emul_info.use_libm_sincos(False)


@pytest.mark.parametrize("rec", RAISED, ids=[f"{r[0].split('/')[-1]}:{r[1]}:{r[2]}" for r in RAISED])
def test_raised_rows_report_the_state_the_kernel_left(fresh_scratch, rec):
    """The golden records on which the reference raises, injected two steps earlier: the raising row is RAISED, never
    TRUNCATED, and its final observation with auto-reset is, bit for bit, the observation the same launch reports for
    that row without auto-reset (the state the abandoned step left)."""
    oracle = fresh_scratch
    from emul import emul_info
    emul_info.use_libm_sincos(True)
    try:
        path, i, t = rec
        preset, env_id, _ = parse_name(path)
        d = np.load(path)
        back = min(t, 2)
        st = state_at(d, i, t - back)
        acts = np.stack([actions_at(d, i, t - q) for q in range(back, -1, -1)])[:, None]
        out = {}
        for auto_reset in (0, 1):
            cfg, ocfg = configs(oracle, preset, env_id, 1, auto_reset)
            b = InfoBatch(oracle, cfg, ocfg, 1)
            b.set_state(0, st)
            out[auto_reset] = b.launch(acts)
            assert not b.diverged
            g = out[auto_reset]
            assert g["err"][back, 0] != 0 and g["flags"][back, 0] == ROW_RAISED and (g["flags"][:back, 0] == 0).all()
        if out[1]["final_h"] is not None:
            assert np.array_equal(out[1]["final_h"][back], out[0]["obs_h"][back], equal_nan=True)
            assert np.array_equal(out[1]["final_g"][back], out[0]["obs_g"][back], equal_nan=True)
    finally:
        emul_info.use_libm_sincos(False)
