"""CPU tier: each row's episode result (rr_step_episodes, include/rr_b200.h) through the host build of the kernel source
(tests/emul emul_episodes: StepOut::counted from step_accounting and the return, length and goal words read before the
auto-reset, as k_step reads them) against a plain restatement over the oracle.

The restatement (EpRef, in the style of test_episode_stats.RefEnv) steps one oracle env per env with the refusal order
of the header and, on the row that counts an episode (done, not a STEP_AFTER_DONE refusal, episode not counted yet),
reports the oracle's step counter and goal state and the return gathered since the env's last reset or rr_set_state.
On every row: whether it counts, its length and its goal words must agree exactly; its return must equal bit for bit the
step-order sum of the host build's own reward rows and the oracle's within the 1e-9 bar; rows that do not count hold
0.0, -1 and zeros.  Per env and launch, the counting rows, the sum of their lengths and the step-order sum of their
returns equal that env's statistics exactly.  Pool rows: an episode continued from a row saved mid-episode has the
row's return plus what follows and continues its step counter; a row saved from a finished episode is refused and
counts nothing.  One K-step launch equals K one-step launches."""
import numpy as np
import pytest

from golden_util import actions_at, parse_name, state_at
from parity_util import close
from test_episode_stats import (BAD_ACTION, EPISODES, GOALS, LENGTH, RAISED, RET_G, RET_H, STEP_AFTER_DONE, V0, V2,
                                RefEnv, bad_action_grid, configs, fresh_scratch, in_field, random_actions, step_near_end)
from test_state_rows import _same, actions, batch, make_cfg

__all__ = ["fresh_scratch"]   # a fixture shared with test_episode_stats


@pytest.fixture(params=["libm", "dd"])
def trig(request):
    """libm: glibc sin/cos in the host build (bit-identical trig to the oracle); dd: the routine the GPU runs."""
    from emul import emul_episodes
    emul_episodes.use_libm_sincos(request.param == "libm")
    yield request.param
    emul_episodes.use_libm_sincos(False)


def oracle_goals(o):
    """rr_goal_state's four words (happy score, grumpy score, destroyed bits, alive-ball bits) of an oracle env."""
    g = o.goal_state()
    return np.array([g["score"][0], g["score"][1], int(g["destroyed"][0]) | int(g["destroyed"][1]) << 1,
                     int(np.sum(g["alive"].astype(np.int64) << np.arange(len(g["alive"]))))], np.int32)


class EpRef(RefEnv):
    """RefEnv whose rows also carry the episode result of the header: (return [2], length, goals [4]) on the row that
    counts an episode, else None."""

    def step(self, a):
        if not self.cfg.discrete and not self.finished() and not in_field(a):
            err, done, rew, ng = BAD_ACTION, 0, np.zeros(2), 0
        else:
            out = self.o.step(a)
            err, done, rew, ng = out["err"], out["done"], out["rew"], out["naughty"]
        if err:
            done, rew, ng = 1, np.zeros(2), 0
        self.ret = self.ret + rew
        ep = None
        if not err & STEP_AFTER_DONE and done and not self.counted:
            self.counted = True
            ep = (self.ret.copy(), int(self.o.get_state()["step"]),
                  oracle_goals(self.o) if self.cfg.goal_scoring else None)
        if done and self.cfg.auto_reset:
            self.reset()
        return err, done, rew, ng, self.o.observe(1), self.o.observe(-1), ep


class EpBatch:
    """The host build's rr_step_episodes launch and the restatement side by side.  An env whose rows leave the 1e-9 bar
    (a last-bit contact flip, parity_util) is counted in `diverged` and no longer compared."""

    def __init__(self, oracle, cfg, ocfg, M):
        from emul.emul import EmulBatch
        self.refs = [EpRef(oracle, cfg, ocfg, i) for i in range(M)]
        r = self.refs[0].o
        self.emul = EmulBatch(cfg, M, r.R, r.B, r.obs_dim)
        self.cfg, self.M = cfg, M
        self.ret = np.zeros((M, 2))      # step-order sum of the host build's own reward rows since the last reset
        self.diverged = set()
        self.episodes = 0
        self.lengths = []

    def set_state(self, i, st):
        self.emul.set_state(i, st)
        self.refs[i].set_state(st)
        self.ret[i] = 0.0

    def reset(self, mask):
        self.emul.reset(mask)
        for i in np.nonzero(mask)[0]:
            self.refs[i].reset()
            self.ret[i] = 0.0

    def launch(self, acts):
        from emul import emul_episodes
        K = acts.shape[0]
        got = emul_episodes.launch(self.emul, acts)
        er, el, eg = got["ep_return"], got["ep_length"], got["ep_goals"]
        assert (el >= -1).all() and (er[el < 0] == 0.0).all()
        if eg is not None:
            assert (eg[el < 0] == 0).all()
        for i in range(self.M):
            for s in range(K):
                err, done, rew, ng, oh, og, ep = self.refs[i].step(acts[s, i])
                if i in self.diverged:
                    continue
                assert got["err"][s, i] == err and got["done"][s, i] == done, (i, s)
                left = err & ~(STEP_AFTER_DONE | BAD_ACTION) and not self.cfg.auto_reset
                if not (close(got["rew"][s, i], rew) and (left or got["obs_h"] is None or
                                                          close(got["obs_h"][s, i], oh) and close(got["obs_g"][s, i], og))):
                    self.diverged.add(i)
                    continue
                self.ret[i] += got["rew"][s, i]
                assert (el[s, i] >= 0) == (ep is not None), (i, s, el[s, i], ep)
                if ep is not None:
                    assert el[s, i] == ep[1], (i, s, el[s, i], ep[1])
                    assert np.array_equal(er[s, i], self.ret[i]) and close(er[s, i], ep[0]), (i, s, er[s, i], ep[0])
                    if eg is not None:
                        assert np.array_equal(eg[s, i], ep[2]), (i, s, eg[s, i], ep[2])
                    self.episodes += 1
                    self.lengths.append(int(el[s, i]))
                if done and self.cfg.auto_reset:
                    self.ret[i] = 0.0
            if i not in self.diverged:
                check_rows_sum_to_stats(er[:, i], el[:, i], got["stats"][i])
        return got


def check_rows_sum_to_stats(er, el, st):
    """One env's rows of one launch: counting rows, the sum of lengths and the step-order sum of returns equal its
    statistics exactly."""
    ret = np.zeros(2)
    for r in er:
        ret = ret + r
    assert (el >= 0).sum() == st[EPISODES] and el[el >= 0].sum() == st[LENGTH], (el, st)
    assert np.array_equal(ret, st[[RET_H, RET_G]]), (ret, st)


@pytest.mark.parametrize("auto_reset", [0, 1])
@pytest.mark.parametrize("preset", ["GAME", "TRAIN"])
def test_time_limit_end(fresh_scratch, preset, auto_reset, trig):
    """Envs from T - 3 to T + 2 over three launches of 3 steps.  The TimeLimit row at T counts with length T; without
    auto-reset the raw row at T + 1 and the refusals after it give -1."""
    oracle = fresh_scratch
    cfg, ocfg = configs(oracle, preset, V2, 1, auto_reset)
    T = 4500 if preset == "GAME" else 300
    starts = [T - 3, T - 2, T - 1, T, T + 1, 0, T - 4, T - 1]
    b = EpBatch(oracle, cfg, ocfg, len(starts))
    for i, st in enumerate(step_near_end(oracle, preset, V2, cfg, starts)):
        b.set_state(i, st)
    rng = np.random.default_rng(1)
    rows = [b.launch(random_actions(rng, cfg, 3, b.M, b.refs[0].o.R))["ep_length"] for _ in range(3)]
    assert not b.diverged, b.diverged
    assert sorted(b.lengths) == [T] * 5 + [T + 1]   # the env injected at T ends on its raw row T + 1
    el = np.concatenate(rows)                     # [9, M]
    assert el[0, 2] == T and el[1, 2] == -1       # the env at T - 1: row T counts, row T + 1 does not
    if not auto_reset:
        assert (el[1:, 2] == -1).all()


@pytest.mark.parametrize("auto_reset", [0, 1])
@pytest.mark.parametrize("env_id", [V2, V0])
@pytest.mark.parametrize("preset", ["GAME", "TRAIN"])
def test_bad_actions_on_live_last_step_and_finished_envs(fresh_scratch, preset, env_id, auto_reset, trig):
    """Unusable actions on live envs, at step T and on finished envs, and as the first step after a reset: that one ends
    an episode of length 0 (the env is left untouched, step counter included)."""
    oracle = fresh_scratch
    cfg, ocfg = configs(oracle, preset, env_id, 1, auto_reset)
    T = 4500 if preset == "GAME" else 300
    R = oracle.OracleEnv(cfg=ocfg).R
    grid = bad_action_grid(cfg, R)
    starts = [0, 10, T - 1, T, T + 1, T + 3]
    M = len(starts) * len(grid)
    b = EpBatch(oracle, cfg, ocfg, M)
    for i, st in enumerate(step_near_end(oracle, preset, env_id, cfg, starts * len(grid))):
        b.set_state(i, st)
    rng = np.random.default_rng(2)
    acts = random_actions(rng, cfg, 4, M, R)
    for i in range(M):
        acts[0 if starts[i % len(starts)] == 0 else 1, i] = grid[i // len(starts)]
    got = b.launch(acts)
    assert not b.diverged, b.diverged
    zero = [i for i in range(M) if starts[i % len(starts)] == 0]
    assert (got["ep_length"][0, zero] == 0).all() and (got["ep_return"][0, zero] == 0.0).all()
    assert 0 in b.lengths


@pytest.mark.parametrize("auto_reset", [0, 1])
@pytest.mark.parametrize("rec", RAISED, ids=[f"{r[0].split('/')[-1]}:{r[1]}:{r[2]}" for r in RAISED])
def test_rows_on_which_the_reference_raises(fresh_scratch, rec, auto_reset):
    """The golden records on which the reference raises, injected two steps earlier: the aborted row counts an episode
    of its length whose return leaves that row's reward out."""
    oracle = fresh_scratch
    from emul import emul_episodes
    emul_episodes.use_libm_sincos(True)
    try:
        path, i, t = rec
        preset, env_id, _ = parse_name(path)
        d = np.load(path)
        cfg, ocfg = configs(oracle, preset, env_id, 1, auto_reset)
        back = min(t, 2)
        st = state_at(d, i, t - back)
        b = EpBatch(oracle, cfg, ocfg, 1)
        b.set_state(0, st)
        acts = np.stack([actions_at(d, i, t - q) for q in range(back, -1, -1)])
        if auto_reset:
            acts = np.concatenate([acts, acts[:2]])
        got = b.launch(acts[:, None])
        assert not b.diverged
        assert got["err"][back, 0] != 0 and got["ep_length"][back, 0] == int(st["step"]) + back + 1
    finally:
        emul_episodes.use_libm_sincos(False)


@pytest.mark.parametrize("preset", ["GAME", "TRAIN"])
def test_set_state_and_reset_discard_the_partial_return(fresh_scratch, preset, trig):
    oracle = fresh_scratch
    cfg, ocfg = configs(oracle, preset, V2, 1, 1)
    T = 4500 if preset == "GAME" else 300
    b = EpBatch(oracle, cfg, ocfg, 6)
    states = step_near_end(oracle, preset, V2, cfg, [T - 8] * 6)
    for i, st in enumerate(states):
        b.set_state(i, st)
    rng = np.random.default_rng(5)
    R = b.refs[0].o.R
    b.launch(random_actions(rng, cfg, 4, 6, R))
    for i in (0, 1):
        b.set_state(i, states[i])
    mask = np.zeros(6, bool); mask[[2, 3]] = True
    b.reset(mask)
    for i in (2, 3):
        st = b.emul.get_state(i); st["step"] = np.int32(T - 3)
        b.set_state(i, st)
    b.launch(random_actions(rng, cfg, 8, 6, R))
    assert not b.diverged and b.episodes == 6 and set(b.lengths) == {T}


@pytest.mark.parametrize("path", GOALS, ids=[p.split("/")[-1] for p in GOALS])
def test_goal_ended_episodes(fresh_scratch, path):
    """Goal scoring (RoboRugby-v0 and the DuelGoals composition): ep_goals of every counting row equals the oracle's goal
    state of that row, destroyed goals and emptied fields included."""
    oracle = fresh_scratch
    from emul import emul_episodes
    emul_episodes.use_libm_sincos(True)
    try:
        preset, env_id, _ = parse_name(path)
        d = np.load(path)
        n, T = d["act"].shape[:2]
        for auto_reset in (0, 1):
            cfg, ocfg = configs(oracle, preset, env_id, 1, auto_reset, goals=True)
            b = EpBatch(oracle, cfg, ocfg, n)
            for i in range(n):
                b.set_state(i, state_at(d, i, 0))
            acts = np.nan_to_num(d["act"], nan=0.0).transpose(1, 0, 2)
            goals = []
            for s0 in range(0, T, 55):
                g = b.launch(acts[s0:s0 + 55])
                goals.append(g["ep_goals"][g["ep_length"] >= 0])
            goals = np.concatenate(goals)
            print(f"{path.split('/')[-1]} auto_reset={auto_reset}: {b.episodes} episodes, {len(b.diverged)} diverged, "
                  f"destroyed bits {np.unique(goals[:, 2])}")
            assert len(b.diverged) <= n // 2 and b.episodes > 0
            assert (goals[:, 2] != 0).any() or (goals[:, 3] == 0).any()   # an episode ended by the goals
    finally:
        emul_episodes.use_libm_sincos(False)


# ------------------------------------------------------------------------------------------ pool rows

def _pool(layout, M, m, seed, before_end=4):
    """A batch and m pool rows saved mid-episode a few steps before the time limit, with what each row holds: its
    return (the step-order sum of the source's reward rows since rr_set_state) and its step counter."""
    from emul import emul_episodes, emul_states
    rng = np.random.default_rng(seed)
    cfg = make_cfg(*layout)
    src = batch(cfg, m)
    T = 4500 if cfg.preset == 0 else 300
    for i in range(m):
        st = src.get_state(i)
        st["step"] = np.int32(T - before_end - 3 - (i % 3))
        src.set_state(i, st)
    g = emul_episodes.launch(src, actions(rng, src, 3))
    assert (g["done"] == 0).all()
    ret = np.zeros((m, 2))
    for s in range(3):
        ret = ret + g["rew"][s]
    steps = np.array([int(src.get_state(i)["step"]) for i in range(m)])
    start = rng.normal(size=(3 * src.R + 2 * src.B, m)) * 100.0
    rows = emul_states.save(src, start)
    a = batch(cfg, M)
    start_a = rng.normal(size=(3 * a.R + 2 * a.B, M)) * 100.0
    return rng, cfg, a, start_a, rows, ret, steps


@pytest.mark.parametrize("layout", [("TRAIN", False, False), ("GAME", True, False), ("TRAIN", True, True)])
def test_pool_row_saved_mid_episode_continues_its_return_and_length(layout):
    """Every episode a pool reset starts ends with return = the row's saved return + the rewards that follow (fp64, in
    step order) and length = the row's step counter + the rows that follow.  The slot each episode started from is
    reset_slot forward-filled over k (INTEGRATION.md §5)."""
    from emul import emul_episodes
    M, m, K = (12, 4, 40) if layout[0] == "TRAIN" else (4, 3, 20)
    rng, cfg, a, start, rows, ret, steps = _pool(layout, M, m, 41)
    a_start = np.full(M, -1)
    from emul import emul_states
    first = rng.integers(0, m, M)
    emul_states.load(a, start, rows, first)
    a_start[:] = first
    g = emul_episodes.launch(a, actions(rng, a, K), start, rows, None, 1.0)
    slot, el, er = g["slot"], g["ep_length"], g["ep_return"]
    n = 0
    for i in range(M):
        origin, acc, length = a_start[i], ret[a_start[i]].copy(), steps[a_start[i]]
        for s in range(K):
            acc = acc + g["rew"][s, i]
            length += 1
            if el[s, i] >= 0:
                assert el[s, i] == length and np.array_equal(er[s, i], acc), (i, s, origin)
                n += 1
            if g["done"][s, i]:
                assert slot[s, i] >= 0
                origin = slot[s, i]
                acc, length = ret[origin].copy(), steps[origin]
        check_rows_sum_to_stats(er[:, i], el[:, i], g["stats"][i])
    print(f"{layout}: {n} episodes continued from pool rows")
    assert n >= 2 * M


def test_pool_row_saved_from_a_finished_episode_counts_nothing():
    """A row saved after its episode was counted: the next step on it is refused (STEP_AFTER_DONE), reports done, -1 and
    0.0, and adds no episode; the reset after it draws again."""
    from emul import emul_episodes, emul_states
    cfg0 = make_cfg("TRAIN", False, False)
    cfg0.auto_reset = 0
    fin = batch(cfg0, 2)
    for i in range(2):
        st = fin.get_state(i)
        st["step"] = np.int32(299)
        fin.set_state(i, st)
    g = emul_episodes.launch(fin, np.zeros((2, 2, 1)))
    assert (g["ep_length"][0] == 300).all() and (g["ep_length"][1] == -1).all()   # counted at T; raw row T + 1
    rows = emul_states.save(fin, np.zeros((5, 2)))
    cfg = make_cfg("TRAIN", False, False)
    a = batch(cfg, 3)
    start = np.zeros((5, 3))
    emul_states.load(a, start, rows, np.array([0, 1, 0]))
    g = emul_episodes.launch(a, np.zeros((2, 3, 1)), start, rows, None, 1.0)
    assert (g["err"][0] == STEP_AFTER_DONE).all() and (g["done"][0] == 1).all()
    assert (g["ep_length"][0] == -1).all() and (g["ep_return"][0] == 0.0).all()
    assert (g["slot"][0] >= 0).all() and (g["err"][1] == STEP_AFTER_DONE).all()   # the pool only holds finished rows
    assert (g["ep_length"] == -1).all() and (g["stats"][:, EPISODES] == 0).all()


@pytest.mark.parametrize("pooled", [False, True])
@pytest.mark.parametrize("layout", [("TRAIN", True, False), ("GAME", False, True)])
def test_one_launch_equals_one_step_launches(layout, pooled):
    """The episode rows of one K-step launch equal those of K one-step launches from the same state, and every other
    output and the final state equal those of rr_step_pool's / rr_step_info's launch (emul_pool / emul_info)."""
    from emul import emul_episodes, emul_info, emul_pool
    M, m, K = (16, 4, 30) if layout[0] == "TRAIN" else (4, 3, 12)
    rng, cfg, a, start_a, rows, _, _ = _pool(layout, M, m, 43)
    from emul import emul_states
    emul_states.load(a, start_a, rows, rng.integers(0, m, M))
    b = batch(cfg, M)
    b.sf[...] = a.sf; b.si[...] = a.si
    c = batch(cfg, M)
    c.sf[...] = a.sf; c.si[...] = a.si
    start_b, start_c = start_a.copy(), start_a.copy()
    acts = actions(rng, a, K)
    pool = (rows, None, 1.0) if pooled else (None, None, 1.0)
    whole = emul_episodes.launch(a, acts, start_a, *pool)
    parts = [emul_episodes.launch(b, acts[s:s + 1], start_b, *pool) for s in range(K)]
    for key in ("ep_return", "ep_length", "ep_goals", "rew", "done", "flags", "slot"):
        if whole[key] is None:
            continue
        assert _same(whole[key], np.concatenate([p[key] for p in parts])), key
    assert _same(a.sf, b.sf) and _same(a.si, b.si) and _same(start_a, start_b)
    ref = emul_pool.launch(c, start_c, acts, rows, None, 1.0) if pooled else emul_info.launch(c, acts, observe=True)
    for key in ("rew", "done", "err", "naughty", "obs_h", "obs_g", "final_h", "final_g", "flags", "stats"):
        assert _same(whole[key], ref[key]), key
    assert _same(a.sf, c.sf) and _same(a.si, c.si)
    assert (whole["done"] != 0).sum() >= M and (whole["ep_length"] >= 0).any()
