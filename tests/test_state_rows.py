"""CPU tier: saved env rows (rr_save_states / rr_load_states, include/rr_b200.h) through the host build of the kernel source
(tests/emul emul_states: rr_sim.cuh's row layout and index rules on EmulBatch columns plus a start array).

A row is every sf column, the starting layout, every si column and zero padding to 16 bytes; its width identifies the
layout.  A save skips indices outside [0, N) and leaves their rows unwritten; a load skips negative indices and indices
>= m and leaves those envs untouched.  A batch loaded from rows saved out of another batch continues that batch's rows bit
for bit: with the same env indices including every auto-reset, in other slots up to the first done row."""
import numpy as np
import pytest

from golden_util import apply_overrides, resolve_env

WIDTHS = {("GAME", False, False): 1104, ("GAME", True, False): 1184, ("GAME", False, True): 1328,
          ("GAME", True, True): 1408, ("TRAIN", False, False): 224, ("TRAIN", True, False): 240,
          ("TRAIN", False, True): 272, ("TRAIN", True, True): 288}
LAYOUTS = sorted(WIDTHS)


def make_cfg(preset, goals, prior, env_id="RoboRugbySimpleDuel-v2", seed=11, env_offset=40):
    from roborugby_b200 import _lib
    if prior:
        env_id = "DuelAllCoordsPrior"
    base, _ = resolve_env(env_id)
    cfg = apply_overrides(_lib.default_config(_lib.PRESET_GAME if preset == "GAME" else _lib.PRESET_TRAIN, base), env_id)
    cfg.goal_scoring, cfg.seed, cfg.env_offset = int(goals), seed, env_offset
    return cfg


def batch(cfg, M):
    from emul.emul import EmulBatch
    R, B = (4, 8) if cfg.preset == 0 else (1, 1)
    D = {1: 5, 2: 11, 4: 6 * R + 4 * B}.get(cfg.observer, 0)
    return EmulBatch(cfg, M, R, B, D)


def start_cols(b, rng):
    """A start array [3R + 2B, M] of arbitrary doubles (the host build has no k_init to record one)."""
    return rng.normal(size=(3 * b.R + 2 * b.B, b.M)) * 100.0


def expected_row(b, start, e, width):
    raw = b"".join(np.ascontiguousarray(a[:, e]).tobytes() for a in (b.sf, start, b.si))
    assert len(raw) <= width < len(raw) + 16 and width % 16 == 0
    return np.frombuffer(raw + bytes(width - len(raw)), np.uint8)


def desync(b, rng, K=6):
    """Episode phases spread as bench.py spreads them, then one launch so that rows carry returns, counted bits, error
    masks, naughty counts and episode counters that are not those of a fresh reset."""
    T = 4500 if b.cfg.preset == 0 else 300
    for i in range(b.M):
        st = b.get_state(i)
        st["step"] = np.int32(T - 1 - 4 * (i // 2) if i % 2 else (i * 37) % (T - 1))   # odd envs end one after another
        b.set_state(i, st)
    b.launch(actions(rng, b, K))


def _same(a, b):
    """Bit-identical (NaN rows included)."""
    if a is None or b is None:
        return a is b
    return np.array_equal(np.ascontiguousarray(a).view(np.uint8), np.ascontiguousarray(b).view(np.uint8))


def actions(rng, b, K):
    if b.cfg.discrete:
        return rng.integers(0, 8, (K, b.M, b.R)).astype(np.float64)
    return rng.choice([-1.0, -0.5, 0.0, 0.5, 1.0], (K, b.M, 2 * b.R))


@pytest.mark.parametrize("layout", LAYOUTS)
def test_row_width_identifies_the_layout(layout):
    from emul import emul_states
    preset, goals, prior = layout
    assert emul_states.row_bytes(make_cfg(preset, goals, prior)) == WIDTHS[layout]
    assert len(set(WIDTHS.values())) == len(WIDTHS)


@pytest.mark.parametrize("layout", LAYOUTS)
def test_round_trip_with_permutation_mask_and_out_of_range_indices(layout):
    from emul import emul_states
    rng = np.random.default_rng(5)
    cfg = make_cfg(*layout)
    M, S = 7, WIDTHS[layout]
    src = batch(cfg, M)
    start = start_cols(src, rng)
    desync(src, rng)
    # save: a permutation with a duplicate, a negative index and two past the end
    envs = np.array([3, -1, 0, M, 6, 3, M + 100, 1, 5])
    rows = np.full((len(envs), S), 0xAB, np.uint8)
    emul_states.save(src, start, envs, rows)
    for j, e in enumerate(envs):
        if 0 <= e < M:
            assert np.array_equal(rows[j], expected_row(src, start, e, S)), (j, e)
        else:
            assert (rows[j] == 0xAB).all(), (j, e)                # an index outside [0, N) leaves its row unwritten
    # two saves of one state are byte-equal, padding included
    assert np.array_equal(emul_states.save(src, start), emul_states.save(src, start))
    # load into another batch: negative slots and slots >= m leave the env as it was
    dst = batch(cfg, M)
    dstart = start_cols(dst, rng)
    desync(dst, rng, K=3)
    before = (dst.sf.copy(), dst.si.copy(), dstart.copy())
    slots = np.array([2, -1, len(envs), 0, -5, 8, len(envs) + 7])
    emul_states.load(dst, dstart, rows, slots)
    for i, r in enumerate(slots):
        got = np.concatenate([np.ascontiguousarray(a[:, i]).view(np.uint8) for a in (dst.sf, dstart, dst.si)])
        if 0 <= r < len(envs):
            assert np.array_equal(got, rows[r][:got.size]), (i, r)
        else:
            for a, b0 in zip((dst.sf, dst.si, dstart), before):
                assert _same(a[:, i], b0[:, i]), (i, r)


@pytest.mark.parametrize("layout", [("GAME", False, False), ("GAME", True, False), ("GAME", False, True),
                                    ("TRAIN", False, False), ("TRAIN", True, True)])
def test_loaded_batch_continues_the_saved_one(layout):
    """Rows saved out of one batch and loaded into a fresh batch (same config) into the same env indices: the next
    launches are bit-identical, auto-resets included (same destination index and episode counter)."""
    from emul import emul_states
    rng = np.random.default_rng(9)
    cfg = make_cfg(*layout)
    M = 6
    src = batch(cfg, M)
    start = start_cols(src, rng)
    desync(src, rng)
    rows = emul_states.save(src, start)
    dst = batch(cfg, M)
    dstart = start_cols(dst, rng)
    emul_states.load(dst, dstart, rows)
    ends = 0
    for _ in range(2):
        acts = actions(rng, src, 8)
        a, b = src.launch(acts, observe=True), dst.launch(acts, observe=True)
        for key in ("rew", "done", "err", "naughty", "obs_h", "obs_g", "stats"):
            assert _same(a[key], b[key]), key
        ends += int(a["done"].sum())
    assert ends                                          # episodes ended and were reset inside the launches
    assert _same(src.sf, dst.sf) and _same(src.si, dst.si) and _same(start, dstart)
    for i in range(M):
        for k, v in src.get_state(i).items():
            assert _same(v, dst.get_state(i)[k]), (i, k)


@pytest.mark.parametrize("layout", [("GAME", True, True), ("TRAIN", False, False)])
def test_loaded_rows_in_other_slots_repeat_the_source_until_its_first_done(layout):
    from emul import emul_states
    rng = np.random.default_rng(13)
    cfg = make_cfg(*layout)
    M = 6
    src = batch(cfg, M)
    start = start_cols(src, rng)
    desync(src, rng)
    perm = rng.permutation(M)
    rows = emul_states.save(src, start, perm)
    dst = batch(cfg, M)
    emul_states.load(dst, start_cols(dst, rng), rows)        # env i <- row i = env perm[i] of src
    acts = actions(rng, src, 10)
    a = src.launch(acts, observe=True)
    b = dst.launch(acts[:, perm], observe=True)            # each env the actions of the env its row came from
    for i in range(M):
        e = perm[i]
        done = np.nonzero(a["done"][:, e])[0]
        last = int(done[0]) if done.size else acts.shape[0] - 1
        for key in ("rew", "done", "err", "naughty"):
            assert _same(a[key][:last + 1, e], b[key][:last + 1, i]), (i, key)
        if a["obs_h"] is not None:
            assert _same(a["obs_h"][:last, e], b["obs_h"][:last, i])
