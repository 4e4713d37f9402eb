"""GPU tier (B200): saved env rows on the device (rr_save_states / rr_load_states, RoboRugbyVecEnv.save_states /
load_states, copy.deepcopy of both env classes).

A load puts back every per-env value a handle keeps between calls: after save, step, load and the same step again, every
output (observations, rewards, done, terminal observations, row flags), the statistics counts and every state accessor
are bit-identical, resets inside the launch included.  The statistics returns are sums whose per-warp atomics may land in
another order, so they are held to 1e-12 relative.  No test here sends an out-of-range index to the device: the skip
rules are tested on the host build (test_state_rows.py), and the refusals below fire before anything is launched."""
import copy

import numpy as np
import pytest

from parity_util import close

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

V0, V2 = "RoboRugby-v0", "RoboRugbySimpleDuel-v2"
RET = [1, 2]
COUNTS = [0, 3, 4, 5, 6, 7]
E_INVALID = -1


def _venv(n, preset="GAME", env_id=V2, **kw):
    from roborugby_b200.vec_env import RoboRugbyVecEnv
    kw.setdefault("time_limit", True)
    kw.setdefault("auto_reset", True)
    kw.setdefault("strict_reset", True)
    return RoboRugbyVecEnv(env_id, n, preset=preset, device="cuda:0", seed=kw.pop("seed", 2026), **kw)


def _desync(env):
    """bench.py's episode phases: resets fall inside every launch."""
    st = env.get_state()
    st["step"][:] = (np.arange(env.num_envs) * 7919) % max(env.max_episode_steps - 1, 1)
    env.set_state(st)


def _actions(env, K, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    if env.discrete:
        return torch.randint(0, 8, (K, env.num_envs, env.action_dim), generator=g, dtype=torch.uint8, device="cuda")
    return torch.rand((K, env.num_envs, env.action_dim), generator=g, device="cuda") * 2 - 1


def _report(env, goals=False):
    """What every host accessor reports for every env."""
    st = env.get_state()
    out = {f"state.{k}": v for k, v in st.items()}
    out["error_mask"] = env.error_mask()
    out["last_naughty"] = env.last_naughty()
    rob3, ball2 = env.get_starting_positions()
    out["start.rob3"], out["start.ball2"] = rob3, ball2
    if goals:
        out.update({f"goal.{k}": v for k, v in env.goal_state().items()})
    if env.obs_dim:
        oh, og = env.observe()
        out["observe.h"], out["observe.g"] = oh.cpu().numpy(), og.cpu().numpy()
        if env.cfg.observer not in (3, 4):
            out["observe_entity"] = env.observe_entity(env.num_robots - 1, env.num_balls - 1).cpu().numpy()
    out["assign_balls"] = env.assign_balls(list(range(env.num_robots))[:2]).cpu().numpy()
    return out


def _bits(a):
    return None if a is None else np.ascontiguousarray(np.asarray(a)).view(np.uint8)


def _eq(a, b):
    """Bit-identical (None only against None)."""
    if a is None or b is None:
        return a is b
    return np.array_equal(_bits(a), _bits(b))


def _assert_same(a, b, where=""):
    assert a.keys() == b.keys()
    for k in a:
        assert _eq(a[k], b[k]), f"{where}{k}"


def _run(env, acts, join=True):
    """One step_k call with final_info; host copies of every output (terminal observations only on done rows)."""
    K = acts.shape[0]
    env.clear_stats()
    obs_h, obs_g, rew, done, info = env.step_k(acts, K, join=join, final_info=True)
    if not join:
        env.join()
    d = done.cpu().numpy()
    out = dict(obs_h=obs_h.cpu().numpy(), obs_g=obs_g.cpu().numpy(), rew=rew.cpu().numpy(), done=d,
               row_flags=info["row_flags"].cpu().numpy(),
               final_h=info["final_obs"].cpu().numpy()[d == 1], final_g=info["final_obs_grumpy"].cpu().numpy()[d == 1])
    stats = env.stats.cpu().numpy()
    return out, stats


def _round_trip(env, K=32, goals=False, seed=1):
    """save all, step_k, load all, the same step_k: every output, the statistics and every accessor bit-identical."""
    _desync(env)
    env.step_k(_actions(env, K, seed + 100), K)          # rows with returns, counted bits, error masks, naughty counts
    before = _report(env, goals)
    rows = env.save_states()
    acts = _actions(env, K, seed)
    out_a, st_a = _run(env, acts)
    after_a = _report(env, goals)
    launches = env.launch_count
    env.load_states(rows)
    assert env.launch_count == launches + 1
    _assert_same(before, _report(env, goals), "after load: ")
    out_b, st_b = _run(env, acts)
    _assert_same(out_a, out_b, "rows: ")
    _assert_same(after_a, _report(env, goals), "after the second step_k: ")
    assert np.array_equal(st_a[COUNTS], st_b[COUNTS]), (st_a, st_b)
    assert np.allclose(st_a[RET], st_b[RET], rtol=1e-12, atol=0), (st_a, st_b)
    assert out_a["done"].any() and st_a[0] > 0                 # episodes ended (and were reset) inside the launch
    return rows


@pytest.mark.parametrize("pipeline", [128, 1])
def test_round_trip_at_the_baseline_configuration(pipeline):
    env = _venv(65536, pipeline=pipeline)
    rows = _round_trip(env)
    assert rows.shape == (65536, 1104) and rows.dtype == torch.uint8 and rows.is_contiguous()
    env.close()


@pytest.mark.parametrize("case", ["train", "goals_wide", "prior", "v0_continuous", "f64"])
def test_round_trip_in_other_configurations(case):
    kw, n, goals, width = {}, 8192, False, 1104
    if case == "train":
        kw, width = dict(preset="TRAIN"), 224
    elif case == "goals_wide":   # one stream-ordered launch over more envs than 384-thread blocks cover: 448 threads
        kw, n, goals, width = dict(goal_scoring=True), 65536, True, 1184
    elif case == "prior":
        kw, width = dict(observer=4, goal_scoring=True), 1408
        goals = True
    elif case == "v0_continuous":
        kw = dict(env_id=V0)
    elif case == "f64":
        kw = dict(out_dtype=torch.float64, pipeline=8)
    env = _venv(n, **kw)
    assert env.state_row_bytes == width
    _round_trip(env, goals=goals)
    env.close()


def test_clone_of_one_env_into_every_slot(oracle):
    N, K = 4096, 32
    env = _venv(N, out_dtype=torch.float64)
    _desync(env)
    env.step_k(_actions(env, 8, 5), 8)
    steps = env.get_state()["step"]
    src = int(np.nonzero((steps > 100) & (steps < env.max_episode_steps - 100))[0][7])   # mid-episode
    src_state = {k: v[src] for k, v in env.get_state().items()}
    row = env.save_states(torch.tensor([src], device="cuda"))
    acts = _actions(env, K, 6)
    want, _ = _run(env, acts)                                  # the source's own continuation
    env.load_states(row, torch.zeros(N, dtype=torch.int64, device="cuda"))
    got, _ = _run(env, acts[:, src:src + 1].expand(K, N, env.action_dim).contiguous())
    d = np.nonzero(want["done"][:, src])[0]
    last = int(d[0]) if d.size else K - 1
    for key in ("obs_h", "obs_g", "rew", "done", "row_flags"):
        w = want[key][:last + 1, src]
        assert np.array_equal(_bits(got[key][:last + 1]), _bits(np.broadcast_to(w[:, None], got[key][:last + 1].shape))), key
    # the source continuation against the oracle from the saved state
    oracle.scratch_mode(1)
    o = oracle.OracleEnv("GAME", V2, time_limit=True)
    o.set_state(src_state)
    a = acts[:, src].cpu().numpy()
    for s in range(last + 1):
        r = o.step(a[s])
        for i in (0, 1000, N - 1):
            assert close(r["rew"], got["rew"][s, i]) and r["done"] == got["done"][s, i], (s, i)
            assert r["done"] or close(r["obs_h"], got["obs_h"][s, i]), (s, i)   # (a done row's obs is after its reset)
    oracle.scratch_mode(0)
    env.close()


def test_permutation_and_mask():
    N = 4096
    env = _venv(N, goal_scoring=True)
    _desync(env)
    env.step_k(_actions(env, 16, 7), 16)
    saved = _report(env, goals=True)
    rows = env.save_states()
    env.step_k(_actions(env, 16, 8), 16)
    current = _report(env, goals=True)
    rng = np.random.default_rng(3)
    slots = rng.permutation(N)
    slots[rng.random(N) < 0.1] = -1
    env.load_states(rows, torch.as_tensor(slots, device="cuda"))
    now = _report(env, goals=True)
    keep = slots < 0
    assert keep.any() and (~keep).any()
    for k in now:
        assert np.array_equal(_bits(now[k][keep]), _bits(current[k][keep])), k
        assert np.array_equal(_bits(now[k][~keep]), _bits(saved[k][slots[~keep]])), k
    env.close()


def test_save_orders_behind_pipelined_steps_and_loads_order_before_them():
    N, K = 16384, 16
    a, b = _venv(N, pipeline=128), _venv(N, pipeline=1)
    for env in (a, b):
        _desync(env)
    acts = [_actions(a, K, 20 + c) for c in range(2)]
    for x in acts:
        a.step_k(x, K, join=False)
        b.step_k(x, K)
    rows_a = a.save_states()                                   # no explicit join
    rows_b = b.save_states()
    assert torch.equal(rows_a, rows_b)
    assert torch.equal(rows_a, a.save_states())                # two saves of one state are byte-equal
    # a load issued behind a pipelined step_k, followed by another one: the second steps the loaded state
    want, _ = _run(b, acts[0])
    a.step_k(acts[1], K, join=False)
    a.load_states(rows_a)
    got, _ = _run(a, acts[0], join=False)
    _assert_same(want, got)
    assert torch.equal(a.save_states(), b.save_states())
    a.close(); b.close()


def test_rows_continue_in_another_handle():
    N, K = 8192, 32
    a, b = _venv(N), _venv(N)
    _desync(a)
    a.step_k(_actions(a, K, 30), K)
    rows = a.save_states()
    b.load_states(rows.cpu().to("cuda"))                       # through host memory, as between processes
    for c in range(3):                                         # resets included: same seed, same env_offset
        acts = _actions(a, K, 31 + c)
        _assert_same(_run(a, acts)[0], _run(b, acts)[0], f"launch {c}: ")
    _assert_same(_report(a), _report(b))
    a.close(); b.close()


def test_refusals_launch_nothing():
    N = 256
    env = _venv(N)
    lib, h, st = env.lib, env._h, env._stream()
    S = env.state_row_bytes
    buf = torch.zeros((N + 2) * S + 16, dtype=torch.uint8, device="cuda")
    idx = torch.zeros(4, dtype=torch.int64, device="cuda")
    n0 = env.launch_count
    p = buf.data_ptr()
    for rc in (lib.rr_save_states(h, None, N, p + 8, st),          # misaligned rows
               lib.rr_load_states(h, p + 8, N, None, st),
               lib.rr_save_states(h, None, 0, p, st),              # m < 1
               lib.rr_load_states(h, p, 0, idx.data_ptr(), st),
               lib.rr_save_states(h, None, N + 1, p, st),          # NULL env indices: m <= N
               lib.rr_load_states(h, p, N - 1, None, st),          # NULL slots: m == N
               lib.rr_save_states(h, idx.data_ptr() + 4, 2, p, st),  # misaligned indices
               lib.rr_save_states(None, None, 1, p, st),
               lib.rr_load_states(h, None, N, None, st)):
        assert rc == E_INVALID
    assert env.launch_count == n0
    rows = env.save_states()
    n1 = env.launch_count
    with pytest.raises(IndexError):
        env.save_states(torch.tensor([0, N]))
    with pytest.raises(IndexError):
        env.save_states(torch.tensor([-1, 0]))
    with pytest.raises(IndexError):
        env.load_states(rows[:4].clone(), torch.tensor([0, 4] + [-1] * (N - 2)))
    for bad in (rows[:, :-16].contiguous(), rows.view(torch.int32), rows.cpu(),
                torch.zeros(N, 2 * S, dtype=torch.uint8, device="cuda")[:, :S]):
        with pytest.raises(ValueError):
            env.load_states(bad)
    with pytest.raises(ValueError):
        env.load_states(rows[:8].clone())                          # no slots: N rows
    with pytest.raises(ValueError):
        env.save_states(out=torch.zeros(N, S - 16, dtype=torch.uint8, device="cuda"))
    assert env.launch_count == n1
    out = torch.empty_like(rows)
    assert env.save_states(out=out) is out and torch.equal(out, rows)
    env.close()


def test_deepcopy_of_a_vec_env_continues_bit_identically():
    N, K = 4096, 32
    env = _venv(N, pipeline=4)
    _desync(env)
    env.step_k(_actions(env, K, 40), K)
    twin = copy.deepcopy(env)
    assert twin.pipeline == 4 and twin._h.value != env._h.value
    assert torch.equal(twin.stats, env.stats)
    for c in range(2):
        acts = _actions(env, K, 41 + c)
        _assert_same(_run(env, acts)[0], _run(twin, acts)[0], f"launch {c}: ")
    env.close(); twin.close()


def test_deepcopy_of_a_gym_env_continues_like_the_original():
    import roborugby_b200 as rr
    env = rr.make(V2)
    env.reset()
    rng = np.random.default_rng(1)
    for _ in range(25):
        env.step(list(rng.integers(0, 8, 4)))
    twin = copy.deepcopy(env)
    assert twin._elapsed == env._elapsed == 25 and twin._reward == env._reward
    assert twin.lstRobots[0]._env is twin
    for _ in range(40):
        a = list(rng.integers(0, 8, 4))
        o1, r1, d1, i1 = env.step(a)
        o2, r2, d2, i2 = twin.step(a)
        assert (r1, d1, dict(i1)) == (r2, d2, dict(i2)) and _eq(i1.adblGrumpyState, i2.adblGrumpyState)
        assert _eq(o1, o2)
    assert twin._elapsed == env._elapsed == 65
    _assert_same(env.get_state(), twin.get_state())
    env.close(); twin.close()
