"""GPU tier (B200): the device statistics vector (RR_STAT_*) against a host sum over the kernel's own rows.

The reference run steps a handle one launch per step and reads, after every call, the fp64 rewards, done,
rr_error_mask(clear=1), rr_last_naughty and the step counter; the host applies the rules of rr_get_stats
(include/rr_b200.h) per env and sums in fp64.  Counts must be exact.  A device return is a sum of the same terms in
another order (warp shuffles, one atomic per warp): |device - fsum| <= n * 2^-52 * sum |terms|.  Every other way of
issuing the same steps (one fused launch, sub-batch pipelines, the host-buffer entry points, NULL outputs) must give
the same."""
import copy
import ctypes
import math
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

STEP_AFTER_DONE, BAD_ACTION = 1, 512
EPISODES, RET_H, RET_G, LENGTH, NAUGHTY, ERRORS, STEPS, REPLAYS = range(8)
INT_STATS = [EPISODES, LENGTH, NAUGHTY, ERRORS, STEPS]
V0, V2 = "RoboRugby-v0", "RoboRugbySimpleDuel-v2"


def _venv(n, preset, env_id=V2, **kw):
    from roborugby_b200.vec_env import RoboRugbyVecEnv
    kw.setdefault("time_limit", True)
    kw.setdefault("auto_reset", True)
    kw.setdefault("out_dtype", torch.float64)
    kw.setdefault("strict_reset", True)
    return RoboRugbyVecEnv(env_id, n, preset=preset, device="cuda:0", seed=kw.pop("seed", 13), **kw)


def _start(env, seed=0):
    """The handle's own placement with step counters spread over the last steps of an episode (and one past it):
    episodes end inside the launches, envs injected past their end are refused and reset."""
    st = env.get_state()
    T = env.max_episode_steps
    rng = np.random.default_rng(seed)
    st["step"] = (T - rng.integers(-1, 9, env.num_envs)).astype(np.int32)
    env.set_state(st)
    return st


def _actions(env, K, seed=1, bad=0.02):
    """Discrete ids 0..7 with a share of ids above 7 (BAD_ACTION rows)."""
    g = np.random.default_rng(seed)
    a = g.integers(0, 8, (K, env.num_envs, env.num_robots))
    a[g.random(a.shape[:2]) < bad, 0] = 9
    return torch.as_tensor(a.astype(np.uint8))


class HostSum:
    """The rules table over one handle's rows, per env: integer statistics and the terms of each return."""

    def __init__(self, n):
        self.counted = np.zeros(n, bool)
        self.ret = np.zeros((n, 2))
        self.ints = np.zeros(8, np.int64)
        self.terms = [[], []]                 # (happy, grumpy) returns of the counted episodes
        self.per_env = np.zeros((n, 8))

    def cleared(self):
        """A copy that goes on from the same envs (returns gathered so far, episodes already counted) with the
        statistics zeroed: what the device vector holds after rr_clear_stats."""
        c = copy.deepcopy(self)
        c.ints[:] = 0
        c.terms = [[], []]
        c.per_env[:] = 0.0
        return c

    def row(self, step_before, rew, done, err, naughty, auto_reset):
        refused = (err & STEP_AFTER_DONE) != 0
        aborted = err != 0
        advanced = ~refused & ((err & BAD_ACTION) == 0)
        length = step_before + advanced
        self.ret += rew
        live = ~refused
        first = live & (done != 0) & ~self.counted
        for q, v in ((STEPS, live), (NAUGHTY, np.where(live & ~aborted, naughty, 0)), (ERRORS, live & aborted),
                     (EPISODES, first), (LENGTH, np.where(first, length, 0))):
            self.ints[q] += int(np.sum(v))
            self.per_env[:, q] += v
        for t in range(2):
            self.terms[t] += self.ret[first, t].tolist()
            self.per_env[first, RET_H + t] += self.ret[first, t]
        self.counted |= first
        if auto_reset:
            d = done != 0
            self.ret[d] = 0.0
            self.counted[d] = False

    def check(self, dev, what):
        dev = np.asarray(dev, np.float64)
        assert np.array_equal(dev[INT_STATS], self.ints[INT_STATS].astype(np.float64)), (what, dev, self.ints)
        for t in range(2):
            terms = self.terms[t]
            bound = len(terms) * 2.0 ** -52 * float(np.sum(np.abs(terms)))
            assert abs(dev[RET_H + t] - math.fsum(terms)) <= bound, (what, t, dev[RET_H + t], math.fsum(terms), bound)


def reference_run(env, acts, auto_reset=True, h=None):
    """One launch per step; the host restatement of the rows (continuing `h`, if given)."""
    N = env.num_envs
    h = HostSum(N) if h is None else h
    env.error_mask(clear=True)
    for s in range(acts.shape[0]):
        before = env.get_state()["step"].astype(np.int64)
        _, _, rew, done = env.step_k(acts[s:s + 1].cuda(), 1)
        rew = rew[0].cpu().numpy(); done = done[0].cpu().numpy()
        err = env.error_mask(clear=True).astype(np.int64)
        h.row(before, np.where((err != 0)[:, None], 0.0, rew), done, err, env.last_naughty(), auto_reset)
        assert np.all(rew[err != 0] == 0), "an aborted row has no reward"
    return h


@pytest.mark.parametrize("preset,N", [("TRAIN", 1), ("GAME", 1), ("TRAIN", 31), ("GAME", 33), ("GAME", 385),
                                      ("TRAIN", 20001), ("GAME", 20001), ("GAME", 384 * 148 + 17)])
def test_gpu_stats_of_a_fused_launch_match_the_host_sum_of_its_rows(preset, N):
    """Batches with padding lanes and partial warps (and, above 384 x 148 GAME envs, the 448-thread k_step).  With one
    env there is one lane and one atomic: the device vector equals the host restatement bit for bit."""
    K = 8 if N < 50000 else 5
    ref = _venv(N, preset)
    _start(ref)
    acts = _actions(ref, K)
    ref.clear_stats()
    h = reference_run(ref, acts)
    h.check(ref.stats.cpu().numpy(), "one launch per step")
    fused = _venv(N, preset)
    _start(fused)
    fused.clear_stats()
    fused.step_k(acts.cuda(), K)
    dev = fused.stats.cpu().numpy()
    h.check(dev, "fused")
    assert h.ints[EPISODES] > 0 and h.ints[ERRORS] > 0 or N == 1
    if N == 1:
        assert np.array_equal(dev[:REPLAYS], h.per_env[0, :REPLAYS]), (dev, h.per_env[0])
    ref.close(); fused.close()


def _null_outputs(env, acts):
    from roborugby_b200 import _lib
    a = acts.cuda().contiguous()
    _lib.check(env.lib.rr_step(env._h, a.data_ptr(), a.shape[2], a.shape[0], None, None, None, None, env._stream()))
    torch.cuda.synchronize()


@pytest.mark.parametrize("preset", ["GAME", "TRAIN"])
def test_gpu_stats_do_not_depend_on_the_entry_point(preset):
    """The same steps as one fused launch, as 7- and 128-group sub-batch pipelines without joins between calls, through
    rr_step_host (zero copy, and staged in up to three launches), rr_step_host_begin / _end, and with every output NULL."""
    N, K = 4099, 8
    ref = _venv(N, preset)
    _start(ref)
    acts = _actions(ref, K, seed=4)
    ref.clear_stats()
    h = reference_run(ref, acts)
    ref.close()

    def run(make, how):
        env = make()
        _start(env)
        env.clear_stats()
        how(env)
        torch.cuda.synchronize()
        env.join()
        h.check(env.stats.cpu().numpy(), how.__name__)
        env.close()

    def fused(env): env.step_k(acts.cuda(), K)
    def split(env):
        for s in range(0, K, 3):
            env.step_k(acts[s:s + 3].cuda(), acts[s:s + 3].shape[0], join=env.pipeline == 1)
        env.join()
    def host(env):
        for s in range(0, K, 4):
            env.step_host(acts[s:s + 4].contiguous().pin_memory(), 4)
    def host_begin_end(env):
        hold = [acts[s:s + 2].contiguous().pin_memory() for s in range(0, K, 2)]
        tickets = [env.step_host_begin(a, 2, j % 3) for j, a in enumerate(hold[:3])]
        env.step_host_end(tickets[0])
        tickets.append(env.step_host_begin(hold[3], 2, 0))
        for t in tickets[1:]:
            env.step_host_end(t)
    def null_outputs(env): _null_outputs(env, acts)

    run(lambda: _venv(N, preset), fused)
    run(lambda: _venv(N, preset, pipeline=7), split)
    run(lambda: _venv(N, preset, pipeline=128), split)
    run(lambda: _venv(N, preset), host)
    os.environ["RR_HOST_ZEROCOPY"], os.environ["RR_HOST_CHUNKS"] = "0", "3"
    try:
        run(lambda: _venv(N, preset), host)
    finally:
        del os.environ["RR_HOST_ZEROCOPY"], os.environ["RR_HOST_CHUNKS"]
    run(lambda: _venv(N, preset), host_begin_end)
    run(lambda: _venv(N, preset), null_outputs)


def test_gpu_stats_buffer_switch_and_clear_while_pipelined():
    """rr_set_stats_buffer to a caller-owned vector (what RoboRugbyVecEnv does) and back to the handle's own; a clear
    issued between pipelined calls drops exactly the calls issued before it."""
    from roborugby_b200 import _lib
    N, K = 2053, 6
    ref = _venv(N, "GAME")
    _start(ref)
    acts = _actions(ref, 2 * K, seed=6)
    ref.clear_stats()
    first = reference_run(ref, acts[:K])
    second = reference_run(ref, acts[K:], h=first.cleared())
    ref.close()

    env = _venv(N, "GAME", pipeline=7)
    _start(env)
    for s in range(K):
        env.step_k(acts[s:s + 1].cuda(), 1, join=False)
    _lib.check(env.lib.rr_clear_stats(env._h, env._stream()))
    for s in range(K, 2 * K, 2):
        env.step_k(acts[s:s + 2].cuda(), 2, join=False)
    env.join()
    second.check(env.stats.cpu().numpy(), "clear between pipelined calls")

    env2 = _venv(N, "GAME")
    _start(env2)
    _lib.check(env2.lib.rr_set_stats_buffer(env2._h, None))          # the handle's own vector
    _lib.check(env2.lib.rr_clear_stats(env2._h, env2._stream()))
    env2.stats.zero_()
    env2.step_k(acts[:K].cuda(), K)
    own = np.zeros(8)
    _lib.check(env2.lib.rr_get_stats(env2._h, own.ctypes.data_as(ctypes.c_void_p)))
    first.check(own, "the handle's own vector")
    assert not env2.stats.any(), "the caller's vector was written after the switch"
    mine = torch.zeros(8, dtype=torch.float64, device="cuda")
    _lib.check(env2.lib.rr_set_stats_buffer(env2._h, mine.data_ptr()))
    env2.step_k(acts[K:].cuda(), K)
    torch.cuda.synchronize()
    second.check(mine.cpu().numpy(), "caller-owned vector")
    env.close(); env2.close()


def test_gpu_two_handles_share_one_vector(oracle):
    """Two handles on one device accumulate into one torch vector; summarize() gives the host restatement's means."""
    from roborugby_b200 import _lib
    from roborugby_b200.stats import summarize
    N, K = 1000, 8
    shared = torch.zeros(8, dtype=torch.float64, device="cuda")
    hs, envs = [], []
    for r in range(2):
        ref = _venv(N, "TRAIN", env_offset=r * N)
        _start(ref, seed=r)
        acts = _actions(ref, K, seed=10 + r)
        hs.append(reference_run(ref, acts))
        ref.close()
        env = _venv(N, "TRAIN", env_offset=r * N)
        _start(env, seed=r)
        _lib.check(env.lib.rr_set_stats_buffer(env._h, shared.data_ptr()))
        env.step_k(acts.cuda(), K)
        envs.append(env)
    torch.cuda.synchronize()
    d = summarize(shared)
    ep = sum(h.ints[EPISODES] for h in hs)
    assert d["episodes"] == ep > 0 and d["steps"] == sum(h.ints[STEPS] for h in hs)
    assert d["mean_length"] == sum(h.ints[LENGTH] for h in hs) / ep
    for t, key in ((0, "mean_return_happy"), (1, "mean_return_grumpy")):
        terms = hs[0].terms[t] + hs[1].terms[t]
        bound = len(terms) * 2.0 ** -52 * float(np.sum(np.abs(terms))) / ep
        assert abs(d[key] - math.fsum(terms) / ep) <= bound + 1e-300, (key, d[key])
    for e in envs:
        e.close()


@pytest.mark.parametrize("preset", ["GAME", "TRAIN"])
def test_gpu_refusal_scenarios_replayed_by_the_oracle(oracle, preset):
    """The scenarios of the CPU tier once on the device: time-limit ends at steps T, T + 1, T + 2 without auto-reset,
    bad actions on live, last-step and finished envs, continuous actions on finished envs, envs injected past their
    end with auto-reset.  The oracle restatement (test_episode_stats.RefEnv) replays every env; the device rows and
    statistics must match it, except envs whose trajectory left the 1e-9 bar on a last-bit contact flip, which are
    counted and bounded."""
    from test_episode_stats import RefEnv, configs, in_field
    T = 4500 if preset == "GAME" else 300
    starts = [10, T - 1, T, T + 1, T + 3]
    oracle.scratch_mode(1)
    try:
        for env_id in (V2, V0):
            for auto_reset in (0, 1):
                cfg, ocfg = configs(oracle, preset, env_id, 1, auto_reset, seed=13, env_offset=0)
                env = _venv(len(starts) * 4, preset, env_id, auto_reset=bool(auto_reset), seed=13)
                N, R = env.num_envs, env.num_robots
                refs = [RefEnv(oracle, cfg, ocfg, i) for i in range(N)]
                st = env.get_state()
                st["step"] = np.array([starts[i % len(starts)] for i in range(N)], np.int32)
                env.set_state(st)
                for i, r in enumerate(refs):
                    r.set_state({k: v[i] for k, v in st.items()})
                g = np.random.default_rng(3)
                K = 4
                if env.discrete:
                    a = g.integers(0, 8, (K, N, R)).astype(np.float64)
                    a[1, :, 0] = np.where(np.arange(N) % 2, 9, 200)
                else:
                    a = g.choice([-1.0, 0.0, 1.0], (K, N, 2 * R))
                    a[1, :, -1] = np.array([np.nan, np.inf, 7.5, -1e10])[np.arange(N) // len(starts)]
                env.clear_stats()
                env.error_mask(clear=True)
                bad = diverged = 0
                h = HostSum(N)
                for s in range(K):
                    before = env.get_state()["step"].astype(np.int64)
                    _, _, rew, done = env.step_k(torch.as_tensor(a[s:s + 1].astype(np.uint8 if env.discrete else np.float32)).cuda(), 1)
                    rew = rew[0].cpu().numpy(); done = done[0].cpu().numpy()
                    err = env.error_mask(clear=True).astype(np.int64)
                    h.row(before, rew, done, err, env.last_naughty(), auto_reset)
                    for i, r in enumerate(refs):
                        e, d, rw, _, _, _ = r.step(a[s, i])
                        if e != err[i] or d != done[i]:
                            bad += 1
                        elif not np.allclose(rw, rew[i], rtol=1e-9, atol=1e-9):
                            diverged += 1
                want = sum((r.st for r in refs), np.zeros(8))
                h.check(env.stats.cpu().numpy(), (env_id, auto_reset))
                assert bad == 0 and diverged <= 1, (env_id, auto_reset, bad, diverged)
                assert np.array_equal(h.ints[INT_STATS], want[INT_STATS].astype(np.int64)), (h.ints, want)
                env.close()
    finally:
        oracle.scratch_mode(0)


def test_gpu_single_env_wrapper_refuses_continuous_actions_on_a_finished_env():
    """RoboRugbyEnv: a NaN thrust on an env past its end raises "Game is over", not the bad-action message."""
    import roborugby_b200 as rr
    env = rr.RoboRugbyEnv("RoboRugby-v0", preset="TRAIN")
    st = env._v.get_state()
    st["step"][:] = env.spec.max_episode_steps + 1
    env._v.set_state(st)
    with pytest.raises(Exception, match="Game is over"):
        env.step([np.nan, 0.0])
    st["step"][:] = 5
    env._v.set_state(st)
    with pytest.raises(Exception, match="invalid action"):
        env.step([np.nan, 0.0])
