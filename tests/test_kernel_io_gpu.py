"""GPU tier: how k_step reads actions and writes result rows (rr_b200.cu warp_store_rows, the element-wise fallback, the
32-bit / byte-wise action loads) and which Launch<...> variant runs, on B200 through the C ABI.

The high-precision reference for every output path is the fp64 run of the same kernel, which test_parity_gpu.py ties to
the oracle: both dtypes compute in double and round once, so fp32 outputs must equal the fp64 outputs cast to float32 bit
for bit.  Result windows are carved out of one larger device buffer between canary bytes, so a stray store is detected
without faulting."""
import itertools

import numpy as np
import pytest

from golden_util import STATE_KEYS
from parity_util import compare_record
from test_action_edges import BAD_ACTION, in_field, thrust_values

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

V0, V2 = "RoboRugby-v0", "RoboRugbySimpleDuel-v2"
CANARY = 0xA5


def _venv(env_id, n, preset, **kw):
    from roborugby_b200.vec_env import RoboRugbyVecEnv
    kw.setdefault("time_limit", False)
    kw.setdefault("auto_reset", False)
    kw.setdefault("out_dtype", torch.float64)
    return RoboRugbyVecEnv(env_id, n, preset=preset, device="cuda:0", **kw)


def lanes_per_chunk(D, size):
    """warp_store_rows: rows of how many lanes one 640-byte staging area takes (0: element-wise stores)."""
    cap, v = 640 // size, 16 // size
    lpc = min(cap // D, 32) if D > 0 else 0
    while 0 < lpc < 32 and (lpc * D) % v:
        lpc -= 1
    return lpc


def vec_bits(N, D, size, aligned=True, act_aligned=True):
    """rr_step's `vec` for torch-allocated (16-byte aligned) buffers: which rows may be written with 128-bit stores."""
    bits = 0
    if aligned and (N * D * size) % 16 == 0:
        bits |= 1
    if aligned and (N * 2 * size) % 16 == 0:
        bits |= 2
    if aligned and N % 16 == 0:
        bits |= 4
    return bits | (8 if act_aligned else 0)


def _same(x, y):
    return np.array_equal(np.asarray(x), np.asarray(y), equal_nan=True)


def _episode_ends_inside(env, K):
    st = env.get_state()
    st["step"][:] = env.max_episode_steps - 1 - (np.arange(env.num_envs) % K)
    env.set_state(st)


# ----------------------------------------------------------------------------------------------- output matrix

def _run_matrix_case(preset, goals, observer, N, pipeline, dtype, acts, K):
    env = _venv(V2, N, preset, seed=17, observer=observer, goal_scoring=goals, out_dtype=dtype, time_limit=True,
                auto_reset=True, pipeline=pipeline)
    _episode_ends_inside(env, K)
    out = [x.cpu().numpy().copy() for x in env.step_k(acts, K)]
    torch.cuda.synchronize()
    res = dict(out=out, state=env.get_state(), err=env.error_mask(), stats=env.get_stats(), D=env.obs_dim,
               launches=env.launch_count)
    env.close()
    return res


@pytest.mark.parametrize("goals", [False, True], ids=["head", "goal_scoring"])
@pytest.mark.parametrize("preset", ["GAME", "TRAIN"])
def test_gpu_fp32_outputs_equal_fp64_cast_on_every_store_path(preset, goals):
    """Observers 0-5 (D = 0, 5, 10, 11, 28, 56) x fp32 / fp64 x one launch / a 7-group sub-batch pipeline, plus (GAME) the
    wide 448-thread variant at 60 000 envs; K = 8 with an episode end (in-kernel auto-reset) in every row.  fp32 rows must
    be the fp64 rows cast to float32 bit for bit; state, error masks and statistics identical."""
    K = 8
    launches = [("single", 2048, 1), ("pipeline7", 2048, 7)]
    if preset == "GAME":
        launches.append(("wide", 60000, 1))
    covered, want = set(), set()
    for (name, N, pipeline), observer in itertools.product(launches, range(6)):
        g = torch.Generator(device="cuda").manual_seed(observer)
        R = 4 if preset == "GAME" else 1
        acts = torch.randint(0, 8, (K, N, R), generator=g, dtype=torch.uint8, device="cuda")
        r64 = _run_matrix_case(preset, goals, observer, N, pipeline, torch.float64, acts, K)
        r32 = _run_matrix_case(preset, goals, observer, N, pipeline, torch.float32, acts, K)
        D = r64["D"]
        why = (name, observer, D)
        for j in range(3):
            assert r32["out"][j].dtype == np.float32 and r64["out"][j].dtype == np.float64
            assert _same(r32["out"][j], r64["out"][j].astype(np.float32)), why + (("obs_h", "obs_g", "rew")[j],)
        assert _same(r32["out"][3], r64["out"][3]) and r32["out"][3].sum() >= N, why
        for k in STATE_KEYS:
            assert np.array_equal(r32["state"][k], r64["state"][k]), why + (k,)
        assert np.array_equal(r32["err"], r64["err"]), why
        for k in ("episodes", "steps", "errors", "length", "naughty"):
            assert r32["stats"][k] == r64["stats"][k], why + (k,)
        for k in ("return_happy", "return_grumpy"):   # atomic additions in any order
            assert np.isclose(r32["stats"][k], r64["stats"][k], rtol=1e-12, atol=1e-9), why + (k,)
        assert r64["launches"] - 1 == (pipeline if pipeline > 1 else 1)
        variant = ("LGame" if preset == "GAME" else "LTrain") + ("Goals" if goals else "") + ("Wide" if name == "wide" else "")
        for size, tag in ((4, "fp32"), (8, "fp64")):
            covered.add((variant, name, tag, D, lanes_per_chunk(D, size), vec_bits(N, D, size)))
        dims = [0, 5, 11, 28, 56, 11] if preset == "GAME" else [0, 5, 11, 5, 10, 11]
        for size, tag in ((4, "fp32"), (8, "fp64")):
            want.add((variant, name, tag, dims[observer], lanes_per_chunk(dims[observer], size),
                      vec_bits(N, dims[observer], size)))
    for t in sorted(covered):
        print("covered (variant, launch, dtype, D, lpc, vec bits):", t)
    assert covered == want
    lpcs = {(t[2], t[4]) for t in covered}
    if preset == "GAME":   # every chunking of warp_store_rows: 32 lanes, 12 (D = 11), 5 (D = 28), 2 (D = 56) for fp32
        assert {("fp32", 32), ("fp32", 12), ("fp32", 5), ("fp32", 2), ("fp64", 16), ("fp64", 6), ("fp64", 2),
                ("fp64", 1)} <= lpcs
    else:
        assert {("fp32", 16), ("fp64", 8)} <= lpcs   # D = 10


# ----------------------------------------------------------------------------------------------- raw store paths

class Carved:
    """Windows of `sizes` bytes at `offset` bytes past a 256-byte boundary of one device buffer, canaries around them."""

    def __init__(self, sizes, offset, pad=64):
        self.spans, cur = [], 0
        for s in sizes:
            p = cur + pad + offset
            self.spans.append((p, s))
            cur = ((p + s + pad + 255) // 256) * 256
        self.pool = torch.full((cur + 256,), CANARY, dtype=torch.uint8, device="cuda")
        for p, s in self.spans:
            self.pool[p:p + s] = 0x5A

    def ptr(self, j):
        return self.pool.data_ptr() + self.spans[j][0] if self.spans[j][1] else None

    def get(self, j, dtype):
        p, s = self.spans[j]
        return self.pool[p:p + s].clone().view(dtype).cpu().numpy()

    def canaries_intact(self):
        keep = torch.ones_like(self.pool, dtype=torch.bool)
        for p, s in self.spans:
            keep[p:p + s] = False
        return bool((self.pool[keep] == CANARY).all())


def _stream():
    return torch.cuda.current_stream().cuda_stream


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64], ids=["fp32", "fp64"])
def test_gpu_result_stores_at_any_alignment_and_with_null_outputs(dtype):
    """rr_step with raw pointers: every output window at 0, 4 or 8 bytes past a 16-byte boundary (whatever keeps the
    elements aligned: 0 or 8 for fp64), batches whose last warp is partial and whose rows are not multiples of 16 bytes (N = 1004: 128-bit rows with a partial last warp), and every
    subset of {obs_h, obs_g, rew, done} passed as NULL.  Each result equals the run into torch buffers, the state is the
    same, and no byte outside the windows changes."""
    from roborugby_b200 import _lib
    K, npt = 3, np.float32 if dtype == torch.float32 else np.float64
    size = np.dtype(npt).itemsize
    for N in (1, 31, 33, 1003, 1004, 4099):
        env = _venv(V2, N, "GAME", seed=N, observer=2, out_dtype=dtype, time_limit=True)
        D = env.obs_dim
        _episode_ends_inside(env, K)
        st0 = env.get_state()
        g = torch.Generator(device="cuda").manual_seed(N)
        acts = torch.randint(0, 8, (K, N, 4), generator=g, dtype=torch.uint8, device="cuda")
        ref = [x.cpu().numpy().copy() for x in env.step_k(acts, K)]
        ref_state = env.get_state()
        sizes = [K * N * D * size, K * N * D * size, K * N * 2 * size, K * N]
        for offset, null in itertools.product((0, 4, 8) if size == 4 else (0, 8), range(16)):
            env.set_state(st0)
            cv = Carved(sizes, offset)
            ptrs = [None if null >> j & 1 else cv.ptr(j) for j in range(4)]
            _lib.check(env.lib.rr_step(env._h, acts.data_ptr(), 4, K, *ptrs, _stream()))
            torch.cuda.synchronize()
            why = (N, offset, null)
            assert cv.canaries_intact(), why
            for j, (want, shape) in enumerate(zip(ref, [(K, N, D), (K, N, D), (K, N, 2), (K, N)])):
                if ptrs[j] is not None:
                    got = cv.get(j, torch.uint8 if j == 3 else dtype).reshape(shape)
                    assert _same(got, want), why + (j,)
            if null in (0, 15):
                st = env.get_state()
                assert all(np.array_equal(st[k], ref_state[k]) for k in STATE_KEYS), why
        env.close()


def test_gpu_observe_and_observe_entity_stores_fp32_equal_fp64_cast():
    """rr_observe (each of obs_h / obs_g may be NULL) and rr_observe_entity into windows at 0, 4 and 8 bytes past a 16-byte
    boundary, for batches with a partial last warp: the fp32 rows are the fp64 rows cast, canaries intact."""
    from roborugby_b200 import _lib
    for N in (1, 31, 33, 1003, 4099):
        e64 = _venv(V2, N, "GAME", seed=5, observer=2, out_dtype=torch.float64)
        e32 = _venv(V2, N, "GAME", seed=5, observer=2, out_dtype=torch.float32)
        D = e64.obs_dim
        ref_h, ref_g = (x.cpu().numpy() for x in e64.observe())
        for offset in (0, 4, 8):
            for null in range(4):
                cv = Carved([N * D * 4, N * D * 4], offset)
                ptrs = [None if null >> j & 1 else cv.ptr(j) for j in range(2)]
                _lib.check(e32.lib.rr_observe(e32._h, ptrs[0], ptrs[1], _stream()))
                torch.cuda.synchronize()
                assert cv.canaries_intact(), (N, offset, null)
                for j, want in enumerate((ref_h, ref_g)):
                    if ptrs[j] is not None:
                        assert _same(cv.get(j, torch.float32).reshape(N, D), want.astype(np.float32)), (N, offset, j)
            for robot in range(e64.num_robots):
                want = e64.observe_entity(robot, robot + 1).cpu().numpy()
                cv = Carved([N * D * 4], offset)
                _lib.check(e32.lib.rr_observe_entity(e32._h, robot, robot + 1, None, cv.ptr(0), _stream()))
                torch.cuda.synchronize()
                assert cv.canaries_intact(), (N, offset, robot)
                assert _same(cv.get(0, torch.float32).reshape(N, D), want.astype(np.float32)), (N, offset, robot)
        e64.close(); e32.close()


# ----------------------------------------------------------------------------------------------- action loads

def _oracle_sample(oracle, preset, env_id, observer, st0, acts, out, state, sample):
    """Replay `sample` envs on the oracle; returns the number whose trajectory left the 1e-9 bar (a contact decision
    flipped on a last-bit difference of sin/cos, test_parity_gpu.py)."""
    K = acts.shape[0]
    diverged = 0
    cfg = oracle.default_config(preset, env_id)
    cfg.observer = observer
    o = oracle.OracleEnv(cfg=cfg)
    for i in sample:
        o.set_state({k: st0[k][i] for k in STATE_KEYS})
        for s in range(K):
            want = o.step(acts[s, i])
            assert want["err"] == 0, (i, s)
            got = dict(obs_h=out[0][s, i], obs_g=out[1][s, i], rew=out[2][s, i], done=out[3][s, i], naughty=want["naughty"])
            last = s == K - 1
            ok = compare_record({k: state[k][i] for k in STATE_KEYS} if last else o.get_state(), got, o.get_state(), want)[0]
            if not ok:
                diverged += 1
                break
    return diverged


@pytest.mark.parametrize("preset", ["GAME", "TRAIN"])
def test_gpu_action_loads_at_any_alignment_and_count(oracle, preset):
    """Discrete ids for 1 to R robots, at byte offsets 0 and 1 of a device buffer (A = 4 at offset 1 takes the byte-wise
    load instead of one 32-bit load per env), and continuous thrust pairs for 1 to R robots: identical to the run from a
    torch tensor, and equal to the oracle on a sample."""
    from roborugby_b200 import _lib
    N, K = 515, 4
    rng = np.random.default_rng(7)
    oracle.scratch_mode(1)
    try:
        for env_id in (V2, V0):
            env = _venv(env_id, N, preset, seed=3, observer=1)
            R = env.num_robots
            st0 = env.get_state()
            counts = range(1, R + 1) if env.discrete else range(2, 2 * R + 1, 2)
            for A in counts:
                if env.discrete:
                    a = rng.integers(0, 8, (K, N, A)).astype(np.uint8)
                else:
                    a = rng.choice(np.float32([-1, -0.5, 0, 0.5, 1, 1.5]), (K, N, A))
                env.set_state(st0)
                ref = [x.cpu().numpy().copy() for x in env.step_k(torch.as_tensor(a).cuda(), K)]
                ref_state, ref_err = env.get_state(), env.error_mask(clear=True)
                for off in ((0, 1, 2, 3) if env.discrete else (0, 4)):
                    raw = torch.zeros(a.nbytes + 64, dtype=torch.uint8, device="cuda")
                    raw[off:off + a.nbytes] = torch.as_tensor(a.reshape(-1).view(np.uint8)).cuda()
                    env.set_state(st0)
                    b = env._out(K)
                    _lib.check(env.lib.rr_step(env._h, raw.data_ptr() + off, A, K, b["obs_h"].data_ptr(),
                                               b["obs_g"].data_ptr(), b["rew"].data_ptr(), b["done"].data_ptr(), _stream()))
                    torch.cuda.synchronize()
                    got = [b[k].cpu().numpy()[..., :env.obs_dim] if k.startswith("obs") else b[k].cpu().numpy()
                           for k in ("obs_h", "obs_g", "rew", "done")]
                    assert all(_same(x, y) for x, y in zip(got, ref)), (env_id, A, off)
                    st = env.get_state()
                    assert all(np.array_equal(st[k], ref_state[k]) for k in STATE_KEYS), (env_id, A, off)
                    assert np.array_equal(env.error_mask(clear=True), ref_err), (env_id, A, off)
                assert (ref_err == 0).all()
                div = _oracle_sample(oracle, preset, env_id, 1, st0, a.astype(np.float64), ref, ref_state, range(0, N, 37))
                assert div <= 1, (env_id, A, div)
            env.close()
    finally:
        oracle.scratch_mode(0)


# ----------------------------------------------------------------------------------------------- action edges

@pytest.mark.parametrize("preset", ["GAME", "TRAIN"])
def test_gpu_thrust_edges_match_oracle(oracle, preset):
    """The CPU tier's grid of thrust values (test_action_edges.py) through rr_step, one case per env, every slot and
    action count: on the GPU a float-to-int conversion saturates and NaN converts to 0, so a missing range check would
    show here as a wrong thrust rather than as undefined behaviour.  Refused exactly where the oracle's int(round(x))
    leaves [-8, 7] (RR_ERR_BAD_ACTION, env untouched, done = 1); everywhere else outputs and state equal the oracle's."""
    cfg = oracle.default_config(preset, V0)
    cfg.observer = 1
    o = oracle.OracleEnv(cfg=cfg)
    o.reset_philox(5, 0, 0)
    base = o.get_state()
    R = o.R
    base["rflag"][:, :2] = np.array([[7, -8], [-8, 7], [3, 3], [0, -1]])[:R]
    vals = thrust_values()
    pairs = [(l, r) for v in vals for l, r in ((v, v), (v, -v), (v, 0.0), (0.0, v), (v, 1.0), (-1.0, v))]
    oracle.scratch_mode(1)
    refused = agreed = 0
    try:
        for n in range(2, 2 * R + 1, 2):
            cases = [(slot, l, r) for slot in range(n // 2) for l, r in pairs]
            N = len(cases)
            a = np.tile(np.float32([1, -1]), (N, R))[:, :n].copy()
            for i, (slot, l, r) in enumerate(cases):
                a[i, 2 * slot], a[i, 2 * slot + 1] = l, r
            env = _venv(V0, N, preset, observer=1)
            st0 = {k: np.stack([base[k]] * N) for k in STATE_KEYS}
            env.set_state(st0)
            out = [x[0].cpu().numpy().copy() for x in env.step_k(torch.as_tensor(a).reshape(1, N, n).cuda(), 1)]
            st, err = env.get_state(), env.error_mask()
            for i, (slot, l, r) in enumerate(cases):
                why = (n, slot, l, r)
                if not in_field(a[i].astype(np.float64)):
                    assert err[i] == BAD_ACTION and out[3][i] == 1, why + (err[i],)
                    assert all(np.array_equal(st[k][i], base[k]) for k in STATE_KEYS), why
                    refused += 1
                    continue
                o.set_state(base)
                want = o.step(a[i].astype(np.float64))
                assert err[i] == want["err"], why + (err[i], want["err"])
                if want["err"]:
                    continue
                got = dict(obs_h=out[0][i], obs_g=out[1][i], rew=out[2][i], done=out[3][i], naughty=want["naughty"])
                ok, _, w, diff = compare_record({k: st[k][i] for k in STATE_KEYS}, got, o.get_state(), want)
                assert ok, why + (diff, w)
                agreed += 1
            env.close()
    finally:
        oracle.scratch_mode(0)
    print(f"{preset}: {agreed} cases equal to the oracle, {refused} refused")
    assert refused > 0 and agreed > 0


@pytest.mark.parametrize("preset", ["GAME", "TRAIN"])
def test_gpu_discrete_ids_above_7_are_refused(oracle, preset):
    """Every uint8 id in every robot slot, with 1 to R actions, through rr_step: ids above 7 raise RR_ERR_BAD_ACTION and
    leave the env untouched, the others equal the oracle."""
    o = oracle.OracleEnv(preset, V2)
    o.reset_philox(6, 1, 0)
    base = o.get_state()
    R = o.R
    oracle.scratch_mode(1)
    try:
        for A in range(1, R + 1):
            cases = [(slot, i) for slot in range(A) for i in range(256)]
            N = len(cases)
            a = np.zeros((N, A), np.uint8)
            for j, (slot, i) in enumerate(cases):
                a[j, slot] = i
            env = _venv(V2, N, preset)
            env.set_state({k: np.stack([base[k]] * N) for k in STATE_KEYS})
            out = [x[0].cpu().numpy().copy() for x in env.step_k(torch.as_tensor(a).reshape(1, N, A).cuda(), 1)]
            st, err = env.get_state(), env.error_mask()
            for j, (slot, i) in enumerate(cases):
                if i > 7:
                    assert err[j] == BAD_ACTION and out[3][j] == 1, (A, slot, i)
                    assert all(np.array_equal(st[k][j], base[k]) for k in STATE_KEYS), (A, slot, i)
                    continue
                o.set_state(base)
                want = o.step(a[j].astype(np.float64))
                assert err[j] == want["err"] == 0, (A, slot, i)
                got = dict(obs_h=out[0][j], obs_g=out[1][j], rew=out[2][j], done=out[3][j], naughty=want["naughty"])
                assert compare_record({k: st[k][j] for k in STATE_KEYS}, got, o.get_state(), want)[0], (A, slot, i)
            env.close()
    finally:
        oracle.scratch_mode(0)


# ----------------------------------------------------------------------------------------------- goal scoring

GOAL_STEPS = 160


def _goal_template(oracle):
    """A GAME RoboRugby-v0 start whose robots and balls are far from the happy goal's corner; negative balls 4 and 5
    parked (at rest) in the happy goal, ball 6 outside its hypotenuse drifting in: the goal is destroyed 150 steps after
    ball 6 arrives.  variant v of the template starts ball 6 further out, so it arrives later."""
    W = 800.0
    o = oracle.OracleEnv("GAME", V0)
    for idx in range(200):
        o.reset_philox(77, idx, 0)
        st = o.get_state()
        if (np.hypot(st["rob"][:, 0] - W, st["rob"][:, 1] - W) > 360).all() and \
                (np.hypot(st["ball"][:, 0] - W, st["ball"][:, 1] - W) > 360).all():
            break
    else:
        raise AssertionError("no start far from the corner")
    for (x, y), b in zip([(W - 40, W - 40), (W - 75, W - 70)], (4, 5)):
        st["ball"][b] = (x, y, x - 7, x + 7, y - 7, y + 7, 0, 0)
    st["rflag"][:] = 0
    st["step"] = np.int32(0)

    def variant(v):
        s = {k: np.array(st[k], copy=True) for k in STATE_KEYS}
        d = (0.5 + v) / np.sqrt(2)          # centre 0.5 + v px outside the hypotenuse x + y = 1360
        x, y = 640 - d, 720 - d
        s["ball"][6] = (x, y, x - 7, x + 7, y - 7, y + 7, 0.2 / np.sqrt(2), 0.2 / np.sqrt(2))
        return s
    return variant


def _goal_config(oracle):
    cfg = oracle.default_config("GAME", V0)
    cfg.goal_scoring = 1
    cfg.observer = 1
    cfg.time_limit = 1
    return cfg


@pytest.mark.parametrize("N", [256, 60000], ids=["LGameGoals", "LGameGoalsWide"])
def test_gpu_goal_destroyed_inside_a_fused_launch_then_auto_reset(oracle, N):
    """Goal scoring with auto_reset: the happy goal is destroyed at a different step of one 160-step launch in each env
    (the third negative ball arrives staggered), done is set on exactly that row, the in-kernel reset clears the goal
    bookkeeping (goal_clear), and the remaining steps follow the oracle from reset_philox(seed, i, 1).  rr_goal_state
    afterwards equals the oracle's: every ball alive, both scores 0, dwell counters as tracked since the reset."""
    from roborugby_b200 import _lib
    seed, K = 2027, GOAL_STEPS
    variant = _goal_template(oracle)
    ocfg = _goal_config(oracle)
    ends = []
    for v in range(8):   # the step (row) at which each variant's goal is destroyed, robots standing still
        o = oracle.OracleEnv(cfg=ocfg)
        o.set_state(variant(v))
        for s in range(K):
            out = o.step(np.zeros(2))
            assert out["err"] == 0
            if out["done"]:
                assert o.goal_state()["destroyed"][0] == 1
                ends.append(s)
                break
    assert len(ends) == 8 and len(set(ends)) > 1 and max(ends) <= K - 4, ends
    env = _venv(V0, N, "GAME", seed=seed, goal_scoring=True, observer=1, auto_reset=True, time_limit=True)
    wide = N > 384 * torch.cuda.get_device_properties(0).multi_processor_count
    vs = [variant(v) for v in range(8)]
    env.set_state({k: np.stack([vs[v][k] for v in range(8)])[np.arange(N) % 8] for k in STATE_KEYS})
    rng = np.random.default_rng(1)
    acts = np.zeros((K, N, 2), np.float32)
    end = np.array([ends[i % 8] for i in range(N)])
    later = np.arange(K)[:, None] > end[None, :]
    acts[later] = rng.choice(np.float32([-1, 0, 1]), (int(later.sum()), 2))
    obs_h, _, _, done = env.step_k(torch.as_tensor(acts).cuda(), K)
    done = done.cpu().numpy()
    assert env.launch_count - 1 == 1 and wide == (N == 60000)
    rows = np.arange(K)[:, None]
    assert (done[end, np.arange(N)] == 1).all() and (done[rows < end[None, :]] == 0).all(), "done on the destroying row"
    # the reference's own placement (strict_reset) can start an episode on which it raises at once: such an env is done
    # again with an error bit, every other env stays in its new episode
    err = env.error_mask()
    again = (done * later).sum(0)
    assert ((again > 0) <= (err != 0)).all() and (err != 0).sum() <= max(2, N // 1000), int((err != 0).sum())
    g = env.goal_state()
    assert (g["alive"] == 1).all() and (g["score"] == 0).all() and (g["destroyed"] == 0).all()
    st = env.get_state()
    clean = np.nonzero(err == 0)[0]
    sample = np.concatenate([clean[:16], clean[-8:]])
    obs_h = obs_h[:, torch.as_tensor(sample, device="cuda")].cpu().numpy()
    oracle.scratch_mode(1)
    try:
        diverged = 0
        for j, i in enumerate(sample):
            o = oracle.OracleEnv(cfg=ocfg)   # the same episode: the placement of a reset starts from the final poses
            o.set_state(vs[i % 8])
            for s in range(end[i] + 1):
                assert o.step(np.zeros(2))["err"] == 0
            o.reset_philox(seed, int(i), 1)
            first = o.observe(1)
            assert np.allclose(obs_h[end[i], j], first, rtol=1e-9, atol=1e-9), i   # the row holds the new episode's first obs
            ok = True
            for s in range(end[i] + 1, K):
                want = o.step(acts[s, i].astype(np.float64))
                assert want["err"] == 0 and want["done"] == 0 == done[s, i], (i, s)
                if not np.allclose(obs_h[s, j], want["obs_h"], rtol=1e-9, atol=1e-9):
                    ok = False
                    break
            if not ok:
                diverged += 1
                continue
            ref, og = o.get_state(), o.goal_state()
            assert int(ref["step"]) == int(st["step"][i]) == K - 1 - end[i], i
            assert np.allclose(ref["rob"], st["rob"][i], rtol=1e-9, atol=1e-9), i
            assert np.array_equal(og["alive"], g["alive"][i]) and np.array_equal(og["score"], g["score"][i]), i
            assert np.array_equal(og["dwell"], g["dwell"][i]), i
        assert diverged <= 1
    finally:
        oracle.scratch_mode(0)
    stats = env.get_stats()
    assert stats["episodes"] == done.sum() and stats["errors"] >= (err != 0).sum()
    env.close()


# ----------------------------------------------------------------------------------------------- rr_set_state

def test_gpu_set_state_rejects_thrusts_the_state_cannot_hold():
    """rr_set_state refuses a stored thrust outside [-8, 7] or a history flag other than 0 / 1 before it copies anything;
    the ends of the range round-trip."""
    from roborugby_b200._lib import RRError
    env = _venv(V0, 8, "GAME", seed=1)
    st = env.get_state()
    st["rflag"][:, :, :2] = np.array([[-8, 7], [7, -8], [0, 0], [-1, 1]])
    env.set_state(st)
    assert np.array_equal(env.get_state()["rflag"], st["rflag"])
    for col, bad in [(0, 8), (1, -9), (0, 127), (1, -128), (2, 2), (2, -1)]:
        x = {k: np.array(v, copy=True) for k, v in st.items()}
        x["rflag"][5, 3, col] = bad
        x["rob"][:, :, 0] += 1.0
        with pytest.raises(RRError, match="rflag of env 5 robot 3"):
            env.set_state(x)
        now = env.get_state()
        assert all(np.array_equal(now[k], st[k]) for k in STATE_KEYS), (col, bad)
    env.close()
