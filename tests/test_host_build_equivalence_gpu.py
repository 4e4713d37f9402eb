"""GPU tier (B200): every k_step variant against the host build of the same source (tests/emul), bit for bit.

The kernels and the host build compile the same rr_sim.cuh with --fmad=false and the same table-driven sin/cos, and
use only IEEE + - * / fma sqrt rint fmod and exact fmin / fmax / fabs; the one intended difference is CUDA's atan,
which only the observers call (angle_degrees).  So the GPU must reproduce the host build exactly: every byte of every
saved env row (rr_save_states), every reward, done flag and row flag, every observation and terminal observation
except the atan-derived columns, and every integer statistic.  What this pins that the CPU tier cannot: the fused
K-step launch and its in-kernel auto-resets, hot fields in shared memory at production block sizes (384 / 448 / 512
threads, partial last block and warp), the branch-free side x line block of the contact paths, the squeeze and
stuck-pair memos, the uint8 action decoding and the sub-batch pipeline's block offsets.

Each case injects starting states on the GPU, warms up with one launch, saves every env's row, loads the rows into the
host build (emul_states.load) and runs the same actions there (use_libm_sincos(False): the GPU's sin/cos routine); then
one launch without and one with the rr_step_info outputs (k_step<L, OutT, false> and <L, OutT, true>) are compared.
The atan columns (BasicLidar column 1, columns 1 and 3 of both 6-way lidars) are held to the suite's parity bar
(1e-9 relative for fp64 outputs, one ulp of the cast host value for fp32) and their bit-equal share is printed.
Statistics returns are sums whose per-warp atomics land in any order: 1e-12 relative."""
import ctypes as C
import os
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from golden_util import STATE_KEYS, parse_name
from conftest import golden_files

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

V0, V2 = "RoboRugby-v0", "RoboRugbySimpleDuel-v2"
OBS_NONE, OBS_BASIC, OBS_L6V2, OBS_ALL, OBS_PRIOR, OBS_L6V1 = 0, 1, 2, 3, 4, 5
ATAN_COLS = {OBS_BASIC: [1], OBS_L6V2: [1, 3], OBS_L6V1: [1, 3]}
COUNTS, RET = [0, 3, 4, 5, 6, 7], [1, 2]   # statistics: episodes, length, naughty, errors, steps, squeeze_replays
NO_SQUEEZE_MEMO = 1
MIXINS_ALL = ["KeepMovingGuys", "DontDriveInGoals", "BaseDestruction", "PushNegBallsFromGoal", "PushPosBallsToGoal",
              "ChasePosBall", "NaughtyBots"]
MIXINS_CUT = ["DontDriveInGoals", "ChasePosBall", "NaughtyBots", "KeepMovingGuys"]
MIXINS_NEG = ["PushNegBallsFromGoal", "KeepMovingGuys", "BaseDestruction"]

# name -> (preset, env id, N, (K without, K with rr_step_info), pipeline, fp64, goal scoring, observer, state pool,
#          other settings).  The sizes put every Launch type at its production block size with a partial last block and
#          a partial last warp: GAME 384 threads (sub-batch pipeline, N > 384 x #SM), 448 (one launch, N > 416 x #SM),
#          TRAIN 512 (N > 480 x #SM).
CASES = {
    "bench_pipeline128": ("GAME", V2, 65536, (32, 8), 128, False, False, None, "bench", {}),
    "bench_single_launch": ("GAME", V2, 65536, (32, 8), 1, False, False, None, "bench", {}),
    "contact_wide_prior": ("GAME", V2, 65529, (16, 8), 1, True, False, OBS_PRIOR, "contact", {}),
    "rich_pipelined_no_memo": ("GAME", V2, 60001, (16, 8), 4, True, False, OBS_BASIC, "rich",
                               dict(flags=NO_SQUEEZE_MEMO, reward_mixins=MIXINS_ALL, others=True)),
    "goals_wide_relaxed": ("GAME", V2, 65529, (16, 8), 1, False, True, OBS_L6V1, "golden+contact",
                           dict(strict_reset=False, others=True)),
    "goals_wide_continuous": ("GAME", V0, 57000, (8, 8), 1, True, True, OBS_ALL, "golden",
                              dict(reward_mixins=MIXINS_CUT)),
    "goals_pipelined_no_auto_reset": ("GAME", V2, 60001, (16, 8), 8, False, True, OBS_L6V2, "rich",
                                      dict(auto_reset=False)),
    "goals_continuous_no_time_limit": ("GAME", V0, 4099, (16, 16), 1, True, True, OBS_NONE, "golden",
                                       dict(time_limit=False)),
    "train": ("TRAIN", V2, 80001, (32, 8), 1, False, False, None, "golden", dict(others=True)),
    "train_continuous_prior": ("TRAIN", V0, 4096, (16, 16), 1, True, False, OBS_PRIOR, "rich",
                               dict(reward_mixins=MIXINS_NEG)),
    "train_goals_relaxed": ("TRAIN", V2, 80001, (32, 8), 1, True, True, OBS_BASIC, "rich", dict(strict_reset=False)),
    "train_goals_no_auto_reset": ("TRAIN", V2, 3001, (16, 16), 2, False, True, OBS_L6V1, "golden",
                                  dict(auto_reset=False, time_limit=False, flags=NO_SQUEEZE_MEMO, others=True)),
}


# ------------------------------------------------------------------------------------------ which k_step runs

def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def pick_block(n, sms, max_block):
    """rr_b200.cu pick_block."""
    b = ((-(-n // sms) + 31) // 32) * 32
    return min(max(b, 32), max_block)


def k_step_variant(preset, goals, n, pipeline, sms):
    """(Launch type, block size, launches) that rr_step picks (rr_b200.cu rr_step_info)."""
    game = preset == "GAME"
    wide = game and pipeline <= 1 and -(-n // 384) > sms
    blk = pick_block(n, sms, 448 if wide else (384 if game else 512))
    nb = -(-n // blk)
    name = ("LGame" if game else "LTrain") + ("Goals" if goals else "") + ("Wide" if wide else "")
    return name, blk, (min(pipeline, nb) if pipeline > 1 else 1)


def test_case_matrix_covers_every_k_step_variant():
    """The 24 instantiations {LGame, LGameWide, LGameGoals, LGameGoalsWide, LTrain, LTrainGoals} x {float, double} x
    {INFO off, on} all run below, and every Launch type runs at its production block size with a partial last block
    and a partial last warp."""
    sms = _sms()
    covered, production = set(), set()
    for name, (preset, _, n, _, pipeline, f64, goals, *_r) in CASES.items():
        launch, blk, _ = k_step_variant(preset, goals, n, pipeline, sms)
        for info in (False, True):
            covered.add((launch, "double" if f64 else "float", info))
        if n % blk and n % 32:
            production.add((launch, blk))
        print(f"{name}: {launch} {'double' if f64 else 'float'}, {blk}-thread blocks, N = {n} "
              f"(last block {n % blk or blk}, last warp {n % 32 or 32})")
    launches = ["LGame", "LGameWide", "LGameGoals", "LGameGoalsWide", "LTrain", "LTrainGoals"]
    want = {(l, t, i) for l in launches for t in ("float", "double") for i in (False, True)}
    print(f"{len(covered)} of 24 k_step variants covered; production blocks with partial ends: {sorted(production)}")
    assert covered == want, sorted(want - covered)
    kmax = {"LGame": 384, "LGameGoals": 384, "LGameWide": 448, "LGameGoalsWide": 448, "LTrain": 512, "LTrainGoals": 512}
    assert {(l, kmax[l]) for l in launches} <= production, sorted(production)


# ------------------------------------------------------------------------------------------ starting states

def _golden_states(preset):
    """Every state the reference stepped in the golden files of `preset` (about-to-collide injections, goal scoring,
    chases, and the states on which it raised)."""
    out = []
    for p in golden_files(f"{preset}_*.npz"):
        d = np.load(p)
        if parse_name(p)[0] != preset or not set(STATE_KEYS) <= set(d.files):   # (the time-limit files hold outputs only)
            continue
        out.append({k: d[k].reshape((-1,) + d[k].shape[2:]) for k in STATE_KEYS})
    return out


def _contact_states(oracle):
    """Squeezes against a wall (with bystanders), pincers and stuck pairs (squeeze_util.py): GAME only."""
    import squeeze_util as sq
    rng = np.random.default_rng(11)
    out = []
    for j in range(96):
        spect = [(rng.uniform(-20, 20), rng.uniform(-20, 20)), (rng.uniform(-40, 40), rng.uniform(-40, 40))] if j % 2 else None
        out.append(sq.oracle_env(oracle, "GAME", sq.scenario(rng, "GAME"), spectators=spect).get_state())
        out.append(sq.pincer_env(oracle, rng).get_state())
        out.append(sq.stuck_pair_env(oracle, rng).get_state())
    return [_stacked(out)]


def _rich_states(preset):
    from test_reward_compositions import _state_set
    return [_stacked([s for s, _, _ in _state_set(preset, True)])]


def _stacked(states):
    return {k: np.stack([np.asarray(s[k]) for s in states]) for k in STATE_KEYS}


def _inject(env, pool_names, oracle, K):
    """Tile the named pools over the batch; a quarter of the envs get a step counter within K of the time limit."""
    N, T = env.num_envs, env.max_episode_steps
    st = env.get_state()
    if pool_names == "bench":
        st["step"][:] = (np.arange(N) * 7919) % max(T - 1, 1)     # bench.py's desynchronisation
        env.set_state(st)
        return 0
    preset = "GAME" if env.num_robots > 1 else "TRAIN"
    parts = []
    for name in pool_names.split("+"):
        parts += {"golden": lambda: _golden_states(preset), "contact": lambda: _contact_states(oracle),
                  "rich": lambda: _rich_states(preset)}[name]()
    pool = {k: np.concatenate([p[k] for p in parts]) for k in STATE_KEYS}
    rng = np.random.default_rng(N)
    pick = rng.integers(0, len(pool["step"]), N)
    for k in STATE_KEYS:
        st[k] = pool[k][pick].astype(st[k].dtype).reshape(st[k].shape)
    near = rng.random(N) < 0.25
    st["step"][near] = T - rng.integers(0, K + 2, int(near.sum()))
    env.set_state(st)
    return len(pool["step"])


def _actions(env, K, seed, contact):
    """Discrete ids (now and then one above 7, which the kernel refuses) or thrust pairs (now and then NaN, infinite or
    out of the field, refused as well).  Contact pools: robots 0 and 1 mostly keep driving forward (id 0 / thrust 1)."""
    rng = np.random.default_rng(seed)
    N, A = env.num_envs, env.action_dim
    if env.discrete:
        a = rng.integers(0, 8, (K, N, A)).astype(np.uint8)
        bad = rng.random((K, N, A)) < 2e-4
        a[bad] = rng.integers(8, 256, int(bad.sum()))
        if contact:
            lead = rng.random((K, N, min(A, 2))) < 0.75
            a[..., :2][lead] = 0
    else:
        vals = np.float32([-1, -0.5, 0, 0.5, 1, 1.4999, 7.4, -8.4, 7.5, np.nan, np.inf, -1e30])
        p = np.array([.2, .1, .2, .1, .2, .1, .05, .04, .0025, .0025, .0025, .0025])
        a = rng.choice(vals, (K, N, A), p=p / p.sum()).astype(np.float32)
    return a


# ------------------------------------------------------------------------------------------ comparison rules

def _same(g, h):
    """Element-wise: bit-identical, or both NaN (NaN payloads are not part of the contract)."""
    g = np.asarray(g); h = np.asarray(h)
    u = np.uint32 if g.dtype == np.float32 else np.uint64
    return (g.view(u) == h.view(u)) | (np.isnan(g) & np.isnan(h))


def _near(g, h, f32):
    """The suite's parity bar for the atan columns: one fp32 ulp of the cast host value, 1e-9 relative in fp64."""
    if f32:
        d = np.abs(g.view(np.int32).astype(np.int64) - h.view(np.int32).astype(np.int64))
        return (d <= 1) | (np.isnan(g) & np.isnan(h))
    with np.errstate(invalid="ignore"):
        return (np.abs(g - h) <= 1e-9 * np.maximum(1.0, np.abs(h))) | (np.isnan(g) & np.isnan(h))


class Tally:
    """Counts of one compared launch (or state) over all chunks, with the first differences found."""

    def __init__(self):
        self.n = {}
        self.first = []

    def add(self, key, v=1):
        self.n[key] = self.n.get(key, 0) + int(v)

    def fail(self, what):
        self.add("differences")
        if len(self.first) < 8:
            self.first.append(what)

    def merge(self, o):
        for k, v in o.n.items():
            self.add(k, v)
        self.first += o.first[:max(0, 8 - len(self.first))]


def _compare_rows(t, tag, g, h, f32, c0, atan=()):
    """g (GPU) [K, m, ...] against h (host, float64 or int) of the same shape; rows are [s, i]; atan columns of
    observations within the parity bar, their bit-equal count tallied."""
    if h.dtype == np.float64 and f32:
        h = h.astype(np.float32)
    if g.dtype.kind == "f":
        h = h.astype(g.dtype)
        ok = _same(g, h)
        if atan:
            exact = ok[..., atan]
            t.add(f"{tag}.atan_values", exact.size)
            t.add(f"{tag}.atan_bit_equal", exact.sum())
            ok[..., atan] = _near(g[..., atan], h[..., atan], f32)
    else:
        ok = g.astype(np.int64) == h.astype(np.int64)
    ok = ok.all(axis=tuple(range(2, ok.ndim)))
    t.add(f"{tag}.rows", ok.size)
    if not ok.all():
        s, i = np.argwhere(~ok)[0]
        t.add(f"{tag}.rows_differing", (~ok).sum())
        t.fail(f"{tag}: {(~ok).sum()} rows differ, first step {s} env {c0 + i}: gpu {g[s, i]} host {h[s, i]}")


def _compare_launch(t, g, h, c0, f32, D, atan, info):
    _compare_rows(t, "rew", g["rew"], h["rew"], f32, c0)
    _compare_rows(t, "done", g["done"], h["done"], f32, c0)
    if info:
        _compare_rows(t, "row_flags", g["flags"], h["flags"], f32, c0)
    if D:
        _compare_rows(t, "obs_h", g["obs_h"], h["obs_h"], f32, c0, atan)
        _compare_rows(t, "obs_g", g["obs_g"], h["obs_g"], f32, c0, atan)
        if info:   # terminal observations: done rows only (the others keep whatever an earlier call left)
            dn = h["done"] != 0
            for key, hk in (("final_h", "final_h"), ("final_g", "final_g")):
                _compare_rows(t, key, g[key][dn][None], h[hk][dn][None], f32, c0, atan)
    t.add("resets", (h["done"] != 0).sum())


def _compare_state(t, tag, g_rows, h_rows, c0):
    """Saved rows, byte for byte (as 8-byte units: the row layout's unit, rr_sim.cuh RowLayout)."""
    gu, hu = g_rows.view(np.uint64), h_rows.view(np.uint64)
    bad = gu != hu
    t.add(f"{tag}.bytes", g_rows.size)
    if bad.any():
        i, u = np.argwhere(bad)[0]
        nbytes = int((g_rows != h_rows).sum())
        t.add(f"{tag}.bytes_differing", nbytes)
        t.fail(f"{tag}: {nbytes} bytes in {bad.any(axis=1).sum()} envs differ, first env {c0 + i} unit {u}: "
               f"gpu {gu[i, u]:#018x} ({gu[i, u:u + 1].view(np.float64)[0]!r}) "
               f"host {hu[i, u]:#018x} ({hu[i, u:u + 1].view(np.float64)[0]!r})")


# ------------------------------------------------------------------------------------------ the host side

def _host_chunk(cfg, env_dims, rows0, c0, c1, launches, f32, atan, others):
    """Envs [c0, c1) in their own EmulBatch (env_offset shifted, so auto-reset draws as for the GPU env): load the
    saved rows, run each launch, compare it and the saved state after it."""
    from emul import emul, emul_info, emul_states
    from roborugby_b200._lib import Config
    R, B, D = env_dims
    c = Config.from_buffer_copy(cfg)
    c.env_offset = cfg.env_offset + c0
    m = c1 - c0
    batch = emul.EmulBatch(c, m, R, B, D)
    start = np.zeros((3 * R + 2 * B, m))
    emul_states.load(batch, start, np.ascontiguousarray(rows0[c0:c1]))
    t = Tally()
    t.stats = []   # per launch: the sums of the envs' contributions to the statistics vector
    for j, L in enumerate(launches):
        a = L["acts"][:, c0:c1].astype(np.float64)
        info = L["info"]
        h = emul_info.launch(batch, a, observe=True) if info else batch.launch(a, observe=True)
        g = {k: v[:, c0:c1] for k, v in L["gpu"].items() if k != "rows"}
        _compare_launch(t, g, h, c0, f32, D, atan, info)
        _compare_state(t, "state", L["gpu"]["rows"][c0:c1], emul_states.save(batch, start), c0)
        t.stats.append(h["stats"].sum(axis=0))
        if j == len(launches) - 1 and others is not None:
            _compare_other_kernels(t, cfg, batch, others, c0, c1, R, D, f32, atan, h)
    return t


def _compare_other_kernels(t, cfg, batch, others, c0, c1, R, D, f32, atan, h_last):
    """rr_observe, rr_observe_entity (every robot, a per-env ball index) and rr_assign_balls on the final state."""
    from emul import emul
    if D:
        for key, team in (("observe_h", "obs_h"), ("observe_g", "obs_g")):
            _compare_rows(t, key, others[key][None, c0:c1], h_last[team][-1:], f32, c0, atan)
    balls = others["balls"][c0:c1]
    for i in range(c1 - c0):
        st = batch.get_state(i)
        if D and cfg.observer not in (OBS_ALL, OBS_PRIOR):
            for r in range(R):
                want = (np.full(D, np.nan) if balls[i] < 0 else emul.observe_entity(cfg, st, r, int(balls[i]), D))
                _compare_rows(t, "observe_entity", others["entity"][r][None, c0 + i:c0 + i + 1], want[None, None], f32,
                              c0 + i, atan)
        got = others["assign"][c0 + i]
        want = emul.assign_balls(cfg, st, list(range(R)))
        t.add("assign_balls.rows")
        if not np.array_equal(got, want):
            t.fail(f"assign_balls env {c0 + i}: gpu {got} host {want}")


def _run_host(env, rows0, launches, f32, atan, others):
    from emul import emul, emul_info, emul_states
    emul_info.use_libm_sincos(False)    # the GPU's sin/cos routine, in both test libraries
    emul_states.lib()                   # (each library is built and loaded once, before the workers start)
    N = env.num_envs
    workers = max(1, os.cpu_count() or 1)
    nchunks = min(max(1, N // 256), 4 * workers)
    bounds = [(N * j // nchunks, N * (j + 1) // nchunks) for j in range(nchunks)]
    dims = (env.num_robots, env.num_balls, env.obs_dim)
    with ThreadPoolExecutor(workers) as ex:   # ctypes releases the GIL; emul_launch / emul_launch_info write no globals
        parts = list(ex.map(lambda b: _host_chunk(env.cfg, dims, rows0, b[0], b[1], launches, f32, atan, others), bounds))
    t = Tally()
    for p in parts:
        t.merge(p)
    t.stats = np.sum([p.stats for p in parts], axis=0)
    return t


# ------------------------------------------------------------------------------------------ the cases

def _gpu_launch(env, acts, K, info):
    env.clear_stats()
    out = env.step_k(torch.as_tensor(acts).cuda(), K, final_info=info)
    g = dict(obs_h=out[0].cpu().numpy(), obs_g=out[1].cpu().numpy(), rew=out[2].cpu().numpy(),
             done=out[3].cpu().numpy())
    if info:
        g.update(final_h=out[4]["final_obs"].cpu().numpy(), final_g=out[4]["final_obs_grumpy"].cpu().numpy(),
                 flags=out[4]["row_flags"].cpu().numpy())
    g["rows"] = env.save_states().cpu().numpy()
    return g, env.stats.cpu().numpy().copy()


@pytest.mark.parametrize("case", list(CASES))
def test_gpu_equals_host_build_bit_for_bit(oracle, case):
    from roborugby_b200.vec_env import RoboRugbyVecEnv
    preset, env_id, N, Ks, pipeline, f64, goals, observer, pools, extra = CASES[case]
    extra = dict(extra)
    others_wanted = extra.pop("others", False)
    kw = dict(time_limit=True, auto_reset=True, strict_reset=True)
    kw.update(extra)
    t0 = time.time()
    env = RoboRugbyVecEnv(env_id, N, preset=preset, device="cuda:0", seed=2026, out_dtype=torch.float64 if f64 else
                          torch.float32, goal_scoring=goals, observer=observer, pipeline=pipeline, **kw)
    f32, D = not f64, env.obs_dim
    atan = ATAN_COLS.get(env.cfg.observer, [])
    launch_type, blk, groups = k_step_variant(preset, goals, N, pipeline, _sms())
    contact = "contact" in pools
    pool_size = _inject(env, pools, oracle, max(Ks))
    if pools != "bench":   # a warm-up launch: returns, counted bits, error masks, naughty counts and prior poses
        env.step_k(torch.as_tensor(_actions(env, 4, 1, contact)).cuda(), 4)
    rows0 = env.save_states().cpu().numpy()
    launches, gpu_stats = [], []
    for j, (K, info) in enumerate(zip(Ks, (False, True))):
        acts = _actions(env, K, 100 + j, contact)
        n0 = env.launch_count
        g, s = _gpu_launch(env, acts, K, info)
        assert env.launch_count - n0 == groups + 1     # k_step launches, then the save
        launches.append(dict(acts=acts, info=info, gpu=g))
        gpu_stats.append(s)
    others = None
    if others_wanted:
        rng = np.random.default_rng(7)
        balls = rng.integers(-1, env.num_balls, N).astype(np.int32)
        others = dict(balls=balls, assign=env.assign_balls(list(range(env.num_robots))).cpu().numpy())
        if D:
            oh, og = env.observe()
            others.update(observe_h=oh.cpu().numpy(), observe_g=og.cpu().numpy())
            if env.cfg.observer not in (OBS_ALL, OBS_PRIOR):
                bt = torch.as_tensor(balls, device="cuda")
                others["entity"] = [env.observe_entity(r, bt).cpu().numpy() for r in range(env.num_robots)]
    t_gpu = time.time() - t0
    t = _run_host(env, rows0, launches, f32, atan, others)
    # statistics: the integer counts exactly, the returns up to summation order
    for j, (got, want) in enumerate(zip(gpu_stats, t.stats)):
        assert np.array_equal(got[COUNTS], want[COUNTS]), (j, got, want)
        assert np.allclose(got[RET], want[RET], rtol=1e-12, atol=1e-9), (j, got, want)
    rows = sum(v for k, v in t.n.items() if k.endswith(".rows"))
    av, ab = t.n.get("obs_h.atan_values", 0) + t.n.get("obs_g.atan_values", 0), \
        t.n.get("obs_h.atan_bit_equal", 0) + t.n.get("obs_g.atan_bit_equal", 0)
    print(f"{case}: {launch_type} {'double' if f64 else 'float'} INFO off + on, {blk}-thread blocks x {groups} launch(es), "
          f"{N} envs ({pool_size} pool states), K = {Ks}: {rows} rows, {t.n.get('state.bytes', 0)} state bytes and "
          f"{t.n['resets']} resets compared; {t.n.get('differences', 0)} differing "
          f"(state bytes {t.n.get('state.bytes_differing', 0)}, rows "
          f"{sum(v for k, v in t.n.items() if k.endswith('rows_differing'))}); squeeze replays "
          f"{int(sum(s[7] for s in gpu_stats))}; atan columns {ab}/{av} bit-equal; "
          f"gpu {t_gpu:.1f} s, host {time.time() - t0 - t_gpu:.1f} s")
    for f in t.first:
        print("  ", f)
    assert not t.first, t.first
    if pools == "bench":
        assert t.n["resets"] > 0 and gpu_stats[0][0] > 0      # episodes ended and were reset inside the launch
    env.close()


def test_gpu_side_x_line_block_equals_the_plain_evaluation():
    """rr_selftest which 1: the branch-free side x line block (sides_x_lines on the device) against
    sides_x_lines_plain on >= 1e8 simulator-shaped and adversarial inputs: nothing differs, and both the block and its
    fallback to ordinary divisions ran."""
    from roborugby_b200 import _lib
    lib = _lib.load()
    out = np.zeros(2, np.int64)
    n = 100_000_000
    rc = lib.rr_selftest(0, 1, n, 20261022, out.ctypes.data_as(C.c_void_p))
    assert rc == 0, lib.rr_last_error()
    print(f"side x line block: {n} inputs, {out[0]} differing, {out[1]} took the fallback")
    assert out[0] == 0, f"{out[0]} inputs differ from sides_x_lines_plain"
    assert 0 < out[1] < n
