"""RoboRugbyVecEnv — N independent RoboRugby episodes advanced in lockstep on one B200.

Host-side mirror of the reference's gym API for the step()/reset() path, batched:

    reference (one env)                      here (N envs, torch tensors on the GPU)
    env.reset() -> obs                       venv.reset() -> obs_happy [N, D]
    env.step(actions) -> obs, r, done, info  venv.step(actions [N, A]) -> obs_happy [N, D], r_happy [N],
                                                                            done [N], info
    info.adblGrumpyState / .dblGrumpyScore   info["obs_grumpy"] [N, D] / info["reward_grumpy"] [N]

(RR_EnvBase.py:202-216, :260-297, :562-566, :617-626.)  Observation, reward and done tensors are
persistent device buffers that every step() overwrites — clone them if they must survive the next
call.  All compute happens in librr_b200.so (hand-written sm_100a kernels) through the C ABI in
include/rr_b200.h; torch is only used for device memory, streams and torch.distributed.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib
from .constants import ENV_IDS, get_preset


class RoboRugbyVecEnv:
    def __init__(self, env_id="RoboRugbySimpleDuel-v2", num_envs=4096, preset="GAME", device="cuda:0", seed=0,
                 env_offset=0, time_limit=True, auto_reset=True, out_dtype=torch.float32, strict_reset=True,
                 n_actions=None, observer=None, reward_mask=None, reward_order=None, reward_mixins=None, flags=0,
                 goal_scoring=False, pipeline=1):
        if env_id not in ENV_IDS:
            raise ValueError(f"unknown env id {env_id!r}; expected one of {ENV_IDS}")
        self.lib = _lib.load()
        self.env_id = env_id
        self.preset = get_preset(preset)
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise ValueError("device must be a CUDA device")
        self.num_envs = int(num_envs)
        cfg = _lib.default_config(self.preset.index, env_id)
        cfg.time_limit = int(bool(time_limit))
        cfg.auto_reset = int(bool(auto_reset))
        cfg.out_f64 = int(out_dtype == torch.float64)
        cfg.strict_reset = int(bool(strict_reset))
        # class composition a la main.py:42-49: another observer / reward-mixin set on top of the id's defaults
        if observer is not None:
            cfg.observer = int(observer)
        if reward_mixins is not None:   # class-definition order, e.g. ("KeepMovingGuys", "ChasePosBall", "NaughtyBots")
            from .constants import reward_config_from_mixins
            reward_mask, reward_order = reward_config_from_mixins(reward_mixins)
        if reward_mask is not None:
            cfg.reward_mask = int(reward_mask)
            cfg.reward_order = 0
        if reward_order is not None:
            cfg.reward_order = int(reward_order)
        cfg.flags = int(flags)
        cfg.goal_scoring = int(bool(goal_scoring))   # goal scoring as intended (include/rr_b200.h); default: the reference's HEAD
        cfg.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
        cfg.env_offset = int(env_offset)
        _lib.check_config(cfg)   # ValueError for a reward_mask / reward_order no class composition produces, etc.
        if not torch.cuda.is_available():
            raise RuntimeError("RoboRugbyVecEnv needs a CUDA device: roborugby_b200 has no CPU fallback")
        self._open(cfg, n_actions, pipeline)

    def _open(self, cfg, n_actions, pipeline):
        """rr_create for cfg and the handle's derived attributes (the constructor and __deepcopy__)."""
        self.cfg = cfg
        self.out_dtype = torch.float64 if cfg.out_f64 else torch.float32
        self.discrete = bool(cfg.discrete)
        dev_index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        self._dev_index = dev_index
        h = C.c_void_p()
        _lib.check(self.lib.rr_create(C.byref(cfg), self.num_envs, dev_index, C.byref(h)))
        self._h = h
        self.num_robots = self.lib.rr_num_robots(h)
        self.num_balls = self.lib.rr_num_balls(h)
        self.obs_dim = self.lib.rr_obs_dim(h)
        self.max_episode_steps = self.lib.rr_max_steps(h)
        self.action_dim = self.num_robots if self.discrete else 2 * self.num_robots
        self.n_actions = self.action_dim if n_actions is None else int(n_actions)
        # statistics live in a torch tensor so torch.distributed can all-reduce them in place
        self.stats = torch.zeros(_lib.NUM_STATS, dtype=torch.float64, device=self.device)
        _lib.check(self.lib.rr_set_stats_buffer(h, self.stats.data_ptr()))
        self._bufs = {}
        self.pipeline = 1
        self._inflight = []
        if pipeline and int(pipeline) > 1:
            self.set_pipeline(pipeline)

    def __deepcopy__(self, memo):
        """copy.deepcopy(venv): a new handle with the same rr_config and pipeline setting whose envs are loaded with every
        env's saved row (save_states / load_states: the copy continues bit for bit, resets included) and a clone of the
        statistics.  Output buffers are not shared and a flush buffer is not carried over."""
        new = object.__new__(type(self))
        memo[id(self)] = new
        new.lib, new.env_id, new.preset, new.device, new.num_envs = self.lib, self.env_id, self.preset, self.device, self.num_envs
        new._open(_lib.Config.from_buffer_copy(self.cfg), self.n_actions, self.pipeline)
        new.load_states(self.save_states())
        new.stats.copy_(self.stats)
        return new

    # ------------------------------------------------------------------ sub-batch pipeline
    def set_pipeline(self, sub_batches):
        """Step the batch as `sub_batches` independent groups of blocks on the handle's own streams (rr_set_pipeline):
        a group held back by its slowest env delays only its own next launch.  With sub_batches > 1, step_k(..., join=False)
        returns without making the current stream wait for the groups, so back-to-back calls overlap; call join() before
        reading results.  Every other method joins by itself.  Results do not depend on the setting."""
        _lib.check(self.lib.rr_set_pipeline(self._h, int(sub_batches)))
        self.pipeline = int(sub_batches)

    def set_flush_buffer(self, buf):
        """Benchmark hygiene: `buf` (a CUDA uint8 tensor larger than the L2, or None) is overwritten in front of every step
        launch on the launching stream (rr_set_flush_buffer)."""
        self._flush = buf
        _lib.check(self.lib.rr_set_flush_buffer(self._h, buf.data_ptr() if buf is not None else None,
                                                buf.numel() if buf is not None else 0))

    def join(self):
        """Make the current stream wait (on the device) for every group's outstanding launches."""
        _lib.check(self.lib.rr_join(self._h, self._stream()))
        if self._inflight:
            # the current stream now waits for the groups; anything it frees after this point is ordered behind them
            self._inflight = []

    # ------------------------------------------------------------------ lifetime
    def close(self):
        if getattr(self, "_h", None):
            self.lib.rr_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ helpers
    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    def _out(self, k):
        """Persistent output buffers for k fused steps."""
        if k not in self._bufs:
            N, D = self.num_envs, max(self.obs_dim, 1)
            mk = lambda *s, dt=self.out_dtype: torch.empty(*s, dtype=dt, device=self.device)
            self._bufs[k] = dict(obs_h=mk(k, N, D), obs_g=mk(k, N, D), rew=mk(k, N, 2),
                                 done=mk(k, N, dt=torch.uint8))
        return self._bufs[k]

    def _check_actions(self, actions, k):
        want = torch.uint8 if self.discrete else torch.float32
        if actions.dtype != want:
            actions = actions.to(want)
        if actions.device != self.device:
            actions = actions.to(self.device, non_blocking=True)
        actions = actions.contiguous()
        if k == 1 and actions.dim() == 2:
            actions = actions.unsqueeze(0)
        if actions.dim() == 2 and actions.shape == (k, self.num_envs):
            actions = actions.unsqueeze(-1)
        if actions.dim() != 3 or actions.shape[0] != k or actions.shape[1] != self.num_envs:
            raise ValueError(f"actions must be [{k}, {self.num_envs}, A], got {tuple(actions.shape)}")
        return actions

    # ------------------------------------------------------------------ gym-like API
    def reset(self, mask=None):
        """reset() for every env (or those where mask is True); returns the happy observation."""
        mp = None
        if mask is not None:
            mask = mask.to(self.device, torch.uint8).contiguous()
            mp = mask.data_ptr()
        _lib.check(self.lib.rr_reset(self._h, mp, self._stream()))
        return self.observe()[0]

    def reset_fixed(self, mask=None, as_constructed=False):
        """reset(bln_randomize_pos=False): back to the stored starting layout (the env's first random placement
        unless set_starting_positions replaced it)."""
        mp = None
        if mask is not None:
            mask = mask.to(self.device, torch.uint8).contiguous()
            mp = mask.data_ptr()
        _lib.check(self.lib.rr_reset_fixed(self._h, mp, int(as_constructed), self._stream()))
        return self.observe()[0]

    def set_starting_positions(self, rob3, ball2):
        """_lst_starting_positions for every env: rob3 [N, R, 3] (x, y, rot) and ball2 [N, B, 2]; a single layout
        [R, 3] / [B, 2] (e.g. constants.config_standard(preset)) is broadcast."""
        N, R, B = self.num_envs, self.num_robots, self.num_balls
        rob3 = np.ascontiguousarray(np.broadcast_to(np.asarray(rob3, np.float64), (N, R, 3)))
        ball2 = np.ascontiguousarray(np.broadcast_to(np.asarray(ball2, np.float64), (N, B, 2)))
        p = lambda a: a.ctypes.data_as(C.c_void_p)
        _lib.check(self.lib.rr_set_starting_positions(self._h, p(rob3), p(ball2)))

    def get_starting_positions(self):
        N, R, B = self.num_envs, self.num_robots, self.num_balls
        rob3 = np.zeros((N, R, 3)); ball2 = np.zeros((N, B, 2))
        p = lambda a: a.ctypes.data_as(C.c_void_p)
        _lib.check(self.lib.rr_get_starting_positions(self._h, p(rob3), p(ball2)))
        return rob3, ball2

    def observe(self):
        b = self._out(1)
        if self.obs_dim:
            _lib.check(self.lib.rr_observe(self._h, b["obs_h"].data_ptr(), b["obs_g"].data_ptr(), self._stream()))
        return b["obs_h"][0, :, :self.obs_dim], b["obs_g"][0, :, :self.obs_dim]

    def observe_entity(self, robot, ball=None):
        """get_game_state(obj_robot=lstRobots[robot], obj_ball=lstBalls[ball]) for every env -> [N, D] (a fresh tensor).
        ball: None (the observer's default ball), an index, or an int32 tensor [N] with one index per env (negative:
        a NaN row).  RR_Observers.py:133-136, :187-203, :304-320."""
        out = torch.empty(self.num_envs, max(self.obs_dim, 1), dtype=self.out_dtype, device=self.device)
        bdev, bidx = None, -1
        if torch.is_tensor(ball):
            ball = ball.to(self.device, torch.int32).contiguous()
            assert ball.shape == (self.num_envs,)
            bdev = ball.data_ptr()
        elif ball is not None:
            bidx = int(ball)
        _lib.check(self.lib.rr_observe_entity(self._h, int(robot), bidx, bdev, out.data_ptr(), self._stream()))
        return out[:, :self.obs_dim]

    def assign_balls(self, robots):
        """The "Stephen" players' greedy nearest-ball assignment (DQN_pytorch_player.py:39-61) for the players driving
        `robots`, in every env -> int32 [N, len(robots)] on the device: ball index, or -1."""
        r = np.ascontiguousarray(robots, np.int32)
        out = torch.empty(self.num_envs, len(r), dtype=torch.int32, device=self.device)
        _lib.check(self.lib.rr_assign_balls(self._h, r.ctypes.data_as(C.c_void_p), len(r), out.data_ptr(), self._stream()))
        return out

    def step(self, actions, final_info=False):
        """One env-step for all envs.  actions: uint8 [N, A] (discrete ids) or float32 [N, A].  final_info=True adds to
        info what auto-reset would otherwise hide (see step_k): "final_observation" / "final_observation_grumpy" [N, D]
        (valid where done), "TimeLimit.truncated" and "raised" (bool [N])."""
        out = self.step_k(actions, 1, final_info=final_info)
        obs_h, obs_g, rew, done = out[:4]
        info = {"obs_grumpy": obs_g[0], "reward_grumpy": rew[0, :, 1]}
        if final_info:
            f = out[4]
            info.update({"final_observation": f["final_obs"][0], "final_observation_grumpy": f["final_obs_grumpy"][0],
                         "TimeLimit.truncated": f["truncated"][0], "raised": f["raised"][0]})
        return obs_h[0], rew[0, :, 0], done[0].bool(), info

    def _final_out(self, k):
        """Persistent rr_step_info buffers for k fused steps."""
        key = ("final", k)
        if key not in self._bufs:
            N, D = self.num_envs, max(self.obs_dim, 1)
            mk = lambda *s, dt=self.out_dtype: torch.empty(*s, dtype=dt, device=self.device)
            self._bufs[key] = dict(final_obs_h=mk(k, N, D), final_obs_g=mk(k, N, D), row_flags=mk(k, N, dt=torch.uint8))
        return self._bufs[key]

    def step_k(self, actions, k, join=True, final_info=False):
        """k fused env-steps in ONE kernel launch (one per group with a sub-batch pipeline).  actions [k, N, A]; returns
        obs_h [k,N,D], obs_g, rew [k,N,2], done [k,N] (uint8).  Envs that finish are reset inside the launch (auto_reset).
        join=False (pipeline > 1 only): do not make the current stream wait for the launches; the caller joins later and
        must not touch `actions` or the returned buffers before that.
        final_info=True (rr_step_info) returns a fifth element, a dict: "final_obs" / "final_obs_grumpy" [k, N, D], the
        observation of the state each done row ended in, before the auto-reset (rows with done == 0 hold whatever an earlier
        call left there); "row_flags" [k, N] (uint8, _lib.ROW_TRUNCATED | _lib.ROW_RAISED); "truncated" and "raised" (bool
        [k, N]): gym's info['TimeLimit.truncated'] and "the reference's step() raised".  A done row with neither is a real
        end of the episode.  The three buffers persist like the others and, with join=False, follow the same rule; since
        "truncated" and "raised" are computed from row_flags on the current stream, with join=False they are None: derive
        them from row_flags after join()."""
        actions = self._check_actions(actions, k)
        A = actions.shape[2]
        b = self._out(k)
        has_obs = self.obs_dim > 0
        f = self._final_out(k) if final_info else None
        _lib.check(self.lib.rr_step_info(self._h, actions.data_ptr(), A, k,
                                         b["obs_h"].data_ptr() if has_obs else None,
                                         b["obs_g"].data_ptr() if has_obs else None,
                                         b["rew"].data_ptr(), b["done"].data_ptr(),
                                         f["final_obs_h"].data_ptr() if f and has_obs else None,
                                         f["final_obs_g"].data_ptr() if f and has_obs else None,
                                         f["row_flags"].data_ptr() if f else None, self._stream()))
        joined = True
        if self.pipeline > 1:
            if join:
                self.join()
            else:
                # keep every action buffer alive until the groups have read it: the groups run on the handle's own streams,
                # which torch's stream-ordered allocator knows nothing about
                self._inflight.append(actions)
                joined = False
                if len(self._inflight) > 256:   # a caller that never joins: bound what is kept alive
                    self.join()
        out = (b["obs_h"][..., :self.obs_dim], b["obs_g"][..., :self.obs_dim], b["rew"], b["done"])
        if not final_info:
            return out
        fl = f["row_flags"]
        info = dict(final_obs=f["final_obs_h"][..., :self.obs_dim], final_obs_grumpy=f["final_obs_g"][..., :self.obs_dim],
                    row_flags=fl, truncated=(fl & _lib.ROW_TRUNCATED).bool() if joined else None,
                    raised=(fl & _lib.ROW_RAISED).bool() if joined else None)
        return out + (info,)

    def step_host(self, actions_host, k, out=None):
        """Same as step_k through the HOST-buffer entry point rr_step_host: `actions_host` is a pinned
        CPU tensor [k, N, A]; results land in pinned CPU tensors (returned, reused across calls)."""
        want = torch.uint8 if self.discrete else torch.float32
        assert actions_host.device.type == "cpu" and actions_host.dtype == want and actions_host.is_contiguous()
        A = actions_host.shape[-1] if actions_host.dim() == 3 else 1
        key = ("host", k)
        if out is None:
            if key not in self._bufs:
                N, D = self.num_envs, max(self.obs_dim, 1)
                mk = lambda *s, dt=self.out_dtype: torch.empty(*s, dtype=dt).pin_memory()
                self._bufs[key] = dict(obs_h=mk(k, N, D), obs_g=mk(k, N, D), rew=mk(k, N, 2),
                                       done=mk(k, N, dt=torch.uint8))
            out = self._bufs[key]
        has_obs = self.obs_dim > 0
        _lib.check(self.lib.rr_step_host(self._h, actions_host.data_ptr(), A, k,
                                         out["obs_h"].data_ptr() if has_obs else None,
                                         out["obs_g"].data_ptr() if has_obs and out.get("obs_g") is not None else None,
                                         out["rew"].data_ptr(), out["done"].data_ptr(), self._stream()))
        return out

    def step_host_begin(self, actions_host, k, slot):
        """rr_step_host_begin: enqueue k fused steps with HOST buffers and return a ticket at once.  `slot` picks one of the
        caller's sets of pinned result buffers (one per call kept in flight, at most 4): begin calls n + 1, n + 2 on other
        slots before ending call n."""
        want = torch.uint8 if self.discrete else torch.float32
        assert actions_host.device.type == "cpu" and actions_host.dtype == want and actions_host.is_contiguous()
        A = actions_host.shape[-1] if actions_host.dim() == 3 else 1
        key = ("host2", k, int(slot))
        if key not in self._bufs:
            N, D = self.num_envs, max(self.obs_dim, 1)
            mk = lambda *s, dt=self.out_dtype: torch.empty(*s, dtype=dt).pin_memory()
            self._bufs[key] = dict(obs_h=mk(k, N, D), obs_g=mk(k, N, D), rew=mk(k, N, 2), done=mk(k, N, dt=torch.uint8))
        out = self._bufs[key]
        has_obs = self.obs_dim > 0
        ticket = C.c_int32(-1)
        _lib.check(self.lib.rr_step_host_begin(self._h, actions_host.data_ptr(), A, k,
                                               out["obs_h"].data_ptr() if has_obs else None,
                                               out["obs_g"].data_ptr() if has_obs else None,
                                               out["rew"].data_ptr(), out["done"].data_ptr(), C.byref(ticket)))
        self._tickets = getattr(self, "_tickets", {})
        self._tickets[ticket.value] = (out, actions_host)
        return ticket.value

    def step_host_end(self, ticket):
        """Block until the call behind `ticket` has delivered its results; returns its pinned result buffers."""
        _lib.check(self.lib.rr_step_host_end(self._h, int(ticket)))
        return self._tickets[int(ticket)][0]

    # ------------------------------------------------------------------ introspection / parity
    def get_state(self):
        """Complete physics state as numpy arrays (layout of oracle/ref_harness.extract, batched)."""
        N, R, B = self.num_envs, self.num_robots, self.num_balls
        st = dict(rob=np.zeros((N, R, 7)), rhist=np.zeros((N, R, 3)), rflag=np.zeros((N, R, 3), np.int32),
                  ball=np.zeros((N, B, 8)), step=np.zeros(N, np.int32))
        p = lambda a: a.ctypes.data_as(C.c_void_p)
        _lib.check(self.lib.rr_get_state(self._h, p(st["rob"]), p(st["rhist"]), p(st["rflag"]), p(st["ball"]),
                                         p(st["step"])))
        return st

    def set_state(self, st):
        N, R, B = self.num_envs, self.num_robots, self.num_balls
        rob = np.ascontiguousarray(st["rob"], np.float64).reshape(N, R, 7)
        rhist = np.ascontiguousarray(st["rhist"], np.float64).reshape(N, R, 3)
        rflag = np.ascontiguousarray(st["rflag"], np.int32).reshape(N, R, 3)
        ball = np.ascontiguousarray(st["ball"], np.float64).reshape(N, B, 8)
        step = np.ascontiguousarray(st["step"], np.int32).reshape(N)
        p = lambda a: a.ctypes.data_as(C.c_void_p)
        _lib.check(self.lib.rr_set_state(self._h, p(rob), p(rhist), p(rflag), p(ball), p(step)))

    # ------------------------------------------------------------------ saved states on the device
    @property
    def state_row_bytes(self):
        """S: the width in bytes of one saved env row (rr_snapshot_bytes_per_env); it identifies the row layout."""
        return int(self.lib.rr_snapshot_bytes_per_env(self._h))

    def _indices(self, idx, n, bound, what):
        """idx as a contiguous int64 tensor on the env's device; ValueError unless it is an integer tensor [n] (n None: any
        length), IndexError, before anything is launched, for an entry >= bound and, for env indices, one < 0 (a negative
        slot keeps its env).  The check is one reduction, and for a device tensor one synchronisation."""
        if not torch.is_tensor(idx) or idx.dtype.is_floating_point or idx.dtype == torch.bool or idx.dim() != 1 or (
                n is not None and idx.numel() != n):
            raise ValueError(f"{what} must be an integer tensor [{'m' if n is None else n}]")
        bad = (idx >= bound) | (idx < 0) if what == "envs" else idx >= bound
        if bool(bad.any()):
            raise IndexError(f"{what} entries must be " + (f"in [0, {bound})" if what == "envs" else f"< {bound}"))
        return idx.to(self.device, torch.int64).contiguous()

    def save_states(self, envs=None, out=None):
        """Save env states on the device (rr_save_states): returns a contiguous uint8 tensor [m, state_row_bytes] on the
        env's device whose row j is env envs[j] (envs: int tensor [m], duplicates allowed; None: every env in order).
        `out` reuses a caller tensor of that shape.  Stream-ordered on the current stream; joins the sub-batch pipeline
        first, so it sees every step issued before it."""
        S = self.state_row_bytes
        ep = None
        if envs is not None:
            envs = self._indices(envs, None, self.num_envs, "envs")
            ep = envs.data_ptr()
        m = self.num_envs if envs is None else envs.numel()
        if m < 1:
            raise ValueError("nothing to save: envs is empty")
        if out is None:
            out = torch.empty(m, S, dtype=torch.uint8, device=self.device)
        else:
            self._check_rows(out, m)
        _lib.check(self.lib.rr_save_states(self._h, ep, m, out.data_ptr(), self._stream()))
        return out

    def load_states(self, rows, slots=None):
        """Load saved rows into the envs on the device (rr_load_states): env i receives rows[slots[i]] (slots: int tensor
        [num_envs]; a negative entry keeps env i; None: env i receives rows[i], and rows has num_envs rows).  rows: a
        contiguous uint8 tensor [m, state_row_bytes] on the env's device, from save_states of this or any handle with the
        same row width.  Every entry point then reports for env i what it reported for the saved env, and stepping it
        continues the saved env bit for bit until a random reset, which draws with env i's own global index.  The
        statistics are not touched.  Stream-ordered on the current stream, like save_states."""
        if not torch.is_tensor(rows) or rows.dim() != 2:
            raise ValueError("rows must be a uint8 tensor [m, state_row_bytes]")
        m = rows.shape[0]
        self._check_rows(rows, m)
        sp = None
        if slots is not None:
            slots = self._indices(slots, self.num_envs, m, "slots")
            sp = slots.data_ptr()
        elif m != self.num_envs:
            raise ValueError(f"without slots rows must have num_envs = {self.num_envs} rows, got {m}")
        _lib.check(self.lib.rr_load_states(self._h, rows.data_ptr(), m, sp, self._stream()))

    def _check_rows(self, rows, m):
        S = self.state_row_bytes
        if rows.dtype != torch.uint8 or tuple(rows.shape) != (m, S) or m < 1:
            raise ValueError(f"rows must be uint8 [{m}, {S}] (state_row_bytes of this env), got {rows.dtype} "
                             f"{tuple(rows.shape)}")
        if rows.device.type != "cuda" or rows.device.index != self._dev_index:
            raise ValueError(f"rows must be on {self.device}, got {rows.device}")
        if not rows.is_contiguous() or rows.data_ptr() % 16:
            raise ValueError("rows must be contiguous and 16-byte aligned")

    def goal_state(self):
        """Goal bookkeeping (goal_scoring=True): dict of numpy arrays alive [N, B] (0/1), score [N, 2] (happy goal,
        grumpy goal), destroyed [N, 2], dwell [N, 2, B]."""
        N, B = self.num_envs, self.num_balls
        alive = np.zeros(N, np.int32); score = np.zeros((N, 2), np.int32); destroyed = np.zeros(N, np.int32)
        dwell = np.zeros((N, 2, B), np.int32)
        p = lambda a: a.ctypes.data_as(C.c_void_p)
        _lib.check(self.lib.rr_goal_state(self._h, p(alive), p(score), p(destroyed), p(dwell)))
        return dict(alive=(alive[:, None] >> np.arange(B)) & 1, score=score,
                    destroyed=(destroyed[:, None] >> np.arange(2)) & 1, dwell=dwell)

    def error_mask(self, clear=False):
        err = np.zeros(self.num_envs, np.uint32)
        _lib.check(self.lib.rr_error_mask(self._h, err.ctypes.data_as(C.c_void_p), int(clear)))
        return err

    def last_naughty(self):
        n = np.zeros(self.num_envs, np.int32)
        _lib.check(self.lib.rr_last_naughty(self._h, n.ctypes.data_as(C.c_void_p)))
        return n

    # ------------------------------------------------------------------ statistics
    def get_stats(self):
        """Episode statistics of THIS shard since the last clear_stats(), as a dict."""
        self.join()
        v = self.stats.cpu().tolist()
        return dict(zip(_lib.STAT_NAMES, v))

    def clear_stats(self):
        self.join()
        self.stats.zero_()

    def reduce_stats(self, group=None):
        """Sum the statistics vector over all ranks (one NCCL all-reduce of 64 bytes over
        NVLink/NVSwitch; the env shards themselves never exchange state).  Returns a dict of the
        GLOBAL statistics; the local vector is left untouched."""
        from .stats import allreduce_stats
        self.join()
        return allreduce_stats(self.stats, group)

    @property
    def launch_count(self):
        return int(self.lib.rr_launch_count(self._h))

    @property
    def state_bytes_per_env(self):
        return int(self.lib.rr_state_bytes_per_env(self._h))
