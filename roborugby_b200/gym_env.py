"""Single-env, drop-in mirror of the reference's gym API on top of the CUDA simulator.

    import roborugby_b200 as rr
    env = rr.make("RoboRugbySimpleDuel-v2")           # robo_rugby/__init__.py:20-26
    obs = env.reset()
    obs, reward, done, info = env.step([3, 0, 1, 7])  # classic gym 4-tuple (RR_EnvBase.py:260-297)
    info.adblGrumpyState, info.dblGrumpyScore          # RR_EnvBase.py:562-566

Every call is one kernel launch on a batch of ONE episode plus a device->host copy, so this class
exists for API compatibility and parity tests; throughput comes from RoboRugbyVecEnv.  Exceptions
of the reference (step after done, too many commands, unresolved collisions) are raised as
`Exception` with the reference's messages.  Rendering is out of scope (SURVEY.md §2 row 12).
"""
import copy

import numpy as np
import torch

from . import _lib
from .constants import TEAM_GRUMPY, TEAM_HAPPY, get_preset
from .vec_env import RoboRugbyVecEnv


class Discrete:
    """gym.spaces.Discrete stand-in (gym is not a dependency)."""

    def __init__(self, n):
        self.n, self.shape, self.dtype = int(n), (), np.dtype(np.int64)

    def sample(self):
        return int(np.random.randint(self.n))

    def contains(self, x):
        return 0 <= int(x) < self.n


class Box:
    """gym.spaces.Box stand-in."""

    def __init__(self, low, high, shape=None, dtype=np.float32):
        shape = tuple(np.asarray(low).shape if shape is None else shape)
        self.shape, self.dtype = shape, np.dtype(dtype)
        self.low = np.broadcast_to(np.asarray(low, dtype), shape).copy()
        self.high = np.broadcast_to(np.asarray(high, dtype), shape).copy()

    def sample(self):
        return np.random.uniform(self.low, self.high).astype(self.dtype)

    def contains(self, x):
        x = np.asarray(x)
        return x.shape == self.shape and bool(np.all(x >= self.low) and np.all(x <= self.high))


class EnvSpec:
    def __init__(self, env_id, max_episode_steps):
        self.id, self.max_episode_steps = env_id, max_episode_steps
        self.nondeterministic, self.reward_threshold = True, 1.0  # robo_rugby/__init__.py:8-9


class DebugInfo(dict):
    """RR_EnvBase.py:562-566."""

    def __init__(self, adblGrumpyState, dblGrumpyScore):
        super().__init__()
        self.adblGrumpyState = adblGrumpyState
        self.dblGrumpyScore = dblGrumpyScore


class _GoalView:
    """sprHappyGoal / sprGrumpyGoal (RR_Goal.py).  At the reference's HEAD scoring is dead code (SURVEY.md §0.4): the
    score is 0 and a goal is never destroyed.  With goal_scoring=True (goal scoring as intended, include/rr_b200.h)
    both reflect the env's goal bookkeeping."""

    def __init__(self, env=None, index=0):
        self._env, self._index = env, index

    def get_score(self):
        if self._env is None:
            return 0
        return int(self._env._v.goal_state()["score"][0, self._index])

    def is_destroyed(self):
        if self._env is None:
            return False
        return bool(self._env._v.goal_state()["destroyed"][0, self._index])


class _RectView:
    """The read-only part of a sprite's FloatRect that scripts look at (MyUtils.py:114-354)."""

    def __init__(self, cx, cy, left, right, top, bottom, rotation=0.0):
        self.centerx, self.centery, self.left, self.right, self.top, self.bottom = cx, cy, left, right, top, bottom
        self.rotation = rotation

    @property
    def center(self):
        return (self.centerx, self.centery)


class RobotView:
    """lstRobots[i] (RR_Robot.py): identity (index, team) plus a snapshot of the pose taken when it is read."""

    def __init__(self, env, index, team):
        self._env, self.index, self.intTeam = env, index, team

    @property
    def rectDbl(self):
        r = self._env.get_state()["rob"][self.index]
        return _RectView(*r[:6], rotation=r[6])

    @property
    def dblRotation(self):
        return float(self._env.get_state()["rob"][self.index][6])

    @property
    def lngLThrust(self):
        return int(self._env.get_state()["rflag"][self.index][0])

    @property
    def lngRThrust(self):
        return int(self._env.get_state()["rflag"][self.index][1])


class BallView:
    """lstBalls[i] (RR_Ball.py): positive balls first (RR_EnvBase.py:62-68, :101-109)."""

    def __init__(self, env, index, positive):
        self._env, self.index, self.is_positive, self.is_negative = env, index, positive, not positive

    @property
    def rectDbl(self):
        return _RectView(*self._env.get_state()["ball"][self.index][:6])

    @property
    def dbl_velocity_x(self):
        return float(self._env.get_state()["ball"][self.index][6])

    @property
    def dbl_velocity_y(self):
        return float(self._env.get_state()["ball"][self.index][7])


# GameEnv_Simple._dct_thrust_from_direction (RR_EnvBase.py:593-602)
_THRUST = {0: (1, 1), 1: (-1, -1), 2: (-1, 1), 3: (1, -1), 4: (0, 1), 5: (1, 0), 6: (-1, 0), 7: (0, -1)}


class RoboRugbyEnv:
    """One episode with the reference's method surface.

    time_limit=False is the raw class (done when lngStepCount > GAME_LENGTH_STEPS, :555-559);
    time_limit=True is what gym.make() returns: the TimeLimit wrapper ends the episode at
    elapsed == max_episode_steps and sets info['TimeLimit.truncated']."""

    metadata = {"render.modes": ["human", "rgb_array"], "video.frames_per_second": 30}
    reward_range = (-float("inf"), float("inf"))

    def __init__(self, env_id, preset="GAME", device="cuda:0", seed=0, time_limit=False, lst_starting_config=None,
                 reward_mixins=None, observer=None, goal_scoring=False):
        """reward_mixins: names of RR_ScoreKeepers.py mixins in class-definition order, composed on top of `env_id`'s
        observer and action space the way main.py:42-49 composes ad-hoc classes (None: the id's own mixins)."""
        self.preset = get_preset(preset)
        self.time_limit = bool(time_limit)
        self._v = RoboRugbyVecEnv(env_id, 1, preset=self.preset, device=device, seed=seed, time_limit=time_limit,
                                  auto_reset=False, out_dtype=torch.float64, strict_reset=True,
                                  reward_mixins=reward_mixins, observer=observer, goal_scoring=goal_scoring)
        self.spec = EnvSpec(env_id, self._v.max_episode_steps)
        R = self._v.num_robots
        if self._v.discrete:
            self.action_space = Discrete(8)  # RR_EnvBase.py:608-610
        else:
            n = 2 * self.preset.num_robots_happy  # :118-123
            self.action_space = Box(-np.ones(n, np.float32), np.ones(n, np.float32), dtype=np.float32)
        hi = max(self.preset.arena_width, self.preset.arena_height, 360)  # RR_Observers.py:30-37
        self.observation_space = Box(-hi, hi, shape=(self._v.obs_dim,), dtype=np.float32) if self._v.obs_dim else None
        self.sprHappyGoal = _GoalView(self, 0) if goal_scoring else _GoalView()
        self.sprGrumpyGoal = _GoalView(self, 1) if goal_scoring else _GoalView()
        # entity lists the reference's scripts index into (main.py:59-63, RR_EnvBase.py:54-68)
        nh, npos = self.preset.num_robots_happy, self.preset.num_ball_pos
        self.lstRobots = [RobotView(self, i, TEAM_HAPPY if i < nh else TEAM_GRUMPY) for i in range(R)]
        self.lstBalls = [BallView(self, i, i < npos) for i in range(self._v.num_balls)]
        self._reward = {TEAM_HAPPY: 0.0, TEAM_GRUMPY: 0.0}
        self._elapsed = 0
        self.np_random = None
        if lst_starting_config is not None:  # GameEnv(lst_starting_config) (RR_EnvBase.py:112-116)
            self._v.set_starting_positions(np.asarray(lst_starting_config[0], np.float64),
                                           np.asarray(lst_starting_config[1], np.float64))
            self._v.reset_fixed(as_constructed=True)

    def __deepcopy__(self, memo):
        """copy.deepcopy(env), as planning code written against the reference branches an env: the episode goes on from
        the same state in a new handle (RoboRugbyVecEnv.__deepcopy__: the env's saved row on the device), and the wrapper's
        own state (TimeLimit's elapsed count, the last rewards, the views, which now look at the copy) is copied."""
        new = object.__new__(type(self))
        memo[id(self)] = new
        for k, v in self.__dict__.items():
            setattr(new, k, copy.deepcopy(v, memo))   # _v through RoboRugbyVecEnv.__deepcopy__; _elapsed, _reward, views
        return new

    # -- gym.Env surface -------------------------------------------------------------------
    @property
    def unwrapped(self):
        return self

    def seed(self, seed=None):  # RR_EnvBase.py:568-570 (the reference never uses this RNG either)
        self.np_random = np.random.RandomState(None if seed is None else int(seed) % (2 ** 32))
        return [seed]

    def close(self):
        self._v.close()

    def render(self, mode="human"):
        raise NotImplementedError("rendering is out of scope for the batched simulator (SURVEY.md §2 row 12)")

    def reset(self, bln_randomize_pos=True):
        if bln_randomize_pos:
            self._v.reset()
        else:  # back to _lst_starting_positions (RR_EnvBase.py:213-214)
            self._v.reset_fixed()
        self._elapsed = 0
        self._reward = {TEAM_HAPPY: 0.0, TEAM_GRUMPY: 0.0}
        return self.get_game_state()

    def step(self, lstArgs):
        arr = np.concatenate(lstArgs, axis=None) if len(lstArgs) else np.zeros(0)  # RR_EnvBase.py:269, :619
        R = self._v.num_robots
        if self._v.discrete:
            if len(arr) > R:
                raise Exception(f"{len(arr)} commands but only {R} robots.")  # :621-622
            act = torch.as_tensor(np.asarray(arr, np.uint8).reshape(1, -1))
        else:
            if len(arr) > 2 * R:
                raise Exception(f"{len(arr)} commands but only {2 * R} robot engines.")  # :270-271
            act = torch.as_tensor(np.asarray(arr, np.float32).reshape(1, -1))
        obs_h, obs_g, rew, done = self._v.step_k(act, 1)
        err = int(self._v.error_mask(clear=True)[0])
        if err:
            msgs = [m for b, m in _lib.ERR_BITS.items() if err & b]
            raise Exception("; ".join(msgs))
        rew = rew[0, 0].tolist()
        self._reward = {TEAM_HAPPY: rew[0], TEAM_GRUMPY: rew[1]}
        self._elapsed += 1
        d = bool(done[0, 0].item())
        info = DebugInfo(self._np_obs(obs_g), rew[1])
        if self.time_limit and self._elapsed >= self.spec.max_episode_steps:
            info["TimeLimit.truncated"] = not self.game_is_done()
        # GameEnv.step returns self.get_game_state() (no team, RR_EnvBase.py:296): None for PosBall_BasicLidar, the
        # happy team's observation for the others
        obs = None if self._v.cfg.observer == _lib.OBS_BASIC_LIDAR else self._np_obs(obs_h)
        return obs, rew[0], d, info

    # -- introspection used by the training scripts --------------------------------------------
    def _np_obs(self, t):
        if self._v.obs_dim == 0:
            return None
        a = t[0, 0].cpu().numpy().astype(np.float64)
        return None if np.isnan(a).all() else a

    @property
    def lstHappyBots(self):
        return self.lstRobots[:self.preset.num_robots_happy]

    @property
    def lstGrumpyBots(self):
        return self.lstRobots[self.preset.num_robots_happy:]

    @property
    def lstPosBalls(self):
        return self.lstBalls[:self.preset.num_ball_pos]

    @property
    def lstNegBalls(self):
        return self.lstBalls[self.preset.num_ball_pos:]

    def _entity_obs(self, robot, ball):
        a = self._v.observe_entity(robot.index, None if ball is None else ball.index)[0].cpu().numpy().astype(np.float64)
        return None if np.isnan(a).all() else a

    def get_game_state(self, int_team=None, obj_robot=None, obj_ball=None):
        """get_game_state(int_team, obj_robot, obj_ball) with every observer's own rules (RR_Observers.py:50-60,
        :133-141, :187-203, :304-320).  obj_robot / obj_ball are entries of lstRobots / lstBalls."""
        ob = self._v.cfg.observer
        if ob == _lib.OBS_NONE:
            return None
        if ob in (_lib.OBS_ALLCOORDS, _lib.OBS_ALLCOORDS_PRIOR):
            if int_team is None:
                int_team = TEAM_HAPPY
            if obj_robot:
                raise NotImplementedError("Robot-specific state output not supported.")  # :59-60
        elif ob == _lib.OBS_BASIC_LIDAR:
            if obj_robot:
                return self._entity_obs(obj_robot, None)  # :134-135 (obj_ball is ignored: lstPosBalls[0])
            if int_team not in (TEAM_HAPPY, TEAM_GRUMPY):
                return None  # :140-141
        else:  # the two 6-way lidar observers, :187-203 / :304-320
            if int_team is not None and obj_robot is not None:
                assert obj_robot.intTeam == int_team
            if obj_robot is not None or obj_ball is not None:
                if obj_robot is None:
                    bots = self.lstHappyBots if int_team in (None, TEAM_HAPPY) else self.lstGrumpyBots
                    if not bots:
                        return None
                    obj_robot = bots[0]
                return self._entity_obs(obj_robot, obj_ball)
            if int_team is None:
                int_team = TEAM_HAPPY
        oh, og = self._v.observe()
        t = oh if int_team == TEAM_HAPPY else og
        a = t[0].cpu().numpy().astype(np.float64)
        return None if np.isnan(a).all() else a

    def get_reward(self, int_team=TEAM_HAPPY):
        return self._reward[TEAM_HAPPY if int_team == TEAM_HAPPY else TEAM_GRUMPY]

    def game_is_done(self):  # RR_EnvBase.py:555-559
        if int(self._v.get_state()["step"][0]) > self.spec.max_episode_steps:
            return True
        if not self._v.cfg.goal_scoring:
            return False
        g = self._v.goal_state()
        return bool(g["destroyed"][0].any() or not g["alive"][0].any())

    @property
    def lngStepCount(self):
        return int(self._v.get_state()["step"][0])

    def _get_positions(self):  # RR_EnvBase.py:125-129
        st = self._v.get_state()
        return [[(r[0], r[1], r[6]) for r in st["rob"][0]], [(b[0], b[1]) for b in st["ball"][0]]]

    @staticmethod
    def thrust_from_direction(direction):  # RR_EnvBase.py:604-606
        return _THRUST[int(direction)]

    # parity harness
    def get_state(self):
        st = self._v.get_state()
        return {k: v[0] for k, v in st.items()}

    def set_state(self, st):
        self._v.set_state({k: np.asarray(v)[None] for k, v in st.items()})


_REGISTRY = {
    "RoboRugby-v0": "GameEnv",
    "RoboRugbySimple-v0": "SimpleChasePos",
    "RoboRugbySimpleDuel-v2": "SimpleDuel2",
    "RoboRugbySimpleDuel-v3": "SimpleDuel3",
}


def spec(env_id, preset="GAME"):
    if env_id not in _REGISTRY:
        raise KeyError(env_id)
    return EnvSpec(env_id, get_preset(preset).game_length_steps)


def make(env_id, preset="GAME", device="cuda:0", seed=0):
    """gym.make(id): the registered class wrapped by TimeLimit(max_episode_steps=GAME_LENGTH_STEPS)."""
    if env_id not in _REGISTRY:
        raise KeyError(f"No registered env with id: {env_id}")
    return RoboRugbyEnv(env_id, preset=preset, device=device, seed=seed, time_limit=True)
