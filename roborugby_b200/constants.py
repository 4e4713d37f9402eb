"""The two constant sets of the reference (robo_rugby/gym_env/RR_Constants.py:4-34).

The reference selects them with one import-time flag, GAME_MODE; here they are two named presets
that can coexist in one process.  Kernels are instantiated for these entity counts.
"""
from dataclasses import dataclass


@dataclass(frozen=True)
class Preset:
    name: str
    index: int             # RR_PRESET_* in include/rr_b200.h
    arena_width: int       # ARENA_WIDTH   :6
    arena_height: int      # ARENA_HEIGHT  :7
    num_robots_happy: int  # :32
    num_robots_grumpy: int  # :33
    num_ball_pos: int      # :30
    num_ball_neg: int      # :31
    game_length_steps: int  # :25
    framerate: int = 30    # :23

    @property
    def num_robots_total(self):
        return self.num_robots_happy + self.num_robots_grumpy

    @property
    def num_balls_total(self):
        return self.num_ball_pos + self.num_ball_neg


GAME = Preset("GAME", 0, 800, 800, 2, 2, 4, 4, 4500)
TRAIN = Preset("TRAIN", 1, 600, 600, 1, 0, 1, 0, 300)
PRESETS = {"GAME": GAME, "TRAIN": TRAIN}

TEAM_HAPPY, TEAM_GRUMPY = 1, -1  # :52-53
MOVES_PER_FRAME = 12             # :12-13

ENV_IDS = ("RoboRugby-v0", "RoboRugbySimple-v0", "RoboRugbySimpleDuel-v2", "RoboRugbySimpleDuel-v3")


def get_preset(p):
    if isinstance(p, Preset):
        return p
    return PRESETS[str(p).upper()]


def config_standard(preset):
    """GameEnv.CONFIG_STANDARD (RR_EnvBase.py:32-52) for a preset: ([R x (x, y, rot)], [B x (x, y)]).

    The reference lists 4 robots and 8 balls, so it only fits the GAME entity counts (with TRAIN constants the
    reference raises "Robot count mismatch", :138-139)."""
    p = get_preset(preset)
    W, H = float(p.arena_width), float(p.arena_height)
    w5, h5 = W / 5, H / 5
    robots = [(W / 2 + 1 * w5, H - 1 * h5, 135.0), (W / 2 + 2 * w5, H - 2 * h5, 135.0),
              (W / 2 - 1 * w5, 1 * h5, 315.0), (W / 2 - 2 * w5, 2 * h5, 315.0)]
    balls = [(w5 * 1, H - h5 * 1), (w5 * 2, H - h5 * 2), (w5 * 3, H - h5 * 3), (w5 * 4, H - h5 * 4),
             (W / 2, h5), (W / 2, H - h5), (w5, H / 2), (W - w5, H / 2)]
    if p.num_robots_total != len(robots) or p.num_balls_total != len(balls):
        raise ValueError(f"Robot count mismatch. {p.num_robots_total} != {len(robots)}.")
    return robots, balls


# Reward mixins (RR_ScoreKeepers.py): name -> (rr_config.reward_mask bit RR_REW_*, rr_config.reward_order id RR_MIX_*)
REWARD_MIXINS = {
    "ChasePosBall": (1, 1), "PushPosBallsToGoal": (2, 2), "NaughtyBots": (4, 3), "DontDriveInGoals": (8, 4),
    "KeepMovingGuys": (16, 5), "BaseDestruction": (32, 6), "PushNegBallsFromGoal": (64, 7),
}


def reward_config_from_mixins(mixins):
    """(reward_mask, reward_order) for a class composed as `class Env(*mixins, Observer, GameEnv_Simple)`.

    Every on_step_end calls super() first and then adds its own terms, so the bodies execute in reverse MRO order;
    NaughtyBots.on_step_end (RR_ScoreKeepers.py:130-135) does not call super(), so the mixins listed AFTER it never
    run theirs (their on_step_begin hooks still do, which is why they stay in the mask)."""
    mask, chain = 0, []
    for name in mixins:
        if name not in REWARD_MIXINS:
            raise ValueError(f"unknown reward mixin {name!r}; expected one of {sorted(REWARD_MIXINS)}")
        if mask & REWARD_MIXINS[name][0]:   # Python refuses such a class: "duplicate base class"
            raise ValueError(f"reward mixin {name!r} listed twice")
        mask |= REWARD_MIXINS[name][0]
    for name in mixins:           # MRO order; the chain of super() calls stops at NaughtyBots
        chain.append(name)
        if name == "NaughtyBots":
            break
    order = 0
    for n, name in enumerate(reversed(chain)):
        order |= REWARD_MIXINS[name][1] << (4 * n)
    return mask, order
