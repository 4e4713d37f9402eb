/* rr_oracle.h — CPU restatement of the RoboRugby reference step()/reset() path.
 *
 * TEST INFRASTRUCTURE ONLY.  This library is the parity oracle: only tests/, the smoke check in
 * __graft_entry__.py and the cpu_baseline / --impl reference legs of bench.py may load it.  The
 * product (roborugby_b200/) never links, imports or calls it and has no CPU fallback.
 *
 * Parity status: PINNED.  The reference ships no tests or golden vectors (SURVEY.md §4); the
 * oracle is pinned against outputs of the reference itself, executed in the build container by
 * oracle/gen_golden.py (stub pygame/gym, unmodified reference sources) and committed under
 * tests/golden/.  tests/test_oracle_golden.py requires bit-for-bit equality on every record.
 *
 * The restatement follows the reference object model (FloatRect with redundant, independently
 * drifting centre/left/right/top/bottom doubles; robot pose history ring; module-global scratch
 * rect) and its exact order of IEEE-754 double operations; it must be compiled with
 * -ffp-contract=off and linked against the same libm CPython uses.
 */
#ifndef RR_ORACLE_H
#define RR_ORACLE_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RRO_MAX_ROBOTS 8
#define RRO_MAX_BALLS 16
#define RRO_MAX_OBS 64

/* reward mixins (RR_ScoreKeepers.py) */
#define RRO_REW_CHASE 1u    /* ChasePosBall        :46-66   */
#define RRO_REW_PUSHPOS 2u  /* PushPosBallsToGoal  :138-157 */
#define RRO_REW_NAUGHTY 4u  /* NaughtyBots         :112-135 */
#define RRO_REW_DONTDRIVE 8u        /* DontDriveInGoals     :69-83   */
#define RRO_REW_KEEPMOVING 16u      /* KeepMovingGuys       :86-98   */
#define RRO_REW_BASEDESTRUCTION 32u /* BaseDestruction      :101-111 */
#define RRO_REW_PUSHNEG 64u         /* PushNegBallsFromGoal :160-179 */
/* on_step_end execution sequence (reward_order): one id per nibble, low nibble first, 0 ends */
#define RRO_MIX_CHASE 1u
#define RRO_MIX_PUSHPOS 2u
#define RRO_MIX_NAUGHTY 3u
#define RRO_MIX_DONTDRIVE 4u
#define RRO_MIX_KEEPMOVING 5u
#define RRO_MIX_BASEDESTRUCTION 6u
#define RRO_MIX_PUSHNEG 7u

/* observers (RR_Observers.py) */
#define RRO_OBS_NONE 0
#define RRO_OBS_BASIC_LIDAR 1 /* PosBall_BasicLidar      :116-166, 5 values  */
#define RRO_OBS_LIDAR6_V2 2   /* SingleBall_6wayLidar_v2 :287-406, 11 values */
#define RRO_OBS_ALLCOORDS 3   /* AllCoords               :47-83, 3R+2B values */
#define RRO_OBS_ALLCOORDS_PRIOR 4 /* AllCoords_WithPrior :86-110, 6R+4B values */
#define RRO_OBS_LIDAR6_V1 5   /* SingleBall_6wayLidar    :168-284, 11 values (what main.py composes for the "Stephen" player) */

/* error bits: the Python exceptions of the path (SURVEY.md §5) */
#define RRO_ERR_STEP_AFTER_DONE 1u      /* RR_EnvBase.py:261-262 */
#define RRO_ERR_TOO_MANY_COMMANDS 2u    /* :270-271, :621-622    */
#define RRO_ERR_BOT_COLLISIONS 4u       /* :312-313              */
#define RRO_ERR_UNDO_FAILED 8u          /* :324-325              */
#define RRO_ERR_ROBOTS_STUCK 16u        /* :327-330              */
#define RRO_ERR_UNRESOLVED_FRAME 32u    /* :417-421              */
#define RRO_ERR_COINCIDENT_BALLS 64u    /* RR_TrashyPhysics.py:249-250 */
#define RRO_ERR_DIV0 128u               /* MyUtils.py:25         */
#define RRO_ERR_BAD_ACTION 512u        /* discrete id outside 0..7 (KeyError, RR_EnvBase.py:593-606); NaN or +-inf thrust
                                           (round() raises, RR_Robot.py:100-102) */

typedef struct {
  int arena_w, arena_h;      /* RR_Constants.py:6-7   */
  int n_happy, n_grumpy;     /* :32-33                */
  int n_pos, n_neg;          /* :30-31                */
  int game_length_steps;     /* :25                   */
  int game_mode;             /* :4 (only changes the behaviour at RR_EnvBase.py:417-421) */
  uint32_t reward_mask;      /* RRO_REW_*             */
  int observer;              /* RRO_OBS_*             */
  int discrete;              /* 1: GameEnv_Simple.step (RR_EnvBase.py:617-626) */
  int time_limit;            /* 1: gym TimeLimit semantics (done at step >= T), 0: raw (step > T) */
  uint32_t reward_order;     /* RRO_MIX_* sequence in which the on_step_end bodies execute: reverse MRO order, cut at
                                NaughtyBots, whose on_step_end does not call super() (RR_ScoreKeepers.py:130-135);
                                0 = Naughty, Chase, PushPos, PushNeg, BaseDestruction, DontDrive, KeepMoving */
  int goal_scoring;          /* 1: goal scoring as intended (RR_Goal.py:54-91 + RR_EnvBase.py:461-511 made live; the
                                reference side is oracle/ref_harness.py _GOAL_SCORING_PATCHES); 0: the reference's HEAD,
                                where that code is dead and scores / destruction are constants. */
} rro_config;

typedef struct rro_env rro_env;

void rro_default_config(rro_config *cfg, int game_mode, const char *env_id);
rro_env *rro_create(const rro_config *cfg);
void rro_destroy(rro_env *e);
int rro_obs_dim(const rro_env *e);
int rro_num_robots(const rro_env *e);
int rro_num_balls(const rro_env *e);

/* State layout = oracle/ref_harness.py extract(): rob[R][7], rhist[R][3], rflag[R][3], ball[B][8]. */
void rro_set_state(rro_env *e, const double *rob, const double *rhist, const int32_t *rflag,
                   const double *ball, int32_t step);
void rro_get_state(const rro_env *e, double *rob, double *rhist, int32_t *rflag, double *ball,
                   int32_t *step);

/* One step.  `actions` holds n_actions values: discrete ids (as doubles) when cfg.discrete, else
 * 2 thrust values per robot.  obs_h / obs_g receive obs_dim doubles (NaN-filled when the
 * reference returns None).  rew[2] = happy, grumpy.  Returns the error mask (0 = ok). */
uint32_t rro_step(rro_env *e, const double *actions, int n_actions, double *obs_h, double *obs_g,
                  double *rew, int32_t *done, int32_t *naughty_count);

/* Observation of the current state (get_game_state(int_team=...)); team = +1 happy, -1 grumpy. */
uint32_t rro_observe(rro_env *e, int team, double *obs);
/* get_game_state(obj_robot=lstRobots[robot], obj_ball=lstBalls[ball]); ball < 0 = default ball.  Returns the error mask,
 * or 0xffffffff when the observer does not support robot-specific output (AllCoords raises NotImplementedError). */
uint32_t rro_observe_entity(rro_env *e, int robot, int ball, double *obs);
/* The "Stephen" players' greedy nearest-ball assignment (DQN_pytorch_player.py:39-61): balls inside either goal's
 * triangle are ignored; (player, ball) pairs by ascending distance, each player one ball, each ball one player.
 * assign[i] = ball index of robots[i], or -1 (the player then returns thrust (0, 0), :68-69). */
void rro_assign_balls(rro_env *e, const int *robots, int n, int *assign);

/* reset(bln_randomize_pos) fed from an explicit stream of randint() results (RR_EnvBase.py:155-216).
 * Returns the number of draws consumed, or -1 if the stream ran out. */
int rro_reset_draws(rro_env *e, int randomize, const int32_t *draws, int n_draws);
/* Same reset, drawing from the counter-based generator the CUDA product uses (Philox4x32-10,
 * key = seed, counter = (env_index, episode, draw/4)); see include/rr_b200.h. */
void rro_reset_philox(rro_env *e, uint64_t seed, uint64_t env_index, uint32_t episode);
/* relaxed = 1: the product's strict_reset = 0 mode, which adds two rejection rules to the placement loop (a robot whose
 * rotated rect intersects an already placed one; a ball within 14 px of another) so that no episode starts in a state
 * on which the reference raises or hangs.  relaxed = 0 is the reference's placement. */
void rro_reset_philox_mode(rro_env *e, uint64_t seed, uint64_t env_index, uint32_t episode, int relaxed);

/* The reference keeps one module-global scratch rect whose centre is updated incrementally
 * (RR_TrashyPhysics.py:29-35,54-55).  mode 0 = faithful (state carried between calls, what the
 * Python process does); mode 1 = fresh (centre assigned exactly; what a batched simulator can
 * do).  rro_scratch_reset() restores the import-time value. */
void rro_scratch_mode(int fresh);
void rro_scratch_reset(void);

void rro_set_starting_positions(rro_env *e, const double *rob3, const double *ball2);
long rro_rollout(rro_env *e, long n_steps, uint64_t seed);

/* Goal bookkeeping of the current state (goal_scoring): alive[B]; score[2] = get_score() of the happy and the grumpy
 * goal; destroyed[2]; dwell[2][B] (steps the ball has stayed in that goal, 0 = not tracked); delta = score change
 * committed by the last step (+ = good for happy). */
void rro_goal_state(const rro_env *e, int32_t *alive, int32_t *score, int32_t *destroyed, int32_t *dwell, int32_t *delta);

/* Test instrumentation: number of physics frames since the last clear in which all ten resolve passes failed and the
 * undo loop ran (RR_EnvBase.py:284-287): the "ball pinned between a robot and a wall" frames. */
long rro_debug_failed_frames(int clear);

/* Philox4x32-10 exposed for the RNG known-answer test. */
void rro_philox4x32(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]);

#ifdef __cplusplus
}
#endif
#endif
