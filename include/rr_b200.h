/* rr_b200.h — C ABI of the B200-native batched RoboRugby simulator (librr_b200.so).
 *
 * Drop-in boundary for ONE path of harman097/RoboRugby: robo_rugby.gym_env step()/reset()
 * (SURVEY.md §8).  The reference has no FFI layer — its boundary is the gym 0.17 Env API of the
 * classes registered in robo_rugby/__init__.py:4-34 — so each entry point below names the Python
 * method it replaces.  roborugby_b200/ mirrors that Python surface on top of this ABI
 * (INTEGRATION.md shows the ctypes stub a reference maintainer would add).
 *
 * Conventions
 *   - plain C: opaque handle, raw pointers and sizes, no torch/C++ types;
 *   - every function returns 0 on success, a negative RR_E_* code otherwise; rr_last_error()
 *     returns a thread-local message;
 *   - "dev" pointers are CUDA device pointers on the handle's device, "host" pointers are
 *     ordinary (ideally pinned) host memory; `stream` is a cudaStream_t passed as void*
 *     (NULL = legacy default stream);
 *   - the handle owns the structure-of-arrays state in HBM; a handle is thread-compatible
 *     (external synchronisation per handle), there is no global state;
 *   - there is no CPU fallback: if no CUDA device is usable rr_create fails.
 *
 * Batch layouts (N = n_envs, R = robots, B = balls, D = obs_dim, K = k_steps)
 *   actions  discrete: uint8  [K][N][A]  A = n_actions <= R     (GameEnv_Simple.Direction ids 0..7)
 *            continuous: float [K][N][A]  A = n_actions <= 2R    (left,right thrust per robot)
 *   obs_h/g  out_t [K][N][D]     rew out_t [K][N][2] (happy, grumpy)     done uint8 [K][N]
 *   out_t = float (default, the dtype the reference declares for observation_space,
 *   RR_Observers.py:36-37) or double when cfg.out_f64 (the dtype its arrays actually hold).
 */
#ifndef RR_B200_H
#define RR_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RR_ABI_VERSION 2

/* presets == the two constant sets behind RR_Constants.py:4 (GAME_MODE) */
#define RR_PRESET_GAME 0  /* 800x800, 2+2 robots, 4+4 balls, 4500 steps */
#define RR_PRESET_TRAIN 1 /* 600x600, 1+0 robots, 1+0 balls, 300 steps  */

/* reward mixins, RR_ScoreKeepers.py */
#define RR_REW_CHASE 1u   /* ChasePosBall :46-66         */
#define RR_REW_PUSHPOS 2u /* PushPosBallsToGoal :138-157 */
#define RR_REW_NAUGHTY 4u /* NaughtyBots :112-135        */
#define RR_REW_DONTDRIVE 8u        /* DontDriveInGoals :69-83 (robot_in_goal RR_TrashyPhysics.py:12-15) */
#define RR_REW_KEEPMOVING 16u      /* KeepMovingGuys :86-98       */
#define RR_REW_BASEDESTRUCTION 32u /* BaseDestruction :101-111 (adds nothing: goals are never destroyed on the live path) */
#define RR_REW_PUSHNEG 64u         /* PushNegBallsFromGoal :160-179 */
/* ids for rr_config.reward_order: the sequence in which the on_step_end bodies run, one id per nibble, low nibble
 * first, 0 ends.  Each on_step_end calls super() before adding its own terms, so the bodies run in REVERSE MRO
 * order, and NaughtyBots.on_step_end does not call super(): mixins listed after it in the class never run.
 * reward_order == 0 selects Naughty, Chase, PushPos, PushNeg, BaseDestruction, DontDrive, KeepMoving (those in the
 * mask), which is the order of the registered ids (RR_Environments.py:11-37).
 * Valid pairs are exactly those a class `class Env(*mixins, Observer, GameEnv_Simple)` with distinct mixins produces:
 * reward_mask has no bits above RR_REW_PUSHNEG, and reward_order is 0 or all of
 *   - its nibbles are distinct ids 1..7, each with its bit in reward_mask, and no non-zero nibble follows the first 0;
 *   - if NAUGHTY is in the mask, the first (lowest) nibble is RR_MIX_NAUGHTY;
 *   - if NAUGHTY is not in the mask, the order lists exactly the mask's mixins.
 * rr_create and rr_check_config refuse any other pair with RR_E_INVALID (rr_sim.cuh rr_reward_config_error). */
#define RR_MIX_CHASE 1u
#define RR_MIX_PUSHPOS 2u
#define RR_MIX_NAUGHTY 3u
#define RR_MIX_DONTDRIVE 4u
#define RR_MIX_KEEPMOVING 5u
#define RR_MIX_BASEDESTRUCTION 6u
#define RR_MIX_PUSHNEG 7u

/* observers, RR_Observers.py */
#define RR_OBS_NONE 0
#define RR_OBS_BASIC_LIDAR 1 /* PosBall_BasicLidar :116-166 (5)        */
#define RR_OBS_LIDAR6_V2 2   /* SingleBall_6wayLidar_v2 :287-406 (11)  */
#define RR_OBS_ALLCOORDS 3   /* AllCoords :47-83 (3R+2B)               */
#define RR_OBS_ALLCOORDS_PRIOR 4 /* AllCoords_WithPrior :86-110 (6R+4B): + rectDblPriorStep of every robot and ball */
#define RR_OBS_LIDAR6_V1 5   /* SingleBall_6wayLidar :168-284 (11): the first 6-way lidar, which main.py:42-49 composes
                                "so Stephen can play" */

/* per-env error bits == the Python exceptions of the path (SURVEY.md §5) */
#define RR_ERR_STEP_AFTER_DONE 1u   /* RR_EnvBase.py:261-262 */
#define RR_ERR_TOO_MANY_COMMANDS 2u /* :270-271, :621-622    */
#define RR_ERR_BOT_COLLISIONS 4u    /* :312-313              */
#define RR_ERR_UNDO_FAILED 8u       /* :324-325              */
#define RR_ERR_ROBOTS_STUCK 16u     /* :327-330              */
#define RR_ERR_UNRESOLVED_FRAME 32u /* :417-421              */
#define RR_ERR_COINCIDENT_BALLS 64u /* RR_TrashyPhysics.py:249-250 */
#define RR_ERR_DIV0 128u            /* MyUtils.py:25         */
#define RR_ERR_RESET_PLACEMENT 256u /* placement loop exceeded its bound (reference: unbounded) */
#define RR_ERR_BAD_ACTION 512u      /* an action the env cannot apply, refused before anything moves: a discrete id > 7
                                       (KeyError in thrust_from_direction, RR_EnvBase.py:593-606, :624), or a thrust whose
                                       int(round(x)) is NaN or +-inf (round() raises, RR_Robot.py:100-102) or lies outside
                                       [-8, 7] (the reference would simulate it; the action space is Box(-1, 1)) */

/* return codes */
#define RR_OK 0
#define RR_E_INVALID (-1)
#define RR_E_CUDA (-2)
#define RR_E_NOMEM (-3)

/* statistics vector (doubles), see rr_get_stats */
#define RR_STAT_EPISODES 0
#define RR_STAT_RETURN_HAPPY 1
#define RR_STAT_RETURN_GRUMPY 2
#define RR_STAT_LENGTH 3
#define RR_STAT_NAUGHTY 4
#define RR_STAT_ERRORS 5
#define RR_STAT_STEPS 6
#define RR_STAT_REPLAYS 7 /* physics frames answered by the squeeze memo (rr_sim.cuh squeeze_contacts) */
#define RR_NUM_STATS 8

/* rr_config.flags */
#define RR_FLAG_NO_SQUEEZE_MEMO 1u /* always recompute a pinned ball's failed frame (A/B switch; results are identical) */

typedef struct rr_config {
  int32_t abi_version;  /* RR_ABI_VERSION */
  int32_t preset;       /* RR_PRESET_*  (entity counts are compile-time in the kernels) */
  uint32_t reward_mask; /* RR_REW_*     (class composition of RR_Environments.py:11-37) */
  int32_t observer;     /* RR_OBS_* */
  int32_t discrete;     /* 1: GameEnv_Simple.step :617-626, 0: GameEnv.step :260-297 */
  int32_t time_limit;   /* 1: done at step >= T (gym TimeLimit via robo_rugby/__init__.py), 0: raw step > T */
  int32_t auto_reset;   /* 1: an env that reports done (or raises) is reset inside the same launch */
  int32_t out_f64;      /* 0: float outputs, 1: double outputs */
  int32_t strict_reset; /* 1: reference placement test verbatim (may leave two balls exactly 14 px
                           apart, a state in which the reference itself never returns);
                           0: additionally reject such ball pairs */
  uint32_t reward_order; /* RR_MIX_* sequence (see above); 0 = canonical order of the mixins in reward_mask */
  uint64_t seed;        /* Philox key */
  int64_t env_offset;   /* global index of this handle's env 0 (rank * n_envs when sharded) */
  uint32_t flags;       /* RR_FLAG_* */
  int32_t goal_scoring; /* 0: the reference's HEAD, where goal scoring is dead code (scores 0, goals never destroyed,
                           balls never removed: SURVEY.md §0.4); 1: goal scoring as intended, i.e. RR_Goal.py:54-91 and
                           the commit block of GameEnv.__old_step (RR_EnvBase.py:461-511) made live: a ball that stays
                           150 steps inside a goal's triangle scores +-500 (added to the scorekeepers' step rewards), is
                           removed from play; three negative balls destroy a goal; done also when a goal is destroyed
                           or no ball is left (:555-559); BaseDestruction pays out */
} rr_config;

typedef struct rr_sim rr_sim;

/* Fill cfg for one of the registered ids (robo_rugby/__init__.py:4-34):
 * "RoboRugby-v0", "RoboRugbySimple-v0", "RoboRugbySimpleDuel-v2", "RoboRugbySimpleDuel-v3". */
int rr_default_config(rr_config *cfg, int preset, const char *env_id);

/* The checks rr_create makes on cfg, without a device: abi_version, preset, observer; discrete, time_limit, auto_reset,
 * out_f64, strict_reset and goal_scoring are 0 or 1; flags has no unknown bits; env_offset >= 0; (reward_mask,
 * reward_order) is a valid pair (see RR_MIX_*).  RR_E_INVALID with a message naming the field otherwise. */
int rr_check_config(const rr_config *cfg);

/* GameEnv.__init__ (RR_EnvBase.py:70-123) for n_envs episodes on CUDA device `device`.  cfg is checked
 * (rr_check_config) before any device is looked at. */
int rr_create(const rr_config *cfg, int64_t n_envs, int device, rr_sim **out);
int rr_destroy(rr_sim *s);
const char *rr_last_error(void);

int rr_num_envs(const rr_sim *s, int64_t *n);
int rr_num_robots(const rr_sim *s);
int rr_num_balls(const rr_sim *s);
int rr_obs_dim(const rr_sim *s);      /* observation_space.shape[0] */
int rr_max_steps(const rr_sim *s);    /* spec.max_episode_steps = GAME_LENGTH_STEPS */

/* GameEnv.reset(bln_randomize_pos=True) (RR_EnvBase.py:202-216) for the envs whose mask byte is
 * non-zero (mask_dev == NULL: all).  Random placement follows :155-200 with a counter-based
 * generator (Philox4x32-10, key = seed, counter = (global env index, episode, draw/4)). */
int rr_reset(rr_sim *s, const uint8_t *mask_dev, void *stream);

/* GameEnv.reset(bln_randomize_pos=False) (RR_EnvBase.py:202-216 -> _set_starting_positions :131-153; caller
 * main.py:107): back to the stored starting layout.  The layout is _lst_starting_positions: after rr_create it is the
 * env's own first random placement (:112-113); rr_set_starting_positions replaces it, e.g. with CONFIG_STANDARD
 * (:35-52).  HOST arrays rob3[N][R][3] = x, y, rot and ball2[N][B][2] = x, y; these two calls synchronise. */
/* as_constructed != 0 reproduces GameEnv(lst_starting_config) (:112-116): the sprites are first put back to their
 * freshly constructed state at the origin instead of running on_reset from the current pose. */
int rr_reset_fixed(rr_sim *s, const uint8_t *mask_dev, int32_t as_constructed, void *stream);
int rr_set_starting_positions(rr_sim *s, const double *rob3, const double *ball2);
int rr_get_starting_positions(rr_sim *s, double *rob3, double *ball2);

/* get_game_state(int_team=HAPPY / GRUMPY) of the current state (RR_Observers.py).  Buffers aligned to out_t. */
int rr_observe(rr_sim *s, void *obs_h_dev, void *obs_g_dev, void *stream);

/* get_game_state(obj_robot=lstRobots[robot], obj_ball=lstBalls[ball]) of the current state for every env
 * (RR_Observers.py:133-136 PosBall_BasicLidar, which ignores the ball; :187-203 SingleBall_6wayLidar; :304-320
 * SingleBall_6wayLidar_v2): obs_dev = out_t [N][D], from the robot's own team's point of view.  ball < 0 selects the
 * default lstPosBalls[0].  ball_dev (int32 [N], device, may be NULL) overrides `ball` with one index per env; a
 * negative entry yields a NaN row (a "Stephen" player without a ball).  RR_E_INVALID for the AllCoords observers
 * ("Robot-specific state output not supported.", :59-60). */
int rr_observe_entity(rr_sim *s, int32_t robot, int32_t ball, const int32_t *ball_dev, void *obs_dev, void *stream);

/* Stephen.__ponder (DQN_pytorch_player.py:39-61) for every env: the greedy nearest-ball assignment of the players that
 * drive robots_host[0..n_robots): balls inside either goal's triangle are ignored, each player gets at most one ball
 * and each ball one player, closest pairs first.  assign_dev = int32 [N][n_robots]: ball index or -1. */
int rr_assign_balls(rr_sim *s, const int32_t *robots_host, int32_t n_robots, int32_t *assign_dev, void *stream);

/* step() x k_steps in ONE fused kernel launch; device buffers (layouts above).  Any output
 * pointer may be NULL.  n_actions = values supplied per env per step (robots beyond it keep
 * their thrust, RR_EnvBase.py:272-273).  A discrete action id above 7 (KeyError in the reference, :603-606), or a
 * continuous thrust whose round-half-to-even value is not finite or lies outside [-8, 7], leaves the env untouched for
 * that step and raises RR_ERR_BAD_ACTION (done = 1; with auto_reset the env is reset).  A step on a finished env (step
 * counter above T, or with goal scoring a destroyed goal or no ball left) is refused with RR_ERR_STEP_AFTER_DONE
 * (done = 1) and changes nothing; continuous actions are not looked at then, as in the reference, while a discrete id
 * above 7 still raises RR_ERR_BAD_ACTION.  With auto_reset every row that reports done resets the env inside the
 * launch, a refused one included.  What each row adds to the statistics: rr_get_stats.
 * Alignment: every buffer to its element type (out_t results, float actions; RR_E_INVALID otherwise), nothing beyond
 * that.  Result rows are written as coalesced 128-bit stores when a buffer is 16-byte aligned and
 * its per-step row (N * D * sizeof(out_t), N * 2 * sizeof(out_t), N bytes) is a multiple of 16 bytes, element by
 * element otherwise; discrete actions with n_actions == 4 are read with one 32-bit load per env when the buffer is
 * 4-byte aligned, byte by byte otherwise. */
int rr_step(rr_sim *s, const void *actions_dev, int32_t n_actions, int32_t k_steps, void *obs_h_dev,
            void *obs_g_dev, void *rew_dev, uint8_t *done_dev, void *stream);

/* row_flags bits (rr_step_info) */
#define RR_ROW_TRUNCATED 1u /* gym 0.17's info['TimeLimit.truncated'] */
#define RR_ROW_RAISED 2u    /* the row's own error bits are non-zero (the reference raised) */

/* rr_step plus what a learner needs at every episode end, which auto_reset otherwise overwrites inside the launch
 * (rr_step is this call with three NULLs).  All three outputs are optional device buffers:
 *   final_obs_h / final_obs_g  out_t [K][N][D]: for every row with done = 1, get_game_state(int_team=HAPPY / GRUMPY) of
 *     the state the row's step ended in, before any auto-reset: what obs_h / obs_g would hold for that row with
 *     auto_reset = 0 (so with auto_reset = 0 the done rows equal the obs rows bit for bit).  A row that raised reports the
 *     state as the kernel left it (what rr_observe reports after it with auto_reset = 0).  Rows with done = 0 are NOT
 *     written: the caller's memory there is left as it was.  Ignored when D = 0 (RR_OBS_NONE).
 *   row_flags  uint8 [K][N], written for every row:
 *     RR_ROW_TRUNCATED  time_limit && step >= T && !game_is_done() on a row that did not raise: the episode was cut by
 *                       the TimeLimit wrapper (gym_env.py restates the rule for one env).  A goal destroyed at step T
 *                       is not truncated, neither is the raw row at T + 1 without auto_reset;
 *     RR_ROW_RAISED     the row's own error bits are non-zero (any RR_ERR_*, RR_ERR_BAD_ACTION and
 *                       RR_ERR_STEP_AFTER_DONE included): the reference's step() raised;
 *     other bits 0.  A done row with neither bit is a real end of the episode (terminated).
 * Everything else (obs, rew and done rows, the state, the error masks, the statistics) is what rr_step computes.  The
 * checks are rr_step's; final observation buffers must be aligned to out_t as well (RR_E_INVALID, nothing launched).
 * row_flags rows are written as 128-bit stores when the buffer is 16-byte aligned and N is a multiple of 16.  With a
 * sub-batch pipeline (rr_set_pipeline) these buffers follow the rule of the others: join before reading them.
 * rr_step_host and rr_step_host_begin do not report these outputs. */
int rr_step_info(rr_sim *s, const void *actions_dev, int32_t n_actions, int32_t k_steps, void *obs_h_dev,
                 void *obs_g_dev, void *rew_dev, uint8_t *done_dev, void *final_obs_h_dev, void *final_obs_g_dev,
                 uint8_t *row_flags_dev, void *stream);

/* Same call with HOST buffers: copies actions host->device, launches, and synchronises the stream before returning.
 * This is what a single-process caller of the reference's env.step() would bind.  When every result buffer is pinned
 * (page-locked, e.g. cudaHostAlloc / torch pin_memory) the kernel writes its rows straight into host memory (zero
 * copy: the device-to-host traffic overlaps the launch and nothing is staged in HBM).  Pageable buffers are staged in
 * HBM and copied; where those copies dominate (TRAIN preset) the k steps then run as up to four launches whose rows
 * travel while the next launch computes.  Results are identical on every path.  RR_HOST_ZEROCOPY=0 / RR_HOST_CHUNKS=n
 * in the environment at rr_create force the staged path / the number of launches. */
int rr_step_host(rr_sim *s, const void *actions_host, int32_t n_actions, int32_t k_steps,
                 void *obs_h_host, void *obs_g_host, void *rew_host, uint8_t *done_host, void *stream);

/* Sub-batch pipeline.  A launch is one wave of blocks and ends with its slowest env (a ball pinned between a robot and
 * a wall costs its block several normal frames per physics frame): at the BASELINE configuration the mean block is done
 * after 14 ms of a 17 ms launch.  rr_set_pipeline(s, n) splits the batch's blocks into n contiguous groups; every
 * rr_step then launches one kernel per group on the handle's own streams, so a group that is held back delays only its
 * OWN next launch while the SMs it leaves idle run the next launch of groups that have finished.  Results do not depend
 * on n (envs never interact; the statistics are accumulated atomically).
 * With n > 1 rr_step is asynchronous with respect to `stream`: the groups wait for the work `stream` holds at the
 * time of the call (the actions, earlier resets, ...), but `stream` does not wait for them.  rr_join(s, stream) makes
 * `stream` wait (on the device, without blocking the host) for everything issued so far; call it before reading
 * results or the state on `stream`.  Every other entry point that takes a stream joins by itself, and those that
 * synchronise the device cover the groups too, so only back-to-back rr_step calls overlap.  n = 1 (the default)
 * restores the single stream-ordered launch.  Replaces: nothing in the reference (one env per process); it is the
 * batched counterpart of running several reference envs in separate processes (Training_DQN_pytorch.py runs one). */
int rr_set_pipeline(rr_sim *s, int32_t sub_batches);
int rr_join(rr_sim *s, void *stream);

/* Benchmark hygiene (bench.py): a device buffer larger than the L2 that is overwritten in front of every rr_step launch,
 * on the stream that launches (with a sub-batch pipeline every group writes its share in front of its own launch), so
 * that no state or action line survives in the L2 from one launch to the next.  bytes = 0 switches it off (default). */
int rr_set_flush_buffer(rr_sim *s, void *buf_dev, int64_t bytes);

/* rr_step_host with up to RR_HOST_TICKETS calls in flight: _begin enqueues a call and returns a ticket (0 ..
 * RR_HOST_TICKETS - 1, handed out round robin) at once, _end blocks until that call's results are in host memory.
 * The result buffers must be pinned (page-locked and mapped); the kernels write into them directly.  The caller
 * rotates as many sets of result buffers as it keeps calls in flight and may begin calls n + 1, n + 2, ... before
 * ending call n (results complete in order); a _begin that finds its ticket still in use first waits for that call.  With a sub-batch pipeline the groups of
 * call n + 1 start while call n's slowest group still runs.  Action buffers are copied before _begin returns control
 * of them only in stream order: keep them unchanged until the call has ended. */
#define RR_HOST_TICKETS 4
int rr_step_host_begin(rr_sim *s, const void *actions_host, int32_t n_actions, int32_t k_steps, void *obs_h_host,
                       void *obs_g_host, void *rew_host, uint8_t *done_host, int32_t *ticket);
int rr_step_host_end(rr_sim *s, int32_t ticket);

/* Complete physics state, HOST buffers, array-of-structs layout used by the parity harness
 * (oracle/ref_harness.py): rob[N][R][7] = cx,cy,left,right,top,bottom,rot (FloatRect fields,
 * MyUtils.py:122-130); rhist[N][R][3] = pose in history slot count-1 (RR_Robot.py:43-58);
 * rflag[N][R][3] = thrust_l, thrust_r (each in [-8, 7]), hist_valid (0 or 1): rr_set_state returns RR_E_INVALID for
 * anything else and changes nothing; ball[N][B][8] = cx,cy,l,r,t,b,vx,vy;
 * step[N] = lngStepCount.  These synchronise the device.  rr_set_state also sets what is derived from the injected
 * pose: rectDblPriorStep of every robot and ball (observer RR_OBS_ALLCOORDS_PRIOR) becomes a copy() of the injected
 * rects, as the reference's on_reset / on_step_begin leave it; goal bookkeeping (goal_scoring) restarts as after a
 * reset.  rr_get_state does not return the prior-step poses (they are visible through rr_observe). */
int rr_set_state(rr_sim *s, const double *rob, const double *rhist, const int32_t *rflag,
                 const double *ball, const int32_t *step);
int rr_get_state(rr_sim *s, double *rob, double *rhist, int32_t *rflag, double *ball, int32_t *step);

/* Saved env states on the device: copy.deepcopy(env) of the reference, batched, without a host round trip (search and
 * lookahead from a common root, "reset to an archived state" curricula, checkpoints of envs mid-episode, replaying an env
 * that raised).  A saved env is one row of S = rr_snapshot_bytes_per_env(s) bytes (rr_sim.cuh RowLayout): every per-env
 * column of the state (robots with their thrusts, history-valid bits and episode-counted bit, balls, episode returns,
 * the AllCoords_WithPrior prior-step poses, step and episode counters, sticky error mask, last naughty count, goal
 * words), the starting layout, then zero padding to a multiple of 16 bytes, so two saves of one state are byte-equal.
 *   GAME  1104 (goal_scoring 1184, RR_OBS_ALLCOORDS_PRIOR 1328, both 1408)
 *   TRAIN  224 (goal_scoring  240, RR_OBS_ALLCOORDS_PRIOR  272, both  288)
 * The eight widths differ, so the width identifies the layout.  A row holds neither the statistics nor the pipeline and
 * flush settings nor anything of rr_config.
 * rr_save_states: for each j < m, row j of rows_dev (m rows of S bytes, 16-byte aligned) receives env env_dev[j]
 *   (env_dev NULL: env j, and m <= N); duplicates are allowed; an index outside [0, N) leaves its row unwritten.
 * rr_load_states: every env i with 0 <= slot_dev[i] < m receives row slot_dev[i]; a negative index (or one >= m) leaves
 *   env i untouched (slot_dev NULL: env i receives row i, and m == N).  A gather: no two rows can write one env.
 * Both are asynchronous and ordered on `stream` like rr_reset: they join the sub-batch pipeline into `stream` first (a
 * save after rr_step sees the stepped state, the next rr_step sees a load), and each adds one launch to rr_launch_count.
 * RR_E_INVALID, nothing launched: a NULL handle or rows pointer, m < 1, rows_dev not 16-byte aligned, an index pointer
 * not 8-byte aligned, or m against the rule of a NULL index pointer.
 * After a load every entry point reports for env i what it reported for the saved env at save time (rr_get_state,
 * rr_observe, rr_observe_entity, rr_assign_balls, rr_goal_state, rr_error_mask, rr_last_naughty,
 * rr_get_starting_positions), and stepping env i gives the saved env's rows bit for bit until a random reset, which
 * draws with the DESTINATION's global env index and the row's episode counter: a row loaded back into the env it came
 * from (same seed and env_offset) repeats even its resets, a clone in another env diverges from its first random reset
 * on.  A row can be loaded into any handle of the same width (another handle, another process through host memory) and
 * continues the same physical state under that handle's reward and observer configuration.  The statistics are not
 * touched; the episode-counted bit travels with the row, so an episode already counted is not counted again and an
 * uncounted one is counted each time a loaded copy of it finishes. */
int64_t rr_snapshot_bytes_per_env(const rr_sim *s);
int rr_save_states(rr_sim *s, const int64_t *env_dev, int64_t m, void *rows_dev, void *stream);
int rr_load_states(rr_sim *s, const void *rows_dev, int64_t m, const int64_t *slot_dev, void *stream);

/* Goal bookkeeping (goal_scoring = 1) to HOST; any pointer may be NULL.  alive[N]: bit b = ball b still in play;
 * score[N][2]: Goal.get_score() of the happy and the grumpy goal (RR_Goal.py:87-88); destroyed[N]: bit 0 happy goal,
 * bit 1 grumpy goal (Goal.is_destroyed, :90-91); dwell[N][2][B]: steps ball b has stayed inside that goal's triangle
 * (0 = not tracked).  Synchronises the device. */
int rr_goal_state(rr_sim *s, int32_t *alive_host, int32_t *score_host, int32_t *destroyed_host, int32_t *dwell_host);

/* Per-env sticky error mask (RR_ERR_*) to HOST; clear != 0 zeroes it afterwards. */
int rr_error_mask(rr_sim *s, uint32_t *err_host, int32_t clear);
/* Naughty-robot count of the last step per env (len(set_naughty_bots)), to HOST. */
int rr_last_naughty(rr_sim *s, int32_t *count_host);

/* Episode statistics accumulated on the device since the last rr_clear_stats: RR_NUM_STATS doubles
 * (finished episodes, sum of happy/grumpy returns, sum of lengths, naughty events, errors, steps, squeeze replays).
 * What one row (one env, one env-step) adds:
 *   steps     1, unless the row is an RR_ERR_STEP_AFTER_DONE refusal
 *   errors    1 if the row counts as a step and raised (any bit, RR_ERR_BAD_ACTION included)
 *   naughty   len(set_naughty_bots) of a completed row (what rr_last_naughty reports); 0 on a row that raised and
 *             without NaughtyBots
 *   episodes, returns, length
 *             at the FIRST row that reports done = 1 and is not a refusal since the env's last reset (rr_create,
 *             rr_reset, rr_reset_fixed, auto-reset) or rr_set_state: 1, the fp64 sum of the rows' rewards since then in
 *             step order (rows that raised add 0), the step counter.  Later done rows of the same episode (the raw
 *             row at T + 1 after the TimeLimit row at T, a bad action on a finished env) add nothing here.
 *   replays   physics frames of the launch answered by the squeeze memo (0 with RR_FLAG_NO_SQUEEZE_MEMO)
 * Each launch sums its rows per warp and adds them with one fp64 atomic per warp and statistic, so the returns of
 * a batch differ from a sequential sum in the last bits.  rr_stats_device_ptr exposes the device vector so a caller
 * can all-reduce it in place (NCCL). */
int rr_get_stats(rr_sim *s, double *stats_host);
int rr_stats_device_ptr(rr_sim *s, double **stats_dev);
int rr_clear_stats(rr_sim *s, void *stream);
/* Accumulate into a caller-owned device vector of RR_NUM_STATS doubles instead (e.g. a torch tensor
 * that torch.distributed all-reduces over NCCL); NULL restores the internal vector. */
int rr_set_stats_buffer(rr_sim *s, double *stats_dev);

/* Kernels launched by this handle so far (bench.py's gpu_launches). */
int64_t rr_launch_count(const rr_sim *s);
/* Bytes of persistent per-env state in HBM (S in DESIGN.md's roofline formula). */
int64_t rr_state_bytes_per_env(const rr_sim *s);

/* Device self-test of a numeric building block that replaces compiler or libm code on the GPU (no reference
 * counterpart: the reference uses CPython's float division and libm).  which 0: the branch-free fp64 division
 * of the contact paths (rr_sim.cuh div_core) against the compiler's division on >= n random operand pairs.
 * out2[0] = results that differ although the routine reported the operands in range (must be 0),
 * out2[1] = operand pairs it reported out of range (those are redone with the ordinary division). */
int rr_selftest(int device, int which, int64_t n, uint64_t seed, int64_t *out2);

#ifdef __cplusplus
}
#endif
#endif
