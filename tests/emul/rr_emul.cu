// rr_emul.cu — HOST execution of the device simulator source (roborugby_b200/csrc/rr_sim.cuh).
//
// TEST INFRASTRUCTURE ONLY.  The product library (librr_b200.so) contains GPU code alone; this
// file builds a separate, test-only library in which the same __host__ __device__ functions are
// compiled for the CPU, so that the CPU-only test tier (-m "not gpu") can check the restructured
// kernel logic against the oracle without a GPU.  Nothing under roborugby_b200/ loads it.
#include <cstring>

#include "../../roborugby_b200/csrc/rr_sim.cuh"

using namespace rr;

template <int NH, int NG, int NP, int NN, bool G = false>
struct HostEnv {
  using E = Env<NH, NG, NP, NN, G>;
  double buf[E::kDoubles];
  double cold[E::kColdDoubles];
  E e;
  HostEnv() { std::memset(buf, 0, sizeof buf); std::memset(cold, 0, sizeof cold); e.base = buf; e.cold = cold; e.stride = 1; e.trig = &kSinCosHost[0][0]; e.thrust = 0x88888888u; e.hvalid = 0; e.step = 0; e.err = 0; e.episode = 0; e.ret_h = e.ret_g = 0; e.sq_watch = 0; e.rr_stuck = 0; e.masks_dirty = true; e.br_near = e.bb_near = e.rr_near = e.wall_near = e.moving = 0; }
};

template <class E>
static void load(E &e, const Consts &k, const double *rob, const double *rhist, const int32_t *rflag,
                 const double *ball, int32_t step) {
  e.hvalid = 0;
  e.thrust = 0x88888888u;
  e.masks_dirty = true;
  e.br_near = e.bb_near = e.rr_near = e.wall_near = e.moving = 0;
  for (int r = 0; r < E::R; r++) {
    const double *p = rob + 7 * r;
    e.rcx(r) = p[0]; e.rcy(r) = p[1]; e.rl(r) = p[2]; e.rr(r) = p[3]; e.rt(r) = p[4]; e.rb(r) = p[5]; e.rrot(r) = p[6];
    e.hx(r) = rhist[3 * r]; e.hy(r) = rhist[3 * r + 1]; e.hrot(r) = rhist[3 * r + 2];
    e.set_thrust(r, rflag[3 * r], rflag[3 * r + 1]);
    if (rflag[3 * r + 2]) e.hvalid |= 1u << r;
    robot_refresh_corners(e, k, r);
  }
  for (int b = 0; b < E::B; b++) {
    const double *p = ball + 8 * b;
    e.bcx(b) = p[0]; e.bcy(b) = p[1]; e.bl(b) = p[2]; e.br(b) = p[3]; e.bt(b) = p[4]; e.bb(b) = p[5];
    e.bvx(b) = p[6]; e.bvy(b) = p[7];
  }
  e.step = step; e.err = 0; e.episode = 0; e.ret_h = e.ret_g = 0;
  e.invalidate_caches();
  e.memo_clear();
  e.goal_clear();
  e.sq_watch = 0; e.rr_stuck = 0;
}

template <class E>
static void store(const E &e, double *rob, double *rhist, int32_t *rflag, double *ball, int32_t *step) {
  for (int r = 0; r < E::R; r++) {
    double *p = rob + 7 * r;
    p[0] = e.rcx(r); p[1] = e.rcy(r); p[2] = e.rl(r); p[3] = e.rr(r); p[4] = e.rt(r); p[5] = e.rb(r); p[6] = e.rrot(r);
    int v = (e.hvalid >> r) & 1;
    rhist[3 * r] = v ? e.hx(r) : 0; rhist[3 * r + 1] = v ? e.hy(r) : 0; rhist[3 * r + 2] = v ? e.hrot(r) : 0;
    rflag[3 * r] = e.thl(r); rflag[3 * r + 1] = e.thr(r); rflag[3 * r + 2] = v;
  }
  for (int b = 0; b < E::B; b++) {
    double *p = ball + 8 * b;
    p[0] = e.bcx(b); p[1] = e.bcy(b); p[2] = e.bl(b); p[3] = e.br(b); p[4] = e.bt(b); p[5] = e.bb(b);
    p[6] = e.bvx(b); p[7] = e.bvy(b);
  }
  *step = e.step;
}

// k_step's action decoding for one env-step of `n` actions given as doubles: discrete ids (the ABI's uint8: 0..255) or
// thrusts (the ABI's float: rounded to float first).  false: the step is refused (RR_ERR_BAD_ACTION).
template <int R>
static bool decode_actions(const Consts &k, const double *a, int n, unsigned &cmd, int &n_cmd) {
  if (k.discrete) {
    uint32_t ids = 0;
    for (int r = 0; r < n && r < R; r++) ids |= ((uint32_t)a[r] & 0xffu) << (8 * r);
    n_cmd = n;
    return decode_discrete<R>(ids, n, cmd);
  }
  float f[2 * R];
  for (int q = 0; q < 2 * R; q++) f[q] = q < n ? (float)a[q] : 0.0f;
  n_cmd = n / 2;
  return decode_continuous<R>(f, n_cmd, cmd);
}

static double g_last_replays = 0.0;  // frames of the last emul_step answered by the squeeze memo
static double g_last_whole = 0.0;    // ... of which whole frames
static double g_last_stuck = 0.0;    // robot-robot phases answered by the stuck-pair memo

template <int NH, int NG, int NP, int NN, bool G = false>
static unsigned step_t(const Consts &k, double *rob, double *rhist, int32_t *rflag, double *ball, int32_t *step,
                       const double *actions, int n_actions, double *obs_h, double *obs_g, double *rew, int32_t *done,
                       int32_t *naughty) {
  HostEnv<NH, NG, NP, NN, G> h;
  auto &e = h.e;
  using E = typename HostEnv<NH, NG, NP, NN, G>::E;
  load(e, k, rob, rhist, rflag, ball, *step);
  unsigned cmd = 0;
  int n_cmd;
  const bool ok = decode_actions<E::R>(k, actions, n_actions, cmd, n_cmd);
  StepOut o;
  { FrameSync fs_; sim_step(e, k, cmd, n_cmd, o, ok, fs_); }
  if (!ok) o.step_err = RR_ERR_BAD_ACTION;
  g_last_replays = e.mm(kMReplays);
  g_last_whole = e.mm(kMFrames);
  g_last_stuck = e.mm(kMStuckReplays);
  unsigned oerr = 0;
  if (obs_h) observe(e, k, 1, obs_h, oerr);
  if (obs_g) observe(e, k, -1, obs_g, oerr);
  rew[0] = o.rew_h; rew[1] = o.rew_g;
  *done = o.done;
  *naughty = rr_popc(o.naughty);
  store(e, rob, rhist, rflag, ball, step);
  return o.step_err;
}

// K discrete env-steps in one call on ONE Env object: like a fused GPU launch, the per-thread memo state (squeeze
// memo, stuck-pair memo) lives across the steps.  Returns the OR of the steps' error bits; stops at the first error.
template <int NH, int NG, int NP, int NN, bool G = false>
static unsigned step_k_t(const Consts &k, double *rob, double *rhist, int32_t *rflag, double *ball, int32_t *step,
                         const double *actions, int n_actions, int K, double *rew_out, double *counters) {
  HostEnv<NH, NG, NP, NN, G> h;
  auto &e = h.e;
  using E = typename HostEnv<NH, NG, NP, NN, G>::E;
  load(e, k, rob, rhist, rflag, ball, *step);
  unsigned errs = 0;
  for (int s = 0; s < K; s++) {
    unsigned cmd = 0;
    int n_cmd;
    const bool ok = decode_actions<E::R>(k, actions + (size_t)s * n_actions, n_actions, cmd, n_cmd);
    StepOut o;
    { FrameSync fs_; sim_step(e, k, cmd, n_cmd, o, ok, fs_); }
    if (!ok) o.step_err = RR_ERR_BAD_ACTION;
    rew_out[2 * s] = o.rew_h; rew_out[2 * s + 1] = o.rew_g;
    errs |= o.step_err;
    if (o.step_err & ~RR_ERR_BAD_ACTION) break;  // a refused step leaves the env untouched: k_step goes on from it
  }
  counters[0] = e.mm(kMReplays); counters[1] = e.mm(kMFrames); counters[2] = e.mm(kMStuckReplays);
  store(e, rob, rhist, rflag, ball, step);
  return errs;
}

// step_k_t for both action kinds, with the goal bookkeeping (goal_scoring) recorded after every step:
// goal[s] = {alive mask, scored masks, done flag}; dwell_out = final dwell counters [2][B]
template <int NH, int NG, int NP, int NN, bool G = false>
static unsigned goal_rollout_t(const Consts &k, double *rob, double *rhist, int32_t *rflag, double *ball, int32_t *step,
                               const double *actions, const int32_t *n_act, int stride, int K, double *rew_out,
                               int32_t *goal, int32_t *dwell_out, int32_t *steps_done) {
  HostEnv<NH, NG, NP, NN, G> h;
  auto &e = h.e;
  using E = typename HostEnv<NH, NG, NP, NN, G>::E;
  load(e, k, rob, rhist, rflag, ball, *step);
  unsigned errs = 0;
  *steps_done = 0;
  for (int s = 0; s < K; s++) {
    unsigned cmd = 0;
    int n_cmd;
    const bool ok = decode_actions<E::R>(k, actions + (size_t)s * stride, n_act[s], cmd, n_cmd);
    StepOut o;
    { FrameSync fs_; sim_step(e, k, cmd, n_cmd, o, ok, fs_); }
    if (!ok) o.step_err = RR_ERR_BAD_ACTION;
    errs |= o.step_err;
    if (o.step_err) break;
    rew_out[2 * s] = o.rew_h; rew_out[2 * s + 1] = o.rew_g;
    goal[3 * s] = (int32_t)e.alive(); goal[3 * s + 1] = (int32_t)e.scored(); goal[3 * s + 2] = o.done;
    *steps_done = s + 1;
  }
  for (int q = 0; q < 2 * E::B; q++) dwell_out[q] = (int32_t)e.gs(2 + q);
  store(e, rob, rhist, rflag, ball, step);
  return errs;
}

template <int NH, int NG, int NP, int NN, bool G = false>
static unsigned reset_t(const Consts &k, double *rob, double *rhist, int32_t *rflag, double *ball, int32_t *step,
                        uint64_t env, uint32_t episode, int construct) {
  HostEnv<NH, NG, NP, NN, G> h;
  auto &e = h.e;
  if (construct) construct_env(e);
  else load(e, k, rob, rhist, rflag, ball, *step);
  e.episode = episode;
  e.err = 0;
  reset_env(e, k, env);
  store(e, rob, rhist, rflag, ball, step);
  return e.err;
}

// ---- k_step launches on the host ---------------------------------------------------------------------------------------
// The persistent state of M envs in the kernels' HBM layout (rr::Columns in rr_sim.cuh), moved in and out of an Env by
// the kernels' own load_columns / store_columns; emul_launch is one k_step launch over all M envs.
template <class E>
static void col_load(E &e, const Consts &k, const double *sf, const int32_t *si, int64_t N, int64_t i) {
  // a launch starts from nothing but the stored columns: every field load_columns does not set holds NaN here
  for (int q = 0; q < E::kDoubles; q++) e.base[q] = HUGE_VAL - HUGE_VAL;
  for (int q = 0; q < E::kColdDoubles; q++) e.cold[q] = HUGE_VAL - HUGE_VAL;
  load_columns(e, k, sf, si, N, i);
}

// One k_step launch: K steps of every env, actions [K][M][A] as doubles (see decode_actions).  Rows: rew [K][M][2],
// done / err (the row's error bits) / naughty [K][M]; obs_h, obs_g [K][M][D] or NULL.  stats [M][RR_NUM_STATS]: each env's
// contribution to the statistics vector before the warp reduction.
template <int NH, int NG, int NP, int NN, bool G = false>
static void launch_t(const Consts &k, double *sf, int32_t *si, int64_t M, const double *actions, int A, int K, double *rew,
                     int32_t *done, int32_t *err, int32_t *naughty, double *obs_h, double *obs_g, double *stats) {
  using E = typename HostEnv<NH, NG, NP, NN, G>::E;
  const int dim = obs_dim_of<E>(k.observer);
  for (int64_t i = 0; i < M; i++) {
    HostEnv<NH, NG, NP, NN, G> h;
    auto &e = h.e;
    col_load(e, k, sf, si, M, i);
    double st[RR_NUM_STATS] = {};
    int last_naughty = 0;
    for (int s = 0; s < K; s++) {
      const int64_t row = (int64_t)s * M + i;
      unsigned cmd = 0;
      int n_cmd = 0;
      bool bad_action = false;
      if (decode_before_refusal(e, k)) bad_action = !decode_actions<E::R>(k, actions + row * A, A, cmd, n_cmd);
      StepOut o;
      { FrameSync fs_; sim_step(e, k, cmd, n_cmd, o, !bad_action, fs_); }
      done[row] = step_bookkeeping(e, k, o, bad_action, st, last_naughty, (uint64_t)(k.env_offset + i));
      rew[2 * row] = o.rew_h; rew[2 * row + 1] = o.rew_g;
      err[row] = (int32_t)o.step_err;
      naughty[row] = last_naughty;
      unsigned oerr = 0;
      if (obs_h) observe(e, k, 1, obs_h + row * dim, oerr);
      if (obs_g) observe(e, k, -1, obs_g + row * dim, oerr);
    }
    st[RR_STAT_REPLAYS] = e.mm(kMReplays);
    store_columns(e, k, sf, si, M, i, last_naughty);
    for (int q = 0; q < RR_NUM_STATS; q++) stats[i * RR_NUM_STATS + q] = st[q];
  }
}

// k_init (rr_create) or k_reset (rr_reset) of the envs whose mask byte is non-zero (mask NULL: all)
template <int NH, int NG, int NP, int NN, bool G = false>
static void cols_reset_t(const Consts &k, double *sf, int32_t *si, int64_t M, const uint8_t *mask, int create) {
  for (int64_t i = 0; i < M; i++) {
    if (mask && !mask[i]) continue;
    HostEnv<NH, NG, NP, NN, G> h;
    auto &e = h.e;
    if (create) {
      construct_env(e);
    } else {
      col_load(e, k, sf, si, M, i);
      e.episode += 1;
    }
    reset_env(e, k, (uint64_t)(k.env_offset + i));
    store_columns(e, k, sf, si, M, i, 0);
  }
}

// the Env type of a configuration: GAME 2 + 2 robots, 4 + 4 balls; TRAIN 1 robot, 1 ball; goal scoring compiled in or not
#define EMUL_DISPATCH(cfg, F, ...)                                                      \
  ((cfg)->goal_scoring ? ((cfg)->preset == RR_PRESET_GAME ? F<2, 2, 4, 4, true>(__VA_ARGS__) \
                                                          : F<1, 0, 1, 0, true>(__VA_ARGS__)) \
                       : ((cfg)->preset == RR_PRESET_GAME ? F<2, 2, 4, 4>(__VA_ARGS__) : F<1, 0, 1, 0>(__VA_ARGS__)))

template <int NH, int NG, int NP, int NN, bool G = false>
static Columns columns_t() {
  return Env<NH, NG, NP, NN, G>::kCols;
}
template <int NH, int NG, int NP, int NN, bool G = false>
static int launch_dispatch_t(const Consts &k, double *sf, int32_t *si, int64_t M, const double *actions, int A, int K,
                             double *rew, int32_t *done, int32_t *err, int32_t *naughty, double *obs_h, double *obs_g,
                             double *stats) {
  launch_t<NH, NG, NP, NN, G>(k, sf, si, M, actions, A, K, rew, done, err, naughty, obs_h, obs_g, stats);
  return 0;
}
template <int NH, int NG, int NP, int NN, bool G = false>
static int reset_dispatch_t(const Consts &k, double *sf, int32_t *si, int64_t M, const uint8_t *mask, int create) {
  cols_reset_t<NH, NG, NP, NN, G>(k, sf, si, M, mask, create);
  return 0;
}

extern "C" {

// dims = {sf columns, si columns, si column of the episode, of the error mask, of the last naughty count}
void emul_cols_dims(const rr_config *cfg, int32_t *dims) {
  const Columns C = EMUL_DISPATCH(cfg, columns_t);
  const int32_t d[] = {C.nf(cfg->observer), C.ni(), C.episode(), C.err(), C.naughty()};
  std::memcpy(dims, d, sizeof d);
}

void emul_cols_set_state(const rr_config *cfg, double *sf, int32_t *si, int64_t M, int64_t i, const double *rob,
                         const double *rhist, const int32_t *rflag, const double *ball, int32_t step) {
  state_to_columns(EMUL_DISPATCH(cfg, columns_t), cfg->observer, sf, si, M, i, rob, rhist, rflag, ball, step);
}

void emul_cols_get_state(const rr_config *cfg, const double *sf, const int32_t *si, int64_t M, int64_t i, double *rob,
                         double *rhist, int32_t *rflag, double *ball, int32_t *step) {
  state_from_columns(EMUL_DISPATCH(cfg, columns_t), sf, si, M, i, rob, rhist, rflag, ball, step);
}

void emul_cols_reset(const rr_config *cfg, double *sf, int32_t *si, int64_t M, const uint8_t *mask, int create) {
  const Consts k = make_consts(*cfg);
  EMUL_DISPATCH(cfg, reset_dispatch_t, k, sf, si, M, mask, create);
}

void emul_launch(const rr_config *cfg, double *sf, int32_t *si, int64_t M, const double *actions, int n_actions, int K,
                 double *rew, int32_t *done, int32_t *err, int32_t *naughty, double *obs_h, double *obs_g, double *stats) {
  Consts k = make_consts(*cfg);
  k.n_actions = n_actions;
  EMUL_DISPATCH(cfg, launch_dispatch_t, k, sf, si, M, actions, n_actions, K, rew, done, err, naughty, obs_h, obs_g, stats);
}

// rr_reward_config_valid over n (mask, order) pairs: ok[i] = 1 for a pair rr_create accepts
void emul_reward_config_valid(const uint32_t *mask, const uint32_t *order, int64_t n, uint8_t *ok) {
  for (int64_t i = 0; i < n; i++) ok[i] = rr_reward_config_valid(mask[i], order[i]) ? 1 : 0;
}

double emul_last_replays(void) { return g_last_replays; }
double emul_last_whole_frames(void) { return g_last_whole; }
double emul_last_stuck_replays(void) { return g_last_stuck; }

unsigned emul_step(const rr_config *cfg, double *rob, double *rhist, int32_t *rflag, double *ball, int32_t *step,
                   const double *actions, int n_actions, double *obs_h, double *obs_g, double *rew, int32_t *done,
                   int32_t *naughty) {
  Consts k = make_consts(*cfg);
  k.n_actions = n_actions;
  if (cfg->goal_scoring) {
    if (cfg->preset == RR_PRESET_GAME)
      return step_t<2, 2, 4, 4, true>(k, rob, rhist, rflag, ball, step, actions, n_actions, obs_h, obs_g, rew, done, naughty);
    return step_t<1, 0, 1, 0, true>(k, rob, rhist, rflag, ball, step, actions, n_actions, obs_h, obs_g, rew, done, naughty);
  }
  if (cfg->preset == RR_PRESET_GAME)
    return step_t<2, 2, 4, 4>(k, rob, rhist, rflag, ball, step, actions, n_actions, obs_h, obs_g, rew, done, naughty);
  return step_t<1, 0, 1, 0>(k, rob, rhist, rflag, ball, step, actions, n_actions, obs_h, obs_g, rew, done, naughty);
}

unsigned emul_step_k(const rr_config *cfg, double *rob, double *rhist, int32_t *rflag, double *ball, int32_t *step,
                     const double *actions, int n_actions, int K, double *rew_out, double *counters) {
  Consts k = make_consts(*cfg);
  k.n_actions = n_actions;
  if (cfg->preset == RR_PRESET_GAME)
    return step_k_t<2, 2, 4, 4>(k, rob, rhist, rflag, ball, step, actions, n_actions, K, rew_out, counters);
  return step_k_t<1, 0, 1, 0>(k, rob, rhist, rflag, ball, step, actions, n_actions, K, rew_out, counters);
}

unsigned emul_goal_rollout(const rr_config *cfg, double *rob, double *rhist, int32_t *rflag, double *ball, int32_t *step,
                           const double *actions, const int32_t *n_act, int stride, int K, double *rew_out, int32_t *goal,
                           int32_t *dwell_out, int32_t *steps_done) {
  Consts k = make_consts(*cfg);
  if (cfg->preset == RR_PRESET_GAME)
    return goal_rollout_t<2, 2, 4, 4, true>(k, rob, rhist, rflag, ball, step, actions, n_act, stride, K, rew_out, goal, dwell_out, steps_done);
  return goal_rollout_t<1, 0, 1, 0, true>(k, rob, rhist, rflag, ball, step, actions, n_act, stride, K, rew_out, goal, dwell_out, steps_done);
}

unsigned emul_reset(const rr_config *cfg, double *rob, double *rhist, int32_t *rflag, double *ball, int32_t *step,
                    uint64_t env, uint32_t episode, int construct) {
  Consts k = make_consts(*cfg);
  if (cfg->preset == RR_PRESET_GAME) return reset_t<2, 2, 4, 4>(k, rob, rhist, rflag, ball, step, env, episode, construct);
  return reset_t<1, 0, 1, 0>(k, rob, rhist, rflag, ball, step, env, episode, construct);
}

unsigned emul_observe(const rr_config *cfg, double *rob, double *rhist, int32_t *rflag, double *ball, int32_t *step,
                      int team, double *obs) {
  Consts k = make_consts(*cfg);
  unsigned err = 0;
  if (cfg->preset == RR_PRESET_GAME) {
    HostEnv<2, 2, 4, 4> h; load(h.e, k, rob, rhist, rflag, ball, *step); observe(h.e, k, team, obs, err);
  } else {
    HostEnv<1, 0, 1, 0> h; load(h.e, k, rob, rhist, rflag, ball, *step); observe(h.e, k, team, obs, err);
  }
  return err;
}

// get_game_state(obj_robot=..., obj_ball=...) and the Stephen assignment through the device source
unsigned emul_observe_entity(const rr_config *cfg, double *rob, double *rhist, int32_t *rflag, double *ball, int32_t *step,
                             int robot, int ball_idx, double *obs) {
  Consts k = make_consts(*cfg);
  unsigned err = 0;
  if (cfg->preset == RR_PRESET_GAME) {
    HostEnv<2, 2, 4, 4> h; load(h.e, k, rob, rhist, rflag, ball, *step); observe_entity(h.e, k, robot, ball_idx, obs, err);
  } else {
    HostEnv<1, 0, 1, 0> h; load(h.e, k, rob, rhist, rflag, ball, *step); observe_entity(h.e, k, robot, ball_idx, obs, err);
  }
  return err;
}

void emul_assign_balls(const rr_config *cfg, double *rob, double *rhist, int32_t *rflag, double *ball, int32_t *step,
                       const int32_t *robots, int n, int32_t *assign) {
  Consts k = make_consts(*cfg);
  unsigned err = 0;
  int rb[8], out[8];
  for (int j = 0; j < n; j++) rb[j] = robots[j];
  if (cfg->preset == RR_PRESET_GAME) {
    HostEnv<2, 2, 4, 4> h; load(h.e, k, rob, rhist, rflag, ball, *step); assign_balls(h.e, k, rb, n, out, err);
  } else {
    HostEnv<1, 0, 1, 0> h; load(h.e, k, rob, rhist, rflag, ball, *step); assign_balls(h.e, k, rb, n, out, err);
  }
  for (int j = 0; j < n; j++) assign[j] = out[j];
}

// For every (robot, robot) and (ball, robot) pair of a GAME state: bit0 = the cheap rejection fired,
// bit1 = the reference predicate is True.  A pair with both bits set would be a parity bug.
void emul_predicates(const rr_config *cfg, double *rob, double *rhist, int32_t *rflag, double *ball, int32_t *step,
                     int32_t *rr_out /*[6]*/, int32_t *br_out /*[32]*/) {
  Consts k = make_consts(*cfg);
  HostEnv<2, 2, 4, 4> h;
  auto &e = h.e;
  load(e, k, rob, rhist, rflag, ball, *step);
  unsigned err = 0;
  int n = 0;
  for (int i = 0; i < 4; i++)
    for (int j = i + 1; j < 4; j++, n++)
      rr_out[n] = (robots_separated(e, i, j) ? 1 : 0) | (robots_collided(e, i, j, err) ? 2 : 0);
  for (int b = 0; b < 8; b++)
    for (int r = 0; r < 4; r++)
      br_out[b * 4 + r] = (ball_clear_of_robot(e, b, r) ? 1 : 0) | (ball_robot_collided(e, k, b, r, err) ? 2 : 0);
}

// n evaluations of the simulator's sin/cos routine (rr_sincos.cuh) on the host.  which 0: rr_sincos_grid (what
// the kernels call: grid fast path, rr_sincos_dd for everything else), 1: rr_sincos_dd alone.
void emul_sincos2(const double *x, int n, double *s, double *c, int which) {
  for (int i = 0; i < n; i++) {
    SinCos r = which ? rr_sincos_dd(x[i], &kSinCosHost[0][0]) : rr_sincos_grid(x[i], &kSinCosHost[0][0]);
    s[i] = r.s; c[i] = r.c;
  }
}
void emul_sincos(const double *x, int n, double *s, double *c) { emul_sincos2(x, n, s, c, 0); }

// 1: glibc sin/cos (what the oracle uses), 0: rr_sincos_dd (what the GPU uses)
void emul_use_libm_sincos(int on) { rr::g_host_libm_sincos = on; }

// reset(False) on one env: `start` = R x (x, y, rot) then B x (x, y), contiguous.
void emul_reset_fixed(const rr_config *cfg, double *rob, double *rhist, int32_t *rflag, double *ball, int32_t *step,
                      const double *start, int as_constructed) {
  Consts k = make_consts(*cfg);
  if (cfg->preset == RR_PRESET_GAME) {
    HostEnv<2, 2, 4, 4> h;
    if (as_constructed) construct_env(h.e); else load(h.e, k, rob, rhist, rflag, ball, *step);
    reset_env_fixed(h.e, k, start, 1);
    store(h.e, rob, rhist, rflag, ball, step);
  } else {
    HostEnv<1, 0, 1, 0> h;
    if (as_constructed) construct_env(h.e); else load(h.e, k, rob, rhist, rflag, ball, *step);
    reset_env_fixed(h.e, k, start, 1);
    store(h.e, rob, rhist, rflag, ball, step);
  }
}
}

