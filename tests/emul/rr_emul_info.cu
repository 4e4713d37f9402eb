// rr_emul_info.cu — HOST execution of rr_step_info's launch (k_step<L, OutT, true>): rr_emul.cu plus one export.
//
// TEST INFRASTRUCTURE ONLY, built into its own test library (tests/emul/emul_info.py).  launch_info_t is launch_t of
// rr_emul.cu with the end of each row taken apart as k_step takes it: step_accounting, step_row_flags and the terminal
// observation, then step_auto_reset (rr_sim.cuh).  launch_t itself calls step_bookkeeping, the composition of the two,
// so a CPU test that runs both over the same states checks that taking the row apart changes nothing else.
#include "rr_emul.cu"

// One rr_step_info launch: rr_emul.cu launch_t's outputs, plus final_h / final_g [K][M][D] (written on done rows only)
// and flags [K][M] (RR_ROW_*), each of which may be NULL.
template <int NH, int NG, int NP, int NN, bool G = false>
static int launch_info_t(const Consts &k, double *sf, int32_t *si, int64_t M, const double *actions, int A, int K,
                         double *rew, int32_t *done, int32_t *err, int32_t *naughty, double *obs_h, double *obs_g,
                         double *stats, double *final_h, double *final_g, int32_t *flags) {
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
      done[row] = step_accounting(e, k, o, bad_action, st, last_naughty);
      unsigned oerr = 0;
      if (flags) flags[row] = (int32_t)step_row_flags(e, k, o);
      if (done[row] && final_h) observe(e, k, 1, final_h + row * dim, oerr);
      if (done[row] && final_g) observe(e, k, -1, final_g + row * dim, oerr);
      step_auto_reset(e, k, done[row], (uint64_t)(k.env_offset + i));
      rew[2 * row] = o.rew_h; rew[2 * row + 1] = o.rew_g;
      err[row] = (int32_t)o.step_err;
      naughty[row] = last_naughty;
      if (obs_h) observe(e, k, 1, obs_h + row * dim, oerr);
      if (obs_g) observe(e, k, -1, obs_g + row * dim, oerr);
    }
    st[RR_STAT_REPLAYS] = e.mm(kMReplays);
    store_columns(e, k, sf, si, M, i, last_naughty);
    for (int q = 0; q < RR_NUM_STATS; q++) stats[i * RR_NUM_STATS + q] = st[q];
  }
  return 0;
}

extern "C" {

void emul_launch_info(const rr_config *cfg, double *sf, int32_t *si, int64_t M, const double *actions, int n_actions, int K,
                      double *rew, int32_t *done, int32_t *err, int32_t *naughty, double *obs_h, double *obs_g, double *stats,
                      double *final_h, double *final_g, int32_t *flags) {
  Consts k = make_consts(*cfg);
  k.n_actions = n_actions;
  EMUL_DISPATCH(cfg, launch_info_t, k, sf, si, M, actions, n_actions, K, rew, done, err, naughty, obs_h, obs_g, stats,
                final_h, final_g, flags);
}
}
