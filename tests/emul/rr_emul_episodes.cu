// rr_emul_episodes.cu — HOST execution of rr_step_episodes' launch (k_step<L, OutT, true> and k_step<L, OutT, true, true>
// with their episode outputs): rr_emul.cu plus one export.
//
// TEST INFRASTRUCTURE ONLY, built into its own test library (tests/emul/emul_episodes.py).  launch_episodes_t is
// launch_pool_t of rr_emul_pool.cu (step_auto_reset without a pool) that also reads each row's episode result where
// k_step reads it: after step_accounting (StepOut::counted), before the auto-reset, goal words through goal_report.
#include "rr_emul.cu"

// One rr_step_episodes launch: launch_pool_t's outputs (slot all -1 without a pool: rows == NULL), plus ep_return
// [K][M][2], ep_length [K][M] and ep_goals [K][M][4] (may be NULL; goal scoring only).
template <int NH, int NG, int NP, int NN, bool G = false>
static int launch_episodes_t(const Consts &k, double *sf, int32_t *si, double *start, int64_t M, const double *actions,
                             int A, int K, double *rew, int32_t *done, int32_t *err, int32_t *naughty, double *obs_h,
                             double *obs_g, double *stats, double *final_h, double *final_g, int32_t *flags,
                             const ResetPool &pool, int32_t *slot, double *ep_return, int32_t *ep_length,
                             int32_t *ep_goals) {
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
      ep_return[2 * row] = o.counted ? e.ret_h : 0.0;
      ep_return[2 * row + 1] = o.counted ? e.ret_g : 0.0;
      ep_length[row] = o.counted ? e.step : -1;
      if (ep_goals) {
        int32_t *g = ep_goals + 4 * row;
        g[0] = g[1] = g[2] = g[3] = 0;
        if constexpr (E::kGoals) {
          if (o.counted) goal_report(e.alive(), e.scored(), E::B, g);
        }
      }
      naughty[row] = last_naughty;  // the row's own count (a pool reset then takes the loaded row's)
      if (pool.rows) {
        slot[row] = step_pool_auto_reset(e, k, done[row], (uint64_t)(k.env_offset + i), pool, start + i, M, last_naughty);
      } else {
        step_auto_reset(e, k, done[row], (uint64_t)(k.env_offset + i));
        slot[row] = -1;
      }
      rew[2 * row] = o.rew_h; rew[2 * row + 1] = o.rew_g;
      err[row] = (int32_t)o.step_err;
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

void emul_launch_episodes(const rr_config *cfg, double *sf, int32_t *si, double *start, int64_t M, const double *actions,
                          int n_actions, int K, double *rew, int32_t *done, int32_t *err, int32_t *naughty, double *obs_h,
                          double *obs_g, double *stats, double *final_h, double *final_g, int32_t *flags,
                          const uint64_t *rows, int64_t m, const double *cdf, double p, int32_t *slot, double *ep_return,
                          int32_t *ep_length, int32_t *ep_goals) {
  Consts k = make_consts(*cfg);
  k.n_actions = n_actions;
  const ResetPool pool{rows, cdf, m, p};
  EMUL_DISPATCH(cfg, launch_episodes_t, k, sf, si, start, M, actions, n_actions, K, rew, done, err, naughty, obs_h, obs_g,
                stats, final_h, final_g, flags, pool, slot, ep_return, ep_length, ep_goals);
}
}
