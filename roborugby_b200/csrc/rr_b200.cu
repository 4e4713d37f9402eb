// rr_b200.cu — kernels and C ABI (include/rr_b200.h) of the B200-native batched RoboRugby simulator.
//
// Build (see __graft_entry__.build()):
//   nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -lineinfo --fmad=false
//        -Xcompiler -fPIC -shared -o roborugby_b200/librr_b200.so roborugby_b200/csrc/rr_b200.cu
//
// HBM layout (DESIGN.md §3): structure of arrays sf (double) and si (int32), env index fastest; the columns are
// defined once, by rr::Columns in rr_sim.cuh.
// One thread owns one env for a whole launch: it loads its column of sf/si with coalesced 8-byte /
// 4-byte transactions, advances k_steps env-steps (12 physics frames each) out of registers / L1,
// streams actions in and observations, rewards and done flags out per step, and writes the column
// back once.  No inter-thread communication is needed except the warp-shuffle reduction of the
// episode statistics at the end of the launch.
#include <cmath>
#include <cstdio>
#include <cstdint>
#include <cstring>
#include <new>
#include <string>
#include <type_traits>
#include <vector>

#include "rr_sim.cuh"

namespace rr {

// Launch geometry.  One block is resident per SM: its warps are re-synchronised every physics frame so that they
// share instruction-cache lines.  A caller that steps one stream-ordered launch at a time gets the batch in one wave
// over all SMs; with the sub-batch pipeline (rr_set_pipeline) the blocks are launched in groups on the handle's own
// streams and their number is free (65 536 GAME envs = 171 blocks of 384 threads, which the SMs work off as they
// become free).  The hot per-env doubles (robot rects) live in shared memory, [field][thread] with the block size as
// stride: GAME 56 doubles x 384 threads = 168 KB; the cold ones (balls, history slots) in a per-thread local array.
template <int NH, int NG, int NP, int NN, bool GOALS = false, int MAXB = 0>
struct Launch {
  static constexpr int R = NH + NG, B = NP + NN;
  using E = Env<NH, NG, NP, NN, GOALS, MAXB>;
  // largest block: bounded by 227 KB of shared memory and by 65 536 registers per SM
  // The register file is per SM sub-partition (4 x 16 384 registers): 12 warps = 3 per sub-partition may use 168 registers
  // per thread, 13 - 16 warps only 128.  GAME: 384 threads x 168 registers beat 448 x 128 by 7.5 % once the sub-batch
  // pipeline (rr_set_pipeline) made the number of blocks a free parameter (171 blocks on 148 SMs no longer means two waves
  // of one launch); measured 416 / 384 / 352 / 320 threads: 139.8 / 151.7 / 142.9 / 135.5 M env-steps/s.
#ifndef RR_MAX_BLOCK_GAME
#define RR_MAX_BLOCK_GAME 384
#endif
#ifndef RR_MAX_BLOCK_TRAIN
#define RR_MAX_BLOCK_TRAIN 512
#endif
  // MAXB != 0: the wide k_step variant (GAME, 448 threads x 128 registers) for a caller that steps a batch of more than
  // 384 x #SM envs one stream-ordered launch at a time: one wave of 448-thread blocks then beats two waves of 384
  static constexpr int kMaxBlock = MAXB ? MAXB : (R > 1 ? RR_MAX_BLOCK_GAME : RR_MAX_BLOCK_TRAIN);
#ifndef RR_STEP_BLOCKS_PER_SM
#define RR_STEP_BLOCKS_PER_SM 1
#endif
  static constexpr int kStepBlocksPerSM = (R > 1 && MAXB == 0) ? RR_STEP_BLOCKS_PER_SM : 1;  // A/B switch (2 x 192 threads: measured slower)
  static constexpr int kTrigDoubles = kTrigRows * 4;  // sin/cos tables staged in front of the env fields
  // behind the env fields: one 640-byte staging area per warp, through which a warp's result rows (160 floats of
  // observations, 64 of rewards, 32 done bytes) are turned into full 128-bit stores (warp_store_rows)
  static constexpr int kStageBytes = 640;
  static constexpr size_t smem_bytes(int block) {
    return sizeof(double) * (kTrigDoubles + E::kDoubles * (size_t)block) + (size_t)kStageBytes * (block / 32);
  }
};

// Block size for n envs: spread over all SMs first (a multiple of one warp), then grow up to kMaxBlock.
static inline int pick_block(int64_t n, int sms, int max_block) {
  int64_t per_sm = (n + sms - 1) / sms;
  int64_t b = ((per_sm + 31) / 32) * 32;
  if (b < 32) b = 32;
  if (b > max_block) b = max_block;
  return (int)b;
}


// Stage the sin/cos table in shared memory (all threads of the block; followed by a barrier).
__device__ __forceinline__ const double *stage_trig_table() {
  const double *src = &kSinCosDev[0][0];
  for (int q = threadIdx.x; q < kTrigRows * 4; q += blockDim.x) rr_smem[q] = src[q];
  __syncthreads();
  return rr_smem;
}
__device__ __forceinline__ double *env_smem_base() { return rr_smem + kTrigRows * 4 + threadIdx.x; }
__device__ __forceinline__ int env_smem_offset() { return kTrigRows * 4 + (int)threadIdx.x; }

// Bind e's hot fields to this thread's column of the shared-memory area and its cold fields to `cold`.
template <class E>
__device__ __forceinline__ void bind_env(E &e, double *cold) {
  e.base = env_smem_base();
  e.boff = env_smem_offset();
  e.cold = cold;
  e.stride = (int)blockDim.x;
}

template <class L>
__device__ __forceinline__ void load_env(typename L::E &e, double *cold, const Consts &k, const double *__restrict__ sf,
                                         const int32_t *__restrict__ si, int64_t N, int64_t i) {
  bind_env(e, cold);
  load_columns(e, k, sf, si, N, i);
}

// Result rows of one warp: lane l holds `dim` values that belong at dst[l * dim .. l * dim + dim), so the warp's 32 rows
// are one contiguous range.  The values are converted, staged in the warp's shared-memory area and written as full
// 128-bit streaming stores (STG.E.128, evict-first: results are never read back by the kernel); a chunk of lanes at a
// time when 32 rows do not fit the area.  `vec` (warp-uniform) = all 32 lanes hold a row and the range is 16-byte
// aligned; otherwise every lane stores its own row element by element.
template <typename OutT, typename SrcT>
__device__ __forceinline__ void warp_store_rows(OutT *__restrict__ dst, const SrcT *vals, int dim, bool has_row, bool vec,
                                                void *stage_area, int lane) {
  constexpr int CAP = 640 / (int)sizeof(OutT), V = 16 / (int)sizeof(OutT);
  int lpc = dim > 0 ? CAP / dim : 0;
  if (lpc > 32) lpc = 32;
  while (lpc > 0 && lpc < 32 && ((lpc * dim) % V)) lpc--;  // every chunk starts on a 16-byte boundary
  if (!vec || lpc == 0) {
    if (has_row)
      for (int q = 0; q < dim; q++) __stcs(&dst[lane * dim + q], (OutT)vals[q]);
    return;
  }
  OutT *stage = (OutT *)stage_area;
#pragma unroll 1
  for (int l0 = 0; l0 < 32; l0 += lpc) {
    const int nl = (32 - l0) < lpc ? (32 - l0) : lpc, n = nl * dim;
    if (lane >= l0 && lane < l0 + nl)
      for (int q = 0; q < dim; q++) stage[(lane - l0) * dim + q] = (OutT)vals[q];
    __syncwarp();
    OutT *d = dst + l0 * dim;
    const int nv = n / V;
    for (int v = lane; v < nv; v += 32) __stcs((uint4 *)d + v, ((const uint4 *)stage)[v]);
    for (int t = nv * V + lane; t < n; t += 32) __stcs(&d[t], stage[t]);
    __syncwarp();
  }
}

struct StepArgs {
  double *sf;
  int32_t *si;
  double *stats;
  const void *actions;  // uint8 or float [K][N][A]
  void *obs_h, *obs_g, *rew;
  uint8_t *done;
  int64_t N;
  int K;
  unsigned vec;  // bit 0 observations, 1 rewards, 2 done, 4 row_flags: the buffer's rows can be written with 128-bit
                 // stores; bit 3: the action buffer is 4-byte aligned (one 32-bit load per env when A == 4)
  int block0;    // first block of this launch's env range (sub-batch launches, rr_set_pipeline); 0 for a whole batch
  void *final_obs_h, *final_obs_g;  // rr_step_info: out_t [K][N][D], written on done rows only (k_step<L, OutT, true>)
  uint8_t *row_flags;               // rr_step_info: RR_ROW_* [K][N]
};
// rr_step_episodes (k_step<L, OutT, true> and the pool variant): each row's episode result, or NULL.  A struct of its
// own, so that the default variants keep their parameter block.
struct InfoStepArgs : StepArgs {
  double *ep_return;   // [K][N][2]; vec bit 6: its rows can be written with 128-bit stores
  int32_t *ep_length;  // [K][N]; vec bit 7
  int32_t *ep_goals;   // [K][N][4] (goal scoring only); vec bit 8
};
// rr_step_pool (k_step<L, OutT, true, true>): the pool, the handle's start columns its resets write, and the slot rows.
// A struct of its own, so that the other variants keep their parameter block.
struct PoolStepArgs : InfoStepArgs {
  double *start;        // [3R + 2B][N]
  ResetPool pool;
  int32_t *reset_slot;  // [K][N] or NULL; vec bit 5: its rows can be written with 128-bit stores
};

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  return v;
}

// The fused multi-step kernel: K env-steps per launch, auto-reset inside.  Padding threads of the
// last block (i >= N) run the control flow without an env so that the per-frame barrier is uniform.
// INFO: also report every row's RR_ROW_* flags and, on done rows, the terminal observation taken before the auto-reset
// (rr_step_info), and each row's episode result taken at the same point (rr_step_episodes).  A template switch, not a
// run-time branch: the default kernels keep their registers and stack.
// POOL (with INFO): a done row's auto-reset may load a row of a reset pool instead (rr_step_pool, pool_reset).
template <class L, typename OutT, bool INFO = false, bool POOL = false>
__global__ void __launch_bounds__(L::kMaxBlock, L::kStepBlocksPerSM) k_step(const __grid_constant__ Consts k,
    const __grid_constant__ typename std::conditional<POOL, PoolStepArgs,
                                                      typename std::conditional<INFO, InfoStepArgs, StepArgs>::type>::type a) {
  static_assert(INFO || !POOL, "the pool variant reports rr_step_info's outputs as well");
  using E = typename L::E;
  constexpr int R = E::R;
  const int64_t i = ((int64_t)a.block0 + blockIdx.x) * blockDim.x + threadIdx.x;
  const bool live = i < a.N;
  double st[RR_NUM_STATS];
#pragma unroll
  for (int q = 0; q < RR_NUM_STATS; q++) st[q] = 0.0;
#ifdef RR_DEBUG_CLOCK
  const long long dbg_t0 = clock64();
#endif
  E e;
  double cold[E::kColdDoubles];
  frame_barrier_init();  // (ordered before the first frame by the barrier inside stage_trig_table)
  e.trig = stage_trig_table();
  FrameSync fs;
#ifdef RR_DEBUG_COUNT
  e.dbg[0] = e.dbg[1] = e.dbg[2] = e.dbg[3] = 0;
#endif
  if (live) {
    load_env<L>(e, cold, k, a.sf, a.si, a.N, i);
  } else {
    bind_env(e, cold);
    e.err = 0; e.step = 0; e.masks_dirty = false; e.sq_watch = 0; e.rr_stuck = 0;
  }
  const int dim = obs_dim_of<E>(k.observer);
  const int A = k.n_actions;
  int last_naughty = 0;
#pragma unroll 1
  for (int s = 0; s < a.K; s++) {
    const int64_t row = (int64_t)s * a.N + i;
    unsigned cmd = 0;
    int n_cmd = 0;
    bool bad_action = false;
    if (live) {
      if (k.discrete) {
        const uint8_t *ap = (const uint8_t *)a.actions + row * A;
        n_cmd = A;
        uint32_t w = 0;
        if (A == 4 && (a.vec & 8u)) {  // one coalesced 32-bit load per env (4-byte aligned buffer)
          w = __ldcs((const uint32_t *)ap);  // streamed once: keep the L2 for the per-thread local arrays
        } else {
#pragma unroll 1
          for (int r = 0; r < A; r++) w |= (uint32_t)ap[r] << (8 * r);
        }
        bad_action = !decode_discrete<R>(w, A, cmd);
      } else if (decode_before_refusal(e, k)) {
        n_cmd = A / 2;
        bad_action = !decode_continuous<R>((const float *)a.actions + row * A, n_cmd, cmd);
      }
    }
    StepOut o;
#ifdef RR_DEBUG_FRAMES
    fs.parity = (unsigned)s;  // (RR_DETACH is off in diagnostics builds: the field is free)
#endif
    sim_step(e, k, cmd, n_cmd, o, live && !bad_action, fs);  // (every thread calls it: block-wide barriers inside)
    int done_flag = 0;
    if (live) done_flag = step_accounting(e, k, o, bad_action, st, last_naughty);
    unsigned char row_flag = 0;
    if constexpr (INFO) {
      if (live) row_flag = (unsigned char)step_row_flags(e, k, o);
      // the terminal observation, before the auto-reset: done rows are rare (GAME 1 / 4500 env-steps), so each done lane
      // observes and stores its own row, without staging
      if (dim > 0 && (a.final_obs_h || a.final_obs_g)) {
        const int lane = threadIdx.x & 31;
        double ob[kMaxObs];
        unsigned oerr = 0;
#pragma unroll 1
        for (int team = 1; team >= -1; team -= 2) {
          OutT *dst = (OutT *)(team > 0 ? a.final_obs_h : a.final_obs_g);
          if (!dst) continue;
          if (live && done_flag) observe(e, k, team, ob, oerr);
          warp_store_rows<OutT>(dst + (row - lane) * dim, ob, dim, live && done_flag, false, nullptr, lane);
        }
      }
      // the episode's result on the row that counted it, before the auto-reset clears it: written on every row, so
      // staged like the results below
      if (a.ep_return || a.ep_length || a.ep_goals) {
        const int lane = threadIdx.x & 31;
        const bool full = __all_sync(0xffffffffu, live);
        const int64_t row0 = row - lane;
        void *stage = (char *)(rr_smem + L::kTrigDoubles + E::kDoubles * (size_t)blockDim.x) + L::kStageBytes * (threadIdx.x >> 5);
        const bool counted = live && o.counted;
        if (a.ep_return) {
          const double er[2] = {counted ? e.ret_h : 0.0, counted ? e.ret_g : 0.0};
          warp_store_rows<double>(a.ep_return + row0 * 2, er, 2, live, full && (a.vec & 64u), stage, lane);
        }
        if (a.ep_length) {
          const int32_t el[1] = {counted ? (int32_t)e.step : -1};
          warp_store_rows<int32_t>(a.ep_length + row0, el, 1, live, full && (a.vec & 128u), stage, lane);
        }
        if constexpr (E::kGoals) {
          if (a.ep_goals) {
            int32_t eg[4] = {0, 0, 0, 0};
            if (counted) goal_report(e.alive(), e.scored(), E::B, eg);
            warp_store_rows<int32_t>(a.ep_goals + row0 * 4, eg, 4, live, full && (a.vec & 256u), stage, lane);
          }
        }
      }
    }
    int32_t slot = -1;
    if constexpr (POOL) {
      if (live) slot = step_pool_auto_reset(e, k, done_flag, (uint64_t)(k.env_offset + i), a.pool, a.start + i, a.N, last_naughty);
    } else {
      if (live) step_auto_reset(e, k, done_flag, (uint64_t)(k.env_offset + i));
    }
    // Results: written once, never read back by this launch.  Every warp turns its 32 rows of each buffer into
    // coalesced 128-bit streaming stores (warp_store_rows); all lanes of the warp take part (no divergence here).
    {
      const int lane = threadIdx.x & 31;
      const bool full = __all_sync(0xffffffffu, live);  // padding lanes only exist in the batch's last warp
      const int64_t row0 = row - lane;                 // the warp's first row
      void *stage = (char *)(rr_smem + L::kTrigDoubles + E::kDoubles * (size_t)blockDim.x) + L::kStageBytes * (threadIdx.x >> 5);
      if (a.rew) {
        const double rw[2] = {o.rew_h, o.rew_g};
        warp_store_rows<OutT>((OutT *)a.rew + row0 * 2, rw, 2, live, full && (a.vec & 2u), stage, lane);
      }
      if (a.done) {
        const unsigned char dn[1] = {(unsigned char)done_flag};
        warp_store_rows<unsigned char>(a.done + row0, dn, 1, live, full && (a.vec & 4u), stage, lane);
      }
      if constexpr (INFO) {
        if (a.row_flags) {
          const unsigned char rf[1] = {row_flag};
          warp_store_rows<unsigned char>(a.row_flags + row0, rf, 1, live, full && (a.vec & 16u), stage, lane);
        }
      }
      if constexpr (POOL) {
        if (a.reset_slot) {
          const int32_t rs[1] = {slot};
          warp_store_rows<int32_t>(a.reset_slot + row0, rs, 1, live, full && (a.vec & 32u), stage, lane);
        }
      }
      if (dim > 0 && (a.obs_h || a.obs_g)) {
        double ob[kMaxObs];
        unsigned oerr = 0;
#pragma unroll 1
        for (int team = 1; team >= -1; team -= 2) {
          OutT *dst = (OutT *)(team > 0 ? a.obs_h : a.obs_g);
          if (!dst) continue;
          if (live) observe(e, k, team, ob, oerr);
          warp_store_rows<OutT>(dst + row0 * dim, ob, dim, live, full && (a.vec & 1u), stage, lane);
        }
      }
    }
  }
#ifdef RR_DEBUG_FRAMES
  __syncthreads();
  if (blockIdx.x == 0 && threadIdx.x == 0 && a.K >= 8) {
    const int nw = (int)(blockDim.x >> 5);
    for (int q = 0; q < a.K * 12 && q < 64 * 12; q++) {
      printf("FR %d", q);
      for (int w = 0; w < nw; w++) printf(" %lld:%x", rr_dbg_arrive[q * 16 + w] - rr_dbg_arrive[0], rr_dbg_paths[q * 16 + w]);
      printf("\n");
    }
  }
#endif
#ifdef RR_DEBUG_CLOCK
  last_naughty = (int)((clock64() - dbg_t0) >> 10);  // per-thread elapsed kilo-cycles (debug builds only)
#endif
#ifdef RR_DEBUG_COUNT
  last_naughty = (int)((min(e.dbg[0], 32767u) << 16) | min(e.dbg[2], 65535u));  // slow passes | precise ball-robot tests
#endif
#if defined(RR_DEBUG_COUNT) && defined(RR_DEBUG_CLOCK)
  // diagnostics build: elapsed cycles >> 12 | warp left the frame barrier | slow resolve passes of this env
  last_naughty = (int)(min((unsigned)((clock64() - dbg_t0) >> 12), 16383u) | (fs.detached ? 1u << 14 : 0u) |
                       (min(e.dbg[0], 65535u) << 15));
#endif
  if (live) {
    st[RR_STAT_REPLAYS] = e.mm(kMReplays);
    store_columns(e, k, a.sf, a.si, a.N, i, last_naughty);
  }
  // episode statistics: warp-shuffle reduction, one atomic per warp and statistic
#pragma unroll
  for (int q = 0; q < RR_NUM_STATS; q++) {
    double v = warp_sum(st[q]);
    if ((threadIdx.x & 31) == 0 && v != 0.0) atomicAdd(&a.stats[q], v);
  }
}

template <class L>
__global__ void __launch_bounds__(L::kMaxBlock, 1) k_init(const __grid_constant__ Consts k, double *sf, int32_t *si, int64_t N,
                                                    double *start) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const double *trig_tab = stage_trig_table();  // every thread of the block takes part (barrier inside)
  if (i >= N) return;
  typename L::E e;
  double cold[L::E::kColdDoubles];
  e.trig = trig_tab;
  bind_env(e, cold);
  construct_env(e);
  reset_env(e, k, (uint64_t)(k.env_offset + i));
  record_start(e, start + i, N);  // _lst_starting_positions = _set_random_positions() (RR_EnvBase.py:112-113)
  store_columns(e, k, sf, si, N, i, 0);
}

template <class L>
__global__ void __launch_bounds__(L::kMaxBlock, 1) k_reset_fixed(const __grid_constant__ Consts k, double *sf, int32_t *si,
                                                           int64_t N, const uint8_t *mask, const double *start,
                                                           int as_constructed) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const double *trig_tab = stage_trig_table();  // every thread of the block takes part (barrier inside)
  if (i >= N) return;
  if (mask && !mask[i]) return;
  typename L::E e;
  double cold[L::E::kColdDoubles];
  e.trig = trig_tab;
  load_env<L>(e, cold, k, sf, si, N, i);
  if (as_constructed) {  // GameEnv(lst_starting_config): sprites freshly constructed at the origin (:85-116)
    const unsigned ep = e.episode;
    construct_env(e);
    e.episode = ep;
  }
  e.episode += 1;
  reset_env_fixed(e, k, start + i, N);
  store_columns(e, k, sf, si, N, i, 0);
}

template <class L>
__global__ void __launch_bounds__(L::kMaxBlock, 1) k_reset(const __grid_constant__ Consts k, double *sf, int32_t *si, int64_t N,
                                                     const uint8_t *mask) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const double *trig_tab = stage_trig_table();  // every thread of the block takes part (barrier inside)
  if (i >= N) return;
  if (mask && !mask[i]) return;
  typename L::E e;
  double cold[L::E::kColdDoubles];
  e.trig = trig_tab;
  load_env<L>(e, cold, k, sf, si, N, i);
  e.episode += 1;
  reset_env(e, k, (uint64_t)(k.env_offset + i));
  store_columns(e, k, sf, si, N, i, 0);
}

template <class L, typename OutT>
__global__ void __launch_bounds__(L::kMaxBlock, 1) k_observe(const __grid_constant__ Consts k, const double *sf, const int32_t *si,
                                                       int64_t N, void *obs_h, void *obs_g) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const double *trig_tab = stage_trig_table();  // every thread of the block takes part (barrier inside)
  if (i >= N) return;
  typename L::E e;
  double cold[L::E::kColdDoubles];
  e.trig = trig_tab;
  load_env<L>(e, cold, k, sf, si, N, i);
  const int dim = obs_dim_of<typename L::E>(k.observer);
  double ob[kMaxObs];
  unsigned oerr = 0;
  if (obs_h) {
    observe(e, k, 1, ob, oerr);
    for (int q = 0; q < dim; q++) ((OutT *)obs_h)[i * dim + q] = (OutT)ob[q];
  }
  if (obs_g) {
    observe(e, k, -1, ob, oerr);
    for (int q = 0; q < dim; q++) ((OutT *)obs_g)[i * dim + q] = (OutT)ob[q];
  }
}

// get_game_state(obj_robot=..., obj_ball=...) for one robot index and a ball index that is the same for every env
// (ball_dev == nullptr) or differs per env (ball_dev[i]; a negative entry gives a NaN row: "no ball assigned")
template <class L, typename OutT>
__global__ void __launch_bounds__(L::kMaxBlock, 1) k_observe_entity(const __grid_constant__ Consts k, const double *sf,
                                                              const int32_t *si, int64_t N, int robot, int ball,
                                                              const int32_t *ball_dev, void *obs) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const double *trig_tab = stage_trig_table();
  if (i >= N) return;
  typename L::E e;
  double cold[L::E::kColdDoubles];
  e.trig = trig_tab;
  load_env<L>(e, cold, k, sf, si, N, i);
  const int dim = obs_dim_of<typename L::E>(k.observer);
  double ob[kMaxObs];
  unsigned oerr = 0;
  const int b = ball_dev ? ball_dev[i] : ball;
  if (ball_dev && b < 0) {
    for (int q = 0; q < dim; q++) ob[q] = rr_nan();
  } else {
    observe_entity(e, k, robot, b, ob, oerr);
  }
  for (int q = 0; q < dim; q++) ((OutT *)obs)[i * dim + q] = (OutT)ob[q];
}

struct RobotList { int n; int idx[8]; };

// Stephen.__ponder for every env: assign[i][j] = ball of the player driving robots.idx[j], or -1
template <class L>
__global__ void __launch_bounds__(L::kMaxBlock, 1) k_assign_balls(const __grid_constant__ Consts k, const double *sf,
                                                            const int32_t *si, int64_t N, const RobotList robots,
                                                            int32_t *assign) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const double *trig_tab = stage_trig_table();
  if (i >= N) return;
  typename L::E e;
  double cold[L::E::kColdDoubles];
  e.trig = trig_tab;
  load_env<L>(e, cold, k, sf, si, N, i);
  int rb[8], out[8];
  for (int j = 0; j < robots.n; j++) rb[j] = robots.idx[j];
  unsigned err = 0;
  assign_balls(e, k, rb, robots.n, out, err);
  for (int j = 0; j < robots.n; j++) assign[i * robots.n + j] = out[j];
}

// Saved env rows (rr_save_states / rr_load_states; the layout is RowLayout in rr_sim.cuh).  A block moves a tile of 32 rows
// through shared memory: the column side is accessed with lane = env, so that every load or store instruction touches one
// column of 32 envs (coalesced when the envs are consecutive), and the row side with 128-bit accesses.  In shared memory a
// row takes an odd number of 16-byte chunks, so that the 128-bit accesses of 32 lanes to chunk q of 32 rows hit distinct
// banks.  Pure data movement: one kernel per direction serves every preset and observer.
constexpr int kRowTile = 32, kRowThreads = 256, kRowWarps = kRowThreads / 32;
RR_HD constexpr int row_tile_chunks(const RowLayout &L) { return (L.bytes() / 16) | 1; }
constexpr size_t row_tile_bytes(const RowLayout &L) { return (size_t)kRowTile * row_tile_chunks(L) * 16; }
constexpr int kRowBatch = 4;  // chunks a lane has in flight in the column-side loop

__global__ void __launch_bounds__(kRowThreads) k_save_rows(const RowLayout L, const uint64_t *__restrict__ sf,
                                                           const uint64_t *__restrict__ start,
                                                           const uint32_t *__restrict__ si, int64_t N,
                                                           const int64_t *__restrict__ env, int64_t m,
                                                           uint4 *__restrict__ rows) {
  extern __shared__ uint4 tile[];
  __shared__ int64_t src[kRowTile];
  const int Q = L.bytes() / 16, QS = row_tile_chunks(L);
  const int64_t j0 = (int64_t)blockIdx.x * kRowTile;
  const int nrows = m - j0 < kRowTile ? (int)(m - j0) : kRowTile;
  if (threadIdx.x < kRowTile) src[threadIdx.x] = (int)threadIdx.x < nrows ? save_source(env, j0 + threadIdx.x, N) : -1;
  __syncthreads();
  // gather: lane = row of the tile, warp w takes chunks w, w + 8, ...
  const int j = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int64_t e = src[j];
  if (e >= 0) {
#pragma unroll 1
    for (int q0 = w; q0 < Q; q0 += kRowWarps * kRowBatch) {
      uint64_t v[2 * kRowBatch];
#pragma unroll
      for (int t = 0; t < kRowBatch; t++) {
        const int q = q0 + t * kRowWarps;
        if (q < Q) { v[2 * t] = row_unit_get(L, sf, start, si, N, e, 2 * q); v[2 * t + 1] = row_unit_get(L, sf, start, si, N, e, 2 * q + 1); }
      }
#pragma unroll
      for (int t = 0; t < kRowBatch; t++) {
        const int q = q0 + t * kRowWarps;
        if (q < Q)
          tile[j * QS + q] = make_uint4((unsigned)v[2 * t], (unsigned)(v[2 * t] >> 32), (unsigned)v[2 * t + 1],
                                        (unsigned)(v[2 * t + 1] >> 32));
      }
    }
  }
  __syncthreads();
  // the tile's rows are one contiguous range of the output: 128-bit stores (rows of skipped indices are not written)
  uint4 *dst = rows + j0 * Q;
#pragma unroll 4
  for (int c = threadIdx.x; c < nrows * Q; c += kRowThreads) {
    const int jj = c / Q;
    if (src[jj] >= 0) dst[c] = tile[jj * QS + (c - jj * Q)];
  }
}

__global__ void __launch_bounds__(kRowThreads) k_load_rows(const RowLayout L, const uint4 *__restrict__ rows, int64_t m,
                                                           const int64_t *__restrict__ slot, int64_t N,
                                                           uint64_t *__restrict__ sf, uint64_t *__restrict__ start,
                                                           uint32_t *__restrict__ si) {
  extern __shared__ uint4 tile[];
  __shared__ int64_t src[kRowTile];
  const int Q = L.bytes() / 16, QS = row_tile_chunks(L);
  const int64_t i0 = (int64_t)blockIdx.x * kRowTile;
  const int nenv = N - i0 < kRowTile ? (int)(N - i0) : kRowTile;
  if (threadIdx.x < kRowTile) src[threadIdx.x] = (int)threadIdx.x < nenv ? load_source(slot, i0 + threadIdx.x, m) : -1;
  __syncthreads();
  // each env's row with 128-bit loads (a row is contiguous; consecutive rows too when the slots are)
#pragma unroll 4
  for (int c = threadIdx.x; c < nenv * Q; c += kRowThreads) {
    const int jj = c / Q;
    const int64_t r = src[jj];
    if (r >= 0) tile[jj * QS + (c - jj * Q)] = rows[r * Q + (c - jj * Q)];
  }
  __syncthreads();
  // scatter: lane = env of the tile, warp w takes chunks w, w + 8, ...; a masked lane stores nothing
  const int j = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (src[j] < 0) return;
  const int64_t i = i0 + j;
#pragma unroll 2
  for (int q = w; q < Q; q += kRowWarps) {
    const uint4 c = tile[j * QS + q];
    row_unit_put(L, sf, start, si, N, i, 2 * q, (uint64_t)c.x | ((uint64_t)c.y << 32));
    row_unit_put(L, sf, start, si, N, i, 2 * q + 1, (uint64_t)c.z | ((uint64_t)c.w << 32));
  }
}

}  // namespace rr

// =============================================================================================
// C ABI

using namespace rr;

struct rr_sim {
  rr_config cfg;
  Consts k;
  int64_t N;
  int device;
  int sms = 148;
  Columns cols;                 // the layout of sf / si (rr_sim.cuh)
  double *sf = nullptr;
  int32_t *si = nullptr;
  double *start = nullptr;      // [3R + 2B][N] starting layout (_lst_starting_positions)
  double *stats = nullptr;      // where kernels accumulate (own_stats or a caller buffer)
  double *own_stats = nullptr;
  // staging for rr_step_host
  void *d_act = nullptr, *d_obs_h = nullptr, *d_obs_g = nullptr, *d_rew = nullptr;
  uint8_t *d_done = nullptr;
  size_t cap_act = 0, cap_obs_h = 0, cap_obs_g = 0, cap_rew = 0, cap_done = 0;
  cudaStream_t copy_stream = nullptr;  // rr_step_host: results of one chunk of steps travel while the next chunk runs
  cudaEvent_t chunk_done[4] = {nullptr, nullptr, nullptr, nullptr};
  int64_t launches = 0;
  // sub-batch pipeline (rr_set_pipeline): the batch's blocks in `pipe` contiguous groups, each stepped by its own kernel
  // on its own stream, so that a group whose slowest env holds it back delays only its own next launch
  int pipe = 1;
  std::vector<cudaStream_t> sub;
  std::vector<cudaEvent_t> sub_done;    // recorded behind a group's latest kernel
  cudaEvent_t pipe_entry = nullptr;     // recorded on the caller's stream at every rr_step: what the groups wait for
  bool pipe_pending = false;            // sub-stream work that the caller's stream has not been joined with yet
  void *flush_buf = nullptr;            // rr_set_flush_buffer: written before every k_step launch (benchmark hygiene)
  size_t flush_bytes = 0;
  // rr_step_host_begin / _end: up to RR_HOST_TICKETS calls in flight, each with its own action staging and completion event
  void *d_act2[RR_HOST_TICKETS] = {};
  size_t cap_act2[RR_HOST_TICKETS] = {};
  cudaEvent_t ticket_done[RR_HOST_TICKETS] = {};
  cudaStream_t ticket_stream[2] = {nullptr, nullptr};  // submission, collection
  int next_ticket = 0;
  int host_chunks = 0;        // RR_HOST_CHUNKS at rr_create (0 = per-preset default)
  bool host_zero_copy = true; // RR_HOST_ZEROCOPY=0 at rr_create forces the staged path
};

static void pipeline_free(rr_sim *s);

// Entry points run on the handle's device and leave the caller's current device as they found it.
struct DeviceGuard {
  int prev = -1;
  bool good = false;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
    good = (prev == dev) || cudaSetDevice(dev) == cudaSuccess;
    if (prev == dev) prev = -1;  // nothing to restore
  }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
  bool ok() const { return good; }
};
#define ON_DEVICE(dev)         \
  DeviceGuard _guard(dev);     \
  if (!_guard.ok()) return fail(RR_E_CUDA, "cudaSetDevice failed")

static thread_local std::string g_err;
const char *rr_last_error(void) { return g_err.c_str(); }

static int fail(int code, const std::string &msg) {
  g_err = msg;
  return code;
}
#define CK(call)                                                                               \
  do {                                                                                         \
    cudaError_t _e = (call);                                                                   \
    if (_e != cudaSuccess)                                                                     \
      return fail(RR_E_CUDA, std::string(#call) + ": " + cudaGetErrorString(_e));              \
  } while (0)

int rr_default_config(rr_config *c, int preset, const char *env_id) {
  if (!c || !env_id) return fail(RR_E_INVALID, "null argument");
  std::memset(c, 0, sizeof *c);
  c->abi_version = RR_ABI_VERSION;
  c->preset = preset;
  c->discrete = 1;
  std::string id(env_id);
  if (id == "RoboRugby-v0") {  // robo_rugby/__init__.py:4-10 -> GameEnv: no reward mixin, no observer
    c->discrete = 0; c->reward_mask = 0; c->observer = RR_OBS_NONE;
  } else if (id == "RoboRugbySimple-v0") {  // :12-18 -> SimpleChasePos (RR_Environments.py:11)
    c->reward_mask = RR_REW_CHASE; c->observer = RR_OBS_BASIC_LIDAR;
  } else if (id == "RoboRugbySimpleDuel-v2") {  // :20-26 -> SimpleDuel2 (RR_Environments.py:19-25)
    c->reward_mask = RR_REW_CHASE | RR_REW_PUSHPOS | RR_REW_NAUGHTY; c->observer = RR_OBS_BASIC_LIDAR;
  } else if (id == "RoboRugbySimpleDuel-v3") {  // :28-34 -> SimpleDuel3 (RR_Environments.py:27-37)
    c->reward_mask = RR_REW_CHASE | RR_REW_PUSHPOS | RR_REW_NAUGHTY; c->observer = RR_OBS_LIDAR6_V2;
  } else {
    return fail(RR_E_INVALID, "unknown env id " + id);
  }
  c->auto_reset = 1;
  c->time_limit = 1;
  c->strict_reset = 1;  // the reference's own placement rules
  return RR_OK;
}

using LGame = Launch<2, 2, 4, 4>;
using LTrain = Launch<1, 0, 1, 0>;
using LGameGoals = Launch<2, 2, 4, 4, true>;   // rr_config.goal_scoring = 1
using LTrainGoals = Launch<1, 0, 1, 0, true>;
using LGameWide = Launch<2, 2, 4, 4, false, 448>;   // k_step only (see Launch::kMaxBlock)
using LGameGoalsWide = Launch<2, 2, 4, 4, true, 448>;

// Every kernel uses more than the default 48 KB of dynamic shared memory: opt in once per device (rr_create), not per
// launch (the attribute call costs more than a K = 1 launch's own CPU time).
template <class L>
static cudaError_t opt_in_shared_memory() {
  const int bytes = (int)L::smem_bytes(L::kMaxBlock);
  cudaError_t e = cudaSuccess;
  auto set = [&](auto kern) {
    cudaError_t r = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e == cudaSuccess) e = r;
  };
  set(k_step<L, float>); set(k_step<L, double>); set(k_step<L, float, true>); set(k_step<L, double, true>);
  set(k_step<L, float, true, true>); set(k_step<L, double, true, true>);
  set(k_init<L>); set(k_reset<L>); set(k_reset_fixed<L>);
  set(k_observe<L, float>); set(k_observe<L, double>);
  set(k_observe_entity<L, float>); set(k_observe_entity<L, double>); set(k_assign_balls<L>);
  return e;
}

// Launch KERNEL<L, ...> for the handle's preset with the block size picked for its batch.
#define LAUNCH_ONE(LTYPE, s, st, KERNEL, ...)                                                               \
  do {                                                                                                      \
    using L = LTYPE;                                                                                        \
    auto kern = KERNEL;                                                                                     \
    const int blk = pick_block((s)->N, (s)->sms, L::kMaxBlock);                                             \
    kern<<<(unsigned)(((s)->N + blk - 1) / blk), blk, L::smem_bytes(blk), st>>>(__VA_ARGS__);               \
  } while (0)
#define LAUNCH_PRESET(s, st, KERNEL, ...)                                                                   \
  do {                                                                                                      \
    const bool game_ = (s)->cfg.preset == RR_PRESET_GAME, goals_ = (s)->cfg.goal_scoring != 0;              \
    if (game_ && !goals_) LAUNCH_ONE(LGame, s, st, KERNEL, __VA_ARGS__);                                    \
    else if (!game_ && !goals_) LAUNCH_ONE(LTrain, s, st, KERNEL, __VA_ARGS__);                             \
    else if (game_) LAUNCH_ONE(LGameGoals, s, st, KERNEL, __VA_ARGS__);                                     \
    else LAUNCH_ONE(LTrainGoals, s, st, KERNEL, __VA_ARGS__);                                               \
  } while (0)

int rr_check_config(const rr_config *cfg) {
  if (!cfg) return fail(RR_E_INVALID, "null argument");
  if (cfg->abi_version != RR_ABI_VERSION) return fail(RR_E_INVALID, "abi_version mismatch");
  if (cfg->preset != RR_PRESET_GAME && cfg->preset != RR_PRESET_TRAIN) return fail(RR_E_INVALID, "unknown preset");
  if (cfg->observer < 0 || cfg->observer > RR_OBS_LIDAR6_V1) return fail(RR_E_INVALID, "unknown observer");
  const struct { const char *name; int32_t v; } bools[] = {
      {"discrete", cfg->discrete},     {"time_limit", cfg->time_limit},     {"auto_reset", cfg->auto_reset},
      {"out_f64", cfg->out_f64},       {"strict_reset", cfg->strict_reset}, {"goal_scoring", cfg->goal_scoring}};
  for (const auto &b : bools)
    if (b.v != 0 && b.v != 1) return fail(RR_E_INVALID, std::string(b.name) + " must be 0 or 1, got " + std::to_string(b.v));
  if (cfg->flags & ~RR_FLAG_NO_SQUEEZE_MEMO)
    return fail(RR_E_INVALID, "flags has unknown bits " + std::to_string(cfg->flags & ~RR_FLAG_NO_SQUEEZE_MEMO));
  if (cfg->env_offset < 0) return fail(RR_E_INVALID, "env_offset must be >= 0");
  if (const char *why = rr_reward_config_error(cfg->reward_mask, cfg->reward_order)) {
    char hex[48];
    snprintf(hex, sizeof hex, " (reward_mask 0x%x, reward_order 0x%x)", cfg->reward_mask, cfg->reward_order);
    return fail(RR_E_INVALID, std::string(why) + hex);
  }
  return RR_OK;
}

int rr_create(const rr_config *cfg, int64_t n_envs, int device, rr_sim **out) {
  if (!cfg || !out || n_envs <= 0) return fail(RR_E_INVALID, "bad arguments");
  if (const int rc = rr_check_config(cfg)) return rc;
  int ndev = 0;
  cudaError_t ce = cudaGetDeviceCount(&ndev);
  if (ce != cudaSuccess || ndev == 0)
    return fail(RR_E_CUDA, std::string("no usable CUDA device (there is no CPU fallback): ") + cudaGetErrorString(ce));
  if (device < 0 || device >= ndev) return fail(RR_E_INVALID, "device index out of range");
  ON_DEVICE(device);
  rr_sim *s = new (std::nothrow) rr_sim();
  if (!s) return fail(RR_E_NOMEM, "host allocation failed");
  s->cfg = *cfg;
  s->k = make_consts(*cfg);
  s->N = n_envs;
  s->device = device;
  if (const char *ev = getenv("RR_HOST_CHUNKS")) s->host_chunks = atoi(ev);
  if (const char *ev = getenv("RR_HOST_ZEROCOPY")) s->host_zero_copy = atoi(ev) != 0;
  cudaDeviceGetAttribute(&s->sms, cudaDevAttrMultiProcessorCount, device);
  if (s->sms <= 0) s->sms = 148;
  const bool game = cfg->preset == RR_PRESET_GAME;
  s->cols = cfg->goal_scoring ? (game ? LGameGoals::E::kCols : LTrainGoals::E::kCols)
                              : (game ? LGame::E::kCols : LTrain::E::kCols);
  if (cudaMalloc(&s->start, sizeof(double) * (3 * s->cols.R + 2 * s->cols.B) * n_envs) != cudaSuccess ||
      cudaMalloc(&s->sf, sizeof(double) * s->cols.nf(cfg->observer) * n_envs) != cudaSuccess ||
      cudaMalloc(&s->si, sizeof(int32_t) * s->cols.ni() * n_envs) != cudaSuccess ||
      cudaMalloc(&s->own_stats, sizeof(double) * RR_NUM_STATS) != cudaSuccess) {
    cudaGetLastError();
    rr_destroy(s);
    return fail(RR_E_NOMEM, "device allocation failed");
  }
  s->stats = s->own_stats;
  if (game) {  // the wide k_step variants
    const int wb = (int)LGameWide::smem_bytes(LGameWide::kMaxBlock);
    cudaError_t we = cudaSuccess;
    auto set = [&](auto kern) {
      cudaError_t r = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, wb);
      if (we == cudaSuccess) we = r;
    };
    if (cfg->goal_scoring) {
      set(k_step<LGameGoalsWide, float>); set(k_step<LGameGoalsWide, double>);
      set(k_step<LGameGoalsWide, float, true>); set(k_step<LGameGoalsWide, double, true>);
      set(k_step<LGameGoalsWide, float, true, true>); set(k_step<LGameGoalsWide, double, true, true>);
    } else {
      set(k_step<LGameWide, float>); set(k_step<LGameWide, double>);
      set(k_step<LGameWide, float, true>); set(k_step<LGameWide, double, true>);
      set(k_step<LGameWide, float, true, true>); set(k_step<LGameWide, double, true, true>);
    }
    if (we != cudaSuccess) { rr_destroy(s); return fail(RR_E_CUDA, std::string("cudaFuncSetAttribute: ") + cudaGetErrorString(we)); }
  }
  {
    cudaError_t ae = cfg->goal_scoring ? (game ? opt_in_shared_memory<LGameGoals>() : opt_in_shared_memory<LTrainGoals>())
                                       : (game ? opt_in_shared_memory<LGame>() : opt_in_shared_memory<LTrain>());
    if (ae != cudaSuccess) { rr_destroy(s); return fail(RR_E_CUDA, std::string("cudaFuncSetAttribute: ") + cudaGetErrorString(ae)); }
  }
  if (cudaMemset(s->stats, 0, sizeof(double) * RR_NUM_STATS) != cudaSuccess) { rr_destroy(s); return fail(RR_E_CUDA, "cudaMemset failed"); }
  LAUNCH_PRESET(s, (cudaStream_t)0, (k_init<L>), s->k, s->sf, s->si, s->N, s->start);
  s->launches++;
  cudaError_t le = cudaGetLastError();
  if (le == cudaSuccess) le = cudaDeviceSynchronize();
  if (le != cudaSuccess) { rr_destroy(s); return fail(RR_E_CUDA, std::string("k_init: ") + cudaGetErrorString(le)); }
  *out = s;
  return RR_OK;
}

int rr_destroy(rr_sim *s) {
  if (!s) return RR_OK;
  DeviceGuard guard(s->device);
  cudaFree(s->sf); cudaFree(s->si); cudaFree(s->own_stats); cudaFree(s->start);
  cudaFree(s->d_act); cudaFree(s->d_obs_h); cudaFree(s->d_obs_g); cudaFree(s->d_rew); cudaFree(s->d_done);
  if (s->copy_stream) cudaStreamDestroy(s->copy_stream);
  for (cudaEvent_t e : s->chunk_done)
    if (e) cudaEventDestroy(e);
  pipeline_free(s);
  for (int t = 0; t < RR_HOST_TICKETS; t++) {
    cudaFree(s->d_act2[t]);
    if (s->ticket_done[t]) cudaEventDestroy(s->ticket_done[t]);
  }
  for (cudaStream_t t : s->ticket_stream)
    if (t) cudaStreamDestroy(t);
  delete s;
  return RR_OK;
}

int rr_num_envs(const rr_sim *s, int64_t *n) { if (!s || !n) return fail(RR_E_INVALID, "null"); *n = s->N; return RR_OK; }
int rr_num_robots(const rr_sim *s) { return s ? s->cols.R : RR_E_INVALID; }
int rr_num_balls(const rr_sim *s) { return s ? s->cols.B : RR_E_INVALID; }
int rr_max_steps(const rr_sim *s) { return s ? s->k.T : RR_E_INVALID; }
int rr_obs_dim(const rr_sim *s) {
  if (!s) return RR_E_INVALID;
  switch (s->cfg.observer) {
    case RR_OBS_BASIC_LIDAR: return 5;
    case RR_OBS_LIDAR6_V2: return 11;
    case RR_OBS_LIDAR6_V1: return 11;
    case RR_OBS_ALLCOORDS: return 3 * s->cols.R + 2 * s->cols.B;
    case RR_OBS_ALLCOORDS_PRIOR: return 6 * s->cols.R + 4 * s->cols.B;
    default: return 0;
  }
}
int64_t rr_launch_count(const rr_sim *s) { return s ? s->launches : 0; }
int64_t rr_state_bytes_per_env(const rr_sim *s) {
  return s ? s->cols.bytes_per_env(s->cfg.observer) : 0;
}

// ---------------------------------------------------------------------------------------------
// Device self-tests of the numeric building blocks that replace compiler / libm code (tests/test_parity_gpu.py).
namespace rr {
__device__ __forceinline__ uint64_t splitmix64(uint64_t &x) {
  uint64_t z = (x += 0x9E3779B97F4A7C15ull);
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}
// a double with random sign and mantissa and an exponent drawn from [-span, span]
__device__ __forceinline__ double random_double(uint64_t &st, int span) {
  const uint64_t u = splitmix64(st);
  const int ex = (int)(splitmix64(st) % (uint64_t)(2 * span + 1)) - span;
  const uint64_t bits = (u & 0x800FFFFFFFFFFFFFull) | ((uint64_t)(1023 + ex) << 52);
  return __longlong_as_double((long long)bits);
}
// which 0: div_core against the compiler's division.  out[0] = cases whose flag said "in range" but whose
// quotient differs from a / b (must be 0), out[1] = cases flagged out of range (redone by the caller).
__global__ void k_selftest_div(uint64_t seed, int64_t per_thread, unsigned long long *out) {
  uint64_t st = seed ^ (0xD1B54A32D192ED03ull * (uint64_t)(blockIdx.x * blockDim.x + threadIdx.x + 1));
  unsigned long long bad = 0, flagged = 0;
  for (int64_t it = 0; it < per_thread; it++) {
    double a, b;
    switch (it & 3) {
      case 0: a = random_double(st, 40); b = random_double(st, 40); break;       // slopes, intercepts
      case 1: a = random_double(st, 1000); b = random_double(st, 1000); break;   // whole exponent range
      case 2: {  // differences of arena coordinates: multiples of 2^-43 below 1024
        a = (double)((int64_t)(splitmix64(st) >> 11) - (1ll << 52)) * 0x1p-43;
        b = (double)((int64_t)(splitmix64(st) >> 11) - (1ll << 52)) * 0x1p-43;
        break;
      }
      default: {  // zeros, subnormals, infinities, NaN now and then
        const uint64_t sel = splitmix64(st) % 6;
        a = sel == 0 ? 0.0 : sel == 1 ? 4.9e-324 * (double)(splitmix64(st) % 1000) : random_double(st, 300);
        b = sel == 2 ? 0.0 : sel == 3 ? HUGE_VAL : sel == 4 ? 1e-310 : sel == 5 ? HUGE_VAL - HUGE_VAL : random_double(st, 300);
      }
    }
    bool ok;
    const double q = div_core(a, b, ok);
    const double ref = a / b;
    if (!ok) flagged++;
    else if (__double_as_longlong(q) != __double_as_longlong(ref)) bad++;
  }
  atomicAdd(&out[0], bad);
  atomicAdd(&out[1], flagged);
}

__device__ __forceinline__ double unit_double(uint64_t &st) { return (double)(splitmix64(st) >> 11) * 0x1p-53; }
__device__ __forceinline__ bool same_value(double a, double b) {  // bit-identical, or both NaN
  return (isnan(a) && isnan(b)) || __double_as_longlong(a) == __double_as_longlong(b);
}

// which 1: the branch-free side x line block of sides_x_lines (the __CUDA_ARCH__ branch) against sides_x_lines_plain, both
// on the device.  Half of the inputs are shaped like the simulator's: robot 0 of a GAME Env bound the way k_step binds
// it (trig table and hot fields in dynamic shared memory), its centre in the arena, its heading on the 0.2-degree grid
// plus rounding drift (exactly 0 / 90 / 180 / 270 and one ulp either side of them now and then), the ball anywhere
// within contact distance (exactly on a corner or a side midpoint now and then), and the ball's diameters as
// ball_robot_collided (buf 0) and apply_force_to_ball (buf 0.5) build them.  The other half are adversarial: lines
// parallel to a side (exact den == 0), vertical / horizontal and zero-length lines, lines through a corner, huge and
// tiny coordinates, NaN and infinity.  out[0] = inputs on which the mask, a point, a slope, an intercept or the error
// bits differ (must be 0), out[1] = inputs on which the block fell back to the ordinary divisions.
__global__ void __launch_bounds__(128, 1) k_selftest_sides(const __grid_constant__ Consts k, uint64_t seed,
                                                           int64_t per_thread, unsigned long long *out) {
  using E = LGame::E;
  E e;
  double cold[E::kColdDoubles];
  e.trig = stage_trig_table();
  bind_env(e, cold);
  e.rrot(0) = rr_nan();  // no heading yet, and no inner-corner offsets cached for one
  e.rc(0, 3) = rr_nan();
  uint64_t st = seed ^ (0x9E6C63D0676A9A99ull * (uint64_t)(blockIdx.x * blockDim.x + threadIdx.x + 1));
  unsigned long long bad = 0, fell = 0;
  for (int64_t it = 0; it < per_thread; it++) {
    P2 rc[4];
    Seg ln[2];
    double buf = 0.0;
    if ((it & 1) == 0) {  // simulator-shaped
      const uint64_t sel = splitmix64(st);
      double rot = 0.2 * (double)(int)(sel % 1800u);
      switch ((sel >> 12) % 8) {
        case 0: break;                                                         // on the grid
        case 1: rot += (unit_double(st) - 0.5) * 1e-11; break;                 // accumulated drift
        case 2: rot = 90.0 * (double)(int)((sel >> 20) % 4u); break;           // axis-aligned
        case 3: rot = nextafter(90.0 * (double)(int)((sel >> 20) % 4u) + (((sel >> 22) & 1) ? 0.0 : 360.0),
                                ((sel >> 22) & 1) ? 400.0 : 0.0) ; break;      // one ulp off an axis
        default: rot += (double)((int)((sel >> 20) % 7u) - 3) * 1e-13; break;  // a few ulps of drift
      }
      rot = norm_rot(rot);
      e.rcx(0) = 30.0 + 740.0 * unit_double(st);
      e.rcy(0) = 30.0 + 740.0 * unit_double(st);
      if (!(e.rrot(0) == rot)) {
        e.rrot(0) = rot;
        robot_refresh_corners(e, k, 0);
      }
      robot_refresh_ltrb(e, 0);
      robot_corners(e, 0, rc);
      double bx, by;
      const uint64_t where = splitmix64(st) % 16u;
      if (where < 4) {  // on a corner
        bx = rc[where].x; by = rc[where].y;
      } else if (where < 8) {  // on a side midpoint
        const Seg s = side_from_corners(rc, (int)where - 4);
        bx = (s.a.x + s.b.x) / 2.0; by = (s.a.y + s.b.y) / 2.0;
      } else {  // anywhere within 7.5 px of the robot, in its own frame
        const double u = (unit_double(st) * 2.0 - 1.0) * 17.5, v = (unit_double(st) * 2.0 - 1.0) * 27.5;
        const double ax = (e.ktrx(0) + e.kbrx(0)) * 0.5, ay = (e.ktry(0) + e.kbry(0)) * 0.5;  // half-length axis
        const double wx = (e.kbrx(0) - e.ktrx(0)) * 0.5, wy = (e.kbry(0) - e.ktry(0)) * 0.5;  // half-width axis
        bx = e.rcx(0) + u * 0.1 * ax + v * 0.05 * wx;
        by = e.rcy(0) + u * 0.1 * ay + v * 0.05 * wy;
      }
      P2 ic[4];
      inner_corners(e, k, 0, bx, by, ic);
      if ((sel >> 30) & 1) {  // ball_robot_collided
        ln[0] = Seg{ic[0], ic[3]}; ln[1] = Seg{ic[1], ic[2]};
      } else {  // apply_force_to_ball, bounce_ball_off_bot (with buf 0)
        ln[0] = Seg{ic[2], ic[1]}; ln[1] = Seg{ic[3], ic[0]};
        buf = ((sel >> 31) & 1) ? 0.5 : 0.0;
      }
    } else {  // adversarial: a rect with small integer corner offsets, so that parallel lines have equal slopes exactly
      const uint64_t sel = splitmix64(st);
      const double cx = (double)(int)(sel % 700u) + 50.0, cy = (double)(int)((sel >> 10) % 700u) + 50.0;
      const double px = (double)((int)((sel >> 20) % 41u) - 20), py = (double)((int)((sel >> 26) % 41u) - 20);
      const double qx = -py, qy = px;  // a perpendicular axis of the same length (a square, possibly degenerate)
      rc[0] = P2{cx - px - qx, cy - py - qy}; rc[1] = P2{cx + px - qx, cy + py - qy};
      rc[2] = P2{cx - px + qx, cy - py + qy}; rc[3] = P2{cx + px + qx, cy + py + qy};
      buf = ((sel >> 32) & 1) ? 0.5 : 0.0;
      for (int q = 0; q < 2; q++) {
        const uint64_t h = splitmix64(st);
        const double ox = (double)((int)(h % 61u) - 30), oy = (double)((int)((h >> 8) % 61u) - 30);
        const P2 a{cx + ox, cy + oy};
        const Seg sd = side_from_corners(rc, (int)((h >> 16) % 4u));
        const P2 cn = rc[(h >> 18) % 4u];
        switch ((h >> 20) % 8) {
          case 0: ln[q] = Seg{P2{sd.a.x + ox, sd.a.y + oy}, P2{sd.b.x + ox, sd.b.y + oy}}; break;  // parallel to a side
          case 1: ln[q] = Seg{a, P2{a.x, a.y + 9.0}}; break;                                          // vertical
          case 2: ln[q] = Seg{a, P2{a.x - 9.0, a.y}}; break;                                          // horizontal
          case 3: ln[q] = Seg{a, a}; break;                                                            // zero length
          case 4: ln[q] = Seg{cn, a}; break;                                                           // through a corner
          case 5: ln[q] = Seg{sd.a, sd.b}; break;                                                      // along a side
          default: ln[q] = Seg{a, P2{cx - ox + (double)((int)((h >> 24) % 7u) - 3), cy - oy}}; break;  // across
        }
      }
      const uint64_t mod = splitmix64(st) % 16u;
      if (mod < 6) {  // the same geometry scaled to huge or tiny coordinates
        const double f = mod == 0 ? 0x1p+900 : mod == 1 ? 0x1p-900 : mod == 2 ? 0x1p+500 : mod == 3 ? 0x1p-1000 : mod == 4 ? 1e-310 : 0x1p+1000;
        for (int i = 0; i < 4; i++) { rc[i].x *= f; rc[i].y *= f; }
        for (int q = 0; q < 2; q++) { ln[q].a.x *= f; ln[q].a.y *= f; ln[q].b.x *= f; ln[q].b.y *= f; }
      } else if (mod == 6 || mod == 7) {  // a NaN or an infinity in one coordinate
        const double v = mod == 6 ? rr_nan() : HUGE_VAL;
        const uint64_t c = splitmix64(st) % 12u;
        if (c < 8) { if (c & 1) rc[c >> 1].y = v; else rc[c >> 1].x = v; }
        else if (c == 8) ln[0].a.x = v; else if (c == 9) ln[0].b.y = v; else if (c == 10) ln[1].a.y = v; else ln[1].b.x = v;
      } else if (mod == 8) {  // arbitrary doubles
        for (int i = 0; i < 4; i++) { rc[i].x = random_double(st, 40); rc[i].y = random_double(st, 40); }
        for (int q = 0; q < 2; q++) {
          ln[q].a.x = random_double(st, 40); ln[q].a.y = random_double(st, 40);
          ln[q].b.x = random_double(st, 40); ln[q].b.y = random_double(st, 40);
        }
      }
    }
    P2 pt[8], pt2[8];
    double lm[2], lb[2], lm2[2], lb2[2];
    unsigned err = 0, err2 = 0;
    bool fb = false;
    const unsigned mask = sides_x_lines(rc, ln, buf, pt, lm, lb, err, &fb);
    const unsigned mask2 = sides_x_lines_plain(rc, ln, buf, pt2, lm2, lb2, err2);
    bool same = mask == mask2 && err == err2;
    for (int i = 0; i < 8; i++) same = same && same_value(pt[i].x, pt2[i].x) && same_value(pt[i].y, pt2[i].y);
    for (int q = 0; q < 2; q++) same = same && same_value(lm[q], lm2[q]) && same_value(lb[q], lb2[q]);
    bad += same ? 0 : 1;
    fell += fb ? 1 : 0;
  }
  atomicAdd(&out[0], bad);
  atomicAdd(&out[1], fell);
}
}  // namespace rr

int rr_selftest(int device, int which, int64_t n, uint64_t seed, int64_t *out2) {
  if (!out2 || n <= 0) return fail(RR_E_INVALID, "bad selftest arguments");
  ON_DEVICE(device);
  unsigned long long *d = nullptr;
  CK(cudaMalloc(&d, 2 * sizeof(unsigned long long)));
  CK(cudaMemset(d, 0, 2 * sizeof(unsigned long long)));
  const int blocks = 148 * 4, threads = which == 1 ? 128 : 256;
  const int64_t per_thread = (n + (int64_t)blocks * threads - 1) / ((int64_t)blocks * threads);
  if (which == 0) {
    rr::k_selftest_div<<<blocks, threads>>>(seed, per_thread, d);
  } else if (which == 1) {
    rr_config cfg;
    rr_default_config(&cfg, RR_PRESET_GAME, "RoboRugbySimpleDuel-v2");
    const size_t sm = LGame::smem_bytes(threads);
    cudaError_t ae = cudaFuncSetAttribute(rr::k_selftest_sides, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
    if (ae != cudaSuccess) { cudaFree(d); CK(ae); }
    rr::k_selftest_sides<<<blocks, threads, sm>>>(make_consts(cfg), seed, per_thread, d);
  } else {
    cudaFree(d);
    return fail(RR_E_INVALID, "unknown selftest");
  }
  cudaError_t e = cudaDeviceSynchronize();
  unsigned long long h[2] = {0, 0};
  if (e == cudaSuccess) e = cudaMemcpy(h, d, sizeof h, cudaMemcpyDeviceToHost);
  cudaFree(d);
  CK(e);
  out2[0] = (int64_t)h[0]; out2[1] = (int64_t)h[1];
  return RR_OK;
}

// Make `st` wait for everything the sub-batch streams have been given (no host blocking).  Every entry point that reads
// or writes the state on the caller's stream calls this first, so only consecutive rr_step calls overlap.
static int join_into(rr_sim *s, cudaStream_t st) {
  if (!s->pipe_pending) return RR_OK;
  for (cudaEvent_t e : s->sub_done) CK(cudaStreamWaitEvent(st, e, 0));
  s->pipe_pending = false;
  return RR_OK;
}

static void pipeline_free(rr_sim *s) {
  for (cudaStream_t t : s->sub) cudaStreamDestroy(t);
  for (cudaEvent_t e : s->sub_done) cudaEventDestroy(e);
  if (s->pipe_entry) cudaEventDestroy(s->pipe_entry);
  s->sub.clear(); s->sub_done.clear(); s->pipe_entry = nullptr; s->pipe = 1; s->pipe_pending = false;
}

int rr_set_pipeline(rr_sim *s, int32_t sub_batches) {
  if (!s) return fail(RR_E_INVALID, "null handle");
  if (sub_batches < 1 || sub_batches > 128) return fail(RR_E_INVALID, "sub_batches must be in [1, 128]");
  ON_DEVICE(s->device);
  CK(cudaDeviceSynchronize());
  pipeline_free(s);
  if (sub_batches == 1) return RR_OK;
  CK(cudaEventCreateWithFlags(&s->pipe_entry, cudaEventDisableTiming));
  for (int j = 0; j < sub_batches; j++) {
    cudaStream_t t; cudaEvent_t e;
    CK(cudaStreamCreateWithFlags(&t, cudaStreamNonBlocking));
    s->sub.push_back(t);
    CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    s->sub_done.push_back(e);
  }
  s->pipe = sub_batches;
  return RR_OK;
}

int rr_set_flush_buffer(rr_sim *s, void *buf_dev, int64_t bytes) {
  if (!s || bytes < 0) return fail(RR_E_INVALID, "bad arguments");
  ON_DEVICE(s->device);
  CK(cudaDeviceSynchronize());
  s->flush_buf = bytes > 0 ? buf_dev : nullptr;
  s->flush_bytes = s->flush_buf ? (size_t)bytes : 0;
  return RR_OK;
}

int rr_join(rr_sim *s, void *stream) {
  if (!s) return fail(RR_E_INVALID, "null handle");
  ON_DEVICE(s->device);
  return join_into(s, (cudaStream_t)stream);
}

int rr_reset(rr_sim *s, const uint8_t *mask_dev, void *stream) {
  if (!s) return fail(RR_E_INVALID, "null handle");
  ON_DEVICE(s->device);
  cudaStream_t st = (cudaStream_t)stream;
  if (int jr = join_into(s, st)) return jr;
  LAUNCH_PRESET(s, st, (k_reset<L>), s->k, s->sf, s->si, s->N, mask_dev);
  s->launches++;
  CK(cudaGetLastError());
  return RR_OK;
}

int rr_reset_fixed(rr_sim *s, const uint8_t *mask_dev, int32_t as_constructed, void *stream) {
  if (!s) return fail(RR_E_INVALID, "null handle");
  ON_DEVICE(s->device);
  cudaStream_t st = (cudaStream_t)stream;
  if (int jr = join_into(s, st)) return jr;
  LAUNCH_PRESET(s, st, (k_reset_fixed<L>), s->k, s->sf, s->si, s->N, mask_dev, s->start, (int)as_constructed);
  s->launches++;
  CK(cudaGetLastError());
  return RR_OK;
}

int rr_set_starting_positions(rr_sim *s, const double *rob3, const double *ball2) {
  if (!s || !rob3 || !ball2) return fail(RR_E_INVALID, "null argument");
  ON_DEVICE(s->device);
  CK(cudaDeviceSynchronize());
  const int64_t N = s->N;
  const int R = s->cols.R, B = s->cols.B;
  std::vector<double> st((size_t)(3 * R + 2 * B) * N);
  for (int64_t i = 0; i < N; i++) {
    for (int q = 0; q < 3 * R; q++) st[(size_t)q * N + i] = rob3[i * 3 * R + q];
    for (int q = 0; q < 2 * B; q++) st[(size_t)(3 * R + q) * N + i] = ball2[i * 2 * B + q];
  }
  CK(cudaMemcpy(s->start, st.data(), sizeof(double) * st.size(), cudaMemcpyHostToDevice));
  return RR_OK;
}

int rr_get_starting_positions(rr_sim *s, double *rob3, double *ball2) {
  if (!s || !rob3 || !ball2) return fail(RR_E_INVALID, "null argument");
  ON_DEVICE(s->device);
  CK(cudaDeviceSynchronize());
  const int64_t N = s->N;
  const int R = s->cols.R, B = s->cols.B;
  std::vector<double> st((size_t)(3 * R + 2 * B) * N);
  CK(cudaMemcpy(st.data(), s->start, sizeof(double) * st.size(), cudaMemcpyDeviceToHost));
  for (int64_t i = 0; i < N; i++) {
    for (int q = 0; q < 3 * R; q++) rob3[i * 3 * R + q] = st[(size_t)q * N + i];
    for (int q = 0; q < 2 * B; q++) ball2[i * 2 * B + q] = st[(size_t)(3 * R + q) * N + i];
  }
  return RR_OK;
}

// The kernels store out_t elements and load float actions / int32 ball indices: a pointer that is not aligned to its
// element type would fault on the device, so the entry points refuse it.
static bool misaligned(const void *p, size_t align) { return ((uintptr_t)p & (align - 1)) != 0; }
static size_t out_size(const rr_sim *s) { return s->cfg.out_f64 ? 8 : 4; }

int rr_observe(rr_sim *s, void *obs_h, void *obs_g, void *stream) {
  if (!s) return fail(RR_E_INVALID, "null handle");
  if (rr_obs_dim(s) == 0) return RR_OK;
  if (misaligned(obs_h, out_size(s)) || misaligned(obs_g, out_size(s)))
    return fail(RR_E_INVALID, "observation buffers must be aligned to their element type");
  ON_DEVICE(s->device);
  cudaStream_t st = (cudaStream_t)stream;
  if (int jr = join_into(s, st)) return jr;
  if (s->cfg.out_f64)
    LAUNCH_PRESET(s, st, (k_observe<L, double>), s->k, s->sf, s->si, s->N, obs_h, obs_g);
  else
    LAUNCH_PRESET(s, st, (k_observe<L, float>), s->k, s->sf, s->si, s->N, obs_h, obs_g);
  s->launches++;
  CK(cudaGetLastError());
  return RR_OK;
}

int rr_observe_entity(rr_sim *s, int32_t robot, int32_t ball, const int32_t *ball_dev, void *obs, void *stream) {
  if (!s || !obs) return fail(RR_E_INVALID, "null argument");
  const int ob = s->cfg.observer;
  if (ob == RR_OBS_ALLCOORDS || ob == RR_OBS_ALLCOORDS_PRIOR)
    return fail(RR_E_INVALID, "Robot-specific state output not supported.");  // RR_Observers.py:59-60
  if (ob == RR_OBS_NONE) return fail(RR_E_INVALID, "this env has no observer");
  if (robot < 0 || robot >= s->cols.R) return fail(RR_E_INVALID, "robot index out of range");
  if (!ball_dev && ball >= s->cols.B) return fail(RR_E_INVALID, "ball index out of range");
  if (misaligned(obs, out_size(s)) || misaligned(ball_dev, 4))
    return fail(RR_E_INVALID, "obs and ball_dev must be aligned to their element types");
  ON_DEVICE(s->device);
  cudaStream_t st = (cudaStream_t)stream;
  if (int jr = join_into(s, st)) return jr;
  if (s->cfg.out_f64)
    LAUNCH_PRESET(s, st, (k_observe_entity<L, double>), s->k, s->sf, s->si, s->N, (int)robot, (int)ball, ball_dev, obs);
  else
    LAUNCH_PRESET(s, st, (k_observe_entity<L, float>), s->k, s->sf, s->si, s->N, (int)robot, (int)ball, ball_dev, obs);
  s->launches++;
  CK(cudaGetLastError());
  return RR_OK;
}

int rr_assign_balls(rr_sim *s, const int32_t *robots_host, int32_t n_robots, int32_t *assign_dev, void *stream) {
  if (!s || !robots_host || !assign_dev) return fail(RR_E_INVALID, "null argument");
  if (n_robots < 1 || n_robots > s->cols.R || n_robots > 8) return fail(RR_E_INVALID, "n_robots out of range");
  RobotList rl{};
  rl.n = n_robots;
  for (int j = 0; j < n_robots; j++) {
    if (robots_host[j] < 0 || robots_host[j] >= s->cols.R) return fail(RR_E_INVALID, "robot index out of range");
    rl.idx[j] = robots_host[j];
  }
  ON_DEVICE(s->device);
  cudaStream_t st = (cudaStream_t)stream;
  if (int jr = join_into(s, st)) return jr;
  LAUNCH_PRESET(s, st, (k_assign_balls<L>), s->k, s->sf, s->si, s->N, rl, assign_dev);
  s->launches++;
  CK(cudaGetLastError());
  return RR_OK;
}

int64_t rr_snapshot_bytes_per_env(const rr_sim *s) { return s ? row_layout(s->cols, s->cfg.observer).bytes() : 0; }

// The checks of rr_save_states / rr_load_states: the kernels never touch memory outside the buffers the caller described.
static int check_rows(const rr_sim *s, const void *rows, int64_t m, const int64_t *idx, bool null_idx_ok, const char *rule) {
  if (!s || !rows) return fail(RR_E_INVALID, "null argument");
  if (m < 1) return fail(RR_E_INVALID, "m must be >= 1");
  if (misaligned(rows, 16)) return fail(RR_E_INVALID, "the rows buffer must be 16-byte aligned");
  if (misaligned(idx, 8)) return fail(RR_E_INVALID, "the index buffer must be 8-byte aligned");
  if (!idx && !null_idx_ok) return fail(RR_E_INVALID, rule);
  return RR_OK;
}

int rr_save_states(rr_sim *s, const int64_t *env_dev, int64_t m, void *rows_dev, void *stream) {
  if (int rc = check_rows(s, rows_dev, m, env_dev, s && m <= s->N, "without env indices m must be <= n_envs")) return rc;
  ON_DEVICE(s->device);
  cudaStream_t st = (cudaStream_t)stream;
  if (int jr = join_into(s, st)) return jr;
  const RowLayout L = row_layout(s->cols, s->cfg.observer);
  k_save_rows<<<(unsigned)((m + kRowTile - 1) / kRowTile), kRowThreads, row_tile_bytes(L), st>>>(
      L, (const uint64_t *)s->sf, (const uint64_t *)s->start, (const uint32_t *)s->si, s->N, env_dev, m, (uint4 *)rows_dev);
  s->launches++;
  CK(cudaGetLastError());
  return RR_OK;
}

int rr_load_states(rr_sim *s, const void *rows_dev, int64_t m, const int64_t *slot_dev, void *stream) {
  if (int rc = check_rows(s, rows_dev, m, slot_dev, s && m == s->N, "without slot indices m must equal n_envs")) return rc;
  ON_DEVICE(s->device);
  cudaStream_t st = (cudaStream_t)stream;
  if (int jr = join_into(s, st)) return jr;
  const RowLayout L = row_layout(s->cols, s->cfg.observer);
  k_load_rows<<<(unsigned)((s->N + kRowTile - 1) / kRowTile), kRowThreads, row_tile_bytes(L), st>>>(
      L, (const uint4 *)rows_dev, m, slot_dev, s->N, (uint64_t *)s->sf, (uint64_t *)s->start, (uint32_t *)s->si);
  s->launches++;
  CK(cudaGetLastError());
  return RR_OK;
}

static int check_actions(const rr_sim *s, int32_t n_actions, int32_t k_steps) {
  if (k_steps <= 0) return fail(RR_E_INVALID, "k_steps must be positive");
  if (n_actions < 0) return fail(RR_E_INVALID, "n_actions must be >= 0");
  // RR_EnvBase.py:621-622 / :270-271: more commands than robots (engines) raises
  if (s->cfg.discrete && n_actions > s->cols.R)
    return fail(RR_E_INVALID, std::to_string(n_actions) + " commands but only " + std::to_string(s->cols.R) + " robots.");
  if (!s->cfg.discrete && (n_actions > 2 * s->cols.R || (n_actions & 1)))
    return fail(RR_E_INVALID, std::to_string(n_actions) + " commands but only " + std::to_string(2 * s->cols.R) + " robot engines.");
  return RR_OK;
}

int rr_step(rr_sim *s, const void *actions, int32_t n_actions, int32_t k_steps, void *obs_h, void *obs_g, void *rew,
            uint8_t *done, void *stream) {
  return rr_step_info(s, actions, n_actions, k_steps, obs_h, obs_g, rew, done, nullptr, nullptr, nullptr, stream);
}

// rr_step_info, and rr_step_episodes when `pool` or an episode output is given (their checks made by the caller)
static int step_launch(rr_sim *s, const void *actions, int32_t n_actions, int32_t k_steps, void *obs_h, void *obs_g,
                       void *rew, uint8_t *done, void *final_obs_h, void *final_obs_g, uint8_t *row_flags,
                       const rr_reset_pool *pool, int32_t *reset_slot, double *ep_return, int32_t *ep_length,
                       int32_t *ep_goals, void *stream) {
  if (!s) return fail(RR_E_INVALID, "null handle");
  int rc = check_actions(s, n_actions, k_steps);
  if (rc) return rc;
  if (n_actions > 0 && !actions) return fail(RR_E_INVALID, "actions is null");
  const size_t osz = out_size(s);
  if (misaligned(obs_h, osz) || misaligned(obs_g, osz) || misaligned(rew, osz) || (!s->cfg.discrete && misaligned(actions, 4)))
    return fail(RR_E_INVALID, "result buffers must be aligned to their element type, continuous actions to 4 bytes");
  if (rr_obs_dim(s) == 0) final_obs_h = final_obs_g = nullptr;  // no observation: nothing to report
  if (misaligned(final_obs_h, osz) || misaligned(final_obs_g, osz))
    return fail(RR_E_INVALID, "final observation buffers must be aligned to their element type");
  const bool pooled = pool != nullptr;
  const bool info = pooled || final_obs_h || final_obs_g || row_flags || ep_return || ep_length || ep_goals;
  ON_DEVICE(s->device);
  cudaStream_t st = (cudaStream_t)stream;
  Consts k = s->k;
  k.n_actions = n_actions;
  // 128-bit result stores need 16-byte aligned buffers whose per-step rows are multiples of 16 bytes
  auto rows16 = [&](const void *p, size_t row_bytes) { return (((uintptr_t)p) & 15u) == 0 && (row_bytes & 15u) == 0; };
  unsigned vec = 0;
  const size_t D = (size_t)rr_obs_dim(s);
  if (rows16(obs_h, s->N * D * osz) && rows16(obs_g, s->N * D * osz)) vec |= 1u;
  if (rows16(rew, s->N * 2 * osz)) vec |= 2u;
  if (rows16(done, (size_t)s->N)) vec |= 4u;
  if ((((uintptr_t)actions) & 3u) == 0) vec |= 8u;
  if (rows16(row_flags, (size_t)s->N)) vec |= 16u;
  if (rows16(reset_slot, (size_t)s->N * 4)) vec |= 32u;
  if (rows16(ep_return, (size_t)s->N * 16)) vec |= 64u;
  if (rows16(ep_length, (size_t)s->N * 4)) vec |= 128u;
  if (rows16(ep_goals, (size_t)s->N * 16)) vec |= 256u;
  PoolStepArgs pa{};
  if (pooled) pa.pool = ResetPool{(const uint64_t *)pool->rows_dev, pool->cdf_dev, pool->m, pool->p_pool};
  pa.start = s->start;
  pa.reset_slot = reset_slot;
  pa.ep_return = ep_return;
  pa.ep_length = ep_length;
  pa.ep_goals = ep_goals;
  InfoStepArgs &ia = pa;  // what the INFO variants take
  StepArgs &a = pa;       // what the default variants take
  a = StepArgs{s->sf, s->si, s->stats, actions, obs_h, obs_g, rew, done, s->N, k_steps, vec, 0, final_obs_h, final_obs_g, row_flags};
  const bool game = s->cfg.preset == RR_PRESET_GAME, goals = s->cfg.goal_scoring != 0, f64 = s->cfg.out_f64 != 0;
  // one stream-ordered launch per call over more envs than 384-thread blocks cover in one wave: 448-thread blocks
  const bool wide = game && s->pipe <= 1 && (s->N + LGame::kMaxBlock - 1) / LGame::kMaxBlock > s->sms &&
                    LGame::kMaxBlock < LGameWide::kMaxBlock;
  const int blk = pick_block(s->N, s->sms, wide ? LGameWide::kMaxBlock : (game ? LGame::kMaxBlock : LTrain::kMaxBlock));
  const int nb = (int)((s->N + blk - 1) / blk);
  auto launch = [&](cudaStream_t on, int block0, int nblocks, int blk) {
    a.block0 = block0;
#define RR_STEP_CASE(LTYPE)                                                                                  \
    do {                                                                                                     \
      const size_t sm = LTYPE::smem_bytes(blk);                                                              \
      if (pooled && f64) k_step<LTYPE, double, true, true><<<(unsigned)nblocks, blk, sm, on>>>(k, pa);       \
      else if (pooled) k_step<LTYPE, float, true, true><<<(unsigned)nblocks, blk, sm, on>>>(k, pa);          \
      else if (info && f64) k_step<LTYPE, double, true><<<(unsigned)nblocks, blk, sm, on>>>(k, ia);          \
      else if (info) k_step<LTYPE, float, true><<<(unsigned)nblocks, blk, sm, on>>>(k, ia);                  \
      else if (f64) k_step<LTYPE, double><<<(unsigned)nblocks, blk, sm, on>>>(k, a);                         \
      else k_step<LTYPE, float><<<(unsigned)nblocks, blk, sm, on>>>(k, a);                                   \
    } while (0)
    if (game && !goals) { if (wide) RR_STEP_CASE(LGameWide); else RR_STEP_CASE(LGame); }
    else if (!game && !goals) RR_STEP_CASE(LTrain);
    else if (game) { if (wide) RR_STEP_CASE(LGameGoalsWide); else RR_STEP_CASE(LGameGoals); }
    else RR_STEP_CASE(LTrainGoals);
#undef RR_STEP_CASE
  };
  const int groups = s->pipe < nb ? s->pipe : nb;
  if (groups <= 1) {
    if (int jr = join_into(s, st)) return jr;
    if (s->flush_buf) CK(cudaMemsetAsync(s->flush_buf, (int)(s->launches & 0xff), s->flush_bytes, st));
    launch(st, 0, nb, blk);
    s->launches++;
  } else {
    // Sub-batch pipeline: the groups wait for what the caller's stream holds so far (the actions, earlier resets, ...)
    // and for their own previous launch (stream order); the caller's stream does NOT wait for them (rr_join).
    CK(cudaEventRecord(s->pipe_entry, st));
    for (int j = 0; j < groups; j++) {
      const int b0 = (int)((int64_t)nb * j / groups), b1 = (int)((int64_t)nb * (j + 1) / groups);
      CK(cudaStreamWaitEvent(s->sub[j], s->pipe_entry, 0));
      if (s->flush_buf) {  // this group's share of the flush, in front of its launch
        const size_t f0 = s->flush_bytes / groups * j, f1 = j + 1 == groups ? s->flush_bytes : s->flush_bytes / groups * (j + 1);
        CK(cudaMemsetAsync((char *)s->flush_buf + f0, (int)(s->launches & 0xff), f1 - f0, s->sub[j]));
      }
      launch(s->sub[j], b0, b1 - b0, blk);
      CK(cudaEventRecord(s->sub_done[j], s->sub[j]));
      s->launches++;
    }
    s->pipe_pending = true;
  }
  CK(cudaGetLastError());
  return RR_OK;
}

int rr_step_info(rr_sim *s, const void *actions, int32_t n_actions, int32_t k_steps, void *obs_h, void *obs_g, void *rew,
                 uint8_t *done, void *final_obs_h, void *final_obs_g, uint8_t *row_flags, void *stream) {
  return step_launch(s, actions, n_actions, k_steps, obs_h, obs_g, rew, done, final_obs_h, final_obs_g, row_flags, nullptr,
                     nullptr, nullptr, nullptr, nullptr, stream);
}

int rr_step_pool(rr_sim *s, const void *actions, int32_t n_actions, int32_t k_steps, void *obs_h, void *obs_g, void *rew,
                 uint8_t *done, void *final_obs_h, void *final_obs_g, uint8_t *row_flags, const rr_reset_pool *pool,
                 int32_t *reset_slot, void *stream) {
  return rr_step_episodes(s, actions, n_actions, k_steps, obs_h, obs_g, rew, done, final_obs_h, final_obs_g, row_flags, pool,
                          reset_slot, nullptr, nullptr, nullptr, stream);
}

int rr_step_episodes(rr_sim *s, const void *actions, int32_t n_actions, int32_t k_steps, void *obs_h, void *obs_g,
                     void *rew, uint8_t *done, void *final_obs_h, void *final_obs_g, uint8_t *row_flags,
                     const rr_reset_pool *pool, int32_t *reset_slot, double *ep_return, int32_t *ep_length,
                     int32_t *ep_goals, void *stream) {
  if (!s) return fail(RR_E_INVALID, "null handle");
  if (pool) {
    if (!pool->rows_dev) return fail(RR_E_INVALID, "reset pool: rows_dev is null");
    if (pool->m < 1 || pool->m > INT32_MAX) return fail(RR_E_INVALID, "reset pool: m must be in [1, INT32_MAX]");
    if (misaligned(pool->rows_dev, 16)) return fail(RR_E_INVALID, "reset pool: rows_dev must be 16-byte aligned");
    if (misaligned(pool->cdf_dev, 8)) return fail(RR_E_INVALID, "reset pool: cdf_dev must be 8-byte aligned");
    if (!(pool->p_pool >= 0.0 && pool->p_pool <= 1.0)) return fail(RR_E_INVALID, "reset pool: p_pool must lie in [0, 1]");
    if (!s->cfg.auto_reset) return fail(RR_E_INVALID, "reset pool: the handle was created with auto_reset = 0");
  }
  if (misaligned(reset_slot, 4)) return fail(RR_E_INVALID, "reset_slot must be 4-byte aligned");
  if (misaligned(ep_return, 8)) return fail(RR_E_INVALID, "ep_return must be 8-byte aligned");
  if (misaligned(ep_length, 4) || misaligned(ep_goals, 4))
    return fail(RR_E_INVALID, "ep_length and ep_goals must be 4-byte aligned");
  if (ep_goals && !s->cfg.goal_scoring) return fail(RR_E_INVALID, "ep_goals: the handle was created without goal_scoring");
  const int rc = step_launch(s, actions, n_actions, k_steps, obs_h, obs_g, rew, done, final_obs_h, final_obs_g, row_flags,
                             pool, reset_slot, ep_return, ep_length, ep_goals, stream);
  if (rc || pool || !reset_slot) return rc;
  // without a pool these are rr_step_info's kernels, and no row is reset from a pool
  ON_DEVICE(s->device);
  CK(cudaMemsetAsync(reset_slot, 0xff, sizeof(int32_t) * (size_t)k_steps * (size_t)s->N, (cudaStream_t)stream));
  return RR_OK;
}

static int ensure(void **p, size_t *cap, size_t need) {
  if (need <= *cap) return RR_OK;
  cudaFree(*p);
  *p = nullptr; *cap = 0;
  if (cudaMalloc(p, need) != cudaSuccess) { cudaGetLastError(); return fail(RR_E_NOMEM, "device staging allocation failed"); }
  *cap = need;
  return RR_OK;
}

// device alias of a pinned (page-locked, mapped) host buffer, or null for pageable memory
static void *pinned_alias(const void *host) {
  if (!host) return nullptr;
  cudaPointerAttributes at;
  if (cudaPointerGetAttributes(&at, host) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  return at.type == cudaMemoryTypeHost ? at.devicePointer : nullptr;
}

int rr_step_host(rr_sim *s, const void *actions, int32_t n_actions, int32_t k_steps, void *obs_h, void *obs_g, void *rew,
                 uint8_t *done, void *stream) {
  if (!s) return fail(RR_E_INVALID, "null handle");
  int rc = check_actions(s, n_actions, k_steps);
  if (rc) return rc;
  ON_DEVICE(s->device);
  cudaStream_t st = (cudaStream_t)stream;
  const size_t osz = s->cfg.out_f64 ? 8 : 4;
  const size_t rows = (size_t)k_steps * (size_t)s->N;
  const size_t act_b = rows * n_actions * (s->cfg.discrete ? 1 : 4);
  const size_t obs_b = rows * rr_obs_dim(s) * osz, rew_b = rows * 2 * osz, done_b = rows;
  if ((rc = ensure(&s->d_act, &s->cap_act, act_b ? act_b : 1))) return rc;
  if (act_b) CK(cudaMemcpyAsync(s->d_act, actions, act_b, cudaMemcpyHostToDevice, st));

  // Pinned result buffers: the kernel writes its rows straight into host memory (coalesced 128-bit streaming stores over
  // PCIe / NVLink-C2C), so the device-to-host traffic overlaps the launch completely and nothing is staged in HBM.
  if (s->host_zero_copy) {
    void *a_oh = pinned_alias(obs_h), *a_og = pinned_alias(obs_g), *a_rw = pinned_alias(rew), *a_dn = pinned_alias(done);
    const bool all_pinned = (!obs_h || !obs_b || a_oh) && (!obs_g || !obs_b || a_og) && (!rew || a_rw) && (!done || a_dn);
    if (all_pinned) {
      rc = rr_step(s, s->d_act, n_actions, k_steps, obs_b ? a_oh : nullptr, obs_b ? a_og : nullptr, a_rw, (uint8_t *)a_dn, stream);
      if (rc) return rc;
      if (int jr = join_into(s, st)) return jr;
      CK(cudaStreamSynchronize(st));
      return RR_OK;
    }
  }

  // Pageable result buffers: staged in HBM and copied.  The K steps run as up to four launches of K/4 steps (same
  // results: the state lives in HBM between launches); the device-to-host copies of one chunk's rows overlap the next
  // chunk's kernel.  Outputs are [K][N][...], so a chunk of steps is one contiguous range of every buffer.  Every launch
  // pays a fixed cost (state load / store, corner tables) and ends with its slowest env, so splitting only pays where the
  // copies dominate: 4 chunks for the light TRAIN preset, 1 for GAME (profiles/README.md).  RR_HOST_CHUNKS (read once,
  // at rr_create) overrides it.
  if ((rc = ensure(&s->d_obs_h, &s->cap_obs_h, obs_b ? obs_b : 1))) return rc;
  if ((rc = ensure(&s->d_obs_g, &s->cap_obs_g, obs_b ? obs_b : 1))) return rc;
  if ((rc = ensure(&s->d_rew, &s->cap_rew, rew_b))) return rc;
  if ((rc = ensure((void **)&s->d_done, &s->cap_done, done_b))) return rc;
  if (!s->copy_stream) {
    CK(cudaStreamCreateWithFlags(&s->copy_stream, cudaStreamNonBlocking));
    for (cudaEvent_t &e : s->chunk_done) CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  }
  int chunks = s->host_chunks > 0 ? s->host_chunks : (s->cols.R > 1 ? 1 : 4);
  if (chunks > 4) chunks = 4;
  if (chunks < 1 || k_steps < chunks) chunks = 1;
  const size_t act_row = (size_t)s->N * n_actions * (s->cfg.discrete ? 1 : 4);
  const size_t obs_row = (size_t)s->N * rr_obs_dim(s) * osz, rew_row = (size_t)s->N * 2 * osz, done_row = (size_t)s->N;
  int k0 = 0;
  for (int c = 0; c < chunks; c++) {
    const int kc = (k_steps - k0) / (chunks - c);
    const size_t r0 = (size_t)k0, rn = (size_t)kc;
    rc = rr_step(s, (const char *)s->d_act + r0 * act_row, n_actions, kc, obs_h ? (char *)s->d_obs_h + r0 * obs_row : nullptr,
                 obs_g ? (char *)s->d_obs_g + r0 * obs_row : nullptr, rew ? (char *)s->d_rew + r0 * rew_row : nullptr,
                 done ? s->d_done + r0 * done_row : nullptr, stream);
    if (rc) return rc;
    if (int jr = join_into(s, st)) return jr;
    CK(cudaEventRecord(s->chunk_done[c], st));
    CK(cudaStreamWaitEvent(s->copy_stream, s->chunk_done[c], 0));
    cudaStream_t cs = s->copy_stream;
    if (obs_h && obs_row) CK(cudaMemcpyAsync((char *)obs_h + r0 * obs_row, (char *)s->d_obs_h + r0 * obs_row, rn * obs_row, cudaMemcpyDeviceToHost, cs));
    if (obs_g && obs_row) CK(cudaMemcpyAsync((char *)obs_g + r0 * obs_row, (char *)s->d_obs_g + r0 * obs_row, rn * obs_row, cudaMemcpyDeviceToHost, cs));
    if (rew) CK(cudaMemcpyAsync((char *)rew + r0 * rew_row, (char *)s->d_rew + r0 * rew_row, rn * rew_row, cudaMemcpyDeviceToHost, cs));
    if (done) CK(cudaMemcpyAsync(done + r0 * done_row, s->d_done + r0 * done_row, rn * done_row, cudaMemcpyDeviceToHost, cs));
    k0 += kc;
  }
  CK(cudaStreamSynchronize(s->copy_stream));
  CK(cudaStreamSynchronize(st));
  return RR_OK;
}

// Several host-buffer calls in flight.  rr_step_host_begin enqueues one call (actions copied from host memory, result rows
// written by the kernels straight into the caller's PINNED buffers) and returns a ticket at once; rr_step_host_end blocks
// until that call's results are in host memory.  With a sub-batch pipeline (rr_set_pipeline) the groups of call n + 1
// start as soon as their own group of call n has finished, while the host still waits for, or consumes, call n.
int rr_step_host_begin(rr_sim *s, const void *actions, int32_t n_actions, int32_t k_steps, void *obs_h, void *obs_g, void *rew,
                       uint8_t *done, int32_t *ticket) {
  if (!s || !ticket) return fail(RR_E_INVALID, "null argument");
  int rc = check_actions(s, n_actions, k_steps);
  if (rc) return rc;
  if (n_actions > 0 && !actions) return fail(RR_E_INVALID, "actions is null");
  ON_DEVICE(s->device);
  const size_t osz = s->cfg.out_f64 ? 8 : 4;
  const size_t rows = (size_t)k_steps * (size_t)s->N;
  const size_t act_b = rows * n_actions * (s->cfg.discrete ? 1 : 4);
  const size_t obs_b = rows * rr_obs_dim(s) * osz;
  void *a_oh = pinned_alias(obs_h), *a_og = pinned_alias(obs_g), *a_rw = pinned_alias(rew), *a_dn = pinned_alias(done);
  if ((obs_h && obs_b && !a_oh) || (obs_g && obs_b && !a_og) || (rew && !a_rw) || (done && !a_dn))
    return fail(RR_E_INVALID, "rr_step_host_begin needs pinned (page-locked, mapped) result buffers; use rr_step_host");
  if (!s->ticket_stream[0]) {
    CK(cudaStreamCreateWithFlags(&s->ticket_stream[0], cudaStreamNonBlocking));  // submission: action copies, entry events
    CK(cudaStreamCreateWithFlags(&s->ticket_stream[1], cudaStreamNonBlocking));  // collection: waits for the groups
    for (cudaEvent_t &e : s->ticket_done) CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  }
  const int t = s->next_ticket;
  s->next_ticket = (t + 1) % RR_HOST_TICKETS;
  CK(cudaEventSynchronize(s->ticket_done[t]));  // the call that used this slot last (no-op if never recorded)
  if ((rc = ensure(&s->d_act2[t], &s->cap_act2[t], act_b ? act_b : 1))) return rc;
  cudaStream_t sub_st = s->ticket_stream[0], col = s->ticket_stream[1];
  if (act_b) CK(cudaMemcpyAsync(s->d_act2[t], actions, act_b, cudaMemcpyHostToDevice, sub_st));
  rc = rr_step(s, s->d_act2[t], n_actions, k_steps, obs_b ? a_oh : nullptr, obs_b ? a_og : nullptr, a_rw, (uint8_t *)a_dn, sub_st);
  if (rc) return rc;
  if (s->pipe_pending) {  // the groups of THIS call (their latest events); the submission stream is not held back
    for (cudaEvent_t e : s->sub_done) CK(cudaStreamWaitEvent(col, e, 0));
    CK(cudaEventRecord(s->ticket_done[t], col));
  } else {
    CK(cudaEventRecord(s->ticket_done[t], sub_st));
  }
  *ticket = t;
  return RR_OK;
}

int rr_step_host_end(rr_sim *s, int32_t ticket) {
  if (!s || ticket < 0 || ticket >= RR_HOST_TICKETS || !s->ticket_done[ticket]) return fail(RR_E_INVALID, "bad ticket");
  ON_DEVICE(s->device);
  CK(cudaEventSynchronize(s->ticket_done[ticket]));
  return RR_OK;
}

int rr_set_state(rr_sim *s, const double *rob, const double *rhist, const int32_t *rflag, const double *ball,
                 const int32_t *step) {
  if (!s || !rob || !rhist || !rflag || !ball || !step) return fail(RR_E_INVALID, "null argument");
  const int64_t N = s->N;
  const int R = s->cols.R, B = s->cols.B;
  for (int64_t q = 0; q < N * R; q++) {  // what the packed si column can hold (Env::thrust: 4 bits per thrust)
    const int32_t *g = rflag + 3 * q;
    if (g[0] < -8 || g[0] > 7 || g[1] < -8 || g[1] > 7 || (g[2] != 0 && g[2] != 1))
      return fail(RR_E_INVALID, "rflag of env " + std::to_string(q / R) + " robot " + std::to_string(q % R) +
                                    ": thrusts must lie in [-8, 7] and hist_valid must be 0 or 1");
  }
  ON_DEVICE(s->device);
  CK(cudaDeviceSynchronize());
  std::vector<double> sf((size_t)s->cols.nf(s->cfg.observer) * N);
  std::vector<int32_t> si((size_t)s->cols.ni() * N);
  CK(cudaMemcpy(si.data(), s->si, sizeof(int32_t) * si.size(), cudaMemcpyDeviceToHost));  // keep episode counters
  for (int64_t i = 0; i < N; i++)
    state_to_columns(s->cols, s->cfg.observer, sf.data(), si.data(), N, i, rob + i * R * 7, rhist + i * R * 3,
                     rflag + i * R * 3, ball + i * B * 8, step[i]);
  CK(cudaMemcpy(s->sf, sf.data(), sizeof(double) * sf.size(), cudaMemcpyHostToDevice));
  CK(cudaMemcpy(s->si, si.data(), sizeof(int32_t) * si.size(), cudaMemcpyHostToDevice));
  return RR_OK;
}

int rr_get_state(rr_sim *s, double *rob, double *rhist, int32_t *rflag, double *ball, int32_t *step) {
  if (!s || !rob || !rhist || !rflag || !ball || !step) return fail(RR_E_INVALID, "null argument");
  ON_DEVICE(s->device);
  CK(cudaDeviceSynchronize());
  const int64_t N = s->N;
  const int R = s->cols.R, B = s->cols.B;
  std::vector<double> sf((size_t)s->cols.nf_base() * N);
  std::vector<int32_t> si((size_t)s->cols.ni() * N);
  CK(cudaMemcpy(sf.data(), s->sf, sizeof(double) * sf.size(), cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(si.data(), s->si, sizeof(int32_t) * si.size(), cudaMemcpyDeviceToHost));
  for (int64_t i = 0; i < N; i++)
    state_from_columns(s->cols, sf.data(), si.data(), N, i, rob + i * R * 7, rhist + i * R * 3, rflag + i * R * 3,
                       ball + i * B * 8, step + i);
  return RR_OK;
}

int rr_goal_state(rr_sim *s, int32_t *alive_host, int32_t *score_host, int32_t *destroyed_host, int32_t *dwell_host) {
  if (!s) return fail(RR_E_INVALID, "null handle");
  if (!s->cfg.goal_scoring) return fail(RR_E_INVALID, "the handle was created without goal_scoring");
  ON_DEVICE(s->device);
  CK(cudaDeviceSynchronize());
  const int64_t N = s->N;
  const int B = s->cols.B;
  std::vector<int32_t> g((size_t)s->cols.G * N);
  CK(cudaMemcpy(g.data(), s->si + (size_t)s->cols.goal(0) * N, sizeof(int32_t) * g.size(), cudaMemcpyDeviceToHost));
  for (int64_t i = 0; i < N; i++) {
    int32_t r[4];
    goal_report((uint32_t)g[(size_t)0 * N + i], (uint32_t)g[(size_t)1 * N + i], B, r);
    if (alive_host) alive_host[i] = r[3];
    if (score_host) { score_host[i * 2] = r[0]; score_host[i * 2 + 1] = r[1]; }
    if (destroyed_host) destroyed_host[i] = r[2];
    if (dwell_host)
      for (int q = 0; q < 2 * B; q++) dwell_host[i * 2 * B + q] = g[(size_t)(2 + q) * N + i];
  }
  return RR_OK;
}

int rr_error_mask(rr_sim *s, uint32_t *err_host, int32_t clear) {
  if (!s || !err_host) return fail(RR_E_INVALID, "null argument");
  ON_DEVICE(s->device);
  CK(cudaDeviceSynchronize());
  int32_t *p = s->si + (size_t)s->cols.err() * s->N;
  CK(cudaMemcpy(err_host, p, sizeof(uint32_t) * s->N, cudaMemcpyDeviceToHost));
  if (clear) CK(cudaMemset(p, 0, sizeof(uint32_t) * s->N));
  return RR_OK;
}

int rr_last_naughty(rr_sim *s, int32_t *count_host) {
  if (!s || !count_host) return fail(RR_E_INVALID, "null argument");
  ON_DEVICE(s->device);
  CK(cudaDeviceSynchronize());
  CK(cudaMemcpy(count_host, s->si + (size_t)s->cols.naughty() * s->N, sizeof(int32_t) * s->N, cudaMemcpyDeviceToHost));
  return RR_OK;
}

int rr_get_stats(rr_sim *s, double *stats_host) {
  if (!s || !stats_host) return fail(RR_E_INVALID, "null argument");
  ON_DEVICE(s->device);
  CK(cudaDeviceSynchronize());
  CK(cudaMemcpy(stats_host, s->stats, sizeof(double) * RR_NUM_STATS, cudaMemcpyDeviceToHost));
  return RR_OK;
}

int rr_stats_device_ptr(rr_sim *s, double **p) {
  if (!s || !p) return fail(RR_E_INVALID, "null argument");
  *p = s->stats;
  return RR_OK;
}

int rr_clear_stats(rr_sim *s, void *stream) {
  if (!s) return fail(RR_E_INVALID, "null handle");
  ON_DEVICE(s->device);
  if (int jr = join_into(s, (cudaStream_t)stream)) return jr;
  CK(cudaMemsetAsync(s->stats, 0, sizeof(double) * RR_NUM_STATS, (cudaStream_t)stream));
  return RR_OK;
}

int rr_set_stats_buffer(rr_sim *s, double *stats_dev) {
  if (!s) return fail(RR_E_INVALID, "null handle");
  s->stats = stats_dev ? stats_dev : s->own_stats;
  return RR_OK;
}
