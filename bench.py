#!/usr/bin/env python
"""bench.py — env-steps/s of the RoboRugby step()/reset() hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--preset GAME|TRAIN] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json configs[2]): RoboRugbySimpleDuel-v2, 65 536 envs per GPU, shipped (GAME)
constants, uniformly random discrete actions for all four robots, fused launches of 32 env-steps
with in-kernel auto-reset.  One bench "step" = one fused launch = 65 536 x 32 env-steps per GPU.

  value    whole-job env-steps/s, inputs (actions) already resident in HBM, CUDA-event timed over the whole region
           (calls issued back to back; with the sub-batch pipeline, rr_set_pipeline, the groups of consecutive calls
           overlap), max over ranks, L2 flushed in front of every launch
  e2e      the same calls through the HOST-buffer C-ABI entry points rr_step_host_begin / _end (three calls in flight):
           actions copied host->device, observations/rewards/done written into pinned host memory and read by the
           caller after every call, all inside the timed region
  roofline HBM: algorithmic bytes per launch / measured kernel time vs MEASURED_PEAKS.json; `secondary` carries the
           ncu figures that actually bound the kernel (fp64 pipe, issue slots, SM busy) and the file they come from
  cpu_baseline  the C oracle (port of the reference algorithm, oracle/) on the host cores, N=1 only
  extras   k1: the same batch stepped ONE env-step per launch (env.step(), the call a policy-in-the-loop consumer
           makes); dqn: env-steps/s inside the vectorised DQN loop (BASELINE configs[4]); per_rank_ms_per_call (N > 1); single_launch: the same calls without the sub-batch pipeline

--impl reference times the reference algorithm's CPU implementation on the host cores (the C
oracle port; the Python reference itself cannot travel to the GPU box — its measured rate in the
build container is recorded in DESIGN.md).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# the tree may be read-only: no bytecode caches there, from this process or the oracle's timing subprocess
sys.dont_write_bytecode = True
os.environ["PYTHONDONTWRITEBYTECODE"] = "1"

ENV_ID = "RoboRugbySimpleDuel-v2"
ENVS_PER_GPU = 65536
FUSED = 32
PIPELINE = 128  # sub-batch groups (rr_set_pipeline): a group held back by its slowest env delays only its own next launch
# Figures from the committed `ncu --set full` captures of the committed kernels (profiles/, see PROFILE_SOURCE).  A bench
# call is 128 kernel launches over groups of blocks (sub-batch pipeline), which ncu cannot capture as one unit, so the
# captures are ONE WAVE of the same kernel: GAME 56 832 envs = 148 blocks of 384 threads x 32 steps (`--envs 56832
# --pipeline 1`), TRAIN 65 536 envs = 147 blocks of 448 threads.  dram__bytes_read.sum + dram__bytes_write.sum is reported
# as roofline.traffic per bench call (the GAME figure scaled by 65 536 / 56 832 envs); the pipe / issue / stall figures
# that bound the kernel as roofline.secondary (the path is not HBM-bound, DESIGN.md §4).  sm_busy_pipelined = sum of
# the block times / (148 SMs x time per call) of the pipelined run, instrumented build (profiles/r02_pipeline_block_chains.txt).
PROFILE_SOURCE = {"GAME": "profiles/r02_k_step_game_by_function.txt", "TRAIN": "profiles/r02_k_step_train_by_function.txt"}
NCU_TRAFFIC_BYTES = {"GAME": (136.85e6 + 1086.35e6) * 65536 / 56832, "TRAIN": 15.41e6 + 126.62e6}
NCU_SECONDARY = {
    "GAME": {"fp64_pipe_pct": 17.8, "issue_slots_busy_pct": 29.0, "warps_active_pct": 18.7, "sm_busy_frac_single_wave": 0.671,
             "sm_busy_pipelined": 0.944, "barrier_stall_per_issue": 2.45, "long_scoreboard_per_issue": 1.12,
             "threads_per_instruction": 21.8, "registers_per_thread": 168, "block": 384},
    "TRAIN": {"fp64_pipe_pct": 18.2, "issue_slots_busy_pct": 33.7, "warps_active_pct": 21.8, "sm_busy_frac_single_wave": 0.878,
              "barrier_stall_per_issue": 2.01, "long_scoreboard_per_issue": 0.91, "threads_per_instruction": 23.5,
              "registers_per_thread": 128, "block": 448},
}
KERNEL_NAME = {"GAME": "rr::k_step<rr::Launch<2, 2, 4, 4, 0, 0>, float>", "TRAIN": "rr::k_step<rr::Launch<1, 0, 1, 0, 0, 0>, float>"}
# The Python reference itself (unmodified, stub pygame/gym) cannot travel to the GPU box; its own rate, measured in the
# build container with oracle/time_reference.py (8 cores, one process per core), is recorded beside the port's.
PY_REFERENCE_NOTE = {"GAME": "Python reference (oracle/time_reference.py, build container, 8 cores): 123 env-steps/s (18.9 per core)",
                     "TRAIN": "Python reference (oracle/time_reference.py, build container, 8 cores): 4467 env-steps/s (657 per core)"}
METRIC = "env_steps_per_sec"
UNIT = "env-steps/s"
# --dump-outputs: the rows of a fixed sample of envs (np.random.default_rng(0), sorted), so that two builds can be compared
# output for output without writing the whole batch (65 536 envs x 32 steps of four outputs is ~110 MB)
DUMP_ENVS = 8192
DUMP_BYTES = 64_000_000


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured"
        except Exception:
            pass
    return 6650.0, "fallback"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu, self.rows, self._stop_evt, self.proc = gpu_index, [], threading.Event(), None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            for line in self.proc.stdout:
                if self._stop_evt.is_set():
                    break
                self.rows.append([x.strip() for x in line.split(",")])
        except Exception:
            pass

    def stop(self):
        self._stop_evt.set()
        if self.proc:
            self.proc.terminate()

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for n, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def run_reference(args, rank, world):
    """--impl reference: the reference algorithm on the host cores (C oracle port)."""
    if rank != 0:
        return
    from oracle import rr_oracle
    cores = os.cpu_count() or 1
    per_core = 4000 if args.preset == "GAME" else 120000  # ~2 s per bench step on each core
    vals, walls = [], []
    for it in range(args.warmup + args.steps):
        v, wall = rr_oracle.timed_rollout(args.preset, args.env_id, per_core, cores)
        if it >= args.warmup:
            vals.append(v); walls.append(wall)
    value = sum(vals) / len(vals)
    sample = f"{per_core} random-action env-steps per core x {cores} cores per bench step, C oracle (oracle/rr_oracle.c)"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * sum(walls) / len(walls), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args, world),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                         "note": PY_REFERENCE_NOTE[args.preset]},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }), flush=True)


def dqn_rate(dev, envs, steps, preset="TRAIN"):
    """env-steps/s inside the vectorised Training_DQN_pytorch loop (roborugby_b200/dqn.py): eps-greedy acting, env step,
    replay store and one learn() per step, all on the device."""
    import torch
    from roborugby_b200.dqn import VecDQNAgent, train
    from roborugby_b200.vec_env import RoboRugbyVecEnv
    env = RoboRugbyVecEnv(ENV_ID, envs, preset=preset, device=dev, seed=5, n_actions=1)
    agent = VecDQNAgent(env.obs_dim, batch_size=2500, max_mem_size=500000, device=dev, seed=1)
    train(env, agent, 10)  # warm-up (cuBLAS handles, allocator)
    out = train(env, agent, steps)
    env.close()
    return {"value": out["env_steps_per_s"], "unit": UNIT, "envs": envs, "steps": steps, "preset": preset,
            "transitions_stored": out["transitions"], "learn_every": 1, "batch_size": 2500,
            "note": "Training_DQN_pytorch.py:317-377 on the GPU VecEnv, K = 1 launches, nothing visits the host"}


def run_dqn(args, rank, world, local_rank):
    """--workload dqn: BASELINE configs[4] as its own line (rank 0 only; the loop does not shard)."""
    if rank != 0:
        return
    import torch
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    r = dqn_rate(dev, envs=args.envs, steps=max(args.steps, 30))
    print(json.dumps({"metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": 1, "steps": r["steps"], "warmup": 10,
                      "ms_per_step": 1e3 * r["envs"] / r["value"], "higher_is_better": True, "scaling": "weak",
                      "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                      "config": {"workload": f"Training_DQN_pytorch loop on {ENV_ID}, TRAIN preset, {r['envs']} envs, learn() every "
                                             "step, batch 2500 (BASELINE configs[4])"}, "dqn": r}), flush=True)


def dump_outputs(path, outs, n_envs):
    """Write the outputs of one step_k call (obs_h, obs_g [K, N, D], rew [K, N, 2], done [K, N]) as float32 .npy files,
    restricted to the sampled envs."""
    import numpy as np
    import torch
    names = ("obs_h", "obs_g", "rew", "done")
    per_env = 4 * sum(x[:, :1].numel() for x in outs)
    n = max(1, min(n_envs, DUMP_ENVS, DUMP_BYTES // per_env))
    idx = np.sort(np.random.default_rng(0).choice(n_envs, n, replace=False))
    sel = torch.as_tensor(idx, device=outs[0].device)
    os.makedirs(path, exist_ok=True)
    for name, x in zip(names, outs):
        if x.numel():   # (no observation arrays for an observer-less env id)
            np.save(os.path.join(path, name + ".npy"), x[:, sel].float().cpu().numpy())


def workload_config(args, world):
    return {"workload": f"{args.env_id} {args.preset} preset, {args.envs} envs/GPU x {world} GPU, random "
                        f"{'continuous thrust' if args.env_id == 'RoboRugby-v0' else 'discrete'} actions, "
                        f"{args.fused} fused env-steps per launch, auto-reset (BASELINE configs[{3 if args.env_id == 'RoboRugby-v0' else 2}])",
            "env_id": args.env_id, "preset": args.preset, "envs_per_gpu": args.envs, "fused_steps": args.fused,
            "parallelism": f"env-shard x{world} (no data-path collective)", "pipeline_groups": args.pipeline,
            "l2": "flushed: every launch is preceded, on its own stream, by a memset of its share of a 256 MB buffer "
                  "(rr_set_flush_buffer), inside the timed region",
            "strict_reset": not args.relaxed_reset, "squeeze_memo": not args.no_squeeze_memo, "out_dtype": "float32"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--preset", default="GAME", choices=["GAME", "TRAIN"])
    ap.add_argument("--envs", type=int, default=ENVS_PER_GPU)
    ap.add_argument("--fused", type=int, default=FUSED)
    ap.add_argument("--pipeline", type=int, default=PIPELINE, help="sub-batch groups stepped on their own streams "
                    "(rr_set_pipeline); 1 = one stream-ordered launch per call, the round-1 measurement")
    ap.add_argument("--env-id", default=ENV_ID, help="another registered id, e.g. RoboRugby-v0 (the full game: continuous "
                    "thrust pairs for all robots, BASELINE configs[3]); the default is the workload the metric is quoted on")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--relaxed-reset", action="store_true", help="strict_reset=0: two extra rejection rules in the reset "
                    "placement (default: the reference's own placement)")
    ap.add_argument("--no-squeeze-memo", action="store_true", help="A/B: recompute every pinned-ball frame (RR_FLAG_NO_SQUEEZE_MEMO)")
    ap.add_argument("--no-extras", action="store_true", help="skip the K = 1 and DQN-loop extras")
    ap.add_argument("--workload", default="rollout", choices=["rollout", "dqn"], help="dqn: BASELINE configs[4], the "
                    "Training_DQN_pytorch loop on the GPU VecEnv (TRAIN constants, as the reference script requires)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed calls, write what the last one returned "
                    "(obs_h, obs_g, rew, done of a fixed sample of rank 0's envs, float32) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.workload == "dqn":
        run_dqn(args, rank, world, local_rank)
        return

    # CPU baseline first (rank 0, N=1 only), before this process touches CUDA
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import rr_oracle
        cores = os.cpu_count() or 1
        per_core = 30000 if args.preset == "GAME" else 800000  # ~12 s of CPU work on every core
        v, wall = rr_oracle.timed_rollout(args.preset, args.env_id, per_core, cores)
        cpu_baseline = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                        "sample": f"{per_core} random-action env-steps per core on {cores} cores ({wall:.1f} s), "
                                  f"C oracle port of the reference algorithm, same env id and preset",
                        "note": PY_REFERENCE_NOTE[args.preset]}

    import torch
    import torch.distributed as dist
    from roborugby_b200 import shard_envs
    from roborugby_b200.vec_env import RoboRugbyVecEnv

    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    N, K = args.envs, args.fused
    total = N * world
    n_local, offset = shard_envs(total, rank, world)
    env = RoboRugbyVecEnv(args.env_id, n_local, preset=args.preset, device=dev, seed=2026, env_offset=offset,
                          time_limit=True, auto_reset=True, out_dtype=torch.float32, strict_reset=not args.relaxed_reset,
                          flags=1 if args.no_squeeze_memo else 0)
    R, D = env.num_robots, env.obs_dim
    g = torch.Generator(device=dev).manual_seed(1 + rank)
    n_sets = 4  # rotate pre-generated action sets so consecutive launches differ
    if env.discrete:
        A = 1 if args.env_id == "RoboRugbySimple-v0" else R
        acts = [torch.randint(0, 8, (K, n_local, A), generator=g, dtype=torch.uint8, device=dev) for _ in range(n_sets)]
    else:  # GameEnv.step: one (left, right) thrust pair per robot, rounded to {-1, 0, 1} by the env (RR_Robot.py:100-102)
        acts = [(torch.rand((K, n_local, 2 * R), generator=g, device=dev) * 2.9 - 1.45).float() for _ in range(n_sets)]
    acts_host = [a.cpu().pin_memory() for a in acts]
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # desynchronise episode phases so resets are spread over launches like a long-running job
    st = env.get_state()
    import numpy as np
    st["step"][:] = (np.arange(n_local) * 7919) % max(env.max_episode_steps - 1, 1)
    env.set_state(st)

    env.set_pipeline(args.pipeline)
    if not os.environ.get("RR_BENCH_NO_FLUSH"):
        env.set_flush_buffer(flush)
    for w in range(args.warmup):
        env.step_k(acts[w % n_sets], K)
    barrier()

    # ---------------- device-resident timing (value) ----------------
    # The calls are issued back to back; with a sub-batch pipeline the groups of call n + 1 start as their own group of
    # call n finishes (no join in between), so the whole region is timed with one event pair on the issuing stream:
    # start before the first call, end after the join behind the last one.
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = env.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_wall0 = time.perf_counter()
    e0.record()
    for s in range(args.steps):
        outs = env.step_k(acts[s % n_sets], K, join=False)
    env.join()
    e1.record()
    barrier()
    t_wall = time.perf_counter() - t_wall0
    if args.dump_outputs and rank == 0:   # before the calls below reuse the output buffers
        dump_outputs(args.dump_outputs, outs, n_local)
    launches = env.launch_count - launches0
    my_ms = e0.elapsed_time(e1)
    kernel_ms = [my_ms / args.steps] * args.steps
    t = torch.tensor([my_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    max_ms = float(t.item())
    value = total * K * args.steps / (max_ms * 1e-3)
    per_rank_ms = [my_ms / args.steps]
    if world > 1:  # per-rank mean time per call: the max over ranks is the shard with the slowest envs (no collective inside)
        allms = [torch.zeros(1, dtype=torch.float64, device=dev) for _ in range(world)]
        dist.all_gather(allms, torch.tensor([my_ms / args.steps], dtype=torch.float64, device=dev))
        per_rank_ms = [float(x.item()) for x in allms]

    # ---------------- end-to-end through the host-buffer C-ABI entry points ----------------
    # rr_step_host_begin / _end with three calls in flight: actions travel host->device, the kernels write the result rows
    # straight into pinned host memory, and the caller reads every call's result on the host before it ends the next one.
    e2e_steps = max(3, min(args.steps, 30))
    depth = 3  # calls in flight (of at most RR_HOST_TICKETS = 4)
    for w in range(4):  # allocates the sets of pinned result buffers + the device staging of all four tickets
        env.step_host_end(env.step_host_begin(acts_host[w % n_sets], K, w % depth))
    barrier()
    t0 = time.perf_counter()
    pending = [env.step_host_begin(acts_host[s % n_sets], K, s % depth) for s in range(min(depth - 1, e2e_steps))]
    for s in range(e2e_steps):
        nx = s + depth - 1
        if nx < e2e_steps:
            pending.append(env.step_host_begin(acts_host[nx % n_sets], K, nx % depth))
        out = env.step_host_end(pending.pop(0))
        _ = float(out["rew"][K - 1, 0, 0])  # the caller reads the step's result on the host
        if os.environ.get("RR_BENCH_TRACE"):
            print("e2e call", s, round((time.perf_counter() - t0) * 1e3, 2), file=sys.stderr)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = total * K * e2e_steps / float(t.item())
    act_bytes = acts[0].element_size() * acts[0].shape[-1]  # per env-step
    h2d = K * n_local * act_bytes
    d2h = K * n_local * (2 * D * 4 + 2 * 4 + 1)
    sampler.stop()
    clocks = sampler.summary()
    per_rank_clocks = None
    if world > 1:  # every rank samples its own GPU: a slower rank is usually a GPU that clocks lower under the fp64 load
        mine = torch.tensor([float(clocks["sm_mhz"] or 0.0), float(len(clocks["reasons"]))], dtype=torch.float64, device=dev)
        allc = [torch.zeros(2, dtype=torch.float64, device=dev) for _ in range(world)]
        dist.all_gather(allc, mine)
        per_rank_clocks = [float(x[0].item()) for x in allc]

    stats = env.reduce_stats()  # the one optional collective: 64-byte all-reduce of episode statistics
    err_envs = int((env.error_mask() != 0).sum())
    local_stats = env.get_stats()
    state_bytes = env.state_bytes_per_env

    # ---------------- extras: one env-step per launch (env.step()), DQN loop ----------------
    extras = {"per_rank_ms_per_call": per_rank_ms}
    if per_rank_clocks is not None:
        extras["per_rank_sm_mhz_median"] = per_rank_clocks
    if not args.no_extras:
        # (a) the same calls one stream-ordered launch at a time (no pipeline): the round-1 definition of `value`
        env.set_pipeline(1)
        for w in range(2):
            env.step_k(acts[w % n_sets], K)
        barrier()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(10)]
        for s, (a0, a1) in enumerate(ev):
            a0.record(); env.step_k(acts[s % n_sets], K); a1.record()
        barrier()
        single_ms = [a0.elapsed_time(a1) for a0, a1 in ev]
        t = torch.tensor([sum(single_ms)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        extras["single_launch"] = {"value": total * K * len(ev) / (float(t.item()) * 1e-3), "unit": UNIT,
                                   "ms_per_launch": float(t.item()) / len(ev), "launches": len(ev),
                                   "note": "pipeline_groups = 1: every call is one kernel over the whole batch and ends with "
                                           "its slowest env; per-launch CUDA events, flush memset inside"}
        env.set_flush_buffer(None)
        # (b) one env-step per call (env.step()), back to back, 16 groups
        env.set_pipeline(min(16, args.pipeline))
        n1 = 256
        a1 = [a[j:j + 1] for a in acts for j in range(K)]  # the same action stream as above, one row per launch
        for w in range(5):
            env.step_k(a1[w % len(a1)], 1)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for s in range(n1):
            env.step_k(a1[(5 + s) % len(a1)], 1, join=False)
        env.join()
        e1.record()
        barrier()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        extras["k1"] = {"value": total * n1 / (float(t.item()) * 1e-3), "unit": UNIT, "launches": n1,
                        "ms_per_launch": float(t.item()) / n1, "pipeline_groups": min(16, args.pipeline),
                        "note": "one env-step per call (RoboRugbyVecEnv.step / GameEnv.step, RR_EnvBase.py:260), "
                                "actions resident, calls issued back to back, no L2 flush"}
        if rank == 0 and world == 1:
            env.close()   # (its buffers are not needed any more)
            extras["dqn"] = dqn_rate(dev, envs=65536, steps=40)

    if rank == 0:
        peak, peak_src = _peaks()
        S = state_bytes
        q = 2.0 * S / K + act_bytes + 2 * D * 4 + 2 * 4 + 1  # algorithmic bytes per env-step (DESIGN.md §4)
        bytes_per_launch = q * n_local * K
        avg_kernel_s = (sum(kernel_ms) / len(kernel_ms)) * 1e-3
        achieved = bytes_per_launch / avg_kernel_s / 1e9
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": max_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": workload_config(args, world),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": e2e_steps, "calls_in_flight": 3},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": (NCU_TRAFFIC_BYTES[args.preset] if (args.envs, args.fused) == (ENVS_PER_GPU, FUSED)
                                     else None),
                         "traffic_source": PROFILE_SOURCE[args.preset] + " (dram bytes read + written by one wave of the kernel, "
                                           "scaled to the envs of one bench call)",
                         "achieved_note": "algorithmic bytes of one bench call / (timed region / calls): the calls overlap "
                                          "(sub-batch pipeline), so this is the sustained rate, not one launch alone",
                         "algorithmic_bytes_per_launch": bytes_per_launch, "peak_source": peak_src, "bytes_per_env_step": q, "state_bytes": S,
                         "kernel": KERNEL_NAME[args.preset],
                         "secondary": dict(NCU_SECONDARY[args.preset], source=PROFILE_SOURCE[args.preset]),
                         "note": "path is fp64-issue / latency bound, not HBM bound (DESIGN.md §4)"},
            "clocks": clocks,
            "episode_stats": {k: stats[k] for k in ("episodes", "mean_return_happy", "mean_return_grumpy", "mean_length",
                                                    "naughty", "errors", "steps")},
            "error_envs": err_envs,
            "errors_per_million_env_steps": 1e6 * stats["errors"] / max(stats["steps"], 1.0),
            "squeeze_replays_rank0": local_stats.get("squeeze_replays"),
            "wall_s_timed_region": t_wall,
            "extras": extras,
        }
        if cpu_baseline is not None:
            line["cpu_baseline"] = cpu_baseline
        print(json.dumps(line), flush=True)
    env.close()   # (idempotent)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
