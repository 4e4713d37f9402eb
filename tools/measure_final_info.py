"""Cost of rr_step_info's outputs (terminal observations of done rows, RR_ROW_* flags) at the BASELINE configuration.

RoboRugbySimpleDuel-v2, GAME constants, 65 536 envs, K = 32 fused env-steps per call, float32 outputs, auto-reset, episode
phases desynchronised as bench.py does, sub-batch pipeline of 128 groups, L2 flushed in front of every launch (a 256 MB
buffer, rr_set_flush_buffer).  Two handles with the same seed step the same actions: one through rr_step (step_k), one
through rr_step_info (step_k(final_info=True)).  Rounds alternate the two so that clock and neighbour noise fall on both;
each round times `--calls` back-to-back calls with one CUDA event pair.  Prints one JSON line with both rates (env-steps/s,
median and spread over rounds), the GPU name and its power limit.

    python tools/measure_final_info.py [--rounds 6] [--calls 20]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = (x.strip() for x in q.split(","))
        return dict(name=name, power_limit=power, max_sm_clock=clock)
    except Exception as e:  # the rates stand without it; say why it is missing
        return dict(error=str(e))


def main():
    import numpy as np
    import torch
    from roborugby_b200.vec_env import RoboRugbyVecEnv

    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--fused", type=int, default=32)
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--pipeline", type=int, default=128)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a GPU"
    N, K = args.envs, args.fused
    envs = {name: RoboRugbyVecEnv("RoboRugbySimpleDuel-v2", N, preset="GAME", device="cuda:0", seed=2026,
                                  time_limit=True, auto_reset=True, out_dtype=torch.float32, strict_reset=True,
                                  pipeline=args.pipeline) for name in ("rr_step", "rr_step_info")}
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")
    for env in envs.values():
        st = env.get_state()
        st["step"][:] = (np.arange(N) * 7919) % max(env.max_episode_steps - 1, 1)
        env.set_state(st)
        env.set_flush_buffer(flush)
    g = torch.Generator(device="cuda").manual_seed(1)
    acts = [torch.randint(0, 8, (K, N, 4), generator=g, dtype=torch.uint8, device="cuda") for _ in range(4)]

    def run(name, calls):
        env, info = envs[name], name == "rr_step_info"
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for s in range(calls):
            env.step_k(acts[s % 4], K, join=False, final_info=info)
        env.join()
        e1.record()
        torch.cuda.synchronize()
        return N * K * calls / (e0.elapsed_time(e1) * 1e-3)

    for name in envs:  # warm-up: modules, buffers
        run(name, 3)
    rates = {name: [] for name in envs}
    for r in range(args.rounds):
        for name in (("rr_step", "rr_step_info") if r % 2 == 0 else ("rr_step_info", "rr_step")):
            rates[name].append(run(name, args.calls))
    out = dict(config=dict(env_id="RoboRugbySimpleDuel-v2", preset="GAME", envs=N, fused=K, out="float32",
                           pipeline=args.pipeline, rounds=args.rounds, calls_per_round=args.calls, l2="flushed"),
               gpu=gpu_info(), unit="env-steps/s")
    for name, v in rates.items():
        out[name] = dict(median=float(np.median(v)), min=float(min(v)), max=float(max(v)), rounds=[float(x) for x in v])
    out["info_over_plain"] = out["rr_step_info"]["median"] / out["rr_step"]["median"]
    print(json.dumps(out), flush=True)
    for env in envs.values():
        env.close()


if __name__ == "__main__":
    main()
