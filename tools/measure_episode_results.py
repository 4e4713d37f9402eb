"""Cost of the per-row episode results (rr_step_episodes) at the benchmark configuration.

RoboRugbySimpleDuel-v2, 65 536 envs, K = 32 env-steps per launch, 128 sub-batch pipeline groups, bench.py's
desynchronised episode phases, L2 flushed in front of every launch (a 256 MB buffer, rr_set_flush_buffer); GAME and
TRAIN.  Two arms, each on its own handle with the same starting state and actions:
  info      rr_step_info (step_k(final_info=True));
  episodes  rr_step_episodes with every output on (step_k(episode_info=True)): the same kernel variant plus the fp64
            returns and the lengths of every row (the goal words need goal scoring, which this env id has off).
Rounds alternate the arms (the order reverses every round) so that clock and neighbour noise fall on both; a round
times `--calls` back-to-back launches with one CUDA event pair after a join.  Prints one JSON line: per preset and arm
the median env-steps/s with its min and max over the rounds, the ratio episodes / info, the episodes counted per
launch, and the GPU name and power limit.

    python tools/measure_episode_results.py [--rounds 7] [--calls 20]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

from tools.measure_state_rows import gpu_info  # noqa: E402


def main():
    import numpy as np
    import torch
    from roborugby_b200.vec_env import RoboRugbyVecEnv

    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--k", type=int, default=32)
    ap.add_argument("--pipeline", type=int, default=128)
    ap.add_argument("--presets", nargs="+", default=["GAME", "TRAIN"])
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--calls", type=int, default=20)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a GPU"
    N, K = args.envs, args.k
    out = dict(config=dict(env_id="RoboRugbySimpleDuel-v2", envs=N, k_steps=K, pipeline=args.pipeline,
                           rounds=args.rounds, calls_per_round=args.calls, l2="flushed"),
               gpu=gpu_info(), unit="env-steps/s")
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")
    for preset in args.presets:
        envs = {a: RoboRugbyVecEnv("RoboRugbySimpleDuel-v2", N, preset=preset, device="cuda:0", seed=2026,
                                   pipeline=args.pipeline) for a in ("info", "episodes")}
        e0 = envs["info"]
        st = e0.get_state()
        st["step"][:] = (np.arange(N) * 7919) % max(e0.max_episode_steps - 1, 1)   # bench.py's desynchronisation
        e0.set_state(st)
        rows0 = e0.save_states()
        for e in envs.values():
            e.load_states(rows0)
            e.set_flush_buffer(flush)
        g = torch.Generator(device="cuda").manual_seed(5)
        acts = [torch.randint(0, 8, (K, N, e0.action_dim), generator=g, device="cuda", dtype=torch.uint8)
                for _ in range(4)]

        def launch(arm, s):
            return envs[arm].step_k(acts[s % 4], K, join=False, final_info=True, episode_info=arm == "episodes")

        def run(arm, calls):
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            ev0.record()
            for s in range(calls):
                launch(arm, s)
            envs[arm].join()
            ev1.record()
            torch.cuda.synchronize()
            return N * K * calls / (ev0.elapsed_time(ev1) * 1e-3)

        for arm in envs:  # warm-up: modules, buffers
            run(arm, 3)
        rates = {arm: [] for arm in envs}
        for r in range(args.rounds):
            order = list(envs) if r % 2 == 0 else list(envs)[::-1]
            for arm in order:
                rates[arm].append(run(arm, args.calls))
        res = {}
        for arm in envs:
            v = rates[arm]
            res[arm] = dict(median=float(np.median(v)), min=float(min(v)), max=float(max(v)), rounds=[float(x) for x in v])
        o = launch("episodes", 0)
        envs["episodes"].join()
        res["episodes"]["episodes_per_launch"] = int((o[4]["episode_length"] >= 0).sum())
        res["episodes_over_info"] = res["episodes"]["median"] / res["info"]["median"]
        out[preset] = res
        for e in envs.values():
            e.close()
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
