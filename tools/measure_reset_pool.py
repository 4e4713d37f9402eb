"""Cost of auto-reset from a reset pool (rr_step_pool) at the benchmark configuration.

RoboRugbySimpleDuel-v2, 65 536 envs, K = 32 env-steps per launch, 128 sub-batch pipeline groups, bench.py's
desynchronised episode phases; GAME and TRAIN.  Three arms, each on its own handle with the same starting state:
  info  rr_step_info without a pool (step_k(final_info=True)): every reset is a random placement;
  p0    the pool kernel with p = 0: the pool draw runs on every reset, every reset is still a random placement;
  p1    the pool kernel with p = 1: every reset loads a row (uniform over 1 024 rows saved mid-episode).
Rounds alternate the arms (the order reverses every round) so that clock and neighbour noise fall on all of them; a
round times `--calls` back-to-back launches with one CUDA event pair after a join.  Prints one JSON line: per preset and
arm the median env-steps/s with its min and max over the rounds, the resets per launch (counted on one extra launch),
the ratios to `info`, and the GPU name and power limit.

    python tools/measure_reset_pool.py [--rounds 7] [--calls 20]
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
    from roborugby_b200.vec_env import ResetPool, RoboRugbyVecEnv

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
                           rounds=args.rounds, calls_per_round=args.calls, pool_rows=1024),
               gpu=gpu_info(), unit="env-steps/s")
    for preset in args.presets:
        envs = {a: RoboRugbyVecEnv("RoboRugbySimpleDuel-v2", N, preset=preset, device="cuda:0", seed=2026,
                                   pipeline=args.pipeline) for a in ("info", "p0", "p1")}
        e0 = envs["info"]
        st = e0.get_state()
        st["step"][:] = (np.arange(N) * 7919) % max(e0.max_episode_steps - 1, 1)   # bench.py's desynchronisation
        e0.set_state(st)
        rows0 = e0.save_states()
        for e in envs.values():
            e.load_states(rows0)
        pool_rows = rows0[torch.randperm(N, device=rows0.device)[:1024]].contiguous()   # mid-episode rows
        pools = {"info": None, "p0": ResetPool(pool_rows, p=0.0), "p1": ResetPool(pool_rows, p=1.0)}
        g = torch.Generator(device="cuda").manual_seed(5)
        acts = torch.randint(0, 8, (K, N, e0.action_dim), generator=g, device="cuda", dtype=torch.uint8)

        def launch(arm):
            if pools[arm] is None:
                return envs[arm].step_k(acts, K, join=False, final_info=True)
            return envs[arm].step_k(acts, K, join=False, reset_pool=pools[arm])

        def run(arm, calls):
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            ev0.record()
            for _ in range(calls):
                launch(arm)
            envs[arm].join()
            ev1.record()
            torch.cuda.synchronize()
            return N * K * calls / (ev0.elapsed_time(ev1) * 1e-3)

        for arm in envs:  # warm-up
            run(arm, 3)
        rates = {arm: [] for arm in envs}
        for r in range(args.rounds):
            order = list(envs) if r % 2 == 0 else list(envs)[::-1]
            for arm in order:
                rates[arm].append(run(arm, args.calls))
        res = {}
        for arm in envs:
            o = launch(arm)
            envs[arm].join()
            done = int(o[3].sum())
            pool_resets = int((o[4]["reset_slot"] >= 0).sum()) if pools[arm] is not None else 0
            v = rates[arm]
            res[arm] = dict(median=float(np.median(v)), min=float(min(v)), max=float(max(v)), resets_per_launch=done,
                            pool_resets_per_launch=pool_resets)
        for arm in ("p0", "p1"):
            res[arm]["over_info"] = res[arm]["median"] / res["info"]["median"]
        out[preset] = res
        for e in envs.values():
            e.close()
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
