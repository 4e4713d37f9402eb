"""Cost of saving and loading every env's state row (rr_save_states / rr_load_states) against a plain device copy.

RoboRugbySimpleDuel-v2, GAME constants (1104-byte rows), at 65 536 and 131 072 envs.  For each size one handle saves all
envs into a row tensor and loads them back; the yardstick is a device-to-device copy of the same number of bytes (torch
copy_, a cudaMemcpyAsync).  Rounds alternate the three so that clock and neighbour noise fall on all of them; each round
times `--calls` back-to-back calls with one CUDA event pair.  The L2 is not flushed between calls: a call reads and writes
72 MB each at 65 536 envs, together more than the 126 MB L2, and 145 MB each at 131 072.  Prints one JSON line: per size and
operation the median time per call, its spread, the achieved GB/s (bytes read + bytes written), the ratio to the copy, and
the GPU name and power limit.

    python tools/measure_state_rows.py [--rounds 7] [--calls 50]
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
    except Exception as e:  # the times stand without it; say why it is missing
        return dict(error=str(e))


def main():
    import numpy as np
    import torch
    from roborugby_b200.vec_env import RoboRugbyVecEnv

    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, nargs="+", default=[65536, 131072])
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--calls", type=int, default=50)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a GPU"
    out = dict(config=dict(env_id="RoboRugbySimpleDuel-v2", preset="GAME", rounds=args.rounds, calls_per_round=args.calls),
               gpu=gpu_info(), unit="ms per call")
    for N in args.envs:
        env = RoboRugbyVecEnv("RoboRugbySimpleDuel-v2", N, preset="GAME", device="cuda:0", seed=2026)
        rows = env.save_states()
        src, dst = torch.empty_like(rows), torch.empty_like(rows)
        ops = {"save": lambda: env.save_states(out=rows), "load": lambda: env.load_states(rows),
               "copy": lambda: dst.copy_(src)}

        def run(op, calls):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(calls):
                ops[op]()
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / calls

        for op in ops:  # warm-up
            run(op, 5)
        t = {op: [] for op in ops}
        for r in range(args.rounds):
            order = list(ops) if r % 2 == 0 else list(ops)[::-1]
            for op in order:
                t[op].append(run(op, args.calls))
        nbytes = rows.numel()
        res = dict(row_bytes=env.state_row_bytes, bytes_each_way=nbytes)
        copy_ms = float(np.median(t["copy"]))
        for op, v in t.items():
            ms = float(np.median(v))
            res[op] = dict(median_ms=ms, min_ms=float(min(v)), max_ms=float(max(v)), gb_per_s=2 * nbytes / (ms * 1e-3) / 1e9,
                           over_copy=ms / copy_ms)
        out[f"envs_{N}"] = res
        env.close()
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
