#!/usr/bin/env python
"""DQN on RoboRugbySimpleDuel-v2 (TRAIN preset, the setting Training_DQN_pytorch.py:233-234 requires) with the GPU VecEnv
feeding torch tensors end to end.  Prints one JSON line with env-steps/s inside the training loop.

    python examples/train_dqn_vec.py --envs 4096 --steps 300
"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def main():
    import torch
    from roborugby_b200.dqn import VecDQNAgent, train
    from roborugby_b200.vec_env import RoboRugbyVecEnv
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--env-id", default="RoboRugbySimpleDuel-v2")
    ap.add_argument("--batch", type=int, default=300 * 8 + 100)  # max_episode_steps * 8 + 100 (:257)
    ap.add_argument("--learn-every", type=int, default=1)
    a = ap.parse_args()
    env = RoboRugbyVecEnv(a.env_id, a.envs, preset="TRAIN", device="cuda:0", seed=1, n_actions=1)
    agent = VecDQNAgent(env.obs_dim, n_actions=8, batch_size=a.batch, device="cuda:0")
    train(env, agent, 20, a.learn_every)  # warm-up (cuBLAS handles, allocator)
    env.clear_stats()
    out = train(env, agent, a.steps, a.learn_every, log_every=50, episode_returns=True)
    # the reference's per-episode line (Training_DQN_pytorch.py:364-371), for the last episode that ended
    rets, avg = out.pop("episode_returns"), out.pop("avg_return_100")
    out.pop("avg_return_100_grumpy")
    out["episodes_ended"] = len(rets)
    if len(rets):
        out["avg_return_100"] = float(avg[-1])
        print(f"episode {len(rets) - 1} score {float(rets[-1, 0]):.2f} average score {float(avg[-1]):.2f}",
              file=sys.stderr)
    out["config"] = vars(a)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
