"""Vectorised DQN on top of RoboRugbyVecEnv (BASELINE.json config 5; SURVEY.md §8f row 1).

Mirror of the reference's agent (Training_DQN_pytorch.py:25-197) with everything on the GPU:

    reference (one env, numpy replay on the host)            here (N envs, torch replay on the device)
    DeepQNetwork obs -> 256 -> 256 -> n_actions  :25-67       same module (torch.nn; library GEMMs are fine here:
                                                             the hot path of this repo is the env, not this MLP)
    store_transition(s, a, r, s_, done)          :119-128     store(s, a, r, s_, done) for N transitions at once
    main loop: happy AND grumpy transition       :317-377     train(): both teams' transitions stored per step, happy
      stored per step, only the happy action                  first; only the happy action applied (drive_grumpy=True
      applied (:343)                                          also applies the grumpy one)
    choose_action: eps-greedy, one forward       :130-141     choose_actions(obs [N, D]) -> uint8 [N]
    learn(): uniform batch without replacement,  :143-189     learn(): identical target r + gamma * max Q_target(s_)
      q_next[terminal] = 0, MSE, Adam,                        (terminal rows zeroed), MSE, Adam, hard target copy
      hard target copy every target_update_freq               whenever mem_cntr crosses a multiple of target_update_freq,
      stored transitions, eps *= eps_dec                      eps <- max(eps * eps_dec, eps_end) per learn()

No observation, action or reward ever visits the host: the env writes torch tensors, the agent
reads them (removes the round trip at :138-141, :166-170 of the reference).
"""
import copy

import torch
import torch.nn as nn
import torch.nn.functional as F


class DeepQNetwork(nn.Module):
    """Training_DQN_pytorch.py:25-61."""

    def __init__(self, input_dim, fc1_dims=256, fc2_dims=256, n_actions=8):
        super().__init__()
        self.fc1 = nn.Linear(input_dim, fc1_dims)
        self.fc2 = nn.Linear(fc1_dims, fc2_dims)
        self.fc3 = nn.Linear(fc2_dims, n_actions)

    def forward(self, state):
        x = F.relu(self.fc1(state.float()))
        x = F.relu(self.fc2(x))
        return self.fc3(x)


class VecDQNAgent:
    def __init__(self, input_dim, n_actions=8, gamma=0.99, epsilon=1.0, lr=5e-4, batch_size=2500,
                 max_mem_size=500000, eps_end=0.2, eps_dec=0.999997, fc1_dims=256, fc2_dims=256,
                 target_update_freq=100000, device="cuda:0", seed=0):
        self.device = torch.device(device)
        self.gamma, self.epsilon, self.eps_end, self.eps_dec = gamma, epsilon, eps_end, eps_dec
        self.n_actions, self.batch_size, self.mem_size = n_actions, int(batch_size), int(max_mem_size)
        self.target_update_freq = int(target_update_freq)
        self.mem_cntr = 0
        self._last_target_epoch = 0
        self.gen = torch.Generator(device=self.device).manual_seed(seed)
        torch.manual_seed(seed)
        self.Q_eval = DeepQNetwork(input_dim, fc1_dims, fc2_dims, n_actions).to(self.device)
        self.Q_target = copy.deepcopy(self.Q_eval)
        self.optimizer = torch.optim.Adam(self.Q_eval.parameters(), lr=lr)
        d = self.device
        self.state_memory = torch.zeros(self.mem_size, input_dim, dtype=torch.float32, device=d)
        self.new_state_memory = torch.zeros(self.mem_size, input_dim, dtype=torch.float32, device=d)
        self.action_memory = torch.zeros(self.mem_size, dtype=torch.int64, device=d)
        self.reward_memory = torch.zeros(self.mem_size, dtype=torch.float32, device=d)
        self.terminal_memory = torch.zeros(self.mem_size, dtype=torch.bool, device=d)

    # -- replay ------------------------------------------------------------------------------
    def store(self, state, action, reward, state_, done):
        """N transitions into the ring (Training_DQN_pytorch.py:119-128, vectorised)."""
        n = state.shape[0]
        idx = (self.mem_cntr + torch.arange(n, device=self.device)) % self.mem_size
        self.state_memory[idx] = state.float()
        self.new_state_memory[idx] = state_.float()
        self.action_memory[idx] = action.long()
        self.reward_memory[idx] = reward.float()
        self.terminal_memory[idx] = done.bool()
        self.mem_cntr += n

    # -- acting ------------------------------------------------------------------------------
    @torch.no_grad()
    def choose_actions(self, obs, epsilon_override=None):
        """eps-greedy for every env (:130-141); returns uint8 [N]."""
        eps = self.epsilon if epsilon_override is None else epsilon_override
        n = obs.shape[0]
        greedy = torch.argmax(self.Q_eval(obs), dim=1)
        rand = torch.randint(0, self.n_actions, (n,), device=self.device, generator=self.gen)
        explore = torch.rand(n, device=self.device, generator=self.gen) <= eps
        return torch.where(explore, rand, greedy).to(torch.uint8)

    # -- learning ----------------------------------------------------------------------------
    def td_target(self, reward, new_state, terminal):
        """reward + gamma * max_a Q_target(s_, a) with terminal rows zeroed (:172-176)."""
        with torch.no_grad():
            q_next = self.Q_target(new_state)
            q_next = torch.where(terminal.unsqueeze(1), torch.zeros_like(q_next), q_next)
            return reward + self.gamma * q_next.max(dim=1)[0]

    def learn(self):
        if self.mem_cntr < self.batch_size:  # :144-147
            return None
        max_mem = min(self.mem_size, self.mem_cntr)
        batch = torch.randperm(max_mem, device=self.device, generator=self.gen)[:self.batch_size]  # replace=False
        s, s_ = self.state_memory[batch], self.new_state_memory[batch]
        a, r, t = self.action_memory[batch], self.reward_memory[batch], self.terminal_memory[batch]
        self.optimizer.zero_grad(set_to_none=True)
        q_eval = self.Q_eval(s).gather(1, a.unsqueeze(1)).squeeze(1)
        loss = F.mse_loss(q_eval, self.td_target(r, s_, t))
        loss.backward()
        self.optimizer.step()
        epoch = self.mem_cntr // self.target_update_freq  # hard copy every target_update_freq transitions (:185-187)
        if epoch != self._last_target_epoch:
            self._last_target_epoch = epoch
            self.Q_target.load_state_dict(self.Q_eval.state_dict())
        self.epsilon = max(self.epsilon * self.eps_dec, self.eps_end)  # :189
        return loss.detach()


def _running_mean(x, n=100):
    """np.mean(scores[-100:]) after each episode (Training_DQN_pytorch.py:364-371), for every prefix of x."""
    c = torch.cat((torch.zeros(1, dtype=x.dtype), x.cumsum(0)))
    i = torch.arange(1, x.numel() + 1)
    lo = (i - n).clamp(min=0)
    return (c[i] - c[lo]) / (i - lo)


def train(env, agent, n_steps, learn_every=1, log_every=0, drive_grumpy=False, episode_returns=False):
    """The reference's main loop (Training_DQN_pytorch.py:317-377) for N envs in lockstep.

    Per iteration, exactly as the reference does per env: an eps-greedy action for the happy observation (:333-336)
    and, when the env has grumpy robots, one for the grumpy observation (:338-339); `env.step([action])` (:343 — the
    reference computes the grumpy action but passes only the happy one, the rest of the list is commented out);
    BOTH transitions are stored, happy first (:351-353: the grumpy one holds the action that was chosen for it, the
    grumpy reward `info.dblGrumpyScore` and next state `info.adblGrumpyState`, and the same done flag); then learn().

    drive_grumpy=True is the loop with the commented-out part of :343 restored: the grumpy action is also applied, to
    the first grumpy robot (robot index num_robots_happy; robots between the two get uniformly random actions, since
    a GameEnv_Simple command list cannot skip a robot, RR_EnvBase.py:617-626).

    episode_returns=True also records every episode that ends (env.step(..., episode_info=True): the whole return, as
    get_stats counts it), as the reference's loop records each episode's score (:364-371): the result adds
    "episode_returns" (float64 [n_episodes, 2], happy and grumpy, in the order the episodes ended, envs in index order
    within a step) and "avg_return_100" / "avg_return_100_grumpy" (float64 [n_episodes]: the mean of the last 100
    episodes after each one, the reference's avg_score).  The rows stay on the device and are gathered every 256 steps.

    Returns a dict with env-steps/s measured with CUDA events around the whole loop."""
    N = env.num_envs
    has_grumpy = env.preset.num_robots_grumpy > 0
    g0 = env.preset.num_robots_happy          # index of the first grumpy robot
    obs = env.reset().clone()
    obs_g = env.observe()[1].clone() if has_grumpy else None   # get_game_state(int_team=TEAM_GRUMPY), :322
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    losses = []
    ends, rets, ended = [], [], []   # per-step episode rows on the device, gathered into `ended` every 256 steps

    def gather():
        if ends:
            ended.append(torch.stack(rets)[torch.stack(ends)])
            ends.clear(); rets.clear()
    ev0.record()
    for it in range(n_steps):
        act = agent.choose_actions(obs)
        act_g = agent.choose_actions(obs_g) if has_grumpy else None
        if has_grumpy and drive_grumpy:
            cmd = torch.randint(0, agent.n_actions, (N, g0 + 1), device=agent.device, generator=agent.gen).to(torch.uint8)
            cmd[:, 0] = act
            cmd[:, g0] = act_g
        else:
            cmd = act.view(-1, 1)
        if episode_returns:
            obs_, rew, done, info = env.step(cmd, episode_info=True)
            ends.append(info["_episode"])
            rets.append(torch.stack((info["episode"]["r"], info["episode"]["r_grumpy"]), 1))
            if len(ends) == 256:
                gather()
        else:
            obs_, rew, done, info = env.step(cmd)
        agent.store(obs, act, rew, obs_, done)
        if has_grumpy:
            agent.store(obs_g, act_g, info["reward_grumpy"], info["obs_grumpy"], done)
        if (it + 1) % learn_every == 0:
            loss = agent.learn()
            if loss is not None and log_every and (it + 1) % log_every == 0:
                losses.append(float(loss))
        obs = obs_.clone()
        if has_grumpy:
            obs_g = info["obs_grumpy"].clone()
    ev1.record()
    torch.cuda.synchronize()
    secs = ev0.elapsed_time(ev1) * 1e-3
    out = {"env_steps": n_steps * N, "seconds": secs, "env_steps_per_s": n_steps * N / secs,
           "transitions": n_steps * N * (2 if has_grumpy else 1),
           "losses": losses, "epsilon": agent.epsilon, "stats": env.get_stats()}
    if episode_returns:
        gather()
        r = torch.cat(ended).cpu() if ended else torch.zeros(0, 2, dtype=torch.float64)
        out.update(episode_returns=r, avg_return_100=_running_mean(r[:, 0]), avg_return_100_grumpy=_running_mean(r[:, 1]))
    return out
