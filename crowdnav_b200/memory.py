"""Replay memory and trajectory recording for batched rollouts (SURVEY.md 8f row 3).

  DeviceReplayMemory   crowd_nav/utils/memory.py:4-28 (ReplayMemory: ring of (state, value) pairs) as two device tensors
  TrajectoryRecorder   crowd_nav/utils/explorer.py:92-125 (Explorer.update_memory): per env slot the rotated joint
                       states and rewards of the running episode; when an episode ends in ReachGoal or Collision its
                       (state_i, value_i) pairs are appended to the memory, with
                         imitation learning:  value_i = sum_{t >= i} pow(gamma, (t - i) * time_step * v_pref) * r_t
                         RL:                  value_i = r_i + gamma_bar * target_model(state_{i+1}),  r_i at the terminal step
The IL return is accumulated forward in t (G_i += pow(...) * r_t as each reward arrives), i.e. in the same order and
with the same pow() factors as the reference's sum(); it agrees to the last ulp of float64 (CPython >= 3.12 sums with
Neumaier compensation) and is identical after the float32 cast the reference applies.
"""
import torch

from . import _abi


class DeviceReplayMemory(object):
    def __init__(self, capacity, human_num, device, feature_dim=13):
        self.capacity = int(capacity)
        self.states = torch.zeros((self.capacity, human_num, feature_dim), dtype=torch.float32, device=device)
        self.values = torch.zeros((self.capacity, 1), dtype=torch.float32, device=device)
        self.position = 0          # memory.py:8,15-19: write pointer, wraps
        self.size = 0

    def push_batch(self, states, values):
        n = states.shape[0]
        if n == 0:
            return
        idx = (torch.arange(n, device=states.device) + self.position) % self.capacity
        self.states[idx] = states
        self.values[idx] = values.reshape(-1, 1).to(torch.float32)
        self.position = (self.position + n) % self.capacity
        self.size = min(self.capacity, self.size + n)

    def is_full(self):
        return self.size == self.capacity

    def __len__(self):
        return self.size

    def __getitem__(self, item):
        return self.states[item], self.values[item]

    def clear(self):
        self.position = 0
        self.size = 0

    def sample(self, batch_size, generator=None):
        idx = torch.randint(0, self.size, (batch_size,), device=self.states.device, generator=generator)
        return self.states[idx], self.values[idx]


class TrajectoryRecorder(object):
    def __init__(self, env, memory, gamma, imitation_learning=True, target_model=None, max_steps=None, om=None):
        """om = None or (cell_num, cell_size, om_channel_size): append the occupancy maps of the current human states to
        every recorded row, as MultiHumanRL.transform does with with_om (multi_human_rl.py:98-104)."""
        self.env, self.memory = env, memory
        self.om = om
        F = 13 + (om[0] * om[0] * om[2] if om else 0)
        self.il, self.target_model = imitation_learning, target_model
        B, N, dev = env.B, env.human_num, env.device
        from .batched import max_episode_steps
        self.T = max_steps or max(128, max_episode_steps(env.time_limit, env.time_step))     # covers the longest episode
        self.states = torch.zeros((B, self.T, N, F), dtype=torch.float32, device=dev)
        self.rewards = torch.zeros((B, self.T), dtype=torch.float64, device=dev)
        self.returns = torch.zeros((B, self.T), dtype=torch.float64, device=dev)
        dt, v_pref = env.time_step, env.robot_v_pref
        # W[t][i] = pow(gamma, max(t - i, 0) * time_step * v_pref) for i <= t, else 0   (explorer.py:104-105), evaluated
        # left to right as the reference does: ((t - i) * dt) * v_pref rounds differently from (t - i) * (dt * v_pref)
        w = [[pow(gamma, (t - i) * dt * v_pref) if i <= t else 0.0 for i in range(self.T)] for t in range(self.T)]
        self.W = torch.tensor(w, dtype=torch.float64, device=dev)
        self.gamma_bar = pow(gamma, dt * v_pref)                         # explorer.py:112
        self._t = None
        self._live = None

    def before_step(self):
        """Record the state each live env decides on: robot.policy.last_state after transform() = rotate(joint state)."""
        env = self.env
        self._t = env.episodes.ep_steps.long().clamp_(max=self.T - 1)
        self._live = env.state.active.bool()
        packed = env.pack_joint()
        if self.om:
            packed = torch.cat([packed, env.occupancy_maps(None, None, *self.om)], dim=2)
        rows = torch.arange(env.B, device=env.device)
        self.states[rows, self._t] = torch.where(self._live.view(-1, 1, 1), packed, self.states[rows, self._t])

    def after_step(self):
        """Book the reward of the step; flush the trajectories of episodes that just ended in success or collision."""
        env = self.env
        rows = torch.arange(env.B, device=env.device)
        r = torch.where(self._live, env.reward, torch.zeros_like(env.reward))
        self.rewards[rows, self._t] = r
        self.returns += self.W[self._t] * r.unsqueeze(1)                 # G_i += pow(gamma, (t-i)*dt*v_pref) * r_t, i <= t
        done = self._live & env.done.bool()
        keep = done & ((env.info == _abi.INFO_REACHGOAL) | (env.info == _abi.INFO_COLLISION))   # explorer.py:67-69
        if bool(keep.any()):
            length = self._t + 1
            steps = torch.arange(self.T, device=env.device).unsqueeze(0)
            sel = keep.unsqueeze(1) & (steps < length.unsqueeze(1))      # [B][T], env-major then time: episode order kept
            st = self.states[sel]
            if self.il:
                val = self.returns[sel]
            else:
                nxt = torch.roll(self.states, shifts=-1, dims=1)[sel]
                with torch.no_grad():
                    boot = self.target_model(nxt).double().view(-1)
                terminal = (steps == (length - 1).unsqueeze(1)).expand_as(sel)[sel]
                val = self.rewards[sel] + torch.where(terminal, torch.zeros_like(boot), self.gamma_bar * boot)
            self.memory.push_batch(st, val)
        if bool(done.any()):
            self.returns[done] = 0.0
            self.rewards[done] = 0.0
