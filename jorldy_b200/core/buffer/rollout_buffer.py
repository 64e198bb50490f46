"""On-policy rollout storage.

`RolloutBuffer` keeps the reference's list semantics for host transitions
(jorldy/core/buffer/rollout_buffer.py:6-24: store appends, sample stacks everything and clears).
`DeviceRollout` is the HBM-resident [N, T, ...] structure-of-arrays the batched collect kernels
write straight into (no host hop): actor-major like the reference's concatenation order
(distributed_manager.py:30), so GAE's `view(-1, n_step)` rows are envs.
"""
import numpy as np
import torch

from ..dev import require_cuda
from .base import BaseBuffer


class RolloutBuffer(BaseBuffer):
    def __init__(self):
        super().__init__()
        self.buffer = list()

    def store(self, transitions):
        if self.first_store:
            self.check_dim(transitions[0])
        self.buffer += transitions

    def sample(self):
        transitions = self.stack_transition(self.buffer)
        self.buffer.clear()
        return transitions

    def sample_batched(self):
        """For transitions whose leading dim is a batch of N envs (one dict per time step): returns
        arrays laid out [N*T, ...] actor-major, i.e. what N reference actors would have produced."""
        out = {}
        for key in self.buffer[0].keys():
            arr = np.stack([np.asarray(b[key]) for b in self.buffer], axis=1)   # [N, T, ...]
            out[key] = arr.reshape((-1,) + arr.shape[2:])
        self.buffer.clear()
        return out

    @property
    def size(self):
        return len(self.buffer)


class DeviceRollout:
    def __init__(self, num_envs, n_step, state_size, action_size, action_type, device=None):
        dev = require_cuda(device)
        N, T = num_envs, n_step
        self.N, self.T, self.device = N, T, dev
        # a shaped state is a uint8 frame stack, kept as the env produces it (4x84x84: 28 224 B a row instead of 4x that
        # as f32); a vector state is f32
        if isinstance(state_size, (list, tuple)):
            shape, sdtype = tuple(state_size), torch.uint8
        else:
            shape, sdtype = (state_size,), torch.float32
        self.state = torch.zeros(N, T, *shape, dtype=sdtype, device=dev)
        if action_type == "discrete":
            self.action = torch.zeros(N, T, dtype=torch.int32, device=dev)
        else:
            self.action = torch.zeros(N, T, action_size, dtype=torch.float32, device=dev)
        self.reward = torch.zeros(N, T, dtype=torch.float32, device=dev)
        self.done = torch.zeros(N, T, dtype=torch.float32, device=dev)
        self.last_next_state = torch.zeros(N, *shape, dtype=sdtype, device=dev)
        self.t = 0

    def write(self, state, action, reward, done, next_state):
        t = self.t
        self.state[:, t].copy_(state)
        if self.action.dtype == torch.int32:
            self.action[:, t].copy_(action.view(self.N))
        else:
            self.action[:, t].copy_(action.view(self.N, -1))
        self.reward[:, t].copy_(reward)
        self.done[:, t].copy_(done)
        if t == self.T - 1:
            self.last_next_state.copy_(next_state)
        self.t = t + 1

    def write_after_step(self, action, reward, done, next_state):
        """Second half of a transition (the pre-step state was already copied into state[:, t])."""
        t = self.t
        if self.action.dtype == torch.int32:
            self.action[:, t].copy_(action.view(self.N))
        else:
            self.action[:, t].copy_(action.view(self.N, -1))
        self.reward[:, t].copy_(reward)
        self.done[:, t].copy_(done)
        if t == self.T - 1:
            self.last_next_state.copy_(next_state)
        self.t = t + 1

    @property
    def full(self):
        return self.t >= self.T

    def clear(self):
        self.t = 0
