"""Value-based agents on the GPU-resident pipeline: DQN and its Double / Dueling / Multistep / PER /
Noisy / C51 / Rainbow / Ape-X variants.

Mirrors jorldy/core/agent/{dqn,double,dueling,multistep,per,noisy,c51,rainbow,ape_x}.py: same
constructor kwargs, bookkeeping (epsilon decay, target-update stamps, learn-period stamps with the
backlog quirk, beta annealing) and result keys.  One learn() = replay gather on the device ->
online/target forwards -> ONE fused target+loss+gradient(+priority) kernel (csrc/dqn.cu, csrc/c51.cu)
-> backward -> (clip +) Adam/RMSprop -> batched sum-tree update (no per-sample .item()).
"""
from collections import deque

import numpy as np
import torch

from ..buffer import FramePERBuffer, FrameReplayBuffer, PERBuffer, ReplayBuffer
from ..dev import C, ptr, require_cuda, stream_ptr
from ..network import Network
from ..optimizer import Optimizer
from .base import BaseAgent


def _action_kind(t):
    return {torch.int64: 0, torch.int32: 1, torch.float32: 2}[t.dtype]


class DQN(BaseAgent):
    action_type = "discrete"
    # how the fused TD kernel is configured for this agent (csrc/dqn.cu)
    _double_q = 0
    _loss_kind = 0      # 0 smooth_l1, 1 IS-weighted MSE
    _order = 0          # 0 dqn.py product order, 1 double.py/per.py order, 2 n-step loop
    _clip = None

    def __init__(self, state_size, action_size, hidden_size=512, optim_config={"name": "adam"},
                 network="discrete_q_network", head="mlp", gamma=0.99, epsilon_init=1.0, epsilon_min=0.1,
                 epsilon_eval=0.0, explore_ratio=0.1, buffer_size=50000, batch_size=64, start_train_step=2000,
                 target_update_period=500, device=None, run_step=1e6, num_workers=1, lr_decay=True, seed=0,
                 frame_replay=False, **kwargs):
        self.device = require_cuda(device)
        self.state_size, self.action_size = state_size, action_size
        self.action_type = "discrete"
        self.seed = int(seed)
        self._build_networks(network, state_size, action_size, hidden_size, head, kwargs)
        self.target_network.copy_from(self.network)
        self.optimizer = Optimizer(**dict(optim_config), params=self.network.parameters())
        self.gamma = gamma
        self.epsilon = epsilon_init
        self.epsilon_init, self.epsilon_min, self.epsilon_eval = epsilon_init, epsilon_min, epsilon_eval
        self.explore_step = run_step * explore_ratio
        self.epsilon_delta = (epsilon_init - epsilon_min) / self.explore_step
        self.buffer_size = buffer_size
        self.frame_replay = frame_replay   # store uint8 frame stacks once per frame (core/buffer/frame_replay.py)
        self.memory = (FrameReplayBuffer if frame_replay else ReplayBuffer)(buffer_size, device=self.device)
        self.batch_size = batch_size
        self.start_train_step = start_train_step
        self.target_update_stamp = 0
        self.target_update_period = target_update_period
        self.num_learn = 0
        self.time_t = 0
        self.num_workers = num_workers
        self.run_step = run_step
        self.lr_decay = lr_decay
        self.n_step = 1
        self.alpha = 0.0
        self.rng_stream_base = 0
        self._row_ctr = {}
        self._eps_rows = None          # per-actor epsilons for batched Ape-X style collection
        self._stats = torch.zeros(4, dtype=torch.float32, device=self.device)
        self.world_size, self.allreduce = 1, None
        self._inject_idx = None        # tests: fixed replay indices for the next learn()

    def _build_networks(self, network, state_size, action_size, hidden_size, head, kwargs):
        self.network = Network(network, state_size, action_size, D_hidden=hidden_size, head=head, device=self.device)
        self.target_network = Network(network, state_size, action_size, D_hidden=hidden_size, head=head,
                                      device=self.device)

    # -------------------------------------------------------------------------------------- act --
    def _q_values(self, state, training, tag="act."):
        M = state.shape[0]
        q = self.network._buf(tag + "q", (M, self.action_size))
        self.network.forward_rows(state, q)
        return q

    def act_device(self, state, training=True, noise=None):
        """state [N, ...] device tensor -> (action int64 [N], q_sel f32 [N])."""
        M = state.shape[0]
        q = self._q_values(state, training)
        eps = self.epsilon if training else self.epsilon_eval
        row_ctr = self._row_ctr.get(M)
        if row_ctr is None:
            row_ctr = self._row_ctr[M] = torch.zeros(M, dtype=torch.int64, device=self.device)
        action = self.network._buf("act.a", (M,), torch.int64)
        q_sel = self.network._buf("act.qsel", (M,))
        eps_rows = self._eps_rows if (training and self._eps_rows is not None and self._eps_rows.shape[0] == M) else None
        C.jb_q_act(ptr(q), M, self.action_size, float(eps), ptr(eps_rows), ptr(noise), self.seed, self.rng_stream_base,
                   ptr(row_ctr), ptr(action), ptr(q_sel), stream_ptr())
        return action, q_sel

    def _state_to_device(self, state):
        if isinstance(state, torch.Tensor):
            return state
        a = np.asarray(state)
        return torch.as_tensor(a, device=self.device)

    def _net_input(self, s):
        """uint8 frames stay uint8 for the CNN head (it scales by 1/255 itself); vectors -> f32 [N, D]."""
        if s.dtype == torch.uint8:
            return s
        return s.to(torch.float32).reshape(s.shape[0], -1)

    @torch.no_grad()
    def act(self, state, training=True):
        self.network.train(training)
        s = self._net_input(self._state_to_device(state))
        action, _ = self.act_device(s, training)
        return {"action": action.cpu().numpy().reshape(-1, 1)}

    # ------------------------------------------------------------------------------------ learn --
    def _sample(self):
        """Returns (batch dict of device tensors, weights f64|None, tree indices|None, stats|None)."""
        idx = None
        if self._inject_idx is not None:
            idx = torch.as_tensor(np.asarray(self._inject_idx), dtype=torch.int64, device=self.device)
        else:
            idx = torch.as_tensor(self.memory.sample_indices(self.batch_size), dtype=torch.int64, device=self.device)
        return self.memory.gather_device(idx), None, None, None

    def _forward_q(self, net, x, tag, is_train=True, noise=None):
        return net.forward(x, tag=tag)

    def _learn_batch(self, batch, weights=None):
        """Shared TD learner. batch: device tensors state, action, reward [B,n], done [B,n], next_state."""
        B = batch["reward"].shape[0]
        A = self.action_size
        state = self._net_input(batch["state"])
        next_state = self._net_input(batch["next_state"])
        reward = batch["reward"].to(torch.float32).reshape(B, -1).contiguous()
        done = batch["done"].to(torch.float32).reshape(B, -1).contiguous()
        action = batch["action"].reshape(B).contiguous()
        if action.dtype not in (torch.int64, torch.int32, torch.float32):
            action = action.to(torch.int64)
        net, tgt = self.network, self.target_network
        noise = getattr(self, "_inject_noise", None) or [None, None, None]
        q = self._forward_q(net, state, "t.", True, noise[0])
        q_next = self._forward_q(net, next_state, "n.", True, noise[1]) if self._double_q else None
        qt_next = self._forward_q(tgt, next_state, "n.", True, noise[2])
        dq = net._buf("t.dq", (B, A))
        prio = net._buf("t.prio", (B,), torch.float64) if weights is not None or self._loss_kind == 1 else None
        C.jb_td_loss(ptr(q), ptr(q_next), ptr(qt_next), ptr(action), _action_kind(action), ptr(reward), ptr(done),
                     ptr(weights), B, A, self.gamma, float(self.alpha), reward.shape[1], self._double_q, self._loss_kind,
                     self._order, ptr(dq), ptr(prio), ptr(self._stats), stream_ptr())
        net.backward(dq, B, tag="t.")
        if self.allreduce is not None:
            self.allreduce(net.grad)
        self.optimizer.step(max_norm=self._clip)
        self.num_learn += 1
        return prio

    def _stats_host(self, stats):
        """stats.cpu().numpy(): learn()'s device->host read.  With the frame replay the same copy carries its overflow
        flag, so a result computed from a stack the pool could no longer hold raises instead of being returned."""
        flag = getattr(self.memory, "overflow_flag", None)
        if flag is None:
            return stats.cpu().numpy()
        both = torch.cat([stats.to(torch.float64), flag.to(torch.float64)]).cpu().numpy()
        self.memory.raise_if_overflow(both[-1] != 0)
        return both[:-1].astype(np.float32)

    def learn(self):
        batch, _, _, _ = self._sample()
        self._learn_batch(batch)
        st = self._stats_host(self._stats[:2])
        return {"loss": float(st[0]), "epsilon": self.epsilon, "max_Q": float(st[1])}

    def update_target(self):
        self.target_network.copy_from(self.network)

    def process(self, transitions, step):
        result = {}
        self.memory.store(transitions)
        delta_t = step - self.time_t
        self.time_t = step
        self.target_update_stamp += delta_t
        if self.memory.size >= self.batch_size and self.time_t >= self.start_train_step:
            result = self.learn()
            if self.lr_decay:
                self.learning_rate_decay(step)
        if self.num_learn > 0:
            self.epsilon_decay(delta_t)
            if self.target_update_stamp >= self.target_update_period:
                self.update_target()
                self.target_update_stamp -= self.target_update_period
        return result

    def epsilon_decay(self, delta_t):
        self.epsilon = max(self.epsilon_min, self.epsilon - delta_t * self.epsilon_delta)

    def set_distributed(self, id):
        self.epsilon = id / self.num_workers
        return self


class Double(DQN):
    _double_q, _order = 1, 1


class Dueling(DQN):
    def __init__(self, network="dueling", **kwargs):
        super().__init__(network=network, **kwargs)


def _nstep_callback(agent, transition, next_from_state=False):
    """multistep.py:90-104 / rainbow.py:294-308 (and ape_x.py:174-199 when next_from_state)."""
    out = {}
    agent.tmp_buffer.append(transition)
    if len(agent.tmp_buffer) == agent.tmp_buffer.maxlen:
        first, last = agent.tmp_buffer[0], agent.tmp_buffer[-1]
        out["state"] = first["state"]
        out["action"] = first["action"]
        out["next_state"] = last["state"] if next_from_state else last["next_state"]
        items = list(agent.tmp_buffer)[:-1] if next_from_state else list(agent.tmp_buffer)
        for key in first.keys():
            if key not in ["state", "action", "next_state"]:
                out[key] = np.stack([np.asarray(t[key]) for t in items], axis=1)
    return out


class Multistep(DQN):
    _order = 2

    def __init__(self, n_step=5, **kwargs):
        super().__init__(**kwargs)
        self.n_step = n_step
        self.tmp_buffer = deque(maxlen=n_step)

    def process(self, transitions, step):
        result = {}
        delta_t = step - self.time_t
        self.memory.store(transitions)
        self.time_t = step
        self.target_update_stamp += delta_t
        if self.memory.size >= self.batch_size and self.time_t >= self.start_train_step:
            result = self.learn()
            if self.lr_decay:
                self.learning_rate_decay(step)
        if self.num_learn > 0:
            self.epsilon_decay(delta_t)
            if self.target_update_stamp >= self.target_update_period:
                self.update_target()
                self.target_update_stamp -= self.target_update_period
        return result

    def interact_callback(self, transition):
        return _nstep_callback(self, transition)


class PER(DQN):
    _double_q, _loss_kind, _order = 1, 1, 1

    def __init__(self, alpha=0.6, beta=0.4, learn_period=16, uniform_sample_prob=1e-3, run_step=1e6, **kwargs):
        super().__init__(run_step=run_step, **kwargs)
        self.memory = (FramePERBuffer if self.frame_replay else PERBuffer)(self.buffer_size, uniform_sample_prob,
                                                                           device=self.device, seed=self.seed)
        self.alpha = alpha
        self.beta = beta
        self.beta_add = (1 - beta) / run_step
        self.learn_period = learn_period
        self.learn_period_stamp = 0
        self._inject_u = None          # tests: (u_a, u_b) uniforms for the next sample

    def _per_sample(self):
        u_a = u_b = None
        if self._inject_u is not None:
            u_a, u_b = (torch.as_tensor(np.asarray(x), dtype=torch.float64, device=self.device) for x in self._inject_u)
        return self.memory.sample_device(self.beta, self.batch_size, u_a, u_b)

    def _per_result(self, stats_per):
        st = self._stats_host(self._stats[:2])
        sp = stats_per.cpu().numpy()
        return float(st[0]), float(st[1]), float(sp[0]), float(sp[1])

    def learn(self):
        batch, weights, indices, stats_per = self._per_sample()
        prio = self._learn_batch(batch, weights)
        self.memory.update_priorities(indices, prio)
        loss, max_q, sampled_p, mean_p = self._per_result(stats_per)
        return {"loss": loss, "epsilon": self.epsilon, "beta": self.beta, "max_Q": max_q, "sampled_p": sampled_p,
                "mean_p": mean_p}

    def _stamped_process(self, transitions, step, counter_attr, decay_eps):
        """per.py:90-122 / rainbow.py:255-283 / ape_x.py:135-164: learn at most once per call while the
        learn-period stamp has backlog."""
        result = {}
        delta_t = step - self.time_t
        self.memory.store(transitions)
        self.time_t = step
        self.target_update_stamp += delta_t
        self.learn_period_stamp += delta_t
        self.beta = min(1.0, self.beta + (self.beta_add * delta_t))
        filled = self.memory.size if counter_attr == "size" else self.memory.buffer_counter
        if (self.learn_period_stamp >= self.learn_period and filled >= self.batch_size
                and self.time_t >= self.start_train_step):
            result = self.learn()
            if self.lr_decay:
                self.learning_rate_decay(step)
            self.learn_period_stamp -= self.learn_period
        if self.num_learn > 0:
            if decay_eps:
                self.epsilon_decay(delta_t)
            if self.target_update_stamp >= self.target_update_period:
                self.update_target()
                self.target_update_stamp -= self.target_update_period
        return result

    def process(self, transitions, step):
        return self._stamped_process(transitions, step, "size", True)


class Noisy(DQN):
    def __init__(self, state_size, action_size, hidden_size=512, network="noisy", head="mlp", noise_type="factorized",
                 **kwargs):
        self._noise_type = noise_type
        super().__init__(state_size, action_size, hidden_size=hidden_size, network=network, head=head, **kwargs)

    def _build_networks(self, network, state_size, action_size, hidden_size, head, kwargs):
        mk = lambda s: Network(network, state_size, action_size, self._noise_type, D_hidden=hidden_size, head=head,
                               device=self.device, seed=s)
        self.network, self.target_network = mk(self.seed), mk(self.seed + 1)

    def _forward_q(self, net, x, tag, is_train=True, noise=None):
        return net.forward(x, is_train, tag=tag, noise=noise)

    def _q_values(self, state, training, tag="act.", noise=None):
        M = state.shape[0]
        q = self.network._buf(tag + "q", (M, self.action_size))
        self.network.forward_rows(state, q, is_train=training, noise=noise)
        return q

    def act_device(self, state, training=True, noise=None):
        """noise: injected NoisyNet draws [(eps_i, eps_j)] x 2 for this forward (parity tests)."""
        M = state.shape[0]
        if training and self.memory.size < max(self.batch_size, self.start_train_step):
            action = torch.randint(0, self.action_size, (M,), device=self.device)      # noisy.py:71-72
            return action, None
        q = self._q_values(state, training, noise=noise)
        return torch.argmax(q, -1), None

    def learn(self):
        batch, _, _, _ = self._sample()
        self._learn_batch(batch)
        st = self._stats_host(self._stats[:2])
        s1, s2 = self.network.get_sig_w_mean()
        return {"loss": float(st[0]), "max_Q": float(st[1]), "sig_w1": float(s1.item()), "sig_w2": float(s2.item())}

    def process(self, transitions, step):
        result = {}
        self.memory.store(transitions)
        delta_t = step - self.time_t
        self.time_t = step
        self.target_update_stamp += delta_t
        if self.memory.size >= self.batch_size and self.time_t >= self.start_train_step:
            result = self.learn()
            if self.lr_decay:
                self.learning_rate_decay(step)
        if self.num_learn > 0 and self.target_update_stamp >= self.target_update_period:
            self.update_target()
            self.target_update_stamp -= self.target_update_period
        return result


class _Distributional:
    """C51 machinery shared by C51 and Rainbow (support z, fused projection/KL kernel)."""

    def _setup_support(self, v_min, v_max, num_support):
        self.v_min, self.v_max, self.num_support = v_min, v_max, num_support
        self.delta_z = (v_max - v_min) / (num_support - 1)
        self.z = torch.linspace(v_min, v_max, num_support, device=self.device).view(1, -1)

    def _dist_learn(self, batch, weights, variant, noise):
        B = batch["reward"].shape[0]
        A, K = self.action_size, self.num_support
        state = self._net_input(batch["state"])
        next_state = self._net_input(batch["next_state"])
        reward = batch["reward"].to(torch.float32).reshape(B, -1).contiguous()
        done = batch["done"].to(torch.float32).reshape(B, -1).contiguous()
        action = batch["action"].reshape(B).contiguous()
        net, tgt = self.network, self.target_network
        logits = self._forward_logits(net, state, "t.", noise[0])
        next_online = self._forward_logits(net, next_state, "n.", noise[1]) if variant == 1 else None
        next_target = self._forward_logits(tgt, next_state, "n.", noise[2])
        dlogits = net._buf("t.dlogits", (B, A, K))
        kl = net._buf("t.kl", (B,))
        prio = net._buf("t.prio", (B,), torch.float64) if variant == 1 else None
        scratch = net._buf("t.c51scratch", (4 * ((B + 7) // 8),))
        C.jb_c51_loss(ptr(logits), ptr(next_online), ptr(next_target), ptr(action), _action_kind(action), ptr(reward),
                      ptr(done), ptr(weights), ptr(self.z), B, A, K, self.gamma, float(self.v_min), float(self.v_max),
                      float(self.alpha), reward.shape[1], variant, ptr(dlogits), ptr(kl), ptr(prio), ptr(self._stats),
                      ptr(scratch), stream_ptr())
        net.backward(dlogits.view(B, A * K), B, tag="t.")
        if self.allreduce is not None:
            self.allreduce(net.grad)
        self.optimizer.step(max_norm=self._clip)
        self.num_learn += 1
        return prio

    def _expected_q(self, logits, M):
        q = self.network._buf("act.q", (M, self.action_size))
        C.jb_c51_q(ptr(logits), ptr(self.z), M, self.action_size, self.num_support, ptr(q), stream_ptr())
        return q


class C51(DQN, _Distributional):
    def __init__(self, state_size, action_size, v_min=-10, v_max=10, num_support=51, **kwargs):
        self._num_support = num_support
        super().__init__(state_size, action_size * num_support, **kwargs)
        self.action_size = action_size
        self._setup_support(v_min, v_max, num_support)

    def _forward_logits(self, net, x, tag, noise=None):
        return net.forward(x, tag=tag)

    def _q_values(self, state, training, tag="act."):
        M = state.shape[0]
        logits = self.network._buf(tag + "logits", (M, self.action_size * self.num_support))
        self.network.forward_rows(state, logits)
        return self._expected_q(logits, M)

    def learn(self):
        batch, _, _, _ = self._sample()
        self._dist_learn(batch, None, 0, [None, None, None])
        st = self._stats_host(self._stats)
        return {"loss": float(st[0]), "epsilon": self.epsilon, "max_Q": float(st[1]), "max_logit": float(st[2]),
                "min_logit": float(st[3])}


class Rainbow(PER, _Distributional):
    def __init__(self, state_size, action_size, hidden_size=512, network="rainbow", head="mlp",
                 optim_config={"name": "adam"}, gamma=0.99, buffer_size=50000, batch_size=64, start_train_step=2000,
                 target_update_period=500, run_step=1e6, lr_decay=True, n_step=4, alpha=0.6, beta=0.4, learn_period=4,
                 uniform_sample_prob=1e-3, noise_type="factorized", v_min=-10, v_max=10, num_support=51, device=None,
                 seed=0, frame_replay=False, **kwargs):
        self._noise_type, self._num_support = noise_type, num_support
        super().__init__(alpha=alpha, beta=beta, learn_period=learn_period, uniform_sample_prob=uniform_sample_prob,
                         run_step=run_step, state_size=state_size, action_size=action_size, hidden_size=hidden_size,
                         network=network, head=head, optim_config=optim_config, gamma=gamma, buffer_size=buffer_size,
                         batch_size=batch_size, start_train_step=start_train_step,
                         target_update_period=target_update_period, lr_decay=lr_decay, device=device, seed=seed,
                         frame_replay=frame_replay)
        self.n_step = n_step
        self.tmp_buffer = deque(maxlen=n_step)
        self._setup_support(v_min, v_max, num_support)
        self._inject_noise = None      # tests: [noise(s), noise(s'), noise_target(s')] each 4 (eps_i, eps_j) pairs

    def _build_networks(self, network, state_size, action_size, hidden_size, head, kwargs):
        mk = lambda s: Network(network, state_size, action_size, self._num_support, self._noise_type,
                               D_hidden=hidden_size, head=head, device=self.device, seed=s)
        self.network, self.target_network = mk(self.seed), mk(self.seed + 1)

    def _forward_logits(self, net, x, tag, noise=None):
        return net.forward(x, True, tag=tag, noise=noise)

    def act_device(self, state, training=True, noise=None):
        """One noisy forward for all rows (the reference's act() with a batch of N states draws its noise once per
        call, rainbow.py:149).  noise: injected draws [(eps_i, eps_j)] x 4 in call order a1, v1, a2, v2."""
        M = state.shape[0]
        if training and self.memory.size < max(self.batch_size, self.start_train_step):
            return torch.randint(0, self.action_size, (M,), device=self.device), None       # rainbow.py:143-147
        logits = self.network._buf("act.logits", (M, self.action_size, self.num_support))
        self.network.forward_rows(state, logits, is_train=training, noise=noise)
        return torch.argmax(self._expected_q(logits, M), -1), None

    def learn(self):
        batch, weights, indices, stats_per = self._per_sample()
        noise = self._inject_noise or [None, None, None]
        prio = self._dist_learn(batch, weights, 1, noise)
        self.memory.update_priorities(indices, prio)
        st = self._stats_host(self._stats)
        sp = stats_per.cpu().numpy()
        return {"loss": float(st[0]), "beta": self.beta, "max_Q": float(st[1]), "max_logit": float(st[2]),
                "min_logit": float(st[3]), "sampled_p": float(sp[0]), "mean_p": float(sp[1])}

    def process(self, transitions, step):
        return self._stamped_process(transitions, step, "counter", False)

    def interact_callback(self, transition):
        return _nstep_callback(self, transition)


class ApeX(PER):
    _double_q, _loss_kind, _order = 1, 1, 2

    def __init__(self, epsilon=0.4, epsilon_alpha=7.0, clip_grad_norm=40.0, alpha=0.6, beta=0.4, learn_period=4,
                 uniform_sample_prob=1e-3, n_step=4, **kwargs):
        super().__init__(alpha=alpha, beta=beta, learn_period=learn_period, uniform_sample_prob=uniform_sample_prob,
                         **kwargs)
        self.epsilon = epsilon
        self.epsilon_alpha = epsilon_alpha
        self.clip_grad_norm = clip_grad_norm
        self._clip = clip_grad_norm
        self.num_transitions = 0
        self.n_step = n_step
        self.tmp_buffer = deque(maxlen=n_step + 1)

    @torch.no_grad()
    def act(self, state, training=True):
        self.network.train(training)
        s = self._net_input(self._state_to_device(state))
        action, q_sel = self.act_device(s, training)
        return {"action": action.cpu().numpy().reshape(-1, 1), "q": q_sel.cpu().numpy()}

    def learn(self):
        batch, weights, indices, stats_per = self._per_sample()
        prio = self._learn_batch(batch, weights)
        self.memory.update_priorities(indices, prio)
        loss, max_q, sampled_p, mean_p = self._per_result(stats_per)
        return {"loss": loss, "max_Q": max_q, "sampled_p": sampled_p, "mean_p": mean_p, "num_learn": self.num_learn,
                "num_transitions": self.num_transitions}

    def process(self, transitions, step):
        self.num_transitions += sum(int(np.shape(t["reward"])[0]) for t in transitions)
        return self._stamped_process(transitions, step, "counter", False)

    def set_distributed(self, id):
        assert self.num_workers > 1
        self.epsilon = self.epsilon ** (1 + (id / (self.num_workers - 1)) * self.epsilon_alpha)
        return self

    def set_actor_epsilons(self, n_actors, first_id=0, total=None):
        """Batched collection: row i of the env batch plays actor first_id+i of `total` (ape_x.py:166-172)."""
        total = total or self.num_workers
        ids = torch.arange(first_id, first_id + n_actors, dtype=torch.float64)
        eps = torch.tensor(self.epsilon, dtype=torch.float64) ** (1 + (ids / (total - 1)) * self.epsilon_alpha)
        self._eps_rows = eps.to(torch.float32).to(self.device)

    def interact_callback(self, transition):
        out = _nstep_callback(self, transition, next_from_state=True)
        if out:
            tb = self.tmp_buffer
            target_q = np.asarray(tb[-1]["q"])
            for i in reversed(range(self.n_step)):
                target_q = np.asarray(tb[i]["reward"]) + (1 - np.asarray(tb[i]["done"])) * self.gamma * target_q
            out["priority"] = abs(target_q - np.asarray(tb[0]["q"]))
            del out["q"]
        return out
