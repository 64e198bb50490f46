"""PPO agent on the GPU-resident pipeline.

Mirror of jorldy/core/agent/ppo.py (act :54-69, learn :71-185, process :187-202) and the parts of
reinforce.py it inherits (:32-64 ctor, :128-142 save/load).  Same constructor kwargs, same result
keys.  What changes is where the work happens:

  act      one batched forward + sampling kernel for all envs (host numpy in/out kept for the
           plugin API; act_device() stays on the GPU)
  learn    pre-pass (value, log_prob_old) -> jb_gae -> n_epoch x shuffled minibatches where one
           minibatch step = forward, fused loss fwd+bwd, backward, clip+Adam, captured once in a
           CUDA graph and replayed with a device-side minibatch cursor; per-minibatch stats are
           accumulated on the device and read back once (the reference does 5 .item() syncs per
           minibatch, ppo.py:171-175)
"""
import numpy as np
import torch

from ..buffer import RolloutBuffer
from ..dev import C, ptr, require_cuda, stream_ptr
from ..network import Network
from ..optimizer import Optimizer
from .base import BaseAgent

GRAPH_CHUNK = 16     # minibatch steps captured per CUDA graph


class PPO(BaseAgent):
    def __init__(
        self,
        state_size,
        action_size,
        hidden_size=512,
        network="discrete_policy_value",
        head="mlp",
        optim_config={"name": "adam"},
        gamma=0.99,
        use_standardization=True,
        run_step=1e6,
        lr_decay=True,
        device=None,
        batch_size=32,
        n_step=128,
        n_epoch=3,
        _lambda=0.95,
        epsilon_clip=0.1,
        vf_coef=1.0,
        ent_coef=0.01,
        clip_grad_norm=1.0,
        num_workers=1,
        seed=0,
        use_cuda_graph=True,
        use_fused=True,
        **kwargs,
    ):
        self.device = require_cuda(device)
        self.action_type = network.split("_")[0]
        assert self.action_type in ["continuous", "discrete"]
        self.state_size, self.action_size = state_size, action_size
        self.network = Network(network, state_size, action_size, D_hidden=hidden_size, head=head,
                               device=self.device)
        # device row layout of a state: uint8 [C, H, W] frame stacks for the CNN head (it scales by 1/255 itself),
        # f32 [D] vectors for the MLP head
        h = self.network.head
        self._row_shape, self._row_dtype = ((h.D_in, torch.uint8) if h.kind == "cnn" else ((h.D_in,), torch.float32))
        optim_config = dict(optim_config)
        self.optimizer = Optimizer(**optim_config, params=self.network.parameters())

        self.gamma = gamma
        self.use_standardization = use_standardization
        self.memory = RolloutBuffer()
        self.run_step = run_step
        self.lr_decay = lr_decay

        self.batch_size = batch_size
        self.n_step = n_step
        self.n_epoch = n_epoch
        self._lambda = _lambda
        self.epsilon_clip = epsilon_clip
        self.vf_coef = vf_coef
        self.ent_coef = ent_coef
        self.clip_grad_norm = clip_grad_norm
        self.num_workers = num_workers
        self.time_t = 0
        self.learn_stamp = 0

        self.seed = int(seed)
        self.rng_stream_base = 0
        self._row_ctr = {}                    # per-row Philox draw counters (device), keyed by batch rows
        self.use_cuda_graph = use_cuda_graph
        self.use_fused = use_fused            # persistent minibatch-loop kernel (csrc/ppo_fused.cu) when eligible
        self._fused = {}
        self._graphs = {}
        self._acc = torch.zeros(8, dtype=torch.float32, device=self.device)
        self._cursor = torch.zeros(1, dtype=torch.int64, device=self.device)
        self.world_size = 1                   # set by parallel.attach() for multi-GPU learners
        self.allreduce = None
        self._inject_perms = None             # tests: list of per-epoch index arrays
        self.n_launches = 0                   # kernels launched by the last learn() (bench bookkeeping)
        self.n_prepass_launches = 0

    # ------------------------------------------------------------------------------------- act --
    @property
    def continuous(self):
        return self.action_type == "continuous"

    def act_device(self, state, training=True, noise=None):
        """state: [N, D] f32 / [N, C, H, W] uint8 device tensor -> action device tensor ([N] int64 / [N, A] f32)."""
        net = self.network
        M = state.shape[0]
        out = net._buf("act.out", (M, net.nout))
        net.forward_rows(state, out)
        A = self.action_size
        row_ctr = self._row_ctr.get(M)
        if row_ctr is None:
            row_ctr = self._row_ctr[M] = torch.zeros(M, dtype=torch.int64, device=self.device)
        if self.continuous:
            action = net._buf("act.a", (M, A))
            C.jb_ppo_act_continuous(ptr(out), M, A, net.nout, ptr(noise), self.seed, self.rng_stream_base,
                                    0, ptr(row_ctr), int(not training), ptr(action), stream_ptr())
        else:
            action = net._buf("act.a", (M,), torch.int64)
            C.jb_ppo_act_discrete(ptr(out), M, A, net.nout, ptr(noise), self.seed, self.rng_stream_base,
                                  0, ptr(row_ctr), int(not training), ptr(action), stream_ptr())
        return action

    def _state_rows(self, state):
        """Host or device states -> device rows in the network's input layout (see _row_shape)."""
        if self._row_dtype == torch.uint8:
            return torch.as_tensor(state, device=self.device).reshape(-1, *self._row_shape)
        s = self.as_tensor(state)
        return s.view(s.shape[0], -1)

    @torch.no_grad()
    def act(self, state, training=True):
        self.network.train(training)
        action = self.act_device(self._state_rows(state), training)
        a = action.cpu().numpy()
        return {"action": a.reshape(a.shape[0], -1)}

    # ----------------------------------------------------------------------------------- learn --
    def _minibatch_step(self, st, idx, B):
        """forward -> fused loss fwd/bwd -> backward -> (all-reduce) -> clip + Adam, for rollout rows idx[B]."""
        net = self.network
        tag = f"mb{B}."
        out = net.forward_raw(st["state"], idx, B, tag=tag)
        dout = net._buf(tag + "dout", (B, net.nout))
        stats = net._buf(tag + "stats", (8 + 4 * ((B + 255) // 256),))
        C.jb_ppo_loss(int(self.continuous), ptr(out), ptr(idx), ptr(st["action"]), ptr(st["adv"]), ptr(st["ret"]),
                      ptr(st["value"]), ptr(st["logp_old"]), B, self.action_size, net.nout, self.epsilon_clip,
                      self.vf_coef, self.ent_coef, ptr(dout), ptr(stats), ptr(self._acc), stream_ptr())
        net.backward_raw(dout, B, tag=tag)
        if self.allreduce is not None:
            self.allreduce(net.grad)
        self.optimizer.step(max_norm=self.clip_grad_norm)

    LAUNCHES_PER_MINIBATCH = 13   # take + in_fwd + gemm + heads + loss + finalize + 2 heads bwd + 3 gemm + sumsq + adam

    def _launches_per_minibatch(self, B):
        """LAUNCHES_PER_MINIBATCH with the input head's own forward / backward kernels (1 + 1 for the MLP head)."""
        h = self.network.head
        return self.LAUNCHES_PER_MINIBATCH - 2 + h.fwd_launches + h.bwd_launches(B)

    def _graph_for(self, st, B):
        """CUDA graph of GRAPH_CHUNK minibatch steps reading indices through the device cursor."""
        key = (B,) + tuple(st[k].data_ptr() for k in ("state", "action", "adv", "ret", "value", "logp_old", "perm"))
        g = self._graphs.get(key)
        if g is not None:
            return g
        cur_idx = self.network._buf(f"mb{B}.cur_idx", (B,), torch.int32)

        def chunk():
            for _ in range(GRAPH_CHUNK):
                C.jb_take_minibatch(ptr(st["perm"]), ptr(self._cursor), B, ptr(cur_idx), stream_ptr())
                self._minibatch_step(st, cur_idx, B)

        # warm-up on a side stream (allocates workspaces), restoring every mutated buffer afterwards
        net, opt = self.network, self.optimizer
        mutated = [net.flat, *opt.state_tensors(), self._acc, self._cursor]
        saved = [t.clone() for t in mutated]
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            C.jb_take_minibatch(ptr(st["perm"]), ptr(self._cursor), B, ptr(cur_idx), stream_ptr())
            self._minibatch_step(st, cur_idx, B)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        for dst, src in zip(mutated, saved):
            dst.copy_(src)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            chunk()
        # capture does not execute, state is untouched
        self._graphs[key] = graph
        return graph

    def _learn_tensors(self, state, action, reward, done, next_state=None, last_next_state=None):
        """Everything is a device tensor; rows are actor-major [N*T, ...]."""
        net = self.network
        NT = state.shape[0]
        T = self.n_step
        N = NT // T
        assert N * T == NT, f"rollout of {NT} rows is not a multiple of n_step={T} (ppo.py:97 view(-1, n_step) would raise)"
        A = self.action_size
        dev = self.device
        s = stream_ptr()
        st = getattr(self, "_st", None)
        if st is None or st["NT"] != NT:
            st = {"NT": NT,
                  "out": torch.empty(NT, net.nout, device=dev),
                  "value": torch.empty(NT, device=dev),
                  "logp_old": torch.empty(NT, A if self.continuous else 1, device=dev),
                  "adv": torch.empty(NT, device=dev), "ret": torch.empty(NT, device=dev),
                  "next_value": torch.empty(NT, device=dev),
                  "perm": torch.empty(NT, dtype=torch.int32, device=dev)}
            self._st = st
        st["state"] = state
        st["action"] = action
        # ---- pre-pass: value and log_prob_old (ppo.py:83-93) ----
        net.forward_rows(state, st["out"])
        if self.continuous:
            C.jb_ppo_prepass_continuous(ptr(st["out"]), ptr(action), NT, A, net.nout, ptr(st["value"]),
                                        ptr(st["logp_old"]), s)
        else:
            C.jb_ppo_prepass_discrete(ptr(st["out"]), ptr(action), NT, A, net.nout, ptr(st["value"]),
                                      ptr(st["logp_old"]), s)
        # ---- V(s') (ppo.py:94) ----
        if next_state is not None:
            nout = net._buf("next.out", (NT, net.nout))
            net.forward_rows(next_state, nout)
            st["next_value"].copy_(nout[:, -1])
            nv, lv = st["next_value"], None
        else:
            lout = net._buf("last.out", (N, net.nout))
            net.forward_rows(last_next_state, lout)
            lv = net._buf("last.v", (N,))
            lv.copy_(lout[:, -1])
            nv = None
        # ---- GAE + returns + standardisation (ppo.py:95-110) ----
        C.jb_gae(ptr(reward), ptr(done), ptr(st["value"]), ptr(nv), ptr(lv), N, T, self.gamma, self._lambda,
                 int(self.use_standardization), ptr(st["adv"]), ptr(st["ret"]), s)
        mean_ret = st["ret"].mean()

        # ---- optimisation epochs (ppo.py:114-175) ----
        B = self.batch_size
        self.optimizer._sync_lr()          # graph replays do not pass through optimizer.step()'s host-side lr check
        self._acc.zero_()
        self._acc[3] = -float("inf")
        self._acc[4] = float("inf")
        n_full = NT // B
        tail = NT - n_full * B
        from . import ppo_fused
        use_fused = self.use_fused and n_full > 0 and ppo_fused.supported(self, B)
        if use_fused and B not in self._fused:
            self._fused[B] = ppo_fused.FusedRunner(self, B)
        use_graph = (not use_fused) and self.use_cuda_graph and n_full >= GRAPH_CHUNK
        n_steps = 0
        for epoch in range(self.n_epoch):
            if self._inject_perms is not None:
                perm = torch.as_tensor(np.asarray(self._inject_perms[epoch]), dtype=torch.int32, device=dev)
            else:
                perm = torch.randperm(NT, device=dev, dtype=torch.int32)
            st["perm"].copy_(perm)
            self._cursor.zero_()
            done_steps = 0
            if use_fused:
                self._fused[B].run(st, n_full)
                done_steps = n_full
            if use_graph:
                g = self._graph_for(st, B)
                for _ in range(n_full // GRAPH_CHUNK):
                    g.replay()
                done_steps = (n_full // GRAPH_CHUNK) * GRAPH_CHUNK
            for k in range(done_steps, n_full):
                self._minibatch_step(st, st["perm"][k * B:(k + 1) * B], B)
            if tail:
                self._minibatch_step(st, st["perm"][n_full * B:], tail)
            n_steps += n_full + (1 if tail else 0)
        per_tail = self._launches_per_minibatch(tail) if tail else 0
        self.n_launches = (self.n_epoch * (1 + per_tail) if use_fused
                           else self.n_epoch * (n_full * self._launches_per_minibatch(B) + per_tail))
        per_pass, rows = net.head.fwd_launches + 2, net.head.max_rows     # head + gemm + heads per inference chunk
        n_next = NT if next_state is not None else N
        # forward chunks + prepass + V(s') chunks + gae
        self.n_prepass_launches = per_pass * -(-NT // rows) + 1 + per_pass * -(-n_next // rows) + 1

        acc = torch.cat([self._acc[:6], mean_ret.view(1), self._acc[7:8]]).cpu().numpy()     # ONE device->host read
        if acc[7] != 0.0:
            dbg = [ws["partials"][200:205].tolist() for ws in (r.ws for r in self._fused.values())]
            raise RuntimeError("persistent PPO kernel: a peer GPU did not reach the gradient exchange (flag wait timed out); "
                               f"[kind 1=grad-ready 2=done-reading, peer, step, seen, target] = {dbg}")
        cnt = max(acc[5], 1.0)
        return {
            "actor_loss": float(acc[0] / cnt),
            "critic_loss": float(acc[1] / cnt),
            "entropy_loss": float(acc[2] / cnt),
            "max_ratio": float(acc[3]),
            "min_prob": float(acc[4]),
            "mean_ret": float(acc[6]),
        }

    def _action_to_device(self, action):
        if self.continuous:
            return torch.as_tensor(action, dtype=torch.float32, device=self.device).reshape(-1, self.action_size)
        return torch.as_tensor(np.asarray(action).reshape(-1), dtype=torch.int32, device=self.device)

    def learn(self):
        buf = self.memory.buffer
        batched = len(buf) > 0 and np.shape(buf[0]["reward"])[0] > 1
        tr = self.memory.sample_batched() if batched else self.memory.sample()
        dev = self.device
        n = len(tr["reward"])
        # host transitions land in PERSISTENT device buffers: captured CUDA graphs bake these pointers
        hin = getattr(self, "_host_in", None)
        if hin is None or hin["n"] != n:
            hin = {"n": n,
                   "state": torch.empty(n, *self._row_shape, dtype=self._row_dtype, device=dev),
                   "next_state": torch.empty(n, *self._row_shape, dtype=self._row_dtype, device=dev),
                   "reward": torch.empty(n, device=dev), "done": torch.empty(n, device=dev),
                   "action": (torch.empty(n, self.action_size, device=dev) if self.continuous
                              else torch.empty(n, dtype=torch.int32, device=dev))}
            self._host_in = hin
        hin["state"].copy_(self._state_rows(tr["state"]))
        hin["next_state"].copy_(self._state_rows(tr["next_state"]))
        hin["reward"].copy_(torch.as_tensor(tr["reward"], dtype=torch.float32, device=dev).reshape(-1))
        hin["done"].copy_(torch.as_tensor(tr["done"], dtype=torch.float32, device=dev).reshape(-1))
        hin["action"].copy_(self._action_to_device(tr["action"]))
        return self._learn_tensors(hin["state"], hin["action"], hin["reward"], hin["done"], next_state=hin["next_state"])

    def learn_rollout(self, rollout):
        """Resident path: `rollout` is a DeviceRollout filled by the batched collect loop."""
        N, T = rollout.N, rollout.T
        res = self._learn_tensors(rollout.state.view(N * T, *self._row_shape), rollout.action.view(N * T, -1) if self.continuous
                                  else rollout.action.view(N * T), rollout.reward.view(N * T),
                                  rollout.done.view(N * T), last_next_state=rollout.last_next_state)
        rollout.clear()
        return res

    def process(self, transitions, step):
        result = {}
        self.memory.store(transitions)
        delta_t = step - self.time_t
        self.time_t = step
        self.learn_stamp += delta_t
        if self.learn_stamp >= self.n_step:
            result = self.learn()
            if self.lr_decay:
                self.learning_rate_decay(step)
            self.learn_stamp = 0
        return result
