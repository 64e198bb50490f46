"""Resident rollout collection: act -> env.step -> write transition, for every env at once, with
no host hop.  Replaces the per-actor loop of jorldy/manager/distributed_manager.py:76-92
(`Actor.run`) and its gather in run_mode.py:180-187: the N ray actors become N rows of one batched
launch sequence, and the whole T-step rollout is captured in ONE CUDA graph (per-row Philox
counters and the env's own episode counters advance on the device, so every replay draws fresh
randomness).
"""
import torch

from .buffer import DeviceRollout


class RolloutCollector:
    def __init__(self, env, agent, n_step=None, use_cuda_graph=True):
        self.env, self.agent = env, agent
        self.T = n_step or agent.n_step
        self.rollout = DeviceRollout(env.num_envs, self.T, env.state_size, env.action_size, env.action_type,
                                     device=agent.device)
        self.use_cuda_graph = use_cuda_graph
        self._graph = None
        # kernels of OUR library per env step: input head + gemm + heads_fwd per inference chunk of envs (one chunk of
        # mlp_in_fwd for the MLP head), then act + env_step (the rollout-row copies are torch plumbing and not counted)
        h = agent.network.head
        self.launches_per_collect = ((h.fwd_launches + 2) * -(-env.num_envs // h.max_rows) + 2) * self.T
        env.reset_device()

    def _collect_eager(self):
        env, agent, ro = self.env, self.agent, self.rollout
        ro.clear()
        for t in range(self.T):
            ro.state[:, t].copy_(env.obs)                      # state acted on (pre-step observation)
            action = agent.act_device(env.obs, training=True)
            next_obs, reward, done = env.step_device(action)   # env.obs <- post-reset observation
            ro.t = t
            ro.write_after_step(action, reward, done, next_obs)

    def collect(self):
        """Fills self.rollout with T steps of all envs; returns it."""
        if not self.use_cuda_graph:
            self._collect_eager()
            return self.rollout
        if self._graph is None:
            # warm-up (allocates workspaces) on a side stream, then capture the T-step sequence
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                self._collect_eager()
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self._collect_eager()
            self._graph = g
        self._graph.replay()
        self.rollout.t = self.T
        return self.rollout


class NStepAssembler:
    """Device-side n-step transition assembly for N batched envs.

    Same windows as the reference's per-actor deques — multistep.py:90-104 / rainbow.py:294-308 (window of
    n steps, next_state = last step's next_state) and ape_x.py:174-199 (window of n+1, next_state = the
    (n+1)-th step's state, actor-side priority |G_n - q_0|) — including their behaviour of NOT clearing at
    episode ends (windows straddle episodes and rely on the (1-done) mask).  One ring [N, L, ...] per field.
    """

    def __init__(self, n_step, apex=False, gamma=0.99):
        self.n, self.apex, self.gamma = n_step, apex, gamma
        self.L = n_step + 1 if apex else n_step
        self.hist, self.count, self.pos = None, 0, 0

    def push(self, tr):
        """tr: dict of device tensors with leading dim N.  Returns an assembled batch dict or None."""
        if self.hist is None:
            self.hist = {k: torch.zeros((v.shape[0], self.L) + tuple(v.shape[1:]), dtype=v.dtype, device=v.device)
                         for k, v in tr.items()}
        for k, v in tr.items():
            self.hist[k][:, self.pos].copy_(v)
        newest = self.pos
        self.pos = (self.pos + 1) % self.L
        self.count = min(self.count + 1, self.L)
        if self.count < self.L:
            return None
        oldest = self.pos                  # after the increment, pos points at the oldest entry
        order = [(oldest + i) % self.L for i in range(self.L)]
        h = self.hist
        out = {"state": h["state"][:, oldest].clone(), "action": h["action"][:, oldest].clone()}
        if self.apex:
            out["next_state"] = h["state"][:, newest].clone()
            steps = order[:-1]
        else:
            out["next_state"] = h["next_state"][:, newest].clone()
            steps = order
        sel = torch.as_tensor(steps, device=h["reward"].device)
        out["reward"] = h["reward"].index_select(1, sel).unsqueeze(-1)      # [N, n, 1]
        out["done"] = h["done"].index_select(1, sel).unsqueeze(-1)
        if self.apex:
            g = h["q"][:, newest].clone()
            for i in reversed(range(self.n)):
                s = steps[i]
                g = h["reward"][:, s] + (1 - h["done"][:, s]) * self.gamma * g
            out["priority"] = (g - h["q"][:, oldest]).abs().to(torch.float64).unsqueeze(-1)
        return out


class ReplayCollector:
    """Off-policy resident loop: `update_period` batched env steps feeding the HBM replay, then one
    agent.process() (the reference's sync loop, run_mode.py:180-187: one learn per round whatever the
    number of transitions that arrived — SURVEY.md row D3)."""

    def __init__(self, env, agent, update_period):
        self.env, self.agent, self.update_period = env, agent, update_period
        n = getattr(agent, "n_step", 1)
        apex = type(agent).__name__ == "ApeX"
        self.assembler = NStepAssembler(n, apex, agent.gamma) if (n > 1 or apex) else None
        if apex:
            agent.set_actor_epsilons(env.num_envs, total=max(agent.num_workers, env.num_envs, 2))
        env.reset_device()

    def run_round(self, step):
        env, agent = self.env, self.agent
        batches = []
        for _ in range(self.update_period):
            state = env.obs.clone()
            action, q_sel = agent.act_device(agent._net_input(state), True)
            next_obs, reward, done = env.step_device(action)
            tr = {"state": state, "action": action.view(action.shape[0], -1).clone(), "reward": reward.clone(), "done": done.clone(),
                  "next_state": next_obs.clone()}
            if self.assembler is not None:
                if self.assembler.apex:
                    tr["q"] = q_sel.clone()
                out = self.assembler.push({k: (v.view(v.shape[0]) if k in ("reward", "done") else v) for k, v in tr.items()})
                if out is not None:
                    batches.append(out)
            else:
                tr["reward"] = tr["reward"].view(-1, 1)
                tr["done"] = tr["done"].view(-1, 1)
                batches.append(tr)
        step += self.update_period
        result = agent.process(batches, step) if batches else {}
        return step, result
