#!/usr/bin/env python
"""Benchmark of the north-star hot path (rollout-collect -> buffer -> learn()) on B200.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--config NAME] [--dump-outputs DIR]

`--config` selects one of BASELINE.json's configurations; the default (what the driver runs) is configs[1]:

  ppo_cartpole    configs[1]  PPO CartPole, 4096 batched envs/GPU, T=128, minibatch 256/GPU, 3 epochs (weak scaling)
  ppo_continuous  configs[4]  PPO continuous obs 11 / act 3 (Hopper dimensions, synthetic dynamics), 8192 envs IN TOTAL,
                              T=2048, 10 epochs, global minibatch 2048 (<= 512 per GPU), Adam 3e-4 (strong scaling)
  rainbow_frames  configs[2]  Rainbow (C51+PER+n-step+Noisy, CNN) on synthetic 84x84x4 uint8 frames, 1M-slot HBM replay
  apex            configs[3]  Ape-X DQN (dueling CNN), 256 actors -> PER sharded over the ranks (32 actors + 250k slots per GPU
                              at 8 GPUs), RMSprop centred, gradient all-reduce

A "step" = one full iteration of the path on every rank:
  PPO      collect T steps of all envs (policy forward + sampling + physics + rollout write, all on the GPU), then learn():
           pre-pass, GAE, n_epoch x shuffled minibatch steps (one launch of the persistent kernel per epoch; at N > 1 the
           per-step gradient average happens inside that kernel over NVLink peer memory);
  replay   ROUNDS rounds of {update_period batched env steps -> n-step assembly -> replay store -> one learn()}.
`value` = env-steps/s over all ranks with inputs resident in HBM; `e2e` = the same loop driven through the
reference-shaped plugin API (agent.act / env.step / agent.interact_callback / agent.process) with HOST numpy buffers,
every host<->device copy inside the timed region.

`--impl reference` times the reference's CPU algorithm for the same path on the host cores (the oracle port: the
reference is pure Python and /root/reference does not travel to the GPU box) on a BOUNDED SAMPLE of the workload: its own
default worker count (8 actors; 1 for the replay agents), NOT the GPU arm's env count.  Its `config` is the GPU arm's
(the contract: "on your arm's config"); `reference_sample`, `reference_actors` and `cpu_baseline.sample` say what ran.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "env_steps_per_sec"
UNIT = "env-steps/s"
CONFIGS = ("ppo_cartpole", "ppo_continuous", "rainbow_frames", "apex", "sac_hopper")


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", type=str, default="b200")
    ap.add_argument("--config", type=str, default="ppo_cartpole", choices=CONFIGS)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the labelled scaled-minibatch variant")
    # shape overrides for quick functional runs (the line is then labelled "override": true and is NOT a config number)
    ap.add_argument("--n-envs", type=int, default=None)
    ap.add_argument("--n-step", type=int, default=None)
    ap.add_argument("--batch", type=int, default=None)
    ap.add_argument("--epochs", type=int, default=None)
    ap.add_argument("--buffer", type=int, default=None)
    ap.add_argument("--rounds", type=int, default=None)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    return args


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


# ------------------------------------------------------------------------------------------------
# clocks sampling (B200_PROFILING.md recipe)
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = sorted(float(r[1]) for r in self.rows if len(r) > 2 and r[1].replace(".", "").isdigit())
        mx = [float(r[2]) for r in self.rows if len(r) > 2 and r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = set()
        for r in self.rows:
            for i, n in enumerate(names):
                if len(r) > 5 + i and r[5 + i].lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


DUMP_MAX_ELEMS = 1 << 20                # per array: 4 MB in float32, 8 MB in float64
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir, arrays, result):
    """Writes each tensor of `arrays` and each number of `result` (as `result.<key>`) to out_dir/<name>.npy: floating
    data as float32, integers and scalars as float64.  An array of more than DUMP_MAX_ELEMS elements is replaced by the
    same seeded sample of that many of its elements (flattened, ascending index) on every run, so that two builds given
    the same arguments can be compared file by file."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    out = {}
    for name, t in arrays.items():
        flat = t.detach().reshape(-1)
        if flat.numel() > DUMP_MAX_ELEMS:
            idx = np.sort(np.random.RandomState(0).randint(0, flat.numel(), DUMP_MAX_ELEMS))
            flat = flat[torch.from_numpy(idx).to(flat.device)]
            a = flat.cpu().numpy()
        else:
            a = flat.cpu().numpy().reshape(tuple(t.shape))
        out[name] = a.astype(np.float32 if a.dtype.kind == "f" else np.float64)
    for k, v in result.items():
        if isinstance(v, (bool, int, float, np.number)):
            out[f"result.{k}"] = np.asarray(v, dtype=np.float64)
    total = sum(a.nbytes for a in out.values())
    if total > DUMP_MAX_BYTES:
        raise ValueError(f"--dump-outputs: {total} bytes exceed the {DUMP_MAX_BYTES}-byte budget")
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    return total


def load_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


# ================================================================================================
# PPO workloads (configs[1] and configs[4])
# ================================================================================================
class PPOWorkload:
    def __init__(self, name, args, world):
        self.name, self.world = name, world
        if name == "ppo_cartpole":
            self.env_name, self.D, self.A, self.continuous = "cartpole", 4, 2, False
            self.n_envs, self.T, self.B, self.epochs, self.lr = 4096, 128, 256, 3, 2.5e-4
            self.scaling = "weak"
            self.ref_cite = "config.ppo.cartpole hyper-parameters, distributed_batch_size 256"
        else:
            self.env_name, self.D, self.A, self.continuous = "hopper", 11, 3, True
            self.n_envs, self.T, self.epochs, self.lr = 8192 // world, 2048, 10, 3e-4
            self.B = min(512, 2048 // world)
            self.scaling = "strong"
            self.ref_cite = "config.ppo.mujoco hyper-parameters (T 2048, 10 epochs, Adam 3e-4), distributed_batch_size 2048 split over the ranks, <= 512 per GPU"
        self.override = any(v is not None for v in (args.n_envs, args.n_step, args.batch, args.epochs))
        self.n_envs = args.n_envs or self.n_envs
        self.T = args.n_step or self.T
        self.B = args.batch or self.B
        self.epochs = args.epochs or self.epochs
        self.H = 512
        self.nout = 2 * self.A + 1 if self.continuous else self.A + 1

    # ---- labels -------------------------------------------------------------------------------
    def config(self):
        w = self.world
        net = f"MLP {self.D}-512-512-({'2x' if self.continuous else ''}{self.A}+1)"
        if self.name == "ppo_cartpole":
            wl = (f"PPO CartPole, {self.n_envs} batched envs/GPU, T={self.T}, minibatch {self.B}/GPU, {self.epochs} epochs, {net} "
                  f"({self.ref_cite})")
        else:
            wl = (f"PPO continuous obs 11 / act 3 (Hopper dimensions, synthetic dynamics s'=tanh(Ws s + Wa a)+0.01 N), "
                  f"{self.n_envs * w} envs in total = {self.n_envs}/GPU, T={self.T}, minibatch {self.B}/GPU, {self.epochs} epochs, {net} "
                  f"({self.ref_cite})")
        c = {"workload": wl, "config_name": self.name, "n_envs_per_gpu": self.n_envs, "n_step": self.T,
             "batch_size_per_gpu": self.B, "n_epoch": self.epochs, "hidden": self.H, "parallelism": f"dp{w}",
             "gradient_exchange": "none (1 GPU)" if w == 1 else
             "in-kernel reduce-scatter + all-gather over NVLink peer memory, once per minibatch step (csrc/ppo_fused.cu, core/parallel.py)",
             "l2": "flushed between timed steps (256 MB fill, > 126 MB L2); every step re-collects its rollout"}
        if self.override:
            c["override"] = True
        return c

    def reference_sample(self):
        return (f"8 actors (the reference's default num_workers, config/ppo/cartpole.py:40) x T={self.T} steps + one PPO.learn() "
                f"(minibatch {self.B}, {self.epochs} epochs) per step on the host cores: a BOUNDED SAMPLE of the configuration named in "
                f"`config` (which is the GPU arm's: {self.n_envs} envs per GPU), not the same number of envs")

    # ---- GPU arm ------------------------------------------------------------------------------
    def build(self, torch, dev, rank):
        from jorldy_b200.core import Agent, Env
        from jorldy_b200.core.collect import RolloutCollector
        self.torch, self.dev, self.rank = torch, dev, rank
        self.env = Env(self.env_name, num_envs=self.n_envs, seed=0, id=rank, device=dev)
        kw = {"network": "continuous_policy_value"} if self.continuous else {}
        self.agent = Agent("ppo", state_size=self.D, action_size=self.A, hidden_size=self.H, batch_size=self.B, n_step=self.T,
                           n_epoch=self.epochs, optim_config={"name": "adam", "lr": self.lr}, device=dev, run_step=10 ** 9,
                           lr_decay=True, seed=1234, **kw)
        self.agent.rng_stream_base = rank << 32
        if self.world > 1:
            from jorldy_b200.core import parallel
            parallel.attach(self.agent, self.world)
        self.col = RolloutCollector(self.env, self.agent)
        self.l2_flush = torch.empty(64 * 1024 * 1024, dtype=torch.float32, device=dev)     # 256 MB > L2
        self.step_no = 0

    def step(self):
        self.l2_flush.fill_(float(self.step_no))
        ro = self.col.collect()
        res = self.agent.learn_rollout(ro)
        self.step_no += self.T
        self.agent.learning_rate_decay(self.step_no)
        return res

    def outputs(self):
        """What the last step handed back: the rollout collect() returned and the network learn() left."""
        ro = self.col.rollout
        out = {f"rollout.{k}": getattr(ro, k) for k in ("state", "action", "reward", "done", "last_next_state")}
        out.update({f"network.{k}": v for k, v in self.agent.network.p.items()})
        return out

    def env_steps_per_step(self):
        return self.n_envs * self.T * self.world

    def learner_transitions_per_step(self):
        return self.n_envs * self.T * self.world * self.epochs

    def launches_per_step(self):
        return self.col.launches_per_collect + self.agent.n_launches + self.agent.n_prepass_launches

    def teardown(self):
        self.agent._graphs.clear()
        self.col._graph = None

    # ---- roofline of the dominant kernel (collective at world > 1: every rank launches it) -----
    def roofline(self, peaks):
        torch, agent = self.torch, self.agent
        runner = agent._fused.get(self.B)
        if runner is None:
            return None
        n_mb = self.n_envs * self.T // self.B
        n_run = min(n_mb, 2048)
        times = []
        for i in range(5):
            agent._cursor.zero_()
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record(); runner.run(agent._st, n_run); a1.record(); torch.cuda.synchronize()
            if i >= 2:
                times.append(a0.elapsed_time(a1))
        dur_ms = sum(times) / len(times)
        flops = float(n_run) * self.B * 6.0 * (self.D * self.H + self.H * self.H + self.H * self.nout)   # fwd + 2x bwd (SURVEY 8d)
        peak = peaks.get("bf16_tflops_sustained", 1400.0)
        ach = flops / (dur_ms * 1e-3) / 1e12
        traffic = None
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "r02_ppo_epoch_kernel_traffic.json")))["dram_bytes_per_launch"]
        except Exception:
            pass
        ffma = 148 * 128 * 2 * 1.965e-3
        return {"kernel": f"ppo_epoch_kernel (persistent cooperative PPO minibatch loop, {n_run} steps/launch)", "bound": "tensor",
                "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
                "traffic": traffic if (self.name == "ppo_cartpole" and n_run == 2048) else None,
                "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained (of measured)" if peaks else "fallback 1400 (of fallback)",
                "algorithmic_flops_per_launch": flops, "ms_per_launch": dur_ms, "us_per_minibatch_step": 1e3 * dur_ms / n_run,
                "fp32_ffma_peak_tflops": ffma, "frac_of_fp32_ffma_peak": ach / ffma, "world": self.world,
                "note": "one launch = one epoch slice of sequential minibatch steps (forward, loss, backward, clip, Adam"
                        + (", gradient exchange over NVLink" if self.world > 1 else "") + "); the step is latency / grid-barrier "
                        "bound at the reference minibatch size (DESIGN.md 3b has the per-phase timeline); frac is against the "
                        "measured bf16 tensor peak as the contract asks, frac_of_fp32_ffma_peak against 148 SMs x 128 FMA/clk x 1.965 GHz"}

    # ---- labelled scaled-minibatch variant (SURVEY 8d: "and a labelled scaled variant (e.g. 16 384)") ----------------
    def extra(self):
        if self.name != "ppo_cartpole" or self.world != 1 or self.override:
            return None
        from jorldy_b200.core import Agent
        torch = self.torch
        B2 = 16384
        big = Agent("ppo", state_size=self.D, action_size=self.A, hidden_size=self.H, batch_size=B2, n_step=self.T,
                    n_epoch=self.epochs, optim_config={"name": "adam", "lr": self.lr}, device=self.dev, run_step=10 ** 9, seed=1234)
        for _ in range(2):
            big.learn_rollout(self.col.collect())
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n = 3
        e0.record()
        for _ in range(n):
            self.l2_flush.fill_(1.0)
            big.learn_rollout(self.col.collect())
        e1.record(); torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / n
        big._graphs.clear()
        return {"label": "scaled minibatch variant, NOT the headline: same rollout (4096 envs x T=128), minibatch 16384, 3 epochs x 32 "
                         "steps through the CUDA-graph path (tcgen05 forward GEMM + FFMA backward tiles)",
                "batch_size": B2, "ms_per_step": ms, "env_steps_per_sec": self.n_envs * self.T / (ms * 1e-3),
                "learner_transitions_per_sec": self.n_envs * self.T * self.epochs / (ms * 1e-3)}

    # ---- e2e through the plugin API ---------------------------------------------------------------
    def e2e(self, np, steps=2):
        import torch.distributed as dist
        from jorldy_b200.core import Agent, Env
        torch, dev, rank, world = self.torch, self.dev, self.rank, self.world
        N, T = self.n_envs, self.T
        env = Env(self.env_name, num_envs=N, seed=1, id=rank, device=dev)
        kw = {"network": "continuous_policy_value"} if self.continuous else {}
        agent = Agent("ppo", state_size=self.D, action_size=self.A, hidden_size=self.H, batch_size=self.B, n_step=T,
                      n_epoch=self.epochs, optim_config={"name": "adam", "lr": self.lr}, device=dev, run_step=10 ** 9, **kw)
        agent.rng_stream_base = rank << 32
        if world > 1:
            from jorldy_b200.core import parallel
            parallel.attach(agent, world)
        state = env.reset()
        cnt = {"h2d": 0, "d2h": 0, "step": 0}

        def iteration():
            nonlocal state
            res = {}
            for _ in range(T):
                action_dict = agent.act(state, True)                          # H2D state, D2H action
                next_state, reward, done = env.step(action_dict["action"])    # H2D action, D2H (ns, r, d)
                tr = {"state": state, "next_state": next_state, "reward": reward, "done": done}
                tr.update(action_dict)
                cnt["step"] += 1
                res = agent.process([tr], cnt["step"])                        # learn() fires on the T-th call: H2D rollout
                cnt["h2d"] += state.nbytes + action_dict["action"].nbytes
                cnt["d2h"] += action_dict["action"].nbytes + next_state.nbytes + 4 * N * 2
                state = env.obs.cpu().numpy()                                 # post-auto-reset observation
                cnt["d2h"] += state.nbytes
            return res

        iteration()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        cnt["h2d"] = cnt["d2h"] = 0
        t0 = time.perf_counter()
        for _ in range(steps):
            iteration()
        torch.cuda.synchronize()
        sec = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([sec], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            sec = float(t.item())
        act_bytes = 4 * self.A if self.continuous else 4
        roll_bytes = N * T * (4 * self.D * 2 + act_bytes + 4 + 4)             # rollout H2D at learn()
        return {"value": world * N * T * steps / sec, "unit": UNIT,
                "h2d_bytes_per_step": world * (cnt["h2d"] // steps + roll_bytes), "d2h_bytes_per_step": world * (cnt["d2h"] // steps + 28),
                "ms_per_step": 1e3 * sec / steps, "api": "Agent.act / Env.step / Agent.process (numpy, pageable host memory)"}

    # ---- reference arm / cpu baseline: the oracle port on host cores -------------------------------
    def cpu_run(self, n_workers, n_rollouts, threads):
        """run_mode.py:180-198 (sync mode) restated around the oracle: n_workers actors collect T transitions each with
        batch-1 policy forwards (Actor.run, distributed_manager.py:76-92), then one PPO.learn() (ppo.py:71-185)."""
        import numpy as np
        import torch
        from oracle import nets
        from oracle import ppo as oppo
        from oracle.classic_control import CartPoleBatch, SyntheticControlBatch
        torch.set_num_threads(threads)
        g = torch.Generator().manual_seed(0)
        H, D, A = self.H, self.D, self.A
        if self.continuous:
            shapes = {"head.l.weight": (H, D), "head.l.bias": (H,), "l.weight": (H, H), "l.bias": (H,), "mu.weight": (A, H),
                      "mu.bias": (A,), "log_std.weight": (A, H), "log_std.bias": (A,), "v.weight": (1, H), "v.bias": (1,)}
        else:
            shapes = {"head.l.weight": (H, D), "head.l.bias": (H,), "l.weight": (H, H), "l.bias": (H,),
                      "pi.weight": (A, H), "pi.bias": (A,), "v.weight": (1, H), "v.bias": (1,)}
        params = {}
        for k, s in shapes.items():
            params[k] = torch.zeros(s) if len(s) == 1 else torch.nn.init.orthogonal_(torch.empty(s), 0.01 if k.startswith("pi") else 1.0, generator=g)
        if self.continuous:
            from jorldy_b200.core.env.synth import synth_weights
            Ws, Wa = synth_weights(D, A, 0)
            envs = [SyntheticControlBatch(1, D, A, seed=0, stream_base=i << 32, auto_reset=False, Ws=Ws, Wa=Wa) for i in range(n_workers)]
        else:
            envs = [CartPoleBatch(1, seed=0, stream_base=i << 32, auto_reset=False) for i in range(n_workers)]
        states = [e.reset() for e in envs]
        hp = {"continuous": self.continuous, "n_step": self.T, "gamma": 0.99, "lambda": 0.95, "standardize": True,
              "batch_size": self.B, "n_epoch": self.epochs, "eps_clip": 0.1, "vf_coef": 1.0, "ent_coef": 0.01, "clip_grad_norm": 1.0}
        opt_state = None
        rs = np.random.RandomState(0)
        t0 = time.perf_counter()
        env_steps = 0
        for _ in range(n_rollouts):
            S, Ac, R, NS, Dn = [], [], [], [], []
            for w, env in enumerate(envs):                      # actor-major order
                for _t in range(self.T):
                    with torch.no_grad():
                        if self.continuous:
                            mu, std, _ = nets.continuous_policy_value(params, torch.from_numpy(states[w]))
                            a = torch.tanh(torch.normal(mu, std)).numpy()
                        else:
                            pi, _ = nets.discrete_policy_value(params, torch.from_numpy(states[w]))
                            a = torch.multinomial(pi, 1).numpy()
                    ns, r, d = env.step(a)
                    S.append(states[w]); Ac.append(a.astype(np.float32)); R.append(np.asarray(r, np.float32).reshape(1, 1)); NS.append(ns)
                    Dn.append(np.asarray(d, np.float32).reshape(1, 1))
                    states[w] = env.reset() if d[0] else ns
                    env_steps += 1
            batch = {"state": torch.from_numpy(np.concatenate(S)), "action": torch.from_numpy(np.concatenate(Ac)),
                     "reward": torch.from_numpy(np.concatenate(R)), "next_state": torch.from_numpy(np.concatenate(NS)),
                     "done": torch.from_numpy(np.concatenate(Dn))}
            NT = n_workers * self.T
            perms = [rs.permutation(NT) for _ in range(self.epochs)]
            out = oppo.learn(params, batch, hp, perms, lr=self.lr, opt_state=opt_state)
            params, opt_state = out["params"], out["opt_state"]
        return env_steps, time.perf_counter() - t0

    def cpu_sample_text(self, n_rollouts):
        return (f"8 {'synthetic Hopper-dimension' if self.continuous else 'CartPole'} actors x {self.T} steps + PPO.learn() "
                f"(batch {self.B}, {self.epochs} epochs) x {n_rollouts} rollout(s), torch-CPU oracle port of run_mode.py:180-198")


# ================================================================================================
# replay workloads (configs[2] Rainbow frames, configs[3] Ape-X)
# ================================================================================================
class ReplayWorkload:
    def __init__(self, name, args, world):
        self.name, self.world = name, world
        self.A, self.K = 4, 51                                     # Breakout's action set (README.md:84), 51 atoms
        if name == "rainbow_frames":
            # config/rainbow/atari.py:16-44
            self.n_actors, self.buffer, self.B, self.n_step, self.update_period = 64, 1_000_000, 32, 3, 4
            self.scaling = "weak"
            self.agent_kw = dict(alpha=0.5, beta=0.4, learn_period=4, uniform_sample_prob=1e-3, v_min=-1, v_max=10, num_support=51,
                                 target_update_period=10000, optim_config={"name": "adam", "lr": 6.25e-5})
            self.agent_name = "rainbow"
        else:
            # config/ape_x/atari.py:16-40,53-55 with num_workers = 256
            self.n_actors, self.buffer, self.n_step, self.update_period = 256 // world, 2_000_000 // world, 3, 100
            self.B = 512 // world
            self.scaling = "strong"
            self.agent_kw = dict(network="dueling", alpha=0.6, beta=0.4, learn_period=4, uniform_sample_prob=1e-3, clip_grad_norm=40.0,
                                 target_update_period=2500, epsilon=0.4, epsilon_alpha=7.0,
                                 optim_config={"name": "rmsprop", "lr": 6.25e-5, "eps": 1.5e-7, "centered": True})
            self.agent_name = "ape_x"
        self.override = any(v is not None for v in (args.n_envs, args.batch, args.buffer, args.rounds))
        self.n_actors = args.n_envs or self.n_actors
        self.B = args.batch or self.B
        self.buffer = args.buffer or self.buffer
        # one bench step = `rounds` rounds of {update_period env steps of every actor, one learn()}
        self.rounds = args.rounds or (32 if name == "rainbow_frames" else 2)
        self.prefill = max(4 * self.B, 2048)                         # transitions in the replay before timing starts

    def config(self):
        w = self.world
        if self.name == "rainbow_frames":
            wl = (f"Rainbow (C51 51 atoms + PER + 3-step + NoisyNet, CNN 4x84x84 -> 512, A=4) on synthetic uint8 frames, {self.n_actors} batched "
                  f"actors, {self.buffer}-slot HBM replay (state + next_state uint8 per slot), B={self.B}, learn every {self.update_period} "
                  f"steps of every actor (config.rainbow.atari hyper-parameters; start_train_step shortened to the prefill)")
        else:
            wl = (f"Ape-X DQN (dueling CNN, A=4), {self.n_actors * w} actors = {self.n_actors}/GPU with per-actor epsilons, PER sharded by rank "
                  f"({self.buffer} slots/GPU), global batch {self.B * w} = {self.B}/GPU, 3-step, RMSprop centred, clip 40, one learn per "
                  f"{self.update_period} steps of every actor (config.ape_x.atari hyper-parameters, num_workers 256)")
        c = {"workload": wl, "config_name": self.name, "n_actors_per_gpu": self.n_actors, "buffer_slots_per_gpu": self.buffer,
             "batch_size_per_gpu": self.B, "n_step": self.n_step, "update_period": self.update_period, "rounds_per_step": self.rounds,
             "parallelism": f"dp{w}", "gradient_exchange": "none (1 GPU)" if w == 1 else "ncclAllReduce(AVG) of the flat gradient per learn()",
             "l2": "inputs exceed L2: every learn() gathers fresh 56 KB/sample frame stacks from the multi-GB replay; 256 MB fill between steps"}
        if self.override:
            c["override"] = True
        return c

    def reference_sample(self):
        return ("ONE actor (batch-1 CNN act, n-step deque, python PER sum-tree capped at 20 000 slots) + learn() every 4 steps on the host "
                "cores: a BOUNDED SAMPLE of the configuration named in `config` (which is the GPU arm's), not the same actor count")

    def build(self, torch, dev, rank):
        from jorldy_b200.core import Agent, Env
        from jorldy_b200.core.collect import ReplayCollector
        self.torch, self.dev, self.rank = torch, dev, rank
        self.env = Env("breakout", num_envs=self.n_actors, seed=0, id=rank, device=dev)
        self.agent = Agent(self.agent_name, state_size=[4, 84, 84], action_size=self.A, hidden_size=512, head="cnn",
                           buffer_size=self.buffer, batch_size=self.B, n_step=self.n_step, start_train_step=0, device=dev,
                           run_step=10 ** 8, num_workers=max(2, self.n_actors * self.world), seed=1234, **self.agent_kw)
        self.agent.rng_stream_base = rank << 32
        if self.world > 1:
            from jorldy_b200.core import parallel
            parallel.attach(self.agent, self.world)
        self.rc = ReplayCollector(self.env, self.agent, self.update_period)
        if self.name == "apex":
            self.agent.set_actor_epsilons(self.n_actors, first_id=rank * self.n_actors, total=self.n_actors * self.world)
        self.l2_flush = torch.empty(64 * 1024 * 1024, dtype=torch.float32, device=dev)
        self.step_no = 0
        # prefill: rounds until the replay holds `prefill` transitions (learn() already runs once size >= B)
        while self.agent.memory.size < self.prefill:
            self.step_no, _ = self.rc.run_round(self.step_no)
        self.learns0 = self.agent.num_learn

    def step(self):
        self.l2_flush.fill_(float(self.step_no))
        res = {}
        for _ in range(self.rounds):
            self.step_no, r = self.rc.run_round(self.step_no)
            res = r or res
        return res

    def outputs(self):
        return {f"network.{k}": v for k, v in self.agent.network.p.items()}

    def env_steps_per_step(self):
        return self.n_actors * self.update_period * self.rounds * self.world

    def learner_transitions_per_step(self):
        # rainbow: learn_period 4 == update_period -> one learn per round; ape_x: one learn per process() call (run_mode.py:185)
        return self.B * self.world * self.rounds

    def launches_per_step(self):
        return None

    def teardown(self):
        pass

    def roofline(self, peaks):
        """Dominant cost of a replay learn(): the CNN forward x3 + backward (SURVEY 8d: ~100 MFLOP per sampled transition) —
        reported for one learn() timed alone on resident replay contents."""
        torch, agent = self.torch, self.agent
        times = []
        for i in range(8):
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record(); agent.learn(); a1.record(); torch.cuda.synchronize()
            if i >= 3:
                times.append(a0.elapsed_time(a1))
        ms = sum(times) / len(times)
        conv = 2.0 * (32 * 20 * 20 * 256 + 64 * 9 * 9 * 512 + 64 * 7 * 7 * 576)          # conv1..3 MACs x2 per frame stack
        if self.name == "rainbow_frames":
            fc = 2.0 * (3136 * 512 + 2 * 512 * 512 + 512 * (self.A * self.K) + 512 * self.K)
        else:
            fc = 2.0 * (2 * 3136 * 512 + 512 * self.A + 512)
        fwd = conv + fc
        flops = self.B * fwd * (3 + 2)                                # 3 forwards (s online, s' online, s' target) + backward = 2 forwards
        peak = peaks.get("bf16_tflops_sustained", 1400.0)
        ach = flops / (ms * 1e-3) / 1e12
        return {"kernel": "learn() of one minibatch: im2col + FFMA tile GEMMs (conv lowering, csrc/conv.cu + csrc/linear.cu) dominate; "
                          "per-kernel shares in profiles/r02_kernels.md", "bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s",
                "frac": ach / peak, "traffic": None,
                "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained (of measured)" if peaks else "fallback 1400 (of fallback)",
                "algorithmic_flops_per_launch": flops, "ms_per_learn": ms, "learner_transitions_per_sec_learn_only": self.B / (ms * 1e-3),
                "replay_gather_bytes_per_learn": self.B * (2 * 28224 + 8 * self.n_step + 8), "world": self.world,
                "note": "latency-bound at B=" + str(self.B) + ": ~60 launches per learn(); fp32 FFMA tiles, not tcgen05, for the minibatch-sized GEMMs"}

    def extra(self):
        return None

    # ---- e2e through the plugin API: numpy frames in / out, per-actor interact_callback deques -----
    def e2e(self, np, steps=1):
        import torch.distributed as dist
        from collections import deque
        from jorldy_b200.core import Agent, Env
        torch, dev, rank, world = self.torch, self.dev, self.rank, self.world
        N = self.n_actors
        env = Env("breakout", num_envs=N, seed=1, id=rank, device=dev)
        agent = Agent(self.agent_name, state_size=[4, 84, 84], action_size=self.A, hidden_size=512, head="cnn",
                      buffer_size=min(self.buffer, 65536), batch_size=self.B, n_step=self.n_step, start_train_step=0, device=dev,
                      run_step=10 ** 8, num_workers=max(2, N * world), seed=99, **self.agent_kw)
        if world > 1:
            from jorldy_b200.core import parallel
            parallel.attach(agent, world)
        if self.name == "apex":
            agent.set_actor_epsilons(N, first_id=rank * N, total=N * world)
        deques = [deque(maxlen=agent.tmp_buffer.maxlen) for _ in range(N)]
        state = env.reset()
        cnt = {"h2d": 0, "d2h": 0, "step": 0}
        rounds = max(1, self.rounds // 8)

        def one_round():
            nonlocal state
            batch = []
            for _ in range(self.update_period):
                ad = agent.act(state, True)                                   # H2D frames, D2H actions (+ q)
                next_state, reward, done = env.step(ad["action"])             # D2H next frames, reward, done
                cnt["h2d"] += state.nbytes + ad["action"].nbytes
                cnt["d2h"] += ad["action"].nbytes + next_state.nbytes + reward.nbytes + done.nbytes
                for i in range(N):                                            # one reference actor per row
                    tr = {"state": state[i:i + 1], "action": ad["action"][i:i + 1], "reward": reward[i:i + 1],
                          "done": done[i:i + 1], "next_state": next_state[i:i + 1]}
                    if "q" in ad:
                        tr["q"] = ad["q"][i:i + 1].reshape(1, 1)
                    agent.tmp_buffer = deques[i]
                    out = agent.interact_callback(tr)
                    if out:
                        batch.append(out)
                state = env.obs.cpu().numpy()
                cnt["d2h"] += state.nbytes
            cnt["step"] += self.update_period
            if batch:
                cnt["h2d"] += sum(sum(np.asarray(v).nbytes for v in t.values()) for t in batch)
                agent.process(batch, cnt["step"])                             # H2D the assembled transitions, learn()
                cnt["d2h"] += 32

        while agent.memory.size < 2 * self.B:
            one_round()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        cnt["h2d"] = cnt["d2h"] = 0
        t0 = time.perf_counter()
        for _ in range(steps * rounds):
            one_round()
        torch.cuda.synchronize()
        sec = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([sec], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            sec = float(t.item())
        n_steps_env = world * N * self.update_period * rounds * steps
        scale = self.rounds / rounds                                          # bytes per bench step (rounds_per_step rounds)
        return {"value": n_steps_env / sec, "unit": UNIT, "h2d_bytes_per_step": int(world * cnt["h2d"] / steps * scale),
                "d2h_bytes_per_step": int(world * cnt["d2h"] / steps * scale), "ms_per_step": 1e3 * sec / steps * scale,
                "rounds_timed": rounds * steps,
                "api": "Agent.act / Env.step / Agent.interact_callback (one deque per actor) / Agent.process (numpy, pageable host memory)"}

    # ---- reference arm: one actor, oracle port ------------------------------------------------------
    def cpu_run(self, n_workers, n_rollouts, threads):
        """run_mode.py:68-91 (single mode) restated around the oracle: act (batch-1 CNN forward) -> synthetic frame ->
        n-step deque -> PER store -> learn() every learn_period steps (rainbow.py:255-283 / ape_x.py:135-164)."""
        import numpy as np
        import torch
        from oracle import collect as oc
        from oracle import dqn as odqn
        from oracle import nets
        from oracle.per import SumTree
        sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
        import gen_inputs as G
        torch.set_num_threads(threads)
        rainbow = self.name == "rainbow_frames"
        case = dict(D=[4, 84, 84], A=self.A, H=512, K=self.K, head="cnn", seed=5, agent="rainbow" if rainbow else "ape_x",
                    net="rainbow" if rainbow else "dueling")
        params = {k: torch.from_numpy(v) for k, v in G.q_params(case).items()}
        tparams = {k: v.clone() for k, v in params.items()}
        hp = {"action_size": self.A, "gamma": 0.99, "n_step": self.n_step, "alpha": 0.5 if rainbow else 0.6, "clip": None if rainbow else 40.0,
              "noise": None, "net": "rainbow" if rainbow else "dueling", "double": True, "loss": "wmse", "order": "nstep"}
        if rainbow:
            hp.update(variant="rainbow", num_support=self.K, v_min=-1, v_max=10)
        optim = self.agent_kw["optim_config"]
        mem = SumTree(20000, 1e-3)
        store = []                                                # transition payloads by ring slot
        win = oc.NStepWindow(self.n_step, apex=not rainbow, gamma=0.99)
        rs = np.random.RandomState(0)
        frame = rs.randint(0, 256, size=(1, 4, 84, 84)).astype(np.uint8)
        opt_state = None
        n_timed = n_rollouts * (128 if rainbow else 32)
        layer_io = [(512, 512), (512, 512), (512, self.A * self.K), (512, self.K)]

        def draw_noise():                                         # network/utils.py:59-60: two randn per noisy layer
            return [(torch.randn(i), torch.randn(o)) for i, o in layer_io]

        t0, t_start, t = None, 0, -1
        while True:
            t += 1
            if t0 is None and mem.counter >= self.B:              # untimed prefill (random actions) until one batch is available
                t0, t_start = time.perf_counter(), t
            if t0 is not None and t - t_start >= n_timed:
                break
            x = torch.from_numpy(frame).float()
            with torch.no_grad():
                if t0 is None:
                    a, q0 = int(rs.randint(self.A)), 0.0
                elif rainbow:
                    a = int(oc.act_rainbow(params, x, self.A, self.K, -1, 10, draw_noise())[0, 0])   # fresh noise per forward
                    q0 = 0.0
                else:
                    q = nets.dueling(params, x).numpy()
                    a = int(np.argmax(q[0])) if rs.rand() > 0.1 else int(rs.randint(self.A))
                    q0 = float(q[0, a])
            nxt = np.concatenate([frame[:, 1:], rs.randint(0, 256, size=(1, 1, 84, 84)).astype(np.uint8)], axis=1)
            tr = {"state": frame, "action": np.array([[a]]), "reward": np.array([[float(rs.choice([-1, 0, 0, 0, 1]))]]),
                  "done": np.array([[rs.rand() < 1e-3]]), "next_state": nxt}
            if not rainbow:
                tr["q"] = np.array([[q0]], np.float32)
            out = win.push(tr)
            frame = nxt
            if out:
                slot = mem.tree_index - mem.first_leaf
                mem.store(1, [float(np.asarray(out["priority"]).reshape(-1)[0])] if "priority" in out else None)
                if slot < len(store):
                    store[slot] = out
                else:
                    store.append(out)
            if t0 is not None and t % 4 == 3:
                idx, w, _, _ = mem.sample(0.4, rs.rand(self.B), rs.rand(self.B))
                rows = [store[i - mem.first_leaf] for i in idx]
                batch = {k: torch.from_numpy(np.concatenate([r[k] for r in rows]).astype(np.float32)) for k in ("state", "next_state", "action", "reward", "done")}
                batch["weights"] = w
                if rainbow:
                    hp["noise"] = [draw_noise(), draw_noise(), draw_noise()]
                res = (odqn.dist_learn if rainbow else odqn.td_learn)(params, tparams, batch, hp, optim, opt_state=opt_state)
                params, opt_state = res["params"], res.get("opt_state")
                for i, p in zip(idx, np.asarray(res["priority"]).reshape(-1)):
                    mem.update(float(p), int(i))
        return n_timed, time.perf_counter() - t0

    def cpu_sample_text(self, n_rollouts):
        return (f"1 actor x {(128 if self.name == 'rainbow_frames' else 32) * n_rollouts} env steps (batch-1 CNN act, 3-step deque, python PER tree) + one learn() (B={self.B}) every 4 steps, "
                "torch-CPU oracle port of run_mode.py:68-91")


# ================================================================================================
# SURVEY 8f-4: the continuous off-policy family, measured on SAC (config/sac/mujoco.py) over the Hopper-dimension task
# ================================================================================================
class ACWorkload:
    """Not a BASELINE.json configuration: the measurement of the section-8f "next" row.  N batched actors step the
    synthetic obs-11 / act-3 task; every `update_period` steps of every actor the learner runs ONE SAC.learn() (the
    reference's sync loop, run_mode.py:180-187).  1024 actors x 2 steps = 2048 transitions per learn() — the data : update
    ratio of config/sac/mujoco.py's distributed setting (16 workers x update_period 128)."""

    def __init__(self, name, args, world):
        self.name, self.world = name, world
        self.D, self.A, self.H = 11, 3, 512
        self.n_actors, self.buffer, self.B, self.update_period = 1024, 1_000_000, 256, 2
        self.scaling = "weak"
        self.optim = {"actor": "adam", "critic": "adam", "alpha": "adam", "actor_lr": 5e-4, "critic_lr": 1e-3, "alpha_lr": 3e-4}
        self.override = any(v is not None for v in (args.n_envs, args.batch, args.buffer, args.rounds))
        self.n_actors = args.n_envs or self.n_actors
        self.B = args.batch or self.B
        self.buffer = args.buffer or self.buffer
        self.rounds = args.rounds or 64
        self.launch_estimate = None

    def config(self):
        c = {"workload": (f"SAC (dynamic alpha, twin critics, MLP 11-512-512, A=3) on the synthetic Hopper-dimension task, {self.n_actors} batched "
                          f"actors/GPU, {self.buffer}-slot HBM replay, B={self.B}, one learn() per {self.update_period} steps of every actor "
                          f"(config.sac.mujoco hyper-parameters; start_train_step shortened to the prefill; buffer enlarged from 50 000 to "
                          f"hold the batched actors' stream)"),
             "config_name": self.name, "n_actors_per_gpu": self.n_actors, "buffer_slots_per_gpu": self.buffer, "batch_size_per_gpu": self.B,
             "update_period": self.update_period, "rounds_per_step": self.rounds, "parallelism": f"replicas x{self.world}",
             "gradient_exchange": "none (independent replicas)",
             "l2": "256 MB fill between steps; every learn() gathers a fresh minibatch from the replay"}
        if self.override:
            c["override"] = True
        return c

    def reference_sample(self):
        return ("ONE actor (batch-1 policy forward, numpy env) x 128 steps then one SAC.learn() (B=256) per round on the host cores "
                "(config/sac/mujoco.py update_period 128): a BOUNDED SAMPLE of the configuration named in `config`, not the same actor count")

    def _agent(self, Agent, dev, seed, n_total):
        return Agent("sac", state_size=self.D, action_size=self.A, hidden_size=self.H, optim_config=dict(self.optim),
                     use_dynamic_alpha=True, gamma=0.99, tau=5e-3, buffer_size=self.buffer, batch_size=self.B, start_train_step=0,
                     run_step=10 ** 8, lr_decay=True, device=dev, seed=seed)

    def build(self, torch, dev, rank):
        from jorldy_b200.core import Agent, Env
        from jorldy_b200.core.collect import ReplayCollector
        self.torch, self.dev, self.rank = torch, dev, rank
        self.env = Env("hopper", num_envs=self.n_actors, seed=0, id=rank, device=dev)
        self.agent = self._agent(Agent, dev, 1234 + rank, self.n_actors)
        self.agent.rng_stream_base = rank << 32
        self.rc = ReplayCollector(self.env, self.agent, self.update_period)
        self.l2_flush = torch.empty(64 * 1024 * 1024, dtype=torch.float32, device=dev)
        self.step_no = 0
        while self.agent.memory.size < max(4 * self.B, 4096):
            self.step_no, _ = self.rc.run_round(self.step_no)
        # launches of OUR kernels per round, counted from the code path: per env step 3 (actor forward) + 1 (sample) + 1 (env) + 5
        # (replay row stores); per learn() 5 (gather) + 78 (forwards, losses, backwards, 4 Adam steps, soft updates, noise fills)
        self.launch_estimate = self.rounds * (10 * self.update_period + 83)

    def step(self):
        self.l2_flush.fill_(float(self.step_no))
        res = {}
        for _ in range(self.rounds):
            self.step_no, r = self.rc.run_round(self.step_no)
            res = r or res
        return res

    def outputs(self):
        out = {f"actor.{k}": v for k, v in self.agent.actor.p.items()}
        for i, c in enumerate(self.agent.critics):
            out.update({f"critic{i + 1}.{k}": v for k, v in c.p.items()})
        out["log_alpha"] = self.agent.log_alpha.flat[:1]
        return out

    def env_steps_per_step(self):
        return self.n_actors * self.update_period * self.rounds * self.world

    def learner_transitions_per_step(self):
        return self.B * self.world * self.rounds

    def launches_per_step(self):
        return self.launch_estimate

    def teardown(self):
        pass

    def extra(self):
        return None

    def roofline(self, peaks):
        """One learn() timed alone: 4 actor-forward equivalents (2 forwards + backward) and 12 critic-forward equivalents
        (2 online + 2 target + 2 on the actor's action, 2 full backwards = 4, 2 input-gradient-only backwards = 2)."""
        torch, agent = self.torch, self.agent
        times = []
        for i in range(13):
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record(); agent.learn(); a1.record(); torch.cuda.synchronize()
            if i >= 3:
                times.append(a0.elapsed_time(a1))
        ms = sum(times) / len(times)
        D, A, H = self.D, self.A, self.H
        actor = 2.0 * (D * H + H * H + H * 2 * A)
        critic = 2.0 * (D * H + A * H + 2 * H * H + H)
        flops = self.B * (4 * actor + 12 * critic)
        peak = peaks.get("bf16_tflops_sustained", 1400.0)
        ach = flops / (ms * 1e-3) / 1e12
        return {"kernel": "SAC.learn() of one minibatch: fp32 FFMA tile GEMMs (csrc/linear.cu) + the row kernels of csrc/actor_critic.cu",
                "bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak, "traffic": None,
                "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained (of measured)" if peaks else "fallback 1400 (of fallback)",
                "algorithmic_flops_per_launch": flops, "ms_per_learn": ms, "learner_transitions_per_sec_learn_only": self.B / (ms * 1e-3),
                "world": self.world, "cuda_graph": bool(agent._graphs),
                "note": f"latency-bound at B={self.B}: ~83 kernels of <= 0.5 GFLOP each per learn(), "
                        + ("replayed as one CUDA graph" if agent._graphs else "launched eagerly")}

    def e2e(self, np, steps=1):
        from jorldy_b200.core import Agent, Env
        torch, dev, rank = self.torch, self.dev, self.rank
        N, rounds = self.n_actors, max(1, self.rounds // 4)
        env = Env("hopper", num_envs=N, seed=1, id=rank, device=dev)
        agent = self._agent(Agent, dev, 99 + rank, N)
        state = env.reset()
        cnt = {"h2d": 0, "d2h": 0, "step": 0}

        def one_round():
            nonlocal state
            batch = []
            for _ in range(self.update_period):
                ad = agent.act(state, True)                                   # H2D state, D2H action
                ns, r, d = env.step(ad["action"])                             # H2D action, D2H (ns, r, d)
                batch.append({"state": state, "action": ad["action"], "reward": r, "done": d, "next_state": ns})
                cnt["h2d"] += state.nbytes + ad["action"].nbytes
                cnt["d2h"] += ad["action"].nbytes + ns.nbytes + 8 * N
                state = env.obs.cpu().numpy()                                 # post-auto-reset observation
                cnt["d2h"] += state.nbytes
                cnt["step"] += 1
            agent.process(batch, cnt["step"])                                 # H2D the transitions, learn(), D2H the stats
            cnt["h2d"] += sum(v.nbytes for tr in batch for v in tr.values())
            cnt["d2h"] += 40

        while agent.memory.size < 2 * self.B:
            one_round()
        torch.cuda.synchronize()
        cnt["h2d"] = cnt["d2h"] = 0
        t0 = time.perf_counter()
        for _ in range(steps * rounds):
            one_round()
        torch.cuda.synchronize()
        sec = time.perf_counter() - t0
        scale = self.rounds / rounds
        return {"value": self.world * N * self.update_period * rounds * steps / sec, "unit": UNIT,
                "h2d_bytes_per_step": int(self.world * cnt["h2d"] / steps * scale), "d2h_bytes_per_step": int(self.world * cnt["d2h"] / steps * scale),
                "ms_per_step": 1e3 * sec / steps * scale, "rounds_timed": rounds * steps,
                "api": "Agent.act / Env.step / Agent.process (numpy, pageable host memory)"}

    def cpu_run(self, n_workers, n_rollouts, threads):
        """run_mode.py:180-198 around the oracle: one actor collects 128 transitions with batch-1 policy forwards, then one
        SAC.learn() (sac.py:162-260) on a uniform minibatch of the python-list replay."""
        import numpy as np
        import torch
        from oracle import actor_critic as oac
        from oracle.classic_control import SyntheticControlBatch
        from jorldy_b200.core.env.synth import synth_weights
        sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
        import gen_inputs as G
        torch.set_num_threads(threads)
        case = dict(D=self.D, A=self.A, H=self.H, agent="sac", seed=7)
        nets = {n: {k: torch.from_numpy(v) for k, v in G.ac_params(case, n).items()} for n in ("actor", "critic1", "critic2")}
        nets["target_critic1"] = {k: v.clone() for k, v in nets["critic1"].items()}
        nets["target_critic2"] = {k: v.clone() for k, v in nets["critic2"].items()}
        Ws, Wa = synth_weights(self.D, self.A, 0)
        env = SyntheticControlBatch(1, self.D, self.A, seed=0, stream_base=0, auto_reset=False, Ws=Ws, Wa=Wa)
        state = env.reset()
        hp = {"gamma": 0.99, "tau": 5e-3, "actor_lr": 5e-4, "critic_lr": 1e-3, "alpha_lr": 3e-4, "use_dynamic_alpha": True,
              "target_entropy": -self.A}
        log_alpha = torch.zeros(1)
        alpha = log_alpha.exp()
        ring, opt_state, rs = [], None, np.random.RandomState(0)
        n_rounds = 8 * n_rollouts
        t0, env_steps = None, 0
        for rnd in range(n_rounds + 2):                              # 2 untimed rounds fill the replay past one batch
            if rnd == 2:
                t0, env_steps = time.perf_counter(), 0
            for _t in range(128):
                with torch.no_grad():
                    mu, std = oac.continuous_policy(nets["actor"], torch.from_numpy(state))
                    a = torch.tanh(torch.normal(mu, std)).numpy()
                ns, r, d = env.step(a)
                ring.append((state, a.astype(np.float32), np.asarray(r, np.float32).reshape(1, 1), ns, np.asarray(d, np.float32).reshape(1, 1)))
                state = env.reset() if d[0] else ns
                env_steps += 1
            if rnd < 1:
                continue
            idx = rs.randint(len(ring), size=self.B)
            cols = list(zip(*[ring[i] for i in idx]))
            batch = {k: torch.from_numpy(np.concatenate(c)) for k, c in zip(("state", "action", "reward", "next_state", "done"), cols)}
            o = oac.sac_learn(nets["actor"], nets["critic1"], nets["critic2"], nets["target_critic1"], nets["target_critic2"], log_alpha,
                              alpha, batch, hp, torch.randn(self.B, self.A), torch.randn(self.B, self.A), opt_state)
            nets.update(actor=o["actor"], critic1=o["critic1"], critic2=o["critic2"])
            nets["target_critic1"] = oac.soft_update(nets["target_critic1"], o["critic1"], hp["tau"])
            nets["target_critic2"] = oac.soft_update(nets["target_critic2"], o["critic2"], hp["tau"])
            log_alpha, alpha, opt_state = o["log_alpha"], o["alpha"], o["opt_state"]
        return env_steps, time.perf_counter() - t0

    def cpu_sample_text(self, n_rollouts):
        return (f"1 actor x {128 * 8 * n_rollouts} env steps (batch-1 policy forward, numpy synthetic env) + one SAC.learn() (B={self.B}) per 128 steps, "
                "torch-CPU oracle port of run_mode.py:180-198")


def make_workload(name, args, world):
    if name == "sac_hopper":
        return ACWorkload(name, args, world)
    return PPOWorkload(name, args, world) if name.startswith("ppo") else ReplayWorkload(name, args, world)


# ------------------------------------------------------------------------------------------------
def args_config_is_ppo(wl):
    return wl.name.startswith("ppo")


def best_cpu_threads(wl, workers):
    """The reference is torch-eager with tiny (batch-1 / minibatch) ops: more intra-op threads than the box can really
    schedule make it SLOWER.  To time the reference at its best, try a few thread counts on one short rollout each."""
    avail = host_cores()
    # 1 thread and "all cores" are both far from the optimum for these op sizes (measured: 1 -> 20x slower, 128 -> 200x
    # slower than 8 on the GPU box's host) and would eat minutes of a bounded baseline: sweep the plausible range only
    cands = sorted({c for c in ((4, 8, 16) if args_config_is_ppo(wl) else (8, 16, 32)) if 1 <= c <= avail}) or [min(avail, 4)]
    best, best_rate, tried = cands[0], 0.0, {}
    for c in cands:
        st, sec = wl.cpu_run(workers, 1, c)
        tried[c] = round(st / sec, 1)
        if st / sec > best_rate:
            best, best_rate = c, st / sec
    return best, tried


def run_reference(args, rank):
    if rank != 0:
        return
    wl = make_workload(args.config, args, 1)
    workers = 8
    threads, tried = best_cpu_threads(wl, workers)          # also serves as warm-up
    tot_steps = tot_sec = 0.0
    for _ in range(args.steps):
        st, sec = wl.cpu_run(workers, 1, threads)
        tot_steps += st; tot_sec += sec
    value = tot_steps / tot_sec
    sample = wl.cpu_sample_text(1) + f" per step; {threads} torch intra-op threads (fastest of env-steps/s by thread count {tried})"
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * tot_sec / args.steps, "higher_is_better": True,
            "scaling": wl.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": make_workload(args.config, args, max(1, args.gpus)).config(),      # the GPU arm's config at this N
            "reference_sample": wl.reference_sample(), "reference_actors": 8 if args.config.startswith("ppo") else 1,
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": host_cores(), "threads": threads, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
def main():
    args = parse()
    rank = int(os.environ.get("RANK", 0))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    from jorldy_b200._lib import LIB_PATH

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    # network initialisation, minibatch permutations and replay sampling draw from the global generators: seeding them
    # gives every run with the same arguments the same inputs
    torch.manual_seed(0)
    np.random.seed(0)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    trace_all = os.environ.get("JB_BENCH_TRACE", "0") == "1"

    def log(msg):
        if rank == 0 or trace_all:
            print(f"[bench {time.strftime('%H:%M:%S')} r{rank}] {msg}", file=sys.stderr, flush=True)

    wl = make_workload(args.config, args, world)
    log(f"world={world} config={args.config}: build")
    wl.build(torch, dev, rank)
    log(f"warm-up ({args.warmup} steps; the first one captures the CUDA graphs)")
    res = {}
    for _w in range(args.warmup):
        res = wl.step()
        if trace_all:
            torch.cuda.synchronize()
            log(f"warm-up step {_w} done")
    log("timing")
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(args.steps):
        res = wl.step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        n = dump_outputs(args.dump_outputs, wl.outputs(), res)
        log(f"outputs of the last timed step ({n} bytes) written to {args.dump_outputs}")
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.barrier()
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    ms_per_step = ms / args.steps
    value = wl.env_steps_per_step() * args.steps / (ms / 1e3)
    learner_tps = wl.learner_transitions_per_step() * args.steps / (ms / 1e3)
    launches = wl.launches_per_step()
    launches = args.steps * launches if launches is not None else None

    peaks = load_peaks()
    log("roofline (dominant kernel timed alone, every rank)")
    roof = wl.roofline(peaks)
    extra = None
    if not args.no_extra:
        extra = wl.extra()
    e2e = None
    if not args.no_e2e:
        log("e2e (plugin API, host numpy buffers) on every rank")
        e2e = wl.e2e(np)
    if rank == 0:
        cpu_base = None
        if not args.no_cpu and world == 1:
            log("cpu baseline (oracle port, bounded sample)")
            threads, tried = best_cpu_threads(wl, 8)
            n_roll = 3 if args.config == "ppo_cartpole" else 1
            st, sec = wl.cpu_run(8, n_roll, threads)
            cpu_base = {"value": st / sec, "unit": UNIT, "cores": host_cores(), "threads": threads, "kind": "port",
                        "sample": wl.cpu_sample_text(n_roll) + f"; fastest thread count of {tried}"}
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": wl.scaling,
                "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": wl.config(),
                "learner_transitions_per_sec": learner_tps, "clocks": clocks, "e2e": e2e, "gpu_launches": launches,
                "roofline": roof, "cpu_baseline": cpu_base, "lib": os.path.relpath(LIB_PATH, ROOT),
                "last_result": res}
        if launches is None:
            line["gpu_launches"] = getattr(wl, "launch_estimate", None)
        if extra:
            line["scaled_minibatch_variant"] = extra
        print(json.dumps(line), flush=True)
    if world > 1:
        # NCCL ops captured inside CUDA graphs make destroy_process_group() hang: drop the graphs, meet at a
        # barrier, flush, and leave without the collective teardown.
        wl.teardown()
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


if __name__ == "__main__":
    try:
        main()
    except BaseException as _e:      # every rank reports its own failure: torchrun's summary carries no traceback
        if not isinstance(_e, SystemExit) or _e.code not in (0, None):
            import traceback
            sys.stderr.write(f"[bench rank {os.environ.get('RANK', 0)}] FAILED: {type(_e).__name__}: {_e}\n{traceback.format_exc()}\n")
            sys.stderr.flush()
        raise
