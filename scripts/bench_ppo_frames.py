"""Speed of PPO with the CNN head on synthetic 4x84x84 uint8 frames (config.ppo.atari in sync mode), on one GPU.

For N in --envs (default 32, 512, 4096) batched envs and T = 128: the agent of config.ppo.atari with its sync-mode
minibatch (batch_size = distributed_batch_size = 1024), a RolloutCollector (the T-step collect captured in one CUDA
graph) and learn_rollout().  After --warmup rounds, collect() and learn_rollout() are timed separately with CUDA events
over --rounds rounds; medians and spread are reported.  FLOPs are the algorithm's, computed here from the layer shapes
(multiply-add = 2 FLOP): per stack forward = conv1 + conv2 + conv3 + l + pi/v heads, backward = 2x forward without
conv1's input gradient.  One env step costs act (1 forward) + pre-pass (1 forward) + n_epoch x (forward + backward).
Prints one JSON line per measurement and appends them to --out; the card's name, power limit and max SM clock are read
in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

STACK = (4, 84, 84)
A = 4                      # breakout's action set
H = 512


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                       capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
    name, power, clock = [x.strip() for x in q[1].split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def layer_flops():
    """Multiply-add FLOPs per stack of each layer: (name, forward, input-gradient flops)."""
    c, h, w = STACK
    out = []
    for name, ci, co, k, s in (("conv1", c, 32, 8, 4), ("conv2", 32, 64, 4, 2), ("conv3", 64, 64, 3, 1)):
        h, w = (h - k) // s + 1, (w - k) // s + 1
        f = 2 * h * w * co * ci * k * k
        out.append((name, f, 0 if name == "conv1" else f))
    feat = 64 * h * w
    out.append(("l", 2 * feat * H, 2 * feat * H))
    out.append(("heads", 2 * H * (A + 1), 2 * H * (A + 1)))
    return out


def flops_per_stack():
    ls = layer_flops()
    fwd = sum(f for _, f, _ in ls)
    bwd = sum(f + dx for _, f, dx in ls)          # weight gradient (= forward) + input gradient
    return fwd, bwd, {n: f for n, f, _ in ls}


def im2col_bytes_per_stack():
    c, h, w = STACK
    oh, ow = (h - 8) // 4 + 1, (w - 8) // 4 + 1
    return oh * ow * c * 8 * 8 * 4


def run(N, T, rounds, warmup, cfg):
    from jorldy_b200.core import Agent, Env
    from jorldy_b200.core.collect import RolloutCollector
    torch.manual_seed(0)
    np.random.seed(0)
    env = Env("breakout", num_envs=N, seed=0, id=0, device="cuda", **cfg.env)
    agent_cfg = dict(cfg.agent, batch_size=cfg.train["distributed_batch_size"], n_step=T)
    agent = Agent(state_size=env.state_size, action_size=env.action_size, optim_config=cfg.optim,
                  run_step=cfg.train["run_step"], num_workers=N, device="cuda", **agent_cfg)
    col = RolloutCollector(env, agent)
    ev = []
    for i in range(warmup + rounds):
        e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        e[0].record()
        ro = col.collect()
        e[1].record()
        res = agent.learn_rollout(ro)
        e[2].record()
        if i >= warmup:
            ev.append(e)
    torch.cuda.synchronize()
    collect_ms = np.array([a.elapsed_time(b) for a, b, _ in ev])
    learn_ms = np.array([b.elapsed_time(c) for _, b, c in ev])
    NT, B = N * T, agent.batch_size
    n_mb = agent.n_epoch * -(-NT // B)
    fwd, bwd, per_layer = flops_per_stack()
    collect_flop = NT * fwd
    learn_flop = NT * (fwd + agent.n_epoch * (fwd + bwd))
    ro = col.rollout
    rollout_bytes = sum(t.numel() * t.element_size() for t in (ro.state, ro.action, ro.reward, ro.done, ro.last_next_state))
    spread = lambda x: {"median": float(np.median(x)), "min": float(x.min()), "max": float(x.max())}
    cm, lm = float(np.median(collect_ms)), float(np.median(learn_ms))
    return {"kind": "ppo_frames", "envs": N, "n_step": T, "batch_size": B, "n_epoch": agent.n_epoch, "rounds": rounds,
            "warmup": warmup, "collect_ms": spread(collect_ms), "learn_ms": spread(learn_ms),
            "ms_per_minibatch_step": lm / n_mb, "minibatch_steps_per_learn": n_mb,
            "env_steps_per_s": NT / (cm * 1e-3), "learner_transitions_per_s": NT / (lm * 1e-3),
            "end_to_end_env_steps_per_s": NT / ((cm + lm) * 1e-3),
            "rollout_bytes": rollout_bytes, "rollout_state_bytes_per_env_step": ro.state[0, 0].numel(),
            "collect_flop_per_s": collect_flop / (cm * 1e-3), "learn_flop_per_s": learn_flop / (lm * 1e-3),
            "learn_finite": bool(all(np.isfinite(v) for v in res.values()))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", default="32,512,4096")
    ap.add_argument("--n-step", type=int, default=128)
    ap.add_argument("--rounds", default="10,5,3", help="timed rounds per --envs entry")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "ppo_frames_b200.jsonl"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_ppo_frames.py measures on a CUDA device; none is available")
    from jorldy_b200 import config
    cfg = config.load("config.ppo.atari")
    fwd, bwd, per_layer = flops_per_stack()
    T = a.n_step
    recs = [{"kind": "device", **gpu_info(), "torch": torch.__version__, "time": time.strftime("%Y-%m-%d %H:%M:%S")},
            {"kind": "shapes", "forward_flop_per_stack": fwd, "backward_flop_per_stack": bwd,
             "forward_flop_by_layer": per_layer, "flop_per_env_step_3_epochs": 2 * fwd + 3 * (fwd + bwd),
             "conv1_im2col_bytes_per_stack": im2col_bytes_per_stack(),
             "rollout_state_bytes_per_env_step_uint8": int(np.prod(STACK)),
             "rollout_state_bytes_per_env_step_f32": 4 * int(np.prod(STACK)),
             "rollout_state_gb_at_4096x128_uint8": 4096 * T * int(np.prod(STACK)) / 1e9,
             "rollout_state_gb_at_4096x128_f32": 4096 * T * 4 * int(np.prod(STACK)) / 1e9}]
    with open(a.out, "a") as fh:
        for r in recs:
            print(json.dumps(r), flush=True)
            fh.write(json.dumps(r) + "\n")
        for N, R in zip([int(x) for x in a.envs.split(",")], [int(x) for x in a.rounds.split(",")]):
            r = run(N, T, R, a.warmup, cfg)
            print(json.dumps(r), flush=True)
            fh.write(json.dumps(r) + "\n")
            fh.flush()
            torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
