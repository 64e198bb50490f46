"""Replay memory and speed of the frame-deduplicated layout (`frame_replay=True`) against the duplicated ring, on one GPU.

Prints one JSON line per measurement (and appends them to --out):
  1. rainbow_frames (64 actors, Rainbow, 1 M slots, B=32, update_period 4): both layouts built side by side with the same
     seeds, an equal prefill, then alternating timed rounds; replay bytes, ms per round, us per store() / gather_device
     (CUDA events), new frames per stored transition; every network parameter must be bit-identical afterwards.
  2. apex (256 actors, Ape-X, 2 M slots): the same, the two layouts one after the other (together they do not fit).
  3. apex with the frame layout alone at 8 M slots (the duplicated ring would need ~452 GB): >= 1 M transitions prefilled,
     then timed rounds.
The hyper-parameters are bench.py's ReplayWorkload ones.  The card's name and power limit are read in the same run.
"""
import argparse
import gc
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

FRAME = 84 * 84


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [x.strip() for x in q.split(",")]
    except Exception as e:                                     # the name still comes from the runtime
        name, power, clock = torch.cuda.get_device_name(0), f"unavailable ({type(e).__name__})", None
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def replay_bytes(mem):
    ts = [getattr(mem, a, None) for a in ("frames", "ref", "min_ref", "ctl", "_tree")]
    ts += [t for v in (mem.fields or {}).values() for t in (v if isinstance(v, list) else [v])]
    return sum(t.numel() * t.element_size() for t in ts if t is not None)


class Timed:
    """Wraps a bound method with CUDA events; durations are read after a synchronise."""

    def __init__(self, fn):
        self.fn, self.ev, self.on = fn, [], False

    def __call__(self, *a, **k):
        if not self.on:
            return self.fn(*a, **k)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = self.fn(*a, **k)
        e1.record()
        self.ev.append((e0, e1))
        return out

    def mean_us(self):
        return 1e3 * float(np.mean([a.elapsed_time(b) for a, b in self.ev])) if self.ev else None


class Arm:
    def __init__(self, cfg, slots, frame_replay, prefill):
        from bench import ReplayWorkload
        from jorldy_b200.core import Agent, Env
        from jorldy_b200.core.collect import ReplayCollector
        args = argparse.Namespace(n_envs=None, batch=None, buffer=slots, rounds=None)
        w = ReplayWorkload(cfg, args, 1)
        self.cfg, self.frame_replay, self.slots = cfg, frame_replay, slots
        torch.manual_seed(0)
        np.random.seed(0)
        self.env = Env("breakout", num_envs=w.n_actors, seed=0, id=0, device="cuda")
        self.agent = Agent(w.agent_name, state_size=[4, 84, 84], action_size=w.A, hidden_size=512, head="cnn",
                           buffer_size=slots, batch_size=w.B, n_step=w.n_step, start_train_step=0, device="cuda",
                           run_step=10 ** 8, num_workers=max(2, w.n_actors), seed=1234, frame_replay=frame_replay,
                           **w.agent_kw)
        self.rc = ReplayCollector(self.env, self.agent, w.update_period)
        if cfg == "apex":
            self.agent.set_actor_epsilons(w.n_actors, first_id=0, total=w.n_actors)
        mem = self.agent.memory
        self.store, self.gather = Timed(mem.store), Timed(mem.gather_device)
        mem.store, mem.gather_device = self.store, self.gather
        torch.cuda.synchronize()
        m0 = torch.cuda.memory_allocated()
        self.step = 0
        while mem.size < prefill:
            self.step, _ = self.rc.run_round(self.step)
        torch.cuda.synchronize()
        self.mem_delta = torch.cuda.memory_allocated() - m0
        self.prefilled = mem.buffer_counter
        self.round_ev = []
        self.store.on = self.gather.on = True
        self.frames0 = self._frames()

    def _frames(self):
        return int(self.agent.memory.ctl[0]) if self.frame_replay else None

    def round(self):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        self.step, res = self.rc.run_round(self.step)
        e1.record()
        self.round_ev.append((e0, e1))
        return res

    def report(self, rounds_timed):
        torch.cuda.synchronize()
        mem = self.agent.memory
        ms = [a.elapsed_time(b) for a, b in self.round_ev]
        rows_per_round = self.rc.update_period * self.env.num_envs
        out = {"config": self.cfg, "slots": self.slots, "frame_replay": self.frame_replay,
               "replay_bytes": replay_bytes(mem), "replay_bytes_per_slot": replay_bytes(mem) / self.slots,
               "memory_allocated_delta_bytes": self.mem_delta, "prefilled_transitions": self.prefilled,
               "timed_rounds": rounds_timed, "ms_per_round_mean": float(np.mean(ms)), "ms_per_round_median": float(np.median(ms)),
               "us_per_store": self.store.mean_us(), "us_per_gather_device": self.gather.mean_us(),
               "learns": self.agent.num_learn}
        if self.frame_replay:
            new = self._frames() - self.frames0
            out["new_frames_per_stored_transition"] = new / (rounds_timed * rows_per_round)
            out["pool_frames"] = mem.num_frames
            out["overflow"] = bool(int(mem.ctl[3]))
        return out


def emit(rec, fh):
    line = json.dumps(rec)
    print(line, flush=True)
    if fh:
        fh.write(line + "\n")
        fh.flush()


def free():
    gc.collect()                                               # an Arm's timed wrappers and its buffer form a cycle
    torch.cuda.empty_cache()


def params(agent):
    return {k: v.detach().clone().cpu() for k, v in agent.network.p.items()}


def same_params(pa, pb):
    return all(torch.equal(pa[k], pb[k]) for k in pa)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="append the JSON lines to this file")
    ap.add_argument("--rainbow-rounds", type=int, default=200)
    ap.add_argument("--apex-rounds", type=int, default=6)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--big-slots", type=int, default=8_000_000)
    ap.add_argument("--skip", default="", help="comma list of parts to skip: rainbow, apex, big")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_frame_replay.py measures on a CUDA device; none is available")
    from jorldy_b200 import build
    build.build()
    fh = open(a.out, "a") if a.out else None
    skip = set(a.skip.split(","))
    emit({"kind": "device", **gpu_info(), "torch": torch.__version__, "time": time.strftime("%Y-%m-%d %H:%M:%S")}, fh)
    ok = True

    if "rainbow" not in skip:
        off, on = Arm("rainbow_frames", 1_000_000, False, 20_000), Arm("rainbow_frames", 1_000_000, True, 20_000)
        for i in range(a.warmup + a.rainbow_rounds):
            if i == a.warmup:
                for arm in (off, on):
                    arm.round_ev, arm.store.ev, arm.gather.ev = [], [], []
                    arm.frames0 = arm._frames()
            ra, rb = off.round(), on.round()
            ok &= ra == rb
        r_off, r_on = off.report(a.rainbow_rounds), on.report(a.rainbow_rounds)
        same = same_params(params(off.agent), params(on.agent)) and ra == rb
        ok &= same
        for r in (r_off, r_on):
            emit({"kind": "layout", **r}, fh)
        emit({"kind": "compare", "config": "rainbow_frames", "params_bit_identical": same,
              "replay_bytes_ratio": r_off["replay_bytes"] / r_on["replay_bytes"],
              "ms_per_round_on_over_off": r_on["ms_per_round_median"] / r_off["ms_per_round_median"]}, fh)
        del off, on, arm
        free()

    if "apex" not in skip:
        recs, ps, res = [], [], []
        for fr in (False, True):
            arm = Arm("apex", 2_000_000, fr, 100_000)
            last = None
            for i in range(1 + a.apex_rounds):
                if i == 1:
                    arm.round_ev, arm.store.ev, arm.gather.ev = [], [], []
                    arm.frames0 = arm._frames()
                last = arm.round()
            recs.append(arm.report(a.apex_rounds))
            ps.append(params(arm.agent))
            res.append(last)
            del arm
            free()
        same = same_params(*ps) and res[0] == res[1]
        ok &= same
        for r in recs:
            emit({"kind": "layout", **r}, fh)
        emit({"kind": "compare", "config": "apex", "params_bit_identical": same,
              "replay_bytes_ratio": recs[0]["replay_bytes"] / recs[1]["replay_bytes"],
              "ms_per_round_on_over_off": recs[1]["ms_per_round_median"] / recs[0]["ms_per_round_median"]}, fh)

    if "big" not in skip:
        slots = a.big_slots
        t0 = time.time()
        arm = Arm("apex", slots, True, 1_000_000)
        prefill_s = time.time() - t0
        for i in range(1 + a.apex_rounds):
            if i == 1:
                arm.round_ev, arm.store.ev, arm.gather.ev = [], [], []
                arm.frames0 = arm._frames()
            arm.round()
        r = arm.report(a.apex_rounds)
        r["prefill_wall_s"] = prefill_s
        r["duplicated_layout_bytes_computed"] = slots * (2 * 4 * FRAME)
        r["peak_memory_allocated_bytes"] = torch.cuda.max_memory_allocated()
        ok &= not r["overflow"]
        emit({"kind": "capacity", **r}, fh)
        del arm
        free()

    emit({"kind": "done", "ok": bool(ok)}, fh)
    if fh:
        fh.close()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
