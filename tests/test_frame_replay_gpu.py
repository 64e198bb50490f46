"""Frame-deduplicated replay (csrc/frame_replay.cu, core/buffer/frame_replay.py) against the duplicated ring it replaces:
every gathered stack bit-identical, device tables equal to oracle/frame_replay.py, PER sampling and whole agents unchanged,
overflow reported on the host, and runs reproducible."""
import numpy as np
import pytest
import torch

from oracle.frame_replay import FrameReplay

pytestmark = pytest.mark.gpu

N_ACTORS, CAP = 16, 1500


def env_rounds(n_step, apex, rounds, n_actors=N_ACTORS, update_period=4, seed=0):
    """Per round the list ReplayCollector.run_round hands to process(): frames env, n-step assembly, step-major rows."""
    from jorldy_b200.core import Env
    from jorldy_b200.core.collect import NStepAssembler
    env = Env("breakout", num_envs=n_actors, seed=seed)
    env.reset_device()
    asm = NStepAssembler(n_step, apex) if (n_step > 1 or apex) else None
    g = torch.Generator(device="cuda").manual_seed(seed)
    for _ in range(rounds):
        batches = []
        for _ in range(update_period):
            state = env.obs.clone()
            q = torch.rand(n_actors, device="cuda", generator=g)
            next_obs, reward, done = env.step_device()
            tr = {"state": state, "action": torch.randint(0, 4, (n_actors, 1), device="cuda", generator=g),
                  "reward": reward.clone(), "done": done.clone(), "next_state": next_obs.clone()}
            if asm is None:
                tr["reward"], tr["done"] = tr["reward"].view(-1, 1), tr["done"].view(-1, 1)
                batches.append(tr)
                continue
            if apex:
                tr["q"] = q
            out = asm.push(tr)
            if out is not None:
                batches.append(out)
        if batches:
            yield batches


def _assert_same_gather(a, b, idx):
    ga, gb = a.gather_device(idx), b.gather_device(idx)
    assert list(ga.keys()) == list(gb.keys())
    for k in ga:
        assert torch.equal(ga[k], gb[k]), k


def _assert_tables(buf, ora):
    torch.cuda.synchronize()
    assert int(buf.ctl[0]) == ora.next_id and int(buf.ctl[2]) == int(ora.counts.sum())
    assert bool(buf.ctl[3]) == ora.overflow
    assert np.array_equal(buf.ref.cpu().numpy(), ora.ref)
    assert np.array_equal(buf.min_ref.cpu().numpy(), ora.min_ref)


@pytest.mark.parametrize("n_step,apex", [(1, False), (3, False), (3, True)], ids=["n1", "rainbow_n3", "apex_n3"])
def test_env_stream_bit_exact_and_tables_match_oracle(n_step, apex):
    from jorldy_b200.core.buffer import FrameReplayBuffer, ReplayBuffer
    ref, buf, ora = ReplayBuffer(CAP, device="cuda"), FrameReplayBuffer(CAP, device="cuda"), FrameReplay(CAP)
    rows = 0
    for batches in env_rounds(n_step, apex, rounds=3 * CAP // (4 * N_ACTORS) + 8):
        batches = [{k: v for k, v in b.items() if k != "priority"} for b in batches]
        ref.store(batches)
        buf.store(batches)
        ora.store([{k: b[k].cpu().numpy() for k in ("state", "next_state")} for b in batches])
        rows += sum(b["state"].shape[0] for b in batches)
        assert (buf.buffer_index, buf.buffer_counter) == (ref.buffer_index, ref.buffer_counter)
        _assert_same_gather(ref, buf, torch.arange(buf.buffer_counter, device="cuda"))
        _assert_tables(buf, ora)
    assert rows >= 3 * CAP
    assert np.array_equal(buf.frames.cpu().numpy(), ora.pool_array(84 * 84))
    # the shift contract holds: about one new frame per stored transition (plus one per reset and per actor start)
    assert buf.new_frames < 1.05 * rows + 8 * N_ACTORS


def test_random_stacks_and_changing_actor_counts():
    from jorldy_b200.core.buffer import FrameReplayBuffer, ReplayBuffer
    cap = 200
    ref, buf, ora = ReplayBuffer(cap, device="cuda"), FrameReplayBuffer(cap, device="cuda", frame_ratio=10.0), FrameReplay(cap, 10.0)
    g = torch.Generator(device="cuda").manual_seed(5)
    prev = None
    for i, n_act in enumerate([3, 3, 5, 1, 7, 7, 2, 4, 4, 4, 6, 3, 3, 8, 8, 8, 5]):
        steps = []
        for t in range(3):
            st = torch.randint(0, 256, (n_act, 4, 16, 16), dtype=torch.uint8, device="cuda", generator=g)
            if i % 2 and prev is not None and prev.shape[0] == n_act:     # sometimes a shifted stack: partly reused frames
                st = torch.cat([prev[:, 1:], st[:, :1]], 1)
            nx = torch.cat([st[:, 1:], torch.randint(0, 256, (n_act, 1, 16, 16), dtype=torch.uint8, device="cuda", generator=g)], 1)
            steps.append({"state": st, "action": torch.zeros(n_act, 1, dtype=torch.int64, device="cuda"),
                          "reward": torch.zeros(n_act, 1, device="cuda"), "next_state": nx})
            prev = nx
        ref.store(steps)
        buf.store(steps)
        ora.store([{k: s[k].cpu().numpy() for k in ("state", "next_state")} for s in steps])
        _assert_same_gather(ref, buf, torch.arange(buf.buffer_counter, device="cuda"))
        _assert_tables(buf, ora)
    assert not ora.overflow
    assert np.array_equal(buf.frames.cpu().numpy(), ora.pool_array(256))
    # numpy input and sample() go through the same layout
    s = buf.sample(8)
    assert s["state"].dtype == np.uint8 and s["state"].shape == (8, 4, 16, 16)


def test_per_buffers_sample_identically():
    from jorldy_b200.core.buffer import FramePERBuffer, PERBuffer
    a, b = PERBuffer(CAP, 1e-3, device="cuda", seed=7), FramePERBuffer(CAP, 1e-3, device="cuda", seed=7)
    g = torch.Generator(device="cuda").manual_seed(1)
    for i, batches in enumerate(env_rounds(3, True, rounds=40)):
        a.store(batches)
        b.store(batches)
        if a.size < 64:
            continue
        ta, wa, ia, sa = a.sample_device(0.4 + 0.01 * i, 64)
        tb, wb, ib, sb = b.sample_device(0.4 + 0.01 * i, 64)
        assert torch.equal(ia, ib) and torch.equal(wa, wb) and torch.equal(sa, sb)
        for k in ta:
            assert torch.equal(ta[k], tb[k]), k
        p = torch.rand(64, dtype=torch.float64, device="cuda", generator=g) + 0.01
        a.update_priorities(ia, p)
        b.update_priorities(ib, p)
    assert torch.equal(a._tree, b._tree)
    ra, rb = a.sample(0.5, 16), b.sample(0.5, 16)
    assert all(np.array_equal(x, y) for x, y in zip(ra[1:3], rb[1:3])) and ra[3:] == rb[3:]
    assert all(np.array_equal(ra[0][k], rb[0][k]) for k in ra[0])


@pytest.mark.parametrize("name", ["rainbow", "ape_x"])
def test_agents_identical_with_and_without_frame_replay(name):
    from jorldy_b200.core import Agent, Env
    from jorldy_b200.core.buffer import FramePERBuffer
    from jorldy_b200.core.collect import ReplayCollector

    def run(frame_replay):
        torch.manual_seed(0)
        np.random.seed(0)
        kw = dict(network="dueling", clip_grad_norm=40.0) if name == "ape_x" else dict(v_min=-1, v_max=10)
        agent = Agent(name, state_size=[4, 84, 84], action_size=4, hidden_size=512, head="cnn", buffer_size=1024,
                      batch_size=32, n_step=3, start_train_step=0, run_step=10 ** 6, num_workers=16, seed=1234,
                      frame_replay=frame_replay, device="cuda", **kw)
        assert isinstance(agent.memory, FramePERBuffer) == frame_replay
        rc = ReplayCollector(Env("breakout", num_envs=16, seed=3), agent, 4)
        step, results = 0, []
        for _ in range(24):
            step, r = rc.run_round(step)
            results.append(r)
        torch.cuda.synchronize()
        return agent, results

    a, ra = run(False)
    b, rb = run(True)
    assert a.num_learn > 10 and ra == rb
    for k, v in a.network.p.items():
        assert torch.equal(v, b.network.p[k]), k


def test_overflow_raises_on_the_host():
    from jorldy_b200.core import Agent, Env
    from jorldy_b200.core.buffer import FramePERBuffer, FrameReplayBuffer
    from jorldy_b200.core.collect import ReplayCollector
    buf = FrameReplayBuffer(64, device="cuda", frame_ratio=0.5)
    mk = lambda: {"state": torch.randint(0, 256, (8, 4, 16, 16), dtype=torch.uint8, device="cuda"),
                  "reward": torch.zeros(8, 1, device="cuda"),
                  "next_state": torch.randint(0, 256, (8, 4, 16, 16), dtype=torch.uint8, device="cuda")}
    buf.store([mk()])                                  # 64 new frames into a 32-frame pool
    with pytest.raises(RuntimeError, match="frame_ratio"):
        buf.sample(4)
    agent = Agent("rainbow", state_size=[4, 84, 84], action_size=4, hidden_size=64, head="cnn", buffer_size=512,
                  batch_size=32, n_step=3, start_train_step=0, run_step=10 ** 6, seed=1, frame_replay=True, device="cuda")
    agent.memory = FramePERBuffer(512, 1e-3, device="cuda", seed=1, frame_ratio=0.3)
    rc = ReplayCollector(Env("breakout", num_envs=16, seed=0), agent, 4)
    step = 0
    with pytest.raises(RuntimeError, match="frame_ratio"):
        for _ in range(40):
            step, _ = rc.run_round(step)


def test_two_runs_build_identical_pools_and_tables():
    from jorldy_b200.core.buffer import FrameReplayBuffer
    bufs = []
    for _ in range(2):
        buf = FrameReplayBuffer(CAP, device="cuda")
        for batches in env_rounds(3, False, rounds=30):
            buf.store(batches)
        bufs.append(buf)
    a, b = bufs
    assert torch.equal(a.frames, b.frames) and torch.equal(a.ref, b.ref) and torch.equal(a.min_ref, b.min_ref)
    assert torch.equal(a.ctl, b.ctl) and torch.equal(a._hist[0], b._hist[0])
