"""The frame-deduplicated replay's store policy (oracle/frame_replay.py) on hand-built streams: shifted stacks, reset tiling,
n-step windows that straddle episodes, the Ape-X (n+1) window, random frames, the overflow check, and pool sizing."""
import numpy as np
import pytest

from oracle.collect import NStepWindow
from oracle.frame_replay import FrameReplay

S = 4


def _frame(actor, k):
    """A 16-byte frame (4x4) that no other (actor, k) shares."""
    return np.array([actor, k], dtype=np.int64).view(np.uint8).reshape(4, 4)


def frame_steps(n_actors, steps, dones=()):
    """Per-step batches of a frames env: stacks shift by one frame per step, next_state is the pre-reset stack, and a
    reset stack is one fresh frame tiled S times.  dones: set of (actor, step) that end an episode."""
    k = [0] * n_actors
    stack = []
    for a in range(n_actors):
        stack.append(np.stack([_frame(a, 0)] * S))
        k[a] = 1
    out = []
    for t in range(steps):
        st, nx, dn = [], [], []
        for a in range(n_actors):
            s = stack[a]
            n = np.concatenate([s[1:], _frame(a, k[a])[None]])
            k[a] += 1
            d = (a, t) in dones
            st.append(s), nx.append(n), dn.append(d)
            if d:
                stack[a] = np.stack([_frame(a, k[a])] * S)
                k[a] += 1
            else:
                stack[a] = n
        out.append({"state": np.stack(st), "next_state": np.stack(nx), "done": np.array(dn, dtype=np.float32)})
    return out


def assemble(batches, n_step, apex):
    """ReplayCollector + NStepAssembler order: one batch per step, row r = actor r."""
    if n_step == 1 and not apex:
        return [{"state": b["state"], "next_state": b["next_state"]} for b in batches]
    N = batches[0]["state"].shape[0]
    wins = [NStepWindow(n_step, apex=apex) for _ in range(N)]
    out = []
    for b in batches:
        rows = []
        for a in range(N):
            tr = {"state": b["state"][a:a + 1], "action": np.zeros((1, 1)), "reward": np.zeros(1), "done": b["done"][a:a + 1],
                  "next_state": b["next_state"][a:a + 1]}
            if apex:
                tr["q"] = np.zeros(1)
            rows.append(wins[a].push(tr))
        if rows[0]:
            out.append({k: np.concatenate([r[k] for r in rows]) for k in ("state", "next_state")})
    return out


def _check_exact(ora, stored):
    """Every live slot gathers the stacks that were stored into it."""
    cap = ora.cap
    rows = np.concatenate([s["state"] for s in stored]), np.concatenate([s["next_state"] for s in stored])
    n = rows[0].shape[0]
    live = np.arange(max(0, n - cap), n)
    slots = live % cap
    for f in range(2):
        np.testing.assert_array_equal(ora.gather(f, slots), rows[f][live])


def _distinct_frames(stored, N):
    seen = set()
    for s in stored:
        for key in ("state", "next_state"):
            for r in range(s[key].shape[0]):
                for fr in s[key][r]:
                    seen.add(fr.tobytes())
    return len(seen)


def test_shift_stream_stores_one_new_frame_per_transition():
    ora = FrameReplay(64, 2.0)
    stored = assemble(frame_steps(3, 10), 1, False)
    ora.store(stored[:4])
    # first row of an actor: the reset frame (tiled) + the next frame; then one new frame per row
    np.testing.assert_array_equal(ora.counts, [2 + 3] * 3)
    ora.store(stored[4:])
    np.testing.assert_array_equal(ora.counts, [6] * 3)
    assert ora.next_id == 3 * 11
    _check_exact(ora, stored)
    assert not ora.overflow


def test_reset_stack_is_one_frame_with_four_references():
    ora = FrameReplay(8)
    stored = assemble(frame_steps(1, 1), 1, False)
    ora.store(stored)
    np.testing.assert_array_equal(ora.ref[0, 0], [0, 0, 0, 0])        # state: the reset frame tiled
    np.testing.assert_array_equal(ora.ref[1, 0], [0, 0, 0, 1])        # next_state: shifted, one new frame
    assert ora.min_ref[0] == 0 and ora.next_id == 2


def test_ids_are_actor_major_in_row_order():
    ora = FrameReplay(16)
    ora.store(assemble(frame_steps(2, 2), 1, False))
    # actor 0 introduces ids 0..2 (reset frame, two next frames), actor 1 ids 3..5; row t*2 + r is actor r
    np.testing.assert_array_equal(ora.ref[1, 0], [0, 0, 0, 1])
    np.testing.assert_array_equal(ora.ref[1, 1], [3, 3, 3, 4])
    np.testing.assert_array_equal(ora.ref[1, 2], [0, 0, 1, 2])
    np.testing.assert_array_equal(ora.ref[0, 3], [3, 3, 3, 4])


@pytest.mark.parametrize("n_step,apex", [(1, False), (3, False), (3, True)])
def test_nstep_windows_straddling_episodes_are_exact_and_store_each_frame_once(n_step, apex):
    dones = {(0, 5), (1, 6), (2, 7), (0, 9), (1, 30), (2, 31), (0, 50)}
    ora = FrameReplay(40, 2.0)
    stored = assemble(frame_steps(3, 64), n_step, apex)
    for i in range(0, len(stored), 4):
        ora.store(stored[i:i + 4])
        _check_exact(ora, stored[:i + 4])
    assert not ora.overflow
    assert ora.next_id == _distinct_frames(stored, 3)


def test_random_frames_round_trip():
    rs = np.random.RandomState(0)
    ora = FrameReplay(30, 8.0)
    stored = [{"state": rs.randint(0, 256, (5, S, 4, 8), dtype=np.uint8),
               "next_state": rs.randint(0, 256, (5, S, 4, 8), dtype=np.uint8)} for _ in range(12)]
    for i in range(0, 12, 3):
        ora.store(stored[i:i + 3])
        np.testing.assert_array_equal(ora.counts, [3 * 2 * S] * 5)
        _check_exact(ora, stored[:i + 3])
    assert not ora.overflow


def test_ragged_step_sizes_are_one_actor():
    ora = FrameReplay(16, 4.0)
    st = frame_steps(3, 2)
    stored = [st[0], {k: v[:2] for k, v in st[1].items()}]
    ora.store([{"state": s["state"], "next_state": s["next_state"]} for s in stored])
    assert ora.counts.shape == (1,)
    _check_exact(ora, [{"state": s["state"], "next_state": s["next_state"]} for s in stored])


def test_overflow_when_live_slots_need_more_frames_than_the_pool():
    rs = np.random.RandomState(1)
    mk = lambda: {"state": rs.randint(0, 256, (4, S, 4, 4), dtype=np.uint8),
                  "next_state": rs.randint(0, 256, (4, S, 4, 4), dtype=np.uint8)}
    ora = FrameReplay(16, 2.0)                 # 32 frames; random rows need 8 each
    ora.store([mk()])
    assert not ora.overflow                    # 32 new frames, nothing older is live
    ora.store([mk()])
    assert ora.overflow                        # the first 4 rows are still live and their frames would be overwritten
    ora2 = FrameReplay(4, 1.0)
    ora2.store([mk()])
    assert ora2.overflow                       # one store needs more frames than the pool has


def test_pool_sizing():
    from jorldy_b200.core.buffer.frame_replay import HISTORY, pool_frames
    import oracle.frame_replay as ofr
    assert pool_frames(1_000_000, 1.25) == 1_250_000
    assert pool_frames(3, 1.25) == 4
    assert pool_frames(10, 0.01) == 1
    assert pool_frames(8_000_000, 1.25) * 84 * 84 == 70_560_000_000     # ~71 GB of frames at 8 M slots
    assert FrameReplay(1_000_000).F == pool_frames(1_000_000, 1.25)
    assert HISTORY == ofr.HISTORY
