"""Frame-deduplicated replay for frame-stack observations (opt-in: the agents' `frame_replay=True`).

The duplicated ring keeps `state` and `next_state` of every slot as full [S, H, W] uint8 stacks (2 x 28 224 B for Atari),
although consecutive transitions of one actor share all but one of those frames.  Here every such field keeps only the S
frame ids of each slot (ref [nf, capacity, S] int64 + min_ref [capacity]); the frames themselves live once in a pool
frames [F, H*W] uint8, F = ceil(frame_ratio * buffer_size), id i at row i % F.  Every other field, the ring bookkeeping
and (FramePERBuffer) the sum-tree are the parents' own, so `gather_device` returns exactly the bytes of ReplayBuffer /
PERBuffer.

Store (csrc/frame_replay.cu): row t*N + r of a store([step_0, ..., step_{T-1}]) call, each step a batch of N rows, is
actor r at step t (the order of ReplayCollector / NStepAssembler); a list whose steps differ in size is one actor.  Each
incoming frame reuses a frame of its actor's history (the last 16 distinct frames it introduced or reused) only after a
byte comparison; otherwise it becomes a new frame.  A wrong guess about actors therefore costs pool space, never
correctness, and arbitrary uint8 data round-trips exactly.  New frames get ids actor-major in row order.  A change of the
actor count resets the histories.

Overflow: the store refuses to overwrite frames that a slot staying live still references and sets a sticky device flag
instead; `sample()` and the agents' learn() (through their one stats read) raise RuntimeError while it is set.
"""
import ctypes
import math

import numpy as np
import torch

from ..dev import C, ptr, stream_ptr
from .per_buffer import PERBuffer
from .replay_buffer import ReplayBuffer

HISTORY = 16                  # csrc/frame_replay.cu HIST
MAX_FIELDS = 4
_EMPTY = -(2 ** 63)
_INT64_MAX = 2 ** 63 - 1


def pool_frames(buffer_size, frame_ratio):
    """Frames in the pool of a `buffer_size`-slot replay."""
    return max(1, int(math.ceil(frame_ratio * buffer_size)))


def frame_stack(val):
    """(S, frame bytes) when a stored field is a uint8 stack [rows, S, H, W] (any further dims belong to the frame) whose
    frames are a multiple of 16 bytes, else None."""
    if isinstance(val, (list, tuple)):
        return None
    is_u8 = val.dtype == torch.uint8 if torch.is_tensor(val) else np.asarray(val).dtype == np.uint8
    shape = tuple(np.shape(val))
    if not is_u8 or len(shape) < 4:
        return None
    fb = int(np.prod(shape[2:]))
    return (shape[1], fb) if fb % 16 == 0 else None


class _FrameRing:
    """The frame layout shared by FrameReplayBuffer and FramePERBuffer (placed before the parent in the MRO)."""

    def __init__(self, *args, frame_ratio=1.25, **kwargs):
        super().__init__(*args, **kwargs)
        self.frame_ratio = float(frame_ratio)
        self.num_frames = pool_frames(self.buffer_size, self.frame_ratio)
        self.frame_keys = []
        self.frames = self.ref = self.min_ref = None
        # {next frame id, first id of the last store, its new frames, overflow flag}
        self.ctl = torch.zeros(4, dtype=torch.int64, device=self.device)
        self._hist = None

    # ---- storage ------------------------------------------------------------------------------
    def _allocate(self, transition):
        self._keys = list(transition.keys())
        stacks = {k: frame_stack(v) for k, v in transition.items()}
        first = next((s for s in stacks.values() if s is not None), None)
        self.frame_keys = [k for k, s in stacks.items() if s is not None and s == first][:MAX_FIELDS]
        super()._allocate({k: v for k, v in transition.items() if k not in self.frame_keys})
        if not self.frame_keys:
            return
        self.stack = tuple(transition[self.frame_keys[0]].shape[1:])
        self.S, self.frame_bytes = first
        for k in self.frame_keys:
            self._np_dtype[k] = None if torch.is_tensor(transition[k]) else np.dtype(np.uint8)
        self.frames = torch.zeros((self.num_frames, self.frame_bytes), dtype=torch.uint8, device=self.device)
        self.ref = torch.zeros((len(self.frame_keys), self.buffer_size, self.S), dtype=torch.int64, device=self.device)
        self.min_ref = torch.full((self.buffer_size,), _INT64_MAX, dtype=torch.int64, device=self.device)

    def _write(self, transitions):
        start = self.buffer_index
        n = super()._write(transitions)
        if self.frame_keys:
            self._store_frames(transitions, start, n)
        return n

    def _store_frames(self, transitions, start, n):
        rows = [int(np.shape(t[self.frame_keys[0]])[0]) for t in transitions]
        if sum(rows) != n:
            raise ValueError(f"frame fields hold {sum(rows)} rows but the transition holds {n}")
        N = rows[0] if all(r == rows[0] for r in rows) else 1
        src = [self._cat([t[k] for t in transitions], torch.uint8, self.device).contiguous() for k in self.frame_keys]
        for s in src:
            if tuple(s.shape[1:]) != self.stack:
                raise ValueError(f"frame stack shape changed from {self.stack} to {tuple(s.shape[1:])}")
        if self._hist is None or self._hist[0].shape[0] != N:
            self._hist = (torch.full((N, HISTORY), _EMPTY, dtype=torch.int64, device=self.device),
                          torch.zeros((N, HISTORY), dtype=torch.int64, device=self.device))
        hist_id, hist_h = self._hist
        nf, K = len(src), len(src) * self.S
        dev = self.device
        hashes = torch.empty(n * K, dtype=torch.int64, device=dev)
        codes = torch.empty(n * K, dtype=torch.int64, device=dev)
        newsrc = torch.empty(n * K, dtype=torch.int64, device=dev)
        counts = torch.empty(N, dtype=torch.int64, device=dev)
        offs = torch.empty(N, dtype=torch.int64, device=dev)
        fields = (ctypes.c_void_p * nf)(*[s.data_ptr() for s in src])
        F, cap, st = self.num_frames, self.buffer_size, stream_ptr()
        C.jb_frame_plan(ctypes.addressof(fields), nf, n, N, self.S, self.frame_bytes, ptr(self.frames), F, ptr(hashes),
                        ptr(self.ctl), ptr(hist_id), ptr(hist_h), ptr(codes), ptr(newsrc), ptr(counts), st)
        C.jb_frame_assign(ptr(counts), N, F, ptr(self.min_ref), cap, start, n, ptr(codes), n * K, ptr(offs), ptr(self.ctl), st)
        C.jb_frame_commit(ctypes.addressof(fields), nf, n, N, self.S, self.frame_bytes, ptr(self.frames), F, ptr(self.ctl),
                          ptr(counts), ptr(offs), ptr(newsrc), ptr(codes), ptr(self.ref), ptr(self.min_ref), cap, start,
                          ptr(hist_id), st)

    # ---- sampling -----------------------------------------------------------------------------
    def _gather_frames(self, f, idx):
        out = torch.empty((idx.shape[0],) + self.stack, dtype=torch.uint8, device=self.device)
        for off in range(0, idx.shape[0], self._MAX_ROWS):
            m = min(self._MAX_ROWS, idx.shape[0] - off)
            C.jb_frame_gather(ptr(self.frames), self.num_frames, self.frame_bytes, ptr(self.ref[f]), self.S,
                              ptr(idx[off:off + m]), m, ptr(out[off:off + m]), stream_ptr())
        return out

    def gather_device(self, idx):
        idx = idx.to(torch.int64).contiguous()
        out = super().gather_device(idx)
        for f, key in enumerate(self.frame_keys):
            out[key] = self._gather_frames(f, idx)
        return {k: out[k] for k in self._keys if k in out}

    # ---- overflow -----------------------------------------------------------------------------
    @property
    def overflow_flag(self):
        """int64 [1] device tensor, non-zero once a store found the pool too small."""
        return self.ctl[3:4]

    def raise_if_overflow(self, flag):
        if flag:
            raise RuntimeError(
                f"frame replay pool overflow: {self.num_frames} frames (frame_ratio={self.frame_ratio} x {self.buffer_size} "
                "slots) cannot hold every frame the live slots reference, so sampled stacks would no longer be exact. "
                "Build the buffer with a larger frame_ratio.")

    def sample(self, *args, **kwargs):
        out = super().sample(*args, **kwargs)
        self.raise_if_overflow(int(self.ctl[3].item()))
        return out

    @property
    def new_frames(self):
        """Frames stored so far (host read)."""
        return int(self.ctl[0].item())

    def replay_bytes(self):
        """Bytes of every device tensor this buffer owns."""
        ts = [self.frames, self.ref, self.min_ref, self.ctl, getattr(self, "_tree", None)]
        ts += [t for v in (self.fields or {}).values() for t in (v if isinstance(v, list) else [v])]
        return sum(t.numel() * t.element_size() for t in ts if t is not None)


class FrameReplayBuffer(_FrameRing, ReplayBuffer):
    """ReplayBuffer(buffer_size, device=None, frame_ratio=1.25) with frame-stack fields stored once per frame."""


class FramePERBuffer(_FrameRing, PERBuffer):
    """PERBuffer(buffer_size, uniform_sample_prob, device, seed, frame_ratio=1.25) with frame-stack fields stored once per
    frame."""
