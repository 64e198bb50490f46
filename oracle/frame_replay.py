"""numpy restatement of the frame-deduplicated replay's store policy (jorldy_b200/core/buffer/frame_replay.py,
csrc/frame_replay.cu): candidate order, reuse or new, id assignment, reference tables and the overflow check.

The device pre-filters candidates by a hash; a frame is only reused after a byte comparison, so the hash never changes
a decision and is not restated here: a frame reuses the first entry of its actor's history (most recently used first)
that holds equal bytes and is still in the pool.
"""
import math

import numpy as np

HISTORY = 16
INT64_MAX = 2 ** 63 - 1


class FrameReplay:
    def __init__(self, buffer_size, frame_ratio=1.25):
        self.cap = int(buffer_size)
        self.F = max(1, int(math.ceil(frame_ratio * buffer_size)))
        self.pool = {}                      # pool row -> frame bytes
        self.next_id = 0
        self.overflow = False
        self.ref = None                     # [nf, cap, S] int64
        self.min_ref = np.full(self.cap, INT64_MAX, dtype=np.int64)
        self.hist = None                    # per actor: [(code, bytes)], most recently used first
        self.index = 0
        self.counter = 0
        self.counts = None                  # new frames per actor of the last store

    def store(self, steps):
        """steps: list of dicts field -> uint8 [rows, S, H, W] (the frame fields, in transition order)."""
        keys = list(steps[0].keys())
        rows = [s[keys[0]].shape[0] for s in steps]
        n = sum(rows)
        N = rows[0] if all(r == rows[0] for r in rows) else 1
        x = {k: np.concatenate([s[k] for s in steps]) for k in keys}
        S = x[keys[0]].shape[1]
        self.shape = x[keys[0]].shape[2:]
        K = len(keys) * S
        if self.ref is None:
            self.ref = np.zeros((len(keys), self.cap, S), dtype=np.int64)
        if self.hist is None or len(self.hist) != N:
            self.hist = [[] for _ in range(N)]
        frame = lambda row, k: x[keys[k // S]][row, k % S].tobytes()
        lo = self.next_id - self.F
        codes = np.zeros((n, K), dtype=np.int64)
        new = [[] for _ in range(N)]
        for r in range(N):
            h = self.hist[r]
            for t in range(n // N):
                row = t * N + r
                for k in range(K):
                    b = frame(row, k)
                    hit = next((w for w, (c, cb) in enumerate(h) if not (0 <= c < lo) and cb == b), None)
                    if hit is not None:
                        entry = h.pop(hit)
                    else:
                        entry = (-(len(new[r]) + 1), b)
                        new[r].append(b)
                        if len(h) == HISTORY:
                            h.pop()
                    h.insert(0, entry)
                    codes[row, k] = entry[0]
        counts = np.array([len(v) for v in new], dtype=np.int64)
        offs = np.concatenate([[0], np.cumsum(counts)[:-1]]).astype(np.int64)
        base, total = self.next_id, int(counts.sum())
        self.next_id += total
        self.counts = counts
        # overflow: neither a slot outside the rows being rewritten nor a reused frame of this store may reference an id
        # the new frames overwrite
        gone = base + total - self.F
        nw = min(n, self.cap)
        rewritten = np.zeros(self.cap, dtype=bool)
        rewritten[(self.index + np.arange(nw)) % self.cap] = True
        if total > self.F or np.any(self.min_ref[~rewritten] < gone) or np.any((codes >= 0) & (codes < gone)):
            self.overflow = True
        if not self.overflow:
            for r in range(N):
                for j, b in enumerate(new[r]):
                    self.pool[(base + offs[r] + j) % self.F] = b
        to_id = lambda c, r: c if c >= 0 else base + offs[r] + (-c - 1)
        for row in range(max(0, n - self.cap), n):
            r, pos = row % N, (self.index + row) % self.cap
            ids = [to_id(int(c), r) for c in codes[row]]
            for k, i in enumerate(ids):
                self.ref[k // S, pos, k % S] = i
            self.min_ref[pos] = min(ids)
        self.hist = [[(to_id(c, r), b) for c, b in h] for r, h in enumerate(self.hist)]
        self.index = (self.index + n) % self.cap
        self.counter = min(self.counter + n, self.cap)

    def gather(self, f, idx):
        """Stacks of field number f at ring slots idx -> uint8 [B, S, ...]."""
        out = [[np.frombuffer(self.pool[int(i) % self.F], dtype=np.uint8).reshape(self.shape) for i in self.ref[f, s]]
               for s in idx]
        return np.array(out, dtype=np.uint8)

    def pool_array(self, frame_bytes):
        """Pool as the device holds it: frames [F, frame_bytes], rows never written are zero."""
        out = np.zeros((self.F, frame_bytes), dtype=np.uint8)
        for row, b in self.pool.items():
            out[row] = np.frombuffer(b, dtype=np.uint8)
        return out
