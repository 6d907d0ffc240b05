"""numpy restatement of the Go-Explore cell archive (include/agarcl_b200.h, agarcl_batch_set_archive): the cell key, the
candidates, the winner of a key, the numbering of new entries, replacement, the selection weights and draws, and the
trajectory base.  The device kernels (archive_kernel.cu) are checked against it after every step."""
import bisect
import math

import numpy as np

from gpu_parity_lib import philox4x32_10_np

SELECT_TAG = 0x41524348  # counter word 1 of a selection draw


def centroid(sv, agent):
    """(cx, cy, total mass) of an agent as agarcl_batch_draw's agent view (and oracle_draw) computes it: fp32 sums in cell order
    of x * (float)mass, over (float)(u32 total mass); None without cells"""
    nc = min(max(int(sv.players["n_cells"][agent]), 0), sv.layout.cap_cells)
    sx, sy, m = np.float32(0), np.float32(0), 0
    for c in sv.cells[agent][:nc]:
        mf = np.float32(int(c["mass"]))
        sx = np.float32(sx + np.float32(c["x"] * mf))
        sy = np.float32(sy + np.float32(c["y"] * mf))
        m = (m + int(c["mass"])) & 0xFFFFFFFF
    if nc == 0 or m == 0:
        return None
    return np.float32(sx / np.float32(m)), np.float32(sy / np.float32(m)), m


def bin_of(c, n, W):
    """clamp((int)(c * (float)n / W), 0, n - 1), each operation one rounded fp32 operation, the conversion truncating"""
    v = np.float32(np.float32(c * np.float32(n)) / np.float32(W))
    return min(max(int(np.trunc(v)), 0), n - 1)


def cell_key(sv, agent, n, W):
    """key (mb * n + by) * n + bx of the agent's cell, -1 without cells"""
    c = centroid(sv, agent)
    if c is None:
        return -1
    cx, cy, m = c
    mb = m.bit_length() - 1
    return (mb * n + bin_of(cy, n, W)) * n + bin_of(cx, n, W)


def weight(chosen):
    """floor(2^20 / (1 + isqrt(chosen))): Go-Explore's 1 / sqrt(C + 1) in integers"""
    return (1 << 20) // (1 + math.isqrt(int(chosen)))


def draw_word(seed, instance, c):
    """the u64 x of draw c of global instance `instance`: words 0 | 1 << 32 of Philox4x32-10 with counter (c, SELECT_TAG,
    instance, 0) and key (seed low, seed high)"""
    w = philox4x32_10_np([c, SELECT_TAG, instance, 0], [int(seed) & 0xFFFFFFFF, (int(seed) >> 32) & 0xFFFFFFFF])
    return int(w[0]) | int(w[1]) << 32


class ArchiveModel:
    def __init__(self, N, A, K, n, agent, W, seed=0, instance_base=0, select=True):
        self.N, self.A, self.K, self.n, self.agent, self.W = N, A, K, n, agent, W
        self.seed, self.instance_base, self.select_on = seed, instance_base, select
        keys = 32 * n * n
        self.cell_of = np.full(N, -1, np.int32)
        self.base_score = np.zeros(N, np.float64)
        self.base_length = np.zeros(N, np.int64)
        self.draws = np.zeros(N, np.int64)
        self.key_entry = np.full(keys, -1, np.int32)
        self.visits = np.zeros(keys, np.uint32)
        self.entry_key = np.full(K, -1, np.int32)
        self.entry_score = np.zeros(K, np.float64)
        self.entry_length = np.zeros(K, np.int64)
        self.entry_chosen = np.zeros(K, np.uint32)
        self.used = self.dropped = self.improved = 0

    def update(self, svs, dones, rewards, ret, steps):
        """one step_autoreset: svs the games after the step (before any reset), dones the game's u8 [N*A] (before the step
        limit), rewards f64 [N*A], ret the episode returns before the step f64 [N*A], steps the episode steps before the step
        [N].  Returns {entry: instance} of the games saved into the pool."""
        A, a = self.A, self.agent
        cands = []
        for i, sv in enumerate(svs):
            key = cell_key(sv, a, self.n, self.W)
            self.cell_of[i] = key
            if key < 0 or dones[i * A:(i + 1) * A].any():
                continue
            s = float(self.base_score[i]) + (float(ret[i * A + a]) + float(rewards[i * A + a]))
            length = int(self.base_length[i]) + int(steps[i]) + 1
            self.visits[key] += 1
            cands.append((key, s, length, i))
        best = {}
        for key, s, length, i in cands:  # highest s, then lowest l (capped at 2^32 - 1, as the device orders it), then lowest i
            rank = (-s, min(length, 0xFFFFFFFF), i)
            if key not in best or rank < best[key][0]:
                best[key] = (rank, s, length, i)
        saves = {}
        for _, s, length, i in sorted(best.values(), key=lambda w: w[3]):
            key = self.cell_of[i]
            e = int(self.key_entry[key])
            if e >= 0:
                if not (s > self.entry_score[e] or (s == self.entry_score[e] and length < self.entry_length[e])):
                    continue
                self.improved += 1
            elif self.used < self.K:
                e = self.used
                self.used += 1
                self.key_entry[key] = e
                self.entry_key[e] = key
            else:
                self.dropped += 1
                continue
            self.entry_score[e], self.entry_length[e] = s, length
            saves[e] = i
        return saves

    def select(self, mask):
        """the picks of a reset of the instances in `mask` (select = 1): {instance: slot or -1}; the counts grow afterwards"""
        used = self.used
        if not self.select_on or not np.asarray(mask).any():
            return {}
        prefix = list(np.cumsum([weight(self.entry_chosen[e]) for e in range(used)], dtype=np.uint64).tolist())
        picks = {}
        for i in np.flatnonzero(mask):
            if used == 0:
                picks[int(i)] = -1
                continue
            x = draw_word(self.seed, self.instance_base + int(i), int(self.draws[i])) % int(prefix[-1])
            picks[int(i)] = bisect.bisect_right(prefix, x)
            self.draws[i] += 1
        for e in picks.values():
            if e >= 0:
                self.entry_chosen[e] += 1
        return picks

    def set_base(self, mask, started_from):
        """the trajectory base of the reset (or restored) instances in `mask`: started_from {instance: slot of the archive's
        pool it started from (start result 1)}; every other one restarts at (0, 0)"""
        for i in np.flatnonzero(mask):
            e = started_from.get(int(i), -1)
            ok = 0 <= e < self.used
            self.base_score[i] = self.entry_score[e] if ok else 0.0
            self.base_length[i] = self.entry_length[e] if ok else 0

    def arrays(self):
        """the read-out of agarcl_batch_archive, as numpy arrays"""
        return {"cell_of": self.cell_of, "base_score": self.base_score, "base_length": self.base_length,
                "key_entry": self.key_entry, "visits": self.visits, "entry_key": self.entry_key, "entry_score": self.entry_score,
                "entry_length": self.entry_length, "entry_chosen": self.entry_chosen,
                "counters": np.array([self.used, self.dropped, self.improved], np.uint64)}
