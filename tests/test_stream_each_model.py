"""CPU model of a streaming receiver whose channels have their own settings and end their streams one by one
(afsk_rx_streams_create_each / _finish_some): the resumable walk (test_stream_gate_model.GateWalk) with each
channel's amp_start / amp_end / timeout, and the retention policy (test_stream_retention_model.Arena) with
partial finishes.  Over random push / finish schedules, each channel's events over each of its successive
streams must be the oracle's listen_gate_multi over that stream with that stream's settings, and every pushed
frame must still cause O(1) moved frames."""
import numpy as np
import pytest

from oracle import oracle as O
from test_stream_gate_model import CHUNK, GateWalk, chunk_amps, random_stream
from test_stream_retention_model import Arena

THRESHOLDS = [(18000, 14000), (14000, 11000), (9000, 8000)]          # the c5 corpus's (amp_start, amp_end) pairs
TIMEOUTS = [0, int(0.1 * 48000), int(0.5 * 48000), 2 * 48000]


class EachHandle:
    """One handle as streams_run keeps it: per channel a walk with that channel's settings, the frames pushed
    to its current stream and the first one retained, and the arena's slots.  ``finish(streams, settings)``
    ends the listed channels' streams and resets them exactly like finish-all resets every channel.
    ``ended[s]`` lists channel s's ended streams as (settings, samples, events of all its pushes and finish)."""

    def __init__(self, settings):
        self.S = len(settings)
        self.settings = list(settings)
        self.walks = [GateWalk(*st) for st in settings]
        self.ar = Arena(self.S)
        self.pushed, self.keep = [0] * self.S, [0] * self.S
        self.cur = [np.zeros(0, np.int16) for _ in range(self.S)]     # the current stream of each channel
        self.events = [[] for _ in range(self.S)]                     # its events so far
        self.ended = [[] for _ in range(self.S)]
        self.total = 0

    def push(self, pieces):
        np_ = [p + len(x) for p, x in zip(self.pushed, pieces)]
        self.ar.push(self.pushed, np_, self.keep)
        out = []
        for s, x in enumerate(pieces):
            old = len(self.cur[s])
            self.cur[s] = np.concatenate([self.cur[s], x])
            out.append(self.walks[s].walk(chunk_amps(self.cur[s])[old // CHUNK:]))
            self.events[s] += out[-1]
            self.keep[s] = self.walks[s].retained_from()
            assert self.ar.base[s] <= self.keep[s] and np_[s] - self.ar.base[s] <= self.ar.cap[s]
        self.pushed = np_
        self.total += sum(len(x) for x in pieces)
        return out

    def finish(self, streams, settings=None):
        """the listed channels' final calls (stream -> list); the others walk no new chunk and emit nothing"""
        out = {}
        for s in range(self.S):
            if s not in streams:
                assert self.walks[s].walk(np.zeros(0, np.int64)) == []
        for i, s in enumerate(streams):
            out[s] = self.walks[s].walk(np.zeros(0, np.int64), finish=True)
            self.ended[s].append((self.settings[s], self.cur[s], self.events[s] + out[s]))
            if settings is not None:
                self.settings[s] = settings[i]
            self.walks[s] = GateWalk(*self.settings[s])
            self.pushed[s] = self.keep[s] = self.ar.base[s] = 0
            self.cur[s], self.events[s] = np.zeros(0, np.int16), []
        return out

    def state(self, s):
        w = self.walks[s]
        return self.pushed[s], (w.mark * CHUNK if w.phase == 2 else -1), self.pushed[s] - self.keep[s]


def random_settings(rng):
    a0, a1 = THRESHOLDS[int(rng.integers(0, len(THRESHOLDS)))]
    return a0, a1, TIMEOUTS[int(rng.integers(0, len(TIMEOUTS)))]


def random_ops(rng, S, steps, piece_max=30000):
    """A random schedule: ("push", S pieces' lengths; some channels get nothing for a while) or ("finish", channel
    ids, new settings per listed channel or None)."""
    ops = []
    for _ in range(steps):
        if rng.random() < 0.25:
            ids = [int(s) for s in rng.permutation(S)[:int(rng.integers(1, S + 1))]]
            ops.append(("finish", ids, [random_settings(rng) for _ in ids] if rng.random() < 0.6 else None))
        else:
            ops.append(("push", [0 if rng.random() < 0.2 else int(rng.integers(0, piece_max)) for _ in range(S)]))
    return ops


def run_ops(h, srcs, ops):
    """Drives the model; returns the model after a final finish of every channel."""
    pos = [0] * h.S
    for op in ops:
        if op[0] == "finish":
            h.finish(op[1], op[2])
            assert all(h.state(s) == (0, -1, 0) for s in op[1])
            continue
        pieces = []
        for s, n in enumerate(op[1]):
            pieces.append(srcs[s][pos[s]:pos[s] + n])
            pos[s] += len(pieces[-1])
        h.push(pieces)
    h.finish(list(range(h.S)))
    return h


@pytest.mark.parametrize("seed", range(6))
def test_each_channels_streams_equal_the_oracle(seed):
    rng = np.random.default_rng(seed)
    S = 6
    h = EachHandle([random_settings(rng) for _ in range(S)])
    srcs = [random_stream(rng, 800, 0) for _ in range(S)]
    run_ops(h, srcs, random_ops(rng, S, 60))
    n_streams = n_calls = 0
    for s in range(S):
        for (a0, a1, t), x, got in h.ended[s]:
            assert got == O.listen_gate_multi(x, a0, a1, t), (s, a0, a1, t, len(x))
            n_streams += 1
            n_calls += len(got)
    assert n_streams > 2 * S and n_calls > 50
    assert h.ar.moved <= 2 * h.total + 2 * CHUNK * S, (h.ar.moved, h.total)


def test_partial_finish_leaves_other_channels_alone():
    """Finishing channel 0 in the middle of a recording on channel 1 changes neither channel 1's walk nor its slot."""
    h = EachHandle([(18000, 14000, 48000), (18000, 14000, 48000)])
    loud = np.full(10 * CHUNK, 25000, np.int16)
    h.push([loud[:3 * CHUNK + 5], loud[:5 * CHUNK + 7]])
    walk1 = vars(h.walks[1]).copy()
    slot1 = (h.ar.off[1], h.ar.cap[1], h.ar.base[1])
    st1 = h.state(1)
    fin = h.finish([0], [(9000, 8000, 0)])
    assert fin == {0: [(True, CHUNK, 3 * CHUNK)]}
    assert vars(h.walks[1]) == walk1 and (h.ar.off[1], h.ar.cap[1], h.ar.base[1]) == slot1 and h.state(1) == st1
    assert h.state(0) == (0, -1, 0) and h.walks[0].lim == 0 and h.walks[0].amp_start == 9000
