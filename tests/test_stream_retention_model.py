"""CPU model of the streaming receiver's retention policy (streams_run in afsk_rx.cu): which retained samples
move, and where, when a piece does not fit behind its channel's slot.  Replayed over long runs with the
resumable walk's retention points (test_stream_gate_model.GateWalk), it checks that every pushed frame
causes O(1) moved frames, also for a recording that stays open beside idle channels for an hour."""
import numpy as np
import pytest

from test_stream_gate_model import CHUNK, GateWalk

PAD = 64


class Arena:
    """Slot bookkeeping of one handle, as in streams_run: per channel slot_off / slot_cap / slot_base,
    the top of the current arena, its capacity in frames, and the frames moved."""

    def __init__(self, S):
        self.off, self.cap, self.base = [0] * S, [0] * S, [0] * S
        self.top, self.frames, self.alloc = 0, [0, 0], [0, 0]
        self.cur, self.moved, self.compactions = 0, 0, 0

    @staticmethod
    def fresh_cap(need):
        return (2 * need + 2 * CHUNK + 7) & ~7

    def grow(self, i, need_frames):
        """grow_device (capacity in bytes: need + need / 4 + 4096), in frames after the pad"""
        need = (need_frames + PAD) * 2
        if need > self.alloc[i]:
            self.alloc[i] = need + need // 4 + 4096
        self.frames[i] = self.alloc[i] // 2 - PAD

    def push(self, pushed, np_, keep):
        S = len(pushed)
        over = [np_[s] - self.base[s] > self.cap[s] for s in range(S)]
        rewind = [2 * (np_[s] - keep[s]) <= self.cap[s] for s in range(S)]
        want = sum(self.fresh_cap(np_[s] - keep[s]) for s in range(S) if over[s] and not rewind[s])
        if any(over) and self.top + want > (self.frames[self.cur] if self.alloc[self.cur] else 0):
            caps = [self.fresh_cap(np_[s] - keep[s]) for s in range(S)]
            total = sum(caps)
            self.grow(self.cur ^ 1, total + total // 2)
            o = 0
            for s in range(S):
                self.moved += pushed[s] - keep[s]
                self.off[s], self.cap[s], self.base[s] = o, caps[s], keep[s]
                o += caps[s]
            self.top, self.cur = total, self.cur ^ 1
            self.compactions += 1
            return
        for s in range(S):
            if not over[s]:
                continue
            if not rewind[s]:
                self.off[s], self.cap[s] = self.top, self.fresh_cap(np_[s] - keep[s])
                self.top += self.cap[s]
            else:                                      # the span lies above the slot start it moves to
                assert keep[s] - self.base[s] >= pushed[s] - keep[s]
            self.moved += pushed[s] - keep[s]
            self.base[s] = keep[s]


def replay(levels, piece, pushes):
    """levels[s]: constant chunk amplitude of channel s.  Returns (arena, pushed frames, walks)."""
    S = len(levels)
    walks = [GateWalk(18000, 14000, 48000) for _ in range(S)]
    ar = Arena(S)
    pushed, keep = [0] * S, [0] * S
    for _ in range(pushes):
        np_ = [p + piece for p in pushed]
        ar.push(pushed, np_, keep)
        for s in range(S):
            walks[s].walk(np.full(np_[s] // CHUNK - pushed[s] // CHUNK, levels[s], np.int64))
            keep[s] = walks[s].retained_from()
            assert ar.base[s] <= keep[s] and np_[s] - ar.base[s] <= ar.cap[s]     # the piece fit behind its slot
            assert ar.off[s] + ar.cap[s] <= ar.top <= ar.frames[ar.cur]
        pushed = np_
    return ar, sum(pushed), walks


@pytest.mark.parametrize("piece,pushes,idle", [(48000, 3600, 1), (48000, 3600, 7), (2048, 8000, 3), (2047, 4000, 3),
                                               (100, 20000, 2)])
def test_moves_per_pushed_frame_are_bounded(piece, pushes, idle):
    """One channel stuck open (its recording grows for the whole run) beside idle channels."""
    ar, total, walks = replay([25000] + [0] * idle, piece, pushes)
    assert walks[0].phase == 2                                     # still recording
    # everything moved, the open recording's doublings and compactions included, is less than what was
    # pushed, and less than three times the open recording (1.1-2.2 times here)
    assert ar.moved <= total, (ar.moved, total)
    assert ar.moved <= 3 * piece * pushes, (ar.moved, piece * pushes)
    assert ar.compactions <= 16


def test_idle_channels_only():
    ar, total, _ = replay([0] * 16, 48000, 2000)
    assert ar.moved <= total // 10                                 # partial chunks only
    assert ar.compactions <= 8
