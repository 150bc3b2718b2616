"""CPU model of the streaming receiver's bits-mode bookkeeping (streams_bits in afsk_rx.cu): when a pending
recording's clock is recovered, which bit windows each push decides, which samples a channel keeps, and the
plane slots, which follow the sample arena's policy (Arena, a plane word counting as four frames).  Checked over
random cuts of streams: every window of every recording is decided exactly once, in word-aligned ranges; the
retained frames stay below max(4096, 33 bit lengths); and a recording open for an hour beside idle channels costs
O(1) moved frames per pushed frame and O(1) moved plane words per decided window."""
import numpy as np
import pytest

from test_stream_gate_model import CHUNK, GateWalk
from test_stream_retention_model import Arena

SYNC = 4096                                  # frames the clock recovery reads
MAX_BF = 2000                                # afsk_rx.cu kWinMaxBf


def bit_frames(baud):
    """the bit length bits mode demodulates at this baud, or 0 where the result follows from length and baud
    (k_preset's statuses: 4800, 960, 1600, 8000, 24000 baud and bauds <= 23)"""
    if baud <= 23 or baud in (4800, 960, 1600, 8000, 24000):
        return 0
    bf = 48000 // baud
    return bf if bf % 4 == 0 and bf <= MAX_BF else -1


def windows_of(n, bf, clk):
    """K = #{k : clk + k bf < n - bf}"""
    span = n - bf - clk
    return 0 if span <= 0 else -(-span // bf)


class BitsPlan:
    """One handle in bits mode: per channel the resumable walk, the frames pushed and kept, the pending recording
    (start, stored clock, windows decided, plane stream position of its window 0), the plane stream's end and
    first kept position (four per word), and the sample and plane arenas.  clock(s, R) gives the clock of channel
    s's recording starting at stream frame R (from its first 4096 frames).  jobs: per push, the window ranges
    decided, as (channel, (stream, recording start), first window, end window)."""

    def __init__(self, settings, bauds, clock):
        self.S = len(settings)
        self.settings, self.bauds, self.clock = list(settings), list(bauds), clock
        self.walks = [GateWalk(*x) for x in self.settings]
        self.ar, self.pl = Arena(self.S), Arena(self.S)
        S = self.S
        self.pushed, self.keep, self.R = [0] * S, [0] * S, [-1] * S
        self.clk, self.dec, self.pw_rec, self.pw_pushed, self.pw_keep = [-1] * S, [0] * S, [0] * S, [0] * S, [0] * S
        self.jobs = []
        self.epoch = [0] * S                     # streams finished per channel (keys recordings with their start)
        self.windows_total = 0

    def _step(self, lens, amps, fin=None):
        S = self.S
        np_ = [p + n for p, n in zip(self.pushed, lens)]
        self.ar.push(self.pushed, np_, self.keep)
        out, jobs = [], []
        new = []
        for s in range(S):
            bf = bit_frames(self.bauds[s])
            w = self.walks[s]
            finish = fin is not None and s in fin
            ev = w.walk(amps[s][self.pushed[s] // CHUNK:np_[s] // CHUNK] if not finish else np.zeros(0, np.int64), finish=finish)
            out.append(ev)
            e = self.pw_pushed[s]
            final = None
            if ev and ev[0][0] and ev[0][1] == self.R[s] and self.clk[s] >= 0:
                K = windows_of(ev[0][2] - ev[0][1], bf, self.clk[s])
                final = (self.R[s], self.clk[s], self.dec[s], K)
                e = max(e, self.pw_rec[s] + 4 * (-(-K // 32)))
            R = w.mark * CHUNK if w.phase == 2 else -1
            same = R >= 0 and R == self.R[s]
            stored = same and self.clk[s] >= 0
            clk = self.clk[s] if same else -1
            if R >= 0 and clk < 0 and bf > 0 and np_[s] - R >= SYNC:
                clk = self.clock(s, R)
            dec, pw0 = 0, 0
            if R >= 0 and clk >= 0:
                span = np_[s] - R - clk
                dec = (span // bf) // 32 * 32 if span > 0 else 0
                pw0 = self.pw_rec[s] if stored else e
                e = max(e, pw0 + 4 * (dec // 32))
            new.append((R, clk, dec, pw0, e, stored, final, bf))
        self.pl.push(self.pw_pushed, [x[4] for x in new], self.pw_keep)
        for s in range(S):
            R, clk, dec, pw0, e, stored, final, bf = new[s]
            if final is not None and final[3] > final[2]:
                jobs.append((s, (self.epoch[s], final[0]), final[2], final[3]))
            d0 = self.dec[s] if stored else 0
            if R >= 0 and clk >= 0 and dec > d0:
                jobs.append((s, (self.epoch[s], R), d0, dec))
            w = self.walks[s]
            on = R >= 0 and clk >= 0
            self.keep[s] = w.pos * CHUNK if R < 0 or bf == 0 else (min(w.pos * CHUNK, R + clk + dec * bf) if on else R)
            self.R[s], self.clk[s] = R, (clk if on else -1)
            self.dec[s], self.pw_rec[s] = (dec if on else 0), (pw0 if on else 0)
            self.pw_pushed[s], self.pw_keep[s] = e, (pw0 if on else e)
            assert self.ar.base[s] <= self.keep[s] and np_[s] - self.ar.base[s] <= self.ar.cap[s]
            assert self.pl.base[s] <= self.pw_keep[s] and e - self.pl.base[s] <= self.pl.cap[s]
        self.pushed = np_
        self.jobs.append(jobs)
        self.windows_total += sum(b - a for _, _, a, b in jobs)
        return out

    def push(self, lens, amps):
        """lens[s] new frames of channel s, whose current stream's chunk amplitudes are amps[s]; -> events per channel"""
        return self._step(lens, amps)

    def finish(self, ids, settings=None, bauds=None):
        out = self._step([0] * self.S, [np.zeros(0, np.int64)] * self.S, fin=set(ids))
        for i, s in enumerate(ids):
            if settings is not None:
                self.settings[s], self.bauds[s] = settings[i], bauds[i]
            self.walks[s] = GateWalk(*self.settings[s])
            self.epoch[s] += 1
            self.pushed[s] = self.keep[s] = self.ar.base[s] = 0
            self.R[s], self.clk[s] = -1, -1
            self.dec[s] = self.pw_rec[s] = self.pw_pushed[s] = self.pw_keep[s] = self.pl.base[s] = 0
        return {s: out[s] for s in ids}

    def state(self, s):
        """afsk_rx_streams_state and _pending_bits of channel s"""
        return (self.pushed[s], self.R[s], self.pushed[s] - self.keep[s]), (self.clk[s] if self.R[s] >= 0 else -1, self.dec[s])


# ---------------------------------------------------------------- CPU checks ----------------------------------------

PIECES = [0, 1, 7, 2047, 2048, 2049, 48000]


def random_amps(rng, n_chunks):
    """chunk amplitudes: idle stretches, recordings of 2 .. 400 chunks, some never closed"""
    a = np.zeros(n_chunks, np.int64)
    i = 0
    while i < n_chunks:
        i += int(rng.integers(0, 30))
        ln = int(rng.integers(1, 400))
        a[i:i + ln] = 25000
        i += ln
    return a


def check_windows(plan, recs):
    """every window [0, K) of every bits-decoded recording decided exactly once, in word-aligned ranges that never
    overlap; recs: (channel, start, K)"""
    seen = {}
    for jobs in plan.jobs:
        for s, R, a, b in jobs:
            assert a % 32 == 0 and b > a
            seen.setdefault((s, R), []).append((a, b))
    for s, R, K in recs:
        rs = sorted(seen.get((s, R), []))
        pos = 0
        for a, b in rs:
            assert a == pos, (s, R, rs)                  # no gap, no overlap
            pos = b
        # windows past K are ones decided before finish cut the recording short; all of [0, K) is covered
        assert pos >= K, (s, R, K, rs)
        for a, b in rs[:-1]:
            assert b < K or b % 32 == 0


@pytest.mark.parametrize("seed", range(4))
def test_every_window_decided_once_and_retention_bounded(seed):
    rng = np.random.default_rng(seed)
    bauds = [300, 1200, 6000, 24, 12000, 4800, 2400, 100]
    S = len(bauds)
    settings = [(18000, 14000, int(rng.choice([0, 48000, 96000]))) for _ in range(S)]
    n_chunks = 300
    amps = [random_amps(rng, n_chunks) for _ in range(S)]
    clocks = {}

    def clock(s, R):
        bf = bit_frames(bauds[s])
        return clocks.setdefault((s, R), int(rng.integers(0, SYNC - 2 * bf)))

    plan = BitsPlan(settings, bauds, clock)
    recs = []
    total = n_chunks * CHUNK
    while min(plan.pushed) < total:
        lens = [min(int(rng.choice(PIECES)), total - p) for p in plan.pushed]
        before = (list(plan.R), list(plan.clk))
        ev = plan.push(lens, amps)
        for s in range(S):
            for k, e in enumerate(ev[s]):
                if e[0] and k == 0 and e[1] == before[0][s] and before[1][s] >= 0:
                    recs.append((s, (plan.epoch[s], e[1]), windows_of(e[2] - e[1], bit_frames(bauds[s]), before[1][s])))
            bf = bit_frames(bauds[s])
            ret = plan.pushed[s] - plan.keep[s]
            assert ret < max(SYNC, 33 * max(bf, 1)), (s, ret)
        if rng.random() < 0.05:
            ids = [int(s) for s in rng.choice(S, int(rng.integers(1, S + 1)), replace=False)]
            before = (list(plan.R), list(plan.clk), list(plan.epoch))
            out = plan.finish(ids)
            for s, evs in out.items():
                for k, e in enumerate(evs):
                    if e[0] and k == 0 and e[1] == before[0][s] and before[1][s] >= 0:
                        recs.append((s, (before[2][s], e[1]), windows_of(e[2] - e[1], bit_frames(bauds[s]), before[1][s])))
                amps[s] = random_amps(rng, n_chunks)
    assert len(recs) > 5
    check_windows(plan, recs)


@pytest.mark.parametrize("baud,piece", [(1200, 48000), (300, 48000), (24, 48000), (6000, 2048), (1200, 2047)])
def test_hour_long_recording_moves_are_bounded(baud, piece):
    """one channel stuck open for an hour beside idle channels"""
    S = 4
    pushes = 3600 * 48000 // piece
    bauds = [baud] * S
    plan = BitsPlan([(18000, 14000, 48000)] * S, bauds, lambda s, R: 100)
    amps = [np.full(pushes * piece // CHUNK + 1, 25000, np.int64)] + [np.zeros(pushes * piece // CHUNK + 1, np.int64)] * (S - 1)
    bf = bit_frames(baud)
    for _ in range(pushes):
        plan.push([piece] * S, amps)
        assert plan.pushed[0] - plan.keep[0] < max(SYNC, 33 * bf)
    assert plan.walks[0].phase == 2
    total = piece * pushes * S
    assert plan.ar.moved <= total // 4, (plan.ar.moved, total)         # O(1) per pushed frame
    windows = plan.dec[0]
    assert windows > 0 and plan.pl.moved // 4 <= 2 * (windows // 32) + 64, (plan.pl.moved, windows)
    assert plan.pl.compactions <= 24
