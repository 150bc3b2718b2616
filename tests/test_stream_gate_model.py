"""CPU model of the streaming receiver's resumable gate walk (k_gate_multi with a saved GateState,
afsk_rx.cu) checked against the oracle's successive receive() calls over the whole stream.

The model keeps the kernel's state fields (pos, mark, call, phase) and transitions.  For every stream
and every way of cutting it into pushes, the calls emitted by all pushes plus finish must be
``oracle.listen_gate_multi`` over the whole stream, and after every push the calls emitted so far must
be exactly the oracle's calls that are final within the prefix pushed so far."""
import numpy as np
import pytest

from oracle import oracle as O

CHUNK = 2048


class GateWalk:
    """One channel: GateState plus the kernel's walk over the amplitudes of the chunks that arrived."""

    def __init__(self, amp_start: int, amp_end: int, timeout_frames: int):
        self.amp_start, self.amp_end = amp_start, amp_end
        self.lim = 0 if timeout_frames <= 0 else -(-timeout_frames // CHUNK)
        self.pos = self.mark = self.call = self.phase = 0

    @staticmethod
    def _find_first(A, c0, lo, hi, hit):
        """first chunk j in [lo, hi) with hit(A[j - c0]), or -1"""
        if hi <= lo:
            return -1
        idx = np.flatnonzero(hit(A[lo - c0:hi - c0]))
        return lo + int(idx[0]) if len(idx) else -1

    def walk(self, amp_new: np.ndarray, finish: bool = False):
        c0 = self.pos
        nch = c0 + len(amp_new)
        A = amp_new                                                    # A[j - c0]: chunk j
        out = []
        while True:
            if self.phase == 0:
                if self.pos >= nch:
                    break
                self.pos += 1                                          # discard
                self.phase, self.mark = 1, self.pos
            rec = (False, 0, 0)
            if self.phase == 1:
                stop = self.mark + self.lim
                o = self._find_first(A, c0, self.pos, min(stop, nch), lambda a: a > self.amp_start)
                if o < 0:
                    if stop > nch:
                        self.pos = nch
                        break
                    self.pos = stop                                    # timed out
                else:
                    self.phase, self.mark, self.pos = 2, o, o + 1
            if self.phase == 2:
                c = self._find_first(A, c0, self.pos, nch, lambda a: a < self.amp_end)
                if c < 0:
                    self.pos = nch
                    break
                rec = (True, self.mark * CHUNK, (c + 1) * CHUNK)
                self.pos = c + 1
            out.append(rec)
            self.phase = 0
        if finish and self.phase == 2:
            out.append((True, self.mark * CHUNK, nch * CHUNK))
            self.phase = 0
        self.call += len(out)
        assert self.pos == nch
        return out

    def retained_from(self) -> int:
        """First frame the device keeps: the pending recording's first chunk, else the partial chunk."""
        return (self.mark if self.phase == 2 else self.pos) * CHUNK


def chunk_amps(x: np.ndarray) -> np.ndarray:
    n = len(x) // CHUNK
    return np.abs(x[:n * CHUNK].astype(np.int64)).reshape(n, CHUNK).sum(axis=1) // CHUNK


def run_schedule(x, cuts, amp_start, amp_end, timeout):
    """Pushes x cut at `cuts`; returns the events of every push and of finish."""
    w = GateWalk(amp_start, amp_end, timeout)
    per_push, pushed = [], 0
    for c in list(cuts) + [len(x)]:
        new_chunks = c // CHUNK - pushed // CHUNK
        amps = chunk_amps(x[:c])[pushed // CHUNK:pushed // CHUNK + new_chunks]
        per_push.append((c, w.walk(amps)))
        assert c - w.retained_from() >= 0
        pushed = c
    return per_push, w.walk(np.zeros(0, np.int64), finish=True), w


def final_prefix(calls, amps_full, nch_prefix, lim, amp_end):
    """How many of the whole stream's calls are final within the first nch_prefix chunks."""
    p, n = 0, 0
    for rec, a, b in calls:
        if not rec:
            end, ok = p + 1 + lim, p + 1 + lim <= nch_prefix
        else:
            end = b // CHUNK
            ok = end <= nch_prefix and amps_full[end - 1] < amp_end and end - 1 > a // CHUNK
        if not ok:
            break
        n += 1
        p = end
    return n


def random_stream(rng, n_chunks, partial):
    levels = np.array([0, 3000, 9000, 16000, 21000, 30000])
    lv = []
    state = 0
    for _ in range(n_chunks):
        if rng.random() < 0.3:
            state = int(rng.integers(0, len(levels)))
        lv.append(levels[state])
    x = np.repeat(np.array(lv, dtype=np.int64), CHUNK)
    x = x * rng.choice([-1, 1], size=len(x))
    x = x + rng.integers(-200, 201, size=len(x))
    x = np.concatenate([x, rng.integers(-30000, 30000, size=partial)])
    return np.clip(x, -32768, 32767).astype(np.int16)


def random_cuts(rng, n):
    cuts, c = [], 0
    while True:
        kind = rng.integers(0, 6)
        if kind == 0:
            step = 0
        elif kind == 1:
            step = 1
        elif kind == 2:                                            # end at 2048k - 1, 2048k or 2048k + 1
            k = c // CHUNK + int(rng.integers(1, 4))
            step = k * CHUNK + int(rng.integers(-1, 2)) - c
        else:
            step = int(rng.integers(0, 20000))
        c = c + max(step, 0)
        if c >= n:
            return cuts
        cuts.append(c)


@pytest.mark.parametrize("timeout", [0, 1, 2048, 3 * 2048, 3 * 2048 + 1, 10 ** 9])
def test_resumable_walk_equals_oracle_on_random_schedules(timeout):
    rng = np.random.default_rng(1000 + timeout % 9973)
    amp_start, amp_end = 18000, 14000
    lim = 0 if timeout <= 0 else -(-timeout // CHUNK)
    checked_final = 0
    for trial in range(25):
        x = random_stream(rng, int(rng.integers(0, 60)), int(rng.integers(0, CHUNK)))
        want = O.listen_gate_multi(x, amp_start, amp_end, timeout)
        amps_full = chunk_amps(x)
        for cuts in (random_cuts(rng, len(x)), [], list(range(CHUNK, len(x), CHUNK)), list(range(CHUNK - 1, len(x), CHUNK - 1))):
            per_push, fin, w = run_schedule(x, cuts, amp_start, amp_end, timeout)
            got = []
            for c, evs in per_push:
                got += evs
                n_final = final_prefix(want, amps_full, c // CHUNK, lim, amp_end)
                assert got == want[:n_final], (trial, c)
                checked_final += n_final
            assert got + fin == want, trial
            assert w.call == len(want)
    assert checked_final > 0


def test_pushes_of_one_frame_and_zero_frames():
    rng = np.random.default_rng(7)
    x = random_stream(rng, 12, 100)
    cuts = sorted(set(range(0, len(x), 1)) | {0})
    cuts = [c for c in cuts for _ in (0, 1)]                      # every push of one frame followed by an empty one
    per_push, fin, _ = run_schedule(x, cuts, 18000, 14000, 4096)
    assert [e for _, ev in per_push for e in ev] + fin == O.listen_gate_multi(x, 18000, 14000, 4096)


def test_positions_beyond_32_bits():
    """Chunk counters and frame positions are 64-bit: a walk resumed far into a stream."""
    w = GateWalk(18000, 14000, 3 * CHUNK)
    w.pos = (1 << 33) + 5                                          # 2^33 chunks: about eleven years at 48 kHz
    ev = w.walk(np.array([0, 20000, 20000, 100, 0, 0, 0, 0], np.int64))
    assert ev == [(True, ((1 << 33) + 6) * CHUNK, ((1 << 33) + 9) * CHUNK), (False, 0, 0)]
    assert ev[0][2] > 1 << 44
