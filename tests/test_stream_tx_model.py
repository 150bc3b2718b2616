"""CPU model of the streaming transmitter (afsk_tx.cu: afsk_tx_streams_send / _pull, k_tx_window): the scheduling of
messages on the shared timeline, the payload arena's retention policy, and k_tx_window's locate arithmetic restated
vector by vector (vector -> row -> overlapping message -> message frame -> pair frame -> bit and phase, var_locate for
unequal tones, then the five-pair walk) — checked against the reference's save() frames (oracle.tx_frames) placed on
each channel's timeline, over random send / pull schedules."""
import numpy as np
import pytest

from oracle import oracle as O

HI, LO = 32767, -32768
TAIL = 4800
ARENA_MIN = 65536


def hamming(v):
    d0, d1, d2, d3 = (v >> 3) & 1, (v >> 2) & 1, (v >> 1) & 1, v & 1
    return (d0 ^ d1 ^ d3) | ((d0 ^ d2 ^ d3) << 1) | (d0 << 2) | ((d1 ^ d2 ^ d3) << 3) | (d1 << 4) | (d2 << 5) | (d3 << 6)


def r16(x):
    return (x + 15) & ~15


class Msg:
    """A queued message: the TxDesc fields k_tx_window reads, its codeword start table, its arena block."""

    def __init__(self, pay: bytes, baud: int, ts_cycles: int):
        self.pay = pay
        self.bf = bf = 48000 // baud
        self.ml, self.sl = 4 * (bf // 4), bf
        self.ts_bits = 2 * ts_cycles
        G = 2 * len(pay)
        self.cws = [hamming(pay[g >> 1] >> 4 if g % 2 == 0 else pay[g >> 1] & 15) for g in range(G)]
        ones = np.array([bin(c).count("1") for c in self.cws], np.int64)
        self.ns = np.zeros(G + 1, np.int64)
        np.cumsum(ones * self.ml + (7 - ones) * self.sl, out=self.ns[1:])
        self.total_bits = self.ts_bits + 4 + 7 * G
        self.out_len = (ts_cycles * (self.ml + self.sl) + self.ml + 3 * self.sl + int(self.ns[G]) + TAIL) & ~1
        self.block = r16(len(pay)) + (r16(8 * (G + 1)) if self.ml != self.sl else 0)
        self.start = self.end = 0

    def tx_bit(self, b):
        if b < self.ts_bits:
            return (~b) & 1
        t = b - self.ts_bits
        if t < 4:
            return 1 if t == 0 else 0
        j = t - 4
        return (self.cws[j // 7] >> (j % 7)) & 1

    def bit(self, b):
        """win_bit: symbol (2 = the zero frames of the tail) and tone length"""
        sym = self.tx_bit(b) if b < self.total_bits else 2
        return sym, (1 << 31) - 1 if sym == 2 else (self.ml if sym else self.bf)

    def locate(self, p):
        """win_locate of even message frame p: (bit, phase)"""
        ml, sl = self.ml, self.sl
        if ml == sl:
            return divmod(p, sl)
        T0 = (self.ts_bits >> 1) * (ml + sl)                 # var_locate
        if p < T0:
            cyc, r = divmod(p, ml + sl)
            return (2 * cyc + 1, r - ml) if r >= ml else (2 * cyc, r)
        t = p - T0
        if t < ml:
            return self.ts_bits, t
        t -= ml
        if t < 3 * sl:
            return self.ts_bits + 1 + t // sl, t % sl
        t -= 3 * sl
        G = len(self.ns) - 1
        if G == 0 or t >= self.ns[G]:
            return self.total_bits, 0
        lo = int(np.searchsorted(self.ns, t, side="right")) - 1
        rem, cw, r = t - int(self.ns[lo]), self.cws[lo], 0
        while r < 6:
            L = ml if (cw >> r) & 1 else sl
            if rem < L:
                break
            rem -= L
            r += 1
        return self.ts_bits + 4 + 7 * lo + r, rem

    def tone(self, sym, ph):
        """tone_pair: the value of a frame at even phase ph"""
        if sym == 2:
            return 0
        q, h = self.bf >> 2, self.bf >> 1
        return HI if ((ph < q or 2 * q <= ph < 3 * q) if sym else ph < h) else LO


def win_find(descs, lo, hi, t):
    while lo < hi:
        mid = (lo + hi) >> 1
        if descs[mid].end <= t:
            lo = mid + 1
        else:
            hi = mid
    return lo


def win_frame(descs, row_off, row, t):
    hi = row_off[row + 1]
    k = win_find(descs, row_off[row], hi, t)
    if k >= hi or descs[k].start > t:
        return 0
    d = descs[k]
    b, u = d.locate((t - d.start) & ~1)
    return d.tone(d.bit(b)[0], u)


def k_tx_window(descs, row_off, P, n, S):
    """The kernel, one 16-byte vector (8 frames) at a time; frames it leaves alone keep the guard value."""
    total = S * n
    out = np.full(total, 0x1234, np.int64)
    for v in range((total + 7) // 8):
        f0 = 8 * v
        row, col = divmod(f0, n)
        t0 = P + col
        if col + 8 <= n:
            hi = row_off[row + 1]
            k = win_find(descs, row_off[row], hi, t0)
            if k >= hi or descs[k].start >= t0 + 8:
                out[f0:f0 + 8] = 0
                continue
            d = descs[k]
            if d.start <= t0 and d.end >= t0 + 8:
                m0 = t0 - d.start
                b, u = d.locate(m0 & ~1)
                sym, L = d.bit(b)
                pv = []
                for _ in range(5):
                    pv.append(d.tone(sym, u))
                    u += 2
                    while u >= L:
                        u -= L
                        b += 1
                        sym, L = d.bit(b)
                for e in range(8):
                    out[f0 + e] = pv[(e + (m0 & 1)) >> 1]
                continue
        for e in range(8):
            if f0 + e >= total:
                break
            out[f0 + e] = win_frame(descs, row_off, row, P + col)
            col += 1
            if col == n:
                col, row = 0, row + 1
    return out.reshape(S, n) if n else out.reshape(S, 0)


class TxModel:
    """afsk_tx_streams_* on the host: per-channel queues, the shared timeline, the payload arena's bookkeeping
    (capacity, top, live bytes, moved bytes, compactions) and, with synth=True, every pull's window."""

    def __init__(self, S, baud, training_time, synth=True):
        self.S, self.baud, self.ts = S, baud, O.ts_cycles(baud, training_time)
        self.synth = synth
        self.P = 0
        self.q = [[] for _ in range(S)]
        self.last_end = [0] * S
        self.cap, self.top, self.live = ARENA_MIN, 0, 0
        self.moved = self.compactions = 0
        self.sent_bytes = 0

    def send(self, streams, payloads):
        msgs = [Msg(p.encode() if isinstance(p, str) else bytes(p), self.baud, self.ts) for p in payloads]
        W = sum(m.block for m in msgs)
        if self.top + W > self.cap:                    # compaction into the other arena, doubled as needed
            while 2 * (self.live + W) > self.cap:
                self.cap *= 2
            self.moved += self.live
            self.compactions += 1
            self.top = self.live
        self.top += W
        self.live += W
        self.sent_bytes += W
        start, end = [], []
        for s, m in zip(streams, msgs):
            m.start = max(self.P, self.last_end[s])
            m.end = self.last_end[s] = m.start + m.out_len
            self.q[s].append(m)
            start.append(m.start)
            end.append(m.end)
        return np.array(start, np.int64), np.array(end, np.int64)

    def pull(self, n):
        out = None
        if self.synth and n > 0:
            descs, row_off = [], [0]
            for s in range(self.S):
                for m in self.q[s]:
                    if m.start >= self.P + n:
                        break
                    descs.append(m)
                row_off.append(len(descs))
            for s in range(self.S):                    # at most ceil(n / 4800) + 1 messages overlap a row's window
                assert row_off[s + 1] - row_off[s] <= -(-n // 4800) + 1
            out = k_tx_window(descs, row_off, self.P, n, self.S)
        if n > 0:
            self.P += n
            for qs in self.q:
                while qs and qs[0].end <= self.P:
                    self.live -= qs.pop(0).block
            if self.live == 0:
                self.top = 0
        return out

    def state(self, s):
        return self.P, self.last_end[s], len(self.q[s])


def timeline(sent, S, length, baud, training_time):
    """The oracle: each channel's frames, with save()'s frames of every message at [start, end)."""
    tl = np.zeros((S, length), np.int16)
    for s, pay, a, b in sent:
        fr = O.tx_frames(pay.encode() if isinstance(pay, str) else pay, baud, training_time)
        assert len(fr) == b - a
        if a < length:
            tl[s, a:min(b, length)] = fr[:max(0, min(b, length) - a)]
    return tl


class TimelineWindow:
    """timeline() one pull at a time, each message with its own baud and training time: add() the messages as they
    are sent, window(P, n) is frames [P, P + n) of every channel.  Each message's frames are made when a window
    first reaches them and dropped once a window has passed its end."""

    def __init__(self, S):
        self.S = S
        self.q = [[] for _ in range(S)]

    def add(self, s, pay, a, b, baud, training_time):
        self.q[s].append([a, b, pay.encode() if isinstance(pay, str) else bytes(pay), baud, training_time, None])

    def window(self, P, n):
        out = np.zeros((self.S, n), np.int16)
        for s, q in enumerate(self.q):
            while q and q[0][1] <= P:
                q.pop(0)
            for m in q:
                a, b = m[0], m[1]
                if a >= P + n:
                    break
                if m[5] is None:
                    m[5] = O.tx_frames(m[2], m[3], m[4])
                    assert len(m[5]) == b - a
                lo, hi = max(a, P), min(b, P + n)
                out[s, lo - P:hi - P] = m[5][lo - a:hi - a]
        return out


def random_payload(rng, hi=12):
    k = int(rng.integers(0, hi + 1))
    return rng.integers(0, 256, size=k, dtype=np.uint8).tobytes()


def schedule(rng, S, n_choice, steps, hi=12):
    """[('send', streams, payloads) | ('pull', n)]: pulls of n_choice (or random sizes), sends in between, several
    messages to one channel in one call, empty payloads, sends while the channel is busy or idle"""
    ops = []
    for _ in range(steps):
        if rng.random() < 0.45:
            k = int(rng.integers(1, 4))
            streams = [int(rng.integers(0, S)) for _ in range(k)]
            if rng.random() < 0.3:
                streams = [streams[0]] * k                 # back-to-back on one channel
            ops.append(("send", streams, [random_payload(rng, hi) for _ in range(k)]))
        else:
            n = int(rng.integers(0, 12000)) if n_choice is None else n_choice
            ops.append(("pull", n))
    return ops


def run_model(ops, S, baud, tt):
    m = TxModel(S, baud, tt)
    sent, got = [], []
    for op in ops:
        if op[0] == "idle_odd":                        # pull until every channel is idle and P is odd
            n = max(max(m.last_end) - m.P, 0)
            op = ("pull", n + 1 - (m.P + n) % 2)
        if op[0] == "send":
            a, b = m.send(op[1], op[2])
            sent += [(s, p, int(x), int(y)) for s, p, x, y in zip(op[1], op[2], a, b)]
        else:
            out = m.pull(op[1])
            got.append(out if out is not None else np.zeros((S, 0), np.int64))
    return m, sent, np.concatenate(got, axis=1) if got else np.zeros((S, 0))


BAUDS = [(1200, 0.02), (4800, 0.01), (24000, 0.0), (8000, 0.005), (12000, 0.0), (300, 0.0)]
CUTS = [0, 1, 3, 7, 8, 9, 2047, 2048, 48000, None]


@pytest.mark.parametrize("baud,tt", BAUDS)
@pytest.mark.parametrize("n", CUTS)
def test_window_model_equals_oracle_timeline(baud, tt, n):
    rng = np.random.default_rng([baud, 99999 if n is None else n])
    S = 3
    if n in (0, 1, 3, 7, 8, 9):
        # small pulls over the start of the timeline (odd P at send included), then larger ones over the rest
        ops = [("send", [0, 1], [random_payload(rng), b""])]
        for i in range(240 if n else 4):
            ops.append(("pull", n))
            if i == 4:
                ops.append(("send", [2], [random_payload(rng)]))         # idle channel, P = 5 * n
            elif i % 37 == 5:
                ops.append(("send", [int(rng.integers(0, S))], [random_payload(rng)]))
        ops += schedule(rng, S, None, 14)
    else:
        ops = schedule(rng, S, n, 24 if n != 48000 else 10)
    ops += [("idle_odd",), ("send", [0, 1, 1], [random_payload(rng), b"", random_payload(rng)])]
    ops += [("pull", n if n else 9000)] * (1 if n is None or n >= 2047 else 3) + [("pull", 20000)]
    m, sent, got = run_model(ops, S, baud, tt)
    want = timeline(sent, S, got.shape[1], baud, tt)
    assert np.array_equal(got, want)
    assert any(a % 2 for _, _, a, _ in sent)                               # a message started on an odd frame


@pytest.mark.parametrize("baud", [4800, 1200])
def test_back_to_back_and_busy_channel_scheduling(baud):
    m = TxModel(2, baud, 0.01, synth=False)
    pays = [b"", b"\x00", b"\xff" * 3, "héllo"]
    a, b = m.send([0, 0, 0, 1], pays)
    lens = [len(O.tx_frames(p.encode() if isinstance(p, str) else p, baud, 0.01)) for p in pays]
    assert list(a) == [0, lens[0], lens[0] + lens[1], 0]
    assert list(b - a) == lens and all(x % 2 == 0 for x in lens)
    m.pull(7)
    a2, _ = m.send([0, 1], [b"x", b"y"])
    assert a2[0] == b[2] and a2[1] == b[3]                 # busy channels: behind their last message
    _, e2 = m.send([1], [b"w"])
    m.pull(int(e2[0]) - m.P + 1)
    assert m.state(1) == (int(e2[0]) + 1, int(e2[0]), 0)
    a3, e3 = m.send([1], [b"z"])
    assert a3[0] == m.P and m.P % 2 == 1                   # idle channel: at P (odd here)
    assert m.state(1) == (m.P, int(e3[0]), 1)


def test_retention_moves_stay_proportional_to_sent_bytes():
    """Many small messages on 64 channels over a long run: every compaction follows at least half an arena of
    sent bytes, so the bytes moved stay below twice the bytes sent, and the arena stays within a small
    multiple of the most bytes ever live."""
    for baud in (1200, 4800):
        rng = np.random.default_rng(baud)
        S = 64
        m = TxModel(S, baud, 0.05, synth=False)
        peak = 0
        for step in range(3000):
            k = int(rng.integers(0, 40))
            m.send([int(x) for x in rng.integers(0, S, k)], [random_payload(rng, 200) for _ in range(k)])
            peak = max(peak, m.live)
            m.pull(int(rng.integers(1, 30000)))
        assert m.compactions >= 5
        assert m.moved <= 2 * m.sent_bytes, (m.moved, m.sent_bytes)
        assert m.cap <= max(4 * peak, ARENA_MIN), (m.cap, peak)


def test_long_idle_stretches_reset_the_top():
    m = TxModel(4, 1200, 0.1, synth=False)
    for _ in range(200):
        m.send([0, 1], [b"a" * 100, b"b" * 50])
        m.pull(200000)                                      # both messages end inside the pull
        assert m.live == 0 and m.top == 0
    assert m.compactions == 0 and m.moved == 0
