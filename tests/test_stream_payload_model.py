"""CPU model of the streaming receiver's payload-mode bookkeeping (streams_bits and k_stream_frame in afsk_rx.cu):
bits mode (test_stream_bits_model.BitsPlan) plus a framing state per pending recording with a stored clock, advanced
every push over the windows of the chunks the gate has walked (K_safe) as far as they are decided; the plane words a
channel keeps from then on; and the payload slots, which follow the sample arena's policy (Arena, two bytes counting
as one frame).  Checked over random decision / quiet sequences and random cuts into pushes, with finishes: the
incremental result equals whole-recording framing (afskmodem.py:362-399, as afsk_oracle_rx_decode does it), the
bytes decoded after every push are a prefix of the final payload, the framing reads only plane words it keeps, and
a one-tone carrier held for an hour keeps O(1) planes."""
import numpy as np
import pytest

from oracle import oracle as O
from test_stream_bits_model import SYNC, BitsPlan, bit_frames, windows_of
from test_stream_gate_model import CHUNK, GateWalk
from test_stream_retention_model import Arena

TRAIN, PAYLOAD, ENDED = 0, 1, 2


class Framing:
    """k_stream_frame's FrameState of one recording"""

    def __init__(self):
        self.phase, self.consumed, self.k0, self.k1, self.nbytes = TRAIN, 0, 0, 0, 0
        self.data = b""                          # the decoded bytes (ArrayFramer only)

    def advance(self, fr, kend, kept_word):
        """frame windows [consumed, kend) with framer fr; kept_word: the first plane word the channel still holds"""
        c = self.consumed
        if self.phase == TRAIN and c < kend:
            t = fr.find_term(c, kend, kept_word)
            if t is None:
                c = kend
            else:
                self.phase, self.k0 = PAYLOAD, t + 1
                c = self.k0
        if self.phase == PAYLOAD:
            q = fr.find_quiet(c, kend, kept_word) if c < kend else None
            if q is not None:
                self.phase, self.k1 = ENDED, q
            c = max(c, kend)
            nb = ((q if q is not None else c) - self.k0) // 14
            if nb > self.nbytes:
                self.data += fr.decode(self.k0, self.nbytes, nb, kept_word)
                self.nbytes = nb
        self.consumed = max(self.consumed, c)

    def result(self, clk, bf, K):
        """the AfskRxResult of the recording that ended with K windows: (status, clock, train_end, nbits, nbytes)"""
        k0 = self.k0 if self.phase >= PAYLOAD else K
        k1 = self.k1 if self.phase == ENDED else K
        nbits = k1 - k0
        return (O.ST_OK if nbits > 0 else O.ST_NO_DATA, clk, clk + k0 * bf, nbits, self.nbytes if nbits > 0 else 0)

    def pending(self, clk, bf):
        """afsk_rx_streams_pending_payload without the bytes: (train_end, nbits, ended, nbytes)"""
        if self.phase == TRAIN:
            return -1, 0, False, self.nbytes
        return clk + self.k0 * bf, (self.k1 if self.phase == ENDED else self.consumed) - self.k0, self.phase == ENDED, self.nbytes


class ArrayFramer:
    """a recording's decision bits and quiet flags as arrays; reads only plane words >= kept_word"""

    def __init__(self, bits, quiet):
        self.bits, self.quiet = np.asarray(bits, np.uint8), np.asarray(quiet, np.uint8)
        self.x = np.concatenate([np.zeros(3, np.uint8), self.bits])    # x[k .. k + 3] = b[k-3 .. k] (0 before window 0)

    def find_term(self, lo, hi, kept_word):
        assert max(lo - 3, 0) // 32 >= kept_word, (lo, kept_word)
        x = self.x
        m = (x[lo:hi] == 1) & (x[lo + 1:hi + 1] == 0) & (x[lo + 2:hi + 2] == 0) & (x[lo + 3:hi + 3] == 0)
        idx = np.flatnonzero(m)
        return lo + int(idx[0]) if len(idx) else None

    def find_quiet(self, lo, hi, kept_word):
        assert lo // 32 >= kept_word
        idx = np.flatnonzero(self.quiet[lo:hi])
        return lo + int(idx[0]) if len(idx) else None

    def decode(self, k0, i0, i1, kept_word):
        assert (k0 + 14 * i0) // 32 >= kept_word
        return decode_bytes(self.bits[k0 + 14 * i0:k0 + 14 * i1])


class MarkFramer:
    """a recording known only by its terminator window t and its first quiet window q >= t + 1 (None: not within the
    stream), e.g. from the oracle's decode of the whole recording; decodes no bytes"""

    def __init__(self, t, q):
        self.t, self.q = t, q

    def find_term(self, lo, hi, kept_word):
        return self.t if self.t is not None and lo <= self.t < hi else None

    def find_quiet(self, lo, hi, kept_word):
        return self.q if self.q is not None and lo <= self.q < hi else None

    def decode(self, k0, i0, i1, kept_word):
        return bytes(i1 - i0)


def decode_bytes(bits):
    """whole 14-bit groups -> bytes: Hamming(7,4) per nibble, first nibble high (:393-399)"""
    n = len(bits) // 14
    return np.packbits(O.ecc_decode(np.asarray(bits[:14 * n], np.uint8))).tobytes()[:n]


def frame_whole(bits, quiet, K, clk, bf):
    """afskmodem.py:362-399 over the first K windows of a recording -> (result, payload)"""
    sr, k0 = 0, K
    for k in range(K):
        sr = ((sr << 1) | int(bits[k])) & 0xF                       # __decodeBits :362-366
        if sr == 0b1000:
            k0 = k + 1
            break
    k1 = K
    for k in range(k0, K):                                          # :372-378
        if quiet[k]:
            k1 = k
            break
    nbits = k1 - k0
    data = decode_bytes(bits[k0:k1]) if nbits > 0 else b""
    return (O.ST_OK if nbits > 0 else O.ST_NO_DATA, clk, clk + k0 * bf, nbits, len(data)), data


def room(f, k):
    """payload slot samples reserved for a recording framed up to window k"""
    b = f.nbytes if f.phase == ENDED else ((f.consumed - f.k0 if f.phase == PAYLOAD else 0) + max(k - f.consumed, 0)) // 14 + 1
    return (b + 1) // 2


class PayloadPlan(BitsPlan):
    """One handle in payload mode.  framer(s, R, clk) gives the framer of channel s's recording starting at stream
    frame R.  results: {(epoch, R): (result, bytes)} of the recordings framed by k_stream_frame's final jobs;
    frame_jobs: per push, (channel, (epoch, R), consumed before, window end, final)."""

    def __init__(self, settings, bauds, clock, framer):
        super().__init__(settings, bauds, clock)
        S = self.S
        self.framer = framer
        self.py = Arena(S)
        self.fs = [Framing() for _ in range(S)]
        self.fr = [None] * S
        self.py_rec, self.py_pushed, self.py_keep = [0] * S, [0] * S, [0] * S
        self.results, self.frame_jobs = {}, []

    def _step(self, lens, amps, fin=None):
        S = self.S
        np_ = [p + n for p, n in zip(self.pushed, lens)]
        self.ar.push(self.pushed, np_, self.keep)
        out, jobs, fjobs, new = [], [], [], []
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
                fin_ended = self.fs[s].phase == ENDED
                final = (self.R[s], self.clk[s], self.dec[s], K, fin_ended)
                if not fin_ended:
                    e = max(e, self.pw_rec[s] + 4 * (-(-K // 32)))
            R = w.mark * CHUNK if w.phase == 2 else -1
            same = R >= 0 and R == self.R[s]
            stored = same and self.clk[s] >= 0
            ended = stored and self.fs[s].phase == ENDED
            clk = self.clk[s] if same else -1
            if R >= 0 and clk < 0 and bf > 0 and np_[s] - R >= SYNC:
                clk = self.clock(s, R)
            dec, pw0 = 0, 0
            if R >= 0 and clk >= 0:
                span = np_[s] - R - clk
                dec = self.dec[s] if ended else ((span // bf) // 32 * 32 if span > 0 else 0)
                pw0 = self.pw_rec[s] if stored else e
                e = max(e, pw0 + 4 * (dec // 32))
            new.append([R, clk, dec, pw0, e, stored, final, bf, ended])
        self.pl.push(self.pw_pushed, [x[4] for x in new], self.pw_keep)
        kend, py0, ynp = [0] * S, [0] * S, [0] * S
        for s in range(S):
            R, clk, dec, pw0, e, stored, final, bf, ended = new[s]
            g = self.walks[s]
            y = self.py_pushed[s]
            if final is not None:
                y = max(y, self.py_rec[s] + room(self.fs[s], final[3]))
            if R >= 0 and clk >= 0:
                if not ended:
                    kend[s] = min(windows_of((g.pos - g.mark) * CHUNK, bf, clk), dec)
                py0[s] = self.py_rec[s] if stored else y
                y = max(y, py0[s] + room(self.fs[s] if stored else Framing(), kend[s]))
            ynp[s] = y
        self.py.push(self.py_pushed, ynp, self.py_keep)
        for s in range(S):
            R, clk, dec, pw0, e, stored, final, bf, ended = new[s]
            if final is not None:
                R0, clk0, dec0, K, fin_ended = final
                if K > dec0 and not fin_ended:
                    jobs.append((s, (self.epoch[s], R0), dec0, K))
                f = self.fs[s]
                fjobs.append((s, (self.epoch[s], R0), f.consumed, K, True))
                f.advance(self.fr[s], K, (self.pw_keep[s] - self.pw_rec[s]) // 4)
                self.results[(s, self.epoch[s], R0)] = (f.result(clk0, bf, K), f.data)
            d0 = self.dec[s] if stored else 0
            if R >= 0 and clk >= 0 and dec > d0:
                jobs.append((s, (self.epoch[s], R), d0, dec))
            if not stored:
                self.fs[s] = Framing()
                self.fr[s] = self.framer(s, R, clk) if R >= 0 and clk >= 0 else None
            f = self.fs[s]
            if kend[s] > f.consumed:
                fjobs.append((s, (self.epoch[s], R), f.consumed, kend[s], False))
                # (a recording new to the planes keeps them from window 0; a stored one as the last push left them)
                f.advance(self.fr[s], kend[s], (self.pw_keep[s] - self.pw_rec[s]) // 4 if stored else 0)
            w = self.walks[s]
            on = R >= 0 and clk >= 0
            fixed = on and f.phase == ENDED
            need = f.k0 + 14 * f.nbytes if f.phase == PAYLOAD else max(f.consumed - 3, 0)
            self.keep[s] = w.pos * CHUNK if R < 0 or bf == 0 or fixed else (min(w.pos * CHUNK, R + clk + dec * bf) if on else R)
            self.R[s], self.clk[s] = R, (clk if on else -1)
            self.dec[s], self.pw_rec[s] = (dec if on else 0), (pw0 if on else 0)
            self.pw_pushed[s] = e
            self.pw_keep[s] = pw0 + 4 * (need // 32) if on and not fixed else e
            self.py_rec[s], self.py_pushed[s], self.py_keep[s] = (py0[s] if on else 0), ynp[s], (py0[s] if on else ynp[s])
            assert self.ar.base[s] <= self.keep[s] and np_[s] - self.ar.base[s] <= self.ar.cap[s]
            assert self.pl.base[s] <= self.pw_keep[s] and e - self.pl.base[s] <= self.pl.cap[s]
            assert self.py.base[s] <= self.py_keep[s] and ynp[s] - self.py.base[s] <= self.py.cap[s]
            assert self.py_rec[s] * 2 + f.nbytes <= ynp[s] * 2 or not on          # every byte fits in the slot
        self.pushed = np_
        self.jobs.append(jobs)
        self.frame_jobs.append(fjobs)
        self.windows_total += sum(b - a for _, _, a, b in jobs)
        return out

    def finish(self, ids, settings=None, bauds=None):
        out = super().finish(ids, settings, bauds)
        for s in ids:
            self.fs[s], self.fr[s] = Framing(), None
            self.py_rec[s] = self.py_pushed[s] = self.py_keep[s] = self.py.base[s] = 0
        return out

    def pending_payload(self, s):
        """afsk_rx_streams_pending_payload of channel s, the bytes as (count, prefix or None)"""
        if self.R[s] < 0 or self.clk[s] < 0:
            return -1, 0, False, 0
        return self.fs[s].pending(self.clk[s], bit_frames(self.bauds[s]))

    def plane_words(self, s):
        return (self.pw_pushed[s] - self.pw_keep[s]) // 4


# ---------------------------------------------------------------- CPU checks ----------------------------------------

PIECES = [0, 1, 7, 2047, 2048, 2049, 48000]


def random_windows(rng, n):
    """decision bits and quiet flags of a recording: a random training run, a terminator somewhere (or none), a payload,
    quiet windows after it (or none); sometimes a quiet window right at k0"""
    kind = int(rng.integers(0, 5))
    bits = rng.integers(0, 2, n).astype(np.uint8)
    quiet = np.zeros(n, np.uint8)
    if kind == 0:                                          # no terminator: alternating, then a stuck tone
        bits[:] = 1
        bits[: n // 2: 2] = 0
        return bits, quiet
    t = int(rng.integers(3, 3000))
    bits[:t - 3] = 1                                       # training ones (no 1,0,0,0 before t)
    bits[t - 3:t + 1] = [1, 0, 0, 0]
    if kind == 1:
        quiet[t + 1:] = rng.random(n - t - 1) < 0.3         # a quiet window at k0 or soon after
        quiet[min(t + 1, n - 1)] = rng.random() < 0.5
    elif kind == 2:
        q = int(rng.integers(t + 1, t + 4000))
        quiet[q:] = 1
    return bits, quiet


def make_framers(rng, recs):
    def framer(s, R, clk):
        return recs.setdefault((s, R, clk), ArrayFramer(*random_windows(rng, 400000)))
    return framer


@pytest.mark.parametrize("seed", range(4))
def test_incremental_framing_equals_whole_recording(seed):
    rng = np.random.default_rng(500 + seed)
    bauds = [300, 1200, 6000, 24, 12000, 4800, 2400, 100, 1200, 6000]
    S = len(bauds)
    settings = [(18000, 14000, int(rng.choice([0, 48000, 96000]))) for _ in range(S)]
    n_chunks = 300
    amps = [random_amps(rng, n_chunks) for _ in range(S)]
    clocks, arrays = {}, {}

    def clock(s, R):
        return clocks.setdefault((s, R), int(rng.integers(0, SYNC - 2 * bit_frames(bauds[s]))))

    plan = PayloadPlan(settings, bauds, clock, make_framers(rng, arrays))
    finals = []                                                      # (channel, epoch, R, clk, K, arrays)
    total = n_chunks * CHUNK
    dropped = 0
    snaps = {}                                                       # bytes decoded after each push, per recording

    def collect(ev, before):
        nonlocal dropped
        for s, evs in ev.items():
            for k, e in enumerate(evs):
                if e[0] and k == 0 and e[1] == before[0][s] and before[1][s] >= 0:
                    bf = bit_frames(bauds[s])
                    K = windows_of(e[2] - e[1], bf, before[1][s])
                    finals.append((s, before[2][s], e[1], before[1][s], K, arrays[(s, e[1], before[1][s])]))
                    dropped += before[3][s] > K                      # windows decided beyond the final K

    while min(plan.pushed) < total:
        lens = [min(int(rng.choice(PIECES)), total - p) for p in plan.pushed]
        before = (list(plan.R), list(plan.clk), list(plan.epoch), list(plan.dec))
        ev = plan.push(lens, amps)
        collect(dict(enumerate(ev)), before)
        for s in range(S):
            f = plan.fs[s]
            if plan.R[s] >= 0 and plan.clk[s] >= 0:
                snaps.setdefault((s, plan.epoch[s], plan.R[s]), []).append(f.data)
                if f.phase == TRAIN:                                  # one word before the search point, and the new ones
                    assert plan.plane_words(s) <= -(-(plan.dec[s] - f.consumed) // 32) + 1, (s, plan.plane_words(s))
                if f.phase == ENDED:
                    assert plan.plane_words(s) == 0
        if rng.random() < 0.05:
            ids = [int(s) for s in rng.choice(S, int(rng.integers(1, S + 1)), replace=False)]
            before = (list(plan.R), list(plan.clk), list(plan.epoch), list(plan.dec))
            out = plan.finish(ids)
            collect(out, before)
            for s in ids:
                amps[s] = random_amps(rng, n_chunks)
    assert len(finals) > 5 and dropped > 0
    phases = set()
    for s, ep, R, clk, K, fr in finals:
        want = frame_whole(fr.bits, fr.quiet, K, clk, bit_frames(bauds[s]))
        assert plan.results[(s, ep, R)] == want, (s, R, K)
        assert all(want[1].startswith(d) for d in snaps.get((s, ep, R), []))
        phases.add(("no_term" if want[0][2] == clk + K * bit_frames(bauds[s]) else "term", want[0][0]))
    assert {("term", O.ST_OK), ("no_term", O.ST_NO_DATA)} <= phases, phases


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


def one_recording(bits, quiet, cuts, baud=1200, clk=100, finish_at=None):
    """one channel whose recording opens at chunk 1 and is loud for the whole stream, pushed in pieces cut at `cuts`
    and finished; -> (plan, final result, bytes after every push)"""
    n = cuts[-1]
    amps = [np.full(n // CHUNK + 2, 25000, np.int64)]
    amps[0][0] = 0
    plan = PayloadPlan([(18000, 14000, 48000 * 3600)], [baud], lambda s, R: clk, lambda s, R, c: ArrayFramer(bits, quiet))
    prev, seen = 0, []
    for c in cuts:
        plan.push([c - prev], amps)
        prev = c
        seen.append((plan.fs[0].phase, plan.fs[0].data))
    out = plan.finish([0])
    (ok, a, b), = out[0]
    return plan, plan.results[(0, 0, a)], seen, windows_of(b - a, bit_frames(baud), clk)


def test_quiet_window_at_k0_is_no_data():
    n = 4000
    bits = np.ones(n, np.uint8)
    bits[50:54] = [1, 0, 0, 0]
    quiet = np.zeros(n, np.uint8)
    quiet[54] = 1
    plan, (res, data), seen, K = one_recording(bits, quiet, [CHUNK * 3 + 5, CHUNK * 20])
    assert res == frame_whole(bits, quiet, K, 100, 40)[0] and res[0] == O.ST_NO_DATA and res[3] == 0 and data == b""
    assert seen[-1][0] == ENDED


def test_terminator_across_a_word_and_a_push_boundary():
    """the terminator's 1 in word 2, its zeros in word 3; the pushes cut between its windows"""
    n = 4000
    bits = np.ones(n, np.uint8)
    bits[62] = 0                                          # (no terminator before: 0 then 1s)
    bits[94:98] = [1, 0, 0, 0]                            # windows 94 .. 97: word 2 / word 3
    quiet = np.zeros(n, np.uint8)
    quiet[2000:] = 1
    rng = np.random.default_rng(7)
    bits[98:2000] = rng.integers(0, 2, 1902)
    clk, bf = 100, 40
    # K_safe = windows of the walked chunks; cut so that one push frames up to window 96, the next past it
    cut = CHUNK + clk + 96 * bf + bf                      # frames after which window 96 is decided
    cuts = [CHUNK * 3, -(-cut // CHUNK) * CHUNK + 1, CHUNK * 30, CHUNK * 45]
    plan, (res, data), seen, K = one_recording(bits, quiet, cuts, clk=clk)
    want = frame_whole(bits, quiet, K, clk, bf)
    assert (res, data) == want and res[0] == O.ST_OK and res[3] == 2000 - 98
    assert [p for p, _ in seen][:2] == [TRAIN, TRAIN] or seen[1][0] == PAYLOAD
    for _, d in seen:
        assert want[1].startswith(d)


@pytest.mark.parametrize("piece", [1, 7, 333, 2047, 2049])
def test_byte_groups_straddle_pushes(piece):
    n = 3000
    rng = np.random.default_rng(piece)
    bits = rng.integers(0, 2, n).astype(np.uint8)
    bits[:20] = 1
    bits[20:24] = [1, 0, 0, 0]
    quiet = np.zeros(n, np.uint8)
    clk, bf = 37, 40
    end = CHUNK * 40
    cuts = list(range(CHUNK * 3, end, piece if piece > 100 else 40 * piece)) + [end]
    plan, (res, data), seen, K = one_recording(bits, quiet, cuts, clk=clk)
    want = frame_whole(bits, quiet, K, clk, bf)
    assert (res, data) == want and res[4] > 50
    sizes = [len(d) for _, d in seen]
    assert sizes == sorted(sizes) and len(set(sizes)) > 5           # bytes appeared push by push
    for _, d in seen:
        assert want[1].startswith(d)


def test_windows_decided_beyond_k_safe_are_dropped_by_finish():
    """the last push ends inside a chunk: bits mode decides windows there, which finish cuts off (the result is
    that of the recording up to its last full chunk)"""
    n = 4000
    bits = np.ones(n, np.uint8)
    bits[10:14] = [1, 0, 0, 0]
    rng = np.random.default_rng(3)
    bits[14:] = rng.integers(0, 2, n - 14)
    quiet = np.zeros(n, np.uint8)
    q = 0
    clk, bf = 100, 40
    # K windows of chunks 1 .. 9; the partial chunk 10 holds more decided windows, and a quiet window among them
    K = windows_of(9 * CHUNK, bf, clk)
    q = K + 5
    quiet[q] = 1
    plan, (res, data), seen, K2 = one_recording(bits, quiet, [CHUNK * 10 + 2000], clk=clk)
    assert K2 == K and plan.dec[0] == 0
    want = frame_whole(bits, quiet, K, clk, bf)
    assert (res, data) == want and res[3] == K - 14                    # the quiet window past K does not count
    assert max(d for jobs in plan.jobs for _, _, _, d in jobs) > K


def test_no_terminator_carrier_for_an_hour_keeps_constant_planes():
    """a one-tone carrier (all ones: no terminator) held open for an hour of 1 s pushes beside idle channels"""
    S, baud, piece = 3, 1200, 48000
    pushes = 3600
    n_win = pushes * piece // 40 + 64
    fr = ArrayFramer(np.ones(n_win, np.uint8), np.zeros(n_win, np.uint8))
    amps = [np.full(pushes * piece // CHUNK + 1, 25000, np.int64)] + [np.zeros(pushes * piece // CHUNK + 1, np.int64)] * (S - 1)
    plan = PayloadPlan([(18000, 14000, 48000)] * S, [baud] * S, lambda s, R: 100, lambda s, R, c: fr)
    words, alloc = [], []
    for i in range(pushes):
        plan.push([piece] * S, amps)
        words.append(plan.plane_words(0))
        alloc.append(sum(plan.pl.alloc) + sum(plan.py.alloc))
    assert plan.walks[0].phase == 2 and plan.fs[0].phase == TRAIN and plan.fs[0].consumed > 4 * 10 ** 6
    assert max(words[2:]) <= 40 + 2                                   # 37.5 words a second, plus one
    assert alloc[-1] == alloc[10]                                      # flat after the first pushes
    assert plan.pl.moved // 4 <= 64 * pushes and plan.py.moved <= 64 * pushes


def test_payload_then_quiet_then_carrier_stops_deciding():
    """a recording whose first quiet window (inside a loud chunk) follows its message: after the push that frames it,
    no window is decided and no plane kept, and the result is fixed"""
    n = 400000
    bits = np.ones(n, np.uint8)
    bits[40:44] = [1, 0, 0, 0]
    rng = np.random.default_rng(11)
    bits[44:44 + 14 * 20] = rng.integers(0, 2, 14 * 20)
    quiet = np.zeros(n, np.uint8)
    quiet[44 + 14 * 20] = 1
    cuts = [48000 * (i + 1) for i in range(60)]
    amps = [np.full(60 * 48000 // CHUNK + 2, 25000, np.int64)]
    amps[0][0] = 0
    plan = PayloadPlan([(18000, 14000, 48000 * 3600)], [1200], lambda s, R: 100, lambda s, R, c: ArrayFramer(bits, quiet))
    prev, decs = 0, []
    for c in cuts:
        plan.push([c - prev], amps)
        prev = c
        decs.append(plan.dec[0])
        if plan.fs[0].phase == ENDED:
            assert plan.plane_words(0) == 0 and plan.pushed[0] - plan.keep[0] < CHUNK
    assert plan.fs[0].phase == ENDED and len(set(decs[1:])) == 1
    out = plan.finish([0])
    (_, a, b), = out[0]
    K = windows_of(b - a, 40, 100)
    assert plan.results[(0, 0, a)] == frame_whole(bits, quiet, K, 100, 40)
    assert plan.results[(0, 0, a)][0][4] == 20
