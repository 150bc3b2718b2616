"""Streaming handles against the oracle at scale.  Receive: every demodulator and clock family decodes streamed
recordings, through host and device planar pushes and interleaved pushes; a recording long enough for k_frame ends in
the same push as short ones at other bauds; 4096 channels with mixed settings, partial finishes and arena compactions.
Transmit: 4096 channels over every TX golden baud, pulled every way, frame-exact against the oracle's timeline across
payload-arena compactions.  Every expected value comes from oracle/oracle.py: listen_gate_multi over each channel's
whole stream, rx_decode of each recorded call, tx_frames of each message at its start frame.

The traffic generators and the retention models below import no torch: tests/test_stream_oracle_plan.py checks on
the CPU that the traffic covers what these tests claim."""
import functools
import json
import os

import numpy as np
import pytest

import afskmodem_b200 as A
from oracle import oracle as O
from test_gpu_stream_each import THRESHOLDS, TIMEOUTS, lim_of, to_device
from test_gpu_streams import golden_cuts, schedule_pieces
from test_stream_gate_model import CHUNK, GateWalk, chunk_amps, final_prefix
from test_stream_retention_model import Arena
from test_stream_tx_model import Msg, TimelineWindow, TxModel, random_payload

pytestmark = pytest.mark.gpu
A.LOG_LEVEL = 5
THREADS = os.cpu_count() or 1
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

# the bauds of test_gpu_parity.py::test_random_sweep_vs_oracle, and 4800 (the reference's load raises there)
SWEEP_BAUDS = [300, 600, 800, 1200, 2400, 4000, 6000, 12000, 100, 24, 375, 1000, 2000, 3000, 1500, 500, 750, 480, 400, 240,
               250, 160, 125, 60, 30]
DEMOD_BAUDS = SWEEP_BAUDS + [4800]
# bauds at which the reference decodes no message: load raises at 4800; at 12000 (4 samples per bit) it recovers the
# clock but never finds the end of the training sequence ("No data.")
NO_MESSAGE = {4800: O.ST_EXC_WAVELEN, 12000: O.ST_NO_DATA}
PIECES = [0, 1, 7, 2047, 2048, 2049, 48000]
K_FRAME_WARP_MAX_WINDOWS = 262144                    # afsk_rx.cu kFrameWarpMaxWindows


# ---------------------------------------------------------------- oracle ------------------------------------------

def render(n, placed, sigma, rng=None, noise=None):
    """n frames: float segments added at their start frames to AWGN of sigma (drawn, or a slice of unit noise),
    rounded and clipped to int16"""
    if noise is not None:
        x = noise * sigma
    else:
        x = rng.normal(0, sigma, n) if sigma else np.zeros(n)
    for at, seg in placed:
        x[at:at + len(seg)] += seg[:n - at]
    return np.clip(np.round(x), -32768, 32767).astype(np.int16)


def oracle_decodes(jobs):
    """[(samples, baud, amp_end)] -> the oracle's (status, clock, train_end, nbits, payload) of each, in blocks"""
    out, i = [], 0
    while i < len(jobs):
        j, tot = i, 0
        while j < len(jobs) and (j == i or tot + len(jobs[j][0]) <= 1 << 26):
            tot += len(jobs[j][0])
            j += 1
        blk = jobs[i:j]
        off = np.zeros(len(blk) + 1, np.int64)
        np.cumsum([len(x) for x, _, _ in blk], out=off[1:])
        datas, res = O.rx_decode_batch(np.concatenate([x for x, _, _ in blk]), off, [b for _, b, _ in blk],
                                       [a for _, _, a in blk], threads=THREADS)
        out += [(r.status, r.clock, r.train_end, r.nbits, d) for r, d in zip(res, datas)]
        i = j
    return out


def oracle_calls(streams, settings):
    """per stream (settings (baud, amp_start, amp_end, timeout s)): its listen_gate_multi calls, and the oracle decode
    of every recorded call, keyed (stream index, start, end)"""
    wants = [O.listen_gate_multi(x, a0, a1, int(t * 48000)) for x, (_, a0, a1, t) in zip(streams, settings)]
    jobs, keys = [], []
    for k, (x, (b, _, a1, _), w) in enumerate(zip(streams, settings, wants)):
        for rec, a, e in w:
            if rec:
                jobs.append((x[a:e], b, a1))
                keys.append((k, a, e))
    return wants, dict(zip(keys, oracle_decodes(jobs)))


def oracle_values(o):
    """what receive() returns for a recording the oracle decodes to o: (string=False, string=True); an exception as
    (type name, message)"""
    if o[0] < 0:
        return O.EXC_TEXT[o[0]], O.EXC_TEXT[o[0]]
    if o[0] != O.ST_OK:
        return b"", b""
    try:
        s = o[4].decode("utf-8")
    except UnicodeDecodeError as e:
        s = (type(e).__name__, str(e))
    return o[4], s


# ---------------------------------------------------------------- traffic -----------------------------------------

def demod_channels(seed=7100):
    """Two channels per baud of DEMOD_BAUDS.  Each: random lead silence, 1-3 messages (the first channel's first one
    clean, with 0.5 s of training; the others 0.02-0.5 s, gains from just below to just above amp_start), one
    full-scale clipped burst after the first message, AWGN of sigma 0-8000; thresholds and timeouts (0 among them)
    mixed.  All channels padded with silence and noise to one length.  -> [dict(baud, a0, a1, timeout, x, pays)]"""
    rng = np.random.default_rng(seed)
    chans = []
    for i, baud in enumerate(DEMOD_BAUDS):
        hi = max(1, min(8, 60000 // (14 * (48000 // baud))))          # at most ~60000 frames of payload
        for j in range(2):
            a0, a1 = THRESHOLDS[(i + j) % 3]
            timeout = (0.5, 1.0, 2.0)[i % 3] if j == 0 else TIMEOUTS[(i + j) % 4]
            sigma = float(rng.choice([0, 1000, 2000])) if j == 0 else float(rng.choice([0, 3000, 5000, 8000]))
            pos = int(rng.integers(0, 30000))
            placed, pays = [], []
            for k in range(int(rng.integers(1, 4))):
                pay = rng.integers(0, 256, int(rng.integers(1, hi + 1)), dtype=np.uint8).tobytes()
                if k == 0 and j == 0:
                    tt, gain = 0.5, 1.0
                else:
                    tt = float(rng.choice([0.02, 0.1, 0.25, 0.5]))
                    gain = min(1.0, a0 / 32767 * rng.uniform(0.9, 1.15))
                seg = O.tx_frames(pay, baud, tt).astype(np.float64) * gain
                placed.append((pos, seg))
                pays.append(pay)
                pos += len(seg) + int(rng.integers(2048, 20000))
                if k == 0:
                    burst = rng.normal(0, 60000, int(rng.integers(3000, 20000)))
                    placed.append((pos, burst))
                    pos += len(burst) + int(rng.integers(2048, 20000))
            chans.append(dict(baud=baud, a0=a0, a1=a1, timeout=timeout, sigma=sigma, placed=placed, pays=pays, n=pos))
    n = max(c["n"] for c in chans) + 30000
    for c in chans:
        c["x"] = render(n, c.pop("placed"), c.pop("sigma"), rng)
        del c["n"]
    return chans


def piece_cuts(n, rng):
    """cuts of pieces of PIECES' lengths, and random ones up to 20000, in shuffled rounds"""
    cuts, c = [], 0
    while True:
        for p in rng.permutation(PIECES + [int(rng.integers(0, 20001))]):
            c += int(p)
            if c >= n:
                return cuts
            cuts.append(c)


def long_frame_channels(seed=7200):
    """Channel 0: a ~20 KB message at 6000 baud (> 262,144 windows).  Channels 1-3: short messages at 1200, 3000 and
    300 baud whose recordings end within 9000 frames before the long one's, so that a schedule of 48000-frame pushes
    finalizes all four in one push.  -> (channels as in demod_channels, long payload, that push's index)"""
    rng = np.random.default_rng(seed)
    long_pay = rng.integers(0, 256, 20000, dtype=np.uint8).tobytes()
    tx = O.tx_frames(long_pay, 6000, 0.1)
    lead = 31337
    loud_end = lead + len(tx) - 4800                                   # save()'s frames end with 4800 silent ones
    placed = [[(lead, tx.astype(np.float64))]]
    pays = [[long_pay]]
    for baud, back in ((1200, 0), (3000, 3000), (300, 9000)):
        pay = rng.integers(0, 256, 6, dtype=np.uint8).tobytes()
        fr = O.tx_frames(pay, baud, 0.1).astype(np.float64)
        placed.append([(loud_end - back - (len(fr) - 4800), fr)])
        pays.append([pay])
    n = loud_end + 60000
    chans = [dict(baud=b, a0=18000, a1=14000, timeout=1.0, x=render(n, p, 1500, rng), pays=q)
             for b, p, q in zip((6000, 1200, 3000, 300), placed, pays)]
    ends = [max(e for rec, _, e in O.listen_gate_multi(c["x"], 18000, 14000, 48000) if rec) for c in chans]
    push = -(-ends[0] // 48000) - 1
    assert all(-(-e // 48000) - 1 == push for e in ends), ends
    return chans, long_pay, push


MANY_S, MANY_PIECE, MANY_PUSHES = 4096, 48000, 4
MANY_BAUDS = [6000, 3000, 2000, 1200, 800, 480, 1500, 750]    # k_clock_q (8 / 16 / 24), k_demod, k_demod_shift, padded
MANY_Q = 2400                                                   # 6000-baud channels


def many_settings(seed=7300):
    """4096 channels: 2400 at 6000 baud, the rest over the other bauds; three threshold pairs, four timeouts (no 0 s
    timeout at 6000 baud, where it would record nothing).  150 other channels are finished after the second push
    with new settings, 150 with their own.  -> (settings [(baud, a0, a1, timeout s)], {id: new settings}, [ids])"""
    rng = np.random.default_rng(seed)
    bauds = [6000] * MANY_Q + [MANY_BAUDS[1 + i % 7] for i in range(MANY_S - MANY_Q)]
    bauds = [bauds[i] for i in rng.permutation(MANY_S)]
    settings = []
    for b in bauds:
        a0, a1 = THRESHOLDS[int(rng.integers(0, 3))]
        settings.append((b, a0, a1, float(rng.choice(TIMEOUTS[1:] if b == 6000 else TIMEOUTS))))
    fin = [int(s) for s in rng.permutation([s for s in range(MANY_S) if bauds[s] != 6000])[:300]]
    new = {}
    for s in sorted(fin[:150]):
        a0, a1 = THRESHOLDS[int(rng.integers(0, 3))]
        new[s] = (MANY_BAUDS[int(rng.integers(0, 8))], a0, a1, float(rng.choice(TIMEOUTS)))
    return settings, new, sorted(fin[150:])


@functools.lru_cache(maxsize=1)
def unit_noise(seed=7301):
    return np.random.default_rng(seed).normal(0, 1, 1 << 20)


def many_channel(s, setting, seed=7300):
    """channel s's 4 s: AWGN of sigma 0-6000 and 1-3 messages, the first near amp_start and 90000-130000 frames long
    (its recording stays pending over the second push's end, and its slot must grow in the third); at 6000 baud two,
    whose recordings both end in the third push"""
    baud, a0 = setting[0], setting[1]
    rng = np.random.default_rng([seed, s])
    n = MANY_PIECE * MANY_PUSHES
    sigma = float(rng.choice([0, 1000, 3000, 6000]))
    bank = unit_noise()
    off = int(rng.integers(0, len(bank) - n))

    def msg(gain, tt, nbytes=None):
        pay = rng.integers(0, 256, nbytes or int(rng.integers(1, 9)), dtype=np.uint8).tobytes()
        return O.tx_frames(pay, baud, tt).astype(np.float64) * gain

    near = min(1.0, a0 / 32767 * rng.uniform(0.9, 1.15))
    if baud == 6000:
        a = msg(near, 0.05, int(rng.integers(80000, 95000)) // 112)
        at = int(rng.integers(0, 10000))
        b = msg(1.0, float(rng.choice([0.02, 0.05, 0.1])))
        placed = [(at, a), (max(at + len(a) + int(rng.integers(2048, 6000)), 100000), b)]
    else:
        placed, pos = [], int(rng.integers(0, 20000))
        for k in range(int(rng.integers(1, 4))):
            long = int(rng.integers(90000, 130000)) // (14 * (48000 // baud)) if k == 0 else None
            seg = msg(near if k == 0 else rng.uniform(0.6, 1.0), float(rng.choice([0.02, 0.1, 0.3])), long)
            if pos + len(seg) > n:
                break
            placed.append((pos, seg))
            pos += len(seg) + int(rng.integers(2048, 40000))
    return render(n, placed, sigma, noise=bank[off:off + n].copy())


class ArenaPlan:
    """EachHandle (test_stream_each_model) fed chunk amplitudes instead of samples: per channel the resumable walk
    with its settings, the frames pushed and retained, the arena's slots (Arena); finish(ids, settings) ends the
    listed channels' streams.  Counts the whole-arena compactions of pushes that began with a recording pending."""

    def __init__(self, settings):
        self.S = len(settings)
        self.settings = list(settings)                             # (amp_start, amp_end, timeout frames)
        self.walks = [GateWalk(*x) for x in settings]
        self.ar = Arena(self.S)
        self.pushed, self.keep = [0] * self.S, [0] * self.S
        self.pending_compactions = 0

    def push(self, lens, amps):
        """lens[s] new frames of channel s, whose current stream's chunk amplitudes are amps[s]; -> events per channel"""
        np_ = [p + n for p, n in zip(self.pushed, lens)]
        c0, pending = self.ar.compactions, any(w.phase == 2 for w in self.walks)
        self.ar.push(self.pushed, np_, self.keep)
        self.pending_compactions += pending and self.ar.compactions > c0
        out = []
        for s in range(self.S):
            out.append(self.walks[s].walk(amps[s][self.pushed[s] // CHUNK:np_[s] // CHUNK]))
            self.keep[s] = self.walks[s].retained_from()
            assert self.ar.base[s] <= self.keep[s] and np_[s] - self.ar.base[s] <= self.ar.cap[s]
        self.pushed = np_
        return out

    def finish(self, ids, settings=None):
        out = {}
        for i, s in enumerate(ids):
            out[s] = self.walks[s].walk(np.zeros(0, np.int64), finish=True)
            if settings is not None:
                self.settings[s] = settings[i]
            self.walks[s] = GateWalk(*self.settings[s])
            self.pushed[s] = self.keep[s] = self.ar.base[s] = 0
        return out


def many_plan():
    """test_4096_receive_channels' traffic as chunk amplitudes through ArenaPlan: -> (settings, the model after the
    last push, per push the recorded events per baud (of the stream that was current))"""
    settings, new, plain = many_settings()
    S, piece, split = MANY_S, MANY_PIECE, 2 * MANY_PIECE
    fin = set(new) | set(plain)
    amps, amps2 = [], {}
    for s in range(S):
        x = many_channel(s, settings[s])
        amps.append(chunk_amps(x[:split] if s in fin else x))
        if s in fin:
            amps2[s] = chunk_amps(x[split:])
    plan = ArenaPlan([(a0, a1, int(t * 48000)) for _, a0, a1, t in settings])
    cur = list(settings)
    per_push = []
    for i in range(MANY_PUSHES):
        ev = plan.push([piece] * S, amps)
        count = {}
        for s in range(S):
            count[cur[s][0]] = count.get(cur[s][0], 0) + sum(1 for e in ev[s] if e[0])
        per_push.append(count)
        if i == 1:
            ids = sorted(new)
            plan.finish(ids, [(new[s][1], new[s][2], int(new[s][3] * 48000)) for s in ids])
            plan.finish(plain)
            for s in fin:
                amps[s] = amps2[s]
                cur[s] = new.get(s, cur[s])
    return settings, plan, per_push


def tx_golden_bauds():
    return sorted({m["baud"] for m in json.load(open(os.path.join(GOLDEN, "tx_cases.json"))) if m["exc"] is None})


TX_PULLS = [0, 1, 7, 8, 9, 2047, 2048, 48000]
TX_TTS = [0.0, 0.01, 0.05, 0.2]


def tx_plan(seed=7400, S=4096, rounds=40):
    """4096 transmit channels, each at a TX golden baud with a training time of TX_TTS.  Three messages of several
    KB on fast channels, then rounds of a send to many channels (a channel listed twice gets its messages back to
    back; empty payloads among them) and a pull of TX_PULLS' sizes in turn; 300 channels configured half way.
    -> (settings [(baud, tt)], ops)"""
    rng = np.random.default_rng(seed)
    bauds = tx_golden_bauds()
    cfg = [(bauds[int(rng.integers(0, len(bauds)))], float(rng.choice(TX_TTS))) for _ in range(S)]
    big = [s for s in range(S) if cfg[s][0] in (8000, 12000, 24000)][:3]
    ops = [("send", big, [rng.integers(0, 256, int(rng.integers(2000, 6000)), dtype=np.uint8).tobytes() for _ in big])]
    for r in range(rounds):
        ids = [int(x) for x in rng.integers(0, S, int(rng.integers(S // 4, S)))]
        ops.append(("send", ids, [random_payload(rng, 12) for _ in ids]))
        ops.append(("pull", TX_PULLS[r % len(TX_PULLS)]))
        if r == rounds // 2:
            ids = [int(x) for x in rng.choice(S, 300, replace=False)]
            ops.append(("configure", ids, [(bauds[int(rng.integers(0, len(bauds)))], float(rng.choice(TX_TTS))) for _ in ids]))
    ops += [("pull", 48000), ("pull", 48000)]
    return cfg, ops


class TxEachModel(TxModel):
    """TxModel with per-channel settings (afsk_tx_streams_create_each / _configure): each message takes its channel's
    baud and training time at send time.  var_across: per compaction, the unequal-tone messages queued across it."""

    def __init__(self, cfg):
        super().__init__(len(cfg), 1200, 0.0, synth=False)
        self.cfg = list(cfg)
        self.var_across = []

    def configure(self, ids, cfg):
        for s, c in zip(ids, cfg):
            self.cfg[s] = c

    def send(self, streams, payloads):
        msgs = [Msg(bytes(p), self.cfg[s][0], O.ts_cycles(*self.cfg[s])) for s, p in zip(streams, payloads)]
        W = sum(m.block for m in msgs)
        if self.top + W > self.cap:
            while 2 * (self.live + W) > self.cap:
                self.cap *= 2
            self.moved += self.live
            self.compactions += 1
            self.top = self.live
            self.var_across.append([m for q in self.q for m in q if m.ml != m.sl])
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


# ---------------------------------------------------------------- GPU drivers -------------------------------------

def take(got, ev, when=None, tag=None):
    """appends (call, recorded, start, end, value, string value, decode) per event to got[channel]; exceptions as
    (type name, message)"""
    def plain(v):
        return (type(v).__name__, str(v)) if isinstance(v, Exception) else v
    vb = ev.values(string=False, errors="return")
    vs = ev.values(string=True, errors="return")
    k = 0
    for i in range(len(ev)):
        s, r = int(ev.stream[i]), None
        if ev.recorded[i]:
            b = ev.batch
            r = (int(b.status[k]), int(b.clock[k]), int(b.train_end[k]), int(b.nbits[k]), b.payload(k))
            k += 1
        got[s].append((int(ev.call[i]), bool(ev.recorded[i]), int(ev.start[i]), int(ev.end[i]), plain(vb[i]), plain(vs[i]), r))
        if when is not None:
            when[s].append(tag)


def push(st, pieces, mode):
    """host / device planar, or interleaved (equal pieces) as bytes, a (n, S) or a flat CUDA tensor"""
    import torch
    if mode == "host":
        return st.push(pieces)
    if mode == "device":
        return st.push(*to_device(pieces))
    X = np.stack(pieces, axis=1)
    if mode == "bytes":
        return st.push_interleaved(X.tobytes())
    t = torch.from_numpy(X).cuda()
    return st.push_interleaved(t if mode == "tensor" else t.reshape(-1))


def check_prefix(st, got, wants, amps, pushed, settings):
    """each channel's calls so far are exactly its oracle calls final within the frames pushed; state agrees"""
    for s in range(len(got)):
        n = final_prefix(wants[s], amps[s], pushed[s] // CHUNK, lim_of(settings[s][3]), settings[s][2])
        assert [g[1:4] for g in got[s]] == wants[s][:n], (s, pushed[s])
        p, pend, ret = st.state(s)
        assert p == pushed[s] and ret == p - (pend if pend >= 0 else p // CHUNK * CHUNK), s


def check_final(calls, want, dec, k):
    """stream k's calls after finish: the oracle's calls, decodes and receive() values"""
    assert [c[0] for c in calls] == list(range(len(calls))), k
    assert [c[1:4] for c in calls] == want, k
    for call, rec, a, b, vb, vs, r in calls:
        if not rec:
            assert vb == b"" and vs == b"", (k, call)
            continue
        o = dec[(k, a, b)]
        assert r == o, (k, call)
        assert (vb, vs) == oracle_values(o), (k, call)


def run_streams(st, streams, ends, modes, wants, settings, when=None):
    """pushes up to ends[i][s] frames of each stream in push i (modes in turn), checking the final prefix after every
    push; then finish"""
    S = len(streams)
    got = [[] for _ in range(S)]
    amps = [chunk_amps(x) for x in streams]
    prev = [0] * S
    for i, e in enumerate(ends):
        take(got, push(st, [x[p:q] for x, p, q in zip(streams, prev, e)], modes[i % len(modes)]), when, i)
        check_prefix(st, got, wants, amps, e, settings)
        prev = e
    take(got, st.finish(), when, len(ends))
    return got


def receivers(settings):
    cache = {}
    return [cache.setdefault(x[:3], A.Receiver(*x[:3])) for x in settings]


@functools.lru_cache(maxsize=1)
def demod_case():
    chans = demod_channels()
    settings = [(c["baud"], c["a0"], c["a1"], c["timeout"]) for c in chans]
    streams = [c["x"] for c in chans]
    return chans, settings, streams, oracle_calls(streams, settings)


@pytest.mark.parametrize("mode", ["host", "device", "interleaved"])
def test_every_demodulator_family_through_one_handle(mode):
    chans, settings, streams, (wants, dec) = demod_case()
    S, n = len(streams), len(streams[0])
    rng = np.random.default_rng(["host", "device", "interleaved"].index(mode))
    if mode == "interleaved":
        ends = [[c] * S for c in piece_cuts(n, rng)] + [[n] * S]
        modes = ["bytes", "tensor", "flat"]
    else:
        cuts = [(golden_cuts(n, rng) + [piece_cuts(n, rng)])[s % 6] for s in range(S)]
        _, bounds = schedule_pieces(streams, cuts)
        ends = [[b[min(i + 1, len(b) - 1)] for b in bounds] for i in range(max(len(b) - 1 for b in bounds))]
        modes = [mode]
    with A.open_receive_streams(receivers(settings), [x[3] for x in settings]) as st:
        got = run_streams(st, streams, ends, modes, wants, settings)
    for s in range(S):
        check_final(got[s], wants[s], dec, s)
    for baud in DEMOD_BAUDS:                                            # not vacuous: every baud decoded a message
        rec = [c for s in range(S) if chans[s]["baud"] == baud for c in got[s] if c[1]]
        sent = [p for c in chans if c["baud"] == baud for p in c["pays"]]
        if baud in NO_MESSAGE:
            assert any(c[6][0] == NO_MESSAGE[baud] for c in rec), baud
        else:
            assert any(c[6][0] == O.ST_OK and c[4] in sent for c in rec), baud
    for bad in (9600, 1100):                                            # the reference's constructor refuses these
        with pytest.raises(Exception, match="Invalid baud rate."):
            A.Receiver(bad)


def test_k_frame_recording_ends_with_short_ones():
    chans, long_pay, final_push = long_frame_channels()
    settings = [(c["baud"], c["a0"], c["a1"], c["timeout"]) for c in chans]
    streams = [c["x"] for c in chans]
    wants, dec = oracle_calls(streams, settings)
    n = len(streams[0])
    ends = [[min(n, (i + 1) * 48000)] * 4 for i in range(-(-n // 48000))]
    when = [[] for _ in chans]
    with A.open_receive_streams(receivers(settings), 1.0) as st:
        got = run_streams(st, streams, ends, ["host", "device"], wants, settings, when)
    for s in range(4):
        check_final(got[s], wants[s], dec, s)
        last = max(i for i, c in enumerate(got[s]) if c[1])
        assert when[s][last] == final_push, s                       # all four end in one push
        assert got[s][last][4] == chans[s]["pays"][0], s           # channel 0: the long payload
    a, b = got[0][max(i for i, c in enumerate(got[0]) if c[1])][2:4]
    assert (b - a) // 8 - 1 > K_FRAME_WARP_MAX_WINDOWS and chans[0]["pays"][0] == long_pay


def test_4096_receive_channels_mixed_settings_through_compactions():
    settings, new, plain = many_settings()
    S, piece, split = MANY_S, MANY_PIECE, 2 * MANY_PIECE
    fin = sorted(set(new) | set(plain))
    X = np.empty((S, piece * MANY_PUSHES), np.int16)
    for s in range(S):
        X[s] = many_channel(s, settings[s])
    # streams: channel s's first stream (its first two pushes if it is finished then), and the second streams
    first = [X[s, :split] if s in new or s in plain else X[s] for s in range(S)]
    second = [X[s, split:] for s in fin]
    set2 = [new.get(s, settings[s]) for s in fin]
    wants, dec = oracle_calls(first + second, settings + set2)
    idx = {s: S + i for i, s in enumerate(fin)}                     # stream index of each finished channel's second stream
    amps = [chunk_amps(x) for x in first + second]
    model = ArenaPlan([(a0, a1, int(t * 48000)) for _, a0, a1, t in settings])
    streams_got = {k: [] for k in range(len(wants))}
    cur = list(range(S))                                            # the stream index each channel is on
    cur_set = list(settings)
    got = [streams_got[k] for k in cur]
    modes = ["device", "tensor", "bytes", "device"]
    busiest, compact_pending, pending = {}, False, False
    with A.open_receive_streams(receivers(settings), [x[3] for x in settings]) as st:
        for i in range(MANY_PUSHES):
            c0 = st.counters()
            ev = push(st, [X[s, i * piece:(i + 1) * piece] for s in range(S)], modes[i])
            take(got, ev)
            model.push([piece] * S, [amps[k] for k in cur])
            c = st.counters()
            compact_pending |= pending and c["compactions"] > c0["compactions"]
            count = {}
            for j in np.flatnonzero(ev.recorded):
                b = cur_set[int(ev.stream[j])][0]
                count[b] = count.get(b, 0) + 1
            if count.get(6000, 0) > busiest.get(6000, 0):
                busiest = count
            pushed = [(i + 1) * piece - (split if cur[s] >= S else 0) for s in range(S)]
            check_prefix(st, got, [wants[k] for k in cur], [amps[k] for k in cur], pushed, cur_set)
            pending = any(st.state(s)[1] >= 0 for s in range(S))
            if i == 1:
                ids = sorted(new)
                take(got, st.finish(ids, receivers([new[s] for s in ids]), [new[s][3] for s in ids]))
                take(got, st.finish(plain))
                model.finish(ids, [(new[s][1], new[s][2], int(new[s][3] * 48000)) for s in ids])
                model.finish(plain)
                for s in fin:
                    cur[s], cur_set[s] = idx[s], new.get(s, settings[s])
                    got[s] = streams_got[cur[s]]
                    assert st.state(s) == (0, -1, 0)
        c = st.counters()
        take(got, st.finish())
    assert c["compactions"] >= 1 and c["moved_frames"] > 0 and compact_pending
    assert (c["moved_frames"], c["compactions"]) == (model.ar.moved, model.ar.compactions)
    assert busiest[6000] > 2000 and len(busiest) >= 4, busiest
    for k, calls in streams_got.items():
        check_final(calls, wants[k], dec, k)


def pull(st, n, mode):
    """mode 0 / 1: pull into host / a device tensor, 2 / 3: pull_interleaved into host / a device tensor; a device
    tensor's guard values past S * n must stay"""
    import torch
    S = st.S
    if mode in (0, 2):
        return (st.pull(n) if mode == 0 else st.pull_interleaved(n)).copy()
    t = torch.full((S * n + 24,), 0x5A5A, dtype=torch.int16, device="cuda")
    assert (st.pull(n, out=t) if mode == 1 else st.pull_interleaved(n, out=t)) is t
    g = t.cpu().numpy()
    assert (g[S * n:] == 0x5A5A).all()
    return g[:S * n].reshape((S, n) if mode == 1 else (n, S))


def test_4096_transmit_channels_every_family():
    cfg, ops = tx_plan()
    S = len(cfg)
    assert {b for b, _ in cfg} == set(tx_golden_bauds()) and len(set(b for b, _ in cfg)) == 15
    txs = {}

    def tx(c):
        return txs.setdefault(c, A.Transmitter(*c))

    model, win = TxEachModel(cfg), TimelineWindow(S)
    sent, P, k, checked = [], 0, 0, 0
    with A.open_transmit_streams([tx(c) for c in cfg]) as st:
        for op in ops:
            if op[0] == "configure":
                st.configure(op[1], [tx(c) for c in op[2]])
                model.configure(op[1], op[2])
            elif op[0] == "send":
                a, b = st.send(op[1], op[2])
                at = [model.cfg[s] for s in op[1]]
                wa, wb = model.send(op[1], op[2])
                assert np.array_equal(a, wa) and np.array_equal(b, wb)
                for s, p, x, y, c in zip(op[1], op[2], a, b, at):
                    win.add(s, p, int(x), int(y), *c)
                    sent.append((s, int(x)))
            else:
                n, mode = op[1], k % 4
                want = win.window(P, n)
                got = pull(st, n, mode)
                assert np.array_equal(got, want if mode < 2 else want.T), (P, n, mode)
                checked += int(want.any(axis=1).sum())
                model.pull(n)
                P += n
                k += 1
                c = st.counters()
                assert (c["moved_bytes"], c["compactions"]) == (model.moved, model.compactions), P
                assert [st.state(s) for s in range(0, S, 61)] == [model.state(s) for s in range(0, S, 61)]
    assert any(a % 2 for _, a in sent) and checked > S
    assert sum(1 for v in model.var_across if any(m.end <= P for m in v)) >= 3
