"""Payload-mode retention (open_receive_streams(..., retain="payload")) against samples mode, the oracle and the CPU
model of its bookkeeping (test_stream_payload_model.PayloadPlan): every demodulator family through host, device and
interleaved pushes; a recording of more than 262,144 windows decoded progressively; 4096 channels with mixed settings
and partial finishes; a one-tone carrier that never ends; a message whose first quiet window lies inside a loud chunk;
and the edge cases of bits mode."""
import numpy as np
import pytest

import afskmodem_b200 as A
from oracle import oracle as O
from test_gpu_stream_bits import edge_case, oracle_clock
from test_gpu_stream_oracle import (MANY_PIECE, MANY_PUSHES, MANY_S, check_final, demod_case, long_frame_channels, many_channel,
                                    many_settings, oracle_calls, piece_cuts, push, receivers, take)
from test_gpu_streams import golden_cuts, schedule_pieces
from test_stream_bits_model import bit_frames, windows_of
from test_stream_gate_model import CHUNK, chunk_amps
from test_stream_payload_model import ENDED, MarkFramer, PayloadPlan

pytestmark = pytest.mark.gpu
A.LOG_LEVEL = 5


def oracle_framer(streams, settings):
    """framer(s, R, clk) of the model: the terminator and first quiet window of the recording from R of channel s's
    current stream, from the oracle's decode of everything the test will push of it"""
    def framer(s, R, clk):
        x = streams[s]() if callable(streams[s]) else streams[s]
        baud, _, a1, _ = settings[s]
        bf = bit_frames(baud)
        o = O.rx_decode(x[R:], baud, a1)
        assert o["clock"] == clk, (s, R)
        Kall = windows_of(len(x) - R, bf, clk)
        k0 = (o["train_end"] - clk) // bf
        if k0 >= Kall:
            return MarkFramer(None, None)
        k1 = k0 + o["nbits"]
        return MarkFramer(k0 - 1, k1 if k1 < Kall else None)
    return framer


def model_of(settings, streams):
    return PayloadPlan([(a0, a1, int(t * 48000)) for _, a0, a1, t in settings], [b for b, *_ in settings],
                       oracle_clock(streams, settings), oracle_framer(streams, settings))


class Prefixes:
    """pending_payload after every push; each snapshot checked against the call's result once it is final"""

    def __init__(self, S):
        self.snaps = [[] for _ in range(S)]
        self.ended_early = 0
        self.checked = 0
        self.gpu_framed = set()              # channels whose open recording the GPU reported framed, with decoded bytes

    def record(self, st, model, S):
        for s in range(S):
            te, nb, ended, data = st.pending_payload(s)
            want = model.pending_payload(s)
            assert (te, nb, ended, len(data)) == want, (s, want)
            if te >= 0 and data:
                self.gpu_framed.add(s)
            if st.state(s)[1] >= 0 and st.pending_bits(s)[0] >= 0:
                self.snaps[s].append((st.state(s)[1], te, nb, ended, data))

    def final(self, got):
        for s, calls in enumerate(got):
            keep = []
            for R, te, nb, ended, data in self.snaps[s]:
                r = [c[6] for c in calls if c[1] and c[2] == R]
                if not r:
                    keep.append((R, te, nb, ended, data))
                    continue
                status, clk, train_end, nbits, pay = r[-1]
                assert pay.startswith(data), (s, R)
                if ended:
                    assert (data, te, nb) == (pay, train_end, nbits), (s, R)
                    self.ended_early += 1
                self.checked += 1
            self.snaps[s] = keep


def check_model(st, model, S):
    for s in range(S):
        want_state, want_bits = model.state(s)
        assert st.state(s) == want_state, s
        assert st.pending_bits(s) == want_bits, s
    c = st.counters()
    assert (c["moved_frames"], c["compactions"]) == (model.ar.moved, model.ar.compactions)
    assert (c["moved_plane_words"], c["plane_compactions"]) == (model.pl.moved // 4, model.pl.compactions)
    assert (c["moved_payload_bytes"], c["payload_compactions"]) == (2 * model.py.moved, model.py.compactions)


def twin_run(settings, streams, ends, modes, finish_some=None):
    """samples- and payload-mode handles fed the same pushes (ends[i][s]: frames of stream s after push i, modes in
    turn): equal events, results, payloads and values after every push and finish; the payload handle's state,
    pending_bits, pending_payload and counters equal the model's.  finish_some: {push index: channel ids}."""
    S = len(streams)
    rx, tmo = receivers(settings), [x[3] for x in settings]
    model = model_of(settings, streams)
    amps = [chunk_amps(x) for x in streams]
    ga, gb = [[] for _ in range(S)], [[] for _ in range(S)]
    pre = Prefixes(S)
    prev = [0] * S
    with A.open_receive_streams(rx, tmo) as sa, A.open_receive_streams(rx, tmo, retain="payload") as sb:
        assert (sa.retain, sb.retain) == ("samples", "payload")
        for i, e in enumerate(ends):
            pieces = [x[p:q] for x, p, q in zip(streams, prev, e)]
            mode = modes[i % len(modes)]
            take(ga, push(sa, pieces, mode))
            take(gb, push(sb, pieces, mode))
            assert ga == gb, i
            model.push([len(x) for x in pieces], amps)
            check_model(sb, model, S)
            pre.final(gb)
            pre.record(sb, model, S)
            prev = e
            if finish_some and i in finish_some:
                ids = finish_some[i]
                keep = {s: (sb.pending_bits(s), sb.pending_payload(s)) for s in range(S) if s not in ids}
                take(ga, sa.finish(ids))
                take(gb, sb.finish(ids))
                assert ga == gb
                model.finish(ids)
                check_model(sb, model, S)
                pre.final(gb)
                # the other channels' framing state untouched
                assert {s: (sb.pending_bits(s), sb.pending_payload(s)) for s in keep} == keep
                for s in ids:
                    streams[s] = streams[s][:prev[s]]
        take(ga, sa.finish())
        take(gb, sb.finish())
        assert ga == gb
        model.finish(list(range(S)))
        check_model(sb, model, S)
        pre.final(gb)
        c = sb.counters()
    return gb, model, c, pre


def framed_bit_lengths(model, settings):
    return {settings[s][0] for jobs in model.frame_jobs for s, *_ in jobs}


@pytest.mark.parametrize("mode", ["host", "device", "interleaved"])
def test_every_demodulator_family_twin_handles(mode):
    chans, settings, streams, (wants, dec) = demod_case()
    S, n = len(streams), len(streams[0])
    rng = np.random.default_rng(200 + ["host", "device", "interleaved"].index(mode))
    if mode == "interleaved":
        ends = [[c] * S for c in piece_cuts(n, rng)] + [[n] * S]
        modes = ["bytes", "tensor", "flat"]
    else:
        cuts = [(golden_cuts(n, rng) + [piece_cuts(n, rng)])[s % 6] for s in range(S)]
        _, bounds = schedule_pieces(streams, cuts)
        ends = [[b[min(i + 1, len(b) - 1)] for b in bounds] for i in range(max(len(b) - 1 for b in bounds))]
        modes = [mode]
    got, model, c, pre = twin_run(settings, list(streams), ends, modes)
    for s in range(S):
        check_final(got[s], wants[s], dec, s)
    # not vacuous: recordings at >= 10 bit lengths framed by k_stream_frame, and some ended before their gate closed.
    # From the device: open recordings whose terminator and decoded bytes pending_payload reported before they ended
    # (only k_stream_frame writes either); from the model: the bit lengths of its frame jobs
    gpu = {settings[s][0] for s in pre.gpu_framed}
    assert len(gpu) >= 10, sorted(gpu)
    framed = framed_bit_lengths(model, settings)
    assert len(framed) >= 10 and all(bit_frames(b) > 0 for b in framed), framed
    assert len(model.results) > 10 and pre.checked > 0 and pre.ended_early >= 1, (len(model.results), pre.checked, pre.ended_early)


def test_long_recording_decoded_progressively():
    chans, long_pay, final_push = long_frame_channels()
    settings = [(c["baud"], c["a0"], c["a1"], c["timeout"]) for c in chans]
    streams = [c["x"] for c in chans]
    wants, dec = oracle_calls(streams, settings)
    n = len(streams[0])
    ends = [[min(n, (i + 1) * 48000)] * 4 for i in range(-(-n // 48000))]
    got, model, _, pre = twin_run(settings, list(streams), ends, ["host", "device"])
    for s in range(4):
        check_final(got[s], wants[s], dec, s)
    rec = [c for c in got[0] if c[1]][-1]
    assert rec[4] == long_pay and (rec[3] - rec[2]) // 8 - 1 > 262144
    # it was framed over several pushes before it ended
    fj = [j for jobs in model.frame_jobs for j in jobs if j[0] == 0 and j[1][1] == rec[2] and not j[4]]
    assert len(fj) >= 3, len(fj)


def test_4096_channels_mixed_settings_partial_finishes():
    settings, new, plain = many_settings()
    S, piece, split = MANY_S, MANY_PIECE, 2 * MANY_PIECE
    fin = sorted(set(new) | set(plain))
    X = np.empty((S, piece * MANY_PUSHES), np.int16)
    for s in range(S):
        X[s] = many_channel(s, settings[s])
    first = [X[s, :split] if s in new or s in plain else X[s] for s in range(S)]
    second = [X[s, split:] for s in fin]
    set2 = [new.get(s, settings[s]) for s in fin]
    wants, dec = oracle_calls(first + second, settings + set2)
    idx = {s: S + i for i, s in enumerate(fin)}
    cur = list(range(S))
    cur_set = list(settings)
    cur_x = [first[s] for s in range(S)]
    model = PayloadPlan([(a0, a1, int(t * 48000)) for _, a0, a1, t in settings], [b for b, *_ in settings],
                        oracle_clock(cur_x, cur_set), oracle_framer(cur_x, cur_set))
    amps = [chunk_amps(x) for x in first + second]
    streams_got = {k: [] for k in range(len(wants))}
    got = [streams_got[k] for k in cur]
    modes = ["device", "tensor", "bytes", "device"]
    bounds = [0, piece // 2, split, split + piece, 2 * split]
    pend = {"compactions": False, "plane_compactions": False, "payload_compactions": False}
    with A.open_receive_streams(receivers(settings), [x[3] for x in settings], retain="payload") as st:
        for i in range(MANY_PUSHES):
            c0 = st.counters()
            pending = any(st.state(s)[1] >= 0 for s in range(S))
            take(got, push(st, [X[s, bounds[i]:bounds[i + 1]] for s in range(S)], modes[i]))
            model.push([bounds[i + 1] - bounds[i]] * S, [amps[k] for k in cur])
            c = st.counters()
            # (the sample arena compacts while recordings are pending; the plane and payload slots stay small in payload
            # mode, so those arenas compact when recordings first fill them, with their planes decided in that push)
            decided = any(st.pending_bits(s)[1] > 0 for s in range(S))
            for k in pend:
                pend[k] |= (pending if k == "compactions" else decided) and c[k] > c0[k]
            check_model(st, model, S)
            for s in range(0, S, 97):
                assert st.pending_payload(s)[:3] == model.pending_payload(s)[:3], s
            if i == 1:
                ids = sorted(new)
                others = [s for s in range(0, S, 13) if s not in fin]
                before = {s: st.pending_payload(s) for s in others}
                take(got, st.finish(ids, receivers([new[s] for s in ids]), [new[s][3] for s in ids]))
                take(got, st.finish(plain))
                model.finish(ids, [(new[s][1], new[s][2], int(new[s][3] * 48000)) for s in ids], [new[s][0] for s in ids])
                model.finish(plain)
                check_model(st, model, S)
                assert {s: st.pending_payload(s) for s in others} == before
                for s in fin:
                    cur[s], cur_set[s] = idx[s], new.get(s, settings[s])
                    cur_x[s] = second[fin.index(s)]
                    got[s] = streams_got[cur[s]]
        take(got, st.finish())
    assert all(pend.values()), pend
    for k, calls in streams_got.items():
        check_final(calls, wants[k], dec, k)


def carrier_channels(S=64, seed=9100):
    """S channels at 300 / 1200 / 2400 / 6000 baud: the modem's mark tone held (every window decides 1: no terminator),
    or a message whose first quiet window lies inside a loud chunk (a short gap between the message and the carrier)"""
    rng = np.random.default_rng(seed)
    settings, heads, blocks, kinds = [], [], [], []
    for s in range(S):
        b = [300, 1200, 2400, 6000][s % 4]
        tone = np.tile(O.tone("mark", b), b)                            # one second
        head = tone.copy()
        kind = s % 2
        if kind:
            pay = rng.integers(0, 256, 4, dtype=np.uint8).tobytes()
            fr = O.tx_frames(pay, b, 0.05)
            fr = fr[:len(fr) - 4800]                                    # no trailing silence
            gap = 3 * (48000 // b)                                      # a few quiet windows inside a loud chunk
            ln = -(-(1000 + len(fr) + gap) // 48000) * 48000
            head = np.tile(tone, ln // 48000)
            head[1000:1000 + len(fr)] = fr
            head[1000 + len(fr):1000 + len(fr) + gap] = 0
        settings.append((b, 18000, 14000, 5.0))
        heads.append(head)
        blocks.append(tone)
        kinds.append(kind)
    return settings, heads, blocks, kinds


def test_stuck_carrier_and_early_end_keep_constant_planes():
    """64 channels for 120 one-second device pushes: a one-tone carrier keeps a constant number of plane words and the
    arenas stay flat; a message ended by a quiet window inside a loud chunk is ended after the push that frames that
    window, decides no more windows, and its result equals the oracle's when the gate finally closes"""
    import torch
    settings, heads, blocks, kinds = carrier_channels()
    S, n_push = len(settings), 120
    secs = [len(h) // 48000 for h in heads]
    n_head = max(secs)
    d_head = torch.from_numpy(np.stack([np.concatenate([h, np.tile(b, n_head - k)]) for h, b, k in zip(heads, blocks, secs)])).cuda()
    d_block = torch.from_numpy(np.stack(blocks)).cuda()
    quiet = np.zeros(48000 * 2, np.int16)

    def host_stream(s):
        return np.concatenate([heads[s], np.tile(blocks[s], n_push - secs[s]), quiet])

    streams = [lambda s=s: host_stream(s) for s in range(S)]
    model = model_of(settings, streams)
    amps = [chunk_amps(host_stream(s)) for s in range(S)]
    rx, tmo = receivers(settings), [x[3] for x in settings]
    got = [[] for _ in range(S)]
    off = np.arange(S + 1, dtype=np.int64) * 48000
    words, nbytes, wins, ended_at = [], [], [[] for _ in range(S)], [None] * S
    with A.open_receive_streams(rx, tmo, retain="payload") as st:
        for i in range(n_push):
            piece = (d_head[:, i * 48000:(i + 1) * 48000] if i < n_head else d_block).contiguous().reshape(-1)
            take(got, st.push(piece, off))
            model.push([48000] * S, amps)
            nbytes.append(st.arena_bytes())
            words.append([model.plane_words(s) for s in range(S)])
            for s in range(S):
                wins[s].append(st.pending_bits(s)[1])
                if ended_at[s] is None and st.pending_payload(s)[2]:
                    ended_at[s] = i
            if i % 20 == 0:
                check_model(st, model, S)
        check_model(st, model, S)
        assert all(st.state(s)[1] >= 0 for s in range(S))
        take(got, st.push(torch.zeros(S * 96000, dtype=torch.int16, device="cuda"), off * 2))   # the gates close
        model.push([96000] * S, amps)
        check_model(st, model, S)
        take(got, st.finish())
    tone = [s for s in range(S) if not kinds[s]]
    msg = [s for s in range(S) if kinds[s]]
    for s in tone:                                                      # training phase for the whole run
        assert model.fs[s].phase == 0 or model.R[s] < 0
        # the words from the search point on: at most the windows of the gate's partial chunk, and one word before them
        bf = bit_frames(settings[s][0])
        assert max(w[s] for w in words[5:]) <= -(-CHUNK // bf) // 32 + 2, (s, max(w[s] for w in words[5:]))
    assert nbytes[-1] == nbytes[10], (nbytes[10], nbytes[-1])
    for s in msg:
        assert ended_at[s] is not None and ended_at[s] < 5, s
        assert len(set(wins[s][ended_at[s] + 1:])) == 1, s               # no window decided after it ended
        assert all(w[s] == 0 for w in words[ended_at[s]:]), s
    for s in range(S):
        wants, dec = oracle_calls([host_stream(s)], [settings[s]])
        check_final(got[s], wants[0], dec, 0)


def test_edge_cases_against_samples_mode_and_oracle():
    """bits mode's edge cases: a recording cut by finish before its clock is stored goes through the plan; 4800 baud;
    a clock stored in the push in which the recording ends; single frames around word boundaries; a finish in the
    middle of a recording, which drops the windows decided in its partial chunk"""
    settings, streams = edge_case()
    S, n = len(streams), len(streams[0])
    at = 2048 * 3
    ends = []
    e = [at + 2048 + 10, 4000, 30000, 2048, 2048, 2048, 20000, 2048]
    ends.append(list(e))
    e = [e[0], 20000, n, n, at + 4096 + 40 * 64 - 3, at + 4096 + 8 * 64 - 3, 26000, 8000]
    ends.append(list(e))
    for _ in range(6):
        e = [e[0], e[1], e[2], e[3], e[4] + 1, e[5] + 1, e[6], e[7]]
        ends.append(list(e))
    ends.append([e[0], n, n, n, n, n, e[6] + 3000, n])
    ends.append([n] * S)
    got, model, _, _ = twin_run(settings, list(streams), ends, ["host", "device"], finish_some={0: [0], 8: [6]})
    wants, dec = oracle_calls([streams[s][:ends[0][0]] if s == 0 else streams[s][:ends[8][6]] if s == 6 else streams[s]
                               for s in range(S)], settings)
    for s in range(S):
        calls = got[s][:len(wants[s])] if s in (0, 6) else got[s]
        check_final(calls, wants[s], dec, s)
    assert [c[6][0] for c in got[0] if c[1]] == [O.ST_NO_CLOCK]


def test_finish_drops_windows_decided_past_the_last_full_chunk():
    """a 6000-baud message still in its payload when the stream ends 1500 frames into a chunk: bits mode has decided
    plane words of that partial chunk, the finish cuts the recording at its last full chunk, and k_stream_frame frames
    it only up to that K"""
    rng = np.random.default_rng(8700)
    at, n = 3 * CHUNK + 100, 60000
    x = np.clip(np.round(rng.normal(0, 500, n)), -32768, 32767)
    fr = O.tx_frames(rng.integers(0, 256, 200, dtype=np.uint8).tobytes(), 6000, 0.1).astype(np.float64)
    x[at:at + len(fr)] += fr                                         # (32 k frames: still sending at the cut)
    x = np.clip(np.round(x), -32768, 32767).astype(np.int16)
    cut = 3 * CHUNK + 6 * CHUNK + 1500
    settings = [(6000, 18000, 14000, 2.0)]
    got, model, _, _ = twin_run(settings, [x[:cut]], [[cut]], ["device"])
    wants, dec = oracle_calls([x[:cut]], settings)
    check_final(got[0], wants[0], dec, 0)
    (_, _, a, b, _, _, r), = [c for c in got[0] if c[1]]
    K = windows_of(b - a, bit_frames(6000), r[1])
    decided = max(j[3] for jobs in model.jobs for j in jobs if j[0] == 0 and j[1][1] == a)
    assert (0, 0, a) in model.results and decided > K and r[0] == O.ST_OK, (decided, K, r[:4])
