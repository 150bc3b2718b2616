"""Bits-mode retention (open_receive_streams(..., retain="bits")) against samples mode, the oracle and the CPU model
of its bookkeeping (test_stream_bits_model.BitsPlan): every demodulator family through host, device and interleaved
pushes; a recording framed by k_frame from its planes; 4096 channels with mixed settings and partial finishes;
config 4 (64 KB at 300 baud) looped back on 4096 channels; recordings that never close; and edge cases."""
import functools

import numpy as np
import pytest

import afskmodem_b200 as A
from afskmodem_b200 import _cabi
from oracle import oracle as O
from test_gpu_stream_oracle import (MANY_PIECE, MANY_PUSHES, MANY_S, THREADS, check_final, demod_case, long_frame_channels,
                                    many_channel, many_settings, oracle_calls, piece_cuts, push, receivers, take)
from test_gpu_streams import golden_cuts, schedule_pieces
from test_stream_bits_model import SYNC, BitsPlan, bit_frames
from test_stream_gate_model import CHUNK, chunk_amps

pytestmark = pytest.mark.gpu
A.LOG_LEVEL = 5


def oracle_clock(streams, settings):
    """clock(s, R) of the model: the oracle's clock of the 4096 frames from R of channel s's current stream"""
    def clock(s, R):
        x = streams[s]()[R:R + SYNC] if callable(streams[s]) else streams[s][R:R + SYNC]
        return int(O.rx_decode(x, settings[s][0], settings[s][2])["clock"])
    return clock


def model_of(settings, streams):
    return BitsPlan([(a0, a1, int(t * 48000)) for _, a0, a1, t in settings], [b for b, *_ in settings],
                    oracle_clock(streams, settings))


def check_model(st, model, S):
    for s in range(S):
        want_state, want_bits = model.state(s)
        assert st.state(s) == want_state, s
        assert st.pending_bits(s) == want_bits, s
    c = st.counters()
    assert (c["moved_frames"], c["compactions"]) == (model.ar.moved, model.ar.compactions)
    assert (c["moved_plane_words"], c["plane_compactions"]) == (model.pl.moved // 4, model.pl.compactions)


def twin_run(settings, streams, ends, modes, finish_some=None):
    """samples- and bits-mode handles fed the same pushes (ends[i][s]: frames of stream s after push i, modes in
    turn): equal events, results, payloads and values after every push and finish; the bits handle's state,
    pending_bits and counters equal the model's.  finish_some: {push index: channel ids finished after it}."""
    S = len(streams)
    rx, tmo = receivers(settings), [x[3] for x in settings]
    model = model_of(settings, streams)
    amps = [chunk_amps(x) for x in streams]
    ga, gb = [[] for _ in range(S)], [[] for _ in range(S)]
    prev = [0] * S
    with A.open_receive_streams(rx, tmo) as sa, A.open_receive_streams(rx, tmo, retain="bits") as sb:
        assert (sa.retain, sb.retain) == ("samples", "bits")
        for i, e in enumerate(ends):
            pieces = [x[p:q] for x, p, q in zip(streams, prev, e)]
            mode = modes[i % len(modes)]
            take(ga, push(sa, pieces, mode))
            take(gb, push(sb, pieces, mode))
            assert ga == gb, i
            model.push([len(x) for x in pieces], amps)
            check_model(sb, model, S)
            prev = e
            if finish_some and i in finish_some:
                ids = finish_some[i]
                bits = {s: sb.pending_bits(s) for s in range(S) if s not in ids}
                take(ga, sa.finish(ids))
                take(gb, sb.finish(ids))
                assert ga == gb
                model.finish(ids)
                check_model(sb, model, S)
                assert {s: sb.pending_bits(s) for s in bits} == bits        # the other channels' plane state untouched
                for s in ids:                                               # (those channels' streams end here)
                    streams[s] = streams[s][:prev[s]]
        take(ga, sa.finish())
        take(gb, sb.finish())
        assert ga == gb
        model.finish(list(range(S)))
        check_model(sb, model, S)
        c = sb.counters()
    return gb, model, c


@pytest.mark.parametrize("mode", ["host", "device", "interleaved"])
def test_every_demodulator_family_twin_handles(mode):
    chans, settings, streams, (wants, dec) = demod_case()
    S, n = len(streams), len(streams[0])
    rng = np.random.default_rng(100 + ["host", "device", "interleaved"].index(mode))
    if mode == "interleaved":
        ends = [[c] * S for c in piece_cuts(n, rng)] + [[n] * S]
        modes = ["bytes", "tensor", "flat"]
    else:
        cuts = [(golden_cuts(n, rng) + [piece_cuts(n, rng)])[s % 6] for s in range(S)]
        _, bounds = schedule_pieces(streams, cuts)
        ends = [[b[min(i + 1, len(b) - 1)] for b in bounds] for i in range(max(len(b) - 1 for b in bounds))]
        modes = [mode]
    got, model, c = twin_run(settings, list(streams), ends, modes)
    for s in range(S):
        check_final(got[s], wants[s], dec, s)
    assert model.windows_total > 0 and c["launches"] > 0
    # not vacuous: recordings at every bit length bits mode demodulates were framed from their planes
    framed = {settings[s][0] for jobs in model.jobs for s, *_ in jobs}
    assert len(framed) >= 10 and all(bit_frames(b) > 0 for b in framed), framed


def test_k_frame_recording_from_its_planes():
    chans, long_pay, final_push = long_frame_channels()
    settings = [(c["baud"], c["a0"], c["a1"], c["timeout"]) for c in chans]
    streams = [c["x"] for c in chans]
    wants, dec = oracle_calls(streams, settings)
    n = len(streams[0])
    ends = [[min(n, (i + 1) * 48000)] * 4 for i in range(-(-n // 48000))]
    got, model, _ = twin_run(settings, list(streams), ends, ["host", "device"])
    for s in range(4):
        check_final(got[s], wants[s], dec, s)
    rec = [c for c in got[0] if c[1]][-1]
    assert rec[4] == long_pay and (rec[3] - rec[2]) // 8 - 1 > 262144
    # the long recording's windows were decided over several pushes before it ended
    assert len([j for jobs in model.jobs for j in jobs if j[0] == 0 and j[1][1] == rec[2]]) >= 3


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
    model = BitsPlan([(a0, a1, int(t * 48000)) for _, a0, a1, t in settings], [b for b, *_ in settings],
                     lambda s, R: int(O.rx_decode(cur_x[s][R:R + SYNC], cur_set[s][0], cur_set[s][2])["clock"]))
    amps = [chunk_amps(x) for x in first + second]
    streams_got = {k: [] for k in range(len(wants))}
    got = [streams_got[k] for k in cur]
    modes = ["device", "tensor", "bytes", "device"]
    # a short first push, then a long one: every channel's tail outgrows its slot while recordings are pending, so the
    # sample arena compacts then (the split after push 2 stays at 2 s)
    bounds = [0, piece // 2, split, split + piece, 2 * split]
    pend_compact = pend_pcompact = False
    with A.open_receive_streams(receivers(settings), [x[3] for x in settings], retain="bits") as st:
        for i in range(MANY_PUSHES):
            c0 = st.counters()
            pending = any(st.state(s)[1] >= 0 for s in range(S))
            take(got, push(st, [X[s, bounds[i]:bounds[i + 1]] for s in range(S)], modes[i]))
            model.push([bounds[i + 1] - bounds[i]] * S, [amps[k] for k in cur])
            c = st.counters()
            pend_compact |= pending and c["compactions"] > c0["compactions"]
            pend_pcompact |= any(st.pending_bits(s)[1] > 0 for s in range(S)) and c["plane_compactions"] > c0["plane_compactions"]
            check_model(st, model, S)
            if i == 1:
                ids = sorted(new)
                take(got, st.finish(ids, receivers([new[s] for s in ids]), [new[s][3] for s in ids]))
                take(got, st.finish(plain))
                model.finish(ids, [(new[s][1], new[s][2], int(new[s][3] * 48000)) for s in ids], [new[s][0] for s in ids])
                model.finish(plain)
                check_model(st, model, S)
                for s in fin:
                    cur[s], cur_set[s] = idx[s], new.get(s, settings[s])
                    cur_x[s] = second[fin.index(s)]
                    got[s] = streams_got[cur[s]]
        take(got, st.finish())
        c = st.counters()
    assert c["compactions"] >= 1 and c["plane_compactions"] >= 1 and pend_compact and pend_pcompact, c
    assert model.windows_total > 10 ** 6
    for k, calls in streams_got.items():
        check_final(calls, wants[k], dec, k)


def test_config4_loopback_4096_channels():
    """64 KB payloads at 300 baud (146.8 M frames each) from a streaming transmitter into a bits-mode receiver, in
    1 s device pieces; samples mode would need about 1.2 TB here"""
    import torch
    S, baud, tt, n_bytes = 4096, 300, 0.1, 65536
    rng = np.random.default_rng(8400)
    pays = [rng.integers(0, 256, n_bytes, dtype=np.uint8).tobytes() for _ in range(S)]
    groups, lead = 8, 257                                   # start frames 0, 257, 514, ...: spread over chunk phases
    rx = A.Receiver(baud)
    bf = 48000 // baud
    with A.open_transmit_streams([A.Transmitter(baud, tt)] * S) as tx, rx.open_streams(S, 10.0, retain="bits") as st:
        starts = np.zeros(S, np.int64)
        ends = np.zeros(S, np.int64)
        buf = torch.empty(S * 48000, dtype=torch.int16, device="cuda")
        got = [[] for _ in range(S)]
        pushed = 0
        for g in range(groups):
            ids = list(range(g, S, groups))
            a, b = tx.send(ids, [pays[s] for s in ids])
            starts[ids], ends[ids] = a, b
            take(got, st.push(tx.pull(lead, out=buf), np.arange(S + 1, dtype=np.int64) * lead))
            pushed += lead
        total = int(ends.max()) + 2 * CHUNK
        # the arena policy with the planes decided by P frames (8 bytes per 32 windows from each channel's start): a plane
        # arena holds slots of at most twice their need plus two chunks (4096 samples = 1024 words) and half as much again
        # free, allocated with grow_device's 1.25; the other arena is the one of the compaction before, at most as large.
        # Sample arenas: tails of under 33 bit lengths plus the 1 s piece, by the same rule.  Staging and scratch: 256 MB.
        def bound(P):
            words = np.maximum(P - starts, 0) // bf // 32 + 1
            planes = int((2 * 1.25 * 1.5 * (2 * 8 * words + 2 * 2 * CHUNK * 2)).sum())
            tails = int(S * 2 * 1.25 * 1.5 * (2 * 2 * (33 * bf + 48000) + 2 * 2 * CHUNK))
            return planes + tails + (1 << 28)
        peak = 0
        while pushed < total:
            n = min(48000, total - pushed)
            take(got, st.push(tx.pull(n, out=buf), np.arange(S + 1, dtype=np.int64) * n))
            pushed += n
            peak = max(peak, st.arena_bytes())
            assert st.arena_bytes() <= bound(pushed), (pushed, st.arena_bytes(), bound(pushed))
        take(got, st.finish())
    # 4096 x 64 KB open at once: 0.94 GB of live planes; the rest are the sample slots that 1 s pieces need (393 MB a push)
    assert peak < 7 << 30, peak
    for s in range(S):
        recs = [c for c in got[s] if c[1]]
        assert len(recs) == 1, (s, len(recs))
        r = recs[0][6]
        assert r[0] == O.ST_OK and r[3] == 917504 and r[4] == pays[s], (s, r[:4])
    for s in (0, 1, 2, S // 2 + 3, S - 1):                 # the oracle on the same frames
        x = np.zeros(total, np.int16)
        fr = O.tx_frames(pays[s], baud, tt)
        x[starts[s]:starts[s] + len(fr)] = fr
        (_, rec, a, e), = [(c[0], c[1], c[2], c[3]) for c in got[s] if c[1]]
        want = O.listen_gate_multi(x, 18000, 14000, 480000)
        assert [w for w in want if w[0]] == [(True, a, e)], s
        o = O.rx_decode(x[a:e], baud, 14000)
        r = [c for c in got[s] if c[1]][0][6]
        assert r == (o["status"], o["clock"], o["train_end"], o["nbits"], o["data"]), s


def stuck_channels():
    """a few dozen channels at 24, 300, 1200 and 6000 baud (and others): a message, then without a quiet chunk a
    continuous full-scale carrier or loud noise.  -> (settings, first second per channel, the 1 s block repeated
    after it per channel)"""
    rng = np.random.default_rng(8500)
    bauds = [24, 300, 1200, 6000, 2400, 600, 150, 48] * 3
    settings, heads, blocks = [], [], []
    t = np.arange(48000)
    noise = np.clip(np.round(rng.normal(0, 20000, 48000)), -32768, 32767).astype(np.int16)
    for i, b in enumerate(bauds):
        pay = rng.integers(0, 256, 3, dtype=np.uint8).tobytes()
        fr = O.tx_frames(pay, b, 0.05)
        fr = fr[:len(fr) - 4800]                                     # no trailing silence
        if i % 2:
            blk = np.round(30000 * np.sin(2 * np.pi * 1200 * t / 48000)).astype(np.int16)
        else:
            blk = noise.copy()
        lead = int(rng.integers(0, 3000))
        ln = -(-(lead + len(fr)) // 48000) * 48000
        head = np.tile(blk, ln // 48000)
        head[lead:lead + len(fr)] = fr
        settings.append((b, 18000, 14000, 5.0))
        heads.append(head)
        blocks.append(blk)
    return settings, heads, blocks


def test_recordings_that_never_close():
    """the streams are made on the device, one second at a time (each channel's first seconds, then its 1 s block again
    and again); the host rebuilds one channel's stream at a time only for the model's chunk amplitudes and the oracle"""
    import torch
    settings, heads, blocks = stuck_channels()
    S, minutes = len(settings), 5
    secs = [len(h) // 48000 for h in heads]
    n_push = max(secs) + 60 * minutes
    n_head = max(secs)
    d_head = torch.from_numpy(np.stack([np.concatenate([h, np.tile(b, n_head - k)]) for h, b, k in zip(heads, blocks, secs)])).cuda()
    d_block = torch.from_numpy(np.stack(blocks)).cuda()

    def host_stream(s):
        return np.concatenate([heads[s], np.tile(blocks[s], n_push - secs[s])])

    rx, tmo = receivers(settings), [x[3] for x in settings]
    model = model_of(settings, [functools.partial(host_stream, s) for s in range(S)])
    amps = [chunk_amps(host_stream(s)) for s in range(S)]
    got = [[] for _ in range(S)]
    samples_bytes, bits_bytes = [], []
    off = np.arange(S + 1, dtype=np.int64) * 48000
    scratch = None
    with A.open_receive_streams(rx, tmo, retain="bits") as st, A.open_receive_streams(rx, tmo) as sa:
        for i in range(n_push):
            piece = (d_head[:, i * 48000:(i + 1) * 48000] if i < n_head else d_block).contiguous().reshape(-1)
            take(got, st.push(piece, off))
            model.push([48000] * S, amps)
            bits_bytes.append(st.arena_bytes())
            # every byte the arenas gained is the model's: sample slots of bounded tails, plane slots of 8 bytes per 32
            # windows decided, by the arena rule (twice the need plus two chunks per slot, 1.5 times the slots per arena,
            # grow_device's 1.25); the handle's other buffers stay as they were after the first push
            arenas = sum(model.ar.alloc) + sum(model.pl.alloc)
            if i == 1:
                scratch = bits_bytes[-1] - arenas
            if i >= 1:
                assert bits_bytes[-1] - arenas == scratch, (i, bits_bytes[-1], arenas, scratch)
            if i < 60:
                sa.push(piece, off)
                samples_bytes.append(sa.arena_bytes())
            if i % 30 == 0:
                check_model(st, model, S)
        assert all(st.state(s)[1] >= 0 and st.pending_bits(s)[1] > 0 for s in range(S))
        check_model(st, model, S)
        c = st.counters()
        take(got, st.finish())
        model.finish(list(range(S)))
    assert c["moved_plane_words"] > 0 and c["plane_compactions"] >= 1, c
    # samples mode grows with the recordings (96 KB per channel-second), bits mode by planes only
    assert samples_bytes[-1] - samples_bytes[10] > 40 * S * 96000 * 0.5
    assert bits_bytes[59] - bits_bytes[10] < (samples_bytes[59] - samples_bytes[10]) / 5
    for s in range(S):                                                  # the oracle over the whole stream
        wants, dec = oracle_calls([host_stream(s)], [settings[s]])
        check_final(got[s], wants[0], dec, 0)


def edge_case(seed=8600):
    """channels: 0 a recording cut by finish after one chunk (NO_CLOCK); 1, 2: 4800 baud spanning pushes, below and above
    4096 frames; 3: a clock that becomes ready in the push where the recording ends; 4, 5: 1-frame pieces across a plane
    word boundary; 6: finished alone in the middle of its recording; 7: a plain 1200-baud message"""
    rng = np.random.default_rng(seed)
    n = 60000
    chans = []
    for k, baud in enumerate([1200, 4800, 4800, 1200, 1200, 6000, 300, 1200]):
        x = np.clip(np.round(rng.normal(0, 500, n)), -32768, 32767)
        pay = rng.integers(0, 256, 4, dtype=np.uint8).tobytes()
        fr = O.tx_frames(pay, baud, 0.1).astype(np.float64)
        at = 2048 * 3 + 100 * k
        if k == 0:
            x[at:] = 30000 * np.sin(np.arange(n - at))
        elif k == 1:
            x[at:at + 3000] = fr[:3000]
        else:
            x[at:at + len(fr)] += fr[:n - at]
        chans.append(((baud, 18000, 14000, 2.0), np.clip(np.round(x), -32768, 32767).astype(np.int16)))
    return [c[0] for c in chans], [c[1] for c in chans]


def test_edge_cases_against_samples_mode_and_oracle():
    settings, streams = edge_case()
    S, n = len(streams), len(streams[0])
    at = 2048 * 3
    ends = []
    # channel 0 is cut by finish one chunk into its recording; 3's recording closes in the push in which its clock is
    # recovered (one big push); 4, 5: single frames around a word boundary of their pending recordings
    e = [at + 2048 + 10, 4000, 30000, 2048, 2048, 2048, 20000, 2048]
    ends.append(list(e))
    e = [e[0], 20000, n, n, at + 4096 + 40 * 64 - 3, at + 4096 + 8 * 64 - 3, 26000, 8000]
    ends.append(list(e))
    for _ in range(6):
        e = [e[0], e[1], e[2], e[3], e[4] + 1, e[5] + 1, e[6], e[7]]
        ends.append(list(e))
    ends.append([e[0], n, n, n, n, n, e[6] + 3000, n])
    ends.append([n] * S)
    got, model, _ = twin_run(settings, list(streams), ends, ["host", "device"], finish_some={0: [0], 8: [6]})
    wants, dec = oracle_calls([streams[s][:ends[0][0]] if s == 0 else streams[s][:ends[8][6]] if s == 6 else streams[s]
                               for s in range(S)], settings)
    for s in range(S):
        if s in (0, 6):
            calls = [c for c in got[s]][:len(wants[s])]
            check_final(calls, wants[s], dec, s)
        else:
            check_final(got[s], wants[s], dec, s)
    assert [c[6][0] for c in got[0] if c[1]] == [O.ST_NO_CLOCK]


def test_retention_is_chosen_before_the_first_push():
    rx = A.Receiver(1200)
    with rx.open_streams(2, 1.0, retain="bits") as st:
        st.push([np.zeros(100, np.int16)] * 2)
        assert _cabi.lib().afsk_rx_streams_set_retention(st._h, 0) == _cabi.AFSK_E_ARG
        assert _cabi.lib().afsk_rx_streams_set_retention(st._h, 7) == _cabi.AFSK_E_ARG
        ev = st.push([np.zeros(5000, np.int16)] * 2)              # still usable, still bits mode
        assert len(ev) == 0 and st.retain == "bits" and st.state(0)[0] == 5100
        st.finish()
    with pytest.raises(ValueError):
        rx.open_streams(1, 1.0, retain="frames")
