"""Streaming receiver (Receiver.open_streams / afsk_rx_streams_*) on the GPU: channels fed piece by
piece must return exactly what successive reference receive() calls return over the whole stream,
whatever the cut, and nothing before it is final."""
import numpy as np
import pytest

import afskmodem_b200 as A
from conftest import gate_multi_stream, load_gate_multi_golden
from oracle import oracle as O
from test_stream_gate_model import chunk_amps, final_prefix
from test_stream_retention_model import replay

pytestmark = pytest.mark.gpu
CHUNK = 2048
A.LOG_LEVEL = 5


def schedule_pieces(streams, cuts):
    """per push: the list of S pieces (cut lists per channel; every stream ends with its last push)"""
    bounds = [[0] + list(c) + [len(x)] for x, c in zip(streams, cuts)]
    n_push = max(len(b) - 1 for b in bounds)
    pushes = []
    for i in range(n_push):
        pushes.append([x[b[i]:b[i + 1]] if i + 1 < len(b) else x[:0] for x, b in zip(streams, bounds)])
    return pushes, bounds


def drive(st, streams, cuts, amp_end=None, lim=None, want=None, device=False, string=False):
    """Pushes every schedule, then finish.  Returns per channel [(call, recorded, start, end, value, result)].
    With want / lim / amp_end: checks after every push that each channel's calls so far are exactly
    its oracle calls that are final within the prefix pushed."""
    import torch
    S = len(streams)
    got = [[] for _ in range(S)]
    pushes, bounds = schedule_pieces(streams, cuts)
    amps = [chunk_amps(x) for x in streams]

    def take(ev):
        vals = ev.values(string=string, errors="return")
        k = 0
        for i in range(len(ev)):
            s = int(ev.stream[i])
            r = None
            if ev.recorded[i]:
                b = ev.batch
                r = (int(b.status[k]), int(b.clock[k]), int(b.train_end[k]), int(b.nbits[k]), b.payload(k))
                k += 1
            got[s].append((int(ev.call[i]), bool(ev.recorded[i]), int(ev.start[i]), int(ev.end[i]), vals[i], r))

    for i, pieces in enumerate(pushes):
        if device:
            off = np.zeros(S + 1, np.int64)
            np.cumsum([len(p) for p in pieces], out=off[1:])
            cat = np.concatenate(pieces) if off[-1] else np.zeros(0, np.int16)
            t = torch.empty(int(off[-1]) + 8, dtype=torch.int16, device="cuda")
            t[:len(cat)] = torch.from_numpy(cat.copy()).cuda()
            take(st.push(t, off))
        else:
            take(st.push(pieces))
        if want is not None:
            for s in range(S):
                pushed = bounds[s][min(i + 1, len(bounds[s]) - 1)]
                n = final_prefix(want[s], amps[s], pushed // CHUNK, lim, amp_end)
                assert [g[1:4] for g in got[s]] == want[s][:n], (s, i)
                p, pend, ret = st.state(s)
                assert p == pushed
                assert ret == pushed - (pend if pend >= 0 else pushed // CHUNK * CHUNK)
    take(st.finish())
    for s in range(S):
        assert [g[0] for g in got[s]] == list(range(len(got[s])))
    return got


def golden_cuts(n, rng):
    return [
        [],                                                                  # one push
        list(range(CHUNK, n, CHUNK)),                                        # 2048-frame pushes
        list(range(CHUNK - 1, n, CHUNK - 1)),                                # 2047-frame pushes
        [e for e in (i * 3000 + i % 8 for i in range(1, n // 3000 + 1)) if e < n],   # ends through all 8 16-byte phases
        sorted(int(c) for c in np.cumsum(rng.integers(0, 20001, size=n // 5000 + 10)) if c < n),   # random 0..20000
    ]


@pytest.mark.parametrize("g", load_gate_multi_golden(), ids=[g["name"] for g in load_gate_multi_golden()])
def test_golden_streams_cut_five_ways(g):
    x = gate_multi_stream(g, O.tx_frames)
    timeout = int(g["timeout"] * 48000)
    want = O.listen_gate_multi(x, g["amp_start"], g["amp_end"], timeout)
    golden = [bytes.fromhex(c["ret_hex"]) for c in g["calls"]]
    cuts = golden_cuts(len(x), np.random.default_rng(len(x)))
    lim = 0 if timeout <= 0 else -(-timeout // CHUNK)
    rx = A.Receiver(g["baud"], g["amp_start"], g["amp_end"])
    with rx.open_streams(len(cuts), g["timeout"]) as st:
        got = drive(st, [x] * len(cuts), cuts, g["amp_end"], lim, [want] * len(cuts))
    whole = rx.receive_all(x, g["timeout"], False, keep_timeouts=True)
    for s, calls in enumerate(got):
        assert [c[1:4] for c in calls] == want, s
        vals = [c[4] for c in calls]
        assert vals[:len(golden)] == golden and len(vals) <= len(golden) + 1, s
        assert vals == whole, s


def sweep_streams(rng, baud, n):
    streams = []
    for _ in range(n):
        parts = [np.zeros(int(rng.integers(0, 30000)), np.int16)]
        for _ in range(int(rng.integers(1, 4))):
            msg = rng.integers(0, 256, size=int(rng.integers(1, 12)), dtype=np.uint8).tobytes()
            tx = O.tx_frames(msg, baud, 0.1).astype(np.float64) * rng.uniform(0.6, 1.0)
            parts += [tx, np.zeros(int(rng.integers(2048, 20000)))]
        x = np.concatenate(parts)
        x = x + np.round(rng.normal(0, 2500, len(x)))
        streams.append(np.clip(x, -32768, 32767).astype(np.int16))
    return streams


@pytest.mark.parametrize("baud", [300, 1200, 6000, 4800])
def test_seeded_sweep_random_schedules(baud):
    rng = np.random.default_rng(baud)
    S, timeout_s = 64, 0.5
    streams = sweep_streams(rng, baud, S)
    timeout = int(timeout_s * 48000)
    lim = -(-timeout // CHUNK)
    want = [O.listen_gate_multi(x, 18000, 14000, timeout) for x in streams]
    cuts = [sorted(int(c) for c in np.cumsum(rng.integers(0, 30000, size=len(x) // 10000 + 5)) if c < len(x)) for x in streams]
    rx = A.Receiver(baud, 18000, 14000)
    with rx.open_streams(S, timeout_s) as st:
        got = drive(st, streams, cuts, 14000, lim, want)
    n_rec = 0
    for s, x in enumerate(streams):
        assert [c[1:4] for c in got[s]] == want[s], s
        for call, rec, a, b, val, r in got[s]:
            if not rec:
                assert val == b""
                continue
            o = O.rx_decode(x[a:b], baud, 14000)
            assert r == (o["status"], o["clock"], o["train_end"], o["nbits"], o["data"]), (s, call)
            if o["status"] < 0:
                assert isinstance(val, Exception)
            else:
                assert val == o["data"]
            n_rec += 1
    assert n_rec >= S


def test_long_recording_and_open_noise_channel():
    rng = np.random.default_rng(5)
    msg = rng.integers(0, 256, size=300, dtype=np.uint8).tobytes()
    tx = O.tx_frames(msg, 1200, 0.5)
    rec = np.concatenate([np.zeros(5000, np.int16), tx, np.zeros(12000, np.int16)])
    noise = (rng.choice([-1, 1], size=len(rec)) * 25000).astype(np.int16)         # opens at once, never quiet
    piece = 4096
    assert len(tx) // piece >= 40
    cuts = [list(range(piece, len(rec), piece))] * 2
    want = [O.listen_gate_multi(x, 18000, 14000, 48000) for x in (rec, noise)]
    rx = A.Receiver(1200, 18000, 14000)
    with rx.open_streams(2, 1.0) as st:
        pushes, _ = schedule_pieces([rec, noise], cuts)
        got = [[], []]
        for i, pieces in enumerate(pushes):
            ev = st.push(pieces)
            for j in range(len(ev)):
                got[int(ev.stream[j])].append((bool(ev.recorded[j]), int(ev.start[j]), int(ev.end[j])))
            retained = sum(st.state(s)[2] for s in range(2))
            pushed, pend, ret = st.state(1)
            assert pend == CHUNK and ret == pushed - CHUNK                          # the open noise recording
            assert st.arena_bytes() <= 16 * retained + 64 * piece + (1 << 20)
        fin = st.finish()
        assert [(bool(fin.recorded[j]), int(fin.start[j]), int(fin.end[j])) for j in range(len(fin))] == [want[1][-1]]
        o = O.rx_decode(noise[want[1][-1][1]:want[1][-1][2]], 1200, 14000)
        b = fin.batch
        assert (int(b.status[0]), int(b.clock[0]), int(b.train_end[0]), int(b.nbits[0]), b.payload(0)) == \
            (o["status"], o["clock"], o["train_end"], o["nbits"], o["data"])
    assert got[0] == want[0] and got[1] == want[1][:-1]
    assert rx.receive_all(rec, 1.0, False) == [msg]


def test_steady_state_pushes_do_not_grow_the_arena():
    rng = np.random.default_rng(9)
    S, piece = 8, 48000
    rx = A.Receiver(1200)
    with rx.open_streams(S, 1.0) as st:
        sizes = []
        for i in range(30):
            pieces = [np.round(rng.normal(0, 2000, piece)).astype(np.int16) for _ in range(S)]
            st.push(pieces)
            sizes.append(st.arena_bytes())
        assert len(set(sizes[10:])) == 1, sizes


def test_device_input_equals_host_input_and_bad_arguments():
    import torch
    rng = np.random.default_rng(11)
    streams = sweep_streams(rng, 1200, 6)
    cuts = [sorted(int(c) for c in np.cumsum(rng.integers(0, 25000, size=len(x) // 10000 + 4)) if c < len(x)) for x in streams]
    rx = A.Receiver(1200)
    with rx.open_streams(6, 0.3) as a, rx.open_streams(6, 0.3) as b:
        host = drive(a, streams, cuts)
        dev = drive(b, streams, cuts, device=True)
    assert host == dev
    assert sum(1 for c in host for e in c if e[1]) >= 6
    x = streams[0]
    with rx.open_streams(2, 0.3) as st:
        h0, h1 = len(x) // 2, len(x) // 3
        t = torch.from_numpy(np.concatenate([x[:h0], x[:h1], np.zeros(16, np.int16)])).cuda()
        off = np.array([0, h0, h0 + h1], np.int64)
        with pytest.raises(A.AfskError):
            st.push(t[1:], off)                                        # misaligned device pointer
        with pytest.raises(A.AfskError):
            st.push(t, np.array([0, 100, 50], np.int64))               # decreasing offsets
        with pytest.raises(ValueError):
            st.push(t, np.array([0, len(t) + 1, len(t) + 1], np.int64))
        assert st.state(0) == (0, -1, 0)
        got = []
        for ev in (st.push(t, off), st.push([x[h0:], x[h1:]]), st.finish()):
            got += [(int(ev.stream[i]), bool(ev.recorded[i]), int(ev.start[i]), int(ev.end[i])) for i in range(len(ev))]
    want = O.listen_gate_multi(x, 18000, 14000, int(0.3 * 48000))
    assert [g[1:] for g in got if g[0] == 0] == want and [g[1:] for g in got if g[0] == 1] == want


def test_finish_then_new_streams_like_a_fresh_receiver():
    rng = np.random.default_rng(13)
    first, second = sweep_streams(rng, 1200, 3), sweep_streams(rng, 1200, 3)
    cuts = lambda xs: [list(range(7000, len(x), 7000)) for x in xs]          # noqa: E731
    rx = A.Receiver(1200)
    with rx.open_streams(3, 0.4) as st:
        drive(st, first, cuts(first))
        reused = drive(st, second, cuts(second))
    with rx.open_streams(3, 0.4) as fresh:
        assert drive(fresh, second, cuts(second)) == reused


def test_retention_moves_match_the_model_and_stay_bounded():
    """A recording open for 60 one-second pushes beside three idle channels: the frames the receiver moves
    to keep retained samples are exactly what the CPU model of its retention policy moves, each of the
    recording's samples is moved at most three times, and the other channels' overflows never move it."""
    piece, pushes = 48000, 60
    rng = np.random.default_rng(17)
    levels = [25000, 0, 0, 0]
    streams = [(rng.choice([-1, 1], size=piece * pushes) * lv).astype(np.int16) for lv in levels]
    rx = A.Receiver(1200)
    with rx.open_streams(len(levels), 1.0) as st:
        for i in range(pushes):
            ev = st.push([x[i * piece:(i + 1) * piece] for x in streams])
            assert not ev.recorded.any()                              # idle channels time out, the open one never closes
        c = st.counters()
        assert st.state(0)[1:] == (CHUNK, piece * pushes - CHUNK)
    ar, total, _ = replay(levels, piece, pushes)
    assert (c["moved_frames"], c["compactions"]) == (ar.moved, ar.compactions)
    assert c["moved_frames"] <= 3 * piece * pushes and c["moved_frames"] <= total
    assert c["launches"] >= 3 * pushes
