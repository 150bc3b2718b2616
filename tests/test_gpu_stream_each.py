"""Stream handles whose channels have their own settings (open_receive_streams / open_transmit_streams,
afsk_rx_streams_create_each / _finish_some, afsk_tx_streams_create_each / _configure) on the GPU.  Each receive
channel must return exactly what a handle created with that channel's settings returns, over each of its
successive streams; each transmit channel must hold exactly save()'s frames of every message, with the settings
its channel had when the message was sent."""
import ctypes as C
import hashlib

import numpy as np
import pytest

import afskmodem_b200 as A
from afskmodem_b200 import _cabi
from conftest import gate_multi_stream, load_gate_multi_golden
from oracle import oracle as O
from test_gpu_stream_tx import CUTS, golden_groups
from test_gpu_streams import golden_cuts, schedule_pieces, sweep_streams
from test_stream_each_model import EachHandle
from test_stream_gate_model import chunk_amps, final_prefix
from test_stream_tx_model import random_payload

pytestmark = pytest.mark.gpu
CHUNK = 2048
A.LOG_LEVEL = 5
RX_BAUDS = [300, 600, 1200, 2400, 4000, 6000, 4800]
THRESHOLDS = [(18000, 14000), (14000, 11000), (9000, 8000)]
TIMEOUTS = [0, 0.1, 0.5, 2]


def lim_of(timeout_s):
    t = int(timeout_s * 48000)
    return 0 if t <= 0 else -(-t // CHUNK)


def to_device(pieces):
    import torch
    off = np.zeros(len(pieces) + 1, np.int64)
    np.cumsum([len(p) for p in pieces], out=off[1:])
    cat = np.concatenate(pieces) if off[-1] else np.zeros(0, np.int16)
    t = torch.empty(int(off[-1]) + 8, dtype=torch.int16, device="cuda")
    t[:len(cat)] = torch.from_numpy(cat.copy()).cuda()
    return t, off


def collect(got, ev):
    """appends (call, recorded, start, end, value, result) per event to got[stream]; a value that is an exception
    is kept as (type name, message) so that results compare by value"""
    vals = [(type(v).__name__, str(v)) if isinstance(v, Exception) else v for v in ev.values(string=False, errors="return")]
    k = 0
    for i in range(len(ev)):
        r = None
        if ev.recorded[i]:
            b = ev.batch
            r = (int(b.status[k]), int(b.clock[k]), int(b.train_end[k]), int(b.nbits[k]), b.payload(k))
            k += 1
        got[int(ev.stream[i])].append((int(ev.call[i]), bool(ev.recorded[i]), int(ev.start[i]), int(ev.end[i]), vals[i], r))


def drive_each(st, streams, cuts, amp_ends=None, lims=None, wants=None, device=False):
    """Pushes every channel's schedule together (the union of their pushes), then finish; with wants: after every
    push each channel's calls so far are exactly its oracle calls final within the prefix pushed, with its own
    lim and amp_end."""
    S = len(streams)
    got = [[] for _ in range(S)]
    pushes, bounds = schedule_pieces(streams, cuts)
    amps = [chunk_amps(x) for x in streams]
    for i, pieces in enumerate(pushes):
        collect(got, st.push(*to_device(pieces)) if device else st.push(pieces))
        if wants is not None:
            for s in range(S):
                pushed = bounds[s][min(i + 1, len(bounds[s]) - 1)]
                n = final_prefix(wants[s], amps[s], pushed // CHUNK, lims[s], amp_ends[s])
                assert [g[1:4] for g in got[s]] == wants[s][:n], (s, i)
                p, pend, ret = st.state(s)
                assert p == pushed and ret == pushed - (pend if pend >= 0 else pushed // CHUNK * CHUNK)
    collect(got, st.finish())
    return got


def check_oracle_values(x, calls, baud, amp_end):
    for call, rec, a, b, val, r in calls:
        if not rec:
            assert val == b""
            continue
        o = O.rx_decode(x[a:b], baud, amp_end)
        assert r == (o["status"], o["clock"], o["train_end"], o["nbits"], o["data"]), (call, baud)
        if o["status"] < 0:
            assert val == O.EXC_TEXT[o["status"]]
        else:
            assert val == o["data"]


def test_golden_cases_as_channels_of_one_handle():
    """Every gate_multi golden case cut five ways: 30 channels of one handle, each with its case's Receiver and
    timeout."""
    cases = load_gate_multi_golden()
    assert len(cases) == 6 and len({(g["baud"], g["amp_start"], g["amp_end"], g["timeout"]) for g in cases}) > 1
    streams, cuts, rxs, timeouts, wants, golden = [], [], [], [], [], []
    for g in cases:
        x = gate_multi_stream(g, O.tx_frames)
        rx = A.Receiver(g["baud"], g["amp_start"], g["amp_end"])
        want = O.listen_gate_multi(x, g["amp_start"], g["amp_end"], int(g["timeout"] * 48000))
        for c in golden_cuts(len(x), np.random.default_rng(len(x))):
            streams.append(x); cuts.append(c); rxs.append(rx); timeouts.append(g["timeout"])
            wants.append(want); golden.append((g, [bytes.fromhex(k["ret_hex"]) for k in g["calls"]]))
    assert len(streams) == 30
    with A.open_receive_streams(rxs, timeouts) as st:
        got = drive_each(st, streams, cuts, [g["amp_end"] for g, _ in golden], [lim_of(t) for t in timeouts], wants)
    whole = {}
    for s, calls in enumerate(got):
        g, gold = golden[s]
        assert [c[0] for c in calls] == list(range(len(calls)))
        assert [c[1:4] for c in calls] == wants[s], s
        vals = [c[4] for c in calls]
        assert vals[:len(gold)] == gold and len(vals) <= len(gold) + 1, s
        if g["name"] not in whole:
            whole[g["name"]] = rxs[s].receive_all(streams[s], g["timeout"], False, keep_timeouts=True)
        assert vals == whole[g["name"]], s


def test_uniform_list_equals_open_streams():
    rng = np.random.default_rng(1200)
    S, t = 64, 0.5
    streams = sweep_streams(rng, 1200, S)
    cuts = [sorted(int(c) for c in np.cumsum(rng.integers(0, 30000, size=len(x) // 10000 + 5)) if c < len(x)) for x in streams]
    rx = A.Receiver(1200, 18000, 14000)
    with A.open_receive_streams([rx] * S, t) as a, rx.open_streams(S, t) as b:
        ga, gb = drive_each(a, streams, cuts), drive_each(b, streams, cuts)
        assert [a.state(s) for s in range(S)] == [b.state(s) for s in range(S)]
        assert a.counters() == b.counters() and a.arena_bytes() == b.arena_bytes()
    assert ga == gb and sum(1 for c in ga for e in c if e[1]) >= S


def mixed_channels(rng, S):
    bauds = [RX_BAUDS[int(i)] for i in rng.integers(0, len(RX_BAUDS), S)]
    thr = [THRESHOLDS[int(i)] for i in rng.integers(0, len(THRESHOLDS), S)]
    tos = [TIMEOUTS[int(i)] for i in rng.integers(0, len(TIMEOUTS), S)]
    return bauds, thr, tos


@pytest.mark.parametrize("device", [False, True])
def test_mixed_sweep_equals_oracle_and_single_setting_handles(device):
    rng = np.random.default_rng(64 + device)
    S = 64
    bauds, thr, tos = mixed_channels(rng, S)
    assert {300, 4800, 6000} <= set(bauds) and len(set(thr)) == 3 and len(set(tos)) == 4
    streams = [sweep_streams(rng, b, 1)[0] for b in bauds]
    cuts = [sorted(int(c) for c in np.cumsum(rng.integers(0, 30000, size=len(x) // 10000 + 5)) if c < len(x)) for x in streams]
    rxs = [A.Receiver(b, a0, a1) for b, (a0, a1) in zip(bauds, thr)]
    wants = [O.listen_gate_multi(x, a0, a1, int(t * 48000)) for x, (a0, a1), t in zip(streams, thr, tos)]
    with A.open_receive_streams(rxs, tos) as st:
        got = drive_each(st, streams, cuts, [a1 for _, a1 in thr], [lim_of(t) for t in tos], wants, device=device)
        launches = st.counters()["launches"]
    n_rec = n_exc = 0
    for s in range(S):
        assert [c[1:4] for c in got[s]] == wants[s], s
        check_oracle_values(streams[s], got[s], bauds[s], thr[s][1])
        with rxs[s].open_streams(1, tos[s]) as one:
            assert drive_each(one, [streams[s]], [cuts[s]], device=device)[0] == got[s], s
        n_rec += sum(1 for c in got[s] if c[1])
        n_exc += sum(1 for c in got[s] if c[1] and isinstance(c[4], tuple))
    assert n_rec >= S and n_exc >= 1                                   # 4800 baud: the reference's exception
    assert launches > 0


def test_partial_finish_and_reopen():
    """Odd channels are finished in random subsets at random pushes, some reopened with other settings; even
    channels are never finished before the end and must match a control handle push for push."""
    rng = np.random.default_rng(77)
    S = 16
    bauds = [1200] * S
    thr = [THRESHOLDS[int(i)] for i in rng.integers(0, 3, S)]
    tos = [TIMEOUTS[int(i)] for i in rng.integers(0, 4, S)]
    src = [np.concatenate(sweep_streams(rng, 1200, 2) + sweep_streams(rng, 300, 1)) for _ in range(S)]
    rxs = [A.Receiver(b, a0, a1) for b, (a0, a1) in zip(bauds, thr)]
    model = EachHandle([(a0, a1, int(t * 48000)) for (a0, a1), t in zip(thr, tos)])
    stream_baud = [[b] for b in bauds]                                  # baud of each of a channel's streams
    got = [[[]] for _ in range(S)]                                      # per channel, per stream: events
    ctl_got = [[] for _ in range(S)]
    pos = [0] * S
    n_partial = n_reopen = 0
    with A.open_receive_streams(rxs, tos) as st, A.open_receive_streams(rxs, tos) as ctl:
        def take(ev, into):
            tmp = [[] for _ in range(S)]
            collect(tmp, ev)
            for s in range(S):
                into[s] += tmp[s]

        for step in range(40):
            if step % 4 == 3:
                ids = [int(s) for s in rng.permutation(range(1, S, 2))[:int(rng.integers(1, S // 2 + 1))]]
                new = None
                if rng.random() < 0.7:
                    new = []
                    for s in ids:
                        if rng.random() < 0.5:
                            new.append((A.Receiver(300, 14000, 11000), 0.5))
                        else:
                            a0, a1 = THRESHOLDS[int(rng.integers(0, 3))]
                            new.append((A.Receiver(1200, a0, a1), TIMEOUTS[int(rng.integers(0, 4))]))
                fin = st.finish(ids, [r for r, _ in new] if new else None, [t for _, t in new] if new else None)
                assert set(int(x) for x in fin.stream) <= set(ids)
                tmp = [[] for _ in range(S)]
                collect(tmp, fin)
                model.finish(ids, [(r._amp_start, r._amp_end, int(t * 48000)) for r, t in new] if new else None)
                for i, s in enumerate(ids):
                    got[s][-1] += tmp[s]
                    got[s].append([])
                    stream_baud[s].append(new[i][0]._baud if new else stream_baud[s][-1])
                    assert st.state(s) == (0, -1, 0)
                n_partial += 1
                n_reopen += bool(new)
            else:
                pieces = []
                for s in range(S):
                    n = 0 if rng.random() < 0.15 else int(rng.integers(0, 40000))
                    pieces.append(src[s][pos[s]:pos[s] + n])
                    pos[s] += len(pieces[-1])
                ev = st.push(pieces)
                tmp = [[] for _ in range(S)]
                collect(tmp, ev)
                for s in range(S):
                    got[s][-1] += tmp[s]
                take(ctl.push([p if s % 2 == 0 else p[:0] for s, p in enumerate(pieces)]), ctl_got)
                model.push(pieces)
                for s in range(0, S, 2):
                    assert st.state(s) == ctl.state(s) and [g for g in got[s][-1]] == ctl_got[s], s
                for s in range(S):
                    assert st.state(s) == model.state(s), s
        moved = st.counters()["moved_frames"]
        fin = st.finish()
        tmp = [[] for _ in range(S)]
        collect(tmp, fin)
        model.finish(list(range(S)))
        take(ctl.finish(), ctl_got)
        for s in range(S):
            got[s][-1] += tmp[s]
            assert st.state(s) == (0, -1, 0)
    assert n_partial >= 8 and n_reopen >= 3
    assert moved == model.ar.moved
    for s in range(S):
        assert len(got[s]) == len(model.ended[s]) == len(stream_baud[s]), s
        for k, ((a0, a1, t), x, want) in enumerate(model.ended[s]):
            assert [g[1:4] for g in got[s][k]] == want == O.listen_gate_multi(x, a0, a1, t), (s, k)
            assert [g[0] for g in got[s][k]] == list(range(len(want)))
            check_oracle_values(x, got[s][k], stream_baud[s][k], a1)
        if s % 2 == 0:
            assert got[s][0] == ctl_got[s]


def test_bad_finish_and_configure_arguments_leave_the_handles_unchanged():
    L = _cabi.lib()
    rng = np.random.default_rng(5)
    x = sweep_streams(rng, 1200, 1)[0]
    rx = A.Receiver(1200)
    n = C.c_int64(0)
    with rx.open_streams(3, 0.3) as st, rx.open_streams(3, 0.3) as ctl:
        h = len(x) // 2
        ga, gb = [[] for _ in range(3)], [[] for _ in range(3)]
        collect(ga, st.push([x[:h]] * 3))
        collect(gb, ctl.push([x[:h]] * 3))
        before = [st.state(s) for s in range(3)]
        b, a, t = np.array([1200, 300], np.int32), np.array([18000, 18000], np.int32), np.array([0, 0], np.int64)
        p32 = lambda v: _cabi.ptr(v, C.c_int32)                        # noqa: E731
        for ids in ([0, 0], [0, 3], [-1, 1]):
            ids = np.array(ids, np.int32)
            assert L.afsk_rx_streams_finish_some(st._h, 2, p32(ids), None, None, None, None, None, C.byref(n)) == _cabi.AFSK_E_ARG
            assert L.afsk_rx_streams_finish_some(st._h, 2, p32(ids), p32(b), p32(a), p32(a), _cabi.ptr(t, C.c_int64), None,
                                                 C.byref(n)) == _cabi.AFSK_E_ARG
        ids = np.array([0, 1], np.int32)
        assert L.afsk_rx_streams_finish_some(st._h, 4, p32(ids), None, None, None, None, None, C.byref(n)) == _cabi.AFSK_E_ARG
        assert L.afsk_rx_streams_finish_some(st._h, 2, p32(ids), p32(b), None, p32(a), _cabi.ptr(t, C.c_int64), None,
                                             C.byref(n)) == _cabi.AFSK_E_ARG            # settings partly given
        tn = np.array([0, -1], np.int64)
        assert L.afsk_rx_streams_finish_some(st._h, 2, p32(ids), p32(b), p32(a), p32(a), _cabi.ptr(tn, C.c_int64), None,
                                             C.byref(n)) == _cabi.AFSK_E_ARG            # negative timeout
        bb = np.array([1200, 9600], np.int32)
        assert L.afsk_rx_streams_finish_some(st._h, 2, p32(ids), p32(bb), p32(a), p32(a), _cabi.ptr(t, C.c_int64), None,
                                             C.byref(n)) == _cabi.AFSK_E_BAUD
        assert "channel 1" in L.afsk_last_error().decode()
        with pytest.raises(ValueError):
            st.finish([0, 1], [rx])                                        # one receiver for two channels
        assert [st.state(s) for s in range(3)] == before
        collect(ga, st.push([x[h:]] * 3))
        collect(gb, ctl.push([x[h:]] * 3))
        collect(ga, st.finish())
        collect(gb, ctl.finish())
        assert ga == gb and st.counters() == ctl.counters()
    want = O.listen_gate_multi(x, 18000, 14000, int(0.3 * 48000))
    assert [g[1:4] for g in ga[0]] == want

    tx = A.Transmitter(1200, 0.05)
    with tx.open_streams(3) as st:
        for ids in ([0, 0], [0, 3], [-1, 1]):
            ids = np.array(ids, np.int32)
            assert L.afsk_tx_streams_configure(st._h, 2, p32(ids), p32(b), _cabi.ptr(t, C.c_int64)) == _cabi.AFSK_E_ARG
        ids = np.array([0, 1], np.int32)
        assert L.afsk_tx_streams_configure(st._h, 4, p32(ids), p32(b), _cabi.ptr(t, C.c_int64)) == _cabi.AFSK_E_ARG
        assert L.afsk_tx_streams_configure(st._h, 2, p32(ids), p32(bb), _cabi.ptr(t, C.c_int64)) == _cabi.AFSK_E_BAUD
        with pytest.raises(ValueError):
            st.configure([0, 1], [tx])
        a0, b0 = st.send([0], [b"abc"])
        want = O.tx_frames(b"abc", 1200, 0.05)
        assert b0[0] - a0[0] == len(want)
        assert np.array_equal(st.pull(len(want) + 10)[0][:len(want)], want)


# ---------------------------------------------------------------- transmitter ----------------------

def test_tx_golden_cases_as_channels_of_one_handle():
    """Every constructible TX golden case, each with its own baud and training time, is one channel of one handle;
    under each pull cut the frames on the timeline are exactly the golden frames."""
    meta, _ = golden_groups()
    txs = [A.Transmitter(m["baud"], m["training_time"]) for m in meta]
    rng = np.random.default_rng(2)
    for cut in CUTS[1:] + [None]:
        sizes = [cut] if cut else CUTS + [int(rng.integers(0, 30000))]
        with A.open_transmit_streams(txs) as st:
            got, placed, i = [], [], 0
            order = rng.permutation(len(meta))
            for k in order:
                m = meta[k]
                a, b = st.send([int(k)], [bytes.fromhex(m["payload_hex"])])
                assert b[0] - a[0] == m["n"]
                placed.append((int(k), m, int(a[0]), int(b[0])))
                got.append(st.pull(sizes[i % len(sizes)]).copy())
                i += 1
            end = max(p[3] for p in placed)
            step = max(sizes[0] or 1, 48000)
            while sum(g.shape[1] for g in got) < end + 5:
                got.append(st.pull(step).copy())
            tl = np.concatenate(got, axis=1)
        covered = np.zeros(tl.shape, bool)
        for s, m, a, b in placed:
            assert hashlib.sha256(tl[s, a:b].astype("<i2").tobytes()).hexdigest() == m["sha256"], (m["name"], cut)
            covered[s, a:b] = True
        assert not tl[~covered].any()


TX_BAUDS = [300, 1200, 6000, 4800, 24000, 8000, 2400]


def tx_sweep_ops(rng, S, steps):
    ops = []
    for _ in range(steps):
        if rng.random() < 0.5:
            k = int(rng.integers(1, 3 * S // 2))
            ops.append(("send", [int(x) for x in rng.integers(0, S, k)], [random_payload(rng, 40) for _ in range(k)]))
        else:
            ops.append(("pull", int(rng.choice([1, 7, 9, 2047, 2048, 48000, int(rng.integers(0, 30000))]))))
    return ops


def test_tx_mixed_sweep_equals_single_setting_handles():
    rng = np.random.default_rng(640)
    S = 64
    cfg = [(TX_BAUDS[int(rng.integers(0, len(TX_BAUDS)))], float(rng.choice([0.0, 0.05, 0.1]))) for _ in range(S)]
    txs = [A.Transmitter(b, tt) for b, tt in cfg]
    ops = tx_sweep_ops(rng, S - 1, 40)                                 # channel S - 1 stays idle until ...
    P = sum(op[1] for op in ops if op[0] == "pull")
    ops += [("pull", 1 if P % 2 == 0 else 2), ("send", [S - 1], [b"odd start"]),     # ... a message starts on an odd frame
            ("send", list(range(S)), [b""] * S), ("pull", 30001)]
    ones = [t.open_streams(1) for t in txs]
    try:
        with A.open_transmit_streams(txs) as st:
            got, want, sent = [], [[] for _ in range(S)], []
            for op in ops:
                if op[0] == "send":
                    a, b = st.send(op[1], op[2])
                    for s, p, x, y in zip(op[1], op[2], a, b):
                        wa, wb = ones[s].send([0], [p])
                        assert (wa[0], wb[0]) == (x, y)
                        sent.append((s, p, int(x), int(y)))
                else:
                    got.append(st.pull(op[1]).copy())
                    for s in range(S):
                        want[s].append(ones[s].pull(op[1])[0].copy())
            got = np.concatenate(got, axis=1)
        assert np.array_equal(got, np.stack([np.concatenate(w) for w in want]))
    finally:
        for o in ones:
            o.close()
    assert {x % 2 for _, _, x, _ in sent} == {0, 1}
    for s, p, a, b in sent[::7]:                                        # and the oracle, on a sample of messages
        if b <= got.shape[1]:
            assert np.array_equal(got[s, a:b], O.tx_frames(p, *cfg[s])), (s, cfg[s])
    n_var = sum(1 for s, _, _, _ in sent if txs[s]._baud in (4800, 24000, 8000))
    assert n_var > 0 and len(sent) - n_var > 0


def test_tx_configure_applies_to_later_messages_only():
    tx_a, tx_b = A.Transmitter(1200, 0.1), A.Transmitter(300, 0.05)
    with A.open_transmit_streams([tx_a, tx_a]) as st:
        a1, b1 = st.send([0, 1], [b"first", b"one"])
        got = [st.pull(777).copy()]
        st.configure([0], tx_b)
        a2, b2 = st.send([0, 1], [b"second", b"two"])
        st.configure([0, 1], [A.Transmitter(4800, 0.0), A.Transmitter(24000, 0.2)])
        assert [t._baud for t in st.transmitters] == [4800, 24000]
        a3, b3 = st.send([1, 0], [b"three", b"third"])
        while sum(g.shape[1] for g in got) < max(b3.max(), b2.max()):
            got.append(st.pull(50000).copy())
    tl = np.concatenate(got, axis=1)
    msgs = [(0, b"first", 1200, 0.1, a1[0], b1[0]), (1, b"one", 1200, 0.1, a1[1], b1[1]),
            (0, b"second", 300, 0.05, a2[0], b2[0]), (1, b"two", 1200, 0.1, a2[1], b2[1]),
            (1, b"three", 24000, 0.2, a3[0], b3[0]), (0, b"third", 4800, 0.0, a3[1], b3[1])]
    for s, p, baud, tt, a, b in msgs:
        fr = O.tx_frames(p, baud, tt)
        assert b - a == len(fr), (p, baud)
        assert np.array_equal(tl[s, a:b], fr), (p, baud)
    assert a2[0] == b1[0] and a3[1] == b2[0]


def test_tx_loopback_into_a_mixed_receiver():
    import torch
    rng = np.random.default_rng(12)
    S, timeout = 12, 1.0
    bauds = [[300, 1200, 2400, 6000][s % 4] for s in range(S)]
    txs = [A.Transmitter(b, 0.5) for b in bauds]
    rxs = [A.Receiver(b) for b in bauds]
    sent, chunks = [], []
    got = [[] for _ in range(S)]
    with A.open_transmit_streams(txs) as st, A.open_receive_streams(rxs, timeout) as rs:
        for rnd in range(4):
            streams = [s for s in range(S) if rng.random() < 0.7]
            pays = [rng.integers(0, 256, int(rng.integers(1, 20)), dtype=np.uint8).tobytes() for _ in streams]
            a, b = st.send(streams, pays)
            sent += [(s, p, int(x), int(y)) for s, p, x, y in zip(streams, pays, a, b)]
            busy = max([y for _, _, _, y in sent] + [st.state(0)[0]])
            gap = int(rng.integers(30000, 60000))
            while st.state(0)[0] < busy + gap:
                n = int(rng.choice([2047, 4096, 9999, 48000]))
                t = torch.empty(S * n + 8, dtype=torch.int16, device="cuda")
                st.pull(n, out=t)
                chunks.append(t[:S * n].view(S, n).cpu().numpy())
                collect(got, rs.push(t, np.arange(S + 1, dtype=np.int64) * n))
        collect(got, rs.finish())
    tl = np.concatenate(chunks, axis=1)
    n_msgs = 0
    for s in range(S):
        x = tl[s]
        want = O.listen_gate_multi(x, 18000, 14000, int(timeout * 48000))
        assert [g[1:4] for g in got[s]] == want, s
        mine = [p for ss, p, _, _ in sent if ss == s]
        assert [g[4] for g in got[s] if g[1]] == mine, s
        n_msgs += len(mine)
    assert n_msgs >= S
