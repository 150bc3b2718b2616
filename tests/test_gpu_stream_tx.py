"""Streaming transmitter (Transmitter.open_streams / afsk_tx_streams_*) on the GPU: every channel's timeline must hold
exactly save()'s frames of each message it was sent, at the frames send() returned, and silence everywhere else,
whatever the cut into pulls; and what it emits must decode through the streaming receiver."""
import ctypes as C
import hashlib
import json
import os

import numpy as np
import pytest

import afskmodem_b200 as A
from afskmodem_b200 import _cabi
from oracle import oracle as O
from test_stream_tx_model import TimelineWindow, TxModel, random_payload, timeline

pytestmark = pytest.mark.gpu
A.LOG_LEVEL = 5
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
CUTS = [0, 1, 3, 7, 8, 9, 2047, 2048, 48000]


def pull_all(st, sizes):
    return np.concatenate([st.pull(n).copy() for n in sizes], axis=1)


def golden_groups():
    meta = [m for m in json.load(open(os.path.join(GOLDEN, "tx_cases.json"))) if m["exc"] is None]
    groups = {}
    for m in meta:
        groups.setdefault((m["baud"], m["training_time"]), []).append(m)
    return meta, groups


def test_golden_cases_on_one_timeline_cut_every_way():
    meta, groups = golden_groups()
    assert len(meta) == 22 and {100, 4800, 8000, 24000, 12000} <= {m["baud"] for m in meta}
    rng = np.random.default_rng(1)
    checked = 0
    for (baud, tt), cases in groups.items():
        with A.Transmitter(baud, tt).open_streams(2) as st:
            got, placed, i = [], [], 0
            sizes = CUTS + [int(rng.integers(0, 30000))]
            for k, m in enumerate(cases):
                a, b = st.send([k % 2], [bytes.fromhex(m["payload_hex"])])
                assert b[0] - a[0] == m["n"]
                placed.append((k % 2, m, int(a[0]), int(b[0])))
                for _ in range(3):                              # a few pulls between sends: odd P at a send
                    got.append(st.pull(sizes[i % len(sizes)]).copy())
                    i += 1
            end = max(p[3] for p in placed)
            while sum(g.shape[1] for g in got) < end + 5:
                got.append(st.pull(sizes[i % len(sizes)] or 1).copy())
                i += 1
            tl = np.concatenate(got, axis=1)
            covered = np.zeros(tl.shape, bool)
            for s, m, a, b in placed:
                assert hashlib.sha256(tl[s, a:b].astype("<i2").tobytes()).hexdigest() == m["sha256"], m["name"]
                covered[s, a:b] = True
                checked += 1
            assert not tl[~covered].any()
    assert checked == 22


def run_schedule(st, model, ops, out=None):
    """drives the GPU transmitter and the CPU model with the same ops; checks send results and state after every
    pull; returns (sent, pulled frames)"""
    sent, got = [], []
    for op in ops:
        if op[0] == "send":
            a, b = st.send(op[1], op[2])
            wa, wb = model.send(op[1], op[2])
            assert np.array_equal(a, wa) and np.array_equal(b, wb)
            sent += [(s, p, int(x), int(y)) for s, p, x, y in zip(op[1], op[2], a, b)]
        else:
            got.append(st.pull(op[1]).copy())
            model.pull(op[1])
            for s in range(model.S):
                assert st.state(s) == model.state(s), (s, st.state(s), model.state(s))
    return sent, np.concatenate(got, axis=1)


def sweep_ops(rng, S, steps):
    ops = []
    for _ in range(steps):
        if rng.random() < 0.5:
            k = int(rng.integers(1, 3 * S // 2))
            streams = [int(x) for x in rng.integers(0, S, k)]
            ops.append(("send", streams, [random_payload(rng, 40) for _ in range(k)]))
        else:
            ops.append(("pull", int(rng.choice([1, 7, 9, 2047, 2048, 48000, int(rng.integers(0, 30000))]))))
    return ops


@pytest.mark.parametrize("baud", [300, 1200, 6000, 4800])
@pytest.mark.parametrize("tt", [0.0, 0.05])
def test_seeded_sweep_64_channels(baud, tt):
    rng = np.random.default_rng([baud, int(tt * 100)])
    S = 64
    model = TxModel(S, baud, tt, synth=False)
    ops = sweep_ops(rng, S, 40) + [("send", list(range(S)), [b""] * S), ("pull", 30001)]
    with A.Transmitter(baud, tt).open_streams(S) as st:
        sent, got = run_schedule(st, model, ops)
        c = st.counters()
    assert any(p == b"" for _, p, _, _ in sent) and any(a % 2 for _, _, a, _ in sent)
    assert np.array_equal(got, timeline(sent, S, got.shape[1], baud, tt))
    assert (c["moved_bytes"], c["compactions"]) == (model.moved, model.compactions)


def test_retention_counters_match_the_model():
    """Many small messages on 64 channels: the arena compacts several times, exactly as the CPU model of the
    retention policy does, and moves less than twice the bytes sent; every frame pulled, before and after each
    compaction, is the oracle's timeline (a payload or codeword start table moved incompletely would show)."""
    rng = np.random.default_rng(7)
    S = 64
    for baud in (1200, 4800):
        model = TxModel(S, baud, 0.05, synth=False)
        win = TimelineWindow(S)
        with A.Transmitter(baud, 0.05).open_streams(S) as st:
            for step in range(300):
                k = int(rng.integers(0, 40))
                streams = [int(x) for x in rng.integers(0, S, k)]
                pays = [random_payload(rng, 400) for _ in range(k)]
                a, b = st.send(streams, pays)
                wa, _ = model.send(streams, pays)
                assert np.array_equal(a, wa)
                for s, p, x, y in zip(streams, pays, a, b):
                    win.add(s, p, int(x), int(y), baud, 0.05)
                n = int(rng.integers(1, 30000))
                assert np.array_equal(st.pull(n), win.window(model.P, n)), (baud, step)
                model.pull(n)
            c = st.counters()
        assert model.compactions >= 3
        assert (c["moved_bytes"], c["compactions"]) == (model.moved, model.compactions)
        assert c["moved_bytes"] <= 2 * model.sent_bytes


def test_64kb_message_at_300_baud_over_many_pulls():
    rng = np.random.default_rng(3)
    msg = rng.integers(0, 256, 65536, dtype=np.uint8).tobytes()
    want = O.tx_frames(msg, 300, 0.5)
    with A.Transmitter(300, 0.5).open_streams(1) as st:
        a, b = st.send([0], [msg])
        assert (a[0], b[0]) == (0, len(want))
        pos, piece, pulls = 0, 960001, 0
        while pos < len(want):
            fr = st.pull(piece)[0]
            k = min(piece, len(want) - pos)
            assert np.array_equal(fr[:k], want[pos:pos + k]), pos
            assert not fr[k:].any()
            pos += piece
            pulls += 1
        assert pulls >= 100 and st.state(0) == (pos, len(want), 0)


def test_device_output_with_guards_equals_host_output():
    import torch
    rng = np.random.default_rng(5)
    S = 13
    ops = sweep_ops(rng, S, 30)
    tx = A.Transmitter(1200, 0.1)
    host, dev = [], []
    with tx.open_streams(S) as a, tx.open_streams(S) as b:
        for op in ops:
            if op[0] == "send":
                ra, rb = a.send(op[1], op[2]), b.send(op[1], op[2])
                assert all(np.array_equal(x, y) for x, y in zip(ra, rb))
                continue
            n = op[1]
            host.append(a.pull(n).copy())
            t = torch.full((S * n + 37,), 0x5A5A, dtype=torch.int16, device="cuda")
            assert b.pull(n, out=t) is t
            g = t.cpu().numpy()
            assert (g[S * n:] == 0x5A5A).all()                  # nothing past S * n is written
            dev.append(g[:S * n].reshape(S, n))
    assert np.array_equal(np.concatenate(host, axis=1), np.concatenate(dev, axis=1))
    assert np.concatenate(host, axis=1).any()


def test_loopback_into_the_streaming_receiver():
    """Pulled into a device tensor and pushed into Receiver.open_streams on the same device: the events and values
    are listen_gate_multi / receive_all of each channel's whole timeline, and the payloads are what was sent."""
    import torch
    rng = np.random.default_rng(11)
    S, baud, tt, timeout = 8, 1200, 0.1, 1.0
    tx, rx = A.Transmitter(baud, tt), A.Receiver(baud)
    model = TxModel(S, baud, tt, synth=False)
    sent, chunks = [], []
    with tx.open_streams(S) as st, rx.open_streams(S, timeout) as rs:
        got = [[] for _ in range(S)]

        def take(ev):
            vals = ev.values(string=False, errors="return")
            for i in range(len(ev)):
                got[int(ev.stream[i])].append((bool(ev.recorded[i]), int(ev.start[i]), int(ev.end[i]), vals[i]))

        for rnd in range(6):
            streams = [s for s in range(S) if rng.random() < 0.7]
            pays = [rng.integers(0, 256, int(rng.integers(1, 30)), dtype=np.uint8).tobytes() for _ in streams]
            a, b = st.send(streams, pays)
            model.send(streams, pays)
            sent += [(s, p, int(x), int(y)) for s, p, x, y in zip(streams, pays, a, b)]
            busy = max([y for _, _, _, y in sent] + [st.state(0)[0]])
            gap = int(rng.integers(30000, 60000))              # silence after the last message of the round
            while st.state(0)[0] < busy + gap:
                n = int(rng.choice([2047, 4096, 9999, 48000]))
                t = torch.empty(S * n + 8, dtype=torch.int16, device="cuda")
                st.pull(n, out=t)
                chunks.append(t[:S * n].view(S, n).cpu().numpy())
                take(rs.push(t, np.arange(S + 1, dtype=np.int64) * n))
        take(rs.finish())
    tl = np.concatenate(chunks, axis=1)
    assert np.array_equal(tl, timeline(sent, S, tl.shape[1], baud, tt))
    n_msgs = 0
    for s in range(S):
        x = tl[s]
        want = O.listen_gate_multi(x, 18000, 14000, int(timeout * 48000))
        assert [g[:3] for g in got[s]] == want, s
        assert [g[3] for g in got[s]] == rx.receive_all(x, timeout, False, keep_timeouts=True), s
        mine = [p for ss, p, _, _ in sent if ss == s]
        assert [g[3] for g in got[s] if g[0]] == mine, s       # noise-free, silent gaps: exactly what was sent
        n_msgs += len(mine)
    assert n_msgs >= S


def test_bad_arguments_leave_the_handle_usable():
    import torch
    L = _cabi.lib()
    tx = A.Transmitter(1200, 0.05)
    with tx.open_streams(3) as st:
        a, _ = st.send([1], [b"abc"])
        with pytest.raises(A.AfskError):
            st.send([3], [b"x"])                               # stream out of range
        with pytest.raises(A.AfskError):
            st.send([-1], [b"x"])
        assert st.state(1)[1:] == (len(O.tx_frames(b"abc", 1200, 0.05)), 1)
        t = torch.zeros(3 * 100 + 16, dtype=torch.int16, device="cuda")
        assert L.afsk_tx_streams_pull(st._h, 100, C.c_void_p(t.data_ptr() + 2), 1, None) == _cabi.AFSK_E_ARG   # misaligned
        assert L.afsk_tx_streams_pull(st._h, -1, C.c_void_p(t.data_ptr()), 1, None) == _cabi.AFSK_E_ARG
        assert L.afsk_tx_streams_pull(st._h, 1 << 62, C.c_void_p(t.data_ptr()), 1, None) == _cabi.AFSK_E_ARG  # S * n overflows
        off = np.array([0, 2, 1], np.int64)
        ids = np.array([0, 1], np.int32)
        z = np.zeros(2, np.int64)
        pay = np.zeros(2, np.uint8)
        assert L.afsk_tx_streams_send(st._h, 2, _cabi.ptr(ids, C.c_int32), _cabi.ptr(off, C.c_int64), _cabi.ptr(pay, C.c_uint8),
                                      _cabi.ptr(z, C.c_int64), _cabi.ptr(z, C.c_int64)) == _cabi.AFSK_E_ARG    # decreasing offsets
        with pytest.raises(ValueError):
            st.pull(5, out=t[:10])                             # too small
        assert st.state(0) == (0, 0, 0)
        want = O.tx_frames(b"abc", 1200, 0.05)
        fr = np.concatenate([st.pull(n)[1].copy() for n in (0, 5, len(want))])
        assert np.array_equal(fr[:len(want)], want) and not fr[len(want):].any()
        assert st.state(1) == (len(want) + 5, len(want), 0)
        assert st.counters()["launches"] == 2 and st.arena_bytes() > 0
    with pytest.raises(Exception, match="Invalid baud rate."):
        A.Transmitter(7)
