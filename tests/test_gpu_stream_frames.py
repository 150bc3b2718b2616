"""Interleaved frames as a column window of a wider card, in int16, int32 and float32 samples, on the GPU
(StreamReceiver.push_interleaved / StreamTransmitter.pull_interleaved with windows and dtype=,
afsk_rx_streams_push_frames / afsk_tx_streams_pull_frames).  A push of a window in any format must be exactly
push_interleaved of the converted, contiguous int16 frames, on twin handles after every call; a pull into a window
must write the converted pull_interleaved there and nothing else."""
import ctypes as C

import numpy as np
import pytest

import afskmodem_b200 as A
from afskmodem_b200 import _cabi
from oracle import oracle as O
from test_gpu_stream_each import RX_BAUDS, THRESHOLDS, TIMEOUTS, collect, mixed_channels
from test_gpu_stream_interleaved import TX_BAUDS, Traffic, handles
from test_stream_frames_model import rule_from_s16, rule_to_s16
from test_stream_tx_model import random_payload

pytestmark = pytest.mark.gpu
A.LOG_LEVEL = 5
FORMATS = [np.int16, np.int32, np.float32]


def in_format(x, dtype, rng):
    """int16 frames x as samples of dtype whose conversion is x, with what the rule discards filled in: the low 16
    bits of int32, a float offset under half a step; a few floats beyond the rule's edges (NaN, +-inf, |v| > 1),
    whose conversion is then no longer x (the twin is fed the converted frames)"""
    if dtype == np.int16:
        return x.copy()
    if dtype == np.int32:
        return (x.astype(np.int32) << 16) | rng.integers(0, 1 << 16, x.shape).astype(np.int32)
    f = ((x.astype(np.float64) + rng.uniform(-0.45, 0.45, x.shape)) / 32768).astype(np.float32)
    if f.size:
        k = rng.integers(0, f.size, max(1, f.size // 500))
        f.reshape(-1)[k] = rng.choice(np.array([np.nan, np.inf, -np.inf, 1.5, -1.25, 1.0, -1.0, 0.5 / 32768], np.float32), len(k))
    return f


def card_with_window(rng, X, dtype, extra, c0):
    """an (n, S + extra) card of dtype whose columns [c0, c0 + S) are X in that format, the others noise"""
    n, S = X.shape
    W = S + extra
    cardv = in_format(rng.integers(-32768, 32768, (n, W), dtype=np.int16), dtype, rng)
    cardv[:, c0:c0 + S] = in_format(X, dtype, rng)
    return cardv


def window_input(cardv, c0, S, kind):
    """the window columns [c0, c0 + S) of the card: a host numpy view, the packed bytes (pyaudio's read), or a view
    of a CUDA tensor"""
    import torch
    if kind == 0:
        return cardv[:, c0:c0 + S]
    if kind == 1:
        return np.ascontiguousarray(cardv[:, c0:c0 + S]).tobytes()
    return torch.from_numpy(cardv).cuda()[:, c0:c0 + S]


def int16_input(X, kind):
    """the twin's contiguous int16 frames, from the same kind of memory"""
    import torch
    if kind == 0:
        return np.ascontiguousarray(X)
    if kind == 1:
        return X.tobytes()
    return torch.from_numpy(np.ascontiguousarray(X)).cuda()


def same(p, q, S, got_p, got_q, arena):
    assert got_p == got_q
    assert [p.state(s) for s in range(S)] == [q.state(s) for s in range(S)]
    assert p.counters() == q.counters()
    if arena:
        assert p.arena_bytes() == q.arena_bytes()


@pytest.mark.parametrize("dtype", FORMATS, ids=["s16", "s32", "f32"])
@pytest.mark.parametrize("S", [1, 7, 64, 65, 4096])
def test_twin_receivers_window_and_converted_frames(S, dtype):
    rng = np.random.default_rng(31000 + 3 * S + FORMATS.index(dtype))
    bauds, thr, tos = mixed_channels(rng, S)
    traffic = Traffic(rng, bauds)
    steps = 10 if S >= 4096 else 27
    n_choices = [0, 1, 7, 9, 2047, 2049, 9000] + ([] if S >= 4096 else [48000])
    got_p, got_q = [[] for _ in range(S)], [[] for _ in range(S)]
    kinds, pos, n_finish = set(), 0, 0
    p, q = handles(bauds, thr, tos)
    with p, q:
        for step in range(steps):
            # device windows first: arena_bytes counts the staging of host input, which holds bytes of the format
            kind = 2 if step < steps // 3 else step % 2         # device window; host window, bytes
            if step % 9 == 8:
                ids = sorted(int(s) for s in rng.choice(S, size=max(1, S // 4), replace=False))
                new = [A.Receiver(RX_BAUDS[int(rng.integers(0, 7))], *THRESHOLDS[int(rng.integers(0, 3))]) for _ in ids]
                to = [TIMEOUTS[int(rng.integers(0, 4))] for _ in ids]
                collect(got_p, p.finish(ids, receivers=new, timeout=to))
                collect(got_q, q.finish(ids, receivers=new, timeout=to))
                n_finish += 1
                same(p, q, S, got_p, got_q, kinds == {2})
                continue
            n = int(rng.choice(n_choices))
            X = np.stack([traffic.frames(s, pos, n) for s in range(S)], axis=1) if n else np.zeros((0, S), np.int16)
            pos += n
            extra = int(rng.choice([0, 1, 7, 67]))
            c0 = int(rng.integers(0, extra + 1)) | (1 if extra else 0)   # an odd column where there is room
            c0 = min(c0, extra)
            cardv = card_with_window(rng, X, dtype, extra, c0)
            conv = rule_to_s16(np.ascontiguousarray(cardv[:, c0:c0 + S]))
            kinds.add(kind)
            collect(got_p, p.push_interleaved(int16_input(conv, kind)))
            collect(got_q, q.push_interleaved(window_input(cardv, c0, S, kind), dtype=dtype))
            same(p, q, S, got_p, got_q, kinds == {2} or dtype == np.int16)
        collect(got_p, p.finish())
        collect(got_q, q.finish())
        same(p, q, S, got_p, got_q, False)
    assert kinds == {0, 1, 2} and n_finish >= 1
    if S > 1:                                                   # (one channel's settings may never open a recording)
        assert sum(1 for c in got_q for e in c if e[1]) >= 1


@pytest.mark.parametrize("dtype", FORMATS, ids=["s16", "s32", "f32"])
def test_two_receivers_over_one_card_equal_one_over_all_columns(dtype):
    import torch
    rng = np.random.default_rng(77 + FORMATS.index(dtype))
    W, k = 37, 13
    bauds, thr, tos = mixed_channels(rng, W)
    traffic = Traffic(rng, bauds)
    rxs = [A.Receiver(b, a0, a1) for b, (a0, a1) in zip(bauds, thr)]
    got_all, got_a, got_b = [[] for _ in range(W)], [[] for _ in range(k)], [[] for _ in range(W - k)]
    pos = 0
    with A.open_receive_streams(rxs, tos) as full, A.open_receive_streams(rxs[:k], tos[:k]) as a, \
            A.open_receive_streams(rxs[k:], tos[k:]) as b:
        for step in range(16):
            n = int(rng.choice([1, 9, 2047, 2049, 30000]))
            X = np.stack([traffic.frames(s, pos, n) for s in range(W)], axis=1)
            pos += n
            cardv = in_format(X, dtype, rng)
            conv = rule_to_s16(cardv)
            dev = step % 2 == 1
            src = torch.from_numpy(cardv).cuda() if dev else cardv
            collect(got_all, full.push_interleaved(torch.from_numpy(conv).cuda() if dev else conv))
            collect(got_a, a.push_interleaved(src[:, :k], dtype=dtype))
            collect(got_b, b.push_interleaved(src[:, k:], dtype=dtype))
            assert got_all == got_a + got_b
            assert [full.state(s) for s in range(W)] == [a.state(s) for s in range(k)] + [b.state(s) for s in range(W - k)]
        collect(got_all, full.finish())
        collect(got_a, a.finish())
        collect(got_b, b.finish())
    assert got_all == got_a + got_b
    assert sum(1 for c in got_all for e in c if e[1]) >= 1


SENT16, SENT32, SENTF = 0x5A5A, 0x5A5A5A5A, np.float32(1234.5)


def sentinel(dtype):
    return {np.int16: SENT16, np.int32: SENT32, np.float32: SENTF}[dtype]


def same_bits(a, b):
    return np.array_equal(np.ascontiguousarray(a).view(np.uint8), np.ascontiguousarray(b).view(np.uint8))


@pytest.mark.parametrize("dtype", FORMATS, ids=["s16", "s32", "f32"])
@pytest.mark.parametrize("S", [1, 7, 64, 65, 4096])
def test_twin_transmitters_pull_into_guarded_windows(S, dtype):
    import torch
    rng = np.random.default_rng(900 + 3 * S + FORMATS.index(dtype))

    def txs(m):
        return [A.Transmitter(TX_BAUDS[int(i)], float(rng.choice([0.0, 0.05]))) for i in rng.integers(0, len(TX_BAUDS), m)]

    settings = txs(S)
    steps = 14 if S >= 4096 else 36
    n_choices = [0, 1, 7, 9, 127, 129, 2047, 9000] + ([] if S >= 4096 else [48000])
    pulled = 0
    with A.open_transmit_streams(settings) as a, A.open_transmit_streams(settings) as b:
        for step in range(steps):
            r = rng.random()
            if r < 0.35:
                m = int(rng.integers(1, 3 * S // 2 + 2))
                streams = [int(x) for x in rng.integers(0, S, m)]
                pays = [random_payload(rng, 20) for _ in range(m)]
                a.send(streams, pays)
                b.send(streams, pays)
                continue
            n = int(rng.choice(n_choices))
            want = rule_from_s16(a.pull_interleaved(n).copy(), dtype)
            extra = int(rng.choice([0, 1, 7, 67]))
            c0 = min(extra, int(rng.integers(0, extra + 1)) | 1)
            tail = int(rng.integers(1, 5))
            guard = np.full((n + tail, S + extra), sentinel(dtype), dtype)
            kind = step % 3
            if kind == 0:                                       # the default pinned view in the format
                got = b.pull_interleaved(n, dtype=dtype)
                assert got.shape == (n, S) and got.dtype == dtype
                assert same_bits(got, want), (step, n)
            elif kind == 1:                                     # a host window of a playback buffer
                out = guard.copy()
                assert b.pull_interleaved(n, out=out[:n, c0:c0 + S], dtype=dtype).base is not None
                expect = guard.copy()
                expect[:n, c0:c0 + S] = want
                assert same_bits(out, expect), (step, n)
            else:                                               # a device window
                t = torch.from_numpy(guard).cuda()
                w = t[:n, c0:c0 + S]
                assert b.pull_interleaved(n, out=w, dtype=dtype) is w
                expect = guard.copy()
                expect[:n, c0:c0 + S] = want
                assert same_bits(t.cpu().numpy(), expect), (step, n)
            pulled += n
            for s in range(S):
                assert a.state(s) == b.state(s)
            assert a.counters() == b.counters()
    assert pulled > 0


@pytest.mark.parametrize("dtype", FORMATS, ids=["s16", "s32", "f32"])
def test_two_transmitters_fill_disjoint_windows_of_one_tensor(dtype):
    import torch
    rng = np.random.default_rng(55 + FORMATS.index(dtype))
    W, k = 41, 17
    settings = [A.Transmitter(TX_BAUDS[int(i)], 0.05) for i in rng.integers(0, len(TX_BAUDS), W)]
    with A.open_transmit_streams(settings) as full, A.open_transmit_streams(settings[:k]) as a, \
            A.open_transmit_streams(settings[k:]) as b:
        for step in range(12):
            if step % 3 == 0:
                streams = [int(x) for x in rng.integers(0, W, 30)]
                pays = [random_payload(rng, 16) for _ in streams]
                full.send(streams, pays)
                for s, p in zip(streams, pays):
                    (a.send([s], [p]) if s < k else b.send([s - k], [p]))
            n = int(rng.choice([1, 7, 2047, 9000]))
            t = torch.full((n + 2, W + 3), float(sentinel(dtype)) if dtype == np.float32 else sentinel(dtype),
                           dtype=getattr(torch, np.dtype(dtype).name), device="cuda")
            ref = t.clone()
            full.pull_interleaved(n, out=ref[:n, 1:1 + W], dtype=dtype)
            a.pull_interleaved(n, out=t[:n, 1:1 + k], dtype=dtype)
            b.pull_interleaved(n, out=t[:n, 1 + k:1 + W], dtype=dtype)
            assert same_bits(t.cpu().numpy(), ref.cpu().numpy()), step


@pytest.mark.parametrize("dtype", [np.float32, np.int32], ids=["f32", "s32"])
def test_device_loopback_in_the_format_on_mixed_settings(dtype):
    """pull_interleaved into a window of a wider device card in the format, push_interleaved of that window: every
    channel decodes exactly what it was sent."""
    import torch
    rng = np.random.default_rng(17 + (dtype == np.int32))
    S, timeout, extra, c0 = 11, 1.0, 5, 3
    bauds = [[300, 1200, 2400, 6000][s % 4] for s in range(S)]
    txs = [A.Transmitter(b, 0.5) for b in bauds]
    rxs = [A.Receiver(b) for b in bauds]
    sent, chunks = [], []
    got = [[] for _ in range(S)]
    tdt = getattr(torch, np.dtype(dtype).name)
    with A.open_transmit_streams(txs) as st, A.open_receive_streams(rxs, timeout) as rs:
        for rnd in range(4):
            streams = [s for s in range(S) if rng.random() < 0.7]
            pays = [rng.integers(0, 256, int(rng.integers(1, 20)), dtype=np.uint8).tobytes() for _ in streams]
            x, y = st.send(streams, pays)
            sent += [(s, p, int(u), int(v)) for s, p, u, v in zip(streams, pays, x, y)]
            busy = max([v for _, _, _, v in sent] + [st.state(0)[0]])
            gap = int(rng.integers(30000, 60000))
            while st.state(0)[0] < busy + gap:
                n = int(rng.choice([2047, 4096, 9999, 48000]))
                cardt = torch.zeros((n, S + extra), dtype=tdt, device="cuda")
                w = st.pull_interleaved(n, out=cardt[:, c0:c0 + S], dtype=dtype)
                chunks.append(rule_to_s16(w.cpu().numpy()).T)
                collect(got, rs.push_interleaved(w, dtype=dtype))
        collect(got, rs.finish())
    tl = np.concatenate(chunks, axis=1)
    n_msgs = 0
    for s in range(S):
        want = O.listen_gate_multi(tl[s], 18000, 14000, int(timeout * 48000))
        assert [g[1:4] for g in got[s]] == want, s
        mine = [p for ss, p, _, _ in sent if ss == s]
        assert [g[4] for g in got[s] if g[1]] == mine, s
        n_msgs += len(mine)
    assert n_msgs >= S


def test_bad_arguments_leave_both_handles_usable():
    import torch
    rng = np.random.default_rng(8)
    S = 5
    bauds, thr, tos = mixed_channels(rng, S)
    traffic = Traffic(rng, bauds)
    L = _cabi.lib()
    ev = C.c_int64(0)
    got_p, got_q = [[] for _ in range(S)], [[] for _ in range(S)]
    p, q = handles(bauds, thr, tos)
    txs = [A.Transmitter(b, 0.05) for b in [1200, 4800, 300, 24000, 1200]]
    with p, q, A.open_transmit_streams(txs) as ta, A.open_transmit_streams(txs) as tb:
        pos = 0
        for step in range(6):
            n = [2047, 9, 48000, 1, 2049, 7][step]
            X = np.stack([traffic.frames(s, pos, n) for s in range(S)], axis=1)
            pos += n
            cardv = card_with_window(rng, X, np.float32, 3, 1)
            t = torch.from_numpy(cardv).cuda()
            ptr = t.data_ptr() + 4
            for fmt, ptr_, nf, pitch in [(3, ptr, n, 8), (-1, ptr, n, 8), (_cabi.SAMPLE_F32, ptr, n, S - 1),
                                         (_cabi.SAMPLE_F32, ptr + 2, n, 8), (_cabi.SAMPLE_S32, ptr + 1, n, 8),
                                         (_cabi.SAMPLE_S16, ptr + 1, n, 8), (_cabi.SAMPLE_F32, None, n, 8),
                                         (_cabi.SAMPLE_F32, ptr, -1, 8), (_cabi.SAMPLE_F32, ptr, 1 << 60, 1 << 20),
                                         (_cabi.SAMPLE_F32, ptr, (1 << 38), 8)]:
                assert L.afsk_rx_streams_push_frames(q._h, C.c_void_p(ptr_) if ptr_ else None, fmt, 1, nf, pitch, None,
                                                     C.byref(ev)) == _cabi.AFSK_E_ARG, (fmt, nf, pitch)
                assert L.afsk_tx_streams_pull_frames(tb._h, nf, C.c_void_p(ptr_) if ptr_ else None, fmt, 1, pitch,
                                                     None) == _cabi.AFSK_E_ARG, (fmt, nf, pitch)
            assert L.afsk_rx_streams_push_frames(q._h, C.c_void_p(ptr), _cabi.SAMPLE_F32, 1, n, 8, None, None) == _cabi.AFSK_E_ARG
            with pytest.raises(ValueError):
                q.push_interleaved(cardv[:, 1:1 + S])                      # float32 without dtype=
            with pytest.raises(ValueError):
                q.push_interleaved(cardv[:, 1:1 + S], dtype=np.int32)      # dtype mismatch
            with pytest.raises(ValueError):
                q.push_interleaved(cardv[:, 1:1 + S], dtype=np.float64)    # unknown format
            with pytest.raises(ValueError):
                q.push_interleaved(t[:, 1:1 + S:2] if S > 2 else t.t(), dtype=np.float32)   # columns not of unit stride
            if n > 1:
                with pytest.raises(ValueError):
                    q.push_interleaved(cardv[::-1, 1:1 + S], dtype=np.float32)             # negative row pitch
            with pytest.raises(ValueError):
                q.push_interleaved(cardv[:, 1:1 + S].tobytes()[:-4], dtype=np.float32)      # not whole frames
            o = torch.zeros((n, S + 3), dtype=torch.float32, device="cuda")
            with pytest.raises(ValueError):
                tb.pull_interleaved(n, out=o[:, 1:1 + S])                  # float32 without dtype=
            with pytest.raises(ValueError):
                tb.pull_interleaved(n, out=o[:, 1:1 + S:2] if S > 2 else o.t(), dtype=np.float32)
            with pytest.raises(ValueError):
                tb.pull_interleaved(n, out=np.zeros((n, S), np.float32)[::-1] if n > 1 else np.zeros((n + 1, S), np.float32),
                                    dtype=np.float32)
            with pytest.raises(ValueError):
                tb.pull_interleaved(n, dtype="int8")
            assert (o == 0).all()
            collect(got_p, p.push_interleaved(rule_to_s16(np.ascontiguousarray(cardv[:, 1:1 + S]))))
            collect(got_q, q.push_interleaved(t[:, 1:1 + S], dtype=np.float32))
            assert got_p == got_q and [p.state(s) for s in range(S)] == [q.state(s) for s in range(S)]
            if step % 3 == 0:
                pays = [random_payload(rng, 12) for _ in range(S)]
                ta.send(list(range(S)), pays)
                tb.send(list(range(S)), pays)
            want = rule_from_s16(ta.pull_interleaved(n).copy(), np.float32)
            assert same_bits(tb.pull_interleaved(n, out=o[:, 2:2 + S], dtype=np.float32).cpu().numpy(), want)
        collect(got_p, p.finish())
        collect(got_q, q.finish())
        assert got_p == got_q


def test_float_rounding_decides_the_gate_at_its_threshold():
    """Chunks whose mean |x| lands on the gate's threshold only by the float rule's rounding: 18000.6 / 32768 is
    18001 (> amp_start: a recording opens), 18000.5 / 32768 is 18000 (round half to even: none opens), -18000.6 /
    32768 is -18001.  The gate's calls are listen_gate_multi's over the converted stream."""
    import torch
    S, timeout = 3, 0.5
    lv = np.array([18000.6, 18000.5, -18000.6])
    x = np.zeros((2048 * 2 + 48000, S), np.float32)
    x[2048:4096] = (lv / 32768).astype(np.float32)
    conv = rule_to_s16(x)
    assert (conv[2048, :] == [18001, 18000, -18001]).all()
    got = [[] for _ in range(S)]
    with A.open_receive_streams([A.Receiver(1200, 18000, 14000)] * S, timeout) as rs:
        t = torch.from_numpy(x).cuda()
        collect(got, rs.push_interleaved(t, dtype=np.float32))
        collect(got, rs.finish())
    opened = []
    for s in range(S):
        want = O.listen_gate_multi(conv[:, s], 18000, 14000, int(timeout * 48000))
        assert [g[1:4] for g in got[s]] == want, s
        opened.append(any(g[1] for g in got[s]))
    assert opened == [True, False, True]


@pytest.mark.parametrize("dtype", FORMATS, ids=["s16", "s32", "f32"])
def test_host_window_of_a_wider_card_through_the_c_abi(dtype):
    """afsk_rx_streams_push_frames given a host window with row_pitch > S (the library copies it row by row into its
    staging buffer; the Python wrapper packs host windows itself and never passes one), against a twin fed the
    converted contiguous int16 frames."""
    rng = np.random.default_rng(400 + FORMATS.index(dtype))
    S = 23
    bauds, thr, tos = mixed_channels(rng, S)
    traffic = Traffic(rng, bauds)
    L = _cabi.lib()
    got_p, got_q = [[] for _ in range(S)], [[] for _ in range(S)]
    pos = 0
    p, q = handles(bauds, thr, tos)
    with p, q:
        for step in range(10):
            n = int(rng.choice([1, 7, 2047, 2049, 30000]))
            X = np.stack([traffic.frames(s, pos, n) for s in range(S)], axis=1)
            pos += n
            extra, c0 = [(1, 1), (7, 3), (67, 5), (67, 66)][step % 4]
            cardv = card_with_window(rng, X, dtype, extra, c0)
            win = cardv[:, c0:c0 + S]
            ev = C.c_int64(0)
            fmt = {np.int16: _cabi.SAMPLE_S16, np.int32: _cabi.SAMPLE_S32, np.float32: _cabi.SAMPLE_F32}[dtype]
            assert L.afsk_rx_streams_push_frames(q._h, C.c_void_p(win.ctypes.data), fmt, 0, n, S + extra, None,
                                                 C.byref(ev)) == _cabi.AFSK_OK
            collect(got_q, q._events(ev.value))
            collect(got_p, p.push_interleaved(rule_to_s16(np.ascontiguousarray(win))))
            same(p, q, S, got_p, got_q, dtype == np.int16)
        collect(got_p, p.finish())
        collect(got_q, q.finish())
        assert got_p == got_q
    assert sum(1 for c in got_q for e in c if e[1]) >= 1


def test_one_channel_int16_device_frames_inside_a_vector():
    """One channel of contiguous int16 device frames that start inside a 16-byte vector (the k_stream_copy route with an
    offset source), against a twin fed the same frames from the host."""
    import torch
    rng = np.random.default_rng(12)
    bauds, thr, tos = [1200], [(18000, 14000)], [0.5]
    traffic = Traffic(rng, bauds)
    got_p, got_q = [[]], [[]]
    pos = 0
    p, q = handles(bauds, thr, tos)
    with p, q:
        for step in range(12):
            n = int(rng.choice([1, 7, 9, 2047, 30000]))
            x = traffic.frames(0, pos, n)
            pos += n
            off = 1 + step % 7                                  # 2 to 14 bytes into the vector
            t = torch.zeros(n + 16, dtype=torch.int16, device="cuda")
            t[off:off + n] = torch.from_numpy(x).cuda()
            assert (t[off:].data_ptr() & 15) != 0
            collect(got_q, q.push_interleaved(t[off:off + n]))
            collect(got_p, p.push_interleaved(x.copy()))
            assert got_p == got_q and p.state(0) == q.state(0) and p.counters() == q.counters()
        collect(got_p, p.finish())
        collect(got_q, q.finish())
        assert got_p == got_q
