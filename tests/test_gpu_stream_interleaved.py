"""Interleaved streaming (StreamReceiver.push_interleaved / StreamTransmitter.pull_interleaved,
afsk_rx_streams_push_interleaved / afsk_tx_streams_pull_interleaved) on the GPU.  A push of n interleaved frames must
be exactly the planar push of the S columns: the same events, values, state, counters and arena bytes, on twin
handles after every call.  A pull must be bitwise the transpose of the planar pull, and write nothing past n * S."""
import ctypes as C

import numpy as np
import pytest

import afskmodem_b200 as A
from afskmodem_b200 import _cabi
from conftest import gate_multi_stream, load_gate_multi_golden
from oracle import oracle as O
from test_gpu_stream_each import RX_BAUDS, THRESHOLDS, TIMEOUTS, collect, mixed_channels
from test_gpu_streams import sweep_streams
from test_stream_tx_model import random_payload

pytestmark = pytest.mark.gpu
A.LOG_LEVEL = 5
N_CHOICES = [0, 1, 7, 8, 9, 2047, 2048, 2049, 48000]


class Traffic:
    """Channel s's stream: a seeded transmission stream at its baud (a pool of a few per baud, each channel
    starting at its own offset), silence once it runs out."""

    def __init__(self, rng, bauds):
        self.pool = {b: sweep_streams(rng, b, 3) for b in sorted(set(bauds))}
        self.src = [(self.pool[b][int(rng.integers(0, 3))], int(rng.integers(0, 20000))) for b in bauds]

    def frames(self, s, a, n):
        x, o = self.src[s]
        out = np.zeros(n, np.int16)
        part = x[o + a:o + a + n]
        out[:len(part)] = part
        return out


def handles(bauds, thr, tos):
    rxs = [A.Receiver(b, a0, a1) for b, (a0, a1) in zip(bauds, thr)]
    return A.open_receive_streams(rxs, tos), A.open_receive_streams(rxs, tos)


def same_handles(p, q, S, got_p, got_q):
    assert got_p == got_q
    assert [p.state(s) for s in range(S)] == [q.state(s) for s in range(S)]
    assert p.counters() == q.counters() and p.arena_bytes() == q.arena_bytes()


def planar_input(X, kind):
    """the planar push of X's columns, from the same kind of memory as as_input(X, kind) (host or device: only host
    input grows the handle's staging buffer, which arena_bytes counts)"""
    import torch
    S = X.shape[1]
    if kind < 2:
        return ([X[:, s].copy() for s in range(S)],)
    t = torch.from_numpy(np.ascontiguousarray(X.T).reshape(-1)).cuda()
    return t, np.arange(S + 1, dtype=np.int64) * X.shape[0]


def as_input(X, kind):
    """X (n, S) int16 as numpy, bytes (what pyaudio's read returns) or a CUDA tensor (2-D or flat)"""
    import torch
    if kind == 0:
        return np.ascontiguousarray(X)
    if kind == 1:
        return X.tobytes()
    t = torch.from_numpy(np.ascontiguousarray(X)).cuda()
    return t if kind == 2 else t.reshape(-1)


@pytest.mark.parametrize("S", [1, 2, 3, 7, 8, 63, 64, 65, 4096])
def test_twin_receivers_planar_and_interleaved(S):
    rng = np.random.default_rng(9000 + S)
    bauds, thr, tos = mixed_channels(rng, S)
    traffic = Traffic(rng, bauds)
    steps = 14 if S >= 4096 else 40
    got_p, got_i = [[] for _ in range(S)], [[] for _ in range(S)]
    kinds, n_finish, n_rec, pos = set(), 0, 0, 0
    big = 0
    p, q = handles(bauds, thr, tos)
    with p, q:
        for step in range(steps):
            if step % 9 == 8:                                   # end some channels' streams, some with new settings
                ids = sorted(int(s) for s in rng.choice(S, size=max(1, S // 5), replace=False))
                if rng.random() < 0.5:
                    new = [A.Receiver(RX_BAUDS[int(rng.integers(0, 7))], *THRESHOLDS[int(rng.integers(0, 3))]) for _ in ids]
                    to = [TIMEOUTS[int(rng.integers(0, 4))] for _ in ids]
                    collect(got_p, p.finish(ids, receivers=new, timeout=to))
                    collect(got_i, q.finish(ids, receivers=new, timeout=to))
                else:
                    collect(got_p, p.finish(ids))
                    collect(got_i, q.finish(ids))
                n_finish += 1
                same_handles(p, q, S, got_p, got_i)
                continue
            n = int(rng.choice(N_CHOICES + [int(rng.integers(1, 6000))]))
            if n == 48000 and S >= 4096:
                if big:
                    n = 2049
                big += 1
            X = np.stack([traffic.frames(s, pos, n) for s in range(S)], axis=1) if n else np.zeros((0, S), np.int16)
            pos += n
            kind = step % 4
            kinds.add(kind)
            collect(got_p, p.push(*planar_input(X, kind)))
            collect(got_i, q.push_interleaved(as_input(X, kind)))
            same_handles(p, q, S, got_p, got_i)
        collect(got_p, p.finish())
        collect(got_i, q.finish())
        same_handles(p, q, S, got_p, got_i)
        n_rec = sum(1 for c in got_i for e in c if e[1])
    assert kinds == {0, 1, 2, 3} and n_finish >= 1
    assert n_rec >= 1                                           # (a 0 s timeout rarely opens a recording)


def test_gate_golden_streams_as_interleaved_channels():
    """The gate_multi golden streams as the channels of one handle fed only by interleaved pushes, each padded with
    silence to the common length pushed: every channel's calls are listen_gate_multi / receive_all of its padded
    stream."""
    cases = load_gate_multi_golden()
    xs = [gate_multi_stream(g, O.tx_frames) for g in cases]
    S = len(cases)
    rxs = [A.Receiver(g["baud"], g["amp_start"], g["amp_end"]) for g in cases]
    rng = np.random.default_rng(6)
    total = max(len(x) for x in xs) + 50000
    got = [[] for _ in range(S)]
    pos = 0
    with A.open_receive_streams(rxs, [g["timeout"] for g in cases]) as st:
        while pos < total:
            n = min(total - pos, int(rng.choice(N_CHOICES + [int(rng.integers(1, 20000))])))
            X = np.zeros((n, S), np.int16)
            for s, x in enumerate(xs):
                part = x[pos:pos + n]
                X[:len(part), s] = part
            collect(got, st.push_interleaved(as_input(X, int(rng.integers(0, 4)))))
            pos += n
        collect(got, st.finish())
    for s, (g, x) in enumerate(zip(cases, xs)):
        padded = np.zeros(total, np.int16)
        padded[:len(x)] = x
        want = O.listen_gate_multi(padded, g["amp_start"], g["amp_end"], int(g["timeout"] * 48000))
        assert [c[1:4] for c in got[s]] == want, g["name"]
        assert [c[4] for c in got[s]] == rxs[s].receive_all(padded, g["timeout"], False, keep_timeouts=True), g["name"]


TX_BAUDS = [1200, 4800, 24000, 300]


@pytest.mark.parametrize("S", [1, 3, 8, 64, 65, 4096])
def test_twin_transmitters_pull_interleaved_is_the_transpose(S):
    import torch
    rng = np.random.default_rng(700 + S)

    def txs(k):
        return [A.Transmitter(TX_BAUDS[int(i)], float(rng.choice([0.0, 0.05]))) for i in rng.integers(0, len(TX_BAUDS), k)]

    settings = txs(S)
    steps = 16 if S >= 4096 else 40
    pulled = big = 0
    with A.open_transmit_streams(settings) as a, A.open_transmit_streams(settings) as b:
        for step in range(steps):
            r = rng.random()
            if r < 0.4:
                k = int(rng.integers(1, 3 * S // 2 + 2))
                streams = [int(x) for x in rng.integers(0, S, k)]
                pays = [random_payload(rng, 20) for _ in range(k)]
                ra, rb = a.send(streams, pays), b.send(streams, pays)
                assert np.array_equal(ra[0], rb[0]) and np.array_equal(ra[1], rb[1])
            elif r < 0.47:
                ids = sorted(int(s) for s in rng.choice(S, size=max(1, S // 3), replace=False))
                new = txs(len(ids))
                a.configure(ids, new)
                b.configure(ids, new)
            else:
                n = int(rng.choice(N_CHOICES + [int(rng.integers(1, 30000))]))
                if n == 48000 and S >= 4096:
                    if big:
                        n = 2047
                    big += 1
                if step % 2:                                    # both twins pull into device memory, or both to the host
                    ta = torch.empty(n * S + 8, dtype=torch.int16, device="cuda")
                    want = a.pull(n, out=ta)[:n * S].view(S, n).cpu().numpy()
                    t = torch.full((n * S + 24,), 0x5A5A, dtype=torch.int16, device="cuda")
                    assert b.pull_interleaved(n, out=t) is t
                    h = t.cpu().numpy()
                    assert (h[n * S:] == 0x5A5A).all()                 # nothing past n * S
                    got = h[:n * S].reshape(n, S)
                else:
                    want = a.pull(n).copy()
                    got = b.pull_interleaved(n)
                    assert got.shape == (n, S) and got.dtype == np.int16
                assert np.array_equal(got, want.T), (step, n)
                pulled += n
                for s in range(S):
                    assert a.state(s) == b.state(s)
                assert a.counters() == b.counters() and a.arena_bytes() == b.arena_bytes()
    assert pulled > 0


def test_loopback_interleaved_on_mixed_settings():
    """pull_interleaved into a CUDA tensor, push_interleaved from it: every channel decodes exactly what it was sent."""
    import torch
    rng = np.random.default_rng(13)
    S, timeout = 11, 1.0
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
                chunks.append(st.pull_interleaved(n, out=t)[:n * S].view(n, S).cpu().numpy().T)
                collect(got, rs.push_interleaved(t[:n * S]))
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
    rng = np.random.default_rng(5)
    S = 5
    bauds, thr, tos = mixed_channels(rng, S)
    traffic = Traffic(rng, bauds)
    L = _cabi.lib()
    ev = C.c_int64(0)
    got_p, got_i = [[] for _ in range(S)], [[] for _ in range(S)]
    p, q = handles(bauds, thr, tos)
    txs = [A.Transmitter(b, 0.05) for b in [1200, 4800, 300, 24000, 1200]]
    with p, q, A.open_transmit_streams(txs) as ta, A.open_transmit_streams(txs) as tb:
        def check_rx():
            for s in range(S):
                assert p.state(s) == q.state(s)
            assert p.counters() == q.counters() and p.arena_bytes() == q.arena_bytes() and got_p == got_i

        def check_tx(n):
            assert np.array_equal(tb.pull_interleaved(n), ta.pull(n).T)
            assert [ta.state(s) for s in range(S)] == [tb.state(s) for s in range(S)] and ta.counters() == tb.counters()

        pos = 0
        for step in range(8):
            n = [2047, 9, 48000, 1, 2049, 7, 30000, 8][step]
            X = np.stack([traffic.frames(s, pos, n) for s in range(S)], axis=1)
            pos += n
            t = torch.from_numpy(X).cuda()
            with pytest.raises(ValueError):
                q.push_interleaved(X.tobytes()[:-2])                       # not whole frames
            with pytest.raises(ValueError):
                q.push_interleaved(X.astype(np.int32))                     # dtype
            with pytest.raises(ValueError):
                q.push_interleaved(np.asfortranarray(X) if n > 1 else X[:, ::2])   # not C-contiguous / shape
            with pytest.raises(ValueError):
                q.push_interleaved(X[:, :S - 1].copy())                    # shape
            with pytest.raises(ValueError):
                q.push_interleaved(t.to(torch.int32))                      # dtype
            with pytest.raises(ValueError):
                q.push_interleaved(torch.from_numpy(X))                    # device
            with pytest.raises(ValueError):
                q.push_interleaved(t.reshape(-1)[:-1])                     # length
            if n > 1:
                with pytest.raises(ValueError):
                    q.push_interleaved(t.t())                              # not contiguous
            flat = torch.zeros(n * S + 16, dtype=torch.int16, device="cuda")
            flat[8:8 + n * S] = t.reshape(-1)
            assert L.afsk_rx_streams_push_interleaved(q._h, C.c_void_p(flat.data_ptr() + 2), 1, n, None, C.byref(ev)) == _cabi.AFSK_E_ARG
            assert L.afsk_rx_streams_push_interleaved(q._h, C.c_void_p(t.data_ptr()), 1, -1, None, C.byref(ev)) == _cabi.AFSK_E_ARG
            assert L.afsk_rx_streams_push_interleaved(q._h, None, 0, n, None, C.byref(ev)) == _cabi.AFSK_E_ARG
            assert L.afsk_rx_streams_push_interleaved(q._h, C.c_void_p(t.data_ptr()), 1, 1 << 62, None, C.byref(ev)) == _cabi.AFSK_E_ARG
            assert L.afsk_rx_streams_push_interleaved(q._h, C.c_void_p(t.data_ptr()), 1, n, None, None) == _cabi.AFSK_E_ARG
            check_rx()
            collect(got_p, p.push(*planar_input(X, 2 if step % 2 else 1)))
            collect(got_i, q.push_interleaved(flat[8:8 + n * S] if step % 2 else X.tobytes()))
            check_rx()

            if step % 3 == 0:
                pays = [random_payload(rng, 12) for _ in range(S)]
                ta.send(list(range(S)), pays)
                tb.send(list(range(S)), pays)
            o = torch.zeros(n * S + 16, dtype=torch.int16, device="cuda")
            with pytest.raises(ValueError):
                tb.pull_interleaved(-1)
            with pytest.raises(ValueError):
                tb.pull_interleaved(n, out=o[:n * S - 1])                  # too small
            with pytest.raises(ValueError):
                tb.pull_interleaved(n, out=o.to(torch.int32))
            with pytest.raises(ValueError):
                tb.pull_interleaved(n, out=o.cpu())
            assert L.afsk_tx_streams_pull_interleaved(tb._h, n, C.c_void_p(o.data_ptr() + 2), 1, None) == _cabi.AFSK_E_ARG
            assert L.afsk_tx_streams_pull_interleaved(tb._h, -1, C.c_void_p(o.data_ptr()), 1, None) == _cabi.AFSK_E_ARG
            assert L.afsk_tx_streams_pull_interleaved(tb._h, n, None, 1, None) == _cabi.AFSK_E_ARG
            assert L.afsk_tx_streams_pull_interleaved(tb._h, 1 << 62, C.c_void_p(o.data_ptr()), 1, None) == _cabi.AFSK_E_ARG
            assert (o == 0).all()
            check_tx(n)
        collect(got_p, p.finish())
        collect(got_i, q.finish())
        check_rx()
    assert sum(1 for c in got_i for e in c if e[1]) >= 1
