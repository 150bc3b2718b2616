"""CPU checks that the traffic of test_gpu_stream_oracle.py covers what its tests claim: with the oracle and the CPU
models of the streaming handles (the resumable walk and the receive retention policy, the transmit arena with
per-channel settings), and no GPU."""
import numpy as np

from oracle import oracle as O
from test_gpu_stream_oracle import (DEMOD_BAUDS, K_FRAME_WARP_MAX_WINDOWS, MANY_Q, NO_MESSAGE, ArenaPlan, TxEachModel,
                                    demod_channels, long_frame_channels, many_plan, tx_golden_bauds, tx_plan)
from test_stream_each_model import EachHandle, random_settings
from test_stream_gate_model import chunk_amps, random_stream
from test_stream_tx_model import TimelineWindow, random_payload, timeline


def test_every_demod_baud_decodes_a_message_it_sent():
    chans = demod_channels()
    assert {c["baud"] for c in chans} == set(DEMOD_BAUDS) and {c["timeout"] for c in chans} >= {0, 0.1, 0.5, 2}
    assert len({(c["a0"], c["a1"]) for c in chans}) == 3 and len({len(c["x"]) for c in chans}) == 1
    for baud in DEMOD_BAUDS:
        ok = False
        for c in (c for c in chans if c["baud"] == baud):
            for rec, a, b in O.listen_gate_multi(c["x"], c["a0"], c["a1"], int(c["timeout"] * 48000)):
                if rec:
                    o = O.rx_decode(c["x"][a:b], baud, c["a1"])
                    if baud in NO_MESSAGE:
                        ok |= o["status"] == NO_MESSAGE[baud]
                    else:
                        ok |= o["status"] == O.ST_OK and o["data"] in c["pays"]
        assert ok, baud


def test_long_recording_needs_k_frame_and_ends_with_the_short_ones():
    chans, long_pay, push = long_frame_channels()            # (asserts that all four end in push `push`)
    assert [c["baud"] for c in chans] == [6000, 1200, 3000, 300]
    rec = [(a, b) for r, a, b in O.listen_gate_multi(chans[0]["x"], 18000, 14000, 48000) if r]
    a, b = rec[-1]
    assert (b - a) // 8 - 1 > K_FRAME_WARP_MAX_WINDOWS
    assert O.rx_decode(chans[0]["x"][a:b], 6000, 14000)["data"] == long_pay


def test_arena_plan_is_each_handle_over_chunk_amplitudes():
    rng = np.random.default_rng(3)
    S = 5
    settings = [random_settings(rng) for _ in range(S)]
    srcs = [random_stream(rng, 200, 0) for _ in range(S)]
    h, p = EachHandle(settings), ArenaPlan(settings)
    amps = [chunk_amps(x) for x in srcs]
    pos = [0] * S
    for step in range(30):
        if step == 12:
            assert h.finish([1, 3], [settings[0], settings[4]]) == p.finish([1, 3], [settings[0], settings[4]])
            for s in (1, 3):
                srcs[s], pos[s] = srcs[s][pos[s]:], 0
                amps[s] = chunk_amps(srcs[s])
            continue
        lens = [int(rng.integers(0, 30000)) for _ in range(S)]
        pieces = [x[q:q + n] for x, q, n in zip(srcs, pos, lens)]
        lens = [len(x) for x in pieces]
        pos = [q + n for q, n in zip(pos, lens)]
        assert h.push(pieces) == p.push(lens, amps)
        assert (h.ar.moved, h.ar.compactions, h.keep) == (p.ar.moved, p.ar.compactions, p.keep)


def test_4096_receive_channels_compact_with_pending_recordings_and_one_push_ends_2000_at_6000_baud():
    settings, plan, per_push = many_plan()
    assert len(settings) == 4096 and sum(1 for s in settings if s[0] == 6000) == MANY_Q
    assert len({s[1:3] for s in settings}) == 3 and len({s[3] for s in settings}) == 4
    assert plan.pending_compactions >= 1 and plan.ar.moved > 0
    assert any(c.get(6000, 0) > 2000 and sum(1 for b, k in c.items() if b != 6000 and k) >= 3 for c in per_push), per_push


def test_transmit_plan_compacts_with_unequal_tone_messages_queued():
    cfg, ops = tx_plan()
    assert {b for b, _ in cfg} == set(tx_golden_bauds()) and len(tx_golden_bauds()) == 15
    assert {4800, 960, 1600, 8000, 24000, 100} <= {b for b, _ in cfg}
    m = TxEachModel(cfg)
    sizes, odd = set(), False
    for op in ops:
        if op[0] == "send":
            a, _ = m.send(op[1], op[2])
            odd |= bool((a % 2).any())
        elif op[0] == "configure":
            m.configure(op[1], op[2])
        else:
            m.pull(op[1])
            sizes.add(op[1])
    assert sizes == {0, 1, 7, 8, 9, 2047, 2048, 48000} and odd
    assert any(op[0] == "send" and any(len(p) >= 2000 for p in op[2]) for op in ops)
    assert any(op[0] == "send" and any(len(p) == 0 for p in op[2]) for op in ops)
    assert sum(1 for v in m.var_across if any(x.end <= m.P for x in v)) >= 3


def test_timeline_window_equals_timeline():
    rng = np.random.default_rng(4)
    S, baud, tt = 3, 4800, 0.01
    m, win = TxEachModel([(baud, tt)] * S), TimelineWindow(S)
    sent, got = [], []
    for step in range(40):
        ids = [int(x) for x in rng.integers(0, S, 2)]
        pays = [random_payload(rng) for _ in ids]
        a, b = m.send(ids, pays)
        for s, p, x, y in zip(ids, pays, a, b):
            sent.append((s, p, int(x), int(y)))
            win.add(s, p, int(x), int(y), baud, tt)
        n = int(rng.choice([0, 1, 7, 2047, 9000]))
        got.append(win.window(m.P, n))
        m.pull(n)
    got = np.concatenate(got, axis=1)
    assert np.array_equal(got, timeline(sent, S, got.shape[1], baud, tt)) and got.any()
