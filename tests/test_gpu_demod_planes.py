"""GPU (-m gpu): every demodulated window against the plain reference of tests/test_demod_planes_model.py, in every
demodulator layout and in the streaming receiver.

The end-to-end results (status, clock, train_end, nbits, payload) hide most demodulator errors: a wrong window in the
alternating training sequence, after the first quiet window or in a capture that ends in "No data." changes nothing,
and Hamming(7,4) absorbs a wrong payload bit.  Here the bit and quiet planes themselves are compared, window by window,
over the crafted batch of demod_batch (tie windows of every class, quiet edges, limiter-edge soup; every baud of
DEMOD_BAUDS) and over the open recordings of a streaming receiver after every push."""
import functools
import os

import numpy as np
import pytest

import afskmodem_b200 as A
from afskmodem_b200 import _cabi
from oracle import oracle as O
from test_demod_planes_model import (CLASSES, N_CLASS, SOUP, SYNC, batch_starts, bit_frames, class_window, demod_batch,
                                     edge_classes, ref_planes, tie_classes, window_classes)
from test_gpu_stream_oracle import check_final, demod_channels, oracle_calls, piece_cuts, receivers, take

pytestmark = pytest.mark.gpu
A.LOG_LEVEL = 5
THREADS = os.cpu_count() or 1
OPT_FUSED, OPT_GROUP_STREAMS = 3, 5                      # AFSK_OPT_* of afsk_b200.h
SWITCHES = ("AFSK_NO_PAD", "AFSK_NO_ROT", "AFSK_NO_LONG_SHIFT", "AFSK_DEMOD_NSUB", "AFSK_DEMOD_STAGES", "AFSK_PAD_WARPS",
            "AFSK_L2_HINT", "AFSK_FUSED", "AFSK_GROUP_STREAMS", "AFSK_DEMOD_TPW_LOG2", "AFSK_CLOCK_KERNEL", "AFSK_FRAME_KERNEL")
PAD_BAUDS = (1500, 750, 375)                                  # 32 / 64 / 128 frames: the padded layout


def _switches(monkeypatch, env):
    for k in SWITCHES:
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)


@functools.lru_cache(maxsize=1)
def batch_case():
    """the crafted batch, the oracle's result of every capture, and the reference planes and window classes of every
    capture with a clock"""
    caps, bauds, thrs, clocks = demod_batch()
    samples = np.concatenate(caps)
    starts = batch_starts(caps)
    lens = np.array([len(x) for x in caps], np.int64)
    datas, res = O.rx_decode_batch(samples, np.append(starts, len(samples)), bauds, thrs, threads=THREADS)
    want = [(r.status, r.clock, r.train_end, r.nbits, r.nbytes, d) for r, d in zip(res, datas)]
    ref, cls = {}, {}
    for i, (x, b, thr, clk) in enumerate(zip(caps, bauds, thrs, clocks)):
        if clk >= 0:
            assert want[i][1] == clk, i                        # crafted to the oracle's clock
            ref[i] = ref_planes(x, b, clk, thr)
            cls[i] = window_classes(x, b, clk, thr)
    return samples, starts, lens, np.array(bauds, np.int32), np.array(thrs, np.int64), want, ref, cls


def _launches(s) -> int:
    import ctypes as C
    n = C.c_int(0)
    _cabi.check(_cabi.lib().afsk_rx_plan_launches(s.plan, C.byref(n)))
    return n.value


def _session(sel, opts=()):
    samples, starts, lens, bauds, thrs = batch_case()[:5]
    s = A.RxSession(starts[sel], bauds[sel], thrs[sel].astype(np.int32), lengths=lens[sel])
    for o, v in opts:
        _cabi.check(_cabi.lib().afsk_rx_plan_set_option(s.plan, o, v))
    s.upload(samples)
    return s


def _check_decode(s, sel, layout):
    """results equal the oracle's; every window of every capture with a clock equals the reference (windows past the
    last one in its pair are 0).  -> window classes per bit length over the compared planes"""
    want, ref, cls = batch_case()[5:]
    s.run()
    b = s.download()
    seen = {}
    for j, i in enumerate(sel):
        got = (int(b.status[j]), int(b.clock[j]), int(b.train_end[j]), int(b.nbits[j]), int(b.nbytes[j]), b.payload(j))
        assert got == want[i], (layout, i, got[:5], want[i][:5])
        if i not in ref:
            continue
        bits, quiet = s.planes(j)
        rb, rq = ref[i]
        K = len(rb)
        assert len(bits) >= K, (layout, i)
        for name, g, r in (("bits", bits, rb), ("quiet", quiet, rq)):
            bad = np.flatnonzero(g[:K] != r)
            assert len(bad) == 0, (layout, i, int(batch_case()[3][i]), name, K, bad[:8].tolist())
            assert not g[K:-(-K // 32) * 32].any(), (layout, i, name, "windows past the last one")
        acc = seen.setdefault(bit_frames(int(batch_case()[3][i])), dict.fromkeys(CLASSES, 0))
        for c, v in cls[i].items():
            acc[c] += v
    return seen


def _assert_not_vacuous(seen, layout):
    assert seen, layout
    for bf, cnt in seen.items():
        for c in tie_classes(bf) + ["E0", "E1"]:
            assert cnt[c] >= N_CLASS, (layout, bf, c, cnt)


LAYOUTS = {
    "default": ({}, (), ()),
    "no_pad": ({"AFSK_NO_PAD": "1"}, (), ()),                  # 1500 / 750 / 375 baud through k_demod, rotated order
    "no_pad_no_rot": ({"AFSK_NO_PAD": "1", "AFSK_NO_ROT": "1"}, (), ()),
    "no_long_shift": ({"AFSK_NO_LONG_SHIFT": "1"}, (), ()),   # 800 / 480 / 400 / 240 baud through k_demod
    "nsub1": ({"AFSK_DEMOD_NSUB": "1"}, (), ()),
    # three sub-tiles make 480 / 240 baud stages of ~307 KB: refused (test_layouts_that_do_not_fit_are_refused)
    "nsub3": ({"AFSK_DEMOD_NSUB": "3"}, (), (480, 240)),
    "stages2": ({"AFSK_DEMOD_STAGES": "2"}, (), ()),
    # four 70 KB stages of the padded layout do not fit a CTA: refused
    "stages4": ({"AFSK_DEMOD_STAGES": "4"}, (), PAD_BAUDS),
    "pad_warps2": ({"AFSK_PAD_WARPS": "2"}, (), ()),
    "pad_warps3": ({"AFSK_PAD_WARPS": "3"}, (), ()),
    "pad_warps4": ({"AFSK_PAD_WARPS": "4"}, (), ()),
    "pad_warps5": ({"AFSK_PAD_WARPS": "5"}, (), ()),
    "l2_hint0": ({"AFSK_L2_HINT": "0"}, (), ()),
    "l2_hint1": ({"AFSK_L2_HINT": "1"}, (), ()),
    "groups_in_turn": ({}, ((OPT_GROUP_STREAMS, 0),), ()),
}


@pytest.mark.parametrize("layout", list(LAYOUTS))
def test_every_window_of_a_mixed_batch_in_every_layout(monkeypatch, layout):
    env, opts, leave_out = LAYOUTS[layout]
    _switches(monkeypatch, env)
    bauds = batch_case()[3]
    sel = np.array([i for i in range(len(bauds)) if int(bauds[i]) not in leave_out])
    s = _session(sel, opts)
    try:
        seen = _check_decode(s, sel, layout)
    finally:
        s.close()
    _assert_not_vacuous(seen, layout)
    assert {bit_frames(b) for b in set(bauds[sel].tolist()) if bit_frames(b) % 4 == 0} == set(seen), layout


@pytest.mark.parametrize("level", [1, 2])
def test_fused_schedules_decide_every_window(monkeypatch, level):
    """AFSK_OPT_FUSED 1 / 2 over the bauds whose groups the fused schedule takes (bit lengths up to 185 frames outside
    the padded layout, and what fits the auxiliary warps' shared memory: asked of the library one baud at a time)"""
    _switches(monkeypatch, {})
    bauds = batch_case()[3]
    ref = batch_case()[6]
    fusable = set()
    for b in sorted({int(x) for x in bauds}):
        i = next(i for i in ref if int(bauds[i]) == b) if any(int(bauds[i]) == b for i in ref) else None
        if i is None or bit_frames(b) > 185 or b in PAD_BAUDS:
            continue
        s = _session(np.array([i]), ((OPT_FUSED, 1),))
        if _launches(s) == 2:                                  # one demodulator launch with its clocks, then k_frame
            fusable.add(b)
        s.close()
    assert {1200, 6000, 2400} <= fusable, sorted(fusable)
    sel = np.array([i for i in range(len(bauds)) if i not in ref or int(bauds[i]) in fusable])
    s = _session(sel, ((OPT_FUSED, level),))
    try:
        groups = len({bit_frames(int(bauds[i])) for i in sel if i in ref})
        assert _launches(s) == groups + 1 + (level == 1), (level, _launches(s))   # + k_preset (spacers, 4800 baud)
        seen = _check_decode(s, sel, f"fused{level}")
    finally:
        s.close()
    _assert_not_vacuous(seen, f"fused{level}")


@pytest.mark.parametrize("env,baud", [({"AFSK_DEMOD_NSUB": "3"}, 480), ({"AFSK_DEMOD_NSUB": "3"}, 240),
                                      ({"AFSK_DEMOD_STAGES": "4"}, 1500), ({"AFSK_DEMOD_STAGES": "4"}, 375)])
def test_layouts_that_do_not_fit_are_refused(monkeypatch, env, baud):
    """a group whose ring would hold no stage, or whose stages exceed a CTA's shared memory, fails plan creation with
    AFSK_E_UNSUPPORTED (the plan is only created: nothing runs)"""
    _switches(monkeypatch, env)
    with pytest.raises(_cabi.AfskError) as e:
        A.RxSession([0, 200000], baud, 14000)
    assert e.value.code == _cabi.AFSK_E_UNSUPPORTED, str(e.value)
    _switches(monkeypatch, {})
    A.RxSession([0, 200000], baud, 14000).close()


# ---------------------------------------------------------------- streaming ---------------------------------------

CRAFTED = [(6000, 1), (4000, 300), (2400, 1), (1200, 300), (1000, 1), (300, 300), (160, 1), (100, 300)]
CRAFTED_WINDOWS = 90                                          # crafted windows of each class per channel
HALF_STEPS = {512: 512.5, 514: 513.5, -512: -512.5}          # int16 sample -> the float32 card value that rounds to it


def crafted_channels(n, seed=9200):
    """channels whose one recording is 12000 frames of a transmission's training (the gate opens there, the clock is
    recovered from it), then up to 100000 frames of limiter-edge soup carrying CRAFTED_WINDOWS windows of every class
    aligned to the recording's clock, then silence.  Thresholds (amp_end 1 or 300) keep every chunk loud through the
    crafted windows.  -> [dict(baud, a0, a1, timeout, x, pays)] as demod_channels"""
    rng = np.random.default_rng(seed)
    chans = []
    for baud, a1 in CRAFTED:
        bf = bit_frames(baud)
        lead, T = int(rng.integers(3000, 30000)), 12000
        L = min(100000, n - lead - T - 20000) // bf * bf
        x = np.zeros(n, np.int64)
        x[lead:lead + T] = O.tx_frames(b"\x00", baud, 0.5)[:T]
        x[lead + T:lead + T + L] = rng.choice(SOUP, L)
        start = O.listen_gate(x.astype(np.int16), 18000, a1, 96000)[1]
        clk = O.rx_decode(x[start:start + SYNC].astype(np.int16), baud, a1)["clock"]
        k0 = -(-(lead + T - start - clk) // bf)
        k1 = (lead + T + L - start - clk) // bf
        cls = tie_classes(bf) + edge_classes(a1, bf)
        at = rng.choice(np.arange(k0, k1), min(k1 - k0, CRAFTED_WINDOWS * len(cls)), replace=False)
        for j, k in enumerate(at):
            w0 = start + clk + k * bf
            x[w0:w0 + bf] = class_window(cls[j % len(cls)], baud, a1, rng)
        x = x.astype(np.int16)
        rec = [(a, e) for r, a, e in O.listen_gate_multi(x, 18000, a1, 96000) if r]
        assert rec[0][0] == start and rec[0][1] >= lead + T + L, (baud, rec)      # one recording over it all
        chans.append(dict(baud=baud, a0=18000, a1=a1, timeout=2.0, x=x, pays=[]))
    return chans


LONG_CHANNELS = 24


def long_channels(n, seed=9300):
    """LONG_CHANNELS channels at 12000 baud, each one recording of ~200000 frames: over 32768 windows, more than its
    first plane slot holds, so that their slots move while they are open and, together, outgrow the plane arena"""
    rng = np.random.default_rng(seed)
    chans = []
    for _ in range(LONG_CHANNELS):
        lead = int(rng.integers(2000, 40000))
        fr = O.tx_frames(rng.integers(0, 256, 3600, dtype=np.uint8).tobytes(), 12000, 0.1).astype(np.float64)
        x = np.zeros(n)
        x[lead:lead + len(fr)] = fr[:n - lead] * rng.uniform(0.6, 1.0)
        x = np.clip(np.round(x + rng.normal(0, 2000, n)), -32768, 32767).astype(np.int16)
        chans.append(dict(baud=12000, a0=18000, a1=14000, timeout=2.0, x=x, pays=[]))
    return chans


@functools.lru_cache(maxsize=1)
def stream_case():
    chans = demod_channels()
    chans = chans + long_channels(len(chans[0]["x"])) + crafted_channels(len(chans[0]["x"]))
    settings = [(c["baud"], c["a0"], c["a1"], c["timeout"]) for c in chans]
    streams = [c["x"] for c in chans]
    return chans, settings, streams, oracle_calls(streams, settings)


def _float_frames(pieces):
    X = np.stack(pieces, axis=1)
    F = X.astype(np.float32) / np.float32(32768)
    for v, h in HALF_STEPS.items():
        F[X == v] = np.float32(h / 32768)
    return F, int(np.isin(X, list(HALF_STEPS)).sum())


@pytest.mark.parametrize("mode", ["bits", "payload"])
def test_streaming_planes_equal_the_reference_after_every_push(mode):
    """bits and payload retention over demod_channels' traffic and the crafted channels, pushed in pieces of PIECES'
    lengths (windows and 32-window words straddle pushes): after every push, each channel's retained windows of its
    open recording equal ref_planes over the recording's frames (start from state(), clock from pending_bits(), counted
    from the recording's first frame).  One push is a float32 card window whose samples sit on half steps at the
    limiter edge.  Plane compactions happen while recordings are open; in bits mode one moves the planes of a recording
    that stays open, and they still match."""
    chans, settings, streams, (wants, dec) = stream_case()
    S, n = len(streams), len(streams[0])
    crafted = range(S - len(CRAFTED), S)
    cuts = piece_cuts(n, np.random.default_rng(["bits", "payload"].index(mode) + 40)) + [n]
    bounds = list(zip([0] + cuts[:-1], cuts))
    halves = [sum(int(np.isin(streams[s][a:b], list(HALF_STEPS)).sum()) for s in crafted) if b - a >= 2048 else 0
              for a, b in bounds]
    fpush = int(np.argmax(halves))
    assert halves[fpush] >= 100, halves
    refs, covered = {}, {}
    got = [[] for _ in range(S)]
    checked = trimmed = 0
    moved = compacted_open = False
    with A.open_receive_streams(receivers(settings), [x[3] for x in settings], retain=mode) as st:
        held = {}
        for i, (a, b) in enumerate(bounds):
            pieces = [x[a:b] for x in streams]
            c0 = st.counters()["plane_compactions"]
            if i == fpush:
                F, nh = _float_frames(pieces)
                assert nh == sum(int(np.isin(pieces[s], list(HALF_STEPS)).sum()) for s in range(S))
                take(got, st.push_interleaved(F, dtype=np.float32))
            else:
                take(got, st.push(pieces))
            compacted = st.counters()["plane_compactions"] > c0
            compacted_open |= compacted and any(st.pending_bits(s)[1] > 0 for s in range(S))
            now = {}
            for s in range(S):
                baud, _, a1, _ = settings[s]
                first, bits, quiet = st.pending_planes(s)
                _, start, _ = st.state(s)
                clk, decided = st.pending_bits(s)
                if len(bits) == 0:
                    continue
                bf = bit_frames(baud)
                assert start >= 0 and clk >= 0 and first % 32 == 0 and first + len(bits) == decided, (s, i, first, decided)
                assert start + clk + (first + len(bits)) * bf <= b, (s, i)          # decided windows lie in frames pushed
                key = (s, start)
                if key not in refs:
                    assert clk == O.rx_decode(streams[s][start:start + SYNC], baud, a1)["clock"], (s, start)
                    end = next(e for r, a0, e in wants[s] if r and a0 == start)
                    refs[key] = (clk, ref_planes(streams[s][start:min(n, end + 4096)], baud, clk, a1))
                    covered[key] = np.zeros(len(refs[key][1][0]), bool)
                rb, rq = refs[key][1]
                assert first + len(bits) <= len(rb), (s, i)
                for name, g, r in (("bits", bits, rb), ("quiet", quiet, rq)):
                    bad = np.flatnonzero(g != r[first:first + len(g)])
                    assert len(bad) == 0, (mode, s, baud, i, name, first, (first + bad[:8]).tolist())
                covered[key][first:first + len(bits)] = True
                checked += len(bits)
                trimmed += first > 0
                now[s] = (start, first, len(bits))
                if compacted and s in held and held[s][0] == start:
                    moved = True                                  # this recording's planes were moved and still match
            held = now
        take(got, st.finish())
    for s in range(S):
        check_final(got[s], wants[s], dec, s)
    assert checked > 0 and compacted_open, (checked, compacted_open)
    if mode == "payload":
        assert trimmed > 0                                       # windows below the framing's need were dropped
        return
    assert moved                                                 # bits mode keeps every window: a compaction moved some
    for s in crafted:                                             # the crafted windows were all compared
        baud, _, a1, _ = settings[s]
        key = next(k for k in covered if k[0] == s)
        cnt = window_classes(streams[s][key[1]:], baud, refs[key][0], a1, 0, int(np.flatnonzero(covered[key])[-1]) + 1)
        for c in tie_classes(bit_frames(baud)) + edge_classes(a1, bit_frames(baud)):
            assert cnt[c] >= N_CLASS, (s, baud, c, cnt)

