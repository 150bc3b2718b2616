"""GPU (-m gpu): every framing path against the plain references of tests/test_frame_cases_model.py, on captures and
recordings crafted to reach the inputs where framing goes wrong.

The batch: every case of batch_cases (terminator positions, ends of capture, first quiet windows, payload layouts,
long captures, each path's search-step edges) at 12000, 6000, 2400, 1200 and 300 baud, in one mixed batch with
capture starts at every residue mod 8.  Each capture's (status, clock, train_end, nbits, nbytes, payload) must equal
the oracle's and the case's reference, and its planes the crafted sequence (so a failure points at framing, not at
the demodulator), under automatic kernel choice, every AFSK_OPT_FRAME_KERNEL and the fused schedule that frames on
its auxiliary warps.

The streaming receiver in payload mode: channels whose one recording carries crafted windows aligned to its clock,
with the terminator, the first quiet window or a byte group's first window at -3 .. +3 windows from a framed-window
limit, fed in three schedules.  After every push pending_payload must equal the k_stream_frame restatement at the
same limit, and pending_planes the recording's planes."""
import ctypes as C
import functools
import os

import numpy as np
import pytest

import afskmodem_b200 as A
from afskmodem_b200 import _cabi
from oracle import oracle as O
from test_demod_planes_model import SYNC, bit_frames, frame, ref_planes
from test_frame_cases_model import (AMP_END, D, MAX_WINDOWS, QUIET, StreamFramer, _tones, batch_cases, frame_cases,
                                    path_cases, pending_of, sequence, stream_tags)
from test_gpu_stream_oracle import check_final, oracle_calls, receivers, take
from test_stream_bits_model import windows_of
from test_stream_gate_model import CHUNK

pytestmark = pytest.mark.gpu
A.LOG_LEVEL = 5
THREADS = os.cpu_count() or 1
OPT_FRAME_KERNEL, OPT_FUSED = 1, 3                       # AFSK_OPT_* of afsk_b200.h
SWITCHES = ("AFSK_FUSED", "AFSK_FRAME_KERNEL", "AFSK_GROUP_STREAMS", "AFSK_CLOCK_KERNEL")


@functools.lru_cache(maxsize=1)
def batch():
    """the cases in shuffled order behind spacer captures (0 .. 7 zero frames: No clock) that put capture starts at
    every residue mod 8; the oracle's result of every capture; the capture index of every case"""
    cases = batch_cases()
    rng = np.random.default_rng(9400)
    caps, bauds, where = [], [], {}
    pos = 0
    for t, i in enumerate(rng.permutation(len(cases))):
        gap = (t % 8 - pos) % 8
        caps.append(np.zeros(gap, np.int16))
        bauds.append(1200)
        pos += gap
        x = cases[i].audio()
        where[len(caps)] = cases[i]
        caps.append(x)
        bauds.append(cases[i].baud)
        pos += len(x)
    samples = np.concatenate(caps)
    lens = np.array([len(x) for x in caps], np.int64)
    starts = np.concatenate([[0], np.cumsum(lens)])[:-1]
    datas, res = O.rx_decode_batch(samples, np.append(starts, len(samples)), bauds, AMP_END, threads=THREADS)
    want = [(r.status, r.clock, r.train_end, r.nbits, r.nbytes, d) for r, d in zip(res, datas)]
    return samples, starts, lens, np.array(bauds, np.int32), want, where


def _launches(s) -> int:
    n = C.c_int(0)
    _cabi.check(_cabi.lib().afsk_rx_plan_launches(s.plan, C.byref(n)))
    return n.value


def _session(sel, opts=()):
    samples, starts, lens, bauds = batch()[:4]
    s = A.RxSession(starts[sel], bauds[sel], np.full(len(sel), AMP_END, np.int32), lengths=lens[sel])
    for o, v in opts:
        _cabi.check(_cabi.lib().afsk_rx_plan_set_option(s.plan, o, v))
    s.upload(samples)
    return s


def _run_observed(s):
    """runs the decode under torch.profiler -> the names of the framing kernels it launched, blanks removed"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        s.run()
        torch.cuda.synchronize()
    return {e.name.replace(" ", "") for e in prof.events() if "k_frame" in e.name}


def _check(s, sel, run):
    """every capture's result equals the oracle's, every case's its reference, every case's planes its crafted
    sequence.  -> (the cases compared, the framing kernels the decode launched)"""
    want, where = batch()[4:]
    launched = _run_observed(s)
    b = s.download()
    seen = []
    for j, i in enumerate(sel):
        got = (int(b.status[j]), int(b.clock[j]), int(b.train_end[j]), int(b.nbits[j]), int(b.nbytes[j]), b.payload(j))
        assert got == want[i], (run, i, got[:5], want[i][:5])
        c = where.get(int(i))
        if c is None:
            continue
        assert got == c.reference(), (run, c.baud, c.name, got[:5], c.reference()[:5])
        bits, quiet = s.planes(j)
        assert np.array_equal(bits[:c.K], c.bits) and np.array_equal(quiet[:c.K], c.quiet), (run, c.baud, c.name)
        seen.append(c)
    return seen, launched


def _assert_reached(seen, path, bauds=None):
    """every family and named residue of the path's cases (at `bauds`, where the run is limited to some) was compared"""
    want = [c for c in path_cases(path) if bauds is None or c.baud in bauds]
    tags = set().union(*(c.tags for c in seen))
    assert {c.family for c in seen} == {c.family for c in want}, path
    missing = set().union(*(c.tags for c in want)) - tags
    assert not missing, (path, sorted(missing))
    got = {(c.baud, c.name) for c in seen}
    assert all((c.baud, c.name) in got for c in want), path


def _select(limit=None, bauds=None):
    _, _, _, bd, _, where = batch()
    return np.array([i for i in range(len(bd)) if i not in where or
                     ((limit is None or where[i].kmax <= limit) and (bauds is None or int(bd[i]) in bauds))])


# the kernel each framing path launches, as the profiler names it (blanks removed)
KERNEL_NAME = {"warp": "k_frame_warp(", "cta128": "k_frame<128,4,int>(", "cta512": "k_frame<512,8,int>(",
               "cta512_64": "k_frame<512,8,longlong>("}


def frame_path(kmaxes, fk):
    """the framing kernel a decode of captures with these windows at clock 0 is meant to launch (afsk_rx.cu
    launch_frame; the CTA variants by the batch's average): what the runs expect of the profiler"""
    m = max(kmaxes)
    if fk == 1 and m > MAX_WINDOWS["warp"]:
        fk = 0
    if fk == 0:
        fk = 1 if m <= MAX_WINDOWS["warp"] else 3 if sum(kmaxes) > 65536 * len(kmaxes) else 2
    return {1: "warp", 2: "cta128", 3: "cta512", 4: "cta512_64"}[fk]


# run: (AFSK_OPT_FRAME_KERNEL or None, path the run frames with, window limit of its captures)
RUNS = {
    "auto": (None, "cta128", None),                    # a capture over 2^18 windows: k_frame<128,4>
    "auto_warp": (None, "warp", MAX_WINDOWS["warp"]),  # every capture within 2^18 windows: k_frame_warp
    "kernel1": (1, "warp", MAX_WINDOWS["warp"]),
    "kernel2": (2, "cta128", None),
    "kernel3": (3, "cta512", None),
    "kernel4": (4, "cta512_64", None),
}


@pytest.mark.parametrize("run", list(RUNS))
def test_framing_kernels_on_crafted_captures(monkeypatch, run):
    for k in SWITCHES:
        monkeypatch.delenv(k, raising=False)
    fk, path, limit = RUNS[run]
    sel = _select(limit)
    where = batch()[5]
    assert frame_path([where[i].kmax for i in sel if i in where], fk or 0) == path, run
    s = _session(sel, ((OPT_FRAME_KERNEL, fk),) if fk is not None else ())
    try:
        seen, launched = _check(s, sel, run)
    finally:
        s.close()
    assert len(launched) == 1 and KERNEL_NAME[path] in next(iter(launched)), (run, launched)
    _assert_reached(seen, path.replace("_64", ""))
    assert (max(c.kmax for c in seen) > MAX_WINDOWS["warp"]) == (limit is None), run


def test_fused_schedule_frames_crafted_captures(monkeypatch):
    """AFSK_OPT_FUSED = 2 (framing on the demodulator's auxiliary warps) over the bauds whose groups the fused schedule
    takes, captures of at most 2^18 windows"""
    for k in SWITCHES:
        monkeypatch.delenv(k, raising=False)
    _, _, _, bd, _, where = batch()
    fusable = set()
    for b in sorted({c.baud for c in where.values()}):
        i = next(i for i, c in where.items() if c.baud == b and c.kmax <= MAX_WINDOWS["warp"])
        s = _session(np.array([i]), ((OPT_FUSED, 1),))
        if _launches(s) == 2:                                  # one demodulator launch with its clocks, then k_frame
            fusable.add(b)
        s.close()
    assert {6000, 2400, 1200} <= fusable, sorted(fusable)
    sel = _select(MAX_WINDOWS["warp"], fusable)
    s = _session(sel, ((OPT_FUSED, 2),))
    try:
        groups = len({int(bd[i]) for i in sel if i in where})
        assert _launches(s) == groups + 1, _launches(s)       # + k_preset (the spacers)
        seen, launched = _check(s, sel, "fused2")
    finally:
        s.close()
    assert not launched, launched                             # the frame jobs ran on the auxiliary warps
    _assert_reached(seen, "warp", fusable)


# ---------------------------------------------------------------- streaming ---------------------------------------

STREAM_BAUDS = (6000, 2400, 1200, 300)
STREAM_FAMILIES = ("term", "quiet", "byte")
STREAM_N = 40 * CHUNK


def limit_after(P, R, bf, clk):
    """the windows a push that ends at stream frame P frames a recording (start R, clock clk) up to: those of the
    chunks the gate has walked, as far as they are decided (streams_bits: min(windows_of(walked), decided & ~31))"""
    span = P - R - clk
    if span <= 0:
        return 0
    return min(windows_of(P // CHUNK * CHUNK - R, bf, clk), (span // bf) // 32 * 32)


def stream_channel(baud, fam, d, rng):
    """one recording: 3 chunks of a real transmission's training (the gate opens, the clock is recovered from it), then
    crafted windows aligned to its clock, then silence ("open": loud to the end of the stream, cut by finish).  Quiet
    windows stay well under a chunk, so the recording stays open over them (asserted with listen_gate_multi).  The
    critical window (terminator, first quiet window, first window of the fourth byte group) sits at d windows from the
    limit E of a push of the 2048-frame schedule.  -> dict(baud, x, start, clk, crit frames, ...)"""
    bf = bit_frames(baud)
    lead, T = int(rng.integers(2000, 9000)), 3 * CHUNK
    tx = O.tx_frames(b"\x00", baud, 0.5)
    x = np.zeros(STREAM_N, np.int64)
    x[lead:lead + T] = tx[:T]
    start = O.listen_gate(x.astype(np.int16), 18000, AMP_END, 96000)[1]
    clk = O.rx_decode(x[start:start + SYNC].astype(np.int16), baud, AMP_END)["clock"]
    kc = -(-(lead + T - start - clk) // bf)
    x[lead + T:start + clk + kc * bf] = tx[T:start + clk + kc * bf - lead]
    m = next(m for m in range(1, 64) if limit_after(m * CHUNK, start, bf, clk) >= kc + 80)
    E = limit_after(m * CHUNK, start, bf, clk)
    if fam == "term":
        k_t, q = E + d, E + d + 1 + 14 * 6 + 5
    elif fam == "quiet":
        k_t, q = E - 40, E + d
    elif fam == "byte":
        k_t, q = E + d - 14 * 3 - 1, E + d + 14 * 4 + 3
    else:
        k_t, q = kc + 30, None
    # loud windows for over two chunks past the last crafted one: the first quiet window ends the result inside a
    # loud recording, which stays open for pushes after it
    n_win = (STREAM_N - start - clk) // bf - 2 if fam == "open" else q + (5 * CHUNK // 2) // bf + int(rng.integers(0, 60))
    bits, quiet = sequence(n_win - kc, k_t - kc, rng, "alt", quiet=[] if q is None else [q - kc])
    bits[:2] = [1, 0]
    W0 = start + clk + kc * bf
    mark, space = _tones(baud)
    Wv = np.where(bits[:, None], mark, space)
    Wv = np.where(quiet[:, None], np.sign(Wv) * QUIET, Wv)
    x[W0:W0 + Wv.size] = Wv.ravel()
    x = x.astype(np.int16)
    rec = [(a, e) for r, a, e in O.listen_gate_multi(x, 18000, AMP_END, 96000) if r]
    assert len(rec) == 1 and rec[0][0] == start, (baud, fam, d, rec)
    rb, rq = ref_planes(x[start:], baud, clk, AMP_END)
    assert np.array_equal(rb[kc:kc + len(bits)], bits) and np.array_equal(rq[kc:kc + len(bits)], quiet), (baud, fam, d)
    assert not rq[:kc].any(), (baud, fam, d)
    crit = {"term": k_t, "quiet": q, "byte": k_t + 1 + 14 * 3, "open": k_t}[fam]
    return dict(baud=baud, fam=fam, d=d, x=x, start=start, clk=clk, bf=bf, planes=(rb, rq), E=E, m=m,
                crit=crit, crit_frame=start + clk + (crit + 1) * bf)


@functools.lru_cache(maxsize=1)
def stream_case():
    rng = np.random.default_rng(9500)
    chans = [stream_channel(b, f, d, rng) for b in STREAM_BAUDS for f in STREAM_FAMILIES for d in D]
    chans += [stream_channel(b, "open", 0, rng) for b in STREAM_BAUDS]
    settings = [(c["baud"], 18000, AMP_END, 2.0) for c in chans]
    streams = [c["x"] for c in chans]
    return chans, settings, streams, oracle_calls(streams, settings)


def schedules(chans):
    n = STREAM_N
    a = list(range(CHUNK, n, CHUNK)) + [n]
    crit = sorted({c["crit_frame"] + e for c in chans for e in (-1, 0, 1)})
    b = sorted(set(crit + list(range(65536, n, 65536)) + [n]))
    one = sorted({c["m"] * CHUNK + e for c in chans for e in range(-2, 3)})
    c = sorted(set(a + one))
    return {"pieces2048": a, "critical_cuts": b, "one_frame": c}


@pytest.mark.parametrize("schedule", ["pieces2048", "critical_cuts", "one_frame"])
def test_streaming_payload_framing_at_every_limit(schedule):
    chans, settings, streams, (wants, dec) = stream_case()
    S = len(chans)
    cuts = schedules(chans)[schedule]
    framers = [StreamFramer(*c["planes"], seed=s) for s, c in enumerate(chans)]
    got = [[] for _ in range(S)]
    compared = np.zeros(S, np.int64)                           # pushes compared per channel
    at_m = np.zeros(S, bool)                                   # compared right after its push m (the limit E)
    prev = 0
    with A.open_receive_streams(receivers(settings), [x[3] for x in settings], retain="payload") as st:
        for P in cuts:
            take(got, st.push([x[prev:P] for x in streams]))
            prev = P
            for s, c in enumerate(chans):
                _, R, _ = st.state(s)
                clk, _ = st.pending_bits(s)
                if R != c["start"] or clk < 0:
                    continue
                assert clk == c["clk"], (s, P)
                fr = framers[s]
                fr.advance(limit_after(P, R, c["bf"], clk))
                te, nb, ended, by = st.pending_payload(s)
                assert (te, nb, ended) == pending_of(fr.F, clk, c["bf"]), (schedule, s, c["baud"], c["fam"], c["d"], P, fr.F)
                assert by == bytes(fr.data), (schedule, s, P, len(by), len(fr.data))
                first, bits, quiet = st.pending_planes(s)
                rb, rq = c["planes"]
                assert np.array_equal(bits, rb[first:first + len(bits)]) and np.array_equal(quiet, rq[first:first + len(quiet)]), (s, P)
                compared[s] += 1
                at_m[s] |= P == c["m"] * CHUNK
        take(got, st.finish())
    for s in range(S):
        check_final(got[s], wants[s], dec, s)
    assert compared.min() >= 1, (schedule, np.flatnonzero(compared == 0).tolist())
    if schedule != "critical_cuts":                            # (its cuts are the critical frames, not the chunk ends)
        assert at_m.all(), (schedule, np.flatnonzero(~at_m).tolist())
    # what the jobs met, per family: the critical window on either side of a limit, and the three named edges
    tags = set().union(*(stream_tags(f.reads) for f in framers))
    assert {"term 1 in previous push and word", "byte cut by limit"} <= tags, (schedule, tags)
    assert {"quiet at job start", "quiet at limit"} & tags, (schedule, tags)
    if schedule == "pieces2048":
        for s, c in enumerate(chans):
            f = framers[s].F
            assert f["phase"] >= 1, (s, c["fam"])
            if c["fam"] == "term":
                assert f["k0"] == c["E"] + c["d"] + 1
            if c["fam"] == "quiet":
                assert f["k1"] == c["E"] + c["d"]
        ended_early = [s for s, c in enumerate(chans) if c["fam"] != "open" and framers[s].F["phase"] == 2]
        assert len(ended_early) == S - len(STREAM_BAUDS)


# ---------------------------------------------------------------- the stream path's cases as recordings ------------

CASE_BAUDS = (6000, 2400, 1200)
E_BAUDS = (2400, 1200)               # bit lengths whose finish-cut K takes every residue mod 32 as the cut moves


@functools.lru_cache(maxsize=None)
def _tx(baud):
    return O.tx_frames(b"\x00", baud, 0.5).astype(np.int64)            # 0.5 s of training: 24000 frames


def _windows(baud, bits, quiet):
    mark, space = _tones(baud)
    W = np.where(np.asarray(bits, bool)[:, None], mark, space)
    return np.where(np.asarray(quiet, bool)[:, None], np.sign(W) * QUIET, W).ravel()


def case_channel(c, rng):
    """one recording carrying case c: real training (the gate opens, the clock is recovered from it) for windows
    0 .. kc - 1, then the case's windows from kc on.
      * T / Q / H: kc is the limit of the push that stores the clock (a multiple of 32: the case's residues and its
        step edges counted from the word where the next framing job starts).  A quiet window follows the case's last
        window (where the case has none, the same result), then over two chunks of loud windows, then silence.
      * E: kc puts the case's last window right before the end of the recording's last full chunk; loud space tones
        (decided 0s, past K in the planes) follow, and the recording is cut there by finish.
    -> dict(case, x, start, clk, bf, kc, b1 (frames of the first push in the two-push schedule), K (E), planes)"""
    bf, tx = bit_frames(c.baud), _tx(c.baud)
    for _ in range(64):
        lead = int(rng.integers(2000, 9000))
        head = np.concatenate([np.zeros(lead, np.int64), tx])
        start = O.listen_gate(head.astype(np.int16), 18000, AMP_END, 96000)[1]
        clk = O.rx_decode(head[start:start + SYNC].astype(np.int16), c.baud, AMP_END)["clock"]
        # the first chunk end whose limit lies past the frames clock recovery reads (the crafted windows must not move
        # the clock) and is a multiple of 32 (at 4 and 8 frames per bit every chunk's limit has the same residue)
        b1 = next((b for b in range(-(-(start + SYNC) // CHUNK) * CHUNK, start + 6 * CHUNK, CHUNK)
                   if clk + limit_after(b, start, bf, clk) * bf >= SYNC and limit_after(b, start, bf, clk) % 32 == 0), None)
        if b1 is None:
            continue
        K = None
        if c.family == "E":
            lo = start + clk + (-(-(SYNC - clk) // bf) + 2 + c.K) * bf
            cand = [M * CHUNK for M in range(-(-lo // CHUNK), -(-lo // CHUNK) + 40)
                    if windows_of(M * CHUNK - start, bf, clk) % 32 == c.K % 32]
            if not cand:
                continue
            K = windows_of(cand[0] - start, bf, clk)
            kc = K - c.K
        else:
            kc = limit_after(b1, start, bf, clk)
        if start + clk + kc * bf <= lead + len(tx) - 4 * bf:
            break
    else:
        raise AssertionError((c.baud, c.name))
    w0 = start + clk + kc * bf
    if c.family == "E":
        tail = _windows(c.baud, np.zeros(CHUNK // bf + 40, bool), np.zeros(CHUNK // bf + 40, bool))
        body = np.concatenate([_windows(c.baud, c.bits, c.quiet), tail])
        n = start + clk + K * bf + CHUNK // 2
        n = -(-n // CHUNK) * CHUNK - CHUNK // 2                          # the last full chunk ends at cand[0]
    else:
        loud = (5 * CHUNK // 2) // bf + 8
        after = np.concatenate([[True], np.zeros(loud, bool)])
        body = np.concatenate([_windows(c.baud, c.bits, c.quiet),
                               _windows(c.baud, rng.integers(0, 2, loud + 1), after)])
        n = w0 + len(body) + 3 * CHUNK
    x = np.zeros(n, np.int64)
    x[lead:w0] = tx[:w0 - lead]
    x[w0:w0 + len(body)] = body[:n - w0]
    x = x.astype(np.int16)
    rec = [(a, e) for r, a, e in O.listen_gate_multi(x, 18000, AMP_END, 96000) if r]
    if c.family == "E":
        assert rec == [(start, n // CHUNK * CHUNK)], (c.baud, c.name, rec)          # open until finish cuts it
    elif len(rec) != 1 or rec[0][0] != start:
        return None                                                      # quiet windows closed a chunk: not usable
    rb, rq = ref_planes(x[start:], c.baud, clk, AMP_END)
    assert np.array_equal(rb[kc:kc + c.K], c.bits) and np.array_equal(rq[kc:kc + c.K], c.quiet), (c.baud, c.name)
    assert not rq[:kc].any() and frame(rb[:kc], rq[:kc], 0, bf)[0] == kc * bf, (c.baud, c.name)   # training only
    if c.family == "E":
        assert windows_of(n // CHUNK * CHUNK - start, bf, clk) == K
    return dict(case=c, x=x, start=start, clk=clk, bf=bf, kc=kc, b1=b1, K=K, planes=(rb, rq))


@functools.lru_cache(maxsize=1)
def case_streams():
    rng = np.random.default_rng(9600)
    chans = []
    for b in CASE_BAUDS:
        for c in frame_cases(b, "stream"):
            if c.family == "E" and b not in E_BAUDS:
                continue
            ch = case_channel(c, rng)
            if ch is not None:
                chans.append(ch)
    settings = [(ch["case"].baud, 18000, AMP_END, 2.0) for ch in chans]
    streams = [ch["x"] for ch in chans]
    return chans, settings, streams, oracle_calls(streams, settings)


def _case_result(ch):
    """the recording's result by the case's reference: (status, clock, train_end, nbits, payload) relative to the
    recording"""
    c = ch["case"]
    st, _, te, nbits, _, data = c.reference()
    k0 = (te - c.lead) // ch["bf"]
    return st, ch["clk"], ch["clk"] + (ch["kc"] + k0) * ch["bf"], nbits, data


@pytest.mark.parametrize("mode,schedule", [("payload", "two_push"), ("payload", "pieces2048"), ("bits", "two_push"),
                                           ("bits", "pieces2048")])
def test_stream_cases_as_recordings(mode, schedule):
    """The stream path's cases (T, E, Q, H and the 1024-window step edges) at 6000, 2400 and 1200 baud, one recording
    per channel.  two_push: the first push of each channel stores its clock and frames the training up to kc, the
    second frames all the rest in one job per recording (payload mode: k_stream_frame's search steps over the case),
    then finish cuts the E recordings (bits mode: their final framing through launch_frame over the stream's planes,
    with decided 0s past K).  pieces2048: 2048-frame pieces.  Payload mode: pending_payload equals the restatement
    after every push.  Every mode: pending_planes equals the planes, every result the oracle's and the case's."""
    chans, settings, streams, (wants, dec) = case_streams()
    S = len(chans)
    lens = [len(x) for x in streams]
    if schedule == "two_push":
        ends = [[ch["b1"] for ch in chans], lens]
    else:
        ends = [[min(L, k * CHUNK) for L in lens] for k in range(1, -(-max(lens) // CHUNK) + 1)]
    framers = [StreamFramer(*ch["planes"], seed=s) for s, ch in enumerate(chans)]
    got = [[] for _ in range(S)]
    compared = np.zeros(S, np.int64)
    prev = [0] * S

    def finals(ev):
        for i in range(len(ev)):
            s = int(ev.stream[i])
            ch = chans[s]
            if ev.recorded[i] and int(ev.start[i]) == ch["start"]:
                K = windows_of(int(ev.end[i]) - ch["start"], ch["bf"], ch["clk"])
                res, data = framers[s].final(K, ch["clk"], ch["bf"])
                assert res[:4] + (data,) == _case_result(ch), (mode, schedule, s, ch["case"].name, res[:4])

    with A.open_receive_streams(receivers(settings), [x[3] for x in settings], retain=mode) as st:
        for e in ends:
            ev = st.push([x[p:q] for x, p, q in zip(streams, prev, e)])
            take(got, ev)
            if mode == "payload":
                finals(ev)
            for s, ch in enumerate(chans):
                _, R, _ = st.state(s)
                clk, _ = st.pending_bits(s)
                if R != ch["start"] or clk < 0:
                    continue
                assert clk == ch["clk"], (s, e[s])
                if mode == "payload":
                    fr = framers[s]
                    fr.advance(limit_after(e[s], R, ch["bf"], clk))
                    te, nb, ended, by = st.pending_payload(s)
                    assert (te, nb, ended) == pending_of(fr.F, clk, ch["bf"]), (schedule, s, ch["case"].name, e[s], fr.F)
                    assert by == bytes(fr.data), (schedule, s, ch["case"].name, e[s])
                first, bits, quiet = st.pending_planes(s)
                rb, rq = ch["planes"]
                assert np.array_equal(bits, rb[first:first + len(bits)]) and np.array_equal(quiet, rq[first:first + len(quiet)]), (s, e[s])
                compared[s] += 1
            prev = e
        ev = st.finish()
        take(got, ev)
        if mode == "payload":
            finals(ev)
    for s, ch in enumerate(chans):
        check_final(got[s], wants[s], dec, s)
        rec = [g for g in got[s] if g[1]]
        assert len(rec) == 1 and rec[0][6] == _case_result(ch), (mode, schedule, s, ch["case"].name, rec[0][6][:4] if rec else None)
    assert compared.min() >= 1, np.flatnonzero(compared == 0).tolist()
    # what reached the GPU: every family, every tag of the stream path's cases at these bauds, E cut by finish
    seen = [ch["case"] for ch in chans]
    want = [c for b in CASE_BAUDS for c in frame_cases(b, "stream")]
    assert {c.family for c in seen} == set("TEQH")
    missing = set().union(*(c.tags for c in want)) - set().union(*(c.tags for c in seen))
    assert not missing, sorted(missing)
    cut = [s for s, ch in enumerate(chans) if ch["case"].family == "E" and got[s][-1][1] and got[s][-1][3] % CHUNK == 0]
    assert len(cut) == sum(ch["case"].family == "E" for ch in chans) >= 2 * 41
    if mode == "payload":
        tags = set().union(*(stream_tags(f.reads) for f in framers))
        need = {"quiet at job start", "byte cut by limit"} if schedule == "pieces2048" else {"term past step", "quiet past step"}
        assert need <= tags, (schedule, tags)
