"""GPU (-m gpu): round-2 features through the public API and the C ABI, bit-exact against the CPU oracle —
one corpus sharded over devices and gathered into one batch, plans re-targeted between layouts, the
host-buffer entry point called repeatedly, every framing-kernel variant (incl. the 64-bit-index one), a
noisy full-size 300-baud capture, the wav staging ring, argument validation, empty transmit batches."""
import ctypes as C
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

A = pytest.importorskip("afskmodem_b200")
from afskmodem_b200 import _cabi, shard  # noqa: E402
from oracle import oracle as O  # noqa: E402


@pytest.fixture(autouse=True, scope="module")
def _quiet_and_loaded():
    A.LOG_LEVEL = 5
    _cabi.require_device(0)      # no CPU fallback: fail loudly if the GPU/library is missing
    yield
    A.LOG_LEVEL = 0


def _mixed_corpus(seed, B, bauds=(300, 600, 1200, 2400, 4000, 6000, 4800, 9600, 1500, 800)):
    rng = np.random.default_rng(seed)
    caps, baud, thr, pls = [], [], [], []
    for i in range(B):
        b = int(rng.choice(bauds))
        btx = 6000 if b == 9600 else b
        pl = rng.integers(0, 256, int(rng.integers(1, 200)), dtype=np.uint8).tobytes()
        fr = O.tx_frames(pl, btx, float(rng.choice([0.5, 0.1, 0.02])))
        x = np.concatenate([np.zeros(int(rng.integers(0, 3000)), np.int16), fr]).astype(np.float64) * float(rng.choice([1.0, 0.7, 0.45]))
        sg = float(rng.choice([0, 2000, 8000, 14000, 19000, 26000]))
        if sg:
            x = x + np.round(rng.normal(0, sg, len(x)))
        caps.append(np.clip(np.trunc(x), -32768, 32767).astype(np.int16))
        baud.append(b); thr.append(int(rng.choice([14000, 11000, 8000]))); pls.append(pl)
    return caps, np.array(baud, np.int32), np.array(thr, np.int32), pls


def _assert_equals_oracle(batch, caps, baud, thr):
    assert len(batch) == len(caps)
    for i, x in enumerate(caps):
        o = O.rx_decode(x, int(baud[i]), int(thr[i]))
        if o["status"] < 0:
            assert int(batch.status[i]) == o["status"], i
            continue
        got = (int(batch.status[i]), int(batch.clock[i]), int(batch.train_end[i]), int(batch.nbits[i]), int(batch.nbytes[i]),
               batch.payload(i))
        want = (o["status"], o["clock"], o["train_end"], o["nbits"], o["nbytes"], o["data"])
        assert got == want, f"capture {i} baud {baud[i]}: {got[:5]} != {want[:5]}"


@pytest.mark.parametrize("devices", [[0, 0], [0, 0, 0, 0, 0], "all"])
def test_sharded_corpus_equals_single_device_and_oracle(devices):
    """ONE corpus cut into contiguous ranges by predicted time, one host thread + session per range, host
    gather in corpus order == the single-device decode == the oracle.  Several ranges on device 0 exercise
    the same code on a one-GPU box; "all" uses every visible GPU."""
    if devices == "all":
        devices = list(range(_cabi.device_count()))
        if len(devices) < 2:
            pytest.skip("needs at least two GPUs")
    caps, baud, thr, _ = _mixed_corpus(21, 96)
    samples, offsets = A.modem._concat(caps)
    rx = A.Receiver(1200)
    single = rx.decode_batch(samples, offsets, baud_rate=baud, amp_end_threshold=thr)
    sharded = rx.decode_batch(samples, offsets, baud_rate=baud, amp_end_threshold=thr, devices=devices)
    sess = rx._cache[1]
    assert isinstance(sess, A.ShardedRxSession) and len(sess.ranges) == len(devices)
    assert sess.ranges[0][0] == 0 and sess.ranges[-1][1] == len(caps)
    assert all(a[1] == b[0] for a, b in zip(sess.ranges, sess.ranges[1:]))
    assert np.array_equal(single.results, sharded.results)
    assert single.payloads() == sharded.payloads()
    _assert_equals_oracle(sharded, caps, baud, thr)
    # pipelined ranges inside every shard, and a repeat call on the cached session
    again = rx.decode_batch(samples, offsets, baud_rate=baud, amp_end_threshold=thr, devices=devices, pipeline=3)
    assert np.array_equal(single.results, again.results) and single.payloads() == again.payloads()
    rx.close()


def test_sharded_more_devices_than_captures_and_empty():
    caps, baud, thr, _ = _mixed_corpus(22, 2, bauds=(1200,))
    rx = A.Receiver(1200)
    b = rx.decode_batch(caps, devices=[0, 0, 0, 0], baud_rate=baud, amp_end_threshold=thr)
    _assert_equals_oracle(b, caps, baud, thr)
    e = rx.decode_batch([], devices=[0, 0])
    assert len(e) == 0 and e.payloads() == []
    rx.close()


def test_pipelined_batch_owns_its_arrays():
    """ADVICE r1: a field view of a pipelined decode must stay valid after the batch object is gone and the
    session has decoded something else (the arrays are copies, not views of pinned staging memory)."""
    caps, baud, thr, _ = _mixed_corpus(23, 24, bauds=(1200, 2400))
    samples, offsets = A.modem._concat(caps)
    rx = A.Receiver(1200)
    st = rx.decode_batch(samples, offsets, baud_rate=baud, amp_end_threshold=thr, pipeline=4).status
    blob = rx.decode_batch(samples, offsets, baud_rate=baud, amp_end_threshold=thr, pipeline=4).blob
    want_st, want_blob = st.copy(), blob.copy()
    assert st.base is None or st.base.flags["OWNDATA"] or st.base.base is None
    noise = [np.zeros(len(c), np.int16) for c in caps]
    for _ in range(3):
        rx.decode_batch(*A.modem._concat(noise), baud_rate=baud, amp_end_threshold=thr, pipeline=4)
    rx.close()
    assert np.array_equal(st, want_st) and np.array_equal(blob, want_blob)


def test_plan_retargeted_between_layouts():
    """Receiver.load-style use: one receiver, a different layout on every call (afsk_rx_plan_reset, grow-only
    buffers) — smaller, larger, empty, mixed baud — every call equal to the oracle."""
    rx = A.Receiver(1200)
    rng = np.random.default_rng(31)
    sess_ids = set()
    for it in range(14):
        B = int(rng.choice([1, 1, 2, 7, 40, 0, 3]))
        caps, baud, thr, _ = _mixed_corpus([31, it], B) if B else ([], np.zeros(0, np.int32), np.zeros(0, np.int32), [])
        b = rx.decode_batch(caps, baud_rate=baud, amp_end_threshold=thr)
        _assert_equals_oracle(b, caps, baud, thr)
        sess_ids.add(id(rx._cache[1]))
    assert len(sess_ids) == 1, "the cached session should have been re-targeted, not rebuilt"
    rx.close()


def test_decode_host_repeated_calls_reuse_context():
    L = _cabi.lib()
    rng = np.random.default_rng(32)
    for it in range(6):
        B = int(rng.integers(1, 9))
        caps, baud, thr, _ = _mixed_corpus([32, it], B, bauds=(1200, 300, 6000, 2400))
        samples, offsets = A.modem._concat(caps)
        cap = np.array([L.afsk_rx_out_capacity(len(c), int(b)) for c, b in zip(caps, baud)], np.int64)
        out_off = np.zeros(B + 1, np.int64); np.cumsum(cap, out=out_off[1:])
        out = np.zeros(int(out_off[-1]), np.uint8)
        res = (_cabi.RxResult * B)()
        _cabi.check(L.afsk_rx_decode_host(0, _cabi.ptr(samples, C.c_int16), _cabi.ptr(offsets, C.c_int64), B,
                                          _cabi.ptr(baud, C.c_int32), _cabi.ptr(thr, C.c_int32), _cabi.ptr(out, C.c_uint8),
                                          _cabi.ptr(out_off, C.c_int64), res))
        for i, x in enumerate(caps):
            o = O.rx_decode(x, int(baud[i]), int(thr[i]))
            assert (res[i].status, res[i].clock, res[i].train_end, res[i].nbits) == (o["status"], o["clock"], o["train_end"], o["nbits"])
            assert out[out_off[i]:out_off[i] + res[i].nbytes].tobytes() == o["data"]
    _cabi.check(L.afsk_rx_host_release(0))


@pytest.mark.parametrize("kernel", [1, 2, 3, 4])
def test_every_framing_kernel_variant(kernel):
    """AFSK_OPT_FRAME_KERNEL forces k_frame_warp / k_frame<128,4,int> / <512,8,int> / <512,8,long long> (the
    variant that is automatic only from 2^30 windows per capture) on ordinary captures: same results."""
    caps, baud, thr, _ = _mixed_corpus(33, 40)
    caps.append(np.zeros(5000, np.int16))                      # no terminator, all quiet
    baud = np.append(baud, 1200).astype(np.int32); thr = np.append(thr, 14000).astype(np.int32)
    samples, offsets = A.modem._concat(caps)
    s = A.RxSession(offsets, baud, thr)
    _cabi.check(_cabi.lib().afsk_rx_plan_set_option(s.plan, _cabi.OPT_FRAME_KERNEL, kernel))
    s.upload(samples); s.run()
    _assert_equals_oracle(s.download(), caps, baud, thr)
    s.close()


@pytest.mark.parametrize("kernel", [1, 2])
def test_framing_search_step_boundaries(kernel):
    """The framing kernels search the packed planes in steps of 256 words per warp (8 words per lane): captures of
    about 20,480 bit windows (640 plane words, two and a half steps) whose data ends inside the last plane words or is
    cut off by the end of the capture, with the terminator in the first plane word, without a terminator, without a
    quiet window, and all quiet — against the oracle."""
    rng = np.random.default_rng(77)
    caps, baud = [], []
    for bd, bf in ((6000, 8), (2400, 20), (1200, 40)):
        for dk in (-33, -32, -31, -2, -1, 0, 1, 2, 31, 32, 33):
            # payload sized so that the data ends inside the last plane words of a 20,480-window capture
            tsec = float(rng.choice([0.02, 0.2]))
            nbytes = (20480 - int(bd * tsec) - 40) // 14 - int(rng.integers(0, 80))   # ends inside the last words, or is cut off
            fr = O.tx_frames(rng.integers(0, 256, nbytes, dtype=np.uint8).tobytes(), bd, tsec)
            n = (20480 + dk) * bf + int(rng.integers(0, bf)) + bf
            x = np.zeros(n, np.int16)
            lead = int(rng.integers(0, 2 * bf))
            m = min(len(fr), n - lead)
            x[lead:lead + m] = fr[:m]
            caps.append(x); baud.append(bd)
        # terminator in the first plane word, data to the very end of the capture (no quiet window)
        fr = O.tx_frames(rng.integers(0, 256, 1400, dtype=np.uint8).tobytes(), bd, 8.0 / bd)
        caps.append(fr[:20470 * bf].copy()); baud.append(bd)
        # no terminator at all: training tone only, then loud noise (never quiet), then silence
        t = O.tx_frames(b"", bd, 1.0)[: 3000 * bf]
        caps.append(np.concatenate([t, rng.integers(-30000, 30000, 500 * bf).astype(np.int16), np.zeros(40 * bf, np.int16)]))
        baud.append(bd)
        caps.append(np.zeros(20480 * bf, np.int16)); baud.append(bd)
    baud = np.array(baud, np.int32); thr = np.full(len(caps), 14000, np.int32)
    samples, offsets = A.modem._concat(caps)
    s = A.RxSession(offsets, baud, thr)
    _cabi.check(_cabi.lib().afsk_rx_plan_set_option(s.plan, _cabi.OPT_FRAME_KERNEL, kernel))
    s.upload(samples); s.run()
    got = s.download()
    windows = [(len(c) - (bf0 := 48000 // int(b)) - max(int(k), 0) + bf0 - 1) // bf0 for c, b, k in zip(caps, baud, got.clock)]
    assert min(windows) < 20480 - 30 and max(windows) > 20480 + 30      # both sides of the bound were exercised
    _assert_equals_oracle(got, caps, baud, thr)
    s.close()


def test_config4_noisy_full_size_capture_vs_oracle():
    """One BASELINE config-4 capture at FULL size (64 KB payload at 300 baud: 146,830,080 frames) with AWGN
    over the whole capture and a lead of silence, decoded by the long-capture path (k_frame<512,8,int>):
    every stage integer and payload byte equal to the oracle's."""
    import torch
    rng = np.random.default_rng(44)
    pl = rng.integers(0, 256, 65536, dtype=np.uint8).tobytes()
    tx = A.TxSession([pl], 300, int(300 * 0.5 / 2))
    tx.upload(); tx.run(); _cabi.stream_sync(0)
    n = int(tx.out_len[0])
    assert n == 146830080
    host = tx.download().samples
    tx.close()
    lead = 1777
    g = torch.Generator(device="cuda"); g.manual_seed(4)
    x = torch.zeros(lead + n, dtype=torch.float32, device="cuda")
    x[lead:] = torch.from_numpy(host[:n]).cuda().to(torch.float32)
    x += torch.round(torch.randn(lead + n, generator=g, device="cuda") * 9000.0)
    noisy = torch.clamp(x, -32768, 32767).to(torch.int16).cpu().numpy()
    del x
    torch.cuda.empty_cache()
    offsets = np.array([0, len(noisy)], np.int64)
    s = A.RxSession(offsets, 300, 14000)
    s.upload(noisy); s.run()
    b = s.download()
    o = O.rx_decode(noisy, 300, 14000)
    got = (int(b.status[0]), int(b.clock[0]), int(b.train_end[0]), int(b.nbits[0]), int(b.nbytes[0]))
    assert got == (o["status"], o["clock"], o["train_end"], o["nbits"], o["nbytes"])
    assert b.payload(0) == o["data"]
    assert o["nbits"] >= 917504                     # the whole message and whatever the noisy tail adds
    s.close()


def test_load_batch_ring_equals_pinned_corpus_mode(tmp_path):
    """afsk_wav_load through the pinned staging ring (no host copy of the corpus) == the one-big-pinned-buffer
    mode == per-file load; with a file the native reader hands to CPython's wave (extensible format), a
    missing file, an empty file, and slots smaller than a file (a file split over several spans)."""
    caps, baud, thr, pls = _mixed_corpus(35, 30, bauds=(1200,))
    names = []
    for i, c in enumerate(caps):
        fn = str(tmp_path / f"c{i:03d}.wav")
        A.write_wav_frames(fn, c)
        names.append(fn)
    # an 8-bit stereo header over the same bytes: the reference pairs the bytes whatever the header says
    import wave
    odd = str(tmp_path / "odd.wav")
    with wave.open(odd, "wb") as f:
        f.setnchannels(2); f.setsampwidth(1); f.setframerate(8000)
        f.writeframes(caps[0].astype("<i2").tobytes())
    names.insert(5, odd)
    names.insert(9, str(tmp_path / "missing.wav"))
    empty = str(tmp_path / "empty.wav")
    A.write_wav_frames(empty, np.zeros(0, np.int16))
    names.append(empty)
    rx = A.Receiver(1200)
    per_file = []
    for fn in names:
        try:
            per_file.append(rx.load(fn, False))
        except Exception as e:  # noqa: BLE001
            per_file.append(type(e))
    norm = lambda out: [type(v) if isinstance(v, Exception) else v for v in out]   # noqa: E731
    for env in ({}, {"AFSK_WAV_SLOT_MB": "1", "AFSK_WAV_SLOTS": "2"}):
        os.environ.update(env)
        try:
            ring = rx.load_batch(names, string=False, errors="return", log=False)
            ring2 = rx.load_batch(names, string=False, errors="return", log=False, threads=3)
        finally:
            for k in env:
                os.environ.pop(k)
        assert norm(ring) == per_file and norm(ring2) == per_file
    pinned = rx.load_batch(names, string=False, errors="return", log=False, keep_host_copy=True)
    assert norm(pinned) == per_file
    assert per_file[0] == O.rx_decode(caps[0], 1200, 14000)["data"]
    rx.close()


def test_python_side_bounds_are_errors_not_device_faults(tmp_path):
    caps, baud, thr, _ = _mixed_corpus(36, 3, bauds=(1200,))
    samples, offsets = A.modem._concat(caps)
    s = A.RxSession(offsets, baud, thr)
    with pytest.raises(ValueError):
        s.upload(samples[:-10])
    with pytest.raises(ValueError):
        s.bind(0x7F0000000010 + 2)                              # misaligned
    with pytest.raises(ValueError):
        s.bind(0x7F0000000000, nsamples=len(samples) - 1)       # short buffer
    d = _cabi.DeviceBuffer(0, 64)
    with pytest.raises(ValueError):
        d.upload(np.zeros(100, np.uint8))
    with pytest.raises(ValueError):
        d.download(np.zeros(100, np.uint8))
    d.close(); s.close()
    p = A.PipelinedRxSession(offsets, baud, thr, 0, 2)
    with pytest.raises(ValueError):
        p.decode(samples[:100])
    p.close()
    with pytest.raises(ValueError):
        A.write_wav_batch([str(tmp_path / "never_written.wav")], samples, [len(samples) - 5], [10])


def test_empty_tx_batch(tmp_path):
    t = A.Transmitter(1200)
    b = t.encode_batch([])
    assert len(b) == 0 and len(b.samples) == 0
    t.save_batch([], [])
    # one empty payload is still a full frame: training + terminator + tail
    one = t.encode_batch([b""])
    assert np.array_equal(one.frames(0), O.tx_frames(b"", 1200))


# ------------------------------------------------------------------------------------------------
# fused schedule: clock recovery and framing as jobs of auxiliary warps inside the streaming kernel
def _decode_with(samples, offsets, baud, thr, fused, frame_kernel=0, repeats=1):
    s = A.RxSession(offsets, baud, thr)
    L = _cabi.lib()
    _cabi.check(L.afsk_rx_plan_set_option(s.plan, _cabi.OPT_FUSED, fused))
    _cabi.check(L.afsk_rx_plan_set_option(s.plan, _cabi.OPT_FRAME_KERNEL, frame_kernel))
    n = C.c_int(0)
    _cabi.check(L.afsk_rx_plan_launches(s.plan, C.byref(n)))
    s.upload(samples)
    out = None
    for _ in range(repeats):
        s.run()
        b = s.download()
        if out is not None:
            assert np.array_equal(out.results, b.results) and out.payloads() == b.payloads(), "repeat decode differs"
        out = b
    s.close()
    return out, n.value


def test_fused_request_with_a_padded_layout_group_keeps_three_kernels():
    """1500 / 750 / 375 baud use the padded layout, whose ring leaves no shared memory for the auxiliary warps at two
    CTAs per SM: a batch holding such a group is decoded by the three kernels whatever AFSK_OPT_FUSED says."""
    caps, baud, thr, _ = _mixed_corpus(53, 60, bauds=(1200, 6000, 1500, 750, 375))
    samples, offsets = A.modem._concat(caps)
    three, n3 = _decode_with(samples, offsets, baud, thr, 0)
    fused, nf = _decode_with(samples, offsets, baud, thr, 2)
    assert nf == n3
    assert np.array_equal(three.results, fused.results) and three.payloads() == fused.payloads()
    _assert_equals_oracle(fused, caps, baud, thr)


def test_fused_equals_three_kernels_and_oracle_mixed():
    caps, baud, thr, _ = _mixed_corpus(51, 160, bauds=(300, 600, 1200, 2400, 4000, 6000, 4800, 9600, 800, 2000, 3000, 480))
    samples, offsets = A.modem._concat(caps)
    three, n3 = _decode_with(samples, offsets, baud, thr, 0)
    fused, nf = _decode_with(samples, offsets, baud, thr, 2, repeats=4)
    assert nf < n3, (nf, n3)                      # one launch per bit length (+ the preset kernel), no k_clock / k_frame
    assert np.array_equal(three.results, fused.results)
    assert three.payloads() == fused.payloads()
    _assert_equals_oracle(fused, caps, baud, thr)
    # fused clocks with a separate framing kernel
    half, nh = _decode_with(samples, offsets, baud, thr, 1)
    assert nh == nf + 1
    assert np.array_equal(three.results, half.results) and three.payloads() == half.payloads()


def test_fused_many_short_captures_and_every_start_alignment():
    """Thousands of captures of one or two tiles each: every CTA completes far more captures than its
    framing queue holds while its auxiliary warps are still busy with clock jobs; every 16-byte phase of the
    capture start; captures just above the 4096-frame minimum; a too-short and an empty one in between."""
    rng = np.random.default_rng(52)
    base = [O.tx_frames(rng.integers(0, 256, n, dtype=np.uint8).tobytes(), 6000, 0.02) for n in (1, 5, 16, 40)]
    caps = []
    for i in range(6000):
        fr = base[i % 4]
        x = np.concatenate([np.zeros(i % 23, np.int16), fr]).astype(np.int32)
        if i % 3:
            x = x + np.round(rng.normal(0, 5000, len(x))).astype(np.int32)
        caps.append(np.clip(x, -32768, 32767).astype(np.int16))
    caps[100] = caps[100][:3000]
    caps[200] = np.zeros(0, np.int16)
    baud = np.full(len(caps), 6000, np.int32)
    thr = np.full(len(caps), 14000, np.int32)
    samples, offsets = A.modem._concat(caps)
    three, _ = _decode_with(samples, offsets, baud, thr, 0)
    fused, _ = _decode_with(samples, offsets, baud, thr, 2, repeats=3)
    assert np.array_equal(three.results, fused.results) and three.payloads() == fused.payloads()
    for i in list(range(0, 6000, 97)) + [100, 200]:
        o = O.rx_decode(caps[i], 6000, 14000)
        assert (int(fused.status[i]), int(fused.clock[i]), int(fused.nbits[i]), fused.payload(i)) == \
               (o["status"], o["clock"], o["nbits"], o["data"]), i


@pytest.mark.parametrize("baud", [6000, 3000, 2000, 4000, 2400, 1200, 600, 300, 1500, 750, 375, 800, 480, 400, 1000, 500, 12000])
def test_fused_clock_every_baud_and_offset(baud):
    """The auxiliary warps' clock search (two passes of 2048 candidates, multiply-shift floor, key minimum) against
    the oracle's first minimum: every capture start phase, clock offsets over a whole training cycle, clean and
    noisy, plus noise-only captures where the minimum is anywhere in the window."""
    rng = np.random.default_rng([53, baud])
    bf = 48000 // baud
    caps = []
    for i in range(2 * bf + 9):
        fr = O.tx_frames(b"clock", baud, 0.25)
        lead = i if i < 2 * bf else int(rng.integers(0, 4000))
        x = np.concatenate([np.zeros(lead, np.int16), fr]).astype(np.int32)
        if i % 2:
            x = x + np.round(rng.normal(0, float(rng.choice([3000, 12000, 30000])), len(x))).astype(np.int32)
        caps.append(np.clip(x, -32768, 32767).astype(np.int16))
    for i in range(24):
        caps.append(np.clip(np.round(rng.normal(0, 9000, 4096 + 37 * i)), -32768, 32767).astype(np.int16))
    b = np.full(len(caps), baud, np.int32)
    thr = np.full(len(caps), 14000, np.int32)
    samples, offsets = A.modem._concat(caps)
    fused, _ = _decode_with(samples, offsets, b, thr, 2)
    _assert_equals_oracle(fused, caps, b, thr)


def test_fused_long_capture_and_retargeted_plan():
    """A capture of more than 2^18 bit windows keeps the separate framing kernel (fused clocks only); the same
    plan is then re-targeted at short captures (fused framing) and back."""
    rng = np.random.default_rng(54)
    pl = rng.integers(0, 256, 40000, dtype=np.uint8).tobytes()
    long_cap = O.tx_frames(pl, 6000, 0.1)                     # 560 K windows of 8 frames
    long_cap = np.clip(long_cap.astype(np.int32) + np.round(rng.normal(0, 6000, len(long_cap))).astype(np.int32), -32768, 32767).astype(np.int16)
    shorts, baud, thr, _ = _mixed_corpus(55, 30, bauds=(6000, 1200))
    rx = A.Receiver(6000)
    os.environ["AFSK_FUSED"] = "2"
    try:
        for caps, bd, th in (([long_cap], np.array([6000], np.int32), np.array([14000], np.int32)), (shorts, baud, thr),
                             ([long_cap, shorts[0]], np.array([6000, baud[0]], np.int32), np.array([14000, thr[0]], np.int32)),
                             (shorts[:3], baud[:3], thr[:3])):
            b = rx.decode_batch(caps, baud_rate=bd, amp_end_threshold=th)
            _cabi.check(_cabi.lib().afsk_rx_plan_set_option(rx._cache[1].plan, _cabi.OPT_FUSED, 2))
            b2 = rx.decode_batch(caps, baud_rate=bd, amp_end_threshold=th)
            assert np.array_equal(b.results, b2.results) and b.payloads() == b2.payloads()
            _assert_equals_oracle(b2, caps, bd, th)
    finally:
        os.environ.pop("AFSK_FUSED")
        rx.close()


@pytest.mark.parametrize("variant", [1, 2])
@pytest.mark.parametrize("baud", [6000, 1200, 300, 2400, 4000, 1500, 800, 3000, 2000])
def test_clock_kernel_variant_2(baud, variant):
    """k_clock for every bit length (AFSK_OPT_CLOCK_KERNEL = 1; the default sends 6000..2000 baud through k_clock_q) and
    k_clock2 (= 2): the one-sweep clock search as a kernel of its own == oracle."""
    rng = np.random.default_rng([61, baud])
    bf = 48000 // baud
    caps = []
    for i in range(40):
        fr = O.tx_frames(rng.integers(0, 256, 12, dtype=np.uint8).tobytes(), baud, 0.2)
        x = np.concatenate([np.zeros(int(rng.integers(0, 2 * bf + 40)), np.int16), fr]).astype(np.int32)
        if i % 2:
            x = x + np.round(rng.normal(0, float(rng.choice([4000, 15000, 30000])), len(x))).astype(np.int32)
        caps.append(np.clip(x, -32768, 32767).astype(np.int16))
    caps.append(np.zeros(3000, np.int16))
    b = np.full(len(caps), baud, np.int32)
    thr = np.full(len(caps), 14000, np.int32)
    samples, offsets = A.modem._concat(caps)
    s = A.RxSession(offsets, b, thr)
    _cabi.check(_cabi.lib().afsk_rx_plan_set_option(s.plan, _cabi.OPT_CLOCK_KERNEL, variant))
    s.upload(samples); s.run()
    _assert_equals_oracle(s.download(), caps, b, thr)
    s.close()


@pytest.mark.parametrize("baud", [6000, 4000, 3000, 2400, 2000])
def test_clock_q_every_start_alignment(baud):
    """k_clock_q (the default at 6000..2000 baud): every capture start modulo 8 samples, lead-ins that put the first minimum
    near both ends of the candidate range, noise-only and constant captures; mixed with a 1200-baud capture and a short
    one so that k_clock runs beside it on the rest of the batch."""
    rng = np.random.default_rng([67, baud])
    bf = 48000 // baud
    caps, bd = [], []
    for i in range(64):
        fr = O.tx_frames(rng.integers(0, 256, 12, dtype=np.uint8).tobytes(), baud, 0.1)
        lead = int(rng.choice([0, 1, bf - 1, 2 * bf + 7, 4096 - 2 * bf - 1, 4096 - 2 * bf, 4090])) if i % 4 == 0 else int(rng.integers(0, 64))
        x = np.concatenate([np.zeros(lead, np.int16), fr]).astype(np.int32)
        if i % 3 == 1:
            x = x + np.round(rng.normal(0, float(rng.choice([4000, 15000, 30000])), len(x))).astype(np.int32)
        if i % 16 == 5:
            x = np.round(rng.normal(0, 12000, len(x))).astype(np.int32)
        if i == 40:
            x = np.full(4500, -32768, np.int32)
        if i == 41:
            x = np.full(4500, 32767, np.int32)
        x = np.clip(x, -32768, 32767).astype(np.int16)
        caps.append(x[:len(x) - int(rng.integers(0, 8))])        # lengths of every residue: the next start moves
        bd.append(baud)
    caps.insert(7, O.tx_frames(b"beside", 1200, 0.1)); bd.insert(7, 1200)
    caps.insert(9, np.zeros(3000, np.int16)); bd.insert(9, baud)
    b = np.array(bd, np.int32)
    thr = np.full(len(caps), 14000, np.int32)
    samples, offsets = A.modem._concat(caps)
    assert len({int(o) % 8 for o in offsets[:-1]}) == 8
    s = A.RxSession(offsets, b, thr)
    s.upload(samples); s.run()
    got = s.download()
    _assert_equals_oracle(got, caps, b, thr)
    _cabi.check(_cabi.lib().afsk_rx_plan_set_option(s.plan, _cabi.OPT_CLOCK_KERNEL, 1))
    s.run()
    ref = s.download()
    assert np.array_equal(got.results, ref.results) and got.payloads() == ref.payloads()
    s.close()
