"""A plain reference of every demodulated window, and generators of the windows where demodulators go wrong (CPU).

``ref_planes`` decides every window of a capture from the reference's rules, written out directly in int64 numpy:
__amplify (afskmodem.py:287-296: > 512 -> 32767, < -512 -> -32768, else 0), getDiff as a floored mean (:101-107),
bit = mark_diff < space_diff (:346-351) and quiet = getAmplitude(chunk) < amp_end (:94-98, :375).  It covers the
windows k with clock + k * bf < n - bf, those the reference's loops visit (:362, :372).  tests/test_gpu_demod_planes.py
compares the GPU's bit and quiet planes with it, window by window, over every demodulator layout and the streaming
receiver.

The generators craft the windows the end-to-end results cannot see into:
  * tie windows: quarters 1 and 2 carry equal c = p - n sums, so the mark and space correlations tie (Um == Us).
    Classes, named by the closed forms of test_demod_algebra_model.py: C1 Um != Us; C2 Um == Us, Ns <= Nm (a 0 without
    looking at the floors); C3 / C4 Um == Us, Ns > Nm with bit 1 / 0 (the floors decide: tie_bit in afsk_rx.cu).
    Ns > Nm comes from (+x, -x) pairs in quarter 1 against sub-limiter samples in quarter 2.  Some bit lengths lack a
    class (tie_classes works them out from the closed forms): at 4 samples per bit a tie has Ns == Nm (no C3 / C4), at
    8 and at several power-of-two multiples a tie with Ns > Nm is always a 0 (no C3).
  * quiet-edge windows: sum|x| is exactly thr * bf (E0, not quiet) or thr * bf - 1 (E1, quiet), -32768 samples among
    them, the end detector's boundary in the kernels' form sum|x| < thr * bf.
  * limiter-edge soup: +-511, +-512, +-513, +-514 and full scale.
``demod_batch`` puts them into captures: a real transmission for the first 4096 frames (clock recovery reads only
those, so the oracle's clock is known before crafting), then whole windows aligned to that clock."""
import functools
import itertools

import numpy as np
import pytest

from oracle import oracle as O
from test_demod_algebra_model import reference_bit
from test_gpu_stream_oracle import DEMOD_BAUDS

HI, LO = 32767, -32768
SYNC = 4096                                   # frames clock recovery reads
N_CLASS = 8                                   # windows of each class per bit length a test must see


def bit_frames(baud: int) -> int:
    return int(48000 / baud)                  # Receiver.__bit_frames :277


@functools.lru_cache(maxsize=None)
def _tones(baud: int):
    return O.tone("mark", baud).astype(np.int64), O.tone("space", baud).astype(np.int64)


def n_windows(n: int, bf: int, clock: int) -> int:
    """#{k >= 0 : clock + k * bf < n - bf}"""
    span = n - bf - clock
    return 0 if span <= 0 else -(-span // bf)


def _windows(x, bf, clock):
    K = n_windows(len(x), bf, clock)
    return np.asarray(x[clock:clock + K * bf], dtype=np.int64).reshape(K, bf)


def ref_planes(x, baud: int, clock: int, amp_end: int):
    """(bits, quiet) bool arrays of every window of x at clock, by the reference's rules"""
    return _decide(_windows(x, bit_frames(baud), clock), baud, amp_end)


def _decide(W, baud, amp_end):
    bf = bit_frames(baud)
    mark, space = _tones(baud)
    amp = np.where(W > 512, HI, np.where(W < -512, LO, 0))                         # __amplify
    mark_diff = np.abs(mark - amp).sum(axis=1) // bf                              # getDiff: int(total / n), total >= 0
    space_diff = np.abs(space - amp).sum(axis=1) // bf
    quiet = np.abs(W).sum(axis=1) // bf < amp_end                                 # getAmplitude(chunk) < amp_end
    return mark_diff < space_diff, quiet


def frame(bits, quiet, clock: int, bf: int):
    """the reference's framing over decided windows (:361-380): (train_end, coded bits)"""
    k0 = len(bits)
    for k in range(3, len(bits)):
        if bits[k - 3] and not bits[k - 2] and not bits[k - 1] and not bits[k]:
            k0 = k + 1
            break
    q = np.flatnonzero(quiet[k0:])
    k1 = k0 + int(q[0]) if len(q) else len(bits)
    return clock + k0 * bf, bits[k0:k1].astype(np.uint8)


# ---------------------------------------------------------------- window classes ----------------------------------

CLASSES = ("C1", "C2", "C3", "C4", "E0", "E1")


def window_classes(x, baud: int, clock: int, amp_end: int, lo: int = 0, hi: int | None = None) -> dict:
    """counts of each class among windows lo .. hi - 1 of x at clock"""
    bf, q = bit_frames(baud), bit_frames(baud) // 4
    W = _windows(x, bf, clock)[lo:hi]
    p, n = (W > 512).astype(np.int64), (W < -512).astype(np.int64)
    quarter = np.arange(bf) // q
    Tm, Ts = np.where(quarter % 2 == 0, 1, -1), np.where(quarter < 2, 1, -1)
    Um, Us, Nm, Ns = (p - n) @ Tm, (p - n) @ Ts, n @ Tm, n @ Ts
    bits, _ = _decide(W, baud, amp_end)
    tie, floors = Um == Us, Ns > Nm
    a = np.abs(W).sum(axis=1)
    return {"C1": int((~tie).sum()), "C2": int((tie & ~floors).sum()), "C3": int((tie & floors & bits).sum()),
            "C4": int((tie & floors & ~bits).sum()), "E0": int((a == amp_end * bf).sum()), "E1": int((a == amp_end * bf - 1).sum())}


P_VALS = [513, 514, 600, 12000, 32767]
N_VALS = [-513, -514, -600, -12000, -32767, -32768]
Z_VALS = [-512, -511, -1, 0, 1, 511, 512]
SOUP = [-32768, -32767, -514, -513, -512, -511, 0, 511, 512, 513, 514, 32767]


def _samples(cls, rng):
    """limiter classes 0 (|x| <= 512), 1 (x > 512), 2 (x < -512) -> samples at and around the limiter edges"""
    out = np.empty(len(cls), np.int64)
    for k, vals in enumerate((Z_VALS, P_VALS, N_VALS)):
        m = cls == k
        out[m] = rng.choice(vals, int(m.sum()))
    return out


def _quarter(p: int, n: int, q: int, rng):
    return rng.permutation(np.repeat([1, 2, 0], [p, n, q - p - n]))


def tie_window(bf: int, rng, floors: bool, want_bit: int = 0):
    """Um == Us: quarter 2 holds quarter 1's limiter classes reshuffled, and d (+x, -x) pairs in quarter 1 against 2d
    sub-limiter samples in quarter 2 (Ns - Nm = 2d).  Without floors the pairs go to quarter 2 (or d = 0).  With floors
    (d >= 1) the bit is 1 iff M mod bf >= bf - 2d, M = 65535 bf / 2 - 32767 Um + Nm: drawn counts of quarters 0 and 3
    and d are rejected until that gives want_bit."""
    q = bf // 4
    cls = rng.integers(0, 3, bf)
    d = int(rng.integers(0, q // 2 + 1))
    if floors:
        for _ in range(64):
            N = 4096
            n0, n3 = rng.integers(0, q + 1, N), rng.integers(0, q + 1, N)
            p0, p3 = (rng.random(N) * (q - n0 + 1)).astype(np.int64), (rng.random(N) * (q - n3 + 1)).astype(np.int64)
            dd = rng.integers(1, q // 2 + 1, N)
            M = 65535 * bf // 2 - 32767 * ((p0 - n0) - (p3 - n3)) + (n0 - n3 - dd)
            ok = np.flatnonzero((M % bf >= bf - 2 * dd) == bool(want_bit))
            if len(ok):
                i = int(ok[0])
                d = int(dd[i])
                cls[:q], cls[3 * q:] = _quarter(int(p0[i]), int(n0[i]), q, rng), _quarter(int(p3[i]), int(n3[i]), q, rng)
                break
        else:
            raise AssertionError(f"no tie window with Ns > Nm decides {want_bit} at {bf} samples per bit")
    base = cls[q:2 * q - 2 * d].copy()
    pairs = np.concatenate([base, np.repeat([1, 2], d)])
    plain = np.concatenate([rng.permutation(base), np.zeros(2 * d, np.int64)])
    a, b = (pairs, plain) if floors else (plain, pairs)
    cls[q:2 * q], cls[2 * q:3 * q] = rng.permutation(a), rng.permutation(b)
    return _samples(cls, rng)


def abs_sum_window(bf: int, total: int, rng):
    """bf samples with sum|x| == total (0 <= total <= 32768 bf), some of them -32768 where the total allows"""
    k = int(rng.integers(0, min(bf, total // 32768) + 1))
    while total - 32768 * k > 32767 * (bf - k):
        k += 1
    rest, n = total - 32768 * k, bf - k
    a = np.zeros(n, np.int64)
    if n:
        w = rng.random(n) ** 3 + 1e-9
        a = np.minimum(np.floor(w / w.sum() * rest).astype(np.int64), 32767)
        r = rest - int(a.sum())
        for i in rng.permutation(n):
            if r == 0:
                break
            d = min(32767 - int(a[i]), r)
            a[i] += d
            r -= d
    x = np.concatenate([np.full(k, LO, np.int64), np.where(rng.random(n) < 0.5, -a, a)])
    return rng.permutation(x)


def class_window(cls: str, baud: int, amp_end: int, rng):
    """one window of class cls"""
    bf = bit_frames(baud)
    if cls in ("E0", "E1"):
        return abs_sum_window(bf, amp_end * bf - (cls == "E1"), rng)
    if cls == "C1":
        return rng.choice(SOUP, bf).astype(np.int64)
    return tie_window(bf, rng, floors=cls != "C2", want_bit=int(cls == "C3"))


def edge_classes(amp_end: int, bf: int):
    """the quiet-edge classes a threshold has (sum|x| ranges over 0 .. 32768 bf)"""
    return [c for c, t in (("E0", amp_end * bf), ("E1", amp_end * bf - 1)) if 0 <= t <= 32768 * bf]


def tie_classes(bf: int):
    """the classes windows of bf samples can fall in.  A tie with Ns > Nm needs 1 <= d = (Ns - Nm) / 2 <= q / 2 (q =
    bf / 4) and is a 1 iff M mod bf >= bf - 2d; M mod bf runs over the residues of 65535 bf / 2 + (-32767 c0 + n0) +
    (32767 c3 - n3) - d, (c, n) = (p - n, n) of quarters 0 and 3."""
    q = bf // 4
    if q < 2:
        return ["C1", "C2"]
    n = np.concatenate([np.full(q + 1 - k, k) for k in range(q + 1)])
    c = np.concatenate([np.arange(q + 1 - k) for k in range(q + 1)]) - n
    U0, U3 = np.unique((-32767 * c + n) % bf), np.unique((32767 * c - n) % bf)
    R = np.unique((65535 * bf // 2 + U0[:, None] + U3[None, :]) % bf)
    d = np.arange(1, q // 2 + 1)
    one = (R[:, None] - d[None, :]) % bf >= bf - 2 * d[None, :]
    return ["C1", "C2"] + ["C3"] * bool(one.any()) + ["C4"] * bool((~one).any())


# ---------------------------------------------------------------- captures ----------------------------------------

# thresholds: those with quiet edges, and the ones the host clamps to [0, 65537] before it forms the int32 thr * bf
EDGE_THRS = [14000, 1, 32768]
OTHER_THRS = [0, 70000, -5, -2 ** 31, 2 ** 31 - 1]
PER_CLASS = 6                                 # crafted windows of each class per capture


def tile_windows(bf: int) -> int:
    """windows per demodulator tile of the default layout (afsk_rx.cu configure_group, Group::wt); for bits longer
    than 48 frames outside the shift and padded layouts an upper bound (very long bits may drop to one sub-tile)"""
    if bf in (8, 16, 24):
        return 256 * {8: 8, 16: 4, 24: 2}[bf]
    if bf in (4, 12, 20, 60, 100, 120, 200):
        wpt = {4: 8, 12: 4, 20: 2, 60: 2, 100: 2, 120: 1, 200: 1}[bf]
        return (1 if bf >= 60 else 2) * 256 * wpt
    if bf in (32, 64, 128):
        return 256 * (128 // bf)
    tpw = 1
    while bf // tpw > 48 and tpw < 8:
        tpw *= 2
    return 2 * 256 // tpw


def crafted_capture(baud: int, amp_end: int, K: int, rng):
    """-> (x, clock): the first SYNC frames of a transmission (its clock is the oracle's), then K windows in all:
    limiter soup and noisy tones with PER_CLASS windows of every class this bit length and threshold have at random
    window positions from frame SYNC on; 1 .. bf frames after window K - 1"""
    bf = bit_frames(baud)
    tx = O.tx_frames(b"\x5a", baud, 0.5)
    lead = int(rng.integers(0, 2 * bf))
    head = np.clip(tx[lead:lead + SYNC].astype(np.float64) + rng.normal(0, 3000, SYNC), LO, HI).astype(np.int64)
    clock = O.rx_decode(head.astype(np.int16), baud, amp_end)["clock"]
    k0 = -(-(SYNC - clock) // bf)
    assert K > k0 + PER_CLASS * 6, (baud, K)
    n = clock + K * bf + int(rng.integers(1, bf + 1))
    x = rng.choice(SOUP, n).astype(np.int64)
    x[:SYNC] = head
    mark, space = _tones(baud)
    tones = np.where(rng.random((K, 1)) < 0.5, mark, space) * rng.choice([1.0, 0.3, 0.02], (K, 1))
    noisy = np.clip(np.round(tones + rng.normal(0, 9000, (K, bf))), LO, HI).astype(np.int64)
    W = x[clock:clock + K * bf].reshape(K, bf)
    pick = rng.random(K) < 0.5
    pick[:k0] = False
    W[pick] = noisy[pick]
    cls = tie_classes(bf) + edge_classes(amp_end, bf)
    at = rng.choice(np.arange(k0, K), PER_CLASS * len(cls), replace=False)
    for i, k in enumerate(at):
        W[k] = class_window(cls[i % len(cls)], baud, amp_end, rng)
    return x.astype(np.int16), clock


@functools.lru_cache(maxsize=1)
def demod_batch(seed: int = 9100):
    """A mixed-baud batch over DEMOD_BAUDS.  Per baud (4800 aside: plain transmissions, which the reference rejects)
    four crafted captures: two over three tiles, two short ones; two thresholds with quiet edges, two among the clamped
    ones.  Window counts run over every residue mod 32 and capture starts over every residue mod 8 (spacer captures
    of 0-7 frames in between), in shuffled order.  -> (captures, bauds, thresholds, clocks (-1: none crafted))"""
    rng = np.random.default_rng(seed)
    jobs = []
    for i, baud in enumerate(DEMOD_BAUDS):
        if bit_frames(baud) % 4:
            for j in range(2):
                jobs.append((baud, EDGE_THRS[j], None))
            continue
        bf = bit_frames(baud)
        k0 = -(-SYNC // bf)
        for j in range(4):
            r = (4 * i + j) % 32
            K = (2 * tile_windows(bf) + 32 if j < 2 else -(-(k0 + 64) // 32) * 32) + r
            thr = EDGE_THRS[(i + j) % 3] if j % 2 == 0 else OTHER_THRS[(2 * i + j) % 5]
            jobs.append((baud, thr, K))
    caps, bauds, thrs, clocks = [], [], [], []
    pos = 0
    for t, idx in enumerate(rng.permutation(len(jobs))):
        baud, thr, K = jobs[idx]
        gap = (t % 8 - pos) % 8
        caps.append(np.zeros(gap, np.int16))
        bauds.append(1200)
        thrs.append(14000)
        clocks.append(-1)
        pos += gap
        if K is None:
            x, clk = O.tx_frames(rng.integers(0, 256, 20, dtype=np.uint8).tobytes(), baud, 0.1), -1
        else:
            x, clk = crafted_capture(baud, thr, K, rng)
        caps.append(x)
        bauds.append(baud)
        thrs.append(thr)
        clocks.append(clk)
        pos += len(x)
    return caps, bauds, thrs, clocks


def batch_starts(caps):
    return np.concatenate([[0], np.cumsum([len(x) for x in caps])])[:-1]


# ---------------------------------------------------------------- self-checks ------------------------------------

@pytest.mark.parametrize("baud", DEMOD_BAUDS)
def test_ref_planes_frame_to_the_oracles_decode(baud):
    """over seeded transmissions (noise, gain, lead silence, truncation, thresholds): the reference's framing of
    ref_planes is the oracle's train_end, coded bits and "No data."; at 4800 baud the oracle finds no clock"""
    rng = np.random.default_rng([11, baud])
    bf = bit_frames(baud)
    seen = set()
    for k in range(8 if baud >= 300 else 3):
        tt = float(rng.choice([0.5, 0.1, 0.05])) if baud >= 300 else 2.0
        fr = O.tx_frames(rng.integers(0, 256, int(rng.integers(1, 24)), dtype=np.uint8).tobytes(), baud, tt)
        x = np.concatenate([np.zeros(int(rng.integers(0, 5000)), np.int64), fr.astype(np.int64)])
        x = x * float(rng.choice([1.0, 0.6, 0.3])) + rng.normal(0, float(rng.choice([0, 3000, 9000, 16000])), len(x))
        x = np.clip(np.trunc(x), LO, HI).astype(np.int16)
        if k % 3 == 2:
            x = x[:int(rng.integers(SYNC, len(x)))]
        thr = int(rng.choice([14000, 8000, 11000]))
        o = O.rx_decode(x, baud, thr, want_bits=True)
        if bf % 4:
            assert o["status"] == O.ST_EXC_WAVELEN
            continue
        assert o["clock"] >= 0, (baud, k)
        bits, quiet = ref_planes(x, baud, o["clock"], thr)
        train_end, coded = frame(bits, quiet, o["clock"], bf)
        assert train_end == o["train_end"] and np.array_equal(coded, o["bits"]), (baud, k)
        assert (o["status"] == O.ST_NO_DATA) == (len(coded) == 0)
        seen.add(o["status"])
    assert bf % 4 or O.ST_OK in seen or baud == 12000


@pytest.mark.parametrize("baud", [b for b in DEMOD_BAUDS if bit_frames(b) % 4 == 0])
def test_ref_planes_equal_the_window_rule_on_sampled_windows(baud):
    """the crafted captures' windows: ref_planes against reference_bit (test_demod_algebra_model.py) and the
    oracle's getAmplitude, window by window"""
    caps, bauds, thrs, clocks = demod_batch()
    rng = np.random.default_rng([12, baud])
    bf = bit_frames(baud)
    for x, b, thr, clk in zip(caps, bauds, thrs, clocks):
        if b != baud or clk < 0:
            continue
        bits, quiet = ref_planes(x, baud, clk, thr)
        for k in rng.choice(len(bits), min(len(bits), 150), replace=False):
            w = x[clk + k * bf:clk + (k + 1) * bf]
            assert bits[k] == reference_bit(w.astype(np.int64), bf), (baud, k)
            assert quiet[k] == (O.amplitude(w) < thr), (baud, k)


def test_generators_reach_their_quotas():
    """every class at every bit length; residues of window counts mod 32 and of capture starts mod 8; the long
    captures over three tiles; each tie window of a class is what its name says"""
    caps, bauds, thrs, clocks = demod_batch()
    starts = batch_starts(caps)
    per_bf, residues, aligns = {}, set(), set()
    for x, b, thr, clk, s0 in zip(caps, bauds, thrs, clocks, starts):
        if clk < 0:
            continue
        bf = bit_frames(b)
        K = n_windows(len(x), bf, clk)
        residues.add(K % 32)
        aligns.add(int(s0) % 8)
        cnt = per_bf.setdefault(bf, dict.fromkeys(CLASSES, 0))
        for c, v in window_classes(x, b, clk, thr).items():
            cnt[c] += v
        per_bf.setdefault(("tiles", bf), []).append(-(-K // tile_windows(bf)))
    assert residues == set(range(32)) and aligns == set(range(8))
    assert {bit_frames(b) for b in DEMOD_BAUDS if bit_frames(b) % 4 == 0} == {k for k in per_bf if isinstance(k, int)}
    for bf, cnt in per_bf.items():
        if isinstance(bf, tuple):
            assert max(cnt) >= 3, bf
            continue
        for c in tie_classes(bf) + ["E0", "E1"]:
            assert cnt[c] >= N_CLASS, (bf, c, cnt)

@pytest.mark.parametrize("bf", [4, 8, 12])
def test_tie_classes_of_short_bits_over_every_limiter_pattern(bf):
    """every limiter pattern of a window (a sample counts only as > 512, < -512 or neither): the classes that exist are
    tie_classes(bf)"""
    cls = np.array(list(itertools.product(range(3), repeat=bf)))
    x = np.choose(cls, [0, 600, -600])
    q = bf // 4
    quarter = np.arange(bf) // q
    p, n = (cls == 1).astype(np.int64), (cls == 2).astype(np.int64)
    Um, Us = (p - n) @ np.where(quarter % 2 == 0, 1, -1), (p - n) @ np.where(quarter < 2, 1, -1)
    Nm, Ns = n @ np.where(quarter % 2 == 0, 1, -1), n @ np.where(quarter < 2, 1, -1)
    bits, _ = _decide(x, 48000 // bf, 14000)
    tie, floors = Um == Us, Ns > Nm
    have = {"C1": (~tie).any(), "C2": (tie & ~floors).any(), "C3": (tie & floors & bits).any(), "C4": (tie & floors & ~bits).any()}
    assert [c for c in ("C1", "C2", "C3", "C4") if have[c]] == tie_classes(bf)


@pytest.mark.parametrize("bf", [4, 8, 40, 2000])
def test_quiet_edge_windows_sit_on_the_threshold(bf):
    rng = np.random.default_rng(bf)
    for thr in EDGE_THRS + [0]:
        for cls in edge_classes(thr, bf):
            x = abs_sum_window(bf, thr * bf - (cls == "E1"), rng)
            assert len(x) == bf and x.min() >= LO and x.max() <= HI
            assert int(np.abs(x).sum()) == thr * bf - (cls == "E1")
            assert (O.amplitude(x.astype(np.int16)) < thr) == (cls == "E1")
    assert (abs_sum_window(bf, 32768 * bf - 1, rng) == LO).sum() == bf - 1
