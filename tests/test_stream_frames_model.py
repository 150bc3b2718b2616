"""CPU model of the windowed, multi-format interleaved kernels, restated from the CUDA source, and of the sample-format
rules of afsk_b200.h (no GPU needed):

  * k_stream_frames<Tin> (afsk_rx.cu): frame f of channel s is element e0 + f * pitch + s of a 16-byte aligned
    buffer (e0: the window's offset in its first vector).  Rows are loaded as aligned 16-byte vectors (8 lanes of 8
    samples for 16-bit, 16 lanes of 4 samples for 32-bit), realigned, converted to int16, and appended through the
    shared tile to each channel's slot.  Checked against a plain slice, conversion and append, with neighbouring
    slots untouched and no vector loaded that holds no window sample.
  * k_tx_window_frames<Tout> (afsk_tx.cu): the frame-major store half into a window of a wider buffer, from the
    row's absolute alignment, checked against the converted transpose of the planar window, with every element
    outside the window untouched.
  * sample_to_s16 / sample_from_s16 at the edges of each format, against the numpy statements of the rules.
"""
import numpy as np
import pytest

from test_stream_interleaved_model import HALO, IL_C, IL_STRIDE, IL_V, KC, KF, POISON, STRIDE, shared_row, slots

FORMATS = [np.int16, np.int32, np.float32]
PITCH_EXTRA = [0, 1, 7, 67]


# ---------------------------------------------------------------- the conversion rules, as numpy statements ----
def rule_to_s16(x: np.ndarray) -> np.ndarray:
    if x.dtype == np.int16:
        return x.copy()
    if x.dtype == np.int32:
        return (x >> 16).astype(np.int16)
    return np.clip(np.rint(np.nan_to_num(x, nan=0.0).astype(np.float64) * 32768), -32768, 32767).astype(np.int16)


def rule_from_s16(s: np.ndarray, dtype) -> np.ndarray:
    if dtype == np.int16:
        return s.astype(np.int16)
    if dtype == np.int32:
        return s.astype(np.int32) << 16
    return (s.astype(np.float32) / np.float32(32768)).astype(np.float32)


# ------------------------------------------------- the kernels' element operations (afsk_common.cuh) ----
def kernel_to_s16(x: np.ndarray) -> np.ndarray:
    """sample_to_s16: int32 >> 16; float: __float2int_rn(x * 32768.f) (round half to even, NaN -> 0, saturating to
    int32), then the clamp"""
    if x.dtype == np.int16:
        return x.copy()
    if x.dtype == np.int32:
        return (x >> np.int32(16)).astype(np.int16)
    y = (x.astype(np.float32) * np.float32(32768)).astype(np.float64)       # exact: a power of two
    r = np.rint(np.where(np.isnan(y), 0.0, y))
    r = np.clip(r, -2.0 ** 31, 2.0 ** 31 - 1).astype(np.int64)             # cvt.rni.s32.f32 saturates
    return np.minimum(np.maximum(r, -32768), 32767).astype(np.int16)


def kernel_from_s16(s: np.ndarray, dtype) -> np.ndarray:
    """sample_from_s16: (uint32)s << 16, s * (1 / 32768.f)"""
    if dtype == np.int16:
        return s.astype(np.int16)
    if dtype == np.int32:
        return ((s.astype(np.int32).view(np.uint32) << np.uint32(16))).view(np.int32)
    return (s.astype(np.float32) * np.float32(1.0 / 32768.0)).astype(np.float32)


def same_bits(a, b):
    return np.array_equal(np.ascontiguousarray(a).view(np.uint8), np.ascontiguousarray(b).view(np.uint8))


# ----------------------------------------------------------------------------- receive ----
def k_stream_frames(buf, e0, pitch, n, S, seg_dst, arena, window_vectors):
    """One launch: buf is the whole 16-byte aligned buffer (its dtype: Tin), the window's frame f of channel s at
    element e0 + f * pitch + s.  Appends to arena through the shared tile, as the kernel does."""
    V = 16 // buf.dtype.itemsize
    L = KC // V
    assert e0 < V
    vecs = buf.reshape(-1, V)                                   # aligned 16-byte vectors
    cblocks, ftiles = -(-S // KC), (n + KF + HALO - 1) // KF
    for b in range(cblocks * ftiles):
        cb, fb = b % cblocks, b // cblocks
        c0, F0 = cb * KC, fb * KF
        nc = min(KC, S - c0)
        sd = seg_dst[c0:c0 + nc]
        T = np.full((KC, STRIDE), POISON, np.int64)
        f_lo, f_hi = max(F0 - HALO, 0), min(F0 + KF, n)
        f = np.arange(f_lo, f_hi)[:, None]
        q = np.arange(L)[None, :]
        q = q[:, :(nc + V - 1) // V]
        row = e0 + f * pitch + c0
        row_end = row + nc
        qs = row + V * q
        sv, k = qs // V, qs % V
        hi_ok = (k != 0) & ((sv + 1) * V < row_end)
        loaded = np.concatenate([sv.reshape(-1), (sv + 1)[hi_ok]])
        assert np.isin(loaded, window_vectors).all()            # only vectors holding window samples
        lo = vecs[sv]
        hi = np.where(hi_ok[..., None], vecs[np.where(hi_ok, sv + 1, 0)], 0)
        w = np.concatenate([lo, hi], -1)                        # (rows, nq, 2V) samples
        vals = np.take_along_axis(w, k[..., None] + np.arange(V), -1)
        vals = kernel_to_s16(vals.reshape(-1)).reshape(vals.shape).astype(np.int64)
        c = np.broadcast_to(V * q[..., None] + np.arange(V), vals.shape)
        cc = np.where(c < nc, c, 0)
        p = f[..., None] - F0 + (sd[cc] & 7)
        ok = (c < nc) & (p >= 0) & (p < KF)
        T[shared_row(cc[ok]), p[ok]] = vals[ok]
        # store half: that of k_stream_deinterleave
        c = np.arange(nc)[:, None]
        jv = np.arange(KF // 8)[None, :]
        g = sd[c]
        d0 = (g >> 3) * 8 + F0 + 8 * jv
        f0 = d0 - g
        e = np.arange(8)
        fe = f0[..., None] + e
        m = (f0 < n)[..., None] & (fe >= 0) & (fe < n)
        v = T[shared_row(c)[..., None], 8 * jv[..., None] + e]
        assert (v[m] != POISON).all()
        arena[(d0[..., None] + e)[m]] = v[m]


def card(rng, dtype, size):
    if dtype == np.float32:
        x = rng.uniform(-1.2, 1.2, size).astype(np.float32)
        x[rng.random(size) < 0.02] = np.nan
        return x
    info = np.iinfo(dtype)
    return rng.integers(info.min, info.max, size, dtype=dtype, endpoint=True)


def window_vectors(e_base, pitch, n, S, V):
    r = e_base + np.arange(n)[:, None] * pitch + np.arange(S)[None, :]
    return np.unique(r // V)


@pytest.mark.parametrize("dtype", FORMATS)
@pytest.mark.parametrize("S", [1, 2, 3, 4, 5, 6, 7, 8, 63, 64, 65, 71, 72, 130])
def test_deinterleave_window_equals_slice_convert_append(S, dtype):
    rng = np.random.default_rng(S * 7 + FORMATS.index(dtype))
    V = 16 // np.dtype(dtype).itemsize
    for n in [1, 7, 9, 128, 129, 300]:
        for extra in PITCH_EXTRA:
            pitch = S + extra
            for e0 in range(V):                                 # every window alignment mod 16 bytes
                col = int(rng.integers(0, extra + 1))           # the window's first column in the card
                e_base = e0 + V * -(-col // V)                  # its first element: e0 mod V, rows start at e_base - col
                total = e_base - col + n * pitch + 2 * V
                total += (-total) % V
                buf = card(rng, dtype, total)
                before = buf.copy()
                win = np.lib.stride_tricks.as_strided(buf[e_base:], shape=(n, S), strides=(pitch * buf.itemsize, buf.itemsize))
                want_x = rule_to_s16(np.array(win))
                dst, size = slots(S, n, rng, rng.integers(0, 8, S))
                arena = rng.integers(-32768, 32768, size, dtype=np.int16).astype(np.int64)
                want = arena.copy()
                for s in range(S):
                    want[dst[s]:dst[s] + n] = want_x[:, s]
                base = buf[e_base - e0:]                        # the 16-byte vector holding the window's first sample
                k_stream_frames(base, e0, pitch, n, S, dst, arena, window_vectors(e0, pitch, n, S, V))
                np.testing.assert_array_equal(arena, want, err_msg=f"S={S} n={n} pitch={pitch} e0={e0} {dtype}")
                assert same_bits(buf, before)


# ---------------------------------------------------------------------------- transmit ----
def k_tx_window_frames(W, S, n, out, e0, pitch):
    """W: the planar int16 window (S, n); out: the 16-byte aligned output buffer (its dtype: Tout), frame f of
    channel s written at element e0 + f * pitch + s"""
    V = 16 // out.dtype.itemsize
    NV = IL_C // V + 1
    cblocks, ftiles = -(-S // IL_C), (n + 8 * IL_V - 1) // (8 * IL_V)
    for b in range(cblocks * ftiles):
        cb, fb = b % cblocks, b // cblocks
        c0, F0 = cb * IL_C, fb * 8 * IL_V
        nc, nf = min(IL_C, S - c0), min(8 * IL_V, n - F0)
        T = np.full((IL_C, IL_STRIDE), POISON, np.int64)
        for c in range(nc):
            for col in range(0, nf, 8):
                m = min(8, nf - col)
                vec = np.zeros(8, np.int64)
                vec[:m] = W[c0 + c, F0 + col:F0 + col + m]
                T[shared_row(c), col:col + 8] = vec
        i = np.arange(nf * NV)
        q, fl = i % NV, i // NV
        a = e0 + (F0 + fl) * pitch + c0
        bnd = a + nc
        d0 = (a // V + q) * V
        live = d0 < bnd
        e = np.arange(V)
        cidx = d0[:, None] + e - a[:, None]
        m = live[:, None] & (cidx >= 0) & (cidx < nc)
        v = T[shared_row(np.where(m, cidx, 0)), fl[:, None]]
        assert (v[m] != POISON).all()
        is_full = live & (d0 >= a) & (d0 + V <= bnd)
        assert (d0[is_full] % V == 0).all() and m[is_full].all()
        assert (np.bincount(fl[live & ~is_full], minlength=nf) <= 2).all()     # only a row's head and tail
        vals = kernel_from_s16(v[m].astype(np.int16), out.dtype.type)
        out[(d0[:, None] + e)[m]] = vals


@pytest.mark.parametrize("dtype", FORMATS)
@pytest.mark.parametrize("S", [1, 2, 3, 4, 5, 6, 7, 8, 63, 64, 65, 71, 130])
def test_tx_window_writes_only_the_window(S, dtype):
    rng = np.random.default_rng(300 + S * 3 + FORMATS.index(dtype))
    V = 16 // np.dtype(dtype).itemsize
    sentinel = {np.int16: 0x5A5A, np.int32: 0x5A5A5A5A, np.float32: np.float32(1234.5)}[dtype]
    for n in [1, 7, 9, 127, 128, 129, 300]:
        W = rng.integers(-32768, 32768, size=(S, n), dtype=np.int16)
        for extra in PITCH_EXTRA:
            pitch = S + extra
            for e0 in range(V):
                col = int(rng.integers(0, extra + 1))
                e_base = e0 + V * (1 + -(-col // V))            # the window's first element, e0 mod V
                total = e_base - col + n * pitch + 3 * V
                total += (-total) % V
                out = np.full(total, sentinel, dtype)
                k_tx_window_frames(W, S, n, out, e_base, pitch)
                want = np.full(total, sentinel, dtype)
                idx = e_base + np.arange(n)[:, None] * pitch + np.arange(S)[None, :]
                want[idx] = rule_from_s16(W.T, dtype)
                assert same_bits(out, want), (S, n, pitch, e0, dtype)


# ------------------------------------------------------------------------------- rules ----
def test_receive_rules_at_the_edges():
    f = np.array([0.0, -0.0, 1.0, -1.0, 0.5 / 32768, -0.5 / 32768, 1.5 / 32768, -1.5 / 32768, 2.5 / 32768,
                  32767.5 / 32768, -32768.5 / 32768, 1.0001, -1.0001, 3.0, -3.0, 1e30, -1e30, np.inf, -np.inf, np.nan,
                  -np.nan, 32767 / 32768, -32768 / 32768, 1e-45, -1e-45, 0.99999994], np.float32)
    want_f = np.array([0, 0, 32767, -32768, 0, 0, 2, -2, 2, 32767, -32768, 32767, -32768, 32767, -32768, 32767, -32768,
                       32767, -32768, 0, 0, 32767, -32768, 0, 0, 32767], np.int16)
    assert np.array_equal(rule_to_s16(f), want_f)
    assert np.array_equal(kernel_to_s16(f), want_f)
    i = np.array([0, -1, 1, 0x7FFFFFFF, -0x80000000, 0xFFFF, 0x10000, -0x10000, -0x10001, -0xFFFF, 0x7FFF0000,
                  -0x7FFFFFFF, 0x12345678, -0x12345678], np.int32)
    want_i = np.array([0, -1, 0, 32767, -32768, 0, 1, -1, -2, -1, 32767, -32768, 0x1234, -0x1235], np.int16)
    assert np.array_equal(rule_to_s16(i), want_i)
    assert np.array_equal(kernel_to_s16(i), want_i)
    s = np.array([-32768, 32767, 0, -1, 1], np.int16)
    assert np.array_equal(kernel_to_s16(s), s)


def test_transmit_then_receive_is_the_identity():
    s = np.arange(-32768, 32768, dtype=np.int32).astype(np.int16)
    for dtype in FORMATS:
        x = kernel_from_s16(s, dtype)
        assert same_bits(x, rule_from_s16(s, dtype))
        assert np.array_equal(kernel_to_s16(x), s) and np.array_equal(rule_to_s16(x), s)
    assert kernel_from_s16(np.array([-32768], np.int16), np.float32)[0] == -1.0
    assert kernel_from_s16(np.array([-32768], np.int16), np.int32)[0] == -0x80000000


def test_random_floats_follow_the_rule():
    rng = np.random.default_rng(1)
    x = np.concatenate([rng.uniform(-1.5, 1.5, 200000), rng.integers(-70000, 70000, 20000) / 65536.0]).astype(np.float32)
    assert np.array_equal(kernel_to_s16(x), rule_to_s16(x))
