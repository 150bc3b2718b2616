"""CPU model of the interleaved streaming kernels' index arithmetic, restated from the CUDA source:

  * k_stream_deinterleave (afsk_rx.cu): tile -> channel / frame ranges, the 7-frame halo, the row loads as
    aligned 16-byte vectors realigned with funnel shifts, the shared tile in destination coordinates and the
    per-channel destination vectors with their head / tail masks.  Checked against a plain transpose-and-append
    into an arena whose other samples (neighbouring slots) must stay untouched, and against reading any vector
    outside the piece.
  * k_tx_window_interleaved (afsk_tx.cu): the tile of channels x column vectors and its frame-major write
    out[f * S + c], checked against the transpose of the planar window, with nothing past n * S written.
"""
import numpy as np
import pytest

KC, KF, HALO, STRIDE = 64, 128, 7, 136            # kDiC, kDiF, kDiHalo, kDiStride
IL_C, IL_V, IL_STRIDE = 64, 16, 136                # kIlC, kIlV, kIlStride
POISON = -(1 << 20)


def shared_row(c):
    return (c & 7) * 8 + (c >> 3)


def funnel_r16(lo, hi):
    return (((hi.astype(np.uint64) << np.uint64(32)) | lo.astype(np.uint64)) >> np.uint64(16)).astype(np.uint32)


def halves(words):
    """uint32 words (..., 4) -> their eight int16 samples, low half first (little-endian)"""
    return np.stack([words & 0xFFFF, words >> 16], -1).reshape(*words.shape[:-1], 8).astype(np.uint16).view(np.int16)


def k_stream_deinterleave(src, n, S, seg_dst, arena):
    """One launch over n frames (src: n * S samples, padded with garbage to a 16-byte multiple).  Returns the
    count of full 16-byte stores and the partial vectors per channel."""
    total = n * S
    words = np.ascontiguousarray(src).view(np.uint32)
    cblocks, ftiles = -(-S // KC), (n + KF + HALO - 1) // KF
    full, partial = 0, np.zeros(S, np.int64)
    for b in range(cblocks * ftiles):
        cb, fb = b % cblocks, b // cblocks
        c0, F0 = cb * KC, fb * KF
        nc = min(KC, S - c0)
        sd = seg_dst[c0:c0 + nc]
        T = np.full((KC, STRIDE), POISON, np.int64)
        f_lo, f_hi = max(F0 - HALO, 0), min(F0 + KF, n)
        assert f_hi > f_lo                                         # every tile has rows to load
        f = np.arange(f_lo, f_hi)[:, None]
        q = np.arange((nc + 7) // 8)[None, :]
        qs = f * S + c0 + 8 * q
        sv, k = qs >> 3, qs & 7
        row_end = f * S + c0 + nc
        assert (sv * 8 < total).all() and (sv >= 0).all()          # lo holds sample qs, inside the piece
        hi_ok = (k != 0) & ((sv + 1) * 8 < row_end)
        assert ((sv + 1) * 8 < total)[hi_ok].all()
        lo = words[(sv * 4)[..., None] + np.arange(4)]
        hi = np.where(hi_ok[..., None], words[np.where(hi_ok, (sv + 1) * 4, 0)[..., None] + np.arange(4)], 0)
        w = np.concatenate([lo, hi], -1).astype(np.uint32)
        j = (k >> 1)[..., None] + np.arange(4)
        x0, x1 = np.take_along_axis(w, j, -1), np.take_along_axis(w, j + 1, -1)
        o = np.where((k & 1)[..., None] == 1, funnel_r16(x0, x1), x0)
        vals = halves(o)                                           # (rows, nq, 8): channels 8q + e
        c = 8 * q[..., None] + np.arange(8)
        c = np.broadcast_to(c, vals.shape)
        cc = np.where(c < nc, c, 0)
        p = f[..., None] - F0 + (sd[cc] & 7)
        ok = (c < nc) & (p >= 0) & (p < KF)
        T[shared_row(cc[ok]), p[ok]] = vals[ok]
        # stores: channel c, destination vector j
        c = np.arange(nc)[:, None]
        jv = np.arange(KF // 8)[None, :]
        g = sd[c]
        d0 = (g >> 3) * 8 + F0 + 8 * jv
        f0 = d0 - g
        live = f0 < n
        e = np.arange(8)
        fe = f0[..., None] + e
        m = live[..., None] & (fe >= 0) & (fe < n)
        v = T[shared_row(c)[..., None], 8 * jv[..., None] + e]
        assert (v[m] != POISON).all()                              # every frame written was loaded
        is_full = live & (f0 >= 0) & (f0 + 8 <= n)
        assert (d0[is_full] % 8 == 0).all()
        full += int(is_full.sum())
        partial[c0:c0 + nc] += (live & ~is_full).sum(1)
        arena[(d0[..., None] + e)[m]] = v[m]
    return full, partial


def slots(S, n, rng, align):
    """per-channel destination offsets in one arena: slot after slot, some back to back, alignments given"""
    dst, at = np.zeros(S, np.int64), 8
    for s in range(S):
        at = (at + 7) // 8 * 8 + int(align[s])
        dst[s] = at
        at += n + int(rng.integers(0, 10))
    return dst, at + 64


N_CASES = [0, 1, 7, 8, 9, 127, 128, 129, 2048, 613]


@pytest.mark.parametrize("S", [1, 2, 3, 5, 8, 9, 63, 64] + [64 + r for r in range(1, 9)])
def test_deinterleave_equals_transpose_and_append(S):
    rng = np.random.default_rng(S)
    for n in N_CASES:
        aligns = [np.full(S, a) for a in range(8)] + [rng.integers(0, 8, S)]
        for align in aligns:
            x = rng.integers(-32768, 32768, size=(n, S), dtype=np.int16)
            src = np.concatenate([x.reshape(-1), rng.integers(-32768, 32768, (-(n * S)) % 8 + 8, dtype=np.int16)])
            dst, size = slots(S, n, rng, align)
            arena = rng.integers(-32768, 32768, size, dtype=np.int16)
            want = arena.copy()
            for s in range(S):
                want[dst[s]:dst[s] + n] = x[:, s]
            if n == 0:                                             # the host launches nothing
                continue
            full, partial = k_stream_deinterleave(src, n, S, dst, arena)
            np.testing.assert_array_equal(arena, want, err_msg=f"S={S} n={n} align={align[:8]}")
            assert (partial <= 2).all()                            # only a channel's head and tail vectors
            assert full >= S * (n // 8 - 2)


def k_tx_window_interleaved(W, S, n, out):
    """W: the planar window (S, n) as win_vec computes it; writes out[f * S + c]"""
    cblocks, ftiles = -(-S // IL_C), (n + 8 * IL_V - 1) // (8 * IL_V)
    for b in range(cblocks * ftiles):
        cb, fb = b % cblocks, b // cblocks
        c0, F0 = cb * IL_C, fb * 8 * IL_V
        nc, nf = min(IL_C, S - c0), min(8 * IL_V, n - F0)
        assert nf > 0
        T = np.full((IL_C, IL_STRIDE), POISON, np.int64)
        for c in range(nc):                                        # phase 1: 8-frame column vectors
            for col in range(0, nf, 8):
                m = min(8, nf - col)
                vec = np.zeros(8, np.int64)
                vec[:m] = W[c0 + c, F0 + col:F0 + col + m]
                T[shared_row(c), col:col + 8] = vec
        i = np.arange(nf * 9)
        q, fl = i % 9, i // 9
        a = (F0 + fl) * S + c0
        bnd = a + nc
        d0 = ((a >> 3) + q) * 8
        live = d0 < bnd
        e = np.arange(8)
        cidx = d0[:, None] + e - a[:, None]
        m = live[:, None] & (cidx >= 0) & (cidx < nc)
        cc = np.where(m, cidx, 0)
        v = T[shared_row(cc), fl[:, None]]
        assert (v[m] != POISON).all()
        is_full = live & (d0 >= a) & (d0 + 8 <= bnd)
        assert (m[is_full]).all()
        # partial vectors only at the row's head and tail
        per_row = np.bincount(fl[live & ~is_full], minlength=nf)
        assert (per_row <= 2).all()
        if S % 8 == 0 and c0 + IL_C <= S:
            assert not (live & ~is_full).any()
        out[(d0[:, None] + e)[m]] = v[m]


@pytest.mark.parametrize("S", [1, 3, 7, 8, 9, 63, 64, 65, 72, 130])
def test_tx_tile_writes_the_transposed_window(S):
    rng = np.random.default_rng(100 + S)
    for n in N_CASES:
        W = rng.integers(-32768, 32768, size=(S, n), dtype=np.int16)
        out = np.full(n * S + 24, 0x5A5A, np.int64)
        if n:
            k_tx_window_interleaved(W, S, n, out)
        np.testing.assert_array_equal(out[:n * S], W.T.reshape(-1))
        assert (out[n * S:] == 0x5A5A).all()
