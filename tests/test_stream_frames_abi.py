"""The windowed, multi-format interleaved entry points are exported, and a call without a handle returns AFSK_E_ARG
whatever its other arguments (no GPU needed).  A handle needs a device, so the checks of each argument (format,
row_pitch, alignment, overflow, grid size) are exercised on live handles in tests/test_gpu_stream_frames.py."""
import ctypes as C

from afskmodem_b200 import _cabi


def test_frames_symbols_are_exported():
    L = _cabi.lib()
    for name in ("afsk_rx_streams_push_frames", "afsk_tx_streams_pull_frames"):
        assert name in _cabi.SYMBOLS
        assert hasattr(L, name)
    assert (_cabi.SAMPLE_S16, _cabi.SAMPLE_S32, _cabi.SAMPLE_F32) == (0, 1, 2)


def test_calls_without_a_handle_are_bad_arguments():
    L = _cabi.lib()
    n = C.c_int64(0)
    buf = (C.c_int32 * 64)()
    p = C.cast(buf, C.c_void_p).value
    cases = [(0, 0, 8, 8), (_cabi.SAMPLE_S32, 0, 8, 8), (3, p, 8, 8), (-1, p, 8, 8), (0, p, 8, 0), (0, p, -1, 8),
             (_cabi.SAMPLE_F32, p + 2, 1, 8), (0, None, 8, 8), (0, p, 1 << 62, 1 << 40)]
    for fmt, ptr, n_frames, pitch in cases:
        assert L.afsk_rx_streams_push_frames(None, ptr, fmt, 0, n_frames, pitch, None, C.byref(n)) == _cabi.AFSK_E_ARG
        assert L.afsk_tx_streams_pull_frames(None, n_frames, ptr, fmt, 0, pitch, None) == _cabi.AFSK_E_ARG
    assert L.afsk_rx_streams_push_frames(None, p, 0, 0, 1, 8, None, None) == _cabi.AFSK_E_ARG
