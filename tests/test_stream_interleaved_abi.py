"""The interleaved streaming entry points are exported, and their argument checks that need no device return
AFSK_E_ARG (no GPU needed)."""
import ctypes as C

from afskmodem_b200 import _cabi


def test_interleaved_symbols_are_exported():
    L = _cabi.lib()
    for name in ("afsk_rx_streams_push_interleaved", "afsk_tx_streams_pull_interleaved"):
        assert name in _cabi.SYMBOLS
        assert hasattr(L, name)


def test_null_handle_is_a_bad_argument():
    L = _cabi.lib()
    n = C.c_int64(0)
    assert L.afsk_rx_streams_push_interleaved(None, None, 0, 0, None, C.byref(n)) == _cabi.AFSK_E_ARG
    assert L.afsk_rx_streams_push_interleaved(None, None, 0, 8, None, C.byref(n)) == _cabi.AFSK_E_ARG
    assert L.afsk_rx_streams_push_interleaved(None, None, 0, -1, None, C.byref(n)) == _cabi.AFSK_E_ARG
    assert L.afsk_tx_streams_pull_interleaved(None, 8, None, 0, None) == _cabi.AFSK_E_ARG
    assert L.afsk_tx_streams_pull_interleaved(None, 0, None, 0, None) == _cabi.AFSK_E_ARG
    assert L.afsk_tx_streams_pull_interleaved(None, -1, None, 1, None) == _cabi.AFSK_E_ARG
