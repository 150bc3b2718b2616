"""The bits-mode retention entry points are exported, and their argument checks that need no device return
AFSK_E_ARG (no GPU needed)."""
import ctypes as C

import pytest

from afskmodem_b200 import _cabi, modem


def test_bits_symbols_are_exported():
    L = _cabi.lib()
    for name in ("afsk_rx_streams_set_retention", "afsk_rx_streams_pending_bits", "afsk_rx_streams_plane_counters",
                 "afsk_rx_streams_pending_planes"):
        assert name in _cabi.SYMBOLS
        assert hasattr(L, name)


def test_null_handle_or_bad_mode_is_a_bad_argument():
    L = _cabi.lib()
    clk, win = C.c_int32(0), C.c_int64(0)
    for mode in (0, 1, 2, -1):
        assert L.afsk_rx_streams_set_retention(None, mode) == _cabi.AFSK_E_ARG
    assert L.afsk_rx_streams_pending_bits(None, 0, C.byref(clk), C.byref(win)) == _cabi.AFSK_E_ARG
    assert L.afsk_rx_streams_plane_counters(None, C.byref(win), C.byref(win)) == _cabi.AFSK_E_ARG
    ptr, first = C.c_void_p(), C.c_int64(0)
    assert L.afsk_rx_streams_pending_planes(None, 0, C.byref(ptr), C.byref(first), C.byref(win)) == _cabi.AFSK_E_ARG


def test_unknown_retention_is_refused_before_any_device_work():
    with pytest.raises(ValueError, match="retain"):
        modem.StreamReceiver([None], 1.0, 0, retain="planes")
