"""Argument checks of afsk_rx_streams_create that run before any device is touched (no GPU needed)."""
import ctypes as C

from afskmodem_b200 import _cabi


def test_create_rejects_bad_baud_and_channel_count():
    L = _cabi.lib()
    h = C.c_void_p()
    assert L.afsk_rx_streams_create(0, 4, 7, 18000, 14000, 48000, C.byref(h)) == _cabi.AFSK_E_BAUD   # 48000 % 7 != 0
    assert L.afsk_rx_streams_create(0, 4, 32000, 18000, 14000, 48000, C.byref(h)) == _cabi.AFSK_E_BAUD
    assert L.afsk_rx_streams_create(0, 0, 1200, 18000, 14000, 48000, C.byref(h)) == _cabi.AFSK_E_ARG
    assert not h.value
