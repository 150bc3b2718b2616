"""Argument checks of afsk_tx_streams_create that run before any device is touched (no GPU needed)."""
import ctypes as C

from afskmodem_b200 import _cabi


def test_create_rejects_bad_baud_and_channel_count():
    L = _cabi.lib()
    h = C.c_void_p()
    assert L.afsk_tx_streams_create(0, 4, 7, 300, C.byref(h)) == _cabi.AFSK_E_BAUD          # 48000 % 7 != 0
    assert L.afsk_tx_streams_create(0, 4, 32000, 300, C.byref(h)) == _cabi.AFSK_E_BAUD
    assert L.afsk_tx_streams_create(0, 0, 1200, 300, C.byref(h)) == _cabi.AFSK_E_ARG
    assert not h.value


def test_null_handle_is_a_bad_argument():
    L = _cabi.lib()
    a = C.c_int64(0)
    assert L.afsk_tx_streams_pull(None, 8, None, 0, None) == _cabi.AFSK_E_ARG
    assert L.afsk_tx_streams_state(None, 0, C.byref(a), C.byref(a), C.byref(a)) == _cabi.AFSK_E_ARG
    assert L.afsk_tx_streams_destroy(None) == _cabi.AFSK_OK
