"""The payload-mode retention entry points are exported, and their argument checks that need no device return
AFSK_E_ARG (no GPU needed)."""
import ctypes as C

import pytest

from afskmodem_b200 import _cabi, modem


def test_payload_symbols_are_exported():
    L = _cabi.lib()
    for name in ("afsk_rx_streams_pending_payload", "afsk_rx_streams_payload_counters"):
        assert name in _cabi.SYMBOLS
        assert hasattr(L, name)
    assert modem.StreamReceiver.RETAIN["payload"] == 2


def test_null_handle_bad_pointers_or_bad_mode_is_a_bad_argument():
    L = _cabi.lib()
    te, nb, n = C.c_int64(0), C.c_int64(0), C.c_int64(0)
    ended = C.c_int32(0)
    buf = (C.c_uint8 * 4)()
    for mode in (0, 1, 2, 3, -1):
        assert L.afsk_rx_streams_set_retention(None, mode) == _cabi.AFSK_E_ARG
    assert L.afsk_rx_streams_pending_payload(None, 0, C.byref(te), C.byref(nb), C.byref(ended), buf, 4, C.byref(n)) == _cabi.AFSK_E_ARG
    assert L.afsk_rx_streams_pending_payload(None, 0, None, None, None, None, 0, None) == _cabi.AFSK_E_ARG
    assert L.afsk_rx_streams_payload_counters(None, C.byref(te), C.byref(nb)) == _cabi.AFSK_E_ARG


def test_unknown_retention_is_refused_before_any_device_work():
    with pytest.raises(ValueError, match="payload"):
        modem.StreamReceiver([None], 1.0, 0, retain="planes")
