"""Argument checks of the per-channel stream entry points (afsk_rx_streams_create_each / _finish_some,
afsk_tx_streams_create_each / _configure) that run before any device is touched (no GPU needed)."""
import ctypes as C

import numpy as np
import pytest

from afskmodem_b200 import _cabi


def rx_create_each(L, baud, amp_start=18000, amp_end=14000, timeout=48000, S=None, null=None):
    S = len(baud) if S is None else S
    n = len(baud)
    arrs = [np.array(baud, np.int32), np.full(n, amp_start, np.int32), np.full(n, amp_end, np.int32),
            np.array(timeout if np.ndim(timeout) else [timeout] * n, np.int64)]
    ptrs = [_cabi.ptr(a, C.c_int32 if a.dtype == np.int32 else C.c_int64) for a in arrs]
    if null is not None:
        ptrs[null] = None
    h = C.c_void_p()
    rc = L.afsk_rx_streams_create_each(0, S, *ptrs, C.byref(h))
    assert not h.value
    return rc


@pytest.mark.parametrize("bad", [7, 9600, 32000])
@pytest.mark.parametrize("at", [0, 2, 4])
def test_rx_create_each_rejects_an_invalid_baud_on_any_channel(bad, at):
    L = _cabi.lib()
    baud = [1200, 300, 2400, 1200, 4800]
    baud[at] = bad
    assert rx_create_each(L, baud) == _cabi.AFSK_E_BAUD
    assert f"channel {at}" in L.afsk_last_error().decode()


def test_rx_create_each_rejects_bad_arguments():
    L = _cabi.lib()
    assert rx_create_each(L, [1200, 300], S=0) == _cabi.AFSK_E_ARG
    assert rx_create_each(L, [1200, 300], S=-1) == _cabi.AFSK_E_ARG
    for i in range(4):
        assert rx_create_each(L, [1200, 300], null=i) == _cabi.AFSK_E_ARG
    assert rx_create_each(L, [1200, 300], timeout=[48000, -1]) == _cabi.AFSK_E_ARG
    h = C.c_void_p()
    b, a, t = np.array([1200], np.int32), np.array([1], np.int32), np.array([0], np.int64)
    assert L.afsk_rx_streams_create_each(0, 1, _cabi.ptr(b, C.c_int32), _cabi.ptr(a, C.c_int32), _cabi.ptr(a, C.c_int32),
                                         _cabi.ptr(t, C.c_int64), None) == _cabi.AFSK_E_ARG


@pytest.mark.parametrize("bad", [7, 9600, 32000])
def test_tx_create_each_rejects_an_invalid_baud_on_any_channel(bad):
    L = _cabi.lib()
    for at in range(3):
        baud = np.array([1200, 24000, 4800], np.int32)
        baud[at] = bad
        ts = np.array([300, 0, 12], np.int64)
        h = C.c_void_p()
        assert L.afsk_tx_streams_create_each(0, 3, _cabi.ptr(baud, C.c_int32), _cabi.ptr(ts, C.c_int64), C.byref(h)) == _cabi.AFSK_E_BAUD
        assert f"channel {at}" in L.afsk_last_error().decode()
        assert not h.value


def test_tx_create_each_rejects_bad_arguments():
    L = _cabi.lib()
    baud, ts = np.array([1200, 300], np.int32), np.array([300, 75], np.int64)
    h = C.c_void_p()
    assert L.afsk_tx_streams_create_each(0, 0, _cabi.ptr(baud, C.c_int32), _cabi.ptr(ts, C.c_int64), C.byref(h)) == _cabi.AFSK_E_ARG
    assert L.afsk_tx_streams_create_each(0, 2, None, _cabi.ptr(ts, C.c_int64), C.byref(h)) == _cabi.AFSK_E_ARG
    assert L.afsk_tx_streams_create_each(0, 2, _cabi.ptr(baud, C.c_int32), None, C.byref(h)) == _cabi.AFSK_E_ARG
    assert L.afsk_tx_streams_create_each(0, 2, _cabi.ptr(baud, C.c_int32), _cabi.ptr(ts, C.c_int64), None) == _cabi.AFSK_E_ARG
    assert not h.value


def test_null_handle_is_a_bad_argument():
    L = _cabi.lib()
    ids = np.array([0], np.int32)
    n = C.c_int64(0)
    assert L.afsk_rx_streams_finish_some(None, 1, _cabi.ptr(ids, C.c_int32), None, None, None, None, None, C.byref(n)) == _cabi.AFSK_E_ARG
    assert L.afsk_rx_streams_finish_some(None, 0, None, None, None, None, None, None, C.byref(n)) == _cabi.AFSK_E_ARG
    b, t = np.array([1200], np.int32), np.array([300], np.int64)
    assert L.afsk_tx_streams_configure(None, 1, _cabi.ptr(ids, C.c_int32), _cabi.ptr(b, C.c_int32), _cabi.ptr(t, C.c_int64)) == _cabi.AFSK_E_ARG
    assert L.afsk_tx_streams_configure(None, 0, None, None, None) == _cabi.AFSK_E_ARG
