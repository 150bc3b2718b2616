"""ctypes binding of libafsk_b200.so (include/afsk_b200.h).  No torch types cross this boundary.

There is no CPU fallback: if the library is missing or CUDA is unavailable every compute call
raises ``AfskError``.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# AFSK_LIB_PATH: a differently built copy of the library, for same-box A/B runs of compile-time variants
LIB_PATH = os.environ.get("AFSK_LIB_PATH") or os.path.join(_HERE, "libafsk_b200.so")

AFSK_OK, AFSK_E_ARG, AFSK_E_CUDA, AFSK_E_BAUD, AFSK_E_UNSUPPORTED = 0, -1, -2, -3, -4
ST_OK, ST_NO_CLOCK, ST_NO_DATA = 0, 1, 2
ST_EXC_WAVELEN, ST_EXC_INDEX, ST_EXC_BAUD = -1, -2, -3
# AFSK_SAMPLE_*: formats of interleaved frames (afsk_rx_streams_push_frames, afsk_tx_streams_pull_frames)
SAMPLE_S16, SAMPLE_S32, SAMPLE_F32 = 0, 1, 2
OPT_FRAME_KERNEL, OPT_L2_HINT, OPT_FUSED, OPT_CLOCK_KERNEL, OPT_GROUP_STREAMS = 1, 2, 3, 4, 5

# every symbol include/afsk_b200.h declares (tests check the library exports them all)
SYMBOLS = [
    "afsk_abi_version", "afsk_last_error", "afsk_device_count", "afsk_device_info", "afsk_malloc",
    "afsk_free", "afsk_host_alloc", "afsk_host_free", "afsk_memcpy_h2d", "afsk_memcpy_d2h",
    "afsk_memset", "afsk_stream_create", "afsk_stream_destroy", "afsk_stream_sync", "afsk_stream_wait_stream",
    "afsk_tone_lengths", "afsk_rx_plan_create", "afsk_rx_plan_create_ranges", "afsk_rx_plan_reset", "afsk_rx_plan_set_option", "afsk_rx_plan_destroy", "afsk_rx_plan_out_offsets",
    "afsk_rx_plan_launches", "afsk_rx_plan_set_timing", "afsk_rx_plan_demod_time", "afsk_rx_decode", "afsk_rx_plan_planes", "afsk_rx_decode_host", "afsk_rx_host_release",
    "afsk_rx_out_capacity", "afsk_rx_gate", "afsk_rx_gate_multi", "afsk_tx_num_samples", "afsk_tx_plan_create",
    "afsk_tx_plan_destroy", "afsk_tx_plan_out_offsets", "afsk_tx_synth", "afsk_tx_synth_host",
    "afsk_wav_probe", "afsk_wav_load", "afsk_wav_save", "afsk_rx_streams_create", "afsk_rx_streams_push",
    "afsk_rx_streams_finish", "afsk_rx_streams_events", "afsk_rx_streams_state", "afsk_rx_streams_arena_bytes",
    "afsk_rx_streams_counters", "afsk_rx_streams_destroy", "afsk_tx_streams_create", "afsk_tx_streams_send",
    "afsk_tx_streams_pull", "afsk_tx_streams_state", "afsk_tx_streams_arena_bytes", "afsk_tx_streams_counters",
    "afsk_tx_streams_destroy", "afsk_rx_streams_create_each", "afsk_rx_streams_finish_some", "afsk_tx_streams_create_each",
    "afsk_tx_streams_configure", "afsk_rx_streams_push_interleaved", "afsk_tx_streams_pull_interleaved",
    "afsk_rx_streams_set_retention", "afsk_rx_streams_pending_bits", "afsk_rx_streams_plane_counters",
    "afsk_rx_streams_pending_payload", "afsk_rx_streams_payload_counters", "afsk_rx_streams_push_frames",
    "afsk_tx_streams_pull_frames", "afsk_rx_streams_pending_planes",
]


class AfskError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libafsk_b200 error {code}: {msg}")
        self.code = code


class RxResult(C.Structure):
    _fields_ = [("status", C.c_int32), ("clock", C.c_int32), ("train_end", C.c_int64),
                ("nbits", C.c_int64), ("nbytes", C.c_int64)]


RX_RESULT_DTYPE = np.dtype([("status", "<i4"), ("clock", "<i4"), ("train_end", "<i8"),
                            ("nbits", "<i8"), ("nbytes", "<i8")])
assert RX_RESULT_DTYPE.itemsize == C.sizeof(RxResult) == 32

# AfskRxStreamEvent
STREAM_EVENT_DTYPE = np.dtype([("stream", "<i4"), ("recorded", "<i4"), ("call", "<i8"), ("start", "<i8"), ("end", "<i8")])
assert STREAM_EVENT_DTYPE.itemsize == 32

_lib = None


def lib():
    """Loads the shared library; raises (loudly) when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise AfskError(AFSK_E_CUDA, f"{LIB_PATH} not built — run `python -m afskmodem_b200.build` "
                                     "(there is no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    vp, i64p, i32p, u8p, i16p = C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int32), C.POINTER(C.c_uint8), \
        C.POINTER(C.c_int16)
    L.afsk_abi_version.restype = C.c_int
    L.afsk_last_error.restype = C.c_char_p
    L.afsk_device_count.argtypes = [C.POINTER(C.c_int)]
    L.afsk_device_info.argtypes = [C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_size_t), C.POINTER(C.c_int)]
    L.afsk_malloc.argtypes = [C.c_int, C.c_size_t, C.POINTER(vp)]
    L.afsk_free.argtypes = [C.c_int, vp]
    L.afsk_host_alloc.argtypes = [C.c_size_t, C.POINTER(vp)]
    L.afsk_host_free.argtypes = [vp]
    L.afsk_memcpy_h2d.argtypes = [C.c_int, vp, vp, C.c_size_t, vp]
    L.afsk_memcpy_d2h.argtypes = [C.c_int, vp, vp, C.c_size_t, vp]
    L.afsk_memset.argtypes = [C.c_int, vp, C.c_int, C.c_size_t, vp]
    L.afsk_stream_create.argtypes = [C.c_int, C.POINTER(vp)]
    L.afsk_stream_destroy.argtypes = [C.c_int, vp]
    L.afsk_stream_sync.argtypes = [C.c_int, vp]
    L.afsk_stream_wait_stream.argtypes = [C.c_int, vp, vp]
    L.afsk_tone_lengths.argtypes = [C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.afsk_rx_plan_create.argtypes = [C.c_int, C.c_int, i64p, i32p, i32p, C.POINTER(vp)]
    L.afsk_rx_plan_create_ranges.argtypes = [C.c_int, C.c_int, i64p, i64p, i32p, i32p, C.POINTER(vp)]
    L.afsk_rx_plan_reset.argtypes = [vp, C.c_int, i64p, i64p, i32p, i32p]
    L.afsk_rx_plan_set_option.argtypes = [vp, C.c_int, C.c_int]
    L.afsk_rx_host_release.argtypes = [C.c_int]
    L.afsk_rx_plan_destroy.argtypes = [vp]
    L.afsk_rx_plan_out_offsets.argtypes = [vp, C.POINTER(i64p)]
    L.afsk_rx_plan_launches.argtypes = [vp, C.POINTER(C.c_int)]
    L.afsk_rx_plan_set_timing.argtypes = [vp, C.c_int]
    L.afsk_rx_plan_demod_time.argtypes = [vp, C.POINTER(C.c_float), C.POINTER(C.c_int)]
    L.afsk_rx_decode.argtypes = [vp, vp, vp, vp, vp]
    L.afsk_rx_plan_planes.argtypes = [vp, C.c_int, C.POINTER(vp), i64p]
    L.afsk_rx_decode_host.argtypes = [C.c_int, i16p, i64p, C.c_int, i32p, i32p, u8p, i64p, C.POINTER(RxResult)]
    L.afsk_rx_out_capacity.argtypes = [C.c_int64, C.c_int]
    L.afsk_rx_out_capacity.restype = C.c_int64
    L.afsk_rx_gate.argtypes = [C.c_int, vp, i64p, C.c_int, C.c_int, C.c_int, C.c_int64, vp, vp]
    L.afsk_rx_gate_multi.argtypes = [C.c_int, vp, i64p, C.c_int, C.c_int, C.c_int, C.c_int64, C.c_int, vp, vp, vp]
    L.afsk_rx_streams_create.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int64, C.POINTER(vp)]
    L.afsk_rx_streams_push.argtypes = [vp, vp, C.c_int, i64p, vp, i64p]
    L.afsk_rx_streams_push_interleaved.argtypes = [vp, vp, C.c_int, C.c_int64, vp, i64p]
    L.afsk_rx_streams_push_frames.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int64, C.c_int64, vp, i64p]
    L.afsk_rx_streams_create_each.argtypes = [C.c_int, C.c_int, i32p, i32p, i32p, i64p, C.POINTER(vp)]
    L.afsk_rx_streams_finish.argtypes = [vp, vp, i64p]
    L.afsk_rx_streams_finish_some.argtypes = [vp, C.c_int, i32p, i32p, i32p, i32p, i64p, vp, i64p]
    L.afsk_rx_streams_events.argtypes = [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), C.POINTER(vp)]
    L.afsk_rx_streams_state.argtypes = [vp, C.c_int, i64p, i64p, i64p]
    L.afsk_rx_streams_arena_bytes.argtypes = [vp, i64p]
    L.afsk_rx_streams_counters.argtypes = [vp, i64p, i64p, i64p]
    L.afsk_rx_streams_destroy.argtypes = [vp]
    L.afsk_rx_streams_set_retention.argtypes = [vp, C.c_int]
    L.afsk_rx_streams_pending_bits.argtypes = [vp, C.c_int, i32p, i64p]
    L.afsk_rx_streams_pending_planes.argtypes = [vp, C.c_int, C.POINTER(vp), i64p, i64p]
    L.afsk_rx_streams_plane_counters.argtypes = [vp, i64p, i64p]
    L.afsk_rx_streams_pending_payload.argtypes = [vp, C.c_int, i64p, i64p, i32p, vp, C.c_int64, i64p]
    L.afsk_rx_streams_payload_counters.argtypes = [vp, i64p, i64p]
    L.afsk_tx_num_samples.argtypes = [C.c_int, C.c_int64, C.c_int64, u8p]
    L.afsk_tx_num_samples.restype = C.c_int64
    L.afsk_tx_plan_create.argtypes = [C.c_int, C.c_int, i64p, i32p, i64p, u8p, C.POINTER(vp)]
    L.afsk_tx_plan_destroy.argtypes = [vp]
    L.afsk_tx_plan_out_offsets.argtypes = [vp, C.POINTER(i64p), C.POINTER(i64p)]
    L.afsk_tx_synth.argtypes = [vp, vp, vp, vp]
    L.afsk_tx_synth_host.argtypes = [C.c_int, u8p, i64p, C.c_int, i32p, i64p, i16p, i64p]
    L.afsk_tx_streams_create.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int64, C.POINTER(vp)]
    L.afsk_tx_streams_create_each.argtypes = [C.c_int, C.c_int, i32p, i64p, C.POINTER(vp)]
    L.afsk_tx_streams_configure.argtypes = [vp, C.c_int, i32p, i32p, i64p]
    L.afsk_tx_streams_send.argtypes = [vp, C.c_int, i32p, i64p, u8p, i64p, i64p]
    L.afsk_tx_streams_pull.argtypes = [vp, C.c_int64, vp, C.c_int, vp]
    L.afsk_tx_streams_pull_interleaved.argtypes = [vp, C.c_int64, vp, C.c_int, vp]
    L.afsk_tx_streams_pull_frames.argtypes = [vp, C.c_int64, vp, C.c_int, C.c_int, C.c_int64, vp]
    L.afsk_tx_streams_state.argtypes = [vp, C.c_int, i64p, i64p, i64p]
    L.afsk_tx_streams_arena_bytes.argtypes = [vp, i64p]
    L.afsk_tx_streams_counters.argtypes = [vp, i64p, i64p, i64p]
    L.afsk_tx_streams_destroy.argtypes = [vp]
    cpp = C.POINTER(C.c_char_p)
    L.afsk_wav_probe.argtypes = [cpp, C.c_int, C.c_int, i64p, i64p, i32p]
    L.afsk_wav_load.argtypes = [cpp, C.c_int, C.c_int, i64p, i64p, i64p, vp, C.c_int, vp, C.c_int64, vp, i32p]
    L.afsk_wav_save.argtypes = [cpp, C.c_int, C.c_int, vp, i64p, i64p, i32p]
    _lib = L
    return L


def check(rc: int) -> None:
    if rc != 0:
        raise AfskError(rc, lib().afsk_last_error().decode("utf-8", "replace"))


def ptr(a: np.ndarray, ctype):
    return a.ctypes.data_as(C.POINTER(ctype))


def device_count() -> int:
    n = C.c_int(0)
    rc = lib().afsk_device_count(C.byref(n))
    return n.value if rc == 0 else 0


def require_device(device: int = 0) -> None:
    n = device_count()
    if n <= device:
        raise AfskError(AFSK_E_CUDA, f"CUDA device {device} not available ({n} visible): the AFSK core has "
                                     "no CPU fallback")


class DeviceBuffer:
    """cudaMalloc'd bytes owned by Python (freed on close/GC)."""

    def __init__(self, device: int, nbytes: int):
        self.device, self.nbytes = device, int(nbytes)
        p = C.c_void_p()
        check(lib().afsk_malloc(device, max(self.nbytes, 16), C.byref(p)))
        self.ptr = p.value
        self._free, self._cptr = lib().afsk_free, p     # kept so that close() works during interpreter shutdown

    def close(self):
        if getattr(self, "ptr", None):
            self._free(self.device, self._cptr)
            self.ptr = None

    __del__ = close

    def upload(self, arr: np.ndarray, stream=None, offset: int = 0):
        arr = np.ascontiguousarray(arr)
        if offset < 0 or offset + arr.nbytes > max(self.nbytes, 16):
            raise ValueError(f"upload of {arr.nbytes} bytes at offset {offset} exceeds the {self.nbytes}-byte device buffer")
        check(lib().afsk_memcpy_h2d(self.device, C.c_void_p(self.ptr + offset), C.c_void_p(arr.ctypes.data),
                                    arr.nbytes, C.c_void_p(stream or 0)))

    def download(self, arr: np.ndarray, stream=None, offset: int = 0):
        if not arr.flags["C_CONTIGUOUS"]:
            raise ValueError("download target must be C-contiguous")
        if offset < 0 or offset + arr.nbytes > max(self.nbytes, 16):
            raise ValueError(f"download of {arr.nbytes} bytes at offset {offset} exceeds the {self.nbytes}-byte device buffer")
        check(lib().afsk_memcpy_d2h(self.device, C.c_void_p(arr.ctypes.data), C.c_void_p(self.ptr + offset),
                                    arr.nbytes, C.c_void_p(stream or 0)))


class PinnedArray:
    """numpy view over cudaMallocHost memory (fast, truly asynchronous H2D/D2H)."""

    def __init__(self, shape, dtype):
        self.dtype = np.dtype(dtype)
        n = int(np.prod(shape)) * self.dtype.itemsize
        p = C.c_void_p()
        check(lib().afsk_host_alloc(max(n, 16), C.byref(p)))
        self._ptr = p.value
        self._free, self._cptr = lib().afsk_host_free, p
        buf = (C.c_uint8 * max(n, 16)).from_address(self._ptr)
        self.array = np.frombuffer(buf, dtype=self.dtype, count=int(np.prod(shape))).reshape(shape)

    def close(self):
        if getattr(self, "_ptr", None):
            self.array = None
            self._free(self._cptr)
            self._ptr = None

    __del__ = close


def c_paths(filenames):
    """list of str/bytes/PathLike -> (char*[n], keep-alive list)"""
    enc = [os.fsencode(f) for f in filenames]
    arr = (C.c_char_p * max(len(enc), 1))(*enc)
    return arr, enc


def stream_sync(device: int, stream=None):
    check(lib().afsk_stream_sync(device, C.c_void_p(stream or 0)))


def stream_create(device: int) -> int:
    s = C.c_void_p()
    check(lib().afsk_stream_create(device, C.byref(s)))
    return s.value


def stream_destroy(device: int, stream: int):
    lib().afsk_stream_destroy(device, C.c_void_p(stream))


def stream_wait_stream(device: int, waiter: int, signaller: int):
    check(lib().afsk_stream_wait_stream(device, C.c_void_p(waiter), C.c_void_p(signaller)))


def tone_lengths(baud: int):
    """(bit_frames, mark_len, space_len) or None where the reference constructor raises."""
    a, b, c = C.c_int(0), C.c_int(0), C.c_int(0)
    rc = lib().afsk_tone_lengths(int(baud), C.byref(a), C.byref(b), C.byref(c))
    return None if rc != 0 else (a.value, b.value, c.value)
