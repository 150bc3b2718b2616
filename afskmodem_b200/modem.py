"""Host-side mirror of the reference's class API (afskmodem.py:19-61 Log, :66-107 Waveforms,
:114-175 ECC, :274-430 Receiver, :436-484 Transmitter) over the CUDA core.

Same names, argument meaning, log text, return types and error behaviour as the reference on the
file path (``load``/``save``); batch entry points (``decode_batch``, ``load_batch``,
``encode_batch``, ``save_batch``) are additions.  All signal processing runs in
``libafsk_b200.so``; this module only validates arguments, moves bytes and formats results.
"""
from __future__ import annotations

import ctypes as C
import wave
from datetime import datetime

import numpy as np

from . import _cabi
from ._cabi import AfskError, DeviceBuffer

# Log level (0: Debug, 1: Info, 2: Warn, 3: Error, 4: Fatal) — same global as afskmodem.py:14.
# The package-level ``afskmodem_b200.LOG_LEVEL`` is the one users set; see __init__.py.
_LEVEL_TAGS = {1: " [ INFO ]  ", 2: " [ WARN ]  ", 3: " [ ERROR ] ", 4: " [ FATAL ] "}


def _log_level() -> int:
    import afskmodem_b200
    return afskmodem_b200.LOG_LEVEL


class Log:
    """Timestamped print logger with the reference's line format (afskmodem.py:19-61)."""

    def __init__(self, class_name: str):
        self._name = class_name

    def _emit(self, level: int, message: str) -> None:
        if level >= _log_level():
            print(datetime.now().strftime("%Y-%m-%d %H:%M:%S") + _LEVEL_TAGS.get(level, " [ DEBUG ] ")
                  + self._name.ljust(24) + ": " + message)

    def debug(self, message: str) -> None:
        self._emit(0, message)

    def info(self, message: str) -> None:
        self._emit(1, message)

    def warn(self, message: str) -> None:
        self._emit(2, message)

    def error(self, message: str) -> None:
        self._emit(3, message)

    def fatal(self, message: str) -> None:
        self._emit(4, message)


class Waveforms:
    """Tone tables and the two waveform metrics (afskmodem.py:66-107), host utilities.

    The receiver/transmitter do not call these (the CUDA kernels use closed forms); they exist so
    code written against the reference's ``Waveforms`` keeps working.
    """

    @staticmethod
    def getSpaceTone(baud_rate: int) -> list[int]:
        if 48000 % baud_rate != 0:
            raise Exception("Invalid baud rate.")
        half = int((48000 / baud_rate) / 2)
        return [32767] * half + [-32768] * half

    @staticmethod
    def getMarkTone(baud_rate: int) -> list[int]:
        if 48000 % baud_rate != 0:
            raise Exception("Invalid baud rate.")
        return Waveforms.getSpaceTone(baud_rate * 2) * 2

    @staticmethod
    def getTrainingCycle(baud_rate: int) -> list[int]:
        return Waveforms.getMarkTone(baud_rate) + Waveforms.getSpaceTone(baud_rate)

    @staticmethod
    def getAmplitude(frames) -> int:
        a = np.asarray(frames, dtype=np.int64)
        return int(int(np.abs(a).sum()) / len(a))

    @staticmethod
    def getDiff(a, b) -> int:
        if len(a) != len(b):
            raise Exception("Comparing two waveforms of different lengths.")
        d = np.asarray(a, dtype=np.int64) - np.asarray(b, dtype=np.int64)
        return int(int(np.abs(d).sum()) / len(a))


class ECC:
    """Hamming(7,4) on '0'/'1' strings (afskmodem.py:114-175), host utility (table driven)."""

    @staticmethod
    def _codeword(nib: int) -> str:
        d0, d1, d2, d3 = (nib >> 3) & 1, (nib >> 2) & 1, (nib >> 1) & 1, nib & 1
        return "".join(str(b) for b in (d0 ^ d1 ^ d3, d0 ^ d2 ^ d3, d0, d1 ^ d2 ^ d3, d1, d2, d3))

    @staticmethod
    def encode(bits: str) -> str:
        table = [ECC._codeword(n) for n in range(16)]
        return "".join(table[int("".join("0" if ch == "0" else "1" for ch in bits[i:i + 4]), 2)]
                       for i in range(0, len(bits) - 3, 4))

    @staticmethod
    def decode(bits: str) -> str:
        out = []
        for i in range(0, len(bits) - 6, 7):
            c = [0 if ch == "0" else 1 for ch in bits[i:i + 7]]
            e = (c[0] ^ c[2] ^ c[4] ^ c[6]) + 2 * (c[1] ^ c[2] ^ c[5] ^ c[6]) + 4 * (c[3] ^ c[4] ^ c[5] ^ c[6])
            if e:
                c[e - 1] ^= 1
            out.append("%d%d%d%d" % (c[2], c[4], c[5], c[6]))
        return "".join(out)


class SoundInput:
    """File half of the reference's SoundInput (afskmodem.py:180-221).  ``loadFromFile`` is the static
    helper ``Receiver.load`` uses (:213-217); the pyaudio stream methods need an audio device and raise."""

    def __init__(self):
        raise RuntimeError("afskmodem_b200 has no live audio input; SoundInput.loadFromFile is available")

    @staticmethod
    def loadFromFile(filename: str) -> list[int]:
        return read_wav_frames(filename).tolist()


class SoundOutput:
    """File half of the reference's SoundOutput (afskmodem.py:226-268): ``writeToFile`` with
    ``__convertFrames``' pair duplication (out[n] = frames[n & ~1], an odd last frame dropped, :239-244)."""

    def __init__(self):
        raise RuntimeError("afskmodem_b200 has no live audio output; SoundOutput.writeToFile is available")

    @staticmethod
    def writeToFile(filename: str, frames) -> None:
        f = np.asarray(frames, dtype=np.int64)
        even = f[0:len(f) - 1:2]
        if len(even) and (even.min() < -32768 or even.max() > 32767):
            raise OverflowError("int too big to convert")            # int.to_bytes(2, signed=True) :242
        write_wav_frames(filename, np.repeat(even.astype(np.int16), 2))


def _check_baud(baud_rate) -> int:
    """Constructor-time validation with the reference's exceptions (afskmodem.py:69-70, 81-83)."""
    Waveforms.getSpaceTone(baud_rate)      # raises Exception("Invalid baud rate.") / ZeroDivisionError
    Waveforms.getMarkTone(baud_rate)
    if int(baud_rate) != baud_rate:
        raise Exception("Invalid baud rate.")
    return int(baud_rate)


def _as_int_threshold(t) -> int:
    # floor(mean) < t  <=>  floor(mean) < ceil(t) for real t
    return int(np.ceil(t))


# ------------------------------------------------------------------------------ receiver ----
PIPELINE_MIN_BYTES = 64 << 20      # decode_batch overlaps copy and kernels from this batch size on
PIPELINE_CHUNKS = 8


class RxBatch:
    """Decoded batch: per-capture stage integers (the reference's debug-log values) and payloads."""

    def __init__(self, results: np.ndarray, blob: np.ndarray, out_off: np.ndarray):
        self.results = results            # structured: status, clock, train_end, nbits, nbytes
        self.blob = blob                  # uint8, capacity layout
        self.out_off = out_off            # int64 [B+1]

    def __len__(self) -> int:
        return len(self.results)

    status = property(lambda self: self.results["status"])
    clock = property(lambda self: self.results["clock"])
    train_end = property(lambda self: self.results["train_end"])
    nbits = property(lambda self: self.results["nbits"])
    nbytes = property(lambda self: self.results["nbytes"])

    def payload(self, i: int) -> bytes:
        o = int(self.out_off[i])
        return self.blob[o:o + int(self.results["nbytes"][i])].tobytes()

    def payloads(self) -> list[bytes]:
        return [self.payload(i) for i in range(len(self))]

    def total_payload_bytes(self) -> int:
        return int(self.results["nbytes"].sum())


class RxSession:
    """A plan plus device buffers for one batch layout on one GPU.

    ``upload`` (H2D) / ``run`` (kernels, async on ``stream``) / ``download`` (D2H) are separate so
    that callers can keep samples resident in HBM (bench ``value``) or time the whole call (``e2e``).
    ``d_samples`` may be an external device pointer (e.g. ``torch.Tensor.data_ptr()``).
    """

    def __init__(self, offsets, baud, amp_end, device: int = 0, lengths=None):
        """``offsets``: CSR offsets (B+1) of adjacent captures, or — with ``lengths`` (B) — the start of
        each capture inside one sample buffer (captures need not be adjacent)."""
        _cabi.require_device(device)
        self.device = device
        self.plan = None
        self._destroy = _cabi.lib().afsk_rx_plan_destroy      # kept for close() during interpreter shutdown
        self.d_out = self.d_res = self.d_samples = None
        self._ext_ptr = None
        self._configure(offsets, baud, amp_end, lengths)

    def reset(self, offsets, baud, amp_end, lengths=None):
        """Re-targets this session at another batch layout (``afsk_rx_plan_reset``): the plan's device
        arena and this session's buffers are reused when large enough, so a receiver that decodes one
        file after another (``Receiver.load``) allocates nothing after its first calls."""
        self._configure(offsets, baud, amp_end, lengths)

    def _configure(self, offsets, baud, amp_end, lengths):
        L = _cabi.lib()
        device = self.device
        self.offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        self.lengths = None if lengths is None else np.ascontiguousarray(lengths, dtype=np.int64)
        self.B = len(self.offsets) - 1 if self.lengths is None else len(self.lengths)
        if self.lengths is not None and len(self.offsets) != self.B:
            raise ValueError("offsets (capture starts) and lengths must have one entry per capture")
        self.baud = np.ascontiguousarray(np.broadcast_to(np.asarray(baud, dtype=np.int32), (self.B,)))
        self.amp_end = np.ascontiguousarray(np.broadcast_to(np.asarray(amp_end, dtype=np.int32), (self.B,)))
        lens_p = None if self.lengths is None else _cabi.ptr(self.lengths, C.c_int64)
        if self.plan is None:
            plan = C.c_void_p()
            if self.lengths is None:
                _cabi.check(L.afsk_rx_plan_create(device, self.B, _cabi.ptr(self.offsets, C.c_int64),
                                                  _cabi.ptr(self.baud, C.c_int32), _cabi.ptr(self.amp_end, C.c_int32),
                                                  C.byref(plan)))
            else:
                _cabi.check(L.afsk_rx_plan_create_ranges(device, self.B, _cabi.ptr(self.offsets, C.c_int64), lens_p,
                                                         _cabi.ptr(self.baud, C.c_int32), _cabi.ptr(self.amp_end, C.c_int32),
                                                         C.byref(plan)))
            self.plan = plan
        else:
            _cabi.check(L.afsk_rx_plan_reset(self.plan, self.B, _cabi.ptr(self.offsets, C.c_int64), lens_p,
                                             _cabi.ptr(self.baud, C.c_int32), _cabi.ptr(self.amp_end, C.c_int32)))
        po = C.POINTER(C.c_int64)()
        _cabi.check(L.afsk_rx_plan_out_offsets(self.plan, C.byref(po)))
        self.out_off = np.ctypeslib.as_array(po, shape=(self.B + 1,)).copy()
        n = C.c_int(0)
        _cabi.check(L.afsk_rx_plan_launches(self.plan, C.byref(n)))
        self.launches = n.value
        if self.lengths is None:
            self.total_samples = int(self.offsets[-1])
        else:
            self.total_samples = int((self.offsets + self.lengths).max()) if self.B else 0
        out_bytes, res_bytes = int(self.out_off[-1]), 32 * max(self.B, 1)
        if self.d_out is None or self.d_out.nbytes < out_bytes:
            regrow = self.d_out is not None
            if regrow:
                self.d_out.close()
            self.d_out = DeviceBuffer(device, out_bytes + (out_bytes // 4 if regrow else 0))
            # payloads are written at capacity offsets: keep the gaps between them defined (zero; stale bytes
            # of an earlier layout after a reset are as good)
            _cabi.check(L.afsk_memset(device, C.c_void_p(self.d_out.ptr), 0, max(self.d_out.nbytes, 16), None))
            _cabi.stream_sync(device)
        if self.d_res is None or self.d_res.nbytes < res_bytes:
            regrow = self.d_res is not None
            if regrow:
                self.d_res.close()
            self.d_res = DeviceBuffer(device, res_bytes + (res_bytes // 4 if regrow else 0))

    def close(self):
        if getattr(self, "plan", None):
            self._destroy(self.plan)
            self.plan = None
        for b in ("d_out", "d_res", "d_samples"):
            buf = getattr(self, b, None)
            if buf is not None:
                buf.close()

    __del__ = close

    def upload(self, samples: np.ndarray, stream=None):
        samples = np.ascontiguousarray(samples, dtype=np.int16)
        if len(samples) < self.total_samples:
            raise ValueError(f"samples holds {len(samples)} frames, the batch layout needs {self.total_samples}")
        self.ensure_samples()
        self.d_samples.upload(samples[:self.total_samples], stream)
        self._ext_ptr = None

    def ensure_samples(self):
        """The session's own device sample buffer, (re)allocated when the layout outgrew it."""
        need = (self.total_samples * 2 + 15) // 16 * 16 + 16
        if self.d_samples is None or self.d_samples.nbytes < need:
            regrow = self.d_samples is not None
            if regrow:
                self.d_samples.close()
            self.d_samples = DeviceBuffer(self.device, need + (need // 4 if regrow else 0))
        return self.d_samples

    def bind(self, device_ptr: int, nsamples: int | None = None):
        """Use caller-owned device samples (16-byte aligned, padded to 16 bytes past the end).
        ``nsamples``: frames the caller's buffer holds — checked against the batch layout so that a
        short buffer is a Python error, not an out-of-bounds device read."""
        if int(device_ptr) % 16:
            raise ValueError("device sample pointer must be 16-byte aligned")
        if nsamples is not None and int(nsamples) < self.total_samples:
            raise ValueError(f"bound buffer holds {int(nsamples)} frames, the batch layout needs {self.total_samples}")
        self._ext_ptr = int(device_ptr)

    def run(self, stream=None):
        p = self._ext_ptr if self._ext_ptr is not None else self.d_samples.ptr
        _cabi.check(_cabi.lib().afsk_rx_decode(self.plan, C.c_void_p(p), C.c_void_p(self.d_out.ptr),
                                               C.c_void_p(self.d_res.ptr), C.c_void_p(stream or 0)))

    def set_timing(self, enable: bool):
        _cabi.check(_cabi.lib().afsk_rx_plan_set_timing(self.plan, 1 if enable else 0))

    def demod_time(self):
        """(summed k_demod milliseconds, launches) since the last query; synchronizes."""
        ms, n = C.c_float(0), C.c_int(0)
        _cabi.check(_cabi.lib().afsk_rx_plan_demod_time(self.plan, C.byref(ms), C.byref(n)))
        return ms.value, n.value

    def download(self, stream=None, res_host: np.ndarray | None = None, blob_host: np.ndarray | None = None,
                 sync: bool = True) -> RxBatch:
        res = res_host if res_host is not None else np.zeros(self.B, dtype=_cabi.RX_RESULT_DTYPE)
        blob = blob_host if blob_host is not None else np.zeros(int(self.out_off[-1]), dtype=np.uint8)
        if self.B:
            self.d_res.download(res, stream)
            self.d_out.download(blob, stream)
        if sync:
            _cabi.stream_sync(self.device, stream)
        return RxBatch(res, blob, self.out_off)

    def planes(self, capture: int):
        """(bits, quiet) numpy bool arrays of capture's windows after a run — stage-level parity."""
        L = _cabi.lib()
        pp, mw = C.c_void_p(), C.c_int64(0)
        _cabi.check(L.afsk_rx_plan_planes(self.plan, capture, C.byref(pp), C.byref(mw)))
        nw = (mw.value + 31) // 32
        words = np.zeros((max(nw, 1), 2), dtype=np.uint32)
        if nw:
            _cabi.check(L.afsk_memcpy_d2h(self.device, C.c_void_p(words.ctypes.data), pp, nw * 8, None))
        _cabi.stream_sync(self.device)
        unpack = lambda col: np.unpackbits(np.ascontiguousarray(words[:, col]).view(np.uint8),  # noqa: E731
                                           bitorder="little")[:mw.value].astype(bool)
        return unpack(0), unpack(1)


class PipelinedRxSession:
    """Host-buffer decode of a large batch with the PCIe copy and the kernels overlapped.

    The batch is cut into ``chunks`` contiguous capture ranges of about equal size in samples
    (``shard.shard_captures``), each with its own plan over the SAME device sample buffer (the plans
    keep the batch's absolute offsets).  A copy stream uploads range after range; the compute stream
    waits for range j's copy (``afsk_stream_wait_stream``) and decodes it while range j+1 is on the
    link, so the call costs the H2D time plus the LAST range's kernels instead of H2D plus all of them.
    Results land in one RxBatch exactly as from a single plan."""

    def __init__(self, offsets, baud, amp_end, device: int, chunks: int):
        from .shard import shard_captures
        self.device = device
        self.offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        self.B = len(self.offsets) - 1
        self.total_samples = int(self.offsets[-1])
        baud = np.ascontiguousarray(np.broadcast_to(np.asarray(baud, dtype=np.int32), (self.B,)))
        amp_end = np.ascontiguousarray(np.broadcast_to(np.asarray(amp_end, dtype=np.int32), (self.B,)))
        self.ranges = [(lo, hi) for lo, hi in shard_captures(np.diff(self.offsets), chunks) if hi > lo]
        self.sessions = [RxSession(self.offsets[lo:hi + 1], baud[lo:hi], amp_end[lo:hi], device) for lo, hi in self.ranges]
        self.d_samples = DeviceBuffer(device, (self.total_samples * 2 + 15) // 16 * 16 + 16)
        for sess in self.sessions:
            sess.bind(self.d_samples.ptr)
        self.copy_stream = _cabi.stream_create(device)
        self.compute_stream = _cabi.stream_create(device)
        self.launches = sum(sess.launches for sess in self.sessions)
        # one host result set for the whole batch; every range downloads into its slice
        self.res_lo, self.blob_lo, self.out_off = self.merged_layout([sess.out_off for sess in self.sessions])
        # pinned staging for the results: the D2H copies are truly asynchronous (range j's results travel
        # while range j+1 is still uploading — the link is full duplex).  The batch handed to the caller
        # OWNS its arrays (copied out of the staging set: ~0.1 % of the sample bytes), so a caller may keep
        # any field view for as long as it likes while the staging set is reused by the next decode.
        self._stage = (_cabi.PinnedArray((max(self.B, 1),), _cabi.RX_RESULT_DTYPE),
                       _cabi.PinnedArray((max(int(self.blob_lo[-1]), 1),), np.uint8))
        # GPUs that share a host link take turns copying (h2d_gate.py; None on boxes where every GPU has its own)
        from .h2d_gate import make_gate
        self.gate = make_gate(device)
        _cabi.stream_sync(device)          # plan set-up (default stream) is complete before the side streams run

    @staticmethod
    def merged_layout(sub_out_offs):
        """Per-range payload offsets (each starting at 0, length B_j + 1) -> (first result index of every
        range, first blob byte of every range, payload offsets of the whole batch)."""
        res_lo = np.cumsum([0] + [len(o) - 1 for o in sub_out_offs]).astype(np.int64)
        blob_lo = np.cumsum([0] + [int(o[-1]) for o in sub_out_offs]).astype(np.int64)
        out_off = np.concatenate([np.asarray(o[:-1], dtype=np.int64) + blob_lo[j] for j, o in enumerate(sub_out_offs)] +
                                 [blob_lo[-1:]]).astype(np.int64)
        return res_lo, blob_lo, out_off

    def decode(self, samples: np.ndarray) -> RxBatch:
        """The returned batch owns its arrays (nothing in it aliases this session's buffers)."""
        samples = np.ascontiguousarray(samples, dtype=np.int16)
        if len(samples) < self.total_samples:
            raise ValueError(f"samples holds {len(samples)} frames, the batch layout needs {self.total_samples}")
        res, blob = (h.array for h in self._stage)
        for j, ((lo, hi), sess) in enumerate(zip(self.ranges, self.sessions)):
            a, b = int(self.offsets[lo]), int(self.offsets[hi])
            if b > a and self.gate is not None:
                with self.gate:            # the link is this GPU's for the length of the copy
                    self.d_samples.upload(samples[a:b], self.copy_stream, offset=2 * a)
                    _cabi.stream_sync(self.device, self.copy_stream)
            elif b > a:
                self.d_samples.upload(samples[a:b], self.copy_stream, offset=2 * a)
            _cabi.stream_wait_stream(self.device, self.compute_stream, self.copy_stream)
            sess.run(self.compute_stream)
            sess.download(self.compute_stream, res[self.res_lo[j]:self.res_lo[j + 1]],
                          blob[self.blob_lo[j]:self.blob_lo[j + 1]], sync=False)
        _cabi.stream_sync(self.device, self.compute_stream)
        return RxBatch(res[:self.B].copy(), blob[:int(self.blob_lo[-1])].copy(), self.out_off)

    def close(self):
        for sess in getattr(self, "sessions", []):
            sess.close()
        self.sessions = []
        if getattr(self, "d_samples", None) is not None:
            self.d_samples.close()
            self.d_samples = None
        for name in ("copy_stream", "compute_stream"):
            st = getattr(self, name, None)
            if st:
                _cabi.stream_destroy(self.device, st)
                setattr(self, name, None)
        for h in getattr(self, "_stage", ()):
            h.close()
        self._stage = ()
        if getattr(self, "gate", None) is not None:
            self.gate.close()
            self.gate = None

    __del__ = close


class ShardedRxSession:
    """ONE corpus decoded on several GPUs from one process (SURVEY §8e: captures are independent,
    afskmodem.py:420-430, so there is no exchange step).

    The corpus is cut into contiguous capture ranges balanced by predicted time
    (``shard.capture_cost`` -> ``shard.shard_captures``), one per device.  Every device gets its own
    host thread, streams and session over its range (a PipelinedRxSession when the range is large, so
    its PCIe copy overlaps its kernels); the per-device results are gathered on the host into ONE
    RxBatch in corpus order.  No collective touches the data path; ctypes releases the GIL during
    every library call, so the device threads really run side by side."""

    def __init__(self, offsets, baud, amp_end, devices, pipeline: int | None = None, weights=None):
        from .shard import capture_cost, shard_captures
        self.devices = [int(d) for d in devices]
        if not self.devices:
            raise ValueError("devices must name at least one GPU")
        for d in self.devices:
            _cabi.require_device(d)
        self.offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        self.B = len(self.offsets) - 1
        self.total_samples = int(self.offsets[-1])
        baud = np.ascontiguousarray(np.broadcast_to(np.asarray(baud, dtype=np.int32), (self.B,)))
        amp_end = np.ascontiguousarray(np.broadcast_to(np.asarray(amp_end, dtype=np.int32), (self.B,)))
        lengths = np.diff(self.offsets)
        self.weights = capture_cost(lengths, baud, resident=False) if weights is None else np.asarray(weights, np.float64)
        self.ranges = shard_captures(lengths, len(self.devices), self.weights)
        self.sessions = []
        for dev, (lo, hi) in zip(self.devices, self.ranges):
            sub = self.offsets[lo:hi + 1] - self.offsets[lo]
            nbytes = int(sub[-1]) * 2
            k = pipeline
            if k is None:
                k = min(PIPELINE_CHUNKS, (hi - lo) // 4) if nbytes >= PIPELINE_MIN_BYTES else 1
            if hi <= lo:
                self.sessions.append(None)
            elif k > 1:
                self.sessions.append(PipelinedRxSession(sub, baud[lo:hi], amp_end[lo:hi], dev, k))
            else:
                self.sessions.append(RxSession(sub, baud[lo:hi], amp_end[lo:hi], dev))
        self.launches = sum(s.launches for s in self.sessions if s is not None)
        self.device_ms = [0.0] * len(self.devices)     # host wall time of every device's last decode

    def _decode_one(self, j: int, samples: np.ndarray, out: list, errs: list):
        import time
        try:
            t0 = time.perf_counter()
            s = self.sessions[j]
            lo, hi = self.ranges[j]
            part = samples[int(self.offsets[lo]):int(self.offsets[hi])]
            if s is None:
                out[j] = None
            elif isinstance(s, PipelinedRxSession):
                out[j] = s.decode(part)
            else:
                s.upload(part)
                s.run()
                out[j] = s.download()
            self.device_ms[j] = (time.perf_counter() - t0) * 1e3
        except BaseException as e:  # noqa: BLE001 - re-raised on the calling thread
            errs.append(e)

    def decode(self, samples: np.ndarray) -> RxBatch:
        import threading

        from .shard import merge_rx_parts
        samples = np.ascontiguousarray(samples, dtype=np.int16)
        if len(samples) < self.total_samples:
            raise ValueError(f"samples holds {len(samples)} frames, the batch layout needs {self.total_samples}")
        out, errs = [None] * len(self.devices), []
        threads = [threading.Thread(target=self._decode_one, args=(j, samples, out, errs)) for j in range(1, len(self.devices))]
        for t in threads:
            t.start()
        self._decode_one(0, samples, out, errs)
        for t in threads:
            t.join()
        if errs:
            raise errs[0]
        parts = [(b.results, b.blob, b.out_off) for b in out if b is not None]
        if not parts:
            return RxBatch(np.zeros(0, dtype=_cabi.RX_RESULT_DTYPE), np.zeros(0, np.uint8), np.zeros(1, np.int64))
        return RxBatch(*merge_rx_parts(parts))

    def close(self):
        for s in getattr(self, "sessions", []):
            if s is not None:
                s.close()
        self.sessions = []

    __del__ = close


def _concat(captures):
    """list of int16 arrays -> (concatenated samples with each capture 16-byte aligned, offsets)."""
    lens = np.array([len(c) for c in captures], dtype=np.int64)
    samples = np.concatenate([np.asarray(c, dtype=np.int16) for c in captures]) if len(captures) else \
        np.zeros(0, np.int16)
    offsets = np.zeros(len(captures) + 1, dtype=np.int64)
    np.cumsum(lens, out=offsets[1:])
    return samples, offsets


def read_wav_frames(filename: str) -> np.ndarray:
    """SoundInput.loadFromFile (afskmodem.py:213-217): all frame bytes, paired little-endian signed,
    whatever the header says about channels/width (the reference does not check either)."""
    with wave.open(filename, "rb") as f:
        raw = f.readframes(f.getnframes())
    return np.frombuffer(raw, dtype="<i2", count=len(raw) // 2)


class WavBatch:
    """Frames of many wav files in ONE pinned int16 buffer (CSR offsets), read by the library's host
    thread pool — SoundInput.loadFromFile (afskmodem.py:213-217) for a batch.  Files the native
    reader does not vouch for (status != 0) go through CPython's ``wave`` module exactly like the
    reference, so whatever ``wave.open`` / ``readframes`` raises there is kept per file in ``errors``."""

    def __init__(self, filenames, threads: int = 0):
        L = _cabi.lib()
        self.filenames = list(filenames)
        n = len(self.filenames)
        self._paths, self._keep = _cabi.c_paths(self.filenames)
        self.nsamples = np.zeros(max(n, 1), dtype=np.int64)
        self.data_pos = np.zeros(max(n, 1), dtype=np.int64)
        self.status = np.zeros(max(n, 1), dtype=np.int32)
        self.threads = threads
        _cabi.check(L.afsk_wav_probe(self._paths, n, threads, _cabi.ptr(self.nsamples, C.c_int64),
                                     _cabi.ptr(self.data_pos, C.c_int64), _cabi.ptr(self.status, C.c_int32)))
        self.errors: dict[int, Exception] = {}
        self.fallback: dict[int, np.ndarray] = {}
        for i in np.nonzero(self.status[:n])[0]:
            try:
                self.fallback[int(i)] = read_wav_frames(self.filenames[i])
                self.nsamples[i] = len(self.fallback[int(i)])
            except Exception as e:  # noqa: BLE001 - what the reference's wave.open raises for this file
                self.errors[int(i)] = e
                self.nsamples[i] = 0
        self.offsets = np.zeros(n + 1, dtype=np.int64)
        np.cumsum(self.nsamples[:n], out=self.offsets[1:])
        self.total = int(self.offsets[-1])
        self.pinned = self.array = None

    def __len__(self) -> int:
        return len(self.filenames)

    def read(self, pinned=None, device: int = 0, d_samples: int | None = None, stream=None):
        """Reads every file into ``pinned`` (a ``_cabi.PinnedArray``, allocated when None or too small;
        a plain numpy int16 array also works, for hosts without a GPU); with ``d_samples`` (device
        pointer) each finished span is copied to the GPU while later files are still being read."""
        n = len(self)
        arr = pinned if isinstance(pinned, np.ndarray) else (pinned.array if pinned is not None else None)
        if arr is None or arr.size < self.total + 64:
            pinned = _cabi.PinnedArray((self.total + 64,), np.int16)
            arr = pinned.array
        self.pinned, self.array = pinned, arr
        for i, fr in self.fallback.items():
            arr[self.offsets[i]:self.offsets[i + 1]] = fr
        ns = self.nsamples.copy()
        for i in list(self.fallback) + list(self.errors):
            ns[i] = 0                                   # not read natively (already in place / unreadable)
        st = np.zeros(max(n, 1), dtype=np.int32)
        _cabi.check(_cabi.lib().afsk_wav_load(self._paths, n, self.threads, _cabi.ptr(self.data_pos, C.c_int64),
                                              _cabi.ptr(ns, C.c_int64), _cabi.ptr(self.offsets, C.c_int64),
                                              C.c_void_p(arr.ctypes.data), device,
                                              C.c_void_p(d_samples) if d_samples else None, 0,
                                              C.c_void_p(stream or 0), _cabi.ptr(st, C.c_int32)))
        for i in np.nonzero(st[:n])[0]:
            self.errors[int(i)] = OSError(f"cannot read {self.filenames[i]!r}")
        return arr[:self.total]

    def read_to_device(self, device: int, d_samples: DeviceBuffer, stream=None) -> None:
        """Streams every file through the library's pinned staging ring straight into ``d_samples`` (same
        CSR offsets): no host copy of the corpus is kept and nothing as large as the corpus is pinned, so
        the first call of a process costs what later calls cost.  Returns once all samples are on the device."""
        n = len(self)
        if d_samples.nbytes < 2 * self.total:
            raise ValueError(f"device buffer of {d_samples.nbytes} bytes cannot hold {self.total} samples")
        ns = self.nsamples.copy()
        for i in list(self.fallback) + list(self.errors):
            ns[i] = 0                                   # not read natively (uploaded below / unreadable)
        st = np.zeros(max(n, 1), dtype=np.int32)
        _cabi.check(_cabi.lib().afsk_wav_load(self._paths, n, self.threads, _cabi.ptr(self.data_pos, C.c_int64),
                                              _cabi.ptr(ns, C.c_int64), _cabi.ptr(self.offsets, C.c_int64),
                                              None, device, C.c_void_p(d_samples.ptr), 0,
                                              C.c_void_p(stream or 0), _cabi.ptr(st, C.c_int32)))
        for i, fr in self.fallback.items():             # after the ring's copies: they cover these ranges too
            if len(fr):
                d_samples.upload(np.ascontiguousarray(fr, dtype=np.int16), stream, offset=2 * int(self.offsets[i]))
        if self.fallback:
            _cabi.stream_sync(device, stream)           # the fallback arrays are pageable host memory
        for i in np.nonzero(st[:n])[0]:
            self.errors[int(i)] = OSError(f"cannot read {self.filenames[i]!r}")

    def frames(self, i: int) -> np.ndarray:
        return self.array[self.offsets[i]:self.offsets[i + 1]]


class Receiver:
    """Receiver(baud_rate, amp_start_threshold, amp_end_threshold) — afskmodem.py:274-430.

    Unlike the reference's, an instance keeps state between calls (the plan and device buffers of the
    last batch layout): use one Receiver per thread, or serialise calls on a shared one."""

    def __init__(self, baud_rate: int = 1200, amp_start_threshold: int = 18000,
                 amp_end_threshold: int = 14000, device: int = 0):
        self._bit_frames = int(48000 / baud_rate)                # :277
        self._baud = _check_baud(baud_rate)                      # raises like :280-282
        self._amp_start = amp_start_threshold                    # live path only (:306)
        self._amp_end = amp_end_threshold
        self._device = device
        self._log = Log("afskmodem.Receiver")
        self._cache = None                                       # (key, RxSession) of the last batch layout

    def _session(self, offsets: np.ndarray, dev, baud=None, amp_end=None, chunks: int = 1):
        """Plan + device buffers are kept between calls with the same batch layout (like an FFT
        plan cache): repeated decode_batch calls then pay only H2D, kernels and D2H.
        chunks > 1: a PipelinedRxSession (copy / compute overlap over capture ranges).
        ``dev``: a device index, or a tuple of them (ShardedRxSession)."""
        baud = self._baud if baud is None else np.ascontiguousarray(baud, dtype=np.int32)
        amp_end = _as_int_threshold(self._amp_end) if amp_end is None else \
            np.ceil(np.asarray(amp_end, dtype=np.float64)).astype(np.int32)
        key = (dev, chunks, baud if np.isscalar(baud) else baud.tobytes(),
               amp_end if np.isscalar(amp_end) else amp_end.tobytes(), offsets.tobytes())
        if self._cache is not None and self._cache[0] == key:
            return self._cache[1]
        cached = self._cache[1] if self._cache is not None else None
        if type(cached) is RxSession and not isinstance(dev, tuple) and chunks <= 1 and cached.device == dev:
            # same kind of session on the same GPU: re-target its plan and buffers instead of rebuilding them
            self._cache = None
            try:
                cached.reset(offsets, baud, amp_end)
            except Exception:
                cached.close()
                raise
            self._cache = (key, cached)
            return cached
        self._drop_session()
        if isinstance(dev, tuple):
            s = ShardedRxSession(offsets, baud, amp_end, dev, pipeline=chunks if chunks > 0 else None)
        elif chunks <= 1:
            s = RxSession(offsets, baud, amp_end, dev)
        else:
            s = PipelinedRxSession(offsets, baud, amp_end, dev, chunks)
        self._cache = (key, s)
        return s

    def _drop_session(self):
        """Releases the cached plan and device buffers (the pinned wav staging buffer is kept: it only grows)."""
        if getattr(self, "_cache", None) is not None:
            self._cache[1].close()
            self._cache = None

    def close(self):
        """Releases everything this receiver holds on the device and in pinned host memory."""
        self._drop_session()
        if getattr(self, "_pinned", None) is not None:
            self._pinned.close()
            self._pinned = None

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001 - interpreter shutdown
            pass

    # -- batch API -------------------------------------------------------------------------
    def decode_batch(self, samples, offsets=None, device: int | None = None, baud_rate=None,
                     amp_end_threshold=None, pipeline: int | None = None, devices=None) -> RxBatch:
        """Decode B captures.  ``samples``: list of int16 arrays, or one concatenated int16 array
        with ``offsets`` (B+1, in samples).  ``baud_rate`` / ``amp_end_threshold`` (arrays of B) override
        this receiver's settings per capture for mixed corpora.  ``pipeline``: number of capture ranges
        whose upload and decode are overlapped (None: 8 for batches of 64 MB and more, else 1).
        ``devices``: several GPUs — the corpus is cut into one contiguous range per device, balanced by
        predicted time, decoded side by side and gathered into ONE batch in corpus order
        (ShardedRxSession).  Raises the reference's exceptions only through ``to_python``; statuses < 0
        mark captures on which ``load`` would raise."""
        if offsets is None:
            samples, offsets = _concat(samples)
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        if devices is not None and len(devices) > 1:
            s = self._session(offsets, tuple(int(d) for d in devices), baud_rate, amp_end_threshold,
                              chunks=0 if pipeline is None else max(int(pipeline), 1))
            return s.decode(samples)
        dev = self._device if device is None else device
        if devices is not None and len(devices) == 1:
            dev = int(devices[0])
        if pipeline is None:
            # overlap pays once the copy is much longer than a launch: >= 64 MB of samples, >= 4 captures per range
            big = len(offsets) > 1 and int(offsets[-1]) * 2 >= PIPELINE_MIN_BYTES
            pipeline = min(PIPELINE_CHUNKS, (len(offsets) - 1) // 4) if big else 1
        s = self._session(offsets, dev, baud_rate, amp_end_threshold, chunks=max(int(pipeline), 1))
        if isinstance(s, PipelinedRxSession):
            return s.decode(samples)
        s.upload(samples)
        s.run()
        return s.download()

    def to_python(self, batch: RxBatch, i: int, string: bool = True, log: bool = True):
        """Capture i of a batch as ``load`` would have returned it (F8 return-type rules), with the
        reference's log lines; raises what ``load`` raises."""
        st = int(batch.status[i])
        lg = self._log if log else _NULL_LOG
        if st == _cabi.ST_EXC_WAVELEN:
            raise Exception("Comparing two waveforms of different lengths.")       # :102-103
        if st == _cabi.ST_EXC_INDEX:
            raise IndexError("list index out of range")                            # :332
        if st == _cabi.ST_EXC_BAUD:
            raise Exception("Invalid baud rate.")
        if st == _cabi.ST_NO_CLOCK:
            lg.warn("Failed to recover clock from received signal.")               # :324
            lg.warn("No data.")                                                    # :423
            return b""
        debug = log and _log_level() <= 0        # the stage lines are built only when they would be printed
        if debug:
            lg.debug("Recovered clock. (frame " + str(int(batch.clock[i])) + ")")       # :338
            lg.debug("Training sequence terminated on frame " + str(int(batch.train_end[i])))   # :368
            lg.debug("Decoded " + str(int(batch.nbits[i])) + " bits. (including ECC)")  # :380
        if st == _cabi.ST_NO_DATA:
            lg.warn("No data.")
            return b""
        data = batch.payload(i)
        if debug:
            lg.debug("Decoded " + str(len(data)) + " bytes.")                          # :427
        if string:
            return data.decode("utf-8")                                            # :428-429
        return data

    def load_batch(self, filenames, string: bool = True, errors: str = "raise", threads: int = 0, log: bool = True,
                   keep_host_copy: bool = False):
        """``load`` over many files in one GPU batch: the library's host threads read the wav files
        through a ring of pinned staging slots while finished spans stream to the GPU, then one decode.
        errors="return" puts the exception object in the list instead of raising at the first
        failing file.  keep_host_copy: read into ONE pinned buffer as large as the corpus instead (kept,
        grow-only, in this receiver; ``self.last_wav_batch.array`` then holds the frames)."""
        wb = WavBatch(filenames, threads)
        dev = self._device
        s = self._session(wb.offsets, dev)
        s.ensure_samples()
        s._ext_ptr = None
        if keep_host_copy:
            wb.read(getattr(self, "_pinned", None), dev, s.d_samples.ptr)
            self._pinned = wb.pinned                             # kept (grow-only) for the next batch
            self.last_wav_batch = wb
        else:
            wb.read_to_device(dev, s.d_samples)
        s.run()
        batch = s.download()
        out = []
        for i in range(len(wb)):
            try:
                if i in wb.errors:
                    raise wb.errors[i]
                out.append(self.to_python(batch, i, string, log))
            except Exception as e:  # noqa: BLE001 - mirrors whatever load raises
                if errors == "raise":
                    raise
                out.append(e)
        return out

    # -- reference API ---------------------------------------------------------------------
    def load(self, filename: str, string: bool = True) -> bytes | str:
        """Reads signal from a file, decodes it, then returns it (or fails) — afskmodem.py:420-430."""
        frames = read_wav_frames(filename)
        return self.to_python(self.decode_batch([frames]), 0, string)

    read = load          # README.md:94 name

    def listen_gate(self, stream_samples, timeout: float, device: int | None = None):
        """Receiver.__listen (:299-319) over recorded streams → list of (recorded, start, end)."""
        streams = stream_samples if isinstance(stream_samples, (list, tuple)) else [stream_samples]
        samples, offsets = _concat(streams)
        dev = self._device if device is None else device
        _cabi.require_device(dev)
        d_s = DeviceBuffer(dev, len(samples) * 2 + 32)
        d_r = DeviceBuffer(dev, 24 * len(streams))
        try:
            d_s.upload(samples)
            _cabi.check(_cabi.lib().afsk_rx_gate(dev, C.c_void_p(d_s.ptr), _cabi.ptr(offsets, C.c_int64),
                                                 len(streams), int(np.floor(self._amp_start)),
                                                 _as_int_threshold(self._amp_end), int(timeout * 48000),
                                                 C.c_void_p(d_r.ptr), None))
            r = np.zeros((len(streams), 3), dtype=np.int64)
            d_r.download(r)
            _cabi.stream_sync(dev)
        finally:
            d_s.close()
            d_r.close()
        return [(bool(a), int(b), int(c)) for a, b, c in r]

    def receive_recording(self, stream_samples, timeout: float, string: bool = True) -> bytes | str:
        """``receive`` (:402-417) with the audio device replaced by a recorded int16 stream."""
        self._log.info("Listening...")
        rec, a, b = self.listen_gate(stream_samples, timeout)[0]
        if not rec:
            self._log.warn("Timed out.")
            return b""
        self._log.debug("Recording started")
        self._log.debug("Recording finished")
        frames = np.asarray(stream_samples, dtype=np.int16)[a:b]
        return self.to_python(self.decode_batch([frames]), 0, string)

    def listen_gate_multi(self, stream_samples, timeout: float, device: int | None = None, d_samples=None):
        """Successive ``__listen`` calls (:299-319) of one receiver over ONE recorded stream →
        [(recorded, start, end), ...], one entry per ``receive`` call that returns before the
        recording ends (recorded False = "Timed out.")."""
        x = np.ascontiguousarray(stream_samples, dtype=np.int16)
        dev = self._device if device is None else device
        _cabi.require_device(dev)
        max_calls = max(1, len(x) // 2048)
        offsets = np.array([0, len(x)], dtype=np.int64)
        own = d_samples is None
        d_s = DeviceBuffer(dev, len(x) * 2 + 32) if own else d_samples
        d_r = DeviceBuffer(dev, 24 * max_calls)
        d_c = DeviceBuffer(dev, 16)
        try:
            if own:
                d_s.upload(x)
            _cabi.check(_cabi.lib().afsk_rx_gate_multi(dev, C.c_void_p(d_s.ptr), _cabi.ptr(offsets, C.c_int64), 1,
                                                       int(np.floor(self._amp_start)), _as_int_threshold(self._amp_end),
                                                       int(timeout * 48000), max_calls, C.c_void_p(d_r.ptr),
                                                       C.c_void_p(d_c.ptr), None))
            cnt = np.zeros(4, dtype=np.int32)
            d_c.download(cnt)
            _cabi.stream_sync(dev)
            r = np.zeros((max(int(cnt[0]), 1), 3), dtype=np.int64)
            if cnt[0]:
                d_r.download(r)
                _cabi.stream_sync(dev)
        finally:
            if own:
                d_s.close()
            d_r.close()
            d_c.close()
        return [(bool(a), int(b), int(c)) for a, b, c in r[:int(cnt[0])]]

    def receive_all(self, stream_samples, timeout: float, string: bool = True, keep_timeouts: bool = False,
                    errors: str = "raise") -> list:
        """What successive ``receive(timeout, string)`` calls (:402-417) of one receiver return over a
        recorded int16 stream holding any number of transmissions: the stream is uploaded once, the
        listen gate cuts it into recordings on the GPU, all recordings are decoded as one batch.
        Timed-out calls (``b""``) are dropped unless ``keep_timeouts``."""
        x = np.ascontiguousarray(stream_samples, dtype=np.int16)
        dev = self._device
        _cabi.require_device(dev)
        d_s = DeviceBuffer(dev, (len(x) * 2 + 15) // 16 * 16 + 32)
        try:
            d_s.upload(x)
            calls = self.listen_gate_multi(x, timeout, dev, d_samples=d_s)
            recs = [(a, b) for rec, a, b in calls if rec]
            batch = None
            if recs:
                sess = RxSession(np.array([a for a, _ in recs], dtype=np.int64), self._baud,
                                 _as_int_threshold(self._amp_end), dev,
                                 lengths=np.array([b - a for a, b in recs], dtype=np.int64))
                try:
                    sess.bind(d_s.ptr)
                    sess.run()
                    batch = sess.download()
                finally:
                    sess.close()
        finally:
            d_s.close()
        return self._receive_values([rec for rec, _, _ in calls], batch, string, keep_timeouts, errors)

    def _receive_values(self, recorded, batch, string: bool, keep_timeouts: bool, errors: str, first: int = 0) -> list:
        """What successive ``receive`` calls return, with the reference's log lines (:402-417): one entry
        per call flagged in ``recorded``; the recorded calls are ``batch``'s captures from ``first`` on, in order."""
        out, k = [], first
        for rec in recorded:
            self._log.info("Listening...")
            if not rec:
                self._log.warn("Timed out.")
                if keep_timeouts:
                    out.append(b"")
                continue
            self._log.debug("Recording started")
            self._log.debug("Recording finished")
            try:
                out.append(self.to_python(batch, k, string))
            except Exception as e:  # noqa: BLE001 - mirrors whatever receive raises
                if errors == "raise":
                    raise
                out.append(e)
            k += 1
        return out

    def open_streams(self, n_streams: int, timeout: float, device: int | None = None, retain: str = "samples") -> StreamReceiver:
        """``receive(timeout)`` called again and again on ``n_streams`` open input streams at once, fed
        piece by piece as the audio arrives (see ``StreamReceiver``; ``retain`` as for ``open_receive_streams``)."""
        return open_receive_streams([self] * int(n_streams), timeout, self._device if device is None else device, retain)

    def receive(self, timeout: float, string: bool = True) -> bytes | str:
        """Live microphone path (:402-417).  Needs an audio device; out of scope for the GPU core —
        record with any tool and use ``receive_recording`` / ``load``."""
        raise RuntimeError("afskmodem_b200 has no live audio input; use receive_recording() or load()")


def open_receive_streams(receivers, timeout, device: int | None = None, retain: str = "samples") -> StreamReceiver:
    """``receive(timeout)`` called again and again on S open input streams at once, channel s by
    ``receivers[s]`` with ``timeout`` (seconds: one for all channels, or S of them).  The same Receiver may
    serve many channels, e.g. ``[rx300] * 2048 + [rx1200] * 2048``.  ``device`` defaults to the first
    receiver's.

    ``retain`` chooses what the device keeps of a recording that is still open.  ``"samples"`` (the default)
    keeps all its samples until it ends: 96 KB per second of audio.  ``"bits"`` demodulates it as it arrives:
    once 4096 frames are in, its clock is recovered, and every push decides its bit windows 32 at a time into
    2 bits per window (1/320 of the samples at 1200 baud); the channel keeps its samples only from its first
    undecided window (less than max(4096, 33 bit lengths) frames).  ``"payload"`` does what ``"bits"`` does and
    also frames the recording as its windows are decided: it finds the training sequence's end, Hamming-decodes
    whole bytes into a payload slot (``pending_payload`` reads them), and keeps only the bit windows it still
    needs; once the first quiet window after the message is found the result is fixed, and the channel keeps no
    windows until the recording ends.  All modes return the same events, results and values.  See
    ``StreamReceiver``."""
    receivers = list(receivers)
    if not receivers:
        raise ValueError("open_receive_streams needs at least one receiver")
    return StreamReceiver(receivers, timeout, receivers[0]._device if device is None else device, retain)


def _timeout_frames(timeout, n: int) -> np.ndarray:
    """receive() timeouts in seconds (one, or n) -> int64 frames; the reference's gate treats a negative timeout
    like 0 (no chunk is examined, :304)"""
    t = [timeout] * n if np.ndim(timeout) == 0 else list(timeout)
    if len(t) != n:
        raise ValueError(f"need one timeout or {n}, got {len(t)}")
    return np.array([max(0, int(float(x) * 48000)) for x in t], dtype=np.int64)


# sample formats of interleaved frames (AFSK_SAMPLE_* of afsk_b200.h)
_FRAME_FORMATS = {np.dtype(np.int16): _cabi.SAMPLE_S16, np.dtype(np.int32): _cabi.SAMPLE_S32,
                  np.dtype(np.float32): _cabi.SAMPLE_F32}


def _frame_format(dtype) -> tuple[np.dtype, int]:
    """dtype (None: int16; a numpy or torch dtype, or its name) -> (numpy dtype, AFSK_SAMPLE_* code)"""
    try:
        dt = np.dtype(np.int16 if dtype is None else str(dtype).removeprefix("torch.") if "torch." in str(dtype) else dtype)
    except TypeError:
        dt = None
    if dt not in _FRAME_FORMATS:
        raise ValueError(f"dtype must be int16, int32 or float32, got {dtype!r}")
    return dt, _FRAME_FORMATS[dt]


def _row_pitch(n: int, S: int, s0: int, s1: int, what: str) -> int:
    """the row pitch (in samples) of an (n, S) window with element strides (s0, s1): rows of unit stride, s0 >= S"""
    if n == 0:                                                  # (an empty array's strides may be anything)
        return S
    if (S > 1 and s1 != 1) or (n > 1 and s0 < S):
        raise ValueError(f"{what} must be rows of unit stride, row_pitch >= {S}: strides ({s0}, {s1}) in samples")
    return int(s0) if n > 1 else S


class StreamEvents:
    """The ``receive`` calls that became final with one push (or ``finish``), ordered by (stream, call):
    numpy arrays ``stream``, ``call``, ``recorded``, ``start``, ``end`` (stream frames of the recording)
    and ``batch``, an RxBatch of the recorded calls' decodes in the same order."""

    def __init__(self, receivers, ev: np.ndarray, batch: RxBatch):
        self._receivers = receivers                             # per channel, as when these calls were made
        self.stream = ev["stream"].astype(np.int64)
        self.call = ev["call"].copy()
        self.recorded = ev["recorded"].astype(bool)
        self.start = ev["start"].copy()
        self.end = ev["end"].copy()
        self.batch = batch

    def __len__(self) -> int:
        return len(self.stream)

    def values(self, string: bool = True, errors: str = "raise") -> list:
        """What each of these ``receive`` calls returned (``b""`` / ``""`` for "Timed out.") with the
        reference's log lines; errors="return" puts the exception a call raises in the list instead."""
        out, i, k, n = [], 0, 0, len(self)
        while i < n:                                            # runs of events whose channels share a Receiver
            rx, j = self._receivers[self.stream[i]], i + 1
            while j < n and self._receivers[self.stream[j]] is rx:
                j += 1
            out += rx._receive_values(self.recorded[i:j], self.batch, string, True, errors, first=k)
            k += int(self.recorded[i:j].sum())
            i = j
        return out


class StreamReceiver:
    """Continuous reception on S channels at once (``open_receive_streams``, ``Receiver.open_streams``).  Each
    channel behaves like its own reference Receiver calling ``receive(timeout)`` again and again on its own open input stream
    (afskmodem.py:283, 299-319, 402-417).  ``push`` appends the next piece of every channel (any length,
    including 0) and returns the calls that became final with it, already decoded: a call that timed
    out, or a recording whose closing quiet chunk has arrived.  A recording still open stays on the
    device.  ``finish`` ends the streams of all or some channels (a pending recording ends at its last full
    chunk, a call that has neither opened nor timed out is dropped); their next push starts new streams, which
    may be received with other settings.  Over any way
    of cutting a stream into pushes, the events of all pushes plus ``finish`` are ``listen_gate_multi``
    over the whole stream, and their values ``receive_all(stream, keep_timeouts=True)``."""

    RETAIN = {"samples": 0, "bits": 1, "payload": 2}             # AFSK_RETAIN_SAMPLES / _BITS / _PAYLOAD

    def __init__(self, receivers, timeout, device: int = 0, retain: str = "samples"):
        if retain not in self.RETAIN:
            raise ValueError(f"retain must be 'samples', 'bits' or 'payload', got {retain!r}")
        _cabi.require_device(device)
        self.receivers, self.S, self.device = tuple(receivers), len(receivers), device
        self.timeout_frames = _timeout_frames(timeout, self.S)
        self._destroy = _cabi.lib().afsk_rx_streams_destroy
        h = C.c_void_p()
        b, a0, a1 = self._settings(self.receivers)
        _cabi.check(_cabi.lib().afsk_rx_streams_create_each(device, self.S, _cabi.ptr(b, C.c_int32), _cabi.ptr(a0, C.c_int32),
                                                             _cabi.ptr(a1, C.c_int32), _cabi.ptr(self.timeout_frames, C.c_int64),
                                                             C.byref(h)))
        self._h = h
        self._pinned = None
        self.retain = retain
        if retain != "samples":
            _cabi.check(_cabi.lib().afsk_rx_streams_set_retention(h, self.RETAIN[retain]))

    @property
    def receiver(self) -> Receiver:
        """channel 0's Receiver (every channel's for ``Receiver.open_streams``)"""
        return self.receivers[0]

    @staticmethod
    def _settings(receivers):
        """int32 arrays (baud, amp_start, amp_end) of the receivers, as the gate and the decoder use them"""
        return (np.array([r._baud for r in receivers], np.int32), np.array([int(np.floor(r._amp_start)) for r in receivers], np.int32),
                np.array([_as_int_threshold(r._amp_end) for r in receivers], np.int32))

    def close(self):
        if getattr(self, "_h", None):
            self._destroy(self._h)
            self._h = None
        if getattr(self, "_pinned", None) is not None:
            self._pinned.close()
            self._pinned = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def _staging(self, n: int) -> np.ndarray:
        """the grow-only pinned int16 buffer host input is copied into (asynchronous copy to the device), >= n samples"""
        if self._pinned is None or self._pinned.array.size < n:
            if self._pinned is not None:
                self._pinned.close()
            self._pinned = _cabi.PinnedArray((max(n + n // 4, 16),), np.int16)
        return self._pinned.array

    def _host_input(self, pieces) -> tuple[np.ndarray, np.ndarray]:
        """S host pieces -> the pinned staging buffer and offsets."""
        offsets = np.zeros(len(pieces) + 1, dtype=np.int64)
        np.cumsum([len(p) for p in pieces], out=offsets[1:])
        buf = self._staging(int(offsets[-1]))
        for p, a, b in zip(pieces, offsets[:-1], offsets[1:]):
            buf[a:b] = p
        return buf, offsets

    def push(self, samples, offsets=None, stream=None) -> StreamEvents:
        """``samples``: a list of S int16 arrays; or one int16 array (numpy, or a CUDA torch tensor on this
        receiver's device) holding the S pieces concatenated, with ``offsets`` (S+1, CSR)."""
        if offsets is None:
            if len(samples) != self.S:
                raise ValueError(f"push needs one piece per stream ({self.S}), got {len(samples)}")
            arr, offsets = self._host_input(samples)
            return self._run(arr.ctypes.data, 0, offsets, stream)
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        if len(offsets) != self.S + 1:
            raise ValueError(f"offsets must have S + 1 = {self.S + 1} entries, got {len(offsets)}")
        if hasattr(samples, "data_ptr"):                       # a torch tensor: passed by device pointer
            if not samples.is_cuda or samples.device.index != self.device:
                raise ValueError(f"device samples must live on cuda:{self.device}")
            if str(samples.dtype) != "torch.int16" or not samples.is_contiguous():
                raise ValueError("device samples must be a contiguous int16 tensor")
            if int(offsets[-1]) > samples.numel():
                raise ValueError(f"tensor holds {samples.numel()} frames, the offsets need {int(offsets[-1])}")
            return self._run(samples.data_ptr(), 1, offsets, stream)
        arr = np.ascontiguousarray(samples, dtype=np.int16)
        if int(offsets[-1]) > len(arr):
            raise ValueError(f"samples holds {len(arr)} frames, the offsets need {int(offsets[-1])}")
        return self._run(arr.ctypes.data, 0, offsets, stream)

    def push_interleaved(self, frames, stream=None, dtype=None) -> StreamEvents:
        """``push`` of the next n frames of every channel, given interleaved as a multi-channel sound card
        delivers them: frame f of channel s is ``frames[f, s]``.  ``dtype`` is the sample format: int16 (the default),
        int32 or float32, converted to int16 by the rules of ``afsk_b200.h`` (int32: the top 16 bits; float32:
        ``clip(rint(x * 32768), -32768, 32767)``, NaN -> 0).  ``frames``: an (n, S) numpy array of that dtype whose
        rows may be a window of wider frames, strides (row_pitch * itemsize, itemsize) with row_pitch >= S (such as
        ``card[:, c0:c0 + S]``), or a C-contiguous (n * S,) one; any buffer (bytes, bytearray, memoryview) of
        n * S little-endian samples, which is what pyaudio's ``Stream.read(n)`` returns for ``channels=S``; or a CUDA
        tensor of that dtype on this receiver's device, (n, S) with strides (row_pitch, 1) or contiguous (n * S,),
        read in place.  Host input is copied once, packed and still in its format, into a pinned buffer; the GPU
        converts and de-interleaves it.  Returns what ``push([x[:, s] for s in range(S)])`` returns, x the frames
        converted to int16."""
        S = self.S
        dt, fmt = _frame_format(dtype)
        if hasattr(frames, "data_ptr"):                         # a torch tensor: passed by device pointer
            if not frames.is_cuda or frames.device.index != self.device:
                raise ValueError(f"device frames must live on cuda:{self.device}")
            if str(frames.dtype) != f"torch.{dt.name}":
                raise ValueError(f"device frames must be a {dt.name} tensor (dtype=), got {frames.dtype}")
            if frames.dim() == 1 and frames.is_contiguous() and frames.numel() % S == 0:
                n, pitch = frames.numel() // S, S
            elif frames.dim() == 2 and frames.shape[1] == S:
                n, pitch = frames.shape[0], _row_pitch(frames.shape[0], S, frames.stride(0), frames.stride(1), "device frames")
            else:
                raise ValueError(f"device frames must have shape (n, {S}) or (n * {S},), got {tuple(frames.shape)}")
            return self._run_frames(frames.data_ptr(), fmt, 1, n, pitch, stream)
        if isinstance(frames, np.ndarray):
            if frames.dtype != dt:
                raise ValueError(f"host frames must be a {dt.name} array (dtype=), got {frames.dtype}")
            if frames.ndim == 1 and frames.flags.c_contiguous and frames.size % S == 0:
                src = frames.reshape(-1, S)
            elif frames.ndim == 2 and frames.shape[1] == S and all(x % dt.itemsize == 0 for x in frames.strides):
                _row_pitch(frames.shape[0], S, frames.strides[0] // dt.itemsize, frames.strides[1] // dt.itemsize, "host frames")
                src = frames
            else:
                raise ValueError(f"host frames must have shape (n, {S}) with rows of unit stride, or (n * {S},), got "
                                 f"{frames.shape} with strides {frames.strides}")
        else:
            mv = memoryview(frames).cast("B")
            if mv.nbytes % (dt.itemsize * S):
                raise ValueError(f"{mv.nbytes} bytes are not whole frames of {S} {dt.name} samples")
            src = np.frombuffer(mv, dtype=dt.newbyteorder("<")).reshape(-1, S)
        n = src.shape[0]
        nbytes = n * S * dt.itemsize
        buf = self._staging((nbytes + 1) // 2).view(np.uint8)[:nbytes].view(dt).reshape(n, S)
        buf[...] = src
        return self._run_frames(buf.ctypes.data, fmt, 0, n, S, stream)

    def _run_frames(self, ptr: int, fmt: int, on_device: int, n_frames: int, pitch: int, stream) -> StreamEvents:
        n = C.c_int64(0)
        _cabi.check(_cabi.lib().afsk_rx_streams_push_frames(self._h, C.c_void_p(ptr), fmt, on_device, n_frames, pitch,
                                                             C.c_void_p(stream or 0), C.byref(n)))
        return self._events(n.value)

    def finish(self, streams=None, receivers=None, timeout=None, stream=None) -> StreamEvents:
        """Ends the streams of the channels ``streams`` (default: all) and returns their final calls.  Each of
        them then starts a new stream at its next push, received by ``receivers`` (one Receiver, or one per
        listed channel) with ``timeout`` (seconds: one, or one per listed channel); either one left out keeps
        the channel's current setting.  Other channels are untouched."""
        n = C.c_int64(0)
        if streams is None and receivers is None and timeout is None:
            _cabi.check(_cabi.lib().afsk_rx_streams_finish(self._h, C.c_void_p(stream or 0), C.byref(n)))
            return self._events(n.value)
        ids = np.arange(self.S, dtype=np.int32) if streams is None else np.ascontiguousarray(streams, dtype=np.int32).reshape(-1)
        new = None
        if receivers is not None or timeout is not None:
            cur = [i if 0 <= i < self.S else 0 for i in ids]      # (the library rejects a channel out of range)
            if receivers is None:
                rxs = [self.receivers[i] for i in cur]
            else:
                rxs = [receivers] * len(ids) if isinstance(receivers, Receiver) else list(receivers)
            if len(rxs) != len(ids):
                raise ValueError(f"finish needs one receiver per listed channel ({len(ids)}), got {len(rxs)}")
            t = self.timeout_frames[cur] if timeout is None else _timeout_frames(timeout, len(ids))
            new = (rxs, t) + self._settings(rxs)
        args = [None] * 4 if new is None else [_cabi.ptr(new[2], C.c_int32), _cabi.ptr(new[3], C.c_int32),
                                               _cabi.ptr(new[4], C.c_int32), _cabi.ptr(new[1], C.c_int64)]
        _cabi.check(_cabi.lib().afsk_rx_streams_finish_some(self._h, len(ids), _cabi.ptr(ids, C.c_int32), *args,
                                                             C.c_void_p(stream or 0), C.byref(n)))
        ev = self._events(n.value)                               # decoded with the settings of the streams that ended
        if new is not None:
            rx = list(self.receivers)
            for i, r, t in zip(ids, new[0], new[1]):
                rx[i] = r
                self.timeout_frames[i] = t
            self.receivers = tuple(rx)
        return ev

    def _run(self, ptr: int, on_device: int, offsets: np.ndarray, stream) -> StreamEvents:
        n = C.c_int64(0)
        _cabi.check(_cabi.lib().afsk_rx_streams_push(self._h, C.c_void_p(ptr), on_device, _cabi.ptr(offsets, C.c_int64),
                                                      C.c_void_p(stream or 0), C.byref(n)))
        return self._events(n.value)

    def _events(self, n: int) -> StreamEvents:
        ev = np.zeros(n, dtype=_cabi.STREAM_EVENT_DTYPE)
        res = np.zeros(n, dtype=_cabi.RX_RESULT_DTYPE)
        off = np.zeros(n + 1, dtype=np.int64)
        blob = np.zeros(0, dtype=np.uint8)
        if n:
            pe, pr, pp, po = C.c_void_p(), C.c_void_p(), C.c_void_p(), C.c_void_p()
            _cabi.check(_cabi.lib().afsk_rx_streams_events(self._h, C.byref(pe), C.byref(pr), C.byref(pp), C.byref(po)))
            C.memmove(ev.ctypes.data, pe, ev.nbytes)
            C.memmove(res.ctypes.data, pr, res.nbytes)
            C.memmove(off.ctypes.data, po, off.nbytes)
            blob = np.zeros(int(off[-1]), dtype=np.uint8)
            if len(blob):
                C.memmove(blob.ctypes.data, pp, blob.nbytes)
        rec = ev["recorded"] != 0
        out_off = np.append(off[:-1][rec], off[-1]).astype(np.int64)
        return StreamEvents(self.receivers, ev, RxBatch(res[rec], blob, out_off))

    def state(self, s: int) -> tuple[int, int, int]:
        """(frames pushed, start of the pending recording or -1, frames retained on the device) of stream s."""
        a, b, c = C.c_int64(0), C.c_int64(0), C.c_int64(0)
        _cabi.check(_cabi.lib().afsk_rx_streams_state(self._h, int(s), C.byref(a), C.byref(b), C.byref(c)))
        return a.value, b.value, c.value

    def counters(self) -> dict:
        """Since this receiver was opened: kernel launches (decodes included), frames moved to keep retained
        samples (appends aside) and whole-arena compactions; in bits and payload mode also the plane words moved to
        keep open recordings' planes and the plane arena's compactions (both 0 in samples mode); in payload mode the
        decoded bytes moved to keep open recordings' payloads and the payload arena's compactions (both 0 otherwise)."""
        a, b, c, d, e, f, g = (C.c_int64(0) for _ in range(7))
        L = _cabi.lib()
        _cabi.check(L.afsk_rx_streams_counters(self._h, C.byref(a), C.byref(b), C.byref(c)))
        _cabi.check(L.afsk_rx_streams_plane_counters(self._h, C.byref(d), C.byref(e)))
        _cabi.check(L.afsk_rx_streams_payload_counters(self._h, C.byref(f), C.byref(g)))
        return {"launches": a.value, "moved_frames": b.value, "compactions": c.value, "moved_plane_words": d.value,
                "plane_compactions": e.value, "moved_payload_bytes": f.value, "payload_compactions": g.value}

    def pending_bits(self, s: int) -> tuple[int, int]:
        """(stored clock, windows decided so far) of stream s's pending recording in bits mode: (-1, 0) while its
        clock is not recovered or no recording is pending; the windows are 0 in samples mode."""
        a, b = C.c_int32(0), C.c_int64(0)
        _cabi.check(_cabi.lib().afsk_rx_streams_pending_bits(self._h, int(s), C.byref(a), C.byref(b)))
        return a.value, b.value

    def pending_planes(self, s: int) -> tuple[int, np.ndarray, np.ndarray]:
        """(first_window, bits, quiet) of stream s's pending recording in bits or payload mode: the decision and quiet
        flags of the windows it keeps on the device, windows first_window, first_window + 1, ... of the recording
        (window k starts at frame ``state(s)[1] + pending_bits(s)[0] + k * bit length``), up to the windows decided.
        Empty in samples mode, with no recording pending, before its clock is recovered, or in payload mode once its
        result is fixed.  For diagnostics and stage-level tests (one device-to-host copy)."""
        L = _cabi.lib()
        pp, first, n = C.c_void_p(), C.c_int64(0), C.c_int64(0)
        _cabi.check(L.afsk_rx_streams_pending_planes(self._h, int(s), C.byref(pp), C.byref(first), C.byref(n)))
        nw = (n.value + 31) // 32
        words = np.zeros((max(nw, 1), 2), dtype=np.uint32)
        if nw:
            _cabi.check(L.afsk_memcpy_d2h(self.device, C.c_void_p(words.ctypes.data), pp, nw * 8, None))
            _cabi.stream_sync(self.device)
        unpack = lambda col: np.unpackbits(np.ascontiguousarray(words[:, col]).view(np.uint8),  # noqa: E731
                                           bitorder="little")[:n.value].astype(bool)
        return first.value, unpack(0), unpack(1)

    def pending_payload(self, s: int) -> tuple[int, int, bool, bytes]:
        """(train_end, nbits, ended, bytes) of stream s's pending recording in payload mode, as framed so far:
        train_end is -1 until the end of the training sequence is seen, nbits the coded bits framed after it, ended
        True once the first quiet window after it was found (the call's result is then fixed), and bytes the payload
        decoded so far, a prefix of what the call returns.  (-1, 0, False, b"") in other modes, with no recording
        pending, or before its clock is recovered."""
        L = _cabi.lib()
        te, nb, n = C.c_int64(0), C.c_int64(0), C.c_int64(0)
        ended = C.c_int32(0)
        _cabi.check(L.afsk_rx_streams_pending_payload(self._h, int(s), C.byref(te), C.byref(nb), C.byref(ended), None, 0, C.byref(n)))
        buf = (C.c_uint8 * max(n.value, 1))()
        if n.value > 0:
            _cabi.check(L.afsk_rx_streams_pending_payload(self._h, int(s), C.byref(te), C.byref(nb), C.byref(ended), buf, n.value,
                                                          C.byref(n)))
        return te.value, nb.value, bool(ended.value), bytes(buf[:n.value])

    def arena_bytes(self) -> int:
        """Device bytes this receiver holds (sample arenas, plane arenas in bits and payload mode, payload arenas
        in payload mode, staging, scratch)."""
        n = C.c_int64(0)
        _cabi.check(_cabi.lib().afsk_rx_streams_arena_bytes(self._h, C.byref(n)))
        return n.value


class _NullLog:
    def debug(self, m): pass
    def info(self, m): pass
    def warn(self, m): pass


_NULL_LOG = _NullLog()


# --------------------------------------------------------------------------- transmitter ----
class TxBatch:
    def __init__(self, samples: np.ndarray, out_off: np.ndarray, out_len: np.ndarray):
        self.samples, self.out_off, self.out_len = samples, out_off, out_len

    def __len__(self) -> int:
        return len(self.out_len)

    def frames(self, i: int) -> np.ndarray:
        o = int(self.out_off[i])
        return self.samples[o:o + int(self.out_len[i])]


class TxSession:
    """Plan + device buffers for one batch of payloads on one GPU (see RxSession)."""

    def __init__(self, payloads, baud, ts_cycles, device: int = 0):
        _cabi.require_device(device)
        L = _cabi.lib()
        self.device = device
        self.B = len(payloads)
        lens = np.array([len(p) for p in payloads], dtype=np.int64)
        self.pay_off = np.zeros(self.B + 1, dtype=np.int64)
        np.cumsum(lens, out=self.pay_off[1:])
        self.payload = np.frombuffer(b"".join(bytes(p) for p in payloads), dtype=np.uint8).copy() \
            if self.pay_off[-1] else np.zeros(1, dtype=np.uint8)
        self.baud = np.ascontiguousarray(np.broadcast_to(np.asarray(baud, dtype=np.int32), (self.B,)))
        self.ts = np.ascontiguousarray(np.broadcast_to(np.asarray(ts_cycles, dtype=np.int64), (self.B,)))
        plan = C.c_void_p()
        rc = L.afsk_tx_plan_create(device, self.B, _cabi.ptr(self.pay_off, C.c_int64), _cabi.ptr(self.baud, C.c_int32),
                                   _cabi.ptr(self.ts, C.c_int64), _cabi.ptr(self.payload, C.c_uint8), C.byref(plan))
        if rc == _cabi.AFSK_E_BAUD:
            raise Exception("Invalid baud rate.")
        if rc == _cabi.AFSK_E_UNSUPPORTED:
            raise NotImplementedError(L.afsk_last_error().decode())
        _cabi.check(rc)
        self.plan = plan
        self._destroy = L.afsk_tx_plan_destroy
        po, pl = C.POINTER(C.c_int64)(), C.POINTER(C.c_int64)()
        _cabi.check(L.afsk_tx_plan_out_offsets(plan, C.byref(po), C.byref(pl)))
        self.out_off = np.ctypeslib.as_array(po, shape=(self.B + 1,)).copy()
        # an empty batch has no length array behind the pointer (std::vector::data() of nothing)
        self.out_len = np.ctypeslib.as_array(pl, shape=(self.B,)).copy() if self.B else np.zeros(0, np.int64)
        self.d_pay = DeviceBuffer(device, len(self.payload))
        self.d_out = DeviceBuffer(device, int(self.out_off[-1]) * 2)

    def close(self):
        if getattr(self, "plan", None):
            self._destroy(self.plan)
            self.plan = None
        for b in ("d_pay", "d_out"):
            buf = getattr(self, b, None)
            if buf is not None:
                buf.close()

    __del__ = close

    def upload(self, stream=None):
        self.d_pay.upload(self.payload, stream)

    def run(self, stream=None):
        _cabi.check(_cabi.lib().afsk_tx_synth(self.plan, C.c_void_p(self.d_pay.ptr), C.c_void_p(self.d_out.ptr),
                                              C.c_void_p(stream or 0)))

    def download(self, stream=None, host: np.ndarray | None = None) -> TxBatch:
        out = host if host is not None else np.zeros(int(self.out_off[-1]), dtype=np.int16)
        if len(out):
            self.d_out.download(out, stream)
        _cabi.stream_sync(self.device, stream)
        return TxBatch(out, self.out_off, self.out_len)


def write_wav_frames(filename: str, frames: np.ndarray) -> None:
    """SoundOutput.writeToFile (afskmodem.py:256-263): 1 channel, 16 bit, 48 kHz."""
    with wave.open(filename, "wb") as f:
        f.setnchannels(1)
        f.setsampwidth(2)
        f.setframerate(48000)
        f.writeframes(np.ascontiguousarray(frames, dtype="<i2").tobytes())


def write_wav_batch(filenames, samples: np.ndarray, starts, lengths, threads: int = 0) -> None:
    """SoundOutput.writeToFile (afskmodem.py:256-263) for many files: file i = samples[starts[i] : starts[i] + lengths[i]]."""
    filenames = list(filenames)
    n = len(filenames)
    samples = np.ascontiguousarray(samples, dtype="<i2")
    starts = np.ascontiguousarray(starts, dtype=np.int64)
    lengths = np.ascontiguousarray(lengths, dtype=np.int64)
    if len(starts) < n or len(lengths) < n:
        raise ValueError("starts and lengths must have one entry per file")
    if n and (int(starts[:n].min()) < 0 or int(lengths[:n].min()) < 0 or int((starts[:n] + lengths[:n]).max()) > len(samples)):
        raise ValueError("a file's [start, start + length) range lies outside the sample buffer")
    paths, _keep = _cabi.c_paths(filenames)
    st = np.zeros(max(n, 1), dtype=np.int32)
    _cabi.check(_cabi.lib().afsk_wav_save(paths, n, threads, C.c_void_p(samples.ctypes.data), _cabi.ptr(starts, C.c_int64),
                                          _cabi.ptr(lengths, C.c_int64), _cabi.ptr(st, C.c_int32)))
    for i in np.nonzero(st[:n])[0]:
        if st[i] == 2:
            write_wav_frames(filenames[i], samples[starts[i]:starts[i] + lengths[i]])   # raises like wave does
        else:
            raise OSError(f"cannot write {filenames[i]!r}")


class Transmitter:
    """Transmitter(baud_rate, training_time) — afskmodem.py:436-484."""

    def __init__(self, baud_rate: int = 1200, training_time: float = 0.5, device: int = 0,
                 training_sequence_time: float | None = None):
        if training_sequence_time is not None:                   # README.md:107 spelling
            training_time = training_sequence_time
        self._ts_cycles = int(baud_rate * training_time / 2)     # :438
        self._baud = _check_baud(baud_rate)                      # raises like :439-441
        self._device = device
        self._log = Log("afskmodem.Transmitter")

    @staticmethod
    def _as_bytes(data) -> bytes:
        return data.encode("utf-8") if isinstance(data, str) else bytes(data)     # :473-474, :482-483

    def encode_batch(self, payloads, device: int | None = None, _host=None) -> TxBatch:
        """Frames ``save`` would write for each payload (str or bytes), synthesized on the GPU."""
        s = TxSession([self._as_bytes(p) for p in payloads], self._baud, self._ts_cycles,
                      self._device if device is None else device)
        try:
            s.upload()
            s.run()
            host = None
            if _host is not None:
                host = _host(int(s.out_off[-1]))
            return s.download(host=host)
        finally:
            s.close()

    def _pinned_frames(self, n: int) -> np.ndarray:
        """grow-only pinned staging buffer for save_batch: the D2H copy runs at link speed and the first touch of
        a fresh pageable array (a page fault per 4 KB) is not paid on every call"""
        cur = getattr(self, "_pinned", None)
        if cur is None or cur.array.size < n:
            if cur is not None:
                cur.close()
            self._pinned = _cabi.PinnedArray((max(n + n // 8, 16),), np.int16)
        return self._pinned.array[:n]

    def save_batch(self, payloads, filenames, threads: int = 0) -> None:
        """``save`` for many payloads: one synthesis on the GPU, files written by the library's host
        threads (byte-identical to the reference's wave output)."""
        batch = self.encode_batch(payloads, _host=self._pinned_frames)
        write_wav_batch(filenames, batch.samples, batch.out_off[:-1], batch.out_len, threads)

    def close(self):
        if getattr(self, "_pinned", None) is not None:
            self._pinned.close()
            self._pinned = None

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001 - interpreter shutdown
            pass

    def save(self, data: str | bytes, filename: str):
        """Transmits the given data, saving the resulting audio to a .wav file — afskmodem.py:481-484."""
        write_wav_frames(filename, self.encode_batch([data]).frames(0))

    write = save         # README.md:119 name

    def open_streams(self, n_streams: int, device: int | None = None) -> StreamTransmitter:
        """``transmit`` called again and again on ``n_streams`` open output streams at once, pulled piece by
        piece as the sound card asks for frames (see ``StreamTransmitter``)."""
        return open_transmit_streams([self] * int(n_streams), self._device if device is None else device)

    def transmit(self, data: str | bytes):
        """Live speaker path (:472-478).  Needs an audio device; out of scope — use ``save``."""
        raise RuntimeError("afskmodem_b200 has no live audio output; use save()")


def open_transmit_streams(transmitters, device: int | None = None) -> StreamTransmitter:
    """``transmit`` called again and again on S open output streams at once, channel s by ``transmitters[s]``
    (the same Transmitter may serve many channels).  ``device`` defaults to the first transmitter's.  See
    ``StreamTransmitter``."""
    transmitters = list(transmitters)
    if not transmitters:
        raise ValueError("open_transmit_streams needs at least one transmitter")
    return StreamTransmitter(transmitters, transmitters[0]._device if device is None else device)


class StreamTransmitter:
    """Continuous transmission on S channels at once (``open_transmit_streams``, ``Transmitter.open_streams``).
    Each channel behaves like its own reference Transmitter whose output stream stays open, calling ``transmit(data)`` again and again
    (afskmodem.py:472-478: ``SoundOutput.play`` writes what ``save`` writes, :247-252).  The channels share one
    timeline, pulled ``n`` frames at a time like the periods of a multi-channel sound card.  ``send`` queues
    messages; one starts at ``max(frames pulled, end of its channel's last message)`` and its frames are exactly
    what ``save`` writes for it; every other frame is silence (0).  Only payload bytes are kept on the device:
    each ``pull`` synthesizes its window from them.  ``configure`` gives channels other settings for the messages
    sent to them afterwards."""

    def __init__(self, transmitters, device: int = 0):
        _cabi.require_device(device)
        self.transmitters, self.S, self.device = tuple(transmitters), len(transmitters), device
        self._destroy = _cabi.lib().afsk_tx_streams_destroy
        h = C.c_void_p()
        b, t = self._settings(self.transmitters)
        _cabi.check(_cabi.lib().afsk_tx_streams_create_each(device, self.S, _cabi.ptr(b, C.c_int32), _cabi.ptr(t, C.c_int64),
                                                             C.byref(h)))
        self._h = h
        self._pinned = None

    @property
    def transmitter(self) -> Transmitter:
        """channel 0's Transmitter (every channel's for ``Transmitter.open_streams``)"""
        return self.transmitters[0]

    @staticmethod
    def _settings(transmitters):
        return (np.array([t._baud for t in transmitters], np.int32), np.array([t._ts_cycles for t in transmitters], np.int64))

    def configure(self, streams, transmitters) -> None:
        """Messages sent from now on to channels ``streams`` use ``transmitters`` (one Transmitter, or one per listed
        channel); messages already queued keep their settings."""
        ids = np.ascontiguousarray(streams, dtype=np.int32).reshape(-1)
        txs = [transmitters] * len(ids) if isinstance(transmitters, Transmitter) else list(transmitters)
        if len(txs) != len(ids):
            raise ValueError(f"configure needs one transmitter per listed channel ({len(ids)}), got {len(txs)}")
        b, t = self._settings(txs)
        _cabi.check(_cabi.lib().afsk_tx_streams_configure(self._h, len(ids), _cabi.ptr(ids, C.c_int32), _cabi.ptr(b, C.c_int32),
                                                           _cabi.ptr(t, C.c_int64)))
        tx = list(self.transmitters)
        for i, x in zip(ids, txs):
            tx[i] = x
        self.transmitters = tuple(tx)

    def close(self):
        if getattr(self, "_h", None):
            self._destroy(self._h)
            self._h = None
        if getattr(self, "_pinned", None) is not None:
            self._pinned.close()
            self._pinned = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def send(self, streams, payloads) -> tuple[np.ndarray, np.ndarray]:
        """Queues ``payloads[i]`` (str is UTF-8 encoded, as in ``save``) on channel ``streams[i]``, in list order.
        Returns the int64 arrays (start, end): the timeline frames of each message."""
        data = [Transmitter._as_bytes(p) for p in payloads]
        ids = np.ascontiguousarray(streams, dtype=np.int32).reshape(-1)
        if len(ids) != len(data):
            raise ValueError(f"send needs one stream per payload, got {len(ids)} streams and {len(data)} payloads")
        off = np.zeros(len(data) + 1, dtype=np.int64)
        np.cumsum([len(p) for p in data], out=off[1:])
        blob = np.frombuffer(b"".join(data), dtype=np.uint8) if off[-1] else np.zeros(1, dtype=np.uint8)
        start, end = np.zeros(len(data), np.int64), np.zeros(len(data), np.int64)
        _cabi.check(_cabi.lib().afsk_tx_streams_send(self._h, len(data), _cabi.ptr(ids, C.c_int32), _cabi.ptr(off, C.c_int64),
                                                     _cabi.ptr(blob, C.c_uint8), _cabi.ptr(start, C.c_int64),
                                                     _cabi.ptr(end, C.c_int64)))
        return start, end

    def pull(self, n: int, out=None, stream=None):
        """The next ``n`` frames of every channel.  Default: a host (S, n) int16 array in a grow-only pinned
        buffer, valid until the next pull unless copied.  ``out``: a contiguous CUDA int16 tensor of at least
        S * n elements on this transmitter's device, written row-major (row s = channel s, no padding) and
        returned; nothing past S * n is written."""
        r = self._pull(_cabi.lib().afsk_tx_streams_pull, n, out, stream)
        return r if out is not None else r.reshape(self.S, int(n))

    def pull_interleaved(self, n: int, out=None, stream=None, dtype=None):
        """``pull`` with the window interleaved, as a multi-channel sound card takes it: frame f of channel s is
        element [f, s], bitwise ``pull(n).T`` converted to ``dtype``: int16 (the default), int32 (``s << 16``) or
        float32 (``s / 32768``, exact).  Default: a host (n, S) array of that dtype in the grow-only pinned buffer,
        valid until the next pull; its ``tobytes()`` is what pyaudio's ``Stream.write`` takes for ``channels=S``.
        ``out``: a CUDA tensor of that dtype on this transmitter's device, contiguous with at least n * S elements
        (written frame-major; nothing past n * S is written), or an (n, S) window of a wider buffer with strides
        (row_pitch, 1); or a host numpy array with such a window layout (strides in bytes), such as
        ``playback[:, c0:c0 + S]``.  Only the window is written, and ``out`` is returned."""
        n = int(n)
        if n < 0:
            raise ValueError("pull needs n >= 0")
        S = self.S
        dt, fmt = _frame_format(dtype)
        fn = _cabi.lib().afsk_tx_streams_pull_frames
        if out is None:
            nbytes = S * n * dt.itemsize
            buf = self._pinned_buffer((nbytes + 1) // 2).view(np.uint8)[:nbytes].view(dt)
            _cabi.check(fn(self._h, n, C.c_void_p(buf.ctypes.data), fmt, 0, S, C.c_void_p(stream or 0)))
            return buf.reshape(n, S)
        if isinstance(out, np.ndarray):
            if out.dtype != dt or out.ndim != 2 or out.shape != (n, S) or any(x % dt.itemsize for x in out.strides) \
                    or not out.flags.writeable:
                raise ValueError(f"host out must be a writable ({n}, {S}) {dt.name} array, got {out.dtype} {out.shape}")
            pitch = _row_pitch(n, S, out.strides[0] // dt.itemsize, out.strides[1] // dt.itemsize, "host out")
            _cabi.check(fn(self._h, n, C.c_void_p(out.ctypes.data), fmt, 0, pitch, C.c_void_p(stream or 0)))
            return out
        if not out.is_cuda or out.device.index != self.device:
            raise ValueError(f"out must live on cuda:{self.device}")
        if str(out.dtype) != f"torch.{dt.name}":
            raise ValueError(f"out must be a {dt.name} tensor (dtype=), got {out.dtype}")
        if out.dim() == 2 and tuple(out.shape) == (n, S):
            pitch = _row_pitch(n, S, out.stride(0), out.stride(1), "out")
        elif out.is_contiguous():
            if out.numel() < S * n:
                raise ValueError(f"out holds {out.numel()} frames, the pull needs {S * n}")
            pitch = S
        else:
            raise ValueError(f"out must be contiguous or an ({n}, {S}) window with strides (row_pitch, 1)")
        _cabi.check(fn(self._h, n, C.c_void_p(out.data_ptr()), fmt, 1, pitch, C.c_void_p(stream or 0)))
        return out

    def _pinned_buffer(self, total: int) -> np.ndarray:
        """the grow-only pinned int16 buffer host output is copied into, >= total samples"""
        if self._pinned is None or self._pinned.array.size < total:
            if self._pinned is not None:
                self._pinned.close()
            self._pinned = _cabi.PinnedArray((max(total + total // 4, 16),), np.int16)
        return self._pinned.array

    def _pull(self, fn, n, out, stream):
        """the next n frames of every channel through fn (the planar pull): into ``out``, or into the pinned buffer,
        returned flat"""
        n = int(n)
        if n < 0:
            raise ValueError("pull needs n >= 0")
        total = self.S * n
        if out is not None:
            if not out.is_cuda or out.device.index != self.device:
                raise ValueError(f"out must live on cuda:{self.device}")
            if str(out.dtype) != "torch.int16" or not out.is_contiguous():
                raise ValueError("out must be a contiguous int16 tensor")
            if out.numel() < total:
                raise ValueError(f"out holds {out.numel()} frames, the pull needs {total}")
            _cabi.check(fn(self._h, n, C.c_void_p(out.data_ptr()), 1, C.c_void_p(stream or 0)))
            return out
        buf = self._pinned_buffer(total)[:total]
        _cabi.check(fn(self._h, n, C.c_void_p(buf.ctypes.data), 0, C.c_void_p(stream or 0)))
        return buf

    def state(self, s: int) -> tuple[int, int, int]:
        """(frames pulled, end of channel s's last message (<= frames pulled: idle), its messages not yet fully pulled)."""
        a, b, c = C.c_int64(0), C.c_int64(0), C.c_int64(0)
        _cabi.check(_cabi.lib().afsk_tx_streams_state(self._h, int(s), C.byref(a), C.byref(b), C.byref(c)))
        return a.value, b.value, c.value

    def counters(self) -> dict:
        """Since this transmitter was opened: kernel launches, payload-arena bytes moved by compactions, compactions."""
        a, b, c = C.c_int64(0), C.c_int64(0), C.c_int64(0)
        _cabi.check(_cabi.lib().afsk_tx_streams_counters(self._h, C.byref(a), C.byref(b), C.byref(c)))
        return {"launches": a.value, "moved_bytes": b.value, "compactions": c.value}

    def arena_bytes(self) -> int:
        """Device bytes this transmitter holds (payload arenas, descriptors, host-output staging)."""
        n = C.c_int64(0)
        _cabi.check(_cabi.lib().afsk_tx_streams_arena_bytes(self._h, C.byref(n)))
        return n.value
