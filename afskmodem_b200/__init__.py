"""afskmodem_b200 — B200-native batch AFSK modem core with the API of lavajuno/afskmodem.

    from afskmodem_b200 import Receiver, Transmitter
    Transmitter(1200).save("Hello World!", "afsk.wav")
    assert Receiver(1200).load("afsk.wav", True) == "Hello World!"

All signal processing runs in hand-written CUDA kernels for sm_100a (libafsk_b200.so, built by
``python -m afskmodem_b200.build``); there is no CPU fallback.
"""
# Log level (0: Debug, 1: Info, 2: Warn, 3: Error, 4: Fatal) — afskmodem.py:14
LOG_LEVEL = 0

from ._cabi import AfskError, LIB_PATH  # noqa: E402
from .modem import (ECC, Log, PipelinedRxSession, Receiver, RxBatch, RxSession, ShardedRxSession, SoundInput,  # noqa: E402
                    SoundOutput, StreamEvents, StreamReceiver, StreamTransmitter, Transmitter, TxBatch, TxSession, Waveforms, WavBatch,
                    open_receive_streams, open_transmit_streams, read_wav_frames, write_wav_batch, write_wav_frames)
from .shard import capture_cost, gather_rx, shard_captures  # noqa: E402

__all__ = ["LOG_LEVEL", "Log", "Waveforms", "ECC", "Receiver", "Transmitter", "RxBatch", "RxSession", "PipelinedRxSession", "ShardedRxSession", "StreamReceiver", "StreamEvents", "StreamTransmitter",
           "open_receive_streams", "open_transmit_streams", "SoundInput", "SoundOutput",
           "TxBatch", "TxSession", "AfskError", "LIB_PATH", "read_wav_frames", "write_wav_frames", "WavBatch", "write_wav_batch",
           "shard_captures", "capture_cost", "gather_rx"]
