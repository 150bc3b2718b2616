"""CPU: host-side logic of the package and the C-ABI surface (no compute calls without a GPU)."""
import ast
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import afskmodem_b200 as A
from afskmodem_b200 import _cabi
from afskmodem_b200.shard import shard_captures
from conftest import ROOT


def test_library_exports_every_declared_symbol():
    """include/afsk_b200.h <-> libafsk_b200.so <-> the ctypes binding agree on the symbol list."""
    hdr = open(os.path.join(ROOT, "include", "afsk_b200.h")).read()
    declared = set(re.findall(r"\b(afsk_[a-z0-9_]+)\s*\(", hdr))
    assert declared == set(_cabi.SYMBOLS)
    L = _cabi.lib()
    for s in declared:
        assert hasattr(L, s), s
    assert L.afsk_abi_version() == 2


def test_tone_lengths_match_reference_rules():
    # SURVEY F1/F2: ctor ok iff 24000 % baud == 0; decodable iff mark_len == space_len
    assert _cabi.tone_lengths(1200) == (40, 40, 40)
    assert _cabi.tone_lengths(4800) == (10, 8, 10)
    assert _cabi.tone_lengths(300) == (160, 160, 160)
    assert _cabi.tone_lengths(6000) == (8, 8, 8)
    for bad in (9600, 3200, 1100, 7, 48000, 0, -5):
        assert _cabi.tone_lengths(bad) is None
    for baud in range(1, 24001):
        got = _cabi.tone_lengths(baud)
        assert (got is not None) == (24000 % baud == 0)
        if got:
            assert got[0] == 48000 // baud and (got[1] == got[2]) == (12000 % baud == 0)


def test_constructor_exceptions_match_reference():
    for bad in (9600, 3200, 1100, 7, 48000):
        with pytest.raises(Exception, match="Invalid baud rate."):
            A.Receiver(bad)
        with pytest.raises(Exception, match="Invalid baud rate."):
            A.Transmitter(bad)
    with pytest.raises(ZeroDivisionError):
        A.Receiver(0)
    A.Receiver(4800), A.Transmitter(4800, training_sequence_time=1.5)     # constructs (F2)
    assert A.Transmitter(1200, 0.5)._ts_cycles == 300 and A.Transmitter(1200, 1.5)._ts_cycles == 900
    assert A.Receiver.read is A.Receiver.load and A.Transmitter.write is A.Transmitter.save


def test_waveforms_and_ecc_utilities():
    assert A.Waveforms.getSpaceTone(1200) == [32767] * 20 + [-32768] * 20
    assert A.Waveforms.getMarkTone(1200) == ([32767] * 10 + [-32768] * 10) * 2
    assert len(A.Waveforms.getMarkTone(4800)) == 8
    assert A.Waveforms.getAmplitude([-32768, 32767, 0, 1]) == 16384
    assert A.Waveforms.getDiff([1, 2, 3], [3, 2, 1]) == 1
    with pytest.raises(Exception, match="different lengths"):
        A.Waveforms.getDiff([1], [1, 2])
    bits = "1011000111110000"
    enc = A.ECC.encode(bits)
    assert len(enc) == 28 and A.ECC.decode(enc) == bits
    flipped = enc[:3] + ("1" if enc[3] == "0" else "0") + enc[4:]
    assert A.ECC.decode(flipped) == bits


def test_log_format(capsys):
    A.LOG_LEVEL = 0
    A.Log("afskmodem.Receiver").debug("Recovered clock. (frame 0)")
    A.Log("afskmodem.Receiver").warn("No data.")
    A.LOG_LEVEL = 3
    A.Log("x").warn("hidden")
    A.LOG_LEVEL = 0
    out = capsys.readouterr().out.splitlines()
    assert re.fullmatch(r"\d{4}-\d\d-\d\d \d\d:\d\d:\d\d \[ DEBUG \] afskmodem\.Receiver      : Recovered clock\. \(frame 0\)", out[0])
    assert out[1].endswith(" [ WARN ]  afskmodem.Receiver      : No data.") and len(out) == 2


def test_shard_captures_balanced_contiguous():
    rng = np.random.default_rng(0)
    for B, W in ((1, 2), (7, 2), (100, 8), (4096, 8), (3, 8)):
        lens = rng.integers(4000, 700000, B)
        r = shard_captures(lens, W)
        assert len(r) == W and r[0][0] == 0 and r[-1][1] == B
        assert all(r[i][1] == r[i + 1][0] for i in range(W - 1))
        if B >= 16 * W:
            loads = [lens[a:b].sum() for a, b in r]
            assert max(loads) <= 1.15 * lens.sum() / W


def test_no_device_means_loud_failure():
    """With no visible CUDA device every compute call raises AfskError.  A fresh process with
    CUDA_VISIBLE_DEVICES empty sees no device on a GPU machine too."""
    code = ("import sys; sys.path.insert(0, sys.argv[1])\n"
            "import numpy as np, pytest, afskmodem_b200 as A\n"
            "with pytest.raises(A.AfskError):\n"
            "    A.Receiver(1200).decode_batch([np.zeros(5000, np.int16)])\n"
            "with pytest.raises(A.AfskError):\n"
            "    A.Transmitter(1200).encode_batch([b'x'])\n")
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    proc = subprocess.run([sys.executable, "-c", code, ROOT], env=env, capture_output=True, text=True, timeout=300)
    assert proc.returncode == 0, proc.stderr


def test_product_never_imports_the_oracle():
    """The oracle is test infrastructure: nothing under afskmodem_b200/ may import or open it."""
    pkg = os.path.join(ROOT, "afskmodem_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            path = os.path.join(dirpath, f)
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(path).read()
                assert "oracle" not in src.lower(), path
            if f.endswith(".py"):
                for node in ast.walk(ast.parse(open(path).read())):
                    if isinstance(node, (ast.Import, ast.ImportFrom)):
                        names = [a.name for a in node.names] + [getattr(node, "module", "") or ""]
                        assert not any("oracle" in n for n in names), path


def test_pipelined_layout_merges_ranges_like_one_plan():
    """PipelinedRxSession keeps one result set for the whole batch: the per-range payload offsets are
    shifted into one blob, results are indexed range after range (pure bookkeeping, no device)."""
    from afskmodem_b200.modem import PipelinedRxSession
    from afskmodem_b200.shard import shard_captures
    rng = np.random.default_rng(5)
    lengths = rng.integers(0, 50_000, 41)
    caps = (lengths // 40 // 14 + 16 + 15) & ~15                 # per-capture capacities as a plan would lay them out
    ranges = [(lo, hi) for lo, hi in shard_captures(lengths, 8) if hi > lo]
    assert ranges[0][0] == 0 and ranges[-1][1] == len(lengths)
    subs = [np.concatenate([[0], np.cumsum(caps[lo:hi])]) for lo, hi in ranges]
    res_lo, blob_lo, out_off = PipelinedRxSession.merged_layout(subs)
    assert list(res_lo) == [lo for lo, _ in ranges] + [len(lengths)]
    assert np.array_equal(out_off, np.concatenate([[0], np.cumsum(caps)]))
    assert list(blob_lo) == [int(out_off[lo]) for lo, _ in ranges] + [int(out_off[-1])]
