"""Generates tests/golden/{rx_cases.npz,rx_cases.json,tx_cases.npz,tx_cases.json,gate_cases.json,gate_multi_cases.json,
random_trials.json}
by running the UNMODIFIED reference (/root/reference/afskmodem.py) in this container through
oracle/ref_harness.py.  The reference ships no golden vectors of its own (SURVEY.md §4), so these
files ARE the pin: the oracle (oracle/afsk_oracle.c) is checked against them on CPU, and the CUDA
path against both on the GPU box, where /root/reference does not exist.

    python tests/golden/make_golden.py          # rewrites the fixtures (needs /root/reference)

Inputs are built from the reference's own Transmitter.save output, then lead silence / gain /
AWGN / truncation applied with numpy (seeded); the exact int16 samples are stored, so the
fixtures do not depend on numpy's RNG stream staying stable.
"""
from __future__ import annotations

import hashlib
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.abspath(os.path.join(HERE, "..", "..")))
from oracle import ref_harness as R  # noqa: E402


def impair(fr, rng, lead=0, gain=1.0, sigma=0.0, cut=None, tail_cut=0):
    x = np.concatenate([np.zeros(lead, np.int16), fr]).astype(np.float64) * gain
    if sigma > 0:
        x = x + np.round(rng.normal(0.0, sigma, size=len(x)))
    x = np.clip(np.trunc(x), -32768, 32767).astype(np.int16)
    if tail_cut:
        x = x[:len(x) - tail_cut]
    if cut is not None:
        x = x[:cut]
    return x


def rx_case_list():
    """(name, baud, amp_start, amp_end, samples)"""
    rng = np.random.default_rng(20261017)
    cases = []
    hello = R.ref_save("Hello World!", 1200)
    cases.append(("readme_hello_1200", 1200, 18000, 14000, hello))
    cases.append(("readme_utf8_1200", 1200, 18000, 14000, R.ref_save("Héellóo World!", 1200)))
    # SURVEY Appendix A edge cases
    for lead in (1, 39, 40, 41, 4015, 4016, 4017, 4096):
        cases.append((f"lead_{lead}", 1200, 18000, 14000, impair(hello, rng, lead=lead)))
    cases.append(("len_4095", 1200, 18000, 14000, hello[:4095].copy()))
    cases.append(("len_4096", 1200, 18000, 14000, hello[:4096].copy()))
    cases.append(("len_0", 1200, 18000, 14000, np.zeros(0, np.int16)))
    cases.append(("tail_removed", 1200, 18000, 14000, hello[:len(hello) - 4800].copy()))
    cases.append(("tail_removed_plus1", 1200, 18000, 14000, hello[:len(hello) - 4799].copy()))
    cases.append(("gain_043", 1200, 18000, 14000, impair(hello, rng, gain=0.43)))
    cases.append(("gain_042", 1200, 18000, 14000, impair(hello, rng, gain=0.42)))
    cases.append(("gain_03_thr8000", 1200, 9000, 8000, impair(hello, rng, gain=0.3)))
    cases.append(("zeros_50000", 1200, 18000, 14000, np.zeros(50000, np.int16)))
    cases.append(("uniform_noise", 1200, 18000, 14000,
                  rng.integers(-32768, 32768, size=20000).astype(np.int16)))
    cases.append(("full_scale_neg", 1200, 18000, 14000, np.full(9000, -32768, np.int16)))
    cases.append(("near_threshold", 1200, 18000, 400,
                  rng.integers(-516, 517, size=12000).astype(np.int16)))
    short = R.ref_save(b"\x00\xffAFSK\x80\x7f", 1200, 0.1)
    for sigma in (2000, 8000, 15000, 20000, 26000, 30000):
        cases.append((f"awgn_{sigma}", 1200, 18000, 14000, impair(short, rng, sigma=sigma)))
    cases.append(("awgn_30000_hello", 1200, 18000, 14000, impair(hello, rng, sigma=30000)))
    # every baud class: valid (12000 % baud == 0), unequal tones (F2), ctor failure (F1), IndexError
    for baud in (300, 600, 800, 1200, 2400, 4000, 6000, 12000, 100, 375):
        fr = R.ref_save(b"Hi!", baud, 0.05 if baud >= 600 else 0.2)
        cases.append((f"baud_{baud}_clean", baud, 18000, 14000, fr))
        cases.append((f"baud_{baud}_noisy", baud, 18000, 14000,
                      impair(fr, rng, lead=int(rng.integers(0, 300)), sigma=6000)))
    for baud in (4800, 960, 1600, 8000):
        fr = R.ref_save(b"Hi!", baud, 0.1)
        cases.append((f"baud_{baud}_unequal", baud, 18000, 14000, fr))
        cases.append((f"baud_{baud}_unequal_short", baud, 18000, 14000, fr[:3000].copy()))
    cases.append(("baud_9600_ctor", 9600, 18000, 14000, hello[:5000].copy()))
    cases.append(("baud_1100_ctor", 1100, 18000, 14000, hello[:5000].copy()))
    cases.append(("baud_20_index", 20, 18000, 14000, hello[:6000].copy()))
    cases.append(("baud_24_scan1", 24, 18000, 14000, hello[:9000].copy()))
    # seeded random sweep
    bauds = [300, 600, 800, 1200, 2400, 4000, 6000]
    thr = [(18000, 14000), (14000, 11000), (9000, 8000)]
    for i in range(28):
        baud = int(rng.choice(bauds))
        pl = rng.integers(0, 256, size=int(rng.integers(1, 10)), dtype=np.uint8).tobytes()
        fr = R.ref_save(pl, baud, float(rng.choice([0.1, 0.05, 0.02])) if baud >= 600 else 0.2)
        a = thr[int(rng.integers(0, 3))]
        x = impair(fr, rng, lead=int(rng.integers(0, 4500)) if rng.random() < 0.5 else 0,
                   gain=float(rng.choice([1.0, 0.7, 0.45, 0.3])),
                   sigma=float(rng.choice([0, 2000, 8000, 14000, 19000, 26000])),
                   cut=int(rng.integers(3000, len(fr))) if rng.random() < 0.2 else None)
        cases.append((f"sweep_{i:02d}_b{baud}", baud, a[0], a[1], x))
    return cases


def tx_case_list():
    rng = np.random.default_rng(7)
    cases = [("readme_hello", "Hello World!".encode(), 1200, 0.5),
             ("readme_utf8", "Héellóo World!".encode(), 1200, 0.5),
             ("empty", b"", 1200, 0.5),
             ("tt_1p5", b"x", 1200, 1.5),
             ("tt_0", b"abc", 1200, 0.0)]
    for baud in (300, 600, 800, 1200, 2400, 4000, 6000, 12000, 100, 375, 4800, 960, 1600, 8000, 24000,
                 9600, 3200, 1100, 7):
        pl = rng.integers(0, 256, size=int(rng.integers(1, 24)), dtype=np.uint8).tobytes()
        cases.append((f"baud_{baud}", pl, baud, float(rng.choice([0.5, 0.1, 0.02, 0.013]))))
    cases.append(("kb_1200", rng.integers(0, 256, size=1024, dtype=np.uint8).tobytes(), 1200, 0.5))
    cases.append(("kb_2400", rng.integers(0, 256, size=300, dtype=np.uint8).tobytes(), 2400, 0.5))
    return cases


def main():
    assert R.available(), "reference not mounted"
    arrays, meta = {}, []
    for name, baud, a0, a1, x in rx_case_list():
        r = R.ref_load(x, baud, a0, a1, string=False)
        rs = R.ref_load(x, baud, a0, a1, string=True)
        ret = r["ret"]
        meta.append({
            "name": name, "baud": baud, "amp_start": a0, "amp_end": a1, "n": int(len(x)),
            "ctor_exc": r["ctor_exc"], "exc": r["exc"],
            "data_hex": ret.hex() if isinstance(ret, (bytes, bytearray)) else None,
            "clock": r.get("clock"), "train_end": r.get("train_end"), "nbits": r.get("nbits"),
            "nbytes": r.get("nbytes"), "no_clock": r.get("no_clock"), "no_data": r.get("no_data"),
            "string_ret_type": type(rs["ret"]).__name__ if rs["ret"] is not None else None,
            "string_ret": rs["ret"] if isinstance(rs["ret"], str) else None,
            "string_exc": rs["exc"][0] if rs["exc"] else None,
        })
        arrays[name] = x
    np.savez_compressed(os.path.join(HERE, "rx_cases.npz"), **arrays)
    json.dump(meta, open(os.path.join(HERE, "rx_cases.json"), "w"), indent=1)

    arrays, meta = {}, []
    for name, pl, baud, tt in tx_case_list():
        try:
            fr = R.ref_save(pl, baud, tt)
            exc = None
        except Exception as e:  # noqa: BLE001
            fr, exc = None, (type(e).__name__, str(e))
        meta.append({"name": name, "payload_hex": pl.hex(), "baud": baud, "training_time": tt, "exc": exc,
                     "n": None if fr is None else int(len(fr)),
                     "sha256": None if fr is None else hashlib.sha256(fr.astype("<i2").tobytes()).hexdigest()})
        if fr is not None and len(fr) <= 120000:
            arrays[name] = fr
    np.savez_compressed(os.path.join(HERE, "tx_cases.npz"), **arrays)
    json.dump(meta, open(os.path.join(HERE, "tx_cases.json"), "w"), indent=1)

    # listen gate (Receiver.receive through the stub stream): recipes are tiny, so store recipes
    hello = R.ref_save("Hello World!", 1200)
    gate = []
    for name, lead, gain, a0, a1, timeout, tailz in [
            ("lead_2048", 2048, 1.0, 18000, 14000, 100.0, 8192),
            ("lead_5000", 5000, 1.0, 18000, 14000, 100.0, 8192),
            ("lead_3x2048", 6144, 1.0, 18000, 14000, 100.0, 8192),
            ("timeout_0p1", 8192, 1.0, 18000, 14000, 0.1, 8192),
            ("timeout_0", 2048, 1.0, 18000, 14000, 0.0, 8192),
            ("quiet_gain", 4096, 0.5, 18000, 14000, 1.0, 8192),
            ("sensitive", 4096, 0.5, 14000, 11000, 1.0, 8192),
            ("timeout_exact", 4096, 1.0, 18000, 14000, 2048 / 48000.0, 8192)]:
        s = np.concatenate([np.zeros(lead, np.int16), (hello.astype(np.float64) * gain).astype(np.int16),
                            np.zeros(tailz, np.int16)])
        r = R.ref_receive(s, 1200, a0, a1, timeout)
        gate.append({"name": name, "lead": lead, "gain": gain, "amp_start": a0, "amp_end": a1,
                     "timeout": timeout, "tail_zeros": tailz, "reads": r["reads"],
                     "timed_out": r["timed_out"], "exc": r["exc"],
                     "ret_hex": r["ret"].hex() if isinstance(r["ret"], (bytes, bytearray)) else None,
                     "clock": r["clock"], "train_end": r["train_end"], "nbits": r["nbits"]})
    json.dump(gate, open(os.path.join(HERE, "gate_cases.json"), "w"), indent=1)

    # several transmissions in one recording: successive receive() calls of ONE reference Receiver
    multi = []
    for name, baud, a0, a1, timeout, segs in [
            # segs: (silence before, message, gain, training_time)
            ("three_msgs", 1200, 18000, 14000, 100.0,
             [(5000, "first message", 1.0, 0.1), (3000, "2nd", 1.0, 0.1), (20000, "the third and last one", 1.0, 0.1), (9000, None, 1.0, 0.1)]),
            ("timeouts_between", 1200, 18000, 14000, 0.1,
             [(5000, "first message", 1.0, 0.1), (3000, "2nd", 1.0, 0.1), (20000, "the third and last one", 1.0, 0.1), (9000, None, 1.0, 0.1)]),
            ("back_to_back", 1200, 18000, 14000, 1.0,
             [(2048, "a", 1.0, 0.05), (0, "b", 1.0, 0.05), (100, "c", 1.0, 0.05), (7000, None, 1.0, 0.05)]),
            ("quiet_and_loud_2400", 2400, 14000, 11000, 0.5,
             [(9000, "loud one", 1.0, 0.1), (30000, "too quiet to open the gate", 0.3, 0.1), (12000, "loud again", 0.6, 0.1), (16000, None, 1.0, 0.1)]),
            ("cut_open_at_end", 1200, 18000, 14000, 1.0,
             [(4096, "complete", 1.0, 0.1), (6000, "this one is cut off by the end of the recording", 1.0, 0.1)]),
            ("timeout_zero", 1200, 18000, 14000, 0.0, [(2048, "never heard", 1.0, 0.1), (8192, None, 1.0, 0.1)]),
    ]:
        parts = []
        for lead, msg, gain, tt in segs:
            parts.append(np.zeros(lead, np.int16))
            if msg is not None:
                parts.append((R.ref_save(msg, baud, tt).astype(np.float64) * gain).astype(np.int16))
        s = np.concatenate(parts)
        if name == "cut_open_at_end":
            s = s[:len(s) - 9000]
        calls = R.ref_receive_many(s, baud, a0, a1, timeout)
        multi.append({"name": name, "baud": baud, "amp_start": a0, "amp_end": a1, "timeout": timeout,
                      "segments": segs, "cut": 9000 if name == "cut_open_at_end" else 0, "n": int(len(s)),
                      "sha256": hashlib.sha256(s.astype("<i2").tobytes()).hexdigest(),
                      "calls": [{"timed_out": c["timed_out"], "exc": c["exc"], "reads_before": c["reads_before"],
                                 "reads_after": c["reads_after"],
                                 "ret_hex": c["ret"].hex() if isinstance(c["ret"], (bytes, bytearray)) else None,
                                 "clock": c["clock"], "train_end": c["train_end"], "nbits": c["nbits"]} for c in calls]})
    json.dump(multi, open(os.path.join(HERE, "gate_multi_cases.json"), "w"), indent=1)

    # the 48 seeded random trials of tests/test_oracle_vs_reference.py: recipes are stored, not samples
    sys.path.insert(0, os.path.dirname(HERE))
    import test_oracle_vs_reference as T
    trials = T.record(R.ref_save, lambda t: T.reference_result(R.ref_load(t["x"], t["baud"], t["amp_start"], t["amp_end"])))
    json.dump({"source": "the unmodified reference, by tests/golden/make_golden.py", "trials": trials},
              open(os.path.join(HERE, "random_trials.json"), "w"), indent=1)
    for f in ("rx_cases.npz", "rx_cases.json", "tx_cases.npz", "tx_cases.json", "gate_cases.json", "gate_multi_cases.json",
              "random_trials.json"):
        print(f, os.path.getsize(os.path.join(HERE, f)))


if __name__ == "__main__":
    main()
