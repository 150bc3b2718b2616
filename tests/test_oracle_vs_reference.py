"""CPU: the oracle against the UNMODIFIED reference on 48 seeded random trials (4 seeds x 12: random baud,
payload, training time, lead silence, gain, AWGN, truncation and thresholds).  The reference's frames and
results of every trial are stored in tests/golden/random_trials.json (with the SHA-256 of each capture, so a
changed recipe or RNG stream fails instead of comparing other inputs).  Where the reference is mounted
(oracle/ref_harness.py) the trials also run on it live and the stored results are checked against it."""
import hashlib
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN
from oracle import oracle as O
from oracle import ref_harness as R

BAUDS = [300, 600, 800, 1200, 2400, 4000, 6000, 12000, 4800, 960, 100]
SEEDS = range(4)
RECIPE = ("baud", "payload_hex", "training_time", "lead", "gain", "sigma", "cut", "amp_start", "amp_end")


def _sha(a) -> str:
    return hashlib.sha256(np.ascontiguousarray(a, dtype="<i2").tobytes()).hexdigest()


def trials(seed, tx_frames):
    """The 12 trials of one seed: the recipe, the frames ``tx_frames(payload, baud, training_time)`` and the
    capture made from them."""
    rng = np.random.default_rng(1000 + seed)
    for _ in range(12):
        baud = int(rng.choice(BAUDS))
        pl = rng.integers(0, 256, size=int(rng.integers(0, 16)), dtype=np.uint8).tobytes()
        tt = float(rng.choice([0.2, 0.1, 0.02]))
        fr = tx_frames(pl, baud, tt)
        lead = int(rng.integers(0, 5000)) if rng.random() < 0.5 else 0
        gain = float(rng.choice([1.0, 0.7, 0.45, 0.3]))
        sigma = float(rng.choice([0, 2000, 8000, 14000, 19000, 26000]))
        x = np.concatenate([np.zeros(lead, np.int16), fr]).astype(np.float64) * gain
        if sigma > 0:
            x = x + np.round(rng.normal(0, sigma, size=len(x)))
        x = np.clip(x, -32768, 32767).astype(np.int16)
        cut = int(rng.integers(1000, len(x))) if rng.random() < 0.2 else None
        if cut is not None:
            x = x[:cut]
        a0, a1 = [(18000, 14000), (14000, 11000), (9000, 8000)][int(rng.integers(0, 3))]
        yield {"baud": baud, "payload_hex": pl.hex(), "training_time": tt, "lead": lead, "gain": gain, "sigma": sigma,
               "cut": cut, "amp_start": a0, "amp_end": a1, "frames": fr, "x": x}


def reference_result(r) -> dict:
    """``ref_harness.ref_load``'s outcome as random_trials.json stores it: the exception, or the payload and
    the four stage integers (a stage the log does not report is -1 / 0, as the oracle reports it)."""
    if r["exc"]:
        return {"exc": list(r["exc"])}
    return {"exc": None, "data_hex": r["ret"].hex(), "clock": -1 if r["clock"] is None else r["clock"],
            "train_end": -1 if r["train_end"] is None else r["train_end"], "nbits": r["nbits"] or 0,
            "nbytes": r["nbytes"] or 0}


def record(tx_frames, result) -> list:
    """What random_trials.json stores for every trial; ``result(trial)`` gives the reference's result."""
    return [{"seed": s, "recipe": {k: t[k] for k in RECIPE}, "frames_sha256": _sha(t["frames"]), "n": int(len(t["x"])),
             "input_sha256": _sha(t["x"]), "result": result(t)} for s in SEEDS for t in trials(s, tx_frames)]


@pytest.fixture(scope="module")
def recorded():
    return json.load(open(os.path.join(GOLDEN, "random_trials.json")))["trials"]


@pytest.mark.parametrize("seed", SEEDS)
def test_random_trials(seed, recorded):
    want_all = [g for g in recorded if g["seed"] == seed]
    assert len(want_all) == 12
    for t, g in zip(trials(seed, O.tx_frames), want_all):
        assert {k: t[k] for k in RECIPE} == g["recipe"]
        assert _sha(t["frames"]) == g["frames_sha256"]                 # the oracle's frames == the reference's
        assert len(t["x"]) == g["n"] and _sha(t["x"]) == g["input_sha256"]
        want = g["result"]
        if R.available():
            assert np.array_equal(R.ref_save(bytes.fromhex(t["payload_hex"]), t["baud"], t["training_time"]), t["frames"])
            assert reference_result(R.ref_load(t["x"], t["baud"], t["amp_start"], t["amp_end"])) == want
        o = O.rx_decode(t["x"], t["baud"], t["amp_end"])
        if want["exc"]:
            assert o["status"] < 0 and list(O.EXC_TEXT[o["status"]]) == want["exc"]
            continue
        assert o["data"].hex() == want["data_hex"]
        assert (o["clock"], o["train_end"]) == (want["clock"], want["train_end"])
        assert (o["nbits"], o["nbytes"]) == (want["nbits"], want["nbytes"])
