"""CPU: host logic added in round 2 — cost-balanced sharding, the host gather of per-rank batches on a
world-size-2 gloo group, the file halves of SoundInput / SoundOutput, the bench corpus recipe and its output dump."""
import os
import socket
import sys

import numpy as np
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)

import afskmodem_b200 as A  # noqa: E402
from afskmodem_b200 import _cabi, shard  # noqa: E402
from oracle import oracle as O  # noqa: E402


def test_shard_by_predicted_cost_balances_mixed_bauds():
    rng = np.random.default_rng(1)
    B = 5000
    baud = rng.choice([300, 1200, 6000, 240, 4800, 9600], B)
    lens = rng.integers(5000, 900000, B)
    cost = shard.capture_cost(lens, baud)
    # a corpus sorted by baud is the bad case for sample-balanced ranges: 240 baud streams at half the rate
    order = np.argsort(baud, kind="stable")
    lens, baud, cost = lens[order], baud[order], cost[order]
    for w in (2, 3, 8):
        by_cost = shard.shard_captures(lens, w, cost)
        by_samples = shard.shard_captures(lens, w)
        for r in (by_cost, by_samples):
            assert r[0][0] == 0 and r[-1][1] == B and all(a[1] == b[0] for a, b in zip(r, r[1:]))
        assert shard.imbalance(cost, by_cost) < 1.01
        assert shard.imbalance(cost, by_cost) <= shard.imbalance(cost, by_samples)
    assert shard.imbalance(cost, shard.shard_captures(lens, 8)) > 1.05
    # captures the reference rejects cost only the fixed part; host-buffer decodes are PCIe-bound
    assert shard.capture_cost([10 ** 6], [9600])[0] == shard.PER_CAPTURE_NS
    assert shard.capture_cost([10 ** 6], [1200], resident=False)[0] > 5 * shard.capture_cost([10 ** 6], [1200])[0]
    with pytest.raises(ValueError):
        shard.shard_captures([1, 2, 3], 2, [1.0])


def test_merge_rx_parts_layout():
    def part(nbytes_list, cap):
        res = np.zeros(len(nbytes_list), dtype=_cabi.RX_RESULT_DTYPE)
        res["nbytes"] = nbytes_list
        off = np.arange(len(nbytes_list) + 1, dtype=np.int64) * cap
        blob = np.zeros(int(off[-1]) + 7, np.uint8)              # capacity may exceed what out_off covers
        for i, n in enumerate(nbytes_list):
            blob[off[i]:off[i] + n] = i + 1 + 10 * len(nbytes_list)
        return res, blob, off
    parts = [part([3, 0], 16), part([], 16), part([5], 32)]
    b = A.RxBatch(*shard.merge_rx_parts(parts))
    assert len(b) == 3 and list(b.out_off) == [0, 16, 32, 64]
    assert b.payload(0) == bytes([21] * 3) and b.payload(1) == b"" and b.payload(2) == bytes([11] * 5)


def _fake_rank_batch(rank):
    """what rank `rank` would have decoded: built from the oracle (this is a test of the gather)"""
    rng = np.random.default_rng([5, rank])
    n = 3 + 2 * rank
    res = np.zeros(n, dtype=_cabi.RX_RESULT_DTYPE)
    off = np.zeros(n + 1, np.int64)
    blobs = []
    for i in range(n):
        pl = rng.integers(0, 256, int(rng.integers(0, 40)), dtype=np.uint8).tobytes()
        o = O.rx_decode(O.tx_frames(pl, 1200, 0.05), 1200, 14000)
        res[i] = (o["status"], o["clock"], o["train_end"], o["nbits"], o["nbytes"])
        cap = (len(o["data"]) + 16 + 15) // 16 * 16
        blobs.append(np.frombuffer(o["data"].ljust(cap, b"\0"), np.uint8))
        off[i + 1] = off[i] + cap
    return A.RxBatch(res, np.concatenate(blobs), off)


def _gather_worker(rank, world, port, out_path):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    merged = shard.gather_rx(_fake_rank_batch(rank), dst=0)
    if rank == 0:
        np.save(out_path, merged.results)
        with open(out_path + ".bin", "wb") as f:
            f.write(b"|".join(p.hex().encode() for p in merged.payloads()))
    else:
        assert merged is None
    dist.barrier()
    dist.destroy_process_group()


def test_gather_rx_two_ranks_gloo(tmp_path):
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    out = str(tmp_path / "res.npy")
    mp.spawn(_gather_worker, args=(2, port, out), nprocs=2, join=True)
    want = [_fake_rank_batch(0), _fake_rank_batch(1)]
    res = np.load(out)
    assert np.array_equal(res, np.concatenate([w.results for w in want]))
    got = open(out + ".bin", "rb").read().split(b"|")
    assert got == [p.hex().encode() for w in want for p in w.payloads()]
    # without a process group the batch comes back unchanged
    assert shard.gather_rx(want[0]) is want[0]


def test_sound_io_file_halves(tmp_path):
    """SoundOutput.writeToFile (afskmodem.py:239-244, 256-263) duplicates even frames and drops an odd last
    one; SoundInput.loadFromFile (:213-217) returns a list of ints.  Against the reference when mounted."""
    from afskmodem import SoundInput, SoundOutput      # the drop-in module name
    rng = np.random.default_rng(3)
    for n in (0, 1, 2, 7, 1000, 1001):
        frames = rng.integers(-32768, 32768, n).tolist()
        fn = str(tmp_path / f"f{n}.wav")
        SoundOutput.writeToFile(fn, frames)
        got = SoundInput.loadFromFile(fn)
        assert isinstance(got, list)
        assert got == [frames[i & ~1] for i in range(len(frames) & ~1)] if n > 1 else got == []
        from oracle import ref_harness
        if ref_harness.available():
            m = ref_harness.module()
            fr = str(tmp_path / f"r{n}.wav")
            m.SoundOutput.writeToFile(fr, frames)
            assert open(fr, "rb").read() == open(fn, "rb").read()
            assert m.SoundInput.loadFromFile(fr) == got
    with pytest.raises(OverflowError):
        SoundOutput.writeToFile(str(tmp_path / "big.wav"), [40000, 0])
    with pytest.raises(RuntimeError):
        SoundInput()


def test_bench_corpus_is_seeded_by_capture_index():
    import bench
    c = bench.Corpus("c5", 3000)
    d = bench.Corpus("c5", 3000)
    assert c.payloads(700, 900) == d.payloads(0, 3000)[700:900]
    lens = c.lens()
    pay = c.payloads(0, 40)
    for i in range(40):
        fr = O.tx_frames(pay[i], int(c.baud_tx[i]), float(c.tt[i]))
        assert lens[i] == c.lead[i] + len(fr), i
    odd = np.nonzero(c.baud_tx == 4800)[0][:5]
    for i in odd:
        fr = O.tx_frames(c.payloads(int(i), int(i) + 1)[0], 4800, float(c.tt[i]))
        assert lens[i] == c.lead[i] + len(fr)
    w = bench.Corpus("c2", 8 * 64)
    assert w.payloads(64, 128) == bench.Corpus("c2", 8 * 64).payloads(0, 512)[64:128]


def _fake_batch(B, seed):
    rng = np.random.default_rng(seed)
    res = np.zeros(B, _cabi.RX_RESULT_DTYPE)
    res["status"] = rng.choice([0, 1, 2, -3], B)
    res["clock"] = rng.integers(-1, 40, B)
    res["train_end"] = rng.integers(2**40, 2**52, B)
    res["nbits"] = rng.integers(0, 9000, B)
    res["nbytes"] = np.where(res["status"] < 0, 0, rng.integers(0, 1100, B))
    out_off = np.zeros(B + 1, np.int64)
    np.cumsum(res["nbytes"] + rng.integers(0, 50, B), out=out_off[1:])
    return A.RxBatch(res, rng.integers(0, 256, int(out_off[-1]), dtype=np.uint8), out_off)


def test_bench_dump_outputs(tmp_path, monkeypatch):
    """--dump-outputs writes every capture's stage integers and payload exactly in float32 / float64; over the
    size budget, the same seeded sample of captures on every run, within the budget."""
    import bench
    b = _fake_batch(300, 5)
    bench.dump_outputs(b, str(tmp_path / "all"))
    got = {f[:-4]: np.load(tmp_path / "all" / f) for f in os.listdir(tmp_path / "all")}
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    assert np.array_equal(got["capture_index"], np.arange(300))
    for f in b.results.dtype.names:
        assert np.array_equal(got[f], b.results[f].astype(np.float64)), f
    off, pay = got["payload_offsets"].astype(np.int64), got["payload_bytes"]
    assert [pay[off[c]:off[c + 1]].astype(np.uint8).tobytes() for c in range(300)] == b.payloads()
    monkeypatch.setattr(bench, "DUMP_BYTES", (1 << 16) + 200_000)
    for run in ("a", "b"):
        bench.dump_outputs(b, str(tmp_path / run))
    total = sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a"))
    assert total <= bench.DUMP_BYTES
    idx = np.load(tmp_path / "a" / "capture_index.npy").astype(np.int64)
    assert 0 < len(idx) < 300 and np.all(np.diff(idx) > 0)
    assert np.array_equal(np.load(tmp_path / "a" / "nbits.npy"), b.nbits[idx].astype(np.float64))
    for f in os.listdir(tmp_path / "a"):
        assert np.array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)), f
    # the sample follows the inputs (the capacity layout), not what was decoded
    other = _fake_batch(300, 6).results
    other["nbytes"] = np.minimum(other["nbytes"], np.diff(b.out_off))
    bench.dump_outputs(A.RxBatch(other, b.blob, b.out_off), str(tmp_path / "c"))
    assert np.array_equal(np.load(tmp_path / "c" / "capture_index.npy"), idx.astype(np.float64))


def test_h2d_gate_serialises_a_group_only(tmp_path, monkeypatch):
    """GPUs that share a host link take turns copying (h2d_gate.py): members of one group never hold the gate
    together, members of different groups do; the policy follows AFSK_H2D_GATE and the number of visible GPUs."""
    import threading
    import time

    from afskmodem_b200 import h2d_gate
    inside, peak, lock = [0], [0], threading.Lock()

    def work(dev):
        g = h2d_gate.H2DGate(dev, 2, 1, root=str(tmp_path))
        for _ in range(30):
            with g:
                with lock:
                    inside[0] += 1
                    peak[0] = max(peak[0], inside[0])
                time.sleep(0.0005)
                with lock:
                    inside[0] -= 1
        g.close()

    for devs, want in (((0, 1), 1), ((0, 2), 2)):
        peak[0] = 0
        ts = [threading.Thread(target=work, args=(d,)) for d in devs]
        [t.start() for t in ts]
        [t.join() for t in ts]
        assert peak[0] <= want and (want == 1 or peak[0] >= 1)
    monkeypatch.delenv("AFSK_H2D_GATE", raising=False)
    assert h2d_gate.default_policy(1) is None and h2d_gate.default_policy(4) is None
    assert h2d_gate.default_policy(8) == (4, 2)
    monkeypatch.setenv("AFSK_H2D_GATE", "off")
    assert h2d_gate.default_policy(8) is None
    monkeypatch.setenv("AFSK_H2D_GATE", "4:2")
    assert h2d_gate.default_policy(2) == (4, 2)
