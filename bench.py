#!/usr/bin/env python
"""bench.py — batched AFSK decode throughput on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Line of record (BASELINE.json configs[1], "c2"): 4096 independent 1200-baud captures per GPU, 1 KB random
payload each, synthesized by the GPU transmitter, 25 % with U[0,4000) frames of lead silence, AWGN sigma
drawn per capture from {0,2k,8k,14k,19k,26k} (weights 1,2,3,2,1,1), all over the whole capture
(SURVEY.md §8d).  ~2.47 G samples = 4.9 GB of int16 per GPU: larger than L2, so no flush is needed
between timed iterations.  A step = one decode of the whole batch.  Every corpus is seeded by CAPTURE
INDEX (never by rank): rank r of N decodes captures [r*B, (r+1)*B) of one global corpus.

  value        decoded Msamples/s, inputs resident in HBM, CUDA events, max over ranks (weak scaling)
  e2e          same metric through Receiver.decode_batch with HOST (pinned) buffers: H2D of all samples,
               kernels, D2H of results + payloads inside the timed region
  roofline     dominant kernel: 2 bytes/sample x samples per launch / its CUDA-event duration vs the
               measured HBM copy peak (MEASURED_PEAKS.json)
  cpu_baseline the C oracle port of the reference algorithm on the host cores (rank 0, N=1), and the
               unmodified Python reference as timed in the build container (profiles/r2_python_reference.json)
  workloads    the other BASELINE configs (c3, c4, c5) at the same N: value, roofline, parity
  sharded      strong scaling: ONE mixed-baud corpus (c5, 100,000 captures) cut into N contiguous ranges
               balanced by predicted time, decoded by the N ranks, gathered on the host into one RxBatch;
               SHA-256 of (results, payloads) is the same at every N
  tx           transmitter (k_synth) roofline, e2e through Transmitter.save_batch, k_synth_var at 4800 baud
  latency      BASELINE configs[0]: single-file Transmitter.save / Receiver.load, and the cold first call

--impl reference times the reference's CPU implementation (the C oracle port; the reference is pure
Python with a pyaudio import and cannot travel to the GPU box, see DESIGN.md) on the FULL batch of the
same workload, all host threads.  --impl reference --python (build container only) times the unmodified
afskmodem.py itself.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

AMP_END = 14000
# name -> (baud, payload bytes, captures per GPU, config id, captures per noise chunk)
#   c3: 6000 baud stand-in for the reference-unsupported 9600 (SURVEY F1)
#   c4: 300 baud, 64 KB payloads, 64 captures of 146.8 M samples per GPU
#   c5: mixed-baud corpus (SURVEY §8d): baud in {300,600,1200,2400,4000,6000} + 1 % each of 4800 / 9600
#       (exception parity), payloads log-uniform 16 B - 4 KB, per-capture thresholds / gains / training times
WORKLOADS = {"c2": (1200, 1024, 4096, 2, 64), "c3": (6000, 1024, 16384, 3, 64), "c4": (300, 65536, 64, 4, 1),
             "c5": (0, 0, 12500, 5, 64)}
C5_CORPUS = 100_000
SIGMAS = np.array([0, 2000, 8000, 14000, 19000, 26000], dtype=np.float64)
SIGMA_W = np.array([1, 2, 3, 2, 1, 1], dtype=np.float64) / 10.0


def resolve_workload(name):
    """c2..c5, or w<baud>: a tuning aid — 1 KB payloads at any decodable baud, about 2.4 G samples."""
    if name in WORKLOADS:
        return WORKLOADS[name]
    if name.startswith("w") and name[1:].isdigit():
        baud = int(name[1:])
        per_capture = (baud // 4 * 2 + 4 + 14 * 1024) * (48000 // baud) + 4800
        return (baud, 1024, max(64, int(2.4e9 // per_capture)), 100 + baud, 64)
    raise SystemExit(f"unknown workload {name!r}")


class Corpus:
    """Per-capture recipe of a workload for ALL captures of one global corpus (SURVEY.md §8d), seeded by
    (config id) for the metadata and (config id, capture chunk) for payload bytes and noise, so any rank
    can rebuild any capture range and gets the same samples."""

    def __init__(self, wl: str, total: int):
        self.wl, self.total = wl, int(total)
        self.baud, self.payload_bytes, self.per_gpu, self.cid, self.chunk = resolve_workload(wl)
        B = self.total
        rng = np.random.default_rng([self.cid, 0])
        if wl != "c5":
            self.plen = np.full(B, self.payload_bytes, np.int64)
            self.lead = np.where(rng.random(B) < 0.25, rng.integers(0, 4000, B), 0).astype(np.int64)
            self.sigma = rng.choice(SIGMAS, size=B, p=SIGMA_W)
            self.gain = np.ones(B)
            self.tt = 0.5 * np.ones(B)
            self.baud_tx = np.full(B, self.baud, np.int32)
            self.baud_rx = np.full(B, self.baud, np.int32)
            self.amp_end = np.full(B, AMP_END, np.int32)
        else:
            baud_rx = rng.choice(np.array([300, 600, 1200, 2400, 4000, 6000, 4800, 9600], np.int32), size=B,
                                 p=[0.1633, 0.1633, 0.1634, 0.1633, 0.1633, 0.1634, 0.01, 0.01])
            self.baud_rx = baud_rx.astype(np.int32)
            self.baud_tx = np.where(baud_rx == 9600, 6000, baud_rx).astype(np.int32)   # nothing can synthesize 9600 (SURVEY F1)
            self.plen = np.exp(rng.uniform(np.log(16), np.log(4096), B)).astype(np.int64)
            pair = rng.integers(0, 3, B)
            self.amp_end = np.array([14000, 11000, 8000], np.int32)[pair]
            self.gain = np.where(pair == 0, rng.choice([1.0, 0.7], B),
                                 np.where(pair == 1, rng.choice([1.0, 0.7, 0.45], B), rng.choice([1.0, 0.7, 0.45, 0.3], B)))
            self.lead = np.where(rng.random(B) < 0.25, rng.integers(0, 4000, B), 0).astype(np.int64)
            self.sigma = rng.choice(SIGMAS, size=B, p=SIGMA_W)
            self.tt = rng.choice([0.5, 1.5, 0.1, 0.02], B)
        self.ts = np.array([int(b * t / 2) for b, t in zip(self.baud_tx, self.tt)], dtype=np.int64)   # afskmodem.py:438
        self._lens = None

    def payloads(self, lo: int, hi: int) -> list[bytes]:
        """payload bytes of captures [lo, hi): one generator per chunk of `chunk` captures"""
        out = []
        for k in (range(lo // self.chunk, (hi - 1) // self.chunk + 1) if hi > lo else ()):
            a, b = k * self.chunk, min((k + 1) * self.chunk, self.total)
            rng = np.random.default_rng([self.cid, 1, k])
            raw = rng.integers(0, 256, int(self.plen[a:b].sum()), dtype=np.uint8)
            cut = np.concatenate([[0], np.cumsum(self.plen[a:b])])
            out += [raw[cut[i]:cut[i + 1]].tobytes() for i in range(b - a) if lo <= a + i < hi]
        return out

    def lens(self) -> np.ndarray:
        """frames per capture (lead silence + what Transmitter.save writes, afskmodem.py:452-469, :239-244)"""
        if self._lens is None:
            bf = 48000 // self.baud_tx.astype(np.int64)
            n = (2 * self.ts + 4 + 14 * self.plen) * bf + 4800
            odd = np.nonzero((12000 % self.baud_tx) != 0)[0]          # mark and space tones of different length
            if len(odd):
                import ctypes

                from afskmodem_b200 import _cabi
                L = _cabi.lib()
                for c in odd:
                    p = np.frombuffer(self.payloads(int(c), int(c) + 1)[0], dtype=np.uint8)
                    n[c] = L.afsk_tx_num_samples(int(self.baud_tx[c]), int(self.ts[c]), len(p),
                                                 p.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8)))
            self._lens = self.lead + (n & ~1)
        return self._lens

    def spec(self, lo: int, hi: int) -> dict:
        return {"payloads": self.payloads(lo, hi), "lead": self.lead[lo:hi], "sigma": self.sigma[lo:hi],
                "gain": self.gain[lo:hi], "tt": self.tt[lo:hi], "baud_tx": self.baud_tx[lo:hi],
                "baud_rx": self.baud_rx[lo:hi], "amp_end": self.amp_end[lo:hi]}

    def name(self, B: int) -> str:
        if self.wl == "c5":
            return (f"c5: {B} mixed-baud captures (300-6000 baud + 1% each 4800/9600), payloads 16 B-4 KB log-uniform, "
                    "per-capture thresholds/gains/training times, AWGN mix")
        return f"{self.wl}: {B} x {self.baud}-baud captures, {self.payload_bytes} B payload, AWGN mix, 25% lead silence"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            for line in self.proc.stdout:
                self.rows.append([c.strip() for c in line.split(",")])
        except Exception:  # noqa: BLE001
            pass

    def stop(self):
        if self.proc:
            self.proc.terminate()
        self.join(timeout=2)
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:  # noqa: BLE001
                continue
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def build_on_gpu(corpus: Corpus, lo: int, hi: int, device: int):
    """Captures [lo, hi) of the corpus on the device: synthesized with the GPU transmitter, then lead
    silence, gain and AWGN with torch (plumbing), chunk by chunk of `corpus.chunk` captures (the noise
    generator is seeded per chunk, so the samples do not depend on who builds them).
    Returns (samples on the device, CSR offsets of [lo, hi))."""
    import ctypes

    import torch

    import afskmodem_b200 as A
    dev = torch.device("cuda", device)
    lens = corpus.lens()
    offsets = np.zeros(hi - lo + 1, dtype=np.int64)
    np.cumsum(lens[lo:hi], out=offsets[1:])
    total = int(offsets[-1])
    samples = torch.zeros(total + 64, dtype=torch.int16, device=dev)
    CH = corpus.chunk
    gen = torch.Generator(device=dev)
    for k in (range(lo // CH, (hi - 1) // CH + 1) if hi > lo else ()):
        a, b = k * CH, min((k + 1) * CH, corpus.total)
        pay = corpus.payloads(a, b)
        tx = A.TxSession(pay, corpus.baud_tx[a:b], corpus.ts[a:b], device)
        tx.upload()
        clean = torch.empty(int(tx.out_off[-1]) + 64, dtype=torch.int16, device=dev)
        synth = lambda: A._cabi.check(A._cabi.lib().afsk_tx_synth(tx.plan, ctypes.c_void_p(tx.d_pay.ptr),       # noqa: E731
                                                                  ctypes.c_void_p(clean.data_ptr()), None))
        synth()
        clean_n = tx.out_len.astype(np.int64)
        assert np.array_equal(clean_n + corpus.lead[a:b], lens[a:b]), "corpus.lens() disagrees with the transmitter plan"
        ln = lens[a:b]
        coff = np.zeros(b - a + 1, dtype=np.int64)
        np.cumsum(ln, out=coff[1:])
        x = torch.zeros(int(coff[-1]), dtype=torch.int16, device=dev)
        for c in range(a, b):
            o = int(coff[c - a]) + int(corpus.lead[c])
            x[o:o + int(clean_n[c - a])] = clean[int(tx.out_off[c - a]):int(tx.out_off[c - a]) + int(clean_n[c - a])]
        tx.close()
        del clean
        lnt = torch.as_tensor(ln, device=dev)
        sig = torch.repeat_interleave(torch.as_tensor(corpus.sigma[a:b], dtype=torch.float32, device=dev), lnt)
        gn = torch.repeat_interleave(torch.as_tensor(corpus.gain[a:b], dtype=torch.float32, device=dev), lnt)
        gen.manual_seed(1_000_003 * corpus.cid + k)
        noise = torch.round(torch.randn(int(coff[-1]), generator=gen, device=dev, dtype=torch.float32) * sig)
        x = torch.clamp(torch.trunc(x.to(torch.float32) * gn) + noise, -32768, 32767).to(torch.int16)
        del sig, gn, noise
        ca, cb = max(a, lo), min(b, hi)                     # captures of this chunk that belong to [lo, hi)
        if cb > ca:
            samples[int(offsets[ca - lo]):int(offsets[cb - lo])] = x[int(coff[ca - a]):int(coff[cb - a])]
        del x
    torch.cuda.synchronize(dev)
    return samples, offsets


def host_sample_batch(corpus: Corpus, lo: int, hi: int, threads: int):
    """Same recipe on the host (oracle transmitter + numpy AWGN, one generator per capture) for the
    reference arm: nothing of the GPU path is used."""
    from concurrent.futures import ThreadPoolExecutor

    from oracle import oracle as O
    pay = corpus.payloads(lo, hi)

    def one(c):
        fr = O.tx_frames(pay[c - lo], int(corpus.baud_tx[c]), float(corpus.tt[c]))
        x = np.concatenate([np.zeros(int(corpus.lead[c]), np.int16), fr]).astype(np.float32)
        x = np.trunc(x * np.float32(corpus.gain[c]))
        if corpus.sigma[c] > 0:
            rng = np.random.default_rng([3, corpus.cid, c])
            x += np.round(rng.standard_normal(len(x), dtype=np.float32) * np.float32(corpus.sigma[c]))
        return np.clip(x, -32768, 32767).astype(np.int16)

    with ThreadPoolExecutor(max(1, threads)) as ex:
        caps = list(ex.map(one, range(lo, hi)))
    lens = np.array([len(c) for c in caps], dtype=np.int64)
    off = np.zeros(hi - lo + 1, dtype=np.int64)
    np.cumsum(lens, out=off[1:])
    return np.concatenate(caps), off


def python_reference_record():
    """The unmodified Python reference as timed in the build container (it cannot travel to the GPU box)."""
    p = os.path.join(ROOT, "profiles", "r2_python_reference.json")
    if os.path.exists(p):
        try:
            return json.load(open(p))
        except Exception:  # noqa: BLE001
            return None
    return None


def run_reference_python(args):
    """--impl reference --python: afskmodem.Receiver.load itself (unmodified, /root/reference) over a prefix
    of the workload as wav files, one process per host core.  Build container only."""
    if not os.path.isdir("/root/reference"):
        print(json.dumps({"impl": "reference", "unavailable": "/root/reference is not mounted on this machine"}))
        return
    import multiprocessing as mp
    import shutil
    import tempfile
    import wave

    from oracle import ref_harness
    corpus = Corpus(args.workload, resolve_workload(args.workload)[2])
    nsample = args.captures if args.captures else 64
    cores = os.cpu_count() or 1
    samples, off = host_sample_batch(corpus, 0, nsample, cores)
    root = "/dev/shm" if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else None
    tmpdir = tempfile.mkdtemp(prefix="afsk_ref_", dir=root)
    try:
        names = []
        for c in range(nsample):
            fn = os.path.join(tmpdir, f"cap{c:05d}.wav")
            with wave.open(fn, "wb") as f:
                f.setnchannels(1); f.setsampwidth(2); f.setframerate(48000)
                f.writeframes(samples[off[c]:off[c + 1]].astype("<i2").tobytes())
            names.append(fn)
        jobs = [(fn, int(corpus.baud_rx[c]), int(corpus.amp_end[c])) for c, fn in enumerate(names)]
        with mp.Pool(cores) as pool:
            pool.map(ref_harness.load_file_job, jobs[:cores])              # warm-up: imports
            t0 = time.perf_counter()
            outs = pool.map(ref_harness.load_file_job, jobs, chunksize=1)
            dt = time.perf_counter() - t0
        t0 = time.perf_counter()
        ref_harness.load_file_job(jobs[0])
        one = time.perf_counter() - t0
    finally:
        shutil.rmtree(tmpdir, ignore_errors=True)
    from oracle import oracle as O
    O.build()
    datas, _ = O.rx_decode_batch(samples, off, corpus.baud_rx[:nsample], corpus.amp_end[:nsample], threads=cores)
    agree = sum(1 for a, b in zip(outs, datas) if a == b)
    val = float(off[-1]) / dt / 1e6
    rec = {"impl": "reference", "kind": "reference (unmodified afskmodem.py, Receiver.load incl. wav read)",
           "metric": "decoded Msamples/s", "value": val, "unit": "Msamples/s", "cores": cores,
           "per_core": float(off[1]) / one / 1e6,
           "sample": f"first {nsample} captures of {corpus.name(corpus.per_gpu)} ({int(off[-1])} samples) as wav files in /dev/shm, "
                     f"multiprocessing.Pool({cores}), {dt:.2f} s wall",
           "payloads_equal_to_oracle_port": agree, "captures": nsample,
           "where": "build container (no GPU); the Python reference cannot travel to the GPU box",
           "python": sys.version.split()[0]}
    print(json.dumps(rec))


def run_reference(args):
    """Reference arm: the oracle port of afskmodem.py's Receiver.load compute on all host threads, the
    FULL batch of the workload per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if args.python:
        return run_reference_python(args)
    from oracle import oracle as O
    O.build()
    cores = os.cpu_count() or 1
    corpus = Corpus(args.workload, resolve_workload(args.workload)[2])
    B = args.captures if args.captures else corpus.per_gpu
    if args.workload == "c4":
        B = min(B, 8)                                   # 147 M samples each: bounded sample
    samples, off = host_sample_batch(corpus, 0, B, cores)
    baud, thr = corpus.baud_rx[:B], corpus.amp_end[:B]
    for _ in range(max(args.warmup, 1)):
        O.rx_decode_batch(samples, off, baud, thr, threads=cores)
    t0 = time.perf_counter()
    nbytes = 0
    for _ in range(args.steps):
        datas, _ = O.rx_decode_batch(samples, off, baud, thr, threads=cores)
        nbytes += sum(len(d) for d in datas)
    dt = time.perf_counter() - t0
    ms = dt / args.steps * 1000
    val = float(off[-1]) / (ms / 1000) / 1e6
    sample = (f"all {B} captures of the {args.workload} recipe ({int(off[-1])} samples) per step, C port of afskmodem.py "
              f"on {cores} threads")
    line = {"impl": "reference", "metric": "decoded Msamples/s", "value": val, "unit": "Msamples/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int16",
            "data": "synthetic", "mbit_s": 8 * nbytes / dt / 1e6,
            "config": {"workload": corpus.name(B), "captures_per_gpu": B, "samples_per_gpu": int(off[-1]),
                       "baud": corpus.baud or "mixed", "payload_bytes": corpus.payload_bytes or "16-4096", "sample": sample},
            "cpu_baseline": {"value": val, "unit": "Msamples/s", "cores": cores, "kind": "port", "sample": sample,
                             "python_reference": python_reference_record()},
            "e2e": {"value": val, "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
class Ctx:
    """process-wide state of the b200 arm"""
    rank = 0
    world = 1
    local = 0
    dev = None
    ndev = 1
    stride = 1


def barrier():
    import torch
    import torch.distributed as dist
    if Ctx.world > 1:
        dist.barrier()
    torch.cuda.synchronize(Ctx.dev)


def allreduce(vals, op="sum"):
    """list of floats -> list of floats reduced over the ranks"""
    import torch
    import torch.distributed as dist
    t = torch.tensor([float(v) for v in vals], dtype=torch.float64, device=Ctx.dev)
    if Ctx.world > 1:
        dist.all_reduce(t, op={"sum": dist.ReduceOp.SUM, "max": dist.ReduceOp.MAX, "min": dist.ReduceOp.MIN}[op])
    return [float(v) for v in t.cpu()]


def allgather_floats(v: float):
    import torch
    import torch.distributed as dist
    t = torch.tensor([float(v)], dtype=torch.float64, device=Ctx.dev)
    if Ctx.world == 1:
        return [float(v)]
    out = [torch.zeros(1, dtype=torch.float64, device=Ctx.dev) for _ in range(Ctx.world)]
    dist.all_gather(out, t)
    return [float(o.item()) for o in out]


def oracle_check(samples, offsets, baud, amp_end, batch, captures, threads):
    """GPU results of `captures` (indices into the batch) against the CPU oracle:
    (checked, failures, seconds the oracle took, samples it decoded)."""
    from oracle import oracle as O
    if not len(captures):
        return 0, 0, 0.0, 0
    captures = list(captures)
    if captures == list(range(captures[0], captures[-1] + 1)):       # a contiguous range: one D2H copy
        a, b = captures[0], captures[-1] + 1
        hs = samples[int(offsets[a]):int(offsets[b])].cpu().numpy()
        off = np.asarray(offsets[a:b + 1], dtype=np.int64) - int(offsets[a])
    else:
        parts = [samples[int(offsets[c]):int(offsets[c + 1])].cpu().numpy() for c in captures]
        off = np.zeros(len(parts) + 1, dtype=np.int64)
        np.cumsum([len(p) for p in parts], out=off[1:])
        hs = np.concatenate(parts)
    t0 = time.perf_counter()
    datas, ores = O.rx_decode_batch(hs, off, np.asarray(baud)[captures], np.asarray(amp_end)[captures], threads=threads)
    dt = time.perf_counter() - t0
    bad = 0
    for i, c in enumerate(captures):
        got = (int(batch.status[c]), int(batch.clock[c]), int(batch.train_end[c]), int(batch.nbits[c]), batch.payload(c))
        want = (int(ores[i].status), int(ores[i].clock), int(ores[i].train_end), int(ores[i].nbits), datas[i])
        if int(ores[i].status) < 0:               # the reference raises: only the status is defined
            got, want = got[:1], want[:1]
        bad += got != want
    return len(captures), bad, dt, int(off[-1])


def time_resident(sess, stream, steps, warmup, preload_s=1.0, sampler=None):
    """W warm-up decodes, ~preload_s of the same load to ramp the clocks, then exactly `steps` decodes
    between CUDA events, barrier + synchronize on both sides.  Returns (elapsed ms of this rank, summed
    dominant-kernel ms, dominant-kernel launches)."""
    import torch
    for _ in range(warmup):
        sess.run(stream)
    if sampler:
        sampler.start()
    t_end = time.time() + preload_s
    while time.time() < t_end:
        sess.run(stream)
        torch.cuda.synchronize(Ctx.dev)
    sess.set_timing(True)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        sess.run(stream)
    e1.record()
    barrier()
    elapsed = e0.elapsed_time(e1)
    demod_ms, demod_launches = sess.demod_time()
    sess.set_timing(False)
    return elapsed, demod_ms, demod_launches


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, copy read+write)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def roofline_record(wl, B, total, steps, elapsed_ms, demod_ms, demod_launches, kernel="k_demod"):
    peak, peak_src = hbm_peak()
    per_decode = demod_ms / steps
    launches = max(demod_launches, 1) / steps
    achieved = 2.0 * total / (per_decode / 1000) / 1e9 if per_decode > 0 else 0.0
    traffic = ceiling = None
    tp = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(tp):
        tj = json.load(open(tp))
        # ncu dram bytes of the dominant launch, full-size default batch of that workload only
        traffic = tj.get(f"k_demod_{wl}_dram_bytes_per_launch") if B == resolve_workload(wl)[2] else None
        ceiling = tj.get("hbm_read_only_ceiling_gbs")
    return {"kernel": kernel, "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
            "frac": achieved / peak, "traffic": traffic,
            "traffic_source": "profiles/roofline_traffic.json (ncu --set full of this workload, not this run)" if traffic else None,
            "peak_source": peak_src,
            # the demodulator only reads; a read-only stream runs above the copy (read+write) peak on this part
            "read_only_ceiling": ceiling, "frac_of_read_only_ceiling": achieved / ceiling if ceiling else None,
            "algorithmic_bytes_per_launch": 2 * total / launches, "avg_launch_ms": per_decode / launches,
            "launches_per_step": launches, "share_of_step": per_decode / (elapsed_ms / steps),
            "step_frac_of_peak": 2.0 * total / (elapsed_ms / steps / 1000) / 1e9 / peak}


DUMP_BYTES = 64 << 20


def dump_outputs(batch, out_dir: str) -> None:
    """--dump-outputs: what a caller of the timed decode receives (an RxBatch) as out_dir/<name>.npy, so that
    two builds run with the same arguments can be compared output for output.  Per capture: its index in the
    corpus and the five stage integers (float64, exact); payload_bytes.npy (float32) holds the payloads one
    after another, payload_offsets.npy where each starts.  When that could pass 64 MB, the captures written
    are a prefix of a fixed permutation (seed 0) of the corpus that fits.  A capture is budgeted at its payload
    capacity, which the plan derives from the inputs alone, so every build writes the same captures."""
    res = batch.results
    fields = res.dtype.names
    nbytes = np.maximum(res["nbytes"].astype(np.int64), 0)
    cost = 8 * (len(fields) + 2) + 4 * np.diff(batch.out_off)    # index, stage integers, offset, payload capacity
    order = np.random.default_rng(0).permutation(len(res))
    keep = np.sort(order[np.cumsum(cost[order]) <= DUMP_BYTES - (1 << 16)])   # room for the headers
    off = np.zeros(len(keep) + 1, dtype=np.int64)
    np.cumsum(nbytes[keep], out=off[1:])
    pay = np.zeros(int(off[-1]), dtype=np.float32)
    for i, c in enumerate(keep):
        o = int(batch.out_off[c])
        pay[off[i]:off[i + 1]] = batch.blob[o:o + int(nbytes[c])]
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"capture_index": keep, "payload_offsets": off, **{f: res[f][keep] for f in fields}}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float64))
    np.save(os.path.join(out_dir, "payload_bytes.npy"), pay)


def results_sha256(batch) -> str:
    """SHA-256 over the stage integers of every capture and its payload bytes, in corpus order."""
    h = hashlib.sha256()
    h.update(np.ascontiguousarray(batch.results).tobytes())
    nb = batch.results["nbytes"]
    for c in range(len(batch)):
        if nb[c] > 0:
            o = int(batch.out_off[c])
            h.update(batch.blob[o:o + int(nb[c])].tobytes())
    return h.hexdigest()


def run_workload(args, wl, captures, steps, main=False):
    """Weak-scaling record of one workload: rank r decodes captures [r*B, (r+1)*B) of one global corpus."""
    import torch

    import afskmodem_b200 as A
    corpus = Corpus(wl, (captures or resolve_workload(wl)[2]) * Ctx.world)
    B = corpus.total // Ctx.world
    lo, hi = Ctx.rank * B, (Ctx.rank + 1) * B
    samples, offsets = build_on_gpu(corpus, lo, hi, Ctx.local)
    spec = corpus.spec(lo, hi)
    total = int(offsets[-1])
    sess = A.RxSession(offsets, spec["baud_rx"], spec["amp_end"], Ctx.local)
    sess.bind(samples.data_ptr(), samples.numel())
    stream = torch.cuda.current_stream(Ctx.dev).cuda_stream

    # ---- correctness against the oracle on EVERY rank (outside every timed region) ----
    sess.run(stream)
    batch = sess.download(stream)
    decoded_bytes = batch.total_payload_bytes()
    threads = max(1, (os.cpu_count() or 1) // Ctx.world)
    raising = (spec["baud_rx"] == 9600) | (spec["baud_rx"] == 4800)
    if wl == "c4":
        picks = list(range(min(B, 8)))
    else:
        n_chk = B if (main and Ctx.world == 1 and not args.no_cpu_baseline) else min(B, args.parity_captures)
        picks = list(range(n_chk))
    cpu = None
    if main and Ctx.world == 1 and not args.no_cpu_baseline:           # warm the oracle's thread pool and page in its code
        oracle_check(samples, offsets, spec["baud_rx"], spec["amp_end"], batch, picks[:min(len(picks), 16)], threads)
    checked, bad, dt_oracle, n_oracle = oracle_check(samples, offsets, spec["baud_rx"], spec["amp_end"], batch, picks, threads)
    exact = int(sum(batch.payload(c) == spec["payloads"][c] for c in range(B)))
    n_raise = int((batch.status < 0).sum())
    bad += int(n_raise != int(raising.sum()))
    checked_all, bad_all, exact_all, raise_all = allreduce([checked, bad, exact, n_raise])
    if bad_all and os.environ.get("AFSK_BENCH_NOPARITY") != "1":
        raise SystemExit(f"PARITY FAILURE ({wl}): {int(bad_all)} of {int(checked_all)} captures differ from the oracle")

    # ---- device-resident timing ----
    sampler = ClockSampler(Ctx.local) if (Ctx.rank == 0 and main) else None
    elapsed, demod_ms, demod_launches = time_resident(sess, stream, steps, args.warmup,
                                                      float(os.environ.get("AFSK_BENCH_PRELOAD_S", "1.0" if main else "0.3")), sampler)
    clocks = sampler.stop() if sampler else None
    if main and args.dump_outputs and args.scaling == "weak":
        from afskmodem_b200 import shard
        final = shard.gather_rx(sess.download(stream), dst=0)      # the last timed decode, all ranks in corpus order
        if Ctx.rank == 0:
            dump_outputs(final, args.dump_outputs)
    rank_ms = allgather_floats(elapsed / steps)
    ms_per_step = max(rank_ms)
    all_samples, all_bytes = allreduce([total, decoded_bytes])
    value = all_samples / (ms_per_step / 1000) / 1e6
    rec = {"value": value, "unit": "Msamples/s", "ms_per_step": ms_per_step, "steps": steps,
           "mbit_s": 8 * all_bytes / (ms_per_step / 1000) / 1e6,
           "workload": corpus.name(B), "captures_per_gpu": B, "samples_per_gpu": total,
           "rank_ms": rank_ms, "payloads_exact": int(exact_all), "captures_raising_like_reference": int(raise_all),
           "parity_checked_vs_oracle": int(checked_all), "parity_failures": int(bad_all),
           "gpu_launches": steps * sess.launches,
           "roofline": roofline_record(wl, B, total, steps, elapsed, demod_ms, demod_launches)}
    if main:
        rec.update({"clocks": clocks})
        if Ctx.world == 1 and not args.no_cpu_baseline and checked > 0:
            # the parity pass above IS the CPU baseline: the oracle decoded these captures on all host threads
            cpu = {"value": float(n_oracle) / dt_oracle / 1e6, "unit": "Msamples/s", "cores": threads, "kind": "port",
                   "sample": f"{'all' if checked == B else 'first'} {checked} captures of the workload ({n_oracle} samples), C port of "
                             f"afskmodem.py Receiver.load compute, {threads} threads, {dt_oracle:.2f} s wall; every payload and "
                             "stage integer equal to the GPU's",
                   "python_reference": python_reference_record()}
        rec["cpu_baseline"] = cpu
    return rec, (corpus, samples, offsets, spec, sess, batch)


def run_e2e(args, state, all_samples):
    """End to end through the public API with host buffers; plus the wav-file leg, the cold first call and
    the single-file latency (rank 0, N=1)."""
    import torch

    import afskmodem_b200 as A
    from afskmodem_b200 import _cabi
    corpus, samples, offsets, spec, sess, batch = state
    total, B = int(offsets[-1]), len(offsets) - 1
    pin = _cabi.PinnedArray((total + 64,), np.int16)
    pin.array[:total] = samples[:total].cpu().numpy()
    rx = A.Receiver(1200, 18000, AMP_END, device=Ctx.local)
    kw = {"baud_rate": spec["baud_rx"], "amp_end_threshold": spec["amp_end"]}     # per-capture settings
    t0 = time.perf_counter()
    rx.decode_batch(pin.array, offsets, **kw)      # first call: plans, device buffers, pinned result staging
    first_ms = (time.perf_counter() - t0) * 1e3
    barrier()
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s0.record()
    for _ in range(args.e2e_steps):
        hb = rx.decode_batch(pin.array, offsets, **kw)
    s1.record()
    barrier()
    e2e_ms = max(allgather_floats(s0.elapsed_time(s1))) / args.e2e_steps
    assert hb.total_payload_bytes() == batch.total_payload_bytes()
    assert np.array_equal(hb.results, batch.results), "host-buffer decode != device-resident decode"
    # what the PCIe link alone allows: the same pinned buffer copied to the device, nothing else
    # (outside the timed region; explains e2e, is not part of it)
    sess_e = rx._cache[1]
    h0, h1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    h0.record()
    for _ in range(2):
        sess_e.d_samples.upload(pin.array[:total])
    h1.record()
    torch.cuda.synchronize(Ctx.dev)
    h2d_ms = h0.elapsed_time(h1) / 2
    e2e = {"value": all_samples / (e2e_ms / 1000) / 1e6, "unit": "Msamples/s", "ms_per_step": e2e_ms,
           "h2d_bytes_per_step": total * 2, "d2h_bytes_per_step": int(32 * B + hb.out_off[-1]),
           "api": "Receiver.decode_batch(pinned int16 samples, offsets, baud_rate=[...], amp_end_threshold=[...])",
           "h2d_overlapped_ranges": len(getattr(sess_e, "sessions", [None])),
           "steps": args.e2e_steps, "first_call_ms": first_ms, "h2d_only_ms": h2d_ms, "h2d_only_gbs": 2.0 * total / h2d_ms / 1e6,
           "share_of_step_in_h2d": h2d_ms / e2e_ms,
           "h2d_gate": (lambda g: None if g is None else f"{g.slots} of every {g.group} consecutive GPUs copy at a time, taking turns range by "
                                                             "range (afskmodem_b200/h2d_gate.py)")(getattr(sess_e, "gate", None)),
           "aggregate_h2d_gbs": 2.0 * all_samples / (e2e_ms / 1000) / 1e9}
    rx.close()
    extra = {}
    # ---- ONE corpus on all the GPUs of this job from ONE process (the product's multi-device call):
    #      rank 0 shards its batch over the N devices the ranks use, the other ranks idle at the barrier
    if Ctx.world > 1 and not args.no_sharded_api:
        if Ctx.rank == 0:
            devs = [r * Ctx.stride for r in range(Ctx.world)]
            rxs = A.Receiver(1200, 18000, AMP_END, device=Ctx.local)
            try:
                rxs.decode_batch(pin.array, offsets, devices=devs, **kw)
                best = 1e9
                for _ in range(args.e2e_steps):
                    t0 = time.perf_counter()
                    sb = rxs.decode_batch(pin.array, offsets, devices=devs, **kw)
                    best = min(best, time.perf_counter() - t0)
                sh = rxs._cache[1]
                extra["e2e_one_process"] = {
                    "value": total / best / 1e6, "unit": "Msamples/s", "ms": best * 1e3, "devices": devs,
                    "api": "Receiver.decode_batch(pinned samples, offsets, devices=[...]) — ShardedRxSession: one host thread + "
                           "streams per device, ranges balanced by predicted time, host gather into one RxBatch",
                    "equal_to_single_device": bool(np.array_equal(sb.results, batch.results) and
                                                   sb.payloads() == batch.payloads()),
                    "device_ms": [round(v, 3) for v in sh.device_ms], "captures_per_device": [hi - lo for lo, hi in sh.ranges]}
            except Exception as e:  # noqa: BLE001 - an extra record must not take the line down
                extra["e2e_one_process"] = {"error": repr(e)[:300]}
            rxs.close()
        barrier()
    # ---- the same path from wav FILES (Receiver.load_batch), a bounded prefix of the batch; cold call and
    #      single-file latency in fresh processes
    if Ctx.rank == 0 and Ctx.world == 1 and not args.no_files:
        import shutil
        import tempfile
        nf = min(B, args.file_captures)
        while nf > 1 and 2 * int(offsets[nf]) > 2_500_000_000:       # keep the temporary files under 2.5 GB
            nf -= 1
        root = "/dev/shm" if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else None
        tmpdir = tempfile.mkdtemp(prefix="afsk_bench_", dir=root)
        try:
            names = [os.path.join(tmpdir, f"cap{c:05d}.wav") for c in range(nf)]
            A.modem.write_wav_batch(names, pin.array, offsets[:nf], np.diff(offsets[:nf + 1]))
            rxf = A.Receiver(corpus.baud or 1200, 18000, AMP_END, device=Ctx.local)
            want = [batch.payload(c) for c in range(nf)]
            res = {}
            for mode, kwf in (("ring", {}), ("pinned_corpus", {"keep_host_copy": True})):
                t0 = time.perf_counter()           # first call of this mode in this process
                rxf.load_batch(names, string=False, errors="return", log=False, **kwf)
                first = (time.perf_counter() - t0) * 1e3
                dtf = 1e9
                for _ in range(3):
                    t0 = time.perf_counter()
                    got = rxf.load_batch(names, string=False, errors="return", log=False, **kwf)
                    dtf = min(dtf, time.perf_counter() - t0)
                assert [g if isinstance(g, bytes) else b"" for g in got] == want, "load_batch != decode"
                res[mode] = {"value": float(offsets[nf]) / dtf / 1e6, "ms": dtf * 1e3, "first_call_ms": first}
                rxf.close()
            extra["e2e_files"] = {"value": res["ring"]["value"], "unit": "Msamples/s", "files": nf, "ms": res["ring"]["ms"],
                                  "first_call_ms": res["ring"]["first_call_ms"], "file_bytes": int(2 * offsets[nf] + 44 * nf),
                                  "where": tmpdir.rsplit("/", 1)[0], "api": "Receiver.load_batch(filenames, string=False)",
                                  "host_threads": os.cpu_count(), "staging": "ring of four pinned 8 MB slots (default)",
                                  "pinned_corpus_mode": res["pinned_corpus"]}
            # cold: the first load_batch of a FRESH process (CUDA initialisation reported separately)
            try:
                out = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "cold_call.py"), str(Ctx.local), tmpdir, str(nf),
                                      str(corpus.baud or 1200)], capture_output=True, text=True, timeout=300)
                extra["e2e_cold"] = json.loads(out.stdout.strip().splitlines()[-1])
                extra["e2e_cold"]["steady_ms"] = res["ring"]["ms"]
                extra["e2e_cold"]["first_over_steady"] = extra["e2e_cold"]["first_load_batch_ms"] / res["ring"]["ms"]
            except Exception as e:  # noqa: BLE001
                extra["e2e_cold"] = {"error": repr(e)[:300]}
        finally:
            shutil.rmtree(tmpdir, ignore_errors=True)
    pin.close()
    return e2e, extra


def run_tx(args):
    """Transmitter as a measured path (rows a12-a14): e2e through Transmitter.save_batch (synthesis, D2H,
    wav files written by the library's host threads) and k_synth_var at 4800 baud."""
    import shutil
    import tempfile

    import torch

    import afskmodem_b200 as A
    out = {}
    rng = np.random.default_rng([8, Ctx.rank])
    peak, _ = hbm_peak()
    # k_synth: the c2 batch (4096 x 1 KB at 1200 baud, 4.9 GB written per launch);
    # k_synth_var: 4800 baud (mark tone 8 frames, space tone 10: bit starts are a prefix sum)
    nb = 4096
    pay = [rng.integers(0, 256, 1024, dtype=np.uint8).tobytes() for _ in range(nb)]
    for name, baud in (("k_synth", 1200), ("k_synth_var_4800", 4800)):
        tx = A.TxSession(pay, baud, int(baud * 0.5 / 2), Ctx.local)
        tx.upload()
        for _ in range(3):
            tx.run()
        torch.cuda.synchronize(Ctx.dev)
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        stream = torch.cuda.current_stream(Ctx.dev).cuda_stream
        t0.record()
        for _ in range(5):
            tx.run(stream)
        t1.record()
        torch.cuda.synchronize(Ctx.dev)
        ms = t0.elapsed_time(t1) / 5
        frames = int(tx.out_len.astype(np.int64).sum())
        out[name] = {"frames": frames, "ms": ms, "msamples_s": frames / ms / 1e3, "achieved_gbs_written": 2.0 * frames / ms / 1e6,
                     "frac": 2.0 * frames / ms / 1e6 / peak, "launches_per_synth": 1 if name == "k_synth" else 2}
        tx.close()
    agg, = allreduce([out["k_synth"]["msamples_s"]])
    out.update({"kernel": "k_synth", "frames": out["k_synth"]["frames"], "ms": out["k_synth"]["ms"],
                "msamples_s": out["k_synth"]["msamples_s"], "msamples_s_all_gpus": agg,
                "achieved_gbs_written": out["k_synth"]["achieved_gbs_written"],
                "roofline": {"kernel": "k_synth", "bound": "hbm", "achieved": out["k_synth"]["achieved_gbs_written"], "peak": peak,
                             "unit": "GB/s", "frac": out["k_synth"]["frac"],
                             "algorithmic_bytes_per_launch": 2 * out["k_synth"]["frames"], "traffic": None}})
    if Ctx.rank == 0 and Ctx.world == 1 and not args.no_files:
        nf = 1024
        root = "/dev/shm" if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else None
        tmpdir = tempfile.mkdtemp(prefix="afsk_txbench_", dir=root)
        try:
            names = [os.path.join(tmpdir, f"tx{c:05d}.wav") for c in range(nf)]
            t = A.Transmitter(1200, 0.5, device=Ctx.local)
            t.save_batch(pay[:nf], names)
            best = 1e9
            for _ in range(3):
                t0 = time.perf_counter()
                t.save_batch(pay[:nf], names)
                best = min(best, time.perf_counter() - t0)
            frames = nf * ((600 + 4 + 14 * 1024) * 40 + 4800)
            out["e2e_save_batch"] = {"value": frames / best / 1e6, "unit": "Msamples/s", "files": nf, "ms": best * 1e3,
                                     "d2h_bytes": 2 * frames, "where": tmpdir.rsplit("/", 1)[0],
                                     "api": "Transmitter.save_batch(payloads, filenames)"}
        finally:
            shutil.rmtree(tmpdir, ignore_errors=True)
    return out


def run_latency(args):
    """BASELINE configs[0]: Transmitter(1200).save -> Receiver(1200).load of 'Hello World!' on one wav
    (reference: 10 ms + 67 ms on one host core, SURVEY §6), warm and in a fresh process."""
    import shutil
    import tempfile

    import afskmodem_b200 as A
    root = "/dev/shm" if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else None
    tmpdir = tempfile.mkdtemp(prefix="afsk_lat_", dir=root)
    try:
        fn = os.path.join(tmpdir, "hello.wav")
        t = A.Transmitter(1200, device=Ctx.local)
        r = A.Receiver(1200, device=Ctx.local)
        t.save("Hello World!", fn)
        assert r.load(fn, True) == "Hello World!"
        fn2 = os.path.join(tmpdir, "other.wav")
        t.save("A different, longer message so that the layout changes between calls.", fn2)
        lat = {"load_ms": [], "save_ms": [], "load_alternating_ms": []}
        for _ in range(50):
            t0 = time.perf_counter(); r.load(fn, True); lat["load_ms"].append((time.perf_counter() - t0) * 1e3)
        for i in range(50):
            t0 = time.perf_counter(); r.load(fn2 if i & 1 else fn, True); lat["load_alternating_ms"].append((time.perf_counter() - t0) * 1e3)
        for _ in range(20):
            t0 = time.perf_counter(); t.save("Hello World!", fn); lat["save_ms"].append((time.perf_counter() - t0) * 1e3)
        rec = {k: {"median": statistics.median(v), "min": min(v)} for k, v in lat.items()}
        rec["what"] = ("Receiver(1200).load / Transmitter(1200).save of 'Hello World!' (35,680 frames), same receiver object; "
                       "load_alternating: two files of different length in turn (plan re-targeted every call)")
        rec["reference_ms"] = {"save": 10, "load": 67, "source": "SURVEY.md §6, one host core of the build container"}
        r.close()
        try:
            out = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "cold_call.py"), str(Ctx.local), fn, "0", "1200"],
                                 capture_output=True, text=True, timeout=300)
            rec["fresh_process"] = json.loads(out.stdout.strip().splitlines()[-1])
        except Exception as e:  # noqa: BLE001
            rec["fresh_process"] = {"error": repr(e)[:300]}
        return rec
    finally:
        shutil.rmtree(tmpdir, ignore_errors=True)


def run_sharded(args, total_captures, steps):
    """Strong scaling on ONE corpus: c5 recipe, `total_captures` captures seeded by capture index, cut into
    world contiguous ranges balanced by predicted time (shard.capture_cost), every rank decodes its range
    from HBM, results gathered on the host into one RxBatch (shard.gather_rx)."""
    import torch

    import afskmodem_b200 as A
    from afskmodem_b200 import shard
    corpus = Corpus("c5", total_captures)
    lens = corpus.lens()
    cost = shard.capture_cost(lens, corpus.baud_rx, resident=True)
    ranges = shard.shard_captures(lens, Ctx.world, cost)
    lo, hi = ranges[Ctx.rank]
    samples, offsets = build_on_gpu(corpus, lo, hi, Ctx.local)
    spec = corpus.spec(lo, hi)
    total = int(offsets[-1])
    sess = A.RxSession(offsets, spec["baud_rx"], spec["amp_end"], Ctx.local)
    sess.bind(samples.data_ptr(), samples.numel())
    stream = torch.cuda.current_stream(Ctx.dev).cuda_stream
    sess.run(stream)
    batch = sess.download(stream)
    threads = max(1, (os.cpu_count() or 1) // Ctx.world)
    B = hi - lo
    picks = sorted(set(np.linspace(0, B - 1, min(B, args.parity_captures)).astype(int).tolist())) if B else []
    checked, bad, _, _ = oracle_check(samples, offsets, spec["baud_rx"], spec["amp_end"], batch, picks, threads)
    raising = (spec["baud_rx"] == 9600) | (spec["baud_rx"] == 4800)
    bad += int(int((batch.status < 0).sum()) != int(raising.sum()))
    checked_all, bad_all = allreduce([checked, bad])
    elapsed, demod_ms, demod_launches = time_resident(sess, stream, steps, args.warmup, 0.3)
    if args.dump_outputs and args.scaling == "strong":
        final = shard.gather_rx(sess.download(stream), dst=0)
        if Ctx.rank == 0:
            dump_outputs(final, args.dump_outputs)
    rank_ms = allgather_floats(elapsed / steps)
    ms = max(rank_ms)
    barrier()
    t0 = time.perf_counter()
    merged = shard.gather_rx(batch, dst=0)
    barrier()
    gather_ms = (time.perf_counter() - t0) * 1e3
    all_samples, = allreduce([total])
    rec = None
    if Ctx.rank == 0:
        sha = results_sha256(merged)
        known = None
        kp = os.path.join(ROOT, "profiles", "c5_corpus_sha256.json")
        if os.path.exists(kp):
            known = json.load(open(kp)).get(str(total_captures))
        rec = {"workload": f"ONE corpus: {corpus.name(total_captures)}; {Ctx.world} contiguous ranges balanced by predicted time",
               "scaling": "strong", "captures": total_captures, "samples": int(all_samples),
               "value": all_samples / (ms / 1000) / 1e6, "unit": "Msamples/s", "ms_per_step": ms, "steps": steps,
               "rank_ms": rank_ms, "imbalance_max_over_mean": ms / (sum(rank_ms) / len(rank_ms)),
               "predicted_imbalance": shard.imbalance(cost, ranges),
               "imbalance_if_sharded_by_samples": shard.imbalance(cost, shard.shard_captures(lens, Ctx.world)),
               "captures_per_rank": [b - a for a, b in ranges],
               "host_gather_ms": gather_ms, "gathered_captures": len(merged),
               "sha256_results_payloads": sha, "sha256_recorded_single_gpu": known,
               "sha256_matches_single_gpu": (sha == known) if known else None,
               "parity_checked_vs_oracle": int(checked_all), "parity_failures": int(bad_all),
               "payload_bytes": merged.total_payload_bytes(),
               "roofline_rank0": roofline_record("c5", B, total, steps, elapsed, demod_ms, demod_launches)}
    sess.close()
    del samples
    torch.cuda.empty_cache()
    if bad_all:
        raise SystemExit(f"PARITY FAILURE (sharded corpus): {int(bad_all)} of {int(checked_all)} captures differ from the oracle")
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--python", action="store_true", help="with --impl reference: the unmodified afskmodem.py (build container only)")
    ap.add_argument("--captures", type=int, default=0, help="captures per GPU (default: the workload's)")
    ap.add_argument("--workload", default="c2", help="c2 (default, the line of record), c3, c4, c5 or w<baud>")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="strong: the line's value is ONE c5 corpus (--corpus-captures) sharded over the ranks")
    ap.add_argument("--corpus-captures", type=int, default=C5_CORPUS)
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--parity-captures", type=int, default=256, help="captures every rank checks against the oracle per record")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-files", action="store_true", help="skip the wav-file legs (load_batch, save_batch, cold call)")
    ap.add_argument("--no-extra", action="store_true", help="skip the c3/c4/c5 sub-records, the sharded corpus, tx and latency")
    ap.add_argument("--no-sharded", action="store_true")
    ap.add_argument("--no-sharded-api", action="store_true")
    ap.add_argument("--file-captures", type=int, default=1024)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the line's last timed decode returned as DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of --impl b200")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist

    import afskmodem_b200 as A
    from afskmodem_b200 import _cabi

    Ctx.rank = int(os.environ.get("RANK", "0"))
    Ctx.world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # Topology-aware placement: with fewer ranks than visible GPUs, spread the ranks over the box
    # (rank r -> GPU r * ndev / world).  Measured on the 8-GPU box: four ranks on GPUs 0-3 copy from pinned
    # host memory at 28.7 GB/s each (two GPUs share one PCIe uplink), on GPUs 0,2,4,6 at 53.1 GB/s each.
    Ctx.ndev = torch.cuda.device_count()
    Ctx.stride = 1
    if Ctx.world > 1 and Ctx.ndev >= 2 * Ctx.world and os.environ.get("AFSK_BENCH_SPREAD", "1") != "0":
        Ctx.stride = Ctx.ndev // Ctx.world
    local *= Ctx.stride
    Ctx.local = local
    A.LOG_LEVEL = 5
    _cabi.require_device(local)              # no CPU fallback
    torch.cuda.set_device(local)
    Ctx.dev = torch.device("cuda", local)
    if Ctx.world > 1:
        dist.init_process_group("nccl", device_id=Ctx.dev)
    main_wl = args.workload
    extras = main_wl == "c2" and not args.no_extra and not args.captures

    rec, state = run_workload(args, main_wl, args.captures, args.steps, main=True)
    all_samples = rec["value"] * rec["ms_per_step"] * 1e3
    e2e, extra = (None, {})
    if not args.no_e2e:
        e2e, extra = run_e2e(args, state, all_samples)
    corpus, samples, offsets, spec, sess, batch = state
    B, total = len(offsets) - 1, int(offsets[-1])
    sess.close()
    del samples, state
    torch.cuda.empty_cache()

    tx = run_tx(args) if not args.no_extra else None
    workloads, sharded, latency = {}, None, None
    if extras:
        for wl in ("c3", "c4", "c5"):
            r, st = run_workload(args, wl, 0, max(5, min(args.steps, 10)))
            st[4].close()
            del st
            torch.cuda.empty_cache()
            workloads[wl] = r
        if Ctx.rank == 0 and Ctx.world == 1 and not args.no_files:
            latency = run_latency(args)
    if (extras and not args.no_sharded) or args.scaling == "strong":
        # as the line's own value the sharded corpus takes --steps; as a sub-record, 5 to 10
        sharded = run_sharded(args, args.corpus_captures, args.steps if args.scaling == "strong" else max(5, min(args.steps, 10)))

    if Ctx.rank != 0:
        if Ctx.world > 1:
            dist.destroy_process_group()
        return

    line = {"metric": "decoded Msamples/s", "value": rec["value"], "unit": "Msamples/s", "n_gpus": Ctx.world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": rec["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "int16", "data": "synthetic",
            "mbit_s": rec["mbit_s"],
            "config": {"workload": rec["workload"], "captures_per_gpu": B, "samples_per_gpu": total,
                       "baud": corpus.baud or "mixed", "payload_bytes": corpus.payload_bytes or "16-4096",
                       "corpus": "one global corpus seeded by capture index; rank r decodes captures [r*B, (r+1)*B)",
                       "l2_policy": f"inputs ({2 * total / 1e9:.1f} GB/GPU) larger than L2; no flush",
                       "gpu_of_rank0": local, "gpus_visible": Ctx.ndev, "rank_to_gpu_stride": Ctx.stride,
                       "payloads_exact": rec["payloads_exact"], "captures_raising_like_reference": rec["captures_raising_like_reference"],
                       "parity_checked_vs_oracle": rec["parity_checked_vs_oracle"], "parity_failures": rec["parity_failures"],
                       "parity_ranks": Ctx.world},
            "rank_ms": rec["rank_ms"],
            "clocks": rec["clocks"], "e2e": e2e, "gpu_launches": rec["gpu_launches"],
            "roofline": rec["roofline"], "cpu_baseline": rec["cpu_baseline"], "tx": tx,
            "workloads": workloads or None, "sharded": sharded, "latency": latency}
    line.update(extra)
    bt = os.path.join(ROOT, "profiles", "r2_baud_sweep.json")
    if os.path.exists(bt) and extras:
        try:
            tj = json.load(open(bt))
            line["baud_table"] = {"source": "profiles/r2_baud_sweep.json (tools/baud_sweep.py on a B200, not this run)",
                                  "demod_gbs_by_baud": {k: v["demod_gbs"] for k, v in tj["table"].items()}}
        except Exception:  # noqa: BLE001
            pass
    if args.scaling == "strong" and sharded:
        # the strong-scaling corpus as the line's own value
        line.update({"value": sharded["value"], "ms_per_step": sharded["ms_per_step"], "scaling": "strong",
                     "steps": sharded["steps"], "weak_scaling_record": {"value": rec["value"], "ms_per_step": rec["ms_per_step"]}})
        line["config"]["workload"] = sharded["workload"]
    print(json.dumps(line))
    if Ctx.world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
