"""Streaming receiver throughput: S channels of 1200-baud transmissions separated by silence, pushed
piece by piece through Receiver.open_streams, host-pinned or device-resident input.

    python tools/stream_bench.py [--S 1,64,4096] [--piece 2048,48000] [--seconds 8] [--mix] [--out FILE]

Channel s hears one long traffic recording from frame s * 12345 on, so recordings land at different
places on every channel.  Each configuration runs its push sequence twice on one receiver (finish in
between) and times the second: host wall time of every push, which ends in a synchronize.  Beside it,
receive_all and listen_gate_multi over whole streams of the same traffic (one stream per call, the
only way they run) on the same card.  Card name and power limit are read in the same run.

--mix splits the channels into six equal groups at 300, 600, 1200, 2400, 4000 and 6000 baud, each hearing
traffic at its own baud, and within a group cycles through the three (amp_start, amp_end) threshold pairs of
the c5 corpus; the handle is then opened with open_receive_streams.  A push then decodes one group per distinct
baud among its final recordings.

--format s16,s32,f32 feeds each piece as the columns of a wider card in that sample format (--pitch-extra K: the card
has S + K columns and the window starts at column 1 when K > 0, an odd column): push_interleaved(card[:, c0:c0 + S],
dtype=...) beside the route it replaces, the slice made contiguous, the conversion to int16 and push_interleaved, with
numpy on the host (a pageable card) or torch on the device, run alternately three times on two receivers.  The profiled
run then times the append kernel in each format over device windows (k_stream_frames; k_stream_deinterleave
for contiguous int16), its bytes/s counted over the bytes it must
read and write (n * S * (sample size + 2)).

--layout interleaved feeds each piece as a multi-channel sound card delivers it, n x S frame-major (host input: a
pageable array, as pyaudio's read returns it), three ways in one run: push_interleaved (the GPU de-interleaves it),
a host numpy transpose into the pinned planar buffer followed by push, and .t().contiguous() on the device followed
by push, which is what a user had to do without push_interleaved.  The profiled run then times
k_stream_deinterleave and k_stream_copy's planar append over the same pieces (4 bytes moved per appended frame).

--retain samples,bits,payload runs every configuration once per retention mode, one after the other, on the same
traffic (open_receive_streams(..., retain=...)), and adds a profiled bits-mode run that times k_stream_windows over
the frames it demodulates (2 bytes read per frame of every window it decides, counted from pending_bits and the final
calls).  --windows-bauds profiles it alone at the given bauds on channels whose recordings never close, --stuck
records arena_bytes() against pushed seconds on such channels for each mode (samples mode stops after 60 s) and each
--stuck-variants entry: "message" (a short message, then a full-scale carrier), "tone" (the mark tone alone: no
message, no terminator) and "gap" (a message, one quiet window inside a loud chunk, then the carrier), and
--loopback S times BASELINE config 4 (64 KB at 300 baud) looped back from a transmitter on S channels in the
--loopback-retain mode."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import afskmodem_b200 as A  # noqa: E402
from afskmodem_b200 import _cabi  # noqa: E402
from oracle import oracle as O  # noqa: E402

SHIFT = 12345
MIX_BAUDS = [300, 600, 1200, 2400, 4000, 6000]
MIX_THRESHOLDS = [(18000, 14000), (14000, 11000), (9000, 8000)]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def traffic(n: int, rng, baud: int = 1200) -> np.ndarray:
    """transmissions (10-60 byte payloads, 0.1 s training) separated by 0.2-1.5 s of silence, light noise"""
    tx = A.Transmitter(baud, 0.1)
    msgs = [rng.integers(0, 256, size=int(rng.integers(10, 61)), dtype=np.uint8).tobytes() for _ in range(64)]
    batch = tx.encode_batch(msgs)
    parts, total = [], 0
    while total < n:
        gap = np.zeros(int(rng.integers(9600, 72000)), np.int16)
        fr = batch.frames(int(rng.integers(0, len(msgs))))
        parts += [gap, fr]
        total += len(gap) + len(fr)
    x = np.concatenate(parts)[:n].astype(np.float64) * 0.8 + rng.normal(0, 1500, n)
    return np.clip(np.round(x), -32768, 32767).astype(np.int16)


def mix_groups(S: int):
    """--mix: (baud, first channel, channels) of the six groups"""
    cuts = [S * g // len(MIX_BAUDS) for g in range(len(MIX_BAUDS) + 1)]
    return [(b, cuts[g], cuts[g + 1] - cuts[g]) for g, b in enumerate(MIX_BAUDS)]


def run_config(base, d_base, S: int, piece: int, T: int, device: bool, timeout: float, mix: bool = False,
               route: str = "planar", retain: str = "samples"):
    """base / d_base: one traffic stream, or with mix one per baud of MIX_BAUDS; route: planar, interleaved,
    host-transpose or device-transpose (see --layout)"""
    import torch
    n_push = T // piece
    offsets = np.arange(S + 1, dtype=np.int64) * piece
    pinned = _cabi.PinnedArray((S * piece + 8,), np.int16)
    out = {"S": S, "piece": piece, "input": "device" if device else "host-pinned", "pushes": n_push, "mix": mix,
           "route": route, "retain": retain}
    if route != "planar" and not device:
        out["input"] = "host"
    if mix:
        groups = mix_groups(S)
        rxs = [A.Receiver(b, *MIX_THRESHOLDS[k % 3]) for b, _, n in groups for k in range(n)]
        st = A.open_receive_streams(rxs, timeout, retain=retain)
    else:
        groups = [(1200, 0, S)]
        st = A.Receiver(1200).open_streams(S, timeout, retain=retain)
        base, d_base = [base], [d_base]
    with st:
        for rep in range(2):
            c0 = st.counters()
            times, n_ev, n_rec, rec_frames, n_dec = [], 0, 0, 0, 0
            for i in range(n_push):
                if device:
                    t = torch.cat([torch.as_strided(d_base[g], (n, piece), (SHIFT, 1), i * piece).reshape(-1)
                                   for g, (_, _, n) in enumerate(groups)])
                    if route != "planar":
                        t = t.view(S, piece).t().contiguous()        # the piece as a sound card delivers it
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    if route == "interleaved":
                        ev = st.push_interleaved(t)
                    elif route == "device-transpose":
                        ev = st.push(t.t().contiguous().view(-1), offsets)
                    else:
                        ev = st.push(t, offsets)
                else:
                    for g, (_, c, n) in enumerate(groups):
                        np.copyto(pinned.array[c * piece:(c + n) * piece].reshape(n, piece),
                                  np.lib.stride_tricks.as_strided(base[g][i * piece:], shape=(n, piece), strides=(SHIFT * 2, 2)))
                    if route != "planar":
                        x = pinned.array[:S * piece].reshape(S, piece).T.copy()   # pageable, frame-major
                    t0 = time.perf_counter()
                    if route == "interleaved":
                        ev = st.push_interleaved(x)
                    elif route == "host-transpose":
                        np.copyto(pinned.array[:S * piece].reshape(S, piece), x.T)
                        ev = st.push(pinned.array, offsets)
                    else:
                        ev = st.push(pinned.array, offsets)
                times.append(time.perf_counter() - t0)
                n_ev += len(ev)
                n_rec += int(ev.recorded.sum())
                rec_frames += int((ev.end - ev.start)[ev.recorded].sum())
                n_dec += int(ev.recorded.any())
            c1 = st.counters()
            arena = st.arena_bytes()
            st.finish()
        frames = S * piece * n_push
        t = np.array(times)
        out.update({
            "frames": frames, "seconds": float(t.sum()), "frames_per_s": frames / float(t.sum()),
            "push_ms_median": float(np.median(t) * 1e3), "push_ms_p90": float(np.percentile(t, 90) * 1e3),
            "push_ms_max": float(t.max() * 1e3), "events": n_ev, "recorded": n_rec,
            "recorded_share": rec_frames / frames,
            # counted by the receiver over the timed pushes (afsk_rx_streams_counters)
            "launches_per_push": (c1["launches"] - c0["launches"]) / n_push, "pushes_with_decode": n_dec,
            "moved_frames": c1["moved_frames"] - c0["moved_frames"], "compactions": c1["compactions"] - c0["compactions"],
            # bytes the kernels move per pushed frame: append reads 2 + writes 2, the amplitudes read 2, the decode reads
            # the recorded share (2 per recorded frame), retention moves read 2 + write 2 per moved frame; the host-input
            # staging copy is not in this figure
            "device_bytes_per_frame": 4 + 2 + (2 * rec_frames + 4 * (c1["moved_frames"] - c0["moved_frames"])) / frames,
            "arena_bytes": arena,
            "moved_plane_words": c1["moved_plane_words"] - c0["moved_plane_words"],
            "plane_compactions": c1["plane_compactions"] - c0["plane_compactions"],
        })
    pinned.close()
    return out


def windows_decided(st, ev, before, bf):
    """windows k_stream_windows decided in one bits-mode push: before[s] = (pending start, clock, windows) of channel s
    before it; a final recording that was pending with its clock stored ends with windows [windows, K)"""
    n = 0
    for i in np.flatnonzero(ev.recorded):
        s = int(ev.stream[i])
        R, clk, w = before[s]
        if int(ev.start[i]) == R and clk >= 0:
            span = int(ev.end[i] - ev.start[i]) - bf - clk
            n += max(0, (span + bf - 1) // bf - w) if span > 0 else 0
            before[s] = (-1, -1, 0)
    for s in range(st.S):
        R, clk, w = before[s]
        pend = st.state(s)[1]
        c, w1 = st.pending_bits(s)
        n += w1 - (w if pend == R and c == clk else 0)
    return n


def profile_bits(d_base, S: int, piece: int, T: int, timeout: float):
    """k_stream_windows in a bits-mode run of its own (torch.profiler): kernel time and GB/s over the frames it
    demodulates"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    n_push = T // piece
    offsets = np.arange(S + 1, dtype=np.int64) * piece
    pieces = [torch.as_strided(d_base, (S, piece), (SHIFT, 1), i * piece).contiguous().view(-1) for i in range(n_push)]
    rx, bf = A.Receiver(1200), 40
    with rx.open_streams(S, timeout, retain="bits") as st:
        for t in pieces:
            st.push(t, offsets)
        st.finish()
        torch.cuda.synchronize()
        wins = 0
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for t in pieces:
                before = [(st.state(s)[1],) + st.pending_bits(s) for s in range(S)]
                ev = st.push(t, offsets)
                wins += windows_decided(st, ev, before, bf)
        st.finish()
    ms = 0.0
    for e in prof.key_averages():
        if "k_stream_windows" in e.key:
            us = getattr(e, "device_time_total", None)
            ms += (us if us is not None else getattr(e, "cuda_time_total", 0.0)) / 1e3
    nbytes = 2 * bf * wins
    return {"S": S, "piece": piece, "pushes": n_push, "kernel": "k_stream_windows", "windows": wins, "frames": bf * wins,
            "kernel_ms": ms, "kernel_us_per_push": ms * 1e3 / n_push, "GBps": nbytes / (ms * 1e-3) / 1e9 if ms else None}


def stuck_carrier(S: int, seconds: int, mode: str, variant: str = "message", samples_cap_s: int = 60):
    """arena_bytes() against pushed seconds on recordings that never close, 1 s device pushes at 1200 baud (samples
    mode stops after samples_cap_s seconds).  variant "message": a short message, then a full-scale 1200 Hz carrier
    with no quiet chunk; "tone": the mark tone alone (every window decides 1: no terminator); "gap": the message, 3
    bit lengths of silence (a quiet window inside a loud chunk), then the carrier"""
    import torch
    t = torch.arange(48000, device="cuda", dtype=torch.float64)
    if variant == "tone":
        block = torch.from_numpy(np.tile(O.tone("mark", 1200), 1200)).cuda()     # the Receiver's mark template
    else:
        block = torch.round(30000 * torch.sin(2 * np.pi * 1200 * t / 48000)).to(torch.int16)
    head = block.clone()
    if variant != "tone":
        fr = torch.from_numpy(A.Transmitter(1200, 0.1).encode_batch([b"stuck"]).frames(0)[:-4800].copy()).cuda()
        head[100:100 + len(fr)] = fr
        if variant == "gap":
            head[100 + len(fr):100 + len(fr) + 120] = 0
    offsets = np.arange(S + 1, dtype=np.int64) * 48000
    out = []
    with A.Receiver(1200).open_streams(S, 5.0, retain=mode) as st:
        for i in range(seconds if mode != "samples" else min(seconds, samples_cap_s)):
            st.push((head if i == 0 else block).repeat(S), offsets)
            out.append([i + 1, st.arena_bytes()])
        ended = sum(st.pending_payload(s)[2] for s in range(S)) if mode == "payload" else None
        st.finish()
    return {"S": S, "retain": mode, "variant": variant, "ended_channels": ended, "seconds_vs_arena_bytes": out}


def profile_windows(baud: int, S: int, pushes: int):
    """k_stream_windows alone at one bit length (torch.profiler): S channels whose recordings never close (a message,
    then a full-scale carrier), 1 s device pushes after the clocks are stored; GB/s over the frames of the windows it
    decides (2 bytes each), counted from pending_bits"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    bf = 48000 // baud
    t = torch.arange(48000, device="cuda", dtype=torch.float64)
    block = torch.round(30000 * torch.sin(2 * np.pi * 1200 * t / 48000)).to(torch.int16).repeat(S)
    offsets = np.arange(S + 1, dtype=np.int64) * 48000
    with A.Receiver(baud).open_streams(S, 5.0, retain="bits") as st:
        for _ in range(3):
            st.push(block, offsets)
        w0 = sum(st.pending_bits(s)[1] for s in range(S))
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(pushes):
                st.push(block, offsets)
        w1 = sum(st.pending_bits(s)[1] for s in range(S))
        st.finish()
    ms = 0.0
    for e in prof.key_averages():
        if "k_stream_windows" in e.key:
            us = getattr(e, "device_time_total", None)
            ms += (us if us is not None else getattr(e, "cuda_time_total", 0.0)) / 1e3
    frames = (w1 - w0) * bf
    return {"baud": baud, "bf": bf, "S": S, "pushes": pushes, "windows": w1 - w0, "frames": frames, "kernel_ms": ms,
            "kernel_us_per_push": ms * 1e3 / pushes, "GBps": 2 * frames / (ms * 1e-3) / 1e9 if ms else None}


def loopback_config4(S: int, retain: str = "bits"):
    """BASELINE config 4 on S channels: 64 KB random payloads at 300 baud (146.8 M frames each) from a streaming
    transmitter, pulled into a device tensor and pushed in 1 s pieces into a bits-mode receiver; start frames spread
    over chunk phases.  Wall time, decoded messages, peak arena_bytes()"""
    import torch
    rng = np.random.default_rng(8400)
    pays = [rng.integers(0, 256, 65536, dtype=np.uint8).tobytes() for _ in range(S)]
    ok, peak = 0, 0
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    with A.open_transmit_streams([A.Transmitter(300, 0.1)] * S) as tx, A.Receiver(300).open_streams(S, 10.0, retain=retain) as st:
        buf = torch.empty(S * 48000, dtype=torch.int16, device="cuda")
        ends, pushed = 0, 0
        for g in range(8):
            ids = list(range(g, S, 8))
            _, e = tx.send(ids, [pays[s] for s in ids])
            ends = max(ends, int(e.max()))
            st.push(tx.pull(257, out=buf), np.arange(S + 1, dtype=np.int64) * 257)
            pushed += 257
        total = ends + 4096
        evs = []
        while pushed < total:
            n = min(48000, total - pushed)
            ev = st.push(tx.pull(n, out=buf), np.arange(S + 1, dtype=np.int64) * n)
            if len(ev):
                evs.append(ev)
            pushed += n
            peak = max(peak, st.arena_bytes())
        evs.append(st.finish())
        for ev in evs:
            b = ev.batch
            k = 0
            for i in np.flatnonzero(ev.recorded):
                ok += int(b.status[k] == 0 and b.nbits[k] == 917504 and b.payload(k) == pays[int(ev.stream[i])])
                k += 1
        torch.cuda.synchronize()
    return {"S": S, "retain": retain, "frames_per_channel": total, "wall_s": time.perf_counter() - t0, "decoded_ok": ok,
            "peak_arena_bytes": peak}


def profile_config(d_base, S: int, piece: int, T: int, timeout: float, out_dir: str | None, route: str = "planar"):
    """Device time of every kernel and copy over one device-input push sequence (torch.profiler, CUDA activity),
    beside the host wall time of the same pushes: what share of a push the GPU is busy.  route interleaved: the
    same pieces frame-major, through push_interleaved."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    n_push = T // piece
    offsets = np.arange(S + 1, dtype=np.int64) * piece
    pieces = [torch.as_strided(d_base, (S, piece), (SHIFT, 1), i * piece).contiguous().view(-1) for i in range(n_push)]
    if route == "interleaved":
        pieces = [t.view(S, piece).t().contiguous() for t in pieces]

    def push(st, t):
        return st.push_interleaved(t) if route == "interleaved" else st.push(t, offsets)
    rx = A.Receiver(1200)
    with rx.open_streams(S, timeout) as st:
        for t in pieces:                                  # warm-up: same shapes
            push(st, t)
        st.finish()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            t0 = time.perf_counter()
            for t in pieces:
                push(st, t)
            wall = time.perf_counter() - t0
        st.finish()
    rows = {}
    for e in prof.key_averages():
        us = getattr(e, "device_time_total", None)
        if us is None:
            us = getattr(e, "cuda_time_total", 0.0)
        if us > 0:
            rows[e.key] = {"count": int(e.count), "ms": us / 1e3}
    busy = sum(r["ms"] for r in rows.values())
    if out_dir:
        prof.export_chrome_trace(os.path.join(out_dir, f"stream_profile_{route}.pt.trace.json"))
    # the append: k_stream_deinterleave, or k_stream_copy's launches (its retention moves included, which the
    # interleaved run also counts under k_stream_copy); 4 bytes per appended frame
    kernel = "k_stream_deinterleave" if route == "interleaved" else "k_stream_copy"
    app_ms = sum(r["ms"] for k, r in rows.items() if kernel in k)
    app_bytes = 4 * S * piece * n_push
    return {"S": S, "piece": piece, "pushes": n_push, "input": "device", "route": route, "host_wall_ms": wall * 1e3,
            "host_ms_per_push": wall * 1e3 / n_push, "append_kernel": kernel, "append_ms": app_ms,
            "append_us_per_push": app_ms * 1e3 / n_push,
            "append_TBps": app_bytes / (app_ms * 1e-3) / 1e12 if app_ms else None,
            "device_busy_ms": busy, "device_busy_share": busy / (wall * 1e3),
            "by_kernel_or_copy": dict(sorted(rows.items(), key=lambda kv: -kv[1]["ms"]))}


FORMATS = {"s16": np.int16, "s32": np.int32, "f32": np.float32}


def run_frames(d_base, S: int, piece: int, T: int, device: bool, fmt: str, extra: int, timeout: float, reps: int = 3):
    """--format: the pieces as a window of an (n, S + extra) card of fmt; route "window" (push_interleaved of the
    window) and "replaced" (contiguous copy, conversion, push_interleaved of int16), alternately on two receivers"""
    import torch
    dt = FORMATS[fmt]
    c0 = 1 if extra else 0
    n_push = max(T // piece, 1)
    cards = []
    for i in range(n_push):
        x = torch.as_strided(d_base, (S, piece), (SHIFT, 1), i * piece).t()
        y = x if dt == np.int16 else x.to(torch.int32) << 16 if dt == np.int32 else x.to(torch.float32) / 32768
        c = torch.zeros((piece, S + extra), dtype=y.dtype, device="cuda")
        c[:, c0:c0 + S] = y
        cards.append(c if device else c.cpu().numpy())
    torch.cuda.synchronize()

    def window(st, c):
        return st.push_interleaved(c[:, c0:c0 + S], dtype=dt)

    def replaced(st, c):
        w = c[:, c0:c0 + S]
        if device:
            w = w.contiguous()
            w = w if dt == np.int16 else (w >> 16).to(torch.int16) if dt == np.int32 else \
                torch.clamp(torch.round(torch.nan_to_num(w, nan=0.0) * 32768), -32768, 32767).to(torch.int16)
        else:
            w = np.ascontiguousarray(w)
            w = w if dt == np.int16 else (w >> 16).astype(np.int16) if dt == np.int32 else \
                np.clip(np.rint(np.nan_to_num(w, nan=0.0).astype(np.float64) * 32768), -32768, 32767).astype(np.int16)
        return st.push_interleaved(w)
    routes = {"window": window, "replaced": replaced}
    times = {r: [] for r in routes}
    rx = A.Receiver(1200)
    events = {}
    with rx.open_streams(S, timeout) as a, rx.open_streams(S, timeout) as b:
        hs = {"window": a, "replaced": b}
        for rep in range(reps + 1):                       # rep 0 warms up every shape
            for r, fn in routes.items():
                n_ev = 0
                for c in cards:
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    n_ev += len(fn(hs[r], c))
                    if rep:
                        times[r].append(time.perf_counter() - t0)
                events[r] = n_ev
    out = []
    for r in routes:
        t = np.array(times[r])
        out.append({"S": S, "piece": piece, "input": "device" if device else "host", "format": fmt, "pitch_extra": extra,
                    "route": r, "pushes": len(t), "push_ms_median": float(np.median(t) * 1e3),
                    "push_ms_min": float(t.min() * 1e3), "push_ms_max": float(t.max() * 1e3),
                    "frames_per_s": S * piece * len(t) / float(t.sum()), "events_last_rep": events[r]})
    return out


def profile_frames(d_base, S: int, piece: int, T: int, fmt: str, extra: int, timeout: float):
    """the append kernel's device time over device-window pushes in one format (torch.profiler)"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    dt = FORMATS[fmt]
    c0 = 1 if extra else 0
    n_push = max(T // piece, 1)
    cards = []
    for i in range(n_push):
        x = torch.as_strided(d_base, (S, piece), (SHIFT, 1), i * piece).t()
        y = x if dt == np.int16 else x.to(torch.int32) << 16 if dt == np.int32 else x.to(torch.float32) / 32768
        c = torch.zeros((piece, S + extra), dtype=y.dtype, device="cuda")
        c[:, c0:c0 + S] = y
        cards.append(c)
    with A.Receiver(1200).open_streams(S, timeout) as st:
        for c in cards:
            st.push_interleaved(c[:, c0:c0 + S], dtype=dt)
        st.finish()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for c in cards:
                st.push_interleaved(c[:, c0:c0 + S], dtype=dt)
    ms = 0.0
    for e in prof.key_averages():
        if "k_stream_frames" in e.key or "k_stream_deinterleave" in e.key:
            us = getattr(e, "device_time_total", None)
            ms += (us if us is not None else getattr(e, "cuda_time_total", 0.0)) / 1e3
    nbytes = S * piece * n_push * (np.dtype(dt).itemsize + 2)
    kernel = "k_stream_deinterleave" if dt == np.int16 and not extra else "k_stream_frames"
    return {"S": S, "piece": piece, "pushes": n_push, "format": fmt, "pitch_extra": extra, "kernel": kernel,
            "kernel_ms": ms, "kernel_us_per_push": ms * 1e3 / n_push, "bytes_read_and_written": nbytes,
            "kernel_TBps": nbytes / (ms * 1e-3) / 1e12 if ms else None}


def whole_stream_reference(base: np.ndarray, T: int, n_streams: int, timeout: float):
    rx = A.Receiver(1200)
    streams = [base[s * SHIFT:s * SHIFT + T] for s in range(n_streams)]
    rx.receive_all(streams[0], timeout, False, keep_timeouts=True)               # warm-up
    t0 = time.perf_counter()
    for x in streams:
        rx.receive_all(x, timeout, False, keep_timeouts=True)
    t_all = time.perf_counter() - t0
    t0 = time.perf_counter()
    for x in streams:
        rx.listen_gate_multi(x, timeout)
    t_gate = time.perf_counter() - t0
    frames = n_streams * T
    return {"streams": n_streams, "frames": frames, "receive_all_frames_per_s": frames / t_all,
            "receive_all_ms_per_stream": t_all / n_streams * 1e3, "listen_gate_multi_frames_per_s": frames / t_gate,
            "listen_gate_multi_ms_per_stream": t_gate / n_streams * 1e3}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--S", default="1,64,4096")
    ap.add_argument("--piece", default="2048,48000")
    ap.add_argument("--seconds", type=float, default=8.0)
    ap.add_argument("--timeout", type=float, default=1.0)
    ap.add_argument("--input", default="host,device")
    ap.add_argument("--mix", action="store_true", help="six bauds and three threshold pairs across the channels")
    ap.add_argument("--layout", default="planar", choices=["planar", "interleaved"])
    ap.add_argument("--stuck", type=int, default=0, help="seconds of stuck-carrier traffic per retention mode")
    ap.add_argument("--stuck-S", type=int, default=256, help="channels of the stuck-carrier run")
    ap.add_argument("--windows-bauds", default="", help="bauds at which to profile k_stream_windows alone (bits mode)")
    ap.add_argument("--stuck-variants", default="message", help="stuck-carrier variants: message,tone,gap")
    ap.add_argument("--loopback", type=int, default=0, help="channels of a config-4 loopback (0: none)")
    ap.add_argument("--loopback-retain", default="bits", help="retention mode of the config-4 loopback")
    ap.add_argument("--retain", default="samples", help="retention modes, run in turn per configuration: samples,bits,payload")
    ap.add_argument("--format", default="", help="sample formats of a window of a wider card: s16,s32,f32")
    ap.add_argument("--pitch-extra", type=int, default=0, help="columns of the card beyond the S of the window")
    ap.add_argument("--out", default=None)
    ap.add_argument("--no-profile", action="store_true", help="skip the profiled run of the largest device configuration")
    a = ap.parse_args()
    import torch
    _cabi.require_device(0)
    A.LOG_LEVEL = 5
    Ss = [int(v) for v in a.S.split(",")]
    pieces = [int(v) for v in a.piece.split(",")]
    T = int(a.seconds * 48000)
    rng = np.random.default_rng(0)
    n = max(Ss) * SHIFT + T + max(pieces)
    if a.mix:
        bases = [traffic(n, rng, b) for b in MIX_BAUDS]
        d_bases = [torch.from_numpy(x).cuda() for x in bases]
    else:
        base = traffic(n, rng)
        d_base = torch.from_numpy(base).cuda()
    res = {"card": card(), "torch_device": torch.cuda.get_device_name(0), "seconds_per_channel": a.seconds,
           "timeout_s": a.timeout, "mix": a.mix, "layout": a.layout, "retain": a.retain, "configs": []}
    modes = a.retain.split(",")
    fmts = [f for f in a.format.split(",") if f]
    if fmts:                                              # the format measurements alone
        res.update({"pitch_extra": a.pitch_extra, "configs": [], "profile_formats": []})
        for S in Ss:
            for piece in pieces:
                for inp in a.input.split(","):
                    for f in fmts:
                        for r in run_frames(d_base, S, piece, T, inp == "device", f, a.pitch_extra, a.timeout):
                            print(json.dumps(r), flush=True)
                            res["configs"].append(r)
        if not a.no_profile:
            for f in fmts:
                r = profile_frames(d_base, max(Ss), max(pieces), T, f, a.pitch_extra, a.timeout)
                print(json.dumps(r), flush=True)
                res["profile_formats"].append(r)
        res["card_after"] = card()
        if a.out:
            os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
            json.dump(res, open(a.out, "w"), indent=1)
        return
    routes = {False: ["planar"], True: ["planar"]}
    if a.layout == "interleaved":
        routes = {False: ["interleaved", "host-transpose"], True: ["interleaved", "device-transpose"]}
    for S in Ss:
        for piece in pieces:
            for inp in a.input.split(","):
                for route in routes[inp == "device"]:
                    for mode in modes:
                        r = run_config(bases, d_bases, S, piece, T, inp == "device", a.timeout, True, route, mode) if a.mix else \
                            run_config(base, d_base, S, piece, T, inp == "device", a.timeout, route=route, retain=mode)
                        print(json.dumps(r), flush=True)
                        res["configs"].append(r)
    if not a.mix and not a.no_profile:                    # the profile and whole-stream lines use uniform traffic
        out_dir = os.path.dirname(os.path.abspath(a.out)) if a.out else None
        res["profile"] = profile_config(d_base, max(Ss), max(pieces), T, a.timeout, out_dir)
        print(json.dumps({k: v for k, v in res["profile"].items() if k != "by_kernel_or_copy"}), flush=True)
        if a.layout == "interleaved":
            res["profile_interleaved"] = profile_config(d_base, max(Ss), max(pieces), T, a.timeout, out_dir, "interleaved")
            print(json.dumps({k: v for k, v in res["profile_interleaved"].items() if k != "by_kernel_or_copy"}), flush=True)
    if a.stuck:
        res["stuck_carrier"] = [stuck_carrier(a.stuck_S, a.stuck, m, v) for v in a.stuck_variants.split(",") for m in modes]
        for r in res["stuck_carrier"]:
            print(json.dumps({"retain": r["retain"], "variant": r["variant"], "ended_channels": r["ended_channels"],
                              "last": r["seconds_vs_arena_bytes"][-1]}), flush=True)
    if a.windows_bauds:
        res["windows_by_baud"] = [profile_windows(int(b), max(Ss), 4) for b in a.windows_bauds.split(",")]
        for r in res["windows_by_baud"]:
            print(json.dumps(r), flush=True)
    if a.loopback:
        res["loopback_config4"] = loopback_config4(a.loopback, a.loopback_retain)
        print(json.dumps(res["loopback_config4"]), flush=True)
    if not a.mix and "bits" in modes:
        res["profile_bits"] = profile_bits(d_base, max(Ss), max(pieces), T, a.timeout)
        print(json.dumps(res["profile_bits"]), flush=True)
    if not a.mix:
        res["whole_stream"] = whole_stream_reference(base, T, 16, a.timeout)
        print(json.dumps(res["whole_stream"]), flush=True)
    res["card_after"] = card()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        json.dump(res, open(a.out, "w"), indent=1)


if __name__ == "__main__":
    main()
