"""Streaming transmitter throughput: S channels of 1200-baud messages separated by silence, pulled window by window
through Transmitter.open_streams into a CUDA tensor or a host (pinned) array.

    python tools/stream_tx_bench.py [--S 1,64,4096] [--pull 2048,48000] [--seconds 8] [--mix] [--out FILE]

Every channel sends a 10-60 byte message (0.1 s training) whenever its previous one has ended and a random gap of
up to twice a message's mean length has passed, so a channel is busy about half the time; the sends due inside a
window go in one send() call before its pull.  Each configuration runs its sequence twice on one transmitter and
times the second: host wall time of every pull (it ends in a synchronize) and of every send.  A separate
torch.profiler run of the largest device-output configuration gives k_tx_window's kernel time (bytes written per
second of kernel time, against the 7.7 TB/s of HBM3e on a B200's data sheet) and the share of a pull the GPU is busy.
Card name and power limit are read in the same run.

--mix splits the channels into six equal groups at 300, 600, 1200, 2400, 4000 and 6000 baud (open_transmit_streams),
each sending messages of its own length at the same duty.

--layout interleaved measures the window as a multi-channel sound card takes it, n x S frame-major, three ways in one
run: pull_interleaved (the GPU writes it interleaved), a planar pull followed by a host numpy transpose into a
preallocated array (host output), and a planar pull into a CUDA tensor followed by .t().contiguous() (device output),
which is what a user had to do without pull_interleaved.  The profiled run then times k_tx_window_interleaved and
k_tx_window over the same sequence (2 bytes written per pulled frame).

--format s16,s32,f32 measures, per format, the window written into columns of a wider playback buffer (--pitch-extra K:
the card has S + K columns and the window starts at column 1 when K > 0, an odd column): pull_interleaved(n,
out=card[:, c0:c0 + S], dtype=...) beside the route it replaces, pull_interleaved(n) of int16 frames, the conversion
(s << 16, s / 32768) and the copy into the card's columns, with numpy on the host or torch on the device.  The
profiled run then times k_tx_window_frames in each format (k_tx_window_interleaved for contiguous int16), its bytes/s
counted over the bytes it writes (n * S * sample size)."""
from __future__ import annotations

import argparse
import json
import os
import re
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import afskmodem_b200 as A  # noqa: E402
from afskmodem_b200 import _cabi  # noqa: E402

HBM_TBS = 7.7
MIX_BAUDS = [300, 600, 1200, 2400, 4000, 6000]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


class Traffic:
    """per channel: the next frame at which it sends, and a pool of payloads"""

    def __init__(self, S: int, baud, seed: int):
        """baud: one for every channel, or an array of S (mean message length per channel)"""
        self.rng = np.random.default_rng(seed)
        self.S = S
        self.msgs = [self.rng.integers(0, 256, size=int(self.rng.integers(10, 61)), dtype=np.uint8).tobytes() for _ in range(256)]
        bf = 48000 // baud
        self.mean_len = (baud // 10) * bf + 5 * bf + 4800 + 35 * 14 * bf
        self.next_at = self.rng.integers(0, 2 * self.mean_len, S).astype(np.int64)

    def due(self, P: int, n: int):
        s = np.nonzero(self.next_at < P + n)[0]
        return s.astype(np.int32), [self.msgs[i] for i in self.rng.integers(0, len(self.msgs), len(s))]

    def sent(self, streams, end):
        hi = 2 * (self.mean_len if np.ndim(self.mean_len) == 0 else self.mean_len[streams])
        self.next_at[streams] = end + self.rng.integers(0, hi, len(streams))


FORMATS = {"s16": np.int16, "s32": np.int32, "f32": np.float32}


def convert_host(x, dt):
    """the transmit rule of afsk_b200.h, with numpy"""
    return x if dt == np.int16 else (x.astype(np.int32) << 16) if dt == np.int32 else x.astype(np.float32) / np.float32(32768)


def frames_route(st, S, n, route, fmt, extra, device):
    """--format: the window of an (n, S + extra) card of format fmt, written by pull_interleaved ("window") or by the
    route it replaces ("replaced": an int16 pull, the conversion, the copy into the card's columns)"""
    import torch
    dt = FORMATS[fmt]
    c0 = 1 if extra else 0
    if device:
        cardt = torch.zeros((n, S + extra), dtype=getattr(torch, np.dtype(dt).name), device="cuda")
        tmp = torch.empty((n, S), dtype=torch.int16, device="cuda")
        if route == "window":
            return lambda: st.pull_interleaved(n, out=cardt[:, c0:c0 + S], dtype=dt)

        def dev():
            x = st.pull_interleaved(n, out=tmp)
            y = x if dt == np.int16 else x.to(torch.int32) << 16 if dt == np.int32 else x.to(torch.float32) / 32768
            cardt[:, c0:c0 + S].copy_(y)
            torch.cuda.synchronize()
        return dev
    cardh = np.zeros((n, S + extra), dt)
    if route == "window":
        return lambda: st.pull_interleaved(n, out=cardh[:, c0:c0 + S], dtype=dt)

    def host():
        cardh[:, c0:c0 + S] = convert_host(st.pull_interleaved(n), dt)
    return host


def pull_route(st, S, n, route, out_t):
    """the pull of one window by route: planar, interleaved, or the planar pull transposed on the host / device"""
    import torch
    if route == "planar":
        return lambda: st.pull(n, out=out_t)
    if route == "interleaved":
        return lambda: st.pull_interleaved(n, out=out_t)
    if route == "host-transpose":
        dst = np.empty((n, S), np.int16)
        return lambda: np.copyto(dst, st.pull(n).T)

    def dev():                                            # device-transpose
        st.pull(n, out=out_t)[:S * n].view(S, n).t().contiguous()
        torch.cuda.synchronize()
    return dev


def run_sequence(st, S, n, n_pull, baud, seed, out_t=None, pull=None):
    tr = Traffic(S, baud, seed)
    t_pull, t_send, busy = [], [], 0
    P = st.state(0)[0]                      # the timeline goes on from the previous sequence
    tr.next_at += P
    for _ in range(n_pull):
        streams, pays = tr.due(P, n)
        t0 = time.perf_counter()
        if len(streams):
            a, b = st.send(streams, pays)
            tr.sent(streams, b)
            busy += int((b - a).sum())
        t1 = time.perf_counter()
        if pull:
            pull()
        else:
            st.pull(n, out=out_t)
        t2 = time.perf_counter()
        t_send.append(t1 - t0)
        t_pull.append(t2 - t1)
        P += n
    return np.array(t_pull), np.array(t_send), busy


def mix_bauds(S: int) -> np.ndarray:
    """--mix: channel s's baud (six equal groups)"""
    return np.array([MIX_BAUDS[s * len(MIX_BAUDS) // S] for s in range(S)], np.int64)


def run_config(S: int, n: int, T: int, device: bool, baud, route: str = "planar", fmt: str | None = None, extra: int = 0):
    """baud: one for every channel, or "mix" (mix_bauds); route: see pull_route, or with fmt frames_route"""
    import torch
    n_pull = max(T // n, 1)
    out_t = torch.empty(S * n, dtype=torch.int16, device="cuda") if device else None
    res = {"S": S, "pull": n, "baud": baud, "output": "device" if device else "host-pinned", "pulls": n_pull, "route": route}
    if fmt:
        res.update({"format": fmt, "pitch_extra": extra, "output": "device" if device else "host"})
    if baud == "mix":
        baud = mix_bauds(S)
        st = A.open_transmit_streams([A.Transmitter(int(b), 0.1) for b in baud])
    else:
        st = A.Transmitter(baud, 0.1).open_streams(S)
    with st:
        pull = frames_route(st, S, n, route, fmt, extra, device) if fmt else pull_route(st, S, n, route, out_t)
        run_sequence(st, S, n, n_pull, baud, 1, out_t, pull)          # warm-up: same shapes
        c0 = st.counters()
        tp, ts, busy = run_sequence(st, S, n, n_pull, baud, 2, out_t, pull)
        c1 = st.counters()
        arena = st.arena_bytes()
    frames = S * n * n_pull
    res.update({
        "frames": frames, "pull_seconds": float(tp.sum()), "send_seconds": float(ts.sum()),
        "frames_per_s": frames / float(tp.sum()), "frames_per_s_with_send": frames / float(tp.sum() + ts.sum()),
        "pull_ms_median": float(np.median(tp) * 1e3), "pull_ms_p90": float(np.percentile(tp, 90) * 1e3),
        "send_ms_median": float(np.median(ts) * 1e3), "busy_fraction": busy / frames,
        "launches_per_pull": (c1["launches"] - c0["launches"]) / n_pull,
        "moved_bytes": c1["moved_bytes"] - c0["moved_bytes"], "compactions": c1["compactions"] - c0["compactions"],
        "arena_bytes": arena,
    })
    return res


def profile_config(S: int, n: int, T: int, baud: int, out_dir: str | None, route: str = "planar", fmt: str | None = None,
                   extra: int = 0):
    """Device time of every kernel and copy over one device-output pull sequence (torch.profiler, CUDA activity),
    beside the host wall time of the same pulls."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    n_pull = max(T // n, 1)
    out_t = torch.empty(S * n, dtype=torch.int16, device="cuda")
    tx = A.Transmitter(baud, 0.1)
    with tx.open_streams(S) as st:
        pull = frames_route(st, S, n, route, fmt, extra, True) if fmt else pull_route(st, S, n, route, out_t)
        run_sequence(st, S, n, n_pull, baud, 1, out_t, pull)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            t0 = time.perf_counter()
            tp, ts, _ = run_sequence(st, S, n, n_pull, baud, 2, out_t, pull)
            wall = time.perf_counter() - t0
    rows = {}
    for e in prof.key_averages():
        us = getattr(e, "device_time_total", None)
        if us is None:
            us = getattr(e, "cuda_time_total", 0.0)
        if us > 0:
            rows[e.key] = {"count": int(e.count), "ms": us / 1e3}
    busy = sum(r["ms"] for r in rows.values())
    kernel = "k_tx_window_interleaved" if route == "interleaved" or (route == "window" and fmt == "s16" and not extra) else \
        "k_tx_window_frames" if route == "window" else "k_tx_window"
    win = [v for k, v in rows.items() if re.search(kernel + r"\b(?!_)", k)]
    win_ms = sum(r["ms"] for r in win)
    win_bytes = (np.dtype(FORMATS[fmt]).itemsize if fmt else 2) * S * n * n_pull
    if out_dir:
        prof.export_chrome_trace(os.path.join(out_dir, f"stream_tx_profile_{route}.pt.trace.json"))
    return {"S": S, "pull": n, "baud": baud, "pulls": n_pull, "output": "device", "route": route, "kernel": kernel,
            "format": fmt, "pitch_extra": extra,
            "host_wall_ms": wall * 1e3,
            "host_ms_per_pull": wall * 1e3 / n_pull, "pull_ms_per_pull": float(tp.sum()) * 1e3 / n_pull,
            "send_ms_per_pull": float(ts.sum()) * 1e3 / n_pull,
            "device_busy_ms": busy, "device_busy_ms_per_pull": busy / n_pull, "device_busy_share": busy / (wall * 1e3),
            "k_tx_window_ms": win_ms, "k_tx_window_us_per_pull": win_ms * 1e3 / n_pull,
            "k_tx_window_bytes_written": win_bytes,
            "k_tx_window_TBps": win_bytes / (win_ms * 1e-3) / 1e12 if win_ms else None,
            "k_tx_window_share_of_hbm_peak": (win_bytes / (win_ms * 1e-3) / 1e12) / HBM_TBS if win_ms else None,
            "by_kernel_or_copy": dict(sorted(rows.items(), key=lambda kv: -kv[1]["ms"]))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--S", default="1,64,4096")
    ap.add_argument("--pull", default="2048,48000")
    ap.add_argument("--seconds", type=float, default=8.0)
    ap.add_argument("--output", default="device,host")
    ap.add_argument("--mix", action="store_true", help="six bauds across the channels")
    ap.add_argument("--layout", default="planar", choices=["planar", "interleaved"])
    ap.add_argument("--format", default="", help="sample formats of a window of a wider card: s16,s32,f32")
    ap.add_argument("--pitch-extra", type=int, default=0, help="columns of the card beyond the S of the window")
    ap.add_argument("--out", default=None)
    ap.add_argument("--no-profile", action="store_true", help="skip the profiled run of the largest device configuration")
    a = ap.parse_args()
    import torch
    _cabi.require_device(0)
    A.LOG_LEVEL = 5
    Ss = [int(v) for v in a.S.split(",")]
    pulls = [int(v) for v in a.pull.split(",")]
    T = int(a.seconds * 48000)
    res = {"card": card(), "torch_device": torch.cuda.get_device_name(0), "seconds_per_channel": a.seconds, "mix": a.mix,
           "configs": []}
    res["layout"] = a.layout
    routes = {False: ["planar"], True: ["planar"]}
    if a.layout == "interleaved":
        routes = {False: ["interleaved", "host-transpose"], True: ["interleaved", "device-transpose"]}
    lines = [(S, n, o == "device", "mix" if a.mix else 1200, r) for S in Ss for n in pulls for o in a.output.split(",")
             for r in routes[o == "device"]]
    if not a.mix:
        lines += [(max(Ss), max(pulls), True, 4800, r) for r in routes[True]]
    fmts = [f for f in a.format.split(",") if f]
    if fmts:
        res["pitch_extra"] = a.pitch_extra
        for S in Ss:
            for n in pulls:
                for o in a.output.split(","):
                    for f in fmts:
                        for route in ("window", "replaced"):
                            r = run_config(S, n, T, o == "device", 1200, route, f, a.pitch_extra)
                            print(json.dumps(r), flush=True)
                            res["configs"].append(r)
        if not a.no_profile:
            res["profile_formats"] = [profile_config(max(Ss), max(pulls), T, 1200, None, "window", f, a.pitch_extra) for f in fmts]
            for r in res["profile_formats"]:
                print(json.dumps({k: v for k, v in r.items() if k != "by_kernel_or_copy"}), flush=True)
        lines = []
    for S, n, dev, baud, route in lines:
        r = run_config(S, n, T, dev, baud, route)
        print(json.dumps(r), flush=True)
        res["configs"].append(r)
    if not a.mix and not a.no_profile and not fmts:
        out_dir = os.path.dirname(os.path.abspath(a.out)) if a.out else None
        res["profile"] = profile_config(max(Ss), max(pulls), T, 1200, out_dir)
        print(json.dumps({k: v for k, v in res["profile"].items() if k != "by_kernel_or_copy"}), flush=True)
        if a.layout == "interleaved":
            res["profile_interleaved"] = profile_config(max(Ss), max(pulls), T, 1200, out_dir, "interleaved")
            print(json.dumps({k: v for k, v in res["profile_interleaved"].items() if k != "by_kernel_or_copy"}), flush=True)
    res["card_after"] = card()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        json.dump(res, open(a.out, "w"), indent=1)


if __name__ == "__main__":
    main()
