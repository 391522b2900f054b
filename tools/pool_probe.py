#!/usr/bin/env python
"""The encoder session pool (Context.encoder_pool, sea_b200_encoder_pool_push) in the shape of a live server: S sessions each
send a 20 ms packet (960 frames at 48 kHz) per round, and one push per round encodes every chunk that completed.  Prints a table
and one JSON line:

  python tools/pool_probe.py [--rounds R] [--warmup W] [--sessions 256,1024,4096,16384]

Rows: stereo CBR-3 and stereo VBR-3 at every S, and one 8-channel CBR-4 row at S = 1024; frames_per_chunk 5120.  Sessions start
at staggered phases (session s first sends s * 5120 / S frames), so in steady state about 1 / 5.33 of them complete a chunk per
round.  Audio: synthetic tone + noise (sea_codec_b200/synth.py), 32 distinct sources cut into 960-frame rows, session s reading
source s mod 32 from its own row offset.  Packets are gathered into a pinned buffer and outputs land in a pinned buffer packed by
push_bound, as a server would lay them out; only the push itself is timed.

Per row: wall ms per push (host clock around the call, which ends in a device synchronise; mean and p99 over the timed rounds),
real-time headroom = 20 ms / mean wall ms, and in a separate traced run the kernel ms per stage (CUDA events, the library's
SEA_B200_TRACE lines: ingest, encode, commit).  At S = 256 and 1024 the same traffic also goes through one sea_b200_encoder handle
per session (make_chunks whenever a session holds a full chunk): ms per round, and whether every session's bytes equal the pool's.
The card's name and power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import re
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

RATE, N, PKT, SOURCES, SPREAD = 48000, 5120, 960, 32, 64
PRIME = (N + PKT - 1) // PKT  # rows a priming packet can span


def start_rows(n_sessions):
    """Row of its source at which session s starts (sessions of one source start at different rows)."""
    return (np.arange(n_sessions) * 7) % SPREAD


def phases(n_sessions):
    """Frames of session s's first (priming) packet: the sessions' chunk boundaries spread evenly over the rounds."""
    return (np.arange(n_sessions, dtype=np.int64) * N) // n_sessions


def packets(sources, n_sessions, r):
    """(frames per session, interleaved packets [n, width]) of round r; round 0 sends the priming packets (up to PRIME rows)."""
    k, r0 = np.arange(n_sessions) % SOURCES, start_rows(n_sessions)
    if r == 0:
        rows = sources[k[:, None], r0[:, None] + np.arange(PRIME)].reshape(n_sessions, -1)
        return phases(n_sessions), rows
    return np.full(n_sessions, PKT, np.int64), sources[k, r0 + PRIME - 1 + r]


TRACE = re.compile(r"pool push: .* ingest ([0-9.]+) ms, encode ([0-9.]+) ms, commit ([0-9.]+) ms")


def card():
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(", ")
        return {"gpu": q[0], "power_limit_w": float(q[1])}
    except Exception as e:
        import torch

        return {"gpu": torch.cuda.get_device_name(0), "power_limit_w": None, "nvidia_smi": str(e)}


def pinned(S, n, dtype):
    p = S.lib().sea_b200_host_alloc(max(1, n * np.dtype(dtype).itemsize))
    if not p:
        raise MemoryError("sea_b200_host_alloc")
    return p, np.ctypeslib.as_array((C.c_uint8 * (n * np.dtype(dtype).itemsize)).from_address(p)).view(dtype)


class Server:
    """S sessions, one pool; round(r) pushes every session's r-th packet (round 0: the staggered priming packets)."""

    def __init__(self, S, ctx, n_sessions, channels, settings, sources):
        self.S, self.ctx, self.n, self.C, self.st = S, ctx, n_sessions, channels, settings
        self.pool = ctx.encoder_pool(channels, RATE, settings, n_sessions)
        self.pool.open(range(n_sessions))
        self.full = self.pool._full
        self.src = sources  # [SOURCES, rows, PKT * C] int16
        self.buffered = np.zeros(n_sessions, np.int64)
        self.sessions = np.arange(n_sessions, dtype=np.uint32)
        self.in_ptr, self.inp = pinned(S, n_sessions * PRIME * PKT * channels, np.int16)
        self.out_cap = n_sessions * self.full + 64
        self.out_ptr, self.outp = pinned(S, self.out_cap, np.uint8)

    def push(self, r):
        frames, rows = packets(self.src, self.n, r)
        self.inp[: rows.size] = rows.reshape(-1)
        pcm_off = np.arange(self.n, dtype=np.uint64) * np.uint64(rows.shape[1])
        tot = self.buffered + frames
        caps = (tot // N * self.full).astype(np.uint64)
        out_off = np.zeros(self.n, np.uint64)
        out_off[1:] = np.cumsum(caps)[:-1]
        t0 = time.perf_counter()
        lens = self.pool.push_host(self.sessions, self.in_ptr, pcm_off, frames.astype(np.uint32), self.out_ptr, out_off, out_caps=caps)
        dt = time.perf_counter() - t0
        self.buffered = tot % N
        return dt, frames, rows, lens, out_off

    def close(self):
        self.pool.close()
        L = self.ctx._L
        L.sea_b200_host_free(C.c_void_p(self.in_ptr))
        L.sea_b200_host_free(C.c_void_p(self.out_ptr))


def traced(fn):
    """fn() with SEA_B200_TRACE set and fd 2 captured; returns the summed (ingest, encode, commit) ms and the push count."""
    os.environ["SEA_B200_TRACE"] = "1"
    sys.stderr.flush()
    saved = os.dup(2)
    with tempfile.TemporaryFile(mode="w+") as tmp:
        os.dup2(tmp.fileno(), 2)
        try:
            fn()
        finally:
            os.dup2(saved, 2)
            os.close(saved)
            os.environ.pop("SEA_B200_TRACE", None)
        tmp.seek(0)
        text = tmp.read()
    acc, n = np.zeros(3), 0
    for m in TRACE.finditer(text):
        acc += [float(m.group(k)) for k in (1, 2, 3)]
        n += 1
    return acc, n


def handles_run(S, ctx, n_sessions, channels, settings, rounds, sources, pool_bytes):
    """The same traffic through one streaming handle per session: make_chunks whenever a session holds a full chunk."""
    L = ctx._L
    st = settings._c()
    hs = []
    for _ in range(n_sessions):
        h = C.c_void_p()
        ctx._check(L.sea_b200_encoder_create(ctx._h, channels, RATE, C.byref(st), C.byref(h)))
        hs.append(h)
    held = [np.zeros(0, np.int16) for _ in range(n_sessions)]
    out = [bytearray() for _ in range(n_sessions)]
    buf = np.empty(70000 * 2, np.uint8)
    times = []
    try:
        for r in range(rounds):
            frames, rows = packets(sources, n_sessions, r)
            t_round = 0.0
            for s in range(n_sessions):
                held[s] = np.concatenate([held[s], rows[s, : frames[s] * channels]])
                k = held[s].size // (N * channels)
                if k:
                    x = np.ascontiguousarray(held[s][: k * N * channels])
                    ln, nck = C.c_uint64(0), C.c_uint32(0)
                    t0 = time.perf_counter()
                    ctx._check(L.sea_b200_encoder_make_chunks(hs[s], x.ctypes.data, x.size, buf.ctypes.data, buf.size, C.byref(ln), C.byref(nck)))
                    t_round += time.perf_counter() - t0
                    out[s] += buf[: ln.value].tobytes()
                    held[s] = held[s][k * N * channels:]
            times.append(t_round)
    finally:
        for h in hs:
            L.sea_b200_encoder_destroy(h)
    same = all(bytes(out[s]) == pool_bytes[s] for s in range(n_sessions))
    return times, same


def row(S, ctx, name, channels, settings, n_sessions, rounds, warmup, sources, with_handles):
    srv = Server(S, ctx, n_sessions, channels, settings, sources)
    keep = with_handles
    got = [bytearray() for _ in range(n_sessions)] if keep else None

    def one(r):
        dt, frames, rows, lens, out_off = srv.push(r)
        if keep:
            for s in np.flatnonzero(lens):
                got[s] += srv.outp[int(out_off[s]): int(out_off[s]) + int(lens[s])].tobytes()
        return dt, int(np.count_nonzero(lens))

    r = 0
    for _ in range(warmup):
        one(r)
        r += 1
    walls, enc = [], []
    for _ in range(rounds):
        dt, k = one(r)
        walls.append(dt)
        enc.append(k)
        r += 1
    state = {"r": r}

    def traced_rounds():
        for _ in range(60 if rounds >= 60 else rounds):
            one(state["r"])
            state["r"] += 1

    stages, n_traced = traced(traced_rounds)
    total_rounds = state["r"]
    srv.close()
    w = np.array(walls) * 1e3
    res = {"row": name, "sessions": n_sessions, "channels": channels, "wall_ms_mean": round(float(w.mean()), 4),
           "wall_ms_p99": round(float(np.percentile(w, 99)), 4), "headroom_x": round(20.0 / float(w.mean()), 2),
           "encoding_sessions_per_push": round(float(np.mean(enc)), 1)}
    if n_traced:
        res.update({"ingest_ms": round(stages[0] / n_traced, 4), "encode_ms": round(stages[1] / n_traced, 4),
                    "commit_ms": round(stages[2] / n_traced, 4)})
    if with_handles:
        times, same = handles_run(S, ctx, n_sessions, channels, settings, total_rounds, sources, [bytes(g) for g in got])
        t = np.array(times[warmup: warmup + rounds]) * 1e3
        res.update({"handles_ms_per_round": round(float(t.mean()), 3), "handles_headroom_x": round(20.0 / float(t.mean()), 2),
                    "pool_bytes_equal_handles": bool(same)})
        assert same, f"{name} S={n_sessions}: the pool's bytes differ from the per-session handles'"
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--sessions", default="256,1024,4096,16384")
    args = ap.parse_args()
    import torch

    import sea_codec_b200 as S
    from sea_codec_b200 import synth

    if not torch.cuda.is_available():
        raise SystemExit("pool_probe needs a CUDA device: nothing is measured without one")
    info = card()
    ctx = S.Context(0)
    n_rows = SPREAD + PRIME + args.warmup + args.rounds + 60
    results = []
    for channels, cfgs in ((2, [("stereo CBR-3", S.EncoderSettings(residual_bits=3.0)),
                                ("stereo VBR-3", S.EncoderSettings(residual_bits=3.0, vbr=True))]),
                           (8, [("8ch CBR-4", S.EncoderSettings(residual_bits=4.0))])):
        src = np.stack([synth.gen_stream(1000 + k, n_rows * PKT, channels, RATE).reshape(n_rows, PKT * channels) for k in range(SOURCES)])
        for name, st in cfgs:
            for n_sessions in ([1024] if channels == 8 else [int(x) for x in args.sessions.split(",")]):
                res = row(S, ctx, name, channels, st, n_sessions, args.rounds, args.warmup, src, n_sessions <= 1024)
                res.update(info)
                results.append(res)
                print(json.dumps(res), flush=True)
    ctx.close()
    hdr = f"{'row':14} {'S':>6} {'wall ms':>8} {'p99':>8} {'x RT':>7} {'enc/push':>8} {'ingest':>7} {'encode':>7} {'commit':>7} {'handles ms':>10} {'x RT':>6} {'same':>5}"
    print(f"# {info.get('gpu')} at {info.get('power_limit_w')} W power limit")
    print(hdr)
    for r in results:
        print(f"{r['row']:14} {r['sessions']:>6} {r['wall_ms_mean']:>8.3f} {r['wall_ms_p99']:>8.3f} {r['headroom_x']:>7.1f} "
              f"{r['encoding_sessions_per_push']:>8.1f} {r.get('ingest_ms', 0):>7.3f} {r.get('encode_ms', 0):>7.3f} {r.get('commit_ms', 0):>7.3f} "
              f"{r.get('handles_ms_per_round', float('nan')):>10.3f} {r.get('handles_headroom_x', float('nan')):>6.1f} "
              f"{str(r.get('pool_bytes_equal_handles', '-')):>5}")
    print(json.dumps({"pool_probe": results}))


if __name__ == "__main__":
    main()
