#!/usr/bin/env python
"""Frame-window decode (sea_b200_decode_windows_device) in the shape of a training data loader: a corpus of .sea streams resident
in HBM, a batch of fixed-length crops at seeded random (stream, start) per call.  Prints one JSON line:

  python tools/window_probe.py [--reps R] [--windows W] [--window-seconds S]

Shapes: 4096 stereo 60 s 44.1 kHz CBR-3 streams, the same at VBR-3, and 256 eight-channel CBR-4 streams; every stream unique
(generated on the device by the library's synth kernel, encoded by encode_batch_device as bench.py does).  For each shape and
both output formats (int16 interleaved, float32 planar): windows/s and window Msamples/s from a host clock around the call (which
ends in a device synchronise), the covered / window sample ratio from the covering-chunk arithmetic, decode and extract kernel ms
(CUDA events, from the library's SEA_B200_TRACE lines), and next to it the full-stream decode_batch_device of the same streams.
The card's name and power limit are read in the same run.  "async" under each format: the registered-corpus form
(Context.corpus + Corpus.decode_windows) on the same windows -- GPU ms per call from CUDA events around back-to-back calls, host
enqueue us per call, graph-replay ms per call with one call captured, the route, and whether its slots and frames_out equal
decode_windows_device's.
"""
from __future__ import annotations

import argparse
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

RATE, N = 44100, 5120
TRACE = re.compile(r"window group \d+: .* decode ([0-9.]+) ms, extract ([0-9.]+) ms")


def card():
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(", ")
        return {"gpu": q[0], "power_limit_w": float(q[1])}
    except Exception as e:  # the run still says which card it was through torch
        import torch

        return {"gpu": torch.cuda.get_device_name(0), "power_limit_w": None, "nvidia_smi": str(e)}


def traced(fn):
    """Runs fn() with SEA_B200_TRACE set and the process's stderr (fd 2) captured; returns (result, summed decode ms, extract ms)."""
    os.environ["SEA_B200_TRACE"] = "1"
    sys.stderr.flush()
    saved = os.dup(2)
    with tempfile.TemporaryFile(mode="w+") as tmp:
        os.dup2(tmp.fileno(), 2)
        try:
            res = fn()
        finally:
            os.dup2(saved, 2)
            os.close(saved)
            os.environ.pop("SEA_B200_TRACE", None)
        tmp.seek(0)
        text = tmp.read()
    dec = ext = 0.0
    for m in TRACE.finditer(text):
        dec += float(m.group(1))
        ext += float(m.group(2))
    return res, dec, ext


def covered_ratio(first, n, total_frames, channels):
    """Samples of the covering chunks over window samples (sea_format.cpp plan_range)."""
    end = np.minimum(first + n, total_frames)
    k0, k1 = first // N, (end + N - 1) // N
    sub = np.minimum(k1 * N, total_frames) - k0 * N
    return float(np.sum(sub) * channels) / float(np.sum(n) * channels)


def shape(ctx, torch, name, n_streams, channels, settings, seconds, n_windows, win_seconds, reps, seed):
    dev = torch.device("cuda:0")
    frames = seconds * RATE
    spp = frames * channels
    pcm = torch.empty(n_streams * spp, dtype=torch.int16, device=dev)
    torch.cuda.synchronize()
    ctx.synth_pcm_device(pcm.data_ptr(), spp, (seed << 16) + np.arange(n_streams, dtype=np.uint32), frames, channels, RATE)
    stride = (ctx.encode_bound(frames, channels, settings) + 15) // 16 * 16
    sea = torch.zeros(n_streams * stride, dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()
    lens = ctx.encode_batch_device(pcm.data_ptr(), np.arange(n_streams, dtype=np.uint64) * spp, np.full(n_streams, frames),
                                   RATE, channels, settings, sea.data_ptr(), np.arange(n_streams, dtype=np.uint64) * stride)
    sea_off = np.arange(n_streams, dtype=np.uint64) * stride
    headers = sea.view(n_streams, stride)[:, :22].cpu().numpy()
    sea_bytes = int(np.sum(lens))

    # full-stream decode of the same corpus (into the PCM buffer, which the encode no longer needs)
    full_ms, full_wall = [], []
    for r in range(reps + 1):
        t0 = time.perf_counter()
        got = ctx.decode_batch_device(sea.data_ptr(), sea_off, lens, headers, pcm.data_ptr(), np.arange(n_streams, dtype=np.uint64) * spp)
        if r:
            full_wall.append(time.perf_counter() - t0)
            full_ms.append(ctx.last_kernel_ms)
    assert np.all(got == spp)

    rng = np.random.default_rng(seed)
    W = win_seconds * RATE
    ws = rng.integers(0, n_streams, size=n_windows).astype(np.uint32)
    ff = rng.integers(0, frames - W + 1, size=n_windows).astype(np.uint64)
    nf = np.full(n_windows, W, dtype=np.uint32)
    oo = np.arange(n_windows, dtype=np.uint64) * (W * channels)
    win_samples = n_windows * W * channels
    row = {"shape": name, "streams": n_streams, "channels": channels, "seconds": seconds, "vbr": bool(settings.vbr),
           "residual_bits": settings.residual_bits, "sea_bytes": sea_bytes, "windows": n_windows, "window_frames": W,
           "covered_over_window_samples": covered_ratio(ff.astype(np.int64), nf.astype(np.int64), frames, channels),
           "full_decode_batch_device": {"kernel_ms": float(np.median(full_ms)), "call_ms": float(np.median(full_wall)) * 1e3,
                                        "msamples_per_s": n_streams * spp / float(np.median(full_wall)) / 1e6}}
    full = pcm.view(n_streams, frames, channels)
    check = rng.choice(n_windows, size=8, replace=False)
    corpus = ctx.corpus(sea, sea_off, lens, headers)
    for planar in (False, True):
        out = torch.empty(win_samples, dtype=torch.float32 if planar else torch.int16, device=dev)
        torch.cuda.synchronize()

        def call():
            return ctx.decode_windows_device(sea.data_ptr(), sea_off, lens, headers, ws, ff, nf, out.data_ptr(), oo, float32_planar=planar)

        call()  # warm-up (scratch allocation, module load)
        walls, kms, decs, exts = [], [], [], []
        for _ in range(reps):
            t0 = time.perf_counter()
            fo, dec, ext = traced(call)
            walls.append(time.perf_counter() - t0)
            kms.append(ctx.last_kernel_ms)
            decs.append(dec)
            exts.append(ext)
        assert np.all(fo == W)
        for w in check:  # every window equals the slice of the full decode
            want = full[int(ws[w]), int(ff[w]): int(ff[w]) + W]
            slot = out[int(oo[w]): int(oo[w]) + W * channels]
            ok = torch.equal(slot.view(channels, W), want.t().float() / 32768.0) if planar else torch.equal(slot.view(W, channels), want)
            assert ok, (name, planar, int(w))
        wall = float(np.median(walls))
        row["f32_planar" if planar else "i16"] = {
            "call_ms": wall * 1e3, "windows_per_s": n_windows / wall, "window_msamples_per_s": win_samples / wall / 1e6,
            "kernel_ms": float(np.median(kms)), "decode_ms": float(np.median(decs)), "extract_ms": float(np.median(exts)),
            "extract_gbs": win_samples * (2 + (4 if planar else 2)) / (float(np.median(exts)) * 1e-3) / 1e9,
            "window_calls_per_full_decode": float(np.median(full_wall)) / wall,
            "async": corpus_async(ctx, torch, corpus, ws, ff, W, planar, out, fo, reps)}
    corpus.close()
    ctx.set_stream(torch.cuda.current_stream().cuda_stream)
    return row


def corpus_async(ctx, torch, corpus, ws, ff, W, planar, ref_out, ref_fo, reps, calls=20):
    """The registered-corpus form on the same windows: GPU ms per call (CUDA events around `calls` back-to-back calls), host enqueue
    us per call, graph-replay ms per call (one captured call), and a check that slots and frames_out equal decode_windows_device's."""
    n = len(ws)
    si = torch.tensor(ws.astype(np.int64), device="cuda")
    fi = torch.tensor(ff.astype(np.int64), device="cuda")
    out = torch.empty_like(ref_out)
    fo = torch.zeros(n, dtype=torch.int32, device="cuda")

    def call():
        corpus.decode_windows(si, fi, W, float32_planar=planar, out=out, frames_out=fo)

    call()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    gpu, enq = [], []
    for _ in range(reps):
        e0.record()
        t0 = time.perf_counter()
        for _ in range(calls):
            call()
        enq.append((time.perf_counter() - t0) / calls)
        e1.record()
        e1.synchronize()
        gpu.append(e0.elapsed_time(e1) / calls)
    equal = bool(torch.equal(out, ref_out)) and bool(np.array_equal(fo.cpu().numpy().astype(np.uint64), ref_fo))
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=side):
        call()
    torch.cuda.synchronize()
    graph = []
    for _ in range(reps):
        e0.record()
        for _ in range(calls):
            g.replay()
        e1.record()
        e1.synchronize()
        graph.append(e0.elapsed_time(e1) / calls)
    corpus.check()
    assert equal, "async slots differ from decode_windows_device's"
    return {"route": corpus.route, "gpu_ms": float(np.median(gpu)), "enqueue_us": float(np.median(enq)) * 1e6,
            "graph_replay_ms": float(np.median(graph)), "equal_to_decode_windows_device": equal}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--windows", type=int, default=4096)
    ap.add_argument("--window-seconds", type=int, default=2)
    ap.add_argument("--seconds", type=int, default=60)
    args = ap.parse_args()
    import torch

    import sea_codec_b200 as S

    if not torch.cuda.is_available():
        raise SystemExit("window_probe.py needs a CUDA device (libsea_b200 has no CPU fallback)")
    torch.cuda.set_device(0)
    ctx = S.Context(0)
    ctx.set_stream(torch.cuda.current_stream().cuda_stream)
    info = {"tool": "window_probe", **card()}
    rows = [
        shape(ctx, torch, "stereo_cbr3", 4096, 2, S.EncoderSettings(residual_bits=3.0), args.seconds, args.windows, args.window_seconds,
              args.reps, 1),
        shape(ctx, torch, "stereo_vbr3", 4096, 2, S.EncoderSettings(residual_bits=3.0, vbr=True), args.seconds, args.windows,
              args.window_seconds, args.reps, 2),
        shape(ctx, torch, "ch8_cbr4", 256, 8, S.EncoderSettings(residual_bits=4.0), args.seconds, args.windows, args.window_seconds,
              args.reps, 3),
    ]
    info["shapes"] = rows
    ctx.close()
    print(json.dumps(info))


if __name__ == "__main__":
    main()
