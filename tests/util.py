"""Shared helpers of the test-suite."""
import hashlib
import json
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REFERENCE_C_GOLDEN = os.path.join(ROOT, "tests", "golden", "reference_c.json")
SENTINEL = -12345


def sha(b) -> str:
    return hashlib.sha256(np.ascontiguousarray(b).tobytes() if isinstance(b, np.ndarray) else b).hexdigest()


def reference_c_result(oracle, key: str, encoded: bytes, lms: bool = False):
    """What the reference's own C decoder (c/sea.h) makes of `encoded`: (sha256 of its PCM, and with lms=True the LMS state it
    holds at the end of every chunk but the last, int16 [chunk][channel][8] -- history[4] then weights[4], mod 2^16).
    Where oracle/_ref is built, c/sea.h runs and must agree with tests/golden/reference_c.json; elsewhere the recorded result
    is used.  Either way `encoded` must be the very input the record belongs to.  The record's "source" says where it came
    from: while it is the oracle rather than c/sea.h, a test without oracle/_ref compares with the oracle's recorded result."""
    with open(REFERENCE_C_GOLDEN) as f:
        rec = json.load(f)["cases"][key]
    assert sha(encoded) == rec["sea_sha"], f"{key}: not the input whose c/sea.h result is recorded"
    want_lms = np.array(rec["lms"], dtype=np.int16) if lms else None
    if oracle.have_ref():
        if lms:
            info, states = oracle.ref_c_decode_lms(encoded)
            assert np.array_equal(states[:-1].astype(np.int16), want_lms), f"{key}: c/sea.h LMS differs from the record"
        else:
            info = oracle.ref_c_decode(encoded)
        assert sha(info.samples) == rec["pcm_sha"], f"{key}: c/sea.h PCM differs from the record"
    return (rec["pcm_sha"], want_lms) if lms else rec["pcm_sha"]


def gen_test_signal(channels: int, frames: int, rate: int = 44100, seed: int = 1) -> np.ndarray:
    """In the spirit of tests/helpers.rs:79-93 (square + sine mix, per-channel delay), but integer-exact: built from
    numpy float64 and rounded once, so every platform produces the same int16 samples."""
    n = np.arange(frames, dtype=np.float64)
    x = np.zeros(frames)

    def seg(a, b):
        return slice(int(frames * a), int(frames * b))

    def square(sl, gain, f):
        period = max(int(rate / f), 2)
        idx = np.arange(sl.stop - sl.start)
        x[sl] += gain * np.where((idx % period) < period // 2, 1.0, -1.0)

    def sine(sl, gain, f):
        idx = np.arange(sl.stop - sl.start)
        x[sl] += gain * np.sin(2 * np.pi * f / rate * idx)

    square(seg(0.0, 0.3), 0.5, 440.0)
    square(seg(0.1, 0.2), 0.3, 2150.1)
    sine(seg(0.1, 0.7), 0.5, 105.0)
    square(seg(0.6, 0.7), 0.5, 14000.0)
    sine(seg(0.5, 0.8), 0.8, 12000.0)
    sine(seg(0.8, 0.9), 1.0, 440.0)
    rng = np.random.default_rng(seed)
    x += rng.uniform(-0.01, 0.01, frames)
    delay = max(rate // 250, 1)
    out = np.zeros((frames, channels))
    for c in range(channels):
        d = min(delay * c, frames)
        out[d:, c] = x[: frames - d]
    return (np.clip(out, -1.0, 1.0) * 32767.0).astype(np.int16).reshape(-1)


def build_host_math():
    src = os.path.join(ROOT, "tests", "csrc", "host_math_check.cpp")
    out_dir = os.path.join(ROOT, "tests", "build")
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, "libhost_math_check.so")
    dep = os.path.join(ROOT, "sea_codec_b200", "csrc", "sea_common.cuh")
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(src), os.path.getmtime(dep)):
        subprocess.run(["g++", "-O2", "-std=c++17", "-x", "c++", "-shared", "-fPIC", "-fwrapv", "-o", so, src], check=True)
    return so


class Packed:
    """.sea streams in one device buffer; `shift` moves every stream off 16-byte alignment."""

    def __init__(self, files, shift=0):
        import torch

        self.files = list(files)
        offs, t = [], 0
        for f in self.files:
            t += shift
            offs.append(t)
            t = (t + len(f) + 15) // 16 * 16
        host = np.zeros(t + 64, dtype=np.uint8)
        for o, f in zip(offs, self.files):
            host[o: o + len(f)] = np.frombuffer(f, dtype=np.uint8)
        self.buf = torch.from_numpy(host).cuda()
        self.offs = np.array(offs, dtype=np.uint64)
        self.lens = np.array([len(f) for f in self.files], dtype=np.uint64)
        self.headers = np.stack([np.frombuffer(f[:22], dtype=np.uint8) for f in self.files])

    def corpus(self, ctx, skip_metadata=False):
        return ctx.corpus(self.buf, self.offs, self.lens, self.headers, skip_metadata=skip_metadata)


def windows(rng, frames, n, W, N=5120):
    """Seeded starts over every stream, with edge starts mixed in: 0, the chunk boundary N, the last frame, past the end, near 2^64."""
    ws = rng.integers(0, len(frames), size=n)
    ff = np.array([int(rng.integers(0, int(frames[s]) + 100)) for s in ws], dtype=np.uint64)
    if n:
        edges = [0, N, N - 1, int(frames[ws[0]]) - 1, int(frames[ws[0]]), 2**64 - 1, 2**64 - N, 2**63]
        for i, e in enumerate(edges[:n]):
            ff[i] = e
    return ws.astype(np.uint32), ff


def run_async(corpus, ws, ff, W, planar, pad=5, status=None):
    """corpus.decode_windows into an odd element offset of a sentinel-filled tensor; checks the sentinels and returns (slots, frames_out)."""
    import torch

    n, ch = len(ws), corpus.channels
    total = n * W * ch
    big = torch.full((total + 2 * pad + 1,), SENTINEL, dtype=torch.float32 if planar else torch.int16, device="cuda")
    out = big[pad: pad + total]
    fo = torch.full((max(n, 1),), -7, dtype=torch.int32, device="cuda")[:n]
    si = torch.tensor(np.asarray(ws, dtype=np.int64), device="cuda")
    fi = torch.tensor(np.asarray(ff, dtype=np.uint64).astype(np.int64), device="cuda")
    corpus.decode_windows(si, fi, W, float32_planar=planar, out=out, frames_out=fo, status=status)
    host = big.cpu().numpy()
    assert np.all(host[:pad] == SENTINEL) and np.all(host[pad + total:] == SENTINEL), "a byte outside the slots was written"
    return host[pad: pad + total], fo.cpu().numpy().astype(np.int64)
