"""Encoder settings at the edges of what make_encode_plan accepts, and host restatements of the choices that decide which code
runs for them.

The .sea format and make_encode_plan (sea_format.cpp) accept 1-255 channels, scale_factor_bits 1-8, scale_factor_frames (F)
1-255 and any frames_per_chunk (N) that is a multiple of F while a chunk stays within 65535 bytes.  SHAPES is a fixed covering
list over that space (not the cross product): every channel count where a kernel changes its mapping, every scale_factor_bits
and residual size, F = 1 / 7 / 20 / 64 / 255, chunks within 1 % of 65535 bytes, ragged last chunks, VBR scratch in global
memory and a 65535-item VBR sort.

The restatements follow the host code line by line:
  plan()            make_encode_plan (sea_format.cpp), with oracle.vbr_params for the VBR bucket counts
  encode_launch()   launch_encode_generic (encode_kernels.cu): fast or generic pass, warps, shared memory, where the VBR scratch
                    lives; `fixed=False` is the sizing before chunk buffers were sized from the job's largest chunk
  latency_smem()    decode_latency_smem (decode_latency.cu): whether the small-job decode kernel takes a geometry
  decode_route()    the kernel family run_decode (capi.cu) sends a uniform job to
  tile_frames_log2  the planar window tile of window_kernels.cu
tests/test_wide_shapes.py checks them on the CPU; tests/test_gpu_wide_shapes.py runs the shapes on the GPU.
No torch import here: the CPU tests run without it.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

from oracle import sea_oracle as O

MAX_CHUNK = 65535
SMEM_CAP = 200 * 1024
SMS = 148


def _ceil8(bits: int) -> int:
    return (bits + 7) // 8


def next_pow2(v: int) -> int:
    p = 2
    while p < v:
        p <<= 1
    return p


def hdr_bits(bits: float) -> int:
    return int(np.floor(np.float32(bits)))


# ------------------------------------------------------------------------------------------------ make_encode_plan

@dataclass(frozen=True)
class Plan:
    channels: int
    N: int
    F: int
    s: int
    bits: float
    vbr: bool
    hdr_bits: int
    base: int
    full_counts: tuple   # [base-1, base, base+1, base+2]
    full_chunk_bytes: int
    max_chunk_bytes: int
    full_chunk_valid: bool

    def counts(self, items: int):
        """vbr_distribution(items, target) of these settings."""
        return O.vbr_params(O.make_settings(self.bits, True, self.s, self.F, self.N), items)[2]


def _full_bytes(channels, s, F, bits, vbr, N):
    """(chunk bytes of a full chunk, VBR base); the size alone, before make_encode_plan's other checks."""
    items = (N // F) * channels
    if not vbr:
        return 4 + 16 * channels + _ceil8(items * s) + _ceil8(N * channels * hdr_bits(bits)), 0
    _, base, counts = O.vbr_params(O.make_settings(bits, True, s, F, N), items)
    return 4 + 16 * channels + _ceil8(items * s) + _ceil8(items * 2) + _ceil8(sum(counts[i] * (base + i - 1) for i in range(4)) * F), base


def plan(channels: int, s: int, F: int, bits: float, vbr: bool, N: int) -> Plan | None:
    """make_encode_plan restated; None where it rejects the settings."""
    if not (1 <= channels <= 255 and 1 <= s <= 8 and 1 <= F <= 255 and 1 <= N <= 65535) or N % F:
        return None
    if not (1.0 <= np.float32(bits) < 9.0):
        return None
    items = (N // F) * channels
    hb = hdr_bits(bits)
    full, base = _full_bytes(channels, s, F, bits, vbr, N)
    if not vbr:
        return None if full > MAX_CHUNK else Plan(channels, N, F, s, bits, False, hb, 0, (0, 0, 0, 0), full, full, True)
    if base < 1 or base + 1 > 8 or items > 65535 or full > MAX_CHUNK:
        return None
    counts = O.vbr_params(O.make_settings(bits, True, s, F, N), items)[2]
    valid = not ((counts[0] and base < 2) or (counts[2] and base + 1 > 8) or (counts[3] and base + 2 > 8))
    worst = 4 + 16 * channels + _ceil8(items * s) + _ceil8(items * 2) + _ceil8(N * channels * (base + 2))
    return Plan(channels, N, F, s, bits, True, hb, base, tuple(counts), full, max(full, worst), valid)


def largest_n(channels: int, s: int, F: int, bits: float, vbr: bool) -> int:
    """The largest N that make_encode_plan accepts: a bisection on the chunk size (which grows with N), then down to the first N
    that passes the plan's other checks."""
    fits = lambda k: (k * F * channels // F <= 65535 or not vbr) and _full_bytes(channels, s, F, bits, vbr, k * F)[0] <= MAX_CHUNK
    lo, hi = 1, 65535 // F
    if fits(hi):
        lo = hi
    while hi - lo > 1:
        mid = (lo + hi) // 2
        lo, hi = (mid, hi) if fits(mid) else (lo, mid)
    k = lo
    while k > 0 and plan(channels, s, F, bits, vbr, k * F) is None:
        k -= 1
    assert k > 0, (channels, s, F, bits, vbr)
    return k * F


def last_chunk_bound(p: Plan, last: int) -> int:
    """What plan_encode (capi.cu) takes as the largest VBR chunk of `last` frames: its own bucket counts with every block at F
    frames (the items past `sortable` keep size base), and no more than `last` frames at base+2 bits."""
    C, F, base = p.channels, p.F, p.base
    items = -(-last // F) * C
    sortable = last * C // F
    c = p.counts(sortable)
    size_sum = c[0] * (base - 1) + (c[1] + items - sortable) * base + c[2] * (base + 1) + c[3] * (base + 2)
    bits = min(size_sum * F, last * C * (base + 2))
    return min(4 + 16 * C + _ceil8(items * p.s) + _ceil8(items * 2) + _ceil8(bits), p.max_chunk_bytes)


def chunk_buf_bytes(p: Plan, stream_frames) -> int:
    """EncodeJob::chunk_buf_bytes: the largest chunk the streams of one job can produce."""
    if not p.vbr:
        return p.max_chunk_bytes
    out = p.full_chunk_bytes if any(f >= p.N for f in stream_frames) else 0
    for f in stream_frames:
        if f % p.N:
            out = max(out, last_chunk_bound(p, f % p.N))
    return out


# ------------------------------------------------------------------------------------------------ launch_encode_generic

ENC_LUT32, ENC_LUT16, ENC_LUT_GLOBAL = 0, 1, 2


def vbr_scratch_bytes(p: Plan) -> int:
    """enc_vbr_scratch_bytes: sort keys, indices, block offsets and row bits, descriptors and sizes of one chunk."""
    if not p.vbr:
        return 0
    nblk = p.N // p.F
    items = nblk * p.channels
    np2 = next_pow2(items)
    return (np2 * 8 + np2 * 4 + nblk * 8 + items * 5 + 255) & ~255


def _lut_entries(fb: int, base: int) -> int:
    if fb > 0:
        return 1 << fb
    lo = base - 1 if base > 1 else 1
    return sum(1 << (lo + i) for i in range(4) if lo + i <= 8)


@dataclass(frozen=True)
class EncLaunch:
    fast: bool
    warps: int
    T: int
    smem: int
    chunk_bytes: int       # the chunk buffer the kernel is given (EncParams::max_chunk_bytes)
    lut_mode: int
    vbr_scratch_shared: bool
    fits: bool             # False: cudaErrorInvalidConfiguration, nothing launched


def encode_launch(p: Plan, stream_frames=None, n_streams: int = 1, fixed: bool = True) -> EncLaunch:
    """launch_encode_generic restated (the split mapping and SEA_B200_ENC_LUT left at their defaults).  stream_frames: the frame
    counts of the job's streams (default: one full chunk each).  fixed=False: the sizing before the chunk buffer and the warp
    count were fitted to 200 KB."""
    C, F, s = p.channels, p.F, p.s
    nsf = 1 << s
    cpw = 32 // min(nsf, 32)
    fast = 3 <= s <= 5 and F == 20 and C <= 16
    warps = min(8, -(-C // cpw))

    def layout(chunk_bytes, warps):
        T = warps * 32
        smem = ((chunk_bytes + 3) // 4 + 2) * 4 + C * 17 * 4 + ((2 * F * T + 15) & ~15) + 16
        lut = ENC_LUT32
        if fast:
            smem += (warps * cpw * F * 2 + 15) & ~15
            fb = 0 if p.vbr else p.hdr_bits
            e = _lut_entries(fb, p.base)
            other = smem + 256 + (vbr_scratch_bytes(p) + 16 if p.vbr else 0)
            budget = 227 * 1024 // ((n_streams + 147) // 148)
            budget = budget - 1280 if budget > 1280 + 28 * 1024 else 28 * 1024
            if not p.vbr:
                lut = ENC_LUT32 if fb <= 7 else (ENC_LUT16 if s == 4 else ENC_LUT_GLOBAL)
            elif other + e * 128 <= budget:
                lut = ENC_LUT32
            elif s == 4 and other + e * 64 <= budget:
                lut = ENC_LUT16
            else:
                lut = ENC_LUT_GLOBAL
            if lut != ENC_LUT_GLOBAL:
                smem += e * (128 if lut == ENC_LUT32 else 64)
            smem += 4 * nsf * 4
        shared = False
        if p.vbr:
            sc = vbr_scratch_bytes(p)
            if sc <= 40 * 1024 and smem + sc + 16 <= SMEM_CAP:
                smem = ((smem + 15) & ~15) + sc
                shared = True
        return smem, lut, shared

    chunk = p.max_chunk_bytes
    smem, lut, shared = layout(chunk, warps)
    if fixed:
        need = chunk_buf_bytes(p, [p.N] if stream_frames is None else stream_frames)
        if smem > SMEM_CAP and need < chunk:
            chunk = need
            smem, lut, shared = layout(chunk, warps)
        while smem > SMEM_CAP and not fast and warps > 1:
            warps -= 1
            smem, lut, shared = layout(chunk, warps)
    return EncLaunch(fast, warps, warps * 32, smem, chunk, lut, shared, smem <= SMEM_CAP)


# ------------------------------------------------------------------------------------------------ decode routes

def latency_row_pitch(N: int) -> int:
    return ((N + 7) & ~7) + 8


def latency_smem(chunk_size: int, N: int, channels: int) -> int:
    """decode_latency_smem: shared memory of the warp-per-chunk kernel, 0 where it does not take the geometry."""
    if channels == 0 or channels > 32:
        return 0
    b = ((chunk_size + 2 + 16 + 15) & ~15) + channels * latency_row_pitch(N) * 2 + N * 6 + 32 + 4096 * 2
    return b if b <= SMEM_CAP else 0


def decode_route(channels: int, N: int, chunk_size: int, F: int, s: int, b: int, vbr: bool, chunks: int, latency_env=None) -> str:
    """The kernel family run_decode sends a uniform job to: "latency" (decode_latency_kernel), "mc" (decode_mc_kernel),
    "fast" (the unrolled / VBR / staged kernels of 1, 2, 3, 5 and 7 channels) or "generic" (decode_generic_kernel).
    latency_env: SEA_B200_DEC_LATENCY ("0", "1" or None).  The fast kernels also need 16-byte aligned input and PCM rows; the
    partial last chunks of an "mc" job run on the generic kernel (or the staged one where it takes the channel count)."""
    sm = latency_smem(chunk_size, N, channels)
    if sm:
        per_sm = min(32, (227 * 1024) // (sm + 1024))
        lat = chunks * 2 <= SMS * per_sm * 5 if latency_env is None else latency_env == "1"
        if lat:
            return "latency"
    mult = {4: 20, 8: 20, 6: 40}.get(channels, 80)
    if not vbr and 3 <= channels <= 8 and F == 20 and 1 <= s <= 6 and 1 <= b <= 8 and N % mult == 0:
        return "mc"
    if channels in (1, 2, 3, 5, 7) and 1 <= s <= 5 and 1 <= b <= 8:
        return "fast"
    return "generic"


def tile_frames_log2(channels: int) -> int:
    """window_kernels.cu: frames per planar tile, a power of two with frames x channels <= 4096 and at least 32 frames."""
    return max(32, 4096 // channels).bit_length() - 1


WIN_TILE_ELEMS = 8192


def tile_staged_elems(channels: int) -> int:
    """The most int16 a planar tile stages: TF frames x channels after up to 7 samples of the previous tile, in 8-sample vectors."""
    return -(-(7 + (1 << tile_frames_log2(channels)) * channels) // 8) * 8


# ------------------------------------------------------------------------------------------------ the shapes

@dataclass(frozen=True)
class Shape:
    channels: int
    s: int
    F: int
    bits: float
    vbr: bool
    N: int
    frames: int   # of the stream the tests encode

    @property
    def id(self) -> str:
        return f"c{self.channels}_s{self.s}_F{self.F}_{'vbr' if self.vbr else 'cbr'}{self.bits}_N{self.N}"

    def settings(self):
        return O.make_settings(self.bits, self.vbr, self.s, self.F, self.N)

    def plan(self) -> Plan:
        return plan(self.channels, self.s, self.F, self.bits, self.vbr, self.N)

    @property
    def decodable(self) -> bool:
        """VBR size codes are written as (size - floor(residual_bits) + 1) & 3 (chunk.rs:245-252): a stream reads back only
        where the base size is floor(residual_bits) - 1 or floor(residual_bits).  Short blocks (F = 1) take s + 2 bits per sample
        off the target, so their base is lower and the reference's decoder refuses what its encoder wrote."""
        p = self.plan()
        return not p.vbr or p.hdr_bits - 1 <= p.base <= p.hdr_bits


# (channels, scale_factor_bits, F, residual bits, vbr, N or None for the largest N the plan accepts, extra frames after the full
# chunks (not a multiple of F: a ragged last chunk), full chunks)
_SPEC = [
    # CBR: residual sizes 1-8, scale_factor_bits 1-8, F = 1 / 7 / 20 / 64 / 255
    (9, 1, 20, 8.0, False, 400, 233, 2),
    (15, 7, 7, 3.0, False, 490, 50, 2),
    (16, 8, 64, 1.0, False, None, 1001, 1),
    (17, 2, 1, 4.0, False, 240, 77, 2),
    (31, 5, 255, 2.0, False, None, 300, 1),
    (32, 3, 20, 5.0, False, 200, 111, 3),
    (33, 6, 64, 7.0, False, 640, 65, 2),
    (64, 4, 20, 6.0, False, None, 47, 1),
    (100, 8, 7, 1.0, False, 700, 13, 2),
    (128, 1, 255, 8.0, False, None, 254, 1),
    (129, 7, 64, 3.0, False, 256, 100, 2),
    # the settings whose CTA exceeded 200 KB before the fix: 160+ channels at F = 255
    (160, 1, 255, 1.0, False, None, 256, 1),
    (200, 8, 255, 1.0, False, None, 1, 1),
    (255, 4, 255, 7.0, False, 255, 254, 1),
    (255, 4, 255, 1.0, False, None, 300, 1),
    # VBR
    (9, 4, 20, 2.5, True, 400, 219, 2),
    (8, 5, 255, 4.5, True, None, 1000, 1),
    (16, 4, 64, 1.5, True, None, 777, 1),
    (16, 4, 20, 1.5, True, None, 333, 1),
    (32, 5, 20, 4.5, True, 1000, 9, 2),
    (33, 2, 7, 5.5, True, 350, 20, 2),
    (64, 7, 64, 7.3, True, 512, 100, 2),
    (100, 2, 255, 5.5, True, None, 256, 1),
    (129, 8, 20, 6.5, True, 600, 57, 2),
    (200, 1, 64, 3.0, True, 256, 65, 2),
    # F = 1 at 255 channels: 257 blocks x 255 channels = 65535 items, sorted by bitonic_sort over 65536 keys in global memory
    # (encode only: see Shape.decodable)
    (255, 1, 1, 7.3, True, 257, 100, 1),
]


def _build():
    out = []
    for C, s, F, bits, vbr, N, extra, full in _SPEC:
        N = largest_n(C, s, F, bits, vbr) if N is None else N
        out.append(Shape(C, s, F, bits, vbr, N, full * N + extra))
    return out


SHAPES = _build()
