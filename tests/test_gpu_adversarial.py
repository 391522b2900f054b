"""Every decode route against the CPU oracle on chunk payloads no encoder writes.

An encoder only writes the LMS headers, scale factors and residual codes that ordinary signals call for.  A decoder must take
any valid chunk, so `craft` rewrites the payload of every chunk of an encoded stream (LMS bytes, scale factors, residual codes;
with `size_codes`, also the VBR size codes) and leaves the file header, the chunk length and chunk header bytes 0-3 alone, which
keeps the stream on the route it was built for.  The patterns reach what encoder-made streams do not: the top scale-factor row,
32-bit wrap-around of the LMS dot product, weights past 2^24 (where FP32 stops being exact) and long runs of saturation at both
ends.  A plain Python LMS (`mirror_decode`) restates the decoder with explicit 32-bit wrap-around; the CPU tests check it against
the oracle and check that the crafted inputs reach those edges, so the inputs can be checked on a machine without a GPU.  The
GPU tests drive the crafted streams through every decode entry point and route knob and compare with oracle.sea_decode."""
import functools
import io

import numpy as np
import pytest

import sea_codec_b200 as S
from oracle import sea_oracle as O
from sea_codec_b200 import api, synth
from util import Packed, run_async, windows

F = 20                    # scale_factor_frames of every stream here
PATTERNS = ("random", "lms_wrap", "sf_top", "saturate")
# (history, weight) in all four taps: sum w*h = 2^32 (wraps to 0), 2^31 (reads back as -2^31: prediction -262144, not
# +262144) and 4 * -32768 * 32767 (wraps to 2^17: prediction +16, not -524272)
LMS_WRAP = ((-32768, -32768), (-32768, -16384), (-32768, 32767))
RUNAWAY_N = 65520         # the largest multiple of 20 frames whose chunk fits the u16 frames_per_chunk


# ------------------------------------------------------------------------------------------------ chunk layout and bits

class Chunk:
    """Byte offsets of one chunk's sections (oracle/sea_oracle.c chunk_from_slice)."""

    def __init__(self, blob, pos, end, frames):
        self.pos, self.end, self.frames = pos, end, frames
        self.C = blob[5]
        self.vbr = blob[pos] == 2
        self.s, self.b, self.F = blob[pos + 1] >> 4, blob[pos + 1] & 15, blob[pos + 2]
        self.items = -(-frames // self.F) * self.C
        self.lms_off = pos + 4
        self.sf_off = self.lms_off + 16 * self.C
        self.vbr_off = self.sf_off + -(-self.items * self.s // 8)
        self.res_off = self.vbr_off + (-(-self.items * 2 // 8) if self.vbr else 0)

    def widths(self, blob):
        """Residual bits of every sample, frame-major: b, or the VBR size of the sample's block and channel."""
        n = self.frames * self.C
        if not self.vbr:
            return np.full(n, self.b, dtype=np.int64)
        sizes = unpack_bits(blob[self.vbr_off: self.res_off], 2, self.items) + self.b - 1
        i = np.arange(n)
        return sizes[(i // self.C) // self.F * self.C + i % self.C]


def chunks(blob):
    cs = int.from_bytes(blob[6:8], "little")
    N = int.from_bytes(blob[8:10], "little")
    total = int.from_bytes(blob[14:18], "little")
    assert total > 0 and int.from_bytes(blob[18:22], "little") == 0, "a stream with total_frames and no metadata"
    out, k = [], 0
    while k * N < total and 22 + k * cs < len(blob):
        pos = 22 + k * cs
        out.append(Chunk(blob, pos, min(pos + cs, len(blob)), min(N, total - k * N)))
        k += 1
    return out


def pack_bits(values, widths):
    """MSB-first bit packing (bits.rs BitPacker), zero-padded to whole bytes."""
    values = np.asarray(values, dtype=np.int64)
    widths = np.broadcast_to(np.asarray(widths, dtype=np.int64), values.shape)
    owner = np.repeat(np.arange(values.size), widths)
    bit = np.arange(owner.size) - np.repeat(np.cumsum(widths) - widths, widths)
    return np.packbits(((values[owner] >> (widths[owner] - 1 - bit)) & 1).astype(np.uint8)).tobytes()


def unpack_bits(data, widths, n):
    widths = np.broadcast_to(np.asarray(widths, dtype=np.int64), (n,))
    bits = np.unpackbits(np.frombuffer(bytes(data), dtype=np.uint8)).astype(np.int64)
    starts = np.cumsum(widths) - widths
    assert n == 0 or starts[-1] + widths[-1] <= bits.size, "section shorter than its codes"
    v = np.zeros(n, dtype=np.int64)
    for j in range(int(widths.max()) if n else 0):
        m = j < widths
        v[m] = v[m] * 2 + bits[starts[m] + j]
    return v


@functools.lru_cache(maxsize=None)
def dqt(b, s):
    """The library's dequantisation table [scale factor][code] (sea_b200_tables)."""
    recip, tab = np.zeros(1 << s, np.int32), np.zeros((1 << s, 1 << b), np.int32)
    assert S.lib().sea_b200_tables(b, s, recip.ctypes.data, tab.ctypes.data) == 0
    return tab


@functools.lru_cache(maxsize=None)
def oracle_dqt(b, s):
    return O.tables(b, s)[1]


# ------------------------------------------------------------------------------------------------ the plain reference

def wrap32(x):
    return ((x + 0x80000000) & 0xFFFFFFFF) - 0x80000000


def lms_step(w, h, d):
    """One sample of lms.rs:33-51 and decoder.rs:38-45 in Python ints: (sample, unclamped sum, whether sum w*h wrapped)."""
    acc = w[0] * h[0] + w[1] * h[1] + w[2] * h[2] + w[3] * h[3]
    v = wrap32((wrap32(acc) >> 13) + d)
    y = min(max(v, -32768), 32767)
    delta = d >> 4
    for i in range(4):
        w[i] = wrap32(w[i] + (delta if h[i] >= 0 else -delta))
    h[0], h[1], h[2], h[3] = h[1], h[2], h[3], y
    return y, v, acc != wrap32(acc)


def mirror_decode(blob, stats=None):
    """Decodes a stream with lms_step and the oracle's tables; `stats` collects which edges the samples reached."""
    out = []
    st = dict(top_sf=0, wrapped=0, sat_hi=0, sat_lo=0, max_w=0) if stats is None else stats
    for ck in chunks(blob):
        C, s = ck.C, ck.s
        lms = np.frombuffer(bytes(blob[ck.lms_off: ck.sf_off]), dtype="<i2").reshape(C, 8).astype(int).tolist()
        state = [(row[4:], row[:4]) for row in lms]
        sf = unpack_bits(blob[ck.sf_off: ck.vbr_off], s, ck.items).tolist()
        widths = ck.widths(blob)
        codes = unpack_bits(blob[ck.res_off: ck.end], widths, ck.frames * C).tolist()
        widths = widths.tolist()
        for i, q in enumerate(codes):
            f, c = divmod(i, C)
            w, h = state[c]
            r = sf[f // ck.F * C + c]
            y, v, wrapped = lms_step(w, h, int(oracle_dqt(widths[i], s)[r, q]))
            out.append(y)
            st["top_sf"] += r == (1 << s) - 1
            st["wrapped"] += wrapped
            st["sat_hi"] += v > 32767
            st["sat_lo"] += v < -32768
            st["max_w"] = max(st["max_w"], max(abs(x) for x in w))
    return np.array(out, dtype=np.int16)


# ------------------------------------------------------------------------------------------------ the crafter

def craft(blob, pattern, seed=0, size_codes=None):
    """`blob` with every chunk's payload rewritten.  Patterns:
      random    seeded LMS bytes, scale factors and codes
      lms_wrap  the LMS_WRAP headers (case (chunk + channel) % 3), seeded scale factors and codes
      sf_top    the encoder's LMS, every scale factor 2^s - 1, seeded codes
      saturate  the encoder's LMS, every scale factor 2^s - 1, runs of 8 blocks of the largest positive dequantised value, then
                8 of the largest negative
      runaway   the encoder's LMS, every scale factor 2^s - 1, each code picked (by lms_step) so that the largest |weight| of
                its channel keeps growing
    VBR size codes are kept; with size_codes = m they are redrawn from 0..m and the residual bytes are seeded noise."""
    rng = np.random.default_rng(seed)
    out = bytearray(blob)
    for k, ck in enumerate(chunks(blob)):
        C, s, n = ck.C, ck.s, ck.frames * ck.C
        top = (1 << s) - 1
        if size_codes is not None:
            assert ck.vbr
            out[ck.vbr_off: ck.res_off] = pack_bits(rng.integers(0, size_codes + 1, ck.items), 2)
            out[ck.sf_off: ck.vbr_off] = pack_bits(rng.integers(0, 1 << s, ck.items), s)
            out[ck.res_off: ck.end] = rng.integers(0, 256, ck.end - ck.res_off, dtype=np.uint8).tobytes()
            continue
        if pattern == "random":
            out[ck.lms_off: ck.sf_off] = rng.integers(-32768, 32768, 8 * C).astype("<i2").tobytes()
        elif pattern == "lms_wrap":
            hw = [LMS_WRAP[(k + c) % 3] for c in range(C)]
            out[ck.lms_off: ck.sf_off] = np.array([[h] * 4 + [w] * 4 for h, w in hw], dtype="<i2").tobytes()
        sf = rng.integers(0, 1 << s, ck.items) if pattern in ("random", "lms_wrap") else np.full(ck.items, top)
        out[ck.sf_off: ck.vbr_off] = pack_bits(sf, s)
        widths = ck.widths(blob)
        if pattern in ("random", "lms_wrap", "sf_top"):
            codes = rng.integers(0, 1 << widths)
        elif pattern == "saturate":
            hi = {wd: int(np.argmax(dqt(wd, s)[top])) for wd in set(widths.tolist())}
            lo = {wd: int(np.argmin(dqt(wd, s)[top])) for wd in set(widths.tolist())}
            blk = np.arange(n) // C // ck.F
            codes = np.array([(hi if (bk // 8) % 2 == 0 else lo)[wd] for bk, wd in zip(blk.tolist(), widths.tolist())])
        else:
            assert pattern == "runaway" and not ck.vbr
            row = dqt(ck.b, s)[top]
            pos, neg = int(np.argmax(row)), int(np.argmin(row))
            lms = np.frombuffer(bytes(blob[ck.lms_off: ck.sf_off]), dtype="<i2").reshape(C, 8).astype(int).tolist()
            state = [(r[4:], r[:4]) for r in lms]
            codes = []
            for i in range(n):
                w, h = state[i % C]
                j = max(range(4), key=lambda t: abs(w[t]))
                # w[j] moves by (d >> 4) * sign(h[j]): pick the sign of d that moves it away from zero
                q = pos if (w[j] >= 0) == (h[j] >= 0) else neg
                codes.append(q)
                lms_step(w, h, int(row[q]))
        packed = pack_bits(codes, widths)
        assert ck.res_off + len(packed) <= ck.end
        out[ck.res_off: ck.res_off + len(packed)] = packed
    return bytes(out)


@functools.lru_cache(maxsize=None)
def base_stream(C, b, s, vbr=False, N=5120, frames=None, seed=0):
    """An oracle-encoded synth stream: two full chunks and a partial one unless `frames` says otherwise."""
    frames = 2 * N + 1234 if frames is None else frames
    pcm = synth.gen_stream(1000 + 97 * C + 13 * s + int(10 * b) + seed, frames, C, 44100)
    return O.sea_encode(pcm, 44100, C, O.make_settings(b, vbr, s, F, N))


# ------------------------------------------------------------------------------------------------ shapes

CBR_SHAPES = [(C, b, s) for C in (1, 2) for b in range(1, 9) for s in range(1, 6)] + \
             [(C, b, s) for C in (3, 5, 8) for b in (1, 4, 8) for s in (2, 4, 6)] + \
             [(C, b, s) for C in (1, 2, 3) for b in (1, 8) for s in (7, 8)]
VBR_SHAPES = [(C, r, s) for C in (1, 2, 3) for r in (2.5, 4.5, 7.3) for s in (3, 4, 5)] + [(2, 4.5, 7), (1, 3.5, 8)]


def _id(shape, vbr):
    C, b, s = shape
    return f"{'vbr' if vbr else 'cbr'}{b}_c{C}_s{s}"


ALL_SHAPES = [pytest.param(sh, False, id=_id(sh, False)) for sh in CBR_SHAPES] + \
             [pytest.param(sh, True, id=_id(sh, True)) for sh in VBR_SHAPES]


def crafted_set(C, b, s, vbr, **kw):
    base = base_stream(C, b, s, vbr, **kw)
    return base, [craft(base, p, seed=31 * i + s) for i, p in enumerate(PATTERNS)]


# ------------------------------------------------------------------------------------------------ CPU: the inputs themselves

def _payload_mask(blob):
    """True on every byte the crafter may change (without size_codes): LMS, scale factors, residuals."""
    m = np.zeros(len(blob), dtype=bool)
    for ck in chunks(blob):
        m[ck.lms_off: ck.vbr_off] = True
        m[ck.res_off: ck.end] = True
    return m


@pytest.mark.parametrize("shape,vbr", ALL_SHAPES)
def test_oracle_accepts_every_crafted_stream_and_headers_stay(shape, vbr):
    base, files = crafted_set(*shape, vbr)
    keep = ~_payload_mask(base)
    for p, f in zip(PATTERNS, files):
        assert len(f) == len(base) and f != base, p
        assert np.array_equal(np.frombuffer(f, np.uint8)[keep], np.frombuffer(base, np.uint8)[keep]), p
        assert O.sea_decode(f).samples.size == O.sea_decode(base).samples.size, p


MIRROR_SHAPES = [((1, 1, 1), False), ((2, 3, 4), False), ((1, 8, 5), False), ((2, 5, 8), False), ((3, 4, 6), False),
                 ((2, 4.5, 4), True), ((1, 2.5, 3), True)]


@pytest.mark.parametrize("shape,vbr", MIRROR_SHAPES)
def test_mirror_equals_oracle_and_crafted_inputs_reach_the_edges(shape, vbr):
    base, files = crafted_set(*shape, vbr, N=1000)
    assert np.array_equal(mirror_decode(base), O.sea_decode(base).samples)
    for p, f in zip(PATTERNS, files):
        st = dict(top_sf=0, wrapped=0, sat_hi=0, sat_lo=0, max_w=0)
        assert np.array_equal(mirror_decode(f, st), O.sea_decode(f).samples), p
        if p == "lms_wrap":
            assert st["wrapped"] > 0, p
        if p in ("sf_top", "saturate"):
            assert st["top_sf"] == O.sea_decode(f).samples.size, p
        if p == "saturate":
            assert st["sat_hi"] > 100 and st["sat_lo"] > 100, (p, st)


def test_lms_wrap_cases_give_the_documented_predictions():
    for (h, w), pred in zip(LMS_WRAP, (0, -262144, 16)):
        ww, hh = [w] * 4, [h] * 4
        y, v, wrapped = lms_step(ww, hh, 0)
        assert wrapped and v == pred
        assert (w * h * 4) >> 13 != pred  # what 64-bit arithmetic would give


@pytest.mark.parametrize("C", [1, 2])
def test_weight_runaway_passes_2_24(C):
    """One full chunk of RUNAWAY_N frames at b = 1, s = 5 (|d| = 8192, so a weight moves 512 per sample): the greedy codes push
    the largest weight of every channel past 2^24 and the prediction wraps."""
    base = base_stream(C, 1, 5, N=RUNAWAY_N, frames=RUNAWAY_N + 1000)
    f = craft(base, "runaway")
    st = dict(top_sf=0, wrapped=0, sat_hi=0, sat_lo=0, max_w=0)
    assert np.array_equal(mirror_decode(f, st), O.sea_decode(f).samples)
    assert st["max_w"] >= 1 << 24, st
    assert st["wrapped"] > 0 and st["sat_hi"] > 0 and st["sat_lo"] > 0, st


# ------------------------------------------------------------------------------------------------ GPU helpers

@pytest.fixture(scope="module")
def lctx():
    """The corpora's own context (a Corpus binds its context to torch's current stream)."""
    c = S.Context(0)
    yield c
    import torch

    torch.cuda.synchronize()


def expected_slots(wants, C, ws, ff, W, planar):
    """Window slots from the oracle's samples: the window's frames, then zeros; float32 planar = int16 / 32768."""
    n = len(ws)
    out = np.zeros((n, W, C), dtype=np.int16)
    fo = np.zeros(n, dtype=np.int64)
    for i, (si, f0) in enumerate(zip(ws, ff)):
        x, f0 = wants[int(si)].reshape(-1, C), int(f0)
        if f0 < len(x):
            k = min(W, len(x) - f0)
            out[i, :k] = x[f0: f0 + k]
            fo[i] = k
    if planar:
        return (out.transpose(0, 2, 1).astype(np.float32) / np.float32(32768)).reshape(-1), fo
    return out.reshape(-1), fo


def launches(ctx, fn):
    n0 = ctx.launch_count
    r = fn()
    return r, ctx.launch_count - n0


def check_corpus(lctx, files, wants, N, route, Ws, rng, n_windows=16):
    """A corpus of `files` on `route`: every window, int16 and planar, equals the oracle's slice; sentinels and frames_out."""
    packed = Packed(files, shift=3)
    corpus = packed.corpus(lctx)
    assert corpus.route == route
    C = corpus.channels
    assert corpus.stream_frames.tolist() == [w.size // C for w in wants]
    for W in Ws:
        for planar in (False, True):
            ws, ff = windows(rng, corpus.stream_frames, n_windows, W, N)
            got, fo = run_async(corpus, ws, ff, W, planar)
            want, fo_want = expected_slots(wants, C, ws, ff, W, planar)
            assert np.array_equal(fo, fo_want), (route, W, planar)
            assert np.array_equal(got, want), (route, W, planar, np.flatnonzero(got != want)[:8])
    corpus.check()
    corpus.close()


def corpus_fast_ok(C, b, s, vbr):
    return not vbr and C <= 2 and s <= 5


# ------------------------------------------------------------------------------------------------ GPU: every route

@pytest.mark.gpu
@pytest.mark.parametrize("shape,vbr", ALL_SHAPES)
def test_every_decode_route_on_crafted_payloads(ctx, lctx, shape, vbr, monkeypatch):
    """The four crafted streams of a shape through the warp-per-chunk kernel, the throughput kernels under every route knob,
    decode_range, decode_windows_device, the streaming decoder and (where the fast corpus test does not cover the shape) the
    generic corpus route, each against the oracle."""
    import torch

    C, b, s = shape
    base, files = crafted_set(C, b, s, vbr)
    wants = [O.sea_decode(f).samples for f in files]
    N = 5120

    # the warp-per-chunk kernel: the same launches as for the encoder's stream
    monkeypatch.setenv("SEA_B200_DEC_LATENCY", "1")
    _, n_base = launches(ctx, lambda: ctx.sea_decode(base))
    for p, f, w in zip(PATTERNS, files, wants):
        got, n = launches(ctx, lambda: ctx.sea_decode(f).samples)
        assert np.array_equal(got, w), ("latency", p)
        assert n == n_base, ("latency", p)
    monkeypatch.setenv("SEA_B200_DEC_LATENCY", "0")

    # the throughput kernels on a uniform batch; a crafted payload must not send the batch to another route than the encoder's
    knobs = [{}, {"SEA_B200_FULL_CTAS": "1"}] + ([{"SEA_B200_VBR_RS": "2"}, {"SEA_B200_VBR_KF": "0"}] if vbr else [])
    for knob in knobs:
        for k, v in knob.items():
            monkeypatch.setenv(k, v)
        _, n_base = launches(ctx, lambda: ctx.decode_batch([base] * (2 * len(files))))
        got, n = launches(ctx, lambda: ctx.decode_batch(files * 2))
        assert n == n_base, knob
        for i, g in enumerate(got):
            assert np.array_equal(g.samples, wants[i % len(files)]), (knob, PATTERNS[i % len(files)])
        for k in knob:
            monkeypatch.delenv(k)

    # decode_range and decode_windows_device
    rng = np.random.default_rng(C * 100 + s * 10 + int(b * 2))
    frames = wants[0].size // C
    for f, w in zip(files, wants):
        for first, n in ((0, 1), (N - 1, 2), (N, N), (int(rng.integers(0, frames)), int(rng.integers(1, 3 * N))), (frames - 5, 100)):
            got = ctx.decode_range(f, first, n).samples
            assert np.array_equal(got, w[first * C: (first + n) * C]), (first, n)
    packed = Packed(files, shift=1)
    for W in (1, N + 7):
        for planar in (False, True):
            ws, ff = windows(rng, np.full(len(files), frames), 24, W, N)
            out = torch.zeros(len(ws) * W * C, dtype=torch.float32 if planar else torch.int16, device="cuda")
            fo = ctx.decode_windows_device(packed.buf.data_ptr(), packed.offs, packed.lens, packed.headers, ws, ff, np.full(len(ws), W),
                                           out.data_ptr(), np.arange(len(ws), dtype=np.uint64) * (W * C), float32_planar=planar)
            want, fo_want = expected_slots(wants, C, ws, ff, W, planar)
            assert np.array_equal(fo.astype(np.int64), fo_want), (W, planar)
            assert np.array_equal(out.cpu().numpy(), want), (W, planar)

    # the streaming decoder: chunk by chunk, and three chunks per launch
    for f, w in zip(files, wants):
        for step in (lambda d: d.decode_frame(), lambda d: d.decode_frames(3)):
            sink = io.BytesIO()
            dec = S.SeaDecoder(io.BytesIO(f), sink, ctx=ctx)
            while step(dec):
                pass
            dec.close()
            assert np.array_equal(np.frombuffer(sink.getvalue(), dtype="<i2"), w)

    # a corpus (the 1- and 2-channel CBR shapes of the fast kernel run in test_corpus_fast_kernel_instances)
    if not corpus_fast_ok(C, b, s, vbr):
        check_corpus(lctx, files, wants, N, "generic", (1, N + 1, 3 * N + 7), rng)


@pytest.mark.gpu
@pytest.mark.parametrize("C", [1, 2])
def test_weight_runaway_on_every_route(ctx, lctx, C, monkeypatch):
    """Weights past 2^24 and a wrapping prediction for most of a 65520-frame chunk, through the throughput kernels (one full
    chunk and a partial one), the warp-per-chunk kernel where it takes the chunk, the streaming decoder and both corpus routes."""
    N = RUNAWAY_N
    base = base_stream(C, 1, 5, N=N, frames=N + 1000)
    f = craft(base, "runaway")
    want = O.sea_decode(f).samples
    for lat in ("1", "0"):
        monkeypatch.setenv("SEA_B200_DEC_LATENCY", lat)
        _, n_base = launches(ctx, lambda: ctx.sea_decode(base))
        got, n = launches(ctx, lambda: ctx.sea_decode(f).samples)
        assert np.array_equal(got, want) and n == n_base, lat
    for knob in ({}, {"SEA_B200_FULL_CTAS": "1"}):
        for k, v in knob.items():
            monkeypatch.setenv(k, v)
        _, n_base = launches(ctx, lambda: ctx.decode_batch([base] * 4))
        got, n = launches(ctx, lambda: ctx.decode_batch([f] * 4))
        assert n == n_base, knob
        assert all(np.array_equal(g.samples, want) for g in got), knob
        for k in knob:
            monkeypatch.delenv(k)
    sink = io.BytesIO()
    dec = S.SeaDecoder(io.BytesIO(f), sink, ctx=ctx)
    while dec.decode_frames(2):
        pass
    assert np.array_equal(np.frombuffer(sink.getvalue(), dtype="<i2"), want)
    rng = np.random.default_rng(C)
    for route in ("generic", "fast"):
        monkeypatch.setenv("SEA_B200_CORPUS_ROUTE", route)
        check_corpus(lctx, [f, f], [want, want], N, route, (1, 33, N - 1, N + 1001), rng, n_windows=8)


# ------------------------------------------------------------------------------------------------ GPU: the corpus fast kernel

CORPUS_FPC = (20, 40, 1000, 5100, 5120)


@pytest.mark.gpu
@pytest.mark.parametrize("s", range(1, 6))
@pytest.mark.parametrize("b", range(1, 9))
@pytest.mark.parametrize("C", [1, 2])
def test_corpus_fast_kernel_instances(lctx, C, b, s, monkeypatch):
    """Every corpus_fast_kernel<C, BT> instance at every scale_factor_bits it takes, each instance over all five chunk lengths
    (20 frames is shorter than a 32-frame tile, 5100 is not a multiple of 32), encoder-made and crafted payloads, int16 and
    float32 planar, against the oracle; then the same corpora on the generic route."""
    N = CORPUS_FPC[(b + s) % len(CORPUS_FPC)]
    lengths = (3 * N + 7, 2 * N, N + N // 2 + 1, 6 * N - 3)  # every stream longer than a chunk keeps the corpus uniform
    enc = [base_stream(C, b, s, N=N, frames=fr, seed=i) for i, fr in enumerate(lengths)]
    crafted = [craft(e, PATTERNS[(i + b) % len(PATTERNS)], seed=i + 7 * s) for i, e in enumerate(enc)]
    Ws = (1, 31, 32, 33, N - 1, N, 3 * N + 7, 7 * N)
    rng = np.random.default_rng(C * 100 + b * 10 + s)
    for files in (enc, crafted):
        wants = [O.sea_decode(f).samples for f in files]
        for route in ("fast", "generic"):
            monkeypatch.setenv("SEA_B200_CORPUS_ROUTE", route)
            check_corpus(lctx, files, wants, N, route, Ws, rng)
        monkeypatch.delenv("SEA_B200_CORPUS_ROUTE")
        assert Packed(files).corpus(lctx).route == "fast"  # what the library picks by itself


# ------------------------------------------------------------------------------------------------ GPU: graph capture, generic route

@pytest.mark.gpu
@pytest.mark.parametrize("C,b,vbr", [(2, 3.5, True), (8, 4, False)])
def test_generic_route_graph_capture_and_replay(lctx, C, b, vbr):
    import torch

    N = 5120
    files = [craft(base_stream(C, b, 4, vbr, frames=N * 3 + 321 * i, seed=i), PATTERNS[i % 4], seed=i) for i in range(4)]
    wants = [O.sea_decode(f).samples for f in files]
    packed = Packed(files, shift=2)
    corpus = packed.corpus(lctx)
    assert corpus.route == "generic"
    n, W = 48, 2 * N + 17
    for planar in (False, True):
        si = torch.zeros(n, dtype=torch.int64, device="cuda")
        fi = torch.zeros(n, dtype=torch.int64, device="cuda")
        fo = torch.zeros(n, dtype=torch.int32, device="cuda")
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            corpus.decode_windows(si, fi, W, float32_planar=planar, frames_out=fo)  # warm-up outside the capture
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            out = corpus.decode_windows(si, fi, W, float32_planar=planar, frames_out=fo)
        rng = np.random.default_rng(9 + C)
        for _ in range(3):
            ws, ff = windows(rng, corpus.stream_frames, n, W, N)
            si.copy_(torch.tensor(ws.astype(np.int64)))
            fi.copy_(torch.tensor(ff.astype(np.int64)))
            g.replay()
            torch.cuda.synchronize()
            want, fo_want = expected_slots(wants, C, ws, ff, W, planar)
            assert np.array_equal(out.cpu().numpy().reshape(-1), want), planar
            assert np.array_equal(fo.cpu().numpy().astype(np.int64), fo_want), planar
    corpus.check()


# ------------------------------------------------------------------------------------------------ GPU: verdicts on random VBR size codes

@pytest.mark.gpu
def test_random_vbr_size_codes_verdicts_agree(ctx, lctx):
    """Seeded size codes (0..m, m cycling 0..3), so that some chunks ask for more residual bits than they hold or for more than
    8 bits a sample.  oracle.sea_decode, ctx.sea_decode, ctx.decode_batch and corpus creation agree on whether the stream is
    valid, the GPU calls on the error code; accepted streams decode, and window, as the oracle does."""
    n_ok = n_bad = 0
    for case in range(48):
        C = 1 + case % 2
        rate = (2.5, 4.5, 6.5, 7.3)[(case // 2) % 4]
        base = base_stream(C, rate, 4, True, N=1000, frames=3000 + 77 * case % 1000)
        f = craft(base, None, seed=case, size_codes=(case // 8) % 4)
        verdicts = []
        try:
            want = O.sea_decode(f).samples
            verdicts.append(0)
        except O.OracleError:
            want = None
            verdicts.append(None)

        def code(fn):
            try:
                fn()
                return 0
            except api.SeaError as e:
                return e.code

        got = {}
        verdicts.append(code(lambda: got.setdefault("one", ctx.sea_decode(f).samples)))
        verdicts.append(code(lambda: got.setdefault("batch", [d.samples for d in ctx.decode_batch([f] * 3)])))
        packed = Packed([f, f])
        verdicts.append(code(lambda: got.setdefault("corpus", packed.corpus(lctx))))
        if want is not None:
            assert verdicts[1:] == [0, 0, 0], (case, verdicts)
            assert np.array_equal(got["one"], want), case
            assert all(np.array_equal(g, want) for g in got["batch"]), case
            rng = np.random.default_rng(case)
            for W in (1, 999, 2500):
                for planar in (False, True):
                    ws, ff = windows(rng, got["corpus"].stream_frames, 12, W, 1000)
                    g, fo = run_async(got["corpus"], ws, ff, W, planar)
                    w, fo_want = expected_slots([want, want], C, ws, ff, W, planar)
                    assert np.array_equal(fo, fo_want) and np.array_equal(g, w), (case, W, planar)
            got["corpus"].close()
            n_ok += 1
        else:
            assert verdicts[1] != 0 and verdicts[1] == verdicts[2] == verdicts[3], (case, verdicts)
            n_bad += 1
    assert n_ok >= 10 and n_bad >= 10, (n_ok, n_bad)


@pytest.mark.gpu
def test_a_corpus_outlives_its_context_safely():
    """A corpus whose context is closed first, or finalised first by the garbage collector in a reference cycle (which is what
    a failing test's traceback makes of a corpus and its context), is released without a call into the destroyed context."""
    import gc

    f = base_stream(2, 3, 4)
    c = S.Context(0)
    corpus = Packed([f]).corpus(c)
    c.close()
    assert not corpus._h.value
    corpus.close()
    for _ in range(3):
        c = S.Context(0)
        cycle = [c, Packed([f]).corpus(c)]
        cycle.append(cycle)
        del c, cycle
        gc.collect()
