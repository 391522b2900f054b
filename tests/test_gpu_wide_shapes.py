"""Every encode and decode route on the wide shapes of tests/wide_shapes.py (up to 255 channels, scale_factor_bits 1-8, blocks
of up to 255 frames, chunks near 65535 bytes), against the CPU oracle: byte for byte for the encoder (and the VBR tie counts),
sample for sample for the decoder, float32 planar = int16 / 32768.  SEA_B200_DEBUG_LAUNCH names the kernels each call ran, so
the tests also check that the warp-per-chunk decode kernel really takes 9-32 channels, that the generic kernel takes the rest,
and that the encoder launches with the threads and shared memory the host restatement predicts."""
import functools
import io
import re

import numpy as np
import pytest

import enc_crafted as G
import sea_codec_b200 as S
import wide_shapes as W
from oracle import sea_oracle as O
from test_gpu_adversarial import PATTERNS, check_corpus, craft, expected_slots
from util import SENTINEL, Packed, windows

pytestmark = pytest.mark.gpu

SHAPES = [pytest.param(sh, id=sh.id) for sh in W.SHAPES]
DECODABLE = [pytest.param(sh, id=sh.id) for sh in W.SHAPES if sh.decodable]
MENU = ("sq10", "noise", "zero", "sq40", "hi", "tone", "lo", "sq2", "dramp")


def crafted_pcm(frames, channels, seed):
    """enc_crafted blocks of 20 frames: full-scale squares, noise, held extremes, silence and a quiet tone rotating over the
    channels, channel 1 the phase-inverted copy of channel 0, and a partial last block."""
    nb = -(-frames // G.BLOCK)
    recipe = []
    for i in range(nb):
        names = tuple("inv" if c == 1 else MENU[(i + c + seed) % len(MENU)] for c in range(channels))
        ent = names if channels > 1 else names[0]
        recipe.append(ent if (i + 1) * G.BLOCK <= frames else [frames - i * G.BLOCK, ent])
    return G.pcm(recipe, channels, seed)


@functools.lru_cache(maxsize=None)
def inputs(shape):
    """Two streams per shape (the second a little shorter, with its own ragged end) and the oracle's encodes and tie counts."""
    xs = [crafted_pcm(shape.frames, shape.channels, 0), crafted_pcm(shape.frames - shape.F - 3, shape.channels, 5)]
    refs = [O.sea_encode(x, 44100, shape.channels, shape.settings(), return_ties=True) for x in xs]
    return xs, [r[0] for r in refs], [r[1] for r in refs]


def enc_settings(shape):
    return S.EncoderSettings(residual_bits=shape.bits, vbr=shape.vbr, scale_factor_bits=shape.s, scale_factor_frames=shape.F,
                             frames_per_chunk=shape.N)


@pytest.fixture
def debug(monkeypatch, capfd):
    """Turns on SEA_B200_DEBUG_LAUNCH; the returned function runs a call and returns (result, [launch lines])."""
    monkeypatch.setenv("SEA_B200_DEBUG_LAUNCH", "1")
    capfd.readouterr()

    def run(fn):
        r = fn()
        return r, [ln for ln in capfd.readouterr().err.splitlines() if re.match(r"^\w+(<[-\d,]+>)?: ", ln)]

    return run


def kernels(lines):
    return [re.match(r"^(\w+)", ln).group(1) for ln in lines]


# ------------------------------------------------------------------------------------------------ encode

@pytest.mark.parametrize("shape", SHAPES)
def test_every_encode_route_matches_the_oracle(ctx, debug, monkeypatch, shape):
    """sea_encode (with the launch the restatement predicts), encode_batch unsliced and in forced one-chunk slices,
    encode_batch_device and the streaming encoder; the VBR tie counts, total and per stream."""
    import torch

    C, st = shape.channels, enc_settings(shape)
    xs, refs, ties = inputs(shape)
    p = shape.plan()
    for x, r, t in zip(xs, refs, ties):
        got, lines = debug(lambda: ctx.sea_encode(x, 44100, C, st))
        assert got == r
        assert not shape.vbr or ctx.last_vbr_ties == t
        want = W.encode_launch(p, [x.size // C])
        m = re.match(r"encode_kernel<(-?\d+),(\d+)>: (\d+) channels, (\d+) threads/CTA, (\d+) B smem, 1 CTAs", lines[0])
        assert len(lines) == 1 and m, lines
        assert (int(m.group(1)) >= 0) == want.fast and int(m.group(4)) == want.T and int(m.group(5)) == want.smem, (lines, want)
    for k in ("0", "1"):
        monkeypatch.setenv("SEA_B200_ENC_SLICE", k)
        assert ctx.encode_batch(xs, 44100, C, st) == refs, k
        assert not shape.vbr or list(ctx.last_vbr_ties_per_stream(len(xs))) == ties, k
    monkeypatch.delenv("SEA_B200_ENC_SLICE")
    frames = np.array([x.size // C for x in xs])
    pcm_off = np.concatenate([[0], np.cumsum(frames * C)[:-1]])
    pcm = torch.from_numpy(np.concatenate(xs)).to("cuda:0")
    stride = (max(ctx.encode_bound(int(f), C, st) for f in frames) + 15) // 16 * 16
    out = torch.zeros(len(xs) * stride, dtype=torch.uint8, device="cuda:0")
    torch.cuda.synchronize()
    lens = ctx.encode_batch_device(pcm.data_ptr(), pcm_off, frames, 44100, C, st, out.data_ptr(), np.arange(len(xs)) * stride)
    host = out.cpu().numpy()
    for i, r in enumerate(refs):
        assert host[i * stride: i * stride + int(lens[i])].tobytes() == r, i
    assert not shape.vbr or list(ctx.last_vbr_ties_per_stream(len(xs))) == ties
    sink = io.BytesIO()
    enc = S.SeaEncoder(C, 44100, xs[0].size // C, st, io.BytesIO(xs[0].astype("<i2").tobytes()), sink, ctx=ctx)
    while enc.encode_frame():
        pass
    enc.finalize()
    assert sink.getvalue() == refs[0]


# ------------------------------------------------------------------------------------------------ decode

@functools.lru_cache(maxsize=None)
def decode_set(shape):
    """The encoder's two streams and three adversarial payloads of the first (patterns rotating over the shapes)."""
    _, refs, _ = inputs(shape)
    k = W.SHAPES.index(shape)
    pats = [PATTERNS[(k + i) % len(PATTERNS)] for i in range(3)]
    files = refs + [craft(refs[0], pat, seed=17 * k + i) for i, pat in enumerate(pats)]
    return files, [O.sea_decode(f).samples for f in files]


def window_slots(ctx, packed, C, ws, ff, W_, planar):
    """decode_windows_device into slots at odd offsets 3 elements apart in a sentinel-filled buffer; checks the gaps."""
    import torch

    n, z = len(ws), W_ * C
    offs = np.arange(n, dtype=np.uint64) * (z + 3) + 1
    total = int(offs[-1]) + z + 5
    out = torch.full((total,), SENTINEL, dtype=torch.float32 if planar else torch.int16, device="cuda")
    torch.cuda.synchronize()
    fo = ctx.decode_windows_device(packed.buf.data_ptr(), packed.offs, packed.lens, packed.headers, ws, ff, np.full(n, W_),
                                   out.data_ptr(), offs, float32_planar=planar)
    host = out.cpu().numpy()
    inside = np.zeros(total, dtype=bool)
    for o in offs:
        inside[int(o): int(o) + z] = True
    assert np.all(host[~inside] == SENTINEL), "a byte outside the slots was written"
    return np.concatenate([host[int(o): int(o) + z] for o in offs]), fo.astype(np.int64)


@pytest.fixture(scope="module")
def lctx():
    c = S.Context(0)
    yield c
    import torch

    torch.cuda.synchronize()


@pytest.mark.parametrize("shape", DECODABLE)
def test_every_decode_route_matches_the_oracle(ctx, lctx, debug, monkeypatch, shape):
    """Each encoder-made stream and three adversarial payloads through the warp-per-chunk kernel (where it takes the geometry)
    and the throughput route, decode_batch plain and pipelined in small groups, decode_range, decode_windows_device (int16 and
    planar), a generic-route corpus with a CUDA-graph replay, and the streaming decoder."""
    import torch

    C, N = shape.channels, shape.N
    files, wants = decode_set(shape)
    p = shape.plan()
    lat = W.latency_smem(p.full_chunk_bytes, N, C) > 0
    for env in ("1", "0"):
        monkeypatch.setenv("SEA_B200_DEC_LATENCY", env)
        route = W.decode_route(C, N, p.full_chunk_bytes, shape.F, shape.s, p.hdr_bits, shape.vbr, 1, env)
        assert (route == "latency") == (env == "1" and lat)
        for f, w in zip(files, wants):
            got, lines = debug(lambda: ctx.sea_decode(f).samples)
            assert np.array_equal(got, w), env
            assert kernels(lines) == ["decode_" + route], (env, lines)
    monkeypatch.setenv("SEA_B200_DEC_LATENCY", "0")
    got, lines = debug(lambda: ctx.decode_batch(files * 2))
    assert all(np.array_equal(g.samples, wants[i % len(files)]) for i, g in enumerate(got))
    assert set(kernels(lines)) == {"decode_generic"} or C < 9, lines
    monkeypatch.setenv("SEA_B200_DEC_GROUP_SAMPLES", str(max(1, wants[0].size // 2)))
    got = ctx.decode_batch(files * 2)
    assert all(np.array_equal(g.samples, wants[i % len(files)]) for i, g in enumerate(got))
    monkeypatch.delenv("SEA_B200_DEC_GROUP_SAMPLES")

    rng = np.random.default_rng(C * 1000 + shape.s * 100 + shape.F)
    for f, w in zip(files, wants):
        frames = w.size // C
        for first, n in ((0, 1), (N - 1, 2), (N, N), (int(rng.integers(0, frames)), int(rng.integers(1, 2 * N))), (frames - 5, 100)):
            assert np.array_equal(ctx.decode_range(f, first, n).samples, w[first * C: (first + n) * C]), (first, n)

    packed = Packed(files, shift=1)
    stream_frames = np.array([w.size // C for w in wants])
    for W_ in (1, 33, N + 7):
        for planar in (False, True):
            ws, ff = windows(rng, stream_frames, 12, W_, N)
            got, fo = window_slots(ctx, packed, C, ws, ff, W_, planar)
            want, fo_want = expected_slots(wants, C, ws, ff, W_, planar)
            assert np.array_equal(fo, fo_want), (W_, planar)
            assert np.array_equal(got, want), (W_, planar, np.flatnonzero(got != want)[:8])

    (_, lines) = debug(lambda: check_corpus(lctx, files, wants, N, "generic", (1, N + 1), rng, n_windows=8))
    assert "corpus_generic" in kernels(lines)
    corpus = Packed(files, shift=2).corpus(lctx)
    n_win, W_ = 8, N + 3
    for planar in (False, True):
        si = torch.zeros(n_win, dtype=torch.int64, device="cuda")
        fi = torch.zeros(n_win, dtype=torch.int64, device="cuda")
        fo = torch.zeros(n_win, dtype=torch.int32, device="cuda")
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            corpus.decode_windows(si, fi, W_, float32_planar=planar, frames_out=fo)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            out = corpus.decode_windows(si, fi, W_, float32_planar=planar, frames_out=fo)
        ws, ff = windows(rng, corpus.stream_frames, n_win, W_, N)
        si.copy_(torch.tensor(ws.astype(np.int64)))
        fi.copy_(torch.tensor(ff.astype(np.int64)))
        g.replay()
        torch.cuda.synchronize()
        want, fo_want = expected_slots(wants, C, ws, ff, W_, planar)
        assert np.array_equal(out.cpu().numpy().reshape(-1), want), planar
        assert np.array_equal(fo.cpu().numpy().astype(np.int64), fo_want), planar
    corpus.check()
    corpus.close()

    for f, w in zip(files, wants):
        for step in (lambda d: d.decode_frame(), lambda d: d.decode_frames(3)):
            sink = io.BytesIO()
            dec = S.SeaDecoder(io.BytesIO(f), sink, ctx=ctx)
            while step(dec):
                pass
            dec.close()
            assert np.array_equal(np.frombuffer(sink.getvalue(), dtype="<i2"), w)


def test_mixed_channel_batch_matches_the_oracle(ctx, debug):
    """One decode_batch of 2, 9, 32 and 255 channels (encoder-made and crafted): not uniform, so every chunk runs on the generic
    kernel."""
    picks = [next(sh for sh in W.SHAPES if sh.channels == c and sh.decodable) for c in (9, 32, 255)]
    files, wants = [], []
    for sh in picks:
        f, w = decode_set(sh)
        files += [f[0], f[2]]
        wants += [w[0], w[2]]
    two = O.sea_encode(crafted_pcm(3000, 2, 1), 44100, 2, O.make_settings(3.0, frames_per_chunk=400))
    files.insert(1, two)
    wants.insert(1, O.sea_decode(two).samples)
    got, lines = debug(lambda: ctx.decode_batch(files))
    for i, (g, w) in enumerate(zip(got, wants)):
        assert np.array_equal(g.samples, w), i
    assert kernels(lines) == ["decode_generic"], lines
