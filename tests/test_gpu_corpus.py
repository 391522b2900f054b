"""Tests of the registered corpus (sea_b200_corpus_*, Context.corpus / Corpus.decode_windows): fixed-length windows decoded from
device-side indices on the current stream.  The contract: every slot and frames_out are bit-identical to what
decode_windows_device writes for the same (stream, first frame, window length) with out_offsets = w * W * channels, nothing outside
the slots is written, a bad stream index zero-fills its slot and sets the status word, and the call captures in a CUDA graph.
The window-plan arithmetic the kernels evaluate on the device is checked against plan_range on the CPU."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import sea_codec_b200 as S
from sea_codec_b200 import api, synth
from util import ROOT, Packed, run_async, windows

N = 5120


# ------------------------------------------------------------------------------------------------ CPU: window plan

PLAN_SRC = r"""
#include "sea_format.cpp"
extern "C" int plan_pair(const uint8_t *hdr22, uint64_t len, uint64_t first, uint64_t n, int skip, uint64_t *out)
{
    sea_b200_header h;
    int rc = sea::parse_file_header(hdr22, 22, &h);
    if (rc) return rc;
    sea::RangePlan p;
    rc = sea::plan_range(h, len, first, n, skip != 0, &p);
    if (rc) return rc;
    const sea::WindowPlan w = sea::window_plan(p.file_frames, h.frames_per_chunk, first, n);
    const uint64_t v[6] = {p.k0, p.skip, p.want, w.k0, w.skip, w.want};
    for (int i = 0; i < 6; i++) out[i] = v[i];
    return 0;
}
"""


def test_window_plan_matches_plan_range(tmp_path):
    """window_plan (sea_common.cuh), which the corpus kernels evaluate per window, gives plan_range's k0 / skip / want over a
    seeded sweep: total_frames and streaming headers, metadata with and without the skip, truncated files, first frames at 0,
    mid-chunk, on a chunk boundary, at the last frame, past the end and near 2^64, window lengths 1, < N, = N, multiples of N and
    longer than the stream."""
    src = tmp_path / "plan.cpp"
    src.write_text(PLAN_SRC)
    so = tmp_path / "libplan.so"
    subprocess.run(["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-I" + os.path.join(ROOT, "sea_codec_b200", "csrc"), "-o", str(so),
                    str(src)], check=True)
    L = C.CDLL(str(so))
    L.plan_pair.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_int, C.c_void_p]
    rng = np.random.default_rng(2024)
    out = np.zeros(6, dtype=np.uint64)
    checked = 0
    for case in range(400):
        fpc = int(rng.choice([1, 7, 20, 1000, 5120, 65535]))
        cs = int(rng.integers(16, 5000))
        n_chunks = int(rng.integers(0, 12))
        meta = int(rng.choice([0, 0, 16, 300]))
        streaming = case % 4 == 0
        total = 0 if streaming else int(rng.integers(1, max(2, n_chunks * fpc + fpc)))
        body_len = n_chunks * cs + int(rng.choice([0, 0, 1, cs // 2, cs - 1]))  # whole chunks or a trailing partial one
        if case % 5 == 1:
            body_len = max(0, body_len - int(rng.integers(1, cs * 2)))  # truncated
        length = 22 + meta + body_len
        hdr = np.zeros(22, dtype=np.uint8)
        hdr[:4] = np.frombuffer(b"seac", dtype=np.uint8)
        hdr[4], hdr[5] = 1, int(rng.integers(1, 9))
        hdr[6:8] = np.frombuffer(np.uint16(cs).tobytes(), dtype=np.uint8)
        hdr[8:10] = np.frombuffer(np.uint16(fpc).tobytes(), dtype=np.uint8)
        hdr[10:14] = np.frombuffer(np.uint32(44100).tobytes(), dtype=np.uint8)
        hdr[14:18] = np.frombuffer(np.uint32(total).tobytes(), dtype=np.uint8)
        hdr[18:22] = np.frombuffer(np.uint32(meta).tobytes(), dtype=np.uint8)
        frames = max(total, n_chunks * fpc)
        firsts = [0, fpc // 2, fpc, 2 * fpc + 3, max(frames - 1, 0), frames, frames + 5, 2**64 - 1, 2**64 - fpc,
                  int(rng.integers(0, frames + 2))]
        lens = [1, max(fpc - 1, 1), fpc, 3 * fpc, frames + fpc + 1, int(rng.integers(1, 4 * fpc + 2)), 0]
        for skip in (0, 1):
            for first in firsts:
                for n in lens:
                    rc = L.plan_pair(hdr.ctypes.data, length, first, n, skip, out.ctypes.data)
                    if rc:
                        continue  # plan_range's own error (body past the end): no window plan
                    assert out[:3].tolist() == out[3:].tolist(), (case, skip, first, n, out.tolist())
                    checked += 1
    assert checked > 20000


# ------------------------------------------------------------------------------------------------ GPU helpers


@pytest.fixture(scope="module")
def lctx():
    """The corpora's own context: Corpus binds its context to torch's current stream (side streams included), which the
    session context of the other test modules must not see."""
    c = S.Context(0)
    yield c
    import torch

    torch.cuda.synchronize()


def _encode(ctx, seed, frames, ch, rate=44100, **kw):
    return ctx.sea_encode(synth.gen_stream(seed, frames, ch, rate), rate, ch, S.EncoderSettings(**kw))


def reference(ctx, packed, ch, ws, ff, W, planar, skip_metadata):
    """decode_windows_device's slots (out_offsets = w * W * ch) and frames_out for the same windows."""
    import torch

    n = len(ws)
    out = torch.zeros(max(n * W * ch, 1), dtype=torch.float32 if planar else torch.int16, device="cuda")
    torch.cuda.synchronize()
    fo = ctx.decode_windows_device(packed.buf.data_ptr(), packed.offs, packed.lens, packed.headers, ws, ff, np.full(n, W), out.data_ptr(),
                                   np.arange(n, dtype=np.uint64) * (W * ch), float32_planar=planar, skip_metadata=skip_metadata)
    return out[: n * W * ch].cpu().numpy(), fo.astype(np.int64)


SHAPES = {
    "mono_cbr3": (1, dict(residual_bits=3.0)),
    "stereo_cbr3": (2, dict(residual_bits=3.0)),
    "stereo_vbr35": (2, dict(residual_bits=3.5, vbr=True)),
    "ch3_cbr4": (3, dict(residual_bits=4.0)),
    "ch8_cbr4": (8, dict(residual_bits=4.0)),
    "stereo_sfb3": (2, dict(residual_bits=3.0, scale_factor_bits=3)),
    "stereo_sfb5": (2, dict(residual_bits=3.0, scale_factor_bits=5)),
    "mono_vbr3_sfb3": (1, dict(residual_bits=3.0, vbr=True, scale_factor_bits=3)),
}
SHAPE_FRAMES = [N * 3 + 777, N * 2, N + 1234, N * 5 + 4097]
FAST_OK = {"mono_cbr3", "stereo_cbr3", "stereo_sfb3", "stereo_sfb5"}


def shape_files(ctx, ch, kw, seed):
    """A partial last chunk, whole chunks only, a short one, and a longer one (every stream longer than a chunk: a stream of one
    partial chunk has its own chunk_size, and the corpus would leave the fast route)."""
    return [_encode(ctx, seed + i, f, ch, **kw) for i, f in enumerate(SHAPE_FRAMES)]


def check_equal(ctx, packed, corpus, ws, ff, W, planar, skip_metadata=False):
    got, fo = run_async(corpus, ws, ff, W, planar)
    want, fo_want = reference(ctx, packed, corpus.channels, ws, ff, W, planar, skip_metadata)
    assert np.array_equal(fo, fo_want), (W, planar)
    assert np.array_equal(got, want), (W, planar, np.flatnonzero(got != want)[:8])


@pytest.mark.gpu
@pytest.mark.parametrize("route", ["auto", "generic", "fast"])
@pytest.mark.parametrize("shape", sorted(SHAPES))
def test_async_windows_equal_decode_windows_device(ctx, lctx, shape, route, monkeypatch):
    ch, kw = SHAPES[shape]
    if route == "fast" and shape not in FAST_OK:
        pytest.skip("the corpus does not qualify for the fast route")
    if route != "auto":
        monkeypatch.setenv("SEA_B200_CORPUS_ROUTE", route)
    packed = Packed(shape_files(ctx, ch, kw, 40 + ch), shift=3)
    corpus = packed.corpus(lctx)
    if route == "auto":
        assert corpus.route == ("fast" if shape in FAST_OK else "generic")
    else:
        assert corpus.route == route
    assert corpus.channels == ch
    assert corpus.stream_frames.tolist() == SHAPE_FRAMES
    rng = np.random.default_rng(len(shape) * 31 + len(route))
    for W in (1, N - 1, N, 3 * N + 7, 6 * N):  # 6N is longer than every stream
        for planar in (False, True):
            ws, ff = windows(rng, corpus.stream_frames, 37, W)
            check_equal(ctx, packed, corpus, ws, ff, W, planar)
    corpus.check()
    corpus.close()


@pytest.mark.gpu
@pytest.mark.parametrize("route", ["generic", "fast"])
def test_many_windows_on_one_stream_and_no_op_calls(ctx, lctx, route, monkeypatch):
    import torch

    monkeypatch.setenv("SEA_B200_CORPUS_ROUTE", route)
    packed = Packed([_encode(ctx, 7, N * 9 + 5, 2)], shift=5)
    corpus = packed.corpus(lctx)
    ws = np.zeros(500, dtype=np.uint32)
    ff = np.random.default_rng(3).integers(0, N * 9 + 100, size=500).astype(np.uint64)
    for planar in (False, True):
        check_equal(ctx, packed, corpus, ws, ff, 2 * N + 11, planar)
    empty = torch.zeros(0, dtype=torch.int64, device="cuda")
    launches = lctx.launch_count
    out = corpus.decode_windows(empty, empty, 1000)
    assert out.shape == (0, 1000, 2)
    one = torch.zeros(3, dtype=torch.int64, device="cuda")
    out = corpus.decode_windows(one, one, 0)
    assert out.shape == (3, 0, 2)
    assert lctx.launch_count == launches  # nothing enqueued
    corpus.check()


@pytest.mark.gpu
@pytest.mark.parametrize("route", ["generic", "fast"])
def test_streaming_header_and_metadata_skip(ctx, lctx, route, monkeypatch):
    monkeypatch.setenv("SEA_B200_CORPUS_ROUTE", route)
    sea = _encode(ctx, 11, N * 4 + 1500, 2)
    streaming = sea[:14] + b"\x00\x00\x00\x00" + sea[18:]  # the trailing partial chunk is not a frame source
    packed = Packed([streaming, sea])
    corpus = packed.corpus(lctx)
    assert corpus.stream_frames.tolist() == [N * 4, N * 4 + 1500]
    rng = np.random.default_rng(5)
    for planar in (False, True):
        ws, ff = windows(rng, corpus.stream_frames, 40, N + 333)
        check_equal(ctx, packed, corpus, ws, ff, N + 333, planar)
    meta = b"title=x\nartist=y"
    with_meta = sea[:18] + len(meta).to_bytes(4, "little") + meta + sea[22:]
    packed = Packed([with_meta, sea], shift=1)
    corpus = packed.corpus(lctx, skip_metadata=True)
    for planar in (False, True):
        ws, ff = windows(rng, corpus.stream_frames, 40, 2 * N)
        check_equal(ctx, packed, corpus, ws, ff, 2 * N, planar, skip_metadata=True)


@pytest.mark.gpu
@pytest.mark.parametrize("route", ["generic", "fast"])
def test_bad_stream_index_sets_status(ctx, lctx, route, monkeypatch):
    import torch

    monkeypatch.setenv("SEA_B200_CORPUS_ROUTE", route)
    packed = Packed([_encode(ctx, 20 + i, N * 3 + 100, 2) for i in range(3)])
    corpus = packed.corpus(lctx)
    ws = np.array([0, 1, 2, 0, 2], dtype=np.uint32)
    ff = np.array([10, N - 5, 2 * N, 0, 3 * N], dtype=np.uint64)
    W = N + 50
    want, fo_want = reference(ctx, packed, 2, ws, ff, W, False, False)
    for bad in (3, -1, 2**40):
        si = torch.tensor(ws.astype(np.int64), device="cuda")
        si[1] = bad
        fo = torch.zeros(5, dtype=torch.int32, device="cuda")
        out = corpus.decode_windows(si, torch.tensor(ff.astype(np.int64), device="cuda"), W, frames_out=fo)
        got = out.cpu().numpy().reshape(-1)
        slot = W * 2
        assert not np.any(got[slot: 2 * slot]) and int(fo[1]) == 0
        mask = np.ones(got.size, dtype=bool)
        mask[slot: 2 * slot] = False
        assert np.array_equal(got[mask], want[mask])
        assert np.array_equal(np.delete(fo.cpu().numpy(), 1), np.delete(fo_want, 1))
        assert int(corpus.status.item()) == api.ERR_INVALID_PARAMETERS
        with pytest.raises(S.SeaError) as e:
            corpus.check()
        assert e.value.code == api.ERR_INVALID_PARAMETERS
        assert int(corpus.status.item()) == 0
    # a status already non-zero is left as it is
    st = torch.tensor([-99], dtype=torch.int32, device="cuda")
    si = torch.tensor([5, 0], dtype=torch.int32, device="cuda")
    corpus.decode_windows(si, torch.zeros(2, dtype=torch.int64, device="cuda"), 100, status=st)
    assert int(st.item()) == -99


@pytest.mark.gpu
def test_mixed_chunk_geometry_takes_the_generic_route(ctx, lctx):
    """A stream of one partial chunk (its own chunk_size) and streams with another frames_per_chunk in one corpus."""
    files = [_encode(ctx, 70, 1234, 2), _encode(ctx, 71, N * 2 + 5, 2), _encode(ctx, 72, 3000 * 3 + 7, 2, frames_per_chunk=3000)]
    packed = Packed(files, shift=7)
    corpus = packed.corpus(lctx)
    assert corpus.route == "generic"
    rng = np.random.default_rng(12)
    for W in (1, 2999, 2 * N + 1):
        for planar in (False, True):
            ws, ff = windows(rng, corpus.stream_frames, 41, W)
            check_equal(ctx, packed, corpus, ws, ff, W, planar)


@pytest.mark.gpu
def test_create_errors(ctx, lctx):
    sea = _encode(ctx, 30, N * 5 + 10, 2)
    hdr = S.parse_header(sea)
    bad = bytearray(sea)
    bad[22 + 3 * hdr.chunk_size] = 7  # chunk 3's type byte
    packed = Packed([sea, bytes(bad)])
    with pytest.raises(S.SeaError) as e:
        packed.corpus(lctx)
    assert e.value.code == api.ERR_INVALID_FRAME
    assert "stream 1, chunk 3" in str(e.value)
    truncated = sea[: 22 + 2 * hdr.chunk_size + 40]  # chunk 2 cut short
    packed = Packed([sea, sea, truncated])
    with pytest.raises(S.SeaError) as e:
        packed.corpus(lctx)
    assert e.value.code == api.ERR_DOMAIN
    assert "stream 2, chunk 2" in str(e.value)
    mono = _encode(ctx, 31, N * 2, 1)
    with pytest.raises(S.SeaError) as e:
        Packed([sea, mono]).corpus(lctx)
    assert e.value.code == api.ERR_INVALID_PARAMETERS


@pytest.mark.gpu
def test_forcing_fast_on_a_corpus_that_does_not_qualify_fails(ctx, lctx, monkeypatch):
    monkeypatch.setenv("SEA_B200_CORPUS_ROUTE", "fast")
    with pytest.raises(S.SeaError) as e:
        Packed([_encode(ctx, 32, N * 2, 2, residual_bits=3.5, vbr=True)]).corpus(lctx)
    assert e.value.code == api.ERR_INVALID_PARAMETERS


@pytest.mark.gpu
@pytest.mark.parametrize("planar", [False, True])
def test_graph_capture_and_replay_with_new_indices(ctx, lctx, planar):
    import torch

    packed = Packed([_encode(ctx, 50 + i, N * 6 + 321 * i, 2) for i in range(4)], shift=2)
    corpus = packed.corpus(lctx)
    assert corpus.route == "fast"
    n, W = 64, 2 * N + 17
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
    rng = np.random.default_rng(9)
    for _ in range(3):
        ws, ff = windows(rng, corpus.stream_frames, n, W)
        si.copy_(torch.tensor(ws.astype(np.int64)))
        fi.copy_(torch.tensor(ff.astype(np.int64)))
        g.replay()
        torch.cuda.synchronize()
        want, fo_want = reference(ctx, packed, 2, ws, ff, W, planar, False)
        assert np.array_equal(out.cpu().numpy().reshape(-1), want)
        assert np.array_equal(fo.cpu().numpy().astype(np.int64), fo_want)
    corpus.check()


@pytest.mark.gpu
def test_side_stream_ordering(ctx, lctx):
    """Indices drawn on a side stream, decoded there and consumed there, with no explicit synchronise in between."""
    import torch

    packed = Packed([_encode(ctx, 60 + i, N * 8 + 99, 1) for i in range(3)])
    corpus = packed.corpus(lctx)
    s = torch.cuda.Stream()
    W, n = 3 * N, 256
    with torch.cuda.stream(s):
        gen = torch.Generator(device="cuda").manual_seed(1)
        idx = torch.randint(0, 3, (n,), device="cuda", generator=gen)
        span = corpus.stream_frames_cuda[idx] - W + 1
        first = (torch.rand(n, device="cuda", generator=gen) * span).long()
        out = corpus.decode_windows(idx, first, W, float32_planar=True)
        doubled = out * 2  # consumed on the same stream
    s.synchronize()
    want, fo_want = reference(ctx, packed, 1, idx.cpu().numpy().astype(np.uint32), first.cpu().numpy().astype(np.uint64), W, True, False)
    assert np.all(fo_want == W)
    assert np.array_equal(out.cpu().numpy().reshape(-1), want)
    assert np.array_equal(doubled.cpu().numpy().reshape(-1), want * 2)
