"""GPU tests of sea_b200_decode_windows_device: many frame windows of device-resident .sea streams in one call.  The contract:
every slot starts with exactly what decode_range returns for its window (frames_out[w] frames), the rest of the slot is zero,
and nothing outside the slots is written.  Expected values are ctx.decode_range of the same bytes, or the oracle's full decode
sliced."""
import ctypes as C

import numpy as np
import pytest

import sea_codec_b200 as S
from sea_codec_b200 import api, synth

pytestmark = pytest.mark.gpu

N = 5120
SENTINEL = -12345
F_STEREO = N * 6 + 777  # six full chunks and a partial one


def _encode(ctx, seed, frames, ch, rate=44100, **kw):
    return ctx.sea_encode(synth.gen_stream(seed, frames, ch, rate), rate, ch, S.EncoderSettings(**kw))


class Corpus:
    """.sea streams packed into one device buffer; `shift` moves every stream off 16-byte alignment."""

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
        self.channels = [S.parse_header(f).channels for f in self.files]


def run(ctx, corpus, wins, planar=False, skip_metadata=False, out_offsets=None):
    """Decodes `wins` = [(stream, first, n)] into a sentinel-filled buffer; checks nothing outside the slots changed and returns
    (frames_out, [slot arrays])."""
    import torch

    sizes = [n * corpus.channels[s] for s, _, n in wins]
    if out_offsets is None:
        out_offsets = np.concatenate([[0], np.cumsum(sizes)[:-1]]).astype(np.uint64)
    total = int(max(int(o) + z for o, z in zip(out_offsets, sizes))) + 37
    out = torch.full((total,), SENTINEL, dtype=torch.float32 if planar else torch.int16, device="cuda")
    torch.cuda.synchronize()
    got = ctx.decode_windows_device(corpus.buf.data_ptr(), corpus.offs, corpus.lens, corpus.headers, [w[0] for w in wins],
                                    [w[1] for w in wins], [w[2] for w in wins], out.data_ptr(), out_offsets, float32_planar=planar,
                                    skip_metadata=skip_metadata)
    host = out.cpu().numpy()
    outside = np.ones(total, dtype=bool)
    for o, z in zip(out_offsets, sizes):
        outside[int(o): int(o) + z] = False
    assert np.all(host[outside] == SENTINEL), "a byte outside the slots was written"
    return got, [host[int(o): int(o) + z] for o, z in zip(out_offsets, sizes)]


def check_against_range(ctx, corpus, wins, got, slots, skip_metadata=False):
    for (s, first, n), fo, slot in zip(wins, got, slots):
        want = ctx.decode_range(corpus.files[s], first, n, skip_metadata=skip_metadata).samples
        assert int(fo) * corpus.channels[s] == want.size, (s, first, n)
        assert np.array_equal(slot[: want.size], want), (s, first, n)
        assert not np.any(slot[want.size:]), (s, first, n)


def check_planar(corpus, wins, slots_i16, slots_f32):
    """float32 planar = the int16 result / 32768, channel row by channel row."""
    for (s, _, n), a, b in zip(wins, slots_i16, slots_f32):
        ch = corpus.channels[s]
        rows = a.reshape(n, ch).T.astype(np.float32) / np.float32(32768.0)
        assert np.array_equal(b.reshape(ch, n), rows), (s, n)


def edge_windows(s, frames):
    """Inside one chunk, straddling a boundary, starting on one, from frame 0, the whole stream, ending at its end, running past
    it, starting past it, empty, and odd starts / lengths."""
    return [(s, 100, 1000), (s, N - 300, 700), (s, N, N), (s, 2 * N, 3), (s, 0, 4000), (s, 0, frames), (s, frames - 2000, 2000),
            (s, frames - 500, 3000), (s, frames, 5), (s, frames + 10, 100), (s, 1234, 0), (s, 7, 1), (s, N - 1, 2),
            (s, 3 * N + 11, 2 * N + 5), (s, 1 << 40, 9)]


def random_windows(rng, corpus, count, max_len=3 * N):
    wins = []
    for _ in range(count):
        s = int(rng.integers(0, len(corpus.files)))
        frames = S.parse_header(corpus.files[s]).total_frames
        first = int(rng.integers(0, frames + 200))
        wins.append((s, first, int(rng.integers(1, max_len))))
    return wins


SHAPES = {
    "stereo_cbr3": (2, F_STEREO, dict(residual_bits=3.0)),
    "stereo_vbr35": (2, F_STEREO, dict(residual_bits=3.5, vbr=True)),
    "mono_cbr3": (1, F_STEREO, dict(residual_bits=3.0)),
    "ch3_cbr4": (3, N * 4 + 1001, dict(residual_bits=4.0)),
    "ch8_cbr4": (8, N * 4 + 999, dict(residual_bits=4.0)),
    "stereo_sfb3": (2, F_STEREO, dict(residual_bits=3.0, scale_factor_bits=3)),
    "stereo_sfb5": (2, F_STEREO, dict(residual_bits=3.0, scale_factor_bits=5)),
    "stereo_whole_chunks": (2, N * 5, dict(residual_bits=3.0)),
}


@pytest.mark.parametrize("shape", sorted(SHAPES))
def test_windows_equal_decode_range(ctx, shape):
    ch, frames, kw = SHAPES[shape]
    corpus = Corpus([_encode(ctx, 300 + i, frames, ch, **kw) for i in range(2)])
    wins = edge_windows(0, frames) + edge_windows(1, frames)[::-1] + random_windows(np.random.default_rng(ch * 7 + frames), corpus, 12)
    got, slots = run(ctx, corpus, wins)
    check_against_range(ctx, corpus, wins, got, slots)
    got_f, slots_f = run(ctx, corpus, wins, planar=True)
    assert np.array_equal(got_f, got)
    check_planar(corpus, wins, slots, slots_f)


def _mixed_corpus(ctx):
    files = [_encode(ctx, 400, F_STEREO, 2, residual_bits=3.0), _encode(ctx, 401, N * 3 + 5, 8, 48000, residual_bits=4.0),
             _encode(ctx, 402, F_STEREO, 1, residual_bits=3.0), _encode(ctx, 403, F_STEREO, 2, residual_bits=3.5, vbr=True),
             _encode(ctx, 404, N * 4 + 77, 3, residual_bits=4.0, scale_factor_bits=5), _encode(ctx, 405, F_STEREO - 99, 2, residual_bits=5.0)]
    return Corpus(files, shift=3)


def _check_mixed_and_uniform(ctx, oracle):
    """Windows of streams with different settings and channel counts in one call, then a uniform stereo batch (the geometry the
    specialised kernels take) with many windows of one stream; expected values from the oracle's full decode, sliced."""
    rng = np.random.default_rng(11)
    for corpus in (_mixed_corpus(ctx), Corpus([_encode(ctx, 500 + i, F_STEREO, 2, residual_bits=3.0) for i in range(3)])):
        full = [oracle.sea_decode(f).samples for f in corpus.files]
        wins = random_windows(rng, corpus, 120) + [(0, int(f), 2 * N + 17) for f in rng.integers(0, F_STEREO, 60)]
        for planar in (False, True):
            got, slots = run(ctx, corpus, wins, planar=planar)
            for (s, first, n), fo, slot in zip(wins, got, slots):
                ch = corpus.channels[s]
                want = full[s].reshape(-1, ch)[first: first + n]
                assert int(fo) == want.shape[0]
                if planar:
                    pad = np.zeros((n, ch), dtype=np.float32)
                    pad[: want.shape[0]] = want.astype(np.float32) / np.float32(32768.0)
                    assert np.array_equal(slot.reshape(ch, n), pad.T), (s, first, n)
                else:
                    assert np.array_equal(slot[: want.size], want.reshape(-1)) and not np.any(slot[want.size:]), (s, first, n)


def test_mixed_batch_default_route(ctx, oracle):
    _check_mixed_and_uniform(ctx, oracle)


@pytest.mark.latency_kernel
def test_mixed_batch_latency_route(ctx, oracle):
    _check_mixed_and_uniform(ctx, oracle)


def test_mixed_batch_full_width_ctas(ctx, oracle, monkeypatch):
    monkeypatch.setenv("SEA_B200_FULL_CTAS", "1")
    _check_mixed_and_uniform(ctx, oracle)


@pytest.mark.parametrize("planar", [False, True])
def test_slots_in_descending_order_with_gaps(ctx, planar):
    corpus = Corpus([_encode(ctx, 600, F_STEREO, 2, residual_bits=3.0), _encode(ctx, 601, N * 2 + 3, 3, residual_bits=4.0)])
    wins = [(0, 5, 1001), (1, 77, 333), (0, N - 3, 17), (1, N * 2, 50), (0, 0, 9), (1, 1, 1), (0, F_STEREO - 4, 13)]
    sizes = [n * corpus.channels[s] for s, _, n in wins]
    offs, o = [], 3
    for z in sizes[::-1]:  # the last window gets the lowest offset; odd gaps between the slots
        offs.append(o)
        o += z + 5
    offs = np.array(offs[::-1], dtype=np.uint64)
    got, slots = run(ctx, corpus, wins, planar=planar, out_offsets=offs)
    if planar:
        got_i, slots_i = run(ctx, corpus, wins)
        assert np.array_equal(got, got_i)
        check_planar(corpus, wins, slots_i, slots)
    else:
        check_against_range(ctx, corpus, wins, got, slots)


def test_multi_group_scratch_gives_the_same_result(ctx, monkeypatch):
    corpus = Corpus([_encode(ctx, 700 + i, F_STEREO, 2, residual_bits=3.0) for i in range(3)])
    wins = random_windows(np.random.default_rng(5), corpus, 40) + [(1, N * 6 + 100, 5), (2, 0, 0)]
    got, slots = run(ctx, corpus, wins)
    n0 = ctx.launch_count
    run(ctx, corpus, wins)
    one_group = ctx.launch_count - n0
    monkeypatch.setenv("SEA_B200_WIN_SCRATCH_SAMPLES", "30000")  # a few windows per group; larger windows alone
    for planar in (False, True):
        n0 = ctx.launch_count
        got_g, slots_g = run(ctx, corpus, wins, planar=planar)
        assert ctx.launch_count - n0 > 4 * one_group, "the scratch cap did not split the call into groups"
        assert np.array_equal(got_g, got)
        if planar:
            check_planar(corpus, wins, slots, slots_g)
        else:
            assert all(np.array_equal(a, b) for a, b in zip(slots, slots_g))
    check_against_range(ctx, corpus, wins, got, slots)


def test_skip_metadata(ctx):
    sea = _encode(ctx, 800, F_STEREO, 2, residual_bits=3.0)
    meta = b"title=x\nartist=y"
    with_meta = sea[:18] + len(meta).to_bytes(4, "little") + meta + sea[22:]
    corpus = Corpus([with_meta, sea])
    wins = [(0, 6000, 3000), (0, 0, N), (0, F_STEREO - 10, 50), (1, 6000, 3000)]
    got, slots = run(ctx, corpus, wins, skip_metadata=True)
    check_against_range(ctx, corpus, wins, got, slots, skip_metadata=True)
    assert np.array_equal(slots[0], slots[3])


def test_streaming_header_counts_whole_chunks_only(ctx):
    sea = _encode(ctx, 900, F_STEREO, 2, residual_bits=3.0)
    streaming = sea[:14] + b"\x00\x00\x00\x00" + sea[18:]
    corpus = Corpus([streaming])
    wins = [(0, 100, 2000), (0, N * 6 - 100, 1000), (0, N * 6, 100), (0, N * 6 + 5, 10), (0, 0, F_STEREO)]
    got, slots = run(ctx, corpus, wins)
    check_against_range(ctx, corpus, wins, got, slots)
    assert list(got) == [2000, 100, 0, 0, N * 6]


def test_errors(ctx):
    sea = _encode(ctx, 1000, F_STEREO, 2, residual_bits=3.0)
    corpus = Corpus([sea])
    import torch

    out = torch.zeros(64, dtype=torch.int16, device="cuda")
    with pytest.raises(S.SeaError) as e:
        ctx.decode_windows_device(corpus.buf.data_ptr(), corpus.offs, corpus.lens, corpus.headers, [0, 1], [0, 0], [10, 10],
                                  out.data_ptr(), [0, 20])
    assert e.value.code == api.ERR_INVALID_PARAMETERS
    ws, ff, nf, oo, fo = (np.zeros(1, dtype=np.uint32), np.zeros(1, dtype=np.uint64), np.full(1, 10, dtype=np.uint32),
                          np.zeros(1, dtype=np.uint64), np.zeros(1, dtype=np.uint64))
    rc = S.lib().sea_b200_decode_windows_device(ctx._h, 1, C.c_void_p(corpus.buf.data_ptr()), corpus.offs.ctypes.data,
                                                corpus.lens.ctypes.data, corpus.headers.ctypes.data, 1, ws.ctypes.data, ff.ctypes.data,
                                                nf.ctypes.data, 4, C.c_void_p(out.data_ptr()), oo.ctypes.data, fo.ctypes.data)
    assert rc == api.ERR_INVALID_PARAMETERS
    # a corrupted chunk (k = 3): inside a window the call fails as decode_range does; covered by no window it changes nothing
    hdr = S.parse_header(sea)
    p = 22 + 3 * hdr.chunk_size
    for at, patch in ((p, b"\x07"), (p + 4, b"\xff" * 36)):  # the chunk type byte; the first scale factors
        bad = bytearray(sea)
        bad[at: at + len(patch)] = patch
        bad = bytes(bad)
        corpus = Corpus([sea, bad])
        inside = [(0, 0, 100), (1, 3 * N + 10, 100)]
        try:
            ctx.decode_range(bad, 3 * N + 10, 100)
            want_code = None
        except S.SeaError as err:
            want_code = err.code
        if want_code is None:  # the corruption still decodes: the window must hold what decode_range returns
            got, slots = run(ctx, corpus, inside)
            check_against_range(ctx, corpus, inside, got, slots)
        else:
            with pytest.raises(S.SeaError) as e:
                run(ctx, corpus, inside)
            assert e.value.code == want_code
        outside = [(1, 0, 2 * N), (1, 4 * N + 1, 3000), (0, 3 * N, 50)]
        got, slots = run(ctx, corpus, outside)
        check_against_range(ctx, corpus, outside, got, slots)
    # the type byte corruption is one decode_range rejects
    bad = bytearray(sea)
    bad[22 + 3 * hdr.chunk_size] = 7
    with pytest.raises(S.SeaError) as e:
        ctx.decode_range(bytes(bad), 3 * N, 10)
    assert e.value.code == api.ERR_INVALID_FRAME
