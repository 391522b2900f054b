"""GPU parity tests (-m gpu): the CUDA path, called through the C-ABI (ctypes), against the CPU oracle on the same seeded
inputs, against the committed golden fixtures, and through size-independent properties.  Bit-exact: integer/byte work."""
import io
import json
import os

import numpy as np
import pytest

import sea_codec_b200 as S
from sea_codec_b200 import api, synth
from util import ROOT, gen_test_signal, sha

pytestmark = pytest.mark.gpu
GOLD = os.path.join(ROOT, "tests", "golden")


def _settings_pair(oracle, **kw):
    return S.EncoderSettings(**kw), oracle.make_settings(**kw)


def _pcm_for(m):
    if m["gen"] == "synth":
        return synth.gen_stream(m["seed"], m["frames"], m["channels"], m["rate"])
    return gen_test_signal(m["channels"], m["frames"], m["rate"], m["seed"])


# ------------------------------------------------------------------------------------------------ golden fixtures

def test_golden_decode(ctx):
    meta = json.load(open(os.path.join(GOLD, "golden.json")))
    for name, m in meta.items():
        gold = open(os.path.join(GOLD, name + ".sea"), "rb").read()
        dec = ctx.sea_decode(gold)
        assert dec.channels == m["channels"] and dec.sample_rate == m["rate"]
        assert dec.samples.size == m["frames"] * m["channels"], name
        assert sha(dec.samples) == m["dec_sha"], name


def test_golden_encode(ctx):
    meta = json.load(open(os.path.join(GOLD, "golden.json")))
    for name, m in meta.items():
        pcm = _pcm_for(m)
        assert sha(pcm) == m["pcm_sha"]
        enc = ctx.sea_encode(pcm, m["rate"], m["channels"], S.EncoderSettings(**m["settings"]))
        gold = open(os.path.join(GOLD, name + ".sea"), "rb").read()
        assert len(enc) == len(gold), name
        assert enc == gold, name
        assert ctx.last_vbr_ties == 0


# ------------------------------------------------------------------------------------------------ decode vs oracle

@pytest.mark.parametrize("channels", [1, 2, 3, 8])
@pytest.mark.parametrize("bits", [1, 2, 3, 4, 5, 6, 7, 8])
def test_decode_cbr_matches_oracle(ctx, oracle, channels, bits):
    frames = 5120 * 2 + 777
    pcm = gen_test_signal(channels, frames, seed=channels * 16 + bits)
    enc = oracle.sea_encode(pcm, 44100, channels, oracle.make_settings(float(bits)))
    ref = oracle.sea_decode(enc).samples
    got = ctx.sea_decode(enc)
    assert got.channels == channels and np.array_equal(got.samples, ref)


@pytest.mark.parametrize("channels,bits", [(1, 1.5), (1, 3.0), (2, 2.0), (2, 3.0), (2, 4.5), (2, 7.3), (3, 3.5), (8, 5.0)])
def test_decode_vbr_matches_oracle(ctx, oracle, channels, bits):
    frames = 5120 * 2 + 1333
    pcm = synth.gen_stream(channels + int(bits * 10), frames, channels, 48000)
    enc = oracle.sea_encode(pcm, 48000, channels, oracle.make_settings(bits, True))
    ref = oracle.sea_decode(enc).samples
    got = ctx.sea_decode(enc)
    assert np.array_equal(got.samples, ref)


@pytest.mark.parametrize("sfb,sff,fpc", [(3, 20, 5120), (5, 20, 5120), (4, 10, 1000), (4, 5, 200), (2, 16, 4096), (6, 32, 320)])
def test_decode_other_geometry(ctx, oracle, sfb, sff, fpc):
    for channels, vbr, bits in ((2, False, 3.0), (1, True, 3.0), (2, True, 4.0)):
        pcm = gen_test_signal(channels, fpc * 3 + sff + 3, seed=sfb)
        st = oracle.make_settings(bits, vbr, sfb, sff, fpc)
        enc = oracle.sea_encode(pcm, 44100, channels, st)
        try:
            ref = oracle.sea_decode(enc).samples
        except oracle.OracleError as e:
            # e.g. N=200, F=5 VBR: base = floor(bits) - 2, the 2-bit size code wraps (chunk.rs:248 masks in release builds) and
            # the reference cannot decode its own file; the GPU path must refuse the same input instead of inventing PCM
            assert e.code == oracle.ERR_PANIC
            with pytest.raises(S.SeaError) as ge:
                ctx.sea_decode(enc)
            assert ge.value.code == api.ERR_DOMAIN
            continue
        assert np.array_equal(ctx.sea_decode(enc).samples, ref)


def test_decode_ragged_lengths(ctx, oracle):
    """tests/test.rs:8-33 restated: lengths straddling multiples of 100, channels 1..3; plus empty-ish inputs."""
    for channels in (1, 2, 3):
        files, refs = [], []
        for mul in (1, 2, 3, 100):
            for frames in range(max(mul * 100 - 2, 1), mul * 100 + 2):
                pcm = gen_test_signal(channels, frames)
                enc = oracle.sea_encode(pcm, 44100, channels, oracle.make_settings(3.0))
                files.append(enc)
                refs.append(oracle.sea_decode(enc).samples)
        outs = ctx.decode_batch(files)
        for o, r in zip(outs, refs):
            assert o.samples.size == r.size and np.array_equal(o.samples, r)


def test_decode_batch_mixed_streams_uses_generic_path(ctx, oracle):
    """Heterogeneous batch (different channel counts / modes) in one launch."""
    files, refs = [], []
    for i, (ch, bits, vbr) in enumerate([(1, 3.0, False), (2, 5.0, True), (3, 2.0, False), (2, 3.0, False), (5, 6.0, False)]):
        pcm = synth.gen_stream(40 + i, 7000 + 13 * i, ch, 44100)
        enc = oracle.sea_encode(pcm, 44100, ch, oracle.make_settings(bits, vbr))
        files.append(enc)
        refs.append(oracle.sea_decode(enc).samples)
    for o, r in zip(ctx.decode_batch(files), refs):
        assert np.array_equal(o.samples, r)


def test_decode_uniform_batch_fast_path(ctx, oracle):
    """Many uniform stereo CBR streams with ragged tails: exercises warp tiles that straddle streams."""
    files, refs = [], []
    for i in range(37):
        frames = 5120 * (1 + i % 3) + (i * 211) % 5120
        pcm = synth.gen_stream(100 + i, frames, 2, 44100)
        enc = oracle.sea_encode(pcm, 44100, 2, oracle.make_settings(3.0))
        files.append(enc)
        refs.append(oracle.sea_decode(enc).samples)
    for o, r in zip(ctx.decode_batch(files), refs):
        assert np.array_equal(o.samples, r)
    # same for mono VBR
    files, refs = [], []
    for i in range(19):
        pcm = synth.gen_stream(200 + i, 5120 + (i * 977) % 9000, 1, 48000)
        enc = oracle.sea_encode(pcm, 48000, 1, oracle.make_settings(3.0, True))
        files.append(enc)
        refs.append(oracle.sea_decode(enc).samples)
    for o, r in zip(ctx.decode_batch(files), refs):
        assert np.array_equal(o.samples, r)


def test_decode_errors(ctx, oracle):
    pcm = synth.gen_stream(3, 6000, 2, 44100)
    enc = bytearray(oracle.sea_encode(pcm, 44100, 2, oracle.make_settings(3.0)))
    bad = bytes(b"saec") + bytes(enc[4:])
    with pytest.raises(S.SeaError) as e:
        ctx.sea_decode(bad)
    assert e.value.code == api.ERR_INVALID_FILE
    bad = bytearray(enc)
    bad[22] = 7  # chunk type (chunk.rs:81-85)
    with pytest.raises(S.SeaError) as e:
        ctx.sea_decode(bytes(bad))
    assert e.value.code == api.ERR_INVALID_FRAME
    with pytest.raises(S.SeaError) as e:  # truncated inside the second chunk: the reference panics on the slice
        ctx.sea_decode(bytes(enc[:-100]))
    assert e.value.code == api.ERR_DOMAIN
    # truncated exactly at a chunk boundary: the reference stops quietly with fewer samples (file.rs:186-188)
    cut = ctx.sea_decode(bytes(enc[: 22 + 4132]))
    assert np.array_equal(cut.samples, oracle.sea_decode(bytes(enc[: 22 + 4132])).samples) and cut.samples.size == 5120 * 2


# ------------------------------------------------------------------------------------------------ encode vs oracle

@pytest.mark.parametrize("channels", [1, 2, 3])
@pytest.mark.parametrize("sfb", [3, 4, 5])
def test_encode_cbr_parameters(ctx, oracle, channels, sfb):
    """tests/test.rs:35-64 sweep (channels 1..3 x sf_bits 3..5 x bits 1..8), bit-exact instead of a PSNR bound."""
    pcm = gen_test_signal(channels, 11025, seed=sfb)
    for bits in range(1, 9):
        st, ost = _settings_pair(oracle, residual_bits=float(bits), scale_factor_bits=sfb)
        assert ctx.sea_encode(pcm, 44100, channels, st) == oracle.sea_encode(pcm, 44100, channels, ost), bits


@pytest.mark.parametrize("bits", [1.5, 2.0, 2.5, 3.0, 3.5, 4.0, 5.0, 6.0, 7.0, 7.3])
def test_encode_vbr_bitrates(ctx, oracle, bits):
    for channels in (1, 2):
        pcm = synth.gen_stream(int(bits * 10) + channels, 5120 * 2 + 2560, channels, 44100)
        st, ost = _settings_pair(oracle, residual_bits=bits, vbr=True)
        ref, ties = oracle.sea_encode(pcm, 44100, channels, ost, return_ties=True)
        assert ties == 0
        got = ctx.sea_encode(pcm, 44100, channels, st)
        assert got == ref
        assert ctx.last_vbr_ties == 0


def _loud_signals(frames, channels):
    """Inputs that push the LMS weights and the dequantised steps far from ordinary audio: the encoder's per-block choice of the
    weights-penalty form (32-bit proved before / after the trial, narrow 64-bit, wide) must not change a bit of the output."""
    rng = np.random.default_rng(99)
    t = np.arange(frames)
    noise = rng.integers(-32768, 32768, size=(frames, channels)).astype(np.int16)
    square = np.where((t[:, None] + np.arange(channels)[None, :]) % 2 == 0, 32767, -32768).astype(np.int16)
    chirp = (32767 * np.sin(2 * np.pi * (0.05 + 0.45 * t / frames) * t))[:, None].repeat(channels, 1).astype(np.int16)
    bursts = np.where((t[:, None] // 37) % 2 == 0, noise, 0).astype(np.int16)
    return {"noise": noise, "square": square, "chirp": chirp, "bursts": bursts}


@pytest.mark.parametrize("name", ["noise", "square", "chirp", "bursts"])
def test_encode_loud_signals_match_oracle(ctx, oracle, name):
    frames = 5120 * 2 + 1500
    pcm = np.ascontiguousarray(_loud_signals(frames, 2)[name]).reshape(-1)
    for kw in ([dict(residual_bits=float(b)) for b in range(1, 9)] +
               [dict(residual_bits=b, vbr=True) for b in (2.0, 3.0, 4.0, 5.5, 7.0)]):
        st, ost = _settings_pair(oracle, **kw)
        ref, ref_ties = oracle.sea_encode(pcm, 44100, 2, ost, return_ties=True)
        got = ctx.sea_encode(pcm, 44100, 2, st)
        # Exact rank ties across a bucket boundary: the reference's order is unspecified there (sort_unstable_by,
        # encoder_vbr.rs:102-103); library and oracle both use (error, index), so their bytes agree regardless and both count
        # the same number of tied boundaries -- recorded, not skipped.
        assert ctx.last_vbr_ties == ref_ties, (name, kw, ctx.last_vbr_ties, ref_ties)
        assert got == ref, (name, kw, f"ties={ref_ties}")
        assert np.array_equal(ctx.sea_decode(got).samples, oracle.sea_decode(ref).samples)


def test_encode_multichannel_and_geometry(ctx, oracle):
    cases = [
        (8, dict(residual_bits=4.0)),
        (8, dict(residual_bits=3.0, vbr=True)),
        (5, dict(residual_bits=2.0, scale_factor_bits=3)),
        (3, dict(residual_bits=3.5, vbr=True, scale_factor_bits=5)),
        (2, dict(residual_bits=3.0, scale_factor_frames=10, frames_per_chunk=1000)),
        (2, dict(residual_bits=4.0, vbr=True, scale_factor_frames=16, frames_per_chunk=4096)),
        (1, dict(residual_bits=5.0, scale_factor_bits=6, scale_factor_frames=32, frames_per_chunk=320)),
        (4, dict(residual_bits=6.0, scale_factor_bits=2)),
        (17, dict(residual_bits=3.0)),
        (1, dict(residual_bits=3.0, vbr=True, scale_factor_frames=5, frames_per_chunk=200)),  # wrapped VBR size codes
        (2, dict(residual_bits=4.0, vbr=True, scale_factor_frames=5, frames_per_chunk=200)),
    ]
    for channels, kw in cases:
        n = kw.get("frames_per_chunk", 5120)
        pcm = synth.gen_stream(channels * 3, n * 2 + n // 2 + 7, channels, 48000)
        st, ost = _settings_pair(oracle, **kw)
        assert ctx.sea_encode(pcm, 48000, channels, st) == oracle.sea_encode(pcm, 48000, channels, ost), (channels, kw)


def test_encode_ragged_and_edge_inputs(ctx, oracle):
    st, ost = _settings_pair(oracle)
    for channels in (1, 2, 3):
        for frames in (1, 2, 19, 20, 21, 99, 100, 101, 5119, 5120, 5121, 10240):
            pcm = gen_test_signal(channels, frames)
            assert ctx.sea_encode(pcm, 44100, channels, st) == oracle.sea_encode(pcm, 44100, channels, ost), (channels, frames)
    # empty input: header only (encoder.rs:73-78)
    assert ctx.sea_encode(np.zeros(0, np.int16), 44100, 2, st) == oracle.sea_encode(np.zeros(0, np.int16), 44100, 2, ost)
    # extreme content: full-scale square wave, silence, alternating extremes (weights penalty / clamps)
    n = 5120 * 2
    sq = np.where((np.arange(n) // 7) % 2 == 0, 32767, -32768).astype(np.int16)
    for sig in (sq, np.zeros(n, np.int16), np.tile(np.array([32767, -32768], np.int16), n // 2)):
        for bits in (1.0, 3.0, 8.0):
            s2, o2 = _settings_pair(oracle, residual_bits=bits)
            assert ctx.sea_encode(sig, 44100, 1, s2) == oracle.sea_encode(sig, 44100, 1, o2)
    # VBR with ragged tails (trap T14: sortable items use the interleaved sample count)
    vs, vo = _settings_pair(oracle, residual_bits=3.0, vbr=True)
    for channels, frames in ((1, 5), (1, 27), (2, 27), (3, 27), (3, 5120 + 27), (2, 5120 * 2 + 19)):
        pcm = synth.gen_stream(frames, frames, channels, 44100)
        assert ctx.sea_encode(pcm, 44100, channels, vs) == oracle.sea_encode(pcm, 44100, channels, vo), (channels, frames)


def test_encode_batch_matches_one_shot(ctx, oracle):
    st, ost = _settings_pair(oracle, residual_bits=4.0)
    streams = [synth.gen_stream(300 + i, 3000 + 517 * i, 2, 44100) for i in range(9)]
    outs = ctx.encode_batch(streams, 44100, 2, st)
    for pcm, enc in zip(streams, outs):
        assert enc == oracle.sea_encode(pcm, 44100, 2, ost)
    vs, vo = _settings_pair(oracle, residual_bits=2.5, vbr=True)
    outs = ctx.encode_batch(streams[:4], 44100, 2, vs)
    for pcm, enc in zip(streams[:4], outs):
        assert enc == oracle.sea_encode(pcm, 44100, 2, vo)


def test_encode_rejects_what_the_reference_panics_on(ctx):
    pcm = synth.gen_stream(1, 6000, 2, 44100)
    for kw in (dict(residual_bits=8.0, vbr=True), dict(residual_bits=1.2, vbr=True), dict(residual_bits=0.5),
               dict(scale_factor_frames=7)):
        with pytest.raises(S.SeaError) as e:
            ctx.sea_encode(pcm, 44100, 2, S.EncoderSettings(**kw))
        assert e.value.code == api.ERR_DOMAIN
    with pytest.raises(S.SeaError) as e:  # one sample for two channels: UnexpectedEof in the reference
        ctx.sea_encode(np.zeros(1, np.int16), 44100, 2, S.EncoderSettings())
    assert e.value.code == api.ERR_DOMAIN


# ------------------------------------------------------------------------------------------------ round trips, streaming

def test_round_trip_config1(ctx, oracle):
    """BASELINE config 1 (10 s 44.1 kHz stereo CBR 3): exact size, encode == oracle, decode == oracle."""
    pcm = synth.gen_stream(0, 441000, 2, 44100)
    enc = ctx.sea_encode(pcm, 44100, 2, S.EncoderSettings())
    assert len(enc) == 355954
    assert enc == oracle.sea_encode(pcm, 44100, 2, oracle.make_settings(3.0))
    assert np.array_equal(ctx.sea_decode(enc).samples, oracle.sea_decode(enc).samples)


def test_streaming_api(ctx, oracle):
    """tests/streaming.rs:51-97: interleaved encode_frame/decode_frame equals the prefix of the one-shot result."""
    pcm = gen_test_signal(1, 44100)
    settings = S.EncoderSettings()
    ref_dec = oracle.sea_decode(oracle.sea_encode(pcm, 44100, 1, oracle.make_settings(3.0))).samples  # the one-shot result, by the oracle

    class Shared(io.RawIOBase):  # the test's SharedBuffer: a FIFO both sides hold
        def __init__(self):
            self.buf = bytearray()

        def write(self, b):
            self.buf += b
            return len(b)

        def read(self, n=-1):
            n = len(self.buf) if n < 0 else min(n, len(self.buf))
            out = bytes(self.buf[:n])
            del self.buf[:n]
            return out

    pipe = Shared()
    enc = S.SeaEncoder(1, 44100, None, settings, io.BytesIO(pcm.astype("<i2").tobytes()), pipe, ctx=ctx)
    assert enc.encode_frame()
    out = io.BytesIO()
    dec = S.SeaDecoder(pipe, out, ctx=ctx)
    for _ in range(3):
        assert enc.encode_frame()
        assert dec.decode_frame()
    got = np.frombuffer(out.getvalue(), dtype="<i2")
    assert got.size == 3 * 5120 and np.array_equal(got, ref_dec[: got.size])
    assert dec.get_header().total_frames == 0 and dec.get_header().chunk_size == enc.chunk_size
    enc.close()
    dec.close()


def test_streaming_encoder_equals_one_shot_bytes(ctx, oracle):
    for kw in (dict(), dict(residual_bits=3.0, vbr=True)):
        settings, ost = _settings_pair(oracle, **kw)
        pcm = synth.gen_stream(11, 5120 * 3 + 100, 2, 44100)
        sink = io.BytesIO()
        enc = S.SeaEncoder(2, 44100, pcm.size // 2, settings, io.BytesIO(pcm.astype("<i2").tobytes()), sink, ctx=ctx)
        while enc.encode_frame():
            pass
        enc.finalize()
        with pytest.raises(S.SeaError) as e:
            enc.encode_frame()
        assert e.value.code == api.ERR_ENCODER_CLOSED
        assert sink.getvalue() == oracle.sea_encode(pcm, 44100, 2, ost)
        out = io.BytesIO()
        dec = S.SeaDecoder(io.BytesIO(sink.getvalue()), out, ctx=ctx)
        while dec.decode_frame():
            pass
        assert np.array_equal(np.frombuffer(out.getvalue(), dtype="<i2"), oracle.sea_decode(sink.getvalue()).samples)


def test_device_resident_batch_and_properties(ctx, oracle):
    """Device-pointer entry points + size-independent properties at a larger size: the decoder applied to the encoder's
    output reproduces the encoder's own reconstruction (checked via re-encode idempotence of chunk headers) and every
    stream of a replicated batch decodes to identical PCM."""
    import torch

    n_streams, frames, ch = 64, 5120 * 20, 2
    settings = S.EncoderSettings()
    dev = torch.device("cuda:0")
    pcm = synth.gen_batch_torch(4, frames, ch, 44100, dev).repeat(n_streams // 4, 1).contiguous()
    bound = ctx.encode_bound(frames, ch, settings)
    stride = (bound + 15) // 16 * 16
    out = torch.zeros(n_streams * stride, dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()
    lens = ctx.encode_batch_device(pcm.data_ptr(), np.arange(n_streams) * frames * ch, np.full(n_streams, frames), 44100, ch,
                                   settings, out.data_ptr(), np.arange(n_streams) * stride)
    assert np.all(lens == bound)
    host = out.cpu().numpy()
    # first four streams against the oracle, the replicas against the first four
    for i in range(4):
        ref = oracle.sea_encode(pcm[i].cpu().numpy(), 44100, ch, oracle.make_settings(3.0))
        assert host[i * stride: i * stride + bound].tobytes() == ref
    for i in range(4, n_streams):
        assert np.array_equal(host[i * stride: i * stride + bound], host[(i % 4) * stride: (i % 4) * stride + bound])
    headers = np.stack([host[i * stride: i * stride + 22] for i in range(n_streams)])
    dec = torch.zeros(n_streams * frames * ch, dtype=torch.int16, device=dev)
    n = ctx.decode_batch_device(out.data_ptr(), np.arange(n_streams) * stride, lens, headers, dec.data_ptr(),
                                np.arange(n_streams) * frames * ch)
    assert np.all(n == frames * ch)
    dec = dec.view(n_streams, -1).cpu().numpy()
    for i in range(4):
        assert np.array_equal(dec[i], oracle.sea_decode(host[i * stride: i * stride + bound].tobytes()).samples)
    for i in range(4, n_streams):
        assert np.array_equal(dec[i], dec[i % 4])
    err = dec[:4].astype(np.float64) - pcm[:4].cpu().numpy()
    assert np.sqrt(np.mean((err / 32767.0) ** 2)) < 0.05


def test_pipelined_host_buffer_decode(ctx, oracle):
    """sea_b200_decode_batch with host buffers splits a large batch into groups and pipelines H2D / kernels / D2H over two
    lanes (capi.cu).  Every group boundary and both lanes must give what the one-shot decode gives: four distinct streams
    (one with a partial last chunk shared by all) against the oracle, 96 replicas against those."""
    n_streams, frames, ch = 96, 5120 * 430 + 777, 2   # 96 x 4.4 M samples = 423 M samples -> 5 groups of <= 96 Mi samples
    settings = S.EncoderSettings()
    uniq = [synth.gen_stream(100 + i, frames, ch, 44100) for i in range(4)]
    files = ctx.encode_batch(uniq, 44100, ch, settings)
    for f, u in zip(files[:2], uniq[:2]):
        assert f == oracle.sea_encode(u, 44100, ch, oracle.make_settings(3.0))
    want = [ctx.sea_decode(f).samples for f in files]
    assert np.array_equal(want[0], oracle.sea_decode(files[0]).samples)
    flen = len(files[0])
    stride = (flen + 15) // 16 * 16
    sea = np.zeros(n_streams * stride, dtype=np.uint8)
    for i in range(n_streams):
        sea[i * stride: i * stride + flen] = np.frombuffer(files[i % 4], dtype=np.uint8)
    spp = frames * ch
    pcm = np.zeros(n_streams * spp, dtype=np.int16)
    n = ctx.decode_batch_host(sea.ctypes.data, np.arange(n_streams) * stride, np.full(n_streams, flen), pcm.ctypes.data,
                              np.arange(n_streams) * spp, np.full(n_streams, spp))
    assert np.all(n == spp)
    pcm = pcm.reshape(n_streams, spp)
    for i in range(n_streams):
        assert np.array_equal(pcm[i], want[i % 4]), f"stream {i} differs after the pipelined decode"
    # scattered layout (streams in reverse order): the grouping must fall back to one range and still be right
    order = np.arange(n_streams)[::-1].copy()
    pcm2 = np.zeros(8 * spp, dtype=np.int16)
    n2 = ctx.decode_batch_host(sea.ctypes.data, order[:8] * stride, np.full(8, flen), pcm2.ctypes.data, np.arange(8) * spp)
    assert np.all(n2 == spp)
    for j in range(8):
        assert np.array_equal(pcm2.reshape(8, spp)[j], want[int(order[j]) % 4])


def test_cpp_host_mirror(ctx, oracle, tmp_path):
    """include/sea_b200.hpp (the compiled-language host mirror of src/encoder.rs, src/decoder.rs, src/lib.rs) driven the way
    tests/streaming.rs drives the crate: one-shot encode, chunk-at-a-time SeaEncoder, SeaDecoder over the result."""
    import subprocess

    from sea_codec_b200 import build as B

    exe = str(tmp_path / "host_mirror_test")  # outside the source tree, which may be read-only
    src = os.path.join(ROOT, "tests", "csrc", "host_mirror_test.cpp")
    lib_dir = os.path.dirname(B.LIB)
    subprocess.run(["g++", "-std=c++17", "-O2", "-o", exe, src, "-L" + lib_dir, "-l:libsea_b200.so", "-Wl,-rpath," + lib_dir], check=True)
    for channels, bits, vbr in ((2, 3.0, 0), (1, 3.0, 1), (3, 5.0, 0)):
        pcm = synth.gen_stream(50 + channels, 5120 * 2 + 777, channels, 44100)
        raw = tmp_path / "in.raw"
        raw.write_bytes(pcm.astype("<i2").tobytes())
        one, stream, dec = tmp_path / "one.sea", tmp_path / "stream.sea", tmp_path / "dec.raw"
        r = subprocess.run([exe, str(raw), str(channels), "44100", str(bits), str(vbr), str(one), str(stream), str(dec)],
                           capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        ref = oracle.sea_encode(pcm, 44100, channels, oracle.make_settings(bits, bool(vbr)))
        assert one.read_bytes() == ref and stream.read_bytes() == ref
        assert np.array_equal(np.frombuffer(dec.read_bytes(), dtype="<i2"), oracle.sea_decode(ref).samples)
