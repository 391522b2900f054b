"""GPU tests added in round 2 (-m gpu): the reference-decoder pin of the encoder's LMS path, the bounds fixes of the
lane-per-chunk decode route, owned-range copies of the host-buffer batch calls, the low-stream-count encode mapping, the
device synth kernel and the per-stream VBR tie counters.  Everything goes through the C-ABI and is compared with the CPU
oracle or with the reference's own C decoder (oracle/_ref)."""
import ctypes as C
import io
import os

import numpy as np
import pytest

import sea_codec_b200 as S
from sea_codec_b200 import api, synth
from util import gen_test_signal, reference_c_result, sha

pytestmark = pytest.mark.gpu


def _settings_pair(oracle, **kw):
    return S.EncoderSettings(**kw), oracle.make_settings(**kw)


# ------------------------------------------------------------------------------------------------ parity pins

@pytest.mark.parametrize("channels", [1, 2, 3, 8])
@pytest.mark.parametrize("bits", [1, 2, 3, 4, 5, 6, 7, 8])
def test_gpu_encoder_lms_against_the_reference_decoder(ctx, oracle, channels, bits):
    """VERDICT r1 missing #1: decode every GPU-encoded CBR stream with the reference's own c/sea.h and require that the LMS
    state the REFERENCE decoder holds at each chunk end (captured before its free, c/sea.h:147-185) equals, mod 2^16
    (lms.rs:64-78), the LMS block the GPU encoder wrote into the next chunk header (file.rs:146-149).  That checks the encoder's
    dequantise / predict / clamp / update path (encoder_base.rs:73-88, lms.rs:33-51) against reference code with no restatement
    in between; the history half is also visible black-box in the PCM c/sea.h emits.  Without oracle/_ref the state and PCM
    come from the record (util.reference_c_result); recorded from the oracle, they pin the GPU encoder and decoder to the
    oracle's bytes and decode."""
    n_chunks, frames = 5, 5120 * 4 + 1000  # whole scale-factor blocks only (c/sea.h:168)
    pcm = synth.gen_stream(900 + channels * 10 + bits, frames, channels, 44100)
    enc = ctx.sea_encode(pcm, 44100, channels, S.EncoderSettings(residual_bits=float(bits)))
    pcm_sha, lms = reference_c_result(oracle, f"gpu_encoder_lms/ch{channels}_b{bits}", enc, lms=True)
    hdr = oracle.chunk_header_lms(enc)
    assert hdr.shape == (n_chunks, channels, 8) and lms.shape == (n_chunks - 1, channels, 8)
    assert np.array_equal(lms, hdr[1:]), "encoder's chunk-header LMS != the reference decoder's end-of-chunk state"
    # the GPU decoder agrees with the reference decoder on the GPU encoder's bytes, so its PCM stands for c/sea.h's below
    dec = ctx.sea_decode(enc).samples
    assert sha(dec) == pcm_sha
    out = dec.reshape(-1, channels)
    for k in range(1, n_chunks):
        assert np.array_equal(hdr[k][:, :4].T, out[k * 5120 - 4: k * 5120])
    assert np.array_equal(hdr[0][:, 4:], np.tile(np.array([0, 0, -8192, 16384], dtype=np.int16), (channels, 1)))


def test_vbr_bytes_equal_the_oracle_even_with_ties_and_ties_are_counted_per_stream(ctx, oracle):
    """The reference's sort_unstable_by (encoder_vbr.rs:102-103) leaves the order of equal errors open; library and oracle both
    order by (error, index), so their bytes agree even on inputs FULL of ties (silence, repeated blocks), and both count the
    blocks that tie across a bucket boundary -- the chunks on which agreement with a Rust binary is undefined."""
    frames, ch = 5120 * 3 + 400, 2
    tone = synth.gen_stream(5, frames, ch, 44100)
    silence = np.zeros(frames * ch, dtype=np.int16)
    half = tone.copy()
    half[: 5120 * 2 * ch] = 0
    period = np.tile(tone[: 20 * ch * 8], frames // (20 * 8) + 1)[: frames * ch].copy()
    streams = [tone, silence, half, period]
    st, ost = _settings_pair(oracle, residual_bits=3.0, vbr=True)
    refs = [oracle.sea_encode(x, 44100, ch, ost, return_ties=True) for x in streams]
    got = ctx.encode_batch(streams, 44100, ch, st)
    per = ctx.last_vbr_ties_per_stream(len(streams))
    assert int(per.sum()) == ctx.last_vbr_ties
    for i, (g, (r, ties)) in enumerate(zip(got, refs)):
        assert g == r, f"stream {i}: GPU and oracle disagree (ties: {ties})"
        assert int(per[i]) == ties, (i, per, ties)
    assert per[0] == 0 and per[1] > 0  # tone + noise: none; digital silence: every boundary ties


# ------------------------------------------------------------------------------------------------ ADVICE r1 (medium) #1

def _uniform_files(oracle, n, channels, frames, first=300, **kw):
    return [oracle.sea_encode(synth.gen_stream(first + i, frames, channels, 44100), 44100, channels, oracle.make_settings(**kw)) for i in range(n)]


@pytest.mark.parametrize("channels,kw", [(2, dict(residual_bits=3.0)), (1, dict(residual_bits=3.0, vbr=True)), (2, dict(residual_bits=3.0, vbr=True)),
                                         (4, dict(residual_bits=4.0)), (8, dict(residual_bits=4.0))])
def test_truncated_stream_in_the_middle_of_a_batch(ctx, oracle, channels, kw):
    """A stream cut in the middle of a chunk, NOT last in the buffer: the lane-per-chunk kernels must not take the cut chunk
    (they never look at data_len and would read the next stream's bytes).  Whatever the oracle says about the cut file alone --
    an error, or a quiet shorter decode -- the batch must say too, for the whole call (error) or for that stream (samples)."""
    files = _uniform_files(oracle, 6, channels, 5120 * 6 + 100, **kw)
    cs = files[0][6] | (files[0][7] << 8)
    for cut_at in (22 + 3 * cs + cs // 2, 22 + 3 * cs + 5, 22 + 2 * cs):  # mid-chunk, inside a chunk header, on a chunk boundary
        batch = list(files)
        batch[2] = files[2][:cut_at]
        try:
            want = [oracle.sea_decode(f).samples for f in batch]
        except oracle.OracleError:
            want = None
        if want is None:
            with pytest.raises(S.SeaError) as e:
                ctx.decode_batch(batch)
            assert e.value.kind in ("Domain", "InvalidFrame")
        else:
            for g, w in zip(ctx.decode_batch(batch), want):
                assert np.array_equal(g.samples, w)


@pytest.mark.parametrize("channels,kw", [(2, dict(residual_bits=3.0)), (2, dict(residual_bits=3.0, vbr=True)), (8, dict(residual_bits=4.0))])
def test_crafted_small_header_chunk_size(ctx, oracle, channels, kw):
    """file.rs:33-38 accepts any chunk_size >= 16.  With the file header patched to 16 while the chunk headers still describe
    the full layout, the reference reads 16 bytes per chunk and panics on the first slice (chunk.rs:95-101); the library must
    report Domain and must not let a lane walk its implied layout past the bytes it was given."""
    files = _uniform_files(oracle, 4, channels, 5120 * 3, **kw)
    bad = []
    for f in files:
        b = bytearray(f)
        b[6], b[7] = 16, 0
        bad.append(bytes(b))
    with pytest.raises(oracle.OracleError):
        oracle.sea_decode(bad[0])
    with pytest.raises(S.SeaError) as e:
        ctx.decode_batch(bad)
    assert e.value.kind == "Domain"
    with pytest.raises(S.SeaError):
        ctx.sea_decode(bad[0])
    # a chunk_size a little short of the layout: every chunk's residual section is cut (slice panic in the reference)
    cs = files[0][6] | (files[0][7] << 8)
    short = []
    for f in files:
        b = bytearray(f)
        b[6], b[7] = (cs - 40) & 255, (cs - 40) >> 8
        short.append(bytes(b))
    try:
        want = [oracle.sea_decode(f).samples for f in short]
    except oracle.OracleError:
        want = None
    if want is None:
        with pytest.raises(S.SeaError):
            ctx.decode_batch(short)
    else:
        for g, w in zip(ctx.decode_batch(short), want):
            assert np.array_equal(g.samples, w)


# ------------------------------------------------------------------------------------------------ ADVICE r1 (medium) #2

def test_host_batch_calls_write_only_the_ranges_they_own(ctx, oracle):
    """sea_b200_decode_batch / encode_batch with gaps between the streams' output ranges, and with ranges in descending
    order: bytes of the caller's buffers outside [offset, offset + length) must come back untouched."""
    ch, frames, n = 2, 5120 * 3 + 333, 5
    pcm_in = [synth.gen_stream(400 + i, frames, ch, 44100) for i in range(n)]
    st, ost = _settings_pair(oracle, residual_bits=3.0)
    files = [oracle.sea_encode(x, 44100, ch, ost) for x in pcm_in]
    want = [oracle.sea_decode(f).samples for f in files]
    flen, spp, gap = len(files[0]), frames * ch, 1000
    sea = np.zeros(n * (flen + 64), dtype=np.uint8)
    sea_off = np.arange(n, dtype=np.uint64) * (flen + 64)
    for i, f in enumerate(files):
        sea[int(sea_off[i]): int(sea_off[i]) + flen] = np.frombuffer(f, dtype=np.uint8)
    for order in (np.arange(n), np.arange(n)[::-1].copy()):
        pcm = np.full(n * (spp + gap) + gap, 0x5A5A, dtype=np.int16)
        pcm_off = (gap + order * (spp + gap)).astype(np.uint64)
        got = ctx.decode_batch_host(sea.ctypes.data, sea_off, np.full(n, flen), pcm.ctypes.data, pcm_off)
        assert np.all(got == spp)
        owned = np.zeros(pcm.size, dtype=bool)
        for i in range(n):
            o = int(pcm_off[i])
            assert np.array_equal(pcm[o: o + spp], want[i])
            owned[o: o + spp] = True
        assert np.all(pcm[~owned] == 0x5A5A), "decode_batch wrote outside the streams' PCM ranges"
        # encode side
        bound = ctx.encode_bound(frames, ch, st)
        out = np.full(n * (bound + gap) + gap, 0xA5, dtype=np.uint8)
        out_off = (gap + order * (bound + gap)).astype(np.uint64)
        flat = np.concatenate(pcm_in)
        lens = ctx.encode_batch_host(flat.ctypes.data, np.arange(n) * spp, np.full(n, frames), 44100, ch, st, out.ctypes.data, out_off)
        owned = np.zeros(out.size, dtype=bool)
        for i in range(n):
            o = int(out_off[i])
            assert out[o: o + int(lens[i])].tobytes() == files[i]
            owned[o: o + int(lens[i])] = True
        assert np.all(out[~owned] == 0xA5), "encode_batch wrote outside the streams' output ranges"


# ------------------------------------------------------------------------------------------------ ADVICE r1 (low)

def test_make_chunk_refuses_a_small_buffer_before_the_state_advances(ctx, oracle):
    ch = 2
    pcm = synth.gen_stream(21, 5120 * 3, ch, 44100)
    st, ost = _settings_pair(oracle, residual_bits=3.0)
    ref = oracle.sea_encode(pcm, 44100, ch, ost)
    L = api.lib()
    stc = st._c()
    h = C.c_void_p()
    assert L.sea_b200_encoder_create(ctx._h, ch, 44100, C.byref(stc), C.byref(h)) == 0
    out = np.zeros(70000, dtype=np.uint8)
    n = C.c_uint64(0)
    chunks = []
    for k in range(3):
        x = np.ascontiguousarray(pcm[k * 5120 * ch: (k + 1) * 5120 * ch])
        if k == 1:  # too small: must fail WITHOUT touching the LMS / prev_scalefactor state ...
            assert L.sea_b200_encoder_make_chunk(h, x.ctypes.data, x.size, out.ctypes.data, 100, C.byref(n)) == api.ERR_CAPACITY
        # ... so that the retry produces what a single call would have
        assert L.sea_b200_encoder_make_chunk(h, x.ctypes.data, x.size, out.ctypes.data, out.size, C.byref(n)) == 0
        chunks.append(out[: n.value].tobytes())
    L.sea_b200_encoder_destroy(h)
    assert b"".join(chunks) == ref[22:]


def test_decode_chunks_checks_scale_factor_bits_like_decode_chunk(ctx, oracle):
    ch = 1
    pcm = synth.gen_stream(22, 5120 * 2, ch, 44100)
    a = oracle.sea_encode(pcm, 44100, ch, oracle.make_settings(3.0, scale_factor_bits=4))
    b = oracle.sea_encode(pcm, 44100, ch, oracle.make_settings(3.0, scale_factor_bits=5))
    cs = a[6] | (a[7] << 8)
    L = api.lib()
    h = C.c_void_p()
    hdr = np.frombuffer(a[:22], dtype=np.uint8)
    assert L.sea_b200_decoder_create(ctx._h, hdr.ctypes.data, 22, C.byref(h)) == 0
    out = np.zeros(5120 * 4, dtype=np.int16)
    n = C.c_uint64(0)
    first = np.frombuffer(a[22: 22 + cs], dtype=np.uint8)
    assert L.sea_b200_decoder_decode_chunks(h, ctx._h, first.ctypes.data, first.size, 5120, out.ctypes.data, out.size, C.byref(n)) == 0
    other = np.frombuffer(b[22: 22 + (b[6] | (b[7] << 8))], dtype=np.uint8)[:cs].copy()  # a chunk with sf bits 5 (decoder.rs:21 assert)
    assert L.sea_b200_decoder_decode_chunks(h, ctx._h, other.ctypes.data, other.size, 5120, out.ctypes.data, out.size, C.byref(n)) == api.ERR_DOMAIN
    L.sea_b200_decoder_destroy(h)


# ------------------------------------------------------------------------------------------------ encode lane mappings

@pytest.fixture
def pin_mapping():
    old = os.environ.get("SEA_B200_ENC_SPLIT")
    yield lambda v: os.environ.__setitem__("SEA_B200_ENC_SPLIT", v)
    if old is None:
        os.environ.pop("SEA_B200_ENC_SPLIT", None)
    else:
        os.environ["SEA_B200_ENC_SPLIT"] = old


@pytest.mark.parametrize("channels", [2, 3, 8])
def test_encode_lane_mappings_agree_with_the_oracle(ctx, oracle, channels, pin_mapping):
    """One warp per channel pair (many streams) and one warp per channel (few streams: BASELINE config 5 over 8 GPUs) are the
    same arithmetic on different lanes: both must reproduce the oracle, CBR 1..8 and VBR, ragged last chunk included."""
    frames = 5120 * 2 + 1234
    pcm = synth.gen_stream(30 + channels, frames, channels, 44100)
    cases = [dict(residual_bits=float(b)) for b in range(1, 9)] + [dict(residual_bits=b, vbr=True) for b in (1.5, 3.0, 4.5, 6.0, 7.3)]
    for kw in cases:
        st, ost = _settings_pair(oracle, **kw)
        ref = oracle.sea_encode(pcm, 44100, channels, ost)
        for mode in ("0", "1"):
            pin_mapping(mode)
            assert ctx.sea_encode(pcm, 44100, channels, st) == ref, (kw, "split" if mode == "1" else "pairs")


def test_encode_batches_small_and_large_match_the_oracle(ctx, oracle):
    """No pinning (the warp-per-pair mapping is the default at every size): 8 and 400 stereo streams -- fewer and more warps than
    sub-partitions -- must match the oracle stream by stream, VBR and CBR."""
    ch, frames = 2, 5120 + 640
    st, ost = _settings_pair(oracle, residual_bits=3.0, vbr=True)
    uniq = [synth.gen_stream(500 + i, frames, ch, 44100) for i in range(8)]
    refs = [oracle.sea_encode(x, 44100, ch, ost) for x in uniq]
    assert ctx.encode_batch(uniq, 44100, ch, st) == refs
    big = ctx.encode_batch([uniq[i % 8] for i in range(400)], 44100, ch, st)
    for i, g in enumerate(big):
        assert g == refs[i % 8], i
    st2, ost2 = _settings_pair(oracle, residual_bits=5.0)
    refs2 = [oracle.sea_encode(x, 44100, ch, ost2) for x in uniq]
    big2 = ctx.encode_batch([uniq[i % 8] for i in range(400)], 44100, ch, st2)
    for i, g in enumerate(big2):
        assert g == refs2[i % 8], i


# ------------------------------------------------------------------------------------------------ bench inputs

def test_device_synth_matches_the_host_recipe(ctx):
    import torch

    frames, ch, rate = 5120 * 3 + 77, 2, 44100
    ids = np.array([0, 1, 47, 48, 1000, 123456], dtype=np.uint32)
    stride = frames * ch + 10
    buf = torch.zeros(ids.size * stride, dtype=torch.int16, device="cuda:0")
    torch.cuda.synchronize()
    ctx.synth_pcm_device(buf.data_ptr(), stride, ids, frames, ch, rate)
    got = buf.cpu().numpy().reshape(ids.size, stride)
    for i, k in enumerate(ids):
        assert np.array_equal(got[i, : frames * ch], synth.gen_stream(int(k), frames, ch, rate)), int(k)
        assert np.all(got[i, frames * ch:] == 0)
    mono = torch.zeros(3 * 1000, dtype=torch.int16, device="cuda:0")
    ctx.synth_pcm_device(mono.data_ptr(), 1000, np.array([7, 8, 9]), 1000, 1, 48000)
    for i, k in enumerate((7, 8, 9)):
        assert np.array_equal(mono.cpu().numpy().reshape(3, 1000)[i], synth.gen_stream(k, 1000, 1, 48000))


# ------------------------------------------------------------------------------------------------ time-sliced host-buffer encode

@pytest.fixture
def force_slices():
    old = os.environ.get("SEA_B200_ENC_SLICE")
    yield lambda v: os.environ.__setitem__("SEA_B200_ENC_SLICE", v)
    if old is None:
        os.environ.pop("SEA_B200_ENC_SLICE", None)
    else:
        os.environ["SEA_B200_ENC_SLICE"] = old


@pytest.mark.parametrize("kw", [dict(residual_bits=3.0), dict(residual_bits=3.0, vbr=True), dict(residual_bits=5.0, scale_factor_bits=5)])
def test_time_sliced_batch_encode_equals_one_shot(ctx, oracle, kw, force_slices):
    """sea_b200_encode_batch cuts long batches into slices of k chunks (upload / kernel / download pipelined, LMS state kept on the
    device between the launches).  Forced here to 2- and 3-chunk slices on a ragged batch: every stream -- full slices, a stream
    that ends early, partial last chunks (CBR: size known on the host; VBR: read back), an empty stream -- must equal the
    oracle's one-shot bytes, in a packed (2-D copies) and in a scattered layout, and nothing outside the owned ranges may change."""
    ch = 2
    lens = [5120 * 7 + 333, 5120 * 7 + 333, 5120 * 3, 5120 * 2 + 17, 0, 5120 * 9 + 4000]
    streams = [synth.gen_stream(600 + i, n, ch, 44100) for i, n in enumerate(lens)]
    st, ost = _settings_pair(oracle, **kw)
    refs = [oracle.sea_encode(x, 44100, ch, ost) for x in streams]
    for k in ("2", "3"):
        force_slices(k)
        assert ctx.encode_batch(streams, 44100, ch, st) == refs, f"{k}-chunk slices, ragged batch"
    # regular layout: equal lengths at a constant stride (the 2-D copy route), with gaps that must stay untouched
    force_slices("2")
    n, frames, gap = 5, 5120 * 5 + 1000, 500
    same = [synth.gen_stream(620 + i, frames, ch, 44100) for i in range(n)]
    want = [oracle.sea_encode(x, 44100, ch, ost) for x in same]
    spp, bound = frames * ch, ctx.encode_bound(frames, ch, st)
    pcm = np.zeros(n * (spp + gap), dtype=np.int16)
    for i, x in enumerate(same):
        pcm[i * (spp + gap): i * (spp + gap) + spp] = x
    out = np.full(n * (bound + gap) + gap, 0xA5, dtype=np.uint8)
    out_off = gap + np.arange(n, dtype=np.uint64) * (bound + gap)
    got = ctx.encode_batch_host(pcm.ctypes.data, np.arange(n) * (spp + gap), np.full(n, frames), 44100, ch, st, out.ctypes.data, out_off)
    owned = np.zeros(out.size, dtype=bool)
    for i in range(n):
        o = int(out_off[i])
        assert out[o: o + int(got[i])].tobytes() == want[i], i
        owned[o: o + int(got[i])] = True
    assert np.all(out[~owned] == 0xA5)


# ------------------------------------------------------------------------------------------------ in-process multi-GPU batch API

def _device_sets():
    import torch

    n = torch.cuda.device_count()
    sets = [[0], [0, 0], [0, 0, 0]]  # several contexts on one GPU exercise the sharding and the host threads on any box
    if n >= 2:
        sets.append(list(range(n)))
    return sets


def test_multi_gpu_batch_calls_equal_the_single_gpu_result(ctx, oracle):
    """sea_b200_multi_{encode,decode}_batch (SURVEY 8e: shard by stream, one host thread + context per GPU, only per-GPU counts
    gathered): same bytes / samples as the single-context call and the oracle, whatever the number of devices; the reported
    ranges tile the batch and the per-device counts add up."""
    ch = 2
    lens = [5120 * 3 + 100 * i for i in range(7)] + [17, 5120]  # (an empty stream encodes to a header the reference refuses to decode)
    streams = [synth.gen_stream(800 + i, n, ch, 44100) for i, n in enumerate(lens)]
    n = len(streams)
    for kw in (dict(residual_bits=3.0), dict(residual_bits=4.5, vbr=True)):
        st, ost = _settings_pair(oracle, **kw)
        refs = [oracle.sea_encode(x, 44100, ch, ost) for x in streams]
        want_pcm = [oracle.sea_decode(r).samples for r in refs]
        pcm_off = np.concatenate([[0], np.cumsum([x.size for x in streams])[:-1]]).astype(np.uint64)
        flat = np.concatenate(streams)
        bounds = np.array([ctx.encode_bound(k, ch, st) for k in lens], dtype=np.uint64)
        out_off = np.concatenate([[0], np.cumsum(bounds + 7)[:-1]]).astype(np.uint64)
        for devs in _device_sets():
            m = S.MultiContext(devs)
            out = np.zeros(int((bounds + 7).sum()), dtype=np.uint8)
            got_lens, first, per = m.encode_batch_host(flat.ctypes.data, pcm_off, np.array(lens, dtype=np.uint32), 44100, ch, st,
                                                       out.ctypes.data, out_off)
            assert first[0] == 0 and np.all(np.diff(first.astype(np.int64)) >= 0) and int(per.sum()) == int(got_lens.sum())
            for i in range(n):
                assert out[int(out_off[i]): int(out_off[i]) + int(got_lens[i])].tobytes() == refs[i], (devs, kw, i)
            # decode what was just encoded, from the same buffer layout
            pcm = np.zeros(flat.size + 16, dtype=np.int16)
            ns, first_d, per_d = m.decode_batch_host(out.ctypes.data, out_off, got_lens, pcm.ctypes.data, pcm_off)
            assert int(per_d.sum()) == int(ns.sum()) == flat.size
            for i in range(n):
                assert np.array_equal(pcm[int(pcm_off[i]): int(pcm_off[i]) + int(ns[i])], want_pcm[i]), (devs, kw, i)
            m.close()
    with pytest.raises(S.SeaError):
        S.MultiContext([99])


# ------------------------------------------------------------------------------------------------ small-job decode kernel

import test_gpu_next_rows as _R  # noqa: E402
import test_gpu_parity as _P  # noqa: E402


@pytest.mark.latency_kernel
def test_latency_kernel_golden_and_errors(ctx, oracle):
    _P.test_golden_decode(ctx)
    _P.test_decode_errors(ctx, oracle)
    _P.test_decode_ragged_lengths(ctx, oracle)
    _R.test_vbr_corrupt_size_codes_match_the_generic_verdict(ctx, oracle)
    _R.test_decode_range_random_access(ctx, oracle)


@pytest.mark.latency_kernel
@pytest.mark.parametrize("channels", [1, 2, 3, 8])
def test_latency_kernel_cbr_and_vbr(ctx, oracle, channels):
    for bits in range(1, 9):
        _P.test_decode_cbr_matches_oracle(ctx, oracle, channels, bits)
    if channels <= 2:
        for bits in (1.5, 3.0, 4.5, 6.0, 7.3):
            _P.test_decode_vbr_matches_oracle(ctx, oracle, channels, bits)
    if channels in (1, 2, 3, 8):
        _R.test_gpu_cbr_decode_against_the_reference_c_decoder(ctx, oracle, channels, 3 if channels != 8 else 4)


@pytest.mark.latency_kernel
def test_latency_kernel_geometries_and_corruption(ctx, oracle):
    for sfb, sff, fpc in ((3, 20, 5120), (5, 20, 5120), (4, 10, 1000), (4, 5, 200), (2, 16, 4096), (6, 32, 320)):
        _P.test_decode_other_geometry(ctx, oracle, sfb, sff, fpc)
    _R.test_randomised_settings_against_oracle(ctx, oracle)
    _R.test_corrupted_files_never_disagree_with_the_oracle(ctx, oracle)
    _R.test_multi_chunk_streaming_equals_chunk_at_a_time(ctx, oracle, False)
    _R.test_multi_chunk_streaming_equals_chunk_at_a_time(ctx, oracle, True)
    for channels, kw in ((2, dict(residual_bits=3.0)), (2, dict(residual_bits=3.0, vbr=True)), (8, dict(residual_bits=4.0))):
        test_truncated_stream_in_the_middle_of_a_batch(ctx, oracle, channels, kw)
        test_crafted_small_header_chunk_size(ctx, oracle, channels, kw)


@pytest.mark.auto_route
def test_decode_route_is_chosen_by_job_size(ctx, oracle):
    """Unpinned: one file (3 chunks) takes the small-job kernel, a batch of 400 x 20 chunks the throughput kernels; both must
    match the oracle, and the launch counter tells the routes apart (one launch against full-chunk + partial-chunk kernels)."""
    pcm = synth.gen_stream(71, 5120 * 2 + 700, 2, 44100)
    enc = oracle.sea_encode(pcm, 44100, 2, oracle.make_settings(3.0))
    want = oracle.sea_decode(enc).samples
    n0 = ctx.launch_count
    assert np.array_equal(ctx.sea_decode(enc).samples, want)
    assert ctx.launch_count - n0 == 1
    long = oracle.sea_encode(synth.gen_stream(72, 5120 * 20 + 700, 2, 44100), 44100, 2, oracle.make_settings(3.0))
    want_long = oracle.sea_decode(long).samples
    n0 = ctx.launch_count
    got = ctx.decode_batch([long] * 400)
    assert ctx.launch_count - n0 == 2
    for g in (got[0], got[199], got[399]):
        assert np.array_equal(g.samples, want_long)


# ------------------------------------------------------------------------------------------------ odd channel counts

@pytest.mark.parametrize("channels", [3, 5, 7])
def test_odd_channel_counts(ctx, oracle, channels):
    """3 (tests/test.rs:10), 5 and 7 channels.  Full CBR chunks with scale_factor_frames 20 and a chunk length that is a multiple
    of 80 frames go through decode_mc_kernel (one lane per chunk, four store phases, PCM words that straddle two frames), the
    partial last chunks and everything else (VBR, other block lengths) through decode_staged_kernel with 32 / C chunks per warp
    and idle tail lanes -- uniform batches, CBR at three sizes and VBR, against the oracle."""
    for kw, launches in ((dict(residual_bits=1.0), 2), (dict(residual_bits=3.0), 2), (dict(residual_bits=8.0), 2),
                         (dict(residual_bits=3.0, vbr=True), 1), (dict(residual_bits=5.0, scale_factor_bits=5), 2),
                         (dict(residual_bits=4.0, scale_factor_frames=10, frames_per_chunk=1000), 1),
                         (dict(residual_bits=3.0, frames_per_chunk=5100), 1), (dict(residual_bits=3.0, frames_per_chunk=80), 2)):
        fpc = kw.get("frames_per_chunk", 5120)
        files = [oracle.sea_encode(synth.gen_stream(1000 + 10 * channels + i, fpc * 2 + 37 * i + (i % 2) * fpc, channels, 44100), 44100, channels,
                                   oracle.make_settings(**kw)) for i in range(12)]
        want = [oracle.sea_decode(f).samples for f in files]
        n0 = ctx.launch_count
        for g, w in zip(ctx.decode_batch(files), want):
            assert np.array_equal(g.samples, w), (channels, kw)
        assert ctx.launch_count - n0 == launches, (kw, "whole-frame kernel + staged kernel for the tails" if launches == 2 else "one staged-kernel launch")


@pytest.mark.parametrize("channels", [3, 4, 5, 6, 7, 8])
@pytest.mark.parametrize("sfb", [1, 3, 5, 6])
def test_multichannel_kernel_other_scale_factor_bits(ctx, oracle, channels, sfb):
    """decode_mc_kernel with scale_factor_bits != 4 (tests/test.rs:37 sweeps 3..5): a block's channels * s scale-factor bits start
    at any bit phase and are cut out of a 64-bit window.  Loud, quiet and ordinary signals so that every scale factor occurs."""
    for bits in (2.0, 5.0, 8.0):
        files, refs = [], []
        for i in range(4):
            frames = 5120 * (1 + i % 2) + (i * 911) % 5120
            if i == 1:
                t = np.arange(frames * channels)
                pcm = np.clip(36000 * np.sin(t * 0.013 * (1 + t % channels)), -32768, 32767).astype(np.int16)
            elif i == 2:
                pcm = np.random.default_rng(90 + i).integers(-300, 301, frames * channels).astype(np.int16)
            else:
                pcm = synth.gen_stream(1500 + i, frames, channels, 48000)
            enc = oracle.sea_encode(pcm, 48000, channels, oracle.make_settings(bits, scale_factor_bits=sfb))
            files.append(enc)
            refs.append(oracle.sea_decode(enc).samples)
        n0 = ctx.launch_count
        for o, r in zip(ctx.decode_batch(files), refs):
            assert np.array_equal(o.samples, r), (bits, sfb)
        assert ctx.launch_count - n0 == 2, "expected the whole-frame kernel plus one launch for the partial last chunks"


# ------------------------------------------------------------------------------------------------ scale_factor_bits 3 and 5 on the fast pass

@pytest.mark.parametrize("sfb", [3, 5])
@pytest.mark.parametrize("channels", [1, 2, 3, 5, 8])
def test_encode_fast_pass_other_scale_factor_bits(ctx, oracle, sfb, channels, pin_mapping):
    """tests/test.rs:37 sweeps scale_factor_bits 3..5: 8 resp. 32 candidates per block = 8 / 32 lanes per chain group, four chains /
    one chain per warp.  CBR 1..8 and VBR, ragged last chunk, batches of streams with different lengths, both lane mappings."""
    frames = 5120 * 2 + 999
    pcm = synth.gen_stream(40 + channels, frames, channels, 44100)
    cases = [dict(residual_bits=float(b), scale_factor_bits=sfb) for b in range(1, 9)] + \
            [dict(residual_bits=b, vbr=True, scale_factor_bits=sfb) for b in (2.0, 3.0, 4.5, 6.5)]
    for kw in cases:
        st, ost = _settings_pair(oracle, **kw)
        try:
            ref = oracle.sea_encode(pcm, 44100, channels, ost)
        except oracle.OracleError:
            with pytest.raises(S.SeaError):
                ctx.sea_encode(pcm, 44100, channels, st)
            continue
        assert ctx.sea_encode(pcm, 44100, channels, st) == ref, kw
    pin_mapping("1")
    st, ost = _settings_pair(oracle, residual_bits=3.0, scale_factor_bits=sfb)
    if channels >= 2:
        assert ctx.sea_encode(pcm, 44100, channels, st) == oracle.sea_encode(pcm, 44100, channels, ost)
    pin_mapping("0")
    streams = [synth.gen_stream(60 + i, 5120 + 777 * i, channels, 44100) for i in range(5)]
    for kw in (dict(residual_bits=3.0, scale_factor_bits=sfb), dict(residual_bits=3.5, vbr=True, scale_factor_bits=sfb)):
        st, ost = _settings_pair(oracle, **kw)
        assert ctx.encode_batch(streams, 44100, channels, st) == [oracle.sea_encode(x, 44100, channels, ost) for x in streams], kw


# ------------------------------------------------------------------------------------------------ lane-per-chunk decode, other scale_factor_bits

@pytest.mark.parametrize("channels", [1, 2])
@pytest.mark.parametrize("sfb", [1, 2, 3, 5, 6, 7])
def test_lane_per_chunk_kernels_other_scale_factor_bits(ctx, oracle, channels, sfb):
    """decode_unrolled_kernel (CBR; scale_factor_bits 3 / 5 as compile-time instances, the rest through the run-time one) and
    decode_vbr_kernel (VBR, scale_factor_bits <= 6) read a round's scale factors as s resp. 2 s whole bytes at any byte phase.
    tests/test.rs:37 sweeps 3..5.  Loud / quiet / ordinary signals so that every scale factor occurs; full chunks plus a tail."""
    cases = [dict(residual_bits=float(b), scale_factor_bits=sfb) for b in (1, 3, 4, 6, 8)]
    if sfb <= 6:
        cases += [dict(residual_bits=b, vbr=True, scale_factor_bits=sfb) for b in (2.0, 3.5, 5.5)]
    for kw in cases:
        files, refs = [], []
        for i in range(5):
            frames = 5120 * (2 + i % 2) + (i * 733) % 5120
            if i == 1:
                t = np.arange(frames * channels)
                pcm = np.clip(37000 * np.sin(t * 0.017), -32768, 32767).astype(np.int16)
            elif i == 2:
                pcm = np.random.default_rng(70 + i).integers(-200, 201, frames * channels).astype(np.int16)
            else:
                pcm = synth.gen_stream(1700 + i, frames, channels, 44100)
            try:
                enc = oracle.sea_encode(pcm, 44100, channels, oracle.make_settings(**kw))
            except oracle.OracleError:
                break
            files.append(enc)
            refs.append(oracle.sea_decode(enc).samples)
        if len(files) < 5:
            continue
        n0 = ctx.launch_count
        for o, r in zip(ctx.decode_batch(files), refs):
            assert np.array_equal(o.samples, r), kw
        if sfb <= 5:  # the staged kernel that takes the tails holds tables up to scale_factor_bits 5; beyond that the generic kernel decodes
            assert ctx.launch_count - n0 == 2, (kw, "expected a lane-per-chunk kernel plus the staged kernel for the partial last chunks")


@pytest.mark.parametrize("channels", [1, 2])
def test_full_width_ctas_and_sector_paired_row_fetch(ctx, oracle, channels, monkeypatch):
    """Large jobs run the unrolled kernel as one full-width CTA per SM (small ones as several narrower CTAs, which is what every
    other test sees): SEA_B200_FULL_CTAS pins that launch shape.  In a build with -DSEA_DEC_PAIRFETCH=1 the rows are then staged
    by sector-paired requests (lanes 2j / 2j+1 fetch the two halves of one 32-byte sector of row j: the lane that decodes a row is
    not the lane that fetched it) and SEA_B200_PAIRFETCH=0 switches back; in the default build both passes run the same kernel.
    Streams of different lengths put stream boundaries inside a warp's 32 rows."""
    monkeypatch.setenv("SEA_B200_FULL_CTAS", "1")
    for bits in range(1, 9):
        files, refs = [], []
        for i in range(7):
            frames = 5120 * (1 + (i * 5) % 4) + (i * 613) % 5120
            pcm = synth.gen_stream(1900 + 10 * bits + i, frames, channels, 44100)
            enc = oracle.sea_encode(pcm, 44100, channels, oracle.make_settings(float(bits)))
            files.append(enc)
            refs.append(oracle.sea_decode(enc).samples)
        for flag in ("1", "0"):
            monkeypatch.setenv("SEA_B200_PAIRFETCH", flag)
            for o, r in zip(ctx.decode_batch(files), refs):
                assert np.array_equal(o.samples, r), (bits, flag)


@pytest.mark.parametrize("channels,fpc,lane_per_chunk", [(2, 5000, True), (2, 1000, True), (2, 200, True), (1, 5040, True), (1, 240, True),
                                                         (2, 5020, False), (1, 5000, False)])
def test_chunk_lengths_with_a_trailing_half_round(ctx, oracle, channels, fpc, lane_per_chunk):
    """The unrolled and the VBR lane-per-chunk kernels stage two halves (four bodies) per round; a chunk length that is a whole
    number of halves but not of rounds (seaconv takes any frames_per_chunk that scale_factor_frames divides: 5000-frame stereo
    chunks are 62.5 rounds) ends with a shorter round.  Lengths that are not whole halves (their PCM rows would not stay 32-byte
    aligned) go to the staged kernel."""
    for kw in (dict(residual_bits=3.0), dict(residual_bits=6.0), dict(residual_bits=8.0, scale_factor_bits=5), dict(residual_bits=3.0, vbr=True),
               dict(residual_bits=6.5, vbr=True)):
        files, refs = [], []
        for i in range(5):
            frames = fpc * (3 + i % 3) + (i * 97) % fpc
            pcm = synth.gen_stream(2100 + i, frames, channels, 44100)
            try:
                enc = oracle.sea_encode(pcm, 44100, channels, oracle.make_settings(frames_per_chunk=fpc, **kw))
            except oracle.OracleError:  # a VBR bitrate whose bucket plan leaves the reference's domain at this chunk length
                break
            files.append(enc)
            refs.append(oracle.sea_decode(enc).samples)
        if len(files) < 5:
            continue
        n0 = ctx.launch_count
        for o, r in zip(ctx.decode_batch(files), refs):
            assert np.array_equal(o.samples, r), (kw, fpc)
        assert ctx.launch_count - n0 == (2 if lane_per_chunk else 1), (kw, fpc)


@pytest.mark.parametrize("seed", [20261019, 7, 424242])
def test_randomised_batches_through_the_lane_per_chunk_kernels(ctx, oracle, seed):
    """Seeded sweep over what the lane-per-chunk decode kernels take (scale_factor_frames 20): 1..8 channels, scale_factor_bits
    1..6, CBR 1..8 / VBR 1.5..7.3, chunk lengths that are whole rounds, end in a short round, or must go to the staged / generic
    kernels, ragged batches of loud / quiet / ordinary / full-scale streams, narrow and full-width CTAs.  Oracle-encoded files,
    decoded PCM must equal the oracle's."""
    import os

    rng = np.random.default_rng(seed)
    checked = 0
    for case in range(72):
        ch = int(rng.integers(1, 9))
        sfb = int(rng.integers(1, 7))
        fpc = 20 * int(rng.choice([2, 4, 8, 10, 12, 16, 25, 50, 63, 64, 100, 128, 250, 256]))
        vbr = bool(rng.integers(0, 3) == 0)
        bits = float(rng.choice([1.5, 2.0, 2.5, 3.0, 3.7, 4.2, 5.0, 5.5, 6.5, 7.3])) if vbr else float(rng.integers(1, 9))
        kw = dict(residual_bits=bits, vbr=vbr, scale_factor_bits=sfb, frames_per_chunk=fpc)
        files, refs = [], []
        for i in range(int(rng.integers(2, 6))):
            frames = fpc * int(rng.integers(1, 5)) + int(rng.integers(0, fpc))
            kind = (case + i) % 4
            t = np.arange(frames * ch, dtype=np.float64)
            if kind == 0:
                pcm = synth.gen_stream(5000 + 10 * case + i, frames, ch, 44100)
            elif kind == 1:
                pcm = np.clip(40000 * np.sin(t * 0.05) + rng.normal(0, 3000, t.size), -32768, 32767).astype(np.int16)
            elif kind == 2:
                pcm = rng.integers(-40, 41, t.size).astype(np.int16)
            else:
                pcm = rng.integers(-32768, 32768, t.size).astype(np.int16)
            try:
                enc = oracle.sea_encode(pcm, 44100, ch, oracle.make_settings(**kw))
            except oracle.OracleError:
                files = None
                break
            try:
                want = oracle.sea_decode(enc).samples
            except oracle.OracleError:  # a VBR plan at the edge of the reference's domain: its own decoder panics on what it wrote
                with pytest.raises(S.SeaError):
                    ctx.decode_batch([enc, enc])
                files = None
                break
            files.append(enc)
            refs.append(want)
        if not files:
            continue
        if case % 3 == 0:
            os.environ["SEA_B200_FULL_CTAS"] = "1"
        try:
            got = ctx.decode_batch(files)
        finally:
            os.environ.pop("SEA_B200_FULL_CTAS", None)
        for o, r in zip(got, refs):
            assert np.array_equal(o.samples, r), (case, ch, kw)
        checked += 1
    assert checked >= 50, checked


# ------------------------------------------------------------------------------------------------ pipelined host-buffer decode

@pytest.mark.gpu
@pytest.mark.parametrize("defer,ahead", [("1", "1"), ("0", "1"), ("1", "0"), ("0", "0")])
def test_pipelined_host_batch_decode_with_deferred_error_words(ctx, oracle, monkeypatch, defer, ahead):
    """sea_b200_decode_batch cuts a long batch into groups and queues them all without waiting for a group's error word
    (SEA_B200_DEC_DEFER, default on); a group whose word is not clean is redone on its own afterwards.  The uploads run ahead of
    the lanes on their own stream into one slot per group (SEA_B200_DEC_UPLOAD_AHEAD, default on).  Small groups forced by
    SEA_B200_DEC_GROUP_SAMPLES: (1) a clean batch, (2) one chunk in a middle group whose reserved header byte is not 0x5A -- the
    reference ignores that byte (chunk.rs:91), the specialised kernels hand the chunk back, the redo decodes it generically --,
    (3) a chunk type the reference rejects (chunk.rs:81-85) in a middle group: the call reports InvalidFrame."""
    ch, frames, n = 2, 5120 * 4 + 777, 14
    files = _uniform_files(oracle, n, ch, frames, first=900, residual_bits=3.0)
    want = [oracle.sea_decode(f).samples for f in files]
    monkeypatch.setenv("SEA_B200_DEC_GROUP_SAMPLES", str(2 * frames * ch))  # two streams per group: 7 groups, both lanes
    monkeypatch.setenv("SEA_B200_DEC_DEFER", defer)
    monkeypatch.setenv("SEA_B200_DEC_UPLOAD_AHEAD", ahead)
    monkeypatch.setenv("SEA_B200_DEC_LATENCY", "0")  # the throughput route is the one that defers
    cs = files[0][6] | (files[0][7] << 8)
    for g, w in zip(ctx.decode_batch(files), want):
        assert np.array_equal(g.samples, w)
    odd = list(files)
    b = bytearray(files[7])
    assert b[22 + 2 * cs + 3] == 0x5A
    b[22 + 2 * cs + 3] = 0x00
    odd[7] = bytes(b)
    assert np.array_equal(oracle.sea_decode(odd[7]).samples, want[7])
    for g, w in zip(ctx.decode_batch(odd), want):
        assert np.array_equal(g.samples, w)
    bad = list(files)
    b = bytearray(files[9])
    b[22 + cs] = 7
    bad[9] = bytes(b)
    with pytest.raises(oracle.OracleError):
        oracle.sea_decode(bad[9])
    with pytest.raises(S.SeaError) as e:
        ctx.decode_batch(bad)
    assert e.value.kind == "InvalidFrame"
    for g, w in zip(ctx.decode_batch(files), want):  # the context is reusable after the error
        assert np.array_equal(g.samples, w)
