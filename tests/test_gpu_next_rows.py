"""GPU tests of the SURVEY 8f "next" rows built on the hot path: seaconv conversions (f1), multi-chunk streaming (f2), the
wasm_api / c/sea.h shaped entry points (f3) and random-access decode (f4).  Every result is compared with the CPU oracle."""
import ctypes as C
import io
import os

import numpy as np
import pytest

import sea_codec_b200 as S
from sea_codec_b200 import api, seaconv, synth, wav
from util import reference_c_result, sha

pytestmark = pytest.mark.gpu


def test_seaconv_wav_to_sea_and_back(ctx, oracle, tmp_path):
    pcm = synth.gen_stream(7, 44100 * 3 + 123, 2, 44100)
    wav_in, sea_out, wav_out = str(tmp_path / "in.wav"), str(tmp_path / "out.sea"), str(tmp_path / "back.wav")
    wav.write_wav(pcm, 2, 44100, wav_in)
    for argv, kw in ((["-b", "3"], dict(residual_bits=3.0)), (["-b", "2.5", "-v", "-c", "2000", "-d", "10", "-s", "5"],
                                                               dict(residual_bits=2.5, vbr=True, frames_per_chunk=2000,
                                                                    scale_factor_frames=10, scale_factor_bits=5))):
        assert seaconv.main([wav_in, sea_out] + argv + ["--chunks-per-launch", "7"]) == 0
        got = open(sea_out, "rb").read()
        assert got == oracle.sea_encode(pcm, 44100, 2, oracle.make_settings(**kw)), argv
        assert seaconv.main([sea_out, wav_out, "--chunks-per-launch", "5"]) == 0
        back = wav.read_wav(wav_out)
        assert back.channels == 2 and back.sample_rate == 44100
        assert np.array_equal(back.samples, oracle.sea_decode(got).samples)


@pytest.mark.parametrize("vbr", [False, True])
def test_multi_chunk_streaming_equals_chunk_at_a_time(ctx, oracle, vbr):
    ch, frames = 2, 5120 * 9 + 1000
    pcm = synth.gen_stream(3, frames, ch, 48000)
    st = S.EncoderSettings(residual_bits=3.0, vbr=vbr)
    ref = oracle.sea_encode(pcm, 48000, ch, oracle.make_settings(3.0, vbr=vbr))
    for per, total in ((1, frames), (4, frames), (64, frames), (3, None)):
        out = io.BytesIO()
        src = pcm if total is not None else pcm[: 5120 * 9 * ch]  # streaming header: whole chunks only
        enc = S.SeaEncoder(ch, 48000, total, st, io.BytesIO(src.astype("<i2").tobytes()), out, ctx=ctx)
        while enc.encode_frames(per):
            pass
        enc.finalize()
        enc.close()
        if total is not None:
            assert out.getvalue() == ref, f"{per} chunks per launch"
        else:
            want = oracle.sea_encode(src, 48000, ch, oracle.make_settings(3.0, vbr=vbr))
            assert out.getvalue()[22:] == want[22:]  # same chunks; the streaming header carries total_frames = 0
            assert out.getvalue()[14:18] == b"\x00\x00\x00\x00"
    want_pcm = oracle.sea_decode(ref).samples
    for per in (1, 2, 5, 100):
        pcm_out = io.BytesIO()
        dec = S.SeaDecoder(io.BytesIO(ref), pcm_out, ctx=ctx)
        while dec.decode_frames(per):
            pass
        dec.close()
        assert np.array_equal(np.frombuffer(pcm_out.getvalue(), dtype="<i2"), want_pcm), f"{per} chunks per launch"


def test_decode_range_random_access(ctx, oracle):
    ch, frames = 2, 5120 * 6 + 777
    pcm = synth.gen_stream(11, frames, ch, 44100)
    for kw in (dict(residual_bits=3.0), dict(residual_bits=3.5, vbr=True)):
        sea = oracle.sea_encode(pcm, 44100, ch, oracle.make_settings(**kw))
        full = oracle.sea_decode(sea).samples.reshape(-1, ch)
        for first, n in ((0, 1), (0, frames), (5119, 2), (5120, 5120), (100, 20000), (5120 * 6, 777), (5120 * 6 + 700, 5000),
                         (frames - 1, 1), (frames, 10), (12345, 0), (1 << 40, 5)):
            got = ctx.decode_range(sea, first, n)
            want = full[first: first + n].reshape(-1) if first < frames else np.zeros(0, dtype=np.int16)
            assert got.sample_rate == 44100 and got.channels == ch
            assert np.array_equal(got.samples, want), (kw, first, n)
    # metadata: the reference never skips it (file.rs:53-54); the flag is the format-compatible fix
    sea = oracle.sea_encode(pcm, 44100, ch, oracle.make_settings(3.0))
    meta = b"title=x\nartist=y"
    with_meta = sea[:18] + len(meta).to_bytes(4, "little") + meta + sea[22:]
    got = ctx.decode_range(with_meta, 6000, 3000, skip_metadata=True)
    assert np.array_equal(got.samples, oracle.sea_decode(sea).samples.reshape(-1, ch)[6000:9000].reshape(-1))


def test_wasm_api_and_csea_shaped_entry_points(ctx, oracle):
    L = S.lib()
    pcm = synth.gen_stream(5, 5120 * 2 + 300, 2, 44100)
    L.sea_b200_wasm_setup()
    for bitrate, vbr in ((3.0, False), (4.0, True)):
        cap = pcm.size * 2 + 4096
        buf = L.sea_b200_wasm_allocate(cap)
        assert buf
        n = L.sea_b200_wasm_sea_encode(pcm.ctypes.data, pcm.size * 2, 44100, 2, bitrate, vbr, buf, cap)
        assert n > 0 and L.sea_b200_wasm_status() == 0
        enc = C.string_at(buf, n)
        assert enc == oracle.sea_encode(pcm, 44100, 2, oracle.make_settings(bitrate, vbr=vbr))
        out = np.zeros(pcm.size, dtype=np.int16)
        rate, ch = C.c_uint32(0), C.c_uint32(0)
        nb = L.sea_b200_wasm_sea_decode(buf, n, out.ctypes.data, out.size * 2, C.byref(rate), C.byref(ch))
        assert nb == pcm.size * 2 and (rate.value, ch.value) == (44100, 2)
        assert np.array_equal(out, oracle.sea_decode(enc).samples)
        # too small an output buffer: the reference asserts (wasm_api.rs:58,81); here 0 + a status
        assert L.sea_b200_wasm_sea_decode(buf, n, out.ctypes.data, 100, C.byref(rate), C.byref(ch)) == 0
        assert L.sea_b200_wasm_status() == api.ERR_CAPACITY
        L.sea_b200_wasm_deallocate(buf, cap)
    # c/sea.h: two-call pattern, return codes 0 / 1 / 2
    enc = np.frombuffer(oracle.sea_encode(pcm, 44100, 2, oracle.make_settings(3.0)), dtype=np.uint8).copy()
    rate, ch, tf = C.c_uint32(0), C.c_uint32(0), C.c_uint32(0)
    assert L.sea_b200_csea_decode(enc.ctypes.data, enc.size, C.byref(rate), C.byref(ch), None, C.byref(tf)) == 0
    assert (rate.value, ch.value, tf.value) == (44100, 2, pcm.size // 2)
    out = np.zeros(tf.value * ch.value, dtype=np.int16)
    assert L.sea_b200_csea_decode(enc.ctypes.data, enc.size, C.byref(rate), C.byref(ch), out.ctypes.data, C.byref(tf)) == 0
    assert np.array_equal(out, oracle.sea_decode(enc.tobytes()).samples)
    bad = enc.copy()
    bad[0] = ord("x")
    assert L.sea_b200_csea_decode(bad.ctypes.data, bad.size, C.byref(rate), C.byref(ch), out.ctypes.data, C.byref(tf)) == 1
    short = enc[: enc.size // 2].copy()
    assert L.sea_b200_csea_decode(short.ctypes.data, short.size, C.byref(rate), C.byref(ch), out.ctypes.data, C.byref(tf)) == 2


def test_cpp_seaconv_matches_python_cli(ctx, oracle, tmp_path):
    """tools/seaconv.cpp (compiled host, include/sea_b200.hpp) produces the same files as the oracle / the Python CLI."""
    import subprocess

    from sea_codec_b200 import build as B
    from util import ROOT

    exe = str(tmp_path / "seaconv")  # outside the source tree, which may be read-only
    lib_dir = os.path.dirname(B.LIB)
    subprocess.run(["g++", "-std=c++17", "-O2", "-I" + os.path.join(ROOT, "include"), "-o", exe, os.path.join(ROOT, "tools", "seaconv.cpp"),
                    "-L" + lib_dir, "-l:libsea_b200.so", "-Wl,-rpath," + lib_dir], check=True)
    pcm = synth.gen_stream(21, 44100 + 321, 1, 22050)
    wav_in, sea_out, wav_out = str(tmp_path / "in.wav"), str(tmp_path / "out.sea"), str(tmp_path / "back.wav")
    wav.write_wav(pcm, 1, 22050, wav_in)
    r = subprocess.run([exe, wav_in, sea_out, "-b", "4", "-c", "4000"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    enc = open(sea_out, "rb").read()
    assert enc == oracle.sea_encode(pcm, 22050, 1, oracle.make_settings(4.0, frames_per_chunk=4000))
    r = subprocess.run([exe, sea_out, wav_out], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    back = wav.read_wav(wav_out)
    assert back.sample_rate == 22050 and back.channels == 1 and np.array_equal(back.samples, oracle.sea_decode(enc).samples)
    r = subprocess.run([exe, wav_in, sea_out, "-b", "9"], capture_output=True, text=True)
    assert r.returncode == 1 and "Bitrate must be between 1.0 and 8.0" in r.stderr


def test_baseline_config2_vbr_mono_full_size(ctx, oracle):
    """BASELINE.json configs[1]: VBR, mono 48 kHz 60 s synthetic tone+noise, bitrate 3 -- bit-exact encode and decode at full
    size (2 880 000 samples: 562 full chunks of 1922 bytes + one of 2560 frames, SURVEY 8d)."""
    frames = 48000 * 60
    pcm = synth.gen_stream(2, frames, 1, 48000)
    enc = ctx.sea_encode(pcm, 48000, 1, S.EncoderSettings(residual_bits=3.0, vbr=True))
    assert ctx.last_vbr_ties == 0, "error ties across a bucket boundary: the reference's sort order would be unspecified here"
    ref = oracle.sea_encode(pcm, 48000, 1, oracle.make_settings(3.0, vbr=True))
    assert enc == ref
    hdr = S.parse_header(enc)
    assert hdr.chunk_size == 1922 and len(enc) == 22 + 562 * 1922 + (len(enc) - 22 - 562 * 1922) and (frames - 562 * 5120) == 2560
    dec = ctx.sea_decode(enc)
    assert dec.sample_rate == 48000 and dec.channels == 1
    assert np.array_equal(dec.samples, oracle.sea_decode(ref).samples)


def test_baseline_config3_eight_channels_cbr4(ctx, oracle):
    """BASELINE.json configs[2]: 8-channel 48 kHz interleaved stream, CBR bitrate 4 (multichannel lane mapping, chunk-parallel
    decode) at full size: 14.4 M frames, 2812 full chunks of 21 636 bytes + one of 2560 frames (SURVEY 8d)."""
    ch, frames = 8, 48000 * 300
    pcm = synth.gen_stream(3, frames, ch, 48000)
    enc = ctx.sea_encode(pcm, 48000, ch, S.EncoderSettings(residual_bits=4.0))
    ref = oracle.sea_encode(pcm, 48000, ch, oracle.make_settings(4.0))
    assert S.parse_header(enc).chunk_size == 21636 and len(enc) == 22 + 2812 * 21636 + 10884
    assert enc == ref
    dec = ctx.sea_decode(enc)
    want = oracle.sea_decode(ref).samples
    assert np.array_equal(dec.samples, want)
    # chunk-parallel property: any chunk range decodes to the same samples as the whole stream (what a 2nd GPU would do)
    n_chunks = (frames + 5119) // 5120
    for k0, k1 in ((0, 1), (1000, 1407), (n_chunks - 3, n_chunks)):
        part = ctx.decode_range(enc, k0 * 5120, (k1 - k0) * 5120)
        assert np.array_equal(part.samples, want[k0 * 5120 * ch: min(frames, k1 * 5120) * ch])


def test_randomised_settings_against_oracle(ctx, oracle):
    """Seeded sweep over the parameter space the grid tests do not enumerate: channels 1-5, scale_factor_bits 2-6, block and
    chunk geometry, CBR 1-8 and VBR 1.5-7.3 bits, ragged lengths, loud / quiet / clipped signals.  Encode bytes and decoded PCM
    must equal the oracle's; settings the reference cannot run (it would panic) must be rejected, not mis-encoded."""
    rng = np.random.default_rng(20261018)
    checked = rejected = 0
    for case in range(48):
        ch = int(rng.integers(1, 6))
        sfb = int(rng.integers(2, 7))
        sff = int(rng.choice([5, 8, 10, 16, 20, 25, 32, 40]))
        fpc = sff * int(rng.integers(8, 200))
        if fpc > 32000:
            fpc = sff * 100
        vbr = bool(rng.integers(0, 2))
        bits = float(rng.choice([1.5, 2.0, 2.5, 3.0, 3.7, 4.2, 5.0, 6.5, 7.3])) if vbr else float(rng.integers(1, 9))
        frames = int(rng.integers(1, 3 * fpc + 50))
        kind = case % 4
        t = np.arange(frames * ch, dtype=np.float64)
        if kind == 0:
            pcm = synth.gen_stream(1000 + case, frames, ch, 44100)
        elif kind == 1:  # loud, clipping
            pcm = np.clip(40000 * np.sin(t * 0.05) + rng.normal(0, 3000, t.size), -32768, 32767).astype(np.int16)
        elif kind == 2:  # quiet
            pcm = rng.integers(-40, 41, t.size).astype(np.int16)
        else:  # white noise, full scale
            pcm = rng.integers(-32768, 32768, t.size).astype(np.int16)
        kw = dict(residual_bits=bits, vbr=vbr, scale_factor_bits=sfb, scale_factor_frames=sff, frames_per_chunk=fpc)
        try:
            enc = ctx.sea_encode(pcm, 44100, ch, S.EncoderSettings(**kw))
        except api.SeaError as e:
            assert e.code in (api.ERR_DOMAIN, api.ERR_INVALID_PARAMETERS), (kw, e)
            rejected += 1
            continue
        ref = oracle.sea_encode(pcm, 44100, ch, oracle.make_settings(**kw))
        assert enc == ref, (case, ch, frames, kw)
        dec = ctx.sea_decode(enc)
        assert np.array_equal(dec.samples, oracle.sea_decode(ref).samples), (case, ch, frames, kw)
        checked += 1
    assert checked >= 30, (checked, rejected)


@pytest.mark.parametrize("channels,bits", [(2, 1.5), (2, 3.0), (2, 5.0), (2, 6.0), (2, 7.3), (1, 2.0), (1, 4.5), (1, 7.0)])
def test_vbr_uniform_batch_throughput_kernel(ctx, oracle, channels, bits):
    """decode_vbr_kernel (lane per chunk, run-time field widths): uniform VBR batches with several full chunks per stream and a
    ragged tail (which the staged kernel takes) must match the oracle for every header size 1..7 and both channel counts."""
    files, refs = [], []
    for i in range(9):
        frames = 5120 * (2 + i % 3) + (i * 733) % 5120
        kind = i % 3
        if kind == 0:
            pcm = synth.gen_stream(300 + i, frames, channels, 44100)
        elif kind == 1:  # loud: exercises the clamp in the pack-saturate path
            t = np.arange(frames * channels)
            pcm = np.clip(36000 * np.sin(t * 0.03) + 2000 * np.cos(t * 1.7), -32768, 32767).astype(np.int16)
        else:  # quiet: ties and small sizes
            pcm = (np.random.default_rng(i).integers(-300, 301, frames * channels)).astype(np.int16)
        enc = oracle.sea_encode(pcm, 44100, channels, oracle.make_settings(bits, True))
        files.append(enc)
        refs.append(oracle.sea_decode(enc).samples)
    for o, r in zip(ctx.decode_batch(files), refs):
        assert np.array_equal(o.samples, r)


def test_vbr_corrupt_size_codes_match_the_generic_verdict(ctx, oracle):
    """A chunk whose size codes ask for more residual bits than it holds is a slice error in the reference (chunk.rs:190-196): the
    throughput kernel must notice and hand the batch to the generic path, which reports Domain -- not decode garbage."""
    pcm = synth.gen_stream(77, 5120 * 3, 2, 44100)
    enc = bytearray(oracle.sea_encode(pcm, 44100, 2, oracle.make_settings(3.0, True)))
    hdr = S.parse_header(bytes(enc))
    vbr_sec = 22 + hdr.chunk_size + 4 + 32 + 256          # second chunk: header, LMS, 512 scale-factor nibbles
    for i in range(128):
        enc[vbr_sec + i] = 0xFF                            # every block asks for header size + 2
    with pytest.raises(api.SeaError) as e:
        ctx.decode_batch([bytes(enc)] * 4)
    assert e.value.code == api.ERR_DOMAIN


def test_corrupted_files_never_disagree_with_the_oracle(ctx, oracle):
    """Seeded corruption sweep: random byte flips, truncations and header edits of CBR and VBR files.  Whatever the oracle says
    (samples, or an error where the reference errors or panics) the GPU path must say too -- alone and as a uniform batch of
    copies, which is what routes through the throughput kernels -- and no input may crash the device."""
    rng = np.random.default_rng(777)
    pcm = synth.gen_stream(9, 5120 * 3 + 1234, 2, 44100)
    bases = [oracle.sea_encode(pcm, 44100, 2, oracle.make_settings(3.0)),
             oracle.sea_encode(pcm, 44100, 2, oracle.make_settings(3.0, True)),
             oracle.sea_encode(pcm[::2].copy(), 44100, 1, oracle.make_settings(5.0, True))]

    def verdict(fn):
        try:
            return True, fn()
        except (api.SeaError, oracle.OracleError):
            return False, None

    n_err = n_ok = 0
    for case in range(90):
        f = bytearray(bases[case % 3])
        kind = (case // 3) % 5
        if kind == 0:      # flips inside chunk payloads / chunk headers
            for _ in range(int(rng.integers(1, 6))):
                f[int(rng.integers(22, len(f)))] ^= int(rng.integers(1, 256))
        elif kind == 1:    # truncation anywhere after the file header
            f = f[: int(rng.integers(22, len(f)))]
        elif kind == 2:    # total_frames edited (shorter, slightly longer, streaming 0)
            tf = int.from_bytes(f[14:18], "little")
            new = int(rng.choice([0, tf - 1, tf - 5120, tf + 1, tf + 5120, 1, 5120]))
            f[14:18] = max(new, 0).to_bytes(4, "little")
        elif kind == 3:    # chunk_size / frames_per_chunk edited
            cs = int.from_bytes(f[6:8], "little")
            if rng.integers(0, 2):
                f[6:8] = int(max(16, cs + int(rng.integers(-40, 41)))).to_bytes(2, "little")
            else:
                f[8:10] = int(rng.choice([5100, 5120 - 20, 5140, 2560, 100])).to_bytes(2, "little")
        else:              # chunk header fields of one chunk: type, sizes byte, scale_factor_frames
            cs = int.from_bytes(f[6:8], "little")
            k = int(rng.integers(0, 3))
            off = 22 + k * cs + int(rng.integers(0, 3))
            if off < len(f):
                f[off] = int(rng.integers(0, 256))
        blob = bytes(f)
        ok_o, want = verdict(lambda: oracle.sea_decode(blob).samples)
        ok_g, got = verdict(lambda: ctx.sea_decode(blob).samples)
        assert ok_o == ok_g, (case, kind, ok_o, ok_g)
        if ok_o:
            assert np.array_equal(got, want), (case, kind)
            n_ok += 1
        else:
            n_err += 1
        ok_b, got_b = verdict(lambda: [d.samples for d in ctx.decode_batch([blob] * 3)])
        assert ok_b == ok_o, (case, kind, "batch")
        if ok_o:
            assert all(np.array_equal(g, want) for g in got_b), (case, kind, "batch")
    assert n_ok >= 10 and n_err >= 10, (n_ok, n_err)


@pytest.mark.parametrize("channels", [3, 4, 5, 6, 7, 8])
@pytest.mark.parametrize("bits", [1, 2, 3, 4, 5, 6, 7, 8])
def test_multichannel_whole_frame_kernel(ctx, oracle, channels, bits):
    """decode_mc_kernel (one lane per chunk with all channels, whole-frame 256-bit stores; two store phases for 6 channels, four
    for 3 / 5 / 7): uniform CBR batches with 3 .. 8 channels, several full chunks per stream plus a ragged tail (taken by the
    generic resp. staged kernel on the side stream), quiet / loud / ordinary signals."""
    files, refs = [], []
    for i in range(5):
        frames = 5120 * (1 + i % 3) + (i * 997) % 5120
        if i % 3 == 1:
            t = np.arange(frames * channels)
            pcm = np.clip(38000 * np.sin(t * 0.011 * (1 + t % channels)), -32768, 32767).astype(np.int16)
        elif i % 3 == 2:
            pcm = np.random.default_rng(50 + i).integers(-500, 501, frames * channels).astype(np.int16)
        else:
            pcm = synth.gen_stream(400 + i, frames, channels, 48000)
        enc = oracle.sea_encode(pcm, 48000, channels, oracle.make_settings(float(bits)))
        files.append(enc)
        refs.append(oracle.sea_decode(enc).samples)
    for o, r in zip(ctx.decode_batch(files), refs):
        assert np.array_equal(o.samples, r)


@pytest.mark.parametrize("channels,fpc", [(6, 5100), (6, 5080), (6, 40), (8, 1000), (8, 20), (4, 60), (4, 5100), (3, 5040), (3, 80), (5, 160), (7, 240),
                                          (3, 5100), (7, 40)])
def test_multichannel_other_chunk_lengths(ctx, oracle, channels, fpc):
    """Chunk lengths the whole-frame kernel takes (8 / 4 channels: any multiple of 20; 6 channels: multiples of 40, whose rows
    stay 32-byte aligned) and the ones that must fall through to the generic kernel (6 channels, N % 40 == 20)."""
    files, refs = [], []
    for i in range(3):
        frames = fpc * (3 + i) + (i * 13) % fpc
        pcm = synth.gen_stream(700 + i, frames, channels, 48000)
        enc = oracle.sea_encode(pcm, 48000, channels, oracle.make_settings(3.0, frames_per_chunk=fpc))
        files.append(enc)
        refs.append(oracle.sea_decode(enc).samples)
    for o, r in zip(ctx.decode_batch(files), refs):
        assert np.array_equal(o.samples, r)


@pytest.mark.parametrize("channels,bits", [(1, 3), (2, 1), (2, 3), (2, 8), (4, 4), (6, 2), (8, 4), (3, 5)])
def test_gpu_cbr_decode_against_the_reference_c_decoder(ctx, oracle, channels, bits):
    """The strongest pin available without a Rust toolchain: the reference's OWN decoder (c/sea.h, compiled into oracle/_ref by
    oracle/Makefile from the read-only reference tree) against the GPU decode kernels, on files the GPU encoder produced --
    no restatement in between.  c/sea.h handles CBR with whole scale-factor blocks only (c/sea.h:131-134, :168).  Without
    oracle/_ref the result comes from the record (util.reference_c_result): the GPU encoder's bytes and the GPU decode must
    equal it, recorded from the oracle, c/sea.h or not."""
    frames = 5120 * 3 + 2000  # a multiple of scale_factor_frames
    pcm = synth.gen_stream(700 + channels * 10 + bits, frames, channels, 44100)
    enc = ctx.sea_encode(pcm, 44100, channels, S.EncoderSettings(residual_bits=float(bits)))
    want = reference_c_result(oracle, f"gpu_cbr_decode/ch{channels}_b{bits}", enc)
    assert sha(ctx.sea_decode(enc).samples) == want
    for got in ctx.decode_batch([enc] * 5):  # the throughput kernels (unrolled / multichannel) + the tail kernels
        assert sha(got.samples) == want
