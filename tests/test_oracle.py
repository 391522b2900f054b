"""CPU tests: the oracle (oracle/sea_oracle.c) against the reference's known answers (SURVEY.md Appendix D), against the
reference's own C decoder (c/sea.h -> oracle/_ref), against the committed golden fixtures, and the invariants the
reference's tests pin (tests/test.rs:8-64, tests/streaming.rs:51-97)."""
import json
import os

import numpy as np
import pytest

from sea_codec_b200 import synth
from util import ROOT, gen_test_signal, reference_c_result, sha

GOLD = os.path.join(ROOT, "tests", "golden")


def test_scale_factors_appendix_d(oracle):
    exp = {
        1: [1, 8, 27, 64, 125, 216, 343, 512, 729, 1000, 1331, 1728, 2197, 2744, 3375, 4096],
        2: [1, 7, 24, 56, 108, 184, 289, 426, 601, 817, 1079, 1390, 1755, 2178, 2662, 3213],
        3: [1, 6, 21, 48, 90, 150, 232, 337, 469, 630, 823, 1051, 1315, 1618, 1963, 2352],
        4: [1, 6, 18, 39, 70, 114, 171, 244, 334, 441, 568, 715, 883, 1075, 1290, 1530],
        5: [1, 5, 14, 28, 48, 75, 108, 150, 199, 257, 323, 398, 483, 578, 682, 797],
        6: [1, 4, 11, 20, 33, 50, 70, 94, 122, 153, 189, 229, 273, 321, 373, 430],
        7: [1, 3, 8, 14, 21, 30, 41, 53, 67, 82, 98, 116, 135, 156, 178, 202],
        8: [1, 3, 6, 9, 14, 19, 25, 31, 38, 45, 53, 61, 70, 79, 88, 99],
    }
    for b, v in exp.items():
        assert oracle.scale_factors(b, 4).tolist() == v
    assert oracle.scale_factors(3, 3).tolist() == [1, 13, 60, 176, 406, 803, 1429, 2352]
    assert oracle.scale_factors(3, 5).tolist()[-3:] == [2035, 2191, 2352]


def test_tables_appendix_d(oracle):
    r3, d3 = oracle.tables(3, 4)
    assert r3.tolist() == [65536, 10922, 3120, 1365, 728, 436, 282, 194, 139, 104, 79, 62, 49, 40, 33, 27]
    r4, d4 = oracle.tables(4, 4)
    assert r4.tolist() == [65536, 10922, 3640, 1680, 936, 574, 383, 268, 196, 148, 115, 91, 74, 60, 50, 42]
    assert d3[0].tolist() == [1, -1, 3, -3, 5, -5, 7, -7]
    assert d3[15].tolist() == [1764, -1764, 5880, -5880, 10584, -10584, 16464, -16464]
    assert oracle.tables(2, 4)[1][15].tolist() == [3582, -3582, 12852, -12852]
    assert d4[15].tolist()[0::2] == [1148, 3825, 6885, 9945, 13005, 16065, 19125, 22950]
    assert oracle.tables(1, 4)[1][15].tolist() == [8192, -8192]


def test_dequant_closed_form(oracle):
    """SURVEY App. B closed form for b >= 3 holds for every scale_factor_bits the boundary accepts."""
    for s in range(1, 9):
        for b in range(3, 9):
            sf = oracle.scale_factors(b, s).astype(np.int64)
            _, d = oracle.tables(b, s)
            last = (1 << (b - 1)) - 1
            for k in range(last + 1):
                if k == 0:
                    mag = (3 * sf + 2) >> 2
                elif k == last:
                    mag = ((1 << b) - 1) * sf
                else:
                    mag = 2 * k * sf + ((sf + 1) >> 1)
                assert np.array_equal(d[:, 2 * k], mag) and np.array_equal(d[:, 2 * k + 1], -mag)


def test_quant_tab_appendix_d(oracle):
    assert oracle.quant_tab(3).tolist() == [7, 7, 7, 5, 5, 3, 3, 1, 0, 0, 2, 2, 4, 4, 6, 6, 6]
    assert oracle.quant_tab(2).tolist() == [3, 3, 1, 1, 0, 0, 0, 2, 2]
    assert oracle.quant_tab(1).tolist() == [1, 1, 0, 0, 0]


def test_vbr_plan_appendix_d(oracle):
    rows = {
        1.5: (1, [0, 214, 41, 1], [0, 426, 83, 3], [0, 1704, 332, 12]),
        2.0: (1, [0, 92, 156, 8], [0, 183, 313, 16], [0, 730, 1254, 64]),
        2.5: (2, [0, 214, 41, 1], [0, 426, 83, 3], [0, 1704, 332, 12]),
        3.0: (2, [0, 92, 156, 8], [0, 183, 313, 16], [0, 730, 1254, 64]),
        3.5: (3, [0, 214, 41, 1], [0, 426, 83, 3], [0, 1704, 332, 12]),
        4.0: (3, [0, 92, 157, 7], [0, 183, 314, 15], [0, 730, 1255, 63]),
        5.0: (4, [0, 92, 156, 8], [0, 183, 313, 16], [0, 730, 1254, 64]),
        6.0: (5, [0, 92, 156, 8], [0, 183, 313, 16], [0, 730, 1254, 64]),
        7.0: (6, [0, 92, 156, 8], [0, 183, 313, 16], [0, 730, 1254, 64]),
        7.3: (6, [0, 19, 226, 11], [0, 37, 452, 23], [0, 146, 1808, 94]),
    }
    for bits, (base, c256, c512, c2048) in rows.items():
        st = oracle.make_settings(bits, True)
        assert oracle.vbr_params(st, 256)[1:] == (base, c256)
        assert oracle.vbr_params(st, 512)[2] == c512
        assert oracle.vbr_params(st, 2048)[2] == c2048
    assert abs(oracle.vbr_params(oracle.make_settings(4.0, True), 256)[0] - 3.62499976) < 1e-7


def test_config1_file_size(oracle):
    """BASELINE config 1: 10 s 44.1 kHz stereo CBR 3 -> 22 + 86*4132 + 580 = 355954 bytes (SURVEY 8d)."""
    pcm = synth.gen_stream(0, 441000, 2, 44100)
    enc = oracle.sea_encode(pcm, 44100, 2, oracle.make_settings(3.0))
    assert len(enc) == 355954
    assert enc[6] | (enc[7] << 8) == 4132
    dec = oracle.sea_decode(enc)
    assert dec.samples.size == pcm.size and dec.channels == 2 and dec.sample_rate == 44100


def test_vbr_chunk_sizes(oracle):
    exp = {1.5: 1923, 2.0: 2563, 2.5: 3203, 3.0: 3843, 3.5: 4483, 4.0: 5120, 5.0: 6403, 6.0: 7683, 7.0: 8963, 7.3: 9345}
    pcm = synth.gen_stream(7, 5120, 2, 44100)
    for bits, size in exp.items():
        enc, ties = oracle.sea_encode(pcm, 44100, 2, oracle.make_settings(bits, True), return_ties=True)
        assert len(enc) == 22 + size and ties == 0
        assert np.array_equal(oracle.sea_decode(enc).samples.shape, pcm.shape)
    # mono config 2 chunk: 4 + 16 + 128 + 64 + 1710 = 1922
    enc = oracle.sea_encode(synth.gen_stream(8, 5120, 1, 48000), 48000, 1, oracle.make_settings(3.0, True))
    assert len(enc) == 22 + 1922


def test_vbr_outside_domain_panics(oracle):
    pcm = synth.gen_stream(7, 5120, 2, 44100)
    for bits in (8.0, 1.2):
        with pytest.raises(oracle.OracleError) as e:
            oracle.sea_encode(pcm, 44100, 2, oracle.make_settings(bits, True))
        assert e.value.code == oracle.ERR_PANIC


@pytest.mark.parametrize("channels,bits,sfb", [(1, 1, 4), (1, 3, 3), (2, 3, 4), (2, 8, 4), (3, 5, 5), (8, 4, 4), (2, 2, 4), (1, 6, 5),
                                               (4, 3, 4), (4, 7, 4), (6, 2, 4), (6, 5, 4), (8, 1, 4), (8, 8, 4), (5, 4, 4), (2, 5, 4), (2, 7, 3)])
def test_oracle_matches_reference_c_decoder(oracle, channels, bits, sfb):
    """CBR decode of the restatement == the reference's own c/sea.h (frames multiple of scale_factor_frames, c/sea.h:168).
    Without oracle/_ref: == the recorded result (util.reference_c_result); recorded from the oracle, that pins the oracle's
    decode against regressions only."""
    frames = 5120 * 2 + 1240
    pcm = gen_test_signal(channels, frames, seed=channels * 10 + bits)
    enc = oracle.sea_encode(pcm, 44100, channels, oracle.make_settings(float(bits), False, sfb))
    a = oracle.sea_decode(enc).samples
    assert sha(a) == reference_c_result(oracle, f"oracle_decode/ch{channels}_b{bits}_sf{sfb}", enc)


@pytest.mark.parametrize("channels,bits,sfb", [(1, 1, 4), (1, 3, 4), (2, 3, 4), (2, 5, 3), (2, 8, 5), (3, 4, 4), (8, 4, 4), (2, 2, 4), (2, 6, 4),
                                               (1, 7, 4)])
def test_reference_decoder_end_state_equals_next_chunk_header(oracle, channels, bits, sfb):
    """Pins the ENCODER's reconstruct/update path with reference code and no restatement in between: c/sea.h decodes the
    encoder's output, and the LMS state it holds when chunk k ends (captured before its free, c/sea.h:147-185, by
    oracle/ref_csea.c) must equal -- mod 2^16, lms.rs:64-78 -- the LMS block the encoder wrote into chunk k+1's header
    (file.rs:146-149).  The last four PCM samples c/sea.h emits per channel are chunk k+1's header history as well.
    Here for the oracle's encoder; tests/test_gpu_round2.py does the same for the GPU encoder.  Without oracle/_ref the state
    and PCM come from the record (util.reference_c_result); recorded from the oracle, that pins the encoder's bytes and the
    oracle's decode against regressions only."""
    frames = 5120 * 4 + 1000
    pcm = gen_test_signal(channels, frames, seed=channels * 10 + bits)
    enc = oracle.sea_encode(pcm, 44100, channels, oracle.make_settings(float(bits), False, sfb))
    pcm_sha, lms = reference_c_result(oracle, f"oracle_lms/ch{channels}_b{bits}_sf{sfb}", enc, lms=True)
    hdr = oracle.chunk_header_lms(enc)
    assert hdr.shape == (5, channels, 8) and lms.shape == (4, channels, 8)
    assert np.array_equal(lms, hdr[1:])
    pcm_out = oracle.sea_decode(enc).samples
    assert sha(pcm_out) == pcm_sha  # the PCM c/sea.h emits
    pcm_out = pcm_out.reshape(-1, channels)
    for k in range(1, 5):  # black-box: history of chunk k's header = the reference decoder's last four frames of chunk k-1
        assert np.array_equal(hdr[k][:, :4].T, pcm_out[k * 5120 - 4: k * 5120])
    assert np.array_equal(hdr[0][:, :4], np.zeros((channels, 4), dtype=np.int16))  # lms.rs:19-32 initial state
    assert np.array_equal(hdr[0][:, 4:], np.tile(np.array([0, 0, -8192, 16384], dtype=np.int16), (channels, 1)))


def test_golden_fixtures(oracle):
    meta = json.load(open(os.path.join(GOLD, "golden.json")))
    assert len(meta) >= 8
    for name, m in meta.items():
        pcm = synth.gen_stream(m["seed"], m["frames"], m["channels"], m["rate"]) if m["gen"] == "synth" else \
            gen_test_signal(m["channels"], m["frames"], m["rate"], m["seed"])
        assert sha(pcm) == m["pcm_sha"], name
        enc = oracle.sea_encode(pcm, m["rate"], m["channels"], oracle.make_settings(**m["settings"]))
        gold = open(os.path.join(GOLD, name + ".sea"), "rb").read()
        assert enc == gold and sha(gold) == m["sea_sha"], name
        assert sha(oracle.sea_decode(gold).samples) == m["dec_sha"], name


def test_sample_len_invariant(oracle):
    """tests/test.rs:8-33: decoded.len() == input.len() for lengths straddling multiples of 100, channels 1..3."""
    for channels in (1, 2, 3):
        for mul in (1, 2, 3, 100):
            for frames in range(max(mul * 100 - 2, 0), mul * 100 + 2):
                pcm = gen_test_signal(channels, frames)
                enc = oracle.sea_encode(pcm, 44100, channels, oracle.make_settings(3.0))
                assert oracle.sea_decode(enc).samples.size == pcm.size


def test_parameters_invariant(oracle):
    """tests/test.rs:35-64: channels 1..3 x sf_bits 3..5 x bits 1..8, rms < 0.2 (their 'psnr < -20')."""
    for channels in (1, 2, 3):
        pcm = gen_test_signal(channels, 11025)
        for sfb in (3, 4, 5):
            for bits in range(1, 9):
                enc = oracle.sea_encode(pcm, 44100, channels, oracle.make_settings(float(bits), False, sfb))
                dec = oracle.sea_decode(enc).samples
                assert dec.size == pcm.size
                rms = np.sqrt(np.mean(((dec.astype(np.float64) - pcm) / 32767.0) ** 2))
                assert rms < 0.2


def test_streaming_equals_one_shot(oracle):
    """tests/streaming.rs:51-97 restated on the oracle: chunk-at-a-time encoding == one-shot prefix."""
    pcm = gen_test_signal(1, 44100)
    st = oracle.make_settings(3.0)
    whole = oracle.sea_encode(pcm, 44100, 1, st)
    enc = oracle.StreamingEncoder(1, 44100, None, st)
    out, pos = enc.initial_bytes, 0
    for _ in range(4):
        more, b, used = enc.encode_frame(pcm[pos:])
        out += b
        pos += used
        assert more
    enc.close()
    # streaming header has total_frames == 0; everything after the 22-byte header is identical
    assert out[22:] == whole[22: len(out)]
    assert out[:14] == whole[:14] and out[14:18] == b"\0\0\0\0"


def test_empty_and_tiny_inputs(oracle):
    st = oracle.make_settings(3.0)
    enc = oracle.sea_encode(np.zeros(0, np.int16), 44100, 2, st)
    assert len(enc) == 22 and enc[6] == 0 and enc[7] == 0  # header only, chunk_size 0
    enc = oracle.sea_encode(np.array([5, -7], np.int16), 44100, 2, st)  # one frame
    assert oracle.sea_decode(enc).samples.size == 2
