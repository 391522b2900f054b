"""Regenerates tests/golden/*.sea and golden.json with the CPU oracle (and cross-checks CBR decodes with the reference's
own C decoder c/sea.h from oracle/_ref).  Run from the repo root: python tests/golden/make_golden.py

python tests/golden/make_golden.py reference_c  writes reference_c.json instead: what c/sea.h makes of the inputs of the tests
that compare with it (util.reference_c_result), so that they run where oracle/_ref cannot be built.  It needs oracle/_ref.
With --from-oracle and no oracle/_ref it records the oracle's decode and the chunk-header LMS instead and says so in the file's
"source": a record of the code under test, so never re-record that way to make a failing comparison pass.

The reference holds no golden vectors of its own (SURVEY.md 8c); these fixtures pin (a) the oracle against regressions and
(b) the CUDA path on the GPU box, where /root/reference does not exist.
"""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from oracle import sea_oracle as O  # noqa: E402
from sea_codec_b200 import synth  # noqa: E402
from util import gen_test_signal, sha  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))

CASES = [
    # name, generator, stream/seed, frames, channels, rate, settings kwargs
    ("stereo_cbr3", "synth", 0, 12000, 2, 44100, dict(residual_bits=3.0)),
    ("mono_vbr3", "synth", 1, 11111, 1, 48000, dict(residual_bits=3.0, vbr=True)),
    ("ch3_cbr5_sf5", "helpers", 3, 7000, 3, 44100, dict(residual_bits=5.0, scale_factor_bits=5)),
    ("ch8_cbr4", "synth", 2, 6000, 8, 48000, dict(residual_bits=4.0)),
    ("stereo_vbr45", "synth", 4, 10300, 2, 44100, dict(residual_bits=4.5, vbr=True)),
    ("mono_cbr1", "synth", 5, 3000, 1, 44100, dict(residual_bits=1.0)),
    ("mono_cbr8", "synth", 6, 3000, 1, 44100, dict(residual_bits=8.0)),
    ("stereo_cbr2_sf3_f10", "helpers", 7, 5000, 2, 44100, dict(residual_bits=2.0, scale_factor_bits=3, scale_factor_frames=10, frames_per_chunk=1000)),
]


def make_pcm(gen, seed, frames, channels, rate):
    if gen == "synth":
        return synth.gen_stream(seed, frames, channels, rate)
    return gen_test_signal(channels, frames, rate, seed)


def main():
    meta = {}
    for name, gen, seed, frames, ch, rate, kw in CASES:
        pcm = make_pcm(gen, seed, frames, ch, rate)
        st = O.make_settings(**kw)
        enc, ties = O.sea_encode(pcm, rate, ch, st, return_ties=True)
        dec = O.sea_decode(enc).samples
        entry = dict(gen=gen, seed=seed, frames=frames, channels=ch, rate=rate, settings=kw, pcm_sha=sha(pcm), sea_sha=sha(enc),
                     sea_len=len(enc), dec_sha=sha(dec), vbr_ties=ties, cref_checked=False)
        if not kw.get("vbr") and frames % kw.get("scale_factor_frames", 20) == 0 and O.have_ref():
            cref = O.ref_c_decode(enc).samples
            assert np.array_equal(cref, dec), name
            entry["cref_checked"] = True
        assert ties == 0, (name, ties)
        with open(os.path.join(HERE, name + ".sea"), "wb") as f:
            f.write(enc)
        meta[name] = entry
        print(name, len(enc), entry["cref_checked"])
    with open(os.path.join(HERE, "golden.json"), "w") as f:
        json.dump(meta, f, indent=1, sort_keys=True)


# the inputs of the four comparisons with c/sea.h: key -> (pcm, channels, settings, capture LMS)
def reference_c_cases():
    for ch, b, sfb in ((1, 1, 4), (1, 3, 3), (2, 3, 4), (2, 8, 4), (3, 5, 5), (8, 4, 4), (2, 2, 4), (1, 6, 5), (4, 3, 4), (4, 7, 4), (6, 2, 4),
                       (6, 5, 4), (8, 1, 4), (8, 8, 4), (5, 4, 4), (2, 5, 4), (2, 7, 3)):  # test_oracle_matches_reference_c_decoder
        yield f"oracle_decode/ch{ch}_b{b}_sf{sfb}", gen_test_signal(ch, 5120 * 2 + 1240, seed=ch * 10 + b), ch, (float(b), False, sfb), False
    for ch, b, sfb in ((1, 1, 4), (1, 3, 4), (2, 3, 4), (2, 5, 3), (2, 8, 5), (3, 4, 4), (8, 4, 4), (2, 2, 4), (2, 6, 4),
                       (1, 7, 4)):  # test_reference_decoder_end_state_equals_next_chunk_header
        yield f"oracle_lms/ch{ch}_b{b}_sf{sfb}", gen_test_signal(ch, 5120 * 4 + 1000, seed=ch * 10 + b), ch, (float(b), False, sfb), True
    # test_gpu_cbr_decode_against_the_reference_c_decoder, and (3, 3) for test_latency_kernel_cbr_and_vbr, which calls it with
    # bits 3 (4 for 8 channels) for each of its channel counts
    for ch, b in ((1, 3), (2, 1), (2, 3), (2, 8), (4, 4), (6, 2), (8, 4), (3, 5), (3, 3)):
        yield f"gpu_cbr_decode/ch{ch}_b{b}", synth.gen_stream(700 + ch * 10 + b, 5120 * 3 + 2000, ch, 44100), ch, (float(b),), False
    for ch in (1, 2, 3, 8):  # test_gpu_encoder_lms_against_the_reference_decoder (the GPU encoder writes the oracle's bytes)
        for b in range(1, 9):
            yield f"gpu_encoder_lms/ch{ch}_b{b}", synth.gen_stream(900 + ch * 10 + b, 5120 * 4 + 1000, ch, 44100), ch, (float(b),), True


def main_reference_c(from_oracle: bool):
    have_ref = O.have_ref()
    if not have_ref and not from_oracle:
        sys.exit("oracle/_ref (c/sea.h) is not built: reference_c.json is left as it is (--from-oracle records the oracle instead)")
    cases = {}
    for key, pcm, ch, st, lms in reference_c_cases():
        enc = O.sea_encode(pcm, 44100, ch, O.make_settings(*st))
        if have_ref:
            if lms:
                info, states = O.ref_c_decode_lms(enc)
                states = states[:-1].astype(np.int16)
            else:
                info = O.ref_c_decode(enc)
            dec = info.samples
        else:
            dec = O.sea_decode(enc).samples
            states = O.chunk_header_lms(enc)[1:]
        cases[key] = dict(sea_sha=sha(enc), pcm_sha=sha(dec), **({"lms": states.tolist()} if lms else {}))
    source = "c/sea.h (oracle/_ref)" if have_ref else (
        "the oracle, not c/sea.h (oracle/_ref was not built): the oracle's decode and the oracle encoder's chunk-header LMS; "
        "where oracle/_ref is built the tests check every value against c/sea.h")
    with open(os.path.join(HERE, "reference_c.json"), "w") as f:  # one case per line
        body = ",\n".join(f"{json.dumps(k)}: {json.dumps(v, sort_keys=True)}" for k, v in sorted(cases.items()))
        f.write(f'{{"source": {json.dumps(source)},\n"cases": {{\n{body}\n}}}}\n')
    print(len(cases), "cases from", source)


if __name__ == "__main__":
    if sys.argv[1:2] == ["reference_c"]:
        main_reference_c("--from-oracle" in sys.argv[2:])
    else:
        main()
