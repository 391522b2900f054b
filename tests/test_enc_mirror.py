"""CPU tests of the encoder mirror (tests/enc_mirror.py) and of the crafted inputs (tests/enc_crafted.py): the mirror equals
oracle.sea_encode byte for byte, every crafted input reaches the encoder path it was made for, and the margin that keeps the
GPU's full-length candidate trials (no early exit) equal to the reference is measured.  No GPU needed."""
import numpy as np
import pytest

import enc_crafted as G
import enc_mirror as M

CBR = [dict(residual_bits=float(b), scale_factor_bits=s, frames_per_chunk=400) for s in (3, 4, 5) for b in (1, 2, 3, 4, 8)]
VBR = [dict(residual_bits=b, vbr=True, scale_factor_bits=s, frames_per_chunk=400) for s, b in ((3, 3.0), (4, 2.5), (4, 5.5), (5, 7.3))]
GENERIC = [dict(residual_bits=3.0, scale_factor_bits=2, frames_per_chunk=400), dict(residual_bits=5.0, scale_factor_bits=6, frames_per_chunk=400),
           dict(residual_bits=4.0, scale_factor_frames=10, frames_per_chunk=400), dict(residual_bits=3.0, vbr=True, scale_factor_frames=32, frames_per_chunk=320)]


def _run(oracle, name, channels, kw):
    st = oracle.make_settings(**kw)
    x = G.crafted(name, channels)
    return x, st, M.encode(x, channels, st)


@pytest.mark.parametrize("kw", CBR + VBR + GENERIC, ids=lambda kw: "-".join(f"{k[:4]}{v}" for k, v in kw.items()))
def test_mirror_equals_the_oracle_on_every_crafted_input(oracle, kw):
    for name in G.RECIPES:
        for channels in ((1, 2) if kw.get("frames_per_chunk") == 400 and not kw.get("vbr") else (2,)):
            x, st, r = _run(oracle, name, channels, kw)
            ref, ties = oracle.sea_encode(x, 44100, channels, st, return_ties=True)
            assert r.data == ref, (name, channels, kw)
            assert r.ties == ties, (name, channels, kw)


def test_mirror_equals_the_oracle_on_ragged_and_multichannel_inputs(oracle):
    for channels, frames, kw in ((3, 1037, dict(residual_bits=3.0, frames_per_chunk=400)),
                                 (3, 845, dict(residual_bits=4.5, vbr=True, frames_per_chunk=400)),
                                 (17, 400, dict(residual_bits=3.0, frames_per_chunk=400)),
                                 (1, 5120 + 33, dict(residual_bits=3.0, vbr=True))):
        x = np.resize(G.crafted("phase", channels).reshape(-1, channels), (frames, channels)).reshape(-1)
        st = oracle.make_settings(**kw)
        assert M.encode(x, channels, st).data == oracle.sea_encode(x, 44100, channels, st), (channels, frames, kw)


def _rollbacks(oracle, name, channels, bits, s=4):
    kw = dict(residual_bits=float(bits), scale_factor_bits=s, frames_per_chunk=400)
    _, st, r = _run(oracle, name, channels, kw)
    return M.warp_trace(r, channels, st), r


@pytest.mark.parametrize("s", [3, 4, 5])
@pytest.mark.parametrize("bits", [4, 8])
def test_crafted_inputs_reach_the_speculative_penalty_edges(oracle, s, bits):
    """try32: a failure in the middle of a chunk, another right after the 8-block skip window, none while the window runs."""
    wt, _ = _rollbacks(oracle, "mid_fail", 1, bits, s)
    assert [b.blk for b in wt if b.rollback] == [6]
    assert [b.spec_skip for b in wt[7:16]] == [8, 7, 6, 5, 4, 3, 2, 1, 0]
    assert not any(b.tried32 for b in wt[7:15]) and wt[15].tried32 and wt[15].form == "sum32"
    assert all(b.form == "sum32" for b in wt[:6])
    wt, _ = _rollbacks(oracle, "refail", 1, bits, s)
    assert [b.blk for b in wt if b.rollback] == [6, 15]
    assert wt[16].spec_skip == 8 and wt[16].form == "narrow"


@pytest.mark.parametrize("s,channels", [(3, 2), (3, 4), (4, 2)])
def test_crafted_input_fails_the_proof_in_one_chain_of_a_warp_only(oracle, s, channels):
    """The vote covers every chain of the warp (2 at S = 4, 4 at S = 3): one failing chain rolls back all of them."""
    wt, r = _rollbacks(oracle, "one_chain", channels, 4, s)
    hit = [b for b in wt if b.split_chain_fail]
    assert len(hit) == 1 and hit[0].blk == 3 and hit[0].rollback
    fails = {b.ch for b in r.blocks if b.blk == 3 and not b.proof_ok}
    assert fails == {0}
    # with one chain per warp (the split mapping) only channel 0's warp rolls back
    split = M.warp_trace(r, channels, r_settings(oracle, 4, s), split=True)
    assert {b.chains for b in split if b.rollback and b.blk == 3} == {(0,)}


def r_settings(oracle, bits, s):
    return oracle.make_settings(float(bits), scale_factor_bits=s, frames_per_chunk=400)


@pytest.mark.parametrize("s", [3, 4, 5])
def test_crafted_inputs_reach_every_arg_min_form_that_pcm_can(oracle, s):
    """saturated: every block takes the exact 64-bit arg-min; the others mix it with the single redux.  No PCM input we found
    reaches a rank of 2^(64 - s) (the explicit compare): see test_no_candidate_rank_can_wrap."""
    for bits in (1, 3, 4, 8):
        wt, r = _rollbacks(oracle, "saturated", 2, bits, s)
        assert all(b.argmin == "butterfly" for b in wt) and len(wt) >= 20
        assert all(b.min_rank >= M.KSAT for b in r.blocks)
        wt, _ = _rollbacks(oracle, "ties", 2, bits, s)
        forms = {b.argmin for b in wt}
        assert forms == {"redux", "butterfly"}, forms


@pytest.mark.parametrize("s,bits,want", [(3, 3, 14), (4, 4, 4), (5, 8, 12)])
def test_crafted_input_ties_the_minimum_with_a_rotated_order(oracle, s, bits, want):
    """Exact ties of the smallest rank where prev != 0: the winner is the first candidate of the rotated visiting order."""
    _, r = _rollbacks(oracle, "ties", 2, bits, s)
    tied = [b for b in r.blocks if b.ties > 1 and b.prev != 0]
    assert len(tied) == want
    for b in tied:  # the first of the tied candidates in the visiting order rotated by prev
        assert b.winner == min(b.tied, key=lambda sf: (sf - b.prev) % (1 << s))
    assert all(b.winner == b.gpu_winner for b in r.blocks)


def _prior32_fraction(r, bits, s):
    """The largest sum_i (|w_i| + 20 * max|delta|)^2 of any block as a fraction of 2^32 (prior32 holds below 1)."""
    _, dqt, _ = M.tables(bits, s)
    lv = {1: 0, 2: 1, 3: 3}[bits]
    grow = max(20 * ((int(dqt[sf, 2 * lv]) + 15) >> 4) for sf in range(1 << s))
    return max(sum((abs(v) + grow) ** 2 for v in b.w0) for b in r.blocks) / 2 ** 32


@pytest.mark.parametrize("s,want", [(3, 123), (4, 190), (5, 154)])
def test_crafted_input_makes_prior32_false_at_cbr3(oracle, s, want):
    """CBR sizes 1-3 take the 32-bit penalty form from a bound checked before the trial.  Three full-scale tones push the
    weights past 20,000 and that bound fails at CBR 3: those blocks run the 64-bit (narrow) form of the direct-quantiser
    instance, with no speculative trial."""
    wt, r = _rollbacks(oracle, "tones", 1, 3, s)
    off = [b for b in wt if b.nf == 20 and b.form != "prior32"]
    assert len(off) == want
    assert all(b.form == "narrow" and not b.tried32 and not b.rollback for b in off)
    assert _prior32_fraction(r, 3, s) > 1.0


def test_prior32_margin_at_cbr1_and_cbr2(oracle):
    """At CBR 1 and 2 no crafted input makes prior32 false: the largest sum of squares over every recipe stays below 2^32
    (the tones reach 0.91 of it at CBR 2, s = 5).  Recorded so that a change which narrows the margin shows up."""
    worst = {}
    for bits in (1, 2):
        for s in (3, 4, 5):
            for name in ("tones", "runaway", "saturated"):
                wt, r = _rollbacks(oracle, name, 1, bits, s)
                assert all(b.form == "prior32" for b in wt if b.nf == 20), (name, bits, s)
                worst[bits] = max(worst.get(bits, 0.0), _prior32_fraction(r, bits, s))
    assert 0.4 < worst[1] < 0.5 and 0.85 < worst[2] < 1.0, worst


def test_runaway_weights_stay_narrow(oracle):
    """The weights the crafted inputs push the search to: past the initial 2^14, below 2^15 and far below 2^23
    (weights_stay_narrow): no block takes the wide 64-bit form."""
    wmax = 0
    for name in ("runaway", "tones"):
        for bits in (1, 3, 4, 8):
            wt, r = _rollbacks(oracle, name, 1, bits)
            wmax = max(wmax, max(b.max_w for b in r.blocks))
            assert all(b.form != "wide" for b in wt)
    assert 24000 < wmax < 2 ** 15


def _wrap_bound(m0):
    """The largest rank a 20-frame block can reach when every weight starts at most m0: each frame adds err^2 < 2^32 and the
    penalty of weights that moved by at most |d >> 4| <= 1578 per frame (|d| <= 255 * 99, dqt.rs)."""
    x = m0 + 20 * 1578
    return 20 * ((1 << 32) + max(0, (4 * x * x >> 18) - 0x8FF) ** 2)


def test_no_candidate_rank_can_wrap(oracle):
    """The reference stops a candidate once its partial rank passes the best so far; the GPU runs every candidate in full.
    The two agree unless a full rank wraps past 2^64.  Over every crafted input and setting: no rank wrapped, the early exit
    never changed a winner, the largest candidate rank stays below 2^37 and the largest chain weight (~24,500, from the
    full-scale tones) leaves a factor of > 300 to the 7.9 M at which _wrap_bound first reaches 2^64 (DESIGN 4.2)."""
    assert _wrap_bound(7_901_905) < 1 << 64 <= _wrap_bound(7_901_906)
    worst_rank, worst_m0, worst_w = 0.0, 0, 0
    for kw in CBR + VBR[:2]:
        for name in G.RECIPES:
            _, _, r = _run(oracle, name, 2, kw)
            for b in r.blocks:
                assert not b.wrapped and b.winner == b.gpu_winner, (name, kw, b)
                assert b.exact_max_rank < _wrap_bound(b.m0)
            worst_rank = max(worst_rank, max(b.exact_max_rank for b in r.blocks))
            worst_m0 = max(worst_m0, max(b.m0 for b in r.blocks))
            worst_w = max(worst_w, max(b.max_w for b in r.blocks))
    assert worst_rank < 2.0 ** 37
    assert 24000 < worst_m0 and worst_m0 * 300 < 7_901_905 and worst_w < 2 ** 15
    assert _wrap_bound(worst_m0) < 2.0 ** 38


@pytest.mark.parametrize("kw,channels,want_sorts", [
    (dict(residual_bits=3.0, vbr=True), 2, {"register"}),        # 5120 frames: 512 items
    (dict(residual_bits=3.0, vbr=True), 3, {"bitonic"}),         # 768 items
    (dict(residual_bits=3.0, vbr=True, frames_per_chunk=400), 2, {"register"}),
])
def test_vbr_sort_paths(oracle, kw, channels, want_sorts):
    st = oracle.make_settings(**kw)
    N = kw.get("frames_per_chunk", 5120)
    x = np.resize(G.crafted("phase", channels).reshape(-1, channels), (N + 333, channels)).reshape(-1)
    r = M.encode(x, channels, st)
    assert r.data == oracle.sea_encode(x, 44100, channels, st)
    paths = {"register" if np2 <= 512 and mx < M.SORT_KEY_LIMIT else "bitonic" for _, _, np2, mx in r.sorts[:1]}
    assert paths == want_sorts
    assert all(mx < M.SORT_KEY_LIMIT for *_, mx in r.sorts)  # the register sort's overflow fallback is out of reach too
    assert r.sorts[-1][1] == (333 * channels) // 20  # the ragged last chunk sorts its whole blocks only


def test_enc_lut_mode_restates_the_host_rule(oracle):
    """400 streams at VBR 3 keep the per-lane layout; at the benchmark's 1024 streams VBR 4.5 needs the shared [code][sf] layout
    (s = 4) or global memory (s = 3, 5), and VBR 5.5 global memory; a pinned layout applies where it fits."""
    st = lambda b, s=4: oracle.make_settings(b, True, s)
    assert M.enc_lut_mode(400, st(3.0), 2) == M.ENC_LUT32
    assert M.enc_lut_mode(1024, st(3.0), 2) == M.ENC_LUT32
    assert M.enc_lut_mode(1024, st(4.5), 2) == M.ENC_LUT16
    assert M.enc_lut_mode(1024, st(4.5, 3), 2) == M.ENC_LUT_GLOBAL
    assert M.enc_lut_mode(1024, st(4.5, 5), 2) == M.ENC_LUT_GLOBAL
    assert M.enc_lut_mode(1024, st(5.5), 2) == M.ENC_LUT_GLOBAL
    assert M.enc_lut_mode(444, st(7.3), 2) == M.ENC_LUT16
    assert M.enc_lut_mode(1, st(3.0), 2, pin="16") == M.ENC_LUT16
    assert M.enc_lut_mode(1, st(3.0, 5), 2, pin="16") == M.ENC_LUT32   # 16 needs s = 4: the natural choice stands
    assert M.enc_lut_mode(1, st(7.3), 2, pin="global") == M.ENC_LUT_GLOBAL
    assert M.enc_lut_mode(1024, st(7.3), 2, pin="32") == M.ENC_LUT32


def test_search_finds_a_recipe_for_a_target(oracle):
    """search() (how the runaway recipe was found): greedy toward a 32-bit proof failure in the block after six quiet ones."""
    st = oracle.make_settings(4.0, frames_per_chunk=400)
    rec = G.search(lambda tr: 0 if tr[-1][0]["proof_ok"] else 1, 1, 1, st, start=["tone"] * 6)
    assert len(rec) == 1 and rec[0] in G.MENU
    x = G.pcm(["tone"] * 6 + rec + ["tone"] * 3, 1, 7)
    r = M.encode(x, 1, st)
    assert r.data == oracle.sea_encode(x, 44100, 1, st)
    assert [b.blk for b in M.warp_trace(r, 1, st) if b.rollback] == [6]
