"""GPU encoder against oracle.sea_encode, byte for byte, on the crafted inputs of tests/enc_crafted.py (which
tests/test_enc_mirror.py shows reach the speculative 32-bit penalty form's rollback and skip window, a proof that fails in one
chain of a warp, the exact 64-bit arg-min, rotated rank ties, and at CBR 3 the direct quantiser's 64-bit form where prior32 fails):
every fast CBR instance under both lane mappings, the VBR
instances under each dequant-table layout, both VBR sorts, the generic search pass and every host route.  Every VBR case also
checks the boundary-tie counts against the oracle's."""
import io
import os

import numpy as np
import pytest

import enc_crafted as G
import enc_mirror as M
import sea_codec_b200 as S

pytestmark = pytest.mark.gpu

NAMES = list(G.RECIPES)


@pytest.fixture
def env():
    """Set encoder knobs for one test; every one is restored afterwards."""
    saved = {}

    def put(k, v):
        saved.setdefault(k, os.environ.get(k))
        if v is None:
            os.environ.pop(k, None)
        else:
            os.environ[k] = v

    yield put
    for k, v in saved.items():
        if v is None:
            os.environ.pop(k, None)
        else:
            os.environ[k] = v


def _pair(oracle, **kw):
    return S.EncoderSettings(**kw), oracle.make_settings(**kw)


def _inputs(channels):
    return [G.crafted(n, channels) for n in NAMES]


@pytest.mark.parametrize("s", [3, 4, 5])
@pytest.mark.parametrize("split", ["0", "1"])
def test_fast_cbr_instances_match_the_oracle(ctx, oracle, env, s, split):
    """encode_kernel<FB, S> for FB 1-8: 1-16 channels (with the split mapping 9-16 channels loop over the 8 warps)."""
    env("SEA_B200_ENC_SPLIT", split)
    for channels in (1, 2, 3, 5, 8, 9, 16):
        xs = _inputs(channels)
        for fb in range(1, 9):
            st, ost = _pair(oracle, residual_bits=float(fb), scale_factor_bits=s, frames_per_chunk=400)
            refs = [oracle.sea_encode(x, 44100, channels, ost) for x in xs]
            got = ctx.encode_batch(xs, 44100, channels, st)
            for name, g, r in zip(NAMES, got, refs):
                assert g == r, (name, channels, fb, s, split)


@pytest.mark.parametrize("s", [3, 4, 5])
@pytest.mark.parametrize("lut", ["32", "16", "global"])
def test_vbr_instances_match_the_oracle_under_each_pinned_layout(ctx, oracle, env, s, lut):
    """SEA_B200_ENC_LUT pins the layout of the VBR dequant table; 16 applies at s = 4 only (elsewhere the natural choice stands)."""
    env("SEA_B200_ENC_LUT", lut)
    for channels in (1, 2, 3):
        xs = _inputs(channels)
        for bits in (2.5, 4.5, 7.3):
            st, ost = _pair(oracle, residual_bits=bits, vbr=True, scale_factor_bits=s, frames_per_chunk=400)
            assert M.enc_lut_mode(1, ost, channels, pin=lut) == ({"32": 0, "16": 1 if s == 4 else 0, "global": 2}[lut])
            for name, x in zip(NAMES, xs):
                ref, ties = oracle.sea_encode(x, 44100, channels, ost, return_ties=True)
                assert ctx.sea_encode(x, 44100, channels, st) == ref, (name, channels, bits, s, lut)
                assert ctx.last_vbr_ties == ties
            got = ctx.encode_batch(xs, 44100, channels, st)
            assert got == [oracle.sea_encode(x, 44100, channels, ost) for x in xs], (channels, bits, s, lut)


@pytest.mark.parametrize("s,bits,n,pin,want", [(4, 4.5, 1024, None, M.ENC_LUT16), (4, 7.3, 444, None, M.ENC_LUT16),
                                               (3, 5.5, 740, None, M.ENC_LUT_GLOBAL), (5, 4.5, 1024, None, M.ENC_LUT_GLOBAL),
                                               (4, 5.5, 1024, None, M.ENC_LUT_GLOBAL), (4, 4.5, 1024, "32", M.ENC_LUT32),
                                               (5, 4.5, 1024, "32", M.ENC_LUT32), (4, 5.5, 1024, "16", M.ENC_LUT16)])
def test_vbr_layouts_chosen_by_batch_size_match_the_oracle(ctx, oracle, env, s, bits, n, pin, want):
    """Unpinned, the batch size alone moves the table to [code][sf] or global memory (as the benchmark's 1024 streams do); pinned,
    SEA_B200_ENC_LUT overrides that choice on the same large batch."""
    env("SEA_B200_ENC_LUT", pin)
    st, ost = _pair(oracle, residual_bits=bits, vbr=True, scale_factor_bits=s)
    assert M.enc_lut_mode(n, ost, 2, pin=pin) == want
    xs = [np.resize(G.crafted(name, 2).reshape(-1, 2), (1000 + 37 * i, 2)).reshape(-1) for i, name in enumerate(NAMES)]
    refs = [oracle.sea_encode(x, 44100, 2, ost, return_ties=True) for x in xs]
    got = ctx.encode_batch([xs[i % len(xs)] for i in range(n)], 44100, 2, st)
    ties = ctx.last_vbr_ties_per_stream(n)
    for i, g in enumerate(got):
        assert g == refs[i % len(xs)][0], (i, s, bits, n, pin)
        assert ties[i] == refs[i % len(xs)][1], (i, s, bits, n, pin)
    assert ctx.last_vbr_ties == sum(refs[i % len(xs)][1] for i in range(n))


@pytest.mark.parametrize("channels", [2, 3])
def test_vbr_sort_paths_and_ragged_chunks(ctx, oracle, env, channels):
    """Stereo 5120-frame chunks sort 512 items in registers; 3 channels (768) take bitonic_sort; ragged last chunks."""
    env("SEA_B200_ENC_LUT", None)
    for s, bits in ((3, 3.0), (4, 4.5), (5, 7.3)):
        st, ost = _pair(oracle, residual_bits=bits, vbr=True, scale_factor_bits=s)
        for name in ("refail", "saturated", "phase"):
            x = np.resize(G.crafted(name, channels).reshape(-1, channels), (5120 * 2 + 333, channels)).reshape(-1)
            ref, ties = oracle.sea_encode(x, 44100, channels, ost, return_ties=True)
            assert ctx.sea_encode(x, 44100, channels, st) == ref, (name, s, bits)
            assert ctx.last_vbr_ties == ties


def test_generic_search_pass_matches_the_oracle(ctx, oracle):
    """search_pass: scale_factor_bits 2 and 6, scale_factor_frames 10 and 32, and 17 channels."""
    cases = [(2, dict(residual_bits=3.0, scale_factor_bits=2, frames_per_chunk=400)),
             (2, dict(residual_bits=5.0, scale_factor_bits=6, frames_per_chunk=400)),
             (2, dict(residual_bits=4.0, scale_factor_frames=10, frames_per_chunk=400)),
             (2, dict(residual_bits=3.0, vbr=True, scale_factor_frames=32, frames_per_chunk=320)),
             (1, dict(residual_bits=4.5, vbr=True, scale_factor_bits=6, frames_per_chunk=400)),
             (17, dict(residual_bits=3.0, frames_per_chunk=400)),
             (17, dict(residual_bits=3.0, vbr=True, frames_per_chunk=400))]
    for channels, kw in cases:
        st, ost = _pair(oracle, **kw)
        for name in NAMES:
            x = G.crafted(name, channels)
            ref, ties = oracle.sea_encode(x, 44100, channels, ost, return_ties=True)
            assert ctx.sea_encode(x, 44100, channels, st) == ref, (name, channels, kw)
            assert ctx.last_vbr_ties == ties


@pytest.mark.parametrize("kw", [dict(residual_bits=4.0), dict(residual_bits=2.0, scale_factor_bits=3), dict(residual_bits=4.5, vbr=True)])
def test_every_host_route_matches_the_oracle(ctx, oracle, env, kw):
    """One-shot, encode_batch in forced 1- and 2-chunk slices, the streaming encoder and encode_batch_device."""
    import torch

    ch = 2
    st, ost = _pair(oracle, frames_per_chunk=400, **kw)
    xs = [np.tile(G.crafted(name, ch).reshape(-1, ch), (3, 1))[: 1150 + 10 * i].reshape(-1) for i, name in enumerate(NAMES)]
    refs, ref_ties = zip(*[oracle.sea_encode(x, 44100, ch, ost, return_ties=True) for x in xs])
    refs, ref_ties = list(refs), list(ref_ties)
    vbr = bool(kw.get("vbr"))
    for x, r, rt in zip(xs, refs, ref_ties):
        assert ctx.sea_encode(x, 44100, ch, st) == r
        assert not vbr or ctx.last_vbr_ties == rt
    for k in ("0", "1", "2"):
        env("SEA_B200_ENC_SLICE", k)
        assert ctx.encode_batch(xs, 44100, ch, st) == refs, k
        assert not vbr or list(ctx.last_vbr_ties_per_stream(len(xs))) == ref_ties, k
    env("SEA_B200_ENC_SLICE", None)
    for x, r in zip(xs[:3], refs[:3]):
        sink = io.BytesIO()
        enc = S.SeaEncoder(ch, 44100, x.size // ch, st, io.BytesIO(x.astype("<i2").tobytes()), sink, ctx=ctx)
        while enc.encode_frame():
            pass
        enc.finalize()
        assert sink.getvalue() == r
    frames = np.array([x.size // ch for x in xs])
    pcm_off = np.concatenate([[0], np.cumsum(frames * ch)[:-1]])
    pcm = torch.from_numpy(np.concatenate(xs)).to("cuda:0")
    bound = max(ctx.encode_bound(int(f), ch, st) for f in frames)
    stride = (bound + 15) // 16 * 16
    out = torch.zeros(len(xs) * stride, dtype=torch.uint8, device="cuda:0")
    torch.cuda.synchronize()
    lens = ctx.encode_batch_device(pcm.data_ptr(), pcm_off, frames, 44100, ch, st, out.data_ptr(), np.arange(len(xs)) * stride)
    host = out.cpu().numpy()
    for i, r in enumerate(refs):
        assert host[i * stride: i * stride + int(lens[i])].tobytes() == r, NAMES[i]
    assert not vbr or list(ctx.last_vbr_ties_per_stream(len(xs))) == ref_ties
