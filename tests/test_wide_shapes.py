"""CPU checks of tests/wide_shapes.py: the oracle takes every wide shape and writes the chunk sizes the plan restatement says,
the shapes reach the code paths they are there for, and the encoder's shared-memory sizing fits every accepted setting."""
import numpy as np
import pytest

import wide_shapes as W
from oracle import sea_oracle as O

IDS = [sh.id for sh in W.SHAPES]

# Settings make_encode_plan accepts whose encoder CTA took more than 200 KB before the chunk buffer and the warp count were fitted
# (launch_encode_generic returned cudaErrorInvalidConfiguration): (channels, s, F, bits, vbr, N, shared memory then)
OVER_200K = [(255, 4, 255, 7.0, False, 255, 209036), (255, 4, 255, 1.0, False, 1785, 209800), (160, 1, 255, 1.0, False, 3060, 205468),
             (200, 8, 255, 1.0, False, 2295, 206564), (100, 2, 255, 5.5, True, 765, 206076), (8, 5, 255, 4.5, True, 14535, 218872)]


def pcm(shape, seed=0):
    """Noise with a loud square on every fourth channel and a phase-inverted copy of channel 0 on channel 1."""
    rng = np.random.default_rng(seed + shape.channels)
    x = rng.integers(-3000, 3000, (shape.frames, shape.channels))
    t = np.arange(shape.frames)
    x[:, ::4] = np.where((t // 7) % 2 == 0, 32767, -32768)[:, None]
    if shape.channels > 1:
        x[:, 1] = np.clip(-x[:, 0], -32768, 32767)
    return x.astype(np.int16).reshape(-1)


def test_shapes_cover_the_settings_space():
    sh = W.SHAPES
    assert {9, 15, 16, 17, 31, 32, 33, 64, 100, 128, 129, 200, 255} <= {x.channels for x in sh}
    assert {x.s for x in sh} == set(range(1, 9))
    assert {1, 7, 8} <= {x.s for x in sh if x.channels >= 9}
    assert {1, 7, 20, 64, 255} <= {x.F for x in sh}
    assert {int(x.bits) for x in sh if not x.vbr} == set(range(1, 9))
    rates = [x.bits for x in sh if x.vbr]
    assert min(rates) == 1.5 and max(rates) == 7.3
    assert sum(x.plan().full_chunk_bytes >= 0.99 * 65535 for x in sh) >= 5
    assert all(x.frames % x.N for x in sh), "every stream ends in a ragged chunk"
    assert sum(x.frames % x.N % x.F != 0 for x in sh) >= 10, "and most in a ragged block"
    assert all(x.plan() is not None for x in sh)
    assert [x.id for x in sh if not x.decodable] == ["c255_s1_F1_vbr7.3_N257"]


def test_shapes_reach_their_routes():
    for x in W.SHAPES:
        p = x.plan()
        lat = W.latency_smem(p.full_chunk_bytes, x.N, x.channels)
        if x.channels > 32:
            assert lat == 0 and W.decode_route(x.channels, x.N, p.full_chunk_bytes, x.F, x.s, p.hdr_bits, x.vbr, 1, "1") == "generic"
        if x.channels >= 9:
            assert W.decode_route(x.channels, x.N, p.full_chunk_bytes, x.F, x.s, p.hdr_bits, x.vbr, 1, "0") == "generic"
    eligible = {x.channels for x in W.SHAPES if W.latency_smem(x.plan().full_chunk_bytes, x.N, x.channels)}
    assert {9, 15, 17, 32} <= eligible, eligible
    # the small-job kernel's own limit: 32 channels, whatever the chunk
    assert W.latency_smem(100, 20, 32) and not W.latency_smem(100, 20, 33)


def test_planar_window_tiles():
    assert [W.tile_frames_log2(c) for c in (9, 16, 17, 32, 33, 64, 65, 128, 129, 255)] == [8, 8, 7, 7, 6, 6, 5, 5, 5, 5]
    for c in range(1, 256):
        assert (1 << W.tile_frames_log2(c)) * c <= max(4096, 32 * c)
        assert W.tile_staged_elems(c) <= W.WIN_TILE_ELEMS, c
    assert W.tile_staged_elems(255) == 8168


def test_vbr_shapes_reach_global_scratch_and_the_65536_key_sort():
    vbr = [x for x in W.SHAPES if x.vbr]
    glob = [x for x in vbr if not W.encode_launch(x.plan(), [x.frames]).vbr_scratch_shared]
    assert sum(W.vbr_scratch_bytes(x.plan()) > 40 * 1024 for x in glob) >= 3
    assert any(W.next_pow2(x.N // x.F * x.channels) == 65536 for x in vbr)
    # the items of a 65535-item chunk fit the u16 indices of encoder_vbr.rs:102 exactly
    assert any(x.N // x.F * x.channels == 65535 for x in vbr)


@pytest.mark.parametrize("shape", W.SHAPES, ids=IDS)
def test_oracle_round_trip_and_chunk_sizes(shape):
    """The oracle encodes each shape and decodes it back to the same length; the header, every full chunk and the ragged last
    chunk have the sizes the plan restatement says."""
    p = shape.plan()
    x = pcm(shape)
    blob, _ = O.sea_encode(x, 44100, shape.channels, shape.settings(), return_ties=True)
    if shape.decodable:
        assert O.sea_decode(blob).samples.size == x.size
    else:
        with pytest.raises(O.OracleError):
            O.sea_decode(blob)
    assert blob[5] == shape.channels
    assert int.from_bytes(blob[6:8], "little") == p.full_chunk_bytes
    assert int.from_bytes(blob[8:10], "little") == shape.N
    assert int.from_bytes(blob[14:18], "little") == shape.frames
    full, last = divmod(shape.frames, shape.N)
    last_bytes = len(blob) - 22 - full * p.full_chunk_bytes
    assert 0 < last_bytes <= W.chunk_buf_bytes(p, [shape.frames])
    if not p.vbr:
        items = -(-last // shape.F) * shape.channels
        assert last_bytes == 4 + 16 * shape.channels + -(-items * shape.s // 8) + -(-last * shape.channels * p.hdr_bits // 8)
    for k in range(full + 1):
        pos = 22 + k * p.full_chunk_bytes
        assert blob[pos] == (2 if p.vbr else 1) and blob[pos + 1] == (shape.s << 4) | p.hdr_bits
        assert blob[pos + 2] == shape.F and blob[pos + 3] == 0x5A


@pytest.mark.parametrize("row", OVER_200K, ids=[f"c{r[0]}_F{r[2]}_{'vbr' if r[4] else 'cbr'}{r[3]}_N{r[5]}" for r in OVER_200K])
def test_settings_over_200k_before_now_fit(row):
    C, s, F, bits, vbr, N, before = row
    p = W.plan(C, s, F, bits, vbr, N)
    assert p is not None and N == W.largest_n(C, s, F, bits, vbr) or N == 255
    for frames in (N, N + F // 2 + 1, 3 * N + 1):
        old = W.encode_launch(p, [frames], fixed=False)
        assert old.smem == before and not old.fits
        new = W.encode_launch(p, [frames])
        assert new.fits and new.smem <= W.SMEM_CAP
        assert new.chunk_bytes >= W.chunk_buf_bytes(p, [frames]) >= p.full_chunk_bytes


def test_shapes_that_fitted_keep_their_launch():
    """The fitted sizing changes nothing for a setting that fitted before: same warps, shared memory and chunk buffer."""
    kept = 0
    for x in W.SHAPES:
        p = x.plan()
        for n in (1, 300, 1024):
            old, new = W.encode_launch(p, [x.frames] * n, n, fixed=False), W.encode_launch(p, [x.frames] * n, n)
            if old.fits:
                assert old == new, x.id
                kept += 1
    assert kept >= 3 * 20


def test_every_accepted_setting_fits_the_encoder():
    """A sweep over channels, scale_factor_bits, F, residual sizes and VBR rates at the largest N each accepts, whole chunks and a
    ragged last chunk: the fitted sizing keeps every CTA within 200 KB (the sizing before refused some of each kind)."""
    refused_before = {"cbr": 0, "vbr": 0}
    for C in (1, 2, 8, 9, 16, 33, 100, 160, 200, 255):
        for s in (1, 2, 4, 6, 8):
            for F in (1, 20, 64, 255):
                for bits, vbr in [(1.0, False), (4.0, False), (8.0, False), (1.5, True), (4.5, True), (7.3, True)]:
                    try:
                        N = W.largest_n(C, s, F, bits, vbr)
                    except AssertionError:
                        continue
                    p = W.plan(C, s, F, bits, vbr, N)
                    for frames in (N, N + F // 2 + 1):
                        if not W.encode_launch(p, [frames], fixed=False).fits:
                            refused_before["vbr" if vbr else "cbr"] += 1
                        assert W.encode_launch(p, [frames]).fits, (C, s, F, bits, vbr, N, frames)
    assert refused_before["cbr"] > 0 and refused_before["vbr"] > 0, refused_before
