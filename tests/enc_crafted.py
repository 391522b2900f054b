"""Crafted PCM for the encoder path tests: each input is a seeded recipe of 20-frame blocks drawn from a small menu of loud
shapes, materialised by pcm().  The runaway recipe was found with search() against the CPU mirror (tests/enc_mirror.py); the
others were shaped by hand and checked against the mirror's trace.  tests/test_enc_mirror.py asserts that each still reaches
its target and tests/test_gpu_encode_paths.py runs them on the GPU.
"""
from __future__ import annotations

import numpy as np

BLOCK = 20
HI, LO = 32767, -32768


def _tones(t):
    return np.sin(2 * np.pi * t / 5.29) + np.sin(2 * np.pi * t / 10.38 + 1) + np.sin(2 * np.pi * t / 17.87 + 2)


_TONES_GAIN = HI / np.abs(_tones(np.arange(5120))).max()  # peak 32767 over the first 5120 frames


def _menu_block(name: str, rng: np.random.Generator, t0: int) -> np.ndarray:
    """One channel's 20 frames."""
    t = np.arange(t0, t0 + BLOCK)
    if name.startswith("sq"):                       # full-scale square of period int(name[2:])
        p = int(name[2:])
        return np.where((t // (p // 2)) % 2 == 0, HI, LO)
    if name == "noise":
        return rng.integers(LO, HI + 1, BLOCK)
    if name == "hi":
        return np.full(BLOCK, HI)
    if name == "lo":
        return np.full(BLOCK, LO)
    if name == "zero":
        return np.zeros(BLOCK, np.int64)
    if name == "ramp":
        return np.linspace(LO, HI, BLOCK).astype(np.int64)
    if name == "dramp":
        return np.linspace(HI, LO, BLOCK).astype(np.int64)
    if name == "tones":                             # three full-scale tones: drive the weights past 2^14 (prior32 fails at CBR 3)
        return np.round(_tones(t) * _TONES_GAIN).astype(np.int64)
    if name == "tone":                              # a quiet tone: ordinary audio between the loud blocks
        return (2000 * np.sin(2 * np.pi * t / 37.0)).astype(np.int64)
    raise KeyError(name)


MENU = ("sq2", "sq4", "sq6", "sq10", "sq40", "noise", "hi", "lo", "zero", "ramp", "dramp", "tone", "tones")


def pcm(recipe, channels: int, seed: int = 0) -> np.ndarray:
    """Interleaved int16 PCM.  recipe: one entry per block; an entry is a menu name (every channel), a tuple of names (one per
    channel; "inv" = the phase-inverted copy of channel 0), and a final partial block may be given as (frames, entry)."""
    rng = np.random.default_rng(seed)
    rows = []
    for i, ent in enumerate(recipe):
        nf = BLOCK
        if isinstance(ent, list):
            nf, ent = ent
        names = (ent,) * channels if isinstance(ent, str) else tuple(ent)
        assert len(names) == channels, (ent, channels)
        blk = np.zeros((BLOCK, channels), np.int64)
        for c, nm in enumerate(names):
            blk[:, c] = np.clip(-blk[:, 0], LO, HI) if nm == "inv" else _menu_block(nm, rng, i * BLOCK)
        rows.append(blk[:nf])
    return np.concatenate(rows).astype(np.int16).reshape(-1)


def search(score, channels: int, n_blocks: int, settings, seed: int = 7, menu=MENU, per_channel=False, beam: int = 1, start=()):
    """Greedy (beam = 1) or beam search over CBR blocks of one chunk: block by block, extend each kept recipe by every menu entry
    and keep the `beam` best by score(traces) -> number, where traces is the list of per-block lists of per-channel
    enc_mirror trace dicts so far.  per_channel: also try entries that differ between channel 0 and the others.  Returns the
    best recipe (after `start`)."""
    import enc_mirror as M

    s = settings.scale_factor_bits
    bits = int(np.floor(np.float32(settings.residual_bits)))
    assert not settings.vbr and settings.scale_factor_frames == BLOCK and settings.frames_per_chunk >= BLOCK * (len(start) + n_blocks)
    choices = list(menu)
    if per_channel and channels >= 2:
        choices += [tuple([a] + [b] * (channels - 1)) for a in menu for b in menu if a != b]
    w = np.tile(np.array([0, 0, -(1 << 13), 1 << 14], np.int64), (channels, 1))
    st0 = (list(start), w, np.zeros((channels, 4), np.int64), np.zeros(channels, np.int64), [])
    x = pcm(list(start), channels, seed).reshape(-1, channels).astype(np.int64) if start else None
    if start:
        recipe, w, h, prev, tr = st0
        for b in range(len(start)):
            prev_, w, h, _, _, t = M._block(x[b * BLOCK:(b + 1) * BLOCK], channels, np.full(channels, bits), s, w, h, prev, True)
            tr = tr + [t]
            prev = prev_
        st0 = (recipe, w, h, prev, tr)
    kept = [st0]
    for _ in range(n_blocks):
        cand = []
        for recipe, w, h, prev, tr in kept:
            for ch in choices:
                blk = pcm(recipe + [ch], channels, seed).reshape(-1, channels)[-BLOCK:].astype(np.int64)
                win, w2, h2, _, _, t = M._block(blk, channels, np.full(channels, bits), s, w, h, prev, True)
                cand.append((score(tr + [t]), (recipe + [ch], w2, h2, win, tr + [t])))
        cand.sort(key=lambda c: -c[0])
        kept = [c[1] for c in cand[:beam]]
    return kept[0][0][len(start):]


def _one(name: str, rest: str, channels: int):
    """name on channel 0, rest on the others."""
    return name if channels == 1 else (name,) + (rest,) * (channels - 1)


# name -> recipe(channels).  The targets (asserted in tests/test_enc_mirror.py, for CBR 4 and 8 at scale_factor_bits 4 unless a
# test says otherwise):
#   mid_fail   the 32-bit proof fails in block 6 of a chunk (not the first block), the block is rolled back
#   refail     ... and fails again in block 15, the first block tried after the 8-block skip window
#   one_chain  the proof fails in channel 0 only: in a warp of several chains one fails and the others pass
#   saturated  every candidate of every block ranks at or above 2^27 - 1 (the exact 64-bit arg-min)
#   ties       exact ties of the minimum rank with a previous scale factor other than 0 (the rotated visiting order decides)
#   runaway    found by beam search for the largest weights the search can be pushed to
#   tones      three full-scale tones for 256 blocks: the weights grow to ~24,000 and prior32 fails at CBR 3 (the 64-bit form of
#              the direct quantiser); at CBR 1 and 2 it stays below the bound
#   phase      a phase-inverted copy of channel 0 on channel 1, a ramp, silence and a held extreme
RECIPES = {
    "mid_fail": lambda C: ["tone"] * 6 + ["noise"] + ["tone"] * 13,
    "refail": lambda C: ["tone"] * 6 + ["noise"] + ["tone"] * 8 + ["sq2"] + ["tone"] * 4,
    "one_chain": lambda C: [_one("tone", "tone", C)] * 3 + [_one("noise", "tone", C)] + [_one("tone", "tone", C)] * 10
    + [_one("sq2", "zero", C)] + [_one("tone", "zero", C)] * 5,
    "saturated": lambda C: ["sq10"] * 20,
    "ties": lambda C: ["hi"] * 10 + ["sq2"] * 10,
    "runaway": lambda C: ["lo", "sq6", "sq40", "sq4", "sq6", "hi", "sq2", "sq40", "sq40", "hi", "sq40", "sq6"] + ["lo", "sq40"] * 14,
    "tones": lambda C: ["tones"] * 256,
    "phase": lambda C: [_one(n, "inv", C) for n in ("sq40", "ramp", "noise", "dramp", "sq6")] + ["zero"] * 3 + ["lo"] * 4
    + [_one("ramp", "inv", C)] * 4 + ["hi"] * 4,
}


def crafted(name: str, channels: int, seed: int = 7) -> np.ndarray:
    return pcm(RECIPES[name](channels), channels, seed)
