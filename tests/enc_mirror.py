"""CPU mirror of the encoder's scale-factor search (oracle/sea_oracle.c, encoder_base.rs) with a per-block trace of what the
fast GPU pass (search_pass_fast in sea_codec_b200/csrc/encode_kernels.cu) decides on the same input.

The 2^s candidates of a block are evaluated together in numpy, each in full (as the GPU does), with the partial rank of every
frame kept in wrapping uint64.  The reference's sequential loop with its early exit is then replayed on those partial ranks, so
encode() reproduces oracle.sea_encode byte for byte, and the trace records whether the GPU's rule -- the smallest full rank,
ties to the earliest visited candidate -- picks the same winner.

The trace groups chains the way a warp does (chains per warp = 32 / 2^s, or one with SEA_B200_ENC_SPLIT=1; a warp's missing
chains duplicate the last channel) and replays the warp-wide votes: prior32 (CBR sizes 1-3), try32 with its proof and the
spec_skip window, weights_stay_narrow, the three arg-min forms, and for VBR the register sort's limits.
"""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np

from oracle import sea_oracle as O

KSAT = (1 << 27) - 1          # encode_kernels.cu: ranks are clamped to this for the single redux
SORT_KEY_LIMIT = 1 << 55      # warp_sort_512 packs (rank, idx) into 64 bits while every rank is below this
WRAP = 1 << 64
_U = np.uint64


def _wrap32(v):
    return ((v + (1 << 31)) & 0xFFFFFFFF) - (1 << 31)


_TABS = {}


def tables(b: int, s: int):
    """(recip[2^s], dqt[2^s][256] zero padded, quant_tab[513] zero padded) of residual size b as int64."""
    key = (b, s)
    if key not in _TABS:
        recip, dqt = O.tables(b, s)
        pad = np.zeros((1 << s, 256), np.int64)
        pad[:, : 1 << b] = dqt
        qt = np.zeros(513, np.int64)
        q = O.quant_tab(b)
        qt[: q.size] = q
        _TABS[key] = (recip.astype(np.int64), pad, qt)
    return _TABS[key]


def next_pow2(v: int) -> int:
    p = 2
    while p < v:
        p <<= 1
    return p


@dataclass
class BlockTrace:
    """One (chunk, pass, block, channel): what every candidate did and which one the reference and the GPU rule keep."""
    chunk: int
    pass_: int            # 0 CBR encode, 1 VBR analysis, 2 VBR encode
    blk: int
    ch: int
    nf: int
    size: int
    prev: int             # previous scale factor (the rotation of the visiting order)
    winner: int           # the reference's scale factor (with early exit)
    gpu_winner: int       # smallest (full wrapping rank, ord)
    min_rank: int         # full ranks of the candidates (wrapping u64)
    max_rank: int
    exact_max_rank: float  # the largest rank without wrap-around
    wrapped: bool          # some candidate's rank passed 2^64
    ties: int              # candidates at the minimum rank
    tied: tuple            # ... their scale factors
    m0: int                # max |w| at the start of the block
    w0: tuple              # the weights at the start of the block
    max_w: int             # largest |w| of any candidate during the block
    prior32_ok: bool       # the bound of the direct quantiser holds for every candidate (meaningful for CBR sizes 1-3)
    proof_ok: bool         # m0 + (sum|d| >> 4) + 20 <= 32767 for every candidate
    narrow_ok: bool        # weights_stay_narrow at F = 20
    big: bool              # some rank >> (64 - s) != 0


@dataclass
class Result:
    data: bytes
    ties: int
    blocks: list = field(default_factory=list)      # BlockTrace
    sorts: list = field(default_factory=list)       # (chunk, items, np2, max_key)

    def chain(self, ch=None, pass_=None):
        return [b for b in self.blocks if (ch is None or b.ch == ch) and (pass_ is None or b.pass_ == pass_)]


def _block(x, C, sizes, s, w0, h0, prev, keep_all):
    """Every candidate of every channel over one block.  x: [nf][C] int64; sizes[C]; w0, h0: [C][4]; prev[C].
    Returns (winner sf, new w, new h, reference rank, list of per-channel trace tuples)."""
    nsf, nf = 1 << s, x.shape[0]
    recip = np.empty((C, nsf), np.int64)
    dqt = np.empty((C, nsf, 256), np.int64)
    qt = np.empty((C, 513), np.int64)
    for c in range(C):
        recip[c], dqt[c], qt[c] = tables(int(sizes[c]), s)
    lim = (1 << np.asarray(sizes, np.int64))[:, None]
    w = np.repeat(w0[:, None, :], nsf, 1).astype(np.int64)    # [C][nsf][4]
    h = np.repeat(h0[:, None, :], nsf, 1).astype(np.int64)
    rank = np.zeros((C, nsf), _U)
    exact = np.zeros((C, nsf), np.float64)
    part = np.zeros((C, nsf, nf), _U)
    dsum = np.zeros((C, nsf), np.int64)
    maxw = np.abs(w0).max(1).astype(np.int64)
    rows = np.arange(C)[:, None]
    cols = np.arange(nsf)[None, :]
    codes = np.zeros((C, nsf, nf), np.int64)
    for f in range(nf):
        xs = x[f][:, None]
        pred = _wrap32((w * h).sum(2)) >> 13
        r = _wrap32(xs - pred)
        n = (r * recip + 32768) >> 16
        scaled = n + (np.sign(r) - np.sign(n))
        scaled = np.clip(scaled, -lim, lim)
        q = qt[rows, scaled + lim]
        d = dqt[rows, cols, q]
        y = np.clip(_wrap32(pred + d), -32768, 32767)
        e = xs - y
        sq = (w.astype(_U) * w.astype(_U)).sum(2, dtype=_U)     # wrapping u64, as the reference's i64 sum in release
        p = (sq.view(np.int64) >> 18) - 0x8FF
        p = np.maximum(p, 0)
        rank += (e * e).astype(_U) + p.astype(_U) * p.astype(_U)
        exact += (e * e).astype(np.float64) + p.astype(np.float64) ** 2
        part[:, :, f] = rank
        dsum += np.abs(d)
        codes[:, :, f] = q
        delta = d >> 4
        w = _wrap32(w + np.where(h < 0, -1, 1) * delta[:, :, None])
        h = np.concatenate([h[:, :, 1:], y[:, :, None]], 2)
        maxw = np.maximum(maxw, np.abs(w).max((1, 2)))
    out = []
    win = np.zeros(C, np.int64)
    wn = np.zeros((C, 4), np.int64)
    hn = np.zeros((C, 4), np.int64)
    ref_rank = np.zeros(C, object)
    win_codes = np.zeros((C, nf), np.int64)
    for c in range(C):
        pv = int(prev[c])
        best, bsf = WRAP - 1, 0
        for i in range(nsf):
            sf = (i + pv) % nsf
            pr = part[c, sf]
            over = np.nonzero(pr > _U(best))[0]
            if over.size:
                continue  # early exit: this rank is above the best so far and never wins
            full = int(pr[-1])
            if full < best:
                best, bsf = full, sf
        full_r = rank[c].astype(object)
        ords = [(sf - pv) % nsf for sf in range(nsf)]
        gsf = min(range(nsf), key=lambda sf: (int(full_r[sf]), ords[sf]))
        win[c], wn[c], hn[c], ref_rank[c] = bsf, w[c, bsf], h[c, bsf], best
        win_codes[c] = codes[c, bsf]
        if keep_all:
            m0 = int(np.abs(w0[c]).max())
            mn = int(min(full_r))
            out.append(dict(
                prev=pv, winner=bsf, gpu_winner=gsf, min_rank=mn, max_rank=int(max(full_r)),
                exact_max_rank=float(exact[c].max()), wrapped=bool(exact[c].max() >= WRAP),
                ties=sum(1 for v in full_r if int(v) == mn), tied=tuple(sf for sf in range(nsf) if int(full_r[sf]) == mn), m0=m0, w0=tuple(int(v) for v in w0[c]), max_w=int(maxw[c]),
                prior32_ok=_prior32(m0, w0[c], int(sizes[c]), s),
                proof_ok=bool(np.all(m0 + (dsum[c] >> 4) + 20 <= 32767)),
                narrow_ok=m0 < (1 << 23) - 1 - 20 * 1600,
                big=any(int(v) >> (64 - s) for v in full_r)))
    return win, wn, hn, ref_rank, win_codes, out


def _prior32(m0, w, size, s):
    """The bound the direct-quantiser instances (CBR sizes 1-3) take before the trial, for every scale factor of the chain."""
    if size > 3:
        return False
    levels = {1: 0, 2: 1, 3: 3}[size]
    _, dqt, _ = tables(size, s)
    for sf in range(1 << s):
        grow = 20 * ((int(dqt[sf, 2 * levels]) + 15) >> 4)
        a = [abs(int(v)) + grow for v in w]
        if not all(v < 65536 for v in a) or sum(v * v for v in a) >> 32:
            return False
    return True


def _pack(vals, widths):
    """Big-endian bit string of the fields, padded to a byte (bits.rs BitPacker)."""
    vals = np.asarray(vals, np.int64)
    widths = np.broadcast_to(np.asarray(widths, np.int64), vals.shape)
    if vals.size == 0:
        return b""
    k = np.arange(8)
    bits = (vals[:, None] >> (widths[:, None] - 1 - k[None, :])) & 1
    bits = bits[k[None, :] < widths[:, None]]
    return np.packbits(bits.astype(np.uint8)).tobytes()


def encode(pcm, channels: int, settings, sample_rate: int = 44100, trace: bool = True) -> Result:
    """oracle.sea_encode restated.  settings: oracle.make_settings(...)."""
    C = channels
    x = np.ascontiguousarray(pcm, np.int16).reshape(-1, C).astype(np.int64)
    frames = x.shape[0]
    s, F, N, vbr = settings.scale_factor_bits, settings.scale_factor_frames, settings.frames_per_chunk, bool(settings.vbr)
    hdr_bits = int(np.floor(np.float32(settings.residual_bits)))
    nsf = 1 << s
    w = np.tile(np.array([0, 0, -(1 << 13), 1 << 14], np.int64), (C, 1))
    h = np.zeros((C, 4), np.int64)
    prev = np.zeros(C, np.int64)
    res = Result(b"", 0)
    chunks = []
    for k in range((frames + N - 1) // N):
        xc = x[k * N: (k + 1) * N]
        nfr = xc.shape[0]
        nblk = (nfr + F - 1) // F
        lms_bytes = b"".join((np.concatenate([h[c], w[c]]) & 0xFFFF).astype("<u2").tobytes() for c in range(C))

        def run(pass_, sizes_of):
            nonlocal w, h, prev
            sfs = np.zeros((nblk, C), np.int64)
            codes = []
            ranks = np.zeros((nblk, C), object)
            for b in range(nblk):
                sizes = sizes_of(b)
                win, w, h, rr, wc, tr = _block(xc[b * F: (b + 1) * F], C, sizes, s, w, h, prev, trace)
                for c, t in enumerate(tr):
                    res.blocks.append(BlockTrace(chunk=k, pass_=pass_, blk=b, ch=c, nf=wc.shape[1], size=int(sizes[c]), **t))
                prev = win.copy()
                sfs[b] = win
                ranks[b] = rr
                codes.append(wc)
            return sfs, codes, ranks

        if not vbr:
            sfs, codes, _ = run(0, lambda b: np.full(C, hdr_bits))
            sizes = np.full((nblk, C), hdr_bits)
        else:
            target, base, counts = O.vbr_params(settings, (nfr * C) // F)
            w_save, h_save = w.copy(), h.copy()
            _, _, ranks = run(1, lambda b: np.full(C, base + 1))
            w, h = w_save, h_save  # restores lms only (the previous scale factors carry over: trap T2)
            sortable = (nfr * C) // F
            keys = [int(v) for v in ranks.reshape(-1)[:sortable]]
            order = sorted(range(sortable), key=lambda i: (keys[i], i))
            res.sorts.append((k, sortable, next_pow2(sortable), max(keys) if keys else 0))
            flat = np.full(nblk * C, base, np.int64)
            m1, p1, p2 = counts[0], counts[2], counts[3]
            lab = np.full(sortable, base, np.int64)
            lab[:m1] = base - 1
            lab[sortable - p2 - p1:] = base + 1
            lab[sortable - p2:] = base + 2
            for pos in range(sortable):
                flat[order[pos]] = lab[pos]
            for bnd in (m1, sortable - p2 - p1, sortable - p2):
                if 0 < bnd < sortable and keys[order[bnd - 1]] == keys[order[bnd]] and lab[bnd - 1] != lab[bnd]:
                    res.ties += 1
            sizes = flat.reshape(nblk, C)
            sfs, codes, _ = run(2, lambda b: sizes[b])
        body = bytes([2 if vbr else 1, (s << 4) | hdr_bits, F, 0x5A]) + lms_bytes
        body += _pack(sfs.reshape(-1), s)
        if vbr:
            body += _pack((sizes.reshape(-1) - hdr_bits + 1) & 3, 2)
        rv, rw = [], []
        for b in range(nblk):
            cb = codes[b]                           # [C][nf]
            rv.append(cb.T.reshape(-1))
            rw.append(np.tile(sizes[b], cb.shape[1]))
        body += _pack(np.concatenate(rv), np.concatenate(rw))
        chunks.append(body)
    head = b"seac" + bytes([1, C]) + int(len(chunks[0]) if chunks else 0).to_bytes(2, "little") + int(N).to_bytes(2, "little")
    head += int(sample_rate).to_bytes(4, "little") + int(frames).to_bytes(4, "little") + bytes(4)
    res.data = head + b"".join(chunks)
    return res


# ------------------------------------------------------------------------------------------------ warp-level votes

@dataclass
class WarpBlock:
    """One (chunk, pass, warp round, block) of search_pass_fast."""
    chunk: int
    pass_: int
    chains: tuple
    blk: int
    nf: int
    form: str        # 'prior32' | 'sum32' | 'narrow' | 'wide' (the form whose rank is kept)
    tried32: bool    # the speculative 32-bit trial ran
    rollback: bool   # ... and its proof failed: the block was run again
    spec_skip: int   # the counter when the block started
    argmin: str      # 'redux' | 'butterfly' | 'explicit'
    split_chain_fail: bool  # the proof failed in some chains of the warp but not all


def warp_rounds(C: int, s: int, split: bool):
    """The chain groups of search_pass_fast: each entry is the tuple of channels one warp runs together."""
    cpw = 1 if split else 32 // (1 << s)
    warps = min(8, C if split else (C + cpw - 1) // cpw)
    slots = warps * cpw
    out = []
    for wp in range(warps):
        cb = wp * cpw
        while cb < C:
            out.append(tuple(min(cb + q, C - 1) for q in range(cpw)))
            cb += slots
    return out


def warp_trace(r: Result, C: int, settings, split: bool = False):
    s, vbr = settings.scale_factor_bits, bool(settings.vbr)
    hdr = int(np.floor(np.float32(settings.residual_bits)))
    direct = not vbr and 1 <= hdr <= 3
    by = {}
    for b in r.blocks:
        by.setdefault((b.chunk, b.pass_), {})[(b.blk, b.ch)] = b
    out = []
    for (k, ps), blocks in sorted(by.items()):
        nblk = 1 + max(bl for bl, _ in blocks)
        for chains in warp_rounds(C, s, split):
            spec = 0
            for bl in range(nblk):
                bt = [blocks[(bl, c)] for c in chains]
                nf = bt[0].nf
                prior = direct and nf == 20 and all(t.prior32_ok for t in bt)
                try32 = not direct and nf == 20 and spec == 0
                start = spec
                if spec:
                    spec -= 1
                proof = all(t.proof_ok for t in bt)
                rollback = try32 and not proof
                if prior:
                    form = "prior32"
                elif try32 and proof:
                    form = "sum32"
                else:
                    form = "narrow" if all(t.narrow_ok for t in bt) else "wide"
                if rollback:
                    spec = 8
                if not any(t.min_rank >= KSAT for t in bt):
                    am = "redux"
                elif not any(t.big for t in bt):
                    am = "butterfly"
                else:
                    am = "explicit"
                real = set(chains)
                fails = {c for c in real if not blocks[(bl, c)].proof_ok}
                out.append(WarpBlock(k, ps, chains, bl, nf, form, try32, rollback, start, am,
                                     bool(try32 and fails and fails != real)))
    return out


# ------------------------------------------------------------------------------------------------ host rule of the LUT layout

ENC_LUT32, ENC_LUT16, ENC_LUT_GLOBAL = 0, 1, 2


def enc_lut_mode(n_streams: int, settings, channels: int, split: bool = False, pin: str | None = None) -> int:
    """The dequant-table layout launch_encode_generic picks for a VBR batch of the fast pass (kEncLut32 / 16 / Global)."""
    s, F, N = settings.scale_factor_bits, settings.scale_factor_frames, settings.frames_per_chunk
    assert settings.vbr and 3 <= s <= 5 and F == 20 and channels <= 16
    nsf = 1 << s
    cpw = 32 // nsf
    target, base, counts = O.vbr_params(settings, (N // F) * channels)
    items = (N // F) * channels
    hdr = int(np.floor(np.float32(settings.residual_bits)))
    full = 4 + 16 * channels + (items * s + 7) // 8 + (items * 2 + 7) // 8 + (sum(counts[i] * (base + i - 1) for i in range(4)) * F + 7) // 8
    worst = 4 + 16 * channels + (items * s + 7) // 8 + (items * 2 + 7) // 8 + (N * channels * (base + 2) + 7) // 8
    max_chunk = max(full, worst)
    del hdr
    split = split and channels >= 2
    warps = min(8, channels if split else (channels + cpw - 1) // cpw)
    T = warps * 32
    smem = ((max_chunk + 3) // 4 + 2) * 4 + channels * 17 * 4 + ((2 * F * T + 15) & ~15) + 16
    smem += (warps * cpw * F * 2 + 15) & ~15
    lo = base - 1 if base > 1 else 1
    e = sum(1 << (lo + i) for i in range(4) if lo + i <= 8)
    nblk = N // F
    np2 = next_pow2(nblk * channels)
    scratch = (np2 * 8 + np2 * 4 + nblk * 8 + nblk * channels * 5 + 255) & ~255
    other = smem + 256 + scratch + 16
    per_sm = (n_streams + 147) // 148
    budget = 227 * 1024 // per_sm
    budget = budget - 1280 if budget > 1280 + 28 * 1024 else 28 * 1024
    if pin is not None:
        want = {"32": ENC_LUT32, "16": ENC_LUT16, "global": ENC_LUT_GLOBAL}[pin]
        if want == ENC_LUT_GLOBAL:
            return want
        if (want == ENC_LUT32 or s == 4) and other + e * (128 if want == ENC_LUT32 else 64) <= 200 * 1024:
            return want
    if other + e * 128 <= budget:
        return ENC_LUT32
    if s == 4 and other + e * 64 <= budget:
        return ENC_LUT16
    return ENC_LUT_GLOBAL
