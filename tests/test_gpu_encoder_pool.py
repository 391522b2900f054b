"""The session pool (Context.encoder_pool, sea_b200_encoder_pool_*): many live streams pushed as ragged packets, every completed
chunk of every session encoded in one launch per push.  Each session's header plus its joined push outputs must be byte for byte
oracle.sea_encode of its whole PCM, whatever the packet sizes, which sessions share a push, and when slots end and reopen.  Also:
refused pushes change nothing, the VBR tie counts come back per session in call order, a push is at most three launches, and the
device form writes nothing outside each session's output."""
import os
import subprocess
import sys

import numpy as np
import pytest

import enc_crafted as G
import sea_codec_b200 as S
from sea_codec_b200 import api
from sea_codec_b200 import synth

pytestmark = pytest.mark.gpu

RATE = 44100
CRAFTED = list(G.RECIPES)


def _pair(oracle, **kw):
    return S.EncoderSettings(**kw), oracle.make_settings(**kw)


def _stream_pcm(rng, channels, N, crafted):
    """One life's PCM: synthetic audio, or crafted blocks (the speculative search paths) joined to about 1-4 chunks."""
    if crafted:
        parts, frames = [], 0
        while frames < N * rng.integers(1, 4):
            x = G.crafted(CRAFTED[rng.integers(len(CRAFTED))], channels, seed=int(rng.integers(1 << 30)))
            parts.append(x.reshape(-1))
            frames += x.size // channels
        return np.concatenate(parts)
    frames = int(rng.integers(0, 4 * N + 50))
    return synth.gen_stream(int(rng.integers(1 << 20)), frames, channels, RATE).reshape(-1)


class Traffic:
    """Seeded live-server traffic over a pool: sessions open, push random packet sizes in random subsets, end and reopen.  Every
    finished life is (pcm, header + joined outputs, summed tie counts)."""

    def __init__(self, ctx, pool, channels, N, n_sessions, seed, crafted_share=0.0):
        self.ctx, self.pool, self.C, self.N = ctx, pool, channels, N
        self.rng = np.random.default_rng(seed)
        self.n = n_sessions
        self.crafted_share = crafted_share
        self.life = {}  # slot -> dict(pcm, pos, out, ties) of the stream it carries
        self.done = []

    def _packet_frames(self, left):
        N = self.N
        menu = [0, 1, N - 1, N, N + 1, 3 * N + 7, int(self.rng.integers(0, 2 * N))]
        return min(left, menu[self.rng.integers(len(menu))])

    def open_some(self, k):
        free = [s for s in range(self.n) if s not in self.life]
        pick = sorted(self.rng.choice(free, size=min(k, len(free)), replace=False).tolist()) if free else []
        if pick:
            self.pool.open(pick)
        for s in pick:
            crafted = self.rng.random() < self.crafted_share
            self.life[s] = dict(pcm=_stream_pcm(self.rng, self.C, self.N, crafted), pos=0, out=[], ties=0)

    def round(self, end_share=0.3):
        open_ = list(self.life)
        if not open_:
            return
        k = int(self.rng.integers(1, len(open_) + 1))
        order = self.rng.permutation(open_)[:k].tolist()
        packets, ends = [], []
        for s in order:
            L = self.life[s]
            left = L["pcm"].size // self.C - L["pos"]
            f = self._packet_frames(left)
            packets.append(L["pcm"][L["pos"] * self.C:(L["pos"] + f) * self.C])
            L["pos"] += f
            ends.append(L["pos"] * self.C == L["pcm"].size and self.rng.random() < end_share)
        outs = self.pool.push(order, packets, end=ends)
        ties = self.ctx.last_vbr_ties_per_stream(len(order))
        for s, o, e, t in zip(order, outs, ends, ties):
            L = self.life[s]
            L["out"].append(o)
            L["ties"] += int(t)
            if e:
                self.done.append((L["pcm"], b"".join(L["out"]), L["ties"]))
                del self.life[s]

    def finish(self):
        """Ends every open life (some with a last packet of 0 frames, some with the rest of their PCM)."""
        while self.life:
            order = list(self.life)
            packets = []
            for s in order:
                L = self.life[s]
                packets.append(L["pcm"][L["pos"] * self.C:])
                L["pos"] = L["pcm"].size // self.C
            outs = self.pool.push(order, packets, end=True)
            ties = self.ctx.last_vbr_ties_per_stream(len(order))
            for s, o, t in zip(order, outs, ties):
                L = self.life.pop(s)
                L["out"].append(o)
                L["ties"] += int(t)
                self.done.append((L["pcm"], b"".join(L["out"]), L["ties"]))


def _file(pool, pcm, chunks, channels, N):
    frames = pcm.size // channels
    first = 0
    if chunks:
        first = pool._full if frames >= N else len(chunks)
    return pool.header(0, first, frames) + chunks


def _run_traffic(ctx, oracle, channels, kw, n_sessions=64, rounds=24, seed=1, crafted_share=0.25, check_ctx=True):
    st, ost = _pair(oracle, **kw)
    N = st.frames_per_chunk
    pool = ctx.encoder_pool(channels, RATE, st, n_sessions)
    try:
        T = Traffic(ctx, pool, channels, N, n_sessions, seed, crafted_share)
        T.open_some(n_sessions * 3 // 4)
        for r in range(rounds):
            T.round()
            if r % 4 == 3:
                T.open_some(n_sessions // 8)  # reopens slots that ended
        T.finish()
        assert len(T.done) >= n_sessions * 3 // 4
        for pcm, chunks, ties in T.done:
            ref, ref_ties = oracle.sea_encode(pcm, RATE, channels, ost, return_ties=True)
            got = _file(pool, pcm, chunks, channels, N)
            assert got == ref, (kw, channels, pcm.size // channels)
            if kw.get("vbr"):
                assert ties == ref_ties, (kw, channels, pcm.size // channels)
        if check_ctx:  # the one-shot encoder agrees on a few of them
            for pcm, chunks, _ in T.done[:4]:
                assert ctx.sea_encode(pcm, RATE, channels, st) == _file(pool, pcm, chunks, channels, N)
    finally:
        pool.close()


@pytest.mark.parametrize("bits", range(1, 9))
def test_random_traffic_cbr_bits(ctx, oracle, bits):
    _run_traffic(ctx, oracle, 2, dict(residual_bits=float(bits)), seed=bits)


@pytest.mark.parametrize("bits", [1.5, 3.0, 4.5])
def test_random_traffic_vbr(ctx, oracle, bits):
    _run_traffic(ctx, oracle, 2, dict(residual_bits=bits, vbr=True), seed=int(bits * 10))


@pytest.mark.parametrize("channels", [1, 3, 8])
def test_random_traffic_channels(ctx, oracle, channels):
    _run_traffic(ctx, oracle, channels, dict(residual_bits=3.0), seed=100 + channels)
    _run_traffic(ctx, oracle, channels, dict(residual_bits=3.0, vbr=True), n_sessions=16, rounds=10, seed=200 + channels,
                 check_ctx=False)


def test_random_traffic_255_channels(ctx, oracle):
    _run_traffic(ctx, oracle, 255, dict(residual_bits=3.0, frames_per_chunk=400), n_sessions=4, rounds=8, seed=255, crafted_share=0.0)


@pytest.mark.parametrize("s", [3, 4, 5])
def test_random_traffic_scale_factor_bits(ctx, oracle, s):
    _run_traffic(ctx, oracle, 2, dict(residual_bits=4.0, scale_factor_bits=s), seed=300 + s)
    _run_traffic(ctx, oracle, 2, dict(residual_bits=3.0, vbr=True, scale_factor_bits=s), n_sessions=16, rounds=10, seed=310 + s,
                 check_ctx=False)


@pytest.mark.parametrize("fpc", [400, 960, 5000])
def test_random_traffic_frames_per_chunk(ctx, oracle, fpc):
    _run_traffic(ctx, oracle, 2, dict(residual_bits=3.0, frames_per_chunk=fpc), seed=400 + fpc)
    _run_traffic(ctx, oracle, 2, dict(residual_bits=3.0, vbr=True, frames_per_chunk=fpc), n_sessions=16, rounds=10, seed=410 + fpc,
                 check_ctx=False)


def test_chunk_aligned_packets_equal_make_chunks(ctx, oracle):
    """Packets of whole chunks: each push's output is what make_chunks gives on a per-session handle fed the same packets."""
    st = S.EncoderSettings(residual_bits=3.0, frames_per_chunk=960)
    N, C, n = 960, 2, 6
    pool = ctx.encoder_pool(C, RATE, st, n)
    pool.open(range(n))
    L = ctx._L
    handles = []
    for _ in range(n):
        h = api.C.c_void_p()
        ctx._check(L.sea_b200_encoder_create(ctx._h, C, RATE, api.C.byref(st._c()), api.C.byref(h)))
        handles.append(h)
    try:
        pcms = [synth.gen_stream(500 + i, N * 6, C, RATE).reshape(-1) for i in range(n)]
        pos = [0] * n
        for r in range(4):
            ks = [(i + r) % 3 for i in range(n)]  # 0, 1 or 2 chunks
            packets = [pcms[i][pos[i]:pos[i] + ks[i] * N * C] for i in range(n)]
            outs = pool.push(list(range(n)), packets)
            for i in range(n):
                pos[i] += ks[i] * N * C
                if not ks[i]:
                    assert outs[i] == b""
                    continue
                buf = np.empty(70000 * ks[i], np.uint8)
                ln, nck = api.C.c_uint64(0), api.C.c_uint32(0)
                p = np.ascontiguousarray(packets[i])
                ctx._check(L.sea_b200_encoder_make_chunks(handles[i], p.ctypes.data, p.size, buf.ctypes.data, buf.size, api.C.byref(ln),
                                                          api.C.byref(nck)))
                assert outs[i] == buf[: ln.value].tobytes(), (r, i)
            assert list(pool.buffered(range(n))) == [0] * n
    finally:
        for h in handles:
            L.sea_b200_encoder_destroy(h)
        pool.close()


def test_short_sessions_empty_end_and_reopen(ctx, oracle):
    st, ost = _pair(oracle, residual_bits=3.0, vbr=True)
    C, N = 2, 5120
    pool = ctx.encoder_pool(C, RATE, st, 4)
    try:
        pool.open([0, 1, 2])
        a = synth.gen_stream(7, 3000, C, RATE).reshape(-1)
        outs = pool.push([0, 1], [a[:1000 * C], a[:0]])
        assert outs == [b"", b""]
        assert list(pool.buffered([0, 1, 2, 3])) == [1000, 0, 0, 0]
        outs = pool.push([0, 1, 2], [a[1000 * C:], a[:0], a[:0]], end=[True, True, False])
        ref = oracle.sea_encode(a, RATE, C, ost)
        assert pool.header(0, len(outs[0]), 3000) + outs[0] == ref  # one short chunk
        assert outs[1] == b"" and outs[2] == b""
        # session 0 reopens: fresh state, nothing buffered
        pool.open([0])
        assert list(pool.buffered([0])) == [0]
        b = synth.gen_stream(8, 2 * N + 17, C, RATE).reshape(-1)
        o1 = pool.push([0], [b[:N * C + 5 * C]])[0]
        o2 = pool.push([0], [b[N * C + 5 * C:]], end=True)[0]
        assert pool.header(0, pool._full, 2 * N + 17) + o1 + o2 == oracle.sea_encode(b, RATE, C, ost)
    finally:
        pool.close()


def test_push_device_equals_push_and_keeps_outside_bytes(ctx, oracle):
    import torch

    st, ost = _pair(oracle, residual_bits=3.0, vbr=True, frames_per_chunk=960)
    C, N, n = 2, 960, 12
    rng = np.random.default_rng(5)
    pa, pb = ctx.encoder_pool(C, RATE, st, n), ctx.encoder_pool(C, RATE, st, n)
    try:
        pa.open(range(n))
        pb.open(range(n))
        dev = torch.device("cuda", ctx.device)
        pcms = [synth.gen_stream(900 + i, int(rng.integers(N, 5 * N)), C, RATE).reshape(-1) for i in range(n)]
        pos = [0] * n
        got_a, got_b = [b""] * n, [b""] * n
        for r in range(6):
            last = r == 5
            sizes = [pcms[i].size // C - pos[i] if last else min(pcms[i].size // C - pos[i], int(rng.integers(0, 2 * N))) for i in range(n)]
            packets = [pcms[i][pos[i] * C:(pos[i] + sizes[i]) * C] for i in range(n)]
            for i in range(n):
                pos[i] += sizes[i]
            ends = [last] * n
            oa = pa.push(range(n), packets, end=ends)
            # device form: odd packet offsets (misaligned sources) and sentinel gaps between the output regions
            caps = [pb.push_bound(i, sizes[i], last) for i in range(n)]
            pcm_off, off = [], 3
            for p in packets:
                pcm_off.append(off)
                off += p.size + 5
            d_pcm = torch.zeros(off + 8, dtype=torch.int16, device=dev)
            for p, o in zip(packets, pcm_off):
                if p.size:
                    d_pcm[o:o + p.size] = torch.from_numpy(np.ascontiguousarray(p)).to(dev)
            out_off, o = [], 7
            for c in caps:
                out_off.append(o)
                o += c + 13
            d_out = torch.full((o + 16,), 0xA5, dtype=torch.uint8, device=dev)
            lens = pb.push_device(range(n), d_pcm.data_ptr(), pcm_off, sizes, d_out.data_ptr(), out_off, end=ends, out_caps=caps)
            torch.cuda.synchronize()
            host = d_out.cpu().numpy()
            mask = np.ones(host.size, bool)
            for i in range(n):
                seg = host[out_off[i]:out_off[i] + int(lens[i])].tobytes()
                assert seg == oa[i], (r, i)
                mask[out_off[i]:out_off[i] + int(lens[i])] = False
                got_a[i] += oa[i]
                got_b[i] += seg
            assert np.all(host[mask] == 0xA5), r
        for i in range(n):
            frames = pcms[i].size // C
            first = pa._full if frames >= N else len(got_a[i])
            assert pa.header(i, first, frames) + got_b[i] == oracle.sea_encode(pcms[i], RATE, C, ost)
    finally:
        pa.close()
        pb.close()


def _code(fn):
    with pytest.raises(S.SeaError) as e:
        fn()
    return e.value.code


def test_refused_pushes_change_nothing(ctx, oracle):
    """Every refusal, then the same sessions carry on: their final bytes still equal the oracle's."""
    import torch

    st, ost = _pair(oracle, residual_bits=3.0, frames_per_chunk=960)
    C, N = 2, 960
    pool = ctx.encoder_pool(C, RATE, st, 4)
    try:
        pool.open([0, 1])
        assert _code(lambda: pool.open([1])) == api.ERR_INVALID_PARAMETERS  # already open
        assert _code(lambda: pool.open([4])) == api.ERR_INVALID_PARAMETERS
        assert _code(lambda: pool.open([2, 2])) == api.ERR_INVALID_PARAMETERS
        assert list(pool.buffered([2])) == [0]
        a = synth.gen_stream(31, 3 * N + 100, C, RATE).reshape(-1)
        b = synth.gen_stream(32, 2 * N + 900, C, RATE).reshape(-1)
        o = pool.push([0, 1], [a[:500 * C], b[:700 * C]])
        outs = {0: [o[0]], 1: [o[1]]}
        pa, pb = a[500 * C:1800 * C], b[700 * C:900 * C]  # session 0 completes a chunk, 1 does not
        L = ctx._L
        before = ctx.launch_count

        def refuse(sessions, packets, code, end=None, caps=None):
            frames = [p.size // C for p in packets]
            pcm = np.concatenate(packets)
            offs = np.cumsum([0] + [p.size for p in packets])[:-1]
            out = np.zeros(200000, np.uint8)
            oo = [0, 100000][: len(sessions)]
            assert _code(lambda: pool.push_host(sessions, pcm.ctypes.data, offs, frames, out.ctypes.data, oo, end=end, out_caps=caps)) == code
            assert list(pool.buffered([0, 1])) == [500, 700]

        refuse([0, 2], [pa, pb], api.ERR_INVALID_PARAMETERS)                    # 2 is not open
        refuse([0, 4], [pa, pb], api.ERR_INVALID_PARAMETERS)                    # past max_sessions
        refuse([0, 0], [pa, pa], api.ERR_INVALID_PARAMETERS)                    # twice
        refuse([1, 0], [pb, pa], api.ERR_CAPACITY, caps=[10**6, pool.push_bound(0, 1300) - 1])
        refuse([0, 1], [pa, pb], api.ERR_CAPACITY, end=[False, True], caps=[10**6, pool.push_bound(1, 200, True) - 1])
        # NULL pointers
        s = np.array([0, 1], np.uint32)
        z = np.zeros(2, np.uint64)
        f = np.array([1, 1], np.uint32)
        lens = np.zeros(2, np.uint64)
        buf = np.zeros(64, np.int16)
        for args in ((None, buf.ctypes.data, z.ctypes.data, f.ctypes.data), (s.ctypes.data, None, z.ctypes.data, f.ctypes.data),
                     (s.ctypes.data, buf.ctypes.data, None, f.ctypes.data), (s.ctypes.data, buf.ctypes.data, z.ctypes.data, None)):
            assert L.sea_b200_encoder_pool_push(pool._h, 2, *args, None, buf.ctypes.data, z.ctypes.data, None, lens.ctypes.data, None) \
                == api.ERR_INVALID_PARAMETERS
        assert L.sea_b200_encoder_pool_push(pool._h, 2, s.ctypes.data, buf.ctypes.data, z.ctypes.data, f.ctypes.data, None, buf.ctypes.data,
                                            z.ctypes.data, None, None, None) == api.ERR_INVALID_PARAMETERS
        # a frame count past 2^32 (nothing is read: the device form with a dangling pointer is refused before any copy)
        d = torch.zeros(8, dtype=torch.int16, device=torch.device("cuda", ctx.device))
        assert _code(lambda: pool.push_device([0], d.data_ptr(), [0], [2**32 - 1], d.data_ptr(), [0])) == api.ERR_TOO_MANY_FRAMES
        assert ctx.launch_count == before
        assert list(pool.buffered([0, 1])) == [500, 700]
        # carry on
        o = pool.push([0, 1], [pa, pb])
        outs[0].append(o[0])
        outs[1].append(o[1])
        o = pool.push([0, 1], [a[1800 * C:], b[900 * C:]], end=True)
        outs[0].append(o[0])
        outs[1].append(o[1])
        for sid, x in ((0, a), (1, b)):
            assert pool.header(sid, pool._full, x.size // C) + b"".join(outs[sid]) == oracle.sea_encode(x, RATE, C, ost)
        assert _code(lambda: pool.push([0], [a[:C]])) == api.ERR_INVALID_PARAMETERS  # closed by end
    finally:
        pool.close()


def test_settings_rejected_at_create(ctx):
    with pytest.raises(S.SeaError):
        ctx.encoder_pool(2, RATE, S.EncoderSettings(residual_bits=9.0), 4)
    with pytest.raises(S.SeaError):
        ctx.encoder_pool(2, RATE, S.EncoderSettings(frames_per_chunk=5121), 4)


def test_vbr_ties_per_session_in_call_order(ctx, oracle):
    """Tie-prone inputs (held extremes and squares): per session, the counts summed over its pushes equal the oracle's."""
    st, ost = _pair(oracle, residual_bits=2.5, vbr=True, frames_per_chunk=400)
    C, n = 2, 8
    pool = ctx.encoder_pool(C, RATE, st, n)
    try:
        pool.open(range(n))
        pcms = [np.concatenate([G.crafted(name, C).reshape(-1) for name in ("ties", "saturated", "ties", "phase")]) for _ in range(n)]
        pcms = [np.roll(p, 2 * C * i) for i, p in enumerate(pcms)]
        pos, ties, outs = [0] * n, [0] * n, [[] for _ in range(n)]
        rng = np.random.default_rng(3)
        total = 0
        while any(pos[i] < pcms[i].size for i in range(n)):
            order = [int(i) for i in rng.permutation(n) if pos[i] < pcms[i].size]
            packets = []
            for i in order:
                f = int(rng.integers(1, 700))
                packets.append(pcms[i][pos[i]:pos[i] + f * C])
                pos[i] += f * C
            ends = [pos[i] >= pcms[i].size for i in order]
            o = pool.push(order, packets, end=ends)
            t = ctx.last_vbr_ties_per_stream(len(order))
            total += int(ctx.last_vbr_ties)
            assert int(ctx.last_vbr_ties) == int(t.sum())
            for i, oi, ti in zip(order, o, t):
                outs[i].append(oi)
                ties[i] += int(ti)
        ref_total = 0
        for i in range(n):
            ref, rt = oracle.sea_encode(pcms[i], RATE, C, ost, return_ties=True)
            assert pool.header(i, pool._full, pcms[i].size // C) + b"".join(outs[i]) == ref
            assert ties[i] == rt, i
            ref_total += rt
        assert total == ref_total
    finally:
        pool.close()


def test_launches_per_push(ctx, oracle):
    st = S.EncoderSettings(residual_bits=3.0)
    C, N, n = 2, 5120, 1000
    pool = ctx.encoder_pool(C, RATE, st, n)
    try:
        pool.open(range(n))
        rng = np.random.default_rng(9)
        sizes = rng.integers(0, 3 * N, n)
        packets = [np.zeros(int(f) * C, np.int16) + np.int16(i) for i, f in enumerate(sizes)]
        before = ctx.launch_count
        pool.push(range(n), packets)
        assert ctx.launch_count - before == 3
        # nobody completes a chunk: the ingest alone
        left = N - pool.buffered(range(n)) - 1
        before = ctx.launch_count
        outs = pool.push(range(n), [np.zeros(int(f) * C, np.int16) for f in left])
        assert ctx.launch_count - before == 1 and all(o == b"" for o in outs)
        assert list(pool.buffered(range(n))) == [N - 1] * n
    finally:
        pool.close()


def test_debug_launch_lines(oracle):
    """A 1000-session push prints one ingest, one encode and one commit line; a push that completes no chunk prints no encode."""
    code = r"""
import numpy as np, sea_codec_b200 as S
ctx = S.Context(0)
pool = ctx.encoder_pool(2, 44100, S.EncoderSettings(), 1000)
pool.open(range(1000))
pool.push(range(1000), [np.zeros((5120 + i) * 2, np.int16) for i in range(1000)])
import sys; sys.stderr.write("--- second\n"); sys.stderr.flush()
pool.push(range(1000), [np.zeros(2, np.int16)] * 1000)
pool.close(); ctx.close()
"""
    env = dict(os.environ, SEA_B200_DEBUG_LAUNCH="1")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=root, env=env, timeout=600)
    assert r.returncode == 0, r.stderr
    first, second = r.stderr.split("--- second\n")
    kinds = lambda t: [ln.split(":")[0].split("<")[0] for ln in t.splitlines() if ln.strip()]
    assert kinds(first) == ["pool_ingest_kernel", "encode_kernel", "pool_commit_kernel"], first
    assert kinds(second) == ["pool_ingest_kernel"], second


def test_side_stream(oracle):
    """A context bound to a torch side stream (its own stream is dropped, so the session fixture's context is not used)."""
    import torch

    st, ost = _pair(oracle, residual_bits=3.0)
    C = 2
    c2 = S.Context(0)
    dev = torch.device("cuda", c2.device)
    side = torch.cuda.Stream(device=dev)
    pool = c2.encoder_pool(C, RATE, st, 8)
    try:
        with torch.cuda.stream(side):
            c2.set_stream(side.cuda_stream)
            pool.open(range(8))
            pcms = [synth.gen_stream(70 + i, 5120 * 2 + 333 * i, C, RATE).reshape(-1) for i in range(8)]
            half = [p[: (p.size // C // 2) * C] for p in pcms]
            o1 = pool.push(range(8), half)
            o2 = pool.push(range(8), [p[h.size:] for p, h in zip(pcms, half)], end=True)
        for i in range(8):
            frames = pcms[i].size // C
            assert pool.header(i, pool._full, frames) + o1[i] + o2[i] == oracle.sea_encode(pcms[i], RATE, C, ost)
    finally:
        pool.close()
        c2.close()
