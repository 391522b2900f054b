// decode_mc.cuh -- throughput decode for uniform CBR batches with MORE than two channels (3 .. 8; BASELINE config 3 is an
// 8-channel stream, the reference's own tests use 3 -- tests/test.rs:10): decode_mc_kernel<CT, B, S4>.  The template lives in a
// header so that the even and the odd channel counts compile as two translation units (decode_mc.cu, decode_mc_odd.cu).
//
// Lane mapping: one lane per chunk with ALL its channels.  In the [frame][channel] bit stream (chunk.rs:254-278) a frame's CT
// codes are adjacent, so the lane walks the residual section front to back with CT independent LMS chains in registers (the ILP
// of the stereo kernel and more) and owns whole PCM frames: they leave as full 32-byte sectors.  (The first versions gave a lane
// one channel pair, then a quad: 4/8-byte stores to 32 different rows per instruction -- the L1 tag stage, not the math,
// bounded 6 channels at 0.67 and 8 at 0.93 Tsamples/s; profiles/r01_decode_mc_v1/v2.)  Everything else is borrowed from
// decode_unrolled_kernel / decode_vbr_kernel: per-lane cp.async ring, a window of big-endian words per body pre-shifted once so
// that every field position inside the body is a compile-time constant, I2IP pack-saturate clamp, LMS signs carried in registers.
//
// Store phases.  A body is HF frames = HF * CT / 2 PCM words.  Where that is not a multiple of the 8 words of a 256-bit store
// (6 channels: 12 words; 3 / 5 / 7 channels: 6 / 10 / 14 words), consecutive bodies start 4 resp. 2 or 6 words further into a
// 32-byte row: the body is instantiated once per phase (2 resp. 4 of them, ParTag) and the words of a row that a body leaves
// open wait in registers for the next one.  With an odd channel count a PCM word also straddles two frames (the last channel of
// an even frame and the first of the odd one): the straddling sample is clamped on its own for the history and packed when its
// partner exists.  S4: scale_factor_bits == 4 and an even channel count (a block's scale factors are CT / 2 whole bytes);
// otherwise the block's CT * s bits are cut out of a 64-bit big-endian window (s <= 6).
#pragma once
#include "sea_device.cuh"

namespace sea {

using namespace dev;

namespace {

template <int V>
struct ParTag {
    static constexpr int value = V;
};

#ifndef SEA_MC_HF8
#define SEA_MC_HF8 10
#endif
#ifndef SEA_MC_WARPS8
#define SEA_MC_WARPS8 12
#endif
#ifndef SEA_MC_WARPS3
#define SEA_MC_WARPS3 16
#endif

template <int CT, int B>
struct MCfg {
    static constexpr int F = 20;
    static constexpr int kChunksPerWarp = 32;
    // frames per looped body (divides F; even, so that a body is whole PCM words): bounded by the window registers (body bits / 32)
    // and by the code size of its phases (4 x 14 KB for 7 channels)
    static constexpr int HF = CT == 4 ? 20 : (CT == 8 ? (B <= 4 ? SEA_MC_HF8 : 4) : 4);
    static constexpr int kBodyWords = HF * CT / 2;      // 32-bit PCM words per body
    static constexpr int kPhaseWords = kBodyWords % 8;  // how far a body moves the position inside a 32-byte row
    static constexpr int kPhases = kPhaseWords == 0 ? 1 : (kPhaseWords == 4 ? 2 : 4);
    static_assert((HF * CT) % 2 == 0 && kPhaseWords % 2 == 0, "a body must be whole PCM words and an even number of them");
    static constexpr int kBodyBits = HF * CT * B;       // bits of the stream one body walks through
    // The window of pre-shifted big-endian words is loaded once per cycle of phases where that is <= 10 words (every phase is its
    // own instantiation of the body, so the fields of a later body are compile-time positions further into the same window;
    // 3 channels: 17 instructions per 48 samples instead of 20 per 12), else once per body.
#ifndef SEA_MC_WIN_CYCLE
#define SEA_MC_WIN_CYCLE 1
#endif
    static constexpr int kWinBodies = (SEA_MC_WIN_CYCLE && kPhases * kBodyBits <= 320) ? kPhases : 1;
    static constexpr int kWinBits = kWinBodies * kBodyBits;
    static constexpr int kNW = (kWinBits + 31 + 31) / 32;   // window words from the first field to the last (any bit phase)
    // The ring is topped up once per cycle of phases (kPhases bodies: a 4-frame body of 3 channels is 12 samples -- the ~10
    // instructions of a top-up slot per body were 1.7 per sample there), so the unit the ring is sized for is that cycle.
    static constexpr int kCycleBytesMax = (kPhases * kBodyBits + 7) / 8 + 1;
    static constexpr int kTopBodies = 2 * kCycleBytesMax + 32 <= 256 ? kPhases : 1;  // bodies per top-up (7 channels x 8 bits: every body)
    static constexpr int kBodyBytesMax = (kTopBodies * kBodyBits + 7) / 8 + 1;
    static constexpr int kRingWords = 64;               // 256-byte ring per lane: two cycles (<= 112 bytes each) plus slack
    static constexpr int kTopUp = (kBodyBytesMax + 15) / 16 + 1;  // granules issued per cycle at most
    // The ring is kept full, so the bytes of a cycle were issued (256 - 32) / cycle bytes - 1 cycles before it is decoded: that many
    // of the newest groups may still be in flight.  (Waiting for all but the newest one stalled every body on loads it would
    // not need for another 4-5 bodies: long_scoreboard 1.35 per issue in profiles/r01_decode_mc_v2.)
    static constexpr int kAhead = (256 - 32) / kBodyBytesMax - 1;
    static constexpr int kKeep = kAhead < 1 ? 1 : (kAhead > 4 ? 4 : kAhead);
    static constexpr int kPitch = 256 + 16;
    static constexpr int kWarpBytes = 32 * kPitch + 64;
    // measured: 4 channels 2.14 ms at 16 warps (2.46 at 12); 8 channels 12 warps (168 registers)
    static constexpr int kWarps = CT == 4 ? 16 : (CT == 3 ? SEA_MC_WARPS3 : SEA_MC_WARPS8);
    static_assert(2 * kBodyBytesMax + 32 <= 256, "ring too small for two cycles of bodies");
    static constexpr int kSfBytesGeneric = (CT * 6 + 7 + 7) / 8;  // bytes that hold a block's CT * s bits at any bit phase, s <= 6
    static_assert(kSfBytesGeneric <= 8, "the scale factors of a block must fit a 64-bit window");
};

}  // namespace

template <int CT, int B, bool S4>
__global__ void __launch_bounds__(MCfg<CT, B>::kWarps * 32, 1)
decode_mc_kernel(const uint8_t *__restrict__ sea, int16_t *__restrict__ pcm, const DecStream *__restrict__ streams, DecFastParams p,
                 const int32_t *__restrict__ tab, int *err)
{
    using Cfg = MCfg<CT, B>;
    static_assert(!S4 || CT % 2 == 0, "the byte-per-pair scale-factor path needs an even channel count");
    extern __shared__ __align__(1024) uint8_t smem[];
    const uint32_t s = S4 ? 4u : p.s;
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;

    // dequant rows of size B as uploaded: lut[sf][code], at the start of the (1024-byte aligned) shared window so that a row's
    // base address has its low B + 2 bits clear and "row | code << 2" needs no add
    const uint32_t nwarps = blockDim.x >> 5;  // chosen per launch (launch_mc): fewer warps per CTA when the grid is only a few waves
    const uint32_t smem_sh = smem_u32(smem), lut_sh = (smem_sh + 1023u) & ~1023u;
    int32_t *lut = reinterpret_cast<int32_t *>(smem + (lut_sh - smem_sh));
    for (uint32_t i = threadIdx.x; i < (1u << (s + B)); i += blockDim.x) lut[i] = tab[tab_dqt_off(s, B) + i];
    __syncthreads();
    const uint32_t rings_off = (lut_sh - smem_sh) + (4u << (s + B));

    uint64_t g = ((uint64_t)blockIdx.x * nwarps + warp) * Cfg::kChunksPerWarp + lane;  // global chunk index
    const bool valid = g < p.total_chunks;
    if (!valid) g = p.total_chunks - 1;  // idle lanes shadow the last chunk and never store

    const DecStream st = streams[find_stream(streams, p.n_streams, g * CT)];
    const uint32_t k = (uint32_t)(g - st.chain_begin / CT);
    const uint64_t ck_off = st.data_off + (uint64_t)k * p.chunk_size;
    const uint8_t *ck = sea + ck_off;
    {
        const uint32_t word = (uint32_t)ck[0] | ((uint32_t)ck[1] << 8) | ((uint32_t)ck[2] << 16) | ((uint32_t)ck[3] << 24);
        if (word != p.hdr_word) report(err, kDevFallback);  // not what this kernel was specialised for: host reruns generically
    }
    int32_t w[CT][4], h[CT][4], sg[CT][4];
#pragma unroll
    for (int c = 0; c < CT; c++) {
        const uint8_t *l = ck + 4u + 16u * c;  // lms.rs:80-94
#pragma unroll
        for (int i = 0; i < 4; i++) {
            h[c][i] = (int16_t)(l[2 * i] | (l[2 * i + 1] << 8));
            w[c][i] = (int16_t)(l[8 + 2 * i] | (l[8 + 2 * i + 1] << 8));
            sg[c][i] = (h[c][i] >> 31) | 1;
        }
    }
    const uint32_t items = (p.N / Cfg::F) * CT;
    const uint64_t sf_off = ck_off + 4u + 16u * CT;              // chunk.rs:108-113
    const uint64_t res_off = sf_off + (items * s + 7u) / 8u;     // the section is padded to a whole byte (bits.rs:120-128)
    const uint8_t *sfp = sea + sf_off;
    uint8_t *out = reinterpret_cast<uint8_t *>(pcm + st.pcm_off + (uint64_t)k * p.N * CT);

    // ---- per-lane ring.  Word w of the 16-byte aligned stream sits at ring word (w & 63).
    const uint64_t a0 = res_off & ~(uint64_t)15;
    const uint8_t *src0 = sea + a0;
    const uint32_t ring_sh = smem_u32(smem + rings_off + warp * Cfg::kWarpBytes) + lane * Cfg::kPitch + (lane >> 3) * 16u;
    uint32_t fetched = 0;                                        // granules issued so far
    uint32_t posg = (uint32_t)(res_off - a0) * 8u;               // bit position of the current body's first field, from a0
#pragma unroll
    for (int t = 0; t < 16; t++) cp_async16_if(true, ring_sh + t * 16, src0 + t * 16);
    fetched = 16;
    cp_async_commit();
    cp_async_commit();
    cp_async_wait<0>();

    const uint32_t n_bodies = p.N / Cfg::HF;
    constexpr int kBodiesPerBlock = Cfg::F / Cfg::HF;
    // Scale factors of a block.  The bytes of the NEXT block are requested when a block starts and only combined when the next
    // one does: consumed right after the load (the first version) every block waited out a global-memory round trip -- 22 % of
    // the stall samples of profiles/r01_decode_mc_v3 sat on the shift behind that load.
    constexpr int kSfBytes = S4 ? CT / 2 : Cfg::kSfBytesGeneric;
    uint32_t sf_raw[kSfBytes];
    uint32_t sf_phase = 0;  // generic path: bit offset of the requested block's first field inside sf_raw[0]
    auto request_sf = [&](uint32_t blk) {
        const uint32_t bit0 = blk * (uint32_t)CT * s;
        const uint8_t *q = sfp + (bit0 >> 3);  // the bytes past the section's end that the last blocks touch are residual bytes of this chunk
        sf_phase = bit0 & 7u;
#pragma unroll
        for (int j = 0; j < kSfBytes; j++) asm volatile("ld.global.nc.u8 %0, [%1];" : "=r"(sf_raw[j]) : "l"(q + j));
    };
    uint32_t rowbase[CT];  // shared-window address of lut[sf of my channel c in the current block][0]
    auto combine_sf = [&]() {
        if (S4) {
            uint32_t v = 0;
#pragma unroll
            for (int j = 0; j < kSfBytes; j++) v = (v << 8) | sf_raw[j];
#pragma unroll
            for (int c = 0; c < CT; c++) rowbase[c] = lut_sh + (((v >> (4 * (CT - 1 - c))) & 15u) << (B + 2));
        } else {
            uint64_t v = 0;
#pragma unroll
            for (int j = 0; j < kSfBytes; j++) v = (v << 8) | (uint64_t)sf_raw[j];
            const uint32_t top = 8u * kSfBytes - sf_phase;  // bits of v from my first field's MSB down
            const uint32_t m = (1u << s) - 1u;
#pragma unroll
            for (int c = 0; c < CT; c++) rowbase[c] = lut_sh + (((uint32_t)(v >> (top - (uint32_t)(c + 1) * s)) & m) << (B + 2));
        }
    };
    request_sf(0);
    const uint32_t n_blocks = p.N / Cfg::F;
    uint32_t blk_next = 0;  // the block whose scale factors are in flight
    uint32_t bib = 0;       // body inside the block

    uint32_t W[Cfg::kNW];   // the window (carried across the bodies of a cycle when kWinBodies > 1)
    uint32_t ow[8];         // the 32-byte store being assembled (carried across bodies when kPhases > 1)
    int32_t pend = 0;       // odd channel counts: the clamped last channel of an even frame, waiting for its word partner
    auto body = [&](uint32_t bd, auto parity_tag) {
        constexpr int kPhase = (decltype(parity_tag)::value * Cfg::kPhaseWords) % 8;  // words of the open 32-byte row before this body
        // ---- top the ring up (first body of a cycle), then wait for everything but that (the bytes of this cycle were issued a cycle ago)
        if (decltype(parity_tag)::value % Cfg::kTopBodies == 0) {
            const uint32_t wq = posg >> 5;
#pragma unroll
            for (int t = 0; t < Cfg::kTopUp; t++) {
                const bool room = fetched * 4u + 4u <= wq + (uint32_t)Cfg::kRingWords;
                cp_async16_if(room, ring_sh + (fetched & 15u) * 16u, src0 + (size_t)fetched * 16u);
                fetched += room ? 1u : 0u;
            }
            cp_async_commit();
            cp_async_wait<Cfg::kKeep>();
        }
        if (bib == 0) {
            combine_sf();
            blk_next++;
            if (blk_next < n_blocks) request_sf(blk_next);
        }
        bib = (kBodiesPerBlock == 1 || bib == (uint32_t)kBodiesPerBlock - 1u) ? 0u : bib + 1u;

        // ---- window: big-endian words from the first field of this body (cycle) on, pre-shifted so that it starts at bit 0 of W[0]
        if (decltype(parity_tag)::value % Cfg::kWinBodies == 0) {
            const uint32_t w0 = posg >> 5, sh = posg & 31u;
            uint32_t V[Cfg::kNW + 1];
#pragma unroll
            for (int t = 0; t < Cfg::kNW + 1; t++) V[t] = __byte_perm(lds_u32(ring_sh + ((w0 + t) & 63u) * 4u), 0, 0x0123);
#pragma unroll
            for (int t = 0; t < Cfg::kNW; t++) W[t] = __funnelshift_l(V[t + 1], V[t], sh);
            posg += Cfg::kWinBits;
        }
        constexpr int kBit0 = (decltype(parity_tag)::value % Cfg::kWinBodies) * Cfg::kBodyBits;  // this body's first bit in W[]

        uint8_t *ob = out + (size_t)bd * (Cfg::kBodyWords * 4) - kPhase * 4;  // the 32-byte row this body starts in
        auto emit = [&](int wb, uint32_t word) {  // wb: word index inside the body (folds to a constant after unrolling)
            const int widx = kPhase + wb;
            ow[widx % 8] = word;
            if (widx % 8 == 7 && valid) st_global_256(ob + (widx / 8) * 32, ow);
        };
#pragma unroll
        for (int fi = 0; fi < Cfg::HF; fi++) {
            constexpr int kGB = CT * B;
            const int bit = kBit0 + fi * CT * B;  // compile-time position of the frame's codes in W[]
            const int wd = bit >> 5, off = bit & 31;
            uint32_t x = 0;  // the frame's CT codes in the low CT*B bits, first channel highest (frames of up to 32 bits)
            if (kGB <= 32) {
                if (off + kGB <= 32) x = W[wd] >> (32 - off - kGB);
                else x = __funnelshift_r(W[wd + 1], W[wd], (64 - off - kGB) & 31);
            }
            int32_t y[CT], d[CT], sgn[CT];
#pragma unroll
            for (int c = 0; c < CT; c++) {
                // the code lands at bit 2 (the table's 4-byte stride) in ONE shift; mask and row base join it in one LOP3
                uint32_t code4;
                constexpr uint32_t kMask4 = ((1u << B) - 1u) << 2;
                if (kGB <= 32) {
                    const int sh2 = B * (CT - 1 - c) - 2;
                    code4 = sh2 >= 0 ? (x >> (sh2 & 31)) : (x << ((-sh2) & 31));
                } else {  // wider frames: every field on its own, still at a compile-time position
                    const int cb = bit + c * B, cw = cb >> 5, co = cb & 31;
                    if (co + B + 2 <= 32) code4 = W[cw] >> (32 - co - B - 2);
                    else if (co + B <= 32) code4 = W[cw] << ((co + B + 2 - 32) & 31);
                    else code4 = __funnelshift_r(W[cw + 1], W[cw], (64 - co - B - 2) & 31);
                }
                d[c] = lds_s32((code4 & kMask4) | rowbase[c]);
                const uint32_t acc = (uint32_t)w[c][0] * (uint32_t)h[c][0] + (uint32_t)w[c][1] * (uint32_t)h[c][1] +
                                     (uint32_t)w[c][2] * (uint32_t)h[c][2] + (uint32_t)w[c][3] * (uint32_t)h[c][3];
                y[c] = (int32_t)((uint32_t)((int32_t)acc >> 13) + (uint32_t)d[c]);  // codec/decoder.rs:38, before the clamp
                sgn[c] = (y[c] >> 31) | 1;                                            // the clamp keeps the sign
            }
            // clamp_i16 (common.rs:5-8) x2 + interleave: one I2IP per PCM word, the clamped values unpacked for the history
            const int s0 = fi * CT;           // sample index of the frame's first channel inside the body
            const int lead = s0 & 1;          // 1: channel 0 completes the word the previous frame left open (odd CT only)
            if (lead) {
                uint32_t pk;
                asm("cvt.pack.sat.s16.s32 %0, %1, %2;" : "=r"(pk) : "r"(y[0]), "r"(pend));
                y[0] = (int32_t)pk >> 16;
                emit(s0 >> 1, pk);
            }
#pragma unroll
            for (int q = 0; q < (CT - lead) / 2; q++) {
                const int c0 = lead + 2 * q;
                uint32_t pk;
                asm("cvt.pack.sat.s16.s32 %0, %1, %2;" : "=r"(pk) : "r"(y[c0 + 1]), "r"(y[c0]));
                y[c0] = (int32_t)(int16_t)(pk & 0xffffu);
                y[c0 + 1] = (int32_t)pk >> 16;
                emit((s0 + c0) >> 1, pk);
            }
            if ((CT - lead) & 1) {  // the last channel opens a word: clamp it for the history, pack it when the next frame's first sample exists
                y[CT - 1] = clamp_i16(y[CT - 1]);
                pend = y[CT - 1];
            }
#pragma unroll
            for (int c = 0; c < CT; c++) {
                const int32_t delta = d[c] >> 4;  // lms.rs:43-51
                w[c][0] += delta * sg[c][0];
                w[c][1] += delta * sg[c][1];
                w[c][2] += delta * sg[c][2];
                w[c][3] += delta * sg[c][3];
                h[c][0] = h[c][1]; h[c][1] = h[c][2]; h[c][2] = h[c][3]; h[c][3] = y[c];
                sg[c][0] = sg[c][1]; sg[c][1] = sg[c][2]; sg[c][2] = sg[c][3]; sg[c][3] = sgn[c];
            }
        }
    };
    for (uint32_t bd = 0; bd < n_bodies; bd += Cfg::kPhases) {
        body(bd, ParTag<0>{});
        if constexpr (Cfg::kPhases > 1) body(bd + 1u, ParTag<1>{});
        if constexpr (Cfg::kPhases > 2) {
            body(bd + 2u, ParTag<2>{});
            body(bd + 3u, ParTag<3>{});
        }
    }
}

// frames per chunk the kernel's store phases need: whole blocks and a whole cycle of phases
template <int CT>
constexpr uint32_t mc_frame_multiple()
{
    // HF does not depend on B where it matters here: 4 channels 20 (1 phase), 8 channels 10 or 4 (1 phase), the others 4
    constexpr uint32_t cycle = (uint32_t)(MCfg<CT, 8>::HF * MCfg<CT, 8>::kPhases);
    return cycle % 20u == 0 ? cycle : (20u % cycle == 0 ? 20u : cycle * 5u);  // lcm(cycle, 20) for cycle in {4, 8, 16, 20}
}

template <int CT, int B, bool S4>
static cudaError_t launch_mc(const uint8_t *d_sea, int16_t *d_pcm, const DecStream *d_streams, const DecFastParams &p, const int32_t *tab,
                             int *d_err, cudaStream_t stream)
{
    using Cfg = MCfg<CT, B>;
    const uint32_t warps = pick_cta_warps(p.total_chunks, Cfg::kChunksPerWarp, Cfg::kWarps);
    const size_t lut = ((size_t)4u << (p.s + B)) + 1024u;
    const size_t smem = (size_t)warps * Cfg::kWarpBytes + lut;
    cudaError_t e = cudaFuncSetAttribute(decode_mc_kernel<CT, B, S4>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)((size_t)Cfg::kWarps * Cfg::kWarpBytes + lut));
    if (e != cudaSuccess) return e;
    const uint64_t chunks_per_cta = (uint64_t)warps * Cfg::kChunksPerWarp;
    const uint64_t blocks = (p.total_chunks + chunks_per_cta - 1) / chunks_per_cta;
    debug_launch("decode_mc<%d,%d,%d>: %u warps/CTA, %zu B smem, %llu CTAs", CT, B, (int)S4, warps, smem, (unsigned long long)blocks);
    decode_mc_kernel<CT, B, S4><<<(unsigned)blocks, warps * 32, smem, stream>>>(d_sea, d_pcm, d_streams, p, tab, d_err);
    return cudaGetLastError();
}

template <int CT, bool S4>
static cudaError_t launch_mc_b(const uint8_t *d_sea, int16_t *d_pcm, const DecStream *d_streams, const DecFastParams &p, const int32_t *tab,
                               int *d_err, cudaStream_t stream)
{
    switch (p.b) {
        case 1: return launch_mc<CT, 1, S4>(d_sea, d_pcm, d_streams, p, tab, d_err, stream);
        case 2: return launch_mc<CT, 2, S4>(d_sea, d_pcm, d_streams, p, tab, d_err, stream);
        case 3: return launch_mc<CT, 3, S4>(d_sea, d_pcm, d_streams, p, tab, d_err, stream);
        case 4: return launch_mc<CT, 4, S4>(d_sea, d_pcm, d_streams, p, tab, d_err, stream);
        case 5: return launch_mc<CT, 5, S4>(d_sea, d_pcm, d_streams, p, tab, d_err, stream);
        case 6: return launch_mc<CT, 6, S4>(d_sea, d_pcm, d_streams, p, tab, d_err, stream);
        case 7: return launch_mc<CT, 7, S4>(d_sea, d_pcm, d_streams, p, tab, d_err, stream);
        default: return launch_mc<CT, 8, S4>(d_sea, d_pcm, d_streams, p, tab, d_err, stream);
    }
}

}  // namespace sea
