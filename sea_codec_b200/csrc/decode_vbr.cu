// decode_vbr.cu -- the throughput decode kernel for uniform VBR batches: decode_vbr_kernel<C, RS, S4, KF> (1 or 2 channels,
// scale_factor_frames = 20, scale_factor_bits <= 6 -- S4: the default 4 as a compile-time constant --, full chunks; everything
// else stays with decode_staged_kernel).
//
// Same mapping as decode_unrolled_kernel (decode_fast.cuh): one CHUNK per lane, all C channels of it in one thread, PCM leaves
// the registers as 256-bit stores, LMS signs carried in registers, I2IP pack-saturate clamp.  What VBR changes
// (chunk.rs:126-139, codec/decoder.rs:52-86): every (block, channel) has its own residual size, so field positions are run-time
// values and every lane walks its bit stream at its own pace:
//   * residual bytes are staged per lane into a 128-byte ring (16-byte cp.async granules, topped up once per block, one block
//     ahead of their use);
//   * a 32-bit window is re-read from the ring every K frames (K * frame bits <= 32), so inside those frames a field is one
//     shift by a per-block register and the window advances with one shift;
//   * the dequant rows of the four sizes a chunk can use (header size - 1 .. + 2) sit in shared memory as uploaded
//     ([size][sf][code], 4-byte stride).
#include <stdlib.h>

#include "sea_device.cuh"

namespace sea {

using namespace dev;

namespace {


template <int C>
struct VCfg {
    static constexpr int F = 20;
    static constexpr int kRows = 32;                 // chunks per warp: one per lane
    static constexpr int kBlkPerBody = 4 / C;        // the looped body is 80 samples: 2 stereo blocks / 4 mono blocks
    static constexpr int kBodyFrames = kBlkPerBody * F;
    static constexpr int kBodiesPerRound = 4;        // a round = 16 scale factors (8 bytes) and 16 size codes (4 bytes)
    static constexpr int kRoundFrames = kBodiesPerRound * kBodyFrames;  // 160 stereo / 320 mono
    static constexpr int K = 4 / C;                  // frames per window re-read: K * C * 8 bits <= 32
    static constexpr int kOutFrames = 16 / C;        // frames per 32-byte store
    static constexpr int kRingWords = 32;            // 128-byte ring per lane
    static constexpr int kPitch = 144;               // ring + one pad granule: consecutive lanes start 4 banks apart
    static constexpr int kWarpBytes = kRows * kPitch + 64;  // rows 8j.. skewed by j granules
#ifndef SEA_VBR_WARPS
#define SEA_VBR_WARPS 12
#endif
    static constexpr int kWarps = SEA_VBR_WARPS;
};

}  // namespace

// The dependent look-up is the busiest shared-memory access of this kernel: with the rows as uploaded (4-byte entries, one copy)
// a warp's 32 look-ups cost ~2.5 wavefronts and the LSU data pipe ran 83 % busy with 60 % of its wavefronts excess
// (profiles/r02_dec_vbr3_*).  Every dequantised value fits 16 bits (|d| <= 255 * 99, dqt.rs), so the table is held as int16 and
// every entry is replicated 2^RS times (copy lane & (2^RS - 1) is the one a lane reads): RS = 5 -- a copy per lane, two lanes per
// bank word -- leaves at most 2-way conflicts; the launcher picks the largest RS whose table fits next to the rings.
//
// KF > 0 ("narrow" chunks: every size <= 7, i.e. header size <= 5 -- VBR up to ~5.5 bits): a window is re-read every KF frames
// (KF * C * largest size <= 31 bits: 3 stereo frames at VBR-3 instead of 2) and is NOT shifted along: the right-shift that puts the
// code of (frame k of the group, channel c) at bit 1 -- the int16 table's stride -- is a per-block register, and one LOP3 masks the
// code and joins it with the row base (the table sits 1 KB-aligned, a row starts at a multiple of its own size).  A field costs
// SHF + LOP3 + LDS (the shifting window: 4 instructions per sample), a re-read is shared by 6 samples instead of 4.  KF = 0: the
// first form, any size.
template <int C, int RS, bool S4, int KF>
__global__ void __launch_bounds__(VCfg<C>::kWarps * 32, 1)
decode_vbr_kernel(const uint8_t *__restrict__ sea, int16_t *__restrict__ pcm, const DecStream *__restrict__ streams, DecFastParams p,
                  const int32_t *__restrict__ tab, int *err)
{
    using Cfg = VCfg<C>;
    extern __shared__ __align__(16) uint8_t smem[];
    const uint32_t s = S4 ? 4u : p.s;
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    const uint32_t hb = p.b;                                    // chunk-header residual size
    const uint32_t lo_size = hb > 1u ? hb - 1u : 1u, hi_size = hb + 2u < 8u ? hb + 2u : 8u;

    // ---- dequant rows of sizes lo_size..hi_size, contiguous in the uploaded table (sea_common.cuh: tab_dqt_off)
    const uint32_t lut_words = tab_dqt_off(s, hi_size + 1u) - tab_dqt_off(s, lo_size);
    static_assert(KF == 0 || RS == 0, "the narrow form reads the single-copy table");
    const uint32_t lut_rel = KF ? ((smem_u32(smem) + Cfg::kWarps * Cfg::kWarpBytes + 1023u) & ~1023u) - smem_u32(smem) : Cfg::kWarps * Cfg::kWarpBytes;
    int16_t *lut = reinterpret_cast<int16_t *>(smem + lut_rel);
    for (uint32_t i = threadIdx.x; i < (lut_words << RS); i += blockDim.x) lut[i] = (int16_t)tab[tab_dqt_off(s, lo_size) + (i >> RS)];
    __syncthreads();
    const uint32_t lut_sh = smem_u32(lut) + (lane & ((1u << RS) - 1u)) * 2u;

    uint64_t g = ((uint64_t)blockIdx.x * Cfg::kWarps + warp) * Cfg::kRows + lane;  // global chunk index
    const bool valid = g < p.total_chunks;
    if (!valid) g = p.total_chunks - 1;  // idle lanes shadow the last chunk and never store

    const DecStream st = streams[find_stream(streams, p.n_streams, g * C)];
    const uint32_t k = (uint32_t)(g - st.chain_begin / C);
    const uint64_t ck_off = st.data_off + (uint64_t)k * p.chunk_size;
    const uint8_t *ck = sea + ck_off;
    {
        const uint32_t word = (uint32_t)ck[0] | ((uint32_t)ck[1] << 8) | ((uint32_t)ck[2] << 16) | ((uint32_t)ck[3] << 24);
        if (word != p.hdr_word) report(err, kDevFallback);  // not what this kernel was specialised for: host reruns generically
    }
    int32_t w[C][4], h[C][4], sg[C][4];
#pragma unroll
    for (int c = 0; c < C; c++) {
        const uint8_t *l = ck + 4u + 16u * c;  // lms.rs:80-94
#pragma unroll
        for (int i = 0; i < 4; i++) {
            h[c][i] = (int16_t)(l[2 * i] | (l[2 * i + 1] << 8));
            w[c][i] = (int16_t)(l[8 + 2 * i] | (l[8 + 2 * i + 1] << 8));
            sg[c][i] = (h[c][i] >> 31) | 1;
        }
    }
    const uint32_t items = (p.N / Cfg::F) * C;
    const uint64_t sf_off = ck_off + 4u + 16u * C;              // chunk.rs:108-113
    const uint64_t vbr_off = sf_off + (items * s + 7u) / 8u;    // the section is padded to a whole byte (bits.rs:120-128)
    const uint64_t res_off = vbr_off + (items * 2u + 7u) / 8u;  // chunk.rs:126-139: 2 bits per item
    const uint64_t res_bits_avail = ((uint64_t)p.chunk_size - (res_off - ck_off)) * 8u;
    uint8_t *out = reinterpret_cast<uint8_t *>(pcm + st.pcm_off + (uint64_t)k * p.N * C);

    // ---- per-lane ring of residual bytes.  Word w of the 16-byte aligned stream sits at ring word (w & 31).
    const uint64_t a0 = res_off & ~(uint64_t)15;                 // aligned start of what this lane stages
    const uint8_t *src0 = sea + a0;
    const uint32_t ring_sh = smem_u32(smem + warp * Cfg::kWarpBytes) + lane * Cfg::kPitch + (lane >> 3) * 16u;
    uint32_t fetched = 0;                                        // granules issued so far
    uint32_t posg = (uint32_t)(res_off - a0) * 8u;               // bit position of the next field, from a0
    const uint32_t pos_begin = posg;
#pragma unroll
    for (int t = 0; t < 8; t++) cp_async16_if(true, ring_sh + t * 16, src0 + t * 16);
    fetched = 8;
    cp_async_commit();
    cp_async_commit();  // keeps the "all but the newest group" wait of the first block meaningful
    cp_async_wait<0>();

    // ---- scale factors (8 bytes per round) and size codes (4 bytes per round): aligned words one round ahead, realigned and
    // byte-swapped by PRMT (per-lane byte phase), rotated at the END of a round so that nothing waits for the loads
    const uint32_t *sfw = reinterpret_cast<const uint32_t *>(sea + (sf_off & ~(uint64_t)3));
    const uint32_t *szw = reinterpret_cast<const uint32_t *>(sea + (vbr_off & ~(uint64_t)3));
    const uint32_t sf_sel = 0x0123u + ((uint32_t)sf_off & 3u) * 0x1111u, sz_sel = 0x0123u + ((uint32_t)vbr_off & 3u) * 0x1111u;
    uint32_t sf_a = 0, sf_b = 0, sf_c = 0, sf_n0 = 0, sf_n1 = 0;
    if (S4) {
        sf_a = __ldg(sfw);
        sf_b = __ldg(sfw + 1);
        sf_c = __ldg(sfw + 2);
    }
    uint32_t sz_a = __ldg(szw), sz_b = __ldg(szw + 1), sz_n = 0;
    // other scale_factor_bits: a round's 16 fields are 2 * s whole bytes (<= 12) at any byte phase -> four aligned words, a round ahead
    uint32_t sg_w[4] = {0, 0, 0, 0}, sg_n[4] = {0, 0, 0, 0};
    auto request_sf = [&](uint32_t r) {  // stays inside the chunk: the size codes and the residual section follow
        const uint32_t *q = reinterpret_cast<const uint32_t *>(sea + ((sf_off + (uint64_t)r * 2u * s) & ~(uint64_t)3));
#pragma unroll
        for (int j = 0; j < 4; j++) asm volatile("ld.global.nc.u32 %0, [%1];" : "=r"(sg_n[j]) : "l"(q + j));
    };
    if (!S4) {
        request_sf(0);
#pragma unroll
        for (int j = 0; j < 4; j++) sg_w[j] = sg_n[j];
    }

    // whole bodies (decode_vbr_supported); the last round may hold fewer than kBodiesPerRound of them
    const uint32_t n_bodies = p.N / Cfg::kBodyFrames, n_rounds = (n_bodies + Cfg::kBodiesPerRound - 1u) / Cfg::kBodiesPerRound;
    bool bad = false;

    for (uint32_t r = 0; r < n_rounds; r++) {
        // big-endian: the round's 16 scale-factor nibbles (first in the top nibble of sfr0) and 16 two-bit size codes (szr)
        uint32_t sfr0, sfr1, sfr2 = 0;  // the round's scale factors, big-endian from bit 31 of sfr0 down
        if (S4) {
            sfr0 = __byte_perm(sf_a, sf_b, sf_sel);
            sfr1 = __byte_perm(sf_b, sf_c, sf_sel);
            asm volatile("ld.global.nc.u32 %0, [%1];" : "=r"(sf_n0) : "l"(sfw + 2 * r + 3));  // both stay inside the chunk
            asm volatile("ld.global.nc.u32 %0, [%1];" : "=r"(sf_n1) : "l"(sfw + 2 * r + 4));
        } else {
            const uint32_t sel = 0x0123u + (((uint32_t)sf_off + r * 2u * s) & 3u) * 0x1111u;
            sfr0 = __byte_perm(sg_w[0], sg_w[1], sel);
            sfr1 = __byte_perm(sg_w[1], sg_w[2], sel);
            sfr2 = __byte_perm(sg_w[2], sg_w[3], sel);
            if (r + 1 < n_rounds) request_sf(r + 1);
        }
        const uint32_t szr = __byte_perm(sz_a, sz_b, sz_sel);
        asm volatile("ld.global.nc.u32 %0, [%1];" : "=r"(sz_n) : "l"(szw + r + 2));

#pragma unroll 1
        for (uint32_t bd = 0; bd < (uint32_t)Cfg::kBodiesPerRound && r * Cfg::kBodiesPerRound + bd < n_bodies; bd++) {
            // items of this body: 4 (block, channel) pairs -> 4 nibbles of sfr, 4 size codes of szr
            // this body's four fields from bit 31 down
            uint32_t sf4;
            if (S4) {
                sf4 = ((bd & 2u) ? sfr1 : sfr0) << (16u * (bd & 1u));
            } else {
                const uint32_t o = bd * 4u * s, wi = o >> 5;
                const uint32_t a = wi == 0u ? sfr0 : (wi == 1u ? sfr1 : sfr2), b = wi == 0u ? sfr1 : (wi == 1u ? sfr2 : 0u);
                sf4 = __funnelshift_l(b, a, o & 31u);
            }
            const uint32_t sz4 = szr >> (24u - 8u * bd);                                    // low 8 bits: this body's codes
            uint8_t *ob = out + ((size_t)(r * Cfg::kBodiesPerRound + bd)) * (Cfg::kBodyFrames * C * 2);
            uint32_t ow[8];
            int32_t y_even = 0;
#pragma unroll
            for (int q = 0; q < Cfg::kBlkPerBody; q++) {
                // ---- top the ring up (<= 3 granules: a block consumes at most 40 bytes; narrow chunks: F * C * largest size bits),
                // then wait for everything but that.  Narrow form: the granule that lands in slot 0 is also written to the pad
                // granule behind the ring, so that the word after ring word 31 is its neighbour and a window is [a], [a + 4].
                {
                    constexpr int kMaxSize = KF == 0 ? 8 : (C == 2 ? (KF >= 5 ? 3 : (KF >= 3 ? 5 : 7)) : (KF >= 6 ? 5 : (KF >= 5 ? 6 : 7)));
                    constexpr int kTop = (Cfg::F * C * kMaxSize / 8 + 15) / 16;
                    const uint32_t wq = posg >> 5;
#pragma unroll
                    for (int t = 0; t < kTop; t++) {
                        const bool room = fetched * 4u + 4u <= wq + (uint32_t)Cfg::kRingWords;
                        const uint8_t *gsrc = src0 + (size_t)fetched * 16u;
                        cp_async16_if(room, ring_sh + (fetched & 7u) * 16u, gsrc);
                        if (KF > 0) cp_async16_if(room && (fetched & 7u) == 0u, ring_sh + 128u, gsrc);
                        fetched += room ? 1u : 0u;
                    }
                    cp_async_commit();
                    cp_async_wait<1>();
                }
                uint32_t size[C], rowbase[C];
                uint32_t st_bits = 0;
#pragma unroll
                for (int c = 0; c < C; c++) {
                    const int item = q * C + c;
                    const uint32_t sfv = (sf4 >> (32u - (uint32_t)(item + 1) * s)) & ((1u << s) - 1u);
                    const uint32_t code = (sz4 >> (6 - 2 * item)) & 3u;
                    if (KF > 0) {
                        // header size 2..5 (launch_decode_vbr): every code is a valid size, size = lo_size + code, and the row of
                        // (size, sf) starts 2^(s + lo_size) * (2^code - 1) + (sf << size) entries into the table
                        size[c] = code + lo_size;
                        rowbase[c] = lut_sh - (2u << (s + lo_size)) + ((2u << (s + lo_size)) << code) + (sfv << (size[c] + 1u));
                    } else {
                        const uint32_t sz = code + hb - 1u;  // chunk.rs:136-138
                        bad |= sz < 1u || sz > 8u;
                        size[c] = sz < lo_size ? lo_size : (sz > hi_size ? hi_size : sz);  // keeps the look-up inside the table
                        rowbase[c] = lut_sh + (((((1u << size[c]) - (1u << lo_size)) << s) + (sfv << size[c])) << (1 + RS));
                    }
                    st_bits += size[c];
                }
                // one reconstructed frame: LMS predict / clamp / update for the C dequantised residuals, PCM into the 32-byte store
                auto lms_frame = [&](int fi, const int32_t (&d)[C]) {
                    int32_t y[C];
#pragma unroll
                    for (int c = 0; c < C; c++) {
                        const uint32_t acc = (uint32_t)w[c][0] * (uint32_t)h[c][0] + (uint32_t)w[c][1] * (uint32_t)h[c][1] +
                                             (uint32_t)w[c][2] * (uint32_t)h[c][2] + (uint32_t)w[c][3] * (uint32_t)h[c][3];
                        y[c] = (int32_t)((uint32_t)((int32_t)acc >> 13) + (uint32_t)d[c]);  // codec/decoder.rs:74, before the clamp
                    }
                    uint32_t packed = 0;
                    int32_t sgn[C];
#pragma unroll
                    for (int c = 0; c < C; c++) sgn[c] = (y[c] >> 31) | 1;  // the clamp keeps the sign
                    if (C == 2) {
                        asm("cvt.pack.sat.s16.s32 %0, %1, %2;" : "=r"(packed) : "r"(y[C - 1]), "r"(y[0]));
                        y[0] = (int32_t)(int16_t)(packed & 0xffffu);
                        y[C - 1] = (int32_t)packed >> 16;
                    } else if ((fi & 1) == 0) {
                        y[0] = clamp_i16(y[0]);
                        y_even = y[0];
                    } else {
                        asm("cvt.pack.sat.s16.s32 %0, %1, %2;" : "=r"(packed) : "r"(y[0]), "r"(y_even));
                        y[0] = (int32_t)packed >> 16;
                    }
#pragma unroll
                    for (int c = 0; c < C; c++) {
                        const int32_t delta = d[c] >> 4;  // lms.rs:43-51
                        w[c][0] += delta * sg[c][0];
                        w[c][1] += delta * sg[c][1];
                        w[c][2] += delta * sg[c][2];
                        w[c][3] += delta * sg[c][3];
                        h[c][0] = h[c][1]; h[c][1] = h[c][2]; h[c][2] = h[c][3]; h[c][3] = y[c];
                        sg[c][0] = sg[c][1]; sg[c][1] = sg[c][2]; sg[c][2] = sg[c][3]; sg[c][3] = sgn[c];
                    }
                    if (C == 2) ow[fi & 7] = packed;
                    else if (fi & 1) ow[(fi >> 1) & 7] = packed;
                    if ((fi % Cfg::kOutFrames) == Cfg::kOutFrames - 1 && valid) st_global_256(ob + (fi / Cfg::kOutFrames) * 32, ow);
                };
                // 32 valid bits of the stream at posg (MSB first): two ring words, byte-swapped, funnel-shifted
                auto window = [&]() -> uint32_t {
                    const uint32_t wi = posg >> 5;
                    const uint32_t a = ring_sh + (wi & 31u) * 4u;
                    const uint32_t r0 = lds_u32(a), r1 = KF > 0 ? lds_u32(a + 4u) : lds_u32(ring_sh + ((wi + 1u) & 31u) * 4u);
                    return __funnelshift_l(__byte_perm(r1, 0, 0x0123), __byte_perm(r0, 0, 0x0123), posg & 31u);
                };
                if constexpr (KF > 0) {
                    uint32_t shv[KF][C], mk[C];
#pragma unroll
                    for (int c = 0; c < C; c++) {
                        mk[c] = ((1u << size[c]) - 1u) << 1;
                        shv[0][c] = 31u - (c == C - 1 ? st_bits : size[0]);
#pragma unroll
                        for (int kk = 1; kk < KF; kk++) shv[kk][c] = shv[kk - 1][c] - st_bits;
                    }
                    const uint32_t adv = (uint32_t)KF * st_bits;
#pragma unroll
                    for (int i0 = 0; i0 < Cfg::F; i0 += KF) {
                        constexpr int kLast = Cfg::F % KF;  // frames of the short last group (0: none)
                        const int G = (i0 + KF <= Cfg::F) ? KF : kLast;
                        const uint32_t win = window();
                        posg += G == KF ? adv : (uint32_t)G * st_bits;
#pragma unroll
                        for (int kk = 0; kk < G; kk++) {
                            int32_t d[C];
#pragma unroll
                            for (int c = 0; c < C; c++) d[c] = lds_s16(((win >> shv[kk][c]) & mk[c]) | rowbase[c]);
                            lms_frame(q * Cfg::F + i0 + kk, d);
                        }
                    }
                } else {
                    const uint32_t sh_frame = 32u - st_bits;      // frame field (both channels) -> low bits
                    const uint32_t m_last = (1u << size[C - 1]) - 1u;
#pragma unroll
                    for (int i0 = 0; i0 < Cfg::F; i0 += Cfg::K) {
                        uint32_t win = window();
                        posg += (uint32_t)Cfg::K * st_bits;
#pragma unroll
                        for (int kk = 0; kk < Cfg::K; kk++) {
                            const uint32_t x = win >> sh_frame;
                            win <<= st_bits;
                            int32_t d[C];
#pragma unroll
                            for (int c = 0; c < C; c++) {
                                const uint32_t code = (c == C - 1) ? (x & m_last) : (x >> size[C - 1]);
                                d[c] = lds_s16(rowbase[c] + (code << (1 + RS)));
                            }
                            lms_frame(q * Cfg::F + i0 + kk, d);
                        }
                    }
                }
            }
        }
        sf_a = sf_c;
        sf_b = sf_n0;
        sf_c = sf_n1;
        sz_a = sz_b;
        sz_b = sz_n;
#pragma unroll
        for (int j = 0; j < 4; j++) sg_w[j] = sg_n[j];
    }
    // a size outside 1..8 panics in the reference (common.rs:34); more residual bits than the chunk holds is a slice error
    if (bad || (uint64_t)(posg - pos_begin) > res_bits_avail) report(err, kDevFallback);
}

bool decode_vbr_supported(const DecFastParams &p)
{
    if (p.channels != 1 && p.channels != 2) return false;
    if ((p.hdr_word & 0xffu) != 2u) return false;  // VBR chunks only
    if (p.F != 20 || p.s < 1 || p.s > 6 || p.b < 1 || p.b > 8) return false;
    const uint32_t body_frames = 80u / p.channels;  // VCfg::kBodyFrames: 40 stereo, 80 mono (whole bodies; 32-byte aligned PCM rows)
    if (p.N == 0 || p.N % body_frames != 0) return false;
    return true;
}

template <int C, int RS, bool S4, int KF>
static cudaError_t launch_vbr(const uint8_t *d_sea, int16_t *d_pcm, const DecStream *d_streams, const DecFastParams &p, const int32_t *tab,
                              int *d_err, size_t lut_bytes, cudaStream_t stream)
{
    using Cfg = VCfg<C>;
    const size_t smem = (size_t)Cfg::kWarps * Cfg::kWarpBytes + ((lut_bytes / 2u) << RS) + (KF ? 1024u : 0u);
    cudaError_t e = cudaFuncSetAttribute(decode_vbr_kernel<C, RS, S4, KF>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    const uint64_t chunks_per_cta = (uint64_t)Cfg::kWarps * Cfg::kRows;
    const uint64_t blocks = (p.total_chunks + chunks_per_cta - 1) / chunks_per_cta;
    debug_launch("decode_vbr<%d,%d,%d,%d>: %u warps/CTA, %zu B smem, %llu CTAs", C, RS, (int)S4, KF, (unsigned)Cfg::kWarps, smem, (unsigned long long)blocks);
    decode_vbr_kernel<C, RS, S4, KF><<<(unsigned)blocks, Cfg::kWarps * 32, smem, stream>>>(d_sea, d_pcm, d_streams, p, tab, d_err);
    return cudaGetLastError();
}

cudaError_t launch_decode_vbr(const uint8_t *d_sea, int16_t *d_pcm, const DecStream *d_streams, const DecFastParams &p, DevTables tabs,
                              int *d_err, cudaStream_t stream)
{
    if (p.total_chunks == 0) return cudaSuccess;
    const int32_t *tab = tabs.by_s[p.s];
    const uint32_t lo = p.b > 1u ? p.b - 1u : 1u, hi = p.b + 2u < 8u ? p.b + 2u : 8u;
    const size_t lut_bytes = (size_t)(tab_dqt_off(p.s, hi + 1u) - tab_dqt_off(p.s, lo)) * 4u;
    // int16 entries, 2^RS copies.  Measured (1024 stereo 60 s streams, profiles/r02_probe2.txt): VBR-3 RS 0 / 3 / 4 / 5 = 4.75 /
    // 5.01 / 5.07 / 4.78 ms, VBR-5.5 4.99 / 5.33 / 5.51 / 5.52 ms -- the bank conflicts are not what bounds the kernel (issue
    // slots and the ALU pipe are), and the larger table costs more than the conflicts it removes: one copy is the default.
    // SEA_B200_VBR_RS=n replicates 2^n times where that fits, for tuning runs.
    const size_t rings = (size_t)VCfg<2>::kWarps * VCfg<2>::kWarpBytes, room = 220u * 1024u - rings;
    int rs = 0;
    if (const char *env = getenv("SEA_B200_VBR_RS")) {
        rs = atoi(env);
        if (rs < 0) rs = 0;
        if (rs > 5) rs = 5;
        while (rs > 0 && ((lut_bytes / 2u) << rs) > room) rs--;
    }
    // Narrow chunks (every code a valid size <= 7: header size 2..5; scale_factor_bits >= 3 keeps a row aligned to its own size): the
    // fixed-window form, re-read every KF frames with KF * C * largest size <= 31.  SEA_B200_VBR_KF=0 pins the first form.
    const bool narrow = p.b >= 2u && hi <= 7u && p.s >= 3u && rs == 0 && !(getenv("SEA_B200_VBR_KF") && atoi(getenv("SEA_B200_VBR_KF")) == 0);
#define SEA_VBR_N(CC, KK)                                                                                             \
    return p.s == 4u ? launch_vbr<CC, 0, true, KK>(d_sea, d_pcm, d_streams, p, tab, d_err, lut_bytes, stream)          \
                     : launch_vbr<CC, 0, false, KK>(d_sea, d_pcm, d_streams, p, tab, d_err, lut_bytes, stream)
    if (narrow && p.channels == 1) {
        if (hi <= 5u) SEA_VBR_N(1, 6);
        if (hi == 6u) SEA_VBR_N(1, 5);
        SEA_VBR_N(1, 4);
    }
    if (narrow) {
        if (hi <= 3u) SEA_VBR_N(2, 5);
        if (hi <= 5u) SEA_VBR_N(2, 3);
        SEA_VBR_N(2, 2);
    }
#undef SEA_VBR_N
    // the tuning copies exist for the default scale_factor_bits only
#define SEA_VBR(CC)                                                                                                  \
    if (p.s != 4u) return launch_vbr<CC, 0, false, 0>(d_sea, d_pcm, d_streams, p, tab, d_err, lut_bytes, stream);    \
    switch (rs) {                                                                                                    \
        case 5: return launch_vbr<CC, 5, true, 0>(d_sea, d_pcm, d_streams, p, tab, d_err, lut_bytes, stream);        \
        case 4: return launch_vbr<CC, 4, true, 0>(d_sea, d_pcm, d_streams, p, tab, d_err, lut_bytes, stream);        \
        case 3: return launch_vbr<CC, 3, true, 0>(d_sea, d_pcm, d_streams, p, tab, d_err, lut_bytes, stream);        \
        case 2: return launch_vbr<CC, 2, true, 0>(d_sea, d_pcm, d_streams, p, tab, d_err, lut_bytes, stream);        \
        case 1: return launch_vbr<CC, 1, true, 0>(d_sea, d_pcm, d_streams, p, tab, d_err, lut_bytes, stream);        \
        default: return launch_vbr<CC, 0, true, 0>(d_sea, d_pcm, d_streams, p, tab, d_err, lut_bytes, stream);       \
    }
    if (p.channels == 1) { SEA_VBR(1) }
    { SEA_VBR(2) }
#undef SEA_VBR
}

}  // namespace sea
