// decode_fast.cuh -- the throughput decode kernel for uniform CBR batches (1 or 2 channels, scale_factor_frames = 20,
// full chunks): decode_unrolled_kernel<C, B, MODE, S>.  A header so that mono and stereo compile as two translation units
// (decode_fast.cu: stereo + routing, decode_fast_mono.cu).
//
// Same work as decode_staged_kernel (chunk.rs:69-213 parse, bits.rs:34-50 unpack, codec/decoder.rs:20-50 reconstruct), laid
// out for what bounds it on B200.  The chain recurrence costs ~18 integer instructions per sample while HBM needs only
// 2.4 B/sample, so the limits are the issue slots, the ALU pipe and the shared-memory data pipe, in that order of discovery
// (profiles/r01_decode_*):
//   * one CHUNK per lane (all C channels of it: C independent recurrences per thread, fields of a frame are adjacent bits), a
//     warp owns 32 consecutive chunks, one CTA per SM;
//   * a round is RF frames with RF*C*B a multiple of 32 bits, so every field position inside a round is a compile-time
//     constant: a field costs one shift and one LOP3 that also forms the look-up address;
//   * every lane stages its own chunk row: 16-byte cp.async granules one round ahead into a row-major tile whose pitch is an
//     odd number of granules (conflict-free 128-bit writes); the window words are then read at a per-round word offset and the
//     byte phase of the unaligned section is undone by the same PRMT that swaps to big-endian;
//   * the dequant row table is replicated per bank (lane l reads bank l) when it fits: the one dependent shared load per
//     sample is conflict free;
//   * PCM goes straight from registers to global memory with 256-bit stores (8 stereo / 16 mono frames = one full 32-byte
//     sector per lane per store), so the output never touches shared memory and costs the L1 tag stage no more than a coalesced
//     store would.  (Earlier variants: TMA bulk stores cost ~6 ALU instructions per sample in elect/broadcast loops; an
//     STS.U16 + LDS/STG tile copy saturated the shared-memory pipe at 85 %; 4-byte cp.async and 16-byte stores per lane hit
//     32 sectors per instruction and choked the L1 tag stage.)
#pragma once
#include <stdio.h>
#include <stdlib.h>

#include "sea_device.cuh"

#ifndef SEA_DEC_WARPS
#define SEA_DEC_WARPS 12
#endif
// PAIR (template parameter of the kernel and its configuration): stage the rows with sector-paired requests.  Otherwise every lane
// fetches its own row, 16 bytes per cp.async: the two halves of a 32-byte sector are asked for by two different instructions
// and L2 sends the sector twice (l1tex__m_xbar2l1tex_read_bytes = 3x the .sea bytes, profiles/r01_decode_unrolled_v12).
// Paired: rows start at a 32-byte boundary of the file and lanes 2j / 2j+1 fetch the two halves of ONE sector of row j (then
// row j + 16) -- the destination of a cp.async is any shared address, the source offset of the served row comes by shuffle --
// so that each sector crosses once.  Costs 24 KB more shared memory per 12-warp CTA (rows 32 bytes longer).  Measured at 4096
// streams (profiles/r02_s2_probe_pairfetch.txt): CBR-3 13.70 against 13.89 ms for one launch and NO difference sustained (14.67 /
// 14.69 ms), CBR-1 2.7 % and CBR-6 4 % slower, CBR-8 2.3 % faster, mono 1.5 % slower -- the L2 -> SM over-fetch costs no time.
// Not compiled by default (-DSEA_DEC_PAIRFETCH=1 adds the PAIR instances for full-width CTAs of the default scale_factor_bits).
#ifndef SEA_DEC_PAIRFETCH
#define SEA_DEC_PAIRFETCH 0
#endif

namespace sea {

using namespace dev;

namespace {

template <int C, int B, bool PAIR = false>
struct UCfg {
    static constexpr int F = 20;                              // scale_factor_frames this kernel is unrolled for
    static constexpr int kRows = 32;                          // chunks per warp: one per lane
    static constexpr int HF = 80 / C;                         // frames per unrolled body ("half"): 80 samples, whole blocks
    static constexpr int kBlk = HF / F;                       // scale-factor blocks per half
    static constexpr int kHalfBits = HF * C * B;              // a multiple of 8: a half starts on a byte boundary of the section
    static constexpr int kHalfBytes = kHalfBits / 8;
    static constexpr int kHalves = 2;                         // halves staged per cp.async round
    static constexpr int RF = kHalves * HF;                   // frames per round
    static constexpr int kRoundBytes = kHalves * kHalfBytes;
    static constexpr int kNW = (kHalfBits + 31) >> 5;         // big-endian words of one half (it starts at bit 0 of W[0])
    static constexpr int kInWords = ((3 + (kHalves - 1) * kHalfBytes) >> 2) + kNW + 1;  // words a round can touch from its first word
    static constexpr int kAlignSlack = PAIR ? 28 : 12;                 // word-aligned start of a round inside its staged row
    static constexpr int kSectors = (kAlignSlack + 4 * kInWords + 31) / 32;         // 32-byte sectors of a round (paired fetch)
    static constexpr int kInGranRaw = PAIR ? 2 * kSectors : (kAlignSlack + 4 * kInWords + 15) / 16;  // 16-byte granules incl. alignment slack
    static constexpr int kInGran = (kInGranRaw % 2) ? kInGranRaw : kInGranRaw + 1; // odd pitch: 8 rows tile all bank groups
    static constexpr int kInPitch = kInGran * 16;
    static constexpr int kBufBytes = kRows * kInPitch + 64;  // rows 8j.. are skewed by j granules: conflict-free 32-bit window reads
    static constexpr int kWarpBytes = 2 * kBufBytes;          // double buffered [row][pitch]
    static constexpr int kOutFrames = 16 / C;                 // frames per 32-byte store
    // warps per CTA (one CTA per SM): as many as fit next to <= 33 KB of table, registers allowing (<= 24), multiple of 4
    static constexpr int kWarpsFit = (190 * 1024 / kWarpBytes) / 4 * 4;
    static constexpr int kWarps = kWarpsFit < SEA_DEC_WARPS ? kWarpsFit : SEA_DEC_WARPS;
};

}  // namespace

// MODE: how the dequantised residual of a code is looked up.
//   kLutPlain     lut1[sf][code], 4-byte stride; one shift + one LOP3 per sample.
//   kLutPair      two adjacent fields (the two channels of a frame, or two consecutive mono frames) are positioned by ONE shift:
//                 the second field indexes lut1 (code stride 2^kShift), the first one, B bits higher, indexes lut0 whose code
//                 stride is 2^(kShift+B); the scale-factor rows of lut0 are interleaved into the gaps, so it is no larger.
//   kLutPairRepl  the same with every entry replicated per bank (stride 128 B, lane l at +4l): conflict-free dependent loads.
enum : int { kLutPlain = 0, kLutPair = 1, kLutPairRepl = 2 };

__host__ __device__ constexpr uint32_t lut_shift(int mode) { return mode == kLutPairRepl ? 7u : 2u; }
__host__ __device__ inline uint32_t lut1_bytes(int mode, uint32_t s, uint32_t b) { return 1u << (s + b + lut_shift(mode)); }
__host__ __device__ inline uint32_t lut0_bytes(int mode, uint32_t s, uint32_t b)
{
    return mode == kLutPlain ? 0u : 1u << (lut_shift(mode) + b + (b > s ? b : s));
}
// offset of row sf inside lut0 (code offset and lane offset are added by the caller)
__host__ __device__ inline uint32_t lut0_row(int mode, uint32_t s, uint32_t b, uint32_t sf)
{
    const uint32_t sh = lut_shift(mode);
    return s <= b ? sf << sh : ((sf & ((1u << b) - 1u)) << sh) + ((sf >> b) << (sh + 2u * b));
}

// S: scale_factor_bits as a compile-time constant (3, 4, 5: what tests/test.rs:37 sweeps and seaconv accepts), 0 = run-time value.
template <int C, int B, int MODE, int S, bool PAIR>
__global__ void __launch_bounds__(UCfg<C, B, PAIR>::kWarps * 32, 1)
decode_unrolled_kernel(const uint8_t *__restrict__ sea, int16_t *__restrict__ pcm, const DecStream *__restrict__ streams,
                       DecFastParams p, const int32_t *__restrict__ tab, int *err)
{
    using Cfg = UCfg<C, B, PAIR>;
    extern __shared__ __align__(1024) uint8_t smem[];
    const uint32_t s = S ? (uint32_t)S : p.s;
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    const uint32_t nwarps = blockDim.x >> 5;  // chosen per launch: narrower CTAs (several resident per SM) when the grid is only a few waves

    // ---- dequant rows of residual size B.  Each table sits after the warp tiles at an address aligned to its own size (a power
    // of two), so "row base | code offset" never carries.
    constexpr int kShift = (int)lut_shift(MODE);  // log2 of the byte stride between consecutive codes of lut1
    constexpr bool kPair = MODE != kLutPlain;
    constexpr bool kRepl = MODE == kLutPairRepl;
    const uint32_t smem_sh = smem_u32(smem);
    const uint32_t l0b = lut0_bytes(MODE, s, B), l1b = lut1_bytes(MODE, s, B);
    const uint32_t a0 = l0b < 1024u ? 1024u : l0b, a1 = l1b < 1024u ? 1024u : l1b;
    const uint32_t lut0_abs = (smem_sh + nwarps * Cfg::kWarpBytes + a0 - 1u) & ~(a0 - 1u);
    const uint32_t lut1_abs = (lut0_abs + l0b + a1 - 1u) & ~(a1 - 1u);
    {
        int32_t *lut0 = reinterpret_cast<int32_t *>(smem + (lut0_abs - smem_sh));
        int32_t *lut1 = reinterpret_cast<int32_t *>(smem + (lut1_abs - smem_sh));
        const uint32_t entries = 1u << (s + B);
        const int32_t *src = tab + tab_dqt_off(s, B);
        const uint32_t reps = kRepl ? 32u : 1u;
        for (uint32_t i = threadIdx.x; i < entries * reps; i += blockDim.x) {
            const uint32_t e = kRepl ? i >> 5 : i, l = kRepl ? i & 31u : 0u;
            const int32_t v = src[e];
            lut1[(e << (kShift - 2)) + l] = v;
            if (kPair) lut0[(lut0_row(MODE, s, B, e >> B) >> 2) + ((e & ((1u << B) - 1u)) << (kShift + B - 2)) + l] = v;
        }
    }
    __syncthreads();
    const uint32_t lut_sh = lut1_abs + (kRepl ? lane * 4u : 0u);
    const uint32_t lut0_sh = lut0_abs + (kRepl ? lane * 4u : 0u);

    uint8_t *in_rows = smem + warp * Cfg::kWarpBytes;  // [2][32 rows][kInPitch]

    uint64_t g = ((uint64_t)blockIdx.x * nwarps + warp) * Cfg::kRows + lane;  // global chunk index
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
    const uint64_t sf_off = ck_off + 4u + 16u * C;
    const uint64_t res_off = sf_off + div_ceil_u32(items * s, 8u);
    uint8_t *out = reinterpret_cast<uint8_t *>(pcm + st.pcm_off + (uint64_t)k * p.N * C);

    // whole halves (decode_unrolled_supported); a chunk with an odd number of them ends with a round of one half
    const uint32_t n_halves = p.N / Cfg::HF, n_rounds = (n_halves + Cfg::kHalves - 1u) / Cfg::kHalves;

    // Each lane fetches its own row's next slice as 16-byte granules, one round ahead.
    const uint32_t my_in_sh = smem_u32(in_rows) + lane * Cfg::kInPitch + (lane >> 3) * 16u;
    auto issue_round = [&](uint32_t r) {
        if constexpr (PAIR) {
        const uint64_t mine = (res_off + (uint64_t)r * Cfg::kRoundBytes) & ~(uint64_t)31;  // my row of this round, from a sector boundary
#pragma unroll
        for (int hf = 0; hf < 2; hf++) {
            const uint32_t rr = (lane >> 1) + 16u * hf;  // the row this lane serves: one half of each of its sectors
            const uint64_t so = __shfl_sync(0xffffffffu, mine, rr);
            const uint8_t *src = sea + so + (lane & 1u) * 16u;
            const uint32_t dst = smem_u32(in_rows) + rr * Cfg::kInPitch + (rr >> 3) * 16u + (r & 1u) * Cfg::kBufBytes + (lane & 1u) * 16u;
#pragma unroll
            for (int t = 0; t < Cfg::kSectors; t++) cp_async16(dst + t * 32, src + t * 32);
        }
        } else {
        const uint8_t *src = sea + ((res_off + (uint64_t)r * Cfg::kRoundBytes) & ~(uint64_t)15);
        const uint32_t dst = my_in_sh + (r & 1u) * Cfg::kBufBytes;
#pragma unroll
        for (int t = 0; t < Cfg::kInGranRaw; t++) cp_async16(dst + t * 16, src + t * 16);
        }
        cp_async_commit();
    };
    // Scale factors.  A round carries 8 fields = s whole bytes of the section: they are read as aligned 32-bit words one round
    // ahead and realigned / byte-swapped by PRMT (per-lane byte phase), so a round costs one (s == 4) or three global loads
    // instead of byte loads per field (the byte loads alone were 1.6 L1 tag requests per warp-sample).
    constexpr int kSfFields = Cfg::kBlk * C;                    // fields per half
    static_assert(Cfg::kHalves * kSfFields == 8, "a round carries 8 scale factors = s bytes");
    constexpr bool kS4 = S == 4;
    const uint32_t *sfw = reinterpret_cast<const uint32_t *>(sea + (sf_off & ~(uint64_t)3));
    const uint32_t sf_sel = 0x0123u + ((uint32_t)sf_off & 3u) * 0x1111u;
    uint32_t sf_lo = 0, sf_hi = 0, sf_new = 0;  // s == 4: aligned words r, r+1 and (in flight) r+2 of the section
    uint32_t sf_w[3] = {0, 0, 0}, sf_n[3] = {0, 0, 0};  // other s: the three aligned words that hold round r's s bytes / round r+1's (in flight)
    auto request_sf = [&](uint32_t r) {  // stays inside the chunk: the residual section follows
        const uint32_t *q = reinterpret_cast<const uint32_t *>(sea + ((sf_off + (uint64_t)r * s) & ~(uint64_t)3));
#pragma unroll
        for (int j = 0; j < 3; j++) asm volatile("ld.global.nc.u32 %0, [%1];" : "=r"(sf_n[j]) : "l"(q + j));
    };
    issue_round(0);
    if (kS4) {
        sf_lo = __ldg(sfw);
        sf_hi = __ldg(sfw + 1);
    } else {
        request_sf(0);
#pragma unroll
        for (int j = 0; j < 3; j++) sf_w[j] = sf_n[j];
    }

    for (uint32_t r = 0; r < n_rounds; r++) {
        // my buffer (r+1)&1 was consumed in round r-1 (only I read my row): refill it, then wait for this round's slice
        if (PAIR) __syncwarp();  // other lanes write my row: nobody refills a buffer that its owner may still be reading
        if (r + 1 < n_rounds) issue_round(r + 1);
        else cp_async_commit();
        cp_async_wait<1>();
        if (PAIR) __syncwarp();  // ... and a row is complete when the lanes that fetched it have waited
        // byte offset of the round's first residual byte inside its staged row (the row starts at a 16-byte boundary of the file)
        const uint32_t rb = (uint32_t)(res_off + (uint64_t)r * Cfg::kRoundBytes) & (PAIR ? 31u : 15u);
        const uint32_t row_sh = my_in_sh + (r & 1u) * Cfg::kBufBytes;

        uint32_t sf_round = 0, sf_round1 = 0;  // big-endian: the fields of the first / second half from bit 31 down
        if (kS4) {  // this round's 8 nibbles; then prefetch the word the next round completes with
            sf_round = __byte_perm(sf_lo, sf_hi, sf_sel);
            sf_round1 = sf_round << 16;
            // stays inside the chunk (the residual section follows); rotated into sf_hi at the END of the round so that nothing
            // waits for it here
            asm volatile("ld.global.nc.u32 %0, [%1];" : "=r"(sf_new) : "l"(sfw + r + 2));
        } else {
            const uint32_t sel = 0x0123u + (((uint32_t)sf_off + r * s) & 3u) * 0x1111u;
            const uint32_t hi = __byte_perm(sf_w[0], sf_w[1], sel), lo = __byte_perm(sf_w[1], sf_w[2], sel);
            sf_round = hi;
            sf_round1 = s == 8u ? lo : __funnelshift_l(lo, hi, 4u * s);
            if (r + 1 < n_rounds) request_sf(r + 1);
        }

        // The body below is ONE half (80 samples, every bit position a compile-time constant); it is looped, not unrolled
        // further, so that the code (~24 KB) stays inside the 32 KB L1.5 instruction cache: with the round unrolled (56 KB) the
        // top stall was "no instruction" (profiles/r01_decode_unrolled_lane_per_chunk_v7).
#pragma unroll 1
        for (uint32_t hh = 0; hh < (uint32_t)Cfg::kHalves && r * Cfg::kHalves + hh < n_halves; hh++) {
            const uint32_t gh = r * Cfg::kHalves + hh;
            // scale factors of this half's blocks
            uint32_t sfv[kSfFields];
            {
                const uint32_t rw = hh ? sf_round1 : sf_round;
#pragma unroll
                for (int q = 0; q < kSfFields; q++) sfv[q] = (rw >> (32u - (uint32_t)(q + 1) * s)) & ((1u << s) - 1u);
            }

            // window of this half: big-endian words W[0..kNW), frame fi / channel c sits at bit (fi*C + c)*B.  The half starts at
            // byte ob of the row: aligned words are loaded and the byte phase is undone by the PRMT that also swaps to big-endian.
            constexpr int kNW = Cfg::kNW;
            const uint32_t ob = rb + hh * Cfg::kHalfBytes;
            const uint32_t wsh = row_sh + (ob & ~3u);
            const uint32_t prmt_sel = 0x0123u + (ob & 3u) * 0x1111u;
            uint32_t V[kNW + 1], W[kNW];
#pragma unroll
            for (int t = 0; t < kNW + 1; t++) V[t] = (uint32_t)lds_s32(wsh + 4 * t);
#pragma unroll
            for (int t = 0; t < kNW; t++) W[t] = __byte_perm(V[t], V[t + 1], prmt_sel);

            uint8_t *oh = out + (size_t)gh * (Cfg::HF * C * 2);
            uint32_t ow[8];  // 32 bytes of interleaved PCM being assembled
            int32_t y_even = 0;  // mono: the clamped even frame waiting to be packed with the odd one
            uint32_t xg = 0;  // the field group (one or two codes) last moved into look-up position
#pragma unroll
            for (int q = 0; q < Cfg::kBlk; q++) {
                uint32_t rowbase[C], rowbase0[C];
#pragma unroll
                for (int c = 0; c < C; c++) {
                    rowbase[c] = lut_sh + (sfv[q * C + c] << (B + kShift));
                    rowbase0[c] = kPair ? lut0_sh + lut0_row(MODE, s, B, sfv[q * C + c]) : 0u;
                }
#pragma unroll
                for (int i = 0; i < Cfg::F; i++) {
                    const int fi = q * Cfg::F + i;  // frame inside the half
                    int32_t y[C], d[C];
#pragma unroll
                    for (int c = 0; c < C; c++) {
                        const int n = fi * C + c;            // sample inside the half
                        const int pb = kPair ? (n & ~1) : n;  // first sample of the group positioned by one shift
                        constexpr int kGB = kPair ? 2 * B : B;
                        if (n == pb) {
                            const int bit = pb * B;  // compile-time position of the group in W[]
                            const int wd = bit >> 5, off = bit & 31;
                            if (off + kGB <= 32) {
                                const int rs = 32 - off - kGB - kShift;
                                xg = rs >= 0 ? (W[wd] >> (rs & 31)) : (W[wd] << ((-rs) & 31));
                            } else {
                                xg = __funnelshift_r(W[wd + 1], W[wd], (64 - off - kGB - kShift) & 31);
                            }
                        }
                        uint32_t addr;
                        if (kPair && n == pb) addr = (xg & (((1u << B) - 1u) << (kShift + B))) | rowbase0[c];
                        else addr = (xg & (((1u << B) - 1u) << kShift)) | rowbase[c];
                        d[c] = lds_s32(addr);
                        const uint32_t acc = (uint32_t)w[c][0] * (uint32_t)h[c][0] + (uint32_t)w[c][1] * (uint32_t)h[c][1] +
                                             (uint32_t)w[c][2] * (uint32_t)h[c][2] + (uint32_t)w[c][3] * (uint32_t)h[c][3];
                        y[c] = (int32_t)((uint32_t)((int32_t)acc >> 13) + (uint32_t)d[c]);  // codec/decoder.rs:38, before the clamp
                    }
                    // clamp_i16 (common.rs:5-8).  Stereo: one I2IP saturates both channels and packs them into the output word
                    // (2 issue slots fewer per frame than 4 VIMNMX + PRMT); the clamped values are unpacked for the history.
                    uint32_t packed = 0;
                    int32_t sgn[C];  // the clamp keeps the sign: take it from the unclamped sum (off the I2IP -> unpack path)
#pragma unroll
                    for (int c = 0; c < C; c++) sgn[c] = (y[c] >> 31) | 1;
                    if (C == 2) {
                        asm("cvt.pack.sat.s16.s32 %0, %1, %2;" : "=r"(packed) : "r"(y[C - 1]), "r"(y[0]));
                        y[0] = (int32_t)(int16_t)(packed & 0xffffu);
                        y[C - 1] = (int32_t)packed >> 16;
                    } else if ((fi & 1) == 0) {
                        y[0] = clamp_i16(y[0]);
                        y_even = y[0];
                    } else {  // mono: the odd frame is saturated while it is packed next to the even one
                        asm("cvt.pack.sat.s16.s32 %0, %1, %2;" : "=r"(packed) : "r"(y[0]), "r"(y_even));
                        y[0] = (int32_t)packed >> 16;
                    }
#pragma unroll
                    for (int c = 0; c < C; c++) {
                        const int32_t delta = d[c] >> 4;
                        w[c][0] += delta * sg[c][0];
                        w[c][1] += delta * sg[c][1];
                        w[c][2] += delta * sg[c][2];
                        w[c][3] += delta * sg[c][3];
                        h[c][0] = h[c][1]; h[c][1] = h[c][2]; h[c][2] = h[c][3]; h[c][3] = y[c];
                        sg[c][0] = sg[c][1]; sg[c][1] = sg[c][2]; sg[c][2] = sg[c][3]; sg[c][3] = sgn[c];
                    }
                    // interleaved i16 PCM: 8 stereo frames or 16 mono frames fill one 32-byte (full sector) store
                    if (C == 2) {
                        ow[fi & 7] = packed;
                    } else {
                        if (fi & 1) ow[(fi >> 1) & 7] = packed;
                    }
                    if ((fi % Cfg::kOutFrames) == Cfg::kOutFrames - 1 && valid) st_global_256(oh + (fi / Cfg::kOutFrames) * 32, ow);
                }
            }
        }
        sf_lo = sf_hi;
        sf_hi = sf_new;
#pragma unroll
        for (int j = 0; j < 3; j++) sf_w[j] = sf_n[j];
    }
}

// Look-up mode of decode_unrolled_kernel<C, B> for scale_factor_bits s.  Pairing without replication was measured and dropped:
// lut0's bank is then a function of the scale factor alone (code stride 2^(2+B) bytes), and the conflicts cost more than the
// saved shift (B = 5: 7.3 ms against 4.9 ms plain).
constexpr int unrolled_mode(int s, int b)
{
    const int hi = b > s ? b : s;
    if (s != 3 && s != 4 && s != 5) return kLutPlain;  // run-time s (the S = 0 instances) keeps to the plain table
    return (s + b <= 7 && b + hi <= 8) ? kLutPairRepl : kLutPlain;  // both tables <= 32 KB with 128-byte entries
}

// Dynamic shared memory of a CTA of `warps` warps (pick_cta_warps): the rows of its warps plus its own copy of the tables.
template <int C, int B, bool PAIR = false>
static size_t unrolled_smem(uint32_t s, uint32_t warps)
{
    using Cfg = UCfg<C, B, PAIR>;
    const int mode = unrolled_mode((int)s, B);
    const uint32_t l0 = lut0_bytes(mode, s, B), l1 = lut1_bytes(mode, s, B);
    return (size_t)warps * Cfg::kWarpBytes + (l0 ? (l0 < 1024u ? 1024u : l0) + l0 : 0u) + (l1 < 1024u ? 1024u : l1) + l1;
}

template <int C, int B>
static bool plan_unrolled(uint32_t s)
{
    return UCfg<C, B>::kWarps >= 8 && unrolled_smem<C, B>(s, UCfg<C, B>::kWarps) <= 227u * 1024u;
}

template <int C, int B, int S, bool PAIR>
static cudaError_t launch_unrolled_p(const uint8_t *d_sea, int16_t *d_pcm, const DecStream *d_streams, const DecFastParams &p,
                                     const int32_t *tab, int *d_err, uint32_t warps, cudaStream_t stream)
{
    using Cfg = UCfg<C, B, PAIR>;
    constexpr int kMode = unrolled_mode(S, B);
    const size_t smem = unrolled_smem<C, B, PAIR>(p.s, warps);
    const uint64_t chunks_per_cta = (uint64_t)warps * Cfg::kRows;
    const uint64_t blocks = (p.total_chunks + chunks_per_cta - 1) / chunks_per_cta;
    cudaError_t e = cudaFuncSetAttribute(decode_unrolled_kernel<C, B, kMode, S, PAIR>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)unrolled_smem<C, B, PAIR>(p.s, Cfg::kWarps));
    if (e != cudaSuccess) return e;
    // The carve-out is left to the driver (the smallest that holds the resident CTAs): the kernel wants its L1 -- pinned to the
    // maximum shared-memory carve-out the config-4 launch takes 17.4 instead of 13.9 ms (profiles/r02_s2_probe_pairfetch.txt).
    debug_launch("decode_unrolled<%d,%d,%d,%d,%d>: %u warps/CTA, %zu B smem, %llu CTAs", C, B, kMode, S, (int)PAIR, warps, smem, (unsigned long long)blocks);
    decode_unrolled_kernel<C, B, kMode, S, PAIR><<<(unsigned)blocks, warps * 32, smem, stream>>>(d_sea, d_pcm, d_streams, p, tab, d_err);
    return cudaGetLastError();
}

template <int C, int B, int S>
static cudaError_t launch_unrolled_s(const uint8_t *d_sea, int16_t *d_pcm, const DecStream *d_streams, const DecFastParams &p,
                                     const int32_t *tab, int *d_err, cudaStream_t stream)
{
    using Cfg = UCfg<C, B>;
    if (!plan_unrolled<C, B>(p.s)) return cudaErrorInvalidConfiguration;
    // narrower CTAs for grids of only a few waves -- as long as the CTAs resident on an SM (each with its own copy of the tables)
    // stay within 196 KB, which leaves the kernel 60 KB of L1
    uint32_t warps = pick_cta_warps(p.total_chunks, Cfg::kRows, Cfg::kWarps);
    while (warps < (uint32_t)Cfg::kWarps && unrolled_smem<C, B>(p.s, warps) * (Cfg::kWarps / warps) > 196u * 1024u) warps *= 2u;
    if constexpr (S == 4 && SEA_DEC_PAIRFETCH) {
        const bool pair = warps == (uint32_t)Cfg::kWarps && UCfg<C, B, true>::kWarps == Cfg::kWarps &&
                          unrolled_smem<C, B, true>(p.s, warps) <= 196u * 1024u && !(getenv("SEA_B200_PAIRFETCH") && getenv("SEA_B200_PAIRFETCH")[0] == '0');
        if (pair) return launch_unrolled_p<C, B, S, true>(d_sea, d_pcm, d_streams, p, tab, d_err, warps, stream);
    }
    return launch_unrolled_p<C, B, S, false>(d_sea, d_pcm, d_streams, p, tab, d_err, warps, stream);
}

template <int C, int B>
static cudaError_t launch_unrolled(const uint8_t *d_sea, int16_t *d_pcm, const DecStream *d_streams, const DecFastParams &p,
                                   const int32_t *tab, int *d_err, cudaStream_t stream)
{
    switch (p.s) {
        case 3: return launch_unrolled_s<C, B, 3>(d_sea, d_pcm, d_streams, p, tab, d_err, stream);
        case 4: return launch_unrolled_s<C, B, 4>(d_sea, d_pcm, d_streams, p, tab, d_err, stream);
        case 5: return launch_unrolled_s<C, B, 5>(d_sea, d_pcm, d_streams, p, tab, d_err, stream);
        default: return launch_unrolled_s<C, B, 0>(d_sea, d_pcm, d_streams, p, tab, d_err, stream);
    }
}

template <int C>
static bool plan_unrolled_b(uint32_t b, uint32_t s)
{
    switch (b) {
        case 1: return plan_unrolled<C, 1>(s);
        case 2: return plan_unrolled<C, 2>(s);
        case 3: return plan_unrolled<C, 3>(s);
        case 4: return plan_unrolled<C, 4>(s);
        case 5: return plan_unrolled<C, 5>(s);
        case 6: return plan_unrolled<C, 6>(s);
        case 7: return plan_unrolled<C, 7>(s);
        case 8: return plan_unrolled<C, 8>(s);
        default: return false;
    }
}

template <int C>
static cudaError_t launch_unrolled_c(const uint8_t *d_sea, int16_t *d_pcm, const DecStream *d_streams, const DecFastParams &p,
                                     const int32_t *tab, int *d_err, cudaStream_t stream)
{
    switch (p.b) {
        case 1: return launch_unrolled<C, 1>(d_sea, d_pcm, d_streams, p, tab, d_err, stream);
        case 2: return launch_unrolled<C, 2>(d_sea, d_pcm, d_streams, p, tab, d_err, stream);
        case 3: return launch_unrolled<C, 3>(d_sea, d_pcm, d_streams, p, tab, d_err, stream);
        case 4: return launch_unrolled<C, 4>(d_sea, d_pcm, d_streams, p, tab, d_err, stream);
        case 5: return launch_unrolled<C, 5>(d_sea, d_pcm, d_streams, p, tab, d_err, stream);
        case 6: return launch_unrolled<C, 6>(d_sea, d_pcm, d_streams, p, tab, d_err, stream);
        case 7: return launch_unrolled<C, 7>(d_sea, d_pcm, d_streams, p, tab, d_err, stream);
        default: return launch_unrolled<C, 8>(d_sea, d_pcm, d_streams, p, tab, d_err, stream);
    }
}

}  // namespace sea
