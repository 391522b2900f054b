// encode_kernels.cu -- SEA encoder for sm_100a: scale-factor search, VBR allocation and bit packing on the device.
//
// Replaces EncoderBase::{calculate_residuals, get_residuals_with_best_scalefactor, get_residuals_for_chunk}
// (encoder_base.rs:44-195), CbrEncoder::encode (encoder_cbr.rs:36-66), VbrEncoder::{analyze,
// choose_residual_len_from_errors, encode} (encoder_vbr.rs:98-214), BitPacker (bits.rs:89-135) and
// SeaChunk::serialize (chunk.rs:215-292).
//
// A stream cannot be split by chunk: the LMS state and prev_scalefactor carry over (encoder_base.rs:181-182).
// One CTA owns one stream.  Within it a chain = one channel; the 2^s scale-factor candidates of a block are
// evaluated by the lanes of a chain group in lock step (no early exit: an aborted candidate can never win,
// SURVEY trap T4), a shuffle arg-min on the key (rank, (sf - prev_sf) mod 2^s) picks what the sequential
// reference loop would have kept (trap T1), and the winner's state is written back before the next block.
// The serialized chunk is assembled in shared memory as a big-endian bit string and written out per chunk.
#include <stdlib.h>
#include <string.h>

#include "sea_kernels.h"

namespace sea {

__device__ __forceinline__ void enc_report(int *err, int code) { atomicCAS(err, 0, code); }

// OR an n <= 8 bit field into the big-endian word view of the chunk at absolute bit position pos.
// The image lives in shared memory: the OR goes out as red.shared on a 32-bit shared-window address (atomicOr on the generic
// pointer made the compiler rebuild the window address -- S2UR SR_CgaCtaId, ULEA -- and branch around every call: 7 % of the
// stall samples of the 1024-stream profile).
__device__ __forceinline__ void red_or_shared(uint32_t addr, uint32_t value)
{
    asm volatile("red.shared.or.b32 [%0], %1;" ::"r"(addr), "r"(value) : "memory");
}
__device__ __forceinline__ void put_bits(uint32_t base, uint32_t pos, uint32_t n, uint32_t value)  // base: shared-window address
{
    const uint32_t word = pos >> 5, off = pos & 31u;
    // MSB-first field as a 64-bit big-endian pair: the second word is zero unless the field straddles (OR of 0 is harmless,
    // and one unconditional pair of reductions is cheaper than a divergent branch)
    const uint64_t v64 = (uint64_t)value << (64u - off - n);
    red_or_shared(base + word * 4u, (uint32_t)(v64 >> 32));
    red_or_shared(base + word * 4u + 4u, (uint32_t)v64);  // zero unless the field straddles (the image has two spare words)
}
__device__ __forceinline__ void put_byte(uint32_t base, uint32_t byte_off, uint32_t v) { put_bits(base, byte_off * 8u, 8u, v & 0xffu); }

struct VbrScratch {
    unsigned long long *keys;  // ranks, then sort keys           [npow2]
    uint32_t *idx;             // item index per sorted position   [npow2]
    uint32_t *blkbit;          // bit offset of each block         [nblk]
    uint32_t *rowbits;         // bits per frame of each block     [nblk]
    uint8_t *sizes;            // residual size per (block, channel)
    uint32_t *desc;            // per (block, channel): size | prefix bits << 4 | frame bits << 12 (second pass)  [items]
    uint32_t desc_sh, blkbit_sh;  // shared-window addresses of desc / blkbit when the scratch lives in shared memory, else 0
};

static __host__ __device__ inline uint32_t next_pow2(uint32_t v)
{
    uint32_t p = 2;
    while (p < v) p <<= 1;
    return p;
}

uint64_t enc_vbr_scratch_bytes(const EncParams &p)
{
    if (!p.vbr) return 0;
    const uint64_t nblk = p.N / p.F, items = nblk * p.channels, np2 = next_pow2((uint32_t)items);
    uint64_t bytes = np2 * 8 + np2 * 4 + nblk * 4 + nblk * 4 + items * 4 + items;
    return (bytes + 255) & ~(uint64_t)255;
}

__device__ __forceinline__ VbrScratch carve_scratch(uint8_t *base, const EncParams &p)
{
    const uint32_t nblk = p.N / p.F, items = nblk * p.channels, np2 = next_pow2(items);
    VbrScratch v;
    v.keys = reinterpret_cast<unsigned long long *>(base);
    v.idx = reinterpret_cast<uint32_t *>(base + (uint64_t)np2 * 8);
    v.blkbit = v.idx + np2;
    v.rowbits = v.blkbit + nblk;
    v.desc = v.rowbits + nblk;
    v.sizes = reinterpret_cast<uint8_t *>(v.desc + items);
    v.desc_sh = v.blkbit_sh = 0;
    return v;
}

// One search pass over a chunk (CBR encode, VBR analysis, or VBR encode).  Warps advance independently: a chain
// only depends on its own history.  mode: 0 = encode with uniform size, 1 = analysis (ranks only), 2 = encode with
// per-(block, channel) sizes.
__device__ void search_pass(int mode, uint32_t uniform_size, const EncParams &p, const int16_t *__restrict__ x0, uint32_t frames,
                            const int32_t *__restrict__ tab, int32_t *st_w, int32_t *st_h, int32_t *st_prev, uint8_t *codes,
                            uint32_t chunk_buf, uint32_t sf_sec_bit, uint32_t res_sec_bit, const VbrScratch &vs)
{
    const uint32_t C = p.channels, F = p.F, s = p.s, nsf = 1u << s;
    const uint32_t lpc = nsf < 32u ? nsf : 32u;  // lanes per chain group
    const uint32_t cpw = 32u / lpc;              // chain groups per warp
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const uint32_t grp = lane / lpc, lic = lane % lpc;
    const uint32_t slots = nwarps * cpw;
    const uint32_t T = blockDim.x;
    const uint32_t nblk = div_ceil_u32(frames, F);

    for (uint32_t blk = 0; blk < nblk; blk++) {
        uint32_t nf = frames - blk * F;
        if (nf > F) nf = F;
        for (uint32_t cb = warp * cpw; cb < C; cb += slots) {  // warp-uniform trip count
            const uint32_t c_raw = cb + grp;
            const bool active = c_raw < C;
            const uint32_t c = active ? c_raw : C - 1u;
            const uint32_t size = mode == 2 ? vs.sizes[blk * C + c] : uniform_size;
            const int32_t *recips = tab + tab_recip_off(s, size);
            const int32_t *rows = tab + tab_dqt_off(s, size);
            const int16_t *x = x0 + (uint64_t)blk * F * C + c;

            int32_t rw[4], rh[4];
#pragma unroll
            for (int i = 0; i < 4; i++) {
                rw[i] = st_w[c * 4 + i];
                rh[i] = st_h[c * 4 + i];
            }
            const uint32_t prev = (uint32_t)st_prev[c];

            unsigned long long best_rank = ~0ull;
            uint32_t best_ord = 0xffffffffu, best_sf = 0, best_buf = 0, cur_buf = 0;
            int32_t bw[4] = {0, 0, 0, 0}, bh[4] = {0, 0, 0, 0};
            for (uint32_t sf = lic; sf < nsf; sf += lpc) {
                const uint32_t ord = (sf - prev) & (nsf - 1u);  // position in the reference's rotated visiting order
                const int32_t recip = __ldg(recips + sf);
                const int32_t *row = rows + (sf << size);
                int32_t w[4], h[4], sg[4];
#pragma unroll
                for (int i = 0; i < 4; i++) {
                    w[i] = rw[i];
                    h[i] = rh[i];
                }
                lms_signs(sg, h);
                unsigned long long rank = 0;
                uint8_t *cbuf = codes + (size_t)cur_buf * F * T + threadIdx.x;
                int32_t x_next = __ldg(x);  // the next frame's sample is requested a step ahead: its latency is off the chain
#pragma unroll 4
                for (uint32_t f = 0; f < nf; f++) {  // encoder_base.rs:64-89
                    const int32_t xs = x_next;
                    x_next = __ldg(x + (uint64_t)(f + 1u < nf ? f + 1u : f) * C);
                    const int32_t pr = lms_predict(w, h);
                    const int32_t r = (int32_t)((uint32_t)xs - (uint32_t)pr);
                    const uint32_t code = quant_code(r, recip, size);
                    const int32_t d = __ldg(row + code);
                    const int32_t y = clamp_i16((int32_t)((uint32_t)pr + (uint32_t)d));
                    const int32_t e = xs - y;
                    rank += (unsigned long long)((long long)e * e) + lms_penalty(w);
                    lms_update_sg(w, h, sg, y, d);
                    cbuf[(size_t)f * T] = (uint8_t)code;
                }
                if (rank < best_rank || (rank == best_rank && ord < best_ord)) {
                    best_rank = rank;
                    best_ord = ord;
                    best_sf = sf;
                    best_buf = cur_buf;
                    cur_buf ^= 1u;
#pragma unroll
                    for (int i = 0; i < 4; i++) {
                        bw[i] = w[i];
                        bh[i] = h[i];
                    }
                }
            }
            // arg-min over the chain group: strict total order (rank, ord) -> every lane agrees on the winner
            unsigned long long g_rank = best_rank;
            uint32_t g_ord = best_ord, g_lane = lane, g_buf = best_buf;
            for (uint32_t o = lpc >> 1; o > 0; o >>= 1) {
                const unsigned long long o_rank = __shfl_xor_sync(0xffffffffu, g_rank, o);
                const uint32_t o_ord = __shfl_xor_sync(0xffffffffu, g_ord, o);
                const uint32_t o_lane = __shfl_xor_sync(0xffffffffu, g_lane, o);
                const uint32_t o_buf = __shfl_xor_sync(0xffffffffu, g_buf, o);
                if (o_rank < g_rank || (o_rank == g_rank && o_ord < g_ord)) {
                    g_rank = o_rank;
                    g_ord = o_ord;
                    g_lane = o_lane;
                    g_buf = o_buf;
                }
            }
            if (active && lane == g_lane) {  // encoder_base.rs:181-186: persist the winner
#pragma unroll
                for (int i = 0; i < 4; i++) {
                    st_w[c * 4 + i] = bw[i];
                    st_h[c * 4 + i] = bh[i];
                }
                st_prev[c] = (int32_t)best_sf;
                if (mode == 1) vs.keys[blk * C + c] = best_rank;
                else put_bits(chunk_buf, sf_sec_bit + (blk * C + c) * s, s, best_sf);
            }
            if (mode != 1 && active) {  // chunk.rs:254-278: residual codes, [frame][channel], MSB first
                uint32_t blockbit, rowbits, prefix;
                if (mode == 2) {
                    blockbit = vs.blkbit[blk];
                    rowbits = vs.rowbits[blk];
                    prefix = 0;
                    for (uint32_t cc = 0; cc < c; cc++) prefix += vs.sizes[blk * C + cc];
                } else {
                    rowbits = C * size;
                    blockbit = blk * F * rowbits;
                    prefix = c * size;
                }
                const uint8_t *wbuf = codes + (size_t)g_buf * F * T + (threadIdx.x - lane + g_lane);
                __syncwarp(__activemask());  // the winner's codes were written by another lane (shuffles do not order memory)
                for (uint32_t f = lic; f < nf; f += lpc)
                    put_bits(chunk_buf, res_sec_bit + blockbit + f * rowbits + prefix, size, wbuf[(size_t)f * T]);
            }
            __syncwarp();  // code buffers are reused by the next chain round
        }
    }
}


// ---------------------------------------------------------------------------------------------------------- fast search pass
// Same result as search_pass for scale_factor_bits = 4 (one candidate per lane, two chains per warp), organised around what
// the profile of the generic pass showed (profiles/r01_encode_generic_v1_*): 95 % of the stall samples sat on the global load of
// the PCM sample inside the 20-step recurrence.  Here the block's samples are staged through shared memory one block ahead, the
// dequant rows live in shared memory as [size][code][sf] (the lane's sf is fixed), FB > 0 makes the residual size a compile-time
// constant, and err^2 / penalty^2 are accumulated with 64-bit fused multiply-adds.
// Where the fast pass keeps its dequant rows.  One CTA per stream and ~7 streams per SM at the benchmark's 1024 streams: the
// tables must leave room for that many CTAs (a [code][32 lanes] table of size 8 alone is 32 KB; 3 CTAs per SM cost 2-3x at the
// high bitrates).  kEncLut32: [code][lane], conflict free.  kEncLut16: [code][sf], the two chains of a warp share a row (same
// scale factors; occasional 2-way conflicts).  kEncLutGlobal: the table as uploaded, read with ld.global.nc (L1 resident;
// slower per step than shared memory, so only when nothing else fits).
enum : int { kEncLut32 = 0, kEncLut16 = 1, kEncLutGlobal = 2 };
__host__ __device__ inline uint32_t enc_lut_entries(int fb, uint32_t vbr_base)  // sum over the sizes in use of 2^size
{
    if (fb > 0) return 1u << fb;
    const uint32_t lo = vbr_base > 1u ? vbr_base - 1u : 1u;
    uint32_t n = 0;
    for (uint32_t i = 0; i < 4u; i++)
        if (lo + i <= 8u) n += 1u << (lo + i);
    return n;
}
// CBR: a function of the residual size alone (compile-time in encode_kernel<FB>); VBR: chosen by the host from the CTA's total
// shared memory (launch_encode_generic) and passed in EncParams::lut_mode.
// (scale_factor_bits other than 4: the [code][16] layout does not apply; size 8 reads the table through L1)
__host__ __device__ constexpr int enc_lut_mode_cbr(int fb, int S = 4) { return fb <= 7 ? kEncLut32 : (S == 4 ? kEncLut16 : kEncLutGlobal); }
template <int M>
struct LutTag {
    static constexpr int value = M;
};

// How a trial accumulates the weights penalty of lms.rs:53-62 (all three are exact; the guards are per block and warp-uniform):
//   kRankWide    any weights: 64-bit sum of squares, 64-bit shift, 64x64 square;
//   kRankNarrow  every |w| < 2^23 during the block: the shifted sum fits 31 bits, one 32x32->64 multiply-add;
//   kRankSum32   every |w_i| <= 32767 during a 20-frame block: sum w^2 < 2^32, so it is four 32-bit multiply-adds, the penalty
//                root is <= (2^32 >> 18) - 0x8ff = 14081 and twenty squares of it fit one 32-bit accumulator (20 * 14081^2 < 2^32)
//                that joins the 64-bit rank after the block.  IMAD.WIDE costs the FMA pipe 4 clocks against 2 for IMAD
//                (profiles/r01_int_ops_ubench.txt), and that pipe bounds this kernel wherever two warps share a sub-partition:
//                20 of its 52 clocks per step were these five wide multiplies.  The bound is checked AFTER the trial, from what
//                the candidate actually did: a weight moves by |d >> 4| <= (|d| >> 4) + 1 per frame (lms.rs:43-51), so
//                max|w(0)| + (sum|d| >> 4) + 20 <= 32767 proves it for every frame of the block; the trajectory (codes, history,
//                weights) never depends on the penalty arithmetic, only the rank does, and a block whose proof fails in any lane is
//                simply run again in the 64-bit form.  The CBR instances with the direct quantiser (sizes 1-3) take the bound
//                sum_i (|w_i| + 20 * max|delta|)^2 < 2^32 before the trial instead (the lane's largest magnitude is a register;
//                it holds at ordinary weights there and costs nothing per step; for the larger sizes it never held).
enum : int { kRankWide = 0, kRankNarrow = 1, kRankSum32 = 2 };
template <int V>
struct RankTag {
    static constexpr int value = V;
};

struct FastLut {
    const int32_t *lut;     // shared memory: per size a table [code][32 lanes] (lane & 15 = scale factor)
    uint32_t lut_sh;        // the same as a shared-window address
    const int32_t *recip;   // shared memory: [slot][16]
    // word offset of the table of `size` in [code][32] units: sum of 32 << z over lo_size <= z < size = (32 << size) - (32 << lo_size)
    // (arithmetic, not an array: a runtime index into this struct put it on the stack -- one LDL per block, 4 % of the VBR profile)
    __device__ __forceinline__ uint32_t slot_off(uint32_t size) const { return (32u << size) - (32u << lo_size); }
    uint32_t lo_size;
    int mode;               // kEncLut32 / kEncLut16 / kEncLutGlobal
#ifdef SEA_ENC_DEBUG_SPEC
    unsigned long long *dbg;  // tuning builds: counts the 20-frame blocks that did NOT finish in the 32-bit penalty form
#endif
};

constexpr uint32_t kCodePitch = 36;  // bytes between the frame rows of a warp's code buffer (search_pass_fast)

// S = scale_factor_bits (3, 4 or 5: what seaconv accepts, seaconv.rs:35-41): 2^S candidates per chain = lanes per chain group,
// 32 / 2^S chains per warp.
template <int FB, int S>
__device__ void search_pass_fast(int mode, uint32_t uniform_size, const EncParams &p, const int16_t *__restrict__ x0, uint32_t frames,
                                 const int32_t *__restrict__ tab, int32_t *st_w, int32_t *st_h, int32_t *st_prev, uint8_t *codes,
                                 uint32_t chunk_buf, uint32_t sf_sec_bit, uint32_t res_sec_bit, const VbrScratch &vs, const FastLut &fl,
                                 int16_t *xbuf_all)
{
    constexpr uint32_t s = S, nsf = 1u << S, lpc = nsf, cpw = 32u / lpc;
    constexpr uint32_t kGroupMask = lpc == 32u ? 0xffffffffu : (1u << (lpc & 31u)) - 1u;
    // scale_factor_frames is the default 20 on this path (launch_encode_generic sends everything else to search_pass).  As a
    // runtime value it costs a software division and several constant-bank reloads per block (40 of ~310 per-block instructions
    // in profiles/r02_enc_cbr3_128_v2_*), so the direct-quantiser instances see it as a constant (-2.5 % at CBR-3).  The
    // table-quantiser instances do NOT: with the constant ptxas schedules their trial 6-8 % slower (same-box A/B,
    // profiles/r02_encode_ab.txt), so they keep reading p.F.
#ifndef SEA_ENC_CONSTF_MASK
#define SEA_ENC_CONSTF_MASK 0x0eu  /* bit FB: FB = 1, 2, 3 (VBR, FB = 0, measured a shade faster with the runtime value) */
#endif
    constexpr bool kConstF = FB >= 0 && ((SEA_ENC_CONSTF_MASK >> (FB < 0 ? 0 : FB)) & 1u) != 0u;
    const uint32_t F = kConstF ? 20u : p.F;
    const uint32_t C = p.channels;
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const uint32_t grp = lane / lpc, sf = lane & (lpc - 1u);
    // p.split (few streams, launch_encode_generic): ONE channel per warp -- BASELINE's "one warp per (stream, channel)".  A warp's
    // step costs the same issue slots whether 16 or 32 of its lanes carry a chain, and with fewer warps than sub-partitions
    // every warp runs alone at its own latency, so halving the chains per warp halves the time.  Both lane groups then run the
    // same chain (identical registers, identical votes); group 0 owns the side effects.
    const bool split = p.split != 0u;
    const uint32_t cstep = split ? 1u : cpw;
    const uint32_t slots = nwarps * cstep;
    const uint32_t T = blockDim.x;
    const uint32_t nblk = div_ceil_u32(frames, F);
    int16_t *xbuf = xbuf_all + warp * (cpw * F);  // [chain group][frame]

    for (uint32_t cb = warp * cstep; cb < C; cb += slots) {  // warp-uniform: this warp's pair of channels (split: its channel)
        const uint32_t c_raw = split ? cb : cb + grp;
        const bool active = c_raw < C && !(split && grp != 0u);
        const uint32_t c = c_raw < C ? c_raw : C - 1u;
        // stage block 0: lane l < F brings frame l of both chains
        {
            const uint32_t nf0 = frames < F ? frames : F;
            if (lane < nf0) {
                const int16_t *px = x0 + (uint64_t)lane * C;
#pragma unroll
                for (uint32_t q = 0; q < cpw; q++) xbuf[q * F + lane] = __ldg(px + (cb + q < C ? cb + q : C - 1u));
            }
        }
        __syncwarp();
        // the chain's LMS state and previous scale factor live in registers for the whole pass (identical in the 16 lanes of
        // the chain group); shared memory holds them only between passes and chunks
        int32_t cw[4], chh[4];
#pragma unroll
        for (int i = 0; i < 4; i++) {
            cw[i] = st_w[c * 4 + i];
            chh[i] = st_h[c * 4 + i];
        }
        uint32_t prev = (uint32_t)st_prev[c];
        // ---- direct quantiser (CBR sizes 1..3): the lane's scale factor never changes, so the quantiser + dequantiser of
        // encoder_base.rs:66-75 collapses to comparisons of A = 2|r| - (r < 0) against <= 3 per-lane thresholds and a select
        // among <= 4 per-lane magnitudes -- no 64-bit multiply, no dependent table load on the step's critical path.
        // k >= j  <=>  |n| >= m_j (m_j = 2j; size 2: 3) with n = (r*recip + 2^15) >> 16:
        //   r >= 0: r >= ceil(X/recip),  r < 0: |r| >= floor(X/recip) + 1,  X = 65536*m_j - 32768;
        // both in one unsigned compare A >= 2*ceil(X/recip) - 1 + [recip divides X] (A is even for r >= 0, odd for r < 0).
        // VBR (FB == 0): the sizes change per block, so the thresholds and magnitudes of sizes 1..3 are prepared once per pass and a
        // block whose two chains both have a size <= 3 selects its set (a size below 3 leaves the unused thresholds at "never").
        constexpr bool kDirect = FB >= 1 && FB <= 3;
        constexpr int kLevels = FB == 0 ? 3 : (FB == 3 ? 3 : (FB == 2 ? 1 : 0));
        uint32_t theta[3] = {0xffffffffu, 0xffffffffu, 0xffffffffu};
        int32_t mag[4] = {0, 0, 0, 0};
        uint32_t theta_by[3][3] = {{0xffffffffu, 0xffffffffu, 0xffffffffu}, {0xffffffffu, 0xffffffffu, 0xffffffffu}, {0xffffffffu, 0xffffffffu, 0xffffffffu}};
        int32_t mag_by[3][4] = {};  // [size - 1][level]
        auto direct_setup = [&](uint32_t z, uint32_t rc, uint32_t *th, int32_t *mg) {
            const uint32_t levels = z == 3u ? 3u : (z == 2u ? 1u : 0u);
            const int32_t *row0 = tab + tab_dqt_off(s, z) + (sf << z);
#pragma unroll
            for (uint32_t j = 0; j < 4u; j++)
                if (j <= levels) mg[j] = __ldg(row0 + 2u * j);  // dqt[sf][2k] = +round(sf * curve[k]) (dqt.rs:114-123)
#pragma unroll
            for (uint32_t j = 1; j < 4u; j++)
                if (j <= levels) {
                    const uint32_t m = z == 2u ? 3u : 2u * j;
                    const uint32_t X = 65536u * m - 32768u, q = X / rc, rem = X - q * rc;
                    th[j - 1u] = rem ? 2u * (q + 1u) - 1u : 2u * q;  // 2*ceil - 1 + [divides]
                }
        };
        if (kDirect) direct_setup(FB > 0 ? FB : 1, (uint32_t)fl.recip[sf], theta, mag);
        if (FB == 0) {
#pragma unroll
            for (uint32_t z = 1; z <= 3u; z++)
                if (z >= fl.lo_size && z <= fl.lo_size + 3u) direct_setup(z, (uint32_t)fl.recip[(z - fl.lo_size) * nsf + sf], theta_by[z - 1u], mag_by[z - 1u]);
        }
        uint32_t spec_skip = 0;  // blocks left before the 32-bit penalty form is tried again after a failed proof
        for (uint32_t blk = 0; blk < nblk; blk++) {
            uint32_t nf = frames - blk * F;
            if (nf > F) nf = F;
            // prefetch the next block's samples into registers; they land in shared memory after this block's steps
            int32_t nx[cpw];
            const uint32_t next_frame = (blk + 1u) * F + lane;
            const bool pre = blk + 1u < nblk && lane < F && next_frame < frames;
            if (pre) {
                const int16_t *px = x0 + (uint64_t)next_frame * C;
#pragma unroll
                for (uint32_t q = 0; q < cpw; q++) nx[q] = __ldg(px + (cb + q < C ? cb + q : C - 1u));
            }
            uint32_t bdesc = 0;  // second VBR pass: size | prefix << 4 | frame bits << 12 of this (block, channel)
            if (FB == 0 && mode == 2) {
                if (vs.desc_sh) asm volatile("ld.shared.u32 %0, [%1];" : "=r"(bdesc) : "r"(vs.desc_sh + (blk * C + c) * 4u));
                else bdesc = vs.desc[blk * C + c];
            }
            const uint32_t size = FB > 0 ? (uint32_t)FB : (mode == 2 ? (bdesc & 15u) : uniform_size);
            const uint32_t slot = FB > 0 ? 0u : size - fl.lo_size;
            const int32_t recip = fl.recip[slot * nsf + sf];
            // shared [code][lane] / [code][sf] (two chains share a row) / global [sf][code]: see kEncLut*
            // Two separate views: a global pointer and a 32-bit shared-window address.  (One pointer selected between the two
            // made the VBR kernel's table reads generic LD.E -- long-scoreboard latency on the step's critical path.)
            const int32_t *row = tab + tab_dqt_off(s, size) + (sf << size);
            const uint32_t row_sh = fl.lut_sh + 4u * (fl.mode == kEncLut32 ? fl.slot_off(size) + lane : (fl.slot_off(size) >> 1) + sf);
            const uint32_t kmax = (1u << (size - 1u)) - 1u;

            // every candidate starts from the chain's state (kept in registers: the winner broadcasts it at the end of the block)
            int32_t w[4], h[4], sg[4];
#pragma unroll
            for (int i = 0; i < 4; i++) {
                w[i] = cw[i];
                h[i] = chh[i];
                sg[i] = (h[i] >> 31) | 1;  // lms.rs:45-46 sign of the history, carried along instead of recomputed per tap
            }
            const uint32_t ord = (sf - prev) & (nsf - 1u);  // position in the reference's rotated visiting order
            unsigned long long rank = 0;
            const int16_t *xs = xbuf + (split ? 0u : grp * F);
            // [frame][lane] per warp, rows 36 bytes apart (9 words: the column read of the winners' codes below is conflict free);
            // constant stride, immediate offsets when unrolled
            uint8_t *cbuf = codes + warp * (F * kCodePitch) + lane;
            // the candidate trial (encoder_base.rs:64-89); NARROW picks the short exact form of the weights penalty
            bool direct_now = kDirect;
            if (FB == 0) {
                direct_now = __all_sync(0xffffffffu, size <= 3u);
                if (direct_now) {
                    const bool z3 = size == 3u, z2 = size == 2u;
                    theta[0] = z3 ? theta_by[2][0] : (z2 ? theta_by[1][0] : 0xffffffffu);
                    theta[1] = z3 ? theta_by[2][1] : 0xffffffffu;
                    theta[2] = z3 ? theta_by[2][2] : 0xffffffffu;
                    mag[0] = z3 ? mag_by[2][0] : (z2 ? mag_by[1][0] : mag_by[0][0]);
                    mag[1] = z3 ? mag_by[2][1] : mag_by[1][1];
                    mag[2] = mag_by[2][2];
                    mag[3] = mag_by[2][3];
                }
            }
            uint32_t pen32 = 0, dsum = 0;  // kRankSum32: the block's penalties and sum |d|
            auto trial = [&](auto rank_tag, auto lut_tag, auto unrolled_tag, auto direct_tag) {
                constexpr int kRank = decltype(rank_tag)::value;
                constexpr int kMode = decltype(lut_tag)::value;
                constexpr bool kUnrolled = decltype(unrolled_tag)::value != 0;
                constexpr bool kDir = decltype(direct_tag)::value != 0;
                auto step = [&](uint32_t f) {
                    const int32_t xv = xs[f];
                    // lms.rs:33-41 as a two-level sum (wrapping adds associate): the newest history value enters last
                    const uint32_t acc = ((uint32_t)w[0] * (uint32_t)h[0] + (uint32_t)w[1] * (uint32_t)h[1]) +
                                         ((uint32_t)w[2] * (uint32_t)h[2] + (uint32_t)w[3] * (uint32_t)h[3]);
                    const int32_t pr = (int32_t)acc >> 13;
                    const int32_t r = (int32_t)((uint32_t)xv - (uint32_t)pr);
                    uint32_t code;
                    int32_t d;
                    if (kDir) {
                        const int32_t ms = r >> 31;                                      // 0 / -1
                        const uint32_t A = ((uint32_t)r << 1) ^ (uint32_t)ms;            // 2|r| - (r < 0)
                        int32_t mg = mag[0];
                        uint32_t k2 = 0;
                        if (kLevels == 3) {  // two select levels instead of a chain of three
                            const bool p1 = A >= theta[0], p2 = A >= theta[1], p3 = A >= theta[2];
                            const int32_t lo = p1 ? mag[1] : mag[0], hi = p3 ? mag[3] : mag[2];
                            mg = p2 ? hi : lo;
                            k2 = p2 ? (p3 ? 6u : 4u) : (p1 ? 2u : 0u);
                        } else {
#pragma unroll
                            for (int j = 0; j < kLevels; j++) {
                                const bool ge = A >= theta[j];
                                mg = ge ? mag[j + 1] : mg;
                                k2 = ge ? 2u * (uint32_t)(j + 1) : k2;
                            }
                        }
                        if (kRank == kRankSum32 && !kDirect) dsum += (uint32_t)mg;       // |d|: the proof of the 32-bit penalty form (VBR)
                        d = (mg ^ ms) - ms;                                              // odd code = negative (dqt.rs:118-121)
                        code = k2 - (uint32_t)ms;                                        // 2k + (r < 0)
                    } else {
                    const int32_t n = (int32_t)(((int64_t)r * (int64_t)recip + 32768) >> 16);
                    const uint32_t an = n < 0 ? 0u - (uint32_t)n : (uint32_t)n;
                    // qt.rs:9-31 closed form: 2*min(an >> 1, kmax) == min(an, 2*kmax + 1) & ~1 (size 2: magnitude index is an >= 3)
                    uint32_t k2 = (an < 2u * kmax + 1u ? an : 2u * kmax + 1u) & ~1u;
                    if ((FB > 0 ? (uint32_t)FB : size) == 2u) k2 = an >= 3u ? 2u : 0u;
                    // the sign bit is known long before k2: fold it into the row pointer so that the table address is one
                    // multiply-add after k2 (code itself is only needed for the bit stream)
                    const uint32_t sbit = (uint32_t)r >> 31;
                    code = k2 + sbit;
                    if (kMode == kEncLutGlobal) {
                        d = __ldg(row + sbit + k2);
                    } else {
                        const uint32_t rs = row_sh + (sbit << (kMode == kEncLut32 ? 7 : 6));
                        asm("ld.shared.s32 %0, [%1];" : "=r"(d) : "r"(rs + (k2 << (kMode == kEncLut32 ? 7 : 6))));
                    }
                    if (kRank == kRankSum32) dsum = __sad(d, 0, dsum);  // + |d|
                    }
                    const int32_t v = (int32_t)((uint32_t)pr + (uint32_t)d);
                    const int32_t y = clamp_i16(v);
                    if (kRank == kRankSum32) {
                        const uint32_t sum = (uint32_t)w[0] * (uint32_t)w[0] + (uint32_t)w[1] * (uint32_t)w[1] +
                                             (uint32_t)w[2] * (uint32_t)w[2] + (uint32_t)w[3] * (uint32_t)w[3];
                        const uint32_t t = (uint32_t)__viaddmax_s32((int32_t)(sum >> 18), -0x8ff, 0);
                        pen32 += t * t;
                        const int32_t e = xv - y;
                        rank += (unsigned long long)((long long)e * (long long)e);
                    } else {
                        rank = rank_step<kRank == kRankNarrow>(rank, xv - y, w);
                    }
                    const int32_t delta = d >> 4;  // lms.rs:43-51
#pragma unroll
                    for (int i = 0; i < 4; i++) w[i] += delta * sg[i];
                    h[0] = h[1]; h[1] = h[2]; h[2] = h[3]; h[3] = y;
                    sg[0] = sg[1]; sg[1] = sg[2]; sg[2] = sg[3]; sg[3] = (v >> 31) | 1;  // the clamp keeps the sign
                    cbuf[f * kCodePitch] = (uint8_t)code;
                };
                if (kUnrolled && FB > 0) {  // the default block: fully unrolled (immediate offsets, no loop control, penalties of one
                                            // step scheduled into the table-load shadow of the next)
#pragma unroll
                    for (uint32_t f = 0; f < 20u; f++) step(f);
                } else if (kUnrolled) {
                    // VBR: the blocks of a chunk alternate between several forms of the trial (direct / table, 32-bit / 64-bit
                    // penalty) and the CTAs of an SM sit in different passes: fully unrolled (13 KB each) the hot forms overflow
                    // the 32 KB instruction cache (VBR-4 ran at half speed).  Four steps per iteration keep the register rotation of
                    // the history free and the forms at 2.5 KB each.
#pragma unroll 4
                    for (uint32_t f = 0; f < 20u; f++) step(f);
                } else {
#pragma unroll 4
                    for (uint32_t f = 0; f < nf; f++) step(f);
                }
            };
            // Per-block choice of the penalty form.  The 32-bit form (kRankSum32) is always TRIED on a default block and proved
            // afterwards from what the candidates did (one vote, shared with nothing else on the way in): the three votes that used
            // to pick a form before the trial -- weights narrow? bound for the direct quantiser? weights small enough to try? -- sat
            // on the block's critical path (~40 instructions and three vote latencies of a ~310-instruction epilogue).
            uint32_t m0 = 0;  // max |w_i| at the start of the block (|INT_MIN| wraps to 2^31: never below the limit)
#pragma unroll
            for (int i = 0; i < 4; i++) {
                const uint32_t a = w[i] < 0 ? 0u - (uint32_t)w[i] : (uint32_t)w[i];
                m0 = a > m0 ? a : m0;
            }
            // CBR sizes 1..3 (direct quantiser in every block): the lane's largest magnitude is a register, so the bound
            // sum_i (|w_i| + 20 * max|delta|)^2 < 2^32 is taken BEFORE the trial instead -- one vote, nothing per step (the
            // per-step |d| accumulation of the proof costs these instances 1-2 % at 1024 streams; profiles/r02_encode_ab.txt)
            bool prior32 = false;
            if (kDirect && nf == 20u) {
                const uint32_t grow = 20u * (((uint32_t)mag[kLevels] + 15u) >> 4);
                unsigned long long g = 0;
                bool ok = true;
#pragma unroll
                for (int i = 0; i < 4; i++) {
                    const uint32_t a = (w[i] < 0 ? 0u - (uint32_t)w[i] : (uint32_t)w[i]) + grow;  // <= 2^31 + 20 * 1600
                    ok &= a < 65536u;
                    g += (unsigned long long)a * a;  // meaningful only while ok: four terms below 2^32
                }
                prior32 = __all_sync(0xffffffffu, ok && (g >> 32) == 0ull);
            }
            const bool try32 = !kDirect && nf == 20u && spec_skip == 0u;
            if (spec_skip) spec_skip--;
            auto run = [&](auto lut_tag, auto direct_tag) {
                if (prior32) {
                    trial(RankTag<kRankSum32>{}, lut_tag, LutTag<1>{}, direct_tag);
                    rank += pen32;
                    return;
                }
                if (try32) {
                    trial(RankTag<kRankSum32>{}, lut_tag, LutTag<1>{}, direct_tag);
                    if (__all_sync(0xffffffffu, m0 + (dsum >> 4) + 20u <= 32767u)) {
                        rank += pen32;
                        return;
                    }
                    spec_skip = 8;  // the weights are running close to 2^15: leave the next blocks to the 64-bit form
                    rank = 0;
#pragma unroll
                    for (int i = 0; i < 4; i++) {
                        w[i] = cw[i];
                        h[i] = chh[i];
                        sg[i] = (h[i] >> 31) | 1;
                    }
                }
#ifdef SEA_ENC_DEBUG_SPEC
                if (lane == 0 && nf == 20u) atomicAdd(fl.dbg, try32 ? (1ull << 20) : 1ull);  // failed proofs << 20 | not tried
#endif
                const bool narrow = __all_sync(0xffffffffu, weights_stay_narrow(w, F));
                if (narrow && nf == 20u) trial(RankTag<kRankNarrow>{}, lut_tag, LutTag<1>{}, direct_tag);
                else if (narrow) trial(RankTag<kRankNarrow>{}, lut_tag, LutTag<0>{}, direct_tag);
                else trial(RankTag<kRankWide>{}, lut_tag, LutTag<0>{}, direct_tag);
            };
            if (FB > 0) run(LutTag<enc_lut_mode_cbr(FB > 0 ? FB : 1, S)>{}, LutTag<kDirect ? 1 : 0>{});
            else if (direct_now) run(LutTag<kEncLut32>{}, LutTag<1>{});  // no table on this path
            else if (fl.mode == kEncLut32) run(LutTag<kEncLut32>{}, LutTag<0>{});
            else if (fl.mode == kEncLut16) run(LutTag<kEncLut16>{}, LutTag<0>{});
            else run(LutTag<kEncLutGlobal>{}, LutTag<0>{});
            // arg-min over the 16 candidates of the chain: strict total order (rank, ord); ord follows from the lane.  (Three
            // REDUX min-reductions -- high word, low word, order -- need a third of the instructions but measured 5 % slower at
            // 1024 streams: their latency sits on the per-block critical path of a latency-bound kernel.)
            uint32_t g_lane;
            // Ordinary audio: the WINNING rank is far below 2^27 (the losers of a block -- scale factors that clip -- are not), so ranks
            // are clamped to 2^27 - 1, (rank, ord) fits 31 bits and ONE redux.sync per chain group finds the minimum; a clamped
            // minimum (every candidate >= 2^27 - 1) takes the exact 64-bit butterfly below instead (four dependent shuffle rounds,
            // ~8 % of a latency-bound block).
            constexpr uint32_t kSat = (1u << 27) - 1u;
            const uint32_t rank27 = (rank >> 27) != 0ull ? kSat : (uint32_t)rank;
            const uint32_t best = __reduce_min_sync(kGroupMask << (grp * (lpc & 31u)), (rank27 << s) | ord);
            if (!__any_sync(0xffffffffu, (best >> s) == kSat)) {
                g_lane = grp * lpc + ((best + prev) & (nsf - 1u));
            } else if (!__any_sync(0xffffffffu, (rank >> (64u - s)) != 0ull)) {
                // the usual case: (rank, ord) fits one 64-bit key, a butterfly of 64-bit minima finds the winner's order and
                // the lane follows from it: sf = (ord + prev) mod 16 (encoder_base.rs:116-117)
                unsigned long long key = (rank << s) | ord;
#pragma unroll
                for (uint32_t o = lpc >> 1; o > 0; o >>= 1) {
                    const unsigned long long other = __shfl_xor_sync(0xffffffffu, key, o);
                    key = other < key ? other : key;
                }
                g_lane = grp * lpc + (((uint32_t)key + prev) & (nsf - 1u));
            } else {  // ranks of 2^60 and more (runaway weights penalty): compare (rank, ord) explicitly
                unsigned long long g_rank = rank;
                g_lane = lane;
#pragma unroll
                for (uint32_t o = lpc >> 1; o > 0; o >>= 1) {
                    const unsigned long long o_rank = __shfl_xor_sync(0xffffffffu, g_rank, o);
                    const uint32_t o_lane = __shfl_xor_sync(0xffffffffu, g_lane, o);
                    const uint32_t g_ord = ((g_lane & (lpc - 1u)) - prev) & (nsf - 1u), o_ord = ((o_lane & (lpc - 1u)) - prev) & (nsf - 1u);
                    if (o_rank < g_rank || (o_rank == g_rank && o_ord < g_ord)) {
                        g_rank = o_rank;
                        g_lane = o_lane;
                    }
                }
            }
            // encoder_base.rs:181-186: the winner's state becomes the chain's state -- broadcast in registers
#pragma unroll
            for (int i = 0; i < 4; i++) {
                cw[i] = __shfl_sync(0xffffffffu, w[i], g_lane);
                chh[i] = __shfl_sync(0xffffffffu, h[i], g_lane);
            }
            prev = g_lane & (lpc - 1u);
            if (mode == 1 && active && lane == g_lane) vs.keys[blk * C + c] = rank;
            if (mode != 1) {  // chunk.rs:254-278: residual codes, [frame][channel], MSB first
                // One lane per FRAME: the codes of the warp's channels are adjacent bits of the frame's row, so lane f reads every
                // winner's code and writes them as one field of up to 32 bits (it was one lane per code: two divergent rounds of
                // put_bits per block -- 14 % of the stall samples of profiles/r02_enc_cbr3_128_*).
                const uint32_t nch = split ? 1u : (C - cb < cpw ? C - cb : cpw);  // chain groups of this warp that carry a real channel
                uint32_t gq[cpw], sq[cpw];
                uint32_t blockbit, rowbits, prefix0;
                if (mode == 2) {
                    if (vs.blkbit_sh) asm volatile("ld.shared.u32 %0, [%1];" : "=r"(blockbit) : "r"(vs.blkbit_sh + blk * 4u));
                    else blockbit = vs.blkbit[blk];
                    const uint32_t d0 = __shfl_sync(0xffffffffu, bdesc, 0);
                    rowbits = d0 >> 12;
                    prefix0 = (d0 >> 4) & 255u;
                } else {
                    rowbits = C * size;
                    blockbit = blk * F * rowbits;
                    prefix0 = cb * size;
                }
#pragma unroll
                for (uint32_t q = 0; q < cpw; q++) {
                    gq[q] = __shfl_sync(0xffffffffu, g_lane, (q * lpc) & 31u);
                    sq[q] = mode == 2 ? (__shfl_sync(0xffffffffu, bdesc, (q * lpc) & 31u) & 15u) : size;
                }
                __syncwarp();  // the winners' codes were written by other lanes
                if (lane < nf) {
                    const uint8_t *row = codes + warp * (F * kCodePitch) + lane * kCodePitch;
                    uint32_t field = 0, n = 0;
#pragma unroll
                    for (uint32_t q = 0; q < cpw; q++)
                        if (q < nch) {
                            field = (field << sq[q]) | row[gq[q]];
                            n += sq[q];
                        }
                    put_bits(chunk_buf, res_sec_bit + blockbit + lane * rowbits + prefix0, n, field);
                } else if (lane == 31u) {  // the block's scale factors of this warp's channels (chunk.rs:228-243): adjacent fields, one write
                    uint32_t field = 0;
#pragma unroll
                    for (uint32_t q = 0; q < cpw; q++)
                        if (q < nch) field = (field << s) | (gq[q] & (lpc - 1u));
                    put_bits(chunk_buf, sf_sec_bit + (blk * C + cb) * s, nch * s, field);
                }
            }
            __syncwarp();  // everybody is done with this block's samples and codes
            if (pre) {
#pragma unroll
                for (uint32_t q = 0; q < cpw; q++) xbuf[q * F + lane] = (int16_t)nx[q];
            }
            __syncwarp();
        }
        if (active && sf == 0u) {  // hand the state to the next pass / chunk
#pragma unroll
            for (int i = 0; i < 4; i++) {
                st_w[c * 4 + i] = cw[i];
                st_h[c * 4 + i] = chh[i];
            }
            st_prev[c] = (int32_t)prev;
        }
        __syncwarp();
    }
}

// CTA-wide bitonic sort of (key, idx) pairs, ascending; idx breaks ties (SURVEY trap T13).
__device__ void bitonic_sort(unsigned long long *keys, uint32_t *idx, uint32_t n)
{
    for (uint32_t k = 2; k <= n; k <<= 1) {
        for (uint32_t j = k >> 1; j > 0; j >>= 1) {
            for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) {
                const uint32_t l = i ^ j;
                if (l > i) {
                    const unsigned long long ki = keys[i], kl = keys[l];
                    const uint32_t ii = idx[i], il = idx[l];
                    const bool gt = ki > kl || (ki == kl && ii > il);
                    const bool up = (i & k) == 0;
                    if (gt == up) {
                        keys[i] = kl;
                        keys[l] = ki;
                        idx[i] = il;
                        idx[l] = ii;
                    }
                }
            }
            __syncthreads();
        }
    }
}

// The same sort for the default shape (one warp per CTA, at most 512 items -- stereo chunks of 256 blocks) held in registers:
// element e = r * 32 + lane lives in register r of its lane, so a compare-exchange at distance j < 32 is a shuffle and at
// j >= 32 an exchange between two registers of one lane.  (rank, idx) packs into one 64-bit key while every rank is below 2^55;
// returns false (nothing written) otherwise and the caller takes the shared-memory sort.  The shared-memory version cost 19 k
// instructions per chunk, most of them waiting on generic loads (8 % of the VBR-3 profile); this one is ~6 k with 16-way ILP.
__device__ bool warp_sort_512(unsigned long long *keys, uint32_t *idx, uint32_t n, uint32_t np2)
{
    const uint32_t lane = threadIdx.x & 31u;
    unsigned long long v[16];
    bool fits = true;
#pragma unroll
    for (uint32_t r = 0; r < 16u; r++) {
        const uint32_t e = r * 32u + lane;
        const unsigned long long k = e < n ? keys[e] : 0ull;
        fits &= (k >> 55) == 0ull;
        v[r] = e < n ? (k << 9) | e : ~0ull;
    }
    if (!__all_sync(0xffffffffu, fits)) return false;
    for (uint32_t k = 2; k <= 512u; k <<= 1) {
        for (uint32_t j = k >> 1; j > 0; j >>= 1) {
            if (j >= 32u) {
                auto exchange = [&](auto jr_tag) {
                    constexpr uint32_t jr = decltype(jr_tag)::value;
#pragma unroll
                    for (uint32_t r = 0; r < 16u; r++) {
                        if (r & jr) continue;
                        const bool up = ((r << 5) & k) == 0u;  // k >= 64: the direction depends on the register index only
                        const unsigned long long a = v[r], b = v[r | jr];
                        const bool swap = (a > b) == up;
                        v[r] = swap ? b : a;
                        v[r | jr] = swap ? a : b;
                    }
                };
                switch (j >> 5) {
                    case 1: exchange(LutTag<1>{}); break;
                    case 2: exchange(LutTag<2>{}); break;
                    case 4: exchange(LutTag<4>{}); break;
                    default: exchange(LutTag<8>{}); break;
                }
            } else {
                const bool lower = (lane & j) == 0u;
#pragma unroll
                for (uint32_t r = 0; r < 16u; r++) {
                    const unsigned long long other = __shfl_xor_sync(0xffffffffu, v[r], j);
                    const bool up = (((r << 5) | lane) & k) == 0u;
                    const bool take_min = lower == up;
                    v[r] = ((other < v[r]) == take_min) ? other : v[r];
                }
            }
        }
    }
#pragma unroll
    for (uint32_t r = 0; r < 16u; r++) {
        const uint32_t e = r * 32u + lane;
        if (e < np2) {
            keys[e] = e < n ? v[r] >> 9 : ~0ull;
            idx[e] = e < n ? (uint32_t)v[r] & 511u : 0xffffffffu;
        }
    }
    __syncwarp();
    return true;
}

// FB = -1: generic search pass (any scale_factor_bits);  FB = 0: fast pass, runtime residual sizes (VBR);  FB = 1..8: fast pass, CBR.
template <int FB, int S>
__global__ void encode_kernel(const int16_t *__restrict__ pcm, uint8_t *__restrict__ out, const EncStream *__restrict__ streams,
                              EncParams p, DevTables tabs, int32_t *state, uint64_t *out_lens, uint32_t *chunk0,
                              unsigned long long *ties, EncWorkspace ws, int *err)
{
    extern __shared__ __align__(16) uint8_t smem[];
    const uint32_t sidx = blockIdx.x;
    const EncStream st = streams[sidx];
    const uint32_t C = p.channels, N = p.N, F = p.F, s = p.s, T = blockDim.x, tid = threadIdx.x;
    const int32_t *tab = tabs.by_s[s];

    const uint32_t buf_words = (p.max_chunk_bytes + 3u) / 4u + 2u;
    uint32_t *chunk_buf = reinterpret_cast<uint32_t *>(smem);
    const uint32_t chunk_sh = (uint32_t)__cvta_generic_to_shared(chunk_buf);  // for the red.shared bit writes
    int32_t *st_w = reinterpret_cast<int32_t *>(chunk_buf + buf_words);
    int32_t *st_h = st_w + 4 * C;
    int32_t *st_prev = st_h + 4 * C;
    int32_t *sv_w = st_prev + C;
    int32_t *sv_h = sv_w + 4 * C;
    uint8_t *codes = reinterpret_cast<uint8_t *>(sv_h + 4 * C);
    __shared__ uint32_t sh_res_bits, sh_sorted;
    // fast pass extras: per-warp sample staging and the dequant tables [size][code][sf]
    FastLut fl = {};
    int16_t *xbuf = nullptr;
    if (FB >= 0) {
        uint8_t *extra = codes + ((2u * (size_t)F * T + 15u) & ~(size_t)15u);
        xbuf = reinterpret_cast<int16_t *>(extra);
        constexpr uint32_t kNsf = 1u << (S > 0 ? S : 4), kCpw = 32u / kNsf;
        int32_t *rcp = reinterpret_cast<int32_t *>(extra + (((T >> 5) * kCpw * F * 2u + 15u) & ~15u));
        int32_t *lut = rcp + 4u * kNsf;
        fl.lut = lut;
        fl.lut_sh = (uint32_t)__cvta_generic_to_shared(lut);
#ifdef SEA_ENC_DEBUG_SPEC
        fl.dbg = ties;
#endif
        fl.recip = rcp;
        fl.lo_size = FB > 0 ? (uint32_t)FB : (p.base > 1u ? p.base - 1u : 1u);
        fl.mode = FB > 0 ? enc_lut_mode_cbr(FB > 0 ? FB : 1, S) : (int)p.lut_mode;
        const uint32_t n_slots = FB > 0 ? 1u : 4u;
        uint32_t off = 0;
        for (uint32_t i = 0; i < n_slots; i++) {
            const uint32_t size = fl.lo_size + i;
            if (size <= 8u) {
                for (uint32_t e = tid; e < kNsf; e += T) rcp[i * kNsf + e] = tab[tab_recip_off(s, size) + e];
                if (fl.mode == kEncLut32) {  // [code][32 lanes]: lane l looks its own scale factor l mod 2^S up
                    const uint32_t n = 32u << size;
                    for (uint32_t e = tid; e < n; e += T) lut[off + e] = tab[tab_dqt_off(s, size) + ((e & (kNsf - 1u)) << size) + (e >> 5)];
                } else if (fl.mode == kEncLut16) {  // S == 4 only: [code][16 scale factors], shared by the two chains of a warp
                    const uint32_t n = 16u << size;
                    for (uint32_t e = tid; e < n; e += T) lut[(off >> 1) + e] = tab[tab_dqt_off(s, size) + ((e & 15u) << size) + (e >> 4)];
                }
                off += 32u << size;  // slot offsets are kept in [code][32] units; kEncLut16 halves them
            }
        }
    }

    VbrScratch vs = {};
    if (p.vbr) {
        vs = carve_scratch(p.vbr_smem_off ? smem + p.vbr_smem_off : ws.vbr_scratch + (uint64_t)sidx * ws.vbr_scratch_stride, p);
        if (p.vbr_smem_off) {  // typed shared-memory access for the per-block reads of the second pass
            vs.desc_sh = (uint32_t)__cvta_generic_to_shared(vs.desc);
            vs.blkbit_sh = (uint32_t)__cvta_generic_to_shared(vs.blkbit);
        }
    }

    // EncoderBase::new (encoder_base.rs:29-41, lms.rs:19-32) or the state kept by a streaming handle
    for (uint32_t c = tid; c < C; c += T) {
        if (state) {
            const int32_t *sp = state + ((uint64_t)sidx * C + c) * kEncStateWords;
            for (int i = 0; i < 4; i++) {
                st_h[c * 4 + i] = sp[i];
                st_w[c * 4 + i] = sp[4 + i];
            }
            st_prev[c] = sp[8];
        } else {
            for (int i = 0; i < 4; i++) st_h[c * 4 + i] = 0;
            st_w[c * 4 + 0] = 0;
            st_w[c * 4 + 1] = 0;
            st_w[c * 4 + 2] = -(1 << 13);
            st_w[c * 4 + 3] = 1 << 14;
            st_prev[c] = 0;
        }
    }
    __syncthreads();

    // the host picks FB > 0 for CBR and FB = 0 for VBR (launch_encode_generic): only the generic kernel carries both branches
    const bool vbr = FB > 0 ? false : (FB == 0 ? true : p.vbr != 0);
    const uint32_t n_chunks = div_ceil_u32(st.n_frames, N);
    uint64_t written = p.raw_chunk_mode ? 0 : kFileHeaderBytes;
    uint32_t first_chunk_bytes = 0;

    for (uint32_t k = 0; k < n_chunks; k++) {
        uint32_t frames = st.n_frames - k * N;
        if (frames > N) frames = N;
        const uint32_t nblk = div_ceil_u32(frames, F), items = nblk * C;
        const int16_t *x0 = pcm + st.pcm_off + (uint64_t)k * N * C;

        for (uint32_t i = tid; i < buf_words; i += T) chunk_buf[i] = 0;
        for (uint32_t i = tid; i < 4 * C; i += T) {  // file.rs:146-149: the chunk header carries the LMS *before* the chunk
            sv_w[i] = st_w[i];
            sv_h[i] = st_h[i];
        }
        __syncthreads();

        const uint32_t sf_sec_bit = (4u + 16u * C) * 8u;
        const uint32_t vbr_sec_bit = sf_sec_bit + div_ceil_u32(items * s, 8u) * 8u;
        const uint32_t res_sec_bit = vbr_sec_bit + (p.vbr ? div_ceil_u32(items * 2u, 8u) * 8u : 0u);

        if (tid == 0) {  // chunk.rs:215-226
            put_byte(chunk_sh, 0, p.vbr ? 2u : 1u);
            put_byte(chunk_sh, 1, (s << 4) | p.hdr_bits);
            put_byte(chunk_sh, 2, F);
            put_byte(chunk_sh, 3, 0x5Au);
        }
        for (uint32_t i = tid; i < 4 * C; i += T) {  // lms.rs:64-78: low 16 bits, history then weights, LE
            const uint32_t c = i >> 2, t = i & 3u;
            const uint32_t hv = (uint32_t)sv_h[i], wv = (uint32_t)sv_w[i];
            const uint32_t base_byte = 4u + 16u * c;
            put_byte(chunk_sh, base_byte + 2u * t, hv);
            put_byte(chunk_sh, base_byte + 2u * t + 1u, hv >> 8);
            put_byte(chunk_sh, base_byte + 8u + 2u * t, wv);
            put_byte(chunk_sh, base_byte + 8u + 2u * t + 1u, wv >> 8);
        }

        if (!vbr) {
            if (FB >= 0) search_pass_fast<FB, (S > 0 ? S : 4)>(0, p.hdr_bits, p, x0, frames, tab, st_w, st_h, st_prev, codes, chunk_sh, sf_sec_bit, res_sec_bit, vs, fl, xbuf);
            else search_pass(0, p.hdr_bits, p, x0, frames, tab, st_w, st_h, st_prev, codes, chunk_sh, sf_sec_bit, res_sec_bit, vs);
            if (tid == 0) sh_res_bits = frames * C * p.hdr_bits;
        } else {
            // ---- analysis at base+1 bits (encoder_vbr.rs:139-171); restores lms only (trap T2)
            if (FB >= 0) search_pass_fast<FB, (S > 0 ? S : 4)>(1, p.base + 1u, p, x0, frames, tab, st_w, st_h, st_prev, codes, chunk_sh, sf_sec_bit, res_sec_bit, vs, fl, xbuf);
            else search_pass(1, p.base + 1u, p, x0, frames, tab, st_w, st_h, st_prev, codes, chunk_sh, sf_sec_bit, res_sec_bit, vs);
            __syncthreads();
            for (uint32_t i = tid; i < 4 * C; i += T) {
                st_w[i] = sv_w[i];
                st_h[i] = sv_h[i];
            }
            // ---- choose_residual_len_from_errors (encoder_vbr.rs:98-137)
            const uint32_t sortable = (frames * C) / F;  // trap T14: interleaved sample count / F
            const bool full = frames == N;
            const uint32_t m1 = full ? p.full_counts[0] : st.last_counts[0];
            const uint32_t p1 = full ? p.full_counts[1] : st.last_counts[1];
            const uint32_t p2 = full ? p.full_counts[2] : st.last_counts[2];
            const uint32_t np2 = next_pow2(sortable);
            for (uint32_t i = tid; i < np2; i += T) {
                if (i >= sortable) vs.keys[i] = ~0ull;
                vs.idx[i] = i < sortable ? i : 0xffffffffu;
            }
            for (uint32_t i = tid; i < items; i += T) vs.sizes[i] = (uint8_t)p.base;
            __syncthreads();
            // register sort by the first warp when the items fit (<= 512: stereo chunks), else / on overflow the CTA-wide one
            if (tid < 32u) {
                const bool ok = np2 <= 512u && warp_sort_512(vs.keys, vs.idx, sortable, np2);
                if (tid == 0) sh_sorted = ok ? 1u : 0u;
            }
            __syncthreads();
            if (!sh_sorted) bitonic_sort(vs.keys, vs.idx, np2);
            for (uint32_t pos = tid; pos < sortable; pos += T) {
                uint32_t size = p.base;
                if (pos < m1) size = p.base - 1u;
                if (pos >= sortable - p2 - p1) size = p.base + 1u;
                if (pos >= sortable - p2) size = p.base + 2u;
                if (size < 1u || size > 8u) enc_report(err, kDevDomain);  // SeaResidualSize::from panics (trap T20)
                vs.sizes[vs.idx[pos]] = (uint8_t)size;
                const bool boundary = pos > 0 && (pos == m1 || pos == sortable - p2 - p1 || pos == sortable - p2);
                if (boundary && vs.keys[pos - 1] == vs.keys[pos]) {
                    uint32_t before = p.base;  // size of position pos-1
                    if (pos - 1 < m1) before = p.base - 1u;
                    if (pos - 1 >= sortable - p2 - p1) before = p.base + 1u;
                    if (pos - 1 >= sortable - p2) before = p.base + 2u;
                    if (before != size) {  // trap T13: tie across a bucket boundary (ties[0] = batch total, ties[1 + i] = stream i)
                        atomicAdd(ties, 1ull);
                        atomicAdd(ties + 1u + sidx, 1ull);
                    }
                }
            }
            __syncthreads();
            if (tid < 32u) {  // bit offset of every block inside the residual section: a run of blocks per lane, then a warp scan
                const uint32_t per = (nblk + 31u) / 32u, b0 = tid * per, b1 = b0 + per < nblk ? b0 + per : nblk;
                uint32_t mine = 0;
                for (uint32_t blk = b0; blk < b1; blk++) {
                    uint32_t rb = 0;
                    for (uint32_t c = 0; c < C; c++) rb += vs.sizes[blk * C + c];
                    uint32_t nf = frames - blk * F;
                    if (nf > F) nf = F;
                    vs.rowbits[blk] = rb;
                    mine += nf * rb;
                }
                uint32_t incl = mine;
#pragma unroll
                for (uint32_t o = 1; o < 32u; o <<= 1) {
                    const uint32_t up = __shfl_up_sync(0xffffffffu, incl, o);
                    if (tid >= o) incl += up;
                }
                uint32_t acc = incl - mine;
                for (uint32_t blk = b0; blk < b1; blk++) {
                    uint32_t nf = frames - blk * F;
                    if (nf > F) nf = F;
                    vs.blkbit[blk] = acc;
                    acc += nf * vs.rowbits[blk];
                }
                if (tid == 31u) sh_res_bits = incl;
            }
            for (uint32_t i = tid; i < items; i += T) {  // chunk.rs:245-252 (release build masks to 2 bits)
                const uint32_t sz = vs.sizes[i], blk_i = i / C, c_i = i - blk_i * C;
                put_bits(chunk_sh, vbr_sec_bit + 2u * i, 2u, (sz - p.hdr_bits + 1u) & 3u);
                uint32_t prefix = 0, rb = 0;
                for (uint32_t cc = 0; cc < C; cc++) {
                    const uint32_t z = vs.sizes[blk_i * C + cc];
                    prefix += cc < c_i ? z : 0u;
                    rb += z;
                }
                vs.desc[i] = sz | (prefix << 4) | (rb << 12);
            }
            __syncthreads();
            // ---- second pass with the chosen sizes (encoder_vbr.rs:193-207)
            if (FB >= 0) search_pass_fast<FB, (S > 0 ? S : 4)>(2, 0, p, x0, frames, tab, st_w, st_h, st_prev, codes, chunk_sh, sf_sec_bit, res_sec_bit, vs, fl, xbuf);
            else search_pass(2, 0, p, x0, frames, tab, st_w, st_h, st_prev, codes, chunk_sh, sf_sec_bit, res_sec_bit, vs);
        }
        __syncthreads();

        const uint32_t chunk_bytes = res_sec_bit / 8u + (sh_res_bits + 7u) / 8u;
        if (chunk_bytes > p.max_chunk_bytes) enc_report(err, kDevDomain);
        // raw chunk mode (make_chunk seam): no file header; consecutive chunks of one call follow each other
        uint8_t *dst = out + st.out_off + (p.raw_chunk_mode ? 0 : (uint64_t)kFileHeaderBytes) + (uint64_t)k * p.full_chunk_bytes;
        for (uint32_t i = tid; i < chunk_bytes && i < p.max_chunk_bytes; i += T)
            dst[i] = (uint8_t)(chunk_buf[i >> 2] >> (24u - 8u * (i & 3u)));
        if (k == 0) first_chunk_bytes = chunk_bytes;
        written += chunk_bytes;
        __syncthreads();
    }

    if (tid == 0) {
        if (!p.raw_chunk_mode) {  // file.rs:78-93; chunk_size = first chunk (file.rs:166-168); total_frames as u32
            uint8_t *hd = out + st.out_off;
            hd[0] = 's'; hd[1] = 'e'; hd[2] = 'a'; hd[3] = 'c';
            hd[4] = 1;
            hd[5] = (uint8_t)C;
            hd[6] = (uint8_t)first_chunk_bytes;
            hd[7] = (uint8_t)(first_chunk_bytes >> 8);
            hd[8] = (uint8_t)N;
            hd[9] = (uint8_t)(N >> 8);
            for (int i = 0; i < 4; i++) hd[10 + i] = (uint8_t)(p.sample_rate >> (8 * i));
            for (int i = 0; i < 4; i++) hd[14 + i] = (uint8_t)(st.n_frames >> (8 * i));
            for (int i = 0; i < 4; i++) hd[18 + i] = 0;
        }
        out_lens[sidx] = written;
        chunk0[sidx] = first_chunk_bytes;
    }
    if (state) {
        for (uint32_t c = tid; c < C; c += T) {
            int32_t *sp = state + ((uint64_t)sidx * C + c) * kEncStateWords;
            for (int i = 0; i < 4; i++) {
                sp[i] = st_h[c * 4 + i];
                sp[4 + i] = st_w[c * 4 + i];
            }
            sp[8] = st_prev[c];
        }
    }
}

template <int FB, int S>
static cudaError_t launch_encode_t(const int16_t *d_pcm, uint8_t *d_out, const EncStream *d_streams, const EncParams &p, DevTables tabs,
                                   int32_t *d_state, uint64_t *d_out_lens, uint32_t *d_chunk0, unsigned long long *d_ties, EncWorkspace ws,
                                   int *d_err, cudaStream_t stream, uint32_t T, size_t smem)
{
    cudaError_t e = cudaFuncSetAttribute(encode_kernel<FB, S>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    // one CTA per stream: residency is bounded by shared memory, so ask for the largest carve-out (the driver's default picked
    // 164 KB of the 228 KB and left a second wave at the high bitrates)
    e = cudaFuncSetAttribute(encode_kernel<FB, S>, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
    if (e != cudaSuccess) return e;
    encode_kernel<FB, S><<<p.n_streams, T, smem, stream>>>(d_pcm, d_out, d_streams, p, tabs, d_state, d_out_lens, d_chunk0, d_ties, ws, d_err);
    return cudaGetLastError();
}

cudaError_t launch_encode_generic(const int16_t *d_pcm, uint8_t *d_out, const EncStream *d_streams, const EncParams &p,
                                  DevTables tabs, int32_t *d_state, uint64_t *d_out_lens, uint32_t *d_chunk0,
                                  unsigned long long *d_ties, EncWorkspace ws, int *d_err, cudaStream_t stream)
{
    if (p.n_streams == 0) return cudaSuccess;
    const uint32_t nsf = 1u << p.s, lpc = nsf < 32u ? nsf : 32u, cpw = 32u / lpc;
    // fast pass: scale_factor_bits 3, 4 or 5 (8 / 16 / 32 lanes per chain group), the default 20 frames per block, every group
    // of 32 / 2^s channels has its own warp
    const bool fast = p.s >= 3u && p.s <= 5u && p.F == 20u && p.channels <= 16u;
    // BASELINE's north star maps "one warp per (stream, channel)".  Built and tested (EncParams::split, search_pass_fast), measured,
    // and NOT selected by default: the two channels of a pair already run concurrently in the two half-warps of one warp and a
    // warp's step costs the same issue slots with 16 or 32 active lanes, so at 128 streams both mappings take 92.1 / 93.1 ms and
    // at 512 the split one is 25 % slower (profiles/r02_split_probe.txt).  SEA_B200_ENC_SPLIT=1 selects it (tests, tuning).
    bool split = false;
    if (const char *env = getenv("SEA_B200_ENC_SPLIT")) split = fast && p.channels >= 2u && env[0] == '1';
    uint32_t warps = split ? p.channels : (p.channels + cpw - 1u) / cpw;
    if (warps > 8u) warps = 8u;
    const uint32_t T = warps * 32u;
    size_t smem = ((size_t)(p.max_chunk_bytes + 3u) / 4u + 2u) * 4u + (size_t)p.channels * 17u * 4u + ((2u * (size_t)p.F * T + 15u) & ~(size_t)15u) + 16u;
    int lut_mode = kEncLut32;
    if (fast) {
        smem += ((size_t)warps * cpw * p.F * 2u + 15u) & ~(size_t)15u;
        {   // One CTA per stream, all of them resident at once if they fit: with k = ceil(streams / 148) CTAs per SM a CTA may use
            // 227 KB / k less the 1 KB the hardware reserves per CTA (31 KB at the benchmark's 1024 streams); with more streams
            // than that would leave 28 KB for, keep the CTA at or under 28 KB (8 per SM, several waves).
            const int fb = p.vbr ? 0 : (int)p.hdr_bits;
            const size_t e = enc_lut_entries(fb, p.base), other = smem + 256u + (p.vbr ? (size_t)enc_vbr_scratch_bytes(p) + 16u : 0u);
            const size_t per_sm = (p.n_streams + 147u) / 148u;
            size_t budget = 227u * 1024u / per_sm;
            budget = budget > 1280u + 28u * 1024u ? budget - 1280u : 28u * 1024u;
            if (!p.vbr) lut_mode = enc_lut_mode_cbr(fb, (int)p.s);
            else if (other + e * 128u <= budget) lut_mode = kEncLut32;
            else if (p.s == 4u && other + e * 64u <= budget) lut_mode = kEncLut16;
            else lut_mode = kEncLutGlobal;
            // SEA_B200_ENC_LUT=32|16|global pins the VBR layout whatever the batch size (tests, tuning); a layout that does not
            // apply (16 needs scale_factor_bits 4) or would take the CTA past 200 KB leaves the choice above
            const char *pin = p.vbr ? getenv("SEA_B200_ENC_LUT") : nullptr;
            if (pin) {
                const int want = !strcmp(pin, "32") ? kEncLut32 : !strcmp(pin, "16") ? kEncLut16 : !strcmp(pin, "global") ? kEncLutGlobal : -1;
                const size_t need = want == kEncLut32 ? e * 128u : (want == kEncLut16 ? e * 64u : 0u);
                if (want >= 0 && (want != kEncLut16 || p.s == 4u) && other + need <= 200u * 1024u) lut_mode = want;
            }
            if (lut_mode != kEncLutGlobal) smem += e * (lut_mode == kEncLut32 ? 128u : 64u);
        }
        smem += 4u * nsf * 4u;  // reciprocals [slot][2^s]
    }
    EncParams pp = p;
    pp.vbr_smem_off = 0;
    pp.lut_mode = (uint32_t)lut_mode;
    pp.split = split ? 1u : 0u;
    if (p.vbr) {  // keep the per-chunk VBR scratch in shared memory when it is small (stereo: 8.7 KB)
        const uint64_t sc = enc_vbr_scratch_bytes(p);
        if (sc <= 40u * 1024u && smem + sc + 16u <= 200u * 1024u) {
            smem = (smem + 15u) & ~(size_t)15u;
            pp.vbr_smem_off = (uint32_t)smem;
            smem += sc;
        }
    }
    if (smem > 200u * 1024u) return cudaErrorInvalidConfiguration;
#define SEA_ENC(FBV, SV) return launch_encode_t<FBV, SV>(d_pcm, d_out, d_streams, pp, tabs, d_state, d_out_lens, d_chunk0, d_ties, ws, d_err, stream, T, smem)
#define SEA_ENC_S(SV)                      \
    {                                      \
        if (p.vbr) SEA_ENC(0, SV);         \
        switch (p.hdr_bits) {              \
            case 1: SEA_ENC(1, SV);        \
            case 2: SEA_ENC(2, SV);        \
            case 3: SEA_ENC(3, SV);        \
            case 4: SEA_ENC(4, SV);        \
            case 5: SEA_ENC(5, SV);        \
            case 6: SEA_ENC(6, SV);        \
            case 7: SEA_ENC(7, SV);        \
            default: SEA_ENC(8, SV);       \
        }                                  \
    }
    if (!fast) SEA_ENC(-1, 0);
    switch (p.s) {
        case 3: SEA_ENC_S(3)
        case 5: SEA_ENC_S(5)
        default: SEA_ENC_S(4)
    }
#undef SEA_ENC_S
#undef SEA_ENC
}

}  // namespace sea
