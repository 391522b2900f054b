// decode_chain.cuh -- the per-chunk checks and the per-chain block loop of decode_generic_kernel (decode_kernels.cu), shared with
// the corpus kernels (corpus_kernels.cu) so that what a chunk must satisfy, and how a chain is decoded, is written once.
//
// Every check reports through `fail(code)` (device error codes kDev*) and makes its function return false; the callers stop there.
#pragma once
#include "sea_device.cuh"

namespace sea {
namespace dev {

// MSB-first field of n <= 8 bits at bit offset `bit` from p (bits.rs:42-46 semantics), p in global memory.
__device__ __forceinline__ uint32_t get_bits_gmem(const uint8_t *p, uint64_t bit, uint32_t n)
{
    uint64_t byte = bit >> 3;
    uint32_t sh = (uint32_t)bit & 7u;
    uint32_t v = (uint32_t)__ldg(p + byte) << 8;
    if (sh + n > 8u) v |= (uint32_t)__ldg(p + byte + 1);
    return (v >> (16u - sh - n)) & ((1u << n) - 1u);
}

// One chunk's header fields and section layout (chunk.rs:69-113).
struct ChunkGeom {
    uint32_t s, b, F;
    bool vbr;
    uint32_t nblk, sf_sec, vbr_sec, res_sec;
    uint64_t res_bits_avail;
};

// The chunk header: `take` bytes present, type, residual and scale-factor bit ranges, F.
template <class Fail>
__device__ __forceinline__ bool chunk_head(const uint8_t *ck, uint32_t take, uint32_t C, ChunkGeom &g, Fail &&fail)
{
    if (take < 4u + 16u * C) { fail(kDevDomain); return false; }  // slice index out of range in chunk.rs:81-101
    const uint32_t type = ck[0];
    g.s = ck[1] >> 4;
    g.b = ck[1] & 15u;
    g.F = ck[2];
    if (type != 1u && type != 2u) { fail(kDevInvalidFrame); return false; }  // chunk.rs:81-85
    if (g.b < 1u || g.b > 8u || g.s < 1u || g.s > 8u || g.F == 0u) { fail(kDevDomain); return false; }
    g.vbr = type == 2u;
    return true;
}

// The sections of a chunk of `frames` frames against the bytes present, and (CBR) that every residual bit is there.
template <class Fail>
__device__ __forceinline__ bool chunk_sections(uint32_t take, uint32_t C, uint32_t frames, ChunkGeom &g, Fail &&fail)
{
    g.nblk = div_ceil_u32(frames, g.F);
    const uint32_t items = g.nblk * C;
    g.sf_sec = 4u + 16u * C;
    g.vbr_sec = g.sf_sec + div_ceil_u32(items * g.s, 8u);
    g.res_sec = g.vbr_sec + (g.vbr ? div_ceil_u32(items * 2u, 8u) : 0u);
    if (g.res_sec > take) { fail(kDevDomain); return false; }
    g.res_bits_avail = (uint64_t)(take - g.res_sec) * 8u;
    if (!g.vbr && (uint64_t)frames * C * g.b > g.res_bits_avail) { fail(kDevDomain); return false; }
    return true;
}

// Chain c of a chunk: the first `frames` frames (of a chunk laid out as g says), block by block, with the VBR size codes (1..8 per
// block and channel) and the residual bits of each block checked.  kDecode: every sample y goes to sink(y) in frame order
// (decoder.rs:38-45); otherwise only the checks run.
template <bool kDecode, class Sink, class Fail>
__device__ __forceinline__ bool chain_blocks(const uint8_t *ck, const ChunkGeom &g, uint32_t C, uint32_t c, uint32_t frames, int32_t (&w)[4],
                                             int32_t (&h)[4], int32_t (&sg)[4], const int32_t *tab, Sink &&sink, Fail &&fail)
{
    const uint32_t s = g.s, b = g.b, F = g.F, nblk = div_ceil_u32(frames, F);
    uint64_t bitpos = 0;  // start of the current frame inside the residual section
    for (uint32_t blk = 0; blk < nblk; blk++) {
        uint32_t sf = 0;
        if constexpr (kDecode) sf = get_bits_gmem(ck + g.sf_sec, (uint64_t)(blk * C + c) * s, s);
        uint32_t size = b, rowbits = C * b, prefix = c * b;
        if (g.vbr) {  // chunk.rs:126-139: size = 2-bit code + residual_size - 1
            rowbits = 0;
            prefix = 0;
            for (uint32_t cc = 0; cc < C; cc++) {
                uint32_t sz = get_bits_gmem(ck + g.vbr_sec, (uint64_t)(blk * C + cc) * 2u, 2u) + b - 1u;
                if (sz < 1u || sz > 8u) { fail(kDevDomain); return false; }
                if (cc < c) prefix += sz;
                if (cc == c) size = sz;
                rowbits += sz;
            }
        }
        uint32_t nf = frames - blk * F;
        if (nf > F) nf = F;
        if (bitpos + (uint64_t)nf * rowbits > g.res_bits_avail) { fail(kDevDomain); return false; }
        if constexpr (kDecode) {
            const int32_t *row = tab + tab_dqt_off(s, size) + (sf << size);
            for (uint32_t f = 0; f < nf; f++) {
                const uint32_t code = get_bits_gmem(ck + g.res_sec, bitpos + prefix, size);
                bitpos += rowbits;
                const int32_t d = __ldg(row + code);
                const int32_t y = clamp_i16((int32_t)((uint32_t)lms_predict(w, h) + (uint32_t)d));  // decoder.rs:38-45
                sink(y);
                lms_update_sg(w, h, sg, y, d);
            }
        } else {
            bitpos += (uint64_t)nf * rowbits;
        }
    }
    return true;
}

}  // namespace dev
}  // namespace sea
