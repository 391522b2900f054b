// decode_kernels.cu -- SEA chunk-parallel decode for sm_100a.
//
// Replaces, per chunk: SeaChunk::from_slice (chunk.rs:69-213), BitUnpacker (bits.rs:34-78) and
// Decoder::decode_cbr / decode_vbr (codec/decoder.rs:20-86).  Every chunk header carries its own LMS state
// (chunk.rs:95-103), so each (stream, chunk, channel) chain is independent: one thread per chain.
//
//   decode_generic_kernel  any per-chunk parameters, any channel count, any alignment; reads the bit stream
//                          straight from global memory.  Correctness fallback.
//   decode_staged_kernel   uniform batches with 1 or 2 channels: a warp owns 32/C consecutive chunks, stages
//                          their packed residuals through shared memory with coalesced 128-bit loads, decodes
//                          one chain per lane and stages the PCM back out for coalesced interleaved stores.
#include "decode_chain.cuh"

namespace sea {

using namespace dev;


// ------------------------------------------------------------------------------------------------ generic

__global__ void __launch_bounds__(128) decode_generic_kernel(const uint8_t *__restrict__ sea, int16_t *__restrict__ pcm,
                                                            const DecStream *__restrict__ streams, uint32_t n_streams,
                                                            uint64_t total_chains, DevTables tabs, int *err)
{
    uint64_t gid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= total_chains) return;
    const DecStream st = streams[find_stream(streams, n_streams, gid)];
    const uint32_t C = st.channels;
    const uint32_t local = (uint32_t)(gid - st.chain_begin);
    const uint32_t k = local / C, c = local - k * C;
    const uint64_t ck_off = (uint64_t)k * st.chunk_size;
    const uint8_t *ck = sea + st.data_off + ck_off;
    const uint64_t rest = st.data_len - ck_off;
    const uint32_t take = rest < st.chunk_size ? (uint32_t)rest : st.chunk_size;
    const uint32_t N = st.frames_per_chunk;
    uint32_t frames = st.total_frames - k * N;
    if (frames > N) frames = N;

    auto fail = [&](int code) { report(err, code); };
    ChunkGeom g;
    if (!chunk_head(ck, take, C, g, fail)) return;
    int32_t w[4], h[4];
    {
        const uint8_t *l = ck + 4u + 16u * c;  // lms.rs:80-94
#pragma unroll
        for (int i = 0; i < 4; i++) {
            h[i] = (int16_t)(l[2 * i] | (l[2 * i + 1] << 8));
            w[i] = (int16_t)(l[8 + 2 * i] | (l[8 + 2 * i + 1] << 8));
        }
    }
    int32_t sg[4];
    lms_signs(sg, h);
    if (!chunk_sections(take, C, frames, g, fail)) return;

    int16_t *out = pcm + st.pcm_off + (uint64_t)k * N * C + c;
    chain_blocks<true>(ck, g, C, c, frames, w, h, sg, tabs.by_s[g.s], [&](int32_t y) {
        *out = (int16_t)y;
        out += C;
    }, fail);
}

cudaError_t launch_decode_generic(const uint8_t *d_sea, int16_t *d_pcm, const DecStream *d_streams, uint32_t n_streams,
                                  uint64_t total_chains, DevTables tabs, int *d_err, cudaStream_t stream)
{
    if (total_chains == 0) return cudaSuccess;
    const uint32_t threads = 128;
    const uint64_t blocks = (total_chains + threads - 1) / threads;
    decode_generic_kernel<<<(unsigned)blocks, threads, 0, stream>>>(d_sea, d_pcm, d_streams, n_streams, total_chains, tabs, d_err);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------ staged

constexpr int kWarpsPerCta = 8;

template <int C, int BT>
struct StagedCfg {
    static constexpr int kRows = 32 / C;                       // chunks per warp
    static constexpr int kTileFrames = 32;                     // frames per round
    static constexpr int kBmax = BT > 0 ? BT : 8;
    static constexpr int kInBytes = ((kTileFrames * C * kBmax + 7) / 8 + 16 + 8 + 15) / 16 * 16;  // + align slack + overread
    static constexpr int kInVecs = kInBytes / 16;
    static constexpr int kOutBytes = kTileFrames * C * 2;      // 64*C, multiple of 16
    static constexpr int kOutPitch = kOutBytes + 16;
    static constexpr int kOutVecs = kOutBytes / 16;
    static constexpr int kWarpBytes = kRows * (kInBytes + kOutPitch) + kRows * 24;
};

// Shared-memory layout per warp: in rows | out rows | row_out ptr (8 B) | row_in offset (8 B) | row_a (8 B)
template <int C, int BT>
__global__ void __launch_bounds__(kWarpsPerCta * 32)
decode_staged_kernel(const uint8_t *__restrict__ sea, uint64_t sea_len, int16_t *__restrict__ pcm,
                     const DecStream *__restrict__ streams, DecFastParams p, const int32_t *__restrict__ tab, int *err)
{
    using Cfg = StagedCfg<C, BT>;
    extern __shared__ __align__(16) uint8_t smem[];
    const uint32_t s = p.s;
    // dequant rows of this scale_factor_bits: all 8 sizes when runtime-sized, else only size BT
    const uint32_t lut_first = BT > 0 ? tab_dqt_off(s, BT) : tab_dqt_off(s, 1);
    const uint32_t lut_words = BT > 0 ? (1u << (s + BT)) : (510u << s);
    int32_t *lut = reinterpret_cast<int32_t *>(smem);
    for (uint32_t i = threadIdx.x; i < lut_words; i += blockDim.x) lut[i] = tab[lut_first + i];
    __syncthreads();

    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    uint8_t *wbase = smem + ((lut_words * 4u + 15u) & ~15u) + warp * Cfg::kWarpBytes;
    uint8_t *in_rows = wbase;
    uint8_t *out_rows = wbase + Cfg::kRows * Cfg::kInBytes;
    uint64_t *row_out = reinterpret_cast<uint64_t *>(out_rows + Cfg::kRows * Cfg::kOutPitch);
    uint64_t *row_in = row_out + Cfg::kRows;
    uint64_t *row_a = row_in + Cfg::kRows;

    const uint32_t j = lane / C, c = lane % C;
    const bool lane_ok = j < (uint32_t)Cfg::kRows;  // channel counts that do not divide 32 leave the last lanes without a chunk
    const uint64_t g = ((uint64_t)blockIdx.x * kWarpsPerCta + warp) * Cfg::kRows + j;  // global chunk index
    uint32_t frames = 0, F = p.F, b = p.b;
    uint64_t res_off = 0, sf_off = 0, vbr_off = 0, res_bits_avail = 0;
    int32_t w[4] = {0, 0, 0, 0}, h[4] = {0, 0, 0, 0};
    int16_t *out = pcm;
    bool vbr = false;
    if (lane_ok && g < p.total_chunks) {
        const DecStream st = streams[find_stream(streams, p.n_streams, g * C)];
        const uint32_t k = (uint32_t)(g - st.chain_begin / C);
        const uint64_t ck_rel = (uint64_t)k * p.chunk_size;
        const uint64_t ck_off = st.data_off + ck_rel;
        const uint64_t rest = st.data_len - ck_rel;
        const uint32_t take = rest < p.chunk_size ? (uint32_t)rest : p.chunk_size;
        frames = st.total_frames - k * p.N;
        if (frames > p.N) frames = p.N;
        const uint8_t *ck = sea + ck_off;
        bool ok = take >= 4u + 16u * C;
        if (ok) {
            const uint32_t word = (uint32_t)ck[0] | ((uint32_t)ck[1] << 8) | ((uint32_t)ck[2] << 16) | ((uint32_t)ck[3] << 24);
            if (BT > 0) ok = word == p.hdr_word;
            else ok = (word | 3u) == (p.hdr_word | 3u) && (ck[0] == 1u || ck[0] == 2u);  // type may vary per chunk
            vbr = ck[0] == 2u;
        }
        const uint32_t items = div_ceil_u32(frames, F) * C;
        sf_off = ck_off + 4u + 16u * C;
        vbr_off = sf_off + div_ceil_u32(items * s, 8u);
        res_off = vbr_off + (vbr ? div_ceil_u32(items * 2u, 8u) : 0u);
        if (ok && res_off - ck_off > take) ok = false;
        if (ok) {
            res_bits_avail = (uint64_t)(take - (uint32_t)(res_off - ck_off)) * 8u;
            if (!vbr && (uint64_t)frames * C * b > res_bits_avail) ok = false;
        }
        if (!ok) {
            report(err, kDevFallback);  // let the generic kernel classify the problem
            frames = 0;
        } else {
            const uint8_t *l = ck + 4u + 16u * c;
#pragma unroll
            for (int i = 0; i < 4; i++) {
                h[i] = (int16_t)(l[2 * i] | (l[2 * i + 1] << 8));
                w[i] = (int16_t)(l[8 + 2 * i] | (l[8 + 2 * i + 1] << 8));
            }
            out = pcm + st.pcm_off + (uint64_t)k * p.N * C;
        }
    }
    int32_t sg[4];
    lms_signs(sg, h);
    if (c == 0 && lane_ok) {
        row_out[j] = reinterpret_cast<uint64_t>(out);
        row_in[j] = res_off;
    }
    // all lanes of a row share frames/res_off; rounds are warp-uniform
    uint32_t max_frames = frames;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) max_frames = max(max_frames, __shfl_xor_sync(0xffffffffu, max_frames, o));
    const uint32_t n_rounds = (max_frames + Cfg::kTileFrames - 1) / Cfg::kTileFrames;

    uint64_t rowpos = 0;            // bit offset of the current frame inside the residual section
    uint32_t blk = 0, blk_left = 0; // current block index (next to load) and frames left in the loaded block
    uint32_t size = b, rowbits = C * b, prefix = c * b;
    const int32_t *lrow = lut;
    uint32_t done = 0;
    uint8_t *my_in = in_rows + j * Cfg::kInBytes;
    int16_t *my_out = reinterpret_cast<int16_t *>(out_rows + j * Cfg::kOutPitch) + c;

    for (uint32_t r = 0; r < n_rounds; r++) {
        // ---- stage the next slice of every row's packed residuals (coalesced 128-bit loads, byte-swapped to
        //      big-endian words so that MSB-first fields become plain shifts)
        const uint64_t a_mine = (res_off + (rowpos >> 3)) & ~(uint64_t)15;
        if (c == 0 && lane_ok) row_a[j] = a_mine;
        __syncwarp();
#pragma unroll
        for (int i = 0; i < (Cfg::kRows * Cfg::kInVecs + 31) / 32; i++) {
            const int v = lane + 32 * i;
            if (v < Cfg::kRows * Cfg::kInVecs) {
                const int row = v / Cfg::kInVecs, col = v % Cfg::kInVecs;
                const uint64_t off = row_a[row] + (uint64_t)col * 16u;
                uint4 q = make_uint4(0, 0, 0, 0);
                if (off + 16u <= sea_len) {
                    q = __ldg(reinterpret_cast<const uint4 *>(sea + off));
                } else if (off < sea_len) {
                    uint8_t tmp[16];
#pragma unroll
                    for (int t = 0; t < 16; t++) tmp[t] = off + t < sea_len ? sea[off + t] : (uint8_t)0;
                    q = *reinterpret_cast<uint4 *>(tmp);
                }
                q.x = __byte_perm(q.x, 0, 0x0123);
                q.y = __byte_perm(q.y, 0, 0x0123);
                q.z = __byte_perm(q.z, 0, 0x0123);
                q.w = __byte_perm(q.w, 0, 0x0123);
                *reinterpret_cast<uint4 *>(in_rows + row * Cfg::kInBytes + col * 16) = q;
            }
        }
        __syncwarp();

        // ---- decode up to kTileFrames frames of my chain
        uint32_t tile = frames - done;
        if (tile > (uint32_t)Cfg::kTileFrames) tile = Cfg::kTileFrames;
        const uint32_t *words = reinterpret_cast<const uint32_t *>(my_in);
        const uint64_t bit_base = (res_off - a_mine) * 8u;  // bits between the row buffer start and the section start
        uint32_t f = 0;
        while (f < tile) {
            if (blk_left == 0) {
                const uint32_t sf = get_bits_gmem(sea + sf_off, (uint64_t)(blk * C + c) * s, s);
                if (BT == 0) {
                    if (vbr) {
                        rowbits = 0;
                        prefix = 0;
                        bool bad = false;
#pragma unroll
                        for (int cc = 0; cc < C; cc++) {
                            const uint32_t sz = get_bits_gmem(sea + vbr_off, (uint64_t)(blk * C + cc) * 2u, 2u) + b - 1u;
                            bad |= sz < 1u || sz > 8u;
                            if (cc < (int)c) prefix += sz;
                            if (cc == (int)c) size = sz;
                            rowbits += sz;
                        }
                        if (bad) {
                            report(err, kDevFallback);
                            size = 1;
                            rowbits = C;
                            prefix = c;
                        }
                    }
                    lrow = lut + (tab_dqt_off(s, size) - tab_dqt_off(s, 1)) + (sf << size);
                } else {
                    lrow = lut + (sf << BT);
                }
                blk_left = frames - blk * F;
                if (blk_left > F) blk_left = F;
                if (rowpos + (uint64_t)blk_left * rowbits > res_bits_avail) {  // truncated VBR chunk (slice OOB in the reference)
                    report(err, kDevFallback);
                    frames = done + f;
                    tile = f;
                    break;
                }
                blk++;
            }
            uint32_t n = tile - f;
            if (n > blk_left) n = blk_left;
            uint32_t rb = (uint32_t)(bit_base + rowpos) + prefix;  // bit offset of my field inside the row buffer
            const uint32_t shr = 32u - (BT > 0 ? (uint32_t)BT : size);
            for (uint32_t i = 0; i < n; i++) {
                const uint32_t wi = rb >> 5;
                const uint32_t code = __funnelshift_l(words[wi + 1], words[wi], rb) >> shr;
                rb += rowbits;
                const int32_t d = lrow[code];
                const int32_t y = clamp_i16((int32_t)((uint32_t)lms_predict(w, h) + (uint32_t)d));
                my_out[(f + i) * C] = (int16_t)y;
                lms_update_sg(w, h, sg, y, d);
            }
            rowpos += (uint64_t)n * rowbits;
            blk_left -= n;
            f += n;
        }
        done += tile;
        __syncwarp();

        // ---- coalesced copy-out: each row's tile is one contiguous run of interleaved i16
        {
            const uint32_t tile_all = __shfl_sync(0xffffffffu, tile, 0);  // fast path when every row is full
            uint32_t uniform = __all_sync(0xffffffffu, tile == tile_all || !lane_ok) && tile_all == (uint32_t)Cfg::kTileFrames;
            const uint64_t round_off = (uint64_t)r * Cfg::kTileFrames * C;  // samples
            if (uniform) {
#pragma unroll
                for (int i = 0; i < (Cfg::kRows * Cfg::kOutVecs + 31) / 32; i++) {
                    const int v = lane + 32 * i;
                    if (v >= Cfg::kRows * Cfg::kOutVecs) break;  // row counts that do not tile the warp (3, 5, 7 channels)
                    const int row = v / Cfg::kOutVecs, col = v % Cfg::kOutVecs;
                    int16_t *dst = reinterpret_cast<int16_t *>(row_out[row]) + round_off;
                    const uint4 q = *reinterpret_cast<const uint4 *>(out_rows + row * Cfg::kOutPitch + col * 16);
                    if ((reinterpret_cast<uint64_t>(dst) & 15u) == 0) {
                        *reinterpret_cast<uint4 *>(reinterpret_cast<uint8_t *>(dst) + col * 16) = q;
                    } else {
                        const uint32_t qs[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
                        for (int t = 0; t < 4; t++) {
                            dst[col * 8 + 2 * t] = (int16_t)(qs[t] & 0xffffu);
                            dst[col * 8 + 2 * t + 1] = (int16_t)(qs[t] >> 16);
                        }
                    }
                }
            } else {
                // ragged tail: element-wise, still coalesced along each row
                for (int row = 0; row < Cfg::kRows; row++) {
                    const uint32_t t_row = __shfl_sync(0xffffffffu, tile, row * C);
                    int16_t *dst = reinterpret_cast<int16_t *>(row_out[row]) + round_off;
                    const int16_t *src = reinterpret_cast<const int16_t *>(out_rows + row * Cfg::kOutPitch);
                    for (uint32_t e = lane; e < t_row * C; e += 32) dst[e] = src[e];
                }
            }
        }
        // the next round's __syncwarp after row_a publication orders these smem reads before the next writes
    }
}

template <int C, int BT>
static cudaError_t launch_staged(const uint8_t *d_sea, uint64_t sea_len, int16_t *d_pcm, const DecStream *d_streams,
                                 const DecFastParams &p, const int32_t *tab, int *d_err, cudaStream_t stream)
{
    using Cfg = StagedCfg<C, BT>;
    const uint32_t lut_words = BT > 0 ? (1u << (p.s + BT)) : (510u << p.s);
    const size_t smem = ((lut_words * 4u + 15u) & ~15u) + (size_t)kWarpsPerCta * Cfg::kWarpBytes;
    cudaError_t e = cudaFuncSetAttribute(decode_staged_kernel<C, BT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    const uint64_t chunks_per_cta = (uint64_t)kWarpsPerCta * Cfg::kRows;
    const uint64_t blocks = (p.total_chunks + chunks_per_cta - 1) / chunks_per_cta;
    decode_staged_kernel<C, BT><<<(unsigned)blocks, kWarpsPerCta * 32, smem, stream>>>(d_sea, sea_len, d_pcm, d_streams, p, tab, d_err);
    return cudaGetLastError();
}

bool decode_fast_supported(const DecFastParams &p)
{
    // 1, 2 and the odd counts (VBR, partial chunks and odd block lengths of 3 / 5 / 7 channels; their full CBR chunks go to the whole-frame
    // kernel of decode_mc.cuh -- 3 is what the reference's tests use, tests/test.rs:10)
    if (p.channels != 1 && p.channels != 2 && p.channels != 3 && p.channels != 5 && p.channels != 7) return false;
    if (p.s < 1 || p.s > 5) return false;  // 510 << s words of LUT must fit shared memory next to the tiles
    if (p.b < 1 || p.b > 8 || p.F == 0) return false;
    return true;
}

cudaError_t launch_decode_fast(const uint8_t *d_sea, uint64_t sea_len, int16_t *d_pcm, const DecStream *d_streams,
                               const DecFastParams &p, DevTables tabs, int *d_err, cudaStream_t stream)
{
    if (p.total_chunks == 0) return cudaSuccess;
    const int32_t *tab = tabs.by_s[p.s];
    const bool cbr = (p.hdr_word & 0xffu) == 1u;
#define SEA_STAGED(CC, BB) return launch_staged<CC, BB>(d_sea, sea_len, d_pcm, d_streams, p, tab, d_err, stream)
#define SEA_STAGED_C(CC)            \
    {                               \
        if (!cbr) SEA_STAGED(CC, 0); \
        switch (p.b) {              \
            case 1: SEA_STAGED(CC, 1); \
            case 2: SEA_STAGED(CC, 2); \
            case 3: SEA_STAGED(CC, 3); \
            case 4: SEA_STAGED(CC, 4); \
            case 5: SEA_STAGED(CC, 5); \
            case 6: SEA_STAGED(CC, 6); \
            case 7: SEA_STAGED(CC, 7); \
            default: SEA_STAGED(CC, 8); \
        }                           \
    }
    switch (p.channels) {
        case 1: SEA_STAGED_C(1)
        case 2: SEA_STAGED_C(2)
        case 3: SEA_STAGED_C(3)
        case 5: SEA_STAGED_C(5)
        default: SEA_STAGED_C(7)
    }
#undef SEA_STAGED_C
#undef SEA_STAGED
}


}  // namespace sea
