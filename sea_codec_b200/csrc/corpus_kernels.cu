// corpus_kernels.cu -- a registered corpus (sea_b200_corpus_*): the create-time validation of every chunk a window can cover, and the
// fused window kernels of sea_b200_corpus_decode_windows_async, which decode the covering chunks straight into the output slots.
//
// Work unit u = (window w, covering-chunk slot j < M), numbered u = j * n_windows + w.  Slot j owns the slot frames [j*N - skip, (j+1)*N - skip) clipped to the window
// (slot 0 from frame 0, slot M-1 up to the window's end), so the units of one window write disjoint frame ranges.  A unit decodes
// chunk k0 + j from its LMS header up to the last frame it owns, stores the frames it owns, and writes zeros where the stream has
// none (past its end, or a bad stream index).  Every chunk was validated at create, so no unit meets a malformed chunk.
//
//   corpus_generic_kernel  any geometry: one thread per (unit, channel) chain, decode_generic_kernel's chain loop (decode_chain.cuh).
//   corpus_fast_kernel     uniform CBR corpora with 1 or 2 channels: a warp owns 32/C units, stages their packed residuals through
//                          shared memory with coalesced 16-byte loads (decode_staged_kernel's scheme), decodes one chain per lane
//                          and writes each 32-frame tile of a unit as a contiguous run of its slot.
#include "../../include/sea_b200.h"
#include "decode_chain.cuh"

namespace sea {

using namespace dev;

// ------------------------------------------------------------------------------------------------ validation

__device__ __forceinline__ uint32_t corpus_find_stream(const CorpusStream *streams, uint32_t n_streams, uint64_t chunk)
{
    uint32_t lo = 0, hi = n_streams;
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        if (streams[mid].chunk_begin <= chunk) lo = mid;
        else hi = mid;
    }
    return lo;
}

__global__ void __launch_bounds__(128) corpus_validate_kernel(const uint8_t *__restrict__ sea, const CorpusStream *__restrict__ streams,
                                                             uint32_t n_streams, uint64_t total, uint32_t C, uint32_t ref_word,
                                                             unsigned long long *first_bad, uint32_t *mixed)
{
    const uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= total) return;
    const CorpusStream st = streams[corpus_find_stream(streams, n_streams, g)];
    const uint64_t k = g - st.chunk_begin, rel = k * st.chunk_size;
    const uint8_t *ck = sea + st.body + rel;
    const uint64_t rest = st.len - rel;
    const uint32_t take = rest < st.chunk_size ? (uint32_t)rest : st.chunk_size;
    const uint64_t left = st.file_frames - k * st.N;
    const uint32_t frames = left < st.N ? (uint32_t)left : st.N;

    auto fail = [&](int code) { atomicMin(first_bad, (unsigned long long)((g << 2) | (uint64_t)code)); };
    ChunkGeom geo;
    if (!chunk_head(ck, take, C, geo, fail)) return;
    const uint32_t word = (uint32_t)ck[0] | ((uint32_t)ck[1] << 8) | ((uint32_t)ck[2] << 16) | ((uint32_t)ck[3] << 24);
    if (word != ref_word) atomicOr(mixed, 1u);
    if (!chunk_sections(take, C, frames, geo, fail)) return;
    int32_t w[4] = {0, 0, 0, 0}, h[4] = {0, 0, 0, 0}, sg[4] = {0, 0, 0, 0};
    chain_blocks<false>(ck, geo, C, 0, frames, w, h, sg, nullptr, [](int32_t) {}, fail);
}

cudaError_t launch_corpus_validate(const uint8_t *d_sea, const CorpusStream *d_streams, uint32_t n_streams, uint64_t total_chunks,
                                   uint32_t channels, uint32_t ref_word, unsigned long long *d_first_bad, uint32_t *d_mixed,
                                   cudaStream_t stream)
{
    if (total_chunks == 0) return cudaSuccess;
    const uint64_t blocks = (total_chunks + 127) / 128;
    debug_launch("corpus_validate: %u channels, %llu CTAs", channels, (unsigned long long)blocks);
    corpus_validate_kernel<<<(unsigned)blocks, 128, 0, stream>>>(d_sea, d_streams, n_streams, total_chunks, channels, ref_word,
                                                                 d_first_bad, d_mixed);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------ work units

struct CorpusUnit {
    uint32_t w, j;
    bool bad;           // the window's stream index is out of range
    uint32_t want;      // frames of the window the stream has (frames_out)
    uint32_t lo, hi;    // slot frames the unit owns
    uint32_t zlo;       // of them, [zlo, hi) are zeros
    uint32_t d_lo, d_hi;  // chunk frames: [0, d_hi) decoded, [d_lo, d_hi) stored at slot frames [lo, ...); d_hi == 0: no chunk
    const uint8_t *ck;  // the chunk (d_hi > 0)
    uint32_t take, nk;  // its bytes present and true frame count
};

__device__ __forceinline__ CorpusUnit corpus_unit(const CorpusLaunch &p, uint64_t u)
{
    CorpusUnit t;
    // slot-major numbering: the units of the last covering-chunk slot, empty for most windows and short otherwise, come last in
    // the grid, so that they (not full-chunk units) are what runs past the first wave
    t.j = (uint32_t)(u / p.n_windows);
    t.w = (uint32_t)(u - (uint64_t)t.j * p.n_windows);
    const uint32_t si = p.win_stream[t.w];
    t.bad = si >= p.n_streams;
    CorpusStream st = {};
    uint32_t N = p.N;  // a bad window's slot is split by the corpus's smallest chunk length
    WindowPlan pl = {0, 0, 0};
    if (!t.bad) {
        st = p.streams[si];
        N = st.N;
        pl = window_plan(st.file_frames, N, p.win_first[t.w], p.W);
    }
    const uint64_t jn = (uint64_t)t.j * N;
    t.lo = t.j == 0 ? 0u : (uint32_t)min((uint64_t)p.W, jn - pl.skip);
    t.hi = t.j == p.M - 1 ? p.W : (uint32_t)min((uint64_t)p.W, jn + N - pl.skip);
    t.want = (uint32_t)pl.want;
    const uint32_t real_hi = min(t.hi, t.want);
    t.zlo = max(t.lo, real_hi);
    t.d_lo = t.d_hi = 0;
    t.ck = nullptr;
    t.take = t.nk = 0;
    if (t.lo < real_hi) {  // chunk k0 + j exists: its first frame is at or before slot frame lo, which the stream has
        const uint64_t k = pl.k0 + t.j, rel = k * st.chunk_size;
        t.ck = p.sea + st.body + rel;
        const uint64_t rest = st.len - rel, left = st.file_frames - k * N;
        t.take = rest < st.chunk_size ? (uint32_t)rest : st.chunk_size;
        t.nk = left < N ? (uint32_t)left : N;
        t.d_lo = (uint32_t)(t.lo + pl.skip - jn);
        t.d_hi = (uint32_t)(real_hi + pl.skip - jn);
    }
    return t;
}

// frames_out and the status word: once per window, by its unit 0
__device__ __forceinline__ void corpus_window_once(const CorpusLaunch &p, const CorpusUnit &t)
{
    if (t.j != 0) return;
    if (p.frames_out) p.frames_out[t.w] = t.want;
    if (t.bad) atomicCAS(reinterpret_cast<int *>(p.status), 0, SEA_B200_ERR_INVALID_PARAMETERS);
}

// ------------------------------------------------------------------------------------------------ generic route

__global__ void __launch_bounds__(128) corpus_generic_kernel(CorpusLaunch p, DevTables tabs, uint64_t total_chains)
{
    const uint64_t gid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= total_chains) return;
    const uint32_t C = p.channels;
    const uint64_t u = gid / C;
    const uint32_t c = (uint32_t)(gid - u * C);
    const CorpusUnit t = corpus_unit(p, u);
    if (c == 0) corpus_window_once(p, t);
    const uint64_t slot = (uint64_t)t.w * p.W * C;
    int16_t *o16 = static_cast<int16_t *>(p.out) + slot + c;             // frame f at o16[f * C]
    float *o32 = static_cast<float *>(p.out) + slot + (uint64_t)c * p.W;  // frame f at o32[f]
    if (t.d_hi) {
        auto nofail = [](int) {};  // validated at create
        ChunkGeom g;
        chunk_head(t.ck, t.take, C, g, nofail);
        int32_t w[4], h[4];
        const uint8_t *l = t.ck + 4u + 16u * c;  // lms.rs:80-94
#pragma unroll
        for (int i = 0; i < 4; i++) {
            h[i] = (int16_t)(l[2 * i] | (l[2 * i + 1] << 8));
            w[i] = (int16_t)(l[8 + 2 * i] | (l[8 + 2 * i + 1] << 8));
        }
        int32_t sg[4];
        lms_signs(sg, h);
        chunk_sections(t.take, C, t.nk, g, nofail);
        uint32_t f = 0;
        const uint32_t shift = t.lo - t.d_lo;  // slot frame = chunk frame + shift (for stored frames)
        chain_blocks<true>(t.ck, g, C, c, t.d_hi, w, h, sg, tabs.by_s[g.s], [&](int32_t y) {
            if (f >= t.d_lo) {
                if (p.planar) o32[f + shift] = (float)y * (1.0f / 32768.0f);
                else o16[(uint64_t)(f + shift) * C] = (int16_t)y;
            }
            f++;
        }, nofail);
    }
    for (uint32_t q = t.zlo; q < t.hi; q++) {
        if (p.planar) o32[q] = 0.0f;
        else o16[(uint64_t)q * C] = 0;
    }
}

// ------------------------------------------------------------------------------------------------ fast route

constexpr int kCorpusWarps = 8;
constexpr uint32_t kCorpusF = 20;  // scale_factor_frames of the fast route

template <int C, int BT>
struct CorpusCfg {
    static constexpr int kRows = 32 / C;  // units per warp
    static constexpr int kTileFrames = 32;
    static constexpr int kInBytes = ((kTileFrames * C * BT + 7) / 8 + 16 + 8 + 15) / 16 * 16;  // + align slack + overread
    static constexpr int kInVecs = kInBytes / 16;
    static constexpr int kOutPitch = kTileFrames * C * 2 + 16;
    static constexpr int kWarpBytes = kRows * (kInBytes + kOutPitch) + kRows * 8;
    static size_t smem(uint32_t s) { return (((size_t)4 << (s + BT)) + 15u) / 16u * 16u + (size_t)kCorpusWarps * kWarpBytes; }
};

// n consecutive int16 of a slot run at dst (any 2-byte alignment) from src (shared memory; null: zeros), as aligned 4-byte words
// spread over the warp's lanes.
__device__ __forceinline__ void put_run_i16(int16_t *dst, const int16_t *src, uint32_t n, uint32_t lane)
{
    const int32_t mis = (int32_t)((reinterpret_cast<uintptr_t>(dst) >> 1) & 1u);
    for (int32_t i = (int32_t)lane; 2 * i < (int32_t)n + mis; i += 32) {
        const int32_t e = 2 * i - mis;  // first element of the aligned word
        const uint32_t v0 = e >= 0 && src ? (uint16_t)src[e] : 0u;
        const uint32_t v1 = e + 1 < (int32_t)n && src ? (uint16_t)src[e + 1] : 0u;
        if (e >= 0 && e + 1 < (int32_t)n) {
            *reinterpret_cast<uint32_t *>(dst + e) = v0 | (v1 << 16);
        } else {
            if (e >= 0) dst[e] = (int16_t)v0;
            if (e + 1 < (int32_t)n) dst[e + 1] = (int16_t)v1;
        }
    }
}

// n consecutive frames of channel row `row` (float32 planar), frame i from src[i * C] (shared memory; null: zeros)
template <int C>
__device__ __forceinline__ void put_run_f32(float *row, const int16_t *src, uint32_t n, uint32_t lane)
{
    for (uint32_t i = lane; i < n; i += 32) row[i] = src ? (float)src[i * C] * (1.0f / 32768.0f) : 0.0f;
}

// Shared-memory layout per warp: in rows | out rows (int16 tiles, interleaved) | row_a (8 B per row)
template <int C, int BT, bool kPlanar>
__global__ void __launch_bounds__(kCorpusWarps * 32) corpus_fast_kernel(CorpusLaunch p, const int32_t *__restrict__ tab, uint64_t n_units)
{
    using Cfg = CorpusCfg<C, BT>;
    extern __shared__ __align__(16) uint8_t smem[];
    const uint32_t s = p.s;
    const uint32_t lut_words = 1u << (s + BT);
    int32_t *lut = reinterpret_cast<int32_t *>(smem);
    for (uint32_t i = threadIdx.x; i < lut_words; i += blockDim.x) lut[i] = tab[tab_dqt_off(s, BT) + i];
    __syncthreads();

    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    uint8_t *wbase = smem + ((lut_words * 4u + 15u) & ~15u) + warp * Cfg::kWarpBytes;
    uint8_t *in_rows = wbase;
    uint8_t *out_rows = wbase + Cfg::kRows * Cfg::kInBytes;
    uint64_t *row_a = reinterpret_cast<uint64_t *>(out_rows + Cfg::kRows * Cfg::kOutPitch);

    const uint32_t j = lane / C, c = lane % C;  // 32 / C rows fill the warp for C = 1, 2
    const uint64_t u = ((uint64_t)blockIdx.x * kCorpusWarps + warp) * Cfg::kRows + j;
    uint32_t frames = 0, d_lo = 0, lo = 0, zlo = 0, hi = 0, wi = 0;
    uint64_t res_off = 0, sf_off = 0;
    int32_t w[4] = {0, 0, 0, 0}, h[4] = {0, 0, 0, 0};
    if (u < n_units) {
        const CorpusUnit t = corpus_unit(p, u);
        if (c == 0) corpus_window_once(p, t);
        wi = t.w;
        lo = t.lo;
        zlo = t.zlo;
        hi = t.hi;
        if (t.d_hi) {
            frames = t.d_hi;
            d_lo = t.d_lo;
            const uint32_t items = div_ceil_u32(t.nk, kCorpusF) * C;  // the layout follows the chunk's true frame count
            sf_off = (uint64_t)(t.ck - p.sea) + 4u + 16u * C;
            res_off = sf_off + div_ceil_u32(items * s, 8u);
            const uint8_t *l = t.ck + 4u + 16u * c;
#pragma unroll
            for (int i = 0; i < 4; i++) {
                h[i] = (int16_t)(l[2 * i] | (l[2 * i + 1] << 8));
                w[i] = (int16_t)(l[8 + 2 * i] | (l[8 + 2 * i + 1] << 8));
            }
        }
    }
    int32_t sg[4];
    lms_signs(sg, h);
    uint32_t max_frames = frames;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) max_frames = max(max_frames, __shfl_xor_sync(0xffffffffu, max_frames, o));
    const uint32_t n_rounds = (max_frames + Cfg::kTileFrames - 1) / Cfg::kTileFrames;
    const uint64_t slot_elems = (uint64_t)p.W * C;

    uint64_t rowpos = 0;             // bit offset of the current frame inside the residual section
    uint32_t blk = 0, blk_left = 0;  // next block to load, frames left in the loaded block
    const uint32_t rowbits = C * BT, prefix = c * BT;
    const int32_t *lrow = lut;
    uint32_t done = 0;
    uint8_t *my_in = in_rows + j * Cfg::kInBytes;
    int16_t *my_out = reinterpret_cast<int16_t *>(out_rows + j * Cfg::kOutPitch) + c;

    for (uint32_t r = 0; r < n_rounds; r++) {
        // ---- stage the next slice of every row's packed residuals (coalesced 16-byte loads, byte-swapped to big-endian words)
        const uint64_t a_mine = (res_off + (rowpos >> 3)) & ~(uint64_t)15;
        if (c == 0) row_a[j] = a_mine;
        __syncwarp();
#pragma unroll
        for (int i = 0; i < (Cfg::kRows * Cfg::kInVecs + 31) / 32; i++) {
            const int v = lane + 32 * i;
            if (v < Cfg::kRows * Cfg::kInVecs) {
                const int row = v / Cfg::kInVecs, col = v % Cfg::kInVecs;
                const uint64_t off = row_a[row] + (uint64_t)col * 16u;
                uint4 q = make_uint4(0, 0, 0, 0);
                if (off + 16u <= p.sea_len) {
                    q = __ldg(reinterpret_cast<const uint4 *>(p.sea + off));
                } else if (off < p.sea_len) {
                    uint8_t tmp[16];
#pragma unroll
                    for (int b = 0; b < 16; b++) tmp[b] = off + b < p.sea_len ? p.sea[off + b] : (uint8_t)0;
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

        // ---- decode up to kTileFrames frames of my chain into the out tile
        uint32_t tile = frames - done;
        if (tile > (uint32_t)Cfg::kTileFrames) tile = Cfg::kTileFrames;
        const uint32_t *words = reinterpret_cast<const uint32_t *>(my_in);
        const uint64_t bit_base = (res_off - a_mine) * 8u;
        uint32_t f = 0;
        while (f < tile) {
            if (blk_left == 0) {
                const uint32_t sf = get_bits_gmem(p.sea + sf_off, (uint64_t)(blk * C + c) * s, s);
                lrow = lut + (sf << BT);
                blk_left = frames - blk * kCorpusF;
                if (blk_left > kCorpusF) blk_left = kCorpusF;
                blk++;
            }
            uint32_t n = tile - f;
            if (n > blk_left) n = blk_left;
            uint32_t rb = (uint32_t)(bit_base + rowpos) + prefix;
            for (uint32_t i = 0; i < n; i++) {
                const uint32_t wj = rb >> 5;
                const uint32_t code = __funnelshift_l(words[wj + 1], words[wj], rb) >> (32u - BT);
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

        // ---- copy-out: the stored part of each row's tile is one run of its slot
        const uint32_t f0 = r * Cfg::kTileFrames;
        for (int row = 0; row < Cfg::kRows; row++) {
            const uint32_t t_row = __shfl_sync(0xffffffffu, tile, row * C);
            const uint32_t dlo_row = __shfl_sync(0xffffffffu, d_lo, row * C);
            const uint32_t a = max(f0, dlo_row), b = f0 + t_row;
            if (a >= b) continue;
            const uint32_t lo_row = __shfl_sync(0xffffffffu, lo, row * C), w_row = __shfl_sync(0xffffffffu, wi, row * C);
            const uint32_t q0 = lo_row + (a - dlo_row);  // slot frame of chunk frame a
            const int16_t *src = reinterpret_cast<const int16_t *>(out_rows + row * Cfg::kOutPitch) + (a - f0) * C;
            if constexpr (kPlanar) {
                float *slot = static_cast<float *>(p.out) + (uint64_t)w_row * slot_elems + q0;
#pragma unroll
                for (int cc = 0; cc < C; cc++) put_run_f32<C>(slot + (uint64_t)cc * p.W, src + cc, b - a, lane);
            } else {
                int16_t *slot = static_cast<int16_t *>(p.out) + (uint64_t)w_row * slot_elems + (uint64_t)q0 * C;
                put_run_i16(slot, src, (b - a) * C, lane);
            }
        }
        // the next round's __syncwarp after row_a publication orders these shared-memory reads before the next writes
    }

    // ---- zeros: slot frames [zlo, hi) of every row
    for (int row = 0; row < Cfg::kRows; row++) {
        const uint32_t z0 = __shfl_sync(0xffffffffu, zlo, row * C), z1 = __shfl_sync(0xffffffffu, hi, row * C);
        if (z0 >= z1) continue;
        const uint32_t w_row = __shfl_sync(0xffffffffu, wi, row * C);
        if constexpr (kPlanar) {
            float *slot = static_cast<float *>(p.out) + (uint64_t)w_row * slot_elems + z0;
#pragma unroll
            for (int cc = 0; cc < C; cc++) put_run_f32<C>(slot + (uint64_t)cc * p.W, nullptr, z1 - z0, lane);
        } else {
            put_run_i16(static_cast<int16_t *>(p.out) + (uint64_t)w_row * slot_elems + (uint64_t)z0 * C, nullptr, (z1 - z0) * C, lane);
        }
    }
}

bool corpus_fast_supported(uint32_t channels, uint32_t s, uint32_t b, uint32_t F, bool vbr)
{
    return !vbr && (channels == 1 || channels == 2) && F == kCorpusF && s >= 1 && s <= 5 && b >= 1 && b <= 8;
}

// The fast route's instance for (channels, b): X(C, BT) is expanded for each and the matching one runs.
#define SEA_CORPUS_FAST(channels, b, X)                                            \
    do {                                                                           \
        if ((channels) == 1) {                                                     \
            switch (b) {                                                           \
                case 1: X(1, 1); case 2: X(1, 2); case 3: X(1, 3); case 4: X(1, 4); \
                case 5: X(1, 5); case 6: X(1, 6); case 7: X(1, 7); default: X(1, 8); \
            }                                                                      \
        }                                                                          \
        switch (b) {                                                               \
            case 1: X(2, 1); case 2: X(2, 2); case 3: X(2, 3); case 4: X(2, 4);     \
            case 5: X(2, 5); case 6: X(2, 6); case 7: X(2, 7); default: X(2, 8);     \
        }                                                                          \
    } while (0)

template <int C, int BT>
static cudaError_t corpus_fast_prepare_t(uint32_t s)
{
    const int smem = (int)CorpusCfg<C, BT>::smem(s);
    cudaError_t e = cudaFuncSetAttribute(corpus_fast_kernel<C, BT, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) return e;
    return cudaFuncSetAttribute(corpus_fast_kernel<C, BT, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
}

cudaError_t corpus_fast_prepare(uint32_t channels, uint32_t s, uint32_t b)
{
#define SEA_PREP(CC, BB) return corpus_fast_prepare_t<CC, BB>(s)
    SEA_CORPUS_FAST(channels, b, SEA_PREP);
#undef SEA_PREP
}

template <int C, int BT>
static cudaError_t launch_corpus_fast(const CorpusLaunch &p, const int32_t *tab, uint64_t units, cudaStream_t stream)
{
    using Cfg = CorpusCfg<C, BT>;
    const uint64_t per_cta = (uint64_t)kCorpusWarps * Cfg::kRows, blocks = (units + per_cta - 1) / per_cta;
    const size_t smem = Cfg::smem(p.s);
    debug_launch("corpus_fast<%d,%d,%d>: %zu B smem, %llu CTAs", C, BT, (int)p.planar, smem, (unsigned long long)blocks);
    if (p.planar) corpus_fast_kernel<C, BT, true><<<(unsigned)blocks, kCorpusWarps * 32, smem, stream>>>(p, tab, units);
    else corpus_fast_kernel<C, BT, false><<<(unsigned)blocks, kCorpusWarps * 32, smem, stream>>>(p, tab, units);
    return cudaGetLastError();
}

cudaError_t launch_corpus_windows(const CorpusLaunch &p, bool fast, DevTables tabs, cudaStream_t stream)
{
    const uint64_t units = (uint64_t)p.n_windows * p.M;
    if (units == 0) return cudaSuccess;
    if (!fast) {
        const uint64_t chains = units * p.channels, blocks = (chains + 127) / 128;
        debug_launch("corpus_generic: %u channels, planar %d, %llu CTAs", p.channels, (int)p.planar, (unsigned long long)blocks);
        corpus_generic_kernel<<<(unsigned)blocks, 128, 0, stream>>>(p, tabs, chains);
        return cudaGetLastError();
    }
    const int32_t *tab = tabs.by_s[p.s];
#define SEA_LAUNCH(CC, BB) return launch_corpus_fast<CC, BB>(p, tab, units, stream)
    SEA_CORPUS_FAST(p.channels, p.b, SEA_LAUNCH);
#undef SEA_LAUNCH
}

#undef SEA_CORPUS_FAST

}  // namespace sea
