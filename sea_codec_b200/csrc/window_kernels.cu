// window_kernels.cu -- the cut of sea_b200_decode_windows_device: the chunks covering every window were decoded into a scratch
// buffer (interleaved int16, each window's covering range at its own 16-sample aligned offset); this kernel writes each window's
// output slot from there, `real` frames starting `skip` frames into the covering range, then zeros up to the slot's length.
// Every window sample passes through here once, so both instances are plain streaming kernels: 16-byte loads, and 16-byte
// stores (int16) or warp-contiguous 128-byte rows (float32 planar).
#include "sea_kernels.h"

namespace sea {

constexpr uint32_t kWinThreads = 256;
constexpr uint32_t kWinSlotSamplesPerCta = 4096;  // grid.x sizing: int16 = 256 threads x 2 vectors x 8, planar ~ one tile
constexpr uint32_t kWinTileElems = 8192;          // planar staging: 32 frames x 255 channels + 14 alignment samples fit

// ---- int16, interleaved --------------------------------------------------------------------------------------------------------

// Keeps the int16 elements [first, first + 2) of word v that lie below lim.
__device__ __forceinline__ uint32_t keep_below(uint32_t v, int first, int64_t lim)
{
    return first + 2 <= lim ? v : (first < lim ? (v & 0xffffu) : 0u);
}

// Output vector j of the body: 8 elements starting `sh` elements into the aligned source vector j; elements at or past `lim`
// (the real samples left) are zero, and a vector with none left reads nothing.
__device__ __forceinline__ uint4 body_vector(const uint4 *__restrict__ sv, uint64_t j, uint32_t sh, int64_t lim)
{
    if (lim <= 0) return make_uint4(0u, 0u, 0u, 0u);
    const uint4 a = __ldg(sv + j);
    uint4 r = a;
    if (sh) {
        const uint4 b = __ldg(sv + j + 1);
        uint32_t w[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
        // shift left by sh >> 1 words with selects on constant indices (a dynamic index would put w in local memory), then by
        // one int16 when sh is odd
        const bool s1 = sh & 2u, s2 = sh & 4u, odd = sh & 1u;
#pragma unroll
        for (int i = 0; i < 7; i++) w[i] = s1 ? w[i + 1] : w[i];
#pragma unroll
        for (int i = 0; i < 5; i++) w[i] = s2 ? w[i + 2] : w[i];
#pragma unroll
        for (int i = 0; i < 4; i++) w[i] = odd ? __funnelshift_r(w[i], w[i + 1], 16) : w[i];
        r = make_uint4(w[0], w[1], w[2], w[3]);
    }
    if (lim < 8) {
        r.x = keep_below(r.x, 0, lim);
        r.y = keep_below(r.y, 2, lim);
        r.z = keep_below(r.z, 4, lim);
        r.w = keep_below(r.w, 6, lim);
    }
    return r;
}

__device__ __forceinline__ void slot_i16(const int16_t *__restrict__ scr, int16_t *__restrict__ out, const WinDesc &d)
{
    const uint64_t n_out = (uint64_t)d.frames * d.channels, n_real = (uint64_t)d.real * d.channels;
    int16_t *o = out + d.dst;
    const int16_t *s = scr + d.src;
    // head: the elements before the slot's first 16-byte boundary; body: whole aligned vectors; tail: what is left
    const uint32_t mis = (uint32_t)(reinterpret_cast<uintptr_t>(o) >> 1) & 7u;
    const uint64_t head = min((uint64_t)((8u - mis) & 7u), n_out);
    const uint64_t nv = (n_out - head) >> 3, tail0 = head + (nv << 3);
    if (blockIdx.x == 0 && threadIdx.x < 16) {
        const uint64_t i = threadIdx.x < 8 ? threadIdx.x : tail0 + threadIdx.x - 8;
        if (threadIdx.x < 8 ? i < head : i < n_out) o[i] = i < n_real ? s[i] : (int16_t)0;
    }
    const uint64_t sb = d.src + head;  // scratch element of body element 0, `sh` elements into an aligned vector
    const uint32_t sh = (uint32_t)sb & 7u;
    const uint4 *sv = reinterpret_cast<const uint4 *>(scr + (sb - sh));
    uint4 *ov = reinterpret_cast<uint4 *>(o + head);
    const int64_t lim0 = (int64_t)n_real - (int64_t)head;
    const uint64_t step = (uint64_t)gridDim.x * kWinThreads * 2u;
    for (uint64_t j = (uint64_t)blockIdx.x * kWinThreads * 2u + threadIdx.x; j < nv; j += step) {
        const uint64_t j1 = j + kWinThreads;
        const uint4 v0 = body_vector(sv, j, sh, lim0 - (int64_t)(j << 3));
        if (j1 < nv) {
            const uint4 v1 = body_vector(sv, j1, sh, lim0 - (int64_t)(j1 << 3));
            ov[j] = v0;
            ov[j1] = v1;
        } else {
            ov[j] = v0;
        }
    }
}

// ---- float32, planar ------------------------------------------------------------------------------------------------------------

// Frames per tile: a power of two with tile frames x channels <= 4096 samples (at least 32 frames, one warp-wide row).
__device__ __forceinline__ uint32_t tile_frames_log2(uint32_t channels)
{
    const uint32_t tf = max(32u, 4096u / channels);
    return 31u - __clz(tf);
}

// A tile = TF frames x all channels.  Its interleaved samples are contiguous in scratch: read as aligned 16-byte vectors into
// shared memory (the first `sh` staged samples belong to the previous tile), then written channel row by channel row, a warp
// covering 32 consecutive frames of one row.
__device__ __forceinline__ void slot_f32_planar(const int16_t *__restrict__ scr, float *__restrict__ out, const WinDesc &d)
{
    __shared__ __align__(16) int16_t tile[kWinTileElems];
    const uint32_t C = d.channels, lg = tile_frames_log2(C), TF = 1u << lg;
    const uint32_t n_tiles = (d.frames + TF - 1u) >> lg;
    for (uint32_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
        const uint32_t f0 = t << lg;
        const uint32_t tf = min(TF, d.frames - f0);                  // slot frames of this tile
        const uint32_t rf = d.real > f0 ? min(tf, d.real - f0) : 0u;  // of them, frames from scratch
        uint32_t sh = 0;
        if (rf) {
            const uint64_t a = d.src + (uint64_t)f0 * C;
            sh = (uint32_t)a & 7u;
            const uint4 *sv = reinterpret_cast<const uint4 *>(scr + (a - sh));
            const uint32_t nvec = (sh + rf * C + 7u) >> 3;
            uint4 *tv = reinterpret_cast<uint4 *>(tile);
            for (uint32_t v = threadIdx.x; v < nvec; v += kWinThreads) tv[v] = __ldg(sv + v);
        }
        __syncthreads();
        float *o = out + d.dst + f0;
        for (uint32_t i = threadIdx.x; i < (C << lg); i += kWinThreads) {
            const uint32_t c = i >> lg, f = i & (TF - 1u);
            if (f < tf) o[(uint64_t)c * d.frames + f] = f < rf ? (float)tile[sh + f * C + c] * (1.0f / 32768.0f) : 0.0f;
        }
        __syncthreads();
    }
}

// blockIdx.y walks the windows, blockIdx.x the vectors / tiles of a window
template <bool kPlanar>
__global__ void __launch_bounds__(kWinThreads) window_extract_kernel(const int16_t *__restrict__ scr, void *__restrict__ out,
                                                                     const WinDesc *__restrict__ desc, uint32_t n_windows)
{
    for (uint32_t w = blockIdx.y; w < n_windows; w += gridDim.y) {
        const WinDesc d = desc[w];
        if constexpr (kPlanar) slot_f32_planar(scr, static_cast<float *>(out), d);
        else slot_i16(scr, static_cast<int16_t *>(out), d);
    }
}

cudaError_t launch_window_extract(const int16_t *d_scratch, void *d_out, const WinDesc *d_desc, uint32_t n_windows, uint64_t max_slot_samples,
                                  bool planar_f32, cudaStream_t stream)
{
    if (n_windows == 0 || max_slot_samples == 0) return cudaSuccess;
    const uint64_t bx = (max_slot_samples + kWinSlotSamplesPerCta - 1u) / kWinSlotSamplesPerCta;
    const dim3 grid((unsigned)(bx < (1u << 20) ? bx : (1u << 20)), n_windows < 65535u ? n_windows : 65535u);
    debug_launch("window_extract<%d>: %u x %u CTAs", (int)planar_f32, grid.x, grid.y);
    if (planar_f32) window_extract_kernel<true><<<grid, kWinThreads, 0, stream>>>(d_scratch, d_out, d_desc, n_windows);
    else window_extract_kernel<false><<<grid, kWinThreads, 0, stream>>>(d_scratch, d_out, d_desc, n_windows);
    return cudaGetLastError();
}

}  // namespace sea
