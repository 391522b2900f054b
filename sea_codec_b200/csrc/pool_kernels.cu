// pool_kernels.cu -- the two kernels around the encoder of a session pool (sea_b200_encoder_pool_push): the ingest, which builds
// the encode launch's contiguous input and the sessions' new carries from ragged packets and gathers the state rows of the
// sessions that encode, and the commit, which scatters their advanced state rows back to the slots.
//
// The host lays the ingest out as a list of plain copies (PoolCopy): carry -> launch input, packet -> launch input, packet ->
// new carry, packet -> end of the current carry, state row -> launch state.  Packets range from one frame to many chunks, so
// the grid is cut by OUTPUT volume, not by session: CTA b writes the 16-byte destination vectors [b * 1024, (b + 1) * 1024) of
// the concatenated copies, whichever copies those are.  A vector whose 8 elements all belong to the copy is one 16-byte store,
// loaded as one aligned vector or, when the source sits at another offset inside its 16 bytes, as two aligned vectors shifted
// together; the at most two partial vectors at a copy's ends are written element by element, so neighbouring copies that share
// a vector never write each other's bytes.
#include "sea_kernels.h"

namespace sea {

constexpr uint32_t kIngestThreads = 256;
constexpr uint32_t kIngestVecsPerCta = 1024;  // 16 KB of output per CTA

__device__ __forceinline__ uint64_t copy_vectors(const PoolCopy &c)
{
    const uint64_t d = reinterpret_cast<uintptr_t>(c.dst);
    return ((d + 2u * c.n + 15u) >> 4) - (d >> 4);
}

// 8 int16 starting `sh` (1..7) elements into the aligned vector at v
__device__ __forceinline__ uint4 shifted_vector(const uint4 *__restrict__ v, uint32_t sh)
{
    const uint4 a = __ldg(v), b = __ldg(v + 1);
    uint32_t w[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
    // by sh >> 1 words with selects on constant indices (a dynamic index would put w in local memory), then by one int16 when
    // sh is odd
    const bool s1 = sh & 2u, s2 = sh & 4u, odd = sh & 1u;
#pragma unroll
    for (int i = 0; i < 7; i++) w[i] = s1 ? w[i + 1] : w[i];
#pragma unroll
    for (int i = 0; i < 5; i++) w[i] = s2 ? w[i + 2] : w[i];
#pragma unroll
    for (int i = 0; i < 4; i++) w[i] = odd ? __funnelshift_r(w[i], w[i + 1], 16) : w[i];
    return make_uint4(w[0], w[1], w[2], w[3]);
}

// Destination vector j (counted from the vector holding c.dst[0]) of copy c.
__device__ __forceinline__ void copy_vector(const PoolCopy &c, uint64_t j)
{
    const uint64_t d = reinterpret_cast<uintptr_t>(c.dst);
    const uint64_t va = ((d >> 4) + j) << 4;  // byte address of the vector
    const uint64_t e0 = va > d ? (va - d) >> 1 : 0u;
    const uint64_t e1 = min(c.n, (uint64_t)((va + 16u - d) >> 1));
    if (e1 - e0 == 8u) {
        const uintptr_t s = reinterpret_cast<uintptr_t>(c.src + e0);
        const uint32_t sh = (uint32_t)(s & 15u) >> 1;
        const uint4 *sv = reinterpret_cast<const uint4 *>(s & ~(uintptr_t)15u);
        *reinterpret_cast<uint4 *>(va) = sh ? shifted_vector(sv, sh) : __ldg(sv);
    } else {
        for (uint64_t e = e0; e < e1; e++) c.dst[e] = c.src[e];
    }
}

// Copies never overlap and no copy reads what another one writes (the host keeps a session's current and next carry in
// different halves of its slot, and a carry that only grows is appended past the frames it already holds).
__global__ void __launch_bounds__(kIngestThreads) pool_ingest_kernel(const PoolCopy *__restrict__ copies, uint32_t n_copies,
                                                                     uint64_t total_vectors)
{
    __shared__ uint32_t first;
    const uint64_t t0 = (uint64_t)blockIdx.x * kIngestVecsPerCta;
    const uint64_t t1 = min(t0 + (uint64_t)kIngestVecsPerCta, total_vectors);
    if (threadIdx.x == 0) {  // the last copy that starts at or before t0 (copies are never empty)
        uint32_t lo = 0, hi = n_copies;
        while (hi - lo > 1u) {
            const uint32_t mid = (lo + hi) >> 1;
            if (copies[mid].v_begin <= t0) lo = mid;
            else hi = mid;
        }
        first = lo;
    }
    __syncthreads();
    for (uint32_t i = first; i < n_copies; i++) {
        const PoolCopy c = copies[i];
        if (c.v_begin >= t1) break;
        const uint64_t nv = copy_vectors(c);
        const uint64_t lo = max(t0, c.v_begin) - c.v_begin, hi = min(t1, c.v_begin + nv) - c.v_begin;
        for (uint64_t j = lo + threadIdx.x; j < hi; j += kIngestThreads) copy_vector(c, j);
    }
}

__global__ void pool_commit_kernel(const int32_t *__restrict__ rows, int32_t *__restrict__ state, const uint32_t *__restrict__ slots,
                                   uint32_t n_rows, uint32_t row_words)
{
    const uint64_t total = (uint64_t)n_rows * row_words;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t r = i / row_words, w = i - r * row_words;
        state[(uint64_t)slots[r] * row_words + w] = rows[i];
    }
}

cudaError_t launch_pool_ingest(const PoolCopy *d_copies, uint32_t n_copies, uint64_t total_vectors, cudaStream_t stream)
{
    if (n_copies == 0 || total_vectors == 0) return cudaSuccess;
    const uint64_t ctas = (total_vectors + kIngestVecsPerCta - 1u) / kIngestVecsPerCta;
    if (ctas > 0x7fffffffull) return cudaErrorInvalidValue;
    debug_launch("pool_ingest_kernel: %u copies, %llu vectors, %llu CTAs", n_copies, (unsigned long long)total_vectors,
                 (unsigned long long)ctas);
    pool_ingest_kernel<<<(unsigned)ctas, kIngestThreads, 0, stream>>>(d_copies, n_copies, total_vectors);
    return cudaGetLastError();
}

cudaError_t launch_pool_commit(const int32_t *d_rows, int32_t *d_state, const uint32_t *d_slots, uint32_t n_rows, uint32_t row_words,
                               cudaStream_t stream)
{
    if (n_rows == 0) return cudaSuccess;
    const uint64_t total = (uint64_t)n_rows * row_words;
    const uint64_t want = (total + 255u) / 256u;
    const unsigned ctas = (unsigned)(want < 148u * 16u ? want : 148u * 16u);
    debug_launch("pool_commit_kernel: %u rows of %u words, %u CTAs", n_rows, row_words, ctas);
    pool_commit_kernel<<<ctas, 256, 0, stream>>>(d_rows, d_state, d_slots, n_rows, row_words);
    return cudaGetLastError();
}

}  // namespace sea
