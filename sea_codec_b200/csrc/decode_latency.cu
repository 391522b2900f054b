// decode_latency.cu -- decode for SMALL jobs: the one-chunk streaming seam (SeaFile::samples_from_reader, file.rs:180-209), a
// handful of chunks per call, one short file (BASELINE config 1: 87 chunks; config 3: one 8-channel stream, 2813 chunks).
//
// The lane-per-chunk throughput kernels need tens of thousands of chunks to fill the machine; a chunk by itself is a serial chain
// per channel (lms.rs:33-51), and what matters then is the length of that chain in cycles.  Here one small CTA (4 warps) owns one
// chunk:
//   A  all threads parse the chunk (chunk.rs:69-213), stage its bytes in shared memory, and turn every residual code into its
//      dequantised value up front (bits.rs:34-78 + dqt.rs tables): d[channel][frame] as int16 in shared memory -- the part of the
//      work that has no dependency at all;
//   B  lane c < channels of the first warp runs channel c's recurrence (codec/decoder.rs:20-86) over the chunk.  The weights of step t depend on
//      samples up to t-2 only, so the one product that waits for sample t-1 is w3 * y(t-1): the chain is IMAD -> shift+add -> clamp,
//      with the look-ups, the other three taps and the four weight updates scheduled beside it.  A channel's row is contiguous:
//      eight d values come in with one 128-bit shared load and eight samples go back with one store, in place;
//   C  all threads interleave the rows into the PCM output with coalesced stores.
// Any per-chunk header (CBR / VBR, 1..8 scale-factor bits, any scale_factor_frames), any channel count up to 32, partial chunks,
// every section checked against the bytes available exactly like decode_generic_kernel (same error codes).
#include "sea_device.cuh"

#ifdef SEA_LAT_DEBUG
#include <stdio.h>
#define LAT_MARK(i) do { if (tid == 0 && blockIdx.x == 0) t_mark[i] = clock64(); } while (0)
#else
#define LAT_MARK(i) do { } while (0)
#endif

namespace sea {

using namespace dev;

namespace {

// MSB-first field of n <= 8 bits at bit offset `bit` of a byte string in shared memory (bits.rs:42-46)
__device__ __forceinline__ uint32_t get_bits_smem(const uint8_t *p, uint32_t bit, uint32_t n)
{
    const uint32_t byte = bit >> 3, sh = bit & 7u;
    const uint32_t v = ((uint32_t)p[byte] << 8) | (uint32_t)p[byte + 1];  // the staged copy has two spare bytes
    return (v >> (16u - sh - n)) & ((1u << n) - 1u);
}

}  // namespace

// Shared memory per CTA: [chunk bytes, padded] [d / pcm: channels rows of row_pitch(frames_per_chunk) int16] [per block: bit
// offset u32, frame bits u16 -- VBR only] [dequant rows, int16].  kLatWarps warps per CTA: all of them parse / dequantise / copy out,
// warp 0 runs the recurrences.
__host__ __device__ inline uint32_t latency_row_pitch(uint32_t frames_per_chunk) { return ((frames_per_chunk + 7u) & ~7u) + 8u; }
constexpr uint32_t kLatencyLutEntries = 4096;  // dequant rows kept in shared memory up to this many entries (8 KB)
constexpr uint32_t kLatWarps = 4, kLatThreads = kLatWarps * 32;

// One pass of phase A2 for eight samples per thread.  VBR picks the per-(block, channel) sizes; branch free so that the eight
// look-up chains of a thread interleave (an index past the end is clamped and its result dropped).
template <bool VBR>
__device__ __forceinline__ void dequant_pass(uint32_t i0, uint32_t tid, uint32_t n_all, uint32_t C, uint32_t F, uint32_t s, uint32_t b,
                                             uint64_t recipC, uint64_t recipF, const uint8_t *cbytes, uint32_t sf_sec, uint32_t vbr_sec,
                                             const uint8_t *res, const uint32_t *blkbit, const uint16_t *rowbits, const int16_t *lut,
                                             bool lut_in_smem, const int32_t *tab, uint32_t lut_first, int16_t *dbuf, uint32_t pitch)
{
    int32_t dv[8];
    uint32_t slot[8];
#pragma unroll
    for (uint32_t u = 0; u < 8u; u++) {
        const uint32_t i_raw = i0 + u * kLatThreads + tid, i = i_raw < n_all ? i_raw : n_all - 1u;
        const uint32_t f = (uint32_t)(((uint64_t)i * recipC) >> 40), c = i - f * C;
        const uint32_t blk = (uint32_t)(((uint64_t)f * recipF) >> 32);
        const uint32_t sf = get_bits_smem(cbytes + sf_sec, (blk * C + c) * s, s);
        uint32_t size = b, pos = i * b;
        if (VBR) {
            uint32_t prefix = 0;
            for (uint32_t cc = 0; cc < c; cc++) prefix += get_bits_smem(cbytes + vbr_sec, (blk * C + cc) * 2u, 2u) + b - 1u;
            size = get_bits_smem(cbytes + vbr_sec, (blk * C + c) * 2u, 2u) + b - 1u;
            pos = blkbit[blk] + (f - blk * F) * rowbits[blk] + prefix;
        }
        const uint32_t code = get_bits_smem(res, pos, size);
        const uint32_t e = tab_dqt_off(s, size) - lut_first + (sf << size) + code;
        dv[u] = lut_in_smem ? (int32_t)lut[e] : __ldg(tab + lut_first + e);
        slot[u] = i_raw < n_all ? c * pitch + f : 0xffffffffu;
    }
#pragma unroll
    for (uint32_t u = 0; u < 8u; u++)
        if (slot[u] != 0xffffffffu) dbuf[slot[u]] = (int16_t)dv[u];
}

__global__ void __launch_bounds__(kLatThreads) decode_latency_kernel(const uint8_t *__restrict__ sea, int16_t *__restrict__ pcm,
                                                                     const DecStream *__restrict__ streams, uint32_t n_streams,
                                                                     uint64_t total_chunks, uint32_t max_chunk_bytes, DevTables tabs, int *err)
{
    extern __shared__ __align__(16) uint8_t smem[];
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
#ifdef SEA_LAT_DEBUG
    long long t_mark[6] = {};
#endif
    LAT_MARK(0);
    const uint64_t g = blockIdx.x;  // global chunk index (chunks of all streams numbered consecutively)
    if (g >= total_chunks) return;
    // streams[].chain_begin counts chains (chunk, channel); every stream of this launch has the same channel count
    const uint32_t C = streams[0].channels;
    const DecStream st = streams[find_stream(streams, n_streams, g * C)];
    const uint32_t k = (uint32_t)(g - st.chain_begin / C);
    const uint64_t ck_off = (uint64_t)k * st.chunk_size;
    const uint8_t *ck = sea + st.data_off + ck_off;
    const uint64_t rest = st.data_len - ck_off;
    const uint32_t take = rest < st.chunk_size ? (uint32_t)rest : st.chunk_size;
    const uint32_t N = st.frames_per_chunk;
    uint32_t frames = st.total_frames - k * N;
    if (frames > N) frames = N;

    // the staged copy keeps the chunk's 16-byte phase, so that its whole granules move as 128-bit loads
    uint8_t *cbytes = smem + (reinterpret_cast<uint64_t>(ck) & 15u);
    int16_t *dbuf = reinterpret_cast<int16_t *>(smem + ((max_chunk_bytes + 2u + 16u + 15u) & ~15u));
    const uint32_t pitch = latency_row_pitch(N);  // int16 per channel row, a multiple of 8: rows start 16-byte aligned
    uint32_t *blkbit = reinterpret_cast<uint32_t *>(dbuf + (size_t)C * pitch);
    const uint64_t recipC = ((1ull << 40) + C - 1u) / C;  // i / C == (i * recipC) >> 40 for i < 2^20, C <= 32

    // ---- A0: stage the chunk (chunks sit at arbitrary byte offsets, 22 + k * chunk_size): bytes up to the first 16-byte boundary,
    // whole granules, bytes after the last boundary -- nothing outside [ck, ck + take) is read
    {
        const uint32_t head = (16u - (uint32_t)(reinterpret_cast<uint64_t>(ck) & 15u)) & 15u;
        const uint32_t h = head < take ? head : take, vecs = (take - h) >> 4, tail0 = h + (vecs << 4);
        if (tid < h) cbytes[tid] = __ldg(ck + tid);
        const uint4 *src = reinterpret_cast<const uint4 *>(ck + h);
        uint4 *dst = reinterpret_cast<uint4 *>(cbytes + h);
        for (uint32_t i = tid; i < vecs; i += kLatThreads) dst[i] = __ldg(src + i);
        if (tail0 + tid < take) cbytes[tail0 + tid] = __ldg(ck + tail0 + tid);
        if (tid < 2u) cbytes[take + tid] = 0;
    }
    __syncthreads();
    LAT_MARK(1);

    // ---- header and section layout (chunk.rs:81-113), validated against the bytes available like the generic kernel (every
    // thread evaluates the same shared bytes: the early exits are CTA-uniform)
    if (take < 4u + 16u * C) {
        if (tid == 0) report(err, kDevDomain);
        return;
    }
    const uint32_t type = cbytes[0], s = cbytes[1] >> 4, b = cbytes[1] & 15u, F = cbytes[2];
    if (type != 1u && type != 2u) {
        if (tid == 0) report(err, kDevInvalidFrame);
        return;
    }
    if (b < 1u || b > 8u || s < 1u || s > 8u || F == 0u) {
        if (tid == 0) report(err, kDevDomain);
        return;
    }
    const bool vbr = type == 2u;
    const uint32_t nblk = div_ceil_u32(frames, F), items = nblk * C;
    const uint32_t sf_sec = 4u + 16u * C;
    const uint32_t vbr_sec = sf_sec + div_ceil_u32(items * s, 8u);
    const uint32_t res_sec = vbr_sec + (vbr ? div_ceil_u32(items * 2u, 8u) : 0u);
    if (res_sec > take) {
        if (tid == 0) report(err, kDevDomain);
        return;
    }
    const uint64_t res_bits_avail = (uint64_t)(take - res_sec) * 8u;
    const int32_t *tab = tabs.by_s[s];
    uint16_t *rowbits = reinterpret_cast<uint16_t *>(blkbit + nblk);
    int16_t *lut = reinterpret_cast<int16_t *>(rowbits + ((nblk + 7u) & ~7u));
    __shared__ uint32_t sh_verdict;  // 0 = fine, else the device error code

    // ---- A1 (warp 0): VBR bit offset and frame width of every block (chunk.rs:126-139) -- a run of blocks per lane, then a warp
    // scan; the size check of the whole chunk (CBR: one product)
    if (warp == 0) {
        bool bad = false;
        uint64_t total_bits = (uint64_t)frames * C * b;
        if (vbr) {
            const uint32_t per = (nblk + 31u) / 32u, b0 = lane * per, b1 = b0 + per < nblk ? b0 + per : nblk;
            uint32_t mine = 0;
            for (uint32_t blk = b0; blk < b1; blk++) {
                uint32_t rb = 0;
                for (uint32_t c = 0; c < C; c++) {
                    const uint32_t sz = get_bits_smem(cbytes + vbr_sec, (blk * C + c) * 2u, 2u) + b - 1u;
                    bad |= sz < 1u || sz > 8u;
                    rb += sz;
                }
                uint32_t nf = frames - blk * F;
                if (nf > F) nf = F;
                rowbits[blk] = (uint16_t)rb;
                mine += nf * rb;
            }
            uint32_t incl = mine;
#pragma unroll
            for (uint32_t o = 1; o < 32u; o <<= 1) {
                const uint32_t up = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += up;
            }
            uint32_t acc = incl - mine;
            for (uint32_t blk = b0; blk < b1; blk++) {
                uint32_t nf = frames - blk * F;
                if (nf > F) nf = F;
                blkbit[blk] = acc;
                acc += nf * rowbits[blk];
            }
            total_bits = __shfl_sync(0xffffffffu, incl, 31);
            bad = __any_sync(0xffffffffu, bad);
        }
        // a size outside 1..8 panics in the reference (common.rs:34); a short residual section is a slice error
        if (lane == 0) sh_verdict = (bad || total_bits > res_bits_avail) ? (uint32_t)kDevDomain : 0u;
    }
    // the dequant rows the chunk can use, as int16, when they are small (CBR-3: 256 B); larger sets are read through L1
    const uint32_t lo_size = vbr ? (b > 1u ? b - 1u : 1u) : b, hi_size = vbr ? (b + 2u < 8u ? b + 2u : 8u) : b;
    const uint32_t lut_first = tab_dqt_off(s, lo_size), lut_entries = tab_dqt_off(s, hi_size + 1u) - lut_first;
    const bool lut_in_smem = lut_entries <= kLatencyLutEntries;
    if (lut_in_smem)
        for (uint32_t i = tid; i < lut_entries; i += kLatThreads) lut[i] = (int16_t)__ldg(tab + lut_first + i);
    __syncthreads();
    if (sh_verdict) {
        if (tid == 0) report(err, (int)sh_verdict);
        return;
    }
    LAT_MARK(2);

    // ---- A2: every residual code -> its dequantised value (|d| <= 255 * 99 fits int16), rows [channel][frame].  One flat loop over
    // the chunk's samples, eight per thread and pass: the look-ups of a pass are independent and issued together (a store to
    // shared memory between them would order every later load behind it: block by block, one warp, this phase cost 2.6x the
    // recurrence).
    const uint8_t *res = cbytes + res_sec;
    const uint32_t n_all = frames * C;
    const uint64_t recipF = ((1ull << 32) + F - 1u) / F;  // f / F == (f * recipF) >> 32 for f < 2^16
    for (uint32_t i0 = 0; i0 < n_all; i0 += 8u * kLatThreads) {
        if (vbr) dequant_pass<true>(i0, tid, n_all, C, F, s, b, recipC, recipF, cbytes, sf_sec, vbr_sec, res, blkbit, rowbits, lut, lut_in_smem, tab, lut_first, dbuf, pitch);
        else dequant_pass<false>(i0, tid, n_all, C, F, s, b, recipC, recipF, cbytes, sf_sec, vbr_sec, res, blkbit, rowbits, lut, lut_in_smem, tab, lut_first, dbuf, pitch);
    }
    __syncthreads();
    LAT_MARK(3);

    // ---- B: the recurrences, one channel per lane of warp 0
    if (warp == 0 && lane < C) {
        int32_t w[4], h[4], sg[4];
        const uint8_t *l = cbytes + 4u + 16u * lane;  // lms.rs:80-94
#pragma unroll
        for (int i = 0; i < 4; i++) {
            h[i] = (int16_t)(l[2 * i] | (l[2 * i + 1] << 8));
            w[i] = (int16_t)(l[8 + 2 * i] | (l[8 + 2 * i + 1] << 8));
            sg[i] = (h[i] >> 31) | 1;
        }
        // eight samples per group, in place in the channel's row: one 128-bit load, one 128-bit store, no predicates (a group may
        // run into the row's padding after the chunk's last frame: those values are computed and never read)
        uint4 *row = reinterpret_cast<uint4 *>(dbuf + (size_t)lane * pitch);
        uint4 nxt = row[0];
        for (uint32_t t0 = 0; t0 < frames; t0 += 8u) {
            const uint4 cur = nxt;
            nxt = row[(t0 >> 3) + 1u];  // the row is padded by one group
            const uint32_t in[4] = {cur.x, cur.y, cur.z, cur.w};
            uint32_t outw[4];
#pragma unroll
            for (uint32_t u = 0; u < 8u; u++) {
                const int32_t d = (u & 1u) ? (int32_t)in[u >> 1] >> 16 : (int32_t)(int16_t)(in[u >> 1] & 0xffffu);
                // everything but w[3] * h[3] is known one sample early: the newest history value enters last
                const uint32_t part = (uint32_t)w[0] * (uint32_t)h[0] + (uint32_t)w[1] * (uint32_t)h[1] + (uint32_t)w[2] * (uint32_t)h[2];
                const uint32_t acc = part + (uint32_t)w[3] * (uint32_t)h[3];
                const int32_t v = (int32_t)((uint32_t)((int32_t)acc >> 13) + (uint32_t)d);
                const int32_t y = clamp_i16(v);
                if (u & 1u) outw[u >> 1] |= (uint32_t)y << 16;
                else outw[u >> 1] = (uint32_t)y & 0xffffu;
                const int32_t delta = d >> 4;
#pragma unroll
                for (int i = 0; i < 4; i++) w[i] += delta * sg[i];
                h[0] = h[1]; h[1] = h[2]; h[2] = h[3]; h[3] = y;
                sg[0] = sg[1]; sg[1] = sg[2]; sg[2] = sg[3]; sg[3] = (v >> 31) | 1;  // the clamp keeps the sign
            }
            row[t0 >> 3] = make_uint4(outw[0], outw[1], outw[2], outw[3]);
        }
    }
    __syncthreads();
    LAT_MARK(4);

    // ---- C: interleave the rows into the PCM output (the chunk's samples are contiguous: pcm_off + k * N * C)
    int16_t *out = pcm + st.pcm_off + (uint64_t)k * N * C;
    const uint32_t n_out = frames * C;
    if ((C & 1u) == 0 && (reinterpret_cast<uint64_t>(out) & 3u) == 0) {  // even channel counts: a channel pair per 32-bit store
        uint32_t *dst32 = reinterpret_cast<uint32_t *>(out);
        const uint32_t hc = C >> 1;
        const uint64_t recipH = ((1ull << 40) + hc - 1u) / hc;
#pragma unroll 4
        for (uint32_t j = tid; j < n_out / 2u; j += kLatThreads) {
            const uint32_t f = (uint32_t)(((uint64_t)j * recipH) >> 40), c = 2u * (j - f * hc);
            dst32[j] = (uint32_t)(uint16_t)dbuf[c * pitch + f] | ((uint32_t)(uint16_t)dbuf[(c + 1u) * pitch + f] << 16);
        }
    } else {
#pragma unroll 4
        for (uint32_t i = tid; i < n_out; i += kLatThreads) {
            const uint32_t f = (uint32_t)(((uint64_t)i * recipC) >> 40), c = i - f * C;
            out[i] = dbuf[c * pitch + f];
        }
    }
    LAT_MARK(5);
#ifdef SEA_LAT_DEBUG
    if (tid == 0 && blockIdx.x == 0)
        printf("latency kernel cycles: stage %lld, parse+scan %lld, dequant %lld, recurrence %lld, copy-out %lld\n", t_mark[1] - t_mark[0],
               t_mark[2] - t_mark[1], t_mark[3] - t_mark[2], t_mark[4] - t_mark[3], t_mark[5] - t_mark[4]);
#endif
}

// Shared-memory footprint of one chunk; 0 when the geometry does not fit (the caller keeps its other kernels then).
size_t decode_latency_smem(uint32_t chunk_size, uint32_t frames_per_chunk, uint32_t channels)
{
    if (channels == 0 || channels > 32u) return 0;
    const size_t bytes = ((chunk_size + 2u + 16u + 15u) & ~(size_t)15u) + (size_t)channels * latency_row_pitch(frames_per_chunk) * 2u +
                         (size_t)frames_per_chunk * 6u + 32u + kLatencyLutEntries * 2u;
    return bytes <= 200u * 1024u ? bytes : 0;
}

cudaError_t launch_decode_latency(const uint8_t *d_sea, int16_t *d_pcm, const DecStream *d_streams, uint32_t n_streams, uint64_t total_chunks,
                                  uint32_t chunk_size, uint32_t frames_per_chunk, uint32_t channels, DevTables tabs, int *d_err,
                                  cudaStream_t stream)
{
    if (total_chunks == 0) return cudaSuccess;
    const size_t smem = decode_latency_smem(chunk_size, frames_per_chunk, channels);
    if (!smem || total_chunks > 0x7fffffffull) return cudaErrorInvalidConfiguration;
    // the attributes are per device and sticky: set them on a device's first launch only (two driver calls are a tenth of what a
    // one-chunk call costs end to end)
    static bool configured[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64 || !configured[dev]) {
        cudaError_t e = cudaFuncSetAttribute(decode_latency_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        if (e != cudaSuccess) return e;
        e = cudaFuncSetAttribute(decode_latency_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
        if (e != cudaSuccess) return e;
        if (dev >= 0 && dev < 64) configured[dev] = true;
    }
    debug_launch("decode_latency: %u channels, %u warps/CTA, %zu B smem, %llu CTAs", channels, kLatWarps, smem, (unsigned long long)total_chunks);
    decode_latency_kernel<<<(unsigned)total_chunks, kLatThreads, smem, stream>>>(d_sea, d_pcm, d_streams, n_streams, total_chunks, chunk_size, tabs,
                                                                        d_err);
    return cudaGetLastError();
}

}  // namespace sea
