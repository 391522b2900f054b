// capi.cu -- the extern "C" boundary of libsea_b200.so (see include/sea_b200.h for what each entry point replaces).
// Host-side work that stays scalar: file headers, launch planning, VBR bucket counts (f32), table generation.
// There is deliberately no CPU implementation of the codec here: a missing or failing GPU is an error return.
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <vector>

#include "../../include/sea_b200.h"
#include "sea_format.h"
#include "sea_kernels.h"

using namespace sea;

namespace {

struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t bytes)
    {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        size_t want = bytes + (bytes >> 3) + 4096;
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release()
    {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
    template <typename T>
    T *as() const { return reinterpret_cast<T *>(p); }
};

}  // namespace

struct sea_b200_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    int32_t *d_tab[9] = {};
    DevTables tabs = {};
    DevBuf in, out, streams, lens, chunk0, scratch, misc;
    int *d_err = nullptr;
    DevBuf ties;  // [0] VBR boundary ties of the last encode, [1 + i] those of its stream i
    std::vector<unsigned long long> h_ties;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    cudaStream_t side = nullptr;                       // partial-chunk decode runs beside the full-chunk kernel
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    // second decode lane: sea_b200_decode_batch pipelines groups of streams (H2D of group i+1 and D2H of group i-1 overlap the
    // kernels of group i), alternating between the primary resources above and these
    struct {
        cudaStream_t stream = nullptr, side = nullptr;
        cudaEvent_t ev_fork = nullptr, ev_join = nullptr, ev0 = nullptr, ev1 = nullptr;
        DevBuf in, out, table;
        int *d_err = nullptr;
    } aux;
    // time-sliced host-buffer encode (sea_b200_encode_batch): upload / kernel / download of neighbouring slices overlap
    struct {
        cudaEvent_t up[2] = {}, kern[2] = {}, down[2] = {};
        DevBuf in[2], out[2], state;
    } pipe;
    // pipelined host-buffer decode: the error words of its groups land here (pinned) and are read once, after the last group was
    // queued; two timing events per group
    int *h_errs = nullptr;
    size_t h_errs_cap = 0;
    std::vector<cudaEvent_t> grp_ev;
    cudaStream_t up = nullptr;  // uploads of a pipelined batch run ahead of the lanes on their own stream
    DevBuf win, win_desc;       // sea_b200_decode_windows_device: decoded covering chunks of a group of windows, their descriptors
    std::string last_error;
    uint64_t launches = 0;
    double last_kernel_ms = 0.0;
    unsigned long long last_ties = 0;
};

struct sea_b200_encoder {
    sea_b200_ctx *ctx;
    sea_b200_settings settings;
    EncodePlan plan;
    uint32_t channels, sample_rate;
    uint32_t chunk_size = 0;
    int32_t *d_state = nullptr;
};

// A slot table of streaming encoders that share one launch per push (sea_b200_encoder_pool_*).  Every slot owns a state row
// (kEncStateWords int32 per channel) and two carry buffers of frames_per_chunk frames: a push that completes a chunk reads the
// current carry into the launch input and writes the new remainder into the other one, so the ingest never reads what it writes.
struct sea_b200_encoder_pool {
    sea_b200_ctx *ctx;
    sea_b200_settings settings;
    EncodePlan plan;
    uint32_t max_sessions, channels, sample_rate;
    int16_t *d_carry = nullptr;  // [max_sessions][2][N * channels]
    int32_t *d_state = nullptr;  // [max_sessions][channels * kEncStateWords]
    int32_t *d_init = nullptr;   // one row of EncoderBase::new state: a freshly opened slot gathers its state from here
    std::vector<uint32_t> carry;                 // frames buffered per slot
    std::vector<uint8_t> half, open, fresh;      // current carry half; open; state row not yet written since open
    std::vector<uint32_t> seen;                  // duplicate check: call stamp per slot
    uint32_t stamp = 0;
    DevBuf pk, in, rows, ob, desc;               // packets (host form), launch input, gathered state rows, output (host form), copies + slots
    uint8_t *h_desc = nullptr;                   // pinned staging of the copy list and the slot list
    size_t h_desc_cap = 0;
    cudaEvent_t ev[4] = {};                      // ingest start, ingest end, encode end, commit end
};

struct sea_b200_decoder {
    sea_b200_ctx *ctx;
    sea_b200_header header;
    int sf_bits = -1;  // Decoder::init on the first chunk (file.rs:193-198)
};

namespace {

int fail(sea_b200_ctx *ctx, int code, const std::string &msg)
{
    if (ctx) ctx->last_error = msg;
    return code;
}
int cuda_fail(sea_b200_ctx *ctx, cudaError_t e, const char *what)
{
    return fail(ctx, e == cudaErrorMemoryAllocation ? SEA_B200_ERR_NOMEM : SEA_B200_ERR_CUDA,
                std::string(what) + ": " + cudaGetErrorString(e));
}
#define CU(call)                                                      \
    do {                                                              \
        cudaError_t e_ = (call);                                      \
        if (e_ != cudaSuccess) return cuda_fail(ctx, e_, #call);      \
    } while (0)

int map_dev_error(sea_b200_ctx *ctx, int dev_err)
{
    switch (dev_err) {
        case kDevOk: return SEA_B200_OK;
        case kDevInvalidFrame: return fail(ctx, SEA_B200_ERR_INVALID_FRAME, "chunk type is neither CBR nor VBR (chunk.rs:81-85)");
        default: return fail(ctx, SEA_B200_ERR_DOMAIN, "chunk data outside the reference's domain (it would panic: truncated or malformed chunk)");
    }
}

// ------------------------------------------------------------------------------------------------ decode core

struct DecodeJob {
    std::vector<DecStream> streams;
    std::vector<uint64_t> n_samples;
    uint64_t total_chains = 0;
    bool uniform = true;
    bool trailing_invalid_frame = false;  // streaming header with a short last chunk (chunk.rs:76-79)
    sea_b200_header first = {};
};

// Resolve how many chunks/frames each stream yields: the host half of SeaDecoder::decode_frame (decoder.rs:33-59)
// and SeaFile::samples_from_reader (file.rs:180-209).
int plan_decode(sea_b200_ctx *ctx, uint32_t n_streams, const uint8_t *headers, size_t header_stride, const uint64_t *sea_offsets,
                const uint64_t *sea_lens, const uint64_t *pcm_offsets, const uint64_t *pcm_caps, DecodeJob *job)
{
    job->streams.resize(n_streams);
    job->n_samples.assign(n_streams, 0);
    uint64_t chain = 0;
    for (uint32_t i = 0; i < n_streams; i++) {
        sea_b200_header h;
        const uint64_t len = sea_lens[i];
        int rc = parse_file_header(headers + (size_t)i * header_stride, len < 22 ? len : 22, &h);
        if (rc) return fail(ctx, rc, "stream " + std::to_string(i) + ": bad .sea header (file.rs:40-72)");
        if (i == 0) job->first = h;
        if (h.channels != job->first.channels || h.chunk_size != job->first.chunk_size || h.frames_per_chunk != job->first.frames_per_chunk)
            job->uniform = false;
        DecStream &d = job->streams[i];
        memset(&d, 0, sizeof(d));
        d.data_off = sea_offsets[i] + kFileHeaderBytes;  // metadata bytes are never skipped by the reference (file.rs:53-54)
        d.data_len = len - kFileHeaderBytes;
        d.pcm_off = pcm_offsets[i];
        d.chunk_size = h.chunk_size;
        d.frames_per_chunk = h.frames_per_chunk;
        d.channels = h.channels;
        const uint64_t avail_chunks = (d.data_len + h.chunk_size - 1) / h.chunk_size;
        uint64_t frames;
        if (h.total_frames > 0) {
            const uint64_t want = ((uint64_t)h.total_frames + h.frames_per_chunk - 1) / h.frames_per_chunk;
            const uint64_t n = std::min(want, avail_chunks);  // read of 0 bytes ends the stream quietly (file.rs:186-188)
            d.n_chunks = (uint32_t)n;
            frames = std::min<uint64_t>(h.total_frames, n * h.frames_per_chunk);
        } else {
            uint64_t n = d.data_len / h.chunk_size;
            if (d.data_len % h.chunk_size) job->trailing_invalid_frame = true;
            d.n_chunks = (uint32_t)n;
            frames = n * h.frames_per_chunk;
            if (frames > 0xffffffffull) return fail(ctx, SEA_B200_ERR_TOO_MANY_FRAMES, "stream longer than 2^32 frames");
        }
        d.total_frames = (uint32_t)frames;
        const uint64_t samples = frames * h.channels;
        if (pcm_caps && samples > pcm_caps[i]) return fail(ctx, SEA_B200_ERR_CAPACITY, "stream " + std::to_string(i) + ": PCM buffer too small");
        job->n_samples[i] = samples;
        if (chain + (uint64_t)d.n_chunks * h.channels > 0xfffffff0ull) return fail(ctx, SEA_B200_ERR_INVALID_PARAMETERS, "batch too large (2^32 chains)");
        d.chain_begin = (uint32_t)chain;
        chain += (uint64_t)d.n_chunks * h.channels;
    }
    job->total_chains = chain;
    return SEA_B200_OK;
}

// The resources one decode launch sequence uses: lane 0 = the context's own stream and buffers, lane 1 = the auxiliary set.
struct DecLane {
    cudaStream_t stream, side;
    cudaEvent_t ev_fork, ev_join, ev0, ev1;
    DevBuf *in, *out, *table;
    int *d_err;
    double kernel_ms;
    // deferred mode (sea_b200_decode_batch's pipeline): the throughput routes leave their error word in *defer (pinned host memory,
    // valid once the stream has drained) instead of waiting for it, and time themselves with k0 / k1; `deferred` tells the caller
    int *defer = nullptr;
    cudaEvent_t k0 = nullptr, k1 = nullptr;
    bool deferred = false;
};
DecLane decode_lane(sea_b200_ctx *ctx, int i)
{
    if (i == 0) return {ctx->stream, ctx->side, ctx->ev_fork, ctx->ev_join, ctx->ev0, ctx->ev1, &ctx->in, &ctx->out, &ctx->streams, ctx->d_err, 0.0};
    return {ctx->aux.stream, ctx->aux.side, ctx->aux.ev_fork, ctx->aux.ev_join, ctx->aux.ev0, ctx->aux.ev1, &ctx->aux.in, &ctx->aux.out,
            &ctx->aux.table, ctx->aux.d_err, 0.0};
}

// d_sea / d_pcm are device pointers; first_hdr_word = first 4 bytes of the first chunk of stream 0 (host copy).
// copy_back / copy_back_bytes: when set and the job takes the small-job route, the PCM is sent to that host address in the same
// stream segment as the kernel and the error word (one synchronisation per call instead of two); *copied tells the caller.
int run_decode(sea_b200_ctx *ctx, DecLane &L, DecodeJob &job, const uint8_t *d_sea, uint64_t sea_len, int16_t *d_pcm, bool have_hdr_word,
               uint32_t hdr_word, int16_t *copy_back = nullptr, size_t copy_back_bytes = 0, bool *copied = nullptr)
{
    const uint32_t n_streams = (uint32_t)job.streams.size();
    if (job.total_chains == 0) return SEA_B200_OK;

    // ---- small jobs (the one-chunk seam, a few chunks per call, one short file): one warp per chunk, decode_latency.cu.  The
    // lane-per-chunk kernels below need tens of thousands of chunks to fill the GPU; under a few waves of warp-sized CTAs the
    // serial chain of a chunk is what the caller waits for.  SEA_B200_DEC_LATENCY = 0 / 1 pins the choice (tests, tuning).
    if (job.uniform) {
        const size_t smem_l = decode_latency_smem(job.first.chunk_size, job.first.frames_per_chunk, job.first.channels);
        const uint64_t chunks = job.total_chains / job.first.channels;
        bool latency = false;
        if (smem_l) {
            int sms = 148;
            cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device);
            const uint64_t per_sm = std::min<uint64_t>(32, (227u * 1024u) / (smem_l + 1024u));
            // measured crossover against the throughput kernels (profiles/r02_decode_route_probe.txt): ~2.5 waves of these CTAs,
            // stereo (2500 of 888 chunks per wave) and 8 channels (888 of 296) alike
            latency = chunks * 2u <= (uint64_t)sms * per_sm * 5u;
            if (const char *env = getenv("SEA_B200_DEC_LATENCY")) latency = env[0] == '1';
        }
        if (latency) {
            CU(L.table->reserve(sizeof(DecStream) * n_streams));
            CU(cudaMemcpyAsync(L.table->p, job.streams.data(), sizeof(DecStream) * n_streams, cudaMemcpyHostToDevice, L.stream));
            CU(cudaMemsetAsync(L.d_err, 0, sizeof(int), L.stream));
            CU(cudaEventRecord(L.ev0, L.stream));
            CU(launch_decode_latency(d_sea, d_pcm, L.table->as<DecStream>(), n_streams, chunks, job.first.chunk_size, job.first.frames_per_chunk,
                                     job.first.channels, ctx->tabs, L.d_err, L.stream));
            ctx->launches++;
            CU(cudaEventRecord(L.ev1, L.stream));
            int dev_err = 0;
            if (copy_back && copy_back_bytes) {  // speculative: worthless (and ignored by the caller) if the error word says so
                CU(cudaMemcpyAsync(copy_back, d_pcm, copy_back_bytes, cudaMemcpyDeviceToHost, L.stream));
                if (copied) *copied = true;
            }
            CU(cudaMemcpyAsync(&dev_err, L.d_err, sizeof(int), cudaMemcpyDeviceToHost, L.stream));
            CU(cudaStreamSynchronize(L.stream));
            float ms = 0;
            cudaEventElapsedTime(&ms, L.ev0, L.ev1);
            L.kernel_ms = ms;
            ctx->last_kernel_ms = ms;
            return map_dev_error(ctx, dev_err);
        }
    }

    DecFastParams fp = {};
    bool fast = false;
    if (job.uniform && have_hdr_word && (reinterpret_cast<uint64_t>(d_sea) & 15u) == 0) {
        fp.channels = job.first.channels;
        fp.N = job.first.frames_per_chunk;
        fp.chunk_size = job.first.chunk_size;
        fp.hdr_word = hdr_word;
        fp.s = (hdr_word >> 12) & 15u;
        fp.b = (hdr_word >> 8) & 15u;
        fp.F = (hdr_word >> 16) & 255u;
        fp.n_streams = n_streams;
        fp.total_chunks = job.total_chains / fp.channels;
        const uint32_t type = hdr_word & 255u;
        fast = (type == 1u || type == 2u) && (hdr_word >> 24) == 0x5Au && decode_fast_supported(fp);
    }
    // Descriptor table on the device: [0, n) every chunk of every stream; when the unrolled kernel applies, [n, 2n) the full
    // chunks it takes and [2n, 3n) what is left for the staged kernel (partial last chunks, chunks too close to the buffer end).
    std::vector<DecStream> table(job.streams);
    const bool use_vbr = fast && decode_vbr_supported(fp);  // the VBR twin of the unrolled kernel: same split, same constraints
    // more than two channels (CBR): one lane per chunk with all its channels, decode_mc.cuh; its left-overs go to the staged kernel
    // where that takes the channel count (3 / 5 / 7: `fast`), else to the generic one
    bool mc = fp.channels > 2 && (fp.hdr_word >> 24) == 0x5Au && decode_mc_supported(fp);
    bool unrolled = ((fast && (use_vbr || decode_unrolled_supported(fp))) || mc) && (reinterpret_cast<uint64_t>(d_pcm) & 31u) == 0;
    // The lane-per-chunk kernels do not look at data_len: every lane walks the layout its chunk header implies.  They therefore
    // only get chunks that are completely present, in streams whose header.chunk_size holds that layout (a crafted small
    // chunk_size -- file.rs:33-38 accepts >= 16 -- would otherwise let a lane read far past its chunk), and `extent` = the most
    // a lane can read from its chunk's first byte must lie inside the buffer.  Everything else goes to the staged / generic
    // kernels, which check every section against the bytes available (chunk.rs:81-196 slice bounds).
    uint64_t extent = 0;
    if (unrolled) {
        const uint64_t items = (uint64_t)(fp.N / fp.F) * fp.channels;
        const uint64_t res_rel = 4u + 16u * fp.channels + (items * fp.s + 7u) / 8u + (use_vbr ? (items * 2u + 7u) / 8u : 0u);
        if (use_vbr) {
            extent = res_rel + (uint64_t)fp.N * fp.channels + 320u;  // sizes are clamped to <= 8 bits per sample inside the kernel
            if (fp.chunk_size < res_rel) unrolled = false;
        } else {
            const uint64_t layout = res_rel + ((uint64_t)fp.N * fp.channels * fp.b + 7u) / 8u;
            extent = layout + (mc ? 512u : 128u);
            if (fp.chunk_size < layout) unrolled = false;
        }
    }
    uint64_t chains_a = 0, chains_b = 0;
    if (unrolled) {
        table.resize((size_t)3 * n_streams);
        for (uint32_t i = 0; i < n_streams && unrolled; i++) {
            const DecStream &d = job.streams[i];
            if (d.pcm_off % 16) unrolled = false;  // 256-bit stores need 32-byte aligned rows
            uint64_t n_full = std::min<uint64_t>(std::min<uint64_t>(d.total_frames / fp.N, d.n_chunks), d.data_len / fp.chunk_size);
            while (n_full > 0 && d.data_off + (n_full - 1u) * fp.chunk_size + extent > sea_len) n_full--;
            DecStream a = d, b = d;
            a.n_chunks = (uint32_t)n_full;
            a.total_frames = (uint32_t)(n_full * fp.N);
            a.chain_begin = (uint32_t)chains_a;
            chains_a += n_full * fp.channels;
            b.data_off += n_full * fp.chunk_size;
            b.data_len -= n_full * fp.chunk_size;
            b.pcm_off += n_full * fp.N * fp.channels;
            b.total_frames -= (uint32_t)(n_full * fp.N);
            b.n_chunks -= (uint32_t)n_full;
            b.chain_begin = (uint32_t)chains_b;
            chains_b += (uint64_t)b.n_chunks * fp.channels;
            table[(size_t)n_streams + i] = a;
            table[(size_t)2 * n_streams + i] = b;
        }
        if (chains_a == 0) unrolled = false;
    }
    if (!unrolled) mc = false;  // everything goes to the staged kernel (`fast`) or the generic one
    CU(L.table->reserve(sizeof(DecStream) * table.size()));
    CU(cudaMemcpyAsync(L.table->p, table.data(), sizeof(DecStream) * table.size(), cudaMemcpyHostToDevice, L.stream));
    CU(cudaMemsetAsync(L.d_err, 0, sizeof(int), L.stream));
    const DecStream *d_all = L.table->as<DecStream>();

    const bool defer = L.defer && (fast || mc);
    CU(cudaEventRecord(defer ? L.k0 : L.ev0, L.stream));
    int dev_err = 0;
    if (fast || mc) {
        if (unrolled) {
            DecFastParams fa = fp, fb = fp;
            fa.total_chunks = chains_a / fp.channels;
            fb.total_chunks = chains_b / fp.channels;
            // The left-over chunks (one partial chunk per stream: a short grid of long serial chains) go first, on the side
            // stream, so that their latency hides under the full-chunk kernel instead of trailing it.
            if (fb.total_chunks) {
                CU(cudaEventRecord(L.ev_fork, L.stream));
                CU(cudaStreamWaitEvent(L.side, L.ev_fork, 0));
                if (mc && !fast) CU(launch_decode_generic(d_sea, d_pcm, d_all + 2 * (size_t)n_streams, n_streams, chains_b, ctx->tabs, L.d_err, L.side));
                else CU(launch_decode_fast(d_sea, sea_len, d_pcm, d_all + 2 * (size_t)n_streams, fb, ctx->tabs, L.d_err, L.side));
                ctx->launches++;
                CU(cudaEventRecord(L.ev_join, L.side));
            }
            if (mc) CU(launch_decode_mc(d_sea, d_pcm, d_all + n_streams, fa, ctx->tabs, L.d_err, L.stream));
            else if (use_vbr) CU(launch_decode_vbr(d_sea, d_pcm, d_all + n_streams, fa, ctx->tabs, L.d_err, L.stream));
            else CU(launch_decode_unrolled(d_sea, d_pcm, d_all + n_streams, fa, ctx->tabs, L.d_err, L.stream));
            ctx->launches++;
            if (fb.total_chunks) CU(cudaStreamWaitEvent(L.stream, L.ev_join, 0));
        } else {
            CU(launch_decode_fast(d_sea, sea_len, d_pcm, d_all, fp, ctx->tabs, L.d_err, L.stream));
            ctx->launches++;
        }
        if (defer) {  // the caller reads the word after its last group (and redoes this one if it is not kDevOk)
            CU(cudaEventRecord(L.k1, L.stream));
            CU(cudaMemcpyAsync(L.defer, L.d_err, sizeof(int), cudaMemcpyDeviceToHost, L.stream));
            L.deferred = true;
            L.kernel_ms = 0.0;
            return SEA_B200_OK;
        }
        CU(cudaMemcpyAsync(&dev_err, L.d_err, sizeof(int), cudaMemcpyDeviceToHost, L.stream));
        CU(cudaStreamSynchronize(L.stream));
        if (dev_err != kDevOk) {  // some chunk is not what the fast path was specialised for: redo everything generically
            fast = false;
            mc = false;
            CU(cudaMemsetAsync(L.d_err, 0, sizeof(int), L.stream));
        }
    }
    if (!fast && !mc) {
        CU(launch_decode_generic(d_sea, d_pcm, d_all, n_streams, job.total_chains, ctx->tabs, L.d_err, L.stream));
        ctx->launches++;
        CU(cudaMemcpyAsync(&dev_err, L.d_err, sizeof(int), cudaMemcpyDeviceToHost, L.stream));
    }
    CU(cudaEventRecord(L.ev1, L.stream));
    CU(cudaStreamSynchronize(L.stream));
    float ms = 0;
    cudaEventElapsedTime(&ms, L.ev0, L.ev1);
    L.kernel_ms = ms;
    ctx->last_kernel_ms = ms;
    return map_dev_error(ctx, dev_err);
}

// ------------------------------------------------------------------------------------------------ encode core

struct EncodeJob {
    EncodePlan plan;
    EncParams params;
    std::vector<EncStream> streams;
    uint32_t chunk_buf_bytes;  // the largest chunk these streams can produce (launch_encode_generic)
};

int plan_encode(sea_b200_ctx *ctx, uint32_t n_streams, const uint64_t *pcm_offsets, const uint32_t *n_frames, uint32_t sample_rate,
                uint32_t channels, const sea_b200_settings *st, const uint64_t *out_offsets, bool raw_chunk_mode, EncodeJob *job)
{
    int rc = make_encode_plan(channels, st, &job->plan);
    if (rc) return fail(ctx, rc, "encoder settings rejected (outside the reference's domain)");
    const EncodePlan &pl = job->plan;
    EncParams &p = job->params;
    memset(&p, 0, sizeof(p));
    p.channels = channels;
    p.N = pl.N;
    p.F = pl.F;
    p.s = pl.s;
    p.hdr_bits = pl.hdr_bits;
    p.vbr = pl.vbr;
    p.base = pl.base;
    p.full_counts[0] = pl.full_counts[0];
    p.full_counts[1] = pl.full_counts[2];
    p.full_counts[2] = pl.full_counts[3];
    p.full_chunk_bytes = pl.full_chunk_bytes;
    p.max_chunk_bytes = pl.max_chunk_bytes;
    p.sample_rate = sample_rate;
    p.raw_chunk_mode = raw_chunk_mode;
    p.n_streams = n_streams;
    job->streams.resize(n_streams);
    bool any_full = false;
    // CBR: every chunk of a job fits max_chunk_bytes exactly.  VBR: a full chunk is full_chunk_bytes exactly; a last chunk of `last`
    // frames is bounded by its own bucket counts with every block taken at F frames (the items past `sortable` keep size `base`)
    // and by `last` frames at base+2 bits.
    job->chunk_buf_bytes = pl.vbr ? 0u : pl.max_chunk_bytes;
    for (uint32_t i = 0; i < n_streams; i++) {
        EncStream &e = job->streams[i];
        memset(&e, 0, sizeof(e));
        e.pcm_off = pcm_offsets[i];
        e.out_off = out_offsets[i];
        e.n_frames = n_frames[i];
        if (n_frames[i] >= pl.N) any_full = true;
        const uint32_t last = n_frames[i] % pl.N;
        if (pl.vbr && last) {
            uint64_t counts[4];
            const uint64_t sortable = ((uint64_t)last * channels) / pl.F;  // trap T14
            vbr_distribution(sortable, pl.vbr_target, counts);
            e.last_counts[0] = (uint32_t)counts[0];
            e.last_counts[1] = (uint32_t)counts[2];
            e.last_counts[2] = (uint32_t)counts[3];
            if ((counts[0] && pl.base < 2) || (counts[2] && pl.base + 1 > 8) || (counts[3] && pl.base + 2 > 8))
                return fail(ctx, SEA_B200_ERR_DOMAIN, "VBR bitrate produces a residual size outside 1..8 (common.rs:34 panics)");
            const uint64_t items = ((uint64_t)last + pl.F - 1) / pl.F * channels;
            const uint64_t size_sum = counts[0] * (pl.base - 1) + (counts[1] + items - sortable) * pl.base + counts[2] * (pl.base + 1) +
                                      counts[3] * (pl.base + 2);
            const uint64_t bits = std::min<uint64_t>(size_sum * pl.F, (uint64_t)last * channels * (pl.base + 2));
            const uint64_t bytes = 4 + 16ull * channels + (items * pl.s + 7) / 8 + (items * 2 + 7) / 8 + (bits + 7) / 8;
            job->chunk_buf_bytes = std::max<uint32_t>(job->chunk_buf_bytes, (uint32_t)std::min<uint64_t>(bytes, pl.max_chunk_bytes));
        }
    }
    if (pl.vbr && any_full) job->chunk_buf_bytes = std::max(job->chunk_buf_bytes, pl.full_chunk_bytes);
    if (any_full && !pl.full_chunk_valid)
        return fail(ctx, SEA_B200_ERR_DOMAIN, "VBR bitrate produces a residual size outside 1..8 (common.rs:34 panics)");
    return SEA_B200_OK;
}

// One encode launch on the context's stream, nothing waited for: `slot` selects which n-entry region of the descriptor / length /
// first-chunk arrays the launch uses (the time-sliced batch encode keeps one per slice and reads them all back at the end).
// The error word and the tie counters are NOT reset here: they accumulate over the launches of one call.
int enqueue_encode(sea_b200_ctx *ctx, EncodeJob &job, const int16_t *d_pcm, uint8_t *d_out, int32_t *d_state, uint32_t slot,
                   bool descriptors_uploaded)
{
    const uint32_t n = job.params.n_streams;
    EncWorkspace ws = {};
    ws.vbr_scratch_stride = enc_vbr_scratch_bytes(job.params);
    if (ws.vbr_scratch_stride) {
        CU(ctx->scratch.reserve(ws.vbr_scratch_stride * n));
        ws.vbr_scratch = ctx->scratch.as<uint8_t>();
    }
    EncStream *d_streams = ctx->streams.as<EncStream>() + (size_t)slot * n;
    if (!descriptors_uploaded)
        CU(cudaMemcpyAsync(d_streams, job.streams.data(), sizeof(EncStream) * n, cudaMemcpyHostToDevice, ctx->stream));
    CU(launch_encode_generic(d_pcm, d_out, d_streams, job.params, ctx->tabs, d_state, ctx->lens.as<uint64_t>() + (size_t)slot * n,
                             ctx->chunk0.as<uint32_t>() + (size_t)slot * n, ctx->ties.as<unsigned long long>(), ws, ctx->d_err, ctx->stream,
                             job.chunk_buf_bytes));
    ctx->launches++;
    return SEA_B200_OK;
}

int run_encode(sea_b200_ctx *ctx, EncodeJob &job, const int16_t *d_pcm, uint8_t *d_out, int32_t *d_state, uint64_t *h_out_lens,
               uint32_t *h_chunk0)
{
    const uint32_t n = job.params.n_streams;
    if (n == 0) return SEA_B200_OK;
    CU(ctx->streams.reserve(sizeof(EncStream) * n));
    CU(ctx->lens.reserve(sizeof(uint64_t) * n));
    CU(ctx->chunk0.reserve(sizeof(uint32_t) * n));
    EncWorkspace ws = {};
    ws.vbr_scratch_stride = enc_vbr_scratch_bytes(job.params);
    if (ws.vbr_scratch_stride) {
        CU(ctx->scratch.reserve(ws.vbr_scratch_stride * n));
        ws.vbr_scratch = ctx->scratch.as<uint8_t>();
    }
    CU(cudaMemcpyAsync(ctx->streams.p, job.streams.data(), sizeof(EncStream) * n, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemsetAsync(ctx->d_err, 0, sizeof(int), ctx->stream));
    CU(ctx->ties.reserve(sizeof(unsigned long long) * ((size_t)n + 1u)));
    CU(cudaMemsetAsync(ctx->ties.p, 0, sizeof(unsigned long long) * ((size_t)n + 1u), ctx->stream));
    ctx->h_ties.assign((size_t)n + 1u, 0ull);
    CU(cudaEventRecord(ctx->ev0, ctx->stream));
    CU(launch_encode_generic(d_pcm, d_out, ctx->streams.as<EncStream>(), job.params, ctx->tabs, d_state, ctx->lens.as<uint64_t>(),
                             ctx->chunk0.as<uint32_t>(), ctx->ties.as<unsigned long long>(), ws, ctx->d_err, ctx->stream, job.chunk_buf_bytes));
    ctx->launches++;
    CU(cudaEventRecord(ctx->ev1, ctx->stream));
    int dev_err = 0;
    CU(cudaMemcpyAsync(&dev_err, ctx->d_err, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    if (job.params.vbr)
        CU(cudaMemcpyAsync(ctx->h_ties.data(), ctx->ties.p, sizeof(unsigned long long) * ((size_t)n + 1u), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaMemcpyAsync(h_out_lens, ctx->lens.p, sizeof(uint64_t) * n, cudaMemcpyDeviceToHost, ctx->stream));
    if (h_chunk0) CU(cudaMemcpyAsync(h_chunk0, ctx->chunk0.p, sizeof(uint32_t) * n, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    float ms = 0;
    cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1);
    ctx->last_kernel_ms = ms;
    ctx->last_ties = ctx->h_ties[0];
    return map_dev_error(ctx, dev_err);
}

// Half-open ranges of a caller buffer that a batch call owns; sorted and coalesced so that one copy serves each run of
// adjacent streams and nothing outside an owned range is ever written.
struct Run {
    uint64_t lo, hi;
};
void merge_runs(std::vector<Run> &runs)
{
    std::sort(runs.begin(), runs.end(), [](const Run &a, const Run &b) { return a.lo < b.lo; });
    size_t n = 0;
    for (const Run &r : runs) {
        if (n && r.lo <= runs[n - 1].hi) runs[n - 1].hi = std::max(runs[n - 1].hi, r.hi);
        else runs[n++] = r;
    }
    runs.resize(n);
}

uint64_t encode_bound_bytes(const EncodePlan &pl, uint64_t n_frames)
{
    const uint64_t full = n_frames / pl.N, rem = n_frames % pl.N;
    uint64_t bytes = kFileHeaderBytes + full * pl.full_chunk_bytes;
    if (rem) {
        const uint64_t items = (rem + pl.F - 1) / pl.F * pl.channels;
        const uint64_t bits = pl.vbr ? pl.base + 2 : pl.hdr_bits;
        bytes += 4 + 16ull * pl.channels + (items * pl.s + 7) / 8 + (pl.vbr ? (items * 2 + 7) / 8 : 0) + (rem * pl.channels * bits + 7) / 8;
    }
    return bytes;
}

// ---- time-sliced host-buffer encode --------------------------------------------------------------------------------------------
// An encoder stream is serial (LMS + prev_scalefactor carry over, encoder_base.rs:181-182), so a batch cannot be pipelined by
// stream groups without starving the kernel of parallel streams.  It is cut in TIME instead: a slice = `K` chunks of every stream;
// slice j+1 is uploaded while slice j is encoded (the per-stream state stays on the device between the launches, exactly like a
// streaming handle's make_chunks) and slice j-1 is downloaded.  Returns 1 when slicing does not apply (short or tiny batches).
int encode_batch_sliced(sea_b200_ctx *ctx, uint32_t n, const int16_t *pcm, const uint64_t *pcm_offsets, const uint32_t *n_frames,
                        uint32_t sample_rate, uint32_t channels, const sea_b200_settings *settings, const EncodePlan &pl, uint8_t *out,
                        const uint64_t *out_offsets, uint64_t *out_lens)
{
    uint64_t forced = 0;  // SEA_B200_ENC_SLICE: 0 = never slice, k > 0 = slices of k chunks whatever the batch size (tests, tuning)
    if (const char *env = getenv("SEA_B200_ENC_SLICE")) {
        if (env[0] == '0') return 1;
        forced = (uint64_t)atoll(env);
    }
    uint64_t max_frames = 0, total_samples = 0;
    for (uint32_t i = 0; i < n; i++) {
        max_frames = std::max<uint64_t>(max_frames, n_frames[i]);
        total_samples += (uint64_t)n_frames[i] * channels;
    }
    if (!forced && total_samples < (32ull << 20)) return 1;
    const uint64_t chunk_samples = (uint64_t)pl.N * channels;
    uint64_t K = (512ull << 20) / std::max<uint64_t>(1, (uint64_t)n * chunk_samples);  // ~1 GB of PCM per slice
    K = forced ? forced : std::min<uint64_t>(std::max<uint64_t>(K, 4), 1024);
    const uint64_t slice_frames = K * pl.N, S = (max_frames + slice_frames - 1) / slice_frames;
    if (S < (forced ? 2u : 3u)) return 1;
    const uint64_t slice_samples = slice_frames * channels, out_region = K * (uint64_t)pl.max_chunk_bytes;

    // regular layouts (equal lengths, equal strides) move a slice with one 2-D copy each way
    bool regular = n > 1;
    const uint64_t pstride = n > 1 ? pcm_offsets[1] - pcm_offsets[0] : 0, ostride = n > 1 ? out_offsets[1] - out_offsets[0] : 0;
    for (uint32_t i = 1; i < n && regular; i++)
        regular = n_frames[i] == n_frames[0] && pcm_offsets[i] == pcm_offsets[0] + i * pstride && out_offsets[i] == out_offsets[0] + i * ostride &&
                  pcm_offsets[1] > pcm_offsets[0] && out_offsets[1] > out_offsets[0];
    if (regular && (pstride < (uint64_t)n_frames[0] * channels || ostride < encode_bound_bytes(pl, n_frames[0]))) regular = false;

    cudaStream_t comp = ctx->stream, up = ctx->aux.stream, down = ctx->aux.side;
    for (int b = 0; b < 2; b++) {
        if (!ctx->pipe.up[b]) CU(cudaEventCreateWithFlags(&ctx->pipe.up[b], cudaEventDisableTiming));
        if (!ctx->pipe.kern[b]) CU(cudaEventCreateWithFlags(&ctx->pipe.kern[b], cudaEventDisableTiming));
        if (!ctx->pipe.down[b]) CU(cudaEventCreateWithFlags(&ctx->pipe.down[b], cudaEventDisableTiming));
        CU(ctx->pipe.in[b].reserve((uint64_t)n * slice_samples * 2 + 64));
        CU(ctx->pipe.out[b].reserve((uint64_t)n * out_region + 64));
    }
    CU(ctx->streams.reserve(sizeof(EncStream) * n * S));
    CU(ctx->lens.reserve(sizeof(uint64_t) * n * S));
    CU(ctx->chunk0.reserve(sizeof(uint32_t) * n * S));
    CU(ctx->ties.reserve(sizeof(unsigned long long) * ((size_t)n + 1u)));
    {   // EncoderBase::new for every stream (encoder_base.rs:29-41, lms.rs:19-32)
        std::vector<int32_t> init((size_t)n * channels * kEncStateWords, 0);
        for (size_t c = 0; c < (size_t)n * channels; c++) {
            init[c * kEncStateWords + 4 + 2] = -(1 << 13);
            init[c * kEncStateWords + 4 + 3] = 1 << 14;
        }
        CU(ctx->pipe.state.reserve(init.size() * sizeof(int32_t)));
        CU(cudaMemcpyAsync(ctx->pipe.state.p, init.data(), init.size() * sizeof(int32_t), cudaMemcpyHostToDevice, comp));
    }
    CU(cudaMemsetAsync(ctx->d_err, 0, sizeof(int), comp));
    CU(cudaMemsetAsync(ctx->ties.p, 0, sizeof(unsigned long long) * ((size_t)n + 1u), comp));
    ctx->h_ties.assign((size_t)n + 1u, 0ull);
    // every slice's launch descriptors, planned and uploaded up front (a pageable upload inside the loop would make the host
    // wait for the previous kernel before it could queue the next copies)
    std::vector<EncodeJob> jobs(S);
    std::vector<uint32_t> all_frames((size_t)S * n);
    {
        std::vector<uint64_t> o_pcm(n), o_out(n);
        std::vector<EncStream> all((size_t)S * n);
        for (uint32_t i = 0; i < n; i++) {
            o_pcm[i] = (uint64_t)i * slice_samples;
            o_out[i] = (uint64_t)i * out_region;
        }
        for (uint64_t j = 0; j < S; j++) {
            uint32_t *fr = all_frames.data() + (size_t)j * n;
            for (uint32_t i = 0; i < n; i++) {
                const uint64_t done = std::min<uint64_t>(n_frames[i], j * slice_frames);
                fr[i] = (uint32_t)std::min<uint64_t>(slice_frames, n_frames[i] - done);
            }
            int prc = plan_encode(ctx, n, o_pcm.data(), fr, sample_rate, channels, settings, o_out.data(), true, &jobs[j]);
            if (prc) return prc;
            std::copy(jobs[j].streams.begin(), jobs[j].streams.end(), all.begin() + (size_t)j * n);
        }
        CU(cudaMemcpyAsync(ctx->streams.p, all.data(), sizeof(EncStream) * all.size(), cudaMemcpyHostToDevice, comp));
    }
    CU(cudaEventRecord(ctx->ev0, comp));
    CU(cudaEventRecord(ctx->pipe.kern[0], comp));  // orders the side streams behind whatever the caller queued on the context's stream
    CU(cudaStreamWaitEvent(up, ctx->pipe.kern[0], 0));
    CU(cudaStreamWaitEvent(down, ctx->pipe.kern[0], 0));

    std::vector<uint64_t> lens_j(n);
    for (uint32_t i = 0; i < n; i++) out_lens[i] = kFileHeaderBytes;
    int rc = SEA_B200_OK;
    for (uint64_t j = 0; j < S && rc == SEA_B200_OK; j++) {
        const int b = (int)(j & 1);
        bool vbr_tail = false;
        const uint32_t *s_frames = all_frames.data() + (size_t)j * n;
        for (uint32_t i = 0; i < n; i++)
            if (pl.vbr && s_frames[i] % pl.N) vbr_tail = true;
        // ---- upload (waits until the kernel that last read this buffer is done)
        if (j >= 2) CU(cudaStreamWaitEvent(up, ctx->pipe.kern[b], 0));
        int16_t *d_in = ctx->pipe.in[b].as<int16_t>();
        if (regular && s_frames[0]) {
            CU(cudaMemcpy2DAsync(d_in, slice_samples * 2, pcm + pcm_offsets[0] + j * slice_samples, pstride * 2, (size_t)s_frames[0] * channels * 2, n,
                                 cudaMemcpyHostToDevice, up));
        } else if (!regular) {
            for (uint32_t i = 0; i < n; i++)
                if (s_frames[i])
                    CU(cudaMemcpyAsync(d_in + (uint64_t)i * slice_samples, pcm + pcm_offsets[i] + j * slice_samples,
                                       (size_t)s_frames[i] * channels * 2, cudaMemcpyHostToDevice, up));
        }
        CU(cudaEventRecord(ctx->pipe.up[b], up));
        // ---- kernel (waits for the upload, and for the download that last read this output buffer)
        CU(cudaStreamWaitEvent(comp, ctx->pipe.up[b], 0));
        if (j >= 2) CU(cudaStreamWaitEvent(comp, ctx->pipe.down[b], 0));
        rc = enqueue_encode(ctx, jobs[j], d_in, ctx->pipe.out[b].as<uint8_t>(), ctx->pipe.state.as<int32_t>(), (uint32_t)j, true);
        if (rc) break;
        CU(cudaEventRecord(ctx->pipe.kern[b], comp));
        // ---- lengths of this slice's output per stream.  Full chunks have the plan's size (CBR and VBR alike, encoder_vbr.rs:66-96
        // gives constant bucket counts); a CBR partial chunk follows from the frame count; a VBR partial chunk has to be read back.
        if (vbr_tail) {
            CU(cudaMemcpyAsync(lens_j.data(), ctx->lens.as<uint64_t>() + (size_t)j * n, sizeof(uint64_t) * n, cudaMemcpyDeviceToHost, comp));
            CU(cudaStreamSynchronize(comp));
        } else {
            for (uint32_t i = 0; i < n; i++) {
                const uint32_t full = s_frames[i] / pl.N, rem = s_frames[i] % pl.N;
                lens_j[i] = (uint64_t)full * pl.full_chunk_bytes + (rem ? cbr_chunk_bytes(rem, channels, pl.s, pl.F, pl.hdr_bits) : 0u);
            }
        }
        // ---- download into the ranges the streams own
        CU(cudaStreamWaitEvent(down, ctx->pipe.kern[b], 0));
        const uint8_t *d_o = ctx->pipe.out[b].as<uint8_t>();
        const uint64_t file_off = kFileHeaderBytes + j * K * (uint64_t)pl.full_chunk_bytes;
        bool same_len = regular;
        for (uint32_t i = 1; i < n && same_len; i++) same_len = lens_j[i] == lens_j[0];
        if (same_len && lens_j[0]) {
            CU(cudaMemcpy2DAsync(out + out_offsets[0] + file_off, ostride, d_o, out_region, lens_j[0], n, cudaMemcpyDeviceToHost, down));
        } else if (!same_len) {
            for (uint32_t i = 0; i < n; i++)
                if (lens_j[i]) CU(cudaMemcpyAsync(out + out_offsets[i] + file_off, d_o + (uint64_t)i * out_region, lens_j[i], cudaMemcpyDeviceToHost, down));
        }
        CU(cudaEventRecord(ctx->pipe.down[b], down));
        for (uint32_t i = 0; i < n; i++) out_lens[i] += lens_j[i];
    }
    CU(cudaEventRecord(ctx->ev1, comp));
    int dev_err = 0;
    CU(cudaMemcpyAsync(&dev_err, ctx->d_err, sizeof(int), cudaMemcpyDeviceToHost, comp));
    if (pl.vbr) CU(cudaMemcpyAsync(ctx->h_ties.data(), ctx->ties.p, sizeof(unsigned long long) * ((size_t)n + 1u), cudaMemcpyDeviceToHost, comp));
    CU(cudaStreamSynchronize(comp));
    CU(cudaStreamSynchronize(up));
    CU(cudaStreamSynchronize(down));
    if (rc) return rc;
    float ms = 0;
    cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1);
    ctx->last_kernel_ms = ms;  // first launch to last, uploads the kernels waited for included
    ctx->last_ties = ctx->h_ties[0];
    if ((rc = map_dev_error(ctx, dev_err)) != SEA_B200_OK) return rc;
    // file headers (file.rs:78-93): chunk_size = the first chunk's size (file.rs:166-168, `as u16`), written by the host
    for (uint32_t i = 0; i < n; i++) {
        const uint64_t first = n_frames[i] >= pl.N ? pl.full_chunk_bytes : out_lens[i] - kFileHeaderBytes;
        write_file_header(out + out_offsets[i], (uint8_t)channels, (uint16_t)first, (uint16_t)pl.N, sample_rate, n_frames[i]);
    }
    return SEA_B200_OK;
}

}  // namespace

// =================================================================================================== C-ABI

extern "C" {

int sea_b200_abi_version(void) { return SEA_B200_ABI_VERSION; }

const char *sea_b200_strerror(int status)
{
    switch (status) {
        case SEA_B200_OK: return "ok";
        case SEA_B200_ERR_READ: return "ReadError";
        case SEA_B200_ERR_INVALID_PARAMETERS: return "InvalidParameters";
        case SEA_B200_ERR_INVALID_FILE: return "InvalidFile";
        case SEA_B200_ERR_INVALID_FRAME: return "InvalidFrame";
        case SEA_B200_ERR_ENCODER_CLOSED: return "EncoderClosed";
        case SEA_B200_ERR_UNSUPPORTED_VERSION: return "UnsupportedVersion";
        case SEA_B200_ERR_TOO_MANY_FRAMES: return "TooManyFrames";
        case SEA_B200_ERR_METADATA_TOO_LARGE: return "MetadataTooLarge";
        case SEA_B200_ERR_IO: return "IoError";
        case SEA_B200_ERR_CAPACITY: return "output buffer too small";
        case SEA_B200_ERR_DOMAIN: return "input outside the reference's domain (the reference panics)";
        case SEA_B200_ERR_CUDA: return "CUDA failure";
        case SEA_B200_ERR_NOMEM: return "out of device memory";
        default: return "unknown";
    }
}

int sea_b200_ctx_create(int device, sea_b200_ctx **out)
{
    if (!out) return SEA_B200_ERR_INVALID_PARAMETERS;
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0 || device < 0 || device >= count) return SEA_B200_ERR_CUDA;
    if (cudaSetDevice(device) != cudaSuccess) return SEA_B200_ERR_CUDA;
    sea_b200_ctx *ctx = new sea_b200_ctx();
    ctx->device = device;
    auto bail = [&](cudaError_t) {
        sea_b200_ctx_destroy(ctx);
        return SEA_B200_ERR_CUDA;
    };
    cudaError_t e;
    if ((e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking)) != cudaSuccess) return bail(e);
    ctx->own_stream = true;
    {   // highest priority: its few long-running CTAs must be placed as soon as an SM frees up, not after the big grid drains
        int prio_lo = 0, prio_hi = 0;
        if ((e = cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi)) != cudaSuccess) return bail(e);
        if ((e = cudaStreamCreateWithPriority(&ctx->side, cudaStreamNonBlocking, prio_hi)) != cudaSuccess) return bail(e);
    }
    if ((e = cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming)) != cudaSuccess) return bail(e);
    if ((e = cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming)) != cudaSuccess) return bail(e);
    {   // auxiliary decode lane
        int prio_lo = 0, prio_hi = 0;
        cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
        if ((e = cudaStreamCreateWithFlags(&ctx->aux.stream, cudaStreamNonBlocking)) != cudaSuccess) return bail(e);
        if ((e = cudaStreamCreateWithPriority(&ctx->aux.side, cudaStreamNonBlocking, prio_hi)) != cudaSuccess) return bail(e);
        if ((e = cudaEventCreateWithFlags(&ctx->aux.ev_fork, cudaEventDisableTiming)) != cudaSuccess) return bail(e);
        if ((e = cudaEventCreateWithFlags(&ctx->aux.ev_join, cudaEventDisableTiming)) != cudaSuccess) return bail(e);
        if ((e = cudaEventCreate(&ctx->aux.ev0)) != cudaSuccess) return bail(e);
        if ((e = cudaEventCreate(&ctx->aux.ev1)) != cudaSuccess) return bail(e);
        if ((e = cudaMalloc(&ctx->aux.d_err, sizeof(int))) != cudaSuccess) return bail(e);
    }
    if ((e = cudaEventCreate(&ctx->ev0)) != cudaSuccess) return bail(e);
    if ((e = cudaEventCreate(&ctx->ev1)) != cudaSuccess) return bail(e);
    if ((e = cudaMalloc(&ctx->d_err, sizeof(int))) != cudaSuccess) return bail(e);
    for (uint32_t s = 1; s <= 8; s++) {  // SeaDequantTab::init for every scale_factor_bits a chunk header can name
        std::vector<int32_t> t = build_tables(s);
        if ((e = cudaMalloc(&ctx->d_tab[s], t.size() * sizeof(int32_t))) != cudaSuccess) return bail(e);
        if ((e = cudaMemcpy(ctx->d_tab[s], t.data(), t.size() * sizeof(int32_t), cudaMemcpyHostToDevice)) != cudaSuccess) return bail(e);
        ctx->tabs.by_s[s] = ctx->d_tab[s];
    }
    ctx->tabs.by_s[0] = nullptr;
    *out = ctx;
    return SEA_B200_OK;
}

void sea_b200_ctx_destroy(sea_b200_ctx *ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    for (int s = 0; s < 9; s++)
        if (ctx->d_tab[s]) cudaFree(ctx->d_tab[s]);
    ctx->in.release();
    ctx->out.release();
    ctx->streams.release();
    ctx->lens.release();
    ctx->chunk0.release();
    ctx->scratch.release();
    ctx->misc.release();
    if (ctx->d_err) cudaFree(ctx->d_err);
    ctx->ties.release();
    for (int i = 0; i < 2; i++) {
        if (ctx->pipe.up[i]) cudaEventDestroy(ctx->pipe.up[i]);
        if (ctx->pipe.kern[i]) cudaEventDestroy(ctx->pipe.kern[i]);
        if (ctx->pipe.down[i]) cudaEventDestroy(ctx->pipe.down[i]);
        ctx->pipe.in[i].release();
        ctx->pipe.out[i].release();
    }
    ctx->pipe.state.release();
    ctx->win.release();
    ctx->win_desc.release();
    if (ctx->aux.stream) { cudaStreamSynchronize(ctx->aux.stream); cudaStreamDestroy(ctx->aux.stream); }
    if (ctx->aux.side) { cudaStreamSynchronize(ctx->aux.side); cudaStreamDestroy(ctx->aux.side); }
    if (ctx->aux.ev_fork) cudaEventDestroy(ctx->aux.ev_fork);
    if (ctx->aux.ev_join) cudaEventDestroy(ctx->aux.ev_join);
    if (ctx->aux.ev0) cudaEventDestroy(ctx->aux.ev0);
    if (ctx->aux.ev1) cudaEventDestroy(ctx->aux.ev1);
    if (ctx->aux.d_err) cudaFree(ctx->aux.d_err);
    if (ctx->h_errs) cudaFreeHost(ctx->h_errs);
    if (ctx->up) { cudaStreamSynchronize(ctx->up); cudaStreamDestroy(ctx->up); }
    for (cudaEvent_t e : ctx->grp_ev) cudaEventDestroy(e);
    ctx->aux.in.release();
    ctx->aux.out.release();
    ctx->aux.table.release();
    if (ctx->side) { cudaStreamSynchronize(ctx->side); cudaStreamDestroy(ctx->side); }
    if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
    if (ctx->ev_join) cudaEventDestroy(ctx->ev_join);
    if (ctx->ev0) cudaEventDestroy(ctx->ev0);
    if (ctx->ev1) cudaEventDestroy(ctx->ev1);
    if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

int sea_b200_ctx_set_stream(sea_b200_ctx *ctx, void *cuda_stream)
{
    if (!ctx) return SEA_B200_ERR_INVALID_PARAMETERS;
    if (ctx->own_stream && ctx->stream) {
        cudaStreamSynchronize(ctx->stream);
        cudaStreamDestroy(ctx->stream);
    }
    ctx->stream = reinterpret_cast<cudaStream_t>(cuda_stream);
    ctx->own_stream = false;
    return SEA_B200_OK;
}

void *sea_b200_ctx_stream(const sea_b200_ctx *ctx) { return ctx ? reinterpret_cast<void *>(ctx->stream) : nullptr; }
const char *sea_b200_last_error(const sea_b200_ctx *ctx) { return ctx ? ctx->last_error.c_str() : ""; }
uint64_t sea_b200_ctx_launch_count(const sea_b200_ctx *ctx) { return ctx ? ctx->launches : 0; }
double sea_b200_last_kernel_ms(const sea_b200_ctx *ctx) { return ctx ? ctx->last_kernel_ms : 0.0; }
uint64_t sea_b200_last_vbr_ties(const sea_b200_ctx *ctx) { return ctx ? ctx->last_ties : 0; }
int sea_b200_last_vbr_ties_per_stream(const sea_b200_ctx *ctx, uint64_t *ties, uint32_t n_streams)
{
    if (!ctx || !ties) return SEA_B200_ERR_INVALID_PARAMETERS;
    for (uint32_t i = 0; i < n_streams; i++) ties[i] = (size_t)i + 1u < ctx->h_ties.size() ? ctx->h_ties[(size_t)i + 1u] : 0u;
    return SEA_B200_OK;
}

void *sea_b200_host_alloc(size_t bytes)
{
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) return nullptr;
    return p;
}
void sea_b200_host_free(void *p)
{
    if (p) cudaFreeHost(p);
}

void sea_b200_default_settings(sea_b200_settings *s)
{
    memset(s, 0, sizeof(*s));
    s->frames_per_chunk = 5120;
    s->scale_factor_bits = 4;
    s->scale_factor_frames = 20;
    s->residual_bits = 3.0f;
    s->vbr = 0;
}

int sea_b200_parse_header(const uint8_t *sea, uint64_t len, sea_b200_header *out)
{
    if (!sea || !out) return SEA_B200_ERR_INVALID_PARAMETERS;
    return parse_file_header(sea, len, out);
}

int sea_b200_encode_bound(uint64_t n_frames, uint32_t channels, const sea_b200_settings *s, uint64_t *bytes)
{
    EncodePlan pl;
    int rc = make_encode_plan(channels, s, &pl);
    if (rc) return rc;
    *bytes = encode_bound_bytes(pl, n_frames);
    return SEA_B200_OK;
}

int sea_b200_full_chunk_bytes(uint32_t channels, const sea_b200_settings *s, uint32_t *bytes)
{
    EncodePlan pl;
    int rc = make_encode_plan(channels, s, &pl);
    if (rc) return rc;
    if (!pl.full_chunk_valid) return SEA_B200_ERR_DOMAIN;
    *bytes = pl.full_chunk_bytes;
    return SEA_B200_OK;
}

int sea_b200_vbr_plan(const sea_b200_settings *s, uint64_t sortable_items, float *target, uint32_t *base, uint64_t counts[4])
{
    if (!s || s->frames_per_chunk == 0 || s->scale_factor_frames == 0) return SEA_B200_ERR_INVALID_PARAMETERS;
    const float t = vbr_normalized_bitrate(s);
    if (target) *target = t;
    if (base) *base = !(t > 0.0f) ? 0u : (t >= 255.0f ? 255u : (uint32_t)t);
    if (counts) vbr_distribution(sortable_items, t, counts);
    return SEA_B200_OK;
}

int sea_b200_tables(uint32_t residual_bits, uint32_t scale_factor_bits, int32_t *recip, int32_t *dqt)
{
    if (residual_bits < 1 || residual_bits > 8 || scale_factor_bits < 1 || scale_factor_bits > 8) return SEA_B200_ERR_INVALID_PARAMETERS;
    std::vector<int32_t> t = build_tables(scale_factor_bits);
    const uint32_t n = 1u << scale_factor_bits;
    if (recip) memcpy(recip, t.data() + tab_recip_off(scale_factor_bits, residual_bits), n * sizeof(int32_t));
    if (dqt) memcpy(dqt, t.data() + tab_dqt_off(scale_factor_bits, residual_bits), ((size_t)n << residual_bits) * sizeof(int32_t));
    return SEA_B200_OK;
}

// ------------------------------------------------------------------------------------------------ decode entry points

int sea_b200_decode_batch_device(sea_b200_ctx *ctx, uint32_t n_streams, const uint8_t *d_sea, const uint64_t *sea_offsets,
                                 const uint64_t *sea_lens, const uint8_t *headers, int16_t *d_pcm, const uint64_t *pcm_offsets,
                                 const uint64_t *pcm_caps, uint64_t *n_samples)
{
    if (!ctx || !sea_offsets || !sea_lens || !headers || !pcm_offsets) return SEA_B200_ERR_INVALID_PARAMETERS;
    if (n_streams == 0) return SEA_B200_OK;
    CU(cudaSetDevice(ctx->device));
    DecodeJob job;
    int rc = plan_decode(ctx, n_streams, headers, kFileHeaderBytes, sea_offsets, sea_lens, pcm_offsets, pcm_caps, &job);
    if (rc) return rc;
    uint64_t sea_len = 0;
    for (uint32_t i = 0; i < n_streams; i++) sea_len = std::max(sea_len, sea_offsets[i] + sea_lens[i]);
    // the first chunk's header word picks the specialised kernel; fetch it from the device copy
    uint32_t hdr_word = 0;
    bool have = false;
    if (job.streams[0].n_chunks > 0 && job.streams[0].data_len >= 4) {
        uint8_t w[4];
        CU(cudaMemcpyAsync(w, d_sea + job.streams[0].data_off, 4, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
        hdr_word = (uint32_t)w[0] | ((uint32_t)w[1] << 8) | ((uint32_t)w[2] << 16) | ((uint32_t)w[3] << 24);
        have = true;
    }
    DecLane L = decode_lane(ctx, 0);
    rc = run_decode(ctx, L, job, d_sea, sea_len, d_pcm, have, hdr_word);
    if (n_samples)
        for (uint32_t i = 0; i < n_streams; i++) n_samples[i] = rc == SEA_B200_OK ? job.n_samples[i] : 0;
    if (rc == SEA_B200_OK && job.trailing_invalid_frame)
        return fail(ctx, SEA_B200_ERR_INVALID_FRAME, "streaming header with a short last chunk (chunk.rs:76-79)");
    return rc;
}

int sea_b200_decode_batch(sea_b200_ctx *ctx, uint32_t n_streams, const uint8_t *sea, const uint64_t *sea_offsets,
                          const uint64_t *sea_lens, int16_t *pcm, const uint64_t *pcm_offsets, const uint64_t *pcm_caps,
                          uint64_t *n_samples)
{
    if (!ctx || !sea || !sea_offsets || !sea_lens || !pcm_offsets) return SEA_B200_ERR_INVALID_PARAMETERS;
    if (n_streams == 0) return SEA_B200_OK;
    CU(cudaSetDevice(ctx->device));
    // host copy of the headers, and the byte range to ship
    std::vector<uint8_t> headers((size_t)n_streams * kFileHeaderBytes, 0);
    uint64_t lo = UINT64_MAX, hi = 0;
    for (uint32_t i = 0; i < n_streams; i++) {
        memcpy(&headers[(size_t)i * kFileHeaderBytes], sea + sea_offsets[i], (size_t)std::min<uint64_t>(sea_lens[i], kFileHeaderBytes));
        lo = std::min(lo, sea_offsets[i]);
        hi = std::max(hi, sea_offsets[i] + sea_lens[i]);
    }
    std::vector<uint64_t> rel_off(n_streams);
    for (uint32_t i = 0; i < n_streams; i++) rel_off[i] = sea_offsets[i] - lo;
    DecodeJob job;
    int rc = plan_decode(ctx, n_streams, headers.data(), kFileHeaderBytes, rel_off.data(), sea_lens, pcm_offsets, pcm_caps, &job);
    if (rc) return rc;
    uint64_t plo = UINT64_MAX, phi = 0;
    for (uint32_t i = 0; i < n_streams; i++) {
        if (job.n_samples[i] == 0) continue;
        plo = std::min(plo, pcm_offsets[i]);
        phi = std::max(phi, pcm_offsets[i] + job.n_samples[i]);
    }
    if (phi == 0) plo = 0;
    if (phi && !pcm) return SEA_B200_ERR_INVALID_PARAMETERS;
    const uint64_t in_bytes = hi - lo, out_samples = phi - plo;

    // ---- group the streams (index order) so that copies and kernels of neighbouring groups overlap: PCIe is the bound of this
    // entry point (2 bytes out per sample against ~0.4 in), so the D2H engine should never wait for a kernel or an upload.
    struct Group {
        uint32_t i0, i1;
        uint64_t lo, hi, plo, phi;  // byte range of the .sea input (relative to the batch range), sample range of the PCM output
    };
    std::vector<Group> groups;
    {
        uint64_t target = 96ull << 20;  // PCM samples per group (192 MB): long enough to amortise launches, short enough to pipeline
        if (const char *env = getenv("SEA_B200_DEC_GROUP_SAMPLES")) target = std::max<uint64_t>(1, strtoull(env, nullptr, 10));  // tests, tuning
        Group g = {0, 0, UINT64_MAX, 0, UINT64_MAX, 0};
        uint64_t acc = 0;
        for (uint32_t i = 0; i < n_streams; i++) {
            g.lo = std::min(g.lo, rel_off[i]);
            g.hi = std::max(g.hi, rel_off[i] + sea_lens[i]);
            if (job.n_samples[i]) {
                g.plo = std::min(g.plo, pcm_offsets[i]);
                g.phi = std::max(g.phi, pcm_offsets[i] + job.n_samples[i]);
            }
            acc += job.n_samples[i];
            // the first group is a short one: nothing overlaps its upload and kernels, the copy-back engine idles until they are done
            if (acc >= (groups.empty() ? (target + 7) / 8 : target) || i + 1 == n_streams) {
                g.i1 = i + 1;
                if (g.phi == 0) g.plo = 0;
                groups.push_back(g);
                g = {i + 1, 0, UINT64_MAX, 0, UINT64_MAX, 0};
                acc = 0;
            }
        }
        uint64_t sum_in = 0, sum_out = 0;
        for (const Group &q : groups) {
            sum_in += q.hi - q.lo;
            sum_out += q.phi - q.plo;
        }
        // scattered or interleaved layouts would make the per-group ranges overlap: ship the batch as one group then
        if (groups.size() < 3 || sum_in > in_bytes + in_bytes / 4 + 4096 || sum_out > out_samples + out_samples / 4 + 4096)
            groups.assign(1, Group{0, n_streams, 0, in_bytes, plo, phi});
    }
    const bool piped = groups.size() > 1;
    uint64_t max_in = 0, max_out = 0;
    for (const Group &q : groups) {
        max_in = std::max(max_in, q.hi - q.lo);
        max_out = std::max(max_out, q.phi - q.plo);
    }
    // Upload-ahead (pipelined batches whose .sea bytes fit a device buffer of <= 8 GB): every group's input has its own slot and
    // all uploads are queued at once on a third stream, a lane only waits for its group's event.  Tied to the lanes (the first
    // form: group i+2's upload queued behind group i's download) every download started together with an upload and ran 5-6 %
    // slower for its whole length (50-53.5 against 53-57 GB/s, profiles/r02_s3_e2e_probe_*.txt); run ahead, the uploads are over
    // after the first five groups and only those downloads are slowed (42 GB/s), the other twenty run at the link's rate: ~2 %
    // per call.  (Plain copies show the same thing, profiles/r02_s3_copy_probe.txt: a download that STARTS while an upload is
    // running stays slow after the upload has ended.  All downloads on one more stream of their own, or the uploads as five growing copies instead of one per group: no change, not kept.)
    // SEA_B200_DEC_UPLOAD_AHEAD=0: the first form.
    bool ahead = piped && in_bytes <= (8ull << 30);
    if (const char *env = getenv("SEA_B200_DEC_UPLOAD_AHEAD")) ahead = ahead && env[0] != '0';
    std::vector<uint64_t> dev_off(groups.size(), 0);  // upload-ahead: the group's slot in ctx->in (256-byte aligned: the kernels want 16)
    if (ahead) {
        uint64_t o = 0;
        for (size_t gi = 0; gi < groups.size(); gi++) {
            dev_off[gi] = o;
            o += (groups[gi].hi - groups[gi].lo + 64 + 255) & ~255ull;
        }
        CU(ctx->in.reserve(o + 64));
        if (!ctx->up) CU(cudaStreamCreateWithFlags(&ctx->up, cudaStreamNonBlocking));
    } else {
        CU(ctx->in.reserve(max_in + 64));
    }
    CU(ctx->out.reserve(max_out * 2 + 64));
    if (piped) {
        if (!ahead) CU(ctx->aux.in.reserve(max_in + 64));
        CU(ctx->aux.out.reserve(max_out * 2 + 64));
        CU(cudaEventRecord(ctx->aux.ev0, ctx->stream));  // order the other streams after whatever the caller queued before us
        CU(cudaStreamWaitEvent(ctx->aux.stream, ctx->aux.ev0, 0));
        if (ahead) CU(cudaStreamWaitEvent(ctx->up, ctx->aux.ev0, 0));
    }
    // events of group gi: kernels begin / end, download begins / ends, upload done
    enum { kEvK0 = 0, kEvK1, kEvD0, kEvD1, kEvUp, kEvPerGroup };
    auto gev = [&](size_t gi, int which) { return ctx->grp_ev[1 + kEvPerGroup * gi + which]; };
    auto upload = [&](size_t gi) -> cudaError_t {
        const Group &q = groups[gi];
        if (ahead) {
            cudaError_t e = cudaMemcpyAsync(ctx->in.as<uint8_t>() + dev_off[gi], sea + lo + q.lo, q.hi - q.lo, cudaMemcpyHostToDevice, ctx->up);
            return e != cudaSuccess ? e : cudaEventRecord(gev(gi, kEvUp), ctx->up);
        }
        DecLane L = decode_lane(ctx, (int)(gi & 1));
        return cudaMemcpyAsync(L.in->p, sea + lo + q.lo, q.hi - q.lo, cudaMemcpyHostToDevice, L.stream);
    };
    // Deferred error words (pipelined batches): a group's kernels report through a word that the host used to wait for before it
    // queued the group's download -- a round trip per group in front of the copy engine this entry point is bound by.  Now the
    // whole batch is queued without a host wait, every group's word lands in pinned memory behind its kernels, and a group whose
    // word is not kDevOk (a chunk the specialised kernel hands back, or a malformed one) is redone on its own, synchronously,
    // after the pipeline drained.  SEA_B200_DEC_DEFER=0 keeps the wait-per-group form (A/B, tests).
    bool defer = piped;
    if (const char *env = getenv("SEA_B200_DEC_DEFER")) defer = piped && env[0] != '0';
    const bool trace = getenv("SEA_B200_TRACE") != nullptr;
    if (defer) {
        if (ctx->h_errs_cap < groups.size()) {
            if (ctx->h_errs) cudaFreeHost(ctx->h_errs);
            ctx->h_errs = nullptr;
            ctx->h_errs_cap = 0;
            CU(cudaHostAlloc(reinterpret_cast<void **>(&ctx->h_errs), sizeof(int) * (groups.size() + 64), cudaHostAllocDefault));
            ctx->h_errs_cap = groups.size() + 64;
        }
        memset(ctx->h_errs, 0, sizeof(int) * groups.size());
    }
    if (defer || trace || ahead)
        while (ctx->grp_ev.size() < 1 + kEvPerGroup * groups.size()) {
            cudaEvent_t e;
            CU(cudaEventCreate(&e));
            ctx->grp_ev.push_back(e);
        }
    double kernel_ms = 0.0;
    std::vector<Run> runs;
    std::vector<char> was_deferred(groups.size(), 0);
    // one group through lane `lane`: kernels (+ the download of what its streams own) queued on the lane's stream
    auto do_group = [&](size_t gi, int lane, bool deferred_mode) -> int {
        const Group &q = groups[gi];
        DecLane L = decode_lane(ctx, lane);
        if (deferred_mode) {
            L.defer = &ctx->h_errs[gi];
            L.k0 = gev(gi, kEvK0);
            L.k1 = gev(gi, kEvK1);
        }
        const uint8_t *d_in = ahead ? ctx->in.as<uint8_t>() + dev_off[gi] : L.in->as<uint8_t>();
        if (ahead) CU(cudaStreamWaitEvent(L.stream, gev(gi, kEvUp), 0));
        DecodeJob sub;
        sub.streams.assign(job.streams.begin() + q.i0, job.streams.begin() + q.i1);
        sub.n_samples.assign(job.n_samples.begin() + q.i0, job.n_samples.begin() + q.i1);
        const uint32_t chain0 = sub.streams.empty() ? 0u : sub.streams[0].chain_begin;
        for (auto &d : sub.streams) {
            d.data_off -= q.lo;
            d.pcm_off -= q.plo;
            d.chain_begin -= chain0;
        }
        const DecStream &last = job.streams[q.i1 - 1];
        sub.total_chains = (uint64_t)last.chain_begin + (uint64_t)last.n_chunks * last.channels - chain0;
        // the group's own first stream decides its specialisation (a mixed batch may still have uniform groups)
        if (parse_file_header(&headers[(size_t)q.i0 * kFileHeaderBytes], kFileHeaderBytes, &sub.first) != SEA_B200_OK) sub.first = job.first;
        sub.uniform = true;
        for (const DecStream &d : sub.streams)
            if (d.channels != sub.first.channels || d.chunk_size != sub.first.chunk_size || d.frames_per_chunk != sub.first.frames_per_chunk)
                sub.uniform = false;
        uint32_t hdr_word = 0;
        bool have = false;
        if (!sub.streams.empty() && sub.streams[0].n_chunks > 0 && sub.streams[0].data_len >= 4) {
            const uint8_t *w = sea + sea_offsets[q.i0] + kFileHeaderBytes;
            hdr_word = (uint32_t)w[0] | ((uint32_t)w[1] << 8) | ((uint32_t)w[2] << 16) | ((uint32_t)w[3] << 24);
            have = true;
        }
        int r = run_decode(ctx, L, sub, d_in, q.hi - q.lo, L.out->as<int16_t>(), have, hdr_word);
        kernel_ms += L.kernel_ms;
        was_deferred[gi] = L.deferred;
        if (r == SEA_B200_OK && q.phi > q.plo) {
            // only the ranges the streams own go back: whatever lies between them in the caller's buffer is not ours to touch
            // (one copy per run of adjacent streams; a packed layout is a single run)
            runs.clear();
            for (uint32_t i = q.i0; i < q.i1; i++)
                if (job.n_samples[i]) runs.push_back({pcm_offsets[i], pcm_offsets[i] + job.n_samples[i]});
            merge_runs(runs);
            if (trace) CU(cudaEventRecord(gev(gi, kEvD0), L.stream));
            for (const Run &rn : runs)
                CU(cudaMemcpyAsync(pcm + rn.lo, L.out->as<int16_t>() + (rn.lo - q.plo), (rn.hi - rn.lo) * 2, cudaMemcpyDeviceToHost, L.stream));
            if (trace) CU(cudaEventRecord(gev(gi, kEvD1), L.stream));
        }
        return r;
    };
    if (trace) CU(cudaEventRecord(ctx->grp_ev[0], ctx->stream));
    if (ahead) {
        for (size_t gi = 0; gi < groups.size(); gi++) CU(upload(gi));
    } else {
        CU(upload(0));
    }
    for (size_t gi = 0; gi < groups.size() && rc == SEA_B200_OK; gi++) {
        if (!ahead && gi + 1 < groups.size()) CU(upload(gi + 1));  // queued behind the other lane's previous download, ahead of our kernels
        rc = do_group(gi, (int)(gi & 1), defer);
    }
    CU(cudaStreamSynchronize(ctx->stream));
    if (piped) CU(cudaStreamSynchronize(ctx->aux.stream));
    if (ahead) CU(cudaStreamSynchronize(ctx->up));
    if (trace && rc == SEA_B200_OK) {
        float t_prev = 0.f;
        for (size_t gi = 0; gi < groups.size(); gi++) {
            float a = 0.f, b = 0.f, k = 0.f, u = 0.f;
            cudaEventElapsedTime(&a, ctx->grp_ev[0], gev(gi, kEvD0));
            cudaEventElapsedTime(&b, ctx->grp_ev[0], gev(gi, kEvD1));
            if (was_deferred[gi]) cudaEventElapsedTime(&k, gev(gi, kEvK0), gev(gi, kEvK1));
            if (ahead) cudaEventElapsedTime(&u, ctx->grp_ev[0], gev(gi, kEvUp));
            fprintf(stderr, "sea_b200 trace: group %zu: upload done %.3f ms, download starts %.3f ms (gap %.3f), takes %.3f ms = %.1f GB/s; kernels %.3f ms\n",
                    gi, u, a, a - t_prev, b - a, (double)(groups[gi].phi - groups[gi].plo) * 2.0 / ((b - a) * 1e6), k);
            t_prev = b;
        }
    }
    if (defer && rc == SEA_B200_OK) {
        for (size_t gi = 0; gi < groups.size() && rc == SEA_B200_OK; gi++) {
            if (!was_deferred[gi]) continue;
            float ms = 0.f;
            cudaEventElapsedTime(&ms, gev(gi, kEvK0), gev(gi, kEvK1));
            kernel_ms += ms;
            if (ctx->h_errs[gi] == kDevOk) continue;
            // redo this group alone with a wait behind its kernels: run_decode falls back to the generic kernel or reports the error
            const Group &q = groups[gi];
            if (!ahead) CU(cudaMemcpyAsync(ctx->in.p, sea + lo + q.lo, q.hi - q.lo, cudaMemcpyHostToDevice, ctx->stream));  // else: still in its slot
            rc = do_group(gi, 0, false);
            CU(cudaStreamSynchronize(ctx->stream));
        }
    }
    ctx->last_kernel_ms = kernel_ms;
    if (n_samples)
        for (uint32_t i = 0; i < n_streams; i++) n_samples[i] = rc == SEA_B200_OK ? job.n_samples[i] : 0;
    if (rc == SEA_B200_OK && job.trailing_invalid_frame)
        return fail(ctx, SEA_B200_ERR_INVALID_FRAME, "streaming header with a short last chunk (chunk.rs:76-79)");
    return rc;
}

int sea_b200_decode(sea_b200_ctx *ctx, const uint8_t *sea, uint64_t len, int16_t *pcm, uint64_t pcm_cap_samples, uint64_t *n_samples,
                    uint32_t *sample_rate, uint32_t *channels)
{
    if (!ctx || !sea) return SEA_B200_ERR_INVALID_PARAMETERS;
    sea_b200_header h;
    int rc = parse_file_header(sea, len, &h);
    if (rc) return fail(ctx, rc, "bad .sea header (file.rs:40-72)");
    if (sample_rate) *sample_rate = h.sample_rate;
    if (channels) *channels = h.channels;
    const uint64_t off = 0, poff = 0;
    if (!pcm) {  // c/sea.h:209-211 two-call pattern: report the size only
        DecodeJob job;
        rc = plan_decode(ctx, 1, sea, kFileHeaderBytes, &off, &len, &poff, nullptr, &job);
        if (rc) return rc;
        if (n_samples) *n_samples = job.n_samples[0];
        return SEA_B200_OK;
    }
    return sea_b200_decode_batch(ctx, 1, sea, &off, &len, pcm, &poff, &pcm_cap_samples, n_samples);
}

// ------------------------------------------------------------------------------------------------ frame windows

// Every non-empty window becomes one DecStream over the chunks that cover it (plan_range, the arithmetic of decode_range), decoded
// by run_decode into a scratch buffer exactly as decode_range decodes its sub-file; window_extract_kernel then cuts each slot out.
// Windows go in index order in groups whose covering ranges fit the scratch cap (one run_decode + one cut per group).
int sea_b200_decode_windows_device(sea_b200_ctx *ctx, uint32_t n_streams, const uint8_t *d_sea, const uint64_t *sea_offsets,
                                   const uint64_t *sea_lens, const uint8_t *headers, uint32_t n_windows, const uint32_t *window_stream,
                                   const uint64_t *first_frames, const uint32_t *n_frames, uint32_t flags, void *d_out,
                                   const uint64_t *out_offsets, uint64_t *frames_out)
{
    if (!ctx || !sea_offsets || !sea_lens || !headers) return SEA_B200_ERR_INVALID_PARAMETERS;
    if (flags & ~(SEA_B200_RANGE_SKIP_METADATA | SEA_B200_WINDOW_F32_PLANAR))
        return fail(ctx, SEA_B200_ERR_INVALID_PARAMETERS, "unknown flag bits");
    if (n_windows == 0) return SEA_B200_OK;
    if (!window_stream || !first_frames || !n_frames || !d_out || !out_offsets) return SEA_B200_ERR_INVALID_PARAMETERS;
    if (frames_out) memset(frames_out, 0, sizeof(uint64_t) * n_windows);
    const bool planar = flags & SEA_B200_WINDOW_F32_PLANAR;
    if (reinterpret_cast<uintptr_t>(d_out) % (planar ? sizeof(float) : sizeof(int16_t)))
        return fail(ctx, SEA_B200_ERR_INVALID_PARAMETERS, "d_out is not aligned to its element type");
    for (uint32_t w = 0; w < n_windows; w++)
        if (window_stream[w] >= n_streams)
            return fail(ctx, SEA_B200_ERR_INVALID_PARAMETERS, "window " + std::to_string(w) + ": stream index out of range");
    std::vector<sea_b200_header> hs(n_streams);
    uint64_t sea_len = 0;
    for (uint32_t i = 0; i < n_streams; i++) {  // as plan_decode checks them
        const uint64_t len = sea_lens[i];
        int rc = parse_file_header(headers + (size_t)i * kFileHeaderBytes, len < 22 ? len : 22, &hs[i]);
        if (rc) return fail(ctx, rc, "stream " + std::to_string(i) + ": bad .sea header (file.rs:40-72)");
        sea_len = std::max(sea_len, sea_offsets[i] + len);
    }
    std::vector<RangePlan> plans(n_windows);
    for (uint32_t w = 0; w < n_windows; w++) {
        const uint32_t s = window_stream[w];
        int rc = plan_range(hs[s], sea_lens[s], first_frames[w], n_frames[w], flags & SEA_B200_RANGE_SKIP_METADATA, &plans[w]);
        if (rc) return fail(ctx, rc, "window " + std::to_string(w) + ": metadata runs past the end of the stream");
        if (plans[w].want && plans[w].sub_frames > 0xffffffffull)
            return fail(ctx, SEA_B200_ERR_TOO_MANY_FRAMES, "window " + std::to_string(w) + ": covering chunks longer than 2^32 frames");
    }
    CU(cudaSetDevice(ctx->device));

    // scratch samples per group: 2 GiB of int16 (SEA_B200_WIN_SCRATCH_SAMPLES: tests, tuning); a window larger than that is a group
    uint64_t cap = 1ull << 30;
    if (const char *env = getenv("SEA_B200_WIN_SCRATCH_SAMPLES")) cap = std::max<uint64_t>(1, strtoull(env, nullptr, 10));
    auto region = [&](uint32_t w) -> uint64_t {  // rows of the lane-per-chunk kernels' 256-bit stores: 16-sample aligned
        return plans[w].want ? (plans[w].sub_frames * hs[window_stream[w]].channels + 15u) & ~15ull : 0u;
    };
    const bool trace = getenv("SEA_B200_TRACE") != nullptr;
    double decode_ms = 0.0, extract_ms = 0.0;
    for (uint32_t w0 = 0, g = 0; w0 < n_windows; g++) {
        uint32_t w1 = w0;
        uint64_t scratch = 0;
        while (w1 < n_windows && (w1 == w0 || scratch + region(w1) <= cap)) scratch += region(w1++);
        DecodeJob job;
        std::vector<WinDesc> desc;
        uint64_t chains = 0, max_slot = 0, off = 0;
        for (uint32_t w = w0; w < w1; w++) {
            const RangePlan &r = plans[w];
            const uint32_t s = window_stream[w];
            const sea_b200_header &h = hs[s];
            WinDesc wd = {};
            wd.dst = out_offsets[w];
            wd.frames = n_frames[w];
            wd.channels = h.channels;
            wd.real = (uint32_t)r.want;
            if (r.want) {
                DecStream d;
                memset(&d, 0, sizeof(d));
                d.data_off = sea_offsets[s] + r.b0;
                d.data_len = r.b1 - r.b0;
                d.pcm_off = off;
                d.total_frames = (uint32_t)r.sub_frames;  // whole covering chunks: a chunk's layout depends on its own frame count
                d.n_chunks = (uint32_t)(r.k1 - r.k0);
                d.chain_begin = (uint32_t)chains;
                d.chunk_size = h.chunk_size;
                d.frames_per_chunk = h.frames_per_chunk;
                d.channels = h.channels;
                if (job.streams.empty()) job.first = h;
                else if (h.channels != job.first.channels || h.chunk_size != job.first.chunk_size || h.frames_per_chunk != job.first.frames_per_chunk)
                    job.uniform = false;
                job.streams.push_back(d);
                chains += (uint64_t)d.n_chunks * h.channels;
                if (chains > 0xfffffff0ull) return fail(ctx, SEA_B200_ERR_INVALID_PARAMETERS, "window group too large (2^32 chains)");
                wd.src = off + r.skip * h.channels;
                off += region(w);
            }
            if (wd.frames) {
                desc.push_back(wd);
                max_slot = std::max(max_slot, (uint64_t)wd.frames * wd.channels);
            }
        }
        job.total_chains = chains;
        // the cut reads whole 16-byte vectors: up to 16 samples past a window's covering range
        CU(ctx->win.reserve((off + 64) * sizeof(int16_t)));
        float ms_dec = 0.f, ms_cut = 0.f;
        if (!job.streams.empty()) {
            const DecStream &d0 = job.streams[0];  // its first chunk's header word picks the specialised kernel
            uint32_t hdr_word = 0;
            bool have = false;
            if (d0.data_len >= 4) {
                uint8_t b[4];
                CU(cudaMemcpyAsync(b, d_sea + d0.data_off, 4, cudaMemcpyDeviceToHost, ctx->stream));
                CU(cudaStreamSynchronize(ctx->stream));
                hdr_word = (uint32_t)b[0] | ((uint32_t)b[1] << 8) | ((uint32_t)b[2] << 16) | ((uint32_t)b[3] << 24);
                have = true;
            }
            DecLane L = decode_lane(ctx, 0);
            int rc = run_decode(ctx, L, job, d_sea, sea_len, ctx->win.as<int16_t>(), have, hdr_word);
            if (rc) return rc;
            ms_dec = (float)L.kernel_ms;
        }
        if (!desc.empty()) {
            CU(ctx->win_desc.reserve(sizeof(WinDesc) * desc.size()));
            CU(cudaMemcpyAsync(ctx->win_desc.p, desc.data(), sizeof(WinDesc) * desc.size(), cudaMemcpyHostToDevice, ctx->stream));
            CU(cudaEventRecord(ctx->ev0, ctx->stream));
            CU(launch_window_extract(ctx->win.as<int16_t>(), d_out, ctx->win_desc.as<WinDesc>(), (uint32_t)desc.size(), max_slot, planar,
                                     ctx->stream));
            ctx->launches++;
            CU(cudaEventRecord(ctx->ev1, ctx->stream));
            CU(cudaStreamSynchronize(ctx->stream));  // the next group reuses the scratch and the events
            cudaEventElapsedTime(&ms_cut, ctx->ev0, ctx->ev1);
        }
        decode_ms += ms_dec;
        extract_ms += ms_cut;
        if (trace)
            fprintf(stderr, "sea_b200 trace: window group %u: windows %u..%u, covering %llu samples, decode %.3f ms, extract %.3f ms\n", g, w0,
                    w1 - 1, (unsigned long long)off, ms_dec, ms_cut);
        w0 = w1;
    }
    ctx->last_kernel_ms = decode_ms + extract_ms;
    if (frames_out)
        for (uint32_t w = 0; w < n_windows; w++) frames_out[w] = plans[w].want;
    return SEA_B200_OK;
}

// ------------------------------------------------------------------------------------------------ registered corpus

}  // extern "C"

struct sea_b200_corpus {
    sea_b200_ctx *ctx;
    uint32_t n_streams, channels;
    bool fast;
    const uint8_t *d_sea;
    uint64_t sea_len;                    // readable bytes from d_sea: the end of the furthest stream
    CorpusStream *d_streams = nullptr;
    std::vector<uint64_t> stream_frames;
    uint32_t N_min, s, b;                // smallest frames_per_chunk; the fast route's header fields
};

extern "C" {

// The stream table and every chunk a window can cover are checked here, once (corpus_validate_kernel): the async call then has no
// malformed-chunk path, no error word to read back and no fallback, which is what lets it run without a host synchronisation.
int sea_b200_corpus_create(sea_b200_ctx *ctx, uint32_t n_streams, const uint8_t *d_sea, const uint64_t *sea_offsets,
                           const uint64_t *sea_lens, const uint8_t *headers, uint32_t flags, sea_b200_corpus **corpus)
{
    if (!ctx || !corpus) return SEA_B200_ERR_INVALID_PARAMETERS;
    *corpus = nullptr;
    if (!d_sea || !sea_offsets || !sea_lens || !headers || n_streams == 0)
        return fail(ctx, SEA_B200_ERR_INVALID_PARAMETERS, "a corpus needs at least one stream and every pointer");
    if (flags & ~SEA_B200_RANGE_SKIP_METADATA) return fail(ctx, SEA_B200_ERR_INVALID_PARAMETERS, "unknown flag bits");
    int force = -1;  // SEA_B200_CORPUS_ROUTE = generic / fast pins the route (tests)
    if (const char *env = getenv("SEA_B200_CORPUS_ROUTE")) {
        if (!strcmp(env, "generic")) force = 0;
        else if (!strcmp(env, "fast")) force = 1;
        else return fail(ctx, SEA_B200_ERR_INVALID_PARAMETERS, "SEA_B200_CORPUS_ROUTE must be generic or fast");
    }
    std::vector<CorpusStream> table(n_streams);
    std::vector<uint64_t> frames(n_streams);
    uint32_t channels = 0, N_min = 0xffffffffu;
    bool uniform = true;
    uint64_t chunks = 0, sea_len = 0;
    for (uint32_t i = 0; i < n_streams; i++) {
        const uint64_t len = sea_lens[i];
        sea_b200_header h;
        int rc = parse_file_header(headers + (size_t)i * kFileHeaderBytes, len < 22 ? len : 22, &h);
        if (rc) return fail(ctx, rc, "stream " + std::to_string(i) + ": bad .sea header (file.rs:40-72)");
        if (i == 0) channels = h.channels;
        if (h.channels != channels)
            return fail(ctx, SEA_B200_ERR_INVALID_PARAMETERS, "stream " + std::to_string(i) + " has " + std::to_string(h.channels) +
                                                                  " channels, stream 0 has " + std::to_string(channels));
        RangePlan rp;
        rc = plan_range(h, len, 0, 0, flags & SEA_B200_RANGE_SKIP_METADATA, &rp);
        if (rc) return fail(ctx, rc, "stream " + std::to_string(i) + ": metadata runs past the end of the stream");
        if (rp.file_frames > 0xffffffffull)
            return fail(ctx, SEA_B200_ERR_TOO_MANY_FRAMES, "stream " + std::to_string(i) + ": longer than 2^32 frames");
        CorpusStream &t = table[i];
        memset(&t, 0, sizeof(t));
        t.body = sea_offsets[i] + rp.body;
        t.len = len - rp.body;
        t.file_frames = rp.file_frames;
        t.chunk_begin = chunks;
        t.chunk_size = h.chunk_size;
        t.N = h.frames_per_chunk;
        t.n_chunks = (uint32_t)((rp.file_frames + t.N - 1) / t.N);
        chunks += t.n_chunks;
        frames[i] = rp.file_frames;
        N_min = std::min(N_min, t.N);
        if (t.chunk_size != table[0].chunk_size || t.N != table[0].N) uniform = false;
        sea_len = std::max(sea_len, sea_offsets[i] + len);
    }
    CU(cudaSetDevice(ctx->device));
    // every chunk is compared with the first chunk of the first stream that has one
    uint32_t ref_word = 0;
    for (uint32_t i = 0; i < n_streams; i++)
        if (table[i].n_chunks) {
            uint8_t b[4] = {0, 0, 0, 0};
            CU(cudaMemcpy(b, d_sea + table[i].body, std::min<uint64_t>(4, table[i].len), cudaMemcpyDeviceToHost));
            ref_word = (uint32_t)b[0] | ((uint32_t)b[1] << 8) | ((uint32_t)b[2] << 16) | ((uint32_t)b[3] << 24);
            break;
        }

    sea_b200_corpus *c = new sea_b200_corpus();
    c->ctx = ctx;
    auto bail = [&](int rc) {
        sea_b200_corpus_destroy(c);
        return rc;
    };
    cudaError_t e = cudaMalloc(&c->d_streams, sizeof(CorpusStream) * n_streams);
    if (e != cudaSuccess) return bail(cuda_fail(ctx, e, "cudaMalloc(corpus stream table)"));
    e = cudaMemcpy(c->d_streams, table.data(), sizeof(CorpusStream) * n_streams, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) return bail(cuda_fail(ctx, e, "cudaMemcpy(corpus stream table)"));
    struct { unsigned long long first_bad; uint32_t mixed, pad; } res = {~0ull, 0u, 0u};
    void *d_res = nullptr;
    if ((e = cudaMalloc(&d_res, sizeof(res))) != cudaSuccess) return bail(cuda_fail(ctx, e, "cudaMalloc(corpus check words)"));
    e = cudaMemcpyAsync(d_res, &res, sizeof(res), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess)
        e = launch_corpus_validate(d_sea, c->d_streams, n_streams, chunks, channels, ref_word, static_cast<unsigned long long *>(d_res),
                                   reinterpret_cast<uint32_t *>(static_cast<uint8_t *>(d_res) + 8), ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(&res, d_res, sizeof(res), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    cudaFree(d_res);
    if (e != cudaSuccess) return bail(cuda_fail(ctx, e, "corpus validation"));
    ctx->launches++;
    if (res.first_bad != ~0ull) {
        const uint64_t g = res.first_bad >> 2;
        uint32_t i = 0;
        while (i + 1 < n_streams && table[i + 1].chunk_begin <= g) i++;
        const int rc = map_dev_error(ctx, (int)(res.first_bad & 3u));
        ctx->last_error = "stream " + std::to_string(i) + ", chunk " + std::to_string(g - table[i].chunk_begin) + ": " + ctx->last_error;
        return bail(rc);
    }
    const uint32_t type = ref_word & 0xffu, s = (ref_word >> 12) & 15u, b = (ref_word >> 8) & 15u, F = (ref_word >> 16) & 0xffu;
    const bool qualifies = chunks > 0 && uniform && !res.mixed && corpus_fast_supported(channels, s, b, F, type == 2u);
    if (force == 1 && !qualifies)
        return bail(fail(ctx, SEA_B200_ERR_INVALID_PARAMETERS,
                         "SEA_B200_CORPUS_ROUTE=fast: the corpus does not qualify (it needs uniform CBR chunks, 1 or 2 channels, "
                         "scale_factor_frames 20, scale_factor_bits <= 5)"));
    c->fast = force >= 0 ? force == 1 : qualifies;
    if (c->fast && (e = corpus_fast_prepare(channels, s, b)) != cudaSuccess) return bail(cuda_fail(ctx, e, "corpus_fast_prepare"));
    c->n_streams = n_streams;
    c->channels = channels;
    c->d_sea = d_sea;
    c->sea_len = sea_len;
    c->stream_frames = std::move(frames);
    c->N_min = N_min == 0xffffffffu ? 1u : N_min;
    c->s = s;
    c->b = b;
    *corpus = c;
    return SEA_B200_OK;
}

void sea_b200_corpus_destroy(sea_b200_corpus *corpus)
{
    if (!corpus) return;
    cudaSetDevice(corpus->ctx->device);
    if (corpus->ctx->stream) cudaStreamSynchronize(corpus->ctx->stream);
    if (corpus->d_streams) cudaFree(corpus->d_streams);  // also waits for the corpus's work on any other stream
    delete corpus;
}

int sea_b200_corpus_info(const sea_b200_corpus *corpus, uint32_t *channels, uint64_t *stream_frames, uint32_t *route)
{
    if (!corpus) return SEA_B200_ERR_INVALID_PARAMETERS;
    if (channels) *channels = corpus->channels;
    if (stream_frames) memcpy(stream_frames, corpus->stream_frames.data(), sizeof(uint64_t) * corpus->n_streams);
    if (route) *route = corpus->fast ? 1u : 0u;
    return SEA_B200_OK;
}

// Enqueues one kernel on the context's stream and nothing else: no allocation, no copy, no synchronisation (graph-capturable).
int sea_b200_corpus_decode_windows_async(sea_b200_corpus *corpus, uint32_t n_windows, const uint32_t *d_window_stream,
                                         const uint64_t *d_first_frames, uint32_t window_frames, uint32_t flags, void *d_out,
                                         uint32_t *d_frames_out, int32_t *d_status)
{
    if (!corpus) return SEA_B200_ERR_INVALID_PARAMETERS;
    sea_b200_ctx *ctx = corpus->ctx;
    if (flags & ~SEA_B200_WINDOW_F32_PLANAR) return fail(ctx, SEA_B200_ERR_INVALID_PARAMETERS, "unknown flag bits");
    if (n_windows == 0 || window_frames == 0) return SEA_B200_OK;
    if (!d_window_stream || !d_first_frames || !d_out || !d_status) return fail(ctx, SEA_B200_ERR_INVALID_PARAMETERS, "NULL pointer");
    const bool planar = flags & SEA_B200_WINDOW_F32_PLANAR;
    if (reinterpret_cast<uintptr_t>(d_out) % (planar ? sizeof(float) : sizeof(int16_t)))
        return fail(ctx, SEA_B200_ERR_INVALID_PARAMETERS, "d_out is not aligned to its element type");
    const uint64_t M = ((uint64_t)window_frames + corpus->N_min - 2u) / corpus->N_min + 1u;  // most chunks a window can touch
    if ((uint64_t)n_windows * M * corpus->channels > (1ull << 38))
        return fail(ctx, SEA_B200_ERR_INVALID_PARAMETERS, "too many windows x covering chunks for one launch");
    CorpusLaunch p = {};
    p.sea = corpus->d_sea;
    p.sea_len = corpus->sea_len;
    p.streams = corpus->d_streams;
    p.n_streams = corpus->n_streams;
    p.channels = corpus->channels;
    p.win_stream = d_window_stream;
    p.win_first = d_first_frames;
    p.n_windows = n_windows;
    p.W = window_frames;
    p.M = (uint32_t)M;
    p.planar = planar;
    p.out = d_out;
    p.frames_out = d_frames_out;
    p.status = d_status;
    p.N = corpus->N_min;
    p.s = corpus->s;
    p.b = corpus->b;
    CU(cudaSetDevice(ctx->device));
    CU(launch_corpus_windows(p, corpus->fast, ctx->tabs, ctx->stream));
    ctx->launches++;
    return SEA_B200_OK;
}

// ------------------------------------------------------------------------------------------------ encode entry points

int sea_b200_encode_batch_device(sea_b200_ctx *ctx, uint32_t n_streams, const int16_t *d_pcm, const uint64_t *pcm_offsets,
                                 const uint32_t *n_frames, uint32_t sample_rate, uint32_t channels, const sea_b200_settings *settings,
                                 uint8_t *d_out, const uint64_t *out_offsets, uint64_t *out_lens)
{
    if (!ctx || !pcm_offsets || !n_frames || !settings || !out_offsets || !out_lens) return SEA_B200_ERR_INVALID_PARAMETERS;
    if (n_streams == 0) return SEA_B200_OK;
    CU(cudaSetDevice(ctx->device));
    EncodeJob job;
    int rc = plan_encode(ctx, n_streams, pcm_offsets, n_frames, sample_rate, channels, settings, out_offsets, false, &job);
    if (rc) return rc;
    return run_encode(ctx, job, d_pcm, d_out, nullptr, out_lens, nullptr);
}

int sea_b200_encode_batch(sea_b200_ctx *ctx, uint32_t n_streams, const int16_t *pcm, const uint64_t *pcm_offsets, const uint32_t *n_frames,
                          uint32_t sample_rate, uint32_t channels, const sea_b200_settings *settings, uint8_t *out,
                          const uint64_t *out_offsets, uint64_t *out_lens)
{
    if (!ctx || !pcm_offsets || !n_frames || !settings || !out || !out_offsets || !out_lens) return SEA_B200_ERR_INVALID_PARAMETERS;
    if (n_streams == 0) return SEA_B200_OK;
    CU(cudaSetDevice(ctx->device));
    EncodeJob job;
    int rc = plan_encode(ctx, n_streams, pcm_offsets, n_frames, sample_rate, channels, settings, out_offsets, false, &job);
    if (rc) return rc;
    uint64_t lo = UINT64_MAX, hi = 0, olo = UINT64_MAX, ohi = 0;
    for (uint32_t i = 0; i < n_streams; i++) {
        const uint64_t ns = (uint64_t)n_frames[i] * channels;
        if (ns) {
            lo = std::min(lo, pcm_offsets[i]);
            hi = std::max(hi, pcm_offsets[i] + ns);
        }
        olo = std::min(olo, out_offsets[i]);
        ohi = std::max(ohi, out_offsets[i] + encode_bound_bytes(job.plan, n_frames[i]));
    }
    if (hi == 0) lo = 0;
    if (hi && !pcm) return SEA_B200_ERR_INVALID_PARAMETERS;
    if (hi) {  // long batches: slices of time pipelined over the copy engines (same bytes; see encode_batch_sliced)
        rc = encode_batch_sliced(ctx, n_streams, pcm, pcm_offsets, n_frames, sample_rate, channels, settings, job.plan, out, out_offsets, out_lens);
        if (rc <= 0) return rc;
    }
    for (auto &e : job.streams) {
        e.pcm_off -= (e.n_frames ? lo : e.pcm_off);
        e.out_off -= olo;
    }
    CU(ctx->in.reserve((hi - lo) * 2 + 64));
    CU(ctx->out.reserve(ohi - olo + 64));
    if (hi) CU(cudaMemcpyAsync(ctx->in.p, pcm + lo, (hi - lo) * 2, cudaMemcpyHostToDevice, ctx->stream));
    rc = run_encode(ctx, job, ctx->in.as<int16_t>(), ctx->out.as<uint8_t>(), nullptr, out_lens, nullptr);
    if (rc) return rc;
    // ship back only what was written, and only into the ranges the streams own (one copy per run of adjacent streams)
    std::vector<Run> runs;
    for (uint32_t i = 0; i < n_streams; i++)
        if (out_lens[i]) runs.push_back({out_offsets[i], out_offsets[i] + out_lens[i]});
    merge_runs(runs);
    for (const Run &r : runs)
        CU(cudaMemcpyAsync(out + r.lo, ctx->out.as<uint8_t>() + (r.lo - olo), r.hi - r.lo, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return SEA_B200_OK;
}

int sea_b200_encode(sea_b200_ctx *ctx, const int16_t *pcm, uint64_t n_samples, uint32_t sample_rate, uint32_t channels,
                    const sea_b200_settings *settings, uint8_t *out, uint64_t out_cap, uint64_t *out_len)
{
    if (!ctx || !settings || !out || !out_len || channels == 0) return SEA_B200_ERR_INVALID_PARAMETERS;
    const uint64_t frames64 = n_samples / channels;  // lib.rs:25 (`as u32`)
    if (frames64 > 0xffffffffull) return fail(ctx, SEA_B200_ERR_TOO_MANY_FRAMES, "more than 2^32 frames");
    if (frames64 == 0 && n_samples != 0)
        return fail(ctx, SEA_B200_ERR_DOMAIN, "fewer samples than channels: the reference fails with UnexpectedEof (encoder.rs:95-99)");
    const uint32_t frames = (uint32_t)frames64;
    uint64_t bound = 0;
    int rc = sea_b200_encode_bound(frames, channels, settings, &bound);
    if (rc) return fail(ctx, rc, "encoder settings rejected (outside the reference's domain)");
    if (bound > out_cap) return fail(ctx, SEA_B200_ERR_CAPACITY, "output buffer smaller than sea_b200_encode_bound");
    const uint64_t off = 0;
    return sea_b200_encode_batch(ctx, 1, pcm, &off, &frames, sample_rate, channels, settings, out, &off, out_len);
}

// ------------------------------------------------------------------------------------------------ streaming seam

int sea_b200_encoder_create(sea_b200_ctx *ctx, uint32_t channels, uint32_t sample_rate, const sea_b200_settings *settings,
                            sea_b200_encoder **out)
{
    if (!ctx || !settings || !out) return SEA_B200_ERR_INVALID_PARAMETERS;
    *out = nullptr;
    EncodePlan pl;
    int rc = make_encode_plan(channels, settings, &pl);
    if (rc) return fail(ctx, rc, "encoder settings rejected (outside the reference's domain)");
    CU(cudaSetDevice(ctx->device));
    sea_b200_encoder *enc = new sea_b200_encoder();
    enc->ctx = ctx;
    enc->settings = *settings;
    enc->plan = pl;
    enc->channels = channels;
    enc->sample_rate = sample_rate;
    std::vector<int32_t> init((size_t)channels * kEncStateWords, 0);
    for (uint32_t c = 0; c < channels; c++) {  // lms.rs:19-32
        init[(size_t)c * kEncStateWords + 4 + 2] = -(1 << 13);
        init[(size_t)c * kEncStateWords + 4 + 3] = 1 << 14;
    }
    cudaError_t e = cudaMalloc(&enc->d_state, init.size() * sizeof(int32_t));
    if (e == cudaSuccess) e = cudaMemcpy(enc->d_state, init.data(), init.size() * sizeof(int32_t), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) {
        if (enc->d_state) cudaFree(enc->d_state);
        delete enc;
        return cuda_fail(ctx, e, "encoder state");
    }
    *out = enc;
    return SEA_B200_OK;
}

uint32_t sea_b200_encoder_chunk_size(const sea_b200_encoder *enc) { return enc ? enc->chunk_size : 0; }

void sea_b200_encoder_destroy(sea_b200_encoder *enc)
{
    if (!enc) return;
    cudaSetDevice(enc->ctx->device);
    if (enc->d_state) cudaFree(enc->d_state);
    delete enc;
}

int sea_b200_encoder_make_chunks(sea_b200_encoder *enc, const int16_t *pcm, uint64_t n_samples, uint8_t *out, uint64_t out_cap,
                                 uint64_t *out_len, uint32_t *n_chunks)
{
    if (!enc || !pcm || !out || !out_len) return SEA_B200_ERR_INVALID_PARAMETERS;
    sea_b200_ctx *ctx = enc->ctx;
    const EncodePlan &pl = enc->plan;
    if (n_samples == 0 || n_samples % enc->channels) return fail(ctx, SEA_B200_ERR_INVALID_PARAMETERS, "make_chunk needs whole frames");
    const uint64_t frames64 = n_samples / enc->channels;
    if (frames64 > 0xffffffffull) return fail(ctx, SEA_B200_ERR_TOO_MANY_FRAMES, "more than 2^32 frames in one call");
    CU(cudaSetDevice(ctx->device));
    const uint32_t frames = (uint32_t)frames64;
    const uint32_t chunks = (frames + pl.N - 1) / pl.N;
    const uint64_t zero = 0;
    EncodeJob job;
    int rc = plan_encode(ctx, 1, &zero, &frames, enc->sample_rate, enc->channels, &enc->settings, &zero, true, &job);
    if (rc) return rc;
    // The kernel advances the handle's LMS / prev_scalefactor state, so a too-small buffer must be refused BEFORE the launch
    // (a caller retrying with a larger one would otherwise encode the same PCM from already-advanced state).
    if (out_cap < encode_bound_bytes(pl, frames) - kFileHeaderBytes)
        return fail(ctx, SEA_B200_ERR_CAPACITY, "chunk buffer smaller than the bound for these frames (sea_b200_encode_bound - 22)");
    CU(ctx->in.reserve(n_samples * 2 + 64));
    CU(ctx->out.reserve((uint64_t)chunks * pl.max_chunk_bytes + 64));
    CU(cudaMemcpyAsync(ctx->in.p, pcm, n_samples * 2, cudaMemcpyHostToDevice, ctx->stream));
    uint64_t len = 0;
    uint32_t first = 0;
    rc = run_encode(ctx, job, ctx->in.as<int16_t>(), ctx->out.as<uint8_t>(), enc->d_state, &len, &first);
    if (rc) return rc;
    if (len > out_cap) return fail(ctx, SEA_B200_ERR_CAPACITY, "chunk buffer too small");  // unreachable: len <= the bound above
    CU(cudaMemcpyAsync(out, ctx->out.p, len, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    if (enc->chunk_size == 0) enc->chunk_size = first & 0xffffu;  // file.rs:166-168 (`as u16`)
    if (frames >= pl.N && enc->chunk_size != (first & 0xffffu))
        return fail(ctx, SEA_B200_ERR_DOMAIN, "full chunk size differs from header.chunk_size (file.rs:173-175 assert)");
    *out_len = len;
    if (n_chunks) *n_chunks = chunks;
    return SEA_B200_OK;
}

int sea_b200_encoder_make_chunk(sea_b200_encoder *enc, const int16_t *pcm, uint64_t n_samples, uint8_t *out, uint64_t out_cap,
                                uint64_t *out_len)
{
    if (!enc) return SEA_B200_ERR_INVALID_PARAMETERS;
    if (n_samples / (enc->channels ? enc->channels : 1) > enc->plan.N)
        return fail(enc->ctx, SEA_B200_ERR_DOMAIN, "more than frames_per_chunk frames (file.rs:173-175 assert)");
    return sea_b200_encoder_make_chunks(enc, pcm, n_samples, out, out_cap, out_len, nullptr);
}

// ------------------------------------------------------------------------------------------------ session pool

int sea_b200_encoder_pool_create(sea_b200_ctx *ctx, uint32_t max_sessions, uint32_t channels, uint32_t sample_rate,
                                 const sea_b200_settings *settings, sea_b200_encoder_pool **pool)
{
    if (!ctx || !settings || !pool) return SEA_B200_ERR_INVALID_PARAMETERS;
    *pool = nullptr;
    if (max_sessions == 0) return fail(ctx, SEA_B200_ERR_INVALID_PARAMETERS, "a pool needs at least one session slot");
    EncodePlan pl;
    int rc = make_encode_plan(channels, settings, &pl);
    if (rc) return fail(ctx, rc, "encoder settings rejected (outside the reference's domain)");
    CU(cudaSetDevice(ctx->device));
    sea_b200_encoder_pool *p = new sea_b200_encoder_pool();
    p->ctx = ctx;
    p->settings = *settings;
    p->plan = pl;
    p->max_sessions = max_sessions;
    p->channels = channels;
    p->sample_rate = sample_rate;
    auto bail = [&](cudaError_t e, const char *what) {
        const int r = cuda_fail(ctx, e, what);
        sea_b200_encoder_pool_destroy(p);
        return r;
    };
    const size_t row = (size_t)channels * kEncStateWords;
    cudaError_t e = cudaMalloc(&p->d_carry, (size_t)max_sessions * 2u * pl.N * channels * sizeof(int16_t));
    if (e != cudaSuccess) return bail(e, "cudaMalloc(pool carry buffers)");
    if ((e = cudaMalloc(&p->d_state, (size_t)max_sessions * row * sizeof(int32_t))) != cudaSuccess) return bail(e, "cudaMalloc(pool state)");
    std::vector<int32_t> init(row, 0);
    for (uint32_t c = 0; c < channels; c++) {  // lms.rs:19-32
        init[(size_t)c * kEncStateWords + 4 + 2] = -(1 << 13);
        init[(size_t)c * kEncStateWords + 4 + 3] = 1 << 14;
    }
    if ((e = cudaMalloc(&p->d_init, row * sizeof(int32_t))) != cudaSuccess) return bail(e, "cudaMalloc(pool initial state)");
    if ((e = cudaMemcpy(p->d_init, init.data(), row * sizeof(int32_t), cudaMemcpyHostToDevice)) != cudaSuccess)
        return bail(e, "cudaMemcpy(pool initial state)");
    for (cudaEvent_t &ev : p->ev)
        if ((e = cudaEventCreate(&ev)) != cudaSuccess) return bail(e, "cudaEventCreate");
    p->carry.assign(max_sessions, 0);
    p->half.assign(max_sessions, 0);
    p->open.assign(max_sessions, 0);
    p->fresh.assign(max_sessions, 1);
    p->seen.assign(max_sessions, 0);
    *pool = p;
    return SEA_B200_OK;
}

void sea_b200_encoder_pool_destroy(sea_b200_encoder_pool *pool)
{
    if (!pool) return;
    cudaSetDevice(pool->ctx->device);
    if (pool->ctx->stream) cudaStreamSynchronize(pool->ctx->stream);
    if (pool->d_carry) cudaFree(pool->d_carry);
    if (pool->d_state) cudaFree(pool->d_state);
    if (pool->d_init) cudaFree(pool->d_init);
    pool->pk.release();
    pool->in.release();
    pool->rows.release();
    pool->ob.release();
    pool->desc.release();
    if (pool->h_desc) cudaFreeHost(pool->h_desc);
    for (cudaEvent_t ev : pool->ev)
        if (ev) cudaEventDestroy(ev);
    delete pool;
}

int sea_b200_encoder_pool_open(sea_b200_encoder_pool *pool, uint32_t n, const uint32_t *sessions)
{
    if (!pool) return SEA_B200_ERR_INVALID_PARAMETERS;
    sea_b200_ctx *ctx = pool->ctx;
    if (n == 0) return SEA_B200_OK;
    if (!sessions) return fail(ctx, SEA_B200_ERR_INVALID_PARAMETERS, "NULL session list");
    if (++pool->stamp == 0) {
        std::fill(pool->seen.begin(), pool->seen.end(), 0u);
        pool->stamp = 1;
    }
    for (uint32_t i = 0; i < n; i++) {
        const uint32_t s = sessions[i];
        if (s >= pool->max_sessions || pool->open[s] || pool->seen[s] == pool->stamp)
            return fail(ctx, SEA_B200_ERR_INVALID_PARAMETERS, "session " + std::to_string(s) + " (entry " + std::to_string(i) + ")" +
                                                                  (s >= pool->max_sessions ? " is past max_sessions" : pool->open[s] ? " is already open" : " appears twice"));
        pool->seen[s] = pool->stamp;
    }
    // host-side only: the slot's first push gathers its state from the EncoderBase::new row
    for (uint32_t i = 0; i < n; i++) {
        const uint32_t s = sessions[i];
        pool->open[s] = 1;
        pool->fresh[s] = 1;
        pool->carry[s] = 0;
        pool->half[s] = 0;
    }
    return SEA_B200_OK;
}

int sea_b200_encoder_pool_buffered(const sea_b200_encoder_pool *pool, uint32_t n, const uint32_t *sessions, uint32_t *frames)
{
    if (!pool) return SEA_B200_ERR_INVALID_PARAMETERS;
    if (n && (!sessions || !frames)) return fail(pool->ctx, SEA_B200_ERR_INVALID_PARAMETERS, "NULL pointer");
    for (uint32_t i = 0; i < n; i++)
        if (sessions[i] >= pool->max_sessions) return fail(pool->ctx, SEA_B200_ERR_INVALID_PARAMETERS, "session past max_sessions");
    for (uint32_t i = 0; i < n; i++) frames[i] = pool->open[sessions[i]] ? pool->carry[sessions[i]] : 0u;
    return SEA_B200_OK;
}

}  // extern "C"

namespace {

// Bytes a push of n_frames more frames gives an open session: k full chunks, plus with `end` the bound of its short final chunk
// (exact for CBR; sea_b200_encode_bound's for VBR, whose last chunk size is only known once it is encoded).
uint64_t pool_bound(const EncodePlan &pl, uint64_t total_frames, bool end)
{
    if (end) return encode_bound_bytes(pl, total_frames) - kFileHeaderBytes;
    return total_frames / pl.N * pl.full_chunk_bytes;
}

int pool_push(sea_b200_encoder_pool *pool, uint32_t n, const uint32_t *sessions, const int16_t *pcm, const uint64_t *pcm_offsets,
              const uint32_t *n_frames, const uint8_t *end, uint8_t *out, const uint64_t *out_offsets, const uint64_t *out_caps,
              uint64_t *out_lens, uint32_t *n_chunks, bool device)
{
    if (!pool) return SEA_B200_ERR_INVALID_PARAMETERS;
    sea_b200_ctx *ctx = pool->ctx;
    if (n == 0) return SEA_B200_OK;
    if (!sessions || !pcm_offsets || !n_frames || !out_offsets || !out_lens) return fail(ctx, SEA_B200_ERR_INVALID_PARAMETERS, "NULL pointer");
    const EncodePlan &pl = pool->plan;
    const uint32_t C = pool->channels, N = pl.N, row = C * kEncStateWords;
    const uint64_t slot_elems = (uint64_t)N * C;

    // ---- every refusal comes before anything is enqueued or any session's bookkeeping moves
    if (++pool->stamp == 0) {
        std::fill(pool->seen.begin(), pool->seen.end(), 0u);
        pool->stamp = 1;
    }
    std::vector<uint32_t> enc_frames(n);
    std::vector<uint64_t> bound(n);
    uint64_t lo = UINT64_MAX, hi = 0, out_total = 0;
    bool vbr_tail = false;  // some session ends with a VBR short chunk: its size is read back before the output can be copied
    for (uint32_t i = 0; i < n; i++) {
        const uint32_t s = sessions[i];
        auto who = [&]() { return "session " + std::to_string(s) + " (entry " + std::to_string(i) + ")"; };
        if (s >= pool->max_sessions) return fail(ctx, SEA_B200_ERR_INVALID_PARAMETERS, who() + " is past max_sessions");
        if (!pool->open[s]) return fail(ctx, SEA_B200_ERR_INVALID_PARAMETERS, who() + " is not open");
        if (pool->seen[s] == pool->stamp) return fail(ctx, SEA_B200_ERR_INVALID_PARAMETERS, who() + " appears twice in one push");
        pool->seen[s] = pool->stamp;
        const uint64_t tot = (uint64_t)pool->carry[s] + n_frames[i];
        if (tot > 0xffffffffull) return fail(ctx, SEA_B200_ERR_TOO_MANY_FRAMES, who() + ": buffered plus pushed frames exceed 2^32");
        const bool e = end && end[i];
        enc_frames[i] = (uint32_t)(e ? tot : tot / N * N);
        bound[i] = pool_bound(pl, tot, e);
        if (out_caps && out_caps[i] < bound[i])
            return fail(ctx, SEA_B200_ERR_CAPACITY, who() + ": out_caps smaller than sea_b200_encoder_pool_push_bound");
        if (e && pl.vbr && tot % N) vbr_tail = true;
        if (n_frames[i]) {
            lo = std::min(lo, pcm_offsets[i]);
            hi = std::max(hi, pcm_offsets[i] + (uint64_t)n_frames[i] * C);
        }
        out_total += bound[i];
    }
    if (hi && !pcm) return fail(ctx, SEA_B200_ERR_INVALID_PARAMETERS, "NULL pcm");
    if (out_total && !out) return fail(ctx, SEA_B200_ERR_INVALID_PARAMETERS, "NULL out");
    if (hi == 0) lo = 0;

    // ---- the encode launch: one stream per session that completes a chunk or ends with frames, in call order
    std::vector<uint32_t> launch;  // call index of launch stream j
    std::vector<uint64_t> in_off, enc_out_off;
    std::vector<uint32_t> frames_j;
    uint64_t in_total = 0, ob_total = 0;
    for (uint32_t i = 0; i < n; i++) {
        if (!enc_frames[i]) continue;
        launch.push_back(i);
        in_off.push_back(in_total);
        in_total += ((uint64_t)enc_frames[i] * C + 7u) & ~7ull;  // 16-byte aligned rows: whole-vector stores for most of them
        frames_j.push_back(enc_frames[i]);
        enc_out_off.push_back(device ? out_offsets[i] : ob_total);
        ob_total += bound[i];
    }
    const uint32_t nl = (uint32_t)launch.size();
    EncodeJob job;
    if (nl) {
        int rc = plan_encode(ctx, nl, in_off.data(), frames_j.data(), pool->sample_rate, C, &pool->settings, enc_out_off.data(), true, &job);
        if (rc) return rc;
    }
    CU(cudaSetDevice(ctx->device));
    // pinned staging: the copy list (at most three copies and a state row per session), the launch's slots, its EncStreams
    const size_t max_copies = (size_t)n * 3u + nl;
    const size_t enc_at = (sizeof(PoolCopy) * max_copies + sizeof(uint32_t) * nl + 15u) & ~(size_t)15u;
    const size_t desc_bytes = enc_at + sizeof(EncStream) * nl;
    CU(pool->desc.reserve(desc_bytes));
    if (pool->h_desc_cap < desc_bytes) {
        if (pool->h_desc) cudaFreeHost(pool->h_desc);
        pool->h_desc = nullptr;
        pool->h_desc_cap = 0;
        CU(cudaHostAlloc(reinterpret_cast<void **>(&pool->h_desc), desc_bytes + (desc_bytes >> 2), cudaHostAllocDefault));
        pool->h_desc_cap = desc_bytes + (desc_bytes >> 2);
    }
    CU(pool->in.reserve(in_total * sizeof(int16_t) + 64));
    CU(pool->rows.reserve((size_t)nl * row * sizeof(int32_t) + 64));
    if (!device) {
        CU(pool->pk.reserve((hi - lo) * sizeof(int16_t) + 64));
        CU(pool->ob.reserve(ob_total + 64));
    }
    if (nl) {
        CU(ctx->streams.reserve(sizeof(EncStream) * nl));
        CU(ctx->lens.reserve(sizeof(uint64_t) * nl));
        CU(ctx->chunk0.reserve(sizeof(uint32_t) * nl));
        CU(ctx->ties.reserve(sizeof(unsigned long long) * ((size_t)nl + 1u)));
    }

    // ---- the ingest's copies, in call order (device pointers are final now)
    PoolCopy *copies = reinterpret_cast<PoolCopy *>(pool->h_desc);
    uint32_t n_copies = 0;
    uint64_t vectors = 0;
    auto add = [&](const int16_t *src, int16_t *dst, uint64_t elems) {
        if (!elems) return;
        PoolCopy &c = copies[n_copies++];
        c.src = src;
        c.dst = dst;
        c.n = elems;
        c.v_begin = vectors;
        const uint64_t d = reinterpret_cast<uintptr_t>(dst);
        vectors += ((d + 2u * elems + 15u) >> 4) - (d >> 4);
    };
    int16_t *d_in = pool->in.as<int16_t>();
    int32_t *d_rows = pool->rows.as<int32_t>();
    for (uint32_t i = 0, j = 0; i < n; i++) {
        const uint32_t s = sessions[i], c = pool->carry[s];
        const int16_t *packet = !n_frames[i] ? nullptr : device ? pcm + pcm_offsets[i] : pool->pk.as<int16_t>() + (pcm_offsets[i] - lo);
        int16_t *cur = pool->d_carry + ((uint64_t)s * 2u + pool->half[s]) * slot_elems;
        int16_t *nxt = pool->d_carry + ((uint64_t)s * 2u + (pool->half[s] ^ 1u)) * slot_elems;
        if (!enc_frames[i]) {  // no chunk completes: the packet is appended behind the carry, in place
            add(packet, cur + (uint64_t)c * C, (uint64_t)n_frames[i] * C);
            continue;
        }
        // carry + the packet's first enc_frames - c frames -> launch input; the remainder -> the other carry half
        int16_t *dst = d_in + in_off[j];
        const uint64_t take = enc_frames[i] - c, rest = (uint64_t)c + n_frames[i] - enc_frames[i];
        add(cur, dst, (uint64_t)c * C);
        add(packet, dst + (uint64_t)c * C, take * C);
        if (rest) add(packet + take * C, nxt, rest * C);
        const int32_t *src_row = pool->fresh[s] ? pool->d_init : pool->d_state + (uint64_t)s * row;
        add(reinterpret_cast<const int16_t *>(src_row), reinterpret_cast<int16_t *>(d_rows + (uint64_t)j * row), 2ull * row);
        j++;
    }
    uint32_t *slots = reinterpret_cast<uint32_t *>(pool->h_desc + sizeof(PoolCopy) * n_copies);
    for (uint32_t j = 0; j < nl; j++) slots[j] = sessions[launch[j]];
    if (nl) memcpy(pool->h_desc + enc_at, job.streams.data(), sizeof(EncStream) * nl);
    const PoolCopy *d_copies = pool->desc.as<PoolCopy>();
    const uint32_t *d_slots = reinterpret_cast<const uint32_t *>(pool->desc.as<uint8_t>() + sizeof(PoolCopy) * n_copies);

    // ---- enqueue, wait, copy back.  From here on a failure leaves the device state of the call's sessions undefined: they are
    // closed.
    std::vector<unsigned long long> dev_ties;
    std::vector<uint64_t> lens_j(nl);
    auto run = [&]() -> int {
        cudaStream_t st = ctx->stream;
        if (!device && hi) CU(cudaMemcpyAsync(pool->pk.p, pcm + lo, (hi - lo) * sizeof(int16_t), cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(pool->desc.p, pool->h_desc, sizeof(PoolCopy) * n_copies + sizeof(uint32_t) * nl, cudaMemcpyHostToDevice, st));
        if (nl) CU(cudaMemcpyAsync(ctx->streams.p, pool->h_desc + enc_at, sizeof(EncStream) * nl, cudaMemcpyHostToDevice, st));
        CU(cudaEventRecord(pool->ev[0], st));
        if (n_copies) {
            CU(launch_pool_ingest(d_copies, n_copies, vectors, st));
            ctx->launches++;
        }
        CU(cudaEventRecord(pool->ev[1], st));
        int dev_err = 0;
        if (nl) {
            CU(cudaMemsetAsync(ctx->d_err, 0, sizeof(int), st));
            CU(cudaMemsetAsync(ctx->ties.p, 0, sizeof(unsigned long long) * ((size_t)nl + 1u), st));
            int rc = enqueue_encode(ctx, job, d_in, device ? out : pool->ob.as<uint8_t>(), d_rows, 0, true);
            if (rc) return rc;
            CU(cudaEventRecord(pool->ev[2], st));
            CU(launch_pool_commit(d_rows, pool->d_state, d_slots, nl, row, st));
            ctx->launches++;
            CU(cudaEventRecord(pool->ev[3], st));
            CU(cudaMemcpyAsync(&dev_err, ctx->d_err, sizeof(int), cudaMemcpyDeviceToHost, st));
            if (pl.vbr) {
                dev_ties.assign((size_t)nl + 1u, 0ull);
                CU(cudaMemcpyAsync(dev_ties.data(), ctx->ties.p, sizeof(unsigned long long) * ((size_t)nl + 1u), cudaMemcpyDeviceToHost, st));
            }
            if (vbr_tail) CU(cudaMemcpyAsync(lens_j.data(), ctx->lens.p, sizeof(uint64_t) * nl, cudaMemcpyDeviceToHost, st));
        } else {
            CU(cudaEventRecord(pool->ev[2], st));
            CU(cudaEventRecord(pool->ev[3], st));
        }
        // a full chunk is full_chunk_bytes exactly and a CBR short chunk follows from its frame count: those sizes are known here,
        // and the output goes back in the same stream segment; a VBR short chunk has to be read back first
        auto copy_back = [&]() -> int {
            if (device) return SEA_B200_OK;
            for (uint32_t j = 0; j < nl;) {  // one copy per run of sessions adjacent both in the staging buffer and in `out`
                uint32_t k = j + 1;
                uint64_t len = lens_j[j];
                while (k < nl && enc_out_off[k] == enc_out_off[j] + len && out_offsets[launch[k]] == out_offsets[launch[j]] + len) len += lens_j[k++];
                if (len) CU(cudaMemcpyAsync(out + out_offsets[launch[j]], pool->ob.as<uint8_t>() + enc_out_off[j], len, cudaMemcpyDeviceToHost, st));
                j = k;
            }
            return SEA_B200_OK;
        };
        if (!vbr_tail) {
            for (uint32_t j = 0; j < nl; j++) {
                const uint32_t f = frames_j[j], rem = f % N;
                lens_j[j] = (uint64_t)(f / N) * pl.full_chunk_bytes + (rem ? cbr_chunk_bytes(rem, C, pl.s, pl.F, pl.hdr_bits) : 0u);
            }
            if (int rc = copy_back()) return rc;
        }
        CU(cudaStreamSynchronize(st));
        if (dev_err != kDevOk) return map_dev_error(ctx, dev_err);
        if (vbr_tail) {
            if (int rc = copy_back()) return rc;
            CU(cudaStreamSynchronize(st));
        }
        return SEA_B200_OK;
    };
    const int rc = run();
    if (rc != SEA_B200_OK) {
        for (uint32_t i = 0; i < n; i++) {
            pool->open[sessions[i]] = 0;
            pool->carry[sessions[i]] = 0;
        }
        return rc;
    }

    // ---- results and the sessions' bookkeeping
    float ms[3] = {0.f, 0.f, 0.f};
    cudaEventElapsedTime(&ms[0], pool->ev[0], pool->ev[1]);
    cudaEventElapsedTime(&ms[1], pool->ev[1], pool->ev[2]);
    cudaEventElapsedTime(&ms[2], pool->ev[2], pool->ev[3]);
    ctx->last_kernel_ms = (double)ms[0] + ms[1] + ms[2];
    if (getenv("SEA_B200_TRACE"))
        fprintf(stderr, "sea_b200 trace: pool push: %u sessions, %u encode, %u copies; ingest %.3f ms, encode %.3f ms, commit %.3f ms\n", n, nl,
                n_copies, ms[0], ms[1], ms[2]);
    ctx->h_ties.assign((size_t)n + 1u, 0ull);  // call order
    for (uint32_t j = 0; j < nl && pl.vbr; j++) ctx->h_ties[1u + launch[j]] = dev_ties[1u + j];
    ctx->h_ties[0] = pl.vbr && nl ? dev_ties[0] : 0ull;
    ctx->last_ties = ctx->h_ties[0];
    for (uint32_t i = 0; i < n; i++) {
        out_lens[i] = 0;
        if (n_chunks) n_chunks[i] = (enc_frames[i] + N - 1u) / N;
    }
    for (uint32_t j = 0; j < nl; j++) out_lens[launch[j]] = lens_j[j];
    for (uint32_t i = 0; i < n; i++) {
        const uint32_t s = sessions[i];
        const uint64_t tot = (uint64_t)pool->carry[s] + n_frames[i];
        if (end && end[i]) {
            pool->open[s] = 0;
            pool->carry[s] = 0;
        } else if (enc_frames[i]) {
            pool->carry[s] = (uint32_t)(tot - enc_frames[i]);
            pool->half[s] ^= 1u;
        } else {
            pool->carry[s] = (uint32_t)tot;
        }
        if (enc_frames[i]) pool->fresh[s] = 0;
    }
    return SEA_B200_OK;
}

}  // namespace

extern "C" {

int sea_b200_encoder_pool_push_bound(const sea_b200_encoder_pool *pool, uint32_t session, uint64_t n_frames, bool end, uint64_t *bytes)
{
    if (!pool || !bytes) return SEA_B200_ERR_INVALID_PARAMETERS;
    if (session >= pool->max_sessions || !pool->open[session])
        return fail(pool->ctx, SEA_B200_ERR_INVALID_PARAMETERS, "session " + std::to_string(session) + " is not open");
    const uint64_t tot = pool->carry[session] + n_frames;
    if (n_frames > 0xffffffffull || tot > 0xffffffffull)
        return fail(pool->ctx, SEA_B200_ERR_TOO_MANY_FRAMES, "buffered plus pushed frames exceed 2^32");
    *bytes = pool_bound(pool->plan, tot, end);
    return SEA_B200_OK;
}

int sea_b200_encoder_pool_push(sea_b200_encoder_pool *pool, uint32_t n, const uint32_t *sessions, const int16_t *pcm,
                               const uint64_t *pcm_offsets, const uint32_t *n_frames, const uint8_t *end, uint8_t *out,
                               const uint64_t *out_offsets, const uint64_t *out_caps, uint64_t *out_lens, uint32_t *n_chunks)
{
    return pool_push(pool, n, sessions, pcm, pcm_offsets, n_frames, end, out, out_offsets, out_caps, out_lens, n_chunks, false);
}

int sea_b200_encoder_pool_push_device(sea_b200_encoder_pool *pool, uint32_t n, const uint32_t *sessions, const int16_t *d_pcm,
                                      const uint64_t *pcm_offsets, const uint32_t *n_frames, const uint8_t *end, uint8_t *d_out,
                                      const uint64_t *out_offsets, const uint64_t *out_caps, uint64_t *out_lens, uint32_t *n_chunks)
{
    return pool_push(pool, n, sessions, d_pcm, pcm_offsets, n_frames, end, d_out, out_offsets, out_caps, out_lens, n_chunks, true);
}

int sea_b200_decoder_create(sea_b200_ctx *ctx, const uint8_t *header22, uint64_t len, sea_b200_decoder **out)
{
    if (!ctx || !header22 || !out) return SEA_B200_ERR_INVALID_PARAMETERS;
    *out = nullptr;
    sea_b200_header h;
    int rc = parse_file_header(header22, len, &h);
    if (rc) return fail(ctx, rc, "bad .sea header (file.rs:40-72)");
    sea_b200_decoder *dec = new sea_b200_decoder();
    dec->ctx = ctx;
    dec->header = h;
    *out = dec;
    return SEA_B200_OK;
}

int sea_b200_decoder_header(const sea_b200_decoder *dec, sea_b200_header *out)
{
    if (!dec || !out) return SEA_B200_ERR_INVALID_PARAMETERS;
    *out = dec->header;
    return SEA_B200_OK;
}

void sea_b200_decoder_destroy(sea_b200_decoder *dec) { delete dec; }

// Decoder::init + the scale_factor_bits assert of codec/decoder.rs:21 for a run of chunks (`stride` bytes apart): the first
// chunk a handle sees fixes scale_factor_bits, every later one must agree.  Shared by decode_chunk and decode_chunks.
__attribute__((visibility("hidden"))) int sea_b200_internal_check_sf_bits(sea_b200_decoder *dec, const uint8_t *chunks, uint64_t len,
                                                                         uint64_t stride)
{
    for (uint64_t off = 0; off + 2 <= len; off += stride) {
        const int sfb = chunks[off + 1] >> 4;
        if (dec->sf_bits < 0) dec->sf_bits = sfb;
        else if (dec->sf_bits != sfb) return fail(dec->ctx, SEA_B200_ERR_DOMAIN, "scale_factor_bits changed between chunks (decoder.rs:21 assert)");
    }
    return SEA_B200_OK;
}

int sea_b200_decoder_decode_chunk(sea_b200_decoder *dec, const uint8_t *chunk, uint64_t len, int64_t remaining_frames, int16_t *pcm,
                                  uint64_t pcm_cap_samples, uint64_t *n_samples)
{
    if (!dec || !chunk || !pcm || !n_samples) return SEA_B200_ERR_INVALID_PARAMETERS;
    sea_b200_ctx *ctx = dec->ctx;
    const sea_b200_header &h = dec->header;
    *n_samples = 0;
    if (len == 0) return fail(ctx, SEA_B200_ERR_INVALID_PARAMETERS, "empty chunk (samples_from_reader returns None before parsing)");
    if (len > h.chunk_size) return fail(ctx, SEA_B200_ERR_DOMAIN, "chunk longer than header.chunk_size (chunk.rs:74 assert)");
    if (remaining_frames < 0 && len < h.chunk_size) return fail(ctx, SEA_B200_ERR_INVALID_FRAME, "short chunk in streaming mode (chunk.rs:76-79)");
    if (len < 4) return fail(ctx, SEA_B200_ERR_DOMAIN, "chunk shorter than its header");
    if (chunk[0] != 1 && chunk[0] != 2) return fail(ctx, SEA_B200_ERR_INVALID_FRAME, "chunk type is neither CBR nor VBR (chunk.rs:81-85)");
    if (int rcs = sea_b200_internal_check_sf_bits(dec, chunk, len, h.chunk_size)) return rcs;
    uint64_t frames = h.frames_per_chunk;
    if (remaining_frames >= 0 && (uint64_t)remaining_frames < frames) frames = (uint64_t)remaining_frames;
    if (frames == 0) return SEA_B200_OK;
    if (frames * h.channels > pcm_cap_samples) return fail(ctx, SEA_B200_ERR_CAPACITY, "PCM buffer too small");
    CU(cudaSetDevice(ctx->device));
    DecodeJob job;
    job.streams.resize(1);
    job.n_samples.assign(1, frames * h.channels);
    DecStream &d = job.streams[0];
    memset(&d, 0, sizeof(d));
    d.data_off = 0;
    d.data_len = len;
    d.pcm_off = 0;
    d.total_frames = (uint32_t)frames;
    d.n_chunks = 1;
    d.chain_begin = 0;
    d.chunk_size = h.chunk_size;
    d.frames_per_chunk = h.frames_per_chunk;
    d.channels = h.channels;
    job.total_chains = h.channels;
    job.first = h;
    // One chunk is a serial chain per channel -- latency, not throughput.  The host already holds the chunk's header word, so
    // mono / stereo chunks go to the staged kernel (residuals through shared memory: ~3x shorter chain steps than the generic
    // kernel's global-memory bit reads); run_decode falls back to the generic kernel for anything it does not cover.
    job.uniform = true;
    const uint32_t hdr_word = (uint32_t)chunk[0] | ((uint32_t)chunk[1] << 8) | ((uint32_t)chunk[2] << 16) | ((uint32_t)chunk[3] << 24);
    CU(ctx->in.reserve(len + 64));
    CU(ctx->out.reserve(frames * h.channels * 2 + 64));
    CU(cudaMemcpyAsync(ctx->in.p, chunk, len, cudaMemcpyHostToDevice, ctx->stream));
    DecLane L = decode_lane(ctx, 0);
    bool copied = false;
    int rc = run_decode(ctx, L, job, ctx->in.as<uint8_t>(), len, ctx->out.as<int16_t>(), true, hdr_word, pcm, frames * h.channels * 2, &copied);
    if (rc) return rc;
    if (!copied) {
        CU(cudaMemcpyAsync(pcm, ctx->out.p, frames * h.channels * 2, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
    }
    *n_samples = frames * h.channels;
    return SEA_B200_OK;
}

// ------------------------------------------------------------------------------------------------ measurement

int sea_b200_synth_pcm_device(sea_b200_ctx *ctx, int16_t *d_pcm, uint64_t stream_stride_samples, uint32_t n_streams, uint32_t n_frames,
                              uint32_t channels, const uint32_t *stream_ids, const uint32_t *phase_steps, const int32_t *sine_table_4096,
                              uint64_t seed, int32_t amplitude, int32_t noise_amplitude)
{
    if (!ctx || !d_pcm || !stream_ids || !phase_steps || !sine_table_4096 || channels == 0 || noise_amplitude < 0)
        return SEA_B200_ERR_INVALID_PARAMETERS;
    if (n_streams == 0 || n_frames == 0) return SEA_B200_OK;
    CU(cudaSetDevice(ctx->device));
    const size_t idb = sizeof(uint32_t) * (size_t)n_streams;
    CU(ctx->misc.reserve(2 * idb + 4096 * sizeof(int32_t) + 256));
    uint8_t *base = ctx->misc.as<uint8_t>();
    const size_t tab_off = (2 * idb + 255) & ~(size_t)255;
    CU(cudaMemcpyAsync(base, stream_ids, idb, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemcpyAsync(base + idb, phase_steps, idb, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemcpyAsync(base + tab_off, sine_table_4096, 4096 * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream));
    CU(launch_synth(d_pcm, stream_stride_samples, n_streams, n_frames, channels, reinterpret_cast<const uint32_t *>(base),
                    reinterpret_cast<const uint32_t *>(base + idb), reinterpret_cast<const int32_t *>(base + tab_off), seed, amplitude,
                    noise_amplitude, ctx->stream));
    ctx->launches += (n_streams + 65534u) / 65535u;
    CU(cudaStreamSynchronize(ctx->stream));  // the id / step / table arrays are the caller's: done with them on return
    return SEA_B200_OK;
}

int sea_b200_int32_peak(sea_b200_ctx *ctx, int mode, double *ops_per_s, double *ms_out)
{
    if (!ctx || mode < 0 || mode > 2) return SEA_B200_ERR_INVALID_PARAMETERS;
    CU(cudaSetDevice(ctx->device));
    CU(ctx->misc.reserve(256));
    uint64_t lane_ops = 0;
    float best = 1e30f;
    for (int rep = 0; rep < 5; rep++) {
        CU(cudaEventRecord(ctx->ev0, ctx->stream));
        CU(launch_int32_peak(mode, ctx->misc.as<uint32_t>(), &lane_ops, ctx->stream));
        ctx->launches++;
        CU(cudaEventRecord(ctx->ev1, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
        float ms = 0;
        cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1);
        if (rep > 0 && ms < best) best = ms;
    }
    if (ms_out) *ms_out = best;
    if (ops_per_s) *ops_per_s = (double)lane_ops / ((double)best * 1e-3);
    return SEA_B200_OK;
}

}  // extern "C"
