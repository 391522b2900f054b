// sea_kernels.h -- launch interface between the C-ABI layer (capi.cu) and the CUDA kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include "sea_common.cuh"

namespace sea {

// Device-side error codes written to the error word by kernels (first failure wins).
enum : int { kDevOk = 0, kDevInvalidFrame = 1, kDevDomain = 2, kDevFallback = 3 /* staged kernel: use the generic path */ };

// ---- decode ------------------------------------------------------------------------------------------------
// One entry per stream; chains (chunk, channel) of all streams are numbered consecutively.
struct DecStream {
    uint64_t data_off;      // byte offset of the first chunk inside the batch buffer
    uint64_t data_len;      // bytes available from data_off
    uint64_t pcm_off;       // sample offset of the stream's PCM inside the output buffer
    uint32_t total_frames;  // frames to produce (resolved by the host, decoder.rs:33-44)
    uint32_t n_chunks;
    uint32_t chain_begin;   // global id of the stream's first chain
    uint16_t chunk_size;
    uint16_t frames_per_chunk;
    uint32_t channels;
    uint32_t pad;
};

// Generic path: any per-chunk (type, sf bits, residual size, sf frames), any channel count, any alignment.
cudaError_t launch_decode_generic(const uint8_t *d_sea, int16_t *d_pcm, const DecStream *d_streams, uint32_t n_streams,
                                  uint64_t total_chains, DevTables tabs, int *d_err, cudaStream_t stream);

// Fast path: uniform batch (every chunk CBR with the same header word, channels C in {1,2}); falls back is the
// caller's job when *d_err reports a chunk whose header differs.
struct DecFastParams {
    uint32_t channels, N, chunk_size, F, s, b;
    uint32_t hdr_word;       // expected little-endian first 4 bytes of every chunk
    uint32_t n_streams;
    uint64_t total_chunks;
};
bool decode_fast_supported(const DecFastParams &p);
cudaError_t launch_decode_fast(const uint8_t *d_sea, uint64_t sea_len, int16_t *d_pcm, const DecStream *d_streams,
                               const DecFastParams &p, DevTables tabs, int *d_err, cudaStream_t stream);

// Throughput path (decode_fast.cuh): CBR, 1 or 2 channels, scale_factor_frames = 20, FULL chunks only (a whole number of 80-sample
// halves), PCM offsets multiples of 16 samples, and >= 128 readable bytes after every chunk it is given (staged rows over-read a little).
bool decode_unrolled_supported(const DecFastParams &p);
cudaError_t launch_decode_unrolled(const uint8_t *d_sea, int16_t *d_pcm, const DecStream *d_streams, const DecFastParams &p,
                                   DevTables tabs, int *d_err, cudaStream_t stream);

// VBR twin (decode_vbr.cu): VBR chunks, 1 or 2 channels, scale_factor_bits <= 6, scale_factor_frames = 20, FULL chunks only (a whole
// number of 80-sample bodies), the same alignment rules, >= 320 readable bytes after every chunk it is given.
bool decode_vbr_supported(const DecFastParams &p);
cudaError_t launch_decode_vbr(const uint8_t *d_sea, int16_t *d_pcm, const DecStream *d_streams, const DecFastParams &p, DevTables tabs,
                              int *d_err, cudaStream_t stream);

// More than two channels (decode_mc.cuh, decode_mc.cu, decode_mc_odd.cu): CBR, 3 .. 8 channels, scale_factor_bits <= 6,
// scale_factor_frames = 20, FULL chunks only (frames per chunk a multiple of 20 / 40 / 80 for 4 and 8 / 6 / odd channel counts), the
// same alignment rules, >= 512 readable bytes after every chunk it is given.
bool decode_mc_supported(const DecFastParams &p);
cudaError_t launch_decode_mc(const uint8_t *d_sea, int16_t *d_pcm, const DecStream *d_streams, const DecFastParams &p, DevTables tabs,
                             int *d_err, cudaStream_t stream);

// Small jobs (decode_latency.cu): one warp per chunk, any per-chunk header, <= 32 channels; every stream of the launch must share
// chunk_size / frames_per_chunk / channels.  decode_latency_smem() == 0: geometry not supported.
size_t decode_latency_smem(uint32_t chunk_size, uint32_t frames_per_chunk, uint32_t channels);
cudaError_t launch_decode_latency(const uint8_t *d_sea, int16_t *d_pcm, const DecStream *d_streams, uint32_t n_streams, uint64_t total_chunks,
                                  uint32_t chunk_size, uint32_t frames_per_chunk, uint32_t channels, DevTables tabs, int *d_err,
                                  cudaStream_t stream);

// Warps per CTA for the lane-per-chunk kernels (one full-width CTA per SM is their design point).  A grid of only a few waves
// of such CTAs ends with most SMs idle while the last wave drains (BASELINE config 3 shape: 2.5 waves -> 16 % lost), so short
// grids are cut into narrower CTAs -- the same warps per SM, several CTAs resident -- until the tail is a small share.
inline uint32_t pick_cta_warps(uint64_t total_chunks, uint32_t chunks_per_warp, uint32_t max_warps)
{
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    uint32_t warps = max_warps;
    if (getenv("SEA_B200_FULL_CTAS")) return warps;  // tests / tuning: the full-width CTA (and what only it selects) whatever the job size
    while (warps > 4u && warps % 2u == 0u) {
        const uint64_t per_cta = (uint64_t)warps * chunks_per_warp;
        const uint64_t ctas = (total_chunks + per_cta - 1) / per_cta;
        if (ctas >= (uint64_t)sms * (max_warps / warps) * 12u) break;  // >= 12 waves: the tail is under ~4 %
        warps /= 2u;
    }
    return warps;
}

// Window cut (window_kernels.cu): one descriptor per window of sea_b200_decode_windows_device.  The covering chunks were decoded
// into a scratch buffer; the kernel writes the slot: `real` frames from scratch, then zeros up to `frames`.
struct WinDesc {
    uint64_t src;       // scratch sample offset of the window's first frame (covering range start + skip * channels)
    uint64_t dst;       // element offset of the slot in the output
    uint32_t real;      // frames copied from scratch
    uint32_t frames;    // frames of the slot
    uint32_t channels;
    uint32_t pad;
};
// planar_f32 = false: int16 interleaved [frames][channels]; true: float32 planar [channels][frames], sample / 32768.
// max_slot_samples: the largest frames * channels of the launch (sizes the grid).
cudaError_t launch_window_extract(const int16_t *d_scratch, void *d_out, const WinDesc *d_desc, uint32_t n_windows, uint64_t max_slot_samples,
                                  bool planar_f32, cudaStream_t stream);

// Registered corpus (corpus_kernels.cu, sea_b200_corpus_*): one entry per stream, made once at create.
struct CorpusStream {
    uint64_t body;         // byte offset of chunk 0 in the corpus buffer (plan_range's body + the stream's offset)
    uint64_t len;          // bytes of the stream from body on
    uint64_t file_frames;  // frames a window can draw from (plan_range's file_frames)
    uint64_t chunk_begin;  // global index of the stream's chunk 0 among the chunks create validates
    uint32_t chunk_size, N, n_chunks;  // n_chunks = ceil(file_frames / N): every chunk a window can cover
    uint32_t pad;
};
// Create-time validation: every chunk of every stream at its true frame count, with decode_generic_kernel's checks.  *d_first_bad:
// min over failing chunks of (global chunk << 2 | kDev code), left at ~0 when none fails.  *d_mixed: nonzero when some chunk's
// 4-byte header word differs from ref_word.
cudaError_t launch_corpus_validate(const uint8_t *d_sea, const CorpusStream *d_streams, uint32_t n_streams, uint64_t total_chunks,
                                   uint32_t channels, uint32_t ref_word, unsigned long long *d_first_bad, uint32_t *d_mixed,
                                   cudaStream_t stream);

// One batch of fixed-length windows (sea_b200_corpus_decode_windows_async): work unit (window, covering-chunk slot j < M).
struct CorpusLaunch {
    const uint8_t *sea;
    uint64_t sea_len;  // readable bytes from sea (the staged loads of the fast route stop there)
    const CorpusStream *streams;
    uint32_t n_streams, channels;
    const uint32_t *win_stream;
    const uint64_t *win_first;
    uint32_t n_windows, W, M;
    bool planar;
    void *out;
    uint32_t *frames_out;  // nullable
    int32_t *status;
    // fast route: the corpus's uniform geometry and header fields
    uint32_t N, chunk_size, s, b;
};
// Fast route: CBR, 1 or 2 channels, scale_factor_frames 20, scale_factor_bits <= 5 (its dequant rows live in shared memory), one
// chunk geometry for every stream.  corpus_fast_prepare (once, at create: not capturable) raises the shared-memory limit of its
// kernels; launch_corpus_windows then only enqueues.
bool corpus_fast_supported(uint32_t channels, uint32_t s, uint32_t b, uint32_t F, bool vbr);
cudaError_t corpus_fast_prepare(uint32_t channels, uint32_t s, uint32_t b);
cudaError_t launch_corpus_windows(const CorpusLaunch &p, bool fast, DevTables tabs, cudaStream_t stream);

// ---- encode ------------------------------------------------------------------------------------------------
struct EncStream {
    uint64_t pcm_off;   // sample offset of the stream's PCM
    uint64_t out_off;   // byte offset of the stream's .sea (or of the raw chunk in chunk mode)
    uint32_t n_frames;
    uint32_t last_counts[3];  // VBR bucket counts [base-1, base+1, base+2] of the partial last chunk
};

struct EncParams {
    uint32_t channels, N, F, s;
    uint32_t hdr_bits;         // chunk header residual size
    uint32_t vbr;              // 0/1
    uint32_t base;             // VBR base size
    uint32_t full_counts[3];   // VBR bucket counts [base-1, base+1, base+2] of a full chunk
    uint32_t full_chunk_bytes;
    uint32_t max_chunk_bytes;
    uint32_t sample_rate;
    uint32_t raw_chunk_mode;   // 1: write only the chunk at out_off, no file header (make_chunk seam)
    uint32_t n_streams;
    uint32_t vbr_smem_off;     // != 0: the VBR scratch (ranks, sort keys, sizes) lives in shared memory at this offset
    uint32_t lut_mode;         // VBR fast pass: where the dequant rows live (encode_kernels.cu kEncLut*); set by the launcher
    uint32_t split;            // fast pass: 1 = one warp per channel (few streams), 0 = one warp per channel pair; set by the launcher
};

// Persistent per-channel encoder state (EncoderBase.lms + prev_scalefactor, encoder_base.rs:15-19): 9 int32 per channel
constexpr int kEncStateWords = 9;

struct EncWorkspace {
    // per-stream VBR scratch (device), sized by enc_vbr_scratch_bytes()
    uint8_t *vbr_scratch;
    uint64_t vbr_scratch_stride;
};
uint64_t enc_vbr_scratch_bytes(const EncParams &p);

// d_state: nullable; when set, n_streams * channels * 9 int32 loaded at start and stored at the end.
// d_out_lens: per stream total bytes written; d_chunk0: per stream size of its first chunk; d_ties: VBR boundary ties.
cudaError_t launch_encode_generic(const int16_t *d_pcm, uint8_t *d_out, const EncStream *d_streams, const EncParams &p,
                                  DevTables tabs, int32_t *d_state, uint64_t *d_out_lens, uint32_t *d_chunk0,
                                  unsigned long long *d_ties, EncWorkspace ws, int *d_err, cudaStream_t stream);

// ---- measurement -------------------------------------------------------------------------------------------
cudaError_t launch_int32_peak(int mode, uint32_t *d_sink, uint64_t *lane_ops, cudaStream_t stream);
// synthetic tone + noise PCM of sea_codec_b200/synth.py, generated in place on the device (bench inputs)
cudaError_t launch_synth(int16_t *d_pcm, uint64_t stream_stride, uint32_t n_streams, uint32_t n_frames, uint32_t channels, const uint32_t *d_ids,
                         const uint32_t *d_steps, const int32_t *d_sine, uint64_t seed, int32_t amp, int32_t noise_amp, cudaStream_t stream);

}  // namespace sea
