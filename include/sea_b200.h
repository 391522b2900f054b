/*
 * sea_b200.h -- C-ABI of the B200-native SEA encode/decode hot path (libsea_b200.so).
 *
 * This is the drop-in boundary for chanderlud/sea-codec: the entry points below are what the crate's
 * FFI for the hot path would bind.  Each one cites the reference interface (file:line under
 * /root/reference) it replaces.  Plain pointers and sizes only; no torch / C++ types.
 *
 * Conventions (precedent: src/wasm_api.rs:32-95 and c/sea.h:189-226):
 *   - the CALLER owns every input and output buffer and passes pointer + capacity; the callee reports
 *     how much it wrote;
 *   - every function returns an int status: 0 (or a small positive "more/eof" value where documented)
 *     on success, a negative SEA_B200_ERR_* otherwise.  Nothing aborts or throws across the boundary;
 *   - there is NO CPU fallback: without a usable CUDA device sea_b200_ctx_create fails with
 *     SEA_B200_ERR_CUDA and no codec call can be made;
 *   - a context is bound to one GPU and one CUDA stream and must be used from one host thread at a
 *     time (the reference types are !Send: src/codec/file.rs:29); contexts are independent.
 */
#ifndef SEA_B200_H
#define SEA_B200_H

#include <stdbool.h>
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SEA_B200_ABI_VERSION 1

/* Status codes.  -1..-9 mirror `enum SeaError` (src/codec/common.rs:53-64) in declaration order. */
enum {
    SEA_B200_OK = 0,
    SEA_B200_ERR_READ = -1,               /* SeaError::ReadError                                        */
    SEA_B200_ERR_INVALID_PARAMETERS = -2, /* SeaError::InvalidParameters                                */
    SEA_B200_ERR_INVALID_FILE = -3,       /* SeaError::InvalidFile       (file.rs:41-44, :68-70)        */
    SEA_B200_ERR_INVALID_FRAME = -4,      /* SeaError::InvalidFrame      (chunk.rs:76-85)               */
    SEA_B200_ERR_ENCODER_CLOSED = -5,     /* SeaError::EncoderClosed     (encoder.rs:107-109)           */
    SEA_B200_ERR_UNSUPPORTED_VERSION = -6,/* SeaError::UnsupportedVersion                               */
    SEA_B200_ERR_TOO_MANY_FRAMES = -7,    /* SeaError::TooManyFrames                                    */
    SEA_B200_ERR_METADATA_TOO_LARGE = -8, /* SeaError::MetadataTooLarge                                 */
    SEA_B200_ERR_IO = -9,                 /* SeaError::IoError (e.g. UnexpectedEof, encoder.rs:95-99)   */
    SEA_B200_ERR_CAPACITY = -20,          /* caller buffer too small (wasm_api.rs:58,81 assert)         */
    SEA_B200_ERR_DOMAIN = -21,            /* input on which the reference panics (assert/unwrap/index), */
                                          /* e.g. VBR >= ~7.375 bits (common.rs:34), chunk > 65535 B    */
    SEA_B200_ERR_CUDA = -30,              /* CUDA runtime / driver failure, no device                   */
    SEA_B200_ERR_NOMEM = -31
};

/* EncoderSettings (src/encoder.rs:16-35); defaults {4, 20, 3.0, 5120, false}. */
typedef struct sea_b200_settings {
    uint8_t scale_factor_bits;   /* 1..8 accepted (seaconv validates 3..5, seaconv.rs:35-41)             */
    uint8_t scale_factor_frames; /* must divide frames_per_chunk (chunk.rs:218)                          */
    uint16_t frames_per_chunk;
    float residual_bits;         /* CBR: floor() in 1..8; VBR: 1.375 <= bits < ~7.375 at defaults        */
    uint8_t vbr;
    uint8_t reserved[3];
} sea_b200_settings;

/* SeaFileHeader (src/codec/file.rs:21-30).  metadata bytes are never consumed by the reference
 * decoder (file.rs:53-54); this library behaves identically: chunk data starts at byte 22. */
typedef struct sea_b200_header {
    uint8_t version;
    uint8_t channels;
    uint16_t chunk_size;
    uint16_t frames_per_chunk;
    uint16_t reserved;
    uint32_t sample_rate;
    uint32_t total_frames;
    uint32_t metadata_size;
} sea_b200_header;

#define SEA_B200_FILE_HEADER_BYTES 22

typedef struct sea_b200_ctx sea_b200_ctx;
typedef struct sea_b200_encoder sea_b200_encoder;
typedef struct sea_b200_decoder sea_b200_decoder;

/* ---------------------------------------------------------------- context */

/* Binds GPU `device`, creates the context's CUDA stream and uploads the quantiser tables
 * (SeaDequantTab::init, dqt.rs:17-38; SeaQuantTab is a closed form on the device). */
int sea_b200_ctx_create(int device, sea_b200_ctx **ctx);
void sea_b200_ctx_destroy(sea_b200_ctx *ctx);
/* Use an existing cudaStream_t (e.g. torch's current stream) for all work of this context. */
int sea_b200_ctx_set_stream(sea_b200_ctx *ctx, void *cuda_stream);
void *sea_b200_ctx_stream(const sea_b200_ctx *ctx);
const char *sea_b200_strerror(int status);
const char *sea_b200_last_error(const sea_b200_ctx *ctx); /* detail of the last failure on ctx */
int sea_b200_abi_version(void);
/* How many kernels of this library the context has launched so far (bench.py "gpu_launches"). */
uint64_t sea_b200_ctx_launch_count(const sea_b200_ctx *ctx);

/* Pinned host memory for the host-buffer entry points (allocate/deallocate, wasm_api.rs:97-111). */
void *sea_b200_host_alloc(size_t bytes);
void sea_b200_host_free(void *p);

/* ---------------------------------------------------------------- format helpers (host only) */

void sea_b200_default_settings(sea_b200_settings *s); /* EncoderSettings::default, encoder.rs:25-35 */
/* SeaFileHeader::from_reader (file.rs:40-72). */
int sea_b200_parse_header(const uint8_t *sea, uint64_t len, sea_b200_header *out);
/* Upper bound of the .sea size for n_frames frames (exact for CBR). */
int sea_b200_encode_bound(uint64_t n_frames, uint32_t channels, const sea_b200_settings *s, uint64_t *bytes);
/* Bytes of a FULL chunk (header.chunk_size; SURVEY App. D formula).  VBR: constant because the bucket
 * counts are constant (encoder_vbr.rs:66-96). */
int sea_b200_full_chunk_bytes(uint32_t channels, const sea_b200_settings *s, uint32_t *bytes);
/* VbrEncoder::get_normalized_vbr_bitrate + interpolate_distribution (encoder_vbr.rs:40-96). */
int sea_b200_vbr_plan(const sea_b200_settings *s, uint64_t sortable_items, float *target, uint32_t *base, uint64_t counts[4]);
/* Quantiser tables as generated on the host for the device (dqt.rs:40-126): recip[2^sfb], dqt[2^sfb * 2^rb]. */
int sea_b200_tables(uint32_t residual_bits, uint32_t scale_factor_bits, int32_t *recip, int32_t *dqt);

/* ---------------------------------------------------------------- one-shot, host buffers */

/* sea_encode (src/lib.rs:13-36): interleaved i16 PCM -> complete .sea byte stream. */
int sea_b200_encode(sea_b200_ctx *ctx, const int16_t *pcm, uint64_t n_samples, uint32_t sample_rate, uint32_t channels,
                    const sea_b200_settings *settings, uint8_t *out, uint64_t out_cap, uint64_t *out_len);
/* sea_decode (src/lib.rs:44-63) / c/sea.h:189 sea_decode: pcm == NULL returns only the header info and the
 * sample count needed (two-call pattern of c/sea.h:209-211). */
int sea_b200_decode(sea_b200_ctx *ctx, const uint8_t *sea, uint64_t len, int16_t *pcm, uint64_t pcm_cap_samples,
                    uint64_t *n_samples, uint32_t *sample_rate, uint32_t *channels);

/* ---------------------------------------------------------------- batch (additive API; independent streams) */

/* n_streams independent sea_encode calls with shared (sample_rate, channels, settings).
 * pcm_offsets[i] / n_frames[i]: sample offset and frame count of stream i inside `pcm`;
 * out_offsets[i]: byte offset of stream i's .sea inside `out` (capacity >= sea_b200_encode_bound);
 * out_lens[i] receives its length.  Host buffers (pinned recommended). */
int sea_b200_encode_batch(sea_b200_ctx *ctx, uint32_t n_streams, const int16_t *pcm, const uint64_t *pcm_offsets,
                          const uint32_t *n_frames, uint32_t sample_rate, uint32_t channels,
                          const sea_b200_settings *settings, uint8_t *out, const uint64_t *out_offsets, uint64_t *out_lens);
/* n_streams independent sea_decode calls.  pcm_offsets[i]: sample offset of stream i's PCM inside `pcm`;
 * pcm_caps[i] its capacity in samples (NULL = trust the headers); n_samples[i] receives the count. */
int sea_b200_decode_batch(sea_b200_ctx *ctx, uint32_t n_streams, const uint8_t *sea, const uint64_t *sea_offsets,
                          const uint64_t *sea_lens, int16_t *pcm, const uint64_t *pcm_offsets, const uint64_t *pcm_caps,
                          uint64_t *n_samples);

/* Same, with `pcm`/`out`/`sea` resident in device memory of the context's GPU (offset/length arrays stay on
 * the host).  decode needs the 22-byte file headers on the host: `headers` = n_streams * 22 bytes. */
int sea_b200_encode_batch_device(sea_b200_ctx *ctx, uint32_t n_streams, const int16_t *d_pcm, const uint64_t *pcm_offsets,
                                 const uint32_t *n_frames, uint32_t sample_rate, uint32_t channels,
                                 const sea_b200_settings *settings, uint8_t *d_out, const uint64_t *out_offsets,
                                 uint64_t *out_lens);
int sea_b200_decode_batch_device(sea_b200_ctx *ctx, uint32_t n_streams, const uint8_t *d_sea, const uint64_t *sea_offsets,
                                 const uint64_t *sea_lens, const uint8_t *headers, int16_t *d_pcm,
                                 const uint64_t *pcm_offsets, const uint64_t *pcm_caps, uint64_t *n_samples);

/* ---------------------------------------------------------------- batch across the GPUs of one box (in-process) */

/* BASELINE north star / SURVEY 8e: streams are partitioned across the GPUs, nothing is exchanged between them, only per-GPU
 * counts are gathered on the host.  A sea_b200_multi owns one context per listed device; a call shards the batch into one
 * contiguous range of streams per GPU (balanced by PCM samples resp. .sea bytes), runs the single-GPU host-buffer call above
 * on every range from one host thread per GPU, and reports where each GPU's range starts and how much it produced.
 * devices == NULL means devices 0 .. n_devices-1.  The arrays first_stream_of_device / *_per_device have n_devices entries
 * and may be NULL.  Results are identical to the single-GPU call on the same arguments. */
typedef struct sea_b200_multi sea_b200_multi;
int sea_b200_multi_create(const int *devices, uint32_t n_devices, sea_b200_multi **multi);
void sea_b200_multi_destroy(sea_b200_multi *multi);
uint32_t sea_b200_multi_device_count(const sea_b200_multi *multi);
sea_b200_ctx *sea_b200_multi_ctx(const sea_b200_multi *multi, uint32_t index); /* the index-th GPU's context (owned by multi) */
const char *sea_b200_multi_last_error(const sea_b200_multi *multi);
int sea_b200_multi_encode_batch(sea_b200_multi *multi, uint32_t n_streams, const int16_t *pcm, const uint64_t *pcm_offsets,
                                const uint32_t *n_frames, uint32_t sample_rate, uint32_t channels,
                                const sea_b200_settings *settings, uint8_t *out, const uint64_t *out_offsets, uint64_t *out_lens,
                                uint32_t *first_stream_of_device, uint64_t *bytes_per_device);
int sea_b200_multi_decode_batch(sea_b200_multi *multi, uint32_t n_streams, const uint8_t *sea, const uint64_t *sea_offsets,
                                const uint64_t *sea_lens, int16_t *pcm, const uint64_t *pcm_offsets, const uint64_t *pcm_caps,
                                uint64_t *n_samples, uint32_t *first_stream_of_device, uint64_t *samples_per_device);

/* ---------------------------------------------------------------- streaming seam (one chunk per call) */

/* SeaFile::new + EncoderBase::new (file.rs:111-129, encoder_base.rs:29-41): per-channel LMS state and
 * prev_scalefactor live on the device for the life of the handle. */
int sea_b200_encoder_create(sea_b200_ctx *ctx, uint32_t channels, uint32_t sample_rate, const sea_b200_settings *settings,
                            sea_b200_encoder **enc);
/* SeaFile::make_chunk (file.rs:142-178): n_samples interleaved i16 (<= frames_per_chunk*channels, multiple of
 * channels) -> one serialized chunk.  The first call fixes header.chunk_size. */
int sea_b200_encoder_make_chunk(sea_b200_encoder *enc, const int16_t *pcm, uint64_t n_samples, uint8_t *out, uint64_t out_cap,
                                uint64_t *out_len);
/* header.chunk_size as fixed by the first chunk (0 before). */
uint32_t sea_b200_encoder_chunk_size(const sea_b200_encoder *enc);
void sea_b200_encoder_destroy(sea_b200_encoder *enc);

/* SeaFile::from_reader (file.rs:131-140): parses the 22-byte header. */
int sea_b200_decoder_create(sea_b200_ctx *ctx, const uint8_t *header22, uint64_t len, sea_b200_decoder **dec);
int sea_b200_decoder_header(const sea_b200_decoder *dec, sea_b200_header *out);
/* SeaFile::samples_from_reader minus the read (file.rs:180-209): `chunk` = the <= chunk_size bytes the reader
 * returned; remaining_frames < 0 means None (streaming, chunk.rs:76-79). */
int sea_b200_decoder_decode_chunk(sea_b200_decoder *dec, const uint8_t *chunk, uint64_t len, int64_t remaining_frames,
                                  int16_t *pcm, uint64_t pcm_cap_samples, uint64_t *n_samples);
void sea_b200_decoder_destroy(sea_b200_decoder *dec);

/* Multi-chunk forms of the two seam calls: the same state machine, several chunks per call (one launch, one H2D, one D2H).
 * make_chunks: n_samples may span any number of chunks; the serialized chunks follow each other in `out` (all but the last
 * are full chunks of sea_b200_encoder_chunk_size() bytes); *n_chunks receives their count.  The LMS state and
 * prev_scalefactor stay on the device between calls (encoder_base.rs:181-182). */
int sea_b200_encoder_make_chunks(sea_b200_encoder *enc, const int16_t *pcm, uint64_t n_samples, uint8_t *out, uint64_t out_cap,
                                 uint64_t *out_len, uint32_t *n_chunks);
/* decode_chunks: `chunks` = consecutive chunks as they lie in the file (every one chunk_size bytes, the last may be the
 * stream's short final chunk when remaining_frames >= 0); decoded chunk-parallel. */
int sea_b200_decoder_decode_chunks(sea_b200_decoder *dec, sea_b200_ctx *ctx, const uint8_t *chunks, uint64_t len,
                                   int64_t remaining_frames, int16_t *pcm, uint64_t pcm_cap_samples, uint64_t *n_samples);

/* ---------------------------------------------------------------- session pool (many live streams, one launch per push) */

/* A slot table of up to max_sessions streaming encoders with one channel count, sample rate and settings (settings are checked
 * as sea_b200_encoder_create checks them).  Each open session is the encoder of one live stream: its LMS state and
 * prev_scalefactor (encoder_base.rs:181-182) and the fewer than frames_per_chunk frames it has buffered stay on the device
 * between calls.  A push takes a packet of any length from each of its sessions and encodes every chunk that has completed,
 * across all of them, in one launch.  A pool uses ctx's current stream, is used from one host thread, and must be destroyed
 * before ctx. */
typedef struct sea_b200_encoder_pool sea_b200_encoder_pool;
int sea_b200_encoder_pool_create(sea_b200_ctx *ctx, uint32_t max_sessions, uint32_t channels, uint32_t sample_rate,
                                 const sea_b200_settings *settings, sea_b200_encoder_pool **pool);
void sea_b200_encoder_pool_destroy(sea_b200_encoder_pool *pool); /* waits for the context's stream */
/* Opens slots sessions[0..n) (each < max_sessions, not open, listed once): each starts from EncoderBase::new state with nothing
 * buffered.  Host-side only. */
int sea_b200_encoder_pool_open(sea_b200_encoder_pool *pool, uint32_t n, const uint32_t *sessions);
/* Frames buffered per session (< frames_per_chunk; 0 for a closed slot). */
int sea_b200_encoder_pool_buffered(const sea_b200_encoder_pool *pool, uint32_t n, const uint32_t *sessions, uint32_t *frames);
/* Bytes a push of n_frames to an open session produces: k * full chunk bytes for the k chunks it completes, and with `end` the
 * bound of its short final chunk on top (exact for CBR). */
int sea_b200_encoder_pool_push_bound(const sea_b200_encoder_pool *pool, uint32_t session, uint64_t n_frames, bool end, uint64_t *bytes);
/* Appends n_frames[i] interleaved frames at pcm + pcm_offsets[i] (samples) to session sessions[i] and writes every chunk now
 * complete, back to back, at out + out_offsets[i] (bytes): out_lens[i] = their byte count, n_chunks[i] (nullable) = their
 * number.  end[i] != 0 (end nullable = none) also encodes what is left as the session's short final chunk and closes the slot.
 * Joining a session's outputs gives exactly the chunks sea_b200_encode writes after its 22-byte header for the session's whole
 * PCM, whatever the packet boundaries and whichever sessions share a call; the header is the caller's, with chunk_size = the
 * session's first chunk's size (file.rs:166-168).  Refused before anything is enqueued, with every session left as it was: a
 * session not open, >= max_sessions or listed twice, a NULL pointer, buffered plus pushed frames past 2^32
 * (SEA_B200_ERR_TOO_MANY_FRAMES), an out_caps[i] (nullable = trust the caller) below push_bound (SEA_B200_ERR_CAPACITY).  A
 * device error closes the call's sessions.  sea_b200_last_vbr_ties_per_stream then holds the call's sessions in call order.
 * Host buffers (pinned recommended); one launch each for ingest, encode (skipped when no chunk completes) and commit. */
int sea_b200_encoder_pool_push(sea_b200_encoder_pool *pool, uint32_t n, const uint32_t *sessions, const int16_t *pcm,
                               const uint64_t *pcm_offsets, const uint32_t *n_frames, const uint8_t *end, uint8_t *out,
                               const uint64_t *out_offsets, const uint64_t *out_caps, uint64_t *out_lens, uint32_t *n_chunks);
/* The same with d_pcm and d_out in device memory of ctx's GPU (offsets and lengths stay on the host); bytes of d_out outside
 * [out_offsets[i], out_offsets[i] + out_lens[i]) are never written. */
int sea_b200_encoder_pool_push_device(sea_b200_encoder_pool *pool, uint32_t n, const uint32_t *sessions, const int16_t *d_pcm,
                                      const uint64_t *pcm_offsets, const uint32_t *n_frames, const uint8_t *end, uint8_t *d_out,
                                      const uint64_t *out_offsets, const uint64_t *out_caps, uint64_t *out_lens, uint32_t *n_chunks);

/* ---------------------------------------------------------------- random access (README.md:125 "seeking" future work) */

/* Decodes frames [first_frame, first_frame + n_frames) of a complete .sea file: only the chunks that cover the range are
 * shipped and decoded (chunk k starts at byte 22 + k*chunk_size, file.rs:185, and carries its own LMS state,
 * chunk.rs:95-103).  The range is clamped to the file; pcm == NULL returns the sample count only.
 * flags: SEA_B200_RANGE_SKIP_METADATA makes chunk data start after the header's metadata bytes -- the format-compatible fix
 * of the reference decoder's metadata bug (file.rs:53-54 reads zero bytes); default 0 mirrors the reference. */
#define SEA_B200_RANGE_SKIP_METADATA 1u
int sea_b200_decode_range(sea_b200_ctx *ctx, const uint8_t *sea, uint64_t len, uint64_t first_frame, uint64_t n_frames,
                          uint32_t flags, int16_t *pcm, uint64_t pcm_cap_samples, uint64_t *n_samples, uint32_t *sample_rate,
                          uint32_t *channels);

/* Output format bit of `flags` (combinable with SEA_B200_RANGE_SKIP_METADATA, which means what it means for decode_range). */
#define SEA_B200_WINDOW_F32_PLANAR 2u
/* n_windows frame windows of device-resident streams in one call (e.g. fixed-length training crops of a corpus kept in HBM).
 * Streams are described as for sea_b200_decode_batch_device (d_sea + host offsets / lengths, n_streams * 22 header bytes on
 * the host).  Window w = frames [first_frames[w], first_frames[w] + n_frames[w]) of stream window_stream[w]; several windows
 * may name the same stream.  Output slot w starts at element out_offsets[w] of d_out (device memory):
 *   default:                    int16, interleaved  [n_frames[w]][channels]   (the library's PCM layout)
 *   SEA_B200_WINDOW_F32_PLANAR: float32, planar     [channels][n_frames[w]], value = sample / 32768.0f
 * The first frames_out[w] frames of a slot are what sea_b200_decode_range(stream, first, n, flags & SKIP_METADATA) returns;
 * frames the stream does not have (past its end, clamped as decode_range clamps them) are written as zeros.  Bytes of d_out
 * outside the slots are never written.  Only the chunks that cover a window are decoded.  A window_stream index >= n_streams
 * or an unknown flag bit is SEA_B200_ERR_INVALID_PARAMETERS; a bad chunk inside a window gives decode_range's code for it. */
int sea_b200_decode_windows_device(sea_b200_ctx *ctx, uint32_t n_streams, const uint8_t *d_sea, const uint64_t *sea_offsets,
                                   const uint64_t *sea_lens, const uint8_t *headers, uint32_t n_windows,
                                   const uint32_t *window_stream, const uint64_t *first_frames, const uint32_t *n_frames,
                                   uint32_t flags, void *d_out, const uint64_t *out_offsets, uint64_t *frames_out);

/* A registered corpus: .sea streams resident in device memory, checked once, then decoded in fixed-length windows from indices
 * that live on the device, stream-ordered and without host synchronisation (a training loader's crops, inside a CUDA graph). */
typedef struct sea_b200_corpus sea_b200_corpus;
/* Registers n_streams .sea streams resident in device memory of ctx's GPU, described as for sea_b200_decode_windows_device
 * (d_sea + host sea_offsets / sea_lens, n_streams * 22 header bytes on the host).  flags: 0 or SEA_B200_RANGE_SKIP_METADATA
 * (fixed for the corpus).  All streams must have the same channel count.  Every chunk any window could cover is validated
 * here, once: a stream the reference could not decode is rejected with the code decode_range would return for it, and
 * last_error names the stream and the chunk.  d_sea must stay valid and unchanged for the life of the corpus, and the corpus
 * must be destroyed before ctx.  Synchronous; not capturable. */
int sea_b200_corpus_create(sea_b200_ctx *ctx, uint32_t n_streams, const uint8_t *d_sea, const uint64_t *sea_offsets,
                           const uint64_t *sea_lens, const uint8_t *headers, uint32_t flags, sea_b200_corpus **corpus);
void sea_b200_corpus_destroy(sea_b200_corpus *corpus); /* waits for work of the corpus still in flight */
/* channels, and per stream the frames a window can draw from (stream_frames: n_streams entries, or NULL); route: 0 generic,
 * 1 fast (informational; SEA_B200_CORPUS_ROUTE=generic|fast pins it at create, for tests). */
int sea_b200_corpus_info(const sea_b200_corpus *corpus, uint32_t *channels, uint64_t *stream_frames, uint32_t *route);
/* n_windows windows of window_frames frames each.  Window w = frames [d_first_frames[w], + window_frames) of stream
 * d_window_stream[w]; both arrays are in DEVICE memory.  Slot w is dense in d_out:
 *   default:                    int16   [n_windows][window_frames][channels]
 *   SEA_B200_WINDOW_F32_PLANAR: float32 [n_windows][channels][window_frames]
 * Slot w equals decode_windows_device's slot for (stream, first, window_frames) with the corpus's metadata flag: what
 * decode_range returns, then zeros (a first frame at or past the stream's end, including any huge value, gives an all-zero
 * slot).  d_frames_out[w] (device, nullable) equals its frames_out.  A stream index >= n_streams zero-fills the slot, writes
 * frames_out 0 and stores SEA_B200_ERR_INVALID_PARAMETERS into *d_status when *d_status is 0 (first error wins; the call never
 * clears it).  Bytes of d_out outside the slots are never written.
 * Stream-ordered on the context's current stream: no host synchronisation, no allocation, no host<->device copy, so the call
 * can be captured in a CUDA graph and replayed with new indices written in place.  For the same reason it does not update
 * sea_b200_last_kernel_ms.  Host-checkable errors (NULL pointers, unknown flag bits, misaligned d_out) return before anything
 * is enqueued; n_windows == 0 or window_frames == 0 enqueues nothing. */
int sea_b200_corpus_decode_windows_async(sea_b200_corpus *corpus, uint32_t n_windows, const uint32_t *d_window_stream,
                                         const uint64_t *d_first_frames, uint32_t window_frames, uint32_t flags, void *d_out,
                                         uint32_t *d_frames_out, int32_t *d_status);

/* ---------------------------------------------------------------- the reference's existing foreign surfaces */

/* src/wasm_api.rs:32-111 (wasm_sea_encode / wasm_sea_decode / allocate / deallocate / setup) with the same argument lists,
 * served by a process-wide context on GPU $SEA_B200_DEVICE (default 0).  Where the reference asserts/panics these return 0
 * and sea_b200_wasm_status() holds the SEA_B200_ERR_* code.  input_length / output_length are BYTES (wasm_api.rs:45,83). */
void sea_b200_wasm_setup(void);
size_t sea_b200_wasm_sea_encode(const int16_t *input_samples, size_t input_length, uint32_t sample_rate, uint32_t channels,
                                float bitrate, bool vbr, uint8_t *output_buffer, size_t output_length);
size_t sea_b200_wasm_sea_decode(const uint8_t *encoded, size_t encoded_length, int16_t *output_buffer, size_t output_length,
                                uint32_t *sample_rate, uint32_t *channels);
uint8_t *sea_b200_wasm_allocate(size_t size);             /* pinned host memory */
void sea_b200_wasm_deallocate(uint8_t *ptr, size_t size);
int sea_b200_wasm_status(void);
/* c/sea.h:189 `int sea_decode(encoded, encoded_len, &sample_rate, &channels, output, &total_frames)`: same arguments, same
 * return codes (0 ok, 1 invalid file, 2 decode error), same two-call pattern (output == NULL fills the header fields only). */
int sea_b200_csea_decode(uint8_t *encoded, uint32_t encoded_len, uint32_t *sample_rate, uint32_t *channels, int16_t *output,
                         uint32_t *total_frames);

/* ---------------------------------------------------------------- measurement helpers */

/* INT32 issue-rate micro-kernel (SURVEY 8d: encoder roofline denominator).  mode 0: IMAD chains (fma pipe),
 * 1: IADD3/LOP3 chains (alu pipe), 2: interleaved.  Returns lane-ops/s in *ops_per_s, kernel ms in *ms. */
int sea_b200_int32_peak(sea_b200_ctx *ctx, int mode, double *ops_per_s, double *ms);
/* Synthetic tone + noise PCM generated in place on the device (bench.py inputs; SURVEY 8d "Synthetic input"): stream i of the
 * batch gets the samples sea_codec_b200/synth.py:gen_stream(stream_ids[i], ...) computes on the host, bit for bit -- interleaved
 * i16 at d_pcm + i*stream_stride_samples.  phase_steps[i] = round(f/rate * 2^32) of the stream's tone and the 4096-entry sine
 * table are computed by the caller in float64 (the device does integer arithmetic only). */
int sea_b200_synth_pcm_device(sea_b200_ctx *ctx, int16_t *d_pcm, uint64_t stream_stride_samples, uint32_t n_streams, uint32_t n_frames,
                              uint32_t channels, const uint32_t *stream_ids, const uint32_t *phase_steps,
                              const int32_t *sine_table_4096, uint64_t seed, int32_t amplitude, int32_t noise_amplitude);
/* Duration (ms, CUDA events on the context's stream) of the kernels launched by the last batch call. */
double sea_b200_last_kernel_ms(const sea_b200_ctx *ctx);
/* VBR blocks whose error tied across a bucket boundary in the last encode (sort_unstable order is unspecified in the
 * reference, encoder_vbr.rs:102-103; this library orders by (error, index)).  0 means bit-exactness is well defined. */
uint64_t sea_b200_last_vbr_ties(const sea_b200_ctx *ctx);
/* The same count per stream of the last batch encode: ties[i] for i < n_streams (bench.py selects tie-free inputs with it). */
int sea_b200_last_vbr_ties_per_stream(const sea_b200_ctx *ctx, uint64_t *ties, uint32_t n_streams);

#ifdef __cplusplus
}
#endif
#endif /* SEA_B200_H */
