// sea_b200.hpp -- C++ host-side mirror of the sea-codec crate API on top of the C-ABI (sea_b200.h).
//
// The reference's host layer is Rust (src/lib.rs, src/encoder.rs, src/decoder.rs); no Rust toolchain exists in the build
// image, so this header is the compiled-language host side: same names, argument meaning and error behaviour.
//   sea::EncoderSettings                          src/encoder.rs:16-35
//   sea::SeaEncoder<R, W>::encode_frame/finalize  src/encoder.rs:50-159   (R: size_t read(void*, size_t); W: void write(const void*, size_t))
//   sea::SeaDecoder<R, W>::decode_frame           src/decoder.rs:22-72
//   sea::sea_encode / sea::sea_decode             src/lib.rs:13-63
//   additions: SeaEncoder::encode_frames(k), SeaDecoder::decode_frames(k) (k chunks per launch), sea::sea_decode_range
// Errors: sea::SeaError carries the SeaError variant (common.rs:53-64) as the C-ABI status code.
#pragma once
#include <cstdint>
#include <cstring>
#include <optional>
#include <stdexcept>
#include <string>
#include <vector>

#include "sea_b200.h"

namespace sea {

struct SeaError : std::runtime_error {
    int code;
    SeaError(int c, const std::string &what) : std::runtime_error(std::string(sea_b200_strerror(c)) + ": " + what), code(c) {}
};

struct EncoderSettings {  // encoder.rs:16-35
    uint8_t scale_factor_bits = 4;
    uint8_t scale_factor_frames = 20;
    float residual_bits = 3.0f;
    uint16_t frames_per_chunk = 5120;
    bool vbr = false;
    sea_b200_settings c() const
    {
        sea_b200_settings s;
        std::memset(&s, 0, sizeof(s));
        s.scale_factor_bits = scale_factor_bits;
        s.scale_factor_frames = scale_factor_frames;
        s.frames_per_chunk = frames_per_chunk;
        s.residual_bits = residual_bits;
        s.vbr = vbr ? 1 : 0;
        return s;
    }
};

struct SeaFileHeader {  // file.rs:21-30
    uint8_t version, channels;
    uint16_t chunk_size, frames_per_chunk;
    uint32_t sample_rate, total_frames;
};

class Context {
public:
    explicit Context(int device = 0)
    {
        int rc = sea_b200_ctx_create(device, &ctx_);
        if (rc) throw SeaError(rc, "no usable CUDA device (libsea_b200 has no CPU fallback)");
    }
    ~Context() { sea_b200_ctx_destroy(ctx_); }
    Context(const Context &) = delete;
    Context &operator=(const Context &) = delete;
    sea_b200_ctx *get() const { return ctx_; }
    void check(int rc) const
    {
        if (rc < 0) throw SeaError(rc, sea_b200_last_error(ctx_));
    }

private:
    sea_b200_ctx *ctx_ = nullptr;
};

// A registered corpus (sea_b200_corpus_*): device-resident streams checked once, then decoded in fixed-length windows from device-side
// indices on the context's stream, without host synchronisation (CUDA-graph capturable).  Destroy it before its Context.
class Corpus {
public:
    Corpus(Context &ctx, uint32_t n_streams, const uint8_t *d_sea, const uint64_t *sea_offsets, const uint64_t *sea_lens,
           const uint8_t *headers, bool skip_metadata = false)
        : ctx_(&ctx)
    {
        ctx.check(sea_b200_corpus_create(ctx.get(), n_streams, d_sea, sea_offsets, sea_lens, headers,
                                         skip_metadata ? SEA_B200_RANGE_SKIP_METADATA : 0u, &corpus_));
        uint32_t route = 0;
        stream_frames_.resize(n_streams);
        ctx.check(sea_b200_corpus_info(corpus_, &channels_, stream_frames_.data(), &route));
        fast_ = route == 1;
    }
    ~Corpus() { sea_b200_corpus_destroy(corpus_); }
    Corpus(const Corpus &) = delete;
    Corpus &operator=(const Corpus &) = delete;
    sea_b200_corpus *get() const { return corpus_; }
    uint32_t channels() const { return channels_; }
    bool fast_route() const { return fast_; }
    const std::vector<uint64_t> &stream_frames() const { return stream_frames_; }
    // see sea_b200_corpus_decode_windows_async; flags: 0 or SEA_B200_WINDOW_F32_PLANAR
    void decode_windows_async(uint32_t n_windows, const uint32_t *d_window_stream, const uint64_t *d_first_frames, uint32_t window_frames,
                              uint32_t flags, void *d_out, uint32_t *d_frames_out, int32_t *d_status) const
    {
        ctx_->check(sea_b200_corpus_decode_windows_async(corpus_, n_windows, d_window_stream, d_first_frames, window_frames, flags, d_out,
                                                         d_frames_out, d_status));
    }

private:
    Context *ctx_;
    sea_b200_corpus *corpus_ = nullptr;
    uint32_t channels_ = 0;
    bool fast_ = false;
    std::vector<uint64_t> stream_frames_;
};

// A pool of streaming encoder sessions (sea_b200_encoder_pool_*): one push per round of packets encodes every chunk that completed
// across all sessions in one launch.  Destroy it before its Context.
class EncoderPool {
public:
    EncoderPool(Context &ctx, uint32_t channels, uint32_t sample_rate, const EncoderSettings &settings, uint32_t max_sessions)
        : ctx_(&ctx)
    {
        sea_b200_settings s = settings.c();
        ctx.check(sea_b200_encoder_pool_create(ctx.get(), max_sessions, channels, sample_rate, &s, &pool_));
    }
    ~EncoderPool() { sea_b200_encoder_pool_destroy(pool_); }
    EncoderPool(const EncoderPool &) = delete;
    EncoderPool &operator=(const EncoderPool &) = delete;
    sea_b200_encoder_pool *get() const { return pool_; }
    void open(uint32_t n, const uint32_t *sessions) { ctx_->check(sea_b200_encoder_pool_open(pool_, n, sessions)); }
    void buffered(uint32_t n, const uint32_t *sessions, uint32_t *frames) const
    {
        ctx_->check(sea_b200_encoder_pool_buffered(pool_, n, sessions, frames));
    }
    uint64_t push_bound(uint32_t session, uint64_t n_frames, bool end) const
    {
        uint64_t b = 0;
        ctx_->check(sea_b200_encoder_pool_push_bound(pool_, session, n_frames, end, &b));
        return b;
    }
    // host buffers; arguments as sea_b200_encoder_pool_push
    void push(uint32_t n, const uint32_t *sessions, const int16_t *pcm, const uint64_t *pcm_offsets, const uint32_t *n_frames,
              const uint8_t *end, uint8_t *out, const uint64_t *out_offsets, const uint64_t *out_caps, uint64_t *out_lens,
              uint32_t *n_chunks = nullptr)
    {
        ctx_->check(sea_b200_encoder_pool_push(pool_, n, sessions, pcm, pcm_offsets, n_frames, end, out, out_offsets, out_caps, out_lens, n_chunks));
    }
    // device buffers of the context's GPU; arguments as sea_b200_encoder_pool_push_device
    void push_device(uint32_t n, const uint32_t *sessions, const int16_t *d_pcm, const uint64_t *pcm_offsets, const uint32_t *n_frames,
                     const uint8_t *end, uint8_t *d_out, const uint64_t *out_offsets, const uint64_t *out_caps, uint64_t *out_lens,
                     uint32_t *n_chunks = nullptr)
    {
        ctx_->check(sea_b200_encoder_pool_push_device(pool_, n, sessions, d_pcm, pcm_offsets, n_frames, end, d_out, out_offsets, out_caps,
                                                      out_lens, n_chunks));
    }

private:
    Context *ctx_;
    sea_b200_encoder_pool *pool_ = nullptr;
};

// Every GPU of the box behind one handle (sea_b200_multi, SURVEY 8e): batch calls shard the streams over the GPUs in-process --
// one context and one host thread per GPU, nothing exchanged between them -- and report per-GPU counts.
class MultiContext {
public:
    struct Shares {
        std::vector<uint32_t> first_stream;  // index of the first stream each GPU took
        std::vector<uint64_t> amount;        // bytes written (encode) / samples produced (decode) per GPU
    };
    explicit MultiContext(const std::vector<int> &devices)
    {
        int rc = sea_b200_multi_create(devices.data(), (uint32_t)devices.size(), &m_);
        if (rc) throw SeaError(rc, "sea_b200_multi_create failed (libsea_b200 has no CPU fallback)");
    }
    ~MultiContext() { sea_b200_multi_destroy(m_); }
    MultiContext(const MultiContext &) = delete;
    MultiContext &operator=(const MultiContext &) = delete;
    uint32_t device_count() const { return sea_b200_multi_device_count(m_); }
    // n independent sea_encode calls (lib.rs:13-36) over all GPUs; arguments as sea_b200_encode_batch
    Shares encode_batch(uint32_t n_streams, const int16_t *pcm, const uint64_t *pcm_offsets, const uint32_t *n_frames, uint32_t sample_rate,
                        uint32_t channels, const sea_b200_settings &settings, uint8_t *out, const uint64_t *out_offsets, uint64_t *out_lens)
    {
        Shares sh{std::vector<uint32_t>(device_count()), std::vector<uint64_t>(device_count())};
        check(sea_b200_multi_encode_batch(m_, n_streams, pcm, pcm_offsets, n_frames, sample_rate, channels, &settings, out, out_offsets, out_lens,
                                          sh.first_stream.data(), sh.amount.data()));
        return sh;
    }
    // n independent sea_decode calls (lib.rs:44-63) over all GPUs; arguments as sea_b200_decode_batch
    Shares decode_batch(uint32_t n_streams, const uint8_t *sea, const uint64_t *sea_offsets, const uint64_t *sea_lens, int16_t *pcm,
                        const uint64_t *pcm_offsets, const uint64_t *pcm_caps, uint64_t *n_samples)
    {
        Shares sh{std::vector<uint32_t>(device_count()), std::vector<uint64_t>(device_count())};
        check(sea_b200_multi_decode_batch(m_, n_streams, sea, sea_offsets, sea_lens, pcm, pcm_offsets, pcm_caps, n_samples,
                                          sh.first_stream.data(), sh.amount.data()));
        return sh;
    }

private:
    void check(int rc) const
    {
        if (rc < 0) throw SeaError(rc, sea_b200_multi_last_error(m_));
    }
    sea_b200_multi *m_ = nullptr;
};

// In-memory reader/writer with the std::io::Read / Write shape the reference is generic over.
struct SliceReader {
    const uint8_t *p;
    size_t len, pos = 0;
    SliceReader(const void *data, size_t n) : p(static_cast<const uint8_t *>(data)), len(n) {}
    size_t read(void *dst, size_t n)
    {
        size_t k = n < len - pos ? n : len - pos;
        std::memcpy(dst, p + pos, k);
        pos += k;
        return k;
    }
};
struct VecWriter {
    std::vector<uint8_t> data;
    void write(const void *src, size_t n)
    {
        const uint8_t *b = static_cast<const uint8_t *>(src);
        data.insert(data.end(), b, b + n);
    }
};

namespace detail {
template <class R>
std::vector<uint8_t> read_max_or_zero(R &r, size_t n)  // common.rs:103-123
{
    std::vector<uint8_t> buf(n);
    size_t got = 0;
    while (got < n) {
        size_t k = r.read(buf.data() + got, n - got);
        if (k == 0) break;
        got += k;
    }
    buf.resize(got);
    return buf;
}
inline void put_header(std::vector<uint8_t> &out, uint8_t channels, uint16_t chunk_size, uint16_t fpc, uint32_t rate, uint32_t total)
{  // file.rs:78-93, empty metadata
    const uint8_t m[4] = {'s', 'e', 'a', 'c'};
    out.insert(out.end(), m, m + 4);
    out.push_back(1);
    out.push_back(channels);
    out.push_back((uint8_t)chunk_size);
    out.push_back((uint8_t)(chunk_size >> 8));
    out.push_back((uint8_t)fpc);
    out.push_back((uint8_t)(fpc >> 8));
    for (int i = 0; i < 4; i++) out.push_back((uint8_t)(rate >> (8 * i)));
    for (int i = 0; i < 4; i++) out.push_back((uint8_t)(total >> (8 * i)));
    for (int i = 0; i < 4; i++) out.push_back(0);
}
}  // namespace detail

template <class R, class W>
class SeaEncoder {  // encoder.rs:37-159
public:
    SeaEncoder(Context &ctx, uint8_t channels, uint32_t sample_rate, std::optional<uint32_t> total_frames, const EncoderSettings &settings,
               R &reader, W &writer)
        : ctx_(ctx), reader_(reader), writer_(writer), settings_(settings), channels_(channels), sample_rate_(sample_rate),
          total_frames_(total_frames.value_or(0))
    {
        sea_b200_settings s = settings.c();
        ctx_.check(sea_b200_encoder_create(ctx.get(), channels, sample_rate, &s, &enc_));
        if (total_frames && *total_frames == 0) {  // encoder.rs:73-78
            std::vector<uint8_t> h;
            detail::put_header(h, channels_, 0, settings_.frames_per_chunk, sample_rate_, 0);
            writer_.write(h.data(), h.size());
            state_ = Writing;
        }
    }
    ~SeaEncoder() { sea_b200_encoder_destroy(enc_); }

    bool encode_frame()  // encoder.rs:106-149: true while more input is expected
    {
        if (state_ == Finished) throw SeaError(SEA_B200_ERR_ENCODER_CLOSED, "encode_frame after the stream ended");
        const size_t fpc = settings_.frames_per_chunk;
        size_t frames = fpc;
        if (total_frames_ > 0) frames = std::min<size_t>(fpc, (size_t)total_frames_ - written_frames_);
        const size_t full = fpc * channels_;
        std::vector<uint8_t> raw = detail::read_max_or_zero(reader_, frames * channels_ * 2);
        if (raw.size() % (2 * (size_t)channels_) != 0) throw SeaError(SEA_B200_ERR_IO, "UnexpectedEof (encoder.rs:95-99)");
        const size_t n = raw.size() / 2;
        const bool eof = n == 0 || n < full;
        if (n) {
            std::vector<uint8_t> chunk(70000);
            uint64_t len = 0;
            ctx_.check(sea_b200_encoder_make_chunk(enc_, reinterpret_cast<const int16_t *>(raw.data()), n, chunk.data(), chunk.size(), &len));
            if (state_ == Start) {  // header goes out once the first chunk fixed chunk_size (encoder.rs:134-138)
                std::vector<uint8_t> h;
                detail::put_header(h, channels_, (uint16_t)sea_b200_encoder_chunk_size(enc_), settings_.frames_per_chunk, sample_rate_, total_frames_);
                writer_.write(h.data(), h.size());
                state_ = Writing;
            }
            writer_.write(chunk.data(), (size_t)len);
            written_frames_ += (uint32_t)frames;
        }
        if (eof) state_ = Finished;
        return !eof;
    }
    // Up to max_chunks encode_frame() steps in ONE launch (sea_b200_encoder_make_chunks): same bytes, same state machine.
    bool encode_frames(size_t max_chunks)
    {
        if (state_ == Finished) throw SeaError(SEA_B200_ERR_ENCODER_CLOSED, "encode_frames after the stream ended");
        const size_t fpc = settings_.frames_per_chunk, want = fpc * max_chunks;
        size_t frames = want;
        if (total_frames_ > 0) frames = std::min<size_t>(want, (size_t)total_frames_ - written_frames_);
        std::vector<uint8_t> raw = detail::read_max_or_zero(reader_, frames * channels_ * 2);
        if (raw.size() % (2 * (size_t)channels_) != 0) throw SeaError(SEA_B200_ERR_IO, "UnexpectedEof (encoder.rs:95-99)");
        const size_t n = raw.size() / 2;
        const bool eof = n == 0 || n < want * channels_;
        if (n) {
            std::vector<uint8_t> chunks(70000 * max_chunks);
            uint64_t len = 0;
            uint32_t n_chunks = 0;
            ctx_.check(sea_b200_encoder_make_chunks(enc_, reinterpret_cast<const int16_t *>(raw.data()), n, chunks.data(), chunks.size(), &len,
                                                    &n_chunks));
            if (state_ == Start) {
                std::vector<uint8_t> h;
                detail::put_header(h, channels_, (uint16_t)sea_b200_encoder_chunk_size(enc_), settings_.frames_per_chunk, sample_rate_, total_frames_);
                writer_.write(h.data(), h.size());
                state_ = Writing;
            }
            writer_.write(chunks.data(), (size_t)len);
            written_frames_ += (uint32_t)(n / channels_);
        }
        if (eof) state_ = Finished;
        return !eof;
    }
    void flush() {}
    void finalize() { state_ = Finished; }

private:
    enum State { Start, Writing, Finished };
    Context &ctx_;
    R &reader_;
    W &writer_;
    EncoderSettings settings_;
    uint8_t channels_;
    uint32_t sample_rate_, total_frames_;
    uint32_t written_frames_ = 0;
    State state_ = Start;
    sea_b200_encoder *enc_ = nullptr;
};

template <class R, class W>
class SeaDecoder {  // decoder.rs:10-72
public:
    SeaDecoder(Context &ctx, R &reader, W &writer) : ctx_(ctx), reader_(reader), writer_(writer)
    {
        std::vector<uint8_t> h = detail::read_max_or_zero(reader_, SEA_B200_FILE_HEADER_BYTES);
        ctx_.check(sea_b200_decoder_create(ctx.get(), h.data(), h.size(), &dec_));
        sea_b200_header hd;
        ctx_.check(sea_b200_decoder_header(dec_, &hd));
        header_ = {hd.version, hd.channels, hd.chunk_size, hd.frames_per_chunk, hd.sample_rate, hd.total_frames};
    }
    ~SeaDecoder() { sea_b200_decoder_destroy(dec_); }

    bool decode_frame()  // decoder.rs:33-59 + file.rs:180-209
    {
        if (header_.total_frames != 0 && header_.total_frames <= frames_read_) return false;
        const int64_t remaining = header_.total_frames > 0 ? (int64_t)(header_.total_frames - frames_read_) : -1;
        std::vector<uint8_t> encoded = detail::read_max_or_zero(reader_, header_.chunk_size);
        if (encoded.empty()) return false;
        std::vector<int16_t> pcm((size_t)header_.frames_per_chunk * header_.channels);
        uint64_t n = 0;
        ctx_.check(sea_b200_decoder_decode_chunk(dec_, encoded.data(), encoded.size(), remaining, pcm.data(), pcm.size(), &n));
        frames_read_ += n / header_.channels;
        writer_.write(pcm.data(), (size_t)n * 2);
        return true;
    }
    // Up to max_chunks decode_frame() steps in one chunk-parallel launch (sea_b200_decoder_decode_chunks).
    bool decode_frames(size_t max_chunks)
    {
        if (header_.total_frames != 0 && header_.total_frames <= frames_read_) return false;
        const int64_t remaining = header_.total_frames > 0 ? (int64_t)(header_.total_frames - frames_read_) : -1;
        std::vector<uint8_t> encoded = detail::read_max_or_zero(reader_, (size_t)header_.chunk_size * max_chunks);
        if (encoded.empty()) return false;
        std::vector<int16_t> pcm((size_t)header_.frames_per_chunk * header_.channels * max_chunks);
        uint64_t n = 0;
        ctx_.check(sea_b200_decoder_decode_chunks(dec_, ctx_.get(), encoded.data(), encoded.size(), remaining, pcm.data(), pcm.size(), &n));
        frames_read_ += n / header_.channels;
        writer_.write(pcm.data(), (size_t)n * 2);
        return true;
    }
    void flush() {}
    void finalize() {}
    SeaFileHeader get_header() const { return header_; }

private:
    Context &ctx_;
    R &reader_;
    W &writer_;
    SeaFileHeader header_{};
    uint64_t frames_read_ = 0;
    sea_b200_decoder *dec_ = nullptr;
};

struct SeaDecodeInfo {  // lib.rs:38-42
    std::vector<int16_t> samples;
    uint32_t sample_rate = 0, channels = 0;
};

// lib.rs:13-36 (one launch over the whole stream instead of a chunk loop)
inline std::vector<uint8_t> sea_encode(Context &ctx, const int16_t *input_samples, size_t n, uint32_t sample_rate, uint32_t channels,
                                       const EncoderSettings &settings)
{
    sea_b200_settings s = settings.c();
    uint64_t bound = 0, len = 0;
    ctx.check(sea_b200_encode_bound(channels ? n / channels : 0, channels, &s, &bound));
    std::vector<uint8_t> out(bound + 64);
    ctx.check(sea_b200_encode(ctx.get(), input_samples, n, sample_rate, channels, &s, out.data(), out.size(), &len));
    out.resize(len);
    return out;
}

// lib.rs:44-63
inline SeaDecodeInfo sea_decode(Context &ctx, const uint8_t *encoded, size_t len)
{
    SeaDecodeInfo info;
    uint64_t n = 0;
    ctx.check(sea_b200_decode(ctx.get(), encoded, len, nullptr, 0, &n, &info.sample_rate, &info.channels));
    info.samples.resize(n ? n : 1);
    ctx.check(sea_b200_decode(ctx.get(), encoded, len, info.samples.data(), info.samples.size(), &n, &info.sample_rate, &info.channels));
    info.samples.resize(n);
    return info;
}

// Random access (README.md:125 "seeking"): frames [first_frame, first_frame + n_frames) of a complete file; only the covering
// chunks are decoded.  skip_metadata = the format-compatible fix of file.rs:53-54.
inline SeaDecodeInfo sea_decode_range(Context &ctx, const uint8_t *encoded, size_t len, uint64_t first_frame, uint64_t n_frames,
                                      bool skip_metadata = false)
{
    SeaDecodeInfo info;
    uint64_t n = 0;
    const uint32_t flags = skip_metadata ? SEA_B200_RANGE_SKIP_METADATA : 0u;
    ctx.check(sea_b200_decode_range(ctx.get(), encoded, len, first_frame, n_frames, flags, nullptr, 0, &n, &info.sample_rate, &info.channels));
    info.samples.resize(n ? n : 1);
    ctx.check(sea_b200_decode_range(ctx.get(), encoded, len, first_frame, n_frames, flags, info.samples.data(), info.samples.size(), &n,
                                    &info.sample_rate, &info.channels));
    info.samples.resize(n);
    return info;
}

}  // namespace sea
