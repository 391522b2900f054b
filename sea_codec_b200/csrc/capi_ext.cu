// capi_ext.cu -- entry points layered on the base C-ABI (capi.cu): random-access decode, multi-chunk streaming decode, and the
// two foreign-function surfaces the reference already ships (src/wasm_api.rs, c/sea.h) re-pointed at the GPU path.
// Nothing here touches a kernel directly; every codec byte still goes through libsea_b200's CUDA kernels (no CPU fallback).
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <mutex>
#include <vector>

#include "../../include/sea_b200.h"
#include "sea_format.h"

// capi.cu (not part of the public header): the decoder.rs:21 scale_factor_bits consistency check over a run of chunks
extern "C" __attribute__((visibility("hidden"))) int sea_b200_internal_check_sf_bits(sea_b200_decoder *dec, const uint8_t *chunks, uint64_t len, uint64_t stride);

namespace {

void put_le16(uint8_t *p, uint32_t v) { p[0] = (uint8_t)v; p[1] = (uint8_t)(v >> 8); }
void put_le32(uint8_t *p, uint32_t v) { for (int i = 0; i < 4; i++) p[i] = (uint8_t)(v >> (8 * i)); }

// file.rs:78-93 with empty metadata
void write_header(uint8_t *dst, const sea_b200_header &h, uint32_t total_frames)
{
    memcpy(dst, "seac", 4);
    dst[4] = h.version;
    dst[5] = h.channels;
    put_le16(dst + 6, h.chunk_size);
    put_le16(dst + 8, h.frames_per_chunk);
    put_le32(dst + 10, h.sample_rate);
    put_le32(dst + 14, total_frames);
    put_le32(dst + 18, 0);
}

// process-wide context for the context-free foreign surfaces below (wasm_api.rs / c/sea.h have no handle argument)
std::mutex g_mu;
sea_b200_ctx *g_ctx = nullptr;
int g_status = 0;

sea_b200_ctx *default_ctx()
{
    if (!g_ctx) {
        const char *dev = getenv("SEA_B200_DEVICE");
        g_status = sea_b200_ctx_create(dev ? atoi(dev) : 0, &g_ctx);
        if (g_status) g_ctx = nullptr;
    }
    return g_ctx;
}

}  // namespace

extern "C" {

int sea_b200_decode_range(sea_b200_ctx *ctx, const uint8_t *sea, uint64_t len, uint64_t first_frame, uint64_t n_frames, uint32_t flags,
                          int16_t *pcm, uint64_t pcm_cap_samples, uint64_t *n_samples, uint32_t *sample_rate, uint32_t *channels)
{
    if (!ctx || !sea || !n_samples) return SEA_B200_ERR_INVALID_PARAMETERS;
    *n_samples = 0;
    sea_b200_header h;
    int rc = sea_b200_parse_header(sea, len, &h);
    if (rc) return rc;
    if (sample_rate) *sample_rate = h.sample_rate;
    if (channels) *channels = h.channels;
    sea::RangePlan r;
    if ((rc = sea::plan_range(h, len, first_frame, n_frames, flags & SEA_B200_RANGE_SKIP_METADATA, &r)) != SEA_B200_OK) return rc;
    if (r.want == 0) return SEA_B200_OK;
    const uint64_t want = r.want * h.channels;
    if (!pcm) {  // size query (c/sea.h:209-211 pattern)
        *n_samples = want;
        return SEA_B200_OK;
    }
    if (want > pcm_cap_samples) return SEA_B200_ERR_CAPACITY;
    const uint64_t sub_frames = r.sub_frames;
    if (sub_frames > 0xffffffffull) return SEA_B200_ERR_TOO_MANY_FRAMES;
    // the sub-file keeps every covered chunk at its true length (see plan_range); the requested frames are cut out afterwards
    std::vector<uint8_t> file(SEA_B200_FILE_HEADER_BYTES + (r.b1 - r.b0));
    write_header(file.data(), h, (uint32_t)sub_frames);
    memcpy(file.data() + SEA_B200_FILE_HEADER_BYTES, sea + r.b0, r.b1 - r.b0);
    const uint64_t skip = r.skip * h.channels;
    if (skip == 0 && want == sub_frames * h.channels) {
        uint64_t got = 0;
        rc = sea_b200_decode(ctx, file.data(), file.size(), pcm, pcm_cap_samples, &got, nullptr, nullptr);
        if (rc == SEA_B200_OK) *n_samples = got;
        return rc;
    }
    std::vector<int16_t> tmp(sub_frames * h.channels);
    uint64_t got = 0;
    rc = sea_b200_decode(ctx, file.data(), file.size(), tmp.data(), tmp.size(), &got, nullptr, nullptr);
    if (rc) return rc;
    const uint64_t n = got > skip ? std::min(want, got - skip) : 0;
    memcpy(pcm, tmp.data() + skip, n * sizeof(int16_t));
    *n_samples = n;
    return SEA_B200_OK;
}

int sea_b200_decoder_decode_chunks(sea_b200_decoder *dec, sea_b200_ctx *ctx, const uint8_t *chunks, uint64_t len, int64_t remaining_frames,
                                   int16_t *pcm, uint64_t pcm_cap_samples, uint64_t *n_samples)
{
    if (!dec || !ctx || !chunks || !pcm || !n_samples) return SEA_B200_ERR_INVALID_PARAMETERS;
    *n_samples = 0;
    sea_b200_header h;
    int rc = sea_b200_decoder_header(dec, &h);
    if (rc) return rc;
    if (len == 0) return SEA_B200_OK;
    const uint64_t n_chunks = (len + h.chunk_size - 1) / h.chunk_size;
    uint64_t frames = n_chunks * h.frames_per_chunk;
    if (remaining_frames >= 0) frames = std::min<uint64_t>(frames, (uint64_t)remaining_frames);
    else if (len % h.chunk_size) return SEA_B200_ERR_INVALID_FRAME;  // chunk.rs:76-79: a short chunk needs a frame count
    if (frames == 0) return SEA_B200_OK;
    if (frames > 0xffffffffull) return SEA_B200_ERR_TOO_MANY_FRAMES;
    if (frames * h.channels > pcm_cap_samples) return SEA_B200_ERR_CAPACITY;
    if ((rc = sea_b200_internal_check_sf_bits(dec, chunks, len, h.chunk_size)) != SEA_B200_OK) return rc;
    std::vector<uint8_t> file(SEA_B200_FILE_HEADER_BYTES + len);
    write_header(file.data(), h, (uint32_t)frames);
    memcpy(file.data() + SEA_B200_FILE_HEADER_BYTES, chunks, len);
    return sea_b200_decode(ctx, file.data(), file.size(), pcm, pcm_cap_samples, n_samples, nullptr, nullptr);
}

// ---------------------------------------------------------------------------------------------- src/wasm_api.rs surface

void sea_b200_wasm_setup(void)
{
    std::lock_guard<std::mutex> lk(g_mu);
    default_ctx();
}

size_t sea_b200_wasm_sea_encode(const int16_t *input_samples, size_t input_length, uint32_t sample_rate, uint32_t channels, float bitrate,
                                bool vbr, uint8_t *output_buffer, size_t output_length)
{
    std::lock_guard<std::mutex> lk(g_mu);
    sea_b200_ctx *ctx = default_ctx();
    if (!ctx || !input_samples || !output_buffer) return 0;
    sea_b200_settings st;
    sea_b200_default_settings(&st);  // EncoderSettings { residual_bits: bitrate, vbr, ..Default::default() } (wasm_api.rs:47-51)
    st.residual_bits = bitrate;
    st.vbr = vbr ? 1 : 0;
    uint64_t out_len = 0;
    g_status = sea_b200_encode(ctx, input_samples, input_length / 2, sample_rate, channels, &st, output_buffer, output_length, &out_len);
    return g_status == SEA_B200_OK ? (size_t)out_len : 0;  // the reference asserts (wasm_api.rs:58); 0 + sea_b200_wasm_status() here
}

size_t sea_b200_wasm_sea_decode(const uint8_t *encoded, size_t encoded_length, int16_t *output_buffer, size_t output_length,
                                uint32_t *sample_rate, uint32_t *channels)
{
    std::lock_guard<std::mutex> lk(g_mu);
    sea_b200_ctx *ctx = default_ctx();
    if (!ctx || !encoded || !output_buffer) return 0;
    uint64_t n = 0;
    g_status = sea_b200_decode(ctx, encoded, encoded_length, output_buffer, output_length / 2, &n, sample_rate, channels);
    return g_status == SEA_B200_OK ? (size_t)n * 2 : 0;  // bytes, like wasm_api.rs:94
}

uint8_t *sea_b200_wasm_allocate(size_t size) { return static_cast<uint8_t *>(sea_b200_host_alloc(size)); }
void sea_b200_wasm_deallocate(uint8_t *ptr, size_t size)
{
    (void)size;
    sea_b200_host_free(ptr);
}
int sea_b200_wasm_status(void) { return g_status; }

// ---------------------------------------------------------------------------------------------- c/sea.h surface

int sea_b200_csea_decode(uint8_t *encoded, uint32_t encoded_len, uint32_t *sample_rate, uint32_t *channels, int16_t *output,
                         uint32_t *total_frames)
{
    if (!encoded || !sample_rate || !channels || !total_frames) return 1;
    sea_b200_header h;
    if (sea_b200_parse_header(encoded, encoded_len, &h) != SEA_B200_OK) {
        fprintf(stderr, "Invalid file\n");  // c/sea.h:196-199
        return 1;
    }
    *sample_rate = h.sample_rate;
    *channels = h.channels;
    *total_frames = h.total_frames;
    if (output == NULL) return 0;  // c/sea.h:209-211
    std::lock_guard<std::mutex> lk(g_mu);
    sea_b200_ctx *ctx = default_ctx();
    uint64_t n = 0;
    g_status = ctx ? sea_b200_decode(ctx, encoded, encoded_len, output, (uint64_t)h.total_frames * h.channels, &n, nullptr, nullptr) : g_status;
    if (!ctx || g_status != SEA_B200_OK || n != (uint64_t)h.total_frames * h.channels) {
        fprintf(stderr, "Decode error\n");  // c/sea.h:218-221
        return 2;
    }
    return 0;
}

}  // extern "C"
