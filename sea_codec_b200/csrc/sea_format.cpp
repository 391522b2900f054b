// sea_format.cpp -- host-side container arithmetic and table generation (see sea_format.h).
// Compiled with -ffp-contract=off: the f32 steps below must be plain IEEE single operations in the order the
// reference performs them (SURVEY.md trap T16).
#include "sea_format.h"

#include <math.h>
#include <string.h>

#include <algorithm>

namespace sea {

static inline uint32_t rd_u16(const uint8_t *p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8); }
static inline uint32_t rd_u32(const uint8_t *p) { return rd_u16(p) | (rd_u16(p + 2) << 16); }

// file.rs:40-72.  Layout: "seac" | version | channels | chunk_size u16 | frames_per_chunk u16 | sample_rate u32 |
// total_frames u32 | metadata_size u32.  validate(): file.rs:33-38.
int parse_file_header(const uint8_t *p, uint64_t len, sea_b200_header *h)
{
    if (len < (uint64_t)kFileHeaderBytes) return SEA_B200_ERR_IO;  // read_exact -> io::Error
    if (memcmp(p, "seac", 4) != 0) return SEA_B200_ERR_INVALID_FILE;
    memset(h, 0, sizeof(*h));
    h->version = p[4];
    h->channels = p[5];
    h->chunk_size = (uint16_t)rd_u16(p + 6);
    h->frames_per_chunk = (uint16_t)rd_u16(p + 8);
    h->sample_rate = rd_u32(p + 10);
    h->total_frames = rd_u32(p + 14);
    h->metadata_size = rd_u32(p + 18);
    if (!(h->channels > 0 && h->chunk_size >= 16 && h->frames_per_chunk > 0 && h->sample_rate > 0))
        return SEA_B200_ERR_INVALID_FILE;
    return SEA_B200_OK;
}

// file.rs:78-93 with empty metadata (encoder.rs:65)
void write_file_header(uint8_t *p, uint8_t channels, uint16_t chunk_size, uint16_t frames_per_chunk, uint32_t sample_rate,
                       uint32_t total_frames)
{
    memcpy(p, "seac", 4);
    p[4] = 1;
    p[5] = channels;
    p[6] = (uint8_t)chunk_size;
    p[7] = (uint8_t)(chunk_size >> 8);
    p[8] = (uint8_t)frames_per_chunk;
    p[9] = (uint8_t)(frames_per_chunk >> 8);
    for (int i = 0; i < 4; i++) p[10 + i] = (uint8_t)(sample_rate >> (8 * i));
    for (int i = 0; i < 4; i++) p[14 + i] = (uint8_t)(total_frames >> (8 * i));
    memset(p + 18, 0, 4);
}

int plan_range(const sea_b200_header &h, uint64_t len, uint64_t first_frame, uint64_t n_frames, bool skip_metadata, RangePlan *p)
{
    memset(p, 0, sizeof(*p));
    p->body = kFileHeaderBytes;
    if (skip_metadata) p->body += h.metadata_size;  // what file.rs:53-54 meant to do
    if (p->body > len) return SEA_B200_ERR_IO;
    const uint64_t N = h.frames_per_chunk, avail_chunks = (len - p->body + h.chunk_size - 1) / h.chunk_size;
    // total_frames clamped to the chunks present (file.rs:186-188) or, streaming, whole chunks
    p->file_frames = h.total_frames ? std::min<uint64_t>(h.total_frames, avail_chunks * N) : (len - p->body) / h.chunk_size * N;
    if (first_frame >= p->file_frames || n_frames == 0) return SEA_B200_OK;
    const uint64_t end_frame = std::min(p->file_frames, first_frame + n_frames);
    p->k0 = first_frame / N;
    p->k1 = (end_frame + N - 1) / N;
    p->b0 = p->body + p->k0 * h.chunk_size;
    p->b1 = std::min<uint64_t>(len, p->body + p->k1 * h.chunk_size);
    // whole chunks only: a chunk's section layout depends on its own frame count (chunk.rs:105-113), so every covered chunk is
    // decoded at its true length and the requested frames are cut out afterwards
    p->sub_frames = std::min(p->file_frames, p->k1 * N) - p->k0 * N;
    p->skip = first_frame - p->k0 * N;
    p->want = end_frame - first_frame;
    return SEA_B200_OK;
}

// encoder_vbr.rs:40-63, evaluated in f32 in source order.
float vbr_normalized_bitrate(const sea_b200_settings *st)
{
    const float dist1 = 0.00f, dist2 = 0.95f, dist3 = 0.05f, dist4 = 0.00f;  // encoder_vbr.rs:21
    float rate = st->residual_bits;
    rate -= (4.0f * 16.0f * 2.0f) / (float)st->frames_per_chunk;
    rate -= (float)st->scale_factor_bits / (float)st->scale_factor_frames;
    rate -= 2.0f / (float)st->scale_factor_frames;
    float fl = floorf(st->residual_bits);
    float mean = dist1 * (fl - 1.0f) + dist2 * fl + dist3 * (fl + 1.0f) + dist4 * (fl + 2.0f);
    float diff = mean - fl;
    rate -= diff;
    return rate;
}

static inline uint64_t trunc_to_u64(float v)  // Rust `as usize`: saturating, NaN -> 0
{
    if (!(v > 0.0f)) return 0;
    if (v >= 18446744073709551616.0f) return UINT64_MAX;
    return (uint64_t)v;
}

// encoder_vbr.rs:66-96: repeated truncating split of what is left; leftovers go to the `base` bucket.
void vbr_distribution(uint64_t items, float target, uint64_t counts[4])
{
    const float dist[6] = {0.00f, 0.00f, 0.95f, 0.05f, 0.00f, 0.00f};
    float frac = target - truncf(target);
    float rest = 1.0f - frac;
    float share[4];
    for (int i = 0; i < 4; i++) share[i] = dist[i] * frac + dist[i + 1] * rest;
    counts[0] = counts[1] = counts[2] = counts[3] = 0;
    uint64_t placed = 0;
    while (placed < items) {
        uint64_t left = items - placed;
        for (int i = 0; i < 4; i++) {
            uint64_t v = trunc_to_u64((float)left * share[i]);
            placed += v;
            counts[i] += v;
        }
        if (items - placed == left) {
            placed += left;
            counts[1] += left;
        }
    }
}

uint32_t vbr_full_chunk_bytes(const EncodePlan &p)
{
    uint32_t items = (p.N / p.F) * p.channels;
    uint64_t bits = 0;
    for (int i = 0; i < 4; i++) bits += (uint64_t)p.full_counts[i] * (uint64_t)(p.base + (uint32_t)i - 1u);
    bits *= p.F;
    return 4u + 16u * p.channels + div_ceil_u32(items * p.s, 8u) + div_ceil_u32(items * 2u, 8u) + (uint32_t)((bits + 7u) / 8u);
}

int make_encode_plan(uint32_t channels, const sea_b200_settings *st, EncodePlan *plan)
{
    if (!st || channels == 0 || channels > 255) return SEA_B200_ERR_INVALID_PARAMETERS;
    if (st->scale_factor_bits < 1 || st->scale_factor_bits > 8) return SEA_B200_ERR_INVALID_PARAMETERS;
    if (st->scale_factor_frames == 0 || st->frames_per_chunk == 0) return SEA_B200_ERR_INVALID_PARAMETERS;
    if (st->frames_per_chunk % st->scale_factor_frames != 0) return SEA_B200_ERR_DOMAIN;  // chunk.rs:218 assert
    if (!(st->residual_bits >= 1.0f && st->residual_bits < 9.0f)) return SEA_B200_ERR_DOMAIN;  // common.rs:34 panic
    memset(plan, 0, sizeof(*plan));
    plan->channels = channels;
    plan->N = st->frames_per_chunk;
    plan->F = st->scale_factor_frames;
    plan->s = st->scale_factor_bits;
    plan->hdr_bits = (uint32_t)floorf(st->residual_bits);
    plan->vbr = st->vbr != 0;
    uint64_t items = (uint64_t)(plan->N / plan->F) * channels;
    if (!plan->vbr) {
        uint64_t bytes = 4ull + 16ull * channels + (items * plan->s + 7) / 8 + ((uint64_t)plan->N * channels * plan->hdr_bits + 7) / 8;
        if (bytes > 65535) return SEA_B200_ERR_DOMAIN;  // header.chunk_size is u16 (file.rs:166-168, :173-175)
        plan->full_chunk_bytes = plan->max_chunk_bytes = (uint32_t)bytes;
        plan->full_chunk_valid = true;
        return SEA_B200_OK;
    }
    plan->vbr_target = vbr_normalized_bitrate(st);
    float t = plan->vbr_target;
    plan->base = !(t > 0.0f) ? 0u : (t >= 255.0f ? 255u : (uint32_t)t);  // `as u8`
    // analysis runs at base+1 (encoder_vbr.rs:140) and every block gets a size from base-1..base+2
    // (SeaResidualSize::from panics outside 1..8: common.rs:24-36, trap T20)
    if (plan->base < 1 || plan->base + 1 > 8) return SEA_B200_ERR_DOMAIN;
    if (items > 65535) return SEA_B200_ERR_DOMAIN;  // u16 indices (encoder_vbr.rs:102)
    uint64_t counts[4];
    vbr_distribution(items, t, counts);
    for (int i = 0; i < 4; i++) plan->full_counts[i] = (uint32_t)counts[i];
    plan->full_chunk_valid = !((counts[0] && plan->base < 2) || (counts[2] && plan->base + 1 > 8) || (counts[3] && plan->base + 2 > 8));
    uint64_t full = vbr_full_chunk_bytes(*plan);
    uint64_t worst = 4ull + 16ull * channels + (items * plan->s + 7) / 8 + (items * 2 + 7) / 8 +
                     ((uint64_t)plan->N * channels * (plan->base + 2) + 7) / 8;
    if (full > 65535) return SEA_B200_ERR_DOMAIN;
    plan->full_chunk_bytes = (uint32_t)full;
    plan->max_chunk_bytes = (uint32_t)(worst > full ? worst : full);
    return SEA_B200_OK;
}

// ---- tables ------------------------------------------------------------------------------------------------

// dqt.rs:75-97: reconstruction levels for one residual size, in units of the scale factor.
static int level_curve(uint32_t b, float *lv)
{
    if (b == 1) {
        lv[0] = 2.0f;
        return 1;
    }
    if (b == 2) {
        lv[0] = 1.115f;
        lv[1] = 4.0f;
        return 2;
    }
    int n = 1 << (b - 1);
    float top = (float)((1 << b) - 1);
    float stride = floorf((top - 0.75f) / (float)(n - 1));
    lv[0] = 0.75f;
    for (int i = 1; i < n - 1; i++) lv[i] = 0.5f + (float)i * stride;
    lv[n - 1] = top;
    return n;
}

std::vector<int32_t> build_tables(uint32_t s)
{
    static const float pow_by_bits[8] = {12.0f, 11.65f, 11.20f, 10.58f, 9.64f, 8.75f, 7.66f, 6.63f};  // dqt.rs:14
    const uint32_t n = 1u << s;
    std::vector<int32_t> tab(tab_words(s), 0);
    std::vector<int32_t> sf(n);
    for (uint32_t b = 1; b <= 8; b++) {
        float e = pow_by_bits[b - 1] / (float)s;                                  // dqt.rs:40-42
        for (uint32_t i = 0; i < n; i++) sf[i] = (int32_t)powf((float)(i + 1), e);  // dqt.rs:49-52 (`as i32` truncates)
        int32_t *recip = tab.data() + tab_recip_off(s, b);
        for (uint32_t i = 0; i < n; i++) recip[i] = (int32_t)(65536.0f / (float)sf[i]);  // dqt.rs:64-67
        float lv[128];
        int levels = level_curve(b, lv);
        int32_t *rows = tab.data() + tab_dqt_off(s, b);
        for (uint32_t i = 0; i < n; i++)
            for (int k = 0; k < levels; k++) {
                int32_t mag = (int32_t)roundf((float)sf[i] * lv[k]);  // dqt.rs:116 (round half away from zero)
                rows[(i << b) + 2 * k] = mag;                           // even code = +, odd code = - (dqt.rs:117-118)
                rows[(i << b) + 2 * k + 1] = -mag;
            }
    }
    return tab;
}

}  // namespace sea
