// sea_format.h -- host-side .sea container arithmetic: file header, chunk geometry, VBR plan, table generation.
// This is the scalar part of the path that stays on the host (SURVEY.md section 7 step 2); the kernels read and
// write the wire layout directly (SURVEY.md Appendix A).
#pragma once
#include <stdint.h>

#include <vector>

#include "../../include/sea_b200.h"
#include "sea_common.cuh"

namespace sea {

// ---- file header: file.rs:40-93 ------------------------------------------------------------------------
int parse_file_header(const uint8_t *p, uint64_t len, sea_b200_header *h);
void write_file_header(uint8_t *p, uint8_t channels, uint16_t chunk_size, uint16_t frames_per_chunk, uint32_t sample_rate,
                       uint32_t total_frames);

// ---- random access: which chunks cover frames [first_frame, first_frame + n_frames) of a file -------------
// Shared by sea_b200_decode_range and sea_b200_decode_windows_device, so that a window holds exactly what decode_range returns.
struct RangePlan {
    uint64_t body;         // byte offset of chunk 0 (22, or 22 + metadata_size with the metadata skip)
    uint64_t file_frames;  // frames the file can deliver: total_frames clamped to the chunks present, or, streaming, whole chunks
    uint64_t k0, k1;       // covering chunks [k0, k1); chunk k starts at body + k * chunk_size (file.rs:185)
    uint64_t b0, b1;       // their bytes [b0, b1) in the file (b1 clamped to its length)
    uint64_t sub_frames;   // frames of the covering chunks: whole chunks, or up to the file's end
    uint64_t skip;         // frames of chunk k0 before first_frame
    uint64_t want;         // frames of the range the file has (0: nothing to decode)
};
// SEA_B200_ERR_IO when the body starts past the file's end; otherwise OK (want == 0 for an empty range).
int plan_range(const sea_b200_header &h, uint64_t len, uint64_t first_frame, uint64_t n_frames, bool skip_metadata, RangePlan *p);

// ---- settings ------------------------------------------------------------------------------------------
// Resolved, validated view of EncoderSettings for one (channels) configuration.
struct EncodePlan {
    uint32_t channels, N, F, s;  // frames_per_chunk, scale_factor_frames, scale_factor_bits
    uint32_t hdr_bits;           // floor(residual_bits): chunk header nibble (chunk.rs:60)
    bool vbr;
    float vbr_target;            // encoder_vbr.rs:40-63
    uint32_t base;               // (u8)vbr_target
    uint32_t full_counts[4];     // interpolate_distribution(N*C/F) -> [base-1, base, base+1, base+2]
    bool full_chunk_valid;       // false when a full chunk would get a size outside 1..8 (the reference panics)
    uint32_t full_chunk_bytes;   // header.chunk_size of a full chunk
    uint32_t max_chunk_bytes;    // upper bound over partial chunks too (smem sizing)
};

// Returns SEA_B200_OK or INVALID_PARAMETERS / DOMAIN (the reference would panic).
int make_encode_plan(uint32_t channels, const sea_b200_settings *st, EncodePlan *plan);

float vbr_normalized_bitrate(const sea_b200_settings *st);                       // encoder_vbr.rs:40-63
void vbr_distribution(uint64_t items, float target, uint64_t counts[4]);         // encoder_vbr.rs:66-96

// chunk bytes of a CBR chunk with `frames` frames (chunk.rs:215-292; SURVEY App. D formula)
inline uint32_t cbr_chunk_bytes(uint32_t frames, uint32_t C, uint32_t s, uint32_t F, uint32_t b)
{
    uint32_t items = div_ceil_u32(frames, F) * C;
    return 4u + 16u * C + div_ceil_u32(items * s, 8u) + (uint32_t)(((uint64_t)frames * C * b + 7u) / 8u);
}
// bytes of a VBR chunk given the bucket counts (sizes base-1, base, base+1, base+2) when every block is full
uint32_t vbr_full_chunk_bytes(const EncodePlan &p);

// ---- quantiser tables: dqt.rs:40-126 ---------------------------------------------------------------------
// Flat table for scale_factor_bits = s in the device layout of sea_common.cuh (tab_words(s) int32 values).
std::vector<int32_t> build_tables(uint32_t s);

}  // namespace sea
