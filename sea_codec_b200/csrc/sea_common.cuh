// sea_common.cuh -- arithmetic shared by the SEA kernels (and callable on the host for unit checks).
//
// Every function states the reference lines (under /root/reference/src/codec) whose result it reproduces.
// Nothing here is a table walk of the reference: the quantiser is a closed form, the LMS keeps signs as
// +-1 multipliers, ranks are accumulated with 64-bit fused multiply-adds.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define SEA_HD __host__ __device__ __forceinline__
#else
#define SEA_HD inline
#endif

namespace sea {

constexpr int kLmsLen = 4;
constexpr int kFileHeaderBytes = 22;

// Device table layout for one scale_factor_bits value `s` (n = 2^s):
//   [0, 8n)            reciprocals   recip[b-1][sf]                      (dqt.rs:57-69)
//   [8n, 8n + 510n)    dequant rows  dqt_b[sf][code] at 8n + n*(2^b-2)   (dqt.rs:99-126)
SEA_HD uint32_t tab_recip_off(uint32_t s, uint32_t b) { return (b - 1u) << s; }
SEA_HD uint32_t tab_dqt_off(uint32_t s, uint32_t b) { return (8u << s) + (((1u << b) - 2u) << s); }
SEA_HD uint32_t tab_words(uint32_t s) { return 518u << s; }

struct DevTables {
    const int32_t *by_s[9];  // index = scale_factor_bits (1..8); device pointers
};

// lms.rs:33-41 -- wrapping i32 dot product, arithmetic shift (release-build semantics, trap T7).
SEA_HD int32_t lms_predict(const int32_t w[4], const int32_t h[4])
{
    uint32_t acc = (uint32_t)w[0] * (uint32_t)h[0] + (uint32_t)w[1] * (uint32_t)h[1] + (uint32_t)w[2] * (uint32_t)h[2] +
                   (uint32_t)w[3] * (uint32_t)h[3];
    return (int32_t)acc >> 13;
}

// common.rs:5-8
SEA_HD int32_t clamp_i16(int32_t v) { return v < -32768 ? -32768 : (v > 32767 ? 32767 : v); }

// lms.rs:43-51 -- w[i] += (h[i] < 0 ? -delta : delta); history shifts in the reconstructed sample.
SEA_HD void lms_update(int32_t w[4], int32_t h[4], int32_t y, int32_t d)
{
    int32_t delta = d >> 4;
    for (int i = 0; i < 4; i++) {  // constant trip count: fully unrolled by nvcc
        int32_t sg = (h[i] >> 31) | 1;  // -1 for negative history, +1 otherwise (zero counts as +, trap T8)
        w[i] = (int32_t)((uint32_t)w[i] + (uint32_t)(delta * sg));
    }
    h[0] = h[1];
    h[1] = h[2];
    h[2] = h[3];
    h[3] = y;
}

// The same update with the history signs carried in registers (sg[i] = h[i] < 0 ? -1 : +1, zero counts as +): the per-tap
// shift+or of lms_update becomes one per sample.  Callers initialise sg from h once per chunk.
SEA_HD void lms_signs(int32_t sg[4], const int32_t h[4])
{
    for (int i = 0; i < 4; i++) sg[i] = (h[i] >> 31) | 1;
}
SEA_HD void lms_update_sg(int32_t w[4], int32_t h[4], int32_t sg[4], int32_t y, int32_t d)
{
    const int32_t delta = d >> 4;
    for (int i = 0; i < 4; i++) w[i] = (int32_t)((uint32_t)w[i] + (uint32_t)(delta * sg[i]));
    h[0] = h[1]; h[1] = h[2]; h[2] = h[3]; h[3] = y;
    sg[0] = sg[1]; sg[1] = sg[2]; sg[2] = sg[3]; sg[3] = (y >> 31) | 1;
}

// lms.rs:53-62 -- max(0, (sum w^2 >> 18) - 0x8ff)^2, wrapping u64 like the release build.
SEA_HD uint64_t lms_penalty(const int32_t w[4])
{
    uint64_t sum = (uint64_t)((int64_t)w[0] * w[0]) + (uint64_t)((int64_t)w[1] * w[1]) + (uint64_t)((int64_t)w[2] * w[2]) +
                   (uint64_t)((int64_t)w[3] * w[3]);
    int64_t p = ((int64_t)sum >> 18) - 0x8ff;
    uint64_t q = p > 0 ? (uint64_t)p : 0;
    return q * q;
}

// rank += err^2 + penalty(w), exactly as encoder_base.rs:78-82 with lms.rs:53-62 (wrapping u64).
// NARROW = true is valid while every |w[i]| < 2^23 (then sum(w^2) < 2^48, the shifted sum fits 31 bits and the square is one
// 32x32->64 multiply-add); callers establish that bound once per block, not per sample.
template <bool NARROW>
SEA_HD uint64_t rank_step(uint64_t rank, int32_t err, const int32_t w[4])
{
    const uint64_t sum = (uint64_t)((int64_t)w[0] * w[0]) + (uint64_t)((int64_t)w[1] * w[1]) + (uint64_t)((int64_t)w[2] * w[2]) +
                         (uint64_t)((int64_t)w[3] * w[3]);
    rank += (uint64_t)((int64_t)err * (int64_t)err);
    if (NARROW) {
#if defined(__CUDA_ARCH__)
        const int32_t t = __viaddmax_s32((int32_t)(uint32_t)(sum >> 18), -0x8ff, 0);  // one VIADDMNMX
#else
        int32_t t = (int32_t)(uint32_t)(sum >> 18) - 0x8ff;
        t = t > 0 ? t : 0;
#endif
        return rank + (uint64_t)(uint32_t)t * (uint64_t)(uint32_t)t;
    }
    const int64_t p = ((int64_t)sum >> 18) - 0x8ff;
    const uint64_t q = p > 0 ? (uint64_t)p : 0;
    return rank + q * q;
}
// a weight moves by at most |d >> 4| <= 1578 per sample (|d| <= 255 * 99, dqt.rs) -> bound over a block of F samples
SEA_HD bool weights_stay_narrow(const int32_t w[4], uint32_t F)
{
    const int32_t lim = (1 << 23) - 1 - (int32_t)F * 1600;
    uint32_t m = 0;  // max |w[i]| (|INT_MIN| wraps to 2^31 as unsigned: still >= lim)
    for (int i = 0; i < 4; i++) {
        const uint32_t a = w[i] < 0 ? 0u - (uint32_t)w[i] : (uint32_t)w[i];
        m = a > m ? a : m;
    }
    return m < (uint32_t)lim;
}

// encoder_base.rs:22-26 (sea_div) + :71-72 (clamp, SeaQuantTab lookup) as one closed form.
//   n = (r*recip + 2^15) >> 16 (i64, floor);  scaled = n + (sgn(r) - sgn(n)).
// Because recip > 0, n never has the opposite sign of r; the fix-up only turns 0 into sgn(r), which does not
// change |scaled| >> 1.  qt.rs:9-31 is the zig-zag  code = 2*min(|c|>>1, 2^(b-1)-1) + (c<0), except b == 2 where
// the magnitude index is (|c| >= 3) (qt.rs:26-30).  Verified exhaustively against the table in tests.
SEA_HD uint32_t quant_code(int32_t r, int32_t recip, uint32_t b)
{
    int64_t n64 = ((int64_t)r * (int64_t)recip + 32768) >> 16;
    int32_t n = (int32_t)n64;
    uint32_t an = n < 0 ? 0u - (uint32_t)n : (uint32_t)n;
    uint32_t kmax = (1u << (b - 1u)) - 1u;
    uint32_t k = an >> 1;
    k = k < kmax ? k : kmax;
    if (b == 2u) k = an >= 3u ? 1u : 0u;
    return 2u * k + ((uint32_t)r >> 31);
}

SEA_HD uint32_t div_ceil_u32(uint32_t a, uint32_t b) { return (a + b - 1u) / b; }

// The window part of plan_range (sea_format.cpp) for a stream that delivers file_frames frames in chunks of N frames: frames
// [first, first + n) start `skip` frames into chunk k0, and the stream has `want` of them.  Past the end (or n == 0): all zero, as
// plan_range leaves them.  The corpus kernels evaluate it per window on the device.
struct WindowPlan {
    uint64_t k0, skip, want;
};
SEA_HD WindowPlan window_plan(uint64_t file_frames, uint32_t N, uint64_t first, uint64_t n)
{
    WindowPlan p = {0, 0, 0};
    if (first >= file_frames || n == 0) return p;
    p.k0 = first / N;
    p.skip = first - p.k0 * N;
    p.want = file_frames - first < n ? file_frames - first : n;
    return p;
}

}  // namespace sea
