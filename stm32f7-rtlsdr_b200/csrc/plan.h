/*
 * plan.h -- host-side launch planning shared by the C-ABI implementation (api.cu) and by the
 * CPU emulation harness of the test-suite: output lengths, tile / segment split, constant blocks.
 */
#ifndef B200_PLAN_H
#define B200_PLAN_H

#include <cstdint>
#include <cstring>

#include "filter_design.h"
#include "spectrum.cuh"
#include "wbfm.cuh"
#include "wbfm_tc.cuh"
#include "am.cuh"

namespace b200 {

inline uint64_t ceil_div(uint64_t a, uint64_t b) { return (a + b - 1) / b; }

/* lengths in complex samples L = bytes / 2 */
inline uint64_t spectrum_frames(uint64_t len_bytes)
{
    const uint64_t n = len_bytes / 2;
    return n < 1024 ? 0 : (n - 1024) / 512 + 1;
}
inline uint64_t wbfm_disc_len(uint64_t len_bytes) { return ceil_div(len_bytes / 2, 10); }
inline uint64_t wbfm_audio_len(uint64_t len_bytes) { return ceil_div(wbfm_disc_len(len_bytes), 5); }
inline uint64_t am_y2_len(uint64_t len_bytes) { return ceil_div(ceil_div(len_bytes / 2, 20), 10); }
inline uint64_t am_audio_len(uint64_t len_bytes) { return ceil_div(2 * am_y2_len(len_bytes), 3); }

/* ---- spectrum: work units of 4 x frames_per_warp consecutive frames, persistent grid ----
 * frames_per_warp follows from the capture LENGTH only -- never from the batch size or the device -- so the
 * summation tree of one capture (frames in a warp, warps in a unit, units in k_spectrum_finalize) and with it
 * every bit of its spectrum is the same for the capture alone, in a batch of 512 and in a 4096 / N shard on
 * any GPU (SURVEY.md section 4(iv): bitwise per-capture results on 1 vs 8 GPUs).  The length rule: as many
 * units as one capture needs to fill every resident CTA slot of a B200 once (2 x 148 slots x 4 warps),
 * at most 64 frames per warp (the partial sums then stay below 2 % of the input bytes); a batch amortises
 * the per-CTA prologue through the persistent grid instead of through longer warps. */
constexpr uint32_t kSpecWarpsToFill = 2u * 148u * B200_SPEC_WARPS; /* a constant, not the device's SM count */
constexpr uint32_t kSpecMaxFramesPerWarp = 64;
struct SpectrumPlan {
    uint32_t frames, frames_per_warp, units_per_capture, grid;
    uint64_t total_units;
};
inline uint32_t spectrum_frames_per_warp(uint64_t frames)
{
    uint64_t fpw = ceil_div(frames, kSpecWarpsToFill);
    if (fpw < 1) fpw = 1;
    if (fpw > kSpecMaxFramesPerWarp) fpw = kSpecMaxFramesPerWarp;
    return (uint32_t)fpw;
}
inline SpectrumPlan plan_spectrum(uint64_t len_bytes, uint32_t n_captures, uint32_t sm_count)
{
    SpectrumPlan pl{};
    pl.frames = (uint32_t)spectrum_frames(len_bytes);
    if (pl.frames == 0) return pl;
    pl.frames_per_warp = spectrum_frames_per_warp(pl.frames);
    pl.units_per_capture = (uint32_t)ceil_div(pl.frames, (uint64_t)pl.frames_per_warp * B200_SPEC_WARPS);
    pl.total_units = (uint64_t)pl.units_per_capture * n_captures;
    /* the device only decides how many CTAs share the units, which no result depends on */
    const uint64_t slots = (uint64_t)sm_count * B200_SPEC_MINB;
    pl.grid = (uint32_t)(pl.total_units < slots ? pl.total_units : slots);
    return pl;
}

/* ---- WBFM ---- */
/* streaming launches: tiles per CTA.  A ring slot is a handful of tiles and the GPU is otherwise idle, so what counts is
 * the slot's latency: one tile per CTA (each CTA after the first also pre-rolls the tile before its own) */
constexpr uint32_t kFmStreamTilesPerSegment = 1;
struct FmPlan {
    uint32_t n_tiles, total_chunks, tiles_per_segment, segments;
    uint64_t m1;
};
/* whole captures (batched path): every stage-1 output m < ceil(L/10) */
inline FmPlan plan_wbfm_batch(uint64_t len_bytes, uint32_t n_captures, uint32_t sm_count)
{
    FmPlan pl{};
    const uint64_t n = len_bytes / 2;
    pl.m1 = ceil_div(n, 10);
    pl.total_chunks = (uint32_t)ceil_div(n, B200_FM_CHUNK);
    pl.n_tiles = (uint32_t)ceil_div(pl.total_chunks, B200_FM_THREADS);
    /* many equal segments (>= ~10 waves of CTAs, so the last partial wave is small) but never shorter
     * than 16 tiles: segments > 0 re-run one tile as pre-roll */
    uint64_t want = ceil_div((uint64_t)sm_count * 40, n_captures ? n_captures : 1);
    uint64_t tps = want ? ceil_div(pl.n_tiles, want) : pl.n_tiles;
    if (tps < 16) tps = 16;
    if (tps > pl.n_tiles) tps = pl.n_tiles ? pl.n_tiles : 1;
    pl.tiles_per_segment = (uint32_t)tps;
    pl.segments = (uint32_t)ceil_div(pl.n_tiles, tps);
    if (pl.segments == 0) pl.segments = 1;
    return pl;
}

inline void fill_fm_taps(FmTaps &t)
{
    const std::vector<double> h1 = design_taps(0), h2 = design_taps(1);
    for (int k = 0; k < B200_FM_T1; ++k) t.h1[k] = (float)h1[k];
    /* raw-byte form of the FIR (cplx2.cuh form C): taps x 2^133, and the -127.5 offset summed over the
     * float taps actually used, so the constant part of the input cancels to rounding */
    double total = 0.0, run = 0.0;
    for (int k = 0; k < B200_FM_T1; ++k) {
        t.h1s[k] = (float)std::ldexp((double)t.h1[k], B200_U8RAW_LOG2);
        total += (double)t.h1[k];
    }
    t.bias_half = (float)(-127.5 * total / 2);
    /* output i of a stream sees real samples through taps k <= 10 i only */
    for (int k = 0; k < B200_FM_T1; ++k) {
        run += (double)t.h1[k];
        if (k % 10 == 0 && k / 10 < 8) t.bias_head[k / 10] = (float)(-127.5 * run);
    }
    for (int k = 0; k < B200_FM_T2; ++k) t.h2[k] = (float)h2[k];
    const double alpha = deemph_alpha(), a = 1.0 - alpha;
    t.alpha = (float)alpha;
    for (int i = 0; i < 32; ++i) t.apow[i] = (float)std::pow(a, i + 1);
    const double a12 = std::pow(a, B200_FM_OPT);
    t.a12 = (float)a12;
    for (int s = 0; s < 5; ++s) t.a12pow[s] = (float)std::pow(a12, double(1 << s));
    t.a384 = (float)std::pow(a12, 32.0);
}

/* ---- WBFM, tensor-core engine (wbfm_tc.cuh) ---- */
struct FmTcPlan {
    uint32_t n_tiles, total_rows, tiles_per_segment, segments, grid;
    uint64_t m1;
};
inline FmTcPlan plan_wbfm_tc(uint64_t len_bytes, uint32_t n_captures, uint32_t sm_count)
{
    FmTcPlan pl{};
    const uint64_t n = len_bytes / 2;
    pl.m1 = ceil_div(n, 10);
    pl.total_rows = (uint32_t)ceil_div(n, B200_TC_ROW_SAMPLES);
    pl.n_tiles = (uint32_t)ceil_div(pl.total_rows, B200_TC_ROWS);
    /* work items = (capture, segment), handed to one persistent CTA per SM round-robin.  Every segment after the first
     * pre-rolls one tile, and the CTA with the most items sets the time, so the segment length is the one that minimises
     * rounds x (tiles per item + 1) -- at least 8 tiles, so the pre-roll stays below 1 in 9 */
    uint64_t best_tps = pl.n_tiles ? pl.n_tiles : 1, best_cost = ~0ull;
    for (uint64_t tps = pl.n_tiles < 8 ? (pl.n_tiles ? pl.n_tiles : 1) : 8; tps <= pl.n_tiles; ++tps) {
        const uint64_t segs = ceil_div(pl.n_tiles, tps), rounds = ceil_div(segs * (n_captures ? n_captures : 1), sm_count);
        const uint64_t cost = rounds * (tps + (segs > 1 ? 1 : 0));
        if (cost < best_cost) { best_cost = cost; best_tps = tps; }
    }
    pl.tiles_per_segment = (uint32_t)best_tps;
    pl.segments = (uint32_t)ceil_div(pl.n_tiles, best_tps);
    if (pl.segments == 0) pl.segments = 1;
    const uint64_t items = (uint64_t)pl.segments * n_captures;
    pl.grid = (uint32_t)(items < sm_count ? items : sm_count);
    return pl;
}
/* The stage-1 taps as three signed 8-bit slices, h[t] 2^e = q0 2^-7 + q1 2^-14 + q2 2^-21 (+ at most 2^-22), the
 * constants of the slice combine, and the B operand as it lies in shared memory (B200_TC_B_BYTES, 128B swizzle).
 * q[s][t] (optional) receives the slices, *e_out the exponent. */
inline void fill_fm_tc(FmTcConsts &c, uint8_t *image, int8_t (*q_out)[B200_FM_T1] = nullptr, int *e_out = nullptr)
{
    const std::vector<double> h1 = design_taps(0), h2 = design_taps(1);
    double hmax = 0.0;
    for (double v : h1) hmax = std::fabs(v) > hmax ? std::fabs(v) : hmax;
    int e = 0;
    while (std::ldexp(hmax, e + 1 + 7) <= 127.0) ++e; /* largest e with |h| 2^e 2^7 <= 127 */
    int8_t q[3][B200_FM_T1];
    double sum[3] = {0, 0, 0};
    for (int t = 0; t < B200_FM_T1; ++t) {
        double r = std::ldexp(h1[t], e);
        for (int s = 0; s < 3; ++s) {
            double v = std::nearbyint(std::ldexp(r, 7 * (s + 1)));
            if (v > 127) v = 127;
            if (v < -127) v = -127;
            q[s][t] = (int8_t)v;
            r -= std::ldexp(v, -7 * (s + 1));
            sum[s] += v;
        }
    }
    const double c0 = std::ldexp(1.0, -7 - e), c1 = std::ldexp(1.0, -14 - e), c2 = std::ldexp(1.0, -21 - e);
    c.c0 = (float)c0; c.c1 = (float)c1; c.c2 = (float)c2;
    c.b0 = (float)(127.5 * sum[0]);
    c.k12 = (float)(-127.5 * (c1 * sum[1] + c2 * sum[2]));
    for (int i = 0; i < 16; ++i) {
        double s0 = 0, s1 = 0, s2 = 0;
        for (int t = 0; t < B200_FM_T1 && t <= 10 * i; ++t) { s0 += q[0][t]; s1 += q[1][t]; s2 += q[2][t]; }
        c.b0_first[i] = (float)(127.5 * s0);
        c.k12_first[i] = (float)(-127.5 * (c1 * s1 + c2 * s2));
    }
    const double alpha = deemph_alpha(), a = 1.0 - alpha, a16 = std::pow(a, B200_TC_OPR);
    c.alpha = (float)alpha;
    for (int i = 0; i < B200_TC_OPR; ++i) c.apow[i] = (float)std::pow(a, i + 1);
    for (int s = 0; s < 5; ++s) c.a16pow[s] = (float)std::pow(a16, double(1 << s));
    for (int t = 0; t < B200_FM_T2; ++t) c.h2[t] = (float)h2[t];
    if (image) {
        /* column (s, j, comp) = slice s of output o = j - 1 of the row on the bytes of component comp; K byte 2 kap + comp is
         * sample kap of the row's window, which starts 96 samples before the row: tap 96 + 10 o - kap */
        memset(image, 0, B200_TC_B_BYTES);
        for (int s = 0; s < 3; ++s)
            for (int j = 0; j <= B200_TC_OPR; ++j)
                for (int comp = 0; comp < 2; ++comp) {
                    const int n = B200_TC_COL(s, j, comp), o = j - 1;
                    for (int kap = 0; kap < B200_TC_K_BYTES / 2; ++kap) {
                        const int t = B200_TC_HIST_SAMPLES + 10 * o - kap;
                        if (t < 0 || t >= B200_FM_T1) continue;
                        image[B200_TC_OP_OFF(B200_TC_N, n, 2 * kap + comp)] = (uint8_t)q[s][t];
                    }
                }
    }
    if (q_out) memcpy(q_out, q, sizeof q);
    if (e_out) *e_out = e;
}

/* ---- AM ---- */
struct AmPlan {
    uint32_t n_tiles, total_chunks, tiles_per_segment, segments;
    uint64_t q_count, audio_len;
};
inline AmPlan plan_am_batch(uint64_t len_bytes, uint32_t n_captures, uint32_t sm_count)
{
    AmPlan pl{};
    const uint64_t n = len_bytes / 2;
    pl.q_count = am_y2_len(len_bytes);
    pl.audio_len = am_audio_len(len_bytes);
    pl.total_chunks = (uint32_t)ceil_div(n, B200_AM_CHUNK);
    pl.n_tiles = (uint32_t)ceil_div(pl.total_chunks, B200_AM_THREADS);
    uint64_t want = ceil_div((uint64_t)sm_count * 30, n_captures ? n_captures : 1);
    uint64_t tps = want ? ceil_div(pl.n_tiles, want) : pl.n_tiles;
    if (tps < 16) tps = 16;
    if (tps > pl.n_tiles) tps = pl.n_tiles ? pl.n_tiles : 1;
    pl.tiles_per_segment = (uint32_t)tps;
    pl.segments = (uint32_t)ceil_div(pl.n_tiles, tps);
    if (pl.segments == 0) pl.segments = 1;
    return pl;
}
inline void fill_am_taps(AmTaps &t)
{
    const std::vector<double> g1 = design_taps(2), g2 = design_taps(3), g3 = design_taps(4);
    for (int k = 0; k < B200_AM_T1; ++k) t.g1[k] = (float)g1[k];
    double total = 0.0, run = 0.0;
    for (int k = 0; k < B200_AM_T1; ++k) { /* see fill_fm_taps */
        t.g1s[k] = (float)std::ldexp((double)t.g1[k], B200_U8RAW_LOG2);
        total += (double)t.g1[k];
    }
    t.bias_half = (float)(-127.5 * total / 2);
    for (int k = 0; k < B200_AM_T1; ++k) {
        run += (double)t.g1[k];
        if (k % 20 == 0 && k / 20 < 4) t.bias_head[k / 20] = (float)(-127.5 * run);
    }
    for (int k = 0; k < B200_AM_T2; ++k) t.g2[k] = (float)g2[k];
    for (int k = 0; k < B200_AM_T3; ++k) t.g3[k] = (float)g3[k];
    const double rho = dcblock_rho(), rho4 = std::pow(rho, B200_AMB_PER);
    t.rho = (float)rho;
    t.rho4 = (float)rho4;
    for (int s = 0; s < 6; ++s) t.rho4_pow[s] = (float)std::pow(rho4, double(1 << s));
    for (int i = 0; i < B200_AMB_PER; ++i) t.rho_i[i] = (float)std::pow(rho, i + 1);
}

inline void fill_twiddles(float2 *tw1024)
{
    for (int m = 0; m < 1024; ++m) {
        const double a = -2.0 * kPi * m / 1024.0;
        tw1024[m].x = (float)std::cos(a);
        tw1024[m].y = (float)std::sin(a);
    }
}

} // namespace b200
#endif
