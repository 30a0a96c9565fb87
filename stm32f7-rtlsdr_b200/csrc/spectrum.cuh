/*
 * spectrum.cuh -- kernel K3: u8 I/Q -> window -> 1024-point FFT -> |X|^2 -> averaged spectrum,
 * fused, one pass over the input bytes.
 *
 * Reference anchor: this is the consumer of `CommItf.buff` the firmware never wrote
 * (README.md:31-32 "next task"; the commented poll at src/main.c:76-79); the intended MCU shape
 * is arm_cfft_f32(1024) + arm_cmplx_mag_squared_f32 (CMSIS/core/arm_math.h:2149, :4693).
 * Definition followed: oracle/golden.c gold_spectrum().
 *
 * Decomposition: 1024 = 32 x 32 "four-step" FFT, ONE WARP PER FRAME, 32 points per lane:
 *   n = t + 32 j   (t = lane, j = 0..31)       k = k1 + 32 k2
 *   pass 1 (lane t):  Y[k1] = sum_j w[n] x[n] W32^{j k1}      in registers (fft32.cuh)
 *   twiddle:          Y[k1] *= W1024^{t k1}                    folded into pass 2's first stage
 *   transpose:        lane t -> lane k1 through a warp-private 32x34 shared tile
 *   pass 2 (lane k1): X[k1+32 k2] = sum_t Y_t[k1] W32^{t k2}   in registers
 *   power:            acc[k2] += |X|^2                          32 bins per lane, in registers
 * The 32 window values and 32 twiddles a lane needs never change, so they are staged through shared
 * memory once per CTA and then held in registers (250 registers, 2 CTAs of 4 warps per SM): the only
 * shared-memory traffic per frame is the transpose (DESIGN.md 5.1 has the measurements behind these choices).
 * Work unit = (capture, 4 x frames_per_warp consecutive frames).  A warp walks `frames_per_warp`
 * consecutive frames (hop 512) and keeps the 32 x 32 bin sums in registers; the four warps of the unit are
 * then added in a fixed order and one 1024-float partial per UNIT goes to a workspace that
 * k_spectrum_finalize (or the split-capture exchange kernel) sums in a fixed order -> deterministic
 * results, no float atomics.  frames_per_warp follows from the capture LENGTH only (plan.h), so the
 * summation tree of a capture -- hence every bit of its spectrum -- is the same whether the capture is
 * processed alone, in a batch of 512 or in a 4096 / N shard on another GPU.  The grid is persistent
 * (one CTA per resident slot): the per-CTA prologue (constants to registers) is paid once however short
 * the units are.  Units are handed out DYNAMICALLY (CTA b starts with unit b, every further one comes from
 * an atomic counter): the two warps that share a scheduler do not get equal shares of it, so with a static
 * split one CTA of every SM finished early and left the other alone on the SM for the last quarter of the
 * kernel -- 11 % slower than handing out units as CTAs become free (measured, profiles/r2_spectrum_units.txt).
 * Which CTA computes a unit never changes its partial, so results stay deterministic.
 *
 * Input access: lane t reads the 2-byte sample n = t + 32 j straight from global memory
 * (a warp reads 64 contiguous bytes per j; both halves of every 128-byte line are used by
 * consecutive j, the second from L1).  Every input byte is fetched from HBM once per frame
 * pair at most (the 50 % overlap re-read hits L2).
 *
 * Roofline: 2 bytes per new complex sample vs ~2100 fp32 lane-operations per frame (512 new
 * samples) -> this chain is bound by the FP32 pipe, not by HBM (SURVEY.md 7.2-1); the packed
 * FFMA2 formulation keeps the issue slots for loads / PRMT / LDS / STS free.
 */
#ifndef B200_SPECTRUM_CUH
#define B200_SPECTRUM_CUH

#include "fft32.cuh"

#define B200_SPEC_MINB 2 /* CTAs per SM the register allocation is tuned for (8 warps/SM, up to 255 registers): the
                            lane's 32 twiddles and 32 window values stay in registers for the whole kernel */
#define B200_SPEC_WARPS 4
#define B200_SPEC_THREADS (32 * B200_SPEC_WARPS)
#define B200_SPEC_XP 34 /* transpose tile row pitch in complex elements: 64-bit accesses conflict-free.
                           34 (even): rows are 16-byte aligned and are read back with 128-bit loads, also conflict-free */
#define B200_SPEC_WP 36 /* window row pitch in floats */

/* shared memory carve-up (bytes) */
#define B200_SPEC_SMEM_WIN 0
#define B200_SPEC_SMEM_TW (32 * B200_SPEC_WP * 4)
#define B200_SPEC_SMEM_XP (B200_SPEC_SMEM_TW + 32 * 32 * 8)
#define B200_SPEC_SMEM_SCHED (B200_SPEC_SMEM_XP + B200_SPEC_WARPS * 32 * B200_SPEC_XP * 8) /* u32 [4]: [2] next unit, [3] last CTA */
#define B200_SPEC_SMEM_BYTES (B200_SPEC_SMEM_SCHED + 16)

#ifdef B200_EMULATED
#define B200_DYN_SMEM(name) unsigned char *name = EMU_DYN_SMEM
#else
#define B200_DYN_SMEM(name) extern __shared__ __align__(1024) unsigned char name[]
#endif

struct SpectrumParams {
    const uint8_t *iq;        /* capture c starts at iq + c * capture_stride                     */
    uint64_t capture_stride;  /* bytes                                                           */
    uint32_t frames;          /* frames per capture (all captures equal length)                  */
    uint32_t frames_per_warp; /* consecutive frames walked by one warp                           */
    const float *window;      /* 1024 floats                                                     */
    const float2 *twiddle;    /* 1024 entries: e^{-2 pi i m / 1024}                              */
    float *partials;          /* [capture][units_per_capture][1024]                              */
    uint32_t units_per_capture; /* ceil(frames / (4 frames_per_warp))                            */
    uint32_t total_units;     /* n_captures x units_per_capture                                  */
    uint32_t *unit_counter;   /* two words, zero before the first launch: [0] units handed out beyond the first
                                 gridDim.x, [1] CTAs finished (the last one leaves both at zero again)     */
    /* single-capture launches of the streaming path: the LAST CTA to finish also does k_spectrum_finalize's job
     * (same arithmetic, same order), which saves a launch per ring slot.  final_out = null: separate finalize kernel. */
    float *final_out;         /* 1024 floats                                                     */
    const float *carry;       /* optional 1024 floats (may alias final_out)                      */
    float final_scale, carry_scale;
    float ema_log2_decay;     /* log2(1 - beta), EMA only                                        */
    float ema_beta;
};

template <bool EMA>
__global__ void __launch_bounds__(B200_SPEC_THREADS, B200_SPEC_MINB) k_spectrum(SpectrumParams p)
{
    B200_DYN_SMEM(smem);
    float *s_win = reinterpret_cast<float *>(smem + B200_SPEC_SMEM_WIN);
    c2 *s_tw = reinterpret_cast<c2 *>(smem + B200_SPEC_SMEM_TW);
    const int tid = (int)threadIdx.x, lane = tid & 31, warp = tid >> 5;
    c2 *s_xp = reinterpret_cast<c2 *>(smem + B200_SPEC_SMEM_XP) + warp * (32 * B200_SPEC_XP);

    /* stage the window per lane in the order pass 1 consumes it: win[t][2 i + h] = w[t + 32 (e_i + 16 h)]
     * with e_i = bitrev5(2 i) -- the two samples of first-stage butterfly i sit side by side --
     * and the twiddles as pairs (see below) */
    for (int i = tid; i < 1024; i += B200_SPEC_THREADS) {
        int t = i & 31, j = i >> 5;
        {
            const int e = j & 15, h = j >> 4;
            const int bi = b200_bitrev5(e) >> 1; /* butterfly index i with bitrev5(2 i) == e */
            s_win[t * B200_SPEC_WP + 2 * bi + h] = __ldg(p.window + i);
        }
        float2 w = __ldg(p.twiddle + ((t * j) & 1023));
        /* pair layout: [e][lane] = (W^{e lane}, W^{(e+16) lane}), e = 0..15: one 16-byte load feeds a
         * first-stage butterfly of pass 2 (elements e and e+16 of lane's column) */
        s_tw[((j & 15) * 32 + t) * 2 + (j >> 4)] = c2_make(w.x, w.y);
    }
    uint32_t *s_sched = reinterpret_cast<uint32_t *>(smem + B200_SPEC_SMEM_SCHED);
    __syncthreads();

    const float *my_win = s_win + lane * B200_SPEC_WP;
    float4 r_tw[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) r_tw[i] = *reinterpret_cast<const float4 *>(s_tw + (b200_bitrev5(2 * i) * 32 + lane) * 2);
    float4 r_win[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) r_win[i] = *reinterpret_cast<const float4 *>(my_win + 4 * i);

    float *s_red = reinterpret_cast<float *>(smem + B200_SPEC_SMEM_XP); /* [warp][1024], pitch 32*XP*2 floats */
    uint32_t unit_g = blockIdx.x;
    while (unit_g < p.total_units) {
    /* ask for the next unit now; the answer is read after this unit's barriers */
    if (tid == 0) s_sched[2] = gridDim.x + atomicAdd(p.unit_counter, 1u);
    const uint32_t capture = unit_g / p.units_per_capture;
    const uint32_t warp_global = (unit_g - capture * p.units_per_capture) * B200_SPEC_WARPS + (uint32_t)warp;
    const uint32_t m_begin = warp_global * p.frames_per_warp;
    uint32_t m_end = m_begin + p.frames_per_warp;
    if (m_end > p.frames) m_end = p.frames;

    float acc[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) acc[i] = 0.0f;

    const uint8_t *cap = p.iq + (uint64_t)capture * p.capture_stride;
    /* software pipeline: the 32 two-byte loads of frame m+1 are issued before the FFT of frame m,
     * so no warp ever waits on HBM/L2 latency with only two warps per scheduler resident */
    const unsigned short *src0 = reinterpret_cast<const unsigned short *>(cap) + (uint32_t)lane;
    uint32_t raw[32];
    if (m_begin < m_end) {
#pragma unroll
        for (int j = 0; j < 32; ++j) raw[j] = __ldg(src0 + (uint64_t)m_begin * 512u + 32 * j);
    }
    for (uint32_t m = m_begin; m < m_end; ++m) {
        c2 v[32];
        /* convert, window and first DIT stage of pass 1 in one go: butterfly i takes samples
         * e = bitrev5(2 i) and e + 16:  X = a wa + b wb,  Y = a wa - b wb  (3 packed ops) */
#pragma unroll
        for (int i2 = 0; i2 < 8; ++i2) {
            const float4 w4 = r_win[i2];
            const float wv[4] = {w4.x, w4.y, w4.z, w4.w};
#pragma unroll
            for (int ii = 0; ii < 2; ++ii) {
                const int i = 2 * i2 + ii, e = b200_bitrev5(2 * i);
                const c2 pa = c2_scale(c2_from_u8_lo(raw[e]), wv[2 * ii]);
                const c2 b = c2_from_u8_lo(raw[e + 16]);
                v[2 * i] = c2_fma_s(b, wv[2 * ii + 1], pa);
                v[2 * i + 1] = c2_fma_s(b, -wv[2 * ii + 1], pa);
            }
        }
        if (m + 1 < m_end) {
            const unsigned short *src = src0 + (uint64_t)(m + 1) * 512u;
#pragma unroll
            for (int j = 0; j < 32; ++j) raw[j] = __ldg(src + 32 * j);
        }
        b200_stage_k<4, 0>::run(v);
        b200_stage_k<8, 0>::run(v);
        b200_stage_k<16, 0>::run(v);
        b200_stage_k<32, 0>::run(v); /* v[k1] = Y[k1] */
        /* transpose through the warp-private tile: row = k1 (the reader's lane), column = source lane t.
         * The barrier that keeps this frame's stores behind the previous frame's loads sits HERE, a whole
         * pass later than those loads, so it never waits on them. */
        __syncwarp();
#pragma unroll
        for (int k1 = 0; k1 < 32; ++k1) s_xp[k1 * B200_SPEC_XP + lane] = v[k1];
        __syncwarp();
#pragma unroll
#ifdef B200_PACKED
        for (int t = 0; t < 32; t += 2) {
            const float4 q = *reinterpret_cast<const float4 *>(s_xp + lane * B200_SPEC_XP + t);
            v[b200_bitrev5(t)] = c2_make(q.x, q.y);
            v[b200_bitrev5(t + 1)] = c2_make(q.z, q.w);
        }
#else /* host emulation: scalar c2 */
        for (int t = 0; t < 32; ++t) v[b200_bitrev5(t)] = s_xp[lane * B200_SPEC_XP + t];
#endif
        /* first DIT stage of pass 2 with the four-step twiddles folded in: slots (2i, 2i+1) hold the
         * elements e = bitrev5(2i) < 16 and e + 16 of this lane's column; X = Ta a + Tb b, Y = Ta a - Tb b
         * = 2 (Ta a) - X: 5 packed ops instead of 2 + 2 (twiddles) + 2 (butterfly) */
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            const int e = b200_bitrev5(2 * i);
            const float4 tw = r_tw[i];
            const c2 pa = (e == 0) ? v[2 * i] : c2_cmul(v[2 * i], tw.x, tw.y);
            const c2 x = c2_cfma(v[2 * i + 1], tw.z, tw.w, pa);
            v[2 * i + 1] = c2_two_a_minus(pa, x);
            v[2 * i] = x;
        }
        b200_stage_k<4, 0>::run(v);
        b200_stage_k<8, 0>::run(v);
        b200_stage_k<16, 0>::run(v);
        b200_stage_k<32, 0>::run(v); /* v[k2] = X[lane + 32 k2] */
        if (EMA) {
            float wgt = p.ema_beta * exp2f((float)(p.frames - 1u - m) * p.ema_log2_decay);
#pragma unroll
            for (int k2 = 0; k2 < 32; ++k2) acc[k2] = fmaf(c2_norm_acc(v[k2], 0.0f), wgt, acc[k2]);
        } else {
#pragma unroll
            for (int k2 = 0; k2 < 32; ++k2) acc[k2] = c2_norm_acc(v[k2], acc[k2]);
        }
    }

    /* fixed-order reduction over the unit's four warps, then one partial per unit (the reduction buffer
     * aliases the transpose tiles: barriers on both sides) */
    __syncthreads();
    float *mine = s_red + warp * (32 * B200_SPEC_XP * 2);
#pragma unroll
    for (int k2 = 0; k2 < 32; ++k2) mine[k2 * 32 + lane] = acc[k2]; /* bin k = lane + 32 k2 */
    __syncthreads();
    float *out = p.partials + (uint64_t)unit_g * 1024u;
    for (int k = tid; k < 1024; k += B200_SPEC_THREADS) {
        float s = 0.0f;
#pragma unroll
        for (int w = 0; w < B200_SPEC_WARPS; ++w) s += s_red[w * (32 * B200_SPEC_XP * 2) + k];
        out[k] = s;
    }
    if (p.final_out) __threadfence(); /* the partial must be visible to whichever CTA finishes last */
    unit_g = s_sched[2];
    __syncthreads(); /* the reduction buffer and s_sched[2] are free again */
    } /* units */
    /* the last CTA out leaves the hand-out counter at zero for the next launch (atomicInc wraps its own word) ... */
    if (tid == 0) {
        const bool last = atomicInc(p.unit_counter + 1, gridDim.x - 1u) == gridDim.x - 1u;
        if (last) p.unit_counter[0] = 0u;
        s_sched[3] = last ? 1u : 0u;
    }
    /* ... and, for a single capture of the streaming path, adds up the partials: out = scale * sum_i partial_i +
     * carry_scale * carry, units in fixed order -- k_spectrum_finalize without the extra launch */
    if (p.final_out) {
        __syncthreads();
        if (s_sched[3]) {
            __threadfence();
            /* a thread owns the bins 4 tid .. 4 tid + 3 and 512 + 4 tid ..; per bin the units are added in order (the same
             * sum as the separate kernel, bit for bit), with 128-bit loads and eight units at a time in flight -- one CTA
             * does this alone, so it is the latency of the loads that counts */
            static_assert(B200_SPEC_THREADS == 128, "folded finalize: 128 threads x 2 x float4 = 1024 bins");
            float sum[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) sum[j] = 0.0f;
#pragma unroll 8
            for (uint32_t i = 0; i < p.total_units; ++i) {
                const float4 *src = reinterpret_cast<const float4 *>(p.partials + (uint64_t)i * 1024u) + tid;
                const float4 a = __ldcg(src), c = __ldcg(src + 128);
                sum[0] += a.x; sum[1] += a.y; sum[2] += a.z; sum[3] += a.w;
                sum[4] += c.x; sum[5] += c.y; sum[6] += c.z; sum[7] += c.w;
            }
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int k = (j < 4 ? 0 : 512) + 4 * tid + (j & 3);
                float r = sum[j] * p.final_scale;
                if (p.carry) r = fmaf(p.carry[k], p.carry_scale, r);
                p.final_out[k] = r;
            }
        }
    }
}

/* out[c][k] = scale * sum_i partials[c][i][k] + carry_scale * carry[k]  (fixed order) */
__global__ void __launch_bounds__(256) k_spectrum_finalize(const float *partials, uint32_t units_per_capture,
                                                           float scale, const float *carry, float carry_scale,
                                                           float *out)
{
    const uint32_t capture = blockIdx.y;
    const uint32_t k = blockIdx.x * 256u + threadIdx.x;
    const float *src = partials + (uint64_t)capture * units_per_capture * 1024u + k;
    float s = 0.0f;
    for (uint32_t i = 0; i < units_per_capture; ++i) s += src[(uint64_t)i * 1024u];
    float r = s * scale;
    if (carry) r = fmaf(carry[(uint64_t)capture * 1024u + k], carry_scale, r);
    out[(uint64_t)capture * 1024u + k] = r;
}

#endif
