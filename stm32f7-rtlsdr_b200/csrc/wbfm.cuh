/*
 * wbfm.cuh -- kernel K4 (FM): u8 I/Q -> /10 polyphase FIR (80 taps) -> quadrature discriminator
 * -> 75 us de-emphasis -> /5 FIR (50 taps) -> 48 kHz audio, fused: the IQ stream crosses HBM once
 * and nothing but audio is written back.
 *
 * Reference anchor: none of this exists in the firmware (README.md:29-34); the planned MCU shape
 * is arm_fir_decimate_f32 (CMSIS/core/arm_math.h:3307).  The RTL2832's own 32-tap hardware FIR
 * (RTL/Inc/usbh_rtlsdr.h:340-345) runs before the bytes reach us.  Definition followed:
 * oracle/golden.c gold_wbfm().
 *
 * Work split.  grid = (segments, captures).  A CTA of B200_FM_THREADS threads walks the tiles of its segment
 * in order; a tile is THREADS x 200 input samples brought in by one TMA bulk copy into a single buffer that
 * is re-armed as soon as the FIR has consumed it (the other CTAs of the SM overlap the rest).
 * A thread's chunk is 200 samples = 20 stage-1 outputs = exactly 4 audio samples, so every stage is balanced
 * over all threads and the /5 FIR reads its window of e[] with aligned 128-bit loads at a fixed offset.
 *
 * Stage 1 is written "input-partitioned": thread t owns input samples [a, a+200), a = tile + 200 t,
 * turns each byte pair into a pair of floats exactly once -- two PRMTs and no arithmetic: the bytes are read
 * as raw (sub)normal floats u * 2^-133 and the -127.5 offset is carried by the accumulators' start values,
 * cplx2.cuh form C -- and scatters it into the (at most
 * 8) outputs y1[m] = sum_k h[k] x[10 m - k] whose window covers it.  Eight packed accumulators
 * rotate; output i of the chunk (centre a + 10 i) completes at sample 10 i:
 *     i = 0..7   partially complete ("heads", started in the previous thread's chunk)
 *     i = 8..19  complete inside the chunk
 *     i = 20..27 started here, finished by the next thread  ("tails", 8 partial sums)
 * Thread t+1 adds thread t's tails to its heads through shared memory; the last thread's tails
 * are carried to the next tile.  So the FIR needs NO input history at all -- a capture (or a
 * stream) starts with the start-of-stream tails (FmTaps::bias_head), which is exactly x[n<0] = 0 -- and
 * costs exactly 8 packed FMAs per input sample with taps held in registers (40 distinct: the filter is
 * symmetric).
 *
 * The 240 kS/s stages run per tile on the fresh outputs: discriminator (atan2 of
 * y[m] conj(y[m-1])), the de-emphasis recurrence as a fixed-shape scan (thread-serial over 20,
 * warp shuffle scan, cross-warp carry, exact carried state between tiles), then the /5 FIR out
 * of a shared-memory window with 49 samples of history (taps outermost: each tap is fetched once
 * for the thread's four outputs).
 *
 * Segments after the first start one tile early with stores suppressed: that warms the carried
 * state up (de-emphasis pole 0.946^1536 ~ 0).  Segment 0 and the streaming path (`state` != 0)
 * carry exact state.
 */
#ifndef B200_WBFM_CUH
#define B200_WBFM_CUH

#include "cplx2.cuh"
#include "tma.cuh"

#define B200_FM_THREADS 128
#define B200_FM_MINB 3                                     /* CTAs per SM (shared memory: 71 KB per CTA)        */
#define B200_FM_WARPS (B200_FM_THREADS / 32)
#define B200_FM_CHUNK 200                                  /* input samples per thread per tile      */
#define B200_FM_OPT 20                                     /* stage-1 outputs per thread per tile    */
#define B200_FM_TILE_IN (B200_FM_THREADS * B200_FM_CHUNK)  /* 25600 (128 threads)                    */
#define B200_FM_TILE_OUT (B200_FM_THREADS * B200_FM_OPT)   /* 2560                                   */
#define B200_FM_TILE_BYTES (2 * B200_FM_TILE_IN)           /* 51200                                  */
#define B200_FM_T1 80
#define B200_FM_T2 50
#define B200_FM_D2 5
#define B200_FM_HIST (B200_FM_T2 - 1) /* 49 */
#define B200_FM_HPAD 52               /* history slots before the tile's e[] (16-byte aligned)        */
#define B200_FM_TAILP (B200_FM_THREADS + 4) /* pitch (in c2) of one row of the transposed tail exchange */
#define B200_FM_APT 4                 /* consecutive audio samples per thread in stage 2 (= OPT / D2) */

/* shared memory carve-up.  ONE raw buffer: the TMA copy of tile t+1 is issued as soon as the
 * scatter FIR of tile t has consumed it and lands while the 240 kS/s stages run, so four CTAs
 * fit on an SM and hide each other's barriers. */
#define B200_FM_SM_RAW 0
#define B200_FM_SM_TAIL (B200_FM_SM_RAW + B200_FM_TILE_BYTES)                           /* c2 [8][132]      */
#define B200_FM_SM_YLAST (B200_FM_SM_TAIL + 8 * B200_FM_TAILP * 8)                      /* c2 [129]         */
#define B200_FM_SM_E (B200_FM_SM_YLAST + (B200_FM_THREADS + 4) * 8)                     /* float [52+1536+16] */
#define B200_FM_SM_WSUM (B200_FM_SM_E + (B200_FM_HPAD + B200_FM_TILE_OUT + 16) * 4)     /* float [8]        */
#define B200_FM_SM_TAILC (B200_FM_SM_WSUM + 32)                                         /* c2 [2][8]        */
#define B200_FM_SM_YLASTC (B200_FM_SM_TAILC + 2 * 8 * 8)                                /* c2 [2]           */
#define B200_FM_SM_BAR (B200_FM_SM_YLASTC + 16)                                         /* u64 mbarrier, 8 spare */
#define B200_FM_SMEM_BYTES (B200_FM_SM_BAR + 16)

#ifndef B200_DYN_SMEM
#ifdef B200_EMULATED
#define B200_DYN_SMEM(name) unsigned char *name = EMU_DYN_SMEM
#else
#define B200_DYN_SMEM(name) extern __shared__ __align__(1024) unsigned char name[]
#endif
#endif

/* state carried between tiles; in global memory it carries a stream from call to call */
struct FmState {
    float tail[16];  /* 8 packed partial sums                                  */
    float ylast[2];  /* y1[m0-1]                                               */
    float e_last;    /* e[m0-1]                                                */
    float pad;
    float e_hist[52]; /* e[m0-49 .. m0-1] in [0..48]                           */
};

struct FmTaps {
    float h1[B200_FM_T1]; /* stage 1, includes 1/127.5                         */
    float h1s[B200_FM_T1]; /* h1 * 2^133: multiplies the raw-byte floats u * 2^-133 (cplx2.cuh form C) */
    float bias_half;       /* -127.5 sum_k h1[k] / 2: start value of EVERY accumulator (form C).  An output that
                              straddles two threads collects one half in each; one that completes inside a thread
                              gets the second half when it is taken out.  Starting at half the offset keeps the
                              partial sums in [-0.5, 0.5] of full scale instead of [-1, 0]: half the rounding error */
    float bias_head[8];    /* -127.5 sum_{k <= 10 i} h1[k]: carried-in part of outputs 0..7 of a stream, whose
                              own part starts from zero (x[n < 0] = 0; small and exact)                       */
    float h2[B200_FM_T2]; /* stage 2, includes the audio gain                  */
    float apow[32];       /* a^(i+1), i = 0..OPT-1, a = 1 - alpha              */
    float alpha;
    float a12;            /* a^OPT: decay over one thread's chunk              */
    float a12pow[5];      /* (a^OPT)^(2^s), s = 0..4                           */
    float a384;           /* (a^OPT)^32: decay over one warp                   */
};

struct FmParams {
    const uint8_t *iq;       /* capture c at iq + c * capture_stride (16-byte aligned)                 */
    uint64_t capture_stride; /* bytes                                                                  */
    uint64_t capture_bytes;  /* valid bytes per capture (multiple of 16 for the batched path)          */
    uint64_t m1;             /* stage-1 outputs per capture to produce: m < m1                         */
    uint64_t m_base;         /* global index of the first stage-1 output of this launch (streaming)    */
    uint32_t n_tiles;        /* tiles per capture                                                      */
    uint32_t total_chunks;   /* 120-sample chunks per capture (the last tile may be partly filled)     */
    uint32_t tiles_per_segment;
    float *audio;            /* [capture][audio_stride]                                                */
    uint64_t audio_stride;
    uint64_t audio_base;     /* audio index of local p = 0 (streaming FIFO offset)                     */
    float *disc;             /* optional [capture][disc_stride]                                        */
    uint64_t disc_stride;
    const FmState *state;    /* optional [capture]: carried state, read by segment 0 (later segments pre-roll) */
    FmState *state_out;      /* optional [capture]: written by the LAST segment; a different buffer than
                                `state` when the launch has more than one segment (they run concurrently) */
    uint32_t *n_audio_out;   /* optional [capture]: number of audio samples written (streaming)        */
};

/* The scatter FIR runs as a LOOP over blocks of 40 samples (5 x 16 bytes): the taps a sample meets repeat every
 * 10 samples with the output index moved on by one, so one block body serves the whole chunk (6.5 KB of code instead
 * of 32 KB unrolled -- the SM's 32 KB instruction cache is shared by every resident warp, and the unrolled form
 * stalled on instruction fetch more than on anything else, profiles/r2_wbfm.txt).
 * J = sample index in the block; local output i (centre 10 i) takes sample J through tap k = 10 i - J and lives in
 * acc[i & 7]; the outputs completing in the block (J = 0, 10, 20, 30) come out in out[0..3] and their slots restart
 * as local outputs 8..11.  Between blocks the caller swaps the two halves of acc[] (local outputs 4..11 become 0..7). */
#define B200_FM_BLK 40
template <int J>
B200_DEV void b200_fm_scatter(c2 x, c2 acc0, const float (&h)[40], c2 (&acc)[8], c2 (&out)[4])
{
#pragma unroll
    for (int i = (J + 9) / 10; i <= (J + 79) / 10; ++i) {
        const int k = 10 * i - J;
        acc[i & 7] = c2_fma_s(x, h[k < 40 ? k : 79 - k], acc[i & 7]);
    }
    if (J % 10 == 0) {
        out[J / 10] = acc[(J / 10) & 7];
        acc[(J / 10) & 7] = acc0; /* local output J/10 + 8 starts here: zero, or half of the -127.5 offset */
    }
}

template <int Q>
struct b200_fm_words {
    B200_DEVM static void run(const uint4 *raw, c2 acc0, const float (&h)[40], c2 (&acc)[8], c2 (&out)[4])
    {
        const uint4 r = raw[Q];
        b200_fm_scatter<8 * Q + 0>(c2_u8raw_lo(r.x), acc0, h, acc, out);
        b200_fm_scatter<8 * Q + 1>(c2_u8raw_hi(r.x), acc0, h, acc, out);
        b200_fm_scatter<8 * Q + 2>(c2_u8raw_lo(r.y), acc0, h, acc, out);
        b200_fm_scatter<8 * Q + 3>(c2_u8raw_hi(r.y), acc0, h, acc, out);
        b200_fm_scatter<8 * Q + 4>(c2_u8raw_lo(r.z), acc0, h, acc, out);
        b200_fm_scatter<8 * Q + 5>(c2_u8raw_hi(r.z), acc0, h, acc, out);
        b200_fm_scatter<8 * Q + 6>(c2_u8raw_lo(r.w), acc0, h, acc, out);
        b200_fm_scatter<8 * Q + 7>(c2_u8raw_hi(r.w), acc0, h, acc, out);
        b200_fm_words<Q + 1>::run(raw, acc0, h, acc, out);
    }
};
template <>
struct b200_fm_words<B200_FM_BLK / 8> {
    B200_DEVM static void run(const uint4 *, c2, const float (&)[40], c2 (&)[8], c2 (&)[4]) {}
};

#ifdef B200_EMULATED
static FmTaps c_fm_taps;
#else
__constant__ FmTaps c_fm_taps;
#endif

B200_DEV float b200_rcp_fast(float x)
{
#ifdef B200_PACKED
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
#else
    return 1.0f / x;
#endif
}

/* atan2(y, x), branch-free, ~1.3e-7 rad: one MUFU.RCP, a degree-15 odd minimax polynomial on
 * [0, 1] (fitted offline against float64 atan), then octant fix-ups.  atan2(0, 0) = 0. */
B200_DEV float b200_atan2(float y, float x)
{
    const float ax = fabsf(x), ay = fabsf(y);
    const float mx = fmaxf(fmaxf(ax, ay), 1e-30f), mn = fminf(ax, ay);
    const float a = mn * b200_rcp_fast(mx); /* MUFU.RCP, ~1 ulp; the IEEE-exact __frcp_rn costs a call */
    const float s = a * a;
    float p = -4.054550054e-03f;
    p = fmaf(p, s, 2.186289528e-02f);
    p = fmaf(p, s, -5.591223568e-02f);
    p = fmaf(p, s, 9.642190620e-02f);
    p = fmaf(p, s, -1.390862694e-01f);
    p = fmaf(p, s, 1.994656515e-01f);
    p = fmaf(p, s, -3.332986075e-01f);
    p = fmaf(p, s, 9.999993356e-01f);
    float r = p * a;
    if (ay > ax) r = 1.57079632679489662f - r;
    if (x < 0.0f) r = 3.14159265358979324f - r;
    return copysignf(r, y);
}

__global__ void __launch_bounds__(B200_FM_THREADS, B200_FM_MINB) k_wbfm(FmParams p)
{
    const FmTaps *taps = &c_fm_taps;
    B200_DYN_SMEM(smem);
    c2 *s_tail = reinterpret_cast<c2 *>(smem + B200_FM_SM_TAIL);
    c2 *s_ylast = reinterpret_cast<c2 *>(smem + B200_FM_SM_YLAST);
    float *s_e = reinterpret_cast<float *>(smem + B200_FM_SM_E);
    float *s_wsum = reinterpret_cast<float *>(smem + B200_FM_SM_WSUM);
    c2 *s_tailc = reinterpret_cast<c2 *>(smem + B200_FM_SM_TAILC);
    c2 *s_ylastc = reinterpret_cast<c2 *>(smem + B200_FM_SM_YLASTC);
    uint64_t *s_bar = reinterpret_cast<uint64_t *>(smem + B200_FM_SM_BAR);

    const int tid = (int)threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t capture = blockIdx.y;
    const uint32_t seg = blockIdx.x;

    /* tiles of this segment; segments > 0 pre-roll one tile with stores suppressed */
    uint32_t t_begin = seg * p.tiles_per_segment;
    uint32_t t_end = t_begin + p.tiles_per_segment;
    if (t_end > p.n_tiles) t_end = p.n_tiles;
    const uint32_t t_first_store = t_begin;
    if (seg > 0) t_begin -= 1;
    const uint32_t my_tiles = t_end > t_begin ? t_end - t_begin : 0;

    const uint8_t *cap = p.iq + (uint64_t)capture * p.capture_stride;

    /* taps and scan constants -> registers */
    float h[40];
#pragma unroll
    for (int k = 0; k < 40; ++k) h[k] = taps->h1s[k];
    const c2 acc0 = c2_make(taps->bias_half, taps->bias_half);
    const float alpha = taps->alpha;
    const float a1 = 1.0f - alpha;
    float lane_pow = 1.0f; /* (a^OPT)^lane */
    for (int i = 0; i < lane; ++i) lane_pow *= taps->a12;

    /* carried state: segment 0 continues the stream exactly; later segments start from zero one tile
     * early (FIR memory is 80 samples, the de-emphasis pole decays to nothing over a tile) */
    const FmState *st_in = (p.state && seg == 0) ? p.state + capture : nullptr;
    if (tid < 8) {
        float tr = 0.0f, ti = 0.0f;
        if (st_in) { tr = st_in->tail[2 * tid]; ti = st_in->tail[2 * tid + 1]; }
        /* first outputs of a capture / stream: x[n < 0] = 0 */
        if (seg == 0 && p.m_base == 0) tr = ti = taps->bias_head[tid];
        s_tailc[8 + tid] = c2_make(tr, ti); /* tile 0 reads carry buffer 1 */
    }
    if (tid == 8) {
        float yr = 0.0f, yi = 0.0f;
        if (st_in) { yr = st_in->ylast[0]; yi = st_in->ylast[1]; }
        s_ylastc[1] = c2_make(yr, yi);
    }
    if (tid == 9) s_wsum[4] = st_in ? st_in->e_last : 0.0f; /* tile carry e[m0-1] */
    for (int i = tid; i < B200_FM_HIST; i += B200_FM_THREADS)
        s_e[B200_FM_HPAD - B200_FM_HIST + i] = st_in ? st_in->e_hist[i] : 0.0f;

    auto issue_tile = [&](uint32_t it) { /* thread 0 only */
        const uint32_t tile = t_begin + it;
        const uint64_t off = (uint64_t)tile * B200_FM_TILE_BYTES;
        uint64_t bytes = p.capture_bytes > off ? p.capture_bytes - off : 0;
        if (bytes > B200_FM_TILE_BYTES) bytes = B200_FM_TILE_BYTES;
        bytes &= ~(uint64_t)15;
        b200_mbar_expect_tx(s_bar, (uint32_t)bytes);
        if (bytes) b200_tma_load_1d(smem + B200_FM_SM_RAW, cap + off, (uint32_t)bytes, s_bar);
    };
    if (tid == 0) {
        b200_mbar_init(s_bar, 1);
        b200_mbar_fence_init();
        if (my_tiles > 0) issue_tile(0);
    }
    __syncthreads();

    for (uint32_t it = 0; it < my_tiles; ++it) {
        const uint32_t tile = t_begin + it;
        const bool store = tile >= t_first_store;
        const uint64_t m0 = (uint64_t)tile * B200_FM_TILE_OUT; /* first stage-1 output of the tile (local index) */
        /* last thread of the tile holding a whole chunk: it owns the carries to the next tile */
        int last = (int)(p.total_chunks - tile * B200_FM_THREADS) - 1;
        if (last > B200_FM_THREADS - 1) last = B200_FM_THREADS - 1;
        const int par = (int)(it & 1);

        /* ---- stage 1: scatter FIR over this thread's 200 samples ---- */
        b200_mbar_wait(s_bar, it & 1);
        c2 acc[8], head[B200_FM_OPT];
        /* the very first chunk of a capture / stream: its outputs 0..7 are the filter's rise from nothing
         * (|y[0]| ~ 1e-6 of full scale) and are kept exact -- own part from zero, carried-in part = the small
         * exact offset of the taps that reach n >= 0 (bias_head) -- instead of two halves of O(0.5) */
        const c2 start = (tid == 0 && it == 0 && seg == 0 && p.m_base == 0) ? c2_zero() : acc0;
#pragma unroll
        for (int i = 0; i < 8; ++i) acc[i] = start;
        unsigned char *my_raw = smem + B200_FM_SM_RAW + tid * (2 * B200_FM_CHUNK);
        /* the 4 outputs a block completes are parked in the part of this thread's OWN raw bytes it has already
         * consumed (32 bytes of results per 80 bytes of input; no other thread ever reads these bytes) and come
         * back into registers after the FIR: that keeps the block body free of chunk-position-dependent code */
        c2 *park = reinterpret_cast<c2 *>(my_raw);
#pragma unroll 1
        for (int blk = 0; blk < B200_FM_CHUNK / B200_FM_BLK; ++blk) {
            c2 out[4];
            b200_fm_words<0>::run(reinterpret_cast<const uint4 *>(my_raw) + blk * (B200_FM_BLK / 8), acc0, h, acc, out);
            /* outputs 8.. of the chunk (blocks 2..) lived in this thread only: they hold one half of the offset, add
             * the other; outputs 0..7 get theirs from the previous thread's tails */
            const c2 fix = blk >= 2 ? acc0 : c2_zero();
#pragma unroll
            for (int q = 0; q < 4; ++q) out[q] = c2_add(out[q], fix);
#pragma unroll
            for (int q = 0; q < 4; ++q) park[4 * blk + q] = out[q];
            /* local outputs 4..11 of this block are 0..7 of the next */
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const c2 t = acc[q];
                acc[q] = acc[q + 4];
                acc[q + 4] = t;
            }
        }
#pragma unroll
        for (int i = 0; i < B200_FM_OPT; ++i) head[i] = park[i];
        /* tails: outputs OPT..OPT+7 are acc[0..7] after the last swap -> next thread's heads 0..7.
         * exchange tile is [i][thread] so a warp's stores / loads are contiguous */
        if (tid == last) {
#pragma unroll
            for (int i = 0; i < 8; ++i) s_tailc[par * 8 + i] = acc[i];
        } else {
#pragma unroll
            for (int i = 0; i < 8; ++i) s_tail[i * B200_FM_TAILP + tid + 1] = acc[i];
        }
        __syncthreads(); /* S1: raw buffer consumed, tails visible */
        if (tid == 0 && it + 1 < my_tiles) issue_tile(it + 1);
        if (tid == 0) {
#pragma unroll
            for (int i = 0; i < 8; ++i) head[i] = c2_add(head[i], s_tailc[(par ^ 1) * 8 + i]);
        } else {
#pragma unroll
            for (int i = 0; i < 8; ++i) head[i] = c2_add(head[i], s_tail[i * B200_FM_TAILP + tid]);
        }
        if (tid == last) s_ylastc[par] = head[B200_FM_OPT - 1];
        else s_ylast[tid + 1] = head[B200_FM_OPT - 1];
        __syncthreads(); /* S2 */

        /* ---- discriminator + thread-serial de-emphasis ---- */
        float e[B200_FM_OPT];
        {
            float pr, pi;
            c2_get(tid == 0 ? s_ylastc[par ^ 1] : s_ylast[tid], pr, pi);
            float d[B200_FM_OPT];
#pragma unroll
            for (int i = 0; i < B200_FM_OPT; ++i) {
                float yr, yi;
                c2_get(head[i], yr, yi);
                float zr = fmaf(yr, pr, yi * pi);
                float zi = fmaf(yi, pr, -(yr * pi));
                d[i] = b200_atan2(zi, zr);
                pr = yr;
                pi = yi;
            }
            if (p.m_base + m0 == 0 && tid == 0) d[0] = 0.0f; /* y1[-1] = 0: defined as d[0] = 0 */
            if (p.disc && store) {
                const uint64_t m = m0 + (uint64_t)tid * B200_FM_OPT;
                float *dst = p.disc + (uint64_t)capture * p.disc_stride + m;
                const int n_valid = p.m1 > m ? (p.m1 - m > B200_FM_OPT ? B200_FM_OPT : (int)(p.m1 - m)) : 0;
#pragma unroll
                for (int i = 0; i < B200_FM_OPT; ++i)
                    if (i < n_valid) dst[i] = d[i];
            }
            float run = 0.0f;
#pragma unroll
            for (int i = 0; i < B200_FM_OPT; ++i) {
                run = fmaf(a1, run, alpha * d[i]);
                e[i] = run;
            }
        }
        /* warp scan of the chunk totals: v_l = sum_{l'<=l} (a^OPT)^(l-l') E_l' */
        float v = e[B200_FM_OPT - 1];
#pragma unroll
        for (int s = 0; s < 5; ++s) {
            float u = __shfl_up_sync(0xffffffffu, v, 1u << s);
            if (lane >= (1 << s)) v = fmaf(taps->a12pow[s], u, v);
        }
        float vprev = __shfl_up_sync(0xffffffffu, v, 1u);
        if (lane == 0) vprev = 0.0f;
        if (lane == 31) s_wsum[warp] = v;
        __syncthreads(); /* S3 */
        {
            float cw = s_wsum[4]; /* carry into warp 0 = e[m0-1] */
            for (int w = 0; w < warp; ++w) cw = fmaf(taps->a384, cw, s_wsum[w]);
            const float cin = fmaf(lane_pow, cw, vprev); /* e just before this thread's chunk */
#pragma unroll
            for (int i = 0; i < B200_FM_OPT; ++i) e[i] = fmaf(taps->apow[i], cin, e[i]);
            float4 *dst = reinterpret_cast<float4 *>(s_e + B200_FM_HPAD + tid * B200_FM_OPT);
#pragma unroll
            for (int q = 0; q < B200_FM_OPT / 4; ++q) dst[q] = make_float4(e[4 * q], e[4 * q + 1], e[4 * q + 2], e[4 * q + 3]);
        }
        __syncthreads(); /* S4 */

        /* ---- stage 2: audio[p] = sum_k h2[k] e[5 p - k].  A tile starts at a multiple of 20 stage-1 outputs
         * (chunks are whole), so thread t owns exactly the four audio samples p = pg_first + 4 t + r whose
         * newest input is its own e[5 r]: the 65-float window e[20 t - 49 .. 20 t + 15] sits at the FIXED
         * offset 3 behind the 16-byte aligned address s_e + 20 t (HPAD - HIST = 3) and is read with 17
         * 128-bit loads; the taps run outermost, so each is fetched once for the four outputs ---- */
        {
            const uint64_t mg0 = p.m_base + m0; /* global stage-1 index of tile start: a multiple of 20 */
            uint64_t mg_end = mg0 + (uint64_t)(last + 1) * B200_FM_OPT;
            if (mg_end > p.m_base + p.m1) mg_end = p.m_base + p.m1;
            const uint64_t pg_first = mg0 / B200_FM_D2;
            const uint64_t pg_end = (mg_end + B200_FM_D2 - 1) / B200_FM_D2;
            const uint64_t pg0 = pg_first + (uint64_t)tid * B200_FM_APT;
            if (pg0 < pg_end) {
                constexpr int WOFF = B200_FM_HPAD - B200_FM_HIST; /* 3 */
                constexpr int NW4 = (WOFF + B200_FM_T2 + B200_FM_D2 * (B200_FM_APT - 1) + 3) / 4; /* 17 */
                const float4 *win = reinterpret_cast<const float4 *>(s_e + tid * B200_FM_OPT);
                float ew[4 * NW4];
#pragma unroll
                for (int j = 0; j < NW4; ++j) {
                    const float4 q = win[j];
                    ew[4 * j] = q.x; ew[4 * j + 1] = q.y; ew[4 * j + 2] = q.z; ew[4 * j + 3] = q.w;
                }
                float au[B200_FM_APT];
#pragma unroll
                for (int r = 0; r < B200_FM_APT; ++r) au[r] = 0.0f;
#pragma unroll
                for (int k = 0; k < B200_FM_T2; ++k) {
                    const float hk = taps->h2[k];
#pragma unroll
                    for (int r = 0; r < B200_FM_APT; ++r) au[r] = fmaf(hk, ew[WOFF + B200_FM_HIST + B200_FM_D2 * r - k], au[r]);
                }
                if (store) {
                    float *dst = p.audio + (uint64_t)capture * p.audio_stride + (pg0 - p.audio_base);
#pragma unroll
                    for (int r = 0; r < B200_FM_APT; ++r)
                        if (pg0 + r < pg_end) dst[r] = au[r];
                }
            }
        }
        __syncthreads(); /* S5 */
        /* e carries for the next tile (tails / ylast travel through the parity buffers) */
        if (tid == 9) s_wsum[4] = s_e[B200_FM_HPAD + (last + 1) * B200_FM_OPT - 1];
        float hv[(B200_FM_HIST + B200_FM_THREADS - 1) / B200_FM_THREADS];
#pragma unroll
        for (int q = 0; q < (B200_FM_HIST + B200_FM_THREADS - 1) / B200_FM_THREADS; ++q) {
            const int i = tid + q * B200_FM_THREADS;
            hv[q] = i < B200_FM_HIST ? s_e[B200_FM_HPAD + (last + 1) * B200_FM_OPT - B200_FM_HIST + i] : 0.0f;
        }
        __syncthreads(); /* S6: history source read before it is overwritten (partial tiles overlap) */
#pragma unroll
        for (int q = 0; q < (B200_FM_HIST + B200_FM_THREADS - 1) / B200_FM_THREADS; ++q) {
            const int i = tid + q * B200_FM_THREADS;
            if (i < B200_FM_HIST) s_e[B200_FM_HPAD - B200_FM_HIST + i] = hv[q];
        }
        /* the next tile's S1..S3 order these writes before their readers */
    }

    if (p.state_out && seg + 1 == gridDim.x) {
        FmState *st_out = p.state_out + capture;
        __syncthreads();
        const int fin = my_tiles ? (int)((my_tiles - 1) & 1) : 1; /* carry buffer written last */
        if (tid < 8) {
            float tr, ti;
            c2_get(s_tailc[fin * 8 + tid], tr, ti);
            st_out->tail[2 * tid] = tr;
            st_out->tail[2 * tid + 1] = ti;
        }
        if (tid == 8) {
            float yr, yi;
            c2_get(s_ylastc[fin], yr, yi);
            st_out->ylast[0] = yr;
            st_out->ylast[1] = yi;
        }
        if (tid == 9) st_out->e_last = s_wsum[4];
        for (int i = tid; i < B200_FM_HIST; i += B200_FM_THREADS)
            st_out->e_hist[i] = s_e[B200_FM_HPAD - B200_FM_HIST + i];
    }
}

#endif
