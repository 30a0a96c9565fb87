/*
 * am.cuh -- kernel K4 (AM): u8 I/Q -> /20 FIR (80 taps) -> /10 FIR (120 taps) -> envelope |y|
 * (k_am_front, one pass over the IQ bytes, writes 4 bytes per 200 input samples), then
 * DC block -> x2 / /3 polyphase resampler -> 8 kHz audio (k_am_back, 12 kS/s, tiny).
 *
 * Reference anchor: planned work only (README.md:29-34; arm_fir_decimate_f32,
 * CMSIS/core/arm_math.h:3307).  Definition followed: oracle/golden.c gold_am().
 *
 * k_am_front uses the same input-partitioned scatter FIR as wbfm.cuh.  A thread owns 200 input
 * samples = 10 stage-1 outputs = exactly ONE stage-2 output, so both stages are perfectly
 * balanced over the CTA:
 *     stage 1: each sample feeds the 4 outputs y1[m] = sum g1[k] x[20 m - k] covering it
 *              (4 rotating packed accumulators; outputs 0..3 need the previous thread's 4
 *              tails, 4..9 complete in-chunk, 10..13 are this thread's tails)
 *     stage 2: y2[q] = sum_{k<120} g2[k] y1[10 q - k], also in scatter form: the thread's ten y1
 *              values (registers) feed 13 outputs; partial sums meet in a shared exchange tile
 *     envelope r[q] = |y2[q]|
 * Only FIRs are involved, so segments that start one tile early reproduce the single-segment
 * result bit for bit.  The DC blocker has a pole at 0.999 (memory ~ 1 s) and therefore runs in
 * k_am_back as an exact scan over the whole capture, one CTA per capture.
 */
#ifndef B200_AM_CUH
#define B200_AM_CUH

#include "cplx2.cuh"
#include "tma.cuh"

#define B200_AM_THREADS 128
#define B200_AM_CHUNK 200                                 /* input samples per thread per tile   */
#define B200_AM_OPT 10                                    /* stage-1 outputs per thread per tile */
#define B200_AM_TILE_IN (B200_AM_THREADS * B200_AM_CHUNK) /* 25600                               */
#define B200_AM_TILE_Y1 (B200_AM_THREADS * B200_AM_OPT)   /* 1280                                */
#define B200_AM_TILE_BYTES (2 * B200_AM_TILE_IN)          /* 51200                               */
#define B200_AM_T1 80
#define B200_AM_T2 120
#define B200_AM_HIST (B200_AM_T2 - 1) /* 119 */
#define B200_AM_T3 48
#define B200_AM_BHIST 24 /* b[] history needed by the resampler */

#define B200_AM_NP 13                       /* a stage-1 chunk (10 outputs) reaches 13 stage-2 outputs */
#define B200_AM_PP (B200_AM_THREADS + 12)   /* slots per row of the partial-sum exchange            */

#define B200_AM_SM_RAW 0
#define B200_AM_SM_TAIL (B200_AM_SM_RAW + B200_AM_TILE_BYTES)                    /* c2 [4][132]       */
#define B200_AM_SM_PART (B200_AM_SM_TAIL + 4 * 132 * 8)                          /* c2 [13][140]      */
#define B200_AM_SM_CARRY (B200_AM_SM_PART + B200_AM_NP * B200_AM_PP * 8)         /* c2 [13][12]       */
#define B200_AM_SM_TAILC (B200_AM_SM_CARRY + B200_AM_NP * 12 * 8)                /* c2 [2][4]         */
#define B200_AM_SM_BAR (B200_AM_SM_TAILC + 2 * 4 * 8)
#define B200_AM_SMEM_BYTES (B200_AM_SM_BAR + 16)

#ifndef B200_DYN_SMEM
#ifdef B200_EMULATED
#define B200_DYN_SMEM(name) unsigned char *name = EMU_DYN_SMEM
#else
#define B200_DYN_SMEM(name) extern __shared__ __align__(1024) unsigned char name[]
#endif
#endif

struct AmFrontState {
    float tail[8];                          /* stage 1: 4 packed partial sums carried to the next chunk */
    float part[2 * B200_AM_NP * 12];        /* stage 2: partial sums of the next 12 outputs, [d][j]      */
};
struct AmBackState {
    float r_last, b_last;
    float b_hist[B200_AM_BHIST]; /* b[q0-24 .. q0-1] */
};

struct AmTaps {
    float g1[B200_AM_T1];
    float g1s[B200_AM_T1]; /* g1 * 2^133 (cplx2.cuh form C) */
    float bias_half;       /* -127.5 sum_k g1[k] / 2 (FmTaps::bias_half)            */
    float bias_head[4];    /* -127.5 sum_{k <= 20 i} g1[k] (FmTaps::bias_head)       */
    float g2[B200_AM_T2];
    float g3[B200_AM_T3];
    float rho;
    float rho4;           /* rho^PER: one thread of k_am_back */
    float rho4_pow[6];    /* (rho^PER)^(2^s) */
    float rho_i[16];      /* rho^(i+1), i = 0..PER-1 (PER = B200_AMB_PER <= 16) */
};

#ifdef B200_EMULATED
static AmTaps c_am_taps;
#else
__constant__ AmTaps c_am_taps;
#endif

struct AmFrontParams {
    const uint8_t *iq;
    uint64_t capture_stride, capture_bytes;
    uint64_t q_count;     /* envelope samples to produce per capture: q < q_count                  */
    uint64_t q_base;      /* global index of the first envelope sample of this launch (streaming)  */
    uint32_t n_tiles, total_chunks, tiles_per_segment;
    float *env;           /* [capture][env_stride] r[q]                                          */
    uint64_t env_stride;
    const AmFrontState *state; /* optional (streaming): carried state, read by segment 0            */
    AmFrontState *state_out;   /* optional: written by the LAST segment (another buffer than `state`
                                  when the launch has several segments: they run concurrently)      */
};

template <int J>
B200_DEV void b200_am_scatter(c2 x, c2 acc0, const float (&g)[40], c2 (&acc)[4], c2 (&head)[B200_AM_OPT])
{
#pragma unroll
    for (int i = (J + 19) / 20; i <= (J + 79) / 20; ++i) {
        const int k = 20 * i - J;
        acc[i & 3] = c2_fma_s(x, g[k < 40 ? k : 79 - k], acc[i & 3]);
    }
    if (J % 20 == 0 && J / 20 < B200_AM_OPT) {
        head[J / 20] = (J / 20 >= 4) ? c2_add(acc[(J / 20) & 3], acc0) : acc[(J / 20) & 3]; /* see wbfm.cuh */
        acc[(J / 20) & 3] = acc0; /* output J/20 + 4 starts here */
    }
}
template <int Q>
struct b200_am_words {
    B200_DEVM static void run(const uint4 *raw, c2 acc0, const float (&g)[40], c2 (&acc)[4], c2 (&head)[B200_AM_OPT])
    {
        const uint4 r = raw[Q];
        b200_am_scatter<8 * Q + 0>(c2_u8raw_lo(r.x), acc0, g, acc, head);
        b200_am_scatter<8 * Q + 1>(c2_u8raw_hi(r.x), acc0, g, acc, head);
        b200_am_scatter<8 * Q + 2>(c2_u8raw_lo(r.y), acc0, g, acc, head);
        b200_am_scatter<8 * Q + 3>(c2_u8raw_hi(r.y), acc0, g, acc, head);
        b200_am_scatter<8 * Q + 4>(c2_u8raw_lo(r.z), acc0, g, acc, head);
        b200_am_scatter<8 * Q + 5>(c2_u8raw_hi(r.z), acc0, g, acc, head);
        b200_am_scatter<8 * Q + 6>(c2_u8raw_lo(r.w), acc0, g, acc, head);
        b200_am_scatter<8 * Q + 7>(c2_u8raw_hi(r.w), acc0, g, acc, head);
        b200_am_words<Q + 1>::run(raw, acc0, g, acc, head);
    }
};
template <>
struct b200_am_words<B200_AM_CHUNK / 8> {
    B200_DEVM static void run(const uint4 *, c2, const float (&)[40], c2 (&)[4], c2 (&)[B200_AM_OPT]) {}
};

__global__ void __launch_bounds__(B200_AM_THREADS, 3) k_am_front(AmFrontParams p)
{
    const AmTaps *taps = &c_am_taps;
    B200_DYN_SMEM(smem);
    c2 *s_tail = reinterpret_cast<c2 *>(smem + B200_AM_SM_TAIL);
    c2 *s_part = reinterpret_cast<c2 *>(smem + B200_AM_SM_PART);
    c2 *s_carry = reinterpret_cast<c2 *>(smem + B200_AM_SM_CARRY);
    c2 *s_tailc = reinterpret_cast<c2 *>(smem + B200_AM_SM_TAILC);
    uint64_t *s_bar = reinterpret_cast<uint64_t *>(smem + B200_AM_SM_BAR);

    const int tid = (int)threadIdx.x;
    const uint32_t capture = blockIdx.y, seg = blockIdx.x;
    uint32_t t_begin = seg * p.tiles_per_segment;
    uint32_t t_end = t_begin + p.tiles_per_segment;
    if (t_end > p.n_tiles) t_end = p.n_tiles;
    const uint32_t t_first_store = t_begin;
    if (seg > 0) t_begin -= 1;
    const uint32_t my_tiles = t_end > t_begin ? t_end - t_begin : 0;
    const uint8_t *cap = p.iq + (uint64_t)capture * p.capture_stride;

    float g[40];
#pragma unroll
    for (int k = 0; k < 40; ++k) g[k] = taps->g1s[k];
    const c2 acc0 = c2_make(taps->bias_half, taps->bias_half);

    /* segment 0 continues the stream exactly; later segments rebuild the FIR state from one pre-roll tile */
    const AmFrontState *st_in = (p.state && seg == 0) ? p.state + capture : nullptr;
    if (tid < 4) {
        float tr = 0.0f, ti = 0.0f;
        if (st_in) { tr = st_in->tail[2 * tid]; ti = st_in->tail[2 * tid + 1]; }
        if (seg == 0 && p.q_base == 0) tr = ti = taps->bias_head[tid]; /* first outputs of a capture / stream */
        s_tailc[4 + tid] = c2_make(tr, ti);
    }
    for (int i = tid; i < B200_AM_NP * 12; i += B200_AM_THREADS) {
        float yr = 0.0f, yi = 0.0f;
        if (st_in) { yr = st_in->part[2 * i]; yi = st_in->part[2 * i + 1]; }
        s_carry[i] = c2_make(yr, yi);
    }

    auto issue_tile = [&](uint32_t it) { /* thread 0 only; single raw buffer */
        const uint32_t tile = t_begin + it;
        const uint64_t off = (uint64_t)tile * B200_AM_TILE_BYTES;
        uint64_t bytes = p.capture_bytes > off ? p.capture_bytes - off : 0;
        if (bytes > B200_AM_TILE_BYTES) bytes = B200_AM_TILE_BYTES;
        bytes &= ~(uint64_t)15;
        b200_mbar_expect_tx(s_bar, (uint32_t)bytes);
        if (bytes) b200_tma_load_1d(smem + B200_AM_SM_RAW, cap + off, (uint32_t)bytes, s_bar);
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
        int last = (int)(p.total_chunks - tile * B200_AM_THREADS) - 1;
        if (last > B200_AM_THREADS - 1) last = B200_AM_THREADS - 1;
        const int par = (int)(it & 1);

        b200_mbar_wait(s_bar, it & 1);
        c2 acc[4], head[B200_AM_OPT];
        const c2 start = (tid == 0 && it == 0 && seg == 0 && p.q_base == 0) ? c2_zero() : acc0; /* wbfm.cuh */
#pragma unroll
        for (int i = 0; i < 4; ++i) acc[i] = start;
        const uint4 *raw = reinterpret_cast<const uint4 *>(smem + B200_AM_SM_RAW + tid * (2 * B200_AM_CHUNK));
        b200_am_words<0>::run(raw, acc0, g, acc, head);
        if (tid == last) {
#pragma unroll
            for (int i = 10; i < 14; ++i) s_tailc[par * 4 + (i - 10)] = acc[i & 3];
        } else {
#pragma unroll
            for (int i = 10; i < 14; ++i) s_tail[(i - 10) * 132 + tid + 1] = acc[i & 3];
        }
        __syncthreads(); /* S1: raw consumed, tails visible */
        if (tid == 0 && it + 1 < my_tiles) issue_tile(it + 1);
        if (tid == 0) {
#pragma unroll
            for (int i = 0; i < 4; ++i) head[i] = c2_add(head[i], s_tailc[(par ^ 1) * 4 + i]);
        } else {
#pragma unroll
            for (int i = 0; i < 4; ++i) head[i] = c2_add(head[i], s_tail[i * 132 + tid]);
        }

        /* stage 2, scatter form again: this thread's ten y1 values (registers) feed the 13 outputs
         * y2[t + d] = sum_k g2[k] y1[10 (t + d) - k], d = 0..12, with tap k = 10 d - i for value i.
         * 120 packed FMAs per thread, no shared-memory reads of the inputs; the 13 partial sums go to
         * row d, slot t + d of the exchange tile, output q then adds column q. */
        {
            c2 part[B200_AM_NP];
#pragma unroll
            for (int d = 0; d < B200_AM_NP; ++d) {
                c2 a = c2_zero();
#pragma unroll
                for (int i = 0; i < B200_AM_OPT; ++i) {
                    const int k = 10 * d - i;
                    if (k >= 0 && k < B200_AM_T2) a = c2_fma_s(head[i], taps->g2[k], a);
                }
                part[d] = a;
            }
#pragma unroll
            for (int d = 0; d < B200_AM_NP; ++d) s_part[d * B200_AM_PP + tid + d] = part[d];
        }
        __syncthreads(); /* S2: partial sums of the tile visible */
        {
            /* column tid: rows d <= tid come from this tile, rows d > tid from the carried partials */
            c2 y = c2_zero();
#pragma unroll
            for (int d = 0; d < B200_AM_NP; ++d) {
                const c2 v = (d <= tid) ? s_part[d * B200_AM_PP + tid] : s_carry[d * 12 + tid];
                y = c2_add(y, v);
            }
            float yr, yi;
            c2_get(y, yr, yi);
            const uint64_t q = (uint64_t)tile * B200_AM_THREADS + (uint64_t)tid;
            if (store && q < p.q_count) p.env[(uint64_t)capture * p.env_stride + q] = sqrtf(fmaf(yr, yr, yi * yi));
        }
        __syncthreads(); /* S3: carried partials consumed */
        /* partial sums that belong to the next 12 outputs: slots last+1 .. last+12 of every row */
        c2 nc[2];
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            const int i = tid + r * B200_AM_THREADS;
            nc[r] = c2_zero();
            if (i < B200_AM_NP * 12) {
                const int d = i / 12, j = i - 12 * d;
                const int q = last + 1 + j; /* tile-local index of the output this entry belongs to */
                if (j < d) {
                    if (q - d >= 0) nc[r] = s_part[d * B200_AM_PP + q];   /* written by thread q - d of this tile */
                    else if (q < 12) nc[r] = s_carry[d * 12 + q];          /* short tile: still owed from before */
                }
            }
        }
        __syncthreads(); /* S4: old carry read before it is replaced */
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            const int i = tid + r * B200_AM_THREADS;
            if (i < B200_AM_NP * 12) s_carry[i] = nc[r];
        }
        /* the next tile's S1/S2 order these writes before their readers and before row d is rewritten */
    }

    if (p.state_out && seg + 1 == gridDim.x) {
        AmFrontState *st_out = p.state_out + capture;
        __syncthreads();
        const int fin = my_tiles ? (int)((my_tiles - 1) & 1) : 1;
        if (tid < 4) {
            float tr, ti;
            c2_get(s_tailc[fin * 4 + tid], tr, ti);
            st_out->tail[2 * tid] = tr;
            st_out->tail[2 * tid + 1] = ti;
        }
        for (int i = tid; i < B200_AM_NP * 12; i += B200_AM_THREADS) {
            float yr, yi;
            c2_get(s_carry[i], yr, yi);
            st_out->part[2 * i] = yr;
            st_out->part[2 * i + 1] = yi;
        }
    }
}

/* ---- back end: b[q] = r[q] - r[q-1] + rho b[q-1];  a[s] = sum_k g3[k] v[3 s - k], v[2 q] = b[q] ---- */
#define B200_AMB_THREADS 256
#define B200_AMB_PER 16
#define B200_AMB_TILE (B200_AMB_THREADS * B200_AMB_PER) /* 4096 envelope samples per tile */

struct AmBackParams {
    const float *env;   /* [capture][env_stride]                                   */
    uint64_t env_stride;
    uint64_t q_count;   /* envelope samples in this launch                         */
    uint64_t q_base;    /* global index of local q = 0 (streaming)                 */
    float *audio;       /* [capture][audio_stride]                                 */
    uint64_t audio_stride;
    uint64_t audio_base; /* global audio index of audio[0] (streaming)              */
    AmBackState *state; /* optional                                                */
};

__global__ void __launch_bounds__(B200_AMB_THREADS) k_am_back(AmBackParams p)
{
    const AmTaps *taps = &c_am_taps;
    __shared__ float s_b[B200_AM_BHIST + B200_AMB_TILE];
    __shared__ float s_wsum[8];
    __shared__ float s_carry[2]; /* r_last, b_last */
    const int tid = (int)threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t capture = blockIdx.x;
    const float *env = p.env + (uint64_t)capture * p.env_stride;

    if (tid < B200_AM_BHIST) s_b[tid] = p.state ? p.state[capture].b_hist[tid] : 0.0f;
    if (tid == 32) s_carry[0] = p.state ? p.state[capture].r_last : 0.0f;
    if (tid == 33) s_carry[1] = p.state ? p.state[capture].b_last : 0.0f;
    float lane_pow = 1.0f; /* (rho^4)^lane */
    for (int i = 0; i < lane; ++i) lane_pow *= taps->rho4;
    __syncthreads();

    const uint64_t n_tiles = (p.q_count + B200_AMB_TILE - 1) / B200_AMB_TILE;
    for (uint64_t tile = 0; tile < n_tiles; ++tile) {
        const uint64_t q0 = tile * B200_AMB_TILE + (uint64_t)tid * B200_AMB_PER;
        float r[B200_AMB_PER], b[B200_AMB_PER];
#pragma unroll
        for (int i = 0; i < B200_AMB_PER; ++i) r[i] = (q0 + i < p.q_count) ? env[q0 + i] : 0.0f;
        /* r[q-1] for the first element: previous thread's last, or the carry */
        float rprev = __shfl_up_sync(0xffffffffu, r[B200_AMB_PER - 1], 1u);
        if (lane == 31) s_wsum[warp] = r[B200_AMB_PER - 1]; /* borrow s_wsum to pass r across warps */
        __syncthreads();
        if (lane == 0) rprev = warp == 0 ? s_carry[0] : s_wsum[warp - 1];
        __syncthreads();
        /* thread-serial recurrence from zero state */
        float run = 0.0f;
#pragma unroll
        for (int i = 0; i < B200_AMB_PER; ++i) {
            run = fmaf(taps->rho, run, r[i] - rprev);
            b[i] = run;
            rprev = r[i];
        }
        float v = run;
#pragma unroll
        for (int s = 0; s < 5; ++s) {
            float u = __shfl_up_sync(0xffffffffu, v, 1u << s);
            if (lane >= (1 << s)) v = fmaf(taps->rho4_pow[s], u, v);
        }
        float vprev = __shfl_up_sync(0xffffffffu, v, 1u);
        if (lane == 0) vprev = 0.0f;
        if (lane == 31) s_wsum[warp] = v;
        __syncthreads();
        float cw = s_carry[1];
        for (int w = 0; w < warp; ++w) cw = fmaf(taps->rho4_pow[5], cw, s_wsum[w]);
        const float cin = fmaf(lane_pow, cw, vprev);
#pragma unroll
        for (int i = 0; i < B200_AMB_PER; ++i) {
            b[i] = fmaf(taps->rho_i[i], cin, b[i]);
            s_b[B200_AM_BHIST + tid * B200_AMB_PER + i] = b[i];
        }
        __syncthreads();
        /* resampler: outputs s with 3 s in [2 Q0, 2 Q0 + 2048), Q0 = global q of the tile start */
        {
            const uint64_t Q0 = p.q_base + tile * B200_AMB_TILE;
            uint64_t q_end = p.q_base + p.q_count; /* first invalid global q */
            const uint64_t s_first = (2 * Q0 + 2) / 3;
            for (uint64_t sg = s_first + (uint64_t)tid;; sg += B200_AMB_THREADS) {
                const uint64_t c = 3 * sg; /* position in the zero-stuffed stream */
                if (c >= 2 * Q0 + 2 * B200_AMB_TILE || c >= 2 * q_end) break;
                float a = 0.0f;
                /* taps k with (c - k) even: k = (c & 1), +2, ...; q = (c - k) / 2 */
                const int k0 = (int)(c & 1u);
                const float *bw = s_b + B200_AM_BHIST + (int)((c - (uint64_t)k0) / 2 - Q0);
#pragma unroll
                for (int j = 0; j < B200_AM_T3 / 2; ++j) a = fmaf(taps->g3[k0 + 2 * j], bw[-j], a);
                p.audio[(uint64_t)capture * p.audio_stride + (sg - p.audio_base)] = a;
            }
        }
        __syncthreads();
        /* carries */
        uint64_t valid = p.q_count - tile * B200_AMB_TILE;
        if (valid > B200_AMB_TILE) valid = B200_AMB_TILE;
        float hb = 0.0f;
        if (tid < B200_AM_BHIST) hb = s_b[(int)valid + tid];
        float nr = 0.0f, nb = 0.0f;
        if (tid == 32) nr = env[tile * B200_AMB_TILE + valid - 1];
        if (tid == 33) nb = s_b[B200_AM_BHIST + (int)valid - 1];
        __syncthreads();
        if (tid < B200_AM_BHIST) s_b[tid] = hb;
        if (tid == 32) s_carry[0] = nr;
        if (tid == 33) s_carry[1] = nb;
        __syncthreads();
    }
    if (p.state) {
        if (tid < B200_AM_BHIST) p.state[capture].b_hist[tid] = s_b[tid];
        if (tid == 32) p.state[capture].r_last = s_carry[0];
        if (tid == 33) p.state[capture].b_last = s_carry[1];
    }
}

#endif
