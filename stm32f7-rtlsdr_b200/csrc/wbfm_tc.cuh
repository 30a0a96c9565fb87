/*
 * wbfm_tc.cuh -- kernel K4 (FM), tensor-core engine (cfg.fir_engine = B200SDR_FIR_ENGINE_TENSOR, batched captures):
 * the same chain as wbfm.cuh -- u8 I/Q -> /10 80-tap FIR -> discriminator -> 75 us de-emphasis -> /5 FIR -> 48 kHz --
 * with the first FIR computed by the 5th-generation tensor cores (tcgen05.mma kind::i8, accumulators in TMEM) as an
 * EXACT integer product, straight from the raw bytes that TMA drops into shared memory.
 *
 * Reference anchor: the planned MCU shape is arm_fir_decimate_f32 (CMSIS/core/arm_math.h:3307); definition followed:
 * oracle/golden.c gold_wbfm().  DESIGN.md 5.2b has the arithmetic, the measurements and why this engine exists next to
 * the CUDA-core kernel (the FP32 pipe caps the scatter FIR at 0.71 of the HBM roofline; this form has no FP32 FIR).
 *
 * The FIR as a banded-Toeplitz GEMM.  A capture is cut into ROWS of 160 samples (320 bytes).  Row R of the A operand is
 * 512 raw bytes: 192 bytes (96 samples) of history, [320 R - 192, 320 R), then the row's own 320 bytes -- unsigned
 * 8-bit, interleaved I,Q exactly as the dongle delivers them, no conversion, no de-interleave.  The row yields the 16
 * stage-1 outputs y1[16 R + o], o = 0..15, and once more the output before them (o = -1), so the discriminator of a row
 * needs nothing from its neighbour.  The B operand is constant: column (s, j, c) holds slice s of the taps of output
 * o = j - 1 (j = 0..16) on the bytes of component c (I or Q), zero on the other component:
 *     B[(s, j, c)][2 kap + c'] = (c' == c) ? q_s[96 + 10 o - kap] : 0                (tap index 0..79, else 0)
 * where the float64-designed taps are cut into three signed 8-bit slices, h[t] 2^e = q0 2^-7 + q1 2^-14 + q2 2^-21
 * (21 bits + sign: 3.6e-7 of the largest tap).  D = A B is u8 x s8 -> s32, exact.  One tile = 125 rows (M = 128 with
 * three idle rows: 125 x 16 = 2000 outputs = 400 audio samples, so every tile starts on an audio sample), N = 112
 * (102 used), K = 512 = 16 MMAs of K = 32.
 *
 * Roles (one CTA of 320 threads per SM, persistent over (capture, segment) work items whose tiles it walks in order):
 *   warp 0      producer: ONE lane issues 8 TMA tensor copies per tile (cp.async.bulk.tensor, 64B swizzle: three
 *               64-byte columns of history from row R - 1, five of the row itself) into one of two operand stages; the
 *               tensor map is the plain (320 bytes, rows, captures) view of the batch, so the row before a capture and
 *               the rows behind its end are out of bounds = zero-filled by the hardware.  A capture whose length is
 *               not a multiple of 320 bytes has its last tile filled by the whole warp with bounds-checked cp.async
 *               instead (same layout);
 *   warp 1      one lane issues the 16 tcgen05.mma per tile into one of two TMEM accumulator stages and commits ONCE to the
 *               tile's "MMAs done" mbarrier, which both frees the operand stage and hands the accumulator on;
 *   warps 2..5 / 6..9   two epilogue GROUPS that take the tiles in turn (group = accumulator stage = tile index mod 2).
 *               Warp w reads TMEM lanes 32 (w % 4) .., a thread owns a ROW: it removes the 127.5 offset from the leading
 *               slice exactly (an integer and a half-integer below 2^23 are exact floats), adds the two small slices, and
 *               runs the 240 kS/s stages on its 16 consecutive outputs: discriminator, de-emphasis as a scan (thread-serial,
 *               then shuffle scans over the warp's 32 rows and the 32 rows before them -- what lies further back has
 *               decayed by a^512 = 4e-13 --, no shared-memory round trip), /5 FIR out of a shared window.  A group meets
 *               at its own 128-thread barrier once per tile; what a tile needs from the tile before it (the other group's:
 *               row totals, the newest 49 e[]) is ordered by a producer / consumer named barrier (bar.arrive / bar.sync)
 *               behind a bounded poll of a counter.  So the
 *               two warps of every scheduler belong to different groups, half a tile apart in time, and the arithmetic
 *               of one hides the latencies of the other.
 * Every wait is bounded (clock64): a protocol error sets *error and ends the kernel, it cannot hang the GPU.
 *
 * Host emulation (tests/emu): only the epilogue groups run (256 fibers); the integer product is computed from the same B
 * image and the same source addressing, so the image layout, the quantisation and everything after TMEM are checked on
 * the CPU.
 */
#ifndef B200_WBFM_TC_CUH
#define B200_WBFM_TC_CUH

#include "wbfm.cuh"
#if defined(__CUDACC__) && !defined(B200_EMULATED)
#include <cuda.h> /* CUtensorMap */
#endif

#define B200_TC_ROW_SAMPLES 160
#define B200_TC_ROW_BYTES 320
#define B200_TC_HIST_SAMPLES 96
#define B200_TC_HIST_BYTES 192                       /* 96 samples in front of the row: 3 columns of 64 bytes   */
#define B200_TC_K_BYTES 512                          /* K of the product = bytes of one A row                   */
#define B200_TC_KSTEPS 16                            /* MMAs of K = 32 per tile                                 */
#define B200_TC_ROWS 125                             /* data rows per tile (TMEM lanes 125..127 idle)           */
#define B200_TC_OPR 16                               /* stage-1 outputs per row = per epilogue thread           */
#define B200_TC_TILE_OUT (B200_TC_ROWS * B200_TC_OPR) /* 2000                                                   */
#define B200_TC_TILE_BYTES (B200_TC_ROWS * B200_TC_ROW_BYTES) /* 40000                                          */
#define B200_TC_SLICE_COLS 34                        /* 17 outputs x (I, Q)                                     */
#define B200_TC_N 112                                /* 3 slices x 34 = 102, padded to a multiple of 16         */
#define B200_TC_BOXES 8                              /* 64-byte K columns: 0..2 history, 3..7 the row           */
#define B200_TC_A_BOX (128 * 64)                     /* 128 rows x 64 bytes of K, 64B swizzle                   */
#define B200_TC_A_STAGE (B200_TC_BOXES * B200_TC_A_BOX)
#define B200_TC_B_BOX (B200_TC_N * 64)
#define B200_TC_B_BYTES (B200_TC_BOXES * B200_TC_B_BOX) /* 57344                                                */
#define B200_TC_TX_BYTES (B200_TC_BOXES * B200_TC_ROWS * 64) /* bytes one tile's TMA copies deliver             */
#define B200_TC_GROUPS 2                             /* epilogue groups, taking the tiles in turn               */
#define B200_TC_EPI 128                              /* threads per epilogue group                              */
#define B200_TC_THREADS (64 + B200_TC_GROUPS * B200_TC_EPI)
#define B200_TC_ACC_COLS 128                         /* TMEM columns per accumulator stage                      */
#define B200_TC_APT 4                                /* audio samples per thread in stage 2 (100 threads)       */
#define B200_TC_EBUF (B200_FM_HPAD + 128 * B200_TC_OPR + 16) /* floats per e[] buffer                           */

#define B200_TC_SM_A 0                                                           /* [2] operand stages        */
#define B200_TC_SM_B (B200_TC_SM_A + 2 * B200_TC_A_STAGE)
#define B200_TC_SM_E (B200_TC_SM_B + B200_TC_B_BYTES)                            /* float [group][2][EBUF]    */
#define B200_TC_SM_TOT (B200_TC_SM_E + B200_TC_GROUPS * 2 * B200_TC_EBUF * 4)    /* float [3][128]            */
#define B200_TC_SM_CNT (B200_TC_SM_TOT + 3 * 128 * 4)                            /* u32 [2] (+ pad)           */
#define B200_TC_SM_BAR (B200_TC_SM_CNT + 16)                                     /* u64 [8]                   */
#define B200_TC_SM_MISC (B200_TC_SM_BAR + 64)                                    /* u32 [4]                   */
#define B200_TC_SMEM_BYTES (B200_TC_SM_MISC + 16)

/* byte offset of element (row n, K byte k) inside an operand of `rows` rows: K-major, 64-byte swizzle
 * (cute Swizzle<2,4,3>): columns of 64 K-bytes, row pitch 64, the 16-byte chunk index XORed with (row / 2) % 4 */
#define B200_TC_OP_OFF(rows, n, k) \
    ((uint32_t)(((k) >> 6) * ((rows) * 64) + (n) * 64 + (((((k) & 63) >> 4) ^ (((n) >> 1) & 3)) << 4) + ((k) & 15)))
/* accumulator column of (slice s, output j of the row's seventeen (o = j - 1), component c) */
#define B200_TC_COL(s, j, c) (B200_TC_SLICE_COLS * (s) + 2 * (j) + (c))

struct FmTcConsts {
    float b0;            /* 127.5 sum q0: the offset's share of the leading slice (exact in fp32)              */
    float c0, c1, c2;    /* 2^-7 / 2^e, 2^-14 / 2^e, 2^-21 / 2^e                                               */
    float k12;           /* -127.5 (c1 sum q1 + c2 sum q2)                                                     */
    float b0_first[16];  /* the same for the first row of a capture, whose history bytes are zero-filled:      */
    float k12_first[16]; /* output o sees real samples through taps t <= 10 o only (x[n < 0] = 0)              */
    float apow[16];      /* a^(i+1)                                                                            */
    float a16pow[5];     /* (a^16)^(2^s): decay over 2^s rows                                                  */
    float alpha;
    float h2[B200_FM_T2];
};

struct FmTcParams {
    const uint8_t *iq;       /* capture c at iq + c * capture_stride (16-byte aligned)                          */
    uint64_t capture_stride; /* bytes                                                                           */
    uint64_t capture_bytes;  /* valid bytes per capture (multiple of 16)                                        */
    uint64_t m1;             /* stage-1 outputs per capture                                                     */
    uint32_t n_tiles;        /* tiles per capture                                                               */
    uint32_t total_rows;     /* rows per capture = ceil(samples / 160)                                          */
    uint32_t tiles_per_segment, segments, n_captures;
    uint32_t manual_from_tile; /* tiles >= this are filled with cp.async instead of TMA (0: no tensor map at all) */
    float *audio;            /* [capture][audio_stride]                                                         */
    uint64_t audio_stride;
    float *disc;             /* optional [capture][disc_stride]                                                 */
    uint64_t disc_stride;
    const uint8_t *b_image;  /* B200_TC_B_BYTES: the B operand as it lies in shared memory                      */
    uint32_t *error;         /* device word, 0 = ok; else which bounded wait expired                            */
    int32_t *dbg_acc;        /* optional [128][112]: raw accumulators of tile 0 of capture 0 (tests)            */
    uint32_t dbg_flags;      /* unused, zero: no kernel reads it; the host emulation harness of tests/emu still sets it */
};

#ifdef B200_EMULATED
static FmTcConsts c_fm_tc;
#else
__constant__ FmTcConsts c_fm_tc;
#endif

#if defined(__CUDACC__) && !defined(B200_EMULATED) /* ------------------------------------ device-only plumbing */

B200_DEV uint32_t b200_tc_smem(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
B200_DEV void b200_tc_bar_init(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(b200_tc_smem(bar)), "r"(count) : "memory");
}

B200_DEV uint64_t b200_tc_desc(uint32_t saddr)
{
    /* cute::UMMA::SmemDescriptor: start >> 4 [0,14), LBO >> 4 [16,30) = 1 (K-major swizzled: unused),
     * SBO >> 4 [32,46) = 512 >> 4 (8 rows x 64 bytes), version 1 [46,48), layout SWIZZLE_64B = 4 [61,64) */
    return (uint64_t)((saddr >> 4) & 0x3fffu) | ((uint64_t)1 << 16) | ((uint64_t)(512 >> 4) << 32) | ((uint64_t)1 << 46) |
           ((uint64_t)4 << 61);
}
/* cute::UMMA::InstrDescriptor: D = S32 (2 at [4,6)), A = unsigned 8-bit (0 at [7,10)), B = signed 8-bit (1 at [10,13)),
 * both K-major, N >> 3 at [17,23), M >> 4 at [24,29) */
#define B200_TC_IDESC ((2u << 4) | (0u << 7) | (1u << 10) | ((uint32_t)(B200_TC_N >> 3) << 17) | ((128u >> 4) << 24))

B200_DEV void b200_tc_mma(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t accumulate)
{
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, {%5, %5, %5, %5}, p;\n\t}\n" ::"r"(tmem_d),
        "l"(da), "l"(db), "r"(B200_TC_IDESC), "r"(accumulate), "r"(0u)
        : "memory");
}
B200_DEV void b200_tc_commit(uint64_t *bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(b200_tc_smem(bar)) : "memory");
}
B200_DEV void b200_tc_arrive(uint64_t *bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(b200_tc_smem(bar)) : "memory");
}
B200_DEV void b200_tc_arrive_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(b200_tc_smem(bar)), "r"(bytes) : "memory");
}
/* one box of the (320 bytes, rows, captures) view: 64 bytes x 125 rows, 64B swizzle, zero fill out of bounds */
B200_DEV void b200_tc_tma_box(uint32_t sdst, const void *tmap, int32_t x, int32_t row, int32_t capture, uint64_t *bar)
{
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(sdst),
                 "l"(tmap), "r"(x), "r"(row), "r"(capture), "r"(b200_tc_smem(bar))
                 : "memory");
}
/* bounded wait; gives up when another role has already failed */
B200_DEV bool b200_tc_wait(uint64_t *bar, uint32_t parity, volatile uint32_t *abort_flag)
{
    const long long t0 = clock64();
    for (;;) {
        uint32_t ok;
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.b32 %0, 1, 0, p;\n\t}\n"
                     : "=r"(ok)
                     : "r"(b200_tc_smem(bar)), "r"(parity)
                     : "memory");
        if (ok) return true;
        if (*abort_flag) return false;
        if (clock64() - t0 > (1ll << 28)) return false;
    }
}
B200_DEV void b200_tc_ld32(uint32_t taddr, uint32_t (&v)[32])
{
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
        "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
          "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
          "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
}
B200_DEV void b200_tc_cp16(uint32_t sdst, const void *gsrc, uint32_t src_bytes)
{
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(sdst), "l"(gsrc), "r"(src_bytes) : "memory");
}
/* named barrier of one epilogue group (128 threads) */
B200_DEV void b200_tc_epi_sync(int grp)
{
    if (grp == 0) asm volatile("bar.sync 1, 128;" ::: "memory");
    else asm volatile("bar.sync 2, 128;" ::: "memory");
}
B200_DEV void b200_tc_ld2(uint32_t taddr, uint32_t &a, uint32_t &b)
{
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0, %1}, [%2];" : "=r"(a), "=r"(b) : "r"(taddr) : "memory");
}
B200_DEV long long b200_tc_clock() { return clock64(); }
/* "phase B of my tile is done" from one epilogue group to the other: the 128 threads of group grp arrive on named barrier
 * 3 + grp, the 128 threads of the other group sync on it (256 participants) */
B200_DEV void b200_tc_group_done(int grp)
{
    if (grp == 0) asm volatile("bar.arrive 3, 256;" ::: "memory");
    else asm volatile("bar.arrive 4, 256;" ::: "memory");
}
B200_DEV void b200_tc_group_wait(int other)
{
    if (other == 0) asm volatile("bar.sync 3, 256;" ::: "memory");
    else asm volatile("bar.sync 4, 256;" ::: "memory");
}

#else

B200_DEV void b200_tc_epi_sync(int grp) { emu::named_barrier(1 + grp, 128); }
B200_DEV long long b200_tc_clock() { emu::yield_now(); return 0; } /* a poll of the other group: let its fibers run */
B200_DEV void b200_tc_group_done(int grp) { emu::named_arrive(3 + grp, 256); }
B200_DEV void b200_tc_group_wait(int other) { emu::named_barrier(3 + other, 256); }

#endif

/* (capture, segment) -> tile range; segments > 0 pre-roll one tile with stores suppressed (de-emphasis / audio-FIR
 * state; the stage-1 FIR and the discriminator have no state here: a row carries its own history bytes) */
struct FmTcItem {
    uint32_t capture, seg, t_begin, t_end, t_first_store;
};
B200_DEV FmTcItem b200_tc_item(const FmTcParams &p, uint32_t item)
{
    FmTcItem w;
    w.capture = item / p.segments;
    w.seg = item % p.segments;
    w.t_begin = w.seg * p.tiles_per_segment;
    w.t_end = w.t_begin + p.tiles_per_segment;
    if (w.t_end > p.n_tiles) w.t_end = p.n_tiles;
    w.t_first_store = w.t_begin;
    if (w.seg > 0) w.t_begin -= 1;
    return w;
}

/* source byte offset (from the capture start) of the 16-byte chunk `chunk` of K column `box` of capture row R, and whether
 * it lies inside the capture: columns 0..2 are the last 192 bytes of row R - 1, columns 3..7 the 320 bytes of row R.
 * This is exactly what the tensor map's bounds give the TMA copies (whole rows) -- refined to 16 bytes for ragged ends. */
B200_DEV bool b200_tc_src(int64_t R, int box, int chunk, uint64_t capture_bytes, int64_t &off)
{
    if (box < 3) {
        off = (R - 1) * B200_TC_ROW_BYTES + 128 + 64 * box + 16 * chunk;
        return R >= 1 && off + 16 <= (int64_t)capture_bytes;
    }
    off = R * B200_TC_ROW_BYTES + 64 * (box - 3) + 16 * chunk;
    return off + 16 <= (int64_t)capture_bytes;
}

/* atan2 as in wbfm.cuh with a degree-13 odd polynomial (7 coefficients, 3.2e-7 rad in fp32) */
B200_DEV float b200_tc_atan2(float y, float x)
{
    const float ax = fabsf(x), ay = fabsf(y);
    const float mx = fmaxf(fmaxf(ax, ay), 1e-30f), mn = fminf(ax, ay);
    const float a = mn * b200_rcp_fast(mx);
    const float s = a * a;
    float p = 6.811790634e-03f;
    p = fmaf(p, s, -3.360421286e-02f);
    p = fmaf(p, s, 7.962366400e-02f);
    p = fmaf(p, s, -1.323334168e-01f);
    p = fmaf(p, s, 1.980781547e-01f);
    p = fmaf(p, s, -3.331736805e-01f);
    p = fmaf(p, s, 9.999961115e-01f);
    float r = p * a;
    if (ay > ax) r = 1.57079632679489662f - r;
    if (x < 0.0f) r = 3.14159265358979324f - r;
    return copysignf(r, y);
}

/* ---- The 240 kS/s stages.  Tile n of the CTA's sequence belongs to epilogue group n & 1 (= its TMEM stage); a thread = a
 * row = 16 outputs.  Per tile, in the group:
 *     A(n)   accumulators -> y1 -> discriminator -> thread-serial de-emphasis of the row (registers), row total -> s_tot[n % 3]
 *     ---- the group's barrier ----
 *     C      /5 FIR of the group's PREVIOUS tile out of its e[] buffer (complete since the barrier)
 *     wait until the other group has finished B(n - 1)
 *     B(n)   shuffle scans of the row totals (this tile's and the last 32 rows of tile n - 1) -> carried-in value -> e[] of
 *            the row -> the group's e[] buffer (n / 2) & 1, with the newest e[] of tile n - 1 in front of it; bump the counter
 * row = TMEM lane, q = row / 32 = the warp's lane quarter, et = index among the group's epilogue threads. ---- */
struct FmTcTile {
    uint32_t tile, it;
    int last;      /* last row of the tile that holds samples */
    bool store;
    uint64_t m0;
};
B200_DEV FmTcTile b200_tc_tile(const FmTcParams &p, const FmTcItem &w, uint32_t tile, uint32_t it)
{
    FmTcTile t;
    t.tile = tile;
    t.it = it;
    t.store = tile >= w.t_first_store;
    t.m0 = (uint64_t)tile * B200_TC_TILE_OUT;
    t.last = (int)(p.total_rows - tile * B200_TC_ROWS) - 1;
    if (t.last > B200_TC_ROWS - 1) t.last = B200_TC_ROWS - 1;
    return t;
}

/* y1 of the row from the three accumulator slices: y = (d0 - 127.5 sum q0) c0 + (128 d1 + d2) c2 - 127.5 (c1 sum q1 + c2
 * sum q2).  The leading slice loses its offset exactly (integer minus half-integer, both below 2^23), the two small
 * slices are joined as integers.  lo[2 j + c] = 128 d1 + d2 as a float, d0[2 j + c] the leading slice.
 * FIRST: the tile holds the first row of a capture (tile 0), whose history bytes are zeros, not samples. */
template <bool FIRST>
B200_DEV void b200_tc_phase_a(const FmTcParams &p, const FmTcItem &w, const FmTcTile &t, const float (&lo)[B200_TC_SLICE_COLS],
                              const uint32_t (&d0)[B200_TC_SLICE_COLS], int row, float (&e)[B200_TC_OPR], float *s_tot)
{
    const FmTcConsts *k = &c_fm_tc;
    const bool first_row = FIRST && row == 0;
    const float c0 = k->c0, c2 = k->c2;
    const float alpha = k->alpha, a1 = 1.0f - alpha;
    float pr, pi, run = 0.0f; /* previous output; de-emphasis state from zero */
    {
        const float b0 = k->b0, k12 = k->k12; /* j = 0 is output -1: of row 0 of a capture it is y1[-1], never used */
        pr = fmaf((float)(int32_t)d0[0] - b0, c0, fmaf(lo[0], c2, k12));
        pi = fmaf((float)(int32_t)d0[1] - b0, c0, fmaf(lo[1], c2, k12));
    }
    float d[B200_TC_OPR];
#pragma unroll
    for (int i = 0; i < B200_TC_OPR; ++i) {
        float b0 = k->b0, k12 = k->k12;
        if (FIRST && first_row) { b0 = k->b0_first[i]; k12 = k->k12_first[i]; }
        const float yr = fmaf((float)(int32_t)d0[2 * i + 2] - b0, c0, fmaf(lo[2 * i + 2], c2, k12));
        const float yi = fmaf((float)(int32_t)d0[2 * i + 3] - b0, c0, fmaf(lo[2 * i + 3], c2, k12));
        const float zr = fmaf(yr, pr, yi * pi);
        const float zi = fmaf(yi, pr, -(yr * pi));
        d[i] = b200_tc_atan2(zi, zr);
        pr = yr;
        pi = yi;
    }
    if (FIRST && row == 0) d[0] = 0.0f; /* y1[-1] = 0: defined as d[0] = 0 */
    if (p.disc && t.store && row < B200_TC_ROWS) { /* lanes 125..127 hold no row of this tile */
        const uint64_t m = t.m0 + (uint64_t)row * B200_TC_OPR;
        float *dst = p.disc + (uint64_t)w.capture * p.disc_stride + m;
        const int n_valid = p.m1 > m ? (p.m1 - m > B200_TC_OPR ? B200_TC_OPR : (int)(p.m1 - m)) : 0;
#pragma unroll
        for (int i = 0; i < B200_TC_OPR; ++i)
            if (i < n_valid) dst[i] = d[i];
    }
#pragma unroll
    for (int i = 0; i < B200_TC_OPR; ++i) {
        run = fmaf(a1, run, alpha * d[i]);
        e[i] = run;
    }
    s_tot[row] = run;
}

/* The de-emphasis state in front of every row.  S[r] = a^16 S[r-1] + tot[r]; what lies more than 512 outputs = 32 rows back
 * has decayed by a^512 = 4e-13 (far below one fp32 ulp), so a warp scans the totals of its own 32 rows and of the 32 rows
 * before them (for the first quarter: rows 93..124 of the previous tile, which is always a full one; zeros at the start of
 * a work item) with two interleaved shuffle scans -- no shared-memory round trip, no carry from warp to warp.  Then e[] of
 * the row gets its carried-in part and goes to the group's e[] buffer. */
B200_DEV void b200_tc_phase_b(const FmTcTile &t, float (&e)[B200_TC_OPR], int row, int et, float lane_pow, float *s_e_cur,
                              const float *s_e_prev, const float *s_tot, const float *s_tot_prev)
{
    const FmTcConsts *k = &c_fm_tc;
    const int lane = row & 31, q = row >> 5;
    /* the 49 (52) newest e[] of the previous tile go in front of this tile's buffer (zeros at the start of a work item;
     * the previous tile of an item is always a full one) */
    if (et < B200_FM_HPAD) s_e_cur[et] = t.it ? s_e_prev[B200_FM_HPAD + B200_TC_TILE_OUT - B200_FM_HPAD + et] : 0.0f;
    float v = s_tot[row];
    float u = q ? s_tot[row - 32] : (t.it ? s_tot_prev[B200_TC_ROWS - 32 + lane] : 0.0f);
#pragma unroll
    for (int s = 0; s < 5; ++s) {
        const float nv = __shfl_up_sync(0xffffffffu, v, 1u << s), nu = __shfl_up_sync(0xffffffffu, u, 1u << s);
        if (lane >= (1 << s)) {
            v = fmaf(k->a16pow[s], nv, v);
            u = fmaf(k->a16pow[s], nu, u);
        }
    }
    float excl = __shfl_up_sync(0xffffffffu, v, 1u); /* state built up inside the quarter in front of this row */
    if (lane == 0) excl = 0.0f;
    const float behind_prev = __shfl_sync(0xffffffffu, u, 31); /* state behind the 32 rows before the quarter */
    const float cin = fmaf(lane_pow, behind_prev, excl);       /* lane_pow = (a^16)^lane */
#pragma unroll
    for (int i = 0; i < B200_TC_OPR; ++i) e[i] = fmaf(k->apow[i], cin, e[i]);
    float4 *de = reinterpret_cast<float4 *>(s_e_cur + B200_FM_HPAD + row * B200_TC_OPR);
#pragma unroll
    for (int i = 0; i < B200_TC_OPR / 4; ++i) de[i] = make_float4(e[4 * i], e[4 * i + 1], e[4 * i + 2], e[4 * i + 3]);
}

/* stage 2 of a tile whose e[] is complete: audio[p] = sum_k h2[k] e[5 p - k].  A tile starts at a multiple of 20 stage-1
 * outputs; thread et < 100 owns the four audio samples p = m0 / 5 + 4 et + r whose window e[20 et - 49 .. 20 et + 15] sits
 * at the fixed offset 3 behind the 16-byte aligned address s_e + 20 et: 17 128-bit loads, taps outermost (wbfm.cuh) */
B200_DEV void b200_tc_phase_c(const FmTcParams &p, uint32_t capture, const FmTcTile &t, int et, const float *s_e)
{
    const FmTcConsts *k = &c_fm_tc;
    uint64_t mg_end = t.m0 + (uint64_t)(t.last + 1) * B200_TC_OPR;
    if (mg_end > p.m1) mg_end = p.m1;
    const uint64_t pg_first = t.m0 / B200_FM_D2;
    const uint64_t pg_end = (mg_end + B200_FM_D2 - 1) / B200_FM_D2;
    const uint64_t pg0 = pg_first + (uint64_t)et * B200_TC_APT;
    if (et < B200_TC_TILE_OUT / (B200_FM_D2 * B200_TC_APT) && pg0 < pg_end) {
        constexpr int WOFF = B200_FM_HPAD - B200_FM_HIST; /* 3 */
        constexpr int NW4 = (WOFF + B200_FM_T2 + B200_FM_D2 * (B200_TC_APT - 1) + 3) / 4; /* 17 */
        const float4 *win = reinterpret_cast<const float4 *>(s_e + et * (B200_FM_D2 * B200_TC_APT));
        float ew[4 * NW4];
#pragma unroll
        for (int j = 0; j < NW4; ++j) {
            const float4 v = win[j];
            ew[4 * j] = v.x; ew[4 * j + 1] = v.y; ew[4 * j + 2] = v.z; ew[4 * j + 3] = v.w;
        }
        float au[B200_TC_APT];
#pragma unroll
        for (int r = 0; r < B200_TC_APT; ++r) au[r] = 0.0f;
#pragma unroll
        for (int tp = 0; tp < B200_FM_T2; ++tp) {
            const float hk = k->h2[tp];
#pragma unroll
            for (int r = 0; r < B200_TC_APT; ++r) au[r] = fmaf(hk, ew[WOFF + B200_FM_HIST + B200_FM_D2 * r - tp], au[r]);
        }
        if (t.store) {
            float *dst = p.audio + (uint64_t)capture * p.audio_stride + pg0;
#pragma unroll
            for (int r = 0; r < B200_TC_APT; ++r)
                if (pg0 + r < pg_end) dst[r] = au[r];
        }
    }
}

/* the epilogue group's walk over the CTA's tiles; `take(w, tile, it, n, e)` fetches the accumulators of the tile with
 * running index n and runs phase A into e[] (device: TMEM loads; emulation: the integer product on the host) */
template <class Take>
B200_DEV bool b200_tc_epilogue_group(const FmTcParams &p, uint32_t n_items, uint32_t first_item, uint32_t item_step, int grp, int row, int et,
                                     unsigned char *smem, volatile uint32_t *abort_flag, Take take)
{
    float *s_e_grp = reinterpret_cast<float *>(smem + B200_TC_SM_E);
    float *s_tot = reinterpret_cast<float *>(smem + B200_TC_SM_TOT);
    volatile uint32_t *s_cnt = reinterpret_cast<volatile uint32_t *>(smem + B200_TC_SM_CNT);
    const int lane = row & 31;
    float lane_pow = 1.0f; /* (a^16)^lane */
#pragma unroll
    for (int s = 0; s < 5; ++s)
        if (lane & (1 << s)) lane_pow *= c_fm_tc.a16pow[s];
    bool have_pend = false;
    uint32_t pend_capture = 0, pend_n = 0;
    FmTcTile pend_t{};
    uint32_t n = 0; /* running tile index of the CTA */
    for (uint32_t item = first_item; item < n_items; item += item_step) {
        const FmTcItem w = b200_tc_item(p, item);
        for (uint32_t tile = w.t_begin, it = 0; tile < w.t_end; ++tile, ++it, ++n) {
            if ((int)(n & 1u) != grp) continue;
            const FmTcTile t = b200_tc_tile(p, w, tile, it);
            float e[B200_TC_OPR];
            if (!take(w, t, n, e, s_tot + (n % 3u) * 128)) return false;
            b200_tc_epi_sync(grp); /* the group's row totals of tile n and its e[] of its previous tile are complete */
            if (have_pend) b200_tc_phase_c(p, pend_capture, pend_t, et, s_e_grp + (grp * 2 + ((pend_n >> 1) & 1u)) * B200_TC_EBUF);
            /* tile n - 1 is the other group's: its phase B (hence its row totals and its e[]) must be done.  Always waited
             * for, also at the start of a work item, so the groups never drift more than one tile apart (buffer reuse) */
            if (n > 0) {
                /* bounded poll of the other group's counter first (a protocol error must end the kernel, not hang it), then
                 * the named barrier its threads have arrived on: that is the synchronisation proper */
                const uint32_t need = 4u * ((n - 1u) / 2u + 1u);
                const long long t0 = b200_tc_clock();
                while (s_cnt[grp ^ 1] < need) {
                    if (*abort_flag || b200_tc_clock() - t0 > (1ll << 28)) return false;
                }
                b200_tc_group_wait(grp ^ 1);
            }
            b200_tc_phase_b(t, e, row, et, lane_pow, s_e_grp + (grp * 2 + ((n >> 1) & 1u)) * B200_TC_EBUF,
                            s_e_grp + ((grp ^ 1) * 2 + (((n - 1u) >> 1) & 1u)) * B200_TC_EBUF, s_tot + (n % 3u) * 128,
                            s_tot + ((n + 2u) % 3u) * 128);
            __threadfence_block();
            __syncwarp();
            if (lane == 0) atomicAdd(const_cast<uint32_t *>(s_cnt) + grp, 1u);
            b200_tc_group_done(grp);
            have_pend = true;
            pend_capture = w.capture;
            pend_t = t;
            pend_n = n;
        }
    }
    if (have_pend) { /* drain: the audio of the group's last tile */
        b200_tc_epi_sync(grp);
        b200_tc_phase_c(p, pend_capture, pend_t, et, s_e_grp + (grp * 2 + ((pend_n >> 1) & 1u)) * B200_TC_EBUF);
    }
    return true;
}

#ifdef B200_EMULATED
/* the integer product as the tensor cores compute it, from the same source addressing and the same B image */
static void b200_tc_emulated_acc(const FmTcParams &p, const FmTcItem &w, uint32_t tile, int row, int32_t (&acc)[3 * B200_TC_SLICE_COLS])
{
    const uint8_t *cap = p.iq + (uint64_t)w.capture * p.capture_stride;
    uint8_t a[B200_TC_K_BYTES];
    for (int kk = 0; kk < B200_TC_K_BYTES; ++kk) {
        int64_t off;
        const bool valid = b200_tc_src((int64_t)tile * B200_TC_ROWS + row, kk >> 6, (kk & 63) >> 4, p.capture_bytes, off);
        a[kk] = valid ? cap[off + (kk & 15)] : 0;
    }
    for (int n = 0; n < 3 * B200_TC_SLICE_COLS; ++n) {
        int64_t sum = 0;
        for (int kk = 0; kk < B200_TC_K_BYTES; ++kk) sum += (int64_t)a[kk] * (int64_t)(int8_t)p.b_image[B200_TC_OP_OFF(B200_TC_N, n, kk)];
        acc[n] = (int32_t)sum;
    }
}
#endif

#if defined(__CUDACC__) && !defined(B200_EMULATED)
__global__ void __launch_bounds__(B200_TC_THREADS, 1) k_wbfm_tc(FmTcParams p, const __grid_constant__ CUtensorMap tmap)
#else
__global__ void __launch_bounds__(B200_TC_THREADS, 1) k_wbfm_tc(FmTcParams p)
#endif
{
    B200_DYN_SMEM(smem);
    const int tid = (int)threadIdx.x;
    const uint32_t n_items = p.segments * p.n_captures;
#ifdef B200_EMULATED
    /* 256 fibers: the two epilogue groups only */
    const int grp = tid >> 7, row = tid & 127;
    uint32_t abort_never = 0;
    if (tid < 2) reinterpret_cast<uint32_t *>(smem + B200_TC_SM_CNT)[tid] = 0u;
    __syncthreads();
    auto take = [&](const FmTcItem &w, const FmTcTile &t, uint32_t, float (&e)[B200_TC_OPR], float *s_tot) -> bool {
        int32_t acc[3 * B200_TC_SLICE_COLS];
        if (row < B200_TC_ROWS) b200_tc_emulated_acc(p, w, t.tile, row, acc);
        else for (int n = 0; n < 3 * B200_TC_SLICE_COLS; ++n) acc[n] = 0x12345 * (n + tid); /* idle lanes hold anything */
        if (p.dbg_acc && w.capture == 0 && t.tile == 0)
            for (int n = 0; n < 3 * B200_TC_SLICE_COLS; ++n) p.dbg_acc[row * B200_TC_N + n] = acc[n];
        float lo[B200_TC_SLICE_COLS];
        uint32_t d0[B200_TC_SLICE_COLS];
        for (int n = 0; n < B200_TC_SLICE_COLS; ++n) {
            lo[n] = (float)(acc[B200_TC_SLICE_COLS + n] * 128 + acc[2 * B200_TC_SLICE_COLS + n]);
            d0[n] = (uint32_t)acc[n];
        }
        if (t.tile == 0) b200_tc_phase_a<true>(p, w, t, lo, d0, row, e, s_tot);
        else b200_tc_phase_a<false>(p, w, t, lo, d0, row, e, s_tot);
        return true;
    };
    b200_tc_epilogue_group(p, n_items, blockIdx.x, gridDim.x, grp, row, row, smem, &abort_never, take);
#else
    const int warp = tid >> 5, lane = tid & 31;
    uint64_t *s_bar = reinterpret_cast<uint64_t *>(smem + B200_TC_SM_BAR);
    uint64_t *bar_full = s_bar, *bar_empty = s_bar + 2, *bar_tfull = s_bar + 4, *bar_tempty = s_bar + 6;
    uint32_t *s_misc = reinterpret_cast<uint32_t *>(smem + B200_TC_SM_MISC); /* [0] TMEM base, [1] abort flag */
    volatile uint32_t *s_abort = s_misc + 1;

    if (tid == 0) {
        for (int i = 0; i < 2; ++i) {
            b200_tc_bar_init(bar_full + i, 1);
            b200_tc_bar_init(bar_empty + i, 1);
            b200_tc_bar_init(bar_tfull + i, 1);
            b200_tc_bar_init(bar_tempty + i, B200_TC_EPI / 32); /* one arrival per warp of the stage's epilogue group */
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        s_misc[1] = 0u;
        reinterpret_cast<uint32_t *>(smem + B200_TC_SM_CNT)[0] = 0u;
        reinterpret_cast<uint32_t *>(smem + B200_TC_SM_CNT)[1] = 0u;
        if (p.manual_from_tile) asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap) : "memory");
    }
    if (warp == 1) { /* TMEM: two accumulator stages of 128 columns */
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(b200_tc_smem(s_misc)), "r"(2u * B200_TC_ACC_COLS)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    { /* the constant B operand */
        const uint4 *src = reinterpret_cast<const uint4 *>(p.b_image);
        uint4 *dst = reinterpret_cast<uint4 *>(smem + B200_TC_SM_B);
        for (int i = tid; i < B200_TC_B_BYTES / 16; i += B200_TC_THREADS) dst[i] = __ldg(src + i);
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); /* generic-proxy stores -> visible to the MMA's async proxy */
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = s_misc[0];
    const uint32_t a_base = b200_tc_smem(smem + B200_TC_SM_A), b_base = b200_tc_smem(smem + B200_TC_SM_B);

    if (warp == 0) {
        /* ===== producer ===== */
        uint32_t g = 0;
        bool ok = true;
        const int chunk = lane & 3, rsub = lane >> 2; /* manual fill: 8 rows x 4 chunks of one 64-byte column per instruction */
        for (uint32_t item = blockIdx.x; item < n_items && ok; item += gridDim.x) {
            const FmTcItem w = b200_tc_item(p, item);
            const uint8_t *cap = p.iq + (uint64_t)w.capture * p.capture_stride;
            for (uint32_t tile = w.t_begin; tile < w.t_end; ++tile, ++g) {
                const uint32_t stage = g & 1u, phase = (g >> 1) & 1u;
                if (!b200_tc_wait(bar_tfull + stage, phase ^ 1u, s_abort)) { ok = false; break; } /* MMAs of the tile two back done */
                const uint32_t a_stage = a_base + stage * B200_TC_A_STAGE;
                const int32_t R0 = (int32_t)(tile * B200_TC_ROWS);
                if (tile < p.manual_from_tile) {
                    if (lane == 0) {
                        b200_tc_arrive_expect_tx(bar_full + stage, B200_TC_TX_BYTES);
#pragma unroll
                        for (int b = 0; b < B200_TC_BOXES; ++b)
                            b200_tc_tma_box(a_stage + b * B200_TC_A_BOX, &tmap, b < 3 ? 128 + 64 * b : 64 * (b - 3), b < 3 ? R0 - 1 : R0,
                                            (int32_t)w.capture, bar_full + stage);
                    }
                } else { /* ragged end of a capture (or no tensor map): bounds-checked 16-byte copies, same layout */
#pragma unroll 1
                    for (int b = 0; b < B200_TC_BOXES; ++b) {
#pragma unroll 2
                        for (int rr = 0; rr < 16; ++rr) {
                            const int r = rr * 8 + rsub;
                            if (r < B200_TC_ROWS) {
                                int64_t off;
                                const bool valid = b200_tc_src((int64_t)R0 + r, b, chunk, p.capture_bytes, off);
                                b200_tc_cp16(a_stage + (uint32_t)(b * B200_TC_A_BOX + r * 64 + ((chunk ^ ((r >> 1) & 3)) << 4)),
                                             cap + (valid ? off : 0), valid ? 16u : 0u);
                            }
                        }
                    }
                    asm volatile("cp.async.commit_group;" ::: "memory");
                    asm volatile("cp.async.wait_group 0;" ::: "memory");
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    __syncwarp();
                    if (lane == 0) b200_tc_arrive(bar_full + stage);
                }
                __syncwarp();
            }
        }
        if (!ok && lane == 0) { *s_abort = 1u; atomicCAS(p.error, 0u, 1u); }
    } else if (warp == 1) {
        /* ===== MMA issuer (one lane) ===== */
        if (lane == 0) {
            uint32_t g = 0;
            uint32_t fail = 0;
            for (uint32_t item = blockIdx.x; item < n_items && !fail; item += gridDim.x) {
                const FmTcItem w = b200_tc_item(p, item);
                for (uint32_t tile = w.t_begin; tile < w.t_end; ++tile, ++g) {
                    const uint32_t stage = g & 1u, phase = (g >> 1) & 1u;
                    if (!b200_tc_wait(bar_full + stage, phase, s_abort)) { fail = 2; break; }
                    if (!b200_tc_wait(bar_tempty + stage, phase ^ 1u, s_abort)) { fail = 3; break; }
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    const uint32_t a_stage = a_base + stage * B200_TC_A_STAGE;
#pragma unroll
                    for (int ks = 0; ks < B200_TC_KSTEPS; ++ks) {
                        const uint64_t da = b200_tc_desc(a_stage + (uint32_t)((ks >> 1) * B200_TC_A_BOX + (ks & 1) * 32));
                        const uint64_t db = b200_tc_desc(b_base + (uint32_t)((ks >> 1) * B200_TC_B_BOX + (ks & 1) * 32));
                        b200_tc_mma(tmem + stage * B200_TC_ACC_COLS, da, db, ks > 0 ? 1u : 0u);
                    }
                    /* ONE commit per tile (each costs the tensor pipe a drain, profiles/r2_wbfm_tc.txt): the same event frees
                     * the operand stage for the producer and hands the accumulator to the epilogue */
                    b200_tc_commit(bar_tfull + stage);
                }
            }
            if (fail) { *s_abort = 1u; atomicCAS(p.error, 0u, fail); }
        }
        __syncwarp();
    } else {
        /* ===== epilogue group grp: the tiles with running index n = grp (mod 2), accumulator stage grp ===== */
        const int grp = (warp - 2) >> 2;
        const int q = warp & 3;              /* TMEM lane quarter this warp may read */
        const int row = q * 32 + lane;
        const int et = (warp - 2 - 4 * grp) * 32 + lane;
        const uint32_t taddr = tmem + ((uint32_t)(q * 32) << 16) + grp * B200_TC_ACC_COLS;
        auto take = [&](const FmTcItem &w, const FmTcTile &t, uint32_t n, float (&e)[B200_TC_OPR], float *s_tot) -> bool {
            if (!b200_tc_wait(bar_tfull + grp, (n >> 1) & 1u, s_abort)) return false;
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            /* the two small slices first, joined as integers; then the leading one */
            float lo[B200_TC_SLICE_COLS];
            {
                uint32_t v1[32], v2[32], w1a, w1b, w2a, w2b;
                b200_tc_ld32(taddr + B200_TC_SLICE_COLS, v1);
                b200_tc_ld2(taddr + B200_TC_SLICE_COLS + 32, w1a, w1b);
                b200_tc_ld32(taddr + 2 * B200_TC_SLICE_COLS, v2);
                b200_tc_ld2(taddr + 2 * B200_TC_SLICE_COLS + 32, w2a, w2b);
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                if (p.dbg_acc && w.capture == 0 && t.tile == 0) {
#pragma unroll
                    for (int c = 0; c < B200_TC_SLICE_COLS; ++c) {
                        p.dbg_acc[row * B200_TC_N + B200_TC_SLICE_COLS + c] = c < 32 ? (int32_t)v1[c < 32 ? c : 0] : (c == 32 ? (int32_t)w1a : (int32_t)w1b);
                        p.dbg_acc[row * B200_TC_N + 2 * B200_TC_SLICE_COLS + c] = c < 32 ? (int32_t)v2[c < 32 ? c : 0] : (c == 32 ? (int32_t)w2a : (int32_t)w2b);
                    }
                }
#pragma unroll
                for (int c = 0; c < 32; ++c) lo[c] = (float)((int32_t)v1[c] * 128 + (int32_t)v2[c]);
                lo[32] = (float)((int32_t)w1a * 128 + (int32_t)w2a);
                lo[33] = (float)((int32_t)w1b * 128 + (int32_t)w2b);
            }
            uint32_t d0[B200_TC_SLICE_COLS];
            {
                uint32_t v0[32];
                b200_tc_ld32(taddr, v0);
                b200_tc_ld2(taddr + 32, d0[32], d0[33]);
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                for (int c = 0; c < 32; ++c) d0[c] = v0[c];
            }
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncwarp();
            if (lane == 0) b200_tc_arrive(bar_tempty + grp); /* the MMA lane may overwrite this accumulator */
            if (p.dbg_acc && w.capture == 0 && t.tile == 0) {
#pragma unroll
                for (int c = 0; c < B200_TC_SLICE_COLS; ++c) p.dbg_acc[row * B200_TC_N + c] = (int32_t)d0[c];
            }
            if (t.tile == 0) b200_tc_phase_a<true>(p, w, t, lo, d0, row, e, s_tot);
            else b200_tc_phase_a<false>(p, w, t, lo, d0, row, e, s_tot);
            return true;
        };
        const bool ok = b200_tc_epilogue_group(p, n_items, blockIdx.x, gridDim.x, grp, row, et, smem, s_abort, take);
        if (!ok && lane == 0) { *s_abort = 1u; atomicCAS(p.error, 0u, 4u); }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(2u * B200_TC_ACC_COLS) : "memory");
#endif
}

#endif
