/*
 * api.cu -- implementation of the C ABI in include/b200sdr.h: context, pinned ingest ring,
 * copy / compute streams, streaming state, batched launches.
 *
 * Reference call shape being replaced (see include/b200sdr.h for the line citations): the
 * superloop polls the class FSM; in RTLSDR_XFER_COMPLETE the 512-byte (or larger) block in
 * `CommItf.buff` is stable until the next URB is submitted.  Here the host driver calls
 * process_samples(block, len, ctx) at that point; the block goes pinned-ring slot -> H2D on the
 * copy stream -> chains on the compute stream, and the caller gets its buffer back at once.
 *
 * No CPU fallback: every result comes from the CUDA kernels in this directory; if CUDA is not
 * usable, b200sdr_create fails.
 */
#include <cuda.h> /* CUtensorMap + the cuTensorMapEncodeTiled prototype; the entry point comes from the runtime, libcuda is not linked */
#include <cuda_runtime.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <vector>

#include "../../include/b200sdr.h"
#include "misc_kernels.cuh"
#include "plan.h"
#include "render.cuh"
#include "exchange.cuh"

namespace {

constexpr uint64_t kStreamSlack = 16384;     /* device stream buffer = ring_slots x slot_bytes + this; the unread
                                                tail carried over a wrap is < 2048 + 400 bytes           */
constexpr uint64_t kWaveBytes = 192ull << 20; /* input bytes per wave of b200sdr_batch_host (two wave buffers)   */

struct AudioFifo {
    float *d_buf = nullptr;   /* device FIFO storage: valid floats are d_buf[head .. head + count)  */
    float *d_spare = nullptr; /* same size; compaction copies into it and swaps (no overlapping)   */
    uint32_t capacity = 0;    /* floats                                                            */
    uint32_t head = 0, count = 0;
};

} // namespace

struct b200sdr_ctx {
    b200sdr_config cfg{};
    int device = 0, sm_count = 148;
    cudaStream_t s_copy = nullptr, s_compute = nullptr, s_d2h = nullptr;
    /* streaming path: one stream per chain (0 spectrum, 1 WBFM, 2 AM, 3 counter).  The chains of a ring slot share
     * nothing but their input bytes, so they run side by side behind the slot's H2D copy; a slot then costs the device
     * the SLOWEST chain instead of their sum (small launches are latency-, not throughput-bound) */
    cudaStream_t s_chain[4] = {nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t ev_chain[4] = {nullptr, nullptr, nullptr, nullptr};
    float *d_partials_stream = nullptr; size_t partials_stream_floats = 0; /* streaming k_spectrum's own workspace ...  */
    uint32_t *d_unit_counter_stream = nullptr;                             /* ... and hand-out counter (it may run next to a batch launch) */
    bool failed = false;     /* sticky: a chain failed after its H2D was enqueued (see commit_slot) */
    uint8_t *d_tc_image = nullptr;  /* tensor-core FIR engine (wbfm_tc.cuh): the B operand as it lies in shared memory ... */
    uint32_t *d_tc_error = nullptr; /* ... and the word its bounded waits report a protocol error in                      */
    bool tc_launched = false;       /* a k_wbfm_tc launch since the last check of d_tc_error                              */
    cudaEvent_t ev_t0 = nullptr, ev_t1 = nullptr;
    uint64_t launches = 0;
    char err[256] = {0};

    /* constants on the device */
    float *d_window[3] = {nullptr, nullptr, nullptr};
    unsigned long long *d_counter_res = nullptr; /* K0 results: [n] break counts, [n] first breaks */
    uint32_t counter_res_cap = 0;
    CounterStreamState *d_cnt_state = nullptr; /* streaming K0: totals + the byte the next block must start with */
    uint64_t cnt_bytes = 0;                    /* stream bytes already checked (absolute index of the next block) */
    float2 *d_twiddle = nullptr;
    float *d_lut = nullptr;
    float *d_thresholds = nullptr;
    std::vector<float> h_taps[5];
    std::vector<float> h_window[3];

    /* workspaces (grown on demand) */
    float *d_partials = nullptr; size_t partials_floats = 0;
    uint32_t *d_unit_counter = nullptr; /* k_spectrum: dynamic hand-out of work units (two words, self-resetting) */
    float *d_env = nullptr; size_t env_floats = 0;
    float *d_res_spec = nullptr, *d_res_fm = nullptr, *d_res_am = nullptr; /* batch_host result staging */
    size_t res_spec_floats = 0, res_fm_floats = 0, res_am_floats = 0;
    uint8_t *d_wave[2] = {nullptr, nullptr}; size_t wave_bytes = 0;
    cudaEvent_t ev_wave_copied[2] = {nullptr, nullptr}, ev_wave_done[2] = {nullptr, nullptr}, ev_wave_out[2] = {nullptr, nullptr};

    /* ingest ring */
    uint8_t *h_ring = nullptr;          /* pinned: ring_slots x slot_bytes                          */
    /* device side of the ring: ONE linear stream buffer.  Every submitted slot is copied behind the
     * previous one, each chain keeps its own read offset, so the kernels see [leftover | new block]
     * contiguously without any device-to-device copy; at the end of the buffer the small unread tail is
     * moved to the front (once per ring_slots submits). */
    uint8_t *d_stream = nullptr;
    uint64_t stream_cap = 0, wpos = 0, spec_off = 0, fm_off = 0, am_off = 0, last_pos = 0;
    cudaEvent_t ev_wrapped = nullptr;
    std::vector<cudaEvent_t> ev_copied;   /* H2D of slot done (pinned slot reusable)                */
    std::vector<uint8_t> slot_used;
    uint32_t ring_head = 0;
    bool slot_acquired = false;
    uint32_t pending = 0;               /* bytes appended to slot ring_head, not yet submitted      */
    uint32_t submit_bytes = 0;          /* submit the open slot once this many bytes are pending    */
    uint64_t bytes_in = 0, blocks_in = 0, busy_returns = 0, submits = 0;
    uint32_t last_len = 0, last_off = 0;

    /* streaming: spectrum */
    float *d_spec_acc = nullptr;    /* running sum (mean) or EMA state, 1024 floats                 */
    uint64_t spec_frames = 0;
    /* streaming: WBFM */
    uint64_t fm_chunks = 0;
    FmState *d_fm_state = nullptr;  /* two FmState: a launch reads [cur] and writes [cur ^ 1] (its segments run concurrently) */
    int fm_state_cur = 0; AudioFifo fm_fifo;
    /* streaming: AM */
    uint64_t am_chunks = 0;
    AmFrontState *d_amf_state = nullptr; /* two, ping-pong like d_fm_state */
    int amf_state_cur = 0;
    AmBackState *d_amb_state = nullptr; AudioFifo am_fifo;
    float *d_am_env_stream = nullptr;
    uint32_t am_env_cap = 0;

    /* split-capture exchange (K6): own mailbox, the peers' mailboxes as mapped here, call counter */
    float *d_mailbox = nullptr;
    uint32_t *d_xchg_status = nullptr; /* pinned, mapped: the kernel raises it, the host reads it without a copy */
    float *peer_mail[B200_XCHG_MAX_WORLD] = {nullptr};
    bool peer_is_ipc[B200_XCHG_MAX_WORLD] = {false};
    uint32_t xchg_world = 0, xchg_rank = 0, xchg_seq = 0;
    bool xchg_connected = false;
};

namespace {

int fail(b200sdr_ctx *c, int code, const char *what, cudaError_t e = cudaSuccess)
{
    if (c) {
        if (e != cudaSuccess) snprintf(c->err, sizeof c->err, "%s: %s", what, cudaGetErrorString(e));
        else snprintf(c->err, sizeof c->err, "%s", what);
    }
    return code;
}

#define CU(call)                                                                      \
    do {                                                                              \
        cudaError_t e_ = (call);                                                      \
        if (e_ != cudaSuccess) return fail(ctx, B200SDR_FAIL, #call, e_);             \
    } while (0)

struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev) { cudaGetDevice(&prev); if (prev != dev) cudaSetDevice(dev); else prev = -1; }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

int ensure_floats(b200sdr_ctx *ctx, float **p, size_t *have, size_t want)
{
    if (*have >= want) return B200SDR_OK;
    if (*p) { CU(cudaStreamSynchronize(ctx->s_compute)); CU(cudaFree(*p)); *p = nullptr; *have = 0; }
    CU(cudaMalloc((void **)p, want * sizeof(float)));
    *have = want;
    return B200SDR_OK;
}

/* ---- launches --------------------------------------------------------------------------- */
int launch_spectrum(b200sdr_ctx *ctx, const uint8_t *iq_dev, uint32_t n_captures, uint64_t stride, uint64_t len_bytes,
                    bool ema, const float *carry, float carry_scale, float scale_override, bool use_scale_override,
                    float *out_dev, bool finalize = true, bool streaming = false)
{
    b200::SpectrumPlan pl = b200::plan_spectrum(len_bytes, n_captures, (uint32_t)ctx->sm_count);
    if (pl.frames == 0) return B200SDR_OK;
    if (pl.total_units > 0xffffffffull) return fail(ctx, B200SDR_NOT_SUPPORTED, "batch too large (32-bit work-unit index)");
    cudaStream_t stream = streaming ? ctx->s_chain[0] : ctx->s_compute;
    float **partials = streaming ? &ctx->d_partials_stream : &ctx->d_partials;
    size_t *partials_cap = streaming ? &ctx->partials_stream_floats : &ctx->partials_floats;
    if (*partials_cap < (size_t)pl.total_units * 1024 && *partials) CU(cudaStreamSynchronize(stream));
    int rc = ensure_floats(ctx, partials, partials_cap, (size_t)pl.total_units * 1024);
    if (rc) return rc;
    float scale = ema ? 1.0f : 1.0f / (float)pl.frames;
    if (use_scale_override) scale = scale_override;
    /* short single captures (ring slots): the last CTA finalizes, one launch less */
    const bool fold = finalize && n_captures == 1 && pl.total_units <= 128;
    SpectrumParams p{};
    p.iq = iq_dev;
    p.capture_stride = stride;
    p.frames = pl.frames;
    p.frames_per_warp = pl.frames_per_warp;
    p.window = ctx->d_window[ctx->cfg.window];
    p.twiddle = ctx->d_twiddle;
    p.partials = *partials;
    p.units_per_capture = pl.units_per_capture;
    p.total_units = (uint32_t)pl.total_units;
    p.unit_counter = streaming ? ctx->d_unit_counter_stream : ctx->d_unit_counter;
    p.ema_beta = ctx->cfg.ema_beta;
    p.ema_log2_decay = log2f(1.0f - ctx->cfg.ema_beta);
    if (fold) { p.final_out = out_dev; p.carry = carry; p.carry_scale = carry_scale; p.final_scale = scale; }
    dim3 grid(pl.grid);
    if (ema) k_spectrum<true><<<grid, B200_SPEC_THREADS, B200_SPEC_SMEM_BYTES, stream>>>(p);
    else k_spectrum<false><<<grid, B200_SPEC_THREADS, B200_SPEC_SMEM_BYTES, stream>>>(p);
    CU(cudaGetLastError());
    ctx->launches += 1;
    if (!finalize || fold) return B200SDR_OK; /* !finalize: the caller reduces ctx->d_partials itself (split-capture exchange) */
    k_spectrum_finalize<<<dim3(4, n_captures), 256, 0, stream>>>(*partials, pl.units_per_capture, scale,
                                                                 carry, carry_scale, out_dev);
    CU(cudaGetLastError());
    ctx->launches += 1;
    return B200SDR_OK;
}

/* the driver's tensor-map encoder through the runtime (no -lcuda) */
typedef CUresult (*tensor_map_encode_fn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                         const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                         CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
tensor_map_encode_fn tensor_map_encoder()
{
    static const tensor_map_encode_fn fn = [] {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q = cudaDriverEntryPointSymbolNotFound;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) p = nullptr;
        return (tensor_map_encode_fn)p;
    }();
    return fn;
}
/* The batch as TMA sees it: (320 bytes, rows of a capture, captures), u8, boxes of 64 bytes x 125 rows, 64B swizzle.
 * Only whole rows are inside the tensor, so everything outside a capture reads as zero.  false: use the cp.async path. */
bool make_tc_tensor_map(CUtensorMap *map, const uint8_t *iq_dev, uint32_t n_captures, uint64_t len_bytes)
{
    memset(map, 0, sizeof *map);
    const tensor_map_encode_fn enc = tensor_map_encoder();
    const uint64_t rows = len_bytes / B200_TC_ROW_BYTES;
    if (!enc || rows == 0) return false;
    const cuuint64_t dims[3] = {B200_TC_ROW_BYTES, rows, n_captures};
    const cuuint64_t strides[2] = {B200_TC_ROW_BYTES, len_bytes};
    const cuuint32_t box[3] = {64, B200_TC_ROWS, 1}, elem[3] = {1, 1, 1};
    return enc(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, (void *)iq_dev, dims, strides, box, elem, CU_TENSOR_MAP_INTERLEAVE_NONE,
               CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

/* cfg.fir_engine = TENSOR: stage 1 on the tensor cores (wbfm_tc.cuh); `dbg_acc` = optional raw accumulators (tests) */
int launch_wbfm_tc_batch(b200sdr_ctx *ctx, const uint8_t *iq_dev, uint32_t n_captures, uint64_t len_bytes, float *audio,
                         float *disc, int32_t *dbg_acc = nullptr)
{
    b200::FmTcPlan pl = b200::plan_wbfm_tc(len_bytes, n_captures, (uint32_t)ctx->sm_count);
    if (pl.n_tiles == 0) return B200SDR_OK;
    FmTcParams p{};
    p.iq = iq_dev;
    p.capture_stride = len_bytes;
    p.capture_bytes = len_bytes;
    p.m1 = pl.m1;
    p.n_tiles = pl.n_tiles;
    p.total_rows = pl.total_rows;
    p.tiles_per_segment = pl.tiles_per_segment;
    p.segments = pl.segments;
    p.n_captures = n_captures;
    p.audio = audio;
    p.audio_stride = b200::wbfm_audio_len(len_bytes);
    p.disc = disc;
    p.disc_stride = pl.m1;
    p.b_image = ctx->d_tc_image;
    p.error = ctx->d_tc_error;
    p.dbg_acc = dbg_acc;
    /* TMA for every tile made of whole rows; the tile with a capture's ragged last row (length not a multiple of 320
     * bytes) is filled with bounds-checked cp.async by the same kernel */
    alignas(64) CUtensorMap tmap;
    const bool have_map = make_tc_tensor_map(&tmap, iq_dev, n_captures, len_bytes);
    const uint64_t whole_rows = len_bytes / B200_TC_ROW_BYTES;
    p.manual_from_tile = !have_map ? 0u : (len_bytes % B200_TC_ROW_BYTES ? (uint32_t)(whole_rows / B200_TC_ROWS) : pl.n_tiles);
    k_wbfm_tc<<<dim3(pl.grid), B200_TC_THREADS, B200_TC_SMEM_BYTES, ctx->s_compute>>>(p, tmap);
    CU(cudaGetLastError());
    ctx->launches += 1;
    ctx->tc_launched = true;
    return B200SDR_OK;
}
/* after the compute stream has been synchronised: did a bounded wait of k_wbfm_tc expire? */
int check_tc_error(b200sdr_ctx *ctx)
{
    if (!ctx->tc_launched) return B200SDR_OK;
    ctx->tc_launched = false;
    uint32_t code = 0;
    CU(cudaMemcpy(&code, ctx->d_tc_error, sizeof code, cudaMemcpyDeviceToHost));
    if (code == 0) return B200SDR_OK;
    CU(cudaMemset(ctx->d_tc_error, 0, sizeof code));
    char msg[96];
    snprintf(msg, sizeof msg, "k_wbfm_tc: pipeline wait expired (role %u); results of that launch are invalid", code);
    return fail(ctx, B200SDR_FAIL, msg);
}

int launch_wbfm_batch(b200sdr_ctx *ctx, const uint8_t *iq_dev, uint32_t n_captures, uint64_t len_bytes, float *audio,
                      float *disc)
{
    if (ctx->cfg.fir_engine == B200SDR_FIR_ENGINE_TENSOR) return launch_wbfm_tc_batch(ctx, iq_dev, n_captures, len_bytes, audio, disc);
    b200::FmPlan pl = b200::plan_wbfm_batch(len_bytes, n_captures, (uint32_t)ctx->sm_count);
    if (pl.n_tiles == 0) return B200SDR_OK;
    FmParams p{};
    p.iq = iq_dev;
    p.capture_stride = len_bytes;
    p.capture_bytes = len_bytes;
    p.m1 = pl.m1;
    p.n_tiles = pl.n_tiles;
    p.total_chunks = pl.total_chunks;
    p.tiles_per_segment = pl.tiles_per_segment;
    p.audio = audio;
    p.audio_stride = b200::wbfm_audio_len(len_bytes);
    p.disc = disc;
    p.disc_stride = pl.m1;
    k_wbfm<<<dim3(pl.segments, n_captures), B200_FM_THREADS, B200_FM_SMEM_BYTES, ctx->s_compute>>>(p);
    CU(cudaGetLastError());
    ctx->launches += 1;
    return B200SDR_OK;
}

int launch_am_batch(b200sdr_ctx *ctx, const uint8_t *iq_dev, uint32_t n_captures, uint64_t len_bytes, float *audio)
{
    b200::AmPlan pl = b200::plan_am_batch(len_bytes, n_captures, (uint32_t)ctx->sm_count);
    if (pl.n_tiles == 0) return B200SDR_OK;
    int rc = ensure_floats(ctx, &ctx->d_env, &ctx->env_floats, (size_t)n_captures * pl.q_count);
    if (rc) return rc;
    AmFrontParams p{};
    p.iq = iq_dev;
    p.capture_stride = len_bytes;
    p.capture_bytes = len_bytes;
    p.q_count = pl.q_count;
    p.n_tiles = pl.n_tiles;
    p.total_chunks = pl.total_chunks;
    p.tiles_per_segment = pl.tiles_per_segment;
    p.env = ctx->d_env;
    p.env_stride = pl.q_count;
    k_am_front<<<dim3(pl.segments, n_captures), B200_AM_THREADS, B200_AM_SMEM_BYTES, ctx->s_compute>>>(p);
    CU(cudaGetLastError());
    AmBackParams b{};
    b.env = ctx->d_env;
    b.env_stride = pl.q_count;
    b.q_count = pl.q_count;
    b.audio = audio;
    b.audio_stride = pl.audio_len;
    k_am_back<<<n_captures, B200_AMB_THREADS, 0, ctx->s_compute>>>(b);
    CU(cudaGetLastError());
    ctx->launches += 2;
    return B200SDR_OK;
}

bool aligned16(const void *p) { return ((uintptr_t)p & 15u) == 0; }
int fifo_reserve(b200sdr_ctx *ctx, AudioFifo &f, uint32_t n, float **where, cudaStream_t stream);
int join_chains(b200sdr_ctx *ctx);

/* ---- streaming steps: all on the compute stream, after the new bytes are in d_stream[.. wpos) ---- */
int stream_spectrum(b200sdr_ctx *ctx)
{
    const uint64_t have = ctx->wpos - ctx->spec_off;
    const uint64_t frames = b200::spectrum_frames(have);
    if (frames == 0) return B200SDR_OK;
    const bool ema = ctx->cfg.avg_mode == B200SDR_AVG_EMA;
    /* mean: acc += sum |X|^2 ; EMA: acc = (1-beta)^F acc + sum beta (1-beta)^(F-1-m) |X_m|^2 */
    const float carry_scale = ema ? powf(1.0f - ctx->cfg.ema_beta, (float)frames) : 1.0f;
    int rc = launch_spectrum(ctx, ctx->d_stream + ctx->spec_off, 1, 0, have, ema, ctx->d_spec_acc, carry_scale, 1.0f, true,
                             ctx->d_spec_acc, true, true);
    if (rc) return rc;
    ctx->spec_frames += frames;
    ctx->spec_off += frames * 1024u; /* 512 samples x 2 bytes per frame; the 512-sample overlap stays unread */
    return B200SDR_OK;
}

int stream_wbfm(b200sdr_ctx *ctx)
{
    const uint32_t n_chunks = (uint32_t)((ctx->wpos - ctx->fm_off) / (2 * B200_FM_CHUNK));
    if (n_chunks == 0) return B200SDR_OK;
    FmParams p{};
    p.iq = ctx->d_stream + ctx->fm_off; /* 16-byte aligned: offsets move by whole 240-byte chunks and 16-byte wraps */
    p.capture_bytes = (uint64_t)n_chunks * 2 * B200_FM_CHUNK;
    p.m1 = (uint64_t)n_chunks * B200_FM_OPT;
    p.m_base = ctx->fm_chunks * B200_FM_OPT;
    p.total_chunks = n_chunks;
    p.n_tiles = (uint32_t)b200::ceil_div(n_chunks, B200_FM_THREADS);
    /* a block of several tiles is spread over CTAs: segment 0 continues the carried state exactly, the
     * others pre-roll one tile (plan.h), so a 256 KiB block costs 3 tile times instead of 9 */
    p.tiles_per_segment = b200::kFmStreamTilesPerSegment;
    const uint32_t segments = (uint32_t)b200::ceil_div(p.n_tiles, p.tiles_per_segment);
    const uint64_t a0 = b200::ceil_div(p.m_base, B200_FM_D2), a1 = b200::ceil_div(p.m_base + p.m1, B200_FM_D2);
    const uint32_t n_audio = (uint32_t)(a1 - a0);
    int frc = fifo_reserve(ctx, ctx->fm_fifo, n_audio, &p.audio, ctx->s_chain[1]);
    if (frc) return frc;
    p.audio_base = a0;
    p.state = ctx->d_fm_state + ctx->fm_state_cur;
    p.state_out = ctx->d_fm_state + (ctx->fm_state_cur ^ 1);
    ctx->fm_state_cur ^= 1;
    k_wbfm<<<dim3(segments, 1), B200_FM_THREADS, B200_FM_SMEM_BYTES, ctx->s_chain[1]>>>(p);
    CU(cudaGetLastError());
    ctx->launches += 1;
    ctx->fm_fifo.count += n_audio;
    ctx->fm_chunks += n_chunks;
    ctx->fm_off += (uint64_t)n_chunks * 2 * B200_FM_CHUNK;
    return B200SDR_OK;
}

int stream_am(b200sdr_ctx *ctx)
{
    const uint32_t n_chunks = (uint32_t)((ctx->wpos - ctx->am_off) / (2 * B200_AM_CHUNK));
    if (n_chunks == 0) return B200SDR_OK;
    if (n_chunks > ctx->am_env_cap) return fail(ctx, B200SDR_FAIL, "AM envelope workspace too small for the pending stream");
    const uint64_t a0 = (2 * ctx->am_chunks + 2) / 3, a1 = (2 * (ctx->am_chunks + n_chunks) + 2) / 3;
    const uint32_t n_audio = (uint32_t)(a1 - a0);
    float *am_out = nullptr;
    int frc = fifo_reserve(ctx, ctx->am_fifo, n_audio, &am_out, ctx->s_chain[2]);
    if (frc) return frc;
    AmFrontParams p{};
    p.iq = ctx->d_stream + ctx->am_off;
    p.capture_bytes = (uint64_t)n_chunks * 2 * B200_AM_CHUNK;
    p.q_count = n_chunks;
    p.q_base = ctx->am_chunks;
    p.total_chunks = n_chunks;
    p.n_tiles = (uint32_t)b200::ceil_div(n_chunks, B200_AM_THREADS);
    p.tiles_per_segment = b200::kFmStreamTilesPerSegment; /* spread over CTAs like stream_wbfm (FIRs only: exact) */
    const uint32_t segments = (uint32_t)b200::ceil_div(p.n_tiles, p.tiles_per_segment);
    p.env = ctx->d_am_env_stream;
    p.state = ctx->d_amf_state + ctx->amf_state_cur;
    p.state_out = ctx->d_amf_state + (ctx->amf_state_cur ^ 1);
    ctx->amf_state_cur ^= 1;
    k_am_front<<<dim3(segments, 1), B200_AM_THREADS, B200_AM_SMEM_BYTES, ctx->s_chain[2]>>>(p);
    CU(cudaGetLastError());
    AmBackParams b{};
    b.env = ctx->d_am_env_stream;
    b.q_count = n_chunks;
    b.q_base = ctx->am_chunks;
    b.audio = am_out;
    b.audio_base = a0;
    b.state = ctx->d_amb_state;
    k_am_back<<<1, B200_AMB_THREADS, 0, ctx->s_chain[2]>>>(b);
    CU(cudaGetLastError());
    ctx->launches += 2;
    ctx->am_fifo.count += n_audio;
    ctx->am_chunks += n_chunks;
    ctx->am_off += (uint64_t)n_chunks * 2 * B200_AM_CHUNK;
    return B200SDR_OK;
}

int stream_counter(b200sdr_ctx *ctx, uint32_t len)
{
    if (len == 0) return B200SDR_OK;
    CounterParams p{};
    p.in = reinterpret_cast<const uint32_t *>(ctx->d_stream + ctx->last_pos); /* blocks are multiples of 4 bytes */
    p.n_words = len / 4u;
    p.stride_words = p.n_words;
    p.expect_first = -1;
    p.stream = ctx->d_cnt_state;
    p.pos_base = ctx->cnt_bytes;
    k_counter_check<<<dim3((unsigned)b200::ceil_div(b200::ceil_div(p.n_words, 4), 1024), 1), 256, 0, ctx->s_chain[3]>>>(p);
    CU(cudaGetLastError());
    ctx->launches += 1;
    ctx->cnt_bytes += len;
    return B200SDR_OK;
}

int reset_counter_state(b200sdr_ctx *ctx)
{
    static const CounterStreamState init = {0ull, ~0ull, 0xffffffffu, 0u};
    ctx->cnt_bytes = 0;
    CU(cudaMemcpyAsync(ctx->d_cnt_state, &init, sizeof init, cudaMemcpyHostToDevice, ctx->s_compute));
    return B200SDR_OK;
}

int reset_stream_state(b200sdr_ctx *ctx)
{
    ctx->wpos = ctx->spec_off = ctx->fm_off = ctx->am_off = ctx->last_pos = 0;
    ctx->spec_frames = 0;
    ctx->fm_chunks = 0; ctx->fm_fifo.count = 0; ctx->fm_fifo.head = 0;
    ctx->am_chunks = 0; ctx->am_fifo.count = 0; ctx->am_fifo.head = 0;
    CU(cudaMemsetAsync(ctx->d_spec_acc, 0, 1024 * sizeof(float), ctx->s_compute));
    CU(cudaMemsetAsync(ctx->d_fm_state, 0, 2 * sizeof(FmState), ctx->s_compute));
    ctx->fm_state_cur = 0;
    CU(cudaMemsetAsync(ctx->d_amf_state, 0, 2 * sizeof(AmFrontState), ctx->s_compute));
    ctx->amf_state_cur = 0;
    CU(cudaMemsetAsync(ctx->d_amb_state, 0, sizeof(AmBackState), ctx->s_compute));
    int rc = reset_counter_state(ctx);
    if (rc) return rc;
    CU(cudaStreamSynchronize(ctx->s_compute)); /* the chain streams start from the cleared state */
    return B200SDR_OK;
}

const float *synth_lut_host()
{
    /* filled by the constructor of a function-local static: C++11 makes that initialisation thread-safe, so
     * contexts created from several threads at once never see a partly filled table */
    struct Lut {
        float v[B200SDR_SYNTH_LUT_SIZE + 1];
        Lut()
        {
            for (unsigned i = 0; i <= B200SDR_SYNTH_LUT_SIZE; ++i)
                v[i] = (float)sin(2.0 * b200::kPi * (double)(i % B200SDR_SYNTH_LUT_SIZE) / (double)B200SDR_SYNTH_LUT_SIZE);
        }
    };
    static const Lut lut;
    return lut.v;
}

/* end of the stream buffer: move the unread tail (what the slowest enabled chain has not consumed:
 * < 2048 + 400 bytes) to the front and rebase all offsets by a multiple of 16 bytes (TMA alignment) */
int wrap_stream(b200sdr_ctx *ctx)
{
    uint64_t lo = ctx->wpos;
    if ((ctx->cfg.chains & B200SDR_CHAIN_SPECTRUM) && ctx->spec_off < lo) lo = ctx->spec_off;
    if ((ctx->cfg.chains & B200SDR_CHAIN_WBFM) && ctx->fm_off < lo) lo = ctx->fm_off;
    if ((ctx->cfg.chains & B200SDR_CHAIN_AM) && ctx->am_off < lo) lo = ctx->am_off;
    const uint64_t shift = lo & ~(uint64_t)15, tail = ctx->wpos - shift;
    if (shift < tail) return fail(ctx, B200SDR_FAIL, "stream buffer too small for the unread tail");
    /* on the compute stream, behind every chain kernel that read the old data; the H2D copies that follow (copy
     * stream, and through its per-slot events the chain streams) wait for the move */
    int jrc = join_chains(ctx);
    if (jrc) return jrc;
    if (tail) CU(cudaMemcpyAsync(ctx->d_stream, ctx->d_stream + shift, tail, cudaMemcpyDeviceToDevice, ctx->s_compute));
    CU(cudaEventRecord(ctx->ev_wrapped, ctx->s_compute));
    CU(cudaStreamWaitEvent(ctx->s_copy, ctx->ev_wrapped, 0));
    ctx->wpos -= shift;
    ctx->spec_off = ctx->spec_off > shift ? ctx->spec_off - shift : 0;
    ctx->fm_off = ctx->fm_off > shift ? ctx->fm_off - shift : 0;
    ctx->am_off = ctx->am_off > shift ? ctx->am_off - shift : 0;
    ctx->last_pos = ctx->last_pos > shift ? ctx->last_pos - shift : 0;
    return B200SDR_OK;
}

int commit_slot(b200sdr_ctx *ctx, uint32_t slot, uint32_t len)
{
    uint8_t *h_slot = ctx->h_ring + (size_t)slot * ctx->cfg.slot_bytes;
    if (ctx->wpos + len > ctx->stream_cap) {
        int wrc = wrap_stream(ctx);
        if (wrc) return wrc;
    }
    CU(cudaMemcpyAsync(ctx->d_stream + ctx->wpos, h_slot, len, cudaMemcpyHostToDevice, ctx->s_copy));
    /* from here on the pinned slot has a copy in flight: it is marked used and the ring moves on whatever
     * happens below, so the slot is never handed out again before ev_copied says so */
    ctx->slot_used[slot] = 1;
    ctx->ring_head = (slot + 1) % ctx->cfg.ring_slots;
    ctx->submits += 1;
    ctx->last_pos = ctx->wpos;
    ctx->wpos += len;
    int rc = B200SDR_OK;
    cudaError_t e = cudaEventRecord(ctx->ev_copied[slot], ctx->s_copy);
    static const uint32_t chain_bit[4] = {B200SDR_CHAIN_SPECTRUM, B200SDR_CHAIN_WBFM, B200SDR_CHAIN_AM, B200SDR_CHAIN_COUNTER};
    for (int c = 0; c < 4 && e == cudaSuccess; ++c)
        if (ctx->cfg.chains & chain_bit[c]) e = cudaStreamWaitEvent(ctx->s_chain[c], ctx->ev_copied[slot], 0);
    if (e != cudaSuccess) rc = fail(ctx, B200SDR_FAIL, "ring slot hand-over", e);
    if (!rc && (ctx->cfg.chains & B200SDR_CHAIN_SPECTRUM)) rc = stream_spectrum(ctx);
    if (!rc && (ctx->cfg.chains & B200SDR_CHAIN_WBFM)) rc = stream_wbfm(ctx);
    if (!rc && (ctx->cfg.chains & B200SDR_CHAIN_AM)) rc = stream_am(ctx);
    if (!rc && (ctx->cfg.chains & B200SDR_CHAIN_COUNTER)) rc = stream_counter(ctx, len);
    if (rc) {
        /* a chain did not run over bytes that are already part of the stream: the chains' read offsets no
         * longer agree with `wpos`, so the stream is dead until b200sdr_reset() starts a new capture.
         * Sticky: every later streaming call returns B200SDR_FAIL instead of computing on a torn stream. */
        ctx->failed = true;
    }
    return rc;
}

/* submit whatever process_samples has appended to the open slot (no-op when nothing is pending) */
int flush_pending(b200sdr_ctx *ctx)
{
    if (ctx->pending == 0) return B200SDR_OK;
    if (ctx->failed) return fail(ctx, B200SDR_FAIL, "stream failed earlier: call b200sdr_reset");
    const uint32_t n = ctx->pending;
    ctx->pending = 0; /* on failure commit_slot latches ctx->failed: the bytes are never silently dropped */
    return commit_slot(ctx, ctx->ring_head, n);
}

/* would this block overflow an audio FIFO?  checked before anything is enqueued */
bool fifo_room(b200sdr_ctx *ctx, uint32_t len)
{
    if ((ctx->cfg.chains & B200SDR_CHAIN_WBFM) && ctx->fm_fifo.count + len / 100 + 8 > ctx->fm_fifo.capacity) return false;
    if ((ctx->cfg.chains & B200SDR_CHAIN_AM) && ctx->am_fifo.count + len / 600 + 8 > ctx->am_fifo.capacity) return false;
    return true;
}

/* is the pinned slot free (its previous H2D finished)? */
int slot_ready(b200sdr_ctx *ctx, uint32_t slot)
{
    if (!ctx->slot_used[slot]) return B200SDR_OK;
    cudaError_t q = cudaEventQuery(ctx->ev_copied[slot]);
    if (q == cudaSuccess) return B200SDR_OK;
    if (q == cudaErrorNotReady) { ctx->busy_returns++; return B200SDR_BUSY; }
    return fail(ctx, B200SDR_FAIL, "cudaEventQuery", q);
}

/* dB thresholds of the 272 LCD rows: T[h] = 10^((db_min + (db_max - db_min) h / 271) / 10) */
int upload_thresholds(b200sdr_ctx *ctx, float db_min, float db_max)
{
    float thr[B200_LCD_H];
    b200_fill_thresholds(thr, db_min, db_max);
    if (!ctx->d_thresholds) CU(cudaMalloc((void **)&ctx->d_thresholds, sizeof thr));
    CU(cudaMemcpyAsync(ctx->d_thresholds, thr, sizeof thr, cudaMemcpyHostToDevice, ctx->s_compute));
    CU(cudaStreamSynchronize(ctx->s_compute)); /* `thr` is a stack buffer */
    return B200SDR_OK;
}

/* contiguous room for n more floats behind the queued ones (compacting if the tail is used up) */
/* every chain stream -> the compute stream: after this, whatever is enqueued on (or synchronised through) s_compute
 * comes after all streaming kernels submitted so far */
int join_chains(b200sdr_ctx *ctx)
{
    for (int c = 0; c < 4; ++c) {
        CU(cudaEventRecord(ctx->ev_chain[c], ctx->s_chain[c]));
        CU(cudaStreamWaitEvent(ctx->s_compute, ctx->ev_chain[c], 0));
    }
    return B200SDR_OK;
}

int fifo_reserve(b200sdr_ctx *ctx, AudioFifo &f, uint32_t n, float **where, cudaStream_t stream)
{
    if (f.count + n > f.capacity) return fail(ctx, B200SDR_FAIL, "audio FIFO overflow");
    if (f.head + f.count + n > f.capacity) {
        CU(cudaMemcpyAsync(f.d_spare, f.d_buf + f.head, (size_t)f.count * sizeof(float), cudaMemcpyDeviceToDevice, stream));
        float *t = f.d_buf; f.d_buf = f.d_spare; f.d_spare = t;
        f.head = 0;
    }
    *where = f.d_buf + f.head + f.count;
    return B200SDR_OK;
}

int pop_fifo(b200sdr_ctx *ctx, AudioFifo &f, float *out, uint32_t capacity, uint32_t *n_out)
{
    int jrc = join_chains(ctx);
    if (jrc) return jrc;
    CU(cudaStreamSynchronize(ctx->s_compute));
    const uint32_t n = f.count < capacity ? f.count : capacity;
    if (n) CU(cudaMemcpy(out, f.d_buf + f.head, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost));
    f.count -= n;
    f.head = f.count ? f.head + n : 0;
    if (n_out) *n_out = n;
    return B200SDR_OK;
}

} // namespace

/* ============================================================================================ */
extern "C" {

const char *b200sdr_version(void) { return "b200sdr 0.1 (sm_100a)"; }

void b200sdr_default_config(b200sdr_config *cfg)
{
    if (!cfg) return;
    memset(cfg, 0, sizeof *cfg);
    cfg->struct_size = (uint32_t)sizeof *cfg;
    cfg->device = 0;
    cfg->chains = B200SDR_CHAIN_SPECTRUM | B200SDR_CHAIN_WBFM | B200SDR_CHAIN_AM;
    cfg->window = B200SDR_WINDOW_HANN;
    cfg->avg_mode = B200SDR_AVG_MEAN;
    cfg->ema_beta = 0.1f;
    cfg->ring_slots = 8;
    cfg->slot_bytes = 262144; /* DEFAULT_BUF_LENGTH, RTL/Inc/usbh_rtlsdr.h:277-278 */
    cfg->audio_capacity = 1u << 20;
}

int32_t b200sdr_create(const b200sdr_config *cfg_in, b200sdr_ctx **out_ctx)
{
    if (!cfg_in || !out_ctx) return B200SDR_FAIL;
    *out_ctx = nullptr;
    b200sdr_config cfg = *cfg_in;
    if (cfg.struct_size != sizeof(b200sdr_config)) return B200SDR_NOT_SUPPORTED;
    if (cfg.window > B200SDR_WINDOW_BLACKMAN || cfg.avg_mode > B200SDR_AVG_EMA) return B200SDR_NOT_SUPPORTED;
    if (cfg.ring_slots < 2 || cfg.ring_slots > 1024) return B200SDR_NOT_SUPPORTED;
    if (cfg.slot_bytes < 4 || (cfg.slot_bytes & 3u)) return B200SDR_NOT_SUPPORTED; /* multiple-of-4 rule */
    if (cfg.avg_mode == B200SDR_AVG_EMA && !(cfg.ema_beta > 0.0f && cfg.ema_beta < 1.0f)) return B200SDR_NOT_SUPPORTED;
    if (cfg.audio_capacity < 4096) cfg.audio_capacity = 4096;
    /* one full slot must fit an EMPTY FIFO, or process_samples would answer BUSY for ever (fifo_room) */
    if ((cfg.chains & B200SDR_CHAIN_WBFM) && cfg.audio_capacity < cfg.slot_bytes / 100 + 16) cfg.audio_capacity = cfg.slot_bytes / 100 + 16;
    if ((cfg.chains & B200SDR_CHAIN_AM) && cfg.audio_capacity < cfg.slot_bytes / 600 + 16) cfg.audio_capacity = cfg.slot_bytes / 600 + 16;
    if (cfg.submit_bytes > cfg.slot_bytes) return B200SDR_NOT_SUPPORTED;
    if (cfg.fir_engine > B200SDR_FIR_ENGINE_TENSOR) return B200SDR_NOT_SUPPORTED;

    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev <= 0 || cfg.device < 0 || cfg.device >= n_dev)
        return B200SDR_FAIL; /* no CUDA device: there is no CPU path */
    b200sdr_ctx *ctx = new (std::nothrow) b200sdr_ctx();
    if (!ctx) return B200SDR_FAIL;
    ctx->cfg = cfg;
    ctx->device = cfg.device;
    ctx->submit_bytes = cfg.submit_bytes ? cfg.submit_bytes : cfg.slot_bytes;
    DeviceGuard guard(ctx->device);
#define CK(call)                                                                               \
    do {                                                                                       \
        cudaError_t e_ = (call);                                                               \
        if (e_ != cudaSuccess) {                                                               \
            fprintf(stderr, "b200sdr_create: %s: %s\n", #call, cudaGetErrorString(e_));        \
            b200sdr_destroy(ctx);                                                              \
            return B200SDR_FAIL;                                                               \
        }                                                                                      \
    } while (0)
    try { /* std::vector growth below may throw; nothing may unwind through the C boundary */
    cudaDeviceProp prop{};
    CK(cudaGetDeviceProperties(&prop, ctx->device));
    if (prop.major < 10) {
        fprintf(stderr, "b200sdr_create: device is sm_%d%d; this library is built for sm_100a only\n", prop.major, prop.minor);
        b200sdr_destroy(ctx);
        return B200SDR_FAIL;
    }
    ctx->sm_count = prop.multiProcessorCount;
    CK(cudaStreamCreateWithFlags(&ctx->s_copy, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&ctx->s_compute, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&ctx->s_d2h, cudaStreamNonBlocking));
    for (int c = 0; c < 4; ++c) {
        CK(cudaStreamCreateWithFlags(&ctx->s_chain[c], cudaStreamNonBlocking));
        CK(cudaEventCreateWithFlags(&ctx->ev_chain[c], cudaEventDisableTiming));
    }
    CK(cudaEventCreate(&ctx->ev_t0));
    CK(cudaEventCreate(&ctx->ev_t1));
    for (int i = 0; i < 2; ++i) {
        CK(cudaEventCreateWithFlags(&ctx->ev_wave_copied[i], cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&ctx->ev_wave_done[i], cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&ctx->ev_wave_out[i], cudaEventDisableTiming));
    }
    CK(cudaFuncSetAttribute(k_spectrum<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, B200_SPEC_SMEM_BYTES));
    CK(cudaFuncSetAttribute(k_spectrum<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, B200_SPEC_SMEM_BYTES));
    CK(cudaFuncSetAttribute(k_wbfm, cudaFuncAttributeMaxDynamicSharedMemorySize, B200_FM_SMEM_BYTES));
    CK(cudaFuncSetAttribute(k_wbfm_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, B200_TC_SMEM_BYTES));
    CK(cudaFuncSetAttribute(k_am_front, cudaFuncAttributeMaxDynamicSharedMemorySize, B200_AM_SMEM_BYTES));

    /* constants */
    for (unsigned w = 0; w < 3; ++w) {
        ctx->h_window[w] = b200::make_window(w, 1024);
        CK(cudaMalloc((void **)&ctx->d_window[w], 1024 * sizeof(float)));
        CK(cudaMemcpy(ctx->d_window[w], ctx->h_window[w].data(), 1024 * sizeof(float), cudaMemcpyHostToDevice));
    }
    {
        std::vector<float2> tw(1024);
        b200::fill_twiddles(tw.data());
        CK(cudaMalloc((void **)&ctx->d_twiddle, 1024 * sizeof(float2)));
        CK(cudaMemcpy(ctx->d_twiddle, tw.data(), 1024 * sizeof(float2), cudaMemcpyHostToDevice));
        CK(cudaMalloc((void **)&ctx->d_lut, (B200SDR_SYNTH_LUT_SIZE + 1) * sizeof(float)));
        CK(cudaMemcpy(ctx->d_lut, synth_lut_host(), (B200SDR_SYNTH_LUT_SIZE + 1) * sizeof(float), cudaMemcpyHostToDevice));
        FmTaps ft{};
        b200::fill_fm_taps(ft);
        CK(cudaMemcpyToSymbol(c_fm_taps, &ft, sizeof ft));
        {
            FmTcConsts tc{};
            std::vector<uint8_t> image(B200_TC_B_BYTES);
            b200::fill_fm_tc(tc, image.data());
            CK(cudaMemcpyToSymbol(c_fm_tc, &tc, sizeof tc));
            CK(cudaMalloc((void **)&ctx->d_tc_image, B200_TC_B_BYTES));
            CK(cudaMemcpy(ctx->d_tc_image, image.data(), B200_TC_B_BYTES, cudaMemcpyHostToDevice));
            CK(cudaMalloc((void **)&ctx->d_tc_error, sizeof(uint32_t)));
            CK(cudaMemset(ctx->d_tc_error, 0, sizeof(uint32_t)));
        }
        AmTaps at{};
        b200::fill_am_taps(at);
        CK(cudaMemcpyToSymbol(c_am_taps, &at, sizeof at));
        /* the raw-byte FIR form (cplx2.cuh form C) multiplies by tap * 2^133: must stay finite */
        bool scaled_ok = true;
        for (float v : ft.h1s) scaled_ok = scaled_ok && std::isfinite(v);
        for (float v : at.g1s) scaled_ok = scaled_ok && std::isfinite(v);
        if (!scaled_ok) {
            fprintf(stderr, "b200sdr_create: a stage-1 FIR tap overflows when scaled by 2^%d\n", B200_U8RAW_LOG2);
            b200sdr_destroy(ctx);
            return B200SDR_FAIL;
        }
        for (unsigned t = 0; t < 5; ++t) {
            std::vector<double> h = b200::design_taps(t);
            ctx->h_taps[t].assign(h.begin(), h.end());
        }
    }
    /* ingest ring + streaming buffers */
    const size_t ring_bytes = (size_t)cfg.ring_slots * cfg.slot_bytes;
    CK(cudaHostAlloc((void **)&ctx->h_ring, ring_bytes, cudaHostAllocDefault));
    ctx->stream_cap = (uint64_t)ring_bytes + kStreamSlack;
    CK(cudaMalloc((void **)&ctx->d_stream, ctx->stream_cap));
    CK(cudaEventCreateWithFlags(&ctx->ev_wrapped, cudaEventDisableTiming));
    ctx->ev_copied.resize(cfg.ring_slots);
    ctx->slot_used.assign(cfg.ring_slots, 0);
    for (uint32_t i = 0; i < cfg.ring_slots; ++i) {
        CK(cudaEventCreateWithFlags(&ctx->ev_copied[i], cudaEventDisableTiming));
    }
    CK(cudaMalloc((void **)&ctx->d_spec_acc, 1024 * sizeof(float)));
    CK(cudaMalloc((void **)&ctx->d_unit_counter, 2 * sizeof(uint32_t)));
    CK(cudaMemset(ctx->d_unit_counter, 0, 2 * sizeof(uint32_t)));
    CK(cudaMalloc((void **)&ctx->d_unit_counter_stream, 2 * sizeof(uint32_t)));
    CK(cudaMemset(ctx->d_unit_counter_stream, 0, 2 * sizeof(uint32_t)));
    CK(cudaMalloc((void **)&ctx->d_cnt_state, sizeof(CounterStreamState)));
    CK(cudaMalloc((void **)&ctx->d_fm_state, 2 * sizeof(FmState)));
    CK(cudaMalloc((void **)&ctx->d_amf_state, 2 * sizeof(AmFrontState)));
    CK(cudaMalloc((void **)&ctx->d_amb_state, sizeof(AmBackState)));
    /* one envelope sample per 400-byte chunk of whatever a launch can see: sized from the whole stream buffer */
    ctx->am_env_cap = (uint32_t)(ctx->stream_cap / (2 * B200_AM_CHUNK) + 8);
    CK(cudaMalloc((void **)&ctx->d_am_env_stream, (size_t)ctx->am_env_cap * sizeof(float)));
    ctx->fm_fifo.capacity = cfg.audio_capacity;
    ctx->am_fifo.capacity = cfg.audio_capacity;
    CK(cudaMalloc((void **)&ctx->fm_fifo.d_buf, (size_t)cfg.audio_capacity * sizeof(float)));
    CK(cudaMalloc((void **)&ctx->am_fifo.d_buf, (size_t)cfg.audio_capacity * sizeof(float)));
    CK(cudaMalloc((void **)&ctx->fm_fifo.d_spare, (size_t)cfg.audio_capacity * sizeof(float)));
    CK(cudaMalloc((void **)&ctx->am_fifo.d_spare, (size_t)cfg.audio_capacity * sizeof(float)));
    if (reset_stream_state(ctx) != B200SDR_OK) { b200sdr_destroy(ctx); return B200SDR_FAIL; }
    CK(cudaStreamSynchronize(ctx->s_compute));
    } catch (...) {
        fprintf(stderr, "b200sdr_create: out of host memory\n");
        b200sdr_destroy(ctx);
        return B200SDR_FAIL;
    }
#undef CK
    *out_ctx = ctx;
    return B200SDR_OK;
}

int32_t b200sdr_destroy(b200sdr_ctx *ctx)
{
    if (!ctx) return B200SDR_FAIL;
    DeviceGuard guard(ctx->device);
    cudaDeviceSynchronize();
    if (ctx->d_mailbox) b200sdr_exchange_destroy(ctx);
    for (auto e : ctx->ev_copied) if (e) cudaEventDestroy(e);
    if (ctx->ev_wrapped) cudaEventDestroy(ctx->ev_wrapped);
    for (int i = 0; i < 2; ++i) {
        if (ctx->ev_wave_copied[i]) cudaEventDestroy(ctx->ev_wave_copied[i]);
        if (ctx->ev_wave_done[i]) cudaEventDestroy(ctx->ev_wave_done[i]);
        if (ctx->ev_wave_out[i]) cudaEventDestroy(ctx->ev_wave_out[i]);
        if (ctx->d_wave[i]) cudaFree(ctx->d_wave[i]);
    }
    if (ctx->ev_t0) cudaEventDestroy(ctx->ev_t0);
    if (ctx->ev_t1) cudaEventDestroy(ctx->ev_t1);
    if (ctx->h_ring) cudaFreeHost(ctx->h_ring);
    void *dev_ptrs[] = {ctx->d_stream, ctx->d_spec_acc, ctx->d_unit_counter, ctx->d_unit_counter_stream, ctx->d_partials_stream, ctx->d_tc_image, ctx->d_tc_error,
                        ctx->d_fm_state, ctx->d_amf_state, ctx->d_amb_state, ctx->d_am_env_stream, ctx->fm_fifo.d_buf,
                        ctx->am_fifo.d_buf, ctx->fm_fifo.d_spare, ctx->am_fifo.d_spare, ctx->d_window[0], ctx->d_window[1], ctx->d_window[2], ctx->d_twiddle,
                        ctx->d_lut, ctx->d_partials, ctx->d_env, ctx->d_thresholds, ctx->d_res_spec, ctx->d_res_fm,
                        ctx->d_res_am, ctx->d_counter_res, ctx->d_cnt_state};
    for (void *p : dev_ptrs) if (p) cudaFree(p);
    if (ctx->s_copy) cudaStreamDestroy(ctx->s_copy);
    if (ctx->s_compute) cudaStreamDestroy(ctx->s_compute);
    if (ctx->s_d2h) cudaStreamDestroy(ctx->s_d2h);
    for (int c = 0; c < 4; ++c) {
        if (ctx->s_chain[c]) cudaStreamDestroy(ctx->s_chain[c]);
        if (ctx->ev_chain[c]) cudaEventDestroy(ctx->ev_chain[c]);
    }
    delete ctx;
    return B200SDR_OK;
}

/* ---- streaming ---------------------------------------------------------------------------- */
int32_t process_samples(const uint8_t *iq, uint32_t len, void *vctx)
{
    b200sdr_ctx *ctx = (b200sdr_ctx *)vctx;
    if (!ctx || !iq) return B200SDR_FAIL;
    if (len == 0) return B200SDR_OK;
    if ((len & 3u) || len > ctx->cfg.slot_bytes) return fail(ctx, B200SDR_NOT_SUPPORTED, "len must be a multiple of 4 and <= slot_bytes");
    if (ctx->slot_acquired) return fail(ctx, B200SDR_FAIL, "a ring slot is acquired; commit it first");
    if (ctx->failed) return fail(ctx, B200SDR_FAIL, "stream failed earlier: call b200sdr_reset");
    DeviceGuard guard(ctx->device);
    /* blocks are appended to the open pinned slot; the slot is submitted (one H2D + one pass of the
     * chains) once cfg.submit_bytes are pending or the next block would not fit */
    if (ctx->pending + len > ctx->cfg.slot_bytes) {
        int rc = flush_pending(ctx);
        if (rc) return rc;
    }
    if (!fifo_room(ctx, ctx->pending + len)) { ctx->busy_returns++; return fail(ctx, B200SDR_BUSY, "audio FIFO full: call b200sdr_get_audio"); }
    const uint32_t slot = ctx->ring_head;
    if (ctx->pending == 0) { /* opening a slot: its previous H2D must have finished */
        int rc = slot_ready(ctx, slot);
        if (rc) return rc;
    }
    memcpy(ctx->h_ring + (size_t)slot * ctx->cfg.slot_bytes + ctx->pending, iq, len);
    ctx->last_off = ctx->pending;
    ctx->last_len = len;
    ctx->pending += len;
    ctx->bytes_in += len;
    ctx->blocks_in += 1;
    if (ctx->pending >= ctx->submit_bytes) return flush_pending(ctx);
    return B200SDR_OK;
}

int32_t b200sdr_ring_acquire(b200sdr_ctx *ctx, uint8_t **slot_ptr, uint32_t *slot_bytes)
{
    if (!ctx || !slot_ptr) return B200SDR_FAIL;
    if (ctx->slot_acquired) return fail(ctx, B200SDR_FAIL, "slot already acquired");
    if (ctx->failed) return fail(ctx, B200SDR_FAIL, "stream failed earlier: call b200sdr_reset");
    DeviceGuard guard(ctx->device);
    int rc = flush_pending(ctx); /* keep stream order: blocks appended by process_samples go first */
    if (rc) return rc;
    const uint32_t slot = ctx->ring_head;
    rc = slot_ready(ctx, slot);
    if (rc) return rc;
    *slot_ptr = ctx->h_ring + (size_t)slot * ctx->cfg.slot_bytes;
    if (slot_bytes) *slot_bytes = ctx->cfg.slot_bytes;
    ctx->slot_acquired = true;
    return B200SDR_OK;
}

int32_t b200sdr_ring_commit(b200sdr_ctx *ctx, uint32_t len)
{
    if (!ctx) return B200SDR_FAIL;
    if (!ctx->slot_acquired) return fail(ctx, B200SDR_FAIL, "no slot acquired");
    if ((len & 3u) || len > ctx->cfg.slot_bytes) return fail(ctx, B200SDR_NOT_SUPPORTED, "len must be a multiple of 4 and <= slot_bytes");
    if (ctx->failed) { ctx->slot_acquired = false; return fail(ctx, B200SDR_FAIL, "stream failed earlier: call b200sdr_reset"); }
    if (!fifo_room(ctx, len)) { ctx->busy_returns++; return fail(ctx, B200SDR_BUSY, "audio FIFO full: call b200sdr_get_audio"); }
    ctx->slot_acquired = false;
    if (len == 0) return B200SDR_OK;
    DeviceGuard guard(ctx->device);
    ctx->last_off = 0;
    ctx->last_len = len;
    ctx->bytes_in += len;
    ctx->blocks_in += 1;
    return commit_slot(ctx, ctx->ring_head, len);
}

int32_t b200sdr_sync(b200sdr_ctx *ctx)
{
    if (!ctx) return B200SDR_FAIL;
    DeviceGuard guard(ctx->device);
    if (!ctx->slot_acquired) {
        int rc = flush_pending(ctx);
        if (rc) return rc;
    }
    CU(cudaStreamSynchronize(ctx->s_copy));
    int jrc = join_chains(ctx);
    if (jrc) return jrc;
    CU(cudaStreamSynchronize(ctx->s_compute));
    return check_tc_error(ctx);
}

int32_t b200sdr_reset(b200sdr_ctx *ctx)
{
    if (!ctx) return B200SDR_FAIL;
    DeviceGuard guard(ctx->device);
    ctx->pending = 0; /* blocks not yet submitted belong to the capture being forgotten */
    ctx->failed = false;
    ctx->slot_acquired = false;
    int rc = b200sdr_sync(ctx);
    if (rc) return rc;
    return reset_stream_state(ctx);
}

int32_t b200sdr_get_spectrum(b200sdr_ctx *ctx, float *out1024, uint64_t *n_frames)
{
    if (!ctx || !out1024) return B200SDR_FAIL;
    DeviceGuard guard(ctx->device);
    if (!ctx->slot_acquired) {
        int rc = flush_pending(ctx);
        if (rc) return rc;
    }
    CU(cudaStreamSynchronize(ctx->s_chain[0]));
    CU(cudaMemcpy(out1024, ctx->d_spec_acc, 1024 * sizeof(float), cudaMemcpyDeviceToHost));
    if (ctx->cfg.avg_mode == B200SDR_AVG_MEAN && ctx->spec_frames) {
        const float s = 1.0f / (float)ctx->spec_frames;
        for (int k = 0; k < 1024; ++k) out1024[k] *= s;
    }
    if (n_frames) *n_frames = ctx->spec_frames;
    return B200SDR_OK;
}

int32_t b200sdr_get_audio(b200sdr_ctx *ctx, uint32_t chain, float *out, uint32_t capacity, uint32_t *n_out)
{
    if (!ctx || !out) return B200SDR_FAIL;
    DeviceGuard guard(ctx->device);
    if (!ctx->slot_acquired) {
        int rc = flush_pending(ctx);
        if (rc) return rc;
    }
    if (chain == B200SDR_CHAIN_WBFM) return pop_fifo(ctx, ctx->fm_fifo, out, capacity, n_out);
    if (chain == B200SDR_CHAIN_AM) return pop_fifo(ctx, ctx->am_fifo, out, capacity, n_out);
    return fail(ctx, B200SDR_NOT_SUPPORTED, "chain has no audio output");
}

int32_t b200sdr_get_counters(b200sdr_ctx *ctx, uint64_t *bytes_in, uint64_t *blocks_in, uint64_t *busy_returns)
{
    if (!ctx) return B200SDR_FAIL;
    if (bytes_in) *bytes_in = ctx->bytes_in;
    if (blocks_in) *blocks_in = ctx->blocks_in;
    if (busy_returns) *busy_returns = ctx->busy_returns;
    return B200SDR_OK;
}

int32_t b200sdr_debug_last_block(b200sdr_ctx *ctx, uint8_t *out, uint32_t capacity, uint32_t *len)
{
    if (!ctx || !out) return B200SDR_FAIL;
    DeviceGuard guard(ctx->device);
    if (!ctx->slot_acquired) {
        int rc = flush_pending(ctx);
        if (rc) return rc;
    }
    CU(cudaStreamSynchronize(ctx->s_copy));
    int jrc = join_chains(ctx);
    if (jrc) return jrc;
    CU(cudaStreamSynchronize(ctx->s_compute));
    uint32_t n = ctx->last_len < capacity ? ctx->last_len : capacity;
    if (n) CU(cudaMemcpy(out, ctx->d_stream + ctx->last_pos + ctx->last_off, n, cudaMemcpyDeviceToHost));
    if (len) *len = ctx->last_len;
    return B200SDR_OK;
}

int32_t b200sdr_debug_wbfm_tc_acc(b200sdr_ctx *ctx, const uint8_t *iq_dev, uint64_t len, int32_t *acc_host, int8_t *slices_host,
                                  int32_t *exponent)
{
    if (!ctx || !iq_dev || !acc_host) return B200SDR_FAIL;
    if (len == 0 || (len & 15u) || ((uintptr_t)iq_dev & 15u)) return B200SDR_NOT_SUPPORTED;
    DeviceGuard guard(ctx->device);
    int32_t *d_acc = nullptr;
    float *d_audio = nullptr;
    CU(cudaMalloc((void **)&d_acc, 128 * B200_TC_N * sizeof(int32_t)));
    CU(cudaMemset(d_acc, 0, 128 * B200_TC_N * sizeof(int32_t)));
    cudaError_t e = cudaMalloc((void **)&d_audio, (b200::wbfm_audio_len(len) + 4) * sizeof(float));
    int rc = e == cudaSuccess ? launch_wbfm_tc_batch(ctx, iq_dev, 1, len, d_audio, nullptr, d_acc) : fail(ctx, B200SDR_FAIL, "cudaMalloc", e);
    if (!rc && cudaStreamSynchronize(ctx->s_compute) != cudaSuccess) rc = fail(ctx, B200SDR_FAIL, "k_wbfm_tc", cudaGetLastError());
    if (!rc) rc = check_tc_error(ctx);
    if (!rc && cudaMemcpy(acc_host, d_acc, 128 * B200_TC_N * sizeof(int32_t), cudaMemcpyDeviceToHost) != cudaSuccess) rc = B200SDR_FAIL;
    cudaFree(d_acc);
    cudaFree(d_audio);
    if (slices_host || exponent) {
        FmTcConsts tc{};
        int8_t q[3][B200_FM_T1];
        int ex = 0;
        b200::fill_fm_tc(tc, nullptr, q, &ex);
        if (slices_host) memcpy(slices_host, q, sizeof q);
        if (exponent) *exponent = ex;
    }
    return rc;
}

/* ---- batched, device-resident -------------------------------------------------------------- */
uint64_t b200sdr_spectrum_frames(uint64_t len_bytes) { return b200::spectrum_frames(len_bytes); }
uint64_t b200sdr_wbfm_disc_len(uint64_t len_bytes) { return b200::wbfm_disc_len(len_bytes); }
uint64_t b200sdr_wbfm_audio_len(uint64_t len_bytes) { return b200::wbfm_audio_len(len_bytes); }
uint64_t b200sdr_am_audio_len(uint64_t len_bytes) { return b200::am_audio_len(len_bytes); }
uint32_t b200sdr_stream_chunk_samples(uint32_t chain)
{
    return chain == B200SDR_CHAIN_WBFM ? B200_FM_CHUNK : chain == B200SDR_CHAIN_AM ? B200_AM_CHUNK : 0u;
}

int32_t b200sdr_batch_spectrum_dev(b200sdr_ctx *ctx, const uint8_t *iq_dev, uint32_t n_captures, uint64_t len_each,
                                   float *spectrum_dev)
{
    if (!ctx || !iq_dev || !spectrum_dev) return B200SDR_FAIL;
    if (n_captures == 0) return B200SDR_OK;
    if ((len_each & 3u) || n_captures > 65535u || ((uintptr_t)iq_dev & 1u))
        return fail(ctx, B200SDR_NOT_SUPPORTED, "len_each must be a multiple of 4, n_captures <= 65535");
    DeviceGuard guard(ctx->device);
    if (b200::spectrum_frames(len_each) == 0) {
        CU(cudaMemsetAsync(spectrum_dev, 0, (size_t)n_captures * 1024 * sizeof(float), ctx->s_compute));
        return B200SDR_OK;
    }
    return launch_spectrum(ctx, iq_dev, n_captures, len_each, len_each, ctx->cfg.avg_mode == B200SDR_AVG_EMA, nullptr,
                           0.0f, 0.0f, false, spectrum_dev);
}

int32_t b200sdr_batch_wbfm_dev(b200sdr_ctx *ctx, const uint8_t *iq_dev, uint32_t n_captures, uint64_t len_each,
                               float *audio_dev, float *disc_dev)
{
    if (!ctx || !iq_dev || !audio_dev) return B200SDR_FAIL;
    if (n_captures == 0 || len_each == 0) return B200SDR_OK;
    if ((len_each & 15u) || !aligned16(iq_dev) || n_captures > 65535u)
        return fail(ctx, B200SDR_NOT_SUPPORTED, "batched WBFM needs 16-byte aligned captures (len_each % 16 == 0)");
    DeviceGuard guard(ctx->device);
    return launch_wbfm_batch(ctx, iq_dev, n_captures, len_each, audio_dev, disc_dev);
}

int32_t b200sdr_batch_am_dev(b200sdr_ctx *ctx, const uint8_t *iq_dev, uint32_t n_captures, uint64_t len_each,
                             float *audio_dev)
{
    if (!ctx || !iq_dev || !audio_dev) return B200SDR_FAIL;
    if (n_captures == 0 || len_each == 0) return B200SDR_OK;
    if ((len_each & 15u) || !aligned16(iq_dev) || n_captures > 65535u)
        return fail(ctx, B200SDR_NOT_SUPPORTED, "batched AM needs 16-byte aligned captures (len_each % 16 == 0)");
    DeviceGuard guard(ctx->device);
    return launch_am_batch(ctx, iq_dev, n_captures, len_each, audio_dev);
}

/* ---- batched, host buffers: captures stream through two device wave buffers so the H2D copy of
 * wave w+1 overlaps the kernels of wave w; results go straight back to host memory ------------ */
int32_t b200sdr_batch_host(b200sdr_ctx *ctx, uint32_t chains, const uint8_t *iq_host, uint32_t n_captures,
                           uint64_t len_each, float *spectrum_host, float *wbfm_audio_host, float *am_audio_host)
{
    if (!ctx || !iq_host) return B200SDR_FAIL;
    if (n_captures == 0 || len_each == 0) return B200SDR_OK;
    if (len_each & 15u) return fail(ctx, B200SDR_NOT_SUPPORTED, "len_each must be a multiple of 16");
    if ((chains & B200SDR_CHAIN_SPECTRUM) && !spectrum_host) return B200SDR_FAIL;
    if ((chains & B200SDR_CHAIN_WBFM) && !wbfm_audio_host) return B200SDR_FAIL;
    if ((chains & B200SDR_CHAIN_AM) && !am_audio_host) return B200SDR_FAIL;
    DeviceGuard guard(ctx->device);
    uint64_t per_wave = kWaveBytes / len_each;
    if (per_wave < 1) per_wave = 1;
    if (per_wave > n_captures) per_wave = n_captures;
    const size_t wave_bytes = (size_t)per_wave * len_each;
    if (ctx->wave_bytes < wave_bytes) {
        CU(cudaDeviceSynchronize());
        for (int i = 0; i < 2; ++i) {
            if (ctx->d_wave[i]) CU(cudaFree(ctx->d_wave[i]));
            ctx->d_wave[i] = nullptr;
            CU(cudaMalloc((void **)&ctx->d_wave[i], wave_bytes));
        }
        ctx->wave_bytes = wave_bytes;
    }
    const uint64_t fm_len = b200::wbfm_audio_len(len_each), am_len = b200::am_audio_len(len_each);
    float *d_spec = nullptr, *d_fm = nullptr, *d_am = nullptr;
    /* per-wave result buffers, double buffered with the wave; kept in the context between calls */
    int rca = B200SDR_OK;
    if (chains & B200SDR_CHAIN_SPECTRUM) { rca = ensure_floats(ctx, &ctx->d_res_spec, &ctx->res_spec_floats, 2 * per_wave * 1024); if (rca) return rca; d_spec = ctx->d_res_spec; }
    if (chains & B200SDR_CHAIN_WBFM) { rca = ensure_floats(ctx, &ctx->d_res_fm, &ctx->res_fm_floats, 2 * per_wave * fm_len); if (rca) return rca; d_fm = ctx->d_res_fm; }
    if (chains & B200SDR_CHAIN_AM) { rca = ensure_floats(ctx, &ctx->d_res_am, &ctx->res_am_floats, 2 * per_wave * am_len); if (rca) return rca; d_am = ctx->d_res_am; }
    /* three streams: H2D of wave w+1 (copy), kernels of wave w (compute), D2H of the results of wave w-1 (d2h) --
     * PCIe is full duplex, and the kernels of the next wave do not wait for a read-back */
    int rc = B200SDR_OK;
    bool used[2] = {false, false};
    uint32_t wave = 0;
    for (uint64_t c0 = 0; c0 < n_captures && rc == B200SDR_OK; c0 += per_wave, ++wave) {
        const int b = (int)(wave & 1);
        const uint32_t nc = (uint32_t)((n_captures - c0 < per_wave) ? n_captures - c0 : per_wave);
        if (used[b]) {
            CU(cudaStreamWaitEvent(ctx->s_copy, ctx->ev_wave_done[b], 0));   /* wave buffer: kernels of wave w-2 done */
            CU(cudaStreamWaitEvent(ctx->s_compute, ctx->ev_wave_out[b], 0)); /* result buffers: read-back of wave w-2 done */
        }
        CU(cudaMemcpyAsync(ctx->d_wave[b], iq_host + c0 * len_each, (size_t)nc * len_each, cudaMemcpyHostToDevice, ctx->s_copy));
        CU(cudaEventRecord(ctx->ev_wave_copied[b], ctx->s_copy));
        CU(cudaStreamWaitEvent(ctx->s_compute, ctx->ev_wave_copied[b], 0));
        float *o_spec = d_spec ? d_spec + (size_t)b * per_wave * 1024 : nullptr;
        float *o_fm = d_fm ? d_fm + (size_t)b * per_wave * fm_len : nullptr;
        float *o_am = d_am ? d_am + (size_t)b * per_wave * am_len : nullptr;
        if (chains & B200SDR_CHAIN_SPECTRUM) { rc = b200sdr_batch_spectrum_dev(ctx, ctx->d_wave[b], nc, len_each, o_spec); if (rc) break; }
        if (chains & B200SDR_CHAIN_WBFM) { rc = launch_wbfm_batch(ctx, ctx->d_wave[b], nc, len_each, o_fm, nullptr); if (rc) break; }
        if (chains & B200SDR_CHAIN_AM) { rc = launch_am_batch(ctx, ctx->d_wave[b], nc, len_each, o_am); if (rc) break; }
        CU(cudaEventRecord(ctx->ev_wave_done[b], ctx->s_compute));
        CU(cudaStreamWaitEvent(ctx->s_d2h, ctx->ev_wave_done[b], 0));
        if (chains & B200SDR_CHAIN_SPECTRUM)
            CU(cudaMemcpyAsync(spectrum_host + c0 * 1024, o_spec, (size_t)nc * 1024 * sizeof(float), cudaMemcpyDeviceToHost, ctx->s_d2h));
        if (chains & B200SDR_CHAIN_WBFM)
            CU(cudaMemcpyAsync(wbfm_audio_host + c0 * fm_len, o_fm, (size_t)nc * fm_len * sizeof(float), cudaMemcpyDeviceToHost, ctx->s_d2h));
        if (chains & B200SDR_CHAIN_AM)
            CU(cudaMemcpyAsync(am_audio_host + c0 * am_len, o_am, (size_t)nc * am_len * sizeof(float), cudaMemcpyDeviceToHost, ctx->s_d2h));
        CU(cudaEventRecord(ctx->ev_wave_out[b], ctx->s_d2h));
        used[b] = true;
    }
    cudaError_t e1 = cudaStreamSynchronize(ctx->s_copy), e2 = cudaStreamSynchronize(ctx->s_compute),
                e3 = cudaStreamSynchronize(ctx->s_d2h);
    if (rc) return rc;
    if (e1 != cudaSuccess) return fail(ctx, B200SDR_FAIL, "copy stream", e1);
    if (e2 != cudaSuccess) return fail(ctx, B200SDR_FAIL, "compute stream", e2);
    if (e3 != cudaSuccess) return fail(ctx, B200SDR_FAIL, "read-back stream", e3);
    return B200SDR_OK;
}

/* ---- K2 ------------------------------------------------------------------------------------ */
int32_t b200sdr_convert_cf32_dev(b200sdr_ctx *ctx, const uint8_t *iq_dev, uint64_t len, uint32_t window, float *out_dev)
{
    if (!ctx || !iq_dev || !out_dev) return B200SDR_FAIL;
    if (window > B200SDR_WINDOW_BLACKMAN) return fail(ctx, B200SDR_NOT_SUPPORTED, "bad window");
    if ((len & 15u) || !aligned16(iq_dev) || !aligned16(out_dev))
        return fail(ctx, B200SDR_NOT_SUPPORTED, "device conversion needs len % 16 == 0 and 16-byte aligned pointers");
    if (len == 0) return B200SDR_OK;
    DeviceGuard guard(ctx->device);
    const uint64_t n_words = len / 4;
    const float *w = window == B200SDR_WINDOW_RECT ? nullptr : ctx->d_window[window];
    k_convert_cf32<<<(unsigned)((n_words + 1023) / 1024), 256, 0, ctx->s_compute>>>((const uint32_t *)iq_dev, (float4 *)out_dev, n_words, w);
    CU(cudaGetLastError());
    ctx->launches += 1;
    return B200SDR_OK;
}

int32_t b200sdr_convert_cf32(b200sdr_ctx *ctx, const uint8_t *iq_host, uint32_t len, uint32_t window, float *out_host)
{
    if (!ctx || !iq_host || !out_host) return B200SDR_FAIL;
    if (len & 3u) return fail(ctx, B200SDR_NOT_SUPPORTED, "len must be a multiple of 4");
    if (len == 0) return B200SDR_OK;
    DeviceGuard guard(ctx->device);
    const uint64_t padded = ((uint64_t)len + 15u) & ~15ull;
    uint8_t *d_in = nullptr;
    float *d_out = nullptr;
    CU(cudaMalloc((void **)&d_in, padded));
    cudaError_t e = cudaMalloc((void **)&d_out, padded * sizeof(float));
    if (e != cudaSuccess) { cudaFree(d_in); return fail(ctx, B200SDR_FAIL, "cudaMalloc", e); }
    int rc = B200SDR_OK;
    do {
        if ((e = cudaMemsetAsync(d_in, 0, padded, ctx->s_compute)) != cudaSuccess) break;
        if ((e = cudaMemcpyAsync(d_in, iq_host, len, cudaMemcpyHostToDevice, ctx->s_compute)) != cudaSuccess) break;
        rc = b200sdr_convert_cf32_dev(ctx, d_in, padded, window, d_out);
        if (rc) break;
        if ((e = cudaMemcpyAsync(out_host, d_out, (size_t)len * sizeof(float), cudaMemcpyDeviceToHost, ctx->s_compute)) != cudaSuccess) break;
        e = cudaStreamSynchronize(ctx->s_compute);
    } while (0);
    cudaFree(d_in);
    cudaFree(d_out);
    if (rc) return rc;
    if (e != cudaSuccess) return fail(ctx, B200SDR_FAIL, "convert", e);
    return B200SDR_OK;
}

/* ---- test-mode counter check (kernel K0) ---------------------------------------------------- */
int32_t b200sdr_counter_check_dev(b200sdr_ctx *ctx, const uint8_t *iq_dev, uint32_t n_captures, uint64_t len_each,
                                  int32_t expect_first, uint64_t *n_breaks_host, uint64_t *first_break_host)
{
    if (!ctx) return B200SDR_FAIL;
    if (n_captures == 0) return B200SDR_OK;
    if (!iq_dev) return fail(ctx, B200SDR_FAIL, "null capture pointer");
    if ((len_each & 3u) || !aligned16(iq_dev) || (n_captures > 1 && (len_each & 15u)) || n_captures > 65535u || expect_first > 255)
        return fail(ctx, B200SDR_NOT_SUPPORTED, "counter check needs len % 4 == 0, a 16-byte aligned pointer and stride, <= 65535 captures");
    DeviceGuard guard(ctx->device);
    if (ctx->counter_res_cap < n_captures) { /* grown on demand, kept: no allocation on the repeated call */
        if (ctx->d_counter_res) { CU(cudaStreamSynchronize(ctx->s_compute)); CU(cudaFree(ctx->d_counter_res)); }
        ctx->d_counter_res = nullptr;
        ctx->counter_res_cap = 0;
        CU(cudaMalloc((void **)&ctx->d_counter_res, 2u * (size_t)n_captures * sizeof(unsigned long long)));
        ctx->counter_res_cap = n_captures;
    }
    unsigned long long *d_res = ctx->d_counter_res;
    cudaError_t e = cudaSuccess;
    do {
        if ((e = cudaMemsetAsync(d_res, 0, n_captures * sizeof(unsigned long long), ctx->s_compute)) != cudaSuccess) break;
        if ((e = cudaMemsetAsync(d_res + n_captures, 0xff, n_captures * sizeof(unsigned long long), ctx->s_compute)) != cudaSuccess) break;
        if (len_each) {
            CounterParams p{};
            p.in = reinterpret_cast<const uint32_t *>(iq_dev);
            p.stride_words = len_each / 4u;
            p.n_words = len_each / 4u;
            p.expect_first = expect_first < 0 ? -1 : expect_first;
            p.n_breaks = d_res;
            p.first_break = d_res + n_captures;
            const uint64_t n_vec = len_each / 16u;
            const uint64_t blocks = n_vec ? b200::ceil_div(n_vec, 1024) : 1;
            if (blocks > 0x3fffffull) return fail(ctx, B200SDR_NOT_SUPPORTED, "capture too long (the kernel indexes vectors with 32 bits)");
            k_counter_check<<<dim3((unsigned)blocks, n_captures), 256, 0, ctx->s_compute>>>(p);
            if ((e = cudaGetLastError()) != cudaSuccess) break;
            ctx->launches += 1;
        }
        static_assert(sizeof(unsigned long long) == sizeof(uint64_t), "result layout");
        if (n_breaks_host &&
            (e = cudaMemcpyAsync(n_breaks_host, d_res, n_captures * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->s_compute)) != cudaSuccess) break;
        if (first_break_host &&
            (e = cudaMemcpyAsync(first_break_host, d_res + n_captures, n_captures * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->s_compute)) != cudaSuccess) break;
        e = cudaStreamSynchronize(ctx->s_compute);
    } while (0);
    if (e != cudaSuccess) return fail(ctx, B200SDR_FAIL, "counter check", e);
    return B200SDR_OK;
}

int32_t b200sdr_get_counter_check(b200sdr_ctx *ctx, uint64_t *n_breaks, uint64_t *first_break)
{
    if (!ctx) return B200SDR_FAIL;
    if (!(ctx->cfg.chains & B200SDR_CHAIN_COUNTER)) return fail(ctx, B200SDR_NOT_SUPPORTED, "B200SDR_CHAIN_COUNTER is not enabled");
    DeviceGuard guard(ctx->device);
    int rc = flush_pending(ctx);
    if (rc) return rc;
    CounterStreamState st{};
    CU(cudaMemcpyAsync(&st, ctx->d_cnt_state, sizeof st, cudaMemcpyDeviceToHost, ctx->s_chain[3]));
    CU(cudaStreamSynchronize(ctx->s_chain[3]));
    if (n_breaks) *n_breaks = st.n_breaks;
    if (first_break) *first_break = st.first_break;
    return B200SDR_OK;
}

int32_t b200sdr_counter_check(b200sdr_ctx *ctx, const uint8_t *iq_host, uint32_t len, int32_t expect_first, uint64_t *n_breaks,
                              uint64_t *first_break)
{
    if (!ctx || (!iq_host && len)) return B200SDR_FAIL;
    if (len & 3u) return fail(ctx, B200SDR_NOT_SUPPORTED, "len must be a multiple of 4");
    if (len == 0) {
        if (n_breaks) *n_breaks = 0;
        if (first_break) *first_break = ~0ull;
        return B200SDR_OK;
    }
    DeviceGuard guard(ctx->device);
    uint8_t *d_in = nullptr;
    CU(cudaMalloc((void **)&d_in, len));
    cudaError_t e = cudaMemcpyAsync(d_in, iq_host, len, cudaMemcpyHostToDevice, ctx->s_compute);
    int rc = B200SDR_OK;
    if (e == cudaSuccess) rc = b200sdr_counter_check_dev(ctx, d_in, 1, len, expect_first, n_breaks, first_break);
    cudaFree(d_in);
    if (e != cudaSuccess) return fail(ctx, B200SDR_FAIL, "counter check copy", e);
    return rc;
}

int32_t b200sdr_get_taps(b200sdr_ctx *ctx, uint32_t which, float *out, uint32_t capacity, uint32_t *n_taps)
{
    if (!ctx || which > 4) return B200SDR_NOT_SUPPORTED;
    const std::vector<float> &h = ctx->h_taps[which];
    if (n_taps) *n_taps = (uint32_t)h.size();
    if (out) {
        if (capacity < h.size()) return fail(ctx, B200SDR_NOT_SUPPORTED, "capacity too small");
        memcpy(out, h.data(), h.size() * sizeof(float));
    }
    return B200SDR_OK;
}

int32_t b200sdr_get_window(b200sdr_ctx *ctx, uint32_t window, float *out1024)
{
    if (!ctx || !out1024 || window > 2) return B200SDR_NOT_SUPPORTED;
    DeviceGuard guard(ctx->device);
    CU(cudaMemcpy(out1024, ctx->d_window[window], 1024 * sizeof(float), cudaMemcpyDeviceToHost)); /* as the kernels see it */
    return B200SDR_OK;
}

/* ---- presentation (section 8f row 3) ------------------------------------------------------- */
int32_t b200sdr_render_spectrum_dev(b200sdr_ctx *ctx, const float *spectra_dev, uint32_t n_spectra, float scale,
                                    float db_min, float db_max, uint32_t *argb_dev)
{
    if (!ctx || !spectra_dev || !argb_dev) return B200SDR_FAIL;
    if (!(db_max > db_min)) return fail(ctx, B200SDR_NOT_SUPPORTED, "db_max must exceed db_min");
    if (n_spectra == 0) return B200SDR_OK;
    DeviceGuard guard(ctx->device);
    int rc = upload_thresholds(ctx, db_min, db_max);
    if (rc) return rc;
    k_render_spectrum<<<n_spectra, B200_LCD_W, 0, ctx->s_compute>>>(spectra_dev, scale, ctx->d_thresholds, argb_dev);
    CU(cudaGetLastError());
    ctx->launches += 1;
    return B200SDR_OK;
}

int32_t b200sdr_render_waterfall_dev(b200sdr_ctx *ctx, const float *spectra_dev, uint32_t n_rows, float scale,
                                     float db_min, float db_max, uint32_t *argb_dev)
{
    if (!ctx || !argb_dev || (!spectra_dev && n_rows)) return B200SDR_FAIL;
    if (!(db_max > db_min)) return fail(ctx, B200SDR_NOT_SUPPORTED, "db_max must exceed db_min");
    DeviceGuard guard(ctx->device);
    int rc = upload_thresholds(ctx, db_min, db_max);
    if (rc) return rc;
    if (n_rows > B200_LCD_H) n_rows = B200_LCD_H; /* the panel has 272 rows */
    k_render_waterfall<<<B200_LCD_H, B200_LCD_W, 0, ctx->s_compute>>>(spectra_dev, n_rows, scale, ctx->d_thresholds, argb_dev);
    CU(cudaGetLastError());
    ctx->launches += 1;
    return B200SDR_OK;
}

int32_t b200sdr_render_waterfall(b200sdr_ctx *ctx, const float *spectra_host, uint32_t n_rows, float db_min, float db_max,
                                 uint32_t *argb_host)
{
    if (!ctx || !argb_host || (!spectra_host && n_rows)) return B200SDR_FAIL;
    DeviceGuard guard(ctx->device);
    if (n_rows > B200_LCD_H) n_rows = B200_LCD_H;
    const size_t img_bytes = (size_t)B200_LCD_W * B200_LCD_H * sizeof(uint32_t);
    const size_t spec_bytes = (size_t)(n_rows ? n_rows : 1) * 1024 * sizeof(float);
    uint32_t *d_img = nullptr;
    float *d_spec = nullptr;
    CU(cudaMalloc((void **)&d_img, img_bytes));
    int rc = B200SDR_OK;
    cudaError_t e = cudaSuccess;
    do {
        if ((e = cudaMalloc((void **)&d_spec, spec_bytes)) != cudaSuccess) break;
        if (n_rows && (e = cudaMemcpyAsync(d_spec, spectra_host, spec_bytes, cudaMemcpyHostToDevice, ctx->s_compute)) != cudaSuccess) break;
        rc = b200sdr_render_waterfall_dev(ctx, d_spec, n_rows, 1.0f, db_min, db_max, d_img);
        if (rc) break;
        if ((e = cudaMemcpyAsync(argb_host, d_img, img_bytes, cudaMemcpyDeviceToHost, ctx->s_compute)) != cudaSuccess) break;
        e = cudaStreamSynchronize(ctx->s_compute);
    } while (0);
    cudaFree(d_img);
    if (d_spec) cudaFree(d_spec);
    if (rc) return rc;
    if (e != cudaSuccess) return fail(ctx, B200SDR_FAIL, "render waterfall", e);
    return B200SDR_OK;
}

int32_t b200sdr_render_spectrum(b200sdr_ctx *ctx, const float *spectrum_host, float db_min, float db_max, uint32_t *argb_host)
{
    if (!ctx || !argb_host) return B200SDR_FAIL;
    DeviceGuard guard(ctx->device);
    if (!spectrum_host && !ctx->slot_acquired) { /* the streaming spectrum must include every accepted block */
        int frc = flush_pending(ctx);
        if (frc) return frc;
    }
    if (!spectrum_host) { /* the render kernel (compute stream) reads what the spectrum chain's stream wrote */
        int jrc = join_chains(ctx);
        if (jrc) return jrc;
    }
    const size_t img_bytes = (size_t)B200_LCD_W * B200_LCD_H * sizeof(uint32_t);
    uint32_t *d_img = nullptr;
    float *d_spec = nullptr;
    CU(cudaMalloc((void **)&d_img, img_bytes));
    int rc = B200SDR_OK;
    cudaError_t e = cudaSuccess;
    do {
        const float *src = ctx->d_spec_acc;
        float scale = 1.0f;
        if (spectrum_host) {
            if ((e = cudaMalloc((void **)&d_spec, 1024 * sizeof(float))) != cudaSuccess) break;
            if ((e = cudaMemcpyAsync(d_spec, spectrum_host, 1024 * sizeof(float), cudaMemcpyHostToDevice, ctx->s_compute)) != cudaSuccess) break;
            src = d_spec;
        } else if (ctx->cfg.avg_mode == B200SDR_AVG_MEAN && ctx->spec_frames) {
            scale = 1.0f / (float)ctx->spec_frames; /* the accumulator holds the sum */
        }
        rc = b200sdr_render_spectrum_dev(ctx, src, 1, scale, db_min, db_max, d_img);
        if (rc) break;
        if ((e = cudaMemcpyAsync(argb_host, d_img, img_bytes, cudaMemcpyDeviceToHost, ctx->s_compute)) != cudaSuccess) break;
        e = cudaStreamSynchronize(ctx->s_compute);
    } while (0);
    cudaFree(d_img);
    if (d_spec) cudaFree(d_spec);
    if (rc) return rc;
    if (e != cudaSuccess) return fail(ctx, B200SDR_FAIL, "render", e);
    return B200SDR_OK;
}

/* ---- synthetic captures -------------------------------------------------------------------- */
int32_t b200sdr_synth_fill_dev(b200sdr_ctx *ctx, uint8_t *iq_dev, uint32_t n_captures, uint64_t len_each, uint32_t kind,
                               uint64_t first_capture)
{
    if (!ctx || !iq_dev) return B200SDR_FAIL;
    if (kind > B200SDR_SYNTH_AM) return fail(ctx, B200SDR_NOT_SUPPORTED, "bad synth kind");
    if ((len_each & 15u) || !aligned16(iq_dev) || n_captures > 65535u)
        return fail(ctx, B200SDR_NOT_SUPPORTED, "len_each must be a multiple of 16");
    if (n_captures == 0 || len_each == 0) return B200SDR_OK;
    DeviceGuard guard(ctx->device);
    const uint64_t groups = len_each / 16;
    k_synth<<<dim3((unsigned)((groups + 255) / 256), n_captures), 256, 0, ctx->s_compute>>>((uint4 *)iq_dev, groups, groups, kind,
                                                                                             first_capture, ctx->d_lut);
    CU(cudaGetLastError());
    ctx->launches += 1;
    return B200SDR_OK;
}

int32_t b200sdr_synth_fill_host(uint8_t *iq_host, uint32_t n_captures, uint64_t len_each, uint32_t kind, uint64_t first_capture)
{
    if (!iq_host || kind > B200SDR_SYNTH_AM || (len_each & 1u)) return B200SDR_NOT_SUPPORTED;
    const float *lut = synth_lut_host();
    for (uint32_t c = 0; c < n_captures; ++c) {
        uint8_t *p = iq_host + (uint64_t)c * len_each;
        const uint64_t seed = B200SDR_SYNTH_SEED_BASE + first_capture + c;
        for (uint64_t n = 0; n < len_each / 2; ++n) b200sdr_synth_sample(lut, kind, seed, n, &p[2 * n], &p[2 * n + 1]);
    }
    return B200SDR_OK;
}

/* ---- split-capture exchange (SURVEY.md section 8e, kernel K6) -------------------------------- */
int32_t b200sdr_exchange_create(b200sdr_ctx *ctx, uint32_t world, uint32_t rank, uint8_t *handle_out64)
{
    if (!ctx) return B200SDR_FAIL;
    if (world < 1 || world > B200_XCHG_MAX_WORLD || rank >= world) return fail(ctx, B200SDR_NOT_SUPPORTED, "bad world / rank");
    if (ctx->d_mailbox) return fail(ctx, B200SDR_FAIL, "exchange already created");
    DeviceGuard guard(ctx->device);
    const size_t bytes = B200_XCHG_MAILBOX_BYTES(world);
    CU(cudaMalloc((void **)&ctx->d_mailbox, bytes));
    CU(cudaMemset(ctx->d_mailbox, 0, bytes));
    CU(cudaHostAlloc((void **)&ctx->d_xchg_status, sizeof(uint32_t), cudaHostAllocMapped));
    *ctx->d_xchg_status = 0;
    ctx->xchg_world = world;
    ctx->xchg_rank = rank;
    ctx->xchg_seq = 0;
    ctx->xchg_connected = false;
    for (uint32_t r = 0; r < B200_XCHG_MAX_WORLD; ++r) { ctx->peer_mail[r] = nullptr; ctx->peer_is_ipc[r] = false; }
    ctx->peer_mail[rank] = ctx->d_mailbox;
    if (handle_out64) {
        static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
        cudaIpcMemHandle_t h;
        CU(cudaIpcGetMemHandle(&h, ctx->d_mailbox));
        memcpy(handle_out64, &h, 64);
    }
    return B200SDR_OK;
}

int32_t b200sdr_exchange_connect(b200sdr_ctx *ctx, const uint8_t *handles /* world x 64 bytes, rank order */)
{
    if (!ctx) return B200SDR_FAIL;
    if (!ctx->d_mailbox) return fail(ctx, B200SDR_FAIL, "call b200sdr_exchange_create first");
    if (!handles && ctx->xchg_world > 1) return fail(ctx, B200SDR_FAIL, "no IPC handles");
    DeviceGuard guard(ctx->device);
    for (uint32_t r = 0; r < ctx->xchg_world; ++r) {
        if (r == ctx->xchg_rank || ctx->peer_mail[r]) continue;
        cudaIpcMemHandle_t h;
        memcpy(&h, handles + 64u * r, 64);
        void *ptr = nullptr;
        CU(cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess));
        ctx->peer_mail[r] = (float *)ptr;
        ctx->peer_is_ipc[r] = true;
    }
    ctx->xchg_connected = true;
    return B200SDR_OK;
}

int32_t b200sdr_exchange_connect_local(b200sdr_ctx *ctx, b200sdr_ctx *const *peers /* world contexts of THIS process */)
{
    if (!ctx || !peers) return B200SDR_FAIL;
    if (!ctx->d_mailbox) return fail(ctx, B200SDR_FAIL, "call b200sdr_exchange_create first");
    DeviceGuard guard(ctx->device);
    for (uint32_t r = 0; r < ctx->xchg_world; ++r) {
        if (r == ctx->xchg_rank) continue;
        b200sdr_ctx *o = peers[r];
        if (!o || !o->d_mailbox || o->xchg_world != ctx->xchg_world || o->xchg_rank != r)
            return fail(ctx, B200SDR_NOT_SUPPORTED, "peer context has no matching exchange");
        if (o->device != ctx->device) {
            int can = 0;
            CU(cudaDeviceCanAccessPeer(&can, ctx->device, o->device));
            if (!can) return fail(ctx, B200SDR_NOT_SUPPORTED, "no peer access between the two devices");
            cudaError_t e = cudaDeviceEnablePeerAccess(o->device, 0);
            if (e == cudaErrorPeerAccessAlreadyEnabled) (void)cudaGetLastError();
            else if (e != cudaSuccess) return fail(ctx, B200SDR_FAIL, "cudaDeviceEnablePeerAccess", e);
        }
        ctx->peer_mail[r] = o->d_mailbox;
    }
    ctx->xchg_connected = true;
    return B200SDR_OK;
}

int32_t b200sdr_split_spectrum_dev(b200sdr_ctx *ctx, const uint8_t *iq_slice_dev, uint64_t len_slice, uint64_t frames_total,
                                   float *spectrum_dev)
{
    if (!ctx || !spectrum_dev || (!iq_slice_dev && len_slice)) return B200SDR_FAIL;
    if (!ctx->xchg_connected) return fail(ctx, B200SDR_FAIL, "exchange not connected");
    if ((len_slice & 3u) || ((uintptr_t)iq_slice_dev & 1u) || frames_total == 0 || ctx->cfg.avg_mode != B200SDR_AVG_MEAN)
        return fail(ctx, B200SDR_NOT_SUPPORTED, "split capture: mean averaging, slice length a multiple of 4");
    DeviceGuard guard(ctx->device);
    /* this rank's frames -> per-CTA partial sums (no finalize: the exchange kernel reduces them) */
    b200::SpectrumPlan pl = b200::plan_spectrum(len_slice, 1, (uint32_t)ctx->sm_count);
    int rc = launch_spectrum(ctx, iq_slice_dev, 1, len_slice, len_slice, false, nullptr, 0.0f, 0.0f, false, nullptr, false);
    if (rc) return rc;
    ExchangeParams p{};
    p.partials = ctx->d_partials;
    p.ctas_per_capture = pl.frames ? pl.units_per_capture : 0; /* a rank without frames contributes zeros */
    p.scale = 1.0f / (float)frames_total;
    p.out = spectrum_dev;
    for (uint32_t r = 0; r < ctx->xchg_world; ++r) p.mail[r] = ctx->peer_mail[r];
    p.world = ctx->xchg_world;
    p.rank = ctx->xchg_rank;
    p.seq = ++ctx->xchg_seq;
    p.status = ctx->d_xchg_status;
    p.timeout_cycles = 10000000000ll; /* ~5 s at 1.965 GHz: a peer that never arrives fails the call */
    k_spectrum_finalize_exchange<<<B200_XCHG_CTAS, 256, 0, ctx->s_compute>>>(p);
    CU(cudaGetLastError());
    ctx->launches += 1;
    return B200SDR_OK;
}

int32_t b200sdr_exchange_wait(b200sdr_ctx *ctx)
{
    if (!ctx) return B200SDR_FAIL;
    if (!ctx->d_xchg_status) return fail(ctx, B200SDR_FAIL, "no exchange");
    DeviceGuard guard(ctx->device);
    CU(cudaStreamSynchronize(ctx->s_compute));
    if (*(volatile uint32_t *)ctx->d_xchg_status) {
        *ctx->d_xchg_status = 0;
        return fail(ctx, B200SDR_FAIL, "split-capture exchange timed out: a peer did not arrive");
    }
    return B200SDR_OK;
}

int32_t b200sdr_exchange_destroy(b200sdr_ctx *ctx)
{
    if (!ctx) return B200SDR_FAIL;
    DeviceGuard guard(ctx->device);
    cudaStreamSynchronize(ctx->s_compute);
    for (uint32_t r = 0; r < B200_XCHG_MAX_WORLD; ++r) {
        if (ctx->peer_is_ipc[r] && ctx->peer_mail[r]) cudaIpcCloseMemHandle(ctx->peer_mail[r]);
        ctx->peer_mail[r] = nullptr;
        ctx->peer_is_ipc[r] = false;
    }
    if (ctx->d_mailbox) cudaFree(ctx->d_mailbox);
    if (ctx->d_xchg_status) cudaFreeHost(ctx->d_xchg_status);
    ctx->d_mailbox = nullptr;
    ctx->d_xchg_status = nullptr;
    ctx->xchg_connected = false;
    ctx->xchg_world = 0;
    return B200SDR_OK;
}

/* ---- memory / timing helpers --------------------------------------------------------------- */
int32_t b200sdr_dev_alloc(b200sdr_ctx *ctx, uint64_t bytes, void **out_dev)
{
    if (!ctx || !out_dev) return B200SDR_FAIL;
    DeviceGuard guard(ctx->device);
    CU(cudaMalloc(out_dev, bytes ? bytes : 16));
    return B200SDR_OK;
}
int32_t b200sdr_dev_free(b200sdr_ctx *ctx, void *dev)
{
    if (!ctx) return B200SDR_FAIL;
    DeviceGuard guard(ctx->device);
    CU(cudaStreamSynchronize(ctx->s_compute));
    CU(cudaFree(dev));
    return B200SDR_OK;
}
int32_t b200sdr_host_alloc_pinned(b200sdr_ctx *ctx, uint64_t bytes, void **out_host)
{
    if (!ctx || !out_host) return B200SDR_FAIL;
    DeviceGuard guard(ctx->device);
    CU(cudaHostAlloc(out_host, bytes ? bytes : 16, cudaHostAllocDefault));
    return B200SDR_OK;
}
int32_t b200sdr_host_free_pinned(b200sdr_ctx *ctx, void *host)
{
    if (!ctx) return B200SDR_FAIL;
    DeviceGuard guard(ctx->device);
    CU(cudaFreeHost(host));
    return B200SDR_OK;
}
int32_t b200sdr_copy_to_host(b200sdr_ctx *ctx, void *dst_host, const void *src_dev, uint64_t bytes)
{
    if (!ctx) return B200SDR_FAIL;
    DeviceGuard guard(ctx->device);
    CU(cudaStreamSynchronize(ctx->s_compute));
    CU(cudaMemcpy(dst_host, src_dev, bytes, cudaMemcpyDeviceToHost));
    return B200SDR_OK;
}
int32_t b200sdr_copy_to_dev(b200sdr_ctx *ctx, void *dst_dev, const void *src_host, uint64_t bytes)
{
    if (!ctx) return B200SDR_FAIL;
    DeviceGuard guard(ctx->device);
    CU(cudaMemcpyAsync(dst_dev, src_host, bytes, cudaMemcpyHostToDevice, ctx->s_compute));
    CU(cudaStreamSynchronize(ctx->s_compute));
    return B200SDR_OK;
}
int32_t b200sdr_timer_start(b200sdr_ctx *ctx)
{
    if (!ctx) return B200SDR_FAIL;
    DeviceGuard guard(ctx->device);
    CU(cudaEventRecord(ctx->ev_t0, ctx->s_compute));
    return B200SDR_OK;
}
int32_t b200sdr_timer_stop_ms(b200sdr_ctx *ctx, float *ms)
{
    if (!ctx || !ms) return B200SDR_FAIL;
    DeviceGuard guard(ctx->device);
    CU(cudaEventRecord(ctx->ev_t1, ctx->s_compute));
    CU(cudaEventSynchronize(ctx->ev_t1));
    CU(cudaEventElapsedTime(ms, ctx->ev_t0, ctx->ev_t1));
    return B200SDR_OK;
}
uint64_t b200sdr_kernel_launches(b200sdr_ctx *ctx) { return ctx ? ctx->launches : 0; }
const char *b200sdr_last_error(b200sdr_ctx *ctx) { return ctx ? ctx->err : "null ctx"; }

} /* extern "C" */
