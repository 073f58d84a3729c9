// p25cu_api.cu -- the C ABI of include/p25cu.h: context, HBM layout, launch sequencing.
//
// Host-side counterpart of the reference's DemodTask (src/demod.rs:44-119) and of the
// RecvTask / ReplayReceiver sample loops (src/recv.rs:140-167, :204-234; src/replay.rs:26-57),
// batched over n_streams.  No CPU compute path exists here: every entry point either queues
// CUDA work or fails with an error code.
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <mutex>
#include <new>

#include "p25cu_internal.cuh"

cudaError_t p25cu_walk_upload_consts();
// wideband channelizer (pfb.cu)
unsigned p25cu_pfb_tail_len();
unsigned p25cu_pfb_channels();
unsigned p25cu_pfb_decimation();
cudaError_t p25cu_pfb_upload(float** d_taps, float2** d_twiddle);
cudaError_t p25cu_launch_pfb(const void* iq, const void* tail_in, void* tail_out, const float* taps, const float2* twiddle,
                             float2* y, unsigned y_rows, float* bb, size_t row_stride, float* power_sum,
                             unsigned long long a0, unsigned long long m0, unsigned n, unsigned n_out, unsigned n_captures,
                             cudaStream_t st, unsigned* launches, const P25DevPlan* plan);

// Per-device launch plans (P25DevPlan): filled once per device, under a mutex, by the first context created on it.
static std::mutex g_plan_mu;
static P25DevPlan g_plans[P25CU_MAX_DEVICES];
static bool g_plan_ok[P25CU_MAX_DEVICES];

struct p25cu_ctx {
    p25cu_config cfg;
    const P25DevPlan* plan;    // launch geometry of cfg.device
    cudaStream_t stream;       // demod kernels (and the walker when it is not overlapped)
    cudaStream_t stream2;      // decode walker, event compaction, event/stat copies
    cudaStream_t stream_copy;  // host -> device copies of caller input (copy of chunk k+1 beside the kernels of chunk k)
    cudaEvent_t ev_bb_ready[2], ev_bb_free[2];
    cudaEvent_t ev_iq_ready[2], ev_iq_free[2];
    int overlap;               // walker of chunk k runs concurrently with ddc_fm of chunk k+1
    int walk_prefilter;        // walker consults the tensor-pipe sync prefilter (mostly idle streams: channelizer contexts)
    char err[512];
    unsigned ht;               // input tail length (samples)
    size_t max_out;            // max baseband samples per stream per chunk
    size_t row_stride;         // floats per baseband row
    unsigned ev_cap;           // event slots per stream
    void* d_iq[2];             // double-buffered staging for host-resident input (lazy)
    size_t d_iq_bytes[2];
    int iq_slot;
    float2* d_tail[2];
    int tail_cur;
    float* d_bb[2];            // double-buffered baseband rows
    int bb_cur;                // buffer the next producer (demod / host baseband) writes
    int bb_last;               // buffer holding the newest undecoded baseband
    float* d_power;
    unsigned* d_work;          // ticket counter of the /50 demod kernel (monotonic)
    // optional per-launch timing of the demod kernel(s): event pairs recorded right around the launch
    int timing;
    unsigned n_timed;
    cudaEvent_t tev[2 * 128];
    unsigned ticket_base;
    WalkStateHbm* d_states;
    unsigned* d_slots;         // [S][ev_cap * P25CU_SLOT_WORDS] packed event records
    p25cu_event* d_dense;      // 80-byte records for p25cu_poll / p25cu_poll_view (lazy)
    unsigned* d_offsets;       // [2 S + 4]: exclusive event / word offsets, totals (events, words, overflow, truncated)
    unsigned long long* d_stats;
    P25DevTables* d_tables;
    uint32_t* d_golay;         // Golay(23,12) syndrome table (referenced from d_tables)
    p25cu_event* h_events;     // pinned staging for p25cu_poll / p25cu_poll_view (grown on demand)
    size_t h_events_cap;
    // packed polls: two mapped pinned buffers the pack kernel writes straight into (the stores are the transfer)
    unsigned* h_ring[2];
    unsigned* h_tot[2];        // 4 words each: events, words, overflow, truncated
    cudaEvent_t ev_poll[2];
    int poll_fence;            // slot + 1 of a started poll whose compaction the next walker on ctx->stream has not been ordered behind yet
    size_t ring_cap_words;
    int ring_head, ring_pending;
    unsigned long long a_abs;  // input samples consumed per stream
    unsigned long long p_abs;  // baseband samples decoded per stream
    size_t last_n_out;
    bool dev_bb_fresh;
    unsigned undecoded;        // device-resident chunks demodulated since the last decode
    unsigned long long launches;
    int n_sm;
    // wideband channelizer mode (decimation 400): input rows are captures, streams are their channels
    unsigned n_captures;       // 0 = one stream per input row
    float* d_pfb_taps;
    float2* d_twiddle;
    float2* d_y;               // [captures][y_rows][1536] channel-filtered spectra of the last chunk (test hook, lazy)
    unsigned y_rows;
    int keep_spectra;
};

static thread_local char g_create_err[512] = "";

#define CK(call)                                                                                         \
    do {                                                                                                 \
        cudaError_t e_ = (call);                                                                         \
        if (e_ != cudaSuccess) {                                                                         \
            snprintf(ctx->err, sizeof ctx->err, "%s:%d %s: %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); \
            return P25CU_ERR_CUDA;                                                                       \
        }                                                                                                \
    } while (0)

static int fail_arg(p25cu_ctx* ctx, const char* msg) {
    snprintf(ctx->err, sizeof ctx->err, "%s", msg);
    return P25CU_ERR_ARG;
}

extern "C" const char* p25cu_last_error(const p25cu_ctx* ctx) { return ctx ? ctx->err : g_create_err; }

extern "C" void p25cu_destroy(p25cu_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->cfg.device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    if (ctx->stream2) cudaStreamSynchronize(ctx->stream2);
    if (ctx->stream_copy) cudaStreamSynchronize(ctx->stream_copy);
    cudaFree(ctx->d_iq[0]);
    cudaFree(ctx->d_iq[1]);
    cudaFree(ctx->d_tail[0]);
    cudaFree(ctx->d_tail[1]);
    cudaFree(ctx->d_bb[0]);
    cudaFree(ctx->d_bb[1]);
    cudaFree(ctx->d_power);
    cudaFree(ctx->d_work);
    for (int i = 0; i < 2 * 128; i++)
        if (ctx->tev[i]) cudaEventDestroy(ctx->tev[i]);
    cudaFree(ctx->d_states);
    cudaFree(ctx->d_slots);
    cudaFree(ctx->d_dense);
    cudaFree(ctx->d_offsets);
    cudaFree(ctx->d_stats);
    cudaFree(ctx->d_tables);
    cudaFree(ctx->d_golay);
    cudaFree(ctx->d_pfb_taps);
    cudaFree(ctx->d_twiddle);
    cudaFree(ctx->d_y);
    cudaFreeHost(ctx->h_events);
    for (int i = 0; i < 2; i++) {
        if (ctx->ev_bb_ready[i]) cudaEventDestroy(ctx->ev_bb_ready[i]);
        if (ctx->ev_bb_free[i]) cudaEventDestroy(ctx->ev_bb_free[i]);
        if (ctx->ev_iq_ready[i]) cudaEventDestroy(ctx->ev_iq_ready[i]);
        if (ctx->ev_iq_free[i]) cudaEventDestroy(ctx->ev_iq_free[i]);
        if (ctx->ev_poll[i]) cudaEventDestroy(ctx->ev_poll[i]);
        cudaFreeHost(ctx->h_ring[i]);
        cudaFreeHost(ctx->h_tot[i]);
    }
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    if (ctx->stream2) cudaStreamDestroy(ctx->stream2);
    if (ctx->stream_copy) cudaStreamDestroy(ctx->stream_copy);
    delete ctx;
}

static int create_impl(p25cu_ctx* ctx) {
    const p25cu_config& cfg = ctx->cfg;
    int ndev = 0;
    CK(cudaGetDeviceCount(&ndev));
    if (cfg.device < 0 || cfg.device >= ndev) return fail_arg(ctx, "device ordinal out of range");
    CK(cudaSetDevice(cfg.device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, cfg.device));
    if (prop.major != 10) {
        snprintf(ctx->err, sizeof ctx->err, "device %d is sm_%d%d; this library is built for sm_100a only", cfg.device,
                 prop.major, prop.minor);
        return P25CU_ERR_CUDA;
    }
    ctx->n_sm = prop.multiProcessorCount;
    if (cfg.device >= P25CU_MAX_DEVICES) return fail_arg(ctx, "device ordinal beyond the library's per-device tables");
    {   // function attributes and occupancy are per device: set up once per device, whichever thread gets here first
        std::lock_guard<std::mutex> lk(g_plan_mu);
        if (!g_plan_ok[cfg.device]) {
            P25DevPlan& pl = g_plans[cfg.device];
            memset(&pl, 0, sizeof pl);
            pl.device = cfg.device;
            pl.n_sm = prop.multiProcessorCount;
            CK(p25cu_ddc_plan_device(&pl));
            CK(p25cu_pfb_plan_device(&pl));
            g_plan_ok[cfg.device] = true;
        }
        ctx->plan = &g_plans[cfg.device];
    }
    {   // stream priorities: demod (stream) first, walker (stream2) last
        int lo = 0, hi = 0;
        CK(cudaDeviceGetStreamPriorityRange(&lo, &hi));
        CK(cudaStreamCreateWithPriority(&ctx->stream, cudaStreamNonBlocking, hi));
        CK(cudaStreamCreateWithPriority(&ctx->stream2, cudaStreamNonBlocking, lo));
        CK(cudaStreamCreateWithFlags(&ctx->stream_copy, cudaStreamNonBlocking));
    }
    for (int i = 0; i < 2; i++) {
        CK(cudaEventCreateWithFlags(&ctx->ev_bb_ready[i], cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&ctx->ev_bb_free[i], cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&ctx->ev_iq_ready[i], cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&ctx->ev_iq_free[i], cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&ctx->ev_poll[i], cudaEventDisableTiming));
    }
    // The walker runs beside the next chunk's demod kernel only where that kernel is HBM-bound (cf32 /50: issue slots
    // are free); the u8 /50, /5 and channelizer kernels are issue-bound themselves and co-running only slows both (measured).
    ctx->overlap = (cfg.decimation == 50 && cfg.format == P25CU_FMT_CF32_IQ) ? 1 : 0;
    ctx->walk_prefilter = cfg.decimation == (int)p25cu_pfb_decimation() ? 1 : 0;
    if (const char* e = getenv("P25CU_WALK_PREFILTER")) ctx->walk_prefilter = atoi(e) ? 1 : 0;   // A/B switch (same output either way)
    const size_t S = cfg.n_streams;
    const bool wide = cfg.decimation == (int)p25cu_pfb_decimation();
    ctx->n_captures = wide ? cfg.n_streams / p25cu_pfb_channels() : 0;
    ctx->ht = wide ? p25cu_pfb_tail_len() : p25cu_ddc_tail_len(cfg.decimation);
    ctx->max_out = cfg.max_chunk_samples / cfg.decimation + 1;
    if (cfg.max_baseband > ctx->max_out) ctx->max_out = cfg.max_baseband;
    ctx->row_stride = (P25CU_BB_HIST + ctx->max_out + 3) & ~(size_t)3;
    ctx->ev_cap = cfg.event_slots ? cfg.event_slots : (unsigned)(ctx->max_out / 200 + 16);

    const size_t tail_rows = wide ? ctx->n_captures : S;
    CK(cudaMalloc(&ctx->d_tail[0], tail_rows * ctx->ht * sizeof(float2)));
    CK(cudaMalloc(&ctx->d_tail[1], tail_rows * ctx->ht * sizeof(float2)));
    CK(cudaMemsetAsync(ctx->d_tail[0], 0, tail_rows * ctx->ht * sizeof(float2), ctx->stream));
    CK(cudaMemsetAsync(ctx->d_tail[1], 0, tail_rows * ctx->ht * sizeof(float2), ctx->stream));
    if (wide) {
        ctx->y_rows = (unsigned)ctx->max_out;
        CK(p25cu_pfb_upload(&ctx->d_pfb_taps, &ctx->d_twiddle));
    }
    for (int i = 0; i < 2; i++) {
        CK(cudaMalloc(&ctx->d_bb[i], S * ctx->row_stride * sizeof(float)));
        CK(cudaMemsetAsync(ctx->d_bb[i], 0, S * ctx->row_stride * sizeof(float), ctx->stream));
    }
    CK(cudaMalloc(&ctx->d_power, S * sizeof(float)));
    CK(cudaMalloc(&ctx->d_work, 64));
    CK(cudaMemsetAsync(ctx->d_work, 0, 64, ctx->stream));
    if ((unsigned long long)S * ctx->ev_cap * P25CU_SLOT_WORDS >= (1ull << 32))
        return fail_arg(ctx, "n_streams x event_slots too large (event word offsets are 32-bit): poll more often with fewer slots");
    CK(cudaMalloc(&ctx->d_states, S * sizeof(WalkStateHbm)));
    CK(cudaMemsetAsync(ctx->d_states, 0, S * sizeof(WalkStateHbm), ctx->stream));  // state SYNC, pos 0
    CK(cudaMalloc(&ctx->d_slots, S * ctx->ev_cap * P25CU_SLOT_WORDS * sizeof(unsigned)));
    CK(cudaMalloc(&ctx->d_offsets, (2 * S + 4) * sizeof(unsigned)));
    CK(cudaMalloc(&ctx->d_stats, S * P25CU_ST_FAMILIES * 3 * sizeof(unsigned long long)));
    CK(cudaMemsetAsync(ctx->d_stats, 0, S * P25CU_ST_FAMILIES * 3 * sizeof(unsigned long long), ctx->stream));
    CK(cudaMalloc(&ctx->d_tables, sizeof(P25DevTables)));
    {
        P25DevTables* t = new (std::nothrow) P25DevTables;
        if (!t) return fail_arg(ctx, "out of host memory");
        memset(t, 0, sizeof *t);
        p25_fill_tables(t);
        cudaError_t e = cudaMalloc(&ctx->d_golay, sizeof(P25_GOLAY23_SYN));
        if (e == cudaSuccess) e = cudaMemcpy(ctx->d_golay, P25_GOLAY23_SYN, sizeof(P25_GOLAY23_SYN), cudaMemcpyHostToDevice);
        t->golay_syn = ctx->d_golay;
        if (e == cudaSuccess) e = cudaMemcpy(ctx->d_tables, t, sizeof *t, cudaMemcpyHostToDevice);
        delete t;
        CK(e);
    }
    CK(p25cu_ddc_upload_taps());
    CK(p25cu_walk_upload_consts());
    CK(cudaStreamSynchronize(ctx->stream));
    return P25CU_OK;
}

extern "C" int p25cu_create(const p25cu_config* cfg, p25cu_ctx** out) {
    if (!cfg || !out) {
        snprintf(g_create_err, sizeof g_create_err, "null argument");
        return P25CU_ERR_ARG;
    }
    *out = nullptr;
    if (cfg->abi_version != P25CU_ABI_VERSION || cfg->n_streams == 0 || cfg->max_chunk_samples == 0 ||
        cfg->max_chunk_samples > (1ull << 30) || cfg->max_baseband > (1ull << 30) ||   /* kernels index a chunk with 32-bit ints */
        (cfg->decimation != 5 && cfg->decimation != 50 && cfg->decimation != (int)p25cu_pfb_decimation()) ||
        (cfg->format != P25CU_FMT_U8_IQ && cfg->format != P25CU_FMT_CF32_IQ) ||
        (cfg->decimation == (int)p25cu_pfb_decimation() &&
         (cfg->format != P25CU_FMT_CF32_IQ || cfg->n_streams % p25cu_pfb_channels() != 0))) {
        snprintf(g_create_err, sizeof g_create_err,
                 "bad config (abi_version %u, n_streams %u, format %d, decimation %d, max_chunk_samples %llu)",
                 cfg->abi_version, cfg->n_streams, cfg->format, cfg->decimation,
                 (unsigned long long)cfg->max_chunk_samples);
        return P25CU_ERR_ARG;
    }
    p25cu_ctx* ctx = new (std::nothrow) p25cu_ctx;
    if (!ctx) return P25CU_ERR_ARG;
    memset(ctx, 0, sizeof *ctx);
    ctx->cfg = *cfg;
    const int rc = create_impl(ctx);
    if (rc != P25CU_OK) {
        snprintf(g_create_err, sizeof g_create_err, "%s", ctx->err);
        p25cu_destroy(ctx);
        return rc;
    }
    *out = ctx;
    return P25CU_OK;
}

// ---------------------------------------------------------------- Surface 1
extern "C" int p25cu_demod(p25cu_ctx* ctx, const void* iq, size_t n, int iq_on_device, float* baseband_out, size_t* n_out_p,
                           float* power_dbm) {
    if (!ctx) return P25CU_ERR_ARG;
    if (!iq && n) return fail_arg(ctx, "iq is null");
    if (n > ctx->cfg.max_chunk_samples) return fail_arg(ctx, "n_in_per_stream exceeds max_chunk_samples");
    CK(cudaSetDevice(ctx->cfg.device));
    const size_t S = ctx->cfg.n_streams;
    const size_t bps = ctx->cfg.format == P25CU_FMT_U8_IQ ? 2 : 8;
    const size_t in_rows = ctx->n_captures ? ctx->n_captures : S;
    const void* d_in = iq;
    int slot = -1;
    if (!iq_on_device && n) {
        // Host input goes through one of two device staging buffers on the copy stream, so the copy of this chunk runs
        // beside the kernels of the previous one; the call returns once ITS copy is complete (see p25cu.h).
        const size_t bytes = in_rows * n * bps;
        slot = ctx->iq_slot;
        ctx->iq_slot ^= 1;
        if (bytes > ctx->d_iq_bytes[slot]) {
            CK(cudaStreamSynchronize(ctx->stream));           // the kernel that last read this buffer
            cudaFree(ctx->d_iq[slot]);
            ctx->d_iq[slot] = nullptr;
            ctx->d_iq_bytes[slot] = 0;
            CK(cudaMalloc(&ctx->d_iq[slot], bytes));
            ctx->d_iq_bytes[slot] = bytes;
        }
        CK(cudaStreamWaitEvent(ctx->stream_copy, ctx->ev_iq_free[slot], 0));
        CK(cudaMemcpyAsync(ctx->d_iq[slot], iq, bytes, cudaMemcpyHostToDevice, ctx->stream_copy));
        CK(cudaEventRecord(ctx->ev_iq_ready[slot], ctx->stream_copy));
        CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_iq_ready[slot], 0));
        d_in = ctx->d_iq[slot];
    }
    const unsigned D = (unsigned)ctx->cfg.decimation;
    DdcParams p;
    memset(&p, 0, sizeof p);
    p.plan = ctx->plan;
    p.iq = d_in;
    p.tail_in = ctx->d_tail[ctx->tail_cur];
    p.tail_out = ctx->d_tail[ctx->tail_cur ^ 1];
    const int buf = ctx->bb_cur;
    CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_bb_free[buf], 0));   // the walker that last read this buffer is done
    p.bb = ctx->d_bb[buf];
    p.row_stride = ctx->row_stride;
    p.power_sum = power_dbm ? ctx->d_power : nullptr;
    p.a0 = ctx->a_abs;
    p.m0 = ctx->a_abs / D;
    p.n = (unsigned)n;
    p.n_out = (unsigned)((ctx->a_abs + n) / D - p.m0);
    p.n_streams = (unsigned)S;
    p.ht = ctx->ht;
    p.work_counter = ctx->d_work;
    p.ticket_base = &ctx->ticket_base;
    // every stream's row must start 16-byte aligned: 2 cf32 or 8 u8 samples per 16-byte load
    p.aligned16 = ((n % (ctx->cfg.format == P25CU_FMT_U8_IQ ? 8 : 2)) == 0) && (((uintptr_t)d_in & 15) == 0);
    if (power_dbm) CK(cudaMemsetAsync(ctx->d_power, 0, S * sizeof(float), ctx->stream));
    const bool timed = ctx->timing && n && ctx->n_timed < 128;
    if (timed) CK(cudaEventRecord(ctx->tev[2 * ctx->n_timed], ctx->stream));
    if (n && ctx->n_captures) {
        // wideband capture -> 1,536 channels per capture (pfb.cu): one cluster kernel writes the per-channel baseband rows; the carried state is the input tail
        const size_t ch = p25cu_pfb_channels();
        unsigned nl = 0;
        if (ctx->keep_spectra && !ctx->d_y) CK(cudaMalloc(&ctx->d_y, (size_t)ctx->n_captures * ctx->y_rows * ch * sizeof(float2)));
        CK(p25cu_launch_pfb(d_in, p.tail_in, p.tail_out, ctx->d_pfb_taps, ctx->d_twiddle, ctx->keep_spectra ? ctx->d_y : nullptr,
                            ctx->y_rows, p.bb, p.row_stride, p.power_sum, p.a0, p.m0, p.n, p.n_out, ctx->n_captures, ctx->stream, &nl,
                            ctx->plan));
        ctx->launches += nl;
        ctx->tail_cur ^= 1;
    } else if (n) {
        CK(p25cu_launch_ddc(p, ctx->cfg.format, ctx->cfg.decimation, ctx->stream));
        ctx->launches++;
        ctx->tail_cur ^= 1;
    }
    if (timed) CK(cudaEventRecord(ctx->tev[2 * ctx->n_timed++ + 1], ctx->stream));
    if (slot >= 0) CK(cudaEventRecord(ctx->ev_iq_free[slot], ctx->stream));
    CK(cudaEventRecord(ctx->ev_bb_ready[buf], ctx->stream));
    ctx->bb_last = buf;
    ctx->bb_cur = buf ^ 1;
    ctx->a_abs += n;
    ctx->last_n_out = p.n_out;
    ctx->dev_bb_fresh = true;
    ctx->undecoded++;
    if (n_out_p) *n_out_p = p.n_out;
    if (baseband_out && p.n_out)
        CK(cudaMemcpy2DAsync(baseband_out, p.n_out * sizeof(float), ctx->d_bb[buf] + P25CU_BB_HIST, ctx->row_stride * sizeof(float),
                             p.n_out * sizeof(float), S, cudaMemcpyDeviceToHost, ctx->stream));
    if (power_dbm) {
        CK(cudaMemcpyAsync(power_dbm, ctx->d_power, S * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        for (size_t s = 0; s < S; s++) {  // reference src/demod.rs:123-134 with R = 1
            const float avg = p.n_out ? power_dbm[s] / (float)p.n_out : 0.f;
            power_dbm[s] = 30.0f + 10.0f * log10f(avg);
        }
    } else if (baseband_out) {
        CK(cudaStreamSynchronize(ctx->stream));
    } else if (slot >= 0) {
        CK(cudaEventSynchronize(ctx->ev_iq_ready[slot]));     // the caller may reuse its buffer as soon as this call returns
    }
    return P25CU_OK;
}

// ---------------------------------------------------------------- Surface 2
extern "C" int p25cu_decode(p25cu_ctx* ctx, const float* baseband, size_t n) {
    if (!ctx) return P25CU_ERR_ARG;
    CK(cudaSetDevice(ctx->cfg.device));
    const size_t S = ctx->cfg.n_streams;
    int buf;
    if (baseband) {
        if (n > ctx->max_out) return fail_arg(ctx, "n_per_stream exceeds the configured maximum");
        buf = ctx->bb_cur;
        CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_bb_free[buf], 0));
        if (n)
            CK(cudaMemcpy2DAsync(ctx->d_bb[buf] + P25CU_BB_HIST, ctx->row_stride * sizeof(float), baseband, n * sizeof(float),
                                 n * sizeof(float), S, cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaEventRecord(ctx->ev_bb_ready[buf], ctx->stream));
        ctx->bb_cur = buf ^ 1;
    } else {
        if (!ctx->dev_bb_fresh) {
            snprintf(ctx->err, sizeof ctx->err, "p25cu_decode(NULL): no undecoded device-resident baseband (call p25cu_demod first)");
            return P25CU_ERR_STATE;
        }
        if (ctx->undecoded > 1 && ctx->p_abs) {
            // the walker's 256-sample history and its absolute sample index assume every demodulated chunk is decoded
            snprintf(ctx->err, sizeof ctx->err, "p25cu_decode(NULL): %u demodulated chunks since the last decode; only the "
                     "newest is still on the device (decode after every p25cu_demod, or use p25cu_process)", ctx->undecoded);
            return P25CU_ERR_STATE;
        }
        buf = ctx->bb_last;
        n = ctx->last_n_out;
    }
    ctx->dev_bb_fresh = false;
    ctx->undecoded = 0;
    cudaStream_t ws = ctx->overlap ? ctx->stream2 : ctx->stream;
    CK(cudaStreamWaitEvent(ws, ctx->ev_bb_ready[buf], 0));
    if (ctx->poll_fence) {
        // an asynchronous poll (p25cu_poll_start) compacts on stream2 and resets the streams' event counters there: a walker
        // on the other stream must not load those counters before it has finished (found by compute-sanitizer's timing:
        // events of chunk k delivered twice)
        if (ws != ctx->stream2) CK(cudaStreamWaitEvent(ws, ctx->ev_poll[ctx->poll_fence - 1], 0));
        ctx->poll_fence = 0;
    }
    WalkParams w;
    memset(&w, 0, sizeof w);
    w.bb = ctx->d_bb[buf];
    w.bb_next = ctx->d_bb[buf ^ 1];
    w.row_stride = ctx->row_stride;
    w.p0 = ctx->p_abs;
    w.n = (unsigned)n;
    w.n_streams = (unsigned)S;
    w.states = ctx->d_states;
    w.slots = ctx->d_slots;
    w.ev_cap = ctx->ev_cap;
    w.stats = ctx->d_stats;
    w.tables = ctx->d_tables;
    // Overlap mode: the walker of chunk k runs beside the demod kernel of chunk k + 1, whose persistent grid holds
    // 3 CTAs x 320 threads x 56 allocated registers per SM.  Two 64-thread walker CTAs fit in the registers that are
    // left (a third would keep a demod CTA from becoming resident: measured 0.51 vs 0.57 ms per step), so the walker
    // is launched as a persistent grid of 2 CTAs per SM that walks the streams in several passes.
    constexpr unsigned walk_ctas_per_sm = 2;
    CK(p25cu_launch_walk(w, ws, ctx->overlap ? (unsigned)ctx->n_sm * walk_ctas_per_sm : 0u, ctx->cfg.device, ctx->walk_prefilter != 0));
    CK(cudaEventRecord(ctx->ev_bb_free[buf], ws));
    if (!ctx->overlap) CK(cudaStreamWaitEvent(ctx->stream2, ctx->ev_bb_free[buf], 0));   // keep stream2 consumers ordered
    ctx->launches++;
    ctx->p_abs += n;
    return P25CU_OK;
}

extern "C" int p25cu_process(p25cu_ctx* ctx, const void* iq, size_t n, int iq_on_device) {
    const int rc = p25cu_demod(ctx, iq, n, iq_on_device, nullptr, nullptr, nullptr);
    if (rc != P25CU_OK) return rc;
    return p25cu_decode(ctx, nullptr, 0);
}

// scan (+ expansion into 80-byte records when `expand`) on stream2; returns the totals
static int compact(p25cu_ctx* ctx, bool expand, unsigned* total, unsigned* overflow) {
    const unsigned S = ctx->cfg.n_streams;
    if (expand && !ctx->d_dense) CK(cudaMalloc(&ctx->d_dense, (size_t)S * ctx->ev_cap * sizeof(p25cu_event)));
    CK(p25cu_launch_compact(ctx->d_states, ctx->d_slots, ctx->ev_cap, S, ctx->d_offsets, expand ? 1 : 0, ctx->d_dense, nullptr, 0,
                            nullptr, ctx->stream2));
    ctx->launches += expand ? 2 : 1;
    unsigned tail[4];
    CK(cudaMemcpyAsync(tail, ctx->d_offsets + 2 * (size_t)S, sizeof tail, cudaMemcpyDeviceToHost, ctx->stream2));
    CK(cudaStreamSynchronize(ctx->stream2));
    *total = tail[0];
    *overflow = tail[2];
    return P25CU_OK;
}

static int no_started_poll(p25cu_ctx* ctx, const char* who) {
    if (!ctx->ring_pending) return P25CU_OK;
    snprintf(ctx->err, sizeof ctx->err, "%s: a poll started with p25cu_poll_start is outstanding; collect it with p25cu_poll_packed first", who);
    return P25CU_ERR_STATE;
}

extern "C" int p25cu_pending(p25cu_ctx* ctx, size_t* n) {
    if (!ctx || !n) return P25CU_ERR_ARG;
    CK(cudaSetDevice(ctx->cfg.device));
    unsigned total, ovf;
    const int rc = compact(ctx, false, &total, &ovf);
    if (rc != P25CU_OK) return rc;
    *n = total;
    return P25CU_OK;
}

// compaction + D2H of all queued events, as 80-byte records, into the pinned staging buffer
static int drain(p25cu_ctx* ctx, unsigned* total_p) {
    unsigned total, ovf;
    int rc = no_started_poll(ctx, "p25cu_poll");
    if (rc != P25CU_OK) return rc;
    rc = compact(ctx, true, &total, &ovf);
    if (rc != P25CU_OK) return rc;
    if (total > ctx->h_events_cap) {
        cudaFreeHost(ctx->h_events);
        ctx->h_events = nullptr;
        ctx->h_events_cap = 0;
        const size_t cap = (size_t)total + total / 2 + 1024;
        CK(cudaHostAlloc((void**)&ctx->h_events, cap * sizeof(p25cu_event), cudaHostAllocDefault));
        ctx->h_events_cap = cap;
    }
    if (total) {
        CK(cudaMemcpyAsync(ctx->h_events, ctx->d_dense, (size_t)total * sizeof(p25cu_event), cudaMemcpyDeviceToHost, ctx->stream2));
        CK(cudaStreamSynchronize(ctx->stream2));
    }
    *total_p = total;
    if (ovf) {
        snprintf(ctx->err, sizeof ctx->err, "event slot overflow: events were dropped (raise event_slots)");
        return P25CU_ERR_OVERFLOW;
    }
    return P25CU_OK;
}

extern "C" int p25cu_poll_view(p25cu_ctx* ctx, const p25cu_event** events, size_t* n) {
    if (!ctx || !events || !n) return P25CU_ERR_ARG;
    CK(cudaSetDevice(ctx->cfg.device));
    unsigned total = 0;
    const int rc = drain(ctx, &total);
    *events = ctx->h_events;
    *n = total;
    return rc;
}

extern "C" int p25cu_poll(p25cu_ctx* ctx, p25cu_event* out, size_t cap, size_t* n) {
    if (!ctx || !n || (!out && cap)) return P25CU_ERR_ARG;
    CK(cudaSetDevice(ctx->cfg.device));
    unsigned total = 0;
    const int rc = drain(ctx, &total);
    if (rc != P25CU_OK && rc != P25CU_ERR_OVERFLOW) return rc;
    const size_t take = total < cap ? total : cap;
    if (take) memcpy(out, ctx->h_events, take * sizeof(p25cu_event));
    *n = take;
    if (take < total) {
        snprintf(ctx->err, sizeof ctx->err, "event overflow: %u queued, %zu returned (cap too small)", total, take);
        return P25CU_ERR_OVERFLOW;
    }
    return rc;
}

// ---- packed polls: compaction writes variable-length records straight into mapped pinned host memory, asynchronously
#ifndef P25CU_POLL_RING_MAX_BYTES
#define P25CU_POLL_RING_MAX_BYTES ((size_t)256 << 20)
#endif
extern "C" int p25cu_poll_start(p25cu_ctx* ctx) {
    if (!ctx) return P25CU_ERR_ARG;
    CK(cudaSetDevice(ctx->cfg.device));
    if (ctx->ring_pending >= 2) {
        snprintf(ctx->err, sizeof ctx->err, "p25cu_poll_start: two polls are already outstanding; collect one with p25cu_poll_packed");
        return P25CU_ERR_STATE;
    }
    const unsigned S = ctx->cfg.n_streams;
    if (!ctx->h_ring[0]) {
        size_t bytes = (size_t)S * ctx->ev_cap * P25CU_SLOT_WORDS * sizeof(unsigned);
        if (bytes > P25CU_POLL_RING_MAX_BYTES) bytes = P25CU_POLL_RING_MAX_BYTES;
        if (bytes < 4096) bytes = 4096;
        for (int i = 0; i < 2; i++) {
            CK(cudaHostAlloc((void**)&ctx->h_ring[i], bytes, cudaHostAllocMapped | cudaHostAllocPortable));
            CK(cudaHostAlloc((void**)&ctx->h_tot[i], 64, cudaHostAllocMapped | cudaHostAllocPortable));
        }
        ctx->ring_cap_words = bytes / sizeof(unsigned);
    }
    if (const char* e = getenv("P25CU_POLL_RING_WORDS")) {   // test hook: a smaller capacity exercises the `more` path
        const size_t w = (size_t)atoll(e);
        if (w >= 32 && w < ctx->ring_cap_words) ctx->ring_cap_words = w;
    }
    const int slot = (ctx->ring_head + ctx->ring_pending) & 1;
    unsigned *d_ring = nullptr, *d_tot = nullptr;
    CK(cudaHostGetDevicePointer((void**)&d_ring, ctx->h_ring[slot], 0));
    CK(cudaHostGetDevicePointer((void**)&d_tot, ctx->h_tot[slot], 0));
    CK(p25cu_launch_compact(ctx->d_states, ctx->d_slots, ctx->ev_cap, S, ctx->d_offsets, 2, nullptr, d_ring, ctx->ring_cap_words,
                            d_tot, ctx->stream2));
    ctx->launches += 2;
    CK(cudaEventRecord(ctx->ev_poll[slot], ctx->stream2));
    ctx->poll_fence = slot + 1;
    ctx->ring_pending++;
    return P25CU_OK;
}

extern "C" int p25cu_poll_packed(p25cu_ctx* ctx, const uint32_t** words, size_t* n_words, size_t* n_events, int* more) {
    if (!ctx || !words || !n_words) return P25CU_ERR_ARG;
    if (!ctx->ring_pending) {
        const int rc = p25cu_poll_start(ctx);
        if (rc != P25CU_OK) return rc;
    }
    CK(cudaSetDevice(ctx->cfg.device));
    const int slot = ctx->ring_head;
    CK(cudaEventSynchronize(ctx->ev_poll[slot]));
    ctx->ring_head ^= 1;
    ctx->ring_pending--;
    const unsigned* t = ctx->h_tot[slot];
    *words = ctx->h_ring[slot];
    *n_words = t[1];
    if (n_events) *n_events = t[0];
    if (more) *more = (int)t[3];
    if (t[2]) {
        snprintf(ctx->err, sizeof ctx->err, "event slot overflow: events were dropped (raise event_slots)");
        return P25CU_ERR_OVERFLOW;
    }
    return P25CU_OK;
}

// host-side expansion of packed records (byte shuffling only)
extern "C" int p25cu_unpack_events(const uint32_t* words, size_t n_words, p25cu_event* out, size_t cap, size_t* n) {
    if ((!words && n_words) || (!out && cap) || !n) return P25CU_ERR_ARG;
    size_t cur = 0, k = 0;
    while (cur + 3 <= n_words) {
        const uint32_t w2 = words[cur + 2];
        const uint32_t len = w2 >> 24, nw = p25cu_packed_words(len);
        if (len > sizeof out->payload || cur + nw > n_words) return P25CU_ERR_ARG;
        if (k < cap) {
            p25cu_event& e = out[k];
            e.stream = words[cur];
            e.kind = (w2 >> 16) & 0xFFu;
            e.sample = (uint64_t)words[cur + 1] | ((uint64_t)(w2 & 0xFFFFu) << 32);
            e.len = len;
            memset(e.payload, 0, sizeof e.payload);
            memcpy(e.payload, words + cur + 3, len);
        }
        k++;
        cur += nw;
    }
    *n = k < cap ? k : cap;
    return (cur != n_words) ? P25CU_ERR_ARG : (k > cap ? P25CU_ERR_OVERFLOW : P25CU_OK);
}

// ---- pinned host buffers for the caller's sample chunks (the reference's buffer pools: src/demod.rs:63, :103;
//      src/sdr.rs:25-33).  Copies from pinned memory are asynchronous DMA at full PCIe rate; pageable memory is staged
//      by the driver.
extern "C" int p25cu_host_alloc(p25cu_ctx* ctx, size_t bytes, void** out) {
    if (!ctx || !out || !bytes) return P25CU_ERR_ARG;
    CK(cudaSetDevice(ctx->cfg.device));
    CK(cudaHostAlloc(out, bytes, cudaHostAllocPortable));
    return P25CU_OK;
}
extern "C" int p25cu_host_free(p25cu_ctx* ctx, void* p) {
    if (!ctx) return P25CU_ERR_ARG;
    CK(cudaSetDevice(ctx->cfg.device));
    CK(cudaStreamSynchronize(ctx->stream_copy));
    CK(cudaFreeHost(p));
    return P25CU_OK;
}
extern "C" int p25cu_host_register(p25cu_ctx* ctx, void* p, size_t bytes) {
    if (!ctx || !p || !bytes) return P25CU_ERR_ARG;
    CK(cudaSetDevice(ctx->cfg.device));
    CK(cudaHostRegister(p, bytes, cudaHostRegisterPortable));
    return P25CU_OK;
}
extern "C" int p25cu_host_unregister(p25cu_ctx* ctx, void* p) {
    if (!ctx || !p) return P25CU_ERR_ARG;
    CK(cudaSetDevice(ctx->cfg.device));
    CK(cudaStreamSynchronize(ctx->stream_copy));
    CK(cudaHostUnregister(p));
    return P25CU_OK;
}

extern "C" int p25cu_resync(p25cu_ctx* ctx, uint32_t stream) {
    if (!ctx || stream >= ctx->cfg.n_streams) return P25CU_ERR_ARG;
    CK(cudaSetDevice(ctx->cfg.device));
    const unsigned one = 1;
    CK(cudaMemcpyAsync((char*)(ctx->d_states + stream) + offsetof(WalkHeader, resync_req), &one, sizeof one,
                       cudaMemcpyHostToDevice, ctx->stream2));
    CK(cudaStreamSynchronize(ctx->stream2));
    return P25CU_OK;
}

extern "C" int p25cu_get_stats(p25cu_ctx* ctx, uint32_t stream, p25cu_stats* out, int clear) {
    if (!ctx || !out || stream >= ctx->cfg.n_streams) return P25CU_ERR_ARG;
    CK(cudaSetDevice(ctx->cfg.device));
    unsigned long long raw[P25CU_ST_FAMILIES * 3];
    unsigned long long* src = ctx->d_stats + (size_t)stream * P25CU_ST_FAMILIES * 3;
    CK(cudaMemcpyAsync(raw, src, sizeof raw, cudaMemcpyDeviceToHost, ctx->stream2));
    if (clear) CK(cudaMemsetAsync(src, 0, sizeof raw, ctx->stream2));
    CK(cudaStreamSynchronize(ctx->stream2));
    for (int f = 0; f < P25CU_ST_FAMILIES; f++) {
        out->code[f].words = raw[3 * f];
        out->code[f].errs = raw[3 * f + 1];
        out->code[f].size = P25_STATS_SIZE[f];
        out->code[f].fixed = raw[3 * f + 2];
    }
    return P25CU_OK;
}

// ---------------------------------------------------------------- measurement helpers
extern "C" void* p25cu_cuda_stream(p25cu_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }
extern "C" int p25cu_sync(p25cu_ctx* ctx) {
    if (!ctx) return P25CU_ERR_ARG;
    CK(cudaSetDevice(ctx->cfg.device));
    CK(cudaStreamSynchronize(ctx->stream_copy));
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream2));
    return P25CU_OK;
}
extern "C" int p25cu_set_overlap(p25cu_ctx* ctx, int on) {
    if (!ctx) return P25CU_ERR_ARG;
    CK(cudaSetDevice(ctx->cfg.device));
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream2));
    ctx->overlap = on ? 1 : 0;
    return P25CU_OK;
}
extern "C" uint64_t p25cu_launch_count(const p25cu_ctx* ctx) { return ctx ? ctx->launches : 0; }
extern "C" int p25cu_demod_timing(p25cu_ctx* ctx, int enable, double* avg_ms, unsigned* count) {
    if (!ctx) return P25CU_ERR_ARG;
    CK(cudaSetDevice(ctx->cfg.device));
    CK(cudaStreamSynchronize(ctx->stream));
    double sum = 0.0;
    for (unsigned i = 0; i < ctx->n_timed; i++) {
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, ctx->tev[2 * i], ctx->tev[2 * i + 1]));
        sum += ms;
    }
    if (avg_ms) *avg_ms = ctx->n_timed ? sum / ctx->n_timed : 0.0;
    if (count) *count = ctx->n_timed;
    ctx->n_timed = 0;
    if (enable && !ctx->tev[0])
        for (int i = 0; i < 2 * 128; i++) CK(cudaEventCreate(&ctx->tev[i]));
    ctx->timing = enable ? 1 : 0;
    return P25CU_OK;
}
extern "C" int p25cu_device_baseband(p25cu_ctx* ctx, const float** ptr, size_t* row_stride, size_t* n_out) {
    if (!ctx || !ptr) return P25CU_ERR_ARG;
    *ptr = ctx->d_bb[ctx->bb_last] + P25CU_BB_HIST;
    if (row_stride) *row_stride = ctx->row_stride;
    if (n_out) *n_out = ctx->last_n_out;
    return P25CU_OK;
}

extern "C" int p25cu_read_baseband(p25cu_ctx* ctx, uint32_t stream, float* out, size_t n) {
    if (!ctx || !out || stream >= ctx->cfg.n_streams || n > ctx->last_n_out) return P25CU_ERR_ARG;
    CK(cudaSetDevice(ctx->cfg.device));
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaMemcpy(out, ctx->d_bb[ctx->bb_last] + (size_t)stream * ctx->row_stride + P25CU_BB_HIST, n * sizeof(float),
                  cudaMemcpyDeviceToHost));
    return P25CU_OK;
}

extern "C" int p25cu_set_keep_spectra(p25cu_ctx* ctx, int on) {
    if (!ctx) return P25CU_ERR_ARG;
    if (!ctx->n_captures) {
        snprintf(ctx->err, sizeof ctx->err, "p25cu_set_keep_spectra: context is not in channelizer mode (decimation 400)");
        return P25CU_ERR_STATE;
    }
    ctx->keep_spectra = on ? 1 : 0;
    return P25CU_OK;
}

extern "C" int p25cu_channelizer_output(p25cu_ctx* ctx, float* out, size_t* n_rows) {
    if (!ctx || !n_rows) return P25CU_ERR_ARG;
    if (!ctx->n_captures || !ctx->keep_spectra || !ctx->d_y) {
        snprintf(ctx->err, sizeof ctx->err, "p25cu_channelizer_output: needs channelizer mode (decimation 400) and "
                 "p25cu_set_keep_spectra(ctx, 1) before the p25cu_demod whose spectra are wanted");
        return P25CU_ERR_STATE;
    }
    CK(cudaSetDevice(ctx->cfg.device));
    *n_rows = ctx->last_n_out;
    if (out && ctx->last_n_out) {
        const size_t ch = p25cu_pfb_channels(), row = ch * sizeof(float2);
        CK(cudaMemcpy2DAsync(out, ctx->last_n_out * row, ctx->d_y, (size_t)ctx->y_rows * row, ctx->last_n_out * row, ctx->n_captures,
                             cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    }
    return P25CU_OK;
}

// ---------------------------------------------------------------- FEC unit entry point
extern "C" int p25cu_fec_selftest(p25cu_ctx* ctx, int kind, void* words, size_t count, int n, int k, void* out_data,
                                  int32_t* out_nerr) {
    if (!ctx || !words || !out_nerr || kind < 0 || kind > 15) return P25CU_ERR_ARG;
    const int base_kind = kind == 10 ? 7 : kind == 11 ? 9 : kind == 12 ? 0 : kind == 13 ? 8 : kind == 15 ? 14 : kind;
    if (base_kind == 7 && (n < 1 || n > 36 || k < 1 || k >= n || ((n - k) != 8 && (n - k) != 12 && (n - k) != 16)))
        return fail_arg(ctx, "rs selftest: unsupported (n, k)");
    if (base_kind != 7 && !out_data) return P25CU_ERR_ARG;
    CK(cudaSetDevice(ctx->cfg.device));
    size_t in_b, out_b;
    switch (base_kind) {
        case 0: in_b = 8; out_b = 4; break;
        case 7: in_b = (size_t)n; out_b = 0; break;
        case 8: in_b = 98; out_b = 12; break;
        case 9: in_b = 72; out_b = 60; break;
        case 14: in_b = 98; out_b = 18; break;
        default: in_b = 4; out_b = 4; break;
    }
    void *d_in = nullptr, *d_out = nullptr;
    int32_t* d_nerr = nullptr;
    int rc = P25CU_OK;
    cudaError_t e;
#define CKF(call) if ((e = (call)) != cudaSuccess) { snprintf(ctx->err, sizeof ctx->err, "%s: %s", #call, cudaGetErrorString(e)); rc = P25CU_ERR_CUDA; goto done; }
    if (count == 0) return P25CU_OK;
    CKF(cudaMalloc(&d_in, count * in_b));
    CKF(cudaMalloc(&d_nerr, count * sizeof(int32_t)));
    if (out_b) CKF(cudaMalloc(&d_out, count * out_b));
    CKF(cudaMemcpyAsync(d_in, words, count * in_b, cudaMemcpyHostToDevice, ctx->stream));
    CKF(p25cu_launch_fec_selftest(ctx->d_tables, kind, d_in, count, n, k, d_out, d_nerr, ctx->stream));
    ctx->launches++;
    if (base_kind == 7) CKF(cudaMemcpyAsync(words, d_in, count * in_b, cudaMemcpyDeviceToHost, ctx->stream));
    if (out_b) CKF(cudaMemcpyAsync(out_data, d_out, count * out_b, cudaMemcpyDeviceToHost, ctx->stream));
    CKF(cudaMemcpyAsync(out_nerr, d_nerr, count * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    CKF(cudaStreamSynchronize(ctx->stream));
done:
    cudaFree(d_in);
    cudaFree(d_out);
    cudaFree(d_nerr);
    return rc;
}
