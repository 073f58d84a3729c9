// p25cu_internal.cuh -- structures shared by the kernels and the C ABI (not installed).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/p25cu.h"
#include "p25_fec.cuh"

// ---------------------------------------------------------------------------
// Data layout in HBM (DESIGN.md section 3)
//
//   iq chunk      [S][n]            cf32 (8 B) or u8 pairs (2 B), stream-major (caller's layout)
//   iq tail       2 x [S][HT]       samples in the stream's own format, last HT inputs of every stream (ping-pong)
//   baseband      [S][row_stride]   f32; row = 256-sample history | this chunk's samples
//   walker state  [S]               WalkStateHbm, 352 B per stream (header + the unit in flight, 4 dibits per byte)
//   event slots   [S][ev_cap * 20]  u32 words: packed variable-length records (3 header words + payload words)
//   event dense   [sum]             (stream, sample)-ordered copy for the host: 80-byte records or packed words
//   stats         [S][12][3]        u64 words / errs / fixed
// ---------------------------------------------------------------------------
#define P25CU_BB_HIST 256          // baseband history kept in front of every row (>= 231 + lock margin)
#define P25CU_MAX_DEVICES 64       // device ordinals the per-device tables cover
#define P25CU_WALK_WARPS 2         // streams (warps) per walker CTA: small enough to co-reside with 3 ddc_fm CTAs per SM
#define P25CU_SLOT_WORDS 20        // u32 words reserved per event slot (the longest packed record takes 18)
#define P25CU_BUF_DIBITS 848       // dibit buffer of the unit in flight (LDU: 784), a multiple of 16

enum { WS_SYNC = 0, WS_NID = 1, WS_PAYLOAD = 2, WS_FLUSH = 3 };

// Receiver state that persists between chunks, in the order it is kept in HBM.  Field-for-field the state of the
// restated MessageReceiver (oracle/p25_oracle.hpp); the sample history lives in the baseband row.
struct __align__(16) WalkHeader {
    unsigned long long next_sym;  // absolute index of the next symbol instant
    unsigned long long pos;       // SYNC: absolute index of the next sample the detector has not seen
    int state, duid, cnt, blocks, part, chunks;
    int have_prev, prev_above;
    float prev_corr, pth, mid, nth;
    unsigned frame_pos;
    unsigned n_events;            // events queued in this stream's slots since the last poll
    unsigned n_words;             // ... and the u32 words they occupy
    unsigned overflow;
    unsigned resync_req;          // set by p25cu_resync, honoured at the next chunk
    unsigned char hex[40];        // hexbits of the link control / crypto sync word being collected
    unsigned char quiet;          // search steps in a row that held no position above threshold (saturates; walker-internal)
    unsigned char pad_[3];
};
static_assert(sizeof(WalkHeader) == 128, "WalkHeader is 8 x 16 bytes");

// HBM record: header + the data dibits of the unit being received, 4 per byte (dibit i at bits 2 (i & 15) of word i / 16).
// Only the first cnt dibits are meaningful, and only they are read and written back (state NID / PAYLOAD).
struct __align__(16) WalkStateHbm {
    WalkHeader h;
    unsigned packed[P25CU_BUF_DIBITS / 16 + 3];   // 53 words, padded to 56
};
static_assert(sizeof(WalkStateHbm) == 352, "WalkStateHbm layout");

// Working copy in shared memory (one per warp): the header plus the dibits one per byte.
struct __align__(16) WalkState : WalkHeader {
    unsigned char buf[P25CU_BUF_DIBITS];
};

struct WalkParams {
    const float* bb;              // baseband rows
    size_t row_stride;            // floats per row
    unsigned long long p0;        // absolute index of the first sample of this chunk
    unsigned n;                   // samples in this chunk (per stream)
    unsigned n_streams;
    WalkStateHbm* states;
    unsigned* slots;              // [S][ev_cap * P25CU_SLOT_WORDS] packed event records
    unsigned ev_cap;              // events per stream between two polls
    unsigned long long* stats;    // [S][12][3]
    const P25DevTables* tables;
    float* bb_next;               // rows the NEXT chunk will be decoded from: receives the 256-sample history
};

// Packed event record (p25cu.h p25cu_poll_packed): word 0 stream, word 1 sample bits 0..31,
// word 2 = sample bits 32..47 | kind << 16 | len << 24, then ceil(len / 4) payload words.
__host__ __device__ inline unsigned p25cu_packed_words(unsigned len) { return 3u + ((len + 3u) >> 2); }

// Launch geometry of one device.  Function attributes (dynamic shared memory opt-in, carve-out) and occupancy are per
// device, and a process may hold one context per GPU on separate host threads (p25cu.h; reference src/main.rs:254-293
// runs one thread per task), so nothing here is cached in function-local statics: the table is filled once per device
// under a mutex at p25cu_create and every launch reads the plan of its own context's device.
struct P25DevPlan {
    int device;
    int n_sm;
    int grid_ddc50;               // persistent grid of fast::p25_ddc_fm_stream_kernel (cf32 /50)
    int grid_w5;                  // w5::p25_ddc5_warp_kernel (cf32 /5)
    int grid_w50i;                // w50i::p25_ddc50_imma_kernel (u8 /50, both decimating stages on the integer tensor pipe)
    int grid_w5i;                 // w5i::p25_ddc5_imma_kernel (u8, decimator on the integer tensor pipe)
    int pfb_slots;                // resident CTAs of the channelizer kernel
};

struct DdcParams {
    const P25DevPlan* plan;       // launch geometry of the context's device
    const void* iq;               // chunk, [S][n]
    const void* tail_in;          // [S][HT] samples in the stream's own format (uchar2 or float2)
    void* tail_out;               // [S][HT]
    float* bb;                    // baseband rows (outputs start at column P25CU_BB_HIST)
    size_t row_stride;
    float* power_sum;             // [S], atomically accumulated sum |c|^2 of this chunk
    unsigned long long a0;        // absolute input index of the first sample of this chunk
    unsigned long long m0;        // absolute output index of the first output of this chunk
    unsigned n;                   // input samples per stream in this chunk
    unsigned n_out;               // outputs per stream in this chunk
    unsigned n_streams;
    unsigned seg_out;             // generic kernel: outputs per segment (whole blocks), set by its launcher
    unsigned n_seg;               // generic kernel: segments per stream, set by its launcher
    unsigned ht;                  // tail length in samples
    int aligned16;                // every chunk row starts 16-byte aligned and holds whole 16-byte groups
    unsigned* work_counter;       // device ticket counter of the /50 kernel's dynamic work split (monotonic)
    unsigned* ticket_base;        // host: tickets consumed by earlier launches
};

// kernels (defined in ddc_fm.cu / decode_walk.cu)
cudaError_t p25cu_launch_ddc(const DdcParams& p, int format, int decimation, cudaStream_t st);
cudaError_t p25cu_ddc_upload_taps();
unsigned p25cu_ddc_tail_len(int decimation);
cudaError_t p25cu_ddc_plan_device(P25DevPlan* plan);   // per-device attribute setup + occupancy (current device)
cudaError_t p25cu_pfb_plan_device(P25DevPlan* plan);
cudaError_t p25cu_launch_walk(const WalkParams& p, cudaStream_t st, unsigned max_blocks, int device, bool prefilter);
// Event compaction.  offsets: [2 S + 4] = exclusive event offsets | exclusive word offsets | total events, total words,
// overflow flag, truncated flag.  mode 0: count only; 1: expand into 80-byte records at dense80; 2: copy the packed
// words to `packed` (device or mapped host memory, at most cap_words; streams that do not fit stay queued) and mirror
// the four totals to `totals_out` (nullable, mapped host memory).
cudaError_t p25cu_launch_compact(WalkStateHbm* states, const unsigned* slots, unsigned ev_cap, unsigned n_streams,
                                 unsigned* offsets, int mode, p25cu_event* dense80, unsigned* packed, unsigned long long cap_words,
                                 unsigned* totals_out, cudaStream_t st);
cudaError_t p25cu_launch_fec_selftest(const P25DevTables* tables, int kind, void* words, size_t count, int n, int k,
                                      void* out_data, int32_t* out_nerr, cudaStream_t st);
