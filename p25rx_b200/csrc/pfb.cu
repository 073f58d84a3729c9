// pfb.cu -- K1b: wideband polyphase channelizer + per-channel C4FM baseband (BASELINE.json configs[2]).
//
// No stage of the reference does this (one RTL-SDR tuner, one channel, retuned by hopping: reference
// src/sdr.rs:61-68, src/recv.rs:127-137); it is the declared extension SURVEY.md section 2.5 names K1b.  A
// 19.2 MS/s cf32 capture is split into 1,536 channels 12.5 kHz apart, each at 48 kS/s, and every channel
// then runs the reference's own 48 kHz stages:
//   channel-select FIR   reference src/demod.rs:93      (static_fir::FirFilter<BandpassFir>)
//   power accumulation   reference src/demod.rs:95-101
//   FM discriminator     reference src/demod.rs:109-111
//   10-tap moving average reference src/demod.rs:114
// so that the decode walker sees 1,536 ordinary streams per capture.
//
// Channel k is defined (spec/p25_spec.py) as mix-down by k * 12.5 kHz, a 6,144-tap prototype low-pass and
// decimation by 400:   y_k[m] = sum_i h[i] x[n_m - i] exp(-2j pi k (n_m - i) / 1536),  n_m = 400 m + 399.
// Writing i = r + 1536 p gives the polyphase form this file computes:
//   v_m[r] = sum_{p<4} h[r + 1536 p] x[n_m - r - 1536 p]           (4 complex-by-real taps per branch)
//   y_k[m] = sum_q v_m[(q + n_m) mod 1536] exp(+2j pi k q / 1536)   (one 1,536-point inverse DFT per output time)
//
// Round 2 folds the channel-select FIR into the prototype and does everything in ONE kernel (below): polyphase
// branches, inverse DFT, discriminator, boxcar, baseband rows.  HBM traffic is the algorithmic minimum: 8 B per input
// sample in, 4 B per channel and output time out (15.4 B per input sample).
#include <cooperative_groups.h>

#include "p25cu_internal.cuh"
#include "p25_pfb_taps.h"

namespace pfb {

constexpr int N = P25_PFB_N, M = P25_PFB_M, P = P25_PFB_P, L = N * P;
static_assert(N == 3 * 8 * 8 * 8, "FFT plan is 3 x 8 x 8 x 8");

__device__ __forceinline__ float2 cmul(float2 a, float2 b) { return make_float2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x); }
// complex add / subtract on the packed FP32 pipe: one FADD2 each
__device__ __forceinline__ float2 cadd(float2 a, float2 b) {
    unsigned long long r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(*reinterpret_cast<const unsigned long long*>(&a)), "l"(*reinterpret_cast<const unsigned long long*>(&b)));
    return *reinterpret_cast<float2*>(&r);
}
__device__ __forceinline__ float2 csub(float2 a, float2 b) {
    unsigned long long r;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(*reinterpret_cast<const unsigned long long*>(&a)), "l"(*reinterpret_cast<const unsigned long long*>(&b)));
    return *reinterpret_cast<float2*>(&r);
}
__device__ __forceinline__ float2 mul_i(float2 a) { return make_float2(-a.y, a.x); }     // a * (+i)
// acc += h * x on both components: one FFMA2
__device__ __forceinline__ float2 cfma(float h, float2 x, float2 acc) {
    unsigned long long r;
    const float2 hh = make_float2(h, h);
    asm("fma.rn.f32x2 %0, %1, %2, %3;"
        : "=l"(r)
        : "l"(*reinterpret_cast<const unsigned long long*>(&hh)), "l"(*reinterpret_cast<const unsigned long long*>(&x)),
          "l"(*reinterpret_cast<const unsigned long long*>(&acc)));
    return *reinterpret_cast<float2*>(&r);
}

// a * w for a twiddle kept as {w, i w} = {w.x, w.y, -w.y, w.x}: a.x * w + a.y * (i w), one FMUL2 + one FFMA2 (the scalar
// factor rides in the packed instructions' broadcast operand)
__device__ __forceinline__ float2 cmulw(float2 a, float4 w) {
    unsigned long long r;
    const float2 ax = make_float2(a.x, a.x), w0 = make_float2(w.x, w.y);
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(*reinterpret_cast<const unsigned long long*>(&ax)), "l"(*reinterpret_cast<const unsigned long long*>(&w0)));
    return cfma(a.y, make_float2(w.z, w.w), *reinterpret_cast<float2*>(&r));
}
__device__ __forceinline__ float4 twiddle4(float2 w) { return make_float4(w.x, w.y, -w.y, w.x); }

// 8-point DFT with the + sign: w[q] = sum_r v[r] exp(+2 pi i r q / 8), in place
__device__ __forceinline__ void dft8(float2 (&v)[8]) {
    const float h = 0.70710678118654752f;
    // radix-2 decimation in time: evens (0,2,4,6), odds (1,3,5,7)
    float2 e0 = cadd(v[0], v[4]), e1 = csub(v[0], v[4]), e2 = cadd(v[2], v[6]), e3 = mul_i(csub(v[2], v[6]));
    float2 o0 = cadd(v[1], v[5]), o1 = csub(v[1], v[5]), o2 = cadd(v[3], v[7]), o3 = mul_i(csub(v[3], v[7]));
    const float2 E0 = cadd(e0, e2), E2 = csub(e0, e2), E1 = cadd(e1, e3), E3 = csub(e1, e3);   // 4-point DFT of the evens
    const float2 O0 = cadd(o0, o2), O2 = csub(o0, o2), O1 = cadd(o1, o3), O3 = csub(o1, o3);   // ... of the odds
    // odd outputs times exp(+2 pi i q / 8), q = 0..3
    const float2 T0 = O0;
    const float2 T1 = make_float2(h * (O1.x - O1.y), h * (O1.x + O1.y));     // * (1 + i) / sqrt 2
    const float2 T2 = mul_i(O2);
    const float2 T3 = make_float2(-h * (O3.x + O3.y), h * (O3.x - O3.y));    // * (-1 + i) / sqrt 2
    v[0] = cadd(E0, T0);
    v[4] = csub(E0, T0);
    v[1] = cadd(E1, T1);
    v[5] = csub(E1, T1);
    v[2] = cadd(E2, T2);
    v[6] = csub(E2, T2);
    v[3] = cadd(E3, T3);
    v[7] = csub(E3, T3);
}

__device__ __forceinline__ float atan2_branchfree(float y, float x) {   // same polynomial as ddc_fm.cu disc_atan2_pair
    const float ax = fabsf(x), ay = fabsf(y);
    const float mx = fmaxf(ax, ay), mn = fminf(ax, ay);
    float rc;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rc) : "f"(fmaxf(mx, 1e-30f)));
    const float t = mn * rc, u = t * t;
    float q = -0.004295386839658022f;
    q = fmaf(q, u, 0.022737378254532814f);
    q = fmaf(q, u, -0.057179518043994904f);
    q = fmaf(q, u, 0.09735459089279175f);
    q = fmaf(q, u, -0.13945257663726807f);
    q = fmaf(q, u, 0.1995391547679901f);
    q = fmaf(q, u, -0.3333050608634949f);
    q = fmaf(q, u, 0.9999995231628418f);
    float r = q * t;
    r = ay > ax ? 1.57079632679489662f - r : r;
    r = x < 0.f ? 3.14159265358979324f - r : r;
    return copysignf(r, y);
}

__device__ __forceinline__ float2 pk_mul(float2 a, float2 b) {
    unsigned long long r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(*reinterpret_cast<const unsigned long long*>(&a)), "l"(*reinterpret_cast<const unsigned long long*>(&b)));
    return *reinterpret_cast<float2*>(&r);
}
__device__ __forceinline__ float2 pk_fma(float2 a, float2 b, float2 c) {
    unsigned long long r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;"
        : "=l"(r)
        : "l"(*reinterpret_cast<const unsigned long long*>(&a)), "l"(*reinterpret_cast<const unsigned long long*>(&b)),
          "l"(*reinterpret_cast<const unsigned long long*>(&c)));
    return *reinterpret_cast<float2*>(&r);
}
// atan2_branchfree for two independent arguments at once (two consecutive output times of the thread's channel): the
// polynomial runs on the packed pipe
__device__ __forceinline__ float2 atan2x2(float2 y, float2 x) {
    const float2 mx = make_float2(fmaxf(fabsf(x.x), fabsf(y.x)), fmaxf(fabsf(x.y), fabsf(y.y)));
    const float2 mn = make_float2(fminf(fabsf(x.x), fabsf(y.x)), fminf(fabsf(x.y), fabsf(y.y)));
    float2 rc;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rc.x) : "f"(fmaxf(mx.x, 1e-30f)));
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rc.y) : "f"(fmaxf(mx.y, 1e-30f)));
    const float2 t = pk_mul(mn, rc), u = pk_mul(t, t);
#define P25_C2(c) make_float2(c, c)
    float2 q = pk_fma(P25_C2(-0.004295386839658022f), u, P25_C2(0.022737378254532814f));
    q = pk_fma(q, u, P25_C2(-0.057179518043994904f));
    q = pk_fma(q, u, P25_C2(0.09735459089279175f));
    q = pk_fma(q, u, P25_C2(-0.13945257663726807f));
    q = pk_fma(q, u, P25_C2(0.1995391547679901f));
    q = pk_fma(q, u, P25_C2(-0.3333050608634949f));
    q = pk_fma(q, u, P25_C2(0.9999995231628418f));
#undef P25_C2
    float2 r = pk_mul(q, t);
    r.x = fabsf(y.x) > fabsf(x.x) ? 1.57079632679489662f - r.x : r.x;
    r.y = fabsf(y.y) > fabsf(x.y) ? 1.57079632679489662f - r.y : r.y;
    r.x = x.x < 0.f ? 3.14159265358979324f - r.x : r.x;
    r.y = x.y < 0.f ? 3.14159265358979324f - r.y : r.y;
    return make_float2(copysignf(r.x, y.x), copysignf(r.y, y.y));
}

// ------------------------------------------------------------------------------------------------ the kernel
// Round 2 folds the per-channel channel-select FIR (41 taps at 48 kS/s, src/demod.rs:93) into the prototype.  Channel k
// after the channel filter is
//     c_k[m] = sum_j hc[j] y_k[m - j] = sum_i heq[i] x[n_m - i] exp(-2j pi k (n_m - i) / N),
//     heq = hp (*) upsample(hc, M)           (6,144 + 40 * 400 = 22,144 taps, zero-padded to PE * N = 23,040)
// i.e. the same polyphase form with PE = 15 taps per branch instead of 4 -- 23,040 complex-by-real MACs per output time
// for all 1,536 channels, instead of 6,144 + 1,536 * 41 = 69,120 -- and no [time][channel] round trip through HBM.
//
// Every one of those MACs pairs a distinct (sample, tap): nothing is reused, so one of the two has to come out of
// shared memory for every FFMA2.  The first round-2 kernel kept the taps in registers and the 23,040-sample window in a
// 192 KB ring (8 bytes per MAC, one CTA per SM, no room left to batch the FFT).  This one turns it round:
//
//   * CLASS-STATIONARY WINDOWS IN REGISTERS.  The samples that feed FFT input q are exactly those with index
//     s = -q (mod N): a thread owns one such residue class and keeps its newest 16 samples in registers as a
//     circular window.  Per MAC only the 4-byte tap comes from shared memory: the 16 taps that go with a window whose
//     newest sample lies d0 = n_m - s_newest inputs back are one table row, tap[k] = heq[d0 + N k] (zero outside
//     0 .. LE - 1), read with four conflict-free LDS.128.  A class receives a new sample in 400 of every 1,536 output
//     times; the 32 classes of a warp are consecutive samples and always advance TOGETHER, at the output time the first
//     of them needs it -- the others then hold a sample up to 62 inputs "from the future" in their newest slot, which
//     the row for their (negative) d0 multiplies by zero.  So the slot that is overwritten is warp-uniform and the
//     branch sum is a jump over 16 compile-time rotations of the same 16 FFMA2.
//   * A CLUSTER OF TWO CTAs PER RUN OF OUTPUT TIMES.  1,536 windows are 46 K registers -- too many beside an FFT on one
//     SM.  CTA b of the pair owns the classes of parity b: 768 windows (23 K registers), only the tap rows of the
//     opposite parity (n_m is odd: 89 KB instead of 178), and the 768-point inverse DFT over its own inputs
//     (q = 2u + b).  The last radix-2 step   c_k' = E[k'] + w^k' O[k'],  c_k'+768 = E[k'] - w^k' O[k']   reads the
//     partner's half through distributed shared memory; CTA b finishes the channels k' in [384 b, 384 b + 384) and
//     k' + 768.
//   * EIGHT OUTPUT TIMES PER PASS.  The 768-point transforms of eight consecutive output times go through the three
//     Stockham passes 8 x 8 x 12 together (96 / 96 / 64 butterflies per time: 768 / 768 / 512 per batch for 768
//     threads), six CTA barriers per eight output times instead of six per time.  The half of the result the partner
//     needs is stored straight into the partner's shared memory (st.async counting bytes on the partner's mbarrier,
//     two buffers deep), and the branch sums of the NEXT batch are computed before the combine step waits for it.
//   * EVERYTHING AFTER THE FFT IS THREAD-LOCAL.  The combine step leaves every thread with the same channel at every
//     output time: c[m-1] for the FM discriminator (src/demod.rs:109-111) and the power sum (src/demod.rs:95-101)
//     stay in its registers, the nine older discriminator values of the 10-tap boxcar (src/demod.rs:114) in its own
//     column of shared memory, and it writes eight consecutive baseband samples of its channel (32 bytes) straight
//     into the walker's rows.
//   * A run starts with 10 warm-up output times (c[m-1] and nine discriminator values), recomputed from the carried
//     input tail instead of carrying discriminator rows between chunks.
// The index arithmetic is restated thread for thread in spec/pfb_dataflow.py and checked against the float64 oracle on
// the CPU (tests/test_pfb_oracle.py).
constexpr int PE = 15;                 // taps per branch of the equivalent prototype
constexpr int LE = N * PE;             // 23,040
constexpr int H = N / 2;               // FFT length per parity / CTA
constexpr int NTH = 768;               // threads per CTA: one class and one channel each (24 warps: the phases are latency-bound)
constexpr int TB = 8;                  // output times per batch
constexpr int WARM = 10;               // warm-up output times of a run
constexpr int WS = 16;                 // window slots per class: 15 taps + one sample that may be early
constexpr int HTX = 27648;             // carried input tail (>= LE + (WARM + 1) * M + 64, a multiple of 128)
constexpr int EARLY = 64;              // a window's newest sample lies at most this far ahead of n_m (a warp spans 62)
constexpr int ROWS = (N + EARLY) / 2;  // tap rows per CTA: d0 = 2 row - EARLY + (1 - b), d0 in [-EARLY, N)
constexpr int FSK = H + H / 8;         // a time's FFT buffer with pad elements (see skew_a(), skew_b())
static_assert(HTX >= LE + (WARM + 1) * M + EARLY && HTX % 128 == 0, "warm-up windows must lie inside the carried tail");
static_assert(M < N && N - M - 62 > 0, "a class receives at most one new sample per output time");

struct SmemC {
    float4 tab[4][ROWS];               // tab[g][row] = taps 4 g .. 4 g + 3 of the row: tap[k] = heq[d0 + N k] or 0
    float2 f0[TB][FSK];                // polyphase sums -> passes A and B in place
    float2 own[TB][H / 2];             // this CTA's transform at the 384 k' it combines itself
    float2 inc[2][TB][H / 2];          // the partner's transform at the same k', written by the partner (st.async), two batches deep
    float hist[P25_BOXCAR - 1][H];     // the nine discriminator values before the current batch, per channel of this CTA
    unsigned long long mbar[2];        // one transaction barrier per incoming buffer
    float4 twB[8][8];                  // w = exp(+2 pi i k r / 64) at [r][k], as {w, i w} (cmulw)
    float2 twC[12][64];                // w = exp(+2 pi i j r / 768) at [r][j]
};

struct PfbParams {
    const float2* iq;          // [captures][n]
    const float2* tail_in;     // [captures][HTX]
    const float* taps;         // [LE] equivalent prototype (prototype (*) upsampled channel filter)
    const float2* twiddle;     // [N] exp(+2 pi i t / N)
    float* bb;                 // baseband rows, stream = capture * N + channel
    size_t row_stride;
    float2* y;                 // nullable: [captures][y_rows][N] channel-filtered spectra c_k[m] of this chunk (test hook)
    float* power_sum;          // nullable: [captures * N]
    unsigned long long a0, m0; // absolute input / output index of the chunk start
    unsigned n, n_out, n_captures;
    unsigned y_rows;
    unsigned runs_per_cap, times_per_run;      // times_per_run is a multiple of TB
};

// sample at logical index l of (carried tail ++ chunk); zeros outside
__device__ __forceinline__ float2 load_logical(const float2* __restrict__ tail, const float2* __restrict__ chunk, int n, int l) {
    const bool in_chunk = l >= HTX;
    const float2* ptr = in_chunk ? chunk + (l - HTX) : tail + l;
    return (l >= 0 && l < HTX + n) ? __ldg(ptr) : make_float2(0.f, 0.f);
}
// Padded positions inside a time's FFT buffer, chosen so that BOTH sides of every pass are free of bank conflicts:
//   pass A writes 8 j + q (lanes: j) and pass B reads j + 96 r (lanes: j) through skew_a: one pad per 16 elements;
//   pass B writes 64 a + k + 8 q (lanes: a, k) and pass C reads j + 64 r (lanes: j) through skew_b: 8 pads per 64.
// (One pad per eight for both, the first version, made every read span an extra wavefront: 9 % of the kernel's
// shared-memory traffic, which is what bounds it.)
__device__ __forceinline__ int skew_a(int i) { return i + (i >> 4); }
__device__ __forceinline__ int skew_b(int i) { return i + 8 * (i >> 6); }
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
// the partner CTA's copy of a shared-memory address of this CTA
__device__ __forceinline__ unsigned map_to_rank(unsigned addr, unsigned rank) {
    unsigned r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
    return r;
}
// 8-byte store into the partner's shared memory that counts its bytes on the partner's transaction barrier: the data
// path needs no cluster-wide barrier and no fence (a release at cluster scope compiles to MEMBAR.ALL.GPU, an acquire to
// CCTL.IVALL: 18 % of all warp stalls in the first version of this kernel)
__device__ __forceinline__ void st_async_f2(unsigned remote_addr, float2 v, unsigned remote_mbar) {
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v2.f32 [%0], {%1, %2}, [%3];"
                 :: "r"(remote_addr), "f"(v.x), "f"(v.y), "r"(remote_mbar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned mbar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(mbar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned mbar, unsigned parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "P25_MBAR_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra P25_MBAR_DONE;\n"
        "bra P25_MBAR_WAIT;\n"
        "P25_MBAR_DONE:\n"
        "}\n" :: "r"(mbar), "r"(parity) : "memory");
}

// 12-point DFT with the + sign, r = 3 a + b, q = q1 + 4 q2: three 4-point DFTs over a, twiddles W12^(b q1), four
// 3-point DFTs over b.  In place: v[q].
__device__ __forceinline__ void dft12(float2 (&v)[12]) {
    const float c6 = 0.86602540378443865f;          // cos(pi / 6) = sin(pi / 3)
    float2 z[3][4];
#pragma unroll
    for (int b = 0; b < 3; b++) {
        const float2 x0 = v[b], x1 = v[3 + b], x2 = v[6 + b], x3 = v[9 + b];
        const float2 s02 = cadd(x0, x2), d02 = csub(x0, x2), s13 = cadd(x1, x3), d13 = mul_i(csub(x1, x3));
        z[b][0] = cadd(s02, s13);
        z[b][1] = cadd(d02, d13);
        z[b][2] = csub(s02, s13);
        z[b][3] = csub(d02, d13);
    }
    // W12^1 = (c6, 1/2), W12^2 = (1/2, c6), W12^3 = i, W12^4 = (-1/2, c6), W12^6 = -1
    z[1][1] = make_float2(c6 * z[1][1].x - 0.5f * z[1][1].y, c6 * z[1][1].y + 0.5f * z[1][1].x);
    z[1][2] = make_float2(0.5f * z[1][2].x - c6 * z[1][2].y, 0.5f * z[1][2].y + c6 * z[1][2].x);
    z[1][3] = mul_i(z[1][3]);
    z[2][1] = make_float2(0.5f * z[2][1].x - c6 * z[2][1].y, 0.5f * z[2][1].y + c6 * z[2][1].x);
    z[2][2] = make_float2(-0.5f * z[2][2].x - c6 * z[2][2].y, -0.5f * z[2][2].y + c6 * z[2][2].x);
    z[2][3] = make_float2(-z[2][3].x, -z[2][3].y);
#pragma unroll
    for (int q1 = 0; q1 < 4; q1++) {
        const float2 s = cadd(z[1][q1], z[2][q1]), d = csub(z[1][q1], z[2][q1]);
        const float2 mid = make_float2(z[0][q1].x - 0.5f * s.x, z[0][q1].y - 0.5f * s.y);
        const float2 rot = make_float2(-c6 * d.y, c6 * d.x);           // i * c6 * (z1 - z2)
        v[q1] = cadd(z[0][q1], s);
        v[q1 + 4] = cadd(mid, rot);
        v[q1 + 8] = csub(mid, rot);
    }
}

// The output times of one class from this one up to (not including) the next window advance, or the end of the batch:
// the newest sample stays in slot K, slot j holds the ((K - j) mod 16)-th newest, consecutive times differ only in the
// tap row (d0 grows by M: M / 2 rows on).  Warp-uniform control flow throughout.
template <int K>
__device__ __forceinline__ void branch_run(float2 (&win)[WS], bool adv, float2 nx0, const float4* __restrict__ tab, float2* __restrict__ out,
                                           int& d0, int& tt, int tt_hi, int lim) {
    if (adv) win[K] = nx0;
    const float4* row = tab + ((d0 + EARLY) >> 1);
    out += tt * FSK;
#pragma unroll 1
    for (;;) {
        const float4 t0 = row[0], t1 = row[ROWS], t2 = row[2 * ROWS], t3 = row[3 * ROWS];
        const float tap[WS] = {t0.x, t0.y, t0.z, t0.w, t1.x, t1.y, t1.z, t1.w, t2.x, t2.y, t2.z, t2.w, t3.x, t3.y, t3.z, t3.w};
        float2 a0 = make_float2(0.f, 0.f), a1 = a0, a2 = a0, a3 = a0;
#pragma unroll
        for (int j = 0; j < WS; j += 4) {
            a0 = cfma(tap[(K - j) & 15], win[j], a0);
            a1 = cfma(tap[(K - j - 1) & 15], win[j + 1], a1);
            a2 = cfma(tap[(K - j - 2) & 15], win[j + 2], a2);
            a3 = cfma(tap[(K - j - 3) & 15], win[j + 3], a3);
        }
        *out = cadd(cadd(a0, a1), cadd(a2, a3));
        tt++;
        if (tt >= tt_hi || d0 >= lim) break;                       // batch done, or the next output time advances the window
        d0 += M;
        row += M / 2;
        out += FSK;
    }
}
#define P25_PFB_CASE(k) \
    case k: branch_run<k>(win, adv, nx0, &sm.tab[0][0], &sm.f0[0][tid], d0, tt, tt_hi, lim); break;

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NTH, 1) p25_pfbc_kernel(const PfbParams p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    SmemC& sm = *reinterpret_cast<SmemC*>(smem_raw);
    cooperative_groups::cluster_group cluster = cooperative_groups::this_cluster();
    const int tid = threadIdx.x, lane = tid & 31;
    const int b = (int)cluster.block_rank();                      // parity of the FFT inputs / classes this CTA owns
    const unsigned run = blockIdx.x >> 1;
    const unsigned cap = run / p.runs_per_cap;
    const int t_first = (int)((run % p.runs_per_cap) * p.times_per_run);          // relative to m0, a multiple of TB
    const int t_last = min(t_first + (int)p.times_per_run, (int)p.n_out);
    if (cap >= p.n_captures || t_first >= t_last) return;         // both CTAs of the cluster take the same way out
    const float2* chunk = p.iq + (size_t)cap * p.n;
    const float2* tail = p.tail_in + (size_t)cap * HTX;
    const int n_in = (int)p.n;
    const unsigned inc_remote = map_to_rank(smem_u32(&sm.inc[0][0][0]), (unsigned)(b ^ 1));
    const unsigned mbar_remote = map_to_rank(smem_u32(&sm.mbar[0]), (unsigned)(b ^ 1));
    constexpr unsigned INC_BYTES = TB * (H / 2) * sizeof(float2);             // one batch of the partner's half
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(smem_u32(&sm.mbar[0])));
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(smem_u32(&sm.mbar[1])));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }

    for (int i = tid; i < 4 * ROWS; i += NTH) {
        const int g = i / ROWS, row = i - g * ROWS;
        const int d0r = 2 * row - EARLY + (1 - b);
        float t[4];
#pragma unroll
        for (int kk = 0; kk < 4; kk++) {
            const int idx = d0r + N * (4 * g + kk);
            t[kk] = (idx >= 0 && idx < LE) ? __ldg(p.taps + idx) : 0.f;
        }
        sm.tab[g][row] = make_float4(t[0], t[1], t[2], t[3]);
    }
    if (tid < 64) sm.twB[tid >> 3][tid & 7] = twiddle4(p.twiddle[24 * (tid >> 3) * (tid & 7)]);
    for (int i = tid; i < 12 * 64; i += NTH) sm.twC[i >> 6][i & 63] = p.twiddle[2 * (i >> 6) * (i & 63)];
#pragma unroll
    for (int i = 0; i < P25_BOXCAR - 1; i++) sm.hist[i][tid] = 0.f;
    // this thread's channel: k' = 384 b + kq (the 384 radix-2 pairs this CTA combines), channel k' or k' + 768
    const int kq = tid < H / 2 ? tid : tid - H / 2;
    const bool upper = tid >= H / 2;                               // warp-uniform: 384 = 12 warps
    const int chan = H / 2 * b + kq + (upper ? H : 0);

    // ---- window state of the thread's class, describing output time t_first - WARM - 1
    // logical index (tail ++ chunk, tail = HTX samples) of n_m for t = 0; every index below fits 32 bits (n <= 2^30)
    const int e_base = (int)((long long)M * (long long)p.m0 + (M - 1) - (long long)p.a0) + HTX;
    float2 win[WS], nx[3];
    int d0, phi = 0;
    {
        const int e_init = e_base + M * (t_first - WARM - 1);
        const int a0m = (int)(p.a0 % (unsigned long long)N);
        const int c = (N - (2 * tid + b)) % N;                    // residue class of the samples behind FFT input q = 2 tid + b
        const int cl = (c + HTX % N + N - a0m) % N;               // ... as a residue of the logical index
        const int rp = (e_init - cl) % N;                         // distance back to the class's latest sample (e_init >= N)
        const int rp0 = __shfl_sync(0xffffffffu, rp, 0);
        // lane i sits 2 i inputs below lane 0; if the warp's last lane would already be a whole N behind, the warp
        // starts one sample ahead (its first lanes then hold an early sample)
        d0 = rp0 + 2 * lane - (rp0 + 62 >= N ? N : 0);
        const int lnew = e_init - d0;
#pragma unroll
        for (int kk = 0; kk < WS; kk++) win[(WS - kk) & 15] = load_logical(tail, chunk, n_in, lnew - N * kk);
#pragma unroll
        for (int i = 0; i < 3; i++) nx[i] = load_logical(tail, chunk, n_in, lnew + N * (i + 1));   // arrivals of the first batch
    }
    float2 cprev = make_float2(0.f, 0.f);
    float pw = 0.f;
    const int t_begin = t_first - WARM;                            // first output time that is computed
    cluster.sync();                                                // both CTAs' barriers are initialised before either one sends

    // Polyphase branch sums of the (up to eight) output times of the batch that starts at tb_, then the prefetch of the
    // (at most three) samples the class receives during the batch after it.
    const auto polyphase = [&](int tb_) {
        const int tt_lo = max(t_begin - tb_, 0), tt_hi = min(t_last - tb_, TB);      // active output times of that batch
        const int lim = N - M - 2 * (31 - lane);                   // the warp's last lane reaches d0 >= N at the next output time
        int tt = tt_lo;
#pragma unroll 1
        while (tt < tt_hi) {
            const bool adv = d0 >= lim;                            // warp-uniform
            d0 += adv ? M - N : M;
            const float2 nx0 = nx[0];
            if (adv) {
                phi = (phi + 1) & 15;
                nx[0] = nx[1];
                nx[1] = nx[2];
            }
            switch (phi) {
                P25_PFB_CASE(0) P25_PFB_CASE(1) P25_PFB_CASE(2) P25_PFB_CASE(3) P25_PFB_CASE(4) P25_PFB_CASE(5)
                P25_PFB_CASE(6) P25_PFB_CASE(7) P25_PFB_CASE(8) P25_PFB_CASE(9) P25_PFB_CASE(10) P25_PFB_CASE(11)
                P25_PFB_CASE(12) P25_PFB_CASE(13) P25_PFB_CASE(14)
                default: branch_run<15>(win, adv, nx0, &sm.tab[0][0], &sm.f0[0][tid], d0, tt, tt_hi, lim); break;
            }
        }
        if (tb_ + TB < t_last) {
            const int l1 = e_base + M * (tb_ + TB - 1) - d0 + N;   // the window describes output time tb_ + TB - 1
            if (__all_sync(0xffffffffu, l1 >= HTX && l1 + 2 * N < HTX + n_in)) {      // the usual case: all inside the chunk
                const float2* src = chunk + (l1 - HTX);
                nx[0] = __ldg(src);
                nx[1] = __ldg(src + N);
                nx[2] = __ldg(src + 2 * N);
            } else {
#pragma unroll
                for (int i = 0; i < 3; i++) nx[i] = load_logical(tail, chunk, n_in, l1 + N * i);
            }
        }
    };
    // Software pipeline over the batches: the branch sums of batch n + 1 are computed between the last FFT pass of batch n
    // (which sends half of its result to the partner) and the combine step of batch n (which needs the partner's half),
    // so the exchange is never waited for (it was 11 % of all warp stalls when the wait followed the send directly).
    polyphase(t_first - 2 * TB);
    unsigned nb = 0;                                               // batch counter: incoming buffer nb & 1, phase (nb >> 1) & 1
    for (int tb = t_first - 2 * TB; tb < t_last; tb += TB, nb++) {
        if (tid == 0) mbar_expect_tx(smem_u32(&sm.mbar[nb & 1]), INC_BYTES);
        const int tt_lo = max(t_begin - tb, 0), tt_hi = min(t_last - tb, TB);        // active output times of this batch
        __syncthreads();                                           // f0 holds this batch's branch sums
        // ---- pass A: radix 8, stride 1, no twiddles; in place (read, barrier, write skewed); one butterfly per thread
        {
            const int tt = tid / 96, j = tid - 96 * tt;
            float2 v[8];
#pragma unroll
            for (int r = 0; r < 8; r++) v[r] = sm.f0[tt][j + 96 * r];
            __syncthreads();
            dft8(v);
#pragma unroll
            for (int q = 0; q < 8; q++) sm.f0[tt][skew_a(8 * j + q)] = v[q];
        }
        __syncthreads();
        // ---- pass B: radix 8, stride 8
        {
            const int tt = tid / 96, j = tid - 96 * tt, k = j & 7;
            float2 v[8];
#pragma unroll
            for (int r = 0; r < 8; r++) v[r] = sm.f0[tt][skew_a(j + 96 * r)];
            __syncthreads();
#pragma unroll
            for (int r = 1; r < 8; r++) v[r] = cmulw(v[r], sm.twB[r][k]);
            dft8(v);
            const int j0 = (j >> 3) * 64 + k;
#pragma unroll
            for (int q = 0; q < 8; q++) sm.f0[tt][skew_b(j0 + 8 * q)] = v[q];
        }
        __syncthreads();
        // ---- pass C: radix 12, stride 64 (512 butterflies).  Outputs k' = j + 64 q: q < 6 lies in CTA 0's combine range,
        // q >= 6 in CTA 1's; the half this CTA combines itself stays here, the other goes straight into the partner's
        // incoming buffer.  The partner cannot still be reading that buffer: it holds the batch before last, and the
        // partner's data of the last batch -- sent after it had finished with that one -- has already been consumed here.
        if (tid < TB * 64) {
            const int tt = tid >> 6, j = tid & 63;
            float2 v[12];
            v[0] = sm.f0[tt][skew_b(j)];
#pragma unroll
            for (int r = 1; r < 12; r++) {
                const float2 w = sm.twC[r][j];                     // 8-byte entries: i w is formed in registers
                v[r] = cmulw(sm.f0[tt][skew_b(j + 64 * r)], make_float4(w.x, w.y, -w.y, w.x));
            }
            dft12(v);
            const unsigned rbase = inc_remote + (unsigned)((((nb & 1) * TB + tt) * (H / 2) + j) * sizeof(float2));
            const unsigned rmbar = mbar_remote + (unsigned)((nb & 1) * sizeof(unsigned long long));
#pragma unroll
            for (int q = 0; q < 6; q++) {
                const float2 mine = b == 0 ? v[q] : v[q + 6], theirs = b == 0 ? v[q + 6] : v[q];
                sm.own[tt][j + 64 * q] = mine;
                st_async_f2(rbase + (unsigned)(64 * q * sizeof(float2)), theirs, rmbar);
            }
        }
        __syncthreads();                                           // own[] complete, f0 free
        if (tb + TB < t_last) polyphase(tb + TB);
        mbar_wait(smem_u32(&sm.mbar[nb & 1]), (nb >> 1) & 1);      // all of the partner's half has landed (long ago)
        // ---- radix-2 combine across the pair, discriminator, boxcar, baseband row: one channel per thread
        {
            const float4 wk = twiddle4(__ldg(p.twiddle + H / 2 * b + kq));
            const bool full = tt_lo == 0 && tt_hi == TB && tb >= t_first;      // the common case: no per-time tests
            float dn[TB];
            if (full && !p.y) {
                float2 cur[TB];
#pragma unroll
                for (int tt = 0; tt < TB; tt++) {
                    const float2 mine = sm.own[tt][kq], theirs = sm.inc[nb & 1][tt][kq];
                    const float2 e = b == 0 ? mine : theirs, wo = cmulw(b == 0 ? theirs : mine, wk);
                    cur[tt] = upper ? csub(e, wo) : cadd(e, wo);
                    pw += cur[tt].x * cur[tt].x + cur[tt].y * cur[tt].y;
                }
#pragma unroll
                for (int tt = 0; tt < TB; tt += 2) {               // two output times per discriminator evaluation
                    const float2 p0 = tt ? cur[tt - 1] : cprev, c0 = cur[tt], c1 = cur[tt + 1];
                    const float2 re = make_float2(c0.x * p0.x + c0.y * p0.y, c1.x * c0.x + c1.y * c0.y);
                    const float2 im = make_float2(c0.y * p0.x - c0.x * p0.y, c1.y * c0.x - c1.x * c0.y);
                    const float2 th = atan2x2(im, re);
                    dn[tt] = th.x * P25_FM_GAIN;
                    dn[tt + 1] = th.y * P25_FM_GAIN;
                }
                cprev = cur[TB - 1];
            } else {
#pragma unroll
                for (int tt = 0; tt < TB; tt++) {
                    float d_t = 0.f;
                    if (tt >= tt_lo && tt < tt_hi) {
                        const float2 mine = sm.own[tt][kq], theirs = sm.inc[nb & 1][tt][kq];
                        const float2 e = b == 0 ? mine : theirs, wo = cmulw(b == 0 ? theirs : mine, wk);
                        const float2 cur = upper ? csub(e, wo) : cadd(e, wo);
                        const float re = cur.x * cprev.x + cur.y * cprev.y;
                        const float im = cur.y * cprev.x - cur.x * cprev.y;
                        d_t = atan2_branchfree(im, re) * P25_FM_GAIN;
                        cprev = cur;
                        if (tb + tt >= t_first) {
                            pw += cur.x * cur.x + cur.y * cur.y;
                            if (p.y) p.y[((size_t)cap * p.y_rows + tb + tt) * N + chan] = cur;
                        }
                    }
                    dn[tt] = d_t;
                }
            }
            // ten-term boxcar over (nine carried values ++ eight new), a tree of pair sums
            float d[17];
#pragma unroll
            for (int i = 0; i < 9; i++) d[i] = sm.hist[i][tid];
#pragma unroll
            for (int i = 0; i < TB; i++) d[9 + i] = dn[i];
#pragma unroll
            for (int i = 0; i < 9; i++) sm.hist[i][tid] = d[8 + i];
            float s2[16], s4[14], box[TB];
#pragma unroll
            for (int i = 0; i < 16; i++) s2[i] = d[i] + d[i + 1];
#pragma unroll
            for (int i = 0; i < 14; i++) s4[i] = s2[i] + s2[i + 2];
#pragma unroll
            for (int i = 0; i < TB; i++) box[i] = ((s4[i] + s4[i + 4]) + s2[i + 8]) * (1.0f / P25_BOXCAR);
            float* out = p.bb + ((size_t)cap * N + chan) * p.row_stride + P25CU_BB_HIST + tb;
            if (full) {
                *reinterpret_cast<float4*>(out) = make_float4(box[0], box[1], box[2], box[3]);
                *reinterpret_cast<float4*>(out + 4) = make_float4(box[4], box[5], box[6], box[7]);
            } else {
#pragma unroll
                for (int i = 0; i < TB; i++)
                    if (tb + i >= t_first && tb + i < t_last) out[i] = box[i];
            }
        }
    }
    cluster.sync();                                                // neither CTA leaves while the other may still send to it
    if (p.power_sum) atomicAdd(p.power_sum + (size_t)cap * N + chan, pw);
}
#undef P25_PFB_CASE

// carried input tail: tail_out[i] = logical[n + i], logical = tail_in ++ chunk (both cf32), i < HTX
__global__ void p25_pfb_tail_kernel(const float2* iq, const float2* tail_in, float2* tail_out, unsigned n) {
    const unsigned cap = blockIdx.y;
    const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (unsigned)HTX) return;
    const unsigned long long l = (unsigned long long)n + i;
    tail_out[(size_t)cap * HTX + i] = l < (unsigned long long)HTX ? tail_in[(size_t)cap * HTX + l] : iq[(size_t)cap * n + (l - HTX)];
}

}  // namespace pfb

// ------------------------------------------------------------------------------------------------ host side
unsigned p25cu_pfb_tail_len() { return (unsigned)pfb::HTX; }
unsigned p25cu_pfb_channels() { return (unsigned)pfb::N; }
unsigned p25cu_pfb_decimation() { return (unsigned)pfb::M; }

// Equivalent prototype heq = hp (*) upsample(hc, M), in double, rounded once to f32; twiddle table.
cudaError_t p25cu_pfb_upload(float** d_taps, float2** d_twiddle) {
    cudaError_t e;
    double* acc = new double[pfb::LE]();
    for (int j = 0; j < P25_TAPS_CHAN; j++)
        for (int i = 0; i < pfb::L; i++) acc[i + pfb::M * j] += (double)P25_TAPS_CHAN_H[j] * (double)P25_TAPS_PFB_H[i];
    float* heq = new float[pfb::LE];
    for (int i = 0; i < pfb::LE; i++) heq[i] = (float)acc[i];
    delete[] acc;
    if ((e = cudaMalloc(d_taps, sizeof(float) * pfb::LE)) == cudaSuccess)
        e = cudaMemcpy(*d_taps, heq, sizeof(float) * pfb::LE, cudaMemcpyHostToDevice);
    delete[] heq;
    if (e != cudaSuccess) return e;
    float2* tw = new float2[pfb::N];
    for (int t = 0; t < pfb::N; t++) {
        const double a = 2.0 * 3.14159265358979323846 * (double)t / (double)pfb::N;
        tw[t] = make_float2((float)cos(a), (float)sin(a));
    }
    if ((e = cudaMalloc(d_twiddle, sizeof(float2) * pfb::N)) == cudaSuccess)
        e = cudaMemcpy(*d_twiddle, tw, sizeof(float2) * pfb::N, cudaMemcpyHostToDevice);
    delete[] tw;
    return e;
}

// Per-device setup (once per device under the library's plan mutex, that device current).
cudaError_t p25cu_pfb_plan_device(P25DevPlan* plan) {
    cudaError_t e = cudaFuncSetAttribute(pfb::p25_pfbc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(pfb::SmemC));
    if (e != cudaSuccess) return e;
    // clusters of two 200 KB CTAs that can be resident at once (at most one per SM pair of a GPC)
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(2 * plan->n_sm);
    cfg.blockDim = dim3(pfb::NTH);
    cfg.dynamicSmemBytes = sizeof(pfb::SmemC);
    int n_clusters = 0;
    e = cudaOccupancyMaxActiveClusters(&n_clusters, pfb::p25_pfbc_kernel, &cfg);
    if (e != cudaSuccess || n_clusters < 1) {
        (void)cudaGetLastError();
        n_clusters = plan->n_sm / 2;
    }
    plan->pfb_slots = n_clusters;
    return cudaSuccess;
}

// One chunk of every capture: baseband rows into bb, new tail.
cudaError_t p25cu_launch_pfb(const void* iq, const void* tail_in, void* tail_out, const float* taps, const float2* twiddle,
                             float2* y, unsigned y_rows, float* bb, size_t row_stride, float* power_sum,
                             unsigned long long a0, unsigned long long m0, unsigned n, unsigned n_out, unsigned n_captures,
                             cudaStream_t st, unsigned* launches, const P25DevPlan* plan) {
    if (n_out) {
        pfb::PfbParams a;
        a.iq = (const float2*)iq;
        a.tail_in = (const float2*)tail_in;
        a.taps = taps;
        a.twiddle = twiddle;
        a.bb = bb;
        a.row_stride = row_stride;
        a.y = y;
        a.power_sum = power_sum;
        a.a0 = a0;
        a.m0 = m0;
        a.n = n;
        a.n_out = n_out;
        a.n_captures = n_captures;
        a.y_rows = y_rows;
        // one wave: every resident cluster gets one run of consecutive output times (each run pays the table load and
        // ten warm-up output times), the captures share the clusters evenly; runs are whole batches of eight
        unsigned per_cap = (unsigned)plan->pfb_slots / n_captures;
        if (per_cap < 1) per_cap = 1;
        unsigned tpr = (n_out + per_cap - 1) / per_cap;
        tpr = (tpr + pfb::TB - 1) / pfb::TB * pfb::TB;
        if (tpr < 4 * pfb::TB) tpr = 4 * pfb::TB;                          // keep the warm-up share below a third
        a.times_per_run = tpr;
        a.runs_per_cap = (n_out + tpr - 1) / tpr;
        pfb::p25_pfbc_kernel<<<2 * a.runs_per_cap * n_captures, pfb::NTH, sizeof(pfb::SmemC), st>>>(a);
        *launches += 1;
    }
    if (n) {
        const dim3 gt((pfb::HTX + 255) / 256, n_captures);
        pfb::p25_pfb_tail_kernel<<<gt, 256, 0, st>>>((const float2*)iq, (const float2*)tail_in, (float2*)tail_out, n);
        *launches += 1;
    }
    return cudaGetLastError();
}
