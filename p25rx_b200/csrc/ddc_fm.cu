// ddc_fm.cu -- K1: IQ -> 48 kHz C4FM baseband for many streams in one launch.
//
// Replaces one iteration of DemodTask::run for every stream (reference src/demod.rs:70-117):
//   u8 IQ -> Complex32 table        src/demod.rs:82-84   (rtlsdr_iq::IQ)
//   /5 decimating FIR               src/demod.rs:87      (static_decimate::Decimator<DecimFir>)
//   channel-select FIR              src/demod.rs:93      (static_fir::FirFilter<BandpassFir>)
//   power accumulation              src/demod.rs:95-101, :123-134
//   FM discriminator                src/demod.rs:109-111 (demod_fm::FmDemod::new(5000, 48000))
//   10-tap moving average           src/demod.rs:114     (moving_avg::MovingAverage::new(10))
// plus a /10 front stage for 2.4 MS/s input (BASELINE.json configs[0]; declared extension).
//
// The whole chain is non-recursive, so every output is a pure function of a window of the logical
// input (tail of the previous chunk ++ this chunk); the only carried state is that raw input tail,
// kept in the stream's own sample format.  Five kernels share the arithmetic; one of the last four takes every
// chunk with outputs and 16-byte aligned rows, of any length, once a whole tail of the stream lies behind it (cf32 /50:
// from the stream start on, given an even decimator phase), and the generic kernel takes the rest:
//
//   p25_ddc_fm_kernel<FRONT,FMT>      generic: any length and alignment, the first chunk of a stream
//                                     (implicit zeros in front of it), odd chunks.  A CTA owns one
//                                     (stream, segment), stages blocks with coalesced loads (u8 through
//                                     a shared-memory copy of the table), runs the decimating stages
//                                     input-stationary and the 48 kHz stages on power-of-two rings.
//   fast::p25_ddc_fm_stream_kernel    cf32 /50 (the bench kernel): TMA bulk copies into a two-stage ring,
//                                     FFMA2 FIRs, persistent grid with a static + ticket work split.
//   w5::p25_ddc5_warp_kernel          cf32 /5: warp-autonomous, every warp is its own pipeline, no CTA
//                                     barriers.
//   w5i::p25_ddc5_imma_kernel         u8 /5: the warp kernel with the /5 decimator as exact integer
//                                     products on the tensor pipe (mma.sync u8 x s8 on the raw IQ bytes).
//   w50i::p25_ddc50_imma_kernel       u8 /50: both decimating stages as one 290-tap integer FIR.
//
// Algorithmic traffic: 8 + 4/D bytes per cf32 input sample, 2 + 4/D per u8 sample (DESIGN.md sec. 4); the cf32 /50
// kernel is HBM-bound (97 %), u8 /50 runs at 78 % of HBM, the /5 kernels are bound by issue slots and the FP32 pipe
// (62 complex-by-real taps per output; u8: 41 once the decimator is on the tensor pipe).
#include "p25cu_internal.cuh"
#include "p25_imma_tables.h"

__constant__ float c_taps_front[P25_TAPS_FRONT];
__constant__ float c_taps_decim[P25_TAPS_DECIM];
__constant__ float c_taps_chan[P25_TAPS_CHAN];
__constant__ float c_iq_lut[256];

static_assert(P25_TAPS_FRONT == 5 * P25_DECIM_FRONT, "front stage is a 10-phase x 5-tap polyphase matrix");
static_assert(P25_TAPS_DECIM == 5 * P25_DECIM_NATIVE, "decimator is a 5-phase x 5-tap polyphase matrix");

// Device primitives of the TMA-staged kernels (fast, w5, w5i, w50i): mbarriers, 1-D bulk copies, packed FP32, and the
// packed atan2 of the warp kernels' discriminator.
namespace prim {

__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
    unsigned ok;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
    } while (!ok);
}
__device__ __forceinline__ void tma_load_1d(void* dst, const void* src, unsigned bytes, unsigned long long* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
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
__device__ __forceinline__ float2 add2(float2 a, float2 b) {
    unsigned long long r;
    asm("add.rn.f32x2 %0, %1, %2;"
        : "=l"(r)
        : "l"(*reinterpret_cast<const unsigned long long*>(&a)), "l"(*reinterpret_cast<const unsigned long long*>(&b)));
    return *reinterpret_cast<float2*>(&r);
}

__device__ __forceinline__ float2 mul2(float2 a, float2 b) {
    unsigned long long r;
    asm("mul.rn.f32x2 %0, %1, %2;"
        : "=l"(r)
        : "l"(*reinterpret_cast<const unsigned long long*>(&a)), "l"(*reinterpret_cast<const unsigned long long*>(&b)));
    return *reinterpret_cast<float2*>(&r);
}
__device__ __forceinline__ float2 fma2s(float2 a, float2 b, float c) {   // a * b + (c, c)
    unsigned long long r;
    const float2 cc = make_float2(c, c);
    asm("fma.rn.f32x2 %0, %1, %2, %3;"
        : "=l"(r)
        : "l"(*reinterpret_cast<const unsigned long long*>(&a)), "l"(*reinterpret_cast<const unsigned long long*>(&b)),
          "l"(*reinterpret_cast<const unsigned long long*>(&cc)));
    return *reinterpret_cast<float2*>(&r);
}
// atan2 for the discriminator, two outputs at once: |error| <= 2e-7 rad (degree-7 minimax in t^2 on [0, 1], spec/gen_tables.py
// style fit; CUDA's atan2f costs ~85 instructions with its special-case branches, this one ~22, branch-free).
// atan2(0, 0) = 0 like std::atan2 on +0 arguments.  The polynomial and the three multiplies run packed (same arithmetic
// per half).
__device__ __forceinline__ float2 disc_atan2_pair(float2 y, float2 x) {
    const float ax0 = fabsf(x.x), ay0 = fabsf(y.x), ax1 = fabsf(x.y), ay1 = fabsf(y.y);
    const float mx0 = fmaxf(ax0, ay0), mn0 = fminf(ax0, ay0), mx1 = fmaxf(ax1, ay1), mn1 = fminf(ax1, ay1);
    float rc0, rc1;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rc0) : "f"(fmaxf(mx0, 1e-30f)));
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rc1) : "f"(fmaxf(mx1, 1e-30f)));
    const float2 t = mul2(make_float2(mn0, mn1), make_float2(rc0, rc1)), u = mul2(t, t);
    float2 q = make_float2(-0.004295386839658022f, -0.004295386839658022f);
    q = fma2s(q, u, 0.022737378254532814f);
    q = fma2s(q, u, -0.057179518043994904f);
    q = fma2s(q, u, 0.09735459089279175f);
    q = fma2s(q, u, -0.13945257663726807f);
    q = fma2s(q, u, 0.1995391547679901f);
    q = fma2s(q, u, -0.3333050608634949f);
    q = fma2s(q, u, 0.9999995231628418f);
    const float2 r = mul2(q, t);
    float r0 = r.x, r1 = r.y;
    r0 = ay0 > ax0 ? 1.57079632679489662f - r0 : r0;
    r1 = ay1 > ax1 ? 1.57079632679489662f - r1 : r1;
    r0 = x.x < 0.f ? 3.14159265358979324f - r0 : r0;
    r1 = x.y < 0.f ? 3.14159265358979324f - r1 : r1;
    return make_float2(copysignf(r0, y.x), copysignf(r1, y.y));
}

}  // namespace prim

template <bool FRONT>
struct Cfg {
    static constexpr int MB = FRONT ? 64 : 256;         // 48 kHz outputs per block
    static constexpr int NT = FRONT ? 320 : 256;        // threads
    static constexpr int DIN = FRONT ? 50 : 5;          // input samples per output
    static constexpr int XN = MB * DIN;                 // input samples per block
    static constexpr int ACOLS = FRONT ? 5 * MB : 0;    // front-stage outputs per block
    static constexpr int RING = FRONT ? 128 : 512;      // >= MB + 40
    static constexpr int HT = FRONT ? 3264 : 1312;      // input tail carried between chunks
};

template <bool FRONT>
struct Smem {
    using C = Cfg<FRONT>;
    float2 xs[C::XN];                        // staged input block
    float2 pa[2][4][FRONT ? C::ACOLS : 1];   // front-stage partial sums (ping-pong)
    float ya_re[FRONT ? C::ACOLS : 1], ya_im[FRONT ? C::ACOLS : 1];
    float2 pd[2][4][C::MB];                  // decimator partial sums (ping-pong)
    float yd_re[C::RING], yd_im[C::RING];    // decimator output ring
    float c_re[C::RING], c_im[C::RING];      // channel filter output ring
    float d[C::RING];                        // discriminator output ring
    float red[32];
    float lut[256];                          // u8 -> f32 table (a per-lane index into __constant__ memory would serialise)
};

// The carried input tail is kept in the stream's own sample format (u8 pairs or cf32).  Samples in front of
// the stream start (absolute index < 0) are zeros: for cf32 the zero-initialised tail says so by itself, for
// u8 (where no byte maps to 0.0) the rule is explicit: logical index l < ht - a0 is zero.
template <int FMT>
struct Elem { using T = float2; };
template <>
struct Elem<P25CU_FMT_U8_IQ> { using T = uchar2; };

template <int FMT>
__device__ __forceinline__ float2 cvt(const float* lut, typename Elem<FMT>::T v) {
    if constexpr (FMT == P25CU_FMT_CF32_IQ) return v;
    else return make_float2(lut[v.x], lut[v.y]);
}

// logical input sample l (0 .. HT+n): tail of the previous chunk, then this chunk; zeros beyond
template <int FMT>
__device__ __forceinline__ typename Elem<FMT>::T load_logical_raw(const DdcParams& p, const void* tail, const void* chunk, long long l) {
    using T = typename Elem<FMT>::T;
    if (l < (long long)p.ht) return ((const T*)tail)[l];
    const long long i = l - p.ht;
    if (i >= (long long)p.n) return T{};
    return __ldcs((const T*)chunk + i);
}

// Stage logical samples [l0, l0 + XN) into sm.xs.  Global loads are 16 bytes wide and aligned to the
// *source* (2 cf32 samples or 8 u8 samples per load); each sample is then stored to its own slot, so
// any decimator phase / chunk parity takes the vector path as long as the rows themselves are aligned.
template <bool FRONT, int FMT>
__device__ __forceinline__ void stage_block(Smem<FRONT>& sm, const DdcParams& p, const void* tail, const void* chunk,
                                            long long l0) {
    using C = Cfg<FRONT>;
    const long long ht = (long long)p.ht;
    const int tid = threadIdx.x;
    // part 1: samples that still come from the previous chunk's tail (HT is even)
    const long long t_end = l0 + C::XN < ht ? l0 + C::XN : ht;
    if (l0 < t_end) {
        if constexpr (FMT == P25CU_FMT_CF32_IQ) {
            for (long long l = (l0 & ~1LL) + 2 * tid; l < t_end; l += 2 * C::NT) {
                const float4 v = *(const float4*)((const float2*)tail + l);
                const long long i = l - l0;
                if (i >= 0) sm.xs[i] = make_float2(v.x, v.y);
                if (i + 1 < C::XN && l + 1 < t_end) sm.xs[i + 1] = make_float2(v.z, v.w);
            }
        } else {
            const long long zero_below = ht - (long long)p.a0;   // logical indices in front of the stream start
            for (long long l = l0 + tid; l < t_end; l += C::NT) {
                const uchar2 b = ((const uchar2*)tail)[l];
                sm.xs[l - l0] = l < zero_below ? make_float2(0.f, 0.f) : make_float2(sm.lut[b.x], sm.lut[b.y]);
            }
        }
    }
    // part 2: samples of this chunk (zeros past its end)
    const long long c_beg = (l0 > ht ? l0 : ht) - ht, c_end = l0 + C::XN - ht;
    if (c_end <= c_beg) return;
    const long long base = ht - l0;   // xs index = chunk index + base
    const long long n = (long long)p.n;
    if (p.aligned16) {
        if (FMT == P25CU_FMT_CF32_IQ) {
            for (long long g = (c_beg & ~1LL) + 2 * tid; g < c_end; g += 2 * C::NT) {
                const float4 v = g < n ? __ldcs((const float4*)((const float2*)chunk + g)) : make_float4(0.f, 0.f, 0.f, 0.f);
                if (g >= c_beg) sm.xs[g + base] = make_float2(v.x, v.y);
                if (g + 1 < c_end) sm.xs[g + 1 + base] = make_float2(v.z, v.w);
            }
        } else {
            for (long long g = (c_beg & ~7LL) + 8 * tid; g < c_end; g += 8 * C::NT) {
                const uint4 v = g < n ? __ldcs((const uint4*)((const uchar2*)chunk + g)) : make_uint4(0x7F7F7F7Fu, 0x7F7F7F7Fu, 0x7F7F7F7Fu, 0x7F7F7F7Fu);
                const unsigned w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                for (int e = 0; e < 8; e++) {
                    const long long jj = g + e;
                    if (jj >= c_beg && jj < c_end) {
                        const unsigned b = w[e >> 1] >> (16 * (e & 1));
                        sm.xs[jj + base] = jj < n ? make_float2(sm.lut[b & 0xFF], sm.lut[(b >> 8) & 0xFF]) : make_float2(0.f, 0.f);
                    }
                }
            }
        }
    } else {
        for (long long jj = c_beg + tid; jj < c_end; jj += C::NT) {
            float2 v = make_float2(0.f, 0.f);
            if (jj < n) v = cvt<FMT>(sm.lut, __ldcs((const typename Elem<FMT>::T*)chunk + jj));
            sm.xs[jj + base] = v;
        }
    }
}

// partial sums of one polyphase column: P_q = sum_p h[D*q + p] * x[D-1-p],  q = 0..4
template <int D>
__device__ __forceinline__ void column_partials(const float2 (&x)[D], const float* __restrict__ h, float2 (&P)[5]) {
#pragma unroll
    for (int q = 0; q < 5; q++) {
        float re = 0.f, im = 0.f;
#pragma unroll
        for (int pp = 0; pp < D; pp++) {
            const float t = h[D * q + pp];
            re = fmaf(t, x[D - 1 - pp].x, re);
            im = fmaf(t, x[D - 1 - pp].y, im);
        }
        P[q] = make_float2(re, im);
    }
}

template <bool FRONT, int FMT>
__global__ void __launch_bounds__(Cfg<FRONT>::NT) p25_ddc_fm_kernel(const DdcParams p) {
    using C = Cfg<FRONT>;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    Smem<FRONT>& sm = *reinterpret_cast<Smem<FRONT>*>(smem_raw);
    const int tid = threadIdx.x;
    const unsigned s = blockIdx.x / p.n_seg, g = blockIdx.x % p.n_seg;

    // zero rings and partial buffers (everything behind xs)
    {
        float* z = reinterpret_cast<float*>(&sm.pa[0][0][0]);
        const int nz = (int)((sizeof(Smem<FRONT>) - sizeof(sm.xs) - sizeof(sm.lut)) / sizeof(float));
        for (int i = tid; i < nz; i += C::NT) z[i] = 0.f;
        for (int i = tid; i < 256; i += C::NT) sm.lut[i] = c_iq_lut[i];
    }

    using ET = typename Elem<FMT>::T;
    const void* tail = (const ET*)p.tail_in + (size_t)s * p.ht;
    const void* chunk = (FMT == P25CU_FMT_CF32_IQ) ? (const void*)((const float2*)p.iq + (size_t)s * p.n)
                                                    : (const void*)((const uchar2*)p.iq + (size_t)s * p.n);
    float* out = p.bb + (size_t)s * p.row_stride + P25CU_BB_HIST;

    const long long M0 = (long long)p.m0;
    const long long mb = M0 + (long long)g * p.seg_out;
    long long me = mb + p.seg_out;
    if (me > M0 + (long long)p.n_out) me = M0 + p.n_out;
    const long long a0 = (long long)p.a0;
    float pw = 0.f;
    int pb = 0;
    __syncthreads();

    for (long long mi = mb - C::MB; mi < me; mi += C::MB, pb ^= 1) {
        // 1. stage the input block [DIN*mi, DIN*(mi+MB)) of the logical input
        stage_block<FRONT, FMT>(sm, p, tail, chunk, (long long)C::DIN * mi - a0 + (long long)p.ht);
        __syncthreads();

        if constexpr (FRONT) {
            // 2. front /10 stage, input-stationary: thread = one column of 10 inputs
            float2 P[5];
            {
                float2 x[10];
                const float4* src = reinterpret_cast<const float4*>(&sm.xs[10 * tid]);
#pragma unroll
                for (int i = 0; i < 5; i++) {
                    const float4 v = src[i];
                    x[2 * i] = make_float2(v.x, v.y);
                    x[2 * i + 1] = make_float2(v.z, v.w);
                }
                column_partials<10>(x, c_taps_front, P);
            }
#pragma unroll
            for (int q = 1; q < 5; q++) sm.pa[pb][q - 1][tid] = P[q];
            __syncthreads();
            // 3. combine with the partials of the 4 previous columns
            float re = P[0].x, im = P[0].y;
#pragma unroll
            for (int q = 1; q < 5; q++) {
                const int c = tid - q;
                const float2 v = c >= 0 ? sm.pa[pb][q - 1][c] : sm.pa[pb ^ 1][q - 1][C::ACOLS + c];
                re += v.x;
                im += v.y;
            }
            sm.ya_re[tid] = re;
            sm.ya_im[tid] = im;
            __syncthreads();
        }

        // 4. /5 decimator, input-stationary: thread = one column of 5 inputs (one 48 kHz output)
        float2 Q[5];
        if (tid < C::MB) {
            float2 x[5];
            if constexpr (FRONT) {
#pragma unroll
                for (int i = 0; i < 5; i++) x[i] = make_float2(sm.ya_re[5 * tid + i], sm.ya_im[5 * tid + i]);
            } else {
#pragma unroll
                for (int i = 0; i < 5; i++) x[i] = sm.xs[5 * tid + i];
            }
            column_partials<5>(x, c_taps_decim, Q);
#pragma unroll
            for (int q = 1; q < 5; q++) sm.pd[pb][q - 1][tid] = Q[q];
        }
        __syncthreads();
        if (tid < C::MB) {
            float re = Q[0].x, im = Q[0].y;
#pragma unroll
            for (int q = 1; q < 5; q++) {
                const int c = tid - q;
                const float2 v = c >= 0 ? sm.pd[pb][q - 1][c] : sm.pd[pb ^ 1][q - 1][C::MB + c];
                re += v.x;
                im += v.y;
            }
            const unsigned r = (unsigned)(mi + tid) & (C::RING - 1);
            sm.yd_re[r] = re;
            sm.yd_im[r] = im;
        }
        __syncthreads();

        // 5. channel-select FIR at 48 kHz: one (output, component) per work item
        for (int w = tid; w < 2 * C::MB; w += C::NT) {
            const int o = w < C::MB ? w : w - C::MB;
            const float* src = w < C::MB ? sm.yd_re : sm.yd_im;
            const unsigned r = (unsigned)(mi + o);
            float acc = 0.f;
#pragma unroll
            for (int k = 0; k < P25_TAPS_CHAN; k++) acc = fmaf(c_taps_chan[k], src[(r - k) & (C::RING - 1)], acc);
            (w < C::MB ? sm.c_re : sm.c_im)[r & (C::RING - 1)] = acc;
        }
        __syncthreads();

        // 6. FM discriminator (+ power of the channel-filtered samples)
        if (tid < C::MB) {
            const long long m = mi + tid;
            const unsigned r = (unsigned)m;
            const float cr = sm.c_re[r & (C::RING - 1)], ci = sm.c_im[r & (C::RING - 1)];
            const float pr = sm.c_re[(r - 1) & (C::RING - 1)], pi = sm.c_im[(r - 1) & (C::RING - 1)];
            const float re = cr * pr + ci * pi;
            const float im = ci * pr - cr * pi;
            sm.d[r & (C::RING - 1)] = atan2f(im, re) * P25_FM_GAIN;
            if (m >= mb && m < me) pw += cr * cr + ci * ci;
        }
        __syncthreads();

        // 7. symbol-period boxcar, store
        if (tid < C::MB) {
            const long long m = mi + tid;
            if (m >= mb && m < me) {
                const unsigned r = (unsigned)m;
                float acc = 0.f;
#pragma unroll
                for (int i = P25_BOXCAR - 1; i >= 0; i--) acc += sm.d[(r - i) & (C::RING - 1)];
                out[m - M0] = acc / (float)P25_BOXCAR;
            }
        }
        // the next block's first barrier orders these ring reads before they are overwritten
    }

    // power: block reduction, one atomic per CTA
    if (p.power_sum) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) pw += __shfl_xor_sync(0xFFFFFFFFu, pw, o);
        __syncthreads();
        if ((tid & 31) == 0) sm.red[tid >> 5] = pw;
        __syncthreads();
        if (tid == 0) {
            float t = 0.f;
            for (int i = 0; i < C::NT / 32; i++) t += sm.red[i];
            atomicAdd(p.power_sum + s, t);
        }
    }

    // the last segment of each stream writes the input tail for the next chunk
    if (g == p.n_seg - 1) {
        ET* tout = (ET*)p.tail_out + (size_t)s * p.ht;
        for (int i = tid; i < (int)p.ht; i += C::NT) tout[i] = load_logical_raw<FMT>(p, tail, chunk, (long long)p.n + i);
    }
}

// =====================================================================================================
// Fast path: cf32 input, /50, 16-byte aligned rows and even decimator phase (the bench workload and any
// caller that feeds even-length chunks).  Same arithmetic as the generic kernel above, restructured:
//   * staging by TMA 1-D bulk copies (cp.async.bulk + mbarrier complete_tx) into a two-stage ring, so the
//     copy of block i+1 is in flight while block i is computed and no thread instruction touches the bytes;
//   * persistent CTAs over a flattened (stream, block) space: every CTA gets the same number of blocks, so
//     there is no partial last wave; a CTA that enters a stream mid-way replays one warm-up block;
//   * FIR inner loops on packed FFMA2 (fma.rn.f32x2): one issue slot per complex-by-real tap, taps broadcast
//     from uniform registers; 48 kHz histories in linear buffers (no ring masking in the inner loops).
// =====================================================================================================
namespace fast {

using namespace prim;

constexpr int MB = 64;            // 48 kHz outputs per block
constexpr int NT = 320;           // threads = front-stage columns per block
constexpr int XN = MB * 50;       // input samples per block
constexpr int ACOLS = 5 * MB;
constexpr int HC = P25_TAPS_CHAN - 1;   // channel filter history (40)
constexpr int HB = P25_BOXCAR - 1;      // boxcar history (9)
#ifndef DDC50_MAXREG
#define DDC50_MAXREG 56
#endif

constexpr int ES = sizeof(float2);      // bytes per sample

struct __align__(128) Smem {
    unsigned char xs[2][XN * ES];  // TMA destinations (blocks start on a 16-byte boundary: even a0)
    float2 pa[4][ACOLS + 4];       // front partials q=1..4; slots 0..3 carry the previous block's last columns
    float2 ya[ACOLS];
    float2 pd[4][MB + 4];
    float2 yd[HC + MB];            // decimator outputs, linear with history
    float2 c[1 + MB];              // channel filter outputs
    float d[HB + MB];              // discriminator outputs
    float red[16];
    unsigned long long full[2];    // mbarriers
};

template <int D>
__device__ __forceinline__ void partials(const float2 (&x)[D], const float* __restrict__ h, float2 (&P)[5]) {
#pragma unroll
    for (int q = 0; q < 5; q++) {
        float2 a = make_float2(0.f, 0.f);
#pragma unroll
        for (int pp = 0; pp < D; pp++) a = cfma(h[D * q + pp], x[D - 1 - pp], a);
        P[q] = a;
    }
}

// issue the bulk copies of logical samples [l0, l0 + XN) (clipped to the data that exists) into xs[stage]
__device__ __forceinline__ void issue_block(Smem& sm, int stage, const DdcParams& p, const unsigned char* tail,
                                            const unsigned char* chunk, long long l0) {
    const long long ht = p.ht, lend = ht + (long long)p.n;
    const long long la = l0 & ~1LL;
    long long l1 = la + XN;
    if (l1 > lend) l1 = lend;
    const long long t1 = l1 < ht ? l1 : ht;       // end of the part served by the tail
    const unsigned nt = la < t1 ? (unsigned)(t1 - la) : 0u;
    const long long cb = la > ht ? la : ht;       // start of the part served by the chunk
    const unsigned nc = cb < l1 ? (unsigned)(l1 - cb) : 0u;
    mbar_expect_tx(&sm.full[stage], (nt + nc) * ES);
    if (nt) tma_load_1d(&sm.xs[stage][0], tail + la * ES, nt * ES, &sm.full[stage]);
    if (nc) tma_load_1d(&sm.xs[stage][(cb - la) * ES], chunk + (cb - ht) * ES, nc * ES, &sm.full[stage]);
}

// Work distribution: the flattened (stream, block) space is split into a static part (n_static consecutive blocks per
// CTA, no extra warm-ups) and a dynamic remainder handed out in DYN_CH-block tickets.  A CTA that becomes resident
// late -- the previous chunk's walker CTAs still hold registers and shared memory on its SM -- simply draws fewer
// tickets instead of stretching the whole launch (with a purely static split that tail cost ~9 % beside the walker).
#ifndef DDC50_DYN_CH
#define DDC50_DYN_CH 16
#endif
#ifndef DDC50_STATIC_NUM
#define DDC50_STATIC_NUM 7
#define DDC50_STATIC_DEN 8
#endif
constexpr unsigned DYN_CH = DDC50_DYN_CH;

// dc = 0 and pw_scale = 1 (the channel filter's start value and the power scale) are launch arguments, not literals:
// with literals ptxas schedules the kernel differently, and that schedule measured 1-2 % slower (NVIDIA B200, 1000 W).
__global__ void __maxnreg__(DDC50_MAXREG) p25_ddc_fm_stream_kernel(const DdcParams p, const unsigned blocks_per_stream,
                                                                  const unsigned n_static, const unsigned n_tickets,
                                                                  const unsigned ticket_base, const float dc, const float pw_scale) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    Smem& sm = *reinterpret_cast<Smem*>(smem_raw);
    __shared__ unsigned s_ticket;
    const int tid = threadIdx.x;

    if (tid == 0) {
        mbar_init(&sm.full[0], 1);
        mbar_init(&sm.full[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    const unsigned long long total = (unsigned long long)p.n_streams * blocks_per_stream;
    const unsigned long long dyn_begin = (unsigned long long)n_static * gridDim.x;
    unsigned long long b = (unsigned long long)n_static * blockIdx.x;      // static share first
    unsigned long long b_end = b + n_static;
    const long long M0 = (long long)p.m0, a0 = (long long)p.a0;
    unsigned use = 0;   // blocks consumed so far by this CTA: stage = use & 1, parity = (use >> 1) & 1
    __syncthreads();

  for (;;) {
    if (b >= b_end) {                                                       // draw the next ticket of the dynamic part
        if (tid == 0) s_ticket = atomicAdd(p.work_counter, 1u) - ticket_base;
        __syncthreads();
        const unsigned c = s_ticket;
        __syncthreads();
        if (c >= n_tickets) break;
        b = dyn_begin + (unsigned long long)c * DYN_CH;
        b_end = b + DYN_CH < total ? b + DYN_CH : total;
    }
    while (b < b_end) {
        const unsigned s = (unsigned)(b / blocks_per_stream);
        const unsigned it0 = (unsigned)(b % blocks_per_stream);
        unsigned it1 = blocks_per_stream;
        if (b_end - b < (unsigned long long)(it1 - it0)) it1 = it0 + (unsigned)(b_end - b);
        b += it1 - it0;
        const unsigned char* tail = (const unsigned char*)p.tail_in + (size_t)s * p.ht * ES;
        const unsigned char* chunk = (const unsigned char*)p.iq + (size_t)s * p.n * ES;
        const long long mb = M0 + (long long)it0 * MB;
        long long me = M0 + (long long)it1 * MB;
        if (me > M0 + (long long)p.n_out) me = M0 + p.n_out;
        float* out = p.bb + (size_t)s * p.row_stride + P25CU_BB_HIST - M0;   // out[m]
        const long long lbase = -a0 + (long long)p.ht;                       // logical index = 50 * m + lbase

        // zero the histories / carries (a fresh piece starts with a warm-up block)
        for (int i = tid; i < 4 * 4; i += NT) {
            sm.pa[i >> 2][i & 3] = make_float2(0.f, 0.f);
            sm.pd[i >> 2][i & 3] = make_float2(0.f, 0.f);
        }
        for (int i = tid; i < HC; i += NT) sm.yd[i] = make_float2(0.f, 0.f);
        if (tid == 0) sm.c[0] = make_float2(0.f, 0.f);
        if (tid < HB) sm.d[tid] = 0.f;
        float pw = 0.f;
        const long long m_first = mb - MB;
        const int nblk = (int)((me - m_first + MB - 1) / MB);
        if (tid == 0) {
            issue_block(sm, use & 1, p, tail, chunk, 50 * m_first + lbase);
            if (nblk > 1) issue_block(sm, (use + 1) & 1, p, tail, chunk, 50 * (m_first + MB) + lbase);
        }
        __syncthreads();

        for (int blk = 0; blk < nblk; blk++, use++) {
            const long long mi = m_first + (long long)blk * MB;
            const int stage = use & 1;
            mbar_wait(&sm.full[stage], (use >> 1) & 1);

            // front /10 stage: thread = column of 10 inputs
            float2 P[5];
            {
                float2 x[10];
                const float4* src = reinterpret_cast<const float4*>(sm.xs[stage]) + 5 * tid;
#pragma unroll
                for (int i = 0; i < 5; i++) {
                    const float4 v = src[i];
                    x[2 * i] = make_float2(v.x, v.y);
                    x[2 * i + 1] = make_float2(v.z, v.w);
                }
                partials<10>(x, c_taps_front, P);
            }
#pragma unroll
            for (int q = 1; q < 5; q++) sm.pa[q - 1][tid + 4] = P[q];
            __syncthreads();                                                  // B1: xs[stage] fully consumed
            if (tid == 0 && blk + 2 < nblk) issue_block(sm, stage, p, tail, chunk, 50 * (mi + 2 * MB) + lbase);
            {
                float2 a = P[0];
#pragma unroll
                for (int q = 1; q < 5; q++) {
                    const float2 v = sm.pa[q - 1][tid + 4 - q];
                    a.x += v.x;
                    a.y += v.y;
                }
                sm.ya[tid] = a;
            }
            __syncthreads();                                                  // B2
            if (tid >= ACOLS - 4) {
#pragma unroll
                for (int q = 1; q < 5; q++) sm.pa[q - 1][tid - (ACOLS - 4)] = P[q];   // carry for the next block
            }
            // /5 decimator, thread = column of 5 front outputs
            float2 Q[5];
            if (tid < MB) {
                float2 x[5];
#pragma unroll
                for (int i = 0; i < 5; i++) x[i] = sm.ya[5 * tid + i];
                partials<5>(x, c_taps_decim, Q);
#pragma unroll
                for (int q = 1; q < 5; q++) sm.pd[q - 1][tid + 4] = Q[q];
            }
            __syncthreads();                                                  // B3
            if (tid < MB) {
                float2 a = Q[0];
#pragma unroll
                for (int q = 1; q < 5; q++) {
                    const float2 v = sm.pd[q - 1][tid + 4 - q];
                    a.x += v.x;
                    a.y += v.y;
                }
                sm.yd[HC + tid] = a;
            }
            __syncthreads();                                                  // B4
            if (tid >= MB - 4 && tid < MB) {
#pragma unroll
                for (int q = 1; q < 5; q++) sm.pd[q - 1][tid - (MB - 4)] = Q[q];
            }
            // channel FIR at 48 kHz (two accumulators for ILP)
            if (tid < MB) {
                float2 e = make_float2(dc, dc), o = make_float2(0.f, 0.f);
                const float2* src = &sm.yd[HC + tid];
#pragma unroll
                for (int k = 0; k + 1 < P25_TAPS_CHAN; k += 2) {
                    e = cfma(c_taps_chan[k], src[-k], e);
                    o = cfma(c_taps_chan[k + 1], src[-k - 1], o);
                }
                e = cfma(c_taps_chan[P25_TAPS_CHAN - 1], src[-(P25_TAPS_CHAN - 1)], e);
                sm.c[1 + tid] = make_float2(e.x + o.x, e.y + o.y);
            }
            __syncthreads();                                                  // B5
            if (tid < MB) {                                                   // FM discriminator
                const float2 cur = sm.c[1 + tid], prv = sm.c[tid];
                const float re = cur.x * prv.x + cur.y * prv.y;
                const float im = cur.y * prv.x - cur.x * prv.y;
                sm.d[HB + tid] = atan2f(im, re) * P25_FM_GAIN;
                const long long m = mi + tid;
                if (m >= mb && m < me) pw += cur.x * cur.x + cur.y * cur.y;
            } else if (tid >= 128 && tid < 128 + HC) {                        // roll the decimator history
                sm.yd[tid - 128] = sm.yd[MB + tid - 128];
            }
            __syncthreads();                                                  // B6
            float bsum = 0.f;
            if (tid < MB) {                                                   // boxcar, store
#pragma unroll
                for (int i = 0; i < P25_BOXCAR; i++) bsum += sm.d[tid + i];
                const long long m = mi + tid;
                if (m >= mb && m < me) out[m] = bsum / (float)P25_BOXCAR;
            } else if (tid == 128) {
                sm.c[0] = sm.c[MB];
            }
            __syncthreads();                                                  // B7: boxcar reads done
            if (tid < HB) sm.d[tid] = sm.d[MB + tid];
        }

        if (p.power_sum) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) pw += __shfl_xor_sync(0xFFFFFFFFu, pw, o);
            if ((tid & 31) == 0) sm.red[tid >> 5] = pw;
            __syncthreads();
            if (tid == 0) {
                float t = 0.f;
                for (int i = 0; i < NT / 32; i++) t += sm.red[i];
                atomicAdd(p.power_sum + s, t * pw_scale);
            }
        }
        if (it1 == blocks_per_stream) {   // this piece ends the stream's chunk: write the tail for the next chunk
            float2* tout = (float2*)p.tail_out + (size_t)s * p.ht;
            for (int i = tid; i < (int)p.ht; i += NT)
                tout[i] = load_logical_raw<P25CU_FMT_CF32_IQ>(p, tail, chunk, (long long)p.n + i);
        }
        __syncthreads();
    }
  }
}

}  // namespace fast


// =====================================================================================================
// Warp-autonomous kernels (w5, w5i, w50i).  The FP32 pipe and the issue slots, not HBM, are the limit of the /5 shapes,
// and CTA barriers between stages that keep only part of a CTA busy would stall both, so every warp is its own pipeline
// and the only synchronisation is __syncwarp:
//   * a warp walks a contiguous share of the flattened (stream, iteration) space, NOUT outputs per iteration, entering
//     each stream or share with one discarded warm-up iteration, so the carried FIR histories live in per-warp shared
//     memory;
//   * lane 0 streams the raw input slices with TMA bulk copies into a per-warp ring of one or two stages;
//   * the kernel's own decimator writes R outputs per lane as rows of the channel filter's window arrays;
//   * the 48 kHz stages are common: the channel filter's R outputs stay in registers for the discriminator (the
//     previous sample arrives by shuffle), only the discriminator rows go back to shared memory for the boxcar; stores
//     are 16 bytes per lane.
// A kernel supplies its slice geometry, its decimator and its shared-memory layout; this namespace does the rest.
// =====================================================================================================
namespace wk {

using namespace prim;

// bulk copy of the slice whose first input has logical index l0 (tail ++ chunk) into xs, completing on bar; 32-bit index
// arithmetic, the slice that still overlaps the carried tail (first iterations of a chunk only) takes the two-copy path.
// CLAMP: the part in front of the tail (l0 < 0: warm-up of a chunk's first piece) is skipped, the destination keeps its
// offset.
template <int ES, int AL, int XLEN, bool CLAMP>
__device__ __forceinline__ void issue_slice(unsigned char* xs, unsigned long long* bar, int ht, int lend,
                                            const unsigned char* tail, const unsigned char* chunk, int l0) {
    const int la0 = l0 & ~(AL - 1);
    const int la = CLAMP ? max(la0, 0) : la0;
    const int lb = min(la0 + XLEN, lend);
    unsigned char* const dst = xs + (la - la0) * ES;
    if (la >= ht) {
        const unsigned bytes = (unsigned)(lb - la) * ES;
        mbar_expect_tx(bar, bytes);
        tma_load_1d(dst, chunk + (size_t)(la - ht) * ES, bytes, bar);
        return;
    }
    const int t1 = min(lb, ht);
    const unsigned nt = (unsigned)(t1 - la), nc = (unsigned)(lb - t1);
    mbar_expect_tx(bar, (nt + nc) * ES);
    tma_load_1d(dst, tail + (size_t)la * ES, nt * ES, bar);
    if (nc) tma_load_1d(dst + nt * ES, chunk, nc * ES, bar);
}

// Walks this warp's share [b0, b1) of the flattened (stream, iteration) space piece by piece: a piece is a run of stored
// iterations of one stream preceded by one warm-up iteration (iteration it_first - 1; -1 = the inputs just before the
// chunk, served by the carried tail) that only rebuilds the filter histories.  Lane 0 keeps NSTAGE slices in flight
// through issue(stage, tail, chunk, l0), NSTAGE iterations ahead (possibly into the next piece); the slice of iteration
// it lands in stage `use % NSTAGE` behind full[stage].  Per iteration dec(stage, it) consumes the slice and writes the
// decimator rows, and back(nv, out, pw) runs the 48 kHz stages and stores nv outputs (none in the warm-up) from out.
// At the end of a piece: power flush, raw-tail carry when the stream's chunk is complete, next stream.
template <int NSTAGE, int WARPS, int R, int NOUT, int XNEW, int ES, typename Issue, typename Dec, typename Back>
__device__ __forceinline__ void walk(const DdcParams& p, const unsigned its_per_stream, const int warp, const int lane,
                                     const int l_base, unsigned long long* const full, const bool want_pw,
                                     const float pw_scale, Issue issue, Dec dec, Back back) {
    const unsigned gw = blockIdx.x * WARPS + warp, GW = gridDim.x * WARPS;
    const unsigned long long total = (unsigned long long)p.n_streams * its_per_stream;
    const unsigned long long b0 = total * gw / GW, b1 = total * (gw + 1ull) / GW;
    if (b0 >= b1) return;
    const int ips = (int)its_per_stream, n_out = (int)p.n_out;
    const size_t row_bytes = (size_t)p.n * ES, tail_bytes = (size_t)p.ht * ES;
    unsigned s = (unsigned)(b0 / its_per_stream);
    int it_first = (int)(b0 % its_per_stream);
    unsigned left = (unsigned)(b1 - b0);                   // stored iterations still to do
    const unsigned char* chunk = (const unsigned char*)p.iq + s * row_bytes;
    const unsigned char* tail = (const unsigned char*)p.tail_in + s * tail_bytes;
    if (lane == 0) {                                        // warm-up (and first stored iteration) of the first piece
#pragma unroll
        for (int k = 0; k < NSTAGE; k++) issue(k, tail, chunk, l_base + XNEW * (it_first - 1 + k));
    }
    unsigned use = 0;

    while (left) {
      const int n_st = min(ips - it_first, (int)left);     // stored iterations of this piece
      const int npiece = n_st + 1;
      left -= (unsigned)n_st;
      float* const out_lane = p.bb + (size_t)s * p.row_stride + P25CU_BB_HIST + R * lane;
      float pw = 0.f;
      for (int j = 0; j < npiece; j++, use++) {
        const int it = it_first - 1 + j;
        const int stage = use % NSTAGE;
        const int nv = j ? min(n_out - NOUT * it, NOUT) : 0;     // j = 0 is the warm-up: nothing is stored
        mbar_wait(&full[stage], (use / NSTAGE) & 1);
        dec(stage, it);
        __syncwarp();                                                                 // S1: slice consumed, rows visible
        if (lane == 0) {
            if (j + NSTAGE < npiece) issue(stage, tail, chunk, l_base + XNEW * (it + NSTAGE));
            // else the next piece's iteration j + NSTAGE - 1 - npiece (its warm-up is -1); with one stage only the last
            // iteration gets here and asks for that warm-up
            else if (left) issue(stage, tail + tail_bytes, chunk + row_bytes, l_base + XNEW * (NSTAGE == 1 ? -1 : j + NSTAGE - 1 - npiece));
        }
        back(nv, out_lane + NOUT * it, pw);
      }
      // ---- end of the piece: flush power, carry the raw input tail when the stream's chunk is complete, next stream
      if (want_pw) {
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) pw += __shfl_xor_sync(0xFFFFFFFFu, pw, o);
          if (lane == 0) atomicAdd(p.power_sum + s, pw * pw_scale);
      }
      if (it_first + n_st == ips) {
          // the next chunk's tail is (tail ++ chunk)[n, n + ht): groups [0, nt) are the end of the old tail when the chunk
          // is shorter than it, the rest the chunk's last bytes (aligned rows: whole 16-byte groups either way)
          const int nt = row_bytes < tail_bytes ? (int)((tail_bytes - row_bytes) / 16) : 0;
          const uint4* src = reinterpret_cast<const uint4*>(chunk + ((long long)p.n - (long long)p.ht) * ES);   // group i >= nt
          uint4* dst = reinterpret_cast<uint4*>((unsigned char*)p.tail_out + s * tail_bytes);
          for (int i = lane; i < nt; i += 32) dst[i] = reinterpret_cast<const uint4*>(tail + row_bytes)[i];
          for (int i = nt + lane; i < (int)(tail_bytes / 16); i += 32) dst[i] = src[i];
      }
      s++;
      it_first = 0;
      chunk += row_bytes;
      tail += tail_bytes;
    }
}

// The 48 kHz stages of one iteration, R outputs per lane on lanes [0, NL) (w5: lane 31 only feeds the decimator):
//   * decimator outputs are rows of R samples split over R / 2 arrays of 16-byte pairs, ys rows apart:
//     yd[q ys + i] = (y[R i + 2 q], y[R i + 2 q + 1]); rows 0 .. HROWS - 1 are the history, row HROWS + lane the lane's
//     own outputs, so a lane's channel-filter window is the consecutive rows lane .. lane + HROWS;
//   * discriminator outputs are rows of R split over R / 4 arrays of four, ds rows apart, DROWS history rows in front;
//   * c_carry is the last channel-filter output of the previous iteration, pw the power of the stored outputs.
template <int R, int NL, int HROWS, int DROWS>
__device__ __forceinline__ void back_end(float4* const yd, const int ys, float4* const d, const int ds, const int lane,
                                         const float dc, float2& c_carry, const bool want_pw, float& pw, const int nv,
                                         float* const out) {
    constexpr int NQ = R / 2, ND = R / 4;
    static_assert(R % 4 == 0 && HROWS * R == P25_TAPS_CHAN - 1 && DROWS * R >= P25_BOXCAR - 1, "history rows");

    // ---- channel-select FIR: outputs R lane + r, window = rows lane .. lane + HROWS (s = 40 + r - k), samples in order
    float2 acc[R];
#pragma unroll
    for (int r = 0; r < R; r++) acc[r] = make_float2(dc, dc);
#pragma unroll
    for (int t = 0; t <= HROWS; t++) {
#pragma unroll
        for (int q = 0; q < NQ; q++) {
            const float4 v = yd[q * ys + lane + t];
            const float2 x[2] = {make_float2(v.x, v.y), make_float2(v.z, v.w)};
#pragma unroll
            for (int e = 0; e < 2; e++) {
#pragma unroll
                for (int r = 0; r < R; r++) {
                    const int k = (P25_TAPS_CHAN - 1) + r - (R * t + 2 * q + e);
                    if (k >= 0 && k < P25_TAPS_CHAN) acc[r] = cfma(c_taps_chan[k], x[e], acc[r]);
                }
            }
        }
    }
    // ---- FM discriminator on the outputs in registers; the sample before comes from the lane below
    float2 prev;
    prev.x = __shfl_up_sync(0xFFFFFFFFu, acc[R - 1].x, 1);
    prev.y = __shfl_up_sync(0xFFFFFFFFu, acc[R - 1].y, 1);
    if (lane == 0) prev = c_carry;
    c_carry.x = __shfl_sync(0xFFFFFFFFu, acc[R - 1].x, NL - 1);
    c_carry.y = __shfl_sync(0xFFFFFFFFu, acc[R - 1].y, NL - 1);
    float dd[R];
#pragma unroll
    for (int r = 0; r < R; r += 2) {
        const float2 c0 = acc[r], c1 = acc[r + 1];
        const float2 re = make_float2(c0.x * prev.x + c0.y * prev.y, c1.x * c0.x + c1.y * c0.y);
        const float2 im = make_float2(c0.y * prev.x - c0.x * prev.y, c1.y * c0.x - c1.x * c0.y);
        const float2 th = disc_atan2_pair(im, re);
        dd[r] = th.x * P25_FM_GAIN;
        dd[r + 1] = th.y * P25_FM_GAIN;
        if (want_pw && R * lane + r < nv) pw += c0.x * c0.x + c0.y * c0.y;
        if (want_pw && R * lane + r + 1 < nv) pw += c1.x * c1.x + c1.y * c1.y;
        prev = c1;
    }
#pragma unroll
    for (int h = 0; h < ND; h++) d[h * ds + DROWS + lane] = make_float4(dd[4 * h], dd[4 * h + 1], dd[4 * h + 2], dd[4 * h + 3]);
    __syncwarp();                                                                     // S2

    // ---- boxcar over d[o - 9 .. o], o = R lane + r: old[i] = d[R lane - 9 + i] from the DROWS rows below the lane's own
    {
        float old[P25_BOXCAR - 1];
#pragma unroll
        for (int i = 0; i < P25_BOXCAR - 1; i++) {
            const int m = R * DROWS - (P25_BOXCAR - 1) + i;                           // sample m of rows lane ..
            const float4 v = d[(m % R) / 4 * ds + lane + m / R];
            old[i] = m % 4 == 0 ? v.x : m % 4 == 1 ? v.y : m % 4 == 2 ? v.z : v.w;
        }
        float sum[R];
        float s0 = old[0] + old[1];
#pragma unroll
        for (int i = 2; i < P25_BOXCAR - 1; i++) s0 += old[i];
        sum[0] = s0 + dd[0];
#pragma unroll
        for (int r = 1; r < R; r++) sum[r] = (sum[r - 1] - old[r - 1]) + dd[r];
        const float kk = 1.0f / P25_BOXCAR;
        const int o0 = R * lane;
        if (o0 < nv) {
            if (o0 + R - 1 < nv) {
#pragma unroll
                for (int h = 0; h < ND; h++)
                    reinterpret_cast<float4*>(out)[h] = make_float4(sum[4 * h] * kk, sum[4 * h + 1] * kk, sum[4 * h + 2] * kk, sum[4 * h + 3] * kk);
            } else {
#pragma unroll
                for (int r = 0; r < R; r++)
                    if (o0 + r < nv) out[r] = sum[r] * kk;
            }
        }
    }
    // ---- roll the histories: rows NL .. of every array move to the front (HROWS decimator rows, DROWS discriminator rows)
    if constexpr (R == 4) {                                 // a lane moves one row of both decimator arrays
        float4 ra = make_float4(0.f, 0.f, 0.f, 0.f), rb = ra, rd = ra;
        if (lane < HROWS) {
            ra = yd[NL + lane];
            rb = yd[ys + NL + lane];
        }
        if (lane < DROWS) rd = d[NL + lane];
        __syncwarp();                                                                 // S3
        if (lane < HROWS) {
            yd[lane] = ra;
            yd[ys + lane] = rb;
        }
        if (lane < DROWS) d[lane] = rd;
    } else {                                                // R = 8: a lane moves one row of one array
        float4 ry = make_float4(0.f, 0.f, 0.f, 0.f), rd = ry;
        const int yq = lane / HROWS, yr = lane - HROWS * yq;
        if (lane < NQ * HROWS) ry = yd[yq * ys + NL + yr];
        if (lane < 2 * DROWS) rd = (lane & 1) ? d[ds + NL + (lane >> 1)] : d[NL + (lane >> 1)];
        __syncwarp();                                                                 // S3
        if (lane < NQ * HROWS) yd[yq * ys + yr] = ry;
        if (lane < 2 * DROWS) {
            if (lane & 1) d[ds + (lane >> 1)] = rd;
            else d[lane >> 1] = rd;
        }
    }
}

}  // namespace wk


// Integer tensor pipe helpers of the u8 kernels (w5i, w50i): mma.sync u8 x s8 with s32 accumulators whose start values
// make them floats (see w5i below).
namespace i8 {

using namespace prim;

__device__ __forceinline__ void imma(int (&d)[4], const unsigned (&a)[4], const uint2 b) {
    asm("mma.sync.aligned.m16n8k32.row.col.s32.u8.s8.s32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+r"(d[0]), "+r"(d[1]), "+r"(d[2]), "+r"(d[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b.x), "r"(b.y));
}
// first k-step of a chain: the start value (one register for all four accumulators) is the C operand
__device__ __forceinline__ void imma0(int (&d)[4], const unsigned (&a)[4], const uint2 b, const int (&c)[4]) {
    asm("mma.sync.aligned.m16n8k32.row.col.s32.u8.s8.s32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%10,%11,%12,%13};"
        : "=r"(d[0]), "=r"(d[1]), "=r"(d[2]), "=r"(d[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b.x), "r"(b.y), "r"(c[0]), "r"(c[1]), "r"(c[2]), "r"(c[3]));
}
// 4-byte shared-memory load the compiler may not fuse with its neighbour (an 8-byte load would need four moves to put
// the words into the fragment's register order)
__device__ __forceinline__ unsigned lds32(unsigned addr) {
    unsigned v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
// the three start values as register quads that stay resident (opaque to the compiler, which otherwise rebuilds a
// quad with four moves in front of every chain: 41 MOV per iteration)
__device__ __forceinline__ void load_init(const int4* g_init, int (&init)[3][4]) {
#pragma unroll
    for (int l = 0; l < 3; l++) {
        const int4 v = g_init[l];
        init[l][0] = v.x; init[l][1] = v.y; init[l][2] = v.z; init[l][3] = v.w;
    }
}
// accumulator pair h ((c0, c1) or (c2, c3)) of the three limbs -> y = 2^16 s2 + 2^8 s1 + s0 as one complex output:
// one FADD2 per limb removes the start value 1.5 * 2^23, two FFMA2 combine the limbs with a single rounding
__device__ __forceinline__ float2 limbs_to_float(const int (&acc)[3][4], const int h) {
    const float2 unmagic = make_float2(-12582912.f, -12582912.f);
    float2 f[3];
#pragma unroll
    for (int l = 0; l < 3; l++)
        f[l] = add2(make_float2(__int_as_float(acc[l][2 * h]), __int_as_float(acc[l][2 * h + 1])), unmagic);
    return cfma(65536.f, f[2], cfma(256.f, f[1], f[0]));
}

}  // namespace i8


// =====================================================================================================
// /5 fast path for cf32 input (the reference's own chain at 240 kS/s; 16-byte aligned rows), a warp kernel (above):
//   * 124 outputs per iteration (31 lanes x 4; lane 31 only contributes its inputs' partial sums to lane 30);
//   * the raw 5.1 KB input slices go into a two-stage ring;
//   * decimator: a lane owns 20 consecutive inputs and forms its four outputs' own part plus the part it contributes
//     to its left neighbour's last outputs, which neighbours exchange by warp shuffle (25 FFMA2 per output);
//   * decimator outputs are kept as rows of four (two 16-byte halves in two arrays): a lane's 44-sample channel
//     filter window is then 22 conflict-free LDS.128 of consecutive rows; stores are 496 contiguous bytes per warp.
// =====================================================================================================
namespace w5 {

using namespace prim;

constexpr int R = 4;                        // outputs per lane
constexpr int NOUT = 31 * R;                // 124 outputs per warp iteration
constexpr int XNEW = 5 * NOUT;              // 620 fresh input samples per iteration
constexpr int XN = 32 * 5 * R;              // 640 samples read (the ghost lane's 20 included)
constexpr int WARPS = 4;                    // per CTA
constexpr int AL = 2, ES = 8;               // samples per 16 bytes, bytes per sample
constexpr int XLEN = (XN + 2 * AL - 2) / AL * AL;
constexpr int XBYTES = (XLEN * ES + 127) / 128 * 128;   // 5.1 KB slices
constexpr int MINB = 4;                     // CTAs per SM
constexpr int HROWS = (P25_TAPS_CHAN - 1) / R;        // 10 history rows of the decimator output
constexpr int DROWS = 3;                    // history rows of the discriminator output (>= 9 samples)
static_assert((P25_TAPS_CHAN - 1) % R == 0 && DROWS * R >= P25_BOXCAR - 1, "history rows");

struct __align__(128) WarpSm {
    unsigned char xs[2][XBYTES];
    float4 ydA[HROWS + 32], ydB[HROWS + 32];    // row i: (yd[4i], yd[4i+1]) | (yd[4i+2], yd[4i+3])
    float4 d4[DROWS + 32];
    unsigned long long full[2];
};
constexpr size_t SMEM = sizeof(WarpSm) * WARPS;         // dynamic shared memory per CTA

__global__ void __launch_bounds__(32 * WARPS, MINB) p25_ddc5_warp_kernel(const DdcParams p, const unsigned its_per_stream,
                                                                         const float dc, const float pw_scale) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    WarpSm& sm = reinterpret_cast<WarpSm*>(smem_raw)[warp];
    if (lane == 0) {
        mbar_init(&sm.full[0], 1);
        mbar_init(&sm.full[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    for (int i = lane; i < HROWS + 32; i += 32) sm.ydA[i] = sm.ydB[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int i = lane; i < DROWS + 32; i += 32) sm.d4[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    __syncwarp();

    const int ht = (int)p.ht, lend = (int)p.ht + (int)p.n;
    const int l_base = (int)(5 * (long long)p.m0 - (long long)p.a0) - 20 + ht;   // logical index of iteration 0's first input
    const bool want_pw = p.power_sum != nullptr;
    float2 c_carry = make_float2(0.f, 0.f);
    wk::walk<2, WARPS, R, NOUT, XNEW, ES>(
        p, its_per_stream, warp, lane, l_base, sm.full, want_pw, pw_scale,
        [&](int stage, const unsigned char* tail, const unsigned char* chunk, int l0) {
            wk::issue_slice<ES, AL, XLEN, false>(sm.xs[stage], &sm.full[stage], ht, lend, tail, chunk, l0);
        },
        [&](int stage, int it) {
            // ---- /5 decimator: lane owns inputs [20 lane, 20 lane + 20)
            const int skew = (l_base + XNEW * it) & (AL - 1);
            float2 own[R];
            float2 x[5 * R];
            const int s0 = skew + 5 * R * lane;
            // 16-byte loads (two samples): half the wavefronts of LDS.64 at this 160-byte lane stride
            const float4* xp = reinterpret_cast<const float4*>(reinterpret_cast<const float2*>(sm.xs[stage]) + (s0 & ~1));
            if (s0 & 1) {
#pragma unroll
                for (int i = 0; i <= 5 * R / 2; i++) {
                    const float4 v = xp[i];
                    if (i > 0) x[2 * i - 1] = make_float2(v.x, v.y);
                    if (i < 5 * R / 2) x[2 * i] = make_float2(v.z, v.w);
                }
            } else {
#pragma unroll
                for (int i = 0; i < 5 * R / 2; i++) {
                    const float4 v = xp[i];
                    x[2 * i] = make_float2(v.x, v.y);
                    x[2 * i + 1] = make_float2(v.z, v.w);
                }
            }
            float2 lft[R];
#pragma unroll
            for (int r = 0; r < R; r++) {
                own[r] = make_float2(0.f, 0.f);
                lft[r] = make_float2(0.f, 0.f);
#pragma unroll
                for (int k = P25_TAPS_DECIM - 1; k >= 0; k--) {
                    if ((P25_TAPS_DECIM_ZERO_MASK >> k) & 1) continue;  // taps that are zero to working precision (4 of 25)
                    const int idx = 5 * r + (P25_TAPS_DECIM - 1) - k;
                    if (idx < 5 * R) own[r] = cfma(c_taps_decim[k], x[idx], own[r]);
                    else lft[r] = cfma(c_taps_decim[k], x[idx - 5 * R], lft[r]);
                }
            }
#pragma unroll
            for (int r = 0; r < R; r++) {
                if (5 * r + (P25_TAPS_DECIM - 1) >= 5 * R) {
                    own[r].x += __shfl_down_sync(0xFFFFFFFFu, lft[r].x, 1);
                    own[r].y += __shfl_down_sync(0xFFFFFFFFu, lft[r].y, 1);
                }
            }
            sm.ydA[HROWS + lane] = make_float4(own[0].x, own[0].y, own[1].x, own[1].y);   // lane 31's row is never read
            sm.ydB[HROWS + lane] = make_float4(own[2].x, own[2].y, own[3].x, own[3].y);
        },
        [&](int nv, float* out, float& pw) {
            wk::back_end<R, 31, HROWS, DROWS>(sm.ydA, (int)(sm.ydB - sm.ydA), sm.d4, 0, lane, dc, c_carry, want_pw, pw, nv, out);
        });
}

}  // namespace w5


// =====================================================================================================
// /5 warp kernel for u8 input with the DECIMATOR ON THE INTEGER TENSOR PIPE (round 2; VERDICT r1 item 4: "integer-domain
// decimator on the raw bytes").  On FFMA2 alone (the warp kernel above) the /5 chain is bound by the FP32 pipe: 21 of its
// 62 FIR FFMA2 per output are the /5 decimator, and every u8 input byte would cost two PRMT + half a FADD2 before it
// could enter an FFMA2.  Here the raw bytes
// go into mma.sync.m16n8k32.s32.u8.s8 as they lie in the TMA-staged slice, without any conversion:
//   * A (16 x 32 bytes per k-step) = sixteen overlapping rows of the slice, row m starting 40 samples (80 bytes) after
//     row m - 1, interleaved I/Q bytes along k; a row's 64-sample window holds the inputs of eight consecutive outputs;
//   * B = the taps as a banded matrix: column 2 n' + c (output n', component c) has tap k = 24 - d at the byte of sample
//     skew + 5 n + d, component c, zero elsewhere.  The taps are 24-bit fixed point, t = round(h 2^25) (an error of
//     2^-26 per tap, the spacing of fp32 at the largest tap), split into three balanced s8 limbs -> three products
//     with s32 accumulators; two n-tiles (outputs 0..3 | 4..7 of every row) x three k-steps each x three limbs =
//     18 IMMA per 128 outputs, 8.35 clocks each per sub-core beside an FFMA2 stream that keeps 85 % of its peak
//     (profiles/pipe_peaks_r02.json);
//   * the sums are exact integers.  The accumulators start at the bit pattern of 1.5 * 2^23 minus 128 * (sum of the
//     limb), so they ARE the floats 1.5 * 2^23 + sum l (u - 128): one FADD2 per limb and two FFMA2 give
//     y = 2^16 s2 + 2^8 s1 + s0 with a single rounding (I2F runs at 32 per clock per SM: not an option).  y is the
//     decimator output in byte units x 2^25; the discriminator does not see the scale, dc and the power scale carry it.
//   * the stream's alignment inside its 16-byte group (skew = 4 a + sk) is constant over a launch: a shifts the row
//     pointers by 8 bytes, sk selects one of four B tables (a window holds sk + 60 <= 63 samples).
//   * the k index is permuted so that a lane's eight words of a row are four 8-byte loads, and mma row g reads slice
//     row 2 (g & 3) + (g >> 2): both halves of the warp then hit 32 different banks (row stride 20 words).
// 128 outputs per iteration on all 32 lanes (no ghost lane); everything after the decimator is the common warp kernel code.
// =====================================================================================================
namespace w5i {

using namespace prim;
using namespace i8;

constexpr int R = 8;                                    // outputs per lane
constexpr int NOUT = 32 * R;                            // 256 outputs per warp iteration: two m-tiles of 16 rows x 8 outputs
constexpr int XNEW = 5 * NOUT;                          // 1280 fresh input samples (2560 bytes: the skew never changes)
constexpr int XREAD = 5 * (NOUT - 1) + P25_TAPS_DECIM;  // 1300 samples read
constexpr int WARPS = 4;
constexpr int AL = 8, ES = 2;
constexpr int XLEN = (XREAD + 2 * AL - 2) / AL * AL;    // 1312
constexpr int XBYTES = (XLEN * ES + 127) / 128 * 128;   // 2688
constexpr int MINB = 4;
constexpr int HROWS = (P25_TAPS_CHAN - 1) / R;          // 5 history rows (of eight) of the decimator output
constexpr int YROWS = HROWS + 32;                       // 37 rows x 4 words = 4 (mod 8) words between the four arrays
constexpr int DROWS = 2;                                // history rows of the discriminator output (>= 9 samples)
constexpr int NB = 18;                                  // B fragments: [n-tile][k-step - n-tile][limb]
constexpr int SCALE_LOG2 = 25;                          // taps as round(h * 2^25): |t| < 2^23
static_assert(XLEN * ES >= 80 * 31 + 8 + 128 && XNEW % (2 * AL) == 0, "A rows inside the slice; constant skew");
static_assert((P25_TAPS_CHAN - 1) % R == 0 && DROWS * R >= P25_BOXCAR - 1 && (YROWS * 4) % 8 == 4, "history rows, store banks");

// decimator outputs as rows of eight, split over four arrays of 16-byte pairs: yd[q][i] = (y[8 i + 2 q], y[8 i + 2 q + 1]).
// A lane's 48-sample channel-filter window is 24 LDS.128 at a 16-byte lane stride (no conflicts), and the fragment
// stores of the decimator (below) hit 32 different banks.
struct __align__(128) WarpSm {
    unsigned char xs[2][XBYTES];
    float4 yd[4][YROWS];
    float4 dA[DROWS + 32], dB[DROWS + 32];      // discriminator outputs: (d[8 i .. 8 i + 3]) | (d[8 i + 4 .. 8 i + 7])
    unsigned long long full[2];
};
constexpr size_t SMEM = sizeof(WarpSm) * WARPS + sizeof(uint2) * NB * 32;   // dynamic shared memory per CTA: + B table

__device__ uint2 g_btab[4][NB][32];             // [sk][fragment][lane] = (b0, b1)
__device__ int4 g_init[3];                      // accumulator start value of every limb, four times (one C operand quad)

template <bool PW>                              // PW: accumulate the channel power (every fourth chunk in the reference's cadence)
__global__ void __launch_bounds__(32 * WARPS, MINB) p25_ddc5_imma_kernel(const DdcParams p, const unsigned its_per_stream,
                                                                         const float dc, const float pw_scale) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    WarpSm& sm = reinterpret_cast<WarpSm*>(smem_raw)[warp];
    uint2* const btab = reinterpret_cast<uint2*>(smem_raw + sizeof(WarpSm) * WARPS);
    const int ht = (int)p.ht, lend = (int)p.ht + (int)p.n;
    const int l_base = (int)(5 * (long long)p.m0 - (long long)p.a0) - 20 + ht;   // logical index of iteration 0's first input
    const int skew = l_base & (AL - 1);                     // the same for every iteration of every stream
    for (int e = threadIdx.x; e < NB * 32; e += 32 * WARPS) btab[e] = (&g_btab[skew & 3][0][0])[e];
    if (lane == 0) {
        mbar_init(&sm.full[0], 1);
        mbar_init(&sm.full[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    for (int i = lane; i < 4 * YROWS; i += 32) (&sm.yd[0][0])[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int i = lane; i < DROWS + 32; i += 32) sm.dA[i] = sm.dB[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    __syncthreads();

    // fragment geometry: mma rows g and g + 8 of m-tile mt read slice rows 16 mt + drow and + 8; a lane's words of a
    // k-step are t and t + 4 of its eight (row stride 20 words: 32 different banks for any row permutation); the row
    // permutation puts the half-warps' stores on rows {0, 2, 4, 6} / {1, 3, 5, 7} (+ 8, + 16 ...) of two arrays each
    const int g = lane >> 2, tig = lane & 3;
    const int drow = ((g & 3) << 1) | (g >> 2);
    const unsigned a_off = 80u * drow + 8u * (skew >> 2) + 4u * tig;
    const uint2* const bl = btab + lane;
    float2* const ydst = reinterpret_cast<float2*>(&sm.yd[tig >> 1][HROWS + drow]) + (tig & 1);
    int init[3][4];
    load_init(g_init, init);
    float2 c_carry = make_float2(0.f, 0.f);
    wk::walk<2, WARPS, R, NOUT, XNEW, ES>(
        p, its_per_stream, warp, lane, l_base, sm.full, PW, pw_scale,
        [&](int stage, const unsigned char* tail, const unsigned char* chunk, int l0) {
            wk::issue_slice<ES, AL, XLEN, false>(sm.xs[stage], &sm.full[stage], ht, lend, tail, chunk, l0);
        },
        [&](int stage, int) {
            // ---- /5 decimator on the integer tensor pipe: 36 IMMA, every B fragment loaded once for both m-tiles
            int acc[2][2][3][4];
            const unsigned xa = smem_u32(sm.xs[stage]) + a_off;
#pragma unroll
            for (int ks = 0; ks < 4; ks++) {
                unsigned a[2][4];
#pragma unroll
                for (int mt = 0; mt < 2; mt++) {
                    const unsigned ad = xa + 1280u * mt + 32u * ks;
                    a[mt][0] = lds32(ad);
                    a[mt][1] = lds32(ad + 640u);
                    a[mt][2] = lds32(ad + 16u);
                    a[mt][3] = lds32(ad + 656u);
                }
#pragma unroll
                for (int nt = 0; nt < 2; nt++) {
                    const int jj = ks - nt;
                    if (jj < 0 || jj > 2) continue;
#pragma unroll
                    for (int l = 0; l < 3; l++) {
                        const uint2 b = bl[32 * ((nt * 3 + jj) * 3 + l)];
#pragma unroll
                        for (int mt = 0; mt < 2; mt++) {
                            if (jj == 0) imma0(acc[mt][nt][l], a[mt], b, init[l]);
                            else imma(acc[mt][nt][l], a[mt], b);
                        }
                    }
                }
            }
            // (c0, c1) = (re, im) of output 128 mt + 8 drow + 4 nt + tig, (c2, c3) of that output + 64
#pragma unroll
            for (int mt = 0; mt < 2; mt++)
#pragma unroll
                for (int nt = 0; nt < 2; nt++)
#pragma unroll
                    for (int h = 0; h < 2; h++) ydst[2 * (2 * nt * YROWS + 16 * mt + 8 * h)] = limbs_to_float(acc[mt][nt], h);
        },
        [&](int nv, float* out, float& pw) {
            wk::back_end<R, 32, HROWS, DROWS>(&sm.yd[0][0], YROWS, sm.dA, (int)(sm.dB - sm.dA), lane, dc, c_carry, PW, pw, nv, out);
        });
}

// host side: the banded tap matrix in fragment order and the accumulator start values (p25_imma_tables.h, plain C++ so that
// the CPU suite can check the very tables this library uploads against the numpy dataflow model)
using Tables = p25imma::Tables5;
static_assert(NB == p25imma::NB5 && SCALE_LOG2 == p25imma::SCALE5 && sizeof(g_btab) == sizeof(Tables::b), "table geometry");
static const Tables& tables() {
    static const Tables t(P25_TAPS_DECIM_H);
    return t;
}

}  // namespace w5i


// =====================================================================================================
// u8 at 2.4 MS/s (/50) with BOTH decimating stages on the integer tensor pipe (round 2).  The /10 front stage and the /5
// decimator are linear and see nothing but bytes in front of them, so their cascade is ONE 290-tap FIR at 2.4 MS/s,
// g[10 k + i] = hd[k] hf[i], decimating by 50 straight to the 48 kHz decimator output -- 290 exact integer MACs per
// output and component instead of 250 + 21 FFMA2 (on FFMA2 the u8 /50 chain is FP32-bound: 30 % of the FFMA2 peak at 28 %
// of HBM).  Same scheme as w5i: raw bytes as the A operand (sixteen overlapping rows of the TMA-staged slice, 200 samples
// = 400 bytes apart, four outputs per row = one n-tile), the taps as a banded s8 matrix in three balanced limbs of
// t = round(g 2^28), accumulators started at the bit pattern of 1.5 * 2^23 - 128 * (limb sum) so that they are floats,
// y = 2^16 s2 + 2^8 s1 + s0 in one FADD2 per limb + two FFMA2.  28 k-steps x 3 limbs = 84 IMMA per 64 outputs; every B
// fragment (21.5 KB table per CTA) is loaded once for the two m-tiles of a 128-output warp iteration.  The row stride of
// 100 words puts the 32 lanes of every fragment load on 32 different banks; the four outputs of a row are one row of
// the channel filter's window arrays.  The 48 kHz stages are the common warp kernel code (4 outputs per lane).
// The warm-up iteration of a piece that starts a chunk reaches 6,640 samples back but only its last 50 outputs (2,740
// samples, inside the 3,264-sample tail) have to be right: bytes in front of the tail are simply not copied, and whatever
// lies in the buffer gives finite garbage in outputs nobody keeps.
// =====================================================================================================
namespace w50i {

using namespace prim;
using namespace i8;

constexpr int D = 50;
constexpr int G = P25_TAPS_FRONT + P25_DECIM_FRONT * (P25_TAPS_DECIM - 1);   // 290 combined taps
constexpr int R = 4;
constexpr int NOUT = 32 * R;                            // 128 outputs per warp iteration: two m-tiles of 16 rows x 4 outputs
constexpr int XNEW = D * NOUT;                          // 6400 fresh input samples per iteration
constexpr int XREAD = D * (NOUT - 1) + G;               // 6640 samples read
constexpr int WARPS = 12;                               // one CTA per SM, three warps per scheduler: 12 x 15 KB + the B table
constexpr int AL = 8, ES = 2;
constexpr int XLEN = (XREAD + 2 * AL - 2) / AL * AL;    // 6648
constexpr int KS = 28;                                  // k-steps: 1 + 150 + 290 = 441 samples <= 448
constexpr int XBYTES = (400 * 31 + 12 + 32 * KS + 127) / 128 * 128;   // 13312: every A load stays inside the stage buffer
constexpr int HROWS = (P25_TAPS_CHAN - 1) / R;          // 10
constexpr int DROWS = 3;
constexpr int NB = KS * 3;                              // B fragments: [k-step][limb]
constexpr int SCALE_LOG2 = 28;                          // taps as round(g * 2^28): |t| < 2^23
static_assert(XBYTES >= XLEN * ES && XNEW % (2 * AL) == 0 && 1 + D * 3 + G <= 16 * KS, "slice, constant skew, window");
static_assert((P25_TAPS_CHAN - 1) % R == 0 && DROWS * R >= P25_BOXCAR - 1, "history rows");

struct __align__(128) WarpSm {
    unsigned char xs[XBYTES];                   // ONE stage: the next slice is requested as soon as this one is consumed and
                                                // lands while the other two warps of the scheduler own the tensor pipe
    float4 ydA[HROWS + 32 + 2];                 // 44 rows: ydB starts 16 banks further (half-warp stores: 32 banks)
    float4 ydB[HROWS + 32];
    float4 d4[DROWS + 32];
    unsigned long long full;
};
constexpr size_t SMEM = sizeof(WarpSm) * WARPS + sizeof(uint2) * NB * 32;   // dynamic shared memory per CTA: + B table

__device__ uint2 g_btab[2][NB][32];             // [skew & 1][fragment][lane]
__device__ int4 g_init[3];

template <bool PW>
__global__ void __launch_bounds__(32 * WARPS, 1) p25_ddc50_imma_kernel(const DdcParams p, const unsigned its_per_stream,
                                                                       const float dc, const float pw_scale) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    WarpSm& sm = reinterpret_cast<WarpSm*>(smem_raw)[warp];
    uint2* const btab = reinterpret_cast<uint2*>(smem_raw + sizeof(WarpSm) * WARPS);
    const int ht = (int)p.ht, lend = (int)p.ht + (int)p.n;
    // logical index (tail ++ chunk) of the first input of iteration 0's window: output m uses 50 m + lbase + [-240, 49]
    const int l_base = (int)(D * (long long)p.m0 - (long long)p.a0) - (G - D) + ht;
    const int skew = l_base & (AL - 1);                     // the same for every iteration of every stream
    for (int e = threadIdx.x; e < NB * 32; e += 32 * WARPS) btab[e] = (&g_btab[skew & 1][0][0])[e];
    if (lane == 0) {
        mbar_init(&sm.full, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    for (int i = lane; i < XBYTES / 16; i += 32) reinterpret_cast<uint4*>(sm.xs)[i] = make_uint4(0u, 0u, 0u, 0u);
    for (int i = lane; i < HROWS + 32; i += 32) sm.ydA[i] = sm.ydB[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int i = lane; i < DROWS + 32; i += 32) sm.d4[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");      // the zeroed stage buffers are overwritten by bulk copies
    __syncthreads();

    // fragment geometry: mma rows g and g + 8 of m-tile mt read slice rows 16 mt + g and + 8 (400 bytes apart); the
    // lane's words of a k-step are t and t + 4 of its eight; (c0, c1) / (c2, c3) are output 4 row + t
    const int g = lane >> 2, tig = lane & 3;
    const unsigned a_off = 400u * g + 4u * (skew >> 1) + 4u * tig;
    const uint2* const bl = btab + lane;
    float2* const ydst = reinterpret_cast<float2*>(tig < 2 ? &sm.ydA[HROWS + g] : &sm.ydB[HROWS + g]) + (tig & 1);
    int init[3][4];
    load_init(g_init, init);
    float2 c_carry = make_float2(0.f, 0.f);
    wk::walk<1, WARPS, R, NOUT, XNEW, ES>(
        p, its_per_stream, warp, lane, l_base, &sm.full, PW, pw_scale,
        [&](int, const unsigned char* tail, const unsigned char* chunk, int l0) {
            wk::issue_slice<ES, AL, XLEN, true>(sm.xs, &sm.full, ht, lend, tail, chunk, l0);
        },
        [&](int, int) {
            // ---- /50: 290-tap FIR on the raw bytes, 168 IMMA
            int acc[2][3][4];
            const unsigned xa = smem_u32(sm.xs) + a_off;
#pragma unroll
            for (int ks = 0; ks < KS; ks++) {
                unsigned a[2][4];
#pragma unroll
                for (int mt = 0; mt < 2; mt++) {
                    const unsigned ad = xa + 6400u * mt + 32u * ks;
                    a[mt][0] = lds32(ad);
                    a[mt][1] = lds32(ad + 3200u);
                    a[mt][2] = lds32(ad + 16u);
                    a[mt][3] = lds32(ad + 3216u);
                }
#pragma unroll
                for (int l = 0; l < 3; l++) {
                    const uint2 b = bl[32 * (ks * 3 + l)];
#pragma unroll
                    for (int mt = 0; mt < 2; mt++) {
                        if (ks == 0) imma0(acc[mt][l], a[mt], b, init[l]);
                        else imma(acc[mt][l], a[mt], b);
                    }
                }
            }
#pragma unroll
            for (int mt = 0; mt < 2; mt++)
#pragma unroll
                for (int h = 0; h < 2; h++) ydst[2 * (16 * mt + 8 * h)] = limbs_to_float(acc[mt], h);
        },
        [&](int nv, float* out, float& pw) {
            wk::back_end<R, 32, HROWS, DROWS>(sm.ydA, (int)(sm.ydB - sm.ydA), sm.d4, 0, lane, dc, c_carry, PW, pw, nv, out);
        });
}

// host side: combined taps (double), limbs, banded matrix in fragment order, accumulator start values (p25_imma_tables.h)
using Tables = p25imma::Tables50;
static_assert(NB == p25imma::NB50 && KS == p25imma::KS50 && SCALE_LOG2 == p25imma::SCALE50 && G == p25imma::G50 &&
              sizeof(g_btab) == sizeof(Tables::b), "table geometry");
static const Tables& tables() {
    static const Tables t(P25_TAPS_FRONT_H, P25_TAPS_DECIM_H);
    return t;
}

}  // namespace w50i

unsigned p25cu_ddc_tail_len(int decimation) { return decimation == 50 ? Cfg<true>::HT : Cfg<false>::HT; }

// the banded tap matrix and the accumulator start values (one C operand quad per limb) of an integer kernel
template <typename T, typename B>
static cudaError_t upload_imma(const T& t, const B& g_btab, const int4 (&g_init)[3]) {
    if (!t.ok) return cudaErrorInvalidValue;
    cudaError_t e = cudaMemcpyToSymbol(g_btab, t.b, sizeof(g_btab));
    if (e != cudaSuccess) return e;
    const int4 q[3] = {make_int4(t.init[0], t.init[0], t.init[0], t.init[0]), make_int4(t.init[1], t.init[1], t.init[1], t.init[1]),
                       make_int4(t.init[2], t.init[2], t.init[2], t.init[2])};
    return cudaMemcpyToSymbol(g_init, q, sizeof(q));
}

cudaError_t p25cu_ddc_upload_taps() {
    cudaError_t e;
    if ((e = cudaMemcpyToSymbol(c_taps_front, P25_TAPS_FRONT_H, sizeof(c_taps_front))) != cudaSuccess) return e;
    if ((e = cudaMemcpyToSymbol(c_taps_decim, P25_TAPS_DECIM_H, sizeof(c_taps_decim))) != cudaSuccess) return e;
    if ((e = cudaMemcpyToSymbol(c_taps_chan, P25_TAPS_CHAN_H, sizeof(c_taps_chan))) != cudaSuccess) return e;
    if ((e = upload_imma(w5i::tables(), w5i::g_btab, w5i::g_init)) != cudaSuccess) return e;
    if ((e = upload_imma(w50i::tables(), w50i::g_btab, w50i::g_init)) != cudaSuccess) return e;
    return cudaMemcpyToSymbol(c_iq_lut, P25_IQ_LUT, sizeof(c_iq_lut));
}

// The generic kernel: one CTA per (stream, segment).  A stream's outputs are split into segments of whole blocks, each
// with its own warm-up block: about 16 CTAs per SM over all streams, but at least 8 blocks per segment.
template <bool FRONT, int FMT>
static cudaError_t launch(const DdcParams& p_in, cudaStream_t st) {
    using C = Cfg<FRONT>;
    DdcParams p = p_in;
    const unsigned iters = (p.n_out + C::MB - 1) / C::MB;
    unsigned want = (unsigned)((size_t)p.plan->n_sm * 16 / p.n_streams);
    const unsigned cap = iters / 8;
    if (want > cap) want = cap;
    if (want < 1) want = 1;
    const unsigned per = (iters + want - 1) / want;
    p.seg_out = (per ? per : 1) * C::MB;
    p.n_seg = p.n_out ? (p.n_out + p.seg_out - 1) / p.seg_out : 1;
    const size_t smem = sizeof(Smem<FRONT>);   // opted in per device by p25cu_ddc_plan_device
    p25_ddc_fm_kernel<FRONT, FMT><<<p.n_streams * p.n_seg, C::NT, smem, st>>>(p);
    return cudaGetLastError();
}

// DC gain of a tap set (double): u8 samples run through the integer kernels in byte units centred on 128,
// x_true = (u - 128 + 0.5) / 127.5 (spec iq_lut), so the half LSB reappears after the filters as 0.5 * (product of gains)
static double tap_gain(const float* h, int n) {
    double g = 0.0;
    for (int k = 0; k < n; k++) g += (double)h[k];
    return g;
}

static cudaError_t launch_fast(const DdcParams& p, cudaStream_t st) {
    const int grid_max = p.plan->grid_ddc50;
    const unsigned bps = (p.n_out + fast::MB - 1) / fast::MB;
    const unsigned long long total = (unsigned long long)p.n_streams * bps;
    const unsigned grid = total < (unsigned long long)grid_max ? (unsigned)total : (unsigned)grid_max;
    // 7/8 of the blocks are split statically, the rest goes out in tickets; the ticket counter only ever grows, every
    // launch consumes n_tickets + grid draws (each CTA stops at its first out-of-range ticket)
    const unsigned n_static = (unsigned)(total / grid * DDC50_STATIC_NUM / DDC50_STATIC_DEN);
    const unsigned long long dyn = total - (unsigned long long)n_static * grid;
    const unsigned n_tickets = (unsigned)((dyn + fast::DYN_CH - 1) / fast::DYN_CH);
    fast::p25_ddc_fm_stream_kernel<<<grid, fast::NT, sizeof(fast::Smem), st>>>(p, bps, n_static, n_tickets, *p.ticket_base, 0.f, 1.f);
    *p.ticket_base += n_tickets + grid;
    return cudaGetLastError();
}

// Launch geometry of a warp kernel: iterations per stream, and a grid of at most grid_max CTAs that gives every warp at
// least ~4 iterations (one warm-up each)
struct WarpGrid {
    unsigned ips, grid;
};
static WarpGrid warp_grid(const DdcParams& p, int nout, int warps, int grid_max) {
    const unsigned ips = (p.n_out + nout - 1) / nout;
    const unsigned long long total = (unsigned long long)p.n_streams * ips;
    unsigned long long want = (total + 3) / 4;
    want = (want + warps - 1) / warps;
    return {ips, want < (unsigned long long)grid_max ? (unsigned)(want ? want : 1) : (unsigned)grid_max};
}

// dc and power scale of an integer kernel: yd is in byte units x 2^scale_log2, so the half LSB of the u8 mapping enters
// the channel filter at that scale
struct ImmaScales {
    float dc, pw_scale;
};
static ImmaScales imma_scales(double gain, int scale_log2) {
    const double sc = (double)(1 << scale_log2);
    return {(float)(0.5 * gain * tap_gain(P25_TAPS_CHAN_H, P25_TAPS_CHAN) * sc), (float)(1.0 / (127.5 * 127.5) / (sc * sc))};
}

static cudaError_t launch_w5(const DdcParams& p, cudaStream_t st) {
    const WarpGrid g = warp_grid(p, w5::NOUT, w5::WARPS, p.plan->grid_w5);
    w5::p25_ddc5_warp_kernel<<<g.grid, 32 * w5::WARPS, w5::SMEM, st>>>(p, g.ips, 0.f, 1.f);
    return cudaGetLastError();
}

static cudaError_t launch_w5i(const DdcParams& p, cudaStream_t st) {
    const WarpGrid g = warp_grid(p, w5i::NOUT, w5i::WARPS, p.plan->grid_w5i);
    const ImmaScales k = imma_scales(w5i::tables().gain, w5i::SCALE_LOG2);
    if (p.power_sum) w5i::p25_ddc5_imma_kernel<true><<<g.grid, 32 * w5i::WARPS, w5i::SMEM, st>>>(p, g.ips, k.dc, k.pw_scale);
    else w5i::p25_ddc5_imma_kernel<false><<<g.grid, 32 * w5i::WARPS, w5i::SMEM, st>>>(p, g.ips, k.dc, k.pw_scale);
    return cudaGetLastError();
}

static cudaError_t launch_w50i(const DdcParams& p, cudaStream_t st) {
    const WarpGrid g = warp_grid(p, w50i::NOUT, w50i::WARPS, p.plan->grid_w50i);
    const ImmaScales k = imma_scales(w50i::tables().gain, w50i::SCALE_LOG2);
    if (p.power_sum) w50i::p25_ddc50_imma_kernel<true><<<g.grid, 32 * w50i::WARPS, w50i::SMEM, st>>>(p, g.ips, k.dc, k.pw_scale);
    else w50i::p25_ddc50_imma_kernel<false><<<g.grid, 32 * w50i::WARPS, w50i::SMEM, st>>>(p, g.ips, k.dc, k.pw_scale);
    return cudaGetLastError();
}

// Per-device setup (called once per device under the library's plan mutex, with that device current): opt every
// kernel into its dynamic shared memory and size the persistent grids from the device's own occupancy.
template <typename K>
static cudaError_t plan_one(K kern, int threads, size_t smem, int n_sm, int* grid) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    int per_sm = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, threads, smem);
    if (e != cudaSuccess) return e;
    *grid = n_sm * (per_sm > 0 ? per_sm : 1);
    return cudaSuccess;
}

cudaError_t p25cu_ddc_plan_device(P25DevPlan* plan) {
    cudaError_t e;
    const int n_sm = plan->n_sm;
    constexpr int U8 = P25CU_FMT_U8_IQ, CF = P25CU_FMT_CF32_IQ;
    if ((e = plan_one(fast::p25_ddc_fm_stream_kernel, fast::NT, sizeof(fast::Smem), n_sm, &plan->grid_ddc50)) != cudaSuccess) return e;
    if ((e = plan_one(w5::p25_ddc5_warp_kernel, 32 * w5::WARPS, w5::SMEM, n_sm, &plan->grid_w5)) != cudaSuccess) return e;
    if ((e = plan_one(w5i::p25_ddc5_imma_kernel<true>, 32 * w5i::WARPS, w5i::SMEM, n_sm, &plan->grid_w5i)) != cudaSuccess) return e;
    if ((e = plan_one(w5i::p25_ddc5_imma_kernel<false>, 32 * w5i::WARPS, w5i::SMEM, n_sm, &plan->grid_w5i)) != cudaSuccess) return e;
    if ((e = plan_one(w50i::p25_ddc50_imma_kernel<true>, 32 * w50i::WARPS, w50i::SMEM, n_sm, &plan->grid_w50i)) != cudaSuccess) return e;
    if ((e = plan_one(w50i::p25_ddc50_imma_kernel<false>, 32 * w50i::WARPS, w50i::SMEM, n_sm, &plan->grid_w50i)) != cudaSuccess) return e;
    // the generic kernels' shared memory (27 - 72 KB) needs the opt-in as well
    if ((e = cudaFuncSetAttribute(p25_ddc_fm_kernel<true, U8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Smem<true>))) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(p25_ddc_fm_kernel<true, CF>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Smem<true>))) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(p25_ddc_fm_kernel<false, U8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Smem<false>))) != cudaSuccess) return e;
    return cudaFuncSetAttribute(p25_ddc_fm_kernel<false, CF>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Smem<false>));
}

cudaError_t p25cu_launch_ddc(const DdcParams& p, int format, int decimation, cudaStream_t st) {
    if (p.n_out == 0 && p.n == 0) return cudaSuccess;
    // warp kernels: aligned rows of any length, any decimator phase, and the whole history inside the stream (no implicit
    // zeros: no u8 byte encodes them)
    const bool warp = p.aligned16 && p.n_out > 0 && p.a0 >= p.ht;
    if (decimation == 5 && warp && p.ht == (unsigned)Cfg<false>::HT)
        return format == P25CU_FMT_CF32_IQ ? launch_w5(p, st) : launch_w5i(p, st);
    if (decimation == 50 && format == P25CU_FMT_CF32_IQ && p.aligned16 && (p.a0 & 1ull) == 0 && p.n_out > 0 &&
        p.ht == (unsigned)Cfg<true>::HT)
        return launch_fast(p, st);
    if (decimation == 50 && format == P25CU_FMT_U8_IQ && warp && p.ht == (unsigned)Cfg<true>::HT) return launch_w50i(p, st);
    if (decimation == 50)
        return format == P25CU_FMT_CF32_IQ ? launch<true, P25CU_FMT_CF32_IQ>(p, st) : launch<true, P25CU_FMT_U8_IQ>(p, st);
    return format == P25CU_FMT_CF32_IQ ? launch<false, P25CU_FMT_CF32_IQ>(p, st) : launch<false, P25CU_FMT_U8_IQ>(p, st);
}
