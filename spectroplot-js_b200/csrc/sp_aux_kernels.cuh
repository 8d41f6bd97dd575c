// sp_aux_kernels.cuh — small non-template kernels (gauges / min-max finalisation, decode tap,
// synthetic capture generator).  Included by sp_engine.cu only.
#pragma once
#include "sp_kernels.cuh"

namespace sp {

// per-frame state for sub-frame mode: ordered-uint encodings of the reference's initial values
__global__ void init_minmax_kernel(unsigned *fmin, unsigned *fmax, long long n)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) { fmin[i] = f2ord(0.0f); fmax[i] = f2ord(-200.0f); }
}

// store into a Uint8ClampedArray (clamp, round half to even, NaN -> 0)
__device__ __forceinline__ unsigned char u8clamped(double v)
{
    if (!(v > 0.0)) return 0;
    if (v >= 255.0) return 255;
    return (unsigned char)__double2int_rn(v);
}

// Decode table of the joint histogram: entry j = (dB bin or -1, colour index), or (-2, 0) when no level maps to j.  It depends only
// on the dB / colour constants of the message, so it is rebuilt (one tiny launch) only when they change; finalize_kernel then
// scatters the joint counters with two atomics per non-empty entry instead of a 32-step bisection each.
__global__ void __launch_bounds__(256) jh_table_kernel(JhConst jc, int cmax, int2 *table)
{
    const int j = blockIdx.x * 256 + threadIdx.x;
    if (j >= JH_BINS) return;
    int bin, g;
    const bool hit = jh_decode(j, jc, cmax, bin, g);
    table[j] = hit ? make_int2(bin, g < 0 ? 0 : g) : make_int2(-2, 0);
}

// gauges (lib/worker.js:128-136), the message-wide min / max (lib/worker.js:124-125) and the two histograms of the reply.
// Every kernel of a render accumulates into engine-owned counters - acc_cb / acc_c (64-bit dB / colour histograms, generic kernel)
// and jh (joint histogram, fused kernels) - which are all zero when a render starts.  Many CTAs of 256 frames each fold the per-frame
// values and scatter jh into acc; the LAST CTA to finish publishes min / max as doubles, copies acc to the reply's histograms and
// zeroes every counter again, so no launch is needed to reset anything before the next render.
// `ordered` says fmin/fmax hold f2ord() encodings (sub-frame mode).  mm = {ordered min, ordered max, done counter}.
// t_end (may be null): the last CTA stores %globaltimer there (the end of the message's device time).
__global__ void __launch_bounds__(256) finalize_kernel(const float *fmin, const float *fmax, const float2 *fmid,
                                                       long long nframes, double range, double gain, int ordered,
                                                       unsigned char *gmin, unsigned char *gmax, unsigned char *gamp,
                                                       unsigned *mm, double *stats /* [2] min, max */,
                                                       unsigned long long *jh, const int2 *jh_table, int cmap_len,
                                                       unsigned long long *acc_cb, unsigned long long *acc_c,
                                                       unsigned long long *cb_hist, unsigned long long *c_hist,
                                                       unsigned long long *t_end)
{
    __shared__ float s_mn[8], s_mx[8];
    __shared__ int s_last;
    // The trigger comes before the wait: the next render may then start on the SMs that the tail of this message's render
    // leaves idle.  That render only reads the capture and constant tables before its own griddep_wait(), which returns once
    // this grid - and so, through the wait below, the render before it - has completed.
    griddep_launch_dependents();
    griddep_wait();
    // joint histogram of the fused kernels -> the reference's two histograms (lib/worker.js:106,113)
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < JH_SIZE; j += gridDim.x * blockDim.x) {
        const unsigned long long c = jh[j];
        if (!c) continue;
        if (j == JH_ZERO) {                          // d0 = -inf pixels were counted in bin 999: they belong to bin 0
            atomicAdd(&acc_cb[0], c);
            atomicAdd(&acc_cb[CB_BINS - 1], 0ull - c);
        } else if (j == JH_BAD) {                    // d0 = +inf / NaN pixels were dropped: they belong to bin 0
            atomicAdd(&acc_cb[0], c);
        } else if (j == JH_NAN) {                    // ~~(0.5 + NaN) == 0 (lib/worker.js:112)
            atomicAdd(&acc_c[0], c);
        } else if (j < JH_BINS) {
            const int2 t = jh_table[j];
            if (t.x >= 0) atomicAdd(&acc_cb[t.x], c);
            if (t.x > -2) atomicAdd(&acc_c[t.y], c);
        }
    }
    float mn = 0.0f, mx = -200.0f;
    const long long x = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (x < nframes) {
        const float a = ordered ? ord2f(reinterpret_cast<const unsigned *>(fmin)[x]) : fmin[x];
        const float b = ordered ? ord2f(reinterpret_cast<const unsigned *>(fmax)[x]) : fmax[x];
        mn = fminf(mn, a); mx = fmaxf(mx, b);
        if (gmin) gmin[x] = u8clamped(__dadd_rn(0.5, __ddiv_rn(__dmul_rn(__dadd_rn(range, (double)a), 256.0), range)));
        if (gmax) gmax[x] = u8clamped(__dadd_rn(0.5, __ddiv_rn(__dmul_rn(__dadd_rn(range, (double)b), 256.0), range)));
        if (gamp) {
            const float2 m = fmid[x];
            const double a2 = __dadd_rn(__dmul_rn((double)m.x, (double)m.x), __dmul_rn((double)m.y, (double)m.y));
            const double amp = __dadd_rn(__dmul_rn(5.0, log10(a2)), gain);                   // :135
            gamp[x] = u8clamped(__dadd_rn(0.5, __ddiv_rn(__dmul_rn(__dadd_rn(range, amp), 256.0), range)));
        }
    }
    for (int off = 16; off > 0; off >>= 1) {
        mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, off));
        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, off));
    }
    if ((threadIdx.x & 31) == 0) { s_mn[threadIdx.x / 32] = mn; s_mx[threadIdx.x / 32] = mx; }
    __syncthreads();                                           // (also: this CTA's scatter atomics have been issued)
    if (threadIdx.x == 0) {
        for (int w = 1; w < (int)(blockDim.x / 32); w++) { mn = fminf(mn, s_mn[w]); mx = fmaxf(mx, s_mx[w]); }
        atomicMin(&mm[0], f2ord(mn));
        atomicMax(&mm[1], f2ord(mx));
        __threadfence();
        s_last = atomicAdd(&mm[2], 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (!s_last) return;
    // last CTA: everything every other CTA added is visible (its fence came before its ticket)
    __threadfence();
    if (threadIdx.x == 0) {
        stats[0] = (double)ord2f(*reinterpret_cast<volatile unsigned *>(&mm[0]));
        stats[1] = (double)ord2f(*reinterpret_cast<volatile unsigned *>(&mm[1]));
        mm[0] = f2ord(0.0f);        // lib/worker.js:35
        mm[1] = f2ord(-200.0f);     // lib/worker.js:36
        mm[2] = 0;
    }
    volatile unsigned long long *vcb = acc_cb, *vc = acc_c;
    for (int i = threadIdx.x; i < CB_BINS; i += blockDim.x) { cb_hist[i] = vcb[i]; vcb[i] = 0; }
    for (int i = threadIdx.x; i < cmap_len; i += blockDim.x) { c_hist[i] = vc[i]; vc[i] = 0; }
    for (int i = threadIdx.x; i < JH_SIZE; i += blockDim.x) jh[i] = 0;
    if (t_end && threadIdx.x == 0) *t_end = globaltimer_ns();
}

// decode tap (sp_decode): same device functions as the fused kernel
__global__ void decode_kernel(const uint8_t *buf, unsigned long long valid_bytes, int fmt, long long first,
                              long long count, float2 *out)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    const long long s = first + i;
    const bool inside = samples_inside(s, 1, sample_width(fmt), valid_bytes);
    out[i] = inside ? decode_fast<FMT_RUNTIME>(buf, s, fmt) : decode_checked(buf, s, fmt, valid_bytes);
}


// ------------------------------------------------------------------ synthetic capture generator
// Same integer arithmetic as oracle/spectro_oracle.c (synth_sample16 / synth_pack): a pure
// function of (seed, sample index, total samples).  lut = 4096-entry int16 sine table.
__device__ __forceinline__ unsigned long long splitmix64(unsigned long long z)
{
    z += 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
__device__ __forceinline__ int sum4x16(unsigned long long r)
{
    return (int)((r & 0xFFFF) + ((r >> 16) & 0xFFFF) + ((r >> 32) & 0xFFFF) + (r >> 48)) - 131070;
}
__device__ __forceinline__ int clamp16(int v) { return v < -32768 ? -32768 : v > 32767 ? 32767 : v; }

__device__ __forceinline__ void synth_sample16(const short *__restrict__ lut, unsigned long long seed,
                                               unsigned long long i, unsigned long long S, int &I, int &Q)
{
    const unsigned ph1 = (unsigned)((i * 512ull) & 4095ull);
    const int c1 = lut[(ph1 + 1024u) & 4095u] >> 1, s1 = lut[ph1] >> 1;
    const unsigned long long f0 = 0ull - (1ull << 62);
    const unsigned long long delta = S ? ((1ull << 63) / S) : 0ull;
    unsigned long long a = i, b = i - 1;
    if (a & 1) b >>= 1; else a >>= 1;
    const unsigned long long ph2 = f0 * i + delta * (a * b);
    const unsigned idx2 = (unsigned)(ph2 >> 52);
    const int c2 = (lut[(idx2 + 1024u) & 4095u] * 3277) >> 15, s2 = (lut[idx2] * 3277) >> 15;
    const int nI = (sum4x16(splitmix64(seed ^ (2 * i))) * 11) >> 12;
    const int nQ = (sum4x16(splitmix64(seed ^ (2 * i + 1))) * 11) >> 12;
    I = clamp16(c1 + c2 + nI);
    Q = clamp16(s1 + s2 + nQ);
}

__global__ void __launch_bounds__(256) synth_kernel(uint8_t *__restrict__ dst, int fmt, unsigned long long first,
                                                    unsigned long long count, unsigned long long total,
                                                    unsigned long long seed, const short *__restrict__ lut_g)
{
    __shared__ short lut[4096];
    for (int j = threadIdx.x; j < 4096; j += blockDim.x) lut[j] = lut_g[j];
    __syncthreads();
    const unsigned long long step = (unsigned long long)gridDim.x * blockDim.x;
    for (unsigned long long k = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; k < count; k += step) {
        int I, Q;
        synth_sample16(lut, seed, first + k, total, I, Q);
        switch (fmt) {
        case CU4: dst[k] = (uint8_t)((((I >> 12) + 8) << 4) | ((Q >> 12) + 8)); break;
        case CS4: dst[k] = (uint8_t)((((I >> 12) & 15) << 4) | ((Q >> 12) & 15)); break;
        case CU8: reinterpret_cast<uchar2 *>(dst)[k] = make_uchar2((uint8_t)((I >> 8) + 128), (uint8_t)((Q >> 8) + 128)); break;
        case CS8: reinterpret_cast<uchar2 *>(dst)[k] = make_uchar2((uint8_t)(I >> 8), (uint8_t)(Q >> 8)); break;
        case CU12: case CS12: {
            const unsigned a = (unsigned)((I >> 4) + (fmt == CU12 ? 2048 : 0)) & 0xFFF;
            const unsigned b = (unsigned)((Q >> 4) + (fmt == CU12 ? 2048 : 0)) & 0xFFF;
            dst[3 * k] = (uint8_t)(a & 0xFF);
            dst[3 * k + 1] = (uint8_t)((a >> 8) | ((b & 0xF) << 4));
            dst[3 * k + 2] = (uint8_t)(b >> 4);
            break;
        }
        case CU16: reinterpret_cast<ushort2 *>(dst)[k] = make_ushort2((unsigned short)(I + 32768), (unsigned short)(Q + 32768)); break;
        case CS16: reinterpret_cast<short2 *>(dst)[k] = make_short2((short)I, (short)Q); break;
        case CU32: reinterpret_cast<uint2 *>(dst)[k] = make_uint2(((unsigned)I << 16) + 0x80000000u, ((unsigned)Q << 16) + 0x80000000u); break;
        case CS32: reinterpret_cast<uint2 *>(dst)[k] = make_uint2((unsigned)I << 16, (unsigned)Q << 16); break;
        case CU64: case CS64: {
            const unsigned long long off = fmt == CU64 ? 0x8000000000000000ull : 0ull;
            reinterpret_cast<ulonglong2 *>(dst)[k] = make_ulonglong2(((unsigned long long)(long long)I << 48) + off,
                                                                    ((unsigned long long)(long long)Q << 48) + off);
            break;
        }
        case CF32: reinterpret_cast<float2 *>(dst)[k] = make_float2((float)I / 32768.0f, (float)Q / 32768.0f); break;
        default: reinterpret_cast<double2 *>(dst)[k] = make_double2((double)I / 32768.0, (double)Q / 32768.0); break;
        }
    }
}

} // namespace sp
