// sp_device.cuh — device building blocks of the B200 spectrogram engine (sm_100a).
//
//  * sample decoders: bit-exact fp32 versions of SampleView.sampleI/Q
//    (reference lib/samples.js:313-400), i.e. gpu == fround(reference double)
//  * register-resident radix-2/4/8/16 butterflies used by the shared-memory FFT, issued as
//    packed-fp32 instructions (FADD2 / FMUL2 / FFMA2)
//    (replaces the radix-2 transform of reference lib/fft_nayuki.js:54-86)
//  * JS number helpers (`~~v`)
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace sp {

enum Format : int {
    CU4 = 0, CS4, CU8, CS8, CU12, CS12, CU16, CS16, CU32, CS32, CU64, CS64, CF32, CF64, FORMAT_COUNT,
    FMT_RUNTIME = -1   // decode through a runtime switch on the format
};

__host__ __device__ constexpr int sample_width(int f)
{
    return (f == CU4 || f == CS4) ? 1 : (f == CU8 || f == CS8) ? 2 : (f == CU12 || f == CS12) ? 3
         : (f == CU16 || f == CS16) ? 4 : (f == CU32 || f == CS32 || f == CF32) ? 8 : 16;
}
__host__ __device__ constexpr int element_size(int f)
{
    return (f <= CS12) ? 1 : (f == CU16 || f == CS16) ? 2 : (f == CF64) ? 8 : 4;
}

// ------------------------------------------------------------------ JS helpers

// log2 for the dB conversion: one MUFU.LG2 (flush-to-zero variant: a power below 1.2e-38, i.e.
// more than 60 dB below the -120 dBFS floor of the parity contract, reads as 0 -> -inf like an
// exact zero).  Relative error 2^-22: 4e-7 dB.
__device__ __forceinline__ float fast_log2(float x)
{
    float r;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
__device__ __forceinline__ float fmin3(float a, float b, float c) { return fminf(fminf(a, b), c); }
__device__ __forceinline__ float fmax3(float a, float b, float c) { return fmaxf(fmaxf(a, b), c); }

// ------------------------------------------------------------------ conversions (raw code -> fp32)
// Each matches fround() of the reference's double expression for EVERY code (SURVEY A.1;
// the three non-power-of-two biases need a correctly rounded IEEE division).

// Correctly rounded x / D for the three non-power-of-two biases without the IEEE-division subroutine:
// q = x * RN(1/D); r = x - q*D (exact in one FMA); q' = q + r * RN(1/D)  (Markstein).  Verified equal to
// RN(x / D) for EVERY code of the three formats with exact rational arithmetic (and by test_decode_bit_exact).
template <int D> __device__ __forceinline__ float div_exact(float x)
{
    constexpr float r = 1.0f / (float)D;
    const float q = __fmul_rn(x, r);
    return fmaf(fmaf(-q, (float)D, x), r, q);
}
__device__ __forceinline__ float cv_u4(int c) { return div_exact<15>((float)(2 * c - 15)); }          // (c-7.5)*(1/7.5)
__device__ __forceinline__ float cv_s4(int c) { return (float)c * 0.125f; }                           // c*(1/8)
__device__ __forceinline__ float cv_u8(int c) { return div_exact<255>((float)(2 * c - 255)); }        // (c-127.5)*(1/127.5)
__device__ __forceinline__ float cv_s8(int c) { return (float)c * 0.0078125f; }                       // c*(1/128)
__device__ __forceinline__ float cv_u12(int c) { return div_exact<4095>((float)(2 * c - 4095)); }     // (c-2047.5)*(1/2047.5)
__device__ __forceinline__ float cv_s12(int c) { return (float)c * 0.00048828125f; }                  // c*(1/2048)
__device__ __forceinline__ float cv_u16(int c) { return (float)(2 * c - 65535) * 1.52587890625e-05f; }// (c-32767.5)/32768, exact
__device__ __forceinline__ float cv_s16(int c) { return (float)c * 3.0517578125e-05f; }               // c/32768, exact
__device__ __forceinline__ float cv_u32(uint32_t c)
{   // (c - 2147483647.5) / 2^31 : exact 33-bit integer, one rounding
    return __ll2float_rn(2ll * (long long)c - 4294967295ll) * 2.3283064365386963e-10f;
}
__device__ __forceinline__ float cv_s32(uint32_t c) { return __int2float_rn((int)c) * 4.656612873077393e-10f; }
__device__ __forceinline__ float cv_u64(uint32_t lo, uint32_t hi)
{   // hi/2^31 + lo/2^64 - 1   (lib/samples.js:368-369; both quotients exact, two roundings like JS)
    double s = __dadd_rn((double)hi * 4.656612873077393e-10, (double)lo * 5.421010862427522e-20);
    return __double2float_rn(__dadd_rn(s, -1.0));
}
__device__ __forceinline__ float cv_s64(uint32_t lo, uint32_t hi)
{   // (hi>>0)/2^31 + lo/2^64   (lib/samples.js:382)
    return __double2float_rn(__dadd_rn((double)(int)hi * 4.656612873077393e-10, (double)lo * 5.421010862427522e-20));
}

__device__ __forceinline__ int sext(int v, int bits) { return (v << (32 - bits)) >> (32 - bits); }

// ------------------------------------------------------------------ fast (in-range) decode of sample s
// `buf` must be 16-byte aligned at sample 0; returns (I, Q).
template <int FMT>
__device__ __forceinline__ float2 decode_fast(const uint8_t *__restrict__ buf, long long s, int rt_fmt)
{
    if constexpr (FMT == FMT_RUNTIME) {
        switch (rt_fmt) {
        case CU4: return decode_fast<CU4>(buf, s, 0);
        case CS4: return decode_fast<CS4>(buf, s, 0);
        case CU8: return decode_fast<CU8>(buf, s, 0);
        case CS8: return decode_fast<CS8>(buf, s, 0);
        case CU12: return decode_fast<CU12>(buf, s, 0);
        case CS12: return decode_fast<CS12>(buf, s, 0);
        case CU16: return decode_fast<CU16>(buf, s, 0);
        case CS16: return decode_fast<CS16>(buf, s, 0);
        case CU32: return decode_fast<CU32>(buf, s, 0);
        case CS32: return decode_fast<CS32>(buf, s, 0);
        case CU64: return decode_fast<CU64>(buf, s, 0);
        case CS64: return decode_fast<CS64>(buf, s, 0);
        case CF32: return decode_fast<CF32>(buf, s, 0);
        default: return decode_fast<CF64>(buf, s, 0);
        }
    } else if constexpr (FMT == CU4) {
        int b = buf[s];
        return make_float2(cv_u4(b >> 4), cv_u4(b & 15));
    } else if constexpr (FMT == CS4) {
        int b = buf[s];
        return make_float2(cv_s4(sext(b >> 4, 4)), cv_s4(sext(b & 15, 4)));
    } else if constexpr (FMT == CU8) {
        unsigned v = *reinterpret_cast<const unsigned short *>(buf + 2 * s);
        return make_float2(cv_u8(v & 255), cv_u8(v >> 8));
    } else if constexpr (FMT == CS8) {
        unsigned v = *reinterpret_cast<const unsigned short *>(buf + 2 * s);
        return make_float2(cv_s8((int)(signed char)(v & 255)), cv_s8((int)(signed char)(v >> 8)));
    } else if constexpr (FMT == CU12 || FMT == CS12) {
        const uint8_t *p = buf + 3 * s;
        int b0 = p[0], b1 = p[1], b2 = p[2];
        int i = ((b1 & 15) << 8) | b0, q = (b2 << 4) | (b1 >> 4);     // lib/samples.js:340,346
        if constexpr (FMT == CU12) return make_float2(cv_u12(i), cv_u12(q));
        return make_float2(cv_s12(sext(i, 12)), cv_s12(sext(q, 12)));
    } else if constexpr (FMT == CU16) {
        unsigned v = *reinterpret_cast<const unsigned *>(buf + 4 * s);
        return make_float2(cv_u16(v & 0xffff), cv_u16(v >> 16));
    } else if constexpr (FMT == CS16) {
        unsigned v = *reinterpret_cast<const unsigned *>(buf + 4 * s);
        return make_float2(cv_s16((int)(short)(v & 0xffff)), cv_s16((int)v >> 16));
    } else if constexpr (FMT == CU32) {
        uint2 v = *reinterpret_cast<const uint2 *>(buf + 8 * s);
        return make_float2(cv_u32(v.x), cv_u32(v.y));
    } else if constexpr (FMT == CS32) {
        uint2 v = *reinterpret_cast<const uint2 *>(buf + 8 * s);
        return make_float2(cv_s32(v.x), cv_s32(v.y));
    } else if constexpr (FMT == CU64) {
        uint4 v = *reinterpret_cast<const uint4 *>(buf + 16 * s);
        return make_float2(cv_u64(v.x, v.y), cv_u64(v.z, v.w));
    } else if constexpr (FMT == CS64) {
        uint4 v = *reinterpret_cast<const uint4 *>(buf + 16 * s);
        return make_float2(cv_s64(v.x, v.y), cv_s64(v.z, v.w));
    } else if constexpr (FMT == CF32) {
        return *reinterpret_cast<const float2 *>(buf + 8 * s);
    } else {
        double2 v = *reinterpret_cast<const double2 *>(buf + 16 * s);
        return make_float2(__double2float_rn(v.x), __double2float_rn(v.y));
    }
}

// ------------------------------------------------------------------ decode with the scale left out
// For the formats whose scale is a power of two the multiplication by the scale commutes exactly
// with the window product (fl(w * (c * 2^-k)) == fl((w * 2^-k) * c)), so the fused kernels fold it
// into the fp32 window table and decode_raw() returns the integer code as a float.  Bit-exactness
// of the decode itself is what decode_fast() (the sp_decode tap) states and tests.
template <int FMT> __host__ __device__ constexpr float raw_scale()
{
    return FMT == CS4 ? 0.125f : FMT == CS8 ? 0.0078125f : FMT == CS12 ? 0.00048828125f
         : FMT == CS16 ? 3.0517578125e-05f : FMT == CU16 ? 1.52587890625e-05f
         : FMT == CS32 ? 4.656612873077393e-10f : 1.0f;
}
__host__ inline float raw_scale_rt(int fmt)
{
    switch (fmt) {
    case CS4: return raw_scale<CS4>();   case CS8: return raw_scale<CS8>();   case CS12: return raw_scale<CS12>();
    case CS16: return raw_scale<CS16>(); case CU16: return raw_scale<CU16>(); case CS32: return raw_scale<CS32>();
    default: return 1.0f;
    }
}
template <int FMT>
__device__ __forceinline__ float2 decode_raw(const uint8_t *__restrict__ buf, long long s, int rt_fmt)
{
    if constexpr (FMT == CS4) {
        int b = buf[s];
        return make_float2((float)sext(b >> 4, 4), (float)sext(b & 15, 4));
    } else if constexpr (FMT == CS8) {
        unsigned v = *reinterpret_cast<const unsigned short *>(buf + 2 * s);
        return make_float2((float)(int)(signed char)(v & 255), (float)(int)(signed char)(v >> 8));
    } else if constexpr (FMT == CS12) {
        const uint8_t *p = buf + 3 * s;
        int b0 = p[0], b1 = p[1], b2 = p[2];
        return make_float2((float)sext(((b1 & 15) << 8) | b0, 12), (float)sext((b2 << 4) | (b1 >> 4), 12));
    } else if constexpr (FMT == CS16) {
        // int16 -> fp32 without the conversion unit (I2F sits behind the same MIO queue as the shared-memory
        // traffic of the fused kernels): bias both halves to unsigned (one LOP3), drop each into the mantissa of
        // 2^23 (one PRMT each: 0x4B00xxxx = 8388608 + x) and subtract 2^23 + 2^15; every step is exact.
        const unsigned v = *reinterpret_cast<const unsigned *>(buf + 4 * s) ^ 0x80008000u;
        const float lo = __uint_as_float(__byte_perm(v, 0x4B000000u, 0x7610));
        const float hi = __uint_as_float(__byte_perm(v, 0x4B000000u, 0x7632));
        return make_float2(__fadd_rn(lo, -8421376.0f), __fadd_rn(hi, -8421376.0f));
    } else if constexpr (FMT == CU16) {
        unsigned v = *reinterpret_cast<const unsigned *>(buf + 4 * s);
        return make_float2((float)(2 * (int)(v & 0xffff) - 65535), (float)(2 * (int)(v >> 16) - 65535));
    } else if constexpr (FMT == CS32) {
        uint2 v = *reinterpret_cast<const uint2 *>(buf + 8 * s);
        return make_float2(__int2float_rn((int)v.x), __int2float_rn((int)v.y));
    } else {
        return decode_fast<FMT>(buf, s, rt_fmt);          // scale 1: the full decode
    }
}

// ------------------------------------------------------------------ bounds-checked decode
// Reference semantics for reads outside the typed array (`undefined`): NaN for the plain
// formats, 0-bits for the packed nibble / 12-bit formats, and for CS64 a missing high word
// is `undefined >> 0 == 0`.  Slow path: only frames that touch the end of a ragged buffer.
__device__ __forceinline__ uint32_t rd_bytes(const uint8_t *buf, long long off, int nb, unsigned long long valid, bool &ok)
{
    ok = off >= 0 && (unsigned long long)(off + nb) <= valid;
    uint32_t v = 0;
    if (ok) for (int i = 0; i < nb; i++) v |= (uint32_t)buf[off + i] << (8 * i);
    return v;
}

static __device__ __noinline__ float2 decode_checked(const uint8_t *__restrict__ buf, long long s, int fmt,
                                              unsigned long long valid_bytes)
{
    const float qnan = __int_as_float(0x7fc00000);
    // typed-array length in whole elements
    const unsigned long long valid = valid_bytes - valid_bytes % (unsigned)element_size(fmt);
    bool ok0, ok1, ok2, ok3;
    float2 r;
    switch (fmt) {
    case CU4: case CS4: {
        int b = (int)rd_bytes(buf, s, 1, valid, ok0);
        if (fmt == CU4) return make_float2(cv_u4(b >> 4), cv_u4(b & 15));
        return make_float2(cv_s4(sext(b >> 4, 4)), cv_s4(sext(b & 15, 4)));
    }
    case CU12: case CS12: {
        int b0 = (int)rd_bytes(buf, 3 * s, 1, valid, ok0);
        int b1 = (int)rd_bytes(buf, 3 * s + 1, 1, valid, ok1);
        int b2 = (int)rd_bytes(buf, 3 * s + 2, 1, valid, ok2);
        int i = ((b1 & 15) << 8) | b0, q = (b2 << 4) | (b1 >> 4);
        if (fmt == CU12) return make_float2(cv_u12(i), cv_u12(q));
        return make_float2(cv_s12(sext(i, 12)), cv_s12(sext(q, 12)));
    }
    case CU8: case CS8: {
        int a = (int)rd_bytes(buf, 2 * s, 1, valid, ok0), b = (int)rd_bytes(buf, 2 * s + 1, 1, valid, ok1);
        r = (fmt == CU8) ? make_float2(cv_u8(a), cv_u8(b)) : make_float2(cv_s8((signed char)a), cv_s8((signed char)b));
        break;
    }
    case CU16: case CS16: {
        int a = (int)rd_bytes(buf, 4 * s, 2, valid, ok0), b = (int)rd_bytes(buf, 4 * s + 2, 2, valid, ok1);
        r = (fmt == CU16) ? make_float2(cv_u16(a), cv_u16(b)) : make_float2(cv_s16((short)a), cv_s16((short)b));
        break;
    }
    case CU32: case CS32: case CF32: {
        uint32_t a = rd_bytes(buf, 8 * s, 4, valid, ok0), b = rd_bytes(buf, 8 * s + 4, 4, valid, ok1);
        r = (fmt == CU32) ? make_float2(cv_u32(a), cv_u32(b))
          : (fmt == CS32) ? make_float2(cv_s32(a), cv_s32(b))
                          : make_float2(__uint_as_float(a), __uint_as_float(b));
        break;
    }
    case CU64: case CS64: {
        uint32_t l0 = rd_bytes(buf, 16 * s, 4, valid, ok0), h0 = rd_bytes(buf, 16 * s + 4, 4, valid, ok1);
        uint32_t l1 = rd_bytes(buf, 16 * s + 8, 4, valid, ok2), h1 = rd_bytes(buf, 16 * s + 12, 4, valid, ok3);
        if (fmt == CU64) {
            r = make_float2(cv_u64(l0, h0), cv_u64(l1, h1));
            ok0 = ok0 && ok1; ok1 = ok2 && ok3;
        } else {
            r = make_float2(cv_s64(l0, h0), cv_s64(l1, h1));   // missing hi word reads as 0
            ok1 = ok2;
        }
        break;
    }
    default: { // CF64
        uint32_t a0 = rd_bytes(buf, 16 * s, 4, valid, ok0), a1 = rd_bytes(buf, 16 * s + 4, 4, valid, ok2);
        uint32_t b0 = rd_bytes(buf, 16 * s + 8, 4, valid, ok1), b1 = rd_bytes(buf, 16 * s + 12, 4, valid, ok3);
        ok0 = ok0 && ok2; ok1 = ok1 && ok3;
        r = make_float2(__double2float_rn(__hiloint2double((int)a1, (int)a0)),
                        __double2float_rn(__hiloint2double((int)b1, (int)b0)));
        break;
    }
    }
    if (!ok0) r.x = qnan;
    if (!ok1) r.y = qnan;
    return r;
}

// ------------------------------------------------------------------ complex helpers
// A complex value lives in one aligned 64-bit register pair (re = low word, im = high word) and
// all FFT arithmetic is issued as Blackwell packed-fp32 instructions (PTX add/sub/mul/fma .f32x2,
// SASS FADD2 / FMUL2 / FFMA2): one issue slot per complex add, two per complex multiply.  The
// pack / unpack `mov.b64` below never reach SASS: ptxas folds them into the operand modifiers of
// the packed instructions (scalar broadcast `R.F32`, swapped halves `R.F32x2.LO_HI`, per-half
// negation `.NP`), so multiplication by +-j is free and a twiddle needs no duplicated registers.

struct cf { unsigned long long u; };

__device__ __forceinline__ cf cpk(float lo, float hi) { cf r; asm("mov.b64 %0, {%1, %2};" : "=l"(r.u) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ cf cpk(float2 a) { return cpk(a.x, a.y); }
__device__ __forceinline__ float2 cun(cf v) { float2 r; asm("mov.b64 {%0, %1}, %2;" : "=f"(r.x), "=f"(r.y) : "l"(v.u)); return r; }
__device__ __forceinline__ float cre(cf v) { return cun(v).x; }
__device__ __forceinline__ float cim(cf v) { return cun(v).y; }
__device__ __forceinline__ cf cld(const float2 *p) { cf r; r.u = *reinterpret_cast<const unsigned long long *>(p); return r; }
__device__ __forceinline__ void cst(float2 *p, cf v) { *reinterpret_cast<unsigned long long *>(p) = v.u; }

__device__ __forceinline__ cf cadd(cf a, cf b) { cf r; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r.u) : "l"(a.u), "l"(b.u)); return r; }
__device__ __forceinline__ cf csub(cf a, cf b) { cf r; asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r.u) : "l"(a.u), "l"(b.u)); return r; }
__device__ __forceinline__ cf cmul2(cf a, cf b) { cf r; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r.u) : "l"(a.u), "l"(b.u)); return r; }
__device__ __forceinline__ cf cfma2(cf a, cf b, cf c) { cf r; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r.u) : "l"(a.u), "l"(b.u), "l"(c.u)); return r; }
// real scale (window coefficient, 1/sqrt2, ...): FMUL2 with a broadcast scalar
__device__ __forceinline__ cf cscale(cf a, float s) { return cmul2(a, cpk(s, s)); }
// a * (w.x + j w.y): FMUL2 + FFMA2
__device__ __forceinline__ cf cmul(cf a, float2 w)
{
    const float2 f = cun(a);
    return cfma2(cpk(f.y, f.x), cpk(-w.y, w.y), cmul2(a, cpk(w.x, w.x)));
}
// multiply by -j (W4^1 of the forward transform) / by +j: operand swizzles, no instruction
__device__ __forceinline__ cf mul_mj(cf a) { const float2 f = cun(a); return cpk(f.y, -f.x); }
__device__ __forceinline__ cf mul_pj(cf a) { const float2 f = cun(a); return cpk(-f.y, f.x); }

// decode_raw() as a packed complex value.  CS16: both halves take the same constant, so the two subtractions are one FADD2
// (one issue slot per sample less in the fused kernels' load phase; every step is exact as in decode_raw).
template <int FMT> __device__ __forceinline__ cf decode_raw_cf(const uint8_t *__restrict__ buf, long long s, int rt_fmt)
{
    if constexpr (FMT == CS16) {
        const unsigned v = *reinterpret_cast<const unsigned *>(buf + 4 * s) ^ 0x80008000u;
        const cf u = cpk(__uint_as_float(__byte_perm(v, 0x4B000000u, 0x7610)), __uint_as_float(__byte_perm(v, 0x4B000000u, 0x7632)));
        return cadd(u, cpk(-8421376.0f, -8421376.0f));
    } else if constexpr (FMT == CU8 || FMT == CS8) {
        // 8-bit codes without the conversion unit (two I2F per sample are 1/8 cycle of the 16-lane XU pipe, which the
        // log2 of the epilogue also needs): each byte is dropped into the mantissa of 2^23 (one PRMT; CS8 is biased to
        // unsigned first), the bias leaves with one FADD2, and the CU8 scaling (2c - 255) / 255 is the same correctly
        // rounded Markstein division as cv_u8(), issued on both components at once.  Every step is exact or identical
        // to decode_fast<>(): the results are bit-identical (tests: test_decode_bit_exact + the fused-kernel parity).
        unsigned v = *reinterpret_cast<const unsigned short *>(buf + 2 * s);
        if constexpr (FMT == CS8) v ^= 0x8080u;
        const cf u = cpk(__uint_as_float(__byte_perm(v, 0x4B000000u, 0x7650)), __uint_as_float(__byte_perm(v, 0x4B000000u, 0x7651)));
        if constexpr (FMT == CS8) return cadd(u, cpk(-8388736.0f, -8388736.0f));            // c = u - 2^23 - 128 (scale 1/128 folded into the window)
        const cf c = cadd(u, cpk(-8388608.0f, -8388608.0f));                                // c = 0 .. 255
        const cf x = cfma2(c, cpk(2.0f, 2.0f), cpk(-255.0f, -255.0f));                      // 2c - 255, exact
        // x / 255 correctly rounded in two instructions: 1/255 = r_hi + r_lo (both fp32), q = RN(x * r_hi + RN(x * r_lo)).  Verified
        // for all 511 values of x against the double-precision quotient (the residual x * r_lo is ~2^-25 of the result, its own
        // rounding error 2^-49): the same bits as div_exact<255> (Markstein, one instruction more) gives
        constexpr float r_hi = 0.003921568859368563f, r_lo = -2.319175823606301e-10f;
        return cfma2(x, cpk(r_hi, r_hi), cmul2(x, cpk(r_lo, r_lo)));
    } else {
        return cpk(decode_raw<FMT>(buf, s, rt_fmt));
    }
}

#define SP_SQRT1_2 0.70710678118654752440f
#define SP_COS_PI_8 0.92387953251128675613f
#define SP_SIN_PI_8 0.38268343236508977173f

// a * W8^1 = (1 - j)/sqrt2 * a   and   a * W8^3 = -(1 + j)/sqrt2 * a : FADD2 + FMUL2
__device__ __forceinline__ cf mul_w8_1(cf a) { return cscale(cadd(a, mul_mj(a)), SP_SQRT1_2); }
__device__ __forceinline__ cf mul_w8_3(cf a) { return cscale(cadd(a, mul_pj(a)), -SP_SQRT1_2); }

// forward DFT-2 / DFT-4 on registers: y[k] = sum_n x[n] * exp(-2 pi j n k / R)
__device__ __forceinline__ void dft2(cf &a, cf &b)
{
    cf t = a; a = cadd(t, b); b = csub(t, b);
}
__device__ __forceinline__ void dft4(cf &a0, cf &a1, cf &a2, cf &a3)
{
    cf t0 = cadd(a0, a2), t1 = csub(a0, a2), t2 = cadd(a1, a3), t3 = mul_mj(csub(a1, a3));
    a0 = cadd(t0, t2); a2 = csub(t0, t2);
    a1 = cadd(t1, t3); a3 = csub(t1, t3);
}

// in place, natural order in -> natural order out
template <int R> __device__ __forceinline__ void dft(cf (&v)[R]);

template <> __device__ __forceinline__ void dft<1>(cf (&)[1]) {}
template <> __device__ __forceinline__ void dft<2>(cf (&v)[2]) { dft2(v[0], v[1]); }
template <> __device__ __forceinline__ void dft<4>(cf (&v)[4]) { dft4(v[0], v[1], v[2], v[3]); }

template <> __device__ __forceinline__ void dft<8>(cf (&v)[8])
{
    // n = 4*n1 + n0, k = k0 + 2*k1 :  W8^{nk} = W2^{n1 k0} * W8^{n0 k0} * W4^{n0 k1}
#pragma unroll
    for (int n0 = 0; n0 < 4; n0++) dft2(v[n0], v[4 + n0]);       // v[n0] : k0 = 0, v[4+n0] : k0 = 1
    dft4(v[0], v[1], v[2], v[3]);   // k0 = 0 : outputs k = 0,2,4,6
    // k0 = 1 : DFT-4 of (x4, W8^1 x5, -j x6, W8^3 x7) with the 1/sqrt2 of the two odd twiddles folded into the
    // FFMA2 of the last butterfly stage (10 packed instructions instead of 12):
    //   W8^1 x5 = s*c5, c5 = x5 - j x5;   W8^3 x7 = -s*c7, c7 = x7 + j x7
    {
        const cf c5 = cadd(v[5], mul_mj(v[5])), c7 = cadd(v[7], mul_pj(v[7]));
        const cf d = csub(c5, c7), e = cadd(c5, c7);               // (a1 + a3)/s, (a1 - a3)/s
        const cf m6 = mul_mj(v[6]);
        const cf t0 = cadd(v[4], m6), t1 = csub(v[4], m6);
        const float2 ef = cun(e);
        const cf es = cpk(ef.y, ef.x);                             // swapped halves: -j*e = (e.im, -e.re)
        v[4] = cfma2(d, cpk(SP_SQRT1_2, SP_SQRT1_2), t0);          // k1 = 0
        v[6] = cfma2(d, cpk(-SP_SQRT1_2, -SP_SQRT1_2), t0);        // k1 = 2
        v[5] = cfma2(es, cpk(SP_SQRT1_2, -SP_SQRT1_2), t1);        // k1 = 1
        v[7] = cfma2(es, cpk(-SP_SQRT1_2, SP_SQRT1_2), t1);        // k1 = 3
    }
    cf y[8];
#pragma unroll
    for (int k1 = 0; k1 < 4; k1++) { y[2 * k1] = v[k1]; y[2 * k1 + 1] = v[4 + k1]; }
#pragma unroll
    for (int i = 0; i < 8; i++) v[i] = y[i];
}

template <> __device__ __forceinline__ void dft<16>(cf (&v)[16])
{
    // n = 4*n1 + n0, k = k0 + 4*k1 :  W16^{nk} = W4^{n1 k0} * W16^{n0 k0} * W4^{n0 k1}
#pragma unroll
    for (int n0 = 0; n0 < 4; n0++) dft4(v[n0], v[4 + n0], v[8 + n0], v[12 + n0]);   // v[4*k0 + n0]
    // twiddles W16^{n0*k0}
    {
        const float C = SP_COS_PI_8, S = SP_SIN_PI_8;
        v[5] = cmul(v[5], make_float2(C, -S));                                  // k0=1,n0=1 : W16^1
        v[6] = mul_w8_1(v[6]);                                                  // k0=1,n0=2 : W16^2
        v[7] = cmul(v[7], make_float2(S, -C));                                  // k0=1,n0=3 : W16^3
        v[9] = mul_w8_1(v[9]);                                                  // k0=2,n0=1 : W16^2
        v[10] = mul_mj(v[10]);                                                  // k0=2,n0=2 : W16^4
        v[11] = mul_w8_3(v[11]);                                                // k0=2,n0=3 : W16^6
        v[13] = cmul(v[13], make_float2(S, -C));                                // k0=3,n0=1 : W16^3
        v[14] = mul_w8_3(v[14]);                                                // k0=3,n0=2 : W16^6
        v[15] = cmul(v[15], make_float2(-C, S));                                // k0=3,n0=3 : W16^9
    }
#pragma unroll
    for (int k0 = 0; k0 < 4; k0++) dft4(v[4 * k0], v[4 * k0 + 1], v[4 * k0 + 2], v[4 * k0 + 3]);  // -> k1
    cf y[16];
#pragma unroll
    for (int k0 = 0; k0 < 4; k0++)
#pragma unroll
        for (int k1 = 0; k1 < 4; k1++) y[k0 + 4 * k1] = v[4 * k0 + k1];
#pragma unroll
    for (int i = 0; i < 16; i++) v[i] = y[i];
}

// ------------------------------------------------------------------ 64-point DFT in registers
// cos(2 pi q / 64), q = 0..16 (double -> fp32 once); the other 47 come from the symmetries
__host__ __device__ constexpr float cos64_q(int q)
{
    constexpr float C[17] = { 1.0f, 0.99518472667219693f, 0.98078528040323043f, 0.95694033573220882f, 0.92387953251128674f,
                              0.88192126434835505f, 0.83146961230254524f, 0.77301045336273699f, 0.70710678118654757f,
                              0.63439328416364549f, 0.55557023301960229f, 0.47139673682599781f, 0.38268343236508984f,
                              0.29028467725446233f, 0.19509032201612833f, 0.09801714032956077f, 0.0f };
    return C[q];
}
__host__ __device__ constexpr float cos64(int m)
{
    int q = m & 63;
    if (q > 32) q = 64 - q;
    return q > 16 ? -cos64_q(32 - q) : cos64_q(q);
}
__host__ __device__ constexpr float sin64(int m) { return cos64(m + 48); }     // sin(x) = cos(x - pi/2)

// a * W64^M (forward sign: exp(-2 pi j M / 64)), M a compile-time constant
template <int M> __device__ __forceinline__ cf mul_w64(cf a)
{
    constexpr int m = M & 63;
    if constexpr (m == 0) return a;
    else if constexpr (m == 16) return mul_mj(a);
    else if constexpr (m == 32) return cpk(-cre(a), -cim(a));
    else if constexpr (m == 48) return mul_pj(a);
    else return cmul(a, make_float2(cos64(m), -sin64(m)));
}

template <int K0> __device__ __forceinline__ void dft64_twiddle_row(cf (&v)[64])
{
    // element v[8*K0 + n0] holds the k0 = K0 output of column n0: times W64^{n0*K0}
    v[8 * K0 + 1] = mul_w64<1 * K0>(v[8 * K0 + 1]); v[8 * K0 + 2] = mul_w64<2 * K0>(v[8 * K0 + 2]);
    v[8 * K0 + 3] = mul_w64<3 * K0>(v[8 * K0 + 3]); v[8 * K0 + 4] = mul_w64<4 * K0>(v[8 * K0 + 4]);
    v[8 * K0 + 5] = mul_w64<5 * K0>(v[8 * K0 + 5]); v[8 * K0 + 6] = mul_w64<6 * K0>(v[8 * K0 + 6]);
    v[8 * K0 + 7] = mul_w64<7 * K0>(v[8 * K0 + 7]);
}

// n = 8*n1 + n0, k = k0 + 8*k1 :  W64^{nk} = W8^{n1 k0} * W64^{n0 k0} * W8^{n0 k1}; natural order in and out
// between(): called once every input has been consumed (after the eight column transforms) - the fused kernels put the
// barrier that releases the buffer the inputs were loaded from there, so that the loads overlap the column transforms
template <class Between> __device__ __forceinline__ void dft64_between(cf (&v)[64], Between between)
{
#pragma unroll
    for (int n0 = 0; n0 < 8; n0++) {                       // DFT-8 over n1 of column n0; result k0 -> v[8*k0 + n0]
        cf u[8];
#pragma unroll
        for (int n1 = 0; n1 < 8; n1++) u[n1] = v[8 * n1 + n0];
        dft<8>(u);
#pragma unroll
        for (int k0 = 0; k0 < 8; k0++) v[8 * k0 + n0] = u[k0];
    }
    between();
    dft64_twiddle_row<1>(v); dft64_twiddle_row<2>(v); dft64_twiddle_row<3>(v); dft64_twiddle_row<4>(v);
    dft64_twiddle_row<5>(v); dft64_twiddle_row<6>(v); dft64_twiddle_row<7>(v);
    cf y[64];
#pragma unroll
    for (int k0 = 0; k0 < 8; k0++) {                       // DFT-8 over n0 of row k0; result k1 -> bin k0 + 8*k1
        cf u[8];
#pragma unroll
        for (int n0 = 0; n0 < 8; n0++) u[n0] = v[8 * k0 + n0];
        dft<8>(u);
#pragma unroll
        for (int k1 = 0; k1 < 8; k1++) y[k0 + 8 * k1] = u[k1];
    }
#pragma unroll
    for (int i = 0; i < 64; i++) v[i] = y[i];
}
template <> __device__ __forceinline__ void dft<64>(cf (&v)[64]) { dft64_between(v, [] {}); }

// 32-point DFT in registers: n = 8*n1 + n0 (n1 < 4), k = k0 + 4*k1 :  W32^{nk} = W4^{n1 k0} * W32^{n0 k0} * W8^{n0 k1}
template <int K0> __device__ __forceinline__ void dft32_twiddle_row(cf (&v)[32])
{
    // element v[8*K0 + n0] holds the k0 = K0 output of column n0: times W32^{n0*K0} = W64^{2*n0*K0}
    v[8 * K0 + 1] = mul_w64<2 * 1 * K0>(v[8 * K0 + 1]); v[8 * K0 + 2] = mul_w64<2 * 2 * K0>(v[8 * K0 + 2]);
    v[8 * K0 + 3] = mul_w64<2 * 3 * K0>(v[8 * K0 + 3]); v[8 * K0 + 4] = mul_w64<2 * 4 * K0>(v[8 * K0 + 4]);
    v[8 * K0 + 5] = mul_w64<2 * 5 * K0>(v[8 * K0 + 5]); v[8 * K0 + 6] = mul_w64<2 * 6 * K0>(v[8 * K0 + 6]);
    v[8 * K0 + 7] = mul_w64<2 * 7 * K0>(v[8 * K0 + 7]);
}
template <> __device__ __forceinline__ void dft<32>(cf (&v)[32])
{
#pragma unroll
    for (int n0 = 0; n0 < 8; n0++) {                       // DFT-4 over n1 of column n0; result k0 -> v[8*k0 + n0]
        dft4(v[n0], v[8 + n0], v[16 + n0], v[24 + n0]);
    }
    dft32_twiddle_row<1>(v); dft32_twiddle_row<2>(v); dft32_twiddle_row<3>(v);
    cf y[32];
#pragma unroll
    for (int k0 = 0; k0 < 4; k0++) {                       // DFT-8 over n0 of row k0; result k1 -> bin k0 + 4*k1
        cf u[8];
#pragma unroll
        for (int n0 = 0; n0 < 8; n0++) u[n0] = v[8 * k0 + n0];
        dft<8>(u);
#pragma unroll
        for (int k1 = 0; k1 < 8; k1++) y[k0 + 4 * k1] = u[k1];
    }
#pragma unroll
    for (int i = 0; i < 32; i++) v[i] = y[i];
}

} // namespace sp
