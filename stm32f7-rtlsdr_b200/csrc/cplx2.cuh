/*
 * cplx2.cuh -- packed complex-float arithmetic on Blackwell's FP32x2 pipe.
 *
 * sm_100 adds add/sub/mul/fma.rn.f32x2 (SASS FADD2 / FMUL2 / FFMA2): one instruction, two
 * IEEE fp32 results, operands are 64-bit register pairs.  ptxas folds half-swaps, per-half
 * negation and scalar broadcast into operand modifiers (R.F32x2.LO_HI.NP, R.F32, UR.F32,
 * immediates), so with a complex number held as the pair (re, im):
 *     a + b, a - b, a -+ j b              one FADD2
 *     a * s + c           (s real)        one FFMA2
 *     (j a) * s + c                       one FFMA2
 *     a + W b             (W constant)    two FFMA2        2 a - X: one FFMA2
 * i.e. a radix-2 butterfly is 3 issue slots instead of 6 (general twiddle) or 2 instead of 4
 * (trivial twiddle).  Everything that is not floating point (loads, byte permutes, address
 * arithmetic) then fits in the issue slots the packed math leaves free.
 *
 * Host build (tests/emu only): the same operations in scalar float, for index-logic checks.
 */
#ifndef B200_CPLX2_CUH
#define B200_CPLX2_CUH

#include <stdint.h>

#if defined(__CUDACC__) && !defined(B200_EMULATED)
#define B200_DEV __device__ __forceinline__
#define B200_DEVM __device__ __forceinline__ /* for static member functions */
#else
#define B200_DEV static inline
#define B200_DEVM inline
#endif

#if defined(__CUDA_ARCH__) && !defined(B200_EMULATED)
#define B200_PACKED 1 /* real device code (inline PTX allowed): complex numbers as fp32x2 pairs */
#endif

#ifdef B200_PACKED

struct c2 { unsigned long long v; };

B200_DEV c2 c2_make(float re, float im)
{
    c2 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r.v) : "f"(re), "f"(im));
    return r;
}
B200_DEV float c2_re(c2 a) { float x, y; asm("mov.b64 {%0, %1}, %2;" : "=f"(x), "=f"(y) : "l"(a.v)); (void)y; return x; }
B200_DEV float c2_im(c2 a) { float x, y; asm("mov.b64 {%0, %1}, %2;" : "=f"(x), "=f"(y) : "l"(a.v)); (void)x; return y; }
B200_DEV void c2_get(c2 a, float &re, float &im) { asm("mov.b64 {%0, %1}, %2;" : "=f"(re), "=f"(im) : "l"(a.v)); }
B200_DEV c2 c2_add(c2 a, c2 b) { c2 r; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r.v) : "l"(a.v), "l"(b.v)); return r; }
B200_DEV c2 c2_sub(c2 a, c2 b) { c2 r; asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r.v) : "l"(a.v), "l"(b.v)); return r; }
B200_DEV c2 c2_mul2(c2 a, c2 b) { c2 r; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r.v) : "l"(a.v), "l"(b.v)); return r; }
B200_DEV c2 c2_fma2(c2 a, c2 b, c2 c)
{
    c2 r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r.v) : "l"(a.v), "l"(b.v), "l"(c.v));
    return r;
}

#else /* scalar fallback: host emulation only */

struct c2 { float re, im; };
B200_DEV c2 c2_make(float re, float im) { c2 r; r.re = re; r.im = im; return r; }
B200_DEV float c2_re(c2 a) { return a.re; }
B200_DEV float c2_im(c2 a) { return a.im; }
B200_DEV void c2_get(c2 a, float &re, float &im) { re = a.re; im = a.im; }
B200_DEV c2 c2_add(c2 a, c2 b) { return c2_make(a.re + b.re, a.im + b.im); }
B200_DEV c2 c2_sub(c2 a, c2 b) { return c2_make(a.re - b.re, a.im - b.im); }
B200_DEV c2 c2_mul2(c2 a, c2 b) { return c2_make(a.re * b.re, a.im * b.im); }
B200_DEV c2 c2_fma2(c2 a, c2 b, c2 c) { return c2_make(a.re * b.re + c.re, a.im * b.im + c.im); }

#endif

/* ---- derived operations (the compiler folds the swaps / signs into operand modifiers) ---- */
B200_DEV c2 c2_zero() { return c2_make(0.0f, 0.0f); }
B200_DEV c2 c2_neg(c2 a) { float x, y; c2_get(a, x, y); return c2_make(-x, -y); }
B200_DEV c2 c2_swap(c2 a) { float x, y; c2_get(a, x, y); return c2_make(y, x); }
/* j a = (-im, re) */
B200_DEV c2 c2_mulj(c2 a) { float x, y; c2_get(a, x, y); return c2_make(-y, x); }
/* a + j b, a - j b */
B200_DEV c2 c2_add_jb(c2 a, c2 b) { return c2_add(a, c2_mulj(b)); }
B200_DEV c2 c2_sub_jb(c2 a, c2 b) { return c2_sub(a, c2_mulj(b)); }
/* a * s, a * s + c with real scalar s */
B200_DEV c2 c2_scale(c2 a, float s) { return c2_mul2(a, c2_make(s, s)); }
B200_DEV c2 c2_fma_s(c2 a, float s, c2 c) { return c2_fma2(a, c2_make(s, s), c); }
/* (j a) * s + c */
/* written as (swap + per-half negate on the DATA operand) x broadcast scalar: that is the form
 * ptxas folds into `-R.F32x2.LO_HI.NP, Rs.F32` with no extra instruction */
B200_DEV c2 c2_fma_js(c2 a, float s, c2 c) { return c2_fma2(c2_mulj(a), c2_make(s, s), c); }
/* a * (wr + j wi) */
B200_DEV c2 c2_cmul(c2 a, float wr, float wi) { return c2_fma_js(a, wi, c2_scale(a, wr)); }
/* c + a * (wr + j wi) */
B200_DEV c2 c2_cfma(c2 a, float wr, float wi, c2 c) { return c2_fma_js(a, wi, c2_fma_s(a, wr, c)); }
/* 2 a - x */
B200_DEV c2 c2_two_a_minus(c2 a, c2 x) { return c2_fma2(a, c2_make(2.0f, 2.0f), c2_neg(x)); }
/* |a|^2 + acc */
B200_DEV float c2_norm_acc(c2 a, float acc)
{
    float x, y;
    c2_get(a, x, y);
    return fmaf(x, x, fmaf(y, y, acc));
}

/* ---- u8 I/Q -> exact float (u - 127.5) without an integer->float conversion.
 *
 * Form A (the spectrum kernel and the cf32 conversion): PRMT drops the byte into mantissa bits [15:8] of 2^15
 * and 0x80 into bits [7:0]: 0x47000080 | (u << 8) is the float 32768.5 + u exactly (ulp of bit 8 at 2^15 is 1),
 * and one FADD of -32896 leaves u - 127.5 exactly.  (The textbook 2^23 + u form cannot subtract
 * 8388735.5 -- it is not representable.)  Per complex sample: 2 PRMT (half rate) + 1 FADD2.
 * `word` holds 4 bytes = 2 complex samples. */
#define B200_U8_MAGIC 0x47000080u
#define B200_U8_BIAS  (-32896.0f)
B200_DEV float b200_u8_to_f32(uint32_t word, int byte_idx) /* byte_idx compile-time 0..3 */
{
    uint32_t sel = 0x7504u | ((uint32_t)byte_idx << 4);
    return __uint_as_float(__byte_perm(word, B200_U8_MAGIC, sel)) + B200_U8_BIAS;
}
B200_DEV c2 c2_from_u8_lo(uint32_t word) /* bytes 0 (I) and 1 (Q) */
{
    float i = __uint_as_float(__byte_perm(word, B200_U8_MAGIC, 0x7504));
    float q = __uint_as_float(__byte_perm(word, B200_U8_MAGIC, 0x7514));
    return c2_add(c2_make(i, q), c2_make(B200_U8_BIAS, B200_U8_BIAS));
}

/* Form C (the FIR kernels): NO conversion arithmetic.  PRMT drops the byte into bits
 * [23:16] of an otherwise zero word.  Read as a float that is u * 2^-133 EXACTLY for every u in 0..255:
 * u < 128 is the subnormal (u << 16) * 2^-149, u >= 128 has exponent field 1 and is
 * 2^-126 (1 + (u - 128) / 128) -- the subnormal / normal boundary is seamless, and FFMA2 (no .ftz)
 * takes subnormal operands at full rate.  The FIR taps carry the factor 2^133 (they are ~1e-3 / 127.5, so
 * tap * 2^133 < 1e37 is representable), the products are u * h exactly as before, and the -127.5 offset
 * becomes one constant per OUTPUT instead of one add per INPUT sample: an accumulator is started at
 * -127.5 * sum(h) instead of 0 (wbfm.cuh / am.cuh).  The FP32 pipe, which bounds those kernels, then sees
 * only the FIR's own FMAs; the two PRMTs run on the integer pipe. */
#define B200_U8RAW_LOG2 133
B200_DEV c2 c2_u8raw_lo(uint32_t word) /* bytes 0 (I) and 1 (Q) -> (I, Q) * 2^-133 */
{
    return c2_make(__uint_as_float(__byte_perm(word, 0u, 0x4044)), __uint_as_float(__byte_perm(word, 0u, 0x4144)));
}
B200_DEV c2 c2_u8raw_hi(uint32_t word) /* bytes 2 (I) and 3 (Q) */
{
    return c2_make(__uint_as_float(__byte_perm(word, 0u, 0x4244)), __uint_as_float(__byte_perm(word, 0u, 0x4344)));
}

#endif /* B200_CPLX2_CUH */
