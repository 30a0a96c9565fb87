/*
 * fft32.cuh -- the stages of a 32-point complex FFT held entirely in one thread's registers.
 *
 * Radix-2 decimation in time, forward transform X[k] = sum_n x[n] e^{-2 pi i k n / 32}.
 * Slot i holds x[bitrev5(i)] (a compile-time permutation of registers, free); after the stages
 * of length 2, 4, .., 32 slot i holds X[i].  Built from the packed-complex primitives of cplx2.cuh:
 *   trivial twiddles (1, -j)   46 butterflies x 2 FADD2
 *   general twiddles           34 butterflies x 3 FFMA2   (X = a + W b: 2, Y = 2a - X: 1)
 * = 194 FP32x2 instructions per transform (388 fp32 lane-operations).
 *
 * The 1024-point transform of the spectrum chain is two of these (32 x 32 "four-step"; spectrum.cuh
 * fuses the first stage of each with the window or the twiddles), the planned CMSIS shape being
 * arm_cfft_f32 with arm_cfft_sR_f32_len1024 (reference CMSIS/core/arm_math.h:2149,
 * arm_const_structs.h:55 -- declared, never called).
 */
#ifndef B200_FFT32_CUH
#define B200_FFT32_CUH

#include "cplx2.cuh"

/* e^{-2 pi i k / 32}, k = 0..15 */
#define B200_W32_RE(k)                                                                                           \
    ((k) == 0 ? 1.0f : (k) == 1 ? 0.98078528040323043f : (k) == 2 ? 0.92387953251128674f                          \
     : (k) == 3 ? 0.83146961230254524f : (k) == 4 ? 0.70710678118654757f : (k) == 5 ? 0.55557023301960218f        \
     : (k) == 6 ? 0.38268343236508978f : (k) == 7 ? 0.19509032201612825f : (k) == 8 ? 0.0f                        \
     : (k) == 9 ? -0.19509032201612825f : (k) == 10 ? -0.38268343236508978f : (k) == 11 ? -0.55557023301960218f   \
     : (k) == 12 ? -0.70710678118654757f : (k) == 13 ? -0.83146961230254524f : (k) == 14 ? -0.92387953251128674f  \
                                                                                          : -0.98078528040323043f)
#define B200_W32_IM(k)                                                                                           \
    ((k) == 0 ? 0.0f : (k) == 1 ? -0.19509032201612825f : (k) == 2 ? -0.38268343236508978f                        \
     : (k) == 3 ? -0.55557023301960218f : (k) == 4 ? -0.70710678118654757f : (k) == 5 ? -0.83146961230254524f     \
     : (k) == 6 ? -0.92387953251128674f : (k) == 7 ? -0.98078528040323043f : (k) == 8 ? -1.0f                     \
     : (k) == 9 ? -0.98078528040323043f : (k) == 10 ? -0.92387953251128674f : (k) == 11 ? -0.83146961230254524f   \
     : (k) == 12 ? -0.70710678118654757f : (k) == 13 ? -0.55557023301960218f : (k) == 14 ? -0.38268343236508978f  \
                                                                                          : -0.19509032201612825f)

B200_DEV int b200_bitrev5(int i)
{
    return ((i & 1) << 4) | ((i & 2) << 2) | (i & 4) | ((i & 8) >> 2) | ((i & 16) >> 4);
}

/* one DIT butterfly with twiddle W32^TW (TW is a constant after unrolling) */
template <int TW>
B200_DEV void b200_bf(c2 &a, c2 &b)
{
    if (TW == 0) {
        c2 t = c2_sub(a, b);
        a = c2_add(a, b);
        b = t;
    } else if (TW == 8) { /* W = -j */
        c2 t = c2_add_jb(a, b);
        a = c2_sub_jb(a, b);
        b = t;
    } else {
        c2 x = c2_cfma(b, B200_W32_RE(TW), B200_W32_IM(TW), a);
        b = c2_two_a_minus(a, x);
        a = x;
    }
}

template <int LEN, int K>
struct b200_stage_k {
    B200_DEVM static void run(c2 (&v)[32])
    {
        constexpr int HALF = LEN / 2;
#pragma unroll
        for (int base = 0; base < 32; base += LEN) b200_bf<K *(32 / LEN)>(v[base + K], v[base + K + HALF]);
        b200_stage_k<LEN, K + 1>::run(v);
    }
};
template <int LEN>
struct b200_stage_k<LEN, LEN / 2> {
    B200_DEVM static void run(c2 (&)[32]) {}
};

#endif
