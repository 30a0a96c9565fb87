// ubench_fft.cu -- what does the spectrum kernel's OWN instruction stream cost when nothing but the
// FP32 pipe is in the way?  Runs a register FFT-32 of csrc/fft32.cuh's stages (the body of k_spectrum, 194 packed
// ops) in a loop, alone and together with the other per-frame ingredients (u8 conversion PRMTs, the
// transpose through shared memory), at the kernel's occupancy (128-thread CTAs, 2 / 3 / 4 per SM).
// Prints FP32-pipe cycles per FFT-32 per scheduler against the nominal 2 cycles per packed op.
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -o build/ubench_fft tools/ubench_fft.cu
#include <cuda_runtime.h>
#include <cstdio>
#include <cstdint>
#include "../stm32f7-rtlsdr_b200/csrc/cplx2.cuh"
#include "../stm32f7-rtlsdr_b200/csrc/fft32.cuh"

/* in-register FFT: slot i holds x[bitrev5(i)] on entry, X[i] on exit */
__device__ __forceinline__ void b200_fft32(c2 (&v)[32])
{
    b200_stage_k<2, 0>::run(v);
    b200_stage_k<4, 0>::run(v);
    b200_stage_k<8, 0>::run(v);
    b200_stage_k<16, 0>::run(v);
    b200_stage_k<32, 0>::run(v);
}

// MODE 0: FFT-32 only          1: + 32 u16 -> c2 conversions (2 PRMT + FADD2 each)
// MODE 2: + transpose (32 STS.64 + 32 LDS.64, pitch 33)      3: all of it
template <int MODE, int MINB>
__global__ void __launch_bounds__(128, MINB) k_fft(float *out, const uint32_t *words, int iters)
{
    __shared__ c2 tile[4][32 * 33];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    c2 v[32];
    uint32_t w[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) {
        v[i] = c2_make(1e-3f * (float)(threadIdx.x + i), 2e-3f * (float)i);
        w[i] = words[(threadIdx.x + i) & 1023];
    }
    for (int it = 0; it < iters; ++it) {
        if (MODE & 1) {
#pragma unroll
            for (int i = 0; i < 32; ++i) {
                v[i] = c2_add(v[i], c2_from_u8_lo(w[i]));
                w[i] += 0x0101u; /* keep the conversion loop-variant (one IADD per word) */
            }
        }
        b200_fft32(v);
        if (MODE & 2) {
            c2 *S = tile[warp];
#pragma unroll
            for (int i = 0; i < 32; ++i) S[i * 33 + lane] = v[i];
            __syncwarp();
#pragma unroll
            for (int i = 0; i < 32; ++i) v[i] = S[lane * 33 + i];
            __syncwarp();
        }
    }
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 32; ++i) s += c2_re(v[i]) + c2_im(v[i]);
    if (s == 1234.5f) out[0] = s;
}

template <int MODE, int MINB>
float timed(float *out, const uint32_t *words, int iters)
{
    cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
    cudaEventRecord(e0);
    k_fft<MODE, MINB><<<148 * MINB, 128>>>(out, words, iters);
    cudaEventRecord(e1);
    cudaDeviceSynchronize();
    float ms; cudaEventElapsedTime(&ms, e0, e1);
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    return ms;
}

// time = launch + iters * per-iteration: two lengths, take the difference (event timing: clock64 inside
// a CTA would miss CTAs that do not run concurrently)
template <int MODE, int MINB>
void run(const char *name, const uint32_t *words, double mhz)
{
    float *out; cudaMalloc(&out, 4);
    cudaFuncSetAttribute(k_fft<MODE, MINB>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    int resident = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&resident, k_fft<MODE, MINB>, 128, 0);
    timed<MODE, MINB>(out, words, 256);
    float best1 = 1e9f, best2 = 1e9f;
    for (int r = 0; r < 3; ++r) {
        best1 = fminf(best1, timed<MODE, MINB>(out, words, 2048));
        best2 = fminf(best2, timed<MODE, MINB>(out, words, 4096));
    }
    const double cycles = (best2 - best1) * 1e-3 * mhz * 1e6; /* for 2048 iterations of MINB warps per scheduler */
    const double per_fft = cycles / (2048.0 * MINB);
    const double nominal = 388.0 + ((MODE & 1) ? 64.0 : 0.0); /* 194 packed ops (+32 FADD2) x 2 cycles */
    printf("%-40s %d CTA/SM (fit %d)  cycles/FFT-32/scheduler %7.1f  nominal %4.0f -> %5.1f %% of FP32 pipe\n", name, MINB, resident,
           per_fft, nominal, 100.0 * nominal / per_fft);
    cudaFree(out);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) printf("  CUDA error: %s\n", cudaGetErrorString(e));
}

int main()
{
    uint32_t *words; cudaMalloc(&words, 4096); cudaMemset(words, 0x5a, 4096);
    int khz = 0; cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, 0);
    const double mhz = khz / 1000.0; /* the boxes run at their maximum SM clock under load (bench.py samples it) */
    printf("SM clock %.0f MHz\n", mhz);
    run<0, 2>("FFT-32 registers only", words, mhz);
    run<0, 3>("FFT-32 registers only", words, mhz);
    run<0, 4>("FFT-32 registers only", words, mhz);
    run<1, 3>("FFT-32 + 32 u8->c2 conversions", words, mhz);
    run<2, 3>("FFT-32 + transpose (STS.64/LDS.64)", words, mhz);
    run<3, 2>("FFT-32 + conversions + transpose", words, mhz);
    run<3, 3>("FFT-32 + conversions + transpose", words, mhz);
    run<3, 4>("FFT-32 + conversions + transpose", words, mhz);
    cudaFree(words);
    return 0;
}
