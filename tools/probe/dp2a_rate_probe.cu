// Standalone probe: issue rate of IDP.2A (dp2a), IMAD and PRMT on one SM, in warp-instructions per SM per clock.
// The LK Newton row (lk.cu, newton_sums) takes its mismatch products on dp2a: 16 IDP per row in place of 8 IDP + 8 IMAD +
// 8 field extracts.  That only pays if IDP issues at (close to) the rate of the other integer pipes.
// One CTA of 1024 threads per SM; each thread runs 8 independent accumulator chains of one instruction kind, so the issue
// rate and not the latency bounds the loop.  SM clocks are read with clock64() around a __syncthreads()-fenced loop; the
// loop's own counter and branch (3 instructions per 64 measured ones) are not counted.  CUDA events give the wall time.
// nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -o dp2a_rate_probe dp2a_rate_probe.cu
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdint.h>

constexpr int CHAINS = 8, PER_ITER = 64, ITERS = 4096, THREADS = 1024;

enum Kind { DP2A_LO, DP2A_HI, IMAD, PRMT, DP2A_PRMT };

template <int K>
__device__ __forceinline__ uint32_t op(uint32_t acc, uint32_t a, uint32_t b)
{
    uint32_t d;
    if (K == DP2A_LO) asm("dp2a.lo.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(acc));
    else if (K == DP2A_HI) asm("dp2a.hi.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(acc));
    else if (K == IMAD) asm("mad.lo.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(acc));
    else asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(acc), "r"(a), "r"(b));
    return d;
}

template <int K>
__global__ void __launch_bounds__(THREADS, 1) rate(uint32_t seed, uint32_t *sink, long long *cycles)
{
    uint32_t acc[CHAINS];
    const uint32_t a = seed ^ threadIdx.x, b = (seed * 0x9e3779b9u) | 0x5140u;
    for (int c = 0; c < CHAINS; c++) acc[c] = a + c;
    __syncthreads();
    const long long t0 = clock64();
#pragma unroll 1
    for (int i = 0; i < ITERS; i++) {
#pragma unroll
        for (int k = 0; k < PER_ITER / CHAINS; k++)
#pragma unroll
            for (int c = 0; c < CHAINS; c++) {
                if (K == DP2A_PRMT) acc[c] = (c & 1) ? op<PRMT>(acc[c], a, b & 0x7777u) : op<DP2A_LO>(acc[c], a, b);
                else acc[c] = op<K>(acc[c], a, K == PRMT ? (b & 0x7777u) : b);
            }
    }
    __syncthreads();
    const long long t1 = clock64();
    uint32_t r = 0;
    for (int c = 0; c < CHAINS; c++) r ^= acc[c];
    if (r == 0x12345678u) sink[blockIdx.x] = r;          // keeps the chains live
    if (threadIdx.x == 0) cycles[blockIdx.x] = t1 - t0;
}

template <int K>
static void run(const char *name, int nsm, uint32_t *sink, long long *cyc)
{
    rate<K><<<nsm, THREADS>>>(1u, sink, cyc);              // warm-up
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    cudaEventRecord(e0);
    rate<K><<<nsm, THREADS>>>(2u, sink, cyc);
    cudaEventRecord(e1);
    cudaError_t e = cudaEventSynchronize(e1);
    if (e != cudaSuccess) { printf("%-10s %s\n", name, cudaGetErrorString(e)); return; }
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    static long long h[1024];
    cudaMemcpy(h, cyc, nsm * sizeof(long long), cudaMemcpyDeviceToHost);
    long long csum = 0;
    for (int i = 0; i < nsm; i++) csum += h[i];
    const double warp_insts = (double)(THREADS / 32) * ITERS * PER_ITER;     // per SM
    printf("%-10s %6.3f warp-inst / SM / clk (mean over SMs; %.0f cycles)  %8.3f ms  %.1f G warp-inst/s whole GPU\n", name,
           warp_insts / ((double)csum / nsm), (double)csum / nsm, ms, warp_insts * nsm / (ms * 1e6));
    cudaEventDestroy(e0); cudaEventDestroy(e1);
}

int main()
{
    cudaDeviceProp p;
    cudaGetDeviceProperties(&p, 0);
    int clk = 0;
    cudaDeviceGetAttribute(&clk, cudaDevAttrClockRate, 0);
    printf("%s, %d SMs, max SM clock %d MHz; %d warps per SM, %d independent chains per thread\n", p.name,
           p.multiProcessorCount, clk / 1000, THREADS / 32, CHAINS);
    uint32_t *sink; long long *cyc;
    cudaMalloc(&sink, p.multiProcessorCount * sizeof(uint32_t));
    cudaMalloc(&cyc, p.multiProcessorCount * sizeof(long long));
    const int n = p.multiProcessorCount;
    run<DP2A_LO>("dp2a.lo", n, sink, cyc);
    run<DP2A_HI>("dp2a.hi", n, sink, cyc);
    run<IMAD>("imad", n, sink, cyc);
    run<PRMT>("prmt", n, sink, cyc);
    run<DP2A_PRMT>("dp2a+prmt", n, sink, cyc);          // 1:1 mix: ~4 when the two share no pipe, ~2 when they do
    cudaFree(sink); cudaFree(cyc);
    return 0;
}
