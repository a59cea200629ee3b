// Microbenchmark: FP64 issue rates on one SM and over the whole GPU, the compute denominator of the linear right-hand
// side's stage kernel (b2ode_linear.cu).
//   * DMMA.8x8x4 (mma.sync.aligned.m8n8k4.row.col.f64, 512 FLOP per warp instruction): cycles per back-to-back MMA of one
//     warp with a single dependent accumulator chain and with 8 independent chains, and the per-SM rate at 1..16 warps.
//   * DFMA (2 FLOP per thread, 64 per warp instruction): the same, dependent and 8 independent chains.
// One block per SM, every SM busy.  Cycles come from clock64() inside the kernel; the SM clock is derived from the same
// launch's CUDA-event time (cycles / seconds), and FP64 FLOP/s is printed at that clock.
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o dmma_rate dmma_rate.cu && ./dmma_rate
#include <cstdio>
#include <cuda_runtime.h>

#define CK(x)                                                                             \
    do {                                                                                  \
        cudaError_t e_ = (x);                                                             \
        if (e_ != cudaSuccess) {                                                          \
            fprintf(stderr, "%s:%d %s -> %s\n", __FILE__, __LINE__, #x, cudaGetErrorString(e_)); \
            return 1;                                                                     \
        }                                                                                 \
    } while (0)

template <int CHAINS>
__global__ void k_dmma(int iters, double seed, unsigned long long *cycles, double *sink) {
    double c[CHAINS][2];
#pragma unroll
    for (int j = 0; j < CHAINS; ++j) c[j][0] = c[j][1] = 0.0;
    const double a = seed + threadIdx.x * 1e-9, b = 1.0 - seed;
    __syncthreads();
    const long long t0 = clock64();
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int j = 0; j < CHAINS; ++j)
            asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};"
                         : "+d"(c[j][0]), "+d"(c[j][1])
                         : "d"(a), "d"(b));
    }
    __syncthreads();
    const long long t1 = clock64();
    double s = 0.0;
#pragma unroll
    for (int j = 0; j < CHAINS; ++j) s += c[j][0] + c[j][1];
    if (s == 12345.678) sink[threadIdx.x] = s;          // never true; keeps the chains alive
    if (threadIdx.x == 0) cycles[blockIdx.x] = (unsigned long long)(t1 - t0);
}

template <int CHAINS>
__global__ void k_dfma(int iters, double seed, unsigned long long *cycles, double *sink) {
    double c[CHAINS];
#pragma unroll
    for (int j = 0; j < CHAINS; ++j) c[j] = j;
    const double a = 1.0 - seed * 1e-3, b = seed + threadIdx.x * 1e-9;
    __syncthreads();
    const long long t0 = clock64();
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int j = 0; j < CHAINS; ++j) asm volatile("fma.rn.f64 %0, %0, %1, %2;" : "+d"(c[j]) : "d"(a), "d"(b));
    }
    __syncthreads();
    const long long t1 = clock64();
    double s = 0.0;
#pragma unroll
    for (int j = 0; j < CHAINS; ++j) s += c[j];
    if (s == 12345.678) sink[threadIdx.x] = s;
    if (threadIdx.x == 0) cycles[blockIdx.x] = (unsigned long long)(t1 - t0);
}

typedef void (*Kern)(int, double, unsigned long long *, double *);

// returns 0; fills per-SM instructions/cycle (mean over blocks) and the clock in MHz
static int run(Kern k, int warps, int chains, int iters, int nsm, unsigned long long *d_cyc, double *d_sink, double *ipc,
               double *mhz, double *ms_out) {
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0));
    CK(cudaEventCreate(&e1));
    k<<<nsm, warps * 32>>>(iters / 10, 0.5, d_cyc, d_sink);      // warm-up
    CK(cudaGetLastError());
    CK(cudaEventRecord(e0));
    k<<<nsm, warps * 32>>>(iters, 0.5, d_cyc, d_sink);
    CK(cudaEventRecord(e1));
    CK(cudaEventSynchronize(e1));
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    static unsigned long long h[1024];
    CK(cudaMemcpy(h, d_cyc, sizeof(unsigned long long) * nsm, cudaMemcpyDeviceToHost));
    double mean = 0.0, mx = 0.0;
    for (int i = 0; i < nsm; ++i) {
        mean += (double)h[i] / nsm;
        if ((double)h[i] > mx) mx = (double)h[i];
    }
    *ipc = (double)warps * chains * iters / mean;
    *mhz = mx / (ms * 1e-3) / 1e6;
    *ms_out = ms;
    CK(cudaEventDestroy(e0));
    CK(cudaEventDestroy(e1));
    return 0;
}

int main() {
    int dev = 0, nsm = 0;
    CK(cudaGetDevice(&dev));
    CK(cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, dev));
    printf("device %s, %d SMs\n", prop.name, nsm);
    unsigned long long *d_cyc;
    double *d_sink;
    CK(cudaMalloc(&d_cyc, sizeof(unsigned long long) * 1024));
    CK(cudaMalloc(&d_sink, sizeof(double) * 1024));
    const int iters = 20000;
    struct Case {
        const char *name;
        Kern k;
        int chains;
        double flop_per_inst;
    } cases[] = {{"DMMA.8x8x4 dependent  ", k_dmma<1>, 1, 512.0}, {"DMMA.8x8x4 8 chains   ", k_dmma<8>, 8, 512.0},
                 {"DFMA dependent        ", k_dfma<1>, 1, 64.0},   {"DFMA 8 chains         ", k_dfma<8>, 8, 64.0}};
    const int warp_list[] = {1, 2, 4, 8, 12, 16};
    double best_dmma = 0.0, best_dfma = 0.0, clk_at_best = 0.0;
    for (const Case &c : cases) {
        for (int w : warp_list) {
            double ipc = 0, mhz = 0, ms = 0;
            if (run(c.k, w, c.chains, iters, nsm, d_cyc, d_sink, &ipc, &mhz, &ms)) return 1;
            const double flops = ipc * c.flop_per_inst * nsm * mhz * 1e6;
            printf("%s warps/SM %2d: %7.2f cycles per instruction per warp, %6.3f warp-instr/cycle/SM, clock %5.0f MHz, "
                   "%7.2f TFLOP/s fp64 (%.2f ms)\n",
                   c.name, w, (double)w / ipc, ipc, mhz, flops * 1e-12, ms);
            if (c.flop_per_inst == 512.0 && flops > best_dmma) {
                best_dmma = flops;
                clk_at_best = mhz;
            }
            if (c.flop_per_inst == 64.0 && flops > best_dfma) best_dfma = flops;
        }
    }
    printf("RESULT dmma_tflops=%.3f dfma_tflops=%.3f clock_mhz=%.0f sms=%d\n", best_dmma * 1e-12, best_dfma * 1e-12, clk_at_best,
           nsm);
    CK(cudaFree(d_cyc));
    CK(cudaFree(d_sink));
    return 0;
}
