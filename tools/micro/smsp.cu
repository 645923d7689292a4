// Two questions behind shkadov's balanced 6/5-point instance, asked of fp64-bound stand-in bodies at its
// launch shape (256 threads, 2 CTAs per SM, one CTA barrier per iteration):
//   * warp-to-sub-partition map: warps w and w + 4 of a CTA share an SMSP.  If so, making warps 0-3
//     heavy (one heavy + one light warp per SMSP) beats making warps 0, 1, 4, 5 heavy (two heavy warps
//     on SMSPs 0 and 1), because the barrier waits for the most loaded SMSP;
//   * instruction cache: two different unrolled bodies of about 14 KB and 12 KB resident at once
//     cost what the mean of the two single-body runs predicts, or more.
// Body of width W: W independent DFMA chains x DEPTH steps, fully unrolled (W = 6: ~0.9 K SASS
// instructions ~ 14 KB, the C = 6 shkadov body is ~15 KB).
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o tools/micro/smsp tools/micro/smsp.cu
#include <cstdio>
#include <cuda_runtime.h>

constexpr int DEPTH = 150;

template <int W> __device__ __forceinline__ double body(double x, double c0, double c1)
{
    double v[W];
#pragma unroll
    for (int k = 0; k < W; k++) v[k] = x + k;
#pragma unroll
    for (int d = 0; d < DEPTH; d++)
#pragma unroll
        for (int k = 0; k < W; k++) v[k] = fma(v[k], (d & 1) ? c0 : c1, (d & 2) ? c1 : c0);
    double s = 0;
#pragma unroll
    for (int k = 0; k < W; k++) s += v[k];
    return s;
}

// MODE 0: all warps W6.  1: all warps W5.  2: warps 0-3 W6, 4-7 W5 (split).  3: warps 0,1,4,5 W6, the
// others W5 (heavy warps paired on two SMSPs under the w / w+4 assumption).
template <int MODE> __global__ void __launch_bounds__(256, 2) probe(double *out, int iters, double c0, double c1)
{
    const int w = threadIdx.x >> 5;
    bool heavy = MODE == 0 || (MODE == 2 && w < 4) || (MODE == 3 && (w & 2) == 0);
    double x = threadIdx.x * 1e-3;
    for (int i = 0; i < iters; i++) {
        x = heavy ? body<6>(x, c0, c1) : body<5>(x, c0, c1);
        __syncthreads();
    }
    out[blockIdx.x * blockDim.x + threadIdx.x] = x;
}

template <int MODE> float run(double *out, int ctas, int iters)
{
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    probe<MODE><<<ctas, 256>>>(out, iters, 0.999, 1e-3);   // warm-up
    cudaEventRecord(e0);
    for (int r = 0; r < 5; r++) probe<MODE><<<ctas, 256>>>(out, iters, 0.999, 1e-3);
    cudaEventRecord(e1);
    cudaEventSynchronize(e1);
    float ms = 0;
    cudaEventElapsedTime(&ms, e0, e1);
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    return ms / 5;
}

int main()
{
    cudaDeviceProp p;
    cudaGetDeviceProperties(&p, 0);
    const int ctas = 2 * p.multiProcessorCount, iters = 400;
    double *out;
    cudaMalloc(&out, (size_t)ctas * 256 * sizeof(double));
    printf("%s, %d SMs, %d CTAs x 256 threads, %d iterations of one body + barrier\n", p.name, p.multiProcessorCount, ctas, iters);
    for (int rep = 0; rep < 3; rep++) {
        float t0 = run<0>(out, ctas, iters), t1 = run<1>(out, ctas, iters), t2 = run<2>(out, ctas, iters), t3 = run<3>(out, ctas, iters);
        printf("rep %d: all W6 %.3f ms | all W5 %.3f ms | split 0-3 W6 %.3f ms (mean of singles %.3f) | paired 0,1,4,5 W6 %.3f ms\n",
               rep, t0, t1, t2, 0.5f * (t0 + t1), t3);
    }
    cudaError_t err = cudaDeviceSynchronize();
    cudaFree(out);
    if (err != cudaSuccess) { printf("CUDA error %s\n", cudaGetErrorString(err)); return 1; }
    return 0;
}
