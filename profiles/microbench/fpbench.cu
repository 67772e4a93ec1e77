// Micro-benchmarks of the Fp primitives (cycles per operation at 1 / 2 / 4 warps per SM sub-partition).
// Not part of the product library; built and run by profiles/microbench/run.sh under gpurun.
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include "../../milagro_bls_b200/csrc/kernels.cuh"

template <int V>
__global__ void __launch_bounds__(128) k_bench(uint32_t* out, int iters, uint32_t seed, long long* cyc) {
    fp x, y, z, w;
#pragma unroll
    for (int i = 0; i < 12; i++) {
        x.l[i] = seed * (i + 1) + threadIdx.x;
        y.l[i] = seed * (i + 7) ^ threadIdx.x;
        z.l[i] = seed * (i + 3) + 5 * threadIdx.x;
        w.l[i] = seed * (i + 11) ^ (3 * threadIdx.x);
    }
    x.l[11] &= 0x0fffffff; y.l[11] &= 0x0fffffff; z.l[11] &= 0x0fffffff; w.l[11] &= 0x0fffffff;
    long long t0 = clock64();
    for (int it = 0; it < iters; it++) {
        if (V == 0) { x = fp_mul_v(x, y); }
        if (V == 1) { x = fp_mul_v(x, x); }
        if (V == 2) { x = fp_mul2_v(x, y, z, w); }
        if (V == 3) { fp_mul_inl(x, x, y); }
        if (V == 4) { fp_mul_inl(x, x, y); fp_mul_inl(z, z, w); }
        if (V == 5) { fp_add(x, x, y); }
        if (V == 6) { fp_sub(x, x, y); }
        if (V == 7) { fp2h a, b; a.v = x; b.v = y; a = fp2h_mul_v(a, b); x = a.v; }
        if (V == 8) { fp2h a; a.v = x; a = fp2h_sqr_v(a); x = a.v; }
        if (V == 9) { fp t; pair_xchg(t, x); fp_add(x, t, y); }
        if (V == 10) { fp2 a, b; a.c0 = x; a.c1 = z; b.c0 = y; b.c1 = w; a = fp2_mul_v(a, b); x = a.c0; z = a.c1; }
        if (V == 11) { fp2 a; a.c0 = x; a.c1 = z; a = fp2_sqr_v(a); x = a.c0; z = a.c1; }
        if (V == 12) { x = fp_sqr_v(x); }
        if (V == 13) { g2h_jac P; P.x.v = x; P.y.v = y; P.z.v = z; pt_dbl(P, P); x = P.x.v; y = P.y.v; z = P.z.v; }
    }
    long long t1 = clock64();
    uint32_t r = 0;
#pragma unroll
    for (int i = 0; i < 12; i++) r ^= x.l[i] ^ z.l[i];
    out[blockIdx.x * blockDim.x + threadIdx.x] = r;
    if (threadIdx.x == 0 && blockIdx.x == 0) *cyc = t1 - t0;
}

template <int V>
static void run(const char* name, int iters, double macs_per_iter) {
    uint32_t* out;
    long long* cyc;
    cudaMalloc(&out, 148 * 16 * 128 * 4);
    cudaMalloc(&cyc, 8);
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    for (int mult = 1; mult <= 4; mult *= 2) {
        k_bench<V><<<148 * mult, 128>>>(out, iters, 12345u, cyc);
        cudaDeviceSynchronize();
        cudaEventRecord(e0);
        k_bench<V><<<148 * mult, 128>>>(out, iters, 777u, cyc);
        cudaEventRecord(e1);
        cudaDeviceSynchronize();
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        long long c = 0;
        cudaMemcpy(&c, cyc, 8, cudaMemcpyDeviceToHost);
        double per_it = (double)c / iters;
        double mac_rate = macs_per_iter * iters * 148.0 * mult * 128 / (ms * 1e-3);
        printf("%-28s warps/SMSP=%d  cycles/iter=%8.1f  ms=%7.3f  GMAC/s=%8.1f  err=%s\n", name, mult, per_it, ms, mac_rate / 1e9,
               cudaGetErrorString(cudaGetLastError()));
    }
    cudaFree(out); cudaFree(cyc);
}

int main() {
    const int N = 2000;
    run<0>("fp_mul_v x=x*y", N, 300);
    run<1>("fp_mul_v x=x*x", N, 300);
    run<2>("fp_mul2_v", N, 444);
    run<3>("fp_mul_inl", N, 300);
    run<4>("2x fp_mul_inl independent", N, 600);
    run<5>("fp_add", N, 0);
    run<6>("fp_sub", N, 0);
    run<7>("fp2h_mul_v (lane pair)", N, 444);
    run<8>("fp2h_sqr_v (lane pair)", N, 300);
    run<9>("pair_xchg + fp_add", N, 0);
    run<10>("fp2_mul_v (1 thread)", N, 888);
    run<11>("fp2_sqr_v (1 thread)", N, 600);
    run<12>("fp_sqr_v (dedicated, 234 MACs)", N, 234);
    run<13>("pt_dbl<fp2h> (lane pair)", N / 8, 0);
    return 0;
}
