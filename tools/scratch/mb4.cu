// prep-chain throughput: cycles per make_record for one warp per SM sub-partition, P independent positions per iteration
#include <cstdio>
#include "../../modulations_b200/csrc/tpf_core.cuh"
using namespace b200dvb::tpf;
template <int P, int MODE>
__global__ void __launch_bounds__(128) prep_probe(int iters, float seed, long long *cyc, float *sink)
{
    float acc = 0.f;
    double y[P][2]; float w[P][2];
    for (int p = 0; p < P; ++p) { y[p][0] = seed + p + threadIdx.x; y[p][1] = seed * 0.5 + p; w[p][0] = seed * 0.25f + p; w[p][1] = seed - p; }
    long long t0 = clock64();
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int p = 0; p < P; ++p) {
            float g[8];
            if (MODE == 0) make_record(y[p][0], y[p][1], w[p][0], w[p][1], g);
            if (MODE == 1) {   // only the 8 f64->f32 conversions + 4 f32->f64
                double a = (double)w[p][0] + y[p][0], b = (double)w[p][1] + y[p][1];
                for (int c = 0; c < 8; ++c) g[c] = d_to_f(a + c * b);
            }
            if (MODE == 2) {   // only fp64 adds (20)
                double a = y[p][0], b = y[p][1];
                for (int c = 0; c < 10; ++c) { a = d_add(a, b); b = d_add(b, a); }
                g[0] = (float)a; for (int c = 1; c < 8; ++c) g[c] = 0.f;
            }
            float s = 0.f;
            for (int c = 0; c < 8; ++c) s += g[c];
            acc += s;
            y[p][0] += s * 1e-3; y[p][1] -= s * 1e-3; w[p][0] += 0.125f; w[p][1] -= 0.25f;
        }
    }
    long long t1 = clock64();
    if (acc == 1234.5f) sink[0] = acc;
    if ((threadIdx.x & 31) == 0) cyc[blockIdx.x * 4 + (threadIdx.x >> 5)] = t1 - t0;
}
template <int P, int MODE> void run(const char *name) {
    long long *d; float *s; cudaMalloc(&d, 8 * 148 * 4); cudaMalloc(&s, 4);
    const int iters = 2000;
    prep_probe<P, MODE><<<148, 128>>>(iters, 1.5f, d, s); prep_probe<P, MODE><<<148, 128>>>(iters, 1.5f, d, s);
    cudaDeviceSynchronize();
    long long h[592]; cudaMemcpy(h, d, sizeof h, cudaMemcpyDeviceToHost);
    double avg = 0; for (int i = 0; i < 592; ++i) avg += h[i]; avg /= 592;
    printf("%-34s P=%d: %.1f cycles per position (1 warp per sub-partition)\n", name, P, avg / iters / P);
}
int main() {
    run<1, 0>("make_record"); run<2, 0>("make_record"); run<4, 0>("make_record");
    run<1, 1>("8 F2F.f32.f64 + adds"); run<4, 1>("8 F2F.f32.f64 + adds");
    run<1, 2>("20 dependent DADD"); run<4, 2>("20 DADD x4 chains");
    return 0;
}
