// tpf_step_probe.cu — cycles per trellis step of the thread-per-frame decoder's arithmetic core, scalar against
// packed (add.rn.f32x2 / sub.rn.f32x2), at the decoder's occupancy: one CTA of 4 warps per SM, i.e. ONE warp per
// SM sub-partition, so nothing but the instruction scheduler hides a dependency.
//   1. pass_step (the "in" passes), records from shared memory, lanes 16-31 in the beta lanes' roles;
//   2. ext_step + bwd_step: one out-phase position (forward step with the extrinsic maxima and one backward step),
//      records from shared memory, no other memory traffic;
//   3. the raw rate: 16 independent chains of FADD (scalar) or of add.rn.f32x2 (packed), cycles per warp-instruction.
// The scalar steps are the decoder's core before the packed rewrite, kept here as the yardstick; the packed ones are
// modulations_b200/csrc/tpf_core.cuh itself.  Both run on the same inputs and their results are compared bit for bit.
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 --fmad=false -o tpf_step_probe tools/tpf_step_probe.cu
#include <cstdio>
#include <cstring>
#include "../modulations_b200/csrc/tpf_core.cuh"

using namespace b200dvb::tpf;

namespace scalar {
__device__ __forceinline__ void pass_step(float (&v)[16], const float (&g)[8], bool isb)
{
    float G[8];
    G[0] = g[0]; G[1] = g[1]; G[6] = g[6]; G[7] = g[7];
    G[2] = isb ? g[3] : g[2]; G[3] = isb ? g[2] : g[3];
    G[4] = isb ? g[5] : g[4]; G[5] = isb ? g[4] : g[5];
    float n[16];
#pragma unroll
    for (int t = 0; t < 8; ++t) {
        const int c = cls(t);
        const float A = (t & 4) ? G[2 * c + 1] : G[2 * c];
        const float B = (t & 4) ? G[2 * c] : G[2 * c + 1];
        n[2 * t] = f_max(f_add(v[t], A), f_add(v[8 + t], B));
        n[2 * t + 1] = f_max(f_add(v[t], B), f_add(v[8 + t], A));
    }
    const float z = n[0];
    v[0] = 0.f;
#pragma unroll
    for (int s = 1; s < 16; ++s) v[s] = f_sub(n[s], z);
}
__device__ __forceinline__ void bwd_step(float (&z)[16], const float (&g)[8])
{
    float n[16];
#pragma unroll
    for (int t = 0; t < 8; ++t) {
        const int c = cls(t);
        const float A = (t & 4) ? g[2 * c + 1] : g[2 * c];
        const float B = (t & 4) ? g[2 * c] : g[2 * c + 1];
        n[t] = f_max(f_add(z[2 * t], A), f_add(z[2 * t + 1], B));
        n[8 + t] = f_max(f_add(z[2 * t], B), f_add(z[2 * t + 1], A));
    }
    const float q = n[0];
    z[0] = 0.f;
#pragma unroll
    for (int s = 1; s < 16; ++s) z[s] = f_sub(n[s], q);
}
__device__ __forceinline__ void ext_step(float (&x)[16], const float (&zs)[16], const float (&g)[8], float (&uv)[4])
{
    float n[16];
    float U0 = 0.f, U3 = 0.f, V1 = 0.f, V2 = 0.f;
#pragma unroll
    for (int t = 0; t < 8; ++t) {
        const int c = cls(t);
        const float gp = g[2 * c], gm = g[2 * c + 1];
        const float hp = g[2 * (3 - c)], hm = g[2 * (3 - c) + 1];
        const int t2 = (t >> 2) & 1;
        const int nP0 = 2 * t + t2, nM0 = 2 * t + 1 - t2;
        const float p0 = f_add(x[t], gp), m0 = f_add(x[t], gm);
        const float p1 = f_add(x[8 + t], gp), m1 = f_add(x[8 + t], gm);
        const float ub0 = f_add(p0, zs[nP0]), ub1 = f_add(p1, zs[nM0]);
        const float vb0 = f_add(m0, zs[nM0]), vb1 = f_add(m1, zs[nP0]);
        const float us0 = f_add(f_sub(x[t], hp), zs[nP0]), us1 = f_add(f_sub(x[8 + t], hp), zs[nM0]);
        const float vs0 = f_add(f_sub(x[t], hm), zs[nM0]), vs1 = f_add(f_sub(x[8 + t], hm), zs[nP0]);
        if (t == 0) {
            U0 = f_max(ub0, ub1); U3 = f_max(us0, us1); V1 = f_max(vb0, vb1); V2 = f_max(vs0, vs1);
        } else {
            U0 = f_max(U0, f_max(ub0, ub1)); U3 = f_max(U3, f_max(us0, us1));
            V1 = f_max(V1, f_max(vb0, vb1)); V2 = f_max(V2, f_max(vs0, vs1));
        }
        n[nP0] = f_max(p0, m1);
        n[nM0] = f_max(m0, p1);
    }
    uv[0] = U0; uv[1] = U3; uv[2] = V1; uv[3] = V2;
    const float q = n[0];
    x[0] = 0.f;
#pragma unroll
    for (int s = 1; s < 16; ++s) x[s] = f_sub(n[s], q);
}
}  // namespace scalar

constexpr int kRec = 32;                  // records per warp in shared memory, used cyclically: [k][2][32 lanes] float4
constexpr int kOut = 20;                  // floats written back per thread

__device__ void fill_records(float4 *mine, int lane)
{
    for (int i = lane; i < kRec * 2 * 32; i += 32) {
        const unsigned h = (unsigned)i * 2654435761u;
        const float v = 0.05f * (float)((h >> 20) & 255) - 6.4f;
        mine[i] = make_float4(v, -0.5f * v + 0.3f, 0.25f * v - 1.1f, 2.3f - v);
    }
}

// PACKED = 0: the scalar yardstick, 1: tpf_core.cuh.  MODE = 0: pass_step; 1: ext_step + bwd_step; 2: raw add rate
// (one "step" = 16 adds, one per chain: 16 FADD or 16 FADD2).
template <int PACKED, int MODE>
__global__ void __launch_bounds__(128, 1) step_probe(int steps, long long *cyc, float *out)
{
    extern __shared__ float4 rec[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const bool isb = lane >= 16;
    float4 *mine = rec + (size_t)warp * kRec * 2 * 32;
    fill_records(mine, lane);
    __syncwarp();
    float v[16], z[16], acc[4] = {-1e30f, -1e30f, -1e30f, -1e30f};
#pragma unroll
    for (int s = 0; s < 16; ++s) { v[s] = 0.01f * s * (lane + 1); z[s] = -0.02f * s * (warp + 1); }
    float4 lo = mine[lane], hi = mine[32 + lane];
    const long long t0 = clock64();
#pragma unroll 4
    for (int k = 0; k < steps; ++k) {
        const int kn = (k + 1) & (kRec - 1);
        const float4 nlo = mine[(kn * 2) * 32 + lane], nhi = mine[(kn * 2 + 1) * 32 + lane];
        const float g[8] = {lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w};
        if (MODE == 0) {
            if (PACKED) pass_step(v, g, isb); else scalar::pass_step(v, g, isb);
        } else if (MODE == 2) {
#pragma unroll
            for (int s = 0; s < 16; ++s) {
                if (PACKED) { const f2 r = add2(f2{v[s], z[s]}, f2{g[2 * (s & 3)], g[2 * (s & 3) + 1]}); v[s] = r.lo; z[s] = r.hi; }
                else v[s] = f_add(v[s], g[s & 7]);
            }
        } else {
            float uv[4];
            if (PACKED) { ext_step(v, z, g, uv); bwd_step(z, g); }
            else        { scalar::ext_step(v, z, g, uv); scalar::bwd_step(z, g); }
#pragma unroll
            for (int i = 0; i < 4; ++i) acc[i] = fmaxf(acc[i], uv[i]);
        }
        lo = nlo; hi = nhi;
    }
    const long long t1 = clock64();
    float *o = out + ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * kOut;
#pragma unroll
    for (int s = 0; s < 16; ++s) o[s] = v[s] + (MODE ? z[s] : 0.f);
#pragma unroll
    for (int i = 0; i < 4; ++i) o[16 + i] = MODE ? acc[i] : 0.f;
    if (lane == 0) cyc[blockIdx.x * 4 + warp] = t1 - t0;
}

static int g_sms = 0;
static size_t g_smem = (size_t)4 * kRec * 2 * 32 * sizeof(float4);

template <int PACKED, int MODE>
static double run(int steps, long long *d_cyc, float *d_out, float *h_out, double *clk_mhz)
{
    auto k = step_probe<PACKED, MODE>;
    cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)g_smem);
    k<<<g_sms, 128, g_smem>>>(steps, d_cyc, d_out);                 // warm-up
    cudaEvent_t a, b;
    cudaEventCreate(&a); cudaEventCreate(&b);
    cudaEventRecord(a);
    k<<<g_sms, 128, g_smem>>>(steps, d_cyc, d_out);
    cudaEventRecord(b);
    const cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) { printf("step_probe<%d,%d> failed: %s\n", PACKED, MODE, cudaGetErrorString(e)); return -1.0; }
    float ms = 0.f;
    cudaEventElapsedTime(&ms, a, b);
    const int nw = g_sms * 4;
    long long *h = new long long[nw];
    cudaMemcpy(h, d_cyc, nw * sizeof(long long), cudaMemcpyDeviceToHost);
    double avg = 0.0, mx = 0.0;
    for (int i = 0; i < nw; ++i) { avg += (double)h[i]; mx = h[i] > mx ? (double)h[i] : mx; }
    avg /= nw;
    delete[] h;
    *clk_mhz = mx / (ms * 1e3);                                     // the slowest warp's cycles over the kernel's time
    cudaMemcpy(h_out, d_out, (size_t)g_sms * 128 * kOut * sizeof(float), cudaMemcpyDeviceToHost);
    return avg / steps;
}

int main()
{
    cudaDeviceProp prop;
    cudaGetDeviceProperties(&prop, 0);
    g_sms = prop.multiProcessorCount;
    printf("# tpf_step_probe on %s (sm_%d%d, %d SMs), one CTA of 4 warps per SM\n", prop.name, prop.major, prop.minor, g_sms);
    const int steps = 1 << 16;
    long long *d_cyc;
    float *d_out;
    const size_t nout = (size_t)g_sms * 128 * kOut;
    cudaMalloc(&d_cyc, (size_t)g_sms * 4 * sizeof(long long));
    cudaMalloc(&d_out, nout * sizeof(float));
    float *hs = new float[nout], *hp = new float[nout];
    double clk;
    for (int rep = 0; rep < 2; ++rep) {
        const double s0 = run<0, 0>(steps, d_cyc, d_out, hs, &clk);
        const double p0 = run<1, 0>(steps, d_cyc, d_out, hp, &clk);
        const bool eq0 = memcmp(hs, hp, nout * sizeof(float)) == 0;
        printf("pass_step           scalar %6.1f  packed %6.1f cycles/step  (%.1f %% fewer; SM clock ~%.0f MHz)  results %s\n",
               s0, p0, 100.0 * (s0 - p0) / s0, clk, eq0 ? "bit-identical" : "DIFFER");
        const double s1 = run<0, 1>(steps, d_cyc, d_out, hs, &clk);
        const double p1 = run<1, 1>(steps, d_cyc, d_out, hp, &clk);
        const bool eq1 = memcmp(hs, hp, nout * sizeof(float)) == 0;
        printf("ext_step + bwd_step scalar %6.1f  packed %6.1f cycles/step  (%.1f %% fewer; SM clock ~%.0f MHz)  results %s\n",
               s1, p1, 100.0 * (s1 - p1) / s1, clk, eq1 ? "bit-identical" : "DIFFER");
        const double s2 = run<0, 2>(steps, d_cyc, d_out, hs, &clk) / 16.0;
        const double p2 = run<1, 2>(steps, d_cyc, d_out, hp, &clk) / 16.0;
        printf("raw rate: FADD %.2f cycles per warp-instruction (%.1f lane-ops/clk/SM), FADD2 %.2f (%.1f lane-ops/clk/SM)\n",
               s2, 4 * 32 / s2, p2, 4 * 64 / p2);
    }
    delete[] hs; delete[] hp;
    cudaFree(d_cyc); cudaFree(d_out);
    return 0;
}
