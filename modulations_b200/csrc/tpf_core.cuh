// tpf_core.cuh — arithmetic core of the thread-per-frame ("TPF") max-log-MAP decoder.
//
// One thread holds all 16 state metrics of one frame and one direction in registers:
// no shuffles, no shared-memory exchange, every step is straight-line FADD2/FMNMX code (two adds per FADD2).
// These functions are __host__ __device__ so that tools/tpf_emulator.cu can replay the
// kernel's schedule on the CPU against the oracle before any GPU time is spent.
//
// Reference arithmetic (dvb_rcs2_turbo.py:116-281): branch metrics are float64 sums
// rounded once to float32 (:131-160); recursions, normalisation by state 0 and the APP
// metrics are float32 (:162-248); the extrinsic is float64 (:250-279).
//
// Trellis facts used (dvb_rcs2_turbo.py:327-396; state s = (s3 s2 s1 s0) = (x, t2 t1 t0)):
//   * ns = 2*(s & 7) + dk: the predecessors of (t, d) are (0, t) and (1, t) — a butterfly.
//   * inputs {00, 11} from s share the next state (dk = s2 ^ s3) and the parity class
//     c(s) = (s0^s1^s2, s1); inputs {01, 10} go to the other next state with class ~c.
//     Rounding is monotone, so max(fl(a+g1), fl(a+g2)) == fl(a + max(g1, g2)): per step only
//     the 8 merged metrics GP[c] = max(P[c], -P[~c]), GM[c] = max(M[~c], -M[c]) are needed
//     (P / M = rounded sums that start from a+b / a-b); the smaller member of a pair is
//     -GP[~c] / -GM[~c], and which member is input 00 (01) is the sign of a+b (a-b).
//   * the backward recursion under bit-reversed state labels has the same register wiring
//     as the forward one; only the GP/GM roles of the classes 1 and 2 swap.  A warp can
//     therefore run alpha lanes and beta lanes through ONE instruction stream.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define TPF_HD __host__ __device__ __forceinline__
#else
#define TPF_HD inline
#endif

namespace b200dvb {
namespace tpf {

TPF_HD float f_add(float a, float b)
{
#ifdef __CUDA_ARCH__
    return __fadd_rn(a, b);
#else
    return a + b;
#endif
}
TPF_HD float f_sub(float a, float b)
{
#ifdef __CUDA_ARCH__
    return __fsub_rn(a, b);
#else
    return a - b;
#endif
}
TPF_HD float f_max(float a, float b)
{
#ifdef __CUDA_ARCH__
    return fmaxf(a, b);
#else
    return a > b ? a : b;
#endif
}
TPF_HD double d_add(double a, double b)
{
#ifdef __CUDA_ARCH__
    return __dadd_rn(a, b);
#else
    return a + b;
#endif
}
TPF_HD double d_sub(double a, double b)
{
#ifdef __CUDA_ARCH__
    return __dsub_rn(a, b);
#else
    return a - b;
#endif
}
TPF_HD double d_mul(double a, double b)
{
#ifdef __CUDA_ARCH__
    return __dmul_rn(a, b);
#else
    return a * b;
#endif
}
TPF_HD float d_to_f(double a)
{
#ifdef __CUDA_ARCH__
    return __double2float_rn(a);
#else
    return (float)a;
#endif
}

// Two float32 lanes added with ONE instruction: add.rn.f32x2 / sub.rn.f32x2 (SASS FADD2, sm_100) round each
// lane exactly like __fadd_rn / __fsub_rn (round to nearest, no flush to zero), so packing two independent adds
// changes no bit — it halves the issue slots they take.  The host version is the two scalar operations.
// FADD2 reads a register pair straight, swapped (.LO_HI) or one register broadcast to both lanes, so the swapped
// record pairs and the (z, z) pairs below cost no instruction; only the pairing of the state vector matters.
struct f2 { float lo, hi; };
TPF_HD f2 add2(f2 a, f2 b)
{
#ifdef __CUDA_ARCH__
    f2 r;
    asm("{\n\t.reg .b64 a, b, d;\n\tmov.b64 a, {%2, %3};\n\tmov.b64 b, {%4, %5};\n\t"
        "add.rn.f32x2 d, a, b;\n\tmov.b64 {%0, %1}, d;\n\t}"
        : "=f"(r.lo), "=f"(r.hi) : "f"(a.lo), "f"(a.hi), "f"(b.lo), "f"(b.hi));
    return r;
#else
    return f2{f_add(a.lo, b.lo), f_add(a.hi, b.hi)};
#endif
}
TPF_HD f2 sub2(f2 a, f2 b)
{
#ifdef __CUDA_ARCH__
    f2 r;
    asm("{\n\t.reg .b64 a, b, d;\n\tmov.b64 a, {%2, %3};\n\tmov.b64 b, {%4, %5};\n\t"
        "sub.rn.f32x2 d, a, b;\n\tmov.b64 {%0, %1}, d;\n\t}"
        : "=f"(r.lo), "=f"(r.hi) : "f"(a.lo), "f"(a.hi), "f"(b.lo), "f"(b.hi));
    return r;
#else
    return f2{f_sub(a.lo, b.lo), f_sub(a.hi, b.hi)};
#endif
}

// parity class of the butterfly t = s & 7: c = 2*(s0^s1^s2) + s1
TPF_HD constexpr int cls(int t) { return 2 * ((t ^ (t >> 1) ^ (t >> 2)) & 1) + ((t >> 1) & 1); }
// 4-bit reversal: natural state index <-> label used by the beta lanes during the passes
TPF_HD constexpr int rho4(int r) { return ((r & 1) << 3) | ((r & 2) << 1) | ((r & 4) >> 1) | ((r & 8) >> 3); }

// Branch-metric record of one trellis step: g[2c] = GP[c], g[2c+1] = GM[c]
// (dvb_rcs2_turbo.py:131-160: float64 left-to-right sums, rounded once to float32).
TPF_HD void make_record(double YA, double YB, float pW, float pY, float (&g)[8])
{
    const double a = d_mul(YA, 0.5), b = d_mul(YB, 0.5);
    const double w = d_mul((double)pW, 0.5), y = d_mul((double)pY, 0.5);
    const double s = d_add(a, b), d = d_sub(a, b);
    float P[4], Mv[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        const double sw = (c & 2) ? -w : w, sy = (c & 1) ? -y : y;
        P[c] = d_to_f(d_add(d_add(s, sw), sy));
        Mv[c] = d_to_f(d_add(d_add(d, sw), sy));
    }
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        g[2 * c] = f_max(P[c], -P[3 - c]);
        g[2 * c + 1] = f_max(Mv[3 - c], -Mv[c]);
    }
}

// One step of the two "in" passes (dvb_rcs2_turbo.py:167-179 forward, :203-213 backward)
// in the shared wiring out[2t+o] = max_i(in[8i+t] + role(i^o)):
//   alpha lanes (isb = false): v = alpha[k] in natural labels  -> alpha[k+1]
//   beta lanes  (isb = true):  v = beta[k+1] in rho4 labels     -> beta[k]
// followed by the normalisation by state 0 (:178-179, :212-213; rho4(0) == 0).
// Packed form: the butterfly's two states are one pair (v[t], v[8+t]), added to the record pair (A, B) and to
// (B, A); R[c] = (G[2c], G[2c+1]) and its swap S[c] provide both.  Every lane operation is the scalar one.
TPF_HD void pass_step(float (&v)[16], const float (&g)[8], bool isb)
{
    f2 R[4], S[4];
    R[0] = f2{g[0], g[1]}; R[3] = f2{g[6], g[7]};
    R[1] = f2{isb ? g[3] : g[2], isb ? g[2] : g[3]};
    R[2] = f2{isb ? g[5] : g[4], isb ? g[4] : g[5]};
#pragma unroll
    for (int c = 0; c < 4; ++c) S[c] = f2{R[c].hi, R[c].lo};
    float n[16];
#pragma unroll
    for (int t = 0; t < 8; ++t) {
        const int c = cls(t);
        const f2 x = f2{v[t], v[8 + t]};
        const f2 e = add2(x, (t & 4) ? S[c] : R[c]);   // (v[t] + A, v[8+t] + B)
        const f2 o = add2(x, (t & 4) ? R[c] : S[c]);   // (v[t] + B, v[8+t] + A)
        n[2 * t] = f_max(e.lo, e.hi);
        n[2 * t + 1] = f_max(o.lo, o.hi);
    }
    const float z = n[0];
    v[0] = 0.f;                                       // fl(z - z): metrics are finite (the reference clips its inputs)
    v[8] = f_sub(n[8], z);
#pragma unroll
    for (int t = 1; t < 8; ++t) {
        const f2 d = sub2(f2{n[t], n[8 + t]}, f2{z, z});
        v[t] = d.lo; v[8 + t] = d.hi;
    }
}

// Backward step in natural labels: z = beta[k+1] -> beta[k] (dvb_rcs2_turbo.py:203-213).
// The butterfly's states are the pair (z[2t], z[2t+1]).
TPF_HD void bwd_step(float (&z)[16], const float (&g)[8])
{
    f2 R[4], S[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) { R[c] = f2{g[2 * c], g[2 * c + 1]}; S[c] = f2{g[2 * c + 1], g[2 * c]}; }
    float n[16];
#pragma unroll
    for (int t = 0; t < 8; ++t) {
        const int c = cls(t);
        const f2 x = f2{z[2 * t], z[2 * t + 1]};
        const f2 e = add2(x, (t & 4) ? S[c] : R[c]);   // (z[2t] + A, z[2t+1] + B)
        const f2 o = add2(x, (t & 4) ? R[c] : S[c]);   // (z[2t] + B, z[2t+1] + A)
        n[t] = f_max(e.lo, e.hi);
        n[8 + t] = f_max(o.lo, o.hi);
    }
    const float q = n[0];
    z[0] = 0.f;
    z[1] = f_sub(n[1], q);
#pragma unroll
    for (int t = 1; t < 8; ++t) {
        const f2 d = sub2(f2{n[2 * t], n[2 * t + 1]}, f2{q, q});
        z[2 * t] = d.lo; z[2 * t + 1] = d.hi;
    }
}

// Extrinsic maxima for step k (dvb_rcs2_turbo.py:239-248) fused with the forward step:
// x = alpha[k] -> alpha[k+1]; zs = beta[k+1]; both in natural labels.
// uv = (U0, U3, V1, V2): max over states of the larger / smaller member of the {00,11}
// pair and of the {01,10} pair, each summed as fl(fl(alpha + gamma) + beta) (:252-253).
// Packed form: with the state pair (x[t], x[8+t]) and the record pairs R[c] = (gp, gm), S[c] = (gm, gp), one add
// gives (p0, m1), which both continue with + zs[nP0], and one gives (m0, p1), which continue with + zs[nM0]; the
// "-h" terms pair up the same way.
TPF_HD void ext_step(float (&x)[16], const float (&zs)[16], const float (&g)[8], float (&uv)[4])
{
    f2 R[4], S[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) { R[c] = f2{g[2 * c], g[2 * c + 1]}; S[c] = f2{g[2 * c + 1], g[2 * c]}; }
    float n[16];
    float U0 = 0.f, U3 = 0.f, V1 = 0.f, V2 = 0.f;
#pragma unroll
    for (int t = 0; t < 8; ++t) {
        const int c = cls(t);
        const int t2 = (t >> 2) & 1;
        // state (0, t): P-branch -> 2t + t2, M-branch -> 2t + 1 - t2;  state (1, t): the other way
        const int nP0 = 2 * t + t2, nM0 = 2 * t + 1 - t2;
        const f2 xs = f2{x[t], x[8 + t]};
        const f2 zP = f2{zs[nP0], zs[nP0]}, zM = f2{zs[nM0], zs[nM0]};
        const f2 pm = add2(xs, R[c]), mp = add2(xs, S[c]);            // (p0, m1), (m0, p1)
        const f2 b01 = add2(pm, zP), b10 = add2(mp, zM);               // (ub0, vb1), (vb0, ub1)
        const f2 s01 = add2(sub2(xs, R[3 - c]), zP);                   // (us0, vs1): x - (hp, hm) + zs[nP0]
        const f2 s10 = add2(sub2(xs, S[3 - c]), zM);                   // (vs0, us1): x - (hm, hp) + zs[nM0]
        const float p0 = pm.lo, m1 = pm.hi, m0 = mp.lo, p1 = mp.hi;
        const float ub0 = b01.lo, vb1 = b01.hi, vb0 = b10.lo, ub1 = b10.hi;
        const float us0 = s01.lo, vs1 = s01.hi, vs0 = s10.lo, us1 = s10.hi;
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
    x[8] = f_sub(n[8], q);
#pragma unroll
    for (int t = 1; t < 8; ++t) {
        const f2 d = sub2(f2{n[t], n[8 + t]}, f2{q, q});
        x[t] = d.lo; x[8 + t] = d.hi;
    }
}

// Extrinsic epilogue for one step (dvb_rcs2_turbo.py:250-279).
TPF_HD void make_extrinsic(const float (&uv)[4], double YA, double YB, double sf, double &ea, double &eb)
{
    // sign of fl(YA/2 + YB/2) == sign of fl(YA + YB): halving commutes with rounding
    const bool sP = d_add(YA, YB) < 0.0, sM = d_sub(YA, YB) < 0.0;
    const float app0 = sP ? uv[1] : uv[0], app3 = sP ? uv[0] : uv[1];
    const float app1 = sM ? uv[3] : uv[2], app2 = sM ? uv[2] : uv[3];
    const float LA = f_sub(f_max(app0, app1), f_max(app2, app3));
    const float LB = f_sub(f_max(app0, app2), f_max(app1, app3));
    ea = d_mul(d_sub((double)LA, YA), sf);
    eb = d_mul(d_sub((double)LB, YB), sf);
    ea = ea > 300.0 ? 300.0 : ea; ea = ea < -300.0 ? -300.0 : ea;
    eb = eb > 300.0 ? 300.0 : eb; eb = eb < -300.0 ? -300.0 : eb;
}

}  // namespace tpf
}  // namespace b200dvb
