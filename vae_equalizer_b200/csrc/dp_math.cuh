// Point-wise math of the DP VAE step shared by every kernel variant (fp32, reference op order).
#pragma once
#include "common.cuh"

namespace vaeq {

// Per-run demapper constants staged once per CTA in shared memory.
struct DemapConst {
    float amp[VAEQ_MAX_LEVELS];   // a_l                       (sf:568)
    float a2[VAEQ_MAX_LEVELS];    // a_l^2
    float nua2[VAEQ_MAX_LEVELS];  // float(nu_sc) * a_l^2       (sf:520 PCS term)
    float P[VAEQ_MAX_LEVELS];     // prior pmf                  (sf:572)
    float var[2];                 // demapper variance per pol  (sf:581)
    float pad[2];
};

__device__ __forceinline__ void load_demap_const(DemapConst *c, const float *amp, const float *P, const float *var,
                                                 float nu_sc, int n_lev) {
    const int t = threadIdx.x;
    if (t < VAEQ_MAX_LEVELS) {
        float a = t < n_lev ? amp[t] : 0.f;
        c->amp[t] = a;
        c->a2[t] = a * a;
        c->nua2[t] = nu_sc * (a * a);
        c->P[t] = (t < n_lev && P != nullptr) ? P[t] : 1.f;
    }
    if (t < 2) c->var[t] = var[t];
}

// q_l = softmin_l( (y-a_l)^2/2/var + nu_sc a_l^2 )   (sf:521-523), max-subtracted like nn.Softmin.
// Also returns the first two posterior moments (sf:108-112).
template <int NL>
__device__ __forceinline__ void demap_component(float y, float var, const DemapConst &c, float (&q)[NL], float &m1,
                                                float &m2) {
    float z[NL];
    float zmin = 3.0e38f;
#pragma unroll
    for (int l = 0; l < NL; ++l) {
        float d = y - c.amp[l];
        z[l] = __fadd_rn(__fdiv_rn(__fmul_rn(__fmul_rn(d, d), 0.5f), var), c.nua2[l]);
        zmin = fminf(zmin, z[l]);
    }
    float s = 0.f;
#pragma unroll
    for (int l = 0; l < NL; ++l) {
        q[l] = expf(zmin - z[l]);
        s += q[l];
    }
    m1 = 0.f;
    m2 = 0.f;
#pragma unroll
    for (int l = 0; l < NL; ++l) {
        q[l] = __fdiv_rn(q[l], s);
        m1 = fmaf(c.amp[l], q[l], m1);
        m2 = fmaf(c.a2[l], q[l], m2);
    }
}

// 2x2 butterfly FIR of one symbol (sf:500-518): x0 is the first sample of the symbol's window in row 0 of four staged sample rows
// (pol 0 I, pol 0 Q, pol 1 I, pol 1 Q) XN floats apart, Ws the taps (2,4,M).  y = (p0 I, p0 Q, p1 I, p1 Q).
__device__ __forceinline__ void fir_butterfly(const float *x0, int XN, const float *Ws, int M, float (&y)[4]) {
    y[0] = y[1] = y[2] = y[3] = 0.f;
    for (int k = 0; k < M; ++k) {
        float xI0 = x0[k], xQ0 = x0[XN + k], xI1 = x0[2 * XN + k], xQ1 = x0[3 * XN + k];
#pragma unroll
        for (int o = 0; o < 2; ++o) {
            float wr0 = Ws[(o * 4 + 0) * M + k], wr1 = Ws[(o * 4 + 1) * M + k];
            float wi0 = Ws[(o * 4 + 2) * M + k], wi1 = Ws[(o * 4 + 3) * M + k];
            y[2 * o] += wr0 * xI0 + wr1 * xI1 - wi0 * xQ0 - wi1 * xQ1;       // sf:505,509
            y[2 * o + 1] += wr0 * xQ0 + wr1 * xQ1 + wi0 * xI0 + wi1 * xI1;   // sf:507,509
        }
    }
}

// entropy contribution  sum_l -q_l log(q_l/P_l + 1e-12)   (sf:132)
template <int NL>
__device__ __forceinline__ float entropy_component(const float (&q)[NL], const DemapConst &c) {
    float e = 0.f;
#pragma unroll
    for (int l = 0; l < NL; ++l) e -= q[l] * logf(__fdiv_rn(q[l], c.P[l]) + 1e-12f);
    return e;
}

// Back-propagate through moments + entropy + softmin for one I/Q component (SURVEY.md §8a-a7):
//   g1 = dL/dE_q[x] (already including -2 E_q[x] dL/dVar), g2 = dL/dE_q[x^2] = dL/dVar,
//   ent_on = 1 if this symbol is inside the entropy window.  Returns dL/dy.
template <int NL>
__device__ __forceinline__ float demap_backward(float y, float var, const DemapConst &c, const float (&q)[NL], float g1,
                                                float g2, bool ent_on) {
    float gq[NL];
    float dot = 0.f;
#pragma unroll
    for (int l = 0; l < NL; ++l) {
        float g = fmaf(c.amp[l], g1, c.a2[l] * g2);
        if (ent_on) {
            float u = __fdiv_rn(q[l], c.P[l]);
            float t = u + 1e-12f;
            g += logf(t) + __fdiv_rn(u, t);
        }
        gq[l] = g;
        dot = fmaf(q[l], g, dot);
    }
    float gy = 0.f;
#pragma unroll
    for (int l = 0; l < NL; ++l) {
        float gz = -q[l] * (gq[l] - dot);
        gy = fmaf(gz, y - c.amp[l], gy);
    }
    return __fdiv_rn(gy, var);
}

// ---------------------------------------------------------------------------------------------
// Fast point-wise math of the register-blocked path (dp_fast.cu) and the persistent small-minibatch kernel (dp_small.cu):
// ex2 / lg2 / rcp approximations, validated against the same tolerances as the precise functions above.
// ---------------------------------------------------------------------------------------------
constexpr float LOG2E = 1.4426950408889634f, LN2 = 0.6931471805599453f;

__device__ __forceinline__ float ex2_approx(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float lg2_approx(float x) {
    float y;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float rcp_approx(float x) {
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

struct FastConst {
    float amp[VAEQ_MAX_LEVELS], a2[VAEQ_MAX_LEVELS], a3[VAEQ_MAX_LEVELS];
    float nua2l[VAEQ_MAX_LEVELS];          // nu_sc a^2 log2(e)
    float lgP[VAEQ_MAX_LEVELS];            // log2 P_l
    float c2[2];                           // log2(e) / (2 var_p)
    float inv_var[2];
    // moment form of the demapper (demap_mom): valid when log2 P_l = alpha + beta a_l^2, the Maxwell-Boltzmann family of sf:572
    float ct[2];                           // c2 + nu_sc log2(e): curvature of the log2-posterior in a_l once the PCS term is folded in
    float eps[2];                          // nu_sc log2(e) / ct: the folded observation is y (1 - eps)
    float alpha, beta;
    float2 namp2[VAEQ_MAX_LEVELS];         // (-a_l, -a_l): operand pairs of the two-symbol packed form (demap_mom2)
    int quad;                              // 1 if the prior is of that family (max residual of the fit below 2e-6 in log2 units)
};

__device__ __forceinline__ void load_fast_const(FastConst *c, const float *amp, const float *P, const float *var, float nu_sc, int n_lev) {
    const int t = threadIdx.x;
    if (t < VAEQ_MAX_LEVELS) {
        const float a = t < n_lev ? amp[t] : 0.f;
        c->amp[t] = a;
        c->a2[t] = a * a;
        c->a3[t] = a * a * a;
        c->namp2[t] = make_float2(-a, -a);
        c->nua2l[t] = nu_sc * (a * a) * LOG2E;
        c->lgP[t] = t < n_lev ? log2f(P[t]) : 0.f;
    }
    if (t < 2) {
        c->c2[t] = LOG2E / (2.f * var[t]);
        c->inv_var[t] = 1.f / var[t];
        const float n = nu_sc * LOG2E, ct = LOG2E / (2.f * var[t]) + n;
        c->ct[t] = ct;
        c->eps[t] = n / ct;
    }
    if (t == 32) {                                          // two-point fit of log2 P over a^2 (innermost / outermost level), checked on all levels
        const int li = n_lev / 2, lo = n_lev - 1;
        const float ai = amp[li], ao = amp[lo], pi = log2f(P[li]), po = log2f(P[lo]);
        const float den = ao * ao - ai * ai;
        const float beta = den > 0.f ? (po - pi) / den : 0.f, alpha = pi - beta * ai * ai;
        float res = 0.f;
        for (int l = 0; l < n_lev; ++l) res = fmaxf(res, fabsf(log2f(P[l]) - fmaf(beta, amp[l] * amp[l], alpha)));
        c->alpha = alpha;
        c->beta = beta;
        c->quad = res <= 2e-6f ? 1 : 0;
    }
}

// soft demapper for one component: q, first two moments and the entropy term  sum_l -q_l ln(q_l / P_l).
// With BWD it also returns the three coefficients of the (linear) backward map of this component,
//     dL/dy = g1 * S1 + g2 * S2 + w * S3,   g1 = dL/dE_q[x], g2 = dL/dE_q[x^2], w = ln2 * [symbol inside the entropy window]
//     S1 = (m2 - m1^2)/var,  S2 = (m3 - m1 m2)/var,  S3 = (dotE (y - m1) - sum_l q_l ge_l (y - a_l))/var,
//     ge_l = log2(q_l / P_l), dotE = sum_l q_l ge_l
// (softmin + moments + entropy backward, closed form in oracle/closed_form.py, regrouped by input; S1 is d m1/dy).
// The backward kernel then needs neither q nor any transcendental.
template <int NL, bool BWD>
__device__ __forceinline__ void demap_fast(float y, float c2, float inv_var, const FastConst &c, float (&q)[NL], float &m1,
                                           float &m2, float &ent, float &S1, float &S2, float &S3) {
    float z[NL];
    float zmin = 3.0e38f;
#pragma unroll
    for (int l = 0; l < NL; ++l) {
        const float d = y - c.amp[l];
        z[l] = fmaf(d * c2, d, c.nua2l[l]);                 // ((y-a)^2/(2 var) + nu_sc a^2) * log2 e   (sf:521)
        zmin = fminf(zmin, z[l]);
    }
    float s = 0.f;
#pragma unroll
    for (int l = 0; l < NL; ++l) {
        z[l] = zmin - z[l];                                 // log2 of the unnormalised posterior
        q[l] = ex2_approx(z[l]);
        s += q[l];
    }
    const float r = rcp_approx(s), lgs = lg2_approx(s);
    m1 = 0.f;
    m2 = 0.f;
    float e = 0.f, m3 = 0.f, ea = 0.f;
#pragma unroll
    for (int l = 0; l < NL; ++l) {
        q[l] *= r;
        const float qa = q[l] * c.amp[l];
        m1 += qa;
        m2 = fmaf(qa, c.amp[l], m2);
        const float ge = z[l] - c.lgP[l];                   // log2(q_l / P_l) + lgs; the 1e-12 of sf:132 only matters where q/P < 1e-9
        e = fmaf(q[l], ge, e);
        if (BWD) {
            m3 = fmaf(qa, c.a2[l], m3);
            ea = fmaf(qa, ge, ea);
        }
    }
    ent = -LN2 * (e - lgs);                                 // sum_l q_l = 1
    if (BWD) {
        // S3 var = dotE (y - m1) - sum_l q_l ge'_l (y - a_l) with ge' = ge - lgs: the y and lgs terms cancel, leaving
        //        = sum_l q_l ge_l a_l - m1 sum_l q_l ge_l
        S1 = (m2 - m1 * m1) * inv_var;
        S2 = (m3 - m1 * m2) * inv_var;
        S3 = fmaf(-e, m1, ea) * inv_var;
    }
}

// Moment form of the same component (prior of the family log2 P_l = alpha + beta a_l^2, FastConst::quad).  The PCS term folds into the
// Gaussian: c2 (y - a)^2 + n a^2 = ct (u_l)^2 + const(y) with u_l = (y - a_l) - eps y, so the log2-posterior is -ct u_l^2 up to a shift.
// Every sum the step needs is a function of the first three moments of u under q (taken about the observation, where the posterior
// mass sits: no cancellation against O(1) level amplitudes):
//     m1 = y(1 - eps) - mu1,  Var = mu2 - mu1^2,  k3 = E[(u - mu1)^3] = mu3 - mu1 (3 Var + mu1^2)
//     S1 = dE_q/dy = Var / var,   T2 = dVar/dy = -k3 / var   (third cumulant of a = -k3)
//     sum_l q_l log2(q~_l / P_l) = zc - ct mu2 - alpha - beta (m1^2 + Var)
//     S3 var = Cov_q(a, log2(q~/P)) = ct (k3 + 2 mu1 Var) - beta (2 m1 Var - k3)
// 11.5 instructions per level instead of 15.5 and one constant table (a_l) instead of five.  Same tolerances as demap_fast
// (checked against it and against float64 in tests/test_dp_step_gpu.py).
template <int NL>
__device__ __forceinline__ void demap_mom(float y, float ct, float eps, float inv_var, const FastConst &c, float (&q)[NL], float &m1,
                                          float &var_q, float &ent, float &S1, float &T2, float &S3) {
    const float ey = eps * y;
    float u[NL], u2[NL];
    float u2min = 3.0e38f;
#pragma unroll
    for (int l = 0; l < NL; ++l) {
        u[l] = (y - c.amp[l]) - ey;                         // y - a_l first: exact for the levels next to y
        u2[l] = u[l] * u[l];
        u2min = fminf(u2min, u2[l]);
    }
    const float zc = ct * u2min;
    float s = 0.f, M1 = 0.f, M2 = 0.f, M3 = 0.f;
#pragma unroll
    for (int l = 0; l < NL; ++l) {
        const float pl = ex2_approx(fmaf(-ct, u2[l], zc));
        q[l] = pl;
        s += pl;
        const float pu = pl * u[l];
        M1 += pu;
        M2 = fmaf(pl, u2[l], M2);
        M3 = fmaf(pu, u2[l], M3);
    }
    const float r = rcp_approx(s), lgs = lg2_approx(s);
#pragma unroll
    for (int l = 0; l < NL; ++l) q[l] *= r;
    const float mu1 = M1 * r, mu2 = M2 * r, mu3 = M3 * r;
    m1 = (y - ey) - mu1;
    const float v = fmaf(-mu1, mu1, mu2);
    const float k3 = fmaf(-mu1, fmaf(mu1, mu1, 3.f * v), mu3);
    var_q = v;
    S1 = v * inv_var;
    T2 = -k3 * inv_var;
    const float e = fmaf(-c.beta, fmaf(m1, m1, v), fmaf(-ct, mu2, zc - c.alpha));
    ent = -LN2 * (e - lgs);
    const float mv2 = 2.f * v;
    S3 = (ct * fmaf(mu1, mv2, k3) - c.beta * fmaf(m1, mv2, -k3)) * inv_var;
}

// demap_mom for TWO symbols at once in packed fp32 (add / mul / fma .f32x2): the moment form is element-wise over the level index, so a
// symbol pair shares every instruction; 6.5 issue slots per level and symbol instead of 11.5 (the FP32 pipe cycles stay the same: the
// point-wise stage turns from issue-bound into pipe-bound).  Per-half operation order = demap_mom: bit-identical results.
__device__ __forceinline__ float2 f2(float a) { return make_float2(a, a); }
template <int NL>
__device__ __forceinline__ void demap_mom2(float2 y, float ct, float eps, float inv_var, const FastConst &c, float2 (&q)[NL], float2 &m1,
                                           float2 &var_q, float2 &ent, float2 &S1, float2 &T2, float2 &S3) {
    const float2 nct = f2(-ct), iv = f2(inv_var);
    const float2 ney = __fmul2_rn(y, f2(-eps));
    float2 u[NL], u2[NL];
    float mx = 3.0e38f, my = 3.0e38f;
#pragma unroll
    for (int l = 0; l < NL; ++l) {
        u[l] = __fadd2_rn(__fadd2_rn(y, c.namp2[l]), ney);
        u2[l] = __fmul2_rn(u[l], u[l]);
        mx = fminf(mx, u2[l].x);
        my = fminf(my, u2[l].y);
    }
    const float2 zc = __fmul2_rn(make_float2(mx, my), f2(ct));
    float2 s = f2(0.f), M1 = f2(0.f), M2 = f2(0.f), M3 = f2(0.f);
#pragma unroll
    for (int l = 0; l < NL; ++l) {
        const float2 z = __ffma2_rn(nct, u2[l], zc);
        const float2 pl = make_float2(ex2_approx(z.x), ex2_approx(z.y));
        q[l] = pl;
        s = __fadd2_rn(s, pl);
        const float2 pu = __fmul2_rn(pl, u[l]);
        M1 = __fadd2_rn(M1, pu);
        M2 = __ffma2_rn(pl, u2[l], M2);
        M3 = __ffma2_rn(pu, u2[l], M3);
    }
    const float2 r = make_float2(rcp_approx(s.x), rcp_approx(s.y)), lgs = make_float2(lg2_approx(s.x), lg2_approx(s.y));
#pragma unroll
    for (int l = 0; l < NL; ++l) q[l] = __fmul2_rn(q[l], r);
    const float2 mu1 = __fmul2_rn(M1, r), mu2 = __fmul2_rn(M2, r), mu3 = __fmul2_rn(M3, r);
    const float2 nmu1 = make_float2(-mu1.x, -mu1.y);
    m1 = __fadd2_rn(__fadd2_rn(y, ney), nmu1);
    const float2 v = __ffma2_rn(nmu1, mu1, mu2);
    const float2 k3 = __ffma2_rn(nmu1, __ffma2_rn(mu1, mu1, __fmul2_rn(f2(3.f), v)), mu3);
    var_q = v;
    S1 = __fmul2_rn(v, iv);
    T2 = __fmul2_rn(k3, f2(-inv_var));
    const float2 nb = f2(-c.beta);
    const float2 e = __ffma2_rn(nb, __ffma2_rn(m1, m1, v), __ffma2_rn(nct, mu2, __fadd2_rn(zc, f2(-c.alpha))));
    ent = __fmul2_rn(__fadd2_rn(e, make_float2(-lgs.x, -lgs.y)), f2(-LN2));
    const float2 mv2 = __fadd2_rn(v, v);
    const float2 nk3 = make_float2(-k3.x, -k3.y);
    S3 = __fmul2_rn(__ffma2_rn(nb, __ffma2_rn(m1, mv2, nk3), __fmul2_rn(f2(ct), __ffma2_rn(mu1, mv2, k3))), iv);
}

// ---------------------------------------------------------------------------------------------
// Adam (torch.optim.Adam single-tensor semantics, see oracle/closed_form.py)
// ---------------------------------------------------------------------------------------------
// Bias corrections of one Adam step (torch single-tensor path: step_size = -lr / (1 - beta1^t), denom uses sqrt(1 - beta2^t));
// double-precision pow is slow and identical for every parameter, so ONE thread computes it per CTA.
__device__ __forceinline__ void adam_bias(int step, double *bc1, float *bc2s) {
    *bc1 = 1.0 - pow(0.9, (double)step);
    *bc2s = (float)sqrt(1.0 - pow(0.999, (double)step));
}
__device__ __forceinline__ void adam_apply(float *param, float g, float *m, float *v, float *vmax, int i, float lr,
                                           bool amsgrad, double bc1, float bc2s) {
    const float b1 = 0.9f, b2 = 0.999f, eps = 1e-8f;
    float mi = m[i], vi = v[i];
    mi = mi + (g - mi) * (1.f - b1);                        // exp_avg.lerp_(grad, 1-beta1)
    vi = vi * b2 + (1.f - b2) * g * g;                      // exp_avg_sq.mul_(beta2).addcmul_(g,g,1-beta2)
    m[i] = mi;
    v[i] = vi;
    const float step_size = (float)(-(double)lr / bc1);
    float vv = vi;
    if (amsgrad) {
        vv = fmaxf(vmax[i], vi);
        vmax[i] = vv;
    }
    const float denom = __fadd_rn(__fdiv_rn(sqrtf(vv), bc2s), eps);
    param[i] = __fadd_rn(param[i], __fmul_rn(step_size, __fdiv_rn(mi, denom)));
}

}  // namespace vaeq
