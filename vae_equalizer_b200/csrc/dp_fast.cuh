// Building blocks of the register-blocked DP kernels (dp_fast.cu, dp_fwd_tc.cu): tile geometry, padded float4 window
// indexing, the 3-multiplication FIR-like contraction and the packed tap-gradient correlation.
#pragma once
#include "dp_math.cuh"
#include "dp_kernels.cuh"

namespace vaeq {

constexpr int FT_NT = 128;                 // threads per CTA.  Every tile is load -> barrier -> FIR -> point-wise -> barrier -> ...,
                                           // so what hides one CTA's load / barrier phases is the OTHER CTAs of the SM: four
                                           // 128-thread CTAs per SM interleave better than two of 256 (0.664 -> 0.627 ms per step,
                                           // profiles/r01c_*), one of 512 is worst (0.782 vs 0.744, profiles/r01_cta_imbalance.txt).
                                           // The tap-gradient kernels need >= 4 warps (one per role), so 128 is the floor.
constexpr int FT_NW = FT_NT / 32;          // warps per CTA
constexpr int FT_CTAS_PER_SM = 512 / FT_NT;   // 128 registers per thread either way
constexpr int FT_R = 4;                    // consecutive symbols per thread
constexpr int FT_TE = FT_NT * FT_R;        // symbols per tile incl. halo (1024)
constexpr int FT_HP = 8;                   // halo per side in symbols (>= MH/2, multiple of 4)
constexpr int FT_T = FT_TE - 2 * FT_HP;    // owned symbols per tile (1008)
constexpr int FT_XOFF = 8;                 // extra margin of the x phase arrays (FIR reaches MH/2 further)
constexpr int FT_XN = FT_TE + 2 * FT_XOFF; // logical length of xe / xo
constexpr int FT_MINB_PW = FT_CTAS_PER_SM; // min CTAs per SM for the point-wise heavy kernels (fwd, bwd1)
constexpr int FT_MINB = FT_CTAS_PER_SM;    // ... and for the tap-gradient kernels (56 live accumulators)

__host__ __device__ constexpr int fdiv4(int c) { return c >= 0 ? c / 4 : -((3 - c) / 4); }
// padded float4 index of logical position 4*l + c (c compile-time, may be negative)
__host__ __device__ constexpr int poff(int c) { return c + fdiv4(c); }
__device__ __forceinline__ int pidx(int i) { return i + (i >> 2); }
__device__ __forceinline__ float f4c(const float4 &v, int r) { return r == 0 ? v.x : r == 1 ? v.y : r == 2 ? v.z : v.w; }
// SoA row helpers: 4 consecutive symbols of one row as a float4
__device__ __forceinline__ float4 ld_row4(const float *base, int64_t ld, int row, int u) {
    return __ldg(reinterpret_cast<const float4 *>(base + (int64_t)row * ld + u));
}
__device__ __forceinline__ void st_row4(float *base, int64_t ld, int row, int u, float4 v) {
    *reinterpret_cast<float4 *>(base + (int64_t)row * ld + u) = v;
}

constexpr int FT_XS = FT_XN + FT_XN / 4 + 4;   // padded lengths (float4)
constexpr int FT_ES = FT_TE + FT_TE / 4 + 4;


// FIR-like contraction  y_o(u) = sum_lag sum_i t_{o,i,lag} * x_i(u + lag)  (complex 2x2, 4 consecutive symbols per thread)
// with the 3-multiplication form of the complex product (Gauss):  for t = tr + j ti, x = xr + j xi
//     P1 = sum tr (xr + xi),  P2 = sum xr (ti - tr),  P3 = sum xi (tr + ti)   =>   Re = P1 - P3,  Im = P1 + P2.
// The three sums run over all lags and both inputs, so the tap-side terms (ti - tr, tr + ti) are tabulated once per kernel
// and the data-side term (xr + xi) once per window element: 3 FMA per complex MAC instead of 4 (-22 % FP32 pipe time in
// these loops incl. the two adds per window element).  Packed as fma.rn.f32x2:
//     P23[r][o] += (xr_i, xi_i) * (td_{o,i}, ts_{o,i})      (window pair x tap pair, i = 0, 1)
//     P1[r][o]  += (tr_{o,0}, tr_{o,1}) * (xs_0, xs_1)      (pair over the two inputs, halves summed at the end)
// Tap table per lag: T0 = {tr00, tr01, tr10, tr11}, T1 = {td00, ts00, td01, ts01}, T2 = {td10, ts10, td11, ts11}  (index o,i).
constexpr int FT_TAPV = 3;                 // float4 per lag in a tap table
struct FirAcc {
    float2 P1[FT_R][2], P23[FT_R][2];
};
struct WinEl {
    float4 x;                              // {re_0, im_0, re_1, im_1}
    float2 s;                              // {re_0 + im_0, re_1 + im_1}
};
__device__ __forceinline__ void fir_acc_zero(FirAcc &a) {
#pragma unroll
    for (int r = 0; r < FT_R; ++r)
#pragma unroll
        for (int o = 0; o < 2; ++o) a.P1[r][o] = a.P23[r][o] = make_float2(0.f, 0.f);
}
__device__ __forceinline__ void fir_acc_finish(const FirAcc &a, float (&acc)[FT_R][4]) {
#pragma unroll
    for (int r = 0; r < FT_R; ++r)
#pragma unroll
        for (int o = 0; o < 2; ++o) {
            const float p1 = a.P1[r][o].x + a.P1[r][o].y;
            acc[r][2 * o] += p1 - a.P23[r][o].y;
            acc[r][2 * o + 1] += p1 + a.P23[r][o].x;
        }
}
// fill one tap-table entry: e in [0,12) within the lag, (tr, ti) supplied by the caller for (o, i)
__device__ __forceinline__ void tap_entry_oi(int e, int &o, int &i) {
    if (e < 4) { o = e >> 1; i = e & 1; }
    else { o = (e - 4) >> 2; i = ((e - 4) >> 1) & 1; }
}
__device__ __forceinline__ float tap_entry_val(int e, float tr, float ti) {
    return e < 4 ? tr : (((e - 4) & 1) ? tr + ti : ti - tr);
}
__device__ __forceinline__ void fir_step(const float4 T0, const float4 T1, const float4 T2, const WinEl &xa, const WinEl &xb,
                                         const WinEl &xc, const WinEl &xd, FirAcc &a) {
    const WinEl *xs[4] = {&xa, &xb, &xc, &xd};
#pragma unroll
    for (int r = 0; r < FT_R; ++r) {
        const float4 x = xs[r]->x;
        const float2 s = xs[r]->s, x0 = make_float2(x.x, x.y), x1 = make_float2(x.z, x.w);
        a.P1[r][0] = __ffma2_rn(make_float2(T0.x, T0.y), s, a.P1[r][0]);
        a.P1[r][1] = __ffma2_rn(make_float2(T0.z, T0.w), s, a.P1[r][1]);
        a.P23[r][0] = __ffma2_rn(x0, make_float2(T1.x, T1.y), a.P23[r][0]);
        a.P23[r][0] = __ffma2_rn(x1, make_float2(T1.z, T1.w), a.P23[r][0]);
        a.P23[r][1] = __ffma2_rn(x0, make_float2(T2.x, T2.y), a.P23[r][1]);
        a.P23[r][1] = __ffma2_rn(x1, make_float2(T2.z, T2.w), a.P23[r][1]);
    }
}

__device__ __forceinline__ void fir4(const float4 *__restrict__ win, int i0, const float4 *__restrict__ taps, int nlag,
                                     float (&out)[FT_R][4]) {
    FirAcc acc;
    fir_acc_zero(acc);
    auto LD = [win](int j) {
        WinEl w;
        w.x = win[j + (j >> 2)];
        w.s = make_float2(w.x.x + w.x.y, w.x.z + w.x.w);
        return w;
    };
    WinEl w0 = LD(i0), w1 = LD(i0 + 1), w2 = LD(i0 + 2), w3;
    int a = 0;
#pragma unroll 1
    for (; a + 4 <= nlag; a += 4) {
        w3 = LD(i0 + 3);
        fir_step(taps[0], taps[1], taps[2], w0, w1, w2, w3, acc);
        w0 = LD(i0 + 4);
        fir_step(taps[3], taps[4], taps[5], w1, w2, w3, w0, acc);
        w1 = LD(i0 + 5);
        fir_step(taps[6], taps[7], taps[8], w2, w3, w0, w1, acc);
        w2 = LD(i0 + 6);
        fir_step(taps[9], taps[10], taps[11], w3, w0, w1, w2, acc);
        i0 += 4;
        taps += 4 * FT_TAPV;
    }
#pragma unroll 1
    for (; a < nlag; ++a) {                  // remainder (nlag % 4 lags): shift the window by register moves
        w3 = LD(i0 + 3);
        fir_step(taps[0], taps[1], taps[2], w0, w1, w2, w3, acc);
        w0 = w1; w1 = w2; w2 = w3;
        i0 += 1;
        taps += FT_TAPV;
    }
    fir_acc_finish(acc, out);
}

// ---------------------------------------------------------------------------------------------
// tap-gradient correlation: acc[a][2(2o+i)+c] += sum_r g[r]_o * conj(win[i0 + r + a]_i),  a < A
// ---------------------------------------------------------------------------------------------
// The window is stored SWIZZLED for these kernels, {re_0, re_1, im_0, im_1} (both inputs' real parts, then both imaginary
// parts), so that one packed fma.rn.f32x2 with a scalar-broadcast g operand updates the pair (i = 0, 1) of an output:
//     RE[o] += g_o.re * (x_0.re, x_1.re) + g_o.im * (x_0.im, x_1.im)      IM[o] += g_o.im * (x.re pair) - g_o.re * (x.im pair)
// 4 FFMA2 per (lag, symbol, o) instead of 8 FFMA: the tap-gradient kernels were issue-bound (66-73 % issue-active, 52-58 % FP32
// pipe, profiles/r01_*), the packed form halves their FMA issue slots.  acc2[a] = {RE[o0], IM[o0], RE[o1], IM[o1]}.
template <int A>
__device__ __forceinline__ void corr4(const float4 *__restrict__ win, int i0, const float4 (&g)[FT_R], float2 (&acc2)[A][4]) {
    float ng[FT_R][2];
#pragma unroll
    for (int r = 0; r < FT_R; ++r) {
        ng[r][0] = -g[r].x;
        ng[r][1] = -g[r].z;
    }
#pragma unroll
    for (int cpos = 0; cpos < A + FT_R - 1; ++cpos) {
        const int j = i0 + cpos;
        const float4 x = win[j + (j >> 2)];
        const float2 xr = make_float2(x.x, x.y), xi = make_float2(x.z, x.w);
#pragma unroll
        for (int r = 0; r < FT_R; ++r) {
            const int a = cpos - r;
            if (a >= 0 && a < A) {
                const float4 gg = g[r];
                acc2[a][0] = __ffma2_rn(make_float2(gg.x, gg.x), xr, acc2[a][0]);
                acc2[a][1] = __ffma2_rn(make_float2(gg.y, gg.y), xr, acc2[a][1]);
                acc2[a][2] = __ffma2_rn(make_float2(gg.z, gg.z), xr, acc2[a][2]);
                acc2[a][3] = __ffma2_rn(make_float2(gg.w, gg.w), xr, acc2[a][3]);
                acc2[a][0] = __ffma2_rn(make_float2(gg.y, gg.y), xi, acc2[a][0]);
                acc2[a][1] = __ffma2_rn(make_float2(ng[r][0], ng[r][0]), xi, acc2[a][1]);
                acc2[a][2] = __ffma2_rn(make_float2(gg.w, gg.w), xi, acc2[a][2]);
                acc2[a][3] = __ffma2_rn(make_float2(ng[r][1], ng[r][1]), xi, acc2[a][3]);
            }
        }
    }
}

}  // namespace vaeq
