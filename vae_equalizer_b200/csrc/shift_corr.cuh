// Shift-search correlation of find_shift / find_shift_symb_full (optical_DP_channel/shared_funcs.py:290-338) as ONE pass over
// the data, shared by the single-run kernel (eval.cu) and the batched sweep kernel (eval_runs.cu).
//
//   S[comp][b][a](i) = sum_t tx[a][comp][t] * E[b][(t - (i - half)) mod N],   i = 0 .. n_shift-1  (sf:300-304, circular roll)
//
// The first version launched one CTA per (shift, chunk): every shift re-read q (64 B/symbol at 64-QAM) and rebuilt
// E = sum_l a_l q_I[l], 21 times over (2.2 ms at N = 2^22 = 2 % of the HBM roofline, profiles/r01d_eval_cma.txt).  Here a CTA
// stages a tile of SC_T symbols ONCE in shared memory -- E for the tile plus the n_shift-1 positions the shifts reach, tx as
// float4 per symbol -- and a lane owns a shift: consecutive lanes read consecutive E positions (conflict-free), tx is a
// broadcast, 8 FMA per 3 shared loads.  A warp owns a 96-symbol slice of the tile; its fp32 partial sums are
// added to double accumulators that live across all tiles of the CTA, then the warps are summed in fixed order
// (deterministic), one [n_shift][8] block of doubles per CTA.
// n_shift <= 24 (the reference searches 21 shifts): a lane owns THREE consecutive shifts and a quarter of the warp's slice (8 shift
// groups x 4 quarters), keeps the three E positions a symbol needs in a sliding register window (one new shared load per row and
// symbol) and updates its 24 sums with packed fma.rn.f32x2 over the (tx pol 0, tx pol 1) pair: 12 FFMA2 per 3 shared loads instead
// of 8 FFMA, all 28 of 32 lanes busy at 21 shifts instead of 21.  Quarters of 24 symbols make the E loads of a warp bank-conflict free
// ({24 q - 3 g} are 32 distinct residues mod 32).
#pragma once
#include "common.cuh"

namespace vaeq {

constexpr int SC_NT = 128, SC_NW = SC_NT / 32;
constexpr int SC_T = 384;                      // symbols per tile
constexpr int SC_SLICE = SC_T / SC_NW;         // symbols per warp and tile
constexpr int SC_MAXSHIFT = 64;
constexpr int SC_MINB = 6;                     // CTAs per SM: the tile loop is load -> barrier -> correlate -> barrier, other CTAs hide the waits

struct ShiftSmem {
    float E[2][SC_T + 2 * SC_MAXSHIFT];        // window of E, starting SC back4 positions before the tile
    float4 X[SC_T];                            // {tx[a=0][comp=0], tx[1][0], tx[0][1], tx[1][1]} = tx rows 0, 2, 1, 3 (pairs over the tx pol a)
    double red[SC_MAXSHIFT][8];
};

__device__ __forceinline__ float4 ld4(const float *p) { return __ldg(reinterpret_cast<const float4 *>(p)); }

constexpr int SC_J = 3, SC_LQ = SC_SLICE / 4;    // shifts per lane and symbols per lane and tile of the blocked correlation (n_shift <= 8 SC_J)
static_assert(SC_LQ % 16 == 8, "quarters of 8 (mod 16) symbols keep the E loads of a warp conflict-free");

// tile part of the blocked correlation: lane (g = lane & 7, quarter = lane >> 3) adds symbols [s0, s1) of the staged tile to its sums for
// shifts 3 g + j; dacc[j][k], k = comp*4 + b*2 + a.  Shifts >= n_shift of the last group accumulate staged data that is never written out.
__device__ __forceinline__ void shift_corr_blocked_tile(const ShiftSmem &sm, int n_shift, int eoff, int tn, double (&dacc)[SC_J][8]) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, g = lane & 7, qtr = lane >> 3;
    const int s0 = wid * SC_SLICE + SC_LQ * qtr, s1 = min(tn, s0 + SC_LQ);
    if (SC_J * g >= n_shift || s0 >= s1) return;
    const int c = n_shift - 1 - SC_J * g + eoff;              // E position of shift 3 g at symbol 0 of the tile
    const float *e0 = sm.E[0] + c, *e1 = sm.E[1] + c;
    float2 F[SC_J][4];
#pragma unroll
    for (int j = 0; j < SC_J; ++j)
#pragma unroll
        for (int k = 0; k < 4; ++k) F[j][k] = make_float2(0.f, 0.f);
    // sliding window: w?[j] = E[s + c - j]
    float a1 = e0[max(s0 - 1, -c)], a2 = e0[max(s0 - 2, -c)], b1 = e1[max(s0 - 1, -c)], b2 = e1[max(s0 - 2, -c)];
#pragma unroll 4
    for (int s = s0; s < s1; ++s) {
        const float a0 = e0[s], b0 = e1[s];
        const float4 x = sm.X[s];
        const float2 xa = make_float2(x.x, x.y), xb = make_float2(x.z, x.w);
        const float aw[SC_J] = {a0, a1, a2}, bw[SC_J] = {b0, b1, b2};
#pragma unroll
        for (int j = 0; j < SC_J; ++j) {
            const float2 A = make_float2(aw[j], aw[j]), B = make_float2(bw[j], bw[j]);
            F[j][0] = __ffma2_rn(xa, A, F[j][0]);             // comp 0, b 0, a = 0 | 1
            F[j][1] = __ffma2_rn(xa, B, F[j][1]);             // comp 0, b 1
            F[j][2] = __ffma2_rn(xb, A, F[j][2]);             // comp 1, b 0
            F[j][3] = __ffma2_rn(xb, B, F[j][3]);             // comp 1, b 1
        }
        a2 = a1; a1 = a0; b2 = b1; b1 = b0;
    }
#pragma unroll
    for (int j = 0; j < SC_J; ++j)
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            dacc[j][2 * k] += (double)F[j][k].x;
            dacc[j][2 * k + 1] += (double)F[j][k].y;
        }
}

// Accumulates symbols [t_lo, t_hi) and writes dst[i * 8 + k], k = comp*4 + b*2 + a, for i < n_shift.  All threads of the CTA call it.
// t_lo must be a multiple of 4 for the vector paths to engage (the callers cut their ranges at multiples of 64).
// ONE_POL: both "polarisations" of E and of tx are polarisation 0 (rows 0 .. 2n-1 of q, rows I / Q of tx): the single-polarisation
// AWGN driver correlates stack((q, q)) with stack((tx, tx)) (AWGN :188-204), so a run needs only its own rows.
template <bool FROM_Q, int NPASS_, bool ONE_POL = false>   // 1: n_shift <= 32, 2: n_shift <= 64 (a lane owns shifts lane, lane + 32), 0: n_shift <= 24, blocked correlation
__device__ __forceinline__ void shift_corr_range(ShiftSmem &sm, const float *__restrict__ q, int64_t ld_q, const float *__restrict__ out,
                                                 int64_t ld_out, const uint16_t *__restrict__ tx, int64_t ld_tx, const float *amp,
                                                 int n_lev, int N, int n_shift, int64_t t_lo, int64_t t_hi, double *dst) {
    constexpr bool blocked = NPASS_ == 0;
    constexpr int NPASS = blocked ? 1 : NPASS_;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int half = n_shift / 2, back = n_shift - 1 - half;      // the shifts reach `back` positions before the tile ...
    const int back4 = (back + 3) & ~3, eoff = back4 - back;       // ... the staged window starts back4 (multiple of 4) before it
    const float *src = FROM_Q ? q : out;
    const int64_t ld_s = FROM_Q ? ld_q : ld_out;
    // 16-byte loads of 4 consecutive positions / 8-byte loads of 4 float16 when the rows allow it
    const bool vec_e = (N % 4 == 0) && (ld_s % 4 == 0) && (reinterpret_cast<uintptr_t>(src) % 16 == 0) && (t_lo % 4 == 0);
    const bool vec_x = (ld_tx % 4 == 0) && (reinterpret_cast<uintptr_t>(tx) % 8 == 0) && (t_lo % 4 == 0);
    float a_l[VAEQ_MAX_LEVELS];
#pragma unroll
    for (int l = 0; l < VAEQ_MAX_LEVELS; ++l) a_l[l] = (FROM_Q && l < n_lev) ? amp[l] : 0.f;
    double dacc[NPASS][8], dblk[SC_J][8];
#pragma unroll
    for (int ps = 0; ps < NPASS; ++ps)
#pragma unroll
        for (int k = 0; k < 8; ++k) dacc[ps][k] = 0.0;
#pragma unroll
    for (int j = 0; j < SC_J; ++j)
#pragma unroll
        for (int k = 0; k < 8; ++k) dblk[j][k] = 0.0;

    for (int64_t t0 = t_lo; t0 < t_hi; t0 += SC_T) {
        const int tn = (int)min((int64_t)SC_T, t_hi - t0);
        __syncthreads();                                          // the previous tile has been consumed
        // ---- E window: positions wb .. wb + wlen - 1 (mod N), 4 per work item ---------------------------------------------------
        const int64_t wb = t0 - back4;
        const int wlen = tn + back4 + half, ngrp = (wlen + 3) >> 2;
        for (int g = tid; g < ngrp; g += SC_NT) {
            const int64_t p0 = wb + 4 * g;
            float e[2][4];
            if (vec_e && p0 >= 0 && p0 + 3 < N) {
#pragma unroll
                for (int b = 0; b < 2; ++b) {
                    if (FROM_Q) {
                        e[b][0] = e[b][1] = e[b][2] = e[b][3] = 0.f;  // E_q[x_I] = sum_l a_l q_I[l]  (sf:297), l ascending
#pragma unroll
                        for (int l = 0; l < VAEQ_MAX_LEVELS; ++l)   // unrolled: the compiler keeps as many loads in flight as registers allow
                            if (l < n_lev) {
                                const float4 v = ld4(q + (int64_t)((ONE_POL ? 0 : b * 2 * n_lev) + l) * ld_q + p0);
                                e[b][0] += a_l[l] * v.x; e[b][1] += a_l[l] * v.y;
                                e[b][2] += a_l[l] * v.z; e[b][3] += a_l[l] * v.w;
                            }
                    } else {
                        const float4 v = ld4(out + (int64_t)(ONE_POL ? 0 : b * 2) * ld_out + p0);      // rx[:,0,:]  (sf:321)
                        e[b][0] = v.x; e[b][1] = v.y; e[b][2] = v.z; e[b][3] = v.w;
                    }
                }
            } else {                                              // window wraps around the ends of the sequence (circular roll)
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    int64_t pos = (p0 + k) % N;
                    if (pos < 0) pos += N;
#pragma unroll
                    for (int b = 0; b < 2; ++b) {
                        float acc;
                        if (FROM_Q) {
                            acc = 0.f;
#pragma unroll
                            for (int l = 0; l < VAEQ_MAX_LEVELS; ++l)
                                if (l < n_lev) acc += a_l[l] * q[(int64_t)((ONE_POL ? 0 : b * 2 * n_lev) + l) * ld_q + pos];
                        } else {
                            acc = out[(int64_t)(ONE_POL ? 0 : b * 2) * ld_out + pos];
                        }
                        e[b][k] = acc;
                    }
                }
            }
#pragma unroll
            for (int b = 0; b < 2; ++b) *reinterpret_cast<float4 *>(&sm.E[b][4 * g]) = make_float4(e[b][0], e[b][1], e[b][2], e[b][3]);
        }
        // ---- tx tile as float4 per symbol ----------------------------------------------------------------------------------------
        for (int g = tid; g < SC_T / 4; g += SC_NT) {
            float x[4][4];                                        // [row][k]
            const int j = 4 * g;
            if (vec_x && j + 3 < tn) {
#pragma unroll
                for (int r = 0; r < 4; ++r) {
                    const uint2 u = __ldg(reinterpret_cast<const uint2 *>(tx + (int64_t)(ONE_POL ? r & 1 : r) * ld_tx + t0 + j));
                    x[r][0] = half_bits_to_float((uint16_t)(u.x & 0xffffu)); x[r][1] = half_bits_to_float((uint16_t)(u.x >> 16));
                    x[r][2] = half_bits_to_float((uint16_t)(u.y & 0xffffu)); x[r][3] = half_bits_to_float((uint16_t)(u.y >> 16));
                }
            } else {
#pragma unroll
                for (int r = 0; r < 4; ++r)
#pragma unroll
                    for (int k = 0; k < 4; ++k) x[r][k] = (j + k < tn) ? half_bits_to_float(tx[(int64_t)(ONE_POL ? r & 1 : r) * ld_tx + t0 + j + k]) : 0.f;
            }
#pragma unroll
            for (int k = 0; k < 4; ++k) sm.X[j + k] = make_float4(x[0][k], x[2][k], x[1][k], x[3][k]);
        }
        __syncthreads();
        if (blocked) {
            shift_corr_blocked_tile(sm, n_shift, eoff, tn, dblk);
            continue;
        }
        const int s_lo = wid * SC_SLICE, s_hi = min(tn, s_lo + SC_SLICE);
#pragma unroll
        for (int ps = 0; ps < NPASS; ++ps) {
            const int i = lane + 32 * ps;
            if (i < n_shift && s_lo < s_hi) {
                const float *e0 = sm.E[0] + (n_shift - 1 - i) + eoff, *e1 = sm.E[1] + (n_shift - 1 - i) + eoff;
                float f[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll 4
                for (int s = s_lo; s < s_hi; ++s) {
                    const float E0 = e0[s], E1 = e1[s];
                    const float4 x = sm.X[s];
                    f[0] += x.x * E0; f[1] += x.y * E0; f[2] += x.x * E1; f[3] += x.y * E1;      // comp 0: (b, a) = 00 01 10 11
                    f[4] += x.z * E0; f[5] += x.w * E0; f[6] += x.z * E1; f[7] += x.w * E1;      // comp 1
                }
#pragma unroll
                for (int k = 0; k < 8; ++k) dacc[ps][k] += (double)f[k];
            }
        }
    }
    if (blocked) {
        // quarters of a warp (lanes g, g + 8, g + 16, g + 24) summed in fixed order, then the lanes of quarter 0 hold shifts 3 g + j
#pragma unroll
        for (int j = 0; j < SC_J; ++j)
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                double v = dblk[j][k];
                v += __shfl_xor_sync(0xffffffffu, v, 8);
                v += __shfl_xor_sync(0xffffffffu, v, 16);
                dblk[j][k] = v;
            }
        for (int w = 0; w < SC_NW; ++w) {
            __syncthreads();
            if (wid == w && lane < 8) {
#pragma unroll
                for (int j = 0; j < SC_J; ++j) {
                    const int i = SC_J * lane + j;
                    if (i < n_shift) {
#pragma unroll
                        for (int k = 0; k < 8; ++k) sm.red[i][k] = (w == 0 ? 0.0 : sm.red[i][k]) + dblk[j][k];
                    }
                }
            }
        }
    } else {
        // warps summed in fixed order
        for (int w = 0; w < SC_NW; ++w) {
            __syncthreads();
            if (wid == w) {
#pragma unroll
                for (int ps = 0; ps < NPASS; ++ps) {
                    const int i = lane + 32 * ps;
                    if (i < n_shift) {
#pragma unroll
                        for (int k = 0; k < 8; ++k) sm.red[i][k] = (w == 0 ? 0.0 : sm.red[i][k]) + dacc[ps][k];
                    }
                }
            }
        }
    }
    __syncthreads();
    for (int idx = tid; idx < n_shift * 8; idx += SC_NT) dst[idx] = sm.red[idx >> 3][idx & 7];
}

}  // namespace vaeq
