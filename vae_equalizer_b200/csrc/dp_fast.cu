// DP VAE step, fast path for B200 (sm_100a): register-blocked tap contractions.
//
// Same math as dp_step.cu (the generic kernels remain the fallback and the in-library cross-check), organised
// for FFMA issue rate, which -- not HBM -- bounds this step at M_est = 25 (DESIGN.md "Roofline"):
//   * a thread owns FT_R = 4 CONSECUTIVE symbols, so a K-lag contraction slides a register window over
//     K + 3 shared-memory float4 loads for 64 K FFMA (the generic kernel does 1 LDS per 2-4 FFMA);
//   * rx is split into its even / odd sample phases (sps = 2), each stored as float4 {I0,Q0,I1,Q1} per
//     position, so every lag of the stride-2 FIR is a unit-stride access; the float4 index is padded
//     (i + i/4) so that the "lane owns 4 consecutive positions" pattern is bank-conflict free with
//     compile-time offsets;
//   * scratch that crosses kernels (residual e, moments, dL/dout) is SoA rows like q, so all global traffic
//     is float4 per thread, 512 B per warp instruction;
//   * point-wise math uses ex2/lg2/rcp approximations, a reciprocal multiply for 1/(2 var) and the analytic
//     log q = (z_min - z_l) - log2 s for the entropy, ~100 instructions per component instead of ~450;
//   * the backward pass is three lean kernels (dE_q + softmin backward -> dL/dout rows; dW; dh) so that no tap
//     accumulators live across the point-wise stage (no spills) and 2-3 CTAs fit per SM;
//   * the sliding-window loops are runtime-parameterised with an unroll-by-4 body (the window rotates through 4
//     register names) instead of being fully unrolled: ~25 KB of SASS per kernel instead of ~110 KB, which
//     removed the instruction-cache stalls ncu showed for the fully unrolled version (profiles/r01_*).
// Reference lines: twoXtwoFIR.forward sf:500-527, loss_function_shaping sf:92-137 (sf = optical_DP_channel/shared_funcs.py).
#include "dp_fast.cuh"

namespace vaeq {

// load the even/odd phase arrays of rx for the tile starting at symbol t0 (logical position 0 <-> symbol t0-HP-XOFF)
// SWZ = false: {I0,Q0,I1,Q1} per position (FIR windows); SWZ = true: {I0,I1,Q0,Q1} (tap-gradient windows, see corr4)
template <bool SWZ = false>
__device__ __forceinline__ void load_x_phases(const DpK &p, int t0, float4 *xe, float4 *xo) {
    const int sym0 = t0 - FT_HP - FT_XOFF;
#pragma unroll 1
    for (int j = threadIdx.x; j < FT_XN / 2; j += FT_NT) {
        const int64_t s0 = 2 * (int64_t)sym0 + 4 * j;           // first of 4 consecutive samples
        float4 v[4];
        if (s0 >= 0 && s0 + 3 < p.L) {
#pragma unroll
            for (int r = 0; r < 4; ++r) v[r] = __ldg(reinterpret_cast<const float4 *>(p.rx + (int64_t)r * p.ld_rx + s0));
        } else {
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                float t[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const int64_t s = s0 + k;
                    t[k] = (s >= 0 && s < p.L) ? p.rx[(int64_t)r * p.ld_rx + s] : 0.f;
                }
                v[r] = make_float4(t[0], t[1], t[2], t[3]);
            }
        }
        constexpr int r1 = SWZ ? 2 : 1, r2 = SWZ ? 1 : 2;
        xe[pidx(2 * j)] = make_float4(v[0].x, v[r1].x, v[r2].x, v[3].x);
        xo[pidx(2 * j)] = make_float4(v[0].y, v[r1].y, v[r2].y, v[3].y);
        xe[pidx(2 * j + 1)] = make_float4(v[0].z, v[r1].z, v[r2].z, v[3].z);
        xo[pidx(2 * j + 1)] = make_float4(v[0].w, v[r1].w, v[r2].w, v[3].w);
    }
}

// ---- asynchronous staging of the NEXT tile's rx (cp.async, 16 bytes, L1 bypass) ---------------------------------------------
// The raw rows (4 rows x 2*FT_XN samples, as they lie in HBM) are copied into a staging buffer while the current tile is being
// computed; at the top of the next iteration they are transposed smem -> smem into the even/odd phase arrays.  This takes
// the HBM/L2 load latency (8.6 % of the forward kernel's stall samples sat on the first use of the tile loader's LDG,
// profiles/r01c_*) off the critical path without holding the tile in registers.
constexpr int FT_RAWROW = FT_XN / 2;                    // float4 per raw row
constexpr int FT_RAW = 4 * FT_RAWROW;                   // float4 of the staging buffer
__device__ __forceinline__ void cp_async16(void *dst_smem, const void *src_gmem) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(dst_smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(src_gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

__device__ __forceinline__ void issue_x_raw(const DpK &p, int t0, float4 *raw) {
    const int sym0 = t0 - FT_HP - FT_XOFF;
#pragma unroll 1
    for (int j = threadIdx.x; j < FT_RAWROW; j += FT_NT) {
        const int64_t s0 = 2 * (int64_t)sym0 + 4 * j;           // chunks are entirely inside or outside [0, L): s0 and L are multiples of 4
        if (s0 >= 0 && s0 + 3 < p.L) {
#pragma unroll
            for (int r = 0; r < 4; ++r) cp_async16(raw + r * FT_RAWROW + j, p.rx + (int64_t)r * p.ld_rx + s0);
        } else {
#pragma unroll
            for (int r = 0; r < 4; ++r) raw[r * FT_RAWROW + j] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
    }
    cp_async_commit();
}
template <bool SWZ = false>
__device__ __forceinline__ void transpose_x_raw(const float4 *raw, float4 *xe, float4 *xo) {
#pragma unroll 1
    for (int j = threadIdx.x; j < FT_RAWROW; j += FT_NT) {
        float4 v[4];
#pragma unroll
        for (int r = 0; r < 4; ++r) v[r] = raw[r * FT_RAWROW + j];
        constexpr int r1 = SWZ ? 2 : 1, r2 = SWZ ? 1 : 2;
        xe[pidx(2 * j)] = make_float4(v[0].x, v[r1].x, v[r2].x, v[3].x);
        xo[pidx(2 * j)] = make_float4(v[0].y, v[r1].y, v[r2].y, v[3].y);
        xe[pidx(2 * j + 1)] = make_float4(v[0].z, v[r1].z, v[r2].z, v[3].z);
        xo[pidx(2 * j + 1)] = make_float4(v[0].w, v[r1].w, v[r2].w, v[3].w);
    }
}

// Tile iteration of a persistent CTA.  Static: tile += gridDim.x (bitwise reproducible partial sums).  Dynamic: the
// next tile index comes from an atomic counter, fetched ONE TILE AHEAD by thread 0 and published through shared memory
// at the barrier that follows the staging of the current tile, so faster CTAs take more tiles and no SM idles at the end
// (profiles/r01_cta_imbalance.txt); the summation order of the per-CTA partials then varies from run to run.
struct TileIter {
    int cur, next;
};
__device__ __forceinline__ void tile_fetch_next(const DpK &p, int k, int cur, int *s_next) {
    if (threadIdx.x == 0) *s_next = p.dyn ? atomicAdd(p.tile_ctr + k, 1) + (int)gridDim.x : cur + (int)gridDim.x;
}

// point-wise stage of the forward kernel for a thread's FT_R symbols: soft demapper, posterior moments, entropy, backward
// coefficients, row stores.  Rolled over the polarisation (code size); y rotates by two components per pass.  Posterior means go
// straight to the shared E_q window (float2 half per polarisation pass): they are not held in registers across the stage, which
// sits at the 128-register cap.  MOM = moment form of the demapper (demap_mom), else the per-level sums (demap_fast).
template <int NL, int MH, bool MOM>
__device__ __forceinline__ void fwd_pointwise(const DpK &p, const FastConst &c, float (&y)[FT_R][4], float4 *m1s, int tid, int u0, bool owned,
                                              bool counted, float &accEnt, float &accV0, float &accV1) {
#pragma unroll 1
    for (int pol = 0; pol < 2; ++pol) {
        float vs[FT_R];
#pragma unroll
        for (int cq = 0; cq < 2; ++cq) {
            const int cc = 2 * pol + cq;
            float qv[FT_R][NL], m1v[FT_R], s1v[FT_R], t2v[FT_R], s3v[FT_R];
            if (MOM) {
#pragma unroll
                for (int r = 0; r < FT_R; r += 2) {                                       // a symbol pair per packed instruction
                    float2 q2[NL], m1p, vp, entp, s1p, t2p, s3p;
                    demap_mom2<NL>(make_float2(y[r][cq], y[r + 1][cq]), c.ct[pol], c.eps[pol], c.inv_var[pol], c, q2, m1p, vp, entp, s1p, t2p, s3p);
#pragma unroll
                    for (int l = 0; l < NL; ++l) { qv[r][l] = q2[l].x; qv[r + 1][l] = q2[l].y; }
                    m1v[r] = m1p.x; m1v[r + 1] = m1p.y;
                    s1v[r] = s1p.x; s1v[r + 1] = s1p.y;
                    t2v[r] = t2p.x; t2v[r + 1] = t2p.y;
                    s3v[r] = s3p.x; s3v[r + 1] = s3p.y;
                    const int u = u0 + r;
                    if (counted && u >= MH && u < p.B - MH) accEnt += entp.x;             // sf:132
                    if (counted && u + 1 >= MH && u + 1 < p.B - MH) accEnt += entp.y;
                    vs[r] = cq ? vs[r] + vp.x : vp.x;
                    vs[r + 1] = cq ? vs[r + 1] + vp.y : vp.y;
                    reinterpret_cast<float *>(&m1s[5 * tid + r])[2 * pol + cq] = m1p.x;
                    reinterpret_cast<float *>(&m1s[5 * tid + r + 1])[2 * pol + cq] = m1p.y;
                }
            } else {
#pragma unroll
                for (int r = 0; r < FT_R; ++r) {
                    float v, ent, m2, S2;
                    demap_fast<NL, true>(y[r][cq], c.c2[pol], c.inv_var[pol], c, qv[r], m1v[r], m2, ent, s1v[r], S2, s3v[r]);
                    t2v[r] = fmaf(-2.f * m1v[r], s1v[r], S2);
                    v = m2 - m1v[r] * m1v[r];                                             // sf:113
                    const int u = u0 + r;
                    if (counted && u >= MH && u < p.B - MH) accEnt += ent;                // sf:132
                    vs[r] = cq ? vs[r] + v : v;
                    reinterpret_cast<float *>(&m1s[5 * tid + r])[2 * pol + cq] = m1v[r];
                }
            }
            if (owned) {
                if (p.q != nullptr) {                // NULL in the frame loops that only keep a section of every window
#pragma unroll
                    for (int l = 0; l < NL; ++l)
                        st_row4(p.q, p.ld_q, cc * NL + l, u0, make_float4(qv[0][l], qv[1][l], qv[2][l], qv[3][l]));
                    st_row4(p.out, p.ld_out, cc, u0, make_float4(y[0][cq], y[1][cq], y[2][cq], y[3][cq]));
                }
                st_row4(p.m1rows, p.B, cc, u0, make_float4(m1v[0], m1v[1], m1v[2], m1v[3]));
                if (p.need_bwd) {
                    st_row4(p.srows, p.B, cc, u0, make_float4(s1v[0], s1v[1], s1v[2], s1v[3]));
                    st_row4(p.srows, p.B, 4 + cc, u0, make_float4(t2v[0], t2v[1], t2v[2], t2v[3]));
                    st_row4(p.srows, p.B, 8 + cc, u0, make_float4(s3v[0], s3v[1], s3v[2], s3v[3]));
                }
                if (p.qk != nullptr && counted) {    // batch-split: the rank that counts a symbol keeps it
                    const int k0 = u0 - p.keep_lo;
                    if (p.keep_vec && k0 >= 0 && k0 + FT_R <= p.keep_n) {            // all four symbols kept, 16-byte aligned destination
                        const int64_t col = p.keep_base + k0;
#pragma unroll
                        for (int l = 0; l < NL; ++l)
                            *reinterpret_cast<float4 *>(p.qk + (int64_t)(cc * NL + l) * p.ld_qk + col) = make_float4(qv[0][l], qv[1][l], qv[2][l], qv[3][l]);
                        *reinterpret_cast<float4 *>(p.outk + (int64_t)cc * p.ld_outk + col) = make_float4(y[0][cq], y[1][cq], y[2][cq], y[3][cq]);
                    } else if (k0 > -FT_R && k0 < p.keep_n) {
#pragma unroll 1
                        for (int r = 0; r < FT_R; ++r) {
                            const int u = u0 + r;
                            if (u >= p.keep_lo && u < p.keep_lo + p.keep_n) {
                                const int64_t col = p.keep_base + (u - p.keep_lo);
                                for (int l = 0; l < NL; ++l)
                                    p.qk[(int64_t)(cc * NL + l) * p.ld_qk + col] = f4c(make_float4(qv[0][l], qv[1][l], qv[2][l], qv[3][l]), r);
                                p.outk[(int64_t)cc * p.ld_outk + col] = f4c(make_float4(y[0][cq], y[1][cq], y[2][cq], y[3][cq]), r);
                            }
                        }
                    }
                }
            }
        }
        if (counted) {
            const float vsum = (vs[0] + vs[1]) + (vs[2] + vs[3]);
            accV0 += pol ? 0.f : vsum;
            accV1 += pol ? vsum : 0.f;
#pragma unroll
            for (int r = 0; r < FT_R; ++r) {
                const int u = u0 + r;
                if (u < MH || u >= p.B - MH) {
                    const int slot = (u < MH) ? u : MH + (u - (p.B - MH));
                    p.edge_vs[2 * MH * pol + slot] = vs[r];
                }
            }
        }
#pragma unroll
        for (int r = 0; r < FT_R; ++r) {             // rotate: the next pass finds its components in slots 0,1
            float t;
            t = y[r][0]; y[r][0] = y[r][2]; y[r][2] = t;
            t = y[r][1]; y[r][1] = y[r][3]; y[r][3] = t;
        }
    }
}

// ---------------------------------------------------------------------------------------------
// forward
// ---------------------------------------------------------------------------------------------
template <int NL, int MH>
__global__ void __launch_bounds__(FT_NT, FT_MINB_PW) k_dp_fwd_fast(DpK p) {
    static_assert(MH % 2 == 0 && MH / 2 <= FT_HP - 2, "fast path needs M_est = 1 (mod 4) and M_est <= 25");
    constexpr int M = 2 * MH + 1, HF = MH / 2, NE = MH + 1, NO = MH;
    extern __shared__ __align__(16) float4 smem4[];
    float4 *xe = smem4, *xo = xe + FT_XS, *m1s = xo + FT_XS;
    float4 *tapF = m1s + FT_ES;                              // FIR taps: [phase][lag][FT_TAPV]
    float4 *tapD = tapF + FT_TAPV * (NE + NO);               // channel taps, reversed per phase
    float4 *raw = tapD + FT_TAPV * (NE + NO);                // staging of the next tile's raw rx rows (cp.async)
    FastConst *cst = reinterpret_cast<FastConst *>(raw + FT_RAW);
    float *red = reinterpret_cast<float *>(cst + 1);
    const int tid = threadIdx.x;

    if ((int)blockIdx.x < p.ntiles) issue_x_raw(p, p.clo + (int)blockIdx.x * FT_T, raw);     // first tile: in flight during the setup
    for (int idx = tid; idx < (NE + NO) * 4 * FT_TAPV; idx += FT_NT) {
        const int la = idx / (4 * FT_TAPV), e = idx - la * (4 * FT_TAPV);
        const int ph = la >= NE, a = ph ? la - NE : la;
        int o, i;
        tap_entry_oi(e, o, i);
        const int k = 2 * a + ph;
        reinterpret_cast<float *>(tapF)[idx] = tap_entry_val(e, p.W[(o * 4 + i) * M + k], p.W[(o * 4 + 2 + i) * M + k]);
        const int j = ph ? (2 * MH - 1 - 2 * a) : (2 * MH - 2 * a);
        reinterpret_cast<float *>(tapD)[idx] = tap_entry_val(e, p.h[((o * 2 + i) * 2 + 0) * M + j], p.h[((o * 2 + i) * 2 + 1) * M + j]);
    }
    load_fast_const(cst, p.amp, p.P, p.var, p.nu_sc, NL);
    cp_async_wait_all();
    __syncthreads();
    const FastConst &c = *cst;

    float accC[2] = {0.f, 0.f}, accEnt = 0.f, accV0 = 0.f, accV1 = 0.f;   // scalars: accV[pol] in the rolled pol loop lived in local memory
    const int i0 = FT_R * tid;                               // local index of this thread's first symbol
    __shared__ int s_next;

#pragma unroll 1
    for (int tile = blockIdx.x; tile < p.ntiles;) {
        const int t0 = p.clo + tile * FT_T;
        tile_fetch_next(p, 0, tile, &s_next);
        transpose_x_raw(raw, xe, xo);                        // this tile's rows were staged while the previous one was computed
        __syncthreads();
        const int tile_next = s_next;
        if (tile_next < p.ntiles) issue_x_raw(p, p.clo + tile_next * FT_T, raw);      // lands during this tile's compute

        const int u0 = t0 - FT_HP + i0;
        const bool in_seq = (u0 >= 0) && (u0 < p.B);         // B % 4 == 0: all four symbols in or out together
        const bool owned = in_seq && (i0 >= FT_HP) && (i0 < FT_HP + FT_T) && (u0 < p.chi);
        const bool counted = owned && (u0 >= p.sym_lo) && (u0 < p.sym_hi);   // sums only over this rank's symbols
        if (!in_seq) {
#pragma unroll
            for (int r = 0; r < FT_R; ++r) m1s[5 * tid + r] = make_float4(0.f, 0.f, 0.f, 0.f);
        } else {
            float y[FT_R][4];
#pragma unroll
            for (int r = 0; r < FT_R; ++r)
#pragma unroll
                for (int k = 0; k < 4; ++k) y[r][k] = 0.f;
            // x[2u + k - MH]: even k = 2a -> xe[u + a - HF], odd k = 2a+1 -> xo[u + a - HF]
#pragma unroll 1
            for (int ph = 0; ph < 2; ++ph)
                fir4(ph ? xo : xe, i0 + FT_XOFF - HF, tapF + (ph ? FT_TAPV * NE : 0), ph ? NO : NE, y);
            // point-wise stage: moment form when the prior is of the Maxwell-Boltzmann family (every reference constellation), else the
            // per-level sums (CTA-uniform branch: one of the two code paths runs for the whole launch)
            if (c.quad) fwd_pointwise<NL, MH, true>(p, c, y, m1s, tid, u0, owned, counted, accEnt, accV0, accV1);
            else fwd_pointwise<NL, MH, false>(p, c, y, m1s, tid, u0, owned, counted, accEnt, accV0, accV1);
        }
        __syncthreads();

        // ---- D = h * E_q for the owned samples, residual e = D - rx ------------------------------------
        if (owned) {
#pragma unroll 1
            for (int ph = 0; ph < 2; ++ph) {
                float d[FT_R][4];
#pragma unroll
                for (int r = 0; r < FT_R; ++r)
#pragma unroll
                    for (int k = 0; k < 4; ++k) d[r][k] = 0.f;
                // even samples: sum_a h[2MH-2a] E_q[u + a - HF];  odd: sum_b h[2MH-1-2b] E_q[u + b - HF + 1]
                fir4(m1s, i0 - HF + ph, tapD + (ph ? FT_TAPV * NE : 0), ph ? NO : NE, d);
                const float4 *xr = ph ? xo : xe;
                float ev[4][FT_R];
#pragma unroll
                for (int r = 0; r < FT_R; ++r) {
                    const int u = u0 + r, s = 2 * u + ph, j = i0 + FT_XOFF + r;
                    const float4 x = xr[j + (j >> 2)];
                    const bool valid = (s >= MH) && (s < p.L - MH);                         // sf:120 "valid" region
                    ev[0][r] = valid ? d[r][0] - x.x : 0.f;
                    ev[1][r] = valid ? d[r][1] - x.y : 0.f;
                    ev[2][r] = valid ? d[r][2] - x.z : 0.f;
                    ev[3][r] = valid ? d[r][3] - x.w : 0.f;
                    if (counted) {
                        accC[0] += ev[0][r] * ev[0][r] + ev[1][r] * ev[1][r];
                        accC[1] += ev[2][r] * ev[2][r] + ev[3][r] * ev[3][r];
                    }
                }
#pragma unroll
                for (int k = 0; k < 4; ++k) st_row4(p.erows, p.B, 4 * ph + k, u0, make_float4(ev[k][0], ev[k][1], ev[k][2], ev[k][3]));
            }
        }
        cp_async_wait_all();
        __syncthreads();
        tile = tile_next;
    }

    float v[5] = {accC[0], accC[1], accEnt, accV0, accV1};
    block_sum<5>(v, red);
    if (tid == 0) {
        double *dst = p.part_fwd + (int64_t)blockIdx.x * 8;
#pragma unroll
        for (int i = 0; i < 5; ++i) dst[i] = (double)v[i];
    }
}

// ---------------------------------------------------------------------------------------------
// backward 1: dL/dE_q (FIR-like over gD = 2 kappa e), then dL/dout = dL/dE_q*S1 + dL/dVar*T2 + w*S3 (coefficients from
// the forward pass) -> dL/dout rows.  No q, no transcendental: 400 FFMA + ~30 other instructions per symbol.
// ---------------------------------------------------------------------------------------------
template <int NL, int MH>
__global__ void __launch_bounds__(FT_NT, FT_MINB_PW) k_dp_bwd1_fast(DpK p) {
    constexpr int M = 2 * MH + 1, HF = MH / 2, NE = MH + 1, NO = MH;
    extern __shared__ __align__(16) float4 smem4[];
    float4 *ge = smem4, *go = ge + FT_ES;
    float4 *tapG = go + FT_ES;                               // 2 kappa_chi conj(h) taps for dE_q: [phase][lag][FT_TAPV]
    float4 *sst = tapG + FT_TAPV * (NE + NO);                // [12][FT_NT]: this thread's S1/T2/S3 float4s, landed by cp.async
    float *PSg = reinterpret_cast<float *>(sst + 12 * FT_NT);         // (2, M+1)
    const int tid = threadIdx.x;
    const float kap0 = p.scal[DP_KAPPA_OFF], kap1 = p.scal[DP_KAPPA_OFF + 1];

    for (int idx = tid; idx < (NE + NO) * 4 * FT_TAPV; idx += FT_NT) {
        const int la = idx / (4 * FT_TAPV), e = idx - la * (4 * FT_TAPV);
        const int ph = la >= NE, a = ph ? la - NE : la;
        int nu, chi;                                              // out index nu, in index chi
        tap_entry_oi(e, nu, chi);
        const int j = 2 * a + ph;
        const float sc = 2.f * (chi ? kap1 : kap0);               // gD = 2 kappa_chi e folded into the taps
        reinterpret_cast<float *>(tapG)[idx] = tap_entry_val(e, sc * p.h[((chi * 2 + nu) * 2 + 0) * M + j], -sc * p.h[((chi * 2 + nu) * 2 + 1) * M + j]);
    }
    if (tid < 2) {
        const int nu = tid;
        float a = 0.f;
        PSg[nu * (M + 1)] = 0.f;
        for (int j = 0; j < M; ++j) {
            const float h0r = p.h[((0 * 2 + nu) * 2 + 0) * M + j], h0i = p.h[((0 * 2 + nu) * 2 + 1) * M + j];
            const float h1r = p.h[((1 * 2 + nu) * 2 + 0) * M + j], h1i = p.h[((1 * 2 + nu) * 2 + 1) * M + j];
            a += kap0 * (h0r * h0r + h0i * h0i) + kap1 * (h1r * h1r + h1i * h1i);
            PSg[nu * (M + 1) + j + 1] = a;
        }
    }
    __syncthreads();
    const int i0 = FT_R * tid;
    __shared__ int s_next;

#pragma unroll 1
    for (int tile = blockIdx.x; tile < p.ntiles;) {
        const int t0 = p.sym_lo + tile * FT_T;
        tile_fetch_next(p, 1, tile, &s_next);
        const int u0 = t0 - FT_HP + i0;
        const bool in_seq = (u0 >= 0) && (u0 < p.B);
        const bool owned = in_seq && (i0 >= FT_HP) && (i0 < FT_HP + FT_T) && (u0 < p.sym_hi);
        if (owned) {                                         // backward coefficients of MY four symbols: in flight during the e staging
#pragma unroll                                               // and the FIR-like loop below, read back by the same thread (no barrier)
            for (int k = 0; k < 12; ++k) cp_async16(sst + k * FT_NT + tid, p.srows + (int64_t)k * p.B + u0);
        }
        cp_async_commit();
        {   // stage the residual e for the tile and its halo (gD = 2 kappa e: the factor sits in the taps)
            float4 er[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) er[k] = in_seq ? ld_row4(p.erows, p.B, k, u0) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int r = 0; r < FT_R; ++r) {
                ge[5 * tid + r] = make_float4(f4c(er[0], r), f4c(er[1], r), f4c(er[2], r), f4c(er[3], r));
                go[5 * tid + r] = make_float4(f4c(er[4], r), f4c(er[5], r), f4c(er[6], r), f4c(er[7], r));
            }
        }
        __syncthreads();
        if (owned) {
            float gE[FT_R][4];
#pragma unroll
            for (int r = 0; r < FT_R; ++r)
#pragma unroll
                for (int k = 0; k < 4; ++k) gE[r][k] = 0.f;
            // dL/dE_q(u) = sum_chi sum_j conj(h[chi][nu][j]) gD_chi(2u - MH + j): even j -> ge[u+a-HF], odd j -> go[u+a-HF]
#pragma unroll 1
            for (int ph = 0; ph < 2; ++ph) fir4(ph ? go : ge, i0 - HF, tapG + (ph ? FT_TAPV * NE : 0), ph ? NO : NE, gE);
            float entw[FT_R];
#pragma unroll
            for (int r = 0; r < FT_R; ++r) {
                const int u = u0 + r;
                entw[r] = (u >= MH && u < p.B - MH) ? LN2 : 0.f;
            }
            cp_async_wait_all();
#pragma unroll 1
            for (int pol = 0; pol < 2; ++pol) {
                float gV[FT_R];
#pragma unroll
                for (int r = 0; r < FT_R; ++r) {
                    const int u = u0 + r;
                    const int jlo = max(0, 2 * MH - 2 * u), jhi = min(M, p.L - 2 * u);
                    gV[r] = PSg[pol * (M + 1) + jhi] - PSg[pol * (M + 1) + jlo];
                }
#pragma unroll
                for (int cq = 0; cq < 2; ++cq) {
                    const int cc = 2 * pol + cq;
                    // dL/dout = dL/dE_q * S1 + dL/dVar * T2 + w * S3 with the coefficients the forward pass left in srows
                    const float4 s1 = sst[cc * FT_NT + tid], t2 = sst[(4 + cc) * FT_NT + tid], s3 = sst[(8 + cc) * FT_NT + tid];
                    float gy[FT_R];
#pragma unroll
                    for (int r = 0; r < FT_R; ++r)
                        gy[r] = fmaf(gE[r][cq], f4c(s1, r), fmaf(gV[r], f4c(t2, r), entw[r] * f4c(s3, r)));
                    st_row4(p.gyrows, p.B, cc, u0, make_float4(gy[0], gy[1], gy[2], gy[3]));
                }
#pragma unroll
                for (int r = 0; r < FT_R; ++r) {
                    gE[r][0] = gE[r][2];
                    gE[r][1] = gE[r][3];
                }
            }
        }
        const int tile_next = s_next;                        // written before the staging barrier of this iteration
        __syncthreads();
        tile = tile_next;
    }
}

// roles: 0 = even phase lags [0, A0e), 1 = even [A0e, NE), 2 = odd [0, A0o), 3 = odd [A0o, NO)
template <int MH>
struct Roles {
    static constexpr int NE = MH + 1, NO = MH;
    static constexpr int A0e = (NE + 1) / 2, A1e = NE - A0e, A0o = (NO + 1) / 2, A1o = NO - A0o;
    static constexpr int AMAX = A0e;
};

// ---------------------------------------------------------------------------------------------
// backward 2 (FAM = 0): dW[o][i][2a+ph]   = sum_u gy_o(u)      conj(x_ph,i[u + a - HF])
// backward 3 (FAM = 1): dh[chi][nu][j(a)] = sum_v gD_ph,chi(v) conj(E_q,nu[v + a - HF + ph]),  j = 2MH - ph - 2a
// Each warp owns one role = (phase, lag half) for the whole kernel (warps w and w+4 share a role and split the
// symbol groups); its AMAX x 8 accumulators live in registers across all tiles of the persistent CTA.
// ---------------------------------------------------------------------------------------------
// The per-symbol operand g (dL/dout rows for dW, residual rows e for dh) is used by its SoA rows directly: a lane's four symbols
// are one float4 per row, so the rows land in shared memory by cp.async exactly as they lie in HBM (double-buffered: the next
// tile's rows are in flight while this tile is correlated) and are "transposed" by register naming only.  The sliding-window
// operand needs one float4 per position: raw rows are staged by cp.async as well and re-laid-out smem -> smem at the top
// of the next iteration (dW: rx phases; dh: E_q rows, by the owning thread, no barrier).
constexpr int FT_GROW = FT_TE / 4;                      // float4 per staged g row
template <int NROW>
__device__ __forceinline__ void issue_g_rows(const float *rows, int64_t ld, int u0, bool owned, float4 *dst) {
    if (owned) {
#pragma unroll
        for (int k = 0; k < NROW; ++k) cp_async16(dst + k * FT_GROW + threadIdx.x, rows + (int64_t)k * ld + u0);
    }
}

template <int MH, int FAM>
__global__ void __launch_bounds__(FT_NT, FT_MINB) k_dp_taps_fast(DpK p) {
    constexpr int M = 2 * MH + 1, HF = MH / 2, NG = FAM == 0 ? 4 : 8;
    using RL = Roles<MH>;
    extern __shared__ __align__(16) float4 smem4[];
    // FAM 0: s0 = xe, s1 = xo (windows), raw = next tile's rx rows, grow = dL/dout rows (4).
    // FAM 1: s0 = s1 = E_q window, raw = next tile's E_q rows (4 x FT_GROW, own slots), grow = residual rows (8: even | odd phase).
    float4 *s0 = smem4, *s1 = FAM == 0 ? s0 + FT_XS : s0;
    float4 *raw = FAM == 0 ? s1 + FT_XS : s0 + FT_ES;
    float4 *grow = raw + (FAM == 0 ? FT_RAW : 4 * FT_GROW);  // [2][NG][FT_GROW]
    float *red = reinterpret_cast<float *>(grow + 2 * NG * FT_GROW);
    const int tid = threadIdx.x, wid = tid >> 5, lane = tid & 31, role = wid & 3, ph = role >> 1;
    const int a0 = (role & 1) ? (ph ? RL::A0o : RL::A0e) : 0;
    const int n_real = role == 0 ? RL::A0e : role == 1 ? RL::A1e : role == 2 ? RL::A0o : RL::A1o;
    const float4 *win = ph ? s1 : s0;
    const int c0 = (FAM == 0 ? FT_XOFF - HF : -HF + ph) + a0, grow0 = FAM == 0 ? 0 : 4 * ph;
    constexpr int BASE = RL::AMAX - 1;                           // = MH / 2 lags per role; A0e = BASE + 1, A1e = A0o = A1o = BASE
    static_assert(BASE >= 1 && RL::A0e == BASE + 1 && RL::A1e == BASE && RL::A0o == BASE && RL::A1o == BASE, "role split");
    const int c0x = (FAM == 0 ? FT_XOFF - HF : -HF) + BASE;      // window offset of the shared lag (even phase, lag BASE)
    const float *grows_g = FAM == 0 ? p.gyrows : p.erows;
    const int i0 = FT_R * tid;

    float2 acc2[RL::AMAX][4];
#pragma unroll
    for (int a = 0; a < RL::AMAX; ++a)
#pragma unroll
        for (int k = 0; k < 4; ++k) acc2[a][k] = make_float2(0.f, 0.f);

    auto issue_tile = [&](int tile_i, int buf) {
        const int t0 = p.sym_lo + tile_i * FT_T, u0 = t0 - FT_HP + i0;
        const bool in_seq = (u0 >= 0) && (u0 < p.B);
        const bool owned = in_seq && (i0 >= FT_HP) && (i0 < FT_HP + FT_T) && (u0 < p.sym_hi);
        issue_g_rows<NG>(grows_g, p.B, u0, owned, grow + buf * NG * FT_GROW);
        if (FAM == 0) {
            issue_x_raw(p, t0, raw);                         // commits the group
        } else {
            if (in_seq) {
#pragma unroll
                for (int k = 0; k < 4; ++k) cp_async16(raw + k * FT_GROW + tid, p.m1rows + (int64_t)k * p.B + u0);
            } else {
#pragma unroll
                for (int k = 0; k < 4; ++k) raw[k * FT_GROW + tid] = make_float4(0.f, 0.f, 0.f, 0.f);
            }
            cp_async_commit();
        }
    };

    __shared__ int s_next;
    int buf = 0;
    if ((int)blockIdx.x < p.ntiles) issue_tile(blockIdx.x, 0);
    cp_async_wait_all();
    __syncthreads();
#pragma unroll 1
    for (int tile = blockIdx.x; tile < p.ntiles;) {
        const int t0 = p.sym_lo + tile * FT_T;
        tile_fetch_next(p, 2 + FAM, tile, &s_next);
        if (FAM == 0) {
            transpose_x_raw<true>(raw, s0, s1);
        } else {
            float4 mr[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) mr[k] = raw[k * FT_GROW + tid];
#pragma unroll
            for (int r = 0; r < FT_R; ++r) s0[5 * tid + r] = make_float4(f4c(mr[0], r), f4c(mr[2], r), f4c(mr[1], r), f4c(mr[3], r));   // swizzled window
        }
        __syncthreads();
        const int tile_next = s_next;
        if (tile_next < p.ntiles) issue_tile(tile_next, buf ^ 1);       // lands while this tile is correlated
        const float4 *gb = grow + (buf * NG + grow0) * FT_GROW;
#pragma unroll 1
        for (int g = (wid >> 2); g < FT_NW; g += FT_NW / 4) {
            const int l = g * 32 + lane;                     // thread-slot whose 4 symbols this lane processes
            const int li0 = FT_R * l, uu0 = t0 - FT_HP + li0;
            if (!((uu0 >= 0) && (uu0 < p.sym_hi) && (li0 >= FT_HP) && (li0 < FT_HP + FT_T))) continue;   // halo slots own nothing
            const float4 r0 = gb[l], r1 = gb[FT_GROW + l], r2 = gb[2 * FT_GROW + l], r3 = gb[3 * FT_GROW + l];
            const float4 gd[FT_R] = {make_float4(r0.x, r1.x, r2.x, r3.x), make_float4(r0.y, r1.y, r2.y, r3.y),
                                     make_float4(r0.z, r1.z, r2.z, r3.z), make_float4(r0.w, r1.w, r2.w, r3.w)};
            // every role correlates BASE = MH/2 lags of its phase; the one lag left over (even phase, lag BASE: 13 = 6 + 1 + 6 even taps at
            // M_est = 25) is shared out by symbol group, so all four roles do the same amount of work between two barriers
            corr4<BASE>(win, li0 + c0, gd, reinterpret_cast<float2(&)[BASE][4]>(acc2));
            if ((g & 3) == role) {
                if (FAM == 1 && ph) {                        // dh: the even-phase residual rows for the shared lag
                    const float4 *ge = grow + (buf * NG) * FT_GROW;
                    const float4 e0 = ge[l], e1 = ge[FT_GROW + l], e2 = ge[2 * FT_GROW + l], e3 = ge[3 * FT_GROW + l];
                    const float4 gx[FT_R] = {make_float4(e0.x, e1.x, e2.x, e3.x), make_float4(e0.y, e1.y, e2.y, e3.y),
                                             make_float4(e0.z, e1.z, e2.z, e3.z), make_float4(e0.w, e1.w, e2.w, e3.w)};
                    corr4<1>(s0, li0 + c0x, gx, reinterpret_cast<float2(&)[1][4]>(acc2[BASE]));
                } else {
                    corr4<1>(s0, li0 + c0x, gd, reinterpret_cast<float2(&)[1][4]>(acc2[BASE]));
                }
            }
        }
        cp_async_wait_all();
        __syncthreads();
        buf ^= 1;
        tile = tile_next;
    }

    // reduce over lanes, then over the two warps of a role, and publish this CTA's partial
    // acc[a][2(2o+i)+c]: c = 0 real, 1 imaginary part of output (o, i)
#pragma unroll
    for (int a = 0; a < RL::AMAX; ++a)
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const float2 v2 = acc2[a][2 * (k >> 2) + (k & 1)];
            const float s = warp_sum(((k >> 1) & 1) ? v2.y : v2.x);
            if (lane == 0) red[wid * (RL::AMAX * 8) + a * 8 + k] = s;
        }
    __syncthreads();
    if (wid < 4) {                                           // warps wid, wid+4, wid+8, ... share this role
        float *dst = p.gpart + (int64_t)blockIdx.x * 16 * M;
        for (int idx = lane; idx < n_real * 8; idx += 32) {
            const int a = idx >> 3, k = idx & 7, oi = k >> 1, cidx = k & 1, o = oi >> 1, i = oi & 1;
            float s = 0.f;
            if (a == BASE) {                                 // the shared lag (role 0 publishes it): partial sums of every warp, fixed order
#pragma unroll
                for (int w = 0; w < FT_NW; ++w) s += red[w * (RL::AMAX * 8) + idx];
            } else {
#pragma unroll
                for (int w = wid; w < FT_NW; w += 4) s += red[w * (RL::AMAX * 8) + idx];
            }
            const int lag = a0 + a;
            if (FAM == 1) dst[8 * M + ((o * 2 + i) * 2 + cidx) * M + (2 * MH - ph - 2 * lag)] = 2.f * p.scal[DP_KAPPA_OFF + o] * s;   // gD = 2 kappa_chi e
            else dst[(o * 4 + 2 * cidx + i) * M + (2 * lag + ph)] = s;
        }
    }
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
template <int MH>
static size_t fast_smem_fwd() {
    return (size_t)(2 * FT_XS + FT_ES + 2 * FT_TAPV * (2 * MH + 1) + FT_RAW) * sizeof(float4) + sizeof(FastConst) + 5 * 32 * sizeof(float) + 64;
}
template <int MH>
static size_t fast_smem_bwd1() {
    return (size_t)(2 * FT_ES + FT_TAPV * (2 * MH + 1) + 12 * FT_NT) * sizeof(float4) + sizeof(FastConst) + (2 * (2 * MH + 2) + 2) * sizeof(float) + 64;
}
template <int MH, int FAM>
static size_t fast_smem_taps() {
    return (size_t)(FAM == 0 ? 2 * FT_XS + FT_RAW + 2 * 4 * FT_GROW : FT_ES + 4 * FT_GROW + 2 * 8 * FT_GROW) * sizeof(float4) +
           FT_NW * Roles<MH>::AMAX * 8 * sizeof(float) + 64;
}

template <typename K>
static int fast_prepare(K kern, size_t smem, int *grid) {
    VAEQ_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per = 0;
    VAEQ_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per, kern, FT_NT, smem));
    *grid = max(1, per) * sm_count();
    return VAEQ_OK;
}

extern bool g_tc_taps, g_tc_fwd;
template <int NL, int MH>
static int dp_run_fast_t(DpK p, int mode, cudaStream_t st, int *grid_bwd_out) {
    static int grids[VAEQ_MAX_DEVICES][4] = {{0}};           // occupancy-derived grids and the shared-memory attribute are per device
    int &gF = grids[cur_device()][0], &g1 = grids[cur_device()][1], &g2 = grids[cur_device()][2], &g3 = grids[cur_device()][3];
    const size_t sf = fast_smem_fwd<MH>(), s1 = fast_smem_bwd1<MH>(), s2 = fast_smem_taps<MH, 0>(), s3 = fast_smem_taps<MH, 1>();
    if (!gF) {
        int rc;
        if ((rc = fast_prepare(k_dp_fwd_fast<NL, MH>, sf, &gF))) return rc;
        if ((rc = fast_prepare(k_dp_bwd1_fast<NL, MH>, s1, &g1))) return rc;
        if ((rc = fast_prepare(k_dp_taps_fast<MH, 0>, s2, &g2))) return rc;
        if ((rc = fast_prepare(k_dp_taps_fast<MH, 1>, s3, &g3))) return rc;
        g2 = g3 = min(g2, g3);                               // both write the same per-CTA partial slots
    }
    p.T = FT_T;
    p.keep_vec = p.qk != nullptr && p.keep_lo % 4 == 0 && p.keep_base % 4 == 0 && p.ld_qk % 4 == 0 && p.ld_outk % 4 == 0 &&
                 (reinterpret_cast<uintptr_t>(p.qk) | reinterpret_cast<uintptr_t>(p.outk)) % 16 == 0;
    const int nt_f = (p.chi - p.clo + FT_T - 1) / FT_T, nt_b = (p.sym_hi - p.sym_lo + FT_T - 1) / FT_T;
    const int gf = min(min(gF, DP_GRID_CAP), nt_f), gb1 = min(min(g1, DP_GRID_CAP), nt_b), gt = min(min(g2, DP_GRID_CAP), nt_b);
    if (mode != DP_MODE_SPLIT_BWD) {
        p.ntiles = nt_f;
        int nparts_f = gf, rc_f = VAEQ_OK;
        if (g_tc_fwd && dp_fwd_tc_launch(p, NL, st, &nparts_f, &rc_f)) {
            if (rc_f) return rc_f;
        } else {
            ktime_begin(VAEQ_K_DP_FWD, st);
            k_dp_fwd_fast<NL, MH><<<gf, FT_NT, sf, st>>>(p);
            ktime_end(VAEQ_K_DP_FWD, st);
            VAEQ_LAUNCH_CHECK("k_dp_fwd_fast");
        }
        *grid_bwd_out = nparts_f;                            // split forward: number of forward partials
        if (mode == DP_MODE_SPLIT_FWD) return VAEQ_OK;
        const int rc = dp_launch_fin(p, nparts_f, st);
        if (rc) return rc;
    }
    if (mode == DP_MODE_FWD) return VAEQ_OK;
    p.ntiles = nt_b;
    ktime_begin(VAEQ_K_DP_BWD, st);
    k_dp_bwd1_fast<NL, MH><<<gb1, FT_NT, s1, st>>>(p);
    ktime_end(VAEQ_K_DP_BWD, st);
    VAEQ_LAUNCH_CHECK("k_dp_bwd1_fast");
    if (g_tc_taps) {
        int rc = VAEQ_OK;
        if (dp_taps_tc_launch(p, st, grid_bwd_out, &rc)) return rc;
    }
    ktime_begin(VAEQ_K_DP_BWD2, st);
    k_dp_taps_fast<MH, 0><<<gt, FT_NT, s2, st>>>(p);
    ktime_end(VAEQ_K_DP_BWD2, st);
    VAEQ_LAUNCH_CHECK("k_dp_taps_fast<W>");
    ktime_begin(VAEQ_K_DP_BWD3, st);
    k_dp_taps_fast<MH, 1><<<gt, FT_NT, s3, st>>>(p);
    ktime_end(VAEQ_K_DP_BWD3, st);
    VAEQ_LAUNCH_CHECK("k_dp_taps_fast<h>");
    *grid_bwd_out = gt;
    return VAEQ_OK;
}

bool g_tc_fwd = true;       // forward kernel with the FIR and the channel convolution on tcgen05 (dp_fwd_tc.cu), default since r02c: with the moment-form
                            // demapper and the magnitude-ordered MMAs it is faster than k_dp_fwd_fast (244 vs 257 us) at a smaller output error
                            // (profiles/r02c_tc_forward.txt); vaeq_dp_tc_forward(0) selects k_dp_fwd_fast, which also serves every (n_lev, M_est)
                            // the tensor-core kernel is not built for

bool g_tc_taps = true;      // both tap-gradient correlations on tcgen05 (dp_taps_tc.cu); false = the two CUDA-core correlation kernels

// returns 1 if the fast path ran (and *grid_bwd_out is the number of gradient partials), 0 if not applicable
int dp_try_fast(const DpK &p, int n_lev, int mode, cudaStream_t st, int *grid_bwd_out, int *rc) {
    const bool no_q = p.q == nullptr;                        // frame loops of the batch-split: only the kept columns are wanted
    const bool aligned = (p.B % 4 == 0) && (p.ld_rx % 4 == 0) && (no_q || ((p.ld_q % 4 == 0) && (p.ld_out % 4 == 0))) &&
                         ((reinterpret_cast<uintptr_t>(p.rx) | reinterpret_cast<uintptr_t>(p.q) | reinterpret_cast<uintptr_t>(p.out)) % 16 == 0);
    if (!aligned || p.B < 2 * FT_T) return 0;                // small batches: the generic kernels (one tile) are as good
    if ((p.sym_lo | p.sym_hi | p.clo | p.chi) % 4 != 0) return 0;
    *rc = VAEQ_OK;
#define FAST_CASE(NL_, MH_)                                             \
    if (n_lev == NL_ && p.mh == MH_) {                                  \
        *rc = dp_run_fast_t<NL_, MH_>(p, mode, st, grid_bwd_out);       \
        return 1;                                                       \
    }
    FAST_CASE(8, 12)
    FAST_CASE(8, 6)
    FAST_CASE(8, 4)
    FAST_CASE(8, 2)
    FAST_CASE(4, 12)
    FAST_CASE(2, 12)
#undef FAST_CASE
    return 0;
}

}  // namespace vaeq

extern "C" int vaeq_dp_tc_forward(int32_t on) {
    vaeq::g_tc_fwd = on != 0;
    return VAEQ_OK;
}

extern "C" int vaeq_dp_tc_taps(int32_t on) {
    if (on != 0 && on != 1) {
        vaeq::set_error("vaeq_dp_tc_taps: %d is not 0 (CUDA-core kernels) or 1 (tensor cores)", on);
        return VAEQ_EINVAL;
    }
    vaeq::g_tc_taps = on != 0;
    return VAEQ_OK;
}
