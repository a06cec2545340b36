// DP VAE step for REFERENCE-SIZE minibatches (batch_len <= 512; Eval_run_DP.py:38 uses 100): persistent frame kernel.
//
// At batch_len = 100 one training step is ~0.5 MFLOP: launched as separate kernels a frame of 100-990 sequential steps
// (func_VAELE_DP_MQAM_shaping.py:57-66, func_VAEflex_DP_MQAM_shaping.py:59-70) is pure launch + global-memory latency.
// Here ONE CTA owns one run for the whole frame:
//   * taps W, channel estimate h, Adam moments and every per-step intermediate (E_q, backward coefficients, residual e,
//     dL/dout, partial sums) live in SHARED MEMORY across all steps; global traffic per step is the rx window in and
//     the kept columns of q / out (+ loss, var_est) out;
//   * the step is a sequence of CTA phases separated by __syncthreads(): FIR over (symbol, output pol) items, soft
//     demapper over (symbol, component) items (ex2/lg2/rcp math of dp_math.cuh, which also yields the backward
//     coefficients S1,T2,S3 so the backward needs no q and no transcendental), channel convolution + residual over
//     (sample, rx pol) items, scalar ELBO assembly, dL/dE_q + dL/dout, the two tap-gradient correlations, Adam;
//   * blockIdx.x = run: independent runs (the sweep cells of Eval_run_DP.py:68-95) are batched in the same launch, one
//     CTA each, 3-4 CTAs per SM.
// Same math as dp_step.cu / dp_fast.cu (closed form restated in oracle/closed_form.py); any odd M_est <= 63.
#include "dp_math.cuh"
#include "dp_kernels.cuh"

namespace vaeq {

// block_sum (common.cuh) with the final reduction on the LAST warp of the CTA: totals valid in all its lanes; ONE barrier (the caller
// uses the scratch once per step)
template <int NV>
__device__ __forceinline__ void block_sum_last(float (&v)[NV], float *scratch) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
#pragma unroll
    for (int i = 0; i < NV; ++i) v[i] = warp_sum(v[i]);
    if (lane == 0) {                                         // no barrier before the stores: the scratch was last read a whole step (ten barriers) ago
#pragma unroll
        for (int i = 0; i < NV; ++i) scratch[i * 32 + wid] = v[i];
    }
    __syncthreads();
    if (wid == nw - 1) {
#pragma unroll
        for (int i = 0; i < NV; ++i) {
            const float x = lane < nw ? scratch[i * 32 + lane] : 0.f;
            v[i] = warp_sum(x);
        }
    }
}

__device__ __forceinline__ float fneg(float v) { return __uint_as_float(__float_as_uint(v) ^ 0x80000000u); }   // sign flip as an integer op

constexpr int SM_NT = 256;

// shared-memory plan (offsets in floats); doubles first (8-byte aligned), then float4 arrays, then floats
struct SmallLayout {
    int XA, XO, SA, SO;                     // phase-array lengths (float4) and zero margins of x and e
    int dsc, xph, m1s, eph, gys, Wt, hD, hG, part4, cst, srow, vsc, PS, Asum, edge, Wf, hf, adam, gfin, hsq, red, scal, total;
};
__host__ __device__ inline SmallLayout small_layout(int B, int M) {
    SmallLayout l;
    const int mh = M / 2;
    l.XO = (mh + 1) / 2 + 1;
    l.XA = B + 2 * l.XO;
    l.SO = (mh + 1) / 2 + 1;
    l.SA = B + 2 * l.SO;
    int off = 0;
    auto take = [&](int nfloats) {
        int o = off;
        off += (nfloats + 3) & ~3;          // keep 16-byte alignment throughout
        return o;
    };
    l.dsc = take(2 * 4);                    // doubles: bc1 (Adam bias correction)
    l.xph = take(2 * 4 * 2 * l.XA);         // double-buffered: the next step's window lands by cp.async during this step
    l.m1s = take(4 * B);
    l.eph = take(4 * 2 * l.SA);
    l.gys = take(4 * B);
    l.Wt = take(4 * 2 * M);
    l.hD = take(4 * 2 * M);
    l.hG = take(4 * 2 * M);
    l.part4 = take(4 * 3 * SM_NT);          // chunk partials of the tap gradients: dW 128 x 4 float4, dh 128 x 2 float4
    l.cst = take((int)(sizeof(FastConst) / 4));
    l.srow = take(12 * B);
    l.vsc = take(4 * B);
    l.PS = take(4 * (M + 1));
    l.Asum = take(4);
    l.edge = take(2 * M);
    l.Wf = take(8 * M);
    l.hf = take(8 * M);
    l.adam = take(48 * M);
    l.gfin = take(16 * M);
    l.hsq = take(4 * M);
    l.red = take(7 * 32);
    l.scal = take(8);
    l.total = off;
    return l;
}

__device__ __forceinline__ void cp_async4(void *dst_smem, const void *src_gmem) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(dst_smem);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(d), "l"(src_gmem) : "memory");
}

constexpr int SM_MINB = 3;   // 3 CTAs (runs) per SM; 98 registers uncapped = 2 CTAs, 64 = 4 CTAs with spills (profiles/r01b_experiments.txt)
// MINB = 3 (80 registers) is the faster kernel per run; MINB = 4 (64 registers, a few spills) is launched when a fourth run per SM saves a
// whole wave of CTAs (e.g. 592 runs on 148 SMs: 444 + a tail of 148 at 3 per SM, one wave at 4 per SM), see dp_small_launch
// MT: M_est at compile time (0 = run time): the tap loops then have constant trip counts and immediate offsets (the kernel is issue-bound:
// 66 % issue-active with a quarter of its instructions integer / address arithmetic, profiles/r02_ncu_misc_summary.md)
template <int NL, int MINB, int MT>
__global__ void __launch_bounds__(SM_NT, MINB) k_dp_frame_fast(DpK p, DpRunsK rs, int n_steps, int stride_sym, int keep_lo_in_dst,
                                                         float lr_w, float lr_h, int amsgrad) {
    extern __shared__ __align__(16) float sm[];
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int B = p.B, L = 2 * p.B, M = MT ? MT : p.M, mh = M / 2, Mh = 2 * mh, run = blockIdx.x;
    const SmallLayout lay = small_layout(B, M);
    const int XA = lay.XA, XO = lay.XO, SA = lay.SA, SO = lay.SO;
    double *dsc = reinterpret_cast<double *>(sm + lay.dsc);
    float4 *xph2 = reinterpret_cast<float4 *>(sm + lay.xph);     // [2 buffers][2 phases][XA]  rx {I0,I1,Q0,Q1}: [ph][a+XO] = rx[:, 2a+ph]
    float4 *m1s = reinterpret_cast<float4 *>(sm + lay.m1s);      // [B]      E_q[x] {p0 I, p1 I, p0 Q, p1 Q}
    float4 *eph = reinterpret_cast<float4 *>(sm + lay.eph);      // [2][SA]  residual D - rx {chi0 re, chi1 re, chi0 im, chi1 im} by sample phase
    float4 *gys = reinterpret_cast<float4 *>(sm + lay.gys);      // [B]      dL/dout
    // every window / table element is {re of both partners, im of both partners}: one fma.rn.f32x2 updates the (partner 0, partner 1) pair
    // of an accumulator, and the per-accumulator operation order is the scalar kernel's (bit-identical results)
    float4 *Wt = reinterpret_cast<float4 *>(sm + lay.Wt);        // [o][k]   {wr<-p0, wr<-p1, wi<-p0, wi<-p1}
    float4 *hD = reinterpret_cast<float4 *>(sm + lay.hD);        // [chi][j] {h_chi,0 re, h_chi,1 re, h_chi,0 im, h_chi,1 im}
    float4 *hG = reinterpret_cast<float4 *>(sm + lay.hG);        // [nu][j]  {h_0,nu re, h_1,nu re, h_0,nu im, h_1,nu im}   (kappa applied at use)
    float4 *part4 = reinterpret_cast<float4 *>(sm + lay.part4);
    FastConst *cst = reinterpret_cast<FastConst *>(sm + lay.cst);
    float *srow = sm + lay.srow, *vsc = sm + lay.vsc, *PS = sm + lay.PS, *Asum = sm + lay.Asum, *edge = sm + lay.edge;
    float *Wf = sm + lay.Wf, *hf = sm + lay.hf, *ad = sm + lay.adam, *gfin = sm + lay.gfin, *hsq = sm + lay.hsq, *red = sm + lay.red;
    float *scal = sm + lay.scal;

    // ---- this run's tensors (blockIdx.x = run) ---------------------------------------------------------------------
    const float *rx0 = p.rx + run * rs.rs_rx;
    float *Wg = p.W + run * rs.rs_W, *hg = p.h + run * rs.rs_h, *adg = p.adam + run * rs.rs_adam;
    float *qk = p.qk ? p.qk + run * rs.rs_qk : nullptr, *outk = p.qk ? p.outk + run * rs.rs_outk : nullptr;
    if (rs.lr_w) lr_w = rs.lr_w[run];
    if (rs.lr_h) lr_h = rs.lr_h[run];
    const float nu_sc = rs.nu_sc ? rs.nu_sc[run] : p.nu_sc;

    // the rx window of step m -> phase arrays of buffer m & 1: 4-byte cp.async scatter (4 rows -> one float4 per position);
    // positions outside [0, L) are the FIR's zero padding, the same in every step: zeroed once below
    auto issue_window = [&](int m) {
        const float *rx = rx0 + (int64_t)m * stride_sym * 2;
        float4 *dst = xph2 + (m & 1) * 2 * XA;
        for (int idx = tid; idx < 2 * XA; idx += SM_NT) {
            const int ph = idx >= XA, a = idx - ph * XA - XO, s = 2 * a + ph;
            if (s >= 0 && s < L) {
                float *d4 = reinterpret_cast<float *>(dst + idx);
#pragma unroll
                for (int r = 0; r < 4; ++r) cp_async4(d4 + ((r & 1) * 2 + (r >> 1)), rx + r * p.ld_rx + s);      // rows p0 I, p0 Q, p1 I, p1 Q -> {I0, I1, Q0, Q1}
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };

    for (int i = tid; i < 8 * M; i += SM_NT) {
        Wf[i] = Wg[i];
        hf[i] = hg[i];
    }
    for (int i = tid; i < 48 * M; i += SM_NT) ad[i] = adg[i];
    for (int i = tid; i < 2 * SA; i += SM_NT) eph[i] = make_float4(0.f, 0.f, 0.f, 0.f);     // margins stay zero for the whole frame
    for (int i = tid; i < 4 * XA; i += SM_NT) xph2[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    load_fast_const(cst, p.amp + run * rs.rs_amp, p.P + run * rs.rs_P, p.var + run * rs.rs_var, nu_sc, NL);
    const int step0 = *reinterpret_cast<const int *>(adg + 48 * M);
    const double width = (double)(L - Mh);
    double b1t = 1.0, b2t = 1.0;                             // beta1^t, beta2^t at the step count the frame starts from
    if (tid == 0) {
        b1t = pow(0.9, (double)step0);
        b2t = pow(0.999, (double)step0);
    }
    __syncthreads();
    if (n_steps > 0) issue_window(0);
    const FastConst &c = *cst;

    for (int m = 0; m < n_steps; ++m) {
        const int64_t keep_base = (int64_t)m * stride_sym + (keep_lo_in_dst ? p.keep_lo : 0);
        const bool last = m == n_steps - 1;
        const float4 *xph = xph2 + (m & 1) * 2 * XA;

        // ---- P0: tap tables from the master copies; |h|^2, its prefix sums over the taps and totals (warp scans) -----------
        for (int idx = tid; idx < 2 * M; idx += SM_NT) {
            const int o = idx / M, k = idx - o * M;
            Wt[idx] = make_float4(Wf[(o * 4 + 0) * M + k], Wf[(o * 4 + 1) * M + k], Wf[(o * 4 + 2) * M + k], Wf[(o * 4 + 3) * M + k]);
            hD[idx] = make_float4(hf[((o * 2 + 0) * 2 + 0) * M + k], hf[((o * 2 + 1) * 2 + 0) * M + k],
                                  hf[((o * 2 + 0) * 2 + 1) * M + k], hf[((o * 2 + 1) * 2 + 1) * M + k]);
            hG[idx] = make_float4(hf[((0 * 2 + o) * 2 + 0) * M + k], hf[((1 * 2 + o) * 2 + 0) * M + k],
                                  hf[((0 * 2 + o) * 2 + 1) * M + k], hf[((1 * 2 + o) * 2 + 1) * M + k]);
        }
        if (tid == 0) {                                      // Adam bias corrections 1 - beta^t: running products (pow once per frame)
            b1t *= 0.9;
            b2t *= 0.999;
            dsc[0] = 1.0 - b1t;
            scal[6] = sqrtf((float)(1.0 - b2t));
        }
        asm volatile("cp.async.wait_group 0;" ::: "memory");      // this step's window (issued during the previous step)
        __syncthreads();
        if (!last) issue_window(m + 1);                      // lands in the other buffer while this step computes
        // |h|^2 and its prefix sums (used from P3 / P4 on) by warps 4-7 AFTER the barrier: they run next to the FIR of warps 0-3 instead of
        // holding every warp at the top of the step
        if (wid >= 4) {                                      // warp 4 + cn: PS[cn][j] = sum_{j' < j} |h_cn,j'|^2, cn = chi * 2 + nu
            const int cn = wid - 4;
            float carry = 0.f;
            if (lane == 0) PS[cn * (M + 1)] = 0.f;
            for (int j0 = 0; j0 < M; j0 += 32) {
                const int j = j0 + lane;
                float v = 0.f;
                if (j < M) {
                    const float hr = hf[(cn * 2 + 0) * M + j], hi = hf[(cn * 2 + 1) * M + j];
                    v = hr * hr + hi * hi;
                    hsq[cn * M + j] = v;
                }
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const float t = __shfl_up_sync(0xffffffffu, v, o);
                    if (lane >= o) v += t;
                }
                v += carry;
                if (j < M) PS[cn * (M + 1) + j + 1] = v;
                carry = __shfl_sync(0xffffffffu, v, 31);
            }
            if (lane == 0) Asum[cn] = carry;
        }

        // ---- P1: butterfly FIR (sf:500-518) + soft demapper, moments, entropy, backward coefficients (sf:511-523, 101-113):
        //      one (symbol, output pol) item per thread, its two components demapped right away ------------------------------
        float accEnt = 0.f, accV0 = 0.f, accV1 = 0.f;
        // FIR: one SYMBOL per item, both output polarisations (the sample-window element of a lag is loaded once for the two of them: the
        // kernel is shared-memory-bandwidth bound); the four outputs go through the dL/dout buffer (dead until P5) to the demapper items
        for (int u = tid; u < B; u += SM_NT) {
            const float2 z2 = make_float2(0.f, 0.f);
            float2 re0 = z2, im0 = z2, re1 = z2, im1 = z2;       // (contribution of input pol 0, of input pol 1) for o = 0 / 1
#pragma unroll
            for (int ph = 0; ph < 2; ++ph) {
                const int k0 = (mh + ph) & 1;                    // taps k = k0, k0+2, ... read samples of phase ph
                const float4 *xb = xph + ph * XA + u + XO + ((k0 - mh - ph) >> 1);
                const float4 *wb0 = Wt + k0, *wb1 = Wt + M + k0;
                const int n = (M - k0 + 1) >> 1;
#pragma unroll 4
                for (int i = 0; i < n; ++i) {
                    const float4 x = xb[i], wa = wb0[2 * i], wc = wb1[2 * i];
                    const float2 xI = make_float2(x.x, x.y), xQ = make_float2(x.z, x.w), nxQ = make_float2(fneg(x.z), fneg(x.w));   // (-wi) xQ = wi (-xQ) bit for bit:
                    const float2 ar = make_float2(wa.x, wa.y), ai = make_float2(wa.z, wa.w), cr = make_float2(wc.x, wc.y), ci = make_float2(wc.z, wc.w);   // FFMA2 negates for free
                    re0 = __ffma2_rn(ar, xI, re0); re0 = __ffma2_rn(ai, nxQ, re0);
                    im0 = __ffma2_rn(ar, xQ, im0); im0 = __ffma2_rn(ai, xI, im0);
                    re1 = __ffma2_rn(cr, xI, re1); re1 = __ffma2_rn(ci, nxQ, re1);
                    im1 = __ffma2_rn(cr, xQ, im1); im1 = __ffma2_rn(ci, xI, im1);
                }
            }
            gys[u] = make_float4(re0.x + re0.y, im0.x + im0.y, re1.x + re1.y, im1.x + im1.y);
        }
        __syncthreads();
        for (int it = tid; it < 2 * B; it += SM_NT) {
            const int o = it >= B, u = it - o * B;
            const float2 y2 = reinterpret_cast<const float2 *>(gys + u)[o];
            const float yc[2] = {y2.x, y2.y};
            const bool keep = qk != nullptr && u >= p.keep_lo && u < p.keep_lo + p.keep_n;      // VAELE_DP:61-62 / VAEflex_DP:64-65
            const int64_t col = keep_base + (u - p.keep_lo);
            float vsum = 0.f;
#pragma unroll
            for (int cq = 0; cq < 2; ++cq) {
                const int cc = 2 * o + cq;
                float q[NL], m1, m2, ent, S1, S2, S3;
                demap_fast<NL, true>(yc[cq], c.c2[o], c.inv_var[o], c, q, m1, m2, ent, S1, S2, S3);
                if (keep) {
#pragma unroll
                    for (int l = 0; l < NL; ++l) qk[(int64_t)(cc * NL + l) * p.ld_qk + col] = q[l];
                    outk[(int64_t)cc * p.ld_outk + col] = yc[cq];
                }
                reinterpret_cast<float *>(m1s + u)[cq * 2 + o] = m1;
                srow[cc * B + u] = S1;
                srow[(4 + cc) * B + u] = fmaf(-2.f * m1, S1, S2);
                srow[(8 + cc) * B + u] = S3;
                vsum += m2 - m1 * m1;                                                    // sf:113
                if (u >= mh && u < B - mh) accEnt += ent;                                // sf:132: [mh:-mh] in SYMBOLS
            }
            vsc[o * B + u] = vsum;                                                       // Var_I + Var_Q of pol o
            if (o) accV1 += vsum; else accV0 += vsum;
        }
        __syncthreads();

        // ---- P3: D = h * E_q on the valid samples, residual e = D - rx (sf:115-134), one (sample, rx pol) item per thread;
        //      then the edge sums of S_nu(j) = V_nu - edge_nu(j) (Var over source symbols outside Mh <= 2u+j < L, sf:128) --------
        float accC0 = 0.f, accC1 = 0.f;
        for (int s = tid; s < L; s += SM_NT) {                   // one SAMPLE per item, both rx polarisations: the E_q window element of a lag is
            float er0 = 0.f, ei0 = 0.f, er1 = 0.f, ei1 = 0.f;    // loaded once for the two of them (the kernel is shared-memory-bandwidth bound)
            if (s >= mh && s < L - mh) {                                             // sf:120 "valid", in SAMPLES
                const float2 z2 = make_float2(0.f, 0.f);
                float2 dr0 = z2, di0 = z2, dr1 = z2, di1 = z2;   // (contribution of tx pol 0, of tx pol 1) for chi = 0 / 1
                const int par = (s + mh) & 1;
                const float4 *hb0 = hD + par, *hb1 = hD + M + par;
                const float4 *mb = m1s + ((s + mh - par) >> 1);                       // E_q[(s + mh - j)/2], j = par + 2i
                const int n = (M - par + 1) >> 1;
#pragma unroll 4
                for (int i = 0; i < n; ++i) {
                    const float4 mm = mb[-i], ha = hb0[2 * i], hc = hb1[2 * i];
                    const float2 mI = make_float2(mm.x, mm.y), mQ = make_float2(mm.z, mm.w), nmQ = make_float2(fneg(mm.z), fneg(mm.w));
                    const float2 ar = make_float2(ha.x, ha.y), ai = make_float2(ha.z, ha.w), cr = make_float2(hc.x, hc.y), ci = make_float2(hc.z, hc.w);
                    dr0 = __ffma2_rn(ar, mI, dr0); dr0 = __ffma2_rn(ai, nmQ, dr0);
                    di0 = __ffma2_rn(ai, mI, di0); di0 = __ffma2_rn(ar, mQ, di0);
                    dr1 = __ffma2_rn(cr, mI, dr1); dr1 = __ffma2_rn(ci, nmQ, dr1);
                    di1 = __ffma2_rn(ci, mI, di1); di1 = __ffma2_rn(cr, mQ, di1);
                }
                const float4 x = xph[(s & 1) * XA + (s >> 1) + XO];
                er0 = (dr0.x + dr0.y) - x.x;
                ei0 = (di0.x + di0.y) - x.z;
                er1 = (dr1.x + dr1.y) - x.y;
                ei1 = (di1.x + di1.y) - x.w;
            }
            eph[(s & 1) * SA + (s >> 1) + SO] = make_float4(er0, er1, ei0, ei1);      // {chi0 re, chi1 re, chi0 im, chi1 im}
            accC0 += er0 * er0 + ei0 * ei0;
            accC1 += er1 * er1 + ei1 * ei1;
        }
        float accB0 = 0.f, accB1 = 0.f;                          // sum_{nu,j} |h_chi,nu,j|^2 edge_nu(j); on the LAST 2M threads,
        for (int idx = tid - (SM_NT - 2 * M); idx >= 0 && idx < 2 * M; idx += SM_NT) {      // which have the fewest D items above
            const int nu = idx / M, j = idx - nu * M;
            const int u_lo = (Mh - j + 1) >> 1, u_hi = (L - 1 - j) >> 1;
            float ed = 0.f;
            for (int u = 0; u < u_lo && u < B; ++u) ed += vsc[nu * B + u];
            for (int u = u_hi + 1; u < B; ++u) ed += vsc[nu * B + u];
            edge[idx] = ed;
            accB0 += hsq[idx] * ed;
            accB1 += hsq[2 * M + idx] * ed;
        }

        // ---- P4: ELBO scalars (sf:131-137): C = sum|e|^2 + sum_nu V_nu A_chi,nu - B_chi, loss, var_est, kappa = (L-Mh)/C ---------
        {
            float v[7] = {accC0, accC1, accEnt, accV0, accV1, accB0, accB1};
            block_sum_last<7>(v, red);                           // its barriers also publish eph and edge; totals in ALL lanes of the LAST warp, which has
            if (wid == SM_NT / 32 - 1 && lane < 2) {             // no P5 item at the reference's batch_len: its two double-precision logs overlap the contraction below
                const int chi = lane;
                const float vC = chi ? v[1] : v[0], vB = chi ? v[6] : v[5], vV = chi ? v[4] : v[3];   // selects, not v[chi]: a run-time index would put
                const double C = (double)vC + ((double)v[3] * (double)Asum[chi * 2] + (double)v[4] * (double)Asum[chi * 2 + 1]) -   // the whole array in local memory
                                 (double)vB;                                         // sf:133-134
                const double term = width * log(C);                                  // sf:136
                scal[chi] = (float)(width / C);                                      // kappa
                scal[2 + chi] = vV;                                                  // V_nu, for S_nu(j) in the Adam phase
                const float ve = (float)(C / width);                                 // sf:137
                if (rs.var_steps) rs.var_steps[((int64_t)run * 2 + chi) * n_steps + m] = ve;
                if (last && rs.var_last) rs.var_last[2 * run + chi] = ve;
                const double term1 = __shfl_sync(0x3u, term, 1);
                if (chi == 0) {
                    const float loss = (float)((-(double)v[2] + term) + term1);
                    if (rs.loss_steps) rs.loss_steps[(int64_t)run * n_steps + m] = loss;
                    if (last && rs.loss_last) rs.loss_last[run] = loss;
                }
            }
        }
        // ---- P5: dL/dE_q = conj(h) (*) gD with gD = 2 kappa_chi e, then dL/dout = dL/dE_q S1 + dL/dVar T2 + w S3;
        //      one symbol (both tx pols) per thread.  The contraction over e does not need kappa (it is linear in kappa_chi, applied after the
        //      sum), so with one item per thread (batch_len <= 256) it runs BEFORE the barrier that publishes kappa, while the last warp
        //      is still at the logs of the ELBO scalars -----------------------------------------------------------------------
        const float2 z2 = make_float2(0.f, 0.f);
        float2 gr0 = z2, gi0 = z2, gr1 = z2, gi1 = z2;           // (chi = 0 terms, chi = 1 terms) for nu = 0 / 1
        auto contract = [&](int u) {
            gr0 = gi0 = gr1 = gi1 = z2;
#pragma unroll
            for (int ph = 0; ph < 2; ++ph) {
                const int j0 = (mh + ph) & 1;                    // gD sample 2u - mh + j has phase ph for j = j0, j0+2, ...
                const float4 *eb = eph + ph * SA + u + SO + ((j0 - mh - ph) >> 1);
                const float4 *hb0 = hG + j0, *hb1 = hG + M + j0;
                const int n = (M - j0 + 1) >> 1;
#pragma unroll 4
                for (int i = 0; i < n; ++i) {
                    const float4 e = eb[i], ha = hb0[2 * i], hc = hb1[2 * i];
                    const float2 eR = make_float2(e.x, e.y), eI = make_float2(e.z, e.w), neR = make_float2(fneg(e.x), fneg(e.y));
                    const float2 ar = make_float2(ha.x, ha.y), ai = make_float2(ha.z, ha.w), cr = make_float2(hc.x, hc.y), ci = make_float2(hc.z, hc.w);
                    gr0 = __ffma2_rn(ar, eR, gr0); gr0 = __ffma2_rn(ai, eI, gr0);
                    gi0 = __ffma2_rn(ar, eI, gi0); gi0 = __ffma2_rn(ai, neR, gi0);
                    gr1 = __ffma2_rn(cr, eR, gr1); gr1 = __ffma2_rn(ci, eI, gr1);
                    gi1 = __ffma2_rn(cr, eI, gi1); gi1 = __ffma2_rn(ci, neR, gi1);
                }
            }
        };
        const bool one_item = B <= SM_NT;
        if (one_item && tid < B) contract(tid);
        __syncthreads();
        const float kap0 = scal[0], kap1 = scal[1];

        for (int u = tid; u < B; u += SM_NT) {
            if (!one_item) contract(u);
            const int jlo = max(0, Mh - 2 * u), jhi = min(M, L - 2 * u);
            const float entw = (u >= mh && u < B - mh) ? LN2 : 0.f;
            float g4[4];
#pragma unroll
            for (int nu = 0; nu < 2; ++nu) {
                const float2 gr2 = nu ? gr1 : gr0, gi2 = nu ? gi1 : gi0;
                const float gr = 2.f * (kap0 * gr2.x + kap1 * gr2.y), gi = 2.f * (kap0 * gi2.x + kap1 * gi2.y);
                const float gV = kap0 * (PS[(0 * 2 + nu) * (M + 1) + jhi] - PS[(0 * 2 + nu) * (M + 1) + jlo]) +
                                 kap1 * (PS[(1 * 2 + nu) * (M + 1) + jhi] - PS[(1 * 2 + nu) * (M + 1) + jlo]);
                const int cc = 2 * nu;
                g4[2 * nu] = fmaf(gr, srow[cc * B + u], fmaf(gV, srow[(4 + cc) * B + u], entw * srow[(8 + cc) * B + u]));
                g4[2 * nu + 1] = fmaf(gi, srow[(cc + 1) * B + u], fmaf(gV, srow[(5 + cc) * B + u], entw * srow[(9 + cc) * B + u]));
            }
            gys[u] = make_float4(g4[0], g4[1], g4[2], g4[3]);
        }
        __syncthreads();

        // ---- P6: tap gradients.  Warps 0-3: dW[o=0,1][in][k] = sum_u gy_o(u) conj(x_in[2u+k-mh]); warps 4-7:
        //      dh[chi=0,1][nu][j] = 2 kappa_chi sum_v e_chi(2v+j-mh) conj(E_q,nu[v]) (warp-uniform roles).  A thread owns a PAIR of
        //      neighbouring taps of one sample phase (k, k+2): their windows are one position apart, so one LDS.128 of the window
        //      and one broadcast of the per-symbol operand feed 16 FMA (the phase was shared-memory-bandwidth bound with one tap
        //      per thread).  The symbol range is cut into `parts` chunks so that all 128 threads of a family work; partials are
        //      summed in fixed order (deterministic).
        {
            const int kf0 = mh & 1, kf1 = (mh + 1) & 1;                               // first tap of phase 0 / 1
            const int np0 = (((M - kf0 + 1) >> 1) + 1) >> 1, np1 = (((M - kf1 + 1) >> 1) + 1) >> 1, nps = np0 + np1;
            const int fam = wid >> 2, ft = tid & 127;
            // dW: an item = a tap pair, BOTH input polarisations at once (the window element {I0, I1, Q0, Q1} is the packed operand);
            // dh: an item = (tx pol, tap pair), both rx polarisations chi at once (window element {re0, re1, im0, im1})
            // Lane mapping: lanes 2i, 2i + 1 share an item and take NEIGHBOURING parts, and the chunk length is odd.  The window positions a
            // quarter-warp's LDS.128 touches are then 2 q + {0, chunk} for four consecutive tap pairs q: eight distinct residues mod 8, i.e.
            // no bank conflict (with lanes = consecutive items the positions 0, 2, ..., 14 collided two by two: 2.7 x the ideal wavefronts
            // in this shared-memory-bound kernel, profiles/r02b_frame_kernel.txt).
            const int items = fam == 0 ? nps : 2 * nps, parts = max(2, 2 * (64 / items)), chunk = ((B + parts - 1) / parts) | 1;
            float4 *pbase = part4 + (fam == 0 ? 0 : 4 * 128);
            if ((ft >> 1) < items * (parts >> 1)) {
                const int item = (ft >> 1) % items, part = 2 * ((ft >> 1) / items) + (ft & 1);
                const int sel = fam == 0 ? 0 : item / nps, q = item - sel * nps, ph = q >= np0, kA = (ph ? kf1 : kf0) + 4 * (ph ? q - np0 : q);
                const int u0 = min(B, part * chunk), u1 = min(B, u0 + chunk), off = (kA - mh - ph) >> 1;
                const float2 z2 = make_float2(0.f, 0.f);
                if (fam == 0) {                                  // f = dL/dout {o0 re, im, o1 re, im}; window = rx of both input pols
                    float2 a0r = z2, a0i = z2, a1r = z2, a1i = z2, b0r = z2, b0i = z2, b1r = z2, b1i = z2;     // (input pol 0, input pol 1)
                    const float4 *wb = xph + ph * XA + XO + off;
                    float4 wa = wb[u0];
#pragma unroll 2
                    for (int u = u0; u < u1; ++u) {
                        const float4 wn = wb[u + 1];
                        const float4 f = gys[u];
                        const float2 fx = make_float2(f.x, f.x), fy = make_float2(f.y, f.y), fz = make_float2(f.z, f.z), fw = make_float2(f.w, f.w);
                        const float2 nfx = make_float2(-f.x, -f.x), nfz = make_float2(-f.z, -f.z);
                        const float2 aI = make_float2(wa.x, wa.y), aQ = make_float2(wa.z, wa.w), nI = make_float2(wn.x, wn.y), nQ = make_float2(wn.z, wn.w);
                        a0r = __ffma2_rn(fx, aI, a0r); a0r = __ffma2_rn(fy, aQ, a0r); a0i = __ffma2_rn(fy, aI, a0i); a0i = __ffma2_rn(nfx, aQ, a0i);
                        a1r = __ffma2_rn(fz, aI, a1r); a1r = __ffma2_rn(fw, aQ, a1r); a1i = __ffma2_rn(fw, aI, a1i); a1i = __ffma2_rn(nfz, aQ, a1i);
                        b0r = __ffma2_rn(fx, nI, b0r); b0r = __ffma2_rn(fy, nQ, b0r); b0i = __ffma2_rn(fy, nI, b0i); b0i = __ffma2_rn(nfx, nQ, b0i);
                        b1r = __ffma2_rn(fz, nI, b1r); b1r = __ffma2_rn(fw, nQ, b1r); b1i = __ffma2_rn(fw, nI, b1i); b1i = __ffma2_rn(nfz, nQ, b1i);
                        wa = wn;
                    }
                    float4 *dst = pbase + ft;                                // [slot = tap of the pair x input pol][thread] -> {o0 re, o0 im, o1 re, o1 im}
                    dst[0] = make_float4(a0r.x, a0i.x, a1r.x, a1i.x);        // (slot-major: consecutive lanes store consecutive float4)
                    dst[128] = make_float4(a0r.y, a0i.y, a1r.y, a1i.y);
                    dst[256] = make_float4(b0r.x, b0i.x, b1r.x, b1i.x);
                    dst[384] = make_float4(b0r.y, b0i.y, b1r.y, b1i.y);
                } else {                                         // window = residual e {chi0 re, chi1 re, chi0 im, chi1 im}; f = E_q of tx pol sel
                    float2 ar = z2, ai = z2, br = z2, bi = z2;                  // (chi 0, chi 1)
                    const float4 *wb = eph + ph * SA + SO + off;
                    const float *fb = reinterpret_cast<const float *>(m1s) + sel;
                    float4 wa = wb[u0];
#pragma unroll 4
                    for (int u = u0; u < u1; ++u) {
                        const float4 wn = wb[u + 1];
                        const float fI = fb[4 * u], fQ = fb[4 * u + 2];
                        const float2 fi2 = make_float2(fI, fI), fq2 = make_float2(fQ, fQ), nq2 = make_float2(-fQ, -fQ);
                        const float2 aR = make_float2(wa.x, wa.y), aI = make_float2(wa.z, wa.w), nR = make_float2(wn.x, wn.y), nI = make_float2(wn.z, wn.w);
                        ar = __ffma2_rn(aR, fi2, ar); ar = __ffma2_rn(aI, fq2, ar); ai = __ffma2_rn(aI, fi2, ai); ai = __ffma2_rn(aR, nq2, ai);
                        br = __ffma2_rn(nR, fi2, br); br = __ffma2_rn(nI, fq2, br); bi = __ffma2_rn(nI, fi2, bi); bi = __ffma2_rn(nR, nq2, bi);
                        wa = wn;
                    }
                    pbase[ft] = make_float4(ar.x, ai.x, ar.y, ai.y);          // [slot = tap of the pair][thread] -> {chi0 re, chi0 im, chi1 re, chi1 im}
                    pbase[128 + ft] = make_float4(br.x, bi.x, br.y, bi.y);
                }
            }
            __syncthreads();
            if (ft < 4 * nps) {                                  // one thread per (tap pair, tap of the pair, pol)
                const int sel = fam == 0 ? (ft & 1) : ft / (2 * nps);
                const int q = fam == 0 ? (ft >> 2) : ((ft % (2 * nps)) >> 1), tb = fam == 0 ? ((ft >> 1) & 1) : (ft & 1);
                const int ph = q >= np0, kA = (ph ? kf1 : kf0) + 4 * (ph ? q - np0 : q);
                const int kk = kA + 2 * tb;
                if (kk < M) {
                    // fixed-order sum of the chunk partials (deterministic)
                    const int item = fam == 0 ? q : sel * nps + q, slot = fam == 0 ? tb * 2 + sel : tb;
                    const float4 *src = pbase + slot * 128 + 2 * item;       // thread of (item, part) = 2 ((part >> 1) items + item) + (part & 1)
                    float4 sacc = src[0];
                    for (int part = 1; part < parts; ++part) {
                        const float4 t4 = src[2 * (part >> 1) * items + (part & 1)];
                        sacc.x += t4.x; sacc.y += t4.y; sacc.z += t4.z; sacc.w += t4.w;
                    }
                    if (fam == 0) {
                        gfin[(0 * 4 + sel) * M + kk] = sacc.x;
                        gfin[(0 * 4 + 2 + sel) * M + kk] = sacc.y;
                        gfin[(1 * 4 + sel) * M + kk] = sacc.z;
                        gfin[(1 * 4 + 2 + sel) * M + kk] = sacc.w;
                    } else {
                        gfin[8 * M + ((0 * 2 + sel) * 2 + 0) * M + kk] = 2.f * kap0 * sacc.x;
                        gfin[8 * M + ((0 * 2 + sel) * 2 + 1) * M + kk] = 2.f * kap0 * sacc.y;
                        gfin[8 * M + ((1 * 2 + sel) * 2 + 0) * M + kk] = 2.f * kap1 * sacc.z;
                        gfin[8 * M + ((1 * 2 + sel) * 2 + 1) * M + kk] = 2.f * kap1 * sacc.w;
                    }
                }
            }
            __syncthreads();
        }

        // ---- P7: E-term of dh (2 kappa_chi h S_nu(j), S = V_nu - edge), Adam on both parameter groups (VAELE_DP:28-31,66) -----
        {
            const double bc1 = dsc[0];
            const float bc2s = scal[6];
            for (int i = tid; i < 16 * M; i += SM_NT) {
                float g = gfin[i];
                if (i >= 8 * M) {
                    const int r = i - 8 * M, j = r % M, cn = r / (2 * M), chi = cn >> 1, nu = cn & 1;
                    const float S = scal[2 + nu] - edge[nu * M + j];
                    g = (float)((double)g + 2.0 * (double)(chi ? kap1 : kap0) * (double)hf[r] * (double)S);
                }
                if (last) {
                    if (i < 8 * M) {
                        if (rs.gW_last) rs.gW_last[(int64_t)run * 8 * M + i] = g;
                    } else if (rs.gh_last) {
                        rs.gh_last[(int64_t)run * 8 * M + i - 8 * M] = g;
                    }
                }
                if (i < 8 * M) adam_apply(Wf, g, ad, ad + 8 * M, ad + 16 * M, i, lr_w, amsgrad != 0, bc1, bc2s);
                else adam_apply(hf, g, ad + 24 * M, ad + 32 * M, ad + 40 * M, i - 8 * M, lr_h, amsgrad != 0, bc1, bc2s);
            }
        }
        __syncthreads();
    }

    // ---- write the trained state back -------------------------------------------------------------------------------
    for (int i = tid; i < 8 * M; i += SM_NT) {
        Wg[i] = Wf[i];
        hg[i] = hf[i];
    }
    for (int i = tid; i < 48 * M; i += SM_NT) adg[i] = ad[i];
    if (tid == 0) *reinterpret_cast<int *>(adg + 48 * M) = step0 + n_steps;
}

static int g_small_per_sm = 0;       // vaeq_dp_frame_runs_per_sm: 0 = choose by waves, 3 / 4 = force that kernel (tests, A/B timing)
size_t dp_small_smem(int B, int M) { return (size_t)small_layout(B, M).total * sizeof(float); }

int dp_small_launch(const DpK &p, const DpRunsK &rs, int n_lev, int n_runs, int n_steps, int stride_sym, int keep_lo_in_dst,
                    float lr_w, float lr_h, int amsgrad, cudaStream_t st) {
    const size_t smem = dp_small_smem(p.B, p.M);
    static SmemAttrCache set_smem[3][2];
    // waves of CTAs at 3 and at 4 runs per SM (shared memory permitting): take the fourth run per SM only when it saves a wave
    const int sms = sm_count(), w3 = (n_runs + SM_MINB * sms - 1) / (SM_MINB * sms), w4 = (n_runs + 4 * sms - 1) / (4 * sms);
    const bool fits4 = 4 * (smem + 1024) <= (size_t)227 * 1024;
    // measured (tools/time_frames.py): 592 runs 2.25 -> 2.08 ms per 100-step frame with the fourth run per SM; with two or more waves
    // either way (1184 runs: 3.97 vs 4.06 ms) the 80-register kernel stays ahead
    const bool four = fits4 && (g_small_per_sm == 4 || (g_small_per_sm == 0 && w4 < w3 && w4 == 1));
    static SmemAttrCache set_smem_m[3][2];                   // the M_est = 25 instantiations (compile-time tap loops)
#define SMALL_LAUNCH(NL_, IDX_, MB_, V_, MT_, CACHE_)                                                                             \
    {                                                                                                                             \
        if (int rc_ = ensure_dyn_smem(k_dp_frame_fast<NL_, MB_, MT_>, smem, CACHE_[IDX_][V_])) return rc_;                        \
        ktime_begin(VAEQ_K_DP_FRAME, st);                                                                                         \
        k_dp_frame_fast<NL_, MB_, MT_><<<n_runs, SM_NT, smem, st>>>(p, rs, n_steps, stride_sym, keep_lo_in_dst, lr_w, lr_h, amsgrad);  \
        ktime_end(VAEQ_K_DP_FRAME, st);                                                                                           \
    }
#define SMALL_CASE(NL_, IDX_)                                                   \
    {                                                                           \
        if (p.M == 25) {                                                        \
            if (four) SMALL_LAUNCH(NL_, IDX_, 4, 1, 25, set_smem_m)             \
            else SMALL_LAUNCH(NL_, IDX_, SM_MINB, 0, 25, set_smem_m)            \
        } else {                                                                \
            if (four) SMALL_LAUNCH(NL_, IDX_, 4, 1, 0, set_smem)                \
            else SMALL_LAUNCH(NL_, IDX_, SM_MINB, 0, 0, set_smem)               \
        }                                                                       \
    }
    if (n_lev == 2) SMALL_CASE(2, 0)
    else if (n_lev == 4) SMALL_CASE(4, 1)
    else SMALL_CASE(8, 2)
#undef SMALL_LAUNCH
#undef SMALL_CASE
    VAEQ_LAUNCH_CHECK("k_dp_frame_fast");
    return VAEQ_OK;
}

}  // namespace vaeq

extern "C" int vaeq_dp_frame_runs_per_sm(int32_t per_sm) {
    if (per_sm != 0 && per_sm != 3 && per_sm != 4) {
        vaeq::set_error("vaeq_dp_frame_runs_per_sm: %d is not 0 (automatic), 3 or 4", per_sm);
        return VAEQ_EINVAL;
    }
    vaeq::g_small_per_sm = per_sm;
    return VAEQ_OK;
}
