// DP VAE-LE / VAE-flex training step for B200 (sm_100a): generic-M reference kernels.
//
// One step = 4 launches on the caller's stream, all persistent over tiles of T symbols:
//   k_dp_fwd   rx -> FIR -> soft demapper -> q, out (HBM), posterior moments -> estimated-channel
//              convolution D -> residual e = D - rx (HBM scratch) -> per-CTA partial sums of C, entropy
//   k_dp_fin   partials -> C, loss, var_est, kappa = (L-Mh)/C, S_nu(j)           (1 CTA)
//   k_dp_bwd   e, moments, q, out, rx -> dL/dE_q -> softmin backward -> dL/dout -> per-CTA partial
//              tap gradients (dW: correlation with rx, dh: correlation of e with E_q)
//   k_dp_adam  deterministic reduction of the partial gradients (+ the E-term of dh) and Adam on
//              both parameter groups                                              (1 CTA)
// Reference: twoXtwoFIR.forward sf:500-527, loss_function_shaping sf:92-137, loss.backward() and
// optimizer.step() at func_VAELE_DP_MQAM_shaping.py:60-66 (sf = optical_DP_channel/shared_funcs.py).
// The closed form implemented here is restated (float64) in oracle/closed_form.py.
#include "dp_math.cuh"
#include "dp_kernels.cuh"

namespace vaeq {

// ---------------------------------------------------------------------------------------------
// forward
// ---------------------------------------------------------------------------------------------
// `cta` of `ncta` CTAs strides over the tiles and publishes partial sums in slot `cta`.  The kernels below pass
// (blockIdx.x, gridDim.x); the persistent frame kernel k_dp_frame_small passes (0, 1): one CTA is the whole run.
template <int NL>
__device__ __forceinline__ void dp_fwd_body(const DpK &p, float *smem, int cta, int ncta) {
    const int M = p.M, mh = p.mh, H = p.H, T = p.T, TE = T + 2 * H, XN = 2 * TE + 2 * mh;
    const int tid = threadIdx.x;
    DemapConst *cst = reinterpret_cast<DemapConst *>(smem);
    float4 *m1s = reinterpret_cast<float4 *>(cst + 1);  // E_q[x] per symbol of tile+halo
    float *red = reinterpret_cast<float *>(m1s + TE);   // 5*32 floats
    float *xs = red + 5 * 32;                           // 4 rows x XN samples (zero padded)
    float *Ws = xs + 4 * XN;                            // (2,4,M)
    float *hs = Ws + 8 * M;                             // (2,2,2,M)

    for (int i = tid; i < 8 * M; i += DP_NT) {
        Ws[i] = p.W[i];
        hs[i] = p.h[i];
    }
    load_demap_const(cst, p.amp, p.P, p.var, p.nu_sc, NL);
    __syncthreads();
    const DemapConst &c = *cst;

    float accC[2] = {0.f, 0.f}, accEnt = 0.f, accV[2] = {0.f, 0.f};

    for (int tile = cta; tile < p.ntiles; tile += ncta) {
        const int t0 = tile * T;
        const int tn = min(T, p.B - t0);
        const int sb = 2 * (t0 - H) - mh;               // first sample held in xs
        for (int j = tid; j < 4 * XN; j += DP_NT) {
            int r = j / XN, jj = j - r * XN, s = sb + jj;
            xs[r * XN + jj] = (s >= 0 && s < p.L) ? p.rx[(int64_t)r * p.ld_rx + s] : 0.f;
        }
        __syncthreads();

        // ---- FIR + demapper for the tile and its halo of H symbols each side -------------------
        for (int i = tid; i < tn + 2 * H; i += DP_NT) {
            const int u = t0 - H + i;
            float4 mom = make_float4(0.f, 0.f, 0.f, 0.f);
            if (u >= 0 && u < p.B && p.from_q) {
                // operator-level loss_function_shaping(q, ...) on a GIVEN q (sf:101-113): posterior moments and entropy only
                const bool owned = (i >= H) && (i < H + tn);
                const bool ent_on = owned && (u >= mh) && (u < p.B - mh);
                float m1v[4];
                float vloc[2] = {0.f, 0.f};
#pragma unroll
                for (int cc = 0; cc < 4; ++cc) {
                    float q[NL], m1 = 0.f, m2 = 0.f;
                    const float *qrow = p.q + (int64_t)(cc * NL) * p.ld_q + u;
#pragma unroll
                    for (int l = 0; l < NL; ++l) {
                        q[l] = qrow[(int64_t)l * p.ld_q];
                        m1 = fmaf(c.amp[l], q[l], m1);
                        m2 = fmaf(c.a2[l], q[l], m2);
                    }
                    m1v[cc] = m1;
                    if (ent_on) accEnt += entropy_component<NL>(q, c);
                    vloc[cc >> 1] += m2 - m1 * m1;
                }
                mom = make_float4(m1v[0], m1v[1], m1v[2], m1v[3]);
                if (owned) {
                    accV[0] += vloc[0];
                    accV[1] += vloc[1];
                    if (u < mh || u >= p.B - mh) {
                        const int slot = (u < mh) ? u : mh + (u - (p.B - mh));
                        p.edge_vs[slot] = vloc[0];
                        p.edge_vs[2 * mh + slot] = vloc[1];
                    }
                    p.m1buf4[u] = mom;
                }
            } else if (u >= 0 && u < p.B) {
                float y[4];                              // (p0 I, p0 Q, p1 I, p1 Q)
                fir_butterfly(xs + 2 * i, XN, Ws, M, y);
                const bool owned = (i >= H) && (i < H + tn);
                const bool ent_on = owned && (u >= mh) && (u < p.B - mh);                // sf:132 [mh:-mh] in symbols
                const bool keep = owned && p.qk != nullptr && (u >= p.keep_lo) && (u < p.keep_lo + p.keep_n);
                float m1v[4];
                float vloc[2] = {0.f, 0.f};
#pragma unroll
                for (int cc = 0; cc < 4; ++cc) {
                    float q[NL], m1, m2;
                    demap_component<NL>(y[cc], c.var[cc >> 1], c, q, m1, m2);
                    m1v[cc] = m1;
                    if (owned) {
                        float *qrow = p.q + (int64_t)(cc * NL) * p.ld_q + u;
#pragma unroll
                        for (int l = 0; l < NL; ++l) qrow[(int64_t)l * p.ld_q] = q[l];
                        p.out[(int64_t)cc * p.ld_out + u] = y[cc];
                        if (keep) {
                            const int64_t col = p.keep_base + (u - p.keep_lo);
                            float *krow = p.qk + (int64_t)(cc * NL) * p.ld_qk + col;
#pragma unroll
                            for (int l = 0; l < NL; ++l) krow[(int64_t)l * p.ld_qk] = q[l];
                            p.outk[(int64_t)cc * p.ld_outk + col] = y[cc];
                        }
                        if (ent_on) accEnt += entropy_component<NL>(q, c);
                    }
                    vloc[cc >> 1] += m2 - m1 * m1;                                       // sf:113
                }
                mom = make_float4(m1v[0], m1v[1], m1v[2], m1v[3]);
                if (owned) {
                    accV[0] += vloc[0];
                    accV[1] += vloc[1];
                    if (u < mh || u >= p.B - mh) {       // S_nu(j) needs the first/last mh symbols individually
                        const int slot = (u < mh) ? u : mh + (u - (p.B - mh));
                        p.edge_vs[slot] = vloc[0];
                        p.edge_vs[2 * mh + slot] = vloc[1];
                    }
                    p.m1buf4[u] = mom;
                }
            }
            m1s[i] = mom;
        }
        __syncthreads();

        // ---- estimated-channel convolution and residual for the owned samples (sf:123-134) -----
        for (int i = tid; i < tn; i += DP_NT) {
            const int u = t0 + i;
#pragma unroll
            for (int ph = 0; ph < 2; ++ph) {
                const int s = 2 * u + ph;
                float4 e = make_float4(0.f, 0.f, 0.f, 0.f);
                if (s >= mh && s < p.L - mh) {                      // "valid" region, in samples
                    float d0r = 0.f, d0i = 0.f, d1r = 0.f, d1i = 0.f;
                    const int j0 = (s + mh) & 1;
                    for (int j = j0; j < M; j += 2) {
                        const int v = (2 * (i + H) + ph + mh - j) >> 1;     // local symbol index of E_q[n-j]
                        const float4 m = m1s[v];
                        // hs[chi][nu][c][j]
                        float h00r = hs[(0 * 4 + 0) * M + j], h00i = hs[(0 * 4 + 1) * M + j];
                        float h01r = hs[(0 * 4 + 2) * M + j], h01i = hs[(0 * 4 + 3) * M + j];
                        float h10r = hs[(1 * 4 + 0) * M + j], h10i = hs[(1 * 4 + 1) * M + j];
                        float h11r = hs[(1 * 4 + 2) * M + j], h11i = hs[(1 * 4 + 3) * M + j];
                        d0r += h00r * m.x - h00i * m.y + h01r * m.z - h01i * m.w;     // sf:124-125
                        d0i += h00i * m.x + h00r * m.y + h01i * m.z + h01r * m.w;     // sf:126-127
                        d1r += h10r * m.x - h10i * m.y + h11r * m.z - h11i * m.w;
                        d1i += h10i * m.x + h10r * m.y + h11i * m.z + h11r * m.w;
                    }
                    const float *xr = xs + 2 * (i + H) + ph + mh;   // rx sample s in the tile buffer
                    e.x = d0r - xr[0];
                    e.y = d0i - xr[XN];
                    e.z = d1r - xr[2 * XN];
                    e.w = d1i - xr[3 * XN];
                    accC[0] += e.x * e.x + e.y * e.y;
                    accC[1] += e.z * e.z + e.w * e.w;
                }
                p.ebuf4[2 * (int64_t)u + ph] = e;
            }
        }
        __syncthreads();
    }

    float v[5] = {accC[0], accC[1], accEnt, accV[0], accV[1]};
    block_sum<5>(v, red);
    if (tid == 0) {
        double *dst = p.part_fwd + (int64_t)cta * 8;
#pragma unroll
        for (int i = 0; i < 5; ++i) dst[i] = (double)v[i];
    }
}

template <int NL>
__global__ void __launch_bounds__(DP_NT) k_dp_fwd(DpK p) {
    extern __shared__ __align__(16) float smem[];
    dp_fwd_body<NL>(p, smem, blockIdx.x, gridDim.x);
}

// ---------------------------------------------------------------------------------------------
// finalize forward: C, loss, var_est, kappa, S_nu(j)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void dp_fin_body(const DpK &p, int nparts) {      // one CTA of 256 ... 1024 threads
    __shared__ double tot[5];
    __shared__ double Esh[2];
    __shared__ float Ssh[2 * VAEQ_MAX_TAPS];
    __shared__ float edge_sh[4 * (VAEQ_MAX_TAPS / 2 + 1)];
    __shared__ float hsq[4 * VAEQ_MAX_TAPS];                // |h[chi][nu][j]|^2
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, M = p.M, mh = p.mh, Mh = 2 * p.mh;
    {   // quantity w = tid & 7 (5 used), slot = tid >> 3: every thread sums a strided share of the CTA partials (592 partials
        // over the 128 slots of the 1024-thread fin CTA = 5 independent loads per thread instead of a chain of 19), then the
        // shares are combined in fixed order (deterministic)
        __shared__ double wq[32][8];
        const int w = tid & 7, slot = tid >> 3, nslot = blockDim.x >> 3, nwarp = blockDim.x >> 5;
        double a = 0.0;
        if (w < 5) {
#pragma unroll 4
            for (int b = slot; b < nparts; b += nslot) a += p.part_fwd[(int64_t)b * 8 + w];
        }
        a += __shfl_xor_sync(0xffffffffu, a, 8);
        a += __shfl_xor_sync(0xffffffffu, a, 16);
        if (lane < 8) wq[wid][lane] = a;
        __syncthreads();
        if (tid < 5) {
            double v = 0.0;
            for (int k = 0; k < nwarp; ++k) v += wq[k][tid];
            tot[tid] = v;
        }
    }
    // stage the edge variances and |h|^2 (one global round trip instead of a chain of dependent loads)
    for (int i = tid; i < 4 * mh; i += blockDim.x) edge_sh[i] = p.edge_vs[i];
    for (int i = tid; i < 4 * M; i += blockDim.x) {
        const int cn = i / M, j = i - cn * M;
        const float hr = p.h[(cn * 2 + 0) * M + j], hi = p.h[(cn * 2 + 1) * M + j];
        hsq[i] = hr * hr + hi * hi;
    }
    __syncthreads();
    // S_nu(j) = sum of (Var_I+Var_Q)[nu] over source symbols u with Mh <= 2u+j < L      (sf:128)
    for (int idx = tid; idx < 2 * M; idx += blockDim.x) {
        const int nu = idx / M, j = idx - nu * M;
        double s = tot[3 + nu];
        const int u_lo = (Mh - j + 1) >> 1;                 // first included symbol
        const int u_hi = (p.L - 1 - j) >> 1;                // last included symbol
        for (int u = 0; u < u_lo && u < mh; ++u) s -= (double)edge_sh[nu * 2 * mh + u];
        for (int u = u_hi + 1; u < p.B; ++u) s -= (double)edge_sh[nu * 2 * mh + mh + (u - (p.B - mh))];
        Ssh[idx] = (float)s;
        p.scal[DP_S_OFF + idx] = (float)s;
    }
    __syncthreads();
    if (wid < 2) {                                          // warp chi: E_chi = sum_{nu,j} |h|^2 S_nu(j)   (sf:129)
        const int chi = wid;
        double E = 0.0;
        for (int idx = lane; idx < 2 * M; idx += 32) E += (double)hsq[chi * 2 * M + idx] * (double)Ssh[idx];
        E = warp_sum(E);
        if (lane == 0) Esh[chi] = E;
    }
    __syncthreads();
    if (tid < 2) {                                          // thread chi: C_chi, its log term; thread 0 assembles the loss
        const int chi = tid;
        const double width = (double)(p.L - Mh);
        const double C = tot[chi] + Esh[chi];                                               // sf:133-134
        const double term = width * log(C);                                                 // sf:136
        p.scal[DP_C_OFF + chi] = (float)C;
        p.scal[DP_KAPPA_OFF + chi] = (float)(width / C);
        const float ve = (float)(C / width);                                                // sf:137
        p.scal[DP_VAREST_OFF + chi] = ve;
        if (p.var_est_out) p.var_est_out[(int64_t)chi * p.var_est_stride] = ve;
        const double term1 = __shfl_sync(0x3u, term, 1);
        if (chi == 0) {
            const double loss = (-tot[2] + term) + term1;
            p.scal[DP_LOSS_OFF] = (float)loss;
            if (p.loss_out) *p.loss_out = (float)loss;
        }
    }
}

__global__ void __launch_bounds__(1024) k_dp_fin(DpK p, int nparts) { dp_fin_body(p, nparts); }

// ---------------------------------------------------------------------------------------------
// backward
// ---------------------------------------------------------------------------------------------
template <int NL>
__device__ __forceinline__ void dp_bwd_body(const DpK &p, float *smem, int cta, int ncta) {
    const int M = p.M, mh = p.mh, Mh = 2 * p.mh, H = p.H, T = p.T, TE = T + 2 * H, XN = 2 * TE + 2 * mh;
    const int tid = threadIdx.x;
    DemapConst *cst = reinterpret_cast<DemapConst *>(smem);
    float4 *es = reinterpret_cast<float4 *>(cst + 1);   // 2*TE: gD per sample of tile+halo
    float4 *m1s = es + 2 * TE;                          // TE
    float4 *gys = m1s + TE;                             // T: dL/dout per owned symbol
    float *xs = reinterpret_cast<float *>(gys + T);     // 4 rows x XN samples
    float *hs = xs + 4 * XN;                            // (2,2,2,M)
    float *PSg = hs + 8 * M;                            // (2, M+1) prefix sums of sum_chi kappa_chi |h|^2

    for (int i = tid; i < 8 * M; i += DP_NT) hs[i] = p.h[i];
    load_demap_const(cst, p.amp, p.P, p.var, p.nu_sc, NL);
    const float kap0 = p.scal[DP_KAPPA_OFF], kap1 = p.scal[DP_KAPPA_OFF + 1];
    __syncthreads();
    if (tid < 2) {
        const int nu = tid;
        float a = 0.f;
        PSg[nu * (M + 1)] = 0.f;
        for (int j = 0; j < M; ++j) {
            float h0r = hs[((0 * 2 + nu) * 2 + 0) * M + j], h0i = hs[((0 * 2 + nu) * 2 + 1) * M + j];
            float h1r = hs[((1 * 2 + nu) * 2 + 0) * M + j], h1i = hs[((1 * 2 + nu) * 2 + 1) * M + j];
            a += kap0 * (h0r * h0r + h0i * h0i) + kap1 * (h1r * h1r + h1i * h1i);
            PSg[nu * (M + 1) + j + 1] = a;
        }
    }
    __syncthreads();
    const DemapConst &c = *cst;

    // each thread owns up to two complex tap-gradient outputs: idx < 4M -> dh(chi,nu,j), else dW(o,in,k)
    float accR[2] = {0.f, 0.f}, accI[2] = {0.f, 0.f};

    for (int tile = cta; tile < p.ntiles; tile += ncta) {
        const int t0 = tile * T;
        const int tn = min(T, p.B - t0);
        const int sb = 2 * (t0 - H) - mh;
        for (int j = tid; j < 4 * XN; j += DP_NT) {
            int r = j / XN, jj = j - r * XN, s = sb + jj;
            xs[r * XN + jj] = (s >= 0 && s < p.L) ? p.rx[(int64_t)r * p.ld_rx + s] : 0.f;
        }
        for (int i = tid; i < 2 * TE; i += DP_NT) {          // gD = 2 kappa_chi (D - r), zero outside the valid region
            const int64_t sidx = 2 * (int64_t)(t0 - H) + i;
            float4 e = make_float4(0.f, 0.f, 0.f, 0.f);
            if (sidx >= 0 && sidx < p.L) e = p.ebuf4[sidx];
            e.x *= 2.f * kap0; e.y *= 2.f * kap0; e.z *= 2.f * kap1; e.w *= 2.f * kap1;
            es[i] = e;
        }
        for (int i = tid; i < TE; i += DP_NT) {
            const int u = t0 - H + i;
            m1s[i] = (u >= 0 && u < p.B) ? p.m1buf4[u] : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        __syncthreads();

        for (int i = tid; i < tn; i += DP_NT) {
            const int u = t0 + i;
            // dL/dE_q(u) = sum_chi sum_j conj(h[chi][nu][j]) gD_chi(2u - mh + j)
            float g0r = 0.f, g0i = 0.f, g1r = 0.f, g1i = 0.f;
            const int sl = 2 * (i + H) - mh;
            for (int j = 0; j < M; ++j) {
                const float4 e = es[sl + j];
                float h00r = hs[(0 * 4 + 0) * M + j], h00i = hs[(0 * 4 + 1) * M + j];
                float h01r = hs[(0 * 4 + 2) * M + j], h01i = hs[(0 * 4 + 3) * M + j];
                float h10r = hs[(1 * 4 + 0) * M + j], h10i = hs[(1 * 4 + 1) * M + j];
                float h11r = hs[(1 * 4 + 2) * M + j], h11i = hs[(1 * 4 + 3) * M + j];
                g0r += h00r * e.x + h00i * e.y + h10r * e.z + h10i * e.w;
                g0i += h00r * e.y - h00i * e.x + h10r * e.w - h10i * e.z;
                g1r += h01r * e.x + h01i * e.y + h11r * e.z + h11i * e.w;
                g1i += h01r * e.y - h01i * e.x + h11r * e.w - h11i * e.z;
            }
            // dL/dVar_nu(u) = sum_chi kappa_chi sum_{j: Mh <= 2u+j < L} |h|^2
            const int jlo = max(0, Mh - 2 * u), jhi = min(M, p.L - 2 * u);
            const float gV0 = PSg[jhi] - PSg[jlo];
            const float gV1 = PSg[(M + 1) + jhi] - PSg[(M + 1) + jlo];
            const float4 mom = m1s[i + H];
            const float m1v[4] = {mom.x, mom.y, mom.z, mom.w};
            const float gE[4] = {g0r, g0i, g1r, g1i};
            const bool ent_on = (u >= mh) && (u < p.B - mh);
            float gy[4];
#pragma unroll
            for (int cc = 0; cc < 4; ++cc) {
                float q[NL];
                const float *qrow = p.q + (int64_t)(cc * NL) * p.ld_q + u;
#pragma unroll
                for (int l = 0; l < NL; ++l) q[l] = qrow[(int64_t)l * p.ld_q];
                const float gV = (cc >> 1) ? gV1 : gV0;
                const float g1 = gE[cc] - 2.f * m1v[cc] * gV;
                if (p.from_q) {                                 // dL/dq_l = a_l dL/dE[x] + a_l^2 dL/dE[x^2] + d(-entropy)/dq_l
                    gy[cc] = 0.f;
                    if (p.gq != nullptr) {
                        float *grow = p.gq + (int64_t)(cc * NL) * p.ld_gq + u;
#pragma unroll
                        for (int l = 0; l < NL; ++l) {
                            float g = fmaf(c.amp[l], g1, c.a2[l] * gV);
                            if (ent_on) {
                                const float uu = __fdiv_rn(q[l], c.P[l]), t = uu + 1e-12f;
                                g += logf(t) + __fdiv_rn(uu, t);
                            }
                            grow[(int64_t)l * p.ld_gq] = g;
                        }
                    }
                    continue;
                }
                const float y = p.out[(int64_t)cc * p.ld_out + u];
                gy[cc] = demap_backward<NL>(y, c.var[cc >> 1], c, q, g1, gV, ent_on);
            }
            gys[i] = make_float4(gy[0], gy[1], gy[2], gy[3]);
        }
        __syncthreads();

        // ---- tap gradients: one complex output per thread slot, summed over the owned samples ----
#pragma unroll
        for (int slot = 0; slot < 2; ++slot) {
            const int idx = tid + slot * DP_NT;
            if (idx < 4 * M) {                               // dh[chi][nu][:, j]
                const int j = idx % M, cn = idx / M, chi = cn >> 1, nu = cn & 1;
                float ar = 0.f, ai = 0.f;
                const int par = (mh + j) & 1;
                for (int sl = 2 * H + par; sl < 2 * H + 2 * tn; sl += 2) {
                    const float4 e = es[sl];
                    const float4 m = m1s[(sl + mh - j) >> 1];
                    const float gr = chi ? e.z : e.x, gi = chi ? e.w : e.y;
                    const float er = nu ? m.z : m.x, ei = nu ? m.w : m.y;
                    ar += gr * er + gi * ei;
                    ai += gi * er - gr * ei;
                }
                accR[slot] += ar;
                accI[slot] += ai;
            } else if (idx < 8 * M) {                        // dW[o][in | 2+in][k]
                const int id2 = idx - 4 * M;
                const int k = id2 % M, oi = id2 / M, o = oi >> 1, in = oi & 1;
                float ar = 0.f, ai = 0.f;
                const float *xI = xs + (2 * in) * XN + 2 * H + k, *xQ = xs + (2 * in + 1) * XN + 2 * H + k;
                for (int i = 0; i < tn; ++i) {
                    const float4 g = gys[i];
                    const float gI = o ? g.z : g.x, gQ = o ? g.w : g.y;
                    const float a = xI[2 * i], b = xQ[2 * i];
                    ar += gI * a + gQ * b;
                    ai += gQ * a - gI * b;
                }
                accR[slot] += ar;
                accI[slot] += ai;
            }
        }
        __syncthreads();
    }

    float *gp = p.gpart + (int64_t)cta * 16 * M;            // layout: gW (2,4,M) then gh (2,2,2,M)
#pragma unroll
    for (int slot = 0; slot < 2; ++slot) {
        const int idx = tid + slot * DP_NT;
        if (idx < 4 * M) {
            const int j = idx % M, cn = idx / M;
            gp[8 * M + (cn * 2 + 0) * M + j] = accR[slot];
            gp[8 * M + (cn * 2 + 1) * M + j] = accI[slot];
        } else if (idx < 8 * M) {
            const int id2 = idx - 4 * M;
            const int k = id2 % M, oi = id2 / M, o = oi >> 1, in = oi & 1;
            gp[(o * 4 + in) * M + k] = accR[slot];
            gp[(o * 4 + 2 + in) * M + k] = accI[slot];
        }
    }
}

template <int NL>
__global__ void __launch_bounds__(DP_NT) k_dp_bwd(DpK p) {
    extern __shared__ __align__(16) float smem[];
    dp_bwd_body<NL>(p, smem, blockIdx.x, gridDim.x);
}

// ---------------------------------------------------------------------------------------------
// gradient reduction + Adam (torch.optim.Adam single-tensor semantics, see oracle/closed_form.py)
// ---------------------------------------------------------------------------------------------
// gradient entry i given the sum `a` of its partials: add the E-term of dh, export, Adam
__device__ __forceinline__ void dp_adam_finish(const DpK &p, int i, double a, int do_update, float lr_w, float lr_h, int amsgrad,
                                               double bc1, float bc2s) {
    const int M = p.M;
    if (i >= 8 * M) {                                       // E-term of dh: 2 kappa_chi h S_nu(j)
        const int r = i - 8 * M, j = r % M, cn = r / (2 * M), chi = cn >> 1, nu = cn & 1;
        a += 2.0 * (double)p.scal[DP_KAPPA_OFF + chi] * (double)p.h[r] * (double)p.scal[DP_S_OFF + nu * M + j];
    }
    const float g = (float)a;
    p.gfinal[i] = g;
    if (i < 8 * M) {
        if (p.gW_out) p.gW_out[i] = g;
    } else {
        if (p.gh_out) p.gh_out[i - 8 * M] = g;
    }
    if (do_update) {
        if (i < 8 * M)
            adam_apply(p.W, g, p.adam, p.adam + 8 * M, p.adam + 16 * M, i, lr_w, amsgrad != 0, bc1, bc2s);
        else
            adam_apply(p.h, g, p.adam + 24 * M, p.adam + 32 * M, p.adam + 40 * M, i - 8 * M, lr_h, amsgrad != 0, bc1, bc2s);
    }
}

// ADAM_TPE threads per tap-gradient entry stride over the per-CTA partials (fixed order -> deterministic; with 592 partials
// each thread has <= 5 independent loads in flight instead of a chain of 19), warp + shared-memory reduction, then one
// thread finishes the entry.  The step counter is bumped by the last CTA to finish.
constexpr int ADAM_TPE = 128, ADAM_EPC = 2;                 // threads per entry, entries per CTA
__global__ void __launch_bounds__(ADAM_TPE * ADAM_EPC) k_dp_adam(DpK p, int nparts, int do_update, float lr_w, float lr_h, int amsgrad) {
    __shared__ double bc1_sh;
    __shared__ float bc2s_sh;
    __shared__ double wsum[ADAM_EPC][ADAM_TPE / 32];
    const int M = p.M, n = 16 * M, lane = threadIdx.x & 31, sub = threadIdx.x % ADAM_TPE, e = threadIdx.x / ADAM_TPE;
    int *step_ptr = p.adam ? reinterpret_cast<int *>(p.adam + 48 * M) : nullptr;
    const int step = do_update ? *step_ptr + 1 : 0;         // every CTA reads the old value before taking its ticket
    if (threadIdx.x == ADAM_TPE * ADAM_EPC - 1) {
        if (do_update) adam_bias(step, &bc1_sh, &bc2s_sh);
        else { bc1_sh = 1.0; bc2s_sh = 1.f; }
    }
    const int i = blockIdx.x * ADAM_EPC + e;
    double a = 0.0;
    if (i < n) {
#pragma unroll 4
        for (int b = sub; b < nparts; b += ADAM_TPE) a += (double)p.gpart[(int64_t)b * n + i];
        a = warp_sum(a);
        if (lane == 0) wsum[e][sub >> 5] = a;
    }
    __syncthreads();
    if (i < n && sub == 0) {
        a = 0.0;
#pragma unroll
        for (int w = 0; w < ADAM_TPE / 32; ++w) a += wsum[e][w];
        dp_adam_finish(p, i, a, do_update, lr_w, lr_h, amsgrad, bc1_sh, bc2s_sh);
    }
    if (do_update) {
        __syncthreads();
        if (threadIdx.x == 0) {
            int *ticket = step_ptr + 1;
            __threadfence();
            if (atomicAdd(ticket, 1) == (int)gridDim.x - 1) {
                *step_ptr = step;
                *ticket = 0;
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// Persistent frame kernel for reference-size minibatches (batch_len <= DP_TILE: the whole minibatch is ONE tile).
// One CTA owns one run and walks its sequential minibatches (VAELE_DP:57-66 / VAEflex_DP:59-70) inside a single
// launch: forward -> fin -> backward -> gradient reduction + Adam, separated by __syncthreads() instead of kernel
// boundaries (at batch_len = 100 a frame is 100-990 steps; launched separately they are launch-latency bound).
// blockIdx.x = run: independent runs (sweep cells: SNR x realisation x lr ..., Eval_run_DP.py:68-95) are batched in the
// same launch, every per-run tensor addressed with a run stride.  The bodies are the generic kernels' own, so a frame
// stepped here is bitwise identical to the same frame stepped launch by launch.
// ---------------------------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ T *byte_off(T *ptr, int64_t bytes) {
    return ptr ? reinterpret_cast<T *>(reinterpret_cast<char *>(ptr) + bytes) : nullptr;
}

template <int NL>
__global__ void __launch_bounds__(DP_NT) k_dp_frame_small(DpK p, DpRunsK rs, int n_steps, int stride_sym, int keep_lo_in_dst,
                                                          float lr_w, float lr_h, int amsgrad) {
    extern __shared__ __align__(16) float smem[];
    __shared__ double bc1_sh;
    __shared__ float bc2s_sh;
    const int run = blockIdx.x, M = p.M, n = 16 * M;
    // ---- this run's tensors ------------------------------------------------------------------
    p.rx += run * rs.rs_rx; p.amp += run * rs.rs_amp; p.P += run * rs.rs_P; p.var += run * rs.rs_var;
    p.W += run * rs.rs_W; p.h += run * rs.rs_h; p.adam += run * rs.rs_adam;
    p.q += run * rs.rs_q; p.out += run * rs.rs_out;
    if (p.qk) { p.qk += run * rs.rs_qk; p.outk += run * rs.rs_outk; }
    {
        const int64_t wo = run * rs.ws_stride;
        p.part_fwd = byte_off(p.part_fwd, wo); p.edge_vs = byte_off(p.edge_vs, wo); p.scal = byte_off(p.scal, wo);
        p.ebuf4 = byte_off(p.ebuf4, wo); p.m1buf4 = byte_off(p.m1buf4, wo); p.gpart = byte_off(p.gpart, wo);
        p.gfinal = byte_off(p.gfinal, wo);
    }
    if (rs.nu_sc) p.nu_sc = rs.nu_sc[run];
    if (rs.lr_w) lr_w = rs.lr_w[run];
    if (rs.lr_h) lr_h = rs.lr_h[run];
    p.gW_out = rs.gW_last ? rs.gW_last + (int64_t)run * 8 * M : nullptr;
    p.gh_out = rs.gh_last ? rs.gh_last + (int64_t)run * 8 * M : nullptr;
    const float *rx0 = p.rx;
    int *step_ptr = reinterpret_cast<int *>(p.adam + 48 * M);

    for (int m = 0; m < n_steps; ++m) {
        p.rx = rx0 + (int64_t)m * stride_sym * 2;
        p.keep_base = (int64_t)m * stride_sym + (keep_lo_in_dst ? p.keep_lo : 0);
        const bool last = m == n_steps - 1;
        p.loss_out = rs.loss_steps ? rs.loss_steps + (int64_t)run * n_steps + m : nullptr;
        p.var_est_out = rs.var_steps ? rs.var_steps + (int64_t)run * 2 * n_steps + m : nullptr;
        p.var_est_stride = n_steps;
        dp_fwd_body<NL>(p, smem, 0, 1);
        __syncthreads();
        dp_fin_body(p, 1);
        __syncthreads();
        if (last && threadIdx.x < 3) {                       // the desc's loss / var_est keep the last step's values
            if (threadIdx.x == 0 && rs.loss_last) rs.loss_last[run] = p.scal[DP_LOSS_OFF];
            if (threadIdx.x > 0 && rs.var_last) rs.var_last[2 * run + threadIdx.x - 1] = p.scal[DP_VAREST_OFF + threadIdx.x - 1];
        }
        dp_bwd_body<NL>(p, smem, 0, 1);
        __syncthreads();
        // gradient "reduction" over the single partial + Adam: one THREAD per entry (same arithmetic as k_dp_adam's lane 0)
        const int step = *step_ptr + 1;
        if (threadIdx.x == 0) adam_bias(step, &bc1_sh, &bc2s_sh);
        __syncthreads();
        for (int i = threadIdx.x; i < n; i += DP_NT) dp_adam_finish(p, i, (double)p.gpart[i], 1, lr_w, lr_h, amsgrad, bc1_sh, bc2s_sh);
        __syncthreads();
        if (threadIdx.x == 0) *step_ptr = step;
    }
}

__global__ void k_adam_generic(float *param, const float *grad, float *state, int n, float lr, int amsgrad,
                               int *step_count, int bump) {
    __shared__ int step_sh;
    __shared__ double bc1_sh;
    __shared__ float bc2s_sh;
    if (threadIdx.x == 0) {
        step_sh = *step_count + (bump ? 1 : 0);
        adam_bias(step_sh, &bc1_sh, &bc2s_sh);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < n; i += blockDim.x)
        adam_apply(param, grad[i], state, state + n, state + 2 * n, i, lr, amsgrad != 0, bc1_sh, bc2s_sh);
    __syncthreads();
    if (threadIdx.x == 0 && bump) *step_count = step_sh;
}

// ---------------------------------------------------------------------------------------------
// soft demapper alone (soft_dec, sf:529-542)
// ---------------------------------------------------------------------------------------------
template <int NL>
__global__ void k_soft_dec(const float *out, int64_t ld_out, const float *var, const float *amp, float nu_sc, int N,
                           float *q, int64_t ld_q, const float *nu_runs = nullptr) {
    __shared__ DemapConst cst;
    out += (int64_t)blockIdx.y * 4 * ld_out;             // blockIdx.y = run of a batch (vaeq_soft_dec_runs)
    q += (int64_t)blockIdx.y * 4 * NL * ld_q;
    load_demap_const(&cst, amp, nullptr, var + 2 * blockIdx.y, nu_runs ? nu_runs[blockIdx.y] : nu_sc, NL);
    __syncthreads();
    for (int64_t u = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; u < N; u += (int64_t)gridDim.x * blockDim.x) {
#pragma unroll
        for (int cc = 0; cc < 4; ++cc) {
            float qv[NL], m1, m2;
            demap_component<NL>(out[(int64_t)cc * ld_out + u], cst.var[cc >> 1], cst, qv, m1, m2);
#pragma unroll
            for (int l = 0; l < NL; ++l) q[(int64_t)(cc * NL + l) * ld_q + u] = qv[l];
        }
    }
}

// Bandwidth version for 16-byte aligned rows and N % 4 == 0: a thread owns 4 consecutive symbols (float4 loads / streaming float4
// stores, 512 B per warp instruction).  The logit z keeps the reference's operation order and roundings -- ((y-a)^2 * 0.5) / var
// + nu_sc a^2 (sf:521) -- with the division by the per-polarisation constant var done as x*r + one fused residual correction
// (r = RN(1/var); q0 = RN(x r); q = RN(q0 + RN(x - q0 var) r): Markstein's correction, the correctly rounded quotient except
// for rare last-bit cases), so hard decisions (argmin z) follow the precise kernel; exp and the normalisation use ex2.approx
// and one reciprocal per component (|dq| < 3e-7).  The precise kernel above took 586 us at N = 2^22 (0.16 of the HBM roofline: 64 IEEE divisions and 32 expf
// per symbol); this one is bound by the q stores.
__device__ __forceinline__ float div_by_const(float x, float c, float rc) {
    const float q0 = x * rc;
    return fmaf(fmaf(-q0, c, x), rc, q0);
}
template <int NL>
__global__ void __launch_bounds__(256) k_soft_dec_vec(const float *__restrict__ out, int64_t ld_out, const float *var, const float *amp,
                                                      float nu_sc, int N, float *__restrict__ q, int64_t ld_q, const float *nu_runs = nullptr) {
    // blockIdx.y = run of a batch (vaeq_soft_dec_runs): tensors advance by their size, var by 2, nu_sc comes from nu_runs
    __shared__ DemapConst cst;
    out += (int64_t)blockIdx.y * 4 * ld_out;
    q += (int64_t)blockIdx.y * 4 * NL * ld_q;
    load_demap_const(&cst, amp, nullptr, var + 2 * blockIdx.y, nu_runs ? nu_runs[blockIdx.y] : nu_sc, NL);
    __syncthreads();
    const int n4 = N >> 2;
    for (int g = blockIdx.x * blockDim.x + threadIdx.x; g < n4; g += gridDim.x * blockDim.x) {
        const int64_t u = 4 * (int64_t)g;
#pragma unroll
        for (int cc = 0; cc < 4; ++cc) {
            const float v = cst.var[cc >> 1], rv = 1.f / v;
            const float4 y4 = ldg_stream(reinterpret_cast<const float4 *>(out + (int64_t)cc * ld_out + u));
            const float y[4] = {y4.x, y4.y, y4.z, y4.w};
            float pq[4][NL], r[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                float z[NL], zmin = 3.0e38f;
#pragma unroll
                for (int l = 0; l < NL; ++l) {
                    const float d = y[k] - cst.amp[l];
                    z[l] = __fadd_rn(div_by_const(__fmul_rn(__fmul_rn(d, d), 0.5f), v, rv), cst.nua2[l]);
                    zmin = fminf(zmin, z[l]);
                }
                float s = 0.f;
#pragma unroll
                for (int l = 0; l < NL; ++l) {
                    pq[k][l] = ex2_approx((zmin - z[l]) * LOG2E);
                    s += pq[k][l];
                }
                r[k] = rcp_approx(s);
            }
#pragma unroll
            for (int l = 0; l < NL; ++l)
                stg_stream(reinterpret_cast<float4 *>(q + (int64_t)(cc * NL + l) * ld_q + u),
                           make_float4(pq[0][l] * r[0], pq[1][l] * r[1], pq[2][l] * r[2], pq[3][l] * r[3]));
        }
    }
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
static size_t dp_fwd_smem(int M, int T, int H, int mh) {
    const int TE = T + 2 * H, XN = 2 * TE + 2 * mh;
    size_t f = sizeof(DemapConst) / 4 + 4 * TE + 5 * 32 + 4 * XN + 16 * M;
    return f * sizeof(float);
}
static size_t dp_bwd_smem(int M, int T, int H, int mh) {
    const int TE = T + 2 * H, XN = 2 * TE + 2 * mh;
    size_t f = sizeof(DemapConst) / 4 + 8 * TE + 4 * TE + 4 * T + 4 * XN + 8 * M + 2 * (M + 1);
    return f * sizeof(float);
}

struct DpWsLayout {
    size_t part_fwd, edge_vs, scal, tile_ctr, ebuf, m1buf, gybuf, sbuf, gpart, gfinal, total;
};
static DpWsLayout dp_ws_layout(int B, int M) {
    DpWsLayout w;
    size_t off = 0;
    auto take = [&](size_t bytes) {
        size_t o = off;
        off = align_up(off + bytes, 256);
        return o;
    };
    w.part_fwd = take((size_t)DP_GRID_CAP * 8 * sizeof(double));
    w.edge_vs = take((size_t)4 * (VAEQ_MAX_TAPS / 2 + 1) * sizeof(float));
    w.scal = take((size_t)(DP_S_OFF + 2 * VAEQ_MAX_TAPS) * sizeof(float));
    w.tile_ctr = take(4 * sizeof(int));
    w.ebuf = take((size_t)B * 8 * sizeof(float));
    w.m1buf = take((size_t)B * 4 * sizeof(float));
    w.gybuf = take((size_t)B * 4 * sizeof(float));
    w.sbuf = take((size_t)B * 12 * sizeof(float));
    w.gpart = take((size_t)DP_GRID_CAP * 16 * M * sizeof(float));
    w.gfinal = take((size_t)16 * M * sizeof(float));
    w.total = off;
    return w;
}

static bool g_dynamic_tiles = true;
static int g_persistent_frames = 1;   // 0: per-step launches, 1: dp_small.cu (default), 2: generic bodies in one launch
static int g_persistent_frames_mode() { return g_persistent_frames; }

// cols_qout >= 0: q / out need only hold that many columns per row (batch-split ranks pass buffers of their own columns)
static int dp_validate(const vaeq_dp_desc *d, bool need_grads, bool need_adam, int64_t cols_qout = -1) {
    VAEQ_CHECK_ARG(d != nullptr, "desc is NULL");
    VAEQ_CHECK_ARG(d->sps == 2, "sps=%d: only sps=2 is implemented (every reference driver uses 2)", d->sps);
    VAEQ_CHECK_ARG(d->M >= 1 && d->M <= VAEQ_MAX_TAPS && (d->M & 1), "M_est=%d must be odd and <= %d", d->M, VAEQ_MAX_TAPS);
    VAEQ_CHECK_ARG(d->n_lev == 2 || d->n_lev == 4 || d->n_lev == 8, "n_lev=%d must be 2, 4 or 8", d->n_lev);
    VAEQ_CHECK_ARG(d->B > 2 * (d->M / 2), "batch_len=%d must exceed M_est-1=%d (the loss's valid region is empty)", d->B, 2 * (d->M / 2));
    // batch-split calls may pass q = out = NULL together with q_keep / out_keep: only the kept section of the window is wanted then
    const bool no_q = cols_qout >= 0 && !d->q && !d->out && (cols_qout == 0 || (d->q_keep && d->out_keep));   // cols 0: the call touches neither
    VAEQ_CHECK_ARG(d->rx && d->amp && d->P && d->var && d->W && d->h && ((d->q && d->out) || no_q), "NULL tensor pointer");
    const int64_t need_cols = no_q ? 0 : cols_qout >= 0 ? cols_qout : (int64_t)d->B;
    VAEQ_CHECK_ARG(d->ld_rx >= (int64_t)d->B * d->sps && d->ld_q >= need_cols && d->ld_out >= need_cols, "row stride smaller than the row");
    VAEQ_CHECK_ARG(!need_grads || need_adam || (d->gW && d->gh), "gW/gh must be given");
    VAEQ_CHECK_ARG(!need_adam || d->adam, "adam state is NULL");
    VAEQ_CHECK_ARG(d->workspace != nullptr, "workspace is NULL");
    if (d->workspace_bytes < vaeq_dp_workspace_bytes(d->B, d->M, d->n_lev)) {
        set_error("workspace too small: %zu < %zu", d->workspace_bytes, vaeq_dp_workspace_bytes(d->B, d->M, d->n_lev));
        return VAEQ_EWORKSPACE;
    }
    if (d->q_keep) VAEQ_CHECK_ARG(d->out_keep && d->keep_n >= 0 && d->keep_lo >= 0, "bad keep window");
    return VAEQ_OK;
}

static DpK dp_make_params(const vaeq_dp_desc *d) {
    DpK p;
    memset(&p, 0, sizeof(p));
    const DpWsLayout w = dp_ws_layout(d->B, d->M);
    char *ws = static_cast<char *>(d->workspace);
    p.rx = d->rx; p.ld_rx = d->ld_rx;
    p.B = d->B; p.L = d->B * d->sps; p.M = d->M; p.mh = d->M / 2; p.H = (p.mh + 1) / 2;
    p.W = d->W; p.h = d->h; p.amp = d->amp; p.P = d->P; p.var = d->var; p.nu_sc = d->nu_sc;
    p.q = d->q; p.ld_q = d->ld_q; p.out = d->out; p.ld_out = d->ld_out;
    p.qk = d->q_keep; p.ld_qk = d->ld_q_keep; p.outk = d->out_keep; p.ld_outk = d->ld_out_keep;
    p.keep_lo = d->keep_lo; p.keep_n = d->keep_n; p.keep_base = 0;
    p.part_fwd = reinterpret_cast<double *>(ws + w.part_fwd);
    p.edge_vs = reinterpret_cast<float *>(ws + w.edge_vs);
    p.scal = reinterpret_cast<float *>(ws + w.scal);
    p.ebuf4 = reinterpret_cast<float4 *>(ws + w.ebuf);
    p.m1buf4 = reinterpret_cast<float4 *>(ws + w.m1buf);
    p.erows = reinterpret_cast<float *>(ws + w.ebuf);
    p.m1rows = reinterpret_cast<float *>(ws + w.m1buf);
    p.gyrows = reinterpret_cast<float *>(ws + w.gybuf);
    p.srows = reinterpret_cast<float *>(ws + w.sbuf);
    p.need_bwd = 1;
    p.gpart = reinterpret_cast<float *>(ws + w.gpart);
    p.gfinal = reinterpret_cast<float *>(ws + w.gfinal);
    p.adam = d->adam;
    p.loss_out = d->loss; p.var_est_out = d->var_est; p.var_est_stride = 1;
    p.gW_out = d->gW; p.gh_out = d->gh;
    p.T = DP_TILE;
    p.ntiles = (d->B + p.T - 1) / p.T;
    p.sym_lo = 0; p.sym_hi = d->B; p.clo = 0; p.chi = d->B;
    p.tile_ctr = reinterpret_cast<int *>(ws + w.tile_ctr);
    p.dyn = g_dynamic_tiles ? 1 : 0;
    return p;
}

int dp_launch_fin(const DpK &p, int nparts, cudaStream_t st) {
    ktime_begin(VAEQ_K_DP_FIN, st);
    k_dp_fin<<<1, nparts > 64 ? 1024 : 256, 0, st>>>(p, nparts);
    ktime_end(VAEQ_K_DP_FIN, st);
    VAEQ_LAUNCH_CHECK("k_dp_fin");
    return VAEQ_OK;
}

static int dp_launch_adam(const DpK &p, int nparts, int mode, float lr_w, float lr_h, int amsgrad, cudaStream_t st) {
    ktime_begin(VAEQ_K_DP_ADAM, st);
    k_dp_adam<<<(16 * p.M + ADAM_EPC - 1) / ADAM_EPC, ADAM_TPE * ADAM_EPC, 0, st>>>(p, nparts, mode == DP_MODE_TRAIN ? 1 : 0, lr_w, lr_h, amsgrad);
    ktime_end(VAEQ_K_DP_ADAM, st);
    VAEQ_LAUNCH_CHECK("k_dp_adam");
    return VAEQ_OK;
}

template <int NL>
static int dp_run(const DpK &p, int mode, float lr_w, float lr_h, int amsgrad, cudaStream_t st) {
    static int grid_fwd_c[VAEQ_MAX_DEVICES][VAEQ_MAX_TAPS + 1] = {{0}}, grid_bwd_c[VAEQ_MAX_DEVICES][VAEQ_MAX_TAPS + 1] = {{0}};   // cached per device and M_est
    static SmemAttrCache set_f, set_b;
    int *grid_fwd = grid_fwd_c[cur_device()], *grid_bwd = grid_bwd_c[cur_device()];
    const size_t sm_f = dp_fwd_smem(p.M, p.T, p.H, p.mh), sm_b = dp_bwd_smem(p.M, p.T, p.H, p.mh);
    if (int rc = ensure_dyn_smem(k_dp_fwd<NL>, sm_f, set_f)) return rc;
    if (int rc = ensure_dyn_smem(k_dp_bwd<NL>, sm_b, set_b)) return rc;
    if (!grid_fwd[p.M]) {
        int per = 0;
        VAEQ_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per, k_dp_fwd<NL>, DP_NT, sm_f));
        grid_fwd[p.M] = max(1, per) * sm_count();
        VAEQ_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per, k_dp_bwd<NL>, DP_NT, sm_b));
        grid_bwd[p.M] = max(1, per) * sm_count();
    }
    const int gf = min(min(grid_fwd[p.M], DP_GRID_CAP), p.ntiles), gb = min(min(grid_bwd[p.M], DP_GRID_CAP), p.ntiles);
    ktime_begin(VAEQ_K_DP_FWD, st);
    k_dp_fwd<NL><<<gf, DP_NT, sm_f, st>>>(p);
    ktime_end(VAEQ_K_DP_FWD, st);
    VAEQ_LAUNCH_CHECK("k_dp_fwd");
    {
        const int rc = dp_launch_fin(p, gf, st);
        if (rc) return rc;
    }
    if (mode == DP_MODE_FWD) return VAEQ_OK;
    ktime_begin(VAEQ_K_DP_BWD, st);
    k_dp_bwd<NL><<<gb, DP_NT, sm_b, st>>>(p);
    ktime_end(VAEQ_K_DP_BWD, st);
    VAEQ_LAUNCH_CHECK("k_dp_bwd");
    return dp_launch_adam(p, gb, mode, lr_w, lr_h, amsgrad, st);
}

static bool g_force_generic = false;

static int dp_dispatch(const DpK &p, int n_lev, int mode, float lr_w, float lr_h, int amsgrad, cudaStream_t st) {
    if (!g_force_generic) {
        int gb = 0, rc = VAEQ_OK;
        if (p.dyn) VAEQ_CUDA(cudaMemsetAsync(p.tile_ctr, 0, 4 * sizeof(int), st));
        if (dp_try_fast(p, n_lev, mode, st, &gb, &rc)) {
            if (rc || mode == DP_MODE_FWD) return rc;
            return dp_launch_adam(p, gb, mode, lr_w, lr_h, amsgrad, st);
        }
    }
    switch (n_lev) {
        case 2: return dp_run<2>(p, mode, lr_w, lr_h, amsgrad, st);
        case 4: return dp_run<4>(p, mode, lr_w, lr_h, amsgrad, st);
        default: return dp_run<8>(p, mode, lr_w, lr_h, amsgrad, st);
    }
}

}  // namespace vaeq

using namespace vaeq;

extern "C" size_t vaeq_dp_workspace_bytes(int32_t B, int32_t M, int32_t n_lev) {
    (void)n_lev;
    if (B <= 0 || M <= 0) return 0;
    return dp_ws_layout(B, M).total;
}

extern "C" size_t vaeq_adam_state_floats(int32_t M) { return (size_t)48 * M + 4; }

extern "C" size_t vaeq_dp_runs_workspace_bytes(int32_t B, int32_t M, int32_t n_lev, int32_t n_runs) {
    if (B <= 0 || M <= 0 || n_runs <= 0) return 0;
    return g_persistent_frames_mode() == 2 ? (size_t)n_runs * vaeq_dp_workspace_bytes(B, M, n_lev) : 256;
}

extern "C" int32_t vaeq_dp_runs_max_batch_len(int32_t M, int32_t n_lev) {
    if (M < 1 || M > VAEQ_MAX_TAPS || !(M & 1) || (n_lev != 2 && n_lev != 4 && n_lev != 8)) return 0;
    return max(vaeq::dp_cluster_max_b(M), vaeq::dp_small_fits(DP_SMALL_MAX_B, M) ? DP_SMALL_MAX_B : 0);
}

extern "C" int vaeq_dp_dynamic_tiles(int32_t on) {
    g_dynamic_tiles = on != 0;
    return VAEQ_OK;
}

extern "C" int vaeq_dp_force_generic(int32_t on) {
    g_force_generic = on != 0;
    return VAEQ_OK;
}

extern "C" int vaeq_dp_forward(const vaeq_dp_desc *d, void *stream) {
    int rc = dp_validate(d, false, false);
    if (rc) return rc;
    return dp_dispatch(dp_make_params(d), d->n_lev, DP_MODE_FWD, 0.f, 0.f, 0, (cudaStream_t)stream);
}

extern "C" int vaeq_dp_forward_backward(const vaeq_dp_desc *d, void *stream) {
    int rc = dp_validate(d, true, false);
    if (rc) return rc;
    return dp_dispatch(dp_make_params(d), d->n_lev, DP_MODE_FWDBWD, 0.f, 0.f, 0, (cudaStream_t)stream);
}

// loss_function_shaping(q, rx, h_est, amp_levels, P) as an operator on an ARBITRARY q (sf:92-137): loss, var_est, and the
// gradients w.r.t. q and h_est.  Generic kernels only (the fused fast path differentiates through the equalizer instead).
extern "C" int vaeq_dp_loss_from_q(const vaeq_dp_desc *d, float *gq, int64_t ld_gq, void *stream) {
    VAEQ_CHECK_ARG(d != nullptr, "desc is NULL");
    VAEQ_CHECK_ARG(d->sps == 2, "sps=%d: only sps=2 is implemented", d->sps);
    VAEQ_CHECK_ARG(d->M >= 1 && d->M <= VAEQ_MAX_TAPS && (d->M & 1), "M_est=%d must be odd and <= %d", d->M, VAEQ_MAX_TAPS);
    VAEQ_CHECK_ARG(d->n_lev == 2 || d->n_lev == 4 || d->n_lev == 8, "n_lev=%d must be 2, 4 or 8", d->n_lev);
    VAEQ_CHECK_ARG(d->B > 2 * (d->M / 2), "batch_len=%d must exceed M_est-1", d->B);
    VAEQ_CHECK_ARG(d->rx && d->amp && d->P && d->h && d->q && d->loss && d->var_est, "NULL tensor pointer (rx, amp, P, h, q, loss, var_est)");
    VAEQ_CHECK_ARG(d->ld_rx >= (int64_t)d->B * d->sps && d->ld_q >= d->B && (!gq || ld_gq >= d->B), "row stride smaller than the row");
    VAEQ_CHECK_ARG(d->workspace != nullptr, "workspace is NULL");
    if (d->workspace_bytes < vaeq_dp_workspace_bytes(d->B, d->M, d->n_lev)) {
        set_error("workspace too small: %zu < %zu", d->workspace_bytes, vaeq_dp_workspace_bytes(d->B, d->M, d->n_lev));
        return VAEQ_EWORKSPACE;
    }
    DpK p = dp_make_params(d);
    p.from_q = 1;
    p.gq = gq;
    p.ld_gq = ld_gq;
    p.qk = nullptr;
    p.W = p.h;                                               // never dereferenced for its values: the FIR is skipped
    p.var = p.amp;                                           // (the demapper constants are unused as well)
    p.gW_out = nullptr;
    const bool need_grads = gq != nullptr || d->gh != nullptr;
    switch (d->n_lev) {
        case 2: return dp_run<2>(p, need_grads ? DP_MODE_FWDBWD : DP_MODE_FWD, 0.f, 0.f, 0, (cudaStream_t)stream);
        case 4: return dp_run<4>(p, need_grads ? DP_MODE_FWDBWD : DP_MODE_FWD, 0.f, 0.f, 0, (cudaStream_t)stream);
        default: return dp_run<8>(p, need_grads ? DP_MODE_FWDBWD : DP_MODE_FWD, 0.f, 0.f, 0, (cudaStream_t)stream);
    }
}

extern "C" int vaeq_dp_train_step(const vaeq_dp_desc *d, float lr_w, float lr_h, void *stream) {
    int rc = dp_validate(d, true, true);
    if (rc) return rc;
    return dp_dispatch(dp_make_params(d), d->n_lev, DP_MODE_TRAIN, lr_w, lr_h, (d->flags & VAEQ_F_AMSGRAD) ? 1 : 0,
                       (cudaStream_t)stream);
}


extern "C" int vaeq_dp_persistent_frames(int32_t mode) {
    VAEQ_CHECK_ARG(mode >= 0 && mode <= 2, "mode must be 0, 1 or 2");
    g_persistent_frames = mode;
    return VAEQ_OK;
}

namespace vaeq {
// one launch for the whole frame of every run (batch_len <= DP_TILE)
static int dp_frame_persistent(const vaeq_dp_desc *d, const vaeq_dp_runs *runs, int n_steps, int stride_sym, int keep_lo_in_dst,
                               float lr_w, float lr_h, float *loss_steps, float *var_est_steps, cudaStream_t st) {
    DpK p = dp_make_params(d);
    p.T = d->B;                                              // the minibatch is the tile: shared memory sized for it
    p.ntiles = 1;
    DpRunsK rs;
    memset(&rs, 0, sizeof(rs));
    const int n_runs = runs ? runs->n_runs : 1;
    if (runs) {
        rs.rs_rx = runs->rs_rx; rs.rs_amp = runs->rs_amp; rs.rs_P = runs->rs_P; rs.rs_var = runs->rs_var;
        rs.rs_W = runs->rs_W; rs.rs_h = runs->rs_h; rs.rs_adam = runs->rs_adam; rs.rs_q = runs->rs_q; rs.rs_out = runs->rs_out;
        rs.rs_qk = runs->rs_q_keep; rs.rs_outk = runs->rs_out_keep;
        rs.nu_sc = runs->nu_sc; rs.lr_w = runs->lr_w; rs.lr_h = runs->lr_h;
    }
    rs.ws_stride = (int64_t)vaeq_dp_workspace_bytes(d->B, d->M, d->n_lev);
    rs.loss_steps = loss_steps; rs.var_steps = var_est_steps;
    rs.loss_last = d->loss; rs.var_last = d->var_est; rs.gW_last = d->gW; rs.gh_last = d->gh;
    const size_t smem = max(dp_fwd_smem(p.M, p.T, p.H, p.mh), dp_bwd_smem(p.M, p.T, p.H, p.mh));
    const int amsgrad = (d->flags & VAEQ_F_AMSGRAD) ? 1 : 0;
    if (g_persistent_frames != 2) {
        if (runs && !dp_small_fits(d->B, d->M))
            return dp_cluster_launch(p, rs, d->n_lev, n_runs, n_steps, stride_sym, keep_lo_in_dst, lr_w, lr_h, amsgrad, st);
        return dp_small_launch(p, rs, d->n_lev, n_runs, n_steps, stride_sym, keep_lo_in_dst, lr_w, lr_h, amsgrad, st);
    }
    static SmemAttrCache set_smem[3];
#define FRAME_CASE(NL_, IDX_)                                                                                             \
    {                                                                                                                     \
        if (int rc_ = ensure_dyn_smem(k_dp_frame_small<NL_>, smem, set_smem[IDX_])) return rc_;                           \
        ktime_begin(VAEQ_K_DP_FRAME, st);                                                                                 \
        k_dp_frame_small<NL_><<<n_runs, DP_NT, smem, st>>>(p, rs, n_steps, stride_sym, keep_lo_in_dst, lr_w, lr_h, amsgrad); \
        ktime_end(VAEQ_K_DP_FRAME, st);                                                                                   \
    }
    if (d->n_lev == 2) FRAME_CASE(2, 0)
    else if (d->n_lev == 4) FRAME_CASE(4, 1)
    else FRAME_CASE(8, 2)
#undef FRAME_CASE
    VAEQ_LAUNCH_CHECK("k_dp_frame_small");
    return VAEQ_OK;
}
}  // namespace vaeq

extern "C" int vaeq_dp_train_frame(const vaeq_dp_desc *d, int32_t n_steps, int32_t stride_sym, int32_t keep_lo_in_dst,
                                   float lr_w, float lr_h, float *loss_steps, float *var_est_steps, void *stream) {
    int rc = dp_validate(d, true, true);
    if (rc) return rc;
    VAEQ_CHECK_ARG(n_steps >= 0 && stride_sym > 0, "bad n_steps/stride");
    VAEQ_CHECK_ARG(d->ld_rx >= ((int64_t)(n_steps - 1) * stride_sym + d->B) * d->sps, "frame shorter than the last window");
    if (n_steps == 0) return VAEQ_OK;
    // mode 1 (dp_small.cu) covers batch_len up to DP_SMALL_MAX_B, i.e. up to where the register-blocked fast path takes over for
    // single steps; mode 2 (generic bodies in one launch) needs the minibatch to be one tile
    if ((g_persistent_frames == 1 && dp_small_fits(d->B, d->M)) ||
        (g_persistent_frames == 2 && d->B <= DP_TILE))
        return dp_frame_persistent(d, nullptr, n_steps, stride_sym, keep_lo_in_dst, lr_w, lr_h, loss_steps, var_est_steps,
                                   (cudaStream_t)stream);
    DpK base = dp_make_params(d);
    for (int m = 0; m < n_steps; ++m) {
        DpK p = base;
        p.rx = d->rx + (int64_t)m * stride_sym * d->sps;
        p.keep_base = (int64_t)m * stride_sym + (keep_lo_in_dst ? d->keep_lo : 0);
        p.loss_out = loss_steps ? loss_steps + m : nullptr;
        p.var_est_out = var_est_steps ? var_est_steps + m : nullptr;
        p.var_est_stride = n_steps;
        rc = dp_dispatch(p, d->n_lev, DP_MODE_TRAIN, lr_w, lr_h, (d->flags & VAEQ_F_AMSGRAD) ? 1 : 0, (cudaStream_t)stream);
        if (rc) return rc;
    }
    return VAEQ_OK;
}

extern "C" int vaeq_dp_train_frame_runs(const vaeq_dp_desc *d, const vaeq_dp_runs *runs, int32_t n_steps, int32_t stride_sym,
                                        int32_t keep_lo_in_dst, float lr_w, float lr_h, float *loss_steps, float *var_est_steps,
                                        void *stream) {
    VAEQ_CHECK_ARG(d != nullptr && runs != nullptr && runs->n_runs >= 1, "desc / runs is NULL or n_runs < 1");
    if (g_persistent_frames == 2)
        VAEQ_CHECK_ARG(d->B <= DP_TILE && dp_small_smem(d->B, d->M) <= 220 * 1024,
                       "batched runs need batch_len <= %d and a shared-memory plan <= 220 KB (one CTA per run), got batch_len %d", DP_SMALL_MAX_B, d->B);
    else if (!dp_small_fits(d->B, d->M) && d->M >= 1 && d->M <= VAEQ_MAX_TAPS)   // above dp_small.cu's range: one cluster per run
        if (int rc = dp_cluster_check(d->B, d->M)) return rc;
    vaeq_dp_desc one = *d;
    static char dummy_ws;                                    // dp_small.cu keeps everything in shared memory: no workspace
    if (g_persistent_frames == 2) {
        one.workspace_bytes = d->workspace_bytes / (size_t)runs->n_runs;  // the generic bodies need a full workspace per run
    } else {
        one.workspace = d->workspace ? d->workspace : &dummy_ws;
        one.workspace_bytes = vaeq_dp_workspace_bytes(d->B, d->M, d->n_lev);
    }
    int rc = dp_validate(&one, true, true);
    if (rc) return rc;
    VAEQ_CHECK_ARG(n_steps >= 0 && stride_sym > 0, "bad n_steps/stride");
    VAEQ_CHECK_ARG(d->ld_rx >= ((int64_t)(n_steps - 1) * stride_sym + d->B) * d->sps, "frame shorter than the last window");
    if (n_steps == 0) return VAEQ_OK;
    return dp_frame_persistent(d, runs, n_steps, stride_sym, keep_lo_in_dst, lr_w, lr_h, loss_steps, var_est_steps, (cudaStream_t)stream);
}

// ---- batch-split phases (SURVEY.md §8e): the host all-reduces `stats` and `grads` between them ----------------
namespace vaeq {
__global__ void k_dp_pack_stats(DpK p, int nparts, double *stats) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (wid < 5) {
        double a = 0.0;
        for (int b = lane; b < nparts; b += 32) a += p.part_fwd[(int64_t)b * 8 + wid];
        a = warp_sum(a);
        if (lane == 0) stats[wid] = a;
    }
    if (threadIdx.x >= 5 && threadIdx.x < 8) stats[threadIdx.x] = 0.0;
    for (int i = threadIdx.x; i < 4 * p.mh; i += blockDim.x) stats[8 + i] = (double)p.edge_vs[i];
}
__global__ void k_dp_unpack_stats(DpK p, const double *stats) {
    if (threadIdx.x < 8) p.part_fwd[threadIdx.x] = stats[threadIdx.x];
    for (int i = threadIdx.x; i < 4 * p.mh; i += blockDim.x) p.edge_vs[i] = (float)stats[8 + i];
}
__global__ void k_dp_reduce_gpart(DpK p, int nparts, float *grads) {
    const int n = 16 * p.M, lane = threadIdx.x & 31, i = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (i >= n) return;
    double a = 0.0;
    for (int b = lane; b < nparts; b += 32) a += (double)p.gpart[(int64_t)b * n + i];
    a = warp_sum(a);
    if (lane == 0) grads[i] = (float)a;
}
// ---- one-shot peer reductions over NVLink (vaeq_dp_split_step_peer) --------------------------------------------------------------
// PUSH model, flag-in-word ("LL") protocol: every rank owns a slot in symmetric memory with one COMPARTMENT per sender.  A reduction is:
// store my partial into compartment `rank` of EVERY peer's slot as 8-byte words {payload32, epoch32} (remote stores pipeline over NVLink;
// nobody reads remote memory; an aligned 8-byte store arrives whole), then poll the words of MY OWN slot (local memory) until each carries
// the epoch of this exchange and add the payloads in rank order, so all ranks compute bit-identical sums (the replicated Adam step depends
// on it).  No fence and no separate flag: one NVLink store latency per exchange, independent of the number of ranks (the fence + epoch-word
// version this replaces cost two more NVLink round trips: fin 10.6 -> 24 us, Adam 10 -> 27 us at N = 4, profiles/r02c_batch_split.txt).
// The two exchanges of a step alternate, which is what makes one buffer per exchange enough: nobody can send exchange k + 1 before
// everybody has read exchange k (see include/vaeq.h).
struct PeerK {
    int rank, world;
    unsigned char *slot[VAEQ_MAX_PEERS];
    int *epoch;                                              // local: [0] ELBO-sum exchanges done, [1] gradient exchanges done
    int comp;                                                // bytes per compartment
};
constexpr int PEER_HDR = 256;                                // reserved
__host__ __device__ inline size_t peer_stats_bytes(int M) { return (size_t)(8 + 4 * (M / 2)) * 2 * sizeof(unsigned long long); }   // a double = two words
__host__ __device__ inline size_t peer_comp_bytes(int M) { return (PEER_HDR + peer_stats_bytes(M) + (size_t)16 * M * sizeof(unsigned long long) + 255) / 256 * 256; }
__device__ __forceinline__ void st_word_sys(unsigned long long *p, unsigned payload, unsigned epoch) {
    const unsigned long long v = ((unsigned long long)epoch << 32) | payload;
    asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long globaltimer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
// spin on a word of my own slot until its epoch half is `epoch` (a sender that never arrives traps after 20 s); returns the payload
__device__ __forceinline__ unsigned ld_word_wait(const unsigned long long *p, unsigned epoch) {
    unsigned long long v;
    asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    if ((unsigned)(v >> 32) != epoch) {
        const unsigned long long t0 = globaltimer_ns();
        do {
            if (globaltimer_ns() - t0 > 20000000000ull) __trap();
            asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
        } while ((unsigned)(v >> 32) != epoch);
    }
    return (unsigned)v;
}
__global__ void __launch_bounds__(256) k_dp_peer_reduce_stats(DpK p, int nparts, PeerK c) {
    __shared__ double st[8 + 4 * (VAEQ_MAX_TAPS / 2)];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, ns = 8 + 4 * p.mh;
    const unsigned e = (unsigned)(*reinterpret_cast<volatile int *>(c.epoch) + 1);
    if (wid < 5) {
        double a = 0.0;
        for (int b = lane; b < nparts; b += 32) a += p.part_fwd[(int64_t)b * 8 + wid];
        a = warp_sum(a);
        if (lane == 0) st[wid] = a;
    }
    if (threadIdx.x >= 5 && threadIdx.x < 8) st[threadIdx.x] = 0.0;
    for (int i = threadIdx.x; i < 4 * p.mh; i += blockDim.x) st[8 + i] = (double)p.edge_vs[i];
    __syncthreads();
    for (int idx = threadIdx.x; idx < c.world * 2 * ns; idx += blockDim.x) {  // my sums -> compartment `rank` of every slot, low / high half of each double
        const int r = idx / (2 * ns), w = idx - r * (2 * ns);
        const unsigned long long bits = (unsigned long long)__double_as_longlong(st[w >> 1]);
        st_word_sys(reinterpret_cast<unsigned long long *>(c.slot[r] + (size_t)c.rank * c.comp + PEER_HDR) + w, (unsigned)(bits >> (32 * (w & 1))), e);
    }
    for (int i = threadIdx.x; i < ns; i += blockDim.x) {
        double a = 0.0;
        for (int r = 0; r < c.world; ++r) {
            const unsigned long long *w = reinterpret_cast<const unsigned long long *>(c.slot[c.rank] + (size_t)r * c.comp + PEER_HDR) + 2 * i;
            const unsigned lo = ld_word_wait(w, e), hi = ld_word_wait(w + 1, e);
            a += __longlong_as_double((long long)(((unsigned long long)hi << 32) | lo));
        }
        if (i < 8) p.part_fwd[i] = a;
        else p.edge_vs[i - 8] = (float)a;
    }
    __syncthreads();                                         // the block's own global writes are visible to the block after the barrier
    if (threadIdx.x == 0) c.epoch[0] = (int)e;
    dp_fin_body(p, 1);                                       // C, loss, var_est, kappa, S_nu(j) from the reduced sums (k_dp_fin's body)
}
// gradients, sender side: a warp sums the per-CTA partials of one gradient entry in the fixed order of k_dp_reduce_gpart (same float) and its
// first `world` lanes store it straight into compartment `rank` of the peers' slots -- the push leaves from the many-CTA reduction kernel, the
// single-CTA kernel below only collects
__global__ void k_dp_reduce_gpart_push(DpK p, int nparts, PeerK c) {
    const int n = 16 * p.M, lane = threadIdx.x & 31, i = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (i >= n) return;
    const unsigned e = (unsigned)(*reinterpret_cast<volatile int *>(c.epoch + 1) + 1);
    double a = 0.0;
    for (int b = lane; b < nparts; b += 32) a += (double)p.gpart[(int64_t)b * n + i];
    a = warp_sum(a);
    const float g = __shfl_sync(0xffffffffu, (float)a, 0);
    if (lane < c.world)
        st_word_sys(reinterpret_cast<unsigned long long *>(c.slot[lane] + (size_t)c.rank * c.comp + PEER_HDR + peer_stats_bytes(p.M)) + i, __float_as_uint(g), e);
}
// gradients, receiver side: the sum over the ranks (rank order), then the replicated Adam step
__global__ void __launch_bounds__(1024) k_dp_peer_reduce_grads_adam(DpK p, PeerK c, float lr_w, float lr_h, int amsgrad) {
    __shared__ float sum_sh[16 * VAEQ_MAX_TAPS];
    const size_t off = PEER_HDR + peer_stats_bytes(p.M);
    const int n = 16 * p.M;
    const unsigned e = (unsigned)(*reinterpret_cast<volatile int *>(c.epoch + 1) + 1);
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        double a = 0.0;
        for (int r = 0; r < c.world; ++r)
            a += (double)__uint_as_float(ld_word_wait(reinterpret_cast<const unsigned long long *>(c.slot[c.rank] + (size_t)r * c.comp + off) + i, e));
        sum_sh[i] = (float)a;                                // a float, like the all-reduced gradient of the NCCL transport
    }
    // ---- replicated Adam on the reduced gradient (k_dp_adam's finish for one "partial"), step counter bumped by this single CTA ----
    __shared__ double bc1_sh;
    __shared__ float bc2s_sh;
    int *step_ptr = reinterpret_cast<int *>(p.adam + 48 * p.M);
    const int step = *step_ptr + 1;
    if (threadIdx.x == blockDim.x - 1) adam_bias(step, &bc1_sh, &bc2s_sh);
    __syncthreads();
    for (int i = threadIdx.x; i < n; i += blockDim.x) dp_adam_finish(p, i, (double)sum_sh[i], 1, lr_w, lr_h, amsgrad, bc1_sh, bc2s_sh);
    __syncthreads();
    if (threadIdx.x == 0) {
        *step_ptr = step;
        c.epoch[1] = (int)e;
    }
}
static int64_t split_cols(const vaeq_dp_desc *d, int32_t lo, int32_t hi) {      // columns a rank writes: its range widened by DP_SPLIT_EXT
    if (d == nullptr || lo < 0 || hi > d->B || lo >= hi) return -1;                // (bad ranges are reported by split_check)
    return (int64_t)min(d->B, hi + DP_SPLIT_EXT) - max(0, lo - DP_SPLIT_EXT);
}
static int split_check(const vaeq_dp_desc *d, int32_t lo, int32_t hi) {
    VAEQ_CHECK_ARG(lo >= 0 && hi <= d->B && lo < hi && lo % 4 == 0 && hi % 4 == 0, "bad symbol range [%d,%d) (multiples of 4 inside [0,B))", lo, hi);
    return VAEQ_OK;
}
}  // namespace vaeq

extern "C" size_t vaeq_dp_split_stats_doubles(int32_t M) { return (size_t)8 + 4 * (M / 2); }

extern "C" int vaeq_dp_split_forward(const vaeq_dp_desc *d, int32_t sym_lo, int32_t sym_hi, double *stats_out, void *stream) {
    int rc = dp_validate(d, false, false, split_cols(d, sym_lo, sym_hi));
    if (rc) return rc;
    if ((rc = split_check(d, sym_lo, sym_hi))) return rc;
    VAEQ_CHECK_ARG(stats_out != nullptr, "stats_out is NULL");
    cudaStream_t st = (cudaStream_t)stream;
    DpK p = dp_make_params(d);
    p.sym_lo = sym_lo; p.sym_hi = sym_hi;
    p.clo = max(0, sym_lo - DP_SPLIT_EXT); p.chi = min(d->B, sym_hi + DP_SPLIT_EXT);
    VAEQ_CUDA(cudaMemsetAsync(p.edge_vs, 0, 4 * (VAEQ_MAX_TAPS / 2 + 1) * sizeof(float), st));
    if (p.dyn) VAEQ_CUDA(cudaMemsetAsync(p.tile_ctr, 0, 4 * sizeof(int), st));
    int nparts = 0, rc2 = VAEQ_OK;
    if (!dp_try_fast(p, d->n_lev, DP_MODE_SPLIT_FWD, st, &nparts, &rc2)) {
        set_error("batch-split needs the fast path: M_est in {5,9,13,25}, 16-byte aligned rows, B %% 4 == 0, B >= 992");
        return VAEQ_EINVAL;
    }
    if (rc2) return rc2;
    ktime_begin(VAEQ_K_DP_FIN, st);
    k_dp_pack_stats<<<1, 256, 0, st>>>(p, nparts, stats_out);
    ktime_end(VAEQ_K_DP_FIN, st);
    VAEQ_LAUNCH_CHECK("k_dp_pack_stats");
    return VAEQ_OK;
}

extern "C" int vaeq_dp_split_backward(const vaeq_dp_desc *d, int32_t sym_lo, int32_t sym_hi, const double *stats_in,
                                      float *grads_out, void *stream) {
    int rc = dp_validate(d, false, false, 0);                // the backward kernels read the scratch rows, not q / out
    if (rc) return rc;
    if ((rc = split_check(d, sym_lo, sym_hi))) return rc;
    VAEQ_CHECK_ARG(stats_in && grads_out, "stats_in / grads_out is NULL");
    cudaStream_t st = (cudaStream_t)stream;
    DpK p = dp_make_params(d);
    p.sym_lo = sym_lo; p.sym_hi = sym_hi;
    p.clo = max(0, sym_lo - DP_SPLIT_EXT); p.chi = min(d->B, sym_hi + DP_SPLIT_EXT);
    k_dp_unpack_stats<<<1, 128, 0, st>>>(p, stats_in);
    VAEQ_LAUNCH_CHECK("k_dp_unpack_stats");
    if ((rc = dp_launch_fin(p, 1, st))) return rc;
    int nparts = 0, rc2 = VAEQ_OK;
    if (!dp_try_fast(p, d->n_lev, DP_MODE_SPLIT_BWD, st, &nparts, &rc2)) {
        set_error("batch-split needs the fast path");
        return VAEQ_EINVAL;
    }
    if (rc2) return rc2;
    ktime_begin(VAEQ_K_DP_ADAM, st);
    k_dp_reduce_gpart<<<(16 * p.M + 7) / 8, 256, 0, st>>>(p, nparts, grads_out);
    ktime_end(VAEQ_K_DP_ADAM, st);
    VAEQ_LAUNCH_CHECK("k_dp_reduce_gpart");
    return VAEQ_OK;
}

extern "C" int vaeq_dp_split_update(const vaeq_dp_desc *d, const float *grads_in, float lr_w, float lr_h, void *stream) {
    int rc = dp_validate(d, true, true, 0);                  // the update touches neither q nor out
    if (rc) return rc;
    VAEQ_CHECK_ARG(grads_in != nullptr, "grads_in is NULL");
    DpK p = dp_make_params(d);
    p.gpart = const_cast<float *>(grads_in);
    return dp_launch_adam(p, 1, DP_MODE_TRAIN, lr_w, lr_h, (d->flags & VAEQ_F_AMSGRAD) ? 1 : 0, (cudaStream_t)stream);
}

extern "C" size_t vaeq_peer_slot_bytes(int32_t M) { return (size_t)VAEQ_MAX_PEERS * peer_comp_bytes(M); }

extern "C" int vaeq_dp_split_step_peer(const vaeq_dp_desc *d, int32_t sym_lo, int32_t sym_hi, const vaeq_peer_comm *comm, float lr_w, float lr_h,
                                       void *stream) {
    int rc = dp_validate(d, true, true, split_cols(d, sym_lo, sym_hi));
    if (rc) return rc;
    if ((rc = split_check(d, sym_lo, sym_hi))) return rc;
    VAEQ_CHECK_ARG(comm != nullptr && comm->world >= 1 && comm->world <= VAEQ_MAX_PEERS && comm->rank >= 0 && comm->rank < comm->world && comm->epoch != nullptr,
                   "bad peer communicator (world 1..%d, rank inside it, epoch counters)", VAEQ_MAX_PEERS);
    PeerK c;
    c.rank = comm->rank; c.world = comm->world; c.epoch = comm->epoch; c.comp = (int)peer_comp_bytes(d->M);
    for (int r = 0; r < VAEQ_MAX_PEERS; ++r) {
        c.slot[r] = r < comm->world ? static_cast<unsigned char *>(comm->slot[r]) : nullptr;
        VAEQ_CHECK_ARG(r >= comm->world || (c.slot[r] != nullptr && reinterpret_cast<uintptr_t>(c.slot[r]) % 16 == 0), "peer slot %d is NULL or unaligned", r);
    }
    cudaStream_t st = (cudaStream_t)stream;
    DpK p = dp_make_params(d);
    p.sym_lo = sym_lo; p.sym_hi = sym_hi;
    p.clo = max(0, sym_lo - DP_SPLIT_EXT); p.chi = min(d->B, sym_hi + DP_SPLIT_EXT);
    VAEQ_CUDA(cudaMemsetAsync(p.edge_vs, 0, 4 * (VAEQ_MAX_TAPS / 2 + 1) * sizeof(float), st));
    if (p.dyn) VAEQ_CUDA(cudaMemsetAsync(p.tile_ctr, 0, 4 * sizeof(int), st));
    int nparts = 0, rc2 = VAEQ_OK;
    if (!dp_try_fast(p, d->n_lev, DP_MODE_SPLIT_FWD, st, &nparts, &rc2)) {
        set_error("batch-split needs the fast path: M_est in {5,9,13,25}, 16-byte aligned rows, B %% 4 == 0, B >= 992");
        return VAEQ_EINVAL;
    }
    if (rc2) return rc2;
    ktime_begin(VAEQ_K_DP_FIN, st);
    k_dp_peer_reduce_stats<<<1, 256, 0, st>>>(p, nparts, c);               // exchange of the ELBO sums + C, loss, var_est, kappa, S_nu(j)
    ktime_end(VAEQ_K_DP_FIN, st);
    VAEQ_LAUNCH_CHECK("k_dp_peer_reduce_stats");
    if (!dp_try_fast(p, d->n_lev, DP_MODE_SPLIT_BWD, st, &nparts, &rc2)) {
        set_error("batch-split needs the fast path");
        return VAEQ_EINVAL;
    }
    if (rc2) return rc2;
    ktime_begin(VAEQ_K_DP_ADAM, st);
    k_dp_reduce_gpart_push<<<(16 * p.M + 7) / 8, 256, 0, st>>>(p, nparts, c);
    k_dp_peer_reduce_grads_adam<<<1, 1024, 0, st>>>(p, c, lr_w, lr_h, (d->flags & VAEQ_F_AMSGRAD) ? 1 : 0);   // exchange of the gradients + Adam
    ktime_end(VAEQ_K_DP_ADAM, st);
    VAEQ_LAUNCH_CHECK("k_dp_peer_reduce_grads_adam");
    return VAEQ_OK;
}

extern "C" int vaeq_adam_update(float *param, const float *grad, float *state, int32_t n, float lr, int32_t amsgrad,
                                int32_t *step_count, int32_t bump_step, void *stream) {
    VAEQ_CHECK_ARG(param && grad && state && step_count && n > 0, "bad adam arguments");
    ktime_begin(VAEQ_K_OTHER, (cudaStream_t)stream);
    k_adam_generic<<<1, 256, 0, (cudaStream_t)stream>>>(param, grad, state, n, lr, amsgrad, step_count, bump_step);
    ktime_end(VAEQ_K_OTHER, (cudaStream_t)stream);
    VAEQ_LAUNCH_CHECK("k_adam_generic");
    return VAEQ_OK;
}

extern "C" int vaeq_soft_dec(const float *out, int64_t ld_out, const float *var, const float *amp, float nu_sc,
                             int32_t n_lev, int32_t N, float *q, int64_t ld_q, void *stream) {
    VAEQ_CHECK_ARG(out && var && amp && q && N > 0, "bad soft_dec arguments");
    VAEQ_CHECK_ARG(n_lev == 2 || n_lev == 4 || n_lev == 8, "n_lev=%d must be 2, 4 or 8", n_lev);
    const int nt = 256;
    cudaStream_t st = (cudaStream_t)stream;
    const bool vec = (N % 4 == 0) && (ld_out % 4 == 0) && (ld_q % 4 == 0) &&
                     ((reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(q)) % 16 == 0);
    if (vec) {
        const int gridv = min((N / 4 + nt - 1) / nt, sm_count() * 8);
        ktime_begin(VAEQ_K_EVAL, st);
        if (n_lev == 2) k_soft_dec_vec<2><<<gridv, nt, 0, st>>>(out, ld_out, var, amp, nu_sc, N, q, ld_q);
        else if (n_lev == 4) k_soft_dec_vec<4><<<gridv, nt, 0, st>>>(out, ld_out, var, amp, nu_sc, N, q, ld_q);
        else k_soft_dec_vec<8><<<gridv, nt, 0, st>>>(out, ld_out, var, amp, nu_sc, N, q, ld_q);
        ktime_end(VAEQ_K_EVAL, st);
        VAEQ_LAUNCH_CHECK("k_soft_dec_vec");
        return VAEQ_OK;
    }
    const int grid = min((N + nt - 1) / nt, sm_count() * 8);
    ktime_begin(VAEQ_K_EVAL, st);
    if (n_lev == 2) k_soft_dec<2><<<grid, nt, 0, st>>>(out, ld_out, var, amp, nu_sc, N, q, ld_q);
    else if (n_lev == 4) k_soft_dec<4><<<grid, nt, 0, st>>>(out, ld_out, var, amp, nu_sc, N, q, ld_q);
    else k_soft_dec<8><<<grid, nt, 0, st>>>(out, ld_out, var, amp, nu_sc, N, q, ld_q);
    ktime_end(VAEQ_K_EVAL, st);
    VAEQ_LAUNCH_CHECK("k_soft_dec");
    return VAEQ_OK;
}

// soft_dec for n_runs independent runs in one launch: out (n_runs,2,2,N), q (n_runs,2,2n,N) contiguous, var (n_runs,2), nu_sc (n_runs);
// the arithmetic per run is that of vaeq_soft_dec (same kernels, blockIdx.y = run)
extern "C" int vaeq_soft_dec_runs(const float *out, const float *var, const float *amp, const float *nu_sc, int32_t n_lev, int32_t N,
                                  int32_t n_runs, float *q, void *stream) {
    VAEQ_CHECK_ARG(out && var && amp && nu_sc && q && N > 0 && n_runs > 0 && n_runs <= 65535, "bad soft_dec_runs arguments");
    VAEQ_CHECK_ARG(n_lev == 2 || n_lev == 4 || n_lev == 8, "n_lev=%d must be 2, 4 or 8", n_lev);
    const int nt = 256;
    cudaStream_t st = (cudaStream_t)stream;
    const bool vec = (N % 4 == 0) && ((reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(q)) % 16 == 0);
    const int per = max(1, sm_count() * 8 / n_runs);
    ktime_begin(VAEQ_K_EVAL, st);
    if (vec) {
        const dim3 grid(max(1, min((N / 4 + nt - 1) / nt, per)), n_runs);
        if (n_lev == 2) k_soft_dec_vec<2><<<grid, nt, 0, st>>>(out, N, var, amp, 0.f, N, q, N, nu_sc);
        else if (n_lev == 4) k_soft_dec_vec<4><<<grid, nt, 0, st>>>(out, N, var, amp, 0.f, N, q, N, nu_sc);
        else k_soft_dec_vec<8><<<grid, nt, 0, st>>>(out, N, var, amp, 0.f, N, q, N, nu_sc);
    } else {
        const dim3 grid(max(1, min((N + nt - 1) / nt, per)), n_runs);
        if (n_lev == 2) k_soft_dec<2><<<grid, nt, 0, st>>>(out, N, var, amp, 0.f, N, q, N, nu_sc);
        else if (n_lev == 4) k_soft_dec<4><<<grid, nt, 0, st>>>(out, N, var, amp, 0.f, N, q, N, nu_sc);
        else k_soft_dec<8><<<grid, nt, 0, st>>>(out, N, var, amp, 0.f, N, q, N, nu_sc);
    }
    ktime_end(VAEQ_K_EVAL, st);
    VAEQ_LAUNCH_CHECK("k_soft_dec (runs)");
    return VAEQ_OK;
}
