// DP VAE frame kernel for minibatches that one CTA's shared memory cannot hold (batched runs above dp_small.cu's range):
// ONE THREAD-BLOCK CLUSTER per run (DESIGN.md §4c).
//
// The K CTAs of a cluster (K = 2, 4 or 8, one per SM) each own a contiguous slice of Bs symbols of the window and keep that slice's rx
// window, E_q, residual, dL/dout and backward coefficients in shared memory, plus a full replica of W, h and the Adam state.  A step is
// dp_small.cu's sequence of phases on the slice; the values that cross slices are read from the peers' shared memory (DSMEM) after a
// cluster barrier, three per step:
//   A  after the demapper:              E_q of the symbols next to the slice (halo of the channel convolution)
//   B  after the residual and partials: the residual e next to the slice (halo of dL/dE_q and dh), every CTA's ELBO partials, and the
//                                       edge variance sums of the first / last CTA (S_nu(j)); every CTA adds them in rank order
//   C  after the tap-gradient partials: every CTA adds the K partial gradients in rank order and runs Adam itself, so the replicas of the
//                                       taps stay bit-identical without a broadcast
// No float atomics: every sum has a fixed order, and K depends on (batch_len, M_est) only, so a run's result does not depend on the
// other runs of the launch.  A CTA rewrites a buffer its peers read only after the next barrier that follows their reads, and the frame
// ends with a cluster barrier so that no CTA exits while a peer may still read its shared memory.
// Same math as dp_small.cu (closed form in oracle/closed_form.py); the demapper takes the moment form when the prior allows it, like the
// single-run fast path.
#include <cooperative_groups.h>
#include "dp_math.cuh"
#include "dp_kernels.cuh"

namespace cg = cooperative_groups;

namespace vaeq {

constexpr int CL_NT = 256;
constexpr size_t CL_SMEM_MAX = 220 * 1024;

__device__ __forceinline__ void cluster_barrier() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ float cl_fneg(float v) { return __uint_as_float(__float_as_uint(v) ^ 0x80000000u); }
__device__ __forceinline__ void cl_cp_async4(void *dst_smem, const void *src_gmem) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(dst_smem);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(d), "l"(src_gmem) : "memory");
}

// per-CTA shared-memory plan (offsets in floats) for a slice of Bs symbols; identical in every CTA of the cluster, so a peer's array
// sits at the same offset as one's own
struct ClusterLayout {
    int XO, XA, SO, SA, HM;                 // margins (symbol positions per sample phase) and lengths of x, e, E_q
    int dsc, xph, m1s, eph, gys, Wt, hD, hG, part4, cst, srow, vsc, PS, Asum, edge, edgep, Wf, hf, adam, gpart, hsq, red, rec, scal, total;
};
__host__ __device__ inline ClusterLayout cluster_layout(int Bs, int M) {
    ClusterLayout l;
    const int mh = M / 2;
    l.XO = (mh + 1) / 2 + 1;
    l.XA = Bs + 2 * l.XO;
    l.SO = l.XO;
    l.SA = Bs + 2 * l.SO;
    l.HM = l.XO;
    int off = 0;
    auto take = [&](int nfloats) {
        int o = off;
        off += (nfloats + 3) & ~3;
        return o;
    };
    l.dsc = take(2 * 4);
    l.xph = take(2 * 4 * 2 * l.XA);         // double-buffered rx window of the slice, mh samples of margin on each side
    l.m1s = take(4 * (Bs + 2 * l.HM));      // E_q of the slice with a halo of HM symbols on each side
    l.eph = take(4 * 2 * l.SA);             // residual of the slice with a halo of SO symbol positions per phase on each side
    l.gys = take(4 * Bs);
    l.Wt = take(4 * 2 * M);
    l.hD = take(4 * 2 * M);
    l.hG = take(4 * 2 * M);
    l.part4 = take(4 * 3 * CL_NT);
    l.cst = take((int)(sizeof(FastConst) / 4));
    l.srow = take(12 * Bs);
    l.vsc = take(2 * Bs);
    l.PS = take(4 * (M + 1));
    l.Asum = take(4);
    l.edge = take(2 * M);
    l.edgep = take(2 * M);                  // first CTA: left edge sums, last CTA: right edge sums (read by every CTA after barrier B)
    l.Wf = take(8 * M);
    l.hf = take(8 * M);
    l.adam = take(48 * M);
    l.gpart = take(16 * M);                 // this CTA's tap-gradient partials (dh without the 2 kappa factor; read after barrier C)
    l.hsq = take(4 * M);
    l.red = take(5 * 32);
    l.rec = take(8);                        // this CTA's ELBO partials C0, C1, entropy, Var0, Var1 (read after barrier B)
    l.scal = take(8);
    l.total = off;
    return l;
}

// slice length and cluster size: the smallest K in {2, 4, 8} whose per-CTA plan fits and whose last slice holds the mh edge symbols and
// the halos its neighbour reads; depends on (B, M) only.  Returns 0 if none fits.
static int cluster_plan(int B, int M, int *Bs_out) {
    const int mh = M / 2;
    for (int K = 2; K <= 8; K *= 2) {
        const int Bs = (B + K - 1) / K, last = B - (K - 1) * Bs;
        const ClusterLayout l = cluster_layout(Bs, M);
        if ((size_t)l.total * sizeof(float) <= CL_SMEM_MAX && last >= mh + 1 && last >= l.HM) {
            *Bs_out = Bs;
            return K;
        }
    }
    return 0;
}

int dp_cluster_max_b(int M) {
    int lo = 0, hi = 1 << 16;                                // the plan grows with B: bisect the largest B that has one
    while (lo < hi) {
        const int mid = (lo + hi + 1) / 2;
        int Bs = 0;
        if (cluster_plan(mid, M, &Bs)) lo = mid;
        else hi = mid - 1;
    }
    return lo;
}

template <int NL, int MT>
__global__ void __launch_bounds__(CL_NT, 1) k_dp_frame_cluster(DpK p, DpRunsK rs, int Bs, int n_steps, int stride_sym, int keep_lo_in_dst,
                                                              float lr_w, float lr_h, int amsgrad) {
    extern __shared__ __align__(16) float sm[];
    cg::cluster_group cluster = cg::this_cluster();
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int rank = (int)cluster.block_rank(), K = (int)cluster.num_blocks(), run = blockIdx.y;
    const int B = p.B, L = 2 * p.B, M = MT ? MT : p.M, mh = M / 2, Mh = 2 * mh;
    const int u0 = rank * Bs, nb = min(Bs, B - u0);         // owned symbols [u0, u0 + nb), samples [2 u0, 2 u0 + 2 nb)
    const ClusterLayout lay = cluster_layout(Bs, M);
    const int XA = lay.XA, XO = lay.XO, SA = lay.SA, SO = lay.SO, HM = lay.HM;
    double *dsc = reinterpret_cast<double *>(sm + lay.dsc);
    // the local arrays are the window's arrays shifted by u0 symbols (2 u0 samples: the sample phases are the global ones)
    float4 *xph2 = reinterpret_cast<float4 *>(sm + lay.xph);     // [2 buffers][2 phases][XA]  [ph][a + XO] = rx[:, 2 (u0 + a) + ph]
    float4 *m1c = reinterpret_cast<float4 *>(sm + lay.m1s) + HM; // [-HM, Bs + HM) E_q {p0 I, p1 I, p0 Q, p1 Q}
    float4 *eph = reinterpret_cast<float4 *>(sm + lay.eph);      // [2][SA] residual {chi0 re, chi1 re, chi0 im, chi1 im}
    float4 *gys = reinterpret_cast<float4 *>(sm + lay.gys);
    float4 *Wt = reinterpret_cast<float4 *>(sm + lay.Wt);
    float4 *hD = reinterpret_cast<float4 *>(sm + lay.hD);
    float4 *hG = reinterpret_cast<float4 *>(sm + lay.hG);
    float4 *part4 = reinterpret_cast<float4 *>(sm + lay.part4);
    FastConst *cst = reinterpret_cast<FastConst *>(sm + lay.cst);
    float *srow = sm + lay.srow, *vsc = sm + lay.vsc, *PS = sm + lay.PS, *Asum = sm + lay.Asum, *edge = sm + lay.edge;
    float *edgep = sm + lay.edgep, *Wf = sm + lay.Wf, *hf = sm + lay.hf, *ad = sm + lay.adam, *gpart = sm + lay.gpart;
    float *hsq = sm + lay.hsq, *red = sm + lay.red, *rec = sm + lay.rec, *scal = sm + lay.scal;

    const float *rx0 = p.rx + run * rs.rs_rx;
    float *Wg = p.W + run * rs.rs_W, *hg = p.h + run * rs.rs_h, *adg = p.adam + run * rs.rs_adam;
    float *qk = p.qk ? p.qk + run * rs.rs_qk : nullptr, *outk = p.qk ? p.outk + run * rs.rs_outk : nullptr;
    if (rs.lr_w) lr_w = rs.lr_w[run];
    if (rs.lr_h) lr_h = rs.lr_h[run];
    const float nu_sc = rs.nu_sc ? rs.nu_sc[run] : p.nu_sc;
    const bool lead = rank == 0;                             // writes the run's scalar outputs and trained state (all CTAs hold the same)

    auto issue_window = [&](int m) {
        const float *rx = rx0 + (int64_t)m * stride_sym * 2;
        float4 *dst = xph2 + (m & 1) * 2 * XA;
        for (int idx = tid; idx < 2 * XA; idx += CL_NT) {
            const int ph = idx >= XA, a = idx - ph * XA - XO, s = 2 * (u0 + a) + ph;
            if (s >= 0 && s < L) {
                float *d4 = reinterpret_cast<float *>(dst + idx);
#pragma unroll
                for (int r = 0; r < 4; ++r) cl_cp_async4(d4 + ((r & 1) * 2 + (r >> 1)), rx + r * p.ld_rx + s);
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };

    for (int i = tid; i < 8 * M; i += CL_NT) {
        Wf[i] = Wg[i];
        hf[i] = hg[i];
    }
    for (int i = tid; i < 48 * M; i += CL_NT) ad[i] = adg[i];
    const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int i = tid; i < 2 * SA; i += CL_NT) eph[i] = z4;   // halos at the true window edges and samples past L stay zero
    for (int i = tid; i < 4 * XA; i += CL_NT) xph2[i] = z4;
    for (int i = tid; i < Bs + 2 * HM; i += CL_NT) m1c[i - HM] = z4;
    load_fast_const(cst, p.amp + run * rs.rs_amp, p.P + run * rs.rs_P, p.var + run * rs.rs_var, nu_sc, NL);
    const int step0 = *reinterpret_cast<const int *>(adg + 48 * M);
    const double width = (double)(L - Mh);
    double b1t = 1.0, b2t = 1.0;
    if (tid == 0) {
        b1t = pow(0.9, (double)step0);
        b2t = pow(0.999, (double)step0);
    }
    __syncthreads();
    issue_window(0);
    const FastConst &c = *cst;
    const bool mom = c.quad != 0;

    for (int m = 0; m < n_steps; ++m) {
        const int64_t keep_base = (int64_t)m * stride_sym + (keep_lo_in_dst ? p.keep_lo : 0);
        const bool last = m == n_steps - 1;
        const float4 *xph = xph2 + (m & 1) * 2 * XA;

        // ---- P0: tap tables, Adam bias corrections, |h|^2 prefix sums (as dp_small.cu) ----------------------------------------
        for (int idx = tid; idx < 2 * M; idx += CL_NT) {
            const int o = idx / M, k = idx - o * M;
            Wt[idx] = make_float4(Wf[(o * 4 + 0) * M + k], Wf[(o * 4 + 1) * M + k], Wf[(o * 4 + 2) * M + k], Wf[(o * 4 + 3) * M + k]);
            hD[idx] = make_float4(hf[((o * 2 + 0) * 2 + 0) * M + k], hf[((o * 2 + 1) * 2 + 0) * M + k],
                                  hf[((o * 2 + 0) * 2 + 1) * M + k], hf[((o * 2 + 1) * 2 + 1) * M + k]);
            hG[idx] = make_float4(hf[((0 * 2 + o) * 2 + 0) * M + k], hf[((1 * 2 + o) * 2 + 0) * M + k],
                                  hf[((0 * 2 + o) * 2 + 1) * M + k], hf[((1 * 2 + o) * 2 + 1) * M + k]);
        }
        if (tid == 0) {
            b1t *= 0.9;
            b2t *= 0.999;
            dsc[0] = 1.0 - b1t;
            scal[6] = sqrtf((float)(1.0 - b2t));
        }
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncthreads();
        if (!last) issue_window(m + 1);
        if (wid >= 4) {
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

        // ---- P1: butterfly FIR of the slice's symbols, then the soft demapper (moments, entropy, backward coefficients) --------
        float accEnt = 0.f, accV0 = 0.f, accV1 = 0.f;
        for (int u = tid; u < nb; u += CL_NT) {
            const float2 z2 = make_float2(0.f, 0.f);
            float2 re0 = z2, im0 = z2, re1 = z2, im1 = z2;
#pragma unroll
            for (int ph = 0; ph < 2; ++ph) {
                const int k0 = (mh + ph) & 1;
                const float4 *xb = xph + ph * XA + u + XO + ((k0 - mh - ph) >> 1);
                const float4 *wb0 = Wt + k0, *wb1 = Wt + M + k0;
                const int n = (M - k0 + 1) >> 1;
#pragma unroll 4
                for (int i = 0; i < n; ++i) {
                    const float4 x = xb[i], wa = wb0[2 * i], wc = wb1[2 * i];
                    const float2 xI = make_float2(x.x, x.y), xQ = make_float2(x.z, x.w), nxQ = make_float2(cl_fneg(x.z), cl_fneg(x.w));
                    const float2 ar = make_float2(wa.x, wa.y), ai = make_float2(wa.z, wa.w), cr = make_float2(wc.x, wc.y), ci = make_float2(wc.z, wc.w);
                    re0 = __ffma2_rn(ar, xI, re0); re0 = __ffma2_rn(ai, nxQ, re0);
                    im0 = __ffma2_rn(ar, xQ, im0); im0 = __ffma2_rn(ai, xI, im0);
                    re1 = __ffma2_rn(cr, xI, re1); re1 = __ffma2_rn(ci, nxQ, re1);
                    im1 = __ffma2_rn(cr, xQ, im1); im1 = __ffma2_rn(ci, xI, im1);
                }
            }
            gys[u] = make_float4(re0.x + re0.y, im0.x + im0.y, re1.x + re1.y, im1.x + im1.y);
        }
        __syncthreads();
        for (int it = tid; it < 2 * nb; it += CL_NT) {
            const int o = it >= nb, u = it - o * nb, ug = u0 + u;
            const float2 y2 = reinterpret_cast<const float2 *>(gys + u)[o];
            const float yc[2] = {y2.x, y2.y};
            const bool keep = qk != nullptr && ug >= p.keep_lo && ug < p.keep_lo + p.keep_n;
            const int64_t col = keep_base + (ug - p.keep_lo);
            float vsum = 0.f;
#pragma unroll
            for (int cq = 0; cq < 2; ++cq) {
                const int cc = 2 * o + cq;
                float q[NL], m1, vq, ent, S1, T2, S3;
                if (mom) {
                    demap_mom<NL>(yc[cq], c.ct[o], c.eps[o], c.inv_var[o], c, q, m1, vq, ent, S1, T2, S3);
                } else {
                    float m2, S2;
                    demap_fast<NL, true>(yc[cq], c.c2[o], c.inv_var[o], c, q, m1, m2, ent, S1, S2, S3);
                    vq = m2 - m1 * m1;
                    T2 = fmaf(-2.f * m1, S1, S2);
                }
                if (keep) {
#pragma unroll
                    for (int l = 0; l < NL; ++l) qk[(int64_t)(cc * NL + l) * p.ld_qk + col] = q[l];
                    outk[(int64_t)cc * p.ld_outk + col] = yc[cq];
                }
                reinterpret_cast<float *>(m1c + u)[cq * 2 + o] = m1;
                srow[cc * Bs + u] = S1;
                srow[(4 + cc) * Bs + u] = T2;
                srow[(8 + cc) * Bs + u] = S3;
                vsum += vq;
                if (ug >= mh && ug < B - mh) accEnt += ent;
            }
            vsc[o * Bs + u] = vsum;
            if (o) accV1 += vsum; else accV0 += vsum;
        }
        cluster_barrier();                                   // A: every slice's E_q is complete

        // E_q halo of the channel convolution from the neighbours' slices
        for (int i = tid; i < 2 * HM; i += CL_NT) {
            const int right = i >= HM, a = right ? nb + i - HM : i - HM;
            if (right ? rank + 1 < K : rank > 0) {
                const float4 *peer = cluster.map_shared_rank(m1c, right ? rank + 1 : rank - 1);
                m1c[a] = peer[right ? a - nb : a + Bs];
            }
        }
        __syncthreads();

        // ---- P3: D = h * E_q and the residual on the slice's samples; ELBO partials; edge variance sums of the end slices ------
        float accC0 = 0.f, accC1 = 0.f;
        for (int s = tid; s < 2 * nb; s += CL_NT) {
            const int sg = 2 * u0 + s;
            float er0 = 0.f, ei0 = 0.f, er1 = 0.f, ei1 = 0.f;
            if (sg >= mh && sg < L - mh) {
                const float2 z2 = make_float2(0.f, 0.f);
                float2 dr0 = z2, di0 = z2, dr1 = z2, di1 = z2;
                const int par = (s + mh) & 1;
                const float4 *hb0 = hD + par, *hb1 = hD + M + par;
                const float4 *mb = m1c + ((s + mh - par) >> 1);
                const int n = (M - par + 1) >> 1;
#pragma unroll 4
                for (int i = 0; i < n; ++i) {
                    const float4 mm = mb[-i], ha = hb0[2 * i], hc = hb1[2 * i];
                    const float2 mI = make_float2(mm.x, mm.y), mQ = make_float2(mm.z, mm.w), nmQ = make_float2(cl_fneg(mm.z), cl_fneg(mm.w));
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
            eph[(s & 1) * SA + (s >> 1) + SO] = make_float4(er0, er1, ei0, ei1);
            accC0 += er0 * er0 + ei0 * ei0;
            accC1 += er1 * er1 + ei1 * ei1;
        }
        // edge_nu(j) = sum of Var over the source symbols u < u_lo(j) (first slice) and u > u_hi(j) (last slice)
        if (lead || rank == K - 1) {
            for (int idx = tid - (CL_NT - 2 * M); idx >= 0 && idx < 2 * M; idx += CL_NT) {
                const int nu = idx / M, j = idx - nu * M;
                float ed = 0.f;
                if (lead) {
                    const int u_lo = (Mh - j + 1) >> 1;
                    for (int u = 0; u < u_lo; ++u) ed += vsc[nu * Bs + u];
                } else {
                    const int u_hi = (L - 1 - j) >> 1;
                    for (int u = u_hi + 1; u < B; ++u) ed += vsc[nu * Bs + u - u0];
                }
                edgep[idx] = ed;
            }
        }
        {                                                    // this CTA's ELBO partials: warp sums, then the warps in order
            float v[5] = {accC0, accC1, accEnt, accV0, accV1};
#pragma unroll
            for (int i = 0; i < 5; ++i) v[i] = warp_sum(v[i]);
            if (lane == 0) {
#pragma unroll
                for (int i = 0; i < 5; ++i) red[i * 32 + wid] = v[i];
            }
            __syncthreads();
            if (tid < 5) {
                float a = red[tid * 32];
                for (int w = 1; w < CL_NT / 32; ++w) a += red[tid * 32 + w];
                rec[tid] = a;
            }
        }
        cluster_barrier();                                   // B: residuals, ELBO partials and edge sums of every slice are complete

        // residual halo of dL/dE_q and dh from the neighbours' slices; the edge sums of the two end slices
        for (int i = tid; i < 4 * SO; i += CL_NT) {
            const int right = i >= 2 * SO, r = i - right * 2 * SO, ph = r >= SO, k = r - ph * SO;
            const int a = right ? nb + k : k - SO;
            if (right ? rank + 1 < K : rank > 0) {
                const float4 *peer = cluster.map_shared_rank(eph, right ? rank + 1 : rank - 1);
                eph[ph * SA + SO + a] = peer[ph * SA + SO + (right ? a - nb : a + Bs)];
            }
        }
        for (int idx = tid; idx < 2 * M; idx += CL_NT)
            edge[idx] = cluster.map_shared_rank(edgep, 0)[idx] + cluster.map_shared_rank(edgep, K - 1)[idx];
        __syncthreads();

        // ---- P4: ELBO scalars from the K partials in rank order (bit-identical in every CTA) -----------------------------------
        if (wid == CL_NT / 32 - 1) {
            float b0 = 0.f, b1 = 0.f;
            for (int idx = lane; idx < 2 * M; idx += 32) {
                b0 += hsq[idx] * edge[idx];
                b1 += hsq[2 * M + idx] * edge[idx];
            }
            b0 = warp_sum(b0);
            b1 = warp_sum(b1);
            float t = 0.f;
            if (lane < 5) {
                for (int r = 0; r < K; ++r) t += cluster.map_shared_rank(rec, r)[lane];
            }
            float v[5];
#pragma unroll
            for (int i = 0; i < 5; ++i) v[i] = __shfl_sync(0xffffffffu, t, i);
            if (lane < 2) {
                const int chi = lane;
                const float vC = chi ? v[1] : v[0], vB = chi ? b1 : b0, vV = chi ? v[4] : v[3];
                const double C = (double)vC + ((double)v[3] * (double)Asum[chi * 2] + (double)v[4] * (double)Asum[chi * 2 + 1]) - (double)vB;
                const double term = width * log(C);
                scal[chi] = (float)(width / C);
                scal[2 + chi] = vV;
                const float ve = (float)(C / width);
                if (lead) {
                    if (rs.var_steps) rs.var_steps[((int64_t)run * 2 + chi) * n_steps + m] = ve;
                    if (last && rs.var_last) rs.var_last[2 * run + chi] = ve;
                }
                const double term1 = __shfl_sync(0x3u, term, 1);
                if (chi == 0 && lead) {
                    const float loss = (float)((-(double)v[2] + term) + term1);
                    if (rs.loss_steps) rs.loss_steps[(int64_t)run * n_steps + m] = loss;
                    if (last && rs.loss_last) rs.loss_last[run] = loss;
                }
            }
        }
        __syncthreads();
        const float kap0 = scal[0], kap1 = scal[1];

        // ---- P5: dL/dE_q = conj(h) (*) 2 kappa e, then dL/dout, one slice symbol (both tx pols) per item ----------------------
        for (int u = tid; u < nb; u += CL_NT) {
            const int ug = u0 + u;
            const float2 z2 = make_float2(0.f, 0.f);
            float2 gr0 = z2, gi0 = z2, gr1 = z2, gi1 = z2;
#pragma unroll
            for (int ph = 0; ph < 2; ++ph) {
                const int j0 = (mh + ph) & 1;
                const float4 *eb = eph + ph * SA + u + SO + ((j0 - mh - ph) >> 1);
                const float4 *hb0 = hG + j0, *hb1 = hG + M + j0;
                const int n = (M - j0 + 1) >> 1;
#pragma unroll 4
                for (int i = 0; i < n; ++i) {
                    const float4 e = eb[i], ha = hb0[2 * i], hc = hb1[2 * i];
                    const float2 eR = make_float2(e.x, e.y), eI = make_float2(e.z, e.w), neR = make_float2(cl_fneg(e.x), cl_fneg(e.y));
                    const float2 ar = make_float2(ha.x, ha.y), ai = make_float2(ha.z, ha.w), cr = make_float2(hc.x, hc.y), ci = make_float2(hc.z, hc.w);
                    gr0 = __ffma2_rn(ar, eR, gr0); gr0 = __ffma2_rn(ai, eI, gr0);
                    gi0 = __ffma2_rn(ar, eI, gi0); gi0 = __ffma2_rn(ai, neR, gi0);
                    gr1 = __ffma2_rn(cr, eR, gr1); gr1 = __ffma2_rn(ci, eI, gr1);
                    gi1 = __ffma2_rn(cr, eI, gi1); gi1 = __ffma2_rn(ci, neR, gi1);
                }
            }
            const int jlo = max(0, Mh - 2 * ug), jhi = min(M, L - 2 * ug);
            const float entw = (ug >= mh && ug < B - mh) ? LN2 : 0.f;
            float g4[4];
#pragma unroll
            for (int nu = 0; nu < 2; ++nu) {
                const float2 gr2 = nu ? gr1 : gr0, gi2 = nu ? gi1 : gi0;
                const float gr = 2.f * (kap0 * gr2.x + kap1 * gr2.y), gi = 2.f * (kap0 * gi2.x + kap1 * gi2.y);
                const float gV = kap0 * (PS[(0 * 2 + nu) * (M + 1) + jhi] - PS[(0 * 2 + nu) * (M + 1) + jlo]) +
                                 kap1 * (PS[(1 * 2 + nu) * (M + 1) + jhi] - PS[(1 * 2 + nu) * (M + 1) + jlo]);
                const int cc = 2 * nu;
                g4[2 * nu] = fmaf(gr, srow[cc * Bs + u], fmaf(gV, srow[(4 + cc) * Bs + u], entw * srow[(8 + cc) * Bs + u]));
                g4[2 * nu + 1] = fmaf(gi, srow[(cc + 1) * Bs + u], fmaf(gV, srow[(5 + cc) * Bs + u], entw * srow[(9 + cc) * Bs + u]));
            }
            gys[u] = make_float4(g4[0], g4[1], g4[2], g4[3]);
        }
        __syncthreads();

        // ---- P6: the slice's tap-gradient partials (dp_small.cu's chunked tap-pair correlations over the slice) ---------------
        {
            const int kf0 = mh & 1, kf1 = (mh + 1) & 1;
            const int np0 = (((M - kf0 + 1) >> 1) + 1) >> 1, np1 = (((M - kf1 + 1) >> 1) + 1) >> 1, nps = np0 + np1;
            const int fam = wid >> 2, ft = tid & 127;
            const int items = fam == 0 ? nps : 2 * nps, parts = max(2, 2 * (64 / items)), chunk = ((nb + parts - 1) / parts) | 1;
            float4 *pbase = part4 + (fam == 0 ? 0 : 4 * 128);
            if ((ft >> 1) < items * (parts >> 1)) {
                const int item = (ft >> 1) % items, part = 2 * ((ft >> 1) / items) + (ft & 1);
                const int sel = fam == 0 ? 0 : item / nps, q = item - sel * nps, ph = q >= np0, kA = (ph ? kf1 : kf0) + 4 * (ph ? q - np0 : q);
                const int ua = min(nb, part * chunk), ub = min(nb, ua + chunk), off = (kA - mh - ph) >> 1;
                const float2 z2 = make_float2(0.f, 0.f);
                if (fam == 0) {
                    float2 a0r = z2, a0i = z2, a1r = z2, a1i = z2, b0r = z2, b0i = z2, b1r = z2, b1i = z2;
                    const float4 *wb = xph + ph * XA + XO + off;
                    float4 wa = wb[ua];
#pragma unroll 2
                    for (int u = ua; u < ub; ++u) {
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
                    float4 *dst = pbase + ft;
                    dst[0] = make_float4(a0r.x, a0i.x, a1r.x, a1i.x);
                    dst[128] = make_float4(a0r.y, a0i.y, a1r.y, a1i.y);
                    dst[256] = make_float4(b0r.x, b0i.x, b1r.x, b1i.x);
                    dst[384] = make_float4(b0r.y, b0i.y, b1r.y, b1i.y);
                } else {
                    float2 ar = z2, ai = z2, br = z2, bi = z2;
                    const float4 *wb = eph + ph * SA + SO + off;
                    const float *fb = reinterpret_cast<const float *>(m1c) + sel;
                    float4 wa = wb[ua];
#pragma unroll 4
                    for (int u = ua; u < ub; ++u) {
                        const float4 wn = wb[u + 1];
                        const float fI = fb[4 * u], fQ = fb[4 * u + 2];
                        const float2 fi2 = make_float2(fI, fI), fq2 = make_float2(fQ, fQ), nq2 = make_float2(-fQ, -fQ);
                        const float2 aR = make_float2(wa.x, wa.y), aI = make_float2(wa.z, wa.w), nR = make_float2(wn.x, wn.y), nI = make_float2(wn.z, wn.w);
                        ar = __ffma2_rn(aR, fi2, ar); ar = __ffma2_rn(aI, fq2, ar); ai = __ffma2_rn(aI, fi2, ai); ai = __ffma2_rn(aR, nq2, ai);
                        br = __ffma2_rn(nR, fi2, br); br = __ffma2_rn(nI, fq2, br); bi = __ffma2_rn(nI, fi2, bi); bi = __ffma2_rn(nR, nq2, bi);
                        wa = wn;
                    }
                    pbase[ft] = make_float4(ar.x, ai.x, ar.y, ai.y);
                    pbase[128 + ft] = make_float4(br.x, bi.x, br.y, bi.y);
                }
            }
            __syncthreads();
            if (ft < 4 * nps) {
                const int sel = fam == 0 ? (ft & 1) : ft / (2 * nps);
                const int q = fam == 0 ? (ft >> 2) : ((ft % (2 * nps)) >> 1), tb = fam == 0 ? ((ft >> 1) & 1) : (ft & 1);
                const int ph = q >= np0, kA = (ph ? kf1 : kf0) + 4 * (ph ? q - np0 : q);
                const int kk = kA + 2 * tb;
                if (kk < M) {
                    const int item = fam == 0 ? q : sel * nps + q, slot = fam == 0 ? tb * 2 + sel : tb;
                    const float4 *src = pbase + slot * 128 + 2 * item;
                    float4 sacc = src[0];
                    for (int part = 1; part < parts; ++part) {
                        const float4 t4 = src[2 * (part >> 1) * items + (part & 1)];
                        sacc.x += t4.x; sacc.y += t4.y; sacc.z += t4.z; sacc.w += t4.w;
                    }
                    if (fam == 0) {
                        gpart[(0 * 4 + sel) * M + kk] = sacc.x;
                        gpart[(0 * 4 + 2 + sel) * M + kk] = sacc.y;
                        gpart[(1 * 4 + sel) * M + kk] = sacc.z;
                        gpart[(1 * 4 + 2 + sel) * M + kk] = sacc.w;
                    } else {
                        gpart[8 * M + ((0 * 2 + sel) * 2 + 0) * M + kk] = sacc.x;
                        gpart[8 * M + ((0 * 2 + sel) * 2 + 1) * M + kk] = sacc.y;
                        gpart[8 * M + ((1 * 2 + sel) * 2 + 0) * M + kk] = sacc.z;
                        gpart[8 * M + ((1 * 2 + sel) * 2 + 1) * M + kk] = sacc.w;
                    }
                }
            }
        }
        cluster_barrier();                                   // C: every slice's gradient partials are complete

        // ---- P7: the K partials in rank order, E-term of dh, Adam on the replicated taps ----------------------------------------
        {
            const double bc1 = dsc[0];
            const float bc2s = scal[6];
            for (int i = tid; i < 16 * M; i += CL_NT) {
                float g = cluster.map_shared_rank(gpart, 0)[i];
                for (int r = 1; r < K; ++r) g += cluster.map_shared_rank(gpart, r)[i];
                if (i >= 8 * M) {
                    const int r = i - 8 * M, j = r % M, cn = r / (2 * M), chi = cn >> 1, nu = cn & 1;
                    const float kap = chi ? kap1 : kap0;
                    g = 2.f * kap * g;
                    const float S = scal[2 + nu] - edge[nu * M + j];
                    g = (float)((double)g + 2.0 * (double)kap * (double)hf[r] * (double)S);
                }
                if (last && lead) {
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
    cluster_barrier();                                       // no CTA leaves while a peer may still read its gradient partials

    if (lead) {
        for (int i = tid; i < 8 * M; i += CL_NT) {
            Wg[i] = Wf[i];
            hg[i] = hf[i];
        }
        for (int i = tid; i < 48 * M; i += CL_NT) adg[i] = ad[i];
        if (tid == 0) *reinterpret_cast<int *>(adg + 48 * M) = step0 + n_steps;
    }
}

int dp_cluster_check(int B, int M) {
    int Bs = 0;
    if (cluster_plan(B, M, &Bs)) return VAEQ_OK;
    set_error("batched runs: batch_len %d at M_est %d fits no thread-block cluster of 2, 4 or 8 CTAs with <= %zu KB of shared memory each; "
              "the largest supported batch_len at M_est %d is %d", B, M, CL_SMEM_MAX / 1024, M, dp_cluster_max_b(M));
    return VAEQ_EINVAL;
}

template <int NL, int MT>
static int cluster_launch(const DpK &p, const DpRunsK &rs, int K, int Bs, int n_runs, int n_steps, int stride_sym, int keep_lo_in_dst,
                          float lr_w, float lr_h, int amsgrad, cudaStream_t st) {
    static SmemAttrCache set_smem;
    const size_t smem = (size_t)cluster_layout(Bs, p.M).total * sizeof(float);
    auto kern = k_dp_frame_cluster<NL, MT>;
    if (int rc = ensure_dyn_smem(kern, smem, set_smem)) return rc;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(K, n_runs, 1);
    cfg.blockDim = dim3(CL_NT, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = K;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    int n_clusters = 0;
    VAEQ_CUDA(cudaOccupancyMaxActiveClusters(&n_clusters, kern, &cfg));
    VAEQ_CHECK_ARG(n_clusters > 0, "batched runs: a cluster of %d CTAs with %zu bytes of shared memory each cannot be scheduled on this device", K, smem);
    ktime_begin(VAEQ_K_DP_FRAME, st);
    const cudaError_t e = cudaLaunchKernelEx(&cfg, kern, p, rs, Bs, n_steps, stride_sym, keep_lo_in_dst, lr_w, lr_h, amsgrad);
    ktime_end(VAEQ_K_DP_FRAME, st);
    if (e != cudaSuccess) {
        set_error("launch of k_dp_frame_cluster failed: %s", cudaGetErrorString(e));
        return (int)e;
    }
    return VAEQ_OK;
}

int dp_cluster_launch(const DpK &p, const DpRunsK &rs, int n_lev, int n_runs, int n_steps, int stride_sym, int keep_lo_in_dst,
                      float lr_w, float lr_h, int amsgrad, cudaStream_t st) {
    int Bs = 0;
    const int K = cluster_plan(p.B, p.M, &Bs);
    if (!K) return dp_cluster_check(p.B, p.M);
    const bool m25 = p.M == 25;
#define CL_CASE(NL_) return m25 ? cluster_launch<NL_, 25>(p, rs, K, Bs, n_runs, n_steps, stride_sym, keep_lo_in_dst, lr_w, lr_h, amsgrad, st) \
                            : cluster_launch<NL_, 0>(p, rs, K, Bs, n_runs, n_steps, stride_sym, keep_lo_in_dst, lr_w, lr_h, amsgrad, st);
    if (n_lev == 2) CL_CASE(2)
    if (n_lev == 4) CL_CASE(4)
    CL_CASE(8)
#undef CL_CASE
}

}  // namespace vaeq
