// AWGN single-polarisation VAE-LE step: one persistent CTA runs forward, loss, backward and Adam(amsgrad).
// Reference (AWGN_channel/func_VAELE_MQAM_shaping.py): twoFIR.forward :214-231, loss_function :63-95,
// optimizer = Adam(amsgrad=True) + add_param_group(h_est) :283-286, training loop :297-306.
// Differences from the DP path that matter (SURVEY.md §8a-a9): taps act as w0 - j*w1; the demapper sees the
// output renormalised THROUGH THE GRAPH by mean|out_c| * amp_mean (:228) -> two more global reductions (forward
// mean, backward sum g*out); metric (y-a)^2/var without /2 or PCS term (:229); scalar C.
#include "dp_math.cuh"
#include "dp_kernels.cuh"

namespace vaeq {

constexpr int AW_NT = 1024;

struct AwK {
    int B, L, M, mh, n_lev;
    float amp_mean, var;
    const float *rx, *amp, *P;
    int64_t ld_rx;  // element stride between the I and Q rows of rx
    float *W, *h, *adam;
    float *q, *out, *loss, *gW_out, *gh_out;
    // scratch
    float *m1;    // (2,B)
    float *vs;    // (B)   Var_I + Var_Q
    float *e;     // (L,2) residual D - rx
    float *gyp;   // (2,B) dL/dy' (normalised demapper input)
    float *gout;  // (2,B) dL/dout
    int mode;
    float lr_w, lr_h;
    int amsgrad;
};

__device__ __forceinline__ void adam_apply_awgn(float *param, float g, float *m, float *v, float *vmax, int i, float lr,
                                                bool amsgrad, double bc1, float bc2s) {
    const float b2 = 0.999f, eps = 1e-8f;
    // torch passes 1 - beta as a double and rounds it to float: 0.1f and 0.001f.  1.f - 0.999f would be 1.3e-5 below 0.001f, about
    // 200 ulp in every exp_avg_sq.
    const float w1 = (float)(1.0 - 0.9), w2 = (float)(1.0 - 0.999);
    float mi = m[i], vi = v[i];
    mi = __fmaf_rn(g - mi, w1, mi);                      // exp_avg.lerp_(grad, 1 - beta1), one fused multiply-add as in torch
    vi = vi * b2 + w2 * g * g;                           // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, value=1 - beta2)
    m[i] = mi;
    v[i] = vi;
    const float step_size = (float)(-(double)lr / bc1);    // bias corrections: two double-precision pow, computed ONCE per step by thread 0
    float vv = vi;
    if (amsgrad) {
        vv = fmaxf(vmax[i], vi);
        vmax[i] = vv;
    }
    param[i] = __fadd_rn(param[i], __fmul_rn(step_size, __fdiv_rn(mi, __fadd_rn(__fdiv_rn(sqrtf(vv), bc2s), eps))));
}

// One step of one run by a whole CTA of AW_NT threads (the single-run kernel and the batched-runs kernel share it, so both give
// the same bits).  Ends with a barrier: the caller may start the next step of the same run right away.
template <int NL>
__device__ __forceinline__ void awgn_step_body(const AwK p) {
    __shared__ DemapConst cst;
    __shared__ float Ws[2 * VAEQ_MAX_TAPS], hs[2 * VAEQ_MAX_TAPS], Ssh[VAEQ_MAX_TAPS], PSg[VAEQ_MAX_TAPS + 1];
    __shared__ double red[4 * 32];
    __shared__ float mu[2], kappa_sh;
    __shared__ double gsum[2];
    const int tid = threadIdx.x, B = p.B, L = p.L, M = p.M, mh = p.mh, Mh = 2 * p.mh;

    for (int i = tid; i < 2 * M; i += AW_NT) {
        Ws[i] = p.W[i];
        hs[i] = p.h[i];
    }
    if (tid < VAEQ_MAX_LEVELS) {
        const float a = tid < NL ? p.amp[tid] : 0.f;
        cst.amp[tid] = a;
        cst.a2[tid] = a * a;
        cst.nua2[tid] = 0.f;
        cst.P[tid] = tid < NL ? p.P[tid] : 1.f;
    }
    if (tid < 2) cst.var[tid] = p.var * 0.5f;        // (y-a)^2/2/(var/2) == (y-a)^2/var bit for bit (:229)
    __syncthreads();

    // ---- phase 1: FIR (cross-correlation, zero pad mh, stride 2)  :216-219 ------------------------
    double acc2[2] = {0.0, 0.0};
    for (int t = tid; t < B; t += AW_NT) {
        float oI = 0.f, oQ = 0.f;
        for (int k = 0; k < M; ++k) {
            const int s = 2 * t + k - mh;
            if (s < 0 || s >= L) continue;
            const float xI = p.rx[s], xQ = p.rx[p.ld_rx + s];
            oI += Ws[k] * xI + Ws[M + k] * xQ;
            oQ += Ws[k] * xQ - Ws[M + k] * xI;
        }
        p.out[t] = oI;
        p.out[B + t] = oQ;
        acc2[0] += (double)fabsf(oI);
        acc2[1] += (double)fabsf(oQ);
    }
    block_sum<2>(acc2, red);
    if (tid == 0) {
        mu[0] = (float)(acc2[0] / (double)B);         // torch.mean(torch.abs(out[c,:]))  :228
        mu[1] = (float)(acc2[1] / (double)B);
    }
    __syncthreads();

    // ---- phase 2: normalise, demap, moments, entropy ------------------------------------------------
    double accE[3] = {0.0, 0.0, 0.0};                 // entropy, total Var
    for (int t = tid; t < B; t += AW_NT) {
        float vsum = 0.f;
#pragma unroll
        for (int c = 0; c < 2; ++c) {
            const float yn = __fmul_rn(__fdiv_rn(p.out[c * B + t], mu[c]), p.amp_mean);
            float q[NL], m1, m2;
            demap_component<NL>(yn, cst.var[0], cst, q, m1, m2);
#pragma unroll
            for (int l = 0; l < NL; ++l) p.q[(int64_t)(c * NL + l) * B + t] = q[l];
            p.m1[c * B + t] = m1;
            vsum += m2 - m1 * m1;
            if (t >= mh && t < B - mh) accE[0] += (double)entropy_component<NL>(q, cst);       // :91
        }
        p.vs[t] = vsum;
        accE[1] += (double)vsum;
    }
    block_sum<3>(accE, red);
    __shared__ double ent_sh, vtot_sh;
    if (tid == 0) {
        ent_sh = accE[0];
        vtot_sh = accE[1];
    }
    __syncthreads();
    // S(j) = sum over source symbols u with Mh <= 2u + j < L of Var(u)
    for (int j = tid; j < M; j += AW_NT) {
        double s = vtot_sh;
        const int u_lo = (Mh - j + 1) >> 1, u_hi = (L - 1 - j) >> 1;
        for (int u = 0; u < u_lo && u < B; ++u) s -= (double)p.vs[u];
        for (int u = u_hi + 1; u < B; ++u) s -= (double)p.vs[u];
        Ssh[j] = (float)s;
    }
    __syncthreads();

    // ---- phase 3: D = h * E_q (valid), residual, C ------------------------------------------------------
    double accC[1] = {0.0};
    for (int s = tid; s < L; s += AW_NT) {
        float er = 0.f, ei = 0.f;
        if (s >= mh && s < L - mh) {
            float dr = 0.f, di = 0.f;
            for (int j = (s + mh) & 1; j < M; j += 2) {
                const int v = (s + mh - j) >> 1;
                const float eI = p.m1[v], eQ = p.m1[B + v];
                dr += hs[j] * eI - hs[M + j] * eQ;                                  // :86
                di += hs[j] * eQ + hs[M + j] * eI;                                  // :87
            }
            er = dr - p.rx[s];
            ei = di - p.rx[p.ld_rx + s];
            accC[0] += (double)(er * er + ei * ei);
        }
        p.e[2 * s] = er;
        p.e[2 * s + 1] = ei;
    }
    block_sum<1>(accC, red);
    if (tid == 0) {
        double E = 0.0;
        for (int j = 0; j < M; ++j) E += (double)(hs[j] * hs[j] + hs[M + j] * hs[M + j]) * (double)Ssh[j];   // :88
        const double C = accC[0] + E, width = (double)(L - Mh);
        *p.loss = (float)(width * log(C) - ent_sh);                                 // :94
        kappa_sh = (float)(width / C);
        float a = 0.f;
        PSg[0] = 0.f;
        for (int j = 0; j < M; ++j) {
            a += kappa_sh * (hs[j] * hs[j] + hs[M + j] * hs[M + j]);
            PSg[j + 1] = a;
        }
    }
    __syncthreads();
    if (p.mode == DP_MODE_FWD) return;
    const float kap2 = 2.f * kappa_sh;

    // ---- phase 4: dL/dE_q, demapper backward -> dL/dy', and sum_t dL/dy' * out -------------------------------
    double accG[2] = {0.0, 0.0};
    for (int t = tid; t < B; t += AW_NT) {
        float gr = 0.f, gi = 0.f;
        for (int j = 0; j < M; ++j) {
            const int s = 2 * t - mh + j;
            if (s < 0 || s >= L) continue;
            const float er = kap2 * p.e[2 * s], ei = kap2 * p.e[2 * s + 1];
            gr += hs[j] * er + hs[M + j] * ei;                                      // conj(h) * gD
            gi += hs[j] * ei - hs[M + j] * er;
        }
        const int jlo = max(0, Mh - 2 * t), jhi = min(M, L - 2 * t);
        const float gV = PSg[jhi] - PSg[jlo];
        const bool ent_on = (t >= mh) && (t < B - mh);
        const float gE[2] = {gr, gi};
#pragma unroll
        for (int c = 0; c < 2; ++c) {
            float q[NL];
#pragma unroll
            for (int l = 0; l < NL; ++l) q[l] = p.q[(int64_t)(c * NL + l) * B + t];
            const float o = p.out[c * B + t];
            const float yn = __fmul_rn(__fdiv_rn(o, mu[c]), p.amp_mean);
            const float g1 = gE[c] - 2.f * p.m1[c * B + t] * gV;
            const float g = demap_backward<NL>(yn, cst.var[0], cst, q, g1, gV, ent_on);
            p.gyp[c * B + t] = g;
            accG[c] += (double)g * (double)o;
        }
    }
    block_sum<2>(accG, red);
    if (tid == 0) {
        gsum[0] = accG[0];
        gsum[1] = accG[1];
    }
    __syncthreads();
    // ---- phase 5: back through y' = out / mean|out| * amp_mean ----------------------------------------------
    for (int t = tid; t < B; t += AW_NT) {
#pragma unroll
        for (int c = 0; c < 2; ++c) {
            const float o = p.out[c * B + t];
            const float sc = p.amp_mean / mu[c];
            const float sgn = (o > 0.f) ? 1.f : ((o < 0.f) ? -1.f : 0.f);
            p.gout[c * B + t] = p.gyp[c * B + t] * sc - sgn * (float)(gsum[c] * (double)sc / ((double)mu[c] * (double)B));
        }
    }
    __syncthreads();
    // ---- phase 6: tap gradients (one output per thread), then Adam -----------------------------------------
    __shared__ int step_sh;
    __shared__ double bc1_sh;
    __shared__ float bc2s_sh;
    int *step_ptr = p.adam ? reinterpret_cast<int *>(p.adam + 12 * M) : nullptr;
    if (tid == 0 && p.mode == DP_MODE_TRAIN) {
        step_sh = *step_ptr + 1;
        bc1_sh = 1.0 - pow(0.9, (double)step_sh);            // (every parameter's thread used to evaluate both pow: FP64 at 1/64 rate)
        bc2s_sh = (float)sqrt(1.0 - pow(0.999, (double)step_sh));
    }
    __syncthreads();
    for (int idx = tid; idx < 4 * M; idx += AW_NT) {
        float g = 0.f;
        if (idx < 2 * M) {                               // dW[0][c][k]
            const int c = idx / M, k = idx - c * M;
            for (int t = 0; t < B; ++t) {
                const int s = 2 * t + k - mh;
                if (s < 0 || s >= L) continue;
                const float gI = p.gout[t], gQ = p.gout[B + t], xI = p.rx[s], xQ = p.rx[p.ld_rx + s];
                g += c ? (gI * xQ - gQ * xI) : (gI * xI + gQ * xQ);
            }
            if (p.gW_out) p.gW_out[idx] = g;
            if (p.mode == DP_MODE_TRAIN)
                adam_apply_awgn(p.W, g, p.adam, p.adam + 2 * M, p.adam + 4 * M, idx, p.lr_w, p.amsgrad != 0, bc1_sh, bc2s_sh);
        } else {                                         // dh[c][j]
            const int r = idx - 2 * M, c = r / M, j = r - c * M;
            for (int s = mh; s < L - mh; ++s) {
                if ((s + mh - j) & 1) continue;
                const int v = (s + mh - j) >> 1;
                const float er = kap2 * p.e[2 * s], ei = kap2 * p.e[2 * s + 1], eI = p.m1[v], eQ = p.m1[B + v];
                g += c ? (ei * eI - er * eQ) : (er * eI + ei * eQ);
            }
            g += kap2 * hs[r] * Ssh[j];
            if (p.gh_out) p.gh_out[r] = g;
            if (p.mode == DP_MODE_TRAIN)
                adam_apply_awgn(p.h, g, p.adam + 6 * M, p.adam + 8 * M, p.adam + 10 * M, r, p.lr_h, p.amsgrad != 0, bc1_sh, bc2s_sh);
        }
    }
    __syncthreads();
    if (tid == 0 && p.mode == DP_MODE_TRAIN) *step_ptr = step_sh;
}

template <int NL>
__global__ void __launch_bounds__(AW_NT) k_awgn_step(AwK p) {
    awgn_step_body<NL>(p);
}

static size_t awgn_ws_floats(int B) { return (size_t)2 * B + B + 4 * (size_t)B + 2 * B + 2 * B + 64; }

static int awgn_launch(const vaeq_awgn_desc *d, int mode, float lr_w, float lr_h, cudaStream_t st) {
    VAEQ_CHECK_ARG(d != nullptr, "desc is NULL");
    VAEQ_CHECK_ARG(d->sps == 2, "sps=%d: only sps=2 is implemented", d->sps);
    VAEQ_CHECK_ARG(d->M >= 1 && d->M <= VAEQ_MAX_TAPS && (d->M & 1), "M_est=%d must be odd and <= %d", d->M, VAEQ_MAX_TAPS);
    VAEQ_CHECK_ARG(d->n_lev == 2 || d->n_lev == 4 || d->n_lev == 8, "n_lev=%d must be 2, 4 or 8", d->n_lev);
    VAEQ_CHECK_ARG(d->B > 2 * (d->M / 2), "batch_len=%d must exceed M_est-1", d->B);
    VAEQ_CHECK_ARG(d->rx && d->amp && d->P && d->W && d->h && d->q && d->out && d->loss && d->workspace, "NULL pointer");
    VAEQ_CHECK_ARG(mode != DP_MODE_TRAIN || d->adam, "adam state is NULL");
    if (d->workspace_bytes < vaeq_awgn_workspace_bytes(d->B, d->M, d->n_lev)) {
        set_error("workspace too small");
        return VAEQ_EWORKSPACE;
    }
    AwK p;
    memset(&p, 0, sizeof(p));
    p.B = d->B; p.L = d->B * 2; p.M = d->M; p.mh = d->M / 2; p.n_lev = d->n_lev; p.ld_rx = p.L;
    p.amp_mean = d->amp_mean; p.var = d->var;
    p.rx = d->rx; p.amp = d->amp; p.P = d->P; p.W = d->W; p.h = d->h; p.adam = d->adam;
    p.q = d->q; p.out = d->out; p.loss = d->loss; p.gW_out = d->gW; p.gh_out = d->gh;
    float *ws = static_cast<float *>(d->workspace);
    p.m1 = ws; ws += 2 * (size_t)d->B;
    p.vs = ws; ws += d->B;
    p.e = ws; ws += 4 * (size_t)d->B;
    p.gyp = ws; ws += 2 * (size_t)d->B;
    p.gout = ws;
    p.mode = mode; p.lr_w = lr_w; p.lr_h = lr_h; p.amsgrad = 1;
    ktime_begin(VAEQ_K_AWGN, st);
    switch (d->n_lev) {
        case 2: k_awgn_step<2><<<1, AW_NT, 0, st>>>(p); break;
        case 4: k_awgn_step<4><<<1, AW_NT, 0, st>>>(p); break;
        default: k_awgn_step<8><<<1, AW_NT, 0, st>>>(p); break;
    }
    ktime_end(VAEQ_K_AWGN, st);
    VAEQ_LAUNCH_CHECK("k_awgn_step");
    return VAEQ_OK;
}

// ---- R independent runs, one CTA each (sweep engine): the per-run values come from device arrays ----------------------------
struct AwRunsK {
    AwK base;                                   // run 0's pointers; per-run fields below
    int64_t rs_rx, fs_rx, rs_W, rs_h, rs_adam, rs_P, rs_q, rs_out, rs_loss, rs_ws;
    const float *lr, *var, *amp_mean;           // (R)
    int n_frames, n_mb;                         // frames of n_mb minibatches of B symbols (train), or 1 x 1 (forward)
};

// blockIdx.x = run.  Train: the epoch loop of :291-306 over n_frames frames, minibatch m of frame f at rx + f*fs_rx + m*sps*B;
// loss of step (f, m) at loss[run][f*n_mb + m].  Forward: one step over the whole rx row (validation, :311-313).
template <int NL>
__global__ void __launch_bounds__(AW_NT) k_awgn_runs(AwRunsK r) {
    const int64_t run = blockIdx.x;
    AwK p = r.base;
    p.var = r.var[run];
    p.amp_mean = r.amp_mean[run];
    p.P = r.base.P + run * r.rs_P;
    p.W = r.base.W + run * r.rs_W;
    p.h = r.base.h + run * r.rs_h;
    p.adam = r.base.adam ? r.base.adam + run * r.rs_adam : nullptr;
    p.q = r.base.q + run * r.rs_q;
    p.out = r.base.out + run * r.rs_out;
    const int64_t wo = run * r.rs_ws;
    p.m1 += wo; p.vs += wo; p.e += wo; p.gyp += wo; p.gout += wo;
    if (p.mode == DP_MODE_TRAIN) p.lr_w = p.lr_h = r.lr[run];    // one lr for both parameter groups (:305-306)
    const float *rx = r.base.rx + run * r.rs_rx;
    float *loss = r.base.loss + run * r.rs_loss;
    for (int f = 0; f < r.n_frames; ++f)
        for (int m = 0; m < r.n_mb; ++m) {
            p.rx = rx + f * r.fs_rx + (int64_t)m * p.L;
            p.loss = loss + (int64_t)f * r.n_mb + m;
            awgn_step_body<NL>(p);
        }
}

static int awgn_runs_launch(const vaeq_awgn_desc *d, const vaeq_awgn_runs *rs, int mode, int64_t ld_rx, int64_t fs_rx, int n_frames,
                            int n_mb, cudaStream_t st) {
    VAEQ_CHECK_ARG(d != nullptr && rs != nullptr, "desc is NULL");
    VAEQ_CHECK_ARG(d->sps == 2, "sps=%d: only sps=2 is implemented", d->sps);
    VAEQ_CHECK_ARG(d->M >= 1 && d->M <= VAEQ_MAX_TAPS && (d->M & 1), "M_est=%d must be odd and <= %d", d->M, VAEQ_MAX_TAPS);
    VAEQ_CHECK_ARG(d->n_lev == 2 || d->n_lev == 4 || d->n_lev == 8, "n_lev=%d must be 2, 4 or 8", d->n_lev);
    VAEQ_CHECK_ARG(d->B > 2 * (d->M / 2), "batch_len=%d must exceed M_est-1", d->B);
    VAEQ_CHECK_ARG(rs->n_runs > 0 && n_frames > 0 && n_mb > 0, "bad sizes (n_runs=%d n_frames=%d minibatches=%d)", rs->n_runs, n_frames, n_mb);
    VAEQ_CHECK_ARG(ld_rx >= (int64_t)d->sps * d->B * n_mb, "ld_rx=%lld is shorter than %d minibatches", (long long)ld_rx, n_mb);
    VAEQ_CHECK_ARG(d->rx && d->amp && d->P && d->W && d->h && d->q && d->out && d->loss && d->workspace && rs->var && rs->amp_mean, "NULL pointer");
    VAEQ_CHECK_ARG(mode != DP_MODE_TRAIN || (d->adam && rs->lr), "adam state / lr is NULL");
    const size_t per = awgn_ws_floats(d->B);
    if (d->workspace_bytes < per * sizeof(float) * (size_t)rs->n_runs) {
        set_error("workspace too small");
        return VAEQ_EWORKSPACE;
    }
    AwRunsK r;
    memset(&r, 0, sizeof(r));
    AwK &p = r.base;
    p.B = d->B; p.L = d->B * 2; p.M = d->M; p.mh = d->M / 2; p.n_lev = d->n_lev; p.ld_rx = ld_rx;
    p.rx = d->rx; p.amp = d->amp; p.P = d->P; p.W = d->W; p.h = d->h; p.adam = d->adam;
    p.q = d->q; p.out = d->out; p.loss = d->loss;
    float *ws = static_cast<float *>(d->workspace);
    p.m1 = ws; ws += 2 * (size_t)d->B;
    p.vs = ws; ws += d->B;
    p.e = ws; ws += 4 * (size_t)d->B;
    p.gyp = ws; ws += 2 * (size_t)d->B;
    p.gout = ws;
    p.mode = mode; p.amsgrad = 1;
    r.rs_rx = rs->rs_rx; r.fs_rx = fs_rx; r.rs_W = rs->rs_W; r.rs_h = rs->rs_h; r.rs_adam = rs->rs_adam; r.rs_P = rs->rs_P;
    r.rs_q = rs->rs_q; r.rs_out = rs->rs_out; r.rs_loss = rs->rs_loss; r.rs_ws = (int64_t)per;
    r.lr = rs->lr; r.var = rs->var; r.amp_mean = rs->amp_mean;
    r.n_frames = n_frames; r.n_mb = n_mb;
    ktime_begin(VAEQ_K_AWGN, st);
    switch (d->n_lev) {
        case 2: k_awgn_runs<2><<<rs->n_runs, AW_NT, 0, st>>>(r); break;
        case 4: k_awgn_runs<4><<<rs->n_runs, AW_NT, 0, st>>>(r); break;
        default: k_awgn_runs<8><<<rs->n_runs, AW_NT, 0, st>>>(r); break;
    }
    ktime_end(VAEQ_K_AWGN, st);
    VAEQ_LAUNCH_CHECK("k_awgn_runs");
    return VAEQ_OK;
}

}  // namespace vaeq

using namespace vaeq;

extern "C" size_t vaeq_awgn_runs_workspace_bytes(int32_t B, int32_t M, int32_t n_lev, int32_t n_runs) {
    (void)M; (void)n_lev;
    return (B > 0 && n_runs > 0) ? awgn_ws_floats(B) * sizeof(float) * (size_t)n_runs : 0;
}
extern "C" int vaeq_awgn_train_frames_runs(const vaeq_awgn_desc *d, const vaeq_awgn_runs *r, int64_t ld_rx, int64_t fs_rx, int32_t n_frames,
                                           int32_t n_mb, void *stream) {
    return awgn_runs_launch(d, r, DP_MODE_TRAIN, ld_rx, fs_rx, n_frames, n_mb, (cudaStream_t)stream);
}
extern "C" int vaeq_awgn_forward_runs(const vaeq_awgn_desc *d, const vaeq_awgn_runs *r, int64_t ld_rx, void *stream) {
    return awgn_runs_launch(d, r, DP_MODE_FWD, ld_rx, 0, 1, 1, (cudaStream_t)stream);
}

extern "C" size_t vaeq_awgn_workspace_bytes(int32_t B, int32_t M, int32_t n_lev) {
    (void)M; (void)n_lev;
    return B > 0 ? awgn_ws_floats(B) * sizeof(float) : 0;
}
extern "C" size_t vaeq_adam_state_floats_awgn(int32_t M) { return (size_t)12 * M + 4; }
extern "C" int vaeq_awgn_forward(const vaeq_awgn_desc *d, void *stream) { return awgn_launch(d, DP_MODE_FWD, 0.f, 0.f, (cudaStream_t)stream); }
extern "C" int vaeq_awgn_forward_backward(const vaeq_awgn_desc *d, void *stream) {
    return awgn_launch(d, DP_MODE_FWDBWD, 0.f, 0.f, (cudaStream_t)stream);
}
extern "C" int vaeq_awgn_train_step(const vaeq_awgn_desc *d, float lr_w, float lr_h, void *stream) {
    return awgn_launch(d, DP_MODE_TRAIN, lr_w, lr_h, (cudaStream_t)stream);
}
