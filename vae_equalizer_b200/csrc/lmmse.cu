// Data-aided LMMSE reference equalizer of the DP sweeps (DESIGN.md §2): per run and frame, the least-squares taps of the 2x2 complex
// butterfly FIR of M_est taps at 2 samples per symbol, fitted on the frame's own transmitted symbols, and the batched FIR that applies
// per-run taps.  No reference counterpart (an extension, like GMI).
//
//   u_n[(i,k)] = x_i[2n + k - mh],  I = [E, N - E), E = ceil(mh/2) + D,  D = n_shift / 2
//   R = sum_I conj(u_n) u_n^T,  r_o(delta) = sum_I conj(u_n) t_o[n - delta],  S_o(delta) = sum_I |t_o[n - delta]|^2
//   w = R^-1 r,  rho = r^H w,  MSE = (S - rho) / |I|,  delta* = argmin MSE,  W = w / beta (beta = rho / S),  var = S (S - rho) / (2 rho |I|)
//
// Two launches per call, one CTA per run each (a run's result does not depend on the other runs of the call):
//   k_lmmse_corr   the correlations the sliding structure needs, summed in double over I.  Along a diagonal of R the entries differ by
//                  the terms entering and leaving I: C_ij(a + 2, d) = C_ij(a, d) + T(N - E) - T(E), so per (pol pair, phase of a) the
//                  2M - 1 lags at the first sample offset of the phase suffice; r slides the same way over (a, delta) -> (a + 2, delta - 1),
//                  M + 4D lags per (pol, tx pol).  Samples and symbols are staged in shared memory as complex doubles (products in
//                  double); a thread owns up to LM_NI correlations and sums its tile's terms in order.  Samples outside the frame are
//                  zero: the first offsets of a phase can reach before the frame, the entries built from them never do.
//   k_lmmse_solve  walks every diagonal (R, packed lower triangle in shared memory) and every (a, delta) chain of r with the edge terms,
//                  S_o(delta) by a block sum and its own sliding, Cholesky R = L L^H, y = L^-1 r for all 2 (2D + 1) right-hand sides,
//                  rho = |y|^2, the delay choice, one back substitution per output pol, and the unbiased taps in the (2,4,M) layout of
//                  twoXtwoFIR.conv_w.weight.  A run whose R is not positive definite in double gets NaN taps / var and ok = 0.
// Every sum runs in a fixed order without atomics: bitwise reproducible, alone or in any batch.
#include "dp_math.cuh"

namespace vaeq {

constexpr int LM_NT = 256;        // threads of both kernels
constexpr int LM_NI = 4;          // correlations per thread of k_lmmse_corr
constexpr int LM_TS = 512;        // symbols per staged tile of k_lmmse_corr
constexpr int LM_SMEM_MAX = 227 * 1024;

struct LmGeom {
    int N, L, M, mh, D, E, nI, nRphi, nE, nitems, n, NR;
};

static inline LmGeom lm_geom(int N, int L, int M, int n_shift) {
    LmGeom g;
    g.N = N;
    g.L = L;
    g.M = M;
    g.mh = M / 2;
    g.D = n_shift / 2;
    g.E = (g.mh + 1) / 2 + g.D;
    g.nI = N - 2 * g.E;
    g.nRphi = 8 * g.mh + 3;                 // per phase: lags of (1,0) [-2mh, 2mh], of (0,0) and (1,1) [-2mh, 0]
    g.nE = 2 * g.D + 1 + g.mh;              // lags e of r per (pol, tx pol, phase): [-D, D + mh]
    g.nitems = 2 * g.nRphi + 8 * g.nE;
    g.n = 2 * M;
    g.NR = 2 * (2 * g.D + 1);
    return g;
}

static inline size_t lm_corr_smem(const LmGeom &g) {
    return sizeof(double2) * (size_t)(2 * (2 * LM_TS + 4 * g.mh) + 2 * (LM_TS + 2 * g.D + g.mh));
}
static inline size_t lm_solve_smem(const LmGeom &g) {
    return sizeof(double2) * ((size_t)g.n * (g.n + 1) / 2 + (size_t)g.NR * g.n) + sizeof(double) * 2 * g.NR + 64;
}

// correlation `it` of a run: rows and offsets of its two factors.  R family: conj(x_i[2n + a0]) x_j[2n + a0 + d];
// r family: conj(x_i[2n + a0]) t_o[n - e].  a0 = -mh + phase.
struct LmItem {
    int i, j, phase, lag, is_t;
};
__host__ __device__ __forceinline__ LmItem lm_item(int it, int mh, int nRphi, int nE, int D) {
    LmItem m;
    if (it < 2 * nRphi) {
        m.phase = it / nRphi;
        const int r = it - m.phase * nRphi;
        m.is_t = 0;
        if (r < 4 * mh + 1) { m.i = 1; m.j = 0; m.lag = r - 2 * mh; }
        else if (r < 6 * mh + 2) { m.i = 0; m.j = 0; m.lag = r - (4 * mh + 1) - 2 * mh; }
        else { m.i = 1; m.j = 1; m.lag = r - (6 * mh + 2) - 2 * mh; }
    } else {
        const int q = it - 2 * nRphi, grp = q / nE;
        m.is_t = 1;
        m.i = grp >> 2;
        m.j = (grp >> 1) & 1;               // tx pol o
        m.phase = grp & 1;
        m.lag = q - grp * nE - D;           // e
    }
    return m;
}

__device__ __forceinline__ void cmac_conj(double2 a, double2 b, double &re, double &im) {   // (re, im) += conj(a) b
    re = fma(a.x, b.x, re);
    re = fma(a.y, b.y, re);
    im = fma(a.x, b.y, im);
    im = fma(-a.y, b.x, im);
}

__global__ void __launch_bounds__(LM_NT) k_lmmse_corr(const float *__restrict__ rx, int64_t ld_rx, int64_t rs_rx, const uint16_t *__restrict__ tx,
                                                      int64_t ld_tx, int64_t rs_tx, LmGeom g, double2 *__restrict__ part) {
    extern __shared__ double2 lm_sm[];
    const int XW = 2 * LM_TS + 4 * g.mh, TW = LM_TS + 2 * g.D + g.mh;
    double2 *xs = lm_sm, *ts = lm_sm + 2 * XW;
    const int run = blockIdx.x, tid = threadIdx.x;
    rx += (int64_t)run * rs_rx;
    tx += (int64_t)run * rs_tx;
    int xo[LM_NI], yo[LM_NI], ys[LM_NI];
    double acc[LM_NI][2];
#pragma unroll
    for (int s = 0; s < LM_NI; ++s) {
        acc[s][0] = acc[s][1] = 0.0;
        const int it = s * LM_NT + tid;
        xo[s] = -1;
        if (it < g.nitems) {
            const LmItem m = lm_item(it, g.mh, g.nRphi, g.nE, g.D);
            const int a0 = -g.mh + m.phase;
            xo[s] = m.i * XW + a0 + 3 * g.mh;                              // x window starts at sample 2 n0 - 3 mh
            if (m.is_t) { yo[s] = 2 * XW + m.j * TW - m.lag + g.D + g.mh; ys[s] = 1; }   // t window starts at symbol n0 - D - mh
            else { yo[s] = m.j * XW + a0 + m.lag + 3 * g.mh; ys[s] = 2; }
        }
    }
    const int nhi = g.N - g.E;
    for (int n0 = g.E; n0 < nhi; n0 += LM_TS) {
        const int tn = min(LM_TS, nhi - n0);
        __syncthreads();
        for (int idx = tid; idx < 2 * XW; idx += LM_NT) {
            const int row = idx / XW, p = idx - row * XW;
            const int64_t s = 2 * (int64_t)n0 - 3 * g.mh + p;
            double2 v = make_double2(0.0, 0.0);
            if (s >= 0 && s < g.L) v = make_double2((double)rx[(int64_t)(2 * row) * ld_rx + s], (double)rx[(int64_t)(2 * row + 1) * ld_rx + s]);
            xs[idx] = v;
        }
        for (int idx = tid; idx < 2 * TW; idx += LM_NT) {
            const int row = idx / TW, p = idx - row * TW;
            const int s = n0 - g.D - g.mh + p;
            double2 v = make_double2(0.0, 0.0);
            if (s >= 0 && s < g.N)
                v = make_double2((double)half_bits_to_float(tx[(int64_t)(2 * row) * ld_tx + s]), (double)half_bits_to_float(tx[(int64_t)(2 * row + 1) * ld_tx + s]));
            ts[idx] = v;
        }
        __syncthreads();
#pragma unroll
        for (int s = 0; s < LM_NI; ++s) {
            if (xo[s] < 0) continue;
            const double2 *px = lm_sm + xo[s], *py = lm_sm + yo[s];
            const int sy = ys[s];
            double re = 0.0, im = 0.0;
#pragma unroll 4
            for (int t = 0; t < tn; ++t) cmac_conj(px[2 * t], py[sy * t], re, im);
            acc[s][0] += re;
            acc[s][1] += im;
        }
    }
#pragma unroll
    for (int s = 0; s < LM_NI; ++s)
        if (xo[s] >= 0) part[(int64_t)run * g.nitems + s * LM_NT + tid] = make_double2(acc[s][0], acc[s][1]);
}

// packed lower triangle, column-major: entry (m, k), m >= k
__device__ __forceinline__ int lm_pk(int m, int k, int n) { return k * n - (k * (k - 1)) / 2 + (m - k); }

__global__ void __launch_bounds__(LM_NT) k_lmmse_solve(const float *__restrict__ rx, int64_t ld_rx, int64_t rs_rx, const uint16_t *__restrict__ tx,
                                                       int64_t ld_tx, int64_t rs_tx, LmGeom g, const double2 *__restrict__ part, float *__restrict__ W,
                                                       float *__restrict__ var_out, int32_t *__restrict__ delay_out, int32_t *__restrict__ ok_out) {
    extern __shared__ double2 lm_sm[];
    const int n = g.n, M = g.M, mh = g.mh, D = g.D, ND = 2 * D + 1, NR = g.NR;
    double2 *A = lm_sm;                                   // packed lower triangle of R, then of L
    double2 *Y = A + n * (n + 1) / 2;                     // [o * ND + delta + D][n]: r, then L^-1 r, then w (chosen delays)
    double *Ssm = reinterpret_cast<double *>(Y + NR * n); // S_o(delta)
    double *rho = Ssm + NR;
    __shared__ double red[32];
    __shared__ int fail;
    __shared__ int dsel[2];
    __shared__ double beta_s[2];
    const int run = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    rx += (int64_t)run * rs_rx;
    tx += (int64_t)run * rs_tx;
    part += (int64_t)run * g.nitems;
    const int hiN = g.N - g.E, loN = g.E;
    auto xg = [&](int i, int s) -> double2 {
        return (s >= 0 && s < g.L) ? make_double2((double)rx[(int64_t)(2 * i) * ld_rx + s], (double)rx[(int64_t)(2 * i + 1) * ld_rx + s])
                                   : make_double2(0.0, 0.0);
    };
    auto tg = [&](int o, int s) -> double2 {
        return (s >= 0 && s < g.N) ? make_double2((double)half_bits_to_float(tx[(int64_t)(2 * o) * ld_tx + s]),
                                                  (double)half_bits_to_float(tx[(int64_t)(2 * o + 1) * ld_tx + s]))
                                   : make_double2(0.0, 0.0);
    };

    // ---- R and r from the correlations, one diagonal / chain per thread --------------------------------------------------------------
    for (int it = tid; it < g.nitems; it += LM_NT) {
        const LmItem m = lm_item(it, mh, g.nRphi, g.nE, D);
        const int a0 = -mh + m.phase;
        double2 C = part[it];
        for (int s = 0;; ++s) {
            const int a = a0 + 2 * s;
            if (a > mh) break;
            if (!m.is_t) {
                const int b = a + m.lag;
                if (b >= -mh && b <= mh) A[lm_pk(m.i * M + a + mh, m.j * M + b + mh, n)] = C;
                if (a + 2 > mh) break;
                double re = C.x, im = C.y;                // C(a + 2) = C(a) + T(N - E) - T(E)
                cmac_conj(xg(m.i, 2 * hiN + a), xg(m.j, 2 * hiN + a + m.lag), re, im);
                double r2 = 0.0, i2 = 0.0;
                cmac_conj(xg(m.i, 2 * loN + a), xg(m.j, 2 * loN + a + m.lag), r2, i2);
                C = make_double2(re - r2, im - i2);
            } else {
                const int dl = m.lag - s;                 // delta of this link of the chain (a0 + 2 s, e - s)
                if (dl >= -D && dl <= D) Y[(m.j * ND + dl + D) * n + m.i * M + a + mh] = C;
                if (a + 2 > mh) break;
                double re = C.x, im = C.y;                // r(a + 2, delta - 1) = r(a, delta) + T'(N - E) - T'(E)
                cmac_conj(xg(m.i, 2 * hiN + a), tg(m.j, hiN - dl), re, im);
                double r2 = 0.0, i2 = 0.0;
                cmac_conj(xg(m.i, 2 * loN + a), tg(m.j, loN - dl), r2, i2);
                C = make_double2(re - r2, im - i2);
            }
        }
    }
    // ---- S_o(0) by a block sum (fixed order), then S_o(delta) by sliding ------------------------------------------------------------
    for (int o = 0; o < 2; ++o) {
        double v = 0.0;
        for (int t = loN + tid; t < hiN; t += LM_NT) {
            const double2 a = tg(o, t);
            v = fma(a.x, a.x, fma(a.y, a.y, v));
        }
        double vv[1] = {v};
        block_sum<1, double>(vv, red);
        if (tid == 0) {
            double S = vv[0];
            Ssm[o * ND + D] = S;
            for (int dl = 0; dl < D; ++dl) {              // S(delta + 1) = S(delta) - |t[N-E-1-delta]|^2 + |t[E-delta-1]|^2
                const double2 p = tg(o, hiN - 1 - dl), q = tg(o, loN - dl - 1);
                S = S - (p.x * p.x + p.y * p.y) + (q.x * q.x + q.y * q.y);
                Ssm[o * ND + D + dl + 1] = S;
            }
            S = vv[0];
            for (int dl = 0; dl > -D; --dl) {             // S(delta - 1) = S(delta) - |t[E-delta]|^2 + |t[N-E-delta]|^2
                const double2 p = tg(o, loN - dl), q = tg(o, hiN - dl);
                S = S - (p.x * p.x + p.y * p.y) + (q.x * q.x + q.y * q.y);
                Ssm[o * ND + D + dl - 1] = S;
            }
        }
        __syncthreads();
    }
    if (tid == 0) fail = 0;
    __syncthreads();

    // ---- Cholesky R = L L^H (right-looking, packed) -----------------------------------------------------------------------------------
    for (int k = 0; k < n; ++k) {
        const int ck = lm_pk(k, k, n);
        if (tid == 0) {
            const double d = A[ck].x;
            if (!(d > 0.0) || !isfinite(d)) fail = 1;
            A[ck] = make_double2(sqrt(d), 0.0);
        }
        __syncthreads();
        if (fail) break;
        const double inv = 1.0 / A[ck].x;
        for (int m = k + 1 + tid; m < n; m += LM_NT) {
            const double2 v = A[ck + m - k];
            A[ck + m - k] = make_double2(v.x * inv, v.y * inv);
        }
        __syncthreads();
        for (int l = k + 1 + wid; l < n; l += LM_NT / 32) {       // A[m][l] -= L[m][k] conj(L[l][k]), m >= l
            const double2 Llk = A[ck + l - k];
            const int cl = lm_pk(l, l, n);
            for (int m = l + lane; m < n; m += 32) {
                const double2 Lmk = A[ck + m - k];
                double2 a = A[cl + m - l];
                a.x -= Lmk.x * Llk.x + Lmk.y * Llk.y;
                a.y -= Lmk.y * Llk.x - Lmk.x * Llk.y;
                A[cl + m - l] = a;
            }
        }
        __syncthreads();
    }
    if (fail) {
        const float nanf_ = __int_as_float(0x7fc00000);
        for (int idx = tid; idx < 8 * M; idx += LM_NT) W[(int64_t)run * 8 * M + idx] = nanf_;
        if (tid < 2) {
            var_out[run * 2 + tid] = nanf_;
            delay_out[run * 2 + tid] = 0;
        }
        if (tid == 0) ok_out[run] = 0;
        return;
    }

    // ---- forward substitution y = L^-1 r for every right-hand side --------------------------------------------------------------------
    for (int k = 0; k < n; ++k) {
        const int ck = lm_pk(k, k, n);
        const double inv = 1.0 / A[ck].x;
        for (int r = tid; r < NR; r += LM_NT) {
            const double2 v = Y[r * n + k];
            Y[r * n + k] = make_double2(v.x * inv, v.y * inv);
        }
        __syncthreads();
        const int rows = n - k - 1;
        for (int idx = tid; idx < NR * rows; idx += LM_NT) {
            const int r = idx / rows, m = k + 1 + (idx - r * rows);
            const double2 L = A[ck + m - k], yk = Y[r * n + k];
            double2 y = Y[r * n + m];
            y.x -= L.x * yk.x - L.y * yk.y;
            y.y -= L.x * yk.y + L.y * yk.x;
            Y[r * n + m] = y;
        }
        __syncthreads();
    }
    for (int r = wid; r < NR; r += LM_NT / 32) {                    // rho = |y|^2, lanes then shuffles in a fixed order
        double v = 0.0;
        for (int k = lane; k < n; k += 32) v = fma(Y[r * n + k].x, Y[r * n + k].x, fma(Y[r * n + k].y, Y[r * n + k].y, v));
        v = warp_sum(v);
        if (lane == 0) rho[r] = v;
    }
    __syncthreads();
    if (tid < 2) {                                                  // delay of least MSE, ties to the smaller |delta|, then the negative one
        const int o = tid;
        int best = 0;
        double bm = 0.0;
        for (int c = 0; c < ND; ++c) {
            const int dl = (c & 1) ? -((c + 1) >> 1) : (c >> 1);
            const int r = o * ND + dl + D;
            const double mse = (Ssm[r] - rho[r]) / (double)g.nI;
            if (c == 0 || mse < bm) { bm = mse; best = dl; }
        }
        const int r = o * ND + best + D;
        const double S = Ssm[r], p = rho[r];
        dsel[o] = r;
        beta_s[o] = p / S;
        var_out[run * 2 + o] = (float)(S * (S - p) / (2.0 * p * (double)g.nI));
        delay_out[run * 2 + o] = best;
    }
    __syncthreads();
    // ---- back substitution L^H w = y for the chosen delay, one warp per output pol ----------------------------------------------------
    if (wid < 2) {
        double2 *y = Y + dsel[wid] * n;
        for (int k = n - 1; k >= 0; --k) {
            const int ck = lm_pk(k, k, n);
            double re = 0.0, im = 0.0;                              // sum_{m > k} conj(L[m][k]) w_m
            for (int m = k + 1 + lane; m < n; m += 32) cmac_conj(A[ck + m - k], y[m], re, im);
            re = warp_sum(re);
            im = warp_sum(im);
            if (lane == 0) {
                const double inv = 1.0 / A[ck].x;
                y[k] = make_double2((y[k].x - re) * inv, (y[k].y - im) * inv);
            }
            __syncwarp();
        }
    }
    __syncthreads();
    for (int idx = tid; idx < 2 * n; idx += LM_NT) {                // W[o][i][k] = Re w / beta, W[o][2 + i][k] = Im w / beta
        const int o = idx / n, p = idx - o * n, i = p / M, k = p - i * M;
        const double2 w = Y[dsel[o] * n + p];
        const double b = beta_s[o];
        float *Wr = W + (int64_t)run * 8 * M + o * 4 * M;
        Wr[i * M + k] = (float)(w.x / b);
        Wr[(2 + i) * M + k] = (float)(w.y / b);
    }
    if (tid == 0) ok_out[run] = 1;
}

// batched 2x2 butterfly FIR with per-run taps: the staged rows of dp_fwd_body, the same fir_butterfly
constexpr int FIR_T = 1024;
__global__ void __launch_bounds__(LM_NT) k_fir_runs(const float *__restrict__ rx, int64_t ld_rx, int64_t rs_rx, int L, const float *__restrict__ W, int M,
                                                    int N, float *__restrict__ out) {
    extern __shared__ float fir_sm[];
    const int mh = M / 2, XN = 2 * FIR_T + 2 * mh;
    float *Ws = fir_sm, *xs = fir_sm + 8 * M;
    const int run = blockIdx.y, t0 = blockIdx.x * FIR_T, tn = min(FIR_T, N - t0), tid = threadIdx.x;
    rx += (int64_t)run * rs_rx;
    for (int i = tid; i < 8 * M; i += LM_NT) Ws[i] = W[(int64_t)run * 8 * M + i];
    const int sb = 2 * t0 - mh;
    for (int j = tid; j < 4 * XN; j += LM_NT) {
        const int r = j / XN, jj = j - r * XN, s = sb + jj;
        xs[j] = (s >= 0 && s < L) ? rx[(int64_t)r * ld_rx + s] : 0.f;
    }
    __syncthreads();
    float *o = out + (int64_t)run * 4 * N;
    for (int i = tid; i < tn; i += LM_NT) {
        float y[4];
        fir_butterfly(xs + 2 * i, XN, Ws, M, y);
#pragma unroll
        for (int c = 0; c < 4; ++c) o[(int64_t)c * N + t0 + i] = y[c];
    }
}

static SmemAttrCache g_lm_corr_attr, g_lm_solve_attr, g_fir_attr;

}  // namespace vaeq

using namespace vaeq;

extern "C" size_t vaeq_lmmse_taps_scratch_bytes(int32_t M, int32_t n_shift, int32_t n_runs) {
    if (M < 1 || n_shift < 1 || n_runs < 1) return 0;
    const LmGeom g = lm_geom(0, 0, M, n_shift);
    return sizeof(double2) * (size_t)g.nitems * (size_t)n_runs;
}

extern "C" int vaeq_lmmse_taps_runs(const float *rx, int64_t ld_rx, int64_t rs_rx, int32_t L, const uint16_t *tx, int64_t ld_tx, int64_t rs_tx,
                                    int32_t N, int32_t M, int32_t n_shift, int32_t n_runs, float *W, float *var, int32_t *delay, int32_t *ok,
                                    void *scratch, size_t scratch_bytes, void *stream) {
    VAEQ_CHECK_ARG(rx && tx && W && var && delay && ok && scratch, "lmmse_taps_runs: NULL pointer");
    VAEQ_CHECK_ARG(M >= 1 && M <= VAEQ_MAX_TAPS && (M & 1), "lmmse_taps_runs: M_est=%d must be odd and <= %d", M, VAEQ_MAX_TAPS);
    VAEQ_CHECK_ARG(n_shift >= 1, "lmmse_taps_runs: n_shift=%d must be >= 1", n_shift);
    VAEQ_CHECK_ARG(n_runs >= 1 && n_runs <= 65535, "lmmse_taps_runs: n_runs=%d must be in [1, 65535]", n_runs);
    VAEQ_CHECK_ARG(N >= 1 && L >= 2 * N, "lmmse_taps_runs: need N >= 1 symbols and L >= 2 N samples, got N=%d, L=%d", N, L);
    VAEQ_CHECK_ARG(ld_rx >= L && ld_tx >= N && (n_runs == 1 || (rs_rx >= 4 * ld_rx && rs_tx >= 2 * ld_tx)),
                   "lmmse_taps_runs: row / run strides too small (ld_rx=%lld rs_rx=%lld ld_tx=%lld rs_tx=%lld)", (long long)ld_rx, (long long)rs_rx,
                   (long long)ld_tx, (long long)rs_tx);
    const LmGeom g = lm_geom(N, L, M, n_shift);
    VAEQ_CHECK_ARG(g.nI >= 2 * M, "lmmse_taps_runs: N=%d leaves %d symbols in the LS range [E, N-E), E=%d; need at least 2 M_est = %d", N, g.nI, g.E,
                   2 * M);
    VAEQ_CHECK_ARG(g.nitems <= LM_NT * LM_NI, "lmmse_taps_runs: n_shift=%d is too large at M_est=%d (%d correlations, at most %d)", n_shift, M,
                   g.nitems, LM_NT * LM_NI);
    const size_t sm_c = lm_corr_smem(g), sm_s = lm_solve_smem(g);
    VAEQ_CHECK_ARG(sm_s <= LM_SMEM_MAX, "lmmse_taps_runs: M_est=%d with n_shift=%d needs %zu bytes of shared memory for the solve, at most %d", M,
                   n_shift, sm_s, LM_SMEM_MAX);
    VAEQ_CHECK_ARG(scratch_bytes >= vaeq_lmmse_taps_scratch_bytes(M, n_shift, n_runs), "lmmse_taps_runs: scratch of %zu bytes, need %zu",
                   scratch_bytes, vaeq_lmmse_taps_scratch_bytes(M, n_shift, n_runs));
    cudaStream_t st = (cudaStream_t)stream;
    int rc = ensure_dyn_smem(k_lmmse_corr, sm_c, g_lm_corr_attr);
    if (rc) return rc;
    rc = ensure_dyn_smem(k_lmmse_solve, sm_s, g_lm_solve_attr);
    if (rc) return rc;
    double2 *part = reinterpret_cast<double2 *>(scratch);
    ktime_begin(VAEQ_K_OTHER, st);
    k_lmmse_corr<<<n_runs, LM_NT, sm_c, st>>>(rx, ld_rx, rs_rx, tx, ld_tx, rs_tx, g, part);
    ktime_end(VAEQ_K_OTHER, st);
    VAEQ_LAUNCH_CHECK("k_lmmse_corr");
    ktime_begin(VAEQ_K_OTHER, st);
    k_lmmse_solve<<<n_runs, LM_NT, sm_s, st>>>(rx, ld_rx, rs_rx, tx, ld_tx, rs_tx, g, part, W, var, delay, ok);
    ktime_end(VAEQ_K_OTHER, st);
    VAEQ_LAUNCH_CHECK("k_lmmse_solve");
    return VAEQ_OK;
}

extern "C" int vaeq_fir_runs(const float *rx, int64_t ld_rx, int64_t rs_rx, int32_t L, const float *W, int32_t M, int32_t N, int32_t n_runs,
                             float *out, void *stream) {
    VAEQ_CHECK_ARG(rx && W && out, "fir_runs: NULL pointer");
    VAEQ_CHECK_ARG(M >= 1 && M <= VAEQ_MAX_TAPS && (M & 1), "fir_runs: M_est=%d must be odd and <= %d", M, VAEQ_MAX_TAPS);
    VAEQ_CHECK_ARG(n_runs >= 1 && n_runs <= 65535 && N >= 1 && L >= 1 && ld_rx >= L && (n_runs == 1 || rs_rx >= 4 * ld_rx),
                   "fir_runs: bad sizes (N=%d L=%d n_runs=%d ld_rx=%lld rs_rx=%lld)", N, L, n_runs, (long long)ld_rx, (long long)rs_rx);
    const size_t sm = sizeof(float) * (size_t)(8 * M + 4 * (2 * FIR_T + 2 * (M / 2)));
    cudaStream_t st = (cudaStream_t)stream;
    int rc = ensure_dyn_smem(k_fir_runs, sm, g_fir_attr);
    if (rc) return rc;
    const dim3 grid((N + FIR_T - 1) / FIR_T, n_runs);
    ktime_begin(VAEQ_K_OTHER, st);
    k_fir_runs<<<grid, LM_NT, sm, st>>>(rx, ld_rx, rs_rx, L, W, M, N, out);
    ktime_end(VAEQ_K_OTHER, st);
    VAEQ_LAUNCH_CHECK("k_fir_runs");
    return VAEQ_OK;
}
