// Per-frame evaluation of R independent runs in a handful of launches (sweep engine, vae_equalizer_b200/sweep.py).
//
// What the VAE drivers do once per frame and per run (func_VAELE_DP_MQAM_shaping.py:70-89, func_VAEflex_DP_MQAM_shaping.py:74-84):
//   find_shift(out_train) -> roll pol by r, roll time by -shift per pol -> [VAE-LE: reshape (m_max, B), drop the last
//   shift[0] + N_cut symbols of every minibatch] -> slice [11 : -11 - max|shift|] -> SER_IQflip; the same with
//   find_shift_symb_full(out_const) and SER_constell_shaping.
// Here the roll / cut / slice are INDEX ARITHMETIC inside the scan kernels (nothing is materialised) and the detected shifts
// stay on the device, so a frame of a sweep needs no host synchronisation and 7 launches for all runs instead of ~40 small
// launches and two syncs per run.  The arithmetic per element is that of eval.cu (same decisions, same counts).
#include "common.cuh"
#include "shift_corr.cuh"

namespace vaeq {

constexpr int ER_NT = 256;
constexpr int ER_NORM_EXTRA = 2048;           // bound of blocks-per-run x runs beyond n_runs (norm partials in the scratch)
constexpr int ER_CHUNKS = 8;                     // at most this many CTAs (partial blocks) per run and estimator in the shift search

struct EvalRunsK {
    const float *q; int64_t ld_q, rs_q;          // (R, 2, 2n, N)  out_train
    const float *out; int64_t ld_out, rs_out;    // (R, 2, 2, N)   out_const
    const uint16_t *tx; int64_t ld_tx, rs_tx;    // (R, 2, 2, N)   float16 bit patterns
    const float *amp;                            // (n)
    const float *var; int64_t rs_var;            // (R, 2)
    const float *nu_sc;                          // (R)
    int n_lev, N, n_shift, n_runs;
    int seg_len, edge, n_cut;                    // seg_len = batch_len (VAE-LE minibatch cut) or 0 (VAE-flex); edge = 11; n_cut = 10
    double *part;                                // [R][2][ER_CHUNKS][n_shift][8]
    int *align;                                  // [R][2][4]: shift_0, shift_1, r, n_eval      (estimator 0: from q, 1: from out)
    double *norms;                               // [R][2]: sum |tx|, sum |rx| over the evaluated region (estimator 1)
    int *counts;                                 // [R][2][16]
    float *ser;                                  // [R][4]: constellation x, y, soft demapper x, y  (rows of SER_valid, VAELE_DP:79,89)
    int chunks;                                  // CTAs per (run, estimator) of the shift search: few when there are many runs
    int which;                                   // bit 0: estimator from q, bit 1: estimator from out
    float *scale;                                // optional [R]: the rescale factor mean|tx| / mean|rx| of sf:242 (estimator from out)
};

__device__ __forceinline__ float er_tx_level(uint16_t bits, float scale) {
    return rintf(__fadd_rn(__fmul_rn(scale, half_bits_to_float(bits)), scale));      // sf:198, sf:239
}

// aligned-coordinate position of evaluated element f (0 <= f < n_eval)
__device__ __forceinline__ int er_map(int f, int edge, int seg_len, int keep) {
    f += edge;
    if (seg_len == 0) return f;
    const int m = f / keep;
    return m * seg_len + (f - m * keep);
}
__device__ __forceinline__ int er_wrap(int t, int N) {
    t %= N;
    return t < 0 ? t + N : t;
}

// ---- shift search, both estimators, all runs: grid (ER_CHUNKS, 2 R); a CTA scans its range of t once for all shifts ------------
template <int NPASS>
__global__ void __launch_bounds__(SC_NT, NPASS == 0 ? 4 : SC_MINB) k_er_shift_corr(EvalRunsK p) {
    __shared__ ShiftSmem sm;
    const int chunk = blockIdx.x, run = blockIdx.y >> 1, est = blockIdx.y & 1, N = p.N;
    if (!((p.which >> est) & 1)) return;
    const int per = ((N + p.chunks - 1) / p.chunks + SC_SLICE - 1) / SC_SLICE * SC_SLICE;
    const int64_t t_lo = min((int64_t)N, (int64_t)chunk * per), t_hi = min((int64_t)N, t_lo + per);
    const float *q = p.q + run * p.rs_q, *out = p.out + run * p.rs_out;
    const uint16_t *tx = p.tx + run * p.rs_tx;
    double *dst = p.part + ((((int64_t)run * 2 + est) * p.chunks + chunk) * p.n_shift) * 8;
    if (est == 0) shift_corr_range<true, NPASS>(sm, q, p.ld_q, nullptr, 0, tx, p.ld_tx, p.amp, p.n_lev, N, p.n_shift, t_lo, t_hi, dst);
    else shift_corr_range<false, NPASS>(sm, nullptr, 0, out, p.ld_out, tx, p.ld_tx, nullptr, 0, N, p.n_shift, t_lo, t_hi, dst);
}

// one warp per (run, estimator): lanes sum the chunk partials of consecutive (i, k) (coalesced), lane 0 replays the torch.max / argmax
// logic of sf:303-314 (first index wins ties), then the cut geometry
constexpr int ER_DEC_NT = 128;
__global__ void __launch_bounds__(ER_DEC_NT) k_er_shift_decide(EvalRunsK p) {
    __shared__ float v_s[ER_DEC_NT / 32][8][SC_MAXSHIFT];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int idx = blockIdx.x * (ER_DEC_NT / 32) + w;
    if (idx >= 2 * p.n_runs) return;                         // whole warps leave together; no block-wide barrier below
    const int run = idx >> 1, est = idx & 1, half = p.n_shift / 2, nidx = p.n_shift * 8;
    if (!((p.which >> est) & 1)) return;
    const double *part = p.part + ((int64_t)run * 2 + est) * p.chunks * nidx;
    for (int j = lane; j < nidx; j += 32) {
        double s = 0.0;
        for (int c = 0; c < p.chunks; ++c) s += part[(int64_t)c * nidx + j];
        v_s[w][j & 7][j >> 3] = fabsf((float)s);
    }
    __syncwarp();
    if (lane != 0) return;
    float cmax[8];
    int cind[8];
    for (int k = 0; k < 8; ++k) {
        cmax[k] = -1.f;
        cind[k] = 0;
        for (int i = 0; i < p.n_shift; ++i) {
            const float v = v_s[w][k][i];
            if (v > cmax[k]) {
                cmax[k] = v;
                cind[k] = i;
            }
        }
    }
    float best[4];
    int which[4];
    for (int ba = 0; ba < 4; ++ba) {
        which[ba] = (cmax[4 + ba] > cmax[ba]) ? 1 : 0;
        best[ba] = which[ba] ? cmax[4 + ba] : cmax[ba];
    }
    int sh0, sh1, r;
    if ((best[0] + best[3]) >= (best[1] + best[2])) {
        sh0 = half - cind[which[0] * 4 + 0];
        sh1 = half - cind[which[3] * 4 + 3];
        r = 0;
    } else {
        sh0 = half - cind[which[1] * 4 + 1];
        sh1 = half - cind[which[2] * 4 + 2];
        r = 1;
    }
    const int tail = p.edge + max(abs(sh0), abs(sh1));
    int total = p.N;
    if (p.seg_len) {
        const int keep = min(p.seg_len, p.seg_len - sh0 - p.n_cut);      // VAELE_DP:73-77; torch's [:keep] slice clamps to the minibatch length
        total = keep > 0 ? (p.N / p.seg_len) * keep : 0;
    }
    int *al = p.align + ((int64_t)run * 2 + est) * 4;
    al[0] = sh0; al[1] = sh1; al[2] = r; al[3] = max(0, total - tail - p.edge);
}

// block reduction of 16 integer counters, one atomic per counter (integer: order independent)
__device__ __forceinline__ void er_publish_counts(int (&cnt)[16], int *red, int *dst) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < 16; ++k) {
        int v = cnt[k];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == 0) red[k * 32 + wid] = v;
    }
    __syncthreads();
    if (threadIdx.x < 16) {
        int v = 0;
        for (int w = 0; w < ER_NT / 32; ++w) v += red[threadIdx.x * 32 + w];
        if (v) atomicAdd(&dst[threadIdx.x], v);
    }
}

// hard decision of one symbol of one polarisation and its errors for the 4 rotations, straight and IQ-flipped (sf:188-222):
// q = the pol's first posterior row at the symbol (rows ld_q apart), tx = its I row at the symbol (Q row ld_tx further);
// cnt[(flip * 2 + pol) * 4 + rotation]
template <int NL>
__device__ __forceinline__ void er_count_q(const float *q, int64_t ld_q, const uint16_t *tx, int64_t ld_tx, int pol, int (&cnt)[16]) {
    const float S = (float)(NL - 1), scale = (float)((NL - 1) / 2.0);
    int d[2];
#pragma unroll
    for (int c = 0; c < 2; ++c) {                                         // torch.argmax: first maximal index
        float best = q[(int64_t)(c * NL) * ld_q];
        int bi = 0;
#pragma unroll
        for (int l = 1; l < NL; ++l) {
            const float v = q[(int64_t)(c * NL + l) * ld_q];
            if (v > best) {
                best = v;
                bi = l;
            }
        }
        d[c] = bi;
    }
    const float dI = (float)d[0], dQ = (float)d[1];
    const float hI[4] = {dI, S - dI, S - dQ, dQ};                         // 0, pi, pi/2, 3pi/2  (sf:201-219)
    const float hQ[4] = {dQ, S - dQ, dI, S - dI};
    const float DI = er_tx_level(tx[0], scale);
    const float DQ = er_tx_level(tx[ld_tx], scale);
    const float DQf = S - DQ;                                             // IQ-flipped reference data (sf:199)
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        cnt[(0 * 2 + pol) * 4 + k] += (DI != hI[k]) || (DQ != hQ[k]);
        cnt[(1 * 2 + pol) * 4 + k] += (DI != hI[k]) || (DQf != hQ[k]);
    }
}

// ---- SER from the posteriors (sf:188-222) on the aligned, cut region: grid (blocks, R) ----------------------------------------
template <int NL>
__global__ void __launch_bounds__(ER_NT) k_er_ser_iqflip(EvalRunsK p) {
    __shared__ int red[16 * 32];
    const int run = blockIdx.y, N = p.N;
    const int *al = p.align + ((int64_t)run * 2 + 0) * 4;
    const int sh[2] = {al[0], al[1]}, r = al[2], n_eval = al[3], keep = p.seg_len ? min(p.seg_len, p.seg_len - sh[0] - p.n_cut) : 0;
    const float *q = p.q + run * p.rs_q;
    const uint16_t *tx = p.tx + run * p.rs_tx;
    int cnt[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) cnt[k] = 0;
    for (int f = blockIdx.x * ER_NT + threadIdx.x; f < n_eval; f += gridDim.x * ER_NT) {
        const int t = er_map(f, p.edge, p.seg_len, keep);
#pragma unroll
        for (int pol = 0; pol < 2; ++pol) {
            const int sp = (pol - r) & 1, ts = er_wrap(t + sh[pol], N);   // out.roll(r, 0)[pol].roll(-shift[pol], -1)  (VAELE_DP:71-72)
            er_count_q<NL>(q + (int64_t)(sp * 2 * NL) * p.ld_q + ts, p.ld_q, tx + (int64_t)(pol * 2) * p.ld_tx + t, p.ld_tx, pol, cnt);
        }
    }
    er_publish_counts(cnt, red, p.counts + ((int64_t)run * 2 + 0) * 16);
}

// ---- constellation SER (sf:225-287): norms of the evaluated region, then the threshold test ---------------------------------
__global__ void __launch_bounds__(ER_NT) k_er_constell_norms(EvalRunsK p) {
    __shared__ double red[2 * 32];
    const int run = blockIdx.y, N = p.N;
    const int *al = p.align + ((int64_t)run * 2 + 1) * 4;
    const int sh[2] = {al[0], al[1]}, r = al[2], n_eval = al[3], keep = p.seg_len ? min(p.seg_len, p.seg_len - sh[0] - p.n_cut) : 0;
    const float *out = p.out + run * p.rs_out;
    const uint16_t *tx = p.tx + run * p.rs_tx;
    double acc[2] = {0.0, 0.0};
    for (int f = blockIdx.x * ER_NT + threadIdx.x; f < n_eval; f += gridDim.x * ER_NT) {
        const int t = er_map(f, p.edge, p.seg_len, keep);
#pragma unroll
        for (int pol = 0; pol < 2; ++pol) {
            const int sp = (pol - r) & 1, ts = er_wrap(t + sh[pol], N);
            const float a = half_bits_to_float(tx[(int64_t)(pol * 2) * p.ld_tx + t]), b = half_bits_to_float(tx[(int64_t)(pol * 2 + 1) * p.ld_tx + t]);
            const float x = out[(int64_t)(sp * 2) * p.ld_out + ts], y = out[(int64_t)(sp * 2 + 1) * p.ld_out + ts];
            acc[0] += (double)sqrtf(__fadd_rn(__fmul_rn(a, a), __fmul_rn(b, b)));
            acc[1] += (double)sqrtf(__fadd_rn(__fmul_rn(x, x), __fmul_rn(y, y)));
        }
    }
    block_sum<2>(acc, red);
    if (threadIdx.x == 0) {                                   // per-CTA partials [run][block][2], summed in fixed order by k_er_ser_constell
        double *dst = p.norms + ((int64_t)run * gridDim.x + blockIdx.x) * 2;
        dst[0] = acc[0];
        dst[1] = acc[1];
    }
}

template <int NL>
__global__ void __launch_bounds__(ER_NT) k_er_ser_constell(EvalRunsK p) {
    __shared__ int red[16 * 32];
    __shared__ float lo[NL], hi[NL];
    const int run = blockIdx.y, N = p.N;
    const int *al = p.align + ((int64_t)run * 2 + 1) * 4;
    const int sh[2] = {al[0], al[1]}, r = al[2], n_eval = al[3], keep = p.seg_len ? min(p.seg_len, p.seg_len - sh[0] - p.n_cut) : 0;
    const float *out = p.out + run * p.rs_out;
    const uint16_t *tx = p.tx + run * p.rs_tx;
    if (threadIdx.x < NL) {
        const int l = threadIdx.x;
        const float f = __fadd_rn(1.f, __fmul_rn(2.f * p.nu_sc[run], p.var[run * p.rs_var]));      // sf:234-236
        lo[l] = (l == 0) ? -INFINITY : __fmul_rn(f, __fadd_rn(p.amp[l - 1], p.amp[l])) * 0.5f;
        hi[l] = (l == NL - 1) ? INFINITY : __fmul_rn(f, __fadd_rn(p.amp[l], p.amp[l + 1])) * 0.5f;
    }
    __syncthreads();
    const double cnt2 = 2.0 * (double)n_eval;
    __shared__ double bc[2];
    double sum_tx = 0.0, sum_rx = 0.0;
    if (threadIdx.x < 32) {                                   // fixed-order sum of the norm partials (no floating-point atomics)
        const double *part = p.norms + (int64_t)run * gridDim.x * 2;
        for (int i = threadIdx.x; i < (int)gridDim.x; i += 32) {
            sum_tx += part[2 * i];
            sum_rx += part[2 * i + 1];
        }
        sum_tx = warp_sum(sum_tx);
        sum_rx = warp_sum(sum_rx);
        if (threadIdx.x == 0) {
            bc[0] = sum_tx;
            bc[1] = sum_rx;
        }
    }
    __syncthreads();
    const float g = __fdiv_rn((float)(bc[0] / cnt2), (float)(bc[1] / cnt2));      // sf:242
    if (p.scale != nullptr && blockIdx.x == 0 && threadIdx.x == 0) p.scale[run] = g;
    const float S = (float)(NL - 1), scale = (float)((NL - 1) / 2.0);
    int cnt[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) cnt[k] = 0;
    for (int f = blockIdx.x * ER_NT + threadIdx.x; f < n_eval; f += gridDim.x * ER_NT) {
        const int t = er_map(f, p.edge, p.seg_len, keep);
#pragma unroll
        for (int pol = 0; pol < 2; ++pol) {
            const int sp = (pol - r) & 1, ts = er_wrap(t + sh[pol], N);
            const float yI = __fmul_rn(out[(int64_t)(sp * 2) * p.ld_out + ts], g), yQ = __fmul_rn(out[(int64_t)(sp * 2 + 1) * p.ld_out + ts], g);
            const float DI = er_tx_level(tx[(int64_t)(pol * 2) * p.ld_tx + t], scale), DQ = er_tx_level(tx[(int64_t)(pol * 2 + 1) * p.ld_tx + t], scale);
            const float DQf = S - DQ;
            const int iI = min(max((int)DI, 0), NL - 1), iQ = min(max((int)DQ, 0), NL - 1), iQf = min(max((int)DQf, 0), NL - 1);
            const float hI[4] = {yI, -yI, -yQ, yQ};                       // sf:245-262
            const float hQ[4] = {yQ, -yQ, yI, -yI};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const bool okI = (lo[iI] <= hI[k]) && (hI[k] < hi[iI]);
                const bool okQ = (lo[iQ] <= hQ[k]) && (hQ[k] < hi[iQ]);
                const bool okQf = (lo[iQf] <= hQ[k]) && (hQ[k] < hi[iQf]);
                cnt[(0 * 2 + pol) * 4 + k] += !(okI && okQ);
                cnt[(1 * 2 + pol) * 4 + k] += !(okI && okQf);
            }
        }
    }
    er_publish_counts(cnt, red, p.counts + ((int64_t)run * 2 + 1) * 16);
}

// torch.amin over (flip, rotation) per pol (sf:221, sf:264): thread = (run, estimator, pol)
__global__ void k_er_ser_min(EvalRunsK p) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= 4 * p.n_runs) return;
    const int run = idx >> 2, est = (idx >> 1) & 1, pol = idx & 1;
    if (!((p.which >> est) & 1)) return;
    const int n_eval = p.align[((int64_t)run * 2 + est) * 4 + 3];
    const int *counts = p.counts + ((int64_t)run * 2 + est) * 16;
    float best = 3.0e38f;
    for (int f = 0; f < 2; ++f)
        for (int k = 0; k < 4; ++k) best = fminf(best, __fdiv_rn((float)counts[(f * 2 + pol) * 4 + k], (float)n_eval));
    p.ser[run * 4 + (est == 0 ? 2 : 0) + pol] = n_eval > 0 ? best : __int_as_float(0x7fc00000);
}

// ---- CMA drivers (CMA_DP:42-48): the aligned copy of the CPE output with the evaluated slice rescaled, all runs -------------------
// oc[run][pol][c][t] = out[run][(pol - r) & 1][c][(t + shift[pol]) mod N] * (edge <= t < N - edge - max|shift| ? g_run : 1):
// out.roll(r, 0), per-pol roll by -shift, and the in-place rescale SER_constell_shaping leaves in the slice it was given (sf:242),
// which soft_dec then sees (CMA_DP:44,48).  align = the estimator-from-out rows of vaeq_frame_eval_runs, g = its scale_out.
__global__ void __launch_bounds__(ER_NT) k_er_align_rescale(const float *out, int64_t ld_out, int64_t rs_out, const int *align, const float *scale,
                                                            int N, int edge, float *oc) {
    const int run = blockIdx.y;
    const int *al = align + ((int64_t)run * 2 + 1) * 4;
    const int sh[2] = {al[0], al[1]}, r = al[2], hi = N - edge - max(abs(al[0]), abs(al[1]));
    const float g = scale[run];
    const float *src = out + run * rs_out;
    float *dst = oc + (int64_t)run * 4 * N;
    for (int t = blockIdx.x * ER_NT + threadIdx.x; t < N; t += gridDim.x * ER_NT) {
        const bool in = t >= edge && t < hi;
#pragma unroll
        for (int pol = 0; pol < 2; ++pol) {
            const int sp = (pol - r) & 1, ts = er_wrap(t + sh[pol], N);
#pragma unroll
            for (int c = 0; c < 2; ++c) {
                const float v = src[(int64_t)(sp * 2 + c) * ld_out + ts];
                dst[(int64_t)(pol * 2 + c) * N + t] = in ? __fmul_rn(v, g) : v;
            }
        }
    }
}

// ---- AWGN single-polarisation driver (processing.py awgn_find_shift + awgn_ser_q, AWGN :188-204, :97-124), R runs ----------------
struct AwgnEvalK {
    const float *q; int64_t ld_q, rs_q;          // (R, 2n, N)
    const uint16_t *tx; int64_t ld_tx, rs_tx;    // (R, 2, N) float16 bits
    const float *amp;
    int n_lev, N, n_shift, n_corr, edge, n_runs, chunks;
    double *part;                                // [R][chunks][n_shift][8]
    int *shift;                                  // [R]
    int *cnt;                                    // [R][16] scratch counters
    int *counts;                                 // [R][4]
    float *ser;                                  // [R]
};

// grid (chunks, R): the correlation of the first n_corr symbols, one SC_T tile per CTA like vaeq_find_shift cuts it, so the partial
// sums and their fixed-order total are those of the single-run search.  q's I rows against itself as both "polarisations"
__global__ void __launch_bounds__(SC_NT, 4) k_aw_shift_corr(AwgnEvalK p) {
    __shared__ ShiftSmem sm;
    const int64_t run = blockIdx.y, t_lo = (int64_t)blockIdx.x * SC_T, t_hi = min((int64_t)p.n_corr, t_lo + SC_T);
    shift_corr_range<true, 0, true>(sm, p.q + run * p.rs_q, p.ld_q, nullptr, 0, p.tx + run * p.rs_tx, p.ld_tx, p.amp, p.n_lev, p.n_corr, p.n_shift,
                                    t_lo, t_hi, p.part + (run * p.chunks + blockIdx.x) * p.n_shift * 8);
}

// thread = run: |corr| with tx I (k = 0) and tx Q (k = 4), summed over the chunks in order as k_shift_decide does, then the rule of
// awgn_find_shift in fp32 like the torch expressions (first index wins ties; 0.02 * N is a Python float compared with a float32 tensor)
__global__ void k_aw_shift_decide(AwgnEvalK p) {
    const int run = blockIdx.x * blockDim.x + threadIdx.x;
    if (run >= p.n_runs) return;
    const int nidx = p.n_shift * 8, half = p.n_shift / 2;
    const double *part = p.part + (int64_t)run * p.chunks * nidx;
    float mI = -1.f, mQ = -1.f;
    int iI = 0, iQ = 0;
    for (int i = 0; i < p.n_shift; ++i) {
        double sI = 0.0, sQ = 0.0;
        for (int c = 0; c < p.chunks; ++c) {
            sI += part[(int64_t)c * nidx + i * 8 + 0];
            sQ += part[(int64_t)c * nidx + i * 8 + 4];
        }
        const float vI = fabsf((float)sI), vQ = fabsf((float)sQ);
        if (vI > mI) { mI = vI; iI = i; }
        if (vQ > mQ) { mQ = vQ; iQ = i; }
    }
    const float thr = (float)(0.02 * (double)p.N);
    const int idx = (mI >= thr) ? iI : ((mQ >= mI) ? iQ : iI);
    p.shift[run] = half - idx;
}

// grid (blocks, R): error counts of q[:, edge + shift : N - edge] against tx[:, edge : N - edge - shift]
template <int NL>
__global__ void __launch_bounds__(ER_NT) k_aw_ser(AwgnEvalK p) {
    __shared__ int red[16 * 32];
    const int64_t run = blockIdx.y;
    const int sh = p.shift[run], n_eval = p.N - 2 * p.edge - sh;
    const float *q = p.q + run * p.rs_q + p.edge + sh;
    const uint16_t *tx = p.tx + run * p.rs_tx + p.edge;
    int cnt[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) cnt[k] = 0;
    for (int f = blockIdx.x * ER_NT + threadIdx.x; f < n_eval; f += gridDim.x * ER_NT) er_count_q<NL>(q + f, p.ld_q, tx + f, p.ld_tx, 0, cnt);
    er_publish_counts(cnt, red, p.cnt + run * 16);
}

// thread = run: the 4 rotation counts (no IQ flip) and min count / symbols in fp32 as torch divides a float32 tensor by a Python int on
// the GPU: times the fp32 reciprocal of the divisor (awgn_ser_q)
__global__ void k_aw_ser_min(AwgnEvalK p) {
    const int run = blockIdx.x * blockDim.x + threadIdx.x;
    if (run >= p.n_runs) return;
    const int n_eval = p.N - 2 * p.edge - p.shift[run];
    int m = INT_MAX;
    for (int k = 0; k < 4; ++k) {
        const int c = p.cnt[run * 16 + k];
        p.counts[run * 4 + k] = c;
        m = min(m, c);
    }
    p.ser[run] = __fmul_rn((float)m, __fdiv_rn(1.f, (float)n_eval));
}

// ---- GMI of the SER's region under the SER's hypothesis (extension, not in the reference) -----------------------------------------
// GMI = H(X) + mean over the evaluated symbols of log2 q(x_tx | y) per polarisation, bit per 2-D symbol, on exactly the symbols the
// soft-demapper SER counts and with the (IQ flip, rotation) whose error count is smallest, so it is invariant under the symmetries the
// SER forgives.  Symbols are split into fixed chunks of GMI_CHUNK: the partial sums of a run depend on its own n_eval only, never on
// the number of runs of the call, so a run's GMI is bit-identical alone or in any batch.
constexpr int GMI_CHUNK = 2048;

struct GmiRunsK {
    const float *q; int64_t ld_q, rs_q;          // DP (R,2,2n,N), AWGN (R,2n,N)
    const uint16_t *tx; int64_t ld_tx, rs_tx;    // DP (R,2,2,N), AWGN (R,2,N) float16 bits
    const float *P; int64_t rs_P;                // (R,n) pmf of each run
    const int *align;                            // DP: (R,2,4) of vaeq_frame_eval_runs_ex (estimator 0 row); AWGN: shift (R)
    const int *counts;                           // DP: (R,2,2,2,4) [est][flip][pol][rotation]; AWGN: (R,4) [rotation]
    int N, seg_len, edge, n_cut, n_runs, max_chunks;
    double *part;                                // [R][max_chunks][2]
    float *gmi;                                  // DP (R,2), AWGN (R)
};

// the hypothesis h = flip * 4 + rotation with the smallest error count, in counter order (flip 0 rotations 0..3, then flip 1);
// the first wins ties.  cnt = the pol's rotation 0 counter, the flip-1 counters flip_stride further
__device__ __forceinline__ int gmi_hypothesis(const int *cnt, int n_flip, int flip_stride) {
    int best = cnt[0], h = 0;
    for (int f = 0; f < n_flip; ++f)
        for (int k = 0; k < 4; ++k) {
            const int c = cnt[f * flip_stride + k];
            if (c < best) {
                best = c;
                h = f * 4 + k;
            }
        }
    return h;
}

// evaluated-region geometry of one run: shifts, polarisation swap and symbol count (DP: estimator 0 of the frame evaluation;
// AWGN: q[:, edge + shift : N - edge] against tx[:, edge : N - edge - shift], as k_aw_ser)
template <int NPOL>
__device__ __forceinline__ void gmi_geometry(const GmiRunsK &p, int run, int (&sh)[2], int &r, int &n_eval, int &keep) {
    if (NPOL == 2) {
        const int *al = p.align + (int64_t)run * 8;
        sh[0] = al[0]; sh[1] = al[1]; r = al[2]; n_eval = al[3];
        keep = p.seg_len ? min(p.seg_len, p.seg_len - sh[0] - p.n_cut) : 0;
    } else {
        sh[0] = sh[1] = p.align[run];
        r = 0; keep = 0;
        // q starts at edge + shift: a shift below -edge (impossible for shifts of awgn_eval_runs with edge >= n_shift / 2) scores
        // nothing rather than reading before the row.  Otherwise n_eval <= N - edge, inside the chunks the grid covers.
        n_eval = p.edge + sh[0] < 0 ? 0 : p.N - 2 * p.edge - sh[0];
    }
}

// grid (max_chunks, R): CTA c sums log2 q of the chosen hypothesis over evaluated symbols [c GMI_CHUNK, (c + 1) GMI_CHUNK) per pol.
// NPOL = 2: the DP drivers (pol swap, circular shift, minibatch cut); NPOL = 1: the AWGN driver (one pol, no flip, no wrap)
template <int NL, int NPOL>
__global__ void __launch_bounds__(ER_NT) k_gmi_runs(GmiRunsK p) {
    __shared__ double red[2 * 32];
    const int run = blockIdx.y, N = p.N;
    int sh[2], r, n_eval, keep;
    gmi_geometry<NPOL>(p, run, sh, r, n_eval, keep);
    const int f0 = blockIdx.x * GMI_CHUNK, f1 = min(n_eval, f0 + GMI_CHUNK);
    if (f0 >= f1) return;                                    // beyond this run's symbols: the finish reads no partial of this CTA
    int hyp[2];
#pragma unroll
    for (int pol = 0; pol < NPOL; ++pol)
        hyp[pol] = NPOL == 2 ? gmi_hypothesis(p.counts + (int64_t)run * 32 + pol * 4, 2, 8) : gmi_hypothesis(p.counts + (int64_t)run * 4, 1, 0);
    const float *q = p.q + run * p.rs_q;
    const uint16_t *tx = p.tx + run * p.rs_tx;
    const float scale = (float)((NL - 1) / 2.0);
    constexpr int S = NL - 1;
    double acc[2] = {0.0, 0.0};
    for (int f = f0 + threadIdx.x; f < f1; f += ER_NT) {
        const int t = er_map(f, p.edge, p.seg_len, keep);
#pragma unroll
        for (int pol = 0; pol < NPOL; ++pol) {
            const int sp = (pol - r) & 1, ts = NPOL == 2 ? er_wrap(t + sh[pol], N) : t + sh[0];
            const int DI = min(max((int)er_tx_level(tx[(int64_t)(pol * 2) * p.ld_tx + t], scale), 0), S);
            const int DQ = min(max((int)er_tx_level(tx[(int64_t)(pol * 2 + 1) * p.ld_tx + t], scale), 0), S);
            const int k = hyp[pol] & 3, DQp = (hyp[pol] >> 2) ? S - DQ : DQ;     // IQ-flipped reference data (sf:199)
            // inverse of er_count_q's hI / hQ: the q levels that rotation k maps onto the tx levels
            const int iI = k == 0 ? DI : k == 1 ? S - DI : k == 2 ? DQp : S - DQp;
            const int iQ = k == 0 ? DQp : k == 1 ? S - DQp : k == 2 ? S - DI : DI;
            const float *qp = q + (int64_t)(sp * 2 * NL) * p.ld_q + ts;
            const float qI = qp[(int64_t)iI * p.ld_q], qQ = qp[(int64_t)(NL + iQ) * p.ld_q];
            acc[pol] += log2((double)fmaxf(qI, 1e-30f)) + log2((double)fmaxf(qQ, 1e-30f));
        }
    }
    block_sum<2>(acc, red);
    if (threadIdx.x == 0) {
        double *dst = p.part + ((int64_t)run * p.max_chunks + blockIdx.x) * 2;
        dst[0] = acc[0];
        dst[1] = acc[1];
    }
}

// thread = (run, pol): the run's chunk partials in chunk order, plus H(X) = -2 sum_l P_l log2 P_l of the run's pmf (as k_gmi_fin)
template <int NPOL>
__global__ void k_gmi_runs_fin(GmiRunsK p, int n_lev) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= NPOL * p.n_runs) return;
    const int run = idx / NPOL, pol = idx % NPOL;
    int sh[2], r, n_eval, keep;
    gmi_geometry<NPOL>(p, run, sh, r, n_eval, keep);
    const int nch = min(p.max_chunks, (max(n_eval, 0) + GMI_CHUNK - 1) / GMI_CHUNK);
    const double *part = p.part + (int64_t)run * p.max_chunks * 2 + pol;
    double s = 0.0;
    for (int c = 0; c < nch; ++c) s += part[2 * c];
    const float *P = p.P + run * p.rs_P;
    double H = 0.0;
    for (int l = 0; l < n_lev; ++l) H -= 2.0 * (double)P[l] * log2((double)P[l]);
    p.gmi[idx] = n_eval > 0 ? (float)(H + s / (double)n_eval) : __int_as_float(0x7fc00000);
}

static int gmi_runs_launch(GmiRunsK &p, int n_lev, int npol, cudaStream_t st) {
    const dim3 grid(p.max_chunks, p.n_runs);
    ktime_begin(VAEQ_K_EVAL, st);
#define GMI_CASE(NL_)                                                                                  \
    if (npol == 2) k_gmi_runs<NL_, 2><<<grid, ER_NT, 0, st>>>(p);                                      \
    else k_gmi_runs<NL_, 1><<<grid, ER_NT, 0, st>>>(p);
    if (n_lev == 2) { GMI_CASE(2) } else if (n_lev == 4) { GMI_CASE(4) } else { GMI_CASE(8) }
#undef GMI_CASE
    ktime_end(VAEQ_K_EVAL, st);
    VAEQ_LAUNCH_CHECK("k_gmi_runs");
    const int n = npol * p.n_runs;
    ktime_begin(VAEQ_K_EVAL, st);
    if (npol == 2) k_gmi_runs_fin<2><<<(n + 127) / 128, 128, 0, st>>>(p, n_lev);
    else k_gmi_runs_fin<1><<<(n + 127) / 128, 128, 0, st>>>(p, n_lev);
    ktime_end(VAEQ_K_EVAL, st);
    VAEQ_LAUNCH_CHECK("k_gmi_runs_fin");
    return VAEQ_OK;
}

static int gmi_max_chunks(int N) { return (N + GMI_CHUNK - 1) / GMI_CHUNK; }

}  // namespace vaeq

using namespace vaeq;

extern "C" size_t vaeq_frame_gmi_scratch_bytes(int32_t n_runs, int32_t N) {
    if (n_runs <= 0 || N <= 0) return 0;
    return (size_t)n_runs * gmi_max_chunks(N) * 2 * sizeof(double);
}

extern "C" size_t vaeq_awgn_gmi_scratch_bytes(int32_t n_runs, int32_t N) { return vaeq_frame_gmi_scratch_bytes(n_runs, N); }

extern "C" int vaeq_frame_gmi_runs(const float *q, int64_t ld_q, int64_t rs_q, const uint16_t *tx, int64_t ld_tx, int64_t rs_tx, const float *P,
                                   int64_t rs_P, const int32_t *align, const int32_t *counts, int32_t n_lev, int32_t N, int32_t n_runs,
                                   int32_t seg_len, int32_t edge, int32_t n_cut, float *gmi_out, void *scratch, void *stream) {
    VAEQ_CHECK_ARG(q && tx && P && align && counts && gmi_out && scratch, "NULL pointer");
    VAEQ_CHECK_ARG(n_lev == 2 || n_lev == 4 || n_lev == 8, "n_lev=%d must be 2, 4 or 8", n_lev);
    VAEQ_CHECK_ARG(N > 0 && edge >= 0 && n_cut >= 0, "bad sizes (N=%d, edge=%d, n_cut=%d)", N, edge, n_cut);
    VAEQ_CHECK_ARG(seg_len == 0 || (seg_len > 0 && N % seg_len == 0), "N=%d must be a multiple of seg_len=%d", N, seg_len);
    VAEQ_CHECK_ARG(n_runs > 0 && n_runs <= 65535, "n_runs=%d must be in 1..65535", n_runs);
    GmiRunsK p;
    p.q = q; p.ld_q = ld_q; p.rs_q = rs_q; p.tx = tx; p.ld_tx = ld_tx; p.rs_tx = rs_tx; p.P = P; p.rs_P = rs_P;
    p.align = align; p.counts = counts; p.N = N; p.seg_len = seg_len; p.edge = edge; p.n_cut = n_cut; p.n_runs = n_runs;
    p.max_chunks = gmi_max_chunks(N); p.part = static_cast<double *>(scratch); p.gmi = gmi_out;
    return gmi_runs_launch(p, n_lev, 2, (cudaStream_t)stream);
}

extern "C" int vaeq_awgn_gmi_runs(const float *q, int64_t ld_q, int64_t rs_q, const uint16_t *tx, int64_t ld_tx, int64_t rs_tx, const float *P,
                                  int64_t rs_P, const int32_t *shift, const int32_t *counts, int32_t n_lev, int32_t N, int32_t n_runs, int32_t edge,
                                  float *gmi_out, void *scratch, void *stream) {
    VAEQ_CHECK_ARG(q && tx && P && shift && counts && gmi_out && scratch, "NULL pointer");
    VAEQ_CHECK_ARG(n_lev == 2 || n_lev == 4 || n_lev == 8, "n_lev=%d must be 2, 4 or 8", n_lev);
    VAEQ_CHECK_ARG(N > 0 && edge >= 0 && N - 2 * edge > 0, "N=%d leaves no symbol to evaluate with edge=%d", N, edge);
    VAEQ_CHECK_ARG(n_runs > 0 && n_runs <= 65535, "n_runs=%d must be in 1..65535", n_runs);
    GmiRunsK p;
    p.q = q; p.ld_q = ld_q; p.rs_q = rs_q; p.tx = tx; p.ld_tx = ld_tx; p.rs_tx = rs_tx; p.P = P; p.rs_P = rs_P;
    p.align = shift; p.counts = counts; p.N = N; p.seg_len = 0; p.edge = edge; p.n_cut = 0; p.n_runs = n_runs;
    p.max_chunks = gmi_max_chunks(N); p.part = static_cast<double *>(scratch); p.gmi = gmi_out;
    return gmi_runs_launch(p, n_lev, 1, (cudaStream_t)stream);
}

extern "C" size_t vaeq_awgn_eval_scratch_bytes(int32_t n_runs, int32_t n_shift, int32_t n_corr) {
    if (n_runs <= 0 || n_shift <= 0 || n_corr <= 0) return 0;
    const size_t chunks = ((size_t)n_corr + SC_T - 1) / SC_T;
    return align_up((size_t)n_runs * chunks * n_shift * 8 * sizeof(double), 256) + (size_t)n_runs * 16 * sizeof(int);
}

extern "C" int vaeq_awgn_eval_runs(const float *q, int64_t ld_q, int64_t rs_q, const uint16_t *tx, int64_t ld_tx, int64_t rs_tx, const float *amp,
                                   int32_t n_lev, int32_t N, int32_t n_shift, int32_t n_corr, int32_t edge, int32_t n_runs, int32_t *shift_out,
                                   int32_t *counts_out, float *ser_out, void *scratch, void *stream) {
    VAEQ_CHECK_ARG(q && tx && amp && shift_out && counts_out && ser_out && scratch, "NULL pointer");
    VAEQ_CHECK_ARG(n_lev == 2 || n_lev == 4 || n_lev == 8, "n_lev=%d must be 2, 4 or 8", n_lev);
    VAEQ_CHECK_ARG(n_shift > 0 && n_shift <= 8 * SC_J && edge >= 0 && n_corr > 0 && n_corr <= N, "bad sizes (n_shift=%d <= %d, n_corr=%d <= N=%d)",
                   n_shift, 8 * SC_J, n_corr, N);
    VAEQ_CHECK_ARG(N - 2 * edge - n_shift / 2 > 0, "N=%d leaves no symbol to evaluate", N);
    VAEQ_CHECK_ARG(n_runs > 0 && n_runs <= 65535, "n_runs=%d must be in 1..65535", n_runs);
    cudaStream_t st = (cudaStream_t)stream;
    AwgnEvalK p;
    p.q = q; p.ld_q = ld_q; p.rs_q = rs_q; p.tx = tx; p.ld_tx = ld_tx; p.rs_tx = rs_tx; p.amp = amp;
    p.n_lev = n_lev; p.N = N; p.n_shift = n_shift; p.n_corr = n_corr; p.edge = edge; p.n_runs = n_runs;
    p.chunks = (n_corr + SC_T - 1) / SC_T;
    const size_t part_b = align_up((size_t)n_runs * p.chunks * n_shift * 8 * sizeof(double), 256);
    p.part = static_cast<double *>(scratch);
    p.cnt = reinterpret_cast<int *>(static_cast<char *>(scratch) + part_b);
    p.shift = shift_out; p.counts = counts_out; p.ser = ser_out;
    VAEQ_CUDA(cudaMemsetAsync(p.cnt, 0, (size_t)n_runs * 16 * sizeof(int), st));
    const int blocks = max(1, min((N + ER_NT - 1) / ER_NT, max(1, sm_count() * 8 / n_runs)));
#define AW_LAUNCH(name, ...)                    \
    ktime_begin(VAEQ_K_EVAL, st);               \
    __VA_ARGS__;                                \
    ktime_end(VAEQ_K_EVAL, st);                 \
    VAEQ_LAUNCH_CHECK(name);
    AW_LAUNCH("k_aw_shift_corr", k_aw_shift_corr<<<dim3(p.chunks, n_runs), SC_NT, 0, st>>>(p))
    AW_LAUNCH("k_aw_shift_decide", k_aw_shift_decide<<<(n_runs + 127) / 128, 128, 0, st>>>(p))
    if (n_lev == 2) { AW_LAUNCH("k_aw_ser", k_aw_ser<2><<<dim3(blocks, n_runs), ER_NT, 0, st>>>(p)) }
    else if (n_lev == 4) { AW_LAUNCH("k_aw_ser", k_aw_ser<4><<<dim3(blocks, n_runs), ER_NT, 0, st>>>(p)) }
    else { AW_LAUNCH("k_aw_ser", k_aw_ser<8><<<dim3(blocks, n_runs), ER_NT, 0, st>>>(p)) }
    AW_LAUNCH("k_aw_ser_min", k_aw_ser_min<<<(n_runs + 127) / 128, 128, 0, st>>>(p))
#undef AW_LAUNCH
    return VAEQ_OK;
}

extern "C" size_t vaeq_frame_eval_scratch_bytes(int32_t n_runs, int32_t n_shift) {
    if (n_runs <= 0 || n_shift <= 0) return 0;
    return align_up((size_t)n_runs * 2 * n_shift * ER_CHUNKS * 8 * sizeof(double), 256) + align_up(((size_t)n_runs + ER_NORM_EXTRA) * 2 * sizeof(double), 256) +
           align_up((size_t)n_runs * 2 * 16 * sizeof(int), 256);
}

extern "C" int vaeq_frame_eval_runs_ex(const float *q, int64_t ld_q, int64_t rs_q, const float *out, int64_t ld_out, int64_t rs_out,
                                       const uint16_t *tx, int64_t ld_tx, int64_t rs_tx, const float *amp, const float *var, int64_t rs_var,
                                       const float *nu_sc, int32_t n_lev, int32_t N, int32_t n_shift, int32_t n_runs, int32_t seg_len,
                                       int32_t edge, int32_t n_cut, int32_t which, int32_t *align_out, int32_t *counts_out, float *ser_out,
                                       float *scale_out, void *scratch, void *stream) {
    VAEQ_CHECK_ARG(which >= 1 && which <= 3, "which=%d: bit 0 = estimator from q, bit 1 = estimator from out", which);
    VAEQ_CHECK_ARG((q || !(which & 1)) && (out || !(which & 2)) && tx && amp && var && nu_sc && align_out && ser_out && scratch, "NULL pointer");
    VAEQ_CHECK_ARG(n_lev == 2 || n_lev == 4 || n_lev == 8, "n_lev=%d must be 2, 4 or 8", n_lev);
    VAEQ_CHECK_ARG(N > 0 && n_runs > 0 && n_shift > 0 && n_shift <= 64 && edge >= 0 && n_cut >= 0, "bad sizes");
    VAEQ_CHECK_ARG(seg_len == 0 || (seg_len > 0 && N % seg_len == 0), "N=%d must be a multiple of seg_len=%d", N, seg_len);
    VAEQ_CHECK_ARG(n_runs <= 32767, "at most 32767 runs per call");
    cudaStream_t st = (cudaStream_t)stream;
    EvalRunsK p;
    p.q = q; p.ld_q = ld_q; p.rs_q = rs_q; p.out = out; p.ld_out = ld_out; p.rs_out = rs_out;
    p.tx = tx; p.ld_tx = ld_tx; p.rs_tx = rs_tx; p.amp = amp; p.var = var; p.rs_var = rs_var; p.nu_sc = nu_sc;
    p.n_lev = n_lev; p.N = N; p.n_shift = n_shift; p.n_runs = n_runs; p.seg_len = seg_len; p.edge = edge; p.n_cut = n_cut;
    char *ws = static_cast<char *>(scratch);
    const size_t part_b = align_up((size_t)n_runs * 2 * n_shift * ER_CHUNKS * 8 * sizeof(double), 256), norm_b = align_up(((size_t)n_runs + ER_NORM_EXTRA) * 2 * sizeof(double), 256);
    p.part = reinterpret_cast<double *>(ws);
    p.norms = reinterpret_cast<double *>(ws + part_b);
    p.counts = counts_out ? counts_out : reinterpret_cast<int *>(ws + part_b + norm_b);
    p.align = align_out; p.ser = ser_out; p.which = which; p.scale = scale_out;
    // enough CTAs to fill the GPU, as few partial blocks as possible: every CTA pays a prologue and a fixed-order reduction
    p.chunks = max(1, min(min(ER_CHUNKS, (N + 2 * SC_T - 1) / (2 * SC_T)), (4 * sm_count() + 2 * n_runs - 1) / (2 * n_runs)));
    VAEQ_CUDA(cudaMemsetAsync(p.counts, 0, (size_t)n_runs * 2 * 16 * sizeof(int), st));
    const int blocks = max(1, min((N + ER_NT - 1) / ER_NT, max(1, min(sm_count() * 8, ER_NORM_EXTRA) / n_runs)));     // n_runs * blocks <= n_runs + ER_NORM_EXTRA norm partials
#define ER_LAUNCH(name, ...)                    \
    ktime_begin(VAEQ_K_EVAL, st);               \
    __VA_ARGS__;                                \
    ktime_end(VAEQ_K_EVAL, st);                 \
    VAEQ_LAUNCH_CHECK(name);
    if (n_shift <= 8 * SC_J) { ER_LAUNCH("k_er_shift_corr", k_er_shift_corr<0><<<dim3(p.chunks, 2 * n_runs), SC_NT, 0, st>>>(p)) }
    else if (n_shift <= 32) { ER_LAUNCH("k_er_shift_corr", k_er_shift_corr<1><<<dim3(p.chunks, 2 * n_runs), SC_NT, 0, st>>>(p)) }
    else { ER_LAUNCH("k_er_shift_corr", k_er_shift_corr<2><<<dim3(p.chunks, 2 * n_runs), SC_NT, 0, st>>>(p)) }
    ER_LAUNCH("k_er_shift_decide", k_er_shift_decide<<<(2 * n_runs + ER_DEC_NT / 32 - 1) / (ER_DEC_NT / 32), ER_DEC_NT, 0, st>>>(p))
    if (which & 1) {
        if (n_lev == 2) { ER_LAUNCH("k_er_ser_iqflip", k_er_ser_iqflip<2><<<dim3(blocks, n_runs), ER_NT, 0, st>>>(p)) }
        else if (n_lev == 4) { ER_LAUNCH("k_er_ser_iqflip", k_er_ser_iqflip<4><<<dim3(blocks, n_runs), ER_NT, 0, st>>>(p)) }
        else { ER_LAUNCH("k_er_ser_iqflip", k_er_ser_iqflip<8><<<dim3(blocks, n_runs), ER_NT, 0, st>>>(p)) }
    }
    if (which & 2) {
        ER_LAUNCH("k_er_constell_norms", k_er_constell_norms<<<dim3(blocks, n_runs), ER_NT, 0, st>>>(p))
        if (n_lev == 2) { ER_LAUNCH("k_er_ser_constell", k_er_ser_constell<2><<<dim3(blocks, n_runs), ER_NT, 0, st>>>(p)) }
        else if (n_lev == 4) { ER_LAUNCH("k_er_ser_constell", k_er_ser_constell<4><<<dim3(blocks, n_runs), ER_NT, 0, st>>>(p)) }
        else { ER_LAUNCH("k_er_ser_constell", k_er_ser_constell<8><<<dim3(blocks, n_runs), ER_NT, 0, st>>>(p)) }
    }
    ER_LAUNCH("k_er_ser_min", k_er_ser_min<<<(4 * n_runs + 127) / 128, 128, 0, st>>>(p))
#undef ER_LAUNCH
    return VAEQ_OK;
}

extern "C" int vaeq_frame_eval_runs(const float *q, int64_t ld_q, int64_t rs_q, const float *out, int64_t ld_out, int64_t rs_out,
                                    const uint16_t *tx, int64_t ld_tx, int64_t rs_tx, const float *amp, const float *var, int64_t rs_var,
                                    const float *nu_sc, int32_t n_lev, int32_t N, int32_t n_shift, int32_t n_runs, int32_t seg_len,
                                    int32_t edge, int32_t n_cut, int32_t *align_out, int32_t *counts_out, float *ser_out, void *scratch,
                                    void *stream) {
    return vaeq_frame_eval_runs_ex(q, ld_q, rs_q, out, ld_out, rs_out, tx, ld_tx, rs_tx, amp, var, rs_var, nu_sc, n_lev, N, n_shift, n_runs,
                                   seg_len, edge, n_cut, 3, align_out, counts_out, ser_out, nullptr, scratch, stream);
}

extern "C" int vaeq_cma_align_rescale(const float *out, int64_t ld_out, int64_t rs_out, const int32_t *align, const float *scale, int32_t N,
                                      int32_t edge, int32_t n_runs, float *oc, void *stream) {
    VAEQ_CHECK_ARG(out && align && scale && oc && N > 0 && edge >= 0 && n_runs > 0 && n_runs <= 32767, "bad align_rescale arguments");
    cudaStream_t st = (cudaStream_t)stream;
    const int blocks = max(1, min((N + ER_NT - 1) / ER_NT, max(1, sm_count() * 8 / n_runs)));
    ktime_begin(VAEQ_K_EVAL, st);
    k_er_align_rescale<<<dim3(blocks, n_runs), ER_NT, 0, st>>>(out, ld_out, rs_out, align, scale, N, edge, oc);
    ktime_end(VAEQ_K_EVAL, st);
    VAEQ_LAUNCH_CHECK("k_er_align_rescale");
    return VAEQ_OK;
}
