// Single-polarisation CMA baseline of the AWGN module (AWGN_channel/func_CMA_MQAM_shaping.py, `cm:` below):
//   CMA :142-168 (complex FIR h[0] + j h[1], tap update after every symbol, NO power normalisation -- unlike the DP version sf:350),
//   SER_CMA :63-93 (in-place rescale, nearest-level decisions, 4 rotations), find_shift_symb :127-140 (non-circular correlation of
//   the first 1000 symbols).  CPE :170-196 (no unwrap) is cma.cu's pipeline with unwrap = 0.
// The output index k = i//sps - mh is negative for the first symbols and wraps to the END of out / e like in the DP version (cm:155).
#include <climits>

#include "common.cuh"

namespace vaeq {

// One frame of the recurrence for the calling warp (cm:147-166): lane `lane` owns taps lane + 32 sl in h0 / h1 (registers, updated
// in place when train != 0).  y: the frame's I row, its Q row ld_y further, N samples.  STORE bit 0 writes the output rows o
// (N / sps apart), bit 1 the error er; the output index wraps like cm:155.
template <int NSLOT, int STORE>
__device__ __forceinline__ void cma1_frame(const float *y, int ld_y, int N, int M, int sps, float R, float lr2, int train, int lane,
                                           float (&h0)[NSLOT], float (&h1)[NSLOT], float *o, float *er) {
    const int mh = M / 2, Nsym = N / sps;
    const int nsym_loop = (N + sps - 1) / sps;
    float n0[NSLOT], n1[NSLOT];                                  // the next symbol's window, loaded one iteration ahead
    auto load_window = [&](int ks) {
#pragma unroll
        for (int sl = 0; sl < NSLOT; ++sl) {
            const int k = lane + 32 * sl, s = ks * sps - mh + k;  // zero padding of mh samples per side (cm:149-150)
            const bool ok = (k < M) && (s >= 0) && (s < N);
            n0[sl] = ok ? y[s] : 0.f;
            n1[sl] = ok ? y[ld_y + s] : 0.f;
        }
    };
    load_window(0);
    for (int ks = 0; ks < nsym_loop; ++ks) {
        float y0[NSLOT], y1[NSLOT];
#pragma unroll
        for (int sl = 0; sl < NSLOT; ++sl) {
            y0[sl] = n0[sl];
            y1[sl] = n1[sl];
        }
        if (ks + 1 < nsym_loop) load_window(ks + 1);
        float a = 0.f, b = 0.f, c = 0.f, d = 0.f;                // y0.h0, y1.h1, y0.h1, y1.h0  (four matmuls, cm:157-158)
#pragma unroll
        for (int sl = 0; sl < NSLOT; ++sl) {
            a = fmaf(y0[sl], h0[sl], a);
            b = fmaf(y1[sl], h1[sl], b);
            c = fmaf(y0[sl], h1[sl], c);
            d = fmaf(y1[sl], h0[sl], d);
        }
        a = warp_sum(a);
        b = warp_sum(b);
        c = warp_sum(c);
        d = warp_sum(d);
        const float o0 = __fsub_rn(a, b), o1 = __fadd_rn(c, d);
        const float err = __fsub_rn(__fsub_rn(R, __fmul_rn(o0, o0)), __fmul_rn(o1, o1));      // cm:160
        if (STORE) {
            int k = (mh + ks * sps) / sps - mh;                  // cm:155
            if (k < 0) k += Nsym;
            if (lane == 0 && k >= 0 && k < Nsym) {
                if (STORE & 1) {
                    o[k] = o0;
                    o[Nsym + k] = o1;
                }
                if (STORE & 2) er[k] = err;
            }
        }
        if (train) {
            const float f = lr2 * err;
#pragma unroll
            for (int sl = 0; sl < NSLOT; ++sl) {                 // cm:163-164
                h0[sl] += f * (o0 * y0[sl] + o1 * y1[sl]);
                h1[sl] += f * (o1 * y0[sl] - o0 * y1[sl]);
            }
        }
    }
}

// one warp per run; lane l owns taps l and l + 32
template <int NSLOT>
__global__ void __launch_bounds__(32) k_cma1_sample(const float *Rx, float *h, float *out, float *e, int N, int M, int sps, float R,
                                                    float lr, int train) {
    const int lane = threadIdx.x, Nsym = N / sps;
    const float *y = Rx + (int64_t)blockIdx.x * 2 * N;
    float *hh = h + (int64_t)blockIdx.x * 2 * M, *o = out + (int64_t)blockIdx.x * 2 * Nsym, *er = e + (int64_t)blockIdx.x * Nsym;
    float h0[NSLOT], h1[NSLOT];
#pragma unroll
    for (int sl = 0; sl < NSLOT; ++sl) {
        const int k = lane + 32 * sl;
        h0[sl] = k < M ? hh[k] : 0.f;
        h1[sl] = k < M ? hh[M + k] : 0.f;
    }
    const float lr2 = 2.f * lr;
    cma1_frame<NSLOT, 3>(y, N, N, M, sps, R, lr2, train, lane, h0, h1, o, er);
    if (train) {
#pragma unroll
        for (int sl = 0; sl < NSLOT; ++sl) {
            const int k = lane + 32 * sl;
            if (k < M) {
                hh[k] = h0[sl];
                hh[M + k] = h1[sl];
            }
        }
    }
}

// A validation period of processing_cma_awgn (cm:221-231) for every run, one 32-thread CTA (one warp) per run: n_frames training
// frames in sequence with the taps in registers (no per-symbol output: the driver discards it), then the no-update pass over the
// validation frame into out_v (2, Nv / sps) per run, then the taps back to h.  The per-symbol arithmetic is cma1_frame, as in
// k_cma1_sample, and lr[run] is the fp32 value the scalar path receives, so run k equals a loop of single calls bit for bit.
template <int NSLOT>
__global__ void __launch_bounds__(32) k_cma1_runs(const float *rxt, int ld_t, int64_t fs_t, int64_t rs_t, int n_frames, int Nt,
                                                  const float *rxv, int ld_v, int64_t rs_v, int Nv, float *h, int M, const float *lr,
                                                  float R, int sps, float *out_v) {
    const int lane = threadIdx.x;
    const int64_t run = blockIdx.x;
    float *hh = h + run * 2 * M;
    float h0[NSLOT], h1[NSLOT];
#pragma unroll
    for (int sl = 0; sl < NSLOT; ++sl) {
        const int k = lane + 32 * sl;
        h0[sl] = k < M ? hh[k] : 0.f;
        h1[sl] = k < M ? hh[M + k] : 0.f;
    }
    const float lr2 = 2.f * lr[run];
    for (int f = 0; f < n_frames; ++f)
        cma1_frame<NSLOT, 0>(rxt + run * rs_t + f * fs_t, ld_t, Nt, M, sps, R, lr2, 1, lane, h0, h1, nullptr, nullptr);
    cma1_frame<NSLOT, 1>(rxv + run * rs_v, ld_v, Nv, M, sps, R, lr2, 0, lane, h0, h1, out_v + run * 2 * (Nv / sps), nullptr);
#pragma unroll
    for (int sl = 0; sl < NSLOT; ++sl) {
        const int k = lane + 32 * sl;
        if (k < M) {
            hh[k] = h0[sl];
            hh[M + k] = h1[sl];
        }
    }
}

// ---- SER_CMA (cm:63-93) --------------------------------------------------------------------------------------------------
constexpr int SC1_NT = 256;

// the CTA's share of sum |tx| and sum |rx| (cm:73) when nb CTAs of SC1_NT threads split N symbols: CTA blk takes t = blk SC1_NT + tid,
// stepping by nb SC1_NT; thread 0 returns the block sums
__device__ __forceinline__ void ser_cma_norms_cta(const float *rx, int64_t ld_rx, const uint16_t *tx, int64_t ld_tx, int N, unsigned blk, unsigned nb,
                                                  double *red, double (&acc)[2]) {
    for (int t = blk * SC1_NT + threadIdx.x; t < N; t += nb * SC1_NT) {
        const float a = half_bits_to_float(tx[t]), b = half_bits_to_float(tx[ld_tx + t]), x = rx[t], y = rx[ld_rx + t];
        acc[0] += (double)sqrtf(__fadd_rn(__fmul_rn(a, a), __fmul_rn(b, b)));
        acc[1] += (double)sqrtf(__fadd_rn(__fmul_rn(x, x), __fmul_rn(y, y)));
    }
    block_sum<2>(acc, red);
}

// the norm partials of nparts CTAs summed in a fixed order by the first warp (no floating-point atomics); thread 0 stores the totals
__device__ __forceinline__ void ser_cma_norms_total(const double *part, int nparts, double *bc) {
    if (threadIdx.x < 32) {
        double s0 = 0.0, s1 = 0.0;
        for (int i = threadIdx.x; i < nparts; i += 32) {
            s0 += part[2 * i];
            s1 += part[2 * i + 1];
        }
        s0 = warp_sum(s0);
        s1 = warp_sum(s1);
        if (threadIdx.x == 0) {
            bc[0] = s0;
            bc[1] = s1;
        }
    }
}

// nearest-level decisions of the rescaled symbol (sI, sQ) (torch.argmin: first minimum, cm:76), the tx levels decoded from fp16 with
// round half to even (cm:72) and the errors of the four rotations (cm:78-91)
template <int NL>
__device__ __forceinline__ void ser_cma_count(float sI, float sQ, uint16_t txI, uint16_t txQ, const float *a, int (&cnt)[4]) {
    const float scale = (float)((NL - 1) / 2.0);
    const int S = NL - 1;
    int dI = 0, dQ = 0;
    float bI = fabsf(__fsub_rn(sI, a[0])), bQ = fabsf(__fsub_rn(sQ, a[0]));
#pragma unroll
    for (int l = 1; l < NL; ++l) {
        const float vI = fabsf(__fsub_rn(sI, a[l])), vQ = fabsf(__fsub_rn(sQ, a[l]));
        if (vI < bI) {
            bI = vI;
            dI = l;
        }
        if (vQ < bQ) {
            bQ = vQ;
            dQ = l;
        }
    }
    const int xI = (int)rintf(__fadd_rn(__fmul_rn(scale, half_bits_to_float(txI)), scale));
    const int xQ = (int)rintf(__fadd_rn(__fmul_rn(scale, half_bits_to_float(txQ)), scale));
    cnt[0] += (xI != dI) || (xQ != dQ);                          // 0
    cnt[1] += (xI != S - dI) || (xQ != S - dQ);                  // pi          (cm:80)
    cnt[2] += (xI != S - dQ) || (xQ != dI);                      // "pi/4"      (cm:84-86)
    cnt[3] += (xI != dQ) || (xQ != S - dI);                      // "3pi/4"     (cm:89-91)
}

// block reduction of the four counters, one integer atomic per counter (order independent)
__device__ __forceinline__ void ser_cma_publish(int (&cnt)[4], int *red, int *counts) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        int v = cnt[k];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == 0) red[k * 32 + wid] = v;
    }
    __syncthreads();
    if (threadIdx.x < 4) {
        int v = 0;
        for (int w = 0; w < SC1_NT / 32; ++w) v += red[threadIdx.x * 32 + w];
        if (v) atomicAdd(&counts[threadIdx.x], v);
    }
}

// CTAs of the single-run SER_CMA over N symbols (vaeq_ser_cma); the norm partials' order depends on it
__host__ __device__ __forceinline__ int ser_cma_grid(int N, int nsm) {
    return max(1, min(min((N + SC1_NT - 1) / SC1_NT, nsm * 8), (int)(VAEQ_EVAL_SCRATCH_BYTES / (2 * sizeof(double)))));
}

__global__ void __launch_bounds__(SC1_NT) k_ser_cma_norms(const float *rx, int64_t ld_rx, const uint16_t *tx, int64_t ld_tx, int N, double *part) {
    __shared__ double red[2 * 32];
    double acc[2] = {0.0, 0.0};
    ser_cma_norms_cta(rx, ld_rx, tx, ld_tx, N, blockIdx.x, gridDim.x, red, acc);
    if (threadIdx.x == 0) {                                      // per-CTA partials, summed in fixed order by the consumer
        part[2 * blockIdx.x] = acc[0];
        part[2 * blockIdx.x + 1] = acc[1];
    }
}

template <int NL>
__global__ void __launch_bounds__(SC1_NT) k_ser_cma(float *rx, int64_t ld_rx, const uint16_t *tx, int64_t ld_tx, const float *amp, int N,
                                                    const double *part, int nparts, int *counts) {
    __shared__ double bc[2];
    __shared__ int red[4 * 32];
    __shared__ float a[NL];
    if (threadIdx.x < NL) a[threadIdx.x] = amp[threadIdx.x];
    ser_cma_norms_total(part, nparts, bc);
    __syncthreads();
    const float g = __fdiv_rn((float)(bc[0] / (double)N), (float)(bc[1] / (double)N));          // cm:73
    int cnt[4] = {0, 0, 0, 0};
    for (int t = blockIdx.x * SC1_NT + threadIdx.x; t < N; t += gridDim.x * SC1_NT) {
        const float sI = __fmul_rn(rx[t], g), sQ = __fmul_rn(rx[ld_rx + t], g);
        rx[t] = sI;                                              // in-place rescale, visible to the caller (cm:73)
        rx[ld_rx + t] = sQ;
        ser_cma_count<NL>(sI, sQ, tx[t], tx[ld_tx + t], a, cnt);
    }
    ser_cma_publish(cnt, red, counts);
}

__global__ void k_ser_cma_min(const int *counts, int N, float *ser) {
    if (threadIdx.x == 0) {
        float best = 1.f;                                        // SER = torch.ones(4) (cm:69)
        for (int r = 0; r < 4; ++r) best = fminf(best, __fdiv_rn((float)counts[r], (float)N));
        ser[0] = best;
    }
}

// ---- find_shift_symb (cm:127-140): corr_c[i] = sum_{t < win - half} tx_c[half + t] rx_I[i + t], i < n_shift, win = 1000 -----------
// the whole search for one run by the calling CTA: a warp per (component, shift), double sums in lane order, then thread 0 decides
__device__ __forceinline__ void find_shift_symb_cta(const float *rx, int n_rx, const uint16_t *tx, int64_t ld_tx, int n_shift, int win,
                                                    float *corr, int *shift, double (&acc)[2][64]) {
    const int half = n_shift / 2, len = win - half, lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    for (int job = wid; job < 2 * n_shift; job += nw) {          // a warp per (component, shift)
        const int c = job / n_shift, i = job - c * n_shift;
        double s = 0.0;
        for (int t = lane; t < len; t += 32) s += (double)half_bits_to_float(tx[(int64_t)c * ld_tx + half + t]) * (double)rx[i + t];
        s = warp_sum(s);
        if (lane == 0) acc[c][i] = s;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        float best[2] = {-1.f, -1.f};
        int arg[2] = {0, 0};
        for (int c = 0; c < 2; ++c)
            for (int i = 0; i < n_shift; ++i) {
                const float v = fabsf((float)acc[c][i]);
                corr[c * n_shift + i] = (float)acc[c][i];
                if (v > best[c]) {                               // torch.argmax: first maximum
                    best[c] = v;
                    arg[c] = i;
                }
            }
        int pick = arg[0];
        if (!(best[0] >= 0.02f * (float)n_rx) && best[1] >= best[0]) pick = arg[1];      // cm:133-140
        shift[0] = pick - half;
    }
}

__global__ void __launch_bounds__(1024) k_find_shift_symb(const float *rx, int n_rx, const uint16_t *tx, int64_t ld_tx, int n_shift, int win,
                                                          float *corr, int *shift) {
    __shared__ double acc[2][64];
    find_shift_symb_cta(rx, n_rx, tx, ld_tx, n_shift, win, corr, shift, acc);
}

// ---- validation scoring of processing_cma_awgn for R runs (cm:227-229), no host sync -------------------------------------------
//   shift = find_shift_symb(y, tx, n_shift);  SER_CMA(y[:, edge + shift : N - edge], tx[:, edge : N - edge - shift])
// The slices are index arithmetic on the device shift; L = N - 2 edge - shift symbols per run.  The norms are split over the CTAs
// the single-run call would use for L (ser_cma_grid) and summed in its order, so the scale g, the counts and the SER are bitwise
// those of the single-run sequence.  The in-place rescale of cm:73 is not written back: the driver never reads the slice again.
struct CmaEvalK {
    const float *y; int64_t ld_y, rs_y;          // (R, 2, N) CPE output
    const uint16_t *tx; int64_t ld_tx, rs_tx;    // (R, 2, N) float16 bits
    const float *amp;
    int N, n_shift, edge, nsm, gmax;
    float *corr;                                 // [R][2][n_shift] scratch
    double *part;                                // [R][gmax][2] scratch: norm partials
    int *shift, *counts;                         // [R], [R][4]
    float *ser;                                  // [R]
};

__global__ void __launch_bounds__(1024) k_cma_eval_shift(CmaEvalK p) {
    __shared__ double acc[2][64];
    const int64_t run = blockIdx.x;
    find_shift_symb_cta(p.y + run * p.rs_y, p.N, p.tx + run * p.rs_tx, p.ld_tx, p.n_shift, 1000, p.corr + run * 2 * p.n_shift,
                        p.shift + run, acc);
}

// grid (gmax, R): CTA b of run r is CTA b of the single-run k_ser_cma_norms over that run's slice (idle when b >= its grid)
__global__ void __launch_bounds__(SC1_NT) k_cma_eval_norms(CmaEvalK p) {
    __shared__ double red[2 * 32];
    const int64_t run = blockIdx.y;
    const int sh = p.shift[run], L = p.N - 2 * p.edge - sh, nb = ser_cma_grid(L, p.nsm);
    if ((int)blockIdx.x >= nb) return;                           // uniform over the CTA
    double acc[2] = {0.0, 0.0};
    ser_cma_norms_cta(p.y + run * p.rs_y + p.edge + sh, p.ld_y, p.tx + run * p.rs_tx + p.edge, p.ld_tx, L, blockIdx.x, nb, red, acc);
    if (threadIdx.x == 0) {
        double *dst = p.part + (run * p.gmax + blockIdx.x) * 2;
        dst[0] = acc[0];
        dst[1] = acc[1];
    }
}

template <int NL>
__global__ void __launch_bounds__(SC1_NT) k_cma_eval_count(CmaEvalK p) {
    __shared__ double bc[2];
    __shared__ int red[4 * 32];
    __shared__ float a[NL];
    const int64_t run = blockIdx.y;
    const int sh = p.shift[run], L = p.N - 2 * p.edge - sh;
    if (threadIdx.x < NL) a[threadIdx.x] = p.amp[threadIdx.x];
    ser_cma_norms_total(p.part + run * p.gmax * 2, ser_cma_grid(L, p.nsm), bc);
    __syncthreads();
    const float g = __fdiv_rn((float)(bc[0] / (double)L), (float)(bc[1] / (double)L));          // cm:73
    const float *y = p.y + run * p.rs_y + p.edge + sh;
    const uint16_t *tx = p.tx + run * p.rs_tx + p.edge;
    int cnt[4] = {0, 0, 0, 0};
    for (int t = blockIdx.x * SC1_NT + threadIdx.x; t < L; t += gridDim.x * SC1_NT)
        ser_cma_count<NL>(__fmul_rn(y[t], g), __fmul_rn(y[p.ld_y + t], g), tx[t], tx[p.ld_tx + t], a, cnt);
    ser_cma_publish(cnt, red, p.counts + run * 4);
}

// thread = run: min(1, count_k / L) as k_ser_cma_min computes it
__global__ void k_cma_eval_min(CmaEvalK p, int n_runs) {
    const int run = blockIdx.x * blockDim.x + threadIdx.x;
    if (run >= n_runs) return;
    const int L = p.N - 2 * p.edge - p.shift[run];
    float best = 1.f;
    for (int r = 0; r < 4; ++r) best = fminf(best, __fdiv_rn((float)p.counts[run * 4 + r], (float)L));
    p.ser[run] = best;
}

}  // namespace vaeq

using namespace vaeq;

extern "C" int vaeq_cma_awgn(const float *Rx, int32_t N, float R, float *h, int32_t M, float lr, int32_t sps, int32_t train, float *out,
                             float *e, int32_t n_runs, void *stream) {
    VAEQ_CHECK_ARG(Rx && h && out && e && N > 0 && n_runs > 0, "bad cma_awgn arguments");
    VAEQ_CHECK_ARG(M >= 1 && M <= VAEQ_MAX_TAPS && (M & 1), "M=%d must be odd and <= %d", M, VAEQ_MAX_TAPS);
    VAEQ_CHECK_ARG(sps >= 1 && N % sps == 0, "N=%d must be a multiple of sps=%d", N, sps);
    cudaStream_t st = (cudaStream_t)stream;
    ktime_begin(VAEQ_K_CMA, st);
    if (M <= 32) k_cma1_sample<1><<<n_runs, 32, 0, st>>>(Rx, h, out, e, N, M, sps, R, lr, train);
    else k_cma1_sample<2><<<n_runs, 32, 0, st>>>(Rx, h, out, e, N, M, sps, R, lr, train);
    ktime_end(VAEQ_K_CMA, st);
    VAEQ_LAUNCH_CHECK("k_cma1_sample");
    return VAEQ_OK;
}

extern "C" int vaeq_cma_awgn_runs(const float *rx_train, int64_t ld_t, int64_t fs_t, int64_t rs_t, int32_t n_frames, int32_t N_train,
                                  const float *rx_valid, int64_t ld_v, int64_t rs_v, int32_t N_valid, float *h, int32_t M, const float *lr,
                                  float R, int32_t sps, float *out_v, int32_t n_runs, void *stream) {
    VAEQ_CHECK_ARG(rx_valid && h && lr && out_v && n_runs > 0 && n_frames >= 0 && (rx_train || n_frames == 0), "bad cma_awgn_runs arguments");
    VAEQ_CHECK_ARG(M >= 1 && M <= VAEQ_MAX_TAPS && (M & 1), "M=%d must be odd and <= %d", M, VAEQ_MAX_TAPS);
    VAEQ_CHECK_ARG(sps >= 1 && N_valid > 0 && N_valid % sps == 0 && (n_frames == 0 || (N_train > 0 && N_train % sps == 0)),
                   "N_train=%d and N_valid=%d must be positive multiples of sps=%d", N_train, N_valid, sps);
    VAEQ_CHECK_ARG(ld_t >= 0 && ld_t <= INT_MAX && ld_v >= 0 && ld_v <= INT_MAX, "row strides must fit in 32 bits");
    cudaStream_t st = (cudaStream_t)stream;
    ktime_begin(VAEQ_K_CMA, st);
    if (M <= 32) k_cma1_runs<1><<<n_runs, 32, 0, st>>>(rx_train, (int)ld_t, fs_t, rs_t, n_frames, N_train, rx_valid, (int)ld_v, rs_v, N_valid, h, M, lr, R, sps, out_v);
    else k_cma1_runs<2><<<n_runs, 32, 0, st>>>(rx_train, (int)ld_t, fs_t, rs_t, n_frames, N_train, rx_valid, (int)ld_v, rs_v, N_valid, h, M, lr, R, sps, out_v);
    ktime_end(VAEQ_K_CMA, st);
    VAEQ_LAUNCH_CHECK("k_cma1_runs");
    return VAEQ_OK;
}

extern "C" int vaeq_ser_cma(float *rx, int64_t ld_rx, const uint16_t *tx, int64_t ld_tx, const float *amp, int32_t n_lev, int32_t N,
                            int32_t *counts_out, float *ser_out, void *scratch, void *stream) {
    VAEQ_CHECK_ARG(rx && tx && amp && counts_out && ser_out && scratch && N > 0, "bad ser_cma arguments");
    VAEQ_CHECK_ARG(n_lev == 2 || n_lev == 4 || n_lev == 8, "n_lev=%d must be 2, 4 or 8", n_lev);
    cudaStream_t st = (cudaStream_t)stream;
    double *part = static_cast<double *>(scratch);
    VAEQ_CUDA(cudaMemsetAsync(counts_out, 0, 4 * sizeof(int), st));
    const int grid = ser_cma_grid(N, sm_count());
    ktime_begin(VAEQ_K_EVAL, st);
    k_ser_cma_norms<<<grid, SC1_NT, 0, st>>>(rx, ld_rx, tx, ld_tx, N, part);
    ktime_end(VAEQ_K_EVAL, st);
    VAEQ_LAUNCH_CHECK("k_ser_cma_norms");
    ktime_begin(VAEQ_K_EVAL, st);
    switch (n_lev) {
        case 2: k_ser_cma<2><<<grid, SC1_NT, 0, st>>>(rx, ld_rx, tx, ld_tx, amp, N, part, grid, counts_out); break;
        case 4: k_ser_cma<4><<<grid, SC1_NT, 0, st>>>(rx, ld_rx, tx, ld_tx, amp, N, part, grid, counts_out); break;
        default: k_ser_cma<8><<<grid, SC1_NT, 0, st>>>(rx, ld_rx, tx, ld_tx, amp, N, part, grid, counts_out); break;
    }
    ktime_end(VAEQ_K_EVAL, st);
    VAEQ_LAUNCH_CHECK("k_ser_cma");
    ktime_begin(VAEQ_K_EVAL, st);
    k_ser_cma_min<<<1, 32, 0, st>>>(counts_out, N, ser_out);
    ktime_end(VAEQ_K_EVAL, st);
    VAEQ_LAUNCH_CHECK("k_ser_cma_min");
    return VAEQ_OK;
}

extern "C" int vaeq_find_shift_symb(const float *rx, int32_t n_rx, const uint16_t *tx, int64_t ld_tx, int32_t n_tx, int32_t n_shift,
                                    float *corr_out, int32_t *shift_out, void *stream) {
    VAEQ_CHECK_ARG(rx && tx && corr_out && shift_out, "NULL pointer");
    VAEQ_CHECK_ARG(n_shift > 0 && n_shift <= 64, "n_shift=%d must be in [1, 64]", n_shift);
    const int win = 1000;                                        // cm:128-131: the first 1000 symbols
    VAEQ_CHECK_ARG(n_tx >= win && n_rx >= win + n_shift / 2, "find_shift_symb needs at least %d symbols (got rx %d, tx %d)", win + n_shift / 2, n_rx, n_tx);
    cudaStream_t st = (cudaStream_t)stream;
    ktime_begin(VAEQ_K_EVAL, st);
    k_find_shift_symb<<<1, 1024, 0, st>>>(rx, n_rx, tx, ld_tx, n_shift, win, corr_out, shift_out);
    ktime_end(VAEQ_K_EVAL, st);
    VAEQ_LAUNCH_CHECK("k_find_shift_symb");
    return VAEQ_OK;
}

static int cma_eval_gmax(int32_t N, int32_t n_shift, int32_t edge, int nsm) { return ser_cma_grid(N - 2 * edge + n_shift / 2, nsm); }

extern "C" size_t vaeq_awgn_cma_eval_scratch_bytes(int32_t n_runs, int32_t N, int32_t n_shift, int32_t edge) {
    if (n_runs <= 0 || N <= 0 || n_shift <= 0 || edge < 0) return 0;
    return align_up((size_t)n_runs * 2 * n_shift * sizeof(float), 256) + (size_t)n_runs * cma_eval_gmax(N, n_shift, edge, sm_count()) * 2 * sizeof(double);
}

extern "C" int vaeq_awgn_cma_eval_runs(const float *y, int64_t ld_y, int64_t rs_y, const uint16_t *tx, int64_t ld_tx, int64_t rs_tx, const float *amp,
                                       int32_t n_lev, int32_t N, int32_t n_shift, int32_t edge, int32_t n_runs, int32_t *shift_out,
                                       int32_t *counts_out, float *ser_out, void *scratch, void *stream) {
    VAEQ_CHECK_ARG(y && tx && amp && shift_out && counts_out && ser_out && scratch, "NULL pointer");
    VAEQ_CHECK_ARG(n_lev == 2 || n_lev == 4 || n_lev == 8, "n_lev=%d must be 2, 4 or 8", n_lev);
    VAEQ_CHECK_ARG(n_shift > 0 && n_shift <= 64 && edge >= n_shift / 2, "n_shift=%d must be in [1, 64] and edge=%d >= n_shift / 2", n_shift, edge);
    const int win = 1000;                                        // cm:128-131: the first 1000 symbols
    VAEQ_CHECK_ARG(N >= win + n_shift / 2, "find_shift_symb needs at least %d symbols (got %d)", win + n_shift / 2, N);
    VAEQ_CHECK_ARG(N - 2 * edge - n_shift / 2 > 0, "N=%d leaves no symbol to evaluate", N);
    VAEQ_CHECK_ARG(n_runs > 0 && n_runs <= 65535, "n_runs=%d must be in 1..65535", n_runs);
    cudaStream_t st = (cudaStream_t)stream;
    CmaEvalK p;
    p.y = y; p.ld_y = ld_y; p.rs_y = rs_y; p.tx = tx; p.ld_tx = ld_tx; p.rs_tx = rs_tx; p.amp = amp;
    p.N = N; p.n_shift = n_shift; p.edge = edge; p.nsm = sm_count(); p.gmax = cma_eval_gmax(N, n_shift, edge, p.nsm);
    p.corr = static_cast<float *>(scratch);
    p.part = reinterpret_cast<double *>(static_cast<char *>(scratch) + align_up((size_t)n_runs * 2 * n_shift * sizeof(float), 256));
    p.shift = shift_out; p.counts = counts_out; p.ser = ser_out;
    VAEQ_CUDA(cudaMemsetAsync(counts_out, 0, (size_t)n_runs * 4 * sizeof(int), st));
    const int blocks = max(1, min((N + SC1_NT - 1) / SC1_NT, max(1, sm_count() * 8 / n_runs)));
#define CE_LAUNCH(name, ...)                    \
    ktime_begin(VAEQ_K_EVAL, st);               \
    __VA_ARGS__;                                \
    ktime_end(VAEQ_K_EVAL, st);                 \
    VAEQ_LAUNCH_CHECK(name);
    CE_LAUNCH("k_cma_eval_shift", k_cma_eval_shift<<<n_runs, 1024, 0, st>>>(p))
    CE_LAUNCH("k_cma_eval_norms", k_cma_eval_norms<<<dim3(p.gmax, n_runs), SC1_NT, 0, st>>>(p))
    if (n_lev == 2) { CE_LAUNCH("k_cma_eval_count", k_cma_eval_count<2><<<dim3(blocks, n_runs), SC1_NT, 0, st>>>(p)) }
    else if (n_lev == 4) { CE_LAUNCH("k_cma_eval_count", k_cma_eval_count<4><<<dim3(blocks, n_runs), SC1_NT, 0, st>>>(p)) }
    else { CE_LAUNCH("k_cma_eval_count", k_cma_eval_count<8><<<dim3(blocks, n_runs), SC1_NT, 0, st>>>(p)) }
    CE_LAUNCH("k_cma_eval_min", k_cma_eval_min<<<(n_runs + 127) / 128, 128, 0, st>>>(p, n_runs))
#undef CE_LAUNCH
    return VAEQ_OK;
}
