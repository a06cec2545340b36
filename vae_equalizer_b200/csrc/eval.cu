// Evaluation kernels: shift search and SER estimators (reference: optical_DP_channel/shared_funcs.py:188-338).
// All are single-pass HBM scans (q: 128 B/symbol at 64-QAM, out: 16 B, tx: 8 B as float16) with integer
// error COUNTS returned next to the float SER so that "bit-exact SER counts" is checkable.
#include "common.cuh"
#include "shift_corr.cuh"
#include "bits.cuh"

namespace vaeq {

constexpr int EV_NT = 256;
constexpr int EV_CHUNKS = 592;         // at most this many CTAs / partial blocks in find_shift (scratch = EV_CHUNKS*n_shift*8 doubles)

__device__ __forceinline__ float tx_level(uint16_t bits, float scale) {
    // round(scale*tx.float()+scale), two fp32 roundings then round-half-even like torch.round (sf:198, sf:239)
    return rintf(__fadd_rn(__fmul_rn(scale, half_bits_to_float(bits)), scale));
}

// V consecutive symbols per thread (V = 4: 16-byte float / 8-byte float16 loads when rows and N allow, else V = 1): the scans
// are HBM-bound and one 4-byte load per row and thread left them at 0.3-0.56 of the roofline (profiles/r01d_eval_cma.txt)
template <int V>
__device__ __forceinline__ void ld_f32(const float *p, float (&v)[V]) {
    if constexpr (V == 4) {
        const float4 x = __ldcs(reinterpret_cast<const float4 *>(p));
        v[0] = x.x; v[1] = x.y; v[2] = x.z; v[3] = x.w;
    } else {
        v[0] = *p;
    }
}
template <int V>
__device__ __forceinline__ void ld_f16(const uint16_t *p, float (&v)[V]) {
    if constexpr (V == 4) {
        const uint2 x = __ldcs(reinterpret_cast<const uint2 *>(p));
        v[0] = half_bits_to_float((uint16_t)(x.x & 0xffffu)); v[1] = half_bits_to_float((uint16_t)(x.x >> 16));
        v[2] = half_bits_to_float((uint16_t)(x.y & 0xffffu)); v[3] = half_bits_to_float((uint16_t)(x.y >> 16));
    } else {
        v[0] = half_bits_to_float(*p);
    }
}
__device__ __forceinline__ float tx_level_f(float x, float scale) { return rintf(__fadd_rn(__fmul_rn(scale, x), scale)); }
static bool ev_vec_ok(const void *a, int64_t ld_a, const void *tx, int64_t ld_tx, int N) {
    return (N % 4 == 0) && (ld_a % 4 == 0) && (ld_tx % 4 == 0) && (reinterpret_cast<uintptr_t>(a) % 16 == 0) &&
           (reinterpret_cast<uintptr_t>(tx) % 8 == 0);
}

// ---------------------------------------------------------------------------------------------
// find_shift / find_shift_symb_full
// ---------------------------------------------------------------------------------------------
// grid (chunks): CTA c scans its contiguous range of t once for ALL shifts (shift_corr.cuh) and writes part[c][i][k],
//   S[comp][b][a] = sum_t tx[a][comp][t] * E[b][(t - (i - half)) mod N]          (sf:300-304, circular roll), k = comp*4 + b*2 + a
template <bool FROM_Q, int NPASS>
__global__ void __launch_bounds__(SC_NT, (FROM_Q || NPASS == 0) ? 4 : SC_MINB) k_shift_corr(const float *q, int64_t ld_q, const float *out, int64_t ld_out,
                                                      const uint16_t *tx, int64_t ld_tx, const float *amp, int n_lev,
                                                      int N, int n_shift, int64_t per, double *part) {
    __shared__ ShiftSmem sm;
    const int64_t t_lo = (int64_t)blockIdx.x * per, t_hi = min((int64_t)N, t_lo + per);
    shift_corr_range<FROM_Q, NPASS>(sm, q, ld_q, out, ld_out, tx, ld_tx, amp, n_lev, N, n_shift, t_lo, t_hi,
                             part + (int64_t)blockIdx.x * n_shift * 8);
}

// one CTA: thread = (chunk group g, idx = (i, k)); consecutive threads read consecutive doubles of a partial block (coalesced),
// a group sums chunks g, g + ng, ...; the groups are then added in fixed order; thread 0 replays the torch.max / argmax logic of
// sf:303-314 (first index wins ties)
__global__ void __launch_bounds__(1024) k_shift_decide(const double *part, int n_shift, int chunks, float *corr_out, int16_t *shift_out, int *r_out) {
    __shared__ float v_s[8][SC_MAXSHIFT];
    __shared__ double ps[1024];
    const int half = n_shift / 2, nidx = n_shift * 8, lanes = (nidx + 31) & ~31, ng = max(1, (int)blockDim.x / lanes);
    const int il = threadIdx.x % lanes, gq = threadIdx.x / lanes;
    double s = 0.0;
    if (gq < ng && il < nidx) {
        int c = gq;
        for (; c + 15 * ng < chunks; c += 16 * ng) {        // 16 independent loads in flight (the kernel is one CTA of pure L2 latency); same order of additions
            double v[16];
#pragma unroll
            for (int k = 0; k < 16; ++k) v[k] = part[(int64_t)(c + k * ng) * nidx + il];
#pragma unroll
            for (int k = 0; k < 16; ++k) s += v[k];
        }
        for (; c < chunks; c += ng) s += part[(int64_t)c * nidx + il];
    }
    ps[threadIdx.x] = s;
    __syncthreads();
    if (threadIdx.x < nidx) {
        double t = 0.0;
        for (int g = 0; g < ng; ++g) t += ps[g * lanes + threadIdx.x];
        const int i = threadIdx.x >> 3, k = threadIdx.x & 7;
        const float v = fabsf((float)t);
        v_s[k][i] = v;
        if (corr_out) corr_out[k * n_shift + i] = v;
    }
    __syncthreads();
    if (threadIdx.x != 0) return;
    float cmax[8];
    int cind[8];
    for (int k = 0; k < 8; ++k) {                            // k = comp*4 + b*2 + a
        cmax[k] = -1.f;
        cind[k] = 0;
        for (int i = 0; i < n_shift; ++i) {
            const float v = v_s[k][i];
            if (v > cmax[k]) {
                cmax[k] = v;
                cind[k] = i;
            }
        }
    }
    float best[4];
    int which[4];
    for (int ba = 0; ba < 4; ++ba) {                         // max over the tx component, first wins
        which[ba] = (cmax[4 + ba] > cmax[ba]) ? 1 : 0;
        best[ba] = which[ba] ? cmax[4 + ba] : cmax[ba];
    }
    // ba index = b*2 + a
    const bool straight = (best[0] + best[3]) >= (best[1] + best[2]);
    if (straight) {
        shift_out[0] = (int16_t)(half - cind[which[0] * 4 + 0]);
        shift_out[1] = (int16_t)(half - cind[which[3] * 4 + 3]);
        *r_out = 0;
    } else {
        shift_out[0] = (int16_t)(half - cind[which[1] * 4 + 1]);
        shift_out[1] = (int16_t)(half - cind[which[2] * 4 + 2]);
        *r_out = 1;
    }
}

// ---------------------------------------------------------------------------------------------
// SER from posteriors: hard decision argmax(q), 4 rotations x IQ flip (sf:188-222)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void count_hypotheses(int (&cnt)[8], float DI, float DQ, float S, const float (&hI)[4],
                                                 const float (&hQ)[4]) {
    const float DQf = S - DQ;                                 // IQ-flipped reference data (sf:199)
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        cnt[r] += (DI != hI[r]) || (DQ != hQ[r]);
        cnt[4 + r] += (DI != hI[r]) || (DQf != hQ[r]);
    }
}

template <int NL, int V>
__global__ void __launch_bounds__(EV_NT) k_ser_iqflip(const float *q, int64_t ld_q, const uint16_t *tx, int64_t ld_tx,
                                                      int N, int *counts) {
    __shared__ int red[16 * 32];
    const float S = (float)(NL - 1), scale = (float)((NL - 1) / 2.0);
    int cnt[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) cnt[k] = 0;
    for (int64_t t = ((int64_t)blockIdx.x * EV_NT + threadIdx.x) * V; t < N; t += (int64_t)gridDim.x * EV_NT * V) {
#pragma unroll
        for (int p = 0; p < 2; ++p) {
            int d[2][V];
#pragma unroll
            for (int c = 0; c < 2; ++c) {                     // torch.argmax: first maximal index
                float best[V], v[V];
                ld_f32<V>(q + (int64_t)(p * 2 * NL + c * NL) * ld_q + t, best);
#pragma unroll
                for (int k = 0; k < V; ++k) d[c][k] = 0;
#pragma unroll
                for (int l = 1; l < NL; ++l) {
                    ld_f32<V>(q + (int64_t)(p * 2 * NL + c * NL + l) * ld_q + t, v);
#pragma unroll
                    for (int k = 0; k < V; ++k)
                        if (v[k] > best[k]) {
                            best[k] = v[k];
                            d[c][k] = l;
                        }
                }
            }
            float xI[V], xQ[V];
            ld_f16<V>(tx + (int64_t)(p * 2 + 0) * ld_tx + t, xI);
            ld_f16<V>(tx + (int64_t)(p * 2 + 1) * ld_tx + t, xQ);
#pragma unroll
            for (int k = 0; k < V; ++k) {
                const float dI = (float)d[0][k], dQ = (float)d[1][k];
                const float hI[4] = {dI, S - dI, S - dQ, dQ};     // 0, pi, pi/2, 3pi/2  (sf:201-219)
                const float hQ[4] = {dQ, S - dQ, dI, S - dI};
                const float DI = tx_level_f(xI[k], scale), DQ = tx_level_f(xQ[k], scale);
                int c8[8] = {0, 0, 0, 0, 0, 0, 0, 0};
                count_hypotheses(c8, DI, DQ, S, hI, hQ);
#pragma unroll
                for (int r = 0; r < 4; ++r) {                     // counts[flip][pol][rot]
                    cnt[(0 * 2 + p) * 4 + r] += c8[r];
                    cnt[(1 * 2 + p) * 4 + r] += c8[4 + r];
                }
            }
        }
    }
    // block reduction of 16 integer counters, then one atomic per counter (integer: order independent)
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
        for (int w = 0; w < EV_NT / 32; ++w) v += red[threadIdx.x * 32 + w];
        if (v) atomicAdd(&counts[threadIdx.x], v);
    }
}

__global__ void k_ser_min(const int *counts, int N, float *ser_out) {
    if (threadIdx.x < 2) {
        const int p = threadIdx.x;
        float best = 3.0e38f;
        for (int f = 0; f < 2; ++f)
            for (int r = 0; r < 4; ++r) best = fminf(best, __fdiv_rn((float)counts[(f * 2 + p) * 4 + r], (float)N));
        ser_out[p] = best;                                    // torch.amin over (flip, rotation)  (sf:221, sf:264)
    }
}


// Sum of per-CTA partial pairs in a FIXED order (no floating-point atomics: the result is bit-reproducible for a given grid):
// warp 0 strides over the partials, then a butterfly; the pair is broadcast through shared memory.  All threads must call.
__device__ __forceinline__ void fixed_order_sum2(const double *part, int n, double *bc /* __shared__ [2] */, double &s0, double &s1) {
    if (threadIdx.x < 32) {
        double a = 0.0, b = 0.0;
        for (int i = threadIdx.x; i < n; i += 32) {
            a += part[2 * i];
            b += part[2 * i + 1];
        }
        a = warp_sum(a);
        b = warp_sum(b);
        if (threadIdx.x == 0) {
            bc[0] = a;
            bc[1] = b;
        }
    }
    __syncthreads();
    s0 = bc[0];
    s1 = bc[1];
}

// ---------------------------------------------------------------------------------------------
// SER from the constellation with PCS-aware thresholds (sf:225-287)
// ---------------------------------------------------------------------------------------------
template <int V>
__global__ void __launch_bounds__(EV_NT) k_constell_norms(const float *rx, int64_t ld_rx, const uint16_t *tx, int64_t ld_tx,
                                                          int N, double *sums) {
    __shared__ double red[2 * 32];
    double acc[2] = {0.0, 0.0};
    for (int64_t t = ((int64_t)blockIdx.x * EV_NT + threadIdx.x) * V; t < N; t += (int64_t)gridDim.x * EV_NT * V) {
#pragma unroll
        for (int p = 0; p < 2; ++p) {
            float a[V], b[V], x[V], y[V];
            ld_f16<V>(tx + (int64_t)(p * 2) * ld_tx + t, a);
            ld_f16<V>(tx + (int64_t)(p * 2 + 1) * ld_tx + t, b);
            ld_f32<V>(rx + (int64_t)(p * 2) * ld_rx + t, x);
            ld_f32<V>(rx + (int64_t)(p * 2 + 1) * ld_rx + t, y);
#pragma unroll
            for (int k = 0; k < V; ++k) {
                acc[0] += (double)sqrtf(__fadd_rn(__fmul_rn(a[k], a[k]), __fmul_rn(b[k], b[k])));
                acc[1] += (double)sqrtf(__fadd_rn(__fmul_rn(x[k], x[k]), __fmul_rn(y[k], y[k])));
            }
        }
    }
    block_sum<2>(acc, red);
    if (threadIdx.x == 0) {                                   // per-CTA partials, summed in fixed order by the consumer
        sums[2 * blockIdx.x] = acc[0];
        sums[2 * blockIdx.x + 1] = acc[1];
    }
}

template <int NL, int V>
__global__ void __launch_bounds__(EV_NT) k_ser_constell(float *rx, int64_t ld_rx, const uint16_t *tx, int64_t ld_tx,
                                                        const float *amp, const float *var, float nu_sc, int N,
                                                        const double *sums, int nparts, int *counts) {
    __shared__ int red[16 * 32];
    __shared__ float lo[NL], hi[NL];
    __shared__ double bc[2];
    double sum_tx, sum_rx;
    fixed_order_sum2(sums, nparts, bc, sum_tx, sum_rx);
    if (threadIdx.x < NL) {
        const int l = threadIdx.x;
        // d = (1 + 2 nu_sc var[0]) (a_l + a_{l+1}) / 2, padded with -inf / +inf  (sf:234-236)
        const float f = __fadd_rn(1.f, __fmul_rn(2.f * nu_sc, var[0]));
        lo[l] = (l == 0) ? -INFINITY : __fmul_rn(f, __fadd_rn(amp[l - 1], amp[l])) * 0.5f;
        hi[l] = (l == NL - 1) ? INFINITY : __fmul_rn(f, __fadd_rn(amp[l], amp[l + 1])) * 0.5f;
    }
    __syncthreads();
    const double cnt2 = 2.0 * (double)N;
    const float g = __fdiv_rn((float)(sum_tx / cnt2), (float)(sum_rx / cnt2));      // sf:242
    const float S = (float)(NL - 1), scale = (float)((NL - 1) / 2.0);
    int cnt[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) cnt[k] = 0;
    for (int64_t t = ((int64_t)blockIdx.x * EV_NT + threadIdx.x) * V; t < N; t += (int64_t)gridDim.x * EV_NT * V) {
#pragma unroll
        for (int p = 0; p < 2; ++p) {
            float *pI = rx + (int64_t)(p * 2) * ld_rx + t, *pQ = rx + (int64_t)(p * 2 + 1) * ld_rx + t;
            float yI[V], yQ[V], xI[V], xQ[V];
            ld_f32<V>(pI, yI);
            ld_f32<V>(pQ, yQ);
            ld_f16<V>(tx + (int64_t)(p * 2) * ld_tx + t, xI);
            ld_f16<V>(tx + (int64_t)(p * 2 + 1) * ld_tx + t, xQ);
#pragma unroll
            for (int k = 0; k < V; ++k) {
                yI[k] = __fmul_rn(yI[k], g);
                yQ[k] = __fmul_rn(yQ[k], g);
            }
            if constexpr (V == 4) {                           // in-place rescale, visible to the caller (sf:242)
                *reinterpret_cast<float4 *>(pI) = make_float4(yI[0], yI[1], yI[2], yI[3]);
                *reinterpret_cast<float4 *>(pQ) = make_float4(yQ[0], yQ[1], yQ[2], yQ[3]);
            } else {
                *pI = yI[0];
                *pQ = yQ[0];
            }
#pragma unroll
            for (int k = 0; k < V; ++k) {
                const float DI = tx_level_f(xI[k], scale), DQ = tx_level_f(xQ[k], scale);
                const float DQf = S - DQ;
                const int iI = min(max((int)DI, 0), NL - 1), iQ = min(max((int)DQ, 0), NL - 1), iQf = min(max((int)DQf, 0), NL - 1);
                const float hI[4] = {yI[k], -yI[k], -yQ[k], yQ[k]};           // sf:245-262
                const float hQ[4] = {yQ[k], -yQ[k], yI[k], -yI[k]};
#pragma unroll
                for (int r = 0; r < 4; ++r) {
                    const bool okI = (lo[iI] <= hI[r]) && (hI[r] < hi[iI]);
                    const bool okQ = (lo[iQ] <= hQ[r]) && (hQ[r] < hi[iQ]);
                    const bool okQf = (lo[iQf] <= hQ[r]) && (hQ[r] < hi[iQf]);
                    cnt[(0 * 2 + p) * 4 + r] += !(okI && okQ);
                    cnt[(1 * 2 + p) * 4 + r] += !(okI && okQf);
                }
            }
        }
    }
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
        for (int w = 0; w < EV_NT / 32; ++w) v += red[threadIdx.x * 32 + w];
        if (v) atomicAdd(&counts[threadIdx.x], v);
    }
}

// ---------------------------------------------------------------------------------------------
// extension (not in the reference): GMI-style achievable rate from the posteriors
// ---------------------------------------------------------------------------------------------
// BITS: the bit-metric rate (BMI) instead, H(X) + the mean of sum_i log2 q(b_i = bit i of g(x_tx) | y) over the I and Q components
// (bits.cuh); it reads every row of q at the thread's symbols, V at a time
template <int NL, int V, bool BITS>
__global__ void __launch_bounds__(EV_NT) k_gmi(const float *q, int64_t ld_q, const uint16_t *tx, int64_t ld_tx, int N, double *sums) {
    __shared__ double red[2 * 32];
    const float scale = (float)((NL - 1) / 2.0);
    double acc[2] = {0.0, 0.0};
    for (int64_t t = ((int64_t)blockIdx.x * EV_NT + threadIdx.x) * V; t < N; t += (int64_t)gridDim.x * EV_NT * V) {
#pragma unroll
        for (int p = 0; p < 2; ++p) {
            float xI[V], xQ[V];
            ld_f16<V>(tx + (int64_t)(p * 2) * ld_tx + t, xI);
            ld_f16<V>(tx + (int64_t)(p * 2 + 1) * ld_tx + t, xQ);
            if constexpr (BITS) {
                float qI[NL][V], qQ[NL][V];
#pragma unroll
                for (int l = 0; l < NL; ++l) {
                    ld_f32<V>(q + (int64_t)(p * 2 * NL + l) * ld_q + t, qI[l]);
                    ld_f32<V>(q + (int64_t)(p * 2 * NL + NL + l) * ld_q + t, qQ[l]);
                }
#pragma unroll
                for (int k = 0; k < V; ++k) {
                    const int iI = min(max((int)tx_level_f(xI[k], scale), 0), NL - 1);
                    const int iQ = min(max((int)tx_level_f(xQ[k], scale), 0), NL - 1);
                    float vI[NL], vQ[NL];
#pragma unroll
                    for (int l = 0; l < NL; ++l) {
                        vI[l] = qI[l][k];
                        vQ[l] = qQ[l][k];
                    }
                    acc[p] += bmi_log2_component<NL>(vI, iI) + bmi_log2_component<NL>(vQ, iQ);
                }
            } else {
#pragma unroll
                for (int k = 0; k < V; ++k) {
                    const int iI = min(max((int)tx_level_f(xI[k], scale), 0), NL - 1);
                    const int iQ = min(max((int)tx_level_f(xQ[k], scale), 0), NL - 1);
                    const float qi = q[(int64_t)(p * 2 * NL + iI) * ld_q + t + k], qq = q[(int64_t)(p * 2 * NL + NL + iQ) * ld_q + t + k];
                    acc[p] += log2((double)fmaxf(qi, 1e-30f)) + log2((double)fmaxf(qq, 1e-30f));
                }
            }
        }
    }
    block_sum<2>(acc, red);
    if (threadIdx.x == 0) {
        sums[2 * blockIdx.x] = acc[0];
        sums[2 * blockIdx.x + 1] = acc[1];
    }
}
__global__ void k_gmi_fin(const double *sums, int nparts, const float *P, int n_lev, int N, float *gmi_out) {
    __shared__ double bc[2];
    double s[2];
    fixed_order_sum2(sums, nparts, bc, s[0], s[1]);
    if (threadIdx.x < 2) {
        double H = 0.0;
        for (int l = 0; l < n_lev; ++l) H -= 2.0 * (double)P[l] * log2((double)P[l]);
        gmi_out[threadIdx.x] = (float)(H + s[threadIdx.x] / (double)N);
    }
}

// Bit LLRs of R runs: q (R, 2, 2n, N) -> llr (R, 2, 2m, N), rows [I bits MSB..LSB | Q bits MSB..LSB] per pol,
// L = ln max(q(b = 0 | y), 1e-30) - ln max(q(b = 1 | y), 1e-30) (positive: bit 0), the bit posteriors of bits.cuh.  grid (blocks, R);
// a thread owns V consecutive symbols (V = 4: 16-byte loads and streaming stores, as k_soft_dec_vec)
template <int NL, int V>
__global__ void __launch_bounds__(EV_NT) k_bit_llr(const float *__restrict__ q, int64_t ld_q, int64_t rs_q, int N, float *__restrict__ llr,
                                                   int64_t ld_llr, int64_t rs_llr) {
    constexpr int m = gray_bits<NL>();
    q += (int64_t)blockIdx.y * rs_q;
    llr += (int64_t)blockIdx.y * rs_llr;
    for (int64_t t = ((int64_t)blockIdx.x * EV_NT + threadIdx.x) * V; t < N; t += (int64_t)gridDim.x * EV_NT * V) {
#pragma unroll
        for (int c = 0; c < 4; ++c) {                          // (pol, component): q rows c NL .., llr rows c m ..
            float qv[NL][V], L[m][V];
#pragma unroll
            for (int l = 0; l < NL; ++l) ld_f32<V>(q + (int64_t)(c * NL + l) * ld_q + t, qv[l]);
#pragma unroll
            for (int k = 0; k < V; ++k) {
                float v[NL], pb[m][2];
#pragma unroll
                for (int l = 0; l < NL; ++l) v[l] = qv[l][k];
                bit_marginals<NL>(v, pb);
#pragma unroll
                for (int i = 0; i < m; ++i) L[i][k] = logf(fmaxf(pb[i][0], 1e-30f)) - logf(fmaxf(pb[i][1], 1e-30f));
            }
#pragma unroll
            for (int i = 0; i < m; ++i) {
                float *dst = llr + (int64_t)(c * m + i) * ld_llr + t;
                if constexpr (V == 4) stg_stream(reinterpret_cast<float4 *>(dst), make_float4(L[i][0], L[i][1], L[i][2], L[i][3]));
                else *dst = L[i][0];
            }
        }
    }
}

static int ev_grid(int N, int V = 1) { return max(1, min(min((N / V + EV_NT - 1) / EV_NT, sm_count() * 8), (int)(VAEQ_EVAL_SCRATCH_BYTES / (2 * sizeof(double))))); }

}  // namespace vaeq

using namespace vaeq;

extern "C" size_t vaeq_find_shift_scratch_bytes(int32_t n_shift) {
    return n_shift > 0 ? (size_t)EV_CHUNKS * n_shift * 8 * sizeof(double) : 0;
}

extern "C" int vaeq_find_shift(const float *q, int64_t ld_q, const float *out, int64_t ld_out, const uint16_t *tx,
                               int64_t ld_tx, const float *amp, int32_t n_lev, int32_t N, int32_t n_shift, float *corr_out,
                               int16_t *shift_out, int32_t *r_out, void *scratch, void *stream) {
    VAEQ_CHECK_ARG((q != nullptr) != (out != nullptr), "exactly one of q / out must be given");
    VAEQ_CHECK_ARG(tx && shift_out && r_out && scratch && N > 0 && n_shift > 0 && n_shift <= 64, "bad find_shift arguments");
    VAEQ_CHECK_ARG(!q || (amp && n_lev >= 1 && n_lev <= VAEQ_MAX_LEVELS), "bad amp / n_lev");
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t tiles = ((int64_t)N + SC_T - 1) / SC_T;
    const int chunks = (int)min((int64_t)min(EV_CHUNKS, 4 * sm_count()), tiles);
    const int64_t per = (tiles + chunks - 1) / chunks * SC_T;
    const int grid = (int)(((int64_t)N + per - 1) / per);
    double *part = static_cast<double *>(scratch);
    const bool one = n_shift <= 32;
    ktime_begin(VAEQ_K_EVAL, st);
    if (q && n_shift <= 8 * SC_J) k_shift_corr<true, 0><<<grid, SC_NT, 0, st>>>(q, ld_q, nullptr, 0, tx, ld_tx, amp, n_lev, N, n_shift, per, part);
    else if (n_shift <= 8 * SC_J) k_shift_corr<false, 0><<<grid, SC_NT, 0, st>>>(nullptr, 0, out, ld_out, tx, ld_tx, nullptr, 0, N, n_shift, per, part);
    else if (q && one) k_shift_corr<true, 1><<<grid, SC_NT, 0, st>>>(q, ld_q, nullptr, 0, tx, ld_tx, amp, n_lev, N, n_shift, per, part);
    else if (q) k_shift_corr<true, 2><<<grid, SC_NT, 0, st>>>(q, ld_q, nullptr, 0, tx, ld_tx, amp, n_lev, N, n_shift, per, part);
    else if (one) k_shift_corr<false, 1><<<grid, SC_NT, 0, st>>>(nullptr, 0, out, ld_out, tx, ld_tx, nullptr, 0, N, n_shift, per, part);
    else k_shift_corr<false, 2><<<grid, SC_NT, 0, st>>>(nullptr, 0, out, ld_out, tx, ld_tx, nullptr, 0, N, n_shift, per, part);
    ktime_end(VAEQ_K_EVAL, st);
    VAEQ_LAUNCH_CHECK("k_shift_corr");
    ktime_begin(VAEQ_K_EVAL, st);
    k_shift_decide<<<1, 1024, 0, st>>>(part, n_shift, grid, corr_out, shift_out, r_out);
    ktime_end(VAEQ_K_EVAL, st);
    VAEQ_LAUNCH_CHECK("k_shift_decide");
    return VAEQ_OK;
}

extern "C" int vaeq_ser_iqflip(const float *q, int64_t ld_q, const uint16_t *tx, int64_t ld_tx, int32_t n_lev, int32_t N,
                               int32_t *counts_out, float *ser_out, void *stream) {
    VAEQ_CHECK_ARG(q && tx && counts_out && ser_out && N > 0, "bad ser_iqflip arguments");
    VAEQ_CHECK_ARG(n_lev == 2 || n_lev == 4 || n_lev == 8, "n_lev=%d must be 2, 4 or 8", n_lev);
    cudaStream_t st = (cudaStream_t)stream;
    VAEQ_CUDA(cudaMemsetAsync(counts_out, 0, 16 * sizeof(int), st));
    const bool vec = ev_vec_ok(q, ld_q, tx, ld_tx, N);
    const int grid = ev_grid(N, vec ? 4 : 1);
    ktime_begin(VAEQ_K_EVAL, st);
#define EV_CASE(NL_)                                                                                         \
    if (vec) k_ser_iqflip<NL_, 4><<<grid, EV_NT, 0, st>>>(q, ld_q, tx, ld_tx, N, counts_out);                \
    else k_ser_iqflip<NL_, 1><<<grid, EV_NT, 0, st>>>(q, ld_q, tx, ld_tx, N, counts_out);
    if (n_lev == 2) { EV_CASE(2) } else if (n_lev == 4) { EV_CASE(4) } else { EV_CASE(8) }
#undef EV_CASE
    ktime_end(VAEQ_K_EVAL, st);
    VAEQ_LAUNCH_CHECK("k_ser_iqflip");
    ktime_begin(VAEQ_K_EVAL, st);
    k_ser_min<<<1, 32, 0, st>>>(counts_out, N, ser_out);
    ktime_end(VAEQ_K_EVAL, st);
    VAEQ_LAUNCH_CHECK("k_ser_min");
    return VAEQ_OK;
}

extern "C" int vaeq_ser_constell(float *rx, int64_t ld_rx, const uint16_t *tx, int64_t ld_tx, const float *amp,
                                 const float *var, float nu_sc, int32_t n_lev, int32_t N, int32_t *counts_out,
                                 float *ser_out, void *scratch, void *stream) {
    VAEQ_CHECK_ARG(rx && tx && amp && var && counts_out && ser_out && scratch && N > 0, "bad ser_constell arguments");
    VAEQ_CHECK_ARG(n_lev == 2 || n_lev == 4 || n_lev == 8, "n_lev=%d must be 2, 4 or 8", n_lev);
    cudaStream_t st = (cudaStream_t)stream;
    double *sums = static_cast<double *>(scratch);           // [grid][2] per-CTA partials (VAEQ_EVAL_SCRATCH_BYTES covers the largest grid)
    VAEQ_CUDA(cudaMemsetAsync(counts_out, 0, 16 * sizeof(int), st));
    const bool vec = ev_vec_ok(rx, ld_rx, tx, ld_tx, N);
    const int grid = ev_grid(N, vec ? 4 : 1);
    ktime_begin(VAEQ_K_EVAL, st);
    if (vec) k_constell_norms<4><<<grid, EV_NT, 0, st>>>(rx, ld_rx, tx, ld_tx, N, sums);
    else k_constell_norms<1><<<grid, EV_NT, 0, st>>>(rx, ld_rx, tx, ld_tx, N, sums);
    ktime_end(VAEQ_K_EVAL, st);
    VAEQ_LAUNCH_CHECK("k_constell_norms");
    ktime_begin(VAEQ_K_EVAL, st);
#define EV_CASE(NL_)                                                                                                          \
    if (vec) k_ser_constell<NL_, 4><<<grid, EV_NT, 0, st>>>(rx, ld_rx, tx, ld_tx, amp, var, nu_sc, N, sums, grid, counts_out);      \
    else k_ser_constell<NL_, 1><<<grid, EV_NT, 0, st>>>(rx, ld_rx, tx, ld_tx, amp, var, nu_sc, N, sums, grid, counts_out);
    if (n_lev == 2) { EV_CASE(2) } else if (n_lev == 4) { EV_CASE(4) } else { EV_CASE(8) }
#undef EV_CASE
    ktime_end(VAEQ_K_EVAL, st);
    VAEQ_LAUNCH_CHECK("k_ser_constell");
    ktime_begin(VAEQ_K_EVAL, st);
    k_ser_min<<<1, 32, 0, st>>>(counts_out, N, ser_out);
    ktime_end(VAEQ_K_EVAL, st);
    VAEQ_LAUNCH_CHECK("k_ser_min");
    return VAEQ_OK;
}

static int rate(const float *q, int64_t ld_q, const uint16_t *tx, int64_t ld_tx, const float *P, int32_t n_lev, int32_t N, float *gmi_out,
                void *scratch, void *stream, bool bits) {
    VAEQ_CHECK_ARG(q && tx && P && gmi_out && scratch && N > 0, "bad gmi arguments");
    VAEQ_CHECK_ARG(n_lev == 2 || n_lev == 4 || n_lev == 8, "n_lev=%d must be 2, 4 or 8", n_lev);
    cudaStream_t st = (cudaStream_t)stream;
    double *sums = static_cast<double *>(scratch);           // [grid][2] per-CTA partials (VAEQ_EVAL_SCRATCH_BYTES covers the largest grid)
    const bool vec = ev_vec_ok(q, ld_q, tx, ld_tx, N);
    const int grid = ev_grid(N, vec ? 4 : 1);
    ktime_begin(VAEQ_K_EVAL, st);
#define EV_CASE(NL_, B_)                                                                    \
    if (vec) k_gmi<NL_, 4, B_><<<grid, EV_NT, 0, st>>>(q, ld_q, tx, ld_tx, N, sums);        \
    else k_gmi<NL_, 1, B_><<<grid, EV_NT, 0, st>>>(q, ld_q, tx, ld_tx, N, sums);
#define EV_LEV(B_)                                                                          \
    if (n_lev == 2) { EV_CASE(2, B_) } else if (n_lev == 4) { EV_CASE(4, B_) } else { EV_CASE(8, B_) }
    if (bits) { EV_LEV(true) } else { EV_LEV(false) }
#undef EV_LEV
#undef EV_CASE
    ktime_end(VAEQ_K_EVAL, st);
    VAEQ_LAUNCH_CHECK("k_gmi");
    ktime_begin(VAEQ_K_EVAL, st);
    k_gmi_fin<<<1, 32, 0, st>>>(sums, grid, P, n_lev, N, gmi_out);
    ktime_end(VAEQ_K_EVAL, st);
    VAEQ_LAUNCH_CHECK("k_gmi_fin");
    return VAEQ_OK;
}

extern "C" int vaeq_gmi(const float *q, int64_t ld_q, const uint16_t *tx, int64_t ld_tx, const float *P, int32_t n_lev,
                        int32_t N, float *gmi_out, void *scratch, void *stream) {
    return rate(q, ld_q, tx, ld_tx, P, n_lev, N, gmi_out, scratch, stream, false);
}

extern "C" int vaeq_bmi(const float *q, int64_t ld_q, const uint16_t *tx, int64_t ld_tx, const float *P, int32_t n_lev,
                        int32_t N, float *bmi_out, void *scratch, void *stream) {
    return rate(q, ld_q, tx, ld_tx, P, n_lev, N, bmi_out, scratch, stream, true);
}

extern "C" int vaeq_bit_llr_runs(const float *q, int64_t ld_q, int64_t rs_q, int32_t n_lev, int32_t N, int32_t n_runs, float *llr,
                                 int64_t ld_llr, int64_t rs_llr, void *stream) {
    VAEQ_CHECK_ARG(q && llr, "NULL pointer");
    VAEQ_CHECK_ARG(n_lev == 2 || n_lev == 4 || n_lev == 8, "n_lev=%d must be 2, 4 or 8", n_lev);
    VAEQ_CHECK_ARG(N > 0, "N=%d must be positive", N);
    VAEQ_CHECK_ARG(n_runs > 0 && n_runs <= 65535, "n_runs=%d must be in 1..65535", n_runs);
    const int m = n_lev == 2 ? 1 : n_lev == 4 ? 2 : 3;
    VAEQ_CHECK_ARG(ld_llr >= N && (n_runs == 1 || rs_llr >= 4 * m * ld_llr), "llr strides (ld_llr=%lld, rs_llr=%lld) overlap rows of N=%d",
                   (long long)ld_llr, (long long)rs_llr, N);
    cudaStream_t st = (cudaStream_t)stream;
    const bool vec = (N % 4 == 0) && (ld_q % 4 == 0) && (rs_q % 4 == 0) && (ld_llr % 4 == 0) && (rs_llr % 4 == 0) &&
                     ((reinterpret_cast<uintptr_t>(q) | reinterpret_cast<uintptr_t>(llr)) % 16 == 0);
    const int V = vec ? 4 : 1;
    const dim3 grid(max(1, min((N / V + EV_NT - 1) / EV_NT, max(1, sm_count() * 8 / n_runs))), n_runs);
    ktime_begin(VAEQ_K_EVAL, st);
#define EV_CASE(NL_)                                                                                              \
    if (vec) k_bit_llr<NL_, 4><<<grid, EV_NT, 0, st>>>(q, ld_q, rs_q, N, llr, ld_llr, rs_llr);                    \
    else k_bit_llr<NL_, 1><<<grid, EV_NT, 0, st>>>(q, ld_q, rs_q, N, llr, ld_llr, rs_llr);
    if (n_lev == 2) { EV_CASE(2) } else if (n_lev == 4) { EV_CASE(4) } else { EV_CASE(8) }
#undef EV_CASE
    ktime_end(VAEQ_K_EVAL, st);
    VAEQ_LAUNCH_CHECK("k_bit_llr");
    return VAEQ_OK;
}
