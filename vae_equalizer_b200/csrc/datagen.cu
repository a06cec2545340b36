// Synthetic dual-polarisation test signal on the device, batched over R independent runs (sweep cells):
// the element-wise stages of generate_data_shaping / simulate_channel / simulate_dispersion
// (optical_DP_channel/shared_funcs.py:38-90) as four fused kernels.  The two DFTs of the dispersion step stay with cuFFT
// (torch.fft; the frame length 2N+2 is dictated by the reference's circular model).  The reference draws from unseeded numpy
// generators, so parity is statistical; here every random number is a Philox4x32-10 output keyed by (seed, run, row, position),
// so a run's data does not depend on what else is in the batch.
//
//   vaeq_gen_levels  sf:75-76   amplitude levels drawn from the run's pmf P (inverse CDF), float rows + the float16 tx slice (sf:89)
//   vaeq_gen_pulse   sf:77-80   zero insertion (sps = 2) + 'valid' convolution with the RRC pulse = two polyphase FIRs on the symbol grid
//   vaeq_gen_jones   sf:41-53   Y = R^T diag(e_pmd, 1/e_pmd) R X * e_cd per frequency bin, R from the run's rotation angle
//   vaeq_gen_noise   sf:83-88   + sigma_n (N(0,1) + j N(0,1)), cut to sps*N samples, split into the (R,2,2,L) float32 layout
//
// vaeq_gen_awgn: the single-polarisation signal of the AWGN module (AWGN_channel/func_VAELE_MQAM_shaping.py generate_data :39-61) for
// R runs x F frames with the same kernels: levels (two rows per frame), one complex 'valid' FIR with rrcfir (*) h_channel (two 'valid'
// convolutions in a row are one with the full convolution of the filters), then sigma_n from the frame's realised power and the noise.
// Draws are keyed by (the run's own seed, frame index, row, position), so a run's frames do not depend on the batch.
#include <curand_kernel.h>
#include "common.cuh"

namespace vaeq {

constexpr int DG_NT = 256;
constexpr int DG_MAXPULSE = 128;

// grid (ceil(n_conv / (4 DG_NT)), nrows, R * frames): a thread draws 4 consecutive levels of one row from one Philox output.
// seeds == NULL: one seed for the batch, draws keyed by (frame z = blockIdx.z, row, position), P row z.  Otherwise frame z is frame
// frame0 + z % frames of run z / frames, keyed by (seeds[run], frame, row, position), P row run.
__global__ void __launch_bounds__(DG_NT) k_gen_levels(const float *amps, const float *P, int n_lev, int n_conv, int N, int tx_off,
                                                      unsigned long long seed, const unsigned long long *seeds, int nrows, int frames,
                                                      int frame0, float *lev, uint16_t *tx) {
    __shared__ float cdf[VAEQ_MAX_LEVELS], a_s[VAEQ_MAX_LEVELS];
    const int row = blockIdx.y, r = blockIdx.z, run = r / frames;
    if (threadIdx.x == 0) {
        float tot = 0.f, acc = 0.f;
        for (int l = 0; l < n_lev; ++l) tot += P[(int64_t)run * n_lev + l];
        for (int l = 0; l < n_lev; ++l) {
            acc += P[(int64_t)run * n_lev + l];
            cdf[l] = acc / tot;
            a_s[l] = amps[l];
        }
    }
    __syncthreads();
    const int g = blockIdx.x * DG_NT + threadIdx.x, groups = (n_conv + 3) >> 2;
    if (g >= groups) return;
    curandStatePhilox4_32_10_t st;
    const unsigned long long key = seeds ? (unsigned long long)(frame0 + r - run * frames) : (unsigned long long)r;
    curand_init(seeds ? seeds[run] : seed, (key * nrows + row) * (unsigned long long)groups + g, 0, &st);
    const float4 u4 = curand_uniform4(&st);                                  // (0, 1]
    const float u[4] = {u4.x, u4.y, u4.z, u4.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int j = 4 * g + k;
        if (j >= n_conv) break;
        int idx = 0;
        for (int l = 0; l < n_lev - 1; ++l) idx += (u[k] > cdf[l]);
        const float a = a_s[idx];
        lev[((int64_t)r * nrows + row) * n_conv + j] = a;
        const int t = j - tx_off;                                            // data[:, T+M-1 : N+T+M-1]  (sf:89)
        if (t >= 0 && t < N) tx[((int64_t)r * nrows + row) * N + t] = __half_as_ushort(__float2half_rn(a));
    }
}

// grid (ceil(n_conv - K/2, DG_NT), nrows / 2 pols, R): thread u produces the even and the odd output sample 2u, 2u+1 (complex) of one pol:
//   shaped[2u]   = sum_t h[K-1-2t] sym[u+t],   shaped[2u+1] = sum_t h[K-2-2t] sym[u+1+t],   t = 0 .. K/2-1
// which is np.convolve(zero-stuffed symbols, h, 'valid') for sps = 2 and an even pulse length K (sf:57-61, 77-80).
// CPLX: h holds K complex taps (re, im interleaved), the composite pulse * channel filter of the AWGN module (:52-53).
template <bool CPLX>
__global__ void __launch_bounds__(DG_NT) k_gen_pulse(const float *lev, const float *h, int K, int n_conv, int nrows, float2 *shaped) {
    __shared__ float2 we[DG_MAXPULSE / 2], wo[DG_MAXPULSE / 2];
    const int half = K >> 1, p = blockIdx.y, r = blockIdx.z, nu = n_conv - half;
    for (int t = threadIdx.x; t < half; t += DG_NT) {
        we[t] = CPLX ? make_float2(h[2 * (K - 1 - 2 * t)], h[2 * (K - 1 - 2 * t) + 1]) : make_float2(h[K - 1 - 2 * t], 0.f);
        wo[t] = CPLX ? make_float2(h[2 * (K - 2 - 2 * t)], h[2 * (K - 2 - 2 * t) + 1]) : make_float2(h[K - 2 - 2 * t], 0.f);
    }
    __syncthreads();
    const int u = blockIdx.x * DG_NT + threadIdx.x;
    if (u >= nu) return;
    const float *re = lev + ((int64_t)r * nrows + 2 * p) * n_conv + u, *im = re + n_conv;
    float er = 0.f, ei = 0.f, orr = 0.f, oi = 0.f;
    float xr = re[0], xi = im[0];
    for (int t = 0; t < half; ++t) {
        const float nr = re[t + 1], ni = im[t + 1];                          // u + half <= n_conv - 1
        const float2 a = we[t], b = wo[t];
        er = fmaf(a.x, xr, er);
        ei = fmaf(a.x, xi, ei);
        orr = fmaf(b.x, nr, orr);
        oi = fmaf(b.x, ni, oi);
        if (CPLX) {
            er = fmaf(-a.y, xi, er);
            ei = fmaf(a.y, xr, ei);
            orr = fmaf(-b.y, ni, orr);
            oi = fmaf(b.y, nr, oi);
        }
        xr = nr;
        xi = ni;
    }
    float4 *dst = reinterpret_cast<float4 *>(shaped + ((int64_t)r * (nrows / 2) + p) * (2 * (int64_t)nu) + 2 * u);
    *dst = make_float4(er, ei, orr, oi);
}

__device__ __forceinline__ float2 cmul(float2 a, float2 b) { return make_float2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x); }
__device__ __forceinline__ float2 cadd(float2 a, float2 b) { return make_float2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ float2 cscale(float2 a, float s) { return make_float2(a.x * s, a.y * s); }

// grid (ceil(n / DG_NT), R): H = R^T diag(p, 1/p) R with R = [[c e0, s e0], [-s e1, c e1]], R^T = [[c e0, -s e0], [s e1, c e1]]  (sf:46-50)
//   H00 = c^2 e0^2 p + s^2 e0 e1 / p     H01 = c s (e0^2 p - e0 e1 / p)
//   H10 = c s (e0 e1 p - e1^2 / p)       H11 = s^2 e0 e1 p + c^2 e1^2 / p
// Pcd = p e_cd and Picd = e_cd / p are tabulated per frame geometry, so Y = H X e_cd (sf:52-53) is 4 complex products per bin and pol.
__global__ void __launch_bounds__(DG_NT) k_gen_jones(float2 *X, const float2 *Pcd, const float2 *Picd, const float *theta, float2 e00,
                                                     float2 e01, float2 e11, int n) {
    const int r = blockIdx.y, b = blockIdx.x * DG_NT + threadIdx.x;
    if (b >= n) return;
    float s, c;
    sincosf(theta[r], &s, &c);
    float2 *x0p = X + ((int64_t)r * 2) * n + b, *x1p = x0p + n;
    const float2 x0 = *x0p, x1 = *x1p, P = Pcd[b], Q = Picd[b];
    const float2 a = cmul(P, e00), d = cmul(Q, e01), f = cmul(P, e01), g = cmul(Q, e11);   // e00 = e0^2, e01 = e0 e1, e11 = e1^2
    const float2 h00 = cadd(cscale(a, c * c), cscale(d, s * s)), h01 = cscale(make_float2(a.x - d.x, a.y - d.y), c * s);
    const float2 h10 = cscale(make_float2(f.x - g.x, f.y - g.y), c * s), h11 = cadd(cscale(f, s * s), cscale(g, c * c));
    *x0p = cadd(cmul(h00, x0), cmul(h01, x1));
    *x1p = cadd(cmul(h10, x0), cmul(h11, x1));
}

// grid (ceil(L / (2 DG_NT)), 2 pols, R): a thread adds complex noise to 2 consecutive samples (4 normals = one Philox output)
__global__ void __launch_bounds__(DG_NT) k_gen_noise(const float2 *sig, const float *sigma, unsigned long long seed, int n, int L, float *rx) {
    const int p = blockIdx.y, r = blockIdx.z, g = blockIdx.x * DG_NT + threadIdx.x, m = 2 * g;
    if (m >= L) return;
    curandStatePhilox4_32_10_t st;
    curand_init(seed, ((unsigned long long)(r * 2 + p)) * (unsigned long long)((L + 1) >> 1) + g, 0, &st);
    const float4 z = curand_normal4(&st);
    const float sg = sigma[r];
    const float2 *s = sig + ((int64_t)r * 2 + p) * n + m;
    float *ri = rx + (((int64_t)r * 2 + p) * 2) * L + m, *rq = ri + L;
    const float2 a = s[0];
    ri[0] = fmaf(sg, z.x, a.x);
    rq[0] = fmaf(sg, z.y, a.y);
    if (m + 1 < L) {
        const float2 b = s[1];
        ri[1] = fmaf(sg, z.z, b.x);
        rq[1] = fmaf(sg, z.w, b.y);
    }
}

// grid (R * frames): one CTA per single-polarisation frame.  sigma_n = sqrt(sps mean|sig|^2 / 2 / 10^(SNR/10)) over the whole 'valid'
// signal of n samples (:55), then rx[z] = (Re, Im)(sig[:L] + sigma_n (N(0,1) + j N(0,1))) (:56-57), 2 samples per Philox output
__global__ void __launch_bounds__(DG_NT) k_gen_awgn_noise(const float2 *sig, const float *snr, const unsigned long long *seeds, int frames,
                                                          int frame0, int n, int L, float *rx) {
    __shared__ double red[32];
    __shared__ float sg_sh;
    const int z = blockIdx.x, run = z / frames;
    const float2 *s = sig + (int64_t)z * n;
    double acc[1] = {0.0};
    for (int m = threadIdx.x; m < n; m += DG_NT) {
        const float2 a = s[m];
        acc[0] += (double)a.x * a.x + (double)a.y * a.y;
    }
    block_sum<1>(acc, red);
    if (threadIdx.x == 0) sg_sh = (float)sqrt(2.0 * (acc[0] / n) / 2.0 / pow(10.0, (double)snr[run] / 10.0));
    __syncthreads();
    const float sg = sg_sh;
    const int groups = (L + 1) >> 1;
    float *ri = rx + (int64_t)z * 2 * L, *rq = ri + L;
    for (int g = threadIdx.x; g < groups; g += DG_NT) {
        curandStatePhilox4_32_10_t st;
        curand_init(seeds[run] ^ 0x9E3779B97F4A7C15ull, (unsigned long long)(frame0 + z - run * frames) * groups + g, 0, &st);
        const float4 w = curand_normal4(&st);
        const int m = 2 * g;
        const float2 a = s[m];
        ri[m] = fmaf(sg, w.x, a.x);
        rq[m] = fmaf(sg, w.y, a.y);
        if (m + 1 < L) {
            const float2 b = s[m + 1];
            ri[m + 1] = fmaf(sg, w.z, b.x);
            rq[m + 1] = fmaf(sg, w.w, b.y);
        }
    }
}

}  // namespace vaeq

using namespace vaeq;

extern "C" int vaeq_gen_awgn(const float *amps, const float *P, int32_t n_lev, const float *taps, int32_t K, int32_t N, int32_t tx_off,
                             int32_t n_conv, const float *snr, const uint64_t *seeds, int32_t frame0, int32_t n_frames, int32_t n_runs,
                             float *lev, float *sig, float *rx, uint16_t *tx, void *stream) {
    VAEQ_CHECK_ARG(amps && P && taps && snr && seeds && lev && sig && rx && tx, "NULL pointer");
    VAEQ_CHECK_ARG(n_lev >= 2 && n_lev <= VAEQ_MAX_LEVELS && N > 0 && tx_off >= 0 && tx_off + N <= n_conv && frame0 >= 0 && n_frames > 0 &&
                   n_runs > 0 && (int64_t)n_runs * n_frames <= 65535, "bad sizes (n_lev=%d N=%d tx_off=%d n_conv=%d frames=%d runs=%d)",
                   n_lev, N, tx_off, n_conv, n_frames, n_runs);
    VAEQ_CHECK_ARG(K >= 2 && K % 2 == 0 && K <= DG_MAXPULSE && n_conv > K / 2, "filter length K=%d must be even and <= %d", K, DG_MAXPULSE);
    const int n = 2 * n_conv - K, L = 2 * N;
    VAEQ_CHECK_ARG(L <= n, "sps*N=%d exceeds the %d filtered samples", L, n);
    VAEQ_CHECK_ARG(reinterpret_cast<uintptr_t>(sig) % 16 == 0, "sig must be 16-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    const int Z = n_runs * n_frames, groups = (n_conv + 3) / 4, nu = n_conv - K / 2;
    const unsigned long long *sd = reinterpret_cast<const unsigned long long *>(seeds);
    ktime_begin(VAEQ_K_OTHER, st);
    k_gen_levels<<<dim3((groups + DG_NT - 1) / DG_NT, 2, Z), DG_NT, 0, st>>>(amps, P, n_lev, n_conv, N, tx_off, 0, sd, 2, n_frames, frame0, lev, tx);
    ktime_end(VAEQ_K_OTHER, st);
    VAEQ_LAUNCH_CHECK("k_gen_levels");
    ktime_begin(VAEQ_K_OTHER, st);
    k_gen_pulse<true><<<dim3((nu + DG_NT - 1) / DG_NT, 1, Z), DG_NT, 0, st>>>(lev, taps, K, n_conv, 2, reinterpret_cast<float2 *>(sig));
    ktime_end(VAEQ_K_OTHER, st);
    VAEQ_LAUNCH_CHECK("k_gen_pulse");
    ktime_begin(VAEQ_K_OTHER, st);
    k_gen_awgn_noise<<<Z, DG_NT, 0, st>>>(reinterpret_cast<const float2 *>(sig), snr, sd, n_frames, frame0, n, L, rx);
    ktime_end(VAEQ_K_OTHER, st);
    VAEQ_LAUNCH_CHECK("k_gen_awgn_noise");
    return VAEQ_OK;
}

extern "C" int vaeq_gen_levels(const float *amps, const float *P, int32_t n_lev, int32_t n_conv, int32_t N, int32_t tx_off, uint64_t seed,
                               float *lev, uint16_t *tx, int32_t n_runs, void *stream) {
    VAEQ_CHECK_ARG(amps && P && lev && tx, "NULL pointer");
    VAEQ_CHECK_ARG(n_lev >= 2 && n_lev <= VAEQ_MAX_LEVELS && n_conv > 0 && N > 0 && tx_off >= 0 && tx_off + N <= n_conv && n_runs > 0 && n_runs <= 65535,
                   "bad sizes (n_lev=%d n_conv=%d N=%d tx_off=%d n_runs=%d)", n_lev, n_conv, N, tx_off, n_runs);
    cudaStream_t st = (cudaStream_t)stream;
    const int groups = (n_conv + 3) / 4;
    ktime_begin(VAEQ_K_OTHER, st);
    k_gen_levels<<<dim3((groups + DG_NT - 1) / DG_NT, 4, n_runs), DG_NT, 0, st>>>(amps, P, n_lev, n_conv, N, tx_off, seed, nullptr, 4, 1, 0, lev,
                                                                                  tx);
    ktime_end(VAEQ_K_OTHER, st);
    VAEQ_LAUNCH_CHECK("k_gen_levels");
    return VAEQ_OK;
}

extern "C" int vaeq_gen_pulse(const float *lev, const float *h, int32_t n_pulse, int32_t n_conv, float *shaped, int32_t n_runs, void *stream) {
    VAEQ_CHECK_ARG(lev && h && shaped, "NULL pointer");
    VAEQ_CHECK_ARG(n_pulse >= 2 && n_pulse % 2 == 0 && n_pulse <= DG_MAXPULSE && n_conv > n_pulse / 2 && n_runs > 0 && n_runs <= 65535,
                   "bad sizes (n_pulse=%d must be even and <= %d, n_conv=%d, n_runs=%d)", n_pulse, DG_MAXPULSE, n_conv, n_runs);
    VAEQ_CHECK_ARG(reinterpret_cast<uintptr_t>(shaped) % 16 == 0, "shaped must be 16-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    const int nu = n_conv - n_pulse / 2;
    ktime_begin(VAEQ_K_OTHER, st);
    k_gen_pulse<false><<<dim3((nu + DG_NT - 1) / DG_NT, 2, n_runs), DG_NT, 0, st>>>(lev, h, n_pulse, n_conv, 4, reinterpret_cast<float2 *>(shaped));
    ktime_end(VAEQ_K_OTHER, st);
    VAEQ_LAUNCH_CHECK("k_gen_pulse");
    return VAEQ_OK;
}

extern "C" int vaeq_gen_jones(float *X, const float *Pcd, const float *Picd, const float *theta, float phi0, float phi1, int32_t n,
                              int32_t n_runs, void *stream) {
    VAEQ_CHECK_ARG(X && Pcd && Picd && theta && n > 0 && n_runs > 0 && n_runs <= 65535, "bad jones arguments");
    cudaStream_t st = (cudaStream_t)stream;
    // e0 = exp(-j phi0), e1 = exp(-j phi1)  (sf:44)
    const float2 e00 = make_float2(cosf(-2.f * phi0), sinf(-2.f * phi0)), e01 = make_float2(cosf(-(phi0 + phi1)), sinf(-(phi0 + phi1))),
                 e11 = make_float2(cosf(-2.f * phi1), sinf(-2.f * phi1));
    ktime_begin(VAEQ_K_OTHER, st);
    k_gen_jones<<<dim3((n + DG_NT - 1) / DG_NT, n_runs), DG_NT, 0, st>>>(reinterpret_cast<float2 *>(X), reinterpret_cast<const float2 *>(Pcd),
                                                                         reinterpret_cast<const float2 *>(Picd), theta, e00, e01, e11, n);
    ktime_end(VAEQ_K_OTHER, st);
    VAEQ_LAUNCH_CHECK("k_gen_jones");
    return VAEQ_OK;
}

extern "C" int vaeq_gen_noise(const float *sig, const float *sigma, uint64_t seed, int32_t n, int32_t L, float *rx, int32_t n_runs, void *stream) {
    VAEQ_CHECK_ARG(sig && sigma && rx && n > 0 && L > 0 && L <= n && n_runs > 0 && n_runs <= 65535, "bad noise arguments (L=%d must be <= n=%d)", L, n);
    cudaStream_t st = (cudaStream_t)stream;
    const int groups = (L + 1) / 2;
    ktime_begin(VAEQ_K_OTHER, st);
    k_gen_noise<<<dim3((groups + DG_NT - 1) / DG_NT, 2, n_runs), DG_NT, 0, st>>>(reinterpret_cast<const float2 *>(sig), sigma, seed, n, L, rx);
    ktime_end(VAEQ_K_OTHER, st);
    VAEQ_LAUNCH_CHECK("k_gen_noise");
    return VAEQ_OK;
}
