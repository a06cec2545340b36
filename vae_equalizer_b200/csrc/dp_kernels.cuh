// Kernel parameter block and workspace constants of the DP VAE step.
#pragma once
#include "common.cuh"

namespace vaeq {

constexpr int DP_NT = 256;        // threads per CTA
constexpr int DP_TILE = 512;      // owned symbols per tile (generic kernels)
constexpr int DP_GRID_CAP = 1184; // upper bound of any persistent grid (8 CTAs x 148 SMs)

// float offsets inside the `scal` scratch block
constexpr int DP_C_OFF = 0;       // C_chi                     (2)
constexpr int DP_KAPPA_OFF = 2;   // (L-Mh)/C_chi              (2)
constexpr int DP_LOSS_OFF = 4;    // loss                      (1)
constexpr int DP_VAREST_OFF = 5;  // C/(L-Mh)                  (2)
constexpr int DP_S_OFF = 8;       // S_nu(j)                   (2*M)

constexpr int DP_MODE_FWD = 0, DP_MODE_FWDBWD = 1, DP_MODE_TRAIN = 2;

struct DpK {
    const float *rx;
    int64_t ld_rx;
    int B, L, M, mh, H;           // H = ceil(mh/2): halo in symbols of the channel convolution
    const float *amp, *P, *var;
    float nu_sc;
    float *W, *h, *adam;
    float *q;
    int64_t ld_q;
    float *out;
    int64_t ld_out;
    float *qk;
    int64_t ld_qk;
    float *outk;
    int64_t ld_outk;
    int keep_lo, keep_n;
    int64_t keep_base;            // destination column of symbol keep_lo
    int keep_vec;                 // fast path: keep_lo, keep_base, the keep strides and pointers allow float4 stores of four kept symbols
    double *part_fwd;             // [grid][8]: C0, C1, entropy, sum Var pol0, sum Var pol1
    float *edge_vs;               // [2][2*mh]: Var_I+Var_Q of the first mh and last mh symbols
    float *scal;
    float4 *ebuf4;                // [L]: residual D - rx per sample (chi0 re, chi0 im, chi1 re, chi1 im)
    float4 *m1buf4;               // [B]: E_q[x] per symbol (p0 I, p0 Q, p1 I, p1 Q)
    // fast path (dp_fast.cu) views of the same scratch as SoA rows of B floats
    float *erows;                 // 8 rows: [phase][chi][re/im]
    float *m1rows;                // 4 rows: (p0 I, p0 Q, p1 I, p1 Q)
    float *gyrows;                // 4 rows: dL/dout
    float *srows;                 // 12 rows: [S1 | T2 | S3][component]: dL/dout = gE*S1 + gV*T2 + w*S3 (see dp_fast.cu)
    int need_bwd;                 // forward kernel also emits srows (skipped in forward-only mode)
    int from_q;                   // generic kernels: q is an INPUT (operator-level loss on an arbitrary q), gq receives dL/dq
    float *gq;
    int64_t ld_gq;
    float *gpart;                 // [grid][16*M]
    float *gfinal;                // [16*M]: gW then gh
    float *loss_out, *var_est_out;
    int64_t var_est_stride;
    float *gW_out, *gh_out;
    int T, ntiles;
    // batch-split across GPUs (SURVEY.md §8e): this rank accumulates sums / gradients over symbols [sym_lo, sym_hi)
    // only, and its forward pass also produces the scratch rows for [clo, chi) = that range widened by DP_SPLIT_EXT
    // symbols, so that the backward halo needs no exchange.  Single GPU: 0, B, 0, B.
    int sym_lo, sym_hi, clo, chi;
    // dynamic tile scheduling of the fast kernels: tile_ctr[k] is the atomic tile counter of kernel k (zeroed per step)
    int *tile_ctr;
    int dyn;
};
constexpr int DP_SPLIT_EXT = 16;

// dp_step.cu
int dp_launch_fin(const DpK &p, int nparts, cudaStream_t st);
// dp_fast.cu: returns 1 if the register-blocked path ran (then *rc is its status, *grid_bwd_out the number of
// gradient partials), 0 if the problem does not qualify (alignment, M_est, size) and the generic kernels must run
int dp_try_fast(const DpK &p, int n_lev, int mode, cudaStream_t st, int *grid_bwd_out, int *rc);
// dp_taps_tc.cu: dW and dh on tcgen05 (after k_dp_bwd1_fast); returns 0 if M_est does not qualify
int dp_taps_tc_launch(const DpK &p, cudaStream_t st, int *nparts, int *rc);
// dp_fwd_tc.cu: the fast path's forward kernel with the FIR and the channel convolution on tcgen05; returns 0 if (n_lev, M_est) is not built
int dp_fwd_tc_launch(const DpK &p, int n_lev, cudaStream_t st, int *nparts, int *rc);
constexpr int DP_MODE_SPLIT_FWD = 3, DP_MODE_SPLIT_BWD = 4;   // forward kernel only / backward kernels only (no fin, no adam)

// batched independent runs of the frame kernels (vaeq_dp_train_frame_runs): blockIdx.x = run
struct DpRunsK {
    int64_t rs_rx, rs_amp, rs_P, rs_var, rs_W, rs_h, rs_adam, rs_q, rs_out, rs_qk, rs_outk;   // elements between runs
    int64_t ws_stride;                      // bytes between the workspaces of consecutive runs
    const float *nu_sc, *lr_w, *lr_h;       // optional per-run values (device), else the scalars
    float *loss_steps, *var_steps;          // (n_runs, n_steps), (n_runs, 2, n_steps); may be NULL
    float *loss_last, *var_last, *gW_last, *gh_last;   // (n_runs,1) (n_runs,2) (n_runs,8M) (n_runs,8M): the desc's loss/var_est/gW/gh
};


// dp_small.cu: persistent frame kernel for batch_len <= DP_SMALL_MAX_B (state and intermediates in shared memory)
constexpr int DP_SMALL_MAX_B = 1000;   // ~200 KB of shared memory at M_est = 25; the fast path starts at 992
size_t dp_small_smem(int B, int M);
int dp_small_launch(const DpK &p, const DpRunsK &rs, int n_lev, int n_runs, int n_steps, int stride_sym, int keep_lo_in_dst,
                    float lr_w, float lr_h, int amsgrad, cudaStream_t st);

}  // namespace vaeq
