/*
 * vaeq.h -- C ABI of libvaeq.so: the B200 (sm_100a) implementation of the VAE blind-equalizer
 * training hot path of kit-cel/vae-equalizer.
 *
 * The reference is pure Python/PyTorch and has no FFI layer (SURVEY.md §8b): its "plugin API" is
 * the Python module surface  optical_DP_channel/shared_funcs.py  that the Eval_run_*.py drivers
 * reach through  func_*_MQAM_shaping.processing().  The entry points below are what a binding for
 * that surface needs; each one cites the reference function (file:line, relative to the reference
 * root, sf = optical_DP_channel/shared_funcs.py) it replaces.  INTEGRATION.md shows the ctypes stub.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer into caller-owned memory unless the name ends in _host;
 *   - tensors are contiguous float32 with time innermost, exactly the reference layouts:
 *       rx (2,2,L) [pol][I/Q][sample], q (2,2n,B) [pol][I rows 0..n-1 | Q rows n..2n-1][symbol],
 *       out (2,2,B), W (2,4,M) [out pol][Re<-p0,Re<-p1,Im<-p0,Im<-p1][tap], h (2,2,2,M) [rx pol][tx pol][Re/Im][tap];
 *     "ld_*" arguments are the distance in elements between consecutive rows, so a window of a
 *     longer frame can be passed without a copy (func_VAELE_DP_MQAM_shaping.py:58 copies instead);
 *   - `stream` is a cudaStream_t passed as void*; nothing synchronises the host;
 *   - return value 0 = ok, otherwise a negative VAEQ_E* code or a positive cudaError_t;
 *     vaeq_last_error() gives the text.  No entry point allocates device memory: scratch comes from
 *     the caller-provided workspace (size from vaeq_dp_workspace_bytes).
 *   - sps == 2 and odd M_est only (what every reference driver uses; even M_est breaks the
 *     reference itself, sf:494 yields B+1 outputs).
 */
#ifndef VAEQ_H_
#define VAEQ_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VAEQ_ABI_VERSION 1

#define VAEQ_OK 0
#define VAEQ_EINVAL (-1)     /* bad argument (shape, sps, even M, n_lev not in {2,4,8}) */
#define VAEQ_EWORKSPACE (-2) /* workspace too small */
#define VAEQ_ENODEV (-3)     /* no sm_100 device / kernel image */

#define VAEQ_MAX_TAPS 63
#define VAEQ_MAX_LEVELS 8

int vaeq_abi_version(void);
const char *vaeq_last_error(void);
/* number of SMs of the current device (persistent grids are sized from it) */
int vaeq_sm_count(void);

/* Measurement hooks (no reference counterpart): kernels are grouped into kinds; every launch is counted,
 * and with timing enabled each launch is bracketed by a CUDA event pair on its own stream.
 * vaeq_kernel_timing(1) resets and enables, (0) disables; vaeq_kernel_timing_read synchronises the recorded
 * events and returns summed milliseconds and launch counts per kind (arrays of VAEQ_NKINDS). */
#define VAEQ_K_DP_FWD 0
#define VAEQ_K_DP_FIN 1
#define VAEQ_K_DP_BWD 2
#define VAEQ_K_DP_ADAM 3
#define VAEQ_K_EVAL 4
#define VAEQ_K_CMA 5
#define VAEQ_K_AWGN 6
#define VAEQ_K_OTHER 7
#define VAEQ_K_DP_BWD2 8
#define VAEQ_K_DP_BWD3 9
#define VAEQ_K_DP_FRAME 10 /* persistent frame kernel: all steps of a frame (and all batched runs) in one launch */
#define VAEQ_NKINDS 11
int vaeq_kernel_timing(int32_t enable);
int vaeq_kernel_timing_read(float *ms_sum, int32_t *count);
int64_t vaeq_launch_count(int32_t kind); /* kind < 0: all kinds */

/* ------------------------------------------------------------------------------------------------
 * DP VAE-LE / VAE-flex training step
 *   replaces  twoXtwoFIR.forward (sf:500-527) + loss_function_shaping (sf:92-137) + loss.backward()
 *   + optim.Adam.step() with two parameter groups (func_VAELE_DP_MQAM_shaping.py:26-31,57-66).
 * ---------------------------------------------------------------------------------------------- */
typedef struct vaeq_dp_desc {
    /* problem */
    int32_t B;       /* symbols in this minibatch (batch_len)                                   */
    int32_t sps;     /* samples per symbol, must be 2                                            */
    int32_t M;       /* M_est, odd, <= VAEQ_MAX_TAPS                                             */
    int32_t n_lev;   /* ASK levels per component: 2, 4 or 8 (4/16/64-QAM)                        */
    float nu_sc;     /* PCS demapper term (sf:570)                                               */
    int32_t flags;   /* VAEQ_F_* below                                                           */
    /* inputs */
    const float *rx; /* (2,2,L=B*sps) window start                                               */
    int64_t ld_rx;   /* row stride of rx in elements                                             */
    const float *amp; /* (n_lev) amplitude levels, ascending (sf:568)                            */
    const float *P;   /* (n_lev) PCS pmf (sf:572)                                                */
    const float *var; /* (2) demapper noise variance per pol (sf:581)                            */
    /* trainable state (updated in place by the *_train_* entry points) */
    float *W;        /* (2,4,M) equalizer taps = twoXtwoFIR.conv_w.weight                        */
    float *h;        /* (2,2,2,M) channel estimate h_est                                         */
    float *adam;     /* Adam state, vaeq_adam_state_floats(M) floats, zero-initialised by caller */
    /* outputs */
    float *q;        /* (2,2n,B) posteriors of the whole minibatch (needed by the backward pass) */
    int64_t ld_q;
    float *out;      /* (2,2,B) equalizer output                                                 */
    int64_t ld_out;
    float *q_keep;   /* optional second copy restricted to symbols [keep_lo, keep_lo+keep_n):    */
    int64_t ld_q_keep; /* what VAE-flex stores (func_VAEflex_DP_MQAM_shaping.py:64-65); may be NULL */
    float *out_keep;
    int64_t ld_out_keep;
    int32_t keep_lo, keep_n;
    float *loss;     /* (1)  ELBO loss of this minibatch (sf:136)                                */
    float *var_est;  /* (2)  C/(L-Mh), the estimated noise variance (sf:137)                     */
    float *gW;       /* optional (2,4,M) gradient of the loss w.r.t. W, may be NULL              */
    float *gh;       /* optional (2,2,2,M) gradient w.r.t. h, may be NULL                        */
    /* scratch */
    void *workspace;
    size_t workspace_bytes;
} vaeq_dp_desc;

#define VAEQ_F_AMSGRAD 1 /* Adam amsgrad=True (AWGN driver, func_VAELE_MQAM_shaping.py:283) */

size_t vaeq_dp_workspace_bytes(int32_t B, int32_t M, int32_t n_lev);
/* floats of Adam state for one run: exp_avg, exp_avg_sq, max_exp_avg_sq for W and h, + step counter */
size_t vaeq_adam_state_floats(int32_t M);

/* Testing hook: != 0 routes every vaeq_dp_* call through the generic-M kernels (dp_step.cu) even when the
 * register-blocked fast path (dp_fast.cu: B % 4 == 0, 16-byte aligned rows, M_est in {5,9,13,25}, B >= 992) applies. */
int vaeq_dp_force_generic(int32_t on);

/* Tile scheduling of the fast path: != 0 (default) lets every persistent CTA pull its next tile from an atomic counter
 * (no SM idles while its slower CTA finishes; ~10 % faster), at the price of run-to-run differences in the LAST BITS of
 * loss / gradients (summation order of the per-CTA partials); 0 = static striding, bitwise reproducible. */
int vaeq_dp_dynamic_tiles(int32_t on);

/* Tap gradients of the fast path: 1 (default) computes both correlations (dW, dh) on tcgen05 tensor cores as block outer products
 * with a 3 x tf32 split and fp32 accumulation in TMEM (dp_taps_tc.cu: 116 us instead of 168 us per 2^22 symbols, agreement with the
 * CUDA-core kernels 3e-7 ... 6e-6 relative, bitwise reproducible); 0 = the two CUDA-core correlation kernels of dp_fast.cu.  This
 * departs from the hot path's stated "no tensor cores" design and was adopted on measurement (DESIGN.md 4a, profiles/r02_tc_taps.txt).
 * Any other value returns VAEQ_EINVAL and leaves the setting unchanged. */
int vaeq_dp_tc_taps(int32_t on);

/* Forward kernel of the fast path: != 0 (default since r02c) runs the 2x2 butterfly FIR and the channel convolution D = h * E_q on
 * tcgen05 tensor cores (dp_fwd_tc.cu: the sample / E_q windows are Hankel operands read straight from the staged rows, tf32 hi + lo
 * split of both operands, fp32 accumulation in TMEM; the tensor core truncates its accumulator, so the MMAs are issued by growing
 * magnitude -- lo parts, outer taps, the K steps with the centre taps last -- and the centre tap itself stays in fp32 on the CUDA
 * cores); 0 = the CUDA-core kernel k_dp_fwd_fast, which also serves the (n_lev, M_est) the tensor-core kernel is not built for.
 * Same outputs within the step tolerances; at batch_len 2^22: 244 us against 257 us, out against float64 max 4.4e-7 / rms 5.3e-8
 * against 6.7e-7 / 6.5e-8 (profiles/r02c_tc_forward.txt). */
int vaeq_dp_tc_forward(int32_t on);

/* forward only: q, out, loss, var_est  (net(minibatch) + loss_function_shaping, no grad) */
int vaeq_dp_forward(const vaeq_dp_desc *d, void *stream);
/* forward + backward: additionally gW, gh (must be non-NULL); parameters are NOT updated */
int vaeq_dp_forward_backward(const vaeq_dp_desc *d, void *stream);
/* loss_function_shaping (sf:92-137) as an operator on an ARBITRARY q: d->q (2,2n,B) is an INPUT here; outputs d->loss, d->var_est,
 * d->gh = dL/dh_est (optional) and gq (2,2n,B, row stride ld_gq) = dL/dq (optional).  d->W / out / var / adam are not used. */
int vaeq_dp_loss_from_q(const vaeq_dp_desc *d, float *gq, int64_t ld_gq, void *stream);

/* Backward of twoXtwoFIR.forward (sf:500-527) alone, for ARBITRARY upstream gradients: gq (2,2n,B) = dL/dq and / or gout (2,2,B) =
 * dL/dout (either may be NULL) -> gW (2,4,M) = dL/dconv_w.weight.  q / out are the forward's outputs (needed when gq != NULL).  What
 * autograd calls when a caller derives something else from q before differentiating; the fused step above does not use it. */
size_t vaeq_eq_backward_scratch_bytes(int32_t B, int32_t M);
int vaeq_eq_backward(const float *rx, int64_t ld_rx, const float *q, int64_t ld_q, const float *out, int64_t ld_out, const float *gq,
                     int64_t ld_gq, const float *gout, int64_t ld_gout, const float *amp, const float *var, int32_t n_lev, int32_t B,
                     int32_t M, float *gW, void *scratch, void *stream);

/* forward + backward + Adam on both groups: lr_w for W (group 0), lr_h for h (group 1);
 * betas (0.9,0.999), eps 1e-8, no weight decay (torch defaults used at func_VAELE_DP_MQAM_shaping.py:28) */
int vaeq_dp_train_step(const vaeq_dp_desc *d, float lr_w, float lr_h, void *stream);

/* A frame of sequential minibatches (func_VAELE_DP_MQAM_shaping.py:57-66 with stride_sym = B,
 * func_VAEflex_DP_MQAM_shaping.py:59-70 with stride_sym = flex_step): step m trains on symbols
 * [m*stride_sym, m*stride_sym + B) of the frame.  d->rx / d->q_keep / d->out_keep address the FRAME
 * (rx_frame (2,2,L_frame), out_train (2,2n,*), out_const (2,2,*)); the kept columns of step m land at
 * column m*stride_sym (+keep_lo when keep_lo_in_dst != 0) of q_keep/out_keep.  d->q / d->out are
 * per-minibatch scratch.  loss_steps (n_steps) and var_est_steps (2,n_steps) receive every step's
 * values (var_est[:,m] at func_VAELE_DP_MQAM_shaping.py:64). */
int vaeq_dp_train_frame(const vaeq_dp_desc *d, int32_t n_steps, int32_t stride_sym, int32_t keep_lo_in_dst,
                        float lr_w, float lr_h, float *loss_steps, float *var_est_steps, void *stream);

/* Reference-size minibatches (batch_len <= 1000, Eval_run_DP.py:38 uses 100): vaeq_dp_train_frame runs the whole frame in
 * ONE persistent launch: one CTA walks the sequential steps with taps, Adam state and all intermediates in shared memory
 * (dp_small.cu).  Testing hook vaeq_dp_persistent_frames(mode): 1 = that kernel (default); 0 = one set of launches per
 * step; 2 = the per-step kernels' own bodies inside one launch (bitwise identical to mode 0). */
int vaeq_dp_persistent_frames(int32_t mode);

/* The same frame for n_runs INDEPENDENT runs in one launch, one CTA per run -- the sweep cells of Eval_run_DP.py:68-95
 * (SNR x realisation x lr ...) that share batch_len, M_est and n_lev.  Every tensor of the desc addresses run 0; run r
 * is found rs_* ELEMENTS further (0 = shared by all runs).  d->loss (n_runs), d->var_est (n_runs,2), d->gW (n_runs,2,4,M),
 * d->gh (n_runs,2,2,2,M) get a leading run dimension; d->workspace holds vaeq_dp_runs_workspace_bytes(B,M,n_lev,n_runs) (the
 * default kernel keeps all scratch in shared memory: 256 bytes; testing mode 2 needs a full workspace per run);
 * loss_steps (n_runs,n_steps), var_est_steps (n_runs,2,n_steps).  nu_sc / lr_w / lr_h: optional per-run device arrays. */
size_t vaeq_dp_runs_workspace_bytes(int32_t B, int32_t M, int32_t n_lev, int32_t n_runs);
typedef struct vaeq_dp_runs {
    int32_t n_runs;
    int64_t rs_rx, rs_amp, rs_P, rs_var, rs_W, rs_h, rs_adam, rs_q, rs_out, rs_q_keep, rs_out_keep;
    const float *nu_sc;
    const float *lr_w, *lr_h;
} vaeq_dp_runs;
int vaeq_dp_train_frame_runs(const vaeq_dp_desc *d, const vaeq_dp_runs *runs, int32_t n_steps, int32_t stride_sym,
                             int32_t keep_lo_in_dst, float lr_w, float lr_h, float *loss_steps, float *var_est_steps,
                             void *stream);
/* The persistent frame kernel exists for 3 runs per SM (80 registers, the faster one per run) and for 4 (64 registers); by default the
 * library takes the fourth run per SM only when that saves a whole wave of CTAs (592 runs on 148 SMs).  Testing hook: 0 = automatic,
 * 3 / 4 = force; both give bitwise identical results. */
int vaeq_dp_frame_runs_per_sm(int32_t per_sm);

/* Batch-split of ONE long minibatch across GPUs (SURVEY.md §8e; the reference has no counterpart, it is what replaces
 * "one process, one device" for func_VAEflex_DP_MQAM_shaping.py at large batch_len).  Every rank holds the whole rx
 * window and the same W/h/Adam state and owns the symbols [sym_lo, sym_hi) (multiples of 4).  Per step:
 *   1. vaeq_dp_split_forward   -> stats_out (vaeq_dp_split_stats_doubles(M) doubles): partial C, entropy, Var sums
 *      host: all-reduce(SUM) stats over the ranks
 *   2. vaeq_dp_split_backward  (stats_in = reduced stats) -> loss, var_est (identical on every rank) and
 *      grads_out (16*M floats: gW then gh, this rank's share, without the rank-independent E-term of gh)
 *      host: all-reduce(SUM) grads
 *   3. vaeq_dp_split_update    (grads_in = reduced grads) -> adds the E-term, Adam on both groups (replicated).
 * q / out are written for the owned symbols (plus a 16-symbol margin each side). */
size_t vaeq_dp_split_stats_doubles(int32_t M);
int vaeq_dp_split_forward(const vaeq_dp_desc *d, int32_t sym_lo, int32_t sym_hi, double *stats_out, void *stream);
int vaeq_dp_split_backward(const vaeq_dp_desc *d, int32_t sym_lo, int32_t sym_hi, const double *stats_in, float *grads_out,
                           void *stream);
int vaeq_dp_split_update(const vaeq_dp_desc *d, const float *grads_in, float lr_w, float lr_h, void *stream);
/* q / out of the three calls above and of vaeq_dp_split_step_peer are touched in the columns [max(0, sym_lo - 16), min(B, sym_hi + 16))
 * only, so a rank may pass a buffer that holds just those columns, its base pointers shifted back by the first column; d->q_keep /
 * d->out_keep (if set) receive the kept columns [keep_lo, keep_lo + keep_n) that lie inside [sym_lo, sym_hi), at column u - keep_lo;
 * with them set, d->q = d->out = NULL is allowed: the window's q / out are then not written at all (the VAE-flex frame loop keeps the
 * middle flex_step symbols of every window and nothing else, func_VAEflex_DP_MQAM_shaping.py:64-67).
 *
 * The same step with BOTH reductions done by the library itself over NVLink peer memory instead of two host-issued all-reduces: every
 * rank allocates a slot of vaeq_peer_slot_bytes(M) bytes, zero-initialised, in memory all peers can address (CUDA IPC / VMM, e.g.
 * torch.distributed._symmetric_memory) and passes the `world` peer-mapped pointers in rank order (slot[rank] = its own) plus two
 * zero-initialised int32 counters in its own device memory.  One call = forward, exchange of the ELBO sums, loss / kappa, backward,
 * exchange of the 16 M gradient floats, replicated Adam: 6 launches (the exchanges are fused with the loss assembly and with Adam), no
 * host synchronisation, graph-capturable.  An exchange is a PUSH with the flag inside every word:
 * a rank stores its partial into its own compartment of EVERY peer's slot as aligned 8-byte words {payload32, epoch32}, then polls the
 * words of its own slot (local memory) until each carries the epoch of this exchange and adds the payloads in rank order -- bit-identical
 * on every rank, no fence, one NVLink store latency whatever the number of ranks.  All ranks must make the same sequence of calls; a peer
 * that does not show up within 20 s traps the kernel. */
#define VAEQ_MAX_PEERS 8
typedef struct vaeq_peer_comm {
    int32_t rank, world;
    void *slot[VAEQ_MAX_PEERS];
    int32_t *epoch;
} vaeq_peer_comm;
size_t vaeq_peer_slot_bytes(int32_t M);
int vaeq_dp_split_step_peer(const vaeq_dp_desc *d, int32_t sym_lo, int32_t sym_hi, const vaeq_peer_comm *comm, float lr_w, float lr_h,
                            void *stream);

/* generic Adam update on n floats (torch.optim.Adam single-tensor semantics); state = [m|v|vmax] (3n floats),
 * step_count is a device int32 incremented by the call when bump_step != 0 */
int vaeq_adam_update(float *param, const float *grad, float *state, int32_t n, float lr, int32_t amsgrad,
                     int32_t *step_count, int32_t bump_step, void *stream);

/* ------------------------------------------------------------------------------------------------
 * soft demapper alone: soft_dec (sf:529-542)
 * ---------------------------------------------------------------------------------------------- */
int vaeq_soft_dec(const float *out, int64_t ld_out, const float *var, const float *amp, float nu_sc,
                  int32_t n_lev, int32_t N, float *q, int64_t ld_q, void *stream);

/* soft_dec for n_runs independent runs in one launch (sweep engine): out (n_runs,2,2,N), q (n_runs,2,2*n_lev,N) contiguous,
 * var (n_runs,2), nu_sc (n_runs); per run the arithmetic of vaeq_soft_dec */
int vaeq_soft_dec_runs(const float *out, const float *var, const float *amp, const float *nu_sc, int32_t n_lev, int32_t N,
                       int32_t n_runs, float *q, void *stream);

/* ------------------------------------------------------------------------------------------------
 * evaluation: shift search and SER estimators (sf:188-338).  tx is the reference's float16
 * data_tensor (2,2,N) (sf:89), passed as uint16_t bit patterns.
 * ---------------------------------------------------------------------------------------------- */
/* find_shift (sf:290-314) when q != NULL (E = sum_l amp_l q_I[l]), find_shift_symb_full (sf:316-338)
 * when q == NULL (E = out[:,0,:]).  corr_out (2 comp,2 eq-pol,2 tx-pol,n_shift) |correlations|,
 * shift_out int16 (2) = n_shift/2 - argmax, r_out int32 (1) in {0,1}.  n_shift <= 64.
 * scratch: vaeq_find_shift_scratch_bytes(n_shift) (per-CTA partial correlations, summed in fixed order). */
size_t vaeq_find_shift_scratch_bytes(int32_t n_shift);
int vaeq_find_shift(const float *q, int64_t ld_q, const float *out, int64_t ld_out, const uint16_t *tx, int64_t ld_tx,
                    const float *amp, int32_t n_lev, int32_t N, int32_t n_shift, float *corr_out, int16_t *shift_out,
                    int32_t *r_out, void *scratch, void *stream);
/* SER_IQflip (sf:188-222): counts int32 (2 flip,2 pol,4 rot) of symbol errors, ser_out float (2) = min/N */
int vaeq_ser_iqflip(const float *q, int64_t ld_q, const uint16_t *tx, int64_t ld_tx, int32_t n_lev, int32_t N,
                    int32_t *counts_out, float *ser_out, void *stream);
/* SER_constell_shaping + dec_on_bound (sf:225-287): rescales rx IN PLACE (sf:242) like the reference.
 * scratch: VAEQ_EVAL_SCRATCH_BYTES (per-CTA partial sums of the two norms, added in a fixed order: no floating-point
 * atomics, so the scale factor and hence every count is bit-reproducible). */
#define VAEQ_EVAL_SCRATCH_BYTES 65536
int vaeq_ser_constell(float *rx, int64_t ld_rx, const uint16_t *tx, int64_t ld_tx, const float *amp, const float *var,
                      float nu_sc, int32_t n_lev, int32_t N, int32_t *counts_out, float *ser_out, void *scratch, void *stream);
/* Per-frame evaluation of n_runs independent runs at once (sweep engine): what func_VAELE_DP_MQAM_shaping.py:70-89 (seg_len =
 * batch_len: the last shift[0] + n_cut symbols of every minibatch are dropped) and func_VAEflex_DP_MQAM_shaping.py:74-84 (seg_len = 0)
 * do per run -- find_shift on out_train and find_shift_symb_full on out_const, roll by (r, -shift), cut, slice [edge : -edge-max|shift|],
 * SER_IQflip and SER_constell_shaping -- with the roll / cut / slice as index arithmetic and the shifts kept on the device.
 * q (R,2,2n,N), out (R,2,2,N), tx (R,2,2,N) float16 bits, run strides rs_* in elements; var (R,2) with run stride rs_var; nu_sc (R).
 * align_out int32 (R,2,4) = {shift_x, shift_y, r, symbols evaluated} for the estimators {from q, from out};
 * counts_out int32 (R,2,2,2,4) optional; ser_out float (R,4) = rows of SER_valid: constellation x, y, soft demapper x, y. */
size_t vaeq_frame_eval_scratch_bytes(int32_t n_runs, int32_t n_shift);
int vaeq_frame_eval_runs(const float *q, int64_t ld_q, int64_t rs_q, const float *out, int64_t ld_out, int64_t rs_out,
                         const uint16_t *tx, int64_t ld_tx, int64_t rs_tx, const float *amp, const float *var, int64_t rs_var,
                         const float *nu_sc, int32_t n_lev, int32_t N, int32_t n_shift, int32_t n_runs, int32_t seg_len,
                         int32_t edge, int32_t n_cut, int32_t *align_out, int32_t *counts_out, float *ser_out, void *scratch,
                         void *stream);

/* vaeq_frame_eval_runs with a choice of estimators (which: bit 0 = from q, bit 1 = from out; the pointer of an unselected one may be
 * NULL, its rows of align_out / counts_out / ser_out are left untouched) and, optionally, the rescale factor mean|tx| / mean|rx| of
 * sf:242 per run (scale_out, estimator from out).  The CMA drivers (CMA_DP:39-52) evaluate in two steps: estimator from out on the CPE
 * output, then soft_dec of the aligned and partially rescaled copy (vaeq_cma_align_rescale) and the estimator from q on it. */
int vaeq_frame_eval_runs_ex(const float *q, int64_t ld_q, int64_t rs_q, const float *out, int64_t ld_out, int64_t rs_out,
                            const uint16_t *tx, int64_t ld_tx, int64_t rs_tx, const float *amp, const float *var, int64_t rs_var,
                            const float *nu_sc, int32_t n_lev, int32_t N, int32_t n_shift, int32_t n_runs, int32_t seg_len,
                            int32_t edge, int32_t n_cut, int32_t which, int32_t *align_out, int32_t *counts_out, float *ser_out,
                            float *scale_out, void *scratch, void *stream);
/* CMA_DP:42-48 for all runs: oc (n_runs,2,2,N) = out rolled by (r, -shift) per run (align = align_out of the call above, estimator
 * from out) with the evaluated slice [edge, N - edge - max|shift|) multiplied by scale[run] -- what SER_constell_shaping leaves behind
 * in the view the drivers pass (sf:242) and soft_dec then reads */
int vaeq_cma_align_rescale(const float *out, int64_t ld_out, int64_t rs_out, const int32_t *align, const float *scale, int32_t N,
                           int32_t edge, int32_t n_runs, float *oc, void *stream);

/* extension, not in the reference: GMI of the soft-demapper SER's region and hypothesis for n_runs runs, without a host sync.
 *   GMI = H(X) + mean over the evaluated symbols of log2 q(x_tx | y), per pol, bit per 2-D symbol; H(X) = -2 sum_l P_l log2 P_l of
 *   the run's pmf; q clamped at 1e-30 before the log; logs and sums in double, one cast to float at the end.
 * The symbols are exactly those the SER counts: estimator 0 (from q) of vaeq_frame_eval_runs_ex, i.e. align (R,2,4) row [run][0] =
 * {shift_x, shift_y, r, n_eval}, cut per minibatch with seg_len (0: no cut).  Per pol the (IQ flip, rotation) with the smallest error
 * count of counts (R,2,2,2,4) [est][flip][pol][rotation] is scored (counter order, the first wins ties), so GMI is invariant under the
 * symmetries the SER forgives.  q (R,2,2n,N), tx (R,2,2,N) float16 bits, P (R,n) with run stride rs_P; gmi_out (R,2); n_eval == 0
 * gives NaN.  A run's result depends on its own inputs only (not on n_runs).  scratch: vaeq_frame_gmi_scratch_bytes. */
size_t vaeq_frame_gmi_scratch_bytes(int32_t n_runs, int32_t N);
int vaeq_frame_gmi_runs(const float *q, int64_t ld_q, int64_t rs_q, const uint16_t *tx, int64_t ld_tx, int64_t rs_tx, const float *P,
                        int64_t rs_P, const int32_t *align, const int32_t *counts, int32_t n_lev, int32_t N, int32_t n_runs, int32_t seg_len,
                        int32_t edge, int32_t n_cut, float *gmi_out, void *scratch, void *stream);

/* extension, not in the reference: achievable-rate estimate H(X)+E[log2 q(x_tx|y)] per pol (bit/2D symbol);
 * scratch: VAEQ_EVAL_SCRATCH_BYTES */
int vaeq_gmi(const float *q, int64_t ld_q, const uint16_t *tx, int64_t ld_tx, const float *P, int32_t n_lev, int32_t N,
             float *gmi_out, void *scratch, void *stream);

/* ------------------------------------------------------------------------------------------------
 * CMA baselines (sf:341-488) and carrier phase estimation (sf:140-186)
 * ---------------------------------------------------------------------------------------------- */
#define VAEQ_CMA_SAMPLE 0 /* CMA      sf:341-379: tap update after every symbol                 */
#define VAEQ_CMA_BATCH 1  /* CMAbatch sf:381-434: k%batchlen==0 && k!=0, window [k-batchlen,k)  */
#define VAEQ_CMA_FLEX 2   /* CMAflex  sf:436-488: k%symb_step==0 && k>=batchlen                 */
/* Rx (2,2,N) samples; h (2,2,2,M) updated in place when train != 0; out (2,2,N/sps); e (N/sps,2).
 * n_runs independent runs may be batched: every pointer then strides by its tensor size per run
 * (Rx by 4*ld... see INTEGRATION.md); n_runs == 1 for the reference call.  scratch: vaeq_cma_scratch_bytes. */
size_t vaeq_cma_scratch_bytes(int32_t N, int32_t M, int32_t n_runs);
int vaeq_cma(int32_t mode, const float *Rx, int32_t N, float R, float *h, int32_t M, float lr, int32_t batchlen,
             int32_t symb_step, int32_t sps, int32_t train, float *out, float *e, int32_t n_runs, void *scratch,
             void *stream);
/* CPE (sf:140-186): y (2,2,N) -> y_corr (2,2,N); scratch: vaeq_cpe_scratch_bytes(N) */
size_t vaeq_cpe_scratch_bytes(int32_t N);
int vaeq_cpe(const float *y, int32_t N, float *y_corr, void *scratch, void *stream);
/* the same for n_runs independent runs: y, y_corr (n_runs,2,2,N); scratch: vaeq_cpe_runs_scratch_bytes(N, n_runs) */
size_t vaeq_cpe_runs_scratch_bytes(int32_t N, int32_t n_runs);
int vaeq_cpe_runs(const float *y, int32_t N, int32_t n_runs, float *y_corr, void *scratch, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Single-polarisation CMA baseline of the AWGN module (AWGN_channel/func_CMA_MQAM_shaping.py, cm:)
 * ---------------------------------------------------------------------------------------------- */
/* CMA (cm:142-168): Rx (2,N) [I,Q], h (2,M) = Re / Im taps updated in place when train != 0, out (2,N/sps), e (N/sps); no power
 * normalisation (unlike the DP version).  n_runs independent runs: every pointer strides by its tensor size per run. */
int vaeq_cma_awgn(const float *Rx, int32_t N, float R, float *h, int32_t M, float lr, int32_t sps, int32_t train, float *out, float *e,
                  int32_t n_runs, void *stream);
/* CPE (cm:170-196): y (n_runs,2,N) -> y_corr, Viterbi-Viterbi WITHOUT unwrapping; scratch: vaeq_cpe_runs_scratch_bytes(N, n_runs) */
int vaeq_cpe_awgn(const float *y, int32_t N, int32_t n_runs, float *y_corr, void *scratch, void *stream);
/* SER_CMA (cm:63-93): rx (2,N) rows with stride ld_rx, RESCALED IN PLACE by mean|tx| / mean|rx| (cm:73); nearest-level decisions;
 * counts_out int32 (4) = symbol errors for the rotations 0, pi, and the two quarter turns; ser_out float (1) = min / N.
 * scratch: VAEQ_EVAL_SCRATCH_BYTES */
int vaeq_ser_cma(float *rx, int64_t ld_rx, const uint16_t *tx, int64_t ld_tx, const float *amp, int32_t n_lev, int32_t N,
                 int32_t *counts_out, float *ser_out, void *scratch, void *stream);
/* find_shift_symb (cm:127-140): correlation of tx[c, n_shift/2 : 1000] with rx[0, i : i + 1000 - n_shift/2], i < n_shift (NOT circular);
 * corr_out float (2, n_shift) for c = I, Q; shift_out int32 (1) = argmax|corr_I| - n_shift/2, or the Q component's when
 * max|corr_I| < 0.02 n_rx and max|corr_Q| >= max|corr_I| */
int vaeq_find_shift_symb(const float *rx, int32_t n_rx, const uint16_t *tx, int64_t ld_tx, int32_t n_tx, int32_t n_shift, float *corr_out,
                         int32_t *shift_out, void *stream);
/* A validation period of the AWGN CMA driver for n_runs runs in ONE launch (one warp per run): n_frames training frames in sequence
 * (cm:142-168 with updates, no per-symbol output), then the pass without updates over the validation frame.  Bit for bit a loop of
 * vaeq_cma_awgn calls per run (n_frames with train = 1, then one with train = 0).
 *   rx_train: frame f of run k at rx_train + k*rs_t + f*fs_t, I row of N_train samples, Q row ld_t further
 *   rx_valid: run k at rx_valid + k*rs_v, I row of N_valid samples, Q row ld_v further
 *   h (n_runs,2,M) taps, updated in place; lr (n_runs) float per run; out_v (n_runs,2,N_valid/sps) */
int vaeq_cma_awgn_runs(const float *rx_train, int64_t ld_t, int64_t fs_t, int64_t rs_t, int32_t n_frames, int32_t N_train,
                       const float *rx_valid, int64_t ld_v, int64_t rs_v, int32_t N_valid, float *h, int32_t M, const float *lr, float R,
                       int32_t sps, float *out_v, int32_t n_runs, void *stream);
/* Validation scoring of the AWGN CMA driver (cm:227-229) for n_runs runs without a host sync: per run
 *   shift = find_shift_symb(y, tx, n_shift), then SER_CMA(y[:, edge+shift : N-edge], tx[:, edge : N-edge-shift]),
 * bit for bit as vaeq_find_shift_symb + vaeq_ser_cma, except that the rescaled values are NOT written back to y (the driver never
 * reads them).  y (n_runs,2,N) float: rows ld_y apart, runs rs_y apart; tx (n_runs,2,N) float16 bits.  Needs N >= 1000 + n_shift/2
 * and edge >= n_shift/2.  Outputs on the device: shift (n_runs) int32, counts (n_runs,4) int32, ser (n_runs) float.
 * scratch: vaeq_awgn_cma_eval_scratch_bytes. */
size_t vaeq_awgn_cma_eval_scratch_bytes(int32_t n_runs, int32_t N, int32_t n_shift, int32_t edge);
int vaeq_awgn_cma_eval_runs(const float *y, int64_t ld_y, int64_t rs_y, const uint16_t *tx, int64_t ld_tx, int64_t rs_tx, const float *amp,
                            int32_t n_lev, int32_t N, int32_t n_shift, int32_t edge, int32_t n_runs, int32_t *shift_out, int32_t *counts_out,
                            float *ser_out, void *scratch, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Synthetic test signal on the device, n_runs independent runs per call (generate_data_shaping sf:65-90, channel 'h0'; the
 * reference's generator is unseeded, parity is statistical).  The host side (vae_equalizer_b200/datagen.py) runs
 *   vaeq_gen_levels -> vaeq_gen_pulse -> FFT -> vaeq_gen_jones -> IFFT -> vaeq_gen_noise
 * with the two DFTs of the dispersion step (sf:40, 54) on cuFFT.  Random numbers are Philox4x32-10 outputs keyed by
 * (seed, run, row, position): a run's data does not depend on the batch it is generated in.
 * ---------------------------------------------------------------------------------------------- */
/* sf:75-76, 89: lev (n_runs,4,n_conv) float rows [pol0 I, pol0 Q, pol1 I, pol1 Q] drawn from amps (n_lev) with pmf P (n_runs,n_lev);
 * tx (n_runs,2,2,N) float16 bit patterns = lev[:, :, tx_off : tx_off + N] */
int vaeq_gen_levels(const float *amps, const float *P, int32_t n_lev, int32_t n_conv, int32_t N, int32_t tx_off, uint64_t seed,
                    float *lev, uint16_t *tx, int32_t n_runs, void *stream);
/* sf:77-80 (simulate_channel sf:56-63 with a one-tap channel): zero insertion by sps = 2 and 'valid' convolution with the pulse h
 * (n_pulse taps, even); shaped (n_runs,2,2*n_conv - n_pulse) complex64, 16-byte aligned */
int vaeq_gen_pulse(const float *lev, const float *h, int32_t n_pulse, int32_t n_conv, float *shaped, int32_t n_runs, void *stream);
/* sf:41-53 in the frequency domain, in place: X (n_runs,2,n) complex64 spectra; Pcd = exp_pmd*exp_cd, Picd = exp_cd/exp_pmd (n) complex64;
 * theta (n_runs) rotation angles; phi0, phi1 the IQ phases (exp_phiIQ = exp(-j phi), sf:44) */
int vaeq_gen_jones(float *X, const float *Pcd, const float *Picd, const float *theta, float phi0, float phi1, int32_t n, int32_t n_runs,
                   void *stream);
/* sf:83-88: rx (n_runs,2,2,L) float32 = Re/Im of sig[:, :, :L] + sigma[run] * N(0,1); sig (n_runs,2,n) complex64, L <= n */
int vaeq_gen_noise(const float *sig, const float *sigma, uint64_t seed, int32_t n, int32_t L, float *rx, int32_t n_runs, void *stream);
/* Single-polarisation signal of the AWGN module (generate_data, AWGN_channel/func_VAELE_MQAM_shaping.py:39-61), n_frames frames
 * (frame indices frame0 ..) of N symbols for each of n_runs runs, all sps = 2:
 *   lev (n_runs, n_frames, 2, n_conv) f32   levels drawn from P (n_runs, n_lev) by inverse CDF
 *   sig (n_runs, n_frames, 2 n_conv - K) complex64   'valid' FIR of the zero-stuffed symbols with taps (K complex, re/im interleaved,
 *       even K: rrcfir (*) h_channel), noise-free
 *   rx  (n_runs, n_frames, 2, 2 N) f32   sig[:2N] + sigma_n (N(0,1) + j N(0,1)), sigma_n from the frame's mean |sig|^2 and snr[run] dB
 *   tx  (n_runs, n_frames, 2, N) float16 bits   lev[:, tx_off : tx_off + N]
 * Every draw is keyed by (seeds[run], frame index, row, position): a run's frames do not depend on the other runs of the call. */
int vaeq_gen_awgn(const float *amps, const float *P, int32_t n_lev, const float *taps, int32_t K, int32_t N, int32_t tx_off, int32_t n_conv,
                  const float *snr, const uint64_t *seeds, int32_t frame0, int32_t n_frames, int32_t n_runs, float *lev, float *sig, float *rx,
                  uint16_t *tx, void *stream);

/* ------------------------------------------------------------------------------------------------
 * AWGN single-polarisation VAE-LE step: twoFIR.forward (AWGN_channel/func_VAELE_MQAM_shaping.py:214-231)
 * + loss_function (:63-95) + backward + Adam(amsgrad=True) (:283-306)
 * ---------------------------------------------------------------------------------------------- */
typedef struct vaeq_awgn_desc {
    int32_t B, sps, M, n_lev;
    float amp_mean; /* :271 */
    float var;      /* 10^(-SNR/10), :272 */
    const float *rx; /* (2,L) [I/Q][sample] */
    const float *amp, *P;
    float *W;       /* (1,2,M) */
    float *h;       /* (2,M)   */
    float *adam;    /* vaeq_adam_state_floats_awgn(M) floats */
    float *q;       /* (2n,B) */
    float *out;     /* (2,B)  */
    float *loss;    /* (1)    */
    float *gW, *gh; /* optional */
    void *workspace;
    size_t workspace_bytes;
} vaeq_awgn_desc;
size_t vaeq_awgn_workspace_bytes(int32_t B, int32_t M, int32_t n_lev);
size_t vaeq_adam_state_floats_awgn(int32_t M);
int vaeq_awgn_forward(const vaeq_awgn_desc *d, void *stream);
int vaeq_awgn_forward_backward(const vaeq_awgn_desc *d, void *stream);
int vaeq_awgn_train_step(const vaeq_awgn_desc *d, float lr_w, float lr_h, void *stream);

/* R independent runs in ONE launch, one CTA of the single-run step kernel per run (sweep engine): bit for bit a loop of
 * vaeq_awgn_train_step / vaeq_awgn_forward per run.  `d` holds run 0's pointers (d->var and d->amp_mean are ignored: per-run
 * values come from `r`); run k's arrays start at d->X + k * r->rs_X (elements).  workspace: vaeq_awgn_runs_workspace_bytes. */
typedef struct vaeq_awgn_runs {
    int32_t n_runs;
    int64_t rs_rx, rs_W, rs_h, rs_adam, rs_P, rs_q, rs_out, rs_loss;
    const float *lr;       /* (n_runs) Adam lr of both parameter groups (:305-306); train only */
    const float *var;      /* (n_runs) 10^(-SNR/10) */
    const float *amp_mean; /* (n_runs) */
} vaeq_awgn_runs;
size_t vaeq_awgn_runs_workspace_bytes(int32_t B, int32_t M, int32_t n_lev, int32_t n_runs);
/* n_frames frames per run, each n_mb minibatches of B = d->B symbols (the epoch loop of :291-306; the frame's remaining symbols are
 * unused): minibatch m of frame f is rx + f*fs_rx + m*sps*B, its Q row ld_rx after its I row.  d->q (2n,B) / d->out (2,B) per run are
 * scratch; d->loss (n_runs, n_frames*n_mb) receives every step's loss (row stride r->rs_loss). */
int vaeq_awgn_train_frames_runs(const vaeq_awgn_desc *d, const vaeq_awgn_runs *r, int64_t ld_rx, int64_t fs_rx, int32_t n_frames,
                                int32_t n_mb, void *stream);
/* forward of every run over B = d->B symbols (rx rows ld_rx apart): q (2n,B), out (2,B) and loss per run */
int vaeq_awgn_forward_runs(const vaeq_awgn_desc *d, const vaeq_awgn_runs *r, int64_t ld_rx, void *stream);
/* Validation scoring of the AWGN driver (processing.py awgn_find_shift + awgn_ser_q, :188-204, :97-124) for n_runs runs without a
 * host sync.  q (n_runs, 2n, N): rows ld_q apart, runs rs_q apart; tx (n_runs, 2, N) float16 bits.  Shift search on the first
 * n_corr symbols (circular), E from q's I rows, correlated with tx I and tx Q; then the counts of q[:, edge+shift : N-edge] against
 * tx[:, edge : N-edge-shift] for the 4 rotations (no IQ flip).  Outputs: shift (n_runs), counts (n_runs, 4), ser (n_runs).
 * scratch: vaeq_awgn_eval_scratch_bytes. */
size_t vaeq_awgn_eval_scratch_bytes(int32_t n_runs, int32_t n_shift, int32_t n_corr);
int vaeq_awgn_eval_runs(const float *q, int64_t ld_q, int64_t rs_q, const uint16_t *tx, int64_t ld_tx, int64_t rs_tx, const float *amp,
                        int32_t n_lev, int32_t N, int32_t n_shift, int32_t n_corr, int32_t edge, int32_t n_runs, int32_t *shift_out,
                        int32_t *counts_out, float *ser_out, void *scratch, void *stream);
/* The GMI of vaeq_frame_gmi_runs for the AWGN driver: one polarisation, no IQ flip.  q[:, edge + shift : N - edge] against
 * tx[:, edge : N - edge - shift] with shift (R) and counts (R,4) [rotation] of vaeq_awgn_eval_runs; gmi_out (R).  Needs
 * edge >= n_shift/2 of that call (the default 11 >= 10), so edge + shift >= 0; a run whose shift is below -edge gives NaN.
 * scratch: vaeq_awgn_gmi_scratch_bytes. */
size_t vaeq_awgn_gmi_scratch_bytes(int32_t n_runs, int32_t N);
int vaeq_awgn_gmi_runs(const float *q, int64_t ld_q, int64_t rs_q, const uint16_t *tx, int64_t ld_tx, int64_t rs_tx, const float *P, int64_t rs_P,
                       const int32_t *shift, const int32_t *counts, int32_t n_lev, int32_t N, int32_t n_runs, int32_t edge, float *gmi_out,
                       void *scratch, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* VAEQ_H_ */
