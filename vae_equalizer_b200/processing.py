"""The per-run `processing(...)` drivers of the reference, re-hosted on the CUDA path.

Positional signatures, return values and the per-frame printed fields are the reference's
(optical_DP_channel/func_VAELE_DP_MQAM_shaping.py:17-95, func_VAEflex_DP_MQAM_shaping.py:16-88,
func_CMA*_DP_MQAM_shaping.py:16-56, AWGN_channel/func_VAELE_MQAM_shaping.py:235-324), so the unmodified
Eval_run_*.py scripts run against them.  One whole frame of sequential minibatches is ONE C-ABI call
(vaeq_dp_train_frame); the host syncs only where the reference does (.item() in the prints and the
data-dependent slicing by the detected shift).  Extra keyword-only arguments (`rng`, `verbose`,
`device`) are additions; the reference's generators are unseeded.
"""
from __future__ import annotations

import numpy as np
import torch

from . import shared_funcs as sfun
from .awgn import AWGNEqualizer, generate_data
from .constants import awgn_constants, upsampled_channel
from .dp import DPEqualizer

N_CUT = 10     # symbols cut per minibatch/frame edge (VAELE_DP:40, CMA_DP:26)


def _make_frame(datagen, N, amps, SNR, h_channel, P, pol, symb_rate, sps, tau_cd, tau_pmd, phiIQ, theta, device, rng, frame_seed):
    """One frame of test signal.  datagen="numpy": the reference's host-side generator restated (sf:65-90);
    datagen="gpu": the same signal model generated on the device (statistical, not bitwise, parity; channels 'h0', 'h1', 'h2');
    datagen=<iterator of (rx (2,2,sps*N) float32, tx (2,2,N) float16)>: replay recorded frames (parity tests feed the frames the
    reference's processing() was given, tests/golden/make_golden_drivers.py)."""
    if hasattr(datagen, "__next__"):
        rx, tx = next(datagen)
        rx, tx = torch.as_tensor(rx, dtype=torch.float32).to(device).contiguous(), torch.as_tensor(tx, dtype=torch.float16).to(device).contiguous()
        if tx.shape[-1] != N or rx.shape[-1] != sps * N:
            raise sfun._lib.VaeqError(f"replayed frame has {tx.shape[-1]} symbols / {rx.shape[-1]} samples, the driver asked for {N} symbols")
        return rx, tx, 0.0
    if datagen == "gpu":
        from .datagen import generate_data_gpu
        return generate_data_gpu(N, amps, SNR, P, sps, theta, device, frame_seed, symb_rate=symb_rate, tau_cd=tau_cd,
                                 tau_pmd=tau_pmd, phiIQ=phiIQ, h_channel=h_channel)
    return sfun.generate_data_shaping(N, amps, SNR, h_channel, P, pol, symb_rate, sps, tau_cd, tau_pmd, phiIQ, theta, device, rng=rng)


def _cuda_device(device):
    if device is None:
        if not torch.cuda.is_available():
            raise sfun._lib.VaeqError("no CUDA device: vae_equalizer_b200 has no CPU path")
        device = torch.device("cuda", torch.cuda.current_device())
    return torch.device(device)


def _align(t, shift_h, r):
    """out.roll(r,0) then per-pol time roll by -shift (VAELE_DP:71-72)."""
    t = t.roll(r, 0)
    t[0], t[1] = t[0].roll(-shift_h[0], -1).clone(), t[1].roll(-shift_h[1], -1).clone()
    return t


def _print_frame(frame, loss, shift_h, r, snr_db, ser):
    print(frame, '\t\ttraining: loss = ', loss, '\tshift_x = ', shift_h[0], '\tshift_y = ', shift_h[1], '\tr = ', r,
          '\tSNR_est = ', snr_db)
    print('\t\t\t\t\t\t\tSER_x = ', ser[0], '\tSER_y = ', ser[1], '\t(constell. with shaping)')
    print('\t\t\t\t\t\t\tSER_x = ', ser[2], '\tSER_y = ', ser[3], '\t(soft demapper)')


def _eval_fused(out_train, out_const, data_tensor, amp_levels, var, nu_sc, seg_len):
    """The per-frame evaluation of the VAE drivers in ONE call sequence without a host sync (vaeq_frame_eval_runs with a single run): the
    same error counts as the find_shift -> roll -> cut -> SER_* sequence (tests/test_frames_gpu.py).  Returns (SER (4,), align (2,4) int32)."""
    ser, al = sfun.frame_eval_runs(out_train.unsqueeze(0), out_const.unsqueeze(0), data_tensor.unsqueeze(0), amp_levels, var.reshape(1, 2),
                                   torch.full((1,), float(nu_sc), device=out_train.device), seg_len, n_cut=N_CUT)
    return ser[0], al[0]


def eval_frame_vae(out_train, out_const, data_tensor, amp_levels, nu_sc, var, seg_len):
    """The per-frame evaluation of the VAE drivers, call by call like the reference: VAELE_DP:70-89 with seg_len = batch_len (the last
    shift[0] + N_cut symbols of every minibatch are dropped before the slice), VAEflex_DP:74-84 with seg_len = 0.
    Returns (SER (4,) [constellation x, y, soft demapper x, y], (shift, r) of find_shift, (shift, r) of find_shift_symb_full)."""
    pol, n2, N = out_train.shape
    ser = torch.empty(4, device=out_train.device, dtype=torch.float32)

    def cut(t, sh):
        if not seg_len:
            return t
        keep = seg_len - sh[0] - N_CUT                 # VAELE_DP:73-77 (a slice bound: clamps to the minibatch, negative counts from its end)
        return t.reshape(pol, t.shape[1], N // seg_len, seg_len)[:, :, :, :keep].reshape(pol, t.shape[1], -1)

    shift, r = sfun.find_shift(out_train, data_tensor, 21, amp_levels, pol)
    sh_q = [int(v) for v in shift.tolist()]
    out_train = _align(out_train, sh_q, r)
    tail = 11 + max(abs(sh_q[0]), abs(sh_q[1]))
    ser[2:] = sfun.SER_IQflip(cut(out_train, sh_q)[:, :, 11:-tail], cut(data_tensor, sh_q)[:, :, 11:-tail])
    shift, r2 = sfun.find_shift_symb_full(out_const, data_tensor, 21)
    sh_c = [int(v) for v in shift.tolist()]
    out_const = _align(out_const, sh_c, r2)
    tail = 11 + max(abs(sh_c[0]), abs(sh_c[1]))
    ser[:2] = sfun.SER_constell_shaping(cut(out_const, sh_c)[:, :, 11:-tail].detach().clone(), cut(data_tensor, sh_c)[:, :, 11:-tail],
                                        amp_levels, nu_sc, var)
    return ser, (sh_q, r), (sh_c, r2)


def eval_frame_cma(out_const, data_tensor, amp_levels, nu_sc, var, pol=2):
    """The per-frame evaluation of the CMA drivers (CMA_DP:39-52): CPE of the equalizer output without its N_cut edge symbols, alignment
    from the constellation, SER_constell_shaping on a VIEW (its in-place rescale, sf:242, is what soft_dec then reads), soft demapper,
    alignment from q, SER_IQflip.  Returns (SER (4,), (shift, r) from out, (shift, r) from q, out_const as soft_dec saw it)."""
    ser = torch.empty(4, device=out_const.device, dtype=torch.float32)
    out_const = sfun.CPE(out_const[:, :, N_CUT:-N_CUT])
    data_tensor = data_tensor[:, :, N_CUT:-N_CUT]
    shift, r = sfun.find_shift_symb_full(out_const, data_tensor, 21)
    sh_c = [int(v) for v in shift.tolist()]
    out_const = _align(out_const, sh_c, r)
    tail = 11 + max(abs(sh_c[0]), abs(sh_c[1]))
    # a VIEW is passed on purpose: the in-place rescale (sf:242) must be visible to soft_dec below (CMA_DP:44,48)
    ser[:2] = sfun.SER_constell_shaping(out_const[:, :, 11:-tail], data_tensor[:, :, 11:-tail], amp_levels, nu_sc, var)
    out_train = sfun.soft_dec(out_const, var, amp_levels, nu_sc)
    shift, r2 = sfun.find_shift(out_train, data_tensor, 21, amp_levels, pol)
    sh_q = [int(v) for v in shift.tolist()]
    out_train = _align(out_train, sh_q, r2)
    tail = 11 + max(abs(sh_q[0]), abs(sh_q[1]))
    ser[2:] = sfun.SER_IQflip(out_train[:, :, 11:-tail], data_tensor[:, :, 11:-tail])
    return ser, (sh_c, r), (sh_q, r2), out_const


def processing_vaele_dp(mod, sps, SNR, nu, M_est, theta_diff, theta, lr_optim, batch_len, N_frame_max, num_frames, flex_step,
                        channel, symb_rate, tau_cd, tau_pmd, phiIQ, N_lrhalf, *, device=None, rng=None, verbose=True, datagen="numpy", seed=0,
                        eval_mode="per_op"):
    """VAE-LE, non-overlapping minibatches (func_VAELE_DP_MQAM_shaping.py:17-95).  eval_mode="per_op" replays the reference's evaluation
    call by call (two host syncs per frame for the detected shifts), "fused" evaluates the frame in one launch sequence without a sync."""
    device = _cuda_device(device)
    if verbose:
        print("We are using the following device for learning:", device)
    h_est, h_channel, P, amp_levels, amps, pol, nu_sc, var, pow_mean = sfun.init(channel, mod, device, nu, sps, M_est, SNR)
    num_lev = amp_levels.shape[0]
    eq = DPEqualizer(M_est, sps, amp_levels, P, var, nu_sc, device=device)
    SER_valid = torch.empty(4, num_frames, device=device, dtype=torch.float32)
    Var_est = torch.empty(pol, num_frames, device=device, dtype=torch.float32)
    m_max = N_frame_max // batch_len
    N_frame = m_max * batch_len
    lr_w = lr_optim
    for frame in range(num_frames):
        if frame % N_lrhalf == 0 and frame != 0:
            lr_w = lr_optim * 0.5                  # param_groups[0] only, not cumulative (VAELE_DP:45-46)
        rx_tensor, data_tensor, _ = _make_frame(datagen, N_frame, amps, SNR, h_channel, P, pol, symb_rate, sps, tau_cd, tau_pmd,
                                                phiIQ, theta, device, rng, seed * 100003 + frame)
        theta += theta_diff
        out_train = torch.empty(pol, 2 * num_lev, N_frame, device=device, dtype=torch.float32)
        out_const = torch.empty(pol, 2, N_frame, device=device, dtype=torch.float32)
        loss_steps, var_est = eq.train_frame(rx_tensor, batch_len, batch_len, m_max, lr_w, lr_optim, out_train, out_const,
                                             0, batch_len, keep_lo_in_dst=True)
        SNR_est = pow_mean / torch.mean(var_est)
        Var_est[:, frame] = torch.mean(var_est, dim=1)

        if eval_mode == "fused":
            SER_valid[:, frame], al = _eval_fused(out_train, out_const, data_tensor, amp_levels, var, nu_sc, batch_len)
            if verbose:
                a = al.tolist()
                _print_frame(frame, loss_steps[-1].item(), a[1][:2], a[1][2], (10 * torch.log10(SNR_est)).item(), SER_valid[:, frame].tolist())
            continue
        SER_valid[:, frame], _, (sh, r) = eval_frame_vae(out_train, out_const, data_tensor, amp_levels, nu_sc, var, batch_len)
        if verbose:
            _print_frame(frame, loss_steps[-1].item(), sh, r, (10 * torch.log10(SNR_est)).item(), SER_valid[:, frame].tolist())
    return SER_valid, Var_est, var


def processing_vaeflex_dp(mod, sps, SNR, nu, M_est, theta_diff, theta, lr_optim, batch_len, N_train_max, num_frames, flex_step,
                          channel, symb_rate, tau_cd, tau_pmd, phiIQ, N_lrhalf, *, device=None, rng=None, verbose=True, datagen="numpy", seed=0,
                          eval_mode="per_op", group=None, split_transport="auto"):
    """VAE-flex, sliding window advanced by flex_step (func_VAEflex_DP_MQAM_shaping.py:16-88).

    group (a torch.distributed process group, or True for the default group; one process per GPU, every rank calls with the same
    arguments): ONE run whose every window is batch-split over the ranks (BASELINE configs[2]; parallel.BatchSplitDP) -- rank 0
    generates the frame and broadcasts rx, every rank trains its symbol range of every window (two tiny reductions per step,
    replicated Adam), the kept columns are gathered on rank 0, which evaluates like the single-GPU driver; the SER / Var_est it returns
    are broadcast, so every rank returns the same tensors."""
    if group is not None:
        return _processing_vaeflex_split(mod, sps, SNR, nu, M_est, theta_diff, theta, lr_optim, batch_len, N_train_max, num_frames, flex_step,
                                         channel, symb_rate, tau_cd, tau_pmd, phiIQ, N_lrhalf, device, rng, verbose, datagen, seed, eval_mode,
                                         group, split_transport)
    device = _cuda_device(device)
    if verbose:
        print("We are using the following device for learning:", device)
    h_est, h_channel, P, amp_levels, amps, pol, nu_sc, var, pow_mean = sfun.init(channel, mod, device, nu, sps, M_est, SNR)
    num_lev = amp_levels.shape[0]
    eq = DPEqualizer(M_est, sps, amp_levels, P, var, nu_sc, device=device)
    SER_valid = torch.empty(4, num_frames, device=device, dtype=torch.float32)
    Var_est = torch.empty(pol, num_frames, device=device, dtype=torch.float32)
    N_frame = (N_train_max // batch_len) * batch_len
    m_max = (N_frame - batch_len) // flex_step * flex_step          # VAEflex_DP:39
    n_steps = m_max // flex_step
    keep_lo, keep_hi = (batch_len - flex_step) // 2, (batch_len + flex_step) // 2     # VAEflex_DP:64-65
    lr_w = lr_optim
    for frame in range(num_frames):
        if frame % N_lrhalf == 0 and frame != 0:
            lr_w = lr_optim * 0.5
        rx_tensor, data_tensor, _ = _make_frame(datagen, N_frame, amps, SNR, h_channel, P, pol, symb_rate, sps, tau_cd, tau_pmd,
                                                phiIQ, theta, device, rng, seed * 100003 + frame)
        data_tensor = data_tensor[:, :, batch_len // 2:m_max + batch_len // 2]                 # VAEflex_DP:51
        theta += theta_diff
        out_train = torch.empty(pol, 2 * num_lev, m_max, device=device, dtype=torch.float32)
        out_const = torch.empty(pol, 2, m_max, device=device, dtype=torch.float32)
        loss_steps, var_est = eq.train_frame(rx_tensor, batch_len, flex_step, n_steps, lr_w, lr_optim, out_train, out_const,
                                             keep_lo, keep_hi - keep_lo, keep_lo_in_dst=False)
        SNR_est = pow_mean / torch.mean(var_est)
        Var_est[:, frame] = torch.mean(var_est, dim=1)

        if eval_mode == "fused":
            SER_valid[:, frame], al = _eval_fused(out_train, out_const, data_tensor, amp_levels, var, nu_sc, 0)
            if verbose:
                a = al.tolist()
                _print_frame(frame, loss_steps[-1].item(), a[1][:2], a[1][2], (10 * torch.log10(SNR_est)).item(), SER_valid[:, frame].tolist())
            continue
        SER_valid[:, frame], _, (sh, r) = eval_frame_vae(out_train, out_const, data_tensor, amp_levels, nu_sc, var, 0)
        if verbose:
            _print_frame(frame, loss_steps[-1].item(), sh, r, (10 * torch.log10(SNR_est)).item(), SER_valid[:, frame].tolist())
    return SER_valid, Var_est, var


def _processing_vaeflex_split(mod, sps, SNR, nu, M_est, theta_diff, theta, lr_optim, batch_len, N_train_max, num_frames, flex_step,
                              channel, symb_rate, tau_cd, tau_pmd, phiIQ, N_lrhalf, device, rng, verbose, datagen, seed, eval_mode, group, transport):
    """processing_vaeflex_dp with every window split over the ranks of `group` (same frame loop: VAEflex_DP:36-86)."""
    import torch.distributed as dist
    from .parallel import BatchSplitDP
    group = None if group is True else group
    device = _cuda_device(device)
    rank = dist.get_rank(group)
    src = dist.get_global_rank(group, 0) if group is not None else 0
    verbose = verbose and rank == 0
    if verbose:
        print("We are using the following device for learning:", device, f"(batch-split over {dist.get_world_size(group)} ranks)")
    h_est, h_channel, P, amp_levels, amps, pol, nu_sc, var, pow_mean = sfun.init(channel, mod, device, nu, sps, M_est, SNR)
    num_lev = amp_levels.shape[0]
    eq = DPEqualizer(M_est, sps, amp_levels, P, var, nu_sc, device=device)
    bs = BatchSplitDP(eq, group, transport)
    SER_valid = torch.zeros(4, num_frames, device=device, dtype=torch.float32)
    Var_est = torch.empty(pol, num_frames, device=device, dtype=torch.float32)
    N_frame = (N_train_max // batch_len) * batch_len
    m_max = (N_frame - batch_len) // flex_step * flex_step          # VAEflex_DP:39
    n_steps = m_max // flex_step
    keep_lo, keep_hi = (batch_len - flex_step) // 2, (batch_len + flex_step) // 2     # VAEflex_DP:64-65
    rx_buf = torch.empty(pol, 2, sps * N_frame, device=device, dtype=torch.float32)   # the same buffers every frame: the frame loop is a CUDA graph
    out_train = torch.empty(pol, 2 * num_lev, m_max, device=device, dtype=torch.float32)
    out_const = torch.empty(pol, 2, m_max, device=device, dtype=torch.float32)
    lr_w = lr_optim
    for frame in range(num_frames):
        if frame % N_lrhalf == 0 and frame != 0:
            lr_w = lr_optim * 0.5
        data_tensor = None
        if rank == 0:
            rx_tensor, data_tensor, _ = _make_frame(datagen, N_frame, amps, SNR, h_channel, P, pol, symb_rate, sps, tau_cd, tau_pmd,
                                                    phiIQ, theta, device, rng, seed * 100003 + frame)
            data_tensor = data_tensor[:, :, batch_len // 2:m_max + batch_len // 2]             # VAEflex_DP:51
            rx_buf.copy_(rx_tensor)
        dist.broadcast(rx_buf, src=src, group=group)
        theta += theta_diff
        out_train.zero_()
        out_const.zero_()
        loss_steps, var_est = bs.train_frame(rx_buf, batch_len, flex_step, n_steps, lr_w, lr_optim, out_train, out_const, keep_lo, keep_hi - keep_lo)
        bs.gather_kept(batch_len, flex_step, n_steps, out_train, out_const, keep_lo, keep_hi - keep_lo, dst=0)
        SNR_est = pow_mean / torch.mean(var_est)
        Var_est[:, frame] = torch.mean(var_est, dim=1)
        if rank == 0:
            if eval_mode == "fused":
                SER_valid[:, frame], al = _eval_fused(out_train, out_const, data_tensor, amp_levels, var, nu_sc, 0)
                sh, r = al.tolist()[1][:2], al.tolist()[1][2]
            else:
                SER_valid[:, frame], _, (sh, r) = eval_frame_vae(out_train.clone(), out_const.clone(), data_tensor, amp_levels, nu_sc, var, 0)
            if verbose:
                _print_frame(frame, loss_steps[-1].item(), sh, r, (10 * torch.log10(SNR_est)).item(), SER_valid[:, frame].tolist())
    dist.broadcast(SER_valid, src=src, group=group)
    return SER_valid, Var_est, var


def _processing_cma(kind, mod, sps, SNR, nu, M_est, theta_diff, theta, lr_optim, batch_len, N_train_max, num_frames, flex_step,
                    channel, symb_rate, tau_cd, tau_pmd, phiIQ, N_lrhalf, *, device=None, rng=None, verbose=True, datagen="numpy", seed=0):
    """CMA / CMAbatch / CMAflex runs (func_CMA_DP_MQAM_shaping.py:16-56 and siblings)."""
    device = _cuda_device(device)
    if verbose:
        print("We are using the following device for learning:", device)
    h_est, h_channel, P, amp_levels, amps, pol, nu_sc, var, pow_mean = sfun.init(channel, mod, device, nu, sps, M_est, SNR)
    h_est = h_est.detach()
    SER_valid = torch.empty(4, num_frames, device=device, dtype=torch.float32)
    Var_est = torch.zeros(pol, num_frames, device=device, dtype=torch.float32)
    R = 1
    for frame in range(num_frames):
        if frame % N_lrhalf == 0 and frame != 0:
            lr_optim *= 0.5                          # cumulative here, unlike the VAE drivers (CMA_DP:31-32)
        rx_tensor, data_tensor, _ = _make_frame(datagen, N_train_max, amps, SNR, h_channel, P, pol, symb_rate, sps, tau_cd, tau_pmd,
                                                phiIQ, theta, device, rng, seed * 100003 + frame)
        if kind == "CMA":
            out_const, h_est, e = sfun.CMA(rx_tensor, R, h_est, lr_optim, sps, True)
        elif kind == "CMAbatch":
            out_const, h_est, e = sfun.CMAbatch(rx_tensor, R, h_est, lr_optim, batch_len, sps, True)
        else:
            out_const, h_est, e = sfun.CMAflex(rx_tensor, R, h_est, lr_optim, batch_len, flex_step, sps, True)
        theta += theta_diff
        SER_valid[:, frame], (sh, r), _, _ = eval_frame_cma(out_const, data_tensor, amp_levels, nu_sc, var, pol)
        if verbose:
            print(frame, '\t\ttraining: loss = ', torch.sum(e).item(), '\tshift_x = ', sh[0], '\tshift_y = ', sh[1], '\tr = ', r)
            print('\t\t\t\t\t\t\tSER_x = ', SER_valid[0, frame].item(), '\tSER_y = ', SER_valid[1, frame].item(), '\t(constell. with shaping)')
            print('\t\t\t\t\t\t\tSER_x = ', SER_valid[2, frame].item(), '\tSER_y = ', SER_valid[3, frame].item(), '\t(soft demapper)')
    return SER_valid, Var_est, var


def processing_cma_dp(*a, **k):
    return _processing_cma("CMA", *a, **k)


def processing_cmabatch_dp(*a, **k):
    return _processing_cma("CMAbatch", *a, **k)


def processing_cmaflex_dp(*a, **k):
    return _processing_cma("CMAflex", *a, **k)


# -------------------------------------------------------------------------------------------------
# AWGN single-polarisation VAE-LE (AWGN_channel/func_VAELE_MQAM_shaping.py:235-324)
# -------------------------------------------------------------------------------------------------
def awgn_find_shift(q, tx, N_shift, amp_levels):
    """find_shift of the AWGN module (:188-204): first 1000 symbols, I first, Q as fallback."""
    n = amp_levels.numel()
    q2 = torch.stack((q[:, :1000], q[:, :1000])).contiguous()
    tx2 = torch.stack((tx[:, :1000], tx[:, :1000])).contiguous()
    _, _, corr = sfun.find_shift(q2, tx2, N_shift, amp_levels, 2, return_corr=True)
    cI, cQ = corr[0, 0, 0].cpu(), corr[1, 0, 0].cpu()
    half = N_shift // 2
    if cI.max() >= 0.02 * q.shape[-1]:
        return half - int(torch.argmax(cI))
    if cQ.max() >= cI.max():
        return half - int(torch.argmax(cQ))
    return half - int(torch.argmax(cI))


def awgn_ser_q(q, tx):
    """SER_q (:97-124): min over 4 rotations, no IQ flip.  Returns (ser float32 0-dim tensor, counts (4,))."""
    q2 = torch.stack((q, q)).contiguous()
    tx2 = torch.stack((tx, tx)).contiguous()
    _, counts = sfun.SER_IQflip(q2, tx2, return_counts=True)
    c = counts[0, 0, :]
    return (c.min().to(torch.float32) / q.shape[-1]), c


def processing_vaele_awgn(mod, sps, SNR, nu, M_est, lr_optim, batch_len, N_valid, N_train, num_epochs, epe, channel, *,
                          device=None, rng=None, verbose=True):
    device = _cuda_device(device)
    if verbose:
        print("We are using the following device for learning:", device)
    if channel not in ("h1", "h2"):
        raise KeyError(f"AWGN driver knows channels h1/h2, got {channel!r}")       # :239-242
    h_channel = upsampled_channel(channel, sps)
    M = (len(h_channel) - 1) // sps + 1
    amps, P, amp_mean, var = awgn_constants(mod, nu, SNR)
    amp_levels = torch.tensor(amps, device=device, dtype=torch.float32)
    eq = AWGNEqualizer(M_est, sps, amp_levels, P, amp_mean, var, device=device)
    SER_valid = torch.empty(num_epochs // epe, device=device, dtype=torch.float32)
    for epoch in range(num_epochs):
        rx_tensor, _ = generate_data(N_train, M, amps, SNR, h_channel, sps, device, P, rng=rng)
        for m in range(N_train // batch_len):
            minibatch = rx_tensor[:, m * batch_len * sps:(m + 1) * batch_len * sps].contiguous()
            _, _, loss = eq.train_step(minibatch, lr_optim, lr_optim)
        if epoch % epe == 0:
            rx_v, data_v = generate_data(N_valid, M, amps, SNR, h_channel, sps, device, P, rng=rng)
            q_v, _, _ = eq.forward(rx_v)
            shift = awgn_find_shift(q_v, data_v, 21, amp_levels)
            ser, _ = awgn_ser_q(q_v[:, 11 + shift:-11], data_v[:, 11:-11 - shift])
            SER_valid[epoch // epe] = ser
            if verbose:
                print(epoch, loss.item(), shift, '\t\t\t\t\t\tSER = ', SER_valid[epoch // epe].item())
    return SER_valid


# -------------------------------------------------------------------------------------------------
# AWGN single-polarisation CMA baseline (AWGN_channel/func_CMA_MQAM_shaping.py:201-256)
# -------------------------------------------------------------------------------------------------
def processing_cma_awgn(mod, sps, SNR, nu, M_est, lr_optim, N_valid, N_train, num_epochs, epe, channel, *, device=None, rng=None,
                        verbose=True, datagen=None):
    """The reference's positional signature and return value (SER_valid float32 [num_epochs // epe]).  Per epoch one CMA pass over a
    fresh training frame; every `epe` epochs a validation frame: CMA without updates -> CPE (no unwrap) -> find_shift_symb -> SER_CMA.
    `datagen`: optional iterator of (rx (2,sps*N) float32, tx (2,N) float16) frames in the order the reference draws them (replay)."""
    from . import awgn_cma as cm
    device = _cuda_device(device)
    if verbose:
        print("We are using the following device for learning:", device)
    if channel not in ("h1", "h2"):
        raise KeyError(f"AWGN driver knows channels h1/h2, got {channel!r}")       # cm:205-208
    h_channel = upsampled_channel(channel, sps)
    M = (len(h_channel) - 1) // sps + 1
    amps, P, _, _ = awgn_constants(mod, nu, SNR)
    amp_levels = torch.tensor(amps, device=device, dtype=torch.float32)
    num_lev = int(amp_levels.numel())
    h_est = torch.zeros(2, M_est, device=device, dtype=torch.float32)              # cm:233-235
    h_est[0, M_est // 2] = 1.0
    SER_valid = torch.empty(num_epochs // epe, device=device, dtype=torch.float32)

    def frame(N):
        if datagen is not None:
            rx, tx = next(datagen)
            return (torch.as_tensor(rx, dtype=torch.float32).to(device).contiguous(), torch.as_tensor(tx, dtype=torch.float16).to(device).contiguous())
        return generate_data(N, M, amps, SNR, h_channel, sps, device, P, rng=rng)

    R = 1
    for epoch in range(num_epochs):
        rx_tensor, _ = frame(N_train)
        _, h_est, e = cm.CMA(rx_tensor, R, h_est, lr_optim, sps, True)
        if epoch % epe == 0:
            rx_v, data_v = frame(N_valid)
            out_v, h_est, _ = cm.CMA(rx_v, R, h_est, lr_optim, sps, False)
            out_cpe = cm.CPE(out_v)
            shift = int(cm.find_shift_symb(out_cpe, data_v, 21))
            SER_valid[epoch // epe] = cm.SER_CMA(out_cpe[:, 11 + shift:-11], data_v[:, 11:-11 - shift], sps, amp_levels, num_lev, device)
            if verbose:
                print(epoch, torch.mean(torch.abs(e)).item(), shift, '\t\t\t\t\t\tSER = ', SER_valid[epoch // epe].item())
    return SER_valid
