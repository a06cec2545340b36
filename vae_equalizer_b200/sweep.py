"""Sweep engine: many independent VAE-LE / VAE-flex runs of the reference's parameter sweep stepped TOGETHER on one GPU.

The reference's Eval_run_DP.py (lines 68-95) walks a 10-deep nest of loops and calls `processing()` once per cell; cells
are independent.  At the reference's batch_len = 100 one run cannot fill a B200 (one CTA's worth of work per step), so
here all cells that share (mod, sps, M_est, batch_len, frame length, flex_step) become ONE batched run set: per frame a
single persistent launch trains every cell's 100-990 sequential minibatches (vaeq_dp_train_frame_runs, one CTA per
cell), then each cell is aligned and scored with the same evaluation kernels as the single-run drivers.  Across GPUs the
cells are dealt round-robin (parallel.shard_cells), no data-path collective.

`sweep_vae_dp` returns the same three result tensors as `processing()` with a leading cell dimension.

The AWGN single-polarisation VAE-LE (AWGN_channel/func_VAELE_MQAM_shaping.py, driven by Eval_run_shaping_vaele.py) has the same
structure: `sweep_vae_awgn` steps all cells of a set together (one launch trains every cell's epochs of a validation period,
one launch runs the validation forward, four score it, no host sync), `run_awgn_sweep` walks the reference's loops.
"""
from __future__ import annotations

import numpy as np
import torch

from . import shared_funcs as sfun
from .datagen import generate_frames_gpu
from .dp import DPEqualizerRuns
from .processing import N_CUT, _align, _cuda_device, _make_frame


def _cell(c, key):
    if key not in c:
        raise KeyError(f"sweep cell {c} lacks {key!r}")
    return c[key]


def sweep_vae_dp(cells, mod, sps, M_est, batch_len, N_frame_max, num_frames, flex_step=None, channel="h0", symb_rate=90e9,
                 tau_cd=-26e-24, tau_pmd=0.1e-12 * np.sqrt(1000), phiIQ=(0.0314, 0.0314), N_lrhalf=None, *, kind="VAE",
                 device=None, datagen="gpu", eval_every=1, eval_mode="batched", verbose=False, gmi=False):
    """Train and score R = len(cells) independent runs in lockstep.

    cells: list of dicts with per-cell values: SNR, nu, lr_optim, theta, theta_diff, and optionally seed.
    datagen: "numpy" (the reference's host generator, per cell), "gpu" (device generator, per cell: a cell's data depends on
    its own seed only, so a cell gives the same result alone or in any batch) or "gpu_batched" (one batched generation for all
    cells per frame, seeded by the first cell's seed: fastest).
    eval_mode: "batched" (default: vaeq_frame_eval_runs, all cells in 7 launches, no host sync) or "per_cell" (the single-run
    drivers' own sequence of calls per cell: find_shift -> roll -> cut -> SER; the two agree to the last error count).
    kind: "VAE" (func_VAELE_DP_MQAM_shaping.py: non-overlapping minibatches) or "VAEflex" (func_VAEflex_DP_MQAM_shaping.py:
    window batch_len advanced by flex_step).  eval_every: score every k-th frame (and the last); unscored frames hold NaN.
    gmi: also score GMI (shared_funcs.gmi_runs: the soft-demapper SER's symbols and hypothesis; eval_mode="batched" only).
    Returns (SER_valid (R,4,num_frames), Var_est (R,2,num_frames), var (R,2)), and GMI (R,2,num_frames) as a 4th tensor with gmi=True
    (NaN on unscored frames)."""
    _gmi_batched_only(gmi, eval_mode)
    device = _cuda_device(device)
    R = len(cells)
    if R == 0:
        raise ValueError("no cells")
    if kind not in ("VAE", "VAEflex"):
        raise KeyError(kind)
    N_lrhalf = num_frames if N_lrhalf is None else N_lrhalf
    phiIQ = np.asarray(phiIQ, dtype=np.complex64)
    init_cache, uniq, which = {}, [], []                                 # cells of a sweep share few (nu, SNR) pairs: sf.init once per pair
    for c in cells:
        key = (float(_cell(c, "nu")), float(_cell(c, "SNR")))
        if key not in init_cache:
            init_cache[key] = len(uniq)
            uniq.append(sfun.init(channel, mod, device, key[0], sps, M_est, key[1]))
        which.append(init_cache[key])
    consts = [uniq[i] for i in which]
    h_channel, amp_levels, amps, pol = consts[0][1], consts[0][3], consts[0][4], consts[0][5]
    num_lev = int(amp_levels.numel())
    widx = torch.tensor(which, dtype=torch.long)
    P_all = torch.stack([torch.as_tensor(k[2], dtype=torch.float32) for k in uniq])[widx]
    var_all = torch.stack([k[7].to(torch.float32).cpu() for k in uniq])[widx]
    nu_sc_all = torch.tensor([k[6] for k in uniq], dtype=torch.float32)[widx]
    pow_mean = [k[8] for k in consts]
    lr0 = torch.tensor([float(_cell(c, "lr_optim")) for c in cells], dtype=torch.float32).to(device)     # on the device: no copy / sync per frame
    theta = [float(c.get("theta", 0.0)) for c in cells]
    theta_diff = [float(c.get("theta_diff", 0.0)) for c in cells]
    seeds = [int(c.get("seed", i)) for i, c in enumerate(cells)]
    rngs = [np.random.default_rng(s) for s in seeds]
    eqr = DPEqualizerRuns(R, M_est, sps, amp_levels, P_all, var_all, nu_sc_all, device=device)
    amp_dev, var_dev, nu_dev = amp_levels.to(device, torch.float32), var_all.to(device), nu_sc_all.to(device)     # evaluation constants: on the device once

    if kind == "VAE":
        m_max = N_frame_max // batch_len
        N_frame = m_max * batch_len                                      # VAELE_DP:38-39
        stride, n_steps, keep_lo, keep_n, N_keep, kd = batch_len, m_max, 0, batch_len, N_frame, True
    else:
        N_frame = (N_frame_max // batch_len) * batch_len
        m_max = (N_frame - batch_len) // flex_step * flex_step           # VAEflex_DP:39
        stride, n_steps = flex_step, m_max // flex_step
        keep_lo, keep_hi = (batch_len - flex_step) // 2, (batch_len + flex_step) // 2
        keep_n, N_keep, kd = keep_hi - keep_lo, m_max, False

    SER_valid = torch.full((R, 4, num_frames), float("nan"), device=device, dtype=torch.float32)
    Var_est = torch.empty(R, pol, num_frames, device=device, dtype=torch.float32)
    GMI = torch.full((R, pol, num_frames), float("nan"), device=device, dtype=torch.float32) if gmi else None
    P_gmi = P_all.to(device) if gmi else None
    rx_all = None if datagen == "gpu_batched" else torch.empty(R, 2, 2, sps * N_frame, device=device, dtype=torch.float32)
    out_train = torch.empty(R, pol, 2 * num_lev, N_keep, device=device, dtype=torch.float32)
    out_const = torch.empty(R, pol, 2, N_keep, device=device, dtype=torch.float32)
    lr_w = lr0
    for frame in range(num_frames):
        if frame % N_lrhalf == 0 and frame != 0:
            lr_w = lr0 * 0.5                                             # group 0 only, not cumulative (VAELE_DP:45-46)
        tx_all = []
        if datagen == "gpu_batched":                                     # all cells' frames in one batched launch sequence
            if len(h_channel) != 1:
                raise sfun._lib.VaeqError("datagen='gpu_batched' implements the optical channel 'h0' only")
            if frame == 0:                                               # per-run parameters live on the device: no copy / sync per frame
                snr_dev = torch.tensor([float(c["SNR"]) for c in cells], dtype=torch.float32, device=device)
                theta_dev = torch.tensor(theta, dtype=torch.float64, device=device)
                theta_diff_dev = torch.tensor(theta_diff, dtype=torch.float64, device=device)
                P_dev = P_all.to(device)
            rx_b, tx_b, _ = generate_frames_gpu(N_frame, amps, snr_dev, P_dev, sps, theta_dev.to(torch.float32), device,
                                                seeds[0] * 100003 + frame, symb_rate=symb_rate, tau_cd=tau_cd, tau_pmd=tau_pmd, phiIQ=phiIQ)
            rx_all = rx_b
            if eval_mode != "batched":
                tx_all = [tx_b[r] if kind == "VAE" else tx_b[r][:, :, batch_len // 2:m_max + batch_len // 2] for r in range(R)]
            theta_dev = theta_dev + theta_diff_dev                       # VAELE_DP:47 theta drift per frame
        else:
            for r in range(R):
                rx, tx, _ = _make_frame(datagen, N_frame, amps, cells[r]["SNR"], h_channel, consts[r][2], pol, symb_rate, sps, tau_cd,
                                        tau_pmd, phiIQ, theta[r], device, rngs[r], seeds[r] * 100003 + frame)
                rx_all[r].copy_(rx)
                tx_all.append(tx if kind == "VAE" else tx[:, :, batch_len // 2:m_max + batch_len // 2])     # VAEflex_DP:51
                theta[r] += theta_diff[r]
        loss_steps, var_steps = eqr.train_frame(rx_all, batch_len, stride, n_steps, lr_w, lr0, out_train, out_const, keep_lo, keep_n,
                                                keep_lo_in_dst=kd)
        Var_est[:, :, frame] = var_steps.mean(dim=2)
        if frame % eval_every and frame != num_frames - 1:
            continue
        if eval_mode == "batched":
            if datagen == "gpu_batched":
                tx_b4 = tx_b if kind == "VAE" else tx_b[:, :, :, batch_len // 2:m_max + batch_len // 2]
            else:
                tx_b4 = torch.stack(tx_all)
            seg_len = batch_len if kind == "VAE" else 0
            ser, al, counts = sfun.frame_eval_runs(out_train, out_const, tx_b4, amp_dev, var_dev, nu_dev, seg_len, n_cut=N_CUT,
                                                   return_counts=True)
            SER_valid[:, :, frame] = ser
            if gmi:
                GMI[:, :, frame] = sfun.gmi_runs(out_train, tx_b4, P_gmi, al, counts, seg_len, n_cut=N_CUT)
            if verbose:
                print(frame, "loss", loss_steps[:, -1].tolist(), "SER", SER_valid[:, :, frame].tolist())
            continue
        # pass 1: both shift searches of every cell, ONE host sync for all of them
        found = [(sfun._find_shift(out_train[r], None, tx_all[r], 21, amp_levels, False, sync=False),
                  sfun._find_shift(None, out_const[r], tx_all[r], 21, None, False, sync=False)) for r in range(R)]
        shifts = torch.stack([torch.cat((a[0].to(torch.int32), a[1], b[0].to(torch.int32), b[1])) for a, b in found]).cpu().tolist()
        # pass 2: align and score (no sync)
        for r in range(R):
            sq, rq, so, ro = shifts[r][0:2], shifts[r][2], shifts[r][3:5], shifts[r][5]
            SER_valid[r, 2:, frame] = _score(kind, "q", _align(out_train[r].clone(), sq, rq), tx_all[r], sq, batch_len, m_max, pol,
                                             num_lev, amp_levels, consts[r])
            SER_valid[r, :2, frame] = _score(kind, "c", _align(out_const[r].clone(), so, ro), tx_all[r], so, batch_len, m_max, pol,
                                             num_lev, amp_levels, consts[r])
        if verbose:
            snr_db = 10 * torch.log10(torch.tensor(pow_mean, device=device) / var_steps.mean(dim=(1, 2)))
            print(frame, "loss", loss_steps[:, -1].tolist(), "SNR_est", snr_db.tolist(), "SER", SER_valid[:, :, frame].tolist())
    if gmi:
        return SER_valid, Var_est, var_all.to(device), GMI
    return SER_valid, Var_est, var_all.to(device)


def _gmi_batched_only(gmi, eval_mode):
    if gmi and eval_mode != "batched":
        raise ValueError(f"gmi=True needs eval_mode='batched' (GMI is scored from the batched evaluation's alignment and counts), got "
                         f"{eval_mode!r}")


def sweep_cma_dp(cells, mod, sps, M_est, batch_len, N_train_max, num_frames, flex_step=None, channel="h0", symb_rate=90e9,
                 tau_cd=-26e-24, tau_pmd=0.1e-12 * np.sqrt(1000), phiIQ=(0.0314, 0.0314), N_lrhalf=None, *, kind="CMA", device=None,
                 datagen="gpu", eval_mode="batched", verbose=False, gmi=False):
    """The CMA / CMAbatch / CMAflex drivers (func_CMA_DP_MQAM_shaping.py:16-56 and siblings) for R = len(cells) independent cells
    in lockstep.  The tap recurrence of a cell is sequential in the symbols, but cells are independent: per frame ONE equalizer
    launch sequence covers all cells that share lr_optim (vaeq_cma n_runs: one warp / one CTA per cell) and ONE batched CPE
    (vaeq_cpe_runs).  The evaluation (CMA_DP:39-52) is batched as well (eval_mode="batched": estimator from the CPE output ->
    aligned, partially rescaled copy -> soft_dec -> estimator from q, 4 calls and no host sync for all cells) or replays the single-run
    drivers' call sequence per cell (eval_mode="per_cell", two host syncs per frame); both give the same error counts.  A cell gives the same SER alone (processing_cma*_dp) or in any batch when
    datagen="gpu" (its data depends on its own seed only); datagen="gpu_batched" generates all cells in one call (fastest).
    gmi: also score GMI of the soft-demapper posteriors q the SER is taken from (shared_funcs.gmi_runs; eval_mode="batched" only).
    Returns (SER_valid (R,4,num_frames), Var_est zeros (R,2,num_frames), var (R,2)), and GMI (R,2,num_frames) as a 4th tensor with gmi=True."""
    from .processing import _make_frame
    _gmi_batched_only(gmi, eval_mode)
    device = _cuda_device(device)
    R = len(cells)
    if R == 0:
        raise ValueError("no cells")
    mode = {"CMA": 0, "CMAbatch": 1, "CMAflex": 2}[kind]
    N_lrhalf = num_frames if N_lrhalf is None else N_lrhalf
    phiIQ = np.asarray(phiIQ, dtype=np.complex64)
    init_cache, consts = {}, []
    for c in cells:
        key = (float(_cell(c, "nu")), float(_cell(c, "SNR")))
        if key not in init_cache:
            init_cache[key] = sfun.init(channel, mod, device, key[0], sps, M_est, key[1])
        consts.append(init_cache[key])
    h_channel, amp_levels, amps, pol = consts[0][1], consts[0][3], consts[0][4], consts[0][5]
    lrs = [float(_cell(c, "lr_optim")) for c in cells]
    lr_groups = {}
    for r, lr in enumerate(lrs):                                         # vaeq_cma takes one lr per call: one sub-batch per distinct lr
        lr_groups.setdefault(lr, []).append(r)
    theta = [float(c.get("theta", 0.0)) for c in cells]
    theta_diff = [float(c.get("theta_diff", 0.0)) for c in cells]
    seeds = [int(c.get("seed", i)) for i, c in enumerate(cells)]
    rngs = [np.random.default_rng(s) for s in seeds]
    h_est = consts[0][0].detach().to(device, torch.float32).unsqueeze(0).repeat(R, 1, 1, 1, 1).contiguous()      # Dirac init per cell (sf:583-585)
    SER_valid = torch.empty(R, 4, num_frames, device=device, dtype=torch.float32)
    Var_est = torch.zeros(R, pol, num_frames, device=device, dtype=torch.float32)
    var_all = torch.stack([k[7].to(device, torch.float32) for k in consts])
    nu_all = torch.tensor([float(k[6]) for k in consts], dtype=torch.float32, device=device)
    GMI = torch.full((R, pol, num_frames), float("nan"), device=device, dtype=torch.float32) if gmi else None
    P_gmi = torch.stack([torch.as_tensor(k[2], dtype=torch.float32) for k in consts]).to(device) if gmi else None
    lr_scale = 1.0
    for frame in range(num_frames):
        if frame % N_lrhalf == 0 and frame != 0:
            lr_scale *= 0.5                                              # cumulative (CMA_DP:31-32)
        if datagen == "gpu_batched":
            if len(h_channel) != 1:
                raise sfun._lib.VaeqError("datagen='gpu_batched' implements the optical channel 'h0' only")
            if frame == 0:                                               # per-run generator parameters live on the device
                P_dev = torch.stack([torch.as_tensor(k[2], dtype=torch.float32) for k in consts]).to(device)
                snr_dev = torch.tensor([float(c["SNR"]) for c in cells], dtype=torch.float32, device=device)
                theta_dev = torch.tensor(theta, dtype=torch.float64, device=device)
                theta_diff_dev = torch.tensor(theta_diff, dtype=torch.float64, device=device)
            rx_all, tx_all, _ = generate_frames_gpu(N_train_max, amps, snr_dev, P_dev, sps, theta_dev.to(torch.float32), device,
                                                    seeds[0] * 100003 + frame, symb_rate=symb_rate, tau_cd=tau_cd, tau_pmd=tau_pmd, phiIQ=phiIQ)
            theta_dev = theta_dev + theta_diff_dev
        else:
            fr = [_make_frame(datagen, N_train_max, amps, cells[r]["SNR"], h_channel, consts[r][2], pol, symb_rate, sps, tau_cd, tau_pmd,
                              phiIQ, theta[r], device, rngs[r], seeds[r] * 100003 + frame) for r in range(R)]
            rx_all, tx_all = torch.stack([f[0] for f in fr]), torch.stack([f[1] for f in fr])
        theta = [t + d for t, d in zip(theta, theta_diff)]
        out_all = torch.empty(R, 2, 2, rx_all.shape[-1] // sps, device=device, dtype=torch.float32)
        for lr, members in lr_groups.items():
            whole = len(members) == R
            rx_g = rx_all if whole else rx_all[members].contiguous()
            h_g = h_est if whole else h_est[members].contiguous()
            out_g, h_g, _ = sfun._cma(mode, rx_g, 1, h_g, lr * lr_scale, batch_len, flex_step or 0, sps, True)
            if whole:
                out_all = out_g
            else:
                out_all[members] = out_g
                h_est[members] = h_g
        out_c = sfun.CPE(out_all[:, :, :, N_CUT:-N_CUT])                 # carrier phase estimation, all cells  (CMA_DP:39)
        tx_c = tx_all[:, :, :, N_CUT:-N_CUT]
        if eval_mode == "batched":
            # CMA_DP:41-46: shift search on the CPE output, alignment as index arithmetic, SER from the constellation; the factor g of sf:242 comes back per cell
            ser_c, al, g = sfun.frame_eval_runs(None, out_c, tx_c, amp_levels, var_all, nu_all, 0, which=2, return_scale=True)
            # CMA_DP:44-48: soft_dec sees the aligned copy with the evaluated slice rescaled in place
            q_all = sfun.soft_dec_runs(sfun.cma_align_rescale(out_c, al, g), var_all, amp_levels, nu_all)
            ser_q, al_q, counts_q = sfun.frame_eval_runs(q_all, None, tx_c, amp_levels, var_all, nu_all, 0, which=1, return_counts=True)  # CMA_DP:49-52
            SER_valid[:, :2, frame] = ser_c[:, :2]
            SER_valid[:, 2:, frame] = ser_q[:, 2:]
            if gmi:
                GMI[:, :, frame] = sfun.gmi_runs(q_all, tx_c, P_gmi, al_q, counts_q, 0)
            if verbose:
                print(frame, "SER", SER_valid[:, :, frame].tolist())
            continue
        # evaluation, CMA_DP:41-52: the single-run sequence of calls per cell; shifts of all cells read back together
        f1 = [sfun._find_shift(None, out_c[r], tx_c[r], 21, None, False, sync=False) for r in range(R)]
        s1 = torch.stack([torch.cat((a.to(torch.int32), b)) for a, b in f1]).cpu().tolist()
        q_al, f2 = [], []
        for r in range(R):
            sh, rr = s1[r][0:2], s1[r][2]
            oc = _align(out_c[r], sh, rr)
            tail = 11 + max(abs(sh[0]), abs(sh[1]))
            # a VIEW is passed on purpose: the in-place rescale (sf:242) must be visible to soft_dec below (CMA_DP:44,48)
            SER_valid[r, :2, frame] = sfun.SER_constell_shaping(oc[:, :, 11:-tail], tx_c[r][:, :, 11:-tail], amp_levels, consts[r][6], consts[r][7])
            q = sfun.soft_dec(oc, consts[r][7], amp_levels, consts[r][6])
            q_al.append(q)
            f2.append(sfun._find_shift(q, None, tx_c[r], 21, amp_levels, False, sync=False))
        s2 = torch.stack([torch.cat((a.to(torch.int32), b)) for a, b in f2]).cpu().tolist()
        for r in range(R):
            sh, rr = s2[r][0:2], s2[r][2]
            qa = _align(q_al[r], sh, rr)
            tail = 11 + max(abs(sh[0]), abs(sh[1]))
            SER_valid[r, 2:, frame] = sfun.SER_IQflip(qa[:, :, 11:-tail], tx_c[r][:, :, 11:-tail])
        if verbose:
            print(frame, "SER", SER_valid[:, :, frame].tolist())
    if gmi:
        return SER_valid, Var_est, var_all, GMI
    return SER_valid, Var_est, var_all


def _score(kind, what, aligned, tx, sh, batch_len, m_max, pol, num_lev, amp_levels, const):
    """Cut the edges like the single-run drivers (VAELE_DP:73-89 / VAEflex_DP:74-84) and run the SER estimator."""
    tail = 11 + max(abs(sh[0]), abs(sh[1]))
    if kind == "VAE":
        keep = batch_len - sh[0] - N_CUT
        rows = aligned.shape[1]
        a = aligned.reshape(pol, rows, m_max, batch_len)[:, :, :, :keep].reshape(pol, rows, -1)
        d = tx.reshape(pol, 2, m_max, batch_len)[:, :, :, :keep].reshape(pol, 2, -1)
    else:
        a, d = aligned, tx
    a, d = a[:, :, 11:-tail], d[:, :, 11:-tail]
    if what == "q":
        return sfun.SER_IQflip(a, d)
    return sfun.SER_constell_shaping(a.detach().clone(), d, amp_levels, const[6], const[7])


def sweep_vae_dp_sharded(cells, *args, rank=0, world=1, group=None, **kw):
    """Round-robin the cells over the ranks (one process per GPU), run each share as one batched run set, and reassemble
    (SER_valid, Var_est, var) -- plus GMI with gmi=True -- for ALL cells on rank 0 (None elsewhere).  No data-path collective."""
    from .parallel import gather_cell_results, shard_cells
    mine = shard_cells(cells, rank, world)
    num_frames = args[5] if len(args) > 5 else kw["num_frames"]
    dev = _cuda_device(kw.get("device"))
    gmi = kw.get("gmi", False)
    if mine:
        res = sweep_vae_dp([c for _, c in mine], *args, **kw)
        ser, ve, var = res[:3]
    loc_ser = {i: ser[k] for k, (i, _) in enumerate(mine)} if mine else {}
    loc_ve = {i: ve[k] for k, (i, _) in enumerate(mine)} if mine else {}
    loc_var = {i: var[k] for k, (i, _) in enumerate(mine)} if mine else {}
    n = len(cells)
    # NaN marks unscored frames: carry it through the sum-based gather with a mask
    ser_g = gather_cell_results({i: torch.nan_to_num(t, nan=-1.0) for i, t in loc_ser.items()}, n, (4, num_frames), rank, world, group, dev)
    ve_g = gather_cell_results(loc_ve, n, (2, num_frames), rank, world, group, dev)
    var_g = gather_cell_results(loc_var, n, (2,), rank, world, group, dev)
    if gmi:                                                          # a collective: every rank takes part, before any rank returns
        loc_g = {i: res[3][k] for k, (i, _) in enumerate(mine)} if mine else {}
        gmi_g = _gather_with_nan(loc_g, n, (2, num_frames), rank, world, group, dev)
    if rank != 0:
        return None
    ser_g = torch.where(ser_g < 0, torch.full_like(ser_g, float("nan")), ser_g)
    if gmi:
        return ser_g, ve_g, var_g, gmi_g
    return ser_g, ve_g, var_g


def _gather_with_nan(local, n_cells, shape, rank, world, group, dev):
    """parallel.gather_cell_results for values of any sign with NaN entries (GMI can be negative, so NaN cannot be carried as a negative
    sentinel): the values with NaN as 0 and a NaN mask travel in one block.  (n_cells, *shape) on rank 0, None elsewhere."""
    from .parallel import gather_cell_results
    packed = {i: torch.stack((torch.where(torch.isnan(t), torch.zeros_like(t), t), torch.isnan(t).to(t.dtype))) for i, t in local.items()}
    g = gather_cell_results(packed, n_cells, (2,) + tuple(shape), rank, world, group, dev)
    if g is None:
        return None
    return torch.where(g[:, 1] > 0, torch.full_like(g[:, 0], float("nan")), g[:, 0])


# -------------------------------------------------------------------------------------------------
# The whole sweep of Eval_run_DP.py (lines 17-114): same parameter lists in, same result arrays and .mat schema out
# -------------------------------------------------------------------------------------------------
AXES = ("SNR", "symb_rate", "nu", "theta_diff", "M", "lr_optim", "batch_len", "flex_step", "theta")   # index order of SER[...] (RUN_DP:52,86)


def run_dp_sweep(mod="64-QAM", sps=2, loss_type="VAE", channel="h0", nu_vec=(0,), symb_rate_vec=(90e9,), theta_vec=(np.pi / 10,),
                 theta_diff_vec=(0.06 * np.pi,), SNR_vec=(23,), M_vec=(25,), batch_len_vec=(100,), flex_step_vec=(10,),
                 lr_optim_vec=(2.5e-3, 2e-3, 3e-3), iter=5, N_lrhalf=170, num_frames=170, N_frame_max=10000,
                 tau_pmd=0.1e-12 * np.sqrt(1000), tau_cd=-26e-24, phiIQ=(0.0314, 0.0314), *, device=None, datagen="gpu_batched",
                 eval_every=1, rank=0, world=1, group=None, runner=None, verbose=False, checkpoint_dir=None, gmi=False):
    """Eval_run_DP.py's ten nested loops (RUN_DP:68-95) as batched run sets.  Cells that share (M, batch_len, flex_step, symb_rate)
    train in the same persistent launch; with world > 1 every rank takes a round-robin share of each set.  Returns the
    reference's result arrays on rank 0 (None elsewhere):
        SER (4, SNR, symb_rate, nu, theta_diff, M, lr, batch_len, flex_step, theta, iter, num_frames), Var_est (2, ...), var_real (2, ..., 1)
    loss_type 'VAE' / 'VAEflex' use the batched VAE engine (sweep_vae_dp), the CMA variants the batched CMA engine (sweep_cma_dp: a cell's tap
    recurrence is sequential in the symbols, the cells of a set run side by side).
    checkpoint_dir: rank 0 writes each finished run set there (one .npz per set, keyed by the set's parameters); a restarted sweep
    loads what it finds instead of recomputing (the reference only saves once, at the very end: RUN_DP:99-114).
    gmi=True: also GMI (2, SNR, ..., iter, num_frames), shaped like Var_est, as a 4th result (sweep_vae_dp / sweep_cma_dp with gmi=True;
    the runner hook is then called with gmi=True).  Its checkpoints hold the GMI and are never mixed up with those of gmi=False."""
    vecs = dict(SNR=list(SNR_vec), symb_rate=list(symb_rate_vec), nu=list(nu_vec), theta_diff=list(theta_diff_vec), M=list(M_vec),
                lr_optim=list(lr_optim_vec), batch_len=list(batch_len_vec), flex_step=list(flex_step_vec), theta=list(theta_vec))
    shape = tuple(len(vecs[a]) for a in AXES) + (iter,)
    dev = torch.device("cpu") if runner is not None and device is None else _cuda_device(device)
    SER = torch.full((4,) + shape + (num_frames,), float("nan"), dtype=torch.float32, device=dev)
    Var_est = torch.zeros((2,) + shape + (num_frames,), dtype=torch.float32, device=dev)
    var_real = torch.zeros((2,) + shape + (1,), dtype=torch.float32, device=dev)
    GMI = torch.full((2,) + shape + (num_frames,), float("nan"), dtype=torch.float32, device=dev) if gmi else None
    gkw = dict(gmi=True) if gmi else {}                              # gmi=False: every call, name and signature exactly as without GMI
    groups = {}
    for idx in np.ndindex(*shape):
        c = {a: vecs[a][i] for a, i in zip(AXES, idx[:-1])}
        c["seed"] = int(np.ravel_multi_index(idx, shape))            # one realisation per (cell, iteration), reproducible
        groups.setdefault((c["M"], c["batch_len"], c["flex_step"], c["symb_rate"]), []).append((idx, c))
    for (M, batch_len, flex_step, symb_rate), members in groups.items():
        cells = [c for _, c in members]
        common = (mod, sps, M, batch_len, N_frame_max, num_frames)
        ck, sig = None, None
        if checkpoint_dir is not None:
            import os
            os.makedirs(checkpoint_dir, exist_ok=True)
            # everything the set's results depend on: the file is only reused by a sweep with the same cells and settings
            sig = _set_signature(loss_type=loss_type, mod=mod, sps=sps, channel=channel, M=M, batch_len=batch_len, flex_step=flex_step,
                                 symb_rate=symb_rate, N_frame_max=N_frame_max, num_frames=num_frames, N_lrhalf=N_lrhalf, tau_cd=tau_cd,
                                 tau_pmd=tau_pmd, phiIQ=list(phiIQ), datagen=datagen, eval_every=eval_every,
                                 cells=[sorted(c.items()) for c in cells], **gkw)
            ck = os.path.join(checkpoint_dir, f"{loss_type}_{mod}_M{M}_B{batch_len}_F{flex_step}_R{symb_rate:g}_n{len(cells)}_f{num_frames}"
                                              f"_{sig[:12]}.npz")
            have = 0
            if rank == 0 and os.path.exists(ck):
                z = np.load(ck)
                if "signature" in z.files and str(z["signature"]) == sig and (not gmi or "gmi" in z.files):
                    have = 1
                    for k, (idx, _) in enumerate(members):
                        SER[(slice(None),) + idx] = torch.from_numpy(z["ser"][k]).to(dev)
                        Var_est[(slice(None),) + idx] = torch.from_numpy(z["ve"][k]).to(dev)
                        var_real[(slice(None),) + idx + (0,)] = torch.from_numpy(z["var"][k]).to(dev)
                        if gmi:
                            GMI[(slice(None),) + idx] = torch.from_numpy(z["gmi"][k]).to(dev)
            if _bcast_flag(have, rank, world, group, dev):           # rank 0 decides (the directory need not be shared); all ranks follow
                continue
        kw = dict(flex_step=flex_step, channel=channel, symb_rate=symb_rate, tau_cd=tau_cd, tau_pmd=tau_pmd, phiIQ=phiIQ, N_lrhalf=N_lrhalf)
        if runner is not None:                                       # test hook: stands for sweep_vae_dp_sharded
            res = runner(cells, *common, **kw, **gkw)
        elif loss_type in ("VAE", "VAEflex"):
            res = sweep_vae_dp_sharded(cells, *common, kind=loss_type, device=dev, datagen=datagen, eval_every=eval_every,
                                       verbose=verbose, rank=rank, world=world, group=group, **kw, **gkw)
        else:
            res = _cma_cells(loss_type, cells, common, kw, dev, rank, world, group, num_frames, datagen=datagen, gmi=gmi)
        if res is None:
            continue
        ser, ve, var = res[:3]
        if ck is not None and rank == 0:
            extra = dict(gmi=res[3].cpu().numpy()) if gmi else {}
            np.savez(ck, ser=ser.cpu().numpy(), ve=ve.cpu().numpy(), var=var.cpu().numpy(), signature=np.array(sig), **extra)
        for k, (idx, _) in enumerate(members):
            SER[(slice(None),) + idx] = ser[k].to(dev)
            Var_est[(slice(None),) + idx] = ve[k].to(dev)
            var_real[(slice(None),) + idx + (0,)] = var[k].to(dev)
            if gmi:
                GMI[(slice(None),) + idx] = res[3][k].to(dev)
    if rank != 0:
        return None
    if gmi:
        return SER, Var_est, var_real, GMI
    return SER, Var_est, var_real


def _set_signature(**params):
    """sha256 of a run set's full parameter dict (floats by repr, so 2.5e-3 and 0.0025 agree)."""
    import hashlib
    import json

    def norm(x):
        if isinstance(x, (list, tuple)):
            return [norm(v) for v in x]
        if isinstance(x, (float, np.floating)):
            return repr(float(x))
        if isinstance(x, (int, np.integer)):
            return int(x)
        return x
    return hashlib.sha256(json.dumps({k: norm(v) for k, v in sorted(params.items())}, sort_keys=True).encode()).hexdigest()


def _bcast_flag(flag, rank, world, group, dev):
    """rank 0's decision on every rank (one tiny broadcast; a no-op for a single process)."""
    import torch.distributed as dist
    if world <= 1 or not (dist.is_available() and dist.is_initialized()):
        return bool(flag)
    on = dev if dist.get_backend(group) == "nccl" else torch.device("cpu")
    t = torch.tensor([int(flag)], dtype=torch.int32, device=on)
    dist.broadcast(t, src=dist.get_global_rank(group, 0) if group is not None else 0, group=group)
    return bool(int(t.item()))


def _cma_cells(loss_type, cells, common, kw, dev, rank, world, group, num_frames, datagen="gpu", gmi=False):
    """This rank's share of the cells of a CMA-family run set through the batched engine (sweep_cma_dp), gathered on rank 0."""
    from .parallel import gather_cell_results, shard_cells
    mod, sps, M, batch_len, N_frame_max, nf = common
    mine = shard_cells(cells, rank, world)
    loc_s, loc_v, loc_r, loc_g = {}, {}, {}, {}
    if mine:
        res = sweep_cma_dp([c for _, c in mine], mod, sps, M, batch_len, N_frame_max, nf, kw["flex_step"], kw["channel"], kw["symb_rate"],
                           kw["tau_cd"], kw["tau_pmd"], kw["phiIQ"], kw["N_lrhalf"], kind=loss_type, device=dev, datagen=datagen,
                           **(dict(gmi=True) if gmi else {}))
        s, v, r = res[:3]
        for k, (i, _) in enumerate(mine):
            loc_s[i], loc_v[i], loc_r[i] = s[k], v[k], r[k]
            if gmi:
                loc_g[i] = res[3][k]
    n = len(cells)
    out = (gather_cell_results(loc_s, n, (4, num_frames), rank, world, group, dev), gather_cell_results(loc_v, n, (2, num_frames), rank, world, group, dev),
           gather_cell_results(loc_r, n, (2,), rank, world, group, dev))
    if gmi:
        out = out + (_gather_with_nan(loc_g, n, (2, num_frames), rank, world, group, dev),)
    return out if rank == 0 else None


def save_mat(path, SER, Var_est, var_real, *, SNR_vec, nu_vec, theta_diff_vec, theta_vec, M_vec, lr_optim_vec, batch_len_vec, symb_rate_vec,
             flex_step_vec, GMI=None):
    """The .mat file of Eval_run_DP.py:99-114: one struct 'dict' with the result arrays and the parameter lists under the same keys.
    GMI (run_dp_sweep(..., gmi=True)), when given, is stored under the extra key 'GMI'; without it the file is exactly the reference's."""
    from scipy import io
    d = {"SER": SER.cpu().numpy(), "Var_est": Var_est.cpu().numpy(), "var_real": var_real.cpu().numpy(),
         "SNR": list(SNR_vec), "nu": list(nu_vec), "theta_diff": list(theta_diff_vec), "theta": list(theta_vec),
         "M": list(M_vec), "lr": list(lr_optim_vec), "batch_len": list(batch_len_vec),
         "symb_rate": list(symb_rate_vec), "symb_step": list(flex_step_vec)}
    if GMI is not None:
        d["GMI"] = GMI.cpu().numpy()
    io.savemat(path, {"dict": d})


# -------------------------------------------------------------------------------------------------
# AWGN single-polarisation VAE-LE (AWGN_channel/func_VAELE_MQAM_shaping.py:235-324, Eval_run_shaping_vaele.py)
# -------------------------------------------------------------------------------------------------
AWGN_VALID_FRAME0 = 1 << 20          # device generator: frame indices of the validation frames (training frames are the epoch index)


def _awgn_check(num_epochs, epe, channel, device):
    if channel not in ("h1", "h2"):
        raise KeyError(f"AWGN driver knows channels h1/h2, got {channel!r}")       # :239-242
    if epe < 1 or num_epochs % epe != 0:
        raise ValueError(f"num_epochs={num_epochs} must be a multiple of epe={epe} (the single-run driver fails on its last validation)")
    dev = _cuda_device(device)
    if dev.type != "cuda":
        raise sfun._lib.VaeqError(f"device {dev}: the AWGN sweep runs on CUDA devices only, there is no CPU path")
    return dev


def _awgn_host_frames(N, F, M, amps, snr, h_channel, sps, dev, P, rngs):
    """F frames of N symbols per run from the host generator, run r drawing from rngs[r] in frame order: rx (R, F, 2, sps*N), tx (R, F, 2, N)."""
    from .awgn import generate_data
    R = len(rngs)
    rx = torch.empty(R, F, 2, sps * N, dtype=torch.float32, device=dev)
    tx = torch.empty(R, F, 2, N, dtype=torch.float16, device=dev)
    for r in range(R):
        for f in range(F):
            rx[r, f], tx[r, f] = generate_data(N, M, amps, snr[r], h_channel, sps, dev, P[r], rng=rngs[r])
    return rx, tx


def sweep_vae_awgn(cells, mod, sps, M_est, batch_len, N_valid, N_train, num_epochs, epe, channel, *, device=None, datagen="gpu", verbose=False,
                   gmi=False):
    """processing_vaele_awgn (:235-324) for R = len(cells) independent cells in lockstep.

    cells: dicts with SNR, nu, lr_optim and optionally seed (default: the cell's index).  Returns SER_valid (R, num_epochs // epe), row k
    being what the single-run driver returns for cell k.  The driver validates after epoch e when e % epe == 0, so a validation period
    is ONE launch training every cell's epochs since the last validation, the validation forward of all cells, and the batched scoring.
    The epe - 1 epochs after the last validation do not change the result and are not trained.
    datagen="gpu": every cell's frames from the device generator, keyed by the cell's seed (a cell gives the same SER alone or in any
    batch); "numpy": each cell's frames from np.random.default_rng(seed) in exactly the order processing_vaele_awgn(rng=...) draws them.
    gmi=True: returns (SER_valid, GMI_valid (R, num_epochs // epe)), GMI scored on the SER's symbols under its best rotation
    (awgn.awgn_gmi_runs)."""
    from .awgn import AWGNEqualizerRuns, awgn_eval_runs, awgn_gmi_runs, generate_frames_awgn_gpu
    from .constants import awgn_constants, upsampled_channel
    dev = _awgn_check(num_epochs, epe, channel, device)
    if datagen not in ("gpu", "numpy"):
        raise ValueError(f"datagen={datagen!r}: 'gpu' or 'numpy'")
    R = len(cells)
    if R == 0:
        raise ValueError("no cells")
    if N_train // batch_len < 1:
        raise ValueError(f"N_train={N_train} holds no minibatch of batch_len={batch_len}")
    h_channel = upsampled_channel(channel, sps)
    M = (len(h_channel) - 1) // sps + 1
    consts = [awgn_constants(mod, float(_cell(c, "nu")), float(_cell(c, "SNR"))) for c in cells]
    amps = consts[0][0]
    amp_levels = torch.tensor(amps, device=dev, dtype=torch.float32)
    P = torch.tensor(np.stack([k[1] for k in consts]), dtype=torch.float32)
    eqr = AWGNEqualizerRuns(R, M_est, sps, amp_levels, P, [k[2] for k in consts], [k[3] for k in consts], device=dev)
    lr = torch.tensor([float(_cell(c, "lr_optim")) for c in cells], dtype=torch.float32, device=dev)
    seeds = [int(c.get("seed", i)) for i, c in enumerate(cells)]
    rngs = [np.random.default_rng(s) for s in seeds]
    snr = [float(c["SNR"]) for c in cells]
    n_val = num_epochs // epe
    SER_valid = torch.empty(R, n_val, device=dev, dtype=torch.float32)
    GMI_valid = torch.empty(R, n_val, device=dev, dtype=torch.float32) if gmi else None
    P_gmi = P.to(dev) if gmi else None

    def host_frames(N, F):
        return _awgn_host_frames(N, F, M, amps, snr, h_channel, sps, dev, [k[1] for k in consts], rngs)

    epoch = 0
    for k in range(n_val):
        n_ep = 1 if k == 0 else epe                                  # epochs epoch .. epoch + n_ep - 1, then validate (epoch % epe == 0)
        if datagen == "gpu":
            rx, _ = generate_frames_awgn_gpu(N_train, amps, snr, P, h_channel, sps, dev, seeds, frame0=epoch, n_frames=n_ep)
            rx_v, tx_v = generate_frames_awgn_gpu(N_valid, amps, snr, P, h_channel, sps, dev, seeds, frame0=AWGN_VALID_FRAME0 + k)
        else:
            rx, _ = host_frames(N_train, n_ep)
            rx_v, tx_v = host_frames(N_valid, 1)
        loss = eqr.train_frames(rx, lr, batch_len, N_train)
        epoch += n_ep
        q_v, _, _ = eqr.forward(rx_v[:, 0])
        shift, counts, ser = awgn_eval_runs(q_v, tx_v[:, 0], amp_levels)
        SER_valid[:, k] = ser
        if gmi:
            GMI_valid[:, k] = awgn_gmi_runs(q_v, tx_v[:, 0], P_gmi, shift, counts)
        if verbose:
            print(epoch - 1, "loss", loss[:, -1].tolist(), "shift", shift.tolist(), "SER", ser.tolist())
    if gmi:
        return SER_valid, GMI_valid
    return SER_valid


def sweep_vae_awgn_sharded(cells, *args, rank=0, world=1, group=None, **kw):
    """sweep_vae_awgn over a round-robin share of the cells per rank (one process per GPU); SER_valid of ALL cells on rank 0 (None
    elsewhere), with gmi=True the pair (SER_valid, GMI_valid).  No data-path collective."""
    from .parallel import gather_cell_results, shard_cells
    mine = shard_cells(cells, rank, world)
    num_epochs, epe = (args[6], args[7]) if len(args) > 7 else (kw["num_epochs"], kw["epe"])
    dev = _cuda_device(kw.get("device"))
    gmi = kw.get("gmi", False)
    loc, loc_g = {}, {}
    if mine:
        res = sweep_vae_awgn([c for _, c in mine], *args, **kw)
        ser = res[0] if gmi else res
        loc = {i: ser[k] for k, (i, _) in enumerate(mine)}
        if gmi:
            loc_g = {i: res[1][k] for k, (i, _) in enumerate(mine)}
    ser_g = gather_cell_results(loc, len(cells), (num_epochs // epe,), rank, world, group, dev)
    if not gmi:
        return ser_g
    gmi_g = _gather_with_nan(loc_g, len(cells), (num_epochs // epe,), rank, world, group, dev)
    return None if rank != 0 else (ser_g, gmi_g)


AWGN_AXES = ("batch_len", "lr_optim", "M", "SNR", "nu")           # loop order of Eval_run_shaping_vaele.py (RUN_AWGN:42-58), then iter


def run_awgn_sweep(mod="64-QAM", sps=2, channel="h1", N_train_vec=(350,), lr_optim_vec=(2e-3,), M_vec=(25,), SNR_vec=(12,), nu_vec=(0.0,),
                   iter=1, N_valid=15000, train_len=1200, num_epochs=500, epe=20, *, device=None, datagen="gpu", rank=0, world=1, group=None,
                   runner=None, verbose=False, checkpoint_dir=None, gmi=False):
    """Eval_run_shaping_vaele.py's loops (RUN_AWGN:42-58) as batched run sets.  As in the reference, the N_train_vec entries are the
    drivers' batch_len and train_len is their N_train (RUN_AWGN:53).  Cells that share (M, batch_len) train in the same launch; with
    world > 1 every rank takes a round-robin share of each set.  Returns on rank 0 (None elsewhere)
        SER (len(N_train_vec), len(lr_optim_vec), len(M_vec), len(SNR_vec), len(nu_vec), iter, num_epochs // epe) and the validation
        epochs (num_epochs // epe,).
    Cell (.., i) is seeded with its flat index.  checkpoint_dir: rank 0 stores every finished set (one .npz, keyed by the set's full
    parameters); a restarted sweep loads what it finds instead of recomputing.
    gmi=True: also GMI shaped like SER as a 3rd result (sweep_vae_awgn(..., gmi=True); the runner hook is then called with gmi=True and
    returns (SER_valid, GMI_valid)).  Its checkpoints hold the GMI and are never mixed up with those of gmi=False."""
    if channel not in ("h1", "h2"):
        raise KeyError(f"AWGN driver knows channels h1/h2, got {channel!r}")
    if epe < 1 or num_epochs % epe != 0:
        raise ValueError(f"num_epochs={num_epochs} must be a multiple of epe={epe}")
    gkw = dict(gmi=True) if gmi else {}                              # gmi=False: every call, name and signature exactly as without GMI
    vecs = dict(batch_len=list(N_train_vec), lr_optim=list(lr_optim_vec), M=list(M_vec), SNR=list(SNR_vec), nu=list(nu_vec))
    dev = torch.device("cpu") if runner is not None and device is None else _cuda_device(device)

    def signature(key, cells):
        M, batch_len = key
        return _set_signature(driver="VAELE_AWGN", mod=mod, sps=sps, channel=channel, M=M, batch_len=batch_len, N_valid=N_valid,
                              train_len=train_len, num_epochs=num_epochs, epe=epe, datagen=datagen, cells=[sorted(c.items()) for c in cells], **gkw)

    def file_name(key, cells, sig):
        M, batch_len = key
        return f"AWGN_{mod}_M{M}_B{batch_len}_n{len(cells)}_e{num_epochs}_{sig[:12]}.npz"

    def run_set(key, cells):
        M, batch_len = key
        args = (cells, mod, sps, M, batch_len, N_valid, train_len, num_epochs, epe, channel)
        if runner is not None:                                       # test hook: stands for sweep_vae_awgn_sharded
            return runner(*args, **gkw)
        return sweep_vae_awgn_sharded(*args, device=dev, datagen=datagen, verbose=verbose, rank=rank, world=world, group=group, **gkw)

    res = _walk_awgn_sets(AWGN_AXES, vecs, ("M", "batch_len"), iter, num_epochs // epe, dev, checkpoint_dir, rank, world, group, signature,
                          file_name, run_set, gmi=gmi)
    if rank != 0:
        return None
    if gmi:
        return res[0], np.arange(0, num_epochs, epe), res[1]
    return res, np.arange(0, num_epochs, epe)


def _walk_awgn_sets(axes, vecs, group_by, iter, n_val, dev, checkpoint_dir, rank, world, group, signature, file_name, run_set, gmi=False):
    """The cells of vecs[axes[0]] x ... x iter, seeded by their flat index, grouped into one run set per value of the `group_by` axes.
    Per set: with checkpoint_dir, rank 0 loads the set's file if its stored signature(key, cells) matches (all ranks then skip it);
    otherwise run_set(key, cells) gives SER_valid (n, n_val) on rank 0 (None elsewhere), which rank 0 stores under
    file_name(key, cells, sig).  Returns SER (shape of the cells, n_val).  gmi=True: run_set gives (SER_valid, GMI_valid), the files
    hold both and (SER, GMI) is returned."""
    import os
    shape = tuple(len(vecs[a]) for a in axes) + (iter,)
    SER = torch.full(shape + (n_val,), float("nan"), dtype=torch.float32, device=dev)
    GMI = torch.full(shape + (n_val,), float("nan"), dtype=torch.float32, device=dev) if gmi else None
    groups = {}
    for idx in np.ndindex(*shape):
        c = {a: vecs[a][i] for a, i in zip(axes, idx[:-1])}
        c["seed"] = int(np.ravel_multi_index(idx, shape))
        groups.setdefault(tuple(c[a] for a in group_by), []).append((idx, c))
    for key, members in groups.items():
        cells = [{k: c[k] for k in ("SNR", "nu", "lr_optim", "seed")} for _, c in members]
        ck, sig = None, None
        if checkpoint_dir is not None:
            os.makedirs(checkpoint_dir, exist_ok=True)
            sig = signature(key, cells)
            ck = os.path.join(checkpoint_dir, file_name(key, cells, sig))
            have = 0
            if rank == 0 and os.path.exists(ck):
                z = np.load(ck)
                if "signature" in z.files and str(z["signature"]) == sig and (not gmi or "gmi" in z.files):
                    have = 1
                    for k, (idx, _) in enumerate(members):
                        SER[idx] = torch.from_numpy(z["ser"][k]).to(dev)
                        if gmi:
                            GMI[idx] = torch.from_numpy(z["gmi"][k]).to(dev)
            if _bcast_flag(have, rank, world, group, dev):
                continue
        res = run_set(key, cells)
        if res is None:
            continue
        ser, g = res if gmi else (res, None)
        if ck is not None and rank == 0:
            extra = dict(gmi=g.cpu().numpy()) if gmi else {}
            np.savez(ck, ser=ser.cpu().numpy(), signature=np.array(sig), **extra)
        for k, (idx, _) in enumerate(members):
            SER[idx] = ser[k].to(dev)
            if gmi:
                GMI[idx] = g[k].to(dev)
    return (SER, GMI) if gmi else SER


# -------------------------------------------------------------------------------------------------
# AWGN single-polarisation CMA baseline (AWGN_channel/func_CMA_MQAM_shaping.py:201-256, `cm:`)
# -------------------------------------------------------------------------------------------------
def sweep_cma_awgn(cells, mod, sps, M_est, N_valid, N_train, num_epochs, epe, channel, *, device=None, datagen="gpu", verbose=False):
    """processing_cma_awgn (cm:201-256) for R = len(cells) independent cells in lockstep.

    cells: dicts with SNR, nu, lr_optim and optionally seed (default: the cell's index).  Returns SER_valid (R, num_epochs // epe), row k
    being what processing_cma_awgn returns for cell k, bit for bit.  A validation period is generation, ONE launch that runs every cell's
    CMA over its training frames since the last validation and then over its validation frame (awgn_cma.CMA_runs), one batched CPE and
    the batched scoring (awgn_cma.awgn_cma_eval_runs): no host sync.  The epe - 1 epochs after the last validation do not change the
    result and are not trained.
    datagen="gpu": frames from the device generator with the frame keys of sweep_vae_awgn (training frame = epoch index, validation
    frame k = AWGN_VALID_FRAME0 + k), so a cell with the same seed, N_train and N_valid sees the same frames in both sweeps and the two
    baselines are compared on identical data; a cell gives the same SER alone or in any batch.  "numpy": each cell's frames from
    np.random.default_rng(seed) in exactly the order processing_cma_awgn(rng=...) draws them.
    No GMI: the AWGN CMA driver makes no posteriors (it decides on the nearest level), so there is no q to score."""
    from . import awgn_cma as cm
    from .awgn import generate_frames_awgn_gpu
    from .constants import awgn_constants, upsampled_channel
    dev = _awgn_check(num_epochs, epe, channel, device)
    if datagen not in ("gpu", "numpy"):
        raise ValueError(f"datagen={datagen!r}: 'gpu' or 'numpy'")
    R = len(cells)
    if R == 0:
        raise ValueError("no cells")
    h_channel = upsampled_channel(channel, sps)
    M = (len(h_channel) - 1) // sps + 1
    consts = [awgn_constants(mod, float(_cell(c, "nu")), float(_cell(c, "SNR"))) for c in cells]
    amps = consts[0][0]
    amp_levels = torch.tensor(amps, device=dev, dtype=torch.float32)
    P = torch.tensor(np.stack([k[1] for k in consts]), dtype=torch.float32)
    lr = torch.tensor([float(_cell(c, "lr_optim")) for c in cells], dtype=torch.float32, device=dev)     # the fp32 value CMA() passes
    seeds = [int(c.get("seed", i)) for i, c in enumerate(cells)]
    rngs = [np.random.default_rng(s) for s in seeds]
    snr = [float(c["SNR"]) for c in cells]
    h = torch.zeros(R, 2, M_est, device=dev, dtype=torch.float32)         # cm:233-235
    h[:, 0, M_est // 2] = 1.0
    n_val = num_epochs // epe
    SER_valid = torch.empty(R, n_val, device=dev, dtype=torch.float32)
    epoch = 0
    for k in range(n_val):
        n_ep = 1 if k == 0 else epe                                  # epochs epoch .. epoch + n_ep - 1, then validate (epoch % epe == 0)
        if datagen == "gpu":
            rx, _ = generate_frames_awgn_gpu(N_train, amps, snr, P, h_channel, sps, dev, seeds, frame0=epoch, n_frames=n_ep)
            rx_v, tx_v = generate_frames_awgn_gpu(N_valid, amps, snr, P, h_channel, sps, dev, seeds, frame0=AWGN_VALID_FRAME0 + k)
        else:
            rx, _ = _awgn_host_frames(N_train, n_ep, M, amps, snr, h_channel, sps, dev, [c[1] for c in consts], rngs)
            rx_v, tx_v = _awgn_host_frames(N_valid, 1, M, amps, snr, h_channel, sps, dev, [c[1] for c in consts], rngs)
        out_v = cm.CMA_runs(rx, rx_v[:, 0], h, lr, sps)
        epoch += n_ep
        shift, _, ser = cm.awgn_cma_eval_runs(cm.CPE(out_v), tx_v[:, 0], amp_levels)
        SER_valid[:, k] = ser
        if verbose:
            print(epoch - 1, "shift", shift.tolist(), "SER", ser.tolist())
    return SER_valid


def sweep_cma_awgn_sharded(cells, *args, rank=0, world=1, group=None, **kw):
    """sweep_cma_awgn over a round-robin share of the cells per rank (one process per GPU); SER_valid of ALL cells on rank 0 (None
    elsewhere).  No data-path collective."""
    from .parallel import gather_cell_results, shard_cells
    mine = shard_cells(cells, rank, world)
    num_epochs, epe = (args[5], args[6]) if len(args) > 6 else (kw["num_epochs"], kw["epe"])
    dev = _cuda_device(kw.get("device"))
    loc = {}
    if mine:
        ser = sweep_cma_awgn([c for _, c in mine], *args, **kw)
        loc = {i: ser[k] for k, (i, _) in enumerate(mine)}
    return gather_cell_results(loc, len(cells), (num_epochs // epe,), rank, world, group, dev)


AWGN_CMA_AXES = ("lr_optim", "M", "SNR", "nu")                     # index order of run_awgn_cma_sweep's SER, then iter


def run_awgn_cma_sweep(mod="64-QAM", sps=2, channel="h1", lr_optim_vec=(5e-4,), M_vec=(25,), SNR_vec=(12,), nu_vec=(0.0,), iter=1, N_valid=15000,
                       N_train=1200, num_epochs=500, epe=20, *, device=None, datagen="gpu", rank=0, world=1, group=None, runner=None,
                       verbose=False, checkpoint_dir=None):
    """A sweep of the AWGN CMA baseline over lr_optim x M x SNR x nu x iter as batched run sets (sweep_cma_awgn_sharded), one set per M.
    The reference's sweep script for this driver is not part of this package: the axis order (that of run_awgn_sweep without its
    batch_len axis) and the defaults (N_valid, N_train, num_epochs and epe as run_awgn_sweep's) are this package's choice.  With
    world > 1 every rank takes a round-robin share of each set.  Returns on rank 0 (None elsewhere)
        SER (len(lr_optim_vec), len(M_vec), len(SNR_vec), len(nu_vec), iter, num_epochs // epe) and the validation epochs (num_epochs // epe,).
    Cell (.., i) is seeded with its flat index, as in run_awgn_sweep.  checkpoint_dir: rank 0 stores every finished set (one .npz named
    AWGNCMA_..., keyed by the set's full parameters; never mistaken for a VAE-LE set of the same directory); a restarted sweep loads what
    it finds instead of recomputing.  runner: stands for sweep_cma_awgn_sharded (called with its positional arguments).
    No GMI (unlike run_awgn_sweep): the AWGN CMA driver makes no posteriors to score."""
    if channel not in ("h1", "h2"):
        raise KeyError(f"AWGN driver knows channels h1/h2, got {channel!r}")
    if epe < 1 or num_epochs % epe != 0:
        raise ValueError(f"num_epochs={num_epochs} must be a multiple of epe={epe}")
    vecs = dict(lr_optim=list(lr_optim_vec), M=list(M_vec), SNR=list(SNR_vec), nu=list(nu_vec))
    dev = torch.device("cpu") if runner is not None and device is None else _cuda_device(device)

    def signature(key, cells):
        return _set_signature(driver="CMA_AWGN", mod=mod, sps=sps, channel=channel, M=key[0], N_valid=N_valid, N_train=N_train,
                              num_epochs=num_epochs, epe=epe, datagen=datagen, cells=[sorted(c.items()) for c in cells])

    def file_name(key, cells, sig):
        return f"AWGNCMA_{mod}_M{key[0]}_n{len(cells)}_e{num_epochs}_{sig[:12]}.npz"

    def run_set(key, cells):
        args = (cells, mod, sps, key[0], N_valid, N_train, num_epochs, epe, channel)
        if runner is not None:
            return runner(*args)
        return sweep_cma_awgn_sharded(*args, device=dev, datagen=datagen, verbose=verbose, rank=rank, world=world, group=group)

    SER = _walk_awgn_sets(AWGN_CMA_AXES, vecs, ("M",), iter, num_epochs // epe, dev, checkpoint_dir, rank, world, group, signature, file_name,
                          run_set)
    if rank != 0:
        return None
    return SER, np.arange(0, num_epochs, epe)
