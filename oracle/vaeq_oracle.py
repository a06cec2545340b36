"""CPU oracle for the VAE blind-equalizer hot path  --  TEST INFRASTRUCTURE, NOT PRODUCT CODE.

This file restates, on the CPU with plain torch/numpy, the algorithm of kit-cel/vae-equalizer's
training hot path.  It exists so that the CUDA path in ``vae_equalizer_b200`` can be checked
against something that runs on a box without ``/root/reference``.  Only ``tests/``,
``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` / ``--impl reference`` legs may
import it; the product package never does (it raises if its CUDA library is missing).

Pinning: the reference ships no tests or golden vectors (SURVEY.md §4), so this oracle is pinned
against OUTPUTS OF THE REFERENCE ITSELF, produced in the build container by
``tests/golden/make_golden.py`` (which imports the unmodified reference) and committed under
``tests/golden/*.npz``; ``tests/test_oracle_golden.py`` replays them.  GMI does not exist in the
reference at all ("parity unpinned" for GMI; the definition lives in ``gmi_from_posteriors``).

Every function cites the reference lines it follows; paths are relative to the reference root,
``sf`` = optical_DP_channel/shared_funcs.py, ``awgn`` = AWGN_channel/func_VAELE_MQAM_shaping.py.
The arithmetic of conv1d / softmax / autograd / Adam lives in PyTorch ATen (requirements_vae.txt
pins torch 1.8.1; this image has 2.11 — same semantics for the ops used).
"""
from __future__ import annotations

import math

import numpy as np
import torch
import torch.nn.functional as F

F32 = torch.float32


# --------------------------------------------------------------------------------------------
# constants / initialisation                                                   sf:544-588
# --------------------------------------------------------------------------------------------
_QAM_SIDE = {"4-QAM": 2, "16-QAM": 4, "64-QAM": 8}
_CHANNELS = {
    "h0": [1.0 + 0.0j],
    "h1": [0.0545 + 0.05j, 0.2823 - 0.11971j, -0.7676 + 0.2788j, -0.0641 - 0.0576j, 0.0466 - 0.02275j],
    "h2": [0.0545 + 0.0165j, -1.3449 - 0.4523j, 1.0067 + 1.1524j, 0.3476 + 0.3153j],
}


def channel_ir(channel: str, sps: int) -> np.ndarray:
    """Zero-stuffed, unit-norm channel impulse response (sf:545-554)."""
    taps = np.asarray(_CHANNELS[channel]).astype(np.complex64)
    up = np.zeros(sps * (taps.shape[-1] - 1) + 1, dtype=np.complex64)
    up[0::sps] = taps
    up /= np.linalg.norm(up)
    return up


def square_qam(mod: str) -> np.ndarray:
    """The reference's constellation table (sf:556-559): row-major over (I level, Q level)."""
    side = _QAM_SIDE[mod]
    lev = np.arange(-(side - 1), side, 2)
    return (np.repeat(lev, side) + 1j * np.tile(lev, side)).astype(np.complex128)


def init(channel, mod, device, nu, sps, M_est, SNR):
    """Host-side constants of one run (sf:544-588).  Returns the reference's 9-tuple."""
    h_channel = channel_ir(channel, sps)
    const = square_qam(mod)
    const = const / np.sqrt(np.mean(np.abs(const) ** 2))
    lev_all = const.real
    n_lev = int(np.sqrt(len(lev_all)))
    amps = lev_all[::n_lev]
    amp_levels = torch.tensor(amps, device=device, dtype=F32)
    sc = np.min(np.abs(amps))
    nu_sc = nu / sc ** 2
    P = np.exp(-nu * np.abs(amps / sc) ** 2)
    P = P / np.sum(P)
    grid = np.tile(P, (n_lev, 1))
    P2 = (grid * grid.T) / np.sum(grid * grid.T)
    pow_mean = np.sum(P2.reshape(-1) * np.abs(const) ** 2)
    var = torch.full((2,), pow_mean / 10 ** (SNR / 10) / 2, device=device, dtype=F32)
    h0 = np.zeros([2, 2, 2, M_est])
    h0[0, 0, 0, M_est // 2] = 1
    h0[1, 1, 0, M_est // 2] = 1
    h_est = torch.tensor(h0, requires_grad=True, dtype=F32, device=device)
    return h_est, h_channel, P, amp_levels, amps, 2, nu_sc, var, pow_mean


def dirac_taps(M_est: int) -> torch.Tensor:
    """Initial equalizer taps (2,4,M): nn.init.dirac_ on Conv1d(4,2,M) (sf:494-495)."""
    w = torch.zeros(2, 4, M_est, dtype=F32)
    w[0, 0, M_est // 2] = 1.0
    w[1, 1, M_est // 2] = 1.0
    return w


# --------------------------------------------------------------------------------------------
# forward: butterfly FIR + soft demapper                                      sf:490-542
# --------------------------------------------------------------------------------------------
def butterfly_fir(x: torch.Tensor, w: torch.Tensor, sps: int) -> torch.Tensor:
    """2x2 complex cross-correlation, zero padded M//2, stride sps (sf:500-518).

    x (2,2,L) [pol, I/Q, sample];  w (2,4,M) rows [Re<-pol0, Re<-pol1, Im<-pol0, Im<-pol1];
    returns out (2,2,N) [pol, I/Q, symbol].
    """
    xi, xq = x[:, 0, :], x[:, 1, :]
    lanes_i = torch.cat((xi, -xq), dim=0).unsqueeze(0)      # sf:505
    lanes_q = torch.cat((xq, xi), dim=0).unsqueeze(0)       # sf:507
    pad = w.shape[-1] // 2
    y_i = F.conv1d(lanes_i, w, stride=sps, padding=pad)[0]
    y_q = F.conv1d(lanes_q, w, stride=sps, padding=pad)[0]
    return torch.stack((y_i, y_q), dim=1)


def soft_demap(out: torch.Tensor, var: torch.Tensor, amp: torch.Tensor, nu_sc: float) -> torch.Tensor:
    """q(x|y) per pol and I/Q component with the PCS term (sf:511-523, same as soft_dec sf:529-542).

    out (2,2,N) -> q (2,2n,N): rows 0..n-1 are the I levels, n..2n-1 the Q levels.
    """
    n = amp.shape[0]
    N = out.shape[-1]
    a = amp.view(n, 1)
    a2 = a ** 2
    q = torch.empty(2, 2 * n, N, dtype=out.dtype)
    for p in range(2):
        for c in range(2):
            metric = (out[p, c, :] - a) ** 2 / 2 / var[p] + nu_sc * a2
            q[p, c * n:(c + 1) * n, :] = F.softmin(metric, dim=0)
    return q


def equalizer_forward(x, w, amp, var, nu_sc, sps):
    """twoXtwoFIR.forward (sf:500-527): returns (q_est, out)."""
    out = butterfly_fir(x, w, sps)
    return soft_demap(out, var, amp, nu_sc), out


# --------------------------------------------------------------------------------------------
# ELBO loss                                                                    sf:92-137
# --------------------------------------------------------------------------------------------
def elbo_loss(q, rx, h, amp, P):
    """loss_function_shaping (sf:92-137): returns (loss, var_est (2,) detached).

    q (2,2n,B), rx (2,2,L), h (2,2,2,M) [rx pol, tx pol, Re/Im, tap], amp (n,), P (n,).
    """
    pol, _, B = q.shape
    L = rx.shape[-1]
    sps = L // B
    n = amp.shape[0]
    mh = h.shape[3] // 2
    Mh = 2 * mh

    qv = q.reshape(pol, 2, n, B)
    w1 = amp.view(1, 1, n, 1)
    m1 = (w1 * qv).sum(dim=2)                     # E_q[x]      sf:108,111
    m2 = ((w1 ** 2) * qv).sum(dim=2)              # E_q[x^2]    sf:109,112
    dt = q.dtype
    Eq = torch.zeros(pol, 2, L, dtype=dt)
    Ex2 = torch.zeros(pol, 2, L, dtype=dt)
    Eq[:, :, ::sps] = m1                          # zero-stuffed onto the sample grid
    Ex2[:, :, ::sps] = m2
    Var = Ex2 - Eq ** 2                           # sf:113
    h_pow = (h ** 2).sum(dim=2)                   # |h|^2 (rx pol, tx pol, tap)   sf:115

    width = L - Mh
    D_re = torch.zeros(2, width, dtype=dt)
    D_im = torch.zeros(2, width, dtype=dt)
    E = torch.zeros(2, dtype=dt)
    for j in range(Mh + 1):                       # true convolution, "valid" part only   sf:123-129
        lo, hi = Mh - j, L - j
        eI0, eQ0 = Eq[0, 0:1, lo:hi], Eq[0, 1:2, lo:hi]
        eI1, eQ1 = Eq[1, 0:1, lo:hi], Eq[1, 1:2, lo:hi]
        D_re = D_re + (h[:, 0, 0:1, j] * eI0 - h[:, 0, 1:2, j] * eQ0
                       + h[:, 1, 0:1, j] * eI1 - h[:, 1, 1:2, j] * eQ1)
        D_im = D_im + (h[:, 0, 1:2, j] * eI0 + h[:, 0, 0:1, j] * eQ0
                       + h[:, 1, 1:2, j] * eI1 + h[:, 1, 0:1, j] * eQ1)
        vs = Var[:, :, lo:hi].sum(dim=(1, 2))
        E = E + (h_pow[:, 0, j] * vs[0] + h_pow[:, 1, j] * vs[1])

    P2 = torch.cat((P, P)).view(2 * n, 1)         # sf:131
    qc = q[:, :, mh:B - mh]
    entropy = torch.sum(-qc[0] * torch.log(qc[0] / P2 + 1e-12) - qc[1] * torch.log(qc[1] / P2 + 1e-12))
    r = rx[:, :, mh:L - mh]
    C = torch.sum(r ** 2, dim=(1, 2))
    C = C + (-2 * torch.sum(r[:, 0, :] * D_re + r[:, 1, :] * D_im, dim=1)
             + torch.sum(D_re ** 2 + D_im ** 2, dim=1) + E)
    loss = torch.sum(width * torch.log(C)) - entropy
    return loss, (C / width).detach()


class DPTrainer:
    """One VAE-LE/VAE-flex run's trainable state, stepped exactly like VAELE_DP:26-31,57-66.

    Adam with two parameter groups: group 0 = equalizer taps W (2,4,M), group 1 = channel estimate
    h (2,2,2,M); ``set_lr_w`` mirrors the reference's "scheduler" that only touches group 0
    (func_VAELE_DP_MQAM_shaping.py:45-46).
    """

    def __init__(self, M_est, sps, lr, W0=None, h0=None, amsgrad=False):
        self.sps = sps
        self.W = (dirac_taps(M_est) if W0 is None else W0.detach().clone().to(F32)).requires_grad_(True)
        if h0 is None:
            h0 = torch.zeros(2, 2, 2, M_est, dtype=F32)
            h0[0, 0, 0, M_est // 2] = 1
            h0[1, 1, 0, M_est // 2] = 1
        self.h = h0.detach().clone().to(F32).requires_grad_(True)
        self.opt = torch.optim.Adam([self.W], lr=lr, amsgrad=amsgrad)
        self.opt.add_param_group({"params": self.h})

    def set_lr_w(self, lr):
        self.opt.param_groups[0]["lr"] = lr

    def forward_loss(self, x, amp, var, nu_sc, P):
        q, out = equalizer_forward(x, self.W, amp, var, nu_sc, self.sps)
        loss, var_est = elbo_loss(q, x, self.h, amp, P)
        return q, out, loss, var_est

    def step(self, x, amp, var, nu_sc, P):
        """zero_grad -> forward -> loss -> backward -> Adam; returns detached (q, out, loss, var_est, gW, gh)."""
        self.opt.zero_grad()
        q, out, loss, var_est = self.forward_loss(x, amp, var, nu_sc, P)
        loss.backward()
        gW, gh = self.W.grad.detach().clone(), self.h.grad.detach().clone()
        self.opt.step()
        return q.detach(), out.detach(), loss.detach(), var_est, gW, gh


# --------------------------------------------------------------------------------------------
# evaluation: SER estimators and shift search                                  sf:188-338
# --------------------------------------------------------------------------------------------
def _tx_levels(tx, n):
    """fp16 amplitudes -> level indices, round(scale*tx+scale) (sf:197-198, sf:238-239)."""
    scale = (n - 1) / 2
    return torch.round(scale * tx.float() + scale).to(torch.int64)


def _eight_hypotheses_counts(dec_fn, data, S):
    """Error counts (flip 2, pol 2, rotation 4) given a per-hypothesis 'is symbol wrong' callback."""
    flipped = data.clone()
    flipped[:, 1, :] = S - data[:, 1, :]                       # IQ flip of the reference data (sf:199)
    counts = torch.zeros(2, 2, 4, dtype=torch.int64)
    for f, ref in enumerate((data, flipped)):
        for r in range(4):
            counts[f, :, r] = dec_fn(r, ref)
    return counts


def ser_iqflip_counts(q, tx):
    """Integer error counts behind SER_IQflip (sf:188-222): (flip, pol, rotation) and N."""
    n = q.shape[1] // 2
    S = n - 1
    data = _tx_levels(tx, n)
    dI = torch.argmax(q[:, :n, :], dim=1)
    dQ = torch.argmax(q[:, n:, :], dim=1)
    rot = ((dI, dQ), (S - dI, S - dQ), (S - dQ, dI), (dQ, S - dI))    # 0, pi, pi/2, 3pi/2  (sf:201-219)

    def wrong(r, ref):
        a, b = rot[r]
        return ((ref[:, 0, :] != a) | (ref[:, 1, :] != b)).sum(dim=-1)

    return _eight_hypotheses_counts(wrong, data, S), q.shape[-1]


def ser_iqflip(q, tx):
    """SER_IQflip (sf:188-222): min over flip and rotation, per polarisation; float32 (2,)."""
    counts, N = ser_iqflip_counts(q, tx)
    ser = counts.to(F32) / N
    return torch.amin(ser, dim=(0, -1))


def constell_thresholds(amp, nu_sc, var):
    """PCS-aware decision thresholds with -inf/+inf guards (sf:234-236)."""
    d = (1 + 2 * nu_sc * var[0]) * (amp[:-1] + amp[1:]) / 2
    inf = torch.full((1,), float("inf"), dtype=d.dtype)
    return torch.cat((-inf, d)), torch.cat((d, inf))


def constell_scale(rx, tx):
    """The in-place renormalisation factor of SER_constell_shaping (sf:242)."""
    num = torch.mean(torch.sqrt(tx[:, 0, :].float() ** 2 + tx[:, 1, :].float() ** 2))
    den = torch.mean(torch.sqrt(rx[:, 0, :] ** 2 + rx[:, 1, :] ** 2))
    return num / den


def ser_constell_counts(rx, tx, amp, nu_sc, var):
    """Counts behind SER_constell_shaping + dec_on_bound (sf:225-287).  MUTATES rx like sf:242."""
    n = amp.shape[0]
    S = n - 1
    lo, hi = constell_thresholds(amp, nu_sc, var)
    data = _tx_levels(tx, n)
    rx *= constell_scale(rx, tx)
    yI, yQ = rx[:, 0, :], rx[:, 1, :]
    rot = ((yI, yQ), (-yI, -yQ), (-yQ, yI), (yQ, -yI))                # sf:245-262

    def wrong(r, ref):
        a, b = rot[r]
        okI = (lo[ref[:, 0, :]] <= a) & (a < hi[ref[:, 0, :]])
        okQ = (lo[ref[:, 1, :]] <= b) & (b < hi[ref[:, 1, :]])
        return (~(okI & okQ)).sum(dim=-1)

    return _eight_hypotheses_counts(wrong, data, S), rx.shape[-1]


def ser_constell(rx, tx, amp, nu_sc, var):
    counts, N = ser_constell_counts(rx, tx, amp, nu_sc, var)
    return torch.amin(counts.to(F32) / N, dim=(0, -1))


def _shift_search(E, tx, N_shift):
    """Common tail of find_shift / find_shift_symb_full (sf:299-314, sf:323-338).

    E (2,N) soft I-component per equalizer output pol; tx (2,2,N).  Returns (shift int16 (2,), r,
    corr_abs (2 comp, 2 out-pol, 2 tx-pol, N_shift)).
    """
    N = E.shape[-1]
    half = N_shift // 2
    rolled = torch.stack([torch.roll(E, i - half, -1) for i in range(N_shift)], dim=-1)   # (2,N,S) circular
    corr = torch.stack([torch.abs(tx[:, c, :N].float() @ rolled) for c in range(2)])     # (c, out-pol, tx-pol, S)
    cmax, cind = torch.max(corr, dim=-1)
    best, which = torch.max(cmax, dim=0)                                                 # over tx component
    straight = torch.stack((cind[which[0, 0], 0, 0], cind[which[1, 1], 1, 1]))
    crossed = torch.stack((cind[which[0, 1], 0, 1], cind[which[1, 0], 1, 0]))
    if (best[0, 0] + best[1, 1]) >= (best[0, 1] + best[1, 0]):
        return (half - straight).to(torch.int16), 0, corr
    return (half - crossed).to(torch.int16), 1, corr


def find_shift(q, tx, N_shift, amp, pol=2, return_corr=False):
    """find_shift (sf:290-314): correlate E_q[x_I] against tx I and Q over N_shift circular lags."""
    n = q.shape[1] // 2
    E = torch.sum(amp.view(1, n, 1) * q[:, :n, :], dim=1)
    s, r, corr = _shift_search(E, tx, N_shift)
    return (s, r, corr) if return_corr else (s, r)


def find_shift_symb_full(rx, tx, N_shift, return_corr=False):
    """find_shift_symb_full (sf:316-338): same search on the equalizer output's I component."""
    s, r, corr = _shift_search(rx[:, 0, :], tx, N_shift)
    return (s, r, corr) if return_corr else (s, r)


# --------------------------------------------------------------------------------------------
# CMA baselines                                                                sf:341-488
# --------------------------------------------------------------------------------------------
def _cma_prepare(Rx, h):
    M = h.shape[-1]
    mh = M // 2
    y = F.pad(Rx.to(F32), (mh, mh))
    y = y / torch.mean(y[:, 0, :] ** 2 + y[:, 1, :] ** 2)        # mean POWER incl. pads (sf:349-350)
    return y.numpy().copy(), M, mh


def _cma_symbol(win, hh):
    """2x2 butterfly output for one symbol from window win (2,2,M) and taps hh (2,2,2,M) (sf:360-364)."""
    yI, yQ = win[:, 0, :], win[:, 1, :]                 # (in-pol, M)
    hr, hi = hh[:, :, 0, :], hh[:, :, 1, :]             # (out-pol, in-pol, M)
    oI = np.einsum("im,oim->o", yI, hr, dtype=np.float32) - np.einsum("im,oim->o", yQ, hi, dtype=np.float32)
    oQ = np.einsum("im,oim->o", yI, hi, dtype=np.float32) + np.einsum("im,oim->o", yQ, hr, dtype=np.float32)
    return oI.astype(np.float32), oQ.astype(np.float32)


def _cma_increment(win, oI, oQ):
    """Per-symbol tap increments before the 2*lr*e factor (sf:370-378 / sf:414-422): (o,i,2,M)."""
    yI, yQ = win[:, 0, :], win[:, 1, :]
    inc = np.empty((2, 2, 2, win.shape[-1]), dtype=np.float32)
    inc[:, :, 0, :] = oI[:, None, None] * yI[None] + oQ[:, None, None] * yQ[None]
    inc[:, :, 1, :] = oQ[:, None, None] * yI[None] - oI[:, None, None] * yQ[None]
    return inc


def _cma_core(Rx, R, h, lr, sps, train, mode, batchlen=0, symb_step=0):
    y, M, mh = _cma_prepare(Rx, h)
    hh = h.detach().numpy().astype(np.float32).copy()
    N = Rx.shape[-1]
    nsym = len(range(mh, N + mh, sps))
    out = np.zeros((2, 2, N // sps), dtype=np.float32)
    e = np.zeros((N // sps, 2), dtype=np.float32)
    buf = np.zeros((nsym, 2, 2, 2, M), dtype=np.float32) if mode != "cma" else None
    lr2 = np.float32(2 * lr)
    R = np.float32(R)
    for ks in range(nsym):
        c = mh + ks * sps                    # centre in the padded signal (sf:355-356)
        k = c // sps - mh                    # sf:357 -- NOT ks: for sps=2 it starts at -(mh//2), and the
        #                                      negative indices wrap to the END of out/e/buf (torch indexing)
        win = y[:, :, c - mh:c + mh + 1]
        oI, oQ = _cma_symbol(win, hh)
        out[:, 0, k], out[:, 1, k] = oI, oQ
        e[k, :] = R - oI * oI - oQ * oQ
        if not train:
            continue
        inc = _cma_increment(win, oI, oQ)
        if mode == "cma":
            hh += (lr2 * e[k, :])[:, None, None, None] * inc                      # every symbol (sf:370-378)
            continue
        buf[k] = inc
        if mode == "batch":
            fire = (k % batchlen == 0 and k != 0)                                 # sf:424
        else:
            fire = (k % symb_step == 0 and k >= batchlen)                         # sf:478
        if fire:
            sl = slice(k - batchlen, k)
            upd = np.einsum("koicm,ko->oicm", buf[sl], e[sl], dtype=np.float32)
            hh += lr2 * upd
    h_new = torch.from_numpy(hh)
    with torch.no_grad():
        h.copy_(h_new)                                                            # in place AND returned
    return torch.from_numpy(out), h, torch.from_numpy(e)


def cma(Rx, R, h, lr, sps, train=True):
    """CMA (sf:341-379): per-symbol tap update."""
    return _cma_core(Rx, R, h, lr, sps, train, "cma")


def cma_batch(Rx, R, h, lr, batchlen, sps, train=True):
    """CMAbatch (sf:381-434): buffered increments applied when k%batchlen==0 and k!=0."""
    return _cma_core(Rx, R, h, lr, sps, train, "batch", batchlen=batchlen)


def cma_flex(Rx, R, h, lr, batchlen, symb_step, sps, train=True):
    """CMAflex (sf:436-488): trailing window of batchlen applied every symb_step symbols."""
    return _cma_core(Rx, R, h, lr, sps, train, "flex", batchlen=batchlen, symb_step=symb_step)


# --------------------------------------------------------------------------------------------
# carrier phase estimation                                                     sf:140-186
# --------------------------------------------------------------------------------------------
def cpe(y, M_ma=501):
    """Viterbi-Viterbi 4th-power phase recovery with 501-tap moving average and pi/2 unwrap (sf:140-186)."""
    a, b = y[:, 0, :], y[:, 1, :]
    a2, b2 = a ** 2, b ** 2
    p4_re = a2 * a2 - 6 * a2 * b2 + b2 * b2                        # sf:152,154
    p4_im = 4 * (a2 * a * b - a * b2 * b)                          # sf:153,155
    stacked = torch.stack((p4_re[0], p4_im[0], p4_re[1], p4_im[1])).unsqueeze(1)
    box = torch.full((1, 1, M_ma), 1 / M_ma, dtype=F32)
    ma = F.conv1d(stacked, box, padding=M_ma // 2)[:, 0, :]        # sf:161
    out = torch.zeros_like(y)
    quarter, half = math.pi / 4, math.pi / 2
    for p in range(2):
        phi = torch.atan2(ma[2 * p + 1], -ma[2 * p]) / 4            # sf:163,172
        d = phi[1:] - phi[:-1]                                     # jumps are judged on the WRAPPED phase
        up = torch.zeros_like(phi)
        up[1:] = torch.cumsum((d < -quarter).to(F32) - (d > quarter).to(F32), 0)
        phi = phi + np.float32(half) * up                          # sf:166-169
        c, s = torch.cos(phi), torch.sin(phi)
        out[p, 0, :] = a[p] * c - b[p] * s                         # sf:182-185
        out[p, 1, :] = b[p] * c + a[p] * s
    return out


# --------------------------------------------------------------------------------------------
# data generation (host side, statistical parity only)                        sf:17-90
# --------------------------------------------------------------------------------------------
def rrc_pulse(T, sps, beta):
    """Root-raised-cosine pulse (sf:27-36)."""
    t = np.arange(-T * sps / 2, T * sps / 2, 1 / sps, dtype=np.float32)
    with np.errstate(divide="ignore", invalid="ignore"):
        h = (np.sin(np.pi * t * (1 - beta)) + 4 * beta * t * np.cos(np.pi * t * (1 + beta))) / (np.pi * t * (1 - (4 * beta * t) ** 2))
    h[np.abs(t) == 1 / 4 / beta] = beta / np.sqrt(2) * ((1 + 2 / np.pi) * np.sin(np.pi / 4 / beta) + (1 - 2 / np.pi) * np.cos(np.pi / 4 / beta))
    h[t == 0] = 1 + beta * (4 / np.pi - 1)
    return h / np.linalg.norm(h)


def dispersion(sig, symb_rate, sps, tau_cd, tau_pmd, phiIQ, theta):
    """Residual CD + PMD + polarisation rotation + IQ phase in the frequency domain (sf:38-54).

    The reference builds the 2x2 Jones matrix as a ragged nested list (sf:49, rejected by
    numpy>=1.24); here it is applied element-wise, which is what numpy 1.18 computed.
    """
    S = np.fft.fft(sig, axis=1)
    f = np.fft.fftfreq(sig.shape[1], 1 / symb_rate / sps)
    e_cd = np.exp(1j * 2 * (np.pi * f) ** 2 * tau_cd)
    e_pmd = np.exp(1j * np.pi * tau_pmd * f)
    c, s = np.cos(theta), np.sin(theta)
    e_iq = np.exp(-1j * phiIQ)
    R = np.array([[c * e_iq[0], s * e_iq[0]], [-s * e_iq[1], c * e_iq[1]]])
    Rt = np.array([[c * e_iq[0], -s * e_iq[0]], [s * e_iq[1], c * e_iq[1]]])
    d0, d1 = e_pmd, 1 / e_pmd
    # H = Rt @ diag(d0,d1) @ R, per frequency bin
    H00 = Rt[0, 0] * d0 * R[0, 0] + Rt[0, 1] * d1 * R[1, 0]
    H01 = Rt[0, 0] * d0 * R[0, 1] + Rt[0, 1] * d1 * R[1, 1]
    H10 = Rt[1, 0] * d0 * R[0, 0] + Rt[1, 1] * d1 * R[1, 0]
    H11 = Rt[1, 0] * d0 * R[0, 1] + Rt[1, 1] * d1 * R[1, 1]
    O = np.zeros((2, sig.shape[1]), dtype=np.complex128)
    O[0] = (H00 * S[0] + H01 * S[1]) * e_cd
    O[1] = (H10 * S[0] + H11 * S[1]) * e_cd
    return np.complex64(np.fft.ifft(O, axis=1))


def generate_data_shaping(N, amps, SNR, h_channel, P, pol, symb_rate, sps, tau_cd, tau_pmd, phiIQ, theta, device, rng=None):
    """PCS symbols -> RRC pulse -> channel IR -> dispersion -> AWGN (sf:65-90).

    ``rng`` (a numpy Generator) makes it reproducible; the reference is unseeded (sf:75, sf:84).
    Returns rx (2,2,sps*N) f32, data (2,2,N) f16, sigma_n.
    """
    T, beta = 8, 0.1
    rng = np.random.default_rng() if rng is None else rng
    M = len(h_channel)
    n_conv = N + M + 4 * T
    data = rng.choice(amps, (pol * 2, n_conv), p=P)
    up = np.zeros((pol, sps * (n_conv - 1) + 1), dtype=np.complex64)
    up[:, ::sps] = data[0::pol, :] + 1j * data[1::pol, :]
    pulse = rrc_pulse(T, sps, beta)
    shaped = np.stack([np.convolve(np.convolve(up[i], pulse, mode="valid"), h_channel, mode="valid") for i in range(pol)]).astype(np.complex64)
    sig = dispersion(shaped, symb_rate, sps, tau_cd, tau_pmd, phiIQ, theta)
    sigma_n = np.sqrt(np.mean(np.abs(sig) ** 2) * sps / 2 / 10 ** (SNR / 10))
    sig = sig + sigma_n * (rng.standard_normal(sig.shape) + 1j * rng.standard_normal(sig.shape))
    rx = torch.from_numpy(np.asarray([sig[:, :sps * N].real, sig[:, :sps * N].imag])).permute(1, 0, 2).to(device, F32)
    sl = slice(T + M - 1, N + T + M - 1)
    tx = torch.from_numpy(np.asarray([data[0::pol, sl], data[1::pol, sl]])).permute(1, 0, 2).to(device, torch.float16)
    return rx.contiguous(), tx.contiguous(), sigma_n


# --------------------------------------------------------------------------------------------
# AWGN single-polarisation variant                                             awgn:63-231
# --------------------------------------------------------------------------------------------
def awgn_forward(x, w, amp, amp_mean, var, sps):
    """twoFIR.forward (awgn:214-231).  x (2,L), w (1,2,M) -> q (2n,N), out (2,N).

    Taps act as w0 - j*w1 (lanes [xI,xQ] and [xQ,-xI], awgn:216-218); the demapper sees the output
    renormalised through the graph by mean|out_c| (awgn:228) and uses (y-a)^2/var (awgn:229).
    """
    pad = (w.shape[-1] - 1) // 2
    lane_i = x.unsqueeze(0)
    lane_q = torch.stack((x[1], -x[0])).unsqueeze(0)
    oI = F.conv1d(lane_i, w, stride=sps, padding=pad)[0, 0]
    oQ = F.conv1d(lane_q, w, stride=sps, padding=pad)[0, 0]
    out = torch.stack((oI, oQ))
    return awgn_demap(out, amp, amp_mean, var), out


def awgn_demap(out, amp, amp_mean, var):
    """The demapper of twoFIR.forward (awgn:228-231): out (2,N) -> q (2n,N)."""
    a = amp.view(-1, 1)
    q = []
    for c in range(2):
        yn = out[c] / torch.mean(torch.abs(out[c])) * amp_mean
        q.append(F.softmin((yn - a) ** 2 / var, dim=0))
    return torch.cat(q, dim=0)


def awgn_loss(q, rx, h, amp, P):
    """loss_function (awgn:63-95): scalar C, entropy with the prior, per-sample E."""
    n = amp.shape[0]
    B = q.shape[1]
    sps = rx.shape[-1] // B
    L = B * sps
    mh = h.shape[1] // 2
    Mh = 2 * mh
    qv = q.reshape(2, n, B)
    m1 = (amp.view(1, n, 1) * qv).sum(1)
    m2 = ((amp ** 2).view(1, n, 1) * qv).sum(1)
    dt = q.dtype                                              # float32 as the reference; float64 as the yardstick of the tests
    Eq = torch.zeros(2, L, dtype=dt)
    Ex2 = torch.zeros(2, L, dtype=dt)
    Eq[:, ::sps] = m1
    Ex2[:, ::sps] = m2
    width = L - Mh
    D_re = torch.zeros(width, dtype=dt)
    D_im = torch.zeros(width, dtype=dt)
    E = torch.zeros(width, dtype=dt)
    for j in range(Mh + 1):                                   # awgn:85-88
        lo, hi = Mh - j, L - j
        D_re = D_re + (h[0, j] * Eq[0, lo:hi] - h[1, j] * Eq[1, lo:hi])
        D_im = D_im + (h[0, j] * Eq[1, lo:hi] + h[1, j] * Eq[0, lo:hi])
        E = E + torch.sum((h[0, j] ** 2 + h[1, j] ** 2) * (Ex2[:, lo:hi] - Eq[:, lo:hi] ** 2), dim=0)
    P2 = torch.cat((P, P)).view(2 * n, 1)
    qc = q[:, mh:B - mh]
    entropy = torch.sum(-qc * torch.log(qc / P2 + 1e-12))
    C = torch.sum(rx[:, mh:L - mh] ** 2)
    C = C + (-2 * torch.sum(rx[0, mh:L - mh] * D_re + rx[1, mh:L - mh] * D_im) + torch.sum(D_re ** 2 + D_im ** 2 + E))
    return width * torch.log(C) - entropy


def awgn_step(rx, W, h, amp, P, amp_mean, var, dtype=F32, want_grads=True):
    """awgn_forward + awgn_loss (+ autograd) in dtype on the CPU: dict of out (2,N), q (2n,N), loss and, with want_grads, gW (1,2,M)
    and gh (2,M).  float32 is the reference's own arithmetic; float64 is the yardstick the float32 paths are measured against."""
    cv = lambda a: torch.as_tensor(np.asarray(a.detach().cpu() if torch.is_tensor(a) else a)).to(dtype)
    x, a = cv(rx), cv(amp)
    Wt = cv(W).reshape(1, 2, -1).requires_grad_(want_grads)
    ht = cv(h).requires_grad_(want_grads)
    with torch.set_grad_enabled(want_grads):
        q, out = awgn_forward(x, Wt, a, amp_mean, var, 2)
        loss = awgn_loss(q, x, ht, a, cv(P))
    res = dict(out=out.detach(), q=q.detach(), loss=loss.detach())
    if want_grads:
        gW, gh = torch.autograd.grad(loss, (Wt, ht))
        res.update(gW=gW, gh=gh)
    return res


def awgn_constants(mod, nu, SNR):
    """amp levels, P, amp_mean, var of the AWGN driver (awgn:252-272)."""
    const = square_qam(mod)
    const = const / np.sqrt(np.mean(np.abs(const) ** 2))
    n = int(np.sqrt(len(const)))
    amps = const.real[::n]
    sc = np.min(np.abs(amps))
    P = np.exp(-nu * np.abs(amps / sc) ** 2)
    P = P / np.sum(P)
    grid = np.tile(P, (n, 1))
    wpts = (grid * grid.T).reshape(-1) * const
    amp_mean = np.sum(np.abs(wpts.real) + np.abs(wpts.imag)) / 2
    return amps, P, amp_mean, 10 ** (-SNR / 10)


def awgn_ser_q_counts(q, tx):
    """SER_q (awgn:97-124): 4 rotations, no IQ flip; returns counts (4,), N."""
    n = q.shape[0] // 2
    S = n - 1
    N = tx.shape[-1]
    data = _tx_levels(tx, n)
    dI = torch.argmax(q[:n, :N], dim=0)
    dQ = torch.argmax(q[n:, :N], dim=0)
    rot = ((dI, dQ), (S - dI, S - dQ), (S - dQ, dI), (dQ, S - dI))
    return torch.stack([((data[0] != a) | (data[1] != b)).sum() for a, b in rot]), N


def awgn_find_shift(q, tx, N_shift, amp):
    """find_shift of the AWGN module (awgn:188-204): first 1000 symbols, I then Q fallback."""
    n = amp.shape[0]
    E = torch.sum(amp.view(n, 1) * q[:n, :1000], dim=0)
    half = N_shift // 2
    rolled = torch.stack([torch.roll(E, i - half, 0) for i in range(N_shift)], dim=-1)
    cI = tx[0, :1000].float() @ rolled
    if torch.max(torch.abs(cI)) >= 0.02 * q.shape[-1]:
        return half - torch.argmax(torch.abs(cI))
    cQ = tx[1, :1000].float() @ rolled
    if torch.max(torch.abs(cQ)) >= torch.max(torch.abs(cI)):
        return half - torch.argmax(torch.abs(cQ))
    return half - torch.argmax(torch.abs(cI))


# --------------------------------------------------------------------------------------------
# AWGN single-polarisation CMA module          AWGN_channel/func_CMA_MQAM_shaping.py (cm:)
# --------------------------------------------------------------------------------------------
def awgn_cma(Rx, R, h, lr, sps, train=True):
    """CMA (cm:142-168): complex FIR h[0] + j h[1] over Rx (2,N), per-symbol tap update, no power normalisation.
    Mutates h in place and returns it, like the reference.  The output index k = i//sps - mh is negative for the
    first symbols and wraps to the end of out / e (cm:155)."""
    M = h.shape[1]
    mh = M // 2
    N = Rx.shape[1]
    y = F.pad(Rx.to(F32), (mh, mh)).numpy()
    hh = h.detach().numpy().astype(np.float32).copy()
    out = np.zeros((2, N // sps), dtype=np.float32)
    e = np.zeros(N // sps, dtype=np.float32)
    lr2, R = np.float32(2 * lr), np.float32(R)
    for i in range(mh, N + mh, sps):
        win = y[:, i - mh:i + mh + 1]
        k = i // sps - mh
        o0 = np.float32(np.dot(win[0], hh[0]) - np.dot(win[1], hh[1]))            # cm:157-158
        o1 = np.float32(np.dot(win[0], hh[1]) + np.dot(win[1], hh[0]))
        out[0, k], out[1, k] = o0, o1
        e[k] = R - o0 * o0 - o1 * o1                                               # cm:160
        if train:
            f = lr2 * e[k]
            hh[0] = hh[0] + f * (o0 * win[0] + o1 * win[1])                        # cm:163-164
            hh[1] = hh[1] + f * (o1 * win[0] - o0 * win[1])
    with torch.no_grad():
        h.copy_(torch.from_numpy(hh))
    return torch.from_numpy(out), h, torch.from_numpy(e)


def awgn_cpe(y, M_ma=501):
    """CPE of the AWGN module (cm:170-196): 4th power, 501-tap moving average, NO unwrapping."""
    a, b = y[0], y[1]
    a2, b2 = a ** 2, b ** 2
    p4 = torch.stack((a2 ** 2 - 6 * a2 * b2 + b2 ** 2, 4 * (a2 * a * b - a * b2 * b))).unsqueeze(1)      # cm:180
    ma = F.conv1d(p4, torch.full((1, 1, M_ma), 1 / M_ma, dtype=F32), padding=M_ma // 2)[:, 0, :]
    phi = torch.atan2(ma[1], -ma[0]) / 4                                             # cm:189
    c, s = torch.cos(phi), torch.sin(phi)
    return torch.stack((a * c - b * s, b * c + a * s))                               # cm:193-194


def awgn_ser_cma_counts(rx, tx, amp):
    """Counts behind SER_CMA (cm:63-93): MUTATES rx (cm:73); nearest-level decisions, rotations 0, pi and the two quarter turns."""
    n = amp.shape[0]
    S = n - 1
    N = tx.shape[1]
    data = _tx_levels(tx, n)
    rx *= torch.mean(torch.sqrt(tx[0].float() ** 2 + tx[1].float() ** 2)) / torch.mean(torch.sqrt(rx[0] ** 2 + rx[1] ** 2))
    dI = torch.argmin(torch.abs(rx[0, :N] - amp.view(n, 1)), dim=0)
    dQ = torch.argmin(torch.abs(rx[1, :N] - amp.view(n, 1)), dim=0)
    rot = ((dI, dQ), (S - dI, S - dQ), (S - dQ, dI), (dQ, S - dI))
    return torch.stack([((data[0] != a) | (data[1] != b)).sum() for a, b in rot]), N


def awgn_ser_cma(rx, tx, amp):
    counts, N = awgn_ser_cma_counts(rx, tx, amp)
    return torch.min(counts.to(F32) / N)


def awgn_find_shift_symb(rx, tx, N_shift):
    """find_shift_symb (cm:127-140): non-circular correlation over the first 1000 symbols, I then Q fallback."""
    half = N_shift // 2
    mat = torch.stack([rx[0, i:1000 - half + i] for i in range(N_shift)], dim=1)
    cI = tx[0, half:1000].float() @ mat
    if torch.max(torch.abs(cI)) >= 0.02 * rx.shape[-1]:
        return torch.argmax(torch.abs(cI)) - half
    cQ = tx[1, half:1000].float() @ mat
    if torch.max(torch.abs(cQ)) >= torch.max(torch.abs(cI)):
        return torch.argmax(torch.abs(cQ)) - half
    return torch.argmax(torch.abs(cI)) - half


# --------------------------------------------------------------------------------------------
# extension (NOT in the reference): GMI from the demapper posteriors
# --------------------------------------------------------------------------------------------
def gmi_from_posteriors(q, tx, P):
    """Symbol-wise achievable rate estimate  H(X) + mean log2 q(x_tx|y)  per pol, in bit/2D-symbol.

    The reference has no GMI code (SURVEY.md fact 3) — parity unpinned; this is the definition the
    CUDA ``vaeq_gmi`` kernel is checked against.
    """
    n = q.shape[1] // 2
    idx = _tx_levels(tx, n)
    Pt = P.to(torch.float64)
    H = -2 * torch.sum(Pt * torch.log2(Pt))
    qi = torch.gather(q[:, :n, :].double(), 1, idx[:, 0:1, :]).squeeze(1)
    qq = torch.gather(q[:, n:, :].double(), 1, idx[:, 1:2, :]).squeeze(1)
    ll = torch.log2(torch.clamp(qi, min=1e-30)) + torch.log2(torch.clamp(qq, min=1e-30))
    return (H + ll.mean(dim=-1)).to(F32)
