"""Closed-form (analytic-gradient) restatement of the DP VAE-LE step in numpy float64.

TEST INFRASTRUCTURE (see oracle/vaeq_oracle.py header for who may import oracle/).

``vaeq_oracle`` follows the reference op by op and lets autograd differentiate it; this file
states the SAME function in closed form, forward and backward, the way the CUDA kernels compute
it (SURVEY.md §8a-a7), in float64.  Tests use it two ways: (1) against autograd of the op-by-op
oracle (proves the derivation), (2) as a high-precision yardstick, so that the fp32 error of the
CUDA path can be compared with the fp32 error of the reference's own torch path.

Reference lines: forward = optical_DP_channel/shared_funcs.py:500-527 and :92-137,
backward = what ``loss.backward()`` does at func_VAELE_DP_MQAM_shaping.py:65,
Adam = torch.optim.Adam as configured at func_VAELE_DP_MQAM_shaping.py:28-31.
"""
from __future__ import annotations

import numpy as np


def dp_step_closed_form(rx, W, h, amp, P, var, nu_sc, sps=2, want_grads=True):
    """rx (2,2,L), W (2,4,M), h (2,2,2,M), amp (n,), P (n,), var (2,), nu_sc -> dict of float64 arrays."""
    f8 = np.float64
    rx, W, h, amp, P, var = (np.asarray(a, dtype=f8) for a in (rx, W, h, amp, P, var))
    nu_sc = f8(nu_sc)
    L = rx.shape[-1]
    B = L // sps
    M = W.shape[-1]
    mh = M // 2
    Mh = 2 * mh
    n = amp.shape[0]
    width = L - Mh

    # ---- butterfly FIR (cross-correlation, zero pad mh, stride sps) --------------- sf:500-518
    x = rx[:, 0] + 1j * rx[:, 1]                              # (i, L)
    w = W[:, 0:2] + 1j * W[:, 2:4]                            # (o, i, M)
    xp = np.pad(x, ((0, 0), (mh, mh)))
    tap_idx = sps * np.arange(B)[:, None] + np.arange(M)[None, :]
    X = xp[:, tap_idx]                                        # (i, B, M)
    y = np.einsum("oik,ibk->ob", w, X)
    yc = np.stack((y.real, y.imag), axis=1)                   # (p, c, B)

    # ---- soft demapper ------------------------------------------------------------- sf:511-523
    a4 = amp[None, None, :, None]
    z = (yc[:, :, None, :] - a4) ** 2 / 2 / var[:, None, None, None] + nu_sc * a4 ** 2
    zs = -(z - z.min(axis=2, keepdims=True))
    ez = np.exp(zs)
    q = ez / ez.sum(axis=2, keepdims=True)                    # (p, c, n, B)

    # ---- posterior moments --------------------------------------------------------- sf:107-113
    m1 = (a4 * q).sum(axis=2)                                 # (p, c, B)
    m2 = (a4 ** 2 * q).sum(axis=2)
    V = m2 - m1 ** 2
    Eq = m1[:, 0] + 1j * m1[:, 1]                             # (nu, B)
    Equp = np.zeros((2, L), dtype=complex)
    Equp[:, ::sps] = Eq
    Vup = np.zeros((2, L))
    Vup[:, ::sps] = V.sum(axis=1)

    # ---- estimated-channel convolution, valid part --------------------------------- sf:115-129
    hc = h[:, :, 0, :] + 1j * h[:, :, 1, :]                   # (chi, nu, M)
    nidx = Mh + np.arange(width)[:, None] - np.arange(M)[None, :]   # D index n -> source sample n-j
    EE = Equp[:, nidx]                                        # (nu, width, M)
    D = np.einsum("xvj,vnj->xn", hc, EE)
    S = Vup[:, nidx].sum(axis=1)                              # (nu, M)   S_nu(j)
    hp = np.abs(hc) ** 2
    Eterm = np.einsum("xvj,vj->x", hp, S)
    r = x[:, mh:L - mh]
    C = (np.abs(r - D) ** 2).sum(axis=1) + Eterm              # sf:133-134 (expanded there)

    # ---- entropy and loss ---------------------------------------------------------- sf:131-137
    qr = q.reshape(2, 2 * n, B)
    P2 = np.concatenate((P, P))[None, :, None]
    qcut = qr[:, :, mh:B - mh]
    ent = np.sum(-qcut * np.log(qcut / P2 + 1e-12))
    loss = np.sum(width * np.log(C)) - ent
    res = dict(out=yc, q=qr, loss=loss, var_est=C / width, C=C, entropy=ent, D=D, Eq=Eq, V=V)
    if not want_grads:
        return res

    # ---- backward ---------------------------------------------------------------------------
    kappa = width / C                                         # dloss/dC_chi
    gD = kappa[:, None] * 2 * (D - r)                         # (chi, width), re + j*im partials
    ghc = np.einsum("xn,vnj->xvj", gD, np.conj(EE)) + 2 * kappa[:, None, None] * hc * S[None]
    gh = np.stack((ghc.real, ghc.imag), axis=2)               # (chi, nu, 2, M)

    gEup = np.zeros((2, L), dtype=complex)
    gVup = np.zeros((2, L))
    for j in range(M):
        lo, hi = Mh - j, L - j
        gEup[:, lo:hi] += np.einsum("xv,xn->vn", np.conj(hc[:, :, j]), gD)
        gVup[:, lo:hi] += np.einsum("x,xv->v", kappa, hp[:, :, j])[:, None]
    gE = gEup[:, ::sps]
    gV = gVup[:, ::sps]                                       # (nu, B), same for both components

    g_m1 = np.stack((gE.real, gE.imag), axis=1) - 2 * m1 * gV[:, None, :]
    gq = a4 * g_m1[:, :, None, :] + a4 ** 2 * gV[:, None, None, :]
    u = q / P[None, None, :, None]
    ent_mask = np.zeros(B)
    ent_mask[mh:B - mh] = 1.0
    gq = gq + ent_mask * (np.log(u + 1e-12) + u / (u + 1e-12))
    gz = -q * (gq - (q * gq).sum(axis=2, keepdims=True))
    gyc = (gz * (yc[:, :, None, :] - a4) / var[:, None, None, None]).sum(axis=2)
    gy = gyc[:, 0] + 1j * gyc[:, 1]
    gw = np.einsum("ob,ibk->oik", gy, np.conj(X))
    gW = np.concatenate((gw.real, gw.imag), axis=1)           # (o, 4, M)
    res.update(gW=gW, gh=gh, gy=gyc, gEq=gE, gV=gV, kappa=kappa)
    return res


class AdamState:
    """torch.optim.Adam single-tensor update restated in numpy (float32 state, double scalars).

    Matches torch/optim/adam.py `_single_tensor_adam` for amsgrad in {False, True}, weight_decay=0,
    maximize=False: bias corrections are Python doubles, the parameter update is
    p += (-lr/bc1) * m / (sqrt(v)/sqrt(bc2) + eps).
    """

    def __init__(self, shape, amsgrad=False, betas=(0.9, 0.999), eps=1e-8):
        self.m = np.zeros(shape, np.float32)
        self.v = np.zeros(shape, np.float32)
        self.vmax = np.zeros(shape, np.float32) if amsgrad else None
        self.t = 0
        self.b1, self.b2 = betas
        self.eps = eps

    def update(self, p, g, lr):
        f4 = np.float32
        g = g.astype(f4)
        self.t += 1
        # exp_avg.lerp_(grad, 1-beta1): torch computes it as ONE fused multiply-add, m + w * (g - m); the float64 product of two floats
        # is exact, so only the float64 sum rounds before the float32 result
        self.m = (self.m.astype(np.float64) + (g - self.m).astype(f4).astype(np.float64) * np.float64(f4(1 - self.b1))).astype(f4)
        self.v = (self.v * f4(self.b2) + f4(1 - self.b2) * g * g).astype(f4)    # mul_(beta2).addcmul_(g,g,1-beta2)
        bc1 = 1 - self.b1 ** self.t
        bc2 = 1 - self.b2 ** self.t
        step = lr / bc1
        bc2s = bc2 ** 0.5
        if self.vmax is not None:
            self.vmax = np.maximum(self.vmax, self.v)
            denom = (np.sqrt(self.vmax) / f4(bc2s) + f4(self.eps)).astype(f4)
        else:
            denom = (np.sqrt(self.v) / f4(bc2s) + f4(self.eps)).astype(f4)
        return (p.astype(f4) + f4(-step) * (self.m / denom)).astype(f4)
