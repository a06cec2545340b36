"""float64 restatement of the data-aided LMMSE reference equalizer of the DP sweeps (DESIGN.md §2), the yardstick of csrc/lmmse.cu:
the regressors u_n are built explicitly and the normal equations solved with numpy, no sliding sums."""
import numpy as np
import torch


def _c(a):
    a = a.detach().cpu().double().numpy() if torch.is_tensor(a) else np.asarray(a, dtype=np.float64)
    return a


def geometry(N, M, n_shift=21):
    mh, D = M // 2, n_shift // 2
    E = (mh + 1) // 2 + D
    return mh, D, E


def regressors(rx, M, N, E):
    """U (|I|, 2M) complex128 with U[n - E, i*M + k] = x_i[2n + k - mh], n in I = [E, N - E)."""
    x = _c(rx)
    xc = x[:, 0] + 1j * x[:, 1]
    mh = M // 2
    n = np.arange(E, N - E)
    idx = 2 * n[:, None] + np.arange(M)[None, :] - mh
    return np.concatenate([xc[0][idx], xc[1][idx]], axis=1)


def lmmse(rx, tx, M, n_shift=21):
    """rx (2,2,2N), tx (2,2,N) of one run -> dict with W (2,4,M), var (2,), delay (2,) int, mse (2, 2D+1) over delta = -D..D, beta (2,),
    rho (2,), S (2,), nI, E, w (2, 2M) complex (the biased solution at the chosen delay)."""
    t = _c(tx)
    N = t.shape[-1]
    mh, D, E = geometry(N, M, n_shift)
    tc = t[:, 0] + 1j * t[:, 1]
    U = regressors(rx, M, N, E)
    nI = U.shape[0]
    Rm = U.conj().T @ U
    n = np.arange(E, N - E)
    res = dict(W=np.zeros((2, 4, M)), var=np.zeros(2), delay=np.zeros(2, dtype=int), mse=np.zeros((2, 2 * D + 1)), beta=np.zeros(2),
               rho=np.zeros(2), S=np.zeros(2), nI=nI, E=E, w=np.zeros((2, 2 * M), dtype=complex))
    order = [0] + [s * k for k in range(1, D + 1) for s in (-1, 1)]          # ties: smaller |delta|, then the negative one
    for o in range(2):
        sols = {}
        for dl in range(-D, D + 1):
            tt = tc[o][n - dl]
            r = U.conj().T @ tt
            w = np.linalg.solve(Rm, r)
            rho = float(np.real(np.vdot(r, w)))
            S = float(np.sum(np.abs(tt) ** 2))
            res["mse"][o, dl + D] = (S - rho) / nI
            sols[dl] = (w, rho, S)
        best = min(order, key=lambda dl: (res["mse"][o, dl + D], order.index(dl)))
        w, rho, S = sols[best]
        beta = rho / S
        res["delay"][o], res["beta"][o], res["rho"][o], res["S"][o], res["w"][o] = best, beta, rho, S, w
        res["var"][o] = S * (S - rho) / (2 * rho * nI)
        res["W"][o, 0:2] = (w.real / beta).reshape(2, M)
        res["W"][o, 2:4] = (w.imag / beta).reshape(2, M)
    return res


def fir64(rx, W):
    """twoXtwoFIR's FIR in float64: rx (2,2,L), W (2,4,M) -> out (2,2,L//2)."""
    from oracle import vaeq_oracle as O
    return O.butterfly_fir(torch.as_tensor(_c(rx)), torch.as_tensor(_c(W)), 2).numpy()


def snr_out_db(res):
    """10 log10 of the mean symbol power over I against twice the fitted noise variance, per output pol."""
    return 10 * np.log10(res["S"] / res["nI"] / (2 * res["var"]))
