"""float64 restatement of the DP signal model's noise-free part (simulate_channel + simulate_dispersion, sf:38-63) on given amplitude
levels, with numpy: the checker that ties the device generator and its torch formulation to the reference's signal model for the ISI
channels.  The RRC pulse and channel IR come from the oracle, the two 'valid' convolutions are applied one after the other, as the
reference does, and nothing is cast to single precision."""
import numpy as np

from oracle import vaeq_oracle as O

ARGS = (90e9, -26e-24, 0.1e-12 * np.sqrt(1000), np.array([0.0314, 0.0314], dtype=np.complex64))   # symb_rate, tau_cd, tau_pmd, phiIQ


def noise_free_signal(lev, channel, theta, sps=2, symb_rate=ARGS[0], tau_cd=ARGS[1], tau_pmd=ARGS[2], phiIQ=ARGS[3]):
    """lev (R, 4, n_conv) rows [pol0 I, pol0 Q, pol1 I, pol1 Q], theta (R,) -> sig (R, 2, 2 n_conv - K) complex128."""
    lev = np.asarray(lev, dtype=np.float64)
    pulse = O.rrc_pulse(8, sps, 0.1).astype(np.float64)
    h = O.channel_ir(channel, sps).astype(np.complex128)
    out = []
    for r in range(lev.shape[0]):
        up = np.zeros((2, sps * (lev.shape[-1] - 1) + 1), dtype=np.complex128)
        up[:, ::sps] = lev[r, 0::2] + 1j * lev[r, 1::2]
        x = np.stack([np.convolve(np.convolve(row, pulse, mode="valid"), h, mode="valid") for row in up])
        S = np.fft.fft(x, axis=1)
        f = np.fft.fftfreq(x.shape[1], 1 / symb_rate / sps)
        e_cd, d0 = np.exp(1j * 2 * (np.pi * f) ** 2 * tau_cd), np.exp(1j * np.pi * tau_pmd * f)
        d1 = 1 / d0
        c, s = np.cos(float(theta[r])), np.sin(float(theta[r]))
        e0, e1 = np.exp(-1j * np.asarray(phiIQ, dtype=np.complex128))
        R = ((c * e0, s * e0), (-s * e1, c * e1))
        Rt = ((c * e0, -s * e0), (s * e1, c * e1))
        H = [[Rt[a][0] * d0 * R[0][b] + Rt[a][1] * d1 * R[1][b] for b in range(2)] for a in range(2)]
        out.append(np.fft.ifft(np.stack([(H[0][0] * S[0] + H[0][1] * S[1]) * e_cd, (H[1][0] * S[0] + H[1][1] * S[1]) * e_cd]), axis=1))
    return np.stack(out)
