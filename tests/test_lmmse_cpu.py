"""The data-aided LMMSE reference of the DP sweeps without a GPU: the float64 restatement (tests/lmmse_ref.py) against its own identities and
against physics on the host generator, and the host logic of run_dp_sweep(loss_type="LMMSE") through a stub runner."""
import numpy as np
import pytest
import torch

import lmmse_ref as LR
from oracle import vaeq_oracle as O

IDEAL = dict(symb_rate=90e9, tau_cd=0.0, tau_pmd=0.0, phiIQ=np.array([0.0, 0.0], dtype=np.complex64), theta=0.0)
DEFAULT = dict(symb_rate=90e9, tau_cd=-26e-24, tau_pmd=0.1e-12 * np.sqrt(1000), phiIQ=np.array([0.0314, 0.0314], dtype=np.complex64),
               theta=np.pi / 10)                                     # Eval_run_DP.py's channel


def host_frame(mod, nu, snr, N, seed, chan=DEFAULT, channel="h0", M=25):
    _, h_ch, P, _, amps, pol, _, _, _ = O.init(channel, mod, "cpu", nu, 2, M, snr)
    rx, tx, _ = O.generate_data_shaping(N, amps, snr, h_ch, P, pol, chan["symb_rate"], 2, chan["tau_cd"], chan["tau_pmd"], chan["phiIQ"],
                                        chan["theta"], "cpu", rng=np.random.default_rng(seed))
    return rx, tx


def test_identities_float64():
    rx, tx = host_frame("16-QAM", 0.0, 18, 3000, 1)
    M = 25
    res = LR.lmmse(rx, tx, M)
    N, E, nI = tx.shape[-1], res["E"], res["nI"]
    z = LR.fir64(rx, res["W"])
    zc = z[:, 0] + 1j * z[:, 1]
    t = tx.double().numpy()
    tc = t[:, 0] + 1j * t[:, 1]
    n = np.arange(E, N - E)
    U = LR.regressors(rx, M, N, E)
    for o in range(2):
        dl = res["delay"][o]
        zo, to = zc[o][n], tc[o][n - dl]
        # the FIR with W over I is u_n^T w / beta: pins the (2,4,M) layout
        assert np.allclose(zo, U @ res["w"][o] / res["beta"][o], rtol=0, atol=1e-10)
        # var from the closed form = half the mean squared error of the unbiased output
        assert res["var"][o] == pytest.approx(0.5 * np.mean(np.abs(zo - to) ** 2), rel=1e-9)
        # beta = regression coefficient of the biased output u^T w on t
        zb = U @ res["w"][o]
        assert res["beta"][o] == pytest.approx(np.real(np.vdot(to, zb)) / np.sum(np.abs(to) ** 2), rel=1e-9)
        assert 0 < res["beta"][o] < 1


@pytest.mark.parametrize("chan", ["ideal", "default"])
@pytest.mark.parametrize("mod", ["16-QAM", "64-QAM"])
@pytest.mark.parametrize("nu", [0.0, 0.0270955])
def test_physics_host_generator(mod, nu, chan):
    """The fitted output SNR is the channel's SNR: a wrong beta, var or delay misses it by decibels."""
    for k, snr in enumerate((12, 18, 24)):
        rx, tx = host_frame(mod, nu, snr, 10000, 100 + k, IDEAL if chan == "ideal" else DEFAULT)
        res = LR.lmmse(rx, tx, 25)
        assert np.all(np.abs(LR.snr_out_db(res) - snr) <= 0.3), (mod, nu, chan, snr, LR.snr_out_db(res), res["delay"])


def test_run_dp_sweep_lmmse_stub(tmp_path):
    from vae_equalizer_b200 import sweep
    calls = []

    def runner(cells, mod, sps, M, batch_len, N_frame_max, num_frames, **kw):
        calls.append((len(cells), M, batch_len, kw))
        R = len(cells)
        out = (torch.full((R, 4, num_frames), 0.25), torch.full((R, 2, num_frames), 0.5), torch.full((R, 2), 0.125))
        return out + tuple(torch.full((R, 2, num_frames), 3.0) for m in ("gmi", "bmi") if kw.get(m))

    kw = dict(SNR_vec=[17, 20], nu_vec=[0.0270955], M_vec=[9, 25], lr_optim_vec=[2.5e-3], iter=2, num_frames=3, N_frame_max=1000)
    SER, Var_est, var_real, GMI, BMI = sweep.run_dp_sweep(loss_type="LMMSE", runner=runner, checkpoint_dir=str(tmp_path), gmi=True, bmi=True, **kw)
    assert SER.shape == (4, 2, 1, 1, 1, 2, 1, 1, 1, 1, 2, 3) and Var_est.shape == (2, 2, 1, 1, 1, 2, 1, 1, 1, 1, 2, 3)
    assert var_real.shape == (2, 2, 1, 1, 1, 2, 1, 1, 1, 1, 2, 1) and GMI.shape == Var_est.shape and BMI.shape == Var_est.shape
    assert bool((SER == 0.25).all()) and bool((GMI == 3.0).all())
    assert [c[:3] for c in calls] == [(4, 9, 100), (4, 25, 100)]
    files = sorted(p.name for p in tmp_path.iterdir())
    assert len(files) == 2 and all(f.startswith("LMMSE_64-QAM_M") for f in files)
    # a restart loads the checkpoints instead of calling the runner
    sweep.run_dp_sweep(loss_type="LMMSE", runner=runner, checkpoint_dir=str(tmp_path), gmi=True, bmi=True, **kw)
    assert len(calls) == 2
    # the VAE sweep over the same lists writes its own files: signatures and names never mixed up
    sweep.run_dp_sweep(loss_type="VAE", runner=runner, checkpoint_dir=str(tmp_path), gmi=True, bmi=True, **kw)
    assert len(calls) == 4
    names = sorted(p.name for p in tmp_path.iterdir())
    assert len(names) == 4 and sum(f.startswith("VAE_") for f in names) == 2
    sig = {f.split("_")[-1] for f in names}
    assert len(sig) == 4
