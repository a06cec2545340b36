"""Host side of the batched DP runs above 1000 symbols (one thread-block cluster per run, DESIGN.md §4c): the supported batch_len
limit and the sweeps' rejection of larger minibatches before any device work."""
import pytest

from vae_equalizer_b200 import _lib, sweep


def test_max_batch_len_per_m_est():
    lib = _lib.load()
    lims = {M: int(lib.vaeq_dp_runs_max_batch_len(M, 8)) for M in (1, 5, 25, 63)}
    assert lims[5] == 9088 and lims[25] == 8640 and lims[63] == 7776                 # K = 8 CTAs of <= 220 KB each
    assert lims[1] >= lims[5] >= lims[25] >= lims[63] > 1000
    assert all(int(lib.vaeq_dp_runs_max_batch_len(25, n)) == lims[25] for n in (2, 4))   # the plan does not depend on n_lev
    assert lib.vaeq_dp_runs_max_batch_len(24, 8) == 0 and lib.vaeq_dp_runs_max_batch_len(25, 3) == 0


def test_sweeps_reject_batch_len_above_the_limit_first():
    """The check runs before the device is even looked up, so it needs no GPU."""
    lim = int(_lib.load().vaeq_dp_runs_max_batch_len(25, 8))
    cell = dict(SNR=20, nu=0.0, lr_optim=2.5e-3, theta=0.0, theta_diff=0.0, seed=1)
    with pytest.raises(_lib.VaeqError, match=str(lim)):
        sweep.sweep_vae_dp([cell], "64-QAM", 2, 25, lim + 1, 2 * (lim + 1), 1, kind="VAE")
    with pytest.raises(_lib.VaeqError, match=str(lim)):
        sweep.run_dp_sweep(loss_type="VAEflex", batch_len_vec=[100, lim + 1], M_vec=[25], iter=1, num_frames=1)
