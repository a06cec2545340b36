"""The data-aided LMMSE reference of the DP sweeps on the GPU (csrc/lmmse.cu: k_lmmse_corr, k_lmmse_solve, k_fir_runs; shared_funcs.lmmse_taps_runs
/ fir_runs, sweep.sweep_lmmse_dp and run_dp_sweep(loss_type="LMMSE")) against the float64 restatement tests/lmmse_ref.py and against physics."""
import numpy as np
import pytest
import torch

import lmmse_ref as LR

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _frames(channel, mod, M, N, snrs, seed, nu=0.0270955):
    """R = len(snrs) device frames (one batched generation), mixed SNR: rx (R,2,2,2N), tx (R,2,2,N)."""
    from vae_equalizer_b200 import shared_funcs as sf
    from vae_equalizer_b200.datagen import generate_frames_gpu
    k = sf.init(channel, mod, DEV, nu, 2, M, float(snrs[0]))
    R = len(snrs)
    P = torch.as_tensor(k[2], dtype=torch.float32).reshape(1, -1).repeat(R, 1).to(DEV)
    snr = torch.tensor([float(s) for s in snrs], dtype=torch.float32, device=DEV)
    theta = torch.full((R,), float(np.pi / 10), dtype=torch.float32, device=DEV)
    rx, tx, _ = generate_frames_gpu(N, k[4], snr, P, 2, theta, DEV, seed, h_channel=k[1])
    return rx.contiguous(), tx.contiguous()


def _check_against_ref(rx, tx, M, W, var, delay, ok):
    W, var, delay = W.cpu().double().numpy(), var.cpu().double().numpy(), delay.cpu().numpy()
    assert bool(ok.all())
    for r in range(rx.shape[0]):
        ref = LR.lmmse(rx[r].cpu(), tx[r].cpu(), M)
        for o in range(2):
            mse = np.sort(ref["mse"][o])
            if (mse[1] - mse[0]) <= 1e-9 * abs(mse[0]):
                continue                                            # a near tie: either delay is right
            assert delay[r, o] == ref["delay"][o], (r, o)
            assert abs(var[r, o] - ref["var"][o]) <= 1e-6 * ref["var"][o], (r, o, var[r, o], ref["var"][o])
            err = np.abs(W[r, o] - ref["W"][o]).max() / np.abs(ref["W"][o]).max()
            assert err <= 1e-5, (r, o, err)


@pytest.mark.parametrize("channel,mod,M,N", [("h0", "4-QAM", 5, None), ("h0", "64-QAM", 25, 10000), ("h1", "16-QAM", 25, 4000),
                                             ("h2", "64-QAM", 63, 3000), ("h2", "4-QAM", 63, None), ("h1", "64-QAM", 5, 600)])
def test_taps_against_float64(channel, mod, M, N):
    from vae_equalizer_b200 import shared_funcs as sf
    mh, D, E = LR.geometry(0, M)
    N = N or 2 * E + 4 * M                                          # |I| = 4 M: short, yet an over-determined fit
    snrs = [12, 17, 20, 23, 26, 30] if M != 63 else [14, 24, 30]
    rx, tx = _frames(channel, mod, M, N, snrs, 7)
    W, var, delay, ok = sf.lmmse_taps_runs(rx, tx, M)
    _check_against_ref(rx, tx, M, W, var, delay, ok)


def test_strided_views_and_mixed_batch_of_37():
    from vae_equalizer_b200 import shared_funcs as sf
    M, N = 25, 2000
    snrs = [12 + (k % 19) for k in range(37)]
    rx, tx = _frames("h1", "64-QAM", M, N, snrs, 3)
    rxl = torch.zeros(37, 2, 2, 2 * N + 13, device=DEV)
    rxl[..., 5:5 + 2 * N] = rx
    txl = torch.zeros(37, 2, 2, N + 6, dtype=torch.float16, device=DEV)
    txl[..., 2:2 + N] = tx
    rv, tv = rxl[..., 5:5 + 2 * N], txl[..., 2:2 + N]
    assert not rv.is_contiguous() and not tv.is_contiguous()
    a = sf.lmmse_taps_runs(rv, tv, M)
    b = sf.lmmse_taps_runs(rx, tx, M)
    for x, y in zip(a, b):
        assert torch.equal(x, y)
    idx = [0, 11, 36]
    _check_against_ref(rx[idx], tx[idx], M, a[0][idx], a[1][idx], a[2][idx], a[3][idx])
    z = sf.fir_runs(rv, a[0])
    assert torch.equal(z, sf.fir_runs(rx, a[0]))


def test_physics_on_device_frames():
    from vae_equalizer_b200 import shared_funcs as sf
    M, N = 25, 10000
    for nu in (0.0, 0.0270955):
        snrs = [12, 18, 24]
        rx, tx = _frames("h0", "64-QAM", M, N, snrs, 11, nu=nu)
        W, var, delay, ok = sf.lmmse_taps_runs(rx, tx, M)
        _, D, E = LR.geometry(N, M)
        t = tx.double()
        for r, snr in enumerate(snrs):
            for o in range(2):
                dl = int(delay[r, o])
                S = float((t[r, o, :, E - dl:N - E - dl] ** 2).sum()) / (N - 2 * E)
                db = 10 * np.log10(S / (2 * float(var[r, o])))
                assert abs(db - snr) <= 0.3, (nu, snr, o, db)


def test_zero_cell_is_nan_and_neighbours_untouched():
    from vae_equalizer_b200 import shared_funcs as sf
    M, N = 25, 3000
    rx, tx = _frames("h0", "16-QAM", M, N, [15, 20, 25, 30], 5)
    rz = rx.clone()
    rz[2] = 0
    W, var, delay, ok = sf.lmmse_taps_runs(rz, tx, M)
    assert ok.tolist() == [True, True, False, True]
    assert bool(torch.isnan(W[2]).all()) and bool(torch.isnan(var[2]).all())
    keep = [0, 1, 3]
    W2, var2, delay2, ok2 = sf.lmmse_taps_runs(rx[keep].contiguous(), tx[keep].contiguous(), M)
    assert torch.equal(W[keep], W2) and torch.equal(var[keep], var2) and torch.equal(delay[keep], delay2)


def test_bad_arguments_raise_before_launch():
    from vae_equalizer_b200 import _lib
    from vae_equalizer_b200 import shared_funcs as sf
    M = 25
    _, _, E = LR.geometry(0, M)
    N = 2 * E + 2 * M - 1
    rx = torch.randn(2, 2, 2, 2 * N, device=DEV)
    tx = torch.ones(2, 2, 2, N, dtype=torch.float16, device=DEV)
    n0 = int(_lib.load().vaeq_launch_count(-1))
    with pytest.raises(_lib.VaeqError, match="LS range"):
        sf.lmmse_taps_runs(rx, tx, M)
    with pytest.raises(_lib.VaeqError, match="odd"):
        sf.lmmse_taps_runs(torch.randn(2, 2, 2, 8000, device=DEV), torch.ones(2, 2, 2, 4000, dtype=torch.float16, device=DEV), 24)
    with pytest.raises(_lib.VaeqError):
        sf.lmmse_taps_runs(rx, tx.float(), M)
    assert int(_lib.load().vaeq_launch_count(-1)) == n0
    W, var, delay, ok = sf.lmmse_taps_runs(torch.randn(2, 2, 2, 2 * N + 2, device=DEV), tx.new_ones(2, 2, 2, N + 1), M)   # |I| = 2 M: accepted
    assert bool(ok.all())


def test_fir_runs_against_dpequalizer_and_float64():
    from vae_equalizer_b200 import shared_funcs as sf
    from vae_equalizer_b200.dp import DPEqualizer
    for M, N in ((5, 1000), (25, 3000), (63, 2000)):
        rx, tx = _frames("h2", "16-QAM", M, N, [18, 24, 30], 9)
        W = 0.1 * torch.randn(3, 2, 4, M, device=DEV)
        W[:, 0, 0, M // 2] += 1
        W[:, 1, 1, M // 2] += 1
        z = sf.fir_runs(rx, W)
        for r in range(3):
            ref = LR.fir64(rx[r].cpu(), W[r].cpu())
            assert np.abs(z[r].cpu().double().numpy() - ref).max() <= 5e-6, (M, r)
            eq = DPEqualizer(M, 2, torch.tensor([-1.0, 1.0]), torch.tensor([0.5, 0.5]), torch.tensor([0.1, 0.1]), 0.0, device=DEV, W0=W[r].cpu())
            out = eq.forward(rx[r])[1]
            assert float((out - z[r]).abs().max()) <= 5e-6, (M, r)


def _cells(snrs, seed0=0):
    return [dict(SNR=s, nu=0.0270955, lr_optim=2.5e-3, theta=np.pi / 10, theta_diff=0.06 * np.pi, seed=seed0 + k) for k, s in enumerate(snrs)]


def test_sweep_alone_equals_in_batch_and_op_by_op():
    from vae_equalizer_b200 import shared_funcs as sf
    from vae_equalizer_b200 import sweep
    cells = _cells([12 + (k % 13) for k in range(37)])
    args = ("64-QAM", 2, 25, 100, 2000, 2)
    full = sweep.sweep_lmmse_dp(cells, *args, device=DEV, datagen="gpu", gmi=True, bmi=True)
    alone = sweep.sweep_lmmse_dp([cells[17]], *args, device=DEV, datagen="gpu", gmi=True, bmi=True)
    for a, b in zip(full, alone):
        assert torch.equal(a[17:18], b)
    base = sweep.sweep_lmmse_dp(cells, *args, device=DEV, datagen="gpu")
    for a, b in zip(full[:3], base):
        assert torch.equal(a, b)
    # op by op on the same frames
    consts, P, var0, nu, frames = sweep._dp_source(cells, "64-QAM", 2, 25, "h0", 2000, 2, "gpu", torch.device(DEV), 90e9, -26e-24,
                                                   0.1e-12 * np.sqrt(1000), (0.0314, 0.0314))
    amp, nu = consts[0][3].to(DEV), nu.to(DEV)
    for f, (rx, tx) in enumerate(frames):
        W, v, dl, ok = sf.lmmse_taps_runs(rx, tx, 25)
        z = sf.fir_runs(rx, W)
        q = sf.soft_dec_runs(z, v, amp, nu)
        ser, al, counts = sf.frame_eval_runs(q, z, tx, amp, v, nu, 0, return_counts=True)
        assert torch.equal(full[0][:, :, f], ser) and torch.equal(full[1][:, :, f], v)
        assert torch.equal(full[3][:, :, f], sf.gmi_runs(q, tx, P.to(DEV), al, counts, 0))
        assert torch.equal(full[4][:, :, f], sf.bmi_runs(q, tx, P.to(DEV), al, counts, 0))


def test_lmmse_and_vae_sets_get_the_same_frames(monkeypatch):
    from vae_equalizer_b200 import sweep
    seen = {}
    real = sweep.generate_frames_gpu

    def recorder(tag):
        def gen(*a, **kw):
            rx, tx, s = real(*a, **kw)
            seen.setdefault(tag, []).append((a[0], a[7], rx.double().sum().item(), tx.double().abs().sum().item(), rx.shape[0]))
            return rx, tx, s
        return gen

    kw = dict(SNR_vec=[17, 23], nu_vec=[0.0270955], M_vec=[9, 25], lr_optim_vec=[2.5e-3], iter=2, num_frames=2, N_frame_max=1050,
              device=DEV, datagen="gpu_batched")
    for lt in ("VAE", "LMMSE"):
        monkeypatch.setattr(sweep, "generate_frames_gpu", recorder(lt))
        sweep.run_dp_sweep(loss_type=lt, **kw)
    assert len(seen["VAE"]) == 4 and seen["VAE"] == seen["LMMSE"]
    assert all(s[0] == 1000 for s in seen["VAE"])                   # (N_frame_max // batch_len) * batch_len


def test_checkpoint_resume(tmp_path, monkeypatch):
    from vae_equalizer_b200 import sweep
    kw = dict(SNR_vec=[20], nu_vec=[0.0], M_vec=[25], lr_optim_vec=[2.5e-3], iter=3, num_frames=2, N_frame_max=2000, device=DEV,
              checkpoint_dir=str(tmp_path), gmi=True)
    first = sweep.run_dp_sweep(loss_type="LMMSE", **kw)
    assert [p.name[:6] for p in tmp_path.iterdir()] == ["LMMSE_"]

    def boom(*a, **k):
        raise AssertionError("recomputed")
    monkeypatch.setattr(sweep, "sweep_lmmse_dp_sharded", boom)
    again = sweep.run_dp_sweep(loss_type="LMMSE", **kw)
    for a, b in zip(first, again):
        assert torch.equal(a.cpu(), b.cpu())


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_gpus_equal_one():
    from vae_equalizer_b200 import sweep
    cells = _cells([14, 18, 22, 26, 30])
    args = ("16-QAM", 2, 25, 100, 2000, 2)
    a = sweep.sweep_lmmse_dp(cells, *args, device="cuda:0", datagen="gpu", gmi=True)
    b = sweep.sweep_lmmse_dp(cells, *args, device="cuda:1", datagen="gpu", gmi=True)
    for x, y in zip(a, b):
        assert torch.equal(x.cpu(), y.cpu())
