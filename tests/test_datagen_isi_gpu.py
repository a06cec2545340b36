"""The device generator on the ISI channels 'h1' and 'h2' (csrc/datagen.cu vaeq_gen_pulse_cplx: one complex 'valid' FIR with the
composite filter rrcfir (*) h_channel, then the Jones / CD / PMD step and the noise of the 'h0' path), and the DP engines and drivers
that use it: the CUDA path against the torch.fft formulation and against the float64 signal model on the same levels, its statistics,
batch independence, argument checks, and the engines' bitwise agreements on these channels."""
import numpy as np
import pytest
import torch

import datagen_ref as ref

pytestmark = pytest.mark.gpu

CHANNELS = ["h1", "h2"]


def consts(mod="64-QAM", nu=0.0270955):
    from vae_equalizer_b200.constants import init
    k = init("h0", mod, "cpu", nu, 2, 25, 23)
    return k[4], np.asarray(k[2], dtype=np.float32)


@pytest.mark.parametrize("channel", CHANNELS)
def test_cuda_isi_generator_against_the_torch_formulation(channel):
    from vae_equalizer_b200 import datagen as dg
    from vae_equalizer_b200.constants import upsampled_channel
    h = upsampled_channel(channel, 2)
    N, sps = 6000, 2
    amps, P64 = consts()
    _, P0 = consts(nu=0.0)
    P = np.stack([P64, P0, P64])
    snr, theta = [23.0, 13.0, 30.0], [0.3, 1.0, -0.7]
    Pt = torch.as_tensor(P, device="cuda")
    rx, tx, sigma, lev, sig = dg._generate_frames_cuda(N, amps, snr, Pt, theta, torch.device("cuda"), 41, *ref.ARGS, return_parts=True,
                                                       h_channel=h)
    K, n_conv = 32 + len(h) - 1, N + len(h) + 4 * dg.PULSE_SPAN
    assert lev.shape == (3, 4, n_conv) and sig.shape == (3, 2, 2 * n_conv - K)
    assert rx.shape == (3, 2, 2, sps * N) and tx.shape == (3, 2, 2, N) and tx.dtype == torch.float16
    off = dg.PULSE_SPAN + len(h) - 1                                      # sf:89
    for p in range(2):
        for c in range(2):
            assert torch.equal(tx[:, p, c], lev[:, 2 * p + c, off:off + N].to(torch.float16))
    # noise-free signal: against the torch.fft formulation and against the float64 signal model, on the same levels
    sig_t = dg._frames_torch_from_levels(lev, N, sps, theta, *ref.ARGS, h_channel=h)
    assert sig_t.shape == sig.shape
    assert float((sig - sig_t).abs().max()) < 3e-5 * float(sig_t.abs().max())
    sig_ref = ref.noise_free_signal(lev.cpu().numpy(), channel, theta)
    assert float(np.abs(sig.cpu().numpy() - sig_ref).max()) < 3e-5 * float(np.abs(sig_ref).max())
    # sigma_n (sf:83)
    pw = (sig_t.abs() ** 2).mean(dim=(1, 2)).cpu().numpy()
    assert np.allclose(sigma.cpu().numpy(), np.sqrt(pw * sps / 2 / 10 ** (np.asarray(snr) / 10)), rtol=1e-4)
    # the levels follow the pmf of the run
    a = np.asarray(amps, dtype=np.float32)
    for r in range(3):
        x = lev[r].cpu().numpy().ravel()
        cnt = np.array([(x == a[l]).sum() for l in range(len(a))])
        assert cnt.sum() == x.size
        exp = P[r] / P[r].sum() * x.size
        assert np.all(np.abs(cnt - exp) < 5 * np.sqrt(exp) + 1)
    # noise: zero mean, unit variance, Gaussian kurtosis, I/Q and neighbouring samples uncorrelated
    clean = torch.stack((sig.real, sig.imag), dim=2)[..., :sps * N]
    z = ((rx - clean) / sigma[:, None, None, None]).double()
    n_el = z[0].numel()
    for r in range(3):
        zr = z[r]
        assert abs(float(zr.mean())) < 5 / np.sqrt(n_el) and abs(float(zr.var()) - 1) < 5 * np.sqrt(2 / n_el)
        assert abs(float((zr ** 4).mean()) - 3) < 0.2
        assert abs(float((zr[:, 0] * zr[:, 1]).mean())) < 5 / np.sqrt(n_el / 2)
        assert abs(float((zr[..., 1:] * zr[..., :-1]).mean())) < 5 / np.sqrt(n_el)
    # same seed -> same data; run 0 alone = run 0 of the batch; another seed differs
    rx2, tx2, _ = dg.generate_frames_gpu(N, amps, snr, P, sps, theta, "cuda", 41, *ref.ARGS, h_channel=h)
    rx1, tx1, _ = dg.generate_frames_gpu(N, amps, snr[:1], P[:1], sps, theta[:1], "cuda", 41, *ref.ARGS, h_channel=h)
    rx3, _, _ = dg.generate_frames_gpu(N, amps, snr, P, sps, theta, "cuda", 42, *ref.ARGS, h_channel=h)
    assert torch.equal(rx2, rx) and torch.equal(tx2, tx) and torch.equal(rx1[0], rx[0]) and torch.equal(tx1[0], tx[0])
    assert not torch.equal(rx3, rx)
    # and the statistics of the full signal agree with the torch generator on the GPU
    rxt, _, sgt = dg._generate_frames_torch(N, amps, snr, Pt, sps, theta, torch.device("cuda"), 41, *ref.ARGS, h_channel=h)
    assert np.allclose(sgt.cpu().numpy(), sigma.cpu().numpy(), rtol=0.05)
    assert np.allclose(rxt.double().var(dim=(1, 2, 3)).cpu().numpy(), rx.double().var(dim=(1, 2, 3)).cpu().numpy(), rtol=0.05)


def test_gen_pulse_cplx_rejects_bad_arguments_and_launches_nothing():
    from vae_equalizer_b200 import VaeqError, _lib
    lib = _lib.load()
    n_conv, R = 200, 2
    lev = torch.zeros(R, 4, n_conv, device="cuda")
    taps = torch.zeros(2 * 130, device="cuda")
    shaped = torch.zeros(R, 2, 2 * n_conv, dtype=torch.complex64, device="cuda")
    st = _lib.current_stream()
    bad = [(39, shaped.data_ptr()), (130, shaped.data_ptr()), (40, shaped.data_ptr() + 8)]     # odd K, K > 128, shaped not 16-byte aligned
    torch.cuda.synchronize()
    n0 = int(lib.vaeq_launch_count(-1))
    for K, dst in bad:
        with pytest.raises(VaeqError):
            _lib.check(lib.vaeq_gen_pulse_cplx(lev.data_ptr(), taps.data_ptr(), K, n_conv, dst, R, st), "vaeq_gen_pulse_cplx")
    torch.cuda.synchronize()
    assert int(lib.vaeq_launch_count(-1)) == n0
    assert float(shaped.abs().max()) == 0.0
    _lib.check(lib.vaeq_gen_pulse_cplx(lev.data_ptr(), taps.data_ptr(), 40, n_conv, shaped.data_ptr(), R, st), "vaeq_gen_pulse_cplx")
    torch.cuda.synchronize()
    assert int(lib.vaeq_launch_count(-1)) == n0 + 1


CELLS = [dict(SNR=20, nu=0.0270955, lr_optim=2.5e-3, theta=np.pi / 10, theta_diff=0.06 * np.pi, seed=3),
         dict(SNR=24, nu=0.0, lr_optim=5e-3, theta=0.2, theta_diff=0.0, seed=4),
         dict(SNR=17, nu=0.0270955, lr_optim=1e-3, theta=0.0, theta_diff=0.01, seed=5)]
COMMON = dict(symb_rate=90e9, tau_cd=-26e-24, tau_pmd=0.1e-12 * np.sqrt(1000), phiIQ=np.array([0.0314, 0.0314], dtype=np.complex64))


@pytest.mark.parametrize("channel", CHANNELS)
def test_vae_sweep_on_isi_channels_equals_single_run_drivers(channel):
    """sweep_vae_dp (VAE, VAEflex) with datagen='gpu': a cell alone equals the same cell in a 3-cell batch, and equals
    processing_vaele_dp / processing_vaeflex_dp for the same cell and seed, bitwise; datagen='gpu_batched' runs."""
    from vae_equalizer_b200.processing import processing_vaele_dp, processing_vaeflex_dp
    from vae_equalizer_b200.sweep import sweep_vae_dp
    for kind, fn, flex in (("VAE", processing_vaele_dp, 10), ("VAEflex", processing_vaeflex_dp, 20)):
        args = ("64-QAM", 2, 25, 100, 2000, 3)
        kw = dict(flex_step=flex, channel=channel, N_lrhalf=2, kind=kind, **COMMON)
        ser, ve, var = sweep_vae_dp(CELLS, *args, eval_mode="per_cell", datagen="gpu", **kw)
        ser_b, ve_b, _ = sweep_vae_dp(CELLS, *args, datagen="gpu", **kw)
        ser1, ve1, _ = sweep_vae_dp(CELLS[1:2], *args, datagen="gpu", **kw)
        torch.cuda.synchronize()
        assert torch.equal(ser1[0], ser_b[1]) and torch.equal(ve1[0], ve_b[1]), kind
        assert torch.isfinite(ser).all() and float(ser.max()) <= 1.0 and (ve > 0).all()
        if kind == "VAE":
            for r, c in enumerate(CELLS):
                s1, v1, var1 = fn("64-QAM", 2, c["SNR"], c["nu"], 25, c["theta_diff"], c["theta"], c["lr_optim"], 100, 2000, 3, flex, channel,
                                  COMMON["symb_rate"], COMMON["tau_cd"], COMMON["tau_pmd"], COMMON["phiIQ"], 2, verbose=False, datagen="gpu",
                                  seed=c["seed"])
                assert torch.equal(s1, ser[r]) and torch.equal(v1, ve[r]) and torch.equal(var1, var[r]), (kind, r)
        else:
            c = CELLS[0]
            s1, v1, _ = fn("64-QAM", 2, c["SNR"], c["nu"], 25, c["theta_diff"], c["theta"], c["lr_optim"], 100, 2000, 3, flex, channel,
                           COMMON["symb_rate"], COMMON["tau_cd"], COMMON["tau_pmd"], COMMON["phiIQ"], 2, verbose=False, datagen="gpu", seed=c["seed"])
            assert torch.equal(s1, ser[0]) and torch.equal(v1, ve[0]), kind
        ser_g, ve_g, _ = sweep_vae_dp(CELLS, *args, datagen="gpu_batched", **kw)
        assert ser_g.shape == (3, 4, 3) and bool(torch.isfinite(ser_g).all()) and (ve_g > 0).all()


@pytest.mark.parametrize("channel", CHANNELS)
def test_cma_sweep_on_isi_channels(channel):
    """sweep_cma_dp with datagen='gpu': a cell alone equals the same cell in a 3-cell batch, bitwise; datagen='gpu_batched' runs."""
    from vae_equalizer_b200 import sweep
    cells = [dict(c, lr_optim=1e-5) for c in CELLS]
    args = ("64-QAM", 2, 25, 100, 3000, 3, 20, channel, COMMON["symb_rate"], COMMON["tau_cd"], COMMON["tau_pmd"], COMMON["phiIQ"], 2)
    ser, _, var = sweep.sweep_cma_dp(cells, *args, kind="CMAbatch", datagen="gpu")
    ser1, _, var1 = sweep.sweep_cma_dp(cells[2:], *args, kind="CMAbatch", datagen="gpu")
    assert torch.equal(ser1[0], ser[2]) and torch.equal(var1[0], var[2])
    assert bool(torch.isfinite(ser).all()) and float(ser.max()) <= 1.0
    ser_g, _, _ = sweep.sweep_cma_dp(cells, *args, kind="CMAbatch", datagen="gpu_batched")
    assert ser_g.shape == (3, 4, 3) and bool(torch.isfinite(ser_g).all())


def test_run_dp_sweep_on_h2_writes_and_reloads_checkpoints(tmp_path):
    from vae_equalizer_b200 import sweep
    lists = dict(nu_vec=[0.0270955], symb_rate_vec=[90e9], theta_vec=[np.pi / 10], theta_diff_vec=[0.0], SNR_vec=[20, 26], M_vec=[25],
                 batch_len_vec=[100], flex_step_vec=[20], lr_optim_vec=[2.5e-3, 2e-3])
    ck = str(tmp_path / "ck")
    a = sweep.run_dp_sweep(channel="h2", iter=2, num_frames=2, N_frame_max=1500, N_lrhalf=170, checkpoint_dir=ck, **lists)
    assert a[0].shape == (4, 2, 1, 1, 1, 1, 2, 1, 1, 1, 2, 2)
    assert torch.isfinite(a[0]).all() and float(a[0].max()) <= 1.0 and (a[1] > 0).all()

    def no_run(*args, **kw):
        raise AssertionError("a checkpointed set was recomputed")

    b = sweep.run_dp_sweep(channel="h2", iter=2, num_frames=2, N_frame_max=1500, N_lrhalf=170, checkpoint_dir=ck, runner=no_run,
                           device="cuda", **lists)
    assert all(torch.equal(x.cpu(), y.cpu()) for x, y in zip(a, b))


def test_vae_le_lowers_its_soft_demapper_ser_on_h1():
    """Convergence sanity check on the device-generated h1 signal: three 16-QAM VAE-LE cells at 25 dB SNR, 10 frames of 10 000 symbols.
    On a B200 their soft-demapper SER went from 0.862-0.872 in the first frame to 0.411-0.436 in the last (the host generator's
    frames follow the same descent); the gates leave about 0.15 of margin on each side."""
    from vae_equalizer_b200.sweep import sweep_vae_dp
    cells = [dict(SNR=25, nu=0.0, lr_optim=2.5e-3, theta=th, theta_diff=0.0, seed=s) for s, th in ((0, 0.3), (1, -0.4), (3, 0.0))]
    ser, _, _ = sweep_vae_dp(cells, "16-QAM", 2, 25, 100, 10000, 10, channel="h1", kind="VAE", N_lrhalf=1000, datagen="gpu", **COMMON)
    soft = ser[:, 2:].mean(1).cpu()                                       # rows 2, 3: soft demapper, per pol
    assert (soft[:, 0] > 0.75).all() and (soft[:, -1] < 0.6).all(), soft.tolist()
