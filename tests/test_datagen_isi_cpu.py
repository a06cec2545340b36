"""The device generator's signal model on the ISI channels 'h1' and 'h2', through its torch.fft formulation on the CPU
(datagen._generate_frames_torch, the path generate_frames_gpu takes without a GPU): the noise-free signal against a float64
restatement of simulate_channel + simulate_dispersion, the reference's frame geometry (tx offset, frame and FFT lengths), sigma_n,
and the channel plumbing of the sweep's frame source.  'h0' stays bitwise on its old path."""
import numpy as np
import pytest
import torch

import datagen_ref as ref

CPU = torch.device("cpu")


def consts(mod="64-QAM", nu=0.0270955):
    from vae_equalizer_b200.constants import init
    k = init("h0", mod, "cpu", nu, 2, 25, 23)
    return k[4], np.asarray(k[2], dtype=np.float32)


@pytest.mark.parametrize("channel", ["h1", "h2"])
def test_torch_formulation_matches_float64_signal_model(channel):
    from vae_equalizer_b200 import datagen as dg
    from vae_equalizer_b200.constants import upsampled_channel
    h = upsampled_channel(channel, 2)
    amps, P = consts()
    N, R, sps = 2500, 3, 2
    # an 'h0' frame whose upsampled length equals the ISI frame's comes first: the cached channel terms must not be shared
    dg.generate_frames_gpu(N + len(h) - 1, amps, [23.0], P[None], sps, [0.3], "cpu", 1)
    snr, theta = [23.0, 13.0, 30.0], [0.3, 1.0, -0.7]
    rx, tx, sigma, lev, sig = dg._generate_frames_torch(N, amps, snr, torch.as_tensor(np.stack([P] * R)), sps, theta, CPU, 5, *ref.ARGS,
                                                        return_parts=True, h_channel=h)
    K = 32 + len(h) - 1
    n_conv = N + len(h) + 4 * dg.PULSE_SPAN
    assert lev.shape == (R, 4, n_conv) and sig.shape == (R, 2, 2 * n_conv - K) and K == {"h1": 40, "h2": 38}[channel]
    assert rx.shape == (R, 2, 2, sps * N) and tx.shape == (R, 2, 2, N) and tx.dtype == torch.float16
    sig_ref = ref.noise_free_signal(lev.numpy(), channel, theta)
    assert float(np.abs(sig.numpy() - sig_ref).max()) < 3e-5 * float(np.abs(sig_ref).max())
    off = dg.PULSE_SPAN + len(h) - 1                                      # sf:89
    for p in range(2):
        for c in range(2):
            assert torch.equal(tx[:, p, c], lev[:, 2 * p + c, off:off + N].to(torch.float16))
    pw = (np.abs(sig.numpy().astype(np.complex128)) ** 2).mean(axis=(1, 2))
    np.testing.assert_allclose(sigma.numpy(), np.sqrt(pw * sps / 2 / 10 ** (np.asarray(snr) / 10)), rtol=1e-5)
    z = (rx - torch.stack((sig.real, sig.imag), dim=2)[..., :sps * N]) / sigma[:, None, None, None]
    for r in range(R):
        assert abs(float(z[r].mean())) < 0.03 and abs(float(z[r].var()) - 1) < 0.03


def test_fft_lengths_at_ten_thousand_symbols():
    """The frame lengths of the three presets at N = 10^4: the dispersion step's DFT runs over n = 2 n_conv - K samples."""
    from vae_equalizer_b200 import datagen as dg
    from vae_equalizer_b200.constants import upsampled_channel
    amps, P = consts()
    for channel, n in (("h0", 20034), ("h1", 20042), ("h2", 20040)):
        _, _, _, _, sig = dg._generate_frames_torch(10000, amps, [20.0], torch.as_tensor(P[None]), 2, [0.0], CPU, 1, *ref.ARGS,
                                                    return_parts=True, h_channel=upsampled_channel(channel, 2))
        assert sig.shape[-1] == n, channel


def test_h0_channel_keyword_is_bitwise_the_default_path():
    from vae_equalizer_b200.constants import upsampled_channel
    from vae_equalizer_b200.datagen import generate_data_gpu, generate_frames_gpu
    amps, P = consts()
    args = (3000, amps, [23, 13, 23], np.stack([P] * 3), 2, [0.3, 0.3, 1.0], "cpu", 11)
    a = generate_frames_gpu(*args)
    b = generate_frames_gpu(*args, h_channel=upsampled_channel("h0", 2))
    assert all(torch.equal(x, y) for x, y in zip(a, b))
    c, d = generate_data_gpu(1500, amps, 20, P, 2, 0.3, "cpu", 7), generate_data_gpu(1500, amps, 20, P, 2, 0.3, "cpu", 7, h_channel=[1.0])
    assert torch.equal(c[0], d[0]) and torch.equal(c[1], d[1]) and c[2] == d[2]


@pytest.mark.parametrize("channel", ["h1", "h2"])
def test_single_run_generator_is_one_run_of_the_batched_generator(channel):
    from vae_equalizer_b200.constants import upsampled_channel
    from vae_equalizer_b200.datagen import generate_data_gpu, generate_frames_gpu
    amps, P = consts("16-QAM", 0.0)
    h = upsampled_channel(channel, 2)
    a, ta, sa = generate_data_gpu(1500, amps, 18, P, 2, 0.3, "cpu", 7, h_channel=h)
    b, tb, sb = generate_frames_gpu(1500, amps, [18], P, 2, [0.3], "cpu", 7, h_channel=h)
    assert torch.equal(a, b[0]) and torch.equal(ta, tb[0]) and sa == float(sb[0])


@pytest.mark.parametrize("datagen", ["gpu", "gpu_batched"])
def test_dp_frame_source_passes_the_channel(datagen):
    """sweep._dp_source on 'h1' (formerly rejected for the device generators): frames of the h1 geometry, each cell's frame the
    generator's output for the cell's key."""
    from vae_equalizer_b200 import sweep
    from vae_equalizer_b200.constants import upsampled_channel
    from vae_equalizer_b200.datagen import generate_data_gpu, generate_frames_gpu
    h = upsampled_channel("h1", 2)
    cells = [dict(SNR=20, nu=0.0270955, theta=0.3, theta_diff=0.1, seed=3), dict(SNR=24, nu=0.0, theta=-0.2, theta_diff=0.0, seed=4)]
    N, F = 800, 2
    consts_, P, _, _, frames = sweep._dp_source(cells, "64-QAM", 2, 25, "h1", N, F, datagen, CPU, *ref.ARGS)
    frames = list(frames)
    assert len(frames) == F and np.array_equal(consts_[0][1], h)
    amps = consts_[0][4]
    for f, (rx, tx) in enumerate(frames):
        assert rx.shape == (2, 2, 2, 2 * N) and tx.shape == (2, 2, 2, N)
        th = [c["theta"] + f * c["theta_diff"] for c in cells]
        if datagen == "gpu_batched":
            rx_e, tx_e, _ = generate_frames_gpu(N, amps, [c["SNR"] for c in cells], P, 2, th, CPU, 3 * 100003 + f, *ref.ARGS, h_channel=h)
            assert torch.allclose(rx, rx_e, atol=1e-6, rtol=0) and torch.equal(tx, tx_e)
        else:
            for r, c in enumerate(cells):
                rx_e, tx_e, _ = generate_data_gpu(N, amps, c["SNR"], P[r].numpy(), 2, th[r], CPU, c["seed"] * 100003 + f, *ref.ARGS, h_channel=h)
                assert torch.allclose(rx[r], rx_e, atol=1e-6, rtol=0) and torch.equal(tx[r], tx_e)
