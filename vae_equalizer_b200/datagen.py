"""Synthetic dual-polarisation test signal (host side): PCS symbols -> RRC pulse -> channel IR ->
residual CD / PMD / polarisation rotation / IQ phase -> AWGN.  Counterpart of the reference's
generate_data_shaping / simulate_channel / simulate_dispersion / rrcfir
(optical_DP_channel/shared_funcs.py:27-90).  The reference draws from unseeded numpy generators, so
parity here is statistical; pass `rng` for reproducible runs.  `generate_data_gpu` is the device
generator used by the benchmark (same statistics, torch.fft on the GPU); it takes the channel presets
'h0', 'h1' and 'h2' through `h_channel`."""
from __future__ import annotations

import numpy as np
import torch

from ._lib import device_guard as _device_guard

PULSE_SPAN, ROLLOFF = 8, 0.1          # sf:66-67


def rrcfir(T, sps, beta):
    t = np.arange(-T * sps / 2, T * sps / 2, 1 / sps, dtype=np.float32)
    with np.errstate(divide="ignore", invalid="ignore"):
        num = np.sin(np.pi * t * (1 - beta)) + 4 * beta * t * np.cos(np.pi * t * (1 + beta))
        h = num / (np.pi * t * (1 - (4 * beta * t) ** 2))
    h[np.abs(t) == 1 / 4 / beta] = beta / np.sqrt(2) * ((1 + 2 / np.pi) * np.sin(np.pi / 4 / beta) + (1 - 2 / np.pi) * np.cos(np.pi / 4 / beta))
    h[t == 0] = 1 + beta * (4 / np.pi - 1)
    return h / np.linalg.norm(h)


def rcfir(T, sps, beta):
    t = np.arange(-T * sps / 2, T * sps / 2, 1 / sps, dtype=np.float32)
    with np.errstate(divide="ignore", invalid="ignore"):
        h = np.sinc(t) * np.cos(np.pi * beta * t) / (1 - (2 * beta * t) ** 2)
    h[np.abs(t) == 1 / 2 / beta] = np.pi / 4 * np.sinc(1 / (2 * beta))
    return h / np.linalg.norm(h)


def jones_response(n, symb_rate, sps, tau_cd, tau_pmd, phiIQ, theta):
    """Per-bin 2x2 transfer matrix R^T diag(e_pmd, 1/e_pmd) R and the CD phase (sf:41-50)."""
    f = np.fft.fftfreq(n, 1 / symb_rate / sps)
    e_cd = np.exp(1j * 2 * (np.pi * f) ** 2 * tau_cd)
    e_pmd = np.exp(1j * np.pi * tau_pmd * f)
    c, s = np.cos(theta), np.sin(theta)
    e0, e1 = np.exp(-1j * np.asarray(phiIQ))
    R = ((c * e0, s * e0), (-s * e1, c * e1))
    Rt = ((c * e0, -s * e0), (s * e1, c * e1))
    d = (e_pmd, 1 / e_pmd)
    H = [[sum(Rt[a][k] * d[k] * R[k][b] for k in range(2)) for b in range(2)] for a in range(2)]
    return H, e_cd


def simulate_dispersion(rx, symb_rate, sps, tau_cd, tau_pmd, phiIQ, theta):
    X = np.fft.fft(rx, axis=1)
    H, e_cd = jones_response(rx.shape[1], symb_rate, sps, tau_cd, tau_pmd, phiIQ, theta)
    Y = np.stack(((H[0][0] * X[0] + H[0][1] * X[1]) * e_cd, (H[1][0] * X[0] + H[1][1] * X[1]) * e_cd))
    return np.complex64(np.fft.ifft(Y, axis=1))


def simulate_channel(tx_up, h_pulse, h_channel):
    return np.stack([np.convolve(np.convolve(row, h_pulse, mode="valid"), h_channel, mode="valid") for row in tx_up]).astype(np.complex64)


def generate_data_shaping(N, amps, SNR, h_channel, P, pol, symb_rate, sps, tau_cd, tau_pmd, phiIQ, theta, device, rng=None):
    """rx (2,2,sps*N) f32, data (2,2,N) f16, sigma_n  -- same contract as the reference (sf:65-90)."""
    rng = np.random.default_rng() if rng is None else rng
    M = len(h_channel)
    n_conv = N + M + 4 * PULSE_SPAN
    data = rng.choice(amps, (pol * 2, n_conv), p=P)
    tx_up = np.zeros((pol, sps * (n_conv - 1) + 1), dtype=np.complex64)
    tx_up[:, ::sps] = data[0::pol, :] + 1j * data[1::pol, :]
    sig = simulate_channel(tx_up, rrcfir(PULSE_SPAN, sps, ROLLOFF), h_channel)
    sig = simulate_dispersion(sig, symb_rate, sps, tau_cd, tau_pmd, phiIQ, theta)
    sigma_n = np.sqrt(np.mean(np.abs(sig) ** 2) * sps / 2 / 10 ** (SNR / 10))
    sig = sig + sigma_n * (rng.standard_normal(sig.shape) + 1j * rng.standard_normal(sig.shape))
    sig = sig[:, :sps * N]
    rx = torch.from_numpy(np.stack((sig.real, sig.imag), axis=1).astype(np.float32)).to(device)
    sl = slice(PULSE_SPAN + M - 1, N + PULSE_SPAN + M - 1)
    tx = torch.from_numpy(np.stack((data[0::pol, sl], data[1::pol, sl]), axis=1)).to(device, torch.float16)
    return rx.contiguous(), tx.contiguous(), sigma_n


def generate_data_gpu(N, amps, SNR, P, sps, theta, device, seed, symb_rate=90e9, tau_cd=-26e-24,
                      tau_pmd=0.1e-12 * np.sqrt(1000), phiIQ=(0.0314, 0.0314), h_channel=None):
    """Device-side generator with the same signal model; statistics, not bits, match the host generator.  h_channel: the upsampled
    channel IR that init returns (None: the optical channel 'h0').  One run of generate_frames_gpu (cached channel terms, no
    per-call host FFT-grid work)."""
    rx, tx, sigma_n = generate_frames_gpu(N, amps, [SNR], np.asarray(P)[None], sps, [theta], device, seed, symb_rate=symb_rate,
                                          tau_cd=tau_cd, tau_pmd=tau_pmd, phiIQ=phiIQ, h_channel=h_channel)
    return rx[0], tx[0], float(sigma_n[0])


def composite_filter(h_channel, sps):
    """rrcfir (*) h_channel in float64: simulate_channel's two 'valid' convolutions in a row are one 'valid' convolution with it."""
    return np.convolve(rrcfir(PULSE_SPAN, sps, ROLLOFF).astype(np.complex128), np.asarray(h_channel, dtype=np.complex64).astype(np.complex128))


def _optical_only(h_channel):
    """True for channel 'h0' (h_channel None or the one unit tap init returns): the real RRC pulse is the whole 'valid' filter."""
    return h_channel is None or (np.size(h_channel) == 1 and complex(np.asarray(h_channel).reshape(-1)[0]) == 1)


def _channel_len(h_channel):
    """len(h_channel) of the reference's frame geometry (sf:72, 89): n_conv = N + M + 4 T, tx = levels [T + M - 1, T + M - 1 + N)."""
    return 1 if h_channel is None else int(np.size(h_channel))


_GPU_CACHE: dict = {}


def _cached_channel_terms(n_up, symb_rate, sps, tau_cd, tau_pmd, device, h_channel=None):
    """Per-bin CD phase and PMD term exp(j pi tau_pmd f) (sf:41-45) and the spectrum of the 'valid' filter, cached per frame geometry
    and filter.  The filter is the real RRC pulse for 'h0' and the composite rrcfir (*) h_channel, cast once to complex64, otherwise;
    its device taps (last entry) are float32, real for 'h0' and (re, im) interleaved otherwise."""
    optical = _optical_only(h_channel)
    key = (n_up, float(symb_rate), sps, float(tau_cd), float(tau_pmd), str(device),
           None if optical else np.asarray(h_channel, dtype=np.complex64).tobytes())
    hit = _GPU_CACHE.get(key)
    if hit is None:
        filt = rrcfir(PULSE_SPAN, sps, ROLLOFF) if optical else composite_filter(h_channel, sps).astype(np.complex64)
        n = n_up - len(filt) + 1                                                     # length after the 'valid' convolution
        f = np.fft.fftfreq(n, 1 / symb_rate / sps)
        e_cd = torch.as_tensor(np.exp(1j * 2 * (np.pi * f) ** 2 * tau_cd), device=device).to(torch.complex64)
        e_pmd = torch.as_tensor(np.exp(1j * np.pi * tau_pmd * f), device=device).to(torch.complex64)
        pulse = torch.as_tensor(filt, device=device).to(torch.complex64)
        n_fft = n_up + pulse.numel() - 1
        if optical:
            taps = torch.as_tensor(filt, device=device).to(torch.float32).contiguous()
        else:
            taps = torch.view_as_real(pulse).reshape(-1).contiguous()
        hit = (e_cd, e_pmd, 1 / e_pmd, torch.fft.fft(pulse, n_fft), n_fft, pulse.numel(), (e_pmd * e_cd).contiguous(), (e_cd / e_pmd).contiguous(),
               taps)
        if len(_GPU_CACHE) > 16:
            _GPU_CACHE.clear()
        _GPU_CACHE[key] = hit
    return hit


def _per_run(v, R, dev):
    """Per-run parameter as a float32 device tensor (R,); a tensor already on the device is used as it is."""
    if torch.is_tensor(v):
        return v.to(dev, torch.float32).reshape(-1).expand(R).contiguous()
    return torch.as_tensor(np.broadcast_to(np.asarray(v, dtype=np.float64), (R,)).copy(), dtype=torch.float32, device=dev)


def _cached_amps(amps, dev):
    a = np.ascontiguousarray(np.asarray(amps, dtype=np.float32))
    key = ("amps", a.tobytes(), str(dev))
    hit = _GPU_CACHE.get(key)
    if hit is None:
        hit = _GPU_CACHE[key] = torch.as_tensor(a, device=dev)
    return hit


_FORCE_TORCH = False      # tests: run the torch.fft formulation on the GPU as the checker of the CUDA kernels


@_device_guard
def _generate_frames_cuda(N, amps, SNR, P, theta, dev, seed, symb_rate, tau_cd, tau_pmd, phiIQ, return_parts=False, h_channel=None):
    """generate_frames_gpu on a CUDA device: the element-wise stages are the vaeq_gen_* kernels (csrc/datagen.cu), the two DFTs of the
    dispersion step are torch.fft (cuFFT).  6.6 -> ~3 ms for 592 runs x 10 000 symbols (profiles/r01d_*); the ISI channels in
    profiles/r03_datagen_isi.txt."""
    from . import _lib
    lib = _lib.load()
    sps, R, n_lev = 2, int(P.shape[0]), int(P.shape[1])
    f32 = torch.float32
    snr, th = _per_run(SNR, R, dev), _per_run(theta, R, dev)      # device tensors pass through: no host->device copy (and no sync) per frame
    amps_t = _cached_amps(amps, dev)
    M = _channel_len(h_channel)
    n_conv = N + M + 4 * PULSE_SPAN
    n_up = sps * (n_conv - 1) + 1
    terms = _cached_channel_terms(n_up, symb_rate, sps, tau_cd, tau_pmd, dev, h_channel)
    n_pulse, Pcd, Picd, pulse = terms[5], terms[6], terms[7], terms[8]
    n = 2 * n_conv - n_pulse
    skey = ("jones_terms_over_n", n, float(symb_rate), float(tau_cd), float(tau_pmd), str(dev))
    scaled = _GPU_CACHE.get(skey)
    if scaled is None:                                        # the 1/n of the inverse DFT folded into the per-bin terms: the Jones kernel's output is
        scaled = _GPU_CACHE[skey] = ((Pcd / n).contiguous(), (Picd / n).contiguous())      # linear in them, and ifft(norm="forward") skips its scaling pass
    Pcd, Picd = scaled
    st = _lib.current_stream()
    seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    lev = torch.empty(R, 4, n_conv, dtype=f32, device=dev)
    tx = torch.empty(R, 2, 2, N, dtype=torch.float16, device=dev)
    P = P.contiguous()
    _lib.check(lib.vaeq_gen_levels(amps_t.data_ptr(), P.data_ptr(), n_lev, n_conv, N, PULSE_SPAN + M - 1, seed, lev.data_ptr(), tx.data_ptr(), R,
                                   st), "vaeq_gen_levels")
    sig = torch.empty(R, 2, n, dtype=torch.complex64, device=dev)
    if _optical_only(h_channel):
        _lib.check(lib.vaeq_gen_pulse(lev.data_ptr(), pulse.data_ptr(), n_pulse, n_conv, sig.data_ptr(), R, st), "vaeq_gen_pulse")
    else:
        _lib.check(lib.vaeq_gen_pulse_cplx(lev.data_ptr(), pulse.data_ptr(), n_pulse, n_conv, sig.data_ptr(), R, st), "vaeq_gen_pulse_cplx")
    X = torch.fft.fft(sig, dim=-1)
    ph = np.asarray(phiIQ)
    phi0, phi1 = float(np.real(ph[0])), float(np.real(ph[1]))
    _lib.check(lib.vaeq_gen_jones(X.data_ptr(), Pcd.data_ptr(), Picd.data_ptr(), th.data_ptr(), phi0, phi1, n, R, st), "vaeq_gen_jones")
    sig = torch.fft.ifft(X, dim=-1, norm="forward")
    power = torch.linalg.vector_norm(torch.view_as_real(sig).reshape(R, -1), dim=1).square() / (2 * n)       # mean |sig|^2 over both pols  (sf:83)
    sigma_n = torch.sqrt(power * sps / 2 / 10 ** (snr / 10))
    rx = torch.empty(R, 2, 2, sps * N, dtype=f32, device=dev)
    _lib.check(lib.vaeq_gen_noise(sig.data_ptr(), sigma_n.contiguous().data_ptr(), seed ^ 0x9E3779B97F4A7C15, n, sps * N, rx.data_ptr(), R, st),
               "vaeq_gen_noise")
    if return_parts:
        return rx, tx, sigma_n, lev, sig
    return rx, tx, sigma_n


def _frames_torch_from_levels(lev, N, sps, theta, symb_rate, tau_cd, tau_pmd, phiIQ, h_channel=None):
    """The noise-free part of generate_frames_gpu's torch.fft formulation for GIVEN amplitude levels lev (R,4,n_conv): checker of the
    CUDA kernels (tests/test_frames_gpu.py, tests/test_datagen_isi_gpu.py)."""
    dev, R = lev.device, lev.shape[0]
    th = _per_run(theta, R, dev)
    n_conv = lev.shape[-1]
    sym = torch.complex(lev[:, 0::2], lev[:, 1::2])
    n_up = sps * (n_conv - 1) + 1
    up = torch.zeros(R, 2, n_up, dtype=torch.complex64, device=dev)
    up[:, :, ::sps] = sym
    e_cd, e_pmd, e_pmd_inv, pulse_f, n_fft, n_pulse = _cached_channel_terms(n_up, symb_rate, sps, tau_cd, tau_pmd, dev, h_channel)[:6]
    shaped = torch.fft.ifft(torch.fft.fft(up, n_fft) * pulse_f)[:, :, n_pulse - 1: n_up]
    return _jones_torch(shaped, th, e_cd, e_pmd, e_pmd_inv, phiIQ)


def _jones_torch(shaped, th, e_cd, e_pmd, e_pmd_inv, phiIQ):
    """H = R^T diag(e_pmd, 1/e_pmd) R with R = [[c e0, s e0], [-s e1, c e1]]  (sf:46-50), per run and per bin."""
    c, s = torch.cos(th)[:, None], torch.sin(th)[:, None]                            # (R,1)
    e0, e1 = np.exp(-1j * np.asarray(phiIQ, dtype=np.complex64))
    R00, R01, R10, R11 = c * complex(e0), s * complex(e0), -s * complex(e1), c * complex(e1)
    T00, T01, T10, T11 = c * complex(e0), -s * complex(e0), s * complex(e1), c * complex(e1)
    H00 = T00 * e_pmd * R00 + T01 * e_pmd_inv * R10
    H01 = T00 * e_pmd * R01 + T01 * e_pmd_inv * R11
    H10 = T10 * e_pmd * R00 + T11 * e_pmd_inv * R10
    H11 = T10 * e_pmd * R01 + T11 * e_pmd_inv * R11
    X = torch.fft.fft(shaped, dim=-1)
    return torch.fft.ifft(torch.stack(((H00 * X[:, 0] + H01 * X[:, 1]) * e_cd, (H10 * X[:, 0] + H11 * X[:, 1]) * e_cd), dim=1), dim=-1)


def generate_frames_gpu(N, amps, SNR, P, sps, theta, device, seed, symb_rate=90e9, tau_cd=-26e-24,
                        tau_pmd=0.1e-12 * np.sqrt(1000), phiIQ=(0.0314, 0.0314), h_channel=None):
    """R frames at once (one batched launch sequence for all runs of a sweep): SNR (R,), P (R,n), theta (R,) per run, one
    seed and one channel for the batch.  Same signal model as generate_data_gpu; h_channel is the upsampled channel IR init returns
    (None: 'h0'), and the frame geometry is generate_data_shaping's (n_conv = N + len(h_channel) + 4 PULSE_SPAN, the FFT length
    2 n_conv - K for the K-tap 'valid' filter, tx from level PULSE_SPAN + len(h_channel) - 1).  Returns rx (R,2,2,sps*N) f32,
    tx (R,2,2,N) f16, sigma_n (R,)."""
    dev = torch.device(device)
    P = P.to(dev, torch.float32) if torch.is_tensor(P) else torch.as_tensor(np.asarray(P), dtype=torch.float32, device=dev)
    if P.dim() == 1:
        P = P[None]
    R = P.shape[0]
    if dev.type == "cuda" and sps == 2 and not _FORCE_TORCH:
        return _generate_frames_cuda(N, amps, SNR, P, theta, dev, seed, symb_rate, tau_cd, tau_pmd, phiIQ, h_channel=h_channel)
    return _generate_frames_torch(N, amps, SNR, P, sps, theta, dev, seed, symb_rate, tau_cd, tau_pmd, phiIQ, h_channel=h_channel)


def _generate_frames_torch(N, amps, SNR, P, sps, theta, dev, seed, symb_rate, tau_cd, tau_pmd, phiIQ, return_parts=False, h_channel=None):
    """generate_frames_gpu as torch ops (the CPU path, and the checker of the CUDA path); with return_parts also the levels
    (R,4,n_conv) and the noise-free signal (R,2,n) complex64."""
    R = P.shape[0]
    snr = _per_run(SNR, R, dev)
    g = torch.Generator(device=dev).manual_seed(int(seed))
    M = _channel_len(h_channel)
    n_conv = N + M + 4 * PULSE_SPAN
    idx = torch.multinomial(P, 4 * n_conv, True, generator=g).view(R, 4, n_conv)
    lev = torch.as_tensor(np.asarray(amps), dtype=torch.float32, device=dev)[idx]
    sig = _frames_torch_from_levels(lev, N, sps, theta, symb_rate, tau_cd, tau_pmd, phiIQ, h_channel)
    sigma_n = torch.sqrt(torch.mean(sig.abs() ** 2, dim=(1, 2)) * sps / 2 / 10 ** (snr / 10))
    noise = torch.complex(torch.randn(sig.shape, device=dev, generator=g), torch.randn(sig.shape, device=dev, generator=g))
    noisy = (sig + sigma_n[:, None, None] * noise)[:, :, :sps * N]
    rx = torch.stack((noisy.real, noisy.imag), dim=2).to(torch.float32).contiguous()
    sl = slice(PULSE_SPAN + M - 1, N + PULSE_SPAN + M - 1)
    tx = torch.stack((lev[:, 0::2][:, :, sl], lev[:, 1::2][:, :, sl]), dim=2).to(torch.float16).contiguous()
    if return_parts:
        return rx, tx, sigma_n, lev, sig
    return rx, tx, sigma_n
