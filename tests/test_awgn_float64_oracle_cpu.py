"""The float64 yardstick of the AWGN VAE-LE step (oracle.vaeq_oracle.awgn_step at torch.float64): it agrees with the reference goldens,
and its autograd gradient is the derivative of its loss.  CPU only; tests/test_awgn_step_float64_gpu.py measures the CUDA step with it."""
import os

import numpy as np
import pytest
import torch

from oracle import vaeq_oracle as O

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
F64 = torch.float64


def rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


@pytest.mark.parametrize("name", ["awgn_16qam_M25_B350", "awgn_64qam_M9_B200"])
def test_float64_oracle_matches_reference_golden(name):
    """Every step of the golden from the reference's own taps before it (teacher-forced), at the tolerances the CUDA step is held to in
    test_awgn_trajectory_against_reference_golden."""
    g = dict(np.load(os.path.join(GOLDEN, name + ".npz")))
    am, var = float(np.float32(g["amp_mean"])), float(np.float32(g["var"]))
    for s in range(g["rx"].shape[0]):
        W, h = (g["W0"], g["h0"]) if s == 0 else (g["W"][s - 1], g["h"][s - 1])
        r = O.awgn_step(g["rx"][s], W, h, g["amp"], g["P"], am, var, dtype=F64)
        assert np.abs(r["out"].numpy() - g["out"][s]).max() < 5e-6, s
        assert np.abs(r["q"].numpy() - g["q"][s]).max() < 5e-5, s
        assert rel(r["loss"], g["loss"][s]) < 1e-4, s
        assert rel(r["gW"], g["gW"][s]) < 2e-4 and rel(r["gh"], g["gh"][s]) < 2e-4, s


def test_float32_path_unchanged_by_dtype_parameter():
    """awgn_step at float32 is the op-by-op reference: bit-identical to awgn_forward + awgn_loss + backward on float32 leaves."""
    g = dict(np.load(os.path.join(GOLDEN, "awgn_16qam_M25_B350.npz")))
    T = torch.from_numpy
    am, var = float(g["amp_mean"]), float(g["var"])
    W, h = T(g["W0"]).clone().requires_grad_(True), T(g["h0"]).clone().requires_grad_(True)
    q, out = O.awgn_forward(T(g["rx"][0]), W, T(g["amp"]), am, var, 2)
    loss = O.awgn_loss(q, T(g["rx"][0]), h, T(g["amp"]), T(g["P"]))
    loss.backward()
    r = O.awgn_step(g["rx"][0], g["W0"], g["h0"], g["amp"], g["P"], am, var)
    assert r["q"].dtype == torch.float32
    for k, v in (("out", out), ("q", q), ("loss", loss), ("gW", W.grad), ("gh", h.grad)):
        assert torch.equal(r[k], v.detach()), k


@pytest.mark.parametrize("mod,M,B,channel,SNR,nu", [("4-QAM", 5, 64, "h1", 10.0, 0.0), ("64-QAM", 25, 350, "h2", 20.0, 0.03)])
def test_float64_gradient_is_derivative_of_loss(mod, M, B, channel, SNR, nu):
    """Central difference of the float64 loss along random directions in W and in h against the autograd gradient."""
    from vae_equalizer_b200.awgn import generate_data
    from vae_equalizer_b200.constants import awgn_constants, upsampled_channel
    hc = upsampled_channel(channel, 2)
    amps, P, am, var = awgn_constants(mod, nu, SNR)
    rng = np.random.default_rng(M * 1000 + B)
    rx, _ = generate_data(B, (len(hc) - 1) // 2 + 1, amps, SNR, hc, 2, "cpu", P, rng=rng)
    W = np.zeros((1, 2, M))
    W[0, 0, M // 2] = 1.0
    h = np.zeros((2, M))
    h[0, M // 2] = 1.0
    W, h = W + 0.05 * rng.standard_normal(W.shape), h + 0.05 * rng.standard_normal(h.shape)
    args = (amps, P, am, var)
    r = O.awgn_step(rx, W, h, *args, dtype=F64)
    loss = lambda W_, h_: float(O.awgn_step(rx, W_, h_, *args, dtype=F64, want_grads=False)["loss"])
    eps = 1e-6
    for _ in range(3):
        for which, grad in (("W", r["gW"].numpy()), ("h", r["gh"].numpy())):
            d = rng.standard_normal(grad.shape)
            d /= np.linalg.norm(d)
            if which == "W":
                fd = (loss(W + eps * d, h) - loss(W - eps * d, h)) / (2 * eps)
            else:
                fd = (loss(W, h + eps * d) - loss(W, h - eps * d)) / (2 * eps)
            ad = float((grad * d).sum())
            err = abs(fd - ad) / np.linalg.norm(grad)
            print(f"{mod} M={M} B={B} d{which}: autograd {ad:.6e} central difference {fd:.6e} rel err {err:.1e}")
            assert err < 1e-6, (which, ad, fd)


@pytest.mark.parametrize("amsgrad", [False, True])
def test_adam_restatement_matches_torch_optim(amsgrad):
    """oracle.closed_form.AdamState against torch.optim.Adam on the CPU, each of 8 steps from torch's own state (gradients shrink from
    step 5 on, so v falls below its running max): exp_avg bit for bit (torch's lerp_ is one fused multiply-add), the rest within 2 ulp
    (torch fuses addcmul_ and addcdiv_ differently on each device)."""
    from oracle import closed_form as CF
    gen = torch.Generator().manual_seed(3 + amsgrad)
    p = torch.nn.Parameter(torch.randn(4096, generator=gen))
    opt = torch.optim.Adam([p], lr=3e-3, amsgrad=amsgrad)
    ad = CF.AdamState((4096,), amsgrad=amsgrad)
    for s in range(8):
        p0 = p.detach().numpy().copy()
        if s:
            st = opt.state[p]
            ad.m, ad.v = st["exp_avg"].numpy().copy(), st["exp_avg_sq"].numpy().copy()
            if amsgrad:
                ad.vmax = st["max_exp_avg_sq"].numpy().copy()
        g = torch.randn(4096, generator=gen) * (0.1 if s >= 4 else 1.0)
        p.grad = g.clone()
        opt.step()
        pn = ad.update(p0, g.numpy(), 3e-3)
        st = opt.state[p]
        assert np.array_equal(st["exp_avg"].numpy(), ad.m), s
        # p within 2 ulp of the largest of p before, p after and the step: where the step nearly cancels p, an ulp of the step is many of p
        p1 = p.detach().numpy()
        pairs = [(st["exp_avg_sq"].numpy(), ad.v, ad.v), (p1, pn, np.maximum(np.abs(p0), np.abs(p1 - p0)))]
        pairs += [(st["max_exp_avg_sq"].numpy(), ad.vmax, ad.vmax)] if amsgrad else []
        for a, b, c in pairs:
            assert (np.abs(a.astype(np.float64) - b) <= 2 * np.spacing(np.maximum.reduce([np.abs(a), np.abs(b), np.abs(c)]))).all(), s
    if amsgrad:
        assert (ad.vmax > ad.v).any()
