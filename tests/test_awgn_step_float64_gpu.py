"""The AWGN single-polarisation VAE-LE step (csrc/awgn.cu awgn_step_body, behind AWGNEqualizer and AWGNEqualizerRuns) against a float64
reference: oracle.vaeq_oracle.awgn_step at torch.float64 (forward + loss + autograd, pinned to the reference goldens and to central
differences by tests/test_awgn_float64_oracle_cpu.py).

Every comparison is one step, or steps teacher-forced from the kernel's own state.  The gate of each quantity is
max(bound, 2 x the error of the float32 oracle), the reference's own arithmetic, against the same float64 values: the kernel has to be
as good as the reference wherever the bound itself is below what float32 can do.  Bounds (DESIGN.md §2): out 5e-6 and q 5e-5 max abs,
loss 1e-5 relative, gW and gh 1e-4 relative to their max-norm."""
import numpy as np
import pytest
import torch

from oracle import closed_form as CF
from oracle import vaeq_oracle as O

pytestmark = pytest.mark.gpu
F64 = torch.float64
MODS = {2: "4-QAM", 4: "16-QAM", 8: "64-QAM"}
BOUND = dict(out=5e-6, q=5e-5, loss=1e-5, gW=1e-4, gh=1e-4)


def _np(a):
    return a.detach().cpu().numpy().astype(np.float64) if torch.is_tensor(a) else np.asarray(a, np.float64)


def _err(key, a, b):
    a, b = _np(a).reshape(-1), _np(b).reshape(-1)
    d = np.abs(a - b).max()
    if key in ("out", "q"):
        return float(d)
    return float(d / max(np.abs(b).max(), 1e-30))


def _setup(n_lev, M, B, channel, SNR, nu, seed, pert=True, zero_head=False):
    """Driver inputs: rx from awgn.generate_data, constants rounded to the float32 the kernel sees, Dirac taps (+ 0.05 N(0,1))."""
    from vae_equalizer_b200.awgn import generate_data
    from vae_equalizer_b200.constants import awgn_constants, upsampled_channel
    hc = upsampled_channel(channel, 2)
    amps, P, am, var = awgn_constants(MODS[n_lev], nu, SNR)
    rng = np.random.default_rng(seed)
    rx, _ = generate_data(B, (len(hc) - 1) // 2 + 1, amps, SNR, hc, 2, "cpu", P, rng=rng)
    if zero_head:
        rx[:, :2 * M] = 0.0
    W = np.zeros((1, 2, M), np.float32)
    W[0, 0, M // 2] = 1.0
    h = np.zeros((2, M), np.float32)
    h[0, M // 2] = 1.0
    if pert:
        W = (W + 0.05 * rng.standard_normal(W.shape)).astype(np.float32)
        h = (h + 0.05 * rng.standard_normal(h.shape)).astype(np.float32)
    c = (np.asarray(amps, np.float32), np.asarray(P, np.float32), float(np.float32(am)), float(np.float32(var)))
    return rx.contiguous(), W, h, c


def _check(tag, got, rx, W, h, c, grads=True):
    """got: the kernel's out, q, loss (and gW, gh).  Prints the kernel's and the float32 oracle's error against float64 per quantity and
    asserts the gates and the hard decisions."""
    amps, P, am, var = c
    ref = O.awgn_step(rx, W, h, amps, P, am, var, dtype=F64, want_grads=grads)
    f32 = O.awgn_step(rx, W, h, amps, P, am, var, dtype=torch.float32, want_grads=grads)
    keys = ("out", "q", "loss", "gW", "gh") if grads else ("out", "q", "loss")
    errs = {k: (_err(k, got[k], ref[k]), _err(k, f32[k], ref[k])) for k in keys}
    print(tag + ": " + ", ".join(f"{k} {e:.2e} (fp32 oracle {o:.2e})" for k, (e, o) in errs.items()))
    for k, (e, o) in errs.items():
        assert e <= max(BOUND[k], 2 * o), (tag, k, e, o)
    # hard decisions per component wherever the float64 top-2 margin is clear; outputs that are exactly 0 tie by symmetry
    n = amps.size
    q64, qk, o64 = _np(ref["q"]), _np(got["q"]), _np(ref["out"])
    for comp in range(2):
        rows = slice(comp * n, (comp + 1) * n)
        top2 = np.sort(q64[rows], axis=0)[-2:]
        clear = (top2[1] - top2[0]) > 1e-4
        assert np.array_equal(qk[rows].argmax(0)[clear], q64[rows].argmax(0)[clear]), (tag, comp)
        live = o64[comp] != 0
        assert clear[live].mean() >= 0.999, (tag, comp, clear[live].mean())


def _equalizer(M, W, h, c):
    from vae_equalizer_b200.awgn import AWGNEqualizer
    amps, P, am, var = c
    return AWGNEqualizer(M, 2, amps, P, am, var, W0=torch.from_numpy(W), h0=torch.from_numpy(h))


def _fwd_bwd(eq, rx):
    q, out, loss, gW, gh = eq.forward_backward(rx.cuda())
    return dict(out=out.clone(), q=q.clone(), loss=loss.clone(), gW=gW.clone(), gh=gh.clone())


# (n_lev, M, B, channel, SNR dB, nu, taps perturbed, first 2M samples of rx zero)
STEP_CASES = [
    (2, 25, 350, "h1", 14.0, 0.0, True, False),      # driver default, every level count on both channels
    (4, 25, 350, "h1", 22.0, 0.05, True, False),
    (8, 25, 350, "h1", 8.0, 0.02, False, False),
    (2, 25, 350, "h2", 8.0, 0.1, False, False),
    (4, 25, 350, "h2", 14.0, 0.0, False, False),
    (8, 25, 350, "h2", 22.0, 0.0, True, False),
    (2, 1, 64, "h1", 14.0, 0.0, True, False),        # mh = 0
    (4, 9, 9, "h2", 22.0, 0.05, True, False),        # minimum B = M
    (8, 63, 63, "h1", 14.0, 0.0, True, False),       # VAEQ_MAX_TAPS at the minimum B
    (8, 25, 1023, "h1", 22.0, 0.02, True, False),    # around one stride of the 1024-thread CTA
    (8, 25, 1024, "h2", 8.0, 0.0, True, False),
    (8, 25, 1025, "h1", 14.0, 0.02, True, False),
    (4, 41, 3000, "h2", 14.0, 0.05, True, False),    # several strides
    (8, 63, 4097, "h1", 22.0, 0.02, True, False),    # widest taps, tail stride
    (2, 9, 8192, "h1", 8.0, 0.0, True, False),       # long serial tap-gradient sums
    (8, 9, 8192, "h2", 22.0, 0.0, True, False),
    (4, 25, 350, "h1", 14.0, 0.0, True, True),       # outputs exactly 0: sgn(0) = 0 in the backward through mean|out|
]


@pytest.mark.parametrize("n_lev,M,B,channel,SNR,nu,pert,zero_head", STEP_CASES)
def test_forward_backward_against_float64(n_lev, M, B, channel, SNR, nu, pert, zero_head):
    rx, W, h, c = _setup(n_lev, M, B, channel, SNR, nu, seed=1000 * M + B, pert=pert, zero_head=zero_head)
    got = _fwd_bwd(_equalizer(M, W, h, c), rx)
    if zero_head:
        assert int((got["out"] == 0).sum()) >= 2 * (M // 2)
    _check(f"{MODS[n_lev]} M={M} B={B} {channel} {SNR:g} dB nu={nu}{' zero head' if zero_head else ''}", got, rx, W, h, c)


@pytest.mark.parametrize("N", [15000, 50000])
@pytest.mark.parametrize("n_lev", [2, 4, 8])
def test_validation_forward_against_float64(n_lev, N):
    """AWGNEqualizer.forward over a whole validation frame (N_valid of the sweeps is 15000): the q every AWGN SER and GMI is computed
    from."""
    rx, W, h, c = _setup(n_lev, 25, N, "h1" if n_lev != 4 else "h2", 14.0 + n_lev, 0.02 * (n_lev == 8), seed=N + n_lev)
    q, out, loss = _equalizer(25, W, h, c).forward(rx.cuda())
    _check(f"forward {MODS[n_lev]} N={N}", dict(out=out, q=q, loss=loss), rx, W, h, c, grads=False)


def test_runs_forward_against_float64():
    """AWGNEqualizerRuns.forward, R = 3 runs with their own var, amp_mean, P, taps and data; rx is a view whose I and Q rows are 517
    samples farther apart than L, so the kernel's ld_rx and run stride are not those of a contiguous (R, 2, L) tensor."""
    from vae_equalizer_b200.awgn import AWGNEqualizerRuns
    R, M, N, pad = 3, 25, 15000, 517
    cases = [_setup(4, M, N, ("h1", "h2", "h1")[r], (10.0, 16.0, 21.0)[r], (0.0, 0.05, 0.1)[r], seed=70 + r) for r in range(R)]
    amps = cases[0][3][0]
    eqr = AWGNEqualizerRuns(R, M, 2, amps, np.stack([c[3][1] for c in cases]), [c[3][2] for c in cases], [c[3][3] for c in cases])
    buf = torch.full((R, 2, 2 * N + pad), float("nan"), device="cuda")
    for r, (rx, W, h, _) in enumerate(cases):
        buf[r, :, :2 * N] = rx.cuda()
        eqr.W[r], eqr.h[r] = torch.from_numpy(W).cuda(), torch.from_numpy(h).cuda()
    view = buf[:, :, :2 * N]
    assert view.stride(-2) == 2 * N + pad and not view.is_contiguous()
    q, out, loss = eqr.forward(view)
    for r, (rx, W, h, c) in enumerate(cases):
        _check(f"runs forward run {r}", dict(out=out[r], q=q[r], loss=loss[r]), rx, W, h, c, grads=False)


def _ulps(a, b, scale=0.0):
    """Largest |a - b| in ulp of max(|a|, |b|, scale): a parameter is measured against the step too, where the step nearly cancels it."""
    a, b = np.asarray(a, np.float32).reshape(-1), np.asarray(b, np.float32).reshape(-1)
    sp = np.spacing(np.maximum(np.maximum(np.abs(a), np.abs(b)), np.abs(np.asarray(scale, np.float32)).reshape(-1)))
    return float((np.abs(a.astype(np.float64) - b.astype(np.float64)) / sp).max())


@pytest.mark.parametrize("step0", [0, 10000])
def test_amsgrad_steps_teacher_forced(step0):
    """8 train_steps with lr_w != lr_h.  Before each: the kernel's gradients at the current state against float64; then the step against
    oracle.closed_form.AdamState(amsgrad=True) (torch's float32 update restated) fed with those gradients and the kernel's own Adam state.
    From step 5 on rx is halved, so that gradients shrink and v falls below its running max (the amsgrad branch)."""
    n_lev, M, B = 4, 25, 350
    lr_w, lr_h = float(np.float32(3e-3)), float(np.float32(1e-3))
    _, W, h, c = _setup(n_lev, M, B, "h1", 16.0, 0.05, seed=step0 + 5)
    eq = _equalizer(M, W, h, c)
    eq.adam.view(torch.int32)[12 * M] = step0
    for s in range(8):
        rx, _, _, _ = _setup(n_lev, M, B, "h1", 16.0, 0.05, seed=step0 + 100 + s)
        if s >= 4:
            rx = rx * 0.5
        W0, h0 = eq.W.cpu().numpy(), eq.h.cpu().numpy()
        buf = eq.adam.cpu().numpy()
        got = _fwd_bwd(eq, rx)
        _check(f"amsgrad step0={step0} step {s + 1}", got, rx, W0, h0, c)
        gW, gh = got["gW"].cpu().numpy(), got["gh"].cpu().numpy()
        eq.train_step(rx.cuda(), lr_w, lr_h)
        assert torch.equal(eq.gW.cpu(), got["gW"].cpu()) and torch.equal(eq.gh.cpu(), got["gh"].cpu())
        after = eq.adam.cpu().numpy()
        assert int(after[12 * M:12 * M + 1].view(np.int32)[0]) == step0 + s + 1
        for off, p0, g, lr, p1 in ((0, W0, gW, lr_w, eq.W), (6 * M, h0, gh, lr_h, eq.h)):
            ad = CF.AdamState(p0.shape, amsgrad=True)
            ad.t = step0 + s
            ad.m, ad.v, ad.vmax = (buf[off + i * 2 * M:off + (i + 1) * 2 * M].reshape(p0.shape).copy() for i in range(3))
            p_ref = ad.update(p0, g, lr)
            got_state = [after[off + i * 2 * M:off + (i + 1) * 2 * M] for i in range(3)]
            p1 = p1.cpu().numpy()
            u = dict(p=_ulps(p1, p_ref, np.maximum(np.abs(p0), np.abs(p1 - p0))), m=_ulps(got_state[0], ad.m), v=_ulps(got_state[1], ad.v),
                     vmax=_ulps(got_state[2], ad.vmax))
            assert max(u.values()) <= 2, (s, off, u)
    v, vmax = after[2 * M:4 * M], after[4 * M:6 * M]
    vh, vmaxh = after[8 * M:10 * M], after[10 * M:12 * M]
    assert (vmax > v).any() or (vmaxh > vh).any()
