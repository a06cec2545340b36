"""The bit-metric decoding rate (BMI) of Gray-labelled bits without a GPU: the float64 reference's (tests/bmi_ref.py) labels, bit posteriors and BMI (tables, reflection
identity, BMI = GMI at n = 2, BMI <= H(X), BMI < GMI on exact posteriors of a Gaussian PAM channel, invariance under the symmetries the SER
forgives), and the host logic of bmi=True in run_dp_sweep / run_awgn_sweep through stub runners: result layout alone and next to GMI,
runner keywords, checkpoint files never mixed up, the .mat key and the inputs the engines reject."""
import os

import numpy as np
import pytest
import torch

import bmi_ref as B

DP = dict(SNR_vec=[20, 23], nu_vec=[0.0], theta_diff_vec=[0.06 * np.pi], theta_vec=[np.pi / 10], M_vec=[9, 25], lr_optim_vec=[2.5e-3],
          batch_len_vec=[100], flex_step_vec=[10], symb_rate_vec=[90e9])
AW = dict(N_train_vec=[200], lr_optim_vec=[2e-3], M_vec=[9, 25], SNR_vec=[12], nu_vec=[0.0, 0.05], iter=1, num_epochs=4, epe=2)


# ---- float64 reference-------------------------------------------------------------------------------------------------------------------
def test_gray_labels_and_reflection_identity():
    assert B.gray_labels(2).tolist() == [0, 1]
    assert B.gray_labels(4).tolist() == [0, 1, 3, 2]
    assert B.gray_labels(8).tolist() == [0, 1, 3, 2, 6, 7, 5, 4]
    for n in (2, 4, 8):
        g, m = B.gray_labels(n), n.bit_length() - 1
        assert all(int(g[n - 1 - l]) == int(g[l]) ^ (1 << (m - 1)) for l in range(n)), n
        assert all(bin(int(g[l]) ^ int(g[l + 1])).count("1") == 1 for l in range(n - 1)), n      # neighbours differ in one bit


def _levels_tx(shape, n, gen):
    S = n - 1
    lev = torch.randint(0, n, shape, generator=gen)
    return ((2 * lev - S).float() / S).to(torch.float16), lev


def _gmi64(q, tx, P):
    """GMI of oracle.gmi_from_posteriors kept in float64 (that function ends in float32)."""
    n = q.shape[1] // 2
    idx = B._tx_levels(tx, n)
    P = torch.as_tensor(P, dtype=torch.float64)
    qi = torch.gather(q[:, :n].double(), 1, idx[:, 0:1]).squeeze(1)
    qq = torch.gather(q[:, n:].double(), 1, idx[:, 1:2]).squeeze(1)
    return -2 * (P * torch.log2(P)).sum() + (torch.log2(qi.clamp(min=1e-30)) + torch.log2(qq.clamp(min=1e-30))).mean(-1)


def test_bit_posteriors_sum_the_labelled_levels():
    gen = torch.Generator().manual_seed(1)
    for n in (2, 4, 8):
        m = n.bit_length() - 1
        q = torch.softmax(torch.randn(2, 2, n, 50, generator=gen, dtype=torch.float64), dim=2).reshape(2, 2 * n, 50)
        pb = B.bit_posteriors(q)
        assert pb.shape == (2, 2 * m, 2, 50)
        g = B.gray_labels(n)
        for c in range(2):
            for i in range(m):
                for v in range(2):
                    levels = [l for l in range(n) if (int(g[l]) >> (m - 1 - i)) & 1 == v]
                    assert torch.allclose(pb[:, c * m + i, v], q[:, c * n + torch.tensor(levels)].sum(1), rtol=0, atol=1e-15)
        L = B.bit_llr_from_posteriors(q)
        assert torch.allclose(L, torch.log(pb[:, :, 0]) - torch.log(pb[:, :, 1]), rtol=0, atol=1e-12)


def test_bmi_equals_gmi_at_two_levels_and_stays_below_entropy():
    gen = torch.Generator().manual_seed(2)
    for n in (2, 4, 8):
        N = 4000
        tx, _ = _levels_tx((2, 2, N), n, gen)
        q = torch.softmax(torch.randn(2, 2, n, N, generator=gen), dim=2).reshape(2, 2 * n, N)      # fp32 posteriors
        P = torch.rand(n, generator=gen) + 0.1
        P = P / P.sum()
        bmi = B.bmi_from_posteriors(q, tx, P)
        H = float(-2 * (P.double() * torch.log2(P.double())).sum())
        assert bmi.dtype == torch.float64 and bool((bmi <= H + 1e-5).all()), (n, bmi.tolist(), H)
        if n == 2:
            assert float((bmi - _gmi64(q, tx, P)).abs().max()) < 1e-12


def test_bmi_below_gmi_on_exact_gaussian_pam_posteriors():
    """Matched posteriors of 64-QAM (8-PAM per component) with Maxwell-Boltzmann shaping nu = 0.03 over AWGN at 8 dB: bit-wise decoding
    loses about 0.1 bit per 2-D symbol against symbol-wise decoding.  Holds for exact posteriors only, not for trained ones."""
    rng = np.random.default_rng(0)
    n, N, nu, snr_db = 8, 200_000, 0.03, 8.0
    a = np.arange(-7, 8, 2.0)
    P = np.exp(-nu * a ** 2)
    P /= P.sum()
    a = a / np.sqrt(2 * np.sum(P * a ** 2))                                        # unit 2-D power
    var = 1 / 10 ** (snr_db / 10) / 2
    idx = rng.choice(n, size=(2, 2, N), p=P)
    y = a[idx] + rng.normal(scale=np.sqrt(var), size=(2, 2, N))
    logit = -(y[..., None] - a) ** 2 / (2 * var) + np.log(P)
    q = np.exp(logit - logit.max(-1, keepdims=True))
    q /= q.sum(-1, keepdims=True)
    q = torch.from_numpy(np.moveaxis(q, -1, 2).reshape(2, 2 * n, N))
    tx = torch.from_numpy((2 * idx - (n - 1)) / (n - 1)).to(torch.float16)
    gmi, bmi = _gmi64(q, tx, torch.from_numpy(P)), B.bmi_from_posteriors(q, tx, torch.from_numpy(P))
    gap = gmi - bmi
    assert bool((gap > 0.06).all()) and bool((gap < 0.14).all()), (gmi.tolist(), bmi.tolist())


def _mirror_q(q, n, flip, k):
    """q of a receiver whose hypothesis (flip, k) is the one that scores the q levels (iI, iQ) below where q scores the tx levels
    (lI, lQ): its I and Q rows are q's, swapped and mirrored (level l -> S - l) as the rotation by k pi/2 and the IQ flip do."""
    rev = lambda t: t.flip(1)
    A, Bp = q[:, :n], (rev(q[:, n:]) if flip else q[:, n:])                       # indexed by lI and by lQp = (S - lQ if flip else lQ)
    return torch.cat([(A, Bp), (rev(A), rev(Bp)), (Bp, rev(A)), (rev(Bp), A)][k], 1)


def test_bmi_invariant_under_rotations_and_iq_flip():
    """q of a receiver rotated by k pi/2 and IQ-flipped, scored at the q levels that hypothesis maps the tx levels onto: the same BMI
    (the Gray labels' reflection identity), for every one of the 8 hypotheses."""
    gen = torch.Generator().manual_seed(4)
    for n in (2, 4, 8):
        N, S = 3000, n - 1
        tx, lev = _levels_tx((2, 2, N), n, gen)
        q = torch.softmax(torch.randn(2, 2, n, N, generator=gen, dtype=torch.float64), dim=2).reshape(2, 2 * n, N)
        P = torch.full((n,), 1.0 / n)
        ref = B.bmi_from_posteriors(q, tx, P)
        for flip in (0, 1):
            for k in range(4):
                q2 = _mirror_q(q, n, flip, k)
                lI, lQ = lev[:, 0], lev[:, 1]
                # the q levels hypothesis (flip, k) scores for tx (lI, lQ): inverse of er_count_q's hI / hQ with DQ flipped
                lQp = S - lQ if flip else lQ
                iI, iQ = [(lI, lQp), (S - lI, S - lQp), (lQp, S - lI), (S - lQp, lI)][k]
                tx2 = torch.stack(((2 * iI - S).float() / S, (2 * iQ - S).float() / S), 1).to(torch.float16)
                got = B.bmi_from_posteriors(q2, tx2, P)
                assert float((got - ref).abs().max()) < 1e-12, (n, flip, k, got.tolist(), ref.tolist())


# ---- engine plumbing through stub runners --------------------------------------------------------------------------------------------
def _dp_runner(calls, offset=0.0):
    """Stands for sweep_vae_dp_sharded: SER / Var_est / var / GMI / BMI encode the cell's seed, BMI = -(GMI + 0.125), NaN on frame 1."""
    def runner(cells, mod, sps, M, batch_len, N_frame_max, num_frames, gmi=False, bmi=False, **kw):
        calls.append((M, len(cells), gmi, bmi))
        n = len(cells)
        seed = torch.tensor([float(c["seed"]) for c in cells])
        ser = seed.view(n, 1, 1).expand(n, 4, num_frames) + offset
        ve, var = 2 * seed.view(n, 1, 1).expand(n, 2, num_frames).clone(), 3 * seed.view(n, 1).expand(n, 2).clone()
        g = (seed.view(n, 1, 1) + torch.arange(2.0).view(1, 2, 1) * 0.5 + offset).expand(n, 2, num_frames).clone()
        g[:, :, 1] = float("nan")
        return (ser, ve, var) + ((g,) if gmi else ()) + ((-(g + 0.125),) if bmi else ())
    return runner


def _aw_runner(calls, offset=0.0):
    def runner(cells, mod, sps, M, batch_len, N_valid, N_train, num_epochs, epe, channel, gmi=False, bmi=False):
        calls.append((M, len(cells), gmi, bmi))
        ser = torch.stack([torch.full((num_epochs // epe,), float(c["seed"]) + offset) for c in cells])
        extra = ((-ser - 0.25,) if gmi else ()) + ((-ser - 0.5,) if bmi else ())
        return (ser,) + extra if extra else ser
    return runner


def test_run_dp_sweep_bmi_layout():
    from vae_equalizer_b200 import sweep
    calls = []
    SER, Var_est, var_real, BMI = sweep.run_dp_sweep(iter=2, num_frames=3, runner=_dp_runner(calls), bmi=True, **DP)
    assert calls and all(c[2:] == (False, True) for c in calls)
    assert BMI.shape == Var_est.shape == (2, 2, 1, 1, 1, 2, 1, 1, 1, 1, 2, 3)
    for idx in np.ndindex(*BMI.shape[1:-1]):
        seed = float(SER[(0,) + idx + (0,)])
        for p in range(2):
            b = BMI[(p,) + idx]
            assert float(b[0]) == -(seed + 0.5 * p + 0.125) and float(b[2]) == float(b[0]) and torch.isnan(b[1]), (idx, p)
    calls2 = []
    res = sweep.run_dp_sweep(iter=2, num_frames=3, runner=_dp_runner(calls2), gmi=True, bmi=True, **DP)
    assert len(res) == 5 and all(c[2:] == (True, True) for c in calls2)
    assert torch.equal(res[0], SER) and torch.equal(res[1], Var_est) and torch.equal(res[2], var_real)
    assert torch.equal(res[4].nan_to_num(7), BMI.nan_to_num(7)) and torch.equal(res[4].nan_to_num(7), (-(res[3] + 0.125)).nan_to_num(7))
    calls3 = []
    res = sweep.run_dp_sweep(iter=2, num_frames=3, runner=_dp_runner(calls3), **DP)
    assert len(res) == 3 and all(c[2:] == (False, False) for c in calls3)


def test_run_awgn_sweep_bmi_layout():
    from vae_equalizer_b200 import sweep
    calls = []
    SER, epochs, BMI = sweep.run_awgn_sweep(mod="16-QAM", runner=_aw_runner(calls), bmi=True, **AW)
    assert all(c[2:] == (False, True) for c in calls) and list(epochs) == [0, 2]
    assert BMI.shape == SER.shape == (1, 1, 2, 1, 2, 1, 2) and torch.equal(BMI, -SER - 0.5)
    calls2 = []
    SER2, _, GMI2, BMI2 = sweep.run_awgn_sweep(mod="16-QAM", runner=_aw_runner(calls2), gmi=True, bmi=True, **AW)
    assert all(c[2:] == (True, True) for c in calls2)
    assert torch.equal(SER2, SER) and torch.equal(GMI2, -SER - 0.25) and torch.equal(BMI2, BMI)


def _files(ck):
    return {f: np.load(os.path.join(ck, f)) for f in sorted(os.listdir(ck))}


def test_dp_bmi_checkpoints_never_mixed_up(tmp_path):
    """Files of gmi / bmi / both / neither are four different sets of files; each kind reloads only its own."""
    from vae_equalizer_b200 import sweep
    ck = str(tmp_path / "ck")
    calls = []
    kinds = [dict(), dict(gmi=True), dict(bmi=True), dict(gmi=True, bmi=True)]
    first = []
    for j, kw in enumerate(kinds):
        n0 = len(calls)
        first.append(sweep.run_dp_sweep(iter=1, num_frames=2, runner=_dp_runner(calls, offset=0.25 * j), checkpoint_dir=ck, **kw, **DP))
        assert len(calls) > n0 and len(os.listdir(ck)) == 2 * (j + 1), kw     # nothing of another kind was loaded
    files = _files(ck)
    assert sum("bmi" in z.files for z in files.values()) == 4 and sum("gmi" in z.files for z in files.values()) == 4
    n0 = len(calls)
    for j, kw in enumerate(kinds):
        again = sweep.run_dp_sweep(iter=1, num_frames=2, runner=_dp_runner(calls, offset=9.0), checkpoint_dir=ck, **kw, **DP)
        assert len(again) == 3 + len(kw)
        assert all(torch.equal(a.nan_to_num(-3), b.nan_to_num(-3)) for a, b in zip(again, first[j])), kw
    assert len(calls) == n0                                                     # every kind reloaded its own files


def test_awgn_bmi_checkpoints_never_mixed_up(tmp_path):
    from vae_equalizer_b200 import sweep
    ck = str(tmp_path / "ck")
    calls = []
    kinds = [dict(gmi=True), dict(bmi=True), dict(gmi=True, bmi=True)]
    first = []
    for j, kw in enumerate(kinds):
        n0 = len(calls)
        first.append(sweep.run_awgn_sweep(mod="16-QAM", runner=_aw_runner(calls, offset=0.25 * j), checkpoint_dir=ck, **kw, **AW))
        assert len(calls) > n0 and len(os.listdir(ck)) == 2 * (j + 1), kw
    n0 = len(calls)
    for j, kw in enumerate(kinds):
        again = sweep.run_awgn_sweep(mod="16-QAM", runner=_aw_runner(calls, offset=9.0), checkpoint_dir=ck, **kw, **AW)
        assert len(again) == 2 + len(kw) and torch.equal(again[0], first[j][0]) and all(torch.equal(a, b) for a, b in zip(again[2:], first[j][2:]))
    assert len(calls) == n0


def test_bmi_checkpoint_without_the_array_is_not_loaded(tmp_path):
    """A file whose signature matches a bmi=True set but that lacks the 'bmi' array is recomputed, not loaded."""
    from vae_equalizer_b200 import sweep
    ck = str(tmp_path / "ck")
    calls = []
    sweep.run_dp_sweep(iter=1, num_frames=2, runner=_dp_runner(calls), checkpoint_dir=ck, bmi=True, **DP)
    for f in os.listdir(ck):
        z = dict(np.load(os.path.join(ck, f)))
        del z["bmi"]
        np.savez(os.path.join(ck, f), **z)
    n0 = len(calls)
    sweep.run_dp_sweep(iter=1, num_frames=2, runner=_dp_runner(calls), checkpoint_dir=ck, bmi=True, **DP)
    assert len(calls) == 2 * n0


def test_save_mat_bmi_key(tmp_path):
    from scipy import io
    from vae_equalizer_b200 import sweep
    SER, Var_est, var_real, GMI, BMI = sweep.run_dp_sweep(iter=1, num_frames=3, runner=_dp_runner([]), gmi=True, bmi=True, **DP)
    lists = dict(SNR_vec=DP["SNR_vec"], nu_vec=DP["nu_vec"], theta_diff_vec=DP["theta_diff_vec"], theta_vec=DP["theta_vec"], M_vec=DP["M_vec"],
                 lr_optim_vec=DP["lr_optim_vec"], batch_len_vec=DP["batch_len_vec"], symb_rate_vec=DP["symb_rate_vec"],
                 flex_step_vec=DP["flex_step_vec"])
    p0, p1, p2 = str(tmp_path / "a.mat"), str(tmp_path / "b.mat"), str(tmp_path / "c.mat")
    sweep.save_mat(p0, SER, Var_est, var_real, **lists)
    sweep.save_mat(p1, SER, Var_est, var_real, BMI=BMI, **lists)
    sweep.save_mat(p2, SER, Var_est, var_real, GMI=GMI, BMI=BMI, **lists)
    d0, d1, d2 = (io.loadmat(p)["dict"] for p in (p0, p1, p2))
    assert set(d1.dtype.names) == set(d0.dtype.names) | {"BMI"} and set(d2.dtype.names) == set(d0.dtype.names) | {"GMI", "BMI"}
    for d in (d1, d2):
        b = d["BMI"][0, 0]
        assert b.shape == tuple(BMI.shape) and np.array_equal(np.isnan(b), torch.isnan(BMI).numpy())
        assert np.array_equal(np.nan_to_num(b), torch.nan_to_num(BMI).numpy())


def test_engines_reject_per_cell_bmi_and_cpu_tensors():
    from vae_equalizer_b200 import sweep
    from vae_equalizer_b200._lib import VaeqError
    from vae_equalizer_b200.awgn import awgn_bmi_runs
    from vae_equalizer_b200.shared_funcs import BMI, bit_llr, bmi_runs
    cells = [dict(SNR=23, nu=0.0, lr_optim=2.5e-3)]
    for kind in ("VAE", "VAEflex"):
        with pytest.raises(ValueError, match="bmi"):
            sweep.sweep_vae_dp(cells, "64-QAM", 2, 25, 100, 1000, 1, 10, kind=kind, eval_mode="per_cell", bmi=True)
    with pytest.raises(ValueError, match="bmi"):
        sweep.sweep_cma_dp(cells, "64-QAM", 2, 25, 100, 1000, 1, eval_mode="per_cell", bmi=True)
    with pytest.raises(VaeqError):
        sweep.sweep_vae_awgn(cells, "16-QAM", 2, 25, 350, 15000, 1200, 20, 10, "h1", device="cpu", bmi=True)
    R, n, N = 2, 4, 300
    q = torch.full((R, 2, 2 * n, N), 1.0 / n)
    tx = torch.zeros(R, 2, 2, N, dtype=torch.float16)
    with pytest.raises(VaeqError):
        bmi_runs(q, tx, torch.full((n,), 1.0 / n), torch.zeros(R, 2, 4, dtype=torch.int32), torch.zeros(R, 2, 2, 2, 4, dtype=torch.int32), 100)
    with pytest.raises(VaeqError):
        awgn_bmi_runs(q[:, 0], tx[:, 0], torch.full((n,), 1.0 / n), torch.zeros(R, dtype=torch.int32), torch.zeros(R, 4, dtype=torch.int32))
    with pytest.raises(VaeqError):
        BMI(q[0], tx[0], torch.full((n,), 1.0 / n))
    for bad in (q, q[0]):
        with pytest.raises(VaeqError):
            bit_llr(bad)


def test_dropin_exports_bmi_and_bit_llr():
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "vae_equalizer_b200", "dropin"))
    try:
        import shared_funcs as drop
    finally:
        sys.path.pop(0)
    from vae_equalizer_b200 import shared_funcs as sfun
    assert drop.BMI is sfun.BMI and drop.bit_llr is sfun.bit_llr and drop.GMI is sfun.GMI


# ---- sharded engines with both metrics: the gathers keep the order GMI, BMI (one rank; the two-rank gathers are those of GMI) ----------
def _stub_dp(cells, *args, gmi=False, bmi=False, **kw):
    n, nf = len(cells), 3
    seed = torch.tensor([float(c["seed"]) for c in cells]).view(n, 1, 1)
    base = (seed.expand(n, 4, nf) * 0.01, torch.zeros(n, 2, nf), torch.ones(n, 2))
    return base + ((seed.expand(n, 2, nf) - 10.0,) if gmi else ()) + ((-seed.expand(n, 2, nf) - 20.0,) if bmi else ())


def _stub_aw(cells, *args, gmi=False, bmi=False, **kw):
    seed = torch.tensor([float(c["seed"]) for c in cells]).view(-1, 1).expand(len(cells), 2)
    extra = ((seed - 10.0,) if gmi else ()) + ((-seed - 20.0,) if bmi else ())
    return (seed * 0.01,) + extra if extra else seed * 0.01


def test_sharded_order_gmi_then_bmi(monkeypatch):
    from vae_equalizer_b200 import sweep
    monkeypatch.setattr(sweep, "sweep_vae_dp", _stub_dp)
    monkeypatch.setattr(sweep, "sweep_cma_dp", _stub_dp)
    monkeypatch.setattr(sweep, "sweep_vae_awgn", _stub_aw)
    cells = [dict(SNR=20, nu=0.0, lr_optim=1e-3, seed=s) for s in range(3)]
    dev = torch.device("cpu")
    kw = dict(flex_step=10, channel="h0", symb_rate=90e9, tau_cd=0.0, tau_pmd=0.0, phiIQ=(0.0, 0.0), N_lrhalf=3)
    for mk in (dict(bmi=True), dict(gmi=True, bmi=True)):
        outs = [sweep.sweep_vae_dp_sharded(cells, "64-QAM", 2, 25, 100, 1000, 3, device=dev, **mk),
                sweep.sweep_cma_dp_sharded(cells, "64-QAM", 2, 25, 100, 1000, 3, kind="CMA", device=dev, **kw, **mk)]
        for out in outs:
            assert len(out) == 3 + len(mk)
            assert float(out[-1][2, 0, 0]) == -22.0 and (len(mk) == 1 or float(out[3][2, 0, 0]) == -8.0)
        aw = sweep.sweep_vae_awgn_sharded(cells, "16-QAM", 2, 25, 200, 3000, 1200, 4, 2, "h1", device=dev, **mk)
        assert len(aw) == 1 + len(mk) and float(aw[-1][1, 0]) == -21.0 and (len(mk) == 1 or float(aw[1][1, 0]) == -9.0)
