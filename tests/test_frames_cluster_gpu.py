"""Batched DP runs above dp_small.cu's range: one thread-block cluster per run (csrc/dp_cluster.cu, DESIGN.md §4c).

Minibatches of more than 1000 symbols (or a shared-memory plan over 220 KB at large M_est) train on K = 2, 4 or 8 CTAs per run.
The cluster kernel is compared with the single-run driver (which steps such a minibatch launch by launch) within the step
tolerances, with the CPU oracle on the first steps, and with itself for batch independence (bitwise)."""
import numpy as np
import pytest
import torch

from oracle import vaeq_oracle as O

pytestmark = pytest.mark.gpu


def synth_frame(mod, M, N, nu, seed, snr=20):
    h_est, h_ch, P, amp, amps, pol, nu_sc, var, pow_mean = O.init("h0", mod, "cpu", nu, 2, M, snr)
    rx, tx, _ = O.generate_data_shaping(N, amps, snr, h_ch, P, 2, 90e9, 2, -26e-24, 0.1e-12 * np.sqrt(1000),
                                        np.array([0.0314, 0.0314], dtype=np.complex64), np.pi / 10, "cpu", rng=np.random.default_rng(seed))
    return dict(P=P, amp=amp, nu_sc=nu_sc, var=var), rx, tx


def run_frame(c, rx, M, B, stride, n_steps, keep_lo, keep_n, keep_lo_in_dst, lr_w, lr_h):
    """One run through DPEqualizer.train_frame: above 1000 symbols that is one set of launches per step."""
    from vae_equalizer_b200 import _lib
    from vae_equalizer_b200.dp import DPEqualizer
    lib = _lib.load()
    n = c["amp"].numel()
    eq = DPEqualizer(M, 2, c["amp"], c["P"], c["var"], c["nu_sc"])
    N_keep = (n_steps - 1) * stride + keep_n + keep_lo
    ot = torch.zeros(2, 2 * n, N_keep, device="cuda")
    oc = torch.zeros(2, 2, N_keep, device="cuda")
    n0 = int(lib.vaeq_launch_count(-1))
    loss, ve = eq.train_frame(rx.cuda(), B, stride, n_steps, lr_w, lr_h, ot, oc, keep_lo, keep_n, keep_lo_in_dst=keep_lo_in_dst)
    torch.cuda.synchronize()
    launches = int(lib.vaeq_launch_count(-1)) - n0
    return dict(loss=loss.cpu(), ve=ve.cpu(), ot=ot.cpu(), oc=oc.cpu(), W=eq.W.cpu(), h=eq.h.cpu(), gW=eq.gW.cpu(), gh=eq.gh.cpu(),
                last_loss=eq.loss.cpu(), last_ve=eq.var_est.cpu(), steps=eq.step_count(), launches=launches)


def make_runs(cs, M):
    from vae_equalizer_b200.dp import DPEqualizerRuns
    return DPEqualizerRuns(len(cs), M, 2, cs[0]["amp"], torch.stack([torch.as_tensor(c["P"], dtype=torch.float32) for c in cs]),
                           torch.stack([torch.as_tensor(c["var"], dtype=torch.float32) for c in cs]),
                           torch.tensor([float(c["nu_sc"]) for c in cs], dtype=torch.float32))


def run_runs(eqr, rx_all, B, stride, n_steps, keep_lo, keep_n, kd, lr_w, lr_h, ot=None, oc=None):
    """All runs of eqr in one vaeq_dp_train_frame_runs call; returns the per-run results on the host and the launch count."""
    from vae_equalizer_b200 import _lib
    lib = _lib.load()
    R, n = eqr.R, eqr.n_lev
    N_keep = (n_steps - 1) * stride + keep_n + keep_lo
    ot = torch.zeros(R, 2, 2 * n, N_keep, device="cuda") if ot is None else ot
    oc = torch.zeros(R, 2, 2, N_keep, device="cuda") if oc is None else oc
    n0 = int(lib.vaeq_launch_count(-1))
    loss, ve = eqr.train_frame(rx_all, B, stride, n_steps, lr_w, lr_h, ot, oc, keep_lo, keep_n, keep_lo_in_dst=kd)
    torch.cuda.synchronize()
    launches = int(lib.vaeq_launch_count(-1)) - n0
    steps = eqr.adam[:, 48 * eqr.M].contiguous().view(torch.int32).cpu()
    return dict(loss=loss.cpu(), ve=ve.cpu(), ot=ot.cpu(), oc=oc.cpu(), W=eqr.W.cpu(), h=eqr.h.cpu(), gW=eqr.gW.cpu(), gh=eqr.gh.cpu(),
                last_loss=eqr.loss.cpu(), last_ve=eqr.var_est.cpu(), steps=steps, launches=launches)


def rel(x, y):
    return float((x.double() - y.double()).abs().max() / y.double().abs().max())


def max_b(M, n_lev=8):
    from vae_equalizer_b200 import _lib
    return int(_lib.load().vaeq_dp_runs_max_batch_len(M, n_lev))


# mod, M, B (None: the largest supported), stride, n_steps, keep_lo, keep_n, keep_lo_in_dst, nu; K in the comment is the cluster size
# the plan takes (the smallest of 2, 4, 8 whose 220 KB per-CTA plan fits)
CLUSTER_CASES = [
    ("64-QAM", 25, 1004, 1004, 3, 0, 1004, True, 0.0270955),    # K = 2, just above dp_small.cu's range
    ("64-QAM", 25, 2000, 2000, 3, 0, 2000, True, 0.0270955),    # K = 2
    ("64-QAM", 25, 4096, 4096, 2, 0, 4096, True, 0.0),          # K = 4
    ("64-QAM", 25, 2000, 100, 5, 950, 100, False, 0.0270955),   # VAE-flex, window 2000 / flex_step 100: kept columns on both sides of a slice edge
    ("16-QAM", 9, 1001, 1001, 3, 0, 1001, True, 0.0),           # K = 2, odd: the single-run side takes the generic kernels
    ("4-QAM", 63, 990, 990, 2, 0, 990, True, 0.05),             # K = 2, below 1000 symbols but over dp_small.cu's 220 KB at M_est 63
    ("64-QAM", 5, None, None, 2, 0, None, True, 0.0270955),     # K = 8, largest supported batch_len at M_est 5
    ("64-QAM", 25, None, None, 2, 0, None, True, 0.0270955),    # K = 8, largest supported batch_len at M_est 25
]


@pytest.mark.parametrize("mod,M,B,stride,n_steps,keep_lo,keep_n,kd,nu", CLUSTER_CASES)
def test_cluster_frame_matches_stepped_frame(mod, M, B, stride, n_steps, keep_lo, keep_n, kd, nu):
    """One run (R = 1) on the cluster kernel against the same frame through the single-run driver, launch by launch: every step's
    loss / var_est, the kept q / out columns, the taps after the frame and the last step's gradients (the gates of
    test_frames_gpu.py's dp_small.cu comparison).  One launch for the whole frame; the step counter advances by n_steps."""
    if B is None:
        B = max_b(M)
        stride, keep_n = B, B
    c, rx, _ = synth_frame(mod, M, (n_steps - 1) * stride + B, nu, seed=B + M)
    a = run_runs(make_runs([c], M), rx[None].cuda().contiguous(), B, stride, n_steps, keep_lo, keep_n, kd, 2.5e-3, 1.5e-3)
    b = run_frame(c, rx, M, B, stride, n_steps, keep_lo, keep_n, kd, 2.5e-3, 1.5e-3)
    assert a["launches"] == 1 and int(a["steps"][0]) == n_steps == b["steps"]
    a = {k: (v[0] if k not in ("launches", "steps") else v) for k, v in a.items()}
    n0 = keep_n + (keep_lo if kd else 0)
    assert float((a["oc"][:, :, :n0] - b["oc"][:, :, :n0]).abs().max()) < 5e-6
    assert float((a["ot"][:, :, :n0] - b["ot"][:, :, :n0]).abs().max()) < 5e-5
    assert rel(a["loss"][:1], b["loss"][:1]) < 1e-5 and rel(a["ve"][:, :1], b["ve"][:, :1]) < 1e-5
    assert float((a["oc"] - b["oc"]).abs().max()) < 1e-4
    assert float((a["ot"] - b["ot"]).abs().max()) < 3e-3
    assert rel(a["loss"], b["loss"]) < 1e-4 and rel(a["ve"], b["ve"]) < 1e-4
    assert rel(a["W"], b["W"]) < 1e-4 and rel(a["h"], b["h"]) < 1e-4
    assert rel(a["gW"], b["gW"]) < 1e-3 and rel(a["gh"], b["gh"]) < 1e-3
    assert torch.equal(a["last_loss"].reshape(()), a["loss"][-1]) and torch.equal(a["last_ve"], a["ve"][:, -1])


def test_cluster_frame_against_cpu_oracle():
    """The first 4 steps of a VAE-LE frame at batch_len 2000 against the torch CPU port (autograd + torch Adam)."""
    M, B, n_steps, lr = 25, 2000, 4, 2.5e-3
    c, rx, _ = synth_frame("64-QAM", M, n_steps * B, 0.0270955, seed=5)
    a = run_runs(make_runs([c], M), rx[None].cuda().contiguous(), B, B, n_steps, 0, B, True, lr, lr)
    a = {k: v[0] for k, v in a.items() if k not in ("launches", "steps")}
    tr = O.DPTrainer(M, 2, lr)
    Pt = torch.tensor(c["P"], dtype=torch.float32)
    for m in range(n_steps):
        qo, oo, lo, vo, gWo, gho = tr.step(rx[:, :, 2 * m * B:2 * (m + 1) * B].contiguous(), c["amp"], c["var"], c["nu_sc"], Pt)
        assert float((a["oc"][:, :, m * B:(m + 1) * B] - oo).abs().max()) < 5e-6, m
        assert float((a["ot"][:, :, m * B:(m + 1) * B] - qo).abs().max()) < 5e-5, m
        assert rel(a["loss"][m], lo.reshape(())) < 1e-4 and rel(a["ve"][:, m], vo) < 1e-4, m
    assert rel(a["W"], tr.W.detach()) < 1e-4 and rel(a["h"], tr.h.detach()) < 1e-4
    assert rel(a["gW"], gWo) < 2e-4 and rel(a["gh"], gho) < 2e-4


def _assert_run_equal(a, r, b):
    for k in ("loss", "ve", "ot", "oc", "W", "h", "gW", "gh", "last_loss", "last_ve"):
        assert torch.equal(a[k][r], b[k][0]), (k, r)


def test_cluster_batched_runs_equal_single_runs():
    """R = 5 runs with different SNR (var), PCS (P, nu_sc), learning rates and data in one launch == each run alone (R = 1), bitwise;
    a second frame continues from the first one's Adam state (again bitwise); two identical calls give identical bits."""
    M, B, n_steps, R = 25, 2000, 4, 5
    cs, rxs = [], []
    for r in range(R):
        c, rx, _ = synth_frame("64-QAM", M, n_steps * B, [0.0, 0.0270955, 0.05, 0.0270955, 0.01][r], seed=100 + r, snr=[17, 20, 23, 26, 29][r])
        cs.append(c)
        rxs.append(rx)
    lr_w = torch.tensor([2.5e-3, 1e-3, 2.5e-3, 5e-3, 2e-3])
    lr_h = torch.tensor([2.5e-3, 2.5e-3, 1e-3, 5e-3, 3e-3])
    rx_all = torch.stack(rxs).cuda().contiguous()
    eqr = make_runs(cs, M)
    a1 = run_runs(eqr, rx_all, B, B, n_steps, 0, B, True, lr_w, lr_h)
    a2 = run_runs(eqr, rx_all, B, B, n_steps, 0, B, True, lr_w, lr_h)
    assert a1["launches"] == 1 and a2["launches"] == 1 and (a2["steps"] == 2 * n_steps).all()
    assert (a2["loss"][:, -1] < a1["loss"][:, 0]).all()
    for r in range(R):
        e = make_runs([cs[r]], M)
        b1 = run_runs(e, rx_all[r:r + 1], B, B, n_steps, 0, B, True, float(lr_w[r]), float(lr_h[r]))
        _assert_run_equal(a1, r, b1)
        b2 = run_runs(e, rx_all[r:r + 1], B, B, n_steps, 0, B, True, float(lr_w[r]), float(lr_h[r]))
        _assert_run_equal(a2, r, b2)
    eqr2 = make_runs(cs, M)
    a3 = run_runs(eqr2, rx_all, B, B, n_steps, 0, B, True, lr_w, lr_h)
    for k in ("loss", "ve", "ot", "oc", "W", "h", "gW", "gh"):
        assert torch.equal(a1[k], a3[k]), k


def test_cluster_runs_over_several_waves_equal_single_runs():
    """40 runs at K = 8 (batch_len 6000, M_est 25): 320 CTAs, more than one wave of clusters on 148 SMs; runs from the first and the
    last wave equal the same runs alone, bitwise."""
    from vae_equalizer_b200.datagen import generate_frames_gpu
    M, B, n_steps, R = 25, 6000, 2, 40
    h_est, h_ch, P, amp, amps, pol, nu_sc, var, pow_mean = O.init("h0", "64-QAM", "cpu", 0.0270955, 2, M, 23)
    snr = [17.0 + 0.3 * r for r in range(R)]
    rx_all, _, _ = generate_frames_gpu(B * n_steps, amps, snr, np.tile(np.asarray(P, dtype=np.float32)[None], (R, 1)), 2,
                                       [0.1 * r for r in range(R)], "cuda", 21)
    rx_all = rx_all.contiguous()
    c = dict(P=P, amp=amp, nu_sc=nu_sc, var=var)
    lr = torch.tensor([1e-3 + 1e-4 * r for r in range(R)])
    a = run_runs(make_runs([c] * R, M), rx_all, B, B, n_steps, 0, B, True, lr, lr)
    assert a["launches"] == 1 and torch.isfinite(a["loss"]).all()
    for r in (0, 17, 39):
        b = run_runs(make_runs([c], M), rx_all[r:r + 1].contiguous(), B, B, n_steps, 0, B, True, float(lr[r]), float(lr[r]))
        _assert_run_equal(a, r, b)


def test_cluster_rejects_batch_len_above_the_limit():
    """One symbol above the largest supported batch_len: VaeqError naming the limit, and nothing is launched (the engine call and the
    sweeps check before any data is generated)."""
    from vae_equalizer_b200 import _lib, sweep
    lib = _lib.load()
    M = 25
    lim = max_b(M)
    assert 4096 < lim < 65536 and max_b(63, 2) < lim < max_b(5)
    c, _, _ = synth_frame("64-QAM", M, 100, 0.0, seed=1)
    eqr = make_runs([c], M)
    rx = torch.zeros(1, 2, 2, 2 * (lim + 1), device="cuda")
    n0 = int(lib.vaeq_launch_count(-1))
    with pytest.raises(_lib.VaeqError, match=str(lim)):
        run_runs(eqr, rx, lim + 1, lim + 1, 1, 0, lim + 1, True, 1e-3, 1e-3)
    assert int(eqr.adam[0, 48 * M:48 * M + 1].view(torch.int32).item()) == 0
    cell = dict(SNR=20, nu=0.0, lr_optim=2.5e-3, theta=0.0, theta_diff=0.0, seed=1)
    with pytest.raises(_lib.VaeqError, match=str(lim)):
        sweep.sweep_vae_dp([cell], "64-QAM", 2, M, lim + 1, 2 * (lim + 1), 1, kind="VAE", datagen="gpu")
    with pytest.raises(_lib.VaeqError, match=str(lim)):
        sweep.run_dp_sweep(batch_len_vec=[100, lim + 1], M_vec=[M], lr_optim_vec=[2.5e-3], iter=1, num_frames=1, N_frame_max=2 * (lim + 1))
    torch.cuda.synchronize()
    assert int(lib.vaeq_launch_count(-1)) == n0


SWEEP_CELLS = [dict(SNR=24, nu=0.0270955, lr_optim=2.5e-3, theta=np.pi / 10, theta_diff=0.06 * np.pi, seed=3),
               dict(SNR=22, nu=0.0, lr_optim=5e-3, theta=0.2, theta_diff=0.0, seed=4),
               dict(SNR=26, nu=0.0270955, lr_optim=1e-3, theta=0.0, theta_diff=0.01, seed=5),
               dict(SNR=20, nu=0.05, lr_optim=2e-3, theta=0.4, theta_diff=0.02, seed=6),
               dict(SNR=28, nu=0.0270955, lr_optim=3e-3, theta=-0.3, theta_diff=0.0, seed=7)]
SWEEP_COMMON = dict(symb_rate=90e9, tau_cd=-26e-24, tau_pmd=0.1e-12 * np.sqrt(1000), phiIQ=np.array([0.0314, 0.0314], dtype=np.complex64))


@pytest.mark.parametrize("kind", ["VAE", "VAEflex"])
@pytest.mark.parametrize("gmi", [False, True])
def test_cluster_sweep_cell_alone_equals_cell_in_batch(kind, gmi):
    """sweep_vae_dp at batch_len 2000 (datagen='gpu': a cell's data depends on its own seed): a cell alone and the same cell inside a
    batch of 5 give identical SER_valid and Var_est (and GMI)."""
    from vae_equalizer_b200.sweep import sweep_vae_dp
    args = ("64-QAM", 2, 25, 2000, 8000, 2)
    kw = dict(flex_step=100, channel="h0", N_lrhalf=1, kind=kind, datagen="gpu", **SWEEP_COMMON, **(dict(gmi=True) if gmi else {}))
    full = sweep_vae_dp(SWEEP_CELLS, *args, **kw)
    one = sweep_vae_dp(SWEEP_CELLS[2:3], *args, **kw)
    torch.cuda.synchronize()
    assert torch.isfinite(full[0]).all() and float(full[0].max()) <= 1.0
    for a, b in zip(full, one):
        assert torch.equal(a[2:3], b)


@pytest.mark.parametrize("kind", ["VAE", "VAEflex"])
def test_cluster_sweep_against_single_run_drivers(kind):
    """sweep_vae_dp at batch_len 2000 against processing_vaele_dp / processing_vaeflex_dp on the same frames (datagen='gpu', same seeds).
    The single-run driver steps these minibatches launch by launch, so the two trajectories agree within the step tolerances, not
    bitwise, and the SER estimates may differ by some decisions.  Measured on a B200 (largest over the 3 cells and 2 frames, SER difference
    x scored symbols): VAE-LE 0 decisions per frame (4 steps per frame), VAE-flex 13 of 6000 (60 steps per frame), Var_est 1.7e-7 and
    5.3e-3 relative.  Bounds: 40 decisions per frame, Var_est 2e-2."""
    from vae_equalizer_b200.processing import processing_vaele_dp, processing_vaeflex_dp
    from vae_equalizer_b200.sweep import sweep_vae_dp
    fn = processing_vaele_dp if kind == "VAE" else processing_vaeflex_dp
    B, N, F, flex = 2000, 8000, 2, 100
    cells = SWEEP_CELLS[:3]
    ser, ve, var = sweep_vae_dp(cells, "64-QAM", 2, 25, B, N, F, flex_step=flex, channel="h0", N_lrhalf=1, kind=kind, datagen="gpu",
                                **SWEEP_COMMON)
    n_eval = N if kind == "VAE" else N - B
    worst, worst_ve = 0.0, 0.0
    for r, c in enumerate(cells):
        s1, v1, var1 = fn("64-QAM", 2, c["SNR"], c["nu"], 25, c["theta_diff"], c["theta"], c["lr_optim"], B, N, F, flex, "h0",
                          SWEEP_COMMON["symb_rate"], SWEEP_COMMON["tau_cd"], SWEEP_COMMON["tau_pmd"], SWEEP_COMMON["phiIQ"], 1,
                          verbose=False, datagen="gpu", seed=c["seed"])
        assert torch.equal(var1.to(var.device), var[r])
        worst = max(worst, float((s1.to(ser.device) - ser[r]).abs().max()) * n_eval)
        worst_ve = max(worst_ve, rel(ve[r].cpu(), v1.cpu()))
    print(f"{kind}: largest SER difference {worst:.2f} decisions per frame, Var_est {worst_ve:.2e} relative")
    assert worst <= 40.0 and worst_ve < 2e-2, (worst, worst_ve)


def test_cluster_run_dp_sweep_mixed_batch_lens(tmp_path):
    """run_dp_sweep with batch_len_vec=[100, 2000]: both sets run; the batch_len-100 set is bitwise what batch_len_vec=[100] alone gives;
    a second call on the same checkpoint directory loads every set and launches nothing.  A cell's seed is its flat index in the result
    array, so every axis before batch_len has one value here (the cells differ by iteration), which keeps the batch_len-100 seeds the
    same in both sweeps."""
    from vae_equalizer_b200 import _lib, sweep
    lib = _lib.load()
    lists = dict(nu_vec=[0.0270955], symb_rate_vec=[90e9], theta_vec=[np.pi / 10], theta_diff_vec=[0.0], SNR_vec=[23], M_vec=[25],
                 flex_step_vec=[100], lr_optim_vec=[2.5e-3])
    kw = dict(loss_type="VAE", iter=2, num_frames=2, N_frame_max=4000, N_lrhalf=170, datagen="gpu", **lists)
    SER, Var_est, var_real = sweep.run_dp_sweep(batch_len_vec=[100, 2000], checkpoint_dir=str(tmp_path), **kw)
    assert SER.shape == (4, 1, 1, 1, 1, 1, 1, 2, 1, 1, 2, 2)
    assert torch.isfinite(SER).all() and float(SER.max()) <= 1.0 and (Var_est > 0).all()
    S1, V1, r1 = sweep.run_dp_sweep(batch_len_vec=[100], **kw)
    assert torch.equal(SER[:, :, :, :, :, :, :, :1], S1) and torch.equal(Var_est[:, :, :, :, :, :, :, :1], V1)
    n0 = int(lib.vaeq_launch_count(-1))
    S2, V2, r2 = sweep.run_dp_sweep(batch_len_vec=[100, 2000], checkpoint_dir=str(tmp_path), **kw)
    assert int(lib.vaeq_launch_count(-1)) == n0
    assert torch.equal(S2.cpu(), SER.cpu()) and torch.equal(V2.cpu(), Var_est.cpu()) and torch.equal(r2.cpu(), var_real.cpu())
