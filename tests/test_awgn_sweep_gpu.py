"""Batched AWGN single-polarisation VAE-LE sweep engine (csrc/awgn.cu k_awgn_runs, csrc/eval_runs.cu vaeq_awgn_eval_runs,
csrc/datagen.cu vaeq_gen_awgn, sweep.sweep_vae_awgn / run_awgn_sweep) against the single-run kernel, the single-run driver and the
reference goldens."""
import os
import socket

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
T = torch.from_numpy


def rel(a, b):
    a = a.detach().cpu().numpy() if torch.is_tensor(a) else np.asarray(a)
    b = b.detach().cpu().numpy() if torch.is_tensor(b) else np.asarray(b)
    return float(np.abs(a.astype(np.float64) - b.astype(np.float64)).max() / max(np.abs(b).max(), 1e-30))


MODS = {2: "4-QAM", 4: "16-QAM", 8: "64-QAM"}


def _frames(R, F, N, mod, M_est, seed, channel="h1", SNR0=14.0):
    from vae_equalizer_b200.awgn import generate_data
    from vae_equalizer_b200.constants import awgn_constants, upsampled_channel
    h = upsampled_channel(channel, 2)
    M = (len(h) - 1) // 2 + 1
    rng = np.random.default_rng(seed)
    consts, rx, tx = [], torch.empty(R, F, 2, 2 * N, device="cuda"), torch.empty(R, F, 2, N, dtype=torch.float16, device="cuda")
    for r in range(R):
        SNR, nu = SNR0 + 2 * r, 0.02 * r
        consts.append(awgn_constants(mod, nu, SNR))
        for f in range(F):
            rx[r, f], tx[r, f] = generate_data(N, M, consts[-1][0], SNR, h, 2, "cuda", consts[-1][1], rng=rng)
    return consts, rx, tx


@pytest.mark.parametrize("n_lev", [2, 4, 8])
@pytest.mark.parametrize("M_est", [9, 25])
@pytest.mark.parametrize("batch_len", [200, 350])
def test_runs_kernel_bitwise_against_single_run_kernel(n_lev, M_est, batch_len):
    """5 runs with different var, P, amp_mean, lr and data over 2 frames: every step's loss, the final taps and the whole Adam state equal
    a loop of AWGNEqualizer.train_step per run bit for bit; so do q and out of the batched validation forward."""
    from vae_equalizer_b200.awgn import AWGNEqualizer, AWGNEqualizerRuns
    R, F, N_train = 5, 2, 1000
    consts, rx, _ = _frames(R, F, N_train, MODS[n_lev], M_est, 10 * n_lev + M_est)
    amps = consts[0][0]
    lr = [1e-3 * (r + 1) for r in range(R)]
    eqr = AWGNEqualizerRuns(R, M_est, 2, amps, np.stack([c[1] for c in consts]), [c[2] for c in consts], [c[3] for c in consts])
    loss = eqr.train_frames(rx, torch.tensor(lr, device="cuda"), batch_len, N_train)
    n_mb = N_train // batch_len
    assert loss.shape == (R, F * n_mb)
    _, rx_v, _ = _frames(R, 1, 15000, MODS[n_lev], M_est, 99)
    q_r, out_r, _ = eqr.forward(rx_v[:, 0])
    for r in range(R):
        eq = AWGNEqualizer(M_est, 2, amps, consts[r][1], consts[r][2], consts[r][3])
        for f in range(F):
            for m in range(n_mb):
                _, _, l1 = eq.train_step(rx[r, f, :, 2 * m * batch_len:2 * (m + 1) * batch_len].contiguous(), lr[r], lr[r])
                assert torch.equal(l1[0], loss[r, f * n_mb + m]), (r, f, m)
        assert torch.equal(eq.W, eqr.W[r]) and torch.equal(eq.h, eqr.h[r]) and torch.equal(eq.adam, eqr.adam[r]), r
        q, out, _ = eq.forward(rx_v[r, 0].contiguous())
        assert torch.equal(q, q_r[r]) and torch.equal(out, out_r[r]), r


@pytest.mark.parametrize("name", ["awgn_16qam_M25_B350", "awgn_64qam_M9_B200"])
def test_runs_kernel_replays_reference_golden(name):
    """The reference's trajectory as run 0 of a 3-run set (the other runs train on other data), step by step, at the tolerances of
    test_awgn_trajectory_against_reference_golden."""
    from vae_equalizer_b200.awgn import AWGNEqualizerRuns
    g = dict(np.load(os.path.join(GOLDEN, name + ".npz")))
    M, B = g["W0"].shape[-1], g["rx"].shape[-1] // 2
    R = 3
    eqr = AWGNEqualizerRuns(R, M, 2, g["amp"], np.stack([g["P"]] * R), [float(g["amp_mean"])] * R, [float(g["var"]), 0.05, 0.1])
    eqr.W[0], eqr.h[0] = T(g["W0"]).cuda(), T(g["h0"]).cuda()
    lr = torch.tensor([float(g["lr"]), 1e-3, 3e-3], device="cuda")
    gen = torch.Generator().manual_seed(3)
    for s in range(g["rx"].shape[0]):
        rx = torch.randn(R, 1, 2, 2 * B, generator=gen).cuda()
        rx[0, 0] = T(g["rx"][s]).cuda()
        q, out, loss = eqr.forward(rx[:, 0])
        assert np.abs(out[0].cpu().numpy() - g["out"][s]).max() < 5e-6, s
        assert np.abs(q[0].cpu().numpy() - g["q"][s]).max() < 5e-5, s
        assert rel(loss[0], g["loss"][s]) < 1e-4, s
        ls = eqr.train_frames(rx, lr, B)
        assert torch.equal(ls[0, 0], loss[0]), s
        assert rel(eqr.W[0], g["W"][s]) < 1e-4 and rel(eqr.h[0], g["h"][s]) < 1e-4, s


def _score_single(q, tx, amp):
    from vae_equalizer_b200.processing import awgn_find_shift, awgn_ser_q
    shift = awgn_find_shift(q, tx, 21, amp)
    ser, c = awgn_ser_q(q[:, 11 + shift:-11], tx[:, 11:-11 - shift])
    return shift, c, ser


def _check_scoring(q, tx, amp):
    from vae_equalizer_b200.awgn import awgn_eval_runs
    shift, counts, ser = awgn_eval_runs(q, tx, amp)
    for r in range(q.shape[0]):
        s1, c1, ser1 = _score_single(q[r], tx[r], amp)
        assert int(shift[r]) == s1 and torch.equal(counts[r], c1.to(torch.int32)) and torch.equal(ser[r], ser1), r
    return shift


def test_scoring_random_posteriors():
    gen = torch.Generator().manual_seed(5)
    amp = torch.tensor([-3.0, -1.0, 1.0, 3.0], device="cuda")
    R, N = 7, 3000
    q = torch.softmax(torch.randn(R, 8, N, generator=gen).view(R, 2, 4, N), dim=2).view(R, 8, N).cuda()
    tx = amp.cpu()[torch.randint(0, 4, (R, 2, N), generator=gen)].to(torch.float16).cuda()
    _check_scoring(q, tx, amp)


def test_scoring_every_shift_on_trained_output():
    """Real validation output of a trained equalizer with tx rolled by every shift in -10..10."""
    from vae_equalizer_b200.awgn import AWGNEqualizerRuns
    consts, rx, _ = _frames(1, 20, 1200, "16-QAM", 25, 1, SNR0=18.0)
    eqr = AWGNEqualizerRuns(1, 25, 2, consts[0][0], consts[0][1][None], [consts[0][2]], [consts[0][3]])
    eqr.train_frames(rx, torch.tensor([5e-3], device="cuda"), 350, 1200)
    _, rx_v, tx_v = _frames(1, 1, 5000, "16-QAM", 25, 2, SNR0=18.0)
    q, _, _ = eqr.forward(rx_v[:, 0])
    amp = torch.tensor(consts[0][0], dtype=torch.float32, device="cuda")
    R = 21
    qR = q.expand(R, -1, -1).contiguous()
    txR = torch.stack([tx_v[0, 0].roll(s, -1) for s in range(-10, 11)])
    shift = _check_scoring(qR, txR, amp)
    assert len(set(shift.tolist())) > 10                             # the rolls move the detected shift


def test_scoring_threshold_branches():
    """I correlation below 0.02 N: Q wins when its maximum is at least I's, else I is kept."""
    amp = torch.tensor([-1.0, 1.0], device="cuda")
    gen = torch.Generator().manual_seed(8)
    N = 4000
    tx = amp.cpu()[torch.randint(0, 2, (2, 2, N), generator=gen)].to(torch.float16).cuda()
    # q: posteriors whose I decision follows tx Q (shifted by 3) weakly, nearly flat otherwise
    p_q = 0.5 + 0.004 * tx[0, 1].float().roll(3)
    q_a = torch.stack((1 - p_q, p_q, torch.full_like(p_q, 0.5), torch.full_like(p_q, 0.5)))
    p_i = 0.5 + 0.004 * tx[1, 0].float().roll(2)                     # ... or follows tx I weakly
    q_b = torch.stack((1 - p_i, p_i, torch.full_like(p_i, 0.5), torch.full_like(p_i, 0.5)))
    q = torch.stack((q_a, q_b)).contiguous()
    txs = torch.stack((tx[0], tx[1])).contiguous()
    import vae_equalizer_b200.shared_funcs as sfun
    from vae_equalizer_b200.processing import awgn_find_shift
    for r in range(2):
        q2 = torch.stack((q[r][:, :1000], q[r][:, :1000])).contiguous()
        _, _, corr = sfun.find_shift(q2, torch.stack((txs[r][:, :1000],) * 2).contiguous(), 21, amp, 2, return_corr=True)
        cI, cQ = corr[0, 0, 0], corr[1, 0, 0]
        assert float(cI.max()) < 0.02 * N
        assert (float(cQ.max()) >= float(cI.max())) == (r == 0), r
        assert isinstance(awgn_find_shift(q[r], txs[r], 21, amp), int)
    _check_scoring(q, txs, amp)


def test_generator_statistics_and_structure():
    from vae_equalizer_b200.awgn import generate_frames_awgn_gpu
    from vae_equalizer_b200.constants import awgn_constants, upsampled_channel
    from vae_equalizer_b200.datagen import PULSE_SPAN, ROLLOFF, rrcfir
    from scipy import stats
    h = upsampled_channel("h1", 2)
    M = (len(h) - 1) // 2 + 1
    amps, P, _, _ = awgn_constants("16-QAM", 0.1, 15.0)
    N, R = 250000, 2
    rx, tx, lev, sig = generate_frames_awgn_gpu(N, amps, [15.0, 15.0], np.stack([P, P]), h, 2, "cuda", [3, 4], n_frames=2, return_parts=True)
    assert rx.shape == (R, 2, 2, 2 * N) and tx.shape == (R, 2, 2, N) and tx.dtype == torch.float16
    levels = lev.cpu().numpy()
    cnt = np.array([(levels == np.float32(a)).sum() for a in amps])
    assert cnt.sum() == levels.size
    chi2 = ((cnt - levels.size * P) ** 2 / (levels.size * P)).sum()
    assert chi2 < stats.chi2.ppf(0.9999, len(amps) - 1), (cnt, P)
    sl = slice(PULSE_SPAN + M - 1, N + PULSE_SPAN + M - 1)
    assert torch.equal(tx.cpu(), lev[..., sl].cpu().to(torch.float16))
    # noise-free signal against np.convolve of the kernel's own levels with rrc, then h_channel ('valid', 2 sps)
    L = levels[0, 0, :, :3000].astype(np.float64)
    up = np.zeros(2 * (L.shape[1] - 1) + 1, dtype=np.complex128)
    up[::2] = L[0] + 1j * L[1]
    ref = np.convolve(np.convolve(up, rrcfir(PULSE_SPAN, 2, ROLLOFF).astype(np.float64), "valid"), h.astype(np.complex128), "valid")
    got = sig[0, 0, :ref.size].cpu().numpy()
    assert np.abs(got - ref).max() < 1e-5
    # realised SNR at 10^6 samples (per frame: 2 * 250000 complex samples, both frames)
    s, x = sig[..., :2 * N].cpu().numpy(), rx.cpu().numpy()
    noise = (x[:, :, 0] - s.real) + 1j * (x[:, :, 1] - s.imag)
    snr = 10 * np.log10(2 * np.mean(np.abs(s) ** 2) / 2 / np.mean(np.abs(noise) ** 2) * 2)
    assert abs(snr - 15.0) < 0.1, snr
    # a run's frames alone and inside a batch of 37
    seeds = list(range(100, 137))
    rx1, tx1 = generate_frames_awgn_gpu(2000, amps, [15.0], P[None], h, 2, "cuda", [seeds[17]], frame0=5, n_frames=3)
    rxb, txb = generate_frames_awgn_gpu(2000, amps, [12.0] * 17 + [15.0] + [18.0] * 19, np.stack([P] * 37), h, 2, "cuda", seeds, frame0=5, n_frames=3)
    assert torch.equal(rx1[0], rxb[17]) and torch.equal(tx1[0], txb[17])


def _cells(n, SNR=20.0, lr=5e-3):
    return [dict(SNR=SNR + (i % 3), nu=0.0 if i % 2 == 0 else 0.05, lr_optim=lr * (1 + 0.25 * (i % 4)), seed=11 + i) for i in range(n)]


@pytest.mark.parametrize("channel", ["h1", "h2"])
def test_sweep_numpy_datagen_equals_driver(channel):
    from vae_equalizer_b200.processing import processing_vaele_awgn
    from vae_equalizer_b200.sweep import sweep_vae_awgn
    cells = _cells(3)
    args = ("16-QAM", 2, 25, 350, 4000, 1200, 24, 6, channel)
    ser = sweep_vae_awgn(cells, *args, datagen="numpy")
    assert ser.shape == (3, 4)
    for r, c in enumerate(cells):
        ref = processing_vaele_awgn("16-QAM", 2, c["SNR"], c["nu"], 25, c["lr_optim"], 350, 4000, 1200, 24, 6, channel,
                                    rng=np.random.default_rng(c["seed"]), verbose=False)
        assert torch.equal(ser[r], ref), (r, ser[r].tolist(), ref.tolist())


def test_sweep_gpu_datagen_batch_independent_and_converges():
    """Blind VAE-LE training from the Dirac start does not converge for every seed: at this setting about 4 cells in 10 stay near SER
    0.8 (the reference algorithm's own behaviour, measured on B200 with the device generator), and WHICH seeds converge moves with any
    last-bit change of the step.  So convergence is asserted over 41 cells: at least a third must end below SER 1e-2 (23 of 41 do; 14
    is about 3 standard deviations below that)."""
    from vae_equalizer_b200.sweep import sweep_vae_awgn
    cells = [dict(SNR=20.0, nu=0.0, lr_optim=5e-3, seed=s) for s in (1, 2, 3, 4)] + _cells(5)
    cells += [dict(SNR=20.0, nu=0.0, lr_optim=5e-3, seed=s) for s in range(100, 132)]
    args = ("16-QAM", 2, 25, 350, 5000, 1200, 200, 50, "h1")       # the setting of test_dropin_awgn_runs, trained longer
    ser = sweep_vae_awgn(cells, *args, datagen="gpu")
    alone = sweep_vae_awgn([cells[2]], *args, datagen="gpu")
    assert torch.equal(alone[0], ser[2])
    assert torch.isfinite(ser).all()
    assert bool((ser[:, 0] > 0.5).all()), ser[:, 0].tolist()        # the validation after the first epoch is far from converged
    converged = int((ser[:, -1] < 0.01).sum())
    assert 3 * converged >= len(cells), ser[:, -1].tolist()


def test_sweep_gpu_datagen_tx_alignment():
    """An equalizer trained on device-generated frames detects the same shift on a device-generated and on a host-generated validation
    frame of the same channel: a misaligned tx slice of the generator would move it."""
    from vae_equalizer_b200 import awgn
    from vae_equalizer_b200.constants import awgn_constants, upsampled_channel
    R = 4
    for channel in ("h1", "h2"):
        h = upsampled_channel(channel, 2)
        amps, P, am, var = awgn_constants("16-QAM", 0.0, 20.0)
        M = (len(h) - 1) // 2 + 1
        seeds = [7, 8, 9, 10]
        rx, _ = awgn.generate_frames_awgn_gpu(1200, amps, [20.0] * R, np.stack([P] * R), h, 2, "cuda", seeds, n_frames=200)
        eqr = awgn.AWGNEqualizerRuns(R, 25, 2, amps, np.stack([P] * R), [am] * R, [var] * R)
        eqr.train_frames(rx, torch.full((R,), 5e-3, device="cuda"), 350, 1200)
        amp_t = torch.tensor(amps, dtype=torch.float32)
        rx_g, tx_g = awgn.generate_frames_awgn_gpu(5000, amps, [20.0] * R, np.stack([P] * R), h, 2, "cuda", seeds, frame0=1 << 20)
        sh_g, _, ser_g = awgn.awgn_eval_runs(eqr.forward(rx_g[:, 0])[0], tx_g[:, 0], amp_t)
        rng = np.random.default_rng(3)
        v = [awgn.generate_data(5000, M, amps, 20.0, h, 2, "cuda", P, rng=rng) for _ in range(R)]
        sh_n, _, ser_n = awgn.awgn_eval_runs(eqr.forward(torch.stack([x[0] for x in v]))[0], torch.stack([x[1] for x in v]), amp_t)
        ok = [r for r in range(R) if float(ser_g[r]) < 0.3]
        assert ok, (channel, ser_g.tolist())
        for r in ok:
            assert float(ser_n[r]) < 0.3 and int(sh_g[r]) == int(sh_n[r]), (channel, r, sh_g.tolist(), sh_n.tolist(), ser_n.tolist())


SWEEP = dict(mod="16-QAM", channel="h1", N_train_vec=[200, 350], lr_optim_vec=[3e-3, 5e-3], M_vec=[25], SNR_vec=[16, 20], nu_vec=[0.0], iter=2,
             N_valid=3000, train_len=1200, num_epochs=6, epe=3)


def _worker(rank, world, port, resq):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        from vae_equalizer_b200.sweep import run_awgn_sweep
        res = run_awgn_sweep(**SWEEP, rank=rank, world=world)
        resq.put((rank, None if res is None else res[0].cpu().numpy()))
    finally:
        dist.destroy_process_group()


def test_run_awgn_sweep_two_gpus_equals_one():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    import torch.multiprocessing as mp
    from vae_equalizer_b200.sweep import run_awgn_sweep
    ser1, _ = run_awgn_sweep(**SWEEP)
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    resq = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, resq)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([resq.get(timeout=300) for _ in range(2)], key=lambda t: t[0])
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    assert res[1][1] is None and np.array_equal(res[0][1], ser1.cpu().numpy())
