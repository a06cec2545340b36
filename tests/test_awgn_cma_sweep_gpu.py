"""Batched AWGN single-polarisation CMA sweep engine (csrc/awgn_cma.cu k_cma1_runs and vaeq_awgn_cma_eval_runs, awgn_cma.CMA_runs /
awgn_cma_eval_runs, sweep.sweep_cma_awgn / run_awgn_cma_sweep) against the single-run operators, the single-run driver
processing_cma_awgn and the reference's driver golden."""
import os
import socket

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
T = torch.from_numpy
MODS = {2: "4-QAM", 4: "16-QAM", 8: "64-QAM"}


def _device_frames(R, F, N, mod="16-QAM", SNR=20.0, seed0=0, frame0=0, channel="h1"):
    from vae_equalizer_b200.awgn import generate_frames_awgn_gpu
    from vae_equalizer_b200.constants import awgn_constants, upsampled_channel
    amps, P, _, _ = awgn_constants(mod, 0.0, SNR)
    rx, tx = generate_frames_awgn_gpu(N, amps, [SNR] * R, np.stack([P] * R), upsampled_channel(channel, 2), 2, "cuda",
                                      list(range(seed0, seed0 + R)), frame0=frame0, n_frames=F)
    return amps, rx, tx


def _dirac(R, M, gen=None, jitter=0.0):
    h = torch.zeros(R, 2, M)
    h[:, 0, M // 2] = 1.0
    if jitter:
        h += jitter * torch.randn(R, 2, M, generator=gen)
    return h.cuda()


@pytest.mark.parametrize("M", [9, 25, 41])
@pytest.mark.parametrize("F", [1, 3])
def test_cma_runs_kernel_bitwise_against_single_calls(M, F):
    """4 runs with their own taps, lr and data: F training calls then the validation call of CMA per run give the batched out_v and taps
    bit for bit (M = 41 takes the two-slot instantiation)."""
    from vae_equalizer_b200 import awgn_cma as cm
    R = 4
    _, rx, _ = _device_frames(R, F, 1500, seed0=10 * M + F)
    _, rx_v, _ = _device_frames(R, 1, 2000, seed0=10 * M + F, frame0=1 << 20)
    lrs = [5e-4, 1e-3 / 3, 7.7e-4, 2e-4]                           # Python floats: the batched path must round them as CMA() does
    h = _dirac(R, M, torch.Generator().manual_seed(M), 0.01)
    h_single = [h[r].clone() for r in range(R)]
    out_v = cm.CMA_runs(rx, rx_v[:, 0], h, torch.tensor(lrs, dtype=torch.float32, device="cuda"), 2)
    assert out_v.shape == (R, 2, 2000)
    for r in range(R):
        for f in range(F):
            cm.CMA(rx[r, f].contiguous(), 1, h_single[r], lrs[r], 2, True)
        ref, _, _ = cm.CMA(rx_v[r, 0].contiguous(), 1, h_single[r], lrs[r], 2, False)
        assert torch.equal(out_v[r], ref), r
        assert torch.equal(h[r], h_single[r]), r


def _score_single(y, tx, amp):
    from vae_equalizer_b200 import awgn_cma as cm
    y = y.clone()
    shift = int(cm.find_shift_symb(y, tx, 21))
    ser, counts = cm.SER_CMA(y[:, 11 + shift:-11], tx[:, 11:-11 - shift], 2, amp, amp.numel(), "cuda", return_counts=True)
    return shift, counts, ser


def _check_scoring(y, tx, amp):
    from vae_equalizer_b200 import awgn_cma as cm
    y_before = y.clone()
    shift, counts, ser = cm.awgn_cma_eval_runs(y, tx, amp)
    assert torch.equal(y, y_before)                                # no in-place rescale
    assert shift.dtype == torch.int32 and counts.shape == (y.shape[0], 4) and ser.dtype == torch.float32
    for r in range(y.shape[0]):
        s1, c1, ser1 = _score_single(y[r], tx[r], amp)
        assert int(shift[r]) == s1 and torch.equal(counts[r], c1) and torch.equal(ser[r], ser1), (r, s1, int(shift[r]))
    return shift


def _trained_cpe_output(n_lev, N_valid=5000):
    """CPE output of a CMA trained on device frames at SNR 20, and the validation frame's tx."""
    from vae_equalizer_b200 import awgn_cma as cm
    amps, rx, _ = _device_frames(1, 12, 1500, MODS[n_lev], seed0=3)
    _, rx_v, tx_v = _device_frames(1, 1, N_valid, MODS[n_lev], seed0=3, frame0=1 << 20)
    out_v = cm.CMA_runs(rx, rx_v[:, 0], _dirac(1, 25), torch.tensor([5e-4], device="cuda"), 2)
    return torch.tensor(amps, dtype=torch.float32, device="cuda"), cm.CPE(out_v), tx_v[:, 0]


@pytest.mark.parametrize("n_lev", [2, 4, 8])
def test_scoring_every_shift_on_trained_output(n_lev):
    """Trained CPE output against its tx rolled by every shift in -10..10: shift, the four counts and the SER of every run equal the
    single-run find_shift_symb + SER_CMA."""
    amp, y, tx = _trained_cpe_output(n_lev)
    R = 21
    yR = y.expand(R, -1, -1).contiguous()
    txR = torch.stack([tx[0].roll(s, -1) for s in range(-10, 11)])
    shift = _check_scoring(yR, txR, amp)
    assert len(set(shift.tolist())) > 10, shift.tolist()           # the rolls move the detected shift


@pytest.mark.parametrize("n_lev", [2, 4, 8])
def test_scoring_threshold_branches(n_lev):
    """Constructed CPE outputs for the three branches of cm:133-140: I above 0.02 N; I below it with Q's maximum at least I's (Q wins);
    I below it and Q weaker (I kept)."""
    from vae_equalizer_b200 import awgn_cma as cm
    from vae_equalizer_b200.constants import awgn_constants
    amps = awgn_constants(MODS[n_lev], 0.0, 20.0)[0]
    amp = torch.tensor(amps, dtype=torch.float32, device="cuda")
    gen = torch.Generator().manual_seed(n_lev)
    R, N = 3, 4000
    tx = amp.cpu()[torch.randint(0, n_lev, (R, 2, N), generator=gen)].to(torch.float16)
    thr = 0.02 * N
    noise = 0.01 * torch.randn(R, 2, N, generator=gen)
    y = noise.clone()
    y[0] = tx[0].float().roll(4, -1) + noise[0]                      # strong: I correlation far above the threshold
    for r, (c, lag) in ((1, (1, 3)), (2, (0, -2))):                  # weak copy of tx Q (run 1) or tx I (run 2) in the I row
        eps = 0.5 * thr / float((tx[r, c, 10:1000].float() ** 2).sum())       # peak correlation about half the threshold
        y[r, 0] = eps * tx[r, c].float().roll(lag, -1) + noise[r, 0]
    y, tx = y.cuda().contiguous(), tx.cuda().contiguous()
    for r in range(R):
        _, corr = cm.find_shift_symb(y[r], tx[r], 21, return_corr=True)
        mI, mQ = float(corr[0].abs().max()), float(corr[1].abs().max())
        assert (mI >= thr) == (r == 0), (r, mI, mQ)
        if r:
            assert (mQ >= mI) == (r == 1), (r, mI, mQ)
    _check_scoring(y, tx, amp)


def test_reference_frames_replayed_as_run_zero():
    """The frames of the reference's driver golden as run 0 of a 3-run set through CMA_runs -> CPE -> awgn_cma_eval_runs: run 0's SER equals
    processing_cma_awgn on the same frames bit for bit and lies within 4 decisions of the reference's."""
    from vae_equalizer_b200 import awgn_cma as cm
    from vae_equalizer_b200.constants import awgn_constants
    from vae_equalizer_b200.processing import processing_cma_awgn
    g = np.load(os.path.join(GOLDEN, "awgncma_drv_16qam.npz"))
    SNR, nu, M, lr, N_valid, N_train, num_epochs, epe = [float(v) for v in g["args"]]
    M, N_valid, num_epochs, epe = int(M), int(N_valid), int(num_epochs), int(epe)
    frames = [(g[f"rx{i}"], g[f"tx{i}"]) for i in range(int(g["n_frames"]))]
    ref = processing_cma_awgn(str(g["mod"]), 2, SNR, nu, M, lr, N_valid, int(N_train), num_epochs, epe, str(g["channel"]), verbose=False,
                              datagen=iter(frames))
    amp = torch.tensor(awgn_constants(str(g["mod"]), nu, SNR)[0], dtype=torch.float32, device="cuda")

    def three(a):                                                    # run 0: the frame; runs 1, 2: other data of the same shape
        a = T(np.ascontiguousarray(a))
        return torch.stack((a, a.flip(0), -a.roll(7, -1))).cuda()
    R = 3
    h = _dirac(R, M)
    lrs = torch.tensor([lr, 2 * lr, 0.5 * lr], dtype=torch.float32, device="cuda")
    it, ser0 = iter(frames), []
    for k in range(num_epochs // epe):
        train = [next(it) for _ in range(1 if k == 0 else epe)]
        rx_v, tx_v = next(it)
        rx_t = torch.stack([three(rx) for rx, _ in train], dim=1)
        out_v = cm.CMA_runs(rx_t, three(rx_v), h, lrs, 2)
        _, _, ser = cm.awgn_cma_eval_runs(cm.CPE(out_v), three(tx_v).to(torch.float16), amp)
        ser0.append(ser[0])
    ser0 = torch.stack(ser0)
    assert torch.equal(ser0, ref), (ser0.tolist(), ref.tolist())
    assert np.abs(ser0.cpu().numpy() - g["SER"]).max() <= 4.0 / (N_valid - 30), (ser0, g["SER"])


def _cells(n, SNR=20.0, lr=5e-4):
    return [dict(SNR=SNR + (i % 3), nu=0.0 if i % 2 == 0 else 0.05, lr_optim=lr * (1 + 0.25 * (i % 4)), seed=11 + i) for i in range(n)]


@pytest.mark.parametrize("channel", ["h1", "h2"])
def test_sweep_numpy_datagen_equals_driver(channel):
    from vae_equalizer_b200.processing import processing_cma_awgn
    from vae_equalizer_b200.sweep import sweep_cma_awgn
    cells = _cells(3)
    args = ("16-QAM", 2, 25, 4000, 1200, 24, 6, channel)
    ser = sweep_cma_awgn(cells, *args, datagen="numpy")
    assert ser.shape == (3, 4)
    for r, c in enumerate(cells):
        ref = processing_cma_awgn("16-QAM", 2, c["SNR"], c["nu"], 25, c["lr_optim"], 4000, 1200, 24, 6, channel,
                                  rng=np.random.default_rng(c["seed"]), verbose=False)
        assert torch.equal(ser[r], ref), (r, ser[r].tolist(), ref.tolist())


def test_sweep_gpu_datagen_batch_independent_and_converges():
    from vae_equalizer_b200.sweep import sweep_cma_awgn
    cells = [dict(SNR=20.0, nu=0.0, lr_optim=5e-4, seed=s) for s in (1, 2, 3, 4)] + _cells(5)
    args = ("16-QAM", 2, 25, 5000, 1200, 20, 5, "h1")
    ser = sweep_cma_awgn(cells, *args, datagen="gpu")
    alone = sweep_cma_awgn([cells[2]], *args, datagen="gpu")
    assert torch.equal(alone[0], ser[2])
    assert torch.isfinite(ser).all()
    for r in range(4):
        assert float(ser[r, -1]) < float(ser[r, 0]), ser[r].tolist()


def test_sweep_gpu_datagen_uses_the_vaele_sweeps_frames(monkeypatch):
    """Both AWGN sweeps draw the same training and validation frames for the same cells: the CMA baseline and the VAE-LE are compared
    on identical data."""
    from vae_equalizer_b200 import awgn, sweep
    real = awgn.generate_frames_awgn_gpu
    seen = {}

    def recording(key):
        def gen(*a, **kw):
            out = real(*a, **kw)
            seen.setdefault(key, []).append((kw.get("frame0"), kw.get("n_frames", 1), out[0].clone(), out[1].clone()))
            return out
        return gen
    cells = _cells(3)
    monkeypatch.setattr(awgn, "generate_frames_awgn_gpu", recording("vae"))
    sweep.sweep_vae_awgn(cells, "16-QAM", 2, 25, 350, 3000, 1200, 6, 3, "h1", datagen="gpu")
    monkeypatch.setattr(awgn, "generate_frames_awgn_gpu", recording("cma"))
    sweep.sweep_cma_awgn(cells, "16-QAM", 2, 25, 3000, 1200, 6, 3, "h1", datagen="gpu")
    assert len(seen["vae"]) == len(seen["cma"]) == 4
    valid = 0
    for (f0a, na, rxa, txa), (f0b, nb, rxb, txb) in zip(seen["vae"], seen["cma"]):
        assert (f0a, na) == (f0b, nb) and torch.equal(rxa, rxb) and torch.equal(txa, txb)
        valid += f0a >= sweep.AWGN_VALID_FRAME0
    assert valid == 2


def test_wrappers_reject_bad_dtypes_and_shapes():
    from vae_equalizer_b200 import awgn_cma as cm
    from vae_equalizer_b200._lib import VaeqError
    rx, rx_v, h, lr = torch.zeros(2, 1, 2, 3000, device="cuda"), torch.zeros(2, 2, 3000, device="cuda"), _dirac(2, 25), torch.ones(2, device="cuda")
    with pytest.raises(VaeqError):
        cm.CMA_runs(rx.double(), rx_v, h, lr, 2)
    with pytest.raises(VaeqError):
        cm.CMA_runs(rx, rx_v[:1], h, lr, 2)
    with pytest.raises(VaeqError):
        cm.CMA_runs(rx, rx_v, h, lr[:1], 2)
    with pytest.raises(VaeqError):
        cm.CMA_runs(rx, rx_v, _dirac(2, 24), lr, 2)                # even M: rejected by the library
    y, tx, amp = torch.zeros(2, 2, 3000, device="cuda"), torch.zeros(2, 2, 3000, dtype=torch.float16, device="cuda"), torch.ones(4, device="cuda")
    with pytest.raises(VaeqError):
        cm.awgn_cma_eval_runs(y, tx.float(), amp)
    with pytest.raises(VaeqError):
        cm.awgn_cma_eval_runs(y, tx[:, :, :2000], amp)
    with pytest.raises(VaeqError):
        cm.awgn_cma_eval_runs(y[:, :, :1005], tx[:, :, :1005], amp)   # find_shift_symb needs 1000 + n_shift // 2 symbols
    with pytest.raises(VaeqError):
        cm.awgn_cma_eval_runs(y, tx, torch.ones(3, device="cuda"))


SWEEP = dict(mod="16-QAM", channel="h1", lr_optim_vec=[3e-4, 5e-4], M_vec=[9, 25], SNR_vec=[16, 20], nu_vec=[0.0], iter=2, N_valid=3000,
             N_train=1200, num_epochs=6, epe=3)


def _worker(rank, world, port, resq):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        from vae_equalizer_b200.sweep import run_awgn_cma_sweep
        res = run_awgn_cma_sweep(**SWEEP, rank=rank, world=world)
        resq.put((rank, None if res is None else res[0].cpu().numpy()))
    finally:
        dist.destroy_process_group()


def test_run_awgn_cma_sweep_two_gpus_equals_one():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    import torch.multiprocessing as mp
    from vae_equalizer_b200.sweep import run_awgn_cma_sweep
    ser1, _ = run_awgn_cma_sweep(**SWEEP)
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
