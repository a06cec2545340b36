"""The bit-metric decoding rate (BMI) of Gray-labelled bits and the bit LLRs on the GPU (csrc/eval_runs.cu k_gmi_runs<.., BITS>,
csrc/eval.cu k_gmi<.., BITS> and k_bit_llr; shared_funcs.bmi_runs / BMI / bit_llr, awgn.awgn_bmi_runs and the bmi=True path of
sweep_vae_dp / sweep_cma_dp / sweep_vae_awgn) against the float64 reference (tests/bmi_ref.py: bmi_from_posteriors, bit_llr_from_posteriors) on the
slice the single-run drivers cut, under the (IQ flip, rotation) hypothesis of the SER."""
import os
import socket

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
PHI = np.array([0.0314, 0.0314], dtype=np.complex64)
TOL = 1e-6                                                                  # absolute, bit per 2-D symbol (the GMI ops' gate)


def _gate(ref):
    """TOL plus half an fp32 ulp of the reference: the kernels sum in double and round once to fp32, so a BMI of magnitude above 16
    (untrained or confidently wrong posteriors) cannot be closer than that rounding to its float64 value."""
    return TOL + 0.5 * float(np.spacing(np.float32(np.abs(ref)).max()))


def _ref():
    import bmi_ref
    return bmi_ref


def _hyp(c):
    """(flip, rotation) of the smallest count in counter order (flip 0 rotations 0..3, then flip 1); the first wins ties."""
    h = int(torch.argmin(c.reshape(-1).cpu()))
    return h // 4, h % 4


def _rotate_tx(I, Q, flip, k):
    """tx rows whose levels are the q levels hypothesis (flip, k) scores (level S - D of a symmetric constellation is amplitude -a)."""
    I, Q = I.clone(), Q.clone()
    Qp = -Q if flip else Q
    return [(I, Qp), (-I, -Qp), (Qp, -I), (-Qp, I)][k]


def _bmi_ref_rows(qs, txs, P, hyps):
    """float64 BMI per pol of a materialised slice qs (2,2n,L), txs (2,2,L) under hyps[pol]."""
    B = _ref()
    out = []
    for pol in range(2):
        tx2 = txs.clone()
        tx2[pol, 0], tx2[pol, 1] = _rotate_tx(txs[pol, 0], txs[pol, 1], *hyps[pol])
        out.append(float(B.bmi_from_posteriors(qs, tx2, P)[pol]) if qs.shape[-1] else float("nan"))
    return out


def _dp_slice(q, tx, al, seg_len, edge=11, n_cut=10):
    """The aligned, cut slice of one run as sweep._score materialises it (VAELE_DP:70-89 / VAEflex_DP:74-84)."""
    from vae_equalizer_b200.processing import _align
    sh, r = [int(al[0]), int(al[1])], int(al[2])
    a = _align(q.clone(), sh, r)
    tail = edge + max(abs(sh[0]), abs(sh[1]))
    d = tx
    if seg_len:
        keep = seg_len - sh[0] - n_cut
        N = q.shape[-1]
        a = a.reshape(2, a.shape[1], N // seg_len, seg_len)[:, :, :, :keep].reshape(2, a.shape[1], -1)
        d = d.reshape(2, 2, N // seg_len, seg_len)[:, :, :, :keep].reshape(2, 2, -1)
    return a[:, :, edge:-tail], d[:, :, edge:-tail]


def _n_eval(sh0, sh1, N, seg_len, edge=11, n_cut=10):
    tail = edge + max(abs(sh0), abs(sh1))
    total = N
    if seg_len:
        keep = min(seg_len, seg_len - sh0 - n_cut)
        total = (N // seg_len) * keep if keep > 0 else 0
    return max(0, total - tail - edge)


def _levels_tx(shape, n, gen):
    S = n - 1
    lev = torch.randint(0, n, shape, generator=gen)
    return ((2 * lev - S).float() / S).to(torch.float16), lev


def _softmax_q(R, n, N, gen, tx_lev=None, peak=0.0):
    z = torch.randn(R, 2, 2, n, N, generator=gen)
    if tx_lev is not None:
        z += peak * torch.nn.functional.one_hot(tx_lev, n).permute(0, 1, 2, 4, 3).float()
    return torch.softmax(z, dim=3).reshape(R, 2, 2 * n, N)


def _counts_selecting(R, gen, first):
    """counts (R,2,2,2,4) whose estimator-0 minimum of (run, pol) sits at hypothesis first[run][pol]; odd runs repeat it at a later
    hypothesis (a tie the first must win)."""
    c = torch.randint(20, 60, (R, 2, 2, 2, 4), generator=gen, dtype=torch.int32)
    for r in range(R):
        for p in range(2):
            h = first[r][p]
            c[r, 0, h // 4, p, h % 4] = 3
            if r % 2 and h < 7:
                h2 = 7 if h != 7 else 6
                c[r, 0, h2 // 4, p, h2 % 4] = 3
    return c


@pytest.mark.parametrize("n_lev", [2, 4, 8])
@pytest.mark.parametrize("seg_len", [100, 0])
def test_frame_bmi_runs_against_float64(n_lev, seg_len):
    """Every shift -10..10 and all 8 hypotheses (ties included), VAE-LE minibatch cut (seg_len 100) and VAE-flex (0); at n_lev = 2 BMI is
    GMI."""
    from vae_equalizer_b200.shared_funcs import bmi_runs, gmi_runs
    gen = torch.Generator().manual_seed(31 * n_lev + seg_len)
    R, N = 5, 2000
    shifts = list(range(-10, 11))
    worst = 0.0
    for call in range(3):
        q = _softmax_q(R, n_lev, N, gen)
        tx, _ = _levels_tx((R, 2, 2, N), n_lev, gen)
        P = torch.rand(R, n_lev, generator=gen) + 0.1
        P = P / P.sum(1, keepdim=True)
        al = torch.zeros(R, 2, 4, dtype=torch.int32)
        for r in range(R):
            s0, s1 = shifts[(call * 2 * R + 2 * r) % 21], shifts[(call * 2 * R + 2 * r + 1) % 21]
            al[r, 0] = torch.tensor([s0, s1, (r + call) % 2, _n_eval(s0, s1, N, seg_len)])
            al[r, 1] = torch.tensor([7, -7, 1, 5])                            # estimator 1 row: never read
        first = [[(call * 10 + 2 * r + p) % 8 for p in range(2)] for r in range(R)]
        counts = _counts_selecting(R, gen, first)
        args = (q.cuda(), tx.cuda(), P.cuda(), al.cuda(), counts.cuda(), seg_len)
        b = bmi_runs(*args).cpu()
        for r in range(R):
            hyps = [_hyp(counts[r, 0, :, p, :]) for p in range(2)]
            assert [h[0] * 4 + h[1] for h in hyps] == first[r]
            qs, ts = _dp_slice(q[r], tx[r], al[r, 0], seg_len)
            ref = np.array(_bmi_ref_rows(qs, ts, P[r], hyps))
            err = float(np.abs(b[r].double().numpy() - ref).max())
            worst = max(worst, err)
            assert err < _gate(ref), (call, r, b[r].tolist(), ref)
        if n_lev == 2:
            assert float((b - gmi_runs(*args).cpu()).abs().max()) < TOL
    al[1, 0, 3] = 0                                                           # nothing evaluated: NaN, like the SER
    b = bmi_runs(q.cuda(), tx.cuda(), P[0].cuda(), al.cuda(), counts.cuda(), seg_len).cpu()
    assert torch.isnan(b[1]).all() and torch.isfinite(b[[0, 2, 3, 4]]).all()
    print(f"bmi_runs n_lev {n_lev} seg_len {seg_len}: largest |error| {worst:.2e}")


@pytest.mark.parametrize("n_lev", [2, 4, 8])
def test_awgn_bmi_runs_against_float64(n_lev):
    from vae_equalizer_b200.awgn import awgn_bmi_runs, awgn_gmi_runs
    B = _ref()
    gen = torch.Generator().manual_seed(7 + n_lev)
    R, N, edge = 7, 3000, 11
    worst = 0.0
    for call in range(3):
        q = torch.softmax(torch.randn(R, 2, n_lev, N, generator=gen), dim=2).reshape(R, 2 * n_lev, N)
        tx, _ = _levels_tx((R, 2, N), n_lev, gen)
        P = torch.rand(R, n_lev, generator=gen) + 0.1
        P = P / P.sum(1, keepdim=True)
        shift = torch.tensor([(call * R + r) % 21 - 10 for r in range(R)], dtype=torch.int32)
        counts = torch.randint(20, 60, (R, 4), generator=gen, dtype=torch.int32)
        for r in range(R):
            k = (call + r) % 4
            counts[r, k] = 2
            if r % 2 and k < 3:
                counts[r, 3] = 2                                              # tie: the first rotation wins
        args = (q.cuda(), tx.cuda(), P.cuda(), shift.cuda(), counts.cuda(), edge)
        b = awgn_bmi_runs(*args).cpu()
        for r in range(R):
            s, k = int(shift[r]), (call + r) % 4
            qs, ts = q[r][:, edge + s:N - edge], tx[r][:, edge:N - edge - s].clone()
            ts[0], ts[1] = _rotate_tx(ts[0], ts[1], 0, k)
            ref = float(B.bmi_from_posteriors(qs[None].repeat(2, 1, 1), ts[None].repeat(2, 1, 1), P[r])[0])
            worst = max(worst, abs(float(b[r]) - ref))
            assert abs(float(b[r]) - ref) < _gate(ref), (call, r, float(b[r]), ref)
        if n_lev == 2:
            assert float((b - awgn_gmi_runs(*args).cpu()).abs().max()) < TOL
    print(f"awgn_bmi_runs n_lev {n_lev}: largest |error| {worst:.2e}")


@pytest.mark.parametrize("n_lev", [2, 4, 8])
def test_single_run_bmi_against_float64(n_lev):
    """shared_funcs.BMI on contiguous rows (16-byte loads) and on a view whose rows start one symbol in (per-symbol path)."""
    from vae_equalizer_b200.shared_funcs import BMI, GMI
    B = _ref()
    gen = torch.Generator().manual_seed(50 + n_lev)
    N = 20001
    tx, lev = _levels_tx((2, 2, N), n_lev, gen)
    q = _softmax_q(1, n_lev, N, gen, lev[None], peak=2.0)[0]
    P = torch.rand(n_lev, generator=gen) + 0.1
    P = P / P.sum()
    for sl in (slice(1, N), slice(0, N - 1)):
        qs, ts = q[:, :, sl], tx[:, :, sl]
        qd = q.cuda()[:, :, sl] if sl.start else qs.contiguous().cuda()
        td = tx.cuda()[:, :, sl] if sl.start else ts.contiguous().cuda()
        b = BMI(qd, td, P.cuda()).cpu().double()
        ref = B.bmi_from_posteriors(qs, ts, P)
        assert float((b - ref).abs().max()) < _gate(ref.numpy()), (sl, b.tolist(), ref.tolist())
        if n_lev == 2:
            assert float((b - GMI(qd, td, P.cuda()).cpu().double()).abs().max()) < TOL


def _llr_check(L, q):
    B = _ref()
    ref = B.bit_llr_from_posteriors(q)
    assert L.shape == ref.shape and L.dtype == torch.float32
    err = (L.double() - ref).abs()
    assert bool((err <= torch.clamp(1e-5 * ref.abs(), min=1e-5)).all()), float(err.max())


@pytest.mark.parametrize("n_lev", [2, 4, 8])
def test_bit_llr_against_float64_and_decisions(n_lev):
    """bit_llr of (R,2,2n,N) and (2,2n,N), aligned and as an unaligned view, against the float64 reference within max(1e-5, 1e-5 |L|).  Where a
    component's largest level posterior exceeds 1/2 (+ the fp32 tolerance of q), that level holds the majority of every bit's mass, so
    sign(L) must give the Gray bits of the argmax decision.  The BMI recomputed from the LLRs agrees with the kernel's BMI."""
    from vae_equalizer_b200.shared_funcs import BMI, bit_llr
    B = _ref()
    gen = torch.Generator().manual_seed(90 + n_lev)
    R, N, m = 3, 4096, n_lev.bit_length() - 1
    tx, lev = _levels_tx((R, 2, 2, N), n_lev, gen)
    q = _softmax_q(R, n_lev, N, gen, lev, peak=2.5)
    q[0, 0, 0, :7] = 0.0                                                        # posteriors of exactly 0: the 1e-30 clamp
    qd = q.cuda()
    L = bit_llr(qd)
    _llr_check(L.cpu(), q)
    _llr_check(bit_llr(qd[1]).cpu(), q[1])
    _llr_check(bit_llr(qd[:, :, :, 3:N - 2]).cpu(), q[:, :, :, 3:N - 2])     # per-symbol path: rows start 3 symbols in
    assert torch.equal(bit_llr(qd[:, :, :, 3:N - 2]).cpu(), L.cpu()[:, :, :, 3:N - 2])   # both paths: the same arithmetic
    bits = B.label_bits(n_lev)                                                 # (m, n)
    qc = q.reshape(R, 2, 2, n_lev, N)
    top, d = qc.max(dim=3)
    sure = top > 0.5 + 1e-6
    sign_bits = (L.cpu().reshape(R, 2, 2, m, N) < 0).long()
    dec_bits = bits[:, d].permute(1, 2, 3, 0, 4)                               # (R, 2, 2, m, N)
    assert int(sure.sum()) > R * 2 * 2 * N // 4
    assert torch.equal(sign_bits.permute(0, 1, 2, 4, 3)[sure], dec_bits.permute(0, 1, 2, 4, 3)[sure])
    # BMI from the LLRs: q(b = tx's bit | y) = sigmoid(+-L), the posteriors of q renormalised per bit
    P = torch.rand(n_lev, generator=gen) + 0.1
    P = P / P.sum()
    for r in range(1, R):                                                      # run 0 has the zeroed posteriors: its bits do not sum to 1
        idx = B._tx_levels(tx[r], n_lev)                                       # (2, 2, N)
        tb = bits[:, idx].permute(1, 2, 0, 3).reshape(2, 2 * m, N)             # tx bits, rows as the LLRs
        Lr = L[r].cpu().double()
        lp = -torch.nn.functional.softplus(torch.where(tb == 0, -Lr, Lr)) / np.log(2)
        H = float(-2 * (P.double() * torch.log2(P.double())).sum())
        from_llr = H + lp.sum(1).mean(-1)
        kern = BMI(qd[r].contiguous(), tx[r].cuda(), P.cuda()).cpu().double()
        assert float((from_llr - kern).abs().max()) < 1e-5, (r, from_llr.tolist(), kern.tolist())


def test_bit_llr_rejects_bad_input():
    from vae_equalizer_b200._lib import VaeqError
    from vae_equalizer_b200.shared_funcs import bit_llr
    q = torch.full((2, 2, 8, 64), 0.25, device="cuda")
    for bad in (q.double(), q[:, :, :6], q.transpose(2, 3), q[:, :, :, ::2]):
        with pytest.raises(VaeqError):
            bit_llr(bad)


# ---- engines --------------------------------------------------------------------------------------------------------------------------
def _dp_cells(n, lr=2.5e-3):
    return [dict(SNR=20 + 2 * i, nu=[0.0, 0.0270955][i % 2], lr_optim=lr, theta=0.1 * i, theta_diff=0.02, seed=11 + i) for i in range(n)]


def _h_f32(P):
    P = torch.as_tensor(P, dtype=torch.float32).double()
    return (-2 * (P * torch.log2(P)).sum(-1)).float()


def _P_of(cells, mod, awgn=False):
    from vae_equalizer_b200.constants import awgn_constants, init
    if awgn:
        return torch.tensor(np.stack([awgn_constants(mod, float(c["nu"]), float(c["SNR"]))[1] for c in cells]), dtype=torch.float32)
    return torch.stack([torch.as_tensor(init("h0", mod, "cpu", float(c["nu"]), 2, 25, float(c["SNR"]))[2], dtype=torch.float32) for c in cells])


def _launches(fn):
    from vae_equalizer_b200 import _lib
    lib = _lib.load()
    n0 = int(lib.vaeq_launch_count(-1))
    res = fn()
    torch.cuda.synchronize()
    return res, int(lib.vaeq_launch_count(-1)) - n0


@pytest.mark.parametrize("kind", ["VAE", "VAEflex"])
def test_bmi_on_trained_posteriors(kind, monkeypatch):
    """One trained frame of 3 cells through sweep_vae_dp: the engine's BMI against the float64 reference on the aligned, cut slice of the trained
    posteriors under the SER's hypothesis."""
    from vae_equalizer_b200 import shared_funcs as sfun, sweep
    calls, orig = [], sfun.bmi_runs

    def spy(q, tx, P, align, counts, seg_len, edge=11, n_cut=10):
        b = orig(q, tx, P, align, counts, seg_len, edge, n_cut)
        calls.append(dict(q=q.cpu(), tx=tx.cpu(), P=torch.as_tensor(P).cpu(), align=align.cpu(), counts=counts.cpu(), seg_len=seg_len, b=b.cpu()))
        return b
    monkeypatch.setattr(sfun, "bmi_runs", spy)
    _, _, _, B = sweep.sweep_vae_dp(_dp_cells(3), "64-QAM", 2, 25, 100, 2000, 1, flex_step=10, kind=kind, datagen="gpu", bmi=True)
    assert len(calls) == 1
    c = calls[0]
    assert torch.equal(c["b"], B[:, :, 0].cpu())
    worst = 0.0
    for r in range(3):
        al = c["align"][r, 0]
        hyps = [_hyp(c["counts"][r, 0, :, p, :]) for p in range(2)]
        qs, ts = _dp_slice(c["q"][r], c["tx"][r], al, c["seg_len"])
        assert qs.shape[-1] == int(al[3]) > 0
        ref = np.array(_bmi_ref_rows(qs, ts, c["P"][r], hyps))
        err = float(np.abs(c["b"][r].double().numpy() - ref).max())
        worst = max(worst, err)
        assert err < _gate(ref), (r, c["b"][r].tolist(), ref)
    print(kind, f"trained posteriors: largest |error| {worst:.2e}, BMI {c['b'].tolist()}")


@pytest.mark.parametrize("kind", ["VAE", "VAEflex"])
def test_vae_dp_engine_bmi(kind):
    from vae_equalizer_b200 import sweep
    cells = _dp_cells(3)
    args = (cells, "64-QAM", 2, 25, 100, 2000, 3)
    kw = dict(flex_step=10, kind=kind, datagen="gpu", eval_every=2)
    base, n_base = _launches(lambda: sweep.sweep_vae_dp(*args, **kw, gmi=True))
    res, n_bmi = _launches(lambda: sweep.sweep_vae_dp(*args, **kw, gmi=True, bmi=True))
    assert n_bmi - n_base == 2 * 2                                              # two launches per scored frame (frames 0 and 2)
    for a, b in zip(res[:4], base):
        assert torch.equal(a.nan_to_num(-7), b.nan_to_num(-7))
    B = res[4]
    assert B.shape == (3, 2, 3) and torch.isnan(B[:, :, 1]).all() and torch.isfinite(B[:, :, [0, 2]]).all()
    H = _h_f32(_P_of(cells, "64-QAM")).cuda()
    assert bool((B[:, :, [0, 2]] <= H.view(3, 1, 1) + 1e-5).all())
    alone = sweep.sweep_vae_dp([cells[1]], *args[1:], **kw, bmi=True)
    assert len(alone) == 4 and torch.equal(alone[3][0].nan_to_num(-7), B[1].nan_to_num(-7))
    print(kind, "BMI", B[:, :, [0, 2]].tolist(), "GMI", res[3][:, :, [0, 2]].tolist())


@pytest.mark.parametrize("kind", ["CMA", "CMAbatch", "CMAflex"])
def test_cma_dp_engine_bmi(kind):
    from vae_equalizer_b200 import sweep
    lr = {"CMA": 1e-3, "CMAbatch": 1e-5, "CMAflex": 1e-6}[kind]
    cells = _dp_cells(3, lr)
    args = (cells, "64-QAM", 2, 25, 100, 3000, 2, 20, "h0", 90e9, -26e-24, 0.1e-12 * np.sqrt(1000), PHI, 2)
    base, n_base = _launches(lambda: sweep.sweep_cma_dp(*args, kind=kind, datagen="gpu", gmi=True))
    res, n_bmi = _launches(lambda: sweep.sweep_cma_dp(*args, kind=kind, datagen="gpu", gmi=True, bmi=True))
    assert n_bmi - n_base == 2 * 2
    for a, b in zip(res[:4], base):
        assert torch.equal(a, b)
    B = res[4]
    assert B.shape == (3, 2, 2) and torch.isfinite(B).all()
    assert bool((B <= _h_f32(_P_of(cells, "64-QAM")).cuda().view(3, 1, 1) + 1e-5).all())
    alone = sweep.sweep_cma_dp([cells[2]], *args[1:], kind=kind, datagen="gpu", bmi=True)
    assert torch.equal(alone[3][0], B[2]) and torch.equal(alone[0][0], res[0][2])


def test_vae_awgn_engine_bmi():
    from vae_equalizer_b200 import sweep
    cells = [dict(SNR=14 + 2 * i, nu=[0.0, 0.05][i % 2], lr_optim=3e-3, seed=5 + i) for i in range(3)]
    args = ("16-QAM", 2, 25, 200, 3000, 1200, 6, 3, "h1")
    (ser0, G0), n_base = _launches(lambda: sweep.sweep_vae_awgn(cells, *args, gmi=True))
    (ser, G, B), n_bmi = _launches(lambda: sweep.sweep_vae_awgn(cells, *args, gmi=True, bmi=True))
    assert n_bmi - n_base == 2 * 2                                              # two validations
    assert torch.equal(ser, ser0) and torch.equal(G, G0) and B.shape == (3, 2) and torch.isfinite(B).all()
    assert bool((B <= _h_f32(_P_of(cells, "16-QAM", awgn=True)).cuda().view(3, 1) + 1e-5).all())
    ser1, B1 = sweep.sweep_vae_awgn([cells[1]], *args, bmi=True)
    assert torch.equal(B1[0], B[1]) and torch.equal(ser1[0], ser[1])
    print("AWGN BMI", B.tolist(), "GMI", G.tolist())


DP_SWEEP = dict(SNR_vec=[18, 24], nu_vec=[0.0, 0.0270955], theta_diff_vec=[0.02], theta_vec=[0.1], M_vec=[25], lr_optim_vec=[2.5e-3],
                batch_len_vec=[100], flex_step_vec=[10], symb_rate_vec=[90e9], iter=1, num_frames=3, N_frame_max=2000, N_lrhalf=2,
                datagen="gpu", eval_every=2)
AW_SWEEP = dict(mod="16-QAM", channel="h1", N_train_vec=[200], lr_optim_vec=[3e-3], M_vec=[25], SNR_vec=[8, 16], nu_vec=[0.0, 0.05], iter=1,
                N_valid=3000, train_len=1200, num_epochs=6, epe=3)


def _all_sweeps(**dist):
    from vae_equalizer_b200.sweep import run_awgn_sweep, run_dp_sweep
    out = []
    for lt in ("VAE", "CMA"):
        res = run_dp_sweep(loss_type=lt, **dict(DP_SWEEP, lr_optim_vec=[2.5e-3] if lt == "VAE" else [1e-3]), gmi=True, bmi=True, **dist)
        out.append(None if res is None else [t.cpu().numpy() for t in res])
    res = run_awgn_sweep(**AW_SWEEP, gmi=True, bmi=True, **dist)
    out.append(None if res is None else [res[0].cpu().numpy(), res[2].cpu().numpy(), res[3].cpu().numpy()])
    return out


def _worker(rank, world, port, resq):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        resq.put((rank, _all_sweeps(rank=rank, world=world)))
    finally:
        dist.destroy_process_group()


def test_two_gpus_equal_one_with_bmi():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    import torch.multiprocessing as mp
    one = _all_sweeps()
    assert np.isnan(one[0][4]).any()                                           # unscored frames travel as NaN
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    resq = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, resq)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([resq.get(timeout=600) for _ in range(2)], key=lambda t: t[0])
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    assert all(o is None for o in res[1][1])
    for a, b in zip(res[0][1], one):
        for x, y in zip(a, b):
            assert np.array_equal(x, y, equal_nan=True)
