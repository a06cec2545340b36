"""GMI next to SER in the batched sweep engines (csrc/eval_runs.cu k_gmi_runs, shared_funcs.gmi_runs, awgn.awgn_gmi_runs and the gmi=True
path of sweep_vae_dp / sweep_cma_dp / sweep_vae_awgn) against a float64 reference built from oracle.gmi_from_posteriors on the slice the
single-run drivers cut, under the (IQ flip, rotation) hypothesis of the SER."""
import os
import socket

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
PHI = np.array([0.0314, 0.0314], dtype=np.complex64)


def _oracle():
    from oracle import vaeq_oracle as O
    return O


def _hyp(c):
    """(flip, rotation) of the smallest count, counter order flip 0 rotations 0..3 then flip 1; the first wins ties."""
    h = int(torch.argmin(c.reshape(-1).cpu()))
    assert int(c.reshape(-1).cpu()[h]) == int(c.min()) and all(int(v) > int(c.min()) for v in c.reshape(-1).cpu()[:h])
    return h // 4, h % 4


def _rotate_tx(I, Q, flip, k):
    """tx rows whose levels index q for hypothesis (flip, k): level S - D of a symmetric constellation is amplitude -a (exact in fp16).
    New tensors, so that the rows may be assigned back into the tensor I and Q are views of."""
    I, Q = I.clone(), Q.clone()
    Qp = -Q if flip else Q
    return [(I, Qp), (-I, -Qp), (Qp, -I), (-Qp, I)][k]


def _gmi_ref_rows(qs, txs, P, hyps):
    """float64 GMI per pol of a materialised slice qs (2,2n,L), txs (2,2,L) under hyps[pol]."""
    O = _oracle()
    out = []
    for pol in range(2):
        tx2 = txs.clone()
        tx2[pol, 0], tx2[pol, 1] = _rotate_tx(txs[pol, 0], txs[pol, 1], *hyps[pol])
        out.append(float(O.gmi_from_posteriors(qs.double(), tx2, torch.as_tensor(P, dtype=torch.float32))[pol]) if qs.shape[-1] else float("nan"))
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
def test_frame_gmi_runs_against_oracle(n_lev, seg_len):
    from vae_equalizer_b200.shared_funcs import gmi_runs
    gen = torch.Generator().manual_seed(17 * n_lev + seg_len)
    R, N = 5, 2000
    shifts = list(range(-10, 11))
    for call in range(3):                                                     # every shift -10..10 across the runs of the calls
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
        g = gmi_runs(q.cuda(), tx.cuda(), P.cuda(), al.cuda(), counts.cuda(), seg_len).cpu()
        for r in range(R):
            hyps = [_hyp(counts[r, 0, :, p, :]) for p in range(2)]
            assert [h[0] * 4 + h[1] for h in hyps] == first[r]
            qs, ts = _dp_slice(q[r], tx[r], al[r, 0], seg_len)
            assert qs.shape[-1] == int(al[r, 0, 3])
            ref = _gmi_ref_rows(qs, ts, P[r], hyps)
            assert np.abs(g[r].double().numpy() - np.array(ref)).max() < 1e-6, (call, r, g[r].tolist(), ref)
    al[1, 0, 3] = 0                                                           # nothing evaluated: NaN, like the SER
    g = gmi_runs(q.cuda(), tx.cuda(), P[0].cuda(), al.cuda(), counts.cuda(), seg_len).cpu()
    assert torch.isnan(g[1]).all() and torch.isfinite(g[[0, 2, 3, 4]]).all()


@pytest.mark.parametrize("n_lev", [2, 4, 8])
def test_awgn_gmi_runs_against_oracle(n_lev):
    from vae_equalizer_b200.awgn import awgn_gmi_runs
    O = _oracle()
    gen = torch.Generator().manual_seed(5 + n_lev)
    R, N, edge = 7, 3000, 11
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
        g = awgn_gmi_runs(q.cuda(), tx.cuda(), P.cuda(), shift.cuda(), counts.cuda(), edge).cpu()
        for r in range(R):
            s, k = int(shift[r]), (call + r) % 4
            qs, ts = q[r][:, edge + s:N - edge], tx[r][:, edge:N - edge - s].clone()
            ts[0], ts[1] = _rotate_tx(ts[0], ts[1], 0, k)
            ref = float(O.gmi_from_posteriors(qs[None].double().repeat(2, 1, 1), ts[None].repeat(2, 1, 1), P[r])[0])
            assert abs(float(g[r]) - ref) < 1e-6, (call, r, float(g[r]), ref)


def test_awgn_gmi_runs_rejects_non_float32_q_and_shifts_before_the_row():
    """q must be float32 (its bits go to the kernel as is); a shift below -edge would start the scored window before the row: that run
    gives NaN and nothing is read, the other runs are unchanged."""
    from vae_equalizer_b200._lib import VaeqError
    from vae_equalizer_b200.awgn import awgn_gmi_runs
    gen = torch.Generator().manual_seed(9)
    R, n, N = 3, 4, 500
    q = torch.softmax(torch.randn(R, 2, n, N, generator=gen), dim=2).reshape(R, 2 * n, N).cuda()
    tx = _levels_tx((R, 2, N), n, gen)[0].cuda()
    P, counts = torch.full((n,), 1.0 / n).cuda(), torch.zeros(R, 4, dtype=torch.int32).cuda()
    for bad in (q.double(), q.half()):
        with pytest.raises(VaeqError):
            awgn_gmi_runs(bad, tx, P, torch.zeros(R, dtype=torch.int32).cuda(), counts)
    ok = awgn_gmi_runs(q, tx, P, torch.tensor([3, -3, 0], dtype=torch.int32).cuda(), counts, edge=3).cpu()       # -3 = -edge: the row's start
    g = awgn_gmi_runs(q, tx, P, torch.tensor([3, -3, -4], dtype=torch.int32).cuda(), counts, edge=3).cpu()
    assert torch.isfinite(ok).all() and torch.isnan(g[2]) and torch.equal(g[:2], ok[:2])


def _dp_cells(n, lr=2.5e-3):
    return [dict(SNR=20 + 2 * i, nu=[0.0, 0.0270955][i % 2], lr_optim=lr, theta=0.1 * i, theta_diff=0.02, seed=11 + i) for i in range(n)]


def _spy_gmi(monkeypatch):
    """Record every shared_funcs.gmi_runs call the engine makes (inputs and result)."""
    from vae_equalizer_b200 import shared_funcs as sfun
    calls, orig = [], sfun.gmi_runs

    def spy(q, tx, P, align, counts, seg_len, edge=11, n_cut=10):
        g = orig(q, tx, P, align, counts, seg_len, edge, n_cut)
        calls.append(dict(q=q.clone(), tx=tx.clone(), P=torch.as_tensor(P).clone(), align=align.clone(), counts=counts.clone(), seg_len=seg_len,
                          g=g.clone()))
        return g
    monkeypatch.setattr(sfun, "gmi_runs", spy)
    return calls


@pytest.mark.parametrize("kind", ["VAE", "VAEflex"])
def test_gmi_on_trained_posteriors(kind, monkeypatch):
    """One trained frame of 3 cells through sweep_vae_dp: the GMI of the engine against the oracle on the aligned, cut slice of the
    trained posteriors, and against shared_funcs.GMI of that slice where the SER's hypothesis is (0, 0)."""
    from vae_equalizer_b200 import shared_funcs as sfun, sweep
    calls = _spy_gmi(monkeypatch)
    _, _, _, G = sweep.sweep_vae_dp(_dp_cells(3), "64-QAM", 2, 25, 100, 2000, 1, flex_step=10, kind=kind, datagen="gpu", gmi=True)
    assert len(calls) == 1
    c = calls[0]
    assert torch.equal(c["g"], G[:, :, 0])
    n00 = 0
    for r in range(3):
        al = c["align"][r, 0].cpu()
        hyps = [_hyp(c["counts"][r, 0, :, p, :]) for p in range(2)]
        qs, ts = _dp_slice(c["q"][r].cpu(), c["tx"][r].cpu(), al, c["seg_len"])
        assert qs.shape[-1] == int(al[3]) > 0
        ref = _gmi_ref_rows(qs, ts, c["P"][r].cpu(), hyps)
        assert np.abs(c["g"][r].cpu().double().numpy() - np.array(ref)).max() < 1e-6, (r, c["g"][r].tolist(), ref)
        # shared_funcs.GMI of the slice: as is where the hypothesis is (0, 0), else with tx mapped onto the levels the hypothesis scores
        tx2 = ts.clone()
        for p in range(2):
            n00 += hyps[p] == (0, 0)
            tx2[p, 0], tx2[p, 1] = _rotate_tx(ts[p, 0], ts[p, 1], *hyps[p])
        g1 = sfun.GMI(qs.cuda().contiguous(), tx2.cuda().contiguous(), c["P"][r].cuda()).cpu()
        assert float((g1 - c["g"][r].cpu()).abs().max()) < 1e-6, (r, g1.tolist(), c["g"][r].tolist())
    print(kind, "pols scored under hypothesis (0, 0):", n00, "of 6")


def test_gmi_invariant_under_rotation_and_iq_flip():
    """q permuted into its pi/2-rotated, IQ-flipped copy: the batched SER counts pick (flip 1, rotation 2) where they picked (0, 0), and
    the GMI is the same."""
    from vae_equalizer_b200.shared_funcs import frame_eval_runs, gmi_runs
    gen = torch.Generator().manual_seed(3)
    for n in (2, 4, 8):
        R, N = 3, 3000
        tx, lev = _levels_tx((R, 2, 2, N), n, gen)
        q = _softmax_q(R, n, N, gen, lev, peak=3.0)
        qI, qQ = q[:, :, :n], q[:, :, n:]
        q2 = torch.cat((qQ.flip(2), qI.flip(2)), dim=2)                        # decisions (S - dQ, S - dI)
        amp = torch.linspace(-1, 1, n)
        P = torch.full((n,), 1.0 / n)
        var, nu = torch.full((R, 2), 0.1), torch.zeros(R)
        res = []
        for qq in (q, q2):
            qq = qq.cuda().contiguous()
            _, al, counts = frame_eval_runs(qq, None, tx.cuda(), amp.cuda(), var, nu, 0, which=1, return_counts=True)
            res.append((al.cpu(), counts.cpu(), gmi_runs(qq, tx.cuda(), P.cuda(), al, counts, 0).cpu()))
        (al1, c1, g1), (al2, c2, g2) = res
        assert torch.equal(al1[:, 0], al2[:, 0])
        for r in range(R):
            for p in range(2):
                assert _hyp(c1[r, 0, :, p, :]) == (0, 0) and _hyp(c2[r, 0, :, p, :]) == (1, 2), (n, r, p)
                assert int(c2[r, 0, 1, p, 2]) == int(c1[r, 0, 0, p, 0])
        assert float((g1 - g2).abs().max()) < 1e-6, (n, g1.tolist(), g2.tolist())


def _h_f32(P):
    P = torch.as_tensor(P, dtype=torch.float32).double()
    return (-2 * (P * torch.log2(P)).sum(-1)).float()


def _P_of(cells, mod, awgn=False):
    from vae_equalizer_b200.constants import awgn_constants, init
    if awgn:
        return torch.tensor(np.stack([awgn_constants(mod, float(c["nu"]), float(c["SNR"]))[1] for c in cells]), dtype=torch.float32)
    return torch.stack([torch.as_tensor(init("h0", mod, "cpu", float(c["nu"]), 2, 25, float(c["SNR"]))[2], dtype=torch.float32) for c in cells])


@pytest.mark.parametrize("kind", ["VAE", "VAEflex"])
def test_vae_dp_engine_gmi(kind):
    from vae_equalizer_b200 import sweep
    cells = _dp_cells(3)
    args = (cells, "64-QAM", 2, 25, 100, 2000, 3)
    kw = dict(flex_step=10, kind=kind, datagen="gpu", eval_every=2)
    base = sweep.sweep_vae_dp(*args, **kw)
    ser, ve, var, G = sweep.sweep_vae_dp(*args, **kw, gmi=True)
    assert torch.equal(ser.nan_to_num(-7), base[0].nan_to_num(-7)) and torch.equal(ve, base[1]) and torch.equal(var, base[2])
    assert G.shape == (3, 2, 3) and torch.isnan(G[:, :, 1]).all() and torch.isfinite(G[:, :, [0, 2]]).all()
    H = _h_f32(_P_of(cells, "64-QAM")).cuda()
    assert bool((G[:, :, [0, 2]] <= H.view(3, 1, 1)).all())
    alone = sweep.sweep_vae_dp([cells[1]], *args[1:], **kw, gmi=True)
    assert torch.equal(alone[3][0].nan_to_num(-7), G[1].nan_to_num(-7)) and torch.equal(alone[0][0].nan_to_num(-7), ser[1].nan_to_num(-7))


@pytest.mark.parametrize("kind", ["CMA", "CMAbatch", "CMAflex"])
def test_cma_dp_engine_gmi(kind):
    from vae_equalizer_b200 import sweep
    lr = {"CMA": 1e-3, "CMAbatch": 1e-5, "CMAflex": 1e-6}[kind]
    cells = _dp_cells(3, lr)
    args = (cells, "64-QAM", 2, 25, 100, 3000, 2, 20, "h0", 90e9, -26e-24, 0.1e-12 * np.sqrt(1000), PHI, 2)
    base = sweep.sweep_cma_dp(*args, kind=kind, datagen="gpu")
    ser, ve, var, G = sweep.sweep_cma_dp(*args, kind=kind, datagen="gpu", gmi=True)
    assert torch.equal(ser, base[0]) and torch.equal(ve, base[1]) and torch.equal(var, base[2])
    assert G.shape == (3, 2, 2) and torch.isfinite(G).all()
    H = _h_f32(_P_of(cells, "64-QAM")).cuda()
    assert bool((G <= H.view(3, 1, 1)).all())
    alone = sweep.sweep_cma_dp([cells[2]], *args[1:], kind=kind, datagen="gpu", gmi=True)
    assert torch.equal(alone[3][0], G[2]) and torch.equal(alone[0][0], ser[2])


def test_vae_awgn_engine_gmi():
    from vae_equalizer_b200 import sweep
    cells = [dict(SNR=14 + 2 * i, nu=[0.0, 0.05][i % 2], lr_optim=3e-3, seed=5 + i) for i in range(3)]
    args = ("16-QAM", 2, 25, 200, 3000, 1200, 6, 3, "h1")
    base = sweep.sweep_vae_awgn(cells, *args)
    ser, G = sweep.sweep_vae_awgn(cells, *args, gmi=True)
    assert torch.equal(ser, base) and G.shape == (3, 2) and torch.isfinite(G).all()
    assert bool((G <= _h_f32(_P_of(cells, "16-QAM", awgn=True)).cuda().view(3, 1)).all())
    ser1, G1 = sweep.sweep_vae_awgn([cells[1]], *args, gmi=True)
    assert torch.equal(G1[0], G[1]) and torch.equal(ser1[0], ser[1])


DP_SWEEP = dict(SNR_vec=[18, 24], nu_vec=[0.0, 0.0270955], theta_diff_vec=[0.02], theta_vec=[0.1], M_vec=[25], lr_optim_vec=[2.5e-3],
                batch_len_vec=[100], flex_step_vec=[10], symb_rate_vec=[90e9], iter=1, num_frames=3, N_frame_max=2000, N_lrhalf=2,
                datagen="gpu", eval_every=2)
AW_SWEEP = dict(mod="16-QAM", channel="h1", N_train_vec=[200], lr_optim_vec=[3e-3], M_vec=[25], SNR_vec=[8, 16], nu_vec=[0.0, 0.05], iter=1,
                N_valid=3000, train_len=1200, num_epochs=6, epe=3)


def _worker(rank, world, port, resq):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        from vae_equalizer_b200.sweep import run_awgn_sweep, run_dp_sweep
        out = []
        for lt in ("VAE", "CMA"):
            res = run_dp_sweep(loss_type=lt, **dict(DP_SWEEP, lr_optim_vec=[2.5e-3] if lt == "VAE" else [1e-3]), rank=rank, world=world, gmi=True)
            out.append(None if res is None else [t.cpu().numpy() for t in res])
        res = run_awgn_sweep(**AW_SWEEP, rank=rank, world=world, gmi=True)
        out.append(None if res is None else [res[0].cpu().numpy(), res[2].cpu().numpy()])
        resq.put((rank, out))
    finally:
        dist.destroy_process_group()


def test_two_gpus_equal_one_with_gmi():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    import torch.multiprocessing as mp
    from vae_equalizer_b200.sweep import run_awgn_sweep, run_dp_sweep
    one = []
    for lt in ("VAE", "CMA"):
        res = run_dp_sweep(loss_type=lt, **dict(DP_SWEEP, lr_optim_vec=[2.5e-3] if lt == "VAE" else [1e-3]), gmi=True)
        one.append([t.cpu().numpy() for t in res])
    res = run_awgn_sweep(**AW_SWEEP, gmi=True)
    one.append([res[0].cpu().numpy(), res[2].cpu().numpy()])
    assert np.isnan(one[0][3]).any()                                           # unscored frames travel as NaN
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
