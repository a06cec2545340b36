"""Host logic of GMI in the sweep engines (run_dp_sweep / run_awgn_sweep with gmi=True): layout of the GMI array through a stub runner,
checkpoint names and signatures unchanged with gmi=False, no reuse across gmi=True / gmi=False files, the .mat GMI key and the inputs
the engines reject.  No GPU."""
import os

import numpy as np
import pytest
import torch

DP = dict(SNR_vec=[20, 23], nu_vec=[0.0], theta_diff_vec=[0.06 * np.pi], theta_vec=[np.pi / 10], M_vec=[9, 25], lr_optim_vec=[2.5e-3],
          batch_len_vec=[100], flex_step_vec=[10], symb_rate_vec=[90e9])
AW = dict(N_train_vec=[200], lr_optim_vec=[2e-3], M_vec=[9, 25], SNR_vec=[12], nu_vec=[0.0, 0.05], iter=1, num_epochs=4, epe=2)

# checkpoint file -> stored signature of the sweeps below with gmi=False, as written before GMI existed
PINNED_DP = {
    "VAE_64-QAM_M25_B100_F10_R9e+10_n2_f2_816092b27ca8.npz": "816092b27ca894eb30649ddd667f91de775ebc324dbb4176db54e13bdf9f8821",
    "VAE_64-QAM_M9_B100_F10_R9e+10_n2_f2_dc4b3c14e6aa.npz": "dc4b3c14e6aa01a9b64cbdce69fb286c3ec039a00a1f74ac078182916920479d",
}
PINNED_AWGN = {
    "AWGN_16-QAM_M25_B200_n2_e4_2bc2104cea30.npz": "2bc2104cea30dc247f193bd239e5f47ccc0a21559ae33dd0aabdfc2dfd833c3c",
    "AWGN_16-QAM_M9_B200_n2_e4_c579a49e0304.npz": "c579a49e030437a4bc05d2bb070891c1fad3fe3ec00e58427855e28ae759aac9",
}


def _dp_runner(calls, offset=0.0):
    """Stands for sweep_vae_dp_sharded: SER / Var_est / var / GMI encode the cell's seed, GMI negative on odd seeds, NaN on frame 1."""
    def runner(cells, mod, sps, M, batch_len, N_frame_max, num_frames, gmi=False, **kw):
        calls.append((M, len(cells), gmi))
        n = len(cells)
        seed = torch.tensor([float(c["seed"]) for c in cells])
        ser = seed.view(n, 1, 1).expand(n, 4, num_frames) + offset
        ve, var = 2 * seed.view(n, 1, 1).expand(n, 2, num_frames).clone(), 3 * seed.view(n, 1).expand(n, 2).clone()
        if not gmi:
            return ser, ve, var
        g = (seed * torch.where(seed % 2 == 1, -1.0, 1.0)).view(n, 1, 1) + torch.arange(2.0).view(1, 2, 1) * 0.5 + offset
        g = g.expand(n, 2, num_frames).clone()
        g[:, :, 1] = float("nan")
        return ser, ve, var, g
    return runner


def _aw_runner(calls, offset=0.0):
    def runner(cells, mod, sps, M, batch_len, N_valid, N_train, num_epochs, epe, channel, gmi=False):
        calls.append((M, len(cells), gmi))
        ser = torch.stack([torch.full((num_epochs // epe,), float(c["seed"]) + offset) for c in cells])
        return (ser, -ser - 0.25) if gmi else ser
    return runner


def test_run_dp_sweep_gmi_layout():
    from vae_equalizer_b200 import sweep
    calls = []
    SER, Var_est, var_real, GMI = sweep.run_dp_sweep(iter=2, num_frames=3, runner=_dp_runner(calls), gmi=True, **DP)
    assert all(c[2] for c in calls)
    assert GMI.shape == Var_est.shape == (2, 2, 1, 1, 1, 2, 1, 1, 1, 1, 2, 3)
    for idx in np.ndindex(*GMI.shape[1:-1]):
        seed = float(SER[(0,) + idx + (0,)])
        sign = -1.0 if int(seed) % 2 else 1.0
        for p in range(2):
            g = GMI[(p,) + idx]
            assert float(g[0]) == sign * seed + 0.5 * p and float(g[2]) == float(g[0]) and torch.isnan(g[1]), (idx, p)
    # gmi=False: exactly the three results of before, runner called without the keyword
    calls2 = []
    res = sweep.run_dp_sweep(iter=2, num_frames=3, runner=_dp_runner(calls2), **DP)
    assert len(res) == 3 and not any(c[2] for c in calls2)
    assert torch.equal(res[0], SER) and torch.equal(res[1], Var_est) and torch.equal(res[2], var_real)


def test_run_awgn_sweep_gmi_layout():
    from vae_equalizer_b200 import sweep
    calls = []
    SER, epochs, GMI = sweep.run_awgn_sweep(mod="16-QAM", runner=_aw_runner(calls), gmi=True, **AW)
    assert all(c[2] for c in calls) and list(epochs) == [0, 2]
    assert GMI.shape == SER.shape == (1, 1, 2, 1, 2, 1, 2)
    assert torch.equal(GMI, -SER - 0.25)
    res = sweep.run_awgn_sweep(mod="16-QAM", runner=_aw_runner([]), **AW)
    assert len(res) == 2 and torch.equal(res[0], SER)


def _files(ck):
    return {f: str(np.load(os.path.join(ck, f))["signature"]) for f in sorted(os.listdir(ck))}


def test_checkpoint_names_and_signatures_pinned_without_gmi(tmp_path):
    from vae_equalizer_b200 import sweep
    ck_dp, ck_aw = str(tmp_path / "dp"), str(tmp_path / "aw")
    sweep.run_dp_sweep(iter=1, num_frames=2, runner=_dp_runner([]), checkpoint_dir=ck_dp, **DP)
    sweep.run_awgn_sweep(mod="16-QAM", runner=_aw_runner([]), checkpoint_dir=ck_aw, **AW)
    assert _files(ck_dp) == PINNED_DP
    assert _files(ck_aw) == PINNED_AWGN
    for ck in (ck_dp, ck_aw):
        for f in os.listdir(ck):
            assert "gmi" not in np.load(os.path.join(ck, f)).files


def test_dp_checkpoints_never_cross_reused(tmp_path):
    from vae_equalizer_b200 import sweep
    ck = str(tmp_path / "ck")
    calls = []
    a = sweep.run_dp_sweep(iter=1, num_frames=2, runner=_dp_runner(calls), checkpoint_dir=ck, **DP)
    n = len(calls)
    b = sweep.run_dp_sweep(iter=1, num_frames=2, runner=_dp_runner(calls, offset=0.5), checkpoint_dir=ck, gmi=True, **DP)
    assert len(calls) == 2 * n and len(os.listdir(ck)) == 4                  # the gmi=False files are not loaded: recomputed, new files
    assert set(PINNED_DP) < set(_files(ck))
    assert torch.equal(b[0], a[0] + 0.5)
    for f in set(_files(ck)) - set(PINNED_DP):
        assert "gmi" in np.load(os.path.join(ck, f)).files
    c = sweep.run_dp_sweep(iter=1, num_frames=2, runner=_dp_runner(calls, offset=1.0), checkpoint_dir=ck, gmi=True, **DP)
    assert len(calls) == 2 * n                                                  # gmi=True reloads its own files, GMI included
    assert all(torch.allclose(x, y, rtol=0, atol=0, equal_nan=True) for x, y in zip(b, c))
    d = sweep.run_dp_sweep(iter=1, num_frames=2, runner=_dp_runner(calls, offset=1.0), checkpoint_dir=ck, **DP)
    assert len(calls) == 2 * n and len(d) == 3 and torch.equal(d[0], a[0])       # gmi=False reloads its own files, not the gmi=True ones


def test_awgn_checkpoints_never_cross_reused(tmp_path):
    from vae_equalizer_b200 import sweep
    ck = str(tmp_path / "ck")
    calls = []
    a = sweep.run_awgn_sweep(mod="16-QAM", runner=_aw_runner(calls), checkpoint_dir=ck, **AW)
    n = len(calls)
    b = sweep.run_awgn_sweep(mod="16-QAM", runner=_aw_runner(calls, offset=0.5), checkpoint_dir=ck, gmi=True, **AW)
    assert len(calls) == 2 * n and len(os.listdir(ck)) == 4 and torch.equal(b[0], a[0] + 0.5)
    c = sweep.run_awgn_sweep(mod="16-QAM", runner=_aw_runner(calls, offset=1.0), checkpoint_dir=ck, gmi=True, **AW)
    assert len(calls) == 2 * n and torch.equal(c[0], b[0]) and torch.equal(c[2], b[2])
    d = sweep.run_awgn_sweep(mod="16-QAM", runner=_aw_runner(calls, offset=1.0), checkpoint_dir=ck, **AW)
    assert len(calls) == 2 * n and len(d) == 2 and torch.equal(d[0], a[0])


def test_save_mat_with_and_without_gmi(tmp_path):
    from scipy import io
    from vae_equalizer_b200 import sweep
    SER, Var_est, var_real, GMI = sweep.run_dp_sweep(iter=1, num_frames=3, runner=_dp_runner([]), gmi=True, **DP)
    lists = dict(SNR_vec=DP["SNR_vec"], nu_vec=DP["nu_vec"], theta_diff_vec=DP["theta_diff_vec"], theta_vec=DP["theta_vec"], M_vec=DP["M_vec"],
                 lr_optim_vec=DP["lr_optim_vec"], batch_len_vec=DP["batch_len_vec"], symb_rate_vec=DP["symb_rate_vec"],
                 flex_step_vec=DP["flex_step_vec"])
    p0, p1 = str(tmp_path / "a.mat"), str(tmp_path / "b.mat")
    sweep.save_mat(p0, SER, Var_est, var_real, **lists)
    sweep.save_mat(p1, SER, Var_est, var_real, GMI=GMI, **lists)
    d0, d1 = io.loadmat(p0)["dict"], io.loadmat(p1)["dict"]
    assert "GMI" not in d0.dtype.names and set(d1.dtype.names) == set(d0.dtype.names) | {"GMI"}
    g = d1["GMI"][0, 0]
    assert g.shape == tuple(GMI.shape) and np.array_equal(np.isnan(g), torch.isnan(GMI).numpy())
    assert np.array_equal(np.nan_to_num(g), torch.nan_to_num(GMI).numpy()) and (g[~np.isnan(g)] < 0).any()
    for k in d0.dtype.names:
        assert np.array_equal(d0[k][0, 0], d1[k][0, 0]), k


def test_engines_reject_per_cell_gmi_and_cpu_tensors():
    from vae_equalizer_b200 import sweep
    from vae_equalizer_b200._lib import VaeqError
    from vae_equalizer_b200.awgn import awgn_gmi_runs
    from vae_equalizer_b200.shared_funcs import gmi_runs
    cells = [dict(SNR=23, nu=0.0, lr_optim=2.5e-3)]
    for kind in ("VAE", "VAEflex"):
        with pytest.raises(ValueError):
            sweep.sweep_vae_dp(cells, "64-QAM", 2, 25, 100, 1000, 1, 10, kind=kind, eval_mode="per_cell", gmi=True)
    with pytest.raises(ValueError):
        sweep.sweep_cma_dp(cells, "64-QAM", 2, 25, 100, 1000, 1, eval_mode="per_cell", gmi=True)
    with pytest.raises(VaeqError):
        sweep.sweep_vae_awgn(cells, "16-QAM", 2, 25, 350, 15000, 1200, 20, 10, "h1", device="cpu", gmi=True)
    R, n, N = 2, 4, 300
    q = torch.full((R, 2, 2 * n, N), 1.0 / n)
    tx = torch.zeros(R, 2, 2, N, dtype=torch.float16)
    with pytest.raises(VaeqError):
        gmi_runs(q, tx, torch.full((n,), 1.0 / n), torch.zeros(R, 2, 4, dtype=torch.int32), torch.zeros(R, 2, 2, 2, 4, dtype=torch.int32), 100)
    with pytest.raises(VaeqError):
        awgn_gmi_runs(q[:, 0], tx[:, 0], torch.full((n,), 1.0 / n), torch.zeros(R, dtype=torch.int32), torch.zeros(R, 4, dtype=torch.int32))


# ---- multi-rank gathers with GMI: two gloo processes, engines replaced by stubs (the gathers are host logic) ----------------------------
NF, NV = 3, 2


def _stub_vals(cells, shape, scale):
    """Per cell: values of either sign from the cell's seed, NaN in the second slot of the last axis."""
    seed = torch.tensor([float(c["seed"]) for c in cells]).view((-1,) + (1,) * len(shape))
    t = (scale * (seed + 1) * torch.where(seed % 2 == 1, -1.0, 1.0)).expand((len(cells),) + shape).clone()
    t[..., 1] = float("nan")
    return t


def _stub_vae_dp(cells, *args, gmi=False, **kw):
    n = len(cells)
    res = (_stub_vals(cells, (4, NF), 0.01).abs(), _stub_vals(cells, (2, NF), 2.0).nan_to_num(0), _stub_vals(cells, (2,), 3.0).nan_to_num(0))
    return res + (_stub_vals(cells, (2, NF), 0.5),) if gmi else res


def _stub_cma_dp(cells, *args, gmi=False, **kw):
    res = (_stub_vals(cells, (4, NF), 0.02).abs(), torch.zeros(len(cells), 2, NF), _stub_vals(cells, (2,), 5.0).nan_to_num(0))
    return res + (_stub_vals(cells, (2, NF), -0.7),) if gmi else res


def _stub_vae_awgn(cells, *args, gmi=False, **kw):
    ser = _stub_vals(cells, (NV,), 0.03).abs().nan_to_num(0)
    return (ser, _stub_vals(cells, (NV,), 0.9)) if gmi else ser


def _sharded_all(rank, world, group=None):
    from vae_equalizer_b200 import sweep
    cells = [dict(SNR=20, nu=0.0, lr_optim=1e-3, seed=s) for s in range(5)]
    dev = torch.device("cpu")
    kw = dict(flex_step=10, channel="h0", symb_rate=90e9, tau_cd=0.0, tau_pmd=0.0, phiIQ=(0.0, 0.0), N_lrhalf=NF)
    out = [sweep.sweep_vae_dp_sharded(cells, "64-QAM", 2, 25, 100, 1000, NF, device=dev, rank=rank, world=world, group=group, gmi=True),
           sweep._cma_cells("CMA", cells, ("64-QAM", 2, 25, 100, 1000, NF), kw, dev, rank, world, group, NF, gmi=True),
           sweep.sweep_vae_awgn_sharded(cells, "16-QAM", 2, 25, 200, 3000, 1200, 2 * NV, 2, "h1", device=dev, rank=rank, world=world,
                                        group=group, gmi=True)]
    from vae_equalizer_b200.parallel import gather_cell_results
    marker = gather_cell_results({rank: torch.full((2,), 7.0 + rank)}, world, (2,), rank, world, group, dev)   # the sequences stayed aligned
    return out, marker


def _gloo_worker(rank, world, port, q):
    import torch.distributed as dist
    from vae_equalizer_b200 import sweep
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        sweep.sweep_vae_dp, sweep.sweep_cma_dp, sweep.sweep_vae_awgn = _stub_vae_dp, _stub_cma_dp, _stub_vae_awgn
        out, marker = _sharded_all(rank, world)
        q.put((rank, None if out[0] is None else [[t.numpy() for t in r] for r in out], None if marker is None else marker.tolist(),
               [r is None for r in out]))
    finally:
        dist.destroy_process_group()


def test_sharded_gmi_gathers_two_ranks_equal_one(monkeypatch):
    """sweep_vae_dp_sharded, _cma_cells and sweep_vae_awgn_sharded with gmi=True over two ranks: every rank takes part in every gather
    (a collective left to rank 0 would pair with another rank's next one), rank 0 gets the one-rank result with its negative and NaN
    GMI entries, the other ranks None."""
    import socket

    import torch.multiprocessing as mp
    from vae_equalizer_b200 import sweep
    monkeypatch.setattr(sweep, "sweep_vae_dp", _stub_vae_dp)
    monkeypatch.setattr(sweep, "sweep_cma_dp", _stub_cma_dp)
    monkeypatch.setattr(sweep, "sweep_vae_awgn", _stub_vae_awgn)
    one, _ = _sharded_all(0, 1)
    assert all(bool(torch.isnan(r[-1]).any()) and bool((r[-1] < 0).any()) for r in one)
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    try:
        res = sorted((q.get(timeout=120) for _ in range(2)), key=lambda t: t[0])
    finally:
        for p in procs:
            p.join(timeout=60)
            if p.is_alive():
                p.kill()
    assert all(p.exitcode == 0 for p in procs)
    (_, out0, marker0, _), (_, out1, marker1, none1) = res
    assert out1 is None and marker1 is None and all(none1)
    assert marker0 == [[7.0, 7.0], [8.0, 8.0]]
    for a, b in zip(out0, one):
        assert len(a) == len(b)
        for x, y in zip(a, b):
            assert np.array_equal(x, y.numpy(), equal_nan=True)
