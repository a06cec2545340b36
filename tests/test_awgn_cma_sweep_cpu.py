"""Host logic of the batched AWGN CMA sweep (sweep.run_awgn_cma_sweep / sweep_cma_awgn): result layout, loop order, seeds and run-set
grouping through a stub runner, checkpoint reuse next to VAE-LE checkpoints, and the inputs the engine rejects.  No GPU."""
import ctypes

import numpy as np
import pytest
import torch

LISTS = dict(lr_optim_vec=[2e-4, 5e-4, 1e-3], M_vec=[9, 25], SNR_vec=[10, 14], nu_vec=[0.0, 0.05], iter=2, num_epochs=6, epe=2)


def _runner(calls, seen=None, offset=0.0):
    def runner(cells, mod, sps, M, N_valid, N_train, num_epochs, epe, channel):
        calls.append((M, len(cells)))
        assert (N_valid, N_train, channel) == (15000, 1200, "h1")
        if seen is not None:
            seen.update({c["seed"]: dict(c, M=M) for c in cells})
        return torch.stack([torch.full((num_epochs // epe,), float(c["seed"] + 1000 * c["SNR"]) + offset) for c in cells])
    return runner


def test_run_awgn_cma_sweep_layout_order_seeds_and_grouping():
    from vae_equalizer_b200 import sweep
    calls, seen = [], {}
    SER, epochs = sweep.run_awgn_cma_sweep(mod="16-QAM", runner=_runner(calls, seen), **LISTS)
    assert SER.shape == (3, 2, 2, 2, 2, 3) and list(epochs) == [0, 2, 4]
    assert sorted(calls) == [(9, 24), (25, 24)]                                       # one set per M: lr x SNR x nu x iter
    shape = SER.shape[:-1]
    assert sorted(seen) == list(range(int(np.prod(shape))))                           # every cell once, seeded by its flat index
    for idx in np.ndindex(*shape):
        l, m, s, n, i = idx
        seed = int(np.ravel_multi_index(idx, shape))
        c = seen[seed]
        assert set(c) == {"SNR", "nu", "lr_optim", "seed", "M"}
        assert (c["lr_optim"], c["M"], c["SNR"], c["nu"]) == (LISTS["lr_optim_vec"][l], LISTS["M_vec"][m], LISTS["SNR_vec"][s],
                                                              LISTS["nu_vec"][n]), idx
        assert (SER[idx] == seed + 1000 * c["SNR"]).all(), idx


def test_run_awgn_cma_sweep_checkpoint_reuse_and_invalidation(tmp_path):
    from vae_equalizer_b200 import sweep
    calls = []
    ck = str(tmp_path / "ck")
    a = sweep.run_awgn_cma_sweep(mod="16-QAM", runner=_runner(calls), checkpoint_dir=ck, **LISTS)
    n = len(calls)
    b = sweep.run_awgn_cma_sweep(mod="16-QAM", runner=_runner(calls), checkpoint_dir=ck, **LISTS)
    assert len(calls) == n and torch.equal(a[0], b[0])
    c = sweep.run_awgn_cma_sweep(mod="16-QAM", runner=_runner(calls), checkpoint_dir=ck, **dict(LISTS, SNR_vec=[11, 15]))
    assert len(calls) == 2 * n and not torch.equal(c[0], a[0])
    d = sweep.run_awgn_cma_sweep(mod="64-QAM", runner=_runner(calls), checkpoint_dir=ck, **LISTS)      # other setting, same lists
    assert len(calls) == 3 * n and torch.equal(d[0], a[0])


def test_cma_and_vaele_checkpoints_do_not_collide(tmp_path):
    """A VAE-LE sweep and a CMA sweep over the same cells in one directory: each loads only its own sets."""
    from vae_equalizer_b200 import sweep
    ck = str(tmp_path / "ck")
    vae_calls = []

    def vae_runner(cells, mod, sps, M, batch_len, N_valid, N_train, num_epochs, epe, channel):
        vae_calls.append(M)
        return torch.stack([torch.full((num_epochs // epe,), -1.0 - c["seed"]) for c in cells])
    common = dict(mod="16-QAM", lr_optim_vec=[5e-4], M_vec=[9, 25], SNR_vec=[14], nu_vec=[0.0], iter=2, num_epochs=6, epe=2,
                  checkpoint_dir=ck)
    v = sweep.run_awgn_sweep(N_train_vec=[1200], train_len=1200, runner=vae_runner, **common)
    cma_calls = []
    c = sweep.run_awgn_cma_sweep(N_train=1200, runner=_runner(cma_calls), **common)
    assert len(cma_calls) == 2 and (c[0] >= 0).all()                                  # nothing taken from the VAE-LE files
    c2 = sweep.run_awgn_cma_sweep(N_train=1200, runner=_runner(cma_calls, offset=0.5), **common)
    v2 = sweep.run_awgn_sweep(N_train_vec=[1200], train_len=1200, runner=vae_runner, **common)
    assert len(cma_calls) == 2 and len(vae_calls) == 2
    assert torch.equal(c2[0], c[0]) and torch.equal(v2[0], v[0]) and (v[0] < 0).all()
    import os
    names = sorted(os.listdir(ck))
    assert sum(n.startswith("AWGNCMA_") for n in names) == 2 and sum(n.startswith("AWGN_") for n in names) == 2


def test_awgn_cma_sweep_rejects_bad_inputs_without_fallback():
    from vae_equalizer_b200 import sweep
    from vae_equalizer_b200._lib import VaeqError
    from vae_equalizer_b200.awgn_cma import CMA_runs, awgn_cma_eval_runs
    cells = [dict(SNR=14, nu=0.0, lr_optim=5e-4)]
    args = ("16-QAM", 2, 25, 15000, 1200)
    with pytest.raises(KeyError):
        sweep.sweep_cma_awgn(cells, *args, 20, 10, "h0")
    with pytest.raises(KeyError):
        sweep.run_awgn_cma_sweep(channel="h0", runner=_runner([]))
    with pytest.raises(ValueError):
        sweep.sweep_cma_awgn(cells, *args, 25, 10, "h1")
    with pytest.raises(ValueError):
        sweep.run_awgn_cma_sweep(num_epochs=25, epe=10, runner=_runner([]))
    with pytest.raises(VaeqError):
        sweep.sweep_cma_awgn(cells, *args, 20, 10, "h1", device="cpu")
    h = torch.zeros(1, 2, 25)
    with pytest.raises(VaeqError):
        CMA_runs(torch.zeros(1, 1, 2, 2400), torch.zeros(1, 2, 3000), h, torch.ones(1), 2)
    with pytest.raises(VaeqError):
        awgn_cma_eval_runs(torch.zeros(1, 2, 3000), torch.zeros(1, 2, 3000, dtype=torch.float16), torch.zeros(4))


def test_library_validates_the_batched_cma_arguments():
    """The C entry points reject bad sizes with VAEQ_EINVAL and a message before they touch a pointer or the device."""
    from vae_equalizer_b200 import _lib
    lib = _lib.load()
    p = ctypes.c_void_p(16)
    ok = dict(M=25, sps=2, Nt=2400, Nv=6000)

    def cma(M=25, sps=2, Nt=2400, Nv=6000):
        return lib.vaeq_cma_awgn_runs(p, Nt, 2 * Nt, 4 * Nt, 1, Nt, p, Nv, 2 * Nv, Nv, p, M, p, 1.0, sps, p, 3, None)
    for bad in (dict(M=24), dict(M=65), dict(M=0), dict(Nv=5999, sps=2), dict(Nt=2401)):
        assert cma(**dict(ok, **bad)) == -1, bad
        assert b"" != lib.vaeq_last_error()

    def ev(n_lev=4, N=3000, n_shift=21, edge=11):
        return lib.vaeq_awgn_cma_eval_runs(p, N, 2 * N, p, N, 2 * N, p, n_lev, N, n_shift, edge, 3, p, p, p, p, None)
    for bad in (dict(n_lev=3), dict(n_lev=16), dict(N=1009), dict(n_shift=65), dict(edge=9)):
        assert ev(**bad) == -1, bad
    assert b"n_lev" in (ev(n_lev=3) and lib.vaeq_last_error())
    assert b"1010" in (ev(N=1009) and lib.vaeq_last_error())
