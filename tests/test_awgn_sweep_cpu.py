"""Host logic of the batched AWGN sweep (sweep.run_awgn_sweep / sweep_vae_awgn): result layout, loop order, seeds and run-set grouping
through a stub runner, checkpoint reuse, and the inputs the engine rejects.  No GPU."""
import numpy as np
import pytest
import torch

LISTS = dict(N_train_vec=[200, 350], lr_optim_vec=[2e-3, 3e-3, 5e-3], M_vec=[9, 25], SNR_vec=[10, 14], nu_vec=[0.0, 0.05], iter=2,
             num_epochs=6, epe=2)


def _runner(calls, seen=None):
    def runner(cells, mod, sps, M, batch_len, N_valid, N_train, num_epochs, epe, channel):
        calls.append((M, batch_len, len(cells)))
        assert (N_valid, N_train, channel) == (15000, 1200, "h1")
        if seen is not None:
            seen.update({c["seed"]: dict(c, M=M, batch_len=batch_len) for c in cells})
        return torch.stack([torch.full((num_epochs // epe,), float(c["seed"] + 1000 * c["SNR"])) for c in cells])
    return runner


def test_run_awgn_sweep_layout_order_seeds_and_grouping():
    from vae_equalizer_b200 import sweep
    calls, seen = [], {}
    SER, epochs = sweep.run_awgn_sweep(mod="16-QAM", runner=_runner(calls, seen), **LISTS)
    assert SER.shape == (2, 3, 2, 2, 2, 2, 3) and list(epochs) == [0, 2, 4]
    assert sorted(calls) == [(9, 200, 24), (9, 350, 24), (25, 200, 24), (25, 350, 24)]      # one set per (M, batch_len): lr x SNR x nu x iter
    shape = SER.shape[:-1]
    assert sorted(seen) == list(range(int(np.prod(shape))))                                # every cell once, seeded by its flat index
    for idx in np.ndindex(*shape):
        b, l, m, s, n, i = idx
        seed = int(np.ravel_multi_index(idx, shape))
        c = seen[seed]
        assert (c["batch_len"], c["lr_optim"], c["M"], c["SNR"], c["nu"]) == (LISTS["N_train_vec"][b], LISTS["lr_optim_vec"][l], LISTS["M_vec"][m],
                                                                              LISTS["SNR_vec"][s], LISTS["nu_vec"][n]), idx
        assert (SER[idx] == seed + 1000 * c["SNR"]).all(), idx


def test_run_awgn_sweep_checkpoint_reuse_and_invalidation(tmp_path):
    from vae_equalizer_b200 import sweep
    calls = []
    ck = str(tmp_path / "ck")
    a = sweep.run_awgn_sweep(mod="16-QAM", runner=_runner(calls), checkpoint_dir=ck, **LISTS)
    n = len(calls)
    b = sweep.run_awgn_sweep(mod="16-QAM", runner=_runner(calls), checkpoint_dir=ck, **LISTS)
    assert len(calls) == n and torch.equal(a[0], b[0])
    c = sweep.run_awgn_sweep(mod="16-QAM", runner=_runner(calls), checkpoint_dir=ck, **dict(LISTS, SNR_vec=[11, 15]))
    assert len(calls) == 2 * n and not torch.equal(c[0], a[0])
    d = sweep.run_awgn_sweep(mod="64-QAM", runner=_runner(calls), checkpoint_dir=ck, **LISTS)      # other setting, same lists
    assert len(calls) == 3 * n and torch.equal(d[0], a[0])


def test_awgn_sweep_rejects_bad_inputs_without_fallback():
    from vae_equalizer_b200 import sweep
    from vae_equalizer_b200._lib import VaeqError
    from vae_equalizer_b200.awgn import AWGNEqualizerRuns, awgn_eval_runs, generate_frames_awgn_gpu
    cells = [dict(SNR=14, nu=0.0, lr_optim=2e-3)]
    args = ("16-QAM", 2, 25, 350, 15000, 1200)
    with pytest.raises(KeyError):
        sweep.sweep_vae_awgn(cells, *args, 20, 10, "h0")
    with pytest.raises(KeyError):
        sweep.run_awgn_sweep(channel="h0", runner=_runner([]))
    with pytest.raises(ValueError):
        sweep.sweep_vae_awgn(cells, *args, 25, 10, "h1")
    with pytest.raises(ValueError):
        sweep.run_awgn_sweep(num_epochs=25, epe=10, runner=_runner([]))
    with pytest.raises(VaeqError):
        sweep.sweep_vae_awgn(cells, *args, 20, 10, "h1", device="cpu")
    with pytest.raises(VaeqError):
        AWGNEqualizerRuns(1, 25, 2, [-1.0, 1.0], [[0.5, 0.5]], [1.0], [0.1], device="cpu")
    with pytest.raises(VaeqError):
        awgn_eval_runs(torch.zeros(1, 8, 100), torch.zeros(1, 2, 100, dtype=torch.float16), torch.zeros(4))
    with pytest.raises(VaeqError):
        generate_frames_awgn_gpu(100, [-1.0, 1.0], [10.0], [[0.5, 0.5]], np.ones(9, np.complex64), 2, "cpu", [0])
