"""CPU-only checks: the C-ABI library loads and exports every symbol include/vaeq.h declares (no compute
without a GPU), host-side constants/data generation match the oracle, and the product path fails loudly
on CPU tensors instead of falling back."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from oracle import vaeq_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    src = open(os.path.join(ROOT, "include", "vaeq.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(vaeq_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from vae_equalizer_b200 import _lib
    assert os.path.exists(_lib.LIB_PATH), "build libvaeq.so first (python -c 'import __graft_entry__ as g; g.build()')"
    lib = ctypes.CDLL(_lib.LIB_PATH)
    names = header_symbols()
    assert len(names) >= 24
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/vaeq.h but not exported"
    assert sorted(_lib.PROTOTYPES) == names, "ctypes prototypes out of sync with the header"
    bound = _lib.load()
    assert bound.vaeq_abi_version() == 1
    assert bound.vaeq_dp_workspace_bytes(100, 25, 8) > 0 and bound.vaeq_adam_state_floats(25) == 48 * 25 + 4


def test_tc_taps_switch_rejects_values_other_than_0_and_1():
    """vaeq_dp_tc_taps selects the tap-gradient kernels (1 = tcgen05, 0 = CUDA cores); any other value is an error, never a
    third mode, and the call only sets a flag, so it runs without a GPU."""
    from vae_equalizer_b200 import _lib
    lib = _lib.load()
    try:
        for bad in (2, 3, 4, 6, -1):
            assert lib.vaeq_dp_tc_taps(bad) == -1                    # VAEQ_EINVAL
            assert b"vaeq_dp_tc_taps" in lib.vaeq_last_error()
        assert lib.vaeq_dp_tc_taps(0) == 0 and lib.vaeq_dp_tc_taps(1) == 0
    finally:
        lib.vaeq_dp_tc_taps(1)


def test_struct_layout_matches_header_field_order():
    from vae_equalizer_b200 import _lib
    src = open(os.path.join(ROOT, "include", "vaeq.h")).read()
    body = re.search(r"typedef struct vaeq_dp_desc \{(.*?)\} vaeq_dp_desc;", src, flags=re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields = []
    for decl in body.split(";"):
        decl = decl.strip()
        if not decl:
            continue
        for part in decl.split(","):
            fields.append(re.sub(r"[\*\s]", " ", part).split()[-1])
    assert fields == [f[0] for f in _lib.DpDesc._fields_]


def test_no_cpu_fallback():
    from vae_equalizer_b200 import VaeqError
    import vae_equalizer_b200.shared_funcs as sfun
    with pytest.raises(VaeqError):
        sfun.soft_dec(torch.zeros(2, 2, 8), torch.ones(2), torch.zeros(4), 0.0)
    with pytest.raises(VaeqError):
        sfun.CPE(torch.zeros(2, 2, 64))
    with pytest.raises(VaeqError):
        sfun.SER_IQflip(torch.zeros(2, 8, 16), torch.zeros(2, 2, 16, dtype=torch.float16))
    if not torch.cuda.is_available():
        from vae_equalizer_b200.dp import DPEqualizer
        with pytest.raises((VaeqError, RuntimeError, AssertionError)):
            DPEqualizer(9, 2, [-1., 1.], [.5, .5], [.1, .1], 0.0, device="cpu")


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "vae_equalizer_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh")):
                txt = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in txt and "from oracle" not in txt, f


@pytest.mark.parametrize("mod,nu,M,snr", [("64-QAM", 0.0270955, 25, 23), ("16-QAM", 0.0, 9, 18), ("4-QAM", 0.1, 5, 12)])
def test_init_matches_oracle(mod, nu, M, snr):
    from vae_equalizer_b200.constants import init
    a, b = init("h1", mod, "cpu", nu, 2, M, snr), O.init("h1", mod, "cpu", nu, 2, M, snr)
    for x, y in zip(a, b):
        x = x.detach().numpy() if torch.is_tensor(x) else np.asarray(x)
        y = y.detach().numpy() if torch.is_tensor(y) else np.asarray(y)
        np.testing.assert_allclose(x, y, rtol=1e-12, atol=0)
    with pytest.raises(KeyError):
        init("h9", mod, "cpu", nu, 2, M, snr)


def test_awgn_constants_match_oracle():
    from vae_equalizer_b200.constants import awgn_constants
    for mod, nu in (("16-QAM", 0.0), ("64-QAM", 0.0872449)):
        for x, y in zip(awgn_constants(mod, nu, 20), O.awgn_constants(mod, nu, 20)):
            np.testing.assert_allclose(np.asarray(x), np.asarray(y), rtol=1e-12)


def test_data_generator_matches_oracle_with_same_rng():
    from vae_equalizer_b200.datagen import generate_data_shaping
    h_est, h_ch, P, amp, amps, pol, nu_sc, var, pow_mean = O.init("h1", "16-QAM", "cpu", 0.0, 2, 9, 18)
    args = (500, amps, 18, h_ch, P, 2, 90e9, 2, -26e-24, 0.1e-12 * np.sqrt(1000), np.array([0.0314, 0.0314], dtype=np.complex64), 0.3, "cpu")
    rx1, tx1, s1 = generate_data_shaping(*args, rng=np.random.default_rng(5))
    rx2, tx2, s2 = O.generate_data_shaping(*args, rng=np.random.default_rng(5))
    assert rx1.shape == (2, 2, 1000) and tx1.shape == (2, 2, 500) and tx1.dtype == torch.float16
    np.testing.assert_allclose(rx1.numpy(), rx2.numpy(), atol=1e-6)
    assert torch.equal(tx1, tx2) and abs(s1 - s2) < 1e-9
    # signal power ~ 1/sps, noise level as requested
    assert abs(float((rx1 ** 2).sum(1).mean()) - 0.5 * (1 + 10 ** -1.8)) < 0.05


def test_batched_frame_generator_matches_single_generator():
    """datagen.generate_frames_gpu (all sweep cells in one batched call) against generate_data_gpu: R = 1 with the same seed draws
    the same symbols and the same noise-free signal; per-run SNR and rotation are honoured."""
    import numpy as np
    import torch
    from vae_equalizer_b200.constants import init
    from vae_equalizer_b200.datagen import generate_data_gpu, generate_frames_gpu
    h_est, h_ch, P, amp, amps, pol, nu_sc, var, pm = init("h0", "64-QAM", "cpu", 0.0270955, 2, 25, 23)
    a, ta, _ = generate_data_gpu(1500, amps, 200, P, 2, 0.3, "cpu", 7)
    b, tb, _ = generate_frames_gpu(1500, amps, [200], P, 2, [0.3], "cpu", 7)
    assert torch.equal(ta, tb[0]) and float((a - b[0]).abs().max()) < 5e-6
    # the drawn symbols follow the PCS pmf (sf:75-76) and the noise-free signal has the constellation's unit power (rotation, CD and
    # PMD are all-pass, the RRC pulse has unit energy)
    _, tbig, _ = generate_frames_gpu(40000, amps, [200], P, 2, [0.3], "cpu", 3)
    lv = torch.tensor(amps, dtype=torch.float32)
    cnt = torch.stack([(tbig.float().reshape(-1) - a_).abs().lt(1e-2).float().mean() for a_ in lv])
    assert float((cnt - torch.tensor(P, dtype=torch.float32)).abs().max()) < 6e-3
    assert abs(float((a ** 2).sum(dim=(0, 1)).mean()) - pm) < 0.05 * pm
    rx, tx, sig = generate_frames_gpu(3000, amps, [23, 13, 23], np.stack([P, P, P]), 2, [0.3, 0.3, 1.0], "cpu", 11)
    assert rx.shape == (3, 2, 2, 6000) and tx.shape == (3, 2, 2, 3000) and tx.dtype == torch.float16
    assert abs(float(sig[1] / sig[0]) - 10 ** 0.5) < 0.05 * 10 ** 0.5          # 10 dB lower SNR -> sqrt(10) more noise
    p0, p2 = float((rx[0] ** 2).mean()), float((rx[2] ** 2).mean())
    assert abs(p0 - p2) / p0 < 0.05                                            # a rotation keeps the power


def test_run_dp_sweep_layout_and_mat_schema(tmp_path):
    """sweep.run_dp_sweep reproduces the index order of Eval_run_DP.py:52,86 and save_mat the .mat schema of :99-114 (stub runner:
    no GPU); cells that share (M, batch_len, flex_step, symb_rate) arrive at the runner as ONE batched set."""
    import numpy as np
    import torch
    from scipy import io
    from vae_equalizer_b200 import sweep
    calls = []

    def runner(cells, mod, sps, M, batch_len, N_frame_max, num_frames, **kw):
        calls.append((M, batch_len, len(cells)))
        ser = torch.stack([torch.full((4, num_frames), 1000.0 * c["SNR"] + 10 * c["lr_optim"] * 1e3 + M + c["seed"] * 1e-3) for c in cells])
        ve = torch.stack([torch.full((2, num_frames), float(c["nu"])) for c in cells])
        var = torch.stack([torch.full((2,), float(c["theta"])) for c in cells])
        return ser, ve, var

    lists = dict(nu_vec=[0, 0.027], symb_rate_vec=[90e9], theta_vec=[0.3], theta_diff_vec=[0.0, 0.1], SNR_vec=[20, 23, 26], M_vec=[9, 25],
                 batch_len_vec=[100], flex_step_vec=[10], lr_optim_vec=[2e-3, 3e-3])
    SER, Var_est, var_real = sweep.run_dp_sweep(iter=2, num_frames=3, runner=runner, **lists)
    assert SER.shape == (4, 3, 1, 2, 2, 2, 2, 1, 1, 1, 2, 3) and Var_est.shape == (2,) + SER.shape[1:] and var_real.shape == (2,) + SER.shape[1:-1] + (1,)
    assert sorted(calls) == [(9, 100, 48), (25, 100, 48)]                         # two batched sets, 3*2*2*2*2 cells each
    # SER[:, s, sr, n, t1, m, l, nt, ss, v, i, :]
    v = float(SER[0, 2, 0, 1, 1, 1, 0, 0, 0, 0, 1, 0])
    assert abs(v - (1000.0 * 26 + 10 * 2.0 + 25)) < 1.0
    assert float(Var_est[1, 0, 0, 1, 0, 0, 0, 0, 0, 0, 0, 2]) == np.float32(0.027) and float(var_real[0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0]) == np.float32(0.3)
    # resume: a second call with the same checkpoint directory recomputes nothing and returns the same arrays
    ck = str(tmp_path / "ck")
    a = sweep.run_dp_sweep(iter=2, num_frames=3, runner=runner, checkpoint_dir=ck, **lists)
    n_calls = len(calls)
    b = sweep.run_dp_sweep(iter=2, num_frames=3, runner=runner, checkpoint_dir=ck, **lists)
    assert len(calls) == n_calls and all(torch.equal(x, y) for x, y in zip(a, b)) and torch.equal(a[0], SER)
    # a sweep with a different SNR list of the same length must NOT pick up the stale files (the signature differs): it recomputes
    lists2 = dict(lists, SNR_vec=[10, 13, 16])
    c = sweep.run_dp_sweep(iter=2, num_frames=3, runner=runner, checkpoint_dir=ck, **lists2)
    assert len(calls) == n_calls + 2 and not torch.equal(c[0], a[0])
    assert abs(float(c[0][0, 2, 0, 1, 1, 1, 0, 0, 0, 0, 1, 0]) - (1000.0 * 16 + 10 * 2.0 + 25)) < 1.0
    c2 = sweep.run_dp_sweep(iter=2, num_frames=3, runner=runner, checkpoint_dir=ck, N_lrhalf=50, **lists2)     # other setting, same lists
    assert len(calls) == n_calls + 4 and torch.equal(c2[0], c[0])
    path = str(tmp_path / "sweep.mat")
    sweep.save_mat(path, SER, Var_est, var_real, SNR_vec=lists["SNR_vec"], nu_vec=lists["nu_vec"], theta_diff_vec=lists["theta_diff_vec"],
                   theta_vec=lists["theta_vec"], M_vec=lists["M_vec"], lr_optim_vec=lists["lr_optim_vec"], batch_len_vec=lists["batch_len_vec"],
                   symb_rate_vec=lists["symb_rate_vec"], flex_step_vec=lists["flex_step_vec"])
    d = io.loadmat(path)["dict"]
    assert set(d.dtype.names) == {"SER", "Var_est", "var_real", "SNR", "nu", "theta_diff", "theta", "M", "lr", "batch_len", "symb_rate", "symb_step"}
    assert d["SER"][0, 0].shape == SER.shape and list(d["SNR"][0, 0].ravel()) == [20, 23, 26]
