"""Frame time of the persistent small-minibatch kernel: one VAE-LE frame of 10 000 symbols at batch_len = 100 (100 sequential
steps, RUN_DP:38-40) for R batched runs, against the launch-by-launch path."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from vae_equalizer_b200 import _lib
from vae_equalizer_b200.constants import init
from vae_equalizer_b200.datagen import generate_data_gpu
from vae_equalizer_b200.dp import DPEqualizer, DPEqualizerRuns

dev = torch.device("cuda", 0)
lib = _lib.load()
M, B, n_steps, lr = 25, int(os.environ.get("B", 100)), int(os.environ.get("STEPS", 100)), 2.5e-3
h_est, h_channel, P, amp, amps, pol, nu_sc, var, pow_mean = init("h0", "64-QAM", "cpu", 0.0270955, 2, M, 23)
N = n_steps * B


def timeit(fn, reps=5):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


rx = generate_data_gpu(N, amps, 23, P, 2, np.pi / 10, dev, 1)[0]
eq = DPEqualizer(M, 2, amp, P, var, nu_sc, device=dev)
ot = torch.empty(2, 16, N, device=dev)
oc = torch.empty(2, 2, N, device=dev)
for persistent in (0, 2, 1):
    _lib.check(lib.vaeq_dp_persistent_frames(persistent))
    ms = timeit(lambda: eq.train_frame(rx, B, B, n_steps, lr, lr, ot, oc, 0, B, keep_lo_in_dst=True))
    print(f"1 run, persistent mode {persistent}: {ms:.3f} ms per frame of {n_steps} steps x {B} symbols = {ms * 1e3 / n_steps:.2f} us/step, {N / ms / 1e3:.3f} M symbols/s")
_lib.check(lib.vaeq_dp_persistent_frames(1))
_lib.check(lib.vaeq_dp_frame_runs_per_sm(int(os.environ.get('PER_SM', 0))))       # 0 = automatic, 3 / 4 = force the kernel variant
for R in [int(v) for v in os.environ.get('RUNS', '1,37,148,296,592,888,1184,2368').split(',')]:
    rxs = torch.stack([generate_data_gpu(N, amps, 23, P, 2, np.pi / 10 + 0.01 * r, dev, 10 + r)[0] for r in range(R)])
    eqr = DPEqualizerRuns(R, M, 2, amp, P, var, nu_sc, device=dev)
    otr = torch.empty(R, 2, 16, N, device=dev)
    ocr = torch.empty(R, 2, 2, N, device=dev)
    ms = timeit(lambda: eqr.train_frame(rxs, B, B, n_steps, lr, lr, otr, ocr, 0, B, keep_lo_in_dst=True), reps=3)
    print(f"{R:5d} runs in one launch: {ms:.3f} ms per frame -> {ms * 1e3 / n_steps:.2f} us/step, aggregate {R * N / ms / 1e3:.2f} M symbols/s; final loss run0 {float(eqr.loss[0]):.2f}")
    del rxs, eqr, otr, ocr
