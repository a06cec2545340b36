"""Time the batched DP frame kernel above 1000 symbols (one thread-block cluster per run, csrc/dp_cluster.cu) on one GPU.

For VAE-LE at batch_len 2000 and 4096 (frames of 100 non-overlapping minibatches) and VAE-flex with a 2000-symbol window advanced by
100 symbols (100 steps), R = 1, 148 and 592 runs per launch: ms per frame (device events, after a warm-up frame) and trained symbols/s
(R x steps x batch_len / time).  In the same process, the single-run driver on one such cell (DPEqualizer.train_frame: one set of
launches per step at this size): R times that is what a sweep paid per frame before the cluster kernel.  Every run of a launch gets
the same frame (the timing does not depend on the data).  The card's name and power limit are read in the same call.

    python tools/time_frames_cluster.py [--frames 3] [--out file]
"""
import argparse
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))

from oracle import vaeq_oracle as O  # noqa: E402
from vae_equalizer_b200.datagen import generate_frames_gpu  # noqa: E402
from vae_equalizer_b200.dp import DPEqualizer, DPEqualizerRuns  # noqa: E402

M, STEPS = 25, 100
CASES = [("VAE-LE", 2000, 2000), ("VAE-LE", 4096, 4096), ("VAE-flex", 2000, 100)]     # name, batch_len, stride (flex_step)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[torch.cuda.current_device()] if q.returncode == 0 else "nvidia-smi unavailable"


def frame_geometry(B, stride):
    keep_lo, keep_n, kd = (0, B, True) if stride == B else ((B - stride) // 2, stride, False)
    n_sym = (STEPS - 1) * stride + B
    n_keep = (STEPS - 1) * stride + keep_n + (keep_lo if kd else 0)
    return keep_lo, keep_n, kd, n_sym, n_keep


def timed(fn, frames):
    fn()                                                    # warm-up: module load, shared-memory attributes
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(frames):
        fn()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / frames


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("needs a CUDA device")
    dev = torch.device("cuda:0")
    h_est, h_ch, P, amp, amps, pol, nu_sc, var, pow_mean = O.init("h0", "64-QAM", "cpu", 0.0270955, 2, M, 23)
    lines = [f"card (name, power limit, max SM clock): {card()}",
             f"64-QAM, M_est {M}, {STEPS} training steps per frame, {a.frames} timed frames after one warm-up, device events"]
    for name, B, stride in CASES:
        keep_lo, keep_n, kd, n_sym, n_keep = frame_geometry(B, stride)
        rx1, _, _ = generate_frames_gpu(n_sym, amps, [23.0], np.asarray(P, dtype=np.float32)[None], 2, [0.3], dev, 7)
        for R in (1, 148, 592):
            eqr = DPEqualizerRuns(R, M, 2, amp, torch.tensor(P, dtype=torch.float32), var, nu_sc, device=dev)
            rx = rx1.expand(R, -1, -1, -1).contiguous()
            ot = torch.empty(R, 2, 16, n_keep, device=dev)
            oc = torch.empty(R, 2, 2, n_keep, device=dev)
            ms = timed(lambda: eqr.train_frame(rx, B, stride, STEPS, 1e-3, 1e-3, ot, oc, keep_lo, keep_n, keep_lo_in_dst=kd), a.frames)
            lines.append(f"{name:8s} batch_len {B:5d} step {stride:5d}  R {R:4d}: {ms:9.3f} ms per frame  "
                         f"{R * STEPS * B / ms * 1e3:.3e} trained symbols/s")
            del eqr, rx, ot, oc
            torch.cuda.empty_cache()
    # the single-run driver's per-step path on one cell
    B, stride = 2000, 2000
    keep_lo, keep_n, kd, n_sym, n_keep = frame_geometry(B, stride)
    rx1, _, _ = generate_frames_gpu(n_sym, amps, [23.0], np.asarray(P, dtype=np.float32)[None], 2, [0.3], dev, 7)
    eq = DPEqualizer(M, 2, amp, torch.tensor(P, dtype=torch.float32), var, nu_sc, device=dev)
    ot = torch.empty(2, 16, n_keep, device=dev)
    oc = torch.empty(2, 2, n_keep, device=dev)
    ms = timed(lambda: eq.train_frame(rx1[0], B, stride, STEPS, 1e-3, 1e-3, ot, oc, keep_lo, keep_n, keep_lo_in_dst=kd), a.frames)
    lines.append(f"single-run driver (DPEqualizer.train_frame, per-step launches) VAE-LE batch_len {B}: {ms:9.3f} ms per frame  "
                 f"{STEPS * B / ms * 1e3:.3e} trained symbols/s; x148 = {148 * ms:.1f} ms, x592 = {592 * ms:.1f} ms")
    text = "\n".join(lines)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
