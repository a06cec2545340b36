"""Event-timed cost of the data-aided LMMSE reference of the DP sweeps, and the table it exists for.  Writes profiles/r03_lmmse_sweep.txt, or the
path given as the first argument.

1. Per launch, 592 cells x 10^4 symbols at 64-QAM (device frames, h0, SNR 12..30 dB), M_est 25 and 63: the taps (k_lmmse_corr + k_lmmse_solve,
   shared_funcs.lmmse_taps_runs), the FIR (fir_runs), soft_dec_runs, the evaluation (frame_eval_runs, seg_len 0) and GMI (gmi_runs).  rx of the
   set is 190 MB, larger than the 126 MB L2.  WARM passes of warm-up, then PASSES timed passes; CUDA events; mean and min per pass.
2. End to end per frame, same call: sweep_lmmse_dp and sweep_vae_dp (VAE-LE, batch_len 100) of the same 592 cells and frames
   (datagen "gpu_batched", generation included, SNR 12..30 dB in 7 values), host clock around F frames ending in a device synchronise
   (set-up included).  The split of the taps launch pair into k_lmmse_corr and k_lmmse_solve comes from torch.profiler in a pass of its own.
3. run_dp_sweep with loss_type "VAE" and "LMMSE" on the same lists (so on the same frames): 64-QAM, nu 0.0270955, h0, SNR {17, 20, 23} x 5
   seeds, 40 frames, M_est 25, batch_len 100: VAE-LE's SER (soft demapper) and GMI over its last 10 frames next to LMMSE's over all 40.
4. -Xptxas -v of csrc/lmmse.cu, compiled in a temporary directory."""
import os
import re
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from time_sweep_gmi import card, timed  # noqa: E402
from vae_equalizer_b200 import shared_funcs as sfun  # noqa: E402
from vae_equalizer_b200 import sweep  # noqa: E402
from vae_equalizer_b200.datagen import generate_frames_gpu  # noqa: E402

R, N = 592, 10000


def frames(dev, M):
    k = sfun.init("h0", "64-QAM", dev, 0.0270955, 2, M, 20.0)
    P = torch.as_tensor(k[2], dtype=torch.float32).reshape(1, -1).repeat(R, 1).to(dev)
    snr = torch.tensor([12 + 18 * r / (R - 1) for r in range(R)], dtype=torch.float32, device=dev)
    theta = torch.full((R,), float(np.pi / 10), device=dev)
    rx, tx, _ = generate_frames_gpu(N, k[4], snr, P, 2, theta, dev, 1, h_channel=k[1])
    return rx.contiguous(), tx.contiguous(), k[3].to(dev), P, torch.full((R,), float(k[6]), device=dev)


def launches(dev, M):
    rx, tx, amp, P, nu = frames(dev, M)
    st = {}

    def taps():
        st["W"], st["v"], st["d"], st["ok"] = sfun.lmmse_taps_runs(rx, tx, M)

    def fir():
        st["z"] = sfun.fir_runs(rx, st["W"])

    def soft():
        st["q"] = sfun.soft_dec_runs(st["z"], st["v"], amp, nu)

    def ev():
        st["ser"], st["al"], st["c"] = sfun.frame_eval_runs(st["q"], st["z"], tx, amp, st["v"], nu, 0, return_counts=True)

    def gm():
        st["gmi"] = sfun.gmi_runs(st["q"], tx, P, st["al"], st["c"], 0)
    mean, mn = timed([taps, fir, soft, ev, gm])
    assert bool(st["ok"].all())
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(5):
            taps()
        torch.cuda.synchronize()
    split = {e.key: e.device_time_total / e.count / 1e3 for e in prof.key_averages() if "lmmse" in e.key}
    return mean, mn, st, split


def end_to_end(dev, F=10):
    cells = [dict(SNR=12 + 3 * (r % 7), nu=0.0270955, lr_optim=2.5e-3, theta=np.pi / 10, theta_diff=0.06 * np.pi, seed=r) for r in range(R)]
    args = ("64-QAM", 2, 25, 100, 10000, F)
    res = {}
    for _ in range(2):                                              # the first round warms up both engines
        for name, fn in (("LMMSE", sweep.sweep_lmmse_dp), ("VAE", sweep.sweep_vae_dp)):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn(cells, *args, device=dev, datagen="gpu_batched")
            torch.cuda.synchronize()
            res[name] = (time.perf_counter() - t0) / F * 1e3
    return res


def table(dev):
    kw = dict(mod="64-QAM", nu_vec=(0.0270955,), SNR_vec=(17, 20, 23), M_vec=(25,), batch_len_vec=(100,), lr_optim_vec=(2.5e-3,), iter=5,
              num_frames=40, N_lrhalf=40, N_frame_max=10000, device=dev, gmi=True)
    vae = sweep.run_dp_sweep(loss_type="VAE", **kw)
    lm = sweep.run_dp_sweep(loss_type="LMMSE", **kw)
    rows = []
    for s, snr in enumerate(kw["SNR_vec"]):
        v_ser = float(vae[0][2:, s, ..., -10:].double().mean())
        v_gmi = float(vae[3][:, s, ..., -10:].double().mean())
        l_ser = float(lm[0][2:, s].double().mean())
        l_gmi = float(lm[3][:, s].double().mean())
        rows.append(f"  {snr:3d} dB   VAE-LE SER {v_ser:.3e}  GMI {v_gmi:.4f}   |   LMMSE SER {l_ser:.3e}  GMI {l_gmi:.4f}   |   GMI gap {l_gmi - v_gmi:+.4f}")
    return rows


def ptxas_lines():
    src = os.path.join(ROOT, "vae_equalizer_b200", "csrc", "lmmse.cu")
    lines = []
    with tempfile.TemporaryDirectory() as tmp:
        try:
            r = subprocess.run(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas", "-v", "-c", "-o",
                                os.path.join(tmp, "lmmse.o"), src], capture_output=True, text=True, timeout=900)
        except Exception as e:                                      # noqa: BLE001
            return [f"nvcc unavailable ({e})"]
        for ln in r.stderr.splitlines():
            m = re.search(r"Compiling entry function '(\S+)'", ln)
            if m:
                lines.append(m.group(1))
            elif "Used" in ln or "spill" in ln:
                lines.append("    " + ln.split(":", 1)[-1].strip())
    return lines


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r03_lmmse_sweep.txt")
    dev = torch.device("cuda")
    torch.cuda.init()
    lines = [f"card: {card()}", f"torch {torch.__version__}, CUDA {torch.version.cuda}", "",
             f"1. per launch, {R} cells x {N} symbols, 64-QAM, h0; CUDA events, mean / min over the timed passes (ms)"]
    for M in (25, 63):
        mean, mn, st, split = launches(dev, M)
        lines.append(f"  M_est {M}")
        for name, a, b in zip(("taps (corr + solve)", "FIR", "soft_dec_runs", "frame_eval_runs", "gmi_runs"), mean, mn):
            lines.append(f"    {name:22s} {a:8.3f} / {b:8.3f}")
        lines.append(f"    sum                    {float(mean.sum()):8.3f}")
        for k, v in sorted(split.items()):
            lines.append(f"    of the taps: {k.split('(')[0]:22s} {v:8.3f} (torch.profiler)")
        print("\n".join(lines), flush=True)
        del st
        torch.cuda.empty_cache()
    e2e = end_to_end(dev)
    lines += ["", f"2. end to end per frame, {R} cells, 64-QAM, M_est 25, batch_len 100, datagen gpu_batched (generation included), host clock",
              f"  sweep_lmmse_dp {e2e['LMMSE']:8.3f} ms / frame", f"  sweep_vae_dp   {e2e['VAE']:8.3f} ms / frame"]
    print("\n".join(lines[-3:]), flush=True)
    lines += ["", "3. 64-QAM, nu 0.0270955, h0, 5 seeds per SNR, 40 frames, M_est 25, batch_len 100, same frames for both (run_dp_sweep);",
              "   SER of the soft demapper (mean of x, y) and GMI (bit / 2D symbol): VAE-LE over its last 10 frames, LMMSE over all 40"]
    lines += table(dev)
    lines += ["", "4. ptxas (nvcc -gencode arch=compute_100a,code=sm_100a -O3 -Xptxas -v) of csrc/lmmse.cu"]
    lines += ptxas_lines()
    text = "\n".join(lines) + "\n"
    print(text)
    os.makedirs(os.path.dirname(out) or ".", exist_ok=True)
    with open(out, "w") as fh:
        fh.write(text)


if __name__ == "__main__":
    main()
