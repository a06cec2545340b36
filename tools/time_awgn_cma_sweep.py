"""Event-timed phases of the batched AWGN CMA sweep engine (sweep.sweep_cma_awgn) per validation period, against the single-run driver
processing_cma_awgn measured in the same process.  Writes profiles/r03_awgn_cma_sweep.txt, or the path given as the first argument.

Workload: 16-QAM and 64-QAM, M_est 25, N_train 1200, N_valid 15000, epe 20, channel h1, R in {1, 148, 592, 2368}.
One validation period = generation of epe training frames and one validation frame for every cell (vaeq_gen_awgn), ONE launch running
every cell's CMA over its epe training frames and then over its validation frame (vaeq_cma_awgn_runs), the batched CPE (vaeq_cpe_awgn)
and the scoring (vaeq_awgn_cma_eval_runs).  One period is warm-up, the next PERIODS are timed.  The compile report of the kernels
(ptxas -v, compiled into a temporary directory) is appended."""
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from vae_equalizer_b200 import awgn_cma as cm  # noqa: E402
from vae_equalizer_b200 import processing as pr  # noqa: E402
from vae_equalizer_b200.awgn import generate_frames_awgn_gpu  # noqa: E402
from vae_equalizer_b200.constants import awgn_constants, upsampled_channel  # noqa: E402

M_EST, N_TRAIN, N_VALID, EPE, CHANNEL, LR = 25, 1200, 15000, 20, "h1", 5e-4
RS, MODS, PERIODS = (1, 148, 592, 2368), ("16-QAM", "64-QAM"), 3


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:                                       # noqa: BLE001
        return f"nvidia-smi unavailable ({e})"


def compile_report():
    """ptxas registers / spills of the kernels of csrc/awgn_cma.cu, built for sm_100a into a temporary directory."""
    src = os.path.join(ROOT, "vae_equalizer_b200", "csrc", "awgn_cma.cu")
    with tempfile.TemporaryDirectory() as tmp:
        r = subprocess.run(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas", "-v", "-c", "-o",
                            os.path.join(tmp, "a.o"), src], capture_output=True, text=True)
    out, name = [], None
    for line in (r.stdout + r.stderr).splitlines():
        if "Compiling entry function" in line:
            name = line.split("'")[1]
        elif name and ("Used" in line or "spill" in line):
            out.append(f"  {name}: {line.split(':', 1)[-1].strip()}")
    return out or [f"  nvcc failed: {r.stderr.strip()[:300]}"]


def driver_ms_per_epoch():
    """processing_cma_awgn, 16-QAM, SNR 12, M_est 25, lr 5e-4, N_valid 15000, N_train 1200, 60 epochs, epe 20, h1 (host data generation
    included, as the driver runs)."""
    args = ("16-QAM", 2, 12, 0.0, M_EST, LR, N_VALID, N_TRAIN, 60, EPE, CHANNEL)
    pr.processing_cma_awgn(*args[:8], 4, 2, CHANNEL, rng=np.random.default_rng(0), verbose=False)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    pr.processing_cma_awgn(*args, rng=np.random.default_rng(1), verbose=False)
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / 60 * 1e3


def time_set(mod, R):
    dev = torch.device("cuda")
    h_ch = upsampled_channel(CHANNEL, 2)
    snr = [10.0 + (r % 8) for r in range(R)]
    consts = [awgn_constants(mod, 0.02 * (r % 3), snr[r]) for r in range(R)]
    amps = consts[0][0]
    P = np.stack([c[1] for c in consts])
    lr = torch.full((R,), LR, device=dev)
    amp = torch.tensor(amps, dtype=torch.float32, device=dev)
    h = torch.zeros(R, 2, M_EST, device=dev)
    h[:, 0, M_EST // 2] = 1.0
    seeds = list(range(R))
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
    acc = np.zeros(4)
    for k in range(PERIODS + 1):
        ev[0].record()
        rx, _ = generate_frames_awgn_gpu(N_TRAIN, amps, snr, P, h_ch, 2, dev, seeds, frame0=k * EPE, n_frames=EPE)
        rx_v, tx_v = generate_frames_awgn_gpu(N_VALID, amps, snr, P, h_ch, 2, dev, seeds, frame0=(1 << 20) + k)
        ev[1].record()
        out_v = cm.CMA_runs(rx, rx_v[:, 0], h, lr, 2)
        ev[2].record()
        y = cm.CPE(out_v)
        ev[3].record()
        _, _, ser = cm.awgn_cma_eval_runs(y, tx_v[:, 0], amp)
        ev[4].record()
        torch.cuda.synchronize()
        if k:
            acc += [ev[i].elapsed_time(ev[i + 1]) for i in range(4)]
        del rx, rx_v, tx_v, out_v, y
    assert torch.isfinite(ser).all()
    return acc / PERIODS / EPE                                    # ms per epoch of the whole set, per phase


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r03_awgn_cma_sweep.txt")
    torch.cuda.init()
    lines = [f"card: {card()}", f"torch {torch.__version__}, CUDA {torch.version.cuda}, {torch.cuda.get_device_properties(0).multi_processor_count} SMs", ""]
    drv = driver_ms_per_epoch()
    lines.append(f"single-run driver processing_cma_awgn (16-QAM, SNR 12, lr {LR}, N_train {N_TRAIN}, N_valid {N_VALID}, epe {EPE}, host data): "
                 f"{drv:.3f} ms per epoch (one cell)")
    lines.append("")
    lines.append(f"batched set, M_est {M_EST}, N_train {N_TRAIN}, N_valid {N_VALID}, epe {EPE}, {CHANNEL}, one 32-thread CTA (one warp) per cell;")
    lines.append("ms per epoch of the WHOLE set (validation work divided over the epe epochs of its period), CUDA events, mean of "
                 f"{PERIODS} periods after one warm-up period")
    lines.append(f"{'mod':7s} {'R':>5s} {'gen':>8s} {'cma':>8s} {'cpe':>8s} {'score':>8s} {'total':>8s} {'ms/cell-ep':>10s} {'Msym/s':>8s} "
                 f"{'Msym/s/cell':>11s} {'speed-up':>8s}")
    for mod in MODS:
        for R in RS:
            g, c, p, s = time_set(mod, R)
            tot = g + c + p + s
            sym = R * (N_TRAIN + N_VALID / EPE) / (c * 1e-3) / 1e6     # CMA symbols (training + validation pass) per second of the CMA launch
            lines.append(f"{mod:7s} {R:5d} {g:8.3f} {c:8.3f} {p:8.3f} {s:8.3f} {tot:8.3f} {tot / R:10.4f} {sym:8.2f} {sym / R:11.3f} "
                         f"{drv / (tot / R):8.1f}")
            print(lines[-1], flush=True)
            torch.cuda.empty_cache()
    lines.append("")
    lines.append("gen = vaeq_gen_awgn (epe training frames + 1 validation frame per cell), cma = vaeq_cma_awgn_runs (one launch: epe training "
                 "frames and the validation pass), cpe = vaeq_cpe_awgn, score = vaeq_awgn_cma_eval_runs; Msym/s = symbols through the CMA "
                 "recurrence per second of the cma phase (Msym/s/cell: per warp); speed-up = driver ms per epoch / set ms per cell-epoch "
                 "(the driver row is 16-QAM).")
    lines.append("")
    lines.append("compile report (ptxas -v, sm_100a):")
    lines += compile_report()
    text = "\n".join(lines) + "\n"
    print(text)
    os.makedirs(os.path.dirname(out) or ".", exist_ok=True)
    with open(out, "w") as fh:
        fh.write(text)


if __name__ == "__main__":
    main()
