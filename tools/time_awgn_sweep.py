"""Event-timed phases of the batched AWGN VAE-LE sweep engine (sweep.sweep_vae_awgn) per validation period, against the single-run driver
(processing_vaele_awgn at the setting of tools/time_awgn.py) measured in the same process.  Writes profiles/r03_awgn_sweep.txt, or the
path given as the first argument.

Workload: 16-QAM and 64-QAM, M_est 25, batch_len 350, N_train 1200, N_valid 15000, epe 20, channel h1, R in {1, 148, 592, 1184}.
One validation period = generation of epe training frames and one validation frame for every cell (vaeq_gen_awgn), ONE launch training
epe epochs of every cell (vaeq_awgn_train_frames_runs), the validation forward (vaeq_awgn_forward_runs) and the scoring
(vaeq_awgn_eval_runs).  One period is warm-up, the next PERIODS are timed."""
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from vae_equalizer_b200 import processing as pr  # noqa: E402
from vae_equalizer_b200.awgn import AWGNEqualizerRuns, awgn_eval_runs, generate_frames_awgn_gpu  # noqa: E402
from vae_equalizer_b200.constants import awgn_constants, upsampled_channel  # noqa: E402

M_EST, BATCH, N_TRAIN, N_VALID, EPE, CHANNEL = 25, 350, 1200, 15000, 20, "h1"
RS, MODS, PERIODS = (1, 148, 592, 1184), ("16-QAM", "64-QAM"), 3


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:                                       # noqa: BLE001
        return f"nvidia-smi unavailable ({e})"


def driver_ms_per_epoch():
    """tools/time_awgn.py: 16-QAM, SNR 12, M_est 25, lr 2e-3, batch_len 350, N_valid 15000, N_train 1200, 60 epochs, epe 20, h1."""
    args = ("16-QAM", 2, 12, 0.0, 25, 2e-3, 350, 15000, 1200, 60, 20, "h1")
    pr.processing_vaele_awgn(*args[:9], 4, 2, args[11], rng=np.random.default_rng(0), verbose=False)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    pr.processing_vaele_awgn(*args, rng=np.random.default_rng(1), verbose=False)
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / 60 * 1e3


def time_set(mod, R):
    dev = torch.device("cuda")
    h = upsampled_channel(CHANNEL, 2)
    snr = [10.0 + (r % 8) for r in range(R)]
    consts = [awgn_constants(mod, 0.02 * (r % 3), snr[r]) for r in range(R)]
    amps = consts[0][0]
    P = np.stack([c[1] for c in consts])
    eqr = AWGNEqualizerRuns(R, M_EST, 2, amps, P, [c[2] for c in consts], [c[3] for c in consts], device=dev)
    lr = torch.full((R,), 2e-3, device=dev)
    amp = torch.tensor(amps, dtype=torch.float32, device=dev)
    seeds = list(range(R))
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
    acc = np.zeros(4)
    for k in range(PERIODS + 1):
        ev[0].record()
        rx, _ = generate_frames_awgn_gpu(N_TRAIN, amps, snr, P, h, 2, dev, seeds, frame0=k * EPE, n_frames=EPE)
        rx_v, tx_v = generate_frames_awgn_gpu(N_VALID, amps, snr, P, h, 2, dev, seeds, frame0=(1 << 20) + k)
        ev[1].record()
        eqr.train_frames(rx, lr, BATCH, N_TRAIN)
        ev[2].record()
        q, _, _ = eqr.forward(rx_v[:, 0])
        ev[3].record()
        _, _, ser = awgn_eval_runs(q, tx_v[:, 0], amp)
        ev[4].record()
        torch.cuda.synchronize()
        if k:
            acc += [ev[i].elapsed_time(ev[i + 1]) for i in range(4)]
        del rx, rx_v, tx_v, q
    assert torch.isfinite(ser).all()
    return acc / PERIODS / EPE                                    # ms per epoch of the whole set, per phase


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r03_awgn_sweep.txt")
    torch.cuda.init()
    lines = [f"card: {card()}", f"torch {torch.__version__}, CUDA {torch.version.cuda}", ""]
    drv = driver_ms_per_epoch()
    lines.append(f"single-run driver processing_vaele_awgn (tools/time_awgn.py setting): {drv:.3f} ms per epoch (one cell)")
    lines.append("")
    lines.append(f"batched set, M_est {M_EST}, batch_len {BATCH}, N_train {N_TRAIN} ({N_TRAIN // BATCH} steps/epoch), N_valid {N_VALID}, epe {EPE}, {CHANNEL};")
    lines.append("ms per epoch of the WHOLE set (validation work divided over the epe epochs of its period), CUDA events, mean of "
                 f"{PERIODS} periods after one warm-up period")
    lines.append(f"{'mod':7s} {'R':>5s} {'gen':>8s} {'train':>8s} {'fwd':>8s} {'score':>8s} {'total':>8s} {'ms/cell-ep':>10s} {'Msym/s':>8s} {'speed-up':>8s}")
    for mod in MODS:
        for R in RS:
            g, t, f, s = time_set(mod, R)
            tot = g + t + f + s
            sym = R * (N_TRAIN // BATCH) * BATCH / (tot * 1e-3) / 1e6
            lines.append(f"{mod:7s} {R:5d} {g:8.3f} {t:8.3f} {f:8.3f} {s:8.3f} {tot:8.3f} {tot / R:10.4f} {sym:8.2f} {drv / (tot / R):8.1f}")
            print(lines[-1], flush=True)
            torch.cuda.empty_cache()
    lines.append("")
    lines.append("gen = vaeq_gen_awgn (epe training frames + 1 validation frame per cell), train = vaeq_awgn_train_frames_runs (one launch, "
                 "epe epochs), fwd = vaeq_awgn_forward_runs, score = vaeq_awgn_eval_runs; Msym/s = trained symbols per second of the set; "
                 "speed-up = driver ms per epoch / set ms per cell-epoch (the driver row is 16-QAM).")
    text = "\n".join(lines) + "\n"
    print(text)
    os.makedirs(os.path.dirname(out) or ".", exist_ok=True)
    with open(out, "w") as fh:
        fh.write(text)


if __name__ == "__main__":
    main()
