"""Device data generator on the channel presets h0, h1 and h2 (profiles/r03_datagen_isi.txt).

- generate_frames_gpu: one 592-cell frame of 10 000 64-QAM symbols per call, per-run parameters on the device (as sweep_vae_dp's
  gpu_batched source passes them), CUDA events around 50 calls after 5 warm-up calls;
- the host generator generate_data_shaping: one cell-frame of 10 000 symbols, host clock over 20 calls, in the same process;
- sweep_vae_dp (VAE-LE, batch_len 100, M_est 25) end to end per frame with datagen='gpu_batched' on 592 cells, h1 and h0 for
  comparison: host clock around num_frames frames ending in a device synchronise, after a 1-frame warm-up of the same set;
- in a separate pass after the timings, the device time of one generate_frames_gpu call per channel by kernel (torch.profiler).
Prints the card's name and power limit first."""
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from vae_equalizer_b200 import sweep  # noqa: E402
from vae_equalizer_b200.constants import init, upsampled_channel  # noqa: E402
from vae_equalizer_b200.datagen import generate_data_shaping, generate_frames_gpu  # noqa: E402

R, N, F = int(os.environ.get("R", 592)), int(os.environ.get("N", 10000)), int(os.environ.get("F", 20))
PHI = np.array([0.0314, 0.0314], dtype=np.complex64)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def device_frame_ms(channel, amps, P, snr, th, n_calls=50):
    h = upsampled_channel(channel, 2)
    for i in range(5):
        generate_frames_gpu(N, amps, snr, P, 2, th, "cuda", i, h_channel=h)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(n_calls):
        generate_frames_gpu(N, amps, snr, P, 2, th, "cuda", 100 + i, h_channel=h)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n_calls


def host_frame_ms(channel, k, n_calls=20):
    rng = np.random.default_rng(0)
    args = (N, k[4], 23, k[1], k[2], 2, 90e9, 2, -26e-24, 0.1e-12 * np.sqrt(1000), PHI, np.pi / 10, "cpu")
    generate_data_shaping(*args, rng=rng)
    t0 = time.perf_counter()
    for _ in range(n_calls):
        generate_data_shaping(*args, rng=rng)
    return (time.perf_counter() - t0) / n_calls * 1e3


def sweep_frame_ms(channel):
    cells = [dict(SNR=15 + 2 * (i % 8), nu=0.0270955, lr_optim=2.5e-3, theta=np.pi / 10, theta_diff=0.06 * np.pi, seed=i) for i in range(R)]
    sweep.sweep_vae_dp(cells, "64-QAM", 2, 25, 100, N, 1, channel=channel, kind="VAE", datagen="gpu_batched")
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ser, _, _ = sweep.sweep_vae_dp(cells, "64-QAM", 2, 25, 100, N, F, channel=channel, kind="VAE", datagen="gpu_batched")
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / F * 1e3, float(ser[:, 2:, -1].mean())


def kernel_breakdown(channel, amps, P, snr, th):
    """torch.profiler table of one warm generate_frames_gpu call, by kernel."""
    from torch.profiler import ProfilerActivity, profile
    h = upsampled_channel(channel, 2)
    generate_frames_gpu(N, amps, snr, P, 2, th, "cuda", 1, h_channel=h)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU]) as prof:
        generate_frames_gpu(N, amps, snr, P, 2, th, "cuda", 2, h_channel=h)
        torch.cuda.synchronize()
    return prof.key_averages().table(sort_by="cuda_time_total", row_limit=14, max_name_column_width=60)


def main():
    torch.cuda.set_device(0)
    print(f"card: {card()}   torch {torch.__version__}, CUDA {torch.version.cuda}, host CPUs {os.cpu_count()}")
    print(f"R = {R} cells x N = {N} symbols, 64-QAM, nu 0.0270955, sps 2\n")
    k = init("h0", "64-QAM", "cpu", 0.0270955, 2, 25, 23)
    amps = k[4]
    P = torch.as_tensor(np.tile(np.asarray(k[2], dtype=np.float32)[None], (R, 1)), device="cuda")
    snr = torch.tensor([15.0 + 2 * (i % 8) for i in range(R)], device="cuda")
    th = torch.full((R,), 0.3, device="cuda")
    print(f"{'channel':8s} {'K':>3s} {'FFT n':>6s} {'device, per 592-cell frame':>27s} {'host, per cell-frame':>21s} {'host x 592':>11s}")
    for channel in ("h0", "h1", "h2"):
        kc = init(channel, "64-QAM", "cpu", 0.0270955, 2, 25, 23)
        L = len(kc[1])
        K, n = 32 + L - 1, 2 * (N + L + 32) - (32 + L - 1)
        d = device_frame_ms(channel, amps, P, snr, th)
        hst = host_frame_ms(channel, kc)
        print(f"{channel:8s} {K:3d} {n:6d} {d:24.3f} ms {hst:18.2f} ms {hst * R / 1e3:9.2f} s")
    print(f"\nsweep_vae_dp, VAE-LE, batch_len 100, M_est 25, datagen='gpu_batched', {R} cells, {F} frames after a 1-frame warm-up:")
    for channel in ("h1", "h0"):
        ms, ser = sweep_frame_ms(channel)
        print(f"  {channel}: {ms:.2f} ms per frame end to end   (mean soft-demapper SER of the last frame {ser:.4f})")
    print("\ndevice time of one generate_frames_gpu call by kernel (torch.profiler, separate pass):")
    for channel in ("h0", "h1", "h2"):
        print(f"  {channel}:")
        print(kernel_breakdown(channel, amps, P, snr, th))


if __name__ == "__main__":
    main()
