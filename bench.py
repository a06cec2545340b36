#!/usr/bin/env python
"""bench.py -- DP VAE-LE training throughput on B200 (BASELINE.json metric) + roofline + CPU baseline.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference algorithm on the host CPU (oracle port)
    python bench.py --steps K --warmup W --dump-outputs DIR  # also write the outputs of the last timed step, to compare builds

A "step" is one full training step (butterfly FIR -> soft demapper -> ELBO -> backward -> Adam on both
parameter groups) over one minibatch of B = 2^22 synthetic DP 64-QAM PCS symbols (BASELINE configs[1]:
func_VAELE_DP, 2x2 butterfly, M_est = 25, sps = 2, SNR 23 dB, nu = 0.0270955).  With N > 1 every rank trains
its own independent sweep point (different noise realisation / seed) -- the reference's sweep is embarrassingly
parallel (Eval_run_DP.py:68-95) -- so scaling is weak and there is no data-path collective.

One JSON line on stdout (rank 0).  Nothing here reads /root/reference.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "DP VAE-LE train symbols/s"
UNIT = "symbols/s"
MOD, NU, SNR, M_EST, SPS, LR = "64-QAM", 0.0270955, 23, 25, 2, 2.5e-3
N_LEV = 8
ALG_BYTES_PER_SYMBOL = 4 * 2 * (2 * SPS + 2 * N_LEV + 2)        # SURVEY.md §8d: read rx once, write q and out once = 176 B
ALG_FLOP_PER_SYMBOL = 5 * 32 * M_EST + 1000                      # SURVEY.md §8d: 5 tap contractions + point-wise work
# dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the dominant kernel (k_dp_fwd_tc<8,12>, the default forward kernel since r02c) at
# batch_len 2^22 from the `ncu --set full` capture summarised in profiles/r02c_ncu_full_summary.json (entry early_staging): 134.3 MB read + 949.7 MB
# written = 258.5 B/symbol
FWD_DRAM_BYTES_PER_SYMBOL = (134.307e6 + 949.731e6) / (1 << 22)
TRAFFIC_SOURCE = "ncu --set full dram__bytes_read.sum + dram__bytes_write.sum of k_dp_fwd_tc<8,12>, profiles/r02c_ncu_full_summary.json, scaled to this batch_len"
CPU_SAMPLE_LOG2 = 17
DUMP_SAMPLE_LOG2 = 18                                            # --dump-outputs: q / out columns kept (2^18 symbols = 36 MiB of float32)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons sampled through NVML every ~2 ms DURING the timed region."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.sm, self.reasons, self.stop_flag, self.smax, self.err = index, [], set(), False, None, None
        self.nv = self.h = None
        try:                                 # NVML is initialised here, before the timed region
            import pynvml as nv
            nv.nvmlInit()
            self.nv, self.h = nv, nv.nvmlDeviceGetHandleByIndex(index)
            self.smax = float(nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM))
        except Exception as e:
            self.err = repr(e)

    def run(self):
        if self.nv is None:
            return
        try:
            nv, h = self.nv, self.h
            bits = {"hw_slowdown": nv.nvmlClocksEventReasonHwSlowdown if hasattr(nv, "nvmlClocksEventReasonHwSlowdown") else 0x8,
                    "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}
            while not self.stop_flag:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for name, b in bits.items():
                    if r & b:
                        self.reasons.add(name)
                time.sleep(0.001)
        except Exception as e:              # NVML unavailable: report that instead of inventing numbers
            self.err = repr(e)

    def finish(self):
        self.stop_flag = True
        self.join(timeout=2.0)
        if not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": self.smax, "reasons": [], "samples": 0, "error": self.err}
        return {"sm_mhz": float(np.median(self.sm)), "sm_max_mhz": self.smax, "reasons": sorted(self.reasons), "samples": len(self.sm)}


def _nvml_index(local_rank):
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local_rank])
        except Exception:
            pass
    return local_rank


def run_constants():
    from vae_equalizer_b200.constants import init
    h_est, h_channel, P, amp_levels, amps, pol, nu_sc, var, pow_mean = init("h0", MOD, "cpu", NU, SPS, M_EST, SNR)
    return dict(P=P, amp=amp_levels, amps=amps, nu_sc=nu_sc, var=var)


def cpu_step_rate(rx_cpu, cst, steps, warmup, max_seconds):
    """The reference algorithm (oracle/vaeq_oracle.py: conv1d + softmin + per-tap gather loop + autograd + torch Adam)
    on this box's host cores, on a bounded sample of the same workload."""
    from oracle import vaeq_oracle as O
    torch.set_num_threads(os.cpu_count() or 1)
    tr = O.DPTrainer(M_EST, SPS, LR)
    Pt = torch.tensor(cst["P"], dtype=torch.float32)
    B = rx_cpu.shape[-1] // SPS
    for _ in range(warmup):
        tr.step(rx_cpu, cst["amp"], cst["var"], cst["nu_sc"], Pt)
    t0 = time.perf_counter()
    done = 0
    for _ in range(steps):
        tr.step(rx_cpu, cst["amp"], cst["var"], cst["nu_sc"], Pt)
        done += 1
        if time.perf_counter() - t0 > max_seconds:
            break
    dt = time.perf_counter() - t0
    return B * done / dt, done, dt, torch.get_num_threads()


def synth_cpu_sample(cst, log2_b, seed):
    from vae_equalizer_b200.datagen import generate_data_shaping
    from vae_equalizer_b200.constants import upsampled_channel
    rng = np.random.default_rng(seed)
    rx, _, _ = generate_data_shaping(1 << log2_b, cst["amps"], SNR, upsampled_channel("h0", SPS), cst["P"], 2, 90e9, SPS, -26e-24,
                                     0.1e-12 * np.sqrt(1000), np.array([0.0314, 0.0314], dtype=np.complex64), np.pi / 10, "cpu", rng=rng)
    return rx


def workload_name(log2_b):
    return (f"DP VAE-LE (func_VAELE_DP) train step, {MOD} PCS nu={NU}, 2x2 butterfly M_est={M_EST}, sps={SPS}, SNR {SNR} dB, "
            f"batch_len=2^{log2_b} symbols/step, synthetic RRC+rotation+CD/PMD channel (BASELINE configs[1])")


def reference_arm(args, rank, world):
    if rank != 0:
        return
    cst = run_constants()
    rx = synth_cpu_sample(cst, CPU_SAMPLE_LOG2, 1234)
    rate, done, dt, cores = cpu_step_rate(rx, cst, args.steps, max(1, min(args.warmup, 2)), max_seconds=150.0)
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": done, "warmup": args.warmup,
        "ms_per_step": 1e3 * dt / max(done, 1), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": workload_name(args.batch_log2), "sample": f"each step = one full training step on 2^{CPU_SAMPLE_LOG2} symbols of the workload"},
        "cpu_baseline": {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{done} steps x 2^{CPU_SAMPLE_LOG2} symbols, oracle/vaeq_oracle.py DPTrainer (torch CPU, autograd, torch Adam)"},
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def dump_outputs(eq, q, out, d):
    """Write what the last train_step handed its caller to d/<name>.npy (float32): q and out on a fixed, seeded sample of
    2^DUMP_SAMPLE_LOG2 symbol columns (all columns at smaller batch_len), loss, var_est, and the taps W and h after its Adam update."""
    B = q.shape[-1]
    n = min(B, 1 << DUMP_SAMPLE_LOG2)
    cols = np.sort(np.random.default_rng(0).choice(B, n, replace=False))
    idx = torch.from_numpy(cols).to(q.device)
    arrays = {"q": q.index_select(2, idx), "out": out.index_select(2, idx), "loss": eq.loss, "var_est": eq.var_est, "W": eq.W, "h": eq.h}
    os.makedirs(d, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(d, name + ".npy"), t.cpu().numpy())


def ours_arm(args, rank, local_rank, world):
    import torch.distributed as dist
    from vae_equalizer_b200 import _lib
    from vae_equalizer_b200.datagen import generate_data_gpu
    from vae_equalizer_b200.dp import DPEqualizer

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()
    cst = run_constants()
    B = 1 << args.batch_log2
    NB = args.buffers
    K, W = args.steps, max(args.warmup, 3)

    # ---- synthetic inputs, resident in HBM before the timed region --------------------------------------------
    theta = np.pi / 10 + 0.06 * np.pi * rank                     # each rank = another sweep point / realisation
    rx_dev = [generate_data_gpu(B, cst["amps"], SNR, cst["P"], SPS, theta, dev, 1234 + 100 * rank + i)[0] for i in range(NB)]
    eq = DPEqualizer(M_EST, SPS, cst["amp"], cst["P"], cst["var"], cst["nu_sc"], device=dev)
    q = torch.empty(2, 2 * N_LEV, B, dtype=torch.float32, device=dev)
    out = torch.empty(2, 2, B, dtype=torch.float32, device=dev)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(W):
        eq.train_step(rx_dev[i % NB], LR, LR, q=q, out=out)
    barrier()

    # ---- timed region: EXACTLY K steps, device timed, no instrumentation inside.  The steps are replayed from a CUDA graph of NB
    # consecutive train_step calls (one per rotating rx batch; DPEqualizer.capture_steps), the remaining K % NB steps are plain calls.
    graph = eq.capture_steps([rx_dev[i % NB] for i in range(NB)], LR, LR, q=q, out=out)
    cap0 = int(lib.vaeq_launch_count(-1))
    eq.train_step(rx_dev[0], LR, LR, q=q, out=out)
    launches_per_step = int(lib.vaeq_launch_count(-1)) - cap0
    sampler = ClockSampler(_nvml_index(local_rank))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    sampler.start()
    e0.record()
    for _ in range(K // NB):
        graph.replay()
    for i in range(K % NB):
        eq.train_step(rx_dev[i], LR, LR, q=q, out=out)
    e1.record()
    while not e1.query():                  # the host is idle while the graphs run: yield to the clock sampler thread
        time.sleep(0.0005)
    barrier()
    ms = e0.elapsed_time(e1)
    clocks = sampler.finish()
    launches = launches_per_step * K
    if args.dump_outputs and rank == 0:                # before the legs below overwrite q / out and step the taps further
        dump_outputs(eq, q, out, args.dump_outputs)
    # ---- the same K steps as plain launches, and once more with the library's per-kernel event pairs on the launching stream
    # (12 event records per step: they cost ~30 us per step, so they stay out of the region `value` is taken from) ------------------
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p0.record()
    for i in range(K):
        eq.train_step(rx_dev[i % NB], LR, LR, q=q, out=out)
    p1.record()
    barrier()
    ms_plain = p0.elapsed_time(p1)
    _lib.check(lib.vaeq_kernel_timing(1))
    k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    k0.record()
    for i in range(K):
        eq.train_step(rx_dev[i % NB], LR, LR, q=q, out=out)
    k1.record()
    barrier()
    ms_events = k0.elapsed_time(k1)
    ms_sum = (C.c_float * 16)()
    cnt = (C.c_int32 * 16)()
    _lib.check(lib.vaeq_kernel_timing_read(ms_sum, cnt))
    _lib.check(lib.vaeq_kernel_timing(0))
    loss_val = float(eq.loss.item())
    if not np.isfinite(loss_val):
        raise SystemExit(f"non-finite loss {loss_val} in the timed region")

    # ---- sustained leg: the same graph replayed for >= 1 s (the K-step region above lasts milliseconds), with its own clock record.
    # It runs AFTER the per-kernel timing pass: 1.6 s under the power cap leave the clocks lower for a while, and the kernel durations
    # of the roofline are to be taken in the clock state of the timed region ----
    sustained = None
    if not args.no_sustained:
        n_rep = max(1, int(np.ceil(args.sustained_seconds * 1e3 / (ms / K * NB))))
        s_sampler = ClockSampler(_nvml_index(local_rank))
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        s_sampler.start()
        s0.record()
        for _ in range(n_rep):
            graph.replay()
        s1.record()
        while not s1.query():
            time.sleep(0.002)
        barrier()
        s_ms = s0.elapsed_time(s1)
        ts = torch.tensor([s_ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ts, op=dist.ReduceOp.MAX)
        sustained = {"value": world * B * NB * n_rep / (float(ts.item()) * 1e-3), "unit": UNIT, "steps": NB * n_rep, "seconds": float(ts.item()) * 1e-3,
                     "ms_per_step": float(ts.item()) / (NB * n_rep), "clocks": s_sampler.finish(),
                     "note": "same CUDA graph as the timed region, replayed back to back; max over ranks"}
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    value = world * B * K / (ms_max * 1e-3)

    # ---- end to end through the public API with HOST buffers: H2D of each step's rx, D2H of loss/var_est ----------
    rx_host = [r.cpu().pin_memory() for r in rx_dev[:2]]
    stage = [torch.empty_like(rx_dev[0]) for _ in range(2)]
    res_host = torch.empty(K + W, 3, dtype=torch.float32).pin_memory()
    copy_stream = torch.cuda.Stream(device=dev)
    main_stream = torch.cuda.current_stream()
    ready = [torch.cuda.Event() for _ in range(2)]
    free = [torch.cuda.Event() for _ in range(2)]

    def e2e_steps(n, base):
        for i in range(n):
            s = i % 2
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(free[s])
                stage[s].copy_(rx_host[(base + i) % 2], non_blocking=True)
                ready[s].record(copy_stream)
            main_stream.wait_event(ready[s])
            eq.train_step(stage[s], LR, LR, q=q, out=out)
            free[s].record(main_stream)
            res_host[base + i, 0:1].copy_(eq.loss, non_blocking=True)
            res_host[base + i, 1:3].copy_(eq.var_est, non_blocking=True)

    for s in range(2):
        free[s].record(main_stream)
    e2e_steps(W, 0)
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    e2e_steps(K, W)
    f1.record()
    barrier()
    t2 = torch.tensor([f0.elapsed_time(f1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t2, op=dist.ReduceOp.MAX)
    e2e_value = world * B * K / (float(t2.item()) * 1e-3)

    # ---- configs[1] at the reference's OWN batch_len = 100 (Eval_run_DP.py:38): one frame = 100 sequential steps in one
    # persistent launch (dp_small.cu); many independent sweep cells batched per launch (configs[4]) --------------------------
    small = None
    if rank == 0 and not args.no_small:
        from vae_equalizer_b200.dp import DPEqualizerRuns
        Bs, ns = 100, 100
        small = {"batch_len": Bs, "steps_per_frame": ns, "note": "VAE-LE frame of 10 000 symbols as 100 sequential minibatches of 100 "
                 "(func_VAELE_DP_MQAM_shaping.py:57-66), one persistent launch per frame; R independent runs batched per launch"}
        for R in (1, 592):
            rxs = torch.stack([generate_data_gpu(Bs * ns, cst["amps"], SNR, cst["P"], SPS, np.pi / 10 + 0.01 * r, dev, 77 + r)[0] for r in range(R)])
            eqr = DPEqualizerRuns(R, M_EST, SPS, cst["amp"], cst["P"], cst["var"], cst["nu_sc"], device=dev)
            otr = torch.empty(R, 2, 2 * N_LEV, Bs * ns, device=dev)
            ocr = torch.empty(R, 2, 2, Bs * ns, device=dev)
            for _ in range(2):
                eqr.train_frame(rxs, Bs, Bs, ns, LR, LR, otr, ocr, 0, Bs, keep_lo_in_dst=True)
            torch.cuda.synchronize()
            h0, h1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            h0.record()
            for _ in range(5):
                eqr.train_frame(rxs, Bs, Bs, ns, LR, LR, otr, ocr, 0, Bs, keep_lo_in_dst=True)
            h1.record()
            torch.cuda.synchronize()
            msf = h0.elapsed_time(h1) / 5
            small[f"runs_{R}"] = {"ms_per_frame": msf, "us_per_step": msf * 1e3 / ns, "symbols_per_s": R * Bs * ns / (msf * 1e-3)}
            del rxs, eqr, otr, ocr
        # the sweep engine end to end (configs[4]): per frame batched data generation + one training launch + batched evaluation
        from vae_equalizer_b200 import sweep as _sweep
        cells = [dict(SNR=15 + 2 * (i % 8), nu=NU, lr_optim=LR, theta=np.pi / 10, theta_diff=0.06 * np.pi, seed=i) for i in range(592)]      # 4 x 148 SMs: one wave of the persistent frame kernel
        n_fr = 24
        _sweep.sweep_vae_dp(cells, MOD, SPS, M_EST, Bs, Bs * ns, n_fr, kind="VAE", datagen="gpu_batched", device=dev)   # warm-up at full size and length (allocator growth, cuFFT plans)
        torch.cuda.synchronize()
        tw = time.perf_counter()
        ser_s, _, _ = _sweep.sweep_vae_dp(cells, MOD, SPS, M_EST, Bs, Bs * ns, n_fr, kind="VAE", datagen="gpu_batched", device=dev)
        torch.cuda.synchronize()
        tw = time.perf_counter() - tw
        small["sweep_end_to_end"] = {"cells": len(cells), "frames": n_fr, "ms_per_frame": tw / n_fr * 1e3, "symbols_per_s": len(cells) * n_fr * Bs * ns / tw,
                                     "note": "sweep.sweep_vae_dp wall clock: on-device data generation + persistent training launch + batched "
                                             "alignment / SER evaluation for all cells, every frame evaluated like the reference"}

    # ---- config 3 (BASELINE configs[2]): ONE VAE-flex run with long windows, every window batch-split over the ranks.  Literally the
    # driver's frame loop (func_VAEflex_DP_MQAM_shaping.py:59-70): batch_len = world x 2^batch_log2, flex_step = batch_len / 2, 8 steps per
    # frame, the kept middle section of every window written to the frame's out_train / out_const; parallel.BatchSplitDP.train_frame
    # replays the frame from a CUDA graph.  Both reduction transports are timed: NVLink peer memory (in-library) and NCCL all-reduces.
    split = None
    if world > 1 and not args.no_split:
        from vae_equalizer_b200.parallel import BatchSplitDP
        del rx_host, stage, q, out, graph, eq
        rx_dev.clear()
        torch.cuda.empty_cache()
        Bt, n_fs = B * world, 8
        stride = Bt // 2
        N_frame = 5 * Bt
        rx_big = torch.empty(2, 2, SPS * N_frame, dtype=torch.float32, device=dev)
        for c in range(5):                                            # same seeds on every rank: the frame is replicated, as the driver broadcasts it
            rx_big[:, :, c * SPS * Bt:(c + 1) * SPS * Bt] = generate_data_gpu(Bt, cst["amps"], SNR, cst["P"], SPS, np.pi / 10, dev, 4321 + c)[0]
        ot = torch.zeros(2, 2 * N_LEV, n_fs * stride, dtype=torch.float32, device=dev)
        oc = torch.zeros(2, 2, n_fs * stride, dtype=torch.float32, device=dev)
        keep_lo = (Bt - stride) // 2
        split = {"unit": UNIT, "batch_len": Bt, "flex_step": stride, "steps_per_frame": n_fs, "scaling": "weak (batch_len grows with N)",
                 "exchange_bytes_per_step": 8 * (8 + 2 * (M_EST - 1)) + 4 * 16 * M_EST,
                 "note": "BASELINE configs[2]: VAE-flex frame loop, every window split in contiguous symbol ranges; per step the ELBO sums and the "
                         "400 tap-gradient floats are reduced over the ranks, Adam is replicated; each rank holds q / out for its own columns only"}
        n_frames = max(3, K // n_fs)
        for transport in ("peer", "nccl"):
            eq2 = DPEqualizer(M_EST, SPS, cst["amp"], cst["P"], cst["var"], cst["nu_sc"], device=dev)
            try:
                bs = BatchSplitDP(eq2, None, transport)
            except Exception as e:                                    # no symmetric memory on this box: say so, keep the NCCL number
                split[transport] = {"unavailable": repr(e)[:200]}
                continue
            for _ in range(2):
                bs.train_frame(rx_big, Bt, stride, n_fs, LR, LR, ot, oc, keep_lo, stride)
            bs.gather_kept(Bt, stride, n_fs, ot, oc, keep_lo, stride, dst=0)      # first call sets up the point-to-point connections
            barrier()
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            g0.record()
            for _ in range(n_frames):
                bs.train_frame(rx_big, Bt, stride, n_fs, LR, LR, ot, oc, keep_lo, stride)
            g1.record()
            barrier()
            t3 = torch.tensor([g0.elapsed_time(g1)], dtype=torch.float64, device=dev)
            dist.all_reduce(t3, op=dist.ReduceOp.MAX)
            h0, h1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            h0.record()
            bs.gather_kept(Bt, stride, n_fs, ot, oc, keep_lo, stride, dst=0)
            h1.record()
            barrier()
            t4 = torch.tensor([h0.elapsed_time(h1)], dtype=torch.float64, device=dev)
            dist.all_reduce(t4, op=dist.ReduceOp.MAX)
            steps = n_frames * n_fs
            split[transport] = {"value": Bt * steps / (float(t3.item()) * 1e-3), "ms_per_step": float(t3.item()) / steps, "steps": steps,
                                "efficiency_vs_n_independent_runs": (Bt * steps / (float(t3.item()) * 1e-3)) / value,
                                "gather_kept_ms_per_frame": float(t4.item()), "final_loss": float(eq2.loss.item())}
            del bs, eq2
        best = max((split[t]["value"] for t in ("peer", "nccl") if "value" in split[t]), default=None)
        split["value"] = best
        del rx_big, ot, oc

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel ---------------------------------------------------------------------------
    names = {0: "k_dp_fwd", 1: "k_dp_fin", 2: "k_dp_bwd1 (dE_q + softmin backward)", 3: "k_dp_adam", 8: "k_dp_taps<W>", 9: "k_dp_taps<h>"}
    per_kernel = {names[k]: {"avg_ms": ms_sum[k] / cnt[k], "launches": int(cnt[k]), "share_of_step": ms_sum[k] / ms_events}
                  for k in names if cnt[k] > 0}
    dom = max((k for k in names if cnt[k] > 0), key=lambda k: ms_sum[k])
    dom_ms = ms_sum[dom] / cnt[dom]
    peak, peak_src = load_peaks()
    achieved = B * ALG_BYTES_PER_SYMBOL / (dom_ms * 1e-3) / 1e9
    step_gbs = B * ALG_BYTES_PER_SYMBOL * K / (ms * 1e-3) / 1e9
    symbols = {"k_dp_fwd": "vaeq::k_dp_fwd_tc<8,12> (FIR and channel convolution on tcgen05, point-wise stage on the CUDA cores; csrc/dp_fwd_tc.cu)",
               "k_dp_taps<W>": "vaeq::k_dp_taps_tc (both tap-gradient correlations in one tcgen05 launch; csrc/dp_taps_tc.cu)"}
    roofline = {"bound": "hbm", "kernel": names[dom], "kernel_symbol": symbols.get(names[dom], names[dom]), "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": (FWD_DRAM_BYTES_PER_SYMBOL * B if names[dom] == "k_dp_fwd" and M_EST == 25 else None),
                "traffic_unit": "bytes per launch", "traffic_source": TRAFFIC_SOURCE + " -- taken from that ncu capture, NOT measured in this run",
                "peak_source": peak_src, "alg_bytes_per_symbol": ALG_BYTES_PER_SYMBOL,
                "alg_bytes_per_launch": B * ALG_BYTES_PER_SYMBOL,
                "whole_step_achieved": step_gbs, "whole_step_frac": step_gbs / peak,
                "fp32_issue": {"alg_flop_per_symbol": ALG_FLOP_PER_SYMBOL, "achieved_tflops": value / world * ALG_FLOP_PER_SYMBOL / 1e12,
                               "peak_tflops": 72.0, "peak_source": "profiles/r01_ffma_issue_microbench.txt (FFMA reg,reg,reg on this pool)",
                               "frac": value / world * ALG_FLOP_PER_SYMBOL / 72.0e12},
                "kernels": per_kernel,
                "kernel_timing": f"CUDA event pairs around every launch on the launching stream, {K} steps right after the timed region "
                                 f"(same inputs and state); that instrumented pass takes {ms_events / K:.4f} ms per step, the same steps as plain "
                                 f"launches {ms_plain / K:.4f} ms, the timed region (CUDA graph replay) {ms / K:.4f} ms"}

    # ---- CPU baseline on a bounded sample (N=1 only) -----------------------------------------------------------------
    cpu = None
    if world == 1 and not args.no_cpu:
        rx_cpu = rx_dev[0][:, :, :SPS << CPU_SAMPLE_LOG2].cpu().contiguous()
        rate, done, dt, cores = cpu_step_rate(rx_cpu, cst, 4, 1, max_seconds=25.0)
        cpu = {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": f"{done} steps x 2^{CPU_SAMPLE_LOG2} symbols (first 2^{CPU_SAMPLE_LOG2} symbols of the workload), "
                         f"oracle/vaeq_oracle.py DPTrainer on torch CPU, {dt:.1f} s"}
        other = {}
        for b_cpu, n_cpu in ((100, 60), (10000, 20)):        # BASELINE.md section 3: the reference's own batch_len and a mid size
            rx_b = rx_dev[0][:, :, :SPS * b_cpu].cpu().contiguous()
            r_b, d_b, t_b, _ = cpu_step_rate(rx_b, cst, n_cpu, 2, max_seconds=8.0)
            other[str(b_cpu)] = {"value": r_b, "unit": UNIT, "steps": d_b, "seconds": t_b}
        cpu["other_batch_len"] = other

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms_max / K,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args.batch_log2), "batch_len": B, "M_est": M_EST, "n_lev": N_LEV,
                   "l2": f"inputs larger than L2: {NB} rotating rx batches of {B * 16 >> 20} MiB, {B * 128 >> 20} MiB of q written per step (L2 = 126 MB)",
                   "parallelism": "independent sweep points, one per GPU, no collective" if world > 1 else "1 GPU",
                   "launch": f"CUDA graph of {NB} consecutive DPEqualizer.train_step calls replayed {K // NB} times + {K % NB} plain calls",
                   "ms_per_step_plain_launches": ms_plain / K,
                   "final_loss": loss_val},
        "roofline": roofline,
        "cpu_baseline": cpu,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": B * 4 * 2 * 2 * SPS, "d2h_bytes_per_step": 12,
                "h2d_gbs": B * 4 * 2 * 2 * SPS * K / (float(t2.item()) * 1e-3) / 1e9,
                "note": "DPEqualizer.train_step on pinned host rx (fp32, 32 B/symbol); H2D double-buffered on a copy stream, loss+var_est "
                        "read back every step; bound by the PCIe Gen5 x16 link (tools/h2d_probe.py measures 55 GB/s on this pool)"},
        "gpu_launches": launches,
        "clocks": clocks,
    }
    # extra legs live under `config` (the driver keeps the nested objects of the contract keys)
    if sustained is not None:
        line["config"]["sustained"] = sustained
    if split is not None:
        line["config"]["batch_split"] = split
    if small is not None:
        line["config"]["reference_batch_len"] = small
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch-log2", type=int, default=22)
    ap.add_argument("--buffers", type=int, default=3)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-small", action="store_true", help="skip the batch_len = 100 persistent-frame leg")
    ap.add_argument("--no-split", action="store_true", help="skip the batch-split (configs[2]) leg at N > 1")
    ap.add_argument("--no-sustained", action="store_true", help="skip the >= 1 s sustained leg")
    ap.add_argument("--sustained-seconds", type=float, default=1.5)
    ap.add_argument("--m-est", type=int, default=M_EST, help="equalizer / channel-estimate taps (default 25 = the BASELINE config; "
                    "5, 9, 13 show the HBM-bound regime, SURVEY.md §8d)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step to DIR/<name>.npy (rank 0; "
                    "q and out on a fixed sample of 2^%d symbols)" % DUMP_SAMPLE_LOG2)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.m_est != M_EST:
        globals()["M_EST"] = args.m_est
        globals()["ALG_FLOP_PER_SYMBOL"] = 5 * 32 * args.m_est + 1000

    if args.gpus > 1 and "RANK" not in os.environ:          # launched bare: re-exec under torchrun (one rank per GPU)
        import socket
        s = socket.socket()
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
        s.close()
        os.execvp(sys.executable, [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
                                   "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.abspath(__file__)] + sys.argv[1:])
    rank = int(os.environ.get("RANK", 0))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if args.impl == "reference":
        reference_arm(args, rank, world)
    else:
        ours_arm(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
