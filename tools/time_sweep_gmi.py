"""Event-timed cost of scoring GMI next to SER in the batched sweep engines, per scored frame of a whole run set.  Writes
profiles/r03_sweep_gmi.txt, or the path given as the first argument.

DP: 592 cells x 10^4 symbols at 64-QAM (VAE-LE geometry: seg_len = batch_len = 100, n_cut 10), posteriors out_train (R,2,16,N) peaked at the
cell's tx levels, rolled by a per-cell shift and polarisation swap, with out_const from the same levels: the existing evaluation
(shared_funcs.frame_eval_runs, both estimators, 7 launches) against the added GMI (shared_funcs.gmi_runs, 2 launches).
AWGN: 592 cells x N_valid 15000 at 16-QAM: awgn.awgn_eval_runs against awgn.awgn_gmi_runs.
Every timed pass runs the evaluation and then the GMI, as the engines do (the GMI reads q right after the evaluation read it; q is larger
than the 126 MB L2).  WARM passes of warm-up, then PASSES timed passes; CUDA events around each call; mean and min per pass."""
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from vae_equalizer_b200 import shared_funcs as sfun  # noqa: E402
from vae_equalizer_b200.awgn import awgn_eval_runs, awgn_gmi_runs  # noqa: E402

R, WARM, PASSES = 592, 3, 20


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:                                       # noqa: BLE001
        return f"nvidia-smi unavailable ({e})"


def posteriors(lev, n, gen, dev, peak=2.5):
    """softmax(noise + peak * onehot(level)) over the levels of each I / Q row: (..., 2, N) levels -> (..., 2n, N)."""
    z = torch.randn(lev.shape[:-2] + (2, n, lev.shape[-1]), generator=gen, device=dev)
    z += peak * torch.nn.functional.one_hot(lev, n).movedim(-1, -2).float()
    return torch.softmax(z, dim=-2).flatten(-3, -2)


def timed(fns):
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(len(fns) + 1)] for _ in range(WARM + PASSES)]
    for k in range(WARM + PASSES):
        ev[k][0].record()
        for i, f in enumerate(fns):
            f()
            ev[k][i + 1].record()
    torch.cuda.synchronize()
    t = np.array([[ev[k][i].elapsed_time(ev[k][i + 1]) for i in range(len(fns))] for k in range(WARM, WARM + PASSES)])
    return t.mean(0), t.min(0)


def dp_set(dev):
    n, N, seg = 8, 10000, 100
    gen = torch.Generator(device=dev).manual_seed(1)
    lev = torch.randint(0, n, (R, 2, 2, N), generator=gen, device=dev)
    S = n - 1
    tx = ((2 * lev - S).float() / S).to(torch.float16)
    amp = torch.linspace(-1, 1, n, device=dev)
    sh = [(r % 11) - 5 for r in range(R)]
    q = posteriors(lev, n, gen, dev)
    out = amp[lev] + 0.05 * torch.randn(R, 2, 2, N, generator=gen, device=dev)
    for r in range(R):                                          # the equalizer's output runs ahead of tx by sh and swaps pols on odd cells
        q[r] = q[r].roll(sh[r], -1).roll(r % 2, 0)
        out[r] = out[r].roll(sh[r], -1).roll(r % 2, 0)
    var, nu = torch.full((R, 2), 0.02, device=dev), torch.zeros(R, device=dev)
    P = torch.full((R, n), 1.0 / n, device=dev)
    st = {}

    def ev():
        st["ser"], st["al"], st["counts"] = sfun.frame_eval_runs(q, out, tx, amp, var, nu, seg, return_counts=True)

    def gm():
        st["gmi"] = sfun.gmi_runs(q, tx, P, st["al"], st["counts"], seg)
    mean, mn = timed([ev, gm])
    n_eval = st["al"][:, 0, 3].double()
    assert torch.isfinite(st["gmi"]).all() and (n_eval > 0).all()
    return mean, mn, float(n_eval.sum()), q.numel() * 4 + tx.numel() * 2


def awgn_set(dev):
    n, N = 4, 15000
    gen = torch.Generator(device=dev).manual_seed(2)
    lev = torch.randint(0, n, (R, 2, N), generator=gen, device=dev)
    S = n - 1
    tx = ((2 * lev - S).float() / S).to(torch.float16)
    q = posteriors(lev, n, gen, dev)
    for r in range(R):
        q[r] = q[r].roll((r % 11) - 5, -1)
    amp = torch.linspace(-1, 1, n, device=dev)
    P = torch.full((R, n), 1.0 / n, device=dev)
    st = {}

    def ev():
        st["shift"], st["counts"], st["ser"] = awgn_eval_runs(q, tx, amp)

    def gm():
        st["gmi"] = awgn_gmi_runs(q, tx, P, st["shift"], st["counts"])
    mean, mn = timed([ev, gm])
    n_eval = (N - 22 - st["shift"]).double()
    assert torch.isfinite(st["gmi"]).all()
    return mean, mn, float(n_eval.sum()), q.numel() * 4 + tx.numel() * 2


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r03_sweep_gmi.txt")
    dev = torch.device("cuda")
    torch.cuda.init()
    lines = [f"card: {card()}", f"torch {torch.__version__}, CUDA {torch.version.cuda}", "",
             f"per scored frame of the WHOLE set of {R} cells; CUDA events, {PASSES} passes after {WARM} warm-up passes (mean / min, ms)", ""]
    for name, fn in (("DP 64-QAM, N 10^4, VAE-LE cut (seg_len 100)", dp_set), ("AWGN 16-QAM, N_valid 15000", awgn_set)):
        (e_mean, g_mean), (e_min, g_min), n_sym, q_bytes = fn(dev)
        lines.append(name)
        lines.append(f"  evaluation (SER)   {e_mean:8.3f} / {e_min:8.3f} ms")
        lines.append(f"  GMI (added)        {g_mean:8.3f} / {g_min:8.3f} ms   = {100 * g_mean / e_mean:5.1f} % of the evaluation, "
                     f"{1e3 * g_mean / R:7.3f} us per cell")
        lines.append(f"  evaluated symbols  {n_sym:.4g} (x 2 pols for DP); GMI {1e6 * g_mean / n_sym:.3f} ns per evaluated symbol")
        lines.append(f"  q + tx arrays      {q_bytes / 1e6:.0f} MB: read once in {g_mean:.3f} ms would be {q_bytes / (g_mean * 1e-3) / 1e12:.2f} TB/s")
        lines.append(f"  minimum the GMI must read (4 q values + 4 fp16 tx per DP symbol, half for AWGN): "
                     f"{(24 if 'DP' in name else 12) * n_sym / 1e6:.0f} MB -> {(24 if 'DP' in name else 12) * n_sym / (g_mean * 1e-3) / 1e12:.2f} TB/s")
        lines.append("")
        print("\n".join(lines[-7:]), flush=True)
        torch.cuda.empty_cache()
    lines.append("The GMI kernel reads the q rows that the tx levels select, so a warp touches up to n_lev rows per 32 symbols: the DRAM traffic "
                 "lies between the minimum above and the whole q array; where in that range it lies was not measured (no hardware-counter profile was taken).")
    text = "\n".join(lines) + "\n"
    print(text)
    os.makedirs(os.path.dirname(out) or ".", exist_ok=True)
    with open(out, "w") as fh:
        fh.write(text)


if __name__ == "__main__":
    main()
