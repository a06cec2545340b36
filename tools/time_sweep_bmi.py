"""Event-timed cost of the bit-metric decoding rate (BMI) in the batched sweep engines and of the bit LLRs.  Writes
profiles/r03_sweep_bmi.txt, or the path given as the first argument.

DP: 592 cells x 10^4 symbols at 64-QAM, VAE-LE geometry (seg_len = batch_len = 100, n_cut 10), the posteriors and alignment of
tools/time_sweep_gmi.py: per scored frame the existing evaluation (shared_funcs.frame_eval_runs, 7 launches), then GMI
(shared_funcs.gmi_runs) and BMI (shared_funcs.bmi_runs, 2 launches each), as the engines run them with gmi=True, bmi=True.
AWGN: 592 cells x N_valid 15000 at 16-QAM: awgn.awgn_eval_runs, awgn_gmi_runs, awgn_bmi_runs.
bit_llr: one run of 2^22 symbols at 64-QAM, (2,16,N) -> (2,6,N): 128 B of q read and 48 B of LLRs written per symbol, against a
device-to-device copy that reads and writes the same 176 B per symbol, timed in the same call and against the 6537 GB/s copy rate of BASELINE.md.
q is larger than the 126 MB L2 in every case.  WARM passes of warm-up, then PASSES timed passes; CUDA events; mean and min per pass.
The -Xptxas -v lines of the new kernel instantiations come from compiling csrc/eval.cu and csrc/eval_runs.cu in a temporary directory."""
import os
import re
import subprocess
import sys
import tempfile

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from time_sweep_gmi import R, card, posteriors, timed  # noqa: E402
from vae_equalizer_b200 import shared_funcs as sfun  # noqa: E402
from vae_equalizer_b200.awgn import awgn_bmi_runs, awgn_eval_runs, awgn_gmi_runs  # noqa: E402

COPY_RATE = 6537e9                     # B/s, the measured HBM copy rate BASELINE.md uses as the roofline denominator


def dp_set(dev):
    n, N, seg = 8, 10000, 100
    gen = torch.Generator(device=dev).manual_seed(1)
    lev = torch.randint(0, n, (R, 2, 2, N), generator=gen, device=dev)
    S = n - 1
    tx = ((2 * lev - S).float() / S).to(torch.float16)
    amp = torch.linspace(-1, 1, n, device=dev)
    q = posteriors(lev, n, gen, dev)
    out = amp[lev] + 0.05 * torch.randn(R, 2, 2, N, generator=gen, device=dev)
    for r in range(R):
        sh = (r % 11) - 5
        q[r] = q[r].roll(sh, -1).roll(r % 2, 0)
        out[r] = out[r].roll(sh, -1).roll(r % 2, 0)
    var, nu = torch.full((R, 2), 0.02, device=dev), torch.zeros(R, device=dev)
    P = torch.full((R, n), 1.0 / n, device=dev)
    st = {}

    def ev():
        st["ser"], st["al"], st["counts"] = sfun.frame_eval_runs(q, out, tx, amp, var, nu, seg, return_counts=True)

    def gm():
        st["gmi"] = sfun.gmi_runs(q, tx, P, st["al"], st["counts"], seg)

    def bm():
        st["bmi"] = sfun.bmi_runs(q, tx, P, st["al"], st["counts"], seg)
    mean, mn = timed([ev, gm, bm])
    assert torch.isfinite(st["bmi"]).all() and bool((st["bmi"] <= st["gmi"] + 1e-6).all())
    return mean, mn, float(st["al"][:, 0, 3].double().sum()) * 2, q.numel() * 4 + tx.numel() * 2, st


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

    def bm():
        st["bmi"] = awgn_bmi_runs(q, tx, P, st["shift"], st["counts"])
    mean, mn = timed([ev, gm, bm])
    assert torch.isfinite(st["bmi"]).all()
    return mean, mn, float((N - 22 - st["shift"]).double().sum()), q.numel() * 4 + tx.numel() * 2, st


def llr_set(dev):
    n, N = 8, 1 << 22
    gen = torch.Generator(device=dev).manual_seed(3)
    lev = torch.randint(0, n, (2, 2, N), generator=gen, device=dev)
    q = posteriors(lev, n, gen, dev)
    src = torch.empty(88 * N // 4, dtype=torch.float32, device=dev).uniform_()     # read + written: the 176 B per symbol of bit_llr
    dst = torch.empty_like(src)
    st = {}

    def llr():
        st["llr"] = sfun.bit_llr(q)

    def copy():
        dst.copy_(src)
    mean, mn = timed([llr, copy])
    assert st["llr"].shape == (2, 6, N) and torch.isfinite(st["llr"]).all()
    return mean, mn, N


def ptxas_lines():
    """-Xptxas -v of csrc/eval.cu and csrc/eval_runs.cu: the BMI (BITS = true) and bit-LLR instantiations."""
    csrc = os.path.join(ROOT, "vae_equalizer_b200", "csrc")
    lines = []
    with tempfile.TemporaryDirectory() as tmp:
        for f in ("eval.cu", "eval_runs.cu"):
            try:
                r = subprocess.run(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas", "-v", "-c", "-o",
                                    os.path.join(tmp, f + ".o"), os.path.join(csrc, f)], capture_output=True, text=True, timeout=900)
            except Exception as e:                               # noqa: BLE001
                return [f"nvcc unavailable ({e})"]
            keep = False
            for ln in r.stderr.splitlines():
                m = re.search(r"Compiling entry function '(\S+)'", ln)
                if m:
                    keep = ("k_gmi" in m.group(1) and "Lb1E" in m.group(1)) or "k_bit_llr" in m.group(1)
                    if keep:
                        lines.append(f"{f}: {m.group(1)}")
                elif keep and ("Used" in ln or "spill" in ln):
                    lines.append("    " + ln.split(":", 1)[-1].strip())
    return lines


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r03_sweep_bmi.txt")
    dev = torch.device("cuda")
    torch.cuda.init()
    lines = [f"card: {card()}", f"torch {torch.__version__}, CUDA {torch.version.cuda}", "",
             f"per scored frame of the WHOLE set of {R} cells; CUDA events, mean / min over the timed passes (ms)", ""]
    for name, fn, need in (("DP 64-QAM, N 10^4, VAE-LE cut (seg_len 100)", dp_set, 2 * 8 * 4 + 4),
                           ("AWGN 16-QAM, N_valid 15000", awgn_set, 2 * 4 * 4 + 4)):
        (e_mean, g_mean, b_mean), (e_min, g_min, b_min), n_sym, q_bytes, st = fn(dev)
        lines.append(name)
        lines.append(f"  evaluation (SER)   {e_mean:8.3f} / {e_min:8.3f} ms")
        lines.append(f"  GMI pair           {g_mean:8.3f} / {g_min:8.3f} ms")
        lines.append(f"  BMI pair (added)   {b_mean:8.3f} / {b_min:8.3f} ms   = {100 * b_mean / e_mean:5.1f} % of the evaluation, "
                     f"{1e3 * b_mean / R:7.3f} us per cell")
        lines.append(f"  scored pol-symbols {n_sym:.4g}; the BMI reads every q row of a scored symbol and its tx pair, {need} B per pol-symbol: "
                     f"{need * n_sym / 1e6:.0f} MB -> {need * n_sym / (b_mean * 1e-3) / 1e12:.2f} TB/s (q + tx arrays {q_bytes / 1e6:.0f} MB)")
        lines.append(f"  mean over the cells: GMI {float(st['gmi'].double().mean()):.4f}, BMI {float(st['bmi'].double().mean()):.4f} bit/2D symbol")
        lines.append("")
        print("\n".join(lines[-7:]), flush=True)
        torch.cuda.empty_cache()
    (l_mean, c_mean), (l_min, c_min), N = llr_set(dev)
    nbytes = 176 * N
    lines.append(f"bit_llr, 64-QAM, one run of N = 2^22 symbols: q (2,16,N) read + LLRs (2,6,N) written = 176 B per symbol, {nbytes / 1e6:.0f} MB")
    lines.append(f"  bit_llr            {l_mean:8.3f} / {l_min:8.3f} ms   = {nbytes / (l_mean * 1e-3) / 1e12:.2f} TB/s, "
                 f"{nbytes / (l_mean * 1e-3) / COPY_RATE:.2f} of the 6537 GB/s copy rate of BASELINE.md")
    lines.append(f"  copy, {nbytes / 2e6:.0f} MB   {c_mean:8.3f} / {c_min:8.3f} ms   = {nbytes / (c_mean * 1e-3) / 1e12:.2f} TB/s read + write, "
                 f"same call; bit_llr takes {l_mean / c_mean:.2f} x the time of this copy of the same bytes")
    lines.append("")
    lines.append("ptxas (nvcc -gencode arch=compute_100a,code=sm_100a -O3 -Xptxas -v): BMI instantiations (BITS = true: k_gmi_runs<NL, NPOL, true>, "
                 "k_gmi<NL, V, true>) and k_bit_llr<NL, V>")
    lines += ptxas_lines()
    text = "\n".join(lines) + "\n"
    print(text)
    os.makedirs(os.path.dirname(out) or ".", exist_ok=True)
    with open(out, "w") as fh:
        fh.write(text)


if __name__ == "__main__":
    main()
