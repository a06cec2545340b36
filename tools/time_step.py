"""Per-kernel CUDA-event times of the DP step at batch_len 2^22 with the tap gradients on the tensor cores and on the CUDA cores
(vaeq_kernel_timing)."""
import ctypes as C, os, sys
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from vae_equalizer_b200 import _lib
from vae_equalizer_b200.constants import init
from vae_equalizer_b200.datagen import generate_data_gpu
from vae_equalizer_b200.dp import DPEqualizer
lib = _lib.load()
M = int(os.environ.get("M_EST", 25))
B = int(os.environ["B_SYMS"]) if "B_SYMS" in os.environ else 1 << int(os.environ.get("LOG2B", 22))
h_est, h_ch, P, amp, amps, pol, nu_sc, var, pow_mean = init("h0", "64-QAM", "cpu", 0.0270955, 2, M, 23)
rxs = [generate_data_gpu(B, amps, 23, P, 2, np.pi / 10, "cuda", 1 + i)[0] for i in range(3)]
q = torch.empty(2, 16, B, device="cuda"); out = torch.empty(2, 2, B, device="cuda")
NK = 11
for tc in [int(a) for a in (sys.argv[1:] or ["1", "0"])]:             # 1: tensor-core tap gradients, 0: the two CUDA-core kernels
    _lib.check(lib.vaeq_dp_tc_taps(tc))
    lib.vaeq_dp_tc_forward(int(os.environ.get('TC_FWD', 1)))
    eq = DPEqualizer(M, 2, amp, P, var, nu_sc)
    for i in range(4):
        eq.train_step(rxs[i % 3], 2.5e-3, 2.5e-3, q=q, out=out)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n = 30
    a.record()
    for i in range(n):
        eq.train_step(rxs[i % 3], 2.5e-3, 2.5e-3, q=q, out=out)
    b.record(); torch.cuda.synchronize()
    plain = a.elapsed_time(b) / n
    lib.vaeq_kernel_timing(1)
    for i in range(n):
        eq.train_step(rxs[i % 3], 2.5e-3, 2.5e-3, q=q, out=out)
    torch.cuda.synchronize()
    ms = (C.c_float * NK)(); cnt = (C.c_int32 * NK)()
    lib.vaeq_kernel_timing_read(ms, cnt)
    lib.vaeq_kernel_timing(0)
    per = {k: ms[k] / cnt[k] * 1e3 for k in range(NK) if cnt[k]}
    print(f"tensor-core taps {tc}: step {plain * 1e3:.1f} us plain launches ({B / plain / 1e6:.2f} G symbols/s); kernels (us, by kind id): "
          + ", ".join(f"{k}: {v:.1f}" for k, v in per.items()) + f"; loss {float(eq.loss):.6g}")
lib.vaeq_dp_tc_taps(1)
lib.vaeq_dp_tc_forward(1)
