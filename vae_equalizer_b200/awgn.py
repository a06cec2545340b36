"""Host-side owners of AWGN single-polarisation VAE-LE runs (reference: AWGN_channel/func_VAELE_MQAM_shaping.py, twoFIR :206-231,
loss_function :63-95, Adam(amsgrad) :283-286): one run (AWGNEqualizer) or R independent runs stepped together (AWGNEqualizerRuns),
the batched validation scoring (awgn_eval_runs) and the on-device signal generator (generate_frames_awgn_gpu)."""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from .datagen import PULSE_SPAN, ROLLOFF, composite_filter, rrcfir

_F32 = torch.float32


class AWGNEqualizer:
    def __init__(self, M_est, sps, amp_levels, P, amp_mean, var, device="cuda", W0=None, h0=None):
        self.lib = _lib.load()
        dev = torch.device(device)
        if dev.type != "cuda":
            raise _lib.VaeqError("AWGNEqualizer needs a CUDA device: there is no CPU path")
        self.device, self.M, self.sps = dev, int(M_est), int(sps)
        self.amp = torch.as_tensor(amp_levels, dtype=_F32).to(dev).contiguous()
        self.P = torch.as_tensor(P, dtype=_F32).to(dev).contiguous()
        self.n_lev = int(self.amp.numel())
        self.amp_mean, self.var = float(amp_mean), float(var)
        M = self.M
        if W0 is None:
            W0 = torch.zeros(1, 2, M, dtype=_F32)
            W0[0, 0, M // 2] = 1.0                         # nn.init.dirac_ on Conv1d(2,1,M)  (:210)
        if h0 is None:
            h0 = torch.zeros(2, M, dtype=_F32)
            h0[0, M // 2] = 1.0                            # :279
        self.W = torch.as_tensor(W0, dtype=_F32).detach().clone().to(dev).contiguous()
        self.h = torch.as_tensor(h0, dtype=_F32).detach().clone().to(dev).contiguous()
        self.adam = torch.zeros(int(self.lib.vaeq_adam_state_floats_awgn(M)), dtype=_F32, device=dev)
        self.gW = torch.zeros(1, 2, M, dtype=_F32, device=dev)
        self.gh = torch.zeros(2, M, dtype=_F32, device=dev)
        self.loss = torch.zeros(1, dtype=_F32, device=dev)
        self._ws, self._ws_B = None, -1

    def _desc(self, rx, q, out, B):
        if not rx.is_cuda or rx.dtype != _F32 or not rx.is_contiguous() or rx.dim() != 2 or rx.shape[0] != 2:
            raise _lib.VaeqError("rx must be a contiguous float32 CUDA tensor of shape (2, L)")
        if self._ws is None or self._ws_B < B:
            self._ws = torch.empty(int(self.lib.vaeq_awgn_workspace_bytes(B, self.M, self.n_lev)), dtype=torch.uint8, device=self.device)
            self._ws_B = B
        d = _lib.AwgnDesc()
        d.B, d.sps, d.M, d.n_lev = B, self.sps, self.M, self.n_lev
        d.amp_mean, d.var = self.amp_mean, self.var
        d.rx, d.amp, d.P = rx.data_ptr(), self.amp.data_ptr(), self.P.data_ptr()
        d.W, d.h, d.adam = self.W.data_ptr(), self.h.data_ptr(), self.adam.data_ptr()
        d.q, d.out, d.loss = q.data_ptr(), out.data_ptr(), self.loss.data_ptr()
        d.gW, d.gh = self.gW.data_ptr(), self.gh.data_ptr()
        d.workspace, d.workspace_bytes = self._ws.data_ptr(), self._ws.numel()
        return d

    @_lib.device_guard
    def _run(self, fn, name, rx, *extra):
        B = rx.shape[-1] // self.sps
        q = torch.empty(2 * self.n_lev, B, dtype=_F32, device=self.device)
        out = torch.empty(2, B, dtype=_F32, device=self.device)
        d = self._desc(rx, q, out, B)
        _lib.check(fn(C.byref(d), *extra, _lib.current_stream()), name)
        return q, out

    def forward(self, rx):
        q, out = self._run(self.lib.vaeq_awgn_forward, "vaeq_awgn_forward", rx)
        return q, out, self.loss

    def forward_backward(self, rx):
        q, out = self._run(self.lib.vaeq_awgn_forward_backward, "vaeq_awgn_forward_backward", rx)
        return q, out, self.loss, self.gW, self.gh

    def train_step(self, rx, lr_w, lr_h=None):
        lr_h = lr_w if lr_h is None else lr_h
        q, out = self._run(self.lib.vaeq_awgn_train_step, "vaeq_awgn_train_step", rx, C.c_float(lr_w), C.c_float(lr_h))
        return q, out, self.loss


def generate_data(N, M, amps, SNR, h_channel, sps, device, P, rng=None):
    """Single-polarisation test signal (reference generate_data, func_VAELE_MQAM_shaping.py:39-61)."""
    rng = np.random.default_rng() if rng is None else rng
    n_conv = N + len(h_channel) + 4 * PULSE_SPAN
    data = rng.choice(amps, (2, n_conv), p=P)
    up = np.zeros(sps * (n_conv - 1) + 1, dtype=np.complex64)
    up[::sps] = data[0] + 1j * data[1]
    sig = np.convolve(np.convolve(up, rrcfir(PULSE_SPAN, sps, ROLLOFF), mode="valid"), h_channel, mode="valid")
    sigma_n = np.sqrt(sps * np.mean(np.abs(sig) ** 2) / 2 / 10 ** (SNR / 10))
    sig = sig + sigma_n * (rng.standard_normal(sig.shape) + 1j * rng.standard_normal(sig.shape))
    rx = torch.from_numpy(np.stack((sig[:sps * N].real, sig[:sps * N].imag)).astype(np.float32)).to(device)
    sl = slice(PULSE_SPAN + M - 1, N + PULSE_SPAN + M - 1)
    tx = torch.from_numpy(np.stack((data[0, sl], data[1, sl]))).to(device, torch.float16)
    return rx.contiguous(), tx.contiguous()


def _need_cuda(t, name):
    if not (torch.is_tensor(t) and t.is_cuda):
        raise _lib.VaeqError(f"{name} must be a CUDA tensor: there is no CPU path")


class AWGNEqualizerRuns:
    """R independent AWGN VAE-LE runs (taps, Adam state, workspaces), trained and evaluated in one launch each: run k behaves bit for bit
    like an AWGNEqualizer with P[k], amp_mean[k], var[k] that is stepped with lr[k] for both parameter groups."""

    def __init__(self, R, M_est, sps, amp_levels, P, amp_mean, var, device="cuda"):
        dev = torch.device(device)
        if dev.type != "cuda":
            raise _lib.VaeqError("AWGNEqualizerRuns needs a CUDA device: there is no CPU path")
        self.lib = _lib.load()
        if dev.index is None:
            dev = torch.device("cuda", torch.cuda.current_device())
        self.R, self.M, self.sps, self.device = int(R), int(M_est), int(sps), dev
        self.amp = torch.as_tensor(amp_levels, dtype=_F32).to(dev).contiguous()
        self.n_lev = int(self.amp.numel())
        self.P = torch.as_tensor(P, dtype=_F32).to(dev).reshape(self.R, self.n_lev).contiguous()
        self.amp_mean = torch.as_tensor(amp_mean, dtype=_F32).to(dev).reshape(self.R).contiguous()
        self.var = torch.as_tensor(var, dtype=_F32).to(dev).reshape(self.R).contiguous()
        M = self.M
        self.W = torch.zeros(self.R, 1, 2, M, dtype=_F32, device=dev)
        self.W[:, 0, 0, M // 2] = 1.0                                  # nn.init.dirac_  (:210)
        self.h = torch.zeros(self.R, 2, M, dtype=_F32, device=dev)
        self.h[:, 0, M // 2] = 1.0                                     # :279
        self.adam = torch.zeros(self.R, int(self.lib.vaeq_adam_state_floats_awgn(M)), dtype=_F32, device=dev)
        self._ws, self._q, self._out = {}, {}, {}

    def _buffers(self, B):
        if B not in self._ws:
            self._ws[B] = torch.empty(int(self.lib.vaeq_awgn_runs_workspace_bytes(B, self.M, self.n_lev, self.R)), dtype=torch.uint8, device=self.device)
        return self._ws[B]

    def _call(self, fn, name, rx, B, q, out, loss, lr, *extra):
        ws = self._buffers(B)
        d = _lib.AwgnDesc()
        d.B, d.sps, d.M, d.n_lev = B, self.sps, self.M, self.n_lev
        d.rx, d.amp, d.P = rx.data_ptr(), self.amp.data_ptr(), self.P.data_ptr()
        d.W, d.h, d.adam = self.W.data_ptr(), self.h.data_ptr(), self.adam.data_ptr()
        d.q, d.out, d.loss = q.data_ptr(), out.data_ptr(), loss.data_ptr()
        d.workspace, d.workspace_bytes = ws.data_ptr(), ws.numel()
        r = _lib.AwgnRuns()
        r.n_runs = self.R
        r.rs_rx, r.rs_W, r.rs_h, r.rs_adam, r.rs_P = int(rx.stride(0)), 2 * self.M, 2 * self.M, int(self.adam.stride(0)), self.n_lev
        r.rs_q, r.rs_out, r.rs_loss = int(q.stride(0)), int(out.stride(0)), int(loss.stride(0))
        r.lr = None if lr is None else lr.data_ptr()
        r.var, r.amp_mean = self.var.data_ptr(), self.amp_mean.data_ptr()
        _lib.check(fn(C.byref(d), C.byref(r), int(rx.stride(-2)), *extra, _lib.current_stream()), name)

    def _check_rx(self, rx, dims):
        _need_cuda(rx, "rx")
        if rx.dtype != _F32 or rx.dim() != dims or rx.shape[0] != self.R or rx.shape[-2] != 2 or rx.stride(-1) != 1:
            raise _lib.VaeqError(f"rx must be float32 ({self.R}, {'F, ' if dims == 4 else ''}2, L) with unit sample stride, got "
                                 f"{tuple(rx.shape)} {rx.dtype}")
        if rx.device != self.device:
            raise _lib.VaeqError(f"rx lives on {rx.device}, the runs on {self.device}")

    @_lib.device_guard
    def train_frames(self, rx, lr, batch_len, N_train=None):
        """The epoch loop of :291-306 over rx (R, F, 2, sps*N_train): per frame N_train // batch_len minibatches of batch_len symbols (the
        rest of the frame is unused), every run with its own lr (R,) for both parameter groups.  Returns the loss of every step (R, F*m)."""
        self._check_rx(rx, 4)
        N_train = rx.shape[-1] // self.sps if N_train is None else int(N_train)
        B, F, n_mb = int(batch_len), int(rx.shape[1]), int(N_train) // int(batch_len)
        if n_mb < 1 or self.sps * N_train > rx.shape[-1]:
            raise _lib.VaeqError(f"a frame of {rx.shape[-1]} samples holds no minibatch of {B} symbols (N_train={N_train})")
        lr = torch.as_tensor(lr, dtype=_F32).to(self.device).reshape(-1).expand(self.R).contiguous()
        q = torch.empty(self.R, 2 * self.n_lev, B, dtype=_F32, device=self.device)
        out = torch.empty(self.R, 2, B, dtype=_F32, device=self.device)
        loss = torch.empty(self.R, F * n_mb, dtype=_F32, device=self.device)
        self._call(self.lib.vaeq_awgn_train_frames_runs, "vaeq_awgn_train_frames_runs", rx, B, q, out, loss, lr, int(rx.stride(1)), F, n_mb)
        return loss

    @_lib.device_guard
    def forward(self, rx):
        """Forward of every run over rx (R, 2, sps*B): q (R, 2n, B), out (R, 2, B), loss (R,)."""
        self._check_rx(rx, 3)
        B = int(rx.shape[-1]) // self.sps
        q = torch.empty(self.R, 2 * self.n_lev, B, dtype=_F32, device=self.device)
        out = torch.empty(self.R, 2, B, dtype=_F32, device=self.device)
        loss = torch.empty(self.R, 1, dtype=_F32, device=self.device)
        self._call(self.lib.vaeq_awgn_forward_runs, "vaeq_awgn_forward_runs", rx, B, q, out, loss, None)
        return q, out, loss[:, 0]


@_lib.device_guard
def awgn_eval_runs(q, tx, amp_levels, n_shift=21, n_corr=1000, edge=11):
    """processing.awgn_find_shift + awgn_ser_q (:188-204, :97-124) for R runs without a host sync: q (R, 2n, N), tx (R, 2, N) float16.
    Returns shift (R,) int32, counts (R, 4) int32 (rotations 0, pi, pi/2, 3pi/2) and ser (R,) float32, all on the device."""
    _need_cuda(q, "q")
    _need_cuda(tx, "tx")
    if tx.dtype != torch.float16:
        raise _lib.VaeqError(f"tx must be float16, got {tx.dtype}")
    if q.dim() != 3 or tx.dim() != 3 or tx.shape[0] != q.shape[0] or tx.shape[1] != 2 or tx.shape[-1] != q.shape[-1] or q.stride(2) != 1 or tx.stride(2) != 1:
        raise _lib.VaeqError(f"need q (R,2n,N) and tx (R,2,N) with unit time stride, got {tuple(q.shape)} {tuple(tx.shape)}")
    lib = _lib.load()
    R, N, n = int(q.shape[0]), int(q.shape[-1]), int(q.shape[1]) // 2
    dev = q.device
    shift = torch.empty(R, dtype=torch.int32, device=dev)
    counts = torch.empty(R, 4, dtype=torch.int32, device=dev)
    ser = torch.empty(R, dtype=_F32, device=dev)
    n_corr = min(int(n_corr), N)                                   # q[:, :1000] of a shorter frame is the whole frame
    scr = torch.empty(int(lib.vaeq_awgn_eval_scratch_bytes(R, int(n_shift), n_corr)), dtype=torch.uint8, device=dev)
    amp = torch.as_tensor(amp_levels, dtype=_F32).to(dev).contiguous()
    _lib.check(lib.vaeq_awgn_eval_runs(q.data_ptr(), int(q.stride(1)), int(q.stride(0)), tx.data_ptr(), int(tx.stride(1)), int(tx.stride(0)),
                                       amp.data_ptr(), n, N, int(n_shift), n_corr, int(edge), R, shift.data_ptr(), counts.data_ptr(),
                                       ser.data_ptr(), scr.data_ptr(), _lib.current_stream()), "vaeq_awgn_eval_runs")
    return shift, counts, ser


def awgn_gmi_runs(q, tx, P, shift, counts, edge=11):
    """EXTENSION (not in the reference): GMI = H(X) + mean log2 q(x_tx|y) (bit/2D-symbol) of R runs on exactly the symbols awgn_eval_runs
    scores (q[:, edge+shift : N-edge] against tx[:, edge : N-edge-shift]) under its best rotation: q (R,2n,N), tx (R,2,N) float16, P (R,n)
    or (n,) pmf, shift (R,) and counts (R,4) int32 from awgn_eval_runs with the same edge.  Returns (R,) float32 on the device; no host sync."""
    return _awgn_rate_runs("vaeq_awgn_gmi_runs", q, tx, P, shift, counts, edge)


def awgn_bmi_runs(q, tx, P, shift, counts, edge=11):
    """EXTENSION (not in the reference): the bit-metric decoding rate of Gray-labelled bits (BMI, DESIGN.md §2) of R runs, bit/2D-symbol.
    Arguments, symbols, rotation and result exactly as awgn_gmi_runs."""
    return _awgn_rate_runs("vaeq_awgn_bmi_runs", q, tx, P, shift, counts, edge)


@_lib.device_guard
def _awgn_rate_runs(fn, q, tx, P, shift, counts, edge):
    """awgn_gmi_runs / awgn_bmi_runs through the C entry `fn` (vaeq_awgn_gmi_runs or vaeq_awgn_bmi_runs: same arguments)."""
    from .dp import _require_cuda
    from .shared_funcs import _run_pmf
    _need_cuda(q, "q")
    _require_cuda(q, "q")                                          # float32 posteriors, on the call's device
    _need_cuda(tx, "tx")
    if tx.dtype != torch.float16:
        raise _lib.VaeqError(f"tx must be float16, got {tx.dtype}")
    if q.dim() != 3 or tx.dim() != 3 or tx.shape[0] != q.shape[0] or tx.shape[1] != 2 or tx.shape[-1] != q.shape[-1] or q.stride(2) != 1 or tx.stride(2) != 1:
        raise _lib.VaeqError(f"need q (R,2n,N) and tx (R,2,N) with unit time stride, got {tuple(q.shape)} {tuple(tx.shape)}")
    lib = _lib.load()
    R, N, n = int(q.shape[0]), int(q.shape[-1]), int(q.shape[1]) // 2
    dev = q.device
    for t, name, shape in ((shift, "shift", (R,)), (counts, "counts", (R, 4))):
        if not torch.is_tensor(t) or t.dtype != torch.int32 or tuple(t.shape) != shape or not t.is_contiguous() or t.device != dev:
            raise _lib.VaeqError(f"{name}: need a contiguous int32 {shape} tensor on {dev} (awgn_eval_runs)")
    Pt, rs_P = _run_pmf(P, R, n, dev)
    rate = torch.empty(R, dtype=_F32, device=dev)
    scr = torch.empty(max(1, int(lib.vaeq_awgn_gmi_scratch_bytes(R, N))), dtype=torch.uint8, device=dev)
    _lib.check(getattr(lib, fn)(q.data_ptr(), int(q.stride(1)), int(q.stride(0)), tx.data_ptr(), int(tx.stride(1)), int(tx.stride(0)),
                                Pt.data_ptr(), rs_P, shift.data_ptr(), counts.data_ptr(), n, N, R, int(edge), rate.data_ptr(), scr.data_ptr(),
                                _lib.current_stream()), fn)
    return rate


_TAPS_CACHE: dict = {}


def _composite_taps(h_channel, sps, dev):
    """rrcfir (*) h_channel as interleaved (re, im) float32 on the device: one 'valid' FIR for the two of generate_data (:52-53)."""
    key = (np.asarray(h_channel, dtype=np.complex64).tobytes(), sps, str(dev))
    if key not in _TAPS_CACHE:
        g = composite_filter(h_channel, sps)
        _TAPS_CACHE[key] = torch.as_tensor(np.stack((g.real, g.imag), -1).astype(np.float32).reshape(-1), device=dev)
    return _TAPS_CACHE[key]


@_lib.device_guard
def generate_frames_awgn_gpu(N, amps, SNR, P, h_channel, sps, device, seeds, frame0=0, n_frames=1, return_parts=False):
    """generate_data (:39-61) on the device for R runs x n_frames frames: SNR (R,), P (R, n), seeds (R,) integers, one per run; frame
    indices frame0 .. frame0 + n_frames - 1.  A run's frames depend only on its seed and the frame index.  Returns rx (R, F, 2, sps*N)
    float32 and tx (R, F, 2, N) float16 (tx = the levels [PULSE_SPAN + M - 1, N + PULSE_SPAN + M - 1), M = symbol-rate channel
    length); with return_parts also the levels (R, F, 2, n_conv) and the noise-free signal (R, F, 2 n_conv - K) complex64."""
    dev = torch.device(device)
    if dev.type != "cuda":
        raise _lib.VaeqError("generate_frames_awgn_gpu needs a CUDA device: there is no CPU path")
    if sps != 2:
        raise _lib.VaeqError(f"sps={sps}: the device generator implements sps=2")
    lib = _lib.load()
    P = torch.as_tensor(np.asarray(P) if not torch.is_tensor(P) else P, dtype=_F32).to(dev)
    P = (P[None] if P.dim() == 1 else P).contiguous()
    R, n_lev, F = int(P.shape[0]), int(P.shape[1]), int(n_frames)
    snr = torch.as_tensor(SNR, dtype=_F32).to(dev).reshape(-1).expand(R).contiguous()
    sd = torch.as_tensor(np.asarray(seeds, dtype=np.uint64).astype(np.int64).reshape(R), device=dev)
    taps = _composite_taps(h_channel, sps, dev)
    K = taps.numel() // 2
    M = (len(h_channel) - 1) // sps + 1
    n_conv = N + len(h_channel) + 4 * PULSE_SPAN                  # :42
    amps_t = torch.as_tensor(np.asarray(amps, dtype=np.float32), device=dev)
    lev = torch.empty(R, F, 2, n_conv, dtype=_F32, device=dev)
    sig = torch.empty(R, F, 2 * n_conv - K, dtype=torch.complex64, device=dev)
    rx = torch.empty(R, F, 2, sps * N, dtype=_F32, device=dev)
    tx = torch.empty(R, F, 2, N, dtype=torch.float16, device=dev)
    _lib.check(lib.vaeq_gen_awgn(amps_t.data_ptr(), P.data_ptr(), n_lev, taps.data_ptr(), K, int(N), PULSE_SPAN + M - 1, n_conv, snr.data_ptr(),
                                 sd.data_ptr(), int(frame0), F, R, lev.data_ptr(), sig.data_ptr(), rx.data_ptr(), tx.data_ptr(),
                                 _lib.current_stream()), "vaeq_gen_awgn")
    return (rx, tx, lev, sig) if return_parts else (rx, tx)
