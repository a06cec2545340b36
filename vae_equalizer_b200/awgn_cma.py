"""B200 implementation of the operator surface of the reference's AWGN CMA module
(`AWGN_channel/func_CMA_MQAM_shaping.py`, cited `cm:`): CMA :142-168, CPE :170-196, SER_CMA :63-93, find_shift_symb :127-140.

Same names, argument order and mutation conventions as the reference: CMA updates `h` in place and returns it, SER_CMA rescales its
`rx` argument in place (cm:73).  Single polarisation: Rx (2,N) [I, Q], h (2,M) = real / imaginary taps.  CUDA tensors only."""
from __future__ import annotations

import torch

from . import _lib

_F32 = torch.float32


def _need(t, name, dtype=_F32):
    if not t.is_cuda:
        raise _lib.VaeqError(f"{name} must be a CUDA tensor: vae_equalizer_b200 has no CPU path")
    if t.dtype != dtype:
        raise _lib.VaeqError(f"{name} must be {dtype}, got {t.dtype}")
    _lib.require_current_device(t, name)


@_lib.device_guard
def CMA(Rx, R, h, lr, sps, eval):
    """Constant-modulus algorithm, complex FIR, tap update after every symbol (cm:142-168); `eval` True = train (sic).
    Rx (2,N) with h (2,M), or S independent streams: Rx (S,2,N) with h (S,2,M).  Returns (out, h, e)."""
    _need(Rx, "Rx")
    _need(h, "h")
    if not (Rx.is_contiguous() and h.is_contiguous()):
        raise _lib.VaeqError("CMA: Rx and h must be contiguous")
    batched = Rx.dim() == 3
    if (batched and (h.dim() != 3 or h.shape[0] != Rx.shape[0])) or (not batched and (Rx.dim() != 2 or h.dim() != 2)) or Rx.shape[-2] != 2:
        raise _lib.VaeqError(f"CMA: need Rx (2,N) with h (2,M) or Rx (S,2,N) with h (S,2,M), got {tuple(Rx.shape)} {tuple(h.shape)}")
    lib = _lib.load()
    S = int(Rx.shape[0]) if batched else 1
    N, M = int(Rx.shape[-1]), int(h.shape[-1])
    out = torch.zeros((S, 2, N // sps) if batched else (2, N // sps), dtype=_F32, device=Rx.device)
    e = torch.empty((S, N // sps) if batched else (N // sps,), dtype=_F32, device=Rx.device)
    _lib.check(lib.vaeq_cma_awgn(Rx.data_ptr(), N, float(R), h.detach().data_ptr(), M, float(lr), int(sps), 1 if eval else 0, out.data_ptr(),
                                 e.data_ptr(), S, _lib.current_stream()), "vaeq_cma_awgn")
    return out, h, e


@_lib.device_guard
def CPE(y):
    """Viterbi-Viterbi carrier phase estimation WITHOUT unwrapping (cm:170-196); y (2,N), or (S,2,N) for S independent runs."""
    _need(y, "y")
    lib = _lib.load()
    y = y.contiguous()
    N = int(y.shape[-1])
    S = int(y.shape[0]) if y.dim() == 3 else 1
    out = torch.empty_like(y)
    scr = torch.empty(int(lib.vaeq_cpe_runs_scratch_bytes(N, S)), dtype=torch.uint8, device=y.device)
    _lib.check(lib.vaeq_cpe_awgn(y.data_ptr(), N, S, out.data_ptr(), scr.data_ptr(), _lib.current_stream()), "vaeq_cpe_awgn")
    return out


def _rows2(t, name):
    if t.dim() != 2 or t.shape[0] != 2 or t.stride(1) != 1:
        raise _lib.VaeqError(f"{name}: need (2,N) with unit time stride, got {tuple(t.shape)} strides {t.stride()}")
    return int(t.stride(0))


@_lib.device_guard
def SER_CMA(rx, tx, sps, amp_levels, num_lev, device=None, return_counts=False):
    """SER from nearest-level decisions, min over the 4 rotations (cm:63-93).  Rescales `rx` IN PLACE (cm:73).  Returns a 0-dim
    float32 tensor (and the int32 error counts (4,) with return_counts)."""
    _need(rx, "rx")
    _need(tx, "tx", torch.float16)
    lib = _lib.load()
    N = int(tx.shape[1])
    if rx.shape[1] != N:
        raise _lib.VaeqError(f"SER_CMA: rx has {rx.shape[1]} symbols, tx {N}")
    amp = amp_levels.to(rx.device, _F32).contiguous()
    counts = torch.empty(4, dtype=torch.int32, device=rx.device)
    ser = torch.empty(1, dtype=_F32, device=rx.device)
    scr = torch.empty(1 << 16, dtype=torch.uint8, device=rx.device)
    _lib.check(lib.vaeq_ser_cma(rx.data_ptr(), _rows2(rx, "rx"), tx.data_ptr(), _rows2(tx, "tx"), amp.data_ptr(), int(amp.numel()), N,
                                counts.data_ptr(), ser.data_ptr(), scr.data_ptr(), _lib.current_stream()), "vaeq_ser_cma")
    return (ser[0], counts) if return_counts else ser[0]


@_lib.device_guard
def find_shift_symb(rx, tx, N_shift, return_corr=False):
    """Time alignment from the first 1000 symbols (cm:127-140): non-circular correlation of tx I (Q as the fallback) with rx I over
    N_shift lags.  Returns the shift as a 0-dim int64 tensor like the reference (`argmax - N_shift//2`)."""
    _need(rx, "rx")
    _need(tx, "tx", torch.float16)
    lib = _lib.load()
    corr = torch.empty(2, N_shift, dtype=_F32, device=rx.device)
    shift = torch.empty(1, dtype=torch.int32, device=rx.device)
    _rows2(rx, "rx")
    _lib.check(lib.vaeq_find_shift_symb(rx.data_ptr(), int(rx.shape[-1]), tx.data_ptr(), _rows2(tx, "tx"), int(tx.shape[-1]), int(N_shift),
                                        corr.data_ptr(), shift.data_ptr(), _lib.current_stream()), "vaeq_find_shift_symb")
    s = shift[0].to(torch.int64)
    return (s, corr) if return_corr else s


@_lib.device_guard
def CMA_runs(rx_train, rx_valid, h, lr, sps, R=1.0):
    """A validation period of processing_cma_awgn for R_runs runs in one launch (one warp per run): CMA with updates over the F training
    frames rx_train (R_runs, F, 2, sps*N_train) in order, then without updates over rx_valid (R_runs, 2, sps*N_valid).  h (R_runs, 2, M)
    is updated in place; lr (R_runs,) is each run's learning rate, used as the fp32 value CMA(..., lr, ...) passes.  Run k equals F calls
    CMA(rx_train[k, f], R, h[k], lr[k], sps, True) followed by CMA(rx_valid[k], R, h[k], lr[k], sps, False), bit for bit.  F may be 0.
    Returns out_v (R_runs, 2, N_valid); the training frames' outputs and errors are not produced."""
    _need(rx_train, "rx_train")
    _need(rx_valid, "rx_valid")
    _need(h, "h")
    _need(lr, "lr")
    if rx_train.dim() != 4 or rx_valid.dim() != 3 or h.dim() != 3 or rx_train.shape[2] != 2 or rx_valid.shape[1] != 2 or h.shape[1] != 2:
        raise _lib.VaeqError(f"CMA_runs: need rx_train (R,F,2,L), rx_valid (R,2,L) and h (R,2,M), got {tuple(rx_train.shape)} "
                             f"{tuple(rx_valid.shape)} {tuple(h.shape)}")
    n = int(h.shape[0])
    if rx_train.shape[0] != n or rx_valid.shape[0] != n or lr.shape != (n,):
        raise _lib.VaeqError(f"CMA_runs: {n} runs in h, but rx_train {tuple(rx_train.shape)}, rx_valid {tuple(rx_valid.shape)}, "
                             f"lr {tuple(lr.shape)}")
    if rx_train.stride(3) != 1 or rx_valid.stride(2) != 1 or not h.is_contiguous() or not lr.is_contiguous():
        raise _lib.VaeqError("CMA_runs: rx needs unit sample stride, h and lr must be contiguous")
    lib = _lib.load()
    F, Nt, Nv, M = int(rx_train.shape[1]), int(rx_train.shape[3]), int(rx_valid.shape[2]), int(h.shape[2])
    out_v = torch.zeros(n, 2, Nv // sps, dtype=_F32, device=h.device)
    _lib.check(lib.vaeq_cma_awgn_runs(rx_train.data_ptr(), int(rx_train.stride(2)), int(rx_train.stride(1)), int(rx_train.stride(0)), F, Nt,
                                      rx_valid.data_ptr(), int(rx_valid.stride(1)), int(rx_valid.stride(0)), Nv, h.detach().data_ptr(), M,
                                      lr.data_ptr(), float(R), int(sps), out_v.data_ptr(), n, _lib.current_stream()), "vaeq_cma_awgn_runs")
    return out_v


@_lib.device_guard
def awgn_cma_eval_runs(out_cpe, tx, amp_levels, n_shift=21, edge=11):
    """The validation lines of processing_cma_awgn (cm:227-229) for R runs without a host sync: per run
    shift = find_shift_symb(out_cpe, tx, n_shift), then SER_CMA(out_cpe[:, edge+shift : -edge], tx[:, edge : -edge-shift]).
    out_cpe (R, 2, N) float32, tx (R, 2, N) float16.  out_cpe is not modified (the single-run SER_CMA rescales its slice in place).
    Returns shift (R,) int32, counts (R, 4) int32 (rotations 0, pi and the two quarter turns) and ser (R,) float32, on the device."""
    _need(out_cpe, "out_cpe")
    _need(tx, "tx", torch.float16)
    if out_cpe.dim() != 3 or tx.dim() != 3 or out_cpe.shape[1] != 2 or tx.shape != out_cpe.shape or out_cpe.stride(2) != 1 or tx.stride(2) != 1:
        raise _lib.VaeqError(f"awgn_cma_eval_runs: need out_cpe and tx (R,2,N) with unit time stride, got {tuple(out_cpe.shape)} "
                             f"{tuple(tx.shape)}")
    lib = _lib.load()
    R, N = int(out_cpe.shape[0]), int(out_cpe.shape[2])
    dev = out_cpe.device
    amp = amp_levels.to(dev, _F32).contiguous() if torch.is_tensor(amp_levels) else torch.as_tensor(amp_levels, dtype=_F32, device=dev)
    shift = torch.empty(R, dtype=torch.int32, device=dev)
    counts = torch.empty(R, 4, dtype=torch.int32, device=dev)
    ser = torch.empty(R, dtype=_F32, device=dev)
    scr = torch.empty(max(1, int(lib.vaeq_awgn_cma_eval_scratch_bytes(R, N, int(n_shift), int(edge)))), dtype=torch.uint8, device=dev)
    _lib.check(lib.vaeq_awgn_cma_eval_runs(out_cpe.data_ptr(), int(out_cpe.stride(1)), int(out_cpe.stride(0)), tx.data_ptr(), int(tx.stride(1)),
                                           int(tx.stride(0)), amp.data_ptr(), int(amp.numel()), N, int(n_shift), int(edge), R,
                                           shift.data_ptr(), counts.data_ptr(), ser.data_ptr(), scr.data_ptr(), _lib.current_stream()),
               "vaeq_awgn_cma_eval_runs")
    return shift, counts, ser
