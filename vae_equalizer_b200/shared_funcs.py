"""B200 implementation of the reference's operator surface `optical_DP_channel/shared_funcs.py`.

Same names, argument order and return conventions as the reference (cited per function, `sf:` =
optical_DP_channel/shared_funcs.py); every tensor argument must live on a CUDA device and every
function enqueues hand-written sm_100a kernels from libvaeq.so on the current torch stream.  There is
no CPU path: CPU tensors raise VaeqError.

Mutation conventions kept from the reference: CMA* update `h` in place and return it (sf:370-379),
SER_constell_shaping rescales its `rx` argument in place (sf:242).
"""
from __future__ import annotations

import ctypes as C
import weakref

import numpy as np
import torch

from . import _lib
from .constants import init  # noqa: F401  (sf:544-588, host-side constants)
from .datagen import generate_data_shaping, rcfir, rrcfir, simulate_channel, simulate_dispersion  # noqa: F401
from .dp import DPEqualizer, _require_cuda

_F32 = torch.float32
EVAL_SCRATCH_BYTES = 1 << 16

def _rows(t: torch.Tensor, name: str):
    """Check the (2, R, N) row-major-with-stride layout the C ABI takes and return the row stride."""
    if t.dim() != 3 or t.stride(2) != 1 or t.stride(0) != t.shape[1] * t.stride(1):
        raise _lib.VaeqError(f"{name}: need (2,R,N) with unit time stride and evenly strided rows, got shape "
                             f"{tuple(t.shape)} strides {t.stride()}")
    return int(t.stride(1))


def _scratch(dev, nbytes=EVAL_SCRATCH_BYTES):
    return torch.empty(nbytes, dtype=torch.uint8, device=dev)


def _tx_bits(tx: torch.Tensor):
    if tx.dtype != torch.float16:
        raise _lib.VaeqError(f"tx must be float16 like the reference's data_tensor (sf:89), got {tx.dtype}")
    if not tx.is_cuda:
        raise _lib.VaeqError("tx must be a CUDA tensor")
    return tx


# -------------------------------------------------------------------------------------------------
# equalizer + demapper                                                         sf:490-542
# -------------------------------------------------------------------------------------------------
class _TapHolder(torch.nn.Module):
    """Stands in for the reference's nn.Conv1d so that `net.conv_w.weight` and `net.parameters()` work."""

    def __init__(self, M_est):
        super().__init__()
        w = torch.zeros(2, 4, M_est, dtype=_F32)
        w[0, 0, M_est // 2] = 1.0                      # nn.init.dirac_  (sf:495)
        w[1, 1, M_est // 2] = 1.0
        self.weight = torch.nn.Parameter(w)


class _FusedLoss(torch.autograd.Function):
    """loss as a function of (W, h_est); gradients come from the fused CUDA backward."""

    @staticmethod
    def forward(ctx, W, h, eq, rx):
        eq.W.copy_(W.detach())
        eq.h.copy_(h.detach())
        q, out, loss, var_est, gW, gh = eq.forward_backward(rx)
        ctx.save_for_backward(gW.clone(), gh.clone())
        ctx.mark_non_differentiable(var_est)
        return loss.reshape(()).clone(), var_est.clone()

    @staticmethod
    def backward(ctx, g_loss, _g_var):
        gW, gh = ctx.saved_tensors
        return g_loss * gW, g_loss * gh, None, None


class twoXtwoFIR(torch.nn.Module):
    """Complex-valued 2x2 butterfly FIR + soft demapper (sf:490-527).

    forward(x, amp_levels, var, nu_sc) -> (q_est (2,2n,N), out (2,2,N)), outputs of one autograd node (_EqualizerFn).
    loss_function_shaping(q, x, h_est, ...) recognises an unmodified q of that node and runs the fused forward+backward
    kernels, handing gradients for `conv_w.weight` and `h_est` to autograd without materialising dL/dq."""

    def __init__(self, M_est, sps):
        super().__init__()
        self.M_est, self.sps = int(M_est), int(sps)
        self.conv_w = _TapHolder(M_est)
        self._eq = None

    def _engine(self, amp_levels, var, nu_sc, P=None):
        """ONE DPEqualizer per (amp_levels, var, nu_sc): forward() needs no prior, loss_function_shaping() sets it in place, so the two
        calls of a minibatch share the engine (and its workspace) instead of rebuilding it twice per step."""
        dev = self.conv_w.weight.device
        key = (amp_levels.data_ptr(), amp_levels._version, var.data_ptr(), var._version, float(nu_sc))
        if self._eq is None or self._eq_key != key:
            n = amp_levels.numel()
            self._eq = DPEqualizer(self.M_est, self.sps, amp_levels, torch.full((n,), 1.0 / n, dtype=_F32), var, float(nu_sc), device=dev)
            self._eq_key = key
        if P is not None:
            self._eq.P.copy_(P.reshape(-1))
        return self._eq

    def forward(self, x, amp_levels, var, nu_sc):
        _require_cuda(x, "x")
        return _EqualizerFn.apply(self.conv_w.weight, x.contiguous(), self, amp_levels, var, float(nu_sc))


class _EqualizerFn(torch.autograd.Function):
    """net(x) = (q, out) as an autograd node.  loss_function_shaping recognises an unmodified q of this node (also through views such as
    the `.squeeze()` the reference drivers apply, VAELE_DP:64) and runs the fused step; anything else derived from q / out differentiates
    through `backward` below (vaeq_eq_backward: softmin + FIR backward for arbitrary upstream gradients)."""

    @staticmethod
    @_lib.device_guard
    def forward(ctx, W, x, net, amp_levels, var, nu_sc):
        eq = net._engine(amp_levels, var, nu_sc)
        eq.W.copy_(W.detach())
        q, out, _, _ = eq.forward(x)
        ctx.net_ref, ctx.x, ctx.x_version = weakref.ref(net), x, x._version
        ctx.consts = (amp_levels, var, nu_sc)
        ctx.save_for_backward(q, out)
        ctx.q_ptr, ctx.q_numel, ctx.q_version, ctx.M = q.data_ptr(), q.numel(), q._version, net.M_est
        return q, out

    @staticmethod
    @_lib.device_guard
    def backward(ctx, gq, gout):
        if gq is None and gout is None:
            return (None,) * 6
        q, out = ctx.saved_tensors
        lib = _lib.load()
        x, (amp, var, _) = ctx.x, ctx.consts
        if x._version != ctx.x_version:
            raise RuntimeError("twoXtwoFIR backward: the input minibatch was modified in place after the forward pass")
        n, B, M = int(amp.numel()), int(q.shape[-1]), int(ctx.M)
        dev = q.device
        gq = None if gq is None else gq.to(_F32).contiguous()
        gout = None if gout is None else gout.to(_F32).contiguous()
        gW = torch.empty(2, 4, M, dtype=_F32, device=dev)
        scr = torch.empty(int(lib.vaeq_eq_backward_scratch_bytes(B, M)), dtype=torch.uint8, device=dev)
        _lib.check(lib.vaeq_eq_backward(x.data_ptr(), int(x.stride(1)), q.data_ptr(), int(q.stride(1)), out.data_ptr(), int(out.stride(1)),
                                        None if gq is None else gq.data_ptr(), B, None if gout is None else gout.data_ptr(), B,
                                        amp.contiguous().data_ptr(), var.contiguous().data_ptr(), n, B, M, gW.data_ptr(), scr.data_ptr(),
                                        _lib.current_stream()), "vaeq_eq_backward")
        return gW, None, None, None, None, None


_VIEW_NODES = ("SqueezeBackward", "UnsqueezeBackward", "ViewBackward", "AliasBackward", "ReshapeAliasBackward", "UnsafeViewBackward")


def _equalizer_node(q):
    """The _EqualizerFn node whose FIRST output `q` is (possibly through shape-only views), else None."""
    fn = q.grad_fn
    for _ in range(8):
        if fn is None:
            return None
        if getattr(fn, "_forward_cls", None) is _EqualizerFn:
            return fn
        if not fn.name().startswith(_VIEW_NODES) or len(fn.next_functions) != 1:
            return None
        fn, nr = fn.next_functions[0]
        if getattr(fn, "_forward_cls", None) is _EqualizerFn and nr != 0:
            return None
    return None


@_lib.device_guard
def soft_dec(out, var, amp_levels, nu_sc):
    """Soft demapper with the PCS correction term (sf:529-542)."""
    _require_cuda(out, "out")
    _lib.require_current_device(var, "var")                  # the kernel dereferences all three on out's device
    _lib.require_current_device(amp_levels, "amp_levels")
    lib = _lib.load()
    n, N = int(amp_levels.numel()), int(out.shape[-1])
    ld = _rows(out, "out")
    q = torch.empty(2, 2 * n, N, dtype=_F32, device=out.device)
    _lib.check(lib.vaeq_soft_dec(out.data_ptr(), ld, var.contiguous().data_ptr(), amp_levels.contiguous().data_ptr(),
                                 float(nu_sc), n, N, q.data_ptr(), N, _lib.current_stream()), "vaeq_soft_dec")
    return q


class _LossFromQ(torch.autograd.Function):
    """loss_function_shaping as a plain operator: loss(q, h_est) for ANY q, with dL/dq and dL/dh_est from vaeq_dp_loss_from_q."""

    @staticmethod
    @_lib.device_guard
    def forward(ctx, q, h, rx, amp, P):
        lib = _lib.load()
        dev = rx.device
        q2, rx2 = q.detach().reshape(2, -1, q.shape[-1]).contiguous(), rx.detach().reshape(2, 2, -1).contiguous()
        h2 = h.detach().contiguous()
        n, B, M = int(amp.numel()), int(q2.shape[-1]), int(h2.shape[-1])
        ws = torch.empty(int(lib.vaeq_dp_workspace_bytes(B, M, n)), dtype=torch.uint8, device=dev)
        loss, var_est = torch.empty(1, dtype=_F32, device=dev), torch.empty(2, dtype=_F32, device=dev)
        gq, gh = torch.empty_like(q2), torch.empty_like(h2)
        d = _lib.DpDesc()
        d.B, d.sps, d.M, d.n_lev = B, rx2.shape[-1] // B, M, n
        d.rx, d.ld_rx = rx2.data_ptr(), int(rx2.stride(1))
        d.amp, d.P, d.h = amp.data_ptr(), P.data_ptr(), h2.data_ptr()
        d.q, d.ld_q = q2.data_ptr(), B
        d.loss, d.var_est, d.gh = loss.data_ptr(), var_est.data_ptr(), gh.data_ptr()
        d.workspace, d.workspace_bytes = ws.data_ptr(), ws.numel()
        _lib.check(lib.vaeq_dp_loss_from_q(C.byref(d), gq.data_ptr(), B, _lib.current_stream()), "vaeq_dp_loss_from_q")
        ctx.save_for_backward(gq.reshape(q.shape), gh.reshape(h.shape))
        ctx.mark_non_differentiable(var_est)
        return loss.reshape(()), var_est

    @staticmethod
    def backward(ctx, g_loss, _g_var):
        gq, gh = ctx.saved_tensors
        return g_loss * gq, g_loss * gh, None, None, None


def loss_function_shaping(q, rx, h_est, amp_levels, P):
    """ELBO loss (sf:92-137): returns (loss, var_est (2,)).

    When `q` is the tensor returned by this package's twoXtwoFIR.forward for the minibatch `rx`, the fused CUDA step runs and the
    gradients reach the equalizer taps and `h_est` without materialising dL/dq.  For any other q (any CUDA tensor (2,2n,B), e.g. a
    posterior from another demapper) the loss is an ordinary autograd operator differentiable w.r.t. `q` and `h_est`."""
    node = _equalizer_node(q)
    net = node.net_ref() if node is not None else None
    fused = (net is not None and q.data_ptr() == node.q_ptr and q.numel() == node.q_numel and q.is_contiguous()
             and q._version == node.q_version and rx.data_ptr() == node.x.data_ptr() and rx.numel() == node.x.numel()
             and node.x._version == node.x_version)
    if not fused:
        _require_cuda(q, "q")
        _require_cuda(rx, "rx")
        amp = torch.as_tensor(amp_levels, dtype=_F32, device=rx.device).contiguous()
        Pt = torch.as_tensor(P, dtype=_F32, device=rx.device).contiguous()
        return _LossFromQ.apply(q, h_est, rx, amp, Pt)
    x, (amp_src, var, nu_sc) = node.x, node.consts
    Pt = torch.as_tensor(P, dtype=_F32, device=rx.device).contiguous()
    eq = net._engine(amp_src, var, nu_sc, P=Pt)
    loss, var_est = _FusedLoss.apply(net.conv_w.weight, h_est, eq, x)
    return loss, var_est


# -------------------------------------------------------------------------------------------------
# evaluation                                                                    sf:188-338
# -------------------------------------------------------------------------------------------------
@_lib.device_guard
def SER_IQflip(q, tx, return_counts=False):
    """SER from hard decisions argmax(q), min over 4 rotations x IQ flip per pol (sf:188-222)."""
    _require_cuda(q, "q")
    tx = _tx_bits(tx)
    lib = _lib.load()
    n, N = q.shape[1] // 2, int(q.shape[-1])
    counts = torch.empty(2, 2, 4, dtype=torch.int32, device=q.device)
    ser = torch.empty(2, dtype=_F32, device=q.device)
    _lib.check(lib.vaeq_ser_iqflip(q.data_ptr(), _rows(q, "q"), tx.data_ptr(), _rows(tx, "tx"), n, N, counts.data_ptr(),
                                   ser.data_ptr(), _lib.current_stream()), "vaeq_ser_iqflip")
    return (ser, counts) if return_counts else ser


@_lib.device_guard
def SER_constell_shaping(rx, tx, amp_levels, nu_sc, var, return_counts=False):
    """SER from the constellation with PCS-aware thresholds (sf:225-287).  Rescales `rx` IN PLACE (sf:242)."""
    _require_cuda(rx, "rx")
    tx = _tx_bits(tx)
    lib = _lib.load()
    n, N = int(amp_levels.numel()), int(rx.shape[-1])
    counts = torch.empty(2, 2, 4, dtype=torch.int32, device=rx.device)
    ser = torch.empty(2, dtype=_F32, device=rx.device)
    scr = _scratch(rx.device)
    _lib.check(lib.vaeq_ser_constell(rx.data_ptr(), _rows(rx, "rx"), tx.data_ptr(), _rows(tx, "tx"),
                                     amp_levels.contiguous().data_ptr(), var.contiguous().data_ptr(), float(nu_sc), n, N,
                                     counts.data_ptr(), ser.data_ptr(), scr.data_ptr(), _lib.current_stream()),
               "vaeq_ser_constell")
    return (ser, counts) if return_counts else ser


@_lib.device_guard
def _find_shift(q, out, tx, N_shift, amp_levels, return_corr, sync=True):
    lib = _lib.load()
    ref = q if q is not None else out
    _require_cuda(ref, "q/rx")
    tx = _tx_bits(tx)
    N = int(ref.shape[-1])
    dev = ref.device
    corr = torch.empty(2, 2, 2, N_shift, dtype=_F32, device=dev)
    shift = torch.empty(2, dtype=torch.int16, device=dev)
    r = torch.empty(1, dtype=torch.int32, device=dev)
    lib = _lib.load()
    scr = _scratch(dev, int(lib.vaeq_find_shift_scratch_bytes(int(N_shift))))
    n = 0 if q is None else q.shape[1] // 2
    _lib.check(lib.vaeq_find_shift(None if q is None else q.data_ptr(), 0 if q is None else _rows(q, "q"),
                                   None if out is None else out.data_ptr(), 0 if out is None else _rows(out, "rx"),
                                   tx.data_ptr(), _rows(tx, "tx"),
                                   None if q is None else amp_levels.contiguous().data_ptr(), n, N, int(N_shift),
                                   corr.data_ptr(), shift.data_ptr(), r.data_ptr(), scr.data_ptr(), _lib.current_stream()),
               "vaeq_find_shift")
    if not sync:                                           # batched callers (sweep.py) read many results with one sync
        return shift, r
    r_host = int(r.item())                                 # the reference returns a Python int here (sf:312,314)
    return (shift, r_host, corr) if return_corr else (shift, r_host)


def find_shift(q, tx, N_shift, amp_levels, pol, return_corr=False):
    """Time/polarisation alignment from E_q[x_I] (sf:290-314): returns (shift int16 (2,), r)."""
    return _find_shift(q, None, tx, N_shift, amp_levels, return_corr)


def find_shift_symb_full(rx, tx, N_shift, return_corr=False):
    """Same search on the equalizer output's in-phase component (sf:316-338)."""
    return _find_shift(None, rx, tx, N_shift, None, return_corr)


@_lib.device_guard
def frame_eval_runs(out_train, out_const, tx, amp_levels, var, nu_sc, seg_len, n_shift=21, edge=11, n_cut=10, return_counts=False, which=3,
                    return_scale=False):
    """The per-frame evaluation of the VAE drivers (VAELE_DP:70-89 with seg_len = batch_len, VAEflex_DP:74-84 with seg_len = 0) for R
    runs in one call and without a host sync: out_train (R,2,2n,N), out_const (R,2,2,N), tx (R,2,2,N) float16 (may be a view into
    longer rows), var (R,2), nu_sc (R,).  Returns ser (R,4) [constellation x, y, soft demapper x, y] and align (R,2,4) int32
    [shift_x, shift_y, r, symbols evaluated] for the estimators (from q, from out)."""
    ref = out_train if out_train is not None else out_const
    if which not in (1, 2, 3) or (which & 1 and out_train is None) or (which & 2 and out_const is None):
        raise _lib.VaeqError(f"which={which}: bit 0 needs out_train, bit 1 needs out_const")
    _require_cuda(ref, "out_train / out_const")
    tx = _tx_bits(tx)
    lib = _lib.load()
    R, N, n = int(ref.shape[0]), int(ref.shape[-1]), int(amp_levels.numel())
    dev = ref.device
    for t, name in ((out_train, "out_train"), (out_const, "out_const"), (tx, "tx")):
        if t is None:
            continue
        if t.dim() != 4 or t.shape[0] != R or t.shape[-1] != N or t.stride(3) != 1 or t.stride(1) != t.shape[2] * t.stride(2):
            raise _lib.VaeqError(f"{name}: need (R,2,rows,N) with unit time stride and evenly strided rows, got {tuple(t.shape)} {t.stride()}")
    var = torch.as_tensor(var, dtype=_F32, device=dev).reshape(R, 2).contiguous()
    nu = torch.as_tensor(nu_sc, dtype=_F32, device=dev).reshape(R).contiguous()
    amp = amp_levels.to(dev, _F32).contiguous()
    align = torch.zeros(R, 2, 4, dtype=torch.int32, device=dev)
    counts = torch.empty(R, 2, 2, 2, 4, dtype=torch.int32, device=dev)
    ser = torch.full((R, 4), float("nan"), dtype=_F32, device=dev)
    scale = torch.empty(R, dtype=_F32, device=dev) if return_scale else None
    scr = _scratch(dev, int(lib.vaeq_frame_eval_scratch_bytes(R, int(n_shift))))
    qa = (out_train.data_ptr(), int(out_train.stride(2)), int(out_train.stride(0))) if out_train is not None else (None, 0, 0)
    oa = (out_const.data_ptr(), int(out_const.stride(2)), int(out_const.stride(0))) if out_const is not None else (None, 0, 0)
    _lib.check(lib.vaeq_frame_eval_runs_ex(*qa, *oa, tx.data_ptr(), int(tx.stride(2)), int(tx.stride(0)), amp.data_ptr(), var.data_ptr(), 2,
                                           nu.data_ptr(), n, N, int(n_shift), R, int(seg_len), int(edge), int(n_cut), int(which), align.data_ptr(),
                                           counts.data_ptr(), ser.data_ptr(), None if scale is None else scale.data_ptr(), scr.data_ptr(),
                                           _lib.current_stream()), "vaeq_frame_eval_runs_ex")
    if return_scale:
        return (ser, align, counts, scale) if return_counts else (ser, align, scale)
    return (ser, align, counts) if return_counts else (ser, align)


def _run_pmf(P, R, n, dev):
    """(R, n) float32 pmf rows on `dev` (one shared row is repeated) and the run stride the C ABI takes."""
    Pt = torch.as_tensor(P, dtype=_F32, device=dev)
    if Pt.dim() == 1:
        Pt = Pt.unsqueeze(0).expand(R, n)
    if tuple(Pt.shape) != (R, n):
        raise _lib.VaeqError(f"P: need (R={R}, n={n}) or (n,), got {tuple(Pt.shape)}")
    Pt = Pt.contiguous()
    return Pt, int(Pt.stride(0))


def gmi_runs(q, tx, P, align, counts, seg_len, edge=11, n_cut=10):
    """EXTENSION (not in the reference): GMI = H(X) + mean log2 q(x_tx|y) per pol (bit/2D-symbol) of R runs, scored on exactly the symbols
    and under the (IQ flip, rotation) hypothesis of the soft-demapper SER of frame_eval_runs: q (R,2,2n,N) and tx (R,2,2,N) float16 as
    given to frame_eval_runs, P (R,n) or (n,) pmf, align (R,2,4) and counts (R,2,2,2,4) from frame_eval_runs(..., return_counts=True)
    with the same seg_len / edge / n_cut.  Returns (R,2) float32 on the device, NaN where no symbol was evaluated; no host sync."""
    return _rate_runs("vaeq_frame_gmi_runs", q, tx, P, align, counts, seg_len, edge, n_cut)


def bmi_runs(q, tx, P, align, counts, seg_len, edge=11, n_cut=10):
    """EXTENSION (not in the reference): the bit-metric decoding rate of Gray-labelled bits (BMI, DESIGN.md §2) per pol (bit/2D-symbol)
    of R runs: H(X) + mean over the symbols of sum over the I and Q bits of log2 q(b_i = tx's bit | y), with the bit posteriors summed
    from q.  Arguments, symbols, hypothesis and result exactly as gmi_runs."""
    return _rate_runs("vaeq_frame_bmi_runs", q, tx, P, align, counts, seg_len, edge, n_cut)


@_lib.device_guard
def _rate_runs(fn, q, tx, P, align, counts, seg_len, edge, n_cut):
    """gmi_runs / bmi_runs through the C entry `fn` (vaeq_frame_gmi_runs or vaeq_frame_bmi_runs: same arguments)."""
    _require_cuda(q, "q")
    tx = _tx_bits(tx)
    lib = _lib.load()
    R, N, n = int(q.shape[0]), int(q.shape[-1]), int(q.shape[2]) // 2 if q.dim() == 4 else 0
    dev = q.device
    for t, name, rows in ((q, "q", 2 * n), (tx, "tx", 2)):
        if t.dim() != 4 or t.shape[0] != R or t.shape[1] != 2 or t.shape[2] != rows or t.shape[-1] != N or t.stride(3) != 1 \
                or t.stride(1) != t.shape[2] * t.stride(2):
            raise _lib.VaeqError(f"{name}: need (R,2,rows,N) with unit time stride and evenly strided rows, got {tuple(t.shape)} {t.stride()}")
    for t, name, shape in ((align, "align", (R, 2, 4)), (counts, "counts", (R, 2, 2, 2, 4))):
        if not torch.is_tensor(t) or t.dtype != torch.int32 or tuple(t.shape) != shape or not t.is_contiguous() or t.device != dev:
            raise _lib.VaeqError(f"{name}: need a contiguous int32 {shape} tensor on {dev} (frame_eval_runs(..., return_counts=True))")
    Pt, rs_P = _run_pmf(P, R, n, dev)
    rate = torch.empty(R, 2, dtype=_F32, device=dev)
    scr = _scratch(dev, max(1, int(lib.vaeq_frame_gmi_scratch_bytes(R, N))))
    _lib.check(getattr(lib, fn)(q.data_ptr(), int(q.stride(2)), int(q.stride(0)), tx.data_ptr(), int(tx.stride(2)), int(tx.stride(0)),
                                Pt.data_ptr(), rs_P, align.data_ptr(), counts.data_ptr(), n, N, R, int(seg_len), int(edge), int(n_cut),
                                rate.data_ptr(), scr.data_ptr(), _lib.current_stream()), fn)
    return rate


@_lib.device_guard
def soft_dec_runs(out, var, amp_levels, nu_sc):
    """soft_dec (sf:529-542) for R independent runs in one launch: out (R,2,2,N), var (R,2), nu_sc (R,) -> q (R,2,2n,N)."""
    _require_cuda(out, "out")
    lib = _lib.load()
    out = out.contiguous()
    R, N, n = int(out.shape[0]), int(out.shape[-1]), int(amp_levels.numel())
    dev = out.device
    var = torch.as_tensor(var, dtype=_F32, device=dev).reshape(R, 2).contiguous()
    nu = torch.as_tensor(nu_sc, dtype=_F32, device=dev).reshape(R).contiguous()
    q = torch.empty(R, 2, 2 * n, N, dtype=_F32, device=dev)
    _lib.check(lib.vaeq_soft_dec_runs(out.data_ptr(), var.data_ptr(), amp_levels.to(dev, _F32).contiguous().data_ptr(), nu.data_ptr(), n, N, R,
                                      q.data_ptr(), _lib.current_stream()), "vaeq_soft_dec_runs")
    return q


def _runs_rows(t, name, R, rows, dtype):
    """Check a (R,2,rows,T) tensor with unit time stride and evenly strided rows (views into longer rows allowed) on the current device."""
    if not t.is_cuda:
        raise _lib.VaeqError(f"{name} must be a CUDA tensor: vae_equalizer_b200 has no CPU path")
    _lib.require_current_device(t, name)
    if t.dtype != dtype:
        raise _lib.VaeqError(f"{name} must be {dtype}, got {t.dtype}")
    if t.dim() != 4 or t.shape[0] != R or t.shape[1] != 2 or t.shape[2] != rows or t.stride(3) != 1 or t.stride(1) != rows * t.stride(2):
        raise _lib.VaeqError(f"{name}: need (R={R},2,{rows},T) with unit time stride and evenly strided rows, got {tuple(t.shape)} {t.stride()}")


@_lib.device_guard
def lmmse_taps_runs(rx, tx, M_est, n_shift=21):
    """EXTENSION (not in the reference): the data-aided LMMSE taps of R runs (DESIGN.md §2), the reference curve of the blind equalizers.
    Per run, the least-squares taps of the 2x2 butterfly FIR of M_est taps (the structure of twoXtwoFIR) that map rx onto the run's own
    transmitted symbols, at the decision delay of least MSE in [-n_shift//2, n_shift//2] per output pol, unbiased.  Correlations and solve in
    double on the device, one launch pair for all runs, no host sync; a run's result does not depend on the other runs.
    rx (R,2,2,2N) float32 and tx (R,2,2,N) float16 (views into longer rows allowed).  Returns W (R,2,4,M_est) float32 in the layout of
    twoXtwoFIR.conv_w.weight, var (R,2) float32 (noise variance per real dimension of the equalized symbols), delay (R,2) int32 and ok (R,)
    bool: False where the run's correlation matrix is not positive definite (its W and var are then NaN)."""
    tx = _tx_bits(tx)
    R, N, M = int(tx.shape[0]), int(tx.shape[-1]), int(M_est)
    _runs_rows(rx, "rx", R, 2, _F32)
    _runs_rows(tx, "tx", R, 2, torch.float16)
    if rx.shape[-1] != 2 * N:
        raise _lib.VaeqError(f"rx has {rx.shape[-1]} samples per row, tx {N} symbols: need 2 samples per symbol")
    lib = _lib.load()
    dev = rx.device
    W = torch.empty(R, 2, 4, M, dtype=_F32, device=dev)
    var = torch.empty(R, 2, dtype=_F32, device=dev)
    delay = torch.empty(R, 2, dtype=torch.int32, device=dev)
    ok = torch.empty(R, dtype=torch.int32, device=dev)
    nb = int(lib.vaeq_lmmse_taps_scratch_bytes(M, int(n_shift), R))
    scr = _scratch(dev, max(nb, 1))
    _lib.check(lib.vaeq_lmmse_taps_runs(rx.data_ptr(), int(rx.stride(2)), int(rx.stride(0)), 2 * N, tx.data_ptr(), int(tx.stride(2)),
                                        int(tx.stride(0)), N, M, int(n_shift), R, W.data_ptr(), var.data_ptr(), delay.data_ptr(), ok.data_ptr(),
                                        scr.data_ptr(), scr.numel(), _lib.current_stream()), "vaeq_lmmse_taps_runs")
    return W, var, delay, ok.bool()


@_lib.device_guard
def fir_runs(rx, W):
    """EXTENSION (not in the reference): twoXtwoFIR's butterfly FIR (sf:500-518, zero padding M//2, stride 2) for R runs with per-run taps in
    one launch: rx (R,2,2,L) float32 (views into longer rows allowed), W (R,2,4,M) float32 -> out (R,2,2,L//2) float32."""
    _require_cuda(W, "W")
    R = int(rx.shape[0]) if rx.dim() == 4 else -1
    _runs_rows(rx, "rx", R, 2, _F32)
    _lib.require_current_device(W, "W")
    if W.dim() != 4 or tuple(W.shape[:3]) != (R, 2, 4) or W.dtype != _F32:
        raise _lib.VaeqError(f"W: need (R={R},2,4,M) float32, got {tuple(W.shape)} {W.dtype}")
    lib = _lib.load()
    L, M = int(rx.shape[-1]), int(W.shape[-1])
    N = L // 2
    W = W.contiguous()
    out = torch.empty(R, 2, 2, N, dtype=_F32, device=rx.device)
    _lib.check(lib.vaeq_fir_runs(rx.data_ptr(), int(rx.stride(2)), int(rx.stride(0)), L, W.data_ptr(), M, N, R, out.data_ptr(),
                                 _lib.current_stream()), "vaeq_fir_runs")
    return out


@_lib.device_guard
def cma_align_rescale(out, align, scale, edge=11):
    """CMA_DP:42-48 for R runs: out (R,2,2,N) rolled by (r, -shift) with the evaluated slice rescaled like SER_constell_shaping leaves it
    (sf:242); align (R,2,4) int32 and scale (R,) from frame_eval_runs(..., which=2, return_scale=True)."""
    _require_cuda(out, "out")
    lib = _lib.load()
    R, N = int(out.shape[0]), int(out.shape[-1])
    if out.dim() != 4 or out.stride(3) != 1 or out.stride(1) != out.shape[2] * out.stride(2):
        raise _lib.VaeqError(f"out: need (R,2,2,N) with unit time stride and evenly strided rows, got {tuple(out.shape)} {out.stride()}")
    oc = torch.empty(R, 2, 2, N, dtype=_F32, device=out.device)
    _lib.check(lib.vaeq_cma_align_rescale(out.data_ptr(), int(out.stride(2)), int(out.stride(0)), align.data_ptr(), scale.data_ptr(), N, int(edge), R,
                                          oc.data_ptr(), _lib.current_stream()), "vaeq_cma_align_rescale")
    return oc


def GMI(q, tx, P):
    """EXTENSION (not in the reference, SURVEY.md fact 3): H(X) + E[log2 q(x_tx|y)] per pol, bit/2D-symbol."""
    return _rate("vaeq_gmi", q, tx, P)


def BMI(q, tx, P):
    """EXTENSION (not in the reference): the bit-metric decoding rate of Gray-labelled bits (DESIGN.md §2) per pol, bit/2D-symbol:
    H(X) + E[sum over the I and Q bits of log2 q(b_i = tx's bit | y)].  Arguments and result as GMI."""
    return _rate("vaeq_bmi", q, tx, P)


@_lib.device_guard
def _rate(fn, q, tx, P):
    _require_cuda(q, "q")
    lib = _lib.load()
    n, N = q.shape[1] // 2, int(q.shape[-1])
    Pt = torch.as_tensor(P, dtype=_F32, device=q.device).contiguous()
    out = torch.empty(2, dtype=_F32, device=q.device)
    scr = _scratch(q.device)
    _lib.check(getattr(lib, fn)(q.data_ptr(), _rows(q, "q"), _tx_bits(tx).data_ptr(), _rows(tx, "tx"), Pt.data_ptr(), n, N,
                                out.data_ptr(), scr.data_ptr(), _lib.current_stream()), fn)
    return out


@_lib.device_guard
def bit_llr(q):
    """EXTENSION (not in the reference): Gray-labelled bit LLRs of the posteriors (DESIGN.md §2), the soft input of a binary decoder.
    q (2,2n,N) or (R,2,2n,N) float32 with unit time stride and evenly strided rows (views allowed) -> (2,2m,N) or (R,2,2m,N) float32,
    m = log2(n), rows [I bits MSB..LSB | Q bits MSB..LSB] per pol; L = ln q(b=0|y) - ln q(b=1|y), each clamped at 1e-30 (positive: bit 0).
    One launch, no host sync."""
    _require_cuda(q, "q")
    single = q.dim() == 3
    q4 = q.unsqueeze(0) if single else q
    if q4.dim() != 4 or q4.shape[1] != 2 or q4.shape[2] not in (4, 8, 16) or q4.stride(3) != 1 or q4.stride(1) != q4.shape[2] * q4.stride(2):
        raise _lib.VaeqError(f"q: need (2,2n,N) or (R,2,2n,N), n in 2/4/8, with unit time stride and evenly strided rows, got "
                             f"{tuple(q.shape)} {q.stride()}")
    lib = _lib.load()
    R, n, N = int(q4.shape[0]), int(q4.shape[2]) // 2, int(q4.shape[3])
    m = n.bit_length() - 1
    llr = torch.empty(R, 2, 2 * m, N, dtype=_F32, device=q.device)
    _lib.check(lib.vaeq_bit_llr_runs(q4.data_ptr(), int(q4.stride(2)), int(q4.stride(0)) if R > 1 else 4 * n * int(q4.stride(2)), n, N, R,
                                     llr.data_ptr(), N, 4 * m * N, _lib.current_stream()), "vaeq_bit_llr_runs")
    return llr[0] if single else llr


# -------------------------------------------------------------------------------------------------
# CMA baselines and CPE                                                         sf:140-186, sf:341-488
# -------------------------------------------------------------------------------------------------
@_lib.device_guard
def _cma(mode, Rx, R, h, lr, batchlen, symb_step, sps, train):
    """Rx (2,2,N), h (2,2,2,M) like the reference -- or a batch of S independent streams: Rx (S,2,2,N), h (S,2,2,2,M), one launch
    sequence for all of them (one warp / one CTA per stream); out and e then carry the leading stream dimension too."""
    _require_cuda(Rx, "Rx")
    _require_cuda(h, "h")
    if not (Rx.is_contiguous() and h.is_contiguous()):
        raise _lib.VaeqError("CMA: Rx and h must be contiguous")
    batched = Rx.dim() == 4
    if (batched and (h.dim() != 5 or h.shape[0] != Rx.shape[0])) or (not batched and (Rx.dim() != 3 or h.dim() != 4)):
        raise _lib.VaeqError(f"CMA: need Rx (2,2,N) with h (2,2,2,M) or Rx (S,2,2,N) with h (S,2,2,2,M), got {tuple(Rx.shape)} {tuple(h.shape)}")
    lib = _lib.load()
    S = int(Rx.shape[0]) if batched else 1
    N, M = int(Rx.shape[-1]), int(h.shape[-1])
    dev = Rx.device
    out = torch.zeros((S, 2, 2, N // sps) if batched else (2, 2, N // sps), dtype=_F32, device=dev)
    e = torch.empty((S, N // sps, 2) if batched else (N // sps, 2), dtype=_F32, device=dev)
    scr = torch.empty(int(lib.vaeq_cma_scratch_bytes(N, M, S)), dtype=torch.uint8, device=dev)
    hd = h.detach()
    _lib.check(lib.vaeq_cma(mode, Rx.data_ptr(), N, float(R), hd.data_ptr(), M, float(lr), int(batchlen), int(symb_step),
                            int(sps), 1 if train else 0, out.data_ptr(), e.data_ptr(), S, scr.data_ptr(),
                            _lib.current_stream()), "vaeq_cma")
    return out, h, e


def CMA(Rx, R, h, lr, sps, eval):
    """Constant-modulus algorithm, tap update after every symbol (sf:341-379); `eval` True = train (sic)."""
    return _cma(0, Rx, R, h, lr, 0, 0, sps, bool(eval))


def CMAbatch(Rx, R, h, lr, batchlen, sps, eval):
    """CMA with buffered, batch-wise tap updates (sf:381-434)."""
    return _cma(1, Rx, R, h, lr, batchlen, 0, sps, bool(eval))


def CMAflex(Rx, R, h, lr, batchlen, symb_step, sps, eval):
    """CMA with a trailing window of `batchlen` applied every `symb_step` symbols (sf:436-488)."""
    return _cma(2, Rx, R, h, lr, batchlen, symb_step, sps, bool(eval))


@_lib.device_guard
def CPE(y):
    """Viterbi-Viterbi carrier phase estimation with unwrap (sf:140-186); y (2,2,N), or (S,2,2,N) for S independent runs in one call."""
    _require_cuda(y, "y")
    lib = _lib.load()
    y = y.contiguous()
    N = int(y.shape[-1])
    S = int(y.shape[0]) if y.dim() == 4 else 1
    out = torch.empty_like(y)
    scr = torch.empty(int(lib.vaeq_cpe_runs_scratch_bytes(N, S)), dtype=torch.uint8, device=y.device)
    _lib.check(lib.vaeq_cpe_runs(y.data_ptr(), N, S, out.data_ptr(), scr.data_ptr(), _lib.current_stream()), "vaeq_cpe_runs")
    return out
