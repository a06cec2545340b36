"""ctypes binding of libvaeq.so (C ABI declared in include/vaeq.h).

There is NO CPU fallback: if the shared library is missing or a call fails this module raises.
"""
from __future__ import annotations

import ctypes as C
import functools
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libvaeq.so")

c_f32p = C.POINTER(C.c_float)


class VaeqError(RuntimeError):
    pass


class DpDesc(C.Structure):
    """Mirror of `struct vaeq_dp_desc` (include/vaeq.h)."""
    _fields_ = [
        ("B", C.c_int32), ("sps", C.c_int32), ("M", C.c_int32), ("n_lev", C.c_int32),
        ("nu_sc", C.c_float), ("flags", C.c_int32),
        ("rx", C.c_void_p), ("ld_rx", C.c_int64),
        ("amp", C.c_void_p), ("P", C.c_void_p), ("var", C.c_void_p),
        ("W", C.c_void_p), ("h", C.c_void_p), ("adam", C.c_void_p),
        ("q", C.c_void_p), ("ld_q", C.c_int64),
        ("out", C.c_void_p), ("ld_out", C.c_int64),
        ("q_keep", C.c_void_p), ("ld_q_keep", C.c_int64),
        ("out_keep", C.c_void_p), ("ld_out_keep", C.c_int64),
        ("keep_lo", C.c_int32), ("keep_n", C.c_int32),
        ("loss", C.c_void_p), ("var_est", C.c_void_p),
        ("gW", C.c_void_p), ("gh", C.c_void_p),
        ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t),
    ]


class DpRuns(C.Structure):
    """Mirror of `struct vaeq_dp_runs`: run strides (elements) of the batched-runs frame call."""
    _fields_ = [
        ("n_runs", C.c_int32),
        ("rs_rx", C.c_int64), ("rs_amp", C.c_int64), ("rs_P", C.c_int64), ("rs_var", C.c_int64),
        ("rs_W", C.c_int64), ("rs_h", C.c_int64), ("rs_adam", C.c_int64), ("rs_q", C.c_int64), ("rs_out", C.c_int64),
        ("rs_q_keep", C.c_int64), ("rs_out_keep", C.c_int64),
        ("nu_sc", C.c_void_p), ("lr_w", C.c_void_p), ("lr_h", C.c_void_p),
    ]


class PeerComm(C.Structure):
    """Mirror of `struct vaeq_peer_comm`: peer-mapped slot pointers of the batch-split ranks (vaeq_dp_split_step_peer)."""
    _fields_ = [("rank", C.c_int32), ("world", C.c_int32), ("slot", C.c_void_p * 8), ("epoch", C.c_void_p)]


class AwgnRuns(C.Structure):
    """Mirror of `struct vaeq_awgn_runs`: run strides (elements) and per-run values of the batched AWGN calls."""
    _fields_ = [
        ("n_runs", C.c_int32),
        ("rs_rx", C.c_int64), ("rs_W", C.c_int64), ("rs_h", C.c_int64), ("rs_adam", C.c_int64), ("rs_P", C.c_int64),
        ("rs_q", C.c_int64), ("rs_out", C.c_int64), ("rs_loss", C.c_int64),
        ("lr", C.c_void_p), ("var", C.c_void_p), ("amp_mean", C.c_void_p),
    ]


class AwgnDesc(C.Structure):
    """Mirror of `struct vaeq_awgn_desc`."""
    _fields_ = [
        ("B", C.c_int32), ("sps", C.c_int32), ("M", C.c_int32), ("n_lev", C.c_int32),
        ("amp_mean", C.c_float), ("var", C.c_float),
        ("rx", C.c_void_p), ("amp", C.c_void_p), ("P", C.c_void_p),
        ("W", C.c_void_p), ("h", C.c_void_p), ("adam", C.c_void_p),
        ("q", C.c_void_p), ("out", C.c_void_p), ("loss", C.c_void_p),
        ("gW", C.c_void_p), ("gh", C.c_void_p),
        ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t),
    ]


# name -> (restype, argtypes); every symbol include/vaeq.h declares
_i32, _i64, _f, _vp, _sz, _u64 = C.c_int32, C.c_int64, C.c_float, C.c_void_p, C.c_size_t, C.c_uint64
PROTOTYPES = {
    "vaeq_abi_version": (C.c_int, []),
    "vaeq_last_error": (C.c_char_p, []),
    "vaeq_sm_count": (C.c_int, []),
    "vaeq_kernel_timing": (C.c_int, [_i32]),
    "vaeq_kernel_timing_read": (C.c_int, [_vp, _vp]),
    "vaeq_launch_count": (C.c_int64, [_i32]),
    "vaeq_dp_workspace_bytes": (_sz, [_i32, _i32, _i32]),
    "vaeq_adam_state_floats": (_sz, [_i32]),
    "vaeq_dp_force_generic": (C.c_int, [_i32]),
    "vaeq_dp_dynamic_tiles": (C.c_int, [_i32]),
    "vaeq_dp_tc_taps": (C.c_int, [_i32]),
    "vaeq_dp_tc_forward": (C.c_int, [_i32]),
    "vaeq_dp_forward": (C.c_int, [C.POINTER(DpDesc), _vp]),
    "vaeq_dp_forward_backward": (C.c_int, [C.POINTER(DpDesc), _vp]),
    "vaeq_dp_loss_from_q": (C.c_int, [C.POINTER(DpDesc), _vp, _i64, _vp]),
    "vaeq_eq_backward_scratch_bytes": (_sz, [_i32, _i32]),
    "vaeq_eq_backward": (C.c_int, [_vp, _i64, _vp, _i64, _vp, _i64, _vp, _i64, _vp, _i64, _vp, _vp, _i32, _i32, _i32, _vp, _vp, _vp]),
    "vaeq_dp_train_step": (C.c_int, [C.POINTER(DpDesc), _f, _f, _vp]),
    "vaeq_dp_train_frame": (C.c_int, [C.POINTER(DpDesc), _i32, _i32, _i32, _f, _f, _vp, _vp, _vp]),
    "vaeq_dp_persistent_frames": (C.c_int, [_i32]),
    "vaeq_dp_frame_runs_per_sm": (C.c_int, [_i32]),
    "vaeq_dp_runs_workspace_bytes": (_sz, [_i32, _i32, _i32, _i32]),
    "vaeq_dp_runs_max_batch_len": (_i32, [_i32, _i32]),
    "vaeq_dp_train_frame_runs": (C.c_int, [C.POINTER(DpDesc), C.POINTER(DpRuns), _i32, _i32, _i32, _f, _f, _vp, _vp, _vp]),
    "vaeq_dp_split_stats_doubles": (_sz, [_i32]),
    "vaeq_dp_split_forward": (C.c_int, [C.POINTER(DpDesc), _i32, _i32, _vp, _vp]),
    "vaeq_dp_split_backward": (C.c_int, [C.POINTER(DpDesc), _i32, _i32, _vp, _vp, _vp]),
    "vaeq_dp_split_update": (C.c_int, [C.POINTER(DpDesc), _vp, _f, _f, _vp]),
    "vaeq_peer_slot_bytes": (_sz, [_i32]),
    "vaeq_dp_split_step_peer": (C.c_int, [C.POINTER(DpDesc), _i32, _i32, C.POINTER(PeerComm), _f, _f, _vp]),
    "vaeq_adam_update": (C.c_int, [_vp, _vp, _vp, _i32, _f, _i32, _vp, _i32, _vp]),
    "vaeq_soft_dec": (C.c_int, [_vp, _i64, _vp, _vp, _f, _i32, _i32, _vp, _i64, _vp]),
    "vaeq_find_shift_scratch_bytes": (_sz, [_i32]),
    "vaeq_find_shift": (C.c_int, [_vp, _i64, _vp, _i64, _vp, _i64, _vp, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp]),
    "vaeq_ser_iqflip": (C.c_int, [_vp, _i64, _vp, _i64, _i32, _i32, _vp, _vp, _vp]),
    "vaeq_ser_constell": (C.c_int, [_vp, _i64, _vp, _i64, _vp, _vp, _f, _i32, _i32, _vp, _vp, _vp, _vp]),
    "vaeq_frame_eval_scratch_bytes": (_sz, [_i32, _i32]),
    "vaeq_frame_eval_runs": (C.c_int, [_vp, _i64, _i64, _vp, _i64, _i64, _vp, _i64, _i64, _vp, _vp, _i64, _vp, _i32, _i32, _i32, _i32, _i32,
                                      _i32, _i32, _vp, _vp, _vp, _vp, _vp]),
    "vaeq_frame_eval_runs_ex": (C.c_int, [_vp, _i64, _i64, _vp, _i64, _i64, _vp, _i64, _i64, _vp, _vp, _i64, _vp, _i32, _i32, _i32, _i32, _i32,
                                         _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp]),
    "vaeq_cma_align_rescale": (C.c_int, [_vp, _i64, _i64, _vp, _vp, _i32, _i32, _i32, _vp, _vp]),
    "vaeq_frame_gmi_scratch_bytes": (_sz, [_i32, _i32]),
    "vaeq_frame_gmi_runs": (C.c_int, [_vp, _i64, _i64, _vp, _i64, _i64, _vp, _i64, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _vp]),
    "vaeq_awgn_gmi_scratch_bytes": (_sz, [_i32, _i32]),
    "vaeq_awgn_gmi_runs": (C.c_int, [_vp, _i64, _i64, _vp, _i64, _i64, _vp, _i64, _vp, _vp, _i32, _i32, _i32, _i32, _vp, _vp, _vp]),
    "vaeq_frame_bmi_runs": (C.c_int, [_vp, _i64, _i64, _vp, _i64, _i64, _vp, _i64, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _vp]),
    "vaeq_awgn_bmi_runs": (C.c_int, [_vp, _i64, _i64, _vp, _i64, _i64, _vp, _i64, _vp, _vp, _i32, _i32, _i32, _i32, _vp, _vp, _vp]),
    "vaeq_soft_dec_runs": (C.c_int, [_vp, _vp, _vp, _vp, _i32, _i32, _i32, _vp, _vp]),
    "vaeq_gmi": (C.c_int, [_vp, _i64, _vp, _i64, _vp, _i32, _i32, _vp, _vp, _vp]),
    "vaeq_bmi": (C.c_int, [_vp, _i64, _vp, _i64, _vp, _i32, _i32, _vp, _vp, _vp]),
    "vaeq_bit_llr_runs": (C.c_int, [_vp, _i64, _i64, _i32, _i32, _i32, _vp, _i64, _i64, _vp]),
    "vaeq_lmmse_taps_scratch_bytes": (_sz, [_i32, _i32, _i32]),
    "vaeq_lmmse_taps_runs": (C.c_int, [_vp, _i64, _i64, _i32, _vp, _i64, _i64, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "vaeq_fir_runs": (C.c_int, [_vp, _i64, _i64, _i32, _vp, _i32, _i32, _i32, _vp, _vp]),
    "vaeq_cma_scratch_bytes": (_sz, [_i32, _i32, _i32]),
    "vaeq_cma": (C.c_int, [_i32, _vp, _i32, _f, _vp, _i32, _f, _i32, _i32, _i32, _i32, _vp, _vp, _i32, _vp, _vp]),
    "vaeq_cpe_scratch_bytes": (_sz, [_i32]),
    "vaeq_gen_levels": (C.c_int, [_vp, _vp, _i32, _i32, _i32, _i32, _u64, _vp, _vp, _i32, _vp]),
    "vaeq_gen_pulse": (C.c_int, [_vp, _vp, _i32, _i32, _vp, _i32, _vp]),
    "vaeq_gen_pulse_cplx": (C.c_int, [_vp, _vp, _i32, _i32, _vp, _i32, _vp]),
    "vaeq_gen_jones": (C.c_int, [_vp, _vp, _vp, _vp, _f, _f, _i32, _i32, _vp]),
    "vaeq_gen_noise": (C.c_int, [_vp, _vp, _u64, _i32, _i32, _vp, _i32, _vp]),
    "vaeq_cpe": (C.c_int, [_vp, _i32, _vp, _vp, _vp]),
    "vaeq_cpe_runs_scratch_bytes": (_sz, [_i32, _i32]),
    "vaeq_cpe_runs": (C.c_int, [_vp, _i32, _i32, _vp, _vp, _vp]),
    "vaeq_cma_awgn": (C.c_int, [_vp, _i32, _f, _vp, _i32, _f, _i32, _i32, _vp, _vp, _i32, _vp]),
    "vaeq_cpe_awgn": (C.c_int, [_vp, _i32, _i32, _vp, _vp, _vp]),
    "vaeq_ser_cma": (C.c_int, [_vp, _i64, _vp, _i64, _vp, _i32, _i32, _vp, _vp, _vp, _vp]),
    "vaeq_find_shift_symb": (C.c_int, [_vp, _i32, _vp, _i64, _i32, _i32, _vp, _vp, _vp]),
    "vaeq_cma_awgn_runs": (C.c_int, [_vp, _i64, _i64, _i64, _i32, _i32, _vp, _i64, _i64, _i32, _vp, _i32, _vp, _f, _i32, _vp, _i32, _vp]),
    "vaeq_awgn_cma_eval_scratch_bytes": (_sz, [_i32, _i32, _i32, _i32]),
    "vaeq_awgn_cma_eval_runs": (C.c_int, [_vp, _i64, _i64, _vp, _i64, _i64, _vp, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp]),
    "vaeq_awgn_workspace_bytes": (_sz, [_i32, _i32, _i32]),
    "vaeq_adam_state_floats_awgn": (_sz, [_i32]),
    "vaeq_awgn_forward": (C.c_int, [C.POINTER(AwgnDesc), _vp]),
    "vaeq_awgn_forward_backward": (C.c_int, [C.POINTER(AwgnDesc), _vp]),
    "vaeq_awgn_train_step": (C.c_int, [C.POINTER(AwgnDesc), _f, _f, _vp]),
    "vaeq_awgn_runs_workspace_bytes": (_sz, [_i32, _i32, _i32, _i32]),
    "vaeq_awgn_train_frames_runs": (C.c_int, [C.POINTER(AwgnDesc), C.POINTER(AwgnRuns), _i64, _i64, _i32, _i32, _vp]),
    "vaeq_awgn_forward_runs": (C.c_int, [C.POINTER(AwgnDesc), C.POINTER(AwgnRuns), _i64, _vp]),
    "vaeq_awgn_eval_scratch_bytes": (_sz, [_i32, _i32, _i32]),
    "vaeq_awgn_eval_runs": (C.c_int, [_vp, _i64, _i64, _vp, _i64, _i64, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp]),
    "vaeq_gen_awgn": (C.c_int, [_vp, _vp, _i32, _vp, _i32, _i32, _i32, _i32, _vp, _vp, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp]),
}

_lib = None


def load():
    """Load libvaeq.so (once) and bind every prototype.  Raises VaeqError when it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise VaeqError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "or vae_equalizer_b200/csrc/build.sh -- there is no CPU fallback")
    lib = C.CDLL(LIB_PATH)
    missing = [name for name in PROTOTYPES if not hasattr(lib, name)]
    if missing:
        raise VaeqError(f"{LIB_PATH} does not export {missing}: header/library mismatch, rebuild")
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.vaeq_abi_version() != 1:
        raise VaeqError(f"libvaeq ABI version {lib.vaeq_abi_version()} != 1")
    _lib = lib
    return lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = load().vaeq_last_error().decode(errors="replace")
        raise VaeqError(f"{what or 'libvaeq call'} failed (code {rc}): {msg}")


def ptr(t):
    """Device pointer of a torch tensor (or None)."""
    return None if t is None else C.c_void_p(t.data_ptr())


def current_stream():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def device_guard(fn):
    """Run `fn` with the CUDA device of its first device-bearing argument (a tensor, or an object with a `.device`) current.

    libvaeq launches on the calling thread's current device and `current_stream()` is that device's stream, so every Python
    entry that reaches the C ABI is wrapped: tensors of `cuda:1` are processed on `cuda:1` whatever the caller's current device is."""
    import torch

    @functools.wraps(fn)
    def wrapper(*args, **kw):
        for a in (*args, *kw.values()):
            d = a if isinstance(a, torch.device) else getattr(a, "device", None)
            if isinstance(d, torch.device) and d.type == "cuda":
                if d.index is None or d.index == torch.cuda.current_device():
                    break
                with torch.cuda.device(d):
                    return fn(*args, **kw)
        return fn(*args, **kw)

    return wrapper


def require_current_device(t, name="tensor"):
    """Raise unless the CUDA tensor `t` lives on the current device (inside a device_guard: the device of the first argument)."""
    import torch
    if t is not None and t.is_cuda and t.device.index != torch.cuda.current_device():
        raise VaeqError(f"{name} lives on {t.device} but the call runs on cuda:{torch.cuda.current_device()}: all tensors of one "
                        "call must be on the same device")
