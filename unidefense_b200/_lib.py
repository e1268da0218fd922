"""ctypes binding of libunidefense_b200.so (the C ABI declared in include/unidefense_b200.h).

The product path has NO CPU fallback: if the shared library is missing, or a tensor is not
a contiguous CUDA fp32 tensor, the call fails loudly.
"""
import ctypes
import os
import threading
import types

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("UD_LIB_PATH") or os.path.join(_HERE, "libunidefense_b200.so")     # (override: A/B builds)
_lib = None
_lock = threading.Lock()

c_p = ctypes.c_void_p
c_i = ctypes.c_int
c_f = ctypes.c_float
c_sz = ctypes.c_size_t

# name -> (restype, argtypes); must list every symbol include/unidefense_b200.h declares
SIGNATURES = {
    "ud_last_error": (ctypes.c_char_p, []),
    "ud_version": (c_i, []),
    "ud_launch_count": (ctypes.c_longlong, []),
    "ud_fft_size_supported": (c_i, [c_i]),
    "ud_fft_size_any": (c_i, [c_i]),
    "ud_recon_tail_workspace_bytes": (c_sz, [c_i] * 6),
    "ud_recon_tail_signs_bytes": (c_sz, [c_i] * 4),
    "ud_recon_tail_fwd": (c_i, [c_p] * 7 + [c_sz] + [c_i] * 7 + [c_p]),
    "ud_recon_tail_bwd": (c_i, [c_p] * 8 + [c_sz] + [c_i] * 7 + [c_p]),
    "ud_in_act_fwd": (c_i, [c_p] * 7 + [c_i] * 3 + [c_f, c_i, c_p]),
    "ud_in_act_bwd_workspace_bytes": (c_sz, [c_i, c_i]),
    "ud_in_act_bwd": (c_i, [c_p] * 11 + [c_sz] + [c_i] * 4 + [c_p]),
    "ud_in_act_fwd_bf16": (c_i, [c_p] * 7 + [c_i] * 3 + [c_f, c_i, c_p]),
    "ud_in_act_bwd_bf16": (c_i, [c_p] * 11 + [c_sz] + [c_i] * 4 + [c_p]),
    "ud_tanh_fwd": (c_i, [c_p, c_p, ctypes.c_longlong, c_p]),
    "ud_tanh_bwd": (c_i, [c_p, c_p, c_p, ctypes.c_longlong, c_p]),
    "ud_bilinear_ac_fwd": (c_i, [c_p, c_p] + [c_i] * 5 + [c_p]),
    "ud_bilinear_ac_bwd": (c_i, [c_p, c_p] + [c_i] * 5 + [c_p]),
    "ud_attn_prep": (c_i, [c_p] * 4 + [c_i] * 9 + [c_p]),
    "ud_attn_prep_bwd": (c_i, [c_p] * 5 + [c_i] * 9 + [c_p]),
    "ud_rfft2_workspace_bytes": (c_sz, [c_i] * 4),
    "ud_rfft2": (c_i, [c_p] * 3 + [c_sz] + [c_i] * 6 + [c_p]),
    "ud_irfft2": (c_i, [c_p] * 4 + [c_sz] + [c_i] * 6 + [c_p]),
    "ud_attn_fuse_fwd": (c_i, [c_p] * 6 + [c_i] * 3 + [c_p]),
    "ud_attn_fuse_bwd_workspace_bytes": (c_sz, [c_i, c_i]),
    "ud_attn_fuse_bwd": (c_i, [c_p] * 10 + [c_sz] + [c_i] * 4 + [c_p]),
    "ud_bn_stats": (c_i, [c_p] * 3 + [c_i] * 3 + [c_p]),
    "ud_bn_bwd_reduce": (c_i, [c_p] * 6 + [c_i] * 3 + [c_p]),
    "ud_bn_bwd_apply": (c_i, [c_p] * 7 + [c_f, c_p] + [c_i] * 3 + [c_p]),
    "ud_proj_m_tiles": (c_i, [c_i] * 4),
    "ud_proj_prep_x": (c_i, [c_p] * 3 + [c_i] * 3 + [c_p]),
    "ud_proj_prep_w": (c_i, [c_p] * 3 + [c_i] * 3 + [c_p]),
    "ud_proj_fwd": (c_i, [c_p] * 8 + [c_i] * 6 + [c_p]),
    "ud_proj_prep_wt": (c_i, [c_p] * 3 + [c_i] * 3 + [c_p]),
    "ud_proj_split": (c_i, [c_p] * 3 + [ctypes.c_longlong, c_p]),
    "ud_proj_wgrad_1x1": (c_i, [c_p] * 5 + [c_i] * 4 + [c_p]),
    "ud_bn_merge_partials": (c_i, [c_p] * 5 + [c_i] * 2 + [c_p]),
    "ud_dyfi_mask_fwd": (c_i, [c_p] * 13 + [c_i] * 6 + [c_p]),
    "ud_dyfi_mask_bwd_workspace_bytes": (c_sz, [c_i, c_i]),
    "ud_dyfi_mask_bwd": (c_i, [c_p] * 19 + [c_sz] + [c_i] * 6 + [c_p]),
    "ud_triplet_fwd": (c_i, [c_p] * 4 + [c_i, c_i, c_p]),
    "ud_factorization_workspace_bytes": (c_sz, [c_i, c_i]),
    "ud_factorization_fwd": (c_i, [c_p] * 5 + [c_sz, c_i, c_i, c_f, c_f, c_p]),
    "ud_mask_kl_workspace_bytes": (c_sz, [c_i]),
    "ud_mask_kl_fwd": (c_i, [c_p] * 5 + [c_sz, c_i, c_i, c_p]),
    "ud_freq_style_workspace_bytes": (c_sz, [c_i] * 4),
    "ud_freq_style_transfer": (c_i, [c_p] * 5 + [c_sz] + [c_i] * 4 + [c_p]),
    "ud_cross_entropy_fwd": (c_i, [c_p] * 4 + [c_i, c_i, c_p]),
    "ud_bce_with_logits_fwd": (c_i, [c_p] * 4 + [c_i, c_p]),
    "ud_spatial_style_workspace_bytes": (c_sz, [c_i] * 3),
    "ud_spatial_style_transfer": (c_i, [c_p] * 5 + [c_sz] + [c_i] * 3 + [c_p]),
    "ud_coral_workspace_bytes": (c_sz, [c_i, c_i]),
    "ud_coral": (c_i, [c_p] * 4 + [c_sz, c_i, c_i, c_p]),
    "ud_gaussian_blur5": (c_i, [c_p, c_p, c_i, c_i, c_i, c_p]),
    "ud_downscale_nearest": (c_i, [c_p, c_p, c_i, c_i, c_i, c_f, c_p]),
    "ud_gaussian_blur5_bwd": (c_i, [c_p, c_p, c_i, c_i, c_i, c_p]),
    "ud_downscale_nearest_bwd": (c_i, [c_p, c_p, c_i, c_i, c_i, c_f, c_p]),
    "ud_sf_pack": (c_i, [c_p, c_p] + [c_i] * 5 + [c_p]),
    "ud_sf_unpack": (c_i, [c_p, c_p] + [c_i] * 5 + [c_p]),
    "ud_sf_mix_fwd": (c_i, [c_p] * 4 + [c_i] * 5 + [c_p]),
    "ud_sf_mix_bwd_workspace_bytes": (c_sz, [c_i] * 3),
    "ud_sf_mix_bwd": (c_i, [c_p] * 8 + [c_sz] + [c_i] * 5 + [c_p]),
    "ud_comm_buffer_bytes": (c_sz, [c_i, c_i]),
    "ud_comm_alloc": (c_i, [c_sz, ctypes.POINTER(c_p), c_p]),
    "ud_comm_open": (c_i, [c_p, ctypes.POINTER(c_p)]),
    "ud_comm_create": (c_i, [ctypes.POINTER(c_p), c_i, c_i, c_i, ctypes.POINTER(c_p)]),
    "ud_comm_gather": (c_i, [c_p, c_p, c_p, c_i, c_i, c_p]),
    "ud_comm_error": (c_i, [c_p]),
    "ud_kl_div_log_target_fwd": (c_i, [c_p] * 5 + [c_sz, c_i, c_i, c_p]),
    "ud_attack_workspace_bytes": (c_sz, [c_i, ctypes.c_longlong]),
    "ud_attack_step": (c_i, [c_p] * 8 + [c_f, c_f, c_i, c_i, ctypes.c_longlong, c_p, c_sz, c_p]),
    "ud_corrupt_workspace_bytes": (c_sz, [c_i] * 4),
    "ud_corrupt": (c_i, [c_p] * 3 + [c_i] * 4 + [c_f, ctypes.c_ulonglong, c_f, c_f, c_p, c_sz, c_p]),
}


def lib():
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                if not os.path.exists(LIB_PATH):
                    raise RuntimeError(
                        f"{LIB_PATH} is missing: build it with `python __graft_entry__.py` "
                        "(or `make -C unidefense_b200/csrc`). There is no CPU/PyTorch fallback.")
                L = ctypes.CDLL(LIB_PATH)
                ns = types.SimpleNamespace(_cdll=L)
                for name, (res, args) in SIGNATURES.items():
                    fn = getattr(L, name)
                    fn.restype = res
                    fn.argtypes = args
                    launches = res is c_i and len(args) > 1 and args[-1] is c_p
                    setattr(ns, name, _timed(fn) if launches else fn)
                _lib = ns
    return _lib


# Optional per-op device timing (bench.py's roofline leg): when PROFILE is a dict, every C-ABI call that
# passes through check() is bracketed by CUDA events on the launching stream: name -> [(start, end), ...].
PROFILE = None
_tls = threading.local()       # start events are per thread: backward runs on autograd's worker thread


def _pending():
    if not hasattr(_tls, "pending"):
        _tls.pending = []
    return _tls.pending


def _timed(fn):
    """Wrap a stream-taking entry point so that, when profiling, a start event precedes its launches."""
    def call(*args):
        if PROFILE is not None:
            ev = torch.cuda.Event(enable_timing=True)
            ev.record(torch.cuda.current_stream())
            _pending().append(ev)
        return fn(*args)
    return call


def check(rc: int, what: str = ""):
    if PROFILE is not None and _pending():
        ev0 = _pending().pop()
        ev1 = torch.cuda.Event(enable_timing=True)
        ev1.record(torch.cuda.current_stream())
        PROFILE.setdefault(what, []).append((ev0, ev1))
    if rc != 0:
        msg = lib().ud_last_error().decode(errors="replace")
        raise RuntimeError(f"unidefense_b200 {what} failed (code {rc}): {msg}")


def profile_summary():
    """-> {op: (calls, total_ms)} after a torch.cuda.synchronize()."""
    out = {}
    for k, evs in (PROFILE or {}).items():
        out[k] = (len(evs), sum(a.elapsed_time(b) for a, b in evs))
    return out


def ptr(t):
    if t is None:
        return None
    return t.data_ptr()


def stream():
    return torch.cuda.current_stream().cuda_stream


def require_cuda_f32(*tensors, also=()):
    """`also`: extra dtypes an entry point accepts for these tensors (the bf16 I/O variants)."""
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise RuntimeError("unidefense_b200 kernels need CUDA tensors (no CPU fallback)")
        if t.device.index != torch.cuda.current_device():
            raise RuntimeError(f"tensor on cuda:{t.device.index} but the current device is cuda:{torch.cuda.current_device()}: "
                               "the stream, workspace and twiddle tables belong to the current device "
                               "(call torch.cuda.set_device(local_rank) as the reference engines do)")
        if t.dtype != torch.float32 and t.dtype not in also:
            raise RuntimeError(f"unidefense_b200 kernels are fp32; got {t.dtype}")
        if not t.is_contiguous():
            raise RuntimeError("unidefense_b200 kernels need contiguous tensors")


_ws = {}
_ws_retired = []


def workspace(nbytes: int, device) -> torch.Tensor:
    """Grow-only byte workspace per (device, stream); safe because every kernel that uses it is enqueued on
    that same stream.  Superseded buffers are kept alive for the process lifetime: a captured CUDA graph may
    still hold their addresses."""
    key = (device.index if device.index is not None else torch.cuda.current_device(), stream())
    t = _ws.get(key)
    if t is None or t.numel() < nbytes:
        if t is not None:
            _ws_retired.append(t)
        t = torch.empty(max(int(nbytes), 1 << 20), dtype=torch.uint8, device=device)
        _ws[key] = t
    return t
