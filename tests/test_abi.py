"""The C-ABI library loads and exports every symbol include/unidefense_b200.h declares; the ctypes
binding table covers exactly that set.  No compute calls (CPU only)."""
import ctypes
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    src = open(os.path.join(ROOT, "include", "unidefense_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"UD_API\s+[\w\s\*]+?\b(ud_\w+)\s*\(", src)))


def test_every_declared_symbol_is_exported_and_bound():
    from unidefense_b200 import _lib
    names = _declared()
    assert len(names) >= 30
    so = ctypes.CDLL(_lib.LIB_PATH)
    for n in names:
        assert hasattr(so, n), f"{n} declared in the header but not exported by the .so"
    assert set(names) == set(_lib.SIGNATURES), (set(names) ^ set(_lib.SIGNATURES))


def test_status_calls_without_gpu():
    from unidefense_b200 import _lib
    L = _lib.lib()
    assert L.ud_version() >= 101
    assert L.ud_fft_size_supported(380) == 1 and L.ud_fft_size_supported(299) == 1
    assert L.ud_fft_size_supported(58) == 0          # 29 is not a mixed-radix factor ...
    assert L.ud_fft_size_any(58) == 1                # ... such sizes run Bluestein
    assert L.ud_fft_size_supported(2048) == 0 and L.ud_fft_size_any(2048) == 0        # > UD_FFT_MAX_N
    assert L.ud_rfft2_workspace_bytes(2, 3, 12, 12) == 0 and L.ud_rfft2_workspace_bytes(2, 3, 95, 95) == 6 * 95 * 48 * 8
    assert L.ud_recon_tail_signs_bytes(2, 3, 380, 380) == 2 * 3 * 380 * 191
    assert L.ud_recon_tail_workspace_bytes(32, 3, 192, 192, 380, 380) > 0
    assert L.ud_launch_count() >= 0
    # invalid arguments are rejected before any CUDA call, with a message
    rc = L.ud_recon_tail_fwd(None, None, None, None, None, None, None, 0, 1, 3, 4, 4, 58, 2058, 1, None)
    assert rc < 0 and b"unsupported" in L.ud_last_error()
    rc = L.ud_factorization_fwd(None, None, None, None, None, 0, 1, 8, 0.005, 1e-6, None)
    assert rc < 0 and b"N >= 2" in L.ud_last_error()
