"""The Fourier-basis definitions of oracle/fourier.py (which csrc/ud_fourier.cu implements) without a GPU: unit norm and
a two-point spectrum of the fp64 basis, canonical pairs and unique counts, the default grid stride, the Philox sign
keying, the batched corrupt.auc against scipy's rank formula, and the C ABI's argument checks."""
import ctypes

import numpy as np
import pytest
import torch
from scipy.stats import rankdata

from oracle import corrupt as C
from oracle import fourier as FO

SIZES = [(380, 380), (299, 299), (45, 67), (64, 96)]


def _freqs(H, W):
    """DC, small and negative u, the Nyquist row and column (u = H/2, v = W/2 where even) and the largest odd-size
    frequencies."""
    us = [0, 1, -1, 7, -13, H // 2, -(H // 2), (H - 1) // 2]
    vs = [0, 1, 5, W // 2, (W - 1) // 2]
    return [(u, v) for u in us for v in vs]


@pytest.mark.parametrize("H,W", SIZES)
def test_basis_has_unit_norm_and_two_spectral_points(H, W):
    worst_norm = worst_leak = 0.0
    for u, v in _freqs(H, W):
        U = FO.basis(u, v, H, W)
        worst_norm = max(worst_norm, abs(float((U * U).sum()) - 1.0))
        spec = np.fft.fft2(U)
        keep = np.zeros(spec.shape, bool)
        keep[u % H, v % W] = keep[(-u) % H, (-v) % W] = True
        e = np.abs(spec) ** 2
        worst_leak = max(worst_leak, float(e[~keep].sum() / e.sum()))
        assert np.array_equal(U, FO.basis(-u, -v, H, W)), (u, v)
    assert worst_norm < 1e-12, worst_norm
    assert worst_leak < 1e-20, worst_leak


@pytest.mark.parametrize("H,W", SIZES + [(64, 64), (1, 7), (8, 1)])
def test_canonical_pairs_and_unique_counts(H, W):
    from unidefense_b200 import fourier
    for u in range(-H, H + 1, max(1, H // 24)):
        for v in range(-W, W + 1, max(1, W // 24)):
            c = FO.canonical(u, v, H, W)
            assert c == FO.canonical(-u, -v, H, W) == fourier.canonical(u, v, H, W)
            assert 0 <= c[0] < H and 0 <= c[1] < W
            assert c <= ((-c[0]) % H, (-c[1]) % W)
    for radius in (1, 2, 4, 15):
        s = FO.default_stride(H, W, radius)
        if s < 1:
            continue
        u, v, groups = FO.grid(H, W, radius)
        brute = {min((a % H, b % W), ((-a) % H, (-b) % W)) for a in u for b in v}
        assert set(groups) == brute
        gu, gv, table, index = fourier.grid(H, W, radius, s)
        assert (gu, gv) == (u, v) and len(table) == len(set(table)) == len(brute)
        for key, pos in groups.items():
            assert all(table[index[i][j]] == key for i, j in pos)


def test_nyquist_column_shrinks_the_unique_count():
    """At 64^2 with radius 4 and stride 8 the v = 32 column is its own mirror: 34 unique points, not the 41 a
    DC-only formula gives."""
    u, v, groups = FO.grid(64, 64, 4, 8)
    assert len(u) * len(v) == 45 and len(groups) == 34
    assert (2 * 4 + 1) * (4 + 1) - 4 == 41


def test_default_stride():
    assert FO.default_stride(380, 380, 15) == 12
    u, v, groups = FO.grid(380, 380, 15)
    assert max(u) == 180 and len(u) == 31 and len(v) == 16 and len(groups) == 481
    assert FO.default_stride(299, 299, 15) == 9
    assert FO.default_stride(64, 96, 15) == 2 and FO.default_stride(64, 96, 4) == 8


def test_signs_known_answers_and_keying():
    seed, ids = 0xDEADBEEF12345678, [0, 5, (1 << 40) + 3, -2]
    r = FO.signs(ids, 128, 12, 7, seed)
    for n, i in enumerate(ids):
        words = C.philox4x32_10(((12 << 16) | 7, i & 0xFFFFFFFF, (i & 0xFFFFFFFFFFFFFFFF) >> 32, 0),
                                (seed & 0xFFFFFFFF, (seed >> 32) ^ 0x464F5552))
        bits = [(int(words[c >> 5]) >> (c & 31)) & 1 for c in range(128)]
        assert r[n].tolist() == [-1.0 if b else 1.0 for b in bits]
    assert FO.SIGN_TAG not in (C.BLOCK_TAG, C.NOISE_TAG, 0x534D5448)
    # Random123's published known answer for the generator under the signs (ctr = key = 0)
    assert [int(w) for w in C.philox4x32_10((0, 0, 0, 0), (0, 0))] == [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]
    # ctr = 0, key = (0, tag): sample 0 at DC with seed 0
    w0 = int(C.philox4x32_10((0, 0, 0, 0), (0, 0x464F5552))[0])
    assert FO.signs([0], 3, 0, 0, 0)[0].tolist() == [-1.0 if (w0 >> c) & 1 else 1.0 for c in range(3)]
    # deterministic, keyed by id, not by position; frequency and seed change them
    assert np.array_equal(FO.signs(ids[::-1], 128, 12, 7, seed), r[::-1])
    assert np.array_equal(FO.signs(ids[2:3], 128, 12, 7, seed), r[2:3])
    assert not np.array_equal(FO.signs(ids, 128, 12, 8, seed), r)
    assert not np.array_equal(FO.signs(ids, 128, 12, 7, seed + 1), r)
    assert 0.4 < (r > 0).mean() < 0.6


def test_perturb_is_the_scaled_basis_plus_clamp():
    H, W = 45, 67
    rng = np.random.default_rng(0)
    x = rng.uniform(-1, 1, (2, 3, H, W)).astype(np.float32)
    uu, vv = FO.canonical(-7, 5, H, W)
    r = FO.signs([0, 1], 3, uu, vv, 9)
    y = FO.perturb(x, uu, vv, 0.5, [0, 1], 9)
    U = FO.basis(-7, 5, H, W)
    want = np.clip(x.astype(np.float64) + 0.5 * r[:, :, None, None] * U, -1, 1)
    assert np.abs(y - want).max() < 1e-7          # s carries the kernel's fp32 rounding of eps*a
    free = (y > -1) & (y < 1)
    assert free.mean() > 0.9


def _auc_scipy(s, y):
    r = rankdata(s)
    npos = int(y.sum())
    return (r[y == 1].sum() - npos * (npos + 1) / 2) / (npos * (len(y) - npos))


def test_batched_auc_matches_scipy_row_by_row():
    from unidefense_b200._evaluator import auc
    rng = np.random.default_rng(4)
    y = np.array([0, 1] * 20)
    s = rng.integers(0, 6, (7, 40)).astype(np.float32) / 5           # many ties
    s[3] = rng.standard_normal(40)
    s[4] = 0.5                                                        # one tie group
    got = auc(torch.from_numpy(s), torch.from_numpy(y))
    assert got.dtype == torch.float64 and got.shape == (7,)
    for i in range(7):
        assert abs(float(got[i]) - _auc_scipy(s[i].astype(np.float64), y)) < 1e-12, i
        assert float(auc(torch.from_numpy(s[i]), torch.from_numpy(y))) == float(got[i])
    s3 = torch.from_numpy(s).view(7, 1, 40).expand(7, 2, 40)
    assert torch.equal(auc(s3, torch.from_numpy(y)), got[:, None].expand(7, 2))
    one = auc(torch.from_numpy(s), torch.zeros(40, dtype=torch.long))
    assert bool(torch.isnan(one).all())


def _auc_parent(scores, labels):
    """corrupt.auc as it stood before it took [..., n]: the 1-D result must not move."""
    n = scores.numel()
    v, order = torch.sort(scores.double())
    pos = (labels[order] == 1).double()
    idx = torch.arange(n, device=scores.device)
    new = torch.ones(n, dtype=torch.bool, device=scores.device)
    new[1:] = v[1:] != v[:-1]
    end = torch.ones_like(new)
    end[:-1] = new[1:]
    first = torch.cummax(torch.where(new, idx, 0), 0).values
    last = torch.flip(torch.cummin(torch.flip(torch.where(end, idx, n - 1), [0]), 0).values, [0])
    rank = (first + last).double() / 2 + 1
    n_pos = pos.sum()
    n_neg = n - n_pos
    return ((rank * pos).sum() - n_pos * (n_pos + 1) / 2) / (n_pos * n_neg)


def test_one_dimensional_auc_is_unchanged():
    from unidefense_b200._evaluator import auc
    rng = np.random.default_rng(5)
    for n in (1, 2, 9, 100, 1001):
        y = torch.from_numpy(rng.integers(0, 2, n))
        for s in (torch.from_numpy(rng.standard_normal(n).astype(np.float32)),
                  torch.from_numpy(rng.integers(0, 4, n).astype(np.float32))):
            a, b = auc(s, y), _auc_parent(s, y)
            assert a.shape == b.shape == () and (torch.equal(a, b) or (bool(a.isnan()) and bool(b.isnan())))


def test_c_abi_rejects_bad_arguments_before_any_cuda_call():
    from unidefense_b200 import _lib
    L = _lib.lib()
    assert L.ud_version() >= 105
    buf = ctypes.create_string_buffer(1 << 16)
    p = ctypes.cast(buf, ctypes.c_void_p).value                # any non-null address: nothing is launched
    q = p + 8192

    def call(x=p, y=q, freqs=p, F=3, f=p, eps=p, seed=p, lo=-1.0, hi=1.0, N=2, Cc=3, H=8, W=8):
        return L.ud_fourier_perturb(x, y, freqs, F, f, eps, None, seed, lo, hi, N, Cc, H, W, None)

    for kw, msg in ((dict(N=0), b"bad shape"), (dict(Cc=0), b"bad shape"), (dict(H=0), b"bad shape"),
                    (dict(W=-1), b"bad shape"), (dict(N=65536), b"65535"), (dict(Cc=129), b"C=129 > 128"),
                    (dict(H=4097, W=1), b"4096"), (dict(H=4096, W=4097), b"4096"), (dict(F=0), b"F=0"),
                    (dict(x=None), b"null pointer"), (dict(y=None), b"null pointer"), (dict(f=None), b"null pointer"),
                    (dict(eps=None), b"null pointer"), (dict(seed=None), b"null pointer"),
                    (dict(freqs=None), b"null pointer"), (dict(lo=1.0, hi=-1.0), b"lo <= hi"),
                    (dict(lo=float("nan")), b"lo <= hi"), (dict(y=p), b"overlaps"), (dict(y=p + 4), b"overlaps"),
                    (dict(x=q + 4 * 2 * 3 * 64 - 4), b"overlaps")):
        rc = call(**kw)
        assert rc < 0 and msg in L.ud_last_error(), (kw, rc, L.ud_last_error())
    assert call(N=65536) == -2 and call(N=0) == -1                 # UD_ERR_UNSUPPORTED, UD_ERR_INVALID
