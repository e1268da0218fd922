"""The attribution and faithfulness definitions of oracle/explain.py (which csrc/ud_explain.cu and the rank mode of
csrc/ud_style_sort.cu implement), without a GPU: trapezoid weights, IG completeness, the SmoothGrad noise stream, the
radix-key rank against numpy's stable argsort, the curve thresholds and AUC, and the C ABI's argument checks."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import corrupt as C
from oracle import explain as E


@pytest.mark.parametrize("m", [1, 2, 7, 32, 64])
def test_trapezoid_weights_sum_to_one(m):
    alpha, w = E.ig_tables(m)
    assert len(alpha) == len(w) == m + 1 and alpha[0] == 0.0 and alpha[-1] == 1.0
    assert abs(w.sum() - 1.0) < 1e-15
    assert w[0] == w[-1] == 0.5 / m


def test_ig_is_exact_on_a_quadratic():
    """The gradient of a quadratic is linear along the straight path, so the trapezoid rule is exact at any m."""
    rng = np.random.default_rng(0)
    A = rng.standard_normal((12, 12))
    A = A + A.T
    c = rng.standard_normal(12)
    f = lambda v: 0.5 * v @ A @ v + c @ v       # noqa: E731
    grad = lambda v: A @ v + c                  # noqa: E731
    x, b = rng.standard_normal(12), rng.standard_normal(12) * 0.1
    for m in (1, 3, 16):
        _, delta = E.integrated_gradients(f, grad, x, b, m)
        assert abs(delta) < 1e-12 * max(1.0, abs(f(x))), (m, delta)


def test_ig_completeness_error_falls_quadratically():
    """On a smooth non-quadratic F the trapezoid error is O(1/m^2): doubling m divides |delta| by about 4."""
    rng = np.random.default_rng(1)
    wv = rng.standard_normal(20)
    f = lambda v: np.log1p(np.exp(v @ wv)) + np.sin(v).sum()             # noqa: E731
    grad = lambda v: wv / (1.0 + np.exp(-(v @ wv))) + np.cos(v)         # noqa: E731
    x, b = rng.uniform(-1, 1, 20), np.full(20, -1.0)
    d = [abs(E.integrated_gradients(f, grad, x, b, m)[1]) for m in (8, 16, 32, 64)]
    for lo_m, hi_m in zip(d, d[1:]):
        assert 3.0 < lo_m / hi_m < 5.0, d


def test_noise_counters_and_keys():
    """Element e of draw k is normal e & 3 of Philox counter (e >> 2, id_lo, id_hi, k) under the SmoothGrad key."""
    P, sid, seed, k = 23, (1 << 40) + 5, 0xDEADBEEF12345678, 3
    z = E.normals(P, sid, seed, k)
    for e in (0, 1, 2, 3, 4, 13, 22):
        words = C.philox4x32_10((e >> 2, sid & 0xFFFFFFFF, sid >> 32, k),
                                ((seed & 0xFFFFFFFF), (seed >> 32) ^ 0x534D5448))
        pair = C.box_muller(words[0], words[1]) if e & 3 < 2 else C.box_muller(words[2], words[3])
        assert float(z[e]) == float(pair[e & 1]), e
    assert E.NOISE_TAG not in (C.BLOCK_TAG, C.NOISE_TAG)
    # Random123's published known answer (ctr = key = 0) for the underlying generator
    got = [int(v) for v in C.philox4x32_10((0, 0, 0, 0), (0, 0))]
    assert got == [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]


def test_noise_moments_over_a_million_draws():
    z = E.normals(1_000_000, 7, 11, 0)
    assert abs(z.mean()) < 5e-3 and abs(z.var() - 1.0) < 5e-3
    assert abs((z ** 3).mean()) < 1e-2 and abs((z ** 4).mean() - 3.0) < 3e-2
    assert abs(np.corrcoef(z[:-1], z[1:])[0, 1]) < 5e-3


def test_noise_is_keyed_by_id_and_draw_not_position():
    a = E.normals(100, 42, 9, 1)
    assert np.array_equal(a, E.normals(100, 42, 9, 1))
    assert np.array_equal(a[:37], E.normals(37, 42, 9, 1))             # a prefix does not depend on the length
    assert not np.allclose(a, E.normals(100, 43, 9, 1))
    assert not np.allclose(a, E.normals(100, 42, 9, 2))
    assert not np.allclose(a, E.normals(100, 42, 10, 1))


def _rank_numpy(m):
    flat = np.asarray(m, np.float32).reshape(m.shape[0], -1)
    order = np.argsort(-flat, axis=1, kind="stable")
    rank = np.empty_like(order)
    for n in range(flat.shape[0]):
        rank[n, order[n]] = np.arange(flat.shape[1])
    return rank.reshape(m.shape)


def test_rank_keys_match_numpy_stable_argsort():
    rng = np.random.default_rng(2)
    maps = [rng.standard_normal((3, 17, 19)).astype(np.float32),
            np.zeros((2, 8, 8), np.float32),                                  # all equal
            np.round(rng.uniform(0, 1, (2, 31, 29)) * 255).astype(np.float32) / 255]   # 8-bit quantised: many ties
    m = rng.standard_normal((2, 16, 16)).astype(np.float32)
    m[0, 0, :5] = np.nan
    m[0, 3, 3] = -np.nan
    m[1, 2, :4] = [np.inf, -np.inf, 0.0, -0.0]
    m[1, 5, :3] = [-0.0, 0.0, -0.0]
    maps.append(m)
    for mp in maps:
        assert np.array_equal(E.rank_desc(mp), _rank_numpy(mp))


def test_thresholds_endpoints_and_auc():
    assert E.thresholds(4, 10) == [0, 2, 5, 7, 10]
    assert E.thresholds(16, 380 * 380)[-1] == 380 * 380 and E.thresholds(16, 380 * 380)[0] == 0
    x = torch.arange(2 * 3 * 2 * 2, dtype=torch.float64).view(2, 3, 2, 2)
    b = torch.full_like(x, -1.0)
    rank = torch.tensor(E.rank_desc(np.random.default_rng(3).standard_normal((2, 2, 2))))
    assert torch.equal(E.masked(x, b, rank, 0, False), x) and torch.equal(E.masked(x, b, rank, 4, False), b)
    assert torch.equal(E.masked(x, b, rank, 0, True), b) and torch.equal(E.masked(x, b, rank, 4, True), x)
    half = E.masked(x, b, rank, 2, False)
    assert torch.equal(half, torch.where((rank < 2)[:, None], b, x))
    s = torch.tensor([[1.0, 0.5, 0.0], [0.2, 0.2, 0.2]], dtype=torch.float64)
    torch.testing.assert_close(E.auc(s), torch.tensor([0.5, 0.2], dtype=torch.float64))


def test_objective_heads_agree():
    """log p(target) of a one-logit head equals that of the two-logit head with logits (0, z)."""
    z = torch.tensor([[-3.0], [0.5], [2.0]], dtype=torch.float64)
    two = torch.cat([torch.zeros_like(z), z], 1)
    for t in ([0, 1, 1], [1, 0, 0]):
        t = torch.tensor(t)
        torch.testing.assert_close(E.objective(z, t), E.objective(two, t))
    assert E.predicted(z).tolist() == E.predicted(two).tolist() == [0, 1, 1]


def test_c_abi_rejects_bad_arguments_before_any_cuda_call():
    from unidefense_b200 import _lib
    L = _lib.lib()
    assert L.ud_version() >= 104
    buf = ctypes.create_string_buffer(1 << 16)
    p = ctypes.cast(buf, ctypes.c_void_p).value                # any non-null address: nothing is launched
    q = p + 4096

    def step(x=p, N=4, Cc=3, H=8, W=8, steps=3, method=0, alpha=p, sigma=None, seed=None, k=p, out=q):
        return L.ud_attrib_step(x, None, 0.0, p, p, out, q + 64, q + 128, k, alpha, p, sigma, None, seed, steps,
                                method, N, Cc, H, W, None)

    for kw, msg in ((dict(N=0), b"bad shape"), (dict(H=0), b"bad shape"), (dict(method=2), b"unknown method"),
                    (dict(steps=0), b"steps=0"), (dict(N=65536), b"65535"), (dict(x=None), b"null pointer"),
                    (dict(k=None), b"null pointer"), (dict(alpha=None), b"step table"),
                    (dict(method=1), b"sigma and seed"), (dict(out=p), b"alias")):
        rc = step(**kw)
        assert rc < 0 and msg in L.ud_last_error(), (kw, rc, L.ud_last_error())

    nws = L.ud_rank_desc_workspace_bytes(2, 64)
    assert nws == 2 * 64 * 16 and L.ud_rank_desc_workspace_bytes(0, 64) == 0
    for args, msg in (((p, q, 0, 64, p, nws), b"bad shape"), ((p, q, 70000, 64, p, nws), b"65535"),
                      ((None, q, 2, 64, p, nws), b"null pointer"), ((p, q, 2, 64, p, nws - 1), b"workspace")):
        rc = L.ud_rank_desc(*args, None)
        assert rc < 0 and msg in L.ud_last_error(), (args, rc, L.ud_last_error())
    assert L.ud_rank_desc(p, q, 2, 64, p, nws - 1, None) == -4                 # UD_ERR_WORKSPACE

    def mask(x=p, y=q, N=2, points=4, ins=0, j=p):
        return L.ud_attrib_mask(x, None, 0.0, p, p, j, points, y, ins, N, 3, 8, 8, None)

    for kw, msg in ((dict(N=0), b"bad shape"), (dict(ins=2), b"insertion must be"), (dict(points=0), b"points=0"),
                    (dict(N=65536), b"65535"), (dict(j=None), b"null pointer"), (dict(y=p), b"alias")):
        rc = mask(**kw)
        assert rc < 0 and msg in L.ud_last_error(), (kw, rc, L.ud_last_error())
