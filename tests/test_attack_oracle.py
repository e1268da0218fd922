"""The PGD / FGSM step composition of oracle/attack.py (which csrc/ud_attack.cu mirrors) in fp64, without a GPU:
the projections keep the iterate in the eps-ball and the input range and are idempotent, FGSM is the closed form, and
best-iterate selection is strict.  Also the C ABI's argument checks, which reject before any CUDA call."""
import ctypes

import pytest
import torch

from oracle import attack as A

LO, HI = -1.0, 1.0


def _case(N=4, shape=(3, 9, 7), seed=0):
    g = torch.Generator().manual_seed(seed)
    x0 = torch.rand(N, *shape, generator=g, dtype=torch.float64) * 2 - 1
    x0[0, 0, 0] = HI                                  # pixels on the range boundary
    x0[0, 0, 1] = LO
    grad = torch.randn(N, *shape, generator=g, dtype=torch.float64)
    grad[1, 1] = 0.0                                  # sign(0) = 0
    eps = torch.tensor([0.0, 0.01, 16 / 255, 0.5], dtype=torch.float64)[:N]
    return x0, grad, eps, g


@pytest.mark.parametrize("norm", ["linf", "l2"])
def test_steps_stay_in_the_ball_and_the_range(norm):
    x0, grad, eps, g = _case()
    step = A.linf_step if norm == "linf" else A.l2_step
    start = A.random_start_linf if norm == "linf" else A.random_start_l2
    alpha = 2.5 * eps / 3
    x = start(x0, eps, LO, HI, g)
    for _ in range(5):
        d = (x - x0).flatten(1)
        radius = d.abs().amax(1) if norm == "linf" else d.norm(dim=1)
        assert bool((radius <= eps * (1 + 1e-12) + 1e-15).all()), (radius, eps)
        assert float(x.min()) >= LO and float(x.max()) <= HI
        x = step(x0, x, grad, eps, alpha, LO, HI)
        grad = torch.randn(x0.shape, generator=g, dtype=torch.float64)
    # eps = 0 pins the iterate to x0
    assert torch.equal(x[0], x0[0])


@pytest.mark.parametrize("norm", ["linf", "l2"])
def test_projection_is_idempotent(norm):
    """A step of length zero (alpha = 0) from a projected point leaves it where it is."""
    x0, grad, eps, g = _case(seed=1)
    step = A.linf_step if norm == "linf" else A.l2_step
    big = torch.full_like(eps, 10.0)                  # far outside the ball: the projection acts
    x1 = step(x0, x0, grad, eps, big, LO, HI)
    x2 = step(x0, x1, grad, eps, torch.zeros_like(eps), LO, HI)
    torch.testing.assert_close(x2, x1, rtol=0, atol=1e-15)
    if norm == "l2":                                  # a long step lands on the sphere (unless the clamp cuts it)
        r = (x1 - x0).flatten(1).norm(dim=1)
        assert float(r[2]) <= float(eps[2]) * (1 + 1e-12)


def test_fgsm_is_the_signed_gradient_step():
    x0, grad, eps, _ = _case(seed=2)
    got = A.linf_step(x0, x0, grad, eps, eps, LO, HI)
    want = torch.clamp(x0 + eps.view(-1, 1, 1, 1) * torch.sign(grad), LO, HI)
    torch.testing.assert_close(got, want, rtol=0, atol=4e-16)


def test_l2_zero_gradient_and_zero_radius():
    x0, grad, eps, _ = _case(seed=3)
    grad.zero_()
    got = A.l2_step(x0, x0, grad, eps, torch.ones_like(eps), LO, HI)       # u = 0 / 1e-12 = 0, d = 0, 0/0 -> 1
    assert torch.equal(got, x0)


def test_select_is_strict_and_nan_never_improves():
    loss = torch.tensor([1.0, 2.0, float("nan"), 0.5], dtype=torch.float64)
    best = torch.tensor([0.5, 2.0, 0.1, float("-inf")], dtype=torch.float64)
    xa = torch.full((4, 3), 7.0, dtype=torch.float64)
    xb = torch.zeros(4, 3, dtype=torch.float64)
    nb, nx, imp = A.select(loss, best, xa, xb)
    assert imp.tolist() == [True, False, False, True]
    assert nb.tolist()[:2] == [1.0, 2.0] and nb[2] == 0.1 and nb[3] == 0.5
    assert torch.equal(nx[imp], xa[imp]) and torch.equal(nx[~imp], xb[~imp])


def test_c_abi_rejects_bad_arguments_before_any_cuda_call():
    from unidefense_b200 import _lib
    L = _lib.lib()
    assert L.ud_version() >= 102
    nws = L.ud_attack_workspace_bytes(4, 3 * 299 * 299)
    assert nws > 0 and L.ud_attack_workspace_bytes(0, 10) == 0
    ws = ctypes.create_string_buffer(nws)
    p = ctypes.cast(ws, ctypes.c_void_p).value                 # any non-null address: nothing is launched

    def call(N=4, P=3 * 299 * 299, norm=0, lo=-1.0, hi=1.0, ws_bytes=nws):
        return L.ud_attack_step(p, p, p, p, p, p, p, p, lo, hi, norm, N, P, p, ws_bytes, None)

    for kw, msg in ((dict(N=0), b"bad shape"), (dict(P=0), b"bad shape"), (dict(norm=1), b"unknown norm"),
                    (dict(lo=1.0, hi=-1.0), b"lo="), (dict(ws_bytes=nws - 1), b"workspace")):
        rc = call(**kw)
        assert rc < 0 and msg in L.ud_last_error(), (kw, rc, L.ud_last_error())
    assert call(ws_bytes=nws - 1) == -4                        # UD_ERR_WORKSPACE
