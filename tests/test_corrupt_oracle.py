"""The corruption definitions of oracle/corrupt.py (which csrc/ud_corrupt.cu implements), without a GPU: Philox known
answers, the JPEG quantisation tables, identities at neutral parameters, structure (blur weights, reflect-101 borders,
block squares, Box-Muller moments), realism (the JPEG definition against libjpeg through PIL; severities that
degrade monotonically), the device-side AUC against scipy, and the C ABI's argument checks."""
import ctypes
import io

import numpy as np
import pytest
import torch

from oracle import corrupt as C

LO, HI = -1.0, 1.0


def _psnr(a, b):
    m = np.mean((a.astype(np.float64) - b.astype(np.float64)) ** 2)
    return 10 * np.log10(255 ** 2 / max(m, 1e-12))


def _u8(x):
    """[3, H, W] in [-1, 1] -> HxWx3 uint8 levels."""
    return C.to_levels(x[None], LO, HI)[0].transpose(1, 2, 0).astype(np.uint8)


def test_philox_known_answers():
    assert [int(v) for v in C.philox4x32_10((0, 0, 0, 0), (0, 0))] == [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]
    m = 0xFFFFFFFF
    assert [int(v) for v in C.philox4x32_10((m, m, m, m), (m, m))] == [0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD]


def test_quantisation_tables():
    assert np.array_equal(C.qtable(C.LUM, 50), C.LUM) and np.array_equal(C.qtable(C.CHR, 50), C.CHR)
    assert (C.qtable(C.LUM, 100) == 1).all() and (C.qtable(C.CHR, 100) == 1).all()
    assert C.qtable(C.LUM, 10)[0, 0] == 80
    assert C.qtable(C.LUM, 1).max() == 255


@pytest.mark.parametrize("kind,param", [("saturation", 1.0), ("contrast", 1.0), ("pixelate", 1), ("blur", 1)])
def test_neutral_parameters_return_the_8bit_input(kind, param):
    x = C.test_images(2, 37, 45, seed=1)
    y, unc = C.corrupt(x, kind, param)
    assert np.array_equal(y, C.from_levels(C.to_levels(x, LO, HI), LO, HI))


def test_levels_round_trip_is_on_the_8bit_grid():
    x = C.test_images(1, 16, 16)
    p = C.to_levels(x, LO, HI)
    assert p.min() >= 0 and p.max() <= 255 and np.array_equal(p, np.rint(p))
    assert np.array_equal(C.to_levels(C.from_levels(p, LO, HI), LO, HI), p)


def test_blur_weights_and_reflect101():
    for k in (1, 7, 9, 13, 17, 21, 31):
        w = C.blur_weights(k)
        assert w.size == k and abs(w.sum() - 1) < 1e-15 and np.allclose(w, w[::-1]) and w.argmax() == k // 2
    n = 6
    assert C.reflect101(np.arange(-3, 0), n).tolist() == [3, 2, 1]        # ... d c b | a b c ...
    assert C.reflect101(np.arange(n, n + 3), n).tolist() == [4, 3, 2]     # ... d e f | e d c ...
    assert C.reflect101(np.arange(n), n).tolist() == list(range(n))


@pytest.mark.parametrize("H,W", [(64, 64), (8, 8), (17, 300)])
def test_block_squares_stay_inside_and_cover_exactly(H, W):
    x = C.test_images(3, H, W, seed=2)
    p = C.to_levels(x, LO, HI)
    p[p == 128] = 127                                   # so that 128 marks the squares only
    x = C.from_levels(p, LO, HI)
    ids = np.array([5, 2 ** 40 + 3, -7])
    y, _ = C.corrupt(x, "block", 80, ids=ids, seed=11)
    q = C.to_levels(y, LO, HI)
    for n in range(3):
        sq = C.block_squares(80, H, W, ids[n], 11)
        assert (sq >= 0).all() and (sq[:, 0] + 8 <= H).all() and (sq[:, 1] + 8 <= W).all()
        cover = np.zeros((H, W), bool)
        for r, c in sq:
            cover[r:r + 8, c:c + 8] = True
        assert np.array_equal(q[n] == 128, np.broadcast_to(cover, q[n].shape))
        assert np.array_equal(q[n][:, ~cover], p[n][:, ~cover])


def test_block_squares_nest_across_severities():
    for k0, k1 in zip(C.LEVELS["block"][:-1], C.LEVELS["block"][1:]):
        assert np.array_equal(C.block_squares(k1, 380, 299, 9, 4)[:k0], C.block_squares(k0, 380, 299, 9, 4))


def test_box_muller_moments():
    z0, z1, z2 = C.noise_normals(1000, 1000, 3, 123)
    for z in (z0, z1, z2):
        z = z.ravel()
        assert abs(z.mean()) < 3 / np.sqrt(z.size)
        assert abs(z.var() - 1) < 0.01
    assert abs(np.corrcoef(z0.ravel(), z1.ravel())[0, 1]) < 0.01


@pytest.mark.parametrize("H,W", [(380, 380), (299, 299), (64, 64)])
def test_jpeg_definition_tracks_libjpeg(H, W):
    """Against PIL's libjpeg at 4:2:0: within 38.3 dB PSNR of its output, and its distortion of the clean image within
    0.7 dB of libjpeg's (the measured 40.3 dB and 0.2 dB, with 2 dB and 0.5 dB of slack)."""
    Image = pytest.importorskip("PIL.Image")
    x = C.test_images(2, H, W, seed=3)
    for q in C.LEVELS["jpeg"]:
        y, _ = C.corrupt(x, "jpeg", q)
        for n in range(2):
            im, ours = _u8(x[n]), _u8(y[n])
            buf = io.BytesIO()
            Image.fromarray(im).save(buf, "JPEG", quality=q, subsampling=2)
            lib = np.asarray(Image.open(io.BytesIO(buf.getvalue())).convert("RGB"))
            assert _psnr(ours, lib) >= 38.3, (H, q, _psnr(ours, lib))
            assert abs(_psnr(ours, im) - _psnr(lib, im)) <= 0.7, (H, q, _psnr(ours, im), _psnr(lib, im))


@pytest.mark.parametrize("kind", C.KINDS)
def test_severities_degrade_monotonically(kind):
    x = C.test_images(4, 96, 80, seed=4)
    clean = C.from_levels(C.to_levels(x, LO, HI), LO, HI)
    mse = [float(np.mean((C.corrupt(x, kind, p, seed=5)[0] - clean) ** 2)) for p in C.LEVELS[kind]]
    assert all(b >= a for a, b in zip(mse[:-1], mse[1:])), mse
    assert mse[0] > 0


def test_uncertain_masks_are_rare():
    x = C.test_images(2, 299, 299, seed=0)          # the GPU tests' images
    for kind in ("noise", "blur", "jpeg"):
        for p in C.LEVELS[kind]:
            _, unc = C.corrupt(x, kind, p)
            assert unc.mean() <= 0.005, (kind, p, unc.mean())


def test_device_auc_matches_the_rank_formula():
    from scipy.stats import rankdata
    from unidefense_b200 import corrupt
    g = torch.Generator().manual_seed(0)
    for n, ties in ((50, False), (64, True), (7, True)):
        s = torch.rand(n, generator=g, dtype=torch.float64)
        if ties:
            s = torch.round(s * 4) / 4
        y = torch.randint(0, 2, (n,), generator=g)
        y[0], y[1] = 0, 1
        r = rankdata(s.numpy())
        npos = int(y.sum())
        want = (r[y.numpy() == 1].sum() - npos * (npos + 1) / 2) / (npos * (n - npos))
        assert abs(float(corrupt.auc(s, y)) - want) < 1e-12
    assert np.isnan(float(corrupt.auc(torch.rand(5), torch.ones(5, dtype=torch.long))))


def test_c_abi_rejects_bad_arguments_before_any_cuda_call():
    from unidefense_b200 import _lib
    L = _lib.lib()
    assert L.ud_version() >= 103
    nws = L.ud_corrupt_workspace_bytes(6, 4, 299, 299)
    assert nws >= 4 * (299 * 299 + 2 * 150 * 150) * 4 and L.ud_corrupt_workspace_bytes(3, 4, 299, 299) == 0
    buf = ctypes.create_string_buffer(16)
    p = ctypes.cast(buf, ctypes.c_void_p).value                # any non-null address: nothing is launched
    x, y = p, p + (1 << 40)

    def call(kind=6, param=50.0, N=4, H=299, W=299, lo=-1.0, hi=1.0, ws_bytes=nws, xp=x):
        return L.ud_corrupt(xp, y, None, N, H, W, kind, param, 0, lo, hi, p, ws_bytes, None)

    cases = ((dict(kind=7), b"unknown kind"), (dict(kind=-1), b"unknown kind"),
             (dict(param=0.0), b"jpeg parameter"), (dict(param=50.5), b"jpeg parameter"),
             (dict(kind=4, param=8.0), b"blur parameter"), (dict(kind=4, param=33.0), b"blur parameter"),
             (dict(kind=0, param=1.5), b"saturation parameter"), (dict(kind=1, param=-0.1), b"contrast parameter"),
             (dict(kind=2, param=3.5), b"block parameter"), (dict(kind=3, param=2.0), b"noise parameter"),
             (dict(kind=5, param=0.0), b"pixelate parameter"),
             (dict(N=0), b"bad shape"), (dict(H=0), b"bad shape"), (dict(N=65536), b"N=65536"),
             (dict(W=9000), b"sides"), (dict(kind=2, param=16.0, H=7), b"H, W >= 8"),
             (dict(kind=4, param=21.0, W=10), b"needs H, W > 10"),
             (dict(lo=1.0, hi=1.0), b"hi > lo"), (dict(lo=float("nan")), b"hi > lo"),
             (dict(xp=y), b"overlap"), (dict(ws_bytes=nws - 1), b"workspace"))
    for kw, msg in cases:
        rc = call(**kw)
        assert rc < 0 and msg in L.ud_last_error(), (kw, rc, L.ud_last_error())
    assert call(ws_bytes=nws - 1) == -4                        # UD_ERR_WORKSPACE
