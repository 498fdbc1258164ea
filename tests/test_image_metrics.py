"""Image quality on the GPU (vbq_image_metrics, `vbq_b200.image_metrics`, `evaluate_compression_quantizer(...,
metrics=True)`) against the NumPy/SciPy restatement in image_metrics_reference.py."""
import ctypes

import numpy as np
import pytest
import torch
from scipy import signal

import image_metrics_reference as R

SHAPES = [(512, 768), (768, 512), (131, 97), (97, 131), (40, 24), (9, 13), (1, 1)]


def images(rng, n, h, w, c, noise=8.0):
    """Image-like originals (smoothed noise) and reconstructions (originals plus rounded Gaussian noise), uint8."""
    base = rng.normal(128, 60, (n, h + 8, w + 8, c))
    base = signal.fftconvolve(base, np.ones((1, 9, 9, 1)) / 81, mode='valid')
    x = np.clip(np.round(base), 0, 255).astype(np.uint8)
    return x, lambda m: np.clip(np.round(x[None] + rng.normal(0, noise, (m,) + x.shape)), 0, 255).astype(np.uint8)


# ---- CPU: the reference itself ------------------------------------------------------------------------------------
def direct_levels(x, y):
    """Independent restatement: separable direct float64 filtering and an explicit 2 x 2 mean with the last row or
    column repeated."""
    a, b = x[0].astype(np.float64), y[0].astype(np.float64)
    ssim, cs = [], []
    for _ in range(5):
        h, w, _ = a.shape
        s = min(11, h, w)
        sigma = s * 1.5 / 11
        u = np.arange(s) - s // 2 + (0.5 if s % 2 == 0 else 0.0)
        g = np.exp(-u ** 2 / (2 * sigma ** 2))
        g /= g.sum()

        def filt(im):
            ho, wo = h - s + 1, w - s + 1
            t = sum(g[k] * im[k:k + ho] for k in range(s))
            return sum(g[k] * t[:, k:k + wo] for k in range(s))
        mu1, mu2 = filt(a), filt(b)
        s11, s22, s12 = filt(a * a) - mu1 * mu1, filt(b * b) - mu2 * mu2, filt(a * b) - mu1 * mu2
        c1, c2 = (0.01 * 255) ** 2, (0.03 * 255) ** 2
        v1, v2 = 2 * s12 + c2, s11 + s22 + c2
        ssim.append(np.mean((2 * mu1 * mu2 + c1) * v1 / ((mu1 * mu1 + mu2 * mu2 + c1) * v2)))
        cs.append(np.mean(v1 / v2))

        def down(im):
            p = np.concatenate([im, im[-1:]], 0) if im.shape[0] % 2 else im
            p = np.concatenate([p, p[:, -1:]], 1) if p.shape[1] % 2 else p
            return 0.25 * (p[0::2, 0::2] + p[1::2, 0::2] + p[0::2, 1::2] + p[1::2, 1::2])
        a, b = down(a), down(b)
    return np.array(ssim), np.array(cs)


@pytest.mark.parametrize("h,w,c", [(131, 97, 3), (40, 24, 3), (9, 13, 1), (24, 40, 1), (1, 1, 3)])
def test_reference_equals_direct_separable_filter(h, w, c):
    rng = np.random.default_rng(h * 1000 + w)
    x, recon = images(rng, 1, h, w, c)
    y = recon(1)[0]
    s_ref, c_ref = R.ms_ssim_levels(x, y)
    s_dir, c_dir = direct_levels(x, y)
    assert np.allclose(s_ref, s_dir, rtol=1e-12, atol=0) and np.allclose(c_ref, c_dir, rtol=1e-12, atol=0)
    assert np.isclose(R.ms_ssim(x, y)[0], R.ms_ssim_from_levels(s_dir, c_dir), rtol=1e-12, atol=0)


def test_reference_identical_images():
    rng = np.random.default_rng(3)
    x, _ = images(rng, 2, 40, 24, 3)
    assert np.array_equal(R.ms_ssim(x, x), [1.0, 1.0])
    assert np.all(np.isinf(R.psnr(x, x)))


@pytest.mark.parametrize("a,b", [(0, 255), (100, 104), (37, 200)])
def test_reference_constant_images_closed_form(a, b):
    x = np.full((1, 40, 24, 3), a, np.uint8)
    y = np.full((1, 40, 24, 3), b, np.uint8)
    c1 = (0.01 * 255) ** 2
    ssim = (2.0 * a * b + c1) / (a * a + b * b + c1)        # sigma11 = sigma22 = sigma12 = 0, so cs = 1
    s_ref, c_ref = R.ms_ssim_levels(x, y)
    assert np.allclose(c_ref, 1.0, rtol=1e-12, atol=0) and np.allclose(s_ref, ssim, rtol=1e-12, atol=0)
    assert np.isclose(R.ms_ssim(x, y)[0], ssim ** R.WEIGHTS[4], rtol=1e-12, atol=0)
    assert R.mse(x, y)[0] == float((a - b) ** 2)
    assert R.psnr(x, y)[0] == 10 * np.log10(255.0 ** 2 / float((a - b) ** 2))


# ---- CPU: argument checks ----------------------------------------------------------------------------------------
def test_abi_rejects_bad_arguments_without_gpu():
    from vbq_b200 import _lib
    lib = _lib.load()
    one = ctypes.c_void_p(256)            # any non-null aligned address: these calls must fail before using it
    ws = lib.vbq_image_metrics_workspace_bytes(24, 16, 512, 768, 3)
    assert ws > 24 * 17 * 512 * 768 * 3                   # the four coarser levels in float32 and the partials
    for bad in ((-1, 1, 8, 8, 3), (1, -1, 8, 8, 3), (1, 1, 0, 8, 3), (1, 1, 8, 0, 3), (1, 1, 8, 8, 0), (1, 1, 8, 8, 5),
                (1, 1, 1 << 16, 1 << 14, 3), (1 << 20, 1 << 12, 8, 8, 3)):
        assert lib.vbq_image_metrics_workspace_bytes(*bad) == -1, bad
        assert lib.vbq_image_metrics(one, one, *bad, one, 1 << 40, one, one, one, None) == 2, bad
    assert lib.vbq_image_metrics(one, one, 1, 1, 8, 8, 5, one, 1 << 40, one, one, one, None) == 2
    assert b"C=5" in lib.vbq_last_error()
    assert lib.vbq_image_metrics(None, one, 2, 3, 8, 8, 3, one, 1 << 40, one, one, one, None) == 1
    assert lib.vbq_image_metrics(one, one, 2, 3, 8, 8, 3, one, 1 << 40, one, None, one, None) == 1
    assert lib.vbq_image_metrics(one, one, 2, 3, 8, 8, 3, ctypes.c_void_p(257), 1 << 40, one, one, one, None) == 7
    need = lib.vbq_image_metrics_workspace_bytes(2, 3, 8, 8, 3)
    assert lib.vbq_image_metrics(one, one, 2, 3, 8, 8, 3, one, need - 1, one, one, one, None) == 5
    assert lib.vbq_image_metrics(one, one, 2, 3, 8, 8, 3, None, need, one, one, one, None) == 5
    # no pairs is no work: null pointers are fine
    assert lib.vbq_image_metrics(None, None, 0, 3, 8, 8, 3, None, 0, None, None, None, None) == 0
    assert lib.vbq_image_metrics(None, None, 2, 0, 8, 8, 3, None, 0, None, None, None, None) == 0


def test_python_argument_checks():
    import vbq_b200
    x = torch.zeros((2, 8, 8, 3), dtype=torch.uint8)
    cases = [
        (x.float(), x, "uint8"), (x, x.to(torch.int16), "uint8"), (x.numpy(), x, "torch.Tensor"),
        (x[0], x, "originals must be"), (x, x[None, :1], "originals must be"), (x, x[:, :, :4], "originals must be"),
        (torch.zeros((2, 8, 8, 5), dtype=torch.uint8), torch.zeros((2, 8, 8, 5), dtype=torch.uint8), "1 <= C"),
        (torch.zeros((2, 0, 8, 3), dtype=torch.uint8), torch.zeros((2, 0, 8, 3), dtype=torch.uint8), "H, W >= 1"),
        (x.transpose(1, 2), x, "contiguous"), (x, x, "CUDA tensor"),
    ]
    for a, b, msg in cases:
        with pytest.raises(ValueError, match=msg):
            vbq_b200.image_metrics(a, b)


# ---- GPU ----------------------------------------------------------------------------------------------------------
def run_and_reference(x, y):
    """GPU kernels and public call on x (N, H, W, C), y (M, N, H, W, C) against the reference."""
    import vbq_b200
    from vbq_b200 import ops
    xd, yd = torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda()
    sse, ssim, cs = (t.cpu().numpy() for t in ops.image_metrics(xd, yd))
    out = vbq_b200.image_metrics(xd, yd)
    M, N = y.shape[:2]
    for k in ("MSE", "PSNR", "MS-SSIM"):
        assert out[k].shape == (M, N) and out[k].dtype == np.float64
    for m in range(M):
        d = x.astype(np.int64) - y[m].astype(np.int64)
        assert np.array_equal(sse[m], np.sum(d * d, axis=(1, 2, 3)))
        assert np.array_equal(out["MSE"][m], R.mse(x, y[m]))
        assert np.array_equal(out["PSNR"][m], R.psnr(x, y[m]))
        for n in range(N):
            s_ref, c_ref = R.ms_ssim_levels(x[n:n + 1], y[m, n:n + 1])
            assert np.allclose(ssim[m, n], s_ref, rtol=1e-12, atol=0), (m, n, ssim[m, n], s_ref)
            assert np.allclose(cs[m, n], c_ref, rtol=1e-12, atol=0), (m, n, cs[m, n], c_ref)
            ref = R.ms_ssim_from_levels(s_ref, c_ref)
            assert np.isclose(out["MS-SSIM"][m, n], ref, rtol=1e-12, atol=0, equal_nan=True), (m, n)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("h,w", SHAPES)
@pytest.mark.parametrize("c", [1, 3])
def test_gpu_equals_reference(h, w, c):
    rng = np.random.default_rng(h * 7919 + w * 31 + c)
    big = h * w >= 100_000
    n, m = (2, 1) if big else (5, 3)
    x, recon = images(rng, n, h, w, c)
    run_and_reference(x, recon(m))


@pytest.mark.gpu
@pytest.mark.parametrize("h,w,c,n", [(40, 24, 3, 24), (131, 97, 1, 4), (9, 13, 3, 24)])
def test_gpu_sixteen_reconstructions(h, w, c, n):
    rng = np.random.default_rng(16 * h + w)
    x, recon = images(rng, n, h, w, c, noise=20.0)
    run_and_reference(x, recon(16))


@pytest.mark.gpu
def test_gpu_one_reconstruction_as_4d_and_identical_images():
    import vbq_b200
    rng = np.random.default_rng(5)
    x, recon = images(rng, 3, 97, 131, 3)
    xd = torch.from_numpy(x).cuda()
    out = vbq_b200.image_metrics(xd, xd.clone())
    assert np.array_equal(out["MS-SSIM"], np.ones((1, 3))) and np.all(np.isinf(out["PSNR"]))
    assert np.array_equal(out["MSE"], np.zeros((1, 3)))
    y = recon(1)
    a = vbq_b200.image_metrics(xd, torch.from_numpy(y[0]).cuda())
    b = vbq_b200.image_metrics(xd, torch.from_numpy(y).cuda())
    for k in a:
        assert np.array_equal(a[k], b[k])


@pytest.mark.gpu
def test_gpu_negative_cs_gives_nan():
    rng = np.random.default_rng(11)
    x = rng.integers(0, 256, (2, 64, 48, 3)).astype(np.uint8)
    y = (255 - x)[None]                                    # anti-correlated: every level's mean cs is negative
    s_ref, c_ref = R.ms_ssim_levels(x[:1], y[0, :1])
    assert np.any(c_ref[:4] < 0)
    out = run_and_reference(x, y)
    assert np.all(np.isnan(out["MS-SSIM"]))


@pytest.mark.gpu
def test_gpu_constant_images():
    a = np.array([0, 100, 37], np.uint8)[:, None, None, None] * np.ones((1, 40, 24, 3), np.uint8)
    b = np.array([255, 104, 200], np.uint8)[:, None, None, None] * np.ones((1, 40, 24, 3), np.uint8)
    run_and_reference(a, b[None])


@pytest.mark.gpu
def test_gpu_deterministic():
    from vbq_b200 import ops
    rng = np.random.default_rng(8)
    x, recon = images(rng, 6, 512, 768, 3)
    xd, yd = torch.from_numpy(x).cuda(), torch.from_numpy(recon(4)).cuda()
    first = ops.image_metrics(xd, yd)
    second = ops.image_metrics(xd, yd)
    for a, b in zip(first, second):
        assert torch.equal(a, b)
        assert a.dtype == torch.int64 or bool(torch.isfinite(a).all())


@pytest.mark.gpu
def test_gpu_argument_checks_and_empty():
    import vbq_b200
    x = torch.zeros((2, 8, 8, 3), dtype=torch.uint8, device="cuda")
    with pytest.raises(ValueError, match="contiguous"):
        vbq_b200.image_metrics(x, x.transpose(1, 2).contiguous().transpose(1, 2))
    with pytest.raises(ValueError, match="CUDA tensor"):
        vbq_b200.image_metrics(x, x.cpu())
    with pytest.raises(ValueError, match="originals must be"):
        vbq_b200.image_metrics(x, x[:1])
    for a, b, shape in ((x[:0], x[:0], (1, 0)), (x, x[None, :0].reshape(0, 2, 8, 8, 3), (0, 2))):
        out = vbq_b200.image_metrics(a, b)
        assert all(v.shape == shape and v.dtype == np.float64 for v in out.values())


@pytest.mark.gpu
def test_evaluation_metrics_column():
    """metrics=True with the fake VAE of test_gpu_golden: the quality columns are image_metrics of the 8-bit arrays
    and the rate columns equal a metrics=False call."""
    import vbq_b200
    from test_gpu_golden import lambs_of, load, make_quantizer
    g = load("learned_c6_n10")
    q = make_quantizer(g)
    lambs = lambs_of(g)
    q.raw_code_length_entropy_models = {l: g["rcl_%d" % i] for i, l in enumerate(lambs)}
    q.entropy_models = {l: g["em_%d" % i] for i, l in enumerate(lambs)}
    means, logvars = torch.from_numpy(g["means"]).cuda(), torch.from_numpy(g["logvars"]).cuda()
    Nimg, Hl, Wl, C = means.shape

    class VAE:
        def encode(self, X):
            return means, logvars

        def decode(self, z):
            m = 0.5 + 0.01 * z.mean(dim=-1, keepdim=True)
            return m.repeat_interleave(16, 1).repeat_interleave(16, 2).repeat_interleave(3, 3)

    rng = np.random.default_rng(2)
    X = rng.uniform(0.3, 0.7, (Nimg, 16 * Hl, 16 * Wl, 3)).astype(np.float32)
    plain = vbq_b200.evaluate_compression_quantizer(q, VAE(), X, lambs)
    assert not {"MSE", "PSNR", "MS-SSIM"} & set(plain)
    res = vbq_b200.evaluate_compression_quantizer(q, VAE(), X, lambs, return_reconstructions=True, metrics=True)
    for k in ("B", "BPP", "BPL", "BPPCL"):
        assert np.array_equal(res[k], plain[k])
    x8 = torch.round(255 * torch.from_numpy(X).cuda()).to(torch.uint8)
    y8 = torch.round(255 * torch.from_numpy(res["reconstructions"]).cuda()).to(torch.uint8)
    direct = vbq_b200.image_metrics(x8, y8)
    for k in ("MSE", "PSNR", "MS-SSIM"):
        assert res[k].shape == (Nimg, len(lambs))
        assert np.array_equal(res[k], direct[k].T)
    only = vbq_b200.evaluate_compression_quantizer(q, VAE(), X, lambs, metrics=True)
    assert "reconstructions" not in only
    for k in res:
        if k != "reconstructions":
            assert np.array_equal(only[k], res[k])
