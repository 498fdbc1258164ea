"""NumPy/SciPy restatement of the image-quality metrics of the reference's evaluation harness
(img_comparison_metrics.py, used by utils.evaluate_compression_quantizer): MSE, PSNR and TF models' MultiScaleSSIM.

This file is the normative definition `vbq_b200.image_metrics` is tested against.  The reference's own
img_comparison_metrics.py is not in this repository, so line-for-line agreement with it is unverified; what the tests
verify is agreement with this restatement.  Inputs are uint8 images (N, H, W, C), max_val = 255."""
import numpy as np
from scipy import signal
from scipy.ndimage import convolve

WEIGHTS = np.array([0.0448, 0.2856, 0.3001, 0.2363, 0.1333])


def mse(x, y):
    """(N,) float64: sum((x - y)^2) over H W C, divided by H W C."""
    d = x.astype(np.float64) - y.astype(np.float64)
    return np.sum(d * d, axis=(1, 2, 3)) / np.prod(x.shape[1:])


def psnr(x, y):
    with np.errstate(divide='ignore'):
        return 10 * np.log10(255.0 ** 2 / mse(x, y))


def fspecial_gauss(size, sigma):
    """_FSpecialGauss: a normalised size x size Gaussian, offset by a half for even sizes."""
    radius = size // 2
    offset = 0.0
    start, stop = -radius, radius + 1
    if size % 2 == 0:
        offset = 0.5
        stop -= 1
    x, y = np.mgrid[offset + start:stop, offset + start:stop]
    g = np.exp(-((x ** 2 + y ** 2) / (2.0 * sigma ** 2)))
    return g / g.sum()


def ssim_for_multiscale(img1, img2, max_val=255, filter_size=11, filter_sigma=1.5, k1=0.01, k2=0.03):
    """(ssim, cs) means of one level of a (1, h, w, C) float64 pair."""
    _, height, width, _ = img1.shape
    size = min(filter_size, height, width)
    sigma = size * filter_sigma / filter_size
    window = np.reshape(fspecial_gauss(size, sigma), (1, size, size, 1))
    mu1 = signal.fftconvolve(img1, window, mode='valid')
    mu2 = signal.fftconvolve(img2, window, mode='valid')
    sigma11 = signal.fftconvolve(img1 * img1, window, mode='valid')
    sigma22 = signal.fftconvolve(img2 * img2, window, mode='valid')
    sigma12 = signal.fftconvolve(img1 * img2, window, mode='valid')
    mu11, mu22, mu12 = mu1 * mu1, mu2 * mu2, mu1 * mu2
    sigma11 -= mu11
    sigma22 -= mu22
    sigma12 -= mu12
    c1 = (k1 * max_val) ** 2
    c2 = (k2 * max_val) ** 2
    v1 = 2.0 * sigma12 + c2
    v2 = sigma11 + sigma22 + c2
    ssim = np.mean((((2.0 * mu12 + c1) * v1) / ((mu11 + mu22 + c1) * v2)))
    cs = np.mean(v1 / v2)
    return ssim, cs


def downsample(im):
    return convolve(im, np.ones((1, 2, 2, 1)) / 4.0, mode='reflect')[:, ::2, ::2, :]


def ms_ssim_levels(x, y):
    """Per-level (ssim, cs) of one (1, H, W, C) pair: two float64 arrays of 5."""
    im1, im2 = x.astype(np.float64), y.astype(np.float64)
    mssim, mcs = [], []
    for _ in range(WEIGHTS.size):
        s, c = ssim_for_multiscale(im1, im2)
        mssim.append(s)
        mcs.append(c)
        im1, im2 = downsample(im1), downsample(im2)
    return np.array(mssim), np.array(mcs)


def ms_ssim_from_levels(mssim, mcs):
    with np.errstate(invalid='ignore'):
        return np.prod(mcs[0:4] ** WEIGHTS[0:4]) * (mssim[4] ** WEIGHTS[4])


def ms_ssim(x, y):
    """(N,) MultiScaleSSIM of each pair x[n], y[n], each as a (1, H, W, C) array."""
    return np.array([ms_ssim_from_levels(*ms_ssim_levels(x[n:n + 1], y[n:n + 1])) for n in range(x.shape[0])])
