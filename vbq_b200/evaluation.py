"""Batched evaluation driver — the caller of the hot path in the reference
(img-compression/utils.py:502-634 `evaluate_compression_quantizer`, post_process.py:159-188).

The reference loops over images one at a time ("TODO: parallelize", utils.py:535) and per image over the settings.
Here all same-sized images go through ONE `quantizer.compress`-style call (one kernel launch for every image and every
lambda), and the per-image bit totals are reduced on the device: the rate statistics `B`, `BPP`, `BPL`, `BPPCL` (the
keys of utils.py:523-527).  With ``metrics=True`` the quality side of each R-D point (MSE, PSNR and MS-SSIM of the
8-bit images, the metrics of the reference's img_comparison_metrics.py) is computed on the device too, by
`image_metrics` (DESIGN.md §8j)."""
from __future__ import annotations

import numpy as np
import torch

from . import _lib, ops, utils

MS_SSIM_WEIGHTS = np.array([0.0448, 0.2856, 0.3001, 0.2363, 0.1333])      # TF models' MultiScaleSSIM


def image_metrics(originals, reconstructions):
    """MSE, PSNR and MS-SSIM of 8-bit images: a dict of float64 NumPy arrays ``MSE``, ``PSNR`` and ``MS-SSIM`` of
    shape (M, N).

    ``originals``: (N, H, W, C) uint8 CUDA tensor; ``reconstructions``: (M, N, H, W, C) uint8 on the same device, M
    reconstructions of each original, or (N, H, W, C) for M = 1; 1 <= C <= 4, contiguous.  max_val is 255.
    MSE = sum((x - y)^2) / (H W C) from the exact integer sum; PSNR = 10 log10(255^2 / MSE), inf for identical
    images; MS-SSIM is TF models' MultiScaleSSIM of each (1, H, W, C) pair (5 levels, 11-tap Gaussian window of
    sigma 1.5 shrunk to the image at coarse levels, k1 = 0.01, k2 = 0.03), NaN where a level's mean cs is negative.
    The sums and the per-level means run in the vbq_image_metrics kernels (float64, fixed summation order, so repeated
    calls give the same bits); the final log and power run on the host.  Bad arguments raise ValueError before any
    launch; N = 0 or M = 0 gives empty arrays without one.  One host synchronisation (the copy of the results)."""
    x, y = originals, reconstructions
    for name, t in (("originals", x), ("reconstructions", y)):
        if not isinstance(t, torch.Tensor):
            raise ValueError("vbq_b200: image_metrics: `%s` must be a torch.Tensor, got %s" % (name, type(t)))
        if t.dtype != torch.uint8:
            raise ValueError("vbq_b200: image_metrics: `%s` must be uint8, got %s" % (name, t.dtype))
    if y.dim() == 4:
        y = y.unsqueeze(0)
    if x.dim() != 4 or y.dim() != 5 or tuple(y.shape[1:]) != tuple(x.shape):
        raise ValueError("vbq_b200: image_metrics: originals must be (N, H, W, C) and reconstructions (M, N, H, W, C) "
                         "or (N, H, W, C), got %s and %s" % (tuple(x.shape), tuple(reconstructions.shape)))
    N, H, W, C = x.shape
    M = y.shape[0]
    if H < 1 or W < 1 or not 1 <= C <= _lib.IMAGE_METRICS_MAX_CHANNELS or H * W * C >= 2 ** 31:
        raise ValueError("vbq_b200: image_metrics: images of shape %s (H, W >= 1, 1 <= C <= %d, H W C < 2^31)"
                         % (tuple(x.shape), _lib.IMAGE_METRICS_MAX_CHANNELS))
    for name, t in (("originals", x), ("reconstructions", y)):
        if not t.is_contiguous():
            raise ValueError("vbq_b200: image_metrics: `%s` must be contiguous" % name)
        if not t.is_cuda:
            raise ValueError("vbq_b200: image_metrics: `%s` must be a CUDA tensor (no CPU fallback exists)" % name)
    if x.device != y.device:
        raise ValueError("vbq_b200: image_metrics: originals on %s, reconstructions on %s" % (x.device, y.device))
    if M * N == 0:
        e = np.zeros((M, N))
        return {'MSE': e, 'PSNR': e.copy(), 'MS-SSIM': e.copy()}
    sse, ssim, cs = ops.image_metrics(x, y)
    sse, ssim, cs = (utils.to_host_numpy(t) for t in (sse, ssim, cs))
    w = MS_SSIM_WEIGHTS
    mse = sse.astype(np.float64) / (H * W * C)
    with np.errstate(divide='ignore', invalid='ignore'):
        psnr = 10 * np.log10(255.0 ** 2 / mse)
        msssim = np.prod(cs[..., :4] ** w[:4], axis=-1) * (ssim[..., 4] ** w[4])
    return {'MSE': mse, 'PSNR': psnr, 'MS-SSIM': msssim}


def to_8bit(x):
    """float images in [0, 1] -> uint8 round(255 x) (round half to even), on x's device; values are clamped to [0, 1]
    first."""
    return torch.round(255 * x.clamp(0, 1)).to(torch.uint8)


def evaluate_compression_quantizer(quantizer, vae, images, settings, return_reconstructions=False, clip=True,
                                   metrics=False):
    """``images``: (N, H, W, 3) float array in [0, 1] (same-sized images, e.g. the 24 Kodak images of one
    orientation).  ``settings``: the lambdas.  Returns a dict with (N, len(settings)) arrays ``B`` (total bits),
    ``BPP`` (bits per pixel), ``BPL`` (bits per latent dimension), ``BPPCL`` (bits per pixel from the raw-depth +
    depth-entropy code lengths, utils.py:552-553) and, optionally, ``reconstructions`` (len(settings), N, H, W, 3).

    ``metrics=True`` adds (N, len(settings)) float64 arrays ``MSE``, ``PSNR`` and ``MS-SSIM``: `image_metrics` of the
    originals and the reconstructions, both clamped to [0, 1] and converted to 8 bits as round(255 x) (round half to
    even) on the device.  The reconstructions are decoded once for both outputs, and without
    ``return_reconstructions`` they never leave the device."""
    X = images if isinstance(images, torch.Tensor) else torch.as_tensor(np.asarray(images))
    N = int(X.shape[0])
    num_pixels = int(X.shape[1]) * int(X.shape[2])
    M = len(settings)
    means, logvars = vae.encode(X)
    dev = quantizer._compress_latents_device(means, logvars, settings)          # (M, N, H', W', C) tensors on the GPU
    num_bits = dev['num_bits'].reshape(M, N, -1)
    nbits = num_bits.sum(dim=2, dtype=torch.float64)                            # (M, N)
    latent_dims = num_bits.shape[2]
    cl = dev['raw_num_bits'].reshape(M, N, -1).sum(dim=2, dtype=torch.float64) if dev['corrected'] else nbits
    results = {
        'B': utils.to_host_numpy(nbits).T.copy(),
        'BPP': utils.to_host_numpy(nbits / num_pixels).T.copy(),
        'BPL': utils.to_host_numpy(nbits / latent_dims).T.copy(),
        'BPPCL': utils.to_host_numpy(cl / num_pixels).T.copy(),
    }
    if return_reconstructions or metrics:
        z = dev['Z_hat'].reshape((-1,) + tuple(means.shape[1:]))
        xh = vae.decode(z)
        xh = xh.detach() if isinstance(xh, torch.Tensor) else torch.as_tensor(np.asarray(xh))
        xh = xh.reshape((M,) + tuple(X.shape))
        if clip:
            xh = xh.clamp(0, 1)
        if metrics:
            d = z.device
            q = image_metrics(to_8bit(X.to(d)).contiguous(), to_8bit(xh.to(d)).contiguous())
            results.update({k: v.T.copy() for k, v in q.items()})
        if return_reconstructions:
            results['reconstructions'] = utils.to_host_numpy(xh.contiguous())
    return results
