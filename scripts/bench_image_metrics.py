"""Image quality on the GPU (vbq_image_metrics, vbq_b200.image_metrics, evaluate_compression_quantizer(...,
metrics=True)) at the size of one Kodak orientation evaluated at 16 lambdas.

  * inputs: 24 seeded 512 x 768 x 3 uint8 originals (smoothed Gaussian noise, seed 10) and 16 seeded reconstructions
    of each (the originals plus rounded Gaussian noise of std 2 .. 32, seed 11): 384 pairs, 453 MB of reconstructions,
    more than the 126 MB of L2.
  * kernel_us: the vbq_image_metrics call (every launch of it: pyramid, five levels, reduction), CUDA events over
    back-to-back calls after a warm-up; call_us: vbq_b200.image_metrics (argument checks, workspace, copy of the
    results, host log and power), host clock from a synchronised start to a synchronised end.
  * fma: the FP64 FMAs the separable filter needs from the shapes (5 moments x s taps, horizontally over every row
    and vertically over the valid rows, per level and pair) and the ones the kernels execute (11 taps over whole
    32 x 32 tiles and their 10 halo rows); the rate is executed FMAs over kernel_us.
  * evaluate: evaluate_compression_quantizer on 24 images x 16 lambdas with and without metrics=True (reconstructions
    stay on the device), with the 6-channel learned code-point table of tests/golden and a stand-in decoder (each
    latent's channel mean upsampled 16x): host clock, synchronised, after a warm-up.
  * reference_cpu_s_per_pair: tests/image_metrics_reference.py (NumPy/SciPy, fftconvolve) on the CPU for one pair,
    over the first three pairs: the cost of computing the same columns on the host.
Writes one JSON document (with the device name, power limit and SM clock read in the same run) to --out."""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

from bench_embedding_coding import power_limit, timed_us   # noqa: E402
from bench_embedding_lookup import call_us                 # noqa: E402

N_IMG, M_REC, H, W, C = 24, 16, 512, 768, 3


def inputs():
    g = torch.Generator(device="cuda").manual_seed(10)
    base = torch.randn((N_IMG, C, H + 8, W + 8), generator=g, device="cuda") * 60 + 128
    base = torch.nn.functional.avg_pool2d(base, 9, stride=1)          # smooth, image-like content
    x = base.round().clamp(0, 255).permute(0, 2, 3, 1).contiguous()
    g.manual_seed(11)
    std = torch.linspace(2, 32, M_REC, device="cuda")[:, None, None, None, None]
    y = (x[None] + std * torch.randn((M_REC,) + tuple(x.shape), generator=g, device="cuda")).round().clamp(0, 255)
    return x.to(torch.uint8), y.to(torch.uint8).contiguous()


def fma_counts(pairs):
    need = run = 0
    h, w = H, W
    for _ in range(5):
        s = min(11, h, w)
        ho, wo = h - s + 1, w - s + 1
        need += pairs * 5 * s * (h * wo * C + ho * wo * C)
        ty, tx = -(-ho // 32), -(-(wo * C) // 32)
        run += pairs * ty * tx * 5 * 11 * (42 * 32 + 32 * 32)
        h, w = (h + 1) // 2, (w + 1) // 2
    return need, run


def evaluate_times(x, min_seconds):
    import vbq_b200
    g = np.load(os.path.join(ROOT, "tests", "golden", "learned_c6_n10.npz"))
    q = vbq_b200.ChannelwisePriorCDFQuantizer(int(g["C"]), int(g["N"]))
    q.set_code_points(g["table"])
    lambs = [2.0 ** k for k in range(-8, 8)]
    q.entropy_models = {l: g["em_%d" % (i % 4)] for i, l in enumerate(lambs)}
    gen = torch.Generator(device="cuda").manual_seed(12)
    means = torch.randn((N_IMG, H // 16, W // 16, 6), generator=gen, device="cuda")
    logvars = torch.randn((N_IMG, H // 16, W // 16, 6), generator=gen, device="cuda") - 3.0

    class VAE:
        def encode(self, X):
            return means, logvars

        def decode(self, z):
            m = 0.5 + 0.05 * z.mean(dim=-1, keepdim=True)
            return m.repeat_interleave(16, 1).repeat_interleave(16, 2).repeat_interleave(3, 3)

    X = x.float() / 255
    out = {}
    for metrics in (False, True):
        us, iters = call_us(lambda: vbq_b200.evaluate_compression_quantizer(q, VAE(), X, lambs, metrics=metrics),
                            min_seconds, 20)
        out["metrics_%s_call_us" % metrics] = us
        out["metrics_%s_iters" % metrics] = iters
    out["lambdas"] = len(lambs)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r10_image_metrics.json"))
    ap.add_argument("--min-seconds", type=float, default=2.0)
    args = ap.parse_args()
    import vbq_b200
    from vbq_b200 import ops
    import image_metrics_reference as R

    x, y = inputs()
    pairs = N_IMG * M_REC
    kernel_us, kernel_iters = timed_us(lambda: ops.image_metrics(x, y), args.min_seconds, 200)
    call, call_iters = call_us(lambda: vbq_b200.image_metrics(x, y), args.min_seconds, 200)
    res = vbq_b200.image_metrics(x, y)
    need, run = fma_counts(pairs)
    xs, ys = x.cpu().numpy(), y.cpu().numpy()
    t0 = time.perf_counter()
    for n in range(3):
        R.ms_ssim(xs[n:n + 1], ys[0, n:n + 1])
        R.psnr(xs[n:n + 1], ys[0, n:n + 1])
    ref_s = (time.perf_counter() - t0) / 3
    doc = {
        "device": torch.cuda.get_device_name(),
        "power_limit_and_max_sm_clock": power_limit(),
        "shape": {"originals": [N_IMG, H, W, C], "reconstructions": [M_REC, N_IMG, H, W, C], "pairs": pairs},
        "kernel_us": kernel_us, "kernel_iters": kernel_iters,
        "call_us": call, "call_iters": call_iters,
        "fp64_fma_needed": need, "fp64_fma_executed": run,
        "fp64_fma_per_s_executed": run / (kernel_us * 1e-6),
        "us_per_pair": kernel_us / pairs,
        "mean_psnr_per_reconstruction": res["PSNR"].mean(axis=1).tolist(),
        "mean_ms_ssim_per_reconstruction": res["MS-SSIM"].mean(axis=1).tolist(),
        "evaluate_compression_quantizer": evaluate_times(x, args.min_seconds),
        "reference_cpu_s_per_pair": ref_s,
        "reference_cpu_note": "tests/image_metrics_reference.py (NumPy/SciPy, scipy.fft's default of one worker) on "
                              "the GPU host's CPU: MS-SSIM and PSNR of one pair, mean of 3",
        "reference_cpu_s_all_pairs_estimate": ref_s * pairs,
    }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(doc, f, indent=1)
    print(json.dumps(doc), flush=True)


if __name__ == "__main__":
    main()
