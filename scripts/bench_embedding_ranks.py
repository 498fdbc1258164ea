"""Exact target ranks (vbq_b200.ranks, CompressedEmbedding.ranks, GaussianCodebook.analogy_sweep) on the posteriors of
bench_embedding_scores.py: 1 M x 300 seeded Gaussian posteriors (seed 77), N = 10, codebook std 1.2356, exact=True,
and the paper's shape 100 k x 100 from the same generator.

  * dense: z_hat = compress_coordinates at beta = 26.8 on both shapes; B = 1, 64, 1,024 and 16,649 seeded
    standard-normal queries with seeded targets, dot and cosine.  kernel_us: the vbq_score_ranks launch (thresholds
    precomputed), CUDA events over back-to-back launches; call_us: vbq_b200.ranks, host clock from a synchronised
    start to a synchronised end; fma_share: B V D over the kernel time as a share of the FP32 FMA bound
    SMs x 128 x the maximum SM clock read in this run.  baseline_call_us: blocked torch.mm in FP32 (TF32 off) over
    row blocks of at most 2^28 scores, the norms for the cosine, the topk keys, compare and sum, on the same queries;
    baseline_rank_diffs: how many of its ranks differ from the contract's (information only: cuBLAS sums in another
    order).
  * compressed: CompressedEmbedding.ranks on the 1 M x 300 blobs at beta = 0.518, 26.8 and 1,931 (default
    segmentation and checkpoint interval), B = 1,024, with its peak extra device memory; against
    lookup(arange(V)) + vbq_b200.ranks.
  * analogy_sweep: five beta on 100 k x 100 with 16,649 seeded synthetic questions (four distinct ids each), cosine;
    the time per beta is the call time over five.
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

from bench_embedding_coding import power_limit, timed_us   # noqa: E402
from bench_embedding_lookup import call_us                 # noqa: E402

BATCHES = [1, 64, 1024, 16649]
BETA = 26.8


def posteriors(V, D):
    g = torch.Generator(device="cuda")
    g.manual_seed(77)
    means = torch.randn((V, D), generator=g, device="cuda") * 1.2329 - 0.08
    stds = torch.exp(torch.randn((V, D), generator=g, device="cuda") * 0.7 + float(np.log(0.04)))
    return means, stds


def keys(s):
    b = s.view(torch.int32).to(torch.int64)
    k = torch.where(b < 0, b ^ 0x7FFFFFFF, b)
    k = torch.where(s == 0, torch.zeros_like(k), k)
    return torch.where(torch.isnan(s), torch.full_like(k, -(1 << 31)), k)


def mm_ranks(Z, q, t, metric):
    """The blocked-mm baseline: q @ Z_block.T in FP32, the target's score from the same product, keys, compare, sum."""
    V, B = Z.shape[0], q.shape[0]
    thr = (q * Z[t]).sum(dim=1)
    if metric == "cosine":
        zn = Z.norm(dim=1)
        qn = q.norm(dim=1)
        thr = thr / (zn[t] * qn).clamp_min(1e-30)
    kt = keys(thr)[:, None]
    counts = torch.ones(B, dtype=torch.int64, device=Z.device)
    R = max(1, (1 << 28) // B)
    for a in range(0, V, R):
        b = min(V, a + R)
        s = q @ Z[a:b].T
        if metric == "cosine":
            s = s / (zn[None, a:b] * qn[:, None]).clamp_min(1e-30)
        k = keys(s)
        ids = torch.arange(a, b, device=Z.device)[None, :]
        counts += ((k > kt) | ((k == kt) & (ids < t[:, None]))).sum(dim=1)
    return counts


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r7_embedding_ranks.json"))
    ap.add_argument("--seconds", type=float, default=0.3, help="about this long per timed configuration")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_embedding_ranks.py needs a CUDA device")
    torch.backends.cuda.matmul.allow_tf32 = False

    import vbq_b200
    from vbq_b200 import ops

    limits = power_limit()
    sm_mhz = float(limits.split(",")[1].split()[0]) if limits else float("nan")
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    fma_per_s = sms * 128 * sm_mhz * 1e6
    cb = vbq_b200.GaussianCodebook(1.2356, 10)
    grid = np.exp(np.linspace(np.log(0.01), np.log(100000), 50))
    doc = dict(device=torch.cuda.get_device_name(), power_limit_and_max_sm_clock=limits, sms=sms,
               fp32_fma_bound_per_s=fma_per_s, torch=torch.__version__, dense=[], compressed=[], analogy_sweep=None)

    for V, D in ((1_000_000, 300), (100_000, 100)):
        means, stds = posteriors(V, D)
        Z, _ = cb.compress_coordinates(means, stds, BETA)
        del means, stds
        for B in BATCHES:
            g = torch.Generator(device="cuda").manual_seed(B)
            q = torch.randn((B, D), generator=g, device="cuda")
            t = torch.randint(0, V, (B,), generator=g, device="cuda")
            for metric in ("dot", "cosine"):
                ar = torch.arange(B, device="cuda")
                thr = ops.pair_scores(Z, q, t, ar, metric)
                counts = torch.zeros(B, dtype=torch.int64, device="cuda")
                k_us, k_n = timed_us(lambda: ops.score_ranks(Z, q, metric, thr, t, counts), args.seconds, 200)
                c_us, c_n = call_us(lambda: vbq_b200.ranks(Z, q, t, metric), args.seconds, 200)
                got = vbq_b200.ranks(Z, q, t, metric)
                b_us, _ = call_us(lambda: mm_ranks(Z, q, t, metric), args.seconds, 50)
                diffs = int((mm_ranks(Z, q, t, metric) != got).sum())
                row = dict(rows=V, dim=D, batch=B, metric=metric, kernel_us=k_us, kernel_launches=k_n, call_us=c_us,
                           calls=c_n, fma_share=B * V * D / (k_us * 1e-6) / fma_per_s, baseline_call_us=b_us,
                           baseline_rank_diffs=diffs)
                doc["dense"].append(row)
                print(json.dumps(row), flush=True)
        del Z
        torch.cuda.empty_cache()

    V, D, B = 1_000_000, 300, 1024
    means, stds = posteriors(V, D)
    betas = [float(grid[i]) for i in (12, 24, 37)]
    blobs = cb.compress_to_bytes(means, stds, betas)
    del means, stds
    g = torch.Generator(device="cuda").manual_seed(5)
    q = torch.randn((B, D), generator=g, device="cuda")
    t = torch.randint(0, V, (B,), generator=g, device="cuda")
    for beta in betas:
        ce = vbq_b200.CompressedEmbedding(blobs[beta])
        for metric in ("dot", "cosine"):
            torch.cuda.synchronize()
            base = torch.cuda.memory_allocated()
            torch.cuda.reset_peak_memory_stats()
            got = ce.ranks(q, t, metric)
            torch.cuda.synchronize()
            peak = torch.cuda.max_memory_allocated() - base
            c_us, c_n = call_us(lambda: ce.ranks(q, t, metric), args.seconds, 20)

            def via_lookup():
                return vbq_b200.ranks(ce.lookup(torch.arange(V, device="cuda")), q, t, metric)
            assert torch.equal(via_lookup(), got), "compressed and dense ranks differ"
            l_us, _ = call_us(via_lookup, args.seconds, 20)
            row = dict(beta=beta, rows=V, dim=D, batch=B, metric=metric, blob_bytes=len(blobs[beta]),
                       device_bytes=ce.nbytes, call_us=c_us, calls=c_n, peak_extra_bytes=int(peak),
                       lookup_ranks_call_us=l_us, workspace_bytes=ce.RANKS_WORKSPACE_BYTES)
            doc["compressed"].append(row)
            print(json.dumps(row), flush=True)
        del ce
    del blobs
    torch.cuda.empty_cache()

    V, D, Bq = 100_000, 100, 16649
    means, stds = posteriors(V, D)
    rng = np.random.default_rng(16649)
    questions = np.stack([rng.choice(V, 4, replace=False) for _ in range(Bq)])
    sweep_betas = [float(grid[i]) for i in (5, 15, 24, 33, 43)]
    cb.analogy_sweep(means, stds, sweep_betas[:1], questions)                  # warm-up
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    table = cb.analogy_sweep(means, stds, sweep_betas, questions)
    torch.cuda.synchronize()
    total = time.perf_counter() - t0
    doc["analogy_sweep"] = dict(rows=V, dim=D, questions=Bq, metric="cosine", betas=sweep_betas,
                                seconds=total, seconds_per_beta=total / len(sweep_betas),
                                table_mrr_acc_hits10_bits=table.tolist())
    print(json.dumps(doc["analogy_sweep"]), flush=True)
    doc["timing"] = ("kernel: CUDA events over back-to-back vbq_score_ranks launches; call, baseline and "
                     "analogy_sweep: host clock from a synchronised start to a synchronised end; peak_extra_bytes: "
                     "torch.cuda.max_memory_allocated above the allocation before the call")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(doc, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
