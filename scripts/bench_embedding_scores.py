"""Query scoring straight from VBQE blobs (CompressedEmbedding.scores / topk, vbq_rans_shared_row_scores) on the
posteriors of bench_embedding_lookup.py: 1 M x 300 seeded Gaussian posteriors, N = 10, codebook std 1.2356,
exact=True, prob_bits 16, default segmentation and checkpoint interval, at beta = 0.518, 26.8 and 1,931, plus
200 k x 300 at beta = 1e5 with two segments.

For B = 1, 8, 64 and 256 queries (seeded standard normal), k = 10, dot and cosine, it reports:
  * scan_kernel_us: one scan of every row (the vbq_rans_shared_row_scores launches of all query tiles), CUDA events
    over back-to-back scans;
  * topk_call_us: CompressedEmbedding.topk, host clock from a synchronised start to a synchronised end;
  * topk_peak_extra_bytes: torch.cuda.max_memory_allocated during topk above what was allocated before it;
and two baselines on the same queries:
  * lookup_mm_topk_call_us: lookup(arange(V)) on the same object, then mm (and the norms for cosine), then topk;
  * dense_mm_topk_call_us: the float32 matrix already on the device, then mm (and norms), then topk: a lower bound
    that needs the dense matrix.
A scan re-reads the payload, which stays in the 126 MB L2 when it fits (beta = 1,931 and 1e5), so those kernel times
are L2-warm.  Writes one JSON document (with the device name, power limit and SM clock read in the same run) to
--out."""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from bench_embedding_coding import power_limit, timed_us   # noqa: E402
from bench_embedding_lookup import call_us                 # noqa: E402

BATCHES = [1, 8, 64, 256]
K_TOP = 10


def dense_topk(Z, q, metric, zn=None):
    s = q @ Z.T
    if metric == "cosine":
        s = s / (zn[None, :] * q.norm(dim=1, keepdim=True)).clamp_min(1e-30)
    return torch.topk(s, K_TOP, dim=1)


def measure(ce, dense, V, B, metric, seconds):
    q = torch.randn((B, 300), generator=torch.Generator(device="cuda").manual_seed(B), device="cuda")
    out = torch.empty((B, V), dtype=torch.float32, device="cuda")
    status = torch.zeros(1, dtype=torch.int32, device="cuda")
    scan_us, scan_n = timed_us(lambda: ce._scores_into(q, 0, V, metric, out, status), seconds, 200)
    assert int(status.item()) == 0
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    vals, ids = ce.topk(q, K_TOP, metric=metric)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    assert torch.equal(vals, out.gather(1, ids)), "topk values differ from the scan"
    topk_us, topk_n = call_us(lambda: ce.topk(q, K_TOP, metric=metric), seconds, 200)

    def via_lookup():
        Z = ce.lookup(torch.arange(V, device="cuda"))
        return dense_topk(Z, q, metric, Z.norm(dim=1) if metric == "cosine" else None)
    look_us, _ = call_us(via_lookup, seconds, 50)
    zn = dense.norm(dim=1) if metric == "cosine" else None
    dense_us, _ = call_us(lambda: dense_topk(dense, q, metric, zn), seconds, 200)
    return dict(batch=B, metric=metric, k=K_TOP, scan_kernel_us=scan_us, scan_launches=scan_n, topk_call_us=topk_us,
                topk_calls=topk_n, topk_peak_extra_bytes=int(peak), lookup_mm_topk_call_us=look_us,
                dense_mm_topk_call_us=dense_us)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r6_embedding_scores.json"))
    ap.add_argument("--rows", type=int, default=1_000_000)
    ap.add_argument("--small-rows", type=int, default=200_000)
    ap.add_argument("--seconds", type=float, default=0.3, help="about this long per timed configuration")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_embedding_scores.py needs a CUDA device")

    import vbq_b200
    from vbq_b200 import serialize

    N, D = 10, 300
    grid = np.exp(np.linspace(np.log(0.01), np.log(100000), 50))
    cb = vbq_b200.GaussianCodebook(1.2356, N)

    def posteriors(V):
        g = torch.Generator(device="cuda")
        g.manual_seed(77)
        means = torch.randn((V, D), generator=g, device="cuda") * 1.2329 - 0.08
        stds = torch.exp(torch.randn((V, D), generator=g, device="cuda") * 0.7 + float(np.log(0.04)))
        return means, stds

    runs = [(args.rows, [float(grid[i]) for i in (12, 24, 37)], None), (args.small_rows, [1e5], "half")]
    results = []
    for V, betas, seg in runs:
        means, stds = posteriors(V)
        seg_rows = None if seg is None else -(-V * D // 32) // 2 + 1
        blobs = cb.compress_to_bytes(means, stds, betas, seg_rows=seg_rows)
        del means, stds
        for beta in betas:
            blob = blobs[beta]
            h = serialize.read_embedding_header(blob)
            dense = cb.decompress_from_bytes(blob)
            ce = vbq_b200.CompressedEmbedding(blob)
            res = dict(beta=beta, rows=V, dim=D, segments=int(h["bounds"].shape[0]), blob_bytes=len(blob),
                       checkpoint_rows=ce.checkpoint_rows, device_bytes=ce.nbytes, dense_bytes=dense.numel() * 4,
                       cases=[])
            for B in BATCHES:
                for metric in ("dot", "cosine"):
                    row = measure(ce, dense, V, B, metric, args.seconds)
                    res["cases"].append(row)
                    print(json.dumps(dict(beta=beta, rows=V, **row)), flush=True)
            results.append(res)
            del dense, ce
            torch.cuda.empty_cache()
    doc = dict(device=torch.cuda.get_device_name(), power_limit_and_max_sm_clock=power_limit(),
               torch=torch.__version__,
               workload="%d x %d Gaussian posteriors (seed 77), N = 10, codebook std 1.2356, exact=True, prob_bits 16, "
                        "default segmentation and checkpoint interval; beta = 1e5 on %d x %d with two segments; "
                        "seeded standard-normal queries, k = %d" % (args.rows, D, args.small_rows, D, K_TOP),
               timing="scan_kernel: CUDA events over back-to-back full scans (every query tile); topk, lookup_mm_topk "
                      "and dense_mm_topk: host clock from a synchronised start to a synchronised end; "
                      "topk_peak_extra_bytes: torch.cuda.max_memory_allocated above the allocation before the call",
               results=results)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(doc, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
