"""Encoding many images: one `compress_many` call against the per-image `compress_to_bytes` loop and against one
`compress_to_bytes` per shape, and the batch encoder against the single-stream encoder (csrc/rans.cu).

Workloads (N = 10, prob_bits 16, one segment per image, learned prior with the reference initialisation, entropy
models fitted on a separate seeded batch as in scripts/bench_rans_batch_decode.py):
  (a) 24 Kodak-shaped images of 32 x 48 latents x 192 channels, one lambda;
  (b) the same 24 images in mixed orientation (12 of 32 x 48, 12 of 48 x 32), three lambdas;
  (c) 64 images of distinct seeded shapes, H' and W' in [16, 64], C = 192, three lambdas.
Reported per workload:
  1. call time (host clock between synchronisations, median) of `compress_many`, of the per-image loop and of one
     `compress_to_bytes` per distinct shape; every blob is checked against the loop's in the same run;
  2. kernel time of encode + scan + compaction (CUDA events around `ops.rans_encode_batch` with every input already on
     the device), back to back with the inputs L2-resident and as single launches after a 256 MB memset;
  3. the host share of a `compress_many` call: (call - kernel) / call;
  4. for (a), `vbq_rans_encode` (encode + scan + compaction) on the equivalent single 24-item stream, the floor.
Writes one JSON document, with the GPU's name, power limit and clocks read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        return r.stdout.strip().splitlines()[torch.cuda.current_device()] if r.returncode == 0 else None
    except Exception:
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r9_rans_batch_encode.json"))
    ap.add_argument("--iters", type=int, default=30)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_rans_batch_encode.py needs a CUDA device")

    import vbq_b200
    from vbq_b200 import coding, ops, serialize
    import vbq_test_helpers as H

    C, N, B, Hh, W = 192, 10, 24, 32, 48
    pr = H.make_prior(C, seed=0)
    q = vbq_b200.ChannelwisePriorCDFQuantizer(C, N)
    q.set_code_points(ops.build_code_points_learned(torch.from_numpy(pr.packed()).cuda(), N))
    lambs = [2.0 ** -6, 0.5, 8.0]
    params = torch.from_numpy(pr.packed()).cuda()

    def latents(seed, rows):      # tests/vbq_test_helpers.make_latents, with F^-1 on the device
        rng = np.random.default_rng(seed)
        mu = ops.learned_inverse_cdf(params, torch.from_numpy(rng.uniform(0.001, 0.999, (rows, C))).cuda())
        return mu.cpu().numpy(), rng.normal(-3.0, 1.5, (rows, C)).astype(np.float32)
    mu_fit, lv_fit = latents(1, B * Hh * W)
    q.build_entropy_models_from_latents(mu_fit, lv_fit, lambs, 1)
    mu, lv = latents(2, B * Hh * W)
    mu, lv = mu.reshape(B, Hh, W, C), lv.reshape(B, Hh, W, C)
    tr = lambda a: np.ascontiguousarray(a.transpose(1, 0, 2))
    rng = np.random.default_rng(3)
    shapes = set()
    while len(shapes) < 64:
        shapes.add(tuple(int(x) for x in rng.integers(16, 65, 2)))
    shapes = sorted(shapes, key=lambda s: rng.random())
    mc, lc = latents(4, sum(h * w for h, w in shapes))
    row0 = np.cumsum([0] + [h * w for h, w in shapes])
    cases = [("(a) 24 Kodak-shaped images (32 x 48), one lambda (0.5)", [mu[b] for b in range(B)],
              [lv[b] for b in range(B)], [0.5]),
             ("(b) 24 images of mixed orientation (12 of 32 x 48, 12 of 48 x 32), three lambdas",
              [mu[b] if b % 2 else tr(mu[b]) for b in range(B)], [lv[b] if b % 2 else tr(lv[b]) for b in range(B)],
              lambs),
             ("(c) 64 images of distinct seeded shapes, H' and W' in [16, 64], three lambdas",
              [mc[row0[i]:row0[i + 1]].reshape(h, w, C) for i, (h, w) in enumerate(shapes)],
              [lc[row0[i]:row0[i + 1]].reshape(h, w, C) for i, (h, w) in enumerate(shapes)], lambs)]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def events(fn, flushed):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        if not flushed:
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(args.iters):
                fn()
            b.record()
            torch.cuda.synchronize()
            return a.elapsed_time(b) * 1e3 / args.iters
        ts = []
        for _ in range(args.iters):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b) * 1e3)
        return float(np.median(ts))

    def call_time(fn):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(args.iters):
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            ts.append((time.perf_counter() - t0) * 1e6)
        return float(np.median(ts))

    def loop(means, logvars, ls):
        out = {l: [] for l in ls}
        for m, v in zip(means, logvars):
            one = q.compress_to_bytes(m[None], v[None], ls)
            for l in ls:
                out[l] += one[l]
        return out

    def per_shape(means, logvars, ls):
        by = {}
        for b, m in enumerate(means):
            by.setdefault(m.shape, []).append(b)
        out = {l: [None] * len(means) for l in ls}
        for idx in by.values():
            got = q.compress_to_bytes(np.stack([means[b] for b in idx]), np.stack([logvars[b] for b in idx]), ls)
            for l in ls:
                for k, b in enumerate(idx):
                    out[l][b] = got[l][k]
        return out

    def batch_kernel(means, logvars, ls):
        """The three launches of compress_many's encode with every input already on the device."""
        rows = [m.shape[0] * m.shape[1] for m in means]
        qi = q.quantize(q._rows_of(means), q._rows_of(logvars), ls, logvar=True, outputs=ops.OUT_QIDX)["qidx"]
        plan = serialize.encode_plan(rows, None, C, list(range(len(ls))))
        dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
        cum = dev(np.stack([coding.cum_table(q.rans_tables(l)) for l in ls]).view(np.int16))
        pb = torch.full((len(ls),), 16, dtype=torch.int32, device="cuda")
        units, ctas, bg = dev(plan["units"]), dev(plan["ctas"]), dev(plan["blob_groups"])
        return qi, lambda: ops.rans_encode_batch(qi, cum, pb, units, ctas, bg, plan["n_groups"], N,
                                                 plan["scratch_words"])

    results = []
    for name, means, logvars, ls in cases:
        many = q.compress_many(means, logvars, ls)
        assert many == loop(means, logvars, ls) == per_shape(means, logvars, ls), name
        _, kern = batch_kernel(means, logvars, ls)
        r = dict(case=name, images=len(means), lambdas=len(ls), distinct_shapes=len({m.shape for m in means}),
                 payload_bytes=sum(len(b) for l in ls for b in many[l]),
                 loop_call_us=call_time(lambda: loop(means, logvars, ls)),
                 per_shape_call_us=call_time(lambda: per_shape(means, logvars, ls)),
                 many_call_us=call_time(lambda: q.compress_many(means, logvars, ls)),
                 many_kernel_us=events(kern, False), many_kernel_us_l2_flushed=events(kern, True))
        r["speedup_vs_loop"] = r["loop_call_us"] / r["many_call_us"]
        r["speedup_vs_per_shape"] = r["per_shape_call_us"] / r["many_call_us"]
        r["many_host_share"] = 1 - r["many_kernel_us"] / r["many_call_us"]
        results.append(r)
        print(json.dumps(r))

    # (a) against the single-stream encoder on the same 24 images as one 24-item stream
    qi, batch = batch_kernel(cases[0][1], cases[0][2], [0.5])
    cum1 = torch.from_numpy(coding.cum_table(q.rans_tables(0.5)[None]).view(np.int16)).cuda()
    single = lambda: ops.rans_encode(qi.reshape(1, B, Hh * W, C), cum1, N, 16, Hh * W)
    # the same groups, coded the same way: the blobs' offset tables and group data add up to the single stream's
    _, size, _ = single()
    _, meta = batch()
    assert int(meta[B].item()) == int(size.item()) // 2, "batch blobs and single stream differ in size"
    floor = dict(single_stream_us=events(single, False), batch_us=events(batch, False),
                 single_stream_us_l2_flushed=events(single, True), batch_us_l2_flushed=events(batch, True))
    floor["ratio"] = floor["batch_us"] / floor["single_stream_us"]
    floor["ratio_l2_flushed"] = floor["batch_us_l2_flushed"] / floor["single_stream_us_l2_flushed"]
    print(json.dumps(floor))

    doc = dict(gpu_name_power_limit_max_sm_clock_sm_clock=gpu_info(), device=torch.cuda.get_device_name(),
               torch=torch.__version__,
               workload="N = 10, C = 192, prob_bits = 16, one segment per image, entropy models fitted on a separate "
                        "seeded batch (add-1); host float32 latents in; blobs as compress_to_bytes returns them",
               timing="call_us: median host clock of a call ending in a device synchronise; kernel_us: CUDA events "
                      "around encode + scan + compaction, mean over back-to-back calls with the inputs on the device "
                      "and L2-resident; *_l2_flushed: median of single calls after a 256 MB memset",
               goals=dict(batch_within_1_2x_of_single_stream_on_a=floor["ratio"] <= 1.2,
                          many_10x_faster_than_loop_on_b_and_c=all(r["speedup_vs_loop"] >= 10 for r in results[1:])),
               iters=args.iters, results=results, batch_vs_single_stream=floor)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(doc, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
