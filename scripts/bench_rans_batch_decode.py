"""Decoding many VBQ2 blobs: the per-blob `decompress_from_bytes` loop against one `decompress_many` call, and the
batch kernel against the single-stream decoder (csrc/rans.cu).

Workload of scripts/bench_rans.py (DESIGN §8c): 24 Kodak-shaped images of 32 x 48 latents x 192 channels, N = 10,
learned prior with the reference initialisation, entropy models fitted on a separate seeded batch, prob_bits 16, one
segment per image.  The blobs are those `compress_to_bytes` returns, one per (lambda, image).  Reported:
  1. call time (host clock between synchronisations, median) of the per-blob loop and of `decompress_many`, and their
     kernel time (CUDA events around the launches alone, inputs already on the device), for 24 blobs of one lambda, 72
     blobs of three lambdas and 24 blobs of mixed orientation (12 of 32 x 48, 12 of 48 x 32);
  2. the batch kernel on the 24 blobs of one lambda against `vbq_rans_decode` on the equivalent single 24-item stream
     (`serialize.encode(items=24)`), the floor;
  3. the host share of each call: (call - kernel) / call.
Kernel times are taken twice: back to back with the inputs L2-resident, and as single launches after a 256 MB memset
that overwrites the L2.  Writes one JSON document, with the GPU's name, power limit and clocks read in the same run."""
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
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r8_rans_batch_decode.json"))
    ap.add_argument("--iters", type=int, default=50)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_rans_batch_decode.py needs a CUDA device")

    import vbq_b200
    from vbq_b200 import coding, ops, serialize
    import vbq_test_helpers as H

    C, N, B, Hh, W = 192, 10, 24, 32, 48
    rows = B * Hh * W
    pr = H.make_prior(C, seed=0)
    q = vbq_b200.ChannelwisePriorCDFQuantizer(C, N)
    q.set_code_points(ops.build_code_points_learned(torch.from_numpy(pr.packed()).cuda(), N))
    lambs = [2.0 ** -6, 0.5, 8.0]
    params = torch.from_numpy(pr.packed()).cuda()

    def latents(seed):      # tests/vbq_test_helpers.make_latents, with F^-1 on the device
        rng = np.random.default_rng(seed)
        mu = ops.learned_inverse_cdf(params, torch.from_numpy(rng.uniform(0.001, 0.999, (rows, C))).cuda())
        return mu.cpu().numpy(), rng.normal(-3.0, 1.5, (rows, C)).astype(np.float32)
    mu_fit, lv_fit = latents(1)
    q.build_entropy_models_from_latents(mu_fit, lv_fit, lambs, 1)
    mu, lv = latents(2)
    mu, lv = mu.reshape(B, Hh, W, C), lv.reshape(B, Hh, W, C)
    blobs = q.compress_to_bytes(mu, lv, lambs)
    tr = q.compress_to_bytes(np.ascontiguousarray(mu.transpose(0, 2, 1, 3)),
                             np.ascontiguousarray(lv.transpose(0, 2, 1, 3)), [0.5])[0.5]
    cp = q.code_points_by_channel
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

    def tables_of(h):
        return [q.rans_tables(l, h["prob_bits"]) for l in h["lambdas"]]

    def loop_kernels(bl):
        """The per-blob launches of decompress_from_bytes with every input already on the device."""
        args_ = []
        for blob in bl:
            h = serialize.read_header(blob)
            words = serialize._payload_words(blob, h)
            t = np.stack(tables_of(h))
            args_.append((torch.from_numpy(words.view(np.int16).copy()).cuda(),
                          torch.from_numpy(serialize._group_bounds(words, h)).cuda(),
                          torch.from_numpy(coding.cum_table(t).view(np.int16)).cuda(), h))
        return lambda: [ops.rans_decode(w, b, c, h["items"], h["item_rows"], h["seg_rows"], N, h["prob_bits"], cp,
                                        False) for w, b, c, h in args_]

    def batch_kernel(bl):
        """The one launch of decompress_many with every input already on the device."""
        headers = [serialize.read_header(b) for b in bl]
        distinct, ids = [], []
        for h in headers:
            row = []
            for t in tables_of(h):
                k = [i for i, d in enumerate(distinct) if d is t]
                if not k:
                    distinct.append(t)
                    k = [len(distinct) - 1]
                row.append(k[0])
            ids.append(row)
        plan = serialize.batch_plan(headers, [serialize._payload_words(b, h) for b, h in zip(bl, headers)], ids)
        w = torch.from_numpy(plan["words"].view(np.int16)).cuda()
        cum = torch.from_numpy(np.stack([coding.cum_table(t) for t in distinct]).view(np.int16)).cuda()
        pb = torch.full((len(distinct),), 16, dtype=torch.int32, device="cuda")
        units, ctas = torch.from_numpy(plan["units"]).cuda(), torch.from_numpy(plan["ctas"]).cuda()
        return lambda: ops.rans_decode_batch(w, cum, pb, units, ctas, len(bl), N, plan["n_out"], cp, False)

    results = []
    cases = [("24 blobs, one lambda (0.5)", blobs[0.5]),
             ("72 blobs, three lambdas", [b for l in lambs for b in blobs[l]]),
             ("24 blobs, mixed orientation (12 of 32 x 48, 12 of 48 x 32), lambda 0.5", blobs[0.5][:12] + tr[:12])]
    for name, bl in cases:
        loop = [q.decompress_from_bytes(b) for b in bl]
        many = q.decompress_many(bl)
        assert all(torch.equal(a, b) for a, b in zip(loop, many)), name
        r = dict(case=name, blobs=len(bl),
                 loop_call_us=call_time(lambda: [q.decompress_from_bytes(b) for b in bl]),
                 many_call_us=call_time(lambda: q.decompress_many(bl)),
                 loop_kernel_us=events(loop_kernels(bl), False), many_kernel_us=events(batch_kernel(bl), False),
                 loop_kernel_us_l2_flushed=events(loop_kernels(bl), True),
                 many_kernel_us_l2_flushed=events(batch_kernel(bl), True))
        r["speedup_call"] = r["loop_call_us"] / r["many_call_us"]
        r["loop_host_share"] = 1 - r["loop_kernel_us"] / r["loop_call_us"]
        r["many_host_share"] = 1 - r["many_kernel_us"] / r["many_call_us"]
        results.append(r)
        print(json.dumps(r))

    # the batch kernel against the single-stream decoder on the same 24 images as one 24-item stream
    qi = q.quantize(torch.from_numpy(mu.reshape(-1, C)).cuda(), torch.from_numpy(lv.reshape(-1, C)).cuda(), [0.5],
                    logvar=True, outputs=ops.OUT_QIDX)["qidx"]
    t = q.rans_tables(0.5)
    stream = serialize.encode(qi, t, N, items=B, lambdas=[0.5], height=Hh)
    h = serialize.read_header(stream)
    words = serialize._payload_words(stream, h)
    sw = torch.from_numpy(words.view(np.int16).copy()).cuda()
    sb = torch.from_numpy(serialize._group_bounds(words, h)).cuda()
    sc = torch.from_numpy(coding.cum_table(t[None]).view(np.int16)).cuda()
    single = lambda: ops.rans_decode(sw, sb, sc, B, Hh * W, Hh * W, N, 16, cp, False)
    batch = batch_kernel(blobs[0.5])
    assert torch.equal(single()[1].reshape(-1), batch()[1]), "batch and single stream differ"
    floor = dict(single_stream_us=events(single, False), batch_us=events(batch, False),
                 single_stream_us_l2_flushed=events(single, True), batch_us_l2_flushed=events(batch, True))
    floor["ratio"] = floor["batch_us"] / floor["single_stream_us"]
    floor["ratio_l2_flushed"] = floor["batch_us_l2_flushed"] / floor["single_stream_us_l2_flushed"]
    print(json.dumps(floor))

    doc = dict(gpu_name_power_limit_max_sm_clock_sm_clock=gpu_info(), device=torch.cuda.get_device_name(),
               torch=torch.__version__,
               workload="Kodak-shaped batch 24 x 32 x 48 x 192, N = 10, prob_bits = 16, one segment per image, "
                        "entropy models fitted on a separate seeded batch (add-1); blobs from compress_to_bytes",
               timing="call_us: median host clock of a call ending in a device synchronise; kernel_us: CUDA events, "
                      "mean over back-to-back launches with the inputs on the device and L2-resident; "
                      "*_l2_flushed: median of single launches (or launch sequences) after a 256 MB memset",
               outputs="z_hat only, as decompress_from_bytes / decompress_many", iters=args.iters,
               results=results, batch_vs_single_stream=floor)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(doc, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
