"""Kernel time and rate of the rANS coder (csrc/rans.cu) on the Kodak-shaped batch of bench.py.

24 images x 32 x 48 latents x 192 channels, N = 10, learned prior with the reference initialisation.  The entropy
models are fitted on a separate seeded batch; the coded batch is quantized at lambda = 2^-6, 0.5, 8 and coded one
lambda per call and all three in one call.  Reported per configuration:
  * encode / decode kernel time (CUDA events; warmed up; back-to-back launches with the symbol planes and payloads
    L2-resident: the int32 planes are 28 MB per lambda, well inside the 126 MB L2 -- and again with the L2 overwritten
    by a 256 MB memset before every launch);
  * symbols per second;
  * coded bits against the sum of num_bits (the fitted models' ideal code lengths) and against the cross-entropy under
    the integer tables, and the flush (32 bits per active lane and group) and offset-table (32 bits per group) bits.
Writes one JSON document (with the device name and power limit read in the same run) to --out."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def power_limit():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip().splitlines()[torch.cuda.current_device()] if r.returncode == 0 else None
    except Exception:
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_rans_bench.json"))
    ap.add_argument("--iters", type=int, default=200)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_rans.py needs a CUDA device")

    import vbq_b200
    from vbq_b200 import _lib, coding, ops
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
    out = q.quantize(torch.from_numpy(mu).cuda(), torch.from_numpy(lv).cuda(), lambs, logvar=True, entropy_bits=True,
                     outputs=ops.OUT_QIDX | ops.OUT_TOTALS)
    qidx = out["qidx"].reshape(3, B, Hh * W, C).contiguous()
    ideal = out["totals"][:, 2].double().cpu().numpy()
    tables = np.stack([q.rans_tables(l) for l in lambs])
    cum_all = torch.from_numpy(coding.cum_table(tables).view(np.int16)).cuda()
    cp = q.code_points_by_channel
    lib = _lib.load()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream

    def timed(fn, flushed):
        for _ in range(5):
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
        for _ in range(max(20, args.iters // 5)):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b) * 1e3)
        return float(np.median(ts))

    results = []
    # one segment per image (the default), and 8 segments of 192 rows per image: 8x the warps, 8x the flush bits
    for sel, seg in (([0], Hh * W), ([1], Hh * W), ([2], Hh * W), ([0, 1, 2], Hh * W), ([1], 192), ([0, 1, 2], 192)):
        L = len(sel)
        planes = qidx[sel].contiguous()
        cum = cum_all[sel].contiguous()
        item_rows = Hh * W
        bound = lib.vbq_rans_payload_bound(L, B, item_rows, C, seg)
        wsb = lib.vbq_rans_workspace_bytes(L, B, item_rows, C, seg)
        payload = torch.empty(bound // 2, dtype=torch.int16, device="cuda")
        size = torch.zeros(1, dtype=torch.int64, device="cuda")
        status = torch.zeros(1, dtype=torch.int32, device="cuda")
        ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")

        def enc():
            _lib.check(lib.vbq_rans_encode(planes.data_ptr(), L, B, item_rows, C, seg, N, 16, cum.data_ptr(),
                                           payload.data_ptr(), bound, size.data_ptr(), status.data_ptr(),
                                           ws.data_ptr(), wsb, stream), "vbq_rans_encode")
        enc()
        torch.cuda.synchronize()
        assert int(status.item()) == 0
        nbytes = int(size.item())
        words = payload[:nbytes // 2].clone()
        host = words.cpu().numpy().view(np.uint16)
        # group ranges from the offset tables, as serialize.decode takes them
        G = B * (item_rows // seg) * ((C + 31) // 32)
        bl, pos = [], 0
        for _ in range(L):
            e = host[pos:pos + 2 * G].astype(np.int64)
            ends = e[0::2] | (e[1::2] << 16)
            base = pos + 2 * G
            bl.append(np.stack([base + np.concatenate([[0], ends[:-1]]), base + ends], 1))
            pos = base + int(ends[-1])
        bounds = torch.from_numpy(np.concatenate(bl)).cuda()
        zh = torch.empty((L, B, item_rows, C), dtype=torch.float32, device="cuda")
        qd = torch.empty((L, B, item_rows, C), dtype=torch.int32, device="cuda")
        dstatus = torch.zeros(1, dtype=torch.int32, device="cuda")

        def dec():
            _lib.check(lib.vbq_rans_decode(words.data_ptr(), words.numel(), bounds.data_ptr(), L, B, item_rows, C, seg, N,
                                           16, cum.data_ptr(), cp.data_ptr(), qd.data_ptr(), zh.data_ptr(),
                                           dstatus.data_ptr(), stream), "vbq_rans_decode")
        dec()
        torch.cuda.synchronize()
        assert int(dstatus.item()) == 0 and torch.equal(qd, planes), "decode mismatch"
        assert torch.equal(zh, torch.gather(cp.unsqueeze(0).unsqueeze(0).expand(L, B, C, -1), 3,
                                            planes.permute(0, 1, 3, 2).long()).permute(0, 1, 3, 2)), "z_hat mismatch"
        t_enc, t_dec = timed(enc, False), timed(dec, False)
        t_enc_f, t_dec_f = timed(enc, True), timed(dec, True)
        n_sym = L * rows * C
        pl = planes.cpu().numpy()
        xent = 0.0
        for i, s in enumerate(sel):
            f = tables[s].T[pl[i].reshape(-1, C), np.arange(C)]
            xent += float(-np.log2(f / 65536.0).sum())
        coded = 8 * nbytes
        flush_bits = 32 * C * B * (item_rows // seg) * L
        offset_bits = 32 * G * L
        sum_nb = float(sum(ideal[s] for s in sel))
        results.append(dict(
            lambdas=[lambs[s] for s in sel], seg_rows=seg, symbols=n_sym, payload_bytes=nbytes,
            encode_us=t_enc, decode_us=t_dec, encode_us_l2_flushed=t_enc_f, decode_us_l2_flushed=t_dec_f,
            encode_symbols_per_s=n_sym / (t_enc * 1e-6), decode_symbols_per_s=n_sym / (t_dec * 1e-6),
            coded_bits=coded, sum_num_bits=sum_nb, xent_bits_int_tables=xent, flush_bits=flush_bits,
            offset_bits=offset_bits, bits_per_symbol=coded / n_sym, ideal_bits_per_symbol=sum_nb / n_sym,
            overhead_tables_pct=100 * (xent - sum_nb) / sum_nb,
            overhead_coder_pct=100 * (coded - flush_bits - offset_bits - xent) / sum_nb,
            overhead_flush_pct=100 * flush_bits / sum_nb, overhead_offsets_pct=100 * offset_bits / sum_nb,
            overhead_total_pct=100 * (coded - sum_nb) / sum_nb))
        print(json.dumps(results[-1]))
    doc = dict(device=torch.cuda.get_device_name(), power_limit_and_max_sm_clock=power_limit(),
               torch=torch.__version__, workload="Kodak-shaped batch 24 x 32 x 48 x 192, N = 10, prob_bits = 16, "
               "seg_rows = 1536 (one segment per image) or 192, entropy models fitted on a separate seeded batch (add-1)",
               timing="CUDA events; 'encode_us'/'decode_us': mean over back-to-back launches, inputs L2-resident; "
                      "'*_l2_flushed': median of single launches after a 256 MB memset",
               encode_kernels="encode + offset scan + compaction (3 launches, 1 memset)",
               decode_outputs="qidx and z_hat", results=results)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(doc, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
