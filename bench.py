#!/usr/bin/env python
"""Benchmark of the VBQ rate-distortion quantization step (BASELINE.json metric: coordinates quantized / second).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
  torchrun --nproc-per-node N bench.py --gpus N ...        (one rank per GPU)

A "step" is one pass of the hot path over one batch: the Kodak-shaped bls2017 latent batch of BASELINE.json
configs[1] (24 images x 32x48 x 192 channels = 7,077,888 coordinates, learned factorized prior at reference init,
max_bits_per_coord=10, single lambda=0.5), written out as sorted quantile index (int32) + code length (float32)
per coordinate, plus the per-lambda rate/distortion totals.  With N>1 every rank processes its own batch of that
shape (weak scaling, no data-path collective) and the totals are all-reduced over NCCL inside the timed region, once
per call (`scaling_variants` also reports four calls per collective).  The same JSON line carries `corrected` (the
reference's production mode: corrected code lengths + entropy-model bits) and `configs` (BASELINE.json configs[2..4]
at this N through sharding.ShardedQuantizer).

`value` is device-resident throughput (CUDA events, max over ranks); `e2e` goes through the reference-facing
ChannelwisePriorCDFQuantizer.compress_batch_channel_latents-level call with pinned HOST buffers (H2D and D2H
inside the timed region); `--impl reference` times the CPU oracle port of the reference's TF-eager quantizer."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

IMAGES, H, W, C, N_BITS = 24, 32, 48, 192, 10
ROWS = IMAGES * H * W
COORDS = ROWS * C
LAMB = 0.5
BYTES_PER_COORD = 16          # read mu, sigma; write quantile index + code length (SURVEY.md §8d)
L2_BYTES = 126 * 2 ** 20
METRIC = "VBQ coordinates quantized per second"
UNIT = "coords/s"
WORKLOAD = "bls2017 Kodak-shaped latents: 24x32x48x192, learned prior (reference init), N=10, lambda=0.5"


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f), "measured"
    return {"hbm_gbs": 6650.0}, "fallback"


class ClockSampler:
    """SM clock and throttle reasons sampled every ~2 ms WHILE the timed region runs (NVML; the fields are the ones
    of the recipe's `nvidia-smi --query-gpu=clocks.sm,clocks.max.sm,clocks_event_reasons.*` line)."""

    def __init__(self, index):
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop = threading.Event()
        self._thread = None

    def __enter__(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[self.index]) if vis and vis.split(",")[self.index].isdigit() else self.index
            h = nv.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {"hw_slowdown": nv.nvmlClocksEventReasonHwSlowdown,
                     "hw_thermal_slowdown": nv.nvmlClocksEventReasonHwThermalSlowdown,
                     "sw_thermal_slowdown": nv.nvmlClocksEventReasonSwThermalSlowdown,
                     "sw_power_cap": nv.nvmlClocksEventReasonSwPowerCap}

            def loop():
                while not self._stop.is_set():
                    try:
                        self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                        r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                        for k, bit in names.items():
                            if r & bit:
                                self.reasons.add(k)
                    except Exception:
                        pass
                    time.sleep(0.002)

            self._thread = threading.Thread(target=loop, daemon=True)
            self._thread.start()
        except Exception:
            self._thread = None
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._thread is not None:
            self._thread.join(timeout=1)

    def summary(self):
        if not self.samples:
            return None
        sm = sorted(self.samples)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(sm)}


# --------------------------------------------------------------------------------------------------------
# synthetic workload
# --------------------------------------------------------------------------------------------------------
def prior_parameters(seed=2, init_scale=10.0):
    """Reference initialisation of BMSHJ2018Prior (learned_prior.py:30-58) in NumPy: constant softplus^-1
    matrices, biases U(-.5,.5), zero factors.  Used by both arms so they quantize against the same prior."""
    rng = np.random.default_rng(seed)
    fdims = (1, 3, 3, 3, 1)
    scale = init_scale ** (1 / 4)
    mats, bs, fs = [], [], []
    for i in range(4):
        init = np.log(np.expm1(1 / scale / fdims[i + 1]))
        mats.append(np.logaddexp(0.0, np.full((C, fdims[i + 1], fdims[i]), init, dtype=np.float32)).astype(np.float32))
        bs.append(rng.uniform(-.5, .5, size=(C, fdims[i + 1], 1)).astype(np.float32))
        if i < 3:
            fs.append(np.zeros((C, fdims[i + 1], 1), dtype=np.float32))
    return mats, bs, fs


def make_prior_and_quantizer(device):
    import vbq_b200
    prior = vbq_b200.BMSHJ2018Prior(C, dims=(3, 3, 3), init_scale=10., device=device)
    prior.set_transformed_parameters(*prior_parameters())
    q = vbq_b200.ChannelwisePriorCDFQuantizer(C, N_BITS, device=device)
    q.build_code_points(prior)
    return prior, q


def make_batch_cpu(table, seed, n_images):
    """CPU-only generator for the reference arm: mu by linear interpolation of the tabulated quantile function at
    u ~ U(0.001, 0.999) (same distribution as `make_batch`), logvar ~ N(-3, 1.5^2)."""
    rng = np.random.default_rng(seed)
    rows = n_images * H * W
    srt = np.sort(table, axis=1)
    xi_sorted = (np.arange(srt.shape[1]) + 1.0) / (srt.shape[1] + 1.0)
    u = rng.uniform(0.001, 0.999, (rows, C))
    mu = np.stack([np.interp(u[:, c], xi_sorted, srt[c]) for c in range(C)], axis=1).astype(np.float32)
    logvar = rng.normal(-3.0, 1.5, (rows, C)).astype(np.float32)
    return mu, (np.exp(logvar) ** np.float32(0.5)).astype(np.float32)


def make_batch(prior, seed, device):
    """mu = F_c^-1(U(0.001,0.999)), logvar ~ N(-3, 1.5^2) (SURVEY.md §8d C2); returns (mu, sigma) (ROWS, C) f32."""
    import torch
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    u = torch.rand((ROWS, C), generator=g, device=device, dtype=torch.float64) * 0.998 + 0.001
    mu = prior.inverse_cdf(u).contiguous()
    logvar = torch.randn((ROWS, C), generator=g, device=device, dtype=torch.float32) * 1.5 - 3.0
    sigma = torch.exp(logvar) ** 0.5
    return mu, sigma.contiguous()


# --------------------------------------------------------------------------------------------------------
# CPU arm: oracle port of the reference's TF-eager quantizer (quantizer.py:156-188 + utils.py:363-423)
# --------------------------------------------------------------------------------------------------------
_W = {}


def _cpu_init(table):
    from oracle import vbq_oracle as O
    oq = O.QuantizerNP(C, N_BITS)
    oq.set_code_points(table, build_grids=True)
    _W["q"] = oq


def _cpu_one_image(args):
    mu, sigma = args
    Z, B = _W["q"].compress_batch_channel_latents(mu, sigma, [LAMB], fast_intervals=False)
    return float(B[LAMB].sum())


def cpu_throughput(table, mu, sigma, n_images, workers, repeats=1):
    """coords/s of the oracle port over ``n_images`` Kodak-shaped images, one image per call like the reference's
    evaluation loop (utils.py:535-542), ``workers`` processes."""
    import multiprocessing as mp
    per = H * W
    jobs = [(mu[i * per:(i + 1) * per], sigma[i * per:(i + 1) * per]) for i in range(n_images)]
    if workers <= 1:
        _cpu_init(table)
        t0 = time.perf_counter()
        for _ in range(repeats):
            for j in jobs:
                _cpu_one_image(j)
        dt = (time.perf_counter() - t0) / repeats
    else:
        with mp.get_context("fork").Pool(workers, initializer=_cpu_init, initargs=(table,)) as pool:
            pool.map(_cpu_one_image, jobs[:workers])           # warm the workers
            t0 = time.perf_counter()
            for _ in range(repeats):
                pool.map(_cpu_one_image, jobs, chunksize=1)
            dt = (time.perf_counter() - t0) / repeats
    return n_images * per * C / dt, dt


def run_reference(args, rank, world):
    """`--impl reference`: the reference's CPU path (oracle port; TensorFlow 1.15 is not installable here) on the
    host cores, rank 0 only."""
    if rank != 0:
        return
    from oracle import vbq_oracle as O
    pr = O.LearnedPriorNP(*prior_parameters())
    xi = O.xi_heap(N_BITS)
    table = pr.inverse_cdf_f64(np.repeat(xi[:, None], C, axis=1), iters=64).T
    mu, sigma = make_batch_cpu(table, 1000, IMAGES)
    cores = os.cpu_count() or 1
    workers = max(1, min(cores, IMAGES))
    import multiprocessing as mp
    per = H * W
    budget_s = 100.0                       # the whole --steps K run stays within a few minutes whatever K is
    with mp.get_context("fork").Pool(workers, initializer=_cpu_init, initargs=(table,)) as pool:
        def run(rows_per_job, n_jobs):
            jobs = [(mu[(i % IMAGES) * per:(i % IMAGES) * per + rows_per_job],
                     sigma[(i % IMAGES) * per:(i % IMAGES) * per + rows_per_job]) for i in range(n_jobs)]
            t0 = time.perf_counter()
            pool.map(_cpu_one_image, jobs, chunksize=1)
            return time.perf_counter() - t0
        run(per, workers)                  # warm the workers (search grids, caches)
        t_img = run(per, workers)          # one image per worker
        for _ in range(max(0, args.warmup - 2)):
            run(per, workers)
        # a step is a bounded sample of the workload: whole images (one per call, like utils.py:535-542) while they fit
        # the per-step share of the budget, otherwise the first rows of one image per worker
        share = budget_s / max(args.steps, 1)
        if share >= t_img:
            n_jobs = int(min(IMAGES, workers * max(1, int(share / t_img))))
            rows_per_job = per
        else:
            n_jobs = workers
            rows_per_job = int(max(64, per * share / t_img))
        t0 = time.perf_counter()
        for _ in range(args.steps):
            run(rows_per_job, n_jobs)
        total = time.perf_counter() - t0
    coords_per_step = n_jobs * rows_per_job * C
    value = coords_per_step * args.steps / total
    sample = "%d jobs of %d rows x %d channels per step (%s), one call per job, %d worker processes" % (
        n_jobs, rows_per_job, C, "whole Kodak-shaped images" if rows_per_job == per else "leading rows of an image",
        workers)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": workers, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# --------------------------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------------------------
def bind_to_gpu_numa_node(index):
    """Pin this rank's host threads to the CPUs that are local to its GPU (NVML affinity) before any pinned host
    buffer is allocated, so that the e2e leg's PCIe traffic does not cross sockets.  Best effort."""
    try:
        import pynvml as nv
        nv.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        phys = int(vis.split(",")[index]) if vis and vis.split(",")[index].isdigit() else index
        nv.nvmlDeviceSetCpuAffinity(nv.nvmlDeviceGetHandleByIndex(phys))
    except Exception:
        pass



def _time_steps(fn, steps, warmup, barrier, finish=None):
    """CUDA-event time of `steps` calls of fn(i) bracketed by barriers; returns milliseconds (this rank)."""
    import torch
    for i in range(warmup):
        fn(i)
    if finish:
        finish()
    barrier()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    t0 = time.perf_counter()
    for i in range(steps):
        fn(warmup + i)
    _time_steps.host_issue_us = 1e6 * (time.perf_counter() - t0) / max(steps, 1)   # host time to ENQUEUE one step
    if finish:
        finish()
    ev[1].record()
    barrier()
    return ev[0].elapsed_time(ev[1])


def dump_outputs(directory, **arrays):
    """Write each device tensor as <directory>/<name>.npy, integers as float32 (exact: code indices are < 2^24) and
    floats at their own precision.  The headline outputs come to 2 x 27 MiB + 32 bytes, so they are written in full
    rather than sampled."""
    os.makedirs(directory, exist_ok=True)
    for name, t in arrays.items():
        a = t.detach().cpu().numpy()
        if a.dtype.kind != "f":
            a = a.astype(np.float32)
        np.save(os.path.join(directory, name + ".npy"), a)


def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    import vbq_b200
    from vbq_b200 import ops, sharding

    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    bind_to_gpu_numa_node(local_rank)
    prior, q = make_prior_and_quantizer(dev)
    pen, length = q._length_tables([LAMB])
    args.flags = ops.search_flags([LAMB], args.flags)   # what the facade passes for this lambda
    if world > 1 and not args.no_reserve:
        args.flags |= ops.FLAG_RESERVE_SM               # leave one SM to the overlapped NCCL all-reduce

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # rotating buffer sets so that no step finds its inputs in the 126 MB L2
    set_bytes = COORDS * BYTES_PER_COORD
    n_sets = max(3, -(-3 * L2_BYTES // set_bytes))
    sets = []
    for s in range(n_sets):
        mu, sigma = make_batch(prior, 1000 + 17 * rank + s, dev)
        sets.append(dict(mu=mu, sigma=sigma,
                         qidx=torch.empty((1, ROWS, C), dtype=torch.int32, device=dev),
                         bits=torch.empty((1, ROWS, C), dtype=torch.float32, device=dev)))

    # ---- headline: device-resident steps ---------------------------------------------------------------------------
    # A step is one prebound vbq_quantize call = one kernel launch incl. the per-lambda totals.  N > 1: the (1, 4) totals
    # are all-reduced over NCCL inside the timed region (sharding.all_reduce_totals, asynchronous on NCCL's stream,
    # overlapping the next kernels): once per call (`collective_every` = 1, the headline) and, for comparison, the totals
    # of n_sets consecutive calls in one collective.
    def headline(every):
        n_buckets = 2 if world > 1 else 1
        buckets = [torch.zeros((every, 1, 4), dtype=torch.float64, device=dev) for _ in range(n_buckets)]
        plans = [[[ops.QuantizePlan(b["mu"], b["sigma"], q.all_code_points, q._packed, pen, length, None, N_BITS,
                                    qidx=b["qidx"], bits=b["bits"], totals=buckets[k][e], flags=args.flags,
                                    graph=args.graph) for b in sets] for e in range(every)] for k in range(n_buckets)]
        pending = [None] * n_buckets
        last = {"i": -1, "totals": None}

        def step(i):
            last["i"] = i
            k, e = (i // every) % n_buckets, i % every
            if e == 0 and pending[k] is not None:
                pending[k].wait()
                pending[k] = None
            last["totals"] = plans[k][e][i % n_sets].run()
            if world > 1 and e == every - 1:
                pending[k] = sharding.all_reduce_totals(buckets[k], async_op=True)

        def drain():
            if world > 1:
                for k in range(n_buckets):
                    if pending[k] is not None:
                        pending[k].wait()
                        pending[k] = None
                i = last["i"]      # a partially filled last bucket is reduced here
                if i >= 0 and i % every != every - 1:
                    sharding.all_reduce_totals(buckets[(i // every) % n_buckets])
                    last["i"] = -1
        return step, drain, last

    # N > 1, headline: NO collective launch at all — while call i runs, an idle lane of its kernel writes the totals of call
    # i-1 into every rank's inbox over NVLink and collects (waits for + adds in rank order) the all-reduced totals of call
    # i-3 (sharding.PeerTotals / vbq_quantize_peer): one exchange per call, hidden behind the search, no stream operation
    # between the kernels, all 148 SMs.  The last calls of a run are flushed by the one-CTA push / collect kernels.
    def headline_peer():
        flags = args.flags & ~ops.FLAG_RESERVE_SM
        peer = sharding.PeerTotals(n_lambda_max=1)
        local = [torch.zeros((1, 4), dtype=torch.float64, device=dev) for _ in sets]
        plans = [ops.QuantizePlan(b["mu"], b["sigma"], q.all_code_points, q._packed, pen, length, None, N_BITS,
                                  qidx=b["qidx"], bits=b["bits"], totals=local[s_], flags=flags, peer=peer)
                 for s_, b in enumerate(sets)]
        glob = [torch.zeros((1, 4), dtype=torch.float64, device=dev) for _ in range(8)]
        calls = []          # (sequence number, buffer set) of the calls of this run

        def step(i):
            calls.append((peer.next_seq(), i % n_sets))
            k = len(calls) - 1
            push = calls[k - 1] if k >= 1 else None           # deliver the previous call's totals (n_sets >= 3: its buffer is intact)
            coll = calls[k - 3] if k >= 3 else None           # collect the call three steps back
            plans[i % n_sets].run_peer(push[0] if push else 0, local[push[1]] if push else None,
                                       coll[0] if coll else 0, glob[(k - 3) % 8] if coll else None)

        def drain():
            n = len(calls)
            if n:
                peer.push(calls[n - 1][0], local[calls[n - 1][1]])
                for k in range(max(0, n - 3), n):
                    peer.collect(calls[k][0], 1, glob[k % 8])
            del calls[:]
        return step, drain, peer, glob, local

    variants = {}
    if world > 1:
        step, drain, peer, glob, local = headline_peer()
        variants["headline"] = "peer inboxes over NVLink: call i delivers the totals of call i-1 and collects those of call i-3 while it runs"
    else:
        step, drain, last = headline(1)
    with ClockSampler(local_rank) as clocks:
        total_ms = max_over_ranks(_time_steps(step, args.steps, args.warmup, barrier, drain))
    value = COORDS * world * args.steps / (total_ms * 1e-3)
    host_issue_us = _time_steps.host_issue_us
    last_k = args.warmup + args.steps - 1      # call index of the last timed step
    if world > 1:
        # the exchanged totals are the NCCL all-reduce of the local ones (last call of the timed region)
        torch.cuda.synchronize()
        want = sharding.all_reduce_totals(local[last_k % n_sets].clone())
        got = glob[(args.steps - 1) % 8]
        assert torch.allclose(got, want, rtol=1e-12), (got, want)
    if args.dump_outputs and rank == 0:
        out = sets[last_k % n_sets]
        dump_outputs(args.dump_outputs, qidx=out["qidx"], bits=out["bits"], totals=got if world > 1 else last["totals"])
    if world > 1:
        for every in (1, n_sets):       # for comparison: the same steps with NCCL all-reduces (147 CTAs + 1 SM for NCCL)
            stepn, drainn, _ = headline(every)
            msn = max_over_ranks(_time_steps(stepn, args.steps, args.warmup, barrier, drainn))
            variants["nccl_collective_every_%d" % every] = {"value": COORDS * world * args.steps / (msn * 1e-3), "unit": UNIT}

    # ---- end to end through the reference-facing call on HOST arrays -------------------------------------------------
    # ChannelwisePriorCDFQuantizer.compress_batch_channel_latents(batch_means, batch_stds, lambs) on pinned NumPy arrays
    # (quantizer.py:156-188): the facade feeds the chunked upload / kernel / download pipeline (vbq_quantize_host) and
    # returns Z_hat_dict, num_bits_dict as host arrays; every byte crosses PCIe inside the timed region.
    h_in = [(b["mu"].cpu().pin_memory().numpy(), b["sigma"].cpu().pin_memory().numpy()) for b in (sets * 2)[:2]]
    state = {}

    def e2e_step(i):
        Z, B = q.compress_batch_channel_latents(h_in[i % 2][0], h_in[i % 2][1], [LAMB])
        state["last"] = (Z[LAMB], B[LAMB])

    e2e_steps = max(3, min(args.steps, 20))
    for i in range(5):      # warm-up: the facade's pinned output buffers come from PyTorch's caching host allocator
        e2e_step(i)             # (the last one, i = 4, used input set 0: checked below)
    # the facade must reproduce the device-resident results exactly: its z_hat is the code point the index names
    step(0)
    drain()
    torch.cuda.synchronize()
    zt = q.code_points_by_channel.t().contiguous()
    want_z = torch.gather(zt, 0, sets[0]["qidx"][0].long()).cpu().numpy()
    assert np.array_equal(state["last"][0], want_z) and np.array_equal(state["last"][1], sets[0]["bits"][0].cpu().numpy().astype(np.int32))
    barrier()
    t0 = time.perf_counter()
    for i in range(e2e_steps):
        e2e_step(i)
    barrier()
    e2e_value = COORDS * world * e2e_steps / max_over_ranks(time.perf_counter() - t0)
    # what the box moves at most: the same bytes per step as bare pinned copies (H2D on one stream, D2H on another)
    d_a = torch.empty((2, ROWS, C), dtype=torch.float32, device=dev)
    h_a = torch.empty((2, ROWS, C), dtype=torch.float32).pin_memory()
    h_b2 = torch.empty((2, ROWS, C), dtype=torch.float32).pin_memory()
    s1, s2 = torch.cuda.Stream(dev), torch.cuda.Stream(dev)

    def copy_step(i):
        with torch.cuda.stream(s1):
            d_a.copy_(h_a, non_blocking=True)
        with torch.cuda.stream(s2):
            h_b2.copy_(d_a, non_blocking=True)

    for i in range(2):
        copy_step(i)
    barrier()
    t0 = time.perf_counter()
    for i in range(e2e_steps):
        copy_step(i)
    barrier()
    ceiling = COORDS * world * e2e_steps / max_over_ranks(time.perf_counter() - t0)
    del d_a, h_a, h_b2

    # ---- the reference's production mode: corrected code lengths + entropy-model bits (quantizer.py:166-180, :223-228) --
    extra = {}
    if not args.headline_only:
        extra["corrected"] = bench_corrected(q, sets, world, dev, barrier, max_over_ranks)
        extra["configs"] = bench_configs(prior, q, rank, world, dev, barrier, max_over_ranks)

    if rank != 0:
        return
    peaks, peak_kind = measured_peaks()
    traffic = None
    tp = os.path.join(ROOT, "profiles", "r2_traffic.json")   # dram__bytes_read+write of one ncu --set full capture
    if os.path.exists(tp):
        with open(tp) as f:
            traffic = json.load(f)["traffic_bytes_per_launch"]
    kern_ms = total_ms / args.steps     # average launch duration over the timed region (launch gaps included): the
    achieved = COORDS * BYTES_PER_COORD / (kern_ms * 1e-3) / 1e9   # steps are back to back, one launch each
    cpu = None
    if world == 1 and not args.no_cpu:
        b = sets[0]
        n_img = IMAGES
        v, dt = cpu_throughput(q.all_code_points.cpu().numpy(), b["mu"][:n_img * H * W].cpu().numpy(),
                               b["sigma"][:n_img * H * W].cpu().numpy(), n_img, 1)
        cpu = {"value": v, "unit": UNIT, "cores": 1, "kind": "port",
               "sample": "%d of the 24 Kodak-shaped images (%d coordinates), one image per call, single process, %.1f s"
                         % (n_img, n_img * H * W * C, dt)}
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "coords_per_step_per_gpu": COORDS, "max_bits_per_coord": N_BITS,
                   "lambdas": [LAMB], "outputs": "sorted quantile index int32 + code length f32 + totals",
                   "l2": "%d rotating input/output sets (%d MB) > 126 MB L2" % (n_sets, n_sets * set_bytes >> 20),
                   "flags": args.flags, "parallelism": "dp%d, totals (n_lambda,4) f64 exchanged once per call (N > 1: peer inboxes over NVLink, written and collected by the search kernel)" % world},
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                     "frac": achieved / peaks["hbm_gbs"], "traffic": traffic, "peak_kind": peak_kind,
                     "kernel": "vbq_bisect_tma_kernel", "kernel_ms": kern_ms,
                     "algorithmic_bytes_per_launch": COORDS * BYTES_PER_COORD},
        "cpu_baseline": cpu,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": 2 * COORDS * 4,
                "d2h_bytes_per_step": 2 * COORDS * 4, "steps": e2e_steps,
                "api": "ChannelwisePriorCDFQuantizer.compress_batch_channel_latents on pinned NumPy arrays (z_hat f32 + "
                       "depth i32 back as NumPy; vbq_quantize_host underneath: 9216-row chunks, 3 streams)",
                "copy_only_ceiling": ceiling, "frac_of_ceiling": e2e_value / ceiling},
        "scaling_variants": variants,
        "gpu_launches": args.steps, "host_issue_us_per_step": host_issue_us,
        "clocks": clocks.summary(),
    }
    line.update(extra)
    print(json.dumps(line))


def bench_corrected(q0, sets, world, dev, barrier, max_over_ranks):
    """Same Kodak batch in the mode every reference call runs in after build_entropy_models (quantizer.py:166-180,
    utils.py:392-396; the path utils.py:542 -> compress -> compress_latents): per-channel corrected code lengths
    n + R_lambda[c, n], z_hat + corrected length + entropy-model bits out.  Entropy models fitted on the batch itself."""
    import torch
    import vbq_b200
    from vbq_b200 import ops
    grid = [float(l) for l in 2.0 ** np.linspace(-8, 7, 16)]
    q = vbq_b200.ChannelwisePriorCDFQuantizer(C, N_BITS, device=dev)
    q.set_code_points(q0.all_code_points)
    b = sets[0]
    logvar = (2.0 * torch.log(b["sigma"])).contiguous()
    q.build_entropy_models_from_latents(b["mu"], logvar, grid, add_n_smoothing=1.0)
    out = {}
    rows = b["mu"].shape[0]
    for name, lambs in (("single_lambda", [LAMB]), ("grid16", grid)):
        # the C-ABI call with caller-owned buffers (ops.QuantizePlan, like the headline): what the kernels take
        L = len(lambs)
        pen, length = q._length_tables(lambs)
        em = q._entropy_model_tensor(lambs)
        z, bl, eb = (torch.empty((L, rows, C), dtype=torch.float32, device=dev) for _ in range(3))
        res = {"lambdas": L, "unit": "coord-lambdas/s",
               "outputs": "z_hat f32 + corrected code length f32 + entropy-model bits f32 + totals"}
        for key, em_, eb_ in (("", em, eb), ("no_entropy_model_bits", None, None)):
            plans = [ops.QuantizePlan(bb["mu"], bb["sigma"], q.all_code_points, q._packed, pen, length, em_, N_BITS, zhat=z,
                                      bits=bl, em_bits=eb_, totals=torch.zeros((L, 4), dtype=torch.float64, device=dev))
                     for bb in sets]
            ms = max_over_ranks(_time_steps(lambda i: plans[i % len(plans)].run(), 20, 3, barrier)) / 20
            r = {"ms_per_call": ms, "value": COORDS * L * world / (ms * 1e-3)}
            if key:
                res[key] = r
            else:
                res.update(r)
            del plans
        # the same through the facade (output allocation and table lookups per call: host-bound for one lambda)

        def fn(i, lambs=lambs):
            bb = sets[i % len(sets)]
            q.quantize(bb["mu"], bb["sigma"], lambs, outputs=ops.OUT_ZHAT | ops.OUT_BITS | ops.OUT_TOTALS, entropy_bits=True)
        del z, bl, eb
        res["facade_ms_per_call"] = max_over_ranks(_time_steps(fn, 10, 3, barrier)) / 10
        out[name] = res
    return out


def bench_configs(prior, q, rank, world, dev, barrier, max_over_ranks):
    """BASELINE.json configs[2..4] at this N, each through vbq_b200.sharding.ShardedQuantizer with ONE all-reduce of the
    totals per call inside the timed region.  Config 3 and 5 run the per-GPU share of the 8-GPU problem (weak scaling:
    512 / 32 images per GPU); config 4 is strong-scaled (1 M rows / N per rank)."""
    import torch
    import vbq_b200
    from vbq_b200 import ops, sharding
    res = {}
    g = torch.Generator(device=dev)
    g.manual_seed(77 + rank)

    # configs[2]: 4096 synthetic 512x768 images (32x48 latents x 192), 64-point lambda sweep, totals only
    imgs = 512
    rows = imgs * H * W
    u = torch.rand((rows, C), generator=g, device=dev, dtype=torch.float64) * 0.998 + 0.001
    mu = prior.inverse_cdf(u).contiguous()
    del u
    sigma = torch.exp(0.5 * (torch.randn((rows, C), generator=g, device=dev) * 1.5 - 3.0)).contiguous()
    sq = sharding.ShardedQuantizer(q)
    lambs = [float(l) for l in 2.0 ** np.linspace(-8, 7, 64)]
    ms = max_over_ranks(_time_steps(lambda i: sq.rd_sweep(mu, sigma, lambs), 3, 2, barrier)) / 3
    res["config3_sweep64"] = {
        "workload": "%d images/GPU x 32x48x192 latents, 64 lambdas 2^linspace(-8,7,64), totals only" % imgs,
        "ms_per_call": ms, "value": rows * C * 64 * world / (ms * 1e-3), "unit": "coord-lambdas/s", "scaling": "weak",
        "hbm_frac_at_8B_per_coord": rows * C * 8 / (ms * 1e-3) / 1e9 / measured_peaks()[0]["hbm_gbs"]}
    del mu, sigma

    # configs[3]: word embeddings 1M x 300, row-sharded (strong scaling): float32 kernel and the default float64 search
    V, K = 1_000_000, 300
    a, b_ = sharding.shard_bounds(V, world, rank)
    means = torch.randn((b_ - a, K), generator=g, device=dev) * 1.2329 - 0.08
    stds = torch.exp(torch.randn((b_ - a, K), generator=g, device=dev) * 0.7 + float(np.log(0.04)))
    cb = vbq_b200.GaussianCodebook(1.2356, 10, device=dev)

    def emb32(i):
        out = cb.quantize(means, stds, [1.0], outputs=ops.OUT_ZHAT | ops.OUT_TOTALS)
        sharding.all_reduce_totals(out["totals"])

    def emb64(i):
        cb.compress_coordinates(means, stds, 1.0, exact=True)

    ms32 = max_over_ranks(_time_steps(emb32, 5, 2, barrier)) / 5
    ms64 = max_over_ranks(_time_steps(emb64, 3, 1, barrier)) / 3
    res["config4_embeddings"] = {
        "workload": "1M x 300 Gaussian posteriors, rows/N per rank, beta = 1, N = 10", "scaling": "strong",
        "float32_kernel": {"ms_per_call": ms32, "value": V * K / (ms32 * 1e-3), "unit": UNIT,
                           "api": "GaussianCodebook.quantize (z_hat + totals, one all-reduce per call)"},
        "float64_default": {"ms_per_call": ms64, "value": V * K / (ms64 * 1e-3), "unit": UNIT,
                            "api": "GaussianCodebook.compress_coordinates(exact=True), the notebook's arithmetic"}}
    del means, stds

    # configs[4]: 256 synthetic 2048x2048 images x 320 channels (128x128 latents), max bit depth 16
    C5, N5, imgs5 = 320, 16, 256 // 8
    rows5 = imgs5 * 128 * 128
    prior5 = vbq_b200.BMSHJ2018Prior(C5, device=dev, seed=5)
    q5 = vbq_b200.ChannelwisePriorCDFQuantizer(C5, N5, device=dev)
    q5.build_code_points(prior5)
    u = torch.rand((rows5, C5), generator=g, device=dev, dtype=torch.float64) * 0.998 + 0.001
    mu5 = prior5.inverse_cdf(u).contiguous()
    del u
    sg5 = torch.exp(0.5 * (torch.randn((rows5, C5), generator=g, device=dev) * 1.5 - 3.0)).contiguous()
    sq5 = sharding.ShardedQuantizer(q5)
    r5 = {"workload": "%d images/GPU x 128x128x320 latents, N = 16, sorted index + code length + totals" % imgs5,
          "scaling": "weak"}
    for name, lamb in (("lambda_0.5", 0.5), ("lambda_2^-8", 2.0 ** -8)):
        ms = max_over_ranks(_time_steps(lambda i: sq5.quantize(mu5, sg5, [lamb], ops.OUT_QIDX | ops.OUT_BITS), 3, 2,
                                        barrier)) / 3
        r5[name] = {"ms_per_call": ms, "value": rows5 * C5 * world / (ms * 1e-3), "unit": UNIT,
                    "roofline_frac": rows5 * C5 * 16 / (ms * 1e-3) / 1e9 / measured_peaks()[0]["hbm_gbs"]}
    res["config5_deep"] = r5
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--flags", type=int, default=0, help="VBQ_FLAG_* bits passed to vbq_quantize")
    ap.add_argument("--chunk-rows", type=int, default=9216, help="rows per chunk of the host pipeline (e2e leg)")
    ap.add_argument("--no-reserve", action="store_true", help="multi-GPU: do not leave an SM to the NCCL kernel")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--headline-only", action="store_true", help="skip the `corrected` and `configs` sections")
    ap.add_argument("--graph", action="store_true", help="replay one CUDA graph per step instead of the prebound eager "
                    "call (the eager launches overlap through programmatic dependent launch and measure faster)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one returned "
                    "(rank 0: qidx, bits as float32 (1, rows, C); totals float64 (1, 4)) as DIR/<name>.npy; the inputs "
                    "are seeded, so two builds run with the same arguments can be compared output for output")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.steps < 1):
        ap.error("--dump-outputs needs --impl ours and --steps >= 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_ours(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
