"""GPU parity tests: the CUDA path (through the C ABI / custom ops) against the CPU oracle.

Protocol (SURVEY.md §8c): (A) kernel code-point table vs oracle table; (B) oracle search run on the
kernel-exported table must match the kernel's z_hat / code length bit for bit; (C) totals; float tolerances are
written next to each assertion."""
import numpy as np
import pytest
import torch

from oracle import vbq_oracle as O
import vbq_test_helpers as H

pytestmark = pytest.mark.gpu

DEV = "cuda"


def _dev(x, dtype=None):
    t = torch.as_tensor(np.ascontiguousarray(x))
    if dtype is not None:
        t = t.to(dtype)
    return t.to(DEV)


def test_division_is_ieee():
    import vbq_b200
    rng = np.random.default_rng(0)
    n = 1 << 22
    a = (rng.standard_normal(n) * np.exp(rng.uniform(-20, 20, n))).astype(np.float32)
    b = np.exp(rng.uniform(-20, 20, n)).astype(np.float32) * rng.choice([-1, 1], n).astype(np.float32)
    out = vbq_b200.ops.selftest_divide(_dev(a), _dev(b)).cpu().numpy()
    assert np.array_equal(out, a / b)


@pytest.mark.parametrize("N,C,fs", [(10, 24, 0.5), (10, 16, 0.0), (12, 5, 0.5)])
def test_learned_table_matches_f64_oracle(N, C, fs):
    import vbq_b200
    pr = H.make_prior(C, seed=11, factor_std=fs)
    params = _dev(pr.packed())
    table = vbq_b200.ops.build_code_points_learned(params, N).cpu().numpy()
    xi = O.xi_heap(N)
    want = pr.inverse_cdf_f64(np.repeat(xi[:, None], C, axis=1)).T
    # correctly rounded float64 root on both sides: at most one float32 ulp apart, almost always identical
    ulp = np.abs(table.view(np.int32).astype(np.int64) - want.view(np.int32).astype(np.int64))
    assert ulp.max() <= 1
    assert (ulp == 0).mean() > 0.999
    # strictly increasing in sorted order => heap order is a binary search tree
    n = np.repeat(np.arange(N + 1), [2 ** k for k in range(N + 1)])
    i = np.concatenate([np.arange(2 ** k) for k in range(N + 1)])
    order = np.argsort(O.heap_to_sorted_rank(n, i, N))
    assert np.all(np.diff(table[:, order], axis=1) > 0)
    # same device routine behind inverse_cdf: bit-identical
    xi_rep = _dev(np.repeat(xi[:, None], C, axis=1))
    z = vbq_b200.ops.learned_inverse_cdf(params, xi_rep).cpu().numpy()
    assert np.array_equal(z.T, table)
    # reference-faithful float32 bisection (learned_prior.py:173-218): 1e-5 of the prior's scale
    ref = pr.inverse_cdf_reference(np.repeat(xi[:, None], C, axis=1)).T
    scale = np.abs(want).max()
    assert np.max(np.abs(ref - table) / np.maximum(np.abs(want), 0.05 * scale)) < 1e-4


def test_learned_cdf_matches_oracle():
    import vbq_b200
    C = 20
    pr = H.make_prior(C, seed=3)
    rng = np.random.default_rng(3)
    x = (rng.standard_normal((1000, C)) * 30).astype(np.float32)
    got = vbq_b200.ops.learned_cdf(_dev(pr.packed()), _dev(x)).cpu().numpy()
    want = pr.cdf(x.astype(np.float64), dtype=np.float64)
    assert np.max(np.abs(got - want)) < 2e-6   # float32 evaluation of a CDF in [0,1]


def test_gaussian_tables_match_scipy():
    import vbq_b200
    N, C = 10, 7
    rng = np.random.default_rng(5)
    mean, std = rng.normal(0, 2, C), np.exp(rng.normal(0, 1, C))
    table = vbq_b200.ops.build_code_points_gaussian(_dev(mean), _dev(std), N).cpu().numpy()
    xi = O.xi_heap(N)
    want64 = O.gaussian_inverse_cdf(np.repeat(xi[:, None], C, axis=1), mean, std)
    z64 = vbq_b200.ops.gaussian_inverse_cdf(_dev(np.repeat(xi[:, None], C, axis=1)), _dev(mean), _dev(std)).cpu().numpy()
    assert np.max(np.abs(z64 - want64) / np.maximum(np.abs(want64), 1e-3)) < 1e-11   # CUDA normcdfinv vs Cephes ndtri, float64
    ulp = np.abs(table.view(np.int32).astype(np.int64) - want64.astype(np.float32).T.view(np.int32).astype(np.int64))
    assert ulp.max() <= 1 and (ulp == 0).mean() > 0.999


def _run_case(N, C, rows, lambs, seed, corrected=False, flags=0, fs=0.5):
    import vbq_b200
    from vbq_b200 import ops
    pr = H.make_prior(C, seed=seed, factor_std=fs)
    table_d = ops.build_code_points_learned(_dev(pr.packed()), N)
    table = table_d.cpu().numpy()
    mu, sigma, _ = H.make_latents(pr, rows, seed + 1, table=table)
    q = vbq_b200.ChannelwisePriorCDFQuantizer(C, N)
    q.set_code_points(table_d)
    oq = O.QuantizerNP(C, N)
    oq.set_code_points(table, build_grids=(N <= 10))
    if corrected:
        rng = np.random.default_rng(seed + 2)
        rcl = {l: (rng.uniform(0.5, 6.0, (C, N + 1))).astype(np.float32) for l in lambs}
        q.raw_code_length_entropy_models = rcl
        oq.raw_code_length_entropy_models = rcl
    out = q.quantize(_dev(mu), _dev(sigma), lambs, flags=flags,
                     outputs=ops.OUT_ZHAT | ops.OUT_QIDX | ops.OUT_LEVEL | ops.OUT_BITS | ops.OUT_TOTALS)
    Zo, Bo, det = oq.compress_batch_channel_latents(mu, sigma, lambs, details=True)
    res = []
    for i, l in enumerate(lambs):
        zk = out["zhat"][i].cpu().numpy()
        bk = out["bits"][i].cpu().numpy()
        lk = out["level"][i].cpu().numpy()
        qk = out["qidx"][i].cpu().numpy()
        res.append(dict(lamb=l, zk=zk, bk=bk, lk=lk, qk=qk, zo=Zo[l], bo=Bo[l], det=det[l],
                        totals=out["totals"][i].cpu().numpy(), mu=mu, sigma=sigma, oq=oq))
    return res


@pytest.mark.parametrize("N,C,rows", [(10, 24, 1000), (10, 16, 64), (10, 5, 333), (4, 33, 257), (1, 3, 40),
                                      (0, 2, 40), (12, 20, 500), (13, 16, 300)])
@pytest.mark.parametrize("flags", [0, 2])
def test_index_parity_raw_lengths(N, C, rows, flags):
    lambs = [2.0 ** -8, 2.0 ** -3, 0.5, 2.0, 128.0]
    for r in _run_case(N, C, rows, lambs, seed=100 + N, flags=flags):
        # (B) bit-exact z_hat and depth against the oracle search on the kernel's own table
        assert np.array_equal(r["zk"], r["zo"]), "lambda=%g" % r["lamb"]
        assert np.array_equal(r["lk"], r["bo"])
        assert np.array_equal(r["bk"], r["bo"].astype(np.float32))
        # sorted index == searchsorted(code_points_by_channel, z_hat)  (quantizer.py:135) and the invariant :136-137
        I = r["oq"].sorted_index(r["zk"])
        assert np.array_equal(r["qk"], I)
        assert np.array_equal(np.take_along_axis(r["oq"].code_points_by_channel.T, I, axis=0), r["zk"])
        # (C) totals: float64 sums of float32 terms, 1e-9 relative
        bits, dist = O.rd_totals(r["mu"], r["sigma"], r["zk"], r["bo"])
        assert r["totals"][0] == bits and r["totals"][1] == bits
        assert abs(r["totals"][3] - dist) <= 1e-6 * max(dist, 1.0)


@pytest.mark.parametrize("N,C,rows", [(10, 24, 700), (6, 17, 300)])
def test_index_parity_corrected_lengths(N, C, rows):
    lambs = [2.0 ** -6, 0.5, 8.0]
    for r in _run_case(N, C, rows, lambs, seed=7, corrected=True):
        assert np.array_equal(r["zk"], r["zo"])
        assert np.array_equal(r["bk"], r["bo"])


def test_fast_mode_differs_only_inside_ties():
    lambs = [2.0 ** -8, 0.5, 8.0]
    tot = out = 0
    for r in _run_case(10, 32, 4000, lambs, seed=21, flags=4):
        n_mis, n_out = H.classify_mismatches(r["det"], r["zk"], r["bk"])
        tot += n_mis
        out += n_out
    print("fast mode: %d mismatches, %d outside the 1e-6 tie band" % (tot, out))
    assert out == 0


def test_prune_equals_no_prune_large():
    a = _run_case(10, 48, 6000, [2.0 ** -8, 0.5, 32.0], seed=33, flags=0)
    b = _run_case(10, 48, 6000, [2.0 ** -8, 0.5, 32.0], seed=33, flags=2)
    for x, y in zip(a, b):
        assert np.array_equal(x["zk"], y["zk"]) and np.array_equal(x["lk"], y["lk"])
        assert np.array_equal(x["zk"], x["zo"])


def test_host_pipeline_matches_device_path():
    """vbq_quantize_host (chunked upload/kernel/download) == vbq_quantize on the same data, incl. ragged last chunk; with
    3 lambdas (penalties also on the host) and with 16 lambdas (more than the pipeline's 64 host penalty floats)."""
    import vbq_b200
    from vbq_b200 import ops
    C, N, rows = 40, 10, 5000
    pr = H.make_prior(C, seed=5)
    q = vbq_b200.ChannelwisePriorCDFQuantizer(C, N)
    q.set_code_points(ops.build_code_points_learned(_dev(pr.packed()), N))
    mu, sigma, _ = H.make_latents(pr, rows, 6, table=q.all_code_points.cpu().numpy())
    for lambs in ([2.0 ** -5, 0.5, 16.0], [float(l) for l in 2.0 ** np.linspace(-8, 6, 16)]):
        _host_pipeline_case(q, C, N, rows, mu, sigma, lambs)


def _host_pipeline_case(q, C, N, rows, mu, sigma, lambs):
    from vbq_b200 import ops
    want = q.quantize(_dev(mu), _dev(sigma), lambs,
                      outputs=ops.OUT_ZHAT | ops.OUT_QIDX | ops.OUT_LEVEL | ops.OUT_BITS | ops.OUT_TOTALS)
    pen, length = q._length_tables(lambs)
    L = len(lambs)
    h = dict(zhat=torch.empty((L, rows, C)).pin_memory(), qidx=torch.empty((L, rows, C), dtype=torch.int32).pin_memory(),
             level=torch.empty((L, rows, C), dtype=torch.int32), bits=torch.empty((L, rows, C)),
             totals=torch.empty((L, 4), dtype=torch.float64))
    pipe = ops.HostPipeline(C, N, L, 768, ops.OUT_ZHAT | ops.OUT_QIDX | ops.OUT_LEVEL | ops.OUT_BITS | ops.OUT_TOTALS)
    pipe.run(torch.from_numpy(mu).pin_memory(), sigma, q.all_code_points, q._packed, pen, length, None, **h)
    pipe.close()
    for k in ("zhat", "qidx", "level", "bits"):
        assert torch.equal(h[k], want[k].cpu()), k
    # chunked accumulation changes the float64 summation order only
    assert torch.allclose(h["totals"], want["totals"].cpu(), rtol=1e-12, atol=0)


@pytest.mark.parametrize("N,C,rows,n_lambda,corrected", [(10, 24, 900, 16, False), (10, 20, 500, 100, True),
                                                         (5, 7, 333, 3, False)])
@pytest.mark.parametrize("fast", [0, 4])
def test_sweep_equals_per_lambda_walks(N, C, rows, n_lambda, corrected, fast):
    """One walk serving all lambdas (sweep kernel, incl. lambda chunking at 100 lambdas) gives exactly the outputs
    of one walk per lambda (VBQ_FLAG_NO_SWEEP); totals agree to 1e-6 (the sweep derives the winner's distortion from
    its float32 score)."""
    import vbq_b200
    from vbq_b200 import ops
    pr = H.make_prior(C, seed=N)
    q = vbq_b200.ChannelwisePriorCDFQuantizer(C, N)
    q.set_code_points(ops.build_code_points_learned(_dev(pr.packed()), N))
    mu, sigma, _ = H.make_latents(pr, rows, 9, table=q.all_code_points.cpu().numpy())
    lambs = [float(l) for l in 2 ** np.linspace(-8, 7, n_lambda)]
    if corrected:
        rng = np.random.default_rng(0)
        q.raw_code_length_entropy_models = {l: rng.uniform(0.5, 6.0, (C, N + 1)).astype(np.float32) for l in lambs}
        q.entropy_models = {l: rng.uniform(0.5, 12.0, (C, q.quantization_levels)).astype(np.float32) for l in lambs}
    outs = ops.OUT_ZHAT | ops.OUT_QIDX | ops.OUT_LEVEL | ops.OUT_BITS | ops.OUT_TOTALS
    a = q.quantize(_dev(mu), _dev(sigma), lambs, outputs=outs, flags=fast, entropy_bits=corrected)
    b = q.quantize(_dev(mu), _dev(sigma), lambs, outputs=outs, flags=fast | ops.FLAG_NO_SWEEP, entropy_bits=corrected)
    for k in ("zhat", "qidx", "level", "bits", "em_bits"):
        assert torch.equal(a[k], b[k]), k
    assert torch.allclose(a["totals"], b["totals"], rtol=1e-6, atol=1e-9)
    # depth sums are integers; raw code lengths too.  Corrected lengths / entropy-model bits are float32 terms that the
    # sweep kernel adds per 64-coordinate tile (units of 2^-16) and the per-lambda kernels per 4 coordinates (2^-24)
    assert torch.equal(a["totals"][:, :1], b["totals"][:, :1])
    if not corrected:
        assert torch.equal(a["totals"][:, :3], b["totals"][:, :3])


def test_strict_mode_equals_reference_walk():
    """Default mode (nearer bracket end + exact tie fallback) vs VBQ_FLAG_REFERENCE_WALK (both ends, two running
    maxima) on 3.1 M coordinates: identical outputs for every lambda."""
    import vbq_b200
    from vbq_b200 import ops
    C, N, rows = 48, 10, 65536
    pr = H.make_prior(C, seed=77)
    q = vbq_b200.ChannelwisePriorCDFQuantizer(C, N)
    q.set_code_points(ops.build_code_points_learned(_dev(pr.packed()), N))
    rng = np.random.default_rng(5)
    srt = q.code_points_by_channel.cpu().numpy()
    idx = rng.integers(0, srt.shape[1], (rows, C))
    mu = (srt[np.arange(C)[None, :], idx] + rng.normal(0, 0.05, (rows, C))).astype(np.float32)
    sigma = np.exp(0.5 * rng.normal(-3, 1.5, (rows, C))).astype(np.float32)
    outs = ops.OUT_ZHAT | ops.OUT_QIDX | ops.OUT_LEVEL
    for lamb in (0.0, 2.0 ** -8, 0.5, 16.0):
        for extra in (0, ops.FLAG_NO_PRUNE):
            a = q.quantize(_dev(mu), _dev(sigma), [lamb], outputs=outs, flags=extra)
            b = q.quantize(_dev(mu), _dev(sigma), [lamb], outputs=outs, flags=extra | ops.FLAG_REFERENCE_WALK)
            for k in ("zhat", "qidx", "level"):
                assert torch.equal(a[k], b[k]), (lamb, extra, k)


@pytest.mark.parametrize("flags", [0, 2, 32])
def test_massive_ties_follow_argmax_order(flags):
    """sigma so large that every distortion term underflows to zero: with lambda = 0 all 2N+1 candidates tie and the
    reference's argmax returns candidate 0 (left_0); with lambda > 0 depth 0 wins outright.  Exercises the tie
    fallback of the default mode."""
    import vbq_b200
    from vbq_b200 import ops
    C, N, rows = 16, 10, 256
    pr = H.make_prior(C, seed=8)
    q = vbq_b200.ChannelwisePriorCDFQuantizer(C, N)
    q.set_code_points(ops.build_code_points_learned(_dev(pr.packed()), N))
    table = q.all_code_points.cpu().numpy()
    mu, _, _ = H.make_latents(pr, rows, 3, table=table)
    sigma = np.full_like(mu, 1e30)
    sigma[::2] = np.float32(3e19)          # t^2 ~ 1e-37: deep in the subnormal range, many equal scores
    oq = O.QuantizerNP(C, N)
    oq.set_code_points(table)
    lambs = [0.0, 1e-30, 0.5]
    Zo, Bo = oq.compress_batch_channel_latents(mu, sigma, lambs)
    for sweep in (ops.FLAG_NO_SWEEP, 0):
        out = q.quantize(_dev(mu), _dev(sigma), lambs, flags=flags | sweep, outputs=ops.OUT_ZHAT | ops.OUT_LEVEL)
        for i, l in enumerate(lambs):
            assert np.array_equal(out["zhat"][i].cpu().numpy(), Zo[l]), (l, sweep)
            assert np.array_equal(out["level"][i].cpu().numpy(), Bo[l]), (l, sweep)


@pytest.mark.parametrize("flags", [0, 4, 32])
def test_garbage_inputs_stay_in_bounds(flags):
    """The reference does not validate inputs (NaNs propagate silently, SURVEY §8b); the kernel must at least terminate
    and keep every index inside its table for NaN / inf / zero / negative posteriors."""
    import vbq_b200
    from vbq_b200 import ops
    C, N, rows = 16, 10, 512
    pr = H.make_prior(C, seed=1)
    q = vbq_b200.ChannelwisePriorCDFQuantizer(C, N)
    q.set_code_points(ops.build_code_points_learned(_dev(pr.packed()), N))
    mu, sigma, _ = H.make_latents(pr, rows, 2)
    bad = [np.nan, np.inf, -np.inf, 0.0, -1.0, 1e-45, 3e38]
    for k, v in enumerate(bad):
        mu[k::32, k % C] = v if k < 3 else mu[k::32, k % C]
        sigma[k::32, (k + 5) % C] = v
    for lambs in ([0.5], [0.0, 0.5, 8.0]):
        out = q.quantize(_dev(mu), _dev(sigma), lambs, flags=flags,
                         outputs=ops.OUT_ZHAT | ops.OUT_QIDX | ops.OUT_LEVEL | ops.OUT_TOTALS)
        torch.cuda.synchronize()
        qi, lv = out["qidx"].cpu().numpy(), out["level"].cpu().numpy()
        assert qi.min() >= 0 and qi.max() < q.quantization_levels
        assert lv.min() >= 0 and lv.max() <= N
        srt = q.code_points_by_channel.cpu().numpy()
        for i in range(len(lambs)):
            assert np.array_equal(np.take_along_axis(srt.T, qi[i].astype(np.int64), axis=0), out["zhat"][i].cpu().numpy())


@pytest.mark.parametrize("N,C,rows", [(10, 48, 20000), (10, 5, 777), (6, 17, 3000), (4, 33, 257), (1, 3, 40), (0, 2, 40),
                                      (12, 20, 3000), (16, 16, 2000), (11, 7, 501)])
def test_bisection_equals_reference_walk(N, C, rows):
    """The default single-lambda kernel (certified bisection: one path node per depth, approximate ranking with a
    guard band, literal search for uncertified coordinates) vs VBQ_FLAG_REFERENCE_WALK and the round-1 bracket walk
    (VBQ_FLAG_BRACKET_WALK): identical outputs for every lambda, prune on and off; totals within 1e-6."""
    import vbq_b200
    from vbq_b200 import ops
    pr = H.make_prior(C, seed=300 + N)
    q = vbq_b200.ChannelwisePriorCDFQuantizer(C, N)
    q.set_code_points(ops.build_code_points_learned(_dev(pr.packed()), N))
    table = q.all_code_points.cpu().numpy()
    mu, sigma, _ = H.make_latents(pr, rows, 41 + N, table=table)
    rng = np.random.default_rng(9)
    # a third of the coordinates sit within a few ulps of code points / of bracket midpoints: near-ties in bulk
    srt = q.code_points_by_channel.cpu().numpy()
    idx = rng.integers(0, srt.shape[1], (rows, C))
    on = srt[np.arange(C)[None, :], idx]
    nxt = srt[np.arange(C)[None, :], np.minimum(idx + 1, srt.shape[1] - 1)]
    pick = rng.integers(0, 6, (rows, C))
    mu = np.where(pick == 0, on, np.where(pick == 1, (0.5 * (on.astype(np.float64) + nxt)).astype(np.float32), mu))
    mu = mu.astype(np.float32)
    outs = ops.OUT_ZHAT | ops.OUT_QIDX | ops.OUT_LEVEL | ops.OUT_BITS | ops.OUT_TOTALS
    for lamb in (0.0, 1e-30, 2.0 ** -8, 0.1, 0.5, 3.0, 16.0, 1e4):
        for extra in (0, ops.FLAG_NO_PRUNE):
            a = q.quantize(_dev(mu), _dev(sigma), [lamb], outputs=outs, flags=extra)
            b = q.quantize(_dev(mu), _dev(sigma), [lamb], outputs=outs, flags=extra | ops.FLAG_REFERENCE_WALK)
            c = q.quantize(_dev(mu), _dev(sigma), [lamb], outputs=outs, flags=extra | ops.FLAG_BRACKET_WALK)
            for k in ("zhat", "qidx", "level", "bits"):
                assert torch.equal(a[k], b[k]), (lamb, extra, k)
                assert torch.equal(a[k], c[k]), (lamb, extra, k)
            assert torch.equal(a["totals"][:, :2], b["totals"][:, :2])
            assert torch.allclose(a["totals"][:, 3], b["totals"][:, 3], rtol=1e-6, atol=1e-9)


def test_bisection_rejects_non_monotone_penalties():
    """Penalties that are not non-decreasing in depth void the one-candidate-per-depth argument; the kernel detects
    them while staging and sends every coordinate through the literal search.  Checked through the raw C ABI with a
    decreasing penalty table against VBQ_FLAG_REFERENCE_WALK."""
    import vbq_b200
    from vbq_b200 import ops
    C, N, rows = 16, 10, 4096
    pr = H.make_prior(C, seed=12)
    q = vbq_b200.ChannelwisePriorCDFQuantizer(C, N)
    q.set_code_points(ops.build_code_points_learned(_dev(pr.packed()), N))
    mu, sigma, _ = H.make_latents(pr, rows, 13, table=q.all_code_points.cpu().numpy())
    rng = np.random.default_rng(2)
    pen = _dev(rng.uniform(0.0, 3.0, (1, 1, N + 1)).astype(np.float32))
    res = []
    for fl in (ops.FLAG_NO_PRUNE, ops.FLAG_NO_PRUNE | ops.FLAG_REFERENCE_WALK, 0):
        z = torch.empty((1, rows, C), dtype=torch.float32, device="cuda")
        lv = torch.empty((1, rows, C), dtype=torch.int32, device="cuda")
        ops.quantize_into(_dev(mu), _dev(sigma), q.all_code_points, q._packed, pen, None, None, N, zhat=z, level=lv,
                          flags=fl)
        res.append((z, lv))
    for z, lv in res[1:]:
        assert torch.equal(z, res[0][0]) and torch.equal(lv, res[0][1])


@pytest.mark.parametrize("N,C,rows,n_lambda", [(10, 48, 9000, 16), (10, 21, 1001, 130), (7, 16, 640, 5), (0, 3, 50, 2)])
def test_bisection_sweep_equals_bracket_walk_sweep(N, C, rows, n_lambda):
    """All lambdas from one certified-bisection walk (vbq_bisect_sweep_kernel, the default for raw code lengths) vs the
    round-1 sweep kernel (VBQ_FLAG_BRACKET_WALK: both bracket ends, IEEE scores, two running maxima) and vs one walk
    per lambda: identical outputs incl. lambda = 0, the chunking beyond 100 lambdas, ragged C; totals within 1e-6."""
    import vbq_b200
    from vbq_b200 import ops
    pr = H.make_prior(C, seed=50 + N)
    q = vbq_b200.ChannelwisePriorCDFQuantizer(C, N)
    q.set_code_points(ops.build_code_points_learned(_dev(pr.packed()), N))
    table = q.all_code_points.cpu().numpy()
    mu, sigma, _ = H.make_latents(pr, rows, 77, table=table)
    srt = q.code_points_by_channel.cpu().numpy()
    rng = np.random.default_rng(3)
    idx = rng.integers(0, srt.shape[1], (rows, C))
    on = srt[np.arange(C)[None, :], idx]
    mu = np.where(rng.integers(0, 5, (rows, C)) == 0, on, mu).astype(np.float32)   # exact hits: ties at lambda = 0
    lambs = [0.0] + [float(l) for l in 2 ** np.linspace(-8, 7, n_lambda - 1)]
    outs = ops.OUT_ZHAT | ops.OUT_QIDX | ops.OUT_LEVEL | ops.OUT_BITS | ops.OUT_TOTALS
    a = q.quantize(_dev(mu), _dev(sigma), lambs, outputs=outs)
    b = q.quantize(_dev(mu), _dev(sigma), lambs, outputs=outs, flags=ops.FLAG_BRACKET_WALK)
    c = q.quantize(_dev(mu), _dev(sigma), lambs, outputs=outs, flags=ops.FLAG_NO_SWEEP | ops.FLAG_REFERENCE_WALK)
    for k in ("zhat", "qidx", "level", "bits"):
        assert torch.equal(a[k], b[k]), k
        assert torch.equal(a[k], c[k]), k
    assert torch.equal(a["totals"][:, :3], b["totals"][:, :3])
    assert torch.allclose(a["totals"][:, 3], b["totals"][:, 3], rtol=1e-6, atol=1e-9)
    t = q.quantize(_dev(mu), _dev(sigma), lambs, outputs=ops.OUT_TOTALS)["totals"]     # totals-only path
    assert torch.allclose(t, a["totals"], rtol=1e-12, atol=0)


@pytest.mark.parametrize("N,C,rows,n_lambda", [(10, 48, 6000, 16), (10, 21, 1001, 1), (7, 16, 640, 60), (3, 5, 333, 4)])
@pytest.mark.parametrize("neg", [False, True])
def test_corrected_lengths_sweep_equals_reference_walk(N, C, rows, n_lambda, neg):
    """Corrected code lengths (per-channel, not monotone in depth) and the entropy-model gather: the default kernels
    (bracket-walk sweep, strict single-lambda kernel) vs one literal two-maxima walk per lambda
    (VBQ_FLAG_NO_SWEEP | VBQ_FLAG_REFERENCE_WALK): identical outputs, one lambda included, with bulk exact hits on code
    points, lambda = 0, ragged C, and (neg) negative corrections, i.e. negative penalties."""
    import vbq_b200
    from vbq_b200 import ops
    pr = H.make_prior(C, seed=70 + N)
    q = vbq_b200.ChannelwisePriorCDFQuantizer(C, N)
    q.set_code_points(ops.build_code_points_learned(_dev(pr.packed()), N))
    table = q.all_code_points.cpu().numpy()
    mu, sigma, _ = H.make_latents(pr, rows, 78, table=table)
    srt = q.code_points_by_channel.cpu().numpy()
    rng = np.random.default_rng(4)
    idx = rng.integers(0, srt.shape[1], (rows, C))
    on = srt[np.arange(C)[None, :], idx]
    mu = np.where(rng.integers(0, 5, (rows, C)) == 0, on, mu).astype(np.float32)
    lambs = ([0.0] if n_lambda > 1 else []) + [float(l) for l in 2 ** np.linspace(-8, 7, max(n_lambda - 1, 1))]
    lo = -3.0 if neg else 0.25
    q.raw_code_length_entropy_models = {l: rng.uniform(lo, 6.0, (C, N + 1)).astype(np.float32) for l in lambs}
    q.entropy_models = {l: rng.uniform(0.5, 12.0, (C, q.quantization_levels)).astype(np.float32) for l in lambs}
    outs = ops.OUT_ZHAT | ops.OUT_QIDX | ops.OUT_LEVEL | ops.OUT_BITS | ops.OUT_TOTALS
    a = q.quantize(_dev(mu), _dev(sigma), lambs, outputs=outs, entropy_bits=True)
    b = q.quantize(_dev(mu), _dev(sigma), lambs, outputs=outs, entropy_bits=True,
                   flags=ops.FLAG_NO_SWEEP | ops.FLAG_REFERENCE_WALK)
    for k in ("zhat", "qidx", "level", "bits", "em_bits"):
        assert torch.equal(a[k], b[k]), k
    assert torch.equal(a["totals"][:, 0], b["totals"][:, 0])
    assert torch.allclose(a["totals"], b["totals"], rtol=1e-6, atol=1e-6)


@pytest.mark.parametrize("graph", [False, True])
def test_quantize_plan_repeats_the_call(graph):
    """ops.QuantizePlan (validated once, prebound C call or CUDA-graph replay, zeroed-workspace flag, programmatic
    dependent launch between back-to-back runs) returns exactly what the one-shot op returns, run after run."""
    import vbq_b200
    from vbq_b200 import ops
    C, N, rows = 32, 10, 4100
    pr = H.make_prior(C, seed=91)
    q = vbq_b200.ChannelwisePriorCDFQuantizer(C, N)
    q.set_code_points(ops.build_code_points_learned(_dev(pr.packed()), N))
    mu, sigma, _ = H.make_latents(pr, rows, 92, table=q.all_code_points.cpu().numpy())
    mu_d, sg_d = _dev(mu), _dev(sigma)
    for lambs in ([0.5], [2.0 ** -6, 0.5, 8.0]):
        want = q.quantize(mu_d, sg_d, lambs, outputs=ops.OUT_QIDX | ops.OUT_BITS | ops.OUT_TOTALS)
        pen, length = q._length_tables(lambs)
        L = len(lambs)
        qidx = torch.empty((L, rows, C), dtype=torch.int32, device="cuda")
        bits = torch.empty((L, rows, C), dtype=torch.float32, device="cuda")
        totals = torch.zeros((L, 4), dtype=torch.float64, device="cuda")
        plan = ops.QuantizePlan(mu_d, sg_d, q.all_code_points, q._packed, pen, length, None, N, qidx=qidx, bits=bits,
                                totals=totals, flags=ops.search_flags(lambs), graph=graph)
        for _ in range(5):
            qidx.fill_(-1)
            t = plan.run()
            plan.run()                      # back to back: the second launch overlaps the first one's tail
        torch.cuda.synchronize()
        assert torch.equal(qidx, want["qidx"]) and torch.equal(bits, want["bits"])
        assert torch.equal(t, want["totals"])
