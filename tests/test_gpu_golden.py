"""GPU tests against the golden vectors produced by the unmodified reference (tests/golden/gen_golden.py).

The kernel is given the REFERENCE's code-point table, so z_hat / code lengths must equal the reference's outputs
bit for bit; the kernel's own table is compared with the reference's separately (tolerance stated below)."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
LEARNED = ["learned_c6_n10", "learned_c20_n6_gated"]


def load(name):
    return np.load(os.path.join(G, name + ".npz"))


def lambs_of(g):
    return [float(l) for l in g["lambs"]]


def make_quantizer(g):
    import vbq_b200
    q = vbq_b200.ChannelwisePriorCDFQuantizer(int(g["C"]), int(g["N"]))
    q.set_code_points(g["table"])
    return q


def make_prior(g):
    import vbq_b200
    p = vbq_b200.BMSHJ2018Prior(int(g["C"]))
    p.set_transformed_parameters([g["matrix%d" % k] for k in range(4)], [g["bias%d" % k] for k in range(4)],
                                 [g["factor%d" % k] for k in range(3)])
    return p


@pytest.mark.parametrize("name", LEARNED)
def test_prior_against_reference(name):
    g = load(name)
    prior = make_prior(g)
    cdf = prior.cdf(g["cdf_in"]).cpu().numpy()
    assert np.max(np.abs(cdf - g["cdf_out"])) < 1e-6            # float32 CDF values in [0,1], different libm
    import vbq_b200
    q = vbq_b200.ChannelwisePriorCDFQuantizer(int(g["C"]), int(g["N"]))
    q.build_code_points(prior)
    table = q.all_code_points.cpu().numpy()
    # reconstructed values within 1e-5 relative (north_star), measured against the prior's range because code
    # points near z=0 make a pure relative test meaningless (SURVEY §7.3-2); the reference's float32 bisection on
    # sigmoid(.)-xi carries up to ~1.6e-5 of its own noise in the upper tail at N=10
    rng_ = np.abs(g["table"]).max()
    assert np.max(np.abs(table - g["table"])) < 2e-5 * rng_
    assert np.median(np.abs(table - g["table"]) / np.maximum(np.abs(g["table"]), 1e-2 * rng_)) < 2e-7
    assert np.array_equal(q.code_points_by_channel.cpu().numpy(), np.sort(table, axis=1))
    # generic route (reference quantizer.py:30-36: prior_model.inverse_cdf(xi_rep)) gives the same table
    q2 = vbq_b200.ChannelwisePriorCDFQuantizer(int(g["C"]), int(g["N"]))
    q2.build_code_points(prior, return_np=True)
    assert np.array_equal(q2.all_code_points.cpu().numpy(), table)


@pytest.mark.parametrize("name", LEARNED)
def test_search_equals_reference(name):
    g = load(name)
    q = make_quantizer(g)
    lambs = lambs_of(g)
    C = int(g["C"])
    means, stds = g["means"].reshape(-1, C), g["stds"]
    Zh, nb = q.compress_batch_channel_latents(means, stds, lambs)
    for i, l in enumerate(lambs):
        assert isinstance(Zh[l], np.ndarray) and nb[l].dtype == np.int32
        assert np.array_equal(Zh[l], g["raw_zhat_%d" % i]), "raw z_hat, lambda=%g" % l
        assert np.array_equal(nb[l], g["raw_bits_%d" % i]), "raw bits, lambda=%g" % l
    # corrected code lengths n + R_lambda[c, n] with the REFERENCE's fitted tables
    q.raw_code_length_entropy_models = {l: g["rcl_%d" % i] for i, l in enumerate(lambs)}
    q.entropy_models = {l: g["em_%d" % i] for i, l in enumerate(lambs)}
    Zh, nb = q.compress_batch_channel_latents(torch.from_numpy(means), torch.from_numpy(stds), lambs, return_np=False)
    for i, l in enumerate(lambs):
        assert Zh[l].is_cuda and nb[l].dtype == torch.float32
        assert np.array_equal(Zh[l].cpu().numpy(), g["cl_zhat_%d" % i])
        assert np.array_equal(nb[l].cpu().numpy(), g["cl_bits_%d" % i])


@pytest.mark.parametrize("name", LEARNED)
def test_entropy_model_fit_and_compress_latents(name):
    """build_entropy_models / compress_latents / compress take log-variances; sigma = sqrt(exp(logvar)) is computed
    inside the kernels (sigma_of_logvar), whose CUDA expf may differ from NumPy's exp by an ulp.  Given the kernels' own
    sigma (ops.selftest_sigma_from_logvar), the oracle reproduces the fitted tables and every output bit for bit; against
    the reference's golden vectors a coordinate may differ only where the kernels' sigma differs from NumPy's."""
    from oracle import vbq_oracle as O
    from vbq_b200 import ops
    g = load(name)
    q = make_quantizer(g)
    lambs = lambs_of(g)
    C = int(g["C"])
    stds_np = np.exp(g["logvars"].astype(np.float32)) ** np.float32(0.5)
    stds_k = ops.selftest_sigma_from_logvar(torch.from_numpy(g["logvars"].astype(np.float32)).cuda()).cpu().numpy()
    sigma_moved = stds_k != stds_np                          # coordinates whose sigma is not the reference's
    oq = O.QuantizerNP(C, int(g["N"]))
    oq.set_code_points(g["table"])

    class VAE:
        def encode(self, X):
            return torch.from_numpy(g["means"]).cuda(), torch.from_numpy(g["logvars"]).cuda()

        def decode(self, z):
            m = 0.5 + 0.01 * z.mean(dim=-1, keepdim=True)
            return m.repeat_interleave(16, 1).repeat_interleave(16, 2).repeat_interleave(3, 3)

    X = np.zeros((g["means"].shape[0], 16 * g["means"].shape[1], 16 * g["means"].shape[2], 3), dtype=np.float32)
    q.build_entropy_models(X, VAE(), lambs, add_n_smoothing=1)
    assert q.lambs == sorted(lambs)
    oq.build_entropy_models_from_latents(g["means"], None, lambs, 1, posterior_stds=stds_k)
    for i, l in enumerate(lambs):
        assert q.raw_code_length_entropy_models[l].dtype == np.float32
        assert np.array_equal(q.raw_code_length_entropy_models[l], oq.raw_code_length_entropy_models[l])
        assert np.array_equal(q.entropy_models[l], oq.entropy_models[l])
        if not sigma_moved.any():
            assert np.array_equal(q.raw_code_length_entropy_models[l], g["rcl_%d" % i])
            assert np.array_equal(q.entropy_models[l], g["em_%d" % i])
    # fed the reference's own float32 sigma = exp(logvar) ** 0.5 (quantizer.py:93) the tables are the reference's, bit for bit
    q_s = make_quantizer(g)
    q_s.build_entropy_models_from_latents(g["means"], None, lambs, add_n_smoothing=1, posterior_stds=stds_np)
    for i, l in enumerate(lambs):
        assert np.array_equal(q_s.raw_code_length_entropy_models[l], g["rcl_%d" % i])
        assert np.array_equal(q_s.entropy_models[l], g["em_%d" % i])
    # with the reference's fitted tables installed, compress() must reproduce the oracle on the kernels' sigma exactly,
    # and the reference's outputs wherever the kernels' sigma is the reference's
    q.raw_code_length_entropy_models = {l: g["rcl_%d" % i] for i, l in enumerate(lambs)}
    q.entropy_models = {l: g["em_%d" % i] for i, l in enumerate(lambs)}
    oq.raw_code_length_entropy_models = dict(q.raw_code_length_entropy_models)
    oq.entropy_models = dict(q.entropy_models)
    want = oq.compress_latents(g["means"], None, lambs, posterior_stds=stds_k)
    out = q.compress(X, VAE(), lambs, clip=True)
    assert set(out) == {"Z_hat", "raw_num_bits", "num_bits_cl", "num_bits", "X_hat"}
    mism = 0
    for i, l in enumerate(lambs):
        assert out["Z_hat"][l].shape == g["compress_Z_hat_%d" % i].shape and out["Z_hat"][l].dtype == np.float32
        for key in ("Z_hat", "raw_num_bits", "num_bits_cl", "num_bits"):
            assert np.array_equal(out[key][l], want[key][l]), key
        same = out["Z_hat"][l] == g["compress_Z_hat_%d" % i]
        assert not (~same & ~sigma_moved).any(), "z_hat differs from the reference where sigma does not"
        mism += int((~same).sum())
        for key in ("raw_num_bits", "num_bits_cl", "num_bits"):
            assert np.array_equal(out[key][l][same], g["compress_%s_%d" % (key, i)][same]), key
        assert out["X_hat"][l].shape == X.shape
        # reconstructions within 1e-5 (decode is linear in z_hat)
        if mism == 0:
            assert np.allclose(out["X_hat"][l], g["compress_X_hat_%d" % i], rtol=1e-5, atol=1e-6)
    print("compress_latents: %d coordinates differ from the reference; %d of %d sigmas differ from NumPy's"
          % (mism, int(sigma_moved.sum()), sigma_moved.size))


def test_embedding_path_against_notebook():
    import vbq_b200
    g = load("notebook_embeddings")
    cb = vbq_b200.GaussianCodebook(float(g["empirical_std"]), 10)
    # norm.ppf on the device in float64 vs SciPy
    assert np.max(np.abs(cb.codepoints - g["codepoints"]) / np.abs(g["codepoints"]).clip(1e-3)) < 1e-11
    assert np.array_equal(cb.lengths, g["lengths"])
    cb.codepoints = g["codepoints"].copy()      # same table on both sides for the search test below
    tot = mism = 0
    for i, beta in enumerate(g["betas"]):
        want = g["optima_%d" % i]
        # float64 kernel: the notebook's arithmetic, bit for bit
        optima, none = cb.compress_coordinates(g["means"], g["stds"], float(beta))
        assert none is None and optima.dtype == np.float32 and optima.shape == g["means"].shape
        assert np.array_equal(optima, want), "beta=%g: %d differ" % (beta, (optima != want).sum())
        # float32 image-path kernel on the same problem: only near-ties may differ
        fast, _ = cb.compress_coordinates(g["means"], g["stds"], float(beta), exact=False)
        bad = fast != want
        if bad.any():
            m, s = g["means"][bad].astype(np.float64), g["stds"][bad].astype(np.float64)
            pen = lambda z: np.array([g["lengths"][np.argmin(np.abs(g["codepoints"] - v))] for v in z])  # noqa: E731
            loss = lambda z: (z - m) ** 2 + 2 * float(beta) * s ** 2 * pen(z)                            # noqa: E731
            la, lb = loss(fast[bad].astype(np.float64)), loss(want[bad].astype(np.float64))
            assert np.all(np.abs(la - lb) <= 1e-5 * np.abs(lb) + 1e-12)
        tot += bad.size
        mism += int(bad.sum())
    print("embeddings, float32 kernel: %d of %d optima differ from the float64 notebook search (near-ties)" % (mism, tot))
    assert mism <= tot // 20000 + 3


def test_empirical_entropy_matches_notebook():
    from vbq_b200.word_embeddings import empirical_entropy
    from oracle import vbq_oracle as O
    g = load("notebook_embeddings")
    for i in range(3):
        v = g["optima_%d" % i]
        want = O.empirical_entropy(v)
        assert abs(empirical_entropy(torch.from_numpy(v).cuda()) - want) <= 1e-9 * max(want, 1.0)
        assert abs(empirical_entropy(v) - want) <= 1e-9 * max(want, 1.0)


def test_embedding_f64_kernel_vs_oracle_large():
    """1.5 M coordinates (SURVEY §8d C1 statistics at half size): float64 kernel == exhaustive notebook restatement."""
    import vbq_b200
    from oracle import vbq_oracle as O
    rng = np.random.default_rng(11)
    means = rng.normal(-0.08, 1.2329, (15000, 100)).astype(np.float32)
    stds = np.exp(rng.normal(np.log(0.04), 0.7, means.shape)).astype(np.float32)
    cb = vbq_b200.GaussianCodebook(vbq_b200.word_embeddings.empirical_std(means), 10)
    for beta in (1.0, np.float64(37.5)):
        got, _ = cb.compress_coordinates(means, stds, beta)
        want, _ = O.compress_coordinates_bracket(means, stds, beta, cb.codepoints, 10,
                                                 pen_f64=isinstance(beta, np.floating))
        assert np.array_equal(got, want)


@pytest.mark.parametrize("name", LEARNED)
def test_intervals_equal_reference(name):
    g = load(name)
    q = make_quantizer(g)
    left, right = q.get_all_N_bit_intervals(g["means"].reshape(-1, int(g["C"])))
    assert np.array_equal(left.cpu().numpy(), g["left"]) and np.array_equal(right.cpu().numpy(), g["right"])


def test_generic_operator_equals_reference():
    """utils.batch_quantize_indep_dims (3-D candidates, int32 lengths, Gaussian fun) vs the reference's NumPy run."""
    from vbq_b200 import utils
    g = load("utils_numpy")
    lambs = [float(l) for l in g["bq_lambs"]]
    B, K = g["bq_loc"].shape
    fun = utils.curry_normal_logpdf(loc=g["bq_loc"], scale=g["bq_scale"], ignore_const=True)
    Zh, nb = utils.batch_quantize_indep_dims((B, K), g["bq_P"], g["bq_L"], fun, lambs)
    for i, l in enumerate(lambs):
        assert np.array_equal(Zh[l], g["bq_zhat_%d" % i])
        assert nb[l].dtype == np.int32 and np.array_equal(nb[l], g["bq_bits_%d" % i])
    # arbitrary callable `fun` (evaluated by the caller on device tensors) + 2-D (K, M) candidates
    P2 = np.sort(np.random.default_rng(0).normal(0, 2, (K, 7)).astype(np.float32), axis=1)
    L2 = np.tile(np.arange(7, dtype=np.int32), (K, 1))
    loc = torch.from_numpy(g["bq_loc"]).cuda()
    Zh2, nb2 = utils.batch_quantize_indep_dims((B, K), P2, L2, lambda z: -torch.abs(z - loc), [0.3])
    Pb = np.repeat(P2.T[:, None, :], B, axis=1)
    Lb = np.repeat(L2.T[:, None, :], B, axis=1)
    s = -np.abs(Pb - g["bq_loc"]) - np.float32(0.3) * Lb.astype(np.float32)
    k = np.argmax(s, axis=0)
    assert np.array_equal(Zh2[0.3], np.take_along_axis(Pb, k[None], 0)[0])
    assert np.array_equal(nb2[0.3], np.take_along_axis(Lb, k[None], 0)[0])


def test_batched_evaluation_driver_equals_per_image_loop():
    """evaluate_compression_quantizer (all images x all lambdas in one launch) reproduces the reference's per-image
    loop (utils.py:535-553) run through `compress`: B, BPP, BPL, BPPCL."""
    import vbq_b200
    g = load("learned_c6_n10")
    q = make_quantizer(g)
    lambs = lambs_of(g)
    q.raw_code_length_entropy_models = {l: g["rcl_%d" % i] for i, l in enumerate(lambs)}
    q.entropy_models = {l: g["em_%d" % i] for i, l in enumerate(lambs)}
    means, logvars = torch.from_numpy(g["means"]).cuda(), torch.from_numpy(g["logvars"]).cuda()
    Nimg, Hl, Wl, C = means.shape

    class VAE:
        def __init__(self, sl=None):
            self.sl = sl

        def encode(self, X):
            return (means, logvars) if self.sl is None else (means[self.sl], logvars[self.sl])

        def decode(self, z):
            m = 0.5 + 0.01 * z.mean(dim=-1, keepdim=True)
            return m.repeat_interleave(16, 1).repeat_interleave(16, 2).repeat_interleave(3, 3)

    X = np.zeros((Nimg, 16 * Hl, 16 * Wl, 3), dtype=np.float32)
    res = vbq_b200.evaluate_compression_quantizer(q, VAE(), X, lambs, return_reconstructions=True)
    assert res["B"].shape == (Nimg, len(lambs)) and res["reconstructions"].shape == (len(lambs),) + X.shape
    npix = X.shape[1] * X.shape[2]
    for n in range(Nimg):
        tmp = q.compress(X[n:n + 1], VAE(slice(n, n + 1)), lambs, clip=True)
        for m, l in enumerate(lambs):
            nb = tmp["num_bits"][l][0]
            assert np.isclose(res["B"][n, m], np.sum(nb, dtype=np.float64), rtol=1e-6)
            assert np.isclose(res["BPP"][n, m], np.sum(nb, dtype=np.float64) / npix, rtol=1e-6)
            assert np.isclose(res["BPL"][n, m], np.sum(nb, dtype=np.float64) / nb.size, rtol=1e-6)
            assert np.isclose(res["BPPCL"][n, m], np.sum(tmp["num_bits_cl"][l][0], dtype=np.float64) / npix, rtol=1e-6)
            assert np.allclose(res["reconstructions"][m, n], tmp["X_hat"][l][0], atol=1e-6)
