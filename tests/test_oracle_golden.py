"""CPU tests: the oracle (oracle/vbq_oracle.py) against the golden vectors produced by the UNMODIFIED reference
(tests/golden/gen_golden.py).  This is what pins the oracle (SURVEY.md §8c): every array below was computed by the
reference's own code, and the oracle must reproduce it bit for bit unless a tolerance is stated."""
import os

import numpy as np
import pytest

from oracle import vbq_oracle as O

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
LEARNED = ["learned_c6_n10", "learned_c20_n6_gated"]


def load(name):
    return np.load(os.path.join(G, name + ".npz"))


def prior_of(g):
    return O.LearnedPriorNP([g["matrix%d" % k] for k in range(4)], [g["bias%d" % k] for k in range(4)],
                            [g["factor%d" % k] for k in range(3)])


def quantizer_of(g):
    q = O.QuantizerNP(int(g["C"]), int(g["N"]))
    q.set_code_points(g["table"])
    return q


def lambs_of(g):
    return [float(l) for l in g["lambs"]]


def test_docstring_known_answers():
    g = load("utils_numpy")
    assert list(g["kat_interval"]) == [0.375, 0.625]                   # utils.py:31-32
    assert O.get_n_bit_interval(0.4375, 2) == [0.375, 0.625]
    assert np.array_equal(g["bin_floats_3"], np.array(O.n_bit_binary_floats(3)))
    for k, x in enumerate(g["xi_x"]):
        for n in range(g["xi_left"].shape[0]):
            assert O.get_n_bit_interval(x, n) == [g["xi_left"][n, k], g["xi_right"][n, k]]


@pytest.mark.parametrize("name", LEARNED)
def test_prior_cdf_and_reference_bisection(name):
    g = load(name)
    pr = prior_of(g)
    assert np.array_equal(pr.cdf(g["cdf_in"]), g["cdf_out"])
    C, N = int(g["C"]), int(g["N"])
    xi_rep = np.repeat(O.xi_heap(N)[:, None], C, axis=1)
    assert np.array_equal(pr.inverse_cdf_reference(xi_rep).T, g["table"])       # learned_prior.py:173-218
    # the float64 logit-space root (the table oracle of the CUDA build) agrees with the reference's float32
    # bisection to 2e-5 of the prior's range; the residue is the reference's own upper-tail noise (SURVEY §7.3-2)
    f64 = pr.inverse_cdf_f64(xi_rep).T
    assert np.max(np.abs(f64 - g["table"])) < 2e-5 * np.abs(g["table"]).max()
    assert np.array_equal(np.sort(g["table"], axis=1), g["sorted_table"])


@pytest.mark.parametrize("name", LEARNED)
def test_brackets(name):
    g = load(name)
    q = quantizer_of(g)
    means = g["means"].reshape(-1, int(g["C"]))
    for fn in (q.get_all_N_bit_intervals, q.get_all_N_bit_intervals_fast):
        left, right = fn(means)
        assert np.array_equal(left, g["left"]) and np.array_equal(right, g["right"])


@pytest.mark.parametrize("name", LEARNED)
def test_search_raw_and_corrected_lengths(name):
    g = load(name)
    q = quantizer_of(g)
    lambs = lambs_of(g)
    C = int(g["C"])
    means, stds = g["means"].reshape(-1, C), g["stds"]
    for fast in (False, True):
        Zh, nb = q.compress_batch_channel_latents(means, stds, lambs, fast_intervals=fast)
        for i, l in enumerate(lambs):
            assert np.array_equal(Zh[l], g["raw_zhat_%d" % i])
            assert np.array_equal(nb[l], g["raw_bits_%d" % i]) and nb[l].dtype == np.int32
    q.build_entropy_models_from_latents(g["means"], g["logvars"], lambs, add_n_smoothing=1)
    for i, l in enumerate(lambs):
        assert np.array_equal(q.raw_code_length_entropy_models[l], g["rcl_%d" % i])
        assert np.array_equal(q.entropy_models[l], g["em_%d" % i])
    Zh, nb = q.compress_batch_channel_latents(means, stds, lambs)
    out = q.compress_latents(g["means"], g["logvars"], lambs)
    for i, l in enumerate(lambs):
        assert np.array_equal(Zh[l], g["cl_zhat_%d" % i])
        assert np.array_equal(nb[l], g["cl_bits_%d" % i]) and nb[l].dtype == np.float32
        for key in ("Z_hat", "raw_num_bits", "num_bits_cl", "num_bits"):
            want = g["compress_%s_%d" % (key, i)]
            assert out[key][l].shape == want.shape and np.array_equal(out[key][l], want), key
        # invariant quantizer.py:136-137: every z_hat is exactly a table entry
        I = q.sorted_index(Zh[l])
        assert np.array_equal(np.take_along_axis(q.code_points_by_channel.T, I, axis=0), Zh[l])


@pytest.mark.parametrize("name", LEARNED)
def test_posterior_stds_replace_logvars(name):
    """posterior_stds= hands the oracle a sigma directly (the GPU tests pass it the kernels' sigma of the log-variances):
    given the reference's own exp(logvar) ** 0.5 it reproduces the reference bit for bit without the log-variances, and
    any other sigma is searched as given."""
    g = load(name)
    lambs = lambs_of(g)
    C = int(g["C"])
    stds = np.exp(g["logvars"].astype(np.float32)) ** np.float32(0.5)
    q = quantizer_of(g)
    q.build_entropy_models_from_latents(g["means"], None, lambs, add_n_smoothing=1, posterior_stds=stds)
    for i, l in enumerate(lambs):
        assert np.array_equal(q.raw_code_length_entropy_models[l], g["rcl_%d" % i])
        assert np.array_equal(q.entropy_models[l], g["em_%d" % i])
    out = q.compress_latents(g["means"], None, lambs, posterior_stds=stds)
    for i, l in enumerate(lambs):
        for key in ("Z_hat", "raw_num_bits", "num_bits_cl", "num_bits"):
            assert np.array_equal(out[key][l], g["compress_%s_%d" % (key, i)]), key
    wide = (stds * np.float32(3.0)).astype(np.float32)
    out = q.compress_latents(g["means"], g["logvars"], lambs, posterior_stds=wide)
    Zh, nb = q.compress_batch_channel_latents(g["means"].reshape(-1, C), wide.reshape(-1, C), lambs)
    assert any(not np.array_equal(Zh[l], g["cl_zhat_%d" % i]) for i, l in enumerate(lambs))
    for l in lambs:
        assert np.array_equal(out["Z_hat"][l].reshape(-1, C), Zh[l]) and np.array_equal(out["raw_num_bits"][l].reshape(-1, C), nb[l])


def test_sorted_rank_formula():
    g = load("learned_c6_n10")
    N = int(g["N"])
    n = np.repeat(np.arange(N + 1), [2 ** k for k in range(N + 1)])
    i = np.concatenate([np.arange(2 ** k) for k in range(N + 1)])
    rank = O.heap_to_sorted_rank(n, i, N)
    for c in range(int(g["C"])):
        assert np.array_equal(g["sorted_table"][c][rank], g["table"][c])


def test_algorithm1_xi_space_equals_z_space_search():
    """utils.encode_vectorized (numba xi-space Algorithm 1) vs the z-space bracket search used everywhere else."""
    g = load("utils_numpy")
    N = 10
    from scipy.stats import norm
    cp = norm.ppf(O.xi_heap(N), scale=float(g["ev_prior_std"]))
    for i, lamb in enumerate(g["ev_lambs"]):
        zh, bits = O.bracket_search_f64(g["ev_mu"], g["ev_sigma"], float(lamb), cp, N)
        same = zh == g["ev_zhat_%d" % i]
        assert same.mean() > 0.999          # xi-space vs z-space bracketing may differ on exact grid hits / ties only
        assert np.array_equal(bits[same], g["ev_bits_%d" % i][same])


def test_generic_operator():
    g = load("utils_numpy")
    lambs = [float(l) for l in g["bq_lambs"]]
    Zh, nb = O.batch_quantize_indep_dims(g["bq_P"], g["bq_L"], g["bq_loc"], g["bq_scale"], lambs)
    for i, l in enumerate(lambs):
        assert np.array_equal(Zh[l], g["bq_zhat_%d" % i]) and np.array_equal(nb[l], g["bq_bits_%d" % i])


def test_notebook_codepoints_and_exhaustive_search():
    g = load("notebook_embeddings")
    cp, ln = O.notebook_codepoints(float(g["empirical_std"]), 10)
    assert np.array_equal(cp, g["codepoints"]) and np.array_equal(ln, g["lengths"])
    for i, beta in enumerate(g["betas"]):
        opt, idx = O.compress_coordinates(g["means"], g["stds"], float(beta), cp, ln)
        assert opt.dtype == np.float32 and np.array_equal(opt, g["optima_%d" % i])
        # "exact same result" claim of ipynb:482: the 2N+1 bracketing candidates suffice
        opt_b, idx_b = O.compress_coordinates_bracket(g["means"], g["stds"], float(beta), cp, 10)
        assert np.array_equal(opt_b, opt) and np.array_equal(idx_b, idx)
