"""CPU checks of the arbitrary-precision prior reference (tests/prior_reference.py): against SciPy's ndtri, against
the float64 table oracle LearnedPriorNP.inverse_cdf_f64, and on priors whose quantiles are known in closed form."""
import numpy as np
import pytest

import prior_reference as R
from oracle import vbq_oracle as O
import vbq_test_helpers as H

mpmath = R.mpmath


def _heap_xi(h):
    h = np.asarray(h, dtype=np.int64)
    n = np.floor(np.log2(h + 1)).astype(np.int64)
    i = h + 1 - (1 << n)
    return (i + 0.5) * np.exp2(-n.astype(np.float64))


def _depth_sample(N, per_depth, seed):
    """Heap indices: both ends and the middle of every depth 0..N plus `per_depth` random entries of each."""
    rng = np.random.default_rng(seed)
    hs = []
    for n in range(N + 1):
        base, w = (1 << n) - 1, 1 << n
        hs += [base, base + w // 2, base + w - 1]
        hs += list(base + rng.integers(0, w, min(per_depth, w)))
    return np.unique(np.asarray(hs, dtype=np.int64))


def test_ndtri_against_scipy():
    from scipy.special import ndtri
    p = np.concatenate([np.logspace(-300, np.log10(0.5), 60), 1 - np.logspace(-1, -15.9, 30),
                        [1 - 2.0 ** -53, 0.5, 0.25, 0.75], _heap_xi(_depth_sample(20, 4, 0))])
    for pk in p:
        want = R.ndtri(pk)
        got = ndtri(pk)
        # Cephes ndtri (SciPy): documented peak relative error 7.2e-16 over (0.125, 1) and 4.6e-16 below it; plus
        # half an ulp for the exact value's own float64 rounding: 8e-16 relative, ~3.6 float64 ulps
        assert abs(mpmath.mpf(float(got)) - want) <= 8e-16 * abs(want), (pk, got, want)
    # symmetry and the centre are exact in the reference
    assert R.ndtri(0.5) == 0
    assert R.ndtri(0.25) + R.ndtri(0.75) == 0


def test_ndtri_known_values():
    # Phi(-1.959963984540054...) = 0.025; Phi^-1(2^-53) from the tail: check the residual in high precision
    for p in (0.025, 2.0 ** -53, 1e-300, 0.3):
        x = R.ndtri(p)
        with mpmath.workdps(60):
            assert abs(mpmath.ncdf(x) / mpmath.mpf(p) - 1) < mpmath.mpf(10) ** -33


def _symmetric_prior(C=2, seed=0):
    """Zero biases: every layer is odd in its input, so logits is odd and the median is exactly 0."""
    pr = H.make_prior(C, seed=seed, factor_std=0.5)
    pr.biases = [np.zeros_like(b) for b in pr.biases]
    return pr


def test_known_answer_symmetric_prior():
    pr = _symmetric_prior()
    for c, p in enumerate(pr.packed()):
        assert R.inverse_cdf(p, 0.5) == 0
        for xi in (0.25, 2.0 ** -20, 0.4375):
            a, b = R.inverse_cdf(p, xi), R.inverse_cdf(p, 1 - xi)
            with mpmath.workdps(R.DPS):
                assert abs(a + b) <= mpmath.mpf(10) ** -34 * abs(a)
        assert R.cdf(p, 0.0) == mpmath.mpf(0.5)


def _logistic_params(scale, shift):
    """One identity path through the network, no gates: logits(x) = x / scale - shift / scale."""
    p = np.zeros(43, dtype=np.float32)
    p[0] = np.float32(1.0 / scale)          # m0[0]
    p[3] = np.float32(-shift / scale)       # b0[0]
    p[9] = p[13] = p[17] = 1.0              # m1 = I
    p[24] = p[28] = p[32] = 1.0             # m2 = I
    p[39] = 1.0                             # m3 = [1, 0, 0]
    return p


@pytest.mark.parametrize("scale,shift", [(1.0, 0.0), (0.125, 3.0), (1024.0, -7.5)])
def test_known_answer_logistic(scale, shift):
    with mpmath.workdps(R.DPS):   # the comparisons below need more than mpmath's default 53 bits
        p = _logistic_params(scale, shift)
        a, b = mpmath.mpf(float(p[0])), mpmath.mpf(float(p[3]))
        for xi in (0.5, 0.3, 2.0 ** -21, 1 - 2.0 ** -21, 1e-300):
            want = (R.logit(xi) - b) / a      # logits(x) = a x + b
            got = R.inverse_cdf(p, xi)
            assert abs(got - want) <= mpmath.mpf(10) ** -34 * max(abs(want), 1), xi
            # the guess only shortens the search
            assert abs(R.inverse_cdf(p, xi, guess=float(want) * (1 + 1e-3) + 1e-3) - want) <= \
                mpmath.mpf(10) ** -34 * max(abs(want), 1)
        x = 0.7
        assert abs(R.cdf(p, x) - 1 / (1 + mpmath.exp(-(a * x + b)))) < mpmath.mpf(10) ** -38


def test_logits_layer_order_matches_numpy_oracle():
    for fs, scale in ((0.0, 10.0), (3.0, 10.0), (0.5, 1000.0), (0.5, 0.01)):
        pr = H.make_prior(3, seed=4, factor_std=fs, init_scale=scale)
        x = np.array([-50.0, -1.5, 0.0, 0.3, 7.0, 1e3]) * scale
        want = pr.logits(np.repeat(x[:, None], 3, axis=1))
        for c, p in enumerate(pr.packed()):
            for k, xk in enumerate(x):
                got = float(R.logits(p, xk))
                bound = R.logits_error_bound(p, xk, R.U64, 1)    # NumPy's float64 evaluation of the same layers
                assert abs(got - want[k, c]) <= bound, (fs, scale, c, xk)


def test_f32_correctly_rounded():
    with mpmath.workdps(R.DPS):
        one = mpmath.mpf(1)
        f, d = R.f32_correctly_rounded(one)
        assert f == np.float32(1) and d > 0
        # halfway between 1 and 1 + 2^-23, nudged either way
        mid = one + mpmath.mpf(2) ** -24
        assert R.f32_correctly_rounded(mid + mpmath.mpf(2) ** -60)[0] == np.nextafter(np.float32(1), np.float32(2))
        assert R.f32_correctly_rounded(mid - mpmath.mpf(2) ** -60)[0] == np.float32(1)
        assert R.f32_correctly_rounded(mid - mpmath.mpf(2) ** -60)[1] < 2.0 ** -35
        # double rounding trap: a value just above a float32 midpoint that float64 rounds onto the midpoint
        v = mid + mpmath.mpf(2) ** -80
        assert np.float32(float(v)) == np.float32(1)                    # float64 first, then float32: ties to even
        assert R.f32_correctly_rounded(v)[0] == np.nextafter(np.float32(1), np.float32(2))
        assert R.f32_correctly_rounded(-mpmath.mpf(3.5))[0] == np.float32(-3.5)
        assert R.f32_correctly_rounded(mpmath.mpf(10) ** 39)[0] == np.float32(np.inf)


@pytest.mark.parametrize("fs,scale,seed", [(0.5, 10.0, 1), (3.0, 1000.0, 2), (0.0, 0.01, 3)])
def test_inverse_cdf_f64_oracle_is_correctly_rounded(fs, scale, seed):
    """LearnedPriorNP.inverse_cdf_f64 (float64 bisection, rounded to float32) returns the correctly rounded float32
    of the true root, except where that root lies within the solver band of a float32 rounding boundary."""
    C = 3
    pr = H.make_prior(C, seed=seed, factor_std=fs, init_scale=scale)
    hs = _depth_sample(20, 3, seed)
    xi = _heap_xi(hs)
    f64 = pr.inverse_cdf_f64(np.repeat(xi[:, None], C, axis=1))
    n_band = 0
    for c, p in enumerate(pr.packed()):
        for k, x in enumerate(xi):
            z = R.inverse_cdf(p, x, guess=float(f64[k, c]))
            want, dist = R.f32_correctly_rounded(z)
            if f64[k, c] != want:
                assert dist <= R.solver_band(p, z, x), (c, x, f64[k, c], want)
                n_band += 1
    assert n_band <= 2
