"""Arbitrary-precision reference for the prior numerics (CPU only): the learned prior's logits, CDF and inverse CDF,
the standard-normal quantile, and correct rounding to float32.

Everything is evaluated with mpmath on the float32 parameters exactly as given (every float32 and float64 is an exact
mpf), so the results are the true values of the operations the kernels approximate, not another float64 restatement.
The root solvers stop at about 35 significant digits, far below any float32 or float64 rounding they are compared with.
"""
import numpy as np
import pytest

mpmath = pytest.importorskip("mpmath")
mp = mpmath.mp
mpf = mpmath.mpf

DPS = 40                      # working precision of every evaluation
ROOT_REL = mpf(10) ** -36     # stop a root solve once the Newton step is below this, relative (~35 digits)
U64 = 2.0 ** -53              # unit roundoff, float64
U32 = 2.0 ** -24              # unit roundoff, float32
F32_MAX = float(np.finfo(np.float32).max)

# packed C-ABI layout of one channel (include/vbq_b200.h): m0 b0 f0 | m1 b1 f1 | m2 b2 f2 | m3 b3
_SLICES = dict(m0=(0, 3), b0=(3, 6), f0=(6, 9), m1=(9, 18), b1=(18, 21), f1=(21, 24), m2=(24, 33), b2=(33, 36),
               f2=(36, 39), m3=(39, 42), b3=(42, 43))


class _Prior:
    """One channel's 43 float32 parameters as exact mpf values (and as float64 for the error bounds)."""

    def __init__(self, params_c):
        p = np.asarray(params_c, dtype=np.float32).reshape(-1)
        assert p.size == 43, "one channel of the packed (C, 43) block"
        self.f64 = {k: p[a:b].astype(np.float64) for k, (a, b) in _SLICES.items()}
        with mp.workdps(DPS):
            self.mp = {k: [mpf(float(v)) for v in p[a:b]] for k, (a, b) in _SLICES.items()}


_PRIORS = {}


def _prior(params_c):
    if isinstance(params_c, _Prior):
        return params_c
    key = np.asarray(params_c, dtype=np.float32).tobytes()
    if key not in _PRIORS:
        _PRIORS[key] = _Prior(params_c)
    return _PRIORS[key]


def _logits_d(P, x):
    """logits(x) and d logits / dx, in the layer order of priors.cu::prior_logits (learned_prior.py:70-107)."""
    q = P.mp
    h, dh = [], []
    for i in range(3):
        v = q["m0"][i] * x + q["b0"][i]
        th = mpmath.tanh(v)
        h.append(v + q["f0"][i] * th)
        dh.append(q["m0"][i] * (1 + q["f0"][i] * (1 - th * th)))
    for m, b, f in (("m1", "b1", "f1"), ("m2", "b2", "f2")):
        g, dg = [], []
        for i in range(3):
            v = q[m][3 * i] * h[0] + q[m][3 * i + 1] * h[1] + q[m][3 * i + 2] * h[2] + q[b][i]
            th = mpmath.tanh(v)
            g.append(v + q[f][i] * th)
            dg.append((q[m][3 * i] * dh[0] + q[m][3 * i + 1] * dh[1] + q[m][3 * i + 2] * dh[2])
                      * (1 + q[f][i] * (1 - th * th)))
        h, dh = g, dg
    lg = q["m3"][0] * h[0] + q["m3"][1] * h[1] + q["m3"][2] * h[2] + q["b3"][0]
    return lg, q["m3"][0] * dh[0] + q["m3"][1] * dh[1] + q["m3"][2] * dh[2]


def logits(params_c, x):
    """The learned prior's logits of one channel at x (a float or mpf), exact to ~DPS digits."""
    with mp.workdps(DPS):
        return _logits_d(_prior(params_c), mpf(x))[0]


def cdf(params_c, x):
    """sigmoid(logits(x)) to ~DPS digits (mpf; no underflow: mpmath exponents are unbounded)."""
    with mp.workdps(DPS):
        return 1 / (1 + mpmath.exp(-_logits_d(_prior(params_c), mpf(x))[0]))


def logit(xi):
    """log(xi) - log1p(-xi) of a float64 xi in (0, 1), to ~DPS digits."""
    with mp.workdps(DPS):
        xi = mpf(float(xi))
        return mpmath.log(xi) - mpmath.log1p(-xi)


def inverse_cdf(params_c, xi, guess=None):
    """The root z of logits(z) = log(xi) - log1p(-xi), xi a float64 in (0, 1), to ~35 significant digits (mpf).

    The root is bracketed first (by doubling from [-1, 1], or by widening around `guess`: a guess only saves
    iterations, the bracket is checked by the sign of the residual either way), then refined by Newton steps that fall
    back to bisection whenever they leave the bracket."""
    P = _prior(params_c)
    with mp.workdps(DPS):
        target = logit(xi)

        def f(z):
            return _logits_d(P, z)[0] - target

        if guess is not None and np.isfinite(guess):
            g = mpf(float(guess))
            d = max(abs(g) * mpf(2) ** -20, mpf(2) ** -120)
            lo, hi = g - d, g + d
            while not f(lo) < 0:
                d *= 16
                lo = g - d
            while not f(hi) > 0:
                d *= 16
                hi = g + d
        else:
            lo, hi = mpf(-1), mpf(1)
            while not f(lo) < 0:
                lo *= 2
            while not f(hi) > 0:
                hi *= 2
        x = (lo + hi) / 2 if guess is None or not np.isfinite(guess) else mpf(float(guess))
        x = min(max(x, lo), hi)
        for _ in range(400):
            v, dv = _logits_d(P, x)
            r = v - target
            if r == 0:
                return x
            if r < 0:
                lo = x
            else:
                hi = x
            xn = x - r / dv if dv > 0 else (lo + hi) / 2
            if not lo < xn < hi:
                xn = (lo + hi) / 2
            step = abs(xn - x)
            x = xn
            if step <= ROOT_REL * abs(x) or hi - lo <= ROOT_REL * max(abs(lo), abs(hi)):
                return x
        raise AssertionError("inverse_cdf did not converge at xi=%r" % xi)


def ndtri(p):
    """The standard-normal quantile Phi^-1(p) of a float64 p in (0, 1), to ~35 significant digits (mpf).

    Newton on log(ncdf(x)) - log(p) in the lower half (the upper half by symmetry, 1 - p being exact), which keeps
    full relative accuracy down to p = 1e-300, where erfinv(2p - 1) at fixed precision has none left."""
    with mp.workdps(DPS):
        p = mpf(float(p))
        assert 0 < p < 1
        if p > mpf(0.5):
            return -ndtri(1 - p)
        if p == mpf(0.5):
            return mpf(0)
        lp = mpmath.log(p)
        # start from the tail asymptote (or 0 near the centre); Newton on a concave log-CDF converges from above
        x = -mpmath.sqrt(-2 * lp) if p < mpf(0.1) else mpf(0)
        for _ in range(200):
            c = mpmath.ncdf(x)
            step = (mpmath.log(c) - lp) * c / mpmath.npdf(x)
            x -= step
            if abs(step) <= ROOT_REL * abs(x):
                return x
        raise AssertionError("ndtri did not converge at p=%r" % p)


def f32_correctly_rounded(v):
    """(the float32 nearest to the mpf v, relative distance from v to the nearest float32 rounding boundary).

    A float64 computation of v that is accurate to a relative error below that distance rounds to the same float32;
    within it, either neighbour is a correct result of a correct-to-float64 computation.  Values beyond the float32
    range round to +-inf (distance measured to the overflow threshold)."""
    with mp.workdps(DPS):
        v = mpf(v)
        if v == 0:
            return np.float32(0.0), np.inf
        big = mpf(F32_MAX) + mpf(2) ** (127 - 24)           # overflow threshold: max + half an ulp
        if abs(v) >= big:
            return np.float32(np.inf if v > 0 else -np.inf), float(abs(abs(v) - big) / abs(v))
        f = np.float32(float(v))                             # within one float32 ulp of v
        cands = [np.nextafter(f, np.float32(-np.inf)), f, np.nextafter(f, np.float32(np.inf))]
        cands = [c for c in cands if np.isfinite(c)]
        best = min(cands, key=lambda c: abs(mpf(float(c)) - v))
        lo = np.nextafter(best, np.float32(-np.inf))
        hi = np.nextafter(best, np.float32(np.inf))
        b = mpf(float(best))
        dist = []
        for nb in (lo, hi):
            if np.isfinite(nb):
                dist.append(abs(v - (b + mpf(float(nb))) / 2))
            else:
                dist.append(abs(abs(v) - big))
        return best, float(min(dist) / abs(v))


# ----------------------------------------------------------------------------------------------------------------------
# a-priori error bounds of the finite-precision evaluations (vectorised over x, float64 arithmetic)
# ----------------------------------------------------------------------------------------------------------------------
def logits_error_bound(params_c, x, u, tanh_ulps):
    """Running (forward) error bound of logits(x) evaluated in a floating-point format of unit roundoff `u`, in the
    layer order of prior_logits, with a tanh accurate to `tanh_ulps` ulps (<= 2 u |tanh| per ulp).

    Per operation: v = sum m*h + b carries sum |m| E_h plus k u (sum |m h| + |b|) for its k = (terms + 1) roundings;
    tanh carries (1 - tanh^2) E_v plus its own error; h = v + f tanh carries E_v + |f| E_tanh plus 2 u (|f tanh| + |h|).
    The bound is first order in u (the neglected terms are O(u^2) relative)."""
    P = _prior(params_c).f64
    x = np.asarray(x, dtype=np.float64)
    with np.errstate(over="ignore", invalid="ignore"):
        h, E = [], []
        for i in range(3):
            v = P["m0"][i] * x + P["b0"][i]
            Ev = 2 * u * (np.abs(P["m0"][i] * x) + np.abs(P["b0"][i]))
            th = np.tanh(v)
            Eth = (1 - th * th) * Ev + tanh_ulps * 2 * u * np.abs(th)
            hi = v + P["f0"][i] * th
            h.append(hi)
            E.append(Ev + abs(P["f0"][i]) * Eth + 2 * u * (np.abs(P["f0"][i] * th) + np.abs(hi)))
        for m, b, f in (("m1", "b1", "f1"), ("m2", "b2", "f2")):
            g, Eg = [], []
            for i in range(3):
                row = P[m][3 * i: 3 * i + 3]
                v = row[0] * h[0] + row[1] * h[1] + row[2] * h[2] + P[b][i]
                mag = np.abs(row[0] * h[0]) + np.abs(row[1] * h[1]) + np.abs(row[2] * h[2]) + abs(P[b][i])
                Ev = abs(row[0]) * E[0] + abs(row[1]) * E[1] + abs(row[2]) * E[2] + 4 * u * mag
                th = np.tanh(v)
                Eth = (1 - th * th) * Ev + tanh_ulps * 2 * u * np.abs(th)
                gi = v + P[f][i] * th
                g.append(gi)
                Eg.append(Ev + abs(P[f][i]) * Eth + 2 * u * (np.abs(P[f][i] * th) + np.abs(gi)))
            h, E = g, Eg
        r = P["m3"]
        mag = np.abs(r[0] * h[0]) + np.abs(r[1] * h[1]) + np.abs(r[2] * h[2]) + abs(P["b3"][0])
        return abs(r[0]) * E[0] + abs(r[1]) * E[1] + abs(r[2]) * E[2] + 4 * u * mag


def solver_band(params_c, z, xi):
    """Relative half-width of the interval in which `solve_inverse_cdf` (float64, priors.cu) may land around the true
    root z of logits = logit(xi): the epsilon band of the float32 comparisons.

      * stopping rule: Newton stops after a step <= 1e-14 |x|; the step before it was >= 1e-7 |x| only if convergence
        was not yet quadratic, and in the quadratic regime the remaining error is far below the last step, so the
        stopping rule contributes at most 1e-14 |x|;
      * the float64 evaluation: the computed residual logits(x) - target is off by at most E_L (logits_error_bound
        with u = 2^-53 and a 2-ulp tanh) plus 2 ulps of the target (log and log1p are each within 1 ulp, and their
        difference adds one rounding), which moves the root by that amount over the slope logits'(z).
    The same band covers LearnedPriorNP.inverse_cdf_f64, whose bisection to float64 resolution adds one float64 ulp."""
    with mp.workdps(DPS):
        _, slope = _logits_d(_prior(params_c), mpf(z))
        target = abs(logit(xi))
    e_eval = float(logits_error_bound(params_c, float(z), U64, 2)) + 4 * U64 * float(target)
    az = max(abs(float(z)), np.finfo(np.float64).tiny)
    return 1e-14 + 2 * U64 + e_eval / (float(slope) * az)
