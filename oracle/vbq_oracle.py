"""CPU oracle for the VBQ rate-distortion quantization path.  TEST INFRASTRUCTURE ONLY.

This module is a NumPy restatement of the reference's algorithm (mandt-lab/vbq).  It is the
*checker* for the CUDA path: only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s
``cpu_baseline`` / ``--impl reference`` legs may import it.  Nothing under ``vbq_b200/`` imports it,
and the product path raises if the CUDA library is missing rather than falling back to this code.

Pinning status: the reference ships no golden vectors for this path (SURVEY.md §4).  The oracle is
pinned against outputs of the *reference's own code run in the build container*:
  * ``tests/golden/gen_golden.py`` imports ``/root/reference/img-compression/utils.py`` (NumPy/numba half,
    unmodified) and executes the notebook cells verbatim, and runs the unmodified
    ``quantizer.py`` / ``learned_prior.py`` / ``vae_models.py`` on a NumPy stand-in for the TF-eager ops
    they call (``oracle/tf_shim``); the resulting vectors live in ``tests/golden/*.npz``.
  * the docstring known-answer ``get_n_bit_interval(0.4375, 2) -> [0.375, 0.625]`` (utils.py:27-37) and
    the invariant "every z_hat is exactly a table entry" (quantizer.py:136-137) are tested directly.
Third-party arithmetic the reference delegates to and that is absent here: TensorFlow 1.15.0 eager kernels
(searchsorted/gather/argmax/matmul/tanh/sigmoid/sort); restated with NumPy float32 ops of the same
published semantics.  SciPy ``norm.ppf`` (pinned 1.3.3) is present at 1.18.

Every function cites the reference file:line it follows (paths relative to /root/reference).
"""
from __future__ import annotations

import numpy as np

F32 = np.float32


# ----------------------------------------------------------------------------------------------
# xi grid (img-compression/utils.py:23-24, quantizer.py:30)
# ----------------------------------------------------------------------------------------------
def n_bit_binary_floats(n):
    """Level-n quantiles (i + 1/2) * 2^-n, i < 2^n.  utils.py:23-24."""
    return [i * 2 ** (-n) + 2 ** (-n - 1) for i in range(2 ** n)]


def xi_heap(N):
    """All Q = 2^(N+1)-1 quantiles in heap order (level-major, ascending in a level).  quantizer.py:30."""
    return np.hstack([n_bit_binary_floats(n) for n in range(N + 1)])


def heap_to_sorted_rank(n, i, N):
    """Rank of code point (level n, index i) in the ascending list of all Q points.

    Equals what quantizer.py:135,223 obtain by searchsorted(code_points_by_channel, z_hat) when the table
    has no duplicates (SURVEY.md §7.2)."""
    return (2 * np.asarray(i, dtype=np.int64) + 1) * (1 << (N - np.asarray(n, dtype=np.int64))) - 1


def get_n_bit_interval(x, n):
    """xi-space bracket used only as a known-answer test (utils.py:27-37 docstring)."""
    if n == 0:
        return [0.5, 0.5]
    w = 2.0 ** (-n)
    off = 0.5 * w
    if x < off:
        return [off, off]
    if x > 1 - off:
        return [1 - off, 1 - off]
    left = np.floor((x - off) / w) * w + off
    return [left, left + w]


# ----------------------------------------------------------------------------------------------
# Learned factorized prior (img-compression/learned_prior.py)
# ----------------------------------------------------------------------------------------------
def softplus(x):
    return np.logaddexp(0.0, x)


class LearnedPriorNP:
    """NumPy restatement of BMSHJ2018Prior's CDF / inverse CDF (learned_prior.py:6-218).

    ``matrices[k]`` (C, d_{k+1}, d_k), ``biases[k]`` (C, d_{k+1}, 1), ``factors[k]`` (C, d_{k+1}, 1) hold the
    *transformed* parameters (softplus / identity / tanh already applied: learned_prior.py:43,57)."""

    def __init__(self, matrices, biases, factors):
        self.matrices = [np.asarray(m, dtype=F32) for m in matrices]
        self.biases = [np.asarray(b, dtype=F32) for b in biases]
        self.factors = [np.asarray(f, dtype=F32) for f in factors]
        self.channels = self.matrices[0].shape[0]

    @classmethod
    def init(cls, channels, dims=(3, 3, 3), init_scale=10.0, rng=None, factor_std=0.0):
        """Reference initialisation (learned_prior.py:30-58): constant softplus^-1 matrices, biases U(-.5,.5),
        zero raw factors.  ``factor_std`` > 0 perturbs the raw factors so the tanh gates are exercised."""
        rng = np.random.default_rng(0) if rng is None else rng
        fdims = (1,) + tuple(dims) + (1,)
        scale = init_scale ** (1 / (len(dims) + 1))
        mats, bs, fs = [], [], []
        for i in range(len(dims) + 1):
            init = np.log(np.expm1(1 / scale / fdims[i + 1]))
            raw = np.full((channels, fdims[i + 1], fdims[i]), init, dtype=F32)
            mats.append(softplus(raw).astype(F32))
            bs.append(rng.uniform(-0.5, 0.5, size=(channels, fdims[i + 1], 1)).astype(F32))
            if i < len(dims):
                rawf = (factor_std * rng.standard_normal((channels, fdims[i + 1], 1))).astype(F32)
                fs.append(np.tanh(rawf).astype(F32))
        return cls(mats, bs, fs)

    def packed(self):
        """(C, 43) float32 block in the C-ABI layout (include/vbq_b200.h): per layer k: matrix row-major,
        bias, factor (k<3)."""
        cols = []
        for k in range(len(self.matrices)):
            C = self.channels
            cols.append(self.matrices[k].reshape(C, -1))
            cols.append(self.biases[k].reshape(C, -1))
            if k < len(self.factors):
                cols.append(self.factors[k].reshape(C, -1))
        return np.ascontiguousarray(np.concatenate(cols, axis=1), dtype=F32)

    # learned_prior.py:70-107
    def logits_cdf(self, x_c1b, dtype=F32):
        logits = np.asarray(x_c1b, dtype=dtype)
        for i in range(len(self.matrices)):
            logits = np.matmul(self.matrices[i].astype(dtype), logits)
            logits = logits + self.biases[i].astype(dtype)
            if i < len(self.factors):
                logits = logits + self.factors[i].astype(dtype) * np.tanh(logits)
        return logits

    # learned_prior.py:109-148 (channel-last in, channel-last out)
    def cdf(self, inputs, dtype=F32):
        x = np.asarray(inputs, dtype=dtype)
        assert x.shape[-1] == self.channels
        xc = np.moveaxis(x, -1, 0).reshape(self.channels, 1, -1)
        lg = self.logits_cdf(xc, dtype=dtype)
        with np.errstate(over="ignore"):
            cdf = 1.0 / (1.0 + np.exp(-lg))
        cdf = cdf.astype(dtype).reshape((self.channels,) + x.shape[:-1])
        return np.moveaxis(cdf, 0, -1)

    def logits(self, inputs, dtype=np.float64):
        x = np.asarray(inputs, dtype=dtype)
        xc = np.moveaxis(x, -1, 0).reshape(self.channels, 1, -1)
        lg = self.logits_cdf(xc, dtype=dtype).reshape((self.channels,) + x.shape[:-1])
        return np.moveaxis(lg, 0, -1)

    # learned_prior.py:173-218, literal float32 restatement (global doubling, min-width stop, returns last mid)
    def inverse_cdf_reference(self, xi, max_iterations=1000, tol=1e-9):
        xi = np.asarray(xi)
        left = np.ones_like(xi, dtype=F32) * F32(-1)
        right = np.ones_like(xi, dtype=F32) * F32(1)

        # the reference passes a float64 ndarray xi; TF's binary-op wrapper converts it to the dtype of the
        # float32 cdf tensor, so the subtraction is float32 arithmetic.
        xi32 = xi.astype(F32)

        def f(z):
            return self.cdf(z, dtype=F32) - xi32

        while not np.all(f(left) < 0):
            left = left * F32(2)
        while not np.all(f(right) > 0):
            right = right * F32(2)
        mid = None
        for _ in range(max_iterations):
            mid = F32(0.5) * (left + right)
            v = f(mid)
            pos = v > 0
            neg = v < 0
            left = left * (~neg).astype(F32) + mid * neg.astype(F32)
            right = right * (~pos).astype(F32) + mid * pos.astype(F32)
            if np.all(~pos & ~neg) or np.min(right - left) <= tol:
                break
        return mid

    def inverse_cdf_f64(self, xi, iters=200):
        """Table-check oracle (SURVEY.md §7.3-2): root of logits_c(z) = logit(xi) with float64 arithmetic on the
        float32 parameters, by bisection to float64 resolution, then rounded to float32."""
        xi = np.asarray(xi, dtype=np.float64)
        target = np.log(xi) - np.log1p(-xi)
        lo = -np.ones_like(xi)
        hi = np.ones_like(xi)
        for _ in range(200):
            bad = self.logits(lo) >= target
            if not bad.any():
                break
            lo = np.where(bad, lo * 2, lo)
        for _ in range(200):
            bad = self.logits(hi) <= target
            if not bad.any():
                break
            hi = np.where(bad, hi * 2, hi)
        for _ in range(iters):
            mid = 0.5 * (lo + hi)
            v = self.logits(mid) - target
            lo = np.where(v < 0, mid, lo)
            hi = np.where(v < 0, hi, mid)
        return (0.5 * (lo + hi)).astype(F32)


# ----------------------------------------------------------------------------------------------
# Gaussian priors (img-compression/vae_models.py:14-43; notebook ipynb:373-390)
# ----------------------------------------------------------------------------------------------
def gaussian_inverse_cdf(xi, mean=None, std=None):
    """norm.ppf(xi, loc, scale) in float64.  vae_models.py:23-25, :40-43."""
    from scipy.stats import norm
    if mean is None:
        return norm.ppf(xi)
    return norm.ppf(xi, loc=mean, scale=std)


def notebook_codepoints(empirical_std, max_codepoint_length=10):
    """Heap-order code points and lengths exactly as ipynb:383-390 (float64 / int)."""
    from scipy.stats import norm
    cl = [(norm.ppf(x, scale=empirical_std), length)
          for length in range(max_codepoint_length + 1)
          for x in np.arange(0.5 ** (length + 1), 1, 0.5 ** length)]
    return np.array([c for c, _ in cl]), np.array([l for _, l in cl])


def compress_coordinates(means, stds, beta, codepoints, bitlengths, chunk=100000):
    """Notebook exhaustive search, ipynb:429-443, with the hard-coded loop bound generalised to len(means).

    Arithmetic follows NumPy's promotion for a Python-float ``beta``: ``(2*beta) * stds**2`` stays float32,
    the product with the int64 ``bitlengths`` and the float64 ``codepoints`` term promote to float64.
    Returns (optima shaped/dtyped like ``means``, heap index of the optimum)."""
    beta = float(beta)
    optima = np.empty_like(means)
    idxs = np.empty(means.size, dtype=np.int64)
    m = means.ravel()
    s = stds.ravel()
    for i in range(0, m.size, chunk):
        squared_errors = (codepoints[np.newaxis, :] - m[i:i + chunk, np.newaxis]) ** 2
        weighted_penalties = (2 * beta) * s[i:i + chunk, np.newaxis] ** 2 * bitlengths[np.newaxis, :]
        k = np.argmin(squared_errors + weighted_penalties, axis=1)
        optima.ravel()[i:i + chunk] = codepoints[k]
        idxs[i:i + chunk] = k
    return optima, idxs.reshape(means.shape)


def compress_coordinates_bracket(means, stds, beta, codepoints, N, pen_f64=False):
    """Same objective and tie rule (first minimum in heap order) as ``compress_coordinates`` but evaluated only
    on the 2N+1 bracketing candidates (SURVEY.md §0; equivalence claimed at ipynb:482).  float64."""
    beta = float(beta)
    m = means.ravel().astype(np.float64)
    if pen_f64:   # NumPy >= 2 with a NumPy float64 `beta`: the product is formed in float64 (SURVEY §7.3-7)
        pen_unit = (2 * beta) * (stds.ravel() ** 2).astype(np.float64)
    else:
        pen_unit = ((2 * beta) * stds.ravel() ** 2).astype(np.float64)  # float32 product promoted afterwards
    best = np.full(m.shape, np.inf)
    best_h = np.zeros(m.shape, dtype=np.int64)
    for n in range(N + 1):
        grid = codepoints[2 ** n - 1: 2 ** (n + 1) - 1]
        r = np.clip(np.searchsorted(grid, m, side="left"), 0, 2 ** n - 1)
        l = np.clip(r - 1, 0, 2 ** n - 1)
        for idx in (l, r):  # lower heap index first => first-minimum tie rule preserved inside a level
            loss = (grid[idx] - m) ** 2 + pen_unit * n
            upd = loss < best
            best = np.where(upd, loss, best)
            best_h = np.where(upd, 2 ** n - 1 + idx, best_h)
    optima = codepoints[best_h].astype(means.dtype).reshape(means.shape)
    return optima, best_h.reshape(means.shape)


def empirical_entropy(values):
    """ipynb:452-455."""
    _, counts = np.unique(np.asarray(values).ravel(), return_counts=True)
    total = counts.sum()
    return total * np.log2(total) - counts.dot(np.log2(counts))


# ----------------------------------------------------------------------------------------------
# ChannelwisePriorCDFQuantizer restatement (img-compression/quantizer.py:13-256)
# ----------------------------------------------------------------------------------------------
class QuantizerNP:
    """Float32 NumPy restatement of ChannelwisePriorCDFQuantizer's hot path."""

    def __init__(self, num_channels, max_bits_per_coord):
        self.N = int(max_bits_per_coord)
        self.C = int(num_channels)
        self.Q = 2 ** (self.N + 1) - 1
        self.raw_code_length_entropy_models = None
        self.entropy_models = None

    # quantizer.py:25-63
    def set_code_points(self, all_code_points, build_grids=True):
        """``all_code_points``: (C, Q) heap order (what quantizer.py:36 stores)."""
        acp = np.asarray(all_code_points, dtype=F32)
        assert acp.shape == (self.C, self.Q)
        self.all_code_points = acp
        self.code_points_by_channel = np.sort(acp, axis=1)
        N = self.N
        self._search_grids = None
        if build_grids:
            grids = np.empty((self.C, N + 1, 2 ** N), dtype=F32)
            for n in range(N + 1):
                lvl = acp[:, 2 ** n - 1: 2 ** (n + 1) - 1]
                if n == 0:
                    grids[:, 0, :] = lvl[:, :1]  # np.pad([p]*2, 2^(N-1)-1, 'edge'): all equal
                else:
                    p = 2 ** (N - 1) - 2 ** (n - 1)
                    grids[:, n, :] = np.pad(lvl, ((0, 0), (p, p)), mode="edge")
            self._search_grids = grids

    def build_code_points(self, inverse_cdf):
        xi = xi_heap(self.N)
        xi_rep = np.repeat(xi[:, None], self.C, axis=1)
        self.set_code_points(np.asarray(inverse_cdf(xi_rep)).astype(F32).T)

    # quantizer.py:65-80 (literal: searchsorted in the edge-padded grids)
    def get_all_N_bit_intervals(self, Z):
        N, C = self.N, self.C
        B = Z.shape[0]
        left = np.empty((C, N + 1, B), dtype=F32)
        right = np.empty((C, N + 1, B), dtype=F32)
        for c in range(C):
            for n in range(N + 1):
                g = self._search_grids[c, n]
                r = np.clip(np.searchsorted(g, Z[:, c], side="left"), 0, 2 ** N - 1)
                l = np.clip(r - 1, 0, 2 ** N - 1)
                right[c, n] = g[r]
                left[c, n] = g[l]
        return left, right

    def get_all_N_bit_intervals_fast(self, Z):
        """Same result without the 2^N-wide padded grids (needed for N=16); edge semantics of quantizer.py:57,75-76:
        mu <= lowest -> left=right=lowest; mu > highest -> left=right=highest for n<N, (second-highest, highest)
        for n=N."""
        N, C = self.N, self.C
        B = Z.shape[0]
        left = np.empty((C, N + 1, B), dtype=F32)
        right = np.empty((C, N + 1, B), dtype=F32)
        for n in range(N + 1):
            lvl = self.all_code_points[:, 2 ** n - 1: 2 ** (n + 1) - 1]
            last = 2 ** n - 1
            for c in range(C):
                g = lvl[c]
                r0 = np.searchsorted(g, Z[:, c], side="left")
                r = np.minimum(r0, last)
                l = np.maximum(r - 1, 0)
                if 0 < n < N:
                    l = np.where(r0 > last, last, l)
                if n == 0:
                    l = r = np.zeros(B, dtype=np.int64)
                right[c, n] = g[r]
                left[c, n] = g[l]
        return left, right

    def code_lengths(self, lambs):
        """(Lambda, N+1, C) float32 lengths in corrected mode, or (N+1,) int32 in raw mode.  quantizer.py:166-180."""
        N, C = self.N, self.C
        if not self.raw_code_length_entropy_models:
            return np.arange(N + 1, dtype=np.int32)
        raw = np.repeat(np.arange(N + 1, dtype=np.int32)[:, None], C, axis=1).astype(F32)
        return np.stack([raw + self.raw_code_length_entropy_models[l].T.astype(F32) for l in lambs])

    # quantizer.py:156-188 + utils.py:307-327,363-423
    def compress_batch_channel_latents(self, batch_means, batch_stds, lambs, fast_intervals=None, details=False):
        Z = np.asarray(batch_means, dtype=F32)
        S = np.asarray(batch_stds, dtype=F32)
        N = self.N
        B, C = Z.shape
        if fast_intervals is None:
            fast_intervals = self._search_grids is None
        left, right = (self.get_all_N_bit_intervals_fast if fast_intervals else self.get_all_N_bit_intervals)(Z)
        left = np.transpose(left, [1, 2, 0])
        right = np.transpose(right, [1, 2, 0])          # (N+1, B, C)
        P = np.concatenate([left, right[1:]], axis=0)   # (2N+1, B, C)   quantizer.py:183
        L = self.code_lengths(lambs)
        with np.errstate(divide="ignore", invalid="ignore"):
            fun_P = F32(-0.5) * ((P - Z) / S) ** 2      # utils.py:318-320, float32 throughout
        Z_hat_dict, bits_dict, det = {}, {}, {}
        cand_level = np.concatenate([np.arange(N + 1), np.arange(1, N + 1)])
        for i, lamb in enumerate(lambs):
            if L.ndim == 3:
                Ln = L[i]                                # (N+1, C) float32
                Lc = np.concatenate([Ln, Ln[1:]], axis=0)[:, None, :]   # (2N+1, 1, C)
            else:
                Lc = np.concatenate([L, L[1:]], axis=0)[:, None, None]  # int32
            pen = F32(lamb) * Lc.astype(F32)             # utils.py:388,393-396: lamb * cast(L, float32)
            scores = fun_P - pen
            k = np.argmax(scores, axis=0)                # first maximum, utils.py:401
            Z_hat = np.take_along_axis(P, k[None], axis=0)[0]
            bits = np.take_along_axis(np.broadcast_to(Lc, P.shape), k[None], axis=0)[0]
            Z_hat_dict[lamb] = Z_hat
            bits_dict[lamb] = bits
            if details:
                det[lamb] = dict(cand=k, level=cand_level[k], scores=scores, P=P)
        if details:
            return Z_hat_dict, bits_dict, det
        return Z_hat_dict, bits_dict

    def sorted_index(self, Z_hat):
        """I = searchsorted(code_points_by_channel, Z_hat^T) -> (B, C).  quantizer.py:135,223."""
        B, C = Z_hat.shape
        I = np.empty((B, C), dtype=np.int64)
        for c in range(C):
            I[:, c] = np.searchsorted(self.code_points_by_channel[c], Z_hat[:, c], side="left")
        return I

    def _stds(self, posterior_logvars, posterior_stds):
        """(rows, C) float32 sigma: exp(logvar) ** 0.5 in float32 (quantizer.py:93, :198), or the given stds."""
        if posterior_stds is not None:
            return np.asarray(posterior_stds, dtype=F32).reshape(-1, self.C)
        return np.exp(np.asarray(posterior_logvars, dtype=F32)).reshape(-1, self.C) ** F32(0.5)

    # quantizer.py:82-150, given latents instead of (X, vae)
    def build_entropy_models_from_latents(self, posterior_means, posterior_logvars, lambs, add_n_smoothing,
                                          posterior_stds=None):
        """``posterior_stds`` (optional) replaces ``posterior_logvars`` by ready-made standard deviations, as the
        facade's parameter of the same name does (e.g. the sigma the kernels derive from the log-variances)."""
        N, C = self.N, self.C
        means = np.asarray(posterior_means, dtype=F32).reshape(-1, C)
        stds = self._stds(posterior_logvars, posterior_stds)
        self.raw_code_length_entropy_models = None
        _, raw_bits = self.compress_batch_channel_latents(means, stds, lambs)
        rcl = {}
        for lamb in lambs:
            counts = np.array([np.bincount(raw_bits[lamb][:, c], minlength=N + 1) for c in range(C)], dtype=F32)
            counts += add_n_smoothing
            freqs = counts / np.sum(counts, axis=1)[:, None]
            rcl[lamb] = -np.log2(freqs)
        self.raw_code_length_entropy_models = rcl
        Z_hat_dict, _ = self.compress_batch_channel_latents(means, stds, lambs)
        em = {}
        for lamb in lambs:
            qidx = self.sorted_index(Z_hat_dict[lamb])
            assert np.array_equal(np.take_along_axis(self.code_points_by_channel.T, qidx, axis=0), Z_hat_dict[lamb])
            counts = np.array([np.bincount(qidx[:, c], minlength=self.Q) for c in range(C)], dtype=F32)
            counts += add_n_smoothing
            freqs = counts / np.sum(counts, axis=1)[:, None]
            em[lamb] = -np.log2(freqs)
        self.entropy_models = em

    # quantizer.py:190-240
    def compress_latents(self, posterior_means, posterior_logvars, lambs, posterior_stds=None):
        """``posterior_stds``: as in `build_entropy_models_from_latents`."""
        C = self.C
        pm = np.asarray(posterior_means, dtype=F32)
        assert pm.shape[-1] == C
        means = pm.reshape(-1, C)
        stds = self._stds(posterior_logvars, posterior_stds)
        Z_hat_dict, raw_dict = self.compress_batch_channel_latents(means, stds, lambs)
        keys = ("Z_hat", "raw_num_bits", "num_bits_cl", "num_bits")
        out = {k: {} for k in keys}
        for lamb in lambs:
            Z_hat = Z_hat_dict[lamb]
            I = self.sorted_index(Z_hat)
            out["Z_hat"][lamb] = Z_hat.reshape(pm.shape)
            out["raw_num_bits"][lamb] = raw_dict[lamb].reshape(pm.shape)
            if self.raw_code_length_entropy_models:
                out["num_bits_cl"][lamb] = raw_dict[lamb].reshape(pm.shape)
            if self.entropy_models:
                nb = np.take_along_axis(self.entropy_models[lamb].T, I, axis=0)
                out["num_bits"][lamb] = nb.reshape(pm.shape)
        return out


# ----------------------------------------------------------------------------------------------
# Parity helpers (north_star harness rules)
# ----------------------------------------------------------------------------------------------
def tie_mask(scores, rel=1e-6):
    """True where the best two candidates with *distinct* score differ by less than ``rel`` relative, or where the
    two best scores are equal: the coordinates the north_star reports separately.  ``scores``: (M, ...) objective
    values (higher is better)."""
    s = np.sort(scores, axis=0)
    top, second = s[-1], s[-2]
    with np.errstate(invalid="ignore"):
        gap = np.abs(top - second)
        return gap <= rel * np.maximum(np.abs(top), np.finfo(F32).tiny)


def rd_totals(Z, S, Z_hat, bits):
    """Per-lambda totals the sharding layer all-reduces (SURVEY.md §8e): total code length and total
    posterior-weighted squared error sum (z_hat-mu)^2/(2 sigma^2), float64."""
    d = (Z_hat.astype(np.float64) - Z.astype(np.float64)) / S.astype(np.float64)
    return float(np.sum(bits, dtype=np.float64)), float(0.5 * np.sum(d * d))


# ----------------------------------------------------------------------------------------------
# Generic forms used by the golden-vector tests
# ----------------------------------------------------------------------------------------------
def bracket_search_f64(mu, sigma, lamb, codepoints_heap, N):
    """Algorithm 1 in z-space, float64: maximise -0.5((z-mu)/sigma)^2 - lamb*n over the bracketing candidates of a
    single shared prior (what utils.encode_vectorized computes in xi-space, utils.py:263-304).  Returns
    (z_hat, num_bits)."""
    mu = np.asarray(mu, dtype=np.float64)
    sigma = np.asarray(sigma, dtype=np.float64)
    best = np.full(mu.shape, -np.inf)
    zhat = np.zeros(mu.shape)
    bits = np.zeros(mu.shape, dtype=np.int64)
    for n in range(N + 1):
        grid = codepoints_heap[2 ** n - 1: 2 ** (n + 1) - 1]
        r = np.clip(np.searchsorted(grid, mu, side="left"), 0, 2 ** n - 1)
        l = np.clip(r - 1, 0, 2 ** n - 1)
        for idx in (l, r):
            s = -0.5 * ((grid[idx] - mu) / sigma) ** 2 - lamb * n
            upd = s > best
            best = np.where(upd, s, best)
            zhat = np.where(upd, grid[idx], zhat)
            bits = np.where(upd, n, bits)
    return zhat, bits


def batch_quantize_indep_dims(P, L, loc, scale, lambs):
    """utils.batch_quantize_indep_dims (utils.py:363-423) for explicit candidates P, L of shape (M, B, K) and the
    float32 Gaussian `fun` of curry_normal_logpdf; returns dicts of (B, K) arrays."""
    P = np.asarray(P, dtype=F32)
    fun_P = F32(-0.5) * ((P - np.asarray(loc, dtype=F32)) / np.asarray(scale, dtype=F32)) ** 2
    Zh, nb = {}, {}
    for lamb in lambs:
        scores = fun_P - lamb * L
        k = np.argmax(scores, axis=0)
        Zh[lamb] = np.take_along_axis(P, k[None], axis=0)[0]
        nb[lamb] = np.take_along_axis(L, k[None], axis=0)[0]
    return Zh, nb


# ----------------------------------------------------------------------------------------------
# Symbol serialisation (SURVEY §8 f4): fixed-width bit packing and per-channel frequency tables
# ----------------------------------------------------------------------------------------------
def pack_indices(q, N):
    """n symbols of N+1 bits each, symbol k in bits [k(N+1), (k+1)(N+1)) (LSB first) of little-endian uint32 words.
    Plain-integer restatement of the format documented in include/vbq_b200.h."""
    q = np.asarray(q).reshape(-1).astype(np.uint64)
    B = N + 1
    n_words = (q.size * B + 31) // 32
    bits = ((q[:, None] >> np.arange(B, dtype=np.uint64)[None, :]) & np.uint64(1)).astype(np.uint8).reshape(-1)
    bits = np.concatenate([bits, np.zeros(n_words * 32 - bits.size, dtype=np.uint8)])
    weights = (np.uint64(1) << np.arange(32, dtype=np.uint64))
    return (bits.reshape(n_words, 32).astype(np.uint64) * weights[None, :]).sum(axis=1).astype(np.uint32)


def unpack_indices(words, n, N):
    B = N + 1
    w = np.asarray(words).astype(np.uint32)
    bits = ((w[:, None] >> np.arange(32, dtype=np.uint32)[None, :]) & np.uint32(1)).astype(np.uint64).reshape(-1)
    bits = bits[:n * B].reshape(n, B)
    return (bits * (np.uint64(1) << np.arange(B, dtype=np.uint64))[None, :]).sum(axis=1).astype(np.int32)


def symbol_histogram(q, Q):
    """quantizer.py:135-146: per-channel np.bincount of the sorted quantile indices, (rows, C) -> (C, Q)."""
    q = np.asarray(q)
    return np.stack([np.bincount(q[:, c], minlength=Q) for c in range(q.shape[1])]).astype(np.int64)
