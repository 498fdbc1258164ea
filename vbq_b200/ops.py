"""PyTorch custom ops (`torch.library`) over the C ABI of libvbq_b200.so.

PyTorch supplies device memory, the current stream and tracing metadata; all arithmetic happens in the
hand-written sm_100a kernels.  Every op raises if the library is missing or the tensors are not CUDA tensors:
there is deliberately no CPU implementation (north_star: "no CPU fallback")."""
from __future__ import annotations

import ctypes
from typing import List, Optional

import torch

from . import _lib

OUT_ZHAT = 1
OUT_QIDX = 2
OUT_LEVEL = 4
OUT_BITS = 8
OUT_EM_BITS = 16
OUT_TOTALS = 32

FLAG_LOGVAR = _lib.FLAG_LOGVAR
FLAG_NO_PRUNE = _lib.FLAG_NO_PRUNE
FLAG_FAST = _lib.FLAG_FAST
FLAG_NO_SWEEP = _lib.FLAG_NO_SWEEP
FLAG_REFERENCE_WALK = _lib.FLAG_REFERENCE_WALK
FLAG_RESERVE_SM = _lib.FLAG_RESERVE_SM
FLAG_BRACKET_WALK = _lib.FLAG_BRACKET_WALK
FLAG_WORKSPACE_ZEROED = _lib.FLAG_WORKSPACE_ZEROED
FLAG_NO_TMA = _lib.FLAG_NO_TMA
FLAG_TABLE_STABLE = _lib.FLAG_TABLE_STABLE
FLAG_NEIGHBOUR_EVERY_DEPTH = _lib.FLAG_NEIGHBOUR_EVERY_DEPTH


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None or t.numel() == 0 else t.data_ptr()


def _stream(device):
    return torch.cuda.current_stream(device).cuda_stream


def _need_cuda(name, t, dtype, ndim=None):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise RuntimeError("vbq_b200: `%s` must be a CUDA tensor (no CPU fallback exists)" % name)
    if t.dtype != dtype:
        raise TypeError("vbq_b200: `%s` must be %s, got %s" % (name, dtype, t.dtype))
    if not t.is_contiguous():
        raise ValueError("vbq_b200: `%s` must be contiguous" % name)
    if ndim is not None and t.dim() != ndim:
        raise ValueError("vbq_b200: `%s` must be %d-D, got shape %s" % (name, ndim, tuple(t.shape)))


_HOST_COPIES = {}     # device pointer of a penalty table -> its host original (dropped when the device tensor dies)
_STABLE_TABLES = set()    # device pointers of packed tables that are known to be complete (see stable_packed)


def with_host_copy(penalty_np, device):
    """Device tensor of a host-made penalty table that remembers its host original (float32, C-contiguous).  The
    search kernels take the penalties of the TMA kernels from the host copy (launch constants / validation,
    vbq_quantize_hp); the device tensor alone works too (other kernels).  The association is by device address, so it
    survives the re-wrapping of tensors by torch.library."""
    import weakref
    import numpy as np
    host = np.ascontiguousarray(penalty_np, dtype=np.float32)
    t = torch.from_numpy(host).to(device)
    key = (t.data_ptr(), tuple(t.shape))
    _HOST_COPIES[key] = host
    weakref.finalize(t, _HOST_COPIES.pop, key, None)
    return t


def _host_penalty_ptr(penalty):
    host = _HOST_COPIES.get((penalty.data_ptr(), tuple(penalty.shape)))
    return None if host is None else host.ctypes.data


def stable_packed(packed):
    """Mark a packed table as complete: the caller has synchronized since vbq_pack_code_points wrote it, so the search
    kernels may read it before earlier kernels of the stream have finished (VBQ_FLAG_TABLE_STABLE).  Returns `packed`."""
    import weakref
    key = packed.data_ptr()
    _STABLE_TABLES.add(key)
    weakref.finalize(packed, _STABLE_TABLES.discard, key)
    return packed


def _table_flags(packed, flags):
    return flags | FLAG_TABLE_STABLE if packed.data_ptr() in _STABLE_TABLES else flags


def search_flags(lambs, flags=0):
    """Flags the facade passes to vbq_quantize for a list of rate-distortion trade-offs.  The sound early exit
    ("every deeper score is <= -penalty") only pays off when the penalty grows quickly with depth; for small lambdas
    the walk reaches the bottom anyway and the exit tests are pure overhead, so they are compiled out.  Results are
    identical either way (tests/test_gpu_parity.py::test_prune_equals_no_prune_large)."""
    if len(lambs) == 1 and float(lambs[0]) < 1.0:
        flags |= FLAG_NO_PRUNE
    return flags


def num_levels(max_bits: int) -> int:
    return 2 ** (max_bits + 1) - 1


# ------------------------------------------------------------------------------------------------------
# raw call with caller-owned outputs (used by the op below and by the benchmark's preallocated plan)
# ------------------------------------------------------------------------------------------------------
def quantize_into(mu, sigma, table, packed, penalty, length, entropy_model, max_bits,
                  zhat=None, qidx=None, level=None, bits=None, em_bits=None, totals=None,
                  workspace=None, flags=0):
    """Direct vbq_quantize call.  Outputs are (n_lambda, rows, C) tensors or None; see include/vbq_b200.h."""
    lib = _lib.load()
    _need_cuda("mu", mu, torch.float32, 2)
    _need_cuda("sigma", sigma, torch.float32, 2)
    _need_cuda("table", table, torch.float32, 2)
    _need_cuda("packed", packed, torch.float32)
    _need_cuda("penalty", penalty, torch.float32, 3)
    if mu.shape != sigma.shape:
        raise ValueError("vbq_b200: mu %s and sigma %s differ in shape" % (tuple(mu.shape), tuple(sigma.shape)))
    rows, C = mu.shape
    Q = num_levels(max_bits)
    if tuple(table.shape) != (C, Q):
        raise ValueError("vbq_b200: table must be (C=%d, Q=%d), got %s" % (C, Q, tuple(table.shape)))
    n_lambda, pen_channels, n1 = penalty.shape
    if n1 != max_bits + 1 or pen_channels not in (1, C):
        raise ValueError("vbq_b200: penalty must be (n_lambda, 1 or C, N+1), got %s" % (tuple(penalty.shape),))
    if packed.numel() != lib.vbq_packed_table_floats(C, max_bits):
        raise ValueError("vbq_b200: packed table has the wrong size")
    if length is not None:
        _need_cuda("length", length, torch.float32, 3)
        if length.shape != penalty.shape:
            raise ValueError("vbq_b200: length must have the shape of penalty")
    if entropy_model is not None:
        _need_cuda("entropy_model", entropy_model, torch.float32, 3)
        if tuple(entropy_model.shape) != (n_lambda, C, Q):
            raise ValueError("vbq_b200: entropy_model must be (n_lambda, C, Q)")
    for name, t, dt in (("zhat", zhat, torch.float32), ("qidx", qidx, torch.int32), ("level", level, torch.int32),
                        ("bits", bits, torch.float32), ("em_bits", em_bits, torch.float32)):
        if t is not None:
            _need_cuda(name, t, dt)
            if tuple(t.shape) != (n_lambda, rows, C):
                raise ValueError("vbq_b200: `%s` must be (n_lambda, rows, C)" % name)
    ws_bytes = 0
    if totals is not None:
        _need_cuda("totals", totals, torch.float64)
        if tuple(totals.shape) != (n_lambda, _lib.TOTALS):
            raise ValueError("vbq_b200: totals must be (n_lambda, %d)" % _lib.TOTALS)
        if workspace is None:
            raise ValueError("vbq_b200: totals need a workspace (see quantize_workspace)")
        ws_bytes = workspace.numel() * workspace.element_size()
    for name, t in (("sigma", sigma), ("table", table), ("packed", packed), ("penalty", penalty), ("length", length),
                    ("entropy_model", entropy_model), ("zhat", zhat), ("qidx", qidx), ("level", level), ("bits", bits),
                    ("em_bits", em_bits), ("totals", totals), ("workspace", workspace)):
        if t is not None and t.device != mu.device:
            raise ValueError("vbq_b200: `%s` lives on %s but `mu` on %s" % (name, t.device, mu.device))
    with torch.cuda.device(mu.device):   # the library launches on the CURRENT device
        st = lib.vbq_quantize_hp(_ptr(mu), _ptr(sigma), rows, C, _ptr(table), _ptr(packed), max_bits,
                                 _ptr(penalty), _host_penalty_ptr(penalty), _ptr(length), n_lambda, pen_channels,
                                 _ptr(entropy_model), _ptr(zhat), _ptr(qidx), _ptr(level), _ptr(bits), _ptr(em_bits),
                                 _ptr(totals), _ptr(workspace), ws_bytes, _table_flags(packed, flags), _stream(mu.device))
    _lib.check(st, "vbq_quantize_hp")


def quantize_workspace(n_lambda, device):
    """Zero-filled totals workspace.  Calls leave its ticket counters zero again, so a workspace from this function
    may always be passed together with FLAG_WORKSPACE_ZEROED (quantize_into does so when `workspace_zeroed`)."""
    n = _lib.load().vbq_quantize_workspace_bytes(n_lambda)
    return torch.zeros((n + 7) // 8, dtype=torch.float64, device=device)


class QuantizePlan:
    """A vbq_quantize call with caller-owned, fixed buffers, validated once.  `run()` re-issues it on the current
    stream with one prebound C call (no Python-side checks); back-to-back runs overlap their launch latency through
    programmatic dependent launch inside the library.  `graph=True` captures the call into a CUDA graph instead and
    replays it (one cudaGraphLaunch per run)."""

    def __init__(self, mu, sigma, table, packed, penalty, length, entropy_model, max_bits, zhat=None, qidx=None,
                 level=None, bits=None, em_bits=None, totals=None, flags=0, graph=False, peer=None):
        self.totals = totals
        self._peer = peer          # sharding.PeerTotals: run(seq) also delivers the totals to every rank's inbox
        self._device = mu.device
        ws = quantize_workspace(penalty.shape[0], mu.device) if totals is not None else None
        self._keep = (mu, sigma, table, packed, penalty, length, entropy_model, zhat, qidx, level, bits, em_bits, totals, ws)
        self._args = (mu, sigma, table, packed, penalty, length, entropy_model, max_bits)
        self._kw = dict(zhat=zhat, qidx=qidx, level=level, bits=bits, em_bits=em_bits, totals=totals, workspace=ws,
                        flags=flags | (FLAG_WORKSPACE_ZEROED if ws is not None else 0))
        quantize_into(*self._args, **self._kw)     # validates everything once (and sets the kernels' attributes)
        rows, C = mu.shape
        n_lambda, pen_channels, _ = penalty.shape
        self._fn = _lib.load().vbq_quantize_hp
        self._cargs = (_ptr(mu), _ptr(sigma), rows, C, _ptr(table), _ptr(packed), max_bits, _ptr(penalty),
                       _host_penalty_ptr(penalty),
                       _ptr(length), n_lambda, pen_channels, _ptr(entropy_model), _ptr(zhat), _ptr(qidx), _ptr(level),
                       _ptr(bits), _ptr(em_bits), _ptr(totals), _ptr(ws),
                       0 if ws is None else ws.numel() * ws.element_size(), _table_flags(packed, self._kw["flags"]))
        self._graph = None
        if graph:
            torch.cuda.synchronize(mu.device)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self._call()
            self._graph = g

    def _call(self):
        if torch.cuda.current_device() != self._device.index:
            with torch.cuda.device(self._device):
                st = self._fn(*self._cargs, _stream(self._device))
        else:
            st = self._fn(*self._cargs, _stream(self._device))
        if st != _lib.OK:
            _lib.check(st, "vbq_quantize_hp")

    def run_peer(self, push_seq=0, push_totals=None, collect_seq=0, collected=None):
        """The call, which also delivers the completed totals of an earlier call (`push_totals`, sequence number
        `push_seq`) to every rank and collects the all-reduced totals of call `collect_seq` into `collected`
        (sharding.PeerTotals; include/vbq_b200.h vbq_quantize_peer)."""
        st = self._peer._lib.vbq_quantize_peer(*self._cargs, _stream(self._device), self._peer._h, int(push_seq),
                                               _ptr(push_totals), int(collect_seq), _ptr(collected))
        if st != _lib.OK:
            _lib.check(st, "vbq_quantize_peer")

    def run(self):
        if self._graph is not None:
            self._graph.replay()
        else:
            self._call()
        return self.totals


# ------------------------------------------------------------------------------------------------------
# torch.library custom ops
# ------------------------------------------------------------------------------------------------------
@torch.library.custom_op("vbq::quantize", mutates_args=())
def quantize(mu: torch.Tensor, sigma: torch.Tensor, table: torch.Tensor, packed: torch.Tensor,
             penalty: torch.Tensor, length: Optional[torch.Tensor], entropy_model: Optional[torch.Tensor],
             max_bits: int, outputs: int, flags: int) -> List[torch.Tensor]:
    """Rate-distortion search for every coordinate and every lambda.

    Returns [zhat f32, qidx i32, level i32, bits f32, em_bits f32, totals f64]; entries whose OUT_* bit is not
    set in ``outputs`` are empty tensors."""
    rows, C = mu.shape
    L = penalty.shape[0]
    dev = mu.device

    def alloc(bit, dtype):
        return torch.empty((L, rows, C), dtype=dtype, device=dev) if outputs & bit else None

    zhat = alloc(OUT_ZHAT, torch.float32)
    qidx = alloc(OUT_QIDX, torch.int32)
    level = alloc(OUT_LEVEL, torch.int32)
    bits = alloc(OUT_BITS, torch.float32)
    em_bits = alloc(OUT_EM_BITS, torch.float32)
    totals = ws = None
    if outputs & OUT_TOTALS:
        totals = torch.empty((L, _lib.TOTALS), dtype=torch.float64, device=dev)
        ws = quantize_workspace(L, dev)
    quantize_into(mu, sigma, table, packed, penalty, length, entropy_model, max_bits,
                  zhat, qidx, level, bits, em_bits, totals, ws, flags)
    empty = lambda dt: torch.empty(0, dtype=dt, device=dev)  # noqa: E731
    return [zhat if zhat is not None else empty(torch.float32),
            qidx if qidx is not None else empty(torch.int32),
            level if level is not None else empty(torch.int32),
            bits if bits is not None else empty(torch.float32),
            em_bits if em_bits is not None else empty(torch.float32),
            totals if totals is not None else empty(torch.float64)]


@quantize.register_fake
def _(mu, sigma, table, packed, penalty, length, entropy_model, max_bits, outputs, flags):
    rows, C = mu.shape
    L = penalty.shape[0]

    def shp(bit):
        return (L, rows, C) if outputs & bit else (0,)

    return [mu.new_empty(shp(OUT_ZHAT)), mu.new_empty(shp(OUT_QIDX), dtype=torch.int32),
            mu.new_empty(shp(OUT_LEVEL), dtype=torch.int32), mu.new_empty(shp(OUT_BITS)),
            mu.new_empty(shp(OUT_EM_BITS)),
            mu.new_empty((L, _lib.TOTALS) if outputs & OUT_TOTALS else (0,), dtype=torch.float64)]


@torch.library.custom_op("vbq::learned_cdf", mutates_args=())
def learned_cdf(params: torch.Tensor, x: torch.Tensor) -> torch.Tensor:
    """BMSHJ2018Prior.cdf on (rows, C) channel-last float32 (learned_prior.py:109-148)."""
    _need_cuda("params", params, torch.float32, 2)
    _need_cuda("x", x, torch.float32, 2)
    C = params.shape[0]
    if params.shape[1] != _lib.PRIOR_PARAMS or x.shape[1] != C:
        raise ValueError("vbq_b200: params must be (C, 43) and x (rows, C)")
    out = torch.empty_like(x)
    st = _lib.load().vbq_learned_cdf(_ptr(params), C, _ptr(x), x.shape[0], _ptr(out), _stream(x.device))
    _lib.check(st, "vbq_learned_cdf")
    return out


@learned_cdf.register_fake
def _(params, x):
    return torch.empty_like(x)


@torch.library.custom_op("vbq::learned_inverse_cdf", mutates_args=())
def learned_inverse_cdf(params: torch.Tensor, xi: torch.Tensor) -> torch.Tensor:
    """BMSHJ2018Prior.inverse_cdf: xi (rows, C) float64 -> float32 (learned_prior.py:173-218)."""
    _need_cuda("params", params, torch.float32, 2)
    _need_cuda("xi", xi, torch.float64, 2)
    C = params.shape[0]
    if params.shape[1] != _lib.PRIOR_PARAMS or xi.shape[1] != C:
        raise ValueError("vbq_b200: params must be (C, 43) and xi (rows, C)")
    out = torch.empty(xi.shape, dtype=torch.float32, device=xi.device)
    st = _lib.load().vbq_learned_inverse_cdf(_ptr(params), C, _ptr(xi), xi.shape[0], _ptr(out), _stream(xi.device))
    _lib.check(st, "vbq_learned_inverse_cdf")
    return out


@learned_inverse_cdf.register_fake
def _(params, xi):
    return xi.new_empty(xi.shape, dtype=torch.float32)


@torch.library.custom_op("vbq::gaussian_inverse_cdf", mutates_args=())
def gaussian_inverse_cdf(xi: torch.Tensor, mean: Optional[torch.Tensor], std: Optional[torch.Tensor]) -> torch.Tensor:
    """norm.ppf(xi, loc=mean, scale=std) in float64; xi (rows, C) (vae_models.py:23-25,40-43; ipynb:385)."""
    _need_cuda("xi", xi, torch.float64, 2)
    C = xi.shape[1]
    for name, t in (("mean", mean), ("std", std)):
        if t is not None:
            _need_cuda(name, t, torch.float64, 1)
            if t.shape[0] != C:
                raise ValueError("vbq_b200: `%s` must have C=%d entries" % (name, C))
    out = torch.empty_like(xi)
    st = _lib.load().vbq_gaussian_inverse_cdf(_ptr(mean), _ptr(std), C, _ptr(xi), xi.shape[0], _ptr(out),
                                              _stream(xi.device))
    _lib.check(st, "vbq_gaussian_inverse_cdf")
    return out


@gaussian_inverse_cdf.register_fake
def _(xi, mean, std):
    return torch.empty_like(xi)


@torch.library.custom_op("vbq::build_code_points_learned", mutates_args=())
def build_code_points_learned(params: torch.Tensor, max_bits: int) -> torch.Tensor:
    """(C, Q) heap-order code-point table of a learned prior (quantizer.py:25-36)."""
    _need_cuda("params", params, torch.float32, 2)
    C = params.shape[0]
    out = torch.empty((C, num_levels(max_bits)), dtype=torch.float32, device=params.device)
    st = _lib.load().vbq_build_code_points_learned(_ptr(params), C, max_bits, _ptr(out), _stream(params.device))
    _lib.check(st, "vbq_build_code_points_learned")
    return out


@build_code_points_learned.register_fake
def _(params, max_bits):
    return params.new_empty((params.shape[0], num_levels(max_bits)))


@torch.library.custom_op("vbq::build_code_points_gaussian", mutates_args=())
def build_code_points_gaussian(mean: torch.Tensor, std: torch.Tensor, max_bits: int) -> torch.Tensor:
    """(C, Q) heap-order code-point table of per-channel Gaussians N(mean[c], std[c]^2)."""
    _need_cuda("mean", mean, torch.float64, 1)
    _need_cuda("std", std, torch.float64, 1)
    C = mean.shape[0]
    out = torch.empty((C, num_levels(max_bits)), dtype=torch.float32, device=mean.device)
    st = _lib.load().vbq_build_code_points_gaussian(_ptr(mean), _ptr(std), C, max_bits, _ptr(out),
                                                    _stream(mean.device))
    _lib.check(st, "vbq_build_code_points_gaussian")
    return out


@build_code_points_gaussian.register_fake
def _(mean, std, max_bits):
    return mean.new_empty((mean.shape[0], num_levels(max_bits)), dtype=torch.float32)


@torch.library.custom_op("vbq::pack_code_points", mutates_args=())
def pack_code_points(table: torch.Tensor, max_bits: int) -> torch.Tensor:
    """Shared-memory image of the table: (groups, min(Q, 2047), 16) (include/vbq_b200.h)."""
    _need_cuda("table", table, torch.float32, 2)
    C = table.shape[0]
    lib = _lib.load()
    out = torch.empty(lib.vbq_packed_table_floats(C, max_bits), dtype=torch.float32, device=table.device)
    st = lib.vbq_pack_code_points(_ptr(table), C, max_bits, _ptr(out), _stream(table.device))
    _lib.check(st, "vbq_pack_code_points")
    return out


@pack_code_points.register_fake
def _(table, max_bits):
    C = table.shape[0]
    g = (C + _lib.GROUP - 1) // _lib.GROUP
    return table.new_empty(g * min(num_levels(max_bits), 2047) * _lib.GROUP)


def selftest_divide(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    _need_cuda("a", a, torch.float32)
    _need_cuda("b", b, torch.float32)
    out = torch.empty_like(a)
    st = _lib.load().vbq_selftest_divide(_ptr(a), _ptr(b), a.numel(), _ptr(out), _stream(a.device))
    _lib.check(st, "vbq_selftest_divide")
    return out


def selftest_sigma_from_logvar(lv: torch.Tensor) -> torch.Tensor:
    """The sigma the search kernels derive from log-variances `lv` (FLAG_LOGVAR), bit for bit."""
    _need_cuda("lv", lv, torch.float32)
    out = torch.empty_like(lv)
    st = _lib.load().vbq_selftest_sigma_from_logvar(_ptr(lv), lv.numel(), _ptr(out), _stream(lv.device))
    _lib.check(st, "vbq_selftest_sigma_from_logvar")
    return out


# ------------------------------------------------------------------------------------------------------
# host-resident latents: chunked upload / kernel / download pipeline (vbq_quantize_host)
# ------------------------------------------------------------------------------------------------------
def _host_ptr(x, dtype, shape, name):
    """Pointer of a contiguous CPU tensor / ndarray (pinned memory recommended); None passes through."""
    if x is None:
        return None
    t = x if isinstance(x, torch.Tensor) else torch.from_numpy(x)
    if t.is_cuda:
        raise RuntimeError("vbq_b200: `%s` must live in host memory for the host pipeline" % name)
    if t.dtype != dtype or not t.is_contiguous() or tuple(t.shape) != tuple(shape):
        raise ValueError("vbq_b200: `%s` must be a contiguous %s host array of shape %s" % (name, dtype, tuple(shape)))
    return t.data_ptr()


class HostPipeline:
    """Owns a `vbq_host_ctx`: three device staging slots + three streams.  `run` quantizes host arrays chunk by
    chunk with upload, kernel and download overlapped, and returns when the results are in host memory."""

    def __init__(self, num_channels, max_bits, n_lambda, chunk_rows, outputs, device=None):
        import ctypes
        self._lib = _lib.load()
        self.C, self.N, self.L = int(num_channels), int(max_bits), int(n_lambda)
        self.outputs = int(outputs)
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        handle = ctypes.c_void_p()
        with torch.cuda.device(self.device):
            st = self._lib.vbq_host_ctx_create(self.C, self.N, self.L, int(chunk_rows), self.outputs,
                                               ctypes.byref(handle))
        _lib.check(st, "vbq_host_ctx_create")
        self._h = handle

    def run(self, h_mu, h_sigma, table, packed, penalty, length=None, entropy_model=None, zhat=None, qidx=None,
            level=None, bits=None, em_bits=None, totals=None, flags=0):
        if self._h is None:
            raise RuntimeError("vbq_b200: HostPipeline is closed")
        rows = int(h_mu.shape[0])
        L, C = self.L, self.C
        _need_cuda("table", table, torch.float32, 2)
        _need_cuda("packed", packed, torch.float32)
        _need_cuda("penalty", penalty, torch.float32, 3)
        if penalty.shape[0] != L or penalty.shape[2] != self.N + 1 or penalty.shape[1] not in (1, C):
            raise ValueError("vbq_b200: penalty must be (n_lambda, 1 or C, N+1)")
        o = (L, rows, C)
        with torch.cuda.device(self.device):
            # the pipeline runs on its own streams: whatever produced the tables on this thread's stream has to be done
            torch.cuda.current_stream(self.device).synchronize()
            st = self._lib.vbq_quantize_host(
                self._h, _host_ptr(h_mu, torch.float32, (rows, C), "h_mu"),
                _host_ptr(h_sigma, torch.float32, (rows, C), "h_sigma"), rows, _ptr(table), _ptr(packed),
                _ptr(penalty), _ptr(length), int(penalty.shape[1]), _ptr(entropy_model),
                _host_ptr(zhat, torch.float32, o, "zhat"), _host_ptr(qidx, torch.int32, o, "qidx"),
                _host_ptr(level, torch.int32, o, "level"), _host_ptr(bits, torch.float32, o, "bits"),
                _host_ptr(em_bits, torch.float32, o, "em_bits"),
                _host_ptr(totals, torch.float64, (L, _lib.TOTALS), "totals"), _table_flags(packed, flags))
        _lib.check(st, "vbq_quantize_host")

    def close(self):
        if getattr(self, "_h", None) is not None:
            self._lib.vbq_host_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# ------------------------------------------------------------------------------------------------------
# stand-alone operator forms
# ------------------------------------------------------------------------------------------------------
@torch.library.custom_op("vbq::intervals", mutates_args=())
def intervals(mu: torch.Tensor, table: torch.Tensor, max_bits: int) -> List[torch.Tensor]:
    """get_all_N_bit_intervals (quantizer.py:65-80): mu (B, C) -> [left, right], each (C, N+1, B)."""
    _need_cuda("mu", mu, torch.float32, 2)
    _need_cuda("table", table, torch.float32, 2)
    rows, C = mu.shape
    if tuple(table.shape) != (C, num_levels(max_bits)):
        raise ValueError("vbq_b200: table must be (C, Q)")
    left = torch.empty((C, max_bits + 1, rows), dtype=torch.float32, device=mu.device)
    right = torch.empty_like(left)
    st = _lib.load().vbq_intervals(_ptr(mu), rows, C, _ptr(table), max_bits, _ptr(left), _ptr(right),
                                   _stream(mu.device))
    _lib.check(st, "vbq_intervals")
    return [left, right]


@intervals.register_fake
def _(mu, table, max_bits):
    rows, C = mu.shape
    e = mu.new_empty((C, max_bits + 1, rows))
    return [e, e.clone()]


def argmax_candidates(P, L, lambs, fun_P=None, loc=None, scale=None):
    """utils.batch_quantize_indep_dims on device tensors: P (M, B, K) float32, L (M, B, K) or (Lambda, M, B, K)
    int32/float32, and either fun_P (M, B, K) or loc/scale (B, K).  Returns (zhat (Lambda,B,K), bits, index)."""
    _need_cuda("P", P, torch.float32, 3)
    M, B, K = P.shape
    if L.dtype not in (torch.int32, torch.float32):
        raise TypeError("vbq_b200: code lengths must be int32 or float32")
    _need_cuda("L", L, L.dtype)
    per_lambda = L.dim() == 4
    n_lambda = len(lambs)
    if tuple(L.shape) != (((n_lambda,) if per_lambda else ()) + (M, B, K)):
        raise ValueError("vbq_b200: L must be (M,B,K) or (n_lambda,M,B,K)")
    lam = torch.tensor([float(l) for l in lambs], dtype=torch.float32, device=P.device)
    if fun_P is not None:
        _need_cuda("fun_P", fun_P, torch.float32, 3)
    else:
        _need_cuda("loc", loc, torch.float32, 2)
        _need_cuda("scale", scale, torch.float32, 2)
    zhat = torch.empty((n_lambda, B, K), dtype=torch.float32, device=P.device)
    bits = torch.empty((n_lambda, B, K), dtype=L.dtype, device=P.device)
    index = torch.empty((n_lambda, B, K), dtype=torch.int32, device=P.device)
    st = _lib.load().vbq_argmax_candidates(_ptr(P), _ptr(L), int(L.dtype == torch.float32), int(per_lambda),
                                           _ptr(fun_P), _ptr(loc), _ptr(scale), _ptr(lam), n_lambda, M, B * K,
                                           _ptr(zhat), _ptr(bits), _ptr(index), _stream(P.device))
    _lib.check(st, "vbq_argmax_candidates")
    return zhat, bits, index


def compress_coordinates_f64(mu, sigma, codepoints, lengths, beta, pen_f32=True, want_index=False, want_level=False):
    """The notebook's float64 search (vbq_compress_coordinates_f64): mu, sigma float32 CUDA tensors of equal shape,
    codepoints (Q,) float64 heap order, lengths (N+1,) float64.  Returns (optima float32, heap index, level)."""
    _need_cuda("mu", mu, torch.float32)
    _need_cuda("sigma", sigma, torch.float32)
    _need_cuda("codepoints", codepoints, torch.float64, 1)
    _need_cuda("lengths", lengths, torch.float64, 1)
    N = lengths.numel() - 1
    if codepoints.numel() != num_levels(N) or mu.shape != sigma.shape:
        raise ValueError("vbq_b200: codepoints must have 2^(N+1)-1 entries and mu/sigma equal shapes")
    optima = torch.empty_like(mu)
    index = torch.empty(mu.shape, dtype=torch.int32, device=mu.device) if want_index else None
    level = torch.empty(mu.shape, dtype=torch.int32, device=mu.device) if want_level else None
    st = _lib.load().vbq_compress_coordinates_f64(_ptr(mu), _ptr(sigma), mu.numel(), _ptr(codepoints), N,
                                                  _ptr(lengths), float(beta), int(bool(pen_f32)), _ptr(optima),
                                                  _ptr(index), _ptr(level), _stream(mu.device))
    _lib.check(st, "vbq_compress_coordinates_f64")
    return optima, index, level


# ------------------------------------------------------------------------------------------------------
# after the search: symbols for an external entropy coder (include/vbq_b200.h, SURVEY §8 f4)
# ------------------------------------------------------------------------------------------------------
def packed_index_words(n: int, max_bits: int) -> int:
    return int(_lib.load().vbq_packed_index_words(int(n), int(max_bits)))


def pack_indices(qidx: torch.Tensor, max_bits: int) -> torch.Tensor:
    """Sorted quantile indices (any shape, int32, CUDA) -> bit stream of max_bits+1 bits per symbol as int32 words."""
    _need_cuda("qidx", qidx, torch.int32)
    q = qidx.contiguous().reshape(-1)
    words = torch.empty(packed_index_words(q.numel(), max_bits), dtype=torch.int32, device=q.device)
    st = _lib.load().vbq_pack_indices(_ptr(q), q.numel(), max_bits, _ptr(words), _stream(q.device))
    _lib.check(st, "vbq_pack_indices")
    return words


def unpack_indices(words: torch.Tensor, n: int, max_bits: int) -> torch.Tensor:
    """Inverse of pack_indices: the first n symbols of the stream as a flat int32 tensor."""
    _need_cuda("words", words, torch.int32, 1)
    if words.numel() < packed_index_words(n, max_bits):
        raise ValueError("vbq_b200: %d words cannot hold %d symbols of %d bits" % (words.numel(), n, max_bits + 1))
    q = torch.empty(int(n), dtype=torch.int32, device=words.device)
    st = _lib.load().vbq_unpack_indices(_ptr(words.contiguous()), int(n), max_bits, _ptr(q), _stream(words.device))
    _lib.check(st, "vbq_unpack_indices")
    return q


def symbol_histogram(qidx: torch.Tensor, max_bits: int, counts: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Per-channel frequency tables of the sorted quantile indices (rows, C) -> (C, Q) int64 counts
    (quantizer.py:135-146 builds them with np.bincount per channel).  `counts` accumulates when given."""
    _need_cuda("qidx", qidx, torch.int32, 2)
    rows, C = qidx.shape
    Q = num_levels(max_bits)
    if counts is None:
        counts = torch.zeros((C, Q), dtype=torch.int64, device=qidx.device)
    else:
        _need_cuda("counts", counts, torch.int64, 2)
        if tuple(counts.shape) != (C, Q):
            raise ValueError("vbq_b200: counts must be (C, Q)")
    st = _lib.load().vbq_symbol_histogram(_ptr(qidx.contiguous()), rows, C, max_bits, _ptr(counts),
                                          _stream(qidx.device))
    _lib.check(st, "vbq_symbol_histogram")
    return counts


# ------------------------------------------------------------------------------------------------------
# entropy coding: interleaved rANS over (item, row segment, 32-channel group) groups (include/vbq_b200.h, csrc/rans.cu)
# ------------------------------------------------------------------------------------------------------
def rans_payload_bound(n_planes: int, items: int, item_rows: int, C: int, seg_rows: int) -> int:
    return int(_lib.load().vbq_rans_payload_bound(n_planes, items, item_rows, C, seg_rows))


def rans_encode(qidx: torch.Tensor, cum: torch.Tensor, max_bits: int, prob_bits: int, seg_rows: int):
    """qidx (n_planes, items, item_rows, C) int32 and cum (n_planes, C, Q) int16 (the uint16 cum tables of
    coding.cum_table) -> (payload int16 words of vbq_rans_payload_bound bytes, payload size in bytes as a 1-element
    int64 tensor, status int32 tensor): one launch for all planes, no synchronisation."""
    _need_cuda("qidx", qidx, torch.int32, 4)
    _need_cuda("cum", cum, torch.int16, 3)
    n_planes, items, item_rows, C = qidx.shape
    lib = _lib.load()
    bound = lib.vbq_rans_payload_bound(n_planes, items, item_rows, C, seg_rows)
    ws_bytes = lib.vbq_rans_workspace_bytes(n_planes, items, item_rows, C, seg_rows)
    if bound < 0 or ws_bytes < 0:
        raise ValueError("vbq_b200: bad rANS shape: %s" % lib.vbq_last_error().decode())
    dev = qidx.device
    payload = torch.empty(max(1, bound // 2), dtype=torch.int16, device=dev)
    size = torch.zeros(1, dtype=torch.int64, device=dev)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    ws = torch.empty(max(1, ws_bytes), dtype=torch.uint8, device=dev)
    st = lib.vbq_rans_encode(_ptr(qidx), n_planes, items, item_rows, C, seg_rows, max_bits, prob_bits, _ptr(cum),
                             payload.data_ptr(), bound, size.data_ptr(), status.data_ptr(), ws.data_ptr(), ws_bytes,
                             _stream(dev))
    _lib.check(st, "vbq_rans_encode")
    return payload, size, status


def rans_decode(words: torch.Tensor, bounds: torch.Tensor, cum: torch.Tensor, items: int, item_rows: int,
                seg_rows: int, max_bits: int, prob_bits: int, code_points: Optional[torch.Tensor] = None,
                want_qidx: bool = True):
    """words: the payload as int16 words; bounds (n_planes * groups, 2) int64 word ranges of the groups; cum
    (n_planes, C, Q) int16.  Returns (qidx or None, zhat or None, status): (n_planes, items, item_rows, C) int32 symbols
    and float32 code_points[c, q] (code_points (C, Q) ascending), and the int32 device status (0 = every group passed
    the integrity check)."""
    _need_cuda("words", words, torch.int16, 1)
    _need_cuda("bounds", bounds, torch.int64, 2)
    _need_cuda("cum", cum, torch.int16, 3)
    n_planes, C, _ = cum.shape
    dev = words.device
    shape = (n_planes, items, item_rows, C)
    q = torch.empty(shape, dtype=torch.int32, device=dev) if want_qidx else None
    z = None
    if code_points is not None:
        _need_cuda("code_points", code_points, torch.float32, 2)
        z = torch.empty(shape, dtype=torch.float32, device=dev)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    st = _lib.load().vbq_rans_decode(_ptr(words), words.numel(), _ptr(bounds), n_planes, items, item_rows, C,
                                     seg_rows, max_bits, prob_bits, _ptr(cum), _ptr(code_points), _ptr(q), _ptr(z),
                                     status.data_ptr(), _stream(dev))
    _lib.check(st, "vbq_rans_decode")
    return q, z, status


BATCH_UNIT_FIELDS = 7       # vbq_rans_batch_unit: start, end, out, rows, table, cg, blob (int64 each)
BATCH_CTA_FIELDS = 4        # vbq_rans_batch_cta: first, count, table, cg (int64 each)


def rans_decode_batch(words: torch.Tensor, cum: torch.Tensor, prob_bits: torch.Tensor, units: torch.Tensor,
                      ctas: torch.Tensor, n_blobs: int, max_bits: int, n_out: int,
                      code_points: Optional[torch.Tensor] = None, want_qidx: bool = True):
    """The work-list decoder of many VBQ2 streams in one launch.  words: the payloads as int16 words; cum (n_tables,
    C, Q) int16; prob_bits (n_tables,) int32; units (n_units, 7) and ctas (n_ctas, 4) int64 (vbq_rans_batch_unit /
    vbq_rans_batch_cta).  Returns (qidx or None, zhat or None, status): flat (n_out,) int32 symbols and float32
    code_points[c, q] (code_points (C, Q) ascending), and the (n_blobs,) int32 device status per blob (bits 1, 2, 4 of
    rans_decode, 8 for a bad unit).  No synchronisation."""
    for name, t, dt, nd in (("words", words, torch.int16, 1), ("cum", cum, torch.int16, 3),
                            ("prob_bits", prob_bits, torch.int32, 1), ("units", units, torch.int64, 2),
                            ("ctas", ctas, torch.int64, 2)):
        _need_cuda(name, t, dt, nd)
    if units.shape[1] != BATCH_UNIT_FIELDS or ctas.shape[1] != BATCH_CTA_FIELDS:
        raise ValueError("vbq_b200: `units` must be (n, %d) and `ctas` (n, %d), got %s and %s" % (
            BATCH_UNIT_FIELDS, BATCH_CTA_FIELDS, tuple(units.shape), tuple(ctas.shape)))
    n_tables, C, _ = cum.shape
    if prob_bits.numel() != n_tables:
        raise ValueError("vbq_b200: %d prob_bits for %d tables" % (prob_bits.numel(), n_tables))
    dev = words.device
    q = torch.empty(n_out, dtype=torch.int32, device=dev) if want_qidx else None
    z = None
    if code_points is not None:
        _need_cuda("code_points", code_points, torch.float32, 2)
        if tuple(code_points.shape) != tuple(cum.shape[1:]):
            raise ValueError("vbq_b200: code_points are %s, need (C, Q) = %s" % (tuple(code_points.shape),
                                                                              tuple(cum.shape[1:])))
        z = torch.empty(n_out, dtype=torch.float32, device=dev)
    status = torch.zeros(n_blobs, dtype=torch.int32, device=dev)
    st = _lib.load().vbq_rans_decode_batch(_ptr(words), words.numel(), _ptr(cum), _ptr(prob_bits), n_tables, C,
                                           max_bits, _ptr(units), units.shape[0], _ptr(ctas), ctas.shape[0], n_blobs,
                                           _ptr(code_points), n_out, _ptr(q), _ptr(z), _ptr(status), _stream(dev))
    _lib.check(st, "vbq_rans_decode_batch")
    return q, z, status


def rans_encode_batch(symbols: torch.Tensor, cum: torch.Tensor, prob_bits: torch.Tensor, units: torch.Tensor,
                      ctas: torch.Tensor, blob_groups: torch.Tensor, n_groups: int, max_bits: int, scratch_words: int):
    """The work-list encoder of many images in one launch each of encode, scan and compaction.  symbols: contiguous
    int32 (read flat); cum (n_tables, C, Q) int16; prob_bits (n_tables,) int32; units (n_units, 7) int64
    (vbq_rans_encode_unit: in, rows, table, cg, group, scratch, blob), ctas (n_ctas, 4) int64 (vbq_rans_batch_cta) and
    blob_groups (n_blobs + 1,) int64 (each blob's first group; [n_blobs] = n_groups); scratch_words: the scratch the
    units' ranges lie in.  Returns (payload, meta): the int16 payload of 2 n_groups + scratch_words words, and one int64
    device tensor meta holding the n_blobs + 1 blob starts (blob b is payload words [meta[b], meta[b + 1])) followed by
    the (n_blobs,) int32 status per blob (bit 1: a symbol outside [0, Q), bit 8: a bad unit), so that one copy brings
    both to the host.  No synchronisation."""
    for name, t, dt, nd in (("symbols", symbols, torch.int32, None), ("cum", cum, torch.int16, 3),
                            ("prob_bits", prob_bits, torch.int32, 1), ("units", units, torch.int64, 2),
                            ("ctas", ctas, torch.int64, 2), ("blob_groups", blob_groups, torch.int64, 1)):
        _need_cuda(name, t, dt, nd)
    if units.shape[1] != BATCH_UNIT_FIELDS or ctas.shape[1] != BATCH_CTA_FIELDS:
        raise ValueError("vbq_b200: `units` must be (n, %d) and `ctas` (n, %d), got %s and %s" % (
            BATCH_UNIT_FIELDS, BATCH_CTA_FIELDS, tuple(units.shape), tuple(ctas.shape)))
    n_tables, C, _ = cum.shape
    if prob_bits.numel() != n_tables:
        raise ValueError("vbq_b200: %d prob_bits for %d tables" % (prob_bits.numel(), n_tables))
    n_blobs = blob_groups.numel() - 1
    if n_blobs < 0:
        raise ValueError("vbq_b200: `blob_groups` needs n_blobs + 1 >= 1 entries")
    lib = _lib.load()
    dev = symbols.device
    ws_bytes = lib.vbq_rans_encode_batch_workspace_bytes(n_groups, scratch_words)
    if ws_bytes < 0:
        raise ValueError("vbq_b200: bad batch encode size: %d groups, %d scratch words" % (n_groups, scratch_words))
    payload_words = 2 * n_groups + scratch_words
    payload = torch.empty(max(1, payload_words), dtype=torch.int16, device=dev)
    meta = torch.empty(n_blobs + 1 + (n_blobs + 1) // 2, dtype=torch.int64, device=dev)
    status = meta[n_blobs + 1:].view(torch.int32)
    ws = torch.empty(max(1, ws_bytes), dtype=torch.uint8, device=dev)
    st = lib.vbq_rans_encode_batch(_ptr(symbols), symbols.numel(), _ptr(cum), _ptr(prob_bits), n_tables, C, max_bits,
                                   _ptr(units), units.shape[0], _ptr(ctas), ctas.shape[0], _ptr(blob_groups), n_blobs,
                                   n_groups, payload.data_ptr(), payload_words, meta.data_ptr(), _ptr(status),
                                   ws.data_ptr(), ws_bytes, _stream(dev))
    _lib.check(st, "vbq_rans_encode_batch")
    return payload, meta


# ------------------------------------------------------------------------------------------------------
# entropy coding with one shared table per plane, symbols as one flat sequence (word embeddings; include/vbq_b200.h)
# ------------------------------------------------------------------------------------------------------
def _seg_array(seg_rows, n_planes):
    seg = [int(seg_rows)] * n_planes if isinstance(seg_rows, int) else [int(x) for x in seg_rows]
    if len(seg) != n_planes:
        raise ValueError("vbq_b200: %d seg_rows for %d planes" % (len(seg), n_planes))
    return (ctypes.c_longlong * n_planes)(*seg)


def rans_shared_payload_bound(n_planes: int, n: int, seg_rows) -> int:
    return int(_lib.load().vbq_rans_shared_payload_bound(n_planes, n, _seg_array(seg_rows, n_planes)))


def rans_shared_encode(qidx: torch.Tensor, cum: torch.Tensor, max_bits: int, prob_bits: int, seg_rows):
    """qidx (n_planes, n) int32 and cum (n_planes, Q+1) int32 (the uint32 cum tables of coding.cum_table_shared);
    seg_rows: an int or one per plane -> (payload int16 words of vbq_rans_shared_payload_bound bytes, payload size in
    bytes as a 1-element int64 tensor, status int32 tensor: bit 1 a symbol outside [0, Q), bit 2 a symbol of
    frequency 0): one launch for all planes, no synchronisation."""
    _need_cuda("qidx", qidx, torch.int32, 2)
    _need_cuda("cum", cum, torch.int32, 2)
    n_planes, n = qidx.shape
    seg = _seg_array(seg_rows, n_planes)
    lib = _lib.load()
    bound = lib.vbq_rans_shared_payload_bound(n_planes, n, seg)
    ws_bytes = lib.vbq_rans_shared_workspace_bytes(n_planes, n, seg)
    if bound < 0 or ws_bytes < 0:
        raise ValueError("vbq_b200: bad rANS shape: %s" % lib.vbq_last_error().decode())
    dev = qidx.device
    payload = torch.empty(max(1, bound // 2), dtype=torch.int16, device=dev)
    size = torch.zeros(1, dtype=torch.int64, device=dev)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    ws = torch.empty(max(1, ws_bytes), dtype=torch.uint8, device=dev)
    st = lib.vbq_rans_shared_encode(_ptr(qidx), n_planes, n, seg, max_bits, prob_bits,
                                    _ptr(cum), payload.data_ptr(), bound, size.data_ptr(),
                                    status.data_ptr(), ws.data_ptr(), ws_bytes, _stream(dev))
    _lib.check(st, "vbq_rans_shared_encode")
    return payload, size, status


def rans_shared_decode(words: torch.Tensor, bounds: torch.Tensor, cum: torch.Tensor, n: int, seg_rows, max_bits: int,
                       prob_bits: int, code_points: Optional[torch.Tensor] = None, want_qidx: bool = True):
    """words: the payload as int16 words; bounds (groups of all planes, 2) int64 word ranges; cum (n_planes, Q+1)
    int32.  Returns (qidx or None, zhat or None, status): (n_planes, n) int32 symbols and float32 code_points[q]
    (code_points (Q,) ascending), and the int32 device status (0 = every group passed the integrity check)."""
    _need_cuda("words", words, torch.int16, 1)
    _need_cuda("bounds", bounds, torch.int64, 2)
    _need_cuda("cum", cum, torch.int32, 2)
    n_planes = cum.shape[0]
    dev = words.device
    q = torch.empty((n_planes, n), dtype=torch.int32, device=dev) if want_qidx else None
    z = None
    if code_points is not None:
        _need_cuda("code_points", code_points, torch.float32, 1)
        z = torch.empty((n_planes, n), dtype=torch.float32, device=dev)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    st = _lib.load().vbq_rans_shared_decode(_ptr(words), words.numel(), _ptr(bounds), n_planes, n,
                                            _seg_array(seg_rows, n_planes), max_bits, prob_bits, _ptr(cum),
                                            _ptr(code_points), _ptr(q), _ptr(z), status.data_ptr(), _stream(dev))
    _lib.check(st, "vbq_rans_shared_decode")
    return q, z, status


# ------------------------------------------------------------------------------------------------------
# row access into one shared-table plane: decoder checkpoints and the row gather (include/vbq_b200.h)
# ------------------------------------------------------------------------------------------------------
LOOKUP_ITEM_FIELDS = 5      # vbq_rans_lookup_item: segment, checkpoint, last_row, lo, hi (int64 each)


def rans_shared_checkpoint_count(n: int, seg_rows: int, checkpoint_rows: int) -> int:
    """Checkpoints of a plane of n symbols in segments of seg_rows rows, one every checkpoint_rows rows; -1 for a bad
    shape."""
    return int(_lib.load().vbq_rans_shared_checkpoint_count(n, seg_rows, checkpoint_rows))


def rans_shared_checkpoints(words: torch.Tensor, bounds: torch.Tensor, cum: torch.Tensor, n: int, seg_rows: int,
                            max_bits: int, prob_bits: int, checkpoint_rows: int):
    """One full decode pass over one plane (words, bounds as for rans_shared_decode; cum (1, Q+1) or (Q+1,) int32) that
    records the checkpoint index.  Returns (offsets (M,) int32, states (M, 32) int32, status): the uint32 fields of
    the index as int32, and the int32 device status of vbq_rans_shared_decode.  No synchronisation."""
    _need_cuda("words", words, torch.int16, 1)
    _need_cuda("bounds", bounds, torch.int64, 2)
    _need_cuda("cum", cum, torch.int32)
    M = rans_shared_checkpoint_count(n, seg_rows, checkpoint_rows)
    if M < 0:
        raise ValueError("vbq_b200: bad checkpoint shape: %s" % _lib.load().vbq_last_error().decode())
    dev = words.device
    offsets = torch.empty(M, dtype=torch.int32, device=dev)
    states = torch.empty((M, 32), dtype=torch.int32, device=dev)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    st = _lib.load().vbq_rans_shared_checkpoints(_ptr(words), words.numel(), _ptr(bounds), n, seg_rows, max_bits,
                                                 prob_bits, _ptr(cum), checkpoint_rows, _ptr(offsets), _ptr(states),
                                                 status.data_ptr(), _stream(dev))
    _lib.check(st, "vbq_rans_shared_checkpoints")
    return offsets, states, status


def rans_shared_decode_rows(words: torch.Tensor, bounds: torch.Tensor, cum: torch.Tensor, n: int, seg_rows: int,
                            max_bits: int, prob_bits: int, checkpoint_rows: int, offsets: torch.Tensor,
                            states: torch.Tensor, items: torch.Tensor, rows: torch.Tensor, row_size: int,
                            code_points: Optional[torch.Tensor] = None, want_qidx: bool = False):
    """The row gather: items (n_items, 5) int64 work list (vbq_rans_lookup_item), rows (n_req,) int64 sorted unique
    embedding rows, row_size = D.  Returns (qidx or None, zhat or None, status): (n_req, D) int32 symbols and float32
    code_points[q], and the int32 device status (8 = a bad work item).  No synchronisation."""
    for name, t, dt, nd in (("words", words, torch.int16, 1), ("bounds", bounds, torch.int64, 2),
                            ("cum", cum, torch.int32, None), ("offsets", offsets, torch.int32, 1),
                            ("states", states, torch.int32, 2), ("items", items, torch.int64, 2),
                            ("rows", rows, torch.int64, 1)):
        _need_cuda(name, t, dt, nd)
    if items.shape[1] != LOOKUP_ITEM_FIELDS:
        raise ValueError("vbq_b200: `items` must be (n_items, %d), got %s" % (LOOKUP_ITEM_FIELDS, tuple(items.shape)))
    dev = words.device
    n_req = rows.numel()
    q = torch.empty((n_req, row_size), dtype=torch.int32, device=dev) if want_qidx else None
    z = None
    if code_points is not None:
        _need_cuda("code_points", code_points, torch.float32, 1)
        z = torch.empty((n_req, row_size), dtype=torch.float32, device=dev)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    st = _lib.load().vbq_rans_shared_decode_rows(_ptr(words), words.numel(), _ptr(bounds), n, seg_rows, max_bits,
                                                 prob_bits, _ptr(cum), checkpoint_rows, _ptr(offsets), _ptr(states),
                                                 _ptr(items), items.shape[0], _ptr(rows), n_req, row_size,
                                                 _ptr(code_points), _ptr(q), _ptr(z), status.data_ptr(), _stream(dev))
    _lib.check(st, "vbq_rans_shared_decode_rows")
    return q, z, status


SCORE_METRICS = {"dot": _lib.SCORE_DOT, "cosine": _lib.SCORE_COSINE}


def rans_shared_score_max_queries(row_size: int) -> int:
    """Queries of length row_size that one vbq_rans_shared_row_scores launch takes (0: none fits)."""
    return int(_lib.load().vbq_rans_shared_score_max_queries(row_size))


def rans_shared_row_scores(words: torch.Tensor, bounds: torch.Tensor, cum: torch.Tensor, n: int, seg_rows: int,
                           max_bits: int, prob_bits: int, checkpoint_rows: int, offsets: torch.Tensor,
                           states: torch.Tensor, row_size: int, row_begin: int, row_end: int, queries: torch.Tensor,
                           code_points: torch.Tensor, metric: str = "dot", out: Optional[torch.Tensor] = None):
    """Scores of queries (B, row_size) float32 against the embedding rows [row_begin, row_end) of one plane, decoded from
    the checkpoint index (arguments as for rans_shared_decode_rows).  Returns (scores (B, row_end - row_begin) float32,
    status int32: bit 1 a group ran out of words, bit 4 a bad group range or restored state).  `out`, if given, is a
    contiguous float32 tensor of that shape.  B <= rans_shared_score_max_queries(row_size).  No synchronisation."""
    for name, t, dt, nd in (("words", words, torch.int16, 1), ("bounds", bounds, torch.int64, 2),
                            ("cum", cum, torch.int32, None), ("offsets", offsets, torch.int32, 1),
                            ("states", states, torch.int32, 2), ("queries", queries, torch.float32, 2),
                            ("code_points", code_points, torch.float32, 1)):
        _need_cuda(name, t, dt, nd)
    if metric not in SCORE_METRICS:
        raise ValueError("vbq_b200: metric must be one of %s, got %r" % (sorted(SCORE_METRICS), metric))
    if queries.shape[1] != row_size:
        raise ValueError("vbq_b200: queries must be (B, %d), got %s" % (row_size, tuple(queries.shape)))
    dev = words.device
    B = queries.shape[0]
    shape = (B, row_end - row_begin)
    if out is None:
        out = torch.empty(shape, dtype=torch.float32, device=dev)
    else:
        _need_cuda("out", out, torch.float32, 2)
        if tuple(out.shape) != shape:
            raise ValueError("vbq_b200: out must be %s, got %s" % (shape, tuple(out.shape)))
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    st = _lib.load().vbq_rans_shared_row_scores(_ptr(words), words.numel(), _ptr(bounds), n, seg_rows, max_bits,
                                                prob_bits, _ptr(cum), checkpoint_rows, _ptr(offsets), _ptr(states),
                                                row_size, row_begin, row_end, _ptr(queries), B, SCORE_METRICS[metric],
                                                _ptr(code_points), _ptr(out), status.data_ptr(), _stream(dev))
    _lib.check(st, "vbq_rans_shared_row_scores")
    return out, status


# ------------------------------------------------------------------------------------------------------
# exact target ranks against dense float32 rows (include/vbq_b200.h, vbq_score_ranks / vbq_pair_scores)
# ------------------------------------------------------------------------------------------------------
def score_ranks(rows: torch.Tensor, queries: torch.Tensor, metric: str, thresholds: torch.Tensor,
                targets: torch.Tensor, counts: torch.Tensor, row_offset: int = 0):
    """Adds to counts (B,) int64 the number of rows of rows (n_rows, D) float32 (global ids row_offset ..) that beat
    each query's target under the score and order contract: queries (B, D) float32, thresholds (B,) float32 = the
    target's score, targets (B,) int64 global ids.  Returns counts.  No synchronisation."""
    for name, t, dt, nd in (("rows", rows, torch.float32, 2), ("queries", queries, torch.float32, 2),
                            ("thresholds", thresholds, torch.float32, 1), ("targets", targets, torch.int64, 1),
                            ("counts", counts, torch.int64, 1)):
        _need_cuda(name, t, dt, nd)
    if metric not in SCORE_METRICS:
        raise ValueError("vbq_b200: metric must be one of %s, got %r" % (sorted(SCORE_METRICS), metric))
    B, D = queries.shape
    if rows.shape[1] != D or not thresholds.numel() == targets.numel() == counts.numel() == B:
        raise ValueError("vbq_b200: score_ranks shapes: rows %s, queries %s, thresholds %s, targets %s, counts %s"
                         % tuple(tuple(t.shape) for t in (rows, queries, thresholds, targets, counts)))
    st = _lib.load().vbq_score_ranks(_ptr(rows), rows.shape[0], D, int(row_offset), _ptr(queries), B,
                                     SCORE_METRICS[metric], _ptr(thresholds), _ptr(targets), _ptr(counts),
                                     _stream(rows.device))
    _lib.check(st, "vbq_score_ranks")
    return counts


def pair_scores(rows: torch.Tensor, queries: torch.Tensor, pair_rows: torch.Tensor, pair_queries: torch.Tensor,
                metric: str = "dot"):
    """float32 (P,) scores of query pair_queries[p] with row pair_rows[p] of rows (n_rows, D) float32, under the
    contract; queries (B, D) float32, both index arrays (P,) int64 (an index out of range gives NaN).  No
    synchronisation."""
    for name, t, dt, nd in (("rows", rows, torch.float32, 2), ("queries", queries, torch.float32, 2),
                            ("pair_rows", pair_rows, torch.int64, 1), ("pair_queries", pair_queries, torch.int64, 1)):
        _need_cuda(name, t, dt, nd)
    if metric not in SCORE_METRICS:
        raise ValueError("vbq_b200: metric must be one of %s, got %r" % (sorted(SCORE_METRICS), metric))
    if rows.shape[1] != queries.shape[1] or pair_rows.numel() != pair_queries.numel():
        raise ValueError("vbq_b200: pair_scores shapes: rows %s, queries %s, pair_rows %s, pair_queries %s"
                         % tuple(tuple(t.shape) for t in (rows, queries, pair_rows, pair_queries)))
    out = torch.empty(pair_rows.numel(), dtype=torch.float32, device=rows.device)
    st = _lib.load().vbq_pair_scores(_ptr(rows), rows.shape[0], rows.shape[1], _ptr(queries), queries.shape[0],
                                     _ptr(pair_rows), _ptr(pair_queries), pair_rows.numel(), SCORE_METRICS[metric],
                                     _ptr(out), _stream(rows.device))
    _lib.check(st, "vbq_pair_scores")
    return out


# image quality: exact SSE and the MS-SSIM levels (include/vbq_b200.h, vbq_image_metrics)
# ---------------------------------------------------------------------------------------
def image_metrics(originals: torch.Tensor, reconstructions: torch.Tensor):
    """originals (N, H, W, C) uint8 and reconstructions (M, N, H, W, C) uint8 on one CUDA device ->
    (sse (M, N) int64, ssim (M, N, 5) float64, cs (M, N, 5) float64): the exact sum of squared errors and the per-level
    means of MultiScaleSSIM's ssim and cs.  No synchronisation."""
    _need_cuda("originals", originals, torch.uint8, 4)
    _need_cuda("reconstructions", reconstructions, torch.uint8, 5)
    if tuple(reconstructions.shape[1:]) != tuple(originals.shape) or reconstructions.device != originals.device:
        raise ValueError("vbq_b200: image_metrics shapes: originals %s on %s, reconstructions %s on %s"
                         % (tuple(originals.shape), originals.device, tuple(reconstructions.shape),
                            reconstructions.device))
    N, H, W, C = originals.shape
    M = reconstructions.shape[0]
    lib = _lib.load()
    nbytes = lib.vbq_image_metrics_workspace_bytes(N, M, H, W, C)
    if nbytes < 0:
        raise ValueError("vbq_b200: image_metrics cannot take images of shape %s (1 <= C <= %d, H W C < 2^31)"
                         % (tuple(originals.shape), _lib.IMAGE_METRICS_MAX_CHANNELS))
    dev = originals.device
    L = _lib.IMAGE_METRICS_LEVELS
    sse = torch.empty((M, N), dtype=torch.int64, device=dev)
    ssim = torch.empty((M, N, L), dtype=torch.float64, device=dev)
    cs = torch.empty((M, N, L), dtype=torch.float64, device=dev)
    if M * N == 0:
        return sse, ssim, cs
    ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    st = lib.vbq_image_metrics(_ptr(originals), _ptr(reconstructions), N, M, H, W, C, _ptr(ws), nbytes, _ptr(sse),
                               _ptr(ssim), _ptr(cs), _stream(dev))
    _lib.check(st, "vbq_image_metrics")
    return sse, ssim, cs
