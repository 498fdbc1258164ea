"""CPU tests of the drop-in boundary: the C-ABI library loads, exports every symbol include/vbq_b200.h declares,
validates its arguments without touching a GPU, and the Python product path refuses to run without CUDA."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    hdr = open(os.path.join(ROOT, "include", "vbq_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    return sorted(set(re.findall(r"\b(vbq_[a-z0-9_]+)\s*\(", hdr)))


def test_library_exports_every_declared_symbol():
    from vbq_b200 import _lib
    lib = ctypes.CDLL(_lib.LIB_PATH)
    syms = declared_symbols()
    assert len(syms) >= 15
    for s in syms:
        assert hasattr(lib, s), "missing export: " + s
    assert sorted(_lib.SIGNATURES) == syms, "ctypes binding table out of sync with include/vbq_b200.h"


def test_version_and_status_strings():
    from vbq_b200 import _lib
    lib = _lib.load()
    assert lib.vbq_version() == 100
    assert lib.vbq_status_string(0) == b"ok"
    assert lib.vbq_status_string(3) == b"bad max_bits_per_coord"
    assert lib.vbq_packed_table_floats(192, 10) == 12 * (2069 * 16 + 40992)
    assert lib.vbq_packed_table_floats(1, 0) == 2069 * 16 + 40992
    assert lib.vbq_packed_table_floats(0, 10) == -1 and lib.vbq_packed_table_floats(4, 21) == -1
    assert lib.vbq_quantize_workspace_bytes(1) == 256 + 1024 * 4 * 8
    assert lib.vbq_quantize_workspace_bytes(0) == -1


def test_argument_validation_needs_no_gpu():
    """Error paths return status codes (never throw, never touch the device)."""
    from vbq_b200 import _lib
    lib = _lib.load()
    one = ctypes.c_void_p(16)      # any non-null, 16-byte aligned address: these calls must fail before using it
    st = lib.vbq_quantize(one, one, -1, 4, one, one, 10, one, None, 1, 1, None, None, None, None, None, None, None,
                          None, 0, 0, None)
    assert st == 2 and b"rows=-1" in lib.vbq_last_error()
    st = lib.vbq_quantize(one, one, 8, 4, one, one, 21, one, None, 1, 1, None, None, None, None, None, None, None,
                          None, 0, 0, None)
    assert st == 3
    st = lib.vbq_quantize(one, one, 8, 4, one, one, 10, one, None, 1, 3, None, None, None, None, None, None, None,
                          None, 0, 0, None)
    assert st == 2                                             # pen_channels not in {1, C}
    st = lib.vbq_quantize(one, one, 8, 4, one, one, 10, one, None, 1, 1, None, None, None, None, None, None, None,
                          None, 0, 1 << 20, None)
    assert st == 4
    st = lib.vbq_quantize(None, one, 8, 4, one, one, 10, one, None, 1, 1, None, None, None, None, None, None, None,
                          None, 0, 0, None)
    assert st == 1
    st = lib.vbq_quantize(one, one, 8, 4, one, one, 10, one, None, 1, 1, None, None, None, None, None, None, one,
                          None, 0, 0, None)
    assert st == 5                                             # totals without workspace
    with pytest.raises(_lib.VbqError):
        _lib.check(st, "vbq_quantize")
    assert lib.vbq_build_code_points_learned(None, 4, 10, one, None) == 1
    assert lib.vbq_pack_code_points(one, 0, 10, one, None) == 2


def test_sigma_selftest_validates_without_gpu():
    """vbq_selftest_sigma_from_logvar rejects null pointers and negative counts, and an empty call is a no-op: all
    before any device work."""
    from vbq_b200 import _lib
    lib = _lib.load()
    one = ctypes.c_void_p(16)
    assert lib.vbq_selftest_sigma_from_logvar(None, 8, one, None) == 1
    assert lib.vbq_selftest_sigma_from_logvar(one, 8, None, None) == 1
    assert b"vbq_selftest_sigma_from_logvar" in lib.vbq_last_error()
    assert lib.vbq_selftest_sigma_from_logvar(one, -1, one, None) == 2 and b"n=-1" in lib.vbq_last_error()
    assert lib.vbq_selftest_sigma_from_logvar(None, 0, None, None) == 0


def test_no_cpu_fallback():
    import vbq_b200
    from vbq_b200 import ops
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        ops.quantize(torch.zeros(4, 2), torch.ones(4, 2), torch.zeros(2, 7), torch.zeros(2069 * 16 + 40992),
                     torch.zeros(1, 1, 3), None, None, 2, ops.OUT_ZHAT, 0)
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        ops.learned_cdf(torch.zeros(2, 43), torch.zeros(3, 2))
    # nothing under vbq_b200/ may import the oracle
    for root, _, files in os.walk(os.path.join(ROOT, "vbq_b200")):
        for f in files:
            if f.endswith(".py"):
                assert "oracle" not in open(os.path.join(root, f)).read(), f


def test_missing_library_fails_loudly(tmp_path, monkeypatch):
    from vbq_b200 import _lib
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", str(tmp_path / "libvbq_b200.so"))
    with pytest.raises(ImportError, match="no CPU fallback"):
        _lib.load()


def test_host_helpers():
    from vbq_b200 import utils
    assert utils.n_bit_binary_floats(2) == [0.125, 0.375, 0.625, 0.875]
    xi = utils.all_bin_floats(3)
    assert len(xi) == 15 and xi[0] == 0.5 and xi[-1] == 1 - 2 ** -4
    N = 5
    n = np.repeat(np.arange(N + 1), [2 ** k for k in range(N + 1)])
    i = np.concatenate([np.arange(2 ** k) for k in range(N + 1)])
    assert np.array_equal(np.argsort(np.argsort(utils.all_bin_floats(N))), utils.heap_to_sorted_index(n, i, N))
    f = utils.curry_normal_logpdf(loc=torch.tensor([1.0]), scale=torch.tensor([2.0]), ignore_const=True)
    assert float(f(torch.tensor([3.0]))) == -0.5


def test_span_cuts_partition_every_tile_exactly_once():
    """The work split of the bisection kernels (same host/device function): monotone cuts from 0 to the tile count,
    balanced within the group-switch charge, for ragged shapes and grids larger than the work."""
    from vbq_b200 import _lib
    lib = _lib.load()
    for rows, C, grid in ((36864, 192, 148), (36864, 192, 147), (1, 1, 148), (5, 33, 7), (1000003, 300, 148),
                          (64, 320, 1), (0, 16, 4), (4097, 17, 1024)):
        out = (ctypes.c_longlong * (grid + 1))()
        assert lib.vbq_selftest_span_cuts(rows, C, grid, out) == 0
        cuts = list(out)
        tiles = ((rows + 3) // 4) * ((C + 15) // 16)
        assert cuts[0] == 0 and cuts[-1] == tiles
        assert all(a <= b for a, b in zip(cuts, cuts[1:]))
        sizes = [b - a for a, b in zip(cuts, cuts[1:])]
        if tiles >= 100 * grid:
            assert max(sizes) - min(sizes) <= 81 + 1           # a CTA that crosses a group boundary gets up to 80 fewer
    assert lib.vbq_selftest_span_cuts(8, 0, 4, (ctypes.c_longlong * 5)()) == 2
