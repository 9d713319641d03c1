"""CPU: the C-ABI library loads and exports every symbol include/dpn_b200.h declares; argument validation
works without a GPU; the product refuses to run without CUDA (no CPU fallback)."""
import ctypes as C
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _lib():
    import __graft_entry__ as g
    g.build()
    from deepphysinet_b200 import _native
    return _native


def test_every_declared_symbol_is_exported():
    N = _lib()
    header = open(os.path.join(ROOT, "include", "dpn_b200.h")).read()
    declared = set(re.findall(r"^\s*(?:int|size_t)\s+(dpn_\w+)\s*\(", header, flags=re.M))
    assert declared == set(N.EXPORTS), (declared, N.EXPORTS)
    L = N.lib()
    for sym in declared:
        assert getattr(L, sym) is not None
    assert L.dpn_abi_version() == N.ABI_VERSION == 2


def test_struct_layouts_match_header_sizes():
    N = _lib()
    assert C.sizeof(N.DpnShape) == 32
    assert C.sizeof(N.DpnConsts) == 8 * 2 + 4 * 2 + 8 + 4 * 2 + 8 * 30 + 8 * 4 + 4 * 48
    assert C.sizeof(N.DpnPoints) == 7 * 8 and C.sizeof(N.DpnWeights) == 13 * 8 and C.sizeof(N.DpnPdeOut) == 3 * 8
    assert C.sizeof(N.DpnMargin) == 5 * 8 and C.sizeof(N.DpnQueryGen) == 6 * 4 + 3 * 8 + 2 * 8 and C.sizeof(N.DpnSampler) == 6 * 4 + 7 * 8


def test_argument_validation_without_gpu():
    N = _lib()
    L = N.lib()
    need = C.c_size_t(0)
    bad = N.DpnShape(B=0, N=10, K=6, mode=0, n_norm=0, seed_scale=1.0, chunk=0)
    assert L.dpn_workspace_bytes(C.byref(bad), C.byref(need)) != 0
    buf = C.create_string_buffer(256)
    L.dpn_last_error(buf, 256)
    assert b"bad shape" in buf.value
    for mode in N.MODES.values():
        ok = N.DpnShape(B=8, N=65536, K=6, mode=mode, n_norm=0, seed_scale=0.125, chunk=0)
        assert L.dpn_workspace_bytes(C.byref(ok), C.byref(need)) == 0 and need.value > 0
    # the 0.25 degree / B=8 / 65k configuration must fit comfortably in 180 GB
    assert need.value < 40 * 2 ** 30


def test_mode_enum_matches_header():
    """Every DPN_MODE_* of the header is reachable from Python under the documented name, and unknown modes are refused."""
    N = _lib()
    header = open(os.path.join(ROOT, "include", "dpn_b200.h")).read()
    declared = {name.lower(): int(val) for name, val in re.findall(r"DPN_MODE_(\w+)\s*=\s*(\d+)", header)}
    assert declared == N.MODES, (declared, N.MODES)
    need = C.c_size_t(0)
    bad = N.DpnShape(B=1, N=128, K=6, mode=max(N.MODES.values()) + 1, n_norm=0, seed_scale=1.0, chunk=0)
    assert N.lib().dpn_workspace_bytes(C.byref(bad), C.byref(need)) != 0
    # the headline shape runs as one pass in every tensor-core mode; all of them keep the same tiles (QM ZH | ZP ZD | seeds | masks),
    # the split modes as two 16-bit planes, the bf16 mode as one: 12.1 vs 6.4 GiB
    sizes = {}
    for name, mode in N.MODES.items():
        shp = N.DpnShape(B=8, N=65536, K=6, mode=mode, n_norm=0, seed_scale=0.125, chunk=0)
        assert N.lib().dpn_workspace_bytes(C.byref(shp), C.byref(need)) == 0
        sizes[name] = need.value
    assert 1.7 < sizes["f16x3"] / sizes["bf16"] < 2.1 and sizes["f16x3"] == sizes["bf16x3"] == sizes["f16x3a"], sizes
    assert max(sizes.values()) < 40 * 2 ** 30, sizes


def test_no_cpu_fallback():
    from deepphysinet_b200 import functional as Fn, testing as T
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    W, pts = T.random_decoder_weights(B=1, N=8, device="cpu")
    with pytest.raises(RuntimeError, match="no CPU path|CUDA"):
        Fn.pde_residual(pts["x"], pts["y"], pts["t"], pts["f"], pts["coord_data"], W)
