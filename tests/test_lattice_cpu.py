"""CPU: lattice inference (dpn_decoder_lattice) - struct layout, argument validation, workspace sizes, and the lattice oracle
against the point-wise oracle pieces."""
import ctypes as C

import numpy as np
import pytest
import torch

from tests import helpers as H


def _N():
    import __graft_entry__ as g
    g.build()
    from deepphysinet_b200 import _native
    return _native


def _bytes(fn, B, Np, mode, chunk=0):
    N = _N()
    need = C.c_size_t(0)
    shp = N.DpnShape(B=B, N=Np, K=6, mode=N.MODES[mode], n_norm=0, seed_scale=1.0, chunk=chunk)
    assert getattr(N.lib(), fn)(C.byref(shp), C.byref(need)) == 0
    return need.value


def test_lattice_struct_layout():
    N = _N()
    assert C.sizeof(N.DpnLattice) == 4 * 4 + 6 * 8
    assert N.DpnLattice.x0.offset == 16 and N.DpnLattice.st.offset == 56


DPN_E_INVALID = 10001
# Never dereferenced: every case below is refused before the library touches a pointer or the device.
_FAKE = 0x10000


def _args(**over):
    """A valid call for a [1,5,4,5,6] coarse stack (x up to 432 km, y up to 324 km, t up to 24 h) on a 3 x 4 x 2 lattice,
    with `over` replacing lattice (nx, ny, nt, x0, ..., st), sampler (sB, sN) or shape (B, N, K) fields."""
    N = _N()
    lat = dict(nx=3, ny=4, nt=2, pad_=0, x0=0.0, y0=0.0, t0=0.0, sx=27000.0, sy=27000.0, st=3600.0)
    lat.update({k: v for k, v in over.items() if k in lat})
    n = lat["nx"] * lat["ny"] * lat["nt"]
    shape = N.DpnShape(B=over.get("B", 1), N=over.get("N", n), K=over.get("K", 6), mode=N.MODE_F16X3, n_norm=0, seed_scale=1.0, chunk=0)
    S = N.DpnSampler(B=over.get("sB", 1), N=over.get("sN", n), Tt=5, Hc=4, Wc=5, pad_=0, dx=27000.0, dy=27000.0, cells_per_coarse=4.0,
                     t_step=21600.0, begin_lat=0.0, deg_per_cell=0.0, omega=0.0)
    W = N.DpnWeights(**{f: _FAKE for f in N.WEIGHT_FIELDS})
    return shape, N.DpnConsts(), N.DpnLattice(**lat), S, W


def _call(shape, consts, lat, S, W, coarse=_FAKE, out=_FAKE):
    N = _N()
    L = N.lib()
    rc = L.dpn_decoder_lattice(C.byref(shape), C.byref(consts), C.byref(lat) if lat is not None else None,
                               C.byref(S) if S is not None else None, coarse, C.byref(W), out, _FAKE, 1 << 40, None)
    buf = C.create_string_buffer(1024)
    L.dpn_last_error(buf, 1024)
    return rc, buf.value.decode()


@pytest.mark.parametrize("over,msg", [
    (dict(nx=0, N=8), "sizes must be positive"),
    (dict(nt=-1, N=6), "sizes must be positive"),
    (dict(sx=0.0), "spacing must be positive"),
    (dict(st=-3600.0), "spacing must be positive"),
    (dict(sy=float("nan")), "spacing must be positive"),
    (dict(N=25), "shape N = 25 but the lattice has nx ny nt = 24 nodes"),
    (dict(sB=2), "does not match shape"),
    (dict(sN=23), "does not match shape"),
    (dict(K=5), "needs K = 6"),
    (dict(x0=-1.0), "lattice x range"),
    (dict(nx=18, N=144), "lattice x range"),                       # last node 17 x 27 km > 432 km
    (dict(y0=300000.0), "lattice y range"),                        # last node 381 km > 324 km
    (dict(t0=-60.0), "lattice t range"),
    (dict(nt=26, N=312), "lattice t range"),                        # last lead 25 h > 24 h
])
def test_validation_rules(over, msg):
    rc, err = _call(*_args(**over))
    assert rc == DPN_E_INVALID and msg in err, (rc, err)


def test_validation_of_null_pointers_and_int32_nodes():
    shape, consts, lat, S, W = _args()
    for rc, err in (_call(shape, consts, None, S, W), _call(shape, consts, lat, None, W),
                    _call(shape, consts, lat, S, W, coarse=None), _call(shape, consts, lat, S, W, out=None)):
        assert rc == DPN_E_INVALID and "NULL" in err, err
    W.W2 = None
    rc, err = _call(shape, consts, lat, S, W)
    assert rc == DPN_E_INVALID and "weight pointer" in err, err
    rc, err = _call(*_args(nx=2048, ny=2048, nt=1024, N=2 ** 31 - 1))
    assert rc == DPN_E_INVALID and "does not fit int32" in err, err


def test_exact_edges_are_inside():
    """A lattice ending exactly on the far edge of the coarse stack in x, y and t is accepted by validation (the call then fails
    only for want of a device / real pointers, never with DPN_E_INVALID)."""
    rc, err = _call(*_args(nx=17, ny=13, nt=25, N=17 * 13 * 25))
    assert rc != DPN_E_INVALID, err


@pytest.mark.parametrize("mode", ["bf16", "bf16x3", "f16x3", "f16x3a"])
def test_lattice_workspace_is_a_tenth_of_the_full_one(mode):
    """configs[3] of bench.py (one sample, 48 hourly leads on the 145 x 257 training grid) as one lattice job."""
    Np = 48 * 145 * 257
    lat = _bytes("dpn_lattice_workspace_bytes", 1, Np, mode)
    full = _bytes("dpn_workspace_bytes", 1, Np, mode)
    assert 10 * lat <= full, (lat, full)


@pytest.mark.parametrize("mode", ["fp32", "bf16", "bf16x3", "f16x3", "f16x3a"])
def test_refined_lattice_workspace_bound(mode):
    """The 4x refined domain (577 x 1025 nodes, 25 leads) for four samples: 14.8 M nodes per sample run through a workspace of
    at most 1.6 GiB (about 2.3 KB per point in flight in the split modes, 1.5 KB in bf16, one sample's chunk at a time in fp32)."""
    assert _bytes("dpn_lattice_workspace_bytes", 4, 577 * 1025 * 25, mode) < 1.6 * 2 ** 30


# dpn_workspace_bytes of the parent commit: the values-only prefix re-orders the carve, it must not change its size.
_PINNED = {
    (1, 300, 0): dict(fp32=24972800, bf16=14781440, bf16x3=28740608, f16x3=28740608, f16x3a=28740608),
    (2, 333, 0): dict(fp32=27722240, bf16=27371520, bf16x3=53127168, f16x3=53127168, f16x3a=53127168),
    (8, 65536, 0): dict(fp32=1362174464, bf16=10090595328, bf16x3=19375801344, f16x3=19375801344, f16x3a=19375801344),
    (1, 1788720, 0): dict(fp32=1362131456, bf16=20137610240, bf16x3=19337219072, f16x3=19337219072, f16x3a=19337219072),
    (4, 14785625, 0): dict(fp32=1362149888, bf16=20145888256, bf16x3=19353754624, f16x3=19353754624, f16x3a=19353754624),
    (3, 8120, 256): dict(fp32=21326336, bf16=25214976, bf16x3=49201152, f16x3=49201152, f16x3a=49201152),
}


@pytest.mark.parametrize("key", sorted(_PINNED))
def test_full_workspace_sizes_unchanged(key):
    B, Np, chunk = key
    for mode, want in _PINNED[key].items():
        assert _bytes("dpn_workspace_bytes", B, Np, mode, chunk) == want, (key, mode)


def test_lattice_oracle_matches_point_oracle():
    """oracle/lattice_oracle on a small refined, cropped lattice with sub-hour leads against a per-node restatement with
    sampler_oracle.trilinear + dpn_oracle.encoding_coord / decode_generated / inverse_norm(with_clip=False)."""
    from deepphysinet_b200.functional import Lattice
    from oracle import dpn_oracle as O, lattice_oracle as LO, sampler_oracle as SO
    g = torch.Generator().manual_seed(11)
    W = dict(W1=0.1 * torch.randn(6, 256, 192, generator=g, dtype=torch.float64), b1=0.1 * torch.randn(6, 256, generator=g, dtype=torch.float64),
             W2=0.06 * torch.randn(6, 256, 256, generator=g, dtype=torch.float64), b2=0.1 * torch.randn(6, 256, generator=g, dtype=torch.float64),
             e=0.1 * torch.randn(6, 256, generator=g, dtype=torch.float64), Wd=0.07 * torch.randn(6, 256, 192, generator=g, dtype=torch.float64),
             bd=0.1 * torch.randn(6, 256, generator=g, dtype=torch.float64), Wa=0.06 * torch.randn(6, 256, 256, generator=g, dtype=torch.float64),
             ba=0.1 * torch.randn(6, 256, generator=g, dtype=torch.float64), Wb=0.06 * torch.randn(6, 256, 256, generator=g, dtype=torch.float64),
             bb=0.1 * torch.randn(6, 256, generator=g, dtype=torch.float64), wo=0.06 * torch.randn(6, 256, generator=g, dtype=torch.float64),
             bo=0.1 * torch.randn(6, generator=g, dtype=torch.float64))
    coarse = torch.randn(5, 4, 5, 6, generator=g, dtype=torch.float64).numpy()
    lat = Lattice(nx=5, ny=3, nt=4, x0=2 * 9000.0, y0=9000.0, t0=1200.0, sx=9000.0, sy=9000.0, st=1200.0)
    geom = dict(lat_size=13, lon_size=17)
    got = LO.lattice_values(coarse, W, lat, **geom)
    assert got.shape == (4, 3, 5, 6) and torch.isfinite(got).all()
    for k in range(lat.nt):
        for j in range(lat.ny):
            for i in range(lat.nx):
                x, y, t = np.float32(lat.x0 + i * lat.sx), np.float32(lat.y0 + j * lat.sy), np.float32(lat.t0 + k * lat.st)
                cd = torch.from_numpy(SO.trilinear(coarse, [x], [y], [t]))
                pe = O.encoding_coord(torch.tensor([[float(x)]], dtype=torch.float64), torch.tensor([[float(y)]], dtype=torch.float64),
                                      torch.tensor([[float(t)]], dtype=torch.float64), 27000.0, 27000.0, 13, 17, 86400.0)
                with torch.no_grad():
                    want = torch.cat(O.inverse_norm(O.decode_generated(pe, cd, W), with_clip=False), 1)[0]
                assert H.rel(got[k, j, i], want) < 1e-14, (k, j, i)
