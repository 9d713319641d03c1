"""GPU (-m gpu): lattice inference, dpn_decoder_lattice / functional.decoder_lattice / InterfacePhysics.predict_lattice."""
import ctypes as C

import numpy as np
import pytest
import torch

from tests import helpers as H

pytestmark = pytest.mark.gpu

MODES = ["fp32", "bf16", "bf16x3", "f16x3", "f16x3a"]
TOL = dict(fp32=1e-4, f16x3=1e-5, f16x3a=1e-5, bf16x3=1e-5, bf16=2e-2)      # values tolerances of test_gpu_decoder.py
GENERATED = ("W1", "b1", "W2", "b2", "e")


@pytest.fixture(scope="module")
def case():
    """A 13 x 17 model (as test_gpu_decoder._interface(img=(13, 17))), three samples with their own encoder input and their own
    [5,4,5,6] coarse stack (which covers the 13 x 17 grid: 3 x 4 coarse cells, 24 h), and the decoder weights of all three."""
    from deepphysinet_b200 import InterfacePhysics
    from deepphysinet_b200.config import DEFAULT_OBS_NORM
    obs = {k: dict(v, norm_type="mean_norm", use_norm=True) for k, v in DEFAULT_OBS_NORM.items()}
    torch.manual_seed(0)
    m = InterfacePhysics(H.META_CFG, H.NET_CFG, obs, None, dict(img_size=(13, 17), dx=27000, dy=27000)).double().cuda()
    g = torch.Generator().manual_seed(8)
    field = torch.randn(3, 159, 2405, generator=g, dtype=torch.float64).cuda()
    fh = torch.full((3, 1, 1), 24.0 / 360.0, dtype=torch.float64).cuda()
    coarse = torch.randn(3, 5, 4, 5, 6, generator=g).cuda()
    with torch.no_grad():
        W = m.physics_net.decoder_weights(field, fh)
    return m, field, fh, coarse, W


def _sample(W, b):
    from deepphysinet_b200.functional import DecoderWeights
    return DecoderWeights(*[(w[b:b + 1] if n in GENERATED else w) for n, w in zip(DecoderWeights._fields, W)])


def _oracle_weights(W, b):
    """Sample b's decoder tensors as the library sees them (fp32), in fp64, oracle layout."""
    from deepphysinet_b200.functional import DecoderWeights
    return {n: (w[b] if n in GENERATED else w).float().double().cpu() for n, w in zip(DecoderWeights._fields, W)}


def _normalised_err(got, want, consts):
    """Worst per-variable relative error of the normalised values (out - mean) / std: the physical values span five decades."""
    errs = []
    for k in range(6):
        a = (got[..., k].double().cpu() - consts.mean[k]) / consts.std[k]
        b = (want[..., k].double().cpu() - consts.mean[k]) / consts.std[k]
        errs.append(H.rel(a, b))
    return max(errs)


def _raw(coarse, W, lat, consts, mode, chunk=0, ws=None, nbytes=None):
    """dpn_decoder_lattice called directly: (return code, out, error text); ws / nbytes default to a fresh buffer of
    dpn_lattice_workspace_bytes."""
    from deepphysinet_b200 import _native as N, functional as Fn
    B = coarse.shape[0]
    g = N.DpnLattice(nx=lat.nx, ny=lat.ny, nt=lat.nt, pad_=0, x0=lat.x0, y0=lat.y0, t0=lat.t0, sx=lat.sx, sy=lat.sy, st=lat.st)
    Np = lat.nx * lat.ny * lat.nt
    shape = Fn._shape(B, Np, 6, mode, chunk=chunk)
    S = N.DpnSampler(B=B, N=Np, Tt=coarse.shape[1], Hc=coarse.shape[2], Wc=coarse.shape[3], pad_=0, dx=consts.dx, dy=consts.dy,
                     cells_per_coarse=4.0, t_step=21600.0, begin_lat=0.0, deg_per_cell=0.0, omega=0.0)
    if ws is None:
        nbytes = lattice_bytes(B, Np, mode, chunk)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=coarse.device)
    ws_f = [Fn._prep(w) for w in W]
    out = torch.empty(B, lat.nt, lat.ny, lat.nx, 6, device=coarse.device)
    rc = N.lib().dpn_decoder_lattice(C.byref(shape), C.byref(N.make_consts(consts)), C.byref(g), C.byref(S), N.ptr(coarse.contiguous()),
                                     C.byref(Fn._weights_struct(ws_f)), N.ptr(out), N.ptr(ws), nbytes, N.stream_ptr())
    torch.cuda.synchronize()
    buf = C.create_string_buffer(1024)
    N.lib().dpn_last_error(buf, 1024)
    return rc, out, buf.value.decode()


def lattice_bytes(B, Np, mode, chunk=0):
    from deepphysinet_b200 import _native as N, functional as Fn
    need = C.c_size_t(0)
    N.check(N.lib().dpn_lattice_workspace_bytes(C.byref(Fn._shape(B, Np, 6, mode, chunk=chunk)), C.byref(need)), "dpn_lattice_workspace_bytes")
    return need.value


@pytest.mark.parametrize("mode", MODES)
def test_training_lattice_matches_predict_grid_bit_for_bit(case, mode):
    """refine = 1, 3-hourly leads: the same nodes predict_grid evaluates, with the same per-point arithmetic (coordinates exact in
    fp32, the same sampler, encoder, pass 1 and two-rounding de-normalisation), in another node order and chunking."""
    from deepphysinet_b200.functional import Lattice
    m, field, fh, coarse, W = case
    m.mode = mode
    W0 = _sample(W, 0)
    grid = m.predict_grid(field[:1], coarse[:1], fh[:1], time_ids=range(0, 25, 3), weights=W0)
    lat = Lattice.domain(m.consts(m._last_factor()), refine=1, st=3 * 3600.0, nt=9)
    got = m.predict_lattice(field[:1], coarse[:1], fh[:1], lat, weights=W0)
    assert got.shape == (1, 9, 13, 17, 6) and got.grad_fn is None
    assert torch.equal(got[0], grid)


_CROP = dict(refine=3, t0=600.0, st=1200.0, nt=3)     # 20-minute leads at 3x the training resolution


def _crop(consts):
    from deepphysinet_b200.functional import Lattice
    lat = Lattice.domain(consts, **_CROP)
    return lat._replace(x0=2 * lat.sx, nx=40, y0=3 * lat.sy, ny=29)          # 40 x 29 x 3 = 3480 nodes: not a multiple of 128


@pytest.fixture(scope="module")
def crop_oracle(case):
    from oracle import lattice_oracle as LO
    m, field, fh, coarse, W = case
    consts = m.consts(m._last_factor())
    lat = _crop(consts)
    return lat, [LO.lattice_values(coarse[b].double().cpu().numpy(), _oracle_weights(W, b), lat, lat_size=13, lon_size=17)
                 for b in range(2)]


@pytest.mark.parametrize("mode", MODES)
def test_refined_cropped_lattice_matches_oracle(case, crop_oracle, mode):
    from deepphysinet_b200 import functional as Fn
    m, field, fh, coarse, W = case
    consts = m.consts(m._last_factor())
    lat, want = crop_oracle
    W2 = Fn.DecoderWeights(*[(w[:2] if n in GENERATED else w) for n, w in zip(Fn.DecoderWeights._fields, W)])
    got = Fn.decoder_lattice(coarse[:2], W2, lat, consts=consts, mode=mode)
    assert got.shape == (2, 3, 29, 40, 6) and torch.isfinite(got).all()
    for b in range(2):
        err = _normalised_err(got[b], want[b], consts)
        assert err < TOL[mode], (mode, b, err)
    assert not torch.equal(got[0], got[1])


@pytest.mark.parametrize("mode", MODES)
def test_batch_and_chunk_independence(case, mode):
    from deepphysinet_b200 import functional as Fn
    m, field, fh, coarse, W = case
    consts = m.consts(m._last_factor())
    lat = _crop(consts)
    all3 = Fn.decoder_lattice(coarse, W, lat, consts=consts, mode=mode)
    for b in range(3):
        one = Fn.decoder_lattice(coarse[b:b + 1], _sample(W, b), lat, consts=consts, mode=mode)
        assert torch.equal(all3[b], one[0]), (mode, b)
    rc, small, err = _raw(coarse, W, lat, consts, mode, chunk=256)            # chunks end mid-row and mid-lead
    assert rc == 0, err
    assert torch.equal(small, all3), mode


@pytest.mark.parametrize("mode", ["fp32", "bf16", "f16x3"])
def test_workspace_bound_is_honoured(case, mode):
    from deepphysinet_b200 import functional as Fn
    m, field, fh, coarse, W = case
    consts = m.consts(m._last_factor())
    lat = _crop(consts)
    need = lattice_bytes(3, lat.nx * lat.ny * lat.nt, mode)
    guard = 1 << 20
    buf = torch.full((need + guard,), 0xA5, dtype=torch.uint8, device="cuda")
    rc, out, err = _raw(coarse, W, lat, consts, mode, ws=buf, nbytes=need)
    assert rc == 0, err
    assert bool((buf[need:] == 0xA5).all()), "the call wrote past dpn_lattice_workspace_bytes"
    assert torch.equal(out, Fn.decoder_lattice(coarse, W, lat, consts=consts, mode=mode))
    rc, _, err = _raw(coarse, W, lat, consts, mode, ws=buf, nbytes=need - 1)
    assert rc == 10002 and "workspace too small" in err, (rc, err)


def test_out_of_domain_lattice_is_refused(case):
    from deepphysinet_b200.functional import Lattice
    m, field, fh, coarse, W = case
    consts = m.consts(m._last_factor())
    lat = Lattice.domain(consts, refine=2, nt=25)
    with pytest.raises(RuntimeError, match="lattice x range"):
        m.predict_lattice(field[:1], coarse[:1], fh[:1], lat._replace(x0=lat.sx), weights=_sample(W, 0))
    with pytest.raises(RuntimeError, match="lattice t range"):
        m.predict_lattice(field[:1], coarse[:1], fh[:1], lat._replace(nt=26), weights=_sample(W, 0))


def test_full_size_refined_domain(case):
    """Lattice.domain(refine=4, nt=25) on the 145 x 257 grid for two samples in f16x3: 29.6 M nodes in one call."""
    from deepphysinet_b200 import _native as N, functional as Fn
    from deepphysinet_b200.config import PhysicsConsts
    from oracle import lattice_oracle as LO
    m, field, fh, _, W = case
    consts = PhysicsConsts(with_clip=False)
    lat = Fn.Lattice.domain(consts, refine=4, nt=25)
    assert (lat.nx, lat.ny, lat.nt) == (1025, 577, 25)
    coarse = torch.randn(2, 5, 37, 65, 6, generator=torch.Generator().manual_seed(4)).cuda()
    W2 = Fn.DecoderWeights(*[(w[:2] if n in GENERATED else w) for n, w in zip(Fn.DecoderWeights._fields, W)])
    W2 = Fn.DecoderWeights(*[w.float().contiguous() for w in W2])
    N.release_workspaces()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    out = Fn.decoder_lattice(coarse, W2, lat, consts=consts, mode="f16x3")
    torch.cuda.synchronize()
    growth = torch.cuda.max_memory_allocated() - base - out.numel() * 4
    ws = lattice_bytes(2, lat.nx * lat.ny * lat.nt, "f16x3")
    print("full-size lattice: peak growth beyond the output %.1f MiB, lattice workspace %.1f MiB" % (growth / 2 ** 20, ws / 2 ** 20))
    assert growth <= ws + 64 * 2 ** 20, (growth, ws)
    assert torch.isfinite(out).all()
    rng = np.random.default_rng(0)
    for b in range(2):
        k, j, i = rng.integers(0, lat.nt, 2048), rng.integers(0, lat.ny, 2048), rng.integers(0, lat.nx, 2048)
        x, y, t = LO.node_coords(lat, k, j, i)
        want = LO.node_values(coarse[b].double().cpu().numpy(), _oracle_weights(W2, b), x, y, t)
        got = out[b][torch.from_numpy(k).cuda(), torch.from_numpy(j).cuda(), torch.from_numpy(i).cuda()]
        err = _normalised_err(got, want, consts)
        assert err < TOL["f16x3"], (b, err)
