"""CPU: the decoder-fields surface without a GPU - argument validation of dpn_decoder_jac_fwd / _bwd, the PyTorch physics of
deepphysinet_b200/physics.py against the fp64 oracle (MSE, L1, SmoothL1; the golden cases of the unmodified reference; a draw
through every branch of the residual physics), and no CPU fallback of decoder_fields."""
import contextlib
import ctypes as C

import numpy as np
import pytest
import torch
import torch.nn as nn

from deepphysinet_b200 import physics
from deepphysinet_b200.config import PhysicsConsts
from oracle import dpn_oracle as O
from oracle import tiefree as TF
from tests import helpers as H

NAMES = ("W1", "b1", "W2", "b2", "e", "Wd", "bd", "Wa", "ba", "Wb", "bb", "wo", "bo")


def _lib():
    import __graft_entry__ as g
    g.build()
    from deepphysinet_b200 import _native
    return _native


# ---------------------------------------------------------------------------------------------------------------------------------
# 1. argument validation
# ---------------------------------------------------------------------------------------------------------------------------------
FAKE = 1 << 20          # 16-byte aligned, never dereferenced: every check runs before the device is touched


def _args(K=6, **pts_kw):
    N = _lib()
    shape = N.DpnShape(B=1, N=128, K=K, mode=0, n_norm=0, seed_scale=1.0, chunk=0)
    pts = dict(x=FAKE, y=FAKE, t=FAKE, f=None, coord_pe=None, coord_data=FAKE, ref=None)
    pts.update(pts_kw)
    w = N.DpnWeights(**{n: FAKE for n in N.WEIGHT_FIELDS})
    return N, shape, N.make_consts(PhysicsConsts()), N.DpnPoints(**pts), w


def _call(which, K=6, seeds=(FAKE, FAKE), grads=True, **pts_kw):
    N, shape, cst, pts, w = _args(K, **pts_kw)
    L = N.lib()
    if which == "fwd":
        rc = L.dpn_decoder_jac_fwd(C.byref(shape), C.byref(cst), C.byref(pts), C.byref(w), FAKE, FAKE, FAKE, 1 << 40, None)
    else:
        g = N.DpnGrads(**{n: FAKE for n in N.WEIGHT_FIELDS})
        rc = L.dpn_decoder_jac_bwd(C.byref(shape), C.byref(cst), C.byref(pts), C.byref(w), seeds[0], seeds[1],
                                   C.byref(g) if grads else None, FAKE, 1 << 40, None)
    buf = C.create_string_buffer(512)
    L.dpn_last_error(buf, 512)
    return rc, buf.value.decode()


CASES = [
    ("x NULL", dict(x=None), "x, y and t are required"),
    ("y NULL", dict(y=None), "x, y and t are required"),
    ("t NULL", dict(t=None), "x, y and t are required"),
    ("coord_pe set", dict(coord_pe=FAKE), "coord_pe must be NULL"),
    ("K = 0", dict(K=0, ref=FAKE), "bad shape"),
    ("K = 7", dict(K=7, ref=FAKE), "bad shape"),
    ("ref NULL with K = 2", dict(K=2), "ref may only be NULL for K = 6"),
]


@pytest.mark.parametrize("which", ["fwd", "bwd"])
@pytest.mark.parametrize("label,kw,text", CASES, ids=[c[0] for c in CASES])
def test_argument_validation(which, label, kw, text):
    kw = dict(kw)
    K = kw.pop("K", 6)
    rc, err = _call(which, K=K, **kw)
    assert rc == 10001 and text in err, (label, rc, err)


def test_backward_seed_and_grads_validation():
    rc, err = _call("bwd", seeds=(None, None))
    assert rc == 10001 and "d_o and d_jac are both NULL" in err, err
    rc, err = _call("bwd", grads=False)
    assert rc == 10001 and "grads is NULL" in err, err


# ---------------------------------------------------------------------------------------------------------------------------------
# 2. physics.py against the oracle in fp64
# ---------------------------------------------------------------------------------------------------------------------------------
def fields64(x, y, t, cd, W, consts):
    """o [N,6] and jac [N,6,3] (d/dx, d/dy, d/dt, before inverse_norm) from fp64 autograd through dpn_oracle.decoder_net, with
    create_graph so that both stay differentiable w.r.t. the weights.  W: oracle layout (sample axis squeezed)."""
    x, y, t = (a.detach().clone().requires_grad_(True) for a in (x, y, t))
    pe = O.encoding_coord(x, y, t, consts.dx, consts.dy, consts.lat_size, consts.lon_size, consts.pred_t_span)
    outs = O.decode_generated(pe, cd, W)
    jac = torch.stack([torch.cat(torch.autograd.grad(o.sum(), (x, y, t), create_graph=True), 1) for o in outs], 1)
    return torch.cat(outs, 1), jac


def _factors(consts):
    return dict(zip(("motion_u_factor", "motion_v_factor", "continuous_factor", "energy_factor", "vapor_factor", "gas_factor"),
                    consts.factor))


@contextlib.contextmanager
def oracle_criterion(criterion):
    """The oracle with another criterion: dpn_oracle.residual_losses calls the module's _mse(lhs, rhs) for each of the six equations,
    with the reference's lhs / rhs split, so swapping that one name gives the reference's place_one_batch with `criterion`."""
    orig = O._mse
    O._mse = criterion
    try:
        yield
    finally:
        O._mse = orig


def _oracle(x, y, t, f, cd, W, consts, criterion):
    with oracle_criterion(criterion):
        return O.place_generated(x, y, t, f, cd, W, dx=consts.dx, dy=consts.dy, lat_size=consts.lat_size, lon_size=consts.lon_size,
                                 pred_t_span=consts.pred_t_span, with_clip=consts.with_clip, factors=_factors(consts),
                                 norm=O.norm_of(consts), c_p=consts.c_p, L=consts.L, R_v=consts.R_v, R_d=consts.R_d)


def _leaves(W, b=0):
    return {n: (w[b] if n in TF.GENERATED else w).detach().double().clone().requires_grad_(True) for n, w in zip(NAMES, W)}


CRITERIA = {"mse": nn.MSELoss(), "l1": nn.L1Loss(), "smoothl1": nn.SmoothL1Loss(beta=0.1)}


def _compare(pts, W, consts, criterion, b=0):
    col = lambda k: pts[k][b].detach().double().cpu().reshape(-1, 1)
    cd = pts["coord_data"][b].detach().double().cpu()
    Wf, Wo = _leaves(W, b), _leaves(W, b)
    o, jac = fields64(col("x"), col("y"), col("t"), cd, Wf, consts)
    terms = physics.residual_terms(o[None], jac[None], col("f").reshape(1, -1), consts, criterion)[0]
    terms.sum().backward()
    total, ref = _oracle(col("x"), col("y"), col("t"), col("f"), cd, Wo, consts, criterion)
    total.backward()
    ref = torch.stack(ref).detach()
    assert terms.dtype == torch.float64
    np.testing.assert_allclose(terms.detach().numpy(), ref.numpy(), rtol=1e-12, atol=0)
    for n in NAMES:
        assert H.rel(Wf[n].grad, Wo[n].grad) < 1e-10, n
    return terms.detach()


@pytest.mark.parametrize("crit", list(CRITERIA))
def test_physics_matches_oracle_random_draw(crit):
    from deepphysinet_b200.testing import random_decoder_weights
    W, pts = random_decoder_weights(B=1, N=96, seed=3, device="cpu")
    _compare(pts, W, PhysicsConsts(), CRITERIA[crit])


@pytest.mark.parametrize("crit", list(CRITERIA))
def test_physics_matches_oracle_in_every_regime(crit):
    """Clipped p, T, q and rho, the q_s floor and the exact tie q = q_s = 1e-6 (oracle/tiefree.py regimes)."""
    consts = PhysicsConsts()
    names = list(TF.regime_table(consts))
    W, pts, _ = TF.tie_free_draw(1, 20 * len(names), 21, 5e-4, consts=consts, regimes=names, min_count=2)
    _compare(pts, W, consts, CRITERIA[crit])


@pytest.mark.parametrize("name", H.CASES)
def test_physics_on_golden_cases(name):
    """The fields of the golden cases through physics.py with MSE give the UNMODIFIED reference's fp64 loss terms."""
    case = H.load_case(name)
    net = H.build_model(case)
    x, y, t, f, cd, field, fh = H.case_inputs(name)
    W = H.leaf_weights(net, field, fh)
    geo = H.geometry(case)
    consts = PhysicsConsts(dx=geo["dx"], dy=geo["dy"], lat_size=geo["lat_size"], lon_size=geo["lon_size"],
                           pred_t_span=geo["pred_t_span"], with_clip=geo["with_clip"])
    o, jac = fields64(x, y, t, cd, W, consts)
    terms = physics.residual_terms(o[None], jac[None], f.reshape(1, -1), consts, nn.MSELoss())[0]
    np.testing.assert_allclose(terms.detach().numpy(), case["terms64"], rtol=1e-9)


# ---------------------------------------------------------------------------------------------------------------------------------
# 3. no CPU fallback
# ---------------------------------------------------------------------------------------------------------------------------------
def test_decoder_fields_refuses_cpu_tensors():
    from deepphysinet_b200 import functional as Fn, testing as T
    W, pts = T.random_decoder_weights(B=1, N=8, device="cpu")
    with pytest.raises(RuntimeError, match="no CPU path|CUDA"):
        Fn.decoder_fields(pts["x"], pts["y"], pts["t"], pts["coord_data"], W)
