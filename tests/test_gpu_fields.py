"""GPU (-m gpu): the decoder fields (functional.decoder_fields: dpn_decoder_jac_fwd / _bwd) in every arithmetic mode.

  * values and Jacobian against fp64 autograd on threshold-free draws, at tile boundaries, for B = 1 / 3 and K = 6 / 2 (with ref);
  * the backward of  sum g_o o + sum g_jac jac  against the fp64 double backward (seeds on o only, on jac only, on both; unchunked
    and chunked) within the strict bounds of tests/test_gpu_strict_parity.py;
  * the forward is the PDE call's pass 1 (o bit-identical, std kappa jac equal to its physical Jacobian to fp32 rounding);
  * physics.residual_terms with MSE on the fields equals the fused pde_residual (terms and gradients);
  * InterfacePhysics.place_one_batch with L1 / SmoothL1 against the fp64 oracle, and with MSE still on the fused operator;
  * no backward kernels without gradients, and CUDA-graph capture of fields + L1 physics + backward.
"""
import pytest
import torch
import torch.nn as nn

from deepphysinet_b200 import _native as NAT
from deepphysinet_b200 import functional as Fn
from deepphysinet_b200 import physics
from oracle import dpn_oracle as O
from oracle import tiefree as TF
from tests import helpers as H
from tests.test_fields_cpu import oracle_criterion
from tests.test_gpu_strict_parity import ALL, BOUNDS, NAMES, STRICT, _draw, _seeds, check, forced_chunk, strict_errors

pytestmark = pytest.mark.gpu


def _consts():
    from deepphysinet_b200.config import PhysicsConsts
    return PhysicsConsts()


def fields_oracle(W, pts, ref_in=None, g_o=None, g_jac=None, consts=None):
    """fp64 autograd through dpn_oracle.decoder_net: vals [B,N,K], jac [B,N,K,3] (d/dx, d/dy, d/dt), jac_scale (sum of |terms| of
    each Jacobian entry, the comparator's cancellation floor) and, with seeds, d(sum g_o o + sum g_jac jac)/dW (double backward)."""
    consts = consts or _consts()
    B, N = pts["x"].shape
    K = W.W1.shape[1]
    leaves = [w.detach().double().cpu().requires_grad_(True) for w in W]
    vals, jacs, scales, total = [], [], [], 0.0
    sc = torch.tensor((1.0 / (consts.dx * (consts.lon_size - 1)), 1.0 / (consts.dy * (consts.lat_size - 1)), 1.0 / consts.pred_t_span),
                      dtype=torch.float64)
    bands = O.freq_bands(32).double()
    for b in range(B):
        Wb = {n: (l[b] if n in TF.GENERATED else l) for n, l in zip(NAMES, leaves)}
        x, y, t = (pts[k][b].detach().double().cpu().reshape(-1, 1).requires_grad_(True) for k in ("x", "y", "t"))
        pe = O.encoding_coord(x, y, t, consts.dx, consts.dy, consts.lat_size, consts.lon_size, consts.pred_t_span)
        cd = pts["coord_data"][b].detach().double().cpu()
        rb = (ref_in[b].detach().double().cpu() if ref_in is not None else cd)
        outs = [O.decoder_net(pe, cd, rb[:, k:k + 1], Wb["W1"][k], Wb["b1"][k], Wb["W2"][k], Wb["b2"][k], Wb["e"][k], O._net_params(Wb, k))
                for k in range(K)]
        jac = torch.stack([torch.cat(torch.autograd.grad(o.sum(), (x, y, t), create_graph=True), 1) for o in outs], 1)
        o = torch.cat(outs, 1)
        # |Jin_j dPE_j| summed per coordinate: pe column f*6 + s*3 + c is sin (s = 0) / cos (s = 1) of z_c band_f
        pv = pe.detach().reshape(N, 32, 2, 3)
        dpe = torch.stack((bands[None, :, None] * pv[:, :, 1], -bands[None, :, None] * pv[:, :, 0]), 2)
        jin = torch.stack([torch.autograd.grad(oo.sum(), pe, retain_graph=True)[0] for oo in outs], 1).reshape(N, K, 32, 2, 3)
        scales.append((jin * dpe[:, None]).abs().sum((2, 3)) * sc)
        if g_o is not None:
            total = total + (o * g_o[b].double().cpu()).sum()
        if g_jac is not None:
            total = total + (jac * g_jac[b].double().cpu()).sum()
        vals.append(o.detach())
        jacs.append(jac.detach())
    out = dict(vals=torch.stack(vals), jac=torch.stack(jacs), jac_scale=torch.stack(scales))
    if g_o is not None or g_jac is not None:
        total.backward()
        out["grads"] = [l.grad if l.grad is not None else torch.zeros_like(l) for l in leaves]
    return out


def run_fields(W, pts, mode, ref=None, g_o=None, g_jac=None, chunk=0):
    leaves = [w.detach().clone().requires_grad_(True) for w in W]
    with forced_chunk(chunk):
        o, jac = Fn.decoder_fields(pts["x"], pts["y"], pts["t"], pts["coord_data"], Fn.DecoderWeights(*leaves), ref=ref, mode=mode)
        loss = 0.0
        if g_o is not None:
            loss = loss + (o * g_o).sum()
        if g_jac is not None:
            loss = loss + (jac * g_jac).sum()
        if g_o is not None or g_jac is not None:
            loss.backward()
    out = dict(vals=o.detach(), jac=jac.detach())
    if g_o is not None or g_jac is not None:
        out["grads"] = [l.grad if l.grad is not None else torch.zeros_like(l) for l in leaves]
    return out


# ---------------------------------------------------------------------------------------------------------------------------------
# 1. forward, strict
# ---------------------------------------------------------------------------------------------------------------------------------
FWD = [(B, N, K) for N in (1, 127, 129, 257, 4225) for B in (1, 3) for K in (6, 2)]


@pytest.mark.parametrize("B,N,K", FWD, ids=["B%d_N%d_K%d" % c for c in FWD])
def test_forward_strict(B, N, K):
    """A one-point sample has no spread to normalise by: its value and Jacobian entries are sums that cancel (measured on the
    B200: fp32 mode 5e-6 on a value, 2.0e-5 on a Jacobian entry; bf16 0.6), so N = 1 checks the padding / single-tile path at
    10x the strict bounds and leaves bf16 out; every other size holds the strict bounds in every mode."""
    W, pts = _draw(B, N, 500 + N + 7 * B + K, pde=False, K=K)
    ref_in = (0.5 * _seeds((B, N, K), 20 + N)).contiguous() if K != 6 else None
    ref = fields_oracle(W, pts, ref_in)
    bad = []
    for mode in (STRICT if N == 1 else ALL):
        got = run_fields(W, pts, mode, ref=ref_in)
        if N == 1:
            bad += [(mode, g, v, w) for g, (v, w) in strict_errors(got, ref).items() if not v <= 10 * BOUNDS[mode][g.replace("_pt", "")]]
        else:
            bad += check(got, ref, mode, "fields B=%d N=%d K=%d" % (B, N, K))
    assert not bad, bad


# ---------------------------------------------------------------------------------------------------------------------------------
# 2. backward, strict
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def bwd_draw():
    return _draw(2, 1000, 510, pde=False)


@pytest.mark.parametrize("seeds", ["o", "jac", "both"])
def test_backward_strict(bwd_draw, seeds):
    """chunk 384: three chunks, the last 232 points (N is no multiple of 128).  Seeding jac alone leaves every bias gradient
    analytically zero (the Jacobian does not depend on the biases): those slices must come out exactly zero."""
    W, pts = bwd_draw
    g_o = _seeds((2, 1000, 6), 30) if seeds in ("o", "both") else None
    g_jac = _seeds((2, 1000, 6, 3), 31) if seeds in ("jac", "both") else None
    ref = fields_oracle(W, pts, g_o=g_o, g_jac=g_jac)
    bad = []
    for chunk in (0, 384):
        for mode in ALL:
            bad += check(run_fields(W, pts, mode, g_o=g_o, g_jac=g_jac, chunk=chunk), ref, mode, "seeds %s, chunk %d" % (seeds, chunk))
    assert not bad, bad


def test_backward_strict_few_nets():
    """K = 2 with ref and seeds on jac: pass 2 with tangent seeds at K < 6."""
    W, pts = _draw(2, 700, 520, pde=False, K=2)
    ref_in = (0.5 * _seeds((2, 700, 2), 32)).contiguous()
    g_o, g_jac = _seeds((2, 700, 2), 33), _seeds((2, 700, 2, 3), 34)
    ref = fields_oracle(W, pts, ref_in, g_o=g_o, g_jac=g_jac)
    bad = []
    for mode in STRICT:
        bad += check(run_fields(W, pts, mode, ref=ref_in, g_o=g_o, g_jac=g_jac), ref, mode, "K=2 with ref, both seeds")
    assert not bad, bad


# ---------------------------------------------------------------------------------------------------------------------------------
# 3. the forward is the PDE path's pass 1
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ALL)
def test_forward_is_pde_pass1(mode):
    from deepphysinet_b200.testing import random_decoder_weights
    consts = _consts()
    W, pts = random_decoder_weights(B=2, N=1000, seed=40)
    with torch.no_grad():
        o, jac = Fn.decoder_fields(pts["x"], pts["y"], pts["t"], pts["coord_data"], W, mode=mode)
        _, _, _, o_pde = Fn.pde_margin_residual(pts["x"], pts["y"], pts["t"], pts["f"], pts["coord_data"], pts["coord_data"], W, mode=mode)
        _, _, _, jac_pde = Fn.pde_residual(pts["x"], pts["y"], pts["t"], pts["f"], pts["coord_data"], W, mode=mode, want_fields=True)
    assert torch.equal(o, o_pde)
    _, phys = physics.physical_fields(o, jac, consts)
    err = ((phys - jac_pde.double()).abs() / jac_pde.double().abs().clamp_min(1e-30)).max().item()
    assert err <= 2.0 ** -22, err


# ---------------------------------------------------------------------------------------------------------------------------------
# 4. the reference physics through the fields equals the fused call
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode,chunk", [(m, 0) for m in ALL] + [("f16x3", 1000)])
def test_fields_physics_equals_fused(mode, chunk):
    from deepphysinet_b200.testing import random_decoder_weights
    consts = _consts()
    W, pts = random_decoder_weights(B=2, N=4096, seed=41)
    a = [w.detach().clone().requires_grad_(True) for w in W]
    b = [w.detach().clone().requires_grad_(True) for w in W]
    with forced_chunk(chunk):
        total, terms = Fn.pde_residual(pts["x"], pts["y"], pts["t"], pts["f"], pts["coord_data"], Fn.DecoderWeights(*a), mode=mode)
        total.backward()
        o, jac = Fn.decoder_fields(pts["x"], pts["y"], pts["t"], pts["coord_data"], Fn.DecoderWeights(*b), mode=mode)
        t2 = physics.residual_terms(o, jac, pts["f"], consts, nn.MSELoss())
        t2.sum(1).mean().backward()
    terr = ((t2.detach() - terms).abs() / terms.abs()).max().item()
    gerr = {n: H.rel(gb.grad, ga.grad) for n, ga, gb in zip(NAMES, a, b)}
    print("mode %s chunk %d: terms %.1e, worst gradient %.1e (%s)" % (mode, chunk, terr, max(gerr.values()), max(gerr, key=gerr.get)))
    assert terr <= 1e-6, terr
    assert max(gerr.values()) <= 1e-5, gerr


# ---------------------------------------------------------------------------------------------------------------------------------
# 5. place_one_batch with other criteria
# ---------------------------------------------------------------------------------------------------------------------------------
def _interface(W):
    from deepphysinet_b200 import InterfacePhysics
    from deepphysinet_b200.config import DEFAULT_OBS_NORM
    obs = {k: dict(v, norm_type="mean_norm", use_norm=True) for k, v in DEFAULT_OBS_NORM.items()}
    torch.manual_seed(0)
    m = InterfacePhysics(H.META_CFG, H.NET_CFG, obs, None, dict(img_size=(145, 257), dx=27000, dy=27000)).cuda()
    m.physics_net.decoder_weights = lambda field, fh: W            # the draw's weights stand in for the encoder's
    return m


def _place(m, pts, crit, mode):
    from deepphysinet_b200.config import DEFAULT_LOSS_FACTOR
    m.mode = mode
    B = pts["x"].shape[0]
    return m.place_one_batch(pts["x"], pts["y"], pts["t"], pts["f"], torch.zeros(B, 1, 1), pts["coord_data"], torch.zeros(B, 1, 1),
                             crit, DEFAULT_LOSS_FACTOR, 0, 0, "cuda:0")


@pytest.mark.parametrize("crit", ["l1", "smoothl1"])
def test_place_one_batch_other_criteria(crit):
    criterion = {"l1": nn.L1Loss(), "smoothl1": nn.SmoothL1Loss(beta=0.1)}[crit]
    consts = _consts()
    B, N = 2, 700
    W, pts = _draw(B, N, 530)
    leaves = [w.detach().double().cpu().requires_grad_(True) for w in W]
    factors = dict(zip(("motion_u_factor", "motion_v_factor", "continuous_factor", "energy_factor", "vapor_factor", "gas_factor"),
                       consts.factor))
    terms, total = [], 0.0
    for b in range(B):
        Wb = {n: (l[b] if n in TF.GENERATED else l) for n, l in zip(NAMES, leaves)}
        col = lambda k: pts[k][b].double().cpu().reshape(-1, 1)
        with oracle_criterion(criterion):
            tb, tt = O.place_generated(col("x"), col("y"), col("t"), col("f"), pts["coord_data"][b].double().cpu(), Wb, factors=factors,
                                       norm=O.norm_of(consts))
        total = total + tb / B
        terms.append(torch.stack([a.detach() for a in tt]))
    total.backward()
    ref = dict(terms=torch.stack(terms), grads=[l.grad for l in leaves])
    bad = []
    for mode in ("fp32", "f16x3"):
        a = [w.detach().clone().requires_grad_(True) for w in W]
        m = _interface(Fn.DecoderWeights(*a))
        loss = _place(m, pts, criterion, mode)
        loss.backward()
        assert abs(loss.item() - total.item()) <= BOUNDS[mode]["terms"] * abs(total.item())
        bad += check(dict(terms=m.last_terms, grads=[l.grad for l in a]), ref, mode, "place_one_batch %s" % crit)
    assert not bad, bad


def test_place_one_batch_mse_stays_fused(monkeypatch):
    calls = []
    orig = Fn.PDEResidualFn.apply
    monkeypatch.setattr(Fn.PDEResidualFn, "apply", lambda *a: calls.append(1) or orig(*a))
    fields = []
    orig_f = Fn.DecoderFieldsFn.apply
    monkeypatch.setattr(Fn.DecoderFieldsFn, "apply", lambda *a: fields.append(1) or orig_f(*a))
    from deepphysinet_b200.testing import random_decoder_weights
    W, pts = random_decoder_weights(B=2, N=300, seed=42)
    m = _interface(W)
    _place(m, pts, nn.MSELoss(), "f16x3")
    assert calls == [1] and not fields
    _place(m, pts, nn.L1Loss(), "f16x3")
    assert calls == [1] and fields == [1]


# ---------------------------------------------------------------------------------------------------------------------------------
# 6. launches without gradients; 7. CUDA graphs
# ---------------------------------------------------------------------------------------------------------------------------------
def test_no_grad_runs_only_the_forward():
    from deepphysinet_b200.testing import random_decoder_weights
    """The launch counter is per thread and autograd runs the backward on its own thread, so the counts compared here are those of
    forward calls on this thread: with gradients, under no_grad and with detached weights they are the same kernels."""
    W, pts = random_decoder_weights(B=2, N=1000, seed=43)
    leaves = [w.detach().clone().requires_grad_(True) for w in W]
    for mode in ("fp32", "f16x3"):
        o, jac = Fn.decoder_fields(pts["x"], pts["y"], pts["t"], pts["coord_data"], Fn.DecoderWeights(*leaves), mode=mode)
        n_fwd = NAT.lib().dpn_last_launch_count()
        assert o.grad_fn is not None and n_fwd > 0
        with torch.no_grad():
            o2, jac2 = Fn.decoder_fields(pts["x"], pts["y"], pts["t"], pts["coord_data"], Fn.DecoderWeights(*leaves), mode=mode)
        assert o2.grad_fn is None and jac2.grad_fn is None
        assert NAT.lib().dpn_last_launch_count() == n_fwd
        o3, _ = Fn.decoder_fields(pts["x"], pts["y"], pts["t"], pts["coord_data"], W, mode=mode)     # detached weights
        assert o3.grad_fn is None and NAT.lib().dpn_last_launch_count() == n_fwd


def test_double_backward_raises():
    from deepphysinet_b200.testing import random_decoder_weights
    W, pts = random_decoder_weights(B=1, N=200, seed=44)
    leaves = [w.detach().clone().requires_grad_(True) for w in W]
    o, jac = Fn.decoder_fields(pts["x"], pts["y"], pts["t"], pts["coord_data"], Fn.DecoderWeights(*leaves))
    g = torch.autograd.grad(jac.pow(2).sum(), leaves[0], create_graph=True)[0]
    with pytest.raises(RuntimeError):
        g.sum().backward()


@pytest.mark.parametrize("mode", ["fp32", "f16x3"])
def test_cuda_graph_l1_step(mode):
    from deepphysinet_b200.testing import random_decoder_weights
    consts = _consts()
    W, pts = random_decoder_weights(B=2, N=2000, seed=45)
    leaves = [w.detach().clone().requires_grad_(True) for w in W]

    def step():
        o, jac = Fn.decoder_fields(pts["x"], pts["y"], pts["t"], pts["coord_data"], Fn.DecoderWeights(*leaves), mode=mode)
        loss = physics.residual_terms(o, jac, pts["f"], consts, nn.L1Loss()).sum(1).mean()
        loss.backward()
        return loss

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            for l in leaves:
                l.grad = None
            eager = step().detach().clone()
    torch.cuda.current_stream().wait_stream(s)
    g_eager = [l.grad.clone() for l in leaves]
    for l in leaves:
        l.grad = None
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        static_loss = step()
    for _ in range(2):
        graph.replay()
        torch.cuda.synchronize()
        assert abs(static_loss.item() - eager.item()) <= 1e-6 * abs(eager.item())
        for n, l, g in zip(NAMES, leaves, g_eager):
            assert H.rel(l.grad, g) <= 1e-6, n
