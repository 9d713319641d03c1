"""torch.autograd.Function wrappers over the C ABI (include/dpn_b200.h).

`PDEResidualFn` is the operator SURVEY.md 8(b) specifies: it replaces everything
`InterfacePhysics.place_one_batch` (interface_physics.py:271-320) does per query point, and the
double-backward graph `train_loss.backward()` (:506) would walk, with one library call that returns
the six loss terms AND the gradients w.r.t. the 13 decoder weight tensors.  Differentiable inputs:
the DecoderWeights tensors.  Not differentiable (as in the reference, where their .grad is never
read): x, y, t, f, coord_data.
"""
import ctypes as C
from typing import NamedTuple, Optional

import torch

from . import _native as N
from .config import PhysicsConsts


class DecoderWeights(NamedTuple):
    """Generated tensors are [B,K,...] (per sample), static ones [K,...]; see include/dpn_b200.h."""
    W1: torch.Tensor
    b1: torch.Tensor
    W2: torch.Tensor
    b2: torch.Tensor
    e: torch.Tensor
    Wd: torch.Tensor
    bd: torch.Tensor
    Wa: torch.Tensor
    ba: torch.Tensor
    Wb: torch.Tensor
    bb: torch.Tensor
    wo: torch.Tensor
    bo: torch.Tensor


def _prep(t, shape=None):
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("deepphysinet_b200 runs on CUDA (sm_100a) only - got a %s tensor; there is no CPU path" % t.device)
    t = t.detach()
    if t.dtype != torch.float32:
        t = t.float()
    if shape is not None:
        t = t.reshape(shape)
    return t.contiguous()


def _check_weights(W: DecoderWeights):
    B, K = W.W1.shape[0], W.W1.shape[1]
    exp = dict(W1=(B, K, 256, 192), b1=(B, K, 256), W2=(B, K, 256, 256), b2=(B, K, 256), e=(B, K, 256),
               Wd=(K, 256, 192), bd=(K, 256), Wa=(K, 256, 256), ba=(K, 256), Wb=(K, 256, 256), bb=(K, 256),
               wo=(K, 256), bo=(K,))
    for name, shp in exp.items():
        if tuple(getattr(W, name).shape) != shp:
            raise ValueError("DecoderWeights.%s has shape %s, expected %s" % (name, tuple(getattr(W, name).shape), shp))
    return B, K


def _weights_struct(ws):
    s = N.DpnWeights()
    for name, t in zip(N.WEIGHT_FIELDS, ws):
        setattr(s, name, t.data_ptr())
    return s


def _grads_struct(gs):
    s = N.DpnGrads()
    for name, t in zip(N.WEIGHT_FIELDS, gs):
        setattr(s, name, t.data_ptr())
    return s


def _shape(B, Np, K, mode, n_norm=0, seed_scale=1.0, chunk=0):
    return N.DpnShape(B=B, N=Np, K=K, mode=N.MODES[mode] if isinstance(mode, str) else int(mode),
                      n_norm=int(n_norm), seed_scale=float(seed_scale), chunk=int(chunk))


class PDEResidualFn(torch.autograd.Function):
    """(total, terms[B,6][, vals, jac][, margin_loss[B], o]) =
           PDEResidualFn.apply(x, y, t, f, coord_data, consts, mode, n_norm, want_fields, margin, *weights)

    x, y, t, f: [B,N] (or [N], [N,1] for B=1); coord_data [B,N,6].
    margin: None, or (target [B,N,6], beta, factor): the supervised SmoothL1 data loss of the train loop on the same points
    (interface_physics.py:464-474), fused into the call (SURVEY 8(f) N1) - then `total` = mean over samples of (six PDE terms +
    margin loss), and margin_loss [B] (float64) and the normalised values o [B,N,6] are returned as non-differentiable extras.
    total = mean over samples of the sum of the six terms (SURVEY D4: DDP sample-mean semantics);
    terms (float64, per sample, non-differentiable) are what place_one_batch logs (:303-318).
    Forward already runs the fused backward kernels and caches d(total)/d(weights); backward only
    scales them by grad_output - valid because `total` is the only differentiable output.
    """

    @staticmethod
    def forward(ctx, x, y, t, f, coord_data, consts: PhysicsConsts, mode, n_norm, want_fields, margin, *weights):
        W = DecoderWeights(*weights)
        B, K = _check_weights(W)
        if K != 6:
            raise ValueError("the PDE residual needs all six nets (u,v,p,T,q,rho)")
        dev = W.W1.device
        cd = _prep(coord_data, (B, -1, 6))
        Np = cd.shape[1]
        xs = [_prep(a, (B, Np)) for a in (x, y, t, f)]
        ws = [_prep(w) for w in W]
        need_grad = any(ctx.needs_input_grad[10:])            # False under no_grad / for detached weights: no backward kernels then
        grads = [torch.empty_like(w) for w in ws] if need_grad else None
        terms = torch.empty(B, 6, dtype=torch.float64, device=dev)
        vals = torch.empty(B, Np, 6, device=dev) if want_fields else None
        jac = torch.empty(B, Np, 6, 3, device=dev) if want_fields else None
        shape = _shape(B, Np, 6, mode, n_norm=n_norm, seed_scale=1.0 / B)
        cst = N.make_consts(consts)
        pts = N.DpnPoints(x=xs[0].data_ptr(), y=xs[1].data_ptr(), t=xs[2].data_ptr(), f=xs[3].data_ptr(),
                          coord_pe=None, coord_data=cd.data_ptr(), ref=None)
        out = N.DpnPdeOut(loss_terms=terms.data_ptr(), vals=None if vals is None else vals.data_ptr(),
                          jac=None if jac is None else jac.data_ptr())
        wstruct = _weights_struct(ws)
        gstruct = _grads_struct(grads) if need_grad else None
        wsbuf, nbytes = N.workspace(shape, dev)
        mstruct = mloss = o_norm = None
        if margin is not None:
            target, beta, factor = margin
            tg = _prep(target, (B, Np, 6))
            mloss = torch.empty(B, dtype=torch.float64, device=dev)
            o_norm = torch.empty(B, Np, 6, device=dev)
            mstruct = N.DpnMargin(target=tg.data_ptr(), beta=float(beta), factor=float(factor), loss=mloss.data_ptr(), o=o_norm.data_ptr())
        N.check(N.lib().dpn_pde_margin_fwd_bwd(C.byref(shape), C.byref(cst), C.byref(pts), C.byref(wstruct),
                                               C.byref(mstruct) if mstruct is not None else None, C.byref(out),
                                               C.byref(gstruct) if need_grad else None,
                                               N.ptr(wsbuf), nbytes, N.stream_ptr()), "dpn_pde_margin_fwd_bwd")
        ctx.grads = grads
        ctx.dtypes = [w.dtype for w in weights]
        total = terms.sum(dim=1).mean() if mloss is None else (terms.sum(dim=1) + mloss).mean()
        total = total.to(torch.float32)
        ctx.mark_non_differentiable(terms)
        ret = (total, terms)
        if want_fields:
            ctx.mark_non_differentiable(vals, jac)
            ret = ret + (vals, jac)
        if mloss is not None:
            ctx.mark_non_differentiable(mloss, o_norm)
            ret = ret + (mloss, o_norm)
        return ret

    @staticmethod
    def backward(ctx, g_total, *unused):
        if ctx.grads is None:
            return (None,) * 23
        gs = [(g * g_total).to(dt) for g, dt in zip(ctx.grads, ctx.dtypes)]
        return (None,) * 10 + tuple(gs)


class DecoderValuesFn(torch.autograd.Function):
    """o[B,N,K] = DecoderValuesFn.apply(coord_pe, x, y, t, coord_data, ref, consts, mode, *weights)
    Values of the K coordinate nets (variable_net.py:67-87).  Either coord_pe [B,N,192] or (x,y,t) is given."""

    @staticmethod
    def forward(ctx, coord_pe, x, y, t, coord_data, ref, consts: PhysicsConsts, mode, *weights):
        W = DecoderWeights(*weights)
        B, K = _check_weights(W)
        dev = W.W1.device
        cd = _prep(coord_data, (B, -1, 6))
        Np = cd.shape[1]
        pe = _prep(coord_pe, (B, Np, 192))
        xs = [_prep(a, (B, Np)) for a in (x, y, t)]
        rf = _prep(ref, (B, Np, K))
        ws = [_prep(w) for w in W]
        o = torch.empty(B, Np, K, device=dev)
        shape = _shape(B, Np, K, mode)
        cst = N.make_consts(consts)
        pts = N.DpnPoints(x=N.ptr(xs[0]), y=N.ptr(xs[1]), t=N.ptr(xs[2]), f=None, coord_pe=N.ptr(pe),
                          coord_data=cd.data_ptr(), ref=N.ptr(rf))
        wstruct = _weights_struct(ws)
        wsbuf, nbytes = N.workspace(shape, dev)
        N.check(N.lib().dpn_decoder_fwd(C.byref(shape), C.byref(cst), C.byref(pts), C.byref(wstruct), N.ptr(o),
                                        N.ptr(wsbuf), nbytes, N.stream_ptr()), "dpn_decoder_fwd")
        ctx.saved = (pe, xs, cd, rf, ws, consts, mode, B, Np, K)
        ctx.dtypes = [w.dtype for w in weights]
        ctx.need = any(ctx.needs_input_grad[8:])
        return o

    @staticmethod
    def backward(ctx, g_o):
        if not ctx.need:
            return (None,) * 21
        pe, xs, cd, rf, ws, consts, mode, B, Np, K = ctx.saved
        dev = g_o.device
        grads = [torch.empty_like(w) for w in ws]
        shape = _shape(B, Np, K, mode)
        cst = N.make_consts(consts)
        pts = N.DpnPoints(x=N.ptr(xs[0]), y=N.ptr(xs[1]), t=N.ptr(xs[2]), f=None, coord_pe=N.ptr(pe),
                          coord_data=cd.data_ptr(), ref=N.ptr(rf))
        wstruct, gstruct = _weights_struct(ws), _grads_struct(grads)
        go = _prep(g_o, (B, Np, K))
        wsbuf, nbytes = N.workspace(shape, dev)
        N.check(N.lib().dpn_decoder_bwd(C.byref(shape), C.byref(cst), C.byref(pts), C.byref(wstruct), N.ptr(go),
                                        C.byref(gstruct), N.ptr(wsbuf), nbytes, N.stream_ptr()), "dpn_decoder_bwd")
        return (None,) * 8 + tuple(g.to(dt) for g, dt in zip(grads, ctx.dtypes))


_DEFAULT_MODE = "f16x3"


def set_default_mode(mode: str):
    """Arithmetic of the dense contractions (include/dpn_b200.h, DESIGN.md section 6):
    'f16x3'  tcgen05, scaled fp16 hi+lo operands, 3 MMAs per contraction - fp32-class accuracy (default)
    'f16x3a' the same with cross-first accumulation of the mask-deciding GEMMs: 2.6x smaller pre-activation error, 6 % slower
    'bf16x3' tcgen05, bf16 hi+lo operands - ~1e-3 class          'bf16' tcgen05, plain bf16 - fastest, ~5e-2 class
    'fp32'   CUDA-core FMA - the reference arithmetic, slowest."""
    global _DEFAULT_MODE
    if mode not in N.MODES:
        raise ValueError("mode must be one of %s" % (tuple(N.MODES),))
    _DEFAULT_MODE = mode


def default_mode():
    return _DEFAULT_MODE


def pde_residual(x, y, t, f, coord_data, W: DecoderWeights, consts: Optional[PhysicsConsts] = None, mode=None,
                 n_norm=0, want_fields=False):
    consts = consts or PhysicsConsts()
    return PDEResidualFn.apply(x, y, t, f, coord_data, consts, mode or _DEFAULT_MODE, n_norm, want_fields, None, *W)


def pde_margin_residual(x, y, t, f, coord_data, target, W: DecoderWeights, beta=0.1, factor=1.0e6,
                        consts: Optional[PhysicsConsts] = None, mode=None, n_norm=0):
    """PDE residual loss AND the supervised margin (data) loss on the same points in one library call (SURVEY 8(f) N1;
    interface_physics.py:464-474 + :489-496): returns (total, terms [B,6], margin_loss [B], o [B,N,6]) with
    total = mean over samples of (sum of the six PDE terms + factor * mean smooth_l1(o - target; beta)), differentiable w.r.t.
    every DecoderWeights tensor; one forward, one reverse sweep and one backward instead of the reference's two passes."""
    consts = consts or PhysicsConsts()
    return PDEResidualFn.apply(x, y, t, f, coord_data, consts, mode or _DEFAULT_MODE, n_norm, False, (target, beta, factor), *W)


def generate_queries(B, Np, seed, offset=0, on_grid=False, consts: Optional[PhysicsConsts] = None, t_steps=25, dt=3600.0,
                     coarse=None, device=None, cells_per_coarse=4.0, t_step=6 * 3600.0, begin_lat=18.0, deg_per_cell=0.25,
                     omega=7.29e-5):
    """On-GPU query-point generator (SURVEY 8(f) N2): Philox4x32-10 draws with the distributions of
    dataset/physics_dataset.py:442-446 (interior: continuous) or :334-338 (on_grid: margin nodes); with `coarse` [B,Tt,Hc,Wc,6]
    the same launch also interpolates coord_data [B,N,6] and evaluates the Coriolis parameter f [B,N].
    Returns (x, y, t) or (x, y, t, coord_data, f), all device tensors."""
    consts = consts or PhysicsConsts()
    dev = torch.device(device) if device is not None else (coarse.device if coarse is not None else torch.device("cuda"))
    if dev.type != "cuda":
        raise RuntimeError("deepphysinet_b200 runs on CUDA (sm_100a) only; there is no CPU path")
    x, y, t = (torch.empty(B, Np, device=dev) for _ in range(3))
    G = N.DpnQueryGen(B=B, N=Np, lat_size=consts.lat_size, lon_size=consts.lon_size, t_steps=int(t_steps), on_grid=int(bool(on_grid)),
                      dx=consts.dx, dy=consts.dy, dt=float(dt), seed=int(seed) & (2 ** 64 - 1), offset=int(offset))
    S = cd = f = cz = None
    if coarse is not None:
        cz = _prep(coarse)
        if cz.dim() != 5 or cz.shape[-1] != 6 or cz.shape[0] != B:
            raise ValueError("coarse must be [B,Tt,Hc,Wc,6], got %s" % (tuple(cz.shape),))
        _, Tt, Hc, Wc, _ = cz.shape
        cd, f = torch.empty(B, Np, 6, device=dev), torch.empty(B, Np, device=dev)
        S = N.DpnSampler(B=B, N=Np, Tt=Tt, Hc=Hc, Wc=Wc, pad_=0, dx=consts.dx, dy=consts.dy, cells_per_coarse=float(cells_per_coarse),
                         t_step=float(t_step), begin_lat=float(begin_lat), deg_per_cell=float(deg_per_cell), omega=float(omega))
    with torch.cuda.device(dev):
        N.check(N.lib().dpn_generate_queries(C.byref(G), C.byref(S) if S is not None else None, N.ptr(cz), N.ptr(x), N.ptr(y), N.ptr(t),
                                             N.ptr(cd), N.ptr(f), N.stream_ptr()), "dpn_generate_queries")
    return (x, y, t) if coarse is None else (x, y, t, cd, f)


def decoder_values(coord_pe, coord_data, W: DecoderWeights, ref=None, xyz=None, consts=None, mode=None):
    """Values o [N,K] (B=1) or [B,N,K] from encoded coordinates (or raw xyz=(x,y,t))."""
    consts = consts or PhysicsConsts()
    x, y, t = xyz if xyz is not None else (None, None, None)
    o = DecoderValuesFn.apply(coord_pe, x, y, t, coord_data, ref, consts, mode or _DEFAULT_MODE, *W)
    return o[0] if coord_data.dim() == 2 else o


def sample_field(coarse, x, y, t, consts: Optional[PhysicsConsts] = None, cells_per_coarse=4.0, t_step=6 * 3600.0,
                 begin_lat=18.0, deg_per_cell=0.25, omega=7.29e-5, want_coriolis=True):
    """On-GPU query-point producer (SURVEY 8(f) N2): trilinear sample of the normalised coarse field stack
    `coarse` [B,Tt,Hc,Wc,6] at the query coordinates x, y, t [B,N] (same units as pde_residual) -> coord_data [B,N,6]
    and the Coriolis parameter f [B,N].  Replaces dataset/physics_dataset.py:477-486 / :521-526.  Not differentiable,
    exactly like the CPU interpolation it replaces."""
    consts = consts or PhysicsConsts()
    cz = _prep(coarse)
    if cz.dim() != 5 or cz.shape[-1] != 6:
        raise ValueError("coarse must be [B,Tt,Hc,Wc,6], got %s" % (tuple(cz.shape),))
    B, Tt, Hc, Wc, _ = cz.shape
    xs = [_prep(a, (B, -1)) for a in (x, y, t)]
    Np = xs[0].shape[1]
    cd = torch.empty(B, Np, 6, device=cz.device)
    f = torch.empty(B, Np, device=cz.device) if want_coriolis else None
    S = N.DpnSampler(B=B, N=Np, Tt=Tt, Hc=Hc, Wc=Wc, pad_=0, dx=consts.dx, dy=consts.dy,
                     cells_per_coarse=float(cells_per_coarse), t_step=float(t_step), begin_lat=float(begin_lat),
                     deg_per_cell=float(deg_per_cell), omega=float(omega))
    N.check(N.lib().dpn_sample_field(C.byref(S), N.ptr(cz), N.ptr(xs[0]), N.ptr(xs[1]), N.ptr(xs[2]), N.ptr(cd), N.ptr(f),
                                     N.stream_ptr()), "dpn_sample_field")
    return cd, f


class Lattice(NamedTuple):
    """Regular space-time lattice (DpnLattice, include/dpn_b200.h): node (k, j, i) sits at x = x0 + i sx, y = y0 + j sy (metres,
    the units of pde_residual) and t = t0 + k st (seconds); decoder_lattice returns [B, nt, ny, nx, 6].  A sub-region is a lattice
    with another origin and fewer nodes, e.g. Lattice.domain(consts, refine=4)._replace(x0=..., nx=...)."""
    nx: int
    ny: int
    nt: int
    x0: float
    y0: float
    t0: float
    sx: float
    sy: float
    st: float

    @classmethod
    def domain(cls, consts: PhysicsConsts, refine=1, t0=0.0, st=3600.0, nt=25):
        """The full lat_size x lon_size domain at `refine` times the training spacing, `nt` leads `st` seconds apart from t0."""
        return cls(nx=(int(consts.lon_size) - 1) * int(refine) + 1, ny=(int(consts.lat_size) - 1) * int(refine) + 1, nt=int(nt),
                   x0=0.0, y0=0.0, t0=float(t0), sx=float(consts.dx) / refine, sy=float(consts.dy) / refine, st=float(st))


@torch.no_grad()
def decoder_lattice(coarse, W: DecoderWeights, lattice: Lattice, consts: Optional[PhysicsConsts] = None, mode=None,
                    cells_per_coarse=4.0, t_step=6 * 3600.0):
    """Physical fields [B, nt, ny, nx, 6] (u,v,p,T,q,rho; inverse_norm without clip, interface_physics.py:533) of the six
    decoders on `lattice` for the B samples of W, with coord_data sampled from `coarse` [B,Tt,Hc,Wc,6] as sample_field does.
    One library call: coordinates and coord_data are generated on the GPU per chunk, and the workspace holds a values-only pass.
    Values only, like sample_field (no grad_fn)."""
    consts = consts or PhysicsConsts()
    Bw, K = _check_weights(W)
    if K != 6:
        raise ValueError("decoder_lattice needs all six nets (u,v,p,T,q,rho)")
    cz = _prep(coarse)
    if cz.dim() != 5 or cz.shape[-1] != 6 or cz.shape[0] != Bw:
        raise ValueError("coarse must be [B,Tt,Hc,Wc,6] with B = %d samples, got %s" % (Bw, tuple(cz.shape)))
    g = N.DpnLattice(nx=int(lattice.nx), ny=int(lattice.ny), nt=int(lattice.nt), pad_=0, x0=float(lattice.x0), y0=float(lattice.y0),
                     t0=float(lattice.t0), sx=float(lattice.sx), sy=float(lattice.sy), st=float(lattice.st))
    Np = g.nx * g.ny * g.nt
    if Np >= 2 ** 31:
        raise ValueError("the lattice has %d nodes per sample; at most 2**31 - 1 fit one call" % Np)
    _, Tt, Hc, Wc, _ = cz.shape
    S = N.DpnSampler(B=Bw, N=Np, Tt=Tt, Hc=Hc, Wc=Wc, pad_=0, dx=consts.dx, dy=consts.dy, cells_per_coarse=float(cells_per_coarse),
                     t_step=float(t_step), begin_lat=0.0, deg_per_cell=0.0, omega=0.0)
    shape = _shape(Bw, Np, 6, mode or _DEFAULT_MODE)
    ws = [_prep(w) for w in W]
    out = torch.empty(Bw, g.nt, g.ny, g.nx, 6, device=cz.device)
    need = C.c_size_t(0)
    N.check(N.lib().dpn_lattice_workspace_bytes(C.byref(shape), C.byref(need)), "dpn_lattice_workspace_bytes")
    with torch.cuda.device(cz.device):
        wsbuf, nbytes = N.workspace(shape, cz.device, need.value)
        N.check(N.lib().dpn_decoder_lattice(C.byref(shape), C.byref(N.make_consts(consts)), C.byref(g), C.byref(S), N.ptr(cz),
                                            C.byref(_weights_struct(ws)), N.ptr(out), N.ptr(wsbuf), nbytes, N.stream_ptr()),
                "dpn_decoder_lattice")
    return out
