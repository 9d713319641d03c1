"""Helpers shared by tests/, bench.py and __graft_entry__.smoke(): synthetic decoder weights and
a comparison of the CUDA library against the CPU oracle.  This is the only product-side file that
imports oracle/ (lazily, inside compare_with_oracle) - it is a checker, not a code path."""
import math

import torch

from . import _native as N
from . import functional as Fn
from .config import PhysicsConsts


def random_decoder_weights(B=1, N=256, seed=0, device="cuda", K=6, out_scale=0.05, consts: PhysicsConsts = None):
    """Weights with the statistics of the reference initialisation (nn.Linear default / hyper-network
    outputs are O(1/sqrt(fan_in))) and query points per SURVEY 8(d).  Cheap: no encoder involved."""
    consts = consts or PhysicsConsts()
    g = torch.Generator().manual_seed(seed)
    u = lambda *s, fan: (torch.rand(*s, generator=g) * 2 - 1) / math.sqrt(fan)
    W = Fn.DecoderWeights(
        W1=u(B, K, 256, 192, fan=192) * 2, b1=u(B, K, 256, fan=192), W2=u(B, K, 256, 256, fan=256) * 2,
        b2=u(B, K, 256, fan=256), e=u(B, K, 256, fan=192),
        Wd=u(K, 256, 192, fan=192), bd=u(K, 256, fan=192), Wa=u(K, 256, 256, fan=256), ba=u(K, 256, fan=256),
        Wb=u(K, 256, 256, fan=256), bb=u(K, 256, fan=256), wo=u(K, 256, fan=256) * out_scale, bo=u(K, fan=256) * out_scale)
    x = torch.rand(B, N, generator=g, dtype=torch.float64) * (consts.lon_size - 1) * consts.dx
    y = torch.rand(B, N, generator=g, dtype=torch.float64) * (consts.lat_size - 1) * consts.dy
    t = torch.randint(0, 25, (B, N), generator=g).double() * 3600.0
    lat = 18.0 + y / consts.dy * 0.25
    f = 2 * 7.29e-5 * torch.sin(lat / 180 * math.pi)
    cd = 0.5 * torch.randn(B, N, 6, generator=g, dtype=torch.float64)
    pts = dict(x=x.float(), y=y.float(), t=t.float(), f=f.float(), coord_data=cd.float())
    dev = torch.device(device)
    W = Fn.DecoderWeights(*[w.to(dev) for w in W])
    pts = {k: v.to(dev) for k, v in pts.items()}
    return W, pts


def run_library(W, pts, consts=None, mode="fp32", want_fields=True, n_norm=0):
    """Library call through the autograd.Function; returns total, terms, grads (+ vals, jac)."""
    leaves = [w.detach().clone().requires_grad_(True) for w in W]
    res = Fn.pde_residual(pts["x"], pts["y"], pts["t"], pts["f"], pts["coord_data"], Fn.DecoderWeights(*leaves),
                          consts=consts, mode=mode, want_fields=want_fields, n_norm=n_norm)
    launches = N.lib().dpn_last_launch_count()
    res[0].backward()
    out = dict(total=res[0].detach(), terms=res[1], grads=[l.grad for l in leaves], launches=launches)
    if want_fields:
        out["vals"], out["jac"] = res[2], res[3]
    return out


def oracle_reference(W, pts, consts=None):
    """fp64 CPU oracle (autograd restatement of the reference) on the same inputs and every constant of `consts`; mean over
    samples."""
    from oracle import dpn_oracle as O
    consts = consts or PhysicsConsts()
    B = W.W1.shape[0]
    leaves = [w.detach().double().cpu().requires_grad_(True) for w in W]
    names = Fn.DecoderWeights._fields
    factors = dict(zip(("motion_u_factor", "motion_v_factor", "continuous_factor", "energy_factor", "vapor_factor",
                        "gas_factor"), consts.factor))
    total = 0.0
    terms, vals, jacs = [], [], []
    for b in range(B):
        Wb = {n: (l[b] if n in ("W1", "b1", "W2", "b2", "e") else l) for n, l in zip(names, leaves)}
        col = lambda k: pts[k][b].detach().double().cpu().reshape(-1, 1)
        tb, tt, v, j = O.place_generated(col("x"), col("y"), col("t"), col("f"), pts["coord_data"][b].detach().double().cpu(),
                                         Wb, dx=consts.dx, dy=consts.dy, lat_size=consts.lat_size, lon_size=consts.lon_size,
                                         pred_t_span=consts.pred_t_span, with_clip=consts.with_clip, factors=factors,
                                         norm=O.norm_of(consts), c_p=consts.c_p, L=consts.L, R_v=consts.R_v, R_d=consts.R_d,
                                         return_fields=True)
        total = total + tb / B
        terms.append(torch.stack([a.detach() for a in tt]))
        vals.append(v)
        jacs.append(j)
    total.backward()
    return dict(total=total.detach(), terms=torch.stack(terms), grads=[l.grad for l in leaves],
                vals=torch.stack(vals), jac=torch.stack(jacs))


def _rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return ((a - b).norm() / b.norm().clamp_min(1e-300)).item()


def compare_with_oracle(W, pts, consts=None, mode="fp32"):
    got = run_library(W, pts, consts, mode)
    ref = oracle_reference(W, pts, consts)
    names = Fn.DecoderWeights._fields
    grel = {n: _rel(g, r) for n, g, r in zip(names, got["grads"], ref["grads"])}
    worst = max(grel, key=grel.get)
    jac_rel = [_rel(got["jac"][..., k, :], ref["jac"][..., k, :]) for k in range(6)]
    return dict(loss_rel=abs(got["total"].item() - ref["total"].item()) / abs(ref["total"].item()),
                terms_rel=((got["terms"].cpu() - ref["terms"]).abs() / ref["terms"].abs().clamp_min(1e-300)).max().item(),
                vals_rel=max(_rel(got["vals"][..., k], ref["vals"][..., k]) for k in range(6)),
                jac_rel=max(jac_rel), grad_rel=grel, grad_rel_max=grel[worst], grad_rel_argmax=worst,
                launches=got["launches"])
