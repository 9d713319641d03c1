"""The residual physics of the reference (interface_physics.py:97-179) as PyTorch on the decoder fields.

`residual_terms(o, jac, f, consts, criterion)` takes what `functional.decoder_fields` returns - the normalised outputs o [B,N,6]
and their Jacobian jac [B,N,6,3] in x, y, t - and gives the six weighted loss terms per sample [B,6].  Every operation is
differentiable, so `terms.sum(1).mean().backward()` sends d(loss)/d(o, jac) through `DecoderFieldsFn` into the library's backward
kernels.  It exists so that a loss the fused kernel does not implement - another criterion (nn.L1Loss, a weighted SmoothL1), a
changed or extra equation, per-term weights that need gradients - is a change to this file or a copy of it, not to CUDA code.

It restates the fused kernel's physics (residual_point in csrc/dpn_common.cuh) and the reference line for line: fp64 arithmetic,
inverse_norm with the clip of p, T, q, rho (torch.clip: derivative 1 on the closed interval), the Jacobian of a clipped field
scaled by that derivative, the reference's .detach() of q_s, the vapour switch and F, the q_s floor and its eps constants, and
criterion(lhs, rhs) with the reference's own lhs / rhs split of each equation, times the equation's factor.
"""
import torch

from .config import PhysicsConsts


def physical_fields(o, jac, consts: PhysicsConsts):
    """inverse_norm (interface_physics.py:232-262) of o [B,N,6] and the chain rule into jac [B,N,6,3]: (vals, jac) in fp64.
    Constants enter as Python scalars (no host-to-device copies), so the function can be captured in a CUDA graph."""
    o, jac = o.double(), jac.double()
    vals, J = [], []
    for k in range(6):
        raw = o[..., k] * consts.std[k] + consts.mean[k]
        jk = jac[..., k, :] * consts.std[k]
        if consts.with_clip and k >= 2:                                     # u, v are never clipped (:256-261)
            inside = ((raw >= consts.lo[k]) & (raw <= consts.hi[k])).to(raw.dtype)
            raw = torch.clip(raw, consts.lo[k], consts.hi[k])
            jk = jk * inside[..., None]
        vals.append(raw)
        J.append(jk)
    return torch.stack(vals, -1), torch.stack(J, -2)


def residual_terms(o, jac, f, consts: PhysicsConsts, criterion):
    """Six loss terms per sample [B,6] (fp64; order motion_u, motion_v, continuous, energy, vapor, gas) from o [B,N,6],
    jac [B,N,6,3] (d/dx, d/dy, d/dt) and the Coriolis parameter f [B,N]; criterion(lhs, rhs) is called per sample and equation
    on [N,1] columns, as the reference calls it."""
    vals, J = physical_fields(o, jac, consts)
    f = f.double().reshape(vals.shape[:2])
    col = lambda a: a[..., None]
    u, v, p, T, q, r = (col(vals[..., k]) for k in range(6))
    gx, gy, gt = (lambda k: col(J[..., k, 0])), (lambda k: col(J[..., k, 1])), (lambda k: col(J[..., k, 2]))
    D = lambda k: gt(k) + u * gx(k) + v * gy(k)                             # material derivative
    c_p, L, R_v, R_d = consts.c_p, consts.L, consts.R_v, consts.R_d
    f = col(f)
    eqs = []
    eqs.append((D(0) + gx(2) / r, f * v))                                   # :97-104
    eqs.append((D(1) + gy(2) / r, -f * u))                                  # :106-114
    cont = D(5) + r * gx(0) + r * gy(1)                                     # :116-124
    eqs.append((cont, torch.zeros_like(cont)))
    Dp, Dq = D(2), D(4)
    en = c_p * D(3) - Dp / (r + 1e-6) + L * Dq                              # :126-144
    eqs.append((en, torch.zeros_like(en)))
    tc = T - 273.15                                                         # :181-185
    e_s = 6.112 * torch.exp(17.67 * tc / (tc + 243.5)) * 100
    q_s = (0.622 * e_s / (p - 0.378 * e_s)).detach()
    q_s = torch.maximum(q_s, torch.ones_like(q_s) * 1e-6)                   # :146-175
    delta = torch.where(torch.logical_and(Dp < 0, torch.ge(q, q_s)), torch.ones_like(Dp), torch.zeros_like(Dp)).detach()
    R = (1 + 0.608 * q) * R_d
    F = ((L * R - c_p * R_v * T) / (c_p * R_v + T * T + L * L * q_s) * q_s * T).detach()
    vap = -Dp * delta * F / (p + 1e-6) + Dq
    eqs.append((vap, torch.zeros_like(vap)))
    eqs.append((p, r * (1 + 0.608 * q) * R_d * T))                          # :177-179
    B = vals.shape[0]
    return torch.stack([torch.stack([criterion(lhs[b], rhs[b]) * fac for (lhs, rhs), fac in zip(eqs, consts.factor)])
                        for b in range(B)])
