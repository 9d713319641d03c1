"""Closed-form (autograd-free) restatement of the hot path in the form the CUDA kernels execute it.

TEST INFRASTRUCTURE ONLY (see oracle/dpn_oracle.py header).  Where dpn_oracle.py follows the
reference's *structure* (autograd double-backward), this file follows the product's *algorithm*
(DESIGN.md section 3) so each CUDA stage has a CPU twin exposing the same intermediate:

  pass 1   value row per point:  a1,h1 -> c -> a3,g -> o ;  reverse sweep for the per-point
           Jacobian vectors  y = 2wo + (u*m3) Wa,  Q = y w2,  Jin = (Q*m1) w1,  o_c = Jin . dPE_c
  residual interface_physics.py:97-179 on (o, o_c) -> six loss sums + seeds dL/do, dL/do_c
  pass 2   ONE combined tangent row per point (input  xt = sum_c dL/do_c dPE_c):  ht, ct, gt
  wgrad    K = points contractions of the J-side and Z-side matrices, plus column sums

It is exact (up to fp rounding) w.r.t. the reference because ReLU / clip masks are constants under
PyTorch double-backward (threshold_backward), see SURVEY.md App. A.  `rnd` emulates the operand
rounding of a tensor-core mode (identity for fp32/fp64; bf16_round, bf16_split_round, f16_split_round for the three tcgen05 modes).
"""
import torch

from . import dpn_oracle as O

MEAN = [O.OBS_NORM[k][0] for k in O.OBS_KEYS]
STD = [O.OBS_NORM[k][1] for k in O.OBS_KEYS]
LO = [O.OBS_NORM[k][2] for k in O.OBS_KEYS]
HI = [O.OBS_NORM[k][3] for k in O.OBS_KEYS]
FACT = [O.LOSS_FACTOR[k] for k in ("motion_u_factor", "motion_v_factor", "continuous_factor",
                                   "energy_factor", "vapor_factor", "gas_factor")]


def bf16_round(a):
    return a.to(torch.bfloat16).to(a.dtype)


def bf16_split_round(a):
    """Operand as the bf16x3 mode sees it: hi = bf16(a) plus lo = bf16(a - hi) (16 mantissa bits).  The emulation keeps
    the lo*lo product the kernels drop (2^-18 relative, below the representation error)."""
    hi = bf16_round(a)
    return hi + bf16_round(a - hi)


def f16_split_round(a):
    """Operand as the f16x3 mode sees it: scaled by a power of two that brings the tile's bound to 2^15 (here: its actual
    maximum, the kernels use rigorous L1-norm bounds a few binades looser - fp16 has the exponent range to absorb that),
    then hi = fp16(v) plus lo = fp16(v - hi) (22 mantissa bits)."""
    m = a.abs().max().clamp_min(1e-300)
    s = torch.exp2(torch.floor(torch.log2(32768.0 / m)))
    v = a * s
    hi = v.to(torch.float16).to(a.dtype)
    return (hi + (v - hi).to(torch.float16).to(a.dtype)) / s


def coord_features(x, y, t, dx, dy, lat_size, lon_size, t_span):
    """PE [N,192] and dPE/dz [N,192] (z-space derivative; column j differentiates w.r.t. z_{j%3})."""
    z = torch.cat((x / dx / (lon_size - 1), y / dy / (lat_size - 1), t / t_span), dim=1)   # [N,3]
    bands = O.freq_bands(32).to(z.dtype)
    arg = z[:, None, :] * bands[:, None]                                                     # [N,32,3]
    s, c = torch.sin(arg), torch.cos(arg)
    pe = torch.stack((s, c), dim=2).reshape(z.shape[0], -1)
    dpe = torch.stack((c * bands[:, None], -s * bands[:, None]), dim=2).reshape(z.shape[0], -1)
    return pe, dpe


def kwargs_of(consts):
    """pde_fwd_bwd keywords carrying every constant of a deepphysinet_b200.config.PhysicsConsts."""
    return dict(dx=consts.dx, dy=consts.dy, lat_size=consts.lat_size, lon_size=consts.lon_size, t_span=consts.pred_t_span,
                with_clip=consts.with_clip,
                phys=dict(mean=consts.mean, std=consts.std, lo=consts.lo, hi=consts.hi, fact=consts.factor, c_p=consts.c_p,
                          L=consts.L, R_v=consts.R_v, R_d=consts.R_d))


def residual_and_seeds(o, od, f, n_total, scales, with_clip=True, fact=FACT, mean=MEAN, std=STD, lo=LO, hi=HI,
                       c_p=1005.0, L=2.5e6, R_v=461.5, R_d=287.0):
    """o [N,6] normalised outputs, od [N,6,3] z-space derivatives, f [N,1]; the constants default to the reference config.
    Returns loss sums [6] (already * factor / n_total), seeds dov [N,6], dod [N,6,3], vals, jac(physical)."""
    dt = o.dtype
    mean, std = torch.tensor(mean, dtype=dt), torch.tensor(std, dtype=dt)
    lo, hi = torch.tensor(lo, dtype=dt), torch.tensor(hi, dtype=dt)
    raw = o * std + mean
    kap = torch.ones_like(raw)
    vals = raw.clone()
    if with_clip:
        kap[:, 2:] = ((raw[:, 2:] >= lo[2:]) & (raw[:, 2:] <= hi[2:])).to(dt)
        vals[:, 2:] = torch.minimum(torch.maximum(raw[:, 2:], lo[2:]), hi[2:])
    sc = torch.tensor(scales, dtype=dt)                                  # (s_x, s_y, s_t)
    jac = od * (std * 1.0)[None, :, None] * kap[:, :, None] * sc[None, None, :]
    u, v, p, T, q, r = [vals[:, i:i + 1] for i in range(6)]
    gx = lambda i: jac[:, i, 0:1]
    gy = lambda i: jac[:, i, 1:2]
    gt = lambda i: jac[:, i, 2:3]
    D = lambda i: gt(i) + u * gx(i) + v * gy(i)
    eps = 1e-6
    r1 = D(0) + gx(2) / r - f * v
    r2 = D(1) + gy(2) / r + f * u
    r3 = D(5) + r * (gx(0) + gy(1))
    r4 = c_p * D(3) - D(2) / (r + eps) + L * D(4)
    tc = T - 273.15
    e_s = 6.112 * torch.exp(17.67 * tc / (tc + 243.5)) * 100
    q_s = torch.clamp_min(0.622 * e_s / (p - 0.378 * e_s), 1e-6)
    delta = ((D(2) < 0) & (q >= q_s)).to(dt)
    Fv = (L * (1 + 0.608 * q) * R_d - c_p * R_v * T) / (c_p * R_v + T * T + L * L * q_s) * q_s * T
    K = delta * Fv / (p + eps)
    r5 = -D(2) * K + D(4)
    r6 = p - r * (1 + 0.608 * q) * R_d * T
    res = [r1, r2, r3, r4, r5, r6]
    losses = torch.stack([fact[e] * (res[e] ** 2).sum() / n_total for e in range(6)])
    a = [2.0 * fact[e] * res[e] / n_total for e in range(6)]
    dv = torch.zeros_like(vals)          # dL/d(physical value)
    dj = torch.zeros_like(jac)           # dL/d(physical derivative) [N,6,3], last = (x,y,t)
    U, V, P, TT, Q, R = range(6)

    def add_D(i, coef):                  # coef * D(i): contributions to jac(i) and to u, v
        dj[:, i, 2:3] += coef
        dj[:, i, 0:1] += coef * u
        dj[:, i, 1:2] += coef * v
        dv[:, U:U + 1] += coef * gx(i)
        dv[:, V:V + 1] += coef * gy(i)

    add_D(U, a[0]); dj[:, P, 0:1] += a[0] / r; dv[:, R:R + 1] += -a[0] * gx(P) / r ** 2; dv[:, V:V + 1] += -a[0] * f
    add_D(V, a[1]); dj[:, P, 1:2] += a[1] / r; dv[:, R:R + 1] += -a[1] * gy(P) / r ** 2; dv[:, U:U + 1] += a[1] * f
    add_D(R, a[2]); dv[:, R:R + 1] += a[2] * (gx(U) + gy(V)); dj[:, U, 0:1] += a[2] * r; dj[:, V, 1:2] += a[2] * r
    add_D(TT, a[3] * c_p); add_D(P, -a[3] / (r + eps)); add_D(Q, a[3] * L)
    dv[:, R:R + 1] += a[3] * D(P) / (r + eps) ** 2
    add_D(P, -a[4] * K); add_D(Q, a[4]); dv[:, P:P + 1] += a[4] * D(P) * delta * Fv / (p + eps) ** 2
    dv[:, P:P + 1] += a[5]
    dv[:, R:R + 1] += -a[5] * (1 + 0.608 * q) * R_d * T
    dv[:, Q:Q + 1] += -a[5] * r * 0.608 * R_d * T
    dv[:, TT:TT + 1] += -a[5] * r * (1 + 0.608 * q) * R_d
    dov = dv * std * kap
    dod = dj * (std[None, :, None] * kap[:, :, None] * sc[None, None, :])
    return losses, dov, dod, vals, jac


def pde_fwd_bwd(x, y, t, f, coord_data, W, *, dx=27000.0, dy=27000.0, lat_size=145, lon_size=257,
                t_span=86400.0, with_clip=True, rnd=lambda a: a, n_total=None, phys=None, return_stages=False):
    """One sample.  W: dict of stacked per-net tensors
       W1 [6,256,192] b1 [6,256] W2 [6,256,256] b2 [6,256] e [6,256]
       Wd [6,256,192] bd [6,256] Wa [6,256,256] ba [6,256] Wb [6,256,256] bb [6,256] wo [6,256] bo [6].
    phys: keywords of residual_and_seeds (normalisation, factors, physical constants); kwargs_of(consts) gives all of them.
    Returns (loss_terms[6], grads dict, vals [N,6], jac [N,6,3]) (+ stages dict)."""
    N = x.shape[0]
    n_total = n_total or N
    pe, dpe = coord_features(x, y, t, dx, dy, lat_size, lon_size, t_span)
    pe6 = O.sine_cos_pe(coord_data, 16)
    scales = (1.0 / (dx * (lon_size - 1)), 1.0 / (dy * (lat_size - 1)), 1.0 / t_span)
    o = torch.zeros(N, 6, dtype=x.dtype)
    od = torch.zeros(N, 6, 3, dtype=x.dtype)
    st = []
    for k in range(6):
        w1, w2, wa, wd = rnd(W["W1"][k]), rnd(W["W2"][k]), rnd(W["Wa"][k]), rnd(W["Wd"][k])
        wo = W["wo"][k]
        uvec = W["Wb"][k].T @ wo                                        # u = Wb^T wo (out_fc folded through cat_fc1.fc.2)
        a1 = rnd(pe) @ w1.T + W["b1"][k]
        h1 = torch.relu(a1)
        c = rnd(h1) @ w2.T + rnd(pe6) @ wd.T + (W["b2"][k] + W["bd"][k] + W["e"][k])
        a3 = rnd(c) @ wa.T + W["ba"][k]
        g = torch.relu(a3)
        o[:, k] = 2.0 * (c @ wo) + g @ uvec + (W["bb"][k] @ wo + W["bo"][k]) + coord_data[:, k]
        m1, m3 = (a1 > 0).to(x.dtype), (a3 > 0).to(x.dtype)
        um = uvec * m3
        yv = rnd(um) @ wa + 2.0 * wo
        qm = (rnd(yv) @ w2) * m1
        jin = rnd(qm) @ w1                                              # [N,192] = do/dPE
        od[:, k, :] = (jin * dpe).reshape(N, 64, 3).sum(1)
        st.append(dict(h1=h1, c=c, g=g, um=um, yv=yv, qm=qm, m1=m1, m3=m3, uvec=uvec, jin=jin))
    losses, dov, dod, vals, jac = residual_and_seeds(o, od, f, n_total, scales, with_clip, **(phys or {}))
    G = {k_: torch.zeros_like(v) for k_, v in W.items()}
    for k in range(6):
        s = st[k]
        w1, w2, wa = rnd(W["W1"][k]), rnd(W["W2"][k]), rnd(W["Wa"][k])
        wo = W["wo"][k]
        dv = dov[:, k:k + 1]
        xt = dod[:, k, :].repeat(1, 64) * dpe                          # column j uses seed of coordinate j%3
        ht = (rnd(xt) @ w1.T) * s["m1"]
        ct = rnd(ht) @ w2.T
        gt = (rnd(ct) @ wa.T) * s["m3"]
        zp, zh, zc, gz = dv * pe + xt, dv * s["h1"] + ht, dv * s["c"] + ct, dv * s["g"] + gt
        G["W1"][k] = rnd(s["qm"]).T @ rnd(zp)
        G["W2"][k] = rnd(s["yv"]).T @ rnd(zh)
        G["Wa"][k] = rnd(s["um"]).T @ rnd(zc)
        G["Wd"][k] = rnd(s["yv"]).T @ rnd(dv * pe6)
        G["b1"][k] = (dv * s["qm"]).sum(0)
        G["b2"][k] = G["bd"][k] = G["e"][k] = (dv * s["yv"]).sum(0)
        G["ba"][k] = (dv * s["um"]).sum(0)
        vc, vg, sdo = zc.sum(0), gz.sum(0), dv.sum()
        G["Wb"][k] = torch.outer(wo, vg)
        G["wo"][k] = 2.0 * vc + W["Wb"][k] @ vg + W["bb"][k] * sdo
        G["bb"][k] = wo * sdo
        G["bo"][k] = sdo
        s.update(xt=xt, ht=ht, ct=ct, gt=gt, zp=zp, zh=zh, zc=zc, gz=gz)
    if return_stages:
        return losses, G, vals, jac, dict(o=o, od=od, dov=dov, dod=dod, nets=st, pe=pe, dpe=dpe, pe6=pe6)
    return losses, G, vals, jac
