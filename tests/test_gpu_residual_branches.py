"""GPU (-m gpu): strict parity of the residual physics (residual_point in csrc/dpn_common.cuh, shared by every mode) in the branches
the default draws never reach, and under constants other than the reference config's.

The draws of tests/test_gpu_strict_parity.py keep every field far inside its bounds except q's lower one, never floor q_s, and use
the default geometry and normalisation.  Here oracle/tiefree.py steers candidate points into named regimes (tiefree.regime_table)
before screening them: p, T, q and rho clipped below lo and above hi (kappa = 0: zero Jacobian row and seeds), q_s floored, the vapour
switch on and off for each of its reasons, and the exact tie q = q_s = 1e-6 (q clipped to its lo while q_s is floored), which the
switch decides by D(p) alone.  rho clipped at 1e-6 multiplies its sample's seeds by 1e7..1e10 and so gets a sample of its own.
Bounds and comparator are those of tests/test_gpu_strict_parity.py; on top of them, clipped fields must come back exactly at the
fp32 image of their bound with an exactly zero Jacobian row.
"""
import dataclasses

import numpy as np
import pytest
import torch

from oracle import closed_form as CF
from oracle import dpn_oracle as O
from oracle import tiefree as TF
from tests import test_gpu_strict_parity as S

pytestmark = pytest.mark.gpu

N_SWEEP = 1000
LATTICE_TOL = dict(fp32=1e-4, f16x3=1e-5, f16x3a=1e-5, bf16x3=1e-5, bf16=2e-2)   # tests/test_gpu_lattice.py


def _default():
    from deepphysinet_b200.config import PhysicsConsts
    return PhysicsConsts()


def custom_consts(with_clip=True):
    """Everything PhysicsConsts carries away from the reference config: dx != dy, a 97 x 181 grid, 6 h time span, a from_cfg
    normalisation whose bounds every field can reach with a shift of at most 9 (so q and rho above hi are steerable), six distinct
    loss factors and perturbed c_p / L / R_v / R_d.  q keeps lo = 1e-6, the q_s floor, so the exact tie exists; T above hi = 420 K
    floors q_s."""
    from deepphysinet_b200.config import FACTOR_KEYS, PhysicsConsts
    obs = dict(u10=dict(norm_factor=[0.5, 4.0], bound=[-500, 500]), v10=dict(norm_factor=[-0.3, 3.5], bound=[-500, 500]),
               pres=dict(norm_factor=[90000.0, 12000.0], bound=[40000, 140000]), t2=dict(norm_factor=[285.0, 20.0], bound=[200, 420]),
               q2=dict(norm_factor=[0.008, 0.006], bound=[1e-6, 0.04]), rio=dict(norm_factor=[1.1, 0.15], bound=[0.5, 1.9]))
    fac = dict(zip(FACTOR_KEYS, (1.1e3, 0.7e3, 1.3e10, 2e1, 0.6e14, 3e-7)))
    c = PhysicsConsts.from_cfg(obs, fac, dx=27000.0, dy=31000.0, lat_size=97, lon_size=181, pred_t_span=21600.0, with_clip=with_clip)
    return dataclasses.replace(c, c_p=1004.0, L=2.45e6, R_v=461.0, R_d=287.05)


def _draw(B, N, seed, regimes, consts=None):
    W, pts, margin = TF.tie_free_draw(B, N, seed, S.GUARD, consts=consts, regimes=regimes, device="cuda")
    assert margin >= S.GUARD
    print("draw %d: " % seed + " | ".join(" ".join("%s %d" % kv for kv in c.items() if kv[1]) for c in TF.branches(W, pts, consts)))
    return W, pts


def run_pde(W, pts, mode, consts, chunk=0, n_norm=0):
    from deepphysinet_b200 import testing as T
    with S.forced_chunk(chunk):
        return T.run_library(W, {k: pts[k] for k in ("x", "y", "t", "f", "coord_data")}, consts=consts, mode=mode, n_norm=n_norm)


def seed_sum_scale(W, pts, consts, n_total=None, extra=None):
    """Per weight tensor, the magnitude of the terms of each gradient entry that is a sum of seeds over points (b1, b2, bd, e, ba,
    bb, bo, wo; zero for the weight matrices), in the layout of pde_oracle's grads.  The PDE seeds change sign from point to point,
    and clipped fields and the q_s floor make some sums cancel to 1e-2..1e-3 of their terms; such a sum has no relative accuracy in
    fp32 accumulation (2.6e-5 of an fp32 bo slice) or bf16 operands.  strict_errors therefore counts no such slice as smaller than
    1/8 of this magnitude: a dropped point or tile still moves it by far more than any bound.  extra [B,N,6]: further seeds dL/do
    of the same call (the margin loss)."""
    B, N = pts["x"].shape
    out = [torch.zeros(w.shape, dtype=torch.float64) for w in W]

    def put(n, b, v):
        g = out[S.NAMES.index(n)]
        if n in TF.GENERATED:
            g[b] += v / B
        else:
            g += v / B
    for b in range(B):
        c = {k: v[b].detach().double().cpu() for k, v in pts.items()}
        Wb = TF.sample_weights(W, b)
        col = lambda k: c[k].reshape(-1, 1)
        st = CF.pde_fwd_bwd(col("x"), col("y"), col("t"), col("f"), c["coord_data"], Wb, return_stages=True,
                            **dict(CF.kwargs_of(consts), n_total=n_total or N))[4]
        dv = st["dov"].abs() + (0 if extra is None else extra[b].abs())                         # [N, 6]
        s = lambda name, x: torch.stack([(dv[:, k:k + 1] * st["nets"][k][x].abs()).sum(0) for k in range(6)])
        put("b1", b, s("b1", "qm"))
        for n in ("b2", "bd", "e"):
            put(n, b, s(n, "yv"))
        put("ba", b, s("ba", "um"))
        put("bo", b, dv.sum(0))
        put("bb", b, Wb["wo"].abs() * dv.sum(0)[:, None])
        put("wo", b, torch.stack([2 * st["nets"][k]["zc"].abs().sum(0) + Wb["Wb"][k].abs() @ st["nets"][k]["gz"].abs().sum(0)
                                  + Wb["bb"][k].abs() * dv[:, k].sum() for k in range(6)]))
    return out


def pde_ref(W, pts, consts, n_total=None):
    return dict(S.pde_oracle(W, pts, consts, n_total=n_total), grad_scale=seed_sum_scale(W, pts, consts, n_total))


def exact_clip_errors(got, ref, consts, label):
    """(label, field, side, count) of clipped points (the oracle's value sits on the bound) whose value is not the fp32 image of
    the bound or whose Jacobian row is not exactly zero; prints the clipped counts."""
    bad, seen = [], []
    vals, jac = got["vals"].cpu(), got["jac"].cpu()
    for k in range(2, 6):
        for side, bound in (("lo", consts.lo[k]), ("hi", consts.hi[k])):
            m = ref["vals"][..., k] == bound
            seen.append("%s %s %d" % (TF.FIELDS[k], side, int(m.sum())))
            wrong = int((vals[..., k][m] != torch.tensor(bound, dtype=torch.float32)).sum()) + int((jac[..., k, :][m] != 0).any(-1).sum())
            if wrong:
                bad.append((label, TF.FIELDS[k], side, wrong))
    print("%-34s clipped: %s" % (label, ", ".join(seen)))
    return bad


def sweep_cases():
    """(id, regimes per sample): each steerable regime of the reference config alone, and one mixed draw with rho below lo in a
    sample of its own."""
    names = [n for n in TF.regime_table(_default()) if n != "free"]
    cases = [(n, [[n], [n]]) for n in names]
    cases.append(("mixed", [["free"] + [n for n in names if n != "rho_lo"], ["free", "rho_lo"]]))
    return cases


SWEEP = sweep_cases()


@pytest.mark.parametrize("name,regimes", SWEEP, ids=[c[0] for c in SWEEP])
def test_branch_sweep(name, regimes):
    """B = 2, N = 1000, unchunked and with 256-point chunks: the clipped points straddle tile and chunk boundaries."""
    consts = _default()
    W, pts = _draw(2, N_SWEEP, 400 + [c[0] for c in SWEEP].index(name), regimes)
    ref = pde_ref(W, pts, consts)
    bad = []
    for chunk in (0, 256):
        for mode in S.ALL:
            got = run_pde(W, pts, mode, consts, chunk=chunk)
            label = "%s chunk %d" % (name, chunk)
            bad += S.check(got, ref, mode, label) + exact_clip_errors(got, ref, consts, label)
    assert not bad, bad


def test_field_clipped_at_every_point_of_a_sample():
    """p below lo at every point of sample 0: that sample's p net gets no seed, so its generated-weight slices must be exactly zero
    (the PDE path through zscale_kernel's clamped scale); sample 1 seeds every net."""
    consts = _default()
    W, pts = _draw(2, 600, 430, [["p_lo"], ["free"]])
    ref = pde_ref(W, pts, consts)
    for n in TF.GENERATED:
        assert not ref["grads"][S.NAMES.index(n)][0, 2].any(), n
    bad = []
    for mode in S.ALL:
        got = run_pde(W, pts, mode, consts)
        bad += S.check(got, ref, mode, "p clipped in all of sample 0") + exact_clip_errors(got, ref, consts, "p clipped, sample 0")
    assert not bad, bad


# ---------------------------------------------------------------------------------------------------------------------------------
# the closed interval [lo, hi]
# ---------------------------------------------------------------------------------------------------------------------------------
def interval_case(N=640, seed=440, guard=S.GUARD, device="cuda"):
    """Nets p and T with wo = bo = 0, so o = coord_data exactly and u = Wb^T wo = 0 (the zero-u scale clamps sWaU, sUM, sY, sQ), and
    a normalisation whose std is a power of two and mean a multiple of it, so o * std + mean is exact: p in [65536, 131072] (mean
    90112 = 11 * 8192, std 8192), T in [240, 368] (mean 288 = 18 * 16, std 16).  Four of five points sit on a bound of p and of T
    or one fp32 ulp outside it, the fifth inside.  Both nets then have a zero Jacobian and zero generated-weight gradients; kappa is
    visible only in their dwo / dbo, which sum the seeds of the points kappa keeps.  The points are screened like tie_free_draw's,
    except for the p and T clip distances, which are zero on purpose."""
    from deepphysinet_b200.testing import random_decoder_weights
    c0 = _default()
    mean, std, lo, hi = list(c0.mean), list(c0.std), list(c0.lo), list(c0.hi)
    mean[2], std[2], lo[2], hi[2] = 90112.0, 8192.0, 65536.0, 131072.0
    mean[3], std[3], lo[3], hi[3] = 288.0, 16.0, 240.0, 368.0
    consts = dataclasses.replace(c0, mean=tuple(mean), std=tuple(std), lo=tuple(lo), hi=tuple(hi))
    pool = 4 * N
    W, cand = random_decoder_weights(1, pool, seed, device="cpu", consts=consts)
    W = W._replace(wo=W.wo.clone(), bo=W.bo.clone())
    W.wo[2:4] = 0
    W.bo[2:4] = 0
    cd = cand["coord_data"].clone()
    f32 = lambda v: torch.tensor(v, dtype=torch.float32)
    i = torch.arange(pool)
    for k in (2, 3):                                              # (lo - mean) / std = -3, (hi - mean) / std = 5 for both
        edge = torch.stack([f32(-3.0), torch.nextafter(f32(-3.0), f32(-1e9)), f32(5.0), torch.nextafter(f32(5.0), f32(1e9))])
        sel = i % 5 < 4
        cd[0, sel, k] = edge[(i[sel] + k) % 4]
    cand = dict(cand, coord_data=cd)
    c = {key: v[0].double() for key, v in cand.items()}
    qs = TF._quantities(TF.sample_weights(W, 0), c["x"], c["y"], c["t"], c["f"], c["coord_data"], consts, True)
    for key in ("clip_lo", "clip_hi"):                            # p and T sit on their bounds on purpose
        d, src = qs[key]
        qs[key] = (d[:, 2:], src[:, 2:])
    m = torch.stack([(d / TF._spread(n, src)).reshape(d.shape[0], -1).amin(1) for n, (d, src) in qs.items()], 1).amin(1)
    keep = torch.nonzero(m >= guard).flatten()[:N]
    assert len(keep) == N
    pts = {key: v[:, keep].contiguous().to(device) for key, v in cand.items()}
    return type(W)(*[w.to(device) for w in W]), pts, consts


def test_closed_interval_at_the_bounds():
    W, pts, consts = interval_case()
    ref = pde_ref(W, pts, consts)
    raw = pts["coord_data"][0, :, 2:4].double().cpu() * torch.tensor(consts.std[2:4]) + torch.tensor(consts.mean[2:4])
    lo, hi = torch.tensor(consts.lo[2:4]), torch.tensor(consts.hi[2:4])
    on, out = ((raw == lo) | (raw == hi)).sum(0), ((raw < lo) | (raw > hi)).sum(0)
    print("p, T on a bound %s, one ulp outside %s" % (on.tolist(), out.tolist()))
    assert (on >= 100).all() and (out >= 100).all()
    bad = []
    for mode in S.ALL:
        got = run_pde(W, pts, mode, consts)
        bad += S.check(got, ref, mode, "closed interval") + exact_clip_errors(got, ref, consts, "closed interval")
        for n in ("W1", "b1", "W2", "b2", "e", "Wd", "bd", "Wa", "ba", "Wb", "bb"):
            g = got["grads"][S.NAMES.index(n)]
            assert not (g[:, 2:4] if n in TF.GENERATED else g[2:4]).any(), (mode, n)
        assert not got["jac"][..., 2:4, :].any(), mode
    assert not bad, bad


# ---------------------------------------------------------------------------------------------------------------------------------
# non-default constants, n_norm
# ---------------------------------------------------------------------------------------------------------------------------------
def _margin_ref(W, pts, consts, target, beta, factor):
    """pde_margin_residual's fp64 composition under `consts` (as test_gpu_strict_parity.test_fused_margin_strict)."""
    B = pts["x"].shape[0]
    ref = S.pde_oracle(W, pts, consts)
    leaves = [w.detach().double().cpu().requires_grad_(True) for w in W]
    mref, o_ref, g_m = [], [], []
    for b in range(B):
        Wb = {n: (l[b] if n in TF.GENERATED else l) for n, l in zip(S.NAMES, leaves)}
        col = lambda k: pts[k][b].double().cpu().reshape(-1, 1)
        pe = O.encoding_coord(col("x"), col("y"), col("t"), consts.dx, consts.dy, consts.lat_size, consts.lon_size, consts.pred_t_span)
        o = torch.cat(O.decode_generated(pe, pts["coord_data"][b].double().cpu(), Wb), 1)
        ml = torch.nn.functional.smooth_l1_loss(o, target[b].double().cpu(), beta=beta, reduction="none").mean() * factor
        g_m.append(torch.autograd.grad(ml, o, retain_graph=True)[0])
        (ml / B).backward()
        mref.append(ml.detach())
        o_ref.append(o.detach())
    return dict(terms=torch.cat([ref["terms"], torch.stack(mref)[:, None]], 1), vals=torch.stack(o_ref),
                grads=[g + l.grad for g, l in zip(ref["grads"], leaves)],
                grad_scale=seed_sum_scale(W, pts, consts, extra=torch.stack(g_m)))


@pytest.mark.parametrize("with_clip", [True, False], ids=["clip", "noclip"])
def test_non_default_constants(with_clip):
    """custom_consts on the PDE call (every mode, unchunked and 384-point chunks), decoder_values + backward and
    pde_margin_residual.  With clip every regime of custom_consts is steered in, q and rho above hi included; without clip the
    fields pass their bounds unclipped (T above 420 K still floors q_s, q below 1e-6 turns the switch off)."""
    from deepphysinet_b200 import functional as Fn
    consts = custom_consts(with_clip)
    names = list(TF.regime_table(consts)) if with_clip else ["free", "T_hi", "q_lo", "p_hi"]
    W, pts = _draw(2, N_SWEEP, 450 + with_clip, names, consts)
    ref = pde_ref(W, pts, consts)
    xyz = (pts["x"], pts["y"], pts["t"])
    g_o = S._seeds((2, N_SWEEP, 6), 14)
    ref_dec = S.decoder_oracle(W, pts["coord_data"], g_o, xyz=xyz, consts=consts)
    beta, factor = 0.1, 1.0e6
    target = pts["coord_data"] + 0.2 * torch.randn(2, N_SWEEP, 6, generator=torch.Generator().manual_seed(15)).cuda()
    ref_m = _margin_ref(W, pts, consts, target, beta, factor)
    tag = "custom consts, %s" % ("clip" if with_clip else "no clip")
    bad = []
    for mode in S.ALL:
        for chunk in (0, 384):
            got = run_pde(W, pts, mode, consts, chunk=chunk)
            bad += S.check(got, ref, mode, "%s, chunk %d" % (tag, chunk))
            if with_clip:
                bad += exact_clip_errors(got, ref, consts, "%s, chunk %d" % (tag, chunk))
        leaves = [w.detach().clone().requires_grad_(True) for w in W]
        o = Fn.decoder_values(None, pts["coord_data"], Fn.DecoderWeights(*leaves), xyz=xyz, consts=consts, mode=mode)
        (o * g_o).sum().backward()
        bad += S.check(dict(vals=o.detach(), grads=[l.grad for l in leaves]), ref_dec, mode, "%s, decoder" % tag)
        if mode in S.STRICT:
            a = [w.detach().clone().requires_grad_(True) for w in W]
            total, terms, mloss, o = Fn.pde_margin_residual(pts["x"], pts["y"], pts["t"], pts["f"], pts["coord_data"], target,
                                                            Fn.DecoderWeights(*a), beta=beta, factor=factor, consts=consts, mode=mode)
            total.backward()
            bad += S.check(dict(terms=torch.cat([terms, mloss[:, None]], 1), vals=o, grads=[l.grad for l in a]), ref_m, mode,
                           "%s, margin" % tag)
    assert not bad, bad


def test_n_norm_differs_from_n():
    """A call on N points whose loss means divide by n_norm = 3N (one shard of a point-sharded batch), in every strict mode."""
    consts = _default()
    W, pts = _draw(2, 700, 460, ["free", "q_lo", "T_hi", "tie"])
    ref = pde_ref(W, pts, consts, n_total=3 * 700)
    bad = []
    for mode in S.STRICT:
        bad += S.check(run_pde(W, pts, mode, consts, n_norm=3 * 700), ref, mode, "n_norm = 3N")
    assert not bad, bad


# ---------------------------------------------------------------------------------------------------------------------------------
# sampler, query generator and lattice away from the default geometry
# ---------------------------------------------------------------------------------------------------------------------------------
GEO = dict(cells_per_coarse=3.0, t_step=3 * 3600.0)
LAT = dict(begin_lat=-12.5, deg_per_cell=0.5)


def test_sampler_queries_and_lattice_at_dx_ne_dy():
    """The geometry of custom_consts (dx 27 km, dy 31 km, 97 x 181 grid), 3 fine cells per coarse cell, a 3 h coarse time step and
    another begin_lat / deg_per_cell.  The coarse stack [B, 9, 33, 61, 6] covers the grid and 24 h."""
    from deepphysinet_b200 import functional as Fn
    from deepphysinet_b200.testing import random_decoder_weights
    from oracle import lattice_oracle as LO
    from oracle import query_oracle as QO
    from oracle import sampler_oracle as SO
    consts = custom_consts()
    B, N = 2, 5000
    coarse = torch.randn(B, 9, 33, 61, 6, generator=torch.Generator().manual_seed(16)).cuda()
    x, y, t, cd, f = Fn.generate_queries(B, N, seed=21, consts=consts, t_steps=9, dt=3 * 3600.0, coarse=coarse, **GEO, **LAT)
    ox, oy, ot = QO.generate(B, N, seed=21, lat_size=97, lon_size=181, t_steps=9, dx=27000.0, dy=31000.0, dt=3 * 3600.0)
    assert np.array_equal(x.cpu().numpy(), ox) and np.array_equal(y.cpu().numpy(), oy) and np.array_equal(t.cpu().numpy(), ot)
    assert y.max().item() > 96 * 27000.0                       # y spans dy * (lat_size - 1), not dx * (lat_size - 1)
    cd2, f2 = Fn.sample_field(coarse, x, y, t, consts=consts, **GEO, **LAT)
    assert torch.equal(cd, cd2) and torch.equal(f, f2)
    worst = [0.0, 0.0]
    for b in range(B):
        want = SO.trilinear(coarse[b].double().cpu().numpy(), ox[b].astype(np.float64), oy[b].astype(np.float64), ot[b].astype(np.float64),
                            dx=consts.dx, dy=consts.dy, **GEO)
        np.testing.assert_allclose(cd[b].cpu().numpy(), want, rtol=2e-6, atol=2e-6)
        fw = SO.coriolis(oy[b].astype(np.float64), dy=consts.dy, **LAT)
        np.testing.assert_allclose(f[b].cpu().numpy(), fw, rtol=1e-6, atol=1e-12)
        worst = [max(worst[0], float(np.abs(cd[b].cpu().numpy() - want).max())), max(worst[1], float(np.abs(f[b].cpu().numpy() - fw).max()))]
    print("sampler at dx != dy: coord_data max abs err %.1e, coriolis %.1e" % tuple(worst))
    W, _ = random_decoder_weights(B, 1, 22, consts=consts)
    lat = Fn.Lattice.domain(consts, refine=2, t0=1800.0, st=2400.0, nt=3)
    lat = lat._replace(x0=5 * lat.sx, nx=37, y0=7 * lat.sy, ny=29)          # 3219 nodes per sample
    want = [LO.lattice_values(coarse[b].double().cpu().numpy(), TF.sample_weights(W, b), lat, dx=consts.dx, dy=consts.dy,
                              lat_size=consts.lat_size, lon_size=consts.lon_size, pred_t_span=consts.pred_t_span, consts=consts, **GEO)
            for b in range(B)]
    for mode in S.ALL:
        got = Fn.decoder_lattice(coarse, W, lat, consts=consts, mode=mode, **GEO)
        err = 0.0
        for b in range(B):
            for k in range(6):
                a = (got[b, ..., k].double().cpu() - consts.mean[k]) / consts.std[k]
                r = (want[b][..., k] - consts.mean[k]) / consts.std[k]
                err = max(err, ((a - r).norm() / r.norm()).item())
        print("lattice at dx != dy, custom normalisation %-6s normalised err %.1e" % (mode, err))
        assert err < LATTICE_TOL[mode], (mode, err)
