"""Threshold-free draws: decoder weights and query points on which no ReLU mask bit, clip bound or vapour switch lies within
rounding distance of its threshold.

TEST INFRASTRUCTURE ONLY (see oracle/dpn_oracle.py header).  A mask bit that flips under a mode's rounding moves the Jacobian and
the J-side gradients of a draw by 1e-4..1e-3 in every arithmetic mode (DESIGN.md section 6), so parity on an arbitrary draw can
only be checked statistically.  On a draw whose every threshold decision clears a guard far above the mode's error, the kernels
compute the same masks as exact arithmetic and can be held to strict per-sample, per-net and per-point bounds
(tests/test_gpu_strict_parity.py).

The margin of a point is computed in fp64 from the point's fp32 inputs and is the minimum of
  * |a1| and |a3| of every unit of every net, each over that unit's standard deviation (a1 = PE W1^T + b1, a3 = c Wa^T + ba);
  * with pde and with_clip: |raw - lo| and |raw - hi| over the field's standard deviation, for p, T, q and rho;
  * with pde and without clip: |rho|, |rho + 1e-6| and |p + 1e-6| over their standard deviation (the poles of the residuals);
  * with pde: the two operands of the vapour switch (D(p) < 0) & (q >= q_s): |D(p)| over its rms (unless p's Jacobian row is exactly
    zero, as when p is clipped: then D(p) = 0 exactly) and |q - q_s| over |q_s|; for
    the exact tie q = q_s = 1e-6 (q clipped to its lo while q_s is floored) the distance of q_s from its floor over 1e-6.
All constants (normalisation, bounds, loss factors, geometry) are those of `consts`.  `regimes` steers candidates into the branches
of the residual physics (regime_table) before they are screened.
The spreads are estimated on the first SCALE_POINTS candidates of each sample; they only set the unit the guard is measured in.
"""
import torch

from . import closed_form as CF
from . import dpn_oracle as O

# guard per mode: 30x or more above f16x3's operand and accumulation error (<= 3e-6 of a unit's spread), ~17x above bf16x3's
# operand error (2.9e-5).  Plain bf16 (operand error ~4e-3) cannot be made threshold-free.
GUARD = dict(fp32=1e-4, f16x3=1e-4, f16x3a=1e-4, bf16x3=5e-4)
SCALE_POINTS = 4096                  # candidates per sample the spreads are estimated on (also the evaluation chunk)
GENERATED = ("W1", "b1", "W2", "b2", "e")
FIELDS = ("u", "v", "p", "T", "q", "rho")

MAX_SHIFT = 40.0


def regime_table(consts):
    """Branch-steering regimes for `consts`: name -> ({field index: shift of coord_data[..., field] in normalised units}, branches of
    `branches` the regime must reach).  The skip input adds to the net's output one-for-one, so a shift of (bound - mean) / std -/+ 2
    puts the field two standard deviations of the normalised outputs beyond its bound.  'tie' clips T above hi (which floors q_s
    when e_s(T_hi) > p / 0.378, as for the reference's 500 K) and q below lo = 1e-6: the exact tie q = q_s = 1e-6.
    Only regimes with every |shift| <= MAX_SHIFT are returned: the kernels form the data-PE argument coord_data * band in fp32, as
    the reference does, and its rounding (|arg| 2^-24, band <= 16) moves values and Wd slices by up to 7e-7 at a shift of 60
    (rho above 10 under the reference config) - too close to the fp32 mode's bounds; q above 10 needs 1600."""
    lo = lambda i: (consts.lo[i] - consts.mean[i]) / consts.std[i] - 2.0
    hi = lambda i: (consts.hi[i] - consts.mean[i]) / consts.std[i] + 2.0
    table = dict(free=({}, ("switch_on", "off_by_Dp", "off_by_q")))
    for i, name in enumerate(FIELDS[2:], 2):
        table[name + "_lo"] = ({i: lo(i)}, (name + "<lo",))
        table[name + "_hi"] = ({i: hi(i)}, (name + ">hi",))
    table["tie"] = ({3: hi(3), 4: lo(4)}, ("tie_on", "tie_off"))
    return {k: v for k, v in table.items() if all(abs(d) <= MAX_SHIFT for d in v[0].values())}


def pool_size(N, guard):
    """Candidates drawn per sample: about 84 % of the points clear 1e-4 and 35 % clear 5e-4 on random_decoder_weights draws."""
    return (2 if guard <= 1e-4 else 4) * N + 64


def sample_weights(W, b, dtype=torch.float64):
    """Per-sample weight dict (closed_form / dpn_oracle layout) of a DecoderWeights batch, on the CPU."""
    return {n: (w[b] if n in GENERATED else w).detach().to("cpu", dtype) for n, w in zip(W._fields, W)}


def preactivations(pe, pe6, Wb):
    """fp64 pre-activations (a1 [N,K,256], a3 [N,K,256]) of the K nets, as closed_form.pde_fwd_bwd forms them."""
    a1s, a3s = [], []
    for k in range(Wb["W1"].shape[0]):
        a1 = pe @ Wb["W1"][k].T + Wb["b1"][k]
        c = torch.relu(a1) @ Wb["W2"][k].T + pe6 @ Wb["Wd"][k].T + (Wb["b2"][k] + Wb["bd"][k] + Wb["e"][k])
        a1s.append(a1)
        a3s.append(c @ Wb["Wa"][k].T + Wb["ba"][k])
    return torch.stack(a1s, 1), torch.stack(a3s, 1)


def _quantities(Wb, x, y, t, f, cd, consts, pde):
    """Threshold distances of n points: dict name -> (distance [n, ...], source of its spread [n, ...]) in fp64."""
    kw = CF.kwargs_of(consts)
    col = lambda a: a.reshape(-1, 1)
    if not pde:
        pe, _ = CF.coord_features(col(x), col(y), col(t), kw["dx"], kw["dy"], kw["lat_size"], kw["lon_size"], kw["t_span"])
        a1, a3 = preactivations(pe, O.sine_cos_pe(cd, 16), Wb)
        return dict(a1=(a1.abs(), a1), a3=(a3.abs(), a3))
    _, _, vals, jac, st = CF.pde_fwd_bwd(col(x), col(y), col(t), col(f), cd, Wb, return_stages=True, **kw)
    a1 = torch.stack([st["pe"] @ Wb["W1"][k].T + Wb["b1"][k] for k in range(6)], 1)
    a3 = torch.stack([st["nets"][k]["c"] @ Wb["Wa"][k].T + Wb["ba"][k] for k in range(6)], 1)
    q = dict(a1=(a1.abs(), a1), a3=(a3.abs(), a3))
    tt = lambda v: torch.tensor(v[2:], dtype=x.dtype)
    raw = st["o"][:, 2:] * tt(consts.std) + tt(consts.mean)                               # p, T, q, rho before the clip
    if consts.with_clip:
        q["clip_lo"] = ((raw - tt(consts.lo)).abs(), raw)
        q["clip_hi"] = ((raw - tt(consts.hi)).abs(), raw)
    else:                   # poles of the residuals: 1/rho, 1/(rho + eps), 1/(p + eps), where rounding is amplified without bound
        p_, r_ = raw[:, 0:1], raw[:, 3:4]
        q["pole"] = (torch.cat([r_.abs(), (r_ + 1e-6).abs(), (p_ + 1e-6).abs()], 1), torch.cat([r_, r_, p_], 1))
    u, v, p, T, qv = vals[:, 0], vals[:, 1], vals[:, 2], vals[:, 3], vals[:, 4]
    dp = jac[:, 2, 2] + u * jac[:, 2, 0] + v * jac[:, 2, 1]                              # D(p) of the vapour switch
    qs_raw = O.saturation_q(p, T)
    q_s = torch.clamp_min(qs_raw, 1e-6)
    # a Jacobian row of p that is exactly zero (p clipped, or a p net with wo = 0) is zero in every arithmetic: D(p) = 0 exactly
    q["dp"] = (torch.where((jac[:, 2] == 0).all(1), torch.inf, dp.abs()), dp)
    # |q - q_s| relative to q_s.  The exact tie q = q_s (q clipped to lo = 1e-6 while q_s is floored to 1e-6) is decided
    # (q >= q_s) in any arithmetic that keeps both constants exact; its margin is that of the floor decision instead.
    tie = qv == q_s
    q["qs"] = (torch.where(tie, (qs_raw - 1e-6).abs() / 1e-6, (qv - q_s).abs() / q_s), None)
    return q


def branches(W, pts, consts=None):
    """Per sample, the number of points that take each branch of the residual physics (fp64, closed_form): raw value below lo /
    above hi per field (with clip: kappa = 0), the q_s floor, the vapour switch on, off because D(p) >= 0 (q >= q_s), off because q < q_s
    (D(p) < 0), and the exact tie q = q_s with the switch on / off.  Returns a list (one dict name -> count per sample)."""
    from deepphysinet_b200.config import PhysicsConsts
    consts = consts or PhysicsConsts()
    kw = CF.kwargs_of(consts)
    out = []
    for b in range(pts["x"].shape[0]):
        c = {k: v[b].detach().double().cpu() for k, v in pts.items()}
        col = lambda k: c[k].reshape(-1, 1)
        _, _, vals, jac, st = CF.pde_fwd_bwd(col("x"), col("y"), col("t"), col("f"), c["coord_data"], sample_weights(W, b),
                                             return_stages=True, **kw)
        raw = st["o"] * torch.tensor(consts.std, dtype=torch.float64) + torch.tensor(consts.mean, dtype=torch.float64)
        n = {}
        for i, name in enumerate(FIELDS[2:], 2):                          # u and v are never clipped
            n[name + "<lo"] = int((raw[:, i] < consts.lo[i]).sum())
            n[name + ">hi"] = int((raw[:, i] > consts.hi[i]).sum())
        u, v, p, T, qv = vals[:, 0], vals[:, 1], vals[:, 2], vals[:, 3], vals[:, 4]
        dp = jac[:, 2, 2] + u * jac[:, 2, 0] + v * jac[:, 2, 1]
        qs_raw = O.saturation_q(p, T)
        q_s = torch.clamp_min(qs_raw, 1e-6)
        on, tie = (dp < 0) & (qv >= q_s), qv == q_s
        n.update({"qs_floor": int((qs_raw < 1e-6).sum()), "switch_on": int(on.sum()), "off_by_Dp": int(((dp >= 0) & (qv >= q_s)).sum()),
                  "off_by_q": int(((dp < 0) & (qv < q_s)).sum()), "tie_on": int((tie & on).sum()), "tie_off": int((tie & ~on).sum())})
        out.append(n)
    return out


def _spread(name, src):
    if src is None:
        return 1.0
    if name == "dp":
        return src.pow(2).mean(0).sqrt().clamp_min(1e-300)
    return src.std(0).clamp_min(1e-300)


def tie_free_draw(B, N, seed, guard, *, pde=True, K=6, consts=None, device="cpu", regimes=None, min_count=4):
    """(W, pts, margin): random_decoder_weights(B, ., seed) weights (bit-identical for any point count: the generator draws the
    weights first) and, per sample, the first N of pool_size(N, guard) candidate points whose margin (module docstring) is at least
    `guard`.  `margin` is the smallest margin among the returned points.  pde=True screens the PDE path (needs K = 6);
    pde=False the values-only decoder (ReLU masks only).

    regimes: names of regime_table(consts), one sequence for every sample or a list of B sequences.  Candidate i of sample b is steered into
    regime regimes[b][i % len(regimes[b])] (its coord_data shifted, then rounded to fp32) before it is screened, so the screen sees
    the point the kernels get; pts["regime"] [B,N] holds each kept point's index into its sample's sequence.  Each regime must
    then keep at least `min_count` points and each of its branches be taken by at least `min_count` of them."""
    from deepphysinet_b200.config import PhysicsConsts
    from deepphysinet_b200.testing import random_decoder_weights
    consts = consts or PhysicsConsts()
    if pde and K != 6:
        raise ValueError("the PDE path needs all six nets")
    if regimes is not None and isinstance(regimes[0], str):
        regimes = [regimes] * B
    table = regime_table(consts)
    pool = pool_size(N, guard)
    W, cand = random_decoder_weights(B, pool, seed, device="cpu", K=K, consts=consts)
    if regimes is not None:
        label = torch.stack([torch.arange(pool) % len(regimes[b]) for b in range(B)])
        cd = cand["coord_data"].double()
        for b in range(B):
            for r, name in enumerate(regimes[b]):
                for k, shift in table[name][0].items():
                    cd[b, label[b] == r, k] += shift
        cand = dict(cand, coord_data=cd.float(), regime=label)
    keep, worst = [], float("inf")
    for b in range(B):
        Wb = sample_weights(W, b)
        c64 = {k: v[b].double() for k, v in cand.items()}
        scale, idx, marg = None, [], []
        for lo in range(0, pool, SCALE_POINTS):
            hi = min(pool, lo + SCALE_POINTS)
            qs = _quantities(Wb, c64["x"][lo:hi], c64["y"][lo:hi], c64["t"][lo:hi], c64["f"][lo:hi], c64["coord_data"][lo:hi],
                             consts, pde)
            if scale is None:                            # spreads from the first SCALE_POINTS candidates
                scale = {name: _spread(name, src) for name, (_, src) in qs.items()}
            m = torch.stack([(d / scale[name]).reshape(d.shape[0], -1).amin(1) for name, (d, _) in qs.items()], 1).amin(1)
            ok = torch.nonzero(m >= guard).flatten()
            idx.append(ok + lo)
            marg.append(m[ok])
            if sum(len(i) for i in idx) >= N:
                break
        idx, marg = torch.cat(idx)[:N], torch.cat(marg)[:N]
        if len(idx) < N:
            raise RuntimeError("tie_free_draw(B=%d, N=%d, seed=%d, guard=%g): only %d of %d candidates of sample %d clear the guard"
                               % (B, N, seed, guard, len(idx), pool, b))
        keep.append(idx)
        worst = min(worst, marg.min().item())
    pts = {k: torch.stack([v[b, keep[b]] for b in range(B)]).contiguous() for k, v in cand.items()}
    if regimes is not None:
        for b in range(B):
            for r, name in enumerate(regimes[b]):
                sel = pts["regime"][b] == r
                got = branches(W, {k: v[b:b + 1, sel] for k, v in pts.items()}, consts)[0] if sel.any() else {}
                short = {n: got.get(n, 0) for n in table[name][1] if got.get(n, 0) < min_count}
                if int(sel.sum()) < min_count or short:
                    raise RuntimeError("tie_free_draw(B=%d, N=%d, seed=%d, guard=%g): regime %s of sample %d keeps %d points, "
                                       "branches short of %d: %s" % (B, N, seed, guard, name, b, int(sel.sum()), min_count, short))
    dev = torch.device(device)
    W = type(W)(*[w.to(dev) for w in W])
    return W, {k: v.to(dev) for k, v in pts.items()}, worst
