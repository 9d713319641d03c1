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
  * with pde: the two operands of the vapour switch (D(p) < 0) & (q >= q_s): |D(p)| over its rms and |q - q_s| over |q_s|.
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
    geo = dict(dx=consts.dx, dy=consts.dy, lat_size=consts.lat_size, lon_size=consts.lon_size)
    col = lambda a: a.reshape(-1, 1)
    if not pde:
        pe, _ = CF.coord_features(col(x), col(y), col(t), t_span=consts.pred_t_span, **geo)
        a1, a3 = preactivations(pe, O.sine_cos_pe(cd, 16), Wb)
        return dict(a1=(a1.abs(), a1), a3=(a3.abs(), a3))
    _, _, vals, jac, st = CF.pde_fwd_bwd(col(x), col(y), col(t), col(f), cd, Wb, t_span=consts.pred_t_span,
                                         with_clip=consts.with_clip, return_stages=True, **geo)
    a1 = torch.stack([st["pe"] @ Wb["W1"][k].T + Wb["b1"][k] for k in range(6)], 1)
    a3 = torch.stack([st["nets"][k]["c"] @ Wb["Wa"][k].T + Wb["ba"][k] for k in range(6)], 1)
    q = dict(a1=(a1.abs(), a1), a3=(a3.abs(), a3))
    if consts.with_clip:
        tt = lambda v: torch.tensor(v[2:], dtype=x.dtype)
        raw = st["o"][:, 2:] * tt(CF.STD) + tt(CF.MEAN)                                   # p, T, q, rho before the clip
        q["clip_lo"] = ((raw - tt(CF.LO)).abs(), raw)
        q["clip_hi"] = ((raw - tt(CF.HI)).abs(), raw)
    u, v, p, T, qv = vals[:, 0], vals[:, 1], vals[:, 2], vals[:, 3], vals[:, 4]
    dp = jac[:, 2, 2] + u * jac[:, 2, 0] + v * jac[:, 2, 1]                              # D(p) of the vapour switch
    q_s = torch.clamp_min(O.saturation_q(p, T), 1e-6)
    q["dp"] = (dp.abs(), dp)
    q["qs"] = ((qv - q_s).abs() / q_s, None)                                                # already relative to |q_s|
    return q


def _spread(name, src):
    if src is None:
        return 1.0
    if name == "dp":
        return src.pow(2).mean(0).sqrt().clamp_min(1e-300)
    return src.std(0).clamp_min(1e-300)


def tie_free_draw(B, N, seed, guard, *, pde=True, K=6, consts=None, device="cpu"):
    """(W, pts, margin): random_decoder_weights(B, ., seed) weights (bit-identical for any point count: the generator draws the
    weights first) and, per sample, the first N of pool_size(N, guard) candidate points whose margin (module docstring) is at least
    `guard`.  `margin` is the smallest margin among the returned points.  pde=True screens the PDE path (needs K = 6);
    pde=False the values-only decoder (ReLU masks only)."""
    from deepphysinet_b200.config import PhysicsConsts
    from deepphysinet_b200.testing import random_decoder_weights
    consts = consts or PhysicsConsts()
    if pde and K != 6:
        raise ValueError("the PDE path needs all six nets")
    pool = pool_size(N, guard)
    W, cand = random_decoder_weights(B, pool, seed, device="cpu", K=K, consts=consts)
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
    dev = torch.device(device)
    W = type(W)(*[w.to(dev) for w in W])
    return W, {k: v.to(dev) for k, v in pts.items()}, worst
