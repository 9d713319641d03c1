"""Function-preserving power-of-two reparametrisations of the decoder and a restatement of the f16x3 scale plan.

TEST INFRASTRUCTURE ONLY (see oracle/dpn_oracle.py header).  ReLU is positively homogeneous and the folded output layer is linear,
so the rescalings below leave values, Jacobian and loss terms unchanged in exact arithmetic while the f16x3 scale plan
(bounds_kernel, plan_kernel, seedmax_kernel, zscale_kernel in deepphysinet_b200/csrc/dpn_tc.cu) sees very different operands:

  R1  per unit j of layer 1, per (sample, net):  W1[j,:] d_j,  b1[j] d_j,  W2[:,j] / d_j
  R2  R1 with one d = 2^a for a whole (sample, net)
  R3  the c path of a net (all samples: it contains the static Wd):  W2, b2, e, Wd, bd, Wb, bb * 2^a,  Wa, wo * 2^-a
  R4  per unit j of layer 3, per net:  Wa[j,:] d_j,  ba[j] d_j,  Wb[:,j] / d_j

Each returns the new weights and the elementwise factor of every tensor.  Because the loss is unchanged, the gradient with respect
to a tensor scaled by f is the old gradient divided by f (transform_grads).  With power-of-two factors every scaled fp32 weight is
exact and every mask keeps its sign.

scale_plan restates the plan in fp32 so that a test can say which scale or product boundary it targets.  Its L1 norms and
P = diag(u) Wa W2 are summed in fp64 and rounded once, where the kernels sum in fp32: a bound that lies within an ulp of a power
of two can land one binade apart, nowhere else.
"""
import torch

S_PE, F16_TOP = 1024.0, 32768.0
CLAMP_LO, CLAMP_HI = 2.0 ** -80, 2.0 ** 80
FP32_LO, FP32_HI = 2.0 ** -126, 2.0 ** 127          # powers of two: normal fp32 range


# ---------------------------------------------------------------------------------------------------------------------------------
# reparametrisations
# ---------------------------------------------------------------------------------------------------------------------------------
def _ones(W):
    return {n: torch.ones(w.shape, dtype=torch.float64) for n, w in zip(W._fields, W)}


def apply(W, factors):
    """W with every tensor multiplied by its factor (exact for powers of two in the fp32 range)."""
    return type(W)(*[(w.double() * factors[n].to(w.device)).to(w.dtype) for n, w in zip(W._fields, W)])


def compose(*fs):
    out = {n: f.clone() for n, f in fs[0].items()}
    for f in fs[1:]:
        for n in out:
            out[n] *= f[n]
    return out


def r1(W, d, b, k):
    """R1 on (sample b, net k): d [256] factors of the units of layer 1."""
    f = _ones(W)
    d = torch.as_tensor(d, dtype=torch.float64)
    f["W1"][b, k] *= d[:, None]
    f["b1"][b, k] *= d
    f["W2"][b, k] /= d[None, :]
    return apply(W, f), f


def r2(W, a, b, k):
    """R2: R1 with d_j = 2^a for every unit of (sample b, net k)."""
    return r1(W, torch.full((256,), 2.0 ** a, dtype=torch.float64), b, k)


def r3(W, a, k):
    """R3 on net k (every sample): c scales by 2^a; a3, u, o and the Jacobian do not change."""
    f = _ones(W)
    for n in ("W2", "b2", "e"):
        f[n][:, k] *= 2.0 ** a
    for n in ("Wd", "bd", "Wb", "bb"):
        f[n][k] *= 2.0 ** a
    for n in ("Wa", "wo"):
        f[n][k] *= 2.0 ** -a
    return apply(W, f), f


def r4(W, d, k):
    """R4 on net k: d [256] factors of the units of layer 3."""
    f = _ones(W)
    d = torch.as_tensor(d, dtype=torch.float64)
    f["Wa"][k] *= d[:, None]
    f["ba"][k] *= d
    f["Wb"][k] /= d[None, :]
    return apply(W, f), f


def unit_spread(s, seed):
    """256 factors 2^e with integer e uniform in [-s, s] (the first unit at -s and the second at +s, so the spread is exactly 2s)."""
    e = torch.randint(-s, s + 1, (256,), generator=torch.Generator().manual_seed(seed)).double()
    e[0], e[1] = -s, s
    return torch.exp2(e)


def transform_grads(grads, factors):
    """Gradients of the reparametrised weights: the loss is unchanged, so d/d(w f) = (d/dw) / f."""
    return [g.double().cpu() / factors[n] for n, g in zip(factors, grads)]


# ---------------------------------------------------------------------------------------------------------------------------------
# scale plan (dpn_tc.cu: scale_for, bounds_kernel, plan_kernel, seedmax_kernel, zscale_kernel)
# ---------------------------------------------------------------------------------------------------------------------------------
def pow2_floor(x):
    """Largest power of two <= x, clamped to [2^-80, 2^80]; 2^-80 for x <= 2^-80, zero or NaN."""
    x = torch.as_tensor(x, dtype=torch.float64)
    _, e = torch.frexp(torch.nan_to_num(x, nan=0.0).clamp_min(CLAMP_LO))
    p = torch.ldexp(torch.ones_like(x), e - 1)
    return torch.where(x > CLAMP_LO, p.clamp(max=CLAMP_HI), torch.full_like(x, CLAMP_LO))


def scale_for(bound):
    """pow2_floor(F16_TOP / max(bound, 1e-30)) with the division in fp32."""
    b = torch.as_tensor(bound, dtype=torch.float64).float().clamp_min(1e-30)
    return pow2_floor((torch.tensor(F16_TOP, dtype=torch.float32) / b).double())


def _f32(x):
    return x.float().double()


def scale_plan(W, seeds=None, chunk=None):
    """Per-(sample, net) scales [B, K] of one call, as the f16x3 kernels choose them (keys as NetScales in dpn_tc.cu).

    seeds: optional (dov [B,N,K], dod [B,N,K,3] or None), the seeds dL/do and dL/do_c of the call; then 'chunks' holds the Z-side
    scales (sZP, sZH, sZD, sDV) of every chunk of `chunk` points (default: one chunk), which zscale_kernel derives from the seed
    maxima of that chunk.  Also returns the bounds the scales come from and T2 [K], the coupled G2 scale of plan_kernel."""
    g = {n: w.detach().double().cpu() for n, w in zip(W._fields, W)}
    B, K = g["W1"].shape[:2]
    bsum = _f32(_f32(g["b2"] + g["bd"]) + g["e"])                        # prep_kernel, in fp32
    uvec = _f32(torch.einsum("kij,ki->kj", g["Wb"], g["wo"]))
    wo2 = 2 * g["wo"]
    P = _f32(uvec[None, :, :, None] * (g["Wa"][None] @ g["W2"]))         # P = diag(u) Wa W2 of fold_gemm_kernel, rounded to fp32
    rowL1 = lambda w: _f32(w.abs().sum(-1))
    l1W1 = rowL1(g["W1"]).amax(-1)
    M1 = _f32(rowL1(g["W1"]) + g["b1"].abs()).amax(-1)
    l1W2, l1Wd = rowL1(g["W2"]).amax(-1), rowL1(g["Wd"]).amax(-1)
    cW2, cWa = _f32(g["W2"].abs().sum(-2)).amax(-1), _f32(g["Wa"].abs().sum(-2)).amax(-1)
    mW1, mW2 = g["W1"].abs().amax((-1, -2)), g["W2"].abs().amax((-1, -2))
    mWd, mWa = g["Wd"].abs().amax((-1, -2)), g["Wa"].abs().amax((-1, -2))
    mBs = bsum.abs().amax(-1)
    Mu, mWo2 = uvec.abs().amax(-1), wo2.abs().amax(-1)
    mP = P.abs().amax((-1, -2))
    Mc = _f32(_f32(l1W2 * M1) + l1Wd + mBs)
    My = _f32(Mu * cWa + mWo2)
    Mq = _f32(My * cW2)
    bk = lambda v: v.expand(B, K) if v.dim() == 1 else v
    t = dict(sW1=scale_for(mW1 * 32), sWa=bk(scale_for(mWa * 32)), sP=scale_for(mP * 32), sWd=bk(scale_for(mWd * 32)),
             sW2=scale_for(mW2), sH1=scale_for(M1), sC=scale_for(Mc), sQ=scale_for(Mq))
    t.update(M1=M1, Mc=Mc, l1W1=l1W1, My=My, Mq=Mq, mP=mP)
    t["cap"] = t["sH1"] * t["sW2"]
    T2 = torch.minimum(S_PE * t["sWd"][0], t["cap"].amin(0))             # plan_kernel: one coupled scale per net
    t["T2"] = T2
    t["sWd"] = (T2 / S_PE).expand(B, K).clone()
    t["sW2"] = T2 / t["sH1"]
    if seeds is not None:
        dov, dod = (s.detach().double().cpu() if s is not None else None for s in seeds)
        N = dov.shape[1]
        chunk = chunk or N
        t["chunks"] = []
        for p0 in range(0, N, chunk):
            DV = _f32(dov[:, p0:p0 + chunk].abs().amax(1))
            RR = 16 * _f32(dod[:, p0:p0 + chunk].abs().amax((1, 3))) if dod is not None else torch.zeros_like(DV)
            t["chunks"].append(dict(DV=DV, RR=RR, sZP=scale_for(DV + RR), sZH=scale_for(_f32(DV * M1) + _f32(RR * l1W1)),
                                    sZD=scale_for(DV), sDV=scale_for(DV)))
    return t


# the scale products the pass-1 epilogues form in one step (k1, k2, i3, i6; i4 = 1 / sP is a single scale)
PASS1_PRODUCTS = dict(k1=("S_PE", "sW1"), k2=("sH1", "sW2"), i3=("sC", "sWa"), i6=("sQ", "sW1"))


def boundaries(t):
    """Names of the plan entries at a boundary: (name, where) for every scale at its 2^-80 / 2^80 clamp and every pass-1
    product of PASS1_PRODUCTS outside the normal fp32 range [2^-126, 2^127].  Empty: every scale is a free power of two, so a
    uniform power-of-two reparametrisation shifts them exactly."""
    out = []
    for n in ("sW1", "sW2", "sWd", "sWa", "sP", "sH1", "sC", "sQ"):
        hit = (t[n] <= CLAMP_LO) | (t[n] >= CLAMP_HI)
        out += [(n, tuple(i)) for i in torch.nonzero(hit).tolist()]
    for n, (a, b) in PASS1_PRODUCTS.items():
        p = (S_PE if a == "S_PE" else t[a]) * t[b]
        bad = (p < FP32_LO) | (p > FP32_HI)
        out += [(n, tuple(i)) for i in torch.nonzero(bad).tolist()]
    return out


def log2(x):
    return torch.log2(torch.as_tensor(x, dtype=torch.float64))


def first_boundary(W, move, exps):
    """The first exponent a of `exps` (in order) at which scale_plan(move(W, a)) reaches a boundary, or None."""
    for a in exps:
        if boundaries(scale_plan(move(W, a))):
            return a
    return None


def f16_split(a, s):
    """An operand as the f16x3 kernels store it under the tile scale s (a power of two, broadcast against a): v = a s,
    hi = fp16(v), lo = fp16(v - hi), returned unscaled in fp64.  fp16 overflow gives inf, fp16 subnormals lose bits."""
    v = a.double() * s
    hi = v.to(torch.float16).double()
    return (hi + (v - hi).to(torch.float16).double()) / s


# binades below 2^15 (a tile's scaled bound) at which the lo plane leaves the fp16 normal range: lo ~ v 2^-11 and the smallest
# normal fp16 is 2^-14, so a value keeps its 22 bits while v >= 2^-3
LO_PLANE_BINADES = 15 - (-14 + 11)
