"""GPU (-m gpu): the f16x3 scale plan across the exponent range, with the comparator, bounds and oracles of
tests/test_gpu_strict_parity.py.

The other strict tests draw every sample from random_decoder_weights, whose magnitudes sit in a narrow band.  Here the plan meets
  a. uniform power-of-two reparametrisations (oracle/rescale.py R2, R3), seeds * 2^k and loss factors * 2^k: every mode must absorb
     them exactly until scale_plan predicts a clamp; values and Jacobian bit-identical, loss terms to 1e-12, gradient slices equal
     to the transformed gradients to 1e-6.  Past the boundary fp32 keeps the strict bounds and no mode returns a non-finite value;
  b. per-unit spreads (R1, R4): fp32 values bit-identical; the split modes strict up to the spread fp16 supports;
  c. one sample of a batch 2^a larger in h1 W2 than the other, which lowers the G2 scale T2 that plan_kernel shares between samples;
  d. seed spreads within a (sample, net, chunk): a hot point over cold ones, hot and cold tiles, chunks 2^30 apart, nets 2^40 apart
     and a sample at 2^-60;
  e. the PDE path with rho clipped at some points of a sample, loss factors from 1e-7 to 1e14, and n_norm far from N.
Every figure is printed; DESIGN.md section 6 states the measured limits these tests assert.
"""
import dataclasses

import pytest
import torch

from oracle import rescale as R
from oracle import tiefree as TF
from tests import test_gpu_residual_branches as RB
from tests import test_gpu_strict_parity as S

pytestmark = pytest.mark.gpu

GRAD_EXACT = 1e-6                 # a transformed gradient slice: equal up to the order of the fp32 reductions
SPLIT = ("f16x3", "f16x3a")
# supported dynamic range of the fp16 split modes (DESIGN.md section 6), asserted below and beyond
UNIT_SPREAD = 8                   # per-unit factors 2^[-s, s]: strict up to s = 8 (16 binades between units)
SAMPLE_RATIO = 20                 # one sample's h1 W2 2^a above another's: strict up to a = 20
COLD_SEEDS = 20                   # rows reached only by seeds 2^-k below the hot seed of their chunk: 1e-4 up to k = 20


@pytest.fixture(scope="module")
def pde_draw():
    return S._draw(2, 700, 801)


@pytest.fixture(scope="module")
def base(pde_draw):
    """Unscaled library calls per mode, the oracle and its seed-sum magnitudes."""
    W, pts = pde_draw
    return {m: S.run_pde(W, pts, m) for m in S.ALL}, S.pde_oracle(W, pts), RB.seed_sum_scale(W, pts, S._consts())


def _cpu(x):
    return x.detach().double().cpu()


def _finite(got):
    return all(bool(torch.isfinite(got[k]).all()) for k in ("terms", "vals", "jac") if k in got) and \
        all(bool(torch.isfinite(g).all()) for g in got["grads"])


def _slice_err(got, want, grad_scale=None):
    """Worst relative error of the gradient slices (per (sample, net) or per net) against `want`."""
    ref = dict(grads=want) if grad_scale is None else dict(grads=want, grad_scale=grad_scale)
    return S.strict_errors(dict(grads=got), ref)["grad"]


def _exact_errors(got, base, factors, seed=1.0, term=1.0, grad_scale=None):
    """Violations of exact absorption: values / Jacobian bit-identical, terms to 1e-12, slices to GRAD_EXACT.  grad_scale: the
    seed-sum magnitudes of the unscaled PDE call (test_gpu_residual_branches.seed_sum_scale): bb and bo are sums of seeds of
    both signs, and their fp32 sums in another order differ by 1e-6 of a slice that cancels."""
    bad = []
    for k in ("vals", "jac"):
        if k in got and not torch.equal(got[k], base[k]):
            bad.append((k, (_cpu(got[k]) - _cpu(base[k])).abs().max().item()))
    if "terms" in got:
        e = ((_cpu(got["terms"]) - term * _cpu(base["terms"])).abs() / (term * _cpu(base["terms"]).abs())).max().item()
        if not e <= 1e-12:
            bad.append(("terms", e))
    want = [g * seed for g in R.transform_grads(base["grads"], factors)]
    if grad_scale is not None:
        grad_scale = [g * seed for g in R.transform_grads(grad_scale, factors)]
    v, where = _slice_err(got["grads"], want, grad_scale)
    if not v <= GRAD_EXACT:
        bad.append(("grad", v, where))
    return bad


# ---------------------------------------------------------------------------------------------------------------------------------
# a. uniform power-of-two reparametrisations, seeds and loss factors
# ---------------------------------------------------------------------------------------------------------------------------------
def _move(name, a):
    return (lambda W: R.r2(W, a, 1, 2)) if name == "R2" else (lambda W: R.r3(W, a, 3))


UNIFORM = [(m, a) for m in ("R2", "R3") for a in (-40, -16, -4, 4, 16, 40)] + \
          [(m, e) for m in ("R2", "R3") for e in ("edge+", "edge-")]


@pytest.mark.parametrize("move,a", UNIFORM, ids=["%s_%s" % c for c in UNIFORM])
def test_uniform_reparametrisation(pde_draw, base, move, a):
    W, pts = pde_draw
    calls, ref, gs = base
    if isinstance(a, str):                       # the first exponent at which scale_plan reaches a clamp, and 12 beyond it
        sign = 1 if a == "edge+" else -1
        edge = R.first_boundary(W, lambda W, e: _move(move, sign * e)(W)[0], range(1, 100))
        a = sign * (edge + 12)
    W2, f = _move(move, a)(W)
    past = R.boundaries(R.scale_plan(W2))
    print("%s a=%d: plan boundaries %s" % (move, a, sorted({n for n, _ in past})))
    bad = []
    for mode in S.ALL:
        got = S.run_pde(W2, pts, mode)
        if not _finite(got):
            bad.append((mode, "non-finite"))
        elif not past:
            bad += [(mode,) + v for v in _exact_errors(got, calls[mode], f, grad_scale=gs)]
        elif mode == "fp32":
            bad += S.check(got, dict(ref, grads=R.transform_grads(ref["grads"], f)), mode, "%s a=%d past the plan" % (move, a))
        if past and mode != "fp32":
            print("%s a=%d %s past the plan: %s" % (move, a, mode, S.strict_errors(got, dict(ref, grads=R.transform_grads(ref["grads"], f)))))
    assert not bad, bad


@pytest.fixture(scope="module")
def dec_draw():
    return S._draw(2, 1024, 802, pde=False)


@pytest.mark.parametrize("k", [-60, -20, 20, 60])
def test_seed_scaling(dec_draw, k):
    """dpn_decoder_bwd with d_o 2^k: gradients exactly 2^k times the unscaled ones."""
    W, pts = dec_draw
    xyz = (pts["x"], pts["y"], pts["t"])
    g_o = S._seeds((2, 1024, 6), 21)
    bad = []
    for mode in S.ALL:
        a = S.run_decoder(W, pts["coord_data"], g_o, mode, xyz=xyz)
        b = S.run_decoder(W, pts["coord_data"], g_o * 2.0 ** k, mode, xyz=xyz)
        bad += [(mode,) + v for v in _exact_errors(b, a, R._ones(W), seed=2.0 ** k)]
    assert not bad, bad


@pytest.mark.parametrize("k", [-20, 20])
def test_loss_factor_scaling(pde_draw, base, k):
    W, pts = pde_draw
    calls, _, gs = base
    c = S._consts()
    c2 = dataclasses.replace(c, factor=tuple(v * 2.0 ** k for v in c.factor))
    bad = []
    for mode in S.ALL:
        got = RB.run_pde(W, pts, mode, c2)
        bad += [(mode,) + v for v in _exact_errors(got, calls[mode], R._ones(W), seed=2.0 ** k, term=2.0 ** k, grad_scale=gs)]
    assert not bad, bad


# ---------------------------------------------------------------------------------------------------------------------------------
# b. per-unit spreads
# ---------------------------------------------------------------------------------------------------------------------------------
def unit_move(kind, s, W):
    """R1 on every (sample, net) or R4 on every net, factors 2^[-s, s]."""
    fs = []
    for k in range(6):
        if kind == "R1":
            for b in range(W.W1.shape[0]):
                W, f = R.r1(W, R.unit_spread(s, 100 * k + b), b, k)
                fs.append(f)
        else:
            W, f = R.r4(W, R.unit_spread(s, 100 + k), k)
            fs.append(f)
    return W, R.compose(*fs)


@pytest.mark.parametrize("kind", ["R1", "R4"])
def test_unit_spread(pde_draw, base, kind):
    W, pts = pde_draw
    calls, ref, _ = base
    bad = []
    for s in (2, 4, 8, 12, 16, 24):
        W2, f = unit_move(kind, s, W)
        ref2 = dict(ref, grads=R.transform_grads(ref["grads"], f))
        for mode in S.STRICT:
            got = S.run_pde(W2, pts, mode)
            label = "%s spread 2^[-%d,%d]" % (kind, s, s)
            if mode == "fp32" and not torch.equal(got["vals"], calls["fp32"]["vals"]):
                bad.append((label, mode, "values not bit-identical"))
            if not _finite(got):
                bad.append((label, mode, "non-finite"))
            v = S.check(got, ref2, mode, label)
            if mode in SPLIT and s > UNIT_SPREAD:
                continue                         # beyond the supported spread: reported above, finite
            bad += v
    assert not bad, bad


# ---------------------------------------------------------------------------------------------------------------------------------
# c. batch independence under mixed magnitudes
# ---------------------------------------------------------------------------------------------------------------------------------
def test_batch_independence(pde_draw):
    """Sample 1's W2 * 2^a (all nets; not function-preserving, and sample 1 is not compared).  Sample 0 must not notice: fp32
    bit-identical values, Jacobian and terms to sample 0 alone, generated-weight slices to 1e-6; the split modes strict up to
    a = SAMPLE_RATIO.  plan_kernel lowers T2 (and with it sample 0's W2 and Wd images) once sample 1's capacity falls below
    S_PE sWd."""
    W, pts = pde_draw
    one = lambda t: t[:1].contiguous()
    W0 = type(W)(*[one(w) if n in TF.GENERATED else w for n, w in zip(W._fields, W)])
    p0 = {k: one(v) for k, v in pts.items()}
    ref = S.pde_oracle(W0, p0)
    alone = {m: S.run_pde(W0, p0, m) for m in S.STRICT}
    bad, first_fail = [], {}
    for a in (0, 4, 8, 12, 16, 20, 24, 32):
        W2 = W.W2.clone()
        W2[1] *= 2.0 ** a
        Wa = W._replace(W2=W2)
        t = R.scale_plan(Wa)
        print("a=%d: T2 2^%s, sample-0 W2 image max 2^%.1f" % (a, R.log2(t["T2"]).tolist(),
                                                             R.log2((W.W2[0].abs().amax((-1, -2)).double().cpu() * t["sW2"][0]).max()).item()))
        for mode in S.STRICT:
            got = S.run_pde(Wa, pts, mode)
            s0 = dict(terms=got["terms"][:1], vals=got["vals"][:1], jac=got["jac"][:1],
                      grads=[2 * g[:1] for n, g in zip(S.NAMES, got["grads"]) if n in TF.GENERATED])
            if not _finite(got):
                bad.append((a, mode, "non-finite"))
            if mode == "fp32":
                for k in ("vals", "jac"):
                    if not torch.equal(s0[k], alone[mode][k]):
                        bad.append((a, mode, k, "differs from the sample alone"))
                e = ((_cpu(s0["terms"]) - _cpu(alone[mode]["terms"])).abs() / _cpu(alone[mode]["terms"]).abs()).max().item()
                if not e <= 1e-12:                  # fp64 sums over blocks, in no fixed order
                    bad.append((a, mode, "terms", e))
                v, where = _slice_err(s0["grads"], [g[:1] for g in alone[mode]["grads"][:5]])
                if not v <= GRAD_EXACT:
                    bad.append((a, mode, "grad", v, where))
            v = S.check(s0, ref, mode, "sample 1 h1 W2 * 2^%d" % a)
            if v and mode not in first_fail:
                first_fail[mode] = a
            if mode not in SPLIT or a <= SAMPLE_RATIO:
                bad += v
    print("first failing exponent per mode:", first_fail)
    assert not bad, bad


# ---------------------------------------------------------------------------------------------------------------------------------
# d. seed spreads within a (sample, net, chunk)
# ---------------------------------------------------------------------------------------------------------------------------------
def _hot_point(pts, b, lo, hi):
    """A point of [lo, hi) of sample b with t = 0: its cos features are exactly 1, so a seed of exactly 1 there puts zp on the
    scaled bound 2^15 (the case a seed scale one binade too high overflows)."""
    return lo + int(torch.nonzero(pts["t"][b, lo:hi].cpu() == 0)[0])


def seed_cases(pts):
    B, N = pts["x"].shape
    g = 0.5 + torch.rand(B, N, 6, generator=torch.Generator().manual_seed(22))      # as S._seeds
    cases = []
    for k in (10, 20, 30):                                      # one hot point among points 2^-k smaller (all in one chunk)
        c = g * 2.0 ** -k
        for b in range(B):
            c[b, _hot_point(pts, b, 0, N)] = 1.0
        cases.append(("hot point, cold 2^-%d" % k, c, 0, k))
    c = g.clone()
    c[:, 128:256] *= 2.0 ** -20                                 # hot and cold tiles
    cases.append(("tile 1 at 2^-20", c, 0, None))
    c = g.clone()
    c[:, :768] *= 2.0 ** -30                                    # chunks 2^30 apart: three cold chunks, then a hot one
    for b in range(B):
        c[b, _hot_point(pts, b, 768, N)] = 1.0
    cases.append(("chunks 2^30 apart", c, 256, None))
    c = g * torch.exp2(-8.0 * torch.arange(6.0))                # nets 2^0 .. 2^-40
    cases.append(("nets 2^0..2^-40", c, 0, None))
    c = g.clone()
    c[1] *= 2.0 ** -60
    cases.append(("sample 1 at 2^-60", c, 0, None))
    return cases


def cold_rows(W, pts, g_o, hot_k):
    """Per (sample, net) the dW1 rows the hot point does not reach (m1 = 0 there): only the cold seeds feed them."""
    from oracle import closed_form as CF
    from oracle import dpn_oracle as O
    c = S._consts()
    out = []
    for b in range(pts["x"].shape[0]):
        hot = int(g_o[b, :, 0].argmax())
        col = lambda k: pts[k][b, hot:hot + 1].double().cpu().reshape(-1, 1)
        pe, _ = CF.coord_features(col("x"), col("y"), col("t"), c.dx, c.dy, c.lat_size, c.lon_size, c.pred_t_span)
        a1, _ = TF.preactivations(pe, O.sine_cos_pe(pts["coord_data"][b, hot:hot + 1].double().cpu(), 16), TF.sample_weights(W, b))
        out.append(a1[0] <= 0)                                   # [6, 256]
    return torch.stack(out)


@pytest.fixture(scope="module")
def seed_draw():
    return S._draw(2, 1024, 803, pde=False)


def test_seed_spreads(seed_draw):
    W, pts = seed_draw
    xyz = (pts["x"], pts["y"], pts["t"])
    bad = []
    for label, g_o, chunk, hot_k in seed_cases(pts):
        ref = S.decoder_oracle(W, pts["coord_data"], g_o, xyz=xyz)
        rows = cold_rows(W, pts, g_o, hot_k) if hot_k else None
        for mode in S.ALL:
            got = S.run_decoder(W, pts["coord_data"], g_o.cuda(), mode, xyz=xyz, chunk=chunk)
            if not _finite(got):
                bad.append((label, mode, "non-finite"))
            v = S.check(got, ref, mode, label)
            if mode == "bf16":
                continue                            # one bf16 plane: a slice led by one point reaches 0.21 (printed above)
            bad += v
            if rows is not None:
                g, r = _cpu(got["grads"][0]), ref["grads"][0]
                # dW1 rows fed by the cold points alone, each over the rms of those rows in its (sample, net) slice (a single row
                # can cancel)
                rn = r.norm(dim=-1)
                rms = (rn.pow(2) * rows).sum(-1, keepdim=True).div(rows.sum(-1, keepdim=True)).sqrt()
                e = ((g - r).norm(dim=-1) / rms)[rows]
                print("%-34s %-6s cold rows %d, worst row %.1e" % (label, mode, int(rows.sum()), e.max().item()))
                if hot_k <= COLD_SEEDS and not e.max() <= S.BOUNDS[mode]["grad"]:
                    bad.append((label, mode, "cold row", e.max().item()))
    assert not bad, bad


# ---------------------------------------------------------------------------------------------------------------------------------
# e. PDE path: rho clipped at some points of a sample, loss factors 1e-7 .. 1e14, n_norm far from N
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("chunk,n_norm", [(0, 0), (256, 0), (0, 4096 * 1000)])
def test_pde_mixed_magnitudes(chunk, n_norm):
    c = dataclasses.replace(S._consts(), factor=(3e-7, 2e4, 1e14, 5e-2, 2e9, 1e-7 * 7))
    W, pts = RB._draw(2, 1000, 804, [["free"], ["free"] * 7 + ["rho_lo"]], consts=c)
    ref = RB.pde_ref(W, pts, c, n_total=n_norm or None)
    bad = []
    for mode in S.ALL:
        got = RB.run_pde(W, pts, mode, c, chunk=chunk, n_norm=n_norm)
        bad += S.check(got, ref, mode, "rho_lo 1 in 8, chunk %d, n_norm %d" % (chunk, n_norm))
    assert not bad, bad
