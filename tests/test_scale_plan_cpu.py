"""CPU: the power-of-two reparametrisations and the restated f16x3 scale plan of oracle/rescale.py, without a GPU.

  * R1..R4 keep values, Jacobian and loss terms of closed_form.pde_fwd_bwd to 1e-14 in fp64, and the fp64 gradients follow
    transform_grads; a threshold-free draw keeps its margin under each of them;
  * scale_plan reproduces hand-computed scales, the cross-sample minimum of plan_kernel, the 2^-80 / 2^80 clamps and the Z-side
    scales of zscale_kernel, and a uniform R2 / R3 shifts exactly the scales it should;
  * mutants of the plan, emulated on the z tile of dW1 with fp16 hi + lo operands: a chunk scaled with the first chunk's seed
    maximum, and a seed scale one binade too high, each break the strict f16x3 bound of tests/test_gpu_strict_parity.py on seeds
    laid out like the chunk case of tests/test_gpu_scale_plan.py (cold chunks, then a hot one), while the correct plan passes it.
"""
import pytest
import torch

from oracle import closed_form as CF
from oracle import rescale as R
from oracle import tiefree as TF
from tests import test_gpu_strict_parity as S


@pytest.fixture(scope="module")
def draw():
    W, pts, _ = TF.tie_free_draw(2, 96, 21, S.GUARD)
    return W, pts


def _closed(W, pts):
    out = []
    for b in range(pts["x"].shape[0]):
        c = {k: v[b].double().reshape(-1, 1) for k, v in pts.items() if k != "coord_data"}
        L, G, v, j = CF.pde_fwd_bwd(c["x"], c["y"], c["t"], c["f"], pts["coord_data"][b].double(), TF.sample_weights(W, b))
        out.append((L, G, v, j))
    return out


def _rel(a, b):
    return ((a - b).abs().max() / b.abs().max().clamp_min(1e-300)).item()


def _r1_r3_r4(W):
    W, f1 = R.r1(W, R.unit_spread(8, 3), 0, 0)
    W, f3 = R.r3(W, -12, 0)
    W, f4 = R.r4(W, R.unit_spread(8, 4), 0)
    return W, R.compose(f1, f3, f4)


MOVES = {
    "R1": lambda W: R.r1(W, R.unit_spread(20, 1), 1, 3),
    "R2": lambda W: R.r2(W, -37, 0, 5),
    "R3": lambda W: R.r3(W, 29, 2),
    "R4": lambda W: R.r4(W, R.unit_spread(20, 2), 4),
    "R1+R3+R4": _r1_r3_r4,
}


@pytest.mark.parametrize("move", list(MOVES))
def test_reparametrisation_preserves_the_function(draw, move):
    W, pts = draw
    W2, f = MOVES[move](W)
    assert not torch.equal(W2.W1, W.W1) or not torch.equal(W2.Wa, W.Wa)
    for b, ((L0, G0, v0, j0), (L1, G1, v1, j1)) in enumerate(zip(_closed(W, pts), _closed(W2, pts))):
        assert _rel(L1, L0) < 1e-14 and _rel(v1, v0) < 1e-14 and _rel(j1, j0) < 1e-14, (move, b)
        for n in S.NAMES:
            want = G0[n] / (f[n][b] if n in TF.GENERATED else f[n])
            assert _rel(G1[n], want) < 1e-12, (move, b, n)


@pytest.mark.parametrize("move", list(MOVES))
def test_tie_free_margin_survives(draw, move):
    """Every threshold distance is measured per unit over that unit's own spread, so the margin of each point is unchanged."""
    W, pts = draw
    W2, _ = MOVES[move](W)

    def margins(W):
        out = []
        for b in range(2):
            c = {k: v[b].double() for k, v in pts.items()}
            qs = TF._quantities(TF.sample_weights(W, b), c["x"], c["y"], c["t"], c["f"], c["coord_data"], S._consts(), True)
            out.append(torch.stack([(d / TF._spread(n, s)).reshape(d.shape[0], -1).amin(1) for n, (d, s) in qs.items()], 1).amin(1))
        return torch.stack(out)
    m0, m1 = margins(W), margins(W2)
    assert _rel(m1, m0) < 1e-9


# ---------------------------------------------------------------------------------------------------------------------------------
# scale_plan
# ---------------------------------------------------------------------------------------------------------------------------------
def _const_weights(B=2, K=2):
    from deepphysinet_b200.functional import DecoderWeights
    z = torch.zeros
    W = DecoderWeights(W1=torch.full((B, K, 256, 192), 2.0 ** -3), b1=z(B, K, 256), W2=torch.full((B, K, 256, 256), 2.0 ** -8),
                       b2=z(B, K, 256), e=z(B, K, 256), Wd=torch.full((K, 256, 192), 2.0 ** -4), bd=z(K, 256),
                       Wa=torch.full((K, 256, 256), 2.0 ** -6), ba=z(K, 256), Wb=z(K, 256, 256), bb=z(K, 256), wo=z(K, 256), bo=z(K))
    return W


def test_kernel_scale_plan_by_hand():
    """mW1 = 2^-3 -> sW1 = pow2_floor(2^15 / 2^2) = 2^13;  M1 = 192 / 8 = 24 -> sH1 = 2^10;  mW2 = 2^-8 -> cap = 2^10 2^23 = 2^33;
    mWd = 2^-4 -> S_PE sWd = 2^10 2^14 = 2^24 = T2 -> sWd = 2^14, sW2 = 2^14;  Mc = L1(W2) M1 + L1(Wd) = 24 + 12 -> sC = 2^9;
    u = 0 and wo = 0 -> P = diag(u) Wa W2 = 0, and sQ, sP at the 2^80 clamp."""
    t = R.scale_plan(_const_weights())
    want = dict(sW1=13, sH1=10, sWd=14, sW2=14, sC=9, sWa=15 - (-6 + 5), sQ=80, sP=80)
    for n, e in want.items():
        assert torch.equal(t[n], torch.full_like(t[n], 2.0 ** e)), (n, R.log2(t[n]))
    assert torch.equal(t["T2"], torch.full((2,), 2.0 ** 24))
    assert {n for n, _ in R.boundaries(t)} == {"sQ", "sP"}


def test_cross_sample_minimum():
    """Sample 1 of net 0 with W2 = 4: cap = 2^10 2^13 = 2^23 < S_PE sWd = 2^24, so T2 = 2^23 moves the Wd image of net 0 and the W2
    image of sample 0 by one binade; net 1 keeps T2 = 2^24."""
    W = _const_weights()
    W2 = W.W2.clone()
    W2[1, 0] = 4.0
    t = R.scale_plan(W._replace(W2=W2))
    assert t["T2"].tolist() == [2.0 ** 23, 2.0 ** 24]
    assert t["sWd"][:, 0].tolist() == [2.0 ** 13] * 2 and t["sWd"][:, 1].tolist() == [2.0 ** 14] * 2
    assert t["sW2"][0].tolist() == [2.0 ** 13, 2.0 ** 14] and t["sW2"][1, 0].item() == 2.0 ** 13
    assert torch.equal(t["sH1"] * t["sW2"], R.S_PE * t["sWd"])                   # G2's coupled accumulator


def test_clamps_and_z_scales():
    W = _const_weights()
    W1 = W.W1.clone()
    W1[0, 0] = 0.0
    W1[0, 1] = 2.0 ** 100
    t = R.scale_plan(W._replace(W1=W1))
    assert t["sW1"][0].tolist() == [2.0 ** 80, 2.0 ** -80]
    assert R.pow2_floor(torch.tensor([0.0, float("nan"), -1.0, 3.0, 2.0 ** 90])).tolist() == [2.0 ** -80] * 3 + [2.0, 2.0 ** 80]
    # Z side: DV = 3, RR = 16 * 0.5 = 8 -> sZP = pow2_floor(2^15 / 11) = 2^11;  sZH: 3 M1 + 8 L1(W1) = 264 -> 2^6;  per chunk
    dov = torch.zeros(2, 300, 2)
    dod = torch.zeros(2, 300, 2, 3)
    dov[:, 5], dod[:, 7, :, 1] = 3.0, -0.5
    dov[:, 290] = 2.0 ** -30
    t = R.scale_plan(W, seeds=(dov, dod), chunk=256)
    c0, c1 = t["chunks"]
    assert torch.equal(c0["sZP"], torch.full((2, 2), 2.0 ** 11)) and torch.equal(c0["sZH"], torch.full((2, 2), 2.0 ** 6))
    assert torch.equal(c1["sDV"], torch.full((2, 2), 2.0 ** 45)) and torch.equal(c1["sZP"], torch.full((2, 2), 2.0 ** 45))


def test_uniform_moves_shift_the_kernel_scales_exactly(draw):
    W, _ = draw
    t0 = R.scale_plan(W)
    # P = diag(u) Wa W2: R2 divides W2 of (1, 2) by 2^16, so sP rises by 16; R3 keeps u = Wb^T wo and multiplies Wa by 2^16 and
    # W2 by 2^-16, so P and sP do not move
    t = R.scale_plan(R.r2(W, 16, 1, 2)[0])
    for n, e in dict(sW1=-16, sH1=-16, sW2=16, sQ=16, sP=16, sWd=0, sC=0, sWa=0).items():
        want = t0[n].clone()
        want[1, 2] *= 2.0 ** e
        assert torch.equal(t[n], want), n
    t = R.scale_plan(R.r3(W, -16, 4)[0])
    for n, e in dict(sC=16, sWa=-16, sWd=16, sW2=16, sH1=0, sW1=0, sQ=0, sP=0).items():
        want = t0[n].clone()
        want[:, 4] *= 2.0 ** e
        assert torch.equal(t[n], want), n


def test_predicted_boundaries_of_the_uniform_sweeps(draw):
    """The sweeps of tests/test_gpu_scale_plan.py stay inside the plan up to +-40 and name their first boundary; no pass-1
    product (k1, k2, i3, i6) leaves the fp32 range before one of its factors is clamped."""
    W, _ = draw
    up = range(1, 100)
    b = {(m, s): R.first_boundary(W, (lambda W, a, m=m, s=s: (R.r2(W, s * a, 0, 0) if m == "R2" else R.r3(W, s * a, 0))[0]), up)
         for m in ("R2", "R3") for s in (1, -1)}
    print("first boundary exponents:", b)
    assert all(v is not None and v > 40 for v in b.values()), b
    for (m, s), a in b.items():
        names = {n for n, _ in R.boundaries(R.scale_plan((R.r2(W, s * a, 0, 0) if m == "R2" else R.r3(W, s * a, 0))[0]))}
        assert not names & set(R.PASS1_PRODUCTS), (m, s, names)


# ---------------------------------------------------------------------------------------------------------------------------------
# mutants of the plan on the z tile of dW1 (dW1 = qm^T zp, zp = dv PE for the decoder path)
# ---------------------------------------------------------------------------------------------------------------------------------
def hot_cold_chunks(pts, spread=30, chunk=256, seed=3):
    """Seeds [B,N,K] of the chunk case: every point 0.5..1, the chunks before the last one 2^-spread of that, and one hot seed of
    exactly 1 on a point with t = 0 in the last chunk (its cos features are exactly 1: zp = DV reaches the scaled bound 2^15)."""
    B, N = pts["x"].shape
    g = 0.5 + 0.5 * torch.rand(B, N, 6, generator=torch.Generator().manual_seed(seed))
    last = (N - 1) // chunk * chunk
    g[:, :last] *= 2.0 ** -spread
    for b in range(B):
        hot = last + int(torch.nonzero(pts["t"][b, last:].cpu() == 0)[0])
        g[b, hot] = 1.0
    return g


def _dW1(W, pts, g_o, sZP_of_chunk, chunk):
    """fp64 dW1 [B,K,256,192] with zp rounded to fp16 hi + lo under the given per-chunk scale [B,K] (None: exact)."""
    B, N = pts["x"].shape
    out = torch.zeros(W.W1.shape, dtype=torch.float64)
    for b in range(B):
        c = {k: v[b].double().cpu().reshape(-1, 1) for k, v in pts.items() if k != "coord_data"}
        st = CF.pde_fwd_bwd(c["x"], c["y"], c["t"], c["f"], pts["coord_data"][b].double().cpu(), TF.sample_weights(W, b),
                            return_stages=True)[4]
        for k in range(6):
            for i, p0 in enumerate(range(0, N, chunk)):
                sl = slice(p0, p0 + chunk)
                zp = g_o[b, sl, k:k + 1].double() * st["pe"][sl]
                if sZP_of_chunk is not None:
                    zp = R.f16_split(zp, sZP_of_chunk(i)[b, k])
                out[b, k] += st["nets"][k]["qm"][sl].T @ zp
    return out


@pytest.fixture(scope="module")
def chunk_draw():
    W, pts, _ = TF.tie_free_draw(1, 512, 601, S.GUARD, pde=False)
    return W, pts


@pytest.mark.parametrize("mutant", [None, "first_chunk_only", "one_binade_high"])
def test_plan_mutants_break_the_strict_bound(chunk_draw, mutant):
    W, pts = chunk_draw
    chunk = 256
    g_o = hot_cold_chunks(pts, chunk=chunk)
    plan = R.scale_plan(W, seeds=(g_o, None), chunk=chunk)["chunks"]
    sZP = {None: lambda i: plan[i]["sZP"], "first_chunk_only": lambda i: plan[0]["sZP"],
           "one_binade_high": lambda i: 2 * plan[i]["sZP"]}[mutant]
    exact = _dW1(W, pts, g_o, None, chunk)
    got = _dW1(W, pts, g_o, sZP, chunk)
    zeros = [torch.zeros(w.shape, dtype=torch.float64) for w in W]
    ref = dict(grads=[exact if n == "W1" else z for n, z in zip(S.NAMES, zeros)])
    E = S.strict_errors(dict(grads=[got if n == "W1" else z for n, z in zip(S.NAMES, zeros)]), ref)
    print(mutant, "dW1 worst slice %.1e %s" % E["grad"])
    rejected = bool(S.violations(E, "f16x3"))
    assert rejected == (mutant is not None), (mutant, E["grad"])
