"""GPU (-m gpu): strict parity of every arithmetic mode with fp64 on threshold-free draws (oracle/tiefree.py), per sample, per net
and per point, at tile, chunk and wgrad-split boundaries.

The statistical tests (tests/test_gpu_f16x3.py, tests/test_gpu_headline_parity.py, tests/test_gpu_bf16x3.py) cover draws that were
not screened for threshold ties: a ReLU mask bit, clip bound or vapour switch within rounding distance of its threshold flips and
moves one net's Jacobian and J-side gradients by 1e-4..1.4e-3, so they accept 3e-3 (1e-2 for bf16x3) per draw on whole-tensor norms
and require only most draws to stay under 1e-4.  That lets a dropped point, a wrongly scaled tile or split, a bug at one size or a
wrong lo plane through.  Here every threshold decision of every point clears a guard of 1e-4 of its spread (5e-4 for bf16x3; the
draws use 5e-4 for all modes), 30x or more above f16x3's error, so the kernels take the masks exact arithmetic takes and each of the
following is bounded separately:

    mode            loss term   gradient slice   Jacobian (sample, net, coordinate)   value per point / rms
    fp32            1e-5        2e-5             2e-5                                 1e-6
    f16x3, f16x3a   5e-5        1e-4             1e-4                                 1e-5
    bf16x3          2e-3        3e-3             3e-3                                 1e-4
    bf16            0.2 everywhere: one bf16 plane cannot be made threshold-free; a structural bug still shows as an O(1) error

Loss terms per sample, values per point over the rms of that sample's field, the Jacobian as a norm per (sample, net, coordinate)
and per point against its rms (10x the slice bound), each generated-weight gradient per (sample, net) slice and each static-weight
gradient per net slice.  A slice whose reference is exactly zero (a net or sample without seeds) must be exactly zero.
The PDE oracle is oracle/closed_form.py per sample (assembled like testing.oracle_reference: total = mean over samples, generated
gradients G_b / B, static ones sum_b G_b / B); the decoder oracle is autograd through dpn_oracle.decoder_net in fp64.
"""
import contextlib
import math

import pytest
import torch

from oracle import closed_form as CF
from oracle import dpn_oracle as O
from oracle import tiefree as TF

pytestmark = pytest.mark.gpu

NAMES = ("W1", "b1", "W2", "b2", "e", "Wd", "bd", "Wa", "ba", "Wb", "bb", "wo", "bo")
STRICT = ("fp32", "f16x3", "f16x3a", "bf16x3")
ALL = STRICT + ("bf16",)
BOUNDS = {"fp32": dict(terms=1e-5, grad=2e-5, jac=2e-5, vals=1e-6),
          "f16x3": dict(terms=5e-5, grad=1e-4, jac=1e-4, vals=1e-5),
          "f16x3a": dict(terms=5e-5, grad=1e-4, jac=1e-4, vals=1e-5),
          "bf16x3": dict(terms=2e-3, grad=3e-3, jac=3e-3, vals=1e-4),
          "bf16": dict(terms=0.2, grad=0.2, jac=0.2, vals=0.2)}
GUARD = max(TF.GUARD.values())            # one draw serves every mode

# ---- the weight-gradient split rule of run_planes (deepphysinet_b200/csrc/dpn_tc.cu), copied so that the shapes below can say
# ---- which T and split count they hit
TP, CLUSTER, SLOTS, WGRAD_TILES, ITEMS = 128, 2, 148, 32, 3


def wgrad_plan(B, P, K=6):
    """(T, splits) of one chunk of P points: T tiles per sample (rounded up to whole clusters) and the wgrad2_kernel point-splits."""
    T = (-(-P // TP) + CLUSTER - 1) // CLUSTER * CLUSTER
    items = B * K * 2 * ITEMS
    splits, best = 1, 0.0
    for sp in range(1, min(8, T) + 1):
        waves = items * sp / SLOTS
        eff = waves / math.ceil(waves)
        if eff > best + 0.02:
            best, splits = eff, sp
    if -(-T // splits) > WGRAD_TILES:
        splits = -(-T // WGRAD_TILES)
    return T, splits


def split_ranges(T, splits):
    return [(T * s // splits, T * (s + 1) // splits) for s in range(splits)]


# (B, N, seed, (T, splits) the shape is meant to hit)
SWEEP = [
    (1, 1, 101, (2, 2)),          # one point; split 1 holds only the cluster's padding tile
    (1, 127, 102, (2, 2)),        # one short tile + padding
    (1, 128, 103, (2, 2)),        # exactly one tile
    (1, 129, 104, (2, 2)),        # last tile holds 1 point
    (1, 255, 105, (2, 2)),
    (1, 257, 106, (4, 4)),        # 3 tiles padded to 4; the 4th split is the padding tile alone
    (1, 383, 107, (4, 4)),        # odd tile count: splits [0,1) [1,2) [2,3) [3,4), the last one padding only
    (1, 640, 108, (6, 4)),        # 5 tiles padded to 6: uneven splits [0,1) [1,3) [3,4) [4,6)
    (3, 1000, 109, (8, 4)),       # sample 1's tiles follow sample 0's; splits [0,2) [2,4) [4,6) [6,8)
    (1, 4225, 110, (34, 4)),      # 4 splits of 8 or 9 tiles; last tile 1 point
    (2, 8321, 111, (66, 3)),      # wave rule gives 2 splits of 33 tiles, the 32-tile flush raises it to 3; last tile 1 point
    (1, 16513, 112, (130, 5)),    # 5 flush splits of 26 tiles; last tile 1 point
]


# ---------------------------------------------------------------------------------------------------------------------------------
# comparator
# ---------------------------------------------------------------------------------------------------------------------------------
def _f(x):
    x = float(x)
    return math.inf if math.isnan(x) else x


def strict_errors(got, ref):
    """group -> (worst figure, where) for every group both dicts carry: terms [B,T], vals [B,N,F], jac [B,N,6,3], grads (13)."""
    E = {}

    def put(group, val, where):
        val = _f(val)
        if group not in E or val > E[group][0]:
            E[group] = (val, where)

    cpu = lambda a: a.detach().double().cpu()
    if "terms" in got and "terms" in ref:
        g, r = cpu(got["terms"]), cpu(ref["terms"])
        e = torch.where(r == 0, torch.where(g == 0, 0.0, math.inf).double(), (g - r).abs() / r.abs())
        i = int(torch.nan_to_num(e, nan=math.inf).argmax())
        put("terms", e.flatten()[i], ("sample, term", divmod(i, r.shape[1])))
    if "vals" in got and "vals" in ref:
        g, r = cpu(got["vals"]), cpu(ref["vals"])
        e = (g - r).abs() / r.pow(2).mean(1, keepdim=True).sqrt().clamp_min(1e-300)
        i = int(torch.nan_to_num(e, nan=math.inf).argmax())
        put("vals", e.flatten()[i], ("sample, point, field", tuple(int(v) for v in torch.unravel_index(torch.tensor(i), e.shape))))
    if "jac" in got and "jac" in ref:
        g, r = cpu(got["jac"]), cpu(ref["jac"])
        d = g - r
        # an entry is a 192-term dot product Jin . dPE; where it cancels, the fp32 encoding of the coordinate alone (6e-8) moves it
        # in every mode (a one-point draw: condition 3.5e3, 2.6e-4 in fp32 mode), so no entry counts as smaller than 1/128 of the
        # magnitude of its terms (jac_scale).  On slices of many points the floor never binds.
        fl = cpu(ref["jac_scale"]) / 128 if "jac_scale" in ref else torch.zeros_like(r)
        e = d.norm(dim=1) / torch.maximum(r.norm(dim=1), fl.norm(dim=1)).clamp_min(1e-300)   # [B,6,3]
        i = int(torch.nan_to_num(e, nan=math.inf).argmax())
        put("jac", e.flatten()[i], ("sample, net, coordinate", tuple(int(v) for v in torch.unravel_index(torch.tensor(i), e.shape))))
        ep = d.abs() / torch.maximum(r.pow(2).mean(1, keepdim=True).sqrt(), fl).clamp_min(1e-300)   # [B,N,6,3]
        i = int(torch.nan_to_num(ep, nan=math.inf).argmax())
        put("jac_pt", ep.flatten()[i], ("sample, point, net, coordinate",
                                        tuple(int(v) for v in torch.unravel_index(torch.tensor(i), ep.shape))))
    if "grads" in got and "grads" in ref:
        for n, g, r in zip(NAMES, got["grads"], ref["grads"]):
            g, r = cpu(g), cpu(r)
            lead = 2 if n in TF.GENERATED else 1
            gs, rs = g.reshape(*r.shape[:lead], -1), r.reshape(*r.shape[:lead], -1)
            for idx in torch.cartesian_prod(*[torch.arange(s) for s in r.shape[:lead]]).reshape(-1, lead).tolist():
                gi, ri = gs[tuple(idx)], rs[tuple(idx)]
                if not torch.isfinite(gi).all():
                    val = math.inf
                elif ri.norm() == 0:
                    val = 0.0 if gi.norm() == 0 else math.inf                   # unseeded slices: exactly zero
                else:
                    den = ri.norm()
                    if "grad_scale" in ref:       # a sum of seeds that cancels has no relative accuracy (see seed_sum_scale)
                        den = torch.maximum(den, cpu(ref["grad_scale"][NAMES.index(n)]).reshape(*r.shape[:lead], -1)[tuple(idx)].norm() / 8)
                    val = ((gi - ri).norm() / den).item()
                put("grad", val, (n,) + tuple(idx))
    return E


def violations(E, mode):
    b = dict(BOUNDS[mode], jac_pt=10 * BOUNDS[mode]["jac"])
    return [(grp, v, where) for grp, (v, where) in E.items() if not v <= b[grp]]


def check(got, ref, mode, label):
    """Print the worst figure of every group; return the violated bounds (empty when the call passes)."""
    E = strict_errors(got, ref)
    print("%-34s %-6s " % (label, mode) + "  ".join("%s %.1e %s" % (g, v, w) for g, (v, w) in E.items() if g != "grad")
          + ("  grad %.1e %s" % E["grad"] if "grad" in E else ""))
    return [(label, mode) + v for v in violations(E, mode)]


# ---------------------------------------------------------------------------------------------------------------------------------
# oracles and library calls
# ---------------------------------------------------------------------------------------------------------------------------------
def _consts():
    from deepphysinet_b200.config import PhysicsConsts
    return PhysicsConsts()


def _jac_scale(st, consts):
    """sum_j |Jin_j dPE_j| per (point, net, coordinate), in the physical units of jac (closed_form.residual_and_seeds)."""
    N = st["pe"].shape[0]
    dt = st["pe"].dtype
    mag = torch.stack([(n["jin"] * st["dpe"]).abs().reshape(N, 64, 3).sum(1) for n in st["nets"]], 1)     # [N,6,3]
    std = torch.tensor(consts.std, dtype=dt)
    kap = torch.ones(N, 6, dtype=dt)
    if consts.with_clip:
        raw = st["o"] * std + torch.tensor(consts.mean, dtype=dt)
        kap[:, 2:] = ((raw[:, 2:] >= torch.tensor(consts.lo[2:], dtype=dt)) & (raw[:, 2:] <= torch.tensor(consts.hi[2:], dtype=dt))).to(dt)
    sc = torch.tensor((1.0 / (consts.dx * (consts.lon_size - 1)), 1.0 / (consts.dy * (consts.lat_size - 1)), 1.0 / consts.pred_t_span),
                      dtype=dt)
    return mag * (std * 1.0)[None, :, None] * kap[:, :, None] * sc


def pde_oracle(W, pts, consts=None, chunk=4096, drop=None, n_total=None):
    """Closed-form fp64 PDE call per sample: terms [B,6], vals [B,N,6], jac [B,N,6,3], grads (d mean_b loss_b / d W).
    drop=(b, index tensor): leave those points of sample b out of the gradients (the terms stay normalised by N);
    n_total: the point count the loss means divide by (the library's n_norm; default N)."""
    consts = consts or _consts()
    B, N = pts["x"].shape
    geo = dict(CF.kwargs_of(consts), n_total=n_total or N)
    grads = [torch.zeros(w.shape, dtype=torch.float64) for w in W]
    terms, vals, jacs, scales = [], [], [], []
    for b in range(B):
        Wb = TF.sample_weights(W, b)
        c = {k: v[b].detach().double().cpu() for k, v in pts.items()}
        keep = torch.ones(N, dtype=torch.bool)
        if drop is not None and drop[0] == b:
            keep[drop[1]] = False
        lt, vb, jb, sb = 0.0, [], [], []
        for lo in range(0, N, chunk):
            sl = slice(lo, min(N, lo + chunk))
            col = lambda k: c[k][sl].reshape(-1, 1)
            L, G, v, j, st = CF.pde_fwd_bwd(col("x"), col("y"), col("t"), col("f"), c["coord_data"][sl], Wb, return_stages=True, **geo)
            lt = lt + L
            vb.append(v)
            jb.append(j)
            sb.append(_jac_scale(st, consts))
            if not keep[sl].all():
                kk = keep[sl]
                _, G, _, _ = CF.pde_fwd_bwd(col("x")[kk], col("y")[kk], col("t")[kk], col("f")[kk], c["coord_data"][sl][kk], Wb, **geo)
            for i, n in enumerate(NAMES):
                if n in TF.GENERATED:
                    grads[i][b] += G[n] / B
                else:
                    grads[i] += G[n] / B
        terms.append(lt)
        vals.append(torch.cat(vb))
        jacs.append(torch.cat(jb))
        scales.append(torch.cat(sb))
    return dict(terms=torch.stack(terms), vals=torch.stack(vals), jac=torch.stack(jacs), jac_scale=torch.stack(scales), grads=grads)


def decoder_oracle(W, cd, g_o, pe=None, xyz=None, ref_in=None, consts=None, rows=None):
    """fp64 autograd through dpn_oracle.decoder_net: vals [B,N,K] (only the rows evaluated) and d sum(o * g_o) / dW.
    pe: [B,N,192] encoded coordinates, or xyz=(x, y, t) [B,N]; ref_in [B,N,K] (default: coord_data[..., k] for net k);
    rows: per sample None (skip) or (lo, hi) to evaluate only those points (the rest carry no seed)."""
    consts = consts or _consts()
    B, N = cd.shape[0], cd.shape[1]
    K = W.W1.shape[1]
    leaves = [w.detach().double().cpu().requires_grad_(True) for w in W]
    vals = torch.zeros(B, N, K, dtype=torch.float64)
    total = 0.0
    for b in range(B):
        lo, hi = (0, N) if rows is None else (rows[b] if rows[b] is not None else (0, 0))
        if hi <= lo:
            continue
        Wb = {n: (l[b] if n in TF.GENERATED else l) for n, l in zip(NAMES, leaves)}
        if pe is not None:
            peb = pe[b, lo:hi].detach().double().cpu()
        else:
            col = lambda a: a[b, lo:hi].detach().double().cpu().reshape(-1, 1)
            peb = O.encoding_coord(col(xyz[0]), col(xyz[1]), col(xyz[2]), consts.dx, consts.dy, consts.lat_size, consts.lon_size,
                                   consts.pred_t_span)
        cdb = cd[b, lo:hi].detach().double().cpu()
        rb = (ref_in if ref_in is not None else cd)[b, lo:hi].detach().double().cpu()
        o = torch.cat([O.decoder_net(peb, cdb, rb[:, k:k + 1], Wb["W1"][k], Wb["b1"][k], Wb["W2"][k], Wb["b2"][k], Wb["e"][k],
                                     O._net_params(Wb, k)) for k in range(K)], 1)
        total = total + (o * g_o[b, lo:hi].detach().double().cpu()).sum()
        vals[b, lo:hi] = o.detach()
    total.backward()
    return dict(vals=vals, grads=[l.grad if l.grad is not None else torch.zeros_like(l) for l in leaves])


@contextlib.contextmanager
def forced_chunk(chunk):
    """Points per chunk of every library call inside (0: the library's default)."""
    from deepphysinet_b200 import functional as Fn
    orig = Fn._shape
    if chunk:
        Fn._shape = lambda *a, **kw: orig(*a, **{**kw, "chunk": chunk})
    try:
        yield
    finally:
        Fn._shape = orig


def run_pde(W, pts, mode, chunk=0):
    from deepphysinet_b200 import testing as T
    with forced_chunk(chunk):
        return T.run_library(W, pts, mode=mode)


def run_decoder(W, cd, g_o, mode, pe=None, xyz=None, ref=None, chunk=0):
    from deepphysinet_b200 import functional as Fn
    leaves = [w.detach().clone().requires_grad_(True) for w in W]
    with forced_chunk(chunk):
        o = Fn.decoder_values(pe, cd, Fn.DecoderWeights(*leaves), ref=ref, xyz=xyz, mode=mode)
        (o * g_o).sum().backward()
    return dict(vals=o.detach(), grads=[l.grad for l in leaves])


def _draw(B, N, seed, pde=True, K=6):
    W, pts, margin = TF.tie_free_draw(B, N, seed, GUARD, pde=pde, K=K, device="cuda")
    assert margin >= GUARD
    return W, pts


def _seeds(shape, seed):
    """Seeds in [0.5, 1.5): the bias gradients are sums of seeds, and a sum of mixed signs that cancels (a 128-point tile whose
    seeds sum to 1e-5 of their magnitudes) has no relative accuracy in any arithmetic."""
    return (0.5 + torch.rand(*shape, generator=torch.Generator().manual_seed(seed))).cuda()


# ---------------------------------------------------------------------------------------------------------------------------------
# a. PDE shape sweep
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,N,seed,plan", SWEEP, ids=["B%d_N%d" % s[:2] for s in SWEEP])
def test_pde_sweep_strict(B, N, seed, plan):
    assert wgrad_plan(B, N) == plan
    W, pts = _draw(B, N, seed)
    ref = pde_oracle(W, pts)
    bad = []
    for mode in STRICT:
        bad += check(run_pde(W, pts, mode), ref, mode, "pde B=%d N=%d T,splits=%s" % (B, N, plan))
    assert not bad, bad


# ---------------------------------------------------------------------------------------------------------------------------------
# b. tile-local seeds through dpn_decoder_bwd
# ---------------------------------------------------------------------------------------------------------------------------------
TILE_B, TILE_N = 2, 8321


def tile_cases(chunk):
    """Global tiles worth a seed of their own at this chunk size: first and last tile of every wgrad split of every chunk, the
    last and first tile around every chunk boundary, and the last (1-point) tile; sample = alternating, so both are covered."""
    chunk = chunk or TILE_N
    real = -(-TILE_N // TP)
    tiles = set()
    for p0 in range(0, TILE_N, chunk):
        P = min(chunk, TILE_N - p0)
        T, splits = wgrad_plan(TILE_B, P)
        g0, last = p0 // TP, -(-P // TP) - 1
        tiles.update({g0, g0 + last})                                   # chunk boundaries
        for t0, t1 in split_ranges(T, splits):
            tiles.update(g0 + t for t in (t0, t1 - 1) if t <= last)
    tiles.add(real - 1)
    return [(i % TILE_B, t) for i, t in enumerate(sorted(tiles))]


@pytest.fixture(scope="module")
def tile_draw():
    return _draw(TILE_B, TILE_N, 201, pde=False)


@pytest.mark.parametrize("chunk", [0, 2560, 2432])
def test_tile_local_seeds(tile_draw, chunk):
    """chunk 2560: 20-tile chunks, the last one 641 points (6 tiles, the last with 1 point); chunk 2432: 19-tile chunks padded to
    20, so the last tile of every chunk has a padding tile as cluster partner, and the last chunk (1025 points) ends with a 1-point
    tile whose partner is padding.  Unchunked: T = 66, splits [0,22) [22,44) [44,66)."""
    W, pts = tile_draw
    xyz = (pts["x"], pts["y"], pts["t"])
    g_all = _seeds((TILE_B, TILE_N, 6), 7)
    bad = []
    for b, tile in tile_cases(chunk):
        lo, hi = tile * TP, min(TILE_N, tile * TP + TP)
        g_o = torch.zeros_like(g_all)
        g_o[b, lo:hi] = g_all[b, lo:hi]
        ref = decoder_oracle(W, pts["coord_data"], g_o, xyz=xyz, rows=[(lo, hi) if s == b else None for s in range(TILE_B)])
        ref.pop("vals")
        for mode in ALL:
            got = run_decoder(W, pts["coord_data"], g_o, mode, xyz=xyz, chunk=chunk)
            got.pop("vals")
            bad += check(got, ref, mode, "tile %d of sample %d, chunk %d" % (tile, b, chunk))
    assert not bad, bad


# ---------------------------------------------------------------------------------------------------------------------------------
# c. nets without seeds; e. chunked calls against the oracle
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def b3_draw():
    return _draw(3, 1000, 109)


def test_unseeded_nets_and_chunk(b3_draw):
    """g_o seeds only u and q, and no point of [256, 512): with chunk 256 the second chunk has no seed at all, and four nets have
    none in any chunk (zscale_kernel's clamped 2^80 scale).  Their gradient slices must be exactly zero."""
    W, pts = b3_draw
    xyz = (pts["x"], pts["y"], pts["t"])
    g_o = _seeds((3, 1000, 6), 8)
    g_o[..., [1, 2, 3, 5]] = 0
    g_o[:, 256:512] = 0
    ref = decoder_oracle(W, pts["coord_data"], g_o, xyz=xyz)
    bad = []
    for chunk in (0, 256):
        for mode in ALL:
            bad += check(run_decoder(W, pts["coord_data"], g_o, mode, xyz=xyz, chunk=chunk), ref, mode, "u,q seeds only, chunk %d" % chunk)
    assert not bad, bad


@pytest.mark.parametrize("chunk", [256, 384])
def test_chunked_calls_against_oracle(b3_draw, chunk):
    W, pts = b3_draw
    ref_pde = pde_oracle(W, pts)
    xyz = (pts["x"], pts["y"], pts["t"])
    g_o = _seeds((3, 1000, 6), 9)
    ref_dec = decoder_oracle(W, pts["coord_data"], g_o, xyz=xyz)
    bad = []
    for mode in ALL:
        bad += check(run_pde(W, pts, mode, chunk=chunk), ref_pde, mode, "pde B=3 N=1000 chunk %d" % chunk)
        bad += check(run_decoder(W, pts["coord_data"], g_o, mode, xyz=xyz, chunk=chunk), ref_dec, mode, "decoder B=3 N=1000 chunk %d" % chunk)
    assert not bad, bad


# ---------------------------------------------------------------------------------------------------------------------------------
# d. pre-encoded coordinates (PhysicsNet.forward) and K < 6 nets with an explicit ref (VariableNet.forward)
# ---------------------------------------------------------------------------------------------------------------------------------
def _encoded(pts):
    c = _consts()
    col = lambda k, b: pts[k][b].double().cpu().reshape(-1, 1)
    return torch.stack([O.encoding_coord(col("x", b), col("y", b), col("t", b), c.dx, c.dy, c.lat_size, c.lon_size, c.pred_t_span)
                        for b in range(pts["x"].shape[0])]).float().cuda()


@pytest.mark.parametrize("B,N", [(1, 700), (2, 333)])
def test_coord_pe_surface(B, N):
    """B = 1 with [N,192] / [N,6] inputs, as PhysicsNet.forward calls it; B = 2 with [B,N,192]."""
    W, pts = _draw(B, N, 300 + B, pde=False)
    pe = _encoded(pts)
    g_o = _seeds((B, N, 6), 10)
    ref = decoder_oracle(W, pts["coord_data"], g_o, pe=pe)
    bad = []
    for mode in STRICT:
        if B == 1:
            got = run_decoder(W, pts["coord_data"][0], g_o[0], mode, pe=pe[0])
            got["vals"] = got["vals"][None]
        else:
            got = run_decoder(W, pts["coord_data"], g_o, mode, pe=pe)
        bad += check(got, ref, mode, "coord_pe B=%d N=%d" % (B, N))
    assert not bad, bad


@pytest.mark.parametrize("K", [1, 2, 5])
def test_few_nets_with_ref(K):
    W, pts = _draw(2, 700, 310 + K, pde=False, K=K)
    pe = _encoded(pts)
    ref_in = (0.5 * _seeds((2, 700, K), 11)).contiguous()
    g_o = _seeds((2, 700, K), 12)
    ref = decoder_oracle(W, pts["coord_data"], g_o, pe=pe, ref_in=ref_in)
    bad = []
    for mode in STRICT:
        bad += check(run_decoder(W, pts["coord_data"], g_o, mode, pe=pe, ref=ref_in), ref, mode, "K=%d with ref" % K)
    assert not bad, bad


# ---------------------------------------------------------------------------------------------------------------------------------
# f. fused margin path against fp64
# ---------------------------------------------------------------------------------------------------------------------------------
def test_fused_margin_strict():
    """pde_margin_residual against the fp64 composition: closed-form PDE terms and gradients plus autograd smooth_l1 of the oracle's
    values (interface_physics.py:464-474); the margin loss of each sample is compared as a seventh loss term."""
    from deepphysinet_b200 import functional as Fn
    B, N, beta, factor = 2, 700, 0.1, 1.0e6
    W, pts = _draw(B, N, 320)
    target = pts["coord_data"] + 0.2 * torch.randn(B, N, 6, generator=torch.Generator().manual_seed(13)).cuda()
    ref = pde_oracle(W, pts)
    leaves = [w.detach().double().cpu().requires_grad_(True) for w in W]
    mref, o_ref = [], []
    for b in range(B):
        Wb = {n: (l[b] if n in TF.GENERATED else l) for n, l in zip(NAMES, leaves)}
        c = _consts()
        col = lambda k: pts[k][b].double().cpu().reshape(-1, 1)
        pe = O.encoding_coord(col("x"), col("y"), col("t"), c.dx, c.dy, c.lat_size, c.lon_size, c.pred_t_span)
        o = torch.cat(O.decode_generated(pe, pts["coord_data"][b].double().cpu(), Wb), 1)
        ml = torch.nn.functional.smooth_l1_loss(o, target[b].double().cpu(), beta=beta, reduction="none").mean() * factor
        (ml / B).backward()
        mref.append(ml.detach())
        o_ref.append(o.detach())
    ref = dict(terms=torch.cat([ref["terms"], torch.stack(mref)[:, None]], 1), vals=torch.stack(o_ref),
               grads=[g + l.grad for g, l in zip(ref["grads"], leaves)])
    bad = []
    for mode in STRICT:
        a = [w.detach().clone().requires_grad_(True) for w in W]
        total, terms, mloss, o = Fn.pde_margin_residual(pts["x"], pts["y"], pts["t"], pts["f"], pts["coord_data"], target,
                                                        Fn.DecoderWeights(*a), beta=beta, factor=factor, mode=mode)
        total.backward()
        got = dict(terms=torch.cat([terms, mloss[:, None]], 1), vals=o, grads=[l.grad for l in a])
        bad += check(got, ref, mode, "margin B=%d N=%d" % (B, N))
    assert not bad, bad
