"""CPU: the branch-steered draws of oracle/tiefree.py and the constants of the oracles, without a GPU.

  * the closed form (the fp64 twin tests/test_gpu_residual_branches.py compares the kernels with) matches the autograd oracle
    in every regime and under non-default constants;
  * steered draws reach every branch, keep the weights of random_decoder_weights and, under each mode's emulated operand rounding,
    keep the exact ReLU masks, clip decisions and vapour switch;
  * the tests bite: a closed form with one kernel-side mistake (kappa = 1 on clipped points, an open interval at the bounds, q's lo
    rounded to fp32, no q_s floor, dx and dy swapped in the Jacobian scale, the u and v loss factors swapped, n_norm ignored) violates
    the fp32 strict bounds on the draw that targets it.
"""
import inspect

import pytest
import torch

from deepphysinet_b200 import testing as T
from oracle import closed_form as CF
from oracle import dpn_oracle as O
from oracle import tiefree as TF
from tests import test_gpu_residual_branches as R
from tests import test_gpu_strict_parity as S


def _worst(E):
    return max(v for v, _ in E.values())


@pytest.mark.parametrize("case", ["default", "custom", "custom_noclip"])
def test_closed_form_matches_autograd_in_every_regime(case):
    consts = R._default() if case == "default" else R.custom_consts(case == "custom")
    names = list(TF.regime_table(consts)) if consts.with_clip else ["free", "T_hi", "q_lo", "p_hi"]
    regimes = [[n for n in names if n != "rho_lo"], ["free", "rho_lo"]] if case == "default" else names
    W, pts, _ = TF.tie_free_draw(2, 20 * len(names), 7, 5e-4, consts=consts, regimes=regimes, min_count=2)
    ref = T.oracle_reference(W, pts, consts)
    E = S.strict_errors(S.pde_oracle(W, pts, consts), ref)
    print(case, {g: "%.1e" % v for g, (v, _) in E.items()})
    assert _worst(E) <= 1e-10, E


def test_oracle_reference_forwards_every_constant():
    """testing.oracle_reference under custom_consts differs from the same call at the default normalisation and physics."""
    import dataclasses
    consts = R.custom_consts()
    W, pts, _ = TF.tie_free_draw(1, 40, 8, 5e-4, consts=consts)
    a = T.oracle_reference(W, pts, consts)
    b = T.oracle_reference(W, pts, dataclasses.replace(R._default(), dx=consts.dx, dy=consts.dy, lat_size=consts.lat_size,
                                                        lon_size=consts.lon_size, pred_t_span=consts.pred_t_span, factor=consts.factor))
    assert not torch.allclose(a["vals"], b["vals"]) and not torch.allclose(a["terms"], b["terms"])


def test_steered_draws_reach_every_branch_and_keep_the_weights():
    from deepphysinet_b200.testing import random_decoder_weights
    seen = {}
    for consts, regimes in ((R._default(), R.SWEEP[-1][1]), (R.custom_consts(), list(TF.regime_table(R.custom_consts())))):
        W, pts, margin = TF.tie_free_draw(2, R.N_SWEEP, 9, 5e-4, consts=consts, regimes=regimes)
        assert margin >= 5e-4
        W0, _ = random_decoder_weights(2, 17, 9, device="cpu", consts=consts)
        assert all(torch.equal(a, b) for a, b in zip(W, W0))
        for c in TF.branches(W, pts, consts):
            print(c)
            for k, v in c.items():
                seen[k] = seen.get(k, 0) + v
    assert all(v > 0 for v in seen.values()), seen
    with pytest.raises(RuntimeError, match="branches short"):
        TF.tie_free_draw(1, 60, 9, 5e-4, regimes=["free", "tie"], min_count=40)


def _decisions(args, consts, rnd):
    """ReLU masks, kappa of p, T, q, rho and the vapour switch of one sample under operand rounding `rnd`."""
    _, _, vals, jac, st = CF.pde_fwd_bwd(*args, rnd=rnd, return_stages=True, **CF.kwargs_of(consts))
    raw = st["o"][:, 2:] * torch.tensor(consts.std[2:], dtype=torch.float64) + torch.tensor(consts.mean[2:], dtype=torch.float64)
    kap = (raw >= torch.tensor(consts.lo[2:])) & (raw <= torch.tensor(consts.hi[2:]))
    u, v, p, T_, q = [vals[:, i] for i in range(5)]
    dp = jac[:, 2, 2] + u * jac[:, 2, 0] + v * jac[:, 2, 1]
    q_s = torch.clamp_min(O.saturation_q(p, T_), 1e-6)
    masks = [torch.stack([n["m1"] for n in st["nets"]]), torch.stack([n["m3"] for n in st["nets"]])]
    return masks + [kap, (dp < 0) & (q >= q_s)]


@pytest.mark.parametrize("rnd,guard", [(lambda a: a.float().double(), 1e-4), (CF.f16_split_round, 1e-4), (CF.bf16_split_round, 5e-4)],
                         ids=["fp32", "f16x3", "bf16x3"])
def test_emulated_rounding_keeps_every_decision(rnd, guard):
    consts = R._default()
    W, pts, _ = TF.tie_free_draw(2, 300, 10, guard, regimes=R.SWEEP[-1][1])
    for b in range(2):
        col = lambda k: pts[k][b].double().reshape(-1, 1)
        args = (col("x"), col("y"), col("t"), col("f"), pts["coord_data"][b].double(), TF.sample_weights(W, b))
        for name, e, g in zip(("m1", "m3", "kappa", "switch"), _decisions(args, consts, lambda a: a), _decisions(args, consts, rnd)):
            assert torch.equal(e, g), (b, name)


# ---------------------------------------------------------------------------------------------------------------------------------
# mutants: each is one kernel-side mistake restated in the closed form
# ---------------------------------------------------------------------------------------------------------------------------------
def _mutant(fn, old, new):
    """fn (a closed_form function) with the source text `old` replaced by `new`, compiled in closed_form's namespace."""
    src = inspect.getsource(fn)
    assert old in src, (fn.__name__, old)
    ns = {}
    exec(compile(src.replace(old, new), CF.__file__, "exec"), vars(CF).copy(), ns)
    return fn.__name__, ns[fn.__name__]


RS = CF.residual_and_seeds
MUTANTS = {
    "kappa_one_on_clipped": _mutant(RS, "kap[:, 2:] = ((raw[:, 2:] >= lo[2:]) & (raw[:, 2:] <= hi[2:])).to(dt)", "pass"),
    "open_interval": _mutant(RS, "(raw[:, 2:] >= lo[2:]) & (raw[:, 2:] <= hi[2:])", "(raw[:, 2:] > lo[2:]) & (raw[:, 2:] < hi[2:])"),
    "q_lo_in_fp32": _mutant(RS, "    raw = o * std + mean\n", "    lo[4] = lo[4].float().double()\n    raw = o * std + mean\n"),
    "no_qs_floor": _mutant(RS, "torch.clamp_min(0.622 * e_s / (p - 0.378 * e_s), 1e-6)", "0.622 * e_s / (p - 0.378 * e_s)"),
    "dx_dy_swapped": _mutant(CF.pde_fwd_bwd, "1.0 / (dx * (lon_size - 1)), 1.0 / (dy * (lat_size - 1))",
                             "1.0 / (dy * (lon_size - 1)), 1.0 / (dx * (lat_size - 1))"),
    "uv_factors_swapped": _mutant(RS, "    dt = o.dtype\n", "    dt = o.dtype\n    fact = (fact[1], fact[0]) + tuple(fact[2:])\n"),
}


def _target(name):
    """(W, pts, consts, n_total of the reference) of the draw each mutant targets."""
    if name == "open_interval":
        W, pts, consts = R.interval_case(device="cpu")
        return W, pts, consts, None
    if name in ("dx_dy_swapped", "uv_factors_swapped"):
        consts = R.custom_consts()
        W, pts, _ = TF.tie_free_draw(1, 300, 11, 5e-4, consts=consts)
        return W, pts, consts, None
    regime = dict(kappa_one_on_clipped=["free", "p_lo", "T_hi", "rho_lo"], q_lo_in_fp32=["tie"], no_qs_floor=["T_hi"],
                  n_norm_ignored=["free"])[name]
    W, pts, _ = TF.tie_free_draw(1, 300, 12, 5e-4, regimes=regime)
    return W, pts, R._default(), (900 if name == "n_norm_ignored" else None)


@pytest.mark.parametrize("name", sorted(MUTANTS) + ["n_norm_ignored"])
def test_mutant_violates_the_fp32_bounds(name, monkeypatch):
    W, pts, consts, n_total = _target(name)
    ref = S.pde_oracle(W, pts, consts, n_total=n_total)
    assert not S.violations(S.strict_errors(S.pde_oracle(W, pts, consts, n_total=n_total), ref), "fp32")
    if name in MUTANTS:
        attr, fn = MUTANTS[name]
        monkeypatch.setattr(CF, attr, fn)
    got = S.pde_oracle(W, pts, consts)                       # n_norm_ignored: the loss means divide by N
    bad = S.violations(S.strict_errors(got, ref), "fp32")
    print(name, bad[:3])
    assert bad, name


def test_seed_sum_floor_still_rejects_a_dropped_point():
    """The floor of seed_sum_scale (1/8 of the terms' magnitude) leaves the strict bounds able to see one dropped point of a
    mixed draw, whichever point it is."""
    consts = R._default()
    W, pts, _ = TF.tie_free_draw(2, 300, 13, 5e-4, regimes=R.SWEEP[-1][1], min_count=2)
    ref = R.pde_ref(W, pts, consts)
    for p in range(0, 300, 37):
        got = dict(ref, grads=S.pde_oracle(W, pts, consts, drop=(p % 2, torch.tensor([p])))["grads"])
        for mode in S.STRICT:
            assert any(v[0] == "grad" for v in S.violations(S.strict_errors(got, ref), mode)), (p, mode)
