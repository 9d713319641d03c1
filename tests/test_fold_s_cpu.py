"""CPU: the second fold of the reverse sweep (DESIGN.md section 3) in fp64 against oracle/closed_form.py.

zc = zh W2^T + zd Wd^T + dov bsum is never formed.  After the last chunk, S = m3^T zc, summed over the samples, comes from the sums
the weight-gradient kernel accumulates anyway:
    S = sum_b (m3^T zh)_b W2_b^T + (sum_b m3^T zd) Wd^T + sum_b sm3_b (x) bsum_b,     sm3 = m3^T dov
and dWa = diag(u) S, dba = u sum_b sm3_b, vg[j] = sum_i Wa[j,i] S[j,i] + ba[j] sum_b sm3_b[j] (dWb = wo (x) vg, dwo = 2vc + Wb vg +
bb sdo), vc = sum_b [(sum_p zh)_b W2_b^T + (sum_p dov)_b bsum_b] + (sum_{b,p} zd) Wd^T.  S is formed unscaled by u: a net with
wo = 0 has u = 0 but still needs vg for dwo.
"""
import pytest
import torch

from oracle import closed_form as CF
from oracle import tiefree as TF
from tests import test_gpu_strict_parity as S
from tests.test_fold_cpu import _rel, stages  # noqa: F401  (stages: the fixture of one sample, with a wo = 0 and a u = 0 net)


def _sums(Ws, st, k):
    """What the weight-gradient kernel accumulates for net k of one sample: m3^T zh, m3^T zd, sm3 and the column sums."""
    s = st["nets"][k]
    dv = st["dov"][:, k:k + 1]
    zh, zd = s["zh"], dv * st["pe6"]
    bsum = Ws["b2"][k] + Ws["bd"][k] + Ws["e"][k]
    return dict(Mh=s["m3"].T @ zh, Md=s["m3"].T @ zd, sm3=s["m3"].T @ dv[:, 0], szh=zh.sum(0), szd=zd.sum(0), sdo=dv.sum(),
                W2=Ws["W2"][k], bsum=bsum)


def _fold_s(per_sample, Ws, k):
    """dWa, dba, vg, vc of net k from the per-sample sums, in the order fold_s_kernel takes them."""
    Wd, Wa, ba = Ws["Wd"][k], Ws["Wa"][k], Ws["ba"][k]
    u = Ws["Wb"][k].T @ Ws["wo"][k]
    Sm = sum(p["Mh"] @ p["W2"].T + torch.outer(p["sm3"], p["bsum"]) for p in per_sample) + sum(p["Md"] for p in per_sample) @ Wd.T
    vc = sum(p["W2"] @ p["szh"] + p["sdo"] * p["bsum"] for p in per_sample) + Wd @ sum(p["szd"] for p in per_sample)
    sm3 = sum(p["sm3"] for p in per_sample)
    vg = (Wa * Sm).sum(1) + ba * sm3
    return u[:, None] * Sm, u * sm3, vg, vc


def _check(name, got, want):
    if want.abs().max() == 0:
        assert got.abs().max() == 0, name
    else:
        assert _rel(got, want) < 1e-12, (name, _rel(got, want))


def _check_net(Ws, G, k, dWa, dba, vg, vc, sdo):
    wo, Wb, bb = Ws["wo"][k], Ws["Wb"][k], Ws["bb"][k]
    _check("Wa", dWa, G["Wa"][k])
    _check("ba", dba, G["ba"][k])
    _check("Wb", torch.outer(wo, vg), G["Wb"][k])
    _check("wo", 2.0 * vc + Wb @ vg + bb * sdo, G["wo"][k])


@pytest.mark.parametrize("k", range(6))
def test_fold_s_one_sample(stages, k):  # noqa: F811
    Ws, G, st = stages
    p = _sums(Ws, st, k)
    dWa, dba, vg, vc = _fold_s([p], Ws, k)
    _check_net(Ws, G, k, dWa, dba, vg, vc, p["sdo"])
    s = st["nets"][k]                                              # and the intermediate vectors themselves
    _check("vc", vc, s["zc"].sum(0))
    _check("vg", vg, s["gz"].sum(0))


def test_fold_s_nets_without_u_keep_vg(stages):  # noqa: F811
    """The wo = 0 and u = 0 nets: dWa = dba = 0 exactly, while vg is not zero and enters dwo."""
    Ws, G, st = stages
    for k in (1, 2):
        u = Ws["Wb"][k].T @ Ws["wo"][k]
        assert u.abs().max() == 0
        dWa, dba, vg, vc = _fold_s([_sums(Ws, st, k)], Ws, k)
        assert dWa.abs().max() == 0 and dba.abs().max() == 0
        assert vg.abs().max() > 0 and _rel(vg, st["nets"][k]["gz"].sum(0)) < 1e-12


@pytest.fixture(scope="module")
def two_samples():
    """A two-sample batch: the generated weights differ per sample, the static ones (Wd, Wa, ba, Wb, wo, ...) are shared; net 1 has
    wo = 0 and net 2 has u = 0 in both samples."""
    W, pts, _ = TF.tie_free_draw(2, 64, 11, S.GUARD)
    out = []
    for b in range(2):
        Ws = {k: v.double().clone() for k, v in TF.sample_weights(W, b).items()}
        Ws["wo"][1] = 0.0
        Ws["Wb"][2] = 0.0
        c = {k: v[b].double().reshape(-1, 1) for k, v in pts.items() if k != "coord_data"}
        L, G, v, j, st = CF.pde_fwd_bwd(c["x"], c["y"], c["t"], c["f"], pts["coord_data"][b].double(), Ws, return_stages=True)
        out.append((Ws, G, st))
    return out


@pytest.mark.parametrize("k", range(6))
def test_fold_s_two_samples(two_samples, k):
    """The sum over samples precedes diag(u) and the dot products with Wa: the static gradients are the sums of the per-sample
    ones of the closed form."""
    per = [_sums(Ws, st, k) for Ws, G, st in two_samples]
    Ws0 = two_samples[0][0]
    for name in ("Wd", "Wa", "ba", "Wb", "wo", "bb", "bo"):
        assert torch.equal(two_samples[0][0][name], two_samples[1][0][name]), name
    dWa, dba, vg, vc = _fold_s(per, Ws0, k)
    G = {n: two_samples[0][1][n] + two_samples[1][1][n] for n in ("Wa", "ba", "Wb", "wo")}
    _check_net(Ws0, G, k, dWa, dba, vg, vc, per[0]["sdo"] + per[1]["sdo"])
