"""CPU: the fold of the reverse sweep (DESIGN.md section 3) in fp64 against oracle/closed_form.py.

Pass 1 never forms y = (u*m3) Wa + 2wo: it contracts the bare mask against P = diag(u) Wa W2 and adds c2 = 2 W2^T wo, and the
weight-gradient kernel contracts the mask against zh / zd, so that dW2, dWd and db2 follow after the last chunk from
Wa^T (diag(u) m3^T z) + 2wo (x) sum_p z.  These identities hold to rounding, also for nets with u = 0 or wo = 0; the epilogue of
G4 takes q sQ = (acc / sP) sQ + c2 sQ in two steps, which stays finite and exact over the whole clamp range of the plan.
"""
import numpy as np
import pytest
import torch

from oracle import closed_form as CF
from oracle import tiefree as TF
from tests import test_gpu_strict_parity as S


@pytest.fixture(scope="module")
def stages():
    W, pts, _ = TF.tie_free_draw(1, 96, 5, S.GUARD)
    Ws = {k: v.double().clone() for k, v in TF.sample_weights(W, 0).items()}
    Ws["wo"][1] = 0.0                     # wo = 0: u = 0 as well, y = 0
    Ws["Wb"][2] = 0.0                     # u = 0 with wo != 0: y = 2wo on every point
    c = {k: v[0].double().reshape(-1, 1) for k, v in pts.items() if k != "coord_data"}
    L, G, v, j, st = CF.pde_fwd_bwd(c["x"], c["y"], c["t"], c["f"], pts["coord_data"][0].double(), Ws, return_stages=True)
    return Ws, G, st


def _rel(a, b):
    return ((a - b).abs().max() / b.abs().max().clamp_min(1e-300)).item()


def _fold(Ws, k):
    u = Ws["Wb"][k].T @ Ws["wo"][k]
    P = u[:, None] * (Ws["Wa"][k] @ Ws["W2"][k])
    c2 = 2.0 * Ws["W2"][k].T @ Ws["wo"][k]
    return u, P, c2


@pytest.mark.parametrize("k", range(6))
def test_q_is_the_mask_against_p(stages, k):
    Ws, G, st = stages
    s = st["nets"][k]
    u, P, c2 = _fold(Ws, k)
    q = (s["m3"] @ P + c2) * s["m1"]
    if s["qm"].abs().max() == 0:
        assert q.abs().max() == 0
    else:
        assert _rel(q, s["qm"]) < 1e-12


@pytest.mark.parametrize("k", range(6))
def test_reassociated_gradients(stages, k):
    Ws, G, st = stages
    s = st["nets"][k]
    u, P, c2 = _fold(Ws, k)
    dv = st["dov"][:, k:k + 1]
    zh, zd = s["zh"], dv * st["pe6"]
    wo2, Wa = 2.0 * Ws["wo"][k], Ws["Wa"][k]
    um3 = u[:, None] * s["m3"].T                                   # diag(u) m3^T, what the weight-gradient kernel contracts
    dW2 = Wa.T @ (um3 @ zh) + torch.outer(wo2, zh.sum(0))
    dWd = Wa.T @ (um3 @ zd) + torch.outer(wo2, zd.sum(0))
    db2 = Wa.T @ (um3 @ dv[:, 0]) + wo2 * dv.sum()
    for name, got in (("W2", dW2), ("Wd", dWd), ("b2", db2), ("e", db2), ("bd", db2)):
        want = G[name][k]
        if want.abs().max() == 0:
            assert got.abs().max() == 0, name
        else:
            assert _rel(got, want) < 1e-12, (name, _rel(got, want))


def _scale_for(bound):
    """dpn_tc.cu scale_for: the largest power of two <= 2^15 / bound, clamped to [2^-80, 2^80]"""
    x = 32768.0 / max(bound, 1e-30)
    return float(min(max(2.0 ** np.floor(np.log2(x)), 2.0 ** -80), 2.0 ** 80))


def test_epilogue_scale_steps_stay_finite():
    """q sQ = (acc * (1 / sP)) * sQ + c2 sQ in fp32, acc = (m3 P) sP, with sP = scale_for(32 max |P|) and sQ = scale_for(Mq): for
    bounds Mq over the fp32 range, every max |P| <= Mq (DESIGN.md section 6) down to P = 0, and values |m3 P| up to
    min(Mq, 256 max |P|), each step is finite and the result is the fp64 value to fp32 rounding - although the one-factor
    form sQ / sP leaves the fp32 range at the corners of the clamps."""
    f32 = np.float32
    for eq in range(-120, 121, 8):
        Mq = 2.0 ** eq + 3.0 * 2.0 ** (eq - 3)
        sQ = _scale_for(Mq)
        for d in (0, 1, 5, 20, 60, 200, None):
            mP = 0.0 if d is None else Mq * 2.0 ** -d
            if mP != 0.0 and mP < 1.2e-38:
                continue
            sP = _scale_for(32.0 * mP)
            for qv in (mP, -0.3 * mP, 2.0 ** -12 * mP, min(Mq, 256.0 * mP)):   # |m3 P| <= min(Mq, 256 max |P|)
                acc = f32(qv * sP)
                with np.errstate(over="raise", invalid="raise", under="ignore"):
                    r = f32(f32(acc * f32(1.0 / sP)) * f32(sQ))
                want = qv * sQ
                assert np.isfinite(r) and abs(float(r) - want) <= 2.0 ** -22 * abs(want) + 1e-30, (eq, d, qv)
    with np.errstate(all="ignore"):
        assert not np.isfinite(f32(2.0 ** 80) / f32(2.0 ** -80)) and f32(2.0 ** -80) / f32(2.0 ** 80) == 0.0
