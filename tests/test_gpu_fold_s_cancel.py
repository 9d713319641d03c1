"""GPU (-m gpu): dWa, dba, dWb and dwo on a draw where the bias bsum = b2 + bd + e cancels most of c = h1 W2^T + PE6 Wd^T + bsum.

The weight-gradient kernel never sees zc = dov c + ct: dWa = diag(u) S, vg and vc come from S = m3^T zc formed after the last chunk
as sum_b (m3^T zh)_b W2_b^T + (sum_b m3^T zd) Wd^T + sum_b sm3_b (x) bsum_b.  Where c is a small difference of h1 W2^T + PE6 Wd^T
and bsum, the three terms of S cancel in the same way.  The draw starts from a threshold-free decoder draw and shifts bd by
delta = -(1 - 1/64) mean_{b,p}(c), and compensates with ba <- ba - Wa delta and bo <- bo - 2wo.delta: the ReLU masks, the values and
the Jacobian do not change (checked in fp64), only c shrinks.  The decoder backward must meet the strict bounds of
tests/test_gpu_strict_parity.py in every split mode, in one chunk and in several.  (The kernels that formed zc and contracted
m3^T zc directly pass it as well: it pins behaviour that no earlier test covered.)
"""
import pytest
import torch

from oracle import dpn_oracle as O
from oracle import tiefree as TF
from tests import test_gpu_strict_parity as S

pytestmark = pytest.mark.gpu


def _stages(W, pts):
    """fp64 per sample: (a1 [N,K,H], a3 [N,K,H], c [N,K,H])"""
    consts = S._consts()
    out = []
    for b in range(pts["x"].shape[0]):
        col = lambda a: a[b].detach().double().cpu().reshape(-1, 1)
        pe = O.encoding_coord(col(pts["x"]), col(pts["y"]), col(pts["t"]), consts.dx, consts.dy, consts.lat_size, consts.lon_size,
                              consts.pred_t_span)
        pe6 = O.sine_cos_pe(pts["coord_data"][b].detach().double().cpu(), 16)
        Wb = TF.sample_weights(W, b)
        a1, a3 = TF.preactivations(pe, pe6, Wb)
        c = torch.einsum("nkl,kil->nki", torch.relu(a1), Wb["W2"]) + torch.einsum("nl,kil->nki", pe6, Wb["Wd"]) + \
            (Wb["b2"] + Wb["bd"] + Wb["e"])[None]
        out.append((a1, a3, c))
    return out


def _cancelling(W, pts, keep=1.0 / 64):
    st = _stages(W, pts)
    delta = -(1.0 - keep) * torch.stack([c.mean(0) for _, _, c in st]).mean(0)          # [K, H]
    Wa, wo = W.Wa.detach().double().cpu(), W.wo.detach().double().cpu()
    dev = W.bd.device
    bd = (W.bd.detach().double().cpu() + delta).float().to(dev)
    ba = (W.ba.detach().double().cpu() - torch.einsum("kji,ki->kj", Wa, delta)).float().to(dev)
    bo = (W.bo.detach().double().cpu() - 2.0 * (wo * delta).sum(1)).float().to(dev)
    return W._replace(bd=bd, ba=ba, bo=bo)


@pytest.fixture(scope="module")
def cancel_draw():
    W, pts = S._draw(2, 1000, 307, pde=False)
    return W, _cancelling(W, pts), pts


def test_shift_keeps_masks_values_and_jacobian(cancel_draw):
    """In fp64: the masks are the same, a3 and the outputs move by the fp32 rounding of the shifted biases only, and the mean of c
    over the draw's points is 1 / 64 of what it was."""
    W0, W, pts = cancel_draw
    xyz = (pts["x"], pts["y"], pts["t"])
    s0, s1 = _stages(W0, pts), _stages(W, pts)
    for (a1, a3, _), (b1, b3, _) in zip(s0, s1):
        assert torch.equal(a1, b1)
        assert torch.equal(a3 > 0, b3 > 0)
        assert ((a3 - b3).abs().max() / a3.abs().max()).item() < 1e-6
    m0, m1 = (torch.stack([c.mean(0) for _, _, c in s]).mean(0) for s in (s0, s1))
    assert (m1.norm() / m0.norm()).item() < 1.0 / 50
    g_o = S._seeds((2, 1000, 6), 37)
    r0 = S.decoder_oracle(W0, pts["coord_data"], g_o, xyz=xyz)
    r1 = S.decoder_oracle(W, pts["coord_data"], g_o, xyz=xyz)
    assert ((r1["vals"] - r0["vals"]).abs().max() / r0["vals"].abs().max()).item() < 1e-6
    # the reverse sweep q = y W2 does not depend on c: dW1 = qm^T zp is unchanged (dWa, dwo are not: they follow c)
    assert ((r1["grads"][0] - r0["grads"][0]).abs().max() / r0["grads"][0].abs().max()).item() < 1e-6


@pytest.mark.parametrize("chunk", [0, 256])
def test_cancelling_bias_strict(cancel_draw, chunk):
    _, W, pts = cancel_draw
    xyz = (pts["x"], pts["y"], pts["t"])
    g_o = S._seeds((2, 1000, 6), 37)
    ref = S.decoder_oracle(W, pts["coord_data"], g_o, xyz=xyz)
    bad = []
    for mode in ("f16x3", "f16x3a", "bf16x3"):
        bad += S.check(S.run_decoder(W, pts["coord_data"], g_o, mode, xyz=xyz, chunk=chunk), ref, mode, "bsum cancels c, chunk %d" % chunk)
    assert not bad, bad
