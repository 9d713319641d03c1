"""GPU (-m gpu): the fold of the reverse sweep on a draw where 2wo cancels most of m3 (diag(u) Wa).

Pass 1 forms q = m3 P + c2 (P = diag(u) Wa W2, c2 = 2 W2^T wo) and the weight-gradient kernel forms dW2, dWd, db2 as
Wa^T (diag(u) m3^T z) + 2wo (x) sum_p z, without ever forming y = m3 (diag(u) Wa) + 2wo.  Where y is a small difference of
two large terms, each of those sums is one too, so this is where the reassociation is most sensitive.  The draw keeps u and the
ReLU masks of a threshold-free decoder draw (they do not depend on wo or Wb) and sets wo so that 2wo cancels 63 / 64 of the
mean of m3 (diag(u) Wa) over the draw's points, with Wb corrected so that u = Wb^T wo is unchanged.  The decoder backward must
meet the strict bounds of tests/test_gpu_strict_parity.py in every split mode, in one chunk and in several.
"""
import pytest
import torch

from oracle import dpn_oracle as O
from oracle import tiefree as TF
from tests import test_gpu_strict_parity as S

pytestmark = pytest.mark.gpu


def _cancelling(W, pts, keep=1.0 / 64):
    consts = S._consts()
    B, N = pts["x"].shape
    col = lambda a, b: a[b].detach().double().cpu().reshape(-1, 1)
    m3 = 0.0
    for b in range(B):
        pe = O.encoding_coord(col(pts["x"], b), col(pts["y"], b), col(pts["t"], b), consts.dx, consts.dy, consts.lat_size,
                              consts.lon_size, consts.pred_t_span)
        pe6 = O.sine_cos_pe(pts["coord_data"][b].detach().double().cpu(), 16)
        _, a3 = TF.preactivations(pe, pe6, TF.sample_weights(W, b))
        m3 = m3 + (a3 > 0).double().mean(0) / B                            # [K, 256]
    Wa, Wb, wo = (w.detach().double().cpu() for w in (W.Wa, W.Wb, W.wo))
    u = torch.einsum("kij,ki->kj", Wb, wo)
    wo_new = -0.5 * (1.0 - keep) * torch.einsum("kl,klj->kj", u * m3, Wa)
    Wb_new = Wb + torch.einsum("ki,kj->kij", wo_new, u - torch.einsum("kij,ki->kj", Wb, wo_new)) / (wo_new * wo_new).sum(1)[:, None, None]
    dev = W.wo.device
    W = W._replace(wo=wo_new.float().to(dev), Wb=Wb_new.float().to(dev))
    u_new = torch.einsum("kij,ki->kj", W.Wb.double().cpu(), W.wo.double().cpu())
    assert ((u_new - u).abs().max() / u.abs().max()).item() < 1e-5
    return W


@pytest.fixture(scope="module")
def cancel_draw():
    W, pts = S._draw(2, 1000, 301, pde=False)
    return _cancelling(W, pts), pts


def test_cancellation_is_strong(cancel_draw):
    """The draw does what it is for: y is smaller than either of its two terms (before the change of wo: 9x larger than
    m3 (diag(u) Wa), 2wo dominating; after it: 0.65x, the point-to-point variation of the mask is what remains)."""
    W, pts = cancel_draw
    consts = S._consts()
    Wb = TF.sample_weights(W, 0)
    col = lambda a: a[0].detach().double().cpu().reshape(-1, 1)
    pe = O.encoding_coord(col(pts["x"]), col(pts["y"]), col(pts["t"]), consts.dx, consts.dy, consts.lat_size, consts.lon_size,
                          consts.pred_t_span)
    _, a3 = TF.preactivations(pe, O.sine_cos_pe(pts["coord_data"][0].detach().double().cpu(), 16), Wb)
    u = torch.einsum("kij,ki->kj", Wb["Wb"], Wb["wo"])
    big = torch.einsum("nkl,klj->nkj", (a3 > 0).double() * u, Wb["Wa"])
    y = big + 2.0 * Wb["wo"]
    assert (y.norm() / big.norm()).item() < 0.7 and (y.norm() / (2.0 * Wb["wo"]).norm() / y.shape[0] ** 0.5).item() < 1.0


@pytest.mark.parametrize("chunk", [0, 256])
def test_cancelling_wo_strict(cancel_draw, chunk):
    W, pts = cancel_draw
    xyz = (pts["x"], pts["y"], pts["t"])
    g_o = S._seeds((2, 1000, 6), 31)
    ref = S.decoder_oracle(W, pts["coord_data"], g_o, xyz=xyz)
    bad = []
    for mode in ("f16x3", "f16x3a", "bf16x3"):
        bad += S.check(S.run_decoder(W, pts["coord_data"], g_o, mode, xyz=xyz, chunk=chunk), ref, mode, "2wo cancels, chunk %d" % chunk)
    assert not bad, bad
