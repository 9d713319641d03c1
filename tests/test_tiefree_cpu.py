"""CPU: threshold-free draws (oracle/tiefree.py) and the strict comparator of tests/test_gpu_strict_parity.py, without a GPU.

  * construction: the returned points clear the guard, the weights are those of random_decoder_weights with the same seed;
  * emulated masks: under each mode's operand rounding the draws take exactly the exact-arithmetic ReLU masks;
  * the comparator bites: a dropped point, a dropped 128-point tile and one (sample, net) gradient slice off by 2^-11 are each
    rejected by the strict bounds, while the per-draw whole-tensor bound of the statistical tests (3e-3) accepts the dropped point
    and the 2^-11 slice.
"""
import pytest
import torch

from oracle import closed_form as CF
from oracle import tiefree as TF
from tests import test_gpu_strict_parity as S

OLD_GRAD = 3e-3                       # per-draw bound on each whole gradient tensor in tests/test_gpu_f16x3.py


@pytest.mark.parametrize("B,N,seed,guard,pde,K", [(1, 300, 1, 1e-4, True, 6), (2, 150, 2, 5e-4, True, 6),
                                                   (2, 200, 3, 5e-4, False, 6), (1, 100, 4, 1e-4, False, 2)])
def test_draw_clears_guard_and_keeps_weights(B, N, seed, guard, pde, K):
    from deepphysinet_b200.testing import random_decoder_weights
    W, pts, margin = TF.tie_free_draw(B, N, seed, guard, pde=pde, K=K)
    assert margin >= guard
    assert pts["x"].shape == (B, N) and pts["coord_data"].shape == (B, N, 6)
    W0, _ = random_decoder_weights(B, 17, seed, device="cpu", K=K)
    for a, b in zip(W, W0):
        assert torch.equal(a, b)
    _, cand = random_decoder_weights(B, TF.pool_size(N, guard), seed, device="cpu", K=K)
    for b in range(B):                                  # the points are candidates, in candidate order
        idx = [int(torch.nonzero(cand["x"][b] == v)[0]) for v in pts["x"][b]]
        assert idx == sorted(set(idx))
        assert torch.equal(cand["coord_data"][b, idx], pts["coord_data"][b])


def test_draw_raises_when_the_pool_runs_out():
    with pytest.raises(RuntimeError, match="clear the guard"):
        TF.tie_free_draw(1, 50, 1, 0.5, pde=False)


def _fp32_operands(a):
    return a.float().double()


@pytest.mark.parametrize("rnd,guard", [(_fp32_operands, 1e-4), (CF.f16_split_round, 1e-4), (CF.bf16_split_round, 5e-4)],
                         ids=["fp32", "f16x3", "bf16x3"])
def test_emulated_rounding_keeps_exact_masks(rnd, guard):
    W, pts, _ = TF.tie_free_draw(2, 400, 5, guard)
    for b in range(2):
        Wb = TF.sample_weights(W, b)
        col = lambda k: pts[k][b].double().reshape(-1, 1)
        args = (col("x"), col("y"), col("t"), col("f"), pts["coord_data"][b].double(), Wb)
        exact = CF.pde_fwd_bwd(*args, return_stages=True)[4]["nets"]
        emul = CF.pde_fwd_bwd(*args, rnd=rnd, return_stages=True)[4]["nets"]
        for k in range(6):
            assert torch.equal(exact[k]["m1"], emul[k]["m1"]), (b, k)
            assert torch.equal(exact[k]["m3"], emul[k]["m3"]), (b, k)


def test_split_rule_copy_matches_the_sweep_comments():
    for B, N, _, plan in S.SWEEP:
        assert S.wgrad_plan(B, N) == plan, (B, N)
    assert S.split_ranges(6, 4) == [(0, 1), (1, 3), (3, 4), (4, 6)]
    assert S.wgrad_plan(2, 8321 - 3 * 2560) == (6, 2)


def _old_grad_rel(got, ref):
    return max(((g - r).norm() / r.norm()).item() for g, r in zip(got["grads"], ref["grads"]))


@pytest.fixture(scope="module")
def draw700():
    W, pts, _ = TF.tie_free_draw(1, 700, 6, 1e-4)
    return W, pts, S.pde_oracle(W, pts)


def test_comparator_accepts_the_reference(draw700):
    W, pts, ref = draw700
    for mode in S.STRICT:
        assert not S.violations(S.strict_errors(ref, ref), mode)


def test_comparator_rejects_a_dropped_point(draw700):
    """Every 50th point in turn: the strict bounds reject each drop; the whole-tensor bound accepts the least visible one."""
    W, pts, ref = draw700
    old = []
    for p in range(0, 700, 50):
        got = dict(ref, grads=S.pde_oracle(W, pts, drop=(0, torch.tensor([p])))["grads"])
        E = S.strict_errors(got, ref)
        old.append(_old_grad_rel(got, ref))
        print("dropped point %d: strict worst slice %.1e %s, whole-tensor %.1e" % (p, E["grad"][0], E["grad"][1], old[-1]))
        for mode in S.STRICT:
            assert any(v[0] == "grad" for v in S.violations(E, mode)), (p, mode)
    assert min(old) < OLD_GRAD, old


def test_comparator_rejects_a_dropped_tile(draw700):
    W, pts, ref = draw700
    got = dict(ref, grads=S.pde_oracle(W, pts, drop=(0, torch.arange(128, 256)))["grads"])
    E = S.strict_errors(got, ref)
    for mode in S.STRICT:
        assert any(v[0] == "grad" for v in S.violations(E, mode)), mode


def test_comparator_rejects_a_slice_off_by_2_pow_minus_11(draw700):
    W, pts, ref = draw700
    grads = [g.clone() for g in ref["grads"]]
    grads[S.NAMES.index("W2")][0, 3] *= 1 + 2.0 ** -11
    got = dict(ref, grads=grads)
    for mode in S.STRICT[:3]:
        assert any(v[0] == "grad" for v in S.violations(S.strict_errors(got, ref), mode)), mode
    assert _old_grad_rel(got, ref) < OLD_GRAD
