"""CPU: the rule of the lifting's backward (oracle/lift_grad_ref.lift_grad_ref, what pn2_lift_views_grad implements) is
the gradient torch autograd computes through the reference's composition -- Projection.apply per (scene, view), then
F.max_pool1d over the views or the first-view fill loop -- in float64, on inputs built to hit every tie."""
import numpy as np
import pytest
import torch

from oracle import lift_grad_ref as lgr


@pytest.mark.parametrize("seed,V", [(1, 3), (2, 4), (3, 2), (4, 5)])
def test_tie_inputs_hit_every_case(seed, V):
    feats, pix, _ = lgr.tie_inputs(seed, V=V)
    cases = lgr.tie_cases(feats, pix)
    for name, count in cases.items():
        assert count > 0, (name, cases)


@pytest.mark.parametrize("reduce", ["max", "first"])
@pytest.mark.parametrize("seed,V", [(1, 3), (2, 4), (3, 2), (4, 5)])
def test_rule_equals_autograd_of_the_reference_composition(reduce, seed, V):
    feats, pix, grad_out = lgr.tie_inputs(seed, V=V)
    want = lgr.composition_grad(feats, pix, grad_out, reduce)
    got = lgr.lift_grad_ref(feats, pix, grad_out, reduce)
    assert got.shape == feats.shape
    torch.testing.assert_close(got, want, rtol=0, atol=0)
    assert want.abs().sum() > 0


@pytest.mark.parametrize("reduce", ["max", "first"])
def test_rule_with_one_view_and_with_random_values(reduce):
    """V = 1 (the reduction is the identity: every seen point passes its gradient on, zero columns included) and
    continuous values (no ties), dyadic grad_out."""
    rng = np.random.default_rng(9)
    for V, cont in ((1, False), (1, True), (3, True)):
        feats, pix, grad_out = lgr.tie_inputs(20 + V, V=V, N=64)
        if cont:
            feats = rng.standard_normal(feats.shape).astype(np.float32)
        want = lgr.composition_grad(feats, pix, grad_out, reduce)
        torch.testing.assert_close(lgr.lift_grad_ref(feats, pix, grad_out, reduce), want, rtol=0, atol=0)


def test_points_nobody_sees_get_no_gradient():
    feats, pix, grad_out = lgr.tie_inputs(5)
    pix[:] = -1
    for reduce in ("max", "first"):
        assert lgr.lift_grad_ref(feats, pix, grad_out, reduce).abs().sum() == 0
        assert lgr.composition_grad(feats, pix, grad_out, reduce).abs().sum() == 0
