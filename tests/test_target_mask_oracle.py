"""CPU checks of the partially labelled DEER loss reference (tests/target_mask_oracle.py): an all-ones mask is the
reference multitask loss, a mask that drops whole rows is the reference on the remaining rows, target values at
unlabelled entries do not matter and get an exactly-zero gradient, and dimensions without labels contribute 0."""
import math

import pytest
import torch

import target_mask_oracle as TMO
from oracle import deer_oracle as O

DIMS = ("valence", "arousal", "dominance")


def inputs(B, seed, D=3):
    g = torch.Generator().manual_seed(seed)
    e = torch.randn(B, D, 4, generator=g, dtype=torch.float64) * 2.0
    e[:, :, 2] = e[:, :, 2].clamp(min=-5.0)
    y = torch.tanh(torch.randn(B, D, generator=g, dtype=torch.float64))
    return e, y


def reference(e, y):
    pred = {}
    for i, d in enumerate(DIMS):
        for k, v in O.nig_from_evidence(e[:, i:i + 1, :]).items():
            pred[f"{d}_{k}"] = v
    return O.multitask_deer_loss(pred, y)


def test_all_ones_mask_is_the_reference():
    e, y = inputs(200, 1)
    got = TMO.masked_loss_from_evidence(e, y, torch.ones_like(y, dtype=torch.bool))
    ref = reference(e, y)
    assert math.isclose(float(got["total_loss"]), float(ref["total_loss"]), rel_tol=1e-12)
    assert math.isclose(float(got["cross_dim_loss"]), float(ref["cross_dim_loss"]), rel_tol=1e-12)
    for i, d in enumerate(DIMS):
        for k in TMO.TERMS:
            assert math.isclose(float(got[f"d{i}_{k}"]), float(ref[f"{d}_{k}"]), rel_tol=1e-12, abs_tol=1e-15), (d, k)


def test_dropping_whole_rows_is_the_reference_on_the_rest():
    e, y = inputs(300, 2)
    keep = torch.rand(300, generator=torch.Generator().manual_seed(3)) < 0.6
    mask = keep[:, None].expand(-1, 3).clone()
    got = TMO.masked_loss_from_evidence(e, y, mask)
    ref = reference(e[keep], y[keep])
    assert math.isclose(float(got["total_loss"]), float(ref["total_loss"]), rel_tol=1e-12)
    for i, d in enumerate(DIMS):
        assert got[f"d{i}_num_labeled"] == int(keep.sum())
        for k in TMO.TERMS:
            assert math.isclose(float(got[f"d{i}_{k}"]), float(ref[f"{d}_{k}"]), rel_tol=1e-12, abs_tol=1e-15), (d, k)


def test_unlabelled_targets_do_not_matter_and_get_zero_gradient():
    e, y = inputs(257, 4)
    mask = torch.rand(257, 3, generator=torch.Generator().manual_seed(5)) > 0.3
    y_bad = y.clone()
    junk = torch.tensor([float("nan"), float("inf"), -float("inf"), 1e30], dtype=torch.float64)
    y_bad[~mask] = junk[torch.arange(int((~mask).sum())) % 4]
    res = []
    for yy in (y, y_bad):
        ed = e.clone().requires_grad_(True)
        out = TMO.masked_loss_from_evidence(ed, yy, mask)
        out["total_loss"].backward()
        res.append((out["vector"].detach(), ed.grad))
    (v0, g0), (v1, g1) = res
    assert torch.isfinite(v1).all() and torch.isfinite(g1).all()
    assert torch.equal(v0, v1) and torch.equal(g0, g1)
    assert torch.equal(g1[~mask], torch.zeros_like(g1[~mask]))
    assert float(g1[mask].abs().max()) > 0


def test_missing_dimension_and_empty_mask():
    e, y = inputs(100, 6)
    mask = torch.ones(100, 3, dtype=torch.bool)
    mask[:, 1] = False
    out = TMO.masked_loss_from_evidence(e, y, mask)
    for k in TMO.TERMS:
        assert float(out[f"d1_{k}"]) == 0.0
    # two dimensions remain: one pair
    u = [(O.nig_from_evidence(e[:, i])["beta"] / (O.nig_from_evidence(e[:, i])["alpha"] - 1 + 1e-8)).mean()
         for i in (0, 2)]
    assert math.isclose(float(out["cross_dim_loss"]), float((u[0] - u[1]) ** 2), rel_tol=1e-12)
    want = (out["d0_total_loss"] + out["d2_total_loss"] + 0.05 * out["cross_dim_loss"]) / 3
    assert math.isclose(float(out["total_loss"]), float(want), rel_tol=1e-12)
    # only one labelled dimension: no pair, no cross-dimension term
    one = torch.zeros(100, 3, dtype=torch.bool)
    one[:, 2] = True
    assert float(TMO.masked_loss_from_evidence(e, y, one)["cross_dim_loss"]) == 0.0
    ed = e.clone().requires_grad_(True)
    empty = TMO.masked_loss_from_evidence(ed, y, torch.zeros(100, 3, dtype=torch.bool))
    assert torch.equal(empty["vector"], torch.zeros(17, dtype=torch.float64))
    assert float(empty["total_loss"]) == 0.0
    assert not empty["total_loss"].requires_grad      # nothing labelled: the loss does not depend on the evidence


@pytest.mark.parametrize("D", [1, 2])
def test_single_dimension_is_the_deer_loss_on_labelled_rows(D):
    e, y = inputs(150, 7 + D, D)
    mask = torch.rand(150, D, generator=torch.Generator().manual_seed(D)) > 0.4
    out = TMO.masked_loss_from_evidence(e, y, mask, cross_dim_weight=0.0)
    p = O.nig_from_evidence(e)
    want = 0.0
    for d in range(D):
        m = mask[:, d]
        r = O.deer_loss(*(t[:, d][m].unsqueeze(-1) for t in (p["mu"], p["nu"], p["alpha"], p["beta"], y)))
        assert math.isclose(float(out[f"d{d}_total_loss"]), float(r["total_loss"]), rel_tol=1e-12)
        want += float(r["total_loss"])
    assert math.isclose(float(out["total_loss"]), want / D, rel_tol=1e-12)
