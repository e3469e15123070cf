"""Pins oracle/loss.py: (1) every known-answer case of the reference's own unit tests
(/root/reference/test/loss/test_RegressionLossEvaluator.py:7-193, restated — not copied — as
data tables), (2) golden vectors generated from the imported reference (oracle/gen_golden.py),
(3) when the original project's sources are importable, a live comparison against the imported reference (no stored
copy of that case exists)."""
import numpy as np
import pytest
import torch

from oracle import loss as ol
from oracle.gen_golden import SELECTIONS, seeded_out_labels
from oracle.refimport import reference_available

T = lambda x: torch.tensor(x, dtype=torch.float32)


# ---- reference KATs (test file line numbers in comments) ------------------------------------
def test_sqdiff_zero_and_offset():  # :9-21
    a = torch.arange(24, dtype=torch.float32).reshape(2, 4, 3)
    assert torch.equal(ol.squared_diff_mean_vector(a, a.clone()), torch.zeros(3))
    assert torch.allclose(ol.squared_diff_mean_vector(a, a + 1.0), torch.ones(3))


def test_sqdiff_errors():  # :23-35
    with pytest.raises(ValueError):
        ol.squared_diff_mean_vector(T([[[1, 2], [3, 4]]]), T([[[1, 2, 3], [4, 5, 6]]]))
    with pytest.raises(ValueError):
        ol.squared_diff_mean_vector(torch.tensor([]), torch.tensor([]))


def test_mask_by_threes_kats():  # :37-87
    x = T([[[1, 0, 0], [0, 2, 0]], [[0, 0, 0], [3, 0, 4]]])
    assert torch.equal(ol.mask_by_threes(x), T([[[1, 1, 1], [1, 1, 1]], [[0, 0, 0], [1, 1, 1]]]))
    x = T([[[1, 0, 0], [0, 2, 0]]])
    assert torch.equal(ol.mask_by_threes(x, 1.5), T([[[0, 0, 0], [1, 1, 1]]]))
    assert torch.equal(ol.mask_by_threes(T([[[0, 0, 0], [0, 0, 0]]])), T([[[0, 0, 0], [0, 0, 0]]]))
    x = T([[[0, 0, 1, 0, 0, 0], [0, 0, 0, 1, 0, 0]]])
    assert torch.equal(ol.mask_by_threes(x), T([[[1, 1, 1, 0, 0, 0], [0, 0, 0, 1, 1, 1]]]))
    for bad in (T([[1, 0, 0]]), torch.empty(0), T([[[1, 0], [0, 2]]])):
        with pytest.raises(ValueError):
            ol.mask_by_threes(bad)


def test_mean_norm_error_kats():  # :89-159
    with pytest.raises(ValueError):
        ol.mean_norm_error(torch.rand(3, 2, 6), torch.rand(3, 2, 9))
    with pytest.raises(ValueError):
        ol.mean_norm_error(torch.rand(2, 6), torch.rand(2, 6))
    with pytest.raises(ValueError):
        ol.mean_norm_error(torch.rand(0, 6), torch.rand(0, 6))
    with pytest.raises(ValueError):
        ol.mean_norm_error(torch.rand(3, 2, 7), torch.rand(3, 2, 7))
    lab = T([[[1, 2, 3], [4, 5, 6]], [[1, 2, 3], [4, 5, 6]]])
    out = T([[[3, -2, 4], [4, 5, 6]], [[3, -2, 4], [4, 5, 6]]])
    assert torch.isclose(ol.mean_norm_error(out, lab), T(0.0))          # last frame only
    out2 = out.clone(); out2[1, 1, 2] = 7.0
    assert torch.isclose(ol.mean_norm_error(out2, lab), T(0.5))
    v = T([[[1, 2, 3, 4, 5, 6]]])
    assert torch.isclose(ol.mean_norm_error(v, v.clone(), 6), T(0.0))
    assert torch.isclose(ol.mean_norm_error(v, torch.zeros_like(v), 6), torch.norm(T([1, 2, 3, 4, 5, 6])))


def test_com_acc_kats():  # :161-192
    with pytest.raises(ValueError):
        ol.com_acc_error(torch.rand(3, 2, 6), torch.rand(4, 2, 6))
    with pytest.raises(ValueError):
        ol.com_acc_error(torch.rand(2, 6), torch.rand(2, 6))
    with pytest.raises(ValueError):
        ol.com_acc_error(torch.empty(0, 0), torch.rand(3, 6))
    with pytest.raises(ValueError):
        ol.com_acc_error(torch.rand(3, 2, 5), torch.rand(3, 2, 5))
    o = T([[[1, 2, 3, 0, 0, 0], [0, 0, 0, 1, 2, 3]]])
    l = T([[[0, 0, 0, 1, 2, 3], [1, 2, 3, 0, 0, 0]]])
    assert torch.isclose(ol.com_acc_error(o, l), T(0.0))


# ---- golden vectors from the imported reference --------------------------------------------
@pytest.mark.parametrize("case", ["b4f10", "b3f1", "b7f50"])
@pytest.mark.parametrize("sel", list(SELECTIONS))
def test_call_matches_golden(golden, case, sel):
    g = golden("loss_call.npz")
    B, F, seed = (int(v) for v in g[f"{case}/meta"])
    o, l = seeded_out_labels(B, F, seed)
    s = [list(x) for x in SELECTIONS[sel]]
    res = ol.regression_loss(o, l, *s)
    for k in ("loss", "force", "cop", "moment", "wrench", "force_report", "moment_report", "cop_report",
              "wrench_report", "wrench_moment_report", "com_acc_report"):
        np.testing.assert_allclose(np.asarray(res[k], dtype=np.float64), g[f"{case}/{sel}/{k}"], rtol=2e-6, atol=1e-7,
                                   err_msg=k)
    grads = ol.regression_loss_grad(o, l, *s)
    for k, v in grads.items():
        np.testing.assert_allclose(v.numpy(), g[f"{case}/{sel}/grad/{k}"], rtol=2e-6, atol=1e-9, err_msg=k)
    assert np.array_equal(ol.mask_by_threes(l[ol.FORCE], 10.0).numpy(), g[f"{case}/mask10"])   # bit-exact


@pytest.mark.skipif(not reference_available(), reason="needs the original project's sources (IBM_REFERENCE_ROOT or oracle/_ref)")
def test_live_against_reference():
    from oracle.gen_golden import run_ref_loss
    from oracle.refimport import load_reference
    ref = load_reference()
    o, l = seeded_out_labels(5, 10, 777)
    sel = SELECTIONS["repeat"]
    res_ref, grads_ref = run_ref_loss(ref, o, l, sel)
    res = ol.regression_loss(o, l, *[list(x) for x in sel])
    assert abs(float(res["loss"]) - float(res_ref["loss"])) <= 2e-6 * abs(float(res_ref["loss"]))
    g = ol.regression_loss_grad(o, l, *[list(x) for x in sel])
    for k in g:
        torch.testing.assert_close(g[k], grads_ref[k], rtol=2e-6, atol=1e-9)
