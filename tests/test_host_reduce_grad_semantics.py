"""The reference's gradient rules that the backward kernels of the masked reductions and of distance_tensor_redux
follow, pinned on the CPU (float64 autograd of oracle/masked.py, which restates the reference op for op).  A torch
release that changed one of them fails here, not as a GPU mismatch."""
import torch

from oracle import masked as om


def _grad(fn, x):
    x = x.clone().requires_grad_(True)
    fn(x).sum().backward()
    return x.grad


def test_min_over_a_dim_tuple_takes_the_first_tie_in_the_caller_order():
    # the dims are reduced one at a time in the caller's order, each picking its first extreme: the last dim reduced
    # is the most significant
    x = torch.tensor([[1., 0.5, 0.5], [0.5, 2., 3.]], dtype=torch.float64)
    assert _grad(lambda t: om.mmin(t, dim=(0, 1), keepdim=True), x).tolist() == [[0., 0., 0.], [1., 0., 0.]]
    assert _grad(lambda t: om.mmin(t, dim=(1, 0), keepdim=True), x).tolist() == [[0., 1., 0.], [0., 0., 0.]]
    assert _grad(lambda t: om.mmax(-t, dim=(1, 0), keepdim=True), x).tolist() == [[0., -1., 0.], [0., 0., 0.]]


def test_min_over_a_dim_takes_the_first_nan_and_drops_an_excluded_pick():
    x = torch.tensor([[1., float("nan"), 0., float("nan")]], dtype=torch.float64)
    assert _grad(lambda t: om.mmin(t, dim=1), x).tolist() == [[0., 1., 0., 0.]]
    # a fully excluded slice: the first position holds the fill value and takes the gradient, which is dropped
    m = torch.tensor([[True, True, True, True]])
    assert _grad(lambda t: om.mmin(t, mask=m, dim=1), torch.zeros(1, 4, dtype=torch.float64)).tolist() == [[0.] * 4]


def test_min_of_everything_spreads_over_the_ties():
    x = torch.tensor([[1., 0.5, 0.5], [0.5, 2., 3.]], dtype=torch.float64)
    assert _grad(lambda t: om.mmin(t), x).tolist() == [[0., 1 / 3, 1 / 3], [1 / 3, 0., 0.]]
    # an excluded position filled with the extreme counts in the split, and its share is dropped
    m = torch.tensor([[False, False, False], [False, True, False]])
    g = _grad(lambda t: om.mmin(t, mask=m, ctt=0.5), x)
    assert g.tolist() == [[0., 0.25, 0.25], [0.25, 0., 0.]]
    # NaN: the split goes over the NaNs
    y = torch.tensor([float("nan"), 1., float("nan")], dtype=torch.float64)
    assert _grad(lambda t: om.mmax(t), y).tolist() == [0.5, 0., 0.5]


def test_meanmin_weights_every_row_by_its_count():
    d = torch.tensor([[[[3., 1., 1.], [1., 2., 5.], [0.5, 0.5, 9.]]]], dtype=torch.float64)
    m = torch.tensor([[[[False, False, True], [False, False, False], [True, False, False]]]])
    g = _grad(lambda t: om.distance_tensor_redux(t, "meanmin", mask=m), d)[0, 0]
    # row minima at the first argmin (row 2: position 0 is excluded and holds inf, the min is at 1), weights cnt_i / C
    assert g.tolist() == [[0., 2 / 7, 0.], [3 / 7, 0., 0.], [0., 2 / 7, 0.]]


def test_minmean_takes_the_first_minimal_row_and_worst_takes_nothing():
    d = torch.tensor([[[[1., 3.], [2., 2.], [0., 4.]]]], dtype=torch.float64)
    g = _grad(lambda t: om.distance_tensor_redux(t, "minmean"), d)[0, 0]
    assert g.tolist() == [[0.5, 0.5], [0., 0.], [0., 0.]]
    assert _grad(lambda t: om.distance_tensor_redux(t, "worst-2"), d).abs().sum() == 0


def test_symmetric_prefix_averages_the_two_orientations():
    d = torch.tensor([[[[3., 1., 1.], [1., 2., 5.], [0.5, 0.5, 9.]]]], dtype=torch.float64)
    g = _grad(lambda t: om.distance_tensor_redux(t, "smin"), d)[0, 0]
    # row-major first minimum (2, 0) and, on the transpose, column-major first minimum (2, 0) again
    assert g.tolist() == [[0., 0., 0.], [0., 0., 0.], [1., 0., 0.]]
    g = _grad(lambda t: om.distance_tensor_redux(t, "smeanmin"), d)[0, 0]
    assert torch.allclose(g, torch.tensor([[0., 1 / 6, 1 / 6], [1 / 6, 0., 0.], [1 / 3, 1 / 6, 0.]], dtype=torch.float64))


def test_bpwr_picks_every_entry_at_or_below_a_round_minimum():
    d = torch.tensor([[[[3., 1., 1.], [1., 2., 5.], [0.5, 0.5, 9.]]]], dtype=torch.float64)
    g = _grad(lambda t: om.distance_tensor_redux(t, "bpwr", eps=0.0), d)[0, 0]
    assert torch.allclose(g, torch.tensor([[0., 0., 1 / 3], [0., 0., 0.], [1 / 3, 1 / 3, 0.]], dtype=torch.float64))
