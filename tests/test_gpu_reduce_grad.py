"""-m gpu: autograd of the masked reductions and of distance_tensor_redux (wealy_masked_reduce_backward,
wealy_distance_redux_backward) against the CPU float64 autograd of oracle/masked.py on the same values."""
import pytest
import torch

from oracle import masked as om

pytestmark = pytest.mark.gpu

DTYPES = [torch.float32, torch.float64, torch.float16, torch.bfloat16]
TOL = {torch.float64: 1e-12, torch.float32: 2e-6, torch.float16: 2e-3, torch.bfloat16: 1.6e-2}
REDUX = ["min", "max", "mean", "minmean", "meanmin", "best", "best-3", "best-100", "worst-2", "bpwr", "bpwr-2", "smin",
         "smeanmin", "sminmean", "sbest-4", "sbpwr", "bestmin-2"]
SHAPES = [(3, 4, 5, 6), (2, 3, 7, 2), (5, 1, 1, 9), (2, 2, 16, 16), (1, 3, 32, 32)]


def _wt():
    from wealy_b200 import tensor_ops as wt
    return wt


def _upstream(shape, seed):
    return torch.randn(shape, generator=torch.Generator().manual_seed(seed), dtype=torch.float64)


def _grads(prod, orac, x, dtype, seed=0):
    """x.grad of prod(x on the GPU in `dtype`) and of orac(the same values in float64 on the CPU) for one upstream g."""
    xr = x.detach().to(dtype)
    xg = xr.cuda().requires_grad_(True)
    out = prod(xg)
    g = _upstream(out.shape, seed).to(dtype)
    out.backward(g.cuda())
    xo = xr.double().clone().requires_grad_(True)
    ref = orac(xo)
    assert ref.numel() == out.numel(), (ref.shape, out.shape)
    ref.backward(g.double().reshape(ref.shape))
    assert xg.grad.dtype == dtype
    return xg.grad.double().cpu(), xo.grad, xr.double()


def _close(a, b, tol):
    assert a.shape == b.shape
    assert torch.equal(torch.isnan(a), torch.isnan(b))
    fin = ~torch.isnan(a)
    err = (a[fin] - b[fin]).abs().max().item() if fin.any() else 0.0
    assert err <= tol * max(1.0, b[fin].abs().max().item() if fin.any() else 1.0), err


def _close_per_tie_group(a, b, vals, mask, tol):
    """best-k: at a tie on the k-th boundary the choice among equal entries is implementation-defined, so compare the
    gradient summed over every group of equal included entries of a block (excluded entries: 0 on both sides)."""
    B = a.shape[0] * a.shape[1]
    a, b, vals = a.reshape(B, -1), b.reshape(B, -1), vals.reshape(B, -1)
    m = torch.zeros_like(vals, dtype=torch.bool) if mask is None else mask.cpu().reshape(B, -1)
    for r in range(B):
        keys = torch.where(m[r], torch.full_like(vals[r], float("nan")), vals[r])
        assert (a[r][m[r]].abs().max().item() if m[r].any() else 0.0) <= tol
        assert (b[r][m[r]].abs().max().item() if m[r].any() else 0.0) <= tol
        for v in torch.unique(keys[~m[r]]):
            sel = (keys == v) & ~m[r]
            assert abs(a[r][sel].sum().item() - b[r][sel].sum().item()) <= tol * max(1.0, b[r][sel].abs().sum().item()), \
                (r, v.item())


def _redux_mask(shape, g):
    mask = torch.rand(*shape, generator=g) < 0.35
    mask[0, 0, 0, :] = True                                    # a fully excluded row
    mask[-1, -1, :, -1] = True                                 # ... column
    if shape[0] > 1:
        mask[1, 0] = True                                      # ... block
    return mask


# ---------------------------------------------------------------------------------------------------------------------
# masked reductions
# ---------------------------------------------------------------------------------------------------------------------
_DIMS = [(None, False), (None, True), (1, False), (-1, True), (0, False), ((0, 2), True), ((2, 0), True), ((1, 2), True),
         ((2, 1), True), ((2, 1, 0), True), ((0, 1, 2), True)]


def _masked_inputs(kind, g):
    shape = (4, 5, 6)
    if kind == "ties":                                         # a coarse grid: every min / max is tied many times
        x = torch.randint(0, 3, shape, generator=g).double() / 2
    else:
        x = torch.randn(shape, generator=g, dtype=torch.float64)
    if kind == "nan":
        x[1, 2, 3] = x[1, 4, 0] = x[3, 0, 5] = float("nan")
    mask = torch.rand(shape, generator=g) < 0.3
    mask[1] = True                                             # empty slices for every dim choice
    mask[:, 2, :] = True
    mask[2, :, 4] = True
    return x, mask


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("kind", ["random", "ties", "nan"])
@pytest.mark.parametrize("fn", ["msum", "mmean", "mmin", "mmax"])
def test_masked_reduction_gradients(fn, kind, dtype):
    wt = _wt()
    g = torch.Generator().manual_seed(10 * len(fn) + len(kind))
    x, mask = _masked_inputs(kind, g)
    f, o = getattr(wt, fn), getattr(om, fn)
    for seed, (dim, keepdim) in enumerate(_DIMS):
        for m in (None, mask):
            mc = None if m is None else m.cuda()
            try:
                o(x.double(), mask=m, dim=dim, keepdim=keepdim)
            except (IndexError, RuntimeError):
                continue                                       # the oracle (the reference) rejects this call
            a, b, _ = _grads(lambda t: f(t, mask=mc, dim=dim, keepdim=keepdim),
                             lambda t: o(t, mask=m, dim=dim, keepdim=keepdim), x, dtype, seed)
            _close(a, b, TOL[dtype])


def test_min_tie_follows_the_caller_dim_order():
    """mmin(dim=(0, 1)) and mmin(dim=(1, 0)) pick different tied entries, like the reference's dim-by-dim reduction."""
    wt = _wt()
    x = torch.tensor([[1., 0.5, 0.5], [0.5, 2., 3.]], dtype=torch.float64)
    for dim in ((0, 1), (1, 0), (-1, -2), (-2, -1)):
        a, b, _ = _grads(lambda t: wt.mmin(t, dim=dim, keepdim=True), lambda t: om.mmin(t, dim=dim, keepdim=True), x,
                         torch.float64)
        assert torch.equal(a, b), (dim, a, b)
    a01 = _grads(lambda t: wt.mmin(t, dim=(0, 1), keepdim=True), lambda t: om.mmin(t, dim=(0, 1), keepdim=True), x,
                 torch.float64)[0]
    a10 = _grads(lambda t: wt.mmin(t, dim=(1, 0), keepdim=True), lambda t: om.mmin(t, dim=(1, 0), keepdim=True), x,
                 torch.float64)[0]
    assert not torch.equal(a01, a10)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_broadcast_masks_and_inputs(dtype):
    """x and mask broadcast together; dx is summed back to x's shape (this is what weights meanmin's row minima).  A
    mask smaller than x only for sum / min / max: the reference's mmean counts the entries of the mask itself."""
    wt = _wt()
    g = torch.Generator().manual_seed(5)
    x = torch.randn(4, 5, 6, generator=g, dtype=torch.float64)
    for m in (torch.rand(5, 6, generator=g) < 0.4, torch.rand(4, 1, 6, generator=g) < 0.4):
        for fn in ("msum", "mmin", "mmax"):
            for dim in (None, -1, (1, 2)):
                a, b, _ = _grads(lambda t: getattr(wt, fn)(t, mask=m.cuda(), dim=dim, keepdim=True),
                                 lambda t: getattr(om, fn)(t, mask=m, dim=dim, keepdim=True), x, dtype)
                _close(a, b, TOL[dtype])
    xs = torch.randn(4, 5, 1, generator=g, dtype=torch.float64)     # x smaller than the mask
    m = torch.rand(4, 5, 6, generator=g) < 0.4
    for fn in ("msum", "mmean", "mmin", "mmax"):
        for dim in (None, -1, (-1, -2)):
            a, b, _ = _grads(lambda t: getattr(wt, fn)(t, mask=m.cuda(), dim=dim, keepdim=True),
                             lambda t: getattr(om, fn)(t, mask=m, dim=dim, keepdim=True), xs, dtype)
            _close(a, b, TOL[dtype])


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("kind", ["random", "ties"])
def test_long_rows_take_the_block_kernel(kind, dtype):
    """3 x 70 000: fewer than 4096 rows of more than 2048 entries run one block per row (ties spread over the warps)."""
    wt = _wt()
    g = torch.Generator().manual_seed(4)
    x = torch.randn(3, 70000, generator=g, dtype=torch.float64) if kind == "random" else \
        torch.randint(0, 4, (3, 70000), generator=g).double()
    m = torch.rand(3, 70000, generator=g) < 0.5
    for fn in ("msum", "mmean", "mmin", "mmax"):
        for dim in (1, None):
            a, b, _ = _grads(lambda t: getattr(wt, fn)(t, mask=m.cuda(), dim=dim),
                             lambda t: getattr(om, fn)(t, mask=m, dim=dim), x, dtype)
            _close(a, b, TOL[dtype])


@pytest.mark.parametrize("dtype", DTYPES)
def test_composite_masked_reductions(dtype, monkeypatch):
    wt = _wt()
    g = torch.Generator().manual_seed(6)
    x = torch.randn(6, 7, 9, generator=g, dtype=torch.float64)
    mask = torch.rand(6, 7, 9, generator=g) < 0.3
    mask[0, 0] = True
    mc = mask.cuda()
    # mbest / mworst: the topk choice at ties is implementation-defined, compare per group of equal entries
    for k in (1, 3, 9):
        for fn in ("mbest", "mworst"):
            a, b, v = _grads(lambda t: getattr(wt, fn)(t, k, mask=mc, dim=-1),
                             lambda t: getattr(om, fn)(t, k, mask=mask, dim=-1), x, dtype)
            _close_per_tie_group(a.reshape(6, 7, 1, 9), b.reshape(6, 7, 1, 9), v.reshape(6, 7, 1, 9),
                                 mask.reshape(6, 7, 1, 9), TOL[dtype])
    # mrand: feed the oracle the product's random keys
    for dim in (-1, (1, 2)):
        xr = x.to(dtype)
        xg = xr.cuda().requires_grad_(True)
        torch.cuda.manual_seed(11)
        keys = torch.rand_like(xg).double().cpu()
        torch.cuda.manual_seed(11)
        out = wt.mrand(xg, mask=mc, dim=dim, keepdim=True)
        up = _upstream(out.shape, 3).to(dtype)
        out.backward(up.cuda())
        monkeypatch.setattr(om.torch, "rand_like", lambda t: keys.to(t.dtype))
        xo = xr.double().clone().requires_grad_(True)
        om.mrand(xo, mask=mask, dim=dim, keepdim=True).backward(up.double())
        monkeypatch.undo()
        _close(xg.grad.double().cpu(), xo.grad, TOL[dtype])


# ---------------------------------------------------------------------------------------------------------------------
# distance_tensor_redux
# ---------------------------------------------------------------------------------------------------------------------
def _redux_check(dist, redux, mask, dtype, fused, seed=0, oracle_eps=1e-7, prod_eps=1e-7):
    wt = _wt()
    mc = None if mask is None else mask.cuda()
    a, b, v = _grads(lambda t: wt.distance_tensor_redux(t, redux, mask=mc, fused=fused, eps=prod_eps),
                     lambda t: om.distance_tensor_redux(t, redux, mask=mask, eps=oracle_eps), dist, dtype, seed)
    if redux.lstrip("s").startswith("best"):
        _close_per_tie_group(a, b, v, mask, TOL[dtype])
    else:
        _close(a, b, TOL[dtype])


def _jitter_free(redux):
    return "bpwr" not in redux


def _half_mask_overflow(dtype, redux, fused, mask):
    """The composition's best-k / worst-k and randmin (always a composition) fill excluded entries with
    torch.where(mask, 1e12, x), which float16 cannot hold (as in the reference)."""
    composed = redux == "randmin" or (not fused and redux.lstrip("s").startswith(("best", "worst")))
    return dtype == torch.float16 and mask is not None and composed


# the reference's "s" branch calls itself without eps, so sbpwr always jitters by 1e-7 * rand: on tie-heavy blocks the
# oracle's own draw decides, and sbpwr is checked there only through the controlled jitter of test_bpwr_gradients_with_jitter
_TIE_SAFE = [r for r in REDUX if r != "sbpwr"]


@pytest.mark.parametrize("fused", [True, False])
@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("redux", REDUX)
def test_redux_gradients(redux, shape, fused):
    """Every strategy of test_fused_redux_equals_the_composition on its shapes and masks, fp32 and fp64.  bpwr with
    eps = 0 (no jitter; the jittered case is below)."""
    g = torch.Generator().manual_seed(sum(shape) + len(redux))
    dist = torch.rand(*shape, generator=g, dtype=torch.float64) * 2
    mask = _redux_mask(shape, g)
    eps = 1e-7 if _jitter_free(redux) else 0.0
    for dtype in (torch.float32, torch.float64):
        for m in (None, mask):
            if not _jitter_free(redux) and m is not None:
                m = m.clone()
                m[..., 0, 0] = False                           # eps = 0: no empty block (the reference divides 0 / 0)
            _redux_check(dist, redux, m, dtype, fused, oracle_eps=eps, prod_eps=eps)


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("redux", _TIE_SAFE)
def test_redux_gradients_half(redux, dtype):
    """fp16 / bf16 on a grid of exactly representable values.  The composition rounds its intermediate row means to
    the half dtype, which can make near-equal rows tie where the float64 oracle does not: minmean there is checked
    through the fused path only."""
    g = torch.Generator().manual_seed(len(redux))
    eps = 1e-7 if _jitter_free(redux) else 0.0
    for shape in SHAPES:
        dist = torch.randint(0, 64, shape, generator=g).double() / 16
        mask = _redux_mask(shape, g)
        if not _jitter_free(redux):
            mask[..., 0, 0] = False
        for fused in (True, False):
            if not fused and "minmean" in redux:
                continue
            for m in (None, mask):
                if _half_mask_overflow(dtype, redux, fused, m):
                    continue
                _redux_check(dist, redux, m, dtype, fused, oracle_eps=eps, prod_eps=eps)


@pytest.mark.parametrize("fused", [True, False])
@pytest.mark.parametrize("redux", _TIE_SAFE)
def test_redux_gradients_on_ties(redux, fused):
    """Tie-heavy blocks (values on a coarse grid): first extreme, first minimal row, first argmin per row, every bpwr
    entry <= a round's minimum, best-k compared per tie group."""
    g = torch.Generator().manual_seed(7 + len(redux))
    eps = 1e-7 if _jitter_free(redux) else 0.0
    for shape in SHAPES:
        dist = torch.randint(0, 3, shape, generator=g).double() / 2
        mask = _redux_mask(shape, g)
        if not _jitter_free(redux):
            mask[..., 0, 0] = False
        for dtype in (torch.float32, torch.float64):
            for m in (None, mask):
                _redux_check(dist, redux, m, dtype, fused, oracle_eps=eps, prod_eps=eps)


@pytest.mark.parametrize("fused", [True, False])
def test_redux_gradients_with_nan(fused):
    g = torch.Generator().manual_seed(8)
    dist = torch.rand(3, 4, 5, 6, generator=g, dtype=torch.float64)
    dist[0, 1, 2, 3] = dist[0, 1, 4, 0] = dist[2, 2, 0, 5] = float("nan")
    for redux in ("min", "max", "smin", "smax", "meanmin", "minmean", "mean"):
        for dtype in (torch.float32, torch.float64):
            _redux_check(dist, redux, None, dtype, fused)


@pytest.mark.parametrize("fused", [True, False])
@pytest.mark.parametrize("redux", ["min", "max", "mean", "minmean", "meanmin", "best", "best-3", "worst", "worst-2",
                                   "bestmin", "bestmin-2", "smin", "smeanmin", "sbest-4"])
def test_redux_gradients_on_golden_inputs(golden, redux, fused):
    G = golden("redux.npz")
    dist, mask = torch.from_numpy(G["dist"]).double(), torch.from_numpy(G["mask"])
    for dtype in (torch.float32, torch.float64):
        for m in (None, mask):
            _redux_check(dist, redux, m, dtype, fused)


@pytest.mark.parametrize("fused", [True, False])
@pytest.mark.parametrize("redux", ["bpwr", "bpwr-2", "sbpwr"])
@pytest.mark.parametrize("shape", [(3, 4, 5, 6), (2, 3, 7, 2), (2, 2, 16, 16)])
def test_bpwr_gradients_with_jitter(redux, shape, fused):
    """The product draws eps * rand_like(dist) from the CUDA generator; the same draw is made here and the oracle is fed
    the jittered tensor with eps = 0 (the jitter's gradient is the identity)."""
    if redux == "sbpwr" and not fused:
        pytest.skip("the composition draws a second jitter for the transposed block")
    wt = _wt()
    eps = 1e-3
    g = torch.Generator().manual_seed(sum(shape))
    dist = torch.randint(0, 4, shape, generator=g).double() / 4          # ties that the jitter breaks
    mask = torch.rand(*shape, generator=g) < 0.3
    mask[..., 0, 0] = False                                              # no empty block (the oracle runs with eps = 0)
    for dtype in (torch.float32, torch.float64):
        for m in (None, mask):
            mc = None if m is None else m.cuda()
            xg = dist.to(dtype).cuda().requires_grad_(True)
            torch.cuda.manual_seed(21)
            if not fused and shape[3] < shape[2]:                        # the composition transposes before drawing
                jit = (eps * torch.rand_like(xg.detach().transpose(2, 3))).transpose(2, 3)
            else:
                jit = eps * torch.rand_like(xg.detach())
            jittered = (xg.detach() + jit).double().cpu()
            torch.cuda.manual_seed(21)
            out = wt.distance_tensor_redux(xg, redux, mask=mc, eps=eps, fused=fused)
            up = _upstream(out.shape, 2).to(dtype)
            out.backward(up.cuda())
            xo = jittered.requires_grad_(True)
            om.distance_tensor_redux(xo, redux, mask=m, eps=0.0).backward(up.double())
            _close(xg.grad.double().cpu(), xo.grad, TOL[dtype])


@pytest.mark.parametrize("redux", REDUX)
def test_gradcheck_fused(redux):
    """torch.autograd.gradcheck on the fused path in float64, tie-free inputs (gaps far above the finite-difference
    step), with and without a mask."""
    wt = _wt()
    g = torch.Generator().manual_seed(len(redux))
    b1, b2, s1, s2 = 2, 2, 3, 4
    # distinct entries at least 1/32 apart, and no exact ties between row / column means either
    vals = (torch.randperm(b1 * b2 * s1 * s2, generator=g).double() + torch.rand(b1 * b2 * s1 * s2, generator=g,
                                                                                 dtype=torch.float64) / 2)
    vals = vals.reshape(b1, b2, s1, s2) / 16
    mask = torch.rand(b1, b2, s1, s2, generator=g) < 0.3
    mask[..., 0, 0] = False
    eps = 1e-7 if _jitter_free(redux) else 0.0
    for m in (None, mask.cuda()):
        d = vals.cuda().requires_grad_(True)
        assert torch.autograd.gradcheck(lambda t: wt.distance_tensor_redux(t, redux, mask=m, eps=eps), (d,))


# ---------------------------------------------------------------------------------------------------------------------
# the forward does not move, and costs nothing new without grad
# ---------------------------------------------------------------------------------------------------------------------
def _same(a, b):
    torch.testing.assert_close(a, b, rtol=0, atol=0, equal_nan=True)


@pytest.mark.parametrize("dtype", DTYPES)
def test_forward_is_bit_identical_with_grad(dtype):
    wt = _wt()
    g = torch.Generator().manual_seed(9)
    for shape in SHAPES:
        dist = (torch.rand(*shape, generator=g) * 2).to(dtype).cuda()
        dist[0, 0, 0, 0] = float("nan")
        mask = _redux_mask(shape, g).cuda()
        for redux in REDUX + ["randmin", "worst"]:
            for fused in (True, False):
                if _half_mask_overflow(dtype, redux, fused, mask):
                    continue
                torch.cuda.manual_seed(5)
                a = wt.distance_tensor_redux(dist, redux, mask=mask, fused=fused)
                torch.cuda.manual_seed(5)
                b = wt.distance_tensor_redux(dist.clone().requires_grad_(True), redux, mask=mask, fused=fused)
                assert b.grad_fn is not None
                _same(a, b.detach())
    x, mask = _masked_inputs("nan", g)
    x, mask = x.to(dtype).cuda(), mask.cuda()
    for fn in ("msum", "mmean", "mmin", "mmax"):
        for dim, keepdim in _DIMS:
            a = getattr(wt, fn)(x, mask=mask, dim=dim, keepdim=keepdim)
            b = getattr(wt, fn)(x.clone().requires_grad_(True), mask=mask, dim=dim, keepdim=keepdim)
            _same(a, b.detach())


def test_no_graph_without_grad():
    wt = _wt()
    x = torch.rand(2, 3, 4, 5, device="cuda")
    xr = x.clone().requires_grad_(True)
    for redux in ("min", "meanmin", "best-2", "bpwr", "smin", "randmin"):
        assert wt.distance_tensor_redux(x, redux).grad_fn is None
        with torch.no_grad():
            assert wt.distance_tensor_redux(xr, redux).grad_fn is None
            assert wt.distance_tensor_redux(xr, redux, fused=False).grad_fn is None
    for fn in ("msum", "mmean", "mmin", "mmax"):
        assert getattr(wt, fn)(x, dim=-1).grad_fn is None
        with torch.no_grad():
            assert getattr(wt, fn)(xr, dim=(1, 2)).grad_fn is None
    assert "ReduxFused" in type(wt.distance_tensor_redux(xr, "min", squeeze=False).grad_fn.next_functions[0][0]).__name__


def test_reduce_grad_is_a_loss_term():
    """The failure the reference user would hit: a loss made only of these functions trains."""
    wt = _wt()
    d = torch.rand(4, 4, 3, 5, device="cuda", requires_grad=True)
    loss = wt.distance_tensor_redux(d, "best-2").mean() + wt.mmin(d, dim=-1).sum()
    loss.backward()
    assert d.grad is not None and d.grad.abs().sum() > 0
