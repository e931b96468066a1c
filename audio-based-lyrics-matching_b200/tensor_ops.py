"""Drop-in for the hot functions of /root/reference/lib/tensor_ops.py, computed on sm_100a.

  pairwise_distance_matrix(x, y, mode="fro", p=2, eps=1e-6)        lib/tensor_ops.py:152-176
  pairwise_euclidean_distance_matrix(x, y, squared=False, eps=1e-6) lib/tensor_ops.py:131-149

Same names, argument meaning, return shape / dtype and error behaviour as the reference
(AssertionError for rank violations, NotImplementedError for unknown modes).  The contraction runs
in the tcgen05 kernel behind wealy_sim_matrix (include/wealy_b200.h); `precision` selects the
tensor-core mode ("fp16x3": fp32-grade hi/lo split, the default; "fp16": one pass, ~1e-4 abs error).
float64 inputs return float64 like the reference: they take a CUDA-core double-precision kernel
(wealy_sim_matrix_f64), gradients included.  Every mode is differentiable (the reference's are: plain
torch ops): cos / cossim / dot / dotsim and the euclidean family (sqeuc / nsqeuc / fro / nfro / euc / neuc
with p = 2, pairwise_euclidean_distance_matrix) run their two gradient products on the same contraction
core.  cdist with p != 2 is not a contraction and raises NotImplementedError (WEALY_ERR_UNSUPPORTED).

  msum / mmean / mmin / mmax / mrand / mbest / mworst                lib/tensor_ops.py:182-282
  distance_tensor_redux(dist, redux, mask=None, ...)                lib/tensor_ops.py:288-373

are differentiable too, with the gradient the reference's autograd gives (first order, with respect to x / dist, not
the mask): every result is a sum of w_e * x_e with weights fixed by a discrete selection, and the backward kernels
(wealy_masked_reduce_backward, wealy_distance_redux_backward) rerun that selection with the reference's tie rules --
first extreme for min / max over given dims (the last dim reduced is the most significant), an even split over the
ties for dim=None, the fused redux's own choice at best-k boundary ties.  Without grad they launch only the forward.
Inputs must be CUDA tensors -- there is no CPU fallback.
"""
import ctypes
import os

import torch
from torch.autograd.function import once_differentiable

from . import _native as N

_PRECISIONS = {"fp16x3": 3, "fp16": 1}
_default_precision = os.environ.get("WEALY_PRECISION", "fp16x3")


def set_default_precision(name):
    global _default_precision
    if name not in _PRECISIONS:
        raise ValueError(f"precision must be one of {sorted(_PRECISIONS)}")
    _default_precision = name


def passes_of(precision=None):
    name = _default_precision if precision is None else precision
    if name not in _PRECISIONS:
        raise ValueError(f"precision must be one of {sorted(_PRECISIONS)}")
    return _PRECISIONS[name]


def _rows(t):
    """2-D view with unit inner stride (the C ABI takes a row stride, not arbitrary strides)."""
    if t.stride(-1) != 1 and t.shape[-1] != 1:
        t = t.contiguous()
    if t.shape[-1] == 1 and t.stride(0) < 1:
        t = t.contiguous()
    return t


def _sim_matrix_f64(x, y, mode, eps, post):
    """float64 operands: CUDA-core DGEMM with the mode epilogue (wealy_sim_matrix_f64)."""
    n, d = x.shape
    m = y.shape[0]
    out = torch.empty((n, m), dtype=torch.float64, device=x.device)
    if n == 0 or m == 0:
        return out
    if d == 0:
        raise NotImplementedError("wealy_b200: zero-width embeddings")
    same = x is y
    x = _rows(x)
    y = x if same else _rows(y)
    with torch.cuda.device(x.device):
        ws_bytes = N.lib.wealy_sim_matrix_f64_workspace_bytes(n, m)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x.device)
        N.check(N.lib.wealy_sim_matrix_f64(x.data_ptr(), n, x.stride(0), y.data_ptr(), m, y.stride(0), d, mode, float(eps),
                                           float(post), out.data_ptr(), out.stride(0), ws.data_ptr(), ws_bytes,
                                           N.stream_ptr(x.device)))
    return out


def _sim_matrix(x, y, mode, eps, post, precision):
    N.require_cuda(x, y)
    if x.dtype != y.dtype:
        raise RuntimeError(f"expected x and y to have the same dtype, got {x.dtype} and {y.dtype}")
    if x.shape[1] != y.shape[1]:
        raise RuntimeError(f"size mismatch: x is {tuple(x.shape)}, y is {tuple(y.shape)}")
    if x.dtype == torch.float64:
        return _sim_matrix_f64(x, y, mode, eps, post)
    code = N.dtype_code(x.dtype)
    n, d = x.shape
    m = y.shape[0]
    out = torch.empty((n, m), dtype=x.dtype, device=x.device)
    if n == 0 or m == 0:
        return out
    if d == 0:
        raise NotImplementedError("wealy_b200: zero-width embeddings")
    same = x is y
    x = _rows(x)
    y = x if same else _rows(y)
    passes = passes_of(precision)
    with torch.cuda.device(x.device):
        ws_bytes = N.lib.wealy_sim_matrix_workspace_bytes(n, m, d, passes)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x.device)
        N.check(N.lib.wealy_sim_matrix(
            x.data_ptr(), n, x.stride(0), y.data_ptr(), m, y.stride(0), d, code, mode, float(eps), float(post),
            passes, out.data_ptr(), out.stride(0), code, ws.data_ptr(), ws_bytes, N.stream_ptr(x.device)))
    return out


class _CosineMatrix(torch.autograd.Function):
    """cos / cossim modes under autograd (the reference differentiates through them, lib/losses.py:45):
    dX^ = G Y^ and dY^ = G^T X^ on the same tcgen05 core, then the Jacobian of x / (|x| + eps)."""

    @staticmethod
    def forward(ctx, x, y, mode, eps, precision):
        ctx.save_for_backward(x, y)
        ctx.cfg = (mode, eps, precision)
        return _sim_matrix(x.detach(), y.detach(), mode, eps, 1.0, precision)

    @staticmethod
    def backward(ctx, g):
        x, y = ctx.saved_tensors
        mode, eps, precision = ctx.cfg
        xx, yy = _rows(x.detach()), _rows(y.detach())
        n, d = xx.shape
        m = yy.shape[0]
        gg = g.to(xx.dtype).contiguous()
        gt = gg.t().contiguous()
        dx = torch.empty((n, d), dtype=xx.dtype, device=xx.device)
        dy = torch.empty((m, d), dtype=xx.dtype, device=xx.device)
        passes = passes_of(precision)
        with torch.cuda.device(xx.device):
            ws_bytes = N.lib.wealy_sim_matrix_backward_workspace_bytes(n, m, d, passes)
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=xx.device)
            N.check(N.lib.wealy_sim_matrix_backward(
                xx.data_ptr(), n, xx.stride(0), yy.data_ptr(), m, yy.stride(0), d, N.dtype_code(xx.dtype), mode,
                float(eps), passes, gg.data_ptr(), gg.stride(0), gt.data_ptr(), gt.stride(0), dx.data_ptr(),
                dx.stride(0), dy.data_ptr(), dy.stride(0), ws.data_ptr(), ws_bytes, N.stream_ptr(xx.device)))
        return (dx if ctx.needs_input_grad[0] else None), (dy if ctx.needs_input_grad[1] else None), None, None, None


class _DotMatrix(torch.autograd.Function):
    """dot / dotsim modes under autograd: dX = G Y, dY = G^T X on the contraction core (no normalisation)."""

    @staticmethod
    def forward(ctx, x, y, mode, eps, precision):
        ctx.save_for_backward(x, y)
        ctx.cfg = (mode, precision)
        return _sim_matrix(x.detach(), y.detach(), mode, eps, 1.0, precision)

    @staticmethod
    def backward(ctx, g):
        x, y = ctx.saved_tensors
        mode, precision = ctx.cfg
        n, d = x.shape
        m = y.shape[0]
        gg = g.to(x.dtype)
        if mode == N.MODE_DOT:                      # out = 1 - x.y
            gg = -gg
        gg = gg.contiguous()
        gt = gg.t().contiguous()
        xt, yt = x.detach().t().contiguous(), y.detach().t().contiguous()
        dx = torch.empty((n, d), dtype=x.dtype, device=x.device)
        dy = torch.empty((m, d), dtype=x.dtype, device=x.device)
        passes = passes_of(precision)
        with torch.cuda.device(x.device):
            ws_bytes = N.lib.wealy_dot_matrix_backward_workspace_bytes(n, m, d, passes)
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x.device)
            N.check(N.lib.wealy_dot_matrix_backward(
                gg.data_ptr(), gg.stride(0), gt.data_ptr(), gt.stride(0), xt.data_ptr(), xt.stride(0), yt.data_ptr(),
                yt.stride(0), n, m, d, N.dtype_code(x.dtype), passes, dx.data_ptr(), dx.stride(0), dy.data_ptr(),
                dy.stride(0), ws.data_ptr(), ws_bytes, N.stream_ptr(x.device)))
        return (dx if ctx.needs_input_grad[0] else None), (dy if ctx.needs_input_grad[1] else None), None, None, None


def _grad_products(h, x, y, precision):
    """(h @ y, h.T @ x) for an upstream-gradient-like matrix h [n, m] on the contraction core (the float64 kernel for
    doubles): the two products every mode's backward is made of."""
    if x.dtype == torch.float64:
        h = h.contiguous()
        return (_sim_matrix_f64(h, y.t().contiguous(), N.MODE_DOTSIM, 0.0, 1.0),
                _sim_matrix_f64(h.t().contiguous(), x.t().contiguous(), N.MODE_DOTSIM, 0.0, 1.0))
    n, d = x.shape
    m = y.shape[0]
    hh = h.to(x.dtype).contiguous()
    ht = hh.t().contiguous()
    xt, yt = x.t().contiguous(), y.t().contiguous()
    hy = torch.empty((n, d), dtype=x.dtype, device=x.device)
    htx = torch.empty((m, d), dtype=x.dtype, device=x.device)
    passes = passes_of(precision)
    with torch.cuda.device(x.device):
        ws_bytes = N.lib.wealy_dot_matrix_backward_workspace_bytes(n, m, d, passes)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x.device)
        N.check(N.lib.wealy_dot_matrix_backward(
            hh.data_ptr(), hh.stride(0), ht.data_ptr(), ht.stride(0), xt.data_ptr(), xt.stride(0), yt.data_ptr(),
            yt.stride(0), n, m, d, N.dtype_code(x.dtype), passes, hy.data_ptr(), hy.stride(0), htx.data_ptr(),
            htx.stride(0), ws.data_ptr(), ws_bytes, N.stream_ptr(x.device)))
    return hy, htx


class _EucMatrix(torch.autograd.Function):
    """Euclidean family under autograd (lib/tensor_ops.py:131-149 and the p = 2 cdist modes, :159-166):
    out = post * D2 (squared) or post * sqrt(D2), D2 = max(|x|^2 - 2 x.y + |y|^2, 0).  With H = dL/dD2 -- zero where the
    distance is zero, like the reference's clamp + masked safe sqrt and like cdist's backward --
        dx = 2 (rowsum(H) x - H y),   dy = 2 (colsum(H) y - H^T x):  the two products run on the contraction core."""

    @staticmethod
    def forward(ctx, x, y, mode, post, precision):
        out = _sim_matrix(x.detach(), y.detach(), mode, 0.0, post, precision)
        ctx.save_for_backward(x, y, out)
        ctx.cfg = (mode, post, precision)
        return out

    @staticmethod
    def backward(ctx, g):
        x, y, out = ctx.saved_tensors
        mode, post, precision = ctx.cfg
        acc = torch.float64 if x.dtype == torch.float64 else torch.float32
        g, o = g.to(acc), out.to(acc)
        xd, yd = x.detach(), y.detach()
        # a distance inside the forward's rounding noise of zero (|x|^2 - 2 x.y + |y|^2 cancels to ~1e-6 of the norms on
        # the fp32-grade path) is a zero distance: no gradient, as for the exact zeros the reference masks out
        noise = (1e-13 if acc == torch.float64 else 1e-6) * \
            ((xd.to(acc) ** 2).sum(dim=1, keepdim=True) + (yd.to(acc) ** 2).sum(dim=1)[None, :])
        d2 = o / post if mode == N.MODE_SQEUC else (o / post) ** 2
        pos = d2 > noise
        if mode == N.MODE_SQEUC:
            h = torch.where(pos, g * post, torch.zeros_like(g))
        else:
            h = torch.where(pos, g * (post * post * 0.5) / torch.where(pos, o, torch.ones_like(o)), torch.zeros_like(g))
        hy, htx = _grad_products(h, xd, yd, precision)
        dx = 2.0 * (h.sum(dim=1, keepdim=True) * xd.to(acc) - hy.to(acc))
        dy = 2.0 * (h.sum(dim=0)[:, None] * yd.to(acc) - htx.to(acc))
        return (dx.to(x.dtype) if ctx.needs_input_grad[0] else None), (dy.to(y.dtype) if ctx.needs_input_grad[1] else None), \
            None, None, None


class _F64Matrix(torch.autograd.Function):
    """cos / cossim / dot / dotsim on float64 operands under autograd: same closed forms as _CosineMatrix / _DotMatrix,
    products on the float64 kernel, the normalisation Jacobian of x / (|x| + eps) as elementwise torch ops."""

    @staticmethod
    def forward(ctx, x, y, mode, eps):
        ctx.save_for_backward(x, y)
        ctx.cfg = (mode, eps)
        return _sim_matrix_f64(x.detach(), y.detach(), mode, eps, 1.0)

    @staticmethod
    def backward(ctx, g):
        x, y = (t.detach() for t in ctx.saved_tensors)
        mode, eps = ctx.cfg
        if mode in (N.MODE_COS, N.MODE_DOT):                       # out = 1 - s
            g = -g
        if mode in (N.MODE_DOTSIM, N.MODE_DOT):
            dx, dy = _grad_products(g, x, y, None)
            return (dx if ctx.needs_input_grad[0] else None), (dy if ctx.needs_input_grad[1] else None), None, None
        rx, ry = x.norm(dim=1, keepdim=True), y.norm(dim=1, keepdim=True)
        xh, yh = x / (rx + eps), y / (ry + eps)
        dxh, dyh = _grad_products(g, xh, yh, None)

        def jac(v, r, dvh):                                        # d/dv of v / (|v| + eps), zero radial term at v = 0
            radial = (v * dvh).sum(dim=1, keepdim=True) / (torch.where(r > 0, r, torch.ones_like(r)) * (r + eps) ** 2)
            return dvh / (r + eps) - torch.where(r > 0, radial, torch.zeros_like(radial)) * v
        return (jac(x, rx, dxh) if ctx.needs_input_grad[0] else None), (jac(y, ry, dyh) if ctx.needs_input_grad[1] else None), \
            None, None


def pairwise_euclidean_distance_matrix(x, y, squared=False, eps=1e-6, precision=None):
    """lib/tensor_ops.py:131-149: |x|^2 - 2 x.y + |y|^2, clamped at 0, optional sqrt (zeros stay 0).
    `eps` only guards the reference's autograd through sqrt(0); neither the forward value nor the gradient (zero at
    zero distance) depends on it."""
    mode = N.MODE_SQEUC if squared else N.MODE_EUC
    if (x.requires_grad or y.requires_grad) and torch.is_grad_enabled() and x.shape[0] > 0 and y.shape[0] > 0:
        return _EucMatrix.apply(x, y, mode, 1.0, precision)
    return _sim_matrix(x, y, mode, 0.0, 1.0, precision)


def pairwise_distance_matrix(x, y, mode="fro", p=2, eps=1e-6, precision=None):
    """lib/tensor_ops.py:152-176.  Returns an (n, m) tensor with x's dtype; differentiable in every mode."""
    assert x.ndim == y.ndim and x.ndim <= 2
    if x.ndim == 1:  # :154-156 -- 1-D inputs are n x 1 column vectors
        x = x.unsqueeze(-1)
        y = y.unsqueeze(-1)
    if x.ndim == 0:
        raise NotImplementedError("wealy_b200: 0-d inputs")
    grad = (x.requires_grad or y.requires_grad) and torch.is_grad_enabled() and \
        x.shape[0] > 0 and y.shape[0] > 0 and x.shape[1] > 0
    if mode == "euc" or mode == "neuc":
        p = 2
    d = x.size(-1)
    if mode in ("fro", "nfro", "euc", "neuc"):
        if p != 2:
            raise NotImplementedError("wealy_b200: cdist modes are built for p=2 only (p-norms with p != 2 are "
                                      "not a contraction; out of the hot path)")
        post = 1.0 if mode in ("fro", "euc") else 1.0 / (d ** (1 / p))
        if grad:
            return _EucMatrix.apply(x, y, N.MODE_EUC, post, precision)
        return _sim_matrix(x, y, N.MODE_EUC, 0.0, post, precision)
    if mode in ("sqeuc", "nsqeuc"):
        post = 1.0 if mode == "sqeuc" else 1.0 / d
        if grad:
            return _EucMatrix.apply(x, y, N.MODE_SQEUC, post, precision)
        return _sim_matrix(x, y, N.MODE_SQEUC, 0.0, post, precision)
    if mode in ("cos", "cossim", "dot", "dotsim"):
        code = {"cossim": N.MODE_COSSIM, "cos": N.MODE_COS, "dotsim": N.MODE_DOTSIM, "dot": N.MODE_DOT}[mode]
        if grad and x.dtype == torch.float64:
            return _F64Matrix.apply(x, y, code, eps)
        if grad and mode in ("cos", "cossim"):
            return _CosineMatrix.apply(x, y, code, eps, precision)
        if grad:
            return _DotMatrix.apply(x, y, code, eps, precision)
        return _sim_matrix(x, y, code, eps, 1.0, precision)
    raise NotImplementedError


# ------------------------------------------------------------------------------------------------
# a3 / a4: masked reductions and the multi-chunk distance reduction
#   lib/tensor_ops.py:182-282 (msum mmean mmin mmax mrand mbest mworst), :288-373 (distance_tensor_redux)
# msum / mmean / mmin / mmax run in one HBM pass of the CUDA kernel behind wealy_masked_reduce; the
# composite reductions (random pick, best-k, redux strategies) are thin compositions of those four
# plus torch.topk / torch.rand_like, with the reference's quirks kept (mask True = EXCLUDED; mworst
# returns 0 -- or NaN when fewer than k entries survive; "bestmin" is shadowed by "best").
# ------------------------------------------------------------------------------------------------
_INF = float("inf")
_OPS = {"sum": 0, "mean": 1, "min": 2, "max": 3}


def _masked_launch(xp, mp, op, fill, eps):
    """wealy_masked_reduce over the columns of the contiguous [rows, cols] xp (mp: its uint8 mask or None) -> [rows]."""
    rows, cols = xp.shape
    out = torch.empty(rows, dtype=xp.dtype, device=xp.device)
    if rows and cols == 0:
        out.fill_({0: 0.0, 1: 0.0, 2: _INF, 3: -_INF}[op])
    elif rows:
        with torch.cuda.device(xp.device):
            N.check(N.lib.wealy_masked_reduce(xp.data_ptr(), mp.data_ptr() if mp is not None else None, rows, cols,
                                              N.dtype_code(xp.dtype, allow_f64=True), op, float(fill), float(eps),
                                              out.data_ptr(), N.stream_ptr(xp.device)))
    return out


class _MaskedReduce(torch.autograd.Function):
    """msum / mmean / mmin / mmax under autograd: dx = g * w, the weights of the forward's selection, rerun by
    wealy_masked_reduce_backward (csrc/masked_kernels.cuh).  `full`: dim=None, where torch.min() spreads the gradient
    over every tied position instead of the first one."""

    @staticmethod
    def forward(ctx, xp, mp, op, fill, eps, full):
        ctx.save_for_backward(xp, mp)
        ctx.cfg = (op, fill, eps, full)
        return _masked_launch(xp.detach(), mp, op, fill, eps)

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        xp, mp = ctx.saved_tensors
        op, fill, eps, full = ctx.cfg
        rows, cols = xp.shape
        dx = torch.empty_like(xp, memory_format=torch.contiguous_format)
        if rows and cols:
            g = g.to(xp.dtype).contiguous()
            with torch.cuda.device(xp.device):
                N.check(N.lib.wealy_masked_reduce_backward(
                    xp.data_ptr(), mp.data_ptr() if mp is not None else None, rows, cols,
                    N.dtype_code(xp.dtype, allow_f64=True), op, float(fill), float(eps), int(full), g.data_ptr(),
                    dx.data_ptr(), N.stream_ptr(xp.device)))
        return dx, None, None, None, None, None


def _reduce(x, mask, dim, keepdim, op, fill=0.0, eps=1e-7):
    N.require_cuda(x)
    N.dtype_code(x.dtype, allow_f64=True)
    grad = x.requires_grad and torch.is_grad_enabled()
    if mask is not None:
        N.require_cuda(mask)
        # like the reference's `included * x` / `torch.where(mask, ctt, x)`, x and mask broadcast together
        # (minmean / meanmin reduce an already-reduced x against the full-size mask); under autograd the expand's
        # backward sums dx back to x's shape
        x, mask = torch.broadcast_tensors(x, mask)
    nd = x.ndim
    if dim is None:
        red = list(range(nd))
    else:
        red = sorted({d % nd for d in ((dim,) if isinstance(dim, int) else tuple(dim))})
    kept = [d for d in range(nd) if d not in red]
    cols_order = red
    if grad and dim is not None and op in (_OPS["min"], _OPS["max"]):
        # the reference reduces the dims one at a time in the caller's order, each taking the first extreme: the last
        # dim reduced is the most significant for ties.  Flatten the columns in that order so that the kernel's
        # "first extreme" is the reference's (the value itself does not depend on the order)
        cols_order = []
        for d in ((dim,) if isinstance(dim, int) else tuple(dim)):
            if d % nd not in cols_order:
                cols_order.append(d % nd)
        cols_order = cols_order[::-1]
    order = kept + cols_order
    kept_shape = [x.shape[d] for d in kept]
    rows = 1
    for s_ in kept_shape:
        rows *= s_
    cols = 1
    for d in red:
        cols *= x.shape[d]
    xp = x.permute(order).contiguous()
    mp = None
    if mask is not None:
        mp = mask.permute(order).contiguous().to(torch.uint8)
    if grad:
        out = _MaskedReduce.apply(xp.view(rows, cols), mp, op, fill, eps, dim is None)
    else:
        out = _masked_launch(xp.view(rows, cols), mp, op, fill, eps)
    out = out.view(kept_shape)
    if keepdim:
        for d in red:
            out = out.unsqueeze(d)
    return out


def msum(x, mask=None, dim=None, keepdim=False):
    return _reduce(x, mask, dim, keepdim, _OPS["sum"])


def mmean(x, mask=None, dim=None, keepdim=False, eps=1e-7):
    return _reduce(x, mask, dim, keepdim, _OPS["mean"], eps=eps)


def mmin(x, mask=None, dim=None, keepdim=False, ctt=torch.inf):
    return _reduce(x, mask, dim, keepdim, _OPS["min"], fill=ctt)


def mmax(x, mask=None, dim=None, keepdim=False, ctt=-torch.inf):
    return _reduce(x, mask, dim, keepdim, _OPS["max"], fill=ctt)


def mrand(x, mask=None, dim=None, keepdim=False, ctt=torch.inf, eps=1e-7):
    keys = torch.rand_like(x)
    if mask is not None:
        keys = torch.where(mask, ctt, keys)
    loser = keys > mmin(keys, mask=mask, dim=dim, keepdim=True, ctt=ctt)
    return mmean(x, mask=loser, dim=dim, keepdim=keepdim, eps=eps)


def mbest(x, k, mask=None, dim=None, keepdim=False, ctt=torch.inf, eps=1e-7):
    assert type(dim) == int
    if mask is not None:
        x = torch.where(mask, ctt, x)
    low = x.topk(k, dim=dim, largest=False)[0]
    return mmean(low, mask=low >= ctt, dim=dim, keepdim=keepdim, eps=eps)


def mworst(x, k, mask=None, dim=None, keepdim=False, ctt=-torch.inf, eps=1e-7):
    assert type(dim) == int
    if mask is not None:
        x = torch.where(mask, ctt, x)
    high = x.topk(k, dim=dim, largest=True)[0]
    return mmean(high, mask=high >= ctt, dim=dim, keepdim=keepdim, eps=eps)   # upstream quirk: excludes everything


def _redux_k(redux, limit):
    return 1 if "-" not in redux else max(1, min(int(redux.split("-")[-1]), limit))


_RDX = {"min": 0, "max": 1, "mean": 2, "minmean": 3, "meanmin": 4}


def _redux_plan(redux):
    """redux string -> (op, karg, symmetric) of wealy_distance_redux, or None when the strategy stays a composition
    (random pick, nested "s" prefixes).  The order of the tests is the reference's (lib/tensor_ops.py:291-368): "best"
    swallows "bestmin", the "s" prefix comes last."""
    sym = 0
    name = redux
    for _ in range(2):
        if name in _RDX:
            return _RDX[name], 0, sym
        if name == "randmin":
            return None
        if name.startswith("bpwr"):
            return 7, (0 if "-" not in name else max(1, int(name.split("-")[-1]))), sym
        if name.startswith("best"):
            return 5, (1 if "-" not in name else max(1, int(name.split("-")[-1]))), sym
        if name.startswith("worst"):
            return 6, (1 if "-" not in name else max(1, int(name.split("-")[-1]))), sym
        if name[:1] == "s" and not sym:
            sym, name = 1, name[1:]
            continue
        break
    return None


def _redux_launch(d, m, plan, eps, inf):
    """wealy_distance_redux on the contiguous (b1, b2, s1, s2) block d (m: its uint8 mask or None) -> (b1, b2)."""
    op, karg, sym = plan
    b1, b2, s1, s2 = d.shape
    out = torch.empty((b1, b2), dtype=d.dtype, device=d.device)
    with torch.cuda.device(d.device):
        N.check(N.lib.wealy_distance_redux(d.data_ptr(), m.data_ptr() if m is not None else None, b1 * b2, s1, s2,
                                           N.dtype_code(d.dtype, allow_f64=True), op, min(karg, 1 << 30), sym, float(eps),
                                           float(inf), out.data_ptr(), N.stream_ptr(d.device)))
    return out


class _ReduxFused(torch.autograd.Function):
    """distance_tensor_redux on the fused path under autograd: d dist = g * w, the weights of the strategy's selection,
    rerun by wealy_distance_redux_backward on the same block (for bpwr the jittered one, whose jitter has gradient 1)."""

    @staticmethod
    def forward(ctx, d, m, plan, eps, inf):
        ctx.save_for_backward(d, m)
        ctx.cfg = (plan, eps, inf)
        return _redux_launch(d.detach(), m, plan, eps, inf)

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        d, m = ctx.saved_tensors
        (op, karg, sym), eps, inf = ctx.cfg
        b1, b2, s1, s2 = d.shape
        dd = torch.empty_like(d, memory_format=torch.contiguous_format)
        g = g.to(d.dtype).contiguous()
        with torch.cuda.device(d.device):
            N.check(N.lib.wealy_distance_redux_backward(
                d.data_ptr(), m.data_ptr() if m is not None else None, b1 * b2, s1, s2,
                N.dtype_code(d.dtype, allow_f64=True), op, min(karg, 1 << 30), sym, float(eps), float(inf), g.data_ptr(),
                dd.data_ptr(), N.stream_ptr(d.device)))
        return dd, None, None, None, None


def _redux_fused(dist, plan, mask, eps, inf):
    """One launch of the fused kernel (csrc/redux_kernels.cuh) -> (b1, b2, 1, 1)."""
    b1, b2, s1, s2 = dist.shape
    if plan[0] == 7:                                    # bpwr: the reference's tie jitter (lib/tensor_ops.py:318)
        dist = dist + eps * torch.rand_like(dist)
    d = dist.contiguous()
    m = None
    if mask is not None:
        m = torch.broadcast_to(mask, dist.shape).contiguous().to(torch.uint8)
    if dist.requires_grad and torch.is_grad_enabled():
        out = _ReduxFused.apply(d, m, plan, eps, inf)
    else:
        out = _redux_launch(d, m, plan, eps, inf)
    return out.view(b1, b2, 1, 1)


def distance_tensor_redux(dist, redux, mask=None, squeeze=True, eps=1e-7, inf=1e12, fused=True):
    """(b1, b2, s1, s2) chunk-vs-chunk distances -> (b1, b2) track-vs-track (lib/tensor_ops.py:288-373).

    Up to 32 chunks per side, every strategy except the random pick runs as ONE kernel launch (one warp per track
    pair, wealy_distance_redux); `fused=False` keeps the composition of masked reductions below (also the path for
    "randmin", nested "s" prefixes and larger blocks), which mirrors the reference branch for branch."""
    if fused and dist.ndim == 4 and dist.is_cuda and 1 <= dist.shape[2] <= 32 and 1 <= dist.shape[3] <= 32:
        plan = _redux_plan(redux)
        if plan is not None:
            out = _redux_fused(dist, plan, mask, eps, inf)
            return out.squeeze((-1, -2)) if squeeze else out
    both = (-1, -2)
    if redux == "min":
        out = mmin(dist, mask=mask, dim=both, keepdim=True, ctt=inf)
    elif redux == "max":
        out = mmax(dist, mask=mask, dim=both, keepdim=True, ctt=-inf)
    elif redux == "mean":
        out = mmean(dist, mask=mask, dim=both, keepdim=True, eps=eps)
    elif redux == "minmean":
        out = mmin(mmean(dist, mask=mask, dim=-1, keepdim=True, eps=eps), mask=mask, dim=both, keepdim=True, ctt=inf)
    elif redux == "meanmin":
        out = mmean(mmin(dist, mask=mask, dim=-1, keepdim=True, ctt=inf), mask=mask, dim=both, keepdim=True, eps=eps)
    elif redux == "randmin":
        out = mrand(mmin(dist, mask=mask, dim=-1, keepdim=True, ctt=inf), mask=mask, dim=both, keepdim=True, ctt=inf,
                    eps=eps)
    elif redux.startswith("bpwr"):  # greedy best pairs without replacement
        if dist.size(3) < dist.size(2):
            dist = dist.transpose(2, 3)
            mask = None if mask is None else mask.transpose(2, 3)
        rounds = dist.size(2) if "-" not in redux else _redux_k(redux, dist.size(2))
        dist = dist + eps * torch.rand_like(dist)
        if mask is None:
            mask = dist > inf
        picked = dist > inf
        for it in range(rounds):
            best = mmin(dist, mask=mask, dim=both, keepdim=True, ctt=inf)
            picked = picked | ((dist <= best) & ~mask)
            if it < rounds - 1:
                mask = (mask | (mmin(dist, mask=mask, dim=-1, keepdim=True, ctt=inf) <= best)
                        | (mmin(dist, mask=mask, dim=-2, keepdim=True, ctt=inf) <= best))
        out = mmean(dist, mask=~picked, dim=both, keepdim=True, eps=eps)
    elif redux.startswith("best"):   # also swallows "bestmin..." exactly like upstream
        k = _redux_k(redux, dist.size(2) * dist.size(3))
        flat = dist.flatten(2).unsqueeze(2)
        fmask = None if mask is None else mask.flatten(2).unsqueeze(2)
        out = mbest(flat, k, mask=fmask, dim=-1, keepdim=True, ctt=inf, eps=eps)
    elif redux.startswith("worst"):
        k = _redux_k(redux, dist.size(2) * dist.size(3))
        flat = dist.flatten(2).unsqueeze(2)
        fmask = None if mask is None else mask.flatten(2).unsqueeze(2)
        out = mworst(flat, k, mask=fmask, dim=-1, keepdim=True, ctt=-inf, eps=eps)
    elif redux[0] == "s":            # symmetrised variant
        fwd = distance_tensor_redux(dist, redux[1:], mask=mask, squeeze=False)
        bwd = distance_tensor_redux(dist.transpose(2, 3), redux[1:],
                                    mask=None if mask is None else mask.transpose(2, 3), squeeze=False)
        out = 0.5 * (fwd + bwd.transpose(2, 3))
    else:
        raise NotImplementedError
    return out.squeeze((-1, -2)) if squeeze else out
