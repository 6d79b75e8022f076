"""The first layer of the policy networks read straight from cell-code grids: `custom` on the V x V view (snk_grid_conv_in
and snk_grid_conv_in_wgrad of include/snk.h; DESIGN.md section 4.16) and `nature` on the 84 x 84 WarpFrame view
(snk_grid_conv84_in and snk_grid_conv84_in_wgrad; section 4.17).

A pixel of view k is one of 7 colours and the colour is set by the cell code alone, so Conv2d(3, 32, 3, 1, 1) over the
view scaled by 1/255 is a lookup per tap in a table T[t][c][o] = sum_rgb W[o, rgb, t] colour[c][rgb] / 255, and its
weight gradient is the same identity backwards through a per-tap, per-class histogram of the incoming gradient.  The
WarpFrame view replicates each cell f = 84 / V times, so nature's Conv2d(3, 32, 8, 4) is a lookup per phase and block of
cells in a table folded through the 0/1 matrix M of include/snk.h.  The parameters are the ordinary Conv2d weight and bias,
so a network trained on grids is the same network as on RGB views.
"""
import ctypes as C
import weakref

import torch

from . import _lib
from ._lib import GRID_CONV_CHANNELS

_COLOURS = {}


def _colours(device):
    """[7, 3] float64: the class colours of snk.h scaled by 1/255."""
    col = _COLOURS.get(device)
    if col is None:
        col = _COLOURS[device] = torch.tensor(_lib.GRID_CONV_COLOURS, dtype=torch.float64, device=device) / 255.0
    return col


def grid_conv_table(weight):
    """T [9, 7, C] float32 of a Conv2d weight [C, 3, 3, 3]: T[3 dy + dx][c][o] = sum_rgb weight[o, rgb, dy, dx] colour[c][rgb] / 255."""
    t = torch.einsum("orhw,cr->hwco", weight.detach().double(), _colours(weight.device))
    return t.reshape(9, len(_lib.GRID_CONV_COLOURS), weight.shape[0]).float().contiguous()


def fold_hist(hist, dtype=torch.float32):
    """(dweight [C, 3, 3, 3], dbias [C]) from the histogram H [9, 7, C] of snk_grid_conv_in_wgrad."""
    h = hist.double()
    dw = torch.einsum("hwco,cr->orhw", h.view(3, 3, h.shape[1], h.shape[2]), _colours(hist.device))
    return dw.to(dtype).contiguous(), h[4].sum(0).to(dtype)


def _stream(device):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _check_grid(grid):
    if not isinstance(grid, torch.Tensor) or not grid.is_cuda or grid.dtype != torch.uint8:
        raise TypeError("grid must be a CUDA uint8 tensor")
    if grid.dim() != 3 or grid.shape[1] != grid.shape[2]:
        raise ValueError("grid must be [n, V, V], got %r" % (tuple(grid.shape),))


class GridConvIn(torch.autograd.Function):
    """relu(conv2d(view `view` of `grid` / 255, weight, bias, padding=1)) without the RGB image."""

    @staticmethod
    def forward(ctx, grid, view, weight, bias):
        _check_grid(grid)
        if weight.dim() != 4 or tuple(weight.shape[1:]) != (3, 3, 3) or tuple(bias.shape) != (weight.shape[0],):
            raise ValueError("weight must be [C, 3, 3, 3] and bias [C], got %r and %r" % (tuple(weight.shape), tuple(bias.shape)))
        if weight.device != grid.device or bias.device != grid.device:
            raise ValueError("grid, weight and bias must be on one device")
        g = grid.contiguous()
        n, V, ch = g.shape[0], g.shape[-1], weight.shape[0]
        out = torch.empty((n, V, V, ch), dtype=torch.float32, device=g.device)
        table = grid_conv_table(weight)
        b = bias.detach().float().contiguous()
        dev = g.device.index or 0
        _lib.check(_lib.lib().snk_grid_conv_in(C.c_void_p(g.data_ptr()), n, V - 2, int(view), C.c_void_p(table.data_ptr()),
                                               C.c_void_p(b.data_ptr()), ch, C.c_void_p(out.data_ptr()), dev, _stream(g.device)))
        y = out.permute(0, 3, 1, 2)
        ctx.view, ctx.dtype = int(view), weight.dtype
        ctx.save_for_backward(g, y)
        return y

    @staticmethod
    def backward(ctx, gy):
        g, y = ctx.saved_tensors
        n, V, ch = g.shape[0], g.shape[-1], y.shape[1]
        o = y.permute(0, 2, 3, 1)                  # the forward's NHWC buffer
        go = gy.permute(0, 2, 3, 1).contiguous()   # no copy when the gradient is channels_last, as conv2's is
        hist = (torch.empty if n else torch.zeros)((9, len(_lib.GRID_CONV_COLOURS), ch), dtype=torch.float32, device=g.device)
        work = torch.empty((_lib.grid_conv_work_bytes(n * V * V) // 4,), dtype=torch.float32, device=g.device)
        dev = g.device.index or 0
        _lib.check(_lib.lib().snk_grid_conv_in_wgrad(C.c_void_p(g.data_ptr()), n, V - 2, ctx.view, C.c_void_p(o.data_ptr()),
                                                     C.c_void_p(go.data_ptr()), ch, C.c_void_p(hist.data_ptr()),
                                                     C.c_void_p(work.data_ptr()), work.numel() * 4, dev, _stream(g.device)))
        dw, db = fold_hist(hist, ctx.dtype)
        return None, None, dw if ctx.needs_input_grad[2] else None, db if ctx.needs_input_grad[3] else None


def grid_conv_in(grid, view, weight, bias):
    """The policy's first layer on cell-code grids: `grid` uint8 [n, V, V] (an env's `obs` in obs_mode 'grid', a rollout
    slot, a minibatch), `view` the snake whose view is read (0 <= view < 32), `weight` [32, 3, 3, 3] and `bias` [32] of a
    Conv2d(3, 32, 3, 1, 1).  Returns relu(conv2d(view / 255)) as a channels_last [n, 32, V, V] float32 tensor, equal to
    the RGB path on expand_views(grid, 1, first_view=view) up to float rounding.  Differentiable in weight and bias (the
    grid is data); the backward is deterministic.  Stream-ordered on the current stream; no synchronisation."""
    return GridConvIn.apply(grid, view, weight, bias)


# ---- nature_cnn's first layer on the WarpFrame view (snk_grid_conv84_*) ----

GRID_CONV84_OUT = 20   # output rows and columns of an 8x8 stride-4 VALID conv over 84 x 84
_GEOM84, _M84, _TABLES84 = {}, {}, {}


def conv84_supported(V):
    """True for the grid sizes snk_grid_conv84_in accepts: V divides 84 and 3 <= V <= 42."""
    return 3 <= V <= 42 and 84 % V == 0


def conv84_geometry(V):
    """(f, P, C) of V x V grids (include/snk.h): f = 84 / V pixels per cell, P = f / gcd(f, 4) phases, C the most cells an
    8-pixel window spans per axis."""
    g = _GEOM84.get(V)
    if g is None:
        if not conv84_supported(V):
            raise ValueError("nature on grids needs V dividing 84 with 3 <= V <= 42, got V = %d" % V)
        f = 84 // V
        P = f // (4 if f % 4 == 0 else 2 if f % 2 == 0 else 1)
        C = max((4 * p + 7) // f - (4 * p) // f + 1 for p in range(P))
        g = _GEOM84[V] = (f, P, C)
    return g


def conv84_fold_matrix(V, device="cpu"):
    """M [P, C, 8] float64: M[phi][a][d] = 1 when kernel row d of a window of phase phi falls in its block row a."""
    key = (V, str(device))
    m = _M84.get(key)
    if m is None:
        f, P, C = conv84_geometry(V)
        m = torch.zeros((P, C, 8), dtype=torch.float64)
        for p in range(P):
            for d in range(8):
                m[p, (4 * p + d) // f - (4 * p) // f, d] = 1.0
        m = _M84[key] = m.to(device)
    return m


def grid_conv84_table(weight, V):
    """T [P, P, C, C, 7, 32] float32 of a Conv2d weight [32, 3, 8, 8] for V x V grids:
    T[py][px][a][b][c][o] = sum_{dy,dx} M[py][a][dy] M[px][b][dx] sum_rgb weight[o, rgb, dy, dx] colour[c][rgb] / 255."""
    m = conv84_fold_matrix(V, weight.device)
    t = torch.einsum("pad,qbe,orde,cr->pqabco", m, m, weight.detach().double(), _colours(weight.device))
    return t.float().contiguous()


def fold_hist84(hist, V, dtype=torch.float32):
    """(dweight [32, 3, 8, 8], dbias [32]) from the histogram H [P, P, C, C, 7, 32] of snk_grid_conv84_in_wgrad."""
    h = hist.double()
    m = conv84_fold_matrix(V, hist.device)
    dw = torch.einsum("pad,qbe,pqabco,cr->orde", m, m, h, _colours(hist.device))
    return dw.to(dtype).contiguous(), h[:, :, 0, 0].sum((0, 1, 2)).to(dtype)


def _table84(weight, V):
    """grid_conv84_table, cached per weight tensor, V and weight._version (in-place updates such as an optimizer step,
    copy_ or load_state_dict bump it), so that the policy calls of a rollout share one table build."""
    key = (id(weight), V)
    ent = _TABLES84.get(key)
    if ent is not None and ent[0]() is weight and ent[1] == (weight._version, weight.data_ptr()):
        return ent[2]
    t = grid_conv84_table(weight, V)
    _TABLES84[key] = (weakref.ref(weight, lambda _r, k=key: _TABLES84.pop(k, None)), (weight._version, weight.data_ptr()), t)
    return t


class GridConv84In(torch.autograd.Function):
    """relu(conv2d(WarpFrame of view `view` of `grid` / 255, weight, bias, stride=4)) without the RGB image."""

    @staticmethod
    def forward(ctx, grid, view, weight, bias):
        _check_grid(grid)
        if tuple(weight.shape) != (GRID_CONV_CHANNELS, 3, 8, 8) or tuple(bias.shape) != (GRID_CONV_CHANNELS,):
            raise ValueError("weight must be [32, 3, 8, 8] and bias [32], got %r and %r" % (tuple(weight.shape), tuple(bias.shape)))
        if weight.device != grid.device or bias.device != grid.device:
            raise ValueError("grid, weight and bias must be on one device")
        g = grid.contiguous()
        n, V = g.shape[0], g.shape[-1]
        _lib.grid_conv84_geometry(V)   # SnkError for an unsupported V, before the table is built
        out = torch.empty((n, GRID_CONV84_OUT, GRID_CONV84_OUT, GRID_CONV_CHANNELS), dtype=torch.float32, device=g.device)
        table = _table84(weight, V)
        b = bias.detach().float().contiguous()
        dev = g.device.index or 0
        _lib.check(_lib.lib().snk_grid_conv84_in(C.c_void_p(g.data_ptr()), n, V - 2, int(view), C.c_void_p(table.data_ptr()),
                                                 C.c_void_p(b.data_ptr()), GRID_CONV_CHANNELS, C.c_void_p(out.data_ptr()), dev,
                                                 _stream(g.device)))
        y = out.permute(0, 3, 1, 2)
        ctx.view, ctx.dtype = int(view), weight.dtype
        ctx.save_for_backward(g, y)
        return y

    @staticmethod
    def backward(ctx, gy):
        g, y = ctx.saved_tensors
        n, V = g.shape[0], g.shape[-1]
        f, P, Cb, work_bytes = _lib.grid_conv84_geometry(V, n)
        o = y.permute(0, 2, 3, 1)                  # the forward's NHWC buffer
        go = gy.permute(0, 2, 3, 1).contiguous()   # no copy when the gradient is channels_last, as conv2's is
        hist = (torch.empty if n else torch.zeros)((P, P, Cb, Cb, 7, GRID_CONV_CHANNELS), dtype=torch.float32, device=g.device)
        work = torch.empty((max(work_bytes, 4) // 4,), dtype=torch.float32, device=g.device)
        dev = g.device.index or 0
        _lib.check(_lib.lib().snk_grid_conv84_in_wgrad(C.c_void_p(g.data_ptr()), n, V - 2, ctx.view, C.c_void_p(o.data_ptr()),
                                                       C.c_void_p(go.data_ptr()), GRID_CONV_CHANNELS, C.c_void_p(hist.data_ptr()),
                                                       C.c_void_p(work.data_ptr()), work.numel() * 4, dev, _stream(g.device)))
        dw, db = fold_hist84(hist, V, ctx.dtype)
        return None, None, dw if ctx.needs_input_grad[2] else None, db if ctx.needs_input_grad[3] else None


def grid_conv84_in(grid, view, weight, bias):
    """nature_cnn's first layer on cell-code grids: `grid` uint8 [n, V, V] with V dividing 84 and 3 <= V <= 42 (an env's
    `obs` in obs_mode 'grid', a rollout slot, a minibatch), `view` the snake whose view is read (0 <= view < 32), `weight`
    [32, 3, 8, 8] and `bias` [32] of a Conv2d(3, 32, 8, 4).  Returns relu(conv2d(WarpFrame(view) / 255, stride 4)) as a
    channels_last [n, 32, 20, 20] float32 tensor, equal to the RGB path on expand_views(grid, 1, first_view=view)
    replicated 84 / V times per cell (the obs_mode 'atari84' view) up to float rounding.  Differentiable in weight and
    bias (the grid is data); the backward is deterministic.  The lookup table is rebuilt only when the weight changes
    (weight._version).  Stream-ordered on the current stream; no synchronisation."""
    return GridConv84In.apply(grid, view, weight, bias)
