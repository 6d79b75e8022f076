"""The first layer of the `custom` policy network read straight from cell-code grids (snk_grid_conv_in and
snk_grid_conv_in_wgrad of include/snk.h; DESIGN.md section 4.16).

A pixel of view k is one of 7 colours and the colour is set by the cell code alone, so Conv2d(3, 32, 3, 1, 1) over the
view scaled by 1/255 is a lookup per tap in a table T[t][c][o] = sum_rgb W[o, rgb, t] colour[c][rgb] / 255, and its
weight gradient is the same identity backwards through a per-tap, per-class histogram of the incoming gradient.  The
parameters are the ordinary Conv2d weight and bias, so a network trained on grids is the same network as on RGB views.
"""
import ctypes as C

import torch

from . import _lib

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
