"""fp64 references of nature_cnn's first layer on grids (snk_grid_conv84_in, include/snk.h): the phase-table lookup, the RGB
path it replaces (expand_grid of test_grid_cpu replicated f x f per cell, then conv2d with stride 4), the weight-gradient
histogram and its fold.  Grids, weights and class rules come from grid_conv_ref."""
import numpy as np
import torch
import torch.nn.functional as F

from grid_conv_ref import cell_classes, colours64
from test_grid_cpu import expand_grid

SUPPORTED_V = (3, 4, 6, 7, 12, 14, 21, 28, 42)
OUT = 20


def geometry(V):
    """(f, P, C, M [P, C, 8] float64) straight from the definitions of include/snk.h."""
    f = 84 // V
    P = f // int(np.gcd(f, 4))
    C = max((4 * p + 7) // f - (4 * p) // f + 1 for p in range(P))
    M = torch.zeros((P, C, 8), dtype=torch.float64)
    for p in range(P):
        for d in range(8):
            M[p, (4 * p + d) // f - (4 * p) // f, d] = 1.0
    return f, P, C, M


def reached(V):
    """[P, P, C, C] bool: block (a, b) is reached by the windows of phase pair (py, px)."""
    M = geometry(V)[3]
    r = M.sum(-1) > 0
    return r[:, None, :, None] & r[None, :, None, :]


def table64(weight, V):
    """T [P, P, C, C, 7, 32] = sum_{dy,dx} M[py][a][dy] M[px][b][dx] sum_rgb W[o, rgb, dy, dx] colour[c][rgb] / 255."""
    M = geometry(V)[3]
    w = torch.as_tensor(weight).double().cpu()
    return torch.einsum("pad,qbe,orde,cr->pqabco", M, M, w, colours64())


def _block_onehots(grid, view):
    """{(a, b): [n, 20, 20, 7]} one-hot class of block (a, b) of every output (all zero where the block lies off the grid),
    and the per-output phase indices py [20], px [20]."""
    cls = cell_classes(grid, view)
    n, V = cls.shape[0], cls.shape[-1]
    f, P, C, _ = geometry(V)
    pad = np.full((n, V + C, V + C), -1, dtype=np.int64)
    pad[:, :V, :V] = cls
    oh = F.one_hot(torch.from_numpy(pad + 1), 8)[..., 1:].double()   # class -1 (off the grid) -> all zero
    o = np.arange(OUT)
    c0 = 4 * o // f
    blocks = {(a, b): oh[:, c0[:, None] + a, c0[None, :] + b] for a in range(C) for b in range(C)}
    return blocks, o % P


def lookup_conv84_64(grid, view, weight, bias):
    """relu(bias + sum_{a,b} T[oy % P][ox % P][a][b][class(grid[cy + a][cx + b])]) as [n, 20, 20, 32] fp64."""
    blocks, ph = _block_onehots(grid, view)
    T = table64(weight, np.asarray(grid).shape[-1])
    acc = torch.as_tensor(bias).double().cpu().reshape(1, 1, 1, -1).expand(np.asarray(grid).shape[0], OUT, OUT, -1).clone()
    for (a, b), oh in blocks.items():
        acc += torch.einsum("nyxc,yxco->nyxo", oh, T[ph[:, None], ph[None, :], a, b])
    return acc.clamp_min(0.0)


def rgb_conv84_64(grid, view, weight, bias, requires_grad=False):
    """relu(conv2d(WarpFrame(expand_grid(grid, 1, view)) / 255, stride 4)) as [n, 20, 20, 32] fp64 (and the fp64 leaves):
    the view replicated 84 / V times per cell, as obs_mode 'atari84' draws it."""
    g = np.asarray(grid)
    f = 84 // g.shape[-1]
    img = expand_grid(g, 1, first_view=view).repeat(f, axis=1).repeat(f, axis=2)
    x = torch.from_numpy(img).double().permute(0, 3, 1, 2) / 255.0
    w = torch.as_tensor(weight).double().cpu().clone().requires_grad_(requires_grad)
    b = torch.as_tensor(bias).double().cpu().clone().requires_grad_(requires_grad)
    return F.relu(F.conv2d(x, w, b, stride=4)).permute(0, 2, 3, 1), w, b


def hist84_64(grid, view, out, gout):
    """H [P, P, C, C, 7, 32]: the sum of (out > 0 ? gout : 0) over outputs of phase pair (py, px) whose block (a, b) has
    class c; zero for blocks the phase does not reach."""
    V = np.asarray(grid).shape[-1]
    _, P, C, _ = geometry(V)
    blocks, ph = _block_onehots(grid, view)
    g = torch.where(torch.as_tensor(out).double().cpu() > 0, torch.as_tensor(gout).double().cpu(), 0.0)
    sel = F.one_hot(torch.from_numpy(ph), P).double()   # [20, P]: output row / column -> phase
    H = torch.zeros((P, P, C, C, 7, g.shape[-1]), dtype=torch.float64)
    for (a, b), oh in blocks.items():
        H[:, :, a, b] = torch.einsum("nyxc,nyxo,yp,xq->pqco", oh, g, sel, sel)
    return H * reached(V)[..., None, None]


def fold84_64(hist, V):
    """(dW [32, 3, 8, 8], dbias [32]) from H through M and the colours."""
    M = geometry(V)[3]
    h = torch.as_tensor(hist).double().cpu()
    return torch.einsum("pad,qbe,pqabco,cr->orde", M, M, h, colours64()), h[:, :, 0, 0].sum((0, 1, 2))


def autograd_grads84_64(grid, view, weight, bias, gout):
    """dW, dbias of sum(relu(conv2d(WarpFrame(view))) * gout) by fp64 autograd."""
    y, w, b = rgb_conv84_64(grid, view, weight, bias, requires_grad=True)
    (y * torch.as_tensor(gout).double().cpu()).sum().backward()
    return w.grad, b.grad


def random_conv1_84(seed=0, channels=32):
    """A Conv2d(3, C, 8, 4) weight and bias, orthogonal like CnnPolicy's, with a nonzero bias."""
    gen = torch.Generator().manual_seed(seed)
    w = torch.empty(channels, 3, 8, 8)
    torch.nn.init.orthogonal_(w, gain=2 ** 0.5, generator=gen)
    b = 0.1 * torch.randn(channels, generator=gen)
    return w, b
