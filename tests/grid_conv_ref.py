"""fp64 references of the grid's first convolution layer (snk_grid_conv_in, include/snk.h): the lookup identity, the RGB
path it replaces (expand_grid of test_grid_cpu + conv2d), the weight-gradient histogram, and the grids they run on."""
import numpy as np
import torch
import torch.nn.functional as F

import snake_oracle as so
from test_grid_cpu import CELL_FRUIT, CELL_WALL, cell_body, cell_head, expand_grid, observation_grid

# the class order of snk.h (SNK_GRID_CONV_CLASSES) and each class's colour in view k
CLASS_COLOURS = ((0, 0, 0), so.COL_FRUIT, so.COL_WALL, so.COL_SELF_BODY,
                 so.COL_SELF_HEAD, so.COL_OTHER_BODY, so.COL_OTHER_HEAD)


def cell_classes(grid, view):
    """[..., V, V] codes -> classes 0..6 of view `view`."""
    g = np.asarray(grid).astype(np.int64)
    cls = np.zeros(g.shape, dtype=np.int64)
    cls[g == CELL_FRUIT] = 1
    cls[g == CELL_WALL] = 2
    snake = (g >= 3) & (g != CELL_WALL)
    own = ((g - 3) >> 1) == view
    head = ((g - 3) & 1) == 1
    cls[snake & own & ~head] = 3
    cls[snake & own & head] = 4
    cls[snake & ~own & ~head] = 5
    cls[snake & ~own & head] = 6
    return cls


def colours64():
    return torch.tensor(CLASS_COLOURS, dtype=torch.float64) / 255.0


def table64(weight):
    """T [9, 7, C]: T[3 dy + dx][c][o] = sum_rgb W[o, rgb, dy, dx] colour[c][rgb] / 255."""
    w = torch.as_tensor(weight).double().cpu()
    return torch.einsum("orhw,cr->hwco", w, colours64()).reshape(9, 7, w.shape[0])


def _padded_onehot(grid, view):
    """[n, V + 2, V + 2, 7] one-hot classes with the SAME padding as class 0."""
    cls = cell_classes(grid, view)
    n, V = cls.shape[0], cls.shape[-1]
    pad = np.zeros((n, V + 2, V + 2), dtype=np.int64)
    pad[:, 1:-1, 1:-1] = cls
    return F.one_hot(torch.from_numpy(pad), 7).double()


def lookup_conv64(grid, view, weight, bias):
    """relu(bias + sum_t T[t][class(grid[p + t])]) as [n, V, V, C] fp64: the identity snk_grid_conv_in computes."""
    oh = _padded_onehot(grid, view)
    V = oh.shape[1] - 2
    T = table64(weight)
    acc = torch.as_tensor(bias).double().cpu().reshape(1, 1, 1, -1).expand(oh.shape[0], V, V, -1).clone()
    for dy in range(3):
        for dx in range(3):
            acc += oh[:, dy:dy + V, dx:dx + V] @ T[3 * dy + dx]
    return acc.clamp_min(0.0)


def rgb_conv64(grid, view, weight, bias, requires_grad=False):
    """relu(conv2d(expand_grid(grid, 1, view) / 255)) as [n, V, V, C] fp64 (and the fp64 leaf weight, bias)."""
    x = torch.from_numpy(expand_grid(np.asarray(grid), 1, first_view=view)).double().permute(0, 3, 1, 2) / 255.0
    w = torch.as_tensor(weight).double().cpu().clone().requires_grad_(requires_grad)
    b = torch.as_tensor(bias).double().cpu().clone().requires_grad_(requires_grad)
    return F.relu(F.conv2d(x, w, b, padding=1)).permute(0, 2, 3, 1), w, b


def hist64(grid, view, out, gout):
    """H [9, 7, C]: H[t][c][o] = sum over cells p with class(grid[p + t]) = c of (out > 0 ? gout : 0)."""
    oh = _padded_onehot(grid, view)
    V = oh.shape[1] - 2
    g = torch.where(torch.as_tensor(out).double().cpu() > 0, torch.as_tensor(gout).double().cpu(), 0.0)
    return torch.stack([torch.einsum("npqc,npqo->co", oh[:, dy:dy + V, dx:dx + V], g) for dy in range(3) for dx in range(3)])


def fold64(hist):
    """(dW [C, 3, 3, 3], dbias [C]) from H: dW[o, rgb, t] = sum_c colour[c][rgb] H[t][c][o], dbias = sum_c H[4][c]."""
    h = torch.as_tensor(hist).double().cpu()
    return torch.einsum("hwco,cr->orhw", h.view(3, 3, 7, -1), colours64()), h[4].sum(0)


def autograd_grads64(grid, view, weight, bias, gout):
    """dW, dbias of sum(relu(conv2d(view)) * gout) by fp64 autograd through expand_grid + conv2d."""
    y, w, b = rgb_conv64(grid, view, weight, bias, requires_grad=True)
    (y * torch.as_tensor(gout).double().cpu()).sum().backward()
    return w.grad, b.grad


def oracle_grids(rules, S, V, n_envs=3, steps=25, seed=0):
    """[n_envs, V, V] grids of the Python oracle after `steps` mostly-straight random steps."""
    vo = so.VecOracle(n_envs, size=V - 2, n_snakes=S, rules=rules, seed=seed)
    vo.reset()
    rng = np.random.default_rng(seed)
    for _ in range(steps):
        a = rng.integers(0, 6 if rules == "cut" else 5, size=(n_envs, S))
        a[rng.random((n_envs, S)) < 0.6] = 0
        vo.step(a)
    return np.stack([observation_grid(e) for e in vo.envs])


def synthetic_grids(S, V, n, seed=0):
    """[n, V, V] codes drawn from every code of S snakes, fruit, wall, empty and the unused code 2, on every cell: the
    edges carry non-empty classes, so the zero padding is exercised on all four sides."""
    rng = np.random.default_rng(seed)
    codes = [0, 0, 0, 1, 2, CELL_WALL] + [c for s in range(S) for c in (cell_body(s), cell_head(s))]
    return np.asarray(rng.choice(codes, size=(n, V, V)), dtype=np.uint8)


def random_conv1(seed=0, channels=32):
    """A Conv2d(3, C, 3) weight and bias, orthogonal like CnnPolicy's, with a nonzero bias."""
    gen = torch.Generator().manual_seed(seed)
    w = torch.empty(channels, 3, 3, 3)
    torch.nn.init.orthogonal_(w, gain=2 ** 0.5, generator=gen)
    b = 0.1 * torch.randn(channels, generator=gen)
    return w, b
