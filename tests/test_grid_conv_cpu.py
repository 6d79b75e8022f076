"""CPU: the identity behind snk_grid_conv_in.  The policy's first layer over view k of a cell-code grid -- Conv2d(3, 32, 3,
padding 1) on the expanded view / 255, then ReLU -- is a per-tap table lookup on the cell classes, and its weight
gradient folds from a per-tap, per-class histogram.  Checked in fp64 against expand_grid + conv2d and autograd, and the
package's own table / fold helpers against the same references."""
import numpy as np
import pytest
import torch

import grid_conv_ref as ref

VIEWS_OF = lambda S: sorted(set(range(S)) | {S, 31})  # noqa: E731  every own view, one past the snakes, the last one


@pytest.mark.parametrize("S", [1, 2, 3, 4, 8, 16])
@pytest.mark.parametrize("rules", ["classic", "adversarial", "cut"])
def test_lookup_equals_conv_on_oracle_grids(rules, S):
    V = {1: 12, 2: 12, 3: 12, 4: 12, 8: 14, 16: 21}[S]
    grids = ref.oracle_grids(rules, S, V, n_envs=3, steps=30, seed=S)
    w, b = ref.random_conv1(seed=S)
    for k in VIEWS_OF(S):
        want, _, _ = ref.rgb_conv64(grids, k, w, b)
        got = ref.lookup_conv64(grids, k, w, b)
        assert torch.allclose(got, want, rtol=0, atol=1e-12), (rules, S, k, float((got - want).abs().max()))


@pytest.mark.parametrize("V", [4, 12, 21, 66])
@pytest.mark.parametrize("S", [1, 2, 3, 4, 8, 16])
def test_lookup_equals_conv_on_any_codes_with_padding_on_every_edge(V, S):
    grids = ref.synthetic_grids(S, V, n=2, seed=V + S)
    for edge in (grids[:, 0], grids[:, -1], grids[:, :, 0], grids[:, :, -1]):   # every edge carries non-empty cells
        assert (ref.cell_classes(edge, 0) != 0).any()
    w, b = ref.random_conv1(seed=V)
    for k in VIEWS_OF(S):
        want, _, _ = ref.rgb_conv64(grids, k, w, b)
        got = ref.lookup_conv64(grids, k, w, b)
        assert torch.allclose(got, want, rtol=0, atol=1e-12), (V, S, k)


@pytest.mark.parametrize("V,S,rules", [(12, 2, "classic"), (21, 16, "adversarial"), (66, 16, "cut"), (4, 3, None), (21, 8, None)])
def test_folded_histogram_equals_autograd(V, S, rules):
    grids = ref.oracle_grids(rules, S, V, n_envs=2, steps=20, seed=V) if rules else ref.synthetic_grids(S, V, n=3, seed=V)
    w, b = ref.random_conv1(seed=S)
    rng = np.random.default_rng(V)
    for k in sorted({0, 1 % S, S, 31}):
        y = ref.lookup_conv64(grids, k, w, b)
        assert (y == 0).any() and (y > 0).any()   # the ReLU mask matters
        gout = torch.from_numpy(rng.standard_normal(tuple(y.shape)))
        dw_want, db_want = ref.autograd_grads64(grids, k, w, b, gout)
        dw, db = ref.fold64(ref.hist64(grids, k, y, gout))
        assert torch.allclose(dw, dw_want, rtol=0, atol=1e-10) and torch.allclose(db, db_want, rtol=0, atol=1e-10), (V, S, k)


def test_package_table_and_fold_match_the_reference():
    """snakes_b200.grid_conv builds the kernel's table and folds its histogram with these formulas (on any device)."""
    from snakes_b200 import _lib, grid_conv
    assert tuple(_lib.GRID_CONV_COLOURS) == tuple(tuple(c) for c in ref.CLASS_COLOURS)
    w, b = ref.random_conv1(seed=5)
    t = grid_conv.grid_conv_table(w)
    assert t.dtype == torch.float32 and tuple(t.shape) == (9, 7, 32) and t.is_contiguous()
    assert torch.allclose(t.double(), ref.table64(w), rtol=0, atol=1e-6) and not t[:, 0].any()
    grids = ref.synthetic_grids(3, 12, n=2, seed=1)
    y = ref.lookup_conv64(grids, 1, w, b)
    gout = torch.from_numpy(np.random.default_rng(0).standard_normal(tuple(y.shape)))
    h = ref.hist64(grids, 1, y, gout)
    dw, db = grid_conv.fold_hist(h.float())
    dw_want, db_want = ref.autograd_grads64(grids, 1, w, b, gout)
    assert dw.dtype == torch.float32 and tuple(dw.shape) == (32, 3, 3, 3)
    assert torch.allclose(dw.double(), dw_want, atol=1e-4) and torch.allclose(db.double(), db_want, atol=1e-4)


def test_workspace_formula_matches_the_header():
    import os
    import re
    from snakes_b200 import _lib
    hdr = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "snk.h")).read()
    val = lambda name: int(re.search(r"#define %s (\d+)" % name, hdr).group(1))  # noqa: E731
    assert _lib.GRID_CONV_CHANNELS == val("SNK_GRID_CONV_CHANNELS") and len(_lib.GRID_CONV_COLOURS) == val("SNK_GRID_CONV_CLASSES")
    assert _lib.GRID_CONV_WGRAD_CELLS_PER_CTA == val("SNK_GRID_CONV_WGRAD_CELLS_PER_CTA")
    assert _lib.GRID_CONV_WGRAD_MAX_CTAS == val("SNK_GRID_CONV_WGRAD_MAX_CTAS")
    assert _lib.grid_conv_work_bytes(1) == _lib.GRID_CONV_PART_FLOATS * 4 == 55 * 32 * 4
    assert _lib.grid_conv_work_bytes(2048 * 3 + 1) == 4 * 55 * 32 * 4
    assert _lib.grid_conv_work_bytes(131072 * 441) == 592 * 55 * 32 * 4


def test_grid_conv_rejects_bad_arguments_before_any_cuda_call():
    """Argument checks of the C entries run before the device is touched: channels, size, view, n, workspace."""
    import ctypes as C
    from snakes_b200 import _lib
    L = _lib.lib()
    p = C.c_void_p(256)   # never dereferenced: every call below is rejected first
    assert L.snk_grid_conv_in(p, 4, 10, 0, p, p, 16, p, 0, None) == -1 and b"channels" in L.snk_last_error()
    assert L.snk_grid_conv_in(p, 4, 255, 0, p, p, 32, p, 0, None) == -1 and b"size" in L.snk_last_error()
    assert L.snk_grid_conv_in(p, 4, 0, 0, p, p, 32, p, 0, None) == -1
    assert L.snk_grid_conv_in(p, 4, 10, 32, p, p, 32, p, 0, None) == -1 and b"view" in L.snk_last_error()
    assert L.snk_grid_conv_in(p, 4, 10, -1, p, p, 32, p, 0, None) == -1
    assert L.snk_grid_conv_in(p, -1, 10, 0, p, p, 32, p, 0, None) == -1
    assert L.snk_grid_conv_in(None, 4, 10, 0, p, p, 32, p, 0, None) == -1
    assert L.snk_grid_conv_in(p, 4, 10, 0, C.c_void_p(260), p, 32, p, 0, None) == -1 and b"aligned" in L.snk_last_error()
    assert L.snk_grid_conv_in(None, 0, 10, 0, None, None, 32, None, 0, None) == 0   # n = 0: nothing to do
    need = _lib.grid_conv_work_bytes(4 * 12 * 12)
    assert L.snk_grid_conv_in_wgrad(p, 4, 10, 0, p, p, 32, p, p, need - 1, 0, None) == -1 and b"workspace" in L.snk_last_error()
    assert L.snk_grid_conv_in_wgrad(p, 4, 10, 0, p, p, 64, p, p, need, 0, None) == -1
    assert L.snk_grid_conv_in_wgrad(p, 4, 10, 40, p, p, 32, p, p, need, 0, None) == -1
    assert L.snk_grid_conv_in_wgrad(None, 0, 10, 0, None, None, 32, None, None, 0, 0, None) == 0
