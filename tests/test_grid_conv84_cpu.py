"""CPU: the identity behind snk_grid_conv84_in.  nature_cnn's first layer over the WarpFrame of view k of a cell-code grid
-- Conv2d(3, 32, 8, stride 4) on the view replicated 84 / V times per cell, / 255, then ReLU -- is a lookup per phase
pair and block of cells, and its weight gradient folds from a per-phase, per-block, per-class histogram.  Checked in fp64
against expand_grid + replication + conv2d and autograd for every supported V; the package's geometry, table and fold
helpers and the C geometry entry against the same definitions."""
import ctypes as C

import numpy as np
import pytest
import torch

import grid_conv84_ref as ref84
import grid_conv_ref as ref

VIEWS_OF = lambda S: sorted({0, 1, S, 31})  # noqa: E731  the first two views, one past the snakes, the last one


@pytest.mark.parametrize("V", ref84.SUPPORTED_V)
def test_lookup_equals_strided_conv_on_synthetic_grids(V):
    """Every supported V, non-empty cells on every edge, every code of up to 16 snakes."""
    S = 16 if V >= 21 else 3
    grids = ref.synthetic_grids(S, V, n=2, seed=V)
    for edge in (grids[:, 0], grids[:, -1], grids[:, :, 0], grids[:, :, -1]):
        assert (ref.cell_classes(edge, 0) != 0).any()
    w, b = ref84.random_conv1_84(seed=V)
    for k in VIEWS_OF(S):
        want, _, _ = ref84.rgb_conv84_64(grids, k, w, b)
        got = ref84.lookup_conv84_64(grids, k, w, b)
        assert got.shape == (2, 20, 20, 32)
        assert torch.allclose(got, want, rtol=0, atol=1e-12), (V, k, float((got - want).abs().max()))


@pytest.mark.parametrize("V,S", [(6, 1), (7, 2), (12, 2), (14, 4), (21, 2), (28, 8), (42, 16)])
@pytest.mark.parametrize("rules", ["classic", "adversarial", "cut"])
def test_lookup_equals_strided_conv_on_oracle_grids(rules, V, S):
    grids = ref.oracle_grids(rules, S, V, n_envs=2, steps=20, seed=V + S)
    w, b = ref84.random_conv1_84(seed=S)
    for k in VIEWS_OF(S):
        want, _, _ = ref84.rgb_conv84_64(grids, k, w, b)
        got = ref84.lookup_conv84_64(grids, k, w, b)
        assert torch.allclose(got, want, rtol=0, atol=1e-12), (rules, V, S, k)


@pytest.mark.parametrize("V", ref84.SUPPORTED_V)
def test_folded_histogram_equals_autograd(V):
    S = 16 if V >= 21 else 3
    grids = ref.oracle_grids("classic", 2, V, n_envs=2, steps=15, seed=V) if V >= 12 else ref.synthetic_grids(S, V, n=3, seed=V)
    w, b = ref84.random_conv1_84(seed=V + 1)
    rng = np.random.default_rng(V)
    for k in (0, 1):
        y = ref84.lookup_conv84_64(grids, k, w, b)
        assert (y == 0).any() and (y > 0).any()   # the ReLU mask matters
        gout = torch.from_numpy(rng.standard_normal(tuple(y.shape)))
        dw_want, db_want = ref84.autograd_grads84_64(grids, k, w, b, gout)
        dw, db = ref84.fold84_64(ref84.hist84_64(grids, k, y, gout), V)
        assert torch.allclose(dw, dw_want, rtol=0, atol=1e-10) and torch.allclose(db, db_want, rtol=0, atol=1e-10), (V, k)


def test_geometry_entry_agrees_with_the_definitions_and_rejects_other_sizes():
    from snakes_b200 import _lib, grid_conv
    L = _lib.lib()
    out = (C.c_int64 * 4)()
    for V in range(1, 100):
        rc = L.snk_grid_conv84_geometry(V - 2, 1, out)
        if V not in ref84.SUPPORTED_V:
            assert rc == -1 and b"size" in L.snk_last_error(), V
            assert not grid_conv.conv84_supported(V)
            with pytest.raises(ValueError):
                grid_conv.conv84_geometry(V)
            continue
        assert rc == 0, V
        f, P, Cb, M = ref84.geometry(V)
        assert tuple(out)[:3] == (f, P, Cb) == grid_conv.conv84_geometry(V), V
        assert torch.equal(grid_conv.conv84_fold_matrix(V), M), V
        assert M.sum((1,)).eq(1).all()   # every kernel row falls in exactly one block
        rows = Cb * Cb * 6 + 1
        assert out[3] == P * P * rows * 32 * 4, V   # n = 1: one CTA per phase pair
        assert _lib.grid_conv84_geometry(V, 0)[3] == 0
        big = _lib.grid_conv84_geometry(V, 131072)[3]
        assert big % (P * P * rows * 32 * 4) == 0 and big <= (592 + P * P) * rows * 32 * 4
    assert L.snk_grid_conv84_geometry(10, -1, out) == -1
    assert L.snk_grid_conv84_geometry(10, 1, None) == -1
    assert {V: ref84.geometry(V)[:3] for V in (12, 21)} == {12: (7, 7, 2), 21: (4, 1, 2)}


def test_package_table_and_fold_match_the_reference():
    from snakes_b200 import grid_conv
    w, b = ref84.random_conv1_84(seed=3)
    for V in (12, 21, 28):
        f, P, Cb, _ = ref84.geometry(V)
        t = grid_conv.grid_conv84_table(w, V)
        assert t.dtype == torch.float32 and tuple(t.shape) == (P, P, Cb, Cb, 7, 32) and t.is_contiguous()
        assert torch.allclose(t.double(), ref84.table64(w, V), rtol=0, atol=1e-6) and not t[..., 0, :].any()
        assert not t[~ref84.reached(V)].any()
        grids = ref.synthetic_grids(3, V, n=2, seed=V)
        y = ref84.lookup_conv84_64(grids, 1, w, b)
        gout = torch.from_numpy(np.random.default_rng(V).standard_normal(tuple(y.shape)))
        dw, db = grid_conv.fold_hist84(ref84.hist84_64(grids, 1, y, gout).float(), V)
        dw_want, db_want = ref84.autograd_grads84_64(grids, 1, w, b, gout)
        assert dw.dtype == torch.float32 and tuple(dw.shape) == (32, 3, 8, 8)
        assert torch.allclose(dw.double(), dw_want, atol=1e-3) and torch.allclose(db.double(), db_want, atol=1e-3), V


def test_nature_grid_policy_has_the_rgb_nature_policy_parameters():
    from snakes_b200 import selfplay
    want = [a.shape for a in selfplay.CnnPolicy((84, 84, 3), 5, "nature").to_tf_list()]
    for V in ref84.SUPPORTED_V:
        net = selfplay.CnnPolicy((V, V, 3), 5, "nature", grid=True)
        assert net.conv_out == (7, 7, 64) and net.grid and net.arch == "nature"
        assert [a.shape for a in net.to_tf_list()] == want, V
        net.from_tf_list(selfplay.CnnPolicy((84, 84, 3), 5, "nature").to_tf_list())
    for V in (11, 5, 84, 2):
        with pytest.raises(ValueError):
            selfplay.CnnPolicy((V, V, 3), 5, "nature", grid=True)


def test_grid_conv84_rejects_bad_arguments_before_any_cuda_call():
    """Argument checks of the C entries run before the device is touched: channels, size, view, n, alignment, workspace."""
    from snakes_b200 import _lib
    L = _lib.lib()
    p = C.c_void_p(256)   # never dereferenced: every call below is rejected first
    assert L.snk_grid_conv84_in(p, 4, 10, 0, p, p, 16, p, 0, None) == -1 and b"channels" in L.snk_last_error()
    for size in (9, 0, 82, 40 + 84, -2):   # V = 11, 2, 84, 126, 0
        assert L.snk_grid_conv84_in(p, 4, size, 0, p, p, 32, p, 0, None) == -1 and b"size" in L.snk_last_error(), size
    assert L.snk_grid_conv84_in(p, 4, 10, 32, p, p, 32, p, 0, None) == -1 and b"view" in L.snk_last_error()
    assert L.snk_grid_conv84_in(p, 4, 10, -1, p, p, 32, p, 0, None) == -1
    assert L.snk_grid_conv84_in(p, -1, 10, 0, p, p, 32, p, 0, None) == -1
    assert L.snk_grid_conv84_in(None, 4, 10, 0, p, p, 32, p, 0, None) == -1 and b"NULL" in L.snk_last_error()
    assert L.snk_grid_conv84_in(p, 4, 10, 0, C.c_void_p(260), p, 32, p, 0, None) == -1 and b"aligned" in L.snk_last_error()
    assert L.snk_grid_conv84_in(p, 4, 10, 0, p, C.c_void_p(264), 32, p, 0, None) == -1
    assert L.snk_grid_conv84_in(p, 4, 10, 0, p, p, 32, C.c_void_p(280 + 4), 0, None) == -1
    assert L.snk_grid_conv84_in(None, 0, 10, 0, None, None, 32, None, 0, None) == 0   # n = 0: nothing to do
    need = _lib.grid_conv84_geometry(12, 4)[3]
    args = lambda wb, **kw: [kw.get("g", p), 4, kw.get("size", 10), kw.get("view", 0), kw.get("o", p), kw.get("go", p),  # noqa: E731
                             kw.get("ch", 32), kw.get("h", p), kw.get("w", p), wb, 0, None]
    assert L.snk_grid_conv84_in_wgrad(*args(need - 4)) == -1 and b"workspace" in L.snk_last_error()
    assert L.snk_grid_conv84_in_wgrad(*args(need, ch=64)) == -1
    assert L.snk_grid_conv84_in_wgrad(*args(need, view=40)) == -1
    assert L.snk_grid_conv84_in_wgrad(*args(need, size=9)) == -1
    for k in ("g", "o", "go", "h", "w"):
        assert L.snk_grid_conv84_in_wgrad(*args(need, **{k: None})) == -1, k
    for k in ("o", "go", "h", "w"):
        assert L.snk_grid_conv84_in_wgrad(*args(need, **{k: C.c_void_p(258)})) == -1 and b"aligned" in L.snk_last_error(), k
    assert L.snk_grid_conv84_in_wgrad(None, 0, 10, 0, None, None, 32, None, None, 0, 0, None) == 0
