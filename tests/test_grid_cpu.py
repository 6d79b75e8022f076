"""CPU: the cell-code grid of obs_mode 'grid' (SNK_CELL_*, include/snk.h) is lossless -- expanded with the colour rule it is
the native observation, pinned against the Python oracle and against the reference's own recordings -- and a grid handle
rejects the debug switches that do not apply to it before any CUDA call."""
import ctypes as C
import os
import zlib

import numpy as np
import pytest

import c_oracle
import helpers
import snake_oracle as so

# The CPU pin of the encoding (SNK_CELL_* of include/snk.h): codes grow in the reference's paint order.
CELL_EMPTY, CELL_FRUIT, CELL_WALL = 0, 1, 255


def cell_body(s):
    return 3 + 2 * s


def cell_head(s):
    return 4 + 2 * s


def observation_grid(env):
    """[V, V] uint8 cell codes of one snake_oracle.SnakeOracle, painted in the order of its observation(): fruits, then the
    snakes by index (body, then head), then the border -- so a fruit outside the board lies under the border."""
    V = env.V
    g = np.zeros(V * V, dtype=np.uint8)
    if env.use_grid:
        g[np.flatnonzero(env.fruit_grid > 0)] = CELL_FRUIT
    else:
        g[env.fruit] = CELL_FRUIT
    for s, b in enumerate(env.body):
        if b:
            g[b] = cell_body(s)
            g[b[0]] = cell_head(s)
    g = g.reshape(V, V)
    g[0, :] = g[V - 1, :] = CELL_WALL
    g[:, 0] = g[:, V - 1] = CELL_WALL
    return g


def expand_grid(grid, n_views, first_view=0):
    """[..., V, V] cell codes -> [..., V, V, 3 n_views]: views first_view .. first_view + n_views - 1 by the colour rule of
    include/snk.h.  The CPU counterpart of snk_expand_views."""
    g = np.asarray(grid, dtype=np.uint8)
    out = np.zeros(g.shape + (n_views, 3), dtype=np.uint8)
    out[g == CELL_FRUIT] = so.COL_FRUIT
    out[g == CELL_WALL] = so.COL_WALL
    snake = (g >= 3) & (g != CELL_WALL)
    owner = (g.astype(np.int64) - 3) >> 1
    head = ((g.astype(np.int64) - 3) & 1) == 1
    for j in range(n_views):
        self_ = snake & (owner == first_view + j)
        other = snake & ~self_
        out[..., j, :][other & ~head] = so.COL_OTHER_BODY
        out[..., j, :][other & head] = so.COL_OTHER_HEAD
        out[..., j, :][self_ & ~head] = so.COL_SELF_BODY
        out[..., j, :][self_ & head] = so.COL_SELF_HEAD
    return out.reshape(g.shape + (3 * n_views,))


def _greedy(env, rng, eps):
    """Fruit-seeking actions from an oracle env's grid: turn toward the nearest fruit onto a free cell, else any free
    cell, with probability eps a uniform action.  Keeps bodies long."""
    g = observation_grid(env).reshape(-1)
    fruits = np.flatnonzero(g == CELL_FRUIT)
    acts = []
    for s in range(env.S):
        b = env.body[s]
        if not b or rng.random() < eps or not len(fruits):
            acts.append(int(rng.integers(env.n_actions)))
            continue
        hx, hy = env.xy(b[0])
        best, best_d = int(rng.integers(1, 5)), None
        for a in range(1, 5):
            nxt = b[0] + env.delta[a]
            if g[nxt] != CELL_EMPTY and g[nxt] != CELL_FRUIT:
                continue
            nx, ny = env.xy(nxt)
            d = min(abs(nx - env.xy(f)[0]) + abs(ny - env.xy(f)[1]) for f in fruits)
            if best_d is None or d < best_d:
                best, best_d = a, d
        acts.append(best)
    return acts


@pytest.mark.parametrize("policy", ["random", "fruit"])
@pytest.mark.parametrize("S", [1, 2, 3, 4, 8])
@pytest.mark.parametrize("rules", ["classic", "adversarial", "cut"])
def test_expanded_grid_is_the_observation(rules, S, policy):
    D = 12 if S == 8 else 10
    vo = so.VecOracle(3, size=D, n_snakes=S, n_views=S + 1, rules=rules, seed=11 + S)
    vo.reset()
    rng = np.random.default_rng(S)
    longest = 0
    for t in range(120):
        if policy == "random":
            acts = rng.integers(0, 6 if rules == "cut" else 5, size=(vo.N, S))
        else:
            acts = np.array([_greedy(e, rng, 0.05) for e in vo.envs])
        vo.step(acts)
        for e in vo.envs:
            g = observation_grid(e)
            assert g.shape == (e.V, e.V) and g.dtype == np.uint8
            for K in sorted({1, S, S + 1}):
                e.K = K
                assert np.array_equal(expand_grid(g, K), e.observation()), (rules, S, K, t)
                if K > 1:  # a run of views is the matching channel slice
                    assert np.array_equal(expand_grid(g, K - 1, first_view=1), e.observation()[..., 3:]), (rules, S, K, t)
            e.K = S + 1
            longest = max(longest, max(len(b) for b in e.body))
    if policy == "fruit" and rules == "classic":
        assert longest >= 6  # the policy did grow bodies


def _grids_from_state(st, V, S):
    """[N, V, V] cell codes of a batch canonical state (snk_dump_state arrays, as the C oracle returns them)."""
    N = len(st["t"])
    g = np.zeros((N, V * V), dtype=np.uint8)
    rows = np.arange(N)
    if "fruit_grid" in st:
        g[st["fruit_grid"] > 0] = CELL_FRUIT
    elif st["fruit"].shape[1]:
        g[rows[:, None], st["fruit"].astype(np.int64)] = CELL_FRUIT
    for s in range(S):
        length = st["len"][:, s].astype(np.int64)
        body = st["body"][:, s].astype(np.int64)
        seg = np.arange(body.shape[1])[None, :] < length[:, None]
        g[np.broadcast_to(rows[:, None], body.shape)[seg], body[seg]] = cell_body(s)
        live = length > 0
        g[rows[live], body[live, 0]] = cell_head(s)
    g = g.reshape(N, V, V)
    g[:, 0, :] = g[:, V - 1, :] = CELL_WALL
    g[:, :, 0] = g[:, :, V - 1] = CELL_WALL
    return g


@pytest.mark.parametrize("name", ["classic_3x10", "classic_2x19", "adversarial_2x10", "adversarial_3x10"])
def test_grid_reproduces_reference_recording(name):
    """Every step of a recording of the reference: the grid of the C oracle's state, expanded, has the recorded crc."""
    g = helpers.load_golden(name)
    N, T, V, S, K = g["N"], min(g["T"], 400), g["D"] + 2, g["S"], g["K"]
    co = c_oracle.COracle(N, size=g["D"], n_snakes=S, n_fruits=g["F"], n_views=K, rules=g["rules"], rng_mode=1)
    co.set_draw_tape(g["tape_vals"], g["tape_bounds"], g["tape_offsets"])
    co.reset()
    assert zlib.crc32(expand_grid(_grids_from_state(co.state(), V, S), K).tobytes()) == int(g["reset_obs_crc"])
    for t in range(T):
        co.step(g["actions"][t])
        grids = _grids_from_state(co.state(), V, S)
        assert zlib.crc32(expand_grid(grids, K).tobytes()) == int(g["obs_crc"][t]), (name, t)


@pytest.fixture(scope="module")
def L():
    import __graft_entry__ as ge
    if not os.path.exists(ge.LIB):
        ge.build()
    from snakes_b200 import _lib
    return _lib


def test_grid_creation_rejects_switches_that_do_not_apply(L):
    lib = L.lib()
    cfg = L.make_config(4, 10, 2, obs_mode=L.OBS_GRID)
    for opts in (b"lane=split", b"delta=1", b"epw=8", b"adaptive=0", b"alt_hi=4", b"force_kernel=tile", b"force_kernel=dense",
                 b"restore_thr=2,lane=fused"):
        out = C.c_void_p()
        assert lib.snk_create_ex(C.byref(cfg), opts, C.byref(out)) == -1 and not out.value, opts
        err = lib.snk_last_error()
        assert opts.split(b",")[-1] in err and b"grid" in err, (opts, err)
    # the switches that keep a meaning get past the check (without a GPU, creation then fails with SNK_ECUDA)
    for opts in (b"", b"force_kernel=lane", b"force_kernel=rows,restore_thr=0"):
        out = C.c_void_p()
        rc = lib.snk_create_ex(C.byref(cfg), opts, C.byref(out))
        assert rc in (0, -2), (opts, rc, lib.snk_last_error())
        if rc == 0:
            lib.snk_destroy(out)
    # a native handle still takes them
    native = L.make_config(4, 10, 2)
    out = C.c_void_p()
    rc = lib.snk_create_ex(C.byref(native), b"lane=split,delta=1", C.byref(out))
    assert rc in (0, -2)
    if rc == 0:
        lib.snk_destroy(out)
    assert lib.snk_create(C.byref(L.make_config(4, 10, 2, obs_mode=3)), C.byref(out)) == -1


def test_expand_views_validates_arguments(L):
    lib = L.lib()
    buf = (C.c_uint8 * 64)()
    p = C.cast(buf, C.c_void_p)
    assert lib.snk_expand_views(None, 1, 10, 0, 1, p, 0, None) == -1
    assert lib.snk_expand_views(p, 1, 10, 0, 1, None, 0, None) == -1
    assert lib.snk_expand_views(p, 0, 10, 0, 1, p, 0, None) == -1
    assert lib.snk_expand_views(p, 1, 1, 0, 1, p, 0, None) == -1 and b"size" in lib.snk_last_error()
    assert lib.snk_expand_views(p, 1, 255, 0, 1, p, 0, None) == -1
    assert lib.snk_expand_views(p, 1, 10, 0, 0, p, 0, None) == -1
    assert lib.snk_expand_views(p, 1, 10, 30, 3, p, 0, None) == -1 and b"views" in lib.snk_last_error()
    assert lib.snk_expand_views(p, 1, 10, -1, 1, p, 0, None) == -1


def test_grid_byte_model(L):
    """The algorithmic bytes of a grid step count one byte per cell for the observation."""
    out = C.c_double(0)
    cfg = L.make_config(131072, 19, 2, 2, 2, "classic", obs_mode=L.OBS_GRID)
    L.check(L.lib().snk_algorithmic_bytes_per_step(C.byref(cfg), 6.0, C.byref(out)))
    assert out.value == 21 * 21 + 19 * 2 + 2 * 6 + 2 * 2 + 30


def test_header_documents_the_codes():
    header = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "snk.h")).read()
    for name, val in (("SNK_OBS_GRID", 2), ("SNK_CELL_EMPTY", 0), ("SNK_CELL_FRUIT", 1), ("SNK_CELL_WALL", 255)):
        assert "#define %s %d" % (name, val) in header
    assert "#define SNK_CELL_BODY(s) (3 + 2 * (s))" in header and "#define SNK_CELL_HEAD(s) (4 + 2 * (s))" in header
    from snakes_b200 import _lib
    assert (_lib.CELL_EMPTY, _lib.CELL_FRUIT, _lib.CELL_WALL, _lib.cell_body(5), _lib.cell_head(5)) == (0, 1, 255, 13, 14)
