"""CPU: argument checks of the per-env state entry points (snk_save_envs / snk_restore_envs / snk_copy_envs) and of the
host-side index validation of SnakeVecEnv.save_envs / restore_envs / copy_envs.  No GPU work."""
import ctypes as C
import os

import numpy as np
import pytest


@pytest.fixture(scope="module")
def L():
    import __graft_entry__ as ge
    if not os.path.exists(ge.LIB):
        ge.build()
    from snakes_b200 import _lib
    return _lib


def test_entry_points_reject_null_arguments(L):
    lib = L.lib()
    buf = (C.c_uint8 * 64)()
    assert lib.snk_save_envs(None, None, 1, buf, 64, None) == -1
    assert b"NULL" in lib.snk_last_error()
    assert lib.snk_restore_envs(None, None, 1, buf, 64, None) == -1
    assert b"NULL" in lib.snk_last_error()
    assert lib.snk_copy_envs(None, None, None, 1, None) == -1
    assert b"NULL" in lib.snk_last_error()
    assert set(L.DEVERR) == {1, 2, 4, 8, 16} and "index" in L.DEVERR[16]


def test_blob_size_follows_the_count_env_layout(L):
    """The device blob of `count` envs is snk_state_layout_of with num_envs = count: what the entry points check
    `bytes` against."""
    lib = L.lib()
    sizes = []
    for n in (1, 2, 131072):
        lay = L.SnkStateLayout()
        L.check(lib.snk_state_layout_of(C.byref(L.make_config(n, 19, 2)), C.byref(lay)))
        sizes.append(lay.total_bytes)
    assert sizes[0] < sizes[1] < sizes[2]
    assert 1500 <= sizes[2] / 131072 <= 1510   # about 1 506 bytes per env at 2 snakes on 19x19


class _Cfg(object):
    def __init__(self, size, n_snakes, n_fruits, rules):
        self.size, self.n_snakes, self.n_fruits, self.rules = size, n_snakes, n_fruits, rules


def _host_env(N):
    """A SnakeVecEnv shell without a handle: enough for the host-side index and geometry checks."""
    import torch
    from snakes_b200 import SnakeVecEnv
    env = SnakeVecEnv.__new__(SnakeVecEnv)
    env.N, env.device, env.cfg = N, torch.device("cpu"), _Cfg(19, 2, 2, 0)
    return env


def test_host_indices_are_checked(L):
    env = _host_env(10)
    t, n, a = env._env_index([3, 1, 3])
    assert n == 3 and t.dtype.is_floating_point is False and list(a) == [3, 1, 3]
    with pytest.raises(IndexError):
        env._env_index([0, 10])
    with pytest.raises(IndexError):
        env._env_index(np.array([-1]))
    with pytest.raises(ValueError):
        env._env_index([2, 2], distinct=True)
    with pytest.raises(ValueError):
        env._env_index([])
    with pytest.raises(TypeError):
        env._env_index([0.5])
    env._check_geometry(_Cfg(19, 2, 2, 0))
    for other in (_Cfg(10, 2, 2, 0), _Cfg(19, 3, 2, 0), _Cfg(19, 2, 1, 0), _Cfg(19, 2, 2, 2)):
        with pytest.raises(ValueError):
            env._check_geometry(other)
