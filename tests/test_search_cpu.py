"""CPU: the rollout-search rule (include/snk.h snk_search_*, snakes_b200/search.py) on hand-built reward and done
streams through the numpy reference (tests/search_ref.py), and the argument checks of the C entry points and of
snk_clone_envs that run before any CUDA call.  No GPU work."""
import ctypes as C
import os

import numpy as np
import pytest

import search_ref as ref


@pytest.fixture(scope="module")
def L():
    import __graft_entry__ as ge
    if not os.path.exists(ge.LIB):
        ge.build()
    from snakes_b200 import _lib
    return _lib


def stream(H, N, S):
    return np.zeros((H, N, S), np.float32), np.zeros((H, N), np.uint8)


def test_slot_numbering():
    M, A, R = 3, 6, 4
    seen = []
    for m in range(M):
        for a in range(A):
            for r in range(R):
                j = (m * A + a) * R + r
                assert ref.slot(m, a, r, A, R) == j
                assert ref.candidate(j, A, R) == a and j // (A * R) == m
                seen.append(j)
    assert seen == list(range(M * A * R))
    acts = np.full((M * A * R + 5, 2), 7, np.int8)
    ret, active = ref.begin(acts, 1, M, A, R)
    assert (acts[:M * A * R, 1] == np.repeat(np.tile(np.arange(A), M), R)).all()
    assert (acts[:, 0] == 7).all() and (acts[M * A * R:, 1] == 7).all()   # other seats and slots beyond M A R untouched
    assert (ret == 0).all() and active.all()


def test_death_on_step_zero_counts_minus_one_and_nothing_after():
    M, A, R, S = 1, 2, 1, 2
    rew, done = stream(4, 2, S)
    rew[0, 0, 1] = -1            # slot 0 (a = 0): seat 1 dies on the first step
    rew[1:, 0, 1] = 5            # never counted (a dead seat gets 0 anyway; the rule stops counting)
    rew[:, 1, 1] = 1             # slot 1 (a = 1) eats every step
    V, a = ref.search(rew, done, 1, M, A, R)
    assert V.tolist() == [[-1.0, 4.0]] and a.tolist() == [1]


def test_done_partway_ends_the_slot():
    M, A, R, S = 1, 2, 2, 1
    rew, done = stream(6, 4, S)
    rew[:, :, 0] = 1
    done[2, 0] = 1               # slot 0 counts steps 0, 1, 2
    done[4, 3] = 1               # slot 3 counts steps 0 .. 4
    V, a = ref.search(rew, done, 0, M, A, R)
    assert V.tolist() == [[3.0 + 6.0, 6.0 + 5.0]] and a.tolist() == [1]


def test_stacked_fruit_reward_above_one():
    M, A, R, S = 1, 3, 1, 2
    rew, done = stream(2, 3, S)
    rew[0, 2, 0] = 3             # three fruits on one cell (adversarial / cut)
    rew[1, 1, 0] = 2
    V, a = ref.search(rew, done, 0, M, A, R)
    assert V.tolist() == [[0.0, 2.0, 3.0]] and a.tolist() == [2]


def test_tie_goes_to_the_lowest_action():
    M, A, R, S = 2, 5, 2, 2
    rew, done = stream(3, M * A * R, S)
    for m in range(M):
        for a in (1, 3):
            rew[0, ref.slot(m, a, 0, A, R), 0] = 1
    V, a = ref.search(rew, done, 0, M, A, R)
    assert a.tolist() == [1, 1]


def test_dead_seat_gives_action_zero():
    """A seat dead at the root gets reward 0 on every step of every slot: every V is 0 and the pick is action 0."""
    M, A, R, S = 3, 6, 2, 3
    rew, done = stream(8, M * A * R, S)
    rew[:, :, 0] = np.random.RandomState(1).randint(-1, 3, size=(8, M * A * R))   # the other seats do not matter
    done[5] = 1
    V, a = ref.search(rew, done, 2, M, A, R)
    assert (V == 0).all() and (a == 0).all()


def test_slots_beyond_the_roots_are_not_counted():
    M, A, R, S = 1, 2, 1, 1
    rew, done = stream(2, 6, S)
    rew[:, 2:, 0] = 9
    V, _ = ref.search(rew, done, 0, M, A, R)
    assert V.tolist() == [[0.0, 0.0]]


def test_search_rejects_bad_arguments(L):
    lib = L.lib()
    n = C.c_void_p(16)   # never dereferenced: every call below fails its checks first
    assert lib.snk_search_begin(None, n, 0, 5, 8, 1, n, n, None) == -1 and "NULL" in lib.snk_last_error().decode()
    assert lib.snk_search_accumulate(None, 0, 5, 8, 1, n, n, None) == -1
    assert lib.snk_search_pick(None, 5, 8, 1, n, n, n, 1, None) == -1
    assert lib.snk_clone_envs(None, n, None, n, 1, None) == -1 and "NULL" in lib.snk_last_error().decode()

