"""CPU: the reference of the scripted fruit-seeking policy (tests/scripted_ref.py) on hand-built states, one per clause of
its contract (snk_gen_scripted_actions, include/snk.h), and its vectorised draw against oracle/snake_oracle.py's scalar one.
tests/test_gpu_scripted.py holds the kernel to the same cases."""
import numpy as np
import pytest

import scripted_ref as ref
import snake_oracle as so

# name -> (size, n_snakes, n_fruits, snakes (board (x, y), head first), velocity codes, fruits (board (x, y)), actions)
# Actions: 1 +x, 2 +y, 3 -x, 4 -y.  Every expected action is worked out by hand in the comment beside it.
CASES = {
    # reversal: the fruit lies just behind a one-cell snake; the reversing action is dropped, the other three tie at 2
    "reverse_vel1": (5, 1, 1, [[(2, 2)]], [1], [(1, 2)], [1]),
    "reverse_vel2": (5, 1, 1, [[(2, 2)]], [2], [(2, 1)], [1]),
    "reverse_vel3": (5, 1, 1, [[(2, 2)]], [3], [(3, 2)], [2]),
    "reverse_vel4": (5, 1, 1, [[(2, 2)]], [4], [(2, 3)], [1]),
    "no_velocity": (5, 1, 1, [[(2, 2)]], [0], [(1, 2)], [3]),          # not moving yet: nothing is a reversal
    # a head on every edge and in every corner, its fruit on the border cell beyond it (distance 0, but a wall);
    # the cells left on the board tie at 2
    "edge_x0": (5, 1, 1, [[(0, 2)]], [0], [(-1, 2)], [1]),
    "edge_x4": (5, 1, 1, [[(4, 2)]], [0], [(5, 2)], [2]),
    "edge_y0": (5, 1, 1, [[(2, 0)]], [0], [(2, -1)], [1]),
    "edge_y4": (5, 1, 1, [[(2, 4)]], [0], [(2, 5)], [1]),
    "corner_00": (5, 1, 1, [[(0, 0)]], [0], [(-1, 0)], [1]),
    "corner_04": (5, 1, 1, [[(0, 4)]], [0], [(-1, 4)], [1]),
    "corner_40": (5, 1, 1, [[(4, 0)]], [0], [(5, 0)], [2]),
    "corner_44": (5, 1, 1, [[(4, 4)]], [0], [(5, 4)], [3]),
    # +x is the snake's own tail (d 2); +y is its neck; -x and -y tie at 4
    "own_tail": (5, 1, 1, [[(1, 1), (1, 2), (2, 2), (2, 1)]], [4], [(4, 1)], [3]),
    # snake 0's +x is snake 1's head, then its tail: -x, +y, -y tie at 3; snake 1 goes for the fruit
    "other_head": (5, 2, 1, [[(2, 2)], [(3, 2)]], [0, 0], [(4, 2)], [2, 1]),
    "other_tail": (5, 2, 1, [[(2, 2)], [(3, 3), (3, 2)]], [0, 2], [(4, 2)], [2, 1]),
    # two-way ties of every pair that includes the winner, and a four-way tie over four fruits
    "tie_1_2": (5, 1, 1, [[(2, 2)]], [0], [(4, 4)], [1]),
    "tie_2_3": (5, 1, 1, [[(2, 2)]], [0], [(0, 4)], [2]),
    "tie_3_4": (5, 1, 1, [[(2, 2)]], [0], [(0, 0)], [3]),
    "tie_1_4": (5, 1, 1, [[(2, 2)]], [0], [(4, 0)], [1]),
    "tie_four_way": (5, 1, 4, [[(2, 2)]], [0], [(0, 2), (4, 2), (2, 0), (2, 4)], [1]),
    "tie_four_way_reversal": (5, 1, 4, [[(2, 2)]], [3], [(0, 2), (4, 2), (2, 0), (2, 4)], [2]),
    # F = 4: the nearest fruit is the last one (d 1 from +y; every other candidate is 3 from its nearest)
    "f4_last_fruit": (5, 1, 4, [[(2, 2)]], [0], [(0, 0), (0, 4), (4, 0), (2, 4)], [2]),
    # F = 0: every distance is the same, so the lowest candidate that is left wins
    "f0_free": (5, 1, 0, [[(2, 2)]], [0], [], [1]),
    "f0_reversal": (5, 1, 0, [[(2, 2)]], [3], [], [2]),
    "f0_blocked": (5, 2, 0, [[(2, 2)], [(3, 2)]], [0, 0], [], [2, 1]),
    # every candidate dropped: action 0.  A 3x3 board filled by one snake (its fruit has no free cell, so it is parked
    # at (0, 0), under the body), and a corner head boxed in by the other snake
    "all_blocked_full": (3, 1, 1, [[(1, 1), (1, 0), (0, 0), (0, 1), (0, 2), (1, 2), (2, 2), (2, 1), (2, 0)]], [2], [(0, 0)], [0]),
    "all_blocked_corner": (5, 2, 1, [[(0, 0)], [(1, 0), (1, 1), (0, 1)]], [0, 4], [(4, 4)], [0, 1]),
    # one free cell left, the fruit still parked at (0, 0) under the tail: the only move is -y
    "parked_fruit": (3, 1, 1, [[(2, 1), (2, 2), (1, 2), (0, 2), (0, 1), (1, 1), (1, 0), (0, 0)]], [4], [(0, 0)], [4]),
    # a dead snake gets 0
    "dead": (5, 2, 1, [[(2, 2)], []], [0, 0], [(2, 4)], [2, 0]),
    # fruits off the board (a restored state may hold any padded id): distances are measured to them all the same
    "fruit_on_border": (5, 1, 1, [[(1, 2)]], [0], [(-1, 2)], [3]),
    "fruit_padded_0": (5, 1, 1, [[(2, 0)]], [0], [(-1, -1)], [3]),
    "fruit_padded_last": (5, 1, 1, [[(4, 3)]], [0], [(5, 5)], [2]),
}


def case_groups():
    """Cases grouped by geometry (size, n_snakes, n_fruits) -> [names]."""
    groups = {}
    for name, c in sorted(CASES.items()):
        groups.setdefault(c[:3], []).append(name)
    return groups


def empty_state(N, size, S, F):
    cap = (size * size + 1 + 7) & ~7
    return {"len": np.zeros((N, S), np.uint16), "grow_to": np.zeros((N, S), np.uint16), "vel": np.zeros((N, S), np.uint8),
            "body": np.zeros((N, S, cap), np.uint16), "fruit": np.zeros((N, F), np.uint16)}


class Cfg(object):
    def __init__(self, size, n_snakes, n_fruits):
        self.size, self.n_snakes, self.n_fruits = size, n_snakes, n_fruits


@pytest.mark.parametrize("name", sorted(CASES))
def test_hand_built_state(name):
    size, S, F, snakes, vels, fruits, want = CASES[name]
    st = empty_state(1, size, S, F)
    ref.fill_state(st, 0, size, snakes, vels, fruits)
    got = ref.scripted_actions(st, Cfg(size, S, F), step=3, seed=1, eps_permille=0, env_id_base=0)
    assert got.tolist() == [want], (name, got.tolist(), want)


def test_cases_in_one_batch():
    """The cases of one geometry side by side in one batch give each its own answer (nothing leaks between envs)."""
    for (size, S, F), names in case_groups().items():
        st = empty_state(len(names), size, S, F)
        for e, n in enumerate(names):
            ref.fill_state(st, e, *((size,) + CASES[n][3:6]))
        got = ref.scripted_actions(st, Cfg(size, S, F), step=0, seed=5, eps_permille=0, env_id_base=77)
        assert got.tolist() == [CASES[n][6] for n in names], names


def _scalar_draws(seed, ids, index):
    return np.array([so.philox_bounded(seed, int(i), 2, index, 5000) for i in ids], dtype=np.int64)


@pytest.mark.parametrize("eps", [0, 1, 999, 1000])
def test_eps_permille(eps):
    """rnd // 5 < eps picks rnd % 5, else the greedy action; a dead snake gets 0 whatever the draw.  eps 1 and 999 each
    take both branches over these 20 000 envs."""
    N, base, step, seed = 20000, 1000, 41, 9
    st = empty_state(N, 5, 2, 1)
    for e in range(N):
        ref.fill_state(st, e, 5, [[(2, 2)], []], [0, 0], [(0, 4)])   # greedy: 2 (tie_2_3)
    got = ref.scripted_actions(st, Cfg(5, 2, 1), step, seed, eps, base)
    rnd = _scalar_draws(seed, np.arange(base, base + N), step * 2)
    rand = rnd // 5 < eps
    assert np.array_equal(got[:, 0], np.where(rand, rnd % 5, 2))
    assert not got[:, 1].any()
    n_rand = int(rand.sum())
    assert n_rand == 0 if eps == 0 else n_rand == N if eps == 1000 else 0 < n_rand < N, n_rand


U64 = (1 << 64) - 1


@pytest.mark.parametrize("seed", [0, 7, (1 << 32) - 1, 1 << 32, (1 << 32) + 12345, (1 << 63) + 3, U64])
def test_draw_equals_scalar_oracle(seed):
    """The vectorised draw is snake_oracle.philox_bounded: indices across the 2^32 word split of the block counter and
    past 2^34 (block counter above 2^32), seeds whose high word feeds the counter, env ids up to 2^32 - 1, every stream."""
    ids = np.array([0, 1, 2, 77, (1 << 31) + 5, (1 << 32) - 1], dtype=np.uint64)
    for index in (0, 1, 2, 3, 4, 5, (1 << 32) - 2, (1 << 32) - 1, 1 << 32, (1 << 32) + 1, (1 << 34) - 1, 1 << 34,
                  (1 << 34) + 6, (1 << 63) + 1, U64):
        for stream in (0, 1, 2):
            for n in (5, 6, 5000):
                got = ref.philox_bounded(seed, ids, stream, index, n)
                want = [so.philox_bounded(seed, int(i), stream, index, n) for i in ids]
                assert got.tolist() == want, (seed, index, stream, n)


@pytest.mark.parametrize("S,step,seed", [(3, (1 << 32) // 3, 5),               # step*S + s: 2^32 - 1, 2^32, 2^32 + 1
                                         (2, (1 << 33) - 1, (1 << 32) + 9),    # the block counter index >> 2 reaches 2^31
                                         (1, (1 << 34) + 2, (1 << 40) + 1),    # block counter above 2^32
                                         (2, U64, U64)])                        # step * S wraps modulo 2^64
def test_counter_and_key_split(S, step, seed):
    """At eps 1000 every live snake's action is the draw itself: (seed, env_id_base + e, 2, step * S + s mod 2^64) % 5."""
    N, base = 64, (1 << 32) - 64
    st = empty_state(N, 5, S, S)
    for e in range(N):
        ref.fill_state(st, e, 5, [[(s, 0)] for s in range(S)], [0] * S, [(4, 4)] * S)
    got = ref.scripted_actions(st, Cfg(5, S, S), step, seed, 1000, base)
    for s in range(S):
        rnd = _scalar_draws(seed, np.arange(base, base + N), (step * S + s) & U64)
        assert np.array_equal(got[:, s], rnd % 5), s
