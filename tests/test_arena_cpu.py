"""CPU: the outcome rule of snk_tally (include/snk.h) on hand-built reward / done streams through the numpy reference
(tests/arena_ref.py), the arena's block partition and seat rotation, and snk_tally's argument checks.  No GPU work."""
import ctypes as C
import os

import numpy as np
import pytest

import arena_ref as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def L():
    import __graft_entry__ as ge
    if not os.path.exists(ge.LIB):
        ge.build()
    from snakes_b200 import _lib
    return _lib


def run(stream, S, group=None, n_groups=1, E=1):
    """stream: list of (reward_all [N][S], done [N]) per step, or ([S], scalar) for one env; the episode length is
    counted here as the handle counts it."""
    N = np.atleast_1d(stream[0][1]).shape[0]
    ref = R.TallyRef(np.zeros(N, int) if group is None else group, n_groups, S, E)
    ep = np.zeros(N, int)
    for rew, done in stream:
        done = np.atleast_1d(np.asarray(done, np.uint8))
        ep += 1
        ref.step(np.asarray(rew, np.float32).reshape(N, S), done, np.where(done, ep, 0))
        ep[done.astype(bool)] = 0
    return ref


def row(counts, s):
    return dict(zip(R.FIELDS, counts[0, s].tolist()))


def test_fields_match_header(L):
    header = open(os.path.join(ROOT, "include", "snk.h")).read()
    for i, name in enumerate(R.FIELDS):
        assert "#define SNK_TALLY_%s %d" % (name.upper(), i) in header
    assert "#define SNK_TALLY_FIELDS %d" % len(R.FIELDS) in header
    assert L.TALLY_FIELDS == R.FIELDS


def test_seat1_dies_first_then_seat0():
    ref = run([([1, 0], 0), ([0, -1], 0), ([2, 0], 0), ([-1, 0], 1)], 2)
    s0, s1 = row(ref.counts, 0), row(ref.counts, 1)
    assert (s0["wins"], s0["draws"], s0["losses"]) == (1, 0, 0)
    assert (s1["wins"], s1["draws"], s1["losses"]) == (0, 0, 1)
    assert s0["fruits"] == 3 and s0["deaths"] == 1 and s0["steps_alive"] == 4 and s0["return_sq"] == 4 and s0["length"] == 4
    assert s1["fruits"] == 0 and s1["deaths"] == 1 and s1["steps_alive"] == 2 and s1["return_sq"] == 1 and s1["length"] == 4


def test_seat0_dies_while_seat1_alive():
    ref = run([([0, 1], 0), ([-1, 1], 1)], 2)
    s0, s1 = row(ref.counts, 0), row(ref.counts, 1)
    assert (s0["wins"], s0["losses"], s1["wins"], s1["losses"]) == (0, 1, 1, 0)
    assert s1["deaths"] == 0 and s1["steps_alive"] == 2 and s1["return_sq"] == 4 and s0["steps_alive"] == 2


def test_simultaneous_deaths_draw():
    ref = run([([0, 0], 0), ([-1, -1], 1)], 2)
    assert row(ref.counts, 0)["draws"] == row(ref.counts, 1)["draws"] == 1
    assert row(ref.counts, 0)["wins"] == row(ref.counts, 1)["losses"] == 0


def test_timeout_both_alive_draws():
    ref = run([([0, 1], 0), ([1, 0], 0), ([0, 0], 1)], 2)
    s0, s1 = row(ref.counts, 0), row(ref.counts, 1)
    assert s0["draws"] == s1["draws"] == 1 and s0["deaths"] == s1["deaths"] == 0
    assert s0["steps_alive"] == s1["steps_alive"] == 3 and s0["return_sq"] == s1["return_sq"] == 1


def test_timeout_after_one_seat_died():
    ref = run([([0, -1], 0), ([1, 0], 0), ([0, 0], 1)], 2)
    s0, s1 = row(ref.counts, 0), row(ref.counts, 1)
    assert s0["wins"] == 1 and s1["losses"] == 1 and s1["steps_alive"] == 1 and s0["steps_alive"] == 3


def test_three_seats_tie_for_last_place():
    # seats 1 and 2 die on step 2, seat 0 survives to the timeout: 0 wins, 1 and 2 both lose
    ref = run([([0, 0, 0], 0), ([0, -1, -1], 0), ([0, 0, 0], 1)], 3)
    assert [row(ref.counts, s)["wins"] for s in range(3)] == [1, 0, 0]
    assert [row(ref.counts, s)["losses"] for s in range(3)] == [0, 1, 1]
    # and a tie for the longest life: seats 0 and 2 alive at the timeout draw, seat 1 loses
    ref = run([([0, -1, 0], 0), ([0, 0, 0], 1)], 3)
    assert [row(ref.counts, s)["draws"] for s in range(3)] == [1, 0, 1]
    assert row(ref.counts, 1)["losses"] == 1


def test_single_seat_always_wins():
    ref = run([([1], 0), ([-1], 1), ([0], 0), ([0], 1)], 1, E=2)
    s0 = row(ref.counts, 0)
    assert s0["wins"] == 2 and s0["draws"] == s0["losses"] == 0
    assert s0["fruits"] == 1 and s0["deaths"] == 1 and s0["steps_alive"] == 4 and s0["return_sq"] == 0 + 0


def test_multi_fruit_steps():
    ref = run([([3, 2], 0), ([1, 0], 0), ([0, -1], 0), ([0, 0], 1)], 2)
    s0, s1 = row(ref.counts, 0), row(ref.counts, 1)
    assert s0["fruits"] == 4 and s0["return_sq"] == 16
    assert s1["fruits"] == 2 and s1["return_sq"] == 1


def test_episodes_after_the_last_are_ignored():
    # env 0 finishes 2 episodes by step 2; its third episode is not counted.  Env 1 finishes one (E = 2: not done).
    stream = [([[-1, 0], [0, 0]], [1, 0]), ([[0, -1], [0, 0]], [1, 0]), ([[5, 0], [0, -1]], [0, 0]),
              ([[-1, 0], [-1, 0]], [1, 1])]
    ref = run(stream, 2, group=np.array([0, 1]), n_groups=2, E=2)
    assert ref.envs_done == 1
    assert ref.counts[0, :, :3].sum() == 4            # two episodes x two seats
    assert ref.counts[0, 0, R.FR] == 0                # the 5 fruits of env 0's third episode are ignored
    assert row(ref.counts[1:], 1)["wins"] == 0 and ref.counts[1, 0, R.W] == 1
    ref.step(np.array([[0, 0], [-1, 0]], np.float32), np.array([0, 1]), np.array([0, 1]))
    assert ref.envs_done == 2


def test_bad_group_is_skipped():
    ref = run([([[-1, 0], [-1, 0]], [1, 1])], 2, group=np.array([0, 3]), n_groups=2)
    assert ref.bad_group and ref.envs_done == 1 and ref.counts[1].sum() == 0


@pytest.mark.parametrize("N,M,S", [(2, 1, 2), (131072, 1, 2), (65537, 3, 3), (1000, 7, 2), (33, 1, 16), (5, 5, 1)])
def test_blocks_partition_and_rotation(L, N, M, S):
    from snakes_b200 import arena
    lay = arena.blocks(N, M, S)
    assert len(lay) == M * S
    assert lay[0][2] == 0 and lay[-1][3] == N
    assert all(a[3] == b[2] for a, b in zip(lay, lay[1:]))
    sizes = [b1 - b0 for _, _, b0, b1 in lay]
    assert max(sizes) - min(sizes) <= 1 and min(sizes) >= 1
    assert [(m, r) for m, r, _, _ in lay] == [(m, r) for m in range(M) for r in range(S)]
    for m in range(M):
        for i in range(S):
            per_seat = np.zeros(S, int)
            for mm, r, b0, b1 in lay:
                if mm == m:
                    per_seat[arena.seat_of(i, r, S)] += b1 - b0
            assert per_seat.min() >= 1 and per_seat.max() - per_seat.min() <= 1
        # in every rotation block the players hold distinct seats
        for r in range(S):
            assert sorted(arena.seat_of(i, r, S) for i in range(S)) == list(range(S))


def test_blocks_reject_too_few_envs(L):
    from snakes_b200 import arena
    with pytest.raises(ValueError):
        arena.blocks(3, 2, 2)
    with pytest.raises(ValueError):
        arena.blocks(10, 0, 2)


def test_tally_rejects_bad_arguments(L):
    lib = L.lib()
    size = (C.c_size_t * 2)()
    assert lib.snk_tally_layout(None, size) == -1
    ok = dict(group=0x1000, work=0x2000, counts=0x3000, done=0x4000)

    def call(h=None, group=ok["group"], n_groups=1, E=1, work=ok["work"], counts=ok["counts"], done=ok["done"]):
        v = lambda x: C.c_void_p(x) if x else None
        return lib.snk_tally(h, v(group), n_groups, E, v(work), v(counts), v(done), None), lib.snk_last_error().decode()

    assert call(n_groups=0) == (-1, "n_groups must be >= 1, got 0")
    assert call(E=0) == (-1, "episodes_per_env must be >= 1, got 0")
    for k in ("group", "work", "counts", "done"):
        assert call(**{k: 0}) == (-1, "NULL argument")
    assert call(group=0x1002)[1] == "d_group must be 4-byte aligned"
    assert call(work=0x2008)[1] == "d_work must be 16-byte aligned"
    assert call(counts=0x3004)[1].startswith("d_counts and d_envs_done")
    assert call(done=0x4004)[1].startswith("d_counts and d_envs_done")
    assert call() == (-1, "handle is NULL")   # every other argument checked first, nothing dereferenced
