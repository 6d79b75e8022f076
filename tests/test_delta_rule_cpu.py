"""CPU: the sector rules of the lane family's delta store (delta_store in snk_lane.cuh), restated in numpy over whole oracle
bodies and checked on C oracle trajectories: the 32-byte sectors a rule stores must cover every byte that differs between
consecutive frames.  This checks the rules, not the kernel: delta_store's own index arithmetic (the k / d offsets, the
fruit pick, the `shifted` test on chain codes) is held to whole-image stores bit for bit by tests/test_gpu_delta.py and
tests/test_gpu_delta_split.py.

The rule stores the sectors of the paint items whose pixel can change: a fruit whose cell changed (new and old cell); for
a snake that moved (new segment i + 1 = old segment i for i < k = min(old length, new length - 1)) its new segments 0 and
1, new segments past k and old segments from k on; every old and new segment of any other snake.  The rule it replaced
(`old_rule`: every new fruit and every new segment) is counted beside it.  An env goes out as sectors only when every old
and new body has at most 17 segments (DELTA_MAX_LEN); the others go out whole and are not counted.

    PYTHONPATH=oracle:tests python tests/test_delta_rule_cpu.py    # sectors per env-step of both rules, headline board
"""
import numpy as np
import pytest

import c_oracle
import scripted_ref

MAX_LEN = 17


def _items(st0, st1, S, F, old_rule):
    """Padded cell ids of the paint items the rule stores, [N][M] with -1 for none, and the envs that qualify."""
    l0, l1 = st0["len"].astype(np.int64), st1["len"].astype(np.int64)
    b0, b1 = st0["body"][:, :, :MAX_LEN + 1].astype(np.int64), st1["body"][:, :, :MAX_LEN + 1].astype(np.int64)
    f0, f1 = st0["fruit"][:, :F].astype(np.int64), st1["fruit"][:, :F].astype(np.int64)
    N = l0.shape[0]
    ok = ((l0 <= MAX_LEN) & (l1 <= MAX_LEN)).all(axis=1)
    moved = f0 != f1
    cols = [np.where(moved, f1, -1) if not old_rule else f1, np.where(moved, f0, -1)]
    seg = np.arange(MAX_LEN)
    for s in range(S):
        k = np.maximum(np.minimum(l0[:, s], l1[:, s] - 1), 0)
        # matched segments: new i + 1 = old i for every i < k
        same = (b1[:, s, 1:MAX_LEN + 1] == b0[:, s, :MAX_LEN]) | (seg[None, :] >= k[:, None])
        k = np.where(same.all(axis=1), k, 0)
        new_keep = seg[None, :] < l1[:, s, None]
        if not old_rule:
            new_keep &= (seg[None, :] < 2) | (seg[None, :] > k[:, None])
        old_keep = (seg[None, :] < l0[:, s, None]) & (seg[None, :] >= k[:, None])
        cols += [np.where(new_keep, b1[:, s, :MAX_LEN], -1), np.where(old_keep, b0[:, s, :MAX_LEN], -1)]
    return np.concatenate(cols, axis=1).reshape(N, -1), ok


def sectors(st0, st1, S, F, V, C, old_rule=False):
    """(emitted [N][n] bool over each env's sectors, stores per env): the 32-byte sectors of the own buffer (envs of
    V*V*C bytes back to back from a 32-byte-aligned start) that the rule stores, counted as distinct sectors and as the
    one or two store instructions per item."""
    E = V * V * C
    pid, ok = _items(st0, st1, S, F, old_rule)
    N = pid.shape[0]
    e = np.broadcast_to(np.arange(N)[:, None], pid.shape)
    first = (np.arange(N) * E) >> 5
    off = e * E + pid * C
    s0, s1 = (off >> 5) - first[:, None], ((off + C - 1) >> 5) - first[:, None]
    live = pid >= 0
    emitted = np.zeros((N, E // 32 + 2), dtype=bool)
    emitted[e[live], s0[live]] = True
    emitted[e[live], s1[live]] = True
    stores = live.sum(axis=1) + (live & (s1 != s0)).sum(axis=1)
    return emitted, stores, ok


def changed(obs0, obs1, E):
    """[N][n] bool: the sectors of each env holding a byte that differs between the two frames."""
    N = obs0.shape[0]
    d = (obs0.reshape(N, E) != obs1.reshape(N, E))
    e, byte = np.nonzero(d)
    out = np.zeros((N, E // 32 + 2), dtype=bool)
    out[e, ((e * E + byte) >> 5) - ((e * E) >> 5)] = True
    return out


def _actions(co, t, seed, mix):
    """Random actions, or (mix) the fruit-seeking policy on two steps of three, as tests/test_gpu_delta.py drives them."""
    if mix and t % 3:
        return scripted_ref.scripted_actions(co.state(), co.cfg, t, seed, 200, 0)
    return c_oracle.gen_actions(co.cfg, t, seed)


def run(N, size, S, F, steps, mix, seed=3, max_steps=2000):
    """Checks coverage on every env-step that qualifies; returns the per-env-step means (changed, new rule distinct,
    new rule stores, old rule distinct, old rule stores) and the share of env-steps that qualify."""
    co = c_oracle.COracle(N, size=size, n_snakes=S, n_fruits=F, seed=seed, max_steps=max_steps)
    V, C = size + 2, 3 * S
    E = V * V * C
    obs0 = co.reset().copy()
    st0 = co.state()
    st0 = {k: v.copy() for k, v in st0.items()}
    tot = np.zeros(5)
    n_ok = 0
    for t in range(steps):
        co.step(_actions(co, t, seed, mix))
        obs1 = co.obs.copy()
        st1 = {k: v.copy() for k, v in co.state().items()}
        em, stores, ok = sectors(st0, st1, S, F, V, C)
        em_old, stores_old, _ = sectors(st0, st1, S, F, V, C, old_rule=True)
        ch = changed(obs0, obs1, E)
        missed = ch & ~em & ok[:, None]
        assert not missed.any(), "step %d: env %d has a changed sector the rule does not store" % (t, np.nonzero(missed)[0][0])
        assert not (em & ~em_old).any(), "the new rule stores a sector the old one did not"
        tot += [ch[ok].sum(), em[ok].sum(), stores[ok].sum(), em_old[ok].sum(), stores_old[ok].sum()]
        n_ok += int(ok.sum())
        obs0, st0 = obs1, st1
    return tot / max(n_ok, 1), n_ok / float(N * steps)


@pytest.mark.parametrize("size", [10, 19])
@pytest.mark.parametrize("S", [1, 2, 3, 4])
@pytest.mark.parametrize("F", [1, 2, 3, 4])
def test_rule_covers_every_changed_byte(size, S, F):
    # short episodes on the small board so that time-limit resets happen too, beside deaths and respawns
    means, share = run(192, size, S, F, 90, mix=(S + F) % 2 == 0, seed=S + 5 * F, max_steps=40 if size == 10 else 2000)
    assert share > 0.5
    print("%dx%d S=%d F=%d: changed %.2f, stored %.2f distinct / %.2f stores, old rule %.2f / %.2f" % ((size, size, S, F) + tuple(means)))


def test_headline_counts():
    """2 snakes on 19x19, random actions: the new rule stores fewer sectors than the old one."""
    means, _ = run(1024, 19, 2, 2, 60, mix=False)
    assert means[2] < means[4]


if __name__ == "__main__":
    print("sectors per env-step that qualifies (bodies <= 17 segments), C oracle trajectories, 2048 envs x 200 steps")
    print("%-34s %8s %8s %8s %8s %8s %7s" % ("", "changed", "new", "new", "old", "old", "share"))
    print("%-34s %8s %8s %8s %8s %8s %7s" % ("", "sectors", "distinct", "stores", "distinct", "stores", ""))
    for name, mix in (("2x19x19 random actions", False), ("2x19x19 fruit-seeking mix (eps .2)", True)):
        m, share = run(2048, 19, 2, 2, 200, mix=mix)
        print("%-34s %8.2f %8.2f %8.2f %8.2f %8.2f %7.3f" % ((name,) + tuple(m) + (share,)))
