"""numpy restatement of the rollout-search bookkeeping (snk_search_begin / _accumulate / _pick of include/snk.h,
snakes_b200/csrc/snk_search.cu): the reference the kernels are checked against bit for bit.  Written from the rule:
slot j = (m A + a) R + r plays candidate a = (j / R) % A, its return is seat's reward summed up to and including the step
on which the seat gets -1 or the env is done, and root m takes the lowest a of maximal V[m][a]."""
import numpy as np


def slot(m, a, r, A, R):
    return (m * A + a) * R + r


def candidate(j, A, R):
    return (np.asarray(j) // R) % A


def begin(actions, seat, M, A, R):
    """Seat's action of slots [0, M A R) of `actions` [N, S] <- their candidate; returns (ret, active) of those slots."""
    n = M * A * R
    actions[:n, seat] = candidate(np.arange(n), A, R)
    return np.zeros(n, np.int32), np.ones(n, bool)


def accumulate(ret, active, reward_all, done, seat):
    """One step's reward_all [N, S] and done [N] into (ret, active) in place."""
    n = len(ret)
    v = np.asarray(reward_all, np.float32)[:n, seat]
    ret[active] += v[active].astype(np.int32)
    active &= ~((v < 0) | np.asarray(done, bool)[:n])


def pick(ret, M, A, R):
    """(V float32 [M, A], action int8 [M]): the lowest a of maximal V[m][a]."""
    V = ret[:M * A * R].astype(np.int64).reshape(M, A, R).sum(-1)
    best = V.max(1, keepdims=True)
    return V.astype(np.float32), np.argmax(V == best, axis=1).astype(np.int8)


def search(rewards, dones, seat, M, A, R):
    """The whole bookkeeping over H steps: rewards [H, N, S], dones [H, N] -> (V, action)."""
    ret, active = np.zeros(M * A * R, np.int32), np.ones(M * A * R, bool)
    for rew, done in zip(rewards, dones):
        accumulate(ret, active, rew, done, seat)
    return pick(ret, M, A, R)
