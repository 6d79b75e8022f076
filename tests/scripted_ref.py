"""Reference for the scripted fruit-seeking policy (snk_gen_scripted_actions, include/snk.h), restated from its contract
in numpy and vectorised over envs.  TEST INFRASTRUCTURE ONLY.

Per env e and snake s of the state at the time of the call:
  1. a dead snake (len 0) gets action 0;
  2. rnd = draw (seed, env_id_base + e, stream 2, index step * S + s) mapped to [0, 5000); if rnd // 5 < eps_permille
     the action is rnd % 5;
  3. otherwise action a = 1..4 proposes the cell head + (+V, +1, -V, -1)[a - 1] (velocity codes: 1 +x, 2 +y, 3 -x, 4 -y),
     dropped when a reverses the stored velocity, when the cell is on the border of the padded V x V grid, or when any
     segment of any snake (tails included) lies on it;
  4. a candidate's distance is the least Manhattan distance, in padded coordinates (x = id // V, y = id % V), to the
     first F fruits (with F = 0 all distances are equal);
  5. the action is the lowest a of strictly smallest distance, or 0 when every candidate is dropped.
The draw is oracle/snake_oracle.py:philox_bounded (Philox4x32-10, hi32(u32 * n)), here for an array of env ids."""
import numpy as np

_M0, _M1, _W0, _W1 = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85
_U32 = np.uint64(0xFFFFFFFF)
_MASK64 = (1 << 64) - 1
STREAM_ACTIONS, STREAM_SCRIPTED = 1, 2


def philox_bounded(seed, env_ids, stream, index, n):
    """Draw `index` of (seed, env id, stream) bounded to [0, n), for every env id of the array `env_ids` (uint64 result).
    Counter (index >> 2 low, high, stream, seed >> 32), key (seed low, env id); word index & 3 of the block."""
    seed, index = int(seed) & _MASK64, int(index) & _MASK64
    ids = np.asarray(env_ids, dtype=np.uint64)
    blk = index >> 2
    c0 = np.full(ids.shape, blk & 0xFFFFFFFF, dtype=np.uint64)
    c1 = np.full(ids.shape, blk >> 32, dtype=np.uint64)
    c2 = np.full(ids.shape, int(stream) & 0xFFFFFFFF, dtype=np.uint64)
    c3 = np.full(ids.shape, seed >> 32, dtype=np.uint64)
    k0 = np.full(ids.shape, seed & 0xFFFFFFFF, dtype=np.uint64)
    k1 = ids & _U32
    for _ in range(10):
        p0 = np.uint64(_M0) * c0
        p1 = np.uint64(_M1) * c2
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & _U32, (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & _U32
        k0 = (k0 + np.uint64(_W0)) & _U32
        k1 = (k1 + np.uint64(_W1)) & _U32
    x = (c0, c1, c2, c3)[index & 3]
    return (x * np.uint64(n)) >> np.uint64(32)


def scripted_actions(state, cfg, step, seed, eps_permille, env_id_base):
    """int8 [N][S]: the policy's actions for the canonical state `state` (split_state of a dump: `len`, `vel`, `body`,
    classic `fruit`) of a configuration with cfg.size, cfg.n_snakes, cfg.n_fruits."""
    S, F, V = int(cfg.n_snakes), int(cfg.n_fruits), int(cfg.size) + 2
    length = state["len"].astype(np.int64)                      # [N][S]
    vel = state["vel"].astype(np.int64)                         # [N][S]
    body = state["body"].astype(np.int64)                       # [N][S][cap], head first
    N, cap = body.shape[0], body.shape[2]
    env = np.arange(N, dtype=np.int64)

    # every segment of every snake, tails included
    occ = np.zeros((N, V * V), dtype=bool)
    seg = np.arange(cap)[None, None, :] < length[:, :, None]
    e_idx = np.broadcast_to(env[:, None, None], body.shape)
    occ[e_idx[seg], body[seg]] = True

    head = body[:, :, 0]
    cx0, cy0 = head // V, head % V
    big = np.iinfo(np.int64).max
    dist = np.empty((N, S, 4), dtype=np.int64)
    for a in range(1, 5):
        dx, dy = ((1, 0), (0, 1), (-1, 0), (0, -1))[a - 1]
        cx, cy = cx0 + dx, cy0 + dy
        reverse = (vel != 0) & (a == ((vel + 1) & 3) + 1)
        border = (cx <= 0) | (cx >= V - 1) | (cy <= 0) | (cy >= V - 1)
        cell = np.clip(cx * V + cy, 0, V * V - 1)
        taken = occ[env[:, None], cell]
        if F:
            fruit = state["fruit"][:, :F].astype(np.int64)      # [N][F]
            fx, fy = fruit // V, fruit % V
            d = (np.abs(cx[:, :, None] - fx[:, None, :]) + np.abs(cy[:, :, None] - fy[:, None, :])).min(axis=2)
        else:
            d = np.zeros((N, S), dtype=np.int64)
        dist[:, :, a - 1] = np.where(reverse | border | taken, big, d)
    best = dist.argmin(axis=2)                                  # the first (lowest a) of the smallest distances
    greedy = np.where(dist[env[:, None], np.arange(S)[None, :], best] == big, 0, best + 1)

    out = np.empty((N, S), dtype=np.int64)
    ids = np.arange(N, dtype=np.uint64) + np.uint64(int(env_id_base))
    for s in range(S):
        rnd = philox_bounded(seed, ids, STREAM_SCRIPTED, int(step) * S + s, 5000).astype(np.int64)
        out[:, s] = np.where(rnd // 5 < int(eps_permille), rnd % 5, greedy[:, s])
    out[length == 0] = 0
    return out.astype(np.int8)


def fill_state(st, e, size, snakes, vels, fruits):
    """Writes env e of the split_state arrays `st` from board coordinates: snakes[s] a list of (x, y) head first, vels[s]
    a velocity code, fruits[f] an (x, y) -- x or y of -1 or `size` is a cell of the border.  grow_to = len + 2, t = 0."""
    V = size + 2
    pid = lambda c: (c[0] + 1) * V + (c[1] + 1)
    for s, b in enumerate(snakes):
        st["len"][e, s] = len(b)
        st["body"][e, s, :] = 0
        st["body"][e, s, :len(b)] = [pid(c) for c in b]
        st["grow_to"][e, s] = len(b) + 2
        st["vel"][e, s] = vels[s]
    st["fruit"][e, :] = [pid(c) for c in fruits]
