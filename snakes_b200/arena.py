"""Head-to-head evaluation of policies on the device: the reference's evaluate_snake.py (two checkpoints in one env on the
host) played over a whole batch of envs at once, with per-seat win / draw / loss and score accounting (snk_tally of
include/snk.h; DESIGN.md section 4.18).

The seats are not symmetric: an episode ends when seat 0 dies or at max_steps, so a snake in seat 0 keeps eating after
its opponents die and one in another seat never gets that time.  `play` therefore splits the envs into one contiguous
block per (match, rotation) and plays every rotation of every match: in block (m, r) player i of match m sits in seat
(i + r) mod S.  Every env counts exactly `episodes` episodes (the kernel ignores an env once it has), so short episodes
are not over-weighted.
"""
import ctypes as C
import math

import numpy as np
import torch

from . import _lib, search

PLAYER_KINDS = ("scripted", "random")


class Search(object):
    """A rollout-search player (search.RolloutSearch): for every env of its block and its seat, each candidate action is
    played from `rollouts` clones of the env, followed by `horizon` steps of the `rollout` policy ('scripted' with
    `eps`, or 'random') keyed by `seed`, and the action of the largest summed return is taken.  It needs no training,
    and with random rollouts it plays every rule-set and every step family."""

    def __init__(self, rollouts=8, horizon=16, rollout="scripted", eps=0.05, seed=1):
        self.rollouts, self.horizon, self.rollout, self.eps, self.seed = int(rollouts), int(horizon), rollout, float(eps), int(seed)

    def __repr__(self):
        return "Search(rollouts=%d, horizon=%d, rollout=%r, eps=%g, seed=%d)" % (
            self.rollouts, self.horizon, self.rollout, self.eps, self.seed)
POLL_STEPS = 32   # steps between two reads of the finished-env counter (one 8-byte copy)


def blocks(N, n_matches, S):
    """[(m, r, b0, b1)] in block order b = m * S + r: len(matches) x S contiguous blocks covering [0, N) whose sizes
    differ by at most one.  ValueError when N < n_matches * S."""
    B = n_matches * S
    if B < 1 or N < B:
        raise ValueError("%d envs cannot hold %d matches x %d seat rotations" % (N, n_matches, S))
    base, extra = divmod(N, B)
    out, b0 = [], 0
    for b in range(B):
        b1 = b0 + base + (b < extra)
        out.append((b // S, b % S, b0, b1))
        b0 = b1
    return out


def seat_of(player, rotation, S):
    """The seat player `player` of a match takes in rotation `rotation`."""
    return (player + rotation) % S


def _net(player):
    return getattr(player, "net", player)


def _check_player(env, p):
    """ValueError for a player that cannot play on this env."""
    if isinstance(p, str):
        if p not in PLAYER_KINDS:
            raise ValueError("a player is a model (anything with .step(ob, view)), 'scripted' or 'random', got %r" % p)
        if p == "scripted" and (env.cfg.rules != _lib.RULES["classic"] or env.launch_info()["kind"] != 0):
            raise ValueError("'scripted' needs a lane-family env with classic rules (snk_gen_scripted_actions)")
        return
    if isinstance(p, Search):
        search.check_args(env, p.rollouts, p.horizon, p.rollout)
        return
    if not callable(getattr(p, "step", None)):
        raise ValueError("a player is a model (anything with .step(ob, view)), 'scripted' or 'random', got %r" % (p,))
    net = _net(p)
    grid = bool(getattr(net, "grid", False))
    if grid != (env.obs_mode == "grid"):
        raise ValueError("an obs_mode %r env needs %s models" % (env.obs_mode, "grid" if env.obs_mode == "grid" else "RGB"))
    n_act = getattr(net, "n_actions", None)
    if n_act is not None and n_act != env.action_space.n:
        raise ValueError("the model has %d actions, the env %d" % (n_act, env.action_space.n))
    shape = getattr(net, "ob_shape", None)
    want = (env.V, env.V, 3) if grid else tuple(env.obs.shape[1:3]) + (3,)
    if shape is not None and tuple(shape) != want:
        raise ValueError("the model reads observations of shape %r, the env gives %r" % (tuple(shape), want))


def _summary(c):
    """Per-player figures from counts [..., fields] summed over the player's seats."""
    f = dict(zip(_lib.TALLY_FIELDS, (int(x) for x in c)))
    n = f["wins"] + f["draws"] + f["losses"]
    ret_sum = f["fruits"] - f["deaths"]
    mean = ret_sum / n if n else float("nan")
    var = (f["return_sq"] - n * mean * mean) / (n - 1) if n > 1 else float("nan")
    return dict(episodes=n, wins=f["wins"], draws=f["draws"], losses=f["losses"],
                score=(f["wins"] + 0.5 * f["draws"]) / n if n else float("nan"),
                return_mean=mean, return_se=math.sqrt(max(var, 0.0) / n) if n > 1 else float("nan"),
                fruits_per_episode=f["fruits"] / n if n else float("nan"),
                death_rate=f["deaths"] / n if n else float("nan"),
                steps_alive=f["steps_alive"] / n if n else float("nan"))


def play(env, matches, episodes=1, seed=1, eps=0.05):
    """Plays every match of `matches` (a list of tuples of env.S players) on `env`, `episodes` episodes per env, in every
    seat rotation.  A player is a model (anything whose .step(ob, view) returns the actions first: selfplay.Model or
    CnnPolicy, grid models on an obs_mode 'grid' env, RGB models otherwise), 'scripted' (the device's fruit-seeking
    policy, gen_scripted_actions with `eps`; lane-family classic envs only), 'random' (gen_actions) or a Search (rollout
    search: one search.RolloutSearch per Search object of the call, sized to the largest block, acts for each of its
    (block, seat) pairs on that block's envs before every step).  `seed` keys the scripted and random action streams.  The env is reset first and must auto-reset and keep its observations on the
    device; an RGB env needs one view per seat (n_views >= S).

    Returns one record per match: {'players': [per-player dict of episodes, wins, draws, losses, score = (wins +
    draws / 2) / episodes, return_mean, return_se (standard error of the mean), fruits_per_episode, death_rate,
    steps_alive (mean, counting the death step)] summed over the player's seat in every rotation, 'counts': int64
    [S rotations][S seats][fields] (fields _lib.TALLY_FIELDS), 'episode_len': the mean episode length, 'envs': envs per
    rotation block, 'steps': steps played}.  Two calls on fresh envs of the same seed, after the same torch.manual_seed,
    give identical records (a reset continues an env's random stream, so a second call on the same env plays other
    games)."""
    S, N = env.S, env.N
    matches = [tuple(m) for m in matches]
    if env.host_io:
        raise ValueError("the arena keeps observations on the device: the env needs host_io=False")
    if not env.cfg.auto_reset:
        raise ValueError("the arena needs an env that auto-resets")
    if int(episodes) < 1:
        raise ValueError("episodes must be >= 1")
    if env.obs_mode != "grid" and env.K < S:
        raise ValueError("an RGB env needs one view per seat (n_views >= n_snakes), got %d < %d" % (env.K, S))
    for m in matches:
        if len(m) != S:
            raise ValueError("a match holds env.S = %d players, got %d" % (S, len(m)))
        for p in m:
            _check_player(env, p)
    layout = blocks(N, len(matches), S)
    dev = env.device
    n_groups = len(layout)
    group = torch.empty(N, dtype=torch.int32, device=dev)
    for b, (_, _, b0, b1) in enumerate(layout):
        group[b0:b1] = b
    L = _lib.lib()
    out = (C.c_size_t * 2)()
    _lib.check(L.snk_tally_layout(env._h, out))
    F = int(out[1])
    work = torch.zeros(-(-int(out[0]) // 16) * 4, dtype=torch.int32, device=dev)
    counts = torch.zeros((n_groups, S, F), dtype=torch.int64, device=dev)
    envs_done = torch.zeros(1, dtype=torch.int64, device=dev)

    # per (block, seat): who acts there; a model plays a block's seat with one forward call on that block
    kinds = sorted({p for m in matches for p in m if isinstance(p, str)})
    from_kind = {k: torch.zeros((N, S), dtype=torch.bool, device=dev) for k in kinds}
    model_calls, search_calls = [], []
    for m, r, b0, b1 in layout:
        for i, p in enumerate(matches[m]):
            s = seat_of(i, r, S)
            if isinstance(p, str):
                from_kind[p][b0:b1, s] = True
            elif isinstance(p, Search):
                search_calls.append((p, b0, b1, s, torch.arange(b0, b1, dtype=torch.int64, device=dev)))
            else:
                model_calls.append((p, b0, b1, s))
    scratch = {k: torch.empty((N, S), dtype=torch.int8, device=dev) for k in kinds}
    actions = torch.zeros((N, S), dtype=torch.int8, device=dev)
    grid = env.obs_mode == "grid"
    largest = max(b1 - b0 for _, _, b0, b1 in layout)
    searchers = {}
    for p, _, _, _, _ in search_calls:
        if p not in searchers:
            searchers[p] = search.RolloutSearch(env, largest, p.rollouts, p.horizon, p.rollout, p.eps, p.seed)

    env.reset()
    stream = env._stream()
    args = (C.c_void_p(group.data_ptr()), n_groups, int(episodes), C.c_void_p(work.data_ptr()),
            C.c_void_p(counts.data_ptr()), C.c_void_p(envs_done.data_ptr()))
    limit = int(episodes) * (env.cfg.max_steps or 2000) + POLL_STEPS   # every episode ends by max_steps
    t = 0
    while True:
        obs = env.obs
        for p, b0, b1, s in model_calls:
            ob = obs[b0:b1] if grid else obs[b0:b1, ..., 3 * s:3 * s + 3]
            actions[b0:b1, s] = p.step(ob, s)[0].to(torch.int8)
        for p, b0, b1, s, roots in search_calls:
            searchers[p].act(s, roots, out=actions[b0:b1, s])
        if "scripted" in kinds:
            env.gen_scripted_actions(t, seed, eps, out=scratch["scripted"])
        if "random" in kinds:
            env.gen_actions(t, seed, out=scratch["random"])
        for k in kinds:
            torch.where(from_kind[k], scratch[k], actions, out=actions)
        env.step(actions)
        _lib.check(L.snk_tally(env._h, *args, stream))
        t += 1
        if t % POLL_STEPS == 0:
            if int(envs_done.item()) == N:
                break
            if t > limit:
                raise RuntimeError("%d of %d envs finished %d episodes in %d steps" % (int(envs_done.item()), N, episodes, t))
    env.check_errors()
    for rs in searchers.values():
        rs.search_env.check_errors()
        rs.close()
    c = counts.cpu().numpy().reshape(len(matches), S, S, F)
    records = []
    for m, match in enumerate(matches):
        cm = c[m]
        players = [_summary(sum(cm[r, seat_of(i, r, S)] for r in range(S))) for i in range(len(match))]
        n_ep = int(cm[:, 0, :3].sum())
        records.append(dict(players=players, counts=cm.copy(),
                            episode_len=float(cm[:, 0, _lib.TALLY_FIELDS.index("length")].sum()) / n_ep,
                            envs=[b1 - b0 for mm, _, b0, b1 in layout if mm == m], steps=t))
    return records


def round_robin(env, players, episodes=1, seed=1, eps=0.05):
    """Every unordered pair of `players` as one `play` call on a two-seat env (both seat orders).  Returns (records,
    score) with records[(i, j)] the match record of players[i] against players[j] (i < j) and score [P][P] the score
    of player i against player j (score[j][i] = 1 - score[i][j]; NaN on the diagonal): the table that ranks a pool of
    checkpoints."""
    if env.S != 2:
        raise ValueError("round_robin plays pairs: it needs a two-seat env, got S = %d" % env.S)
    P = len(players)
    score = np.full((P, P), np.nan)
    records = {}
    for i in range(P):
        for j in range(i + 1, P):
            rec = play(env, [(players[i], players[j])], episodes, seed, eps)[0]
            records[(i, j)] = rec
            score[i, j], score[j, i] = rec["players"][0]["score"], rec["players"][1]["score"]
    return records, score
