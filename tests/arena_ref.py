"""numpy restatement of snk_tally (include/snk.h, snakes_b200/csrc/snk_arena.cu): the reference the kernel is checked
against bit for bit.  Written from the outcome rule, not from the kernel: the death step of every seat is kept per env,
and at the end of an episode every seat's outcome is decided by comparing it with every other seat."""
import numpy as np

FIELDS = ("wins", "draws", "losses", "fruits", "deaths", "steps_alive", "return_sq", "length")
W, D, LOSS, FR, DE, SA, RSQ, LEN = range(len(FIELDS))
INF = np.iinfo(np.int64).max


def outcome(d):
    """Outcome index (W, D or LOSS) of every seat for death steps d [..., S] (INF: alive at the end), straight from the
    rule: s wins if d_s > d_j for every j != s, draws if d_s >= d_j for every j and d_s == d_j for some j != s."""
    d = np.asarray(d, dtype=np.int64)
    S = d.shape[-1]
    other = ~np.eye(S, dtype=bool)                       # [s, j]: j != s
    gt = (d[..., :, None] > d[..., None, :]) | ~other    # vacuous for j == s
    ge = (d[..., :, None] >= d[..., None, :]) | ~other
    eq = (d[..., :, None] == d[..., None, :]) & other
    win, draw = gt.all(-1), ge.all(-1) & eq.any(-1)
    return np.where(win, W, np.where(draw, D, LOSS))


class TallyRef:
    """Feeds one step's reward_all [N, S], done [N], episode_len [N] at a time, as the kernel sees them."""

    def __init__(self, group, n_groups, S, episodes_per_env):
        self.group = np.asarray(group, dtype=np.int64)
        N = len(self.group)
        self.S, self.E = S, episodes_per_env
        self.t = np.zeros(N, np.int64)
        self.death = np.zeros((N, S), np.int64)   # 0 = alive
        self.fruits = np.zeros((N, S), np.int64)
        self.episodes = np.zeros(N, np.int64)
        self.active = np.ones(N, bool)
        self.counts = np.zeros((n_groups, S, len(FIELDS)), np.int64)
        self.bad_group = False

    @property
    def envs_done(self):
        return int((self.episodes >= self.E).sum())

    def step(self, reward_all, done, ep_len):
        r = np.asarray(reward_all, dtype=np.float32).reshape(len(self.t), self.S)
        done = np.asarray(done).astype(bool)
        ep_len = np.asarray(ep_len, dtype=np.int64)
        a = self.active
        self.t[a] += 1
        dies = a[:, None] & (r < 0)
        self.death[dies] = np.broadcast_to(self.t[:, None], dies.shape)[dies]
        eats = a[:, None] & (r > 0)
        self.fruits[eats] += r[eats].astype(np.int64)
        fin = a & done
        bad = fin & ((self.group < 0) | (self.group >= len(self.counts)))
        if bad.any():
            self.bad_group = True
            self.active[bad] = False
        e = np.nonzero(fin & ~bad)[0]
        if len(e):
            g, death, fruits = self.group[e], self.death[e], self.fruits[e]
            died = death > 0
            o = outcome(np.where(died, death, INF))                  # [n, S]
            ret = fruits - died
            L = np.broadcast_to(ep_len[e][:, None], died.shape)
            per = np.zeros(died.shape + (len(FIELDS),), np.int64)   # [n, S, fields]
            np.put_along_axis(per, o[..., None], 1, axis=-1)
            per[..., FR], per[..., DE] = fruits, died
            per[..., SA] = np.where(died, death, L)
            per[..., RSQ], per[..., LEN] = ret * ret, L
            np.add.at(self.counts, g, per)
            self.death[e] = 0
            self.fruits[e] = 0
            self.t[e] = 0
            self.episodes[e] += 1
            self.active[e[self.episodes[e] >= self.E]] = False
