"""GPU: the arena (snakes_b200.arena, snk_tally of include/snk.h).

- k_tally against the numpy reference tests/arena_ref.py bit for bit (counters and finished-env count), on live steps of
  both step families, every rule-set, S = 1..16, few and many groups (the shared-memory and the global-memory counters),
  E = 1, 2, 3 and N past the first wave of CTAs.
- Exact invariants of `play`, the scripted policy against random play, grid against native envs, model players (both
  observation modes, reproducibility, checkpoints) and the arguments `play` rejects."""
import ctypes as C

import numpy as np
import pytest
import torch

import arena_ref as R

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def sb():
    import snakes_b200
    return snakes_b200


class Tally:
    """snk_tally on an env with caller-owned work area and counters."""

    def __init__(self, env, group, n_groups, E):
        from snakes_b200 import _lib
        self.env, self.L, self.n_groups, self.E = env, _lib.lib(), n_groups, E
        out = (C.c_size_t * 2)()
        _lib.check(self.L.snk_tally_layout(env._h, out))
        self.work = torch.zeros(-(-int(out[0]) // 4), dtype=torch.int32, device=env.device)
        self.counts = torch.zeros((n_groups, env.S, int(out[1])), dtype=torch.int64, device=env.device)
        self.envs_done = torch.zeros(1, dtype=torch.int64, device=env.device)
        self.group = torch.as_tensor(group, dtype=torch.int32, device=env.device)
        self._lib = _lib

    def __call__(self):
        p = lambda t: C.c_void_p(t.data_ptr())
        self._lib.check(self.L.snk_tally(self.env._h, p(self.group), self.n_groups, self.E, p(self.work), p(self.counts),
                                         p(self.envs_done), self.env._stream()))


# (name, rules, S, size, N, E, n_groups, max_steps, scripted share)
CASES = [
    ("classic_2x19_131072", "classic", 2, 19, 131072, 2, 5, 150, True),
    ("cut_3x10_65536", "cut", 3, 10, 65536, 1, 3, 100, False),
    ("adversarial_3x10", "adversarial", 3, 10, 4096, 3, 2, 30, False),
    ("ring_cut_16x64", "cut", 16, 64, 300, 1, 4, 200, False),
    ("classic_2x10_37_groups", "classic", 2, 10, 20000, 1, 37, 80, True),
    ("classic_2x10_global_counters", "classic", 2, 10, 8192, 1, 400, 60, False),
    ("classic_1x10", "classic", 1, 10, 2048, 2, 1, 50, True),
]


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_tally_matches_reference(sb, case):
    name, rules, S, size, N, E, G, max_steps, scripted = case
    env = sb.SnakeVecEnv(N, size=size, n_snakes=S, rules=rules, max_steps=max_steps, seed=11)
    if name.startswith("ring"):
        assert env.launch_info()["kind"] != 0
    elif scripted:
        assert env.launch_info()["kind"] == 0
    rng = np.random.default_rng(5)
    group = rng.integers(0, G, N) if G > 1 else np.zeros(N, int)
    if G > 1:
        group[:G] = np.arange(G)   # every group present; sizes are uneven
    tal = Tally(env, group, G, E)
    ref = R.TallyRef(group, G, S, E)
    env.reset()
    rnd = torch.empty((N, S), dtype=torch.int8, device=env.device)
    scr = torch.empty_like(rnd)
    half = (torch.arange(N, device=env.device) % 2 == 0)[:, None]
    t, extra, limit = 0, 0, E * max_steps + 10
    while extra < 5:
        a = env.gen_actions(t, 3, out=rnd)
        if scripted:
            a = torch.where(half, env.gen_scripted_actions(t, 3, 0.05, out=scr), a)
        env.step(a)
        tal()
        ref.step(env.rewards_all.cpu().numpy(), env._done_u8.cpu().numpy(), env.episode_len.cpu().numpy())
        t += 1
        if t % 25 == 0:
            assert int(tal.envs_done.item()) == ref.envs_done, "finished count differs at step %d" % t
        extra += ref.envs_done == N
        assert t <= limit
    env.check_errors()
    got = tal.counts.cpu().numpy()
    assert int(tal.envs_done.item()) == N == ref.envs_done
    np.testing.assert_array_equal(got, ref.counts)
    assert got[..., :3].sum() == N * E * S
    assert (got[..., R.LEN].sum(1) == S * got[:, 0, R.LEN]).all()
    print("%s: %d steps, %d episodes, %d wins / %d draws / %d losses" % (name, t, N * E, got[..., 0].sum(), got[..., 1].sum(),
                                                                        got[..., 2].sum()))
    env.close()


def test_tally_flags_a_bad_group(sb):
    N = 1024
    env = sb.SnakeVecEnv(N, size=10, n_snakes=2, seed=2)
    group = np.zeros(N, int)
    group[7] = 2
    tal = Tally(env, group, 2, 1)
    env.reset()
    for t in range(400):
        env.step(env.gen_actions(t, 1))
        tal()
    flags = C.c_uint32(0)
    from snakes_b200 import _lib
    _lib.check(_lib.lib().snk_check_errors(env._h, C.byref(flags), env._stream()))
    assert flags.value == 16
    assert int(tal.envs_done.item()) == N - 1
    assert tal.counts[0, :, :3].sum().item() == 2 * (N - 1) and tal.counts[1].sum().item() == 0
    env.close()


def _rec_equal(a, b):
    assert len(a) == len(b)
    for x, y in zip(a, b):
        np.testing.assert_array_equal(x["counts"], y["counts"])
        assert x["players"] == y["players"] and x["episode_len"] == y["episode_len"]


def test_play_invariants(sb):
    env = sb.SnakeVecEnv(4099, size=10, n_snakes=2, max_steps=100, seed=4)
    E = 2
    rec, = sb.arena.play(env, [("scripted", "random")], episodes=E, seed=9)
    a, b = rec["players"]
    assert a["wins"] == b["losses"] and a["losses"] == b["wins"] and a["draws"] == b["draws"]
    assert a["episodes"] == b["episodes"] == 4099 * E
    assert a["score"] + b["score"] == pytest.approx(1.0)
    c = rec["counts"]
    for r in range(2):
        assert (c[r, :, :3].sum(-1) == rec["envs"][r] * E).all()
    assert sorted(rec["envs"]) == [2049, 2050]
    env.close()


def test_scripted_beats_random(sb):
    """Scripted against random on 2x19x19 classic, 16 384 envs, 2 episodes each.  Measured on one NVIDIA B200 (1 000 W):
    the scripted player scores 0.939 (30 095 wins, 1 338 draws, 1 335 losses of 32 768 episodes); the bound leaves a
    wide margin."""
    env = sb.SnakeVecEnv(16384, size=19, n_snakes=2, seed=1)
    rec, = sb.arena.play(env, [("scripted", "random")], episodes=2, seed=3)
    s, r = rec["players"]
    print("scripted vs random:", s, r, "episode_len %.2f" % rec["episode_len"])
    assert s["score"] > 0.8 and s["fruits_per_episode"] > r["fruits_per_episode"]
    env.close()


def test_grid_and_native_give_the_same_records(sb):
    recs = []
    for mode in ("native", "grid"):
        env = sb.SnakeVecEnv(4096, size=19, n_snakes=2, max_steps=300, seed=21, obs_mode=mode)
        recs.append(sb.arena.play(env, [("scripted", "random"), ("random", "scripted")], episodes=2, seed=5))
        env.close()
    _rec_equal(*recs)


def _models(sb, env, grid, n=2):
    from snakes_b200.selfplay import Model
    torch.manual_seed(1234)
    shape = (env.V, env.V, 3) if grid else tuple(env.obs.shape[1:3]) + (3,)
    return [Model(shape, env.action_space.n, device=env.device, trainable=False, grid=grid) for _ in range(n)]


@pytest.mark.parametrize("mode", ["grid", "native"])
def test_model_players(sb, tmp_path, mode):
    """Records depend on the env seed and the torch seed alone: each play runs on a fresh env of the same seed (a reset
    continues an env's random stream, so a second play on the same env meets other fruit)."""
    from snakes_b200.selfplay import Model
    grid = mode == "grid"

    def fresh():
        return sb.SnakeVecEnv(2048, size=10, n_snakes=2, max_steps=200, seed=8, obs_mode=mode)

    def run(matches, **kw):
        env = fresh()
        torch.manual_seed(7)
        out = sb.arena.play(env, matches, episodes=1, seed=2, **kw)
        env.close()
        return out

    env = fresh()
    A, B = _models(sb, env, grid)
    env.close()
    first = run([(A, B), (A, "random")])
    _rec_equal(first, run([(A, B), (A, "random")]))
    a, b = first[0]["players"]
    assert a["wins"] == b["losses"] and a["episodes"] == b["episodes"] == 2048 // 2
    # a checkpoint written by Model.save and read by Model.load plays the same games as the live model
    path = str(tmp_path / "a.joblib")
    A.save(path)
    A2 = Model(A.net.ob_shape, A.net.n_actions, device=A.net.pi.weight.device, trainable=False, grid=grid)
    A2.load(path)
    _rec_equal(first, run([(A2, B), (A2, "random")]))
    # round robin over three players: one play per pair, scores mirror
    env = fresh()
    records, score = sb.arena.round_robin(env, [A, B, "random"], episodes=1, seed=2)
    assert sorted(records) == [(0, 1), (0, 2), (1, 2)]
    assert np.isnan(np.diag(score)).all()
    off = ~np.eye(3, dtype=bool)
    assert np.allclose((score + score.T)[off], 1.0)
    env.close()


def test_play_rejects_bad_arguments(sb):
    from snakes_b200.selfplay import Model
    adv = sb.SnakeVecEnv(64, size=10, n_snakes=2, rules="adversarial", seed=1)
    with pytest.raises(ValueError, match="scripted"):
        sb.arena.play(adv, [("scripted", "random")])
    adv.close()
    grid = sb.SnakeVecEnv(64, size=10, n_snakes=2, seed=1, obs_mode="grid")
    rgb_model = Model((12, 12, 3), 5, device=grid.device, trainable=False)
    with pytest.raises(ValueError, match="grid"):
        sb.arena.play(grid, [(rgb_model, "random")])
    with pytest.raises(ValueError, match="players"):
        sb.arena.play(grid, [("random", "random", "random")])
    with pytest.raises(ValueError, match="actions"):
        sb.arena.play(grid, [(Model((12, 12, 3), 6, device=grid.device, trainable=False, grid=True), "random")])
    with pytest.raises(ValueError, match="envs"):
        sb.arena.play(grid, [("random", "random")] * 40)
    with pytest.raises(ValueError):
        sb.arena.play(grid, [("random", "greedy")])
    grid.close()
    host = sb.SnakeVecEnv(64, size=10, n_snakes=2, seed=1, host_io=True)
    with pytest.raises(ValueError, match="host_io"):
        sb.arena.play(host, [("random", "random")])
    host.close()
    few_views = sb.SnakeVecEnv(64, size=10, n_snakes=2, n_views=1, seed=1)
    with pytest.raises(ValueError, match="view"):
        sb.arena.play(few_views, [("random", "random")])
    few_views.close()
    three = sb.SnakeVecEnv(64, size=10, n_snakes=3, seed=1)
    with pytest.raises(ValueError, match="two-seat"):
        sb.arena.round_robin(three, ["random", "random"])
    three.close()
