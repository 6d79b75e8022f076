"""GPU: obs_mode 'grid' (SNK_OBS_GRID).  Twin handles -- native and grid, same configuration, seed and actions -- step in
lockstep, and every step expand_views(grid.obs, K) equals the native obs bit for bit; rewards, dones, num_snakes and
Monitor's r / l are equal, and so are the state dumps.  Lane family (k_lane_logic + k_lane_grid) and ring family (the rows
kernel's grid form, for every geometry the native path puts on tile, dense or rows)."""
import numpy as np
import pytest

import helpers

pytestmark = pytest.mark.gpu

# name -> (constructor kwargs, num_envs, native kernel kind: 0 lane, 1 tile, 2 dense, 3 rows).  The grid handle is on
# the lane family whenever S, F <= 4 and size <= 32, whatever K is, and on the rows kernel's grid form otherwise.
CASES = {
    "lane_classic_2x19": (dict(size=19, n_snakes=2, rules="classic"), 2048, 0),
    "lane_classic_2x10_k3": (dict(size=10, n_snakes=2, n_views=3, rules="classic"), 1024, 0),
    "dense_native_classic_2x19_k3": (dict(size=19, n_snakes=2, n_views=3, rules="classic"), 1024, 2),
    "lane_classic_1x10": (dict(size=10, n_snakes=1, rules="classic"), 600, 0),
    "lane_cut_3x10": (dict(size=10, n_snakes=3, rules="cut"), 1000, 0),
    "lane_adversarial_3x10": (dict(size=10, n_snakes=3, rules="adversarial"), 1000, 0),
    "lane_classic_4x12": (dict(size=12, n_snakes=4, rules="classic"), 700, 0),
    "lane_ragged_1003": (dict(size=10, n_snakes=2, rules="classic"), 1003, 0),
    "tile_classic_6x12": (dict(size=12, n_snakes=6, rules="classic"), 300, 1),
    "dense_adversarial_5x41": (dict(size=41, n_snakes=5, rules="adversarial"), 40, 2),
    "rows_cut_16x64": (dict(size=64, n_snakes=16, rules="cut"), 24, 3),
}


@pytest.fixture(scope="module")
def sb():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import snakes_b200
    return snakes_b200


def _twins(sb, case, seed=3, **extra):
    kw, N, kind = CASES[case]
    kw = dict(kw, **extra)
    nat = sb.SnakeVecEnv(N, seed=seed, **kw)
    grd = sb.SnakeVecEnv(N, seed=seed, obs_mode="grid", **kw)
    assert nat.launch_info()["kind"] == kind, nat.launch_info()
    lane = kw["n_snakes"] <= 4 and kw.get("n_fruits", kw["n_snakes"]) <= 4 and kw["size"] <= 32
    want = "k_lane_logic + k_lane_grid" if lane else "k_step_rows (grid)"
    assert grd.launch_info()["kernel"] == want, grd.launch_info()
    assert tuple(grd.obs.shape) == (N, grd.V, grd.V) and grd.observation_space.shape == (grd.V, grd.V)
    return nat, grd


def _actions(env, t, rng):
    import torch
    a = rng.randint(0, env.action_space.n, size=(env.N, env.S)).astype(np.int8)
    a[rng.rand(env.N, env.S) < 0.5] = 0   # mostly straight on: bodies survive a while
    return torch.as_tensor(a, device=env.device)


def _same_obs(sb, nat, grd, where):
    import torch
    got = sb.expand_views(grd.obs, grd.K)
    if not torch.equal(got, nat.obs):
        bad = (got != nat.obs).reshape(nat.N, -1).any(1).nonzero().flatten()[:5].tolist()
        raise AssertionError("%s: expanded grid differs from the native obs in envs %s" % (where, bad))


def _same_step(nat, grd, r, where):
    import torch
    (_, rn, dn, infn), (_, rg, dg, infg) = r
    assert torch.equal(rn, rg) and torch.equal(dn, dg), where
    assert torch.equal(nat.num_alive, grd.num_alive), where
    d = dn.bool()
    assert torch.equal(nat.episode_return[d], grd.episode_return[d]) and torch.equal(nat.episode_len[d], grd.episode_len[d]), where


def _same_state(nat, grd, where):
    a, b = nat.dump_state(), grd.dump_state()
    for k in a:
        assert np.array_equal(a[k], b[k]), (where, k)


def _lockstep(sb, nat, grd, steps, rng, state_every=16):
    for t in range(steps):
        a = _actions(nat, t, rng)
        r = (nat.step(a), grd.step(a))
        _same_step(nat, grd, r, t)
        _same_obs(sb, nat, grd, "step %d" % t)
        if t % state_every == 0 or t == steps - 1:
            _same_state(nat, grd, t)
    nat.check_errors(); grd.check_errors()


@pytest.mark.parametrize("case", sorted(CASES))
def test_grid_twin_lockstep(sb, case):
    import torch
    nat, grd = _twins(sb, case)
    rng = np.random.RandomState(7)
    nat.reset(); grd.reset()
    _same_obs(sb, nat, grd, "reset")
    _lockstep(sb, nat, grd, 60, rng)
    # long bodies (multi-word chain codes; ring wrap-around once stepped), loaded into both and re-encoded
    blob = helpers.random_long_snake_states(nat.lay, nat.cfg, np.random.RandomState(5))
    for e in (nat, grd):
        e.load_state_blob(blob)
        e.reset(mask=torch.zeros(e.N, dtype=torch.bool, device=e.device))
    _same_obs(sb, nat, grd, "load")
    _lockstep(sb, nat, grd, 24, rng, state_every=8)
    # a masked reset
    m = torch.as_tensor(rng.rand(nat.N) < 0.3, device=nat.device)
    nat.reset(mask=m); grd.reset(mask=m)
    _same_obs(sb, nat, grd, "masked reset")
    _same_state(nat, grd, "masked reset")
    nat.close(); grd.close()


def test_grid_headline_shard(sb):
    """131 072 envs of 2 snakes on 19x19: a few steps of the full-size shard."""
    import torch
    nat = sb.SnakeVecEnv(131072, size=19, n_snakes=2, seed=0)
    grd = sb.SnakeVecEnv(131072, size=19, n_snakes=2, seed=0, obs_mode="grid")
    assert grd.launch_info()["kernel"] == "k_lane_logic + k_lane_grid"
    nat.reset(); grd.reset()
    _same_obs(sb, nat, grd, "reset")
    for t in range(6):
        a = nat.gen_actions(t, 1).clone()
        r = (nat.step(a), grd.step(a))
        _same_step(nat, grd, r, t)
        _same_obs(sb, nat, grd, "step %d" % t)
    assert torch.equal(sb.expand_views(grd.obs[:7], 1, first_view=1), nat.obs[:7, ..., 3:6])
    nat.close(); grd.close()


def test_grid_scripted_long_bodies(sb):
    """The fruit-seeking policy (bodies over 17 segments: more than one chain word) gives the same actions on both twins,
    although the native handle reads occupancy from its image and the grid handle walks the bodies; then the scripted
    graph on both."""
    import torch
    nat = sb.SnakeVecEnv(4096, size=19, n_snakes=2, seed=5)
    grd = sb.SnakeVecEnv(4096, size=19, n_snakes=2, seed=5, obs_mode="grid")
    nat.reset(); grd.reset()
    longest = 0
    for t in range(400):
        an = nat.gen_scripted_actions(t, seed=2, eps=0.02).clone()
        ag = grd.gen_scripted_actions(t, seed=2, eps=0.02).clone()
        assert torch.equal(an, ag), t
        r = (nat.step(an), grd.step(ag))
        _same_step(nat, grd, r, t)
        if t % 25 == 0 or t > 380:
            _same_obs(sb, nat, grd, "scripted step %d" % t)
            longest = max(longest, int(grd.dump_state()["len"].max()))
    assert longest > 17, longest
    _same_state(nat, grd, "scripted")
    gn, gg = nat.make_scripted_graph(50, step0=400, seed=2, eps=0.02), grd.make_scripted_graph(50, step0=400, seed=2, eps=0.02)
    gn.launch(); gg.launch()
    torch.cuda.synchronize()
    _same_obs(sb, nat, grd, "scripted graph")
    _same_state(nat, grd, "scripted graph")
    gn.close(); gg.close()
    nat.close(); grd.close()


def test_grid_rollout_equals_eager(sb):
    """A graph rollout writes [T, N, V, V]; every slot expands to the native obs of the same eager step."""
    import torch
    kw = dict(size=10, n_snakes=3, rules="cut")
    nat = sb.SnakeVecEnv(777, seed=9, **kw)
    grd = sb.SnakeVecEnv(777, seed=9, obs_mode="grid", **kw)
    nat.reset(); grd.reset()
    rng = np.random.RandomState(1)
    T = 12
    acts = torch.stack([_actions(nat, t, rng) for t in range(T)])
    obs, rew, done = grd.rollout(acts)
    assert tuple(obs.shape) == (T, 777, 12, 12)
    for t in range(T):
        _, rn, dn, _ = nat.step(acts[t])
        assert torch.equal(sb.expand_views(obs[t], grd.K), nat.obs), t
        assert torch.equal(rew[t], rn) and torch.equal(done[t], dn), t
    assert torch.equal(sb.expand_views(obs, grd.K)[T - 1], nat.obs)  # a [T, N, V, V] batch at once
    _same_state(nat, grd, "rollout")
    nat.close(); grd.close()


def test_grid_host_io_equals_device(sb):
    import torch
    dev = sb.SnakeVecEnv(513, size=19, n_snakes=2, seed=4, obs_mode="grid")
    host = sb.SnakeVecEnv(513, size=19, n_snakes=2, seed=4, obs_mode="grid", host_io=True)
    assert host.observation_space.shape == (21, 21)
    o0 = host.reset()
    assert isinstance(o0, np.ndarray) and o0.shape == (513, 21, 21)
    assert np.array_equal(o0, dev.reset().cpu().numpy())
    for t in range(20):
        a = dev.gen_actions(t, 1).clone()
        ho, hr, hd, _ = host.step(a.cpu().numpy())
        do, dr, dd, _ = dev.step(a)
        assert np.array_equal(ho, do.cpu().numpy()) and np.array_equal(hr, dr.cpu().numpy().astype(np.float64)), t
        assert np.array_equal(hd, dd.cpu().numpy()), t
    with pytest.raises(ValueError):
        sb.SnakeVecEnv(8, size=10, n_snakes=2, obs_mode="grid", host_io=True, host_views=1)
    with pytest.raises(ValueError):
        dev.set_main_view_target(torch.empty((513, 21, 21, 3), dtype=torch.uint8, device=dev.device))
    dev.close(); host.close()


def test_grid_restore_copy_observe(sb):
    import torch
    nat, grd = _twins(sb, "lane_classic_2x19")
    nat.reset(); grd.reset()
    rng = np.random.RandomState(2)
    _lockstep(sb, nat, grd, 10, rng, state_every=100)
    saved = (nat.save_envs([1, 2, 3]), grd.save_envs([1, 2, 3]))
    _lockstep(sb, nat, grd, 5, rng, state_every=100)
    nat.restore_envs(saved[0], [10, 20, 30]); grd.restore_envs(saved[1], [10, 20, 30])
    _same_obs(sb, nat, grd, "restore")
    nat.copy_envs([5, 5, 6], [40, 41, 42]); grd.copy_envs([5, 5, 6], [40, 41, 42])
    _same_obs(sb, nat, grd, "copy")
    _lockstep(sb, nat, grd, 8, rng)
    nat.close(); grd.close()
    # ring family too
    nat, grd = _twins(sb, "tile_classic_6x12")
    nat.reset(); grd.reset()
    _lockstep(sb, nat, grd, 6, rng, state_every=100)
    nat.copy_envs(torch.tensor([0, 1], device=nat.device), torch.tensor([7, 8], device=nat.device))
    grd.copy_envs(torch.tensor([0, 1], device=grd.device), torch.tensor([7, 8], device=grd.device))
    _same_obs(sb, nat, grd, "ring copy")
    nat.close(); grd.close()


def test_expand_views_subsets_and_out(sb):
    import torch
    for case in ("lane_classic_4x12", "rows_cut_16x64"):
        nat, grd = _twins(sb, case)
        nat.reset(); grd.reset()
        _lockstep(sb, nat, grd, 5, np.random.RandomState(0), state_every=100)
        K = nat.K
        for first, n in ((0, 1), (1, 1), (K - 1, 1), (0, 2), (1, 2), (0, 3), (1, 3), (0, K), (K - 3, 3)):
            got = sb.expand_views(grd.obs, n, first_view=first)
            assert torch.equal(got, nat.obs[..., 3 * first:3 * (first + n)]), (case, first, n)
        # views beyond S have no self snake: every snake in the other colours
        far = sb.expand_views(grd.obs, 1, first_view=nat.S)
        assert torch.equal(far, sb.expand_views(grd.obs, 1, first_view=31))
        # a gathered minibatch, an unaligned output and `out=`
        idx = torch.tensor([3, 0, 2], device=grd.device)
        assert torch.equal(sb.expand_views(grd.obs[idx], K), nat.obs[idx])
        buf = torch.empty(grd.obs[:2].numel() * 3 * K + 1, dtype=torch.uint8, device=grd.device)
        sb.expand_views(grd.obs[:2], K, out=buf[1:].view(tuple(grd.obs[:2].shape) + (3 * K,)))
        assert torch.equal(buf[1:].view_as(nat.obs[:2]), nat.obs[:2])
        out = torch.empty_like(nat.obs)
        assert sb.expand_views(grd.obs, K, out=out) is out and torch.equal(out, nat.obs)
        with pytest.raises(ValueError):
            sb.expand_views(grd.obs, K, out=torch.empty(3, dtype=torch.uint8, device=grd.device))
        with pytest.raises(sb.SnkError):
            sb.expand_views(grd.obs, 2, first_view=31)
        nat.close(); grd.close()


def test_grid_render_and_interfaces(sb):
    nat = sb.SnakeVecEnv(64, size=10, n_snakes=2, seed=8)
    grd = sb.SnakeVecEnv(64, size=10, n_snakes=2, seed=8, obs_mode="grid")
    nat.reset(); grd.reset()
    for t in range(30):
        a = nat.gen_actions(t, 1).clone()
        nat.step(a); grd.step(a)
    for i in (0, 17, 63):
        assert np.array_equal(nat.render(env_index=i), grd.render(env_index=i)), i
    # K < S: the native render cannot rebuild the world view, the grid one can
    g1 = sb.SnakeVecEnv(8, size=10, n_snakes=3, n_views=1, seed=1, obs_mode="grid")
    g1.reset()
    w = g1.render()
    assert w.shape == (12, 12, 3) and (w == (255, 255, 255)).all(-1)[0].all()
    # through the registry, and the learner refuses it
    v = sb.make("snake-multiple-v0", num_envs=16, obs_mode="grid")
    assert tuple(v.obs.shape) == (16, 12, 12)
    b = sb.make_basic_env("snake-multiple-v0", 16, seed=0, obs_mode="grid")
    assert b.obs_mode == "grid"
    from snakes_b200 import selfplay
    with pytest.raises(ValueError):
        selfplay.Runner(b, None, [], 8)
    for e in (nat, grd, g1, v, b):
        e.close()


def test_grid_save_load_keeps_mode(sb, tmp_path):
    import torch
    grd = sb.SnakeVecEnv(100, size=10, n_snakes=2, seed=6, obs_mode="grid")
    grd.reset()
    for t in range(12):
        grd.step(grd.gen_actions(t, 1))
    path = str(tmp_path / "g.npz")
    grd.save(path)
    back = sb.SnakeVecEnv.load(path)
    assert back.obs_mode == "grid" and torch.equal(back.obs, grd.obs)
    grd.close(); back.close()
