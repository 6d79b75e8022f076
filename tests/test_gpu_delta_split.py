"""GPU: the two-kernel form's sector store (k_lane_logic keeps the old paint items, k_lane_paint2 stores only the 32-byte
sectors a step changes) against whole-image stores (SNK_DEBUG delta=0), bit for bit every step, and every event after which
the own buffer no longer shows the records."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SPLIT = "k_lane_logic + k_lane_paint2"


@pytest.fixture(scope="module")
def sb():
    import snakes_b200
    return snakes_b200


def _pair(sb, N, kw, debug="lane=split"):
    """(sector store forced on, whole images), both in the two-kernel form unless `debug` says otherwise."""
    sep = "," if debug else ""
    a = sb.SnakeVecEnv(N, debug=debug + sep + "delta=1", **kw)
    b = sb.SnakeVecEnv(N, debug=debug + sep + "delta=0", **kw)
    return a, b


def _same(a, b, what):
    import torch
    assert torch.equal(a.obs, b.obs), "observations differ: %s" % what
    assert torch.equal(a.rewards, b.rewards) and torch.equal(a._done_u8, b._done_u8), "reward / done differ: %s" % what


def _actions(a, t, seed=3, eps=0.2):
    """Random actions and the fruit-seeking policy, so that bodies grow, snakes eat, die and respawn."""
    return a.gen_scripted_actions(t, seed=seed, eps=eps).clone() if t % 3 else a.gen_actions(t, seed).clone()


def _steps(a, b, t0, n, what, seed=3, eps=0.2):
    for t in range(t0, t0 + n):
        x = _actions(a, t, seed, eps)
        a.step(x)
        b.step(x)
        _same(a, b, "%s step %d" % (what, t))


def _close(*envs):
    for e in envs:
        e.check_errors()
        e.close()


def test_headline_eager_and_graph(sb):
    """131 072 envs of 2 snakes on 19x19: 200 eager steps, then a 200-step graph on the own buffer."""
    import torch
    N, kw = 131072, dict(size=19, n_snakes=2, rules="classic", seed=0)
    a, b = _pair(sb, N, kw)
    assert a.launch_info()["kernel"] == SPLIT
    a.reset(); b.reset()
    _same(a, b, "reset")
    _steps(a, b, 0, 200, "eager")
    acts = torch.stack([a.gen_actions(1000 + t, 9).clone() for t in range(16)])
    ga, gb = a.make_graph(acts, T=200), b.make_graph(acts, T=200)
    ga.launch(); gb.launch()
    _same(a, b, "after a 200-step graph")
    assert np.array_equal(a.dump_state_blob(), b.dump_state_blob())
    ga.close(); gb.close()
    _close(a, b)


@pytest.mark.parametrize("S,F", [(1, 1), (1, 4), (2, 1), (2, 3), (3, 2), (3, 4), (4, 1), (4, 4)])
def test_every_snake_and_fruit_count(sb, S, F):
    N, kw = 3001, dict(size=10, n_snakes=S, n_fruits=F, rules="classic", seed=4 + S + 7 * F)
    a, b = _pair(sb, N, kw)
    assert a.launch_info()["kernel"] == SPLIT
    a.reset(); b.reset()
    _steps(a, b, 0, 120, "S=%d F=%d" % (S, F))
    _close(a, b)


def test_bodies_past_17_segments(sb):
    """The fruit-seeking policy grows bodies past the 17 segments of the record's first chain word: images holding such
    an env go out whole, the others as sectors, in the same launch."""
    N, kw = 4096, dict(size=19, n_snakes=2, rules="classic", seed=11)
    a, b = _pair(sb, N, kw)
    a.reset(); b.reset()
    _steps(a, b, 0, 400, "long bodies", seed=5, eps=0.02)
    length = a.dump_state()["len"]
    assert (length > 17).any() and (length[(length > 0)] <= 17).any(), "no mix of short and long bodies"
    _close(a, b)


def test_regime_switch(sb):
    """The adaptive pair with its threshold lowered: fused -> two kernels -> fused, both storing sectors."""
    import torch
    N, kw = 4736, dict(size=19, n_snakes=2, rules="classic", seed=21)
    a, b = _pair(sb, N, kw, "alt_hi=6,epw=32")
    a.reset(); b.reset()
    plans = []
    for t in range(330):
        x = a.gen_scripted_actions(t, seed=5, eps=0.05).clone() if t < 200 else a.gen_actions(t, 5).clone()
        a.step(x); b.step(x)
        _same(a, b, "regime step %d" % t)
        torch.cuda.synchronize()
        plans.append(a.launch_info()["kernel"])
    assert plans[0] == plans[-1] == "k_step_lane" and SPLIT in plans, set(plans)
    _close(a, b)


def test_invalidation(sb):
    """Every way the own buffer can stop showing the records, each followed by steps that must still match."""
    import torch
    N, kw = 2048, dict(size=19, n_snakes=2, rules="classic", seed=6)
    a, b = _pair(sb, N, kw)
    a.reset(); b.reset()
    _steps(a, b, 0, 20, "warm-up")
    old = a.dump_state_blob()
    _steps(a, b, 20, 30, "before load")
    a.load_state_blob(old); b.load_state_blob(old)
    _steps(a, b, 50, 1, "first step after load_state_blob")
    _steps(a, b, 51, 10, "after load_state_blob")
    ta, tb = torch.zeros_like(a.obs), torch.zeros_like(b.obs)
    a.set_obs_target(ta); b.set_obs_target(tb)
    _steps(a, b, 61, 5, "into an obs target")
    a.set_obs_target(None); b.set_obs_target(None)
    _steps(a, b, 66, 5, "after set_obs_target(None)")
    acts = torch.stack([a.gen_actions(200 + t, 2).clone() for t in range(6)])
    oa, ra, da = a.rollout(acts)
    ob, rb, db = b.rollout(acts)
    assert torch.equal(oa, ob) and torch.equal(ra, rb) and torch.equal(da, db)
    _steps(a, b, 71, 5, "after rollout")
    mask = torch.arange(N, device=a.device) % 3 == 0
    a.reset(mask); b.reset(mask)
    _same(a, b, "masked reset")
    _steps(a, b, 76, 10, "after masked reset")
    # restore / copy without re-encoding: the next step must write the rewritten envs' images whole
    idx = np.arange(0, N, 5)
    sa, sb_ = a.save_envs(idx), b.save_envs(idx)
    _steps(a, b, 86, 4, "before restore_envs")
    a.restore_envs(sa, idx, observe=False); b.restore_envs(sb_, idx, observe=False)
    _steps(a, b, 90, 3, "after restore_envs(observe=False)")
    src, dst = np.arange(1, 200, 2), np.arange(400, 500)
    a.copy_envs(src, dst, observe=False); b.copy_envs(src, dst, observe=False)
    _steps(a, b, 93, 3, "after copy_envs(observe=False)")
    a.copy_envs(src, dst + 500); b.copy_envs(src, dst + 500)
    _same(a, b, "copy_envs(observe=True)")
    _steps(a, b, 96, 3, "after copy_envs(observe=True)")
    gacts = torch.stack([a.gen_actions(300 + t, 4).clone() for t in range(4)])
    ga, gb = a.make_graph(gacts, T=4), b.make_graph(gacts, T=4)
    ga.launch(); gb.launch()
    _same(a, b, "graph")
    a.load_state_blob(old); b.load_state_blob(old)
    ga.launch(); gb.launch()
    _same(a, b, "graph launched after load_state_blob")
    _steps(a, b, 99, 5, "after the graph")
    ga.close(); gb.close()
    _close(a, b)


def test_delta_store_is_taken(sb):
    """The writer really stores sectors: bytes of the own buffer that no step touches keep what was there, until an event
    clears frame_ok and the next step writes whole images again."""
    N, kw = 512, dict(size=19, n_snakes=2, rules="classic", seed=7)
    a, b = _pair(sb, N, kw)
    assert a.launch_info()["kernel"] == SPLIT
    a.reset(); b.reset()
    _steps(a, b, 0, 5, "warm-up")
    a.obs[:, 5:15, 5:15, :] = 77      # breaks the contract on purpose
    x = a.gen_actions(5, 3).clone()
    a.step(x); b.step(x)
    assert (a.obs != b.obs).any(), "every byte was rewritten: the sector store did not run"
    blob = a.dump_state_blob()
    a.load_state_blob(blob); b.load_state_blob(blob)
    _steps(a, b, 6, 3, "after load_state_blob")
    _close(a, b)
