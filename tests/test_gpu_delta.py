"""GPU: the fused lane kernel's delta store (only the 32-byte sectors a step changes are written into the own observation
buffer) against whole-image stores (SNK_DEBUG delta=0), bit for bit every step, and every event after which the own
buffer no longer shows the records (frame_ok must be cleared or rewritten)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def sb():
    import snakes_b200
    return snakes_b200


def _pair(sb, N, kw, debug=""):
    """(delta store forced on, whole images).  Shards with fewer than 32 envs per warp batch store whole images by
    default, so delta=1 makes those geometries take the sector path too."""
    sep = "," if debug else ""
    return sb.SnakeVecEnv(N, debug=debug + sep + "delta=1", **kw), sb.SnakeVecEnv(N, debug=debug + sep + "delta=0", **kw)


def _same(a, b, what):
    import torch
    assert torch.equal(a.obs, b.obs), "observations differ: %s" % what
    assert torch.equal(a.rewards, b.rewards) and torch.equal(a._done_u8, b._done_u8), "reward / done differ: %s" % what


def _actions(a, t, seed=3):
    """A mix of random actions and the fruit-seeking policy, so that bodies grow, snakes eat, die and respawn."""
    return a.gen_scripted_actions(t, seed=seed, eps=0.2).clone() if t % 3 else a.gen_actions(t, seed).clone()


def _steps(a, b, t0, n, what, seed=3):
    for t in range(t0, t0 + n):
        x = _actions(a, t, seed)
        a.step(x)
        b.step(x)
        _same(a, b, "%s step %d" % (what, t))


def _close(*envs):
    for e in envs:
        e.check_errors()
        e.close()


def test_headline_eager_and_graph(sb):
    """131 072 envs of 2 snakes on 19x19 (the headline): 300 eager steps, then a 200-step graph on the own buffer."""
    import torch
    N, kw = 131072, dict(size=19, n_snakes=2, rules="classic", seed=0)
    a, b = _pair(sb, N, kw)
    a.reset(); b.reset()
    _same(a, b, "reset")
    _steps(a, b, 0, 300, "eager")
    acts = torch.stack([a.gen_actions(1000 + t, 9).clone() for t in range(16)])
    ga, gb = a.make_graph(acts, T=200), b.make_graph(acts, T=200)
    ga.launch(); gb.launch()
    _same(a, b, "after a 200-step graph")
    assert np.array_equal(a.dump_state_blob(), b.dump_state_blob())
    ga.close(); gb.close()
    _close(a, b)


@pytest.mark.parametrize("epw", [16, 8, 4])
def test_small_shard_batches(sb, epw):
    """epw=<n> (n envs per warp batch, n / 8 images): ragged last batch and last image."""
    N, kw = 1003, dict(size=10, n_snakes=2, rules="classic", seed=8)
    a, b = _pair(sb, N, kw, "epw=%d" % epw)
    assert a.launch_info()["envs_per_warp_batch"] == epw
    a.reset(); b.reset()
    _steps(a, b, 0, 150, "epw=%d" % epw)
    _close(a, b)


@pytest.mark.parametrize("S", [1, 2, 3, 4])
def test_fused_every_snake_count(sb, S):
    N, kw = 3001, dict(size=10, n_snakes=S, rules="classic", seed=4 + S)
    a, b = _pair(sb, N, kw, "lane=fused")
    assert a.launch_info()["kernel"] == "k_step_lane"
    a.reset(); b.reset()
    _steps(a, b, 0, 120, "S=%d" % S)
    _close(a, b)


def test_regime_switch(sb):
    """fused -> two kernels -> fused on one handle: the two-kernel form writes whole images and sets frame_ok, so the
    fused kernel may store sectors again as soon as it is back."""
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
    assert plans[0] == plans[-1] == "k_step_lane" and "k_lane_logic + k_lane_paint2" in plans, set(plans)
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
    # an older state under a newer frame: one step must repaint from scratch
    a.load_state_blob(old); b.load_state_blob(old)
    _steps(a, b, 50, 1, "first step after load_state_blob")
    _steps(a, b, 51, 10, "after load_state_blob")
    # steps into an obs target, then back to the own buffer (which holds an older frame)
    ta, tb = torch.zeros_like(a.obs), torch.zeros_like(b.obs)
    a.set_obs_target(ta); b.set_obs_target(tb)
    _steps(a, b, 61, 5, "into an obs target")
    a.set_obs_target(None); b.set_obs_target(None)
    _steps(a, b, 66, 5, "after set_obs_target(None)")
    # a rollout into its own buffers, then steps on the own buffer
    acts = torch.stack([a.gen_actions(200 + t, 2).clone() for t in range(6)])
    oa, ra, da = a.rollout(acts)
    ob, rb, db = b.rollout(acts)
    assert torch.equal(oa, ob) and torch.equal(ra, rb) and torch.equal(da, db)
    _steps(a, b, 71, 5, "after rollout")
    # a masked reset
    mask = torch.arange(N, device=a.device) % 3 == 0
    a.reset(mask); b.reset(mask)
    _same(a, b, "masked reset")
    _steps(a, b, 76, 10, "after masked reset")
    # a graph captured before, launched after load_state_blob
    gacts = torch.stack([a.gen_actions(300 + t, 4).clone() for t in range(4)])
    ga, gb = a.make_graph(gacts, T=4), b.make_graph(gacts, T=4)
    ga.launch(); gb.launch()
    _same(a, b, "graph")
    a.load_state_blob(old); b.load_state_blob(old)
    ga.launch(); gb.launch()
    _same(a, b, "graph launched after load_state_blob")
    _steps(a, b, 86, 5, "after the graph")
    ga.close(); gb.close()
    _close(a, b)


def test_delta_store_is_taken(sb):
    """The sector store really runs: bytes of the own buffer that no step touches keep what was there (which is why
    callers must not write into it), until an event clears frame_ok and the next step writes whole images again."""
    N, kw = 512, dict(size=19, n_snakes=2, rules="classic", seed=7)
    a, b = _pair(sb, N, kw)
    a.reset(); b.reset()
    _steps(a, b, 0, 5, "warm-up")
    a.obs[:, 5:15, 5:15, :] = 77      # breaks the contract on purpose
    x = a.gen_actions(5, 3).clone()
    a.step(x); b.step(x)
    assert (a.obs != b.obs).any(), "every byte was rewritten: the delta store did not run"
    blob = a.dump_state_blob()
    a.load_state_blob(blob); b.load_state_blob(blob)
    _steps(a, b, 6, 3, "after load_state_blob")
    _close(a, b)
