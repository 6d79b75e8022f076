"""GPU: the scripted fruit-seeking policy kernel (k_scripted_actions, behind snk_gen_scripted_actions and
snk_graph_create_scripted) against its reference, tests/scripted_ref.py, bit for bit: on the hand-built states of
tests/test_scripted_ref_cpu.py, on live states of every lane (S, K) combination the policy drives itself into, after
every way the handle's observations can stop or start describing the state (the kernel then walks the bodies or reads
the green bytes of the native image), and inside the captured scripted graph against an eagerly stepped twin."""
import numpy as np
import pytest

import scripted_ref as ref
from test_scripted_ref_cpu import CASES, case_groups

pytestmark = pytest.mark.gpu

U64 = (1 << 64) - 1


@pytest.fixture(scope="module")
def sb():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import snakes_b200
    return snakes_b200


def _check(env, step, seed, eps, where):
    """gen_scripted_actions against the reference on the state dumped just before the call; returns the device actions."""
    st = env.dump_state()
    dev = env.gen_scripted_actions(step, seed=seed, eps=eps / 1000.0)
    got = dev.cpu().numpy()
    want = ref.scripted_actions(st, env.cfg, step, seed, eps, env.cfg.env_id_base)
    if not np.array_equal(got, want):
        bad = np.flatnonzero((got != want).any(axis=1))
        e = int(bad[0])
        raise AssertionError("%s: %d of %d envs differ from the reference; env %d: kernel %s, reference %s, len %s, vel %s, "
                             "heads %s, fruits %s" % (where, len(bad), env.N, e, got[e].tolist(), want[e].tolist(),
                                                      st["len"][e].tolist(), st["vel"][e].tolist(),
                                                      st["body"][e, :, 0].tolist(), st["fruit"][e].tolist()))
    return dev


def _grow(env, t0, steps, seed, eps):
    """The policy drives the env for `steps` steps (step indices t0, t0 + 1, ...): long bodies on a crowded board."""
    for t in range(t0, t0 + steps):
        env.step(env.gen_scripted_actions(t, seed=seed, eps=eps / 1000.0))


def test_hand_built_states(sb):
    """Every case of the CPU file, loaded into a device env: the kernel's answer after load_state (it walks the bodies)
    and after the observations are re-encoded (it reads them), native and grid."""
    import torch
    for (size, S, F), names in sorted(case_groups().items()):
        for mode in ("native", "grid"):
            env = sb.SnakeVecEnv(len(names), size=size, n_snakes=S, n_fruits=F, seed=1, env_id_base=40, obs_mode=mode)
            blob = np.zeros(env.lay.total_bytes, dtype=np.uint8)
            st = sb.split_state(blob, env.lay, env.cfg)
            for e, n in enumerate(names):
                ref.fill_state(st, e, *((size,) + CASES[n][3:6]))
            env.load_state_blob(blob)
            back = env.dump_state()
            for k in ("len", "vel", "body", "fruit"):
                assert np.array_equal(back[k], st[k]), (names, k)
            want = [CASES[n][6] for n in names]
            assert _check(env, 3, 1, 0, "%s %s loaded" % (mode, names)).cpu().tolist() == want, (mode, names)
            env.reset(mask=torch.zeros(env.N, dtype=torch.bool, device=env.device))
            assert _check(env, 3, 1, 0, "%s %s observed" % (mode, names)).cpu().tolist() == want, (mode, names)
            env.check_errors()
            env.close()


# name -> (n_snakes, n_views, size, n_fruits, eps permille, num_envs, env_id_base, seed, first step index, steps)
LIVE = {
    "s1k1_d32_f1": (1, 1, 32, 1, 50, 1000, 3, 11, 0, 400),
    "s2k2_d3_f2": (2, 2, 3, 2, 50, 4097, 7, 12, 0, 120),
    "s3k3_d5_f4": (3, 3, 5, 4, 0, 1000, 0, (1 << 32) + 5, 0, 150),
    "s4k4_d4_f0": (4, 4, 4, 0, 50, 4097, 123456, 14, 0, 120),
    "s1k3_d10_f1_eps1000": (1, 3, 10, 1, 1000, 1000, 9, 15, 0, 60),
    "s2k3_d12_f4_counter_2e32": (2, 3, 12, 4, 50, 4097, 1 << 31, 16, (1 << 31) - 100, 250),
    "s2k2_d19_f2_headline": (2, 2, 19, 2, 50, 131072, 0, 17, 0, 150),
}


@pytest.mark.parametrize("name", sorted(LIVE))
def test_live_states(sb, name):
    """The policy drives the env (native observations: the kernel reads occupancy from the image the last step wrote);
    at chosen steps the actions equal the reference on the state dumped just before the call."""
    S, K, D, F, eps, N, base, seed, t0, steps = LIVE[name]
    env = sb.SnakeVecEnv(N, size=D, n_snakes=S, n_fruits=F, n_views=K, seed=21, env_id_base=base)
    assert env.launch_info()["kind"] == 0, env.launch_info()
    env.reset()
    checks = {steps - 1} if N > 100000 else {0, 1, steps // 2, steps - 1}
    longest = 0
    for t in range(t0, t0 + steps):
        if t - t0 in checks:
            longest = max(longest, int(env.dump_state()["len"].max()))
            a = _check(env, t, seed, eps, "%s step %d" % (name, t))
        else:
            a = env.gen_scripted_actions(t, seed=seed, eps=eps / 1000.0)
        env.step(a)
    env.check_errors()
    env.close()
    if eps < 1000 and F:
        assert longest > 3, longest   # the policy ate fruit: bodies past their first growth


# the occupancy sources: constructor kwargs and what is done to the env before the kernel is checked
SOURCES = ["delta=1", "delta=0", "atari84", "grid", "obs_target", "load_state", "restore_unobserved", "restore_observed",
           "copy_unobserved", "copy_observed"]


@pytest.mark.parametrize("source", SOURCES)
def test_occupancy_source(sb, source):
    """Each way the handle can come to a state, with the kernel's occupancy read from the observations or from a walk
    of the bodies, gives the reference's actions."""
    import torch
    seed, eps, N = 31, 50, 1000
    kw = dict(size=10, n_snakes=2, n_views=3, seed=8, env_id_base=300)
    if source.startswith("delta"):
        kw["debug"] = source
    elif source in ("atari84", "grid"):
        kw["obs_mode"] = source
    env = sb.SnakeVecEnv(N, **kw)
    env.reset()
    _grow(env, 0, 150, seed, eps)
    _check(env, 150, seed, eps, source)
    t = 151
    if source == "obs_target":
        slots = torch.zeros((2,) + tuple(env.obs.shape), dtype=torch.uint8, device=env.device)
        for k in range(4):
            env.set_obs_target(slots[k % 2])
            env.step(_check(env, t, seed, eps, "%s slot %d" % (source, k)))
            t += 1
        env.set_obs_target(None)
    elif source == "load_state":
        blob = env.dump_state_blob()
        _grow(env, t, 5, seed, eps)
        t += 5
        env.load_state_blob(blob)
        env.step(_check(env, t, seed, eps, "%s loaded" % source))
        t += 1
        env.load_state_blob(blob)
        env.reset(mask=torch.zeros(N, dtype=torch.bool, device=env.device))
        _check(env, t, seed, eps, "%s re-encoded" % source)
    elif source.startswith("restore"):
        idx = torch.arange(0, N, 3, device=env.device)
        saved = env.save_envs(idx)
        _grow(env, t, 7, seed, eps)
        t += 7
        env.restore_envs(saved, idx, observe=source == "restore_observed")
        env.step(_check(env, t, seed, eps, "%s restored" % source))
        t += 1
    elif source.startswith("copy"):
        src = torch.arange(0, 100, device=env.device)
        dst = torch.arange(N - 100, N, device=env.device).flip(0)
        env.copy_envs(src, dst, observe=source == "copy_observed")
        env.step(_check(env, t, seed, eps, "%s copied" % source))
        t += 1
    for k in range(3):   # and the steps after it, on the observations those steps wrote
        env.step(_check(env, t, seed, eps, "%s step %d after" % (source, t)))
        t += 1
    env.check_errors()
    env.close()


def _same_env(a, b, where):
    import torch
    sa, sb_ = a.dump_state(), b.dump_state()
    for k in sa:
        assert np.array_equal(sa[k], sb_[k]), (where, k)
    assert torch.equal(a.obs, b.obs), where
    assert torch.equal(a.rewards, b.rewards) and torch.equal(a._done_u8, b._done_u8), where
    assert a.stats(False) == b.stats(False), where


@pytest.mark.parametrize("mode,T", [("native", 1), ("native", 4), ("atari84", 1), ("atari84", 4), ("grid", 4)])
def test_scripted_graph(sb, mode, T):
    """make_scripted_graph(T) against a twin stepped eagerly with the reference's actions: step 0 of a launch walks the
    bodies, steps 1..T-1 read the observations the previous captured step wrote.  Two launches of one graph, then an
    eager call that reads the observations the launch left."""
    import torch
    kw = dict(size=10, n_snakes=2, seed=4, obs_mode=mode, env_id_base=500)
    N, step0, seed, eps = 1000, 1000, 7, 50
    A, B = sb.SnakeVecEnv(N, **kw), sb.SnakeVecEnv(N, **kw)
    A.reset(); B.reset()
    for t in range(120):
        for env in (A, B):
            env.step(env.gen_scripted_actions(t, seed=3, eps=0.05))
    _same_env(A, B, "warm-up")
    g = A.make_scripted_graph(T, step0=step0, seed=seed, eps=eps / 1000.0)
    for launch in range(2):
        g.launch()
        for t in range(T):
            a = ref.scripted_actions(B.dump_state(), B.cfg, step0 + t, seed, eps, B.cfg.env_id_base)
            B.step(torch.as_tensor(a, device=B.device))
        torch.cuda.synchronize()
        _same_env(A, B, "%s T=%d launch %d" % (mode, T, launch))
    _check(A, step0 + T, seed, eps, "%s eager call after the graph" % mode)
    g.close()
    A.check_errors(); B.check_errors()
    A.close(); B.close()


def test_rejections(sb):
    """eps outside 0..1000, a ring-family handle and non-classic rules are refused by the eager call and the graph."""
    lane = sb.SnakeVecEnv(64, size=10, n_snakes=2)
    ring = sb.SnakeVecEnv(64, size=12, n_snakes=6)
    adv = sb.SnakeVecEnv(64, size=10, n_snakes=3, rules="adversarial")
    assert ring.launch_info()["kind"] != 0 and adv.launch_info()["kind"] == 0
    for env in (lane, ring, adv):
        env.reset()
    for eps in (0.0, 1.0):
        lane.gen_scripted_actions(0, eps=eps)
        lane.make_scripted_graph(1, eps=eps).close()
    for env, eps in ((lane, -0.001), (lane, 1.001), (ring, 0.05), (adv, 0.05)):
        with pytest.raises(sb._lib.SnkError):
            env.gen_scripted_actions(0, eps=eps)
        with pytest.raises(sb._lib.SnkError):
            env.make_scripted_graph(2, eps=eps)
    for env in (lane, ring, adv):
        env.close()


def test_uniform_stream_counter_and_key_split(sb):
    """The uniform action stream (snk_gen_actions, stream 1) at the top of the env id range, with step * S + s across
    2^32 and beyond, and seeds above 2^32."""
    N, S = 1000, 3
    base = (1 << 32) - 1 - N   # the last ids a handle may hold: base + N <= 2^32 - 1
    env = sb.SnakeVecEnv(N, size=10, n_snakes=S, rules="cut", env_id_base=base)
    ids = np.arange(N, dtype=np.uint64) + np.uint64(base)
    for step, seed in (((1 << 32) // S, 5), ((1 << 34) + 2, (1 << 40) + 1), (U64, U64)):
        got = env.gen_actions(step, seed).cpu().numpy()
        want = np.stack([ref.philox_bounded(seed, ids, ref.STREAM_ACTIONS, (step * S + s) & U64, env.action_space.n)
                         for s in range(S)], axis=1)
        assert np.array_equal(got, want), (step, seed)
    env.close()
