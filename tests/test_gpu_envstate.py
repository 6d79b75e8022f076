"""GPU: per-env state on the device -- save_envs / restore_envs / copy_envs (snk_save_envs, snk_restore_envs,
snk_copy_envs).  Every check is bit for bit, on the lane family (chain-coded bodies) and on the ring family (tile, dense
and rows kernels), with long bodies (multi-word chain codes, ring wrap-around once stepped)."""
import numpy as np
import pytest

import c_oracle
import helpers

pytestmark = pytest.mark.gpu

# name -> (constructor kwargs, SNK_DEBUG string, num_envs)
CASES = {
    "lane_classic_2x19": (dict(size=19, n_snakes=2, rules="classic"), "", 2048),
    "lane_cut_3x10": (dict(size=10, n_snakes=3, rules="cut"), "", 1000),
    "lane_adversarial_3x10": (dict(size=10, n_snakes=3, rules="adversarial"), "", 1000),
    "lane_classic_1x10": (dict(size=10, n_snakes=1, rules="classic"), "", 600),
    "lane_classic_4x10": (dict(size=10, n_snakes=4, rules="classic"), "", 600),
    "tile_classic_2x19": (dict(size=19, n_snakes=2, rules="classic"), "force_kernel=tile", 96),
    "dense_cut_16x64": (dict(size=64, n_snakes=16, rules="cut"), "force_kernel=dense", 12),
    "rows_cut_16x64": (dict(size=64, n_snakes=16, rules="cut"), "force_kernel=rows", 12),
}


@pytest.fixture(scope="module")
def sb():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import snakes_b200
    return snakes_b200


def _make(sb, case, seed=1, debug_extra="", **extra):
    kw, dbg, N = CASES[case]
    dbg = ",".join(x for x in (dbg, debug_extra) if x)
    kw = dict(kw, **extra)
    return sb.SnakeVecEnv(N, seed=seed, debug=dbg, **kw)


def _variants(sb, case, seed=1):
    """Lane-family classic handles come as delta=1 / delta=0 twins (sector store forced on / whole images), so that a
    restore that failed to clear frame_ok shows up as stale observation bytes."""
    kw, dbg, _ = CASES[case]
    if dbg == "" and kw["rules"] == "classic":
        return [_make(sb, case, seed, "delta=1"), _make(sb, case, seed, "delta=0")]
    return [_make(sb, case, seed)]


def _actions(env, rng):
    import torch
    a = rng.randint(0, env.action_space.n, size=(env.N, env.S)).astype(np.int8)
    a[rng.rand(env.N, env.S) < 0.6] = 0   # mostly straight on, so that long bodies survive a while
    return torch.as_tensor(a, device=env.device)


def _prime(env, rng, steps=6):
    """Long random bodies loaded through the host path, re-encoded, then a few steps (ring wrap-around, carries)."""
    import torch
    env.load_state_blob(helpers.random_long_snake_states(env.lay, env.cfg, rng))
    env.reset(mask=torch.zeros(env.N, dtype=torch.bool, device=env.device))
    for _ in range(steps):
        env.step(_actions(env, rng))
    env.check_errors()


def _expected_blob(sb, env, whole, idx):
    """The canonical blob of envs `idx`, built on the host from a whole-handle dump."""
    cfg, lay = env._sub_config(len(idx))
    blob = np.zeros(lay.total_bytes, dtype=np.uint8)
    st = sb.split_state(blob, lay, cfg)
    for k in st:
        st[k][...] = whole[k][np.asarray(idx)]
    return blob


def _outputs(env):
    return [x.clone() for x in (env.obs, env.rewards, env._done_u8, env.num_alive, env.episode_return, env.episode_len)]


def _same_outputs(a, b, what):
    import torch
    names = ("obs", "reward", "done", "num_alive", "episode_return", "episode_len")
    for n, x, y in zip(names, a, b):
        assert torch.equal(x, y), "%s: %s differs" % (what, n)


def _np(t):
    """numpy copy of a torch view of an EnvStates blob (unsigned 16 / 32-bit views go through their signed twins)."""
    import torch
    if t.dtype == torch.uint16:
        return t.view(torch.int16).cpu().numpy().view(np.uint16)
    if t.dtype == torch.uint32:
        return t.view(torch.int32).cpu().numpy().view(np.uint32)
    return t.cpu().numpy()


# ---------------------------------------------------------------------------------------------------- 1. save = host dump
@pytest.mark.parametrize("case", list(CASES))
def test_save_equals_host_dump(sb, case):
    import torch
    env = _make(sb, case)
    rng = np.random.RandomState(11)
    _prime(env, rng)
    N = env.N
    whole = env.dump_state()
    sets = [None, rng.randint(0, N, size=min(N, 257)), [0], [N - 1], [N - 1, 0, N - 1, 3 % N]]
    for idx in sets:
        n = N if idx is None else len(idx)
        out = sb.EnvStates.empty(env, n)
        out.blob.fill_(0xA5)                      # every byte, alignment gaps included, must be written
        got = env.save_envs(idx, out=out)
        assert got is out and got.count == n
        expect = _expected_blob(sb, env, whole, np.arange(N) if idx is None else idx)
        assert np.array_equal(got.numpy(), expect), (case, None if idx is None else len(idx))
    # the host blob itself, and a range through snk_dump_state_range
    assert np.array_equal(env.save_envs().numpy(), env.dump_state_blob())
    first, count = N // 3, max(1, N // 4)
    part = env.dump_state_range(first, count)
    st = sb.split_state(env.save_envs(np.arange(first, first + count)).numpy(), *env._sub_config(count)[::-1])
    for k in part:
        assert np.array_equal(st[k], part[k]), k
    # a CUDA index tensor (int64 and int32) is used as is; arrays() are views with split_state's names and shapes
    sel = rng.randint(0, N, size=min(N, 64))
    for dt in (torch.int64, torch.int32):
        got = env.save_envs(torch.as_tensor(sel, dtype=dt, device=env.device))
        assert np.array_equal(got.numpy(), _expected_blob(sb, env, whole, sel))
        host = sb.split_state(got.numpy(), got.lay, got.cfg)
        arrs = got.arrays()
        assert set(arrs) == set(host)
        for k in host:
            assert tuple(arrs[k].shape) == host[k].shape and np.array_equal(_np(arrs[k]), host[k]), k
    env.check_errors()
    env.close()


# ---------------------------------------------------------------------------------------------------- 2. round trip
def _record(env, acts):
    rec = []
    for a in acts:
        env.step(a)
        rec.append(_outputs(env) + [env.dump_state_blob()])
    return rec


def _replay(env, acts, rec, what):
    for t, a in enumerate(acts):
        env.step(a)
        _same_outputs(_outputs(env), rec[t][:6], "%s step %d" % (what, t))
        assert np.array_equal(env.dump_state_blob(), rec[t][6]), "%s step %d: state" % (what, t)


@pytest.mark.parametrize("mode", ["eager", "graph", "no_observe"])
@pytest.mark.parametrize("case", list(CASES))
def test_round_trip(sb, case, mode):
    """Save at t0, step k times recording everything; restore; the same k actions give the same outputs and states."""
    import torch
    for env in _variants(sb, case):
        rng = np.random.RandomState(5)
        _prime(env, rng)
        k = 10
        acts = [_actions(env, rng) for _ in range(k)]
        states = env.save_envs()
        at_t0 = _outputs(env)
        blob_t0 = env.dump_state_blob()
        if mode == "graph":
            # captured BEFORE the restore, launched after it: steps into the handle's own buffer, then per-step slots
            g = env.make_graph(torch.stack(acts), T=k)
            O = torch.empty((k,) + tuple(env.obs.shape), dtype=torch.uint8, device=env.device)
            R = torch.empty((k, env.N), dtype=torch.float32, device=env.device)
            Dn = torch.empty((k, env.N), dtype=torch.uint8, device=env.device)
            g2 = env.make_graph(torch.stack(acts), T=k, obs_out=O, rewards_out=R, dones_out=Dn)
            g.launch()
            first = (env.obs.clone(), env.rewards.clone(), env._done_u8.clone(), env.dump_state_blob())
            env.restore_envs(states, observe=False)
            g.launch()
            assert torch.equal(env.obs, first[0]) and torch.equal(env.rewards, first[1]) and torch.equal(env._done_u8, first[2])
            assert np.array_equal(env.dump_state_blob(), first[3])
            env.restore_envs(states, observe=False)
            g2.launch()
            O1, R1, D1 = O.clone(), R.clone(), Dn.clone()
            env.restore_envs(states, observe=False)
            g2.launch()
            assert torch.equal(O, O1) and torch.equal(R, R1) and torch.equal(Dn, D1)
            assert np.array_equal(env.dump_state_blob(), first[3])
            g.close(); g2.close()
        else:
            rec = _record(env, acts)
            env.restore_envs(states, observe=(mode == "eager"))
            assert np.array_equal(env.dump_state_blob(), blob_t0)
            if mode == "eager":
                assert torch.equal(env.obs, at_t0[0]), "re-encoded observations differ from the saved frame"
            _replay(env, acts, rec, "%s %s %s" % (case, mode, env._debug))
        env.check_errors()
        env.close()


# ---------------------------------------------------------------------------------------------------- 3. untouched envs
@pytest.mark.parametrize("case", ["lane_classic_2x19", "lane_cut_3x10", "tile_classic_2x19", "rows_cut_16x64"])
def test_untouched_envs_stay_untouched(sb, case):
    import torch
    for env in _variants(sb, case):
        rng = np.random.RandomState(7)
        _prime(env, rng)
        N = env.N
        perm = rng.permutation(N)
        m = max(2, N // 8)
        src, dst = perm[:m], perm[m:2 * m]
        rest = np.setdiff1d(np.arange(N), dst)
        for op in ("restore", "copy"):
            for observe in (False, True):
                before = env.dump_state()
                obs0 = env.obs.clone()
                if op == "restore":
                    env.restore_envs(env.save_envs(src), dst, observe=observe)
                else:
                    env.copy_envs(src, dst, observe=observe)
                after = env.dump_state()
                for k in before:
                    assert np.array_equal(after[k][rest], before[k][rest]), (op, observe, k)
                    assert np.array_equal(after[k][dst], before[k][src]), (op, observe, k)
                keep = torch.as_tensor(rest, device=env.device)
                assert torch.equal(env.obs[keep], obs0[keep]), (op, observe)
                if not observe:
                    assert torch.equal(env.obs, obs0), "observe=False must not touch the observations"
                env.step(_actions(env, rng))
        env.check_errors()
        env.close()


# ---------------------------------------------------------------------------------------------------- 4. oracle parity
def _compare_step(env, co, a, what):
    obs, rew, done, _ = env.step(a)
    cobs, crew, cdone, cinfo = co.step(a.cpu().numpy())
    assert np.array_equal(rew.cpu().numpy(), crew), what + " reward"
    assert np.array_equal(done.cpu().numpy(), cdone), what + " done"
    assert np.array_equal(env.num_alive.cpu().numpy(), cinfo["num_snakes"]), what + " num_snakes"
    assert np.array_equal(env.episode_return.cpu().numpy(), cinfo["episode_r"]), what + " episode r"
    assert np.array_equal(env.episode_len.cpu().numpy(), cinfo["episode_l"]), what + " episode l"
    assert np.array_equal(obs.cpu().numpy(), cobs), what + " obs"


@pytest.mark.parametrize("case", list(CASES))
def test_restore_copy_then_oracle_parity(sb, case):
    """A permuted host-built blob of long bodies restored into the whole handle, a 1 -> many broadcast copy, then lock
    step with the oracle loaded from the handle's own dump (clones keep the DESTINATION env's RNG key)."""
    import torch
    env = _make(sb, case, seed=3)
    N = env.N
    rng = np.random.RandomState(13)
    src_blob = helpers.random_long_snake_states(env.lay, env.cfg, rng)
    src = sb.split_state(src_blob, env.lay, env.cfg)
    perm = rng.permutation(N)
    blob = np.zeros_like(src_blob)
    st = sb.split_state(blob, env.lay, env.cfg)
    for k in st:
        st[k][...] = src[k][perm]
    env.restore_envs(torch.as_tensor(blob, device=env.device))
    assert np.array_equal(env.dump_state_blob(), blob)
    # broadcast: env a into many slots, env b into a few more
    a, b = int(perm[0]), int(perm[1])
    others = np.setdiff1d(np.arange(N), [a, b])
    dst = rng.choice(others, size=max(2, min(len(others), N // 2)), replace=False)
    srcs = np.where(np.arange(len(dst)) < (2 * len(dst)) // 3, a, b)
    pre = env.save_envs()
    pre_st = sb.split_state(pre.numpy(), pre.lay, pre.cfg)
    env.copy_envs(torch.as_tensor(srcs, device=env.device), torch.as_tensor(dst, device=env.device))
    post = env.save_envs()
    post_st = sb.split_state(post.numpy(), post.lay, post.cfg)
    rest = np.setdiff1d(np.arange(N), dst)
    for k in pre_st:
        assert np.array_equal(post_st[k][dst], pre_st[k][srcs]), k
        assert np.array_equal(post_st[k][rest], pre_st[k][rest]), k
    kw, _, _ = CASES[case]
    co = c_oracle.COracle(N, seed=3, **kw)
    co.load_state(env.dump_state_blob())
    assert np.array_equal(env.obs.cpu().numpy(), co.observe()), "re-encoded observations differ from the oracle's"
    for t in range(40):
        _compare_step(env, co, _actions(env, rng), "%s step %d" % (case, t))
    assert np.array_equal(env.dump_state_blob(), co.dump_state())
    env.check_errors()
    env.close()


# ---------------------------------------------------------------------------------------------------- 5. restore = load
@pytest.mark.parametrize("case", list(CASES))
def test_restore_equals_load(sb, case):
    import torch
    a, b = _make(sb, case, seed=4), _make(sb, case, seed=4)
    rng = np.random.RandomState(17)
    blob = helpers.random_long_snake_states(a.lay, a.cfg, rng)
    a.reset(); b.reset()
    a.restore_envs(blob)
    b.load_state_blob(blob)
    b.reset(mask=torch.zeros(b.N, dtype=torch.bool, device=b.device))
    assert np.array_equal(a.dump_state_blob(), b.dump_state_blob())
    assert torch.equal(a.obs, b.obs)
    for t in range(15):
        x = _actions(a, rng)
        a.step(x); b.step(x)
        _same_outputs(_outputs(a), _outputs(b), "%s step %d" % (case, t))
        assert np.array_equal(a.dump_state_blob(), b.dump_state_blob())
    a.check_errors(); b.check_errors()
    a.close(); b.close()


# ---------------------------------------------------------------------------------------------------- 6. rejection
@pytest.mark.parametrize("debug", ["", "force_kernel=tile"])
def test_restore_rejects_bad_states(sb, debug):
    """The bad blobs of test_load_state_rejects_bad_blobs, restored into a subset: the bad-state flag, and the state
    load_state_blob leaves for the same rows."""
    import torch
    kw = dict(size=10, n_snakes=2, seed=1)
    a, b = sb.SnakeVecEnv(8, debug=debug, **kw), sb.SnakeVecEnv(8, debug=debug, **kw)
    lane = a.launch_info()["kind"] == 0
    a.reset(); b.reset()
    x = a.gen_actions(0, 1).clone()
    a.step(x); b.step(x)
    good = a.dump_state_blob()
    idx = [3, 2, 6]
    cases = [("len", 5000, True), ("body", 60000, True), ("vel", 9, True), ("adjacency", None, lane)]
    for field, value, rejected in cases:
        bad = good.copy()
        st = sb.split_state(bad, a.lay, a.cfg)
        if field == "body":
            st["body"][3, 1, 0] = value
        elif field == "adjacency":
            st["len"][2, 0] = 3
            st["body"][2, 0, :3] = [14, 15, 40]   # 15 -> 40 is not a neighbour step
        else:
            st[field][3, 1] = value
        a.load_state_blob(good); b.load_state_blob(good)
        sub = _expected_blob(sb, a, st, idx)
        a.restore_envs(sub, idx, observe=False)
        if rejected:
            with pytest.raises(sb.SnkError, match="bad state"):
                a.check_errors()
            with pytest.raises(sb.SnkError):
                b.load_state_blob(bad)
        else:
            a.check_errors()
            b.load_state_blob(bad)
        assert np.array_equal(a.dump_state_blob(), b.dump_state_blob()), field
    # an out-of-range device index raises the flag and writes nothing for its entry
    a.load_state_blob(good)
    before = a.dump_state()
    states = a.save_envs([5, 1])
    a.restore_envs(states, torch.as_tensor([0, 8 + 5], device=a.device), observe=False)
    with pytest.raises(sb.SnkError, match="index out of range"):
        a.check_errors()
    after = a.dump_state()
    for k in before:
        assert np.array_equal(after[k][0], before[k][5]) and np.array_equal(after[k][1:], before[k][1:]), k
    a.copy_envs(torch.as_tensor([1, -1], device=a.device), torch.as_tensor([-7, 4], device=a.device), observe=False)
    with pytest.raises(sb.SnkError):
        a.check_errors()
    for k, v in a.dump_state().items():
        assert np.array_equal(v, after[k]), k
    out = sb.EnvStates.empty(a, 2)
    a.save_envs(torch.as_tensor([9, 4], device=a.device), out=out)
    with pytest.raises(sb.SnkError):
        a.check_errors()
    part = sb.split_state(out.numpy(), out.lay, out.cfg)
    for k in part:
        assert np.array_equal(part[k][1], after[k][4]), k
    # host indices are checked on the host
    with pytest.raises(IndexError):
        a.restore_envs(states, [0, 8])
    with pytest.raises(ValueError):
        a.restore_envs(states, [1, 1])
    with pytest.raises(ValueError):
        a.copy_envs([1, 2], [2, 3])
    a.close(); b.close()


# ---------------------------------------------------------------------------------------------------- 7. across handles
def test_states_move_across_handles(sb):
    kw = dict(size=19, n_snakes=2, rules="classic")
    A = sb.SnakeVecEnv(4096, seed=1, **kw)
    B = sb.SnakeVecEnv(1000, seed=2, env_id_base=77, **kw)
    rng = np.random.RandomState(19)
    _prime(A, rng)
    B.reset()
    ia = rng.choice(A.N, size=300, replace=False)
    ib = rng.choice(B.N, size=300, replace=False)
    states = A.save_envs(ia)
    B.restore_envs(states, ib)
    sa, sbst = A.dump_state(), B.dump_state()
    for k in sa:
        assert np.array_equal(sbst[k][ib], sa[k][ia]), k
    for _ in range(5):
        B.step(B.gen_actions(0, 3))
    B.check_errors()
    C = sb.SnakeVecEnv(16, size=10, n_snakes=2, seed=1)
    with pytest.raises(ValueError):
        C.restore_envs(sb.EnvStates.empty(A, 16))
    with pytest.raises(ValueError):
        C.save_envs(out=sb.EnvStates.empty(A, 16))
    with pytest.raises(ValueError):
        sb.SnakeVecEnv(16, size=19, n_snakes=2, rules="cut").restore_envs(sb.EnvStates.empty(A, 16))
    for e in (A, B, C):
        e.close()


# ---------------------------------------------------------------------------------------------------- 8. graph capture
@pytest.mark.parametrize("case", ["lane_classic_2x19", "lane_adversarial_3x10", "tile_classic_2x19"])
def test_graph_capture(sb, case):
    """save_envs(out=...), restore_envs(observe=False) and copy_envs(observe=False) recorded into one torch CUDA graph
    and replayed equal the eager sequence: none of them synchronises or allocates."""
    import torch
    a, b = _make(sb, case, seed=6), _make(sb, case, seed=6)
    rng_a, rng_b = np.random.RandomState(23), np.random.RandomState(23)
    _prime(a, rng_a); _prime(b, rng_b)
    N = a.N
    rng = np.random.RandomState(29)
    perm = rng.permutation(N)
    m = max(2, N // 8)
    save_idx = rng.randint(0, N, size=m)
    restore_idx = perm[:m]
    cs, cd = np.repeat(perm[m], m), perm[m + 1:2 * m + 1]
    dev = lambda v: torch.as_tensor(v, dtype=torch.int64, device=a.device)
    ta = [dev(v) for v in (save_idx, restore_idx, cs, cd)]
    tb = [dev(v) for v in (save_idx, restore_idx, cs, cd)]
    out_a, out_b = sb.EnvStates.empty(a, m), sb.EnvStates.empty(b, m)
    torch.cuda.synchronize()

    def seq(env, out, t):
        env.save_envs(t[0], out=out)
        env.restore_envs(out, t[1], observe=False)
        env.copy_envs(t[2], t[3], observe=False)

    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        seq(a, out_a, ta)
    assert np.array_equal(a.dump_state_blob(), b.dump_state_blob()), "capture must not run the work"
    seq(b, out_b, tb)
    g.replay()
    torch.cuda.synchronize()
    assert np.array_equal(out_a.numpy(), out_b.numpy())
    assert np.array_equal(a.dump_state_blob(), b.dump_state_blob())
    for t in range(8):
        x = _actions(a, rng)
        a.step(x); b.step(x)
        _same_outputs(_outputs(a), _outputs(b), "%s step %d after the graph" % (case, t))
    g.replay(); seq(b, out_b, tb)
    torch.cuda.synchronize()
    assert np.array_equal(a.dump_state_blob(), b.dump_state_blob())
    a.check_errors(); b.check_errors()
    del g
    a.close(); b.close()


# ---------------------------------------------------------------------------------------------------- 9. re-encoding
@pytest.mark.parametrize("target", ["atari84", "main_view"])
def test_observe_reencodes_like_load(sb, target):
    import torch
    kw = dict(size=19, n_snakes=2, rules="classic", seed=8)
    if target == "atari84":
        kw["obs_mode"] = "atari84"
    N = 512
    a, b = sb.SnakeVecEnv(N, **kw), sb.SnakeVecEnv(N, **kw)
    rng = np.random.RandomState(31)
    _prime(a, rng)
    b.load_state_blob(a.dump_state_blob())
    H = a.obs.shape[1]
    slots = [torch.zeros((N, H, H, 3), dtype=torch.uint8, device=a.device) for _ in range(2)]
    if target == "main_view":
        a.set_main_view_target(slots[0]); b.set_main_view_target(slots[1])
    blob = helpers.random_long_snake_states(a.lay, a.cfg, rng)
    idx = rng.choice(N, size=N // 3, replace=False)
    whole = sb.split_state(blob, a.lay, a.cfg)
    a.restore_envs(_expected_blob(sb, a, whole, np.arange(len(idx))), idx)
    full = b.dump_state()
    for k in full:
        full[k][idx] = whole[k][:len(idx)]
    fb = np.zeros(b.lay.total_bytes, dtype=np.uint8)
    fst = sb.split_state(fb, b.lay, b.cfg)
    for k in fst:
        fst[k][...] = full[k]
    b.load_state_blob(fb)
    b.reset(mask=torch.zeros(N, dtype=torch.bool, device=b.device))
    assert np.array_equal(a.dump_state_blob(), b.dump_state_blob())
    assert torch.equal(a.obs, b.obs)
    if target == "main_view":
        assert torch.equal(slots[0], slots[1]) and torch.equal(slots[0], a.obs[..., 0:3])
    a.copy_envs(idx[:4], np.setdiff1d(np.arange(N), idx)[:4])
    b.load_state_blob(a.dump_state_blob())
    b.reset(mask=torch.zeros(N, dtype=torch.bool, device=b.device))
    assert torch.equal(a.obs, b.obs)
    if target == "main_view":
        assert torch.equal(slots[0], slots[1])
    a.check_errors(); b.check_errors()
    a.close(); b.close()
