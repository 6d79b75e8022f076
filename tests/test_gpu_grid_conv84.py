"""GPU: nature_cnn's first layer read from cell-code grids (snk_grid_conv84_in / snk_grid_conv84_in_wgrad, grid_conv84_in)
and the self-play learner with arch 'nature' on obs_mode 'grid' envs.  The kernels against the fp64 references of
grid_conv84_ref; a nature grid CnnPolicy against the RGB nature CnnPolicy on the WarpFrame view of an obs_mode 'atari84'
twin with the same weights; Runner.run and learn on a grid env against replaying twins and RGB models."""
import os

import numpy as np
import pytest

import grid_conv84_ref as ref84
import grid_conv_ref as ref

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def sb():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import snakes_b200
    return snakes_b200


@pytest.fixture
def no_tf32():
    import torch
    old = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def _forward(sb, grids, k, w, b):
    import torch
    g = torch.as_tensor(np.ascontiguousarray(grids)).cuda()
    y = sb.grid_conv84_in(g, k, w.cuda(), b.cuda())
    assert tuple(y.shape) == (g.shape[0], 32, 20, 20) and y.dtype == torch.float32
    assert y.is_contiguous(memory_format=torch.channels_last)
    return y.permute(0, 2, 3, 1).cpu().double()


def _close(got, want, atol=1e-5):
    err = float((got - want).abs().max()) if got.numel() else 0.0
    assert err <= atol, err


@pytest.mark.parametrize("S", [1, 2, 3, 4, 8, 16])
@pytest.mark.parametrize("rules", ["classic", "adversarial", "cut"])
def test_forward_matches_fp64_on_oracle_grids(sb, rules, S):
    V = {1: 12, 2: 12, 3: 12, 4: 14, 8: 21, 16: 28}[S]
    grids = ref.oracle_grids(rules, S, V, n_envs=3, steps=30, seed=S)
    w, b = ref84.random_conv1_84(seed=S)
    for k in sorted(set(range(S)) | {S, 31}):
        _close(_forward(sb, grids, k, w, b), ref84.lookup_conv84_64(grids, k, w, b))


@pytest.mark.parametrize("n", [0, 1, 257, 1003])
@pytest.mark.parametrize("V", ref84.SUPPORTED_V)
def test_forward_every_size_ragged_and_edges(sb, V, n):
    """Every supported V, n = 0 and 1, batches whose last work item is ragged, non-empty cells on every edge."""
    S = 16 if V >= 21 else 3
    grids = ref.synthetic_grids(S, V, n, seed=V * 7 + n)
    w, b = ref84.random_conv1_84(seed=V)
    for k in ((0, 1, S, 31) if n < 1000 else (0, S)):
        got = _forward(sb, grids, k, w, b)
        assert got.shape == (n, 20, 20, 32)
        if n:
            _close(got, ref84.lookup_conv84_64(grids, k, w, b))


@pytest.mark.parametrize("case", ["lane", "ring"])
def test_forward_on_live_env_grids(sb, case):
    kw, N = (dict(size=19, n_snakes=2, rules="classic"), 2048) if case == "lane" else (dict(size=40, n_snakes=16, rules="cut"), 24)
    env = sb.SnakeVecEnv(N, seed=5, obs_mode="grid", **kw)
    assert ("k_lane_grid" in env.launch_info()["kernel"]) == (case == "lane")
    env.reset()
    for t in range(40):
        env.step(env.gen_actions(t, 1))
    grids = env.obs.cpu().numpy()
    w, b = ref84.random_conv1_84(seed=3)
    for k in (0, 1, env.S - 1, env.S):
        _close(_forward(sb, grids, k, w, b), ref84.lookup_conv84_64(grids, k, w, b))
    env.close()


@pytest.mark.parametrize("V,n,S,rules", [(12, 64, 2, "classic"), (21, 1024, 2, None), (21, 24, 16, "adversarial"),
                                         (42, 9, 16, "cut"), (4, 301, 3, None), (28, 50, 3, None)])
def test_backward_matches_fp64_autograd_and_is_deterministic(sb, V, n, S, rules):
    import torch
    grids = ref.oracle_grids(rules, S, V, n_envs=n, steps=20, seed=V) if rules else ref.synthetic_grids(S, V, n, seed=V)
    w0, b0 = ref84.random_conv1_84(seed=S)
    g = torch.as_tensor(grids).cuda()
    w = w0.cuda().requires_grad_(True)
    b = b0.cuda().requires_grad_(True)
    rng = np.random.default_rng(n)
    for k in sorted({0, 1, S}):
        y = sb.grid_conv84_in(g, k, w, b)
        gout = torch.from_numpy(rng.standard_normal((n, 20, 20, 32)).astype(np.float32))
        gy = gout.cuda().permute(0, 3, 1, 2)   # channels_last, like conv2's input gradient
        dw, db = torch.autograd.grad(y, (w, b), gy, retain_graph=True)
        dw2, db2 = torch.autograd.grad(y, (w, b), gy.contiguous())   # a second call, and an NCHW-contiguous gradient
        assert torch.equal(dw, dw2) and torch.equal(db, db2)
        dw_want, db_want = ref84.autograd_grads84_64(grids, k, w0, b0, gout.double())
        mag_w, mag_b = ref84.autograd_grads84_64(grids, k, w0, b0, gout.double().abs())   # sum of the terms' magnitudes
        assert ((dw.cpu().double() - dw_want).abs() <= 1e-4 * mag_w + 1e-6).all(), (k, float((dw.cpu().double() - dw_want).abs().max()))
        assert ((db.cpu().double() - db_want).abs() <= 1e-4 * mag_b + 1e-6).all(), k


def test_invalid_arguments_raise(sb):
    import ctypes as C
    import torch
    from snakes_b200 import _lib
    g = torch.zeros((4, 12, 12), dtype=torch.uint8, device="cuda")
    w, b = ref84.random_conv1_84(seed=0)
    w, b = w.cuda(), b.cuda()
    with pytest.raises(ValueError):
        sb.grid_conv84_in(g, 0, torch.zeros((16, 3, 8, 8), device="cuda"), torch.zeros(16, device="cuda"))   # C = 16
    for V in (11, 84, 2):
        with pytest.raises(sb.SnkError):
            sb.grid_conv84_in(torch.zeros((2, V, V), dtype=torch.uint8, device="cuda"), 0, w, b)
    with pytest.raises(sb.SnkError):
        sb.grid_conv84_in(g, 32, w, b)
    with pytest.raises(sb.SnkError):
        sb.grid_conv84_in(g, -1, w, b)
    y = sb.grid_conv84_in(g, 0, w, b).permute(0, 2, 3, 1).contiguous()
    gy = torch.ones_like(y)
    hist = torch.empty((7, 7, 2, 2, 7, 32), device="cuda")
    need = _lib.grid_conv84_geometry(12, 4)[3]
    work = torch.empty(need // 4, device="cuda")
    L, st = _lib.lib(), C.c_void_p(torch.cuda.current_stream().cuda_stream)
    args = lambda wb: (C.c_void_p(g.data_ptr()), 4, 10, 0, C.c_void_p(y.data_ptr()), C.c_void_p(gy.data_ptr()), 32,  # noqa: E731
                       C.c_void_p(hist.data_ptr()), C.c_void_p(work.data_ptr()), wb, 0, st)
    with pytest.raises(sb.SnkError):
        _lib.check(L.snk_grid_conv84_in_wgrad(*args(need - 4)))
    _lib.check(L.snk_grid_conv84_in_wgrad(*args(need)))
    torch.cuda.synchronize()
    assert torch.isfinite(hist).all()


def _twins(sb, N, size, S, seed, steps):
    """A grid env and an atari84 env with the same config and seed, stepped with the same actions."""
    envs = [sb.SnakeVecEnv(N, size=size, n_snakes=S, seed=seed, obs_mode=m) for m in ("grid", "atari84")]
    for e in envs:
        e.reset()
    for t in range(steps):
        a = envs[0].gen_actions(t, 1)
        for e in envs:
            e.step(a)
    return envs


def _nature_pair(V, seed=1):
    """A nature grid policy on V x V grids and the RGB nature policy with the same weights (and a nonzero conv1 bias)."""
    import torch
    from snakes_b200 import selfplay
    torch.manual_seed(seed)
    gnet = selfplay.CnnPolicy((V, V, 3), 5, "nature", grid=True).cuda().to(memory_format=torch.channels_last)
    rnet = selfplay.CnnPolicy((84, 84, 3), 5, "nature").cuda().to(memory_format=torch.channels_last)
    with torch.no_grad():
        gnet.convs[0].bias.uniform_(-0.1, 0.1)
    rnet.load_state_dict(gnet.state_dict())
    return gnet, rnet


@pytest.mark.parametrize("size", [10, 19])
def test_lockstep_grid_nature_policy_equals_atari84_rgb_policy(sb, no_tf32, size):
    import torch
    genv, aenv = _twins(sb, 512, size, 2, seed=2, steps=25)
    gnet, rnet = _nature_pair(genv.V)
    for k in (0, 1):
        lg, vg = gnet(genv.obs, k)
        lr, vr = rnet(aenv.obs[..., 3 * k:3 * k + 3].contiguous())
        assert torch.allclose(lg, lr, rtol=1e-4, atol=1e-5) and torch.allclose(vg, vr, rtol=1e-4, atol=1e-5), k
    genv.close(); aenv.close()


def test_checkpoints_move_between_grid_and_rgb_nature_models(sb, tmp_path, no_tf32):
    import torch
    from snakes_b200 import selfplay
    genv, aenv = _twins(sb, 256, 10, 2, seed=4, steps=10)
    for src_grid in (True, False):
        torch.manual_seed(7)
        src = selfplay.Model((12, 12, 3) if src_grid else (84, 84, 3), 5, arch="nature", device=genv.device, grid=src_grid)
        dst = selfplay.Model((84, 84, 3) if src_grid else (12, 12, 3), 5, arch="nature", device=genv.device, trainable=False,
                             grid=not src_grid)
        path = str(tmp_path / ("m%d.pkl" % src_grid))
        src.save(path)
        dst.load(path)
        gm, rm = (src, dst) if src_grid else (dst, src)
        assert torch.allclose(gm.net(genv.obs)[0], rm.net(aenv.obs[..., :3].contiguous())[0], rtol=1e-4, atol=1e-5)
    genv.close(); aenv.close()


def test_table_cache_follows_train_and_set_params(sb, no_tf32):
    """The cached lookup table is rebuilt after an optimizer step and after set_params: the grid model still equals the RGB
    model given the same weights."""
    import torch
    from snakes_b200 import selfplay
    genv, aenv = _twins(sb, 256, 10, 2, seed=6, steps=12)
    torch.manual_seed(3)
    gm = selfplay.Model((12, 12, 3), 5, arch="nature", device=genv.device, grid=True)
    rm = selfplay.Model((84, 84, 3), 5, arch="nature", device=genv.device, trainable=False)
    x_rgb = aenv.obs[..., :3].contiguous()

    def same():
        rm.set_params(gm.get_params())
        with torch.no_grad():
            lg, vg = gm.net(genv.obs)
            lr, vr = rm.net(x_rgb)
        return torch.allclose(lg, lr, rtol=1e-4, atol=1e-5) and torch.allclose(vg, vr, rtol=1e-4, atol=1e-5)

    assert same()
    n = genv.num_envs
    for _ in range(2):
        w_before = gm.net.convs[0].weight.detach().clone()
        gm.train(1e-3, 0.2, genv.obs, torch.randn(n, device="cuda"), None, torch.randint(0, 5, (n,), device="cuda"),
                 torch.zeros(n, device="cuda"), torch.full((n,), 1.6, device="cuda"))
        assert not torch.equal(w_before, gm.net.convs[0].weight)
        assert same()
    other = selfplay.Model((84, 84, 3), 5, arch="nature", device=genv.device, trainable=False)
    gm.set_params(other.get_params())
    assert same()
    genv.close(); aenv.close()


class _Recording(object):
    """An opponent model that records the view index it is asked for and the actions it plays."""

    def __init__(self, model):
        self.model, self.net, self.views, self.actions = model, model.net, [], []

    def step(self, ob, view=0):
        a, v, nlp = self.model.step(ob, view)
        self.views.append(view)
        self.actions.append(a.clone())
        return a, v, nlp


def test_runner_rollout_on_grid_env_with_nature_models(sb, no_tf32):
    """mb_obs holds the grids a replaying twin produces; values / neglogps are the RGB nature model's on the WarpFrame of
    the slots; returns are GAE over the twin's rewards."""
    import torch
    import gae_oracle
    from snakes_b200 import selfplay
    torch.manual_seed(0)
    T, N, V = 8, 130, 12
    kw = dict(size=V - 2, n_snakes=2, seed=11)
    env, twin, atwin = sb.SnakeVecEnv(N, obs_mode="grid", **kw), sb.SnakeVecEnv(N, obs_mode="grid", **kw), sb.SnakeVecEnv(N, obs_mode="atari84", **kw)
    model = selfplay.Model((V, V, 3), 5, arch="nature", device=env.device, grid=True)
    opp = _Recording(selfplay.Model((V, V, 3), 5, arch="nature", device=env.device, trainable=False, grid=True))
    runner = selfplay.Runner(env, model, [opp], nsteps=T)
    rnet = selfplay.CnnPolicy((84, 84, 3), 5, "nature").cuda().to(memory_format=torch.channels_last)
    rnet.load_state_dict(model.net.state_dict())
    for rollout in range(2):
        opp.actions.clear()
        obs, returns, dones, actions, values, neglogp, _, ep = runner.run()
        assert tuple(runner.mb_obs.shape) == (T, N, V, V) and tuple(obs.shape) == (N * T, V, V)
        assert opp.views == [1] * T * (rollout + 1)
        o, ao = (twin.reset(), atwin.reset()) if rollout == 0 else (twin.obs, atwin.obs)
        a_tn = actions.reshape(N, T).t()
        prev_done = torch.zeros(N, dtype=torch.bool, device=env.device) if rollout == 0 else prev_done
        rew = []
        for t in range(T):
            assert torch.equal(runner.mb_obs[t], o), (rollout, t)
            assert torch.equal(dones.reshape(N, T)[:, t], prev_done)
            with torch.no_grad():
                lg, v = rnet(ao[..., :3].contiguous())
            assert torch.allclose(values.reshape(N, T)[:, t], v, rtol=1e-4, atol=1e-5)
            nlp = torch.nn.functional.cross_entropy(lg, a_tn[t], reduction="none")
            assert torch.allclose(neglogp.reshape(N, T)[:, t], nlp, rtol=1e-4, atol=1e-4)
            full = torch.stack([a_tn[t].to(torch.int8), opp.actions[t].to(torch.int8)], 1).contiguous()
            o, r, d, _ = twin.step(full)
            ao = atwin.step(full)[0]
            rew.append(r.clone()); prev_done = d.clone()
        assert torch.equal(env.obs, o)
        with torch.no_grad():
            last_v = rnet(ao[..., :3].contiguous())[1]
        advs, rets = gae_oracle.gae(torch.stack(rew).cpu().numpy(), values.reshape(N, T).t().cpu().numpy(),
                                    dones.reshape(N, T).t().cpu().numpy(), last_v.cpu().numpy(), prev_done.cpu().numpy(), 0.99, 0.95)
        assert np.allclose(returns.reshape(N, T).t().cpu().numpy(), rets, atol=1e-4)
    env.close(); twin.close(); atwin.close()


def test_two_snake_self_play_nature_grid_pool_and_checkpoints(sb, tmp_path):
    """learn(grid_env, arch='nature'): opponent files are written and the final checkpoint is an RGB nature policy that
    agrees with the grid model on the atari84 twin's observations."""
    import joblib
    import torch
    from snakes_b200 import selfplay
    torch.manual_seed(0)
    N, T, U = 256, 16, 5
    env = sb.SnakeVecEnv(N, size=10, n_snakes=2, seed=3, obs_mode="grid")
    d = str(tmp_path / "ppo")
    model, log = selfplay.learn(env, nsteps=T, total_timesteps=N * T * U, log_interval=1, model_dir=d, arch="nature",
                                opponent_save_interval=2, csv_path=str(tmp_path / "ppo.csv"), save_interval=2)
    env.check_errors()
    assert model.net.grid and model.net.arch == "nature"
    assert sorted(f for f in os.listdir(d) if f.startswith("opponent")) == ["opponent0_0.pkl", "opponent0_1.pkl", "opponent0_2.pkl"]
    assert log.rows[-1]["num_opponents"] == 3 and len(log.rows) == U
    params = joblib.load(os.path.join(d, "snake_model_num2_final.pkl"))
    assert len(params) == 12 and params[0].shape == (8, 8, 3, 32) and params[6].shape == (7 * 7 * 64, 512)
    m2 = selfplay.Model((84, 84, 3), 5, arch="nature", device=env.device, trainable=False)
    m2.load(os.path.join(d, "snake_model_num2_final.pkl"))
    twin = sb.SnakeVecEnv(N, size=10, n_snakes=2, seed=3, obs_mode="atari84")
    twin.restore_envs(env.save_envs())   # the learner env's current state, observed as the WarpFrame
    with torch.no_grad():
        assert torch.allclose(m2.net(twin.obs[..., :3].contiguous())[0], model.net(env.obs)[0], atol=1e-4)
    env.close(); twin.close()


def test_single_snake_ppo_learns_on_device_grid_nature():
    """The nature twin of test_single_snake_ppo_learns_on_device_grid, with the same thresholds and the same budget
    (36 updates of 1 024 envs x 32 steps): measured on one B200, eprewmean 100 goes from -0.94 to 1.80 and eplenmean from
    7.3 to 201.8 at that budget, so no larger budget (and no atari84 run to calibrate one) is needed."""
    import torch
    import snakes_b200
    from snakes_b200 import selfplay
    torch.manual_seed(0)
    env = snakes_b200.SnakeVecEnv(1024, size=10, n_snakes=1, seed=0, obs_mode="grid")
    model, log = selfplay.learn(env, nsteps=32, total_timesteps=1024 * 32 * 36, log_interval=6, seed=0, arch="nature")
    env.check_errors()
    assert model.net.grid and model.net.arch == "nature"
    first, last = log.rows[0], log.rows[-1]
    assert first["eprewmean 100"] < -0.8
    assert last["eprewmean 100"] > first["eprewmean 100"] + 0.5, (first, last)
    assert last["eplenmean"] > 3 * first["eplenmean"]
    env.close()
