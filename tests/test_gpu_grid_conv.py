"""GPU: the policy's first layer read from cell-code grids (snk_grid_conv_in / snk_grid_conv_in_wgrad, grid_conv_in) and the
self-play learner on obs_mode 'grid' envs.  The kernels against the fp64 references of grid_conv_ref; a grid CnnPolicy
against the RGB CnnPolicy on expand_views with the same weights; Runner.run on a grid env against a replaying twin."""
import ctypes as C
import os

import numpy as np
import pytest

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
    y = sb.grid_conv_in(g, k, w.cuda(), b.cuda())
    n, V = g.shape[0], g.shape[-1]
    assert tuple(y.shape) == (n, 32, V, V) and y.dtype == torch.float32
    assert y.is_contiguous(memory_format=torch.channels_last)
    return y.permute(0, 2, 3, 1).cpu().double()


def _close(got, want, atol=1e-5):
    err = float((got - want).abs().max()) if got.numel() else 0.0
    assert err <= atol, err


@pytest.mark.parametrize("S", [1, 2, 3, 4, 8, 16])
@pytest.mark.parametrize("rules", ["classic", "adversarial", "cut"])
def test_forward_matches_fp64_on_oracle_grids(sb, rules, S):
    V = {1: 12, 2: 12, 3: 12, 4: 12, 8: 14, 16: 21}[S]
    grids = ref.oracle_grids(rules, S, V, n_envs=3, steps=30, seed=S)
    w, b = ref.random_conv1(seed=S)
    for k in sorted(set(range(S)) | {S, 31}):
        _close(_forward(sb, grids, k, w, b), ref.lookup_conv64(grids, k, w, b))


@pytest.mark.parametrize("V,n", [(3, 5), (4, 1), (4, 257), (12, 0), (12, 1), (12, 1003), (21, 333), (66, 7), (256, 2)])
def test_forward_sizes_ragged_and_edges(sb, V, n):
    """Any V, n = 0 and 1, batches whose last chunk is ragged, and non-empty cells on all four edges (zero padding)."""
    S = 16 if V >= 21 else 3
    grids = ref.synthetic_grids(S, V, n, seed=V * 7 + n)
    w, b = ref.random_conv1(seed=V)
    for k in (0, 1, S, 31):
        got = _forward(sb, grids, k, w, b)
        assert got.shape == (n, V, V, 32)
        _close(got, ref.lookup_conv64(grids, k, w, b) if n else got)


@pytest.mark.parametrize("case", ["lane", "rows"])
def test_forward_on_live_env_grids(sb, case):
    kw, N = (dict(size=19, n_snakes=2, rules="classic"), 2048) if case == "lane" else (dict(size=64, n_snakes=16, rules="cut"), 24)
    env = sb.SnakeVecEnv(N, seed=5, obs_mode="grid", **kw)
    assert ("k_lane_grid" in env.launch_info()["kernel"]) == (case == "lane")
    env.reset()
    for t in range(40):
        env.step(env.gen_actions(t, 1))
    grids = env.obs.cpu().numpy()
    w, b = ref.random_conv1(seed=3)
    for k in (0, 1, env.S - 1, env.S):
        _close(_forward(sb, grids, k, w, b), ref.lookup_conv64(grids, k, w, b))
    env.close()


@pytest.mark.parametrize("V,n,S,rules", [(12, 64, 2, "classic"), (21, 4096, 2, None), (21, 24, 16, "adversarial"),
                                         (66, 9, 16, "cut"), (5, 1001, 3, None)])
def test_backward_matches_fp64_autograd_and_is_deterministic(sb, V, n, S, rules):
    import torch
    grids = ref.oracle_grids(rules, S, V, n_envs=n, steps=20, seed=V) if rules else ref.synthetic_grids(S, V, n, seed=V)
    w0, b0 = ref.random_conv1(seed=S)
    g = torch.as_tensor(grids).cuda()
    w = w0.cuda().requires_grad_(True)
    b = b0.cuda().requires_grad_(True)
    rng = np.random.default_rng(n)
    for k in sorted({0, 1, S}):
        y = sb.grid_conv_in(g, k, w, b)
        gout = torch.from_numpy(rng.standard_normal((n, V, V, 32)).astype(np.float32))
        gy = gout.cuda().permute(0, 3, 1, 2)   # channels_last, like conv2's input gradient
        dw, db = torch.autograd.grad(y, (w, b), gy, retain_graph=True)
        dw2, db2 = torch.autograd.grad(y, (w, b), gy.contiguous())   # a second call, and an NCHW-contiguous gradient
        assert torch.equal(dw, dw2) and torch.equal(db, db2)
        dw_want, db_want = ref.autograd_grads64(grids, k, w0, b0, gout.double())
        mag_w, mag_b = ref.autograd_grads64(grids, k, w0, b0, gout.double().abs())   # sum of the terms' magnitudes
        assert ((dw.cpu().double() - dw_want).abs() <= 1e-4 * mag_w + 1e-6).all(), (k, float((dw.cpu().double() - dw_want).abs().max()))
        assert ((db.cpu().double() - db_want).abs() <= 1e-4 * mag_b + 1e-6).all(), k


def test_invalid_arguments_raise(sb):
    import torch
    from snakes_b200 import _lib
    g = torch.zeros((4, 12, 12), dtype=torch.uint8, device="cuda")
    w, b = ref.random_conv1(seed=0)
    w, b = w.cuda(), b.cuda()
    with pytest.raises(sb.SnkError):
        sb.grid_conv_in(g, 0, torch.zeros((16, 3, 3, 3), device="cuda"), torch.zeros(16, device="cuda"))   # C = 16
    with pytest.raises(sb.SnkError):
        sb.grid_conv_in(torch.zeros((2, 258, 258), dtype=torch.uint8, device="cuda"), 0, w, b)           # V = 258
    with pytest.raises(sb.SnkError):
        sb.grid_conv_in(torch.zeros((2, 2, 2), dtype=torch.uint8, device="cuda"), 0, w, b)               # V = 2
    with pytest.raises(sb.SnkError):
        sb.grid_conv_in(g, 32, w, b)
    with pytest.raises(sb.SnkError):
        sb.grid_conv_in(g, -1, w, b)
    y = sb.grid_conv_in(g, 0, w, b).permute(0, 2, 3, 1).contiguous()
    gy = torch.ones_like(y)
    hist = torch.empty((9, 7, 32), device="cuda")
    need = _lib.grid_conv_work_bytes(4 * 144)
    work = torch.empty(need // 4, device="cuda")
    L, st = _lib.lib(), C.c_void_p(torch.cuda.current_stream().cuda_stream)
    args = lambda wb: (C.c_void_p(g.data_ptr()), 4, 10, 0, C.c_void_p(y.data_ptr()), C.c_void_p(gy.data_ptr()), 32,  # noqa: E731
                       C.c_void_p(hist.data_ptr()), C.c_void_p(work.data_ptr()), wb, 0, st)
    with pytest.raises(sb.SnkError):
        _lib.check(L.snk_grid_conv_in_wgrad(*args(need - 4)))
    _lib.check(L.snk_grid_conv_in_wgrad(*args(need)))
    torch.cuda.synchronize()
    assert torch.isfinite(hist).all()


def _policies(V, grid_first=True):
    import torch
    from snakes_b200 import selfplay
    torch.manual_seed(1)
    a = selfplay.CnnPolicy((V, V, 3), 5, grid=grid_first).cuda().to(memory_format=torch.channels_last)
    bnet = selfplay.CnnPolicy((V, V, 3), 5, grid=not grid_first).cuda().to(memory_format=torch.channels_last)
    bnet.load_state_dict(a.state_dict())
    with torch.no_grad():
        a.convs[0].bias.uniform_(-0.1, 0.1)   # a nonzero bias, copied below
        bnet.convs[0].bias.copy_(a.convs[0].bias)
    return (a, bnet) if grid_first else (bnet, a)


def test_grid_policy_equals_rgb_policy(sb, no_tf32):
    import torch
    from snakes_b200 import selfplay
    env = sb.SnakeVecEnv(512, size=10, n_snakes=2, seed=2, obs_mode="grid")
    env.reset()
    for t in range(25):
        env.step(env.gen_actions(t, 1))
    gnet, rnet = _policies(env.V)
    for k in (0, 1):
        lg, vg = gnet(env.obs, k)
        lr, vr = rnet(sb.expand_views(env.obs, 1, first_view=k))
        assert torch.allclose(lg, lr, rtol=1e-4, atol=1e-5) and torch.allclose(vg, vr, rtol=1e-4, atol=1e-5), k
    with pytest.raises(ValueError):
        selfplay.CnnPolicy((84, 84, 3), 5, arch="nature", grid=True)
    env.close()


def test_checkpoints_move_between_grid_and_rgb_models(sb, tmp_path, no_tf32):
    import torch
    from snakes_b200 import selfplay
    env = sb.SnakeVecEnv(256, size=10, n_snakes=2, seed=4, obs_mode="grid")
    env.reset()
    for t in range(10):
        env.step(env.gen_actions(t, 1))
    rgb_view = sb.expand_views(env.obs, 1)
    for src_grid in (True, False):
        torch.manual_seed(7)
        src = selfplay.Model((12, 12, 3), 5, device=env.device, grid=src_grid)
        dst = selfplay.Model((12, 12, 3), 5, device=env.device, trainable=False, grid=not src_grid)
        path = str(tmp_path / ("m%d.pkl" % src_grid))
        src.save(path)
        dst.load(path)
        gm, rm = (src, dst) if src_grid else (dst, src)
        assert torch.allclose(gm.net(env.obs)[0], rm.net(rgb_view)[0], rtol=1e-4, atol=1e-5)
    env.close()


class _Recording(object):
    """An opponent model that records the view index it is asked for and the actions it plays."""

    def __init__(self, model):
        self.model, self.net, self.views, self.actions = model, model.net, [], []

    def step(self, ob, view=0):
        a, v, nlp = self.model.step(ob, view)
        self.views.append(view)
        self.actions.append(a.clone())
        return a, v, nlp


def test_runner_rollout_on_grid_env(sb, no_tf32):
    """mb_obs holds the grids a replaying twin produces; values / neglogps are the RGB model's on expand_views of the
    slots; returns are GAE over the twin's rewards; the runner refuses RGB models and env.obs is the current grid."""
    import torch
    import gae_oracle
    from snakes_b200 import selfplay
    torch.manual_seed(0)
    T, N = 8, 130    # N * V * V = 15 730: the runner pads its slots to 16-byte multiples
    kw = dict(size=9, n_snakes=2, seed=11, obs_mode="grid")
    env, twin = sb.SnakeVecEnv(N, **kw), sb.SnakeVecEnv(N, **kw)
    with pytest.raises(ValueError):
        selfplay.Runner(env, selfplay.Model((11, 11, 3), 5, device=env.device), [], T)
    model = selfplay.Model((11, 11, 3), 5, device=env.device, grid=True)
    opp = _Recording(selfplay.Model((11, 11, 3), 5, device=env.device, trainable=False, grid=True))
    runner = selfplay.Runner(env, model, [opp], nsteps=T)
    rnet = selfplay.CnnPolicy((11, 11, 3), 5).cuda().to(memory_format=torch.channels_last)
    rnet.load_state_dict(model.net.state_dict())
    for rollout in range(2):
        opp.actions.clear()
        obs, returns, dones, actions, values, neglogp, _, ep = runner.run()
        assert tuple(runner.mb_obs.shape) == (T, N, 11, 11) and tuple(obs.shape) == (N * T, 11, 11)
        assert opp.views == [1] * T * (rollout + 1)
        o = twin.reset() if rollout == 0 else twin.obs
        a_tn = actions.reshape(N, T).t()
        prev_done = torch.zeros(N, dtype=torch.bool, device=env.device) if rollout == 0 else prev_done
        rew = []
        for t in range(T):
            assert torch.equal(runner.mb_obs[t], o), (rollout, t)
            assert torch.equal(obs.reshape(N, T, 11, 11)[:, t], o)
            assert torch.equal(dones.reshape(N, T)[:, t], prev_done)
            with torch.no_grad():
                lg, v = rnet(sb.expand_views(o, 1))
            assert torch.allclose(values.reshape(N, T)[:, t], v, rtol=1e-4, atol=1e-5)
            nlp = torch.nn.functional.cross_entropy(lg, a_tn[t], reduction="none")
            assert torch.allclose(neglogp.reshape(N, T)[:, t], nlp, rtol=1e-4, atol=1e-4)
            full = torch.stack([a_tn[t].to(torch.int8), opp.actions[t].to(torch.int8)], 1).contiguous()
            o, r, d, _ = twin.step(full)
            rew.append(r.clone()); prev_done = d.clone()
        assert torch.equal(env.obs, o)   # env.obs is the current grid, in the env's own buffer
        assert not any(env.obs.data_ptr() == runner.mb_obs[t].data_ptr() for t in range(T))
        with torch.no_grad():
            last_v = rnet(sb.expand_views(o, 1))[1]
        advs, rets = gae_oracle.gae(torch.stack(rew).cpu().numpy(), values.reshape(N, T).t().cpu().numpy(),
                                    dones.reshape(N, T).t().cpu().numpy(), last_v.cpu().numpy(), prev_done.cpu().numpy(), 0.99, 0.95)
        assert np.allclose(returns.reshape(N, T).t().cpu().numpy(), rets, atol=1e-4)
    env.close(); twin.close()


def test_single_snake_ppo_learns_on_device_grid():
    """The grid twin of test_single_snake_ppo_learns_on_device, with the same thresholds."""
    import torch
    import snakes_b200
    from snakes_b200 import selfplay
    torch.manual_seed(0)
    env = snakes_b200.SnakeVecEnv(1024, size=10, n_snakes=1, seed=0, obs_mode="grid")
    model, log = selfplay.learn(env, nsteps=32, total_timesteps=1024 * 32 * 36, log_interval=6, seed=0)
    env.check_errors()
    assert model.net.grid
    first, last = log.rows[0], log.rows[-1]
    assert first["eprewmean 100"] < -0.8
    assert last["eprewmean 100"] > first["eprewmean 100"] + 0.5, (first, last)
    assert last["eplenmean"] > 3 * first["eplenmean"]
    for k in ("num_opponents", "serial_timesteps", "nupdates", "total_timesteps", "explained_variance", "eprewmean 100",
              "eplenmean", "time_elapsed", "ep_rew_mean", "policy_loss", "value_loss", "policy_entropy", "approxkl", "clipfrac"):
        assert k in last
    env.close()


def test_two_snake_self_play_pool_and_checkpoints_grid(tmp_path):
    """The grid twin of test_two_snake_self_play_pool_and_checkpoints: the checkpoint restores an RGB policy."""
    import joblib
    import torch
    import snakes_b200
    from snakes_b200 import selfplay
    torch.manual_seed(0)
    env = snakes_b200.SnakeVecEnv(256, size=10, n_snakes=2, seed=3, obs_mode="grid")
    d = str(tmp_path / "ppo")
    model, log = selfplay.learn(env, nsteps=16, total_timesteps=256 * 16 * 5, log_interval=1, model_dir=d,
                                opponent_save_interval=2, csv_path=str(tmp_path / "ppo.csv"), save_interval=2)
    env.check_errors()
    assert sorted(f for f in os.listdir(d) if f.startswith("opponent")) == ["opponent0_0.pkl", "opponent0_1.pkl", "opponent0_2.pkl"]
    assert log.rows[-1]["num_opponents"] == 3 and len(log.rows) == 5
    assert os.path.exists(os.path.join(d, "snake_model_num2_final.pkl"))
    params = joblib.load(os.path.join(d, "snake_model_num2_final.pkl"))
    assert len(params) == 14 and params[0].shape == (3, 3, 3, 32)
    m2 = selfplay.Model((12, 12, 3), 5, device=env.device, trainable=False)
    m2.load(os.path.join(d, "snake_model_num2_final.pkl"))
    assert torch.allclose(m2.net(snakes_b200.expand_views(env.obs, 1))[0], model.net(env.obs)[0], atol=1e-5)
    env.close()
