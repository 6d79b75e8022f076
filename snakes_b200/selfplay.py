"""On-device self-play PPO around the batched env (SURVEY.md section 8f, rows f2-f4).

The env step is the product of this repo; this module is the CALLER on the other side of the
rollout buffer, kept deliberately thin and in plain PyTorch: it exists so that the loop the
reference runs -- policy forward for the main snake and every opponent, env step, rollout buffer,
GAE, PPO2 update, opponent pool -- closes on the GPU with no host round trip, and so that the
interchange formats of the reference (joblib list of ndarrays in TF variable order, baselines
logger key names) have a writer / reader here.

Reference structure mirrored (src/ of the reference):
  policies.py:12-67            nature_cnn / custom_cnn / CnnPolicy  -> CnnPolicy
  ppo_multi_agent_new.py:20-46  MultiModel.multi_step                -> Runner._act
  ppo_multi_agent_new.py:48-135 Model (PPO2 loss, Adam eps=1e-5, global-norm clip, save / load)
  ppo_multi_agent_new.py:138-220 Runner.run (+ sf01)                 -> Runner.run
  ppo_multi_agent_new.py:234-390 learn (opponent pool: save every 50 updates, <= 1000, uniform)
  config.py:13-14               OPPONENT_SAVE_INTERVAL / MAX_SAVED_OPPONENTS
"""
import csv
import math
import os
import random
import time
from collections import deque

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from . import rollout as _rollout
from .grid_conv import conv84_supported, grid_conv84_in, grid_conv_in

OPPONENT_SAVE_INTERVAL = 50   # config.py:13
MAX_SAVED_OPPONENTS = 1000    # config.py:14


def _ortho_(w, scale):
    """baselines.a2c.utils.ortho_init: orthogonal over (prod(other dims), out)."""
    nn.init.orthogonal_(w, gain=scale)
    return w


class CnnPolicy(nn.Module):
    """policies.py:40-67.  `arch='custom'` is custom_cnn (four 3x3 SAME convs 32-32-64-64, fc 512;
    Config.USE_ATARI_SIZE False), `arch='nature'` is nature_cnn (8/4, 4/2, 3/1 VALID convs, fc 512; 84x84
    input).  Input: uint8 [B, H, W, C] exactly as the env writes it (NHWC); scaled by 1/255 here.

    `grid=True`: the input is a cell-code grid uint8 [B, V, V] (obs_mode 'grid') and the first conv, its bias and ReLU
    are computed from view `view` of it: the RGB view is never built.  `custom` (grid_conv_in) is the network of the RGB
    policy of ob_shape (V, V, 3); `nature` (grid_conv84_in, V dividing 84 with 3 <= V <= 42) is nature_cnn on the 84x84
    WarpFrame of the view, the network of the RGB policy of ob_shape (84, 84, 3) on an obs_mode 'atari84' env.  The
    parameters are the same, so checkpoints and to_tf_list / from_tf_list move between the two."""

    def __init__(self, ob_shape, n_actions, arch="custom", grid=False):
        super().__init__()
        h, w, c = ob_shape
        self.ob_shape, self.n_actions, self.arch, self.grid = tuple(ob_shape), int(n_actions), arch, bool(grid)
        if grid and c != 3:
            raise ValueError("grid=True needs ob_shape (V, V, 3), got %r" % (tuple(ob_shape),))
        if grid and arch == "nature":
            if h != w or not conv84_supported(h):
                raise ValueError("grid=True with arch 'nature' needs V dividing 84 with 3 <= V <= 42, got V = %d" % h)
            h = w = 84   # the network sees the WarpFrame view
        if arch == "nature":
            spec = [(32, 8, 4, 0), (64, 4, 2, 0), (64, 3, 1, 0)]
        elif arch == "custom":
            spec = [(32, 3, 1, 1), (32, 3, 1, 1), (64, 3, 1, 1), (64, 3, 1, 1)]
        else:
            raise ValueError("arch must be 'custom' or 'nature'")
        convs, cin = [], c
        for nf, rf, stride, pad in spec:
            conv = nn.Conv2d(cin, nf, rf, stride, pad)
            _ortho_(conv.weight, math.sqrt(2)); nn.init.zeros_(conv.bias)
            convs.append(conv)
            cin = nf
            h = (h + 2 * pad - rf) // stride + 1
            w = (w + 2 * pad - rf) // stride + 1
        self.convs = nn.ModuleList(convs)
        self.conv_out = (h, w, cin)
        self.fc1 = nn.Linear(h * w * cin, 512)
        self.pi = nn.Linear(512, self.n_actions)
        self.v = nn.Linear(512, 1)
        _ortho_(self.fc1.weight, math.sqrt(2)); nn.init.zeros_(self.fc1.bias)
        _ortho_(self.pi.weight, 0.01); nn.init.zeros_(self.pi.bias)
        _ortho_(self.v.weight, 1.0); nn.init.zeros_(self.v.bias)

    def forward(self, ob, view=0):
        """(logits, value).  `view`: which snake's view of a grid input is read (a grid policy only; an RGB input is
        already one view)."""
        if self.grid:
            conv_in = grid_conv84_in if self.arch == "nature" else grid_conv_in
            x = conv_in(ob, view, self.convs[0].weight, self.convs[0].bias)
            convs = self.convs[1:]
        else:
            x = ob.permute(0, 3, 1, 2).float() * (1.0 / 255.0)
            x = x.contiguous(memory_format=torch.channels_last)
            convs = self.convs
        for conv in convs:
            x = F.relu(conv(x))
        # conv_to_fc flattens NHWC (baselines.a2c.utils.conv_to_fc): keep that order so fc1 is interchangeable
        x = x.permute(0, 2, 3, 1).reshape(x.shape[0], -1)
        hid = F.relu(self.fc1(x))
        return self.pi(hid), self.v(hid)[:, 0]

    @torch.no_grad()
    def step(self, ob, view=0):
        """a0 = pd.sample(), vf, neglogp0 (policies.py:53-59); CategoricalPd samples with the Gumbel trick."""
        logits, v = self.forward(ob, view)
        u = torch.rand_like(logits).clamp_(1e-20, 1.0)
        a = torch.argmax(logits - torch.log(-torch.log(u)), dim=-1)
        return a, v, F.cross_entropy(logits, a, reduction="none")

    @torch.no_grad()
    def value(self, ob, view=0):
        return self.forward(ob, view)[1]

    # ---- interchange with the reference's checkpoints (ppo_multi_agent_new.py:104-125, evaluate_snake.py:21-40):
    # joblib list of ndarrays in tf.trainable_variables order: c1/w, c1/b, ..., fc1/w, fc1/b, pi/w, pi/b, v/w, v/b
    def to_tf_list(self):
        out = []
        for conv in self.convs:
            out.append(conv.weight.detach().permute(2, 3, 1, 0).cpu().numpy().copy())  # [kh, kw, in, out]
            out.append(conv.bias.detach().cpu().numpy().copy())
        for fc in (self.fc1, self.pi, self.v):
            out.append(fc.weight.detach().t().cpu().numpy().copy())                    # [in, out]
            out.append(fc.bias.detach().cpu().numpy().copy())
        return out

    @torch.no_grad()
    def from_tf_list(self, params):
        params = list(params)
        want = 2 * len(self.convs) + 6
        if len(params) != want:
            raise ValueError("expected %d arrays, got %d" % (want, len(params)))
        it = iter(params)
        for conv in self.convs:
            w, b = np.asarray(next(it)), np.asarray(next(it))
            if tuple(w.shape) != tuple(conv.weight.permute(2, 3, 1, 0).shape):
                raise ValueError("conv weight shape %s does not fit %s" % (w.shape, tuple(conv.weight.shape)))
            conv.weight.copy_(torch.from_numpy(w).permute(3, 2, 0, 1))
            conv.bias.copy_(torch.from_numpy(b))
        for fc in (self.fc1, self.pi, self.v):
            w, b = np.asarray(next(it)), np.asarray(next(it))
            if tuple(w.shape) != (fc.in_features, fc.out_features):
                raise ValueError("fc weight shape %s does not fit (%d, %d)" % (w.shape, fc.in_features, fc.out_features))
            fc.weight.copy_(torch.from_numpy(w).t())
            fc.bias.copy_(torch.from_numpy(b))
        return self


def ppo_loss(logits, vpred, actions, advs, returns, old_neglogp, old_v, cliprange, ent_coef, vf_coef):
    """The loss graph of Model.__init__ (ppo_multi_agent_new.py:62-77); returns (loss, stats[5])."""
    neglogp = F.cross_entropy(logits, actions, reduction="none")
    logp_all = F.log_softmax(logits, dim=-1)
    entropy = -(logp_all.exp() * logp_all).sum(-1).mean()
    vclipped = old_v + torch.clamp(vpred - old_v, -cliprange, cliprange)
    vf_loss = 0.5 * torch.maximum((vpred - returns) ** 2, (vclipped - returns) ** 2).mean()
    ratio = torch.exp(old_neglogp - neglogp)
    pg_loss = torch.maximum(-advs * ratio, -advs * torch.clamp(ratio, 1.0 - cliprange, 1.0 + cliprange)).mean()
    approxkl = 0.5 * ((neglogp - old_neglogp) ** 2).mean()
    clipfrac = ((ratio - 1.0).abs() > cliprange).float().mean()
    loss = pg_loss - entropy * ent_coef + vf_loss * vf_coef
    return loss, torch.stack([pg_loss, vf_loss, entropy, approxkl, clipfrac]).detach()


class Model(object):
    """ppo_multi_agent_new.py:48-135: one policy network with its PPO2 trainer, save / load.  `grid=True`: the network
    reads cell-code grids (CnnPolicy grid=True); `step` / `value` take the view index, `train` reads view 0."""

    loss_names = ["policy_loss", "value_loss", "policy_entropy", "approxkl", "clipfrac"]

    def __init__(self, ob_shape, n_actions, ent_coef=0.01, vf_coef=0.5, max_grad_norm=0.5, arch="custom", device="cuda",
                 trainable=True, grid=False):
        self.net = CnnPolicy(ob_shape, n_actions, arch, grid).to(device).to(memory_format=torch.channels_last)
        self.ent_coef, self.vf_coef, self.max_grad_norm = ent_coef, vf_coef, max_grad_norm
        self.opt = torch.optim.Adam(self.net.parameters(), lr=2.5e-4, eps=1e-5) if trainable else None
        self.step, self.value = self.net.step, self.net.value
        self.initial_state = None

    def train(self, lr, cliprange, obs, returns, masks, actions, values, neglogpacs, states=None):
        advs = returns - values
        advs = (advs - advs.mean()) / (advs.std(unbiased=False) + 1e-8)   # numpy std (:82-83)
        for g in self.opt.param_groups:
            g["lr"] = lr
        logits, vpred = self.net(obs)
        loss, stats = ppo_loss(logits, vpred, actions, advs, returns, neglogpacs, values, cliprange, self.ent_coef, self.vf_coef)
        self.opt.zero_grad(set_to_none=True)
        loss.backward()
        if torch.distributed.is_available() and torch.distributed.is_initialized() and torch.distributed.get_world_size() > 1:
            ws = torch.distributed.get_world_size()   # data-parallel learner: envs are sharded, gradients averaged
            for prm in self.net.parameters():
                torch.distributed.all_reduce(prm.grad)
                prm.grad.div_(ws)
        if self.max_grad_norm is not None:
            nn.utils.clip_grad_norm_(self.net.parameters(), self.max_grad_norm)
        self.opt.step()
        return stats

    def save(self, path):
        import joblib
        joblib.dump(self.net.to_tf_list(), path)

    def load(self, path):
        import joblib
        self.net.from_tf_list(joblib.load(path))

    def get_params(self):
        return [p.detach().clone() for p in self.net.parameters()]

    @torch.no_grad()
    def set_params(self, params):
        for p, q in zip(self.net.parameters(), params):
            p.copy_(q)


def _dist_world():
    d = torch.distributed
    return d.get_world_size() if d.is_available() and d.is_initialized() else 1


def sync_model_across_ranks(model, src=0):
    """Data-parallel learner: every rank builds its network from its own RNG, so the replicas must be made identical
    before the first update (gradients are averaged afterwards, Model.train).  Broadcasts parameters from `src`."""
    if _dist_world() > 1:
        for prm in model.net.parameters():
            torch.distributed.broadcast(prm.data, src)
    return model


def _is_rank0():
    return _dist_world() == 1 or torch.distributed.get_rank() == 0


def sf01(t):
    """swap and then flatten axes 0 and 1 (:222-227)."""
    return t.transpose(0, 1).reshape(t.shape[0] * t.shape[1], *t.shape[2:])


class Runner(object):
    """Runner of ppo_multi_agent_new.py:138-220 with every buffer on the device.

    On an obs_mode 'grid' env (with grid models only) the rollout keeps cell-code grids: mb_obs is uint8 [nsteps, N, V, V],
    the main model reads view 0 of a slot and opponent i view i + 1 of the same slot."""

    def __init__(self, env, model, opponent_models, nsteps, gamma=0.99, lam=0.95):
        self.env, self.model, self.opponents = env, model, list(opponent_models)
        self.nsteps, self.gamma, self.lam = nsteps, gamma, lam
        N, dev = env.num_envs, env.device
        self.grid = getattr(env, "obs_mode", "native") == "grid"
        if self.grid:
            self._init_grid(N, dev)
            return
        h, w, c = env.observation_space.shape
        if c < 3 * (1 + len(self.opponents)):
            raise ValueError("the env must emit one view per controlled snake (n_views >= n_snakes)")
        self.obs = env.reset()                      # uint8 [N, H, W, 3K], aliased device buffer
        self.dones = torch.zeros(N, dtype=torch.bool, device=dev)
        self.mb_obs = torch.empty((nsteps, N, h, w, 3), dtype=torch.uint8, device=dev)
        self.mb_rewards = torch.empty((nsteps, N), dtype=torch.float32, device=dev)
        self.mb_actions = torch.empty((nsteps, N), dtype=torch.int64, device=dev)
        self.mb_values = torch.empty((nsteps, N), dtype=torch.float32, device=dev)
        self.mb_neglogp = torch.empty((nsteps, N), dtype=torch.float32, device=dev)
        self.mb_dones = torch.empty((nsteps, N), dtype=torch.bool, device=dev)
        self.full_actions = torch.zeros((N, env.S), dtype=torch.int8, device=dev)
        self.main_spare = torch.empty((N, h, w, 3), dtype=torch.uint8, device=dev)  # main view after the rollout's last step
        self.main_next = None

    def _init_grid(self, N, dev):
        env, nsteps = self.env, self.nsteps
        if not all(getattr(getattr(m, "net", None), "grid", False) for m in [self.model] + [o for o in self.opponents if o is not None]):
            raise ValueError("a grid env needs grid models (Model(..., grid=True)): the rollout keeps cell-code grids, not RGB views")
        if 1 + len(self.opponents) > env.S:
            raise ValueError("%d models for %d snakes: one model per controlled snake" % (1 + len(self.opponents), env.S))
        V = env.V
        # slots 16-byte aligned: the env writes a step's grid straight into one (set_obs_target)
        slot = -(-N * V * V // 16) * 16
        self.mb_obs = torch.empty((nsteps, slot), dtype=torch.uint8, device=dev)[:, :N * V * V].view(nsteps, N, V, V)
        self.obs = env.reset()
        self.dones = torch.zeros(N, dtype=torch.bool, device=dev)
        self.mb_rewards = torch.empty((nsteps, N), dtype=torch.float32, device=dev)
        self.mb_actions = torch.empty((nsteps, N), dtype=torch.int64, device=dev)
        self.mb_values = torch.empty((nsteps, N), dtype=torch.float32, device=dev)
        self.mb_neglogp = torch.empty((nsteps, N), dtype=torch.float32, device=dev)
        self.mb_dones = torch.empty((nsteps, N), dtype=torch.bool, device=dev)
        self.full_actions = torch.zeros((N, env.S), dtype=torch.int8, device=dev)

    def _act_grid(self, grid):
        """MultiModel.multi_step on one grid: the main model reads view 0, opponent i view i + 1."""
        a, v, nlp = self.model.step(grid, 0)
        self.full_actions[:, 0] = a.to(torch.int8)
        for i, opp in enumerate(self.opponents):
            self.full_actions[:, i + 1] = 1 if opp is None else opp.step(grid, i + 1)[0].to(torch.int8)
        return a, v, nlp

    def _run_grid(self):
        """run() on a grid env: the env writes each step's grid into mb_obs[t + 1] through set_obs_target, and the last
        step's into its own buffer (the target is switched off), so env.obs is the current grid, the env never holds a
        pointer into the runner's memory, and slot 0 of the next rollout is one copy of it.  No view is expanded and no
        step is copied."""
        env = self.env
        before = env.stats(False)
        self.mb_obs[0].copy_(env.obs)
        for t in range(self.nsteps):
            a, v, nlp = self._act_grid(self.mb_obs[t])
            self.mb_actions[t], self.mb_values[t], self.mb_neglogp[t] = a, v, nlp
            self.mb_dones[t] = self.dones
            env.set_obs_target(self.mb_obs[t + 1] if t + 1 < self.nsteps else None)
            _, rew, dones, _ = env.step(self.full_actions)
            self.mb_rewards[t] = rew
            self.dones = dones.clone()
        self.obs = env.obs
        last_values = self.model.value(env.obs, 0)
        advs, returns = _rollout.gae(self.mb_rewards, self.mb_values, self.mb_dones, last_values, self.dones, self.gamma, self.lam)
        after = env.stats(False)
        ep = {k: after[k] - before[k] for k in ("episodes", "return_sum", "length_sum")}
        return (sf01(self.mb_obs), sf01(returns), sf01(self.mb_dones), sf01(self.mb_actions), sf01(self.mb_values),
                sf01(self.mb_neglogp), None, ep)

    def _views(self):
        """use_multi_agent_obs (:161-165): view 0 is the main snake's, view i + 1 opponent i's."""
        return [self.obs[..., 3 * i:3 * (i + 1)] for i in range(1 + len(self.opponents))]

    def _act(self, views):
        """MultiModel.multi_step (:24-41): the main model samples, every opponent acts on ITS view;
        an absent opponent plays action 1."""
        a, v, nlp = self.model.step(views[0])
        self.full_actions[:, 0] = a.to(torch.int8)
        for i, opp in enumerate(self.opponents):
            self.full_actions[:, i + 1] = 1 if opp is None else opp.step(views[i + 1])[0].to(torch.int8)
        return a, v, nlp

    def run(self):
        """The rollout loop of Runner.run (:178-198).  The env writes the main snake's view of the observation a step
        returns straight into the slot the NEXT step's policy call reads it from (set_main_view_target: mb_obs[t + 1],
        the last one into a spare slot), so mb_obs is filled by the env and the policy reads a contiguous [N,H,W,3]
        tensor; the opponents' views stay in the env's own transient buffer."""
        if self.grid:
            return self._run_grid()
        env = self.env
        before = env.stats(False)
        for t in range(self.nsteps):
            views = self._views()
            if t == 0:
                self.mb_obs[0].copy_(self.main_next if self.main_next is not None else views[0])
            a, v, nlp = self._act([self.mb_obs[t]] + views[1:])
            self.mb_actions[t], self.mb_values[t], self.mb_neglogp[t] = a, v, nlp
            self.mb_dones[t] = self.dones
            env.set_main_view_target(self.mb_obs[t + 1] if t + 1 < self.nsteps else self.main_spare)
            self.obs, rew, dones, _ = env.step(self.full_actions)
            self.mb_rewards[t] = rew
            self.dones = dones.clone()
        env.set_main_view_target(None)
        self.main_next = self.main_spare
        last_values = self.model.value(self.main_spare)
        advs, returns = _rollout.gae(self.mb_rewards, self.mb_values, self.mb_dones, last_values, self.dones, self.gamma, self.lam)
        after = env.stats(False)
        # Monitor's episode records of this rollout in aggregate (every finished episode, not a sample)
        ep = {k: after[k] - before[k] for k in ("episodes", "return_sum", "length_sum")}
        return (sf01(self.mb_obs), sf01(returns), sf01(self.mb_dones), sf01(self.mb_actions), sf01(self.mb_values),
                sf01(self.mb_neglogp), None, ep)


class KVLogger(object):
    """The key/value rows `learn` writes through baselines.logger.CSVOutputFormat (:249, :357-377):
    same key names, one CSV row per logged update (keys are fixed by the first row)."""

    def __init__(self, csv_path=None, echo=False):
        self.kvs, self.rows, self.echo = {}, [], echo
        self._fh, self._writer = (open(csv_path, "w", newline="") if csv_path else None), None

    def logkv(self, k, v):
        self.kvs[k] = v

    def dumpkvs(self):
        row = dict(self.kvs)
        self.rows.append(row)
        if self._fh:
            if self._writer is None:
                self._writer = csv.DictWriter(self._fh, fieldnames=list(row.keys()), extrasaction="ignore")
                self._writer.writeheader()
            self._writer.writerow(row)
            self._fh.flush()
        if self.echo:
            print(" | ".join("%s %s" % (k, ("%.4g" % v) if isinstance(v, float) else v) for k, v in row.items()), flush=True)
        self.kvs = {}
        return row

    def close(self):
        if self._fh:
            self._fh.close()
            self._fh = None


def explained_variance(ypred, y):
    """baselines.common.math_util.explained_variance: 1 - Var[y - ypred] / Var[y]."""
    vary = y.var(unbiased=False)
    return float("nan") if float(vary) == 0 else float(1 - (y - ypred).var(unbiased=False) / vary)


def learn(env, nsteps=128, total_timesteps=int(1e6), ent_coef=0.01, lr=2.5e-4, vf_coef=0.5, max_grad_norm=0.5,
          gamma=0.99, lam=0.95, log_interval=10, nminibatches=4, noptepochs=4, cliprange=0.2, save_interval=0,
          arch="custom", model_dir=None, csv_path=None, echo=False, opponent_save_interval=OPPONENT_SAVE_INTERVAL,
          max_saved_opponents=MAX_SAVED_OPPONENTS, seed=0, max_minibatch=32768):
    """learn of ppo_multi_agent_new.py:234-390: self-play PPO2 against a pool of past selves.

    `lr` / `cliprange`: floats or callables of the remaining fraction.  The opponent pool lives on the
    device (and, with `model_dir`, also as the reference's opponent{i}_{k}.pkl joblib files).  Returns
    (model, logger)."""
    lr_fn = lr if callable(lr) else (lambda _f, _v=lr: _v)
    clip_fn = cliprange if callable(cliprange) else (lambda _f, _v=cliprange: _v)
    rng = random.Random(seed)
    N, S, dev = env.num_envs, env.S, env.device
    h, w = env.observation_space.shape[:2]
    ob_shape = (h, w, 3)
    grid = getattr(env, "obs_mode", "native") == "grid"   # grid models: the rollout and the minibatches hold cell codes
    n_act = env.action_space.n
    nbatch = N * nsteps
    assert nbatch % nminibatches == 0
    nbatch_train = nbatch // nminibatches
    mk = lambda trainable: Model(ob_shape, n_act, ent_coef, vf_coef, max_grad_norm, arch, dev, trainable, grid)
    model = sync_model_across_ranks(mk(True))   # one model, N replicas: identical weights from the first update on
    opponent_models = [mk(False) for _ in range(S - 1)]
    # opponent sampling uses `rng`, seeded identically on every rank, so all ranks load the same past selves
    write = model_dir is not None and _is_rank0()   # checkpoints and opponent files are written by rank 0 only
    runner = Runner(env, model, opponent_models, nsteps, gamma, lam)
    logger = KVLogger(csv_path if _is_rank0() else None, echo and _is_rank0())
    epbuf = deque()          # (episodes, return_sum, length_sum) per rollout, newest last; covers >= 100 episodes
    maxlen = 100
    if write:
        os.makedirs(model_dir, exist_ok=True)
    pool = [[] for _ in range(S - 1)]
    idx = [0] * (S - 1)

    def save_opponent(i):
        snap = model.get_params()
        if idx[i] < len(pool[i]):
            pool[i][idx[i]] = snap
        else:
            pool[i].append(snap)
        if write:
            model.save(os.path.join(model_dir, "opponent%d_%d.pkl" % (i, idx[i])))
        idx[i] = (idx[i] + 1) % max_saved_opponents

    for i in range(S - 1):
        save_opponent(i)
    nupdates = max(total_timesteps // nbatch, 1)
    t_first = time.time()
    for update in range(1, nupdates + 1):
        for i, opp in enumerate(opponent_models):                      # :300-304
            opp.set_params(pool[i][rng.randint(0, max(len(pool[i]) - 1, 0))])
        frac = 1.0 - (update - 1.0) / nupdates
        lrnow, clipnow = lr_fn(frac), clip_fn(frac)
        obs, returns, masks, actions, values, neglogpacs, _, ep = runner.run()
        epbuf.append(ep)
        while len(epbuf) > 1 and sum(e["episodes"] for e in list(epbuf)[1:]) >= maxlen:
            epbuf.popleft()
        losses = []
        chunk = min(nbatch_train, max_minibatch)
        for _ in range(noptepochs):                                    # :317-324
            inds = torch.randperm(nbatch, device=dev)
            for start in range(0, nbatch, chunk):
                mb = inds[start:start + chunk]
                losses.append(model.train(lrnow, clipnow, obs[mb], returns[mb], masks[mb], actions[mb], values[mb], neglogpacs[mb]))
        for i in range(S - 1):                                         # :332-341
            if update % opponent_save_interval == 0:
                save_opponent(i)
        if update % log_interval == 0 or update == 1:
            n_ep = sum(e["episodes"] for e in epbuf)
            ep_rew_mean = sum(e["return_sum"] for e in epbuf) / n_ep if n_ep else float("nan")
            ep_len_mean = sum(e["length_sum"] for e in epbuf) / n_ep if n_ep else float("nan")
            lossvals = torch.stack(losses).mean(0).tolist()
            logger.logkv("num_opponents", len(pool[0]) if pool else 0)
            logger.logkv("serial_timesteps", update * nsteps)
            logger.logkv("nupdates", update)
            logger.logkv("total_timesteps", update * nbatch)
            logger.logkv("explained_variance", explained_variance(values, returns))
            logger.logkv("eprewmean %d" % maxlen, ep_rew_mean)
            logger.logkv("eplenmean", ep_len_mean)
            logger.logkv("time_elapsed", time.time() - t_first)
            logger.logkv("ep_rew_mean", ep_rew_mean)
            for name, val in zip(Model.loss_names, lossvals):
                logger.logkv(name, val)
            logger.dumpkvs()
        if save_interval and write and (update % save_interval == 0 or update == 1):
            model.save(os.path.join(model_dir, "snake_model_num%d_%d.pkl" % (S, update)))
    if write:
        model.save(os.path.join(model_dir, "snake_model_num%d_final.pkl" % S))
    logger.close()
    return model, logger
