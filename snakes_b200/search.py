"""Rollout search on the device: a player that needs no training (DESIGN.md section 4.19).

For every root env it clones the env into A x R slots of a second handle (A candidate actions, R rollouts each), plays
each candidate on the first step and a rollout policy after it for H steps, and picks the candidate of the largest summed
return.  The clones live in their own handle (snk_clone_envs), so the game env is only read.
"""
import ctypes as C

import torch

from . import _lib
from .vec_env import SnakeVecEnv

ROLLOUT_POLICIES = ("scripted", "random")


def check_args(env, rollouts, horizon, rollout):
    """ValueError unless a search with these arguments can run on `env`."""
    if rollout not in ROLLOUT_POLICIES:
        raise ValueError("rollout must be 'scripted' or 'random', got %r" % (rollout,))
    if rollout == "scripted" and (env.cfg.rules != _lib.RULES["classic"] or env.launch_info()["kind"] != 0):
        raise ValueError("scripted rollouts need a lane-family env with classic rules (snk_gen_scripted_actions)")
    if int(rollouts) < 1:
        raise ValueError("rollouts must be >= 1, got %d" % rollouts)
    if int(horizon) < 1:
        raise ValueError("horizon must be >= 1, got %d" % horizon)


def _layout(env):
    """What snk_clone_envs needs to match beyond the configuration: the body family and the ring capacity (record, chain
    and fruit-grid sizes follow from them and the configuration)."""
    return env.launch_info()["kind"] == 0, int(env.lay.cap)


class RolloutSearch(object):
    """Picks one seat's action for up to `max_roots` envs of `env` by rollouts on a handle of its own.

    The search handle holds max_roots x A x R envs, A = env.action_space.n (5, or 6 under cut rules, where strike is a
    candidate) and R = `rollouts`.  It has the game env's configuration, seed and debug string with obs_mode 'grid' (the
    rollouts never read an image); when that handle cannot be created or its private layout differs from the game
    env's, it takes the game env's own obs_mode.  It is reset once when the search is built.

    act(seat, roots) with M = len(roots) follows this rule exactly; `calls` is the number of earlier act calls:
      1. slot j = (m A + a) R + r is cloned from env roots[m] of the game env (m < M, a < A, r < R);
      2. for k = 0 .. H-1 (H = `horizon`) the rollout policy writes every seat's actions of every slot of the search
         handle: gen_scripted_actions(calls H + k, seed, eps) for 'scripted', gen_actions(calls H + k, seed) for
         'random';
      3. at k = 0, seat `seat`'s action of slot j is overwritten with its candidate a = (j / R) % A;
      4. the search handle steps, then each slot adds seat's reward to its return; the step on which the seat gets -1
         (it died) or the slot's env is done is the slot's last counted step;
      5. after the last step V[m][a] = the sum of the returns of the R slots of (m, a), and the action of root m is the
         lowest a of maximal V[m][a].
    Slots at and beyond M A R step too but are never counted.  The game env is not touched: its state, statistics and
    observations are as they were.  Everything runs on the device without a synchronisation; V of the last call is
    `values[:M]` (float [M, A])."""

    def __init__(self, env, max_roots, rollouts=8, horizon=16, rollout="scripted", eps=0.05, seed=1):
        check_args(env, rollouts, horizon, rollout)
        if int(max_roots) < 1:
            raise ValueError("max_roots must be >= 1, got %d" % max_roots)
        self.env = env
        self.max_roots, self.R, self.H = int(max_roots), int(rollouts), int(horizon)
        self.A = env.action_space.n
        self.rollout, self.eps, self.seed = rollout, float(eps), int(seed)
        self.calls = 0
        N = self.max_roots * self.A * self.R
        self.search_env = se = self._make(env, N)
        se.reset()
        dev = env.device
        self._slots = torch.arange(N, dtype=torch.int64, device=dev)
        self._actions = torch.zeros((N, env.S), dtype=torch.int8, device=dev)
        self._ret = torch.zeros(N, dtype=torch.int32, device=dev)
        self._active = torch.zeros(N, dtype=torch.uint8, device=dev)
        self.values = torch.zeros((self.max_roots, self.A), dtype=torch.float32, device=dev)
        self._pick = torch.zeros(self.max_roots, dtype=torch.int8, device=dev)

    @staticmethod
    def _make(env, N):
        c = env.cfg
        kw = dict(size=c.size, n_snakes=c.n_snakes, n_fruits=c.n_fruits, n_views=c.n_views, rules=c.rules, seed=c.seed,
                  device=c.device, auto_reset=bool(c.auto_reset), max_steps=c.max_steps, debug=env._debug)
        if env.obs_mode != "grid":
            try:
                se = SnakeVecEnv(N, obs_mode="grid", **kw)
            except _lib.SnkError:
                se = None
            if se is not None:
                if _layout(se) == _layout(env):
                    return se
                se.close()
        return SnakeVecEnv(N, obs_mode=env.obs_mode, **kw)

    def act(self, seat, roots, out=None):
        """Seat `seat`'s action for each env of `roots` (int64 CUDA tensor of M <= max_roots game-env indices), by the
        rule of the class docstring.  Returns int8 [M]: `out` when given (any int8 CUDA view of M elements, such as
        column `seat` of rows of the game env's [N, S] action tensor), else a buffer the next call overwrites."""
        S = self.env.S
        if isinstance(seat, bool) or not isinstance(seat, int) or not 0 <= seat < S:
            raise ValueError("seat must be an int in [0, %d), got %r" % (S, seat))
        if not isinstance(roots, torch.Tensor) or not roots.is_cuda or roots.dtype != torch.int64 or roots.dim() != 1:
            raise TypeError("roots must be a 1-D int64 CUDA tensor")
        M = int(roots.numel())
        if not 1 <= M <= self.max_roots:
            raise ValueError("%d roots outside [1, max_roots = %d]" % (M, self.max_roots))
        if out is None:
            out = self._pick[:M]
        elif (not isinstance(out, torch.Tensor) or out.dtype != torch.int8 or out.device != self.env.device
              or out.dim() != 1 or out.numel() != M or out.stride(0) < 1):
            raise ValueError("out must be an int8 tensor of %d elements on %s" % (M, self.env.device))
        A, R, H = self.A, self.R, self.H
        n = M * A * R
        se = self.search_env
        L, h, stream = se._L, se._h, se._stream()
        se.clone_envs_from(self.env, roots.contiguous().repeat_interleave(A * R), self._slots[:n], observe=False)
        acts = C.c_void_p(self._actions.data_ptr())
        ret, active = C.c_void_p(self._ret.data_ptr()), C.c_void_p(self._active.data_ptr())
        for k in range(H):
            t = self.calls * H + k
            if self.rollout == "scripted":
                se.gen_scripted_actions(t, self.seed, self.eps, out=self._actions)
            else:
                se.gen_actions(t, self.seed, out=self._actions)
            if k == 0:
                _lib.check(L.snk_search_begin(h, acts, seat, A, R, M, ret, active, stream))
            se.step(self._actions)
            _lib.check(L.snk_search_accumulate(h, seat, A, R, M, ret, active, stream))
        _lib.check(L.snk_search_pick(h, A, R, M, ret, C.c_void_p(self.values.data_ptr()), C.c_void_p(out.data_ptr()),
                                     out.stride(0), stream))
        self.calls += 1
        return out

    def close(self):
        self.search_env.close()
