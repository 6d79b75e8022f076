"""SnakeVecEnv -- the reference's VecEnv protocol over the CUDA library.

Drop-in for what `utils.make_basic_env` returns in the reference (src/utils.py:34-49):
a `SubprocVecEnv` (src/baselines/common/vec_env/subproc_vec_env.py:31) of
`Monitor(SnakeEnv)` instances.  Same attributes and methods -- `num_envs`,
`observation_space`, `action_space`, `reset()`, `step_async()`, `step_wait()`, `step()`,
`close()` (src/baselines/common/vec_env/__init__.py:22-88) -- but all N envs live in HBM and
one fused kernel steps them.  Observations, rewards and dones are returned as CUDA tensors that
alias the library's buffers (no copy, no host round trip: consume them before the next step, or
clone); `host_io=True` returns numpy arrays like SubprocVecEnv.step_wait (`:57-61`): float64
rewards, bool dones, fresh arrays every step (`host_copy=False` hands out views of the pinned
staging buffers instead, for callers that consume an observation before the next step).
"""
import ctypes as C
import weakref

import numpy as np
import torch

from . import _lib
from .spaces import Box, Discrete


class _DevPtr(object):
    """A raw device pointer presented through __cuda_array_interface__ so torch can alias it."""

    def __init__(self, ptr, shape, typestr):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (int(ptr), False), "version": 2}


def _alias(ptr, shape, typestr, device):
    return torch.as_tensor(_DevPtr(ptr, shape, typestr), device=device)


def tile_images(img_nhwc):
    """N images -> one P x Q mosaic, P = ceil(sqrt(N)), Q = ceil(N / P), missing tiles black
    (the layout of baselines/common/tile_images.py:3-22)."""
    img = np.asarray(img_nhwc)
    n, h, w, c = img.shape
    P = int(np.ceil(np.sqrt(n)))
    Q = int(np.ceil(float(n) / P))
    canvas = np.zeros((P * Q, h, w, c), dtype=img.dtype)
    canvas[:n] = img
    return canvas.reshape(P, Q, h, w, c).transpose(0, 2, 1, 3, 4).reshape(P * h, Q * w, c)


class Infos(object):
    """Lazily materialised `infos` of one step: behaves like the tuple of per-env dicts that
    SubprocVecEnv returns ({'ale.lives': 1, 'num_snakes': n[, 'episode': {'r','l','t'}]},
    snake_multiple_test.py:197 + monitor.py:62-76) but only touches the host when indexed.

    Like SubprocVecEnv's infos it describes ITS step for good: the env snapshots the (small)
    device arrays behind an Infos object that is still alive and unread when the next step is
    launched (`_freeze`), so reading it later never reports the next step's episodes."""

    def __init__(self, num_alive, done, ep_ret, ep_len, elapsed, block=None):
        self._dev = (num_alive, done, ep_ret, ep_len)
        self._block = block      # the one device block the four arrays live in (snk_buffers.d_info_block)
        self._host = None
        self._elapsed = elapsed
        self._n = int(done.shape[0])

    def _freeze(self):
        """Called by the env before it overwrites the live buffers: keep this step's values."""
        if self._host is not None or not isinstance(self._dev[0], torch.Tensor):
            return
        if self._block is not None:
            snap = self._block.clone()   # one copy: the four arrays share a block
            base = self._block.data_ptr()
            self._dev = tuple(snap[x.data_ptr() - base: x.data_ptr() - base + x.numel() * x.element_size()].view(x.dtype)
                              for x in self._dev)
        else:
            self._dev = tuple(x.clone() for x in self._dev)
        self._block = None

    def _fetch(self):
        if self._host is None:
            self._host = tuple(np.asarray(x.cpu() if isinstance(x, torch.Tensor) else x) for x in self._dev)
            self._dev = self._block = None
        return self._host

    def __len__(self):
        return self._n

    def __getitem__(self, i):
        alive, done, ret, length = self._fetch()
        if i < 0:
            i += self._n
        if not 0 <= i < self._n:
            raise IndexError(i)
        info = {"ale.lives": 1, "num_snakes": int(alive[i])}
        if done[i]:
            info["episode"] = {"r": round(float(ret[i]), 6), "l": int(length[i]), "t": self._elapsed}
        return info

    def __iter__(self):
        return (self[i] for i in range(self._n))

    def episodes(self):
        """[{'r','l','t'}] of the envs that finished this step (what Runner.run collects,
        ppo_multi_agent_new.py:189-192) without building N dicts."""
        _, done, ret, length = self._fetch()
        idx = np.flatnonzero(done)
        return [{"r": round(float(ret[i]), 6), "l": int(length[i]), "t": self._elapsed} for i in idx]


class MonitorCSV(object):
    """The per-episode log baselines' Monitor writes when it is given a file name (bench/monitor.py:27-36, :62-76):
    a `#{"t_start": ..., "env_id": ...}` header line, then `r,l,t` rows, one per finished episode, in the order the
    episodes ended.  (The reference's make_basic_env passes filename=None, utils.py:40, so it writes none; this is for
    callers that want the file the plotting scripts read.)  Feed it the `infos` of every step."""

    EXT = "monitor.csv"

    def __init__(self, path, env_id="snake", t_start=None):
        import json
        import time
        if not path.endswith(self.EXT):
            path = path + "." + self.EXT if not path.endswith(".") else path + self.EXT
        self.path = path
        self.f = open(path, "wt")
        self.f.write("#%s\n" % json.dumps({"t_start": time.time() if t_start is None else t_start, "env_id": env_id}))
        self.f.write("r,l,t\n")
        self.f.flush()
        self.episodes = 0

    def write(self, infos):
        for ep in infos.episodes():
            self.f.write("%s,%d,%s\n" % (ep["r"], ep["l"], ep["t"]))
            self.episodes += 1
        self.f.flush()

    def close(self):
        if self.f:
            self.f.close()
            self.f = None


class StepGraph(object):
    """T env steps captured as one CUDA graph (snk_graph_create): a single launch per rollout,
    kernels linked by programmatic dependent-launch edges, no Python in the loop."""

    def __init__(self, env, handle, keep):
        self._env, self._g, self._keep = env, handle, keep

    def launch(self):
        self._env._before_overwrite()
        _lib.check(self._env._L.snk_graph_launch(self._g, self._env._stream()))

    def close(self):
        if self._g is not None and not self._env.closed:
            torch.cuda.synchronize(self._env.device)
            self._env._L.snk_graph_destroy(self._g)
        self._g = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class SnakeVecEnv(object):
    """N multi-snake envs stepped in lockstep on one GPU.

    kwargs follow NewMultipleSnakes.__init__ (gym_snake/envs/snake_multiple_env_new.py:10):
    `size`, `n_snakes`, `n_fruits`, `screen_res` (accepted, unused: no pyglet viewer), plus the
    batch / device ones: `num_envs`, `rules` ('classic' | 'adversarial' | 'cut'), `n_views`
    (K; the reference's SnakeEnv emits 3, snake_multiple_test.py:93-95), `seed`, `device`,
    `env_id_base` (global id of env 0: shard offset under multi-GPU), `auto_reset`, `obs_mode`
    ('native' [V,V,3K] or 'atari84' [84,84,3K]: the reference's WarpFrame, utils.py:15-31; exact
    pixel replication, so it needs 84 % (size + 2) == 0, e.g. size 10 or 19; or 'grid' [V,V]: one
    cell code per cell (CELL_* constants), lossless for all K views at 1/(3K) of the bytes --
    `expand_views(obs, K)` is the native observation).
    Host I/O: `host_io=True` (numpy in / numpy out), `host_views` (how many views of each pixel
    come back, default all K; 1 = the main snake's view only, ppo_multi_agent_new.py:181; not with 'grid'),
    `host_copy` (default True: fresh arrays every step like np.stack; False: views of the pinned,
    NUMA-local staging buffers).  `debug`: experiment switches, a "key=value,..." string
    (include/snk.h, snk_create_ex); None reads the SNK_DEBUG environment variable.
    `obs` (device tensor [N, H, W, 3K]) is the handle's own observation buffer and is read-only for callers: a step
    rewrites only the 32-byte pieces of it that can have changed since the previous frame, so whatever is written into
    it between steps may survive them.  Copy it (or use set_obs_target / rollout buffers) to modify observations.
    """

    def __init__(self, num_envs, size=(10, 10), n_snakes=2, n_fruits=None, n_views=None, rules="classic",
                 seed=0, device=0, env_id_base=0, auto_reset=True, max_steps=2000, screen_res=300, host_io=False,
                 obs_mode="native", host_views=None, host_copy=True, debug=None):
        import time
        self.closed = True
        self._L = _lib.lib()
        if isinstance(device, torch.device):
            device = device.index or 0
        elif isinstance(device, str):
            device = torch.device(device).index or 0
        if obs_mode not in _lib.OBS_MODES:
            raise ValueError("obs_mode must be 'native', 'atari84' or 'grid'")
        if obs_mode == "grid" and host_views is not None:
            raise ValueError("obs_mode 'grid' returns the whole grid: host_views must be None (expand views on the device)")
        self.obs_mode = obs_mode
        self.cfg = _lib.make_config(num_envs, size, n_snakes, n_fruits, n_views, rules, max_steps, auto_reset,
                                    obs_mode=_lib.OBS_MODES[obs_mode],
                                    device=device, env_id_base=env_id_base, seed=seed)
        self.device = torch.device("cuda", self.cfg.device)
        torch.cuda.init()
        h = C.c_void_p()
        self._debug = debug
        if debug is None:
            _lib.check(self._L.snk_create(C.byref(self.cfg), C.byref(h)))
        else:
            _lib.check(self._L.snk_create_ex(C.byref(self.cfg), str(debug).encode(), C.byref(h)))
        self._h = h
        self.closed = False
        self.lay = _lib.SnkStateLayout()
        _lib.check(self._L.snk_state_layout_of(C.byref(self.cfg), C.byref(self.lay)))
        self.num_envs = self.N = self.cfg.num_envs
        self.S, self.F, self.K, self.D = self.cfg.n_snakes, self.cfg.n_fruits, self.cfg.n_views, self.cfg.size
        self.V = self.D + 2
        self.rules = rules
        self.screen_res = screen_res
        self.host_io = host_io
        self.host_copy = bool(host_copy)
        self.host_views = None if obs_mode == "grid" else self.K if not host_views else int(host_views)
        if obs_mode != "grid" and not 1 <= self.host_views <= self.K:
            raise ValueError("host_views must be 1..n_views")
        self._last_infos = None
        self._graphs = {}
        self.action_space = Discrete(6 if self.cfg.rules == _lib.RULES["cut"] else 5)
        self._bind_buffers()
        self.observation_space = Box(0, 255, tuple(self.obs.shape[1:]), np.uint8)
        self._actions = torch.zeros((self.N, self.S), dtype=torch.int8, device=self.device)
        self._pending = False
        self._tstart = time.time()
        self._time = time
        self.host_numa_node = None
        if host_io:
            # pinned staging buffers from the C layer, placed on the GPU's NUMA node (snk_host_alloc)
            oshape = tuple(self.obs.shape) if obs_mode == "grid" else tuple(self.obs.shape[:3]) + (3 * self.host_views,)
            self._h_actions = self._host_array((self.N, self.S), np.int8)
            self._h_obs = self._host_array(oshape, np.uint8)
            self._h_reward = self._host_array((self.N,), np.float32)
            self._h_done = self._host_array((self.N,), np.uint8)
            self._h_alive = self._host_array((self.N,), np.uint8)
            self.observation_space = Box(0, 255, oshape[1:], np.uint8)

    def _host_array(self, shape, dtype):
        n = int(np.prod(shape)) * np.dtype(dtype).itemsize
        ptr, node = C.c_void_p(), C.c_int32(-1)
        _lib.check(self._L.snk_host_alloc(self._h, max(n, 1), C.byref(ptr), C.byref(node)))
        self.host_numa_node = node.value
        buf = (C.c_uint8 * max(n, 1)).from_address(ptr.value)
        return np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)

    def _bind_buffers(self):
        b = _lib.SnkBuffers()
        _lib.check(self._L.snk_get_buffers(self._h, C.byref(b)))
        N, S, dev = self.N, self.S, self.device
        shape = (N, b.obs_h, b.obs_w) if self.obs_mode == "grid" else (N, b.obs_h, b.obs_w, b.obs_c)
        self.obs = _alias(b.d_obs, shape, "|u1", dev)
        self.rewards = _alias(b.d_reward, (N,), "<f4", dev)
        self.rewards_all = _alias(b.d_reward_all, (N, S), "<f4", dev)
        self._done_u8 = _alias(b.d_done, (N,), "|u1", dev)
        self.num_alive = _alias(b.d_num_alive, (N,), "|u1", dev)
        self.episode_return = _alias(b.d_episode_return, (N,), "<f4", dev)
        self.episode_len = _alias(b.d_episode_len, (N,), "<i4", dev)
        self._stats = _alias(b.d_stats, (_lib.NSTATS,), "<f8", dev)
        self._info_block = _alias(b.d_info_block, (b.info_block_bytes,), "|u1", dev)
        self._own = (self.obs, self.rewards, self._done_u8)   # the handle's buffers (a rollout re-points the live names)

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    # ------------------------------------------------------------------ VecEnv protocol
    def seed(self, seed=None):
        """env.seed(seed + rank) of utils.py:39: re-keys the counter-based RNG.  Takes effect on a
        fresh handle, so it is only allowed before the first reset."""
        if seed is None:
            return [int(self.cfg.seed)]
        state = self.dump_state()
        fresh = not state["t"].any() and not state["len"].any()
        if not fresh:
            raise _lib.SnkError("seed() must be called before the first reset()")
        self.close()
        self.__init__(self.N, self.D, self.S, self.F, self.K, self.rules, seed, self.cfg.device, self.cfg.env_id_base,
                      bool(self.cfg.auto_reset), self.cfg.max_steps, self.screen_res, self.host_io, self.obs_mode,
                      self.host_views, self.host_copy, self._debug)
        return [int(seed)]

    def _before_overwrite(self):
        """The live buffers are about to change: freeze the previous step's infos if somebody still holds them."""
        li = self._last_infos() if self._last_infos is not None else None
        if li is not None:
            li._freeze()
        self._last_infos = None
        self.obs, self.rewards, self._done_u8 = self._own

    def _host_obs(self):
        """[N,H,W,3K] (or the first host_views views; [N,V,V] in grid mode) of the current device observations as numpy."""
        if self.host_views is None or self.host_views == self.K:
            return self.obs.cpu().numpy()
        return self.obs[..., :3 * self.host_views].contiguous().cpu().numpy()

    def reset(self, mask=None):
        """VecEnv.reset (subproc_vec_env.py:63-66).  `mask` (bool [N], optional extension) resets a subset."""
        m = None
        if mask is not None:
            m = torch.as_tensor(mask, device=self.device).to(torch.uint8).contiguous()
        self._before_overwrite()
        _lib.check(self._L.snk_reset(self._h, C.c_void_p(m.data_ptr()) if m is not None else None, self._stream()))
        if self.host_io:
            return self._host_obs()
        return self.obs

    def step_async(self, actions):
        """actions: [N][S] ints -- a CUDA int8 tensor is used as is; sequences of tuples (what
        MultiModel.multi_step builds, ppo_multi_agent_new.py:35-37) and numpy arrays are copied.
        The step (with host_io: the H2D copy, the step and the D2H copies) is enqueued here;
        step_wait hands out the results."""
        if self._pending:
            raise _lib.SnkError("already running an async step")
        self._before_overwrite()
        if self.host_io:
            self._h_actions[...] = np.asarray(actions).reshape(self.N, self.S)
            p = lambda a: C.c_void_p(a.ctypes.data)
            _lib.check(self._L.snk_step_host_async(self._h, p(self._h_actions), p(self._h_obs), self.host_views or 0, p(self._h_reward),
                                                   p(self._h_done), p(self._h_alive), self._stream()))
        else:
            if isinstance(actions, torch.Tensor) and actions.is_cuda and actions.dtype == torch.int8 and actions.is_contiguous():
                a = actions.view(self.N, self.S)
            else:
                a = torch.as_tensor(np.asarray(actions) if not isinstance(actions, torch.Tensor) else actions)
                self._actions.copy_(a.reshape(self.N, self.S).to(torch.int8), non_blocking=True)
                a = self._actions
            self._a_live = a  # keep alive until step_wait
            _lib.check(self._L.snk_step(self._h, C.c_void_p(a.data_ptr()), self._stream()))
        self._pending = True

    def step_wait(self):
        if not self._pending:
            raise _lib.SnkError("not running an async step")
        self._pending = False
        elapsed = round(self._time.time() - self._tstart, 6)
        if self.host_io:
            # Monitor's r / l of the envs that finished, fetched behind the big copies (two [N] arrays)
            ret, length = self.episode_return.cpu().numpy(), self.episode_len.cpu().numpy()  # synchronises the stream
            done = self._h_done.astype(bool)
            infos = Infos(self._h_alive.copy(), done, ret, length, elapsed)
            obs = self._h_obs.copy() if self.host_copy else self._h_obs
            return obs, self._h_reward.astype(np.float64), done, infos  # np.stack of python floats is float64 (:61)
        dones = self._done_u8.view(torch.bool)
        infos = Infos(self.num_alive, self._done_u8, self.episode_return, self.episode_len, elapsed, self._info_block)
        self._last_infos = weakref.ref(infos)
        return self.obs, self.rewards, dones, infos

    def step(self, actions):
        self.step_async(actions)
        return self.step_wait()

    # ------------------------------------------------------------------ pipelined host step, observations stay in HBM
    SCALAR_SLOTS = 4   # SNK_SCALAR_SLOTS of include/snk.h
    def step_scalars_async(self, actions):
        """The step for a learner that lives on the GPU but is driven from the host (north_star: observations never
        leave HBM): numpy `actions` [N][S] go through a pinned, NUMA-local slot to the device, the fused kernel steps,
        and reward / done / num_snakes / Monitor r, l come back as ONE block into the slot's pinned memory
        (snk_step_scalars_async: the copies run on streams of their own beside the step stream, so the H2D of the next
        step and the D2H of the previous one overlap the kernel).  Nothing synchronises; four steps may be in flight, and
        the call blocks only when the slot it is about to reuse (four steps back) has not arrived yet.  Returns a
        ticket for `wait_scalars`.  The observations of the step are `self.obs` (device tensor, stream-ordered) or the
        rollout slot set with set_obs_target / set_main_view_target; `self.rewards` etc. are NOT written."""
        ring = getattr(self, "_ring", None)
        if ring is None:
            lay = (C.c_size_t * 6)()
            _lib.check(self._L.snk_scalars_layout(self._h, lay))
            ring = []
            for _ in range(self.SCALAR_SLOTS):
                act = self._host_array((self.N, self.S), np.int8)
                blk = self._host_array((int(lay[0]),), np.uint8)
                part = lambda k, dt: blk[int(lay[1 + k]):int(lay[1 + k]) + self.N * np.dtype(dt).itemsize].view(dt)
                ring.append((act, blk, (part(0, np.float32), part(1, np.uint8), part(2, np.uint8), part(3, np.float32), part(4, np.int32))))
            self._ring, self._ring_head = ring, 0
        if self._pending:
            raise _lib.SnkError("already running an async step")
        slot = self._ring_head % self.SCALAR_SLOTS
        act, blk, _ = ring[slot]
        _lib.check(self._L.snk_scalars_wait(self._h, slot))   # the slot's previous trip is over (H2D read, D2H written)
        np.copyto(act, np.asarray(actions).reshape(self.N, self.S), casting="unsafe")
        self._before_overwrite()
        _lib.check(self._L.snk_step_scalars_async(self._h, C.c_void_p(act.ctypes.data), C.c_void_p(blk.ctypes.data), slot, self._stream()))
        self._ring_head += 1
        return self._ring_head - 1

    def wait_scalars(self, ticket):
        """(reward float32, done uint8, num_snakes uint8, episode return float32, episode length int32), each [N], of the
        step `ticket`: views of its pinned slot, valid until three further steps have been enqueued.  The last two are
        Monitor's r / l where done (monitor.py:62-76)."""
        if not self._ring_head - self.SCALAR_SLOTS <= ticket < self._ring_head:
            raise _lib.SnkError("ticket %d is no longer (or not yet) in flight" % ticket)
        _lib.check(self._L.snk_scalars_wait(self._h, ticket % self.SCALAR_SLOTS))
        return self._ring[ticket % self.SCALAR_SLOTS][2]

    def close(self):
        if not getattr(self, "closed", True) and getattr(self, "_h", None):
            torch.cuda.synchronize(self.device)
            for g in list(self._graphs.values()):
                g.close()
            self._graphs = {}
            self._L.snk_destroy(self._h)
            self._h = None
            self._ring = None   # views of pinned memory the library has just freed
        self.closed = True

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    _WORLD_COLOURS = (((0, 204, 0), (191, 242, 191)), ((0, 51, 204), (128, 154, 230)),
                      ((204, 0, 119), (230, 128, 188)), ((119, 0, 204), (188, 128, 230)))

    def render(self, mode="rgb_array", env_index=0):
        """World view of one env as the reference's get_ob_world draws it (snake_multiple_test.py:60-91):
        one [V, V, 3] uint8 image, fruit red, snake i in the i-th colour pair, white border.  It is
        rebuilt on the host from the env's K views (snake k is the green one of view k), so it needs
        K >= S and the native observation mode -- or, in grid mode, straight from the cell codes, for any K;
        there is no pyglet window on a GPU box."""
        if mode != "rgb_array":
            raise NotImplementedError("only mode='rgb_array'")
        if self.obs_mode == "grid":
            g = self.obs[env_index].cpu().numpy()
            world = np.zeros((self.V, self.V, 3), dtype=np.uint8)
            world[g == _lib.CELL_FRUIT] = (255, 0, 0)
            for s in range(min(self.S, 4)):   # the reference has 4 colour pairs
                body_c, head_c = self._WORLD_COLOURS[s]
                world[g == _lib.cell_body(s)] = body_c
                world[g == _lib.cell_head(s)] = head_c
            world[g == _lib.CELL_WALL] = (255, 255, 255)
            return world
        if self.obs_mode != "native" or self.K < min(self.S, 4):
            return self.obs[env_index, :, :, 0:3].cpu().numpy()
        ob = self.obs[env_index].cpu().numpy().reshape(self.V, self.V, self.K, 3)
        world = np.zeros((self.V, self.V, 3), dtype=np.uint8)
        v0 = ob[:, :, 0]
        world[(v0 == (255, 0, 0)).all(-1)] = (255, 0, 0)
        for k in range(min(self.S, 4)):
            body_c, head_c = self._WORLD_COLOURS[k]
            world[(ob[:, :, k] == (0, 204, 0)).all(-1)] = body_c
            world[(ob[:, :, k] == (191, 242, 191)).all(-1)] = head_c
        world[(v0 == (255, 255, 255)).all(-1)] = (255, 255, 255)
        return world

    def get_images(self):
        """VecEnv.get_images (baselines/common/vec_env/__init__.py): the world view of every env, [N, V, V, 3]."""
        return np.stack([self.render("rgb_array", i) for i in range(self.N)])

    def render_tiled(self, max_envs=64):
        """VecEnv.render's big image: the first `max_envs` world views tiled into one P x Q mosaic."""
        n = min(self.N, max_envs)
        return tile_images(np.stack([self.render("rgb_array", i) for i in range(n)]))

    @property
    def unwrapped(self):
        return self

    # ------------------------------------------------------------------ extensions
    def set_obs_target(self, tensor):
        """Write observations straight into `tensor` (e.g. rollout[t], ppo_multi_agent_new.py:181)."""
        if tensor is None:
            _lib.check(self._L.snk_set_obs_target(self._h, None, 0))
        else:
            assert tensor.is_cuda and tensor.dtype == torch.uint8 and tensor.is_contiguous()
            _lib.check(self._L.snk_set_obs_target(self._h, C.c_void_p(tensor.data_ptr()), tensor.numel()))
        self._bind_buffers()

    def set_main_view_target(self, tensor):
        """Every following step / reset also writes the MAIN snake's view of all envs, packed [N,H,W,3], into `tensor`
        (slot t of the learner's [nsteps,N,H,W,3] rollout buffer, ppo_multi_agent_new.py:181); None switches it off.
        Not in grid mode: expand_views(obs, 1) gives view 0."""
        if self.obs_mode == "grid":
            raise ValueError("obs_mode 'grid' has no main-view target: use expand_views(env.obs, 1)")
        if tensor is None:
            _lib.check(self._L.snk_set_main_view_target(self._h, None, 0))
        else:
            assert tensor.is_cuda and tensor.dtype == torch.uint8 and tensor.is_contiguous()
            _lib.check(self._L.snk_set_main_view_target(self._h, C.c_void_p(tensor.data_ptr()), tensor.numel()))
        self._main_target = tensor   # keep it alive

    def make_graph(self, actions, T=None, obs_out=None, rewards_out=None, dones_out=None, sync_back=False):
        """T steps as one CUDA graph launch (snk_graph_create).  actions: int8 CUDA tensor [B, N, S]; step t plays
        batch t % B (T defaults to B).  obs_out [T,N,H,W,3K] ([T,N,V,V] in grid mode) / rewards_out [T,N] f32 / dones_out [T,N] u8 redirect the
        per-step outputs into rollout slots; without them every step writes the env's own buffers."""
        a = actions
        assert a.is_cuda and a.dtype == torch.int8 and a.is_contiguous() and tuple(a.shape[1:]) == (self.N, self.S)
        B = int(a.shape[0])
        T = B if T is None else int(T)
        ptr = lambda t: None if t is None else C.c_void_p(t.data_ptr())
        g = C.c_void_p()
        _lib.check(self._L.snk_graph_create(self._h, ptr(a), B, T, ptr(obs_out), ptr(rewards_out), ptr(dones_out),
                                            _lib.GRAPH_SYNC_BACK if sync_back else 0, C.byref(g)))
        return StepGraph(self, g, (a, obs_out, rewards_out, dones_out))

    def make_scripted_graph(self, T, step0=0, seed=1, eps=0.05):
        """T steps of [fruit-seeking policy kernel, step kernel] as one CUDA graph launch (snk_graph_create_scripted)."""
        g = C.c_void_p()
        _lib.check(self._L.snk_graph_create_scripted(self._h, int(T), int(step0), int(seed), int(round(eps * 1000)), C.byref(g)))
        return StepGraph(self, g, None)

    def rollout(self, actions, obs_out=None, rewards_out=None, dones_out=None):
        """T steps back to back into rollout buffers on the device (the mb_obs / mb_rewards /
        mb_dones of Runner.run, ppo_multi_agent_new.py:178-198) with no host round trip: ONE graph
        launch (cached per buffer set).  actions: int8 CUDA tensor [T, N, S].  Returns (obs
        [T,N,H,W,3K] u8, rewards [T,N] f32, dones [T,N] bool); afterwards `env.obs` / `env.rewards`
        are the last slot of those buffers (no copy back) until the next step() or reset()."""
        a = torch.as_tensor(actions, device=self.device).to(torch.int8).contiguous()
        T = int(a.shape[0])
        assert tuple(a.shape) == (T, self.N, self.S)
        shape = (T,) + tuple(self._own[0].shape)
        if obs_out is None:
            obs_out = torch.empty(shape, dtype=torch.uint8, device=self.device)
        if rewards_out is None:
            rewards_out = torch.empty((T, self.N), dtype=torch.float32, device=self.device)
        if dones_out is None:
            dones_out = torch.empty((T, self.N), dtype=torch.uint8, device=self.device)
        assert obs_out.is_contiguous() and tuple(obs_out.shape) == shape and obs_out.dtype == torch.uint8
        d8 = dones_out.view(torch.uint8) if dones_out.dtype == torch.bool else dones_out
        key = (a.data_ptr(), T, obs_out.data_ptr(), rewards_out.data_ptr(), d8.data_ptr())
        g = self._graphs.get(key)
        if g is None:
            for old in self._graphs.values():   # one cached rollout graph at a time
                old.close()
            self._graphs = {}
            g = self._graphs[key] = self.make_graph(a, T, obs_out, rewards_out, d8)
        g.launch()
        self.obs, self.rewards, self._done_u8 = obs_out[T - 1], rewards_out[T - 1], d8[T - 1]
        return obs_out, rewards_out, d8.view(torch.bool)

    def set_draw_tape(self, vals, bounds, offsets):
        """Replay mode: recorded reference draws, CSR per env (parity tests)."""
        vals = np.ascontiguousarray(vals, dtype=np.uint32)
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        assert len(offsets) == self.N + 1
        b = None if bounds is None else np.ascontiguousarray(bounds, dtype=np.uint32)
        _lib.check(self._L.snk_set_draw_tape(self._h, vals.ctypes.data_as(C.c_void_p),
                                             None if b is None else b.ctypes.data_as(C.c_void_p),
                                             offsets.ctypes.data_as(C.c_void_p)))
        self.cfg.rng_mode = _lib.RNG_TAPE

    def dump_state_blob(self):
        blob = np.zeros(self.lay.total_bytes, dtype=np.uint8)
        _lib.check(self._L.snk_dump_state(self._h, blob.ctypes.data_as(C.c_void_p), blob.nbytes))
        return blob

    def load_state_blob(self, blob):
        blob = np.ascontiguousarray(blob, dtype=np.uint8)
        _lib.check(self._L.snk_load_state(self._h, blob.ctypes.data_as(C.c_void_p), blob.nbytes))

    def dump_state(self):
        return split_state(self.dump_state_blob(), self.lay, self.cfg)

    def dump_state_range(self, first, count):
        """Canonical state of envs [first, first + count) only (snk_dump_state_range)."""
        sub = _lib.SnkConfig.from_buffer_copy(self.cfg)
        sub.num_envs, sub.env_id_base = int(count), self.cfg.env_id_base + int(first)
        lay = _lib.SnkStateLayout()
        _lib.check(self._L.snk_state_layout_of(C.byref(sub), C.byref(lay)))
        blob = np.zeros(lay.total_bytes, dtype=np.uint8)
        _lib.check(self._L.snk_dump_state_range(self._h, int(first), int(count), blob.ctypes.data_as(C.c_void_p), blob.nbytes))
        return split_state(blob, lay, sub)

    # ------------------------------------------------------------------ per-env state on the device
    def _sub_config(self, count):
        """This handle's geometry with `count` envs: the configuration of a `count`-env state blob."""
        sub = _lib.SnkConfig.from_buffer_copy(self.cfg)
        sub.num_envs, sub.env_id_base = int(count), 0
        lay = _lib.SnkStateLayout()
        _lib.check(self._L.snk_state_layout_of(C.byref(sub), C.byref(lay)))
        return sub, lay

    def _env_index(self, idx, distinct=False):
        """(int64 CUDA tensor, count) for an index argument.  A CUDA integer tensor is used as is (trusted: an index
        outside [0, N) only raises the device error flag, duplicates are not detected); host ints / numpy are checked."""
        if isinstance(idx, torch.Tensor) and idx.is_cuda:
            if idx.dtype.is_floating_point or idx.dtype == torch.bool:
                raise TypeError("env indices must be integers, got %s" % idx.dtype)
            t = idx.reshape(-1)
            if t.dtype != torch.int64:
                t = t.to(torch.int64)
            return t.contiguous(), int(t.numel()), None
        a = np.asarray(idx.cpu() if isinstance(idx, torch.Tensor) else idx)
        if a.dtype.kind not in "iu" and a.size:
            raise TypeError("env indices must be integers, got %s" % a.dtype)
        a = a.astype(np.int64).reshape(-1)
        if a.size == 0:
            raise ValueError("no env indices given")
        if a.min() < 0 or a.max() >= self.N:
            raise IndexError("env index out of range [0, %d)" % self.N)
        if distinct and len(np.unique(a)) != a.size:
            raise ValueError("destination env indices must be distinct")
        return torch.from_numpy(a).to(self.device), int(a.size), a

    def _check_geometry(self, cfg):
        mine = (self.cfg.size, self.cfg.n_snakes, self.cfg.n_fruits, self.cfg.rules)
        theirs = (cfg.size, cfg.n_snakes, cfg.n_fruits, cfg.rules)
        if mine != theirs:
            raise ValueError("env states of geometry (size, n_snakes, n_fruits, rules) = %r do not fit this env's %r" % (theirs, mine))

    def _observe(self):
        """Re-encode every env's observation from its state (snk_reset with an all-zero mask), as SnakeVecEnv.load does."""
        if getattr(self, "_no_reset_mask", None) is None:
            self._no_reset_mask = torch.zeros(self.N, dtype=torch.uint8, device=self.device)
        _lib.check(self._L.snk_reset(self._h, C.c_void_p(self._no_reset_mask.data_ptr()), self._stream()))

    def save_envs(self, idx=None, out=None):
        """Canonical state of envs `idx` (default: all) into a device blob, stream-ordered, no host round trip
        (snk_save_envs).  Returns an EnvStates; `out` (an EnvStates of len(idx) envs of this geometry) is reused instead
        of allocating, so the call can be recorded into a CUDA graph.  Indices may repeat."""
        i, n, _ = (None, self.N, None) if idx is None else self._env_index(idx)
        if out is None:
            out = EnvStates.empty(self, n)
        else:
            if not isinstance(out, EnvStates):
                raise TypeError("out must be an EnvStates")
            self._check_geometry(out.cfg)
            if out.count != n:
                raise ValueError("out holds %d envs, %d are saved" % (out.count, n))
        _lib.check(self._L.snk_save_envs(self._h, None if i is None else C.c_void_p(i.data_ptr()), n,
                                         C.c_void_p(out.blob.data_ptr()), out.blob.numel(), self._stream()))
        return out

    def restore_envs(self, states, idx=None, observe=True):
        """Env idx[j] (default: env j) <- entry j of `states` (snk_restore_envs): an EnvStates, or a uint8 torch / numpy
        blob of a len(idx)-env layout.  The states may come from another handle of the same geometry (size, n_snakes,
        n_fruits, rules); a rejected body raises the bad-state device flag (check_errors) and leaves that snake empty.
        Everything else a step returns (rewards, dones, infos, statistics) is untouched and the RNG key stays the
        destination env's.  observe=True re-encodes every env's observation from its state afterwards, as after a
        reset; observe=False leaves the observation buffers as they were (the next step writes the restored envs'
        images whole) and launches nothing but the restore."""
        if isinstance(states, EnvStates):
            self._check_geometry(states.cfg)
            blob, count = states.blob, states.count
        else:
            blob, count = states, None
        i, n, _ = (None, None, None) if idx is None else self._env_index(idx, distinct=True)
        count = count if count is not None else (n if n is not None else self.N)
        if n is not None and n != count:
            raise ValueError("%d indices for %d saved envs" % (n, count))
        if n is None and count > self.N:
            raise ValueError("%d saved envs do not fit %d envs" % (count, self.N))
        if not isinstance(states, EnvStates):
            if isinstance(blob, torch.Tensor):
                if blob.dtype != torch.uint8:
                    raise TypeError("a state blob must be uint8")
                blob = blob.reshape(-1).to(self.device).contiguous()
            else:
                blob = torch.from_numpy(np.ascontiguousarray(blob, dtype=np.uint8).reshape(-1)).to(self.device)
            if blob.data_ptr() % 16:
                blob = blob.clone()
        if observe:
            self._before_overwrite()
        _lib.check(self._L.snk_restore_envs(self._h, None if i is None else C.c_void_p(i.data_ptr()), count,
                                            C.c_void_p(blob.data_ptr()), blob.numel(), self._stream()))
        if observe:
            self._observe()

    def copy_envs(self, src, dst, observe=True):
        """Env dst[j] <- env src[j] on the device (snk_copy_envs): src may repeat (one env cloned into many slots),
        dst must be distinct and disjoint from src.  A clone keeps its own RNG key, so it equals its source until the
        next random draw.  `observe` as in restore_envs."""
        s, ns, hs = self._env_index(src)
        d, nd, hd = self._env_index(dst, distinct=True)
        if ns != nd:
            raise ValueError("%d sources for %d destinations" % (ns, nd))
        if hs is not None and hd is not None and np.intersect1d(hs, hd).size:
            raise ValueError("destination envs must not also be sources")
        if observe:
            self._before_overwrite()
        _lib.check(self._L.snk_copy_envs(self._h, C.c_void_p(s.data_ptr()), C.c_void_p(d.data_ptr()), ns, self._stream()))
        if observe:
            self._observe()

    def clone_envs_from(self, src_env, src, dst, observe=True):
        """Env dst[j] of this env <- env src[j] of `src_env` on the device (snk_clone_envs): copy_envs across handles.
        src_env is only read.  Both handles must be on one device with the same size, n_snakes, n_fruits and rules and
        the same private layout (a grid-mode and a native handle of one configuration can differ there: SnkError).
        src may repeat; dst must be distinct.  A clone keeps this env's RNG key, so it equals its source until the next
        random draw.  `observe` as in restore_envs."""
        if src_env is self:
            raise ValueError("src_env is this env: use copy_envs")
        s, ns, _ = src_env._env_index(src)
        d, nd, _ = self._env_index(dst, distinct=True)
        if ns != nd:
            raise ValueError("%d sources for %d destinations" % (ns, nd))
        if observe:
            self._before_overwrite()
        _lib.check(self._L.snk_clone_envs(src_env._h, C.c_void_p(s.data_ptr()), self._h, C.c_void_p(d.data_ptr()), ns,
                                          self._stream()))
        if observe:
            self._observe()

    def save(self, path):
        """Checkpoint of the env state (the reference never checkpoints it; its learner only saves
        model parameters, ppo_multi_agent_new.py:104-106).  A .npz with the constructor arguments
        and the canonical state blob; `SnakeVecEnv.load(path)` resumes bit-exactly."""
        c = self.cfg
        np.savez_compressed(path, blob=self.dump_state_blob(), num_envs=c.num_envs, size=c.size, n_snakes=c.n_snakes,
                            n_fruits=c.n_fruits, n_views=c.n_views, rules=self.rules, max_steps=c.max_steps,
                            auto_reset=c.auto_reset, env_id_base=c.env_id_base, seed=np.uint64(c.seed), obs_mode=self.obs_mode)

    @classmethod
    def load(cls, path, device=0, host_io=False):
        z = np.load(path if str(path).endswith(".npz") else str(path) + ".npz")
        env = cls(int(z["num_envs"]), int(z["size"]), int(z["n_snakes"]), int(z["n_fruits"]), int(z["n_views"]), str(z["rules"]),
                  int(z["seed"]), device, int(z["env_id_base"]), bool(z["auto_reset"]), int(z["max_steps"]), host_io=host_io,
                  obs_mode=str(z["obs_mode"]))
        env.load_state_blob(z["blob"])
        env.reset(mask=torch.zeros(env.N, dtype=torch.bool, device=env.device))  # re-encode the observations
        return env

    def gen_actions(self, step, seed=1, out=None):
        """Synthetic uniform action stream (Philox key (seed, global env id)), generated on device."""
        out = self._actions if out is None else out
        _lib.check(self._L.snk_gen_actions(self._h, C.c_void_p(out.data_ptr()), int(step), int(seed),
                                           self.action_space.n, self._stream()))
        return out

    def gen_scripted_actions(self, step, seed=1, eps=0.05, out=None):
        """Benchmark policy computed on the device from the current state: turn toward the nearest
        fruit unless the next cell is a wall or a body, with probability `eps` a random action."""
        out = self._actions if out is None else out
        _lib.check(self._L.snk_gen_scripted_actions(self._h, C.c_void_p(out.data_ptr()), int(step), int(seed),
                                                    int(round(eps * 1000)), self._stream()))
        return out

    def stats(self, reduce=True):
        """Running episode statistics (Monitor's aggregate role).  With torch.distributed
        initialised and reduce=True the 8 doubles are summed over all ranks on demand (a
        torch.distributed all-reduce); the in-loop form is init_comm() + stats_global()."""
        from .sharding import all_reduce_stats
        s = self._stats.clone()
        if reduce:
            all_reduce_stats(s)
        return dict(zip(_lib.STAT_NAMES, s.cpu().tolist()))

    def init_comm(self, group=None, mode="p2p"):
        """Sets up the path's one exchange: from now on every step sums the 8-double statistics vector over all ranks,
        read about one step late through stats_global().
        mode 'p2p' (default): fused into the step kernel -- its first CTA stores the rank's running sums (as of the
        previous step) into every peer's inbox over NVLink (cudaIpc-mapped peer memory, posted 8-byte stores); no
        collective kernel, no fence, no rendezvous (snk_peer_export / snk_peer_connect).  mode 'nccl': a raw ncclAllReduce per step issued by the C layer on a side
        stream (snk_comm_init).  The handles / the NCCL id travel over the existing torch.distributed group; without
        one (single process) both forms degenerate to one rank."""
        import torch.distributed as dist
        world = dist.get_world_size(group) if dist.is_available() and dist.is_initialized() else 1
        rank = dist.get_rank(group) if world > 1 else 0
        on_gpu = world > 1 and dist.get_backend(group) == "nccl"
        if mode == "p2p":
            mine = np.zeros(64, dtype=np.uint8)
            _lib.check(self._L.snk_peer_export(self._h, mine.ctypes.data_as(C.c_void_p)))
            handles = mine[None]
            if world > 1:
                t = torch.from_numpy(mine).to(self.device if on_gpu else "cpu")
                out = [torch.empty_like(t) for _ in range(world)]
                dist.all_gather(out, t, group=group)
                handles = np.ascontiguousarray(torch.stack(out).cpu().numpy())
            torch.cuda.synchronize(self.device)
            _lib.check(self._L.snk_peer_connect(self._h, handles.ctypes.data_as(C.c_void_p), world, rank))
            if world > 1:
                dist.barrier(group=group)   # every rank has mapped every inbox before anybody pushes
            self.comm_mode = "p2p"
            return world
        if mode != "nccl":
            raise ValueError("mode must be 'p2p' or 'nccl'")
        ident = np.zeros(128, dtype=np.uint8)
        if rank == 0:
            _lib.check(self._L.snk_comm_unique_id(ident.ctypes.data_as(C.c_void_p)))
        if world > 1:
            t = torch.from_numpy(ident).to(self.device if on_gpu else "cpu")
            dist.broadcast(t, src=dist.get_global_rank(group, 0) if group is not None else 0, group=group)
            ident = np.ascontiguousarray(t.cpu().numpy())
        torch.cuda.synchronize(self.device)
        _lib.check(self._L.snk_comm_init(self._h, ident.ctypes.data_as(C.c_void_p), world, rank))
        self.comm_mode = "nccl"
        return world

    def comm_enable(self, on=True):
        """A/B switch of the per-step reduction (graphs made afterwards follow it)."""
        _lib.check(self._L.snk_comm_enable(self._h, 1 if on else 0))

    def stats_global(self):
        """Statistics summed over all ranks (after init_comm).  NCCL form: as of the last completed per-step all-reduce.
        Peer form: this rank's sums plus what the peers last pushed -- about one step old while the ranks are stepping;
        called by all ranks after their last step it is exact (it pushes the final sums, waits at a barrier of the
        torch.distributed group, then adds up)."""
        out = np.zeros(_lib.NSTATS, dtype=np.float64)
        _lib.check(self._L.snk_get_stats_global(self._h, out.ctypes.data_as(C.c_void_p), self._stream()))
        if getattr(self, "comm_mode", None) == "p2p":
            import torch.distributed as dist
            if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
                dist.barrier()   # every rank's final push has been issued and completed (the call above synchronised)
                _lib.check(self._L.snk_get_stats_global(self._h, out.ctypes.data_as(C.c_void_p), self._stream()))
        return dict(zip(_lib.STAT_NAMES, out.tolist()))

    def comm_latency_us(self, iters=200):
        """Mean duration of one all-reduce of the statistics vector (CUDA events on the side stream; collective call)."""
        out = C.c_double(0)
        _lib.check(self._L.snk_comm_bench(self._h, int(iters), C.byref(out)))
        return out.value

    def comm_info(self):
        out = (C.c_int32 * 4)()
        _lib.check(self._L.snk_comm_info(self._h, out))
        return dict(zip(("ranks", "rank", "allreduces", "nccl_version"), list(out)))

    def reset_stats(self):
        _lib.check(self._L.snk_reset_stats(self._h, self._stream()))

    def check_errors(self):
        flags = C.c_uint32(0)
        _lib.check(self._L.snk_check_errors(self._h, C.byref(flags), self._stream()))
        if flags.value:
            raise _lib.SnkError("device error flags: " + ", ".join(v for k, v in _lib.DEVERR.items() if flags.value & k))

    def launch_count(self):
        n = C.c_uint64(0)
        _lib.check(self._L.snk_launch_count(self._h, C.byref(n)))
        return n.value

    def launch_info(self):
        out = (C.c_int32 * 6)()
        _lib.check(self._L.snk_launch_info(self._h, out))
        d = dict(zip(("kind", "grid", "block", "smem", "occupancy", "envs_per_cta"), list(out)))
        d["kernel"] = ("k_step_lane", "k_step_tile", "k_step_dense", "k_step_rows")[d["kind"]]
        f = (C.c_int32 * 4)()
        _lib.check(self._L.snk_launch_form(self._h, f))
        if self.obs_mode == "grid" and d["kind"] == 3:
            d["kernel"] = "k_step_rows (grid)"
        if d["kind"] == 0:  # the lane path has three forms; the handle may move between the fused and the two-kernel one by itself
            d["kernel"] = {0: "k_step_lane", 1: "k_step_lane_ws", 3: "k_lane_logic + k_lane_paint2"}[f[0]]
            if self.obs_mode == "grid":
                d["kernel"] = "k_lane_logic + k_lane_grid"
            d["envs_per_warp_batch"], d["envs_per_image"], d["adaptive"] = int(f[1]), int(f[2]), bool(f[3])
        return d

    def algorithmic_bytes_per_step(self, mean_sum_len):
        out = C.c_double(0)
        _lib.check(self._L.snk_algorithmic_bytes_per_step(C.byref(self.cfg), float(mean_sum_len), C.byref(out)))
        return out.value


def expand_views(grid, n_views, first_view=0, out=None):
    """Cell-code grids (obs_mode 'grid') -> RGB views on the device (snk_expand_views).  `grid`: a CUDA uint8 tensor whose
    last two dims are (V, V) -- an env's `obs`, a [T, N, V, V] rollout, a gathered minibatch.  Returns
    [..., V, V, 3 * n_views]: views first_view .. first_view + n_views - 1 of every cell, byte-identical to those channels
    of the native observation, so expand_views(env.obs, env.K) equals a native env's `obs` of the same state.  `out`
    (uint8, that shape, contiguous, on the grid's device) is written instead of allocating.  Stream-ordered on the
    current stream; no synchronisation."""
    if not isinstance(grid, torch.Tensor) or not grid.is_cuda or grid.dtype != torch.uint8:
        raise TypeError("grid must be a CUDA uint8 tensor")
    if grid.dim() < 2 or grid.shape[-1] != grid.shape[-2]:
        raise ValueError("the last two dims of a grid are (V, V), got %r" % (tuple(grid.shape),))
    V, n_views, first_view = int(grid.shape[-1]), int(n_views), int(first_view)
    shape = tuple(grid.shape) + (3 * n_views,)
    if out is None:
        out = torch.empty(shape, dtype=torch.uint8, device=grid.device)
    elif (not isinstance(out, torch.Tensor) or tuple(out.shape) != shape or out.dtype != torch.uint8 or not out.is_contiguous()
          or out.device != grid.device):
        raise ValueError("out must be a contiguous uint8 tensor of shape %r on %s" % (shape, grid.device))
    n = grid.numel() // (V * V)
    if n == 0:
        return out
    g = grid.contiguous()
    dev = grid.device.index or 0
    stream = C.c_void_p(torch.cuda.current_stream(grid.device).cuda_stream)
    _lib.check(_lib.lib().snk_expand_views(C.c_void_p(g.data_ptr()), n, V - 2, first_view, n_views, C.c_void_p(out.data_ptr()), dev, stream))
    return out


class EnvStates(object):
    """Canonical states of `count` envs in a device uint8 blob (SnakeVecEnv.save_envs): the blob of a `count`-env
    configuration of the env's geometry, byte for byte what dump_state_range writes for the same envs.  `cfg` is that
    configuration and `lay` its SnkStateLayout.  States move between handles of the same size, n_snakes, n_fruits and
    rules (another num_envs, seed or env_id_base is fine)."""

    def __init__(self, blob, cfg, lay):
        assert isinstance(blob, torch.Tensor) and blob.is_cuda and blob.dtype == torch.uint8 and blob.numel() >= lay.total_bytes
        self.blob, self.cfg, self.lay = blob, cfg, lay
        self.count = int(cfg.num_envs)

    @classmethod
    def empty(cls, env, count):
        """An uninitialised buffer for `count` envs of `env`'s geometry (for save_envs(out=...))."""
        cfg, lay = env._sub_config(count)
        return cls(torch.empty(int(lay.total_bytes), dtype=torch.uint8, device=env.device), cfg, lay)

    def __len__(self):
        return self.count

    def arrays(self):
        """Named torch views of the blob, with the names and shapes of split_state."""
        N, S, F, V, lay = self.count, self.cfg.n_snakes, self.cfg.n_fruits, self.cfg.size + 2, self.lay

        def arr(off, dtype, shape):
            n = int(np.prod(shape)) * torch.empty(0, dtype=dtype).element_size()
            return self.blob[off:off + n].view(dtype).reshape(shape)

        out = {"t": arr(lay.off_t, torch.int32, (N,)), "spare": arr(lay.off_spare, torch.uint32, (N,)),
               "draw_ctr": arr(lay.off_draw_ctr, torch.uint32, (N,)), "ep_ret": arr(lay.off_ep_ret, torch.float32, (N,)),
               "ep_len": arr(lay.off_ep_len, torch.int32, (N,)), "len": arr(lay.off_len, torch.uint16, (N, S)),
               "grow_to": arr(lay.off_grow_to, torch.uint16, (N, S)), "vel": arr(lay.off_vel, torch.uint8, (N, S)),
               "body": arr(lay.off_body, torch.uint16, (N, S, lay.cap))}
        if lay.fruit_is_grid:
            out["fruit_grid"] = arr(lay.off_fruit, torch.uint8, (N, V * V))
        else:
            out["fruit"] = arr(lay.off_fruit, torch.uint16, (N, F))
        return out

    def numpy(self):
        """The blob on the host (synchronises), usable with split_state(blob, states.lay, states.cfg)."""
        return self.blob[:self.lay.total_bytes].cpu().numpy()


def split_state(blob, lay, cfg):
    """Named numpy views of a canonical state blob (snk_state_layout, include/snk.h)."""
    N, S, F, V = cfg.num_envs, cfg.n_snakes, cfg.n_fruits, cfg.size + 2
    b = np.frombuffer(blob, dtype=np.uint8)

    def arr(off, dtype, shape):
        n = int(np.prod(shape)) * np.dtype(dtype).itemsize
        return b[off:off + n].view(dtype).reshape(shape)

    out = {"t": arr(lay.off_t, np.int32, (N,)), "spare": arr(lay.off_spare, np.uint32, (N,)),
           "draw_ctr": arr(lay.off_draw_ctr, np.uint32, (N,)), "ep_ret": arr(lay.off_ep_ret, np.float32, (N,)),
           "ep_len": arr(lay.off_ep_len, np.int32, (N,)), "len": arr(lay.off_len, np.uint16, (N, S)),
           "grow_to": arr(lay.off_grow_to, np.uint16, (N, S)), "vel": arr(lay.off_vel, np.uint8, (N, S)),
           "body": arr(lay.off_body, np.uint16, (N, S, lay.cap))}
    if lay.fruit_is_grid:
        out["fruit_grid"] = arr(lay.off_fruit, np.uint8, (N, V * V))
    else:
        out["fruit"] = arr(lay.off_fruit, np.uint16, (N, F))
    return out
