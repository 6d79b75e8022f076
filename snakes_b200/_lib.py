"""ctypes binding of libsnk.so -- the C ABI declared in include/snk.h.

The library is the product: if it is missing the import fails loudly (there is no CPU
fallback).  Build it with `python __graft_entry__.py build` (nvcc, sm_100a).
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SNK_LIB") or os.path.join(_HERE, "libsnk.so")  # SNK_LIB: A/B builds during kernel work

RULES = {"classic": 0, "adversarial": 1, "cut": 2}
OBS_NATIVE, OBS_ATARI84, OBS_GRID = 0, 1, 2
OBS_MODES = {"native": OBS_NATIVE, "atari84": OBS_ATARI84, "grid": OBS_GRID}
# cell codes of obs_mode 'grid' (SNK_CELL_* of include/snk.h); snake s: body 3 + 2s, head 4 + 2s
CELL_EMPTY, CELL_FRUIT, CELL_WALL = 0, 1, 255


def cell_body(s):
    return 3 + 2 * s


def cell_head(s):
    return 4 + 2 * s

# snk_grid_conv_in (SNK_GRID_CONV_* of include/snk.h): classes of a cell in view k, their RGB colours, the workspace
GRID_CONV_CHANNELS = 32
GRID_CONV_COLOURS = ((0, 0, 0), (255, 0, 0), (255, 255, 255), (0, 204, 0), (191, 242, 191), (0, 51, 204), (128, 154, 230))
GRID_CONV_WGRAD_CELLS_PER_CTA, GRID_CONV_WGRAD_MAX_CTAS = 2048, 592
GRID_CONV_PART_FLOATS = (9 * (len(GRID_CONV_COLOURS) - 1) + 1) * GRID_CONV_CHANNELS


def grid_conv_work_bytes(n_cells):
    """SNK_GRID_CONV_WORK_BYTES: the workspace snk_grid_conv_in_wgrad needs for n_cells = n * V * V."""
    ctas = min(-(-int(n_cells) // GRID_CONV_WGRAD_CELLS_PER_CTA), GRID_CONV_WGRAD_MAX_CTAS)
    return ctas * GRID_CONV_PART_FLOATS * 4


def grid_conv84_geometry(V, n=0):
    """snk_grid_conv84_geometry for V x V grids: (f, P, C, workspace bytes of snk_grid_conv84_in_wgrad for n grids).
    Raises SnkError for a V that does not divide 84 or lies outside 3..42."""
    out = (C.c_int64 * 4)()
    check(lib().snk_grid_conv84_geometry(int(V) - 2, int(n), out))
    return tuple(int(x) for x in out)


RNG_PHILOX, RNG_TAPE = 0, 1
NSTATS = 8
STAT_NAMES = ("env_steps", "episodes", "return_sum", "length_sum", "fruits", "deaths", "body_cells", "draws")
DEVERR = {1: "draw tape underrun", 2: "draw tape bound mismatch", 4: "fruit count overflow", 8: "body ring overflow",
          16: "bad state (non-adjacent segments, cell id or length out of range) or env index out of range"}
GRAPH_SYNC_BACK = 1
# snk_tally counters (SNK_TALLY_* of include/snk.h): [n_groups][S][fields] int64, in this order
TALLY_FIELDS = ("wins", "draws", "losses", "fruits", "deaths", "steps_alive", "return_sq", "length")


class SnkConfig(C.Structure):
    _fields_ = [("size", C.c_int32), ("n_snakes", C.c_int32), ("n_fruits", C.c_int32), ("n_views", C.c_int32),
                ("rules", C.c_int32), ("max_steps", C.c_int32), ("auto_reset", C.c_int32), ("obs_mode", C.c_int32),
                ("device", C.c_int32), ("rng_mode", C.c_int32), ("num_envs", C.c_int64), ("env_id_base", C.c_int64),
                ("seed", C.c_uint64)]


class SnkBuffers(C.Structure):
    _fields_ = [("d_obs", C.c_void_p), ("d_reward", C.c_void_p), ("d_reward_all", C.c_void_p), ("d_done", C.c_void_p),
                ("d_num_alive", C.c_void_p), ("d_episode_return", C.c_void_p), ("d_episode_len", C.c_void_p),
                ("d_stats", C.c_void_p), ("obs_bytes", C.c_size_t), ("obs_h", C.c_int32), ("obs_w", C.c_int32),
                ("obs_c", C.c_int32), ("d_info_block", C.c_void_p), ("info_block_bytes", C.c_size_t)]


class SnkStateLayout(C.Structure):
    _fields_ = [(n, C.c_size_t) for n in ("total_bytes", "off_t", "off_spare", "off_draw_ctr", "off_ep_ret",
                                          "off_ep_len", "off_len", "off_grow_to", "off_vel", "off_body", "off_fruit")]
    _fields_ += [("cap", C.c_int32), ("fruit_is_grid", C.c_int32)]


# every symbol include/snk.h declares, with its argument types
_SIGNATURES = {
    "snk_version": (C.c_int, []),
    "snk_last_error": (C.c_char_p, []),
    "snk_create": (C.c_int, [C.POINTER(SnkConfig), C.POINTER(C.c_void_p)]),
    "snk_create_ex": (C.c_int, [C.POINTER(SnkConfig), C.c_char_p, C.POINTER(C.c_void_p)]),
    "snk_destroy": (C.c_int, [C.c_void_p]),
    "snk_get_config": (C.c_int, [C.c_void_p, C.POINTER(SnkConfig)]),
    "snk_get_buffers": (C.c_int, [C.c_void_p, C.POINTER(SnkBuffers)]),
    "snk_reset": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "snk_step": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "snk_step_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "snk_step_host_views": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "snk_step_host_async": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "snk_scalars_layout": (C.c_int, [C.c_void_p, C.POINTER(C.c_size_t)]),
    "snk_step_scalars_async": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "snk_scalars_wait": (C.c_int, [C.c_void_p, C.c_int32]),
    "snk_host_alloc": (C.c_int, [C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p), C.POINTER(C.c_int32)]),
    "snk_host_free": (C.c_int, [C.c_void_p, C.c_void_p]),
    "snk_graph_create": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32,
                                   C.POINTER(C.c_void_p)]),
    "snk_graph_create_scripted": (C.c_int, [C.c_void_p, C.c_int32, C.c_uint64, C.c_uint64, C.c_int32, C.POINTER(C.c_void_p)]),
    "snk_graph_launch": (C.c_int, [C.c_void_p, C.c_void_p]),
    "snk_graph_destroy": (C.c_int, [C.c_void_p]),
    "snk_rollout": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "snk_set_obs_target": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t]),
    "snk_set_main_view_target": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t]),
    "snk_set_draw_tape": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "snk_state_layout_of": (C.c_int, [C.POINTER(SnkConfig), C.POINTER(SnkStateLayout)]),
    "snk_dump_state": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t]),
    "snk_dump_state_range": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_size_t]),
    "snk_load_state": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t]),
    "snk_save_envs": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_size_t, C.c_void_p]),
    "snk_restore_envs": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_size_t, C.c_void_p]),
    "snk_copy_envs": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "snk_clone_envs": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "snk_get_stats": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "snk_reset_stats": (C.c_int, [C.c_void_p, C.c_void_p]),
    "snk_check_errors": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint32), C.c_void_p]),
    "snk_peer_export": (C.c_int, [C.c_void_p, C.c_void_p]),
    "snk_peer_connect": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32]),
    "snk_comm_enable": (C.c_int, [C.c_void_p, C.c_int32]),
    "snk_comm_unique_id": (C.c_int, [C.c_void_p]),
    "snk_comm_init": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32]),
    "snk_get_stats_global": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "snk_comm_bench": (C.c_int, [C.c_void_p, C.c_int32, C.POINTER(C.c_double)]),
    "snk_comm_info": (C.c_int, [C.c_void_p, C.POINTER(C.c_int32)]),
    "snk_gen_actions": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_int32, C.c_void_p]),
    "snk_gen_scripted_actions": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_int32, C.c_void_p]),
    "snk_gae": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_double, C.c_int32, C.c_int64,
                          C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "snk_expand_views": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p]),
    "snk_grid_conv_in": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p,
                                   C.c_int32, C.c_void_p]),
    "snk_grid_conv_in_wgrad": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32,
                                         C.c_void_p, C.c_void_p, C.c_size_t, C.c_int32, C.c_void_p]),
    "snk_grid_conv84_geometry": (C.c_int, [C.c_int32, C.c_int64, C.POINTER(C.c_int64)]),
    "snk_grid_conv84_in": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p,
                                     C.c_int32, C.c_void_p]),
    "snk_grid_conv84_in_wgrad": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32,
                                           C.c_void_p, C.c_void_p, C.c_size_t, C.c_int32, C.c_void_p]),
    "snk_tally_layout": (C.c_int, [C.c_void_p, C.POINTER(C.c_size_t)]),
    "snk_tally": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "snk_search_begin": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int64, C.c_void_p, C.c_void_p,
                                   C.c_void_p]),
    "snk_search_accumulate": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "snk_search_pick": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                                  C.c_void_p]),
    "snk_algorithmic_bytes_per_step":(C.c_int, [C.POINTER(SnkConfig), C.c_double, C.POINTER(C.c_double)]),
    "snk_launch_count": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint64)]),
    "snk_launch_info": (C.c_int, [C.c_void_p, C.POINTER(C.c_int32)]),
    "snk_launch_form": (C.c_int, [C.c_void_p, C.POINTER(C.c_int32)]),
}

_lib = None


class SnkError(RuntimeError):
    pass


def lib():
    """Loads libsnk.so (once).  Raises if it has not been built: there is no fallback path."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise SnkError("%s not found: build the CUDA library first (python __graft_entry__.py build)" % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype, fn.argtypes = res, args
        _lib = L
    return _lib


def check(rc):
    if rc != 0:
        raise SnkError("libsnk error %d: %s" % (rc, lib().snk_last_error().decode()))


def make_config(num_envs, size=10, n_snakes=2, n_fruits=None, n_views=None, rules="classic", max_steps=2000,
                auto_reset=True, obs_mode=OBS_NATIVE, device=0, rng_mode=RNG_PHILOX, env_id_base=0, seed=0):
    if isinstance(rules, str):
        if rules not in RULES:
            raise ValueError("rules must be one of %s" % sorted(RULES))
        rules = RULES[rules]
    if hasattr(size, "__len__"):
        if len(size) != 2 or size[0] != size[1]:
            raise ValueError("only square boards are supported, got size=%r" % (size,))
        size = size[0]
    return SnkConfig(int(size), int(n_snakes), int(n_snakes if n_fruits is None else n_fruits),
                     int(n_snakes if n_views is None else n_views), int(rules), int(max_steps), int(bool(auto_reset)),
                     int(obs_mode), int(device), int(rng_mode), int(num_envs), int(env_id_base), int(seed))
