/* snk.h -- C ABI of the B200-native batched multi-snake environment (libsnk.so).
 *
 * The reference (jdubkim/Self-play-on-Multi-Snakes-Environment) has no native boundary: its hot
 * path is a per-instance Python `gym.Env` stepped by one OS process per env.  This header is the
 * boundary a native replacement of that path exports; every entry point names the reference
 * interface it replaces (paths relative to the reference's `src/`).  Plain pointers and sizes
 * only -- no torch / Python types -- so it binds from ctypes, cffi, pybind11 or any FFI.
 *
 * Conventions
 *   - every function returns 0 on success or a negative SNK_E* code; no exception crosses;
 *     `snk_last_error()` gives the text of the calling thread's last failure.
 *   - `d_` pointers are device memory of the handle's CUDA device, `h_` pointers are host memory.
 *   - `stream` is a `cudaStream_t` passed as `void*` (NULL = legacy default stream).  All device
 *     work is stream-ordered on it; no entry point synchronises unless its comment says so.
 *   - one handle per GPU (per shard of the global env range); a handle is not thread-safe.
 *
 * Geometry.  D = board edge, V = D + 2 (one-cell border).  A cell (x, y) -- x is the FIRST
 * observation index, `ob[x+1][y+1]` in gym_snake/envs/snake_multiple_test.py:31 -- is stored as
 * the padded id  pid = (x + 1) * V + (y + 1)  (uint16), which can also hold a head that is one
 * step outside the board.
 */
#ifndef SNK_H_
#define SNK_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SNK_VERSION 350 /* 0.3.5 */

/* error codes */
#define SNK_OK 0
#define SNK_EINVAL (-1)   /* bad argument / unsupported configuration */
#define SNK_ECUDA (-2)    /* CUDA runtime failure (text in snk_last_error) */
#define SNK_ENOMEM (-3)
#define SNK_ESTATE (-4)   /* device-side error flag raised (see SNK_DEVERR_*) */
#define SNK_ECOMM (-5)    /* NCCL missing or an NCCL call failed (text in snk_last_error) */

/* device error flags (sticky; read + cleared by snk_check_errors) */
#define SNK_DEVERR_TAPE_UNDERRUN 1u   /* replay tape exhausted for some env */
#define SNK_DEVERR_TAPE_BOUND 2u      /* replayed draw was recorded with another bound */
#define SNK_DEVERR_FRUIT_OVERFLOW 4u  /* >255 fruits on one cell (adversarial / cut grid) */
#define SNK_DEVERR_BODY_OVERFLOW 8u   /* ring capacity exceeded (cannot happen for cap = D*D+1) */
#define SNK_DEVERR_BAD_STATE 16u      /* a rejected state (snk_load_state, snk_restore_envs: see there) or an env index outside
                                       * [0, N) given to snk_save_envs / snk_restore_envs / snk_copy_envs (entry skipped) */

/* rule-sets */
#define SNK_RULES_CLASSIC 0      /* gym_snake/envs/snake_multiple_test.py  (SnakeEnv) */
#define SNK_RULES_ADVERSARIAL 1  /* gym_snake/envs/snake_adversarial_env.py (dead body -> fruit, spare_fruits) */
#define SNK_RULES_CUT 2          /* README.md:11 "body-cut"; no reference code -- spec in DESIGN.md, parity unpinned */

/* observation modes */
#define SNK_OBS_NATIVE 0   /* uint8 [N][V][V][3K], the reference's get_multi_snake_ob() stacked by np.stack */
#define SNK_OBS_ATARI84 1  /* uint8 [N][84][84][3K]: utils.py:27-31 WarpFrame; exact when 84 % V == 0 */
#define SNK_OBS_GRID 2     /* uint8 [N][V][V]: one cell code (SNK_CELL_*) per padded cell, row-major like the native image;
                            * snk_buffers reports obs_h = obs_w = V, obs_c = 1, obs_bytes = N*V*V.  Lossless for all K views:
                            * snk_expand_views turns it into the native image or any run of its views. */

/* Cell codes of SNK_OBS_GRID.  They grow in the reference's paint order (get_ob_for_snake :35-58: fruits, then the
 * snakes by index, body then head, then the border), so "a later item overwrites an earlier one" holds code by code,
 * and S <= 32 keeps every code in a byte.  Code 2 is unused.  A fruit outside the board (adversarial rules: a dead body's
 * cells become fruit, and a head may die one step outside) lies under the border, as in the reference.
 * View k (0 <= k < K) of a cell, as the native observation draws it:
 *   SNK_CELL_EMPTY  black (0, 0, 0)            SNK_CELL_FRUIT  red (255, 0, 0)       SNK_CELL_WALL  white (255, 255, 255)
 *   code >= 3       snake s = (code - 3) >> 1, head if (code - 3) & 1, else body; the self colours (green: body (0, 204, 0),
 *                   head (191, 242, 191)) when s == k, the other colours (blue: body (0, 51, 204), head (128, 154, 230))
 *                   otherwise.  Views k >= S have no self snake. */
#define SNK_CELL_EMPTY 0
#define SNK_CELL_FRUIT 1
#define SNK_CELL_BODY(s) (3 + 2 * (s))
#define SNK_CELL_HEAD(s) (4 + 2 * (s))
#define SNK_CELL_WALL 255

/* RNG modes */
#define SNK_RNG_PHILOX 0   /* Philox4x32-10, key (seed, global env id), counter = per-env draw index */
#define SNK_RNG_TAPE 1     /* replay recorded reference draws (snk_set_draw_tape) */

/* Constructor arguments.  Replaces the env kwargs of
 * gym_snake/envs/snake_multiple_env_new.py:10 (`size, n_snakes, n_fruits`), `Config.NUM_SNAKES`
 * (config.py:16, read at snake_multiple_test.py:223), `env.seed(seed + rank)` (utils.py:39) and the
 * `[make_env(i) for i in range(num_env)]` fan-out of utils.py:49. */
typedef struct snk_config {
  int32_t size;        /* D, 2..254 */
  int32_t n_snakes;    /* S, 1..32 */
  int32_t n_fruits;    /* F, 0..32; the reference uses F = S (snake_multiple_test.py:223-225) */
  int32_t n_views;     /* K, 1..32; 0 = S.  SnakeEnv emits K = 3 (snake_multiple_test.py:93-95) */
  int32_t rules;       /* SNK_RULES_* */
  int32_t max_steps;   /* episode cap, reference 2000 (snake_multiple_test.py:195); 0 = 2000 */
  int32_t auto_reset;  /* 1 = SubprocVecEnv worker contract (baselines/common/vec_env/subproc_vec_env.py:13-16) */
  int32_t obs_mode;    /* SNK_OBS_*; SNK_OBS_GRID takes none of the debug switches lane, delta, epw, adaptive, alt_hi,
                        * force_kernel=tile|dense (snk_create_ex fails with SNK_EINVAL and names the switch) */
  int32_t device;      /* CUDA device ordinal */
  int32_t rng_mode;    /* SNK_RNG_* */
  int64_t num_envs;    /* N, envs held by THIS handle */
  int64_t env_id_base; /* global id of this handle's env 0 (shard offset; keys the RNG); >= 0, base + N <= 2^32 */
  uint64_t seed;
} snk_config;

/* Device buffers owned by the handle (valid until snk_destroy).  Replaces the tuple returned by
 * SubprocVecEnv.step_wait (subproc_vec_env.py:57-61) and Monitor's info['episode']
 * (baselines/bench/monitor.py:62-76). */
typedef struct snk_buffers {
  uint8_t* d_obs;          /* [N][H][W][3K] uint8 (H = W = V native, 84 atari); may be redirected.  READ-ONLY for
                            * callers: the step writes only the bytes that changed into the handle's own buffer (the
                            * sectors a step can change, when the handle knows the buffer still shows the previous
                            * frame), so anything written into it between steps may survive them.  Copy it instead. */
  float* d_reward;         /* [N]    reward of snake 0 (the reference's scalar reward) */
  float* d_reward_all;     /* [N][S] extension: per-snake reward */
  uint8_t* d_done;         /* [N]    1 = episode ended this step (obs is then the reset obs if auto_reset) */
  uint8_t* d_num_alive;    /* [N]    info['num_snakes'] */
  float* d_episode_return; /* [N]    valid where d_done: Monitor 'r' */
  int32_t* d_episode_len;  /* [N]    valid where d_done: Monitor 'l' */
  double* d_stats;         /* [SNK_NSTATS] running sums since snk_reset_stats */
  size_t obs_bytes;        /* N*H*W*3K (SNK_OBS_GRID: N*V*V) */
  int32_t obs_h, obs_w, obs_c;  /* bytes per pixel: 3K, or 1 for SNK_OBS_GRID */
  uint8_t* d_info_block;   /* d_done, d_num_alive, d_episode_return, d_episode_len live in this one block (in this */
  size_t info_block_bytes; /* order, each 16-byte aligned): one copy snapshots a step's infos */
} snk_buffers;

/* indices into d_stats / snk_get_stats */
#define SNK_STAT_ENV_STEPS 0
#define SNK_STAT_EPISODES 1
#define SNK_STAT_RETURN_SUM 2
#define SNK_STAT_LENGTH_SUM 3
#define SNK_STAT_FRUITS 4     /* fruits eaten by any snake */
#define SNK_STAT_DEATHS 5     /* snakes that died */
#define SNK_STAT_BODY_CELLS 6 /* sum over env-steps of total live body length after the step (mean SigmaL = this / ENV_STEPS) */
#define SNK_STAT_DRAWS 7      /* RNG draws consumed */
#define SNK_NSTATS 8

/* Offsets (bytes) of the canonical state arrays inside a snk_dump_state blob.  Bodies are stored
 * head-first and zero-padded, so two blobs are byte-comparable. */
typedef struct snk_state_layout {
  size_t total_bytes;
  size_t off_t;          /* int32  [N]       step counter t */
  size_t off_spare;      /* uint32 [N]       adversarial spare_fruits (snake_adversarial_env.py:14) */
  size_t off_draw_ctr;   /* uint32 [N]       draws consumed so far */
  size_t off_ep_ret;     /* float  [N]       running episode return (Monitor) */
  size_t off_ep_len;     /* int32  [N]       running episode length (Monitor) */
  size_t off_len;        /* uint16 [N][S]    body length, 0 = dead */
  size_t off_grow_to;    /* uint16 [N][S] */
  size_t off_vel;        /* uint8  [N][S]    0 none, 1 +x, 2 +y, 3 -x, 4 -y */
  size_t off_body;       /* uint16 [N][S][cap] padded ids, head first */
  size_t off_fruit;      /* classic: uint16 [N][F] padded ids;  adversarial/cut: uint8 [N][V*V] counts */
  int32_t cap;           /* D*D + 1 rounded up to a multiple of 8 */
  int32_t fruit_is_grid; /* 0 list, 1 count grid */
} snk_state_layout;

typedef struct snk_handle snk_handle;

int snk_version(void);
const char* snk_last_error(void);

/* gym.make(id) + env.__init__(**kwargs) + env.seed()  (utils.py:37-39), for N envs at once.
 * snk_create reads ONE environment variable, SNK_DEBUG: a comma-separated key=value list of experiment switches
 * (force_kernel, lane, adaptive, alt_hi, epw, delta, restore_thr; DESIGN.md section 4.7).  None of them changes results;
 * unset is the production configuration.  An unknown key, or a force_kernel / lane value that is not listed there, is
 * SNK_EINVAL.  snk_create_ex takes that string explicitly (NULL = production) and reads no environment. */
int snk_create(const snk_config* cfg, snk_handle** out);
int snk_create_ex(const snk_config* cfg, const char* debug_opts, snk_handle** out);
/* VecEnv.close()  (subproc_vec_env.py:73-83). */
int snk_destroy(snk_handle* h);
int snk_get_config(const snk_handle* h, snk_config* out);
int snk_get_buffers(const snk_handle* h, snk_buffers* out);

/* VecEnv.reset()  (subproc_vec_env.py:63-66 -> SnakeEnv.reset, snake_multiple_test.py:219-232).
 * d_mask == NULL resets every env; otherwise only envs with d_mask[i] != 0 (their obs is rewritten,
 * the others are left untouched). */
int snk_reset(snk_handle* h, const uint8_t* d_mask, void* stream);

/* VecEnv.step_async + step_wait  (subproc_vec_env.py:52-61 -> SnakeEnv.step,
 * snake_multiple_test.py:166-197, get_multi_snake_ob :93-95, Monitor.step monitor.py:57-78).
 * d_actions: int8 [N][S]; values outside the rule-set's action range are no-ops
 * (snake_multiple_test.py:108-115).  One fused kernel launch. */
int snk_step(snk_handle* h, const int8_t* d_actions, void* stream);

/* Same step through HOST buffers, the shape in which SubprocVecEnv hands data to the learner
 * (numpy arrays): copies actions H2D, steps, copies results D2H and synchronises `stream`.
 * Any of the h_ output pointers may be NULL to skip that copy.  Host buffers should be pinned. */
int snk_step_host(snk_handle* h, const int8_t* h_actions, uint8_t* h_obs, float* h_reward,
                  uint8_t* h_done, uint8_t* h_num_alive, void* stream);
/* Same, but h_obs receives only the first n_views_out views of every pixel, packed as [N][H][W][3 n_views_out]
 * (1 <= n_views_out <= 4, or 0 / K for all views).  The reference learner keeps view 0 alone in its rollout
 * (ppo_multi_agent_new.py:181, `obs[..., 0:3]`), so with n_views_out = 1 the D2H copy carries 1/K of the bytes; the
 * views are gathered on the device by a small kernel first. */
/* SNK_OBS_GRID: h_obs receives the [N][V][V] grid; n_views_out other than 0 is SNK_EINVAL (expand on the device first). */
int snk_step_host_views(snk_handle* h, const int8_t* h_actions, uint8_t* h_obs, int32_t n_views_out, float* h_reward,
                        uint8_t* h_done, uint8_t* h_num_alive, void* stream);
/* VecEnv.step_async proper: enqueues the H2D copy, the step and the D2H copies and returns; the caller synchronises
 * `stream` (VecEnv.step_wait) before reading the host buffers. */
int snk_step_host_async(snk_handle* h, const int8_t* h_actions, uint8_t* h_obs, int32_t n_views_out, float* h_reward,
                        uint8_t* h_done, uint8_t* h_num_alive, void* stream);

/* The same step for a learner that keeps the observations in HBM (north_star) but is driven from the host: N*S action
 * bytes in, the per-env scalars out, nothing else crosses PCIe.  SNK_SCALAR_SLOTS slots (slot = step index modulo the
 * slots the caller uses, at least 2) let the copies run on streams of their own beside the step stream: the H2D of step
 * t+1 and the D2H of step t-1 overlap the kernel of step t, so `stream` carries kernels only.  h_out (pinned, snk_scalars_layout bytes) receives ONE block per step:
 *   reward float[N] | done uint8[N] | num_alive uint8[N] | episode return float[N] | episode length int32[N]
 * (the last two valid where done: Monitor's r / l), each part 16-byte aligned at the offsets snk_scalars_layout reports
 * (out[0] = block bytes, out[1..5] = offsets in that order).  The call returns at once; snk_scalars_wait(slot) blocks
 * until the block of the slot's last step has arrived.  Before a slot is reused its previous block must have been
 * consumed (the call orders the device side itself; the host side is the caller's: wait, read, then step again).
 * These steps write the observations as usual (handle buffer / snk_set_obs_target) but NOT the handle's own scalar
 * buffers of snk_get_buffers.  Replaces the `obs, rewards, dones, infos = env.step(actions)` round trip of Runner.run
 * (ppo_multi_agent_new.py:186-192) for an on-device learner. */
#define SNK_SCALAR_SLOTS 4
int snk_scalars_layout(const snk_handle* h, size_t* out /*[6]*/);
int snk_step_scalars_async(snk_handle* h, const int8_t* h_actions, uint8_t* h_out, int32_t slot, void* stream);
int snk_scalars_wait(snk_handle* h, int32_t slot);

/* Pinned host memory for the h_ buffers above, placed on the NUMA node the handle's GPU is attached to (sysfs
 * numa_node of its PCI device; pages bound with set_mempolicy around cudaHostAlloc).  With one process per GPU this
 * keeps every rank's D2H stream on its own socket.  *numa_node (may be NULL) receives the node, or -1 when the
 * placement could not be applied (the memory is still pinned).  Freed by snk_host_free or snk_destroy. */
int snk_host_alloc(snk_handle* h, size_t bytes, void** out, int32_t* numa_node);
int snk_host_free(snk_handle* h, void* ptr);

/* Write observations straight into a caller-owned device buffer (e.g. slot t of the learner's
 * rollout buffer, ppo_multi_agent_new.py:181) instead of the handle's own d_obs.
 * NULL restores the internal buffer.  Must be 16-byte aligned. */
int snk_set_obs_target(snk_handle* h, uint8_t* d_obs, size_t bytes);

/* The learner's rollout keeps the MAIN snake's view alone (ppo_multi_agent_new.py:181 `mb_obs.append(self.main_obs)`,
 * with main_obs = obs[..., 0:3], :162); the opponents' views are needed once, for their action, and then dropped.
 * With a main-view target set, every snk_step / snk_reset additionally writes view 0 of all envs, packed as
 * [N][H][W][3], into d_main (slot t of a [nsteps][N][H][W][3] buffer) while all K views stay in the handle's own,
 * transient observation buffer.  NULL switches it off.  (A gather kernel behind the step kernel: the interleaved
 * [N][H][W][3K] layout of the reference is what the step kernel streams out; see DESIGN.md section 4.9 for why a planar
 * store was not adopted.) */
/* SNK_OBS_GRID: SNK_EINVAL (the grid is already compact; snk_expand_views with n_views = 1 gives view 0). */
int snk_set_main_view_target(snk_handle* h, uint8_t* d_main, size_t bytes);

/* T steps back to back into a caller-owned rollout buffer, no host round trip: step t reads
 * d_actions[t] (int8 [T][N][S]) and writes its observations into d_obs[t] ([T][N][H][W][3K]), its
 * rewards into d_reward[t] (float [T][N]) and its dones into d_done[t] (uint8 [T][N]).  Replaces the
 * rollout loop of Runner.run (ppo_multi_agent_new.py:178-198: mb_obs / mb_rewards / mb_dones appends)
 * for a scripted or pre-sampled action stream.  d_reward / d_done may be NULL.  Afterwards the
 * handle's own buffers (snk_get_buffers) hold the last step, as after T calls of snk_step. */
int snk_rollout(snk_handle* h, const int8_t* d_actions, int32_t T, uint8_t* d_obs, float* d_reward,
                uint8_t* d_done, void* stream);

/* The step loop as ONE launch: T consecutive steps captured into a CUDA graph (kernel nodes linked by programmatic
 * dependent-launch edges, plus, after snk_comm_init, one NCCL all-reduce node per step on a forked branch).  Replaces
 * the Python `for _ in range(self.nsteps): ... self.env.step(actions)` loop of Runner.run (ppo_multi_agent_new.py:178-198)
 * for pre-sampled / scripted action streams, and is what snk_rollout launches internally (it caches the graph of its
 * last argument set).  Step t reads action batch t % n_batches of d_actions (int8 [n_batches][N][S]).  d_obs / d_reward /
 * d_done as in snk_rollout, each may be NULL (the handle's own buffers, or the snk_set_obs_target target current at
 * creation, are then written by every step).  flags: SNK_GRAPH_SYNC_BACK copies the last rollout slot back into the
 * handle's own buffers.  A graph stays valid while the handle and the buffers it was created with live. */
#define SNK_GRAPH_SYNC_BACK 1u
typedef struct snk_graph snk_graph;
int snk_graph_create(snk_handle* h, const int8_t* d_actions, int32_t n_batches, int32_t T, uint8_t* d_obs,
                     float* d_reward, uint8_t* d_done, uint32_t flags, snk_graph** out);
/* The scripted fruit-seeking policy in the loop: every step is the policy kernel (snk_gen_scripted_actions with step index
 * step0 + t, reading the state the previous step left) followed by the step kernel, T times, one launch. */
int snk_graph_create_scripted(snk_handle* h, int32_t T, uint64_t step0, uint64_t seed, int32_t eps_permille, snk_graph** out);
int snk_graph_launch(snk_graph* g, void* stream);
int snk_graph_destroy(snk_graph* g);

/* Generalised advantage estimation over a rollout, on the device (the numpy loop at the end of
 * Runner.run, ppo_multi_agent_new.py:205-218), bit-exact with that loop's mixed precision: float32
 * inputs, gamma * next_value in float32, everything else in float64, advantages rounded to float32,
 * returns = advs + values in float32.  d_dones[t] is the done flag BEFORE step t (mb_dones[t]);
 * d_last_dones / d_last_values are the flags / value estimates after the last step.  All arrays
 * [T][N] (or [N]) on `device`.  Not tied to a handle. */
int snk_gae(const float* d_rewards, const float* d_values, const uint8_t* d_dones, const float* d_last_values,
            const uint8_t* d_last_dones, double gamma, double lam, int32_t T, int64_t N, float* d_advs,
            float* d_returns, int32_t device, void* stream);

/* SNK_OBS_GRID -> RGB views.  d_grid: uint8 [n][V][V] cell codes (V = size + 2, 3 <= V <= 256), e.g. a handle's grid
 * observations, a [T][N][V][V] rollout (n = T*N) or a gathered minibatch.  d_out: uint8 [n][V][V][3 n_views] receives
 * views first_view .. first_view + n_views - 1 of every cell (the colour rule at SNK_CELL_*), byte-identical to those
 * channels of the native observation of the same state; with first_view = 0 and n_views = K it IS the native
 * observation.  0 <= first_view, 1 <= n_views, first_view + n_views <= 32.  Not tied to a handle; stream-ordered on
 * `stream` on `device`, no allocation, no synchronisation, so it can be recorded into a CUDA graph.  16-byte aligned
 * buffers take the vector path; any alignment is accepted. */
int snk_expand_views(const uint8_t* d_grid, int64_t n, int32_t size, int32_t first_view, int32_t n_views,
                     uint8_t* d_out, int32_t device, void* stream);

/* SNK_OBS_GRID -> the first layer of a policy network: a 3x3 SAME convolution 3 -> C (C = 32, the `custom` network of
 * the reference's policies.py), + bias, ReLU, over view `view` of the grid scaled by 1/255, without the RGB image.
 * Class order (the colour of view k at SNK_CELL_*, as c = 0..6):
 *   0 empty (0, 0, 0)   1 fruit (255, 0, 0)   2 wall (255, 255, 255)   3 self body (0, 204, 0)   4 self head (191, 242, 191)
 *   5 other body (0, 51, 204)   6 other head (128, 154, 230)
 * A snake cell is "self" when its snake index equals `view`, so views >= S have no self cells; code 2 is class 0.  The
 * zero padding of SAME is class 0.  Taps t = 3 dy + dx, dy, dx = 0..2 row-major over the kernel window, cell (y + dy - 1,
 * x + dx - 1), as Conv2d's cross-correlation indexes weight[o][rgb][dy][dx].
 * snk_grid_conv_in: d_table float [9][7][C], d_table[t][c][o] = sum_rgb weight[o][rgb][t] colour[c][rgb] / 255 (rows
 * c = 0 are zero, since empty is black, and are not read: empty taps are skipped); d_bias float [C].  d_out float [n][V][V][C] (NHWC: a channels_last [n, C, V, V] tensor) receives
 *   out[i][p][o] = max(0, bias[o] + sum_t table[t][class(grid[i][p + t])][o])   (taps summed in increasing t).
 * snk_grid_conv_in_wgrad: d_out is that output (its zeros are the ReLU mask) and d_gout float [n][V][V][C] the gradient
 * of the loss with respect to it.  d_hist float [9][7][C] receives
 *   hist[t][c][o] = sum over cells p of every grid with class(grid[p + t]) == c of (out[p][o] > 0 ? gout[p][o] : 0),
 * from which dweight[o][rgb][t] = sum_c colour[c][rgb] / 255 hist[t][c][o] and dbias[o] = sum_c hist[4][c][o].  Class 0
 * is computed as the total minus classes 1..6.  Deterministic: the same inputs give the same bits on every call (per-CTA
 * partials in shared memory, written to d_work, added up in a fixed order; no atomics).  d_work: at least
 * SNK_GRID_CONV_WORK_BYTES(n * V * V) bytes, 4-byte aligned; never more than SNK_GRID_CONV_WORK_BYTES_MAX.
 * Rejected (SNK_EINVAL): channels other than SNK_GRID_CONV_CHANNELS; size outside 1..254 (3 <= V <= 256); view outside
 * 0..31; n < 0; a NULL buffer or, for snk_grid_conv_in, d_table / d_bias / d_out not 16-byte aligned; for the wgrad
 * d_out / d_gout / d_hist / d_work not 4-byte aligned or work_bytes below the formula.  n = 0 does nothing (d_hist is
 * not written).  Not tied to a handle; stream-ordered on `stream` on `device`, no allocation, no synchronisation, so
 * both can be recorded into a CUDA graph. */
#define SNK_GRID_CONV_CHANNELS 32
#define SNK_GRID_CONV_CLASSES 7
#define SNK_GRID_CONV_WGRAD_CELLS_PER_CTA 2048
#define SNK_GRID_CONV_WGRAD_MAX_CTAS 592
#define SNK_GRID_CONV_PART_FLOATS ((9 * (SNK_GRID_CONV_CLASSES - 1) + 1) * SNK_GRID_CONV_CHANNELS) /* per CTA */
#define SNK_GRID_CONV_WORK_BYTES(n_cells)                                                                              \
  ((size_t)((((n_cells) + SNK_GRID_CONV_WGRAD_CELLS_PER_CTA - 1) / SNK_GRID_CONV_WGRAD_CELLS_PER_CTA) <                \
                    SNK_GRID_CONV_WGRAD_MAX_CTAS                                                                       \
                ? (((n_cells) + SNK_GRID_CONV_WGRAD_CELLS_PER_CTA - 1) / SNK_GRID_CONV_WGRAD_CELLS_PER_CTA)            \
                : SNK_GRID_CONV_WGRAD_MAX_CTAS) *                                                                      \
   SNK_GRID_CONV_PART_FLOATS * 4)
#define SNK_GRID_CONV_WORK_BYTES_MAX ((size_t)SNK_GRID_CONV_WGRAD_MAX_CTAS * SNK_GRID_CONV_PART_FLOATS * 4)
int snk_grid_conv_in(const uint8_t* d_grid, int64_t n, int32_t size, int32_t view, const float* d_table,
                     const float* d_bias, int32_t channels, float* d_out, int32_t device, void* stream);
int snk_grid_conv_in_wgrad(const uint8_t* d_grid, int64_t n, int32_t size, int32_t view, const float* d_out,
                           const float* d_gout, int32_t channels, float* d_hist, void* d_work, size_t work_bytes,
                           int32_t device, void* stream);

/* SNK_OBS_GRID -> the first layer of the reference's `nature_cnn` on its WarpFrame view: an 8x8 stride-4 VALID
 * convolution 3 -> C (C = 32) + bias, ReLU, over view `view` replicated f x f per cell to 84 x 84 and scaled by 1/255
 * (the observation of SNK_OBS_ATARI84), without the image.  V = size + 2 must divide 84 with 3 <= V <= 42 (V = 3, 4, 6,
 * 7, 12, 14, 21, 28, 42); f = 84 / V pixels per cell.  Classes and colours are those of snk_grid_conv_in.
 * Output pixel (oy, ox), 0 <= oy, ox < 20, reads pixel rows 4 oy .. 4 oy + 7, i.e. cell rows floor(4 oy / f) + a.  How
 * the 8 kernel rows fall on those cells depends only on the phase oy mod P, P = f / gcd(f, 4):
 *   M[phi][a][d] = 1 if floor((4 phi + d) / f) - floor(4 phi / f) == a else 0     (0 <= a < C, 0 <= d < 8)
 * with C the most cells a window spans per axis; block a of phase phi is reached when M[phi][a] is not all zero.
 * snk_grid_conv84_geometry: out[0..3] = f, P, C and the workspace bytes snk_grid_conv84_in_wgrad needs for n grids.  Pure
 * host arithmetic.  SNK_EINVAL for an unsupported size, n < 0 or a NULL out.
 * snk_grid_conv84_in: d_table float [P][P][C][C][7][C_out],
 *   table[py][px][a][b][c][o] = sum_{dy,dx} M[py][a][dy] M[px][b][dx] sum_rgb weight[o][rgb][dy][dx] colour[c][rgb] / 255
 * (rows c = 0 are zero and not read: empty blocks are skipped); d_bias float [C_out].  d_out float [n][20][20][C_out]
 * (NHWC: a channels_last [n, C_out, 20, 20] tensor) receives
 *   out[i][oy][ox][o] = max(0, bias[o] + sum_{a,b} table[oy % P][ox % P][a][b][class(grid[i][cy + a][cx + b])][o]),
 *   cy = floor(4 oy / f), cx = floor(4 ox / f), blocks summed in increasing a C + b, unreached blocks skipped.
 * snk_grid_conv84_in_wgrad: d_out is that output (its zeros are the ReLU mask), d_gout float [n][20][20][C_out] the
 * gradient of the loss with respect to it.  d_hist float [P][P][C][C][7][C_out] receives
 *   hist[py][px][a][b][c][o] = sum over outputs (oy, ox) of every grid with oy % P = py, ox % P = px and
 *                              class(grid[cy + a][cx + b]) == c of (out > 0 ? gout : 0)
 * (zero for unreached blocks; class 0 is the phase's total minus classes 1..6), from which
 *   dweight[o][rgb][dy][dx] = sum M[py][a][dy] M[px][b][dx] colour[c][rgb] / 255 hist[py][px][a][b][c][o]
 *   dbias[o] = sum_{py,px,c} hist[py][px][0][0][c][o].
 * Deterministic: the work is split by phase pair and the CTA count depends on (n, V) only; each CTA adds its warps' bins
 * in warp order into one partial in d_work, and the partials are added in CTA order.  No atomics.  d_work: at least
 * geometry's out[3] bytes, 4-byte aligned.
 * Rejected (SNK_EINVAL): channels other than SNK_GRID_CONV_CHANNELS; an unsupported size; view outside 0..31; n < 0; a
 * NULL buffer or, for snk_grid_conv84_in, d_table / d_bias / d_out not 16-byte aligned; for the wgrad d_out / d_gout /
 * d_hist / d_work not 4-byte aligned or work_bytes below geometry's figure.  n = 0 does nothing (d_hist is not written).
 * Not tied to a handle; stream-ordered on `stream` on `device`, no allocation, no synchronisation, so both can be
 * recorded into a CUDA graph. */
#define SNK_GRID_CONV84_OUT 20 /* output rows and columns */
#define SNK_GRID_CONV84_WGRAD_OUTPUTS_PER_CTA 2048
#define SNK_GRID_CONV84_WGRAD_MAX_CTAS 592
int snk_grid_conv84_geometry(int32_t size, int64_t n, int64_t* out /*[4]: f, P, C, workspace bytes for n grids*/);
int snk_grid_conv84_in(const uint8_t* d_grid, int64_t n, int32_t size, int32_t view, const float* d_table,
                       const float* d_bias, int32_t channels, float* d_out, int32_t device, void* stream);
int snk_grid_conv84_in_wgrad(const uint8_t* d_grid, int64_t n, int32_t size, int32_t view, const float* d_out,
                             const float* d_gout, int32_t channels, float* d_hist, void* d_work, size_t work_bytes,
                             int32_t device, void* stream);

/* Replay mode: per-env tapes of the reference's np_random.randint draws
 * (snake_multiple_test.py:200, :215).  CSR: env i owns vals/bounds[offsets[i] .. offsets[i+1]).
 * Host arrays, copied to the device (synchronous).  Switches the handle to SNK_RNG_TAPE. */
int snk_set_draw_tape(snk_handle* h, const uint32_t* h_vals, const uint32_t* h_bounds,
                      const uint64_t* h_offsets);

/* Canonical state (parity tests, checkpoint / resume) through HOST memory.  Synchronous. */
int snk_state_layout_of(const snk_config* cfg, snk_state_layout* out);
int snk_dump_state(snk_handle* h, void* h_dst, size_t bytes);
/* Envs [first, first + count) only, as the blob of a `count`-env configuration (snk_state_layout_of with num_envs =
 * count): parity checks of a slice of a large batch without moving the whole state. */
int snk_dump_state_range(snk_handle* h, int64_t first, int64_t count, void* h_dst, size_t bytes);
/* Rejects (SNK_ESTATE, offending snakes left empty) bodies longer than the board, cell ids outside the padded grid,
 * velocity codes above 4 and consecutive segments that are not adjacent cells. */
int snk_load_state(snk_handle* h, const void* h_src, size_t bytes);

/* Per-env state on the device: start episodes from stored states, paired evaluation from the same start states, search by
 * cloning one env into many slots.  None of the three synchronises, allocates or touches host memory; all work is
 * stream-ordered on `stream`, so they can be recorded into a CUDA graph.  Indices are int64 device arrays (the dtype of a
 * PyTorch index tensor).  An index outside [0, N) raises SNK_DEVERR_BAD_STATE (read it with snk_check_errors) and nothing is written for
 * that entry; the launch itself still runs.  Device blobs must be 16-byte aligned.
 *   What moves: all of the canonical state -- t, spare, draw_ctr, Monitor's running ep_ret / ep_len, bodies, grow_to, vel
 *   and fruits.  What does not: the per-step outputs (d_reward, d_done, d_num_alive, d_episode_*), the running d_stats
 *   sums, and the RNG key, which stays (seed, global id of the DESTINATION env).  A restored or copied env continues with
 *   the source's draw_ctr on its own Philox stream, so a clone is identical to its source only until the next random
 *   draw (a fruit respawn, an auto-reset).  In tape mode draw_ctr indexes the destination env's tape.
 *   Observations are not re-encoded (as after snk_load_state): restored / copied envs are marked so that the next step
 *   writes their images whole; call snk_reset with an all-zero mask to re-encode every env's observation at once. */
/* Canonical state of envs d_idx[0..count) (NULL: envs [0, count)) into the DEVICE buffer d_blob, laid out as the blob of a
 * `count`-env configuration (snk_state_layout_of with num_envs = count): byte-identical to what snk_dump_state_range
 * writes for the same envs.  Indices may repeat. */
int snk_save_envs(snk_handle* h, const int64_t* d_idx, int64_t count, void* d_blob, size_t bytes, void* stream);
/* Env d_idx[j] (NULL: env j) <- entry j of the device blob d_blob (a `count`-env blob).  Validates exactly what
 * snk_load_state validates; a rejected snake is left empty and SNK_DEVERR_BAD_STATE is raised.  Destination indices must
 * be distinct.  The blob may come from a handle of another num_envs / seed / env_id_base, as long as size, n_snakes,
 * n_fruits and rules are the same. */
int snk_restore_envs(snk_handle* h, const int64_t* d_idx, int64_t count, const void* d_blob, size_t bytes, void* stream);
/* Env d_dst[j] <- env d_src[j], private layout to private layout (record, chain words / ring row, fruit grid + bitmap):
 * about 1/12 of the bytes of a save + restore through a blob at 2 snakes on 19x19.  d_src may repeat (1 -> many); d_dst
 * must be distinct and disjoint from d_src. */
int snk_copy_envs(snk_handle* h, const int64_t* d_src, const int64_t* d_dst, int64_t count, void* stream);
/* snk_copy_envs across handles: env d_dst[j] of `dst` <- env d_src[j] of `src`, private layout to private layout, one
 * kernel.  `src` is only read.  Everything else is as for snk_copy_envs: d_src may repeat, d_dst must be distinct (and,
 * when src == dst, disjoint from d_src); the RNG key stays (seed, global id) of the destination; the destination's
 * observations are not re-encoded.  An index outside [0, N) of its own handle raises SNK_DEVERR_BAD_STATE on `dst` and
 * that entry is skipped.  Rejected (SNK_EINVAL naming the field, before any CUDA call): a NULL argument, count < 1,
 * handles on different devices, of another size, n_snakes, n_fruits or rules, or of another private layout (body family,
 * record words, chain words, ring capacity, fruit grid stride or bitmap words).  The family follows the launch plan, which
 * follows the observation size, so two handles of one configuration in different obs_modes may be rejected: states are
 * not converted between layouts (save_envs / restore_envs do that through the canonical blob). */
int snk_clone_envs(const snk_handle* src, const int64_t* d_src, snk_handle* dst, const int64_t* d_dst, int64_t count, void* stream);

/* Episode statistics (Monitor's aggregate role).  snk_get_stats synchronises `stream`. */
int snk_get_stats(snk_handle* h, double* h_stats /*[SNK_NSTATS]*/, void* stream);
int snk_reset_stats(snk_handle* h, void* stream);
/* Reads and clears the sticky device error flags (synchronises `stream`). */
int snk_check_errors(snk_handle* h, uint32_t* flags, void* stream);

/* The path's ONE collective (SURVEY.md section 8e): with envs sharded over G GPUs, one process and one handle per GPU,
 * every step's local statistics vector is summed over the ranks -- Monitor's per-step episode records
 * (monitor.py:57-78, collected every step by Runner.run, ppo_multi_agent_new.py:189-192) in aggregate.  After
 * snk_comm_init each snk_step / graph step ends with the last CTA copying the handle's running sums into a snapshot
 * slot; a high-priority side stream all-reduces that slot (ncclAllReduce, 8 doubles, NVLink / NVSwitch) while the next
 * step runs, and the result is read one step late.  No other inter-GPU traffic exists on the path.
 *   snk_comm_unique_id  rank 0 creates the 128-byte NCCL id; the caller ships it to the other ranks (any channel).
 *   snk_comm_init       collective over all ranks; NCCL is bound at run time (dlopen of libnccl.so.2), no link dependency.
 *   snk_get_stats_global  sums over all ranks as of the last completed reduction (synchronises `stream`); without a
 *                       communicator it equals snk_get_stats. */
/* The same reduction WITHOUT a collective library and without a kernel of its own -- the default of the Python layer.
 * Every rank exports a small inbox (cudaIpc) and maps its peers' inboxes (snk_peer_connect, after the caller has gathered
 * the 64-byte handles of all ranks in rank order over any channel).  From then on the FIRST CTA of every step kernel
 * stores the rank's running sums -- complete as of the previous step -- into its slot of every peer's inbox: eight
 * aligned 8-byte stores per peer over NVLink / NVSwitch, posted, draining while the CTA steps its envs.  Every statistic
 * is a monotonic sum and an aligned 8-byte store is one transaction, so there are no fences, no versions and no
 * rendezvous: a rank never waits for another, and compute step and exchange are one kernel.  snk_get_stats_global pushes
 * the rank's final sums and returns own sums + the peers' latest pushes: the global statistics as of about one step ago,
 * exact once every rank has made that call after its last step (call it, barrier, call it again).  Ranks must be
 * processes of one node with peer access between their GPUs; at most 16.
 * snk_comm_enable(h, 0) switches the per-step reduction of either form off (A/B measurements), 1 on again. */
int snk_peer_export(snk_handle* h, uint8_t* out64);
int snk_peer_connect(snk_handle* h, const uint8_t* handles /*[n_ranks][64]*/, int32_t n_ranks, int32_t rank);
int snk_comm_enable(snk_handle* h, int32_t on);
int snk_comm_unique_id(uint8_t* out128);
int snk_comm_init(snk_handle* h, const uint8_t* id128, int32_t n_ranks, int32_t rank);
int snk_get_stats_global(snk_handle* h, double* h_stats /*[SNK_NSTATS]*/, void* stream);
int snk_comm_info(const snk_handle* h, int32_t* out /*[4]: ranks, rank, all-reduces issued, NCCL version code*/);
/* Mean duration (microseconds, CUDA events on the side stream) of `iters` back-to-back all-reduces of the statistics
 * vector: the latency bench.py reports for the collective.  Collective over all ranks; synchronises the device. */
int snk_comm_bench(snk_handle* h, int32_t iters, double* mean_us);

/* Synthetic uniform action stream for benchmarks: Philox key (seed, global env id), stream 1,
 * counter = step * S + snake, value in [0, n_actions).  d_actions: int8 [N][S]. */
int snk_gen_actions(snk_handle* h, int8_t* d_actions, uint64_t step, uint64_t seed,
                    int32_t n_actions, void* stream);

/* Scripted policy for benchmarks (SURVEY.md section 8d second stream): every live snake turns toward
 * its nearest fruit unless the next cell is a wall or a body cell, else keeps going; with probability
 * eps_permille / 1000 a uniform random action instead (Philox stream 2).  Keeps snakes long (larger
 * SigmaL, fewer resets).  Lane-family configurations with classic fruit lists only; eps_permille outside 0..1000 is
 * SNK_EINVAL.  Exactly, per env e and snake s: a dead snake gets 0.  The draw rnd is the Philox value of key (seed, global
 * env id), stream 2, counter step * S + s (as for snk_gen_actions) bounded to [0, 5000); rnd / 5 < eps_permille gives
 * action rnd % 5.  Otherwise action a = 1..4 is a candidate unless it reverses the velocity, its cell is on the border,
 * or a segment of any snake (tails included) lies there; its distance is the least Manhattan distance from that cell to
 * the first F fruits (with F = 0 all distances are equal).  The lowest a of strictly smallest distance wins; with no
 * candidate left the action is 0, which keeps the snake going in its current direction. */
int snk_gen_scripted_actions(snk_handle* h, int8_t* d_actions, uint64_t step, uint64_t seed,
                             int32_t eps_permille, void* stream);

/* Head-to-head evaluation (the reference's evaluate_snake.py, played over many envs at once; DESIGN.md section 4.18).
 * Outcome of one episode of one env: let d_s be the step within the episode at which seat s got reward -1 (it died), or
 * +infinity if it never did.  Seat s WINS if d_s > d_j for every other seat j, DRAWS if d_s >= d_j for every j and
 * d_s == d_j for at least one j != s, and otherwise LOSES.  Under the reference's rules (an episode ends when seat 0 dies
 * or at max_steps) both seats alive at the timeout is a draw, dying on the same step is a draw, seat 1 dying first and
 * seat 0 later is a win for seat 0, and at S = 1 every episode is a win (only the score fields mean anything).
 * Per seat the counters also hold the fruits (sum of positive rewards; more than 1 on a step when fruit stacks on a cell
 * under the adversarial and cut rules), deaths, steps alive (counting the death step; the episode length for a seat
 * that survives), the sum of squared episode returns (return = fruits - 1 if the seat died, else fruits) and the sum of
 * episode lengths.  Every counter is an int64 sum of integers, so a result is the same bits on every run.
 * snk_tally_layout: out[0] = bytes of the work area for the handle (int32 step counter and episodes counted [N], death
 * step and fruits [N][S] of the running episode, each part 16-byte aligned), out[1] = SNK_TALLY_FIELDS.  Host only.
 * snk_tally, launched after every snk_step on the step's stream (one kernel): reads the handle's d_reward_all, d_done and
 * d_episode_len, and d_group (int32 [N]: the counter group of every env).  Every finished episode of an env adds its
 * outcome per seat to d_counts (int64 [n_groups][S][SNK_TALLY_FIELDS]) row d_group[env].  An env that has counted
 * episodes_per_env episodes is ignored from then on, and *d_envs_done (int64) counts such envs: poll it until it
 * reaches N and every env has contributed exactly episodes_per_env episodes.  The caller zeroes d_work, d_counts and
 * d_envs_done when it resets the envs (snk_reset), and the handle must auto-reset.  Stream-ordered, no allocation, no
 * synchronisation, so it can be recorded into a CUDA graph.
 * Rejected (SNK_EINVAL, before any CUDA call): n_groups < 1, episodes_per_env < 1, a NULL argument, d_group not 4-byte,
 * d_work not 16-byte, d_counts or d_envs_done not 8-byte aligned.  A group id outside [0, n_groups) raises
 * SNK_DEVERR_BAD_STATE (read it with snk_check_errors) and that env is skipped: it is never counted and never finished. */
#define SNK_TALLY_WINS 0
#define SNK_TALLY_DRAWS 1
#define SNK_TALLY_LOSSES 2
#define SNK_TALLY_FRUITS 3
#define SNK_TALLY_DEATHS 4
#define SNK_TALLY_STEPS_ALIVE 5
#define SNK_TALLY_RETURN_SQ 6
#define SNK_TALLY_LENGTH 7
#define SNK_TALLY_FIELDS 8
int snk_tally_layout(const snk_handle* h, size_t* out /*[2]*/);
int snk_tally(snk_handle* h, const int32_t* d_group, int32_t n_groups, int32_t episodes_per_env, void* d_work,
              int64_t* d_counts, int64_t* d_envs_done, void* stream);

/* Rollout search (DESIGN.md section 4.19): the bookkeeping of a search handle whose slots are clones of roots.  With
 * A = n_actions and R = rollouts, slot j < n_roots * A * R belongs to root m = j / (A R) and candidate action
 * a = (j / R) % A.  Slots at and beyond n_roots * A * R are never read or written.  The caller keeps d_ret (int32 [slots],
 * 4-byte aligned) and d_active (uint8 [slots]) between the calls; each is one kernel, stream-ordered, without allocation
 * or synchronisation.
 *   snk_search_begin, before the search's first snk_step: seat `seat`'s action of slot j in d_actions (int8 [N][S], the
 *     step's action array) <- a; d_ret[j] <- 0; d_active[j] <- 1.
 *   snk_search_accumulate, after every snk_step: an active slot adds the handle's d_reward_all[j][seat] (an integer) to
 *     d_ret[j].  The step where that reward is -1 (the seat died, the death rule of snk_tally) or where d_done[j] is set
 *     is the slot's last counted step: d_active[j] <- 0 after it.
 *   snk_search_pick: V[m][a] = sum of d_ret over the R slots of (m, a), written as float to d_value [n_roots][A]; the
 *     lowest a of maximal V[m][a] is written to d_pick[m * pick_stride] (int8; pick_stride = S puts it straight into a
 *     column of an [N][S] action array).  Every sum is of integers, so the result is the same bits in any order.
 * Rejected (SNK_EINVAL, before any CUDA call): a NULL handle or array, seat outside [0, S), n_actions outside 1..127,
 * rollouts < 1, n_roots < 1 or n_roots * A * R > N, pick_stride < 1, d_ret or d_value not 4-byte aligned. */
int snk_search_begin(snk_handle* h, int8_t* d_actions, int32_t seat, int32_t n_actions, int32_t rollouts, int64_t n_roots,
                     int32_t* d_ret, uint8_t* d_active, void* stream);
int snk_search_accumulate(snk_handle* h, int32_t seat, int32_t n_actions, int32_t rollouts, int64_t n_roots, int32_t* d_ret,
                          uint8_t* d_active, void* stream);
int snk_search_pick(snk_handle* h, int32_t n_actions, int32_t rollouts, int64_t n_roots, const int32_t* d_ret, float* d_value,
                    int8_t* d_pick, int64_t pick_stride, void* stream);

/* Algorithmic bytes of one env-step (SURVEY.md section 8d): obs K*H*W*3 + state 19S + 2*SigmaL + 2F + 30. */
int snk_algorithmic_bytes_per_step(const snk_config* cfg, double mean_sum_len, double* out);

/* Number of kernels launched by this handle since creation (bench.py's gpu_launches). */
int snk_launch_count(const snk_handle* h, uint64_t* out);
/* The launch plan of the step kernel (bench.py's config.kernel): kind (0 lane, 1 tile, 2 dense, 3 rows), grid, block,
 * dynamic shared memory bytes, resident CTAs per SM, envs per CTA. */
int snk_launch_info(const snk_handle* h, int32_t* out /*[6]*/);
/* Which form of the lane path the NEXT eager step will launch (it follows the body-length regime, DESIGN.md 4.8; a classic
 * step recorded into a graph that stores sectors into the own buffer follows thresholds of its own, DESIGN.md 4.20):
 * out[0] = 0 fused kernel, 1 warp-specialised kernel, 3 two kernels (k_lane_logic + k_lane_paint2, or + k_lane_grid in
 * SNK_OBS_GRID, which always uses this form), -1 not a lane-family
 * configuration (2 is no longer reported); out[1] = envs stepped per warp batch of the fused kernel;
 * out[2] = envs per shared-memory image; out[3] = 1 when the handle switches forms by itself. */
int snk_launch_form(const snk_handle* h, int32_t* out /*[4]*/);

#ifdef __cplusplus
}
#endif
#endif /* SNK_H_ */
