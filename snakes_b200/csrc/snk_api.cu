// snk_api.cu -- the extern "C" boundary of libsnk.so (include/snk.h): handle lifetime, device
// buffers, launch planning.  No torch, no Python: plain pointers and sizes.
#include <dlfcn.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/syscall.h>
#include <unistd.h>

#include <algorithm>
#include <string>
#include <vector>

#include "snk_device.cuh"
#include "snk_launch.h"

static thread_local char g_err[512] = "";

static int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

#define CUDA_TRY(expr)                                                                         \
  do {                                                                                         \
    cudaError_t _e = (expr);                                                                   \
    if (_e != cudaSuccess) return fail(SNK_ECUDA, "%s: %s", #expr, cudaGetErrorString(_e));    \
  } while (0)

struct snk_graph;

// ---- NCCL, bound at run time (dlopen): libsnk.so has no link-time dependency on it, and inside a PyTorch process the
// soname resolves to the libnccl.so.2 torch already loaded, so there is one NCCL in the process.
typedef struct ncclComm* ncclComm_t;
typedef struct { char internal[128]; } ncclUniqueId;
struct NcclApi {
  void* so;
  int (*GetUniqueId)(ncclUniqueId*);
  int (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int);
  int (*CommInitRankConfig)(ncclComm_t*, int, ncclUniqueId, int, void* /*ncclConfig_t*/);
  int (*CommDestroy)(ncclComm_t);
  int (*AllReduce)(const void*, void*, size_t, int /*ncclDataType_t*/, int /*ncclRedOp_t*/, ncclComm_t, cudaStream_t);
  const char* (*GetErrorString)(int);
  int (*GetVersion)(int*);
};
static const int kNcclFloat64 = 8, kNcclSum = 0;  // nccl.h: ncclFloat64 = 8, ncclSum = 0 (stable since NCCL 2.0)
// ncclConfig_t as of NCCL 2.18 (nccl.h: size / magic / version head the struct precisely so that a caller built against an
// older layout keeps working: fields beyond `size` take their defaults)
struct NcclConfig218 {
  size_t size; unsigned magic, version;
  int blocking, cgaClusterSize, minCTAs, maxCTAs;
  const char* netName;
  int splitShare;
};

struct snk_handle {
  snk_config cfg;
  snk_state_layout lay;
  Params p;
  LaunchPlan plan;
  int n_sm;
  uint8_t* d_obs_own;     // native observations (the step kernels' output)
  // regime-adaptive lane path: `plan` is the fused kernel, `plan_alt` the two-kernel form (k_lane_logic + k_lane_paint2)
  LaunchPlan plan_alt;
  bool have_alt, use_alt, use_alt_sec;  // use_alt_sec: the form of a graph-captured step that stores sectors (regime_update)
  double* h_regime;            // mapped pinned host memory [2]: env-steps, body cells (Params::regime_out)
  double reg_steps0, reg_cells0, alt_hi, alt_lo, sec_hi, sec_lo;
  const uint8_t* obs_current;  // where the native observations of the CURRENT state are (NULL: not encoded since the state changed)
  uint8_t* d_obs84_own;   // obs_mode atari84: the 84x84 images handed to the caller
  uint8_t* d_obs_user;    // what snk_get_buffers reports: own buffer or the caller's target
  uint8_t* d_main_target; // snk_set_main_view_target: view 0 of every step, packed [N][H][W][3] (NULL = off)
  size_t obs_out_env_bytes;
  int8_t* d_actions_own;
  uint8_t* d_blob;  // staging for dump / load
  uint32_t* d_tape_vals;
  uint32_t* d_tape_bounds;
  uint64_t* d_tape_off;
  size_t blob_bytes;
  uint8_t* d_info;        // done | num_alive | fin_ret | fin_len, contiguous (snk_buffers.d_info_block)
  size_t info_bytes;
  uint8_t* d_views;       // host-buffer step with fewer views than K: packed staging [N][V][V][3 n]
  size_t views_bytes;
  std::vector<void*> allocs;
  std::vector<std::pair<void*, size_t>> host_allocs;  // snk_host_alloc: pinned, NUMA-local
  uint64_t launches;
  // per-step statistics all-reduce (snk_comm_init)
  ncclComm_t comm;
  int comm_ranks, comm_rank;
  cudaStream_t side;           // high-priority side stream the all-reduce runs on
  cudaStream_t cap_stream;     // private stream graphs are captured on
  double* d_snap;              // [2][SNK_NSTATS] per-step snapshots of the local sums (written by the step kernel)
  double* d_global;            // [2][SNK_NSTATS] their sums over all ranks
  cudaEvent_t ev_step[2], ev_red[2], cev_step[2], cev_red[2];  // eager / capture-time fork + join events
  bool ev_red_valid[2];
  uint64_t step_seq;           // steps launched so far: slot = step_seq & 1
  uint64_t collectives;
  int last_slot;
  double* d_global_last;       // the all-reduced vector of the most recent step (a slot of d_global or of a graph)
  // peer-memory form (snk_peer_export / snk_peer_connect)
  uint8_t* d_inbox;            // this rank's inbox (cudaMalloc, exported through cudaIpc)
  void* peer_mapped[SNK_MAX_PEERS];  // the peers' inboxes as opened in this process
  PeerArgs peer;               // ranks == 0: peer form not connected
  bool reduce_enabled;         // snk_comm_enable: A/B switch of the per-step reduction
  snk_graph* rollout_cache;    // the graph of the last snk_rollout call (re-launched when the arguments repeat)
  // snk_step_scalars_async: device slots (actions in, per-env scalars out) and the copy streams beside the step stream
  struct ScalarSlot { int8_t* d_act; uint8_t* d_out; cudaEvent_t ev_in, ev_k, ev_out; bool used, host_synced; } sc[SNK_SCALAR_SLOTS];
  cudaStream_t s_in, s_out;
  size_t sc_bytes, sc_off[5];  // block size; offsets of reward, done, num_alive, episode return, episode length
  std::string debug;
};

static size_t align16(size_t x) { return (x + 15) & ~(size_t)15; }
static int gcd(int a, int b) { return b ? gcd(b, a % b) : a; }

// ---- experiment switches.  ONE string of key=value pairs separated by ',', ' ' or ';', given explicitly to snk_create_ex
// or, for snk_create, read from the single environment variable SNK_DEBUG.  None changes results (all are parity-tested);
// an unset / empty string is the production configuration.  Keys: force_kernel=lane|tile|rows|dense, lane=fused|ws|split,
// adaptive=0, alt_hi=<body cells>, epw=<n>, delta=0|1, restore_thr=<n>.  dbg_check rejects anything else.
static std::vector<std::string> dbg_tokens(const std::string& opts) {
  std::vector<std::string> out;
  for (size_t pos = 0; pos < opts.size();) {
    size_t end = opts.find_first_of(", ;", pos);
    if (end == std::string::npos) end = opts.size();
    if (end > pos) out.push_back(opts.substr(pos, end - pos));
    pos = end + 1;
  }
  return out;
}
static bool dbg_get(const std::string& opts, const char* key, std::string* out) {
  const size_t klen = strlen(key);
  for (const std::string& t : dbg_tokens(opts)) {
    if (t.size() > klen && t.compare(0, klen, key) == 0 && t[klen] == '=') {
      *out = t.substr(klen + 1);
      return true;
    }
  }
  return false;
}
static int dbg_int(const std::string& opts, const char* key, int dflt) {
  std::string v;
  return dbg_get(opts, key, &v) ? atoi(v.c_str()) : dflt;
}
// A stale or mistyped switch would otherwise be ignored and the run would measure the production path without a word.
static int dbg_check(const std::string& opts) {
  static const char* const keys[] = {"force_kernel", "lane", "adaptive", "alt_hi", "epw", "delta", "restore_thr"};
  for (const std::string& t : dbg_tokens(opts)) {
    const size_t eq = t.find('=');
    const std::string key = t.substr(0, eq), val = eq == std::string::npos ? "" : t.substr(eq + 1);
    bool ok = eq != std::string::npos && std::any_of(std::begin(keys), std::end(keys), [&](const char* k) { return key == k; });
    if (key == "force_kernel") ok = ok && (val == "lane" || val == "tile" || val == "rows" || val == "dense");
    if (key == "lane") ok = ok && (val == "fused" || val == "ws" || val == "split");
    if (!ok) return fail(SNK_EINVAL, "unknown debug option '%s'", t.c_str());
  }
  return SNK_OK;
}

// SNK_OBS_GRID has one writer per family (k_lane_grid behind k_lane_logic; k_step_rows<RULES, true>), so the switches
// that choose between RGB writers or tune them would silently measure something else there.  force_kernel=lane|rows and
// restore_thr keep their meaning.
static int dbg_check_grid(const std::string& opts) {
  static const char* const keys[] = {"lane", "delta", "epw", "adaptive", "alt_hi"};
  for (const std::string& t : dbg_tokens(opts)) {
    const size_t eq = t.find('=');
    const std::string key = t.substr(0, eq), val = eq == std::string::npos ? "" : t.substr(eq + 1);
    const bool bad = std::any_of(std::begin(keys), std::end(keys), [&](const char* k) { return key == k; }) ||
                     (key == "force_kernel" && (val == "tile" || val == "dense"));
    if (bad) return fail(SNK_EINVAL, "debug option '%s' does not apply to obs_mode grid", t.c_str());
  }
  return SNK_OK;
}

// Un-paint by zero-fill + border redraw (lane_restore / cta_restore) once a lane would walk more than restore_thr segments.
// `threads` share an image buffer (32: a warp of the fused / ws kernel; 64: k_lane_paint2).  The restore costs each of
// them one 16-byte store per 16 * threads bytes of image plus its share of one env's border units; a walked segment costs
// about 16 instructions.  Measured on B200 (2x19x19, 131072 envs, fruit-seeking policy, sum of lengths 22): thresholds
// 3 / 5 / 8 / 12 -> 145.9 / 145.1 / 146.8 / 152.9 us, always-walk 161.1 us; random actions (sum of lengths 4.4)
// unchanged.  The restore_thr switch overrides it (0 = always walk).
static int restore_threshold(const Params& p, int threads) {
  const int U = (p.C & 1) ? 1 : 2, lanes_per_env = threads / p.TE;
  const int border_units = (2 * (p.V * p.C + p.C) + (p.V - 3) * 2 * p.C) / U;
  const int stores = (int)((size_t)p.TE * p.E / (16 * threads)) + border_units / lanes_per_env;
  return stores / 16 < 3 ? 3 : stores / 16;
}

// Launch planning: fills h->plan, h->plan_alt and the lane geometry of h->p.  Decisions, in order: the kernel family,
// a forced kernel, the lane path's form, small-shard batches, the regime-adaptive alternative.
static int plan_launch(snk_handle* h) {
  const std::string& dbg = h->debug;
  Params& p = h->p;
  const bool grid = h->cfg.obs_mode == SNK_OBS_GRID;
  const int D = p.D, V = p.V, S = p.S, F = p.F, K = p.K;
  const long long N = p.N;
  LaunchPlan& plan = h->plan;
  // grid = work: the CTAs it takes to cover every env
  auto finish = [&](LaunchPlan& pl) {
    return snk_plan(h->cfg.rules, pl, h->n_sm, S, K, (N + pl.envs_per_cta - 1) / pl.envs_per_cta);
  };
  // lane form `form` at te envs per warp image and epw envs per warp batch.  `threads` is what restore_threshold counts
  // as sharing an image buffer: k_lane_grid and the adaptive alternative count k_lane_paint2's 64, the other lane
  // plans a warp's 32.
  auto plan_lane = [&](LaunchPlan& pl, int form, int te, int epw, int threads) {
    p.TE = te; p.EPW = epw;
    p.tile_stride = (int)(((size_t)te * p.E + 127) & ~(size_t)127);
    p.n_groups = (N + epw - 1) / epw;
    const bool two = form == FORM_LANE_SPLIT || form == FORM_LANE_GRID;  // the observation writer: one image per CTA
    pl.form = form;
    pl.block = form == FORM_LANE_WS ? 32 * (WS_PAINT_WARPS + WS_LOGIC_WARPS) : 64;
    pl.smem = (size_t)(two ? 1 : 2) * p.tile_stride;
    pl.envs_per_cta = two ? te : form == FORM_LANE_WS ? 32 * WS_LOGIC_WARPS : 2 * epw;  // fused: 2 warps per CTA
    pl.restore_thr = dbg_int(dbg, "restore_thr", restore_threshold(p, threads));
    return finish(pl);
  };

  // lane kernel (chain-coded bodies, lane per env) for small boards; otherwise the warp-per-env tile kernel while
  // W observations + template + scratch leave room for >= 2 CTAs per SM; otherwise the CTA-per-env rows / dense kernel.
  std::string force;
  dbg_get(dbg, "force_kernel", &force);
  int TE = 0;
  if ((grid || snk_lane_supported(S, K)) && S <= 4 && F <= 4 && D <= 32) {  // grid: k_lane_grid exists for every K
    const int cand[3] = {32, 16, 8};
    for (int i = 0; i < 3 && !TE; ++i)
      if (cand[i] % p.G == 0 && (size_t)cand[i] * p.E <= 28 * 1024) TE = cand[i];
    if (!TE && p.G <= 8 && (size_t)8 * p.E <= 48 * 1024) TE = 8;
  }
  const int W = p.G > 8 ? p.G : 8;
  const size_t smem_tile = (size_t)(W + p.G) * p.E + (size_t)W * (REC_SNAKE0 + 2 * S + (F + 1) / 2 + 3 + p.bm_words) * 4;
  // rows kernel: chunks of R image rows must be 16-byte multiples (TMA) and fit a ~24 KB buffer
  int R = 0;
  if (p.E % 16 == 0 && !grid) {
    const int unit = 16 / gcd(V * p.C, 16);
    // chunk size and CTA shape measured on B200 at 16 snakes on 64x64: 4 warps (1 producer + 3 consumers) give 7 CTAs
    // per SM, and 8 KB chunks beat 12 KB (32 768 envs: classic 1280 us, cut 1502 vs 1551 us)
    const size_t lim = 8 * 1024;
    for (int r = unit; r <= V && ((size_t)r * V * p.C <= lim || !R); r += unit) { if ((size_t)r * V * p.C > 48 * 1024) break; R = r; }
  }
  int form = TE ? FORM_LANE : smem_tile <= 110 * 1024 ? FORM_TILE : R ? FORM_ROWS : FORM_DENSE;
  // grid: every ring-family geometry goes to the rows kernel's grid form (the producer's code grid IS the observation)
  if (grid && form != FORM_LANE) form = FORM_ROWS;
  if (force == "dense") form = FORM_DENSE;
  if (force == "rows") {
    if (!R && !grid) return fail(SNK_EINVAL, "rows kernel does not support this configuration");
    form = FORM_ROWS;
  }
  if (force == "tile" && smem_tile <= 200 * 1024) form = FORM_TILE;
  if (force == "lane" && !TE) return fail(SNK_EINVAL, "lane kernel does not support this configuration");
  p.family = form == FORM_LANE;
  if (form == FORM_LANE) {
    // lane path forms (lane=fused|ws|split): every warp steps 32 envs then streams their images (default: fastest
    // measured), warp-specialised single kernel, or two kernels
    std::string lv;
    const bool have_lv = dbg_get(dbg, "lane", &lv);
    // measured on B200: with a small image per env (3 views of 12x12: 1296 B) the step is bound by the
    // logic's latency and the warp-specialised form (more logic warps per image buffer) is 1.4x faster;
    // with 2646 B per env (2 views of 21x21) the image stream dominates and the fused form wins
    // ... unless there are too few 32-env batches to give every SM a few (4 096 envs of 2x10x10: one
    // batch per SM at most): then a warp that steps AND paints its batch has the shortest critical path
    // (13.8 us vs 19.0 us per step)
    // Since the respawns became warp-cooperative function calls the register-capped warp-specialised kernel pays for
    // them in spills, and for S >= 2 the two-kernel form (logic at full occupancy, then the observation writer) is the
    // fastest small-image form (65 536 envs, 10x10: 3 snakes cut 53.0 vs 61.3 us, 3 snakes classic 44.0 vs 48.8,
    // 2 snakes 34.6 vs 38.8; 1 M envs cut 648 vs 751 us); a single snake stays warp-specialised (23.6 vs 29.2 us).
    const bool small_image = p.E < 2048 && (N + 31) / 32 >= 2LL * h->n_sm;
    if (grid) form = FORM_LANE_GRID;
    else if (have_lv ? lv == "ws" : (small_image && S == 1)) form = FORM_LANE_WS;
    else if (have_lv ? lv == "split" : (small_image && S > 1)) form = FORM_LANE_SPLIT;
    p.RW = (REC_SNAKE0 + 2 * S + 2 + 3) & ~3;
    p.W = 32;
    int te = TE, epw = 32;
    if (form == FORM_LANE) {
      // Small shards.  A warp's pass (logic of its batch, then one image after the other) is a serial chain, and a lane
      // per env keeps 32 envs on it; when the shard has fewer 32-env batches than the GPU holds warps (4 096 envs of
      // 2x10x10 = 128 warps on 148 SMs: 14 us per step, all of it one warp's latency) the batch shrinks to 16 / 8 / 4 envs
      // -- the idle lanes cost issue slots nobody wants, the chain gets shorter (one image, painted by 32/epw lanes per
      // env) -- as long as every batch still finds a resident warp.  epw=<n> overrides.
      const int forced = dbg_int(dbg, "epw", 0);
      for (int cand = 16; cand >= 4; cand >>= 1) {
        if (cand % p.G != 0 || (forced && cand < forced)) break;
        CUDA_TRY(plan_lane(plan, form, cand < TE ? cand : TE, cand, 32));
        if (!forced && (N + cand - 1) / cand > (long long)plan.max_grid * 2) break;  // more batches than resident warps (2 per CTA)
        te = p.TE; epw = cand;
      }
    }
    CUDA_TRY(plan_lane(plan, form, te, epw, form == FORM_LANE_GRID ? 64 : 32));
  } else {
    if (form == FORM_TILE) {
      p.W = W; plan.block = 32 * W; plan.smem = smem_tile;
    } else if (form == FORM_ROWS) {
      if (grid) form = FORM_ROWS_GRID;
      p.W = 1; p.R = R; plan.block = 128;  // 1 producer warp + 3 consumer warps
      p.tile_stride = (int)(((size_t)R * V * p.C + 127) & ~(size_t)127);  // grid: R = 0, no chunk buffers
      plan.smem = 2 * (((size_t)p.VV + 127) & ~(size_t)127) + 2 * (size_t)p.tile_stride + (size_t)(p.RW + p.bm_words) * 4;
    } else {
      p.W = 1; plan.block = 256; plan.smem = align16((size_t)p.VV) + (size_t)(p.RW + p.bm_words) * 4;
      if (plan.smem > 200 * 1024) return fail(SNK_EINVAL, "board too large for shared memory");
    }
    p.n_groups = (N + p.W - 1) / p.W;
    plan.form = form;
    plan.envs_per_cta = p.W;
    CUDA_TRY(finish(plan));
  }
  // Regime-adaptive lane path: `plan` the fused kernel, `plan_alt` the two-kernel form (k_lane_logic + k_lane_paint2).  The
  // fused kernel's warps are serial chains (logic of a batch, then its images, ten warps per SM); the two kernels run the
  // logic at full occupancy in one wave and pay for a second launch.  Two pairs of thresholds in body cells per env, with
  // hysteresis, pick between them (launch()):
  //  * alt_hi / alt_lo: a step that stores whole images, or an eager step.  With short bodies the fused kernel wins
  //    (2x19x19, 131 072 envs, random actions: 64.5 us against 73.3 us for the two-kernel form with whole images); with
  //    long bodies its warps fall behind.  Measured on one box, body cells per env 5.8 / 8.6 / 12.8 / 22.2 (fruit-seeking
  //    policy with 70 / 40 / 20 / 5 % random actions): fused 72.6 / 83.0 / 92.4 / 109.9 us, two kernels 75.9 / 79.8 /
  //    85.6 / 93.4 us; 8 cells at 2646 bytes of image per env, scaled with the image.  Eager steps keep these thresholds
  //    even when they store sectors: a second launch per step costs an eager loop with per-step copies more than the
  //    two-kernel form saves (bench.py e2e_obs_resident, 131 072 envs: 4.09e9 against 4.54e9 agent-steps/s, §4.20).
  //  * sec_hi / sec_lo: a classic step recorded into a graph that stores sectors into the own buffer (native
  //    observations).  Both forms then store sectors.  Measured on B200 (2x19x19, same states and actions; body cells
  //    4.3 random, then 5.0 / 6.0 / 7.6 / 11.2 fruit-seeking as above), two kernels / fused:
  //      131 072 envs: 0.93 / 0.80 / 0.74 / 0.70 / 0.77     1 M envs: 0.96 / 0.79 / 0.68 / 0.70 / 0.83
  //       32 768 envs: 1.04 / 0.96 / 0.92 / 0.90 / 0.95
  //    So once the fused kernel's warps must step more than one batch each, the two-kernel form wins at every body
  //    length (sec_hi = 0); with one batch per warp the forms cross near 5 body cells per env, scaled with the image.
  // The host cannot know the regime without the statistics, so the first CTA of every step posts the running sums into
  // mapped host memory (peer_push) and regime_update() reads them -- no synchronisation, a step or two late, which is
  // early enough for a quantity that moves over hundreds of steps.  Results are bit-identical either way.  adaptive=0
  // turns it off; alt_hi=<n> sets both thresholds.
  std::string lv;
  if (form == FORM_LANE && p.EPW == 32 && !dbg_get(dbg, "lane", &lv) && dbg_int(dbg, "adaptive", 1) != 0) {
    const bool one_round = (N + 31) / 32 <= (long long)plan.max_grid * 2;  // every 32-env batch finds a resident warp
    // the alternative steps the same 32-env batches: p's lane geometry stays as it is
    h->have_alt = plan_lane(h->plan_alt, FORM_LANE_SPLIT, p.TE, 32, 64) == cudaSuccess;
    cudaGetLastError();
    const int hi = dbg_int(dbg, "alt_hi", 0);
    h->alt_hi = hi > 0 ? (double)hi : 8.0 * (double)p.E / 2646.0;
    h->sec_hi = hi > 0 ? (double)hi : one_round ? 5.0 * (double)p.E / 2646.0 : 0.0;
    h->alt_lo = 0.75 * h->alt_hi;
    h->sec_lo = 0.75 * h->sec_hi;
    // the forms for a fresh reset: every snake one cell long
    h->use_alt = (double)S > h->alt_hi;
    h->use_alt_sec = (double)S > h->sec_hi;
  }
  return SNK_OK;
}

static int cfg_check(const snk_config* c) {
  if (!c) return fail(SNK_EINVAL, "config is NULL");
  if (c->size < 2 || c->size > 254) return fail(SNK_EINVAL, "size must be 2..254, got %d", c->size);
  if (c->n_snakes < 1 || c->n_snakes > 32) return fail(SNK_EINVAL, "n_snakes must be 1..32, got %d", c->n_snakes);
  if (c->n_fruits < 0 || c->n_fruits > 32) return fail(SNK_EINVAL, "n_fruits must be 0..32, got %d", c->n_fruits);
  if (c->n_views < 0 || c->n_views > 32) return fail(SNK_EINVAL, "n_views must be 0..32, got %d", c->n_views);
  if (c->rules < 0 || c->rules > 2) return fail(SNK_EINVAL, "unknown rules %d", c->rules);
  if (c->num_envs < 1) return fail(SNK_EINVAL, "num_envs must be >= 1");
  if (c->max_steps < 0 || c->max_steps > 65535) return fail(SNK_EINVAL, "max_steps must be 0..65535");
  if (c->obs_mode != SNK_OBS_NATIVE && c->obs_mode != SNK_OBS_ATARI84 && c->obs_mode != SNK_OBS_GRID)
    return fail(SNK_EINVAL, "unknown obs_mode %d", c->obs_mode);
  if (c->obs_mode == SNK_OBS_ATARI84 && 84 % (c->size + 2) != 0)
    return fail(SNK_EINVAL, "obs_mode atari84 needs 84 %% (size + 2) == 0 (exact pixel replication); size=%d", c->size);
  if (c->obs_mode == SNK_OBS_ATARI84 && (c->n_views ? c->n_views : c->n_snakes) > 8)
    return fail(SNK_EINVAL, "obs_mode atari84 supports at most 8 views");
  if (c->rng_mode != SNK_RNG_PHILOX && c->rng_mode != SNK_RNG_TAPE) return fail(SNK_EINVAL, "unknown rng_mode %d", c->rng_mode);
  if (c->env_id_base < 0) return fail(SNK_EINVAL, "env_id_base must be >= 0");
  if ((uint64_t)c->env_id_base + (uint64_t)c->num_envs > 0xffffffffull) return fail(SNK_EINVAL, "global env ids must fit 32 bits");
  return SNK_OK;
}

extern "C" int snk_version(void) { return SNK_VERSION; }
extern "C" const char* snk_last_error(void) { return g_err; }

extern "C" int snk_state_layout_of(const snk_config* c, snk_state_layout* o) {
  int rc = cfg_check(c);
  if (rc) return rc;
  if (!o) return fail(SNK_EINVAL, "layout is NULL");
  const size_t N = (size_t)c->num_envs, S = (size_t)c->n_snakes, F = (size_t)c->n_fruits, D = (size_t)c->size, V = D + 2;
  const int cap = (int)((D * D + 1 + 7) & ~(size_t)7);
  size_t off = 0;
  o->off_t = off;        off = align16(off + 4 * N);
  o->off_spare = off;    off = align16(off + 4 * N);
  o->off_draw_ctr = off; off = align16(off + 4 * N);
  o->off_ep_ret = off;   off = align16(off + 4 * N);
  o->off_ep_len = off;   off = align16(off + 4 * N);
  o->off_len = off;      off = align16(off + 2 * N * S);
  o->off_grow_to = off;  off = align16(off + 2 * N * S);
  o->off_vel = off;      off = align16(off + N * S);
  o->off_body = off;     off = align16(off + 2 * N * S * (size_t)cap);
  o->off_fruit = off;
  o->fruit_is_grid = c->rules != SNK_RULES_CLASSIC;
  off = align16(off + (o->fruit_is_grid ? N * V * V : 2 * N * F));
  o->total_bytes = off;
  o->cap = cap;
  return SNK_OK;
}

template <typename T>
static int dev_alloc(snk_handle* h, T** out, size_t count, bool zero) {
  void* ptr = nullptr;
  const size_t bytes = align16(count * sizeof(T) + 16);
  cudaError_t e = cudaMalloc(&ptr, bytes);
  if (e != cudaSuccess) return fail(SNK_ENOMEM, "cudaMalloc(%zu bytes): %s", bytes, cudaGetErrorString(e));
  h->allocs.push_back(ptr);
  if (zero) CUDA_TRY(cudaMemset(ptr, 0, bytes));
  *out = (T*)ptr;
  return SNK_OK;
}

static void dev_free(snk_handle* h, void* ptr) {
  if (!ptr) return;
  auto it = std::find(h->allocs.begin(), h->allocs.end(), ptr);
  if (it != h->allocs.end()) h->allocs.erase(it);
  cudaFree(ptr);
}

// ------------------------------------------------------------------ NCCL binding
static NcclApi g_nccl = {};
static int nccl_load() {
  if (g_nccl.so) return SNK_OK;
  void* so = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
  if (!so) so = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
  if (!so) return fail(SNK_ECOMM, "libnccl.so.2 not found: %s", dlerror());
  NcclApi a = {};
  a.so = so;
  *(void**)&a.GetUniqueId = dlsym(so, "ncclGetUniqueId");
  *(void**)&a.CommInitRank = dlsym(so, "ncclCommInitRank");
  *(void**)&a.CommInitRankConfig = dlsym(so, "ncclCommInitRankConfig");
  *(void**)&a.CommDestroy = dlsym(so, "ncclCommDestroy");
  *(void**)&a.AllReduce = dlsym(so, "ncclAllReduce");
  *(void**)&a.GetErrorString = dlsym(so, "ncclGetErrorString");
  *(void**)&a.GetVersion = dlsym(so, "ncclGetVersion");
  if (!a.GetUniqueId || !a.CommInitRank || !a.CommDestroy || !a.AllReduce || !a.GetErrorString)
    return fail(SNK_ECOMM, "libnccl.so.2 lacks a required symbol");
  g_nccl = a;
  return SNK_OK;
}
#define NCCL_TRY(expr)                                                                            \
  do {                                                                                            \
    int _r = (expr);                                                                              \
    if (_r != 0) return fail(SNK_ECOMM, "%s: %s", #expr, g_nccl.GetErrorString(_r));             \
  } while (0)

struct snk_graph {
  snk_handle* h;
  cudaGraph_t graph;
  cudaGraphExec_t exec;
  int T;
  uint64_t launches_per_run, collectives_per_run;
  // arguments it was captured with (snk_rollout's cache key)
  const int8_t* d_actions; int32_t n_batches; uint8_t* d_obs; float* d_reward; uint8_t* d_done; uint32_t flags;
  uint8_t* obs_target; bool with_comm, with_push;
  const uint8_t* last_native_obs;  // where the graph's last step leaves the native observations
  double* d_slots;  // with a communicator: [T] snapshot slots + [T] all-reduced slots, one pair per step (no reuse inside a launch)
};

extern "C" int snk_graph_destroy(snk_graph* g) {
  if (!g) return SNK_OK;
  if (g->h && g->h->rollout_cache == g) g->h->rollout_cache = nullptr;
  if (g->exec) cudaGraphExecDestroy(g->exec);
  if (g->graph) cudaGraphDestroy(g->graph);
  if (g->h && g->h->d_global_last >= g->d_slots && g->d_slots && g->h->d_global_last < g->d_slots + 2 * (size_t)g->T * SNK_NSTATS)
    g->h->d_global_last = nullptr;
  if (g->d_slots) cudaFree(g->d_slots);
  delete g;
  return SNK_OK;
}

extern "C" int snk_destroy(snk_handle* h) {
  if (!h) return SNK_OK;
  cudaSetDevice(h->cfg.device);
  cudaDeviceSynchronize();
  if (h->rollout_cache) snk_graph_destroy(h->rollout_cache);
  if (h->comm && g_nccl.so) g_nccl.CommDestroy(h->comm);
  for (int i = 0; i < SNK_MAX_PEERS; ++i)
    if (h->peer_mapped[i]) cudaIpcCloseMemHandle(h->peer_mapped[i]);
  for (int i = 0; i < 2; ++i) {
    if (h->ev_step[i]) cudaEventDestroy(h->ev_step[i]);
    if (h->ev_red[i]) cudaEventDestroy(h->ev_red[i]);
    if (h->cev_step[i]) cudaEventDestroy(h->cev_step[i]);
    if (h->cev_red[i]) cudaEventDestroy(h->cev_red[i]);
  }
  for (int i = 0; i < SNK_SCALAR_SLOTS; ++i) {
    if (h->sc[i].ev_in) cudaEventDestroy(h->sc[i].ev_in);
    if (h->sc[i].ev_k) cudaEventDestroy(h->sc[i].ev_k);
    if (h->sc[i].ev_out) cudaEventDestroy(h->sc[i].ev_out);
  }
  if (h->s_in) cudaStreamDestroy(h->s_in);
  if (h->s_out) cudaStreamDestroy(h->s_out);
  if (h->side) cudaStreamDestroy(h->side);
  if (h->cap_stream) cudaStreamDestroy(h->cap_stream);
  for (void* q : h->allocs) cudaFree(q);
  for (auto& q : h->host_allocs) cudaFreeHost(q.first);
  delete h;
  return SNK_OK;
}

#define TRY(expr) do { int _rc = (expr); if (_rc) { snk_destroy(h); return _rc; } } while (0)
#define CUDA_TRY_H(expr)                                                                        \
  do {                                                                                          \
    cudaError_t _e = (expr);                                                                    \
    if (_e != cudaSuccess) { snk_destroy(h); return fail(SNK_ECUDA, "%s: %s", #expr, cudaGetErrorString(_e)); } \
  } while (0)

extern "C" int snk_create_ex(const snk_config* cfg, const char* debug_opts, snk_handle** out) {
  int rc = cfg_check(cfg);
  if (rc) return rc;
  if ((rc = dbg_check(debug_opts ? debug_opts : ""))) return rc;
  const bool grid = cfg->obs_mode == SNK_OBS_GRID;
  if (grid && (rc = dbg_check_grid(debug_opts ? debug_opts : ""))) return rc;
  if (!out) return fail(SNK_EINVAL, "out is NULL");
  int n_dev = 0;
  CUDA_TRY(cudaGetDeviceCount(&n_dev));
  if (cfg->device < 0 || cfg->device >= n_dev) return fail(SNK_EINVAL, "device %d of %d", cfg->device, n_dev);
  CUDA_TRY(cudaSetDevice(cfg->device));
  snk_handle* h = new snk_handle();
  h->cfg = *cfg;
  if (h->cfg.n_views == 0) h->cfg.n_views = cfg->n_snakes;
  if (h->cfg.max_steps == 0) h->cfg.max_steps = 2000;
  h->launches = 0;
  h->d_main_target = nullptr;
  h->obs_current = nullptr; h->have_alt = false; h->use_alt = h->use_alt_sec = false; h->h_regime = nullptr; h->reg_steps0 = h->reg_cells0 = 0.0;
  h->d_obs_own = nullptr; h->d_actions_own = nullptr; h->d_blob = nullptr; h->blob_bytes = 0; h->d_views = nullptr; h->views_bytes = 0;
  h->d_tape_vals = h->d_tape_bounds = nullptr; h->d_tape_off = nullptr;
  h->comm = nullptr; h->comm_ranks = 1; h->comm_rank = 0; h->side = nullptr; h->cap_stream = nullptr;
  h->d_snap = h->d_global = nullptr; h->step_seq = 0; h->collectives = 0; h->last_slot = 0; h->rollout_cache = nullptr;
  h->d_global_last = nullptr;
  h->d_inbox = nullptr; memset(&h->peer, 0, sizeof(h->peer)); h->reduce_enabled = true;
  for (int i = 0; i < SNK_MAX_PEERS; ++i) h->peer_mapped[i] = nullptr;
  for (int i = 0; i < 2; ++i) { h->ev_step[i] = h->ev_red[i] = h->cev_step[i] = h->cev_red[i] = nullptr; h->ev_red_valid[i] = false; }
  h->debug = debug_opts ? debug_opts : "";
  const std::string& dbg = h->debug;
  snk_state_layout_of(&h->cfg, &h->lay);
  cudaDeviceProp prop;
  CUDA_TRY_H(cudaGetDeviceProperties(&prop, cfg->device));
  h->n_sm = prop.multiProcessorCount;

  Params& p = h->p;
  memset(&p, 0, sizeof(p));
  const int D = cfg->size, V = D + 2, S = cfg->n_snakes, F = cfg->n_fruits, K = h->cfg.n_views;
  const long long N = cfg->num_envs;
  p.D = D; p.V = V; p.VV = V * V; p.S = S; p.F = F; p.K = K; p.C = grid ? 1 : 3 * K;  // grid: one code byte per cell
  p.cap = h->lay.cap;
  p.CW = (p.cap - 1 + 15) / 16;
  p.RW = (REC_SNAKE0 + 2 * S + (F + 1) / 2 + 3) & ~3;
  p.E = p.VV * p.C;
  p.G = 16 / gcd(p.E, 16);
  p.grid_stride = (int)align16((size_t)p.VV);
  p.bm_words = (D * D + 31) / 32;
  p.magicV = 65536u / (uint32_t)V + 1u; p.magicD = 65536u / (uint32_t)D + 1u;
  p.max_steps = h->cfg.max_steps; p.auto_reset = cfg->auto_reset != 0; p.rng_mode = cfg->rng_mode;
  p.N = N; p.env_id_base = cfg->env_id_base; p.seed = cfg->seed;

  TRY(plan_launch(h));
  if (h->have_alt) {  // regime_update() reads the running sums the step kernels post here (Params::regime_out)
    h->have_alt = false;
    void* hp = nullptr;
    if (cudaHostAlloc(&hp, 2 * sizeof(double), cudaHostAllocMapped) == cudaSuccess) {
      void* dp = nullptr;
      if (cudaHostGetDevicePointer(&dp, hp, 0) == cudaSuccess) {
        h->h_regime = (double*)hp; h->h_regime[0] = h->h_regime[1] = 0.0;
        h->host_allocs.push_back(std::make_pair(hp, 2 * sizeof(double)));
        p.regime_out = (double*)dp;
        h->have_alt = true;
      } else cudaFreeHost(hp);
    }
    cudaGetLastError();
  }

  // device buffers
  TRY(dev_alloc(h, &p.rec, (size_t)N * p.RW, true));
  if (p.family == 1) TRY(dev_alloc(h, &p.chain, (size_t)N * S * p.CW, true));
  else TRY(dev_alloc(h, &p.body, (size_t)N * S * p.cap, true));
  if (cfg->rules != SNK_RULES_CLASSIC) TRY(dev_alloc(h, &p.grid, (size_t)N * p.grid_stride, true));
  p.GBW = (p.VV + 31) / 32;
  if (cfg->rules != SNK_RULES_CLASSIC && p.family == 1) TRY(dev_alloc(h, &p.gbits, (size_t)N * p.GBW, true));
  TRY(dev_alloc(h, &h->d_obs_own, (size_t)N * p.E, true));
  p.obs = h->d_obs_own;
  if (p.family == 1) {
    // frame_ok[e] = 1 <=> d_obs_own holds exactly the image of env e's record (cleared here and by every restore / copy, written
    // by every lane-family kernel that writes a record).  With it the lane path's classic step (fused kernel and two-kernel
    // form) stores only the sectors a step changes; delta=0 always stores whole images.  Sectors never cross env boundaries because the first and last
    // (V+1)*C bytes of an env image are border (needs >= 32) and the buffer is 32-byte aligned.  Default: 32-env batches
    // only.  A small shard (smaller batches, §4.10 of DESIGN.md) is bound by one warp's serial chain, not by the stream,
    // and there the sector loop is longer than one bulk-store issue (2x10x10, 4 096 envs on B200: 10.39 vs 9.86 us per
    // step); the headline shard gains 64.5 -> 52.7 us.  delta=0 / delta=1 turn it off / on regardless.
    const int dm = dbg_int(dbg, "delta", -1);
    // Default: 32-env batches of the fused kernel and its adaptive pair.  The small-image two-kernel form (§4.8) keeps whole
    // images: there the sector store is slower (3x10x10 classic, 65 536 envs on B200: 45.8 us per step with sectors, 41.9 us whole).
    p.delta = !grid && cfg->rules == SNK_RULES_CLASSIC && (V + 1) * p.C >= 32 && ((uintptr_t)h->d_obs_own & 31) == 0 &&
              (dm < 0 ? p.EPW == 32 && h->plan.form != FORM_LANE_SPLIT : dm != 0);
  }
  h->d_obs84_own = nullptr;
  h->obs_out_env_bytes = (size_t)p.E;
  h->d_obs_user = h->d_obs_own;
  if (cfg->obs_mode == SNK_OBS_ATARI84) {
    h->obs_out_env_bytes = (size_t)84 * 84 * p.C;
    TRY(dev_alloc(h, &h->d_obs84_own, (size_t)N * h->obs_out_env_bytes, true));
    h->d_obs_user = h->d_obs84_own;
  }
  TRY(dev_alloc(h, &p.reward, (size_t)N, true));
  TRY(dev_alloc(h, &p.reward_all, (size_t)N * S, true));
  {  // done | num_alive | episode return | episode length in ONE block: a caller that must keep a step's infos past the
     // next step snapshots them with a single copy
    const size_t nb = align16((size_t)N);
    h->info_bytes = 2 * nb + 2 * align16(4 * (size_t)N);
    TRY(dev_alloc(h, &h->d_info, h->info_bytes, true));
    p.done = h->d_info; p.num_alive = h->d_info + nb;
    p.fin_ret = reinterpret_cast<float*>(h->d_info + 2 * nb);
    p.fin_len = reinterpret_cast<int32_t*>(h->d_info + 2 * nb + align16(4 * (size_t)N));
  }
  TRY(dev_alloc(h, &p.stats, (size_t)SNK_NSTATS, true));
  TRY(dev_alloc(h, &p.err, (size_t)1, true));
  TRY(dev_alloc(h, &p.ticket, (size_t)1, true));
  TRY(dev_alloc(h, &h->d_actions_own, (size_t)N * S, true));
  if (p.family == 1) {
    // frame_ok, and the two-kernel form's writer learns the old state from k_lane_logic: DeltaPrev entries (8 words per env
    // for S <= 2, 12 for S <= 4) from the first 256-byte boundary past the flags (delta_prev() in snk_lane.cuh).  Allocated
    // whenever p.delta is set, whatever the form: a launch's Params::delta never exceeds the handle's, so every launch that
    // may write or read the entries finds them.  Last of the per-env buffers, so that the entries move no other buffer.
    TRY(dev_alloc(h, &p.frame_ok, p.delta ? (size_t)((N + 255) & ~255LL) + (size_t)N * 4 * ((2 * S + 6) & ~3) : (size_t)N, true));
  }

  // lookup tables: padded id -> (outside?, y-major board index incl. the reference's aliasing), and back
  std::vector<uint32_t> cellinfo((size_t)p.VV);
  std::vector<uint16_t> idx2pid((size_t)D * D);
  for (int px = 0; px < V; ++px)
    for (int py = 0; py < V; ++py) {
      const int x = px - 1, y = py - 1;
      const bool outside = x < 0 || x >= D || y < 0 || y >= D;
      const long idx = (long)y * D + x;  // snake_multiple_test.py:209, not bounds-checked
      uint32_t v = (idx >= 0 && idx < (long)D * D) ? (uint32_t)idx : 0x7fffffffu;
      if (outside) v |= 0x80000000u;
      cellinfo[(size_t)px * V + py] = v;
      if (!outside) idx2pid[(size_t)idx] = (uint16_t)(px * V + py);
    }
  uint32_t* d_cellinfo; uint16_t* d_idx2pid; uint8_t* d_tmpl;
  TRY(dev_alloc(h, &d_cellinfo, cellinfo.size(), false));
  TRY(dev_alloc(h, &d_idx2pid, idx2pid.size(), false));
  CUDA_TRY_H(cudaMemcpy(d_cellinfo, cellinfo.data(), cellinfo.size() * 4, cudaMemcpyHostToDevice));
  CUDA_TRY_H(cudaMemcpy(d_idx2pid, idx2pid.data(), idx2pid.size() * 2, cudaMemcpyHostToDevice));
  p.cellinfo = d_cellinfo; p.idx2pid = d_idx2pid;
  // border-only observation of one 16-byte-aligned group of G envs (snake_multiple_test.py:52-56)
  std::vector<uint8_t> tmpl((size_t)p.G * p.E, 0);
  for (int g = 0; g < p.G; ++g)
    for (int i = 0; i < V; ++i) {
      const int ring_cells[4] = {i, (V - 1) * V + i, i * V, i * V + V - 1};
      for (int q = 0; q < 4; ++q) memset(&tmpl[(size_t)g * p.E + (size_t)ring_cells[q] * p.C], 255, (size_t)p.C);
    }
  TRY(dev_alloc(h, &d_tmpl, tmpl.size(), false));
  CUDA_TRY_H(cudaMemcpy(d_tmpl, tmpl.data(), tmpl.size(), cudaMemcpyHostToDevice));
  p.tmpl = d_tmpl;
  CUDA_TRY_H(cudaStreamCreateWithFlags(&h->cap_stream, cudaStreamNonBlocking));
  CUDA_TRY_H(cudaDeviceSynchronize());
  *out = h;
  return SNK_OK;
}

extern "C" int snk_create(const snk_config* cfg, snk_handle** out) { return snk_create_ex(cfg, getenv("SNK_DEBUG"), out); }

extern "C" int snk_get_config(const snk_handle* h, snk_config* out) {
  if (!h || !out) return fail(SNK_EINVAL, "NULL argument");
  *out = h->cfg;
  return SNK_OK;
}

extern "C" int snk_get_buffers(const snk_handle* h, snk_buffers* out) {
  if (!h || !out) return fail(SNK_EINVAL, "NULL argument");
  const Params& p = h->p;
  out->d_obs = h->d_obs_user; out->d_reward = p.reward; out->d_reward_all = p.reward_all; out->d_done = p.done;
  out->d_num_alive = p.num_alive; out->d_episode_return = p.fin_ret; out->d_episode_len = p.fin_len;
  const int side = h->cfg.obs_mode == SNK_OBS_ATARI84 ? 84 : p.V;
  out->d_info_block = h->d_info; out->info_block_bytes = h->info_bytes;
  out->d_stats = p.stats; out->obs_bytes = (size_t)p.N * h->obs_out_env_bytes; out->obs_h = side; out->obs_w = side; out->obs_c = p.C;
  return SNK_OK;
}

struct RolloutSlot {  // per-step output redirection (rollout graphs, snk_step_scalars_async); NULL = the handle's own buffer
  uint8_t* obs = nullptr;
  float* reward = nullptr;
  uint8_t* done = nullptr;
  uint8_t* alive = nullptr;
  float* fin_ret = nullptr;
  int32_t* fin_len = nullptr;
};

// One step (or reset / re-encode) on `stream`.  `capturing`: the call is being recorded into a CUDA graph (snk_graph_create);
// the per-step statistics all-reduce then forks onto the side stream with capture-time events.
struct CaptureCtx {  // a step being recorded into a CUDA graph
  int step;
  double* slots;     // the graph's own [T] snapshot + [T] result slots (NULL without a communicator)
  int T;
};

// Fused or two-kernel form for the next launch (see snk_create_ex): mean body cells per env over the steps since the last
// decision, from the sums the step kernels post into mapped host memory.
static void regime_update(snk_handle* h) {
  if (!h->have_alt) return;
  const double steps = ((volatile double*)h->h_regime)[0], cells = ((volatile double*)h->h_regime)[1];
  if (steps < h->reg_steps0 || cells < h->reg_cells0) { h->reg_steps0 = steps; h->reg_cells0 = cells; return; }  // statistics were reset
  if (steps - h->reg_steps0 < (double)h->p.N) return;  // less than one whole step of news
  const double mean = (cells - h->reg_cells0) / (steps - h->reg_steps0);
  h->reg_steps0 = steps; h->reg_cells0 = cells;
  if (mean > h->alt_hi) h->use_alt = true;
  else if (mean < h->alt_lo) h->use_alt = false;
  if (mean > h->sec_hi) h->use_alt_sec = true;
  else if (mean < h->sec_lo) h->use_alt_sec = false;
}

static int launch(snk_handle* h, int mode, const int8_t* d_actions, const uint8_t* d_mask, cudaStream_t stream,
                  const RolloutSlot* slot = nullptr, const CaptureCtx* cap = nullptr) {
  const bool capturing = cap != nullptr;
  CUDA_TRY(cudaSetDevice(h->cfg.device));
  Params p = h->p;
  uint8_t* obs_user = h->d_obs_user;
  if (slot) {
    if (slot->reward) p.reward = slot->reward;
    if (slot->done) p.done = slot->done;
    if (slot->alive) p.num_alive = slot->alive;
    if (slot->fin_ret) p.fin_ret = slot->fin_ret;
    if (slot->fin_len) p.fin_len = slot->fin_len;
    if (slot->obs) {
      obs_user = slot->obs;
      if (h->cfg.obs_mode != SNK_OBS_ATARI84) p.obs = slot->obs;
    }
  }
  p.mode = mode; p.actions = d_actions; p.mask = d_mask;
  // the step kernels write every env's image into p.obs (frame_ok is about RGB images: a grid handle never has one)
  p.frame_own = p.obs == h->d_obs_own && h->cfg.obs_mode != SNK_OBS_GRID;
  p.delta = p.delta && p.frame_own && mode == MODE_STEP;
  p.tape_vals = h->d_tape_vals; p.tape_bounds = h->d_tape_bounds; p.tape_off = h->d_tape_off;
  if (p.rng_mode == SNK_RNG_TAPE && !p.tape_vals) return fail(SNK_EINVAL, "rng_mode is TAPE but no tape was set");
  const bool reduce = h->comm && h->reduce_enabled && mode == MODE_STEP;   // NCCL form: snapshot + all-reduce on the side stream
  const bool push = h->peer.ranks > 0 && h->reduce_enabled && mode == MODE_STEP;  // peer form: the step kernel's first CTA pushes
  if (push) p.peer = h->peer;
  int sl = 0;
  double* snap = nullptr;
  double* glob = nullptr;
  if (reduce) {
    if (capturing) {
      // inside a graph every step has its own pair of slots: nothing is reused within a launch, so a step kernel depends
      // on its predecessor alone (the programmatic edge) and the all-reduces form an independent side branch
      snap = cap->slots + (size_t)cap->step * SNK_NSTATS;
      glob = cap->slots + (size_t)(cap->T + cap->step) * SNK_NSTATS;
    } else {
      sl = (int)(h->step_seq & 1);
      snap = h->d_snap + sl * SNK_NSTATS;
      glob = h->d_global + sl * SNK_NSTATS;
      // the all-reduce that last read this snapshot slot (two steps ago) must be done before the kernel rewrites it
      if (h->ev_red_valid[sl]) CUDA_TRY(cudaStreamWaitEvent(stream, h->ev_red[sl], 0));
    }
  }
  p.snap = snap;
  if (mode == MODE_STEP) regime_update(h);
  // a graph-captured classic step that stores sectors into the own buffer follows sec_hi / sec_lo (plan_launch)
  const bool sectors = capturing && p.delta && h->cfg.obs_mode == SNK_OBS_NATIVE;
  const bool alt = h->have_alt && (sectors ? h->use_alt_sec : h->use_alt);
  const LaunchPlan& plan = alt ? h->plan_alt : h->plan;
  p.restore_thr = plan.restore_thr;
  CUDA_TRY(snk_launch_step(p, plan, stream));
  if (!capturing) h->obs_current = p.obs;
  h->launches += (plan.logic && mode != MODE_OBSERVE) ? 2 : 1;
  if (reduce) {
    // side stream: all-reduce this step's snapshot while the next step runs; its result is read one step late
    cudaEvent_t es = capturing ? h->cev_step[0] : h->ev_step[sl], er = capturing ? h->cev_red[0] : h->ev_red[sl];
    CUDA_TRY(cudaEventRecord(es, stream));
    CUDA_TRY(cudaStreamWaitEvent(h->side, es, 0));
    NCCL_TRY(g_nccl.AllReduce(snap, glob, SNK_NSTATS, kNcclFloat64, kNcclSum, h->comm, h->side));
    CUDA_TRY(cudaEventRecord(er, h->side));
    if (!capturing) { h->ev_red_valid[sl] = true; h->step_seq++; h->collectives++; h->last_slot = sl; h->d_global_last = glob; }
  }
  if (push && !capturing) h->collectives++;
  if (h->cfg.obs_mode == SNK_OBS_ATARI84) {
    CUDA_TRY(snk_launch_upscale84(p.obs, obs_user, p.N, p.V, p.C, h->n_sm, stream));
    h->launches++;
  }
  if (h->d_main_target && !capturing) {  // the main snake's view alone, packed, for the learner's rollout slot
    const size_t px = (size_t)p.N * (h->obs_out_env_bytes / (size_t)p.C);
    CUDA_TRY(snk_launch_extract_views(obs_user, h->d_main_target, (long long)px, p.C, 1, stream));
    h->launches++;
  }
  return SNK_OK;
}

// before work that is not ordered behind the side stream by events of its own (graph launches, stats read-back)
static int join_side(snk_handle* h, cudaStream_t stream) {
  for (int i = 0; i < 2; ++i)
    if (h->ev_red_valid[i]) CUDA_TRY(cudaStreamWaitEvent(stream, h->ev_red[i], 0));
  return SNK_OK;
}

extern "C" int snk_reset(snk_handle* h, const uint8_t* d_mask, void* stream) {
  if (!h) return fail(SNK_EINVAL, "handle is NULL");
  return launch(h, MODE_RESET, nullptr, d_mask, (cudaStream_t)stream);
}

extern "C" int snk_step(snk_handle* h, const int8_t* d_actions, void* stream) {
  if (!h || !d_actions) return fail(SNK_EINVAL, "NULL argument");
  return launch(h, MODE_STEP, d_actions, nullptr, (cudaStream_t)stream);
}

// ------------------------------------------------------------------ CUDA graphs: T steps, one launch
struct ScriptedArgs { uint64_t step0, seed; int eps_permille; };

static int graph_create_impl(snk_handle* h, const int8_t* d_actions, int32_t n_batches, int32_t T, uint8_t* d_obs,
                             float* d_reward, uint8_t* d_done, uint32_t flags, const ScriptedArgs* scripted, snk_graph** out) {
  if (!h || !d_actions || !out || T < 1 || n_batches < 1) return fail(SNK_EINVAL, "bad argument");
  const Params& p = h->p;
  const size_t obs_step = (size_t)p.N * h->obs_out_env_bytes;
  if (d_obs) {
    if (((uintptr_t)d_obs & 15) != 0) return fail(SNK_EINVAL, "rollout obs buffer must be 16-byte aligned");
    if (obs_step % 16 != 0 && T > 1) return fail(SNK_EINVAL, "N * obs bytes per env must be a multiple of 16 for a rollout");
  }
  CUDA_TRY(cudaSetDevice(h->cfg.device));
  snk_graph* g = new snk_graph();
  g->h = h; g->graph = nullptr; g->exec = nullptr; g->T = T;
  g->d_actions = d_actions; g->n_batches = n_batches; g->d_obs = d_obs; g->d_reward = d_reward; g->d_done = d_done; g->flags = flags;
  const bool reducing = h->comm && h->reduce_enabled;                   // NCCL form: per-step slots and a forked branch
  const bool pushing = h->peer.ranks > 0 && h->reduce_enabled;          // peer form: nothing beside the step kernels
  g->obs_target = h->d_obs_user; g->with_comm = reducing; g->with_push = pushing; g->d_slots = nullptr;
  if (reducing) {
    const size_t bytes = sizeof(double) * 2 * (size_t)T * SNK_NSTATS;
    if (cudaMalloc(&g->d_slots, bytes) != cudaSuccess || cudaMemset(g->d_slots, 0, bytes) != cudaSuccess) {
      delete g;
      return fail(SNK_ENOMEM, "cudaMalloc of the graph's statistics slots");
    }
  }
  const uint64_t l0 = h->launches;
  cudaStream_t s = h->cap_stream;
  cudaError_t ce = cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal);
  if (ce != cudaSuccess) { delete g; return fail(SNK_ECUDA, "cudaStreamBeginCapture: %s", cudaGetErrorString(ce)); }
  int rc = SNK_OK;
  for (int32_t t = 0; t < T && rc == SNK_OK; ++t) {
    RolloutSlot slot;
    slot.obs = d_obs ? d_obs + (size_t)t * obs_step : nullptr;
    slot.reward = d_reward ? d_reward + (size_t)t * p.N : nullptr;
    slot.done = d_done ? d_done + (size_t)t * p.N : nullptr;
    if (scripted) {  // the policy kernel reads the state step t-1 left and writes this step's actions
      // (occupancy from the previous captured step's observations; step 0 walks the bodies: the graph cannot know where
      // the observations of the state it will be launched on are)
      if (snk_launch_scripted_actions(h->p, h->d_actions_own, scripted->step0 + (uint64_t)t, scripted->seed, scripted->eps_permille,
                                      t && h->cfg.obs_mode != SNK_OBS_GRID ? g->last_native_obs : nullptr, s) != cudaSuccess)
        rc = fail(SNK_ECUDA, "capture: scripted policy kernel");
      h->launches++;
    }
    const CaptureCtx cap = {t, g->d_slots, T};
    if (rc == SNK_OK) rc = launch(h, MODE_STEP, d_actions + (size_t)(t % n_batches) * p.N * p.S, nullptr, s, &slot, &cap);
    g->last_native_obs = (slot.obs && h->cfg.obs_mode != SNK_OBS_ATARI84) ? slot.obs : h->p.obs;
  }
  if (rc == SNK_OK && reducing) {  // join the side branch (its last all-reduce) back into the origin stream
    if (cudaStreamWaitEvent(s, h->cev_red[0], 0) != cudaSuccess) rc = fail(SNK_ECUDA, "cudaStreamWaitEvent (capture join)");
  }
  if (rc == SNK_OK && d_obs && (flags & SNK_GRAPH_SYNC_BACK)) {
    // leave the handle's own buffers as after T calls of snk_step
    const uint8_t* last = d_obs + (size_t)(T - 1) * obs_step;
    if (cudaMemcpyAsync(h->d_obs_user, last, obs_step, cudaMemcpyDeviceToDevice, s) != cudaSuccess) rc = fail(SNK_ECUDA, "capture: obs copy-back");
    if (d_reward && cudaMemcpyAsync(p.reward, d_reward + (size_t)(T - 1) * p.N, (size_t)p.N * 4, cudaMemcpyDeviceToDevice, s) != cudaSuccess)
      rc = fail(SNK_ECUDA, "capture: reward copy-back");
    if (d_done && cudaMemcpyAsync(p.done, d_done + (size_t)(T - 1) * p.N, (size_t)p.N, cudaMemcpyDeviceToDevice, s) != cudaSuccess)
      rc = fail(SNK_ECUDA, "capture: done copy-back");
  }
  ce = cudaStreamEndCapture(s, &g->graph);
  g->launches_per_run = h->launches - l0;
  h->launches = l0;  // nothing ran yet
  g->collectives_per_run = (reducing || pushing) ? (uint64_t)T : 0;
  if (rc != SNK_OK) { snk_graph_destroy(g); return rc; }
  if (ce != cudaSuccess) { snk_graph_destroy(g); return fail(SNK_ECUDA, "cudaStreamEndCapture: %s", cudaGetErrorString(ce)); }
  ce = cudaGraphInstantiate(&g->exec, g->graph, 0);
  if (ce != cudaSuccess) { snk_graph_destroy(g); return fail(SNK_ECUDA, "cudaGraphInstantiate: %s", cudaGetErrorString(ce)); }
  // move the executable graph to the device now, not inside the caller's first launch (a short rollout would pay it per step)
  if (cudaGraphUpload(g->exec, h->cap_stream) == cudaSuccess) cudaStreamSynchronize(h->cap_stream);
  cudaGetLastError();
  *out = g;
  return SNK_OK;
}

extern "C" int snk_graph_create(snk_handle* h, const int8_t* d_actions, int32_t n_batches, int32_t T, uint8_t* d_obs,
                                float* d_reward, uint8_t* d_done, uint32_t flags, snk_graph** out) {
  return graph_create_impl(h, d_actions, n_batches, T, d_obs, d_reward, d_done, flags, nullptr, out);
}

extern "C" int snk_graph_create_scripted(snk_handle* h, int32_t T, uint64_t step0, uint64_t seed, int32_t eps_permille, snk_graph** out) {
  if (!h || eps_permille < 0 || eps_permille > 1000) return fail(SNK_EINVAL, "bad argument");
  if (h->p.family != 1 || h->cfg.rules != SNK_RULES_CLASSIC)
    return fail(SNK_EINVAL, "the scripted policy needs a lane-family configuration with classic rules");
  ScriptedArgs a = {step0, seed, eps_permille};
  return graph_create_impl(h, h->d_actions_own, 1, T, nullptr, nullptr, nullptr, 0, &a, out);
}

extern "C" int snk_graph_launch(snk_graph* g, void* stream) {
  if (!g || !g->exec) return fail(SNK_EINVAL, "graph is NULL");
  snk_handle* h = g->h;
  cudaStream_t s = (cudaStream_t)stream;
  CUDA_TRY(cudaSetDevice(h->cfg.device));
  if (g->with_comm) {
    int rc = join_side(h, s);  // eager all-reduces still reading the snapshot slots
    if (rc) return rc;
  }
  CUDA_TRY(cudaGraphLaunch(g->exec, s));
  h->obs_current = g->last_native_obs;
  h->launches += g->launches_per_run;
  h->collectives += g->collectives_per_run;
  if (g->with_comm) {
    h->d_global_last = g->d_slots + (size_t)(2 * g->T - 1) * SNK_NSTATS;  // the result slot of the graph's last step
    h->ev_red_valid[0] = h->ev_red_valid[1] = false;  // the graph joined its own all-reduces; stream order covers them
  }
  return SNK_OK;
}

extern "C" int snk_rollout(snk_handle* h, const int8_t* d_actions, int32_t T, uint8_t* d_obs, float* d_reward, uint8_t* d_done,
                           void* stream) {
  if (!h || !d_actions || !d_obs || T < 1) return fail(SNK_EINVAL, "bad argument");
  snk_graph* g = h->rollout_cache;
  const uint32_t flags = SNK_GRAPH_SYNC_BACK;
  if (g && !(g->d_actions == d_actions && g->n_batches == T && g->T == T && g->d_obs == d_obs && g->d_reward == d_reward &&
             g->d_done == d_done && g->flags == flags && g->obs_target == h->d_obs_user &&
             g->with_comm == (h->comm && h->reduce_enabled) && g->with_push == (h->peer.ranks > 0 && h->reduce_enabled))) {
    CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));  // the cached graph may still be running
    snk_graph_destroy(g);
    g = nullptr;
  }
  if (!g) {
    int rc = snk_graph_create(h, d_actions, T, T, d_obs, d_reward, d_done, flags, &g);
    if (rc) return rc;
    h->rollout_cache = g;
  }
  return snk_graph_launch(g, stream);
}

// ------------------------------------------------------------------ host-buffer step
static int step_host_impl(snk_handle* h, const int8_t* h_actions, uint8_t* h_obs, int32_t n_views_out, float* h_reward,
                          uint8_t* h_done, uint8_t* h_num_alive, void* stream, bool sync) {
  if (!h || !h_actions) return fail(SNK_EINVAL, "NULL argument");
  cudaStream_t s = (cudaStream_t)stream;
  const Params& p = h->p;
  if (h->cfg.obs_mode == SNK_OBS_GRID && n_views_out != 0)
    return fail(SNK_EINVAL, "obs_mode grid copies the grid: n_views_out must be 0 (snk_expand_views gives views)");
  if (n_views_out <= 0 || n_views_out > p.K) n_views_out = p.K;
  if (n_views_out < p.K && n_views_out > 4) return fail(SNK_EINVAL, "a view subset holds at most 4 views");
  CUDA_TRY(cudaSetDevice(h->cfg.device));
  CUDA_TRY(cudaMemcpyAsync(h->d_actions_own, h_actions, (size_t)p.N * p.S, cudaMemcpyHostToDevice, s));
  int rc = launch(h, MODE_STEP, h->d_actions_own, nullptr, s);
  if (rc) return rc;
  // the small arrays first: the learner's bookkeeping can start while the observations are still in flight
  if (h_reward) CUDA_TRY(cudaMemcpyAsync(h_reward, p.reward, (size_t)p.N * 4, cudaMemcpyDeviceToHost, s));
  if (h_done) CUDA_TRY(cudaMemcpyAsync(h_done, p.done, (size_t)p.N, cudaMemcpyDeviceToHost, s));
  if (h_num_alive) CUDA_TRY(cudaMemcpyAsync(h_num_alive, p.num_alive, (size_t)p.N, cudaMemcpyDeviceToHost, s));
  if (h_obs) {
    const size_t px_per_env = h->obs_out_env_bytes / (size_t)p.C;
    if (n_views_out == p.K) {
      CUDA_TRY(cudaMemcpyAsync(h_obs, h->d_obs_user, (size_t)p.N * h->obs_out_env_bytes, cudaMemcpyDeviceToHost, s));
    } else {
      const size_t bytes = (size_t)p.N * px_per_env * 3 * (size_t)n_views_out;
      if (h->views_bytes < bytes) {
        dev_free(h, h->d_views); h->d_views = nullptr; h->views_bytes = 0;
        if ((rc = dev_alloc(h, &h->d_views, bytes, false))) return rc;
        h->views_bytes = bytes;
      }
      CUDA_TRY(snk_launch_extract_views(h->d_obs_user, h->d_views, (long long)((size_t)p.N * px_per_env), p.C, n_views_out, s));
      h->launches++;
      CUDA_TRY(cudaMemcpyAsync(h_obs, h->d_views, bytes, cudaMemcpyDeviceToHost, s));
    }
  }
  if (sync) CUDA_TRY(cudaStreamSynchronize(s));
  return SNK_OK;
}

extern "C" int snk_step_host(snk_handle* h, const int8_t* h_actions, uint8_t* h_obs, float* h_reward, uint8_t* h_done,
                             uint8_t* h_num_alive, void* stream) {
  return step_host_impl(h, h_actions, h_obs, 0, h_reward, h_done, h_num_alive, stream, true);
}

extern "C" int snk_step_host_views(snk_handle* h, const int8_t* h_actions, uint8_t* h_obs, int32_t n_views_out, float* h_reward,
                                   uint8_t* h_done, uint8_t* h_num_alive, void* stream) {
  return step_host_impl(h, h_actions, h_obs, n_views_out, h_reward, h_done, h_num_alive, stream, true);
}

extern "C" int snk_step_host_async(snk_handle* h, const int8_t* h_actions, uint8_t* h_obs, int32_t n_views_out, float* h_reward,
                                   uint8_t* h_done, uint8_t* h_num_alive, void* stream) {
  return step_host_impl(h, h_actions, h_obs, n_views_out, h_reward, h_done, h_num_alive, stream, false);
}

// ------------------------------------------------------------------ pipelined host step, observations stay in HBM
// The learner sits on the GPU (north_star) but is driven from the host: per step it sends N*S action bytes and wants the
// per-env scalars back.  On ONE stream that is H2D -> kernel -> D2H, each copy a PCIe round trip the next kernel waits
// for (measured: 120 us per step around a 66 us kernel).  Here the copies run on two streams of their own and every step
// writes its scalars into one of SNK_SCALAR_SLOTS device slots, so the step stream carries kernels only: the H2D of step
// t + 1 and the D2H of step t - 1 overlap the kernel of step t, and a host that reads a step's scalars two steps late
// never waits for the device.
static void scalars_layout(const snk_handle* h, size_t* bytes, size_t off[5]) {
  const size_t N = (size_t)h->p.N;
  off[0] = 0;                          // reward          float [N]
  off[1] = off[0] + align16(4 * N);    // done            uint8 [N]
  off[2] = off[1] + align16(N);        // num_alive       uint8 [N]
  off[3] = off[2] + align16(N);        // episode return  float [N]  (valid where done)
  off[4] = off[3] + align16(4 * N);    // episode length  int32 [N]  (valid where done)
  *bytes = off[4] + align16(4 * N);
}

extern "C" int snk_scalars_layout(const snk_handle* h, size_t* out) {
  if (!h || !out) return fail(SNK_EINVAL, "NULL argument");
  scalars_layout(h, &out[0], &out[1]);
  return SNK_OK;
}

static int scalars_init(snk_handle* h) {
  if (h->s_in) return SNK_OK;
  scalars_layout(h, &h->sc_bytes, h->sc_off);
  CUDA_TRY(cudaStreamCreateWithFlags(&h->s_in, cudaStreamNonBlocking));
  CUDA_TRY(cudaStreamCreateWithFlags(&h->s_out, cudaStreamNonBlocking));
  for (int i = 0; i < SNK_SCALAR_SLOTS; ++i) {
    int rc;
    if ((rc = dev_alloc(h, &h->sc[i].d_act, (size_t)h->p.N * h->p.S, true))) return rc;
    if ((rc = dev_alloc(h, &h->sc[i].d_out, h->sc_bytes, true))) return rc;
    CUDA_TRY(cudaEventCreateWithFlags(&h->sc[i].ev_in, cudaEventDisableTiming));
    CUDA_TRY(cudaEventCreateWithFlags(&h->sc[i].ev_k, cudaEventDisableTiming));
    CUDA_TRY(cudaEventCreateWithFlags(&h->sc[i].ev_out, cudaEventDisableTiming));
    h->sc[i].used = false;
  }
  CUDA_TRY(cudaDeviceSynchronize());  // the memsets above ran on the legacy stream
  return SNK_OK;
}

extern "C" int snk_step_scalars_async(snk_handle* h, const int8_t* h_actions, uint8_t* h_out, int32_t slot, void* stream) {
  if (!h || !h_actions || !h_out || slot < 0 || slot >= SNK_SCALAR_SLOTS) return fail(SNK_EINVAL, "bad argument");
  CUDA_TRY(cudaSetDevice(h->cfg.device));
  int rc = scalars_init(h);
  if (rc) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  snk_handle::ScalarSlot& q = h->sc[slot];
  const Params& p = h->p;
  // actions: after the kernel that read this slot's action buffer two steps ago (implied when the host has already
  // waited for that step's scalars -- snk_scalars_wait -- as a caller that reuses the slot's host block must)
  const bool ordered = !q.used || q.host_synced;
  if (!ordered) CUDA_TRY(cudaStreamWaitEvent(h->s_in, q.ev_k, 0));
  CUDA_TRY(cudaMemcpyAsync(q.d_act, h_actions, (size_t)p.N * p.S, cudaMemcpyHostToDevice, h->s_in));
  CUDA_TRY(cudaEventRecord(q.ev_in, h->s_in));
  CUDA_TRY(cudaStreamWaitEvent(s, q.ev_in, 0));
  if (!ordered) CUDA_TRY(cudaStreamWaitEvent(s, q.ev_out, 0));  // this slot's previous scalars have left the device
  RolloutSlot rs;
  rs.reward = reinterpret_cast<float*>(q.d_out + h->sc_off[0]);
  rs.done = q.d_out + h->sc_off[1];
  rs.alive = q.d_out + h->sc_off[2];
  rs.fin_ret = reinterpret_cast<float*>(q.d_out + h->sc_off[3]);
  rs.fin_len = reinterpret_cast<int32_t*>(q.d_out + h->sc_off[4]);
  if ((rc = launch(h, MODE_STEP, q.d_act, nullptr, s, &rs))) return rc;
  CUDA_TRY(cudaEventRecord(q.ev_k, s));
  CUDA_TRY(cudaStreamWaitEvent(h->s_out, q.ev_k, 0));
  CUDA_TRY(cudaMemcpyAsync(h_out, q.d_out, h->sc_bytes, cudaMemcpyDeviceToHost, h->s_out));
  CUDA_TRY(cudaEventRecord(q.ev_out, h->s_out));
  q.used = true; q.host_synced = false;
  return SNK_OK;
}

extern "C" int snk_scalars_wait(snk_handle* h, int32_t slot) {
  if (!h || slot < 0 || slot >= SNK_SCALAR_SLOTS) return fail(SNK_EINVAL, "bad argument");
  if (!h->s_in || !h->sc[slot].used) return SNK_OK;
  CUDA_TRY(cudaEventSynchronize(h->sc[slot].ev_out));
  h->sc[slot].host_synced = true;
  return SNK_OK;
}

// Pinned host memory on the NUMA node the handle's GPU hangs off: with one process per GPU all writing ~350 MB of
// observations per step into host DRAM, buffers that land on one socket (first touch by whichever core ran the
// allocation) make seven of eight GPUs cross the inter-socket link.  The node comes from sysfs; the pages are placed by
// a temporary MPOL_BIND memory policy around cudaHostAlloc (raw syscall, no libnuma).
static int gpu_numa_node(int device) {
  char bus[32] = "";
  if (cudaDeviceGetPCIBusId(bus, sizeof(bus), device) != cudaSuccess) return -1;
  for (char* c = bus; *c; ++c) if (*c >= 'A' && *c <= 'Z') *c += 'a' - 'A';
  char path[128];
  snprintf(path, sizeof(path), "/sys/bus/pci/devices/%s/numa_node", bus);
  FILE* f = fopen(path, "r");
  if (!f) return -1;
  int node = -1;
  if (fscanf(f, "%d", &node) != 1) node = -1;
  fclose(f);
  return node;
}

extern "C" int snk_host_alloc(snk_handle* h, size_t bytes, void** out, int32_t* numa_node) {
  if (!h || !out || !bytes) return fail(SNK_EINVAL, "bad argument");
  CUDA_TRY(cudaSetDevice(h->cfg.device));
  const int node = gpu_numa_node(h->cfg.device);
  bool bound = false;
#ifdef SYS_set_mempolicy
  if (node >= 0 && node < 1024) {
    unsigned long mask[16] = {0};
    mask[node / (8 * sizeof(unsigned long))] |= 1ul << (node % (8 * sizeof(unsigned long)));
    bound = syscall(SYS_set_mempolicy, 2 /*MPOL_BIND*/, mask, (unsigned long)(8 * sizeof(mask))) == 0;
  }
#endif
  void* ptr = nullptr;
  cudaError_t e = cudaHostAlloc(&ptr, bytes, cudaHostAllocDefault);
  if (e == cudaSuccess) memset(ptr, 0, bytes);  // first touch under the policy
#ifdef SYS_set_mempolicy
  if (bound) syscall(SYS_set_mempolicy, 0 /*MPOL_DEFAULT*/, nullptr, 0ul);
#endif
  if (e != cudaSuccess) return fail(SNK_ENOMEM, "cudaHostAlloc(%zu bytes): %s", bytes, cudaGetErrorString(e));
  h->host_allocs.push_back(std::make_pair(ptr, bytes));
  *out = ptr;
  if (numa_node) *numa_node = bound ? node : -1;
  return SNK_OK;
}

extern "C" int snk_host_free(snk_handle* h, void* ptr) {
  if (!h || !ptr) return SNK_OK;
  for (size_t i = 0; i < h->host_allocs.size(); ++i)
    if (h->host_allocs[i].first == ptr) {
      cudaFreeHost(ptr);
      h->host_allocs.erase(h->host_allocs.begin() + (long)i);
      return SNK_OK;
    }
  return fail(SNK_EINVAL, "pointer was not allocated by snk_host_alloc on this handle");
}

extern "C" int snk_set_obs_target(snk_handle* h, uint8_t* d_obs, size_t bytes) {
  if (!h) return fail(SNK_EINVAL, "handle is NULL");
  const bool atari = h->cfg.obs_mode == SNK_OBS_ATARI84;
  if (!d_obs) {
    h->d_obs_user = atari ? h->d_obs84_own : h->d_obs_own;
    if (!atari) h->p.obs = h->d_obs_own;
    return SNK_OK;
  }
  if (((uintptr_t)d_obs & 15) != 0) return fail(SNK_EINVAL, "obs target must be 16-byte aligned");
  const size_t need = (size_t)h->p.N * h->obs_out_env_bytes;
  if (bytes < need) return fail(SNK_EINVAL, "obs target too small: %zu < %zu", bytes, need);
  h->d_obs_user = d_obs;
  if (!atari) h->p.obs = d_obs;  // native mode: the step kernel writes straight into the target
  return SNK_OK;
}

extern "C" int snk_set_main_view_target(snk_handle* h, uint8_t* d_main, size_t bytes) {
  if (!h) return fail(SNK_EINVAL, "handle is NULL");
  if (!d_main) { h->d_main_target = nullptr; return SNK_OK; }
  if (h->cfg.obs_mode == SNK_OBS_GRID) return fail(SNK_EINVAL, "obs_mode grid has no main-view target: expand view 0 with snk_expand_views");
  const size_t need = (size_t)h->p.N * (h->obs_out_env_bytes / (size_t)h->p.C) * 3;
  if (bytes < need) return fail(SNK_EINVAL, "main-view target too small: %zu < %zu", bytes, need);
  h->d_main_target = d_main;
  return SNK_OK;
}

extern "C" int snk_set_draw_tape(snk_handle* h, const uint32_t* h_vals, const uint32_t* h_bounds, const uint64_t* h_offsets) {
  if (!h || !h_vals || !h_offsets) return fail(SNK_EINVAL, "NULL argument");
  CUDA_TRY(cudaSetDevice(h->cfg.device));
  CUDA_TRY(cudaDeviceSynchronize());
  const size_t N = (size_t)h->p.N, n = (size_t)h_offsets[N];
  dev_free(h, h->d_tape_vals); dev_free(h, h->d_tape_bounds); dev_free(h, h->d_tape_off);  // a previous tape
  h->d_tape_vals = h->d_tape_bounds = nullptr; h->d_tape_off = nullptr;
  int rc;
  if ((rc = dev_alloc(h, &h->d_tape_vals, n + 1, false))) return rc;
  if ((rc = dev_alloc(h, &h->d_tape_off, N + 1, false))) return rc;
  CUDA_TRY(cudaMemcpy(h->d_tape_vals, h_vals, n * 4, cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMemcpy(h->d_tape_off, h_offsets, (N + 1) * 8, cudaMemcpyHostToDevice));
  if (h_bounds) {
    if ((rc = dev_alloc(h, &h->d_tape_bounds, n + 1, false))) return rc;
    CUDA_TRY(cudaMemcpy(h->d_tape_bounds, h_bounds, n * 4, cudaMemcpyHostToDevice));
  }
  h->p.rng_mode = SNK_RNG_TAPE;
  h->cfg.rng_mode = SNK_RNG_TAPE;
  return SNK_OK;
}

static int ensure_blob(snk_handle* h, size_t bytes) {
  if (h->d_blob && h->blob_bytes >= bytes) return SNK_OK;
  dev_free(h, h->d_blob);
  h->d_blob = nullptr; h->blob_bytes = 0;
  int rc = dev_alloc(h, &h->d_blob, bytes, true);
  if (rc == SNK_OK) h->blob_bytes = bytes;
  return rc;
}

// the blob layout of a `count`-env configuration of this handle's geometry
static int sub_layout(const snk_handle* h, int64_t count, snk_state_layout* lay) {
  snk_config sub = h->cfg;
  sub.num_envs = count; sub.env_id_base = 0;
  return snk_state_layout_of(&sub, lay);
}

extern "C" int snk_dump_state_range(snk_handle* h, int64_t first, int64_t count, void* h_dst, size_t bytes) {
  if (!h || !h_dst) return fail(SNK_EINVAL, "NULL argument");
  if (first < 0 || count < 1 || first + count > h->p.N) return fail(SNK_EINVAL, "env range [%lld, %lld) outside [0, %lld)",
                                                                    (long long)first, (long long)(first + count), h->p.N);
  snk_state_layout lay;
  int rc = sub_layout(h, count, &lay);
  if (rc) return rc;
  if (bytes < lay.total_bytes) return fail(SNK_EINVAL, "buffer too small: %zu < %zu", bytes, lay.total_bytes);
  CUDA_TRY(cudaSetDevice(h->cfg.device));
  if ((rc = ensure_blob(h, lay.total_bytes))) return rc;
  CUDA_TRY(cudaDeviceSynchronize());
  CUDA_TRY(snk_launch_save(h->p, nullptr, first, count, h->d_blob, lay, 0));  // writes every byte of the blob
  h->launches++;
  CUDA_TRY(cudaMemcpy(h_dst, h->d_blob, lay.total_bytes, cudaMemcpyDeviceToHost));
  return SNK_OK;
}

extern "C" int snk_dump_state(snk_handle* h, void* h_dst, size_t bytes) {
  if (!h) return fail(SNK_EINVAL, "NULL argument");
  return snk_dump_state_range(h, 0, h->p.N, h_dst, bytes);
}

extern "C" int snk_load_state(snk_handle* h, const void* h_src, size_t bytes) {
  if (!h || !h_src) return fail(SNK_EINVAL, "NULL argument");
  if (bytes < h->lay.total_bytes) return fail(SNK_EINVAL, "buffer too small: %zu < %zu", bytes, h->lay.total_bytes);
  CUDA_TRY(cudaSetDevice(h->cfg.device));
  int rc = ensure_blob(h, h->lay.total_bytes);
  if (rc) return rc;
  CUDA_TRY(cudaDeviceSynchronize());
  CUDA_TRY(cudaMemcpy(h->d_blob, h_src, h->lay.total_bytes, cudaMemcpyHostToDevice));
  h->obs_current = nullptr;
  CUDA_TRY(snk_launch_restore(h->p, nullptr, h->p.N, h->d_blob, h->lay, 0));  // clears frame_ok: the own buffer no longer shows the records
  h->launches++;
  CUDA_TRY(cudaDeviceSynchronize());
  uint32_t flags = 0;
  CUDA_TRY(cudaMemcpy(&flags, h->p.err, 4, cudaMemcpyDeviceToHost));
  if (flags & SNK_DEVERR_BAD_STATE) {
    flags &= ~SNK_DEVERR_BAD_STATE;
    CUDA_TRY(cudaMemcpy(h->p.err, &flags, 4, cudaMemcpyHostToDevice));
    return fail(SNK_ESTATE, "state blob rejected: a body that is too long, leaves the padded grid, has a velocity code above 4 "
                            "or whose consecutive segments are not adjacent cells (those snakes were left empty)");
  }
  return SNK_OK;
}

// A state change the host did not see while a graph is being recorded on `stream`: the recorded work has not run, so the
// host-side view of the state (obs_current) stays as it is, the way launch() treats a captured step.
static bool stream_capturing(cudaStream_t stream) {
  cudaStreamCaptureStatus st = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(stream, &st) != cudaSuccess) {
    cudaGetLastError();
    return true;  // the legacy stream while another stream captures globally: a capture is under way
  }
  return st != cudaStreamCaptureStatusNone;
}

static int envs_check(const snk_handle* h, const void* d_blob, int64_t count, size_t bytes, bool idx_null, snk_state_layout* lay) {
  if (!h || !d_blob) return fail(SNK_EINVAL, "NULL argument");
  if (count < 1) return fail(SNK_EINVAL, "count must be >= 1, got %lld", (long long)count);
  if (idx_null && count > h->p.N) return fail(SNK_EINVAL, "count %lld > num_envs %lld without indices", (long long)count, h->p.N);
  if (((uintptr_t)d_blob & 15) != 0) return fail(SNK_EINVAL, "device blob must be 16-byte aligned");
  int rc = sub_layout(h, count, lay);
  if (rc) return rc;
  if (bytes < lay->total_bytes) return fail(SNK_EINVAL, "blob too small: %zu < %zu bytes for %lld envs", bytes, lay->total_bytes,
                                            (long long)count);
  return SNK_OK;
}

extern "C" int snk_save_envs(snk_handle* h, const int64_t* d_idx, int64_t count, void* d_blob, size_t bytes, void* stream) {
  snk_state_layout lay;
  int rc = envs_check(h, d_blob, count, bytes, d_idx == nullptr, &lay);
  if (rc) return rc;
  CUDA_TRY(cudaSetDevice(h->cfg.device));
  CUDA_TRY(snk_launch_save(h->p, d_idx, 0, count, (uint8_t*)d_blob, lay, (cudaStream_t)stream));
  h->launches++;
  return SNK_OK;
}

extern "C" int snk_restore_envs(snk_handle* h, const int64_t* d_idx, int64_t count, const void* d_blob, size_t bytes, void* stream) {
  snk_state_layout lay;
  int rc = envs_check(h, d_blob, count, bytes, d_idx == nullptr, &lay);
  if (rc) return rc;
  CUDA_TRY(cudaSetDevice(h->cfg.device));
  CUDA_TRY(snk_launch_restore(h->p, d_idx, count, (const uint8_t*)d_blob, lay, (cudaStream_t)stream));
  h->launches++;
  if (!stream_capturing((cudaStream_t)stream)) h->obs_current = nullptr;
  return SNK_OK;
}

extern "C" int snk_copy_envs(snk_handle* h, const int64_t* d_src, const int64_t* d_dst, int64_t count, void* stream) {
  if (!h || !d_src || !d_dst) return fail(SNK_EINVAL, "NULL argument");
  if (count < 1) return fail(SNK_EINVAL, "count must be >= 1, got %lld", (long long)count);
  CUDA_TRY(cudaSetDevice(h->cfg.device));
  CUDA_TRY(snk_launch_copy(h->p, h->p, d_src, d_dst, count, (cudaStream_t)stream));
  h->launches++;
  if (!stream_capturing((cudaStream_t)stream)) h->obs_current = nullptr;
  return SNK_OK;
}

extern "C" int snk_clone_envs(const snk_handle* src, const int64_t* d_src, snk_handle* dst, const int64_t* d_dst, int64_t count,
                              void* stream) {
  if (!src || !dst || !d_src || !d_dst) return fail(SNK_EINVAL, "NULL argument");
  if (count < 1) return fail(SNK_EINVAL, "count must be >= 1, got %lld", (long long)count);
  const snk_config &a = src->cfg, &b = dst->cfg;
  if (a.device != b.device) return fail(SNK_EINVAL, "device differs: %d vs %d", a.device, b.device);
  if (a.size != b.size) return fail(SNK_EINVAL, "size differs: %d vs %d", a.size, b.size);
  if (a.n_snakes != b.n_snakes) return fail(SNK_EINVAL, "n_snakes differs: %d vs %d", a.n_snakes, b.n_snakes);
  if (a.n_fruits != b.n_fruits) return fail(SNK_EINVAL, "n_fruits differs: %d vs %d", a.n_fruits, b.n_fruits);
  if (a.rules != b.rules) return fail(SNK_EINVAL, "rules differ: %d vs %d", a.rules, b.rules);
  // the private layout: the family follows the launch plan (the image size), so one configuration can have two
  const Params &ps = src->p, &pd = dst->p;
  const struct { const char* name; int s, d; } layout[] = {
      {"family", ps.family, pd.family}, {"RW", ps.RW, pd.RW}, {"CW", ps.CW, pd.CW}, {"cap", ps.cap, pd.cap},
      {"grid_stride", ps.grid_stride, pd.grid_stride}, {"GBW", ps.GBW, pd.GBW}};
  for (const auto& f : layout)
    if (f.s != f.d) return fail(SNK_EINVAL, "private layout differs: %s %d vs %d", f.name, f.s, f.d);
  CUDA_TRY(cudaSetDevice(b.device));
  CUDA_TRY(snk_launch_copy(ps, pd, d_src, d_dst, count, (cudaStream_t)stream));
  dst->launches++;
  if (!stream_capturing((cudaStream_t)stream)) dst->obs_current = nullptr;
  return SNK_OK;
}

extern "C" int snk_get_stats(snk_handle* h, double* h_stats, void* stream) {
  if (!h || !h_stats) return fail(SNK_EINVAL, "NULL argument");
  CUDA_TRY(cudaSetDevice(h->cfg.device));
  CUDA_TRY(cudaMemcpyAsync(h_stats, h->p.stats, sizeof(double) * SNK_NSTATS, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));
  return SNK_OK;
}

extern "C" int snk_reset_stats(snk_handle* h, void* stream) {
  if (!h) return fail(SNK_EINVAL, "handle is NULL");
  CUDA_TRY(cudaSetDevice(h->cfg.device));
  CUDA_TRY(cudaMemsetAsync(h->p.stats, 0, sizeof(double) * SNK_NSTATS, (cudaStream_t)stream));
  return SNK_OK;
}

extern "C" int snk_check_errors(snk_handle* h, uint32_t* flags, void* stream) {
  if (!h || !flags) return fail(SNK_EINVAL, "NULL argument");
  CUDA_TRY(cudaSetDevice(h->cfg.device));
  CUDA_TRY(cudaMemcpyAsync(flags, h->p.err, 4, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  CUDA_TRY(cudaMemsetAsync(h->p.err, 0, 4, (cudaStream_t)stream));
  CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));
  return SNK_OK;
}

// ------------------------------------------------------------------ the path's one collective
extern "C" int snk_comm_unique_id(uint8_t* out128) {
  if (!out128) return fail(SNK_EINVAL, "NULL argument");
  int rc = nccl_load();
  if (rc) return rc;
  ncclUniqueId id;
  NCCL_TRY(g_nccl.GetUniqueId(&id));
  memcpy(out128, &id, sizeof(id));
  return SNK_OK;
}

// what both forms of the per-step reduction share: the high-priority side stream, the fork / join events (eager and
// capture-time sets) and the two eager snapshot / result slots
static int ensure_side(snk_handle* h) {
  if (h->side) return SNK_OK;
  int lo = 0, hi = 0;
  CUDA_TRY(cudaDeviceGetStreamPriorityRange(&lo, &hi));
  CUDA_TRY(cudaStreamCreateWithPriority(&h->side, cudaStreamNonBlocking, hi));
  for (int i = 0; i < 2; ++i) {
    CUDA_TRY(cudaEventCreateWithFlags(&h->ev_step[i], cudaEventDisableTiming));
    CUDA_TRY(cudaEventCreateWithFlags(&h->ev_red[i], cudaEventDisableTiming));
    CUDA_TRY(cudaEventCreateWithFlags(&h->cev_step[i], cudaEventDisableTiming));
    CUDA_TRY(cudaEventCreateWithFlags(&h->cev_red[i], cudaEventDisableTiming));
  }
  int rc;
  if ((rc = dev_alloc(h, &h->d_snap, (size_t)2 * SNK_NSTATS, true))) return rc;
  if ((rc = dev_alloc(h, &h->d_global, (size_t)2 * SNK_NSTATS, true))) return rc;
  return SNK_OK;
}

extern "C" int snk_comm_init(snk_handle* h, const uint8_t* id128, int32_t n_ranks, int32_t rank) {
  if (!h || !id128 || n_ranks < 1 || rank < 0 || rank >= n_ranks) return fail(SNK_EINVAL, "bad argument");
  if (h->comm || h->peer.ranks > 0) return fail(SNK_EINVAL, "a reduction is already set up on this handle");
  int rc = nccl_load();
  if (rc) return rc;
  CUDA_TRY(cudaSetDevice(h->cfg.device));
  ncclUniqueId id;
  memcpy(&id, id128, sizeof(id));
  ncclComm_t comm = nullptr;
  if (g_nccl.CommInitRankConfig) {
    // a 64-byte all-reduce needs ONE CTA: every further channel is a CTA that has to wait for room on an SM the step
    // kernel fills (measured at 2 GPUs: the default cost 2 us per step, 3 %)
    NcclConfig218 cfg;
    cfg.size = sizeof(cfg); cfg.magic = 0xcafebeefu; cfg.version = 21800;
    const int undef = (int)0x80000000;  // NCCL_CONFIG_UNDEF_INT
    cfg.blocking = undef; cfg.cgaClusterSize = undef; cfg.minCTAs = 1; cfg.maxCTAs = 1; cfg.netName = nullptr; cfg.splitShare = undef;
    NCCL_TRY(g_nccl.CommInitRankConfig(&comm, n_ranks, id, rank, &cfg));
  } else {
    NCCL_TRY(g_nccl.CommInitRank(&comm, n_ranks, id, rank));
  }
  if ((rc = ensure_side(h))) return rc;
  // one eager all-reduce now: NCCL sets its connections up on first use, which must not happen inside a stream capture
  NCCL_TRY(g_nccl.AllReduce(h->d_snap, h->d_global, SNK_NSTATS, kNcclFloat64, kNcclSum, comm, h->side));
  CUDA_TRY(cudaStreamSynchronize(h->side));
  h->comm = comm; h->comm_ranks = n_ranks; h->comm_rank = rank;
  if (h->rollout_cache) snk_graph_destroy(h->rollout_cache);  // captured without the collective
  return SNK_OK;
}

extern "C" int snk_peer_export(snk_handle* h, uint8_t* out64) {
  if (!h || !out64) return fail(SNK_EINVAL, "NULL argument");
  CUDA_TRY(cudaSetDevice(h->cfg.device));
  if (!h->d_inbox) {
    const size_t bytes = (size_t)SNK_MAX_PEERS * SNK_INBOX_STRIDE;
    void* ptr = nullptr;
    cudaError_t e = cudaMalloc(&ptr, bytes);  // its own allocation: cudaIpc exports whole allocations
    if (e != cudaSuccess) return fail(SNK_ENOMEM, "cudaMalloc(inbox): %s", cudaGetErrorString(e));
    h->allocs.push_back(ptr);
    CUDA_TRY(cudaMemset(ptr, 0, bytes));
    h->d_inbox = (uint8_t*)ptr;
  }
  cudaIpcMemHandle_t ipc;
  static_assert(sizeof(ipc) == 64, "cudaIpcMemHandle_t is 64 bytes");
  CUDA_TRY(cudaIpcGetMemHandle(&ipc, h->d_inbox));
  memcpy(out64, &ipc, sizeof(ipc));
  return SNK_OK;
}

extern "C" int snk_peer_connect(snk_handle* h, const uint8_t* handles, int32_t n_ranks, int32_t rank) {
  if (!h || !handles || n_ranks < 1 || n_ranks > SNK_MAX_PEERS || rank < 0 || rank >= n_ranks) return fail(SNK_EINVAL, "bad argument");
  if (!h->d_inbox) return fail(SNK_EINVAL, "snk_peer_export first");
  if (h->peer.ranks > 0 || h->comm) return fail(SNK_EINVAL, "a reduction is already set up on this handle");
  CUDA_TRY(cudaSetDevice(h->cfg.device));
  PeerArgs a;
  memset(&a, 0, sizeof(a));
  for (int g = 0; g < n_ranks; ++g) {
    if (g == rank) { a.inbox[g] = h->d_inbox; continue; }
    cudaIpcMemHandle_t ipc;
    memcpy(&ipc, handles + (size_t)g * sizeof(ipc), sizeof(ipc));
    void* ptr = nullptr;
    cudaError_t e = cudaIpcOpenMemHandle(&ptr, ipc, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) return fail(SNK_ECOMM, "cudaIpcOpenMemHandle(rank %d): %s", g, cudaGetErrorString(e));
    h->peer_mapped[g] = ptr;
    a.inbox[g] = (uint8_t*)ptr;
  }
  int rc;
  if (!h->d_global && (rc = dev_alloc(h, &h->d_global, (size_t)2 * SNK_NSTATS, true))) return rc;
  a.ranks = n_ranks; a.rank = rank;
  h->peer = a;
  h->comm_ranks = n_ranks; h->comm_rank = rank;
  if (h->rollout_cache) snk_graph_destroy(h->rollout_cache);  // captured without the exchange
  return SNK_OK;
}

extern "C" int snk_comm_enable(snk_handle* h, int32_t on) {
  if (!h) return fail(SNK_EINVAL, "handle is NULL");
  h->reduce_enabled = on != 0;
  if (h->rollout_cache) snk_graph_destroy(h->rollout_cache);
  return SNK_OK;
}

extern "C" int snk_get_stats_global(snk_handle* h, double* h_stats, void* stream) {
  if (!h || !h_stats) return fail(SNK_EINVAL, "NULL argument");
  if (h->peer.ranks > 0) {  // own running sums + the peers' latest pushes, as of now
    cudaStream_t s = (cudaStream_t)stream;
    CUDA_TRY(cudaSetDevice(h->cfg.device));
    CUDA_TRY(snk_launch_sum_inbox(h->peer, h->p.stats, h->d_global, s));
    CUDA_TRY(cudaMemcpyAsync(h_stats, h->d_global, sizeof(double) * SNK_NSTATS, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    return SNK_OK;
  }
  if (!h->comm) return snk_get_stats(h, h_stats, stream);  // one shard: the local sums are the global ones
  cudaStream_t s = (cudaStream_t)stream;
  CUDA_TRY(cudaSetDevice(h->cfg.device));
  int rc = join_side(h, s);
  if (rc) return rc;
  if (!h->d_global_last) return snk_get_stats(h, h_stats, stream);  // no step since snk_comm_init (or its graph is gone)
  CUDA_TRY(cudaMemcpyAsync(h_stats, h->d_global_last, sizeof(double) * SNK_NSTATS, cudaMemcpyDeviceToHost, s));
  CUDA_TRY(cudaStreamSynchronize(s));
  return SNK_OK;
}

extern "C" int snk_comm_bench(snk_handle* h, int32_t iters, double* mean_us) {
  if (!h || !mean_us || iters < 1) return fail(SNK_EINVAL, "bad argument");
  if (!h->comm) return fail(SNK_EINVAL, "no communicator (snk_comm_init)");
  CUDA_TRY(cudaSetDevice(h->cfg.device));
  CUDA_TRY(cudaDeviceSynchronize());
  cudaEvent_t a, b;
  CUDA_TRY(cudaEventCreate(&a)); CUDA_TRY(cudaEventCreate(&b));
  double* scratch = h->d_global;  // in place on the result slots: the values are rewritten by the next step's reduction
  for (int i = 0; i < 5; ++i) NCCL_TRY(g_nccl.AllReduce(h->d_snap, scratch, SNK_NSTATS, kNcclFloat64, kNcclSum, h->comm, h->side));
  CUDA_TRY(cudaEventRecord(a, h->side));
  for (int i = 0; i < iters; ++i) NCCL_TRY(g_nccl.AllReduce(h->d_snap, scratch, SNK_NSTATS, kNcclFloat64, kNcclSum, h->comm, h->side));
  CUDA_TRY(cudaEventRecord(b, h->side));
  CUDA_TRY(cudaStreamSynchronize(h->side));
  float ms = 0.f;
  CUDA_TRY(cudaEventElapsedTime(&ms, a, b));
  cudaEventDestroy(a); cudaEventDestroy(b);
  *mean_us = (double)ms * 1e3 / iters;
  return SNK_OK;
}

extern "C" int snk_comm_info(const snk_handle* h, int32_t* out /*[4]: ranks, rank, collectives issued (low 31 bits), nccl version*/) {
  if (!h || !out) return fail(SNK_EINVAL, "NULL argument");
  out[0] = (h->comm || h->peer.ranks > 0) ? h->comm_ranks : 1; out[1] = h->comm_rank; out[2] = (int32_t)(h->collectives & 0x7fffffff);
  int v = 0;
  if (g_nccl.so && g_nccl.GetVersion) g_nccl.GetVersion(&v);
  out[3] = v;
  return SNK_OK;
}

extern "C" int snk_gen_actions(snk_handle* h, int8_t* d_actions, uint64_t step, uint64_t seed, int32_t n_actions, void* stream) {
  if (!h || !d_actions || n_actions < 1) return fail(SNK_EINVAL, "bad argument");
  CUDA_TRY(cudaSetDevice(h->cfg.device));
  CUDA_TRY(snk_launch_gen_actions(d_actions, h->p.N, h->p.S, h->p.env_id_base, step, seed, n_actions, (cudaStream_t)stream));
  h->launches++;
  return SNK_OK;
}

extern "C" int snk_gen_scripted_actions(snk_handle* h, int8_t* d_actions, uint64_t step, uint64_t seed, int32_t eps_permille, void* stream) {
  if (!h || !d_actions || eps_permille < 0 || eps_permille > 1000) return fail(SNK_EINVAL, "bad argument");
  if (h->p.family != 1 || h->cfg.rules != SNK_RULES_CLASSIC)
    return fail(SNK_EINVAL, "the scripted policy needs a lane-family configuration with classic rules");
  CUDA_TRY(cudaSetDevice(h->cfg.device));
  // the policy reads occupancy from the green bytes of a native image; a grid handle's kernel walks the bodies instead
  const uint8_t* occ = h->cfg.obs_mode == SNK_OBS_GRID ? nullptr : h->obs_current;
  CUDA_TRY(snk_launch_scripted_actions(h->p, d_actions, step, seed, eps_permille, occ, (cudaStream_t)stream));
  h->launches++;
  return SNK_OK;
}

extern "C" int snk_gae(const float* d_rewards, const float* d_values, const uint8_t* d_dones, const float* d_last_values,
                       const uint8_t* d_last_dones, double gamma, double lam, int32_t T, int64_t N, float* d_advs, float* d_returns,
                       int32_t device, void* stream) {
  if (!d_rewards || !d_values || !d_dones || !d_last_values || !d_last_dones || !d_advs || !d_returns || T < 1 || N < 1)
    return fail(SNK_EINVAL, "bad argument");
  CUDA_TRY(cudaSetDevice(device));
  CUDA_TRY(snk_launch_gae(d_rewards, d_values, d_dones, d_last_values, d_last_dones, gamma, lam, T, N, d_advs, d_returns,
                          (cudaStream_t)stream));
  return SNK_OK;
}

extern "C" int snk_expand_views(const uint8_t* d_grid, int64_t n, int32_t size, int32_t first_view, int32_t n_views,
                                uint8_t* d_out, int32_t device, void* stream) {
  if (!d_grid || !d_out) return fail(SNK_EINVAL, "NULL argument");
  if (n < 1) return fail(SNK_EINVAL, "n must be >= 1, got %lld", (long long)n);
  if (size < 2 || size > 254) return fail(SNK_EINVAL, "size must be 2..254, got %d", size);
  if (n_views < 1 || first_view < 0 || first_view + n_views > 32)
    return fail(SNK_EINVAL, "views [%d, %d) outside [0, 32) or empty", first_view, first_view + n_views);
  CUDA_TRY(cudaSetDevice(device));
  const long long VV = (long long)(size + 2) * (size + 2);
  CUDA_TRY(snk_launch_expand_views(d_grid, n * VV, first_view, n_views, d_out, (cudaStream_t)stream));
  return SNK_OK;
}

static int grid_conv_check(int64_t n, int32_t size, int32_t view, int32_t channels) {
  if (channels != SNK_GRID_CONV_CHANNELS)
    return fail(SNK_EINVAL, "channels must be %d, got %d", SNK_GRID_CONV_CHANNELS, channels);
  if (size < 1 || size > 254) return fail(SNK_EINVAL, "size must be 1..254, got %d", size);
  if (view < 0 || view > 31) return fail(SNK_EINVAL, "view must be 0..31, got %d", view);
  if (n < 0) return fail(SNK_EINVAL, "n must be >= 0, got %lld", (long long)n);
  return SNK_OK;
}

static bool misaligned(const void* p, uintptr_t a) { return ((uintptr_t)p & (a - 1)) != 0; }

// the work area of snk_tally: t [N] | episodes [N] | death [N][S] | fruits [N][S], each part 16-byte aligned
static size_t tally_work_bytes(long long N, int S, size_t off[4]) {
  const size_t env = align16((size_t)N * 4), seat = align16((size_t)N * S * 4);
  off[0] = 0; off[1] = env; off[2] = 2 * env; off[3] = 2 * env + seat;
  return 2 * env + 2 * seat;
}

extern "C" int snk_tally_layout(const snk_handle* h, size_t* out) {
  if (!h || !out) return fail(SNK_EINVAL, "NULL argument");
  size_t off[4];
  out[0] = tally_work_bytes(h->p.N, h->p.S, off);
  out[1] = SNK_TALLY_FIELDS;
  return SNK_OK;
}

extern "C" int snk_tally(snk_handle* h, const int32_t* d_group, int32_t n_groups, int32_t episodes_per_env, void* d_work,
                         int64_t* d_counts, int64_t* d_envs_done, void* stream) {
  if (n_groups < 1) return fail(SNK_EINVAL, "n_groups must be >= 1, got %d", n_groups);
  if (episodes_per_env < 1) return fail(SNK_EINVAL, "episodes_per_env must be >= 1, got %d", episodes_per_env);
  if (!d_group || !d_work || !d_counts || !d_envs_done) return fail(SNK_EINVAL, "NULL argument");
  if (misaligned(d_group, 4)) return fail(SNK_EINVAL, "d_group must be 4-byte aligned");
  if (misaligned(d_work, 16)) return fail(SNK_EINVAL, "d_work must be 16-byte aligned");
  if (misaligned(d_counts, 8) || misaligned(d_envs_done, 8)) return fail(SNK_EINVAL, "d_counts and d_envs_done must be 8-byte aligned");
  if (!h) return fail(SNK_EINVAL, "handle is NULL");
  CUDA_TRY(cudaSetDevice(h->cfg.device));
  const Params& p = h->p;
  size_t off[4];
  tally_work_bytes(p.N, p.S, off);
  uint8_t* w = (uint8_t*)d_work;
  TallyArgs a;
  a.reward_all = p.reward_all; a.done = p.done; a.ep_len = p.fin_len; a.group = d_group;
  a.t = (int32_t*)(w + off[0]); a.episodes = (int32_t*)(w + off[1]); a.death = (int32_t*)(w + off[2]); a.fruits = (int32_t*)(w + off[3]);
  a.counts = d_counts; a.envs_done = d_envs_done; a.err = p.err;
  a.N = p.N; a.S = p.S; a.n_groups = n_groups; a.episodes_per_env = episodes_per_env;
  CUDA_TRY(snk_launch_tally(a, (cudaStream_t)stream));
  h->launches++;
  return SNK_OK;
}

// rollout search bookkeeping (snk_search.cu): slots j < n_roots * n_actions * rollouts of the handle
static int search_check(const snk_handle* h, int32_t seat, int32_t n_actions, int32_t rollouts, int64_t n_roots, const void* d_ret) {
  if (!h) return fail(SNK_EINVAL, "handle is NULL");
  if (!d_ret) return fail(SNK_EINVAL, "NULL argument");
  if (seat < 0 || seat >= h->p.S) return fail(SNK_EINVAL, "seat %d outside [0, %d)", seat, h->p.S);
  if (n_actions < 1 || n_actions > 127) return fail(SNK_EINVAL, "n_actions must be 1..127, got %d", n_actions);
  if (rollouts < 1) return fail(SNK_EINVAL, "rollouts must be >= 1, got %d", rollouts);
  if (n_roots < 1 || n_roots * n_actions * rollouts > h->p.N)
    return fail(SNK_EINVAL, "n_roots %lld x %d actions x %d rollouts outside [1, num_envs = %lld]", (long long)n_roots, n_actions,
                rollouts, h->p.N);
  if (misaligned(d_ret, 4)) return fail(SNK_EINVAL, "d_ret must be 4-byte aligned");
  return SNK_OK;
}

static SearchArgs search_args(const snk_handle* h, int32_t seat, int32_t n_actions, int32_t rollouts, int64_t n_roots,
                              int32_t* d_ret, uint8_t* d_active) {
  SearchArgs a;
  a.reward_all = h->p.reward_all; a.done = h->p.done; a.ret = d_ret; a.active = d_active;
  a.S = h->p.S; a.seat = seat; a.n_actions = n_actions; a.rollouts = rollouts; a.n_roots = n_roots;
  return a;
}

extern "C" int snk_search_begin(snk_handle* h, int8_t* d_actions, int32_t seat, int32_t n_actions, int32_t rollouts, int64_t n_roots,
                                int32_t* d_ret, uint8_t* d_active, void* stream) {
  int rc = search_check(h, seat, n_actions, rollouts, n_roots, d_ret);
  if (rc) return rc;
  if (!d_actions || !d_active) return fail(SNK_EINVAL, "NULL argument");
  CUDA_TRY(cudaSetDevice(h->cfg.device));
  CUDA_TRY(snk_launch_search_begin(search_args(h, seat, n_actions, rollouts, n_roots, d_ret, d_active), d_actions, (cudaStream_t)stream));
  h->launches++;
  return SNK_OK;
}

extern "C" int snk_search_accumulate(snk_handle* h, int32_t seat, int32_t n_actions, int32_t rollouts, int64_t n_roots, int32_t* d_ret,
                                     uint8_t* d_active, void* stream) {
  int rc = search_check(h, seat, n_actions, rollouts, n_roots, d_ret);
  if (rc) return rc;
  if (!d_active) return fail(SNK_EINVAL, "NULL argument");
  CUDA_TRY(cudaSetDevice(h->cfg.device));
  CUDA_TRY(snk_launch_search_accumulate(search_args(h, seat, n_actions, rollouts, n_roots, d_ret, d_active), (cudaStream_t)stream));
  h->launches++;
  return SNK_OK;
}

extern "C" int snk_search_pick(snk_handle* h, int32_t n_actions, int32_t rollouts, int64_t n_roots, const int32_t* d_ret,
                               float* d_value, int8_t* d_pick, int64_t pick_stride, void* stream) {
  int rc = search_check(h, 0, n_actions, rollouts, n_roots, d_ret);
  if (rc) return rc;
  if (!d_value || !d_pick) return fail(SNK_EINVAL, "NULL argument");
  if (pick_stride < 1) return fail(SNK_EINVAL, "pick_stride must be >= 1, got %lld", (long long)pick_stride);
  if (misaligned(d_value, 4)) return fail(SNK_EINVAL, "d_value must be 4-byte aligned");
  CUDA_TRY(cudaSetDevice(h->cfg.device));
  SearchArgs a = search_args(h, 0, n_actions, rollouts, n_roots, (int32_t*)d_ret, nullptr);
  CUDA_TRY(snk_launch_search_pick(a, d_value, d_pick, pick_stride, (cudaStream_t)stream));
  h->launches++;
  return SNK_OK;
}

extern "C" int snk_grid_conv_in(const uint8_t* d_grid, int64_t n, int32_t size, int32_t view, const float* d_table,
                                const float* d_bias, int32_t channels, float* d_out, int32_t device, void* stream) {
  int rc = grid_conv_check(n, size, view, channels);
  if (rc) return rc;
  if (n == 0) return SNK_OK;
  if (!d_grid || !d_table || !d_bias || !d_out) return fail(SNK_EINVAL, "NULL argument");
  if (misaligned(d_table, 16) || misaligned(d_bias, 16) || misaligned(d_out, 16))
    return fail(SNK_EINVAL, "d_table, d_bias and d_out must be 16-byte aligned");
  CUDA_TRY(cudaSetDevice(device));
  const long long V = size + 2;
  CUDA_TRY(snk_launch_grid_conv_in(d_grid, n * V * V, (int)V, view, d_table, d_bias, d_out, (cudaStream_t)stream));
  return SNK_OK;
}

extern "C" int snk_grid_conv_in_wgrad(const uint8_t* d_grid, int64_t n, int32_t size, int32_t view, const float* d_out,
                                      const float* d_gout, int32_t channels, float* d_hist, void* d_work, size_t work_bytes,
                                      int32_t device, void* stream) {
  int rc = grid_conv_check(n, size, view, channels);
  if (rc) return rc;
  if (n == 0) return SNK_OK;
  if (!d_grid || !d_out || !d_gout || !d_hist || !d_work) return fail(SNK_EINVAL, "NULL argument");
  if (misaligned(d_out, 4) || misaligned(d_gout, 4) || misaligned(d_hist, 4) || misaligned(d_work, 4))
    return fail(SNK_EINVAL, "d_out, d_gout, d_hist and d_work must be 4-byte aligned");
  const long long V = size + 2, n_cells = n * V * V;
  if (work_bytes < SNK_GRID_CONV_WORK_BYTES(n_cells))
    return fail(SNK_EINVAL, "workspace too small: %zu < %zu bytes", work_bytes, (size_t)SNK_GRID_CONV_WORK_BYTES(n_cells));
  CUDA_TRY(cudaSetDevice(device));
  CUDA_TRY(snk_launch_grid_conv_in_wgrad(d_grid, n_cells, (int)V, view, d_out, d_gout, d_hist, (float*)d_work,
                                         (cudaStream_t)stream));
  return SNK_OK;
}

extern "C" int snk_grid_conv84_geometry(int32_t size, int64_t n, int64_t* out) {
  GridConv84Geometry g;
  if (!out) return fail(SNK_EINVAL, "out is NULL");
  if (n < 0) return fail(SNK_EINVAL, "n must be >= 0, got %lld", (long long)n);
  if (size < 1 || size > 40 || !snk_grid_conv84_geometry_of(size + 2, n, g))
    return fail(SNK_EINVAL, "size %d: V = size + 2 must divide 84 with 3 <= V <= 42", size);
  out[0] = g.f; out[1] = g.P; out[2] = g.C; out[3] = (int64_t)g.work_bytes;
  return SNK_OK;
}

static int grid_conv84_check(int64_t n, int32_t size, int32_t view, int32_t channels, GridConv84Geometry& g) {
  if (channels != SNK_GRID_CONV_CHANNELS)
    return fail(SNK_EINVAL, "channels must be %d, got %d", SNK_GRID_CONV_CHANNELS, channels);
  if (view < 0 || view > 31) return fail(SNK_EINVAL, "view must be 0..31, got %d", view);
  if (n < 0) return fail(SNK_EINVAL, "n must be >= 0, got %lld", (long long)n);
  if (size < 1 || size > 40 || !snk_grid_conv84_geometry_of(size + 2, n, g))
    return fail(SNK_EINVAL, "size %d: V = size + 2 must divide 84 with 3 <= V <= 42", size);
  return SNK_OK;
}

extern "C" int snk_grid_conv84_in(const uint8_t* d_grid, int64_t n, int32_t size, int32_t view, const float* d_table,
                                  const float* d_bias, int32_t channels, float* d_out, int32_t device, void* stream) {
  GridConv84Geometry g;
  int rc = grid_conv84_check(n, size, view, channels, g);
  if (rc) return rc;
  if (n == 0) return SNK_OK;
  if (!d_grid || !d_table || !d_bias || !d_out) return fail(SNK_EINVAL, "NULL argument");
  if (misaligned(d_table, 16) || misaligned(d_bias, 16) || misaligned(d_out, 16))
    return fail(SNK_EINVAL, "d_table, d_bias and d_out must be 16-byte aligned");
  CUDA_TRY(cudaSetDevice(device));
  CUDA_TRY(snk_launch_grid_conv84_in(d_grid, n, size + 2, view, d_table, d_bias, d_out, (cudaStream_t)stream));
  return SNK_OK;
}

extern "C" int snk_grid_conv84_in_wgrad(const uint8_t* d_grid, int64_t n, int32_t size, int32_t view, const float* d_out,
                                        const float* d_gout, int32_t channels, float* d_hist, void* d_work, size_t work_bytes,
                                        int32_t device, void* stream) {
  GridConv84Geometry g;
  int rc = grid_conv84_check(n, size, view, channels, g);
  if (rc) return rc;
  if (n == 0) return SNK_OK;
  if (!d_grid || !d_out || !d_gout || !d_hist || !d_work) return fail(SNK_EINVAL, "NULL argument");
  if (misaligned(d_out, 4) || misaligned(d_gout, 4) || misaligned(d_hist, 4) || misaligned(d_work, 4))
    return fail(SNK_EINVAL, "d_out, d_gout, d_hist and d_work must be 4-byte aligned");
  if (work_bytes < g.work_bytes) return fail(SNK_EINVAL, "workspace too small: %zu < %zu bytes", work_bytes, g.work_bytes);
  CUDA_TRY(cudaSetDevice(device));
  CUDA_TRY(snk_launch_grid_conv84_in_wgrad(d_grid, n, size + 2, view, d_out, d_gout, d_hist, (float*)d_work,
                                           (cudaStream_t)stream));
  return SNK_OK;
}

extern "C" int snk_algorithmic_bytes_per_step(const snk_config* c, double mean_sum_len, double* out) {
  int rc = cfg_check(c);
  if (rc) return rc;
  if (!out) return fail(SNK_EINVAL, "out is NULL");
  const double V = c->size + 2.0, S = c->n_snakes, F = c->n_fruits, K = c->n_views ? c->n_views : c->n_snakes;
  const double side = c->obs_mode == SNK_OBS_ATARI84 ? 84.0 : V, obs = c->obs_mode == SNK_OBS_GRID ? V * V : K * side * side * 3.0;
  *out = obs + 19.0 * S + 2.0 * mean_sum_len + 2.0 * F + 30.0;  // SURVEY.md section 8d
  return SNK_OK;
}

extern "C" int snk_launch_count(const snk_handle* h, uint64_t* out) {
  if (!h || !out) return fail(SNK_EINVAL, "NULL argument");
  *out = h->launches;
  return SNK_OK;
}

// include/snk.h's numbers for each form: snk_launch_info's kind (0 lane, 1 tile, 2 dense, 3 rows) and snk_launch_form's
// code (0 fused, 1 warp-specialised, 3 two kernels, -1 not the lane family)
static const struct { int32_t kind, code; } kFormCodes[FORM_COUNT] = {
    {0, 0}, {0, 1}, {0, 3}, {0, 3}, {1, -1}, {2, -1}, {3, -1}, {3, -1}};

extern "C" int snk_launch_form(const snk_handle* h, int32_t* out /*[4]*/) {
  if (!h || !out) return fail(SNK_EINVAL, "NULL argument");
  const LaunchPlan& pl = (h->have_alt && h->use_alt) ? h->plan_alt : h->plan;
  out[0] = kFormCodes[pl.form].code;
  out[1] = h->p.family ? h->p.EPW : 0; out[2] = h->p.family ? h->p.TE : 0; out[3] = h->have_alt ? 1 : 0;
  return SNK_OK;
}

extern "C" int snk_launch_info(const snk_handle* h, int32_t* out /*[6]: kind, grid, block, smem, occupancy, envs per CTA*/) {
  if (!h || !out) return fail(SNK_EINVAL, "NULL argument");
  const LaunchPlan& pl = (h->have_alt && h->use_alt) ? h->plan_alt : h->plan;
  out[0] = kFormCodes[pl.form].kind; out[1] = pl.grid; out[2] = pl.block; out[3] = (int32_t)pl.smem; out[4] = pl.occupancy; out[5] = pl.envs_per_cta;
  return SNK_OK;
}
