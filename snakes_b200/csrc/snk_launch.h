// snk_launch.h -- host-visible launch interface between snk_api.cu and snk_kernels.cu.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>

#include "../../include/snk.h"

struct Params;
struct PeerArgs;
// k_step_lane_ws: paint warps (each owning a shared-memory image) and logic warps per CTA
enum { WS_PAINT_WARPS = 2, WS_LOGIC_WARPS = 3 };

// The kernel sequences a step runs.  snk_api.cu's plan_launch picks one; resolve<RULES> in snk_kernels.cu is the only code
// that names their kernels.  The lane family keeps bodies chain-coded with a lane per env; the others keep ring bodies.
enum Form {
  FORM_LANE,        // k_step_lane: a warp steps its batch, then streams its images
  FORM_LANE_WS,     // k_step_lane_ws: paint warps + logic warps per CTA
  FORM_LANE_SPLIT,  // k_lane_logic (thread per env) + k_lane_paint2 (observation writer)
  FORM_LANE_GRID,   // SNK_OBS_GRID: k_lane_logic + k_lane_grid
  FORM_TILE,        // k_step_tile, warp per env, instantiated for 256 and 512 threads (chosen by the block)
  FORM_DENSE,       // k_step_dense, CTA per env
  FORM_ROWS,        // k_step_rows<RULES, false>, CTA per env
  FORM_ROWS_GRID,   // SNK_OBS_GRID: k_step_rows<RULES, true>
  FORM_COUNT
};

struct LaunchPlan {
  int form;
  const void* logic;   // k_lane_logic<S, RULES>, launched before `kernel` except in MODE_OBSERVE; NULL for one-kernel forms
  const void* kernel;  // the step kernel, or the observation writer behind `logic`
  bool pdl;            // programmatic stream serialization for `logic` and `kernel`
  int grid, block;
  size_t smem;
  int occupancy;       // resident CTAs per SM
  int max_grid;        // SMs * occupancy: persistent grid size
  int envs_per_cta;
  int restore_thr;     // Params::restore_thr under this plan
};

// Resolves plan.form (and plan.block) to its kernels, sets their shared-memory limit, and fills pdl, occupancy, max_grid
// and grid = work clamped to [1, max_grid].  cudaErrorInvalidConfiguration: no kernel for this form, S and K.
cudaError_t snk_plan(int rules, LaunchPlan& plan, int n_sm, int S, int K, long long work);
bool snk_lane_supported(int S, int K);
cudaError_t snk_launch_step(const Params& p, const LaunchPlan& plan, cudaStream_t stream);
cudaError_t snk_launch_upscale84(const uint8_t* native, uint8_t* out, long long N, int V, int C, int n_sm, cudaStream_t stream);
// env state (k_save_envs / k_restore_envs / k_copy_envs): entry j is env idx[j], or env first + j when idx is NULL
cudaError_t snk_launch_save(const Params& p, const int64_t* idx, long long first, long long count, uint8_t* blob,
                            const snk_state_layout& lay, cudaStream_t stream);
cudaError_t snk_launch_restore(const Params& p, const int64_t* idx, long long count, const uint8_t* blob, const snk_state_layout& lay,
                               cudaStream_t stream);
// k_copy_envs: env src[j] of `ps` -> env dst[j] of `pd` (one handle, or two of the same private layout)
cudaError_t snk_launch_copy(const Params& ps, const Params& pd, const int64_t* src, const int64_t* dst, long long count,
                            cudaStream_t stream);
cudaError_t snk_launch_sum_inbox(const PeerArgs& a, const double* stats, double* glob, cudaStream_t stream);
cudaError_t snk_launch_expand_views(const uint8_t* grid, long long n_cells, int first_view, int n_views, uint8_t* out, cudaStream_t stream);
// snk_grid_conv.cu: the grid's first convolution layer (n_cells = n * V * V) and the CTA count of its weight gradient
cudaError_t snk_launch_grid_conv_in(const uint8_t* grid, long long n_cells, int V, int view, const float* table,
                                    const float* bias, float* out, cudaStream_t stream);
cudaError_t snk_launch_grid_conv_in_wgrad(const uint8_t* grid, long long n_cells, int V, int view, const float* out,
                                          const float* gout, float* hist, float* work, cudaStream_t stream);
int snk_grid_conv_wgrad_ctas(long long n_cells);
// snk_grid_conv84.cu: nature_cnn's first layer on the WarpFrame view of a grid (n grids of V x V).  Geometry: f, P, C of
// include/snk.h, K weight-gradient CTAs per phase pair and the workspace; false for an unsupported V or n < 0.
struct GridConv84Geometry {
  int f, P, C, K;
  size_t work_bytes;
};
bool snk_grid_conv84_geometry_of(int V, long long n, GridConv84Geometry& g);
cudaError_t snk_launch_grid_conv84_in(const uint8_t* grid, long long n, int V, int view, const float* table, const float* bias,
                                      float* out, cudaStream_t stream);
cudaError_t snk_launch_grid_conv84_in_wgrad(const uint8_t* grid, long long n, int V, int view, const float* out, const float* gout,
                                            float* hist, float* work, cudaStream_t stream);
cudaError_t snk_launch_extract_views(const uint8_t* src, uint8_t* dst, long long n_pixels, int C, int n_out, cudaStream_t stream);
cudaError_t snk_launch_scripted_actions(const Params& p, int8_t* actions, uint64_t step, uint64_t seed, int eps_permille,
                                        const uint8_t* occ_obs, cudaStream_t stream);
cudaError_t snk_launch_gae(const float* rewards, const float* values, const uint8_t* dones, const float* last_values,
                           const uint8_t* last_dones, double gamma, double lam, int T, long long N, float* advs, float* returns,
                           cudaStream_t stream);
cudaError_t snk_launch_gen_actions(int8_t* actions, long long N, int S, long long env_id_base, uint64_t step,
                                   uint64_t seed, int n_actions, cudaStream_t stream);
// snk_arena.cu: per-seat match accounting after a step (snk_tally).  The work area of include/snk.h split into its parts.
struct TallyArgs {
  const float* reward_all;  // [N][S] the handle's per-step outputs
  const uint8_t* done;
  const int32_t* ep_len;
  const int32_t* group;     // [N]
  int32_t* t;               // [N] step within the running episode, -1 once the env has counted episodes_per_env episodes
  int32_t* episodes;        // [N] episodes counted
  int32_t* death;           // [N][S] step of the seat's death in the running episode, 0 = alive
  int32_t* fruits;          // [N][S] fruits of the running episode
  int64_t* counts;          // [n_groups][S][SNK_TALLY_FIELDS]
  int64_t* envs_done;
  uint32_t* err;
  long long N;
  int S, n_groups, episodes_per_env;
};
cudaError_t snk_launch_tally(const TallyArgs& a, cudaStream_t stream);
// snk_search.cu: rollout-search bookkeeping (snk_search_begin / _accumulate / _pick).  Slot j < n_roots * n_actions *
// rollouts of the search handle is root j / (n_actions * rollouts), candidate action (j / rollouts) % n_actions.
struct SearchArgs {
  const float* reward_all;  // [N][S] the search handle's per-step outputs
  const uint8_t* done;      // [N]
  int32_t* ret;             // [slots] return of `seat` over the counted steps
  uint8_t* active;          // [slots] 1 until the slot's last counted step has been added
  int S, seat, n_actions, rollouts;
  long long n_roots;
};
cudaError_t snk_launch_search_begin(const SearchArgs& a, int8_t* actions, cudaStream_t stream);
cudaError_t snk_launch_search_accumulate(const SearchArgs& a, cudaStream_t stream);
cudaError_t snk_launch_search_pick(const SearchArgs& a, float* value, int8_t* pick, long long pick_stride, cudaStream_t stream);
