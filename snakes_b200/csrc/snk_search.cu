// snk_search.cu -- the bookkeeping of a rollout search behind the step kernels (snk_search_*; DESIGN.md section 4.19).
//
// A search handle holds n_roots x n_actions x rollouts slots, slot j = (m * n_actions + a) * rollouts + r a clone of root
// m that plays candidate action a with seat `seat` on its first step and then follows a rollout policy.  Three kernels,
// one thread per slot (per root for pick), stream-ordered on the step's stream, no allocation, no synchronisation:
//   begin       before the first step: seat's action of slot j <- a, return <- 0, active <- 1
//   accumulate  after every step: an active slot adds seat's reward; the step where the seat gets -1 (it died, the
//               death rule of snk_tally) or where the env is done is its last counted step
//   pick        V[m][a] = sum of the returns of the slot's rollouts; the lowest a of maximal V is the root's action
// Rewards are integers, so every return and every V is exact whatever order the sums run in.
#include <cuda_runtime.h>
#include <stdint.h>

#include "snk_launch.h"

static constexpr int SEARCH_THREADS = 256;

__global__ void __launch_bounds__(SEARCH_THREADS) k_search_begin(const SearchArgs a, int8_t* actions, long long slots) {
  const long long j = (long long)blockIdx.x * SEARCH_THREADS + threadIdx.x;
  if (j >= slots) return;
  actions[j * a.S + a.seat] = (int8_t)((j / a.rollouts) % a.n_actions);
  a.ret[j] = 0;
  a.active[j] = 1;
}

__global__ void __launch_bounds__(SEARCH_THREADS) k_search_accumulate(const SearchArgs a, long long slots) {
  const long long j = (long long)blockIdx.x * SEARCH_THREADS + threadIdx.x;
  if (j >= slots || !a.active[j]) return;
  const float v = a.reward_all[j * a.S + a.seat];
  a.ret[j] += (int32_t)v;
  if (v < 0.f || a.done[j]) a.active[j] = 0;
}

__global__ void __launch_bounds__(SEARCH_THREADS) k_search_pick(const SearchArgs a, float* value, int8_t* pick, long long pick_stride) {
  const long long m = (long long)blockIdx.x * SEARCH_THREADS + threadIdx.x;
  if (m >= a.n_roots) return;
  const int32_t* r = a.ret + m * a.n_actions * a.rollouts;
  long long best = 0;
  int best_a = 0;
  for (int c = 0; c < a.n_actions; ++c, r += a.rollouts) {
    long long v = 0;
    for (int k = 0; k < a.rollouts; ++k) v += r[k];
    value[m * a.n_actions + c] = (float)v;
    if (c == 0 || v > best) { best = v; best_a = c; }
  }
  pick[m * pick_stride] = (int8_t)best_a;
}

static unsigned blocks_of(long long n) { return (unsigned)((n + SEARCH_THREADS - 1) / SEARCH_THREADS); }

cudaError_t snk_launch_search_begin(const SearchArgs& a, int8_t* actions, cudaStream_t stream) {
  const long long slots = a.n_roots * a.n_actions * a.rollouts;
  k_search_begin<<<blocks_of(slots), SEARCH_THREADS, 0, stream>>>(a, actions, slots);
  return cudaGetLastError();
}

cudaError_t snk_launch_search_accumulate(const SearchArgs& a, cudaStream_t stream) {
  const long long slots = a.n_roots * a.n_actions * a.rollouts;
  k_search_accumulate<<<blocks_of(slots), SEARCH_THREADS, 0, stream>>>(a, slots);
  return cudaGetLastError();
}

cudaError_t snk_launch_search_pick(const SearchArgs& a, float* value, int8_t* pick, long long pick_stride, cudaStream_t stream) {
  k_search_pick<<<blocks_of(a.n_roots), SEARCH_THREADS, 0, stream>>>(a, value, pick, pick_stride);
  return cudaGetLastError();
}
