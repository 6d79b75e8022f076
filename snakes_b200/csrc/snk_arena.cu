// snk_arena.cu -- per-seat match accounting behind the step kernels (snk_tally; DESIGN.md section 4.18).
//
// One thread per env, launched after every step on the step's stream.  It reads only the step's outputs (reward_all,
// done, episode_len), so it serves every step family, rule-set and S = 1..32.  A seat's reward is -1 on the step it
// dies, 0 on every later step and otherwise the fruits it ate, so the running values of an episode are, per seat, the
// step of its death (0 = alive) and its fruits, plus the env's step counter.  On done the finished episode becomes
// outcomes (snk.h: the unique longest survivor wins, seats tied for longest draw) added to int64 counters
// [n_groups][S][SNK_TALLY_FIELDS]; the step has already auto-reset the env, so its running values are cleared.
//
// Up to a tenth of the envs finish on one step and, with few groups, every one of them would add into the same
// addresses: each CTA first adds into a shared-memory copy of the counters and then adds its non-zero words into global
// memory.  Integer atomics, so the result is the same bits whatever order they land in.
#include <cuda_runtime.h>
#include <stdint.h>

#include "snk_launch.h"

typedef unsigned long long u64;

static constexpr int TALLY_THREADS = 256;
static constexpr int TALLY_SHARED_WORDS = 48 * 1024 / 8;  // counters kept in shared memory up to the default 48 KB

// SHARED: the CTA's counters live in shared memory (shared_words of them) and are added to global memory at the end;
// otherwise (more counters than fit) every outcome is added to global memory directly
template <bool SHARED>
__global__ void __launch_bounds__(TALLY_THREADS) k_tally(const TallyArgs a, int shared_words) {
  extern __shared__ u64 s_acc[];
  u64* acc = SHARED ? s_acc : (u64*)a.counts;
  if (SHARED) {
    for (int i = threadIdx.x; i < shared_words; i += TALLY_THREADS) s_acc[i] = 0;
    __syncthreads();
  }
  const long long e = (long long)blockIdx.x * TALLY_THREADS + threadIdx.x;
  const int S = a.S;
  bool finished = false, counted = false;
  if (e < a.N) {
    // the loads every env makes are issued together: the kernel is bound by their latency, not by its 2-3 MB
    int t = a.t[e];
    const bool done = a.done[e];
    const int g = a.group[e], L = a.ep_len[e];
    const float r0 = a.reward_all[e * S];
    if (t >= 0) {  // -1: the env has counted episodes_per_env episodes
      t += 1;
      const float* r = a.reward_all + e * S;
      int32_t* death = a.death + e * S;
      int32_t* fruits = a.fruits + e * S;
      for (int s = 0; s < S; ++s) {
        const float v = s ? r[s] : r0;
        if (v < 0.f) death[s] = t;
        else if (v > 0.f) fruits[s] += (int32_t)v;
      }
      if (done) {
        if (g < 0 || g >= a.n_groups) {
          atomicOr(a.err, (unsigned)SNK_DEVERR_BAD_STATE);
          t = -1;  // skipped: never counted, never finished
        } else {
          int last = 0, n_last = 0;  // the latest death step (INT_MAX: alive at the end) and how many seats share it
          for (int s = 0; s < S; ++s) {
            const int d = death[s] ? death[s] : 0x7fffffff;
            if (d > last) { last = d; n_last = 1; }
            else if (d == last) ++n_last;
          }
          u64* c = acc + (size_t)g * S * SNK_TALLY_FIELDS;
          for (int s = 0; s < S; ++s, c += SNK_TALLY_FIELDS) {
            const int d = death[s], f = fruits[s];
            const bool top = (d ? d : 0x7fffffff) == last;
            atomicAdd(c + (!top ? SNK_TALLY_LOSSES : n_last == 1 ? SNK_TALLY_WINS : SNK_TALLY_DRAWS), 1ull);
            const long long ret = (long long)f - (d ? 1 : 0);
            if (f) atomicAdd(c + SNK_TALLY_FRUITS, (u64)f);
            if (d) atomicAdd(c + SNK_TALLY_DEATHS, 1ull);
            atomicAdd(c + SNK_TALLY_STEPS_ALIVE, (u64)(d ? d : L));
            if (ret) atomicAdd(c + SNK_TALLY_RETURN_SQ, (u64)(ret * ret));
            atomicAdd(c + SNK_TALLY_LENGTH, (u64)L);
            death[s] = 0;
            fruits[s] = 0;
          }
          counted = true;
          const int n = a.episodes[e] + 1;
          a.episodes[e] = n;
          finished = n >= a.episodes_per_env;
          t = finished ? -1 : 0;
        }
      }
      a.t[e] = t;
    }
  }
  const unsigned fin = __ballot_sync(0xffffffffu, finished);
  if (fin && (threadIdx.x & 31) == 0) atomicAdd((u64*)a.envs_done, (u64)__popc(fin));
  if (SHARED && __syncthreads_or(counted)) {
    for (int i = threadIdx.x; i < shared_words; i += TALLY_THREADS) {
      const u64 v = s_acc[i];
      if (v) atomicAdd((u64*)a.counts + i, v);
    }
  }
}

cudaError_t snk_launch_tally(const TallyArgs& a, cudaStream_t stream) {
  const long long words = (long long)a.n_groups * a.S * SNK_TALLY_FIELDS;
  const unsigned blocks = (unsigned)((a.N + TALLY_THREADS - 1) / TALLY_THREADS);
  if (words <= TALLY_SHARED_WORDS)
    k_tally<true><<<blocks, TALLY_THREADS, (size_t)words * 8, stream>>>(a, (int)words);
  else
    k_tally<false><<<blocks, TALLY_THREADS, 0, stream>>>(a, 0);
  return cudaGetLastError();
}
