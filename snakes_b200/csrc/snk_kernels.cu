// snk_kernels.cu -- the fused env-step kernels (sm_100a) and their launchers.
//
// k_step_tile  : one WARP per env, W consecutive envs per CTA, persistent grid.  The CTA keeps a
//                shared-memory image of its W observations; each iteration restores it from a
//                border-only template, the warps paint the few non-background cells of their env,
//                and ONE thread hands the whole image to the TMA engine
//                (cp.async.bulk.global.shared::cta) which streams it to HBM while the warps are
//                already stepping the next group.  SM issue slots go to game logic, not to stores.
// k_step_dense : one CTA per env for boards whose observation does not fit the tile scheme
//                (e.g. 16 snakes on 64x64: 209 KB per env); same logic, cell-code grid in shared
//                memory, dense colour mapping with coalesced stores.
// Both fuse: action decode, head advance, eating + respawn, simultaneous collision test, body
// clearing, reward / done, Monitor accounting, in-place auto-reset and the RGB encoding of
// all K views (reference: gym_snake/envs/snake_multiple_test.py:166-197 + :35-58 + :93-95).
#include "snk_device.cuh"
#include "snk_lane.cuh"
#include "snk_launch.h"

// ------------------------------------------------------------------ TMA bulk-copy wrappers
__device__ __forceinline__ void bulk_store_s2g(void* gdst, const void* ssrc, u32 bytes) {
  const u32 s = (u32)__cvta_generic_to_shared(ssrc);
  const u64 g = (u64)__cvta_generic_to_global(gdst);
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(g), "r"(s), "r"(bytes) : "memory");
}
// same, with an L2 evict-first policy: the observation stream is write-once and larger than L2, so
// it should not push the (re-read every step) env records out of the cache
__device__ __forceinline__ u64 l2_evict_first_policy() {
  u64 pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ void bulk_store_s2g_hint(void* gdst, const void* ssrc, u32 bytes, u64 pol) {
  const u32 s = (u32)__cvta_generic_to_shared(ssrc);
  const u64 g = (u64)__cvta_generic_to_global(gdst);
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;" ::"l"(g), "r"(s), "r"(bytes), "l"(pol)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
// global -> shared bulk copy completing on an mbarrier (used once per warp to fetch the border image)
__device__ __forceinline__ void mbar_init(u64* bar, u32 count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"((u32)__cvta_generic_to_shared(bar)), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(u64* bar, u32 bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"((u32)__cvta_generic_to_shared(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_load_g2s(void* sdst, const void* gsrc, u32 bytes, u64* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   (u32)__cvta_generic_to_shared(sdst)),
               "l"((u64)__cvta_generic_to_global(gsrc)), "r"(bytes), "r"((u32)__cvta_generic_to_shared(bar))
               : "memory");
}
__device__ __forceinline__ void mbar_wait(u64* bar, u32 parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tWAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE_%=;\n\tbra WAIT_%=;\n\tDONE_%=:\n\t}" ::"r"((u32)__cvta_generic_to_shared(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void flush_stats(const Params& p, const WarpStats& st, u32 errs, double* s_stats, int lane) {
  if (lane == 0) {
    atomicAdd(&s_stats[SNK_STAT_ENV_STEPS], (double)st.steps);
    atomicAdd(&s_stats[SNK_STAT_EPISODES], (double)st.episodes);
    atomicAdd(&s_stats[SNK_STAT_RETURN_SUM], (double)st.ret_sum);
    atomicAdd(&s_stats[SNK_STAT_LENGTH_SUM], (double)st.len_sum);
    atomicAdd(&s_stats[SNK_STAT_FRUITS], (double)st.fruits);
    atomicAdd(&s_stats[SNK_STAT_DEATHS], (double)st.deaths);
    atomicAdd(&s_stats[SNK_STAT_BODY_CELLS], (double)st.cells);
    atomicAdd(&s_stats[SNK_STAT_DRAWS], (double)st.draws);
    if (errs) atomicOr(p.err, errs);
  }
}

// The path's one inter-GPU exchange, fused into the step kernel and free of any rendezvous (snk_peer_connect).
// Every statistic is a monotonic running sum, and an aligned 8-byte store is one transaction on NVLink, so the exchange
// needs neither fences nor versions: at the START of step t + 1 eight threads of the first CTA read the rank's sums --
// complete as of step t, the launch has just waited for the previous grid -- and store each into this rank's slot of
// every peer's inbox (cudaIpc-mapped peer memory).  The stores are posted and drain while the CTA goes on to step its
// envs: nothing waits for them, no collective kernel runs beside the step, no rank ever waits for another.  A reader sums
// its own running sums and the eight-byte values the peers last pushed: the global statistics as of about one step ago
// (monitor.py:57-78 aggregated over all shards; SURVEY.md section 8e), exact once every rank has pushed its final sums
// (snk_get_stats_global does that push).
__device__ __forceinline__ void peer_push(const Params& p, int tid) {
  // the same moment serves the host's choice between the fused and the two-kernel form of the lane path (snk_api.cu,
  // regime_update): running env-steps and body cells as of the previous step, two posted 8-byte stores into mapped host
  // memory, read there without any synchronisation
  if (p.regime_out && blockIdx.x == 0 && tid < 2 && p.mode == MODE_STEP)
    reinterpret_cast<volatile double*>(p.regime_out)[tid] = __ldcg(&p.stats[tid ? SNK_STAT_BODY_CELLS : SNK_STAT_ENV_STEPS]);
  if (p.peer.ranks > 1 && blockIdx.x == 0 && tid < SNK_NSTATS && p.mode == MODE_STEP) {
    const double v = __ldcg(&p.stats[tid]);
    for (int g = 0; g < p.peer.ranks; ++g)
      if (g != p.peer.rank) reinterpret_cast<volatile double*>(p.peer.inbox[g] + (size_t)p.peer.rank * SNK_INBOX_STRIDE)[tid] = v;
  }
}

// End of every step kernel: the CTA's sums go to the handle's running statistics.  In the NCCL form of the per-step
// reduction (snk_comm_init: Params::snap set) the LAST CTA to arrive also copies the vector into the snapshot slot of
// this step, which a side stream hands to ncclAllReduce beside the next step.  (The peer-memory form pushes at the START
// of the next step instead, peer_push: anything done here, at the very end of a launch, sits on the critical path --
// a fenced push from the last CTA was measured at 7.5 us per step, because the next launch waits for this grid.)
__device__ __forceinline__ void publish_stats(const Params& p, const double* s_stats, int tid) {
  __shared__ int s_last;
  __syncthreads();
  if (tid < SNK_NSTATS && s_stats[tid] != 0.0) atomicAdd(&p.stats[tid], s_stats[tid]);
  if (p.snap) {
    __threadfence();
    __syncthreads();
    if (tid == 0) s_last = atomicAdd(p.ticket, 1u) == gridDim.x - 1;
    __syncthreads();
    if (s_last) {
      __threadfence();
      if (tid < SNK_NSTATS) p.snap[tid] = __ldcg(&p.stats[tid]);
      if (tid == 0) *p.ticket = 0;
    }
  }
}

template <int RULES>
__device__ __forceinline__ void advance_env(const Params& p, long long e, int lane, u32* sc, u32* bm, u32& errs, WarpStats& st) {
  u16* rings = p.body + e * p.S * p.cap;
  u8* grid = p.grid ? p.grid + e * p.grid_stride : nullptr;
  load_rec(p, e, lane, sc);
  if (p.mode == MODE_STEP) {
    step_env_warp<RULES>(p, e, lane, sc, bm, rings, grid, errs, st);
  } else if (p.mode == MODE_RESET) {
    if (!p.mask || p.mask[e]) reset_env_warp<RULES>(p, e, lane, sc, rings, grid, errs, st);
  }
  __syncwarp();
  if (p.mode != MODE_OBSERVE) store_rec(p, e, lane, sc);
}

// Paint the non-background cells of env e into its slot of the CTA's observation image
// (get_ob_for_snake :35-58): fruits first, then snakes in index order (a later snake overwrites an
// earlier one and any fruit), head over body.  The border is already in the image and is never
// touched: cells outside the board are skipped, which equals the reference painting them and then
// overwriting them with the wall (:52-56).  Interleaved layout: pixel pid, view k at pid*3K + 3k.
template <int RULES>
__device__ __forceinline__ void paint_env(const Params& p, long long e, int lane, const u32* sc, u8* img) {
  const int S = p.S, F = p.F, K = p.K, C = p.C, cap = p.cap;
  if (RULES == SNK_RULES_CLASSIC) {
    const u16* fr = reinterpret_cast<const u16*>(sc + REC_SNAKE0 + 2 * S);
    if (lane < F) {
      u8* px = img + (int)fr[lane] * C;
      for (int k = 0; k < K; ++k) px[3 * k] = 255;  // G and B of the restored image are 0
    }
  } else {
    const u8* grid = p.grid + e * p.grid_stride;
    for (int pid = lane; pid < p.VV; pid += 32) {
      if (grid[pid] && !(__ldg(p.cellinfo + pid) >> 31)) {
        u8* px = img + pid * C;
        for (int k = 0; k < K; ++k) px[3 * k] = 255;
      }
    }
  }
  __syncwarp();
  const u16* rings = p.body + e * S * cap;
  for (int s = 0; s < S; ++s) {
    const u32 a = sc[REC_SNAKE0 + 2 * s];
    const int len = a >> 16, hs = a & 0xffff;
    if (len == 0) continue;
    for (int i = lane; i < len; i += 32) {
      u8* px = img + ring_at(rings + s * cap, hs, i, cap) * C;
      for (int k = 0; k < K; ++k) {
        const u32 rgb = snake_rgb(s == k, i == 0);
        px[3 * k] = (u8)rgb; px[3 * k + 1] = (u8)(rgb >> 8); px[3 * k + 2] = (u8)(rgb >> 16);
      }
    }
    __syncwarp();
  }
}

template <int RULES, int BLOCK>
__global__ void __launch_bounds__(BLOCK) k_step_tile(const Params p) {
  extern __shared__ __align__(128) u8 smem[];
  __shared__ double s_stats[SNK_NSTATS];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nthr = blockDim.x;
  const int W = p.W, E = p.E;
  const int tile_bytes = W * E, tmpl_bytes = p.G * E;  // both multiples of 16
  u8* tile = smem;
  u8* tmpl = smem + tile_bytes;
  u32* sc = reinterpret_cast<u32*>(tmpl + tmpl_bytes) + warp * (p.RW + p.bm_words);
  u32* bm = sc + p.RW;
  if (tid < SNK_NSTATS) s_stats[tid] = 0.0;
  peer_push(p, tid);  // the running sums as of the previous step, to every peer (posted stores)
  {
    const uint4* src = reinterpret_cast<const uint4*>(p.tmpl);
    uint4* dst = reinterpret_cast<uint4*>(tmpl);
    for (int i = tid; i < tmpl_bytes / 16; i += nthr) dst[i] = src[i];
  }
  __syncthreads();
  WarpStats st = {0, 0, 0, 0, 0, 0, 0, 0};
  u32 errs = 0;
  for (long long grp = blockIdx.x; grp < p.n_groups; grp += gridDim.x) {
    const long long e = grp * W + warp;
    const bool valid = e < p.N;
    if (valid) advance_env<RULES>(p, e, lane, sc, bm, errs, st);
    if (tid == 0) bulk_wait_read();  // the TMA engine has finished reading the previous image
    __syncthreads();
    {
      const uint4* src = reinterpret_cast<const uint4*>(tmpl);
      const int n16 = tmpl_bytes / 16;
      for (int c = 0; c < W / p.G; ++c) {
        uint4* dst = reinterpret_cast<uint4*>(tile + c * tmpl_bytes);
        for (int i = tid; i < n16; i += nthr) dst[i] = src[i];
      }
    }
    __syncthreads();
    if (valid) paint_env<RULES>(p, e, lane, sc, tile + warp * E);
    fence_async_smem();  // generic-proxy writes -> visible to the async (TMA) proxy
    __syncthreads();
    u8* gdst = p.obs + grp * (long long)tile_bytes;
    if ((grp + 1) * W <= p.N) {
      if (tid == 0) {
        for (int off = 0; off < tile_bytes; off += 16384)
          bulk_store_s2g(gdst + off, tile + off, (u32)min(16384, tile_bytes - off));
        bulk_commit();
      }
    } else {  // last, partial group: plain stores for the valid envs only
      const int bytes = (int)(p.N - grp * W) * E;
      for (int b = tid; b < bytes; b += nthr) gdst[b] = tile[b];
    }
  }
  if (tid == 0) bulk_wait_all();
  flush_stats(p, st, errs, s_stats, lane);
  publish_stats(p, s_stats, tid);
}


// Stream one painted image (TE envs, 16-byte aligned in HBM) out of shared memory, shared by the `nthr` threads that own
// the buffer.  A whole image goes out as TMA bulk copies issued by thread 0, which then waits until the engine has READ
// the image, so it may be modified; the last, partial image is copied byte by byte by all of them.
constexpr int LANE_BULK = 16384;  // bytes per bulk copy
__device__ __forceinline__ void store_image(const Params& p, const u8* tile, int tile_bytes, long long e0, int tid, int nthr) {
  const long long left = p.N - e0;
  u8* gdst = p.obs + e0 * (long long)p.E;
  if (left >= p.TE) {
    if (tid == 0) {
      const u64 pol = l2_evict_first_policy();
      for (int off = 0; off < tile_bytes; off += LANE_BULK)
        bulk_store_s2g_hint(gdst + off, tile + off, (u32)min(LANE_BULK, tile_bytes - off), pol);
      bulk_commit();
      bulk_wait_read();
    }
  } else {
    const int bytes = (int)left * p.E;
    for (int i = tid; i < bytes; i += nthr) gdst[i] = tile[i];
  }
}

__device__ __forceinline__ void init_border_image(const Params& p, u8* tile, int lane) {
  const uint4* src = reinterpret_cast<const uint4*>(p.tmpl);
  const int n16 = p.G * p.E / 16;
  for (int c = 0; c < p.TE / p.G; ++c) {
    uint4* dst = reinterpret_cast<uint4*>(tile + c * p.G * p.E);
    for (int i = lane; i < n16; i += 32) dst[i] = src[i];
  }
}

__device__ __forceinline__ void reduce_lane_stats(const Params& p, LaneStats st, u32 errs, double* s_stats, int lane) {
#pragma unroll
  for (int o = 16; o; o >>= 1) {
    st.steps += __shfl_xor_sync(FULL, st.steps, o); st.episodes += __shfl_xor_sync(FULL, st.episodes, o);
    st.ret_sum += __shfl_xor_sync(FULL, st.ret_sum, o); st.len_sum += __shfl_xor_sync(FULL, st.len_sum, o);
    st.fruits += __shfl_xor_sync(FULL, st.fruits, o); st.deaths += __shfl_xor_sync(FULL, st.deaths, o);
    st.cells += __shfl_xor_sync(FULL, st.cells, o); st.draws += __shfl_xor_sync(FULL, st.draws, o);
    errs |= __shfl_xor_sync(FULL, errs, o);
  }
  WarpStats ws = {st.steps, st.episodes, st.ret_sum, st.len_sum, st.fruits, st.deaths, st.cells, st.draws};
  flush_stats(p, ws, errs, s_stats, lane);
}

// ---- split form of the lane path: game logic at full occupancy, then the observation writer.
// k_lane_logic: one THREAD per env, no shared-memory image, so many warps per SM hide the HBM
// latency of the record / chain / action loads.
// 7 CTAs per SM (72 registers) for one or two snakes: 131 072 envs are 1 024 CTAs, one wave on 148 x 7 slots where the
// compiler's own 92 registers (5 CTAs per SM) made it two (long bodies: 96.7 -> 92.1 us per step); three and four snakes
// would spill (120-320 bytes) and stay as they are
template <int S, int RULES>
__global__ void __launch_bounds__(128, (S <= 2 ? 7 : 1)) k_lane_logic(const Params p) {
  __shared__ double s_stats[SNK_NSTATS];
  __shared__ u32 s_bm[4][SPAWN_WORDS];  // per warp: scratch of group_spawn
  __shared__ uint2 s_hop[256];          // displacements after 1..4 chain codes of a byte (lane_step<HOP>)
  const int tid = threadIdx.x, lane = tid & 31;
  if (tid < SNK_NSTATS) s_stats[tid] = 0.0;
  build_hop_lut(s_hop, p.V, tid, 128);
  asm volatile("griddepcontrol.wait;" ::: "memory");  // the previous step's observation writer still reads the records
  peer_push(p, tid);  // the running sums as of the previous step, to every peer (posted stores)
  __syncthreads();
  LaneStats st = {0, 0, 0, 0, 0, 0, 0, 0};
  u32 errs = 0;
  const long long e = (long long)blockIdx.x * blockDim.x + tid;
  {
    const bool valid = e < p.N;
    LaneEnv<S> env;
#pragma unroll
    for (int s = 0; s < S; ++s) { env.head[s] = 0; env.len[s] = 0; env.c0[s] = 0; env.grow[s] = 0; env.vel[s] = 0; }
    env.fruit[0] = env.fruit[1] = env.fruit[2] = env.fruit[3] = 0;
    env.spare = 0;
    LaneRng rng;
    rng.have = false; rng.blk = 0;
    const FruitSet grid = fruit_set(p, e);
    LaneRaw<S> raw;
    raw.act = 0;
    if (valid) {
      raw = lane_fetch<S>(p, e, p.mode == MODE_STEP);
      if (RULES == SNK_RULES_CLASSIC && p.delta) delta_prev_store<S>(p, e, raw);  // for the writer's sector store
      lane_unpack<S>(raw, env);
    }
    if (p.mode == MODE_STEP) {
      lane_step<S, RULES, true>(p, e, valid, env, raw.act, rng, grid, s_bm[tid >> 5], errs, st, s_hop);
    } else if (valid && (!p.mask || p.mask[e])) {
      lane_reset<S, RULES>(p, e, env, rng, grid, errs, st.draws);
    }
    if (valid) lane_store<S>(p, e, env);
  }
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");  // the observation writer may start its prologue
  reduce_lane_stats(p, st, errs, s_stats, lane);
  publish_stats(p, s_stats, tid);
}

// k_lane_paint2: the observation writer, TWO warps per image buffer.  The image buffers are what an SM runs out of
// (10 at 2x19x19); with one warp each, every warp would be a serial chain paint -> bulk store -> wait -> un-paint.
// The 64 threads of a CTA share one buffer (LPE = 64/TE lanes per env), which halves the trips of every per-env loop
// (an image takes as long as its longest snake) and the zero-fill of the restore, and doubles the warps that cover each
// other's latencies.  CTA-wide barriers order the phases.  Launched programmatically behind k_lane_logic: the border
// image is fetched before griddepcontrol.wait.
template <int C>
__device__ __forceinline__ void cta_restore(u8* tile, int n16, u8* img, int V, int sub, int LPE, int tid, int NT) {
  constexpr int U = (C & 1) ? 1 : 2, PU = 2 * C / U;
  uint4* t4 = reinterpret_cast<uint4*>(tile);
  const uint4 z = make_uint4(0u, 0u, 0u, 0u);
  for (int i = tid; i < n16; i += NT) t4[i] = z;
  __syncthreads();
  const int RB = V * C;
  const int n_edge = (RB + C) / U;
  u8* bot = img + RB * (V - 1) - C;
  for (int j = sub; j < n_edge; j += LPE) {
    if (U == 2) { *reinterpret_cast<u16*>(img + 2 * j) = 0xffffu; *reinterpret_cast<u16*>(bot + 2 * j) = 0xffffu; }
    else { img[j] = 0xff; bot[j] = 0xff; }
  }
  for (int x = 1 + sub; x <= V - 3; x += LPE) {
    u8* q = img + x * RB + RB - C;
#pragma unroll
    for (int r = 0; r < PU; ++r) {
      if (U == 2) *reinterpret_cast<u16*>(q + 2 * r) = 0xffffu; else q[r] = 0xff;
    }
  }
}

// A lane's share of one image, worked out before any shared memory is touched: per snake the contiguous run
// [i, i1) of segments this lane paints, the cell of segment i and the chain word holding the code that leads on from it.
// Everything here reads global memory and registers only, so for a CTA's first image it runs while the TMA engine is still
// fetching the border image into the buffer.
template <int S>
struct PaintRuns {
  int i[S], i1[S], pos[S];
  u32 w[S];
};
template <int S>
__device__ __forceinline__ PaintRuns<S> cta_paint_prepare(const Params& p, const PaintEnv<S>& pe, long long e_owner, int sub, int LPE) {
  PaintRuns<S> r;
  const int sh = 31 - __clz(LPE);
#pragma unroll
  for (int s = 0; s < S; ++s) {
    r.i[s] = r.i1[s] = 0; r.pos[s] = 0; r.w[s] = 0;
    if (pe.valid) {
      // lane `sub` takes the contiguous run [sub * n, sub * n + n) of the snake's segments: one popcount position, then
      // it walks the chain codes (5 instructions per segment)
      const u32* ch = p.chain + (e_owner * S + s) * p.CW;
      const int len = pe.len[s], n = (len + LPE - 1) >> sh;
      const int i = sub * n;
      r.i[s] = i; r.i1[s] = min(i + n, len);
      if (i < r.i1[s]) {
        r.pos[s] = chain_pos(pe.head[s], pe.c0[s], ch, p.V, i);
        r.w[s] = (i >> 4) ? ch[i >> 4] : pe.c0[s];  // the word holding the code of the move from segment i to i + 1
      }
    }
  }
  return r;
}

// fruits, then the snakes in index order (get_ob_for_snake :35-58); `paint` false = the same walk writes zeros.
// GRID: the image is the cell-code grid of SNK_OBS_GRID (one byte per cell, K does not enter), the same walk writes codes.
template <int S, int RULES, int K, bool GRID = false>
__device__ __forceinline__ void cta_paint(const Params& p, const PaintEnv<S>& pe, const PaintRuns<S>& runs, long long e_owner, int sub, int LPE,
                                          u8* img, bool paint) {
  constexpr int C = GRID ? 1 : 3 * K;
  const int V = p.V, F = p.F;
  const u8 red = paint ? (GRID ? SNK_CELL_FRUIT : 255) : 0;
  if (RULES == SNK_RULES_CLASSIC) {
#pragma unroll
    for (int f = 0; f < 4; ++f) {
      if (pe.valid && f < F && (f & (LPE - 1)) == sub) {
        if (GRID) img[pe.fruit[f]] = red;
        else {
#pragma unroll
          for (int k = 0; k < K; ++k) img[pe.fruit[f] * C + 3 * k] = red;
        }
      }
    }
  } else if (pe.valid) {
    const u32* gb = p.gbits + e_owner * p.GBW;
    for (int w = sub; w < p.GBW; w += LPE) {
      for (u32 bits = gb[w]; bits; bits &= bits - 1) {
        const int pid = 32 * w + __ffs(bits) - 1;
        // cells outside the board lie under the border (the reference paints them, then the wall over them, :52-56)
        const u32 px = ((u32)pid * p.magicV) >> 16, py = (u32)pid - px * (u32)V;
        if (px - 1u < (u32)(V - 2) && py - 1u < (u32)(V - 2)) {
          if (GRID) img[pid] = red;
          else {
#pragma unroll
            for (int k = 0; k < K; ++k) img[pid * C + 3 * k] = red;
          }
        }
      }
    }
  }
  if (paint) __syncthreads();  // un-painting writes zeros only: its groups need no order
#pragma unroll
  for (int s = 0; s < S; ++s) {
    if (runs.i[s] < runs.i1[s]) {
      const u32* ch = p.chain + (e_owner * S + s) * p.CW;
      int i = runs.i[s], pos = runs.pos[s];
      const int i1 = runs.i1[s];
      u32 w = runs.w[s];
      for (;;) {
        if (GRID) img[pos] = paint ? (u8)(i == 0 ? SNK_CELL_HEAD(s) : SNK_CELL_BODY(s)) : 0;
        else put_pixel<S, K>(img + pos * C, s, i == 0, paint);
        if (i + 1 >= i1) break;
        pos -= chain_delta((w >> (2 * (i & 15))) & 3, V);
        ++i;
        if ((i & 15) == 0) w = ch[i >> 4];
      }
    }
    if (paint && s + 1 < S) __syncthreads();
  }
}

// Un-paint.  Short bodies: the same walk writes zeros.  Long bodies (`restore`): the threads zero-fill the buffer and
// redraw the border (cta_restore).  A CTA's last image is not un-painted at all.
// With Params::delta (classic RGB step) an image whose envs all qualify (delta_eligible, on the old state k_lane_logic left
// at delta_prev()) goes out as its changed sectors (delta_store) instead of one bulk store.
// GRID: the same writer for SNK_OBS_GRID (k_lane_grid), images of TE cell-code grids of V*V bytes.
template <int S, int RULES, int K, bool GRID>
__device__ __forceinline__ void lane_paint2_body(const Params& p, u8* smem, u64& s_bar) {
  const int tid = threadIdx.x, NT = 64;
  const int TE = p.TE, LPE = NT / TE, E = p.E;
  const int tile_bytes = TE * E;
  u8* tile = smem;
  if (tid == 0) {
    mbar_init(&s_bar, 1);
    mbar_expect_tx(&s_bar, (u32)tile_bytes);
    for (int c = 0; c < TE / p.G; ++c) bulk_load_g2s(tile + c * p.G * E, p.tmpl, (u32)(p.G * E), &s_bar);
  }
  __syncthreads();
  const int slot = tid / LPE, sub = tid - slot * LPE;
  u8* img = tile + slot * E;
  const long long n_items = (p.N + TE - 1) / TE;
  const long long stride = gridDim.x;
  long long item = blockIdx.x;
  const bool delta = !GRID && RULES == SNK_RULES_CLASSIC && p.delta;
  asm volatile("griddepcontrol.wait;" ::: "memory");  // the records of this step come from k_lane_logic
  PaintEnv<S> cur = paint_env_from_memory<S>(p, item < n_items ? item * TE + slot : p.N);
  DeltaOld<S> cur_old;
  bool cur_frame = false;
  if (delta && cur.valid) cur_old = delta_prev_load<S>(p, item * TE + slot, cur_frame);
  bool have_image = false;  // the border image has arrived in the buffer
  const int sh = 31 - __clz(LPE);
  while (item < n_items) {
    const long long next = item + stride;
    const PaintEnv<S> nxt = paint_env_from_memory<S>(p, next < n_items ? next * TE + slot : p.N);
    DeltaOld<S> nxt_old;
    bool nxt_frame = false;
    if (delta && nxt.valid) nxt_old = delta_prev_load<S>(p, next * TE + slot, nxt_frame);
    const long long e0 = item * TE;
    int trips = 0;
#pragma unroll
    for (int s = 0; s < S; ++s) trips += (cur.len[s] + LPE - 1) >> sh;
    const PaintRuns<S> runs = cta_paint_prepare<S>(p, cur, e0 + slot, sub, LPE);
    const bool ok = delta && (!cur.valid || delta_eligible<S>(cur_old, cur_frame, cur.len));
    if (!have_image) { mbar_wait(&s_bar, 0); have_image = true; }
    cta_paint<S, RULES, K, GRID>(p, cur, runs, e0 + slot, sub, LPE, img, true);
    fence_async_smem();
    // the barriers that order the phases also take the CTA's votes
    const bool sectors = __syncthreads_and(ok);
    if (!GRID && RULES == SNK_RULES_CLASSIC && sectors) delta_store<S, K, true>(p, cur, cur_old, slot, sub, LPE, tile, (int)min((long long)TE, p.N - e0) * E, e0);
    else store_image(p, tile, tile_bytes, e0, tid, NT);
    if (next < n_items) {  // the last image of a CTA leaves its buffer as it is
      if (__syncthreads_or(p.restore_thr > 0 && trips > p.restore_thr)) cta_restore<GRID ? 1 : 3 * K>(tile, tile_bytes >> 4, img, p.V, sub, LPE, tid, NT);
      else cta_paint<S, RULES, K, GRID>(p, cur, runs, e0 + slot, sub, LPE, img, false);
      __syncthreads();
    }
    cur = nxt;
    cur_old = nxt_old;
    cur_frame = nxt_frame;
    item = next;
  }
  if (!have_image) mbar_wait(&s_bar, 0);  // never leave with a bulk copy into our shared memory in flight
  if (tid == 0) bulk_wait_all();
  // the dependent launch is released only once this CTA's images have left: with a policy kernel between two steps an
  // earlier release (before the drain, or before the last un-paint that this kernel no longer does) cost 5 us per step
  // (fruit-seeking stream 114.5 vs 109.1 us), and nothing without one (88.7 vs 89.2 us)
  __syncthreads();
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}

template <int S, int RULES, int K>
__global__ void __launch_bounds__(64) k_lane_paint2(const Params p) {
  extern __shared__ __align__(128) u8 smem[];
  __shared__ __align__(8) u64 s_bar;
  lane_paint2_body<S, RULES, K, false>(p, smem, s_bar);
}

// k_lane_grid: the observation writer of SNK_OBS_GRID behind k_lane_logic.  A grid image is 1/(3K) of the RGB one, so a
// CTA's buffer holds TE = 32 envs' grids (16 when they exceed 28 KB); K does not enter, the kernel exists per (S, rules).
template <int S, int RULES>
__global__ void __launch_bounds__(64) k_lane_grid(const Params p) {
  extern __shared__ __align__(128) u8 smem[];
  __shared__ __align__(8) u64 s_bar;
  lane_paint2_body<S, RULES, 1, true>(p, smem, s_bar);
}


// k_step_lane_ws: ONE fused launch, warp-specialised.  Each CTA has PW "paint" warps, each owning a
// shared-memory image (the scarce resource: 10 per SM at 2x19x19), and LW "logic" warps that own
// nothing but registers.  Logic warps step 32 envs per iteration (one per lane) and publish a
// per-warp round counter in shared memory; paint warps wait for the counter of the batch they
// need, read its records back from L2, paint -> stream out -> un-paint.  Logic never waits, so the
// record / action latency of later batches hides under the HBM write stream of earlier ones.
template <int S, int RULES, int K>
__global__ void __launch_bounds__(32 * (WS_PAINT_WARPS + WS_LOGIC_WARPS), 5) k_step_lane_ws(const Params p) {
  constexpr int PW = WS_PAINT_WARPS, LW = WS_LOGIC_WARPS;
  extern __shared__ __align__(128) u8 smem[];
  __shared__ double s_stats[SNK_NSTATS];
  __shared__ int s_ready[LW];
  __shared__ u32 s_bm[PW + LW][SPAWN_WORDS];  // per warp: scratch of group_spawn (logic warps)
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int TE = p.TE, LPE = 32 / TE, E = p.E, IPB = 32 / TE;  // images per 32-env batch
  if (tid < SNK_NSTATS) s_stats[tid] = 0.0;
  peer_push(p, tid);  // the running sums as of the previous step, to every peer (posted stores)
  if (tid < LW) s_ready[tid] = 0;
  __syncthreads();
  const long long n_batches = (p.N + 31) / 32;
  LaneStats st = {0, 0, 0, 0, 0, 0, 0, 0};
  u32 errs = 0;
  if (warp < PW) {
    // ------------------------------------------------------------ paint warp
    const int tile_bytes = TE * E;
    u8* tile = smem + warp * p.tile_stride;
    init_border_image(p, tile, lane);
    __syncwarp();
    const int slot = lane / LPE, sub = lane - slot * LPE;
    u8* img = tile + slot * E;
    volatile int* ready = s_ready;
    for (int r = 0;; ++r) {
      const long long base_b = ((long long)r * gridDim.x + blockIdx.x) * LW;
      if (base_b >= n_batches) break;
      for (int j = warp; j < LW * IPB; j += PW) {
        const int l = j / IPB, q = j - l * IPB;
        const long long e0 = (base_b + l) * 32 + (long long)q * TE;
        if (e0 >= p.N) continue;
        while (ready[l] <= r) __nanosleep(64);
        __threadfence_block();
        const PaintEnv<S> pe = paint_env_from_memory<S>(p, e0 + slot);
        const bool restore = lane_wants_restore<S>(p, pe.len, LPE);
        lane_paint<S, RULES, K>(p, pe, e0 + slot, sub, LPE, img, true);
        fence_async_smem();
        __syncwarp();
        store_image(p, tile, tile_bytes, e0, lane, 32);
        __syncwarp();
        lane_unpaint<S, RULES, K>(p, pe, e0 + slot, sub, LPE, tile, tile_bytes, img, lane, restore);
        __syncwarp();
      }
    }
    if (lane == 0) bulk_wait_all();
  } else {
    // ------------------------------------------------------------ logic warp
    const int lw = warp - PW;
    for (int r = 0;; ++r) {
      const long long base_b = ((long long)r * gridDim.x + blockIdx.x) * LW;
      if (base_b >= n_batches) break;
      const long long e = (base_b + lw) * 32 + lane;
      if (p.mode != MODE_OBSERVE) {
        const bool valid = e < p.N;
        LaneEnv<S> env;
#pragma unroll
        for (int s = 0; s < S; ++s) { env.head[s] = 0; env.len[s] = 0; env.c0[s] = 0; env.grow[s] = 0; env.vel[s] = 0; }
        env.fruit[0] = env.fruit[1] = env.fruit[2] = env.fruit[3] = 0;
        env.spare = 0;
        LaneRng rng;
        rng.have = false; rng.blk = 0;
        const FruitSet grid = fruit_set(p, e);
        LaneRaw<S> raw;
        raw.act = 0;
        if (valid) { raw = lane_fetch<S>(p, e, p.mode == MODE_STEP); lane_unpack<S>(raw, env); }
        if (p.mode == MODE_STEP) {
          lane_step<S, RULES>(p, e, valid, env, raw.act, rng, grid, s_bm[warp], errs, st);
        } else if (valid && (!p.mask || p.mask[e])) {
          lane_reset<S, RULES>(p, e, env, rng, grid, errs, st.draws);
        }
        if (valid) lane_store<S>(p, e, env);
      }
      __threadfence_block();  // records / chain words / fruit grid before the round counter
      __syncwarp();
      if (lane == 0) *(volatile int*)&s_ready[lw] = r + 1;
    }
  }
  reduce_lane_stats(p, st, errs, s_stats, lane);
  publish_stats(p, s_stats, tid);
}


// k_step_lane: see snk_lane.cuh.  A warp is an independent worker: 32 envs of logic (one per lane),
// then 32/TE rounds of paint -> TMA bulk store -> un-paint on its private image.  No __syncthreads.
// With Params::delta an image whose envs all qualify (delta_eligible) goes out as its changed sectors instead (delta_store).
// Three and four snakes: left to itself ptxas caps the kernel at 168 registers and spills (up to 136 bytes); asking for
// 4 CTAs per SM (up to 256 registers) keeps it spill-free.  One and two snakes keep the compiler's own choice.
template <int S, int RULES, int K>
__global__ void __launch_bounds__(64, (S >= 3 ? 4 : 0)) k_step_lane(const Params p) {
  extern __shared__ __align__(128) u8 smem[];
  __shared__ double s_stats[SNK_NSTATS];
  __shared__ __align__(8) u64 s_bar[2];
  __shared__ u32 s_bm[2][SPAWN_WORDS];  // per warp: scratch of group_spawn
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, wpc = blockDim.x >> 5;
  const int TE = p.TE, LPE = 32 / TE, E = p.E, EPW = p.EPW;  // EPW envs per warp batch: 32, fewer when the shard is small (snk_api.cu)
  const int tile_bytes = TE * E;
  u8* tile = smem + warp * p.tile_stride;
  // the border-only image arrives through the TMA engine while the first batch is being stepped
  if (lane == 0) {
    mbar_init(&s_bar[warp], 1);
    mbar_expect_tx(&s_bar[warp], (u32)tile_bytes);
    for (int c = 0; c < TE / p.G; ++c) bulk_load_g2s(tile + c * p.G * E, p.tmpl, (u32)(p.G * E), &s_bar[warp]);
  }
  if (tid < SNK_NSTATS) s_stats[tid] = 0.0;
  __syncthreads();
  LaneStats st = {0, 0, 0, 0, 0, 0, 0, 0};
#ifdef SNK_PHASE_LOGIC
  st.ph[0] = st.ph[1] = st.ph[2] = st.ph[3] = 0;
#endif
  u32 errs = 0;
  const int slot = lane / LPE, sub = lane - slot * LPE;
  u8* img = tile + slot * E;
  const long long n_batches = (p.N + EPW - 1) / EPW;
  const long long stride = (long long)gridDim.x * wpc;
  const bool stepping = p.mode == MODE_STEP;
  const bool delta = RULES == SNK_RULES_CLASSIC && stepping && p.delta;
  const u32 tile_mask = TE == 32 ? ~0u : (1u << TE) - 1u;
  long long b = (long long)blockIdx.x * wpc + warp;
  LaneRaw<S> raw;
  // Programmatic dependent launch: everything above (shared-memory carve-up, mbarrier, border image
  // fetch) may overlap the tail of the previous launch in the stream; records, actions and every
  // output are only touched after the previous grid has completed and flushed.
  asm volatile("griddepcontrol.wait;" ::: "memory");
  peer_push(p, tid);  // the running sums as of the previous step, to every peer (posted stores)
  if (b < n_batches && lane < EPW && b * EPW + lane < p.N) raw = lane_fetch<S>(p, b * EPW + lane, stepping);
  bool have_image = false;
#ifdef SNK_PHASE_TIMING  // experiment build (tools/phase.py): cycles per phase, summed over warps
  long long tA = 0, tB = 0, tC = 0, tD = 0; const long long tStart = clock64();
#endif
  for (; b < n_batches; b += stride) {
#ifdef SNK_PHASE_TIMING
    long long t0 = clock64();
#endif
    const long long e = b * EPW + lane;
    const bool valid = lane < EPW && e < p.N;  // lanes past EPW idle through the logic and join the painting
    LaneEnv<S> env;
#pragma unroll
    for (int s = 0; s < S; ++s) { env.head[s] = 0; env.len[s] = 0; env.c0[s] = 0; env.grow[s] = 0; env.vel[s] = 0; }
    env.fruit[0] = env.fruit[1] = env.fruit[2] = env.fruit[3] = 0;
    env.spare = 0;
    {
      LaneRng rng;
      rng.have = false; rng.blk = 0;
      const FruitSet grid = fruit_set(p, e);
      if (valid) lane_unpack<S>(raw, env);
      if (stepping) {
        lane_step<S, RULES>(p, e, valid, env, raw.act, rng, grid, s_bm[warp], errs, st);
      } else if (valid && p.mode == MODE_RESET) {
        if (!p.mask || p.mask[e]) lane_reset<S, RULES>(p, e, env, rng, grid, errs, st.draws);
      }
      if (valid && p.mode != MODE_OBSERVE) lane_store<S>(p, e, env);
    }
    // delta store: the old state's paint items, and the lanes whose env must go out as a whole image
    DeltaOld<S> old;
    u32 whole = ~0u;
    if (delta) {
      old = delta_old<S>(raw);
      whole = __ballot_sync(FULL, valid && !delta_eligible<S>(old, raw.frame, env.len));
    }
    // records + actions of this warp's NEXT batch: in flight while the current one is painted
    if (b + stride < n_batches && lane < EPW && (b + stride) * EPW + lane < p.N) raw = lane_fetch<S>(p, (b + stride) * EPW + lane, stepping);
    const bool restore = lane_wants_restore<S>(p, env.len, LPE);  // one decision for the batch's 32/TE images
    if (!have_image) { mbar_wait(&s_bar[warp], 0); have_image = true; }
    __syncwarp();  // chain words / fruit grid written by the owner lane are read by the painting lanes
#ifdef SNK_PHASE_TIMING
    { const long long t1 = clock64(); tA += t1 - t0; t0 = t1; }
#endif
    for (int q = 0; q * TE < EPW; ++q) {
      const long long e0 = b * EPW + (long long)q * TE;
      if (e0 >= p.N) break;
      const PaintEnv<S> pe = paint_env_from_lane<S>(env, valid, q * TE + slot);
      lane_paint<S, RULES, K>(p, pe, e0 + slot, sub, LPE, img, true);
      fence_async_smem();  // generic-proxy writes -> visible to the async (TMA) proxy
      __syncwarp();
#ifdef SNK_PHASE_TIMING
      { const long long t1 = clock64(); tB += t1 - t0; t0 = t1; }
#endif
      if (((whole >> (q * TE)) & tile_mask) == 0) {
        const DeltaOld<S> po = delta_old_from_lane<S>(old, q * TE + slot);
        delta_store<S, K, false>(p, pe, po, slot, sub, LPE, tile, (int)min((long long)TE, p.N - e0) * E, e0);
      } else {
        store_image(p, tile, tile_bytes, e0, lane, 32);
      }
      __syncwarp();
#ifdef SNK_PHASE_TIMING
      { const long long t1 = clock64(); tC += t1 - t0; t0 = t1; }
#endif
      // the warp's last image of the launch leaves the buffer as it is (small shards: its only image)
      if (b + stride < n_batches || ((q + 1) * TE < EPW && e0 + TE < p.N))
        lane_unpaint<S, RULES, K>(p, pe, e0 + slot, sub, LPE, tile, tile_bytes, img, lane, restore);
      __syncwarp();
#ifdef SNK_PHASE_TIMING
      { const long long t1 = clock64(); tD += t1 - t0; t0 = t1; }
#endif
    }
  }
#ifdef SNK_PHASE_TIMING
  if (lane == 0) {  // the last five statistics carry the cycle sums instead (total, logic, paint, store + wait, un-paint)
    atomicAdd(&p.stats[3], (double)(clock64() - tStart)); atomicAdd(&p.stats[4], (double)tA); atomicAdd(&p.stats[5], (double)tB);
    atomicAdd(&p.stats[6], (double)tC); atomicAdd(&p.stats[7], (double)tD);
  }
#ifdef SNK_PHASE_LOGIC  // the four slots carry move+push / respawns / death test / tail+reset of the logic instead
  if (lane == 0) {
    atomicAdd(&p.stats[4], (double)(st.ph[0] - tA)); atomicAdd(&p.stats[5], (double)(st.ph[1] - tB));
    atomicAdd(&p.stats[6], (double)(st.ph[2] - tC)); atomicAdd(&p.stats[7], (double)(st.ph[3] - tD));
  }
#endif
  st.len_sum = st.fruits = st.deaths = st.cells = st.draws = 0.f;
#endif
  if (!have_image) mbar_wait(&s_bar[warp], 0);  // never leave with a bulk copy into our shared memory in flight
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");  // the next launch may start its prologue
  reduce_lane_stats(p, st, errs, s_stats, lane);  // (the last images drain while the statistics are folded)
  publish_stats(p, s_stats, tid);
  if (lane == 0) bulk_wait_all();
}

template <int RULES>
__global__ void __launch_bounds__(256) k_step_dense(const Params p) {
  extern __shared__ __align__(128) u8 smem[];
  __shared__ double s_stats[SNK_NSTATS];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nthr = blockDim.x;
  const int S = p.S, F = p.F, K = p.K, VV = p.VV, V = p.V, cap = p.cap;
  u8* code = smem;  // [VV] 0 empty, 1 fruit, 2 wall, 3+2s body of s, 4+2s head of s
  u32* sc = reinterpret_cast<u32*>(smem + ((VV + 15) & ~15));
  u32* bm = sc + p.RW;
  if (tid < SNK_NSTATS) s_stats[tid] = 0.0;
  peer_push(p, tid);  // the running sums as of the previous step, to every peer (posted stores)
  __syncthreads();
  WarpStats st = {0, 0, 0, 0, 0, 0, 0, 0};
  u32 errs = 0;
  for (long long e = blockIdx.x; e < p.N; e += gridDim.x) {
    if (warp == 0) advance_env<RULES>(p, e, lane, sc, bm, errs, st);
    for (int i = tid; i < VV; i += nthr) code[i] = 0;
    __syncthreads();
    if (RULES == SNK_RULES_CLASSIC) {
      const u16* fr = reinterpret_cast<const u16*>(sc + REC_SNAKE0 + 2 * S);
      if (tid < F) code[fr[tid]] = 1;
    } else {
      const u8* grid = p.grid + e * p.grid_stride;
      const u32* g32 = reinterpret_cast<const u32*>(grid);  // grid_stride is a multiple of 16
      for (int w = tid; w < (VV + 3) / 4; w += nthr) {
        u32 word = g32[w];
        for (int q = 0; word; ++q, word >>= 8) if ((word & 0xff) && 4 * w + q < VV) code[4 * w + q] = 1;
      }
    }
    __syncthreads();
    const u16* rings = p.body + e * S * cap;
    for (int s = 0; s < S; ++s) {
      const u32 a = sc[REC_SNAKE0 + 2 * s];
      const int len = a >> 16, hs = a & 0xffff;
      if (len == 0) continue;  // block-uniform
      for (int i = tid; i < len; i += nthr) code[ring_at(rings + s * cap, hs, i, cap)] = (u8)(3 + 2 * s + (i == 0));
      __syncthreads();
    }
    for (int i = tid; i < V; i += nthr) {
      code[i] = 2; code[(V - 1) * V + i] = 2; code[i * V] = 2; code[i * V + V - 1] = 2;
    }
    __syncthreads();
    u8* out = p.obs + e * (long long)p.E;
    for (int j = tid; j < VV * K; j += nthr) {  // j = pixel * K + view: 3 consecutive bytes
      const int px = j / K, k = j - px * K;
      const int c = code[px];
      u32 rgb = 0;
      if (c == 1) rgb = 255u;
      else if (c == 2) rgb = 0xffffffu;
      else if (c >= 3) rgb = snake_rgb(((c - 3) >> 1) == k, (c - 3) & 1);
      out[3 * j] = (u8)rgb; out[3 * j + 1] = (u8)(rgb >> 8); out[3 * j + 2] = (u8)(rgb >> 16);
    }
    __syncthreads();
  }
  if (warp == 0) flush_stats(p, st, errs, s_stats, lane);
  publish_stats(p, s_stats, tid);
}


// k_step_rows: large fields (e.g. 16 snakes on 64x64: 209 KB of observation per env).  One CTA per
// env: warp 0 runs the warp-cooperative logic, all threads build the cell-code grid in shared
// memory (fruits, snakes in index order, border: the reference's paint order, get_ob_for_snake
// :35-58), then the image leaves in chunks of R rows: each thread expands whole pixels (one code ->
// 3K bytes, written once, 16-byte vector stores) into one of two chunk buffers and a TMA bulk copy
// streams the buffer out while the next chunk is being expanded.
__device__ __forceinline__ void pattern3(u32 rgb, u32& w0, u32& w1, u32& w2) {  // RGBRGB... as 3 periodic words
  const u32 r = rgb & 255, g = (rgb >> 8) & 255, b = (rgb >> 16) & 255;
  w0 = r | g << 8 | b << 16 | r << 24; w1 = g | b << 8 | r << 16 | g << 24; w2 = b | r << 8 | g << 16 | b << 24;
}

__device__ __forceinline__ void consumer_sync(int n) { asm volatile("bar.sync 1, %0;" ::"r"(n) : "memory"); }

// One cell code -> the C bytes of its pixel in a chunk buffer (16-byte vector stores).  CT = compile-time
// pixel size (48 = 16 views, the large-field configuration: the per-word phase of the RGB pattern and the
// store loop then fold to constants), 0 = run time.
template <int CT>
__device__ __forceinline__ void rows_emit(u8* __restrict__ tile, int i, int cd, int C_, int K) {
  const int C = CT > 0 ? CT : C_;
  u32 rgb = 0;
  int self = -1;
  if (cd == 1) rgb = 255u;
  else if (cd == 255) rgb = 0xffffffu;
  else if (cd >= 3) { self = (cd - 3) >> 1; rgb = snake_rgb(false, (cd - 3) & 1); }
  u32 w0, w1, w2;
  pattern3(rgb, w0, w1, w2);
  u8* px = tile + i * C;
  if ((C & 15) == 0) {
    uint4* q = reinterpret_cast<uint4*>(px);
    const int n16 = C / 16;
#pragma unroll
    for (int j = 0; j < n16; ++j) {  // word index 4j: period 3 words
      const int ph = (4 * j) % 3;
      const u32 a0 = ph == 0 ? w0 : ph == 1 ? w1 : w2, a1 = ph == 0 ? w1 : ph == 1 ? w2 : w0, a2 = ph == 0 ? w2 : ph == 1 ? w0 : w1;
      q[j] = make_uint4(a0, a1, a2, a0);
    }
  } else {
    for (int j = 0; j < C; ++j) px[j] = (u8)(rgb >> (8 * (j % 3)));
  }
  if (self >= 0 && self < K) {
    const u32 own = snake_rgb(true, (cd - 3) & 1);
    px[3 * self] = (u8)own; px[3 * self + 1] = (u8)(own >> 8); px[3 * self + 2] = (u8)(own >> 16);
  }
}

// Expand the `cells` cell codes of one chunk, one thread per cell.
template <int CT>
__device__ __forceinline__ void rows_expand(const u8* __restrict__ code, u8* __restrict__ tile, int cells, int C, int K, int ct, int cn) {
  for (int i = ct; i < cells; i += cn) rows_emit<CT>(tile, i, code[i], C, K);
}

// GRID (SNK_OBS_GRID): the consumers store the finished code grid itself, V*V bytes at obs + e*V*V (not 16-byte aligned
// in general: plain coalesced stores), and there are no chunk buffers.
template <int RULES, bool GRID>
__global__ void __launch_bounds__(160, 5) k_step_rows(const Params p) {
  extern __shared__ __align__(128) u8 smem[];
  __shared__ double s_stats[SNK_NSTATS];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int S = p.S, F = p.F, K = p.K, C = p.C, VV = p.VV, V = p.V, cap = p.cap, R = p.R;
  const int code_stride = (VV + 127) & ~127;
  u8* codes = smem;  // two grids [VV]: 0 empty, 1 fruit, 3+2s body of s, 4+2s head of s, 255 border
  u8* tiles = smem + 2 * code_stride;
  u32* sc = reinterpret_cast<u32*>(tiles + 2 * p.tile_stride);
  u32* bm = sc + p.RW;
  if (tid < SNK_NSTATS) s_stats[tid] = 0.0;
  peer_push(p, tid);  // the running sums as of the previous step, to every peer (posted stores)
  __syncthreads();
  WarpStats st = {0, 0, 0, 0, 0, 0, 0, 0};
  u32 errs = 0;
  const int n_chunks = GRID ? 0 : (V + R - 1) / R;
  int issued = 0;  // chunks handed to the TMA engine so far (bulk groups of the consumers' thread 0)
#ifdef SNK_PHASE_TIMING  // experiment build (tools/phase_rows.py)
  long long tA = 0, tB = 0, tC = 0, tD = 0; const long long tStart = clock64();
#endif
  // Software pipeline over envs: warp 0 (producer) steps env e_next and builds its code grid while
  // warps 1..4 (consumers) expand and stream out the image of env e from the other grid.
  long long e = blockIdx.x;
  for (int it = 0;; ++it, e += gridDim.x) {
    if (warp == 0) {
      // iteration `it` consumes grid it & 1 (env e) and builds grid (it + 1) & 1 (env e + gridDim.x);
      // iteration 0 first builds grid 0 as well
      const long long eb = it == 0 ? e : e + gridDim.x;
      for (int rep = 0; rep < (it == 0 ? 2 : 1); ++rep) {
        const long long en = rep == 0 ? eb : eb + gridDim.x;
        u8* code = codes + ((it == 0 ? rep : it + 1) & 1) * code_stride;
        if (en >= p.N) continue;
#ifdef SNK_PHASE_TIMING
        const long long ta0 = clock64();
#endif
        {
          // L2 prefetch: the fruit count grid of this env (read at the end of the build, after the whole step)
          // and the record + actions of the env this warp steps next (a whole env period ahead)
          if (RULES != SNK_RULES_CLASSIC) {
            const u8* g = p.grid + en * p.grid_stride;
            for (int off = lane * 128; off < p.grid_stride; off += 32 * 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(g + off));
          }
          const long long nx = en + gridDim.x;
          if (nx < p.N) {
            if (lane < (p.RW * 4 + 127) / 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(reinterpret_cast<const u8*>(p.rec + nx * p.RW) + lane * 128));
            if (lane == 31 && p.actions) asm volatile("prefetch.global.L2 [%0];" ::"l"(p.actions + nx * S));
          }
        }
        advance_env<RULES>(p, en, lane, sc, bm, errs, st);
#ifdef SNK_PHASE_TIMING
        const long long ta1 = clock64(); tA += ta1 - ta0;
#endif
        uint4* c16 = reinterpret_cast<uint4*>(code);
        for (int i = lane; i < code_stride / 16; i += 32) c16[i] = make_uint4(0, 0, 0, 0);
        __syncwarp();
        if (RULES == SNK_RULES_CLASSIC) {
          const u16* fr = reinterpret_cast<const u16*>(sc + REC_SNAKE0 + 2 * S);
          if (lane < F) code[fr[lane]] = 1;
        } else {
          // count-grid rules: cells holding fruit get code 1 here, read with independent 16-byte loads (the
          // grid was last written by this warp); snakes and the border overwrite it below
          const uint4* g16 = reinterpret_cast<const uint4*>(p.grid + en * p.grid_stride);
          const int n16 = p.grid_stride / 16;
#pragma unroll 3
          for (int i = lane; i < n16; i += 32) {
            const uint4 v = g16[i];
            if (v.x | v.y | v.z | v.w) {
              const u32 w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
              for (int k = 0; k < 16; ++k)
                if (((w[k >> 2] >> (8 * (k & 3))) & 0xffu) && 16 * i + k < VV) code[16 * i + k] = 1;
            }
          }
        }
        __syncwarp();
        // codes grow in paint order, so "later overwrites earlier" is a per-cell max: all snakes at
        // once, repeated until no lane had to raise a cell (cells shared by two snakes are rare)
        const u16* rings = p.body + en * S * cap;
        {
          // all snakes' segments as one list, 32 per pass (seg_scan / seg_locate, snk_device.cuh): the ring
          // reads of a pass are independent loads
          const u32 a_mine = lane < S ? sc[REC_SNAKE0 + 2 * lane] : 0u;
          const int len_mine = a_mine >> 16;
          const SegScan sg = seg_scan(len_mine, lane);
          for (int pass = 0; pass < 64; ++pass) {
            int changed = 0;
            for (int t0 = 0; t0 < sg.total; t0 += 32) {
              int j, i;
              const bool have = seg_locate(sg, len_mine, S, t0 + lane, j, i);
              const int hs = __shfl_sync(FULL, (int)(a_mine & 0xffff), j);
              if (have) {
                const int cell = ring_at(rings + j * cap, hs, i, cap);
                const u8 mine = (u8)(3 + 2 * j + (i == 0));
                if (code[cell] < mine) { code[cell] = mine; changed = 1; }
              }
            }
            __syncwarp();
            if (!__any_sync(FULL, changed)) break;
          }
        }
        for (int i = lane; i < V; i += 32) { code[i] = 255; code[(V - 1) * V + i] = 255; code[i * V] = 255; code[i * V + V - 1] = 255; }
        __syncwarp();
#ifdef SNK_PHASE_TIMING
        tB += clock64() - ta1;
#endif
      }
    }
    if (it == 0) __syncthreads();  // grid 0 ready
    if (e >= p.N) break;
    if (GRID && warp > 0) {
      const u8* code = codes + (it & 1) * code_stride;
      u8* out = p.obs + e * (long long)VV;
      for (int i = tid - 32; i < VV; i += blockDim.x - 32) out[i] = code[i];
    } else if (warp > 0) {
      const int ct = tid - 32, cn = blockDim.x - 32;
      const u8* code = codes + (it & 1) * code_stride;
      u8* out = p.obs + e * (long long)p.E;
#ifdef SNK_PHASE_TIMING
      const long long tc0 = clock64();
#endif
      for (int c = 0; c < n_chunks; ++c) {
        u8* tile = tiles + (issued & 1) * p.tile_stride;
#ifdef SNK_PHASE_TIMING
        const long long tw0 = clock64();
#endif
        if (issued >= 2) {  // the copy that last used this buffer has been read by the engine
          if (ct == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
          consumer_sync(cn);
        }
#ifdef SNK_PHASE_TIMING
        tD += clock64() - tw0;
#endif
        const int r0 = c * R, rows = min(R, V - r0), cells = rows * V;
        if (C == 48) rows_expand<48>(code + r0 * V, tile, cells, C, K, ct, cn);
        else rows_expand<0>(code + r0 * V, tile, cells, C, K, ct, cn);
        fence_async_smem();
        consumer_sync(cn);
        if (ct == 0) {
          const int bytes = cells * C;
          for (int off = 0; off < bytes; off += 16384)
            bulk_store_s2g(out + (long long)r0 * V * C + off, tile + off, (u32)min(16384, bytes - off));
          bulk_commit();
        }
        ++issued;
      }
#ifdef SNK_PHASE_TIMING
      tC += clock64() - tc0;
#endif
    }
    __syncthreads();  // grid (it + 1) & 1 built, grid it & 1 consumed
  }
  if (!GRID && tid == 32) bulk_wait_all();
#ifdef SNK_PHASE_TIMING  // total, producer logic, producer grid build, consumers, of which TMA read-wait
  if (tid == 0) { atomicAdd(&p.stats[3], (double)(clock64() - tStart)); atomicAdd(&p.stats[4], (double)tA); atomicAdd(&p.stats[5], (double)tB); }
  if (tid == 32) { atomicAdd(&p.stats[6], (double)tC); atomicAdd(&p.stats[7], (double)tD); }
  st.len_sum = st.fruits = st.deaths = st.cells = st.draws = 0.f;
#endif
  if (warp == 0) flush_stats(p, st, errs, s_stats, lane);
  publish_stats(p, s_stats, tid);
}

// The file can be compiled as one translation unit (SNK_TU undefined) or as four that build in
// parallel: SNK_TU = 0 / 1 / 2 instantiates the step kernels of one rule-set, SNK_TU = 3 holds the
// remaining kernels and the host dispatch.
#ifndef SNK_TU
#define SNK_TU (-1)
#endif
#if SNK_TU == -1 || SNK_TU == 3
// k_upscale84: obs_mode = SNK_OBS_ATARI84, the reference's WarpFrame (utils.py:27-31):
// cv2.resize(frame, (84, 84), INTER_AREA), which for 84 % V == 0 is exact r x r pixel replication
// (r = 84 / V).  One CTA per env: the native [V][V][3K] image is staged in shared memory, every
// thread replicates source pixels into the 84x84 image (also in shared memory), and one TMA bulk
// copy streams the 7056*3K bytes out (always a multiple of 16, so every env is an aligned unit).
// one source pixel -> R rows of R copies; compile-time pixel size C and factor R (0 = runtime)
template <int CT, int RT>
__device__ __forceinline__ void upscale_pixel(const u8* spx, u8* dst0, int C, int r) {
  if constexpr (CT > 0 && (CT % 2) == 0 && ((RT * CT) % 8) == 0) {
    // the R*C-byte run is a periodic pattern of C/2 halfwords: build it once as 64-bit words
    constexpr int NH = CT / 2, NQ = RT * CT / 8;
    u64 h[NH];
#pragma unroll
    for (int j = 0; j < NH; ++j) h[j] = reinterpret_cast<const u16*>(spx)[j];
    u64 q[NQ];
#pragma unroll
    for (int w = 0; w < NQ; ++w) q[w] = h[(4 * w) % NH] | h[(4 * w + 1) % NH] << 16 | h[(4 * w + 2) % NH] << 32 | h[(4 * w + 3) % NH] << 48;
#pragma unroll
    for (int dx = 0; dx < RT; ++dx) {
      u64* row = reinterpret_cast<u64*>(dst0 + dx * 84 * CT);
#pragma unroll
      for (int w = 0; w < NQ; ++w) row[w] = q[w];
    }
  } else if constexpr (CT > 0) {
    u8 v[CT];
#pragma unroll
    for (int j = 0; j < CT; ++j) v[j] = spx[j];
#pragma unroll
    for (int dx = 0; dx < RT; ++dx) {
      u8* row = dst0 + dx * 84 * CT;
#pragma unroll
      for (int dy = 0; dy < RT; ++dy)
#pragma unroll
        for (int j = 0; j < CT; ++j) row[dy * CT + j] = v[j];
    }
  } else {
    for (int dx = 0; dx < r; ++dx) {
      u8* row = dst0 + dx * 84 * C;
      for (int j = 0; j < C; ++j) {
        const u8 v = spx[j];
        for (int dy = 0; dy < r; ++dy) row[dy * C + j] = v;
      }
    }
  }
}

// The 84x84 image leaves in TWO parts (native rows [0, rows_a) and [rows_a, V); rows_a = V: one part), each its own bulk
// group: while the engine streams part A out, the threads expand part B, and while B streams they expand part A of the
// next env, whose native image was fetched into registers a whole env earlier.  The first form (expand the whole image,
// hand it over, wait) left the SM's store path idle a third of the time: 1 070 us per 131 072 envs of 2 views 21x21
// (5.5 TB/s) -- see DESIGN.md 4.11.
__device__ __forceinline__ void bulk_wait_read1() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }

template <int CT, int RT>
__global__ void __launch_bounds__(256) k_upscale84(const u8* __restrict__ native, u8* __restrict__ out, long long N, int V, int C_, int rows_a) {
  extern __shared__ __align__(128) u8 smem[];
  const int tid = threadIdx.x, nthr = 256;
  const int C = CT > 0 ? CT : C_, r = RT > 0 ? RT : 84 / V;
  const int E = V * V * C, OUT = 84 * 84 * C;
  u8* dst = smem;
  u8* src = smem + ((OUT + 127) & ~127);
  // halfwords of one native image per thread, known at compile time for the specialised shapes (V = 84 / RT)
  constexpr int PF = (CT > 0 && RT > 0 && ((84 / (RT > 0 ? RT : 1)) * (84 / (RT > 0 ? RT : 1)) * CT) % 2 == 0)
                         ? ((84 / (RT > 0 ? RT : 1)) * (84 / (RT > 0 ? RT : 1)) * CT / 2 + 255) / 256 : 0;
  u16 pf[PF > 0 ? PF : 1];
  const bool two = rows_a < V;
  const int px_a = rows_a * V, bytes_a = rows_a * r * 84 * C;
  long long e = blockIdx.x;
  if (PF > 0 && e < N) {
    const u16* g16 = reinterpret_cast<const u16*>(native + e * (long long)E);
#pragma unroll
    for (int k = 0; k < PF; ++k) { const int i = tid + k * nthr; pf[k] = i < E / 2 ? g16[i] : (u16)0; }
  }
  for (; e < N; e += gridDim.x) {
    if (PF > 0) {
      u16* s16 = reinterpret_cast<u16*>(src);
#pragma unroll
      for (int k = 0; k < PF; ++k) { const int i = tid + k * nthr; if (i < E / 2) s16[i] = pf[k]; }
      const long long en = e + gridDim.x;
      if (en < N) {  // the next env's native image: in flight while this one is expanded and streamed
        const u16* g16 = reinterpret_cast<const u16*>(native + en * (long long)E);
#pragma unroll
        for (int k = 0; k < PF; ++k) { const int i = tid + k * nthr; pf[k] = i < E / 2 ? g16[i] : (u16)0; }
      }
    } else {
      const u8* g = native + e * (long long)E;
      for (int i = tid; i < E; i += nthr) src[i] = g[i];
    }
    for (int part = 0; part < (two ? 2 : 1); ++part) {
      // the part's region of the image buffer was last read by the bulk group issued two groups ago
      if (tid == 0) { if (two) bulk_wait_read1(); else bulk_wait_read(); }
      __syncthreads();  // also: src is complete
      const int p0 = part ? px_a : 0, p1 = (two && !part) ? px_a : V * V;
      for (int sp = p0 + tid; sp < p1; sp += nthr) {
        const int x = sp / V, y = sp - x * V;
        upscale_pixel<CT, RT>(src + sp * C, dst + ((x * r) * 84 + y * r) * C, C, r);
      }
      fence_async_smem();
      __syncthreads();
      if (tid == 0) {
        const int o0 = part ? bytes_a : 0, o1 = (two && !part) ? bytes_a : OUT;
        u8* gd = out + e * (long long)OUT;
        for (int off = o0; off < o1; off += 16384) bulk_store_s2g(gd + off, dst + off, (u32)min(16384, o1 - off));
        bulk_commit();
      }
    }
    // (the barrier before the last part's hand-over also ended every read of src: the next iteration may overwrite it)
  }
  if (tid == 0) bulk_wait_all();
}

template <int CT, int RT>
static cudaError_t launch_upscale(const uint8_t* native, uint8_t* out, long long N, int V, int C, int n_sm, cudaStream_t stream) {
  const size_t smem = (((size_t)84 * 84 * C + 127) & ~(size_t)127) + (size_t)V * V * C + 16;
  cudaError_t err = cudaFuncSetAttribute(k_upscale84<CT, RT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (err) return err;
  int occ = 0;
  if ((err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_upscale84<CT, RT>, 256, smem))) return err;
  if (occ < 1) return cudaErrorInvalidConfiguration;
  long long grid = (long long)n_sm * occ;
  if (grid > N) grid = N;
  // two parts: the split nearest the middle whose first part is a whole number of 16-byte units (TMA); none: one part
  const int r = 84 / V;
  int rows_a = V;
  for (int d = 0; d < V / 2 && rows_a == V; ++d)
    for (int k : {V / 2 + d, V / 2 - d})
      if (k > 0 && k < V && ((size_t)k * r * 84 * C) % 16 == 0) { rows_a = k; break; }
  k_upscale84<CT, RT><<<(unsigned)grid, 256, smem, stream>>>(native, out, N, V, C, rows_a);
  return cudaGetLastError();
}


// k_scripted_actions: greedy fruit seeking on the device (benchmark action stream).  One thread per
// env, registers only: the up-to-four candidate cells of every snake are compared against every
// segment in ONE walk of the chain codes (the first form kept a V*V-bit occupancy bitmap in local
// memory: 25 us per 131 072 envs, as long as a quarter of the step it feeds).
// `occ_obs` (may be NULL): the native observations of the state the policy acts on.  A cell holds a snake segment or lies
// outside the board exactly when the green byte of its pixel in view 0 is non-zero (snake_rgb / the white border; fruit
// and empty cells have G = 0), so six byte loads replace the walk of both bodies -- which, one env per lane, cost every
// warp its longest pair of snakes: 31 us per 131 072 envs under this policy, a third of the step it feeds.
// The contract (draw, candidates, distances, tie-break) is stated at snk_gen_scripted_actions in include/snk.h;
// tests/scripted_ref.py restates it in numpy and tests/test_gpu_scripted.py holds this kernel to it.
template <int S>
__global__ void __launch_bounds__(128) k_scripted_actions(const Params p, int8_t* actions, u64 step, u64 seed, int eps_permille,
                                                          const u8* __restrict__ occ_obs) {
  const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  // launched programmatically between two step kernels: wait for the step that produced the state, then let the next
  // step's prologue in right away (it waits for this grid's completion itself before it touches the actions)
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  if (e >= p.N) return;
  LaneEnv<S> env;
  lane_load<S>(p, e, env);
  const int V = p.V, F = p.F;
  int cand[S][4];   // cell a snake would enter with action a+1, or -1: not a candidate (dead, reversal, outside)
#pragma unroll
  for (int s = 0; s < S; ++s) {
#pragma unroll
    for (int a = 1; a <= 4; ++a) {
      int c = -1;
      if (env.len[s] && !(env.vel[s] && a == (((env.vel[s] + 1) & 3) + 1))) {  // reversal is ignored by the env anyway
        c = env.head[s] + chain_delta((u32)(a - 1), V);
        if (!occ_obs && (__ldg(p.cellinfo + c) >> 31)) c = -1;  // (from the observations: the border's G byte blocks it below)
      }
      cand[s][a - 1] = c;
    }
  }
  u32 blocked = 0;  // bit 4s + a-1: some segment of some snake lies on cand[s][a-1]
  if (occ_obs) {
    const u8* o = occ_obs + e * (long long)p.E + 1;
#pragma unroll
    for (int s = 0; s < S; ++s) {
#pragma unroll
      for (int a = 0; a < 4; ++a) if (cand[s][a] >= 0 && __ldg(o + cand[s][a] * p.C) != 0) blocked |= 1u << (4 * s + a);
    }
  } else
#pragma unroll
  for (int j = 0; j < S; ++j)
    chain_walk(env.head[j], env.len[j], env.c0[j], p.chain + (e * S + j) * p.CW, V, [&](int, int pid) {
#pragma unroll
      for (int s = 0; s < S; ++s) {
#pragma unroll
        for (int a = 0; a < 4; ++a) if (pid == cand[s][a]) blocked |= 1u << (4 * s + a);
      }
    });
  int fx[4], fy[4];
#pragma unroll
  for (int f = 0; f < 4; ++f) { fx[f] = env.fruit[f] / V; fy[f] = env.fruit[f] - fx[f] * V; }
  u32 packed = 0;
#pragma unroll
  for (int s = 0; s < S; ++s) {
    int best = 0;
    if (env.len[s]) {
      const u32 rnd = philox_bounded(seed, (u64)(p.env_id_base + e), 2, step * (u64)S + (u64)s, 1000u * 5u);
      if ((int)(rnd / 5u) < eps_permille) {
        best = (int)(rnd % 5u);
      } else {
        int best_d = 0x7fffffff;
#pragma unroll
        for (int a = 1; a <= 4; ++a) {
          const int c = cand[s][a - 1];
          if (c < 0 || ((blocked >> (4 * s + a - 1)) & 1)) continue;
          const int cx = c / V, cy = c - cx * V;
          int d = 0x7ffffffe;
#pragma unroll
          for (int f = 0; f < 4; ++f)
            if (f < F) d = min(d, abs(cx - fx[f]) + abs(cy - fy[f]));
          if (d < best_d) { best_d = d; best = a; }
        }
      }
    }
    packed |= (u32)best << (8 * s);
  }
  if (S == 2) *reinterpret_cast<u16*>(actions + e * S) = (u16)packed;
  else if (S == 4) *reinterpret_cast<u32*>(actions + e * S) = packed;
  else {
#pragma unroll
    for (int s = 0; s < S; ++s) actions[e * S + s] = (int8_t)(packed >> (8 * s));
  }
}


// k_gae: the reversed GAE loop of Runner.run (ppo_multi_agent_new.py:209-218), one thread per env.
// The reference mixes precisions (float32 arrays, `1.0 - dones` is float64, python-float gamma): every
// operation below is the same IEEE operation in the same order, with explicit _rn intrinsics so that
// nothing is contracted into an FMA.
__global__ void k_gae(const float* __restrict__ rewards, const float* __restrict__ values, const u8* __restrict__ dones,
                      const float* __restrict__ last_values, const u8* __restrict__ last_dones, double gamma, double lam, int T,
                      long long N, float* __restrict__ advs, float* __restrict__ returns) {
  const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  const float gamma32 = (float)gamma;          // python float * float32 array -> float32 product
  const double gl = __dmul_rn(gamma, lam);     // python float * python float
  double last = 0.0;
  for (int t = T - 1; t >= 0; --t) {
    const bool tail = t == T - 1;
    const double nonterm = __dsub_rn(1.0, (double)(tail ? last_dones[n] : dones[(long long)(t + 1) * N + n]));
    const float nextv = tail ? last_values[n] : values[(long long)(t + 1) * N + n];
    const float v = values[(long long)t * N + n];
    const double gvn = __dmul_rn((double)__fmul_rn(gamma32, nextv), nonterm);
    const double delta = __dsub_rn(__dadd_rn((double)rewards[(long long)t * N + n], gvn), (double)v);
    last = __dadd_rn(delta, __dmul_rn(__dmul_rn(gl, nonterm), last));
    const float a = (float)last;
    advs[(long long)t * N + n] = a;
    returns[(long long)t * N + n] = __fadd_rn(a, v);
  }
}

// ------------------------------------------------------------------ env state: canonical blob <-> private layout
// snk_save_envs / snk_restore_envs / snk_copy_envs, and through them snk_dump_state(_range) / snk_load_state.  One warp
// per entry: its snakes one after the other, then the entry's scalars and fruits.  Entry j of a launch is env idx[j]
// of the handle (idx == NULL: env first + j) and row j of a `count`-env blob.  An index outside [0, N) raises
// SNK_DEVERR_BAD_STATE and nothing is written for that entry.  Body rows move as 16-byte vectors by consecutive lanes.
__device__ __forceinline__ bool entry_env(const Params& p, const int64_t* idx, long long first, long long j, bool report,
                                          long long& e) {
  e = idx ? (long long)idx[j] : first + j;
  if (e >= 0 && e < p.N) return true;
  if (report) atomicOr(p.err, SNK_DEVERR_BAD_STATE);
  return false;
}

// the alignment gaps between the arrays of a blob (zero in every blob, so two blobs are byte-comparable)
__device__ __noinline__ void blob_zero_gaps(u8* blob, const snk_state_layout lay, long long n, int S, int F, int VV) {
  const size_t end[10] = {lay.off_t + 4 * n, lay.off_spare + 4 * n, lay.off_draw_ctr + 4 * n, lay.off_ep_ret + 4 * n,
                          lay.off_ep_len + 4 * n, lay.off_len + 2 * n * S, lay.off_grow_to + 2 * n * S, lay.off_vel + n * S,
                          lay.off_body + 2 * n * S * lay.cap, lay.off_fruit + (lay.fruit_is_grid ? n * VV : 2 * n * F)};
  const size_t next[10] = {lay.off_spare, lay.off_draw_ctr, lay.off_ep_ret, lay.off_ep_len, lay.off_len, lay.off_grow_to,
                           lay.off_vel, lay.off_body, lay.off_fruit, lay.total_bytes};
#pragma unroll
  for (int k = 0; k < 10; ++k)
    for (size_t b = end[k]; b < next[k]; ++b) blob[b] = 0;
}

// private -> canonical.  Lane family: lane w expands chain word w (16 segments, two 16-byte stores of the row); the id of
// its first segment is the head minus the displacement of all earlier words, an exclusive warp scan of the per-word
// displacements (codes_disp).  Word 0 is the record's c0 word; words >= 1 are read only where the body reaches them.
// Ring family: lane l takes 8 consecutive segments (ring_at) per 16-byte store.  Padding zeros are stored too.
__global__ void __launch_bounds__(256) k_save_envs(const Params p, const int64_t* __restrict__ idx, long long first,
                                                   long long count, u8* __restrict__ blob, const snk_state_layout lay) {
  const int lane = threadIdx.x & 31, S = p.S, cap = p.cap, V = p.V;
  if (blockIdx.x == 0 && threadIdx.x == 0) blob_zero_gaps(blob, lay, count, S, p.F, p.VV);
  const long long j = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;  // entry j
  if (j >= count) return;
  long long e;
  if (!entry_env(p, idx, first, j, lane == 0, e)) return;
  const u32* r = p.rec + e * p.RW;
  for (int s = 0; s < S; ++s) {
    const long long u = j * S + s;
    const u32 a = r[REC_SNAKE0 + 2 * s], b = r[REC_SNAKE0 + 2 * s + 1];
    const int len = a >> 16, hs = a & 0xffff;
    if (lane == 0) {
      reinterpret_cast<u16*>(blob + lay.off_len)[u] = (u16)len;
      reinterpret_cast<u16*>(blob + lay.off_grow_to)[u] = (u16)(b & 0xffff);
      (blob + lay.off_vel)[u] = (u8)(b >> 16);
    }
    uint4* dst = reinterpret_cast<uint4*>(blob + lay.off_body + (size_t)u * cap * 2);
    if (p.family == 1) {  // chain code: hs is the head id
      const u32 c0 = r[s < 3 ? 5 + s : p.RW - 2];  // LaneRec::c0_word
      const u32* ch = p.chain + (e * S + s) * p.CW;
      int base = hs;  // id of the first segment of the current 32 words
      for (int w0 = 0; 16 * w0 < cap; w0 += 32) {
        const int w = w0 + lane, k0 = 16 * w;
        const u32 word = k0 < len ? (w == 0 ? c0 : ch[w]) : 0u;
        const int disp = k0 < len ? codes_disp(word, V, 16) : 0;
        const int incl = warp_incl_scan(disp, lane);
        int pid = base - (incl - disp);
        base -= __shfl_sync(FULL, incl, 31);
        u32 o[8];
  #pragma unroll
        for (int q = 0; q < 16; ++q) {
          const u32 v = k0 + q < len ? (u32)pid : 0u;
          o[q >> 1] = (q & 1) ? (o[q >> 1] | (v << 16)) : v;
          pid -= chain_delta((word >> (2 * q)) & 3, V);
        }
        if (k0 + 8 <= cap) dst[2 * w] = make_uint4(o[0], o[1], o[2], o[3]);
        if (k0 + 16 <= cap) dst[2 * w + 1] = make_uint4(o[4], o[5], o[6], o[7]);
      }
    } else {
      const u16* ring = p.body + (e * S + s) * cap;
      for (int k0 = 8 * lane; k0 < cap; k0 += 256) {
        u32 o[4];
  #pragma unroll
        for (int q = 0; q < 8; ++q) {
          const u32 v = k0 + q < len ? (u32)ring_at(ring, hs, k0 + q, cap) : 0u;
          o[q >> 1] = (q & 1) ? (o[q >> 1] | (v << 16)) : v;
        }
        dst[k0 >> 3] = make_uint4(o[0], o[1], o[2], o[3]);
      }
    }
  }
  if (lane == 0) {
    reinterpret_cast<u32*>(blob + lay.off_t)[j] = r[REC_T];
    reinterpret_cast<u32*>(blob + lay.off_spare)[j] = r[REC_SPARE];
    reinterpret_cast<u32*>(blob + lay.off_draw_ctr)[j] = r[REC_DRAW_CTR];
    reinterpret_cast<u32*>(blob + lay.off_ep_ret)[j] = r[REC_EP_RET];
    reinterpret_cast<u32*>(blob + lay.off_ep_len)[j] = r[REC_EP_LEN];
  }
  if (lay.fruit_is_grid) {  // lane family: a count is valid only where its gbits bit is set
    const u8* g = p.grid + e * p.grid_stride;
    const u32* gb = p.family == 1 ? p.gbits + e * p.GBW : nullptr;
    u8* out = blob + lay.off_fruit + (size_t)j * p.VV;
    for (int k = lane; k < p.VV; k += 32) out[k] = (!gb || ((gb[k >> 5] >> (k & 31)) & 1)) ? g[k] : (u8)0;
  } else if (lane < p.F) {
    reinterpret_cast<u16*>(blob + lay.off_fruit)[j * p.F + lane] = reinterpret_cast<const u16*>(r + REC_SNAKE0 + 2 * S)[lane];
  }
}

// canonical -> private, trusting nothing: a body longer than the board, a cell id outside the padded grid, a velocity code
// above 4 or (lane family) two consecutive segments that are not adjacent cells raise SNK_DEVERR_BAD_STATE and leave that
// snake empty; a classic fruit id outside the grid is flagged and replaced by cell (0, 0).  Lane family: lane w reads
// segments 16w .. 16w+16 (two 16-byte loads and its neighbour's first id), builds chain word w and checks its part of the
// body; a warp vote collects the verdict.  Chain words the body does not reach are not written (nothing reads them).
// Clears frame_ok: the own observation buffer no longer shows the env.
__global__ void __launch_bounds__(256) k_restore_envs(const Params p, const int64_t* __restrict__ idx, long long count,
                                                      const u8* __restrict__ blob, const snk_state_layout lay) {
  const int lane = threadIdx.x & 31, S = p.S, cap = p.cap, V = p.V;
  const long long j = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
  if (j >= count) return;
  long long e;
  if (!entry_env(p, idx, 0, j, lane == 0, e)) return;
  u32* r = p.rec + e * p.RW;
  for (int s = 0; s < S; ++s) {
    const long long u = j * S + s;
    u32 len = reinterpret_cast<const u16*>(blob + lay.off_len)[u];
    const u32 grow = reinterpret_cast<const u16*>(blob + lay.off_grow_to)[u];
    u32 vel = (blob + lay.off_vel)[u];
    const uint4* src = reinterpret_cast<const uint4*>(blob + lay.off_body + (size_t)u * cap * 2);
    bool bad = len > (u32)(p.D * p.D + 1) || len > (u32)cap || vel > 4u;
    const int n = bad ? 0 : (int)len;
    u32 c0 = 0, head = 0;
    if (p.family == 1) {
      u32* ch = p.chain + (e * S + s) * p.CW;
      for (int w0 = 0; w0 == 0 || 16 * w0 < n; w0 += 32) {
        const int w = w0 + lane, k0 = 16 * w;
        u32 v[8];
  #pragma unroll
        for (int q = 0; q < 8; ++q) v[q] = 0;
        if (k0 < n || w == 0) {  // word 0 without waiting for len: most bodies fit it
          const uint4 x = src[2 * w];
          v[0] = x.x; v[1] = x.y; v[2] = x.z; v[3] = x.w;
          if (k0 + 8 < n || (w == 0 && cap >= 16)) { const uint4 y = src[2 * w + 1]; v[4] = y.x; v[5] = y.y; v[6] = y.z; v[7] = y.w; }
        }
        int nxt = __shfl_down_sync(FULL, (int)(v[0] & 0xffff), 1);
        if (lane == 31 && k0 + 16 < n) nxt = reinterpret_cast<const u16*>(src)[k0 + 16];
        u32 word = 0;
        bool lbad = false;
  #pragma unroll
        for (int q = 0; q < 16; ++q) {
          const int cur = (int)((v[q >> 1] >> (16 * (q & 1))) & 0xffff);
          const int nx = q < 15 ? (int)((v[(q + 1) >> 1] >> (16 * ((q + 1) & 1))) & 0xffff) : nxt;
          if (k0 + q < n) lbad |= cur >= p.VV;
          if (k0 + q + 1 < n) {
            const int diff = cur - nx;
            lbad |= !(diff == V || diff == 1 || diff == -V || diff == -1);
            word |= (diff == V ? 0u : diff == 1 ? 1u : diff == -V ? 2u : 3u) << (2 * q);
          }
        }
        bad |= __any_sync(FULL, lbad);
        if (w0 == 0) { c0 = __shfl_sync(FULL, word, 0); head = __shfl_sync(FULL, v[0] & 0xffff, 0); }
        if (w >= 1 && k0 + 1 < n) ch[w] = word;  // words holding at least one code
      }
    } else {  // the whole ring row, zeros past the body (as snk_load_state has always written it), head at slot 0
      u16* ring = p.body + (e * S + s) * cap;
      bool lbad = false;
      for (int k0 = 8 * lane; k0 < cap; k0 += 256) {
        u32 v[4] = {0u, 0u, 0u, 0u};
        if (k0 < n) { const uint4 x = src[k0 >> 3]; v[0] = x.x; v[1] = x.y; v[2] = x.z; v[3] = x.w; }
  #pragma unroll
        for (int q = 0; q < 8; ++q) {
          const u32 id = (v[q >> 1] >> (16 * (q & 1))) & 0xffff;
          if (k0 + q >= n) v[q >> 1] &= (q & 1) ? 0x0000ffffu : 0xffff0000u;
          else lbad |= id >= (u32)p.VV;
        }
        reinterpret_cast<uint4*>(ring)[k0 >> 3] = make_uint4(v[0], v[1], v[2], v[3]);
      }
      bad |= __any_sync(FULL, lbad);
    }
    if (bad) { len = 0; vel = 0; c0 = 0; }
    if (lane == 0) {
      if (bad) atomicOr(p.err, SNK_DEVERR_BAD_STATE);
      r[REC_SNAKE0 + 2 * s] = (p.family == 1 && len ? head : 0u) | (len << 16);
      r[REC_SNAKE0 + 2 * s + 1] = grow | (vel << 16);
      if (p.family == 1) r[s < 3 ? 5 + s : p.RW - 2] = c0;  // LaneRec::c0_word
    }
  }
  if (lane == 0) {
    r[REC_T] = reinterpret_cast<const u32*>(blob + lay.off_t)[j];
    r[REC_SPARE] = reinterpret_cast<const u32*>(blob + lay.off_spare)[j];
    r[REC_DRAW_CTR] = reinterpret_cast<const u32*>(blob + lay.off_draw_ctr)[j];
    r[REC_EP_RET] = reinterpret_cast<const u32*>(blob + lay.off_ep_ret)[j];
    r[REC_EP_LEN] = reinterpret_cast<const u32*>(blob + lay.off_ep_len)[j];
    if (p.family == 0) r[5] = r[6] = r[7] = 0;
    if (p.frame_ok) p.frame_ok[e] = 0;
  }
  if (lay.fruit_is_grid) {  // counts, and the lane family's bitmap of the cells whose count is > 0 (one vote per word)
    u8* g = p.grid + e * p.grid_stride;
    const u8* in = blob + lay.off_fruit + (size_t)j * p.VV;
    for (int c = 0; 32 * c < p.VV; ++c) {
      const int k = 32 * c + lane;
      const u8 v = k < p.VV ? in[k] : (u8)0;
      if (k < p.VV) g[k] = v;
      const u32 bits = __ballot_sync(FULL, v != 0);
      if (p.family == 1 && lane == 0) p.gbits[e * p.GBW + c] = bits;
    }
  } else if (lane < p.F) {
    u16 f = reinterpret_cast<const u16*>(blob + lay.off_fruit)[j * p.F + lane];
    if (f >= (u32)p.VV) { atomicOr(p.err, SNK_DEVERR_BAD_STATE); f = (u16)(p.V + 1); }
    reinterpret_cast<u16*>(r + REC_SNAKE0 + 2 * S)[lane] = f;
  }
}

// private -> private, one warp per (src, dst) pair: the record, the chain words >= 1 each body reaches (lane family) or the
// whole ring row (ring family), the fruit count grid and the lane family's fruit bitmap; clears frame_ok[dst].  Env src[j]
// of handle `ps` into env dst[j] of handle `pd`: the same handle for snk_copy_envs, two handles of one private layout
// (family, RW, CW, cap, grid_stride, GBW, checked by snk_clone_envs) otherwise.  `ps` is only read.
__global__ void k_copy_envs(const Params ps, const Params pd, const int64_t* __restrict__ src,
                            const int64_t* __restrict__ dst, long long count) {
  const int lane = threadIdx.x & 31, S = pd.S;
  const long long j = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
  if (j >= count) return;
  const long long es = src[j], ed = dst[j];
  if (es < 0 || es >= ps.N || ed < 0 || ed >= pd.N) {
    if (lane == 0) atomicOr(pd.err, SNK_DEVERR_BAD_STATE);
    return;
  }
  const u32* rs = ps.rec + es * pd.RW;
  u32* rd = pd.rec + ed * pd.RW;
  for (int w = lane; w < pd.RW; w += 32) rd[w] = rs[w];
  if (pd.family == 1) {
    for (int s = 0; s < S; ++s) {
      const int len = rs[REC_SNAKE0 + 2 * s] >> 16;
      const int nw = len >= 2 ? ((len - 2) >> 4) + 1 : 0;  // words holding codes 0 .. len-2; word 0 is in the record
      const u32* cs = ps.chain + (es * S + s) * pd.CW;
      u32* cd = pd.chain + (ed * S + s) * pd.CW;
      for (int w = 1 + lane; w < nw; w += 32) cd[w] = cs[w];
    }
    if (lane == 0) pd.frame_ok[ed] = 0;
  } else {
    const uint4* bs = reinterpret_cast<const uint4*>(ps.body + es * S * pd.cap);
    uint4* bd = reinterpret_cast<uint4*>(pd.body + ed * S * pd.cap);
    for (int k = lane; k < S * pd.cap / 8; k += 32) bd[k] = bs[k];
  }
  if (pd.grid) {
    const uint4* gs = reinterpret_cast<const uint4*>(ps.grid + es * pd.grid_stride);
    uint4* gd = reinterpret_cast<uint4*>(pd.grid + ed * pd.grid_stride);
    for (int k = lane; k < pd.grid_stride / 16; k += 32) gd[k] = gs[k];
    if (pd.gbits)
      for (int w = lane; w < pd.GBW; w += 32) pd.gbits[ed * pd.GBW + w] = ps.gbits[es * pd.GBW + w];
  }
}

// ------------------------------------------------------------------ action stream, views
// The first n_out views of every pixel, packed: [pixels][3K] -> [pixels][3 n_out].  Used by the host-buffer step when
// the caller only keeps the main snake's view (ppo_multi_agent_new.py:181 stores obs[..., 0:3] alone: the D2H copy then
// carries n_out / K of the bytes) and by snk_set_main_view_target (the learner's rollout slot).
// k_extract_main<C>: the main view alone (n_out = 1) for C = 6 / 9 / 12 bytes per pixel.  A thread takes 16 pixels:
// C 16-byte loads (its 16 C contiguous bytes), twelve output words assembled with byte permutes whose selectors are
// compile-time constants, three 16-byte stores.  HBM-bound: reads N V V 3K, writes N V V 3.  (The first form, one thread
// per 4 pixels with byte loads, took 173 us per 131 072 envs of 2x19x19 -- 2.6x the step kernel it follows.)
template <int C>
__global__ void __launch_bounds__(256) k_extract_main(const uint4* __restrict__ src, uint4* __restrict__ dst, long long n16) {
  const long long g = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (g >= n16) return;
  u32 w[4 * C];
#pragma unroll
  for (int i = 0; i < C; ++i) {
    const uint4 v = __ldcs(src + g * C + i);  // streamed: every byte is read once
    w[4 * i] = v.x; w[4 * i + 1] = v.y; w[4 * i + 2] = v.z; w[4 * i + 3] = v.w;
  }
  u32 o[12];
#pragma unroll
  for (int k = 0; k < 12; ++k) {
    // output byte t = 4k + b is channel t % 3 of pixel t / 3, i.e. input byte (t / 3) * C + t % 3
    const int i0 = ((4 * k) / 3) * C + (4 * k) % 3, i1 = ((4 * k + 1) / 3) * C + (4 * k + 1) % 3;
    const int i2 = ((4 * k + 2) / 3) * C + (4 * k + 2) % 3, i3 = ((4 * k + 3) / 3) * C + (4 * k + 3) % 3;
    const u32 lo = __byte_perm(w[i0 >> 2], w[i1 >> 2], (u32)((i0 & 3) | (((i1 & 3) + 4) << 4)));
    const u32 hi = __byte_perm(w[i2 >> 2], w[i3 >> 2], (u32)((i2 & 3) | (((i3 & 3) + 4) << 4)));
    o[k] = __byte_perm(lo, hi, 0x5410u);
  }
  dst[g * 3] = make_uint4(o[0], o[1], o[2], o[3]);
  dst[g * 3 + 1] = make_uint4(o[4], o[5], o[6], o[7]);
  dst[g * 3 + 2] = make_uint4(o[8], o[9], o[10], o[11]);
}

// general form (any C, n_out <= 4, ragged tails, unaligned destinations): one thread per 4 pixels
__global__ void k_extract_views(const u8* __restrict__ src, u8* __restrict__ dst, long long px_first, long long n_pixels, int C, int n_out) {
  const long long g = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  const long long px0 = px_first + g * 4;
  if (px0 >= n_pixels) return;
  const int CO = 3 * n_out;
  if (px0 + 4 <= n_pixels && (reinterpret_cast<uintptr_t>(dst) & 3) == 0) {
    u32 w[12];  // n_out <= 4
    u8* b = reinterpret_cast<u8*>(w);
    for (int q = 0; q < 4; ++q)
      for (int j = 0; j < CO; ++j) b[q * CO + j] = src[(px0 + q) * C + j];
    u32* d = reinterpret_cast<u32*>(dst + px0 * CO);
    for (int j = 0; j < CO; ++j) d[j] = w[j];
  } else {  // the ragged tail, or a destination that is not word aligned (an odd slot of an odd-sized rollout buffer)
    for (long long q = px0; q < n_pixels && q < px0 + 4; ++q)
      for (int j = 0; j < CO; ++j) dst[q * CO + j] = src[q * C + j];
  }
}

// ------------------------------------------------------------------ SNK_OBS_GRID -> RGB views (snk_expand_views)
// A pure write stream: one code byte in, 3 n_views bytes out per cell.  The colours of one cell: `other` for every view
// but the one of its own snake, `own` for that view, whose index relative to first_view is `rel` (-1 / out of range:
// none).  Packed R | G << 8 | B << 16 like snake_rgb.
__device__ __forceinline__ void cell_colours(u32 c, int first_view, u32& other, u32& own, int& rel) {
  other = c == SNK_CELL_FRUIT ? 255u : c == SNK_CELL_WALL ? 0xffffffu : 0u;
  own = other;
  rel = -1;
  if (c >= 3 && c != SNK_CELL_WALL) {
    other = snake_rgb(false, (c - 3) & 1);
    own = snake_rgb(true, (c - 3) & 1);
    rel = (int)((c - 3) >> 1) - first_view;
  }
}

// k_expand_views<NV>: NV views, compile time.  A thread takes P cells, the fewest whose P * 3 NV output bytes are whole
// 16-byte words (NV = 1: 16 cells, 2: 8, 3: 16, 16: 1), so the byte positions of the period fold to constants.  The warp
// stages its 32 periods in shared memory and stores them as consecutive 16-byte words: one 512-byte run per store
// instruction instead of 32 pieces 3 NV * P bytes apart.  B200, 131 072 envs of 21x21: 2 views 95.7 -> 90.3 us, 3 views
// 184.5 -> 102.4, 16 views 717 -> 543; one view 57.2 -> 64.3 (DESIGN.md section 4.15).
template <int NV>
__global__ void __launch_bounds__(256) k_expand_views(const u8* __restrict__ grid, uint4* __restrict__ out, long long n_periods, int first_view) {
  constexpr int C = 3 * NV, P = 16 / (C % 16 == 0 ? 16 : C % 8 == 0 ? 8 : C % 4 == 0 ? 4 : C % 2 == 0 ? 2 : 1), W = P * C / 4, Q = W / 4;
  __shared__ uint4 s_out[8][32 * Q];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long g = blockIdx.x * (long long)blockDim.x + threadIdx.x, g0 = g - lane;
  if (g0 >= n_periods) return;  // warp-uniform
  if (g < n_periods) {
    u32 other[P], own[P];
    int rel[P];
#pragma unroll
    for (int q = 0; q < P; ++q) cell_colours(__ldg(grid + g * P + q), first_view, other[q], own[q], rel[q]);
    u32 w[W];
#pragma unroll
    for (int i = 0; i < W; ++i) {
      u32 v = 0;
#pragma unroll
      for (int b = 0; b < 4; ++b) {
        const int j = 4 * i + b, q = j / C, view = (j % C) / 3, ch = j % 3;
        v |= (((rel[q] == view ? own[q] : other[q]) >> (8 * ch)) & 0xffu) << (8 * b);
      }
      w[i] = v;
    }
#pragma unroll
    for (int i = 0; i < Q; ++i) s_out[warp][lane * Q + i] = make_uint4(w[4 * i], w[4 * i + 1], w[4 * i + 2], w[4 * i + 3]);
  }
  __syncwarp();
  const int n16 = (int)min(32LL, n_periods - g0) * Q;
  for (int i = lane; i < n16; i += 32) __stcs(out + g0 * Q + i, s_out[warp][i]);
}

// any view count, ragged tails, unaligned destinations: one thread per cell, byte stores
__global__ void k_expand_views_any(const u8* __restrict__ grid, u8* __restrict__ out, long long first_cell, long long n_cells,
                                   int first_view, int n_views) {
  const long long i = first_cell + blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= n_cells) return;
  u32 other, own;
  int rel;
  cell_colours(__ldg(grid + i), first_view, other, own, rel);
  u8* px = out + i * 3 * n_views;
  for (int k = 0; k < n_views; ++k) {
    const u32 v = k == rel ? own : other;
    px[3 * k] = (u8)v; px[3 * k + 1] = (u8)(v >> 8); px[3 * k + 2] = (u8)(v >> 16);
  }
}

// snk_get_stats_global in the peer-memory form: push the rank's CURRENT sums to the peers (the final step's, which no
// later step would push) and add up the own sums and what the peers have pushed so far
__global__ void k_sum_inbox(const PeerArgs a, const double* __restrict__ stats, double* __restrict__ glob) {
  const int k = threadIdx.x;
  if (k >= SNK_NSTATS) return;
  const double v = __ldcg(stats + k);
  double sum = v;
  for (int g = 0; g < a.ranks; ++g) {
    if (g == a.rank) continue;
    reinterpret_cast<volatile double*>(a.inbox[g] + (size_t)a.rank * SNK_INBOX_STRIDE)[k] = v;
    sum += reinterpret_cast<const volatile double*>(a.inbox[a.rank] + (size_t)g * SNK_INBOX_STRIDE)[k];
  }
  glob[k] = sum;
}

__global__ void k_gen_actions(int8_t* actions, long long N, int S, long long env_id_base, u64 step, u64 seed, int n_actions) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= N * S) return;
  const long long e = i / S;
  const int s = (int)(i - e * S);
  actions[i] = (int8_t)philox_bounded(seed, (u64)(env_id_base + e), 1, step * (u64)S + (u64)s, (u32)n_actions);
}

#endif  // misc kernels

// ------------------------------------------------------------------ launchers
// (S, K) pairs the lane kernel is compiled for: one view per snake, or the 3 views SnakeEnv emits
#ifdef LANE_COMBOS_OVERRIDE  // quick A/B builds (tools/build_variant.sh): the two bench shapes only
#define LANE_COMBOS(X) X(2, 2) X(3, 3)
#else
#define LANE_COMBOS(X) X(1, 1) X(2, 2) X(3, 3) X(4, 4) X(1, 3) X(2, 3)
#endif

#if SNK_TU == -1 || SNK_TU == 3
bool snk_lane_supported(int S, int K) {
#define X(s, k) if (S == s && K == k) return true;
  LANE_COMBOS(X)
#undef X
  return false;
}
#endif

// SNK_OBS_GRID, lane family: k_lane_logic + k_lane_grid, instantiated per snake count (the views do not enter)
#define GRID_SNAKES(X) X(1) X(2) X(3) X(4)

// plan.logic and plan.kernel of plan.form for S snakes and K views under RULES
template <int RULES>
cudaError_t resolve(LaunchPlan& plan, int S, int K) {
  const void* logic = nullptr;
  const void* kernel = nullptr;
  switch (plan.form) {
    case FORM_LANE:
    case FORM_LANE_WS:
    case FORM_LANE_SPLIT:
#define X(s, k)                                                                  \
  if (S == s && K == k) {                                                        \
    if (plan.form == FORM_LANE) {                                                \
      kernel = (const void*)k_step_lane<s, RULES, k>;                            \
    } else if (plan.form == FORM_LANE_WS) {                                      \
      kernel = (const void*)k_step_lane_ws<s, RULES, k>;                         \
    } else {                                                                     \
      logic = (const void*)k_lane_logic<s, RULES>;                               \
      kernel = (const void*)k_lane_paint2<s, RULES, k>;                          \
    }                                                                            \
  }
      LANE_COMBOS(X)
#undef X
      break;
    case FORM_LANE_GRID:
#define X(s)                                     \
  if (S == s) {                                  \
    logic = (const void*)k_lane_logic<s, RULES>; \
    kernel = (const void*)k_lane_grid<s, RULES>; \
  }
      GRID_SNAKES(X)
#undef X
      break;
    case FORM_TILE: kernel = plan.block <= 256 ? (const void*)k_step_tile<RULES, 256> : (const void*)k_step_tile<RULES, 512>; break;
    case FORM_DENSE: kernel = (const void*)k_step_dense<RULES>; break;
    case FORM_ROWS: kernel = (const void*)k_step_rows<RULES, false>; break;
    case FORM_ROWS_GRID: kernel = (const void*)k_step_rows<RULES, true>; break;
  }
  plan.logic = logic;
  plan.kernel = kernel;
  return kernel ? cudaSuccess : cudaErrorInvalidConfiguration;
}

#if SNK_TU >= 0 && SNK_TU <= 2
template cudaError_t resolve<SNK_TU>(LaunchPlan&, int, int);
#elif SNK_TU == 3
extern template cudaError_t resolve<SNK_RULES_CLASSIC>(LaunchPlan&, int, int);
extern template cudaError_t resolve<SNK_RULES_ADVERSARIAL>(LaunchPlan&, int, int);
extern template cudaError_t resolve<SNK_RULES_CUT>(LaunchPlan&, int, int);
#endif
#if SNK_TU == -1 || SNK_TU == 3
cudaError_t snk_plan(int rules, LaunchPlan& plan, int n_sm, int S, int K, long long work) {
  cudaError_t err = rules == SNK_RULES_CLASSIC       ? resolve<SNK_RULES_CLASSIC>(plan, S, K)
                    : rules == SNK_RULES_ADVERSARIAL ? resolve<SNK_RULES_ADVERSARIAL>(plan, S, K)
                                                     : resolve<SNK_RULES_CUT>(plan, S, K);
  if (err) return err;
  // programmatic launches for the fused kernel and both kernels of the two-kernel forms; the warp-specialised, tile,
  // dense and rows kernels launch without
  plan.pdl = plan.form == FORM_LANE || plan.form == FORM_LANE_SPLIT || plan.form == FORM_LANE_GRID;
  int occ = 0;
  if ((err = cudaFuncSetAttribute(plan.kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)plan.smem))) return err;
  if ((err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, plan.kernel, plan.block, plan.smem))) return err;
  if (occ < 1) return cudaErrorInvalidConfiguration;
  plan.occupancy = occ;
  plan.max_grid = n_sm * occ;
  plan.grid = (int)(work < plan.max_grid ? work : plan.max_grid);
  if (plan.grid < 1) plan.grid = 1;
  return cudaSuccess;
}

cudaError_t snk_launch_step(const Params& p, const LaunchPlan& plan, cudaStream_t stream) {
  // programmatic launches: a kernel's prologue overlaps the tail of the launch before it
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cudaLaunchConfig_t cfg = {};
  cfg.stream = stream;
  cfg.attrs = attr;
  cfg.numAttrs = plan.pdl ? 1 : 0;
  void* args[] = {const_cast<Params*>(&p)};
  if (plan.logic && p.mode != MODE_OBSERVE) {  // thread per env
    cfg.gridDim = dim3((unsigned)((p.N + 127) / 128));
    cfg.blockDim = dim3(128);
    cudaError_t err = cudaLaunchKernelExC(&cfg, plan.logic, args);
    if (err != cudaSuccess) return err;
  }
  cfg.gridDim = dim3(plan.grid);
  cfg.blockDim = dim3(plan.block);
  cfg.dynamicSmemBytes = plan.smem;
  return cudaLaunchKernelExC(&cfg, plan.kernel, args);
}

cudaError_t snk_launch_upscale84(const uint8_t* native, uint8_t* out, long long N, int V, int C, int n_sm, cudaStream_t stream) {
  const int r = 84 / V;
  if (C == 6 && r == 4) return launch_upscale<6, 4>(native, out, N, V, C, n_sm, stream);   // 2 views of 21x21 (the headline board)
  if (C == 12 && r == 4) return launch_upscale<12, 4>(native, out, N, V, C, n_sm, stream);  // 4 views of 21x21
  if (C == 6 && r == 7) return launch_upscale<6, 7>(native, out, N, V, C, n_sm, stream);    // 2 views of 12x12
  if (C == 9 && r == 7) return launch_upscale<9, 7>(native, out, N, V, C, n_sm, stream);    // 3 views of 12x12 (SnakeEnv's K = 3)
  if (C == 9 && r == 4) return launch_upscale<9, 4>(native, out, N, V, C, n_sm, stream);    // 3 views of 21x21
  if (C == 3 && r == 7) return launch_upscale<3, 7>(native, out, N, V, C, n_sm, stream);
  if (C == 3 && r == 4) return launch_upscale<3, 4>(native, out, N, V, C, n_sm, stream);
  return launch_upscale<0, 0>(native, out, N, V, C, n_sm, stream);
}

cudaError_t snk_launch_save(const Params& p, const int64_t* idx, long long first, long long count, u8* blob,
                            const snk_state_layout& lay, cudaStream_t stream) {
  k_save_envs<<<(unsigned)((count + 7) / 8), 256, 0, stream>>>(p, idx, first, count, blob, lay);
  return cudaGetLastError();
}

cudaError_t snk_launch_restore(const Params& p, const int64_t* idx, long long count, const u8* blob, const snk_state_layout& lay,
                               cudaStream_t stream) {
  k_restore_envs<<<(unsigned)((count + 7) / 8), 256, 0, stream>>>(p, idx, count, blob, lay);
  return cudaGetLastError();
}

cudaError_t snk_launch_copy(const Params& ps, const Params& pd, const int64_t* src, const int64_t* dst, long long count,
                            cudaStream_t stream) {
  k_copy_envs<<<(unsigned)((count + 7) / 8), 256, 0, stream>>>(ps, pd, src, dst, count);
  return cudaGetLastError();
}

cudaError_t snk_launch_sum_inbox(const PeerArgs& a, const double* stats, double* glob, cudaStream_t stream) {
  k_sum_inbox<<<1, 32, 0, stream>>>(a, stats, glob);
  return cudaGetLastError();
}



cudaError_t snk_launch_extract_views(const uint8_t* src, uint8_t* dst, long long n_pixels, int C, int n_out, cudaStream_t stream) {
  long long done = 0;
  const bool aligned = ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) & 15) == 0;
  if (n_out == 1 && aligned && (C == 6 || C == 9 || C == 12) && n_pixels >= 16) {
    const long long n16 = n_pixels / 16;
    const unsigned grid = (unsigned)((n16 + 255) / 256);
    const uint4* s4 = reinterpret_cast<const uint4*>(src);
    uint4* d4 = reinterpret_cast<uint4*>(dst);
    if (C == 6) k_extract_main<6><<<grid, 256, 0, stream>>>(s4, d4, n16);
    else if (C == 9) k_extract_main<9><<<grid, 256, 0, stream>>>(s4, d4, n16);
    else k_extract_main<12><<<grid, 256, 0, stream>>>(s4, d4, n16);
    done = n16 * 16;
    if (done == n_pixels) return cudaGetLastError();
  }
  const long long n = (n_pixels - done + 3) / 4;
  k_extract_views<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(src, dst, done, n_pixels, C, n_out);
  return cudaGetLastError();
}

template <int NV>
static long long launch_expand(const u8* grid, long long n_cells, int first_view, u8* out, cudaStream_t stream) {
  constexpr int C = 3 * NV, P = 16 / (C % 16 == 0 ? 16 : C % 8 == 0 ? 8 : C % 4 == 0 ? 4 : C % 2 == 0 ? 2 : 1);
  const long long n_periods = n_cells / P;
  if (n_periods > 0)
    k_expand_views<NV><<<(unsigned)((n_periods + 255) / 256), 256, 0, stream>>>(grid, reinterpret_cast<uint4*>(out), n_periods, first_view);
  return n_periods * P;
}

cudaError_t snk_launch_expand_views(const uint8_t* grid, long long n_cells, int first_view, int n_views, uint8_t* out, cudaStream_t stream) {
  long long done = 0;
  if ((reinterpret_cast<uintptr_t>(out) & 15) == 0) {
    switch (n_views) {
      case 1: done = launch_expand<1>(grid, n_cells, first_view, out, stream); break;
      case 2: done = launch_expand<2>(grid, n_cells, first_view, out, stream); break;
      case 3: done = launch_expand<3>(grid, n_cells, first_view, out, stream); break;
      case 16: done = launch_expand<16>(grid, n_cells, first_view, out, stream); break;
      default: break;
    }
  }
  if (done < n_cells) {
    const long long n = n_cells - done;
    k_expand_views_any<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(grid, out, done, n_cells, first_view, n_views);
  }
  return cudaGetLastError();
}

cudaError_t snk_launch_scripted_actions(const Params& p, int8_t* actions, u64 step, u64 seed, int eps_permille, const uint8_t* occ_obs,
                                        cudaStream_t stream) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)((p.N + 127) / 128)); cfg.blockDim = dim3(128); cfg.dynamicSmemBytes = 0; cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  switch (p.S) {
    case 1: return cudaLaunchKernelEx(&cfg, k_scripted_actions<1>, p, actions, step, seed, eps_permille, occ_obs);
    case 2: return cudaLaunchKernelEx(&cfg, k_scripted_actions<2>, p, actions, step, seed, eps_permille, occ_obs);
    case 3: return cudaLaunchKernelEx(&cfg, k_scripted_actions<3>, p, actions, step, seed, eps_permille, occ_obs);
    default: return cudaLaunchKernelEx(&cfg, k_scripted_actions<4>, p, actions, step, seed, eps_permille, occ_obs);
  }
  return cudaGetLastError();
}

cudaError_t snk_launch_gae(const float* rewards, const float* values, const uint8_t* dones, const float* last_values,
                           const uint8_t* last_dones, double gamma, double lam, int T, long long N, float* advs, float* returns,
                           cudaStream_t stream) {
  k_gae<<<(unsigned)((N + 127) / 128), 128, 0, stream>>>(rewards, values, dones, last_values, last_dones, gamma, lam, T, N, advs, returns);
  return cudaGetLastError();
}

cudaError_t snk_launch_gen_actions(int8_t* actions, long long N, int S, long long env_id_base, u64 step, u64 seed,
                                   int n_actions, cudaStream_t stream) {
  const long long n = N * S;
  k_gen_actions<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(actions, N, S, env_id_base, step, seed, n_actions);
  return cudaGetLastError();
}
#endif  // host dispatch
