// snk_device.cuh -- device-side building blocks of the fused env-step kernels (sm_100a).
//
// Everything here is warp-cooperative: one warp owns one env.  Scalar game logic runs
// warp-uniform (all 32 lanes compute the same values, no divergence); every scan over body
// segments, fruits or bitmap words is lane-parallel.  What each function reproduces is cited
// against the reference (/root/reference/src/gym-snake/gym_snake/envs/snake_multiple_test.py
// unless another file is named).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/snk.h"

typedef uint8_t u8;
typedef uint16_t u16;
typedef uint32_t u32;
typedef uint64_t u64;

#define FULL 0xffffffffu
#define SNK_MAX_PEERS 16        // ranks of one node that can share statistics through peer memory
#define SNK_INBOX_STRIDE 64     // bytes per sender in an inbox: its SNK_NSTATS running sums

// ---- private per-env record (u32 words); snakes start at word REC_SNAKE0, two words each:
//      word A = head_slot | len << 16, word B = grow_to | vel << 16; classic fruits follow as u16.
#define REC_T 0
#define REC_EP_LEN 1
#define REC_DRAW_CTR 2
#define REC_EP_RET 3
#define REC_SPARE 4
#define REC_SNAKE0 8

enum { MODE_STEP = 0, MODE_RESET = 1, MODE_OBSERVE = 2 };

// peer-memory form of the statistics reduction (snk_peer_connect): every rank's inbox as mapped into this process
struct PeerArgs {
  int ranks, rank;              // ranks == 0: off
  u8* inbox[SNK_MAX_PEERS];     // cudaIpc mappings; [rank] is the local one
};

struct Params {
  int D, V, VV, S, F, K, C;     // C = 3K bytes per pixel
  int cap, RW, E;               // ring capacity, record words, obs bytes per env
  int G, W;                     // envs per 16-byte-aligned obs group, warps (envs) per CTA
  int grid_stride, bm_words;    // bytes per env of the fruit count grid, words of the spawn bitmap
  int GBW;                      // lane family: words of the per-env fruit bitmap (adversarial / cut)
  int family, CW;               // 0 = ring bodies (tile / dense kernels), 1 = chain-coded bodies (lane kernel); chain words per snake
  int TE, tile_stride;          // lane kernel: envs per warp image, bytes between warp images
  int EPW;                      // fused lane kernel: envs stepped per warp batch (32; 16/8/4 when the shard is too small to give every resident warp a batch)
  int R;                        // rows kernel: image rows per chunk buffer
  u32 magicV, magicD;           // n / V == (n * magicV) >> 16 for n < V*V, n / D likewise for n < D*D (65536 / d + 1; exact while n * d < 65536)
  int restore_thr;              // lane kernel: un-paint an image by zero-fill + border redraw when a lane would walk more segments than this (0 = always walk)
  int delta;                    // lane family (fused and two-kernel form), classic step into the own buffer: an image whose envs all have frame_ok stores only the 32-byte sectors the step can change
  int frame_own;                // this launch writes a complete image of every env into the handle's own observation buffer (lane_store writes it to frame_ok)
  int max_steps, auto_reset, rng_mode, mode;
  long long N, env_id_base, n_groups;
  u64 seed;
  u32* rec;
  u16* body;
  u32* chain;                   // [N][S][CW] 2-bit directions, 16 per word (lane kernel)
  u8* grid;
  u32* gbits;                   // [N][GBW] lane family: bit per padded cell, set = fruit count valid and > 0
  const int8_t* actions;
  const u8* mask;
  u8* obs;
  u8* frame_ok;                 // [N] lane family: 1 = the own observation buffer holds exactly the image of the env's record
                                // (with `delta`, followed by the two-kernel form's DeltaPrev entries: delta_prev(); allocated whenever the handle's `delta` is set)
  float* reward;
  float* reward_all;
  u8* done;
  u8* num_alive;
  float* fin_ret;
  int32_t* fin_len;
  double* stats;
  double* snap;                 // per-step copy of `stats` written by the last CTA of a step kernel (NULL: no per-step reduction)
  u32* ticket;                  // arrival counter behind `snap`
  double* regime_out;           // mapped host memory [2]: running env-steps / body cells, posted by the first CTA of every step (NULL: off)
  PeerArgs peer;                // peer-memory form: the first CTA of every step pushes the running sums to the peers
  u32* err;
  const u32* tape_vals;
  const u32* tape_bounds;
  const u64* tape_off;
  const u32* cellinfo;  // [VV] bit31 = outside the board, low bits = y*D+x (or 0x7fffffff: aliases nothing)
  const u16* idx2pid;   // [D*D] y-major board index -> padded id
  const u8* tmpl;       // [G*E] border-only observation of one group
};

struct WarpStats {
  float steps, episodes, ret_sum, len_sum, fruits, deaths, cells, draws;
};

// ------------------------------------------------------------------ Philox4x32-10
struct Philox4 { u32 w[4]; };

// not inlined: ~100 instructions, called from many (rare) sites; inlining it bloated the step kernels past the I-cache
static __device__ __noinline__ Philox4 philox_block(u32 c0, u32 c1, u32 c2, u32 c3, u32 k0, u32 k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const u32 hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const u32 hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    c0 = hi1 ^ c1 ^ k0; c1 = lo1; c2 = hi0 ^ c3 ^ k1; c3 = lo0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  Philox4 o; o.w[0] = c0; o.w[1] = c1; o.w[2] = c2; o.w[3] = c3;
  return o;
}

// Draw `index` of stream (seed, env_id, stream): one Philox block (counter = index >> 2) serves four
// consecutive draws (word = index & 3); bounded by hi32(x * n).
__device__ __forceinline__ u32 philox_bounded(u64 seed, u64 env_id, u32 stream, u64 index, u32 n) {
  const u64 blk = index >> 2;
  const Philox4 o = philox_block((u32)blk, (u32)(blk >> 32), stream, (u32)(seed >> 32), (u32)seed, (u32)env_id);
  const u32 sel = (u32)index & 3;
  const u32 x = sel == 0 ? o.w[0] : sel == 1 ? o.w[1] : sel == 2 ? o.w[2] : o.w[3];
  return __umulhi(x, n);
}

// Draw number `idx` of env e, bounded by n: np_random.randint(n) at :200 and :215, either
// replayed from the recorded tape or generated by the counter-based production RNG.
__device__ __forceinline__ u32 draw_at(const Params& p, long long e, u32 idx, u32 n, u32& errs) {
  if (p.rng_mode == SNK_RNG_TAPE) {
    const u64 pos = p.tape_off[e] + idx;
    if (pos >= p.tape_off[e + 1]) { errs |= SNK_DEVERR_TAPE_UNDERRUN; return 0; }
    if (p.tape_bounds && p.tape_bounds[pos] != n) errs |= SNK_DEVERR_TAPE_BOUND;
    return p.tape_vals[pos];
  }
  return philox_bounded(p.seed, (u64)(p.env_id_base + e), 0, idx, n);
}

__device__ __forceinline__ int warp_sum(int v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
  return v;
}

__device__ __forceinline__ int warp_incl_scan(int v, int lane) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int n = __shfl_up_sync(FULL, v, o);
    if (lane >= o) v += n;
  }
  return v;
}

__device__ __forceinline__ int ring_at(const u16* ring, int hs, int i, int cap) {
  int slot = hs + i;
  if (slot >= cap) slot -= cap;
  return ring[slot];
}

// Flattened view of the bodies of one env: lane j holds len_j (0 for lanes >= S); segment t of the
// concatenation belongs to snake j = #{k : incl_k <= t}, at index i = t - (incl_j - len_j).
struct SegScan {
  int incl, total;
};
__device__ __forceinline__ SegScan seg_scan(int my_len, int lane) {
  SegScan sg;
  sg.incl = warp_incl_scan(my_len, lane);
  sg.total = __shfl_sync(FULL, sg.incl, 31);
  return sg;
}
// every lane must call it (shuffles); returns false for t >= total (j, i are then valid dummies: 0, 0)
__device__ __forceinline__ bool seg_locate(const SegScan& sg, int my_len, int S, int t, int& j, int& i) {
  const bool have = t < sg.total;
  j = 0;
  for (int k = 0; k < S; ++k) j += (__shfl_sync(FULL, sg.incl, k) <= t) ? 1 : 0;
  if (!have) j = 0;
  const int excl = __shfl_sync(FULL, sg.incl - my_len, j);
  i = have ? t - excl : 0;
  return have;
}

__device__ __forceinline__ void grid_inc(u8* grid, int pid, u32& errs) {
  const u8 c = grid[pid];
  if (c == 255) errs |= SNK_DEVERR_FRUIT_OVERFLOW; else grid[pid] = c + 1;
}

// safe_choose_cell (:202-217): k-th free board index in y-major order, every live body cell
// removed WITHOUT a bounds check (cellinfo holds the aliased index of out-of-board heads); no
// draw when nothing is free.  Warp-cooperative; bm = per-warp bitmap scratch in shared memory.
static __device__ __noinline__ int spawn_cell(const Params& p, long long e, int lane, const u32* sc, u32* bm, const u16* rings,
                          u32& ctr, u32& errs, WarpStats& st) {
  const int S = p.S, cap = p.cap, DD = p.D * p.D, nW = p.bm_words;
  for (int w = lane; w < nW; w += 32) bm[w] = 0;
  __syncwarp();
  for (int s = 0; s < S; ++s) {
    const u32 a = sc[REC_SNAKE0 + 2 * s];
    const int len = a >> 16, hs = a & 0xffff;
    for (int i = lane; i < len; i += 32) {
      const u32 idx = __ldg(p.cellinfo + ring_at(rings + s * cap, hs, i, cap)) & 0x7fffffffu;
      if (idx < (u32)DD) atomicOr(&bm[idx >> 5], 1u << (idx & 31));
    }
  }
  __syncwarp();
  int total = 0;
  for (int w0 = 0; w0 < nW; w0 += 32) {
    const int w = w0 + lane;
    u32 fr = 0;
    if (w < nW) { fr = ~bm[w]; if (w == nW - 1 && (DD & 31)) fr &= (1u << (DD & 31)) - 1; }
    total += warp_sum(__popc(fr));
  }
  if (total == 0) return 1 * p.V + 1;  // (0,0); the reference does not draw here
  const int k = (int)draw_at(p, e, ctr, (u32)total, errs);
  ctr++; st.draws += 1.f;
  int running = 0, found = 0;
  for (int w0 = 0; w0 < nW; w0 += 32) {
    const int w = w0 + lane;
    u32 fr = 0;
    if (w < nW) { fr = ~bm[w]; if (w == nW - 1 && (DD & 31)) fr &= (1u << (DD & 31)) - 1; }
    const int cnt = __popc(fr);
    const int incl = warp_incl_scan(cnt, lane);
    const int lo = running + incl - cnt;
    const bool mine = k >= lo && k < lo + cnt;
    const int idx = mine ? w * 32 + (int)__fns(fr, 0, k - lo + 1) : 0;
    const u32 who = __ballot_sync(FULL, mine);
    if (who) { found = __shfl_sync(FULL, idx, __ffs(who) - 1); break; }
    running += __shfl_sync(FULL, incl, 31);
  }
  return p.idx2pid[found];
}

// reset (:219-232): snake_i.x, snake_i.y, fruit_i.x, fruit_i.y interleaved, each randint(D), no
// overlap checks; grow_to 3, vel (0,0), t 0.  Lanes draw in parallel (draw q has index ctr + q).
// Monitor accumulators are cleared; adversarial `spare` survives (snake_adversarial_env.py:14).
template <int RULES>
__device__ void reset_env_warp(const Params& p, long long e, int lane, u32* sc, u16* rings, u8* grid, u32& errs,
                               WarpStats& st) {
  const int S = p.S, F = p.F, V = p.V, cap = p.cap;
  u32 ctr = sc[REC_DRAW_CTR];
  const int n_pairs = S > F ? S : F;  // pair i: snake i (if i < S) then fruit i (if i < F)
  if (RULES != SNK_RULES_CLASSIC) {
    u32* g32 = reinterpret_cast<u32*>(grid);
    for (int w = lane; w < p.grid_stride / 4; w += 32) g32[w] = 0;
  }
  __syncwarp();
  u16* fr = reinterpret_cast<u16*>(sc + REC_SNAKE0 + 2 * S);
  int base = 0;
  for (int i0 = 0; i0 < n_pairs; i0 += 8) {  // up to 8 pairs = 32 draws per round
    // lane -> (pair, which of 4 slots); slots that do not exist (i >= S or i >= F) draw nothing
    const int i = i0 + (lane >> 2), slot = lane & 3;
    const bool is_snake = slot < 2;
    const bool live = i < n_pairs && (is_snake ? i < S : i < F);
    const u32 bal = __ballot_sync(FULL, live);
    const int my_idx = base + __popc(bal & ((1u << lane) - 1));
    const int v = live ? (int)draw_at(p, e, ctr + my_idx, (u32)p.D, errs) : 0;
    const int vy = __shfl_down_sync(FULL, v, 1);
    if (live && (slot == 0 || slot == 2)) {
      const int pid = (v + 1) * V + (vy + 1);
      if (slot == 0) {
        rings[i * cap] = (u16)pid;
        sc[REC_SNAKE0 + 2 * i] = 0u | (1u << 16);
        sc[REC_SNAKE0 + 2 * i + 1] = 3u;
      } else if (RULES == SNK_RULES_CLASSIC) {
        fr[i] = (u16)pid;
      }
    }
    if (RULES != SNK_RULES_CLASSIC) {  // count grid: duplicates possible, add one at a time
      for (int j = 0; j < 8; ++j) {
        const int pid = __shfl_sync(FULL, (v + 1) * V + (vy + 1), 4 * j + 2);
        if (lane == 0 && i0 + j < F) grid_inc(grid, pid, errs);
      }
    }
    base += __popc(bal);
  }
  ctr += base;
  st.draws += (float)base;
  if (lane == 0) {
    sc[REC_T] = 0; sc[REC_EP_LEN] = 0; sc[REC_DRAW_CTR] = ctr; sc[REC_EP_RET] = 0;
  }
  __syncwarp();
}

// One env step (:166-197): update_snake for every snake in index order (:97-145), then the
// simultaneous death test (:147-164), clearing, reward / t / done, Monitor accounting
// (baselines/bench/monitor.py:57-78) and the SubprocVecEnv auto-reset
// (baselines/common/vec_env/subproc_vec_env.py:13-16).  sc holds the record on entry and exit.
template <int RULES>
__device__ void step_env_warp(const Params& p, long long e, int lane, u32* sc, u32* bm, u16* rings, u8* grid,
                              u32& errs, WarpStats& st) {
  const int S = p.S, F = p.F, V = p.V, cap = p.cap;
  u32 ctr = sc[REC_DRAW_CTR];
  u32 spare = sc[REC_SPARE];
  u16* fr = reinterpret_cast<u16*>(sc + REC_SNAKE0 + 2 * S);
  const int act = lane < S ? (int)p.actions[e * S + lane] : 0;
  u32 was_alive = 0, moved = 0, strike = 0;
  int my_eaten = 0, eaten_total = 0, eaten0 = 0;
  // all S old heads in one parallel pass (lane s holds snake s): the per-snake loop below must not
  // pay one dependent HBM round trip per snake
  int old_head = 0;
  if (lane < S) {
    const u32 a = sc[REC_SNAKE0 + 2 * lane];
    if (a >> 16) old_head = rings[lane * cap + (a & 0xffff)];
  }
  // count-grid rules: the fruit count under every snake's next head, fetched in the same parallel
  // pass; it stays valid until some snake eats (respawn is the only thing that edits the grid here)
  int pre_cnt = 0;
  if (RULES != SNK_RULES_CLASSIC && lane < S) {
    const u32 a = sc[REC_SNAKE0 + 2 * lane];
    int v = sc[REC_SNAKE0 + 2 * lane + 1] >> 16;
    if (act >= 1 && act <= 4 && v != (((act + 1) & 3) + 1)) v = act;
    if ((a >> 16) && v) pre_cnt = grid[old_head + (v == 1 ? V : v == 2 ? 1 : v == 3 ? -V : -1)];
  }

  for (int s = 0; s < S; ++s) {
    const u32 wa = sc[REC_SNAKE0 + 2 * s], wb = sc[REC_SNAKE0 + 2 * s + 1];
    int len = wa >> 16, hs = wa & 0xffff, grow = wb & 0xffff, vel = wb >> 16;
    if (len == 0) continue;
    was_alive |= 1u << s;
    const int a = __shfl_sync(FULL, act, s);
    if (a >= 1 && a <= 4 && vel != (((a + 1) & 3) + 1)) vel = a;  // :108-115, reversal ignored
    if (RULES == SNK_RULES_CUT && a == 5) strike |= 1u << s;
    if (vel == 0) continue;                                         // :119, has not started moving
    const int delta = vel == 1 ? V : vel == 2 ? 1 : vel == 3 ? -V : -1;
    const int head = __shfl_sync(FULL, old_head, s) + delta;
    int n_eat;
    u32 hitmask = 0;
    if (RULES == SNK_RULES_CLASSIC) {
      hitmask = __ballot_sync(FULL, lane < F && fr[lane] == head);    // :126-132, several fruits may share a cell
      n_eat = __popc(hitmask);
    } else {
      const int pc = __shfl_sync(FULL, pre_cnt, s);
      n_eat = eaten_total == 0 ? pc : (int)grid[head];
    }
    grow += 2 * n_eat;
    if (len >= grow) len--;                                          // :134-135 pop before insert
    hs = hs ? hs - 1 : cap - 1;
    len++;
    if (lane == 0) {
      rings[s * cap + hs] = (u16)head;                               // :137
      sc[REC_SNAKE0 + 2 * s] = (u32)hs | ((u32)len << 16);
      sc[REC_SNAKE0 + 2 * s + 1] = (u32)grow | ((u32)vel << 16);
    }
    __syncwarp();
    if (RULES == SNK_RULES_CLASSIC) {
      while (hitmask) {                                              // :139-140, current half-updated world
        const int i = __ffs(hitmask) - 1;
        hitmask &= hitmask - 1;
        const int cell = spawn_cell(p, e, lane, sc, bm, rings, ctr, errs, st);
        if (lane == 0) fr[i] = (u16)cell;
        __syncwarp();
      }
    } else {
      for (int i = 0; i < n_eat; ++i) {
        if (RULES == SNK_RULES_ADVERSARIAL && spare > 0) {           // snake_adversarial_env.py:138-139
          spare--;
        } else {
          const int cell = spawn_cell(p, e, lane, sc, bm, rings, ctr, errs, st);
          if (lane == 0) { grid[head]--; grid_inc(grid, cell, errs); }
          __syncwarp();
        }
      }
    }
    moved |= 1u << s;
    if (lane == s) my_eaten = n_eat;
    if (s == 0) eaten0 = n_eat;
    eaten_total += n_eat;
  }

  // ---- death test on the post-move bodies of all snakes, before anything is cleared
  const u32 my_a = lane < S ? sc[REC_SNAKE0 + 2 * lane] : 0;
  const int my_len = my_a >> 16;
  const int my_head = my_len ? (int)rings[lane * cap + (my_a & 0xffff)] : -1;  // lane s: head of snake s
  const bool my_oob = my_len && (__ldg(p.cellinfo + my_head) >> 31);
  u32 hit_own = 0, hit_head = 0, hit_body = 0;  // bit s: head of snake s touches ...
  {
    // All segments of all snakes as ONE list dealt to the lanes 32 at a time (segment t belongs to the
    // snake j whose running length sum first exceeds t): the ring reads of a pass are independent, so the
    // test costs one memory round trip per 32 segments instead of one per snake.
    const SegScan sg = seg_scan(my_len, lane);
    for (int t0 = 0; t0 < sg.total; t0 += 32) {
      int j, i;
      const bool have = seg_locate(sg, my_len, S, t0 + lane, j, i);
      const int hs = __shfl_sync(FULL, (int)(my_a & 0xffff), j);
      const int pid = have ? ring_at(rings + j * cap, hs, i, cap) : -2;
      for (int s = 0; s < S; ++s) {
        const int h = __shfl_sync(FULL, my_head, s);
        if (pid == h && !(j == s && i == 0)) {
          if (j == s) hit_own |= 1u << s; else if (i == 0) hit_head |= 1u << s; else hit_body |= 1u << s;
        }
      }
    }
  }
  hit_own = __reduce_or_sync(FULL, hit_own);
  hit_head = __reduce_or_sync(FULL, hit_head);
  hit_body = __reduce_or_sync(FULL, hit_body);
  const u32 smask = S == 32 ? FULL : (1u << S) - 1;
  const u32 empty = ~__ballot_sync(FULL, my_len > 0) & smask;
  const u32 oob = __ballot_sync(FULL, my_oob);
  u32 dead = empty | oob | hit_own | hit_head | hit_body;
  if (RULES == SNK_RULES_CUT) {
    // strike: a head that only touches body segments (k >= 1) of OTHER snakes survives and cuts them
    const u32 saved = strike & moved & hit_body & ~(empty | oob | hit_own | hit_head);
    dead &= ~saved;
    if (saved) {
      for (int j = 0; j < S; ++j) {
        const u32 a = sc[REC_SNAKE0 + 2 * j];
        const int len = a >> 16, hs = a & 0xffff;
        int cut = 0x7fffffff;
        for (int i0 = 0; i0 < len; i0 += 32) {
          const int i = i0 + lane;
          const int pid = i < len ? ring_at(rings + j * cap, hs, i, cap) : -2;
          for (u32 m = saved & ~(1u << j); m; m &= m - 1) {
            const int h = __shfl_sync(FULL, my_head, __ffs(m) - 1);  // every lane takes part in the shuffle
            if (i >= 1 && pid == h) cut = min(cut, i);
          }
        }
#pragma unroll
        for (int o = 16; o; o >>= 1) cut = min(cut, __shfl_xor_sync(FULL, cut, o));
        if (cut < len) {
          for (int i0 = cut; i0 < len; i0 += 32) {   // removed segments become fruit unless a striker's head is there
            const int i = i0 + lane;
            const int pid = i < len ? ring_at(rings + j * cap, hs, i, cap) : -2;
            bool under_head = false;
            for (u32 m = saved; m; m &= m - 1) under_head |= pid == __shfl_sync(FULL, my_head, __ffs(m) - 1);
            if (i < len && !under_head) grid_inc(grid, pid, errs);
          }
          if (lane == 0) {
            sc[REC_SNAKE0 + 2 * j] = (u32)hs | ((u32)cut << 16);
            sc[REC_SNAKE0 + 2 * j + 1] = (u32)cut | (sc[REC_SNAKE0 + 2 * j + 1] & 0xffff0000u);
          }
          __syncwarp();
        }
      }
    }
  }
  if (RULES == SNK_RULES_ADVERSARIAL) {
    // snake_adversarial_env.py:180-186: every cell of a dead body (even an out-of-board head) becomes
    // a fruit and spare_fruits grows by len for EACH cell, i.e. by len^2
    for (u32 m = dead & ~empty; m; m &= m - 1) {
      const int j = __ffs(m) - 1;
      const u32 a = sc[REC_SNAKE0 + 2 * j];
      const int len = a >> 16, hs = a & 0xffff;
      for (int i = 1 + lane; i < len; i += 32) grid_inc(grid, ring_at(rings + j * cap, hs, i, cap), errs);
      __syncwarp();
      if (lane == 0) grid_inc(grid, rings[j * cap + hs], errs);  // the head may lie on its own body
      __syncwarp();
      spare += (u32)(len * len);
    }
  }
  // ---- clear the dead (:184-185), reward (:187-190), t (:192-193), done (:195)
  if (lane < S && ((dead >> lane) & 1)) sc[REC_SNAKE0 + 2 * lane] &= 0xffffu;
  __syncwarp();
  int cells = 0;
  for (int s = 0; s < S; ++s) cells += sc[REC_SNAKE0 + 2 * s] >> 16;
  const bool main_dead = dead & 1u;
  const float r0 = main_dead ? -1.f : (float)eaten0;
  const u32 t = sc[REC_T] + 1;
  const bool done = t >= (u32)p.max_steps || main_dead;
  const float ep_ret = __uint_as_float(sc[REC_EP_RET]) + r0;
  const u32 ep_len = sc[REC_EP_LEN] + 1;
  const int n_alive = S - __popc(dead);
  if (lane < S) {
    const bool d = (dead >> lane) & 1;
    float r = d ? (((was_alive >> lane) & 1) ? -1.f : 0.f) : (float)my_eaten;
    if (lane == 0) r = r0;
    p.reward_all[e * S + lane] = r;
  }
  if (lane == 0) {
    p.reward[e] = r0;
    p.done[e] = done;
    p.num_alive[e] = (u8)n_alive;
    p.fin_ret[e] = done ? ep_ret : 0.f;
    p.fin_len[e] = done ? (int)ep_len : 0;
    sc[REC_T] = t; sc[REC_EP_LEN] = ep_len; sc[REC_DRAW_CTR] = ctr;
    sc[REC_EP_RET] = __float_as_uint(ep_ret); sc[REC_SPARE] = spare;
  }
  __syncwarp();
  st.steps += 1.f;
  st.fruits += (float)eaten_total;
  st.deaths += (float)__popc(dead & was_alive);
  st.cells += (float)cells;
  if (done) {
    st.episodes += 1.f; st.ret_sum += ep_ret; st.len_sum += (float)ep_len;
    if (p.auto_reset) reset_env_warp<RULES>(p, e, lane, sc, rings, grid, errs, st);
  }
}

__device__ __forceinline__ void load_rec(const Params& p, long long e, int lane, u32* sc) {
  const u32* g = p.rec + e * p.RW;
  for (int w = lane; w < p.RW; w += 32) sc[w] = g[w];
  __syncwarp();
}

__device__ __forceinline__ void store_rec(const Params& p, long long e, int lane, const u32* sc) {
  u32* g = p.rec + e * p.RW;
  for (int w = lane; w < p.RW; w += 32) g[w] = sc[w];
}

// colours of get_ob_for_snake (:43-50): self green body/head, every other snake blue body/head
__device__ __forceinline__ u32 snake_rgb(bool self, bool head) {
  // packed R | G << 8 | B << 16
  return self ? (head ? (191u | 242u << 8 | 191u << 16) : (0u | 204u << 8 | 0u << 16))
              : (head ? (128u | 154u << 8 | 230u << 16) : (0u | 51u << 8 | 204u << 16));
}
