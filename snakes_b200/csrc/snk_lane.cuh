// snk_lane.cuh -- k_step_lane: the fast path for small boards (S <= 4, F <= 4, D <= 32).
//
// One LANE per env for the game logic, one WARP per batch of 32 consecutive envs, no CTA-wide
// synchronisation.  Differences from the warp-per-env kernels (snk_kernels.cu), all driven by the
// round-1 profile (944 warp-instructions per env-step, issue-bound at 24 % of the HBM roofline):
//
//  * body = chain code.  Consecutive segments are always adjacent cells, so a body is its head id
//    plus 2 bits per further segment (direction of the move that created segment i from i+1).  The
//    first 16 directions live in one register (one u32 in HBM); longer bodies spill to `chain`
//    words.  Advancing = shift in 2 bits; popping the tail = len-1; walking = register ALU only.
//  * the scalar logic of 32 envs runs in the 32 lanes at once (it ran 32x redundantly before).
//  * each warp owns a shared-memory image of TE (8/16/32) observations holding the border; LPE =
//    32/TE lanes paint one env by walking its chain (each lane owns fixed byte positions of a pixel,
//    so the reference's paint order -- fruits, snakes by index -- is kept without barriers), lane 0
//    hands the image to the TMA engine (cp.async.bulk.global.shared::cta), and after the engine has
//    read it the same walk un-paints.  No template restore, no lists, any body length.
//
// Reference semantics: gym_snake/envs/snake_multiple_test.py (cited per block below),
// snake_adversarial_env.py:137-141,180-186, subproc_vec_env.py:13-16, monitor.py:57-78.
#pragma once
#include "snk_device.cuh"

template <int S>
struct LaneRec {  // record words of the lane family: header 8, snakes 2S, room for 4 fruits
  static constexpr int RW = (REC_SNAKE0 + 2 * S + 2 + 3) & ~3;
  // the first chain word (16 directions) of every snake lives INSIDE the record, so a typical step
  // touches one contiguous 64-byte record per env and nothing else: words 5..7, snake 3 -> RW-2
  __host__ __device__ static constexpr int c0_word(int s) { return s < 3 ? 5 + s : RW - 2; }
};

template <int S>
struct LaneEnv {
  u32 t, ep_len, ctr, spare;
  float ep_ret;
  int head[S], len[S], grow[S], vel[S];
  u32 c0[S];
  int fruit[4];
};

struct LaneRng {  // one cached Philox block: four consecutive draws cost one evaluation
  u32 blk;
  bool have;
  Philox4 o;
};

__device__ __forceinline__ int chain_delta(u32 d, int V) {  // d = vel-1: +V, +1, -V, -1
  const int dv = (d & 1) ? 1 : V;
  return (d & 2) ? -dv : dv;
}

// visit(i, pid) for every segment, head first
template <class Fn>
__device__ __forceinline__ void chain_walk(int head, int len, u32 c0, const u32* __restrict__ ch, int V, Fn visit) {
  int pid = head;
  u32 w = c0;
  for (int i = 0; i < len; ++i) {
    visit(i, pid);
    const int j = i & 15;
    if (j == 0 && i) w = ch[i >> 4];
    pid -= chain_delta((w >> (2 * j)) & 3, V);
  }
}

// the raw Philox word of draw index env.ctr (no side effect but the one-block cache)
template <int S>
__device__ __forceinline__ u32 lane_philox_peek(const Params& p, long long e, const LaneEnv<S>& env, LaneRng& rng) {
  const u32 idx = env.ctr, blk = idx >> 2;
  if (!rng.have || rng.blk != blk) {
    rng.o = philox_block(blk, 0, 0, (u32)(p.seed >> 32), (u32)p.seed, (u32)(p.env_id_base + e));
    rng.blk = blk; rng.have = true;
  }
  const u32 sel = idx & 3;
  return sel == 0 ? rng.o.w[0] : sel == 1 ? rng.o.w[1] : sel == 2 ? rng.o.w[2] : rng.o.w[3];
}

template <int S>
__device__ __forceinline__ u32 lane_draw(const Params& p, long long e, LaneEnv<S>& env, LaneRng& rng, u32 n, u32& errs, float& draws) {
  draws += 1.f;
  if (p.rng_mode == SNK_RNG_TAPE) {
    const u32 idx = env.ctr++;
    const u64 pos = p.tape_off[e] + idx;
    if (pos >= p.tape_off[e + 1]) { errs |= SNK_DEVERR_TAPE_UNDERRUN; return 0; }
    if (p.tape_bounds && p.tape_bounds[pos] != n) errs |= SNK_DEVERR_TAPE_BOUND;
    return p.tape_vals[pos];
  }
  const u32 x = lane_philox_peek<S>(p, e, env, rng);
  env.ctr++;
  return __umulhi(x, n);
}

// Displacement from segment 0 to segment r (0..16) of the codes in word w: V * (#(+V) - #(-V)) + (#(+1) - #(-1)).
__device__ __forceinline__ int codes_disp(u32 w, int V, int r) {
  const u32 m = r >= 16 ? 0x55555555u : ((1u << (2 * r)) - 1u) & 0x55555555u;
  const u32 lo = w & m, hi = (w >> 1) & m;
  return V * (r - __popc(lo | hi) - __popc(hi & ~lo)) + (__popc(lo & ~hi) - __popc(lo & hi));
}

// Position of segment i without walking: the 2-bit codes before it are counted per direction with
// popcounts, pid_i = head - V*(#(+V) - #(-V)) - (#(+1) - #(-1)).
template <bool AT_L2 = false>  // AT_L2: the chain words were written by another lane a moment ago -- read them at the L2
__device__ __forceinline__ int chain_pos(int head, u32 c0, const u32* __restrict__ ch, int V, int i) {
  int nV = 0, n1 = 0;
  u32 w = c0;
  int k = 0;
  for (; i - 16 * k > 16; ++k) {  // whole words before the one holding code i-1 (bodies longer than 17)
    const u32 lo = w & 0x55555555u, hi = (w >> 1) & 0x55555555u;
    nV += 16 - __popc(lo | hi) - __popc(hi & ~lo);
    n1 += __popc(lo & ~hi) - __popc(lo & hi);
    w = AT_L2 ? __ldcg(ch + k + 1) : ch[k + 1];
  }
  return head - V * nV - n1 - codes_disp(w, V, i - 16 * k);
}

// chain_pos for a lane that visits segments in increasing order (i, i + LPE, ...): the whole words before the current
// one are folded into `base` once per word instead of once per segment.
struct ChainCursor {
  int base, k;
  u32 w;
  __device__ __forceinline__ ChainCursor(int head, u32 c0) : base(head), k(0), w(c0) {}
  __device__ __forceinline__ int at(const u32* ch, int V, int i) {
    while (i - 16 * k > 16) {
      const u32 lo = w & 0x55555555u, hi = (w >> 1) & 0x55555555u;
      base -= V * (16 - __popc(lo | hi) - __popc(hi & ~lo)) + __popc(lo & ~hi) - __popc(lo & hi);
      w = ch[k + 1];
      ++k;
    }
    return base - codes_disp(w, V, i - 16 * k);  // 0..16 codes of word k
  }
};

// safe_choose_cell (:202-217), warp-cooperative.  Under a policy that eats, about six lanes of every warp respawn a
// fruit on every step; a one-lane form (a serial walk of all bodies with a bitmap in local memory, about 5 k cycles;
// the first version of this kernel) then sits on the warp's critical path.  Here the warp serves up to FOUR envs
// ("owners", the lowest set bits of `mm`) per pass, eight lanes each: lane `sub` of a group takes segments sub,
// sub+8, ... of each body of its owner (chain_pos is O(1)) and ORs their y-major bits (cellinfo: the reference's
// un-bounds-checked aliasing of an out-of-board head) into the group's 32 words of shared memory; each lane then
// counts the free cells of four words, a 3-step shuffle scan gives the total, the owner turns its Philox word
// (`raw`, fetched by all owners at once before the pass) or its tape value into k, and the lane whose words hold the
// k-th free cell looks it up.  Same draws, same cell as the reference.  ALL 32 lanes must call it; `bm` = SPAWN_WORDS
// words of shared memory private to the warp.  Returns true in the lanes that were served, with their cell.
// The two phases are real function calls (one copy per kernel instead of one per snake: with the walks inlined S times
// the kernel outgrew the instruction cache -- 9 000 instructions ran the headline 12 % slower than 6 900), so they
// take values, not references: a reference to the env or to Params would force those into local memory.
#define SPAWN_WORDS 136  // 4 groups x 32 bitmap words, 4 totals, 4 cells
template <int S>
struct SpawnBodies {  // the bodies of one env as the lane that owns it holds them
  long long e;
  int head[S], len[S];
  u32 c0[S];
};

// phase 1: bitmaps of the (up to four) owners of this pass; returns the number of free cells to the served owners
template <int S>
__device__ __noinline__ u32 spawn_totals(SpawnBodies<S> me, u32 mm, u32* bm, const u32* chain, int CW, int V, int D, u32 magicV, int nW, int DD) {
  const int lane = threadIdx.x & 31, g = lane >> 3, sub = lane & 7;
  u32 m = mm;
  for (int t = 0; t < g; ++t) m &= m - 1;
  const bool active = m != 0;                      // my group serves the (g+1)-th owner
  const int src = active ? __ffs(m) - 1 : lane;
  const long long eo = __shfl_sync(FULL, me.e, src);
  u32* b = bm + g * 32;
  b[sub] = 0; b[sub + 8] = 0; b[sub + 16] = 0; b[sub + 24] = 0;
  __syncwarp();  // also orders the owners' chain-word stores before the other lanes' loads
#pragma unroll
  for (int s = 0; s < S; ++s) {
    const int h = __shfl_sync(FULL, me.head[s], src);
    int l = __shfl_sync(FULL, me.len[s], src);
    if (!active) l = 0;
    const u32 c0 = __shfl_sync(FULL, me.c0[s], src);
    const u32* ch = chain + (eo * S + s) * CW;
    ChainCursor cur(h, c0);
    for (int i = sub; i < l; i += 8) {
      // y*D + x, not bounds-checked (:209): an out-of-board head aliases another cell or nothing, exactly as cellinfo
      // tabulates it -- computed here because the 27 KB of L1 left beside the images rarely holds the table
      const u32 pid = (u32)cur.at(ch, V, i);
      const u32 px = (pid * magicV) >> 16, py = pid - px * (u32)V;
      const u32 idx = (u32)(((int)py - 1) * D + (int)px - 1);
      if (idx < (u32)DD) atomicOr(&b[idx >> 5], 1u << (idx & 31));
    }
  }
  __syncwarp();
  int c = 0;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int w = 4 * sub + j;
    u32 f = w < nW ? ~b[w] : 0u;
    if (w == nW - 1 && (DD & 31)) f &= (1u << (DD & 31)) - 1;
    b[w] = f;                                      // the words now hold the FREE cells (phase 2 reads them back)
    c += __popc(f);
  }
#pragma unroll
  for (int o = 1; o < 8; o <<= 1) {
    const int v = __shfl_up_sync(FULL, c, o, 8);
    if (sub >= o) c += v;
  }
  if (sub == 7) bm[128 + g] = (u32)c;
  __syncwarp();
  const int rank = __popc(mm & ((1u << lane) - 1u));  // an owner's rank among the set bits = the group that served it
  return (((mm >> lane) & 1u) && rank < 4) ? bm[128 + rank] : 0u;
}

// phase 2: k = the owner's draw (or -1); returns the k-th free cell (y-major order) to the served owners
static __device__ __noinline__ int spawn_pick(int k, u32 mm, u32* bm, int V, int D, u32 magicD) {
  const int lane = threadIdx.x & 31, g = lane >> 3, sub = lane & 7;
  u32 m = mm;
  for (int t = 0; t < g; ++t) m &= m - 1;
  const int src = m ? __ffs(m) - 1 : lane;
  int kk = __shfl_sync(FULL, k, src);
  if (!m) kk = -1;
  const u32* b = bm + g * 32;
  int c = 0;
  u32 fr[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) { fr[j] = b[4 * sub + j]; c += __popc(fr[j]); }
  int incl = c;
#pragma unroll
  for (int o = 1; o < 8; o <<= 1) {
    const int v = __shfl_up_sync(FULL, incl, o, 8);
    if (sub >= o) incl += v;
  }
  if (kk >= incl - c && kk < incl) {
    int r = kk - (incl - c), idx = 0;
    bool found = false;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int cj = __popc(fr[j]);
      if (!found && r < cj) { idx = (4 * sub + j) * 32 + (int)__fns(fr[j], 0, r + 1); found = true; }
      r -= cj;
    }
    const u32 y = ((u32)idx * magicD) >> 16, x = (u32)idx - y * (u32)D;  // cell (idx % D, idx // D) (:216)
    bm[132 + g] = (x + 1) * (u32)V + y + 1;
  }
  __syncwarp();
  const int rank = __popc(mm & ((1u << lane) - 1u));
  const int cell = (((mm >> lane) & 1u) && rank < 4) ? (int)bm[132 + rank] : 0;
  __syncwarp();  // the next pass zeroes the words
  return cell;
}

// one pass: returns true in the lanes that were served, with their cell
template <int S>
__device__ __forceinline__ bool group_spawn(const Params& p, long long e, LaneEnv<S>& env, LaneRng& rng, u32 raw, u32 mm, u32* bm, u32& errs,
                                            float& draws, int& cell) {
  const int lane = threadIdx.x & 31;
  SpawnBodies<S> me;
  me.e = e;
#pragma unroll
  for (int s = 0; s < S; ++s) { me.head[s] = env.head[s]; me.len[s] = env.len[s]; me.c0[s] = env.c0[s]; }
  const u32 total = spawn_totals<S>(me, mm, bm, p.chain, p.CW, p.V, p.D, p.magicV, p.bm_words, p.D * p.D);
  const bool served = ((mm >> lane) & 1u) && __popc(mm & ((1u << lane) - 1u)) < 4;
  int k = -1;
  if (served && total > 0) {
    if (p.rng_mode == SNK_RNG_TAPE) k = (int)lane_draw<S>(p, e, env, rng, total, errs, draws);
    else { env.ctr++; draws += 1.f; k = (int)__umulhi(raw, total); }
  }
  const int c = spawn_pick(k, mm, bm, p.V, p.D, p.magicD);
  cell = k >= 0 ? c : p.V + 1;                     // (0,0), no draw, when nothing is free (:212-215)
  return served;
}


// Fruit multiset of the adversarial / cut rule-sets in the lane family: `gbits` holds one bit per
// padded cell (set = at least one fruit), `grid` the count, VALID ONLY WHERE THE BIT IS SET.  Reset
// therefore clears GBW words instead of V*V bytes and painting scans GBW words instead of the grid.
struct FruitSet {
  u8* cnt;    // [VV]
  u32* bits;  // [GBW]
};
__device__ __forceinline__ FruitSet fruit_set(const Params& p, long long e) {
  FruitSet f;
  f.cnt = p.grid ? p.grid + e * p.grid_stride : nullptr;
  f.bits = p.gbits ? p.gbits + e * p.GBW : nullptr;
  return f;
}
__device__ __forceinline__ int fruit_count(const FruitSet& f, int pid) {
  return ((f.bits[pid >> 5] >> (pid & 31)) & 1) ? (int)f.cnt[pid] : 0;
}
__device__ __forceinline__ void fruit_inc(const FruitSet& f, int pid, u32& errs) {
  const u32 w = f.bits[pid >> 5], m = 1u << (pid & 31);
  if (w & m) {
    const u8 c = f.cnt[pid];
    if (c == 255) errs |= SNK_DEVERR_FRUIT_OVERFLOW; else f.cnt[pid] = c + 1;
  } else {
    f.cnt[pid] = 1;
    f.bits[pid >> 5] = w | m;
  }
}
__device__ __forceinline__ void fruit_dec(const FruitSet& f, int pid) {
  const u8 c = f.cnt[pid] - 1;
  f.cnt[pid] = c;
  if (c == 0) f.bits[pid >> 5] &= ~(1u << (pid & 31));
}

// reset (:219-232): snake_i.x, snake_i.y, fruit_i.x, fruit_i.y interleaved, randint(D) each
template <int S, int RULES>
__device__ __forceinline__ void lane_reset(const Params& p, long long e, LaneEnv<S>& env, LaneRng& rng, const FruitSet& fs, u32& errs, float& draws) {
  const int F = p.F, V = p.V;
  if (RULES != SNK_RULES_CLASSIC) {
    for (int w = 0; w < p.GBW; ++w) fs.bits[w] = 0;
  }
  // the draws in a rolled loop (two inlined copies of lane_draw instead of twelve: the kernel lives off the instruction
  // cache), the cells parked in a small local array, then dealt out in the reference's interleaved order
  int cells[8];
  const int nc = S + F;
#pragma unroll 1
  for (int c = 0; c < nc; ++c) {
    const int x = (int)lane_draw<S>(p, e, env, rng, (u32)p.D, errs, draws);
    const int y = (int)lane_draw<S>(p, e, env, rng, (u32)p.D, errs, draws);
    cells[c] = (x + 1) * V + (y + 1);
  }
  int r = 0;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    if (i < S) {
      env.head[i < S ? i : 0] = cells[r++];
      env.len[i < S ? i : 0] = 1; env.grow[i < S ? i : 0] = 3; env.vel[i < S ? i : 0] = 0; env.c0[i < S ? i : 0] = 0;
    }
    if (i < F) {
      const int pid = cells[r++];
      if (RULES == SNK_RULES_CLASSIC) env.fruit[i] = pid; else fruit_inc(fs, pid, errs);
    }
  }
  env.t = 0; env.ep_len = 0; env.ep_ret = 0.f;  // `spare` survives (snake_adversarial_env.py:14)
}

struct LaneStats {
  float steps, episodes, ret_sum, len_sum, fruits, deaths, cells, draws;
#ifdef SNK_PHASE_LOGIC  // experiment build: warp cycles of the four parts of lane_step (move+push, respawns, death test, tail+reset)
  long long ph[4];
#endif
};
#ifdef SNK_PHASE_LOGIC
#define SNK_LOGIC_MARK(k) { __syncwarp(__activemask()); const long long t_now = clock64(); st.ph[k] += t_now - t_mark; t_mark = t_now; }
#define SNK_LOGIC_START long long t_mark; { __syncwarp(__activemask()); t_mark = clock64(); }
#else
#define SNK_LOGIC_MARK(k)
#define SNK_LOGIC_START
#endif

// One env step in one lane (:166-197).
// Called by ALL 32 lanes of the warp (the respawns are warp-cooperative); lanes without an env pass valid = false
// and an env whose snakes all have length 0.  `bm` = SPAWN_WORDS words of shared memory private to the warp.
//
// HOP (the two-kernel form's k_lane_logic): the death test takes the chain codes four at a time.  A 256-entry table in
// shared memory (build_hop_lut) holds, for every byte of codes, the displacement after one, two, three and four of them
// as four 16-bit fields, so a group of four segments costs one 8-byte load, four subtractions and 4 S compares, with no
// branch inside: 9 instructions per segment instead of 21 in the test that, one env per lane, costs every warp its
// longest pair of snakes (43 % of the kernel's instructions under the fruit-seeking policy).  Same hits.
__device__ __forceinline__ void build_hop_lut(uint2* lut, int V, int tid, int nthreads) {
  for (int b = tid; b < 256; b += nthreads) {
    int d = 0;
    u32 f[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) { d += chain_delta((u32)(b >> (2 * k)) & 3, V); f[k] = (u32)d & 0xffffu; }
    lut[b] = make_uint2(f[0] | (f[1] << 16), f[2] | (f[3] << 16));
  }
}

template <int S, int RULES, bool HOP = false>
__device__ __forceinline__ void lane_step(const Params& p, long long e, bool valid, LaneEnv<S>& env, u32 act_packed, LaneRng& rng, const FruitSet& fs,
                                          u32* bm, u32& errs, LaneStats& st, const uint2* hop_lut = nullptr) {
  const int V = p.V, F = p.F;
  const u32* chain_e = p.chain + e * S * p.CW;
  int act[S];
#pragma unroll
  for (int s = 0; s < S; ++s) act[s] = (int)(int8_t)(act_packed >> (8 * s));
  u32 was_alive = 0, moved = 0, strike = 0;
  int eaten[S];
  SNK_LOGIC_START
  // ---- update_snake for every snake in index order (:97-145)
#pragma unroll
  for (int s = 0; s < S; ++s) {
    eaten[s] = 0;
    u32 hitmask = 0;   // classic: fruit slots to respawn; other rule-sets: number of respawns
    int n_spawn = 0, head = 0;
    if (env.len[s] != 0) {
      was_alive |= 1u << s;
      const int a = act[s];
      int vel = env.vel[s];
      if (a >= 1 && a <= 4 && vel != (((a + 1) & 3) + 1)) vel = a;   // :108-115
      if (RULES == SNK_RULES_CUT && a == 5) strike |= 1u << s;
      if (vel != 0) {                                                  // :119
        head = env.head[s] + chain_delta((u32)(vel - 1), V);
        int n_eat = 0;
        if (RULES == SNK_RULES_CLASSIC) {
#pragma unroll
          for (int f = 0; f < 4; ++f) if (f < F && env.fruit[f] == head) { hitmask |= 1u << f; ++n_eat; }   // :126-132
        } else {
          n_eat = fruit_count(fs, head);
        }
        const int grow = env.grow[s] + 2 * n_eat;
        int len = env.len[s];
        if (len >= grow) len--;                                          // :134-135
        len++;                                                           // :137
        {  // push the new direction: segment 0 -> 1 was created by `vel`
          u32* ch = p.chain + (e * S + s) * p.CW;
          const int nw = (len - 1 + 15) >> 4;
          u32 carry = env.c0[s] >> 30;
          env.c0[s] = (env.c0[s] << 2) | (u32)(vel - 1);
          for (int k = 1; k < nw; ++k) { const u32 w = ch[k]; ch[k] = (w << 2) | carry; carry = w >> 30; }
        }
        env.head[s] = head; env.len[s] = len; env.grow[s] = grow; env.vel[s] = vel;
        if (RULES == SNK_RULES_ADVERSARIAL) {                          // snake_adversarial_env.py:138-139: spare fruits first
          const int use = min((int)min(env.spare, 0x7fffffffu), n_eat);
          env.spare -= (u32)use;
          n_spawn = n_eat - use;
        } else if (RULES == SNK_RULES_CUT) {
          n_spawn = n_eat;
        }
        moved |= 1u << s;
        eaten[s] = n_eat;
      }
    }
    SNK_LOGIC_MARK(0)
    // respawns (:139-140, against the half-updated world): up to four envs per pass by the whole warp
    for (;;) {
      const bool need = RULES == SNK_RULES_CLASSIC ? hitmask != 0 : n_spawn > 0;
      u32 mm = __ballot_sync(FULL, need);
      if (!mm) break;
      u32 raw = 0;
      if (need && p.rng_mode != SNK_RNG_TAPE) raw = lane_philox_peek<S>(p, e, env, rng);  // all owners at once
      while (mm) {
        int cell;
        if (group_spawn<S>(p, e, env, rng, raw, mm, bm, errs, st.draws, cell)) {
          if (RULES == SNK_RULES_CLASSIC) {
            const int f = __ffs(hitmask) - 1;
#pragma unroll
            for (int g = 0; g < 4; ++g) if (g == f) env.fruit[g] = cell;
            hitmask &= hitmask - 1;
          } else {
            fruit_dec(fs, head); fruit_inc(fs, cell, errs);
            --n_spawn;
          }
        }
#pragma unroll
        for (int t = 0; t < 4; ++t) mm &= mm - 1;  // the four owners of this pass are done
      }
    }
    SNK_LOGIC_MARK(1)
  }
  // ---- is_snake_alive for all snakes on the post-move bodies, before anything is cleared (:147-164, :178-182)
  u32 empty = 0, oob = 0, hit_own = 0, hit_head = 0, hit_body = 0;
#pragma unroll
  for (int s = 0; s < S; ++s) {
    if (env.len[s] == 0) empty |= 1u << s;
    else {  // outside the board (:150-152), by arithmetic: a table load here sits on every batch's critical path
      const u32 px = ((u32)env.head[s] * p.magicV) >> 16, py = (u32)env.head[s] - px * (u32)V;
      if (px - 1u >= (u32)p.D || py - 1u >= (u32)p.D) oob |= 1u << s;
    }
  }
  int live_head[S];  // head of a live snake, or an id no cell has: one compare per segment and snake in the walks
#pragma unroll
  for (int s = 0; s < S; ++s) live_head[s] = env.len[s] ? env.head[s] : -1;
  if (HOP) {
#pragma unroll
    for (int j = 0; j < S; ++j) {
      const u32* ch = chain_e + j * p.CW;
      const int len = env.len[j];
      int pid = env.head[j];
      u32 w = env.c0[j];
      for (int i = 0; i < len; i += 4) {
        if ((i & 15) == 0 && i) w = ch[i >> 4];
        const uint2 d = hop_lut[(w >> (2 * (i & 15))) & 0xffu];
        const int n = len - i;  // segments i .. i+3 exist while k < n
        const int q1 = pid - (int)(short)(d.x & 0xffffu), q2 = pid - ((int)d.x >> 16), q3 = pid - (int)(short)(d.y & 0xffffu);
#pragma unroll
        for (int s = 0; s < S; ++s) {
          const int t = live_head[s];
          const bool h0 = pid == t, h123 = (q1 == t && n > 1) || (q2 == t && n > 2) || (q3 == t && n > 3);
          if (j == s) { if ((h0 && i) || h123) hit_own |= 1u << s; }
          else {
            if (h0 && !i) hit_head |= 1u << s;
            if ((h0 && i) || h123) hit_body |= 1u << s;
          }
        }
        pid -= (int)d.y >> 16;
      }
    }
  } else {
#pragma unroll
  for (int j = 0; j < S; ++j) {
    chain_walk(env.head[j], env.len[j], env.c0[j], chain_e + j * p.CW, V, [&](int i, int pid) {
#pragma unroll
      for (int s = 0; s < S; ++s) {
        if (pid == live_head[s]) {
          if (i == 0) { if (j != s) hit_head |= 1u << s; }
          else if (j == s) hit_own |= 1u << s;
          else hit_body |= 1u << s;
        }
      }
    });
  }
  }
  u32 dead = empty | oob | hit_own | hit_head | hit_body;
  if (RULES == SNK_RULES_CUT) {
    const u32 saved = strike & moved & hit_body & ~(empty | oob | hit_own | hit_head);
    dead &= ~saved;
    if (saved) {
#pragma unroll
      for (int j = 0; j < S; ++j) {
        int cut = 0x7fffffff;
        chain_walk(env.head[j], env.len[j], env.c0[j], chain_e + j * p.CW, V, [&](int i, int pid) {
#pragma unroll
          for (int s = 0; s < S; ++s)
            if (s != j && ((saved >> s) & 1) && i >= 1 && pid == env.head[s] && i < cut) cut = i;
        });
        if (cut < env.len[j]) {
          chain_walk(env.head[j], env.len[j], env.c0[j], chain_e + j * p.CW, V, [&](int i, int pid) {
            if (i < cut) return;
            bool under = false;
#pragma unroll
            for (int s = 0; s < S; ++s) under |= ((saved >> s) & 1) && pid == env.head[s];
            if (!under) fruit_inc(fs, pid, errs);
          });
          env.len[j] = cut; env.grow[j] = cut;
        }
      }
    }
  }
  if (RULES == SNK_RULES_ADVERSARIAL) {  // snake_adversarial_env.py:180-186
#pragma unroll
    for (int j = 0; j < S; ++j) {
      if (!((dead & ~empty) >> j & 1)) continue;
      chain_walk(env.head[j], env.len[j], env.c0[j], chain_e + j * p.CW, V, [&](int, int pid) { fruit_inc(fs, pid, errs); });
      env.spare += (u32)(env.len[j] * env.len[j]);
    }
  }
  SNK_LOGIC_MARK(2)
  // ---- clear (:184-185), reward (:187-190), t (:192-193), done (:195), Monitor (monitor.py:57-78)
  int cells = 0;
#pragma unroll
  for (int s = 0; s < S; ++s) { if ((dead >> s) & 1) env.len[s] = 0; cells += env.len[s]; }
  const bool main_dead = dead & 1u;
  const float r0 = main_dead ? -1.f : (float)eaten[0];
  env.t += 1;
  const bool done = env.t >= (u32)p.max_steps || main_dead;
  env.ep_ret += r0;
  env.ep_len += 1;
  if (valid) {
    int fruits = 0;
#pragma unroll
    for (int s = 0; s < S; ++s) {
      const bool d = (dead >> s) & 1;
      const float r = s == 0 ? r0 : d ? (((was_alive >> s) & 1) ? -1.f : 0.f) : (float)eaten[s];
      p.reward_all[e * S + s] = r;
      fruits += eaten[s];
    }
    p.reward[e] = r0;
    p.done[e] = done;
    p.num_alive[e] = (u8)(S - __popc(dead));
    p.fin_ret[e] = done ? env.ep_ret : 0.f;
    p.fin_len[e] = done ? (int)env.ep_len : 0;
    st.steps += 1.f;
    st.fruits += (float)fruits;
    st.deaths += (float)__popc(dead & was_alive);
    st.cells += (float)cells;
    if (done) {
      st.episodes += 1.f; st.ret_sum += env.ep_ret; st.len_sum += (float)env.ep_len;
      if (p.auto_reset) lane_reset<S, RULES>(p, e, env, rng, fs, errs, st.draws);  // subproc_vec_env.py:13-16
    }
  }
  SNK_LOGIC_MARK(3)
}

// The record and the actions of one env as they sit in HBM: fetched early (the loads stay in flight
// while the warp paints the previous batch) and unpacked when the step starts.
template <int S>
struct LaneRaw {
  uint4 v[LaneRec<S>::RW / 4];
  u32 act;     // S int8 actions, little-endian
  bool frame;  // frame_ok: the own observation buffer holds this record's image
};

template <int S>
__device__ __forceinline__ LaneRaw<S> lane_fetch(const Params& p, long long e, bool with_actions) {
  constexpr int RW = LaneRec<S>::RW;
  LaneRaw<S> raw;
  const uint4* g = reinterpret_cast<const uint4*>(p.rec + e * RW);
  u64 pol;  // keep the records L2-resident across steps (they are re-read by the next launch)
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
#pragma unroll
  for (int i = 0; i < RW / 4; ++i)
    asm volatile("ld.global.L2::cache_hint.v4.u32 {%0, %1, %2, %3}, [%4], %5;"
                 : "=r"(raw.v[i].x), "=r"(raw.v[i].y), "=r"(raw.v[i].z), "=r"(raw.v[i].w) : "l"(g + i), "l"(pol));
  raw.frame = p.frame_ok[e] != 0;
  raw.act = 0;
  if (with_actions) {
    const int8_t* a = p.actions + e * S;
    if (S == 2) raw.act = *reinterpret_cast<const u16*>(a);
    else if (S == 4) raw.act = *reinterpret_cast<const u32*>(a);
    else {
#pragma unroll
      for (int s = 0; s < S; ++s) raw.act |= (u32)(u8)a[s] << (8 * s);
    }
  }
  return raw;
}

template <int S>
__device__ __forceinline__ void lane_unpack(const LaneRaw<S>& raw, LaneEnv<S>& env) {
  constexpr int RW = LaneRec<S>::RW;
  u32 r[RW];
#pragma unroll
  for (int i = 0; i < RW / 4; ++i) { r[4 * i] = raw.v[i].x; r[4 * i + 1] = raw.v[i].y; r[4 * i + 2] = raw.v[i].z; r[4 * i + 3] = raw.v[i].w; }
  env.t = r[REC_T]; env.ep_len = r[REC_EP_LEN]; env.ctr = r[REC_DRAW_CTR]; env.ep_ret = __uint_as_float(r[REC_EP_RET]);
  env.spare = r[REC_SPARE];
#pragma unroll
  for (int s = 0; s < S; ++s) {
    env.head[s] = r[REC_SNAKE0 + 2 * s] & 0xffff; env.len[s] = r[REC_SNAKE0 + 2 * s] >> 16;
    env.grow[s] = r[REC_SNAKE0 + 2 * s + 1] & 0xffff; env.vel[s] = r[REC_SNAKE0 + 2 * s + 1] >> 16;
    env.c0[s] = r[LaneRec<S>::c0_word(s)];
  }
  env.fruit[0] = r[REC_SNAKE0 + 2 * S] & 0xffff; env.fruit[1] = r[REC_SNAKE0 + 2 * S] >> 16;
  env.fruit[2] = r[REC_SNAKE0 + 2 * S + 1] & 0xffff; env.fruit[3] = r[REC_SNAKE0 + 2 * S + 1] >> 16;
}

template <int S>
__device__ __forceinline__ void lane_load(const Params& p, long long e, LaneEnv<S>& env) {
  const LaneRaw<S> raw = lane_fetch<S>(p, e, false);
  lane_unpack<S>(raw, env);
}

template <int S>
__device__ __forceinline__ void lane_store(const Params& p, long long e, const LaneEnv<S>& env) {
  constexpr int RW = LaneRec<S>::RW;
  u32 r[RW];
#pragma unroll
  for (int i = 0; i < RW; ++i) r[i] = 0;
  r[REC_T] = env.t; r[REC_EP_LEN] = env.ep_len; r[REC_DRAW_CTR] = env.ctr; r[REC_EP_RET] = __float_as_uint(env.ep_ret);
  r[REC_SPARE] = env.spare;
#pragma unroll
  for (int s = 0; s < S; ++s) {
    r[REC_SNAKE0 + 2 * s] = (u32)env.head[s] | ((u32)env.len[s] << 16);
    r[REC_SNAKE0 + 2 * s + 1] = (u32)env.grow[s] | ((u32)env.vel[s] << 16);
    r[LaneRec<S>::c0_word(s)] = env.c0[s];
  }
  r[REC_SNAKE0 + 2 * S] = (u32)env.fruit[0] | ((u32)env.fruit[1] << 16);
  r[REC_SNAKE0 + 2 * S + 1] = (u32)env.fruit[2] | ((u32)env.fruit[3] << 16);
  uint4* g = reinterpret_cast<uint4*>(p.rec + e * RW);
  p.frame_ok[e] = (u8)p.frame_own;
  u64 pol;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
#pragma unroll
  for (int i = 0; i < RW / 4; ++i)
    asm volatile("st.global.L2::cache_hint.v4.u32 [%0], {%1, %2, %3, %4}, %5;" ::"l"(g + i), "r"(r[4 * i]), "r"(r[4 * i + 1]),
                 "r"(r[4 * i + 2]), "r"(r[4 * i + 3]), "l"(pol) : "memory");
}

// all C = 3K bytes of one pixel: snake s seen by every view k (self colours iff s == k)
template <int S, int K>
__device__ __forceinline__ void put_pixel(u8* px, int s, bool is_head, bool paint) {
  if (K % 2 == 0) {  // 6 bytes per pair of views at an even address: three 16-bit stores instead of six bytes
#pragma unroll
    for (int m = 0; m < K / 2; ++m) {
      const u32 a = paint ? snake_rgb(s == 2 * m, is_head) : 0u, b = paint ? snake_rgb(s == 2 * m + 1, is_head) : 0u;
      u16* q = reinterpret_cast<u16*>(px + 6 * m);
      q[0] = (u16)a; q[1] = (u16)((a >> 16) | ((b & 0xffu) << 8)); q[2] = (u16)(b >> 8);
    }
  } else {
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const u32 rgb = paint ? snake_rgb(s == k, is_head) : 0u;
      px[3 * k] = (u8)rgb; px[3 * k + 1] = (u8)(rgb >> 8); px[3 * k + 2] = (u8)(rgb >> 16);
    }
  }
}

// What painting needs of one env: heads, lengths, first chain words, classic fruit ids.
template <int S>
struct PaintEnv {
  int head[S], len[S];
  u32 c0[S];
  int fruit[4];
  bool valid;
};

// fused kernel: the painting lane fetches the env of lane `owner` through shuffles
template <int S>
__device__ __forceinline__ PaintEnv<S> paint_env_from_lane(const LaneEnv<S>& env, bool valid, int owner) {
  PaintEnv<S> pe;
  pe.valid = __shfl_sync(FULL, (int)valid, owner);
#pragma unroll
  for (int f = 0; f < 4; ++f) pe.fruit[f] = __shfl_sync(FULL, env.fruit[f], owner);
#pragma unroll
  for (int s = 0; s < S; ++s) {
    pe.head[s] = __shfl_sync(FULL, env.head[s], owner);
    pe.len[s] = __shfl_sync(FULL, env.len[s], owner);
    pe.c0[s] = __shfl_sync(FULL, env.c0[s], owner);
  }
  return pe;
}

// split kernels: the painting lane reads the env's record from HBM / L2
template <int S>
__device__ __forceinline__ PaintEnv<S> paint_env_from_memory(const Params& p, long long e) {
  constexpr int RW = LaneRec<S>::RW;
  PaintEnv<S> pe;
  pe.valid = e < p.N;
#pragma unroll
  for (int s = 0; s < S; ++s) { pe.head[s] = 0; pe.len[s] = 0; pe.c0[s] = 0; }
  pe.fruit[0] = pe.fruit[1] = pe.fruit[2] = pe.fruit[3] = 0;
  if (pe.valid) {
    const u32* r = p.rec + e * RW;  // __ldcg: read at L2, the line may have just been written by another warp
#pragma unroll
    for (int s = 0; s < S; ++s) {
      const u32 a = __ldcg(r + REC_SNAKE0 + 2 * s);
      pe.head[s] = a & 0xffff; pe.len[s] = a >> 16;
      pe.c0[s] = __ldcg(r + LaneRec<S>::c0_word(s));
    }
    const u32 f0 = __ldcg(r + REC_SNAKE0 + 2 * S), f1 = __ldcg(r + REC_SNAKE0 + 2 * S + 1);
    pe.fruit[0] = f0 & 0xffff; pe.fruit[1] = f0 >> 16; pe.fruit[2] = f1 & 0xffff; pe.fruit[3] = f1 >> 16;
  }
  return pe;
}

// Paint (PAINT) or un-paint the TE envs of one image.  The LPE lanes that share an env split its
// fruits and, per snake, its segments (segment i goes to lane i % LPE; chain_pos makes that O(1)).
// The reference's paint order (fruits, then snakes by index, get_ob_for_snake :35-58) is kept by a
// __syncwarp between the groups; within a group two items never overlap with different colours.
// Out-of-board cells are skipped (the reference paints them under the border, :52-56).
// `paint` is a run-time flag: one copy of the walk serves painting and un-painting (code size, see lane_reset).
template <int S, int RULES, int K>
__device__ __forceinline__ void lane_paint(const Params& p, const PaintEnv<S>& pe, long long e_owner, int sub, int LPE, u8* img, bool paint) {
  constexpr int C = 3 * K;
  const int V = p.V, F = p.F;
  const u8 red = paint ? 255 : 0;
  if (RULES == SNK_RULES_CLASSIC) {
#pragma unroll
    for (int f = 0; f < 4; ++f) {
      if (pe.valid && f < F && (f & (LPE - 1)) == sub) {
#pragma unroll
        for (int k = 0; k < K; ++k) img[pe.fruit[f] * C + 3 * k] = red;
      }
    }
  } else if (pe.valid) {
    const u32* gb = p.gbits + e_owner * p.GBW;
    for (int w = sub; w < p.GBW; w += LPE) {
      for (u32 bits = gb[w]; bits; bits &= bits - 1) {
        const int pid = 32 * w + __ffs(bits) - 1;
        if (!(__ldg(p.cellinfo + pid) >> 31)) {
#pragma unroll
          for (int k = 0; k < K; ++k) img[pid * C + 3 * k] = red;
        }
      }
    }
  }
  __syncwarp();
#pragma unroll
  for (int s = 0; s < S; ++s) {
    if (pe.valid) {
      const u32* ch = p.chain + (e_owner * S + s) * p.CW;
      ChainCursor cur(pe.head[s], pe.c0[s]);
      for (int i = sub; i < pe.len[s]; i += LPE) put_pixel<S, K>(img + cur.at(ch, V, i) * C, s, i == 0, paint);
    }
    __syncwarp();
  }
}

// Un-paint without walking: the interior of every image is black and the border white, so the warp
// zero-fills its whole image buffer (16-byte stores) and the LPE lanes of each env redraw the border
// spans -- [0, row + 1 px), the (last px of row x, first px of row x+1) pairs, [last px of row V-2, end).
// Fixed cost per image (about 100 stores per lane at 8 envs of 2 views 21x21), independent of the body
// lengths; the kernel uses it when the walk would be longer (Params::restore_thr).
template <int K>
__device__ __noinline__ void lane_restore(u8* tile, int n16, u8* img, int V, int sub, int LPE, int lane) {
  constexpr int C = 3 * K, U = (C & 1) ? 1 : 2, PU = 2 * C / U;
  uint4* t4 = reinterpret_cast<uint4*>(tile);
  const uint4 z = make_uint4(0u, 0u, 0u, 0u);
  for (int i = lane; i < n16; i += 32) t4[i] = z;
  __syncwarp();
  const int RB = V * C;
  const int n_edge = (RB + C) / U;
  u8* bot = img + RB * (V - 1) - C;
  for (int j = sub; j < n_edge; j += LPE) {
    if (U == 2) { *reinterpret_cast<u16*>(img + 2 * j) = 0xffffu; *reinterpret_cast<u16*>(bot + 2 * j) = 0xffffu; }
    else { img[j] = 0xff; bot[j] = 0xff; }
  }
  // rows 1..V-3: the (last px of row x, first px of row x+1) pair, one row per lane and trip
  for (int x = 1 + sub; x <= V - 3; x += LPE) {
    u8* q = img + x * RB + RB - C;
#pragma unroll
    for (int r = 0; r < PU; ++r) {
      if (U == 2) *reinterpret_cast<u16*>(q + 2 * r) = 0xffffu; else q[r] = 0xff;
    }
  }
}

// Un-paint decision: lane_restore when some lane of the warp would walk more than Params::restore_thr segments
// (warp-uniform, bit-identical result either way).  Taken BEFORE the image is painted and handed to the TMA engine,
// so that the warp reduction is off the critical path between the engine's read and the next paint.
template <int S>
__device__ __forceinline__ bool lane_wants_restore(const Params& p, const int* len, int LPE) {
  if (p.restore_thr <= 0) return false;
  const int sh = 31 - __clz(LPE);
  int it = 0;
#pragma unroll
  for (int s = 0; s < S; ++s) it += (len[s] + LPE - 1) >> sh;
  return __reduce_max_sync(FULL, it) > p.restore_thr;
}

template <int S, int RULES, int K>
__device__ __forceinline__ void lane_unpaint(const Params& p, const PaintEnv<S>& pe, long long e_owner, int sub, int LPE, u8* tile, int tile_bytes,
                                             u8* img, int lane, bool restore) {
  if (restore) lane_restore<K>(tile, tile_bytes >> 4, img, p.V, sub, LPE, lane);
  else lane_paint<S, RULES, K>(p, pe, e_owner, sub, LPE, img, false);
}

// ---- Delta store (Params::delta): the fused kernel's image store when the own observation buffer already holds the
// previous frame.  Both frames of an env are the border over a black interior with fruits and bodies painted on top, so
// a pixel painted in neither the old frame nor the new one is the same in both: writing every 32-byte sector that holds a
// pixel of the OLD state's classic fruits and bodies or of the NEW state's turns the old image into the new one.  The
// bytes come from the new image the warp has painted in shared memory; painting and un-painting stay as they are.
// The first and last (V+1)*C >= 32 bytes of an env image are border (the planner checks it), so a sector holding an
// interior pixel lies inside its own env and no two warps ever write the same sector.  Bodies of up to
// DELTA_MAX_LEN segments: the whole chain is in the record's first chain word.
#define DELTA_MAX_LEN 17

template <int S>
struct DeltaOld {  // the paint items of the state the record held before the step (= what the old frame shows)
  u32 hl[S], c0[S];  // head | len << 16, first chain word
  u32 fr[2];         // classic fruit ids, two u16 per word
};

template <int S>
__device__ __forceinline__ DeltaOld<S> delta_old(const LaneRaw<S>& raw) {
  constexpr int RW = LaneRec<S>::RW;
  u32 r[RW];
#pragma unroll
  for (int i = 0; i < RW / 4; ++i) { r[4 * i] = raw.v[i].x; r[4 * i + 1] = raw.v[i].y; r[4 * i + 2] = raw.v[i].z; r[4 * i + 3] = raw.v[i].w; }
  DeltaOld<S> o;
#pragma unroll
  for (int s = 0; s < S; ++s) { o.hl[s] = r[REC_SNAKE0 + 2 * s]; o.c0[s] = r[LaneRec<S>::c0_word(s)]; }
  o.fr[0] = r[REC_SNAKE0 + 2 * S]; o.fr[1] = r[REC_SNAKE0 + 2 * S + 1];
  return o;
}

// the verdict for one env: the old frame is in the buffer and every old and new body fits the first chain word
template <int S>
__device__ __forceinline__ bool delta_eligible(const DeltaOld<S>& o, bool frame, const int (&len)[S]) {
  bool ok = frame;
#pragma unroll
  for (int s = 0; s < S; ++s) ok = ok && (o.hl[s] >> 16) <= DELTA_MAX_LEN && len[s] <= DELTA_MAX_LEN;
  return ok;
}

// The two-kernel form: k_lane_logic keeps the old state's paint items and frame_ok of every env (W words: hl[S], c0[S],
// fr[2], frame), written right after lane_fetch, for the observation writer behind it.  They live in the frame_ok
// allocation, from the first 256-byte boundary past its N flags; snk_create_ex allocates them whenever the handle's
// Params::delta is set, and no launch sets it otherwise.
template <int S>
struct DeltaPrev {
  static constexpr int W = (2 * S + 3 + 3) & ~3;  // 32 bytes for S <= 2, 48 for S <= 4
};
__device__ __forceinline__ u32* delta_prev(const Params& p) { return reinterpret_cast<u32*>(p.frame_ok + ((p.N + 255) & ~255LL)); }

template <int S>
__device__ __forceinline__ void delta_prev_store(const Params& p, long long e, const LaneRaw<S>& raw) {
  constexpr int RW = LaneRec<S>::RW, W = DeltaPrev<S>::W;
  u32 r[RW], q[W];
#pragma unroll
  for (int i = 0; i < RW / 4; ++i) { r[4 * i] = raw.v[i].x; r[4 * i + 1] = raw.v[i].y; r[4 * i + 2] = raw.v[i].z; r[4 * i + 3] = raw.v[i].w; }
#pragma unroll
  for (int i = 0; i < W; ++i) q[i] = 0;
#pragma unroll
  for (int s = 0; s < S; ++s) { q[s] = r[REC_SNAKE0 + 2 * s]; q[S + s] = r[LaneRec<S>::c0_word(s)]; }
  q[2 * S] = r[REC_SNAKE0 + 2 * S]; q[2 * S + 1] = r[REC_SNAKE0 + 2 * S + 1]; q[2 * S + 2] = raw.frame;
  uint4* g = reinterpret_cast<uint4*>(delta_prev(p) + e * W);
  u64 pol;  // read once by the writer right behind, then rewritten by the next step: keep it in the L2 like the records
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
#pragma unroll
  for (int i = 0; i < W / 4; ++i)
    asm volatile("st.global.L2::cache_hint.v4.u32 [%0], {%1, %2, %3, %4}, %5;" ::"l"(g + i), "r"(q[4 * i]), "r"(q[4 * i + 1]),
                 "r"(q[4 * i + 2]), "r"(q[4 * i + 3]), "l"(pol) : "memory");
}

// the writer's read of it (at the L2: k_lane_logic wrote it a moment ago); `frame` = the old frame_ok
template <int S>
__device__ __forceinline__ DeltaOld<S> delta_prev_load(const Params& p, long long e, bool& frame) {
  constexpr int W = DeltaPrev<S>::W;
  const uint4* g = reinterpret_cast<const uint4*>(delta_prev(p) + e * W);
  u32 q[W];
#pragma unroll
  for (int i = 0; i < W / 4; ++i) { const uint4 v = __ldcg(g + i); q[4 * i] = v.x; q[4 * i + 1] = v.y; q[4 * i + 2] = v.z; q[4 * i + 3] = v.w; }
  DeltaOld<S> o;
#pragma unroll
  for (int s = 0; s < S; ++s) { o.hl[s] = q[s]; o.c0[s] = q[S + s]; }
  o.fr[0] = q[2 * S]; o.fr[1] = q[2 * S + 1];
  frame = q[2 * S + 2] != 0;
  return o;
}

template <int S>
__device__ __forceinline__ DeltaOld<S> delta_old_from_lane(const DeltaOld<S>& o, int owner) {
  DeltaOld<S> d;
#pragma unroll
  for (int s = 0; s < S; ++s) { d.hl[s] = __shfl_sync(FULL, o.hl[s], owner); d.c0[s] = __shfl_sync(FULL, o.c0[s], owner); }
  d.fr[0] = __shfl_sync(FULL, o.fr[0], owner); d.fr[1] = __shfl_sync(FULL, o.fr[1], owner);
  return d;
}

// One sector: two 16-byte shared loads (an image starts 16-byte aligned in HBM, so a sector is 16-byte aligned in
// shared memory), one 32-byte global store (STG.E.ENL2.256) with the observation stream's L2 evict-first policy `pol`.
// The data is in registers before the store issues, so the image may be un-painted right after.
__device__ __forceinline__ void store_sector(u8* g, const u8* s, u64 pol) {
  const uint4 a = *reinterpret_cast<const uint4*>(s), b = *reinterpret_cast<const uint4*>(s + 16);
  asm volatile("st.global.L2::cache_hint.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8}, %9;" ::"l"(g), "r"(a.x), "r"(a.y), "r"(a.z),
               "r"(a.w), "r"(b.x), "r"(b.y), "r"(b.z), "r"(b.w), "l"(pol) : "memory");
}

// the one or two sectors of the C-byte pixel at byte `off` of the image; `a` = the image's HBM address mod 32.  A sector
// outside [0, bytes) is skipped: only a border cell could produce one, and those are never painted.
template <int C>
__device__ __forceinline__ void delta_pixel(u8* g, const u8* tile, int bytes, int a, int off, u64 pol) {
  const int r0 = ((off + a) & ~31) - a, r1 = ((off + C - 1 + a) & ~31) - a;
  if ((u32)r0 <= (u32)(bytes - 32)) store_sector(g + r0, tile + r0, pol);
  if (r1 != r0 && (u32)r1 <= (u32)(bytes - 32)) store_sector(g + r1, tile + r1, pol);
}

// Store the sectors of one env of the image: the paint items whose pixel can differ between the two frames.
//  * Every new fruit and the old cell of a fruit that moved; TIGHT: only a fruit whose cell changed, new and old cell (a
//    fruit that stayed paints the same pixel in both frames).
//  * A snake that moved (`shifted`: neither killed nor reset) has new segment i + 1 = old segment i for i < k =
//    min(old length, new length - 1): of its old body only the segments from k on (the popped tail).  Every new segment;
//    TIGHT: only new segments 0 and 1 (the new head, the old head turned body) and those past k -- the others are
//    body-coloured in both frames.
//  * Any other snake: every old and every new segment.
// A cell where none of these lies holds the same items in the same paint order in both frames, so its pixel is unchanged
// (tests/test_delta_rule_cpu.py checks both rules on oracle trajectories).  The fused kernel keeps the wider rule: there
// the tight one's extra instructions cost more than its 42 % fewer stores save (2x19x19, 131 072 envs on B200: 54.7 vs
// 52.8 us per step); in the observation writer of the two-kernel form the tight rule wins (49.3 vs 51.7 us).
// The items are dealt round-robin to the env's LPE lanes; one loop with one store site keeps the code small (the fused
// kernel lives off the instruction cache, see lane_reset).  `bytes` = bytes of the image that belong to valid envs.
template <int S, int K, bool TIGHT>
__device__ __forceinline__ void delta_store(const Params& p, const PaintEnv<S>& pe, const DeltaOld<S>& po, int slot, int sub, int LPE,
                                            const u8* tile, int bytes, long long e0) {
  constexpr int C = 3 * K;
  if (!pe.valid) return;
  const int V = p.V, F = p.F;
  const long long t0 = e0 * (long long)p.E;
  u8* g = p.obs + t0;
  const int a = (int)(t0 & 31), base = slot * p.E;
  u64 pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  u32 fm = 0;  // TIGHT: the fruits whose cell changed
  if (TIGHT) {
#pragma unroll
    for (int f = 0; f < 4; ++f)
      if (f < F && (int)((po.fr[f >> 1] >> (16 * (f & 1))) & 0xffffu) != pe.fruit[f]) fm |= 1u << f;
  }
  const int nf = TIGHT ? 2 * __popc(fm) : 2 * F;
  // per snake: k[s] matched segments, of which the old ones are left out; TIGHT also leaves out the d[s] = k - 1 new
  // segments 2..k
  int n = nf, k[S], d[S];
#pragma unroll
  for (int s = 0; s < S; ++s) {
    const int nl = pe.len[s], oh = (int)(po.hl[s] & 0xffffu), ol = (int)(po.hl[s] >> 16);
    const u32 m = ol >= 17 ? ~0u : (1u << (2 * max(ol - 1, 0))) - 1u;  // the codes of the old body
    const bool shifted = nl >= 1 && pe.head[s] - codes_disp(pe.c0[s], V, 1) == oh && (((pe.c0[s] >> 2) ^ po.c0[s]) & m) == 0;
    k[s] = shifted ? min(ol, nl - 1) : 0;
    d[s] = TIGHT ? max(k[s] - 1, 0) : 0;
    n += nl - d[s] + ol - k[s];
  }
  for (int j = sub; j < n; j += LPE) {
    int pid = 0;
    if (j < nf) {
      if (TIGHT) {
        const int f = (int)__fns(fm, 0, (j >> 1) + 1);
#pragma unroll
        for (int q = 0; q < 4; ++q)
          if (q == f) pid = (j & 1) ? (int)((po.fr[q >> 1] >> (16 * (q & 1))) & 0xffffu) : pe.fruit[q];
      } else {
#pragma unroll
        for (int f = 0; f < 4; ++f) {
          const int of = (int)((po.fr[f >> 1] >> (16 * (f & 1))) & 0xffffu);
          if (f < F && j == f) pid = pe.fruit[f];
          if (f < F && j == F + f) pid = of == pe.fruit[f] ? -1 : of;  // a fruit that stayed is one of the new items
        }
      }
    } else {
      int i = j - nf, head = 0;
      u32 w = 0;
      bool found = false;
#pragma unroll
      for (int s = 0; s < S; ++s) {
        const int nn = pe.len[s] - d[s], on = (int)(po.hl[s] >> 16) - k[s];
        if (!found && i < nn) { head = pe.head[s]; w = pe.c0[s]; if (TIGHT && i >= 2) i += d[s]; found = true; }
        else if (!found) i -= nn;
        if (!found && i < on) { head = (int)(po.hl[s] & 0xffffu); w = po.c0[s]; i += k[s]; found = true; }
        else if (!found) i -= on;
      }
      pid = head - codes_disp(w, V, i);
    }
    if (pid >= 0) delta_pixel<C>(g, tile, bytes, a, base + pid * C, pol);
  }
}
