// snk_grid_conv84.cu -- the first convolution of nature_cnn on the 84x84 WarpFrame view, read straight from SNK_OBS_GRID
// cell codes (snk_grid_conv84_in, snk_grid_conv84_in_wgrad; DESIGN.md section 4.17).
//
// The view is the grid replicated f = 84 / V times per cell, so an 8x8 stride-4 window over it covers at most C cells per
// axis, and how its 8 rows (columns) fall on those cells depends only on the phase oy mod P, P = f / gcd(f, 4).  With
// the kernel folded per phase and block (a, b) into a table T[py][px][a][b][class][o] (include/snk.h),
//   out[oy][ox][o] = relu(bias[o] + sum_{a,b} T[oy % P][ox % P][a][b][class(grid[cy + a][cx + b])][o])
// and the weight gradient is the same identity backwards through a per-phase, per-block, per-class histogram.  Both
// kernels work phase pair by phase pair, so a CTA needs one phase's C x C x 7 x 32 table slice (3.5 KB for C = 2), not
// the whole table (172 KB at V = 12), and a warp's bins are one phase's.  Each output's C x C block classes are packed
// into one key (block a C + b in bits 3 (a C + b) ..) and only non-empty blocks are visited.
#include <cuda_runtime.h>
#include <stdint.h>

#include "snk_grid_class.cuh"
#include "snk_launch.h"

typedef unsigned char u8;

static constexpr int G8_C = SNK_GRID_CONV_CHANNELS, G8_CLS = SNK_GRID_CONV_CLASSES, G8_OUT = SNK_GRID_CONV84_OUT;
static constexpr int G8_PIX = G8_OUT * G8_OUT;
static constexpr int FW_THREADS = 256, FW_OUTS = 1024;  // forward: outputs of one phase pair per work item (128 KB)

template <int CB> struct Key;  // C x C blocks of 3 bits
template <> struct Key<2> { typedef unsigned T; };
template <> struct Key<4> { typedef unsigned long long T; };
static __device__ __forceinline__ int lowest_bit(unsigned k) { return __ffs(k) - 1; }
static __device__ __forceinline__ int lowest_bit(unsigned long long k) { return __ffsll((long long)k) - 1; }

// cells a window of phase `ph` spans per axis (blocks 0 .. span - 1 are reached)
static __device__ __forceinline__ int span_of(int ph, int f) { return (4 * ph + 7) / f - (4 * ph) / f + 1; }

template <int CB> static constexpr __host__ __device__ int wg_warps() { return CB == 2 ? 8 : 3; }  // 25.6 / 37.2 KB of bins per CTA
template <int CB> static constexpr __host__ __device__ int wg_rows() { return CB * CB * (G8_CLS - 1) + 1; }  // blocks x classes 1..6, total

// the key and the output pixel (sample * 400 + oy * 20 + ox) of output j of phase pair (py, px)
template <int CB>
static __device__ __forceinline__ typename Key<CB>::T out_key(const u8* __restrict__ grid, long long j, int m, int nx, int py,
                                                              int px, int P, int V, int f, int view, long long& pix) {
  const long long s = j / m;
  const int r = (int)(j - s * m), iy = r / nx, oy = py + P * iy, ox = px + P * (r - iy * nx);
  const int cy = 4 * oy / f, cx = 4 * ox / f, sy = span_of(py, f), sx = span_of(px, f);
  const u8* g = grid + s * V * V + cy * V + cx;
  typename Key<CB>::T key = 0;
  for (int a = 0; a < sy; ++a)
    for (int b = 0; b < sx; ++b) key |= (typename Key<CB>::T)cell_class(__ldg(g + a * V + b), view) << (3 * (a * CB + b));
  pix = s * G8_PIX + oy * G8_OUT + ox;
  return key;
}

// k_grid_conv84_in: work item = FW_OUTS consecutive outputs of one phase pair (phase-major order; outputs of a phase in
// (sample, iy, ix) order); each CTA takes a contiguous range of items, so it reloads its table slice only when the phase
// changes.  Per item one key and pixel per output go to shared memory, then thread (output, q) adds the table's float4
// rows for channels 4q .. 4q + 3 and stores them with st.global.cs: whole 128-byte channel rows.
template <int CB>
__global__ void __launch_bounds__(FW_THREADS) k_grid_conv84_in(const u8* __restrict__ grid, long long n, int V, int f, int P,
                                                              int view, const float4* __restrict__ table,
                                                              const float4* __restrict__ bias, float4* __restrict__ out,
                                                              long long per_phase, long long n_items) {
  constexpr int SLICE = CB * CB * G8_CLS * (G8_C / 4);
  __shared__ float4 s_tab[SLICE];
  __shared__ typename Key<CB>::T s_key[FW_OUTS];
  __shared__ long long s_pix[FW_OUTS];
  const int tid = threadIdx.x, q = tid & 7;
  const float4 b = bias[q];
  const long long it0 = n_items * blockIdx.x / gridDim.x, it1 = n_items * (blockIdx.x + 1) / gridDim.x;
  long long loaded = -1;
  for (long long it = it0; it < it1; ++it) {
    const long long ph = it / per_phase, j0 = (it - ph * per_phase) * FW_OUTS;
    const int py = (int)(ph / P), px = (int)(ph - (long long)py * P);
    const int ny = (G8_OUT - py + P - 1) / P, nx = (G8_OUT - px + P - 1) / P, m = ny * nx;
    const long long total = n * m;
    if (j0 >= total) continue;  // the phase has fewer outputs than the largest one
    const int cnt = (int)min((long long)FW_OUTS, total - j0);
    __syncthreads();  // the previous item's keys (and table slice) are consumed
    if (ph != loaded) {
      for (int i = tid; i < SLICE; i += FW_THREADS) s_tab[i] = table[ph * SLICE + i];
      loaded = ph;
    }
    for (int i = tid; i < cnt; i += FW_THREADS) {
      long long pix;
      s_key[i] = out_key<CB>(grid, j0 + i, m, nx, py, px, P, V, f, view, pix);
      s_pix[i] = pix;
    }
    __syncthreads();
    for (int i = tid; i < cnt * 8; i += FW_THREADS) {  // i & 7 == q
      typename Key<CB>::T key = s_key[i >> 3];
      float4 a = b;
      while (key) {
        const int bit = lowest_bit(key), blk = bit / 3;
        const unsigned cls = (unsigned)(key >> (3 * blk)) & 7u;
        key &= ~((typename Key<CB>::T)7u << (3 * blk));
        const float4 w = s_tab[(blk * G8_CLS + (int)cls) * (G8_C / 4) + q];
        a.x += w.x; a.y += w.y; a.z += w.z; a.w += w.w;
      }
      a.x = fmaxf(a.x, 0.f); a.y = fmaxf(a.y, 0.f); a.z = fmaxf(a.z, 0.f); a.w = fmaxf(a.w, 0.f);
      __stcs(out + (s_pix[i >> 3] << 3) + q, a);
    }
  }
}

// k_grid_conv84_in_wgrad: CTA t works on phase pair t / K only (K CTAs per phase pair), warp per 32 consecutive outputs of
// that phase, lane = channel.  Lane j computes output j's key and pixel; then, output by output, every lane reads its
// channel of the saved output (the ReLU mask) and of the gradient (two 128-byte rows per output, eight outputs in flight)
// and adds the masked gradient to the bins of the output's non-empty blocks and to its running total.  The bins are the
// warp's own, lane j owns column j: no atomics, no races.  At the end the CTA adds up its warps in warp order and writes
// one partial [ROWS][32] to the workspace.
template <int CB>
__global__ void __launch_bounds__(wg_warps<CB>() * 32) k_grid_conv84_in_wgrad(const u8* __restrict__ grid, long long n, int V,
                                                                             int f, int P, int view, int K,
                                                                             const float* __restrict__ out,
                                                                             const float* __restrict__ gout,
                                                                             float* __restrict__ part) {
  constexpr int WARPS = wg_warps<CB>(), ROWS = wg_rows<CB>();
  __shared__ float s_bin[WARPS][ROWS][G8_C];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int ph = blockIdx.x / K, k = blockIdx.x - ph * K, py = ph / P, px = ph - py * P;
  const int ny = (G8_OUT - py + P - 1) / P, nx = (G8_OUT - px + P - 1) / P, m = ny * nx;
  float* bin = &s_bin[warp][0][0];
  for (int i = 0; i < ROWS - 1; ++i) bin[i * G8_C + lane] = 0.f;
  float tot = 0.f;
  const long long total = n * m, n_rounds = (total + 31) / 32;
  for (long long r = (long long)k * WARPS + warp; r < n_rounds; r += (long long)K * WARPS) {
    const long long j0 = r * 32;
    const int cnt = (int)min(32LL, total - j0);
    long long own_pix = 0;
    const typename Key<CB>::T own = lane < cnt ? out_key<CB>(grid, j0 + lane, m, nx, py, px, P, V, f, view, own_pix) : 0;
    for (int u0 = 0; u0 < cnt; u0 += 8) {
      float o[8], d[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const long long p = __shfl_sync(0xffffffffu, own_pix, (u0 + u) & 31);
        const bool ok = u0 + u < cnt;
        o[u] = ok ? __ldcs(out + p * G8_C + lane) : 0.f;
        d[u] = ok ? __ldcs(gout + p * G8_C + lane) : 0.f;
      }
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const float v = o[u] > 0.f ? d[u] : 0.f;
        tot += v;
        typename Key<CB>::T key = __shfl_sync(0xffffffffu, own, (u0 + u) & 31);
        if (u0 + u >= cnt) key = 0;
        while (key) {
          const int blk = lowest_bit(key) / 3;
          const int cls = (int)(key >> (3 * blk)) & 7;
          key &= ~((typename Key<CB>::T)7u << (3 * blk));
          bin[(blk * (G8_CLS - 1) + cls - 1) * G8_C + lane] += v;
        }
      }
    }
  }
  bin[(ROWS - 1) * G8_C + lane] = tot;
  __syncthreads();
  for (int i = threadIdx.x; i < ROWS * G8_C; i += WARPS * 32) {
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < WARPS; ++w) s += (&s_bin[w][0][0])[i];
    part[(long long)blockIdx.x * (ROWS * G8_C) + i] = s;
  }
}

// H of phase pair blockIdx.x from its K partials, in CTA order.  Class 0 is the phase's total minus classes 1..6 (every
// output has exactly one class per block); blocks the phase's windows do not reach are zero.
template <int CB>
__global__ void __launch_bounds__(256) k_grid_conv84_in_hist(const float* __restrict__ part, int K, int f, int P,
                                                            float* __restrict__ hist) {
  constexpr int ROWS = wg_rows<CB>(), SLICE = CB * CB * G8_CLS * G8_C;
  __shared__ float s[ROWS * G8_C];
  const int ph = blockIdx.x, sy = span_of(ph / P, f), sx = span_of(ph % P, f);
  const float* p = part + (long long)ph * K * (ROWS * G8_C);
  for (int i = threadIdx.x; i < ROWS * G8_C; i += 256) {
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
    int b = 0;
    for (; b + 4 <= K; b += 4) {
      a0 += p[(long long)b * (ROWS * G8_C) + i];
      a1 += p[(long long)(b + 1) * (ROWS * G8_C) + i];
      a2 += p[(long long)(b + 2) * (ROWS * G8_C) + i];
      a3 += p[(long long)(b + 3) * (ROWS * G8_C) + i];
    }
    for (; b < K; ++b) a0 += p[(long long)b * (ROWS * G8_C) + i];
    s[i] = (a0 + a1) + (a2 + a3);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < SLICE; i += 256) {
    const int o = i % G8_C, c = (i / G8_C) % G8_CLS, blk = i / (G8_CLS * G8_C);
    float h = 0.f;
    if (blk / CB < sy && blk % CB < sx) {
      if (c) {
        h = s[(blk * (G8_CLS - 1) + c - 1) * G8_C + o];
      } else {
        h = s[(ROWS - 1) * G8_C + o];
        for (int k = 1; k < G8_CLS; ++k) h -= s[(blk * (G8_CLS - 1) + k - 1) * G8_C + o];
      }
    }
    hist[(long long)ph * SLICE + i] = h;
  }
}

bool snk_grid_conv84_geometry_of(int V, long long n, GridConv84Geometry& g) {
  if (V < 3 || V > 42 || 84 % V != 0 || n < 0) return false;
  int f = 84 / V, gcd4 = f % 4 == 0 ? 4 : f % 2 == 0 ? 2 : 1, C = 0;
  g.f = f;
  g.P = f / gcd4;
  for (int ph = 0; ph < g.P; ++ph) {
    const int s = (4 * ph + 7) / f - (4 * ph) / f + 1;
    C = s > C ? s : C;
  }
  g.C = C <= 2 ? 2 : 4;  // blocks per axis the kernels are instantiated for (C = 3 never occurs for V | 84)
  if (g.C != C) return false;
  const long long P2 = (long long)g.P * g.P, per = (G8_OUT + g.P - 1) / g.P;
  const long long want = (n * per * per + SNK_GRID_CONV84_WGRAD_OUTPUTS_PER_CTA - 1) / SNK_GRID_CONV84_WGRAD_OUTPUTS_PER_CTA;
  long long cap = (SNK_GRID_CONV84_WGRAD_MAX_CTAS + P2 - 1) / P2;
  g.K = (int)(want < cap ? want : cap);
  g.work_bytes = (size_t)(P2 * g.K * (C * C * (G8_CLS - 1) + 1) * G8_C * 4);
  return true;
}

cudaError_t snk_launch_grid_conv84_in(const uint8_t* grid, long long n, int V, int view, const float* table, const float* bias,
                                      float* out, cudaStream_t stream) {
  GridConv84Geometry g;
  if (!snk_grid_conv84_geometry_of(V, n, g)) return cudaErrorInvalidValue;
  int dev = 0, n_sm = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e == cudaSuccess) e = cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
  if (e != cudaSuccess) return e;
  const long long per = (G8_OUT + g.P - 1) / g.P, per_phase = (n * per * per + FW_OUTS - 1) / FW_OUTS;
  const long long n_items = (long long)g.P * g.P * per_phase, resident = 8LL * n_sm;  // 8 CTAs of 256 threads per SM
  const unsigned ctas = (unsigned)(n_items < resident ? n_items : resident);
  const float4* t4 = reinterpret_cast<const float4*>(table);
  const float4* b4 = reinterpret_cast<const float4*>(bias);
  float4* o4 = reinterpret_cast<float4*>(out);
  if (g.C == 2)
    k_grid_conv84_in<2><<<ctas, FW_THREADS, 0, stream>>>(grid, n, V, g.f, g.P, view, t4, b4, o4, per_phase, n_items);
  else
    k_grid_conv84_in<4><<<ctas, FW_THREADS, 0, stream>>>(grid, n, V, g.f, g.P, view, t4, b4, o4, per_phase, n_items);
  return cudaGetLastError();
}

cudaError_t snk_launch_grid_conv84_in_wgrad(const uint8_t* grid, long long n, int V, int view, const float* out, const float* gout,
                                            float* hist, float* work, cudaStream_t stream) {
  GridConv84Geometry g;
  if (!snk_grid_conv84_geometry_of(V, n, g)) return cudaErrorInvalidValue;
  const unsigned ctas = (unsigned)(g.P * g.P * g.K);
  if (g.C == 2)
    k_grid_conv84_in_wgrad<2><<<ctas, wg_warps<2>() * 32, 0, stream>>>(grid, n, V, g.f, g.P, view, g.K, out, gout, work);
  else
    k_grid_conv84_in_wgrad<4><<<ctas, wg_warps<4>() * 32, 0, stream>>>(grid, n, V, g.f, g.P, view, g.K, out, gout, work);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  if (g.C == 2)
    k_grid_conv84_in_hist<2><<<g.P * g.P, 256, 0, stream>>>(work, g.K, g.f, g.P, hist);
  else
    k_grid_conv84_in_hist<4><<<g.P * g.P, 256, 0, stream>>>(work, g.K, g.f, g.P, hist);
  return cudaGetLastError();
}
