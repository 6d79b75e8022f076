// snk_grid_conv.cu -- the policy's first convolution read straight from SNK_OBS_GRID cell codes (snk_grid_conv_in,
// snk_grid_conv_in_wgrad; DESIGN.md section 4.16).
//
// A pixel of view k is one of 7 colours, chosen by the cell code alone, and the SAME padding's zeros are the colour of
// an empty cell.  So a 3x3 SAME convolution C_in = 3 -> C over the expanded view is a table lookup per tap:
//   out[p][o] = relu(bias[o] + sum_t T[t][class_k(grid[p + t])][o]),   T[t][c][o] = sum_rgb W[o][rgb][t] colour[c][rgb] / 255
// and its weight gradient is the same identity backwards, through the histogram
//   H[t][c][o] = sum over cells p with class_k(grid[p + t]) = c of g[p][o] (g: incoming gradient behind the ReLU).
// T[t][0] is zero (empty is black), so a cell whose nine taps are all empty is bias + ReLU.  Each cell's nine tap
// classes are packed into one 27-bit key (tap t = 3 (dy + 1) + (dx + 1) in bits 3t .. 3t + 2) and only the non-empty
// taps are visited.
#include <cuda_runtime.h>
#include <stdint.h>

#include "snk_grid_class.cuh"
#include "snk_launch.h"

typedef unsigned char u8;

static constexpr int GC_C = SNK_GRID_CONV_CHANNELS, GC_CLS = SNK_GRID_CONV_CLASSES, GC_TAPS = 9;
static constexpr int FW_THREADS = 256, FW_CELLS = 1024;  // forward: cells per chunk (128 KB of output)
static constexpr int WG_WARPS = 6;                        // wgrad: warps per CTA, each with private bins (41 KB of shared per CTA)
static constexpr int WG_ROWS = SNK_GRID_CONV_PART_FLOATS / GC_C;  // 9 taps x classes 1..6, then the total row
static_assert(WG_ROWS == GC_TAPS * (GC_CLS - 1) + 1, "the partial layout of snk.h");

// the nine tap classes of cell (y, x); `cls` points at the cell in a row-major class image of width V that holds its
// rows y - 1 .. y + 1 (rows outside 0 .. V - 1 are not read: off the image is empty)
static __device__ __forceinline__ unsigned cell_key(const u8* cls, int y, int x, int V) {
  unsigned key = 0;
#pragma unroll
  for (int dy = -1; dy <= 1; ++dy) {
    if (y + dy < 0 || y + dy >= V) continue;
#pragma unroll
    for (int dx = -1; dx <= 1; ++dx)
      if (x + dx >= 0 && x + dx < V) key |= (unsigned)cls[dy * V + dx] << (3 * (3 * (dy + 1) + dx + 1));
  }
  return key;
}

// the same key from the codes in global memory (the backward computes it once per cell, one cell per lane)
static __device__ __forceinline__ unsigned cell_key_codes(const u8* __restrict__ grid, long long c, int V, int view) {
  const long long r = c / V;
  const int x = (int)(c - r * V), y = (int)(r % V);
  unsigned key = 0;
#pragma unroll
  for (int dy = -1; dy <= 1; ++dy) {
    if (y + dy < 0 || y + dy >= V) continue;
#pragma unroll
    for (int dx = -1; dx <= 1; ++dx)
      if (x + dx >= 0 && x + dx < V)
        key |= cell_class(__ldg(grid + c + dy * V + dx), view) << (3 * (3 * (dy + 1) + dx + 1));
  }
  return key;
}

// pops the lowest non-empty tap of `key`: its tap index and class
static __device__ __forceinline__ void pop_tap(unsigned& key, int& t, unsigned& cls) {
  t = (__ffs(key) - 1) / 3;
  cls = (key >> (3 * t)) & 7u;
  key &= ~(7u << (3 * t));
}

// k_grid_conv_in: persistent CTAs over chunks of FW_CELLS consecutive cells of the [n][V][V] batch.  Per chunk the
// classes of its rows and the halo row above and below (rows of the neighbouring envs are staged but masked by the row
// test of cell_key) go to shared memory once per cell, then one key per cell, then thread (cell, q) writes channels
// 4q .. 4q + 3 of its cell: a warp stores 4 whole 128-byte channel rows, 512 contiguous bytes, as streaming stores.
__global__ void __launch_bounds__(FW_THREADS) k_grid_conv_in(const u8* __restrict__ grid, long long n_cells, int V, int view,
                                                            const float4* __restrict__ table, const float4* __restrict__ bias,
                                                            float4* __restrict__ out) {
  __shared__ float4 s_tab[GC_TAPS * GC_CLS * GC_C / 4];
  __shared__ u8 s_cls[FW_CELLS + 4 * 256];  // at most (cells - 1) / V + 4 rows of V <= 256
  __shared__ unsigned s_key[FW_CELLS];
  const int tid = threadIdx.x, q = tid & 7;
  for (int i = tid; i < GC_TAPS * GC_CLS * GC_C / 4; i += FW_THREADS) s_tab[i] = table[i];
  const float4 b = bias[q];
  for (long long c0 = blockIdx.x * (long long)FW_CELLS; c0 < n_cells; c0 += gridDim.x * (long long)FW_CELLS) {
    const int cells = (int)min((long long)FW_CELLS, n_cells - c0);
    const long long r0 = c0 / V - 1;  // first staged row: the halo row above the chunk
    const int nst = (int)((c0 + cells - 1) / V + 2 - r0) * V;
    __syncthreads();  // the previous chunk's classes and keys are consumed
    for (int i = tid; i < nst; i += FW_THREADS) {
      const long long g = r0 * V + i;
      s_cls[i] = g >= 0 && g < n_cells ? (u8)cell_class(__ldg(grid + g), view) : (u8)0;
    }
    __syncthreads();
    for (int i = tid; i < cells; i += FW_THREADS) {
      const long long c = c0 + i, r = c / V;
      const int x = (int)(c - r * V);
      s_key[i] = cell_key(s_cls + (r - r0) * V + x, (int)(r % V), x, V);
    }
    __syncthreads();
    for (int i = tid; i < cells * 8; i += FW_THREADS) {  // i & 7 == q
      unsigned key = s_key[i >> 3];
      float4 a = b;
      while (key) {
        int t;
        unsigned cls;
        pop_tap(key, t, cls);
        const float4 w = s_tab[(t * GC_CLS + cls) * (GC_C / 4) + q];
        a.x += w.x; a.y += w.y; a.z += w.z; a.w += w.w;
      }
      a.x = fmaxf(a.x, 0.f); a.y = fmaxf(a.y, 0.f); a.z = fmaxf(a.z, 0.f); a.w = fmaxf(a.w, 0.f);
      __stcs(out + (c0 << 3) + i, a);
    }
  }
}

// k_grid_conv_in_wgrad: warp per 32 consecutive cells, lane = channel.  Lane j first computes the key of cell j; then,
// cell by cell, every lane reads its channel of the saved output (the ReLU mask) and of the incoming gradient (two
// 128-byte rows per cell, eight cells in flight) and adds the masked gradient to the bins of the cell's non-empty taps
// and to its running total.  The bins are the warp's own, lane j owns column j: no atomics, no races.  At the end the CTA
// adds up its warps in warp order and writes one partial [WG_ROWS][C] to the workspace.
__global__ void __launch_bounds__(WG_WARPS * 32) k_grid_conv_in_wgrad(const u8* __restrict__ grid, long long n_cells, int V,
                                                                     int view, const float* __restrict__ out,
                                                                     const float* __restrict__ gout, float* __restrict__ part) {
  __shared__ float s_bin[WG_WARPS][WG_ROWS][GC_C];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float* bin = &s_bin[warp][0][0];
  for (int i = 0; i < WG_ROWS - 1; ++i) bin[i * GC_C + lane] = 0.f;
  float tot = 0.f;
  const long long n_rounds = (n_cells + 31) / 32;
  for (long long r = blockIdx.x * (long long)WG_WARPS + warp; r < n_rounds; r += gridDim.x * (long long)WG_WARPS) {
    const long long c0 = r * 32;
    const int m = (int)min(32LL, n_cells - c0);
    const unsigned own = lane < m ? cell_key_codes(grid, c0 + lane, V, view) : 0u;
    const float* po = out + c0 * GC_C + lane;
    const float* pg = gout + c0 * GC_C + lane;
    for (int j0 = 0; j0 < m; j0 += 8) {
      float o[8], d[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const bool ok = j0 + u < m;
        o[u] = ok ? __ldcs(po + (j0 + u) * GC_C) : 0.f;
        d[u] = ok ? __ldcs(pg + (j0 + u) * GC_C) : 0.f;
      }
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const float v = o[u] > 0.f ? d[u] : 0.f;
        tot += v;
        unsigned key = __shfl_sync(0xffffffffu, own, (j0 + u) & 31);
        if (j0 + u >= m) key = 0u;
        while (key) {
          int t;
          unsigned cls;
          pop_tap(key, t, cls);
          bin[(t * (GC_CLS - 1) + (int)cls - 1) * GC_C + lane] += v;
        }
      }
    }
  }
  bin[(WG_ROWS - 1) * GC_C + lane] = tot;
  __syncthreads();
  for (int i = threadIdx.x; i < WG_ROWS * GC_C; i += WG_WARPS * 32) {
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < WG_WARPS; ++w) s += (&s_bin[w][0][0])[i];
    part[(long long)blockIdx.x * (WG_ROWS * GC_C) + i] = s;
  }
}

// H from the partials of `n_part` CTAs, in CTA order: CTA t of 9 builds tap t, thread (c, o) class c, channel o.  Class 0
// is the total minus classes 1..6: every (cell, tap) pair has exactly one class, off-image taps included.
__global__ void __launch_bounds__(GC_CLS * GC_C) k_grid_conv_in_hist(const float* __restrict__ part, int n_part,
                                                                    float* __restrict__ hist) {
  __shared__ float s[GC_CLS][GC_C];
  const int t = blockIdx.x, c = threadIdx.x / GC_C, o = threadIdx.x % GC_C;
  const int row = c == 0 ? WG_ROWS - 1 : t * (GC_CLS - 1) + c - 1;
  const float* p = part + row * GC_C + o;
  float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
  int b = 0;
  for (; b + 4 <= n_part; b += 4) {
    a0 += p[(long long)b * (WG_ROWS * GC_C)];
    a1 += p[(long long)(b + 1) * (WG_ROWS * GC_C)];
    a2 += p[(long long)(b + 2) * (WG_ROWS * GC_C)];
    a3 += p[(long long)(b + 3) * (WG_ROWS * GC_C)];
  }
  for (; b < n_part; ++b) a0 += p[(long long)b * (WG_ROWS * GC_C)];
  s[c][o] = (a0 + a1) + (a2 + a3);
  __syncthreads();
  float h = s[c][o];
  if (c == 0)
    for (int k = 1; k < GC_CLS; ++k) h -= s[k][o];
  hist[(t * GC_CLS + c) * GC_C + o] = h;
}

int snk_grid_conv_wgrad_ctas(long long n_cells) {
  const long long want = (n_cells + SNK_GRID_CONV_WGRAD_CELLS_PER_CTA - 1) / SNK_GRID_CONV_WGRAD_CELLS_PER_CTA;
  return (int)(want < SNK_GRID_CONV_WGRAD_MAX_CTAS ? want : SNK_GRID_CONV_WGRAD_MAX_CTAS);
}

cudaError_t snk_launch_grid_conv_in(const uint8_t* grid, long long n_cells, int V, int view, const float* table,
                                    const float* bias, float* out, cudaStream_t stream) {
  int dev = 0, n_sm = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e == cudaSuccess) e = cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
  if (e != cudaSuccess) return e;
  const long long chunks = (n_cells + FW_CELLS - 1) / FW_CELLS, resident = 8LL * n_sm;  // 8 CTAs of 256 threads per SM
  k_grid_conv_in<<<(unsigned)(chunks < resident ? chunks : resident), FW_THREADS, 0, stream>>>(
      grid, n_cells, V, view, reinterpret_cast<const float4*>(table), reinterpret_cast<const float4*>(bias),
      reinterpret_cast<float4*>(out));
  return cudaGetLastError();
}

cudaError_t snk_launch_grid_conv_in_wgrad(const uint8_t* grid, long long n_cells, int V, int view, const float* out,
                                          const float* gout, float* hist, float* work, cudaStream_t stream) {
  const int g = snk_grid_conv_wgrad_ctas(n_cells);
  k_grid_conv_in_wgrad<<<g, WG_WARPS * 32, 0, stream>>>(grid, n_cells, V, view, out, gout, work);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  k_grid_conv_in_hist<<<GC_TAPS, GC_CLS * GC_C, 0, stream>>>(work, g, hist);
  return cudaGetLastError();
}
