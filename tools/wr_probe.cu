// wr_probe.cu -- what does this box sustain for a WRITE-ONLY stream issued the way the env kernels issue theirs?
// (timing aid, not product code)   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o tools/wr_probe tools/wr_probe.cu
//
// Every CTA owns one or two shared-memory buffers holding a constant pattern and streams "pieces" of `piece` bytes to
// global memory: piece p = blockIdx.x + k * gridDim.x (the env kernels' assignment: at any moment the CTAs write one
// contiguous window of gridDim.x pieces).  Variants: TMA bulk stores (one thread issues, `depth` pieces in flight per CTA)
// or 16-byte st.global by all threads; piece size; CTAs per SM.  Prints GB/s per variant.
//
// `wr_probe scatter [envs] [env_bytes]`: the delta store of the fused lane kernel instead.  A buffer of envs x env_bytes
// (default 131 072 x 2 646 = 347 MB, the headline observation buffer) is written as scattered 32-byte sectors, about 6.6
// per env at hashed positions inside the env's interior, in the env kernel's piece order (2 warps per CTA, each warp a
// batch of 32 envs = 4 images of 8 envs, 4 lanes per env, batches strided over the grid).  Variants: full sectors
// (st.global.v8.b32, STG.E.ENL2.256) with the L2 evict-first policy and without, and 16-byte half-sector stores (which
// make the L2 fetch the rest of the sector from DRAM before it can write).  The full TMA stream of the same buffer is
// timed beside them.  Prints us per pass (one pass = one step's worth of stores).
#include <cstdio>
#include <cstdlib>
#include <cstdint>
#include <cstring>
#include <cuda_runtime.h>

__device__ __forceinline__ void bulk_store(void* g, const void* s, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"((uint64_t)__cvta_generic_to_global(g)),
               "r"((uint32_t)__cvta_generic_to_shared(s)), "r"(bytes) : "memory");
}

template <int DEPTH>
__global__ void __launch_bounds__(256) k_tma(uint8_t* out, long long n_pieces, int piece, int spin) {
  extern __shared__ __align__(128) uint8_t smem[];
  for (int i = threadIdx.x; i < piece * DEPTH / 4; i += blockDim.x) reinterpret_cast<uint32_t*>(smem)[i] = 0x01020304u * (i & 63);
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  __syncthreads();
  int buf = 0;
  for (long long p = blockIdx.x; p < n_pieces; p += gridDim.x) {
    if (threadIdx.x == 0) {
      if (DEPTH == 1) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
      else asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
      uint8_t* g = out + p * (long long)piece;
      const uint8_t* s = smem + buf * piece;
      for (int off = 0; off < piece; off += 16384) bulk_store(g + off, s + off, (uint32_t)min(16384, piece - off));
      asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    }
    if (spin) {  // stand-in for the work between two pieces (expansion / painting): all threads, `spin` dependent FMAs
      float x = (float)threadIdx.x;
      for (int i = 0; i < spin; ++i) x = x * 1.0001f + 0.5f;
      if (x == 12345.f) out[0] = 1;
      __syncthreads();
    }
    buf = (buf + 1) % DEPTH;
  }
  if (threadIdx.x == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

__global__ void __launch_bounds__(256) k_stg(uint8_t* out, long long n_pieces, int piece) {
  const uint4 v = make_uint4(1, 2, 3, threadIdx.x);
  for (long long p = blockIdx.x; p < n_pieces; p += gridDim.x) {
    uint4* g = reinterpret_cast<uint4*>(out + p * (long long)piece);
    for (int i = threadIdx.x; i < piece / 16; i += blockDim.x) __stcs(g + i, v);
  }
}

__device__ __forceinline__ uint32_t hash32(uint32_t x) {
  x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16;
  return x;
}

// MODE 0: 32-byte sector, evict-first; 1: 32-byte sector, no policy; 2: 16-byte half sector, evict-first
template <int MODE>
__global__ void __launch_bounds__(64) k_scatter(uint8_t* out, long long n_envs, int env_bytes, uint32_t salt) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int slot = lane >> 2, sub = lane & 3;  // 8 envs per image, 4 lanes per env
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  const long long n_batches = (n_envs + 31) / 32;
  for (long long b = (long long)blockIdx.x * 2 + warp; b < n_batches; b += (long long)gridDim.x * 2) {
    for (int q = 0; q < 4; ++q) {
      const long long e = b * 32 + q * 8 + slot;
      if (e >= n_envs) continue;
      const uint32_t h0 = hash32((uint32_t)e * 2654435761u + salt);
      const int n_sec = 6 + ((h0 & 1023) < 614);  // 6.6 sectors per env on average
      const int interior = env_bytes - 2 * 132;
      for (int j = sub; j < n_sec; j += 4) {
        const uint32_t h = hash32(h0 + (uint32_t)j * 0x9e3779b9u);
        const long long off = (e * env_bytes + 132 + (long long)(h % (uint32_t)interior)) & ~31ll;
        uint8_t* g = out + off;
        const uint32_t v = h;
        if (MODE == 0)
          asm volatile("st.global.L2::cache_hint.v8.b32 [%0], {%1, %1, %1, %1, %1, %1, %1, %1}, %2;" ::"l"(g), "r"(v), "l"(pol) : "memory");
        else if (MODE == 1)
          asm volatile("st.global.v8.b32 [%0], {%1, %1, %1, %1, %1, %1, %1, %1};" ::"l"(g), "r"(v) : "memory");
        else
          asm volatile("st.global.L2::cache_hint.v4.b32 [%0], {%1, %1, %1, %1}, %2;" ::"l"(g), "r"(v), "l"(pol) : "memory");
      }
    }
  }
}

static int scatter_main(int argc, char** argv) {
  const long long n_envs = argc > 2 ? atoll(argv[2]) : 131072;
  const int env_bytes = argc > 3 ? atoi(argv[3]) : 2646;
  const size_t total = (size_t)n_envs * env_bytes;
  uint8_t* d;
  if (cudaMalloc(&d, total + (1 << 20)) != cudaSuccess) { printf("alloc failed\n"); return 1; }
  cudaMemset(d, 0, total);
  int n_sm = 0;
  cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, 0);
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0); cudaEventCreate(&e1);
  printf("scatter: %lld envs x %d B = %.1f MB, %d SMs, 5 CTAs of 2 warps per SM, 20 passes per timing, best of 5\n", n_envs, env_bytes,
         total / 1e6, n_sm);
  const int grid = n_sm * 5;
  auto time_it = [&](const char* tag, double bytes_per_pass, auto launch) {
    float best = 1e9f;
    for (int rep = 0; rep < 6; ++rep) {
      cudaEventRecord(e0);
      for (int k = 0; k < 20; ++k) launch(rep * 20 + k);
      cudaEventRecord(e1);
      cudaEventSynchronize(e1);
      float ms; cudaEventElapsedTime(&ms, e0, e1);
      if (rep && ms < best) best = ms;
    }
    const double us = best * 1e3 / 20;
    cudaError_t err = cudaGetLastError();
    printf("%-44s %8.2f us per pass  %7.0f GB/s of stored bytes %s\n", tag, us, bytes_per_pass / (us * 1e-6) / 1e9, err ? cudaGetErrorString(err) : "");
  };
  const double sec_bytes = 6.6 * 32.0 * (double)n_envs;
  time_it("sectors 32 B, st.v8, L2 evict-first", sec_bytes, [&](int k) { k_scatter<0><<<grid, 64>>>(d, n_envs, env_bytes, (uint32_t)k); });
  time_it("sectors 32 B, st.v8, no L2 policy", sec_bytes, [&](int k) { k_scatter<1><<<grid, 64>>>(d, n_envs, env_bytes, (uint32_t)k); });
  time_it("half sectors 16 B, st.v4, L2 evict-first", sec_bytes / 2, [&](int k) { k_scatter<2><<<grid, 64>>>(d, n_envs, env_bytes, (uint32_t)k); });
  // the whole-image stream of the same buffer: TMA bulk stores of 8-env images (21 168 B at 2 646 B), 10 per SM
  const int piece = 8 * env_bytes;
  if (piece % 16 == 0 && piece <= 48 * 1024) {
    cudaFuncSetAttribute(k_tma<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, piece);
    time_it("whole images, TMA bulk, 10 CTAs/SM", (double)total, [&](int) { k_tma<1><<<n_sm * 10, 256, piece>>>(d, (long long)(total / piece), piece, 0); });
  }
  cudaFree(d);
  return 0;
}

int main(int argc, char** argv) {
  if (argc > 1 && !strcmp(argv[1], "scatter")) return scatter_main(argc, argv);
  const size_t total = argc > 1 ? (size_t)atoll(argv[1]) : (size_t)131072 * 42336;
  uint8_t* d;
  if (cudaMalloc(&d, total + (1 << 20)) != cudaSuccess) { printf("alloc failed\n"); return 1; }
  cudaMemset(d, 0, total);
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0); cudaEventCreate(&e1);
  int n_sm = 0;
  cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, 0);
  const int pieces[] = {42336, 21168, 10080, 4032, 2016 * 16};
  const int ctas[] = {2, 5, 10};
  printf("total %.1f MB, %d SMs\n", total / 1e6, n_sm);
  auto run = [&](const char* tag, int piece, int per_sm, int depth, int spin, int stg) {
    const long long n = (long long)(total / piece);
    const int grid = n_sm * per_sm;
    const size_t smem = (size_t)piece * depth;
    if (!stg && smem * per_sm > 220 * 1024) return;
    if (!stg) {
      if (depth == 1) cudaFuncSetAttribute(k_tma<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      else cudaFuncSetAttribute(k_tma<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    }
    float best = 1e9f;
    for (int rep = 0; rep < 4; ++rep) {
      cudaEventRecord(e0);
      if (stg) k_stg<<<grid, 256>>>(d, n, piece);
      else if (depth == 1) k_tma<1><<<grid, 256, smem>>>(d, n, piece, spin);
      else k_tma<2><<<grid, 256, smem>>>(d, n, piece, spin);
      cudaEventRecord(e1);
      cudaEventSynchronize(e1);
      float ms; cudaEventElapsedTime(&ms, e0, e1);
      if (rep && ms < best) best = ms;
    }
    cudaError_t err = cudaGetLastError();
    printf("%-4s piece %6d  %2d CTAs/SM  depth %d  spin %5d : %8.1f us  %7.0f GB/s %s\n", tag, piece, per_sm, depth, spin, best * 1e3,
           (double)n * piece / (best * 1e-3) / 1e9, err ? cudaGetErrorString(err) : "");
  };
  for (int piece : pieces)
    for (int c : ctas) {
      run("tma", piece, c, 1, 0, 0);
      run("tma", piece, c, 2, 0, 0);
    }
  for (int c : {5, 10}) { run("tma", 42336, c > 5 ? 5 : c, 1, 2000, 0); run("tma", 21168, c, 2, 1000, 0); }
  for (int piece : {42336, 4032}) for (int c : {5, 8}) run("stg", piece, c, 1, 0, 1);
  // a window that advances linearly at fine grain: pieces of 4 KB with many CTAs = the fill kernel's pattern
  run("stg", 4096, 8, 1, 0, 1);
  run("tma", 4096, 10, 2, 0, 0);
  return 0;
}
