// Shared helpers for the CUDA translation units of libeigd_b200.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>

void eigd_set_error(const char* fmt, ...);

extern cudaStream_t g_eigd_stream;
extern int64_t g_eigd_launches;

#define EIGD_CUDA(call)                                                                   \
  do {                                                                                    \
    cudaError_t e_ = (call);                                                              \
    if (e_ != cudaSuccess) {                                                              \
      eigd_set_error("%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); \
      return 100 + (int)e_;                                                               \
    }                                                                                     \
  } while (0)

// launch bookkeeping: every kernel launch of the library goes through this macro
#define EIGD_LAUNCH(kernel, grid, block, smem, ...)                                       \
  do {                                                                                    \
    kernel<<<(grid), (block), (smem), g_eigd_stream>>>(__VA_ARGS__);                      \
    ++g_eigd_launches;                                                                    \
  } while (0)

#define EIGD_CHECK_LAUNCH()                                                               \
  do {                                                                                    \
    cudaError_t e_ = cudaGetLastError();                                                  \
    if (e_ != cudaSuccess) {                                                              \
      eigd_set_error("%s:%d kernel launch -> %s", __FILE__, __LINE__, cudaGetErrorString(e_)); \
      return 100 + (int)e_;                                                               \
    }                                                                                     \
  } while (0)

static inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ---- cooperative kernels with a software grid barrier (dense.cu mgs_sweep, block_krylov.cu block_step) ----
// All of them share one monotonic arrival counter: every CTA adds 1 per barrier, so a launch on G CTAs with b
// barriers adds b * G, and the next launch (stream-ordered) waits for targets counted from the new base.
__device__ __forceinline__ void coop_grid_barrier(unsigned long long* ctr, unsigned long long target) {
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long v;
    asm volatile("red.release.gpu.global.add.u64 [%0], 1;" ::"l"(ctr) : "memory");
    do {
      asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(ctr) : "memory");
    } while (v < target);
  }
  __syncthreads();
}

// The counter of the current device (allocated and zeroed on first use) and the arrivals enqueued so far; the caller
// adds its launch's barriers x grid to *base after the launch.  Defined in dense.cu.
int coop_counter(unsigned long long** ctr, unsigned long long** base);

// Largest co-resident grid of a 256-thread kernel: SMs x min(occupancy, per_sm), at most cap; computed once (*max_grid)
template <class Kernel>
static int coop_max_grid(Kernel kernel, int per_sm, int cap, int* max_grid) {
  if (*max_grid > 0) return 0;
  int dev = 0, sms = 0, occ = 0;
  EIGD_CUDA(cudaGetDevice(&dev));
  EIGD_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  EIGD_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, 256, 0));
  if (occ < 1) { eigd_set_error("cooperative kernel does not fit on an SM"); return 7; }
  int g = sms * (occ < per_sm ? occ : per_sm);
  *max_grid = g > cap ? cap : g;
  return 0;
}
