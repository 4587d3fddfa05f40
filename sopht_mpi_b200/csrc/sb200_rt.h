// Runtime shim: the kernels in this directory are CUDA (sm_100a).  When built
// with -DSB200_EMU (g++, no nvcc) the same sources compile into a host-thread
// emulation used ONLY by tests/emu to check kernel logic in the GPU-less build
// container.  The emulation is never loaded by the product path.
#pragma once
#include <cstddef>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <cmath>

#ifndef SB200_EMU
// ------------------------------------------------------------------ CUDA ---
#include <cuda_runtime.h>
#define SB_DYN_SMEM(name) extern __shared__ __align__(16) unsigned char name[]
// kernel launch: grid, block, dynamic smem bytes, stream
#define SB_LAUNCH(kernel, grid, block, smem, stream, ...) \
  kernel<<<(grid), (block), (smem), (cudaStream_t)(stream)>>>(__VA_ARGS__)
#define SB_LAUNCH_COOP SB_LAUNCH
#define SB_KERNEL_ATTR_SMEM(kernel, bytes) \
  cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(bytes))
static inline int sb_memset_async(void* p, int v, size_t n, void* stream) {
  return (int)cudaMemsetAsync(p, v, n, (cudaStream_t)stream);
}
static inline int sb_last_launch_error() { return (int)cudaGetLastError(); }
static inline const char* sb_error_string(int e) { return cudaGetErrorString((cudaError_t)e); }
#else
// ------------------------------------------------------------- emulation ---
#include <barrier>
#include <functional>
#include <memory>
#include <thread>
#include <type_traits>
#include <vector>
struct uint3 { unsigned x, y, z; };
struct dim3 {
  unsigned x, y, z;
  dim3(unsigned x_ = 1, unsigned y_ = 1, unsigned z_ = 1) : x(x_), y(y_), z(z_) {}
};
struct float2 { float x, y; };
struct double2 { double x, y; };
struct alignas(16) float4 { float x, y, z, w; };
static inline float2 make_float2(float x, float y) { return float2{x, y}; }
static inline double2 make_double2(double x, double y) { return double2{x, y}; }
static inline float4 make_float4(float x, float y, float z, float w) { return float4{x, y, z, w}; }

#define __global__
#define __device__
#define __host__
#define __forceinline__ inline
#define __shared__ static
#define __launch_bounds__(...)
#define __ldg(p) (*(p))

namespace sbemu {
struct BlockCtx {
  std::unique_ptr<std::barrier<>> block_bar;
  std::vector<std::unique_ptr<std::barrier<>>> warp_bar;
  std::vector<uint64_t> xchg;  // one slot per thread
  std::vector<unsigned char> dyn_smem;
};
extern thread_local uint3 t_threadIdx, t_blockIdx;
extern thread_local dim3 t_blockDim, t_gridDim;
extern thread_local BlockCtx* t_ctx;
extern thread_local unsigned t_linear_tid;
void launch(dim3 grid, dim3 block, size_t smem, bool coop, const std::function<void()>& body);
// Records the address of a launched kernel in the runtime's launch log (sb200_emu_launched_kernels).
// Taking the address also gives every instantiation a symbol of its own where g++ inlines the call.
// Weak: a runtime that keeps no launch log still links, and then nothing is recorded.
__attribute__((weak)) void note_launch(const void* kernel);
}  // namespace sbemu
#define threadIdx (sbemu::t_threadIdx)
#define blockIdx (sbemu::t_blockIdx)
#define blockDim (sbemu::t_blockDim)
#define gridDim (sbemu::t_gridDim)
#define SB_DYN_SMEM(name) unsigned char* name = sbemu::t_ctx->dyn_smem.data()
#define SB_EMU_NOTE_LAUNCH(kernel) (sbemu::note_launch ? sbemu::note_launch((const void*)&kernel) : void())
#define SB_LAUNCH(kernel, grid, block, smem, stream, ...) \
  (SB_EMU_NOTE_LAUNCH(kernel), sbemu::launch((grid), (block), (smem), false, [&]() { kernel(__VA_ARGS__); }))
#define SB_LAUNCH_COOP(kernel, grid, block, smem, stream, ...) \
  (SB_EMU_NOTE_LAUNCH(kernel), sbemu::launch((grid), (block), (smem), true, [&]() { kernel(__VA_ARGS__); }))
#define SB_KERNEL_ATTR_SMEM(kernel, bytes) (0)

static inline void __syncthreads() { sbemu::t_ctx->block_bar->arrive_and_wait(); }
static inline void __threadfence_block() { __atomic_thread_fence(__ATOMIC_SEQ_CST); }
static inline void __syncwarp(unsigned = 0xffffffffu) {
  sbemu::t_ctx->warp_bar[sbemu::t_linear_tid / 32]->arrive_and_wait();
}
template <typename T>
static inline T sb_emu_shfl(T v, unsigned src_lane) {
  static_assert(sizeof(T) <= 8, "shfl payload");
  auto* c = sbemu::t_ctx;
  unsigned tid = sbemu::t_linear_tid, w = tid / 32;
  uint64_t bits = 0;
  std::memcpy(&bits, &v, sizeof(T));
  c->xchg[tid] = bits;
  c->warp_bar[w]->arrive_and_wait();
  uint64_t r = c->xchg[w * 32 + (src_lane & 31)];
  c->warp_bar[w]->arrive_and_wait();
  T out;
  std::memcpy(&out, &r, sizeof(T));
  return out;
}
template <typename T>
static inline T __shfl_xor_sync(unsigned, T v, int m) { return sb_emu_shfl(v, (sbemu::t_linear_tid % 32) ^ m); }
template <typename T>
static inline T __shfl_down_sync(unsigned, T v, unsigned d) {
  unsigned l = sbemu::t_linear_tid % 32;
  return sb_emu_shfl(v, l + d < 32 ? l + d : l);
}
template <typename T>
static inline T __shfl_up_sync(unsigned, T v, unsigned d) {
  unsigned l = sbemu::t_linear_tid % 32;
  return sb_emu_shfl(v, l >= d ? l - d : l);
}
template <typename T>
static inline T __shfl_sync(unsigned, T v, int src) { return sb_emu_shfl(v, (unsigned)src); }

template <typename T>
static inline T atomicAdd(T* p, T v) {
  using U = typename std::conditional<sizeof(T) == 4, uint32_t, uint64_t>::type;
  U* up = reinterpret_cast<U*>(p);
  U expect = __atomic_load_n(up, __ATOMIC_RELAXED);
  for (;;) {
    T cur;
    std::memcpy(&cur, &expect, sizeof(T));
    T nxt = cur + v;
    U desired;
    std::memcpy(&desired, &nxt, sizeof(T));
    if (__atomic_compare_exchange_n(up, &expect, desired, false, __ATOMIC_RELAXED, __ATOMIC_RELAXED))
      return cur;
  }
}
static inline unsigned long long atomicMax(unsigned long long* p, unsigned long long v) {
  unsigned long long e = __atomic_load_n(p, __ATOMIC_RELAXED);
  while (e < v && !__atomic_compare_exchange_n(p, &e, v, false, __ATOMIC_RELAXED, __ATOMIC_RELAXED)) {}
  return e;
}
static inline unsigned atomicMax(unsigned* p, unsigned v) {
  unsigned e = __atomic_load_n(p, __ATOMIC_RELAXED);
  while (e < v && !__atomic_compare_exchange_n(p, &e, v, false, __ATOMIC_RELAXED, __ATOMIC_RELAXED)) {}
  return e;
}
static inline void sincospif(float a, float* s, float* c) {
  *s = (float)std::sin(M_PI * (double)a);
  *c = (float)std::cos(M_PI * (double)a);
}
static inline void sincospi(double a, double* s, double* c) {
  *s = std::sin(M_PI * a);
  *c = std::cos(M_PI * a);
}
static inline int sb_memset_async(void* p, int v, size_t n, void*) {
  std::memset(p, v, n);
  return 0;
}
static inline int sb_last_launch_error() { return 0; }
static inline const char* sb_error_string(int) { return "emu"; }
#endif

// ------------------------------------------------------------- common ------
#define SB_HD __host__ __device__ __forceinline__
#define SB_D __device__ __forceinline__
