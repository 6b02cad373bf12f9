// Shared device/host helpers for the tgp_b200 kernels (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include "../../include/tgp_b200.h"

namespace tgp {

constexpr int kWarp = 32;
constexpr unsigned kFull = 0xffffffffu;

// Process-wide launch counter (bench.py reports it) and optional per-launch checking
// (TGPB200_DEBUG_SYNC=1: synchronise after every kernel and name the first one that fails).
long long& launch_counter();
bool debug_sync_enabled();
void report_launch_failure(const char* name, cudaError_t e);

inline int launch_status() {
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? TGPB200_OK : TGPB200_ERR_CUDA;
}

// Optional per-kernel timing (bench.py): kernels whose name contains the filter are bracketed by CUDA events on
// their own launch stream; tgpb200_debug_kernel_time_ms() averages the recorded pairs.
bool timing_match(const char* name);
void timing_begin(cudaStream_t st);
void timing_end(cudaStream_t st);

template <typename... KArgs, typename... Args>
inline void launch(const char* name, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                   Args... args) {
  ++launch_counter();
  const bool timed = timing_match(name);
  if (timed) timing_begin(st);
  kernel<<<grid, block, smem, st>>>(args...);
  if (timed) timing_end(st);
  if (debug_sync_enabled()) {
    cudaError_t e = cudaStreamSynchronize(st);
    if (e == cudaSuccess) e = cudaPeekAtLastError();
    if (e != cudaSuccess) report_launch_failure(name, e);
  }
}

// Same as launch() for a kernel that runs as thread-block clusters of `cluster` CTAs along x (grid.x % cluster == 0).
template <typename... KArgs, typename... Args>
inline void launch_cluster(const char* name, void (*kernel)(KArgs...), unsigned grid, unsigned block, unsigned cluster,
                           size_t smem, cudaStream_t st, Args... args) {
  ++launch_counter();
  const bool timed = timing_match(name);
  if (timed) timing_begin(st);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid, 1, 1);
  cfg.blockDim = dim3(block, 1, 1);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = cluster;
  at[0].val.clusterDim.y = 1;
  at[0].val.clusterDim.z = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
  if (timed) timing_end(st);
  if (debug_sync_enabled()) {
    cudaError_t e = cudaStreamSynchronize(st);
    if (e == cudaSuccess) e = cudaPeekAtLastError();
    if (e != cudaSuccess) report_launch_failure(name, e);
  }
}

inline size_t align_up(size_t x, size_t a = 256) { return (x + a - 1) / a * a; }

// Bump allocator over the caller-provided workspace (the torch shim owns the memory).
struct Workspace {
  char* base;
  size_t cap;
  size_t off;
  bool ok;
  Workspace(void* p = nullptr, size_t bytes = 0) : base(static_cast<char*>(p)), cap(bytes), off(0), ok(true) {}
  template <typename T>
  T* take(size_t n) {
    size_t bytes = align_up(n * sizeof(T));
    if (base == nullptr || off + bytes > cap) {
      ok = false;
      off += bytes;
      return nullptr;
    }
    T* r = reinterpret_cast<T*>(base + off);
    off += bytes;
    return r;
  }
  // A region of `bytes` taken from this workspace, as a workspace of its own: a primitive's scratch in a layout.
  Workspace sub(size_t bytes) { return Workspace(take<char>(bytes), bytes); }
};

// Bytes a layout carves: every workspace layout is a struct whose constructor takes all of its regions from a
// Workspace, so its size query builds it over a null workspace (every take fails and is counted).
template <typename Layout, typename... Args>
inline size_t layout_bytes(Args... args) {
  Workspace ws(nullptr, 0);
  Layout l(ws, args...);
  (void)l;
  return ws.off;
}

inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

// 128-bit accesses need a 16-byte aligned base: a contiguous tensor need not have one (a view at a storage offset)
__host__ __device__ inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(kFull, v, o));
  return v;
}
__device__ __forceinline__ int warp_sum_i(int v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
  return v;
}

// Block-wide sum (all threads get the result). `red` must hold >= 32 floats.
__device__ __forceinline__ float block_sum(float v, float* red) {
  int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  v = warp_sum(v);
  __syncthreads();
  if (lane == 0) red[w] = v;
  __syncthreads();
  float r = (lane < nw) ? red[lane] : 0.f;
  r = warp_sum(r);
  return r;
}
__device__ __forceinline__ float block_max(float v, float* red) {
  int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  v = warp_max(v);
  __syncthreads();
  if (lane == 0) red[w] = v;
  __syncthreads();
  float r = (lane < nw) ? red[lane] : -INFINITY;
  r = warp_max(r);
  return r;
}

// 128-bit streaming loads/stores (no L1 allocation) for data touched once.
__device__ __forceinline__ float4 ld_stream_f4(const float4* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ void st_stream_f4(float4* p, const float4& v) {
  asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z),
               "f"(v.w));
}

template <typename T>
__device__ __forceinline__ float to_f32(T v);
template <>
__device__ __forceinline__ float to_f32<float>(float v) {
  return v;
}
template <>
__device__ __forceinline__ float to_f32<__nv_bfloat16>(__nv_bfloat16 v) {
  return __bfloat162float(v);
}
template <typename T>
__device__ __forceinline__ T from_f32(float v);
template <>
__device__ __forceinline__ float from_f32<float>(float v) {
  return v;
}
template <>
__device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float v) {
  return __float2bfloat16_rn(v);
}

}  // namespace tgp
