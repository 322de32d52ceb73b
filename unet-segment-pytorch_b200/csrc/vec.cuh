// Small helpers shared by the bandwidth-bound kernels: 128-bit bf16x8 vectors,
// warp / block reductions, grid sizing.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace ub2 {

struct F8 {
  float v[8];
};

__device__ __forceinline__ F8 unpack8(const uint4& u) {
  F8 r;
  r.v[0] = __uint_as_float(u.x << 16);
  r.v[1] = __uint_as_float(u.x & 0xFFFF0000u);
  r.v[2] = __uint_as_float(u.y << 16);
  r.v[3] = __uint_as_float(u.y & 0xFFFF0000u);
  r.v[4] = __uint_as_float(u.z << 16);
  r.v[5] = __uint_as_float(u.z & 0xFFFF0000u);
  r.v[6] = __uint_as_float(u.w << 16);
  r.v[7] = __uint_as_float(u.w & 0xFFFF0000u);
  return r;
}
__device__ __forceinline__ uint32_t pack2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ uint4 pack8(const F8& f) {
  uint4 u;
  u.x = pack2(f.v[0], f.v[1]);
  u.y = pack2(f.v[2], f.v[3]);
  u.z = pack2(f.v[4], f.v[5]);
  u.w = pack2(f.v[6], f.v[7]);
  return u;
}
__device__ __forceinline__ F8 load8(const __nv_bfloat16* p) {
  return unpack8(__ldg(reinterpret_cast<const uint4*>(p)));
}
// streaming variants: data touched once
__device__ __forceinline__ F8 load8_stream(const __nv_bfloat16* p) {
  uint4 u;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(u.x), "=r"(u.y), "=r"(u.z), "=r"(u.w)
               : "l"(p));
  return unpack8(u);
}
__device__ __forceinline__ uint4 ld_stream16(const void* p) {   // any 16 bytes: 8 bf16 or 4 fp32
  uint4 u;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(u.x), "=r"(u.y), "=r"(u.z), "=r"(u.w)
               : "l"(p));
  return u;
}
__device__ __forceinline__ void store8(__nv_bfloat16* p, const F8& f) {
  *reinterpret_cast<uint4*>(p) = pack8(f);
}
__device__ __forceinline__ F8 loadf8(const float* p) {
  F8 r;
  const float4 a = __ldg(reinterpret_cast<const float4*>(p));
  const float4 b = __ldg(reinterpret_cast<const float4*>(p) + 1);
  r.v[0] = a.x; r.v[1] = a.y; r.v[2] = a.z; r.v[3] = a.w;
  r.v[4] = b.x; r.v[5] = b.y; r.v[6] = b.z; r.v[7] = b.w;
  return r;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Deterministic cross-block reduction of per-block partial rows laid out [row][NS][C] (doubles).
// Launch with blockDim = (32, 32): x = channel lane (coalesced), y = row group.  Threads with
// threadIdx.y == 0 return the totals for channel `c`.
template <int NS>
__device__ __forceinline__ void rows_sum(const double* __restrict__ partials, int rows, int C, int c,
                                         double (&out)[NS], double* smem /* [NS][32][33] */) {
  double acc[NS];
#pragma unroll
  for (int k = 0; k < NS; ++k) acc[k] = 0.0;
  if (c < C) {
    for (int r = threadIdx.y; r < rows; r += 32) {
#pragma unroll
      for (int k = 0; k < NS; ++k) acc[k] += partials[(static_cast<size_t>(r) * NS + k) * C + c];
    }
  }
#pragma unroll
  for (int k = 0; k < NS; ++k) smem[(k * 32 + threadIdx.y) * 33 + threadIdx.x] = acc[k];
  __syncthreads();
  if (threadIdx.y == 0) {
#pragma unroll
    for (int k = 0; k < NS; ++k) {
      double s = 0.0;
      for (int y = 0; y < 32; ++y) s += smem[(k * 32 + y) * 33 + threadIdx.x];
      out[k] = s;
    }
  }
}

// The same reduction for blockDim = (8, 128): 8 channels per block (grid = ceil(C / 8)), 128 row
// lanes, so a few hundred rows are one or two independent loads per thread followed by a
// shared-memory tree — the latency of these tiny kernels is what they cost.  Fixed order.
template <int NS>
__device__ __forceinline__ void rows_sum_wide(const double* __restrict__ partials, int rows, int C, int c,
                                              double (&out)[NS], double* smem /* [NS][128][9] */) {
  double acc[NS];
#pragma unroll
  for (int k = 0; k < NS; ++k) acc[k] = 0.0;
  if (c < C) {
#pragma unroll 4
    for (int r = threadIdx.y; r < rows; r += 128) {
#pragma unroll
      for (int k = 0; k < NS; ++k) acc[k] += partials[(static_cast<size_t>(r) * NS + k) * C + c];
    }
  }
#pragma unroll
  for (int k = 0; k < NS; ++k) smem[(k * 128 + threadIdx.y) * 9 + threadIdx.x] = acc[k];
  __syncthreads();
  for (int s = 64; s >= 1; s >>= 1) {
    if (threadIdx.y < s) {
#pragma unroll
      for (int k = 0; k < NS; ++k)
        smem[(k * 128 + threadIdx.y) * 9 + threadIdx.x] += smem[(k * 128 + threadIdx.y + s) * 9 + threadIdx.x];
    }
    __syncthreads();
  }
  if (threadIdx.y == 0) {
#pragma unroll
    for (int k = 0; k < NS; ++k) out[k] = smem[(k * 128) * 9 + threadIdx.x];
  }
}

// Host-side argument checks: the pointer is a multiple of `bytes` (NULL passes; callers check it separately).
inline bool aligned_to(const void* p, uintptr_t bytes) { return (reinterpret_cast<uintptr_t>(p) & (bytes - 1)) == 0; }

// Grid for a bandwidth-bound grid-stride kernel: a multiple of the SM count.
inline int stream_grid(long long work_items, int threads, int sms, int blocks_per_sm = 8) {
  long long need = (work_items + threads - 1) / threads;
  long long cap = static_cast<long long>(sms) * blocks_per_sm;
  if (need >= cap) return static_cast<int>(cap);
  return static_cast<int>(need < 1 ? 1 : need);
}

}  // namespace ub2
