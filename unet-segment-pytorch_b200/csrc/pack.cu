// Parameter layout conversion at the boundary.  Parameters stay torch-owned fp32 tensors in
// the reference's OIHW layout (the checkpoint wire format, SURVEY.md App. A); the tensor-core
// kernels read bf16 packs that are rebuilt from them:
//   fwd pack   (Cout, taps, Cin)         : K-major B operand of the forward implicit GEMM
//   dgrad pack (Cin, taps flipped, Cout) : the same kernel computes the data gradient
// and the split-K partial weight gradients are folded back into the OIHW fp32 .grad.
#include "launch.cuh"
#include "../../include/unetb200.h"
#include "conv.h"
#include "vec.cuh"

namespace ub2 {

// One block = a 16 (co) x 16 (ci) x TAPS tile, one or nine elements per thread with every load
// issued before the first store.  The OIHW rows are read contiguously (16*TAPS floats per co),
// rounded to bf16 into shared memory, and both packs are written in 32-byte runs along their own
// fastest axis (ci for the forward pack, co for the data-gradient pack).
static constexpr int kPackT = 16;

// FULL: Cin and Cout are multiples of 16, so every index split below divides by a constant (with
// run-time tile extents the integer divisions make the kernel instruction bound).
template <int TAPS, bool FULL>
__device__ __forceinline__ void pack_tile(const float* __restrict__ w, __nv_bfloat16* __restrict__ fwd,
                                          __nv_bfloat16* __restrict__ dgrad, int Cout, int Cin,
                                          const float* __restrict__ out_scale, int ci_tile, int co_tile,
                                          __nv_bfloat16 (*tile)[kPackT * 9 + 2]) {
  const int ci0 = ci_tile * kPackT, co0 = co_tile * kPackT;
  const int nci = FULL ? kPackT : min(kPackT, Cin - ci0), nco = FULL ? kPackT : min(kPackT, Cout - co0);
  const int row = nci * TAPS;  // contiguous floats per output channel in this tile
  const int tid = threadIdx.x;
  float v[TAPS];
#pragma unroll
  for (int k = 0; k < TAPS; ++k) {
    const int idx = tid + k * 256;
    const int col = idx / row, j = idx - col * row;
    v[k] = 0.f;
    if (col < nco) {
      v[k] = __ldg(w + (static_cast<size_t>(co0 + col) * Cin + ci0) * TAPS + j);
      if (out_scale != nullptr) v[k] *= __ldg(out_scale + co0 + col);  // BatchNorm folded (eval)
    }
  }
#pragma unroll
  for (int k = 0; k < TAPS; ++k) {
    const int idx = tid + k * 256;
    const int col = idx / row, j = idx - col * row;
    if (col < nco) tile[col][j] = __float2bfloat16_rn(v[k]);
  }
  __syncthreads();
  if (FULL) {
    // 16-byte stores: a chunk is 8 consecutive bf16 of one output row (2 chunks per row of 16)
    constexpr int kChunks = kPackT * TAPS * 2;
    if (fwd != nullptr) {
      for (int c = tid; c < kChunks; c += 256) {
        const int half = c & 1, t = (c >> 1) % TAPS, col = (c >> 1) / TAPS;
        uint32_t r[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const __nv_bfloat16 lo = tile[col][(half * 8 + 2 * i) * TAPS + t];
          const __nv_bfloat16 hi = tile[col][(half * 8 + 2 * i + 1) * TAPS + t];
          r[i] = static_cast<uint32_t>(__bfloat16_as_ushort(lo)) | (static_cast<uint32_t>(__bfloat16_as_ushort(hi)) << 16);
        }
        *reinterpret_cast<uint4*>(fwd + (static_cast<size_t>(co0 + col) * TAPS + t) * Cin + ci0 + half * 8) =
            make_uint4(r[0], r[1], r[2], r[3]);
      }
    }
    if (dgrad != nullptr) {
      for (int c = tid; c < kChunks; c += 256) {
        const int half = c & 1, t = (c >> 1) % TAPS, cil = (c >> 1) / TAPS;
        uint32_t r[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const __nv_bfloat16 lo = tile[half * 8 + 2 * i][cil * TAPS + t];
          const __nv_bfloat16 hi = tile[half * 8 + 2 * i + 1][cil * TAPS + t];
          r[i] = static_cast<uint32_t>(__bfloat16_as_ushort(lo)) | (static_cast<uint32_t>(__bfloat16_as_ushort(hi)) << 16);
        }
        *reinterpret_cast<uint4*>(dgrad + (static_cast<size_t>(ci0 + cil) * TAPS + (TAPS - 1 - t)) * Cout + co0 + half * 8) =
            make_uint4(r[0], r[1], r[2], r[3]);
      }
    }
    return;
  }
  if (fwd != nullptr) {
#pragma unroll
    for (int k = 0; k < TAPS; ++k) {
      const int idx = tid + k * 256;
      const int cil = idx % nci;
      const int t = (idx / nci) % TAPS;
      const int col = idx / row;
      if (col < nco)
        fwd[(static_cast<size_t>(co0 + col) * TAPS + t) * Cin + ci0 + cil] = tile[col][cil * TAPS + t];
    }
  }
  if (dgrad != nullptr) {
#pragma unroll
    for (int k = 0; k < TAPS; ++k) {
      const int idx = tid + k * 256;
      const int col = idx % nco;
      const int t = (idx / nco) % TAPS;
      const int cil = idx / (nco * TAPS);
      if (cil < nci)
        dgrad[(static_cast<size_t>(ci0 + cil) * TAPS + (TAPS - 1 - t)) * Cout + co0 + col] =
            tile[col][cil * TAPS + t];
    }
  }
}

template <int TAPS, bool FULL>
__global__ void __launch_bounds__(256)
pack_weight_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ fwd,
                   __nv_bfloat16* __restrict__ dgrad, int Cout, int Cin,
                   const float* __restrict__ out_scale) {
  pdl_trigger();
  pdl_wait();
  __shared__ __nv_bfloat16 tile[kPackT][kPackT * 9 + 2];
  pack_tile<TAPS, FULL>(w, fwd, dgrad, Cout, Cin, out_scale, blockIdx.x, blockIdx.y, tile);
}

// Every conv weight of the network in one launch (the packs are rebuilt once per optimizer step):
// desc[t] = {w, fwd, dgrad, Cout, Cin, taps} as int64, blocks[b] = {tensor, ci tile, co tile, edge}.
// edge = 0: a whole 16x16 tile with Cin and Cout multiples of 8 (16-byte stores); otherwise the
// generic tile (partial extents, element stores).
// (min 8 blocks per SM: the register budget of the whole tiles alone; the edge path may spill)
__global__ void __launch_bounds__(256, 8)
pack_weights_multi_kernel(const long long* __restrict__ desc, const int4* __restrict__ blocks) {
  pdl_trigger();
  pdl_wait();
  __shared__ __nv_bfloat16 tile[kPackT][kPackT * 9 + 2];
  const int4 b = blocks[blockIdx.x];
  const long long* d = desc + 6 * b.x;
  const float* w = reinterpret_cast<const float*>(d[0]);
  __nv_bfloat16* fwd = reinterpret_cast<__nv_bfloat16*>(d[1]);
  __nv_bfloat16* dgrad = reinterpret_cast<__nv_bfloat16*>(d[2]);
  const int Cout = static_cast<int>(d[3]), Cin = static_cast<int>(d[4]);
  if (b.w != 0) {
    if (d[5] == 9) pack_tile<9, false>(w, fwd, dgrad, Cout, Cin, nullptr, b.y, b.z, tile);
    else pack_tile<1, false>(w, fwd, dgrad, Cout, Cin, nullptr, b.y, b.z, tile);
  } else if (d[5] == 9) {
    pack_tile<9, true>(w, fwd, dgrad, Cout, Cin, nullptr, b.y, b.z, tile);
  } else {
    pack_tile<1, true>(w, fwd, dgrad, Cout, Cin, nullptr, b.y, b.z, tile);
  }
}

// Stage 1 of the split-K fold when there are many splits: partial[0][i] = sum_s partial[s][i],
// float4 columns x 8 split lanes per block, fixed summation order (deterministic).  In place: every
// element of slot 0 is read (by lane 0) before the block-wide barrier and written after it.
__global__ void __launch_bounds__(256)
wgrad_presum_kernel(float* __restrict__ partial, int splits, long long quads) {
  pdl_trigger();
  pdl_wait();
  __shared__ float4 s_red[8][32];
  const long long q = static_cast<long long>(blockIdx.x) * 32 + threadIdx.x;
  float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
  if (q < quads) {
    const float4* src = reinterpret_cast<const float4*>(partial) + q;
#pragma unroll 4
    for (int s = threadIdx.y; s < splits; s += 8) {
      const float4 v = src[static_cast<size_t>(s) * quads];
      a.x += v.x; a.y += v.y; a.z += v.z; a.w += v.w;
    }
  }
  s_red[threadIdx.y][threadIdx.x] = a;
  __syncthreads();
  if (threadIdx.y == 0 && q < quads) {
    float4 t = s_red[0][threadIdx.x];
#pragma unroll
    for (int y = 1; y < 8; ++y) {
      const float4 v = s_red[y][threadIdx.x];
      t.x += v.x; t.y += v.y; t.z += v.z; t.w += v.w;
    }
    reinterpret_cast<float4*>(partial)[q] = t;
  }
}

// grad[co][ci][t] (+)= sum_s partial[s][t*Cin + ci][co].  One block = 32 co x 8 ci x TAPS: the
// partial rows are read along co (coalesced; a thread's TAPS rows are independent loads in
// flight together), transposed through shared memory, and each output channel's 8*TAPS
// consecutive OIHW floats are written together.  Fixed summation order (deterministic).
static constexpr int kRedCi = 8;

template <int TAPS>
__device__ __forceinline__ void reduce_tile(const float* __restrict__ partial, int splits, int Cout, int Cin,
                                            float* __restrict__ grad, int accumulate, int co_tile,
                                            int ci_tile, float (*tile)[kRedCi * 9 + 1]) {
  const int co0 = co_tile * 32, ci0 = ci_tile * kRedCi;
  const int nci = min(kRedCi, Cin - ci0);
  const size_t total = static_cast<size_t>(Cout) * Cin * TAPS;
  const int co = co0 + threadIdx.x;
  const int cil = threadIdx.y;      // blockDim.y == kRedCi: one source channel per thread row
  float a[TAPS];
#pragma unroll
  for (int t = 0; t < TAPS; ++t) a[t] = 0.f;
  if (co < Cout && cil < nci) {
    const float* src = partial + static_cast<size_t>(ci0 + cil) * Cout + co;
    for (int s = 0; s < splits; ++s) {
#pragma unroll
      for (int t = 0; t < TAPS; ++t) a[t] += __ldg(src + s * total + static_cast<size_t>(t) * Cin * Cout);
    }
  }
#pragma unroll
  for (int t = 0; t < TAPS; ++t) tile[threadIdx.x][cil * TAPS + t] = a[t];
  __syncthreads();
  const int row = nci * TAPS;
  for (int col = threadIdx.y; col < 32 && co0 + col < Cout; col += 8) {
    float* dst = grad + (static_cast<size_t>(co0 + col) * Cin + ci0) * TAPS;
    for (int j = threadIdx.x; j < row; j += 32) {
      const float v = tile[col][j];
      dst[j] = accumulate ? dst[j] + v : v;
    }
  }
}

template <int TAPS>
__global__ void __launch_bounds__(256)
wgrad_reduce_kernel(const float* __restrict__ partial, int splits, int Cout, int Cin,
                    float* __restrict__ grad, int accumulate) {
  pdl_trigger();
  pdl_wait();
  __shared__ float tile[32][kRedCi * 9 + 1];
  reduce_tile<TAPS>(partial, splits, Cout, Cin, grad, accumulate, blockIdx.x, blockIdx.y, tile);
}

// Several layers per launch (one launch per gradient bucket instead of one or two per layer).
// The item table travels as a kernel argument, so the launch can sit in a captured graph.
struct ReduceItems {
  Ub2ReduceItem item[UB2_REDUCE_MAX_ITEMS];
  int first_block[UB2_REDUCE_MAX_ITEMS + 1];
  int n;
};

__device__ __forceinline__ int find_item(const ReduceItems& t, int block) {
  int i = 0;
  while (i + 1 < t.n && block >= t.first_block[i + 1]) ++i;
  return i;
}

__global__ void __launch_bounds__(256)
wgrad_presum_multi_kernel(const __grid_constant__ ReduceItems t) {
  pdl_trigger();
  pdl_wait();
  __shared__ float4 s_red[8][32];
  const int i = find_item(t, blockIdx.x);
  const Ub2ReduceItem& it = t.item[i];
  const long long quads = static_cast<long long>(it.Cout) * it.Cin * it.taps / 4;
  const long long q = static_cast<long long>(blockIdx.x - t.first_block[i]) * 32 + threadIdx.x;
  float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
  if (q < quads) {
    const float4* src = reinterpret_cast<const float4*>(it.partial) + q;
#pragma unroll 4
    for (int s = threadIdx.y; s < it.splits; s += 8) {
      const float4 v = src[static_cast<size_t>(s) * quads];
      a.x += v.x; a.y += v.y; a.z += v.z; a.w += v.w;
    }
  }
  s_red[threadIdx.y][threadIdx.x] = a;
  __syncthreads();
  if (threadIdx.y == 0 && q < quads) {
    float4 r = s_red[0][threadIdx.x];
#pragma unroll
    for (int y = 1; y < 8; ++y) {
      const float4 v = s_red[y][threadIdx.x];
      r.x += v.x; r.y += v.y; r.z += v.z; r.w += v.w;
    }
    reinterpret_cast<float4*>(it.partial)[q] = r;
  }
}

__global__ void __launch_bounds__(256)
wgrad_reduce_multi_kernel(const __grid_constant__ ReduceItems t, int accumulate) {
  pdl_trigger();
  pdl_wait();
  __shared__ float tile[32][kRedCi * 9 + 1];
  const int i = find_item(t, blockIdx.x);
  const Ub2ReduceItem& it = t.item[i];
  const int local = blockIdx.x - t.first_block[i];
  const int co_tiles = (it.Cout + 31) / 32;
  if (it.taps == 9)
    reduce_tile<9>(it.partial, it.splits, it.Cout, it.Cin, it.grad, accumulate, local % co_tiles, local / co_tiles, tile);
  else
    reduce_tile<1>(it.partial, it.splits, it.Cout, it.Cin, it.grad, accumulate, local % co_tiles, local / co_tiles, tile);
}

}  // namespace ub2

using namespace ub2;

extern "C" {

int ub2_version(void) { return 100; }

int ub2_pack_conv_weight(const float* w, void* fwd, void* dgrad, int Cout, int Cin, int taps,
                         const float* out_scale, void* stream) {
  if (Cout <= 0 || Cin <= 0 || (taps != 1 && taps != 9)) return UB2_ERR_SHAPE;
  const dim3 grid((Cin + kPackT - 1) / kPackT, (Cout + kPackT - 1) / kPackT);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  __nv_bfloat16* f = static_cast<__nv_bfloat16*>(fwd);
  __nv_bfloat16* d = static_cast<__nv_bfloat16*>(dgrad);
  const bool full = Cin % kPackT == 0 && Cout % kPackT == 0;
  if (taps == 9 && full) launch(pack_weight_kernel<9, true>, grid, 256, 0, st, w, f, d, Cout, Cin, out_scale);
  else if (taps == 9) launch(pack_weight_kernel<9, false>, grid, 256, 0, st, w, f, d, Cout, Cin, out_scale);
  else if (full) launch(pack_weight_kernel<1, true>, grid, 256, 0, st, w, f, d, Cout, Cin, out_scale);
  else launch(pack_weight_kernel<1, false>, grid, 256, 0, st, w, f, d, Cout, Cin, out_scale);
  return static_cast<int>(cudaGetLastError());
}

int ub2_wgrad_reduce_multi(const Ub2ReduceItem* items, int n, int accumulate, void* stream) {
  if (items == nullptr || n <= 0 || n > UB2_REDUCE_MAX_ITEMS) return UB2_ERR_SHAPE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  ReduceItems pre{}, red{};
  int pre_blocks = 0, red_blocks = 0;
  for (int i = 0; i < n; ++i) {
    const Ub2ReduceItem& it = items[i];
    if (it.Cout <= 0 || it.Cin <= 0 || it.splits <= 0 || (it.taps != 1 && it.taps != 9)) return UB2_ERR_SHAPE;
    const long long total = static_cast<long long>(it.Cout) * it.Cin * it.taps;
    Ub2ReduceItem r = it;
    if (it.splits > 8 && total % 4 == 0) {   // many splits: column sums first, all SMs busy
      pre.item[pre.n] = it;
      pre.first_block[pre.n] = pre_blocks;
      pre_blocks += static_cast<int>((total / 4 + 31) / 32);
      ++pre.n;
      r.splits = 1;
    }
    red.item[i] = r;
    red.first_block[i] = red_blocks;
    red_blocks += ((it.Cout + 31) / 32) * ((it.Cin + kRedCi - 1) / kRedCi);
  }
  red.n = n;
  pre.first_block[pre.n] = pre_blocks;
  red.first_block[n] = red_blocks;
  if (pre.n > 0) launch(wgrad_presum_multi_kernel, pre_blocks, dim3(32, 8), 0, st, pre);
  launch(wgrad_reduce_multi_kernel, red_blocks, dim3(32, kRedCi), 0, st, red, accumulate);
  return static_cast<int>(cudaGetLastError());
}

int ub2_pack_conv_weights_multi(const long long* desc, const int* blocks, int nblocks, void* stream) {
  if (nblocks <= 0) return UB2_ERR_SHAPE;
  launch(pack_weights_multi_kernel, nblocks, 256, 0, static_cast<cudaStream_t>(stream), desc, reinterpret_cast<const int4*>(blocks));
  return static_cast<int>(cudaGetLastError());
}

int ub2_wgrad_reduce(float* partial, int splits, int Cout, int Cin, int taps, float* grad,
                     int accumulate, void* stream) {
  if (Cout <= 0 || Cin <= 0 || splits <= 0 || (taps != 1 && taps != 9)) return UB2_ERR_SHAPE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const long long total = static_cast<long long>(Cout) * Cin * taps;
  if (splits > 8 && total % 4 == 0) {  // many splits: column sums first, all SMs busy
    const long long quads = total / 4;
    launch(wgrad_presum_kernel, static_cast<unsigned>((quads + 31) / 32), dim3(32, 8), 0, st, partial, splits, quads);
    splits = 1;
  }
  const dim3 grid((Cout + 31) / 32, (Cin + kRedCi - 1) / kRedCi);
  if (taps == 9)
    launch(wgrad_reduce_kernel<9>, grid, dim3(32, kRedCi), 0, st, partial, splits, Cout, Cin, grad, accumulate);
  else
    launch(wgrad_reduce_kernel<1>, grid, dim3(32, kRedCi), 0, st, partial, splits, Cout, Cin, grad, accumulate);
  return static_cast<int>(cudaGetLastError());
}

}  // extern "C"
