// The two ends of the network, both far below the tensor-core ridge (SURVEY.md App. B):
//
//  * conv_in: the first 3x3 convolution (inc.double_conv.0, layers.py:32) with Cin = n_channels
//    (1 for CT slices): K = 9*Cin, arithmetic intensity ~9 flop/B -> a direct fp32 CUDA-core
//    convolution reading the fp32 NCHW input and writing NHWC bf16 + BatchNorm statistics,
//    its weight gradient, and its data gradient dx (fp32 NCHW, the network input's layout) for
//    callers that differentiate with respect to the input (saliency maps, adversarial steps, a
//    U-Net behind another trainable stage).  The data-gradient kernels are templated over the dy
//    element type and serve both precisions (bf16 dy here, fp32 dy of the fp32 / TF32 mode).
//  * outc: OutConv's 1x1 conv with bias (layers.py:120) C -> n_classes, writing fp32 NCHW
//    logits, and its backward (data gradient NHWC bf16, weight / bias gradients).
#include "launch.cuh"
#include "../../include/unetb200.h"
#include "conv.h"
#include "vec.cuh"

namespace ub2 {

static constexpr int kHeadThreads = 256;
static constexpr int kMaxClasses = 8;
static constexpr int kMaxCin = 4;

// ------------------------------------------------------------------------------ conv_in
// REGW: Cin == 1 and the thread's 8x9 weights live in registers (the shared-memory weight reads
// otherwise bound the kernel: 18 conflicted LDS.128 per pixel).
template <bool REGW>
__global__ void __launch_bounds__(kHeadThreads)
conv_in_fwd_kernel(const float* __restrict__ x, const float* __restrict__ w, __nv_bfloat16* __restrict__ y,
                   int ld_y, double* partials, int N, int Cin, int H, int W, int Cout) {
  pdl_trigger();
  pdl_wait();
  extern __shared__ float s_dyn[];
  float* s_w = s_dyn;                         // [Cin*9][Cout]
  float* s_red = s_dyn + Cin * 9 * Cout;      // [lanes][cgs][16]
  for (int i = threadIdx.x; i < Cout * Cin * 9; i += blockDim.x) {
    const int co = i / (Cin * 9), r = i % (Cin * 9);
    s_w[r * Cout + co] = w[i];
  }
  __syncthreads();
  const int cgs = Cout / 8;
  const int lanes = blockDim.x / cgs;
  const int lane = threadIdx.x / cgs, cg = threadIdx.x % cgs;
  const bool active = lane < lanes;
  const int rows = N * H;
  float wr[REGW ? 9 : 1][8];
  if (REGW) {
#pragma unroll
    for (int t = 0; t < (REGW ? 9 : 1); ++t)
#pragma unroll
      for (int k = 0; k < 8; ++k) wr[t][k] = s_w[t * Cout + cg * 8 + k];
  }
  float s1[8], s2[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) s1[k] = s2[k] = 0.f;
  if (active) {
    // block walks image rows; its pixel lanes walk the row (no per-pixel integer division)
    for (int row = blockIdx.x; row < rows; row += gridDim.x) {
      const int n = row / H, hq = row % H;
      for (int wq = lane; wq < W; wq += lanes) {
        const size_t pix = static_cast<size_t>(row) * W + wq;
        float acc[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) acc[k] = 0.f;
        for (int ci = 0; ci < Cin; ++ci) {
          const float* xp = x + (static_cast<size_t>(n) * Cin + ci) * H * W;
#pragma unroll
          for (int t = 0; t < 9; ++t) {
            const int hh = hq + t / 3 - 1, ww = wq + t % 3 - 1;
            const float xv = (hh >= 0 && hh < H && ww >= 0 && ww < W) ? __ldg(xp + static_cast<size_t>(hh) * W + ww) : 0.f;
            if (REGW) {
#pragma unroll
              for (int k = 0; k < 8; ++k) acc[k] = fmaf(xv, wr[REGW ? t : 0][k], acc[k]);
            } else {
              const float* wrow = s_w + (ci * 9 + t) * Cout + cg * 8;
#pragma unroll
              for (int k = 0; k < 8; ++k) acc[k] = fmaf(xv, wrow[k], acc[k]);
            }
          }
        }
        F8 o;
#pragma unroll
        for (int k = 0; k < 8; ++k) o.v[k] = acc[k];
        const uint4 packed = pack8(o);
        *reinterpret_cast<uint4*>(y + pix * ld_y + cg * 8) = packed;
        const F8 r = unpack8(packed);
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          s1[k] += r.v[k];
          s2[k] = fmaf(r.v[k], r.v[k], s2[k]);
        }
      }
    }
  }
  if (partials != nullptr) {
    float* mine = s_red + (static_cast<size_t>(lane) * cgs + cg) * 16;
    if (active) {
#pragma unroll
      for (int k = 0; k < 8; ++k) { mine[k] = s1[k]; mine[8 + k] = s2[k]; }
    }
    __syncthreads();
    for (int idx = threadIdx.x; idx < cgs * 16; idx += blockDim.x) {
      double a = 0.0;
      for (int l = 0; l < lanes; ++l) a += static_cast<double>(s_red[static_cast<size_t>(l) * cgs * 16 + idx]);
      const int cgi = idx / 16, k = idx % 16;
      partials[(static_cast<size_t>(blockIdx.x) * 2 + (k >> 3)) * Cout + cgi * 8 + (k & 7)] = a;
    }
  }
}

// Cin == 1, W % 4 == 0: a thread owns 4 consecutive pixels x 8 channels; its 72 weights and the
// 3x6 input window live in registers (288 FMAs per 18 loads and 4 stores).
__global__ void __launch_bounds__(kHeadThreads)
conv_in_fwd4_kernel(const float* __restrict__ x, const float* __restrict__ w, __nv_bfloat16* __restrict__ y,
                    int ld_y, double* partials, int N, int H, int W, int Cout) {
  pdl_trigger();
  pdl_wait();
  extern __shared__ float s_red[];  // [lanes][cgs][16]
  const int cgs = Cout / 8;
  const int lanes = blockDim.x / cgs;
  const int lane = threadIdx.x / cgs, cg = threadIdx.x % cgs;
  const bool active = lane < lanes;
  const int rows = N * H;
  float wr[9][8];
#pragma unroll
  for (int t = 0; t < 9; ++t)
#pragma unroll
    for (int k = 0; k < 8; ++k) wr[t][k] = __ldg(w + (cg * 8 + k) * 9 + t);
  float s1[8], s2[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) s1[k] = s2[k] = 0.f;
  if (active) {
    for (int row = blockIdx.x; row < rows; row += gridDim.x) {
      const int hq = row % H;
      const float* xrow = x + static_cast<size_t>(row) * W;
      for (int wq = lane * 4; wq < W; wq += lanes * 4) {
        float xv[3][6];
#pragma unroll
        for (int r = 0; r < 3; ++r) {
          const int hh = hq + r - 1;
          const bool rv = hh >= 0 && hh < H;
          const float* xp = xrow + (r - 1) * W + wq;
          xv[r][0] = (rv && wq > 0) ? __ldg(xp - 1) : 0.f;
          const float4 mid = rv ? __ldg(reinterpret_cast<const float4*>(xp)) : make_float4(0.f, 0.f, 0.f, 0.f);
          xv[r][1] = mid.x; xv[r][2] = mid.y; xv[r][3] = mid.z; xv[r][4] = mid.w;
          xv[r][5] = (rv && wq + 4 < W) ? __ldg(xp + 4) : 0.f;
        }
#pragma unroll
        for (int px = 0; px < 4; ++px) {
          float acc[8];
#pragma unroll
          for (int k = 0; k < 8; ++k) acc[k] = 0.f;
#pragma unroll
          for (int r = 0; r < 3; ++r)
#pragma unroll
            for (int s = 0; s < 3; ++s)
#pragma unroll
              for (int k = 0; k < 8; ++k) acc[k] = fmaf(xv[r][px + s], wr[r * 3 + s][k], acc[k]);
          F8 o;
#pragma unroll
          for (int k = 0; k < 8; ++k) o.v[k] = acc[k];
          const uint4 packed = pack8(o);
          *reinterpret_cast<uint4*>(y + (static_cast<size_t>(row) * W + wq + px) * ld_y + cg * 8) = packed;
          const F8 rr = unpack8(packed);
#pragma unroll
          for (int k = 0; k < 8; ++k) {
            s1[k] += rr.v[k];
            s2[k] = fmaf(rr.v[k], rr.v[k], s2[k]);
          }
        }
      }
    }
  }
  if (partials != nullptr) {
    float* mine = s_red + (static_cast<size_t>(lane) * cgs + cg) * 16;
    if (active) {
#pragma unroll
      for (int k = 0; k < 8; ++k) { mine[k] = s1[k]; mine[8 + k] = s2[k]; }
    }
    __syncthreads();
    for (int idx = threadIdx.x; idx < cgs * 16; idx += blockDim.x) {
      double a = 0.0;
      for (int l = 0; l < lanes; ++l) a += static_cast<double>(s_red[static_cast<size_t>(l) * cgs * 16 + idx]);
      const int cgi = idx / 16, k = idx % 16;
      partials[(static_cast<size_t>(blockIdx.x) * 2 + (k >> 3)) * Cout + cgi * 8 + (k & 7)] = a;
    }
  }
}

// dW[co][ci][t] = sum_p dy[p][co] * x[p + shift_t][ci]; blockIdx.y = ci; rows of [9][Cout] doubles
__global__ void __launch_bounds__(kHeadThreads)
conv_in_wgrad_kernel(const float* __restrict__ x, const __nv_bfloat16* __restrict__ dy, int ld_dy,
                     double* partials, int N, int Cin, int H, int W, int Cout) {
  pdl_trigger();
  pdl_wait();
  extern __shared__ float s_red[];  // [lanes][cgs][8]
  const int ci = blockIdx.y;
  const int cgs = Cout / 8;
  const int lanes = blockDim.x / cgs;
  const int lane = threadIdx.x / cgs, cg = threadIdx.x % cgs;
  const bool active = lane < lanes;
  const int pixels = static_cast<int>(N) * H * W;
  float acc[9][8];
#pragma unroll
  for (int t = 0; t < 9; ++t)
#pragma unroll
    for (int k = 0; k < 8; ++k) acc[t][k] = 0.f;
  if (active) {
    for (int pix = static_cast<int>(blockIdx.x) * lanes + lane; pix < pixels;
         pix += static_cast<int>(gridDim.x) * lanes) {
      const int wq = static_cast<int>(pix % W);
      const int hq = static_cast<int>((pix / W) % H);
      const int n = static_cast<int>(pix / (static_cast<int>(W) * H));
      const F8 d = load8_stream(dy + static_cast<size_t>(pix) * ld_dy + cg * 8);
      const float* xp = x + (static_cast<size_t>(n) * Cin + ci) * H * W;
#pragma unroll
      for (int t = 0; t < 9; ++t) {
        const int hh = hq + t / 3 - 1, ww = wq + t % 3 - 1;
        const float xv = (hh >= 0 && hh < H && ww >= 0 && ww < W) ? __ldg(xp + static_cast<size_t>(hh) * W + ww) : 0.f;
#pragma unroll
        for (int k = 0; k < 8; ++k) acc[t][k] = fmaf(xv, d.v[k], acc[t][k]);
      }
    }
  }
  double* row = partials + (static_cast<size_t>(blockIdx.x) * Cin + ci) * 9 * Cout;
#pragma unroll
  for (int t = 0; t < 9; ++t) {
    float* mine = s_red + (static_cast<size_t>(lane) * cgs + cg) * 8;
    if (active) {
#pragma unroll
      for (int k = 0; k < 8; ++k) mine[k] = acc[t][k];
    }
    __syncthreads();
    for (int idx = threadIdx.x; idx < cgs * 8; idx += blockDim.x) {
      double a = 0.0;
      for (int l = 0; l < lanes; ++l) a += static_cast<double>(s_red[static_cast<size_t>(l) * cgs * 8 + idx]);
      row[t * Cout + idx] = a;
    }
    __syncthreads();
  }
}

// Cin == 1, W % 4 == 0: an item is 4 consecutive pixels x 8 channels (as conv_in_fwd4): four
// 128-bit dy loads in flight (the next item's are issued before this item's 288 FMAs), the 3x6
// input window shared by the 4 pixels, no per-pixel index arithmetic.
__global__ void __launch_bounds__(kHeadThreads, 2)
conv_in_wgrad4_kernel(const float* __restrict__ x, const __nv_bfloat16* __restrict__ dy, int ld_dy,
                      double* partials, int N, int H, int W, int Cout) {
  pdl_trigger();
  pdl_wait();
  extern __shared__ float s_red[];  // [lanes][cgs][8]
  const int cgs = Cout / 8;
  const int lanes = blockDim.x / cgs;
  const int lane = threadIdx.x / cgs, cg = threadIdx.x % cgs;
  const bool active = lane < lanes;
  const unsigned wq4 = static_cast<unsigned>(W) >> 2;
  const unsigned items = static_cast<unsigned>(N) * H * wq4;
  const unsigned stride = gridDim.x * lanes;
  float acc[9][8];
#pragma unroll
  for (int t = 0; t < 9; ++t)
#pragma unroll
    for (int k = 0; k < 8; ++k) acc[t][k] = 0.f;
  if (active) {
    unsigned item = blockIdx.x * lanes + lane;
    uint4 d[4];
    auto load_dy = [&](unsigned it) {
      const __nv_bfloat16* p = dy + static_cast<size_t>(it) * 4 * ld_dy + cg * 8;
#pragma unroll
      for (int px = 0; px < 4; ++px) d[px] = ld_stream16(p + static_cast<size_t>(px) * ld_dy);
    };
    if (item < items) load_dy(item);
    for (; item < items; item += stride) {
      const unsigned row = item / wq4;
      const int wq = static_cast<int>(item - row * wq4) << 2;
      const int hq = static_cast<int>(row % static_cast<unsigned>(H));
      const float* xrow = x + static_cast<size_t>(row) * W;
      float xv[3][6];
#pragma unroll
      for (int r = 0; r < 3; ++r) {
        const int hh = hq + r - 1;
        const bool rv = hh >= 0 && hh < H;
        const float* xp = xrow + (r - 1) * W + wq;
        xv[r][0] = (rv && wq > 0) ? __ldg(xp - 1) : 0.f;
        const float4 mid = rv ? __ldg(reinterpret_cast<const float4*>(xp)) : make_float4(0.f, 0.f, 0.f, 0.f);
        xv[r][1] = mid.x; xv[r][2] = mid.y; xv[r][3] = mid.z; xv[r][4] = mid.w;
        xv[r][5] = (rv && wq + 4 < W) ? __ldg(xp + 4) : 0.f;
      }
      F8 cur[4];
#pragma unroll
      for (int px = 0; px < 4; ++px) cur[px] = unpack8(d[px]);
      if (item + stride < items) load_dy(item + stride);
#pragma unroll
      for (int px = 0; px < 4; ++px)
#pragma unroll
        for (int r = 0; r < 3; ++r)
#pragma unroll
          for (int sft = 0; sft < 3; ++sft)
#pragma unroll
            for (int k = 0; k < 8; ++k) acc[r * 3 + sft][k] = fmaf(xv[r][px + sft], cur[px].v[k], acc[r * 3 + sft][k]);
    }
  }
  double* rowp = partials + static_cast<size_t>(blockIdx.x) * 9 * Cout;
#pragma unroll
  for (int t = 0; t < 9; ++t) {
    float* mine = s_red + (static_cast<size_t>(lane) * cgs + cg) * 8;
    if (active) {
#pragma unroll
      for (int k = 0; k < 8; ++k) mine[k] = acc[t][k];
    }
    __syncthreads();
    for (int idx = threadIdx.x; idx < cgs * 8; idx += blockDim.x) {
      double a = 0.0;
      for (int l = 0; l < lanes; ++l) a += static_cast<double>(s_red[static_cast<size_t>(l) * cgs * 8 + idx]);
      rowp[t * Cout + idx] = a;
    }
    __syncthreads();
  }
}

// grad[co][ci][t] += sum_rows partials[row][ci][t][co];  blockDim = (32, 32)
__global__ void conv_in_wgrad_finalize_kernel(const double* __restrict__ partials, int rows, int Cin,
                                              int Cout, float* grad) {
  pdl_trigger();
  pdl_wait();
  __shared__ double smem[32 * 33];
  const int total = Cout * Cin * 9;
  const int i = blockIdx.x * 32 + threadIdx.x;  // index into the [ci][t][co] row layout
  double s[1];
  rows_sum<1>(partials, rows, total, i, s, smem);
  if (threadIdx.y != 0 || i >= total) return;
  const int co = i % Cout, r = i / Cout;
  grad[co * Cin * 9 + r] += static_cast<float>(s[0]);
}

// dx[n][ci][h][w] = sum_{r,s} sum_co dy[n][h-r+1][w-s+1][co] * W[co][ci][r][s]  (dy outside the image = 0)
//
// dy is read as 16-byte vectors of V channels (8 bf16 or 4 fp32).  Every element offset is 64-bit: N*H*W*ld_dy
// passes 2^31 at batch 128 of 512^2 x 64.  No pointer to a dy row outside the image is formed.
template <typename T>
struct DyVec;
template <>
struct DyVec<__nv_bfloat16> {
  static constexpr int V = 8;
  __device__ __forceinline__ static void load(const __nv_bfloat16* p, float (&v)[V]) {
    const F8 f = unpack8(__ldg(reinterpret_cast<const uint4*>(p)));
#pragma unroll
    for (int k = 0; k < V; ++k) v[k] = f.v[k];
  }
  __device__ __forceinline__ static float one(const __nv_bfloat16* p) {
    return __uint_as_float(static_cast<unsigned>(__ldg(reinterpret_cast<const unsigned short*>(p))) << 16);
  }
};
template <>
struct DyVec<float> {
  static constexpr int V = 4;
  __device__ __forceinline__ static void load(const float* p, float (&v)[V]) {
    const float4 f = __ldg(reinterpret_cast<const float4*>(p));
    v[0] = f.x; v[1] = f.y; v[2] = f.z; v[3] = f.w;
  }
  __device__ __forceinline__ static float one(const float* p) { return __ldg(p); }
};

// Cin == 1, W % 4 == 0, dy / dx 16-byte aligned (as conv_in_fwd4): a thread owns 4 consecutive pixels x one
// V-channel group of dy with its 9*V weights in registers, reads the 3x6 window of dy vectors around them and
// does 36*V FMAs into 4 per-pixel partial sums.  The Cout/V group partials of a pixel group are then folded in a
// fixed order — by xor shuffles when Cout/V is a power of two <= 32 (the group threads are adjacent lanes of one
// warp), else through shared memory — and written with one float4 store.  The block walks trips of
// (image row, chunk of lanes*4 columns) together, so the fold's barriers are reached by every thread.
template <typename T, bool SHFL>
__global__ void __launch_bounds__(kHeadThreads, 2)
conv_in_dgrad4_kernel(const T* __restrict__ dy, int ld_dy, const float* __restrict__ w, float* __restrict__ dx,
                      int N, int H, int W, int Cout) {
  pdl_trigger();
  pdl_wait();
  constexpr int V = DyVec<T>::V;
  extern __shared__ float4 s_part[];  // [lanes][cgs] (SHFL == false)
  const int cgs = Cout / V;
  const int lanes = blockDim.x / cgs;
  const int lane = threadIdx.x / cgs, cg = threadIdx.x % cgs;
  const int span = lanes * 4;
  const int chunks = (W + span - 1) / span;
  const int trips = N * H * chunks;  // host: < 2^31
  float wr[9][V];
#pragma unroll
  for (int t = 0; t < 9; ++t)
#pragma unroll
    for (int k = 0; k < V; ++k) wr[t][k] = __ldg(w + static_cast<size_t>(cg * V + k) * 9 + t);
  for (int trip = blockIdx.x; trip < trips; trip += gridDim.x) {
    const int row = trip / chunks;  // n*H + h
    const int wq = (trip - row * chunks) * span + lane * 4;
    const int hq = row % H;
    const bool active = wq < W;
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    if (active) {
#pragma unroll
      for (int r = 0; r < 3; ++r) {  // dy row hq + r - 1 meets the weight row 2 - r
        const int hh = hq + r - 1;
        if (hh < 0 || hh >= H) continue;
        const T* p = dy + (static_cast<size_t>(row + r - 1) * W + wq) * ld_dy + cg * V;
        float v[6][V];
        if (wq > 0) DyVec<T>::load(p - ld_dy, v[0]);
        else {
#pragma unroll
          for (int k = 0; k < V; ++k) v[0][k] = 0.f;
        }
#pragma unroll
        for (int c = 1; c < 5; ++c) DyVec<T>::load(p + static_cast<size_t>(c - 1) * ld_dy, v[c]);
        if (wq + 4 < W) DyVec<T>::load(p + static_cast<size_t>(4) * ld_dy, v[5]);
        else {
#pragma unroll
          for (int k = 0; k < V; ++k) v[5][k] = 0.f;
        }
        // pixel wq+px takes dy column wq+px+j-1 (window column px+j) with weight column 2-j
#pragma unroll
        for (int px = 0; px < 4; ++px)
#pragma unroll
          for (int j = 0; j < 3; ++j)
#pragma unroll
            for (int k = 0; k < V; ++k) acc[px] = fmaf(v[px + j][k], wr[(2 - r) * 3 + (2 - j)][k], acc[px]);
      }
    }
    if (SHFL) {
#pragma unroll
      for (int px = 0; px < 4; ++px)
        for (int o = cgs >> 1; o > 0; o >>= 1) acc[px] += __shfl_xor_sync(0xffffffffu, acc[px], o);
    } else {
      s_part[threadIdx.x] = make_float4(acc[0], acc[1], acc[2], acc[3]);
      __syncthreads();
      if (cg == 0 && active) {
        for (int c = 1; c < cgs; ++c) {
          const float4 q = s_part[lane * cgs + c];
          acc[0] += q.x; acc[1] += q.y; acc[2] += q.z; acc[3] += q.w;
        }
      }
      __syncthreads();
    }
    if (cg == 0 && active)
      *reinterpret_cast<float4*>(dx + static_cast<size_t>(row) * W + wq) = make_float4(acc[0], acc[1], acc[2], acc[3]);
  }
}

// Every other Cin, W or alignment: one dx element per thread (NCHW order, coalesced stores), weights in shared
// memory as [ci][tap][co], every tap bounds-checked, dy read one element at a time.
template <typename T>
__global__ void __launch_bounds__(kHeadThreads)
conv_in_dgrad_kernel(const T* __restrict__ dy, int ld_dy, const float* __restrict__ w, float* __restrict__ dx,
                     int N, int Cin, int H, int W, int Cout) {
  pdl_trigger();
  pdl_wait();
  extern __shared__ float s_w[];  // [Cin*9][Cout]
  for (int i = threadIdx.x; i < Cout * Cin * 9; i += blockDim.x) {
    const int co = i / (Cin * 9), r = i % (Cin * 9);
    s_w[r * Cout + co] = w[i];
  }
  __syncthreads();
  const long long total = static_cast<long long>(N) * Cin * H * W;
  for (long long e = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; e < total;
       e += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int wq = static_cast<int>(e % W);
    const long long q = e / W;
    const int hq = static_cast<int>(q % H);
    const long long nc = q / H;
    const int ci = static_cast<int>(nc % Cin);
    const long long n = nc / Cin;
    float acc = 0.f;
    for (int r = 0; r < 3; ++r) {
      const int hh = hq - r + 1;
      if (hh < 0 || hh >= H) continue;
      for (int s = 0; s < 3; ++s) {
        const int ww = wq - s + 1;
        if (ww < 0 || ww >= W) continue;
        const T* p = dy + ((n * H + hh) * W + ww) * static_cast<long long>(ld_dy);
        const float* wp = s_w + (ci * 9 + r * 3 + s) * Cout;
#pragma unroll 4
        for (int co = 0; co < Cout; ++co) acc = fmaf(DyVec<T>::one(p + co), wp[co], acc);
      }
    }
    dx[e] = acc;
  }
}

// Variant choice and launch, after the entry point's argument checks.  The general variant's weights must fit the
// 48 KB of dynamic shared memory that needs no opt-in (Cin * 9 * Cout <= 12288).
template <typename T>
static int conv_in_dgrad_launch(const T* dy, int ld_dy, const float* w, float* dx, int N, int Cin, int H, int W,
                                int Cout, void* stream) {
  constexpr int V = DyVec<T>::V;
  const int cgs = Cout / V;
  const long long rows = static_cast<long long>(N) * H;
  const bool aligned16 = ((reinterpret_cast<uintptr_t>(dy) | reinterpret_cast<uintptr_t>(dx)) & 15) == 0;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (Cin == 1 && W % 4 == 0 && aligned16 && cgs <= kHeadThreads) {
    const int lanes = kHeadThreads / cgs;
    const int block = lanes * cgs;
    const long long span = lanes * 4;
    const long long trips = rows * ((W + span - 1) / span);
    if (trips < (1LL << 31) && W + span < (1LL << 31)) {  // the kernel's 32-bit trip and column indices
      const bool shfl = (cgs & (cgs - 1)) == 0 && cgs <= 32;
      const size_t smem = shfl ? 0 : static_cast<size_t>(block) * sizeof(float4);
      const int grid = stream_grid(trips, 1, num_sms(), 4);
      if (shfl)
        launch(conv_in_dgrad4_kernel<T, true>, grid, block, smem, s, dy, ld_dy, w, dx, N, H, W, Cout);
      else
        launch(conv_in_dgrad4_kernel<T, false>, grid, block, smem, s, dy, ld_dy, w, dx, N, H, W, Cout);
      return static_cast<int>(cudaGetLastError());
    }
  }
  const size_t smem = static_cast<size_t>(Cin) * 9 * Cout * sizeof(float);
  if (smem > 48 * 1024) return UB2_ERR_SHAPE;
  const int grid = stream_grid(static_cast<long long>(N) * Cin * H * W, kHeadThreads, num_sms(), 8);
  launch(conv_in_dgrad_kernel<T>, grid, kHeadThreads, smem, s, dy, ld_dy, w, dx, N, Cin, H, W, Cout);
  return static_cast<int>(cudaGetLastError());
}

// ------------------------------------------------------------------------------ outc
struct HeadGeom {
  int C, cgs, tpp, slots, K;
  int pixels, HW;
};

// KMAX >= n_classes.  `tpp` threads share a pixel (8 channels each, C <= 256: one group per
// thread, its weights in registers); 4 pixels per trip keep 4 independent 128-bit loads in flight.
template <int KMAX>
__global__ void __launch_bounds__(kHeadThreads)
outc_fwd_kernel(const __nv_bfloat16* __restrict__ a, int ld_a, const float* __restrict__ w,
                const float* __restrict__ bias, float* __restrict__ logits, HeadGeom g) {
  pdl_trigger();
  pdl_wait();
  const int slot = threadIdx.x / g.tpp, j = threadIdx.x % g.tpp;
  const bool single = g.cgs <= g.tpp;
  F8 wreg[KMAX];
  float breg[KMAX];
#pragma unroll
  for (int k = 0; k < KMAX; ++k) {
    breg[k] = (bias != nullptr && k < g.K) ? __ldg(bias + k) : 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i)
      wreg[k].v[i] = (single && k < g.K && j < g.cgs) ? __ldg(w + static_cast<size_t>(k) * g.C + j * 8 + i) : 0.f;
  }
  const int stride = static_cast<int>(gridDim.x) * g.slots;
  for (int base = static_cast<int>(blockIdx.x) * g.slots; base < g.pixels; base += 4 * stride) {
    float dot[4][KMAX];
    F8 v[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int pix = base + u * stride + slot;
#pragma unroll
      for (int i = 0; i < 8; ++i) v[u].v[i] = 0.f;
      if (single && pix < g.pixels && j < g.cgs) v[u] = load8_stream(a + static_cast<size_t>(pix) * ld_a + j * 8);
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int pix = base + u * stride + slot;
      const bool pv = pix < g.pixels;
#pragma unroll
      for (int k = 0; k < KMAX; ++k) dot[u][k] = 0.f;
      if (single) {
#pragma unroll
        for (int k = 0; k < KMAX; ++k)
#pragma unroll
          for (int i = 0; i < 8; ++i) dot[u][k] = fmaf(v[u].v[i], wreg[k].v[i], dot[u][k]);
      } else if (pv) {
        for (int cg = j; cg < g.cgs; cg += g.tpp) {
          const F8 vv = load8_stream(a + static_cast<size_t>(pix) * ld_a + cg * 8);
#pragma unroll
          for (int k = 0; k < KMAX; ++k) {
            if (k < g.K) {
              const F8 wv = loadf8(w + static_cast<size_t>(k) * g.C + cg * 8);
#pragma unroll
              for (int i = 0; i < 8; ++i) dot[u][k] = fmaf(vv.v[i], wv.v[i], dot[u][k]);
            }
          }
        }
      }
#pragma unroll
      for (int k = 0; k < KMAX; ++k)
        for (int o = g.tpp >> 1; o > 0; o >>= 1) dot[u][k] += __shfl_xor_sync(0xffffffffu, dot[u][k], o);
      if (pv && j == 0) {
        const int n = pix / g.HW, r = pix % g.HW;
#pragma unroll
        for (int k = 0; k < KMAX; ++k)
          if (k < g.K) logits[(static_cast<size_t>(n) * g.K + k) * g.HW + r] = dot[u][k] + breg[k];
      }
    }
  }
}

// dA[p][c] = sum_k dl[k][p] W[k][c];  partial rows: [K][C] (dW) then [K] (db), as doubles
template <int KMAX, int G>
__global__ void __launch_bounds__(kHeadThreads)
outc_bwd_kernel(const float* __restrict__ dl, const __nv_bfloat16* __restrict__ a, int ld_a,
                const float* __restrict__ w, __nv_bfloat16* __restrict__ da, int ld_da,
                double* partials, HeadGeom g) {
  pdl_trigger();
  pdl_wait();
  extern __shared__ float s_red[];  // [256][8]
  const int slot = threadIdx.x / g.tpp, j = threadIdx.x % g.tpp;
  // G channel groups per thread (C <= 256*G), KMAX >= n_classes
  constexpr int kMaxClasses = KMAX;
  float accw[G][kMaxClasses][8];
  float accb[kMaxClasses];
#pragma unroll
  for (int gi = 0; gi < G; ++gi)
#pragma unroll
    for (int k = 0; k < kMaxClasses; ++k)
#pragma unroll
      for (int i = 0; i < 8; ++i) accw[gi][k][i] = 0.f;
#pragma unroll
  for (int k = 0; k < kMaxClasses; ++k) accb[k] = 0.f;
  // U pixels per trip (their loads are issued together); with few classes the weights stay in registers
  constexpr int U = (G == 1 && KMAX <= 2) ? 4 : ((G == 1 && KMAX <= 4) ? 2 : 1);
  constexpr bool kHoist = G * KMAX <= 4;
  F8 wreg[kHoist ? G : 1][kHoist ? KMAX : 1];
  if (kHoist) {
#pragma unroll
    for (int gi = 0; gi < G; ++gi)
#pragma unroll
      for (int k = 0; k < kMaxClasses; ++k) {
        const int cg = j + gi * g.tpp;
#pragma unroll
        for (int i = 0; i < 8; ++i)
          wreg[kHoist ? gi : 0][kHoist ? k : 0].v[i] =
              (k < g.K && cg < g.cgs) ? __ldg(w + static_cast<size_t>(k) * g.C + cg * 8 + i) : 0.f;
      }
  }
  const int stride = static_cast<int>(gridDim.x) * g.slots;
  for (int base = static_cast<int>(blockIdx.x) * g.slots; base < g.pixels; base += U * stride) {
    float d[U][kMaxClasses];
    uint4 v[U][G];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int pix = base + u * stride + slot;
      const bool pv = pix < g.pixels;
      const int n = pv ? pix / g.HW : 0, r = pv ? pix % g.HW : 0;
#pragma unroll
      for (int k = 0; k < kMaxClasses; ++k) d[u][k] = (pv && k < g.K) ? __ldg(dl + (n * g.K + k) * g.HW + r) : 0.f;
#pragma unroll
      for (int gi = 0; gi < G; ++gi) {
        const int cg = j + gi * g.tpp;
        v[u][gi] = (pv && cg < g.cgs) ? ld_stream16(a + static_cast<size_t>(pix) * ld_a + cg * 8) : make_uint4(0u, 0u, 0u, 0u);
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int pix = base + u * stride + slot;
      if (pix >= g.pixels) continue;
#pragma unroll
      for (int k = 0; k < kMaxClasses; ++k)
        if (j == 0) accb[k] += d[u][k];
#pragma unroll
      for (int gi = 0; gi < G; ++gi) {
        const int cg = j + gi * g.tpp;
        if (cg < g.cgs) {
          const F8 vv = unpack8(v[u][gi]);
          F8 o;
#pragma unroll
          for (int i = 0; i < 8; ++i) o.v[i] = 0.f;
#pragma unroll
          for (int k = 0; k < kMaxClasses; ++k) {
            if (k < g.K) {
              F8 wv;
              if (kHoist) wv = wreg[kHoist ? gi : 0][kHoist ? k : 0];
              else wv = loadf8(w + static_cast<size_t>(k) * g.C + cg * 8);
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                o.v[i] = fmaf(d[u][k], wv.v[i], o.v[i]);
                accw[gi][k][i] = fmaf(d[u][k], vv.v[i], accw[gi][k][i]);
              }
            }
          }
          if (da != nullptr) store8(da + static_cast<size_t>(pix) * ld_da + cg * 8, o);
        }
      }
    }
  }
  double* row = partials + static_cast<size_t>(blockIdx.x) * (static_cast<size_t>(g.K) * g.C + g.K);
#pragma unroll
  for (int gi = 0; gi < G; ++gi) {
#pragma unroll
    for (int k = 0; k < kMaxClasses; ++k) {
      if (k >= g.K) continue;
#pragma unroll
      for (int i = 0; i < 8; ++i) s_red[(slot * g.tpp + j) * 8 + i] = accw[gi][k][i];
      __syncthreads();
      for (int idx = threadIdx.x; idx < g.tpp * 8; idx += blockDim.x) {
        const int jj = idx >> 3, i = idx & 7;
        const int cg = jj + gi * g.tpp;
        if (cg < g.cgs) {
          double s = 0.0;
          for (int sl = 0; sl < g.slots; ++sl) s += static_cast<double>(s_red[(sl * g.tpp + jj) * 8 + i]);
          row[static_cast<size_t>(k) * g.C + cg * 8 + i] = s;
        }
      }
      __syncthreads();
    }
  }
#pragma unroll
  for (int k = 0; k < kMaxClasses; ++k) {
    if (k >= g.K) continue;
    const float ws = warp_sum(accb[k]);
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = ws;
    __syncthreads();
    if (threadIdx.x == 0) {
      double s = 0.0;
      for (int i = 0; i < (blockDim.x >> 5); ++i) s += static_cast<double>(s_red[i]);
      row[static_cast<size_t>(g.K) * g.C + k] = s;
    }
    __syncthreads();
  }
}

// blockDim = (32, 32)
__global__ void outc_bwd_finalize_kernel(const double* __restrict__ partials, int rows, int K, int C,
                                         float* dw, float* db) {
  pdl_trigger();
  pdl_wait();
  __shared__ double smem[32 * 33];
  const int total = K * C + K;
  const int i = blockIdx.x * 32 + threadIdx.x;
  double s[1];
  rows_sum<1>(partials, rows, total, i, s, smem);
  if (threadIdx.y != 0 || i >= total) return;
  if (i < K * C) {
    if (dw) dw[i] += static_cast<float>(s[0]);
  } else if (db) {
    db[i - K * C] += static_cast<float>(s[0]);
  }
}

static int head_geom(HeadGeom* g, int N, int H, int W, int C, int K) {
  if (C <= 0 || C % 8 != 0 || K < 1 || K > kMaxClasses || N <= 0 || H <= 0 || W <= 0) return UB2_ERR_SHAPE;
  if (static_cast<double>(N) * H * W * K >= 2.0e9) return UB2_ERR_SHAPE;  // 32-bit pixel indices
  g->C = C; g->cgs = C / 8; g->K = K;
  int t = 1;
  while (t < g->cgs && t < 32) t *= 2;
  g->tpp = t;
  g->slots = kHeadThreads / t;
  g->HW = static_cast<int>(H) * W;
  g->pixels = g->HW * N;
  return 0;
}

}  // namespace ub2

using namespace ub2;

extern "C" {

int ub2_conv_in_rows(int N, int H, int W, int Cout) {
  if (Cout <= 0 || Cout % 8 != 0 || Cout / 8 > kHeadThreads || N <= 0 || H <= 0 || W <= 0) return UB2_ERR_SHAPE;
  const int lanes = kHeadThreads / (Cout / 8);
  return stream_grid(static_cast<int>(N) * H * W, lanes, num_sms(), 4);
}

int ub2_conv_in_fwd(const float* x, const float* w, void* y, int ld_y, double* partials, int rows, int N,
                    int Cin, int H, int W, int Cout, void* stream) {
  if (Cout % 8 != 0 || Cout / 8 > kHeadThreads || Cin < 1 || Cin > kMaxCin) return UB2_ERR_SHAPE;
  if (static_cast<double>(N) * H * W * Cin >= 2.0e9) return UB2_ERR_SHAPE;  // 32-bit pixel indices
  const int cgs = Cout / 8;
  const int block = cgs * (kHeadThreads / cgs);
  const int lanes = block / cgs;
  const int grid = stream_grid(static_cast<int>(N) * H * W, lanes, num_sms(), 4);
  if (partials != nullptr && grid != rows) return UB2_ERR_WORKSPACE;
  const size_t smem = (static_cast<size_t>(Cin) * 9 * Cout + static_cast<size_t>(lanes) * cgs * 16) * sizeof(float);
  if (Cin == 1 && W % 4 == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0)
    launch(conv_in_fwd4_kernel, grid, block, static_cast<size_t>(lanes) * cgs * 16 * sizeof(float), static_cast<cudaStream_t>(stream), x, w, static_cast<__nv_bfloat16*>(y), ld_y, partials, N, H, W, Cout);
  else if (Cin == 1)
    launch(conv_in_fwd_kernel<true>, grid, block, smem, static_cast<cudaStream_t>(stream), x, w, static_cast<__nv_bfloat16*>(y), ld_y, partials, N, Cin, H, W, Cout);
  else
    launch(conv_in_fwd_kernel<false>, grid, block, smem, static_cast<cudaStream_t>(stream), x, w, static_cast<__nv_bfloat16*>(y), ld_y, partials, N, Cin, H, W, Cout);
  return static_cast<int>(cudaGetLastError());
}

int ub2_conv_in_wgrad(const float* x, const void* dy, int ld_dy, double* partials, int rows, float* grad,
                      int N, int Cin, int H, int W, int Cout, void* stream) {
  if (Cout % 8 != 0 || Cout / 8 > kHeadThreads || Cin < 1 || Cin > kMaxCin) return UB2_ERR_SHAPE;
  if (static_cast<double>(N) * H * W * Cin >= 2.0e9) return UB2_ERR_SHAPE;  // 32-bit pixel indices
  const int cgs = Cout / 8;
  const int block = cgs * (kHeadThreads / cgs);
  const int lanes = block / cgs;
  const int grid = stream_grid(static_cast<int>(N) * H * W, lanes, num_sms(), 4);
  if (grid != rows) return UB2_ERR_WORKSPACE;
  const size_t smem = static_cast<size_t>(lanes) * cgs * 8 * sizeof(float);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (Cin == 1 && W % 4 == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0 &&
      static_cast<double>(N) * H * W < 4.0e9)
    launch(conv_in_wgrad4_kernel, grid, block, smem, s, x, static_cast<const __nv_bfloat16*>(dy), ld_dy, partials, N, H, W, Cout);
  else
    launch(conv_in_wgrad_kernel, dim3(grid, Cin), block, smem, s, x, static_cast<const __nv_bfloat16*>(dy), ld_dy, partials, N, Cin, H, W, Cout);
  const int total = Cout * Cin * 9;
  launch(conv_in_wgrad_finalize_kernel, (total + 31) / 32, dim3(32, 32), 0, s, partials, grid, Cin, Cout, grad);
  return static_cast<int>(cudaGetLastError());
}

int ub2_conv_in_dgrad(const void* dy, int ld_dy, const float* w, float* dx, int N, int Cin, int H, int W, int Cout,
                      void* stream) {
  if (dy == nullptr || w == nullptr || dx == nullptr || N <= 0 || H <= 0 || W <= 0) return UB2_ERR_SHAPE;
  if (Cout <= 0 || Cout % 8 != 0 || Cout / 8 > kHeadThreads || Cin < 1 || Cin > kMaxCin || ld_dy < Cout) return UB2_ERR_SHAPE;
  if (static_cast<double>(N) * H * W * Cin >= 2.0e9) return UB2_ERR_SHAPE;  // the forward's limit
  if (ld_dy % 8 != 0 || (reinterpret_cast<uintptr_t>(dy) & 1) || (reinterpret_cast<uintptr_t>(w) & 3) ||
      (reinterpret_cast<uintptr_t>(dx) & 3))
    return UB2_ERR_ALIGN;
  return conv_in_dgrad_launch(static_cast<const __nv_bfloat16*>(dy), ld_dy, w, dx, N, Cin, H, W, Cout, stream);
}

int ub2_f32_conv_in_dgrad(const float* dy, int ld_dy, const float* w, float* dx, int N, int Cin, int H, int W, int Cout,
                          void* stream) {
  if (dy == nullptr || w == nullptr || dx == nullptr || N <= 0 || H <= 0 || W <= 0) return UB2_ERR_SHAPE;
  if (Cout <= 0 || Cout % 4 != 0 || Cin < 1 || ld_dy < Cout) return UB2_ERR_SHAPE;
  if (ld_dy % 4 != 0 || ((reinterpret_cast<uintptr_t>(dy) | reinterpret_cast<uintptr_t>(w) | reinterpret_cast<uintptr_t>(dx)) & 3))
    return UB2_ERR_ALIGN;
  return conv_in_dgrad_launch(dy, ld_dy, w, dx, N, Cin, H, W, Cout, stream);
}

int ub2_outc_rows(int N, int H, int W, int C) {
  HeadGeom g;
  int rc = head_geom(&g, N, H, W, C, 1);
  if (rc) return rc;
  return stream_grid(g.pixels, g.slots, num_sms(), 4);
}

int ub2_outc_fwd(const void* a, int ld_a, const float* w, const float* bias, float* logits, int N, int H,
                 int W, int C, int K, void* stream) {
  HeadGeom g;
  int rc = head_geom(&g, N, H, W, C, K);
  if (rc) return rc;
  const int grid = stream_grid((g.pixels + 3) / 4, g.slots, num_sms(), 8);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const __nv_bfloat16* ap = static_cast<const __nv_bfloat16*>(a);
  if (K <= 2) launch(outc_fwd_kernel<2>, grid, kHeadThreads, 0, s, ap, ld_a, w, bias, logits, g);
  else if (K <= 4) launch(outc_fwd_kernel<4>, grid, kHeadThreads, 0, s, ap, ld_a, w, bias, logits, g);
  else launch(outc_fwd_kernel<8>, grid, kHeadThreads, 0, s, ap, ld_a, w, bias, logits, g);
  return static_cast<int>(cudaGetLastError());
}

int ub2_outc_bwd(const float* dlogits, const void* a, int ld_a, const float* w, void* da, int ld_da,
                 double* partials, int rows, float* dw, float* db, int N, int H, int W, int C, int K,
                 void* stream) {
  HeadGeom g;
  int rc = head_geom(&g, N, H, W, C, K);
  if (rc) return rc;
  if (g.cgs > 2 * g.tpp) return UB2_ERR_SHAPE;
  const int grid = stream_grid(g.pixels, g.slots, num_sms(), 4);
  if (grid != rows) return UB2_ERR_WORKSPACE;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const size_t smem = kHeadThreads * 8 * sizeof(float);
  const __nv_bfloat16* ap = static_cast<const __nv_bfloat16*>(a);
  __nv_bfloat16* dap = static_cast<__nv_bfloat16*>(da);
  const bool two = g.cgs > g.tpp;
#define UB2_OUTC_BWD(KM)                                                                              \
  do {                                                                                                \
    if (two) launch(outc_bwd_kernel<KM, 2>, grid, kHeadThreads, smem, s, dlogits, ap, ld_a, w, dap, ld_da, partials, g); \
    else launch(outc_bwd_kernel<KM, 1>, grid, kHeadThreads, smem, s, dlogits, ap, ld_a, w, dap, ld_da, partials, g);    \
  } while (0)
  if (K <= 2) UB2_OUTC_BWD(2);
  else if (K <= 4) UB2_OUTC_BWD(4);
  else UB2_OUTC_BWD(8);
#undef UB2_OUTC_BWD
  const int total = K * C + K;
  launch(outc_bwd_finalize_kernel, (total + 31) / 32, dim3(32, 32), 0, s, partials, grid, K, C, dw, db);
  return static_cast<int>(cudaGetLastError());
}

}  // extern "C"
