// Bandwidth-bound BatchNorm / ReLU / MaxPool passes over NHWC bf16 activations.
//
// Train-mode forward of one conv->BN->ReLU stage (layers.py:32-34) is
//   conv kernel (raw bf16 output + per-CTA sum / sum-sq rows)
//   -> bn_finalize (batch mean / biased var, running-stat update, scale/shift)
//   -> bn_act     (a = relu(scale*y + shift); optionally the 2x2 max-pooled copy
//                  that Down (layers.py:56) feeds to the next stage).
// Backward: bn_bwd<false> reduces sum(dz), sum(dz*xhat); bn_bwd_finalize turns them
// into dgamma/dbeta (+ the three per-channel coefficients); bn_bwd<true> writes
// dy = gamma*invstd*(dz - mean(dz) - xhat*mean(dz*xhat)).  The gradient arriving through
// the max-pool is routed to the window's first maximum, recomputed from y.
//
// Threads walk 2x2 pixel windows x 8-channel (128-bit) vectors; a thread's channel
// group is fixed so per-channel coefficients live in registers.
#include "launch.cuh"
#include "../../include/unetb200.h"
#include "conv.h"
#include "vec.cuh"

namespace ub2 {

static constexpr int kBnThreads = 256;

// ------------------------------------------------------------------------------ finalize
// blockDim = (8, 128): see rows_sum_wide in vec.cuh
__global__ void bn_finalize_kernel(const double* __restrict__ partials, int rows, int C, double count,
                                   const float* __restrict__ gamma, const float* __restrict__ beta,
                                   float* running_mean, float* running_var, long long* nbt,
                                   float momentum, float eps, float* scale, float* shift, float* mean,
                                   float* invstd) {
  pdl_trigger();
  pdl_wait();
  __shared__ double smem[2 * 128 * 9];
  const int c = blockIdx.x * 8 + threadIdx.x;
  if (blockIdx.x == 0 && threadIdx.x == 0 && threadIdx.y == 0 && nbt != nullptr) *nbt += 1;
  double s[2];
  rows_sum_wide<2>(partials, rows, C, c, s, smem);
  if (threadIdx.y != 0 || c >= C) return;
  const double m = s[0] / count;
  double var = s[1] / count - m * m;
  if (var < 0.0) var = 0.0;
  const double inv = 1.0 / sqrt(var + static_cast<double>(eps));
  const float g = gamma ? gamma[c] : 1.f;
  const float b = beta ? beta[c] : 0.f;
  scale[c] = static_cast<float>(g * inv);
  shift[c] = static_cast<float>(b - m * g * inv);
  mean[c] = static_cast<float>(m);
  invstd[c] = static_cast<float>(inv);
  if (running_mean != nullptr) {
    const double unbiased = count > 1.0 ? var * count / (count - 1.0) : var;
    running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * static_cast<float>(m);
    running_var[c] = (1.f - momentum) * running_var[c] + momentum * static_cast<float>(unbiased);
  }
}

__global__ void bn_eval_coeffs_kernel(const float* __restrict__ gamma, const float* __restrict__ beta,
                                      const float* __restrict__ rm, const float* __restrict__ rv,
                                      float eps, int C, float* scale, float* shift) {
  pdl_trigger();
  pdl_wait();
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const float inv = 1.f / sqrtf(rv[c] + eps);
  const float g = gamma ? gamma[c] : 1.f;
  scale[c] = g * inv;
  shift[c] = (beta ? beta[c] : 0.f) - rm[c] * g * inv;
}

// ------------------------------------------------------------------------------ window walk
struct WinGeom {
  int N, H, W, C, cgs, Hc, Wc;
  int windows;
};
// Device loops index pixels with 32-bit integers.
static bool fits32(int N, int H, int W, int C) {
  return static_cast<double>(N) * H * W * (C > 8 ? C / 8 : 1) < 2.0e9;
}
static WinGeom make_geom(int N, int H, int W, int C) {
  WinGeom g;
  g.N = N; g.H = H; g.W = W; g.C = C; g.cgs = C / 8;
  g.Hc = (H + 1) / 2; g.Wc = (W + 1) / 2;
  g.windows = static_cast<int>(N) * g.Hc * g.Wc;
  return g;
}

// ------------------------------------------------------------------------------ forward apply
// fp32 pair -> packed bf16x2 with the ReLU folded into the conversion (one instruction instead of two max + one cvt)
__device__ __forceinline__ uint32_t pack2_relu(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}

// POOL: also emit the 2x2 max-pooled copy (+ window index); RELU: compile-time so that the conversion carries it.
// The decoder's ten launches per step have no pool: its compare / select work is not even compiled into theirs.
template <bool POOL, bool RELU>
__global__ void __launch_bounds__(kBnThreads, 4)
bn_act_kernel(const __nv_bfloat16* __restrict__ y, int ld_y, const float* __restrict__ scale,
              const float* __restrict__ shift, __nv_bfloat16* a, int ld_a, __nv_bfloat16* pooled,
              int ld_p, unsigned char* pidx, WinGeom g) {
  pdl_trigger();
  pdl_wait();
  const int lanes = blockDim.x / g.cgs;
  const int lane = threadIdx.x / g.cgs;
  const int cg = threadIdx.x % g.cgs;
  if (lane >= lanes) return;
  F8 sc, sh;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    sc.v[i] = scale ? scale[cg * 8 + i] : 1.f;
    sh.v[i] = shift ? shift[cg * 8 + i] : 0.f;
  }
  const int Hp = g.H / 2, Wp = g.W / 2;
  for (int wi = static_cast<int>(blockIdx.x) * lanes + lane; wi < g.windows;
       wi += static_cast<int>(gridDim.x) * lanes) {
    const int wc = static_cast<int>(wi % g.Wc);
    const int hc = static_cast<int>((wi / g.Wc) % g.Hc);
    const int n = static_cast<int>(wi / (static_cast<int>(g.Wc) * g.Hc));
    F8 mx;
    unsigned arg[8];  // window position of the first maximum, per channel
#pragma unroll
    for (int i = 0; i < 8; ++i) arg[i] = 0u;
#pragma unroll
    for (int i = 0; i < 8; ++i) mx.v[i] = -INFINITY;
    // the window's four 128-bit loads are in flight together (kept packed: 16 registers); with a
    // load -> store chain per pixel the kernel is latency bound at ~4.4 TB/s
    uint4 raw[4];
#pragma unroll
    for (int d = 0; d < 4; ++d) {
      const int h = hc * 2 + (d >> 1), w = wc * 2 + (d & 1);
      raw[d] = make_uint4(0u, 0u, 0u, 0u);
      if (h < g.H && w < g.W) {
        const size_t pix = (static_cast<size_t>(n) * g.H + h) * g.W + w;
        raw[d] = ld_stream16(y + pix * ld_y + cg * 8);
      }
    }
#pragma unroll
    for (int d = 0; d < 4; ++d) {
      const int h = hc * 2 + (d >> 1), w = wc * 2 + (d & 1);
      if (h < g.H && w < g.W) {
        const size_t pix = (static_cast<size_t>(n) * g.H + h) * g.W + w;
        F8 v = unpack8(raw[d]);
        uint4 packed;
#pragma unroll
        for (int i = 0; i < 8; ++i) v.v[i] = fmaf(v.v[i], sc.v[i], sh.v[i]);
        if (RELU) {
          packed.x = pack2_relu(v.v[0], v.v[1]);
          packed.y = pack2_relu(v.v[2], v.v[3]);
          packed.z = pack2_relu(v.v[4], v.v[5]);
          packed.w = pack2_relu(v.v[6], v.v[7]);
        } else {
          packed = pack8(v);
        }
        if (a != nullptr) *reinterpret_cast<uint4*>(a + pix * ld_a + cg * 8) = packed;
        if (POOL) {
          const F8 r = unpack8(packed);
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            if (r.v[i] > mx.v[i]) {  // strict: the first maximum wins, as in ATen's max_pool2d
              mx.v[i] = r.v[i];
              arg[i] = d;
            }
          }
        }
      }
    }
    if (POOL && pooled != nullptr && hc < Hp && wc < Wp) {
      const size_t pp = (static_cast<size_t>(n) * Hp + hc) * Wp + wc;
      store8(pooled + pp * ld_p + cg * 8, mx);
      if (pidx != nullptr) {
        uint2 packed;  // one byte per channel
        packed.x = arg[0] | (arg[1] << 8) | (arg[2] << 16) | (arg[3] << 24);
        packed.y = arg[4] | (arg[5] << 8) | (arg[6] << 16) | (arg[7] << 24);
        *reinterpret_cast<uint2*>(pidx + pp * g.C + cg * 8) = packed;
      }
    }
  }
}

// ------------------------------------------------------------------------------ backward
// g = (dA + dP routed through the 2x2 max-pool) * [scale*y + shift > 0]
//   reduce : s1 = sum g, s2 = sum g*y          (raw y: the finalize turns s2 into sum g*xhat)
//   apply  : dy = A*g + B*y + C                (coef rows A, B, C from the finalize)
struct BwdArgs {
  const __nv_bfloat16* dA; int ld_da;
  const __nv_bfloat16* dP; int ld_dp;
  const unsigned char* pidx;
  const __nv_bfloat16* y; int ld_y;
  const float* scale; const float* shift; const float* coef;
  __nv_bfloat16* dY; int ld_dy;
  double* partials;
  int relu;
};

template <bool POOL, bool APPLY>
__global__ void __launch_bounds__(kBnThreads, 2)
bn_bwd_kernel(BwdArgs a, WinGeom g) {
  pdl_trigger();
  pdl_wait();
  extern __shared__ float s_red[];
  const int lanes = blockDim.x / g.cgs;
  const int lane = threadIdx.x / g.cgs;
  const int cg = threadIdx.x % g.cgs;
  const bool active = lane < lanes;
  F8 sc, sh, cA, cB, cC, s1, s2;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int c = cg * 8 + i;
    sc.v[i] = a.scale[c]; sh.v[i] = a.shift[c];
    if (APPLY) { cA.v[i] = a.coef[c]; cB.v[i] = a.coef[g.C + c]; cC.v[i] = a.coef[2 * g.C + c]; }
    s1.v[i] = s2.v[i] = 0.f;
  }
  auto one_pixel = [&](size_t pix, const F8& yv, F8 gv) {
    F8 out;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      float gs = gv.v[i];
      if (a.relu && !(fmaf(yv.v[i], sc.v[i], sh.v[i]) > 0.f)) gs = 0.f;
      if (APPLY) {
        out.v[i] = fmaf(cA.v[i], gs, fmaf(cB.v[i], yv.v[i], cC.v[i]));
      } else {
        s1.v[i] += gs;
        s2.v[i] = fmaf(gs, yv.v[i], s2.v[i]);
      }
    }
    if (APPLY) store8(a.dY + pix * a.ld_dy + cg * 8, out);
  };
  if (active) {
    if (!POOL) {
      const int pixels = static_cast<int>(g.N) * g.H * g.W;
      const int stride = static_cast<int>(gridDim.x) * lanes;
      int pix = static_cast<int>(blockIdx.x) * lanes + lane;
      // 4 pixels per trip: 8 independent 128-bit loads in flight per thread
      for (; pix + 3 * stride < pixels; pix += 4 * stride) {
        F8 yv[4], gv[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const size_t p = static_cast<size_t>(pix + u * stride);
          yv[u] = load8_stream(a.y + p * a.ld_y + cg * 8);
          gv[u] = load8_stream(a.dA + p * a.ld_da + cg * 8);
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) one_pixel(static_cast<size_t>(pix + u * stride), yv[u], gv[u]);
      }
      for (; pix < pixels; pix += stride) {
        const size_t p = static_cast<size_t>(pix);
        one_pixel(p, load8_stream(a.y + p * a.ld_y + cg * 8), load8_stream(a.dA + p * a.ld_da + cg * 8));
      }
    } else {
      const int Hp = g.H / 2, Wp = g.W / 2;
      for (int wi = static_cast<int>(blockIdx.x) * lanes + lane; wi < g.windows;
           wi += static_cast<int>(gridDim.x) * lanes) {
        const int wc = static_cast<int>(wi % g.Wc);
        const int hc = static_cast<int>((wi / g.Wc) % g.Hc);
        const int n = static_cast<int>(wi / (static_cast<int>(g.Wc) * g.Hc));
        const size_t pix0 = (static_cast<size_t>(n) * g.H + hc * 2) * g.W + wc * 2;
        if (hc < Hp && wc < Wp) {
          // complete window (the common case): all ten 128-bit loads are issued up front
          const size_t pp = (static_cast<size_t>(n) * Hp + hc) * Wp + wc;
          const size_t px[4] = {pix0, pix0 + 1, pix0 + g.W, pix0 + g.W + 1};
          F8 yv[4], gv[4];
#pragma unroll
          for (int d = 0; d < 4; ++d) yv[d] = load8_stream(a.y + px[d] * a.ld_y + cg * 8);
          const F8 gp = load8_stream(a.dP + pp * a.ld_dp + cg * 8);
          const uint2 amax = __ldg(reinterpret_cast<const uint2*>(a.pidx + pp * g.C + cg * 8));
          if (a.dA != nullptr) {
#pragma unroll
            for (int d = 0; d < 4; ++d) gv[d] = load8_stream(a.dA + px[d] * a.ld_da + cg * 8);
          } else {
#pragma unroll
            for (int d = 0; d < 4; ++d)
#pragma unroll
              for (int i = 0; i < 8; ++i) gv[d].v[i] = 0.f;
          }
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const unsigned pos = ((i < 4 ? amax.x : amax.y) >> (8 * (i & 3))) & 3u;
#pragma unroll
            for (int d = 0; d < 4; ++d) gv[d].v[i] += (pos == static_cast<unsigned>(d)) ? gp.v[i] : 0.f;
          }
#pragma unroll
          for (int d = 0; d < 4; ++d) one_pixel(px[d], yv[d], gv[d]);
        } else {
          // window cut by an odd image edge: its pixels are not pooled (MaxPool2d floors)
#pragma unroll
          for (int d = 0; d < 4; ++d) {
            const int h = hc * 2 + (d >> 1), w = wc * 2 + (d & 1);
            if (h >= g.H || w >= g.W) continue;
            const size_t pix = (static_cast<size_t>(n) * g.H + h) * g.W + w;
            F8 gv;
            if (a.dA != nullptr) {
              gv = load8_stream(a.dA + pix * a.ld_da + cg * 8);
            } else {
#pragma unroll
              for (int i = 0; i < 8; ++i) gv.v[i] = 0.f;
            }
            one_pixel(pix, load8_stream(a.y + pix * a.ld_y + cg * 8), gv);
          }
        }
      }
    }
  }
  if (!APPLY) {
    // block reduction over pixel lanes: s_red[lane][cg][16]
    float* mine = s_red + (static_cast<size_t>(lane) * g.cgs + cg) * 16;
    if (active) {
#pragma unroll
      for (int i = 0; i < 8; ++i) { mine[i] = s1.v[i]; mine[8 + i] = s2.v[i]; }
    }
    __syncthreads();
    for (int idx = threadIdx.x; idx < g.cgs * 16; idx += blockDim.x) {
      double acc = 0.0;
      for (int l = 0; l < lanes; ++l) acc += static_cast<double>(s_red[static_cast<size_t>(l) * g.cgs * 16 + idx]);
      const int cgi = idx / 16, k = idx % 16;
      const int c = cgi * 8 + (k & 7);
      a.partials[(static_cast<size_t>(blockIdx.x) * 2 + (k >> 3)) * g.C + c] = acc;
    }
  }
}

// s1 = sum g, s2 = sum g*y  ->  dbeta = s1, dgamma = invstd*(s2 - mean*s1) (accumulated into the
// fp32 .grad tensors) and the apply coefficients: dy = A*g + B*y + C with
//   A = gamma*invstd, B = -A*invstd*dgamma/M, C = -A*dbeta/M - B*mean     (B = C = 0 when frozen)
__global__ void bn_bwd_finalize_kernel(const double* __restrict__ partials, int rows, int C,
                                       double count, const float* __restrict__ gamma,
                                       const float* __restrict__ mean, const float* __restrict__ invstd,
                                       int frozen, float* dgamma, float* dbeta, float* coef) {
  pdl_trigger();
  pdl_wait();
  __shared__ double smem[2 * 128 * 9];
  const int c = blockIdx.x * 8 + threadIdx.x;
  double s[2];
  rows_sum_wide<2>(partials, rows, C, c, s, smem);
  if (threadIdx.y != 0 || c >= C) return;
  const double mu = mean[c], is = invstd[c];
  const double db = s[0];
  const double dg = is * (s[1] - mu * s[0]);
  if (dbeta) dbeta[c] += static_cast<float>(db);
  if (dgamma) dgamma[c] += static_cast<float>(dg);
  const double g = gamma ? gamma[c] : 1.0;
  const double A = g * is;
  const double B = frozen ? 0.0 : -A * is * dg / count;
  const double Cc = frozen ? 0.0 : -A * db / count - B * mu;
  coef[c] = static_cast<float>(A);
  coef[C + c] = static_cast<float>(B);
  coef[2 * C + c] = static_cast<float>(Cc);
}

static int bn_block(int cgs) { return cgs * (kBnThreads / cgs); }
static bool al16(const void* p) { return aligned_to(p, 16); }

}  // namespace ub2

using namespace ub2;

extern "C" {

int ub2_bn_finalize(const double* partials, int rows, int C, double count, const float* gamma,
                    const float* beta, float* running_mean, float* running_var, long long* nbt,
                    float momentum, float eps, float* scale, float* shift, float* mean, float* invstd,
                    void* stream) {
  if (C <= 0 || rows <= 0) return UB2_ERR_SHAPE;
  launch(bn_finalize_kernel, (C + 7) / 8, dim3(8, 128), 0, static_cast<cudaStream_t>(stream), partials, rows, C, count, gamma, beta, running_mean, running_var, nbt, momentum, eps, scale, shift, mean, invstd);
  return static_cast<int>(cudaGetLastError());
}

int ub2_bn_eval_coeffs(const float* gamma, const float* beta, const float* running_mean,
                       const float* running_var, float eps, int C, float* scale, float* shift,
                       void* stream) {
  if (C <= 0 || running_mean == nullptr || running_var == nullptr || scale == nullptr || shift == nullptr)
    return UB2_ERR_SHAPE;
  launch(bn_eval_coeffs_kernel, (C + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream), gamma, beta, running_mean, running_var, eps, C, scale, shift);
  return static_cast<int>(cudaGetLastError());
}

int ub2_bn_act(const void* y, int ld_y, const float* scale, const float* shift, void* a, int ld_a,
               void* pooled, int ld_p, unsigned char* pidx, int N, int H, int W, int C, int relu,
               void* stream) {
  if (C <= 0 || C % 8 != 0 || C / 8 > kBnThreads || N <= 0 || H <= 0 || W <= 0 || !fits32(N, H, W, C))
    return UB2_ERR_SHAPE;
  if (y == nullptr || ld_y < C || (a && ld_a < C) || (pooled && ld_p < C)) return UB2_ERR_SHAPE;
  if (ld_y % 8 || (a && ld_a % 8) || (pooled && ld_p % 8)) return UB2_ERR_ALIGN;
  if (!al16(y) || !al16(a) || !al16(pooled) || !aligned_to(pidx, 8)) return UB2_ERR_ALIGN;
  WinGeom g = make_geom(N, H, W, C);
  const int block = bn_block(g.cgs);
  const int lanes = block / g.cgs;
  const int grid = stream_grid(g.windows, lanes, num_sms(), 8);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const __nv_bfloat16* yb = static_cast<const __nv_bfloat16*>(y);
  __nv_bfloat16* ab = static_cast<__nv_bfloat16*>(a);
  __nv_bfloat16* pb = static_cast<__nv_bfloat16*>(pooled);
  if (pooled != nullptr) {
    if (relu) launch(bn_act_kernel<true, true>, grid, block, 0, s, yb, ld_y, scale, shift, ab, ld_a, pb, ld_p, pidx, g);
    else launch(bn_act_kernel<true, false>, grid, block, 0, s, yb, ld_y, scale, shift, ab, ld_a, pb, ld_p, pidx, g);
  } else {
    if (relu) launch(bn_act_kernel<false, true>, grid, block, 0, s, yb, ld_y, scale, shift, ab, ld_a, pb, ld_p, pidx, g);
    else launch(bn_act_kernel<false, false>, grid, block, 0, s, yb, ld_y, scale, shift, ab, ld_a, pb, ld_p, pidx, g);
  }
  return static_cast<int>(cudaGetLastError());
}

// Arguments shared by the reduce and apply passes: dA and dP optional (not both; dP needs pidx), every other
// pointer required, channel strides >= C and multiples of 8, 128-bit-accessed pointers 16-byte aligned.
static int bwd_check(const void* dA, int ld_da, const void* dP, int ld_dp, const unsigned char* pidx, const void* y,
                     int ld_y, const float* scale, const float* shift, int N, int H, int W, int C) {
  if (C <= 0 || C % 8 != 0 || C / 8 > kBnThreads || N <= 0 || H <= 0 || W <= 0 || !fits32(N, H, W, C))
    return UB2_ERR_SHAPE;
  if ((dA == nullptr && dP == nullptr) || (dP != nullptr && pidx == nullptr)) return UB2_ERR_SHAPE;
  if (y == nullptr || scale == nullptr || shift == nullptr) return UB2_ERR_SHAPE;
  if (ld_y < C || (dA && ld_da < C) || (dP && ld_dp < C)) return UB2_ERR_SHAPE;
  if (ld_y % 8 || (dA && ld_da % 8) || (dP && ld_dp % 8)) return UB2_ERR_ALIGN;
  if (!al16(y) || !al16(dA) || !al16(dP) || !aligned_to(pidx, 8)) return UB2_ERR_ALIGN;
  return 0;
}

static int bwd_items(const WinGeom& g, bool pool) {
  return pool ? g.windows : static_cast<int>(g.N) * g.H * g.W;
}

int ub2_bn_bwd_rows(int N, int H, int W, int C, int pool) {
  if (C <= 0 || C % 8 != 0 || C / 8 > kBnThreads || N <= 0 || H <= 0 || W <= 0) return UB2_ERR_SHAPE;
  WinGeom g = make_geom(N, H, W, C);
  const int lanes = bn_block(g.cgs) / g.cgs;
  return stream_grid((bwd_items(g, pool != 0) + 3) / 4, lanes, num_sms(), 2);
}

int ub2_bn_bwd_reduce(const void* dA, int ld_da, const void* dP, int ld_dp, const unsigned char* pidx,
                      const void* y, int ld_y, const float* scale, const float* shift, double* partials,
                      int rows, int N, int H, int W, int C, int relu, void* stream) {
  const int rc = bwd_check(dA, ld_da, dP, ld_dp, pidx, y, ld_y, scale, shift, N, H, W, C);
  if (rc) return rc;
  if (partials == nullptr) return UB2_ERR_SHAPE;
  if (!aligned_to(partials, 8)) return UB2_ERR_ALIGN;
  WinGeom g = make_geom(N, H, W, C);
  const bool pool = dP != nullptr;
  const int block = bn_block(g.cgs);
  const int lanes = block / g.cgs;
  const int grid = stream_grid((bwd_items(g, pool) + 3) / 4, lanes, num_sms(), 2);
  if (grid != rows) return UB2_ERR_WORKSPACE;
  const size_t smem = static_cast<size_t>(lanes) * g.cgs * 16 * sizeof(float);
  BwdArgs a{static_cast<const __nv_bfloat16*>(dA), ld_da, static_cast<const __nv_bfloat16*>(dP), ld_dp, pidx,
            static_cast<const __nv_bfloat16*>(y), ld_y, scale, shift, nullptr, nullptr, 0, partials, relu};
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (pool) launch_co(bn_bwd_kernel<true, false>, grid, block, smem, s, a, g);
  else launch_co(bn_bwd_kernel<false, false>, grid, block, smem, s, a, g);
  return static_cast<int>(cudaGetLastError());
}

int ub2_bn_bwd_finalize(const double* partials, int rows, int C, double count, const float* gamma,
                        const float* mean, const float* invstd, int frozen, float* dgamma, float* dbeta,
                        float* coef, void* stream) {
  if (C <= 0 || rows <= 0) return UB2_ERR_SHAPE;
  launch_co(bn_bwd_finalize_kernel, (C + 7) / 8, dim3(8, 128), 0, static_cast<cudaStream_t>(stream), partials, rows, C, count, gamma, mean, invstd, frozen, dgamma, dbeta, coef);
  return static_cast<int>(cudaGetLastError());
}

int ub2_bn_bwd_apply(const void* dA, int ld_da, const void* dP, int ld_dp, const unsigned char* pidx,
                     const void* y, int ld_y, const float* scale, const float* shift, const float* coef,
                     void* dY, int ld_dy, int N, int H, int W, int C, int relu, void* stream) {
  const int rc = bwd_check(dA, ld_da, dP, ld_dp, pidx, y, ld_y, scale, shift, N, H, W, C);
  if (rc) return rc;
  if (coef == nullptr || dY == nullptr || ld_dy < C) return UB2_ERR_SHAPE;
  if (ld_dy % 8 || !al16(dY)) return UB2_ERR_ALIGN;
  WinGeom g = make_geom(N, H, W, C);
  const bool pool = dP != nullptr;
  const int block = bn_block(g.cgs);
  const int lanes = block / g.cgs;
  const int grid = stream_grid((bwd_items(g, pool) + 3) / 4, lanes, num_sms(), 4);
  BwdArgs a{static_cast<const __nv_bfloat16*>(dA), ld_da, static_cast<const __nv_bfloat16*>(dP), ld_dp, pidx,
            static_cast<const __nv_bfloat16*>(y), ld_y, scale, shift, coef,
            static_cast<__nv_bfloat16*>(dY), ld_dy, nullptr, relu};
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (pool) launch_co(bn_bwd_kernel<true, true>, grid, block, 0, s, a, g);
  else launch_co(bn_bwd_kernel<false, true>, grid, block, 0, s, a, g);
  return static_cast<int>(cudaGetLastError());
}

}  // extern "C"
