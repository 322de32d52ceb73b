// fp32 / TF32 evaluation mode (BASELINE configs[0]: AttentionUNet fp32 forward; north_star:
// "in fp32/TF32 mode logits must match within 1e-3").  Activations are fp32 NHWC, the 3x3 / 1x1
// convolutions run on the tensor cores as kind::tf32 (conv_fwd.cu, operands rounded to TF32 where
// they are produced), BatchNorm is folded with the running statistics (eval mode), and the passes
// around the convolutions are the plain fp32 kernels below.  Forward only: training runs in bf16.
//
//   f32_pack_weight : OIHW fp32 -> (Cout, taps, Cin) fp32, TF32-rounded                 (layers.py:32,35)
//   f32_conv_in     : first conv (Cin = n_channels) + folded BN + ReLU, NCHW -> NHWC    (layers.py:32-34)
//   f32_maxpool     : MaxPool2d(2)                                                       (layers.py:56)
//   f32_upsample    : bilinear align_corners=True (+ F.pad border)                       (layers.py:78,98-102)
//   f32_gate        : AttentionGate.forward after the two 1x1 projections                (layers.py:183-192)
//   f32_outc        : OutConv, NHWC -> NCHW logits                                       (layers.py:120)
#include "launch.cuh"
#include "../../include/unetb200.h"
#include "conv.h"
#include "ptx.cuh"
#include "resample.cuh"
#include "vec.cuh"

namespace ub2 {

__global__ void f32_pack_weight_kernel(const float* __restrict__ w, float* __restrict__ out, int Cout, int Cin,
                                       int taps) {
  pdl_trigger();
  pdl_wait();
  const long long total = static_cast<long long>(Cout) * Cin * taps;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    // i indexes the pack: ((co*taps + t)*Cin + ci)
    const int ci = static_cast<int>(i % Cin);
    const int t = static_cast<int>((i / Cin) % taps);
    const int co = static_cast<int>(i / (static_cast<long long>(Cin) * taps));
    out[i] = tf32_round(__ldg(w + (static_cast<size_t>(co) * Cin + ci) * taps + t));
  }
}

// thread = (pixel, 4 output channels)
__global__ void __launch_bounds__(256)
f32_conv_in_kernel(const float* __restrict__ x, const float* __restrict__ w, const float* __restrict__ scale,
                   const float* __restrict__ shift, float* __restrict__ out, int N, int Cin, int H, int W,
                   int Cout) {
  pdl_trigger();
  pdl_wait();
  const int c4s = Cout / 4;
  const long long total = static_cast<long long>(N) * H * W * c4s;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c4 = static_cast<int>(i % c4s);
    const long long pix = i / c4s;
    const int wq = static_cast<int>(pix % W);
    const int hq = static_cast<int>((pix / W) % H);
    const int n = static_cast<int>(pix / (static_cast<long long>(W) * H));
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    for (int ci = 0; ci < Cin; ++ci) {
      const float* xp = x + (static_cast<size_t>(n) * Cin + ci) * H * W;
#pragma unroll
      for (int t = 0; t < 9; ++t) {
        const int hh = hq + t / 3 - 1, ww = wq + t % 3 - 1;
        if (hh < 0 || hh >= H || ww < 0 || ww >= W) continue;
        const float xv = __ldg(xp + static_cast<size_t>(hh) * W + ww);
#pragma unroll
        for (int k = 0; k < 4; ++k)
          acc[k] = fmaf(xv, __ldg(w + (static_cast<size_t>(c4 * 4 + k) * Cin + ci) * 9 + t), acc[k]);
      }
    }
    float4 o;
    float* po = &o.x;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int c = c4 * 4 + k;
      po[k] = tf32_round(fmaxf(fmaf(acc[k], __ldg(scale + c), __ldg(shift + c)), 0.f));
    }
    *reinterpret_cast<float4*>(out + pix * Cout + c4 * 4) = o;
  }
}

__global__ void __launch_bounds__(256)
f32_maxpool_kernel(const float* __restrict__ in, float* __restrict__ out, int N, int H, int W, int C) {
  pdl_trigger();
  pdl_wait();
  const int c4s = C / 4, Hp = H / 2, Wp = W / 2;
  const long long total = static_cast<long long>(N) * Hp * Wp * c4s;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c4 = static_cast<int>(i % c4s);
    const long long pp = i / c4s;
    const int wp = static_cast<int>(pp % Wp);
    const int hp = static_cast<int>((pp / Wp) % Hp);
    const int n = static_cast<int>(pp / (static_cast<long long>(Wp) * Hp));
    const float* base = in + ((static_cast<size_t>(n) * H + hp * 2) * W + wp * 2) * C + c4 * 4;
    const float4 a = __ldg(reinterpret_cast<const float4*>(base));
    const float4 b = __ldg(reinterpret_cast<const float4*>(base + C));
    const float4 c = __ldg(reinterpret_cast<const float4*>(base + static_cast<size_t>(W) * C));
    const float4 d = __ldg(reinterpret_cast<const float4*>(base + static_cast<size_t>(W) * C + C));
    float4 o;
    o.x = fmaxf(fmaxf(a.x, b.x), fmaxf(c.x, d.x));
    o.y = fmaxf(fmaxf(a.y, b.y), fmaxf(c.y, d.y));
    o.z = fmaxf(fmaxf(a.z, b.z), fmaxf(c.z, d.z));
    o.w = fmaxf(fmaxf(a.w, b.w), fmaxf(c.w, d.w));
    *reinterpret_cast<float4*>(out + pp * C + c4 * 4) = o;
  }
}

__device__ __forceinline__ float4 lerp4(const float* __restrict__ base, int win, int C, int h0, int h1, int w0,
                                        int w1, float a0, float a1, float b0, float b1, int c) {
  const float4 v00 = __ldg(reinterpret_cast<const float4*>(base + (static_cast<size_t>(h0) * win + w0) * C + c));
  const float4 v01 = __ldg(reinterpret_cast<const float4*>(base + (static_cast<size_t>(h0) * win + w1) * C + c));
  const float4 v10 = __ldg(reinterpret_cast<const float4*>(base + (static_cast<size_t>(h1) * win + w0) * C + c));
  const float4 v11 = __ldg(reinterpret_cast<const float4*>(base + (static_cast<size_t>(h1) * win + w1) * C + c));
  float4 o;
  o.x = a0 * (b0 * v00.x + b1 * v01.x) + a1 * (b0 * v10.x + b1 * v11.x);
  o.y = a0 * (b0 * v00.y + b1 * v01.y) + a1 * (b0 * v10.y + b1 * v11.y);
  o.z = a0 * (b0 * v00.z + b1 * v01.z) + a1 * (b0 * v10.z + b1 * v11.z);
  o.w = a0 * (b0 * v00.w + b1 * v01.w) + a1 * (b0 * v10.w + b1 * v11.w);
  return o;
}

// (hin,win) -> (hu,wu) resampled, centred inside a zero (Ho,Wo) canvas
__global__ void __launch_bounds__(256)
f32_upsample_kernel(const float* __restrict__ in, float* __restrict__ out, int N, int hin, int win, int hu,
                    int wu, int Ho, int Wo, int C, float rh, float rw) {
  pdl_trigger();
  pdl_wait();
  const int c4s = C / 4;
  const int pt = (Ho - hu) / 2, pl = (Wo - wu) / 2;
  const long long total = static_cast<long long>(N) * Ho * Wo * c4s;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c4 = static_cast<int>(i % c4s);
    const long long pix = i / c4s;
    const int wo = static_cast<int>(pix % Wo);
    const int ho = static_cast<int>((pix / Wo) % Ho);
    const int n = static_cast<int>(pix / (static_cast<long long>(Wo) * Ho));
    const int uh = ho - pt, uw = wo - pl;
    float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
    if (uh >= 0 && uh < hu && uw >= 0 && uw < wu) {
      int h0, h1, w0, w1;
      float a0, a1, b0, b1;
      src_index(rh, uh, hin, h0, h1, a0, a1);
      src_index(rw, uw, win, w0, w1, b0, b1);
      o = lerp4(in + static_cast<size_t>(n) * hin * win * C, win, C, h0, h1, w0, w1, a0, a1, b0, b1, c4 * 4);
      o.x = tf32_round(o.x); o.y = tf32_round(o.y); o.z = tf32_round(o.z); o.w = tf32_round(o.w);
    }
    *reinterpret_cast<float4*>(out + pix * C + c4 * 4) = o;
  }
}

// One warp per pixel: psi = w_psi . relu(BN_g(up q) + BN_x(xp)); a = sigmoid(BN_psi(psi)); out = x * a
__global__ void __launch_bounds__(256)
f32_gate_kernel(const float* __restrict__ q, const float* __restrict__ xp, const float* __restrict__ x,
                const float* __restrict__ sg, const float* __restrict__ hg, const float* __restrict__ sx,
                const float* __restrict__ hx, const float* __restrict__ wpsi, const float* __restrict__ spsi,
                const float* __restrict__ hpsi, float* __restrict__ out, int N, int hin, int win, int H, int W,
                int Ci, int Cx, float rh, float rw) {
  pdl_trigger();
  pdl_wait();
  const int lane = threadIdx.x & 31;
  const long long pixels = static_cast<long long>(N) * H * W;
  const long long warps = static_cast<long long>(gridDim.x) * (blockDim.x >> 5);
  for (long long pix = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5); pix < pixels;
       pix += warps) {
    const int wo = static_cast<int>(pix % W);
    const int ho = static_cast<int>((pix / W) % H);
    const int n = static_cast<int>(pix / (static_cast<long long>(W) * H));
    int h0, h1, w0, w1;
    float a0, a1, b0, b1;
    src_index(rh, ho, hin, h0, h1, a0, a1);
    src_index(rw, wo, win, w0, w1, b0, b1);
    const float* qb = q + static_cast<size_t>(n) * hin * win * Ci;
    float dot = 0.f;
    for (int c = lane * 4; c < Ci; c += 128) {
      const float4 u = lerp4(qb, win, Ci, h0, h1, w0, w1, a0, a1, b0, b1, c);
      const float4 v = __ldg(reinterpret_cast<const float4*>(xp + pix * Ci + c));
      const float uu[4] = {u.x, u.y, u.z, u.w}, vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float t = fmaf(uu[k], __ldg(sg + c + k), __ldg(hg + c + k)) +
                        fmaf(vv[k], __ldg(sx + c + k), __ldg(hx + c + k));
        dot = fmaf(fmaxf(t, 0.f), __ldg(wpsi + c + k), dot);
      }
    }
    dot = warp_sum(dot);
    const float z = fmaf(dot, __ldg(spsi), __ldg(hpsi));
    const float a = 1.f / (1.f + expf(-z));
    for (int c = lane * 4; c < Cx; c += 128) {
      float4 v = __ldg(reinterpret_cast<const float4*>(x + pix * Cx + c));
      v.x = tf32_round(v.x * a); v.y = tf32_round(v.y * a); v.z = tf32_round(v.z * a); v.w = tf32_round(v.w * a);
      *reinterpret_cast<float4*>(out + pix * Cx + c) = v;
    }
  }
}

// thread = pixel; K <= 8 classes
__global__ void __launch_bounds__(256)
f32_outc_kernel(const float* __restrict__ a, const float* __restrict__ w, const float* __restrict__ bias,
                float* __restrict__ logits, int N, int H, int W, int C, int K) {
  pdl_trigger();
  pdl_wait();
  const long long HW = static_cast<long long>(H) * W;
  const long long pixels = static_cast<long long>(N) * HW;
  for (long long pix = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; pix < pixels;
       pix += static_cast<long long>(gridDim.x) * blockDim.x) {
    float acc[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) acc[k] = (k < K && bias != nullptr) ? __ldg(bias + k) : 0.f;
    for (int c = 0; c < C; c += 4) {
      const float4 v = __ldg(reinterpret_cast<const float4*>(a + pix * C + c));
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        if (k < K) {
          const float* wr = w + static_cast<size_t>(k) * C + c;
          acc[k] = fmaf(v.x, __ldg(wr), fmaf(v.y, __ldg(wr + 1), fmaf(v.z, __ldg(wr + 2), fmaf(v.w, __ldg(wr + 3), acc[k]))));
        }
      }
    }
    const long long n = pix / HW, hw = pix % HW;
#pragma unroll
    for (int k = 0; k < 8; ++k)
      if (k < K) logits[(n * K + k) * HW + hw] = acc[k];
  }
}

static float ratio(int in, int out) {
  return out > 1 ? static_cast<float>(in - 1) / static_cast<float>(out - 1) : 0.f;
}

}  // namespace ub2

using namespace ub2;

extern "C" {

// Argument checks as in fp32_train.cu, before the device is touched: counts <= 0, channel counts that are not
// multiples of 4, Ho < hu or NULL pointers (bias alone is optional) return UB2_ERR_SHAPE; a pointer that a float4
// access cannot use, UB2_ERR_ALIGN.
static bool c4(int C) { return C > 0 && C % 4 == 0; }
static bool al16(const void* p) { return aligned_to(p, 16); }
static bool al4(const void* p) { return aligned_to(p, 4); }

int ub2_f32_pack_weight(const float* w, float* out, int Cout, int Cin, int taps, void* stream) {
  if (w == nullptr || out == nullptr || Cout <= 0 || Cin <= 0 || (taps != 1 && taps != 9)) return UB2_ERR_SHAPE;
  if (!al4(w) || !al4(out)) return UB2_ERR_ALIGN;
  const long long total = static_cast<long long>(Cout) * Cin * taps;
  launch(f32_pack_weight_kernel, stream_grid(total, 256, num_sms(), 8), 256, 0, static_cast<cudaStream_t>(stream), w, out, Cout, Cin, taps);
  return static_cast<int>(cudaGetLastError());
}

int ub2_f32_conv_in(const float* x, const float* w, const float* scale, const float* shift, float* out, int N,
                    int Cin, int H, int W, int Cout, void* stream) {
  if (x == nullptr || w == nullptr || scale == nullptr || shift == nullptr || out == nullptr || !c4(Cout) || Cin <= 0 ||
      N <= 0 || H <= 0 || W <= 0)
    return UB2_ERR_SHAPE;
  if (!al4(x) || !al4(w) || !al4(scale) || !al4(shift) || !al16(out)) return UB2_ERR_ALIGN;
  const long long total = static_cast<long long>(N) * H * W * (Cout / 4);
  launch(f32_conv_in_kernel, stream_grid(total, 256, num_sms(), 8), 256, 0, static_cast<cudaStream_t>(stream), x, w, scale, shift, out, N, Cin, H, W, Cout);
  return static_cast<int>(cudaGetLastError());
}

int ub2_f32_maxpool(const float* in, float* out, int N, int H, int W, int C, void* stream) {
  if (in == nullptr || out == nullptr || !c4(C) || H < 2 || W < 2 || N <= 0) return UB2_ERR_SHAPE;
  if (!al16(in) || !al16(out)) return UB2_ERR_ALIGN;
  const long long total = static_cast<long long>(N) * (H / 2) * (W / 2) * (C / 4);
  launch(f32_maxpool_kernel, stream_grid(total, 256, num_sms(), 8), 256, 0, static_cast<cudaStream_t>(stream), in, out, N, H, W, C);
  return static_cast<int>(cudaGetLastError());
}

int ub2_f32_upsample(const float* in, float* out, int N, int hin, int win, int hu, int wu, int Ho, int Wo, int C,
                     void* stream) {
  if (in == nullptr || out == nullptr || !c4(C) || N <= 0 || hin <= 0 || win <= 0 || hu <= 0 || wu <= 0 || Ho < hu || Wo < wu)
    return UB2_ERR_SHAPE;
  if (!al16(in) || !al16(out)) return UB2_ERR_ALIGN;
  const long long total = static_cast<long long>(N) * Ho * Wo * (C / 4);
  launch(f32_upsample_kernel, stream_grid(total, 256, num_sms(), 8), 256, 0, static_cast<cudaStream_t>(stream), in, out, N, hin, win, hu, wu, Ho, Wo, C, ratio(hin, hu), ratio(win, wu));
  return static_cast<int>(cudaGetLastError());
}

int ub2_f32_gate(const float* q, const float* xp, const float* x, const float* scale_g, const float* shift_g,
                 const float* scale_x, const float* shift_x, const float* w_psi, const float* scale_psi,
                 const float* shift_psi, float* out, int N, int hin, int win, int H, int W, int Ci, int Cx,
                 void* stream) {
  if (q == nullptr || xp == nullptr || x == nullptr || scale_g == nullptr || shift_g == nullptr || scale_x == nullptr ||
      shift_x == nullptr || w_psi == nullptr || scale_psi == nullptr || shift_psi == nullptr || out == nullptr)
    return UB2_ERR_SHAPE;
  if (!c4(Ci) || !c4(Cx) || N <= 0 || hin <= 0 || win <= 0 || H <= 0 || W <= 0) return UB2_ERR_SHAPE;
  if (!al16(q) || !al16(xp) || !al16(x) || !al16(out) || !al4(scale_g) || !al4(shift_g) || !al4(scale_x) || !al4(shift_x) ||
      !al4(w_psi) || !al4(scale_psi) || !al4(shift_psi))
    return UB2_ERR_ALIGN;
  const long long pixels = static_cast<long long>(N) * H * W;
  launch(f32_gate_kernel, stream_grid(pixels, 8, num_sms(), 8), 256, 0, static_cast<cudaStream_t>(stream), q, xp, x, scale_g, shift_g, scale_x, shift_x, w_psi, scale_psi, shift_psi, out, N, hin, win, H, W, Ci, Cx, ratio(hin, H), ratio(win, W));
  return static_cast<int>(cudaGetLastError());
}

int ub2_f32_outc(const float* a, const float* w, const float* bias, float* logits, int N, int H, int W, int C,
                 int K, void* stream) {
  if (a == nullptr || w == nullptr || logits == nullptr || !c4(C) || K <= 0 || K > 8 || N <= 0 || H <= 0 || W <= 0)
    return UB2_ERR_SHAPE;
  if (!al16(a) || !al4(w) || !al4(bias) || !al4(logits)) return UB2_ERR_ALIGN;
  const long long pixels = static_cast<long long>(N) * H * W;
  launch(f32_outc_kernel, stream_grid(pixels, 256, num_sms(), 8), 256, 0, static_cast<cudaStream_t>(stream), a, w, bias, logits, N, H, W, C, K);
  return static_cast<int>(cudaGetLastError());
}

}  // extern "C"
