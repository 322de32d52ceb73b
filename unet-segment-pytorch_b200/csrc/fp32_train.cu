// fp32 / TF32 TRAINING mode (north_star: "in fp32/TF32 mode, logits and gradients must match within 1e-3";
// the reference's own training runs in fp32: scripts/train.py:132-136).  Activations and their gradients
// are fp32 NHWC, stored unrounded.
//
// A single TF32 pass is NOT enough for the gradients: its 2^-11 operand rounding moves ~2e-4 of the
// pre-activations across zero, and every ReLU decision that differs from the reference's costs a whole
// gradient element (measured per module: outputs 3e-4, gradients 1-3e-2).  So forward and data-gradient
// convolutions run as 3xTF32 on the tensor cores: each operand is split into two TF32 numbers
// x = hi + lo (f32_split_tf32 writes [hi | lo] along the channel axis), the weights likewise, and ONE launch
// of the kind::tf32 implicit-GEMM kernel (conv_fwd.cu) walks the K axis [a_hi | a_lo | a_hi] against
// [w_hi | w_hi | w_lo] (f32_pack_weight3) — its two virtual-concat sources are the split tensor and a view of
// its first half — accumulating a_hi.w_hi + a_lo.w_hi + a_hi.w_lo in fp32 in TMEM (error ~2^-21).
// kind::tf32 has no MN-major operand mode (tools/probe/umma_tf32_mn.cu: the instruction returns zeros), so
// the weight gradient — whose operands are channel-contiguous — runs on the bf16 kernels with each fp32
// operand split into hi + lo bf16 halves (x = hi + lo to 2^-16): dW = a_hi.dy_hi + a_lo.dy_hi + a_hi.dy_lo,
// three launches into the same fp32 split-K fold.  Everything around the convolutions is the plain fp32 kernels below:
// this is the accuracy mode, written for clarity and determinism (fixed-order fp64 folds of per-block
// partial rows, shared with the bf16 path's finalize kernels), not tuned to the roofline like the bf16 path.
//
//   f32_channel_stats   per-channel sum / sum of squares                     BatchNorm2d train statistics
//   f32_affine_act      a = relu(scale*y + shift),                           layers.py:33-34
//   f32_maxpool_idx     MaxPool2d(2) + window position of the maximum        layers.py:56
//   f32_act_bwd_reduce / _apply   BatchNorm + ReLU (+ max-pool routing) backward
//   f32_upsample_bwd    transpose of the bilinear resampling (gather form)   layers.py:78, :98-102
//   f32_gate_*          AttentionGate.forward / backward around the 1x1 projections   layers.py:171-192
//   f32_outc_bwd        OutConv backward                                     layers.py:120
//   f32_conv_in_wgrad   first convolution's weight gradient (Cin = n_channels)
//   f32_split_bf16      x -> (hi, lo) bf16
//   f32_split_tf32 / f32_pack_weight3   the 3xTF32 operand split and weight packs
//   f32_upsample_fwd    bilinear resampling, unrounded
#include "launch.cuh"
#include "../../include/unetb200.h"
#include "conv.h"
#include "ptx.cuh"
#include "resample.cuh"
#include "vec.cuh"

namespace ub2 {

static constexpr int kFT = 256;   // threads per block

__device__ __forceinline__ float4 ld4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ void st4(float* p, const float4& v) { *reinterpret_cast<float4*>(p) = v; }
// training keeps full fp32 values: the convolutions split their operands themselves (3xTF32, see above)
__device__ __forceinline__ float4 round4(float4 v) { return v; }

// ---- per-channel reductions: thread = (pixel lane, 4 channels), channel group fixed per thread ----------------
// Fold the per-thread sums of NS statistics over the pixel lanes of the block; one fp64 row [NS][C] per block.
template <int NS>
__device__ __forceinline__ void fold_channels(float (&acc)[NS][4], int lane, int lanes, int c4, int c4s, int C,
                                              double* row, float* smem /* [kFT * 4] */) {
#pragma unroll
  for (int s = 0; s < NS; ++s) {
    if (lane < lanes) {
#pragma unroll
      for (int k = 0; k < 4; ++k) smem[(lane * c4s + c4) * 4 + k] = acc[s][k];
    }
    __syncthreads();
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
      double t = 0.0;
      for (int l = 0; l < lanes; ++l) t += static_cast<double>(smem[(l * c4s + (c >> 2)) * 4 + (c & 3)]);
      row[static_cast<size_t>(s) * C + c] = t;
    }
    __syncthreads();
  }
}
static int chan_lanes(int C) { return kFT / (C / 4) > 0 ? kFT / (C / 4) : 1; }
static int chan_grid(long long pixels, int C) { return stream_grid(pixels, chan_lanes(C), num_sms(), 4); }

__global__ void __launch_bounds__(kFT)
f32_channel_stats_kernel(const float* __restrict__ x, int ld, long long pixels, int C, double* partials) {
  pdl_trigger();
  pdl_wait();
  __shared__ float smem[kFT * 4];
  const int c4s = C / 4, lanes = blockDim.x / c4s, lane = threadIdx.x / c4s, c4 = threadIdx.x % c4s;
  float acc[2][4] = {};
  if (lane < lanes) {
    for (long long p = static_cast<long long>(blockIdx.x) * lanes + lane; p < pixels; p += static_cast<long long>(gridDim.x) * lanes) {
      const float4 v = ld4(x + p * ld + c4 * 4);
      acc[0][0] += v.x; acc[0][1] += v.y; acc[0][2] += v.z; acc[0][3] += v.w;
      acc[1][0] = fmaf(v.x, v.x, acc[1][0]); acc[1][1] = fmaf(v.y, v.y, acc[1][1]);
      acc[1][2] = fmaf(v.z, v.z, acc[1][2]); acc[1][3] = fmaf(v.w, v.w, acc[1][3]);
    }
  }
  fold_channels<2>(acc, lane, lanes, c4, c4s, C, partials + static_cast<size_t>(blockIdx.x) * 2 * C, smem);
}

// per-pixel scalar field (the gate's psi): rows of (sum, sum of squares)
__global__ void __launch_bounds__(kFT)
f32_scalar_stats_kernel(const float* __restrict__ x, long long n, double* partials) {
  pdl_trigger();
  pdl_wait();
  __shared__ float smem[2][kFT / 32];
  float s = 0.f, q = 0.f;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float v = __ldg(x + i);
    s += v;
    q = fmaf(v, v, q);
  }
  s = warp_sum(s);
  q = warp_sum(q);
  if ((threadIdx.x & 31) == 0) { smem[0][threadIdx.x >> 5] = s; smem[1][threadIdx.x >> 5] = q; }
  __syncthreads();
  if (threadIdx.x < 2) {
    double t = 0.0;
    for (int i = 0; i < kFT / 32; ++i) t += static_cast<double>(smem[threadIdx.x][i]);
    partials[static_cast<size_t>(blockIdx.x) * 2 + threadIdx.x] = t;
  }
}

// ---- BatchNorm apply + ReLU, max-pool ---------------------------------------------------------------------------
__global__ void __launch_bounds__(kFT)
f32_affine_act_kernel(const float* __restrict__ y, const float* __restrict__ scale, const float* __restrict__ shift,
                      float* __restrict__ out, long long pixels, int C, int relu) {
  pdl_trigger();
  pdl_wait();
  const int c4s = C / 4;
  const long long total = pixels * c4s;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i % c4s) * 4;
    float4 v = ld4(y + i * 4);
    const float4 sc = ld4(scale + c), sh = ld4(shift + c);
    v.x = fmaf(v.x, sc.x, sh.x); v.y = fmaf(v.y, sc.y, sh.y); v.z = fmaf(v.z, sc.z, sh.z); v.w = fmaf(v.w, sc.w, sh.w);
    if (relu) { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f); }
    st4(out + i * 4, round4(v));
  }
}

// p = max over the 2x2 window, idx = position (row*2 + col) of the FIRST maximum (ATen's tie rule)
__global__ void __launch_bounds__(kFT)
f32_maxpool_idx_kernel(const float* __restrict__ a, float* __restrict__ p, unsigned char* __restrict__ idx, int N, int H,
                       int W, int C) {
  pdl_trigger();
  pdl_wait();
  const int c4s = C / 4, Hp = H / 2, Wp = W / 2;
  const long long total = static_cast<long long>(N) * Hp * Wp * c4s;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c4 = static_cast<int>(i % c4s);
    const long long pp = i / c4s;
    const int wp = static_cast<int>(pp % Wp);
    const int hp = static_cast<int>((pp / Wp) % Hp);
    const int n = static_cast<int>(pp / (static_cast<long long>(Wp) * Hp));
    const float* base = a + ((static_cast<size_t>(n) * H + hp * 2) * W + wp * 2) * C + c4 * 4;
    float best[4];
    unsigned arg[4] = {0u, 0u, 0u, 0u};
#pragma unroll
    for (int d = 0; d < 4; ++d) {
      const float4 v = ld4(base + (static_cast<size_t>(d >> 1) * W + (d & 1)) * C);
      const float vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        if (d == 0 || vv[k] > best[k]) {
          best[k] = vv[k];
          arg[k] = d;
        }
      }
    }
    st4(p + pp * C + c4 * 4, make_float4(best[0], best[1], best[2], best[3]));
    *reinterpret_cast<uchar4*>(idx + pp * C + c4 * 4) = make_uchar4(arg[0], arg[1], arg[2], arg[3]);
  }
}

// gradient reaching the activation of pixel (n,h,w): dA (optional) + the pooled gradient routed to the maximum
__device__ __forceinline__ float4 act_grad(const float* __restrict__ dA, int ld_da, const float* __restrict__ dP,
                                           const unsigned char* __restrict__ idx, long long pix, int n, int h, int w,
                                           int H, int W, int C, int c) {
  float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
  if (dA != nullptr) g = ld4(dA + pix * ld_da + c);
  if (dP != nullptr) {
    const int Hp = H / 2, Wp = W / 2, hp = h >> 1, wp = w >> 1;
    if (hp < Hp && wp < Wp) {
      const long long pp = (static_cast<long long>(n) * Hp + hp) * Wp + wp;
      const uchar4 a = *reinterpret_cast<const uchar4*>(idx + pp * C + c);
      const float4 d = ld4(dP + pp * C + c);
      const unsigned pos = (h & 1) * 2 + (w & 1);
      if (a.x == pos) g.x += d.x;
      if (a.y == pos) g.y += d.y;
      if (a.z == pos) g.z += d.z;
      if (a.w == pos) g.w += d.w;
    }
  }
  return g;
}

// rows of (sum dz, sum dz*y), dz = g * [scale*y + shift > 0]  (bn_bwd_finalize's convention)
__global__ void __launch_bounds__(kFT)
f32_act_bwd_reduce_kernel(const float* __restrict__ dA, int ld_da, const float* __restrict__ dP,
                          const unsigned char* __restrict__ idx, const float* __restrict__ y,
                          const float* __restrict__ scale, const float* __restrict__ shift, double* partials, int N, int H,
                          int W, int C, int relu) {
  pdl_trigger();
  pdl_wait();
  __shared__ float smem[kFT * 4];
  const int c4s = C / 4, lanes = blockDim.x / c4s, lane = threadIdx.x / c4s, c4 = threadIdx.x % c4s;
  const long long pixels = static_cast<long long>(N) * H * W;
  float acc[2][4] = {};
  if (lane < lanes) {
    const float4 sc = ld4(scale + c4 * 4), sh = ld4(shift + c4 * 4);
    for (long long p = static_cast<long long>(blockIdx.x) * lanes + lane; p < pixels; p += static_cast<long long>(gridDim.x) * lanes) {
      const int w = static_cast<int>(p % W), h = static_cast<int>((p / W) % H), n = static_cast<int>(p / (static_cast<long long>(W) * H));
      float4 g = act_grad(dA, ld_da, dP, idx, p, n, h, w, H, W, C, c4 * 4);
      const float4 v = ld4(y + p * C + c4 * 4);
      if (relu) {
        if (fmaf(v.x, sc.x, sh.x) <= 0.f) g.x = 0.f;
        if (fmaf(v.y, sc.y, sh.y) <= 0.f) g.y = 0.f;
        if (fmaf(v.z, sc.z, sh.z) <= 0.f) g.z = 0.f;
        if (fmaf(v.w, sc.w, sh.w) <= 0.f) g.w = 0.f;
      }
      acc[0][0] += g.x; acc[0][1] += g.y; acc[0][2] += g.z; acc[0][3] += g.w;
      acc[1][0] = fmaf(g.x, v.x, acc[1][0]); acc[1][1] = fmaf(g.y, v.y, acc[1][1]);
      acc[1][2] = fmaf(g.z, v.z, acc[1][2]); acc[1][3] = fmaf(g.w, v.w, acc[1][3]);
    }
  }
  fold_channels<2>(acc, lane, lanes, c4, c4s, C, partials + static_cast<size_t>(blockIdx.x) * 2 * C, smem);
}

// dy = coef0*dz + coef1*y + coef2, unrounded (the convolutions that take it split it themselves)
__global__ void __launch_bounds__(kFT)
f32_act_bwd_apply_kernel(const float* __restrict__ dA, int ld_da, const float* __restrict__ dP,
                         const unsigned char* __restrict__ idx, const float* __restrict__ y,
                         const float* __restrict__ scale, const float* __restrict__ shift, const float* __restrict__ coef,
                         float* __restrict__ dy, int N, int H, int W, int C, int relu) {
  pdl_trigger();
  pdl_wait();
  const int c4s = C / 4;
  const long long total = static_cast<long long>(N) * H * W * c4s;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i % c4s) * 4;
    const long long p = i / c4s;
    const int w = static_cast<int>(p % W), h = static_cast<int>((p / W) % H), n = static_cast<int>(p / (static_cast<long long>(W) * H));
    float4 g = act_grad(dA, ld_da, dP, idx, p, n, h, w, H, W, C, c);
    const float4 v = ld4(y + p * C + c);
    if (relu) {
      const float4 sc = ld4(scale + c), sh = ld4(shift + c);
      if (fmaf(v.x, sc.x, sh.x) <= 0.f) g.x = 0.f;
      if (fmaf(v.y, sc.y, sh.y) <= 0.f) g.y = 0.f;
      if (fmaf(v.z, sc.z, sh.z) <= 0.f) g.z = 0.f;
      if (fmaf(v.w, sc.w, sh.w) <= 0.f) g.w = 0.f;
    }
    const float4 a = ld4(coef + c), b = ld4(coef + C + c), d = ld4(coef + 2 * C + c);
    float4 o;
    o.x = fmaf(a.x, g.x, fmaf(b.x, v.x, d.x)); o.y = fmaf(a.y, g.y, fmaf(b.y, v.y, d.y));
    o.z = fmaf(a.z, g.z, fmaf(b.z, v.z, d.z)); o.w = fmaf(a.w, g.w, fmaf(b.w, v.w, d.w));
    st4(dy + p * C + c, round4(o));
  }
}

// ---- bilinear resampling, transpose (gather form: deterministic) ------------------------------------------------
// destination rows / columns whose interpolation touches source index i
__device__ __forceinline__ void f32_dst_range(float r, int i, int out, int& lo, int& hi) {
  if (r <= 0.f) { lo = 0; hi = out - 1; return; }
  lo = static_cast<int>(ceilf((static_cast<float>(i) - 1.f) / r)) - 1;
  hi = static_cast<int>(floorf((static_cast<float>(i) + 1.f) / r)) + 1;
  if (lo < 0) lo = 0;
  if (hi > out - 1) hi = out - 1;
}
__device__ __forceinline__ float f32_tap_weight(float r, int dst, int in, int i) {
  int i0, i1;
  float l0, l1;
  src_index(r, dst, in, i0, i1, l0, l1);
  float wgt = 0.f;
  if (i0 == i) wgt += l0;
  if (i1 == i) wgt += l1;
  return wgt;
}
__global__ void __launch_bounds__(kFT)
f32_upsample_bwd_kernel(const float* __restrict__ dout, int ld_dout, float* __restrict__ din, int N, int hin, int win,
                        int hu, int wu, int Ho, int Wo, int C, float rh, float rw) {
  pdl_trigger();
  pdl_wait();
  const int c4s = C / 4;
  const int pt = (Ho - hu) / 2, pl = (Wo - wu) / 2;
  const long long total = static_cast<long long>(N) * hin * win * c4s;
  for (long long t = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; t < total; t += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(t % c4s) * 4;
    const long long sp = t / c4s;
    const int j = static_cast<int>(sp % win), i = static_cast<int>((sp / win) % hin);
    const int n = static_cast<int>(sp / (static_cast<long long>(win) * hin));
    int ylo, yhi, xlo, xhi;
    f32_dst_range(rh, i, hu, ylo, yhi);
    f32_dst_range(rw, j, wu, xlo, xhi);
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int yy = ylo; yy <= yhi; ++yy) {
      const float wy = f32_tap_weight(rh, yy, hin, i);
      if (wy == 0.f) continue;
      for (int xx = xlo; xx <= xhi; ++xx) {
        const float wx = f32_tap_weight(rw, xx, win, j);
        if (wx == 0.f) continue;
        const float4 v = ld4(dout + ((static_cast<size_t>(n) * Ho + yy + pt) * Wo + xx + pl) * ld_dout + c);
        const float ww = wy * wx;
        acc.x = fmaf(ww, v.x, acc.x); acc.y = fmaf(ww, v.y, acc.y); acc.z = fmaf(ww, v.z, acc.z); acc.w = fmaf(ww, v.w, acc.w);
      }
    }
    st4(din + sp * C + c, round4(acc));
  }
}

// ---- attention gate: one warp per pixel, a lane owns channels lane*4 + 128*i (Ci <= 512) ------------------------
static constexpr int kGI = 4;   // 128-channel slices per lane

// psi_raw = w_psi . relu(sg*u + sx*xp + hg + hx);  u = up(q) materialised (fp32 mode keeps the passes plain)
__global__ void __launch_bounds__(kFT)
f32_gate_psi_kernel(const float* __restrict__ u, const float* __restrict__ xp, const float* __restrict__ sg,
                    const float* __restrict__ hg, const float* __restrict__ sx, const float* __restrict__ hx,
                    const float* __restrict__ wpsi, float* __restrict__ psi_raw, long long pixels, int Ci) {
  pdl_trigger();
  pdl_wait();
  const int lane = threadIdx.x & 31;
  const long long warps = static_cast<long long>(gridDim.x) * (blockDim.x >> 5);
  for (long long pix = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5); pix < pixels; pix += warps) {
    float dot = 0.f;
    for (int c = lane * 4; c < Ci; c += 128) {
      const float4 a = ld4(u + pix * Ci + c), b = ld4(xp + pix * Ci + c);
      const float4 s1 = ld4(sg + c), s2 = ld4(sx + c), h1 = ld4(hg + c), h2 = ld4(hx + c), wv = ld4(wpsi + c);
      dot = fmaf(wv.x, fmaxf(fmaf(a.x, s1.x, fmaf(b.x, s2.x, h1.x + h2.x)), 0.f), dot);
      dot = fmaf(wv.y, fmaxf(fmaf(a.y, s1.y, fmaf(b.y, s2.y, h1.y + h2.y)), 0.f), dot);
      dot = fmaf(wv.z, fmaxf(fmaf(a.z, s1.z, fmaf(b.z, s2.z, h1.z + h2.z)), 0.f), dot);
      dot = fmaf(wv.w, fmaxf(fmaf(a.w, s1.w, fmaf(b.w, s2.w, h1.w + h2.w)), 0.f), dot);
    }
    dot = warp_sum(dot);
    if (lane == 0) psi_raw[pix] = dot;
  }
}

// a = sigmoid(spsi*psi_raw + hpsi); out = x * a (TF32-rounded)
__global__ void __launch_bounds__(kFT)
f32_gate_apply_kernel(const float* __restrict__ psi_raw, const float* __restrict__ spsi, const float* __restrict__ hpsi,
                      const float* __restrict__ x, float* __restrict__ out, float* __restrict__ a_out, long long pixels,
                      int Cx) {
  pdl_trigger();
  pdl_wait();
  const float s = __ldg(spsi), h = __ldg(hpsi);
  const int c4s = Cx / 4;
  const long long total = pixels * c4s;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long pix = i / c4s;
    const float a = 1.f / (1.f + expf(-fmaf(__ldg(psi_raw + pix), s, h)));
    float4 v = ld4(x + i * 4);
    v.x *= a; v.y *= a; v.z *= a; v.w *= a;
    st4(out + i * 4, round4(v));
    if (a_out != nullptr && (i % c4s) == 0) a_out[pix] = a;
  }
}

// da = sum_c dOut_c x_c ; dn = da * a (1-a) ; dx_direct = dOut * a ; rows of (sum dn, sum dn*psi_raw)
__global__ void __launch_bounds__(kFT)
f32_gate_bwd_a_kernel(const float* __restrict__ dout, int ld_do, const float* __restrict__ x, const float* __restrict__ a,
                      const float* __restrict__ psi_raw, float* __restrict__ dx, float* __restrict__ dpsin, double* partials,
                      long long pixels, int Cx) {
  pdl_trigger();
  pdl_wait();
  __shared__ float smem[2][kFT / 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long warps = static_cast<long long>(gridDim.x) * (blockDim.x >> 5);
  float st0 = 0.f, st1 = 0.f;
  for (long long pix = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + warp; pix < pixels; pix += warps) {
    const float av = __ldg(a + pix);
    float dot = 0.f;
    for (int c = lane * 4; c < Cx; c += 128) {
      float4 d = ld4(dout + pix * ld_do + c);
      const float4 xv = ld4(x + pix * Cx + c);
      dot = fmaf(d.x, xv.x, fmaf(d.y, xv.y, fmaf(d.z, xv.z, fmaf(d.w, xv.w, dot))));
      d.x *= av; d.y *= av; d.z *= av; d.w *= av;
      st4(dx + pix * Cx + c, d);
    }
    dot = warp_sum(dot);
    if (lane == 0) {
      const float dn = dot * av * (1.f - av);
      dpsin[pix] = dn;
      st0 += dn;
      st1 = fmaf(dn, __ldg(psi_raw + pix), st1);
    }
  }
  if (lane == 0) { smem[0][warp] = st0; smem[1][warp] = st1; }
  __syncthreads();
  if (threadIdx.x < 2) {
    double t = 0.0;
    for (int i = 0; i < kFT / 32; ++i) t += static_cast<double>(smem[threadIdx.x][i]);
    partials[static_cast<size_t>(blockIdx.x) * 2 + threadIdx.x] = t;
  }
}

// ds_c = dpsi_raw * w_psi_c * [t_c > 0]; rows of (sum ds, sum ds*xp, sum ds*u, sum dpsi_raw*relu(t)) per channel
__global__ void __launch_bounds__(kFT)
f32_gate_bwd_s_kernel(const float* __restrict__ dpsin, const float* __restrict__ psi_raw, const float* __restrict__ coef_psi,
                      const float* __restrict__ u, const float* __restrict__ xp, const float* __restrict__ sg,
                      const float* __restrict__ hg, const float* __restrict__ sx, const float* __restrict__ hx,
                      const float* __restrict__ wpsi, float* __restrict__ ds, double* partials, long long pixels, int Ci) {
  pdl_trigger();
  pdl_wait();
  extern __shared__ float dyn[];   // [warps][4][Ci]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const long long warps = static_cast<long long>(gridDim.x) * nw;
  const float cA = __ldg(coef_psi), cB = __ldg(coef_psi + 1), cC = __ldg(coef_psi + 2);
  float acc[kGI][4][4] = {};
  for (long long pix = static_cast<long long>(blockIdx.x) * nw + warp; pix < pixels; pix += warps) {
    const float dpr = fmaf(cA, __ldg(dpsin + pix), fmaf(cB, __ldg(psi_raw + pix), cC));   // BN_psi backward
#pragma unroll
    for (int i = 0; i < kGI; ++i) {
      const int c = lane * 4 + 128 * i;
      if (c < Ci) {
        const float4 a = ld4(u + pix * Ci + c), b = ld4(xp + pix * Ci + c);
        const float4 s1 = ld4(sg + c), s2 = ld4(sx + c), h1 = ld4(hg + c), h2 = ld4(hx + c), wv = ld4(wpsi + c);
        const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
        const float s1v[4] = {s1.x, s1.y, s1.z, s1.w}, s2v[4] = {s2.x, s2.y, s2.z, s2.w};
        const float hv[4] = {h1.x + h2.x, h1.y + h2.y, h1.z + h2.z, h1.w + h2.w}, wvv[4] = {wv.x, wv.y, wv.z, wv.w};
        float o[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const float t = fmaf(av[k], s1v[k], fmaf(bv[k], s2v[k], hv[k]));
          const float d = (t > 0.f) ? dpr * wvv[k] : 0.f;
          o[k] = d;
          acc[i][0][k] += d;
          acc[i][1][k] = fmaf(d, bv[k], acc[i][1][k]);
          acc[i][2][k] = fmaf(d, av[k], acc[i][2][k]);
          acc[i][3][k] = fmaf(dpr, fmaxf(t, 0.f), acc[i][3][k]);
        }
        st4(ds + pix * Ci + c, make_float4(o[0], o[1], o[2], o[3]));
      }
    }
  }
#pragma unroll
  for (int i = 0; i < kGI; ++i) {
    const int c = lane * 4 + 128 * i;
    if (c < Ci) {
#pragma unroll
      for (int s = 0; s < 4; ++s)
#pragma unroll
        for (int k = 0; k < 4; ++k) dyn[(static_cast<size_t>(warp) * 4 + s) * Ci + c + k] = acc[i][s][k];
    }
  }
  __syncthreads();
  for (int e = threadIdx.x; e < 4 * Ci; e += blockDim.x) {
    double t = 0.0;
    for (int wv = 0; wv < nw; ++wv) t += static_cast<double>(dyn[static_cast<size_t>(wv) * 4 * Ci + e]);
    partials[static_cast<size_t>(blockIdx.x) * 4 * Ci + e] = t;
  }
}

// dxp = coef0*ds + coef1*xp + coef2 ; du = coef3*ds + coef4*u + coef5  (gate_bwd_finalize's coefficients)
__global__ void __launch_bounds__(kFT)
f32_gate_bwd_xg_kernel(const float* __restrict__ ds, const float* __restrict__ xp, const float* __restrict__ u,
                       const float* __restrict__ coef, float* __restrict__ dxp, float* __restrict__ du, long long pixels,
                       int Ci) {
  pdl_trigger();
  pdl_wait();
  const int c4s = Ci / 4;
  const long long total = pixels * c4s;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i % c4s) * 4;
    const float4 d = ld4(ds + i * 4), xv = ld4(xp + i * 4), uv = ld4(u + i * 4);
    const float4 c0 = ld4(coef + c), c1 = ld4(coef + Ci + c), c2 = ld4(coef + 2 * Ci + c);
    const float4 c3 = ld4(coef + 3 * Ci + c), c4 = ld4(coef + 4 * Ci + c), c5 = ld4(coef + 5 * Ci + c);
    float4 ox, og;
    ox.x = fmaf(c0.x, d.x, fmaf(c1.x, xv.x, c2.x)); ox.y = fmaf(c0.y, d.y, fmaf(c1.y, xv.y, c2.y));
    ox.z = fmaf(c0.z, d.z, fmaf(c1.z, xv.z, c2.z)); ox.w = fmaf(c0.w, d.w, fmaf(c1.w, xv.w, c2.w));
    og.x = fmaf(c3.x, d.x, fmaf(c4.x, uv.x, c5.x)); og.y = fmaf(c3.y, d.y, fmaf(c4.y, uv.y, c5.y));
    og.z = fmaf(c3.z, d.z, fmaf(c4.z, uv.z, c5.z)); og.w = fmaf(c3.w, d.w, fmaf(c4.w, uv.w, c5.w));
    st4(dxp + i * 4, round4(ox));
    st4(du + i * 4, og);
  }
}

// ---- output head backward: thread = pixel; K <= 8 classes ------------------------------------------------------
// da[c] = sum_k dl[k] w[k][c]; rows of (dw[k][c] = sum dl[k] a[c], db[k] = sum dl[k]) per block
__global__ void __launch_bounds__(kFT)
f32_outc_bwd_kernel(const float* __restrict__ dlogits, const float* __restrict__ a, const float* __restrict__ w,
                    float* __restrict__ da, double* partials, int N, int H, int W, int C, int K) {
  pdl_trigger();
  pdl_wait();
  extern __shared__ float dyn[];   // [warps][K*C + K]
  const long long HW = static_cast<long long>(H) * W, pixels = static_cast<long long>(N) * HW;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const int cols = K * C + K;
  for (int e = threadIdx.x; e < nw * cols; e += blockDim.x) dyn[e] = 0.f;
  __syncthreads();
  float* mine = dyn + static_cast<size_t>(warp) * cols;
  // a warp walks pixels one at a time; lanes split the channels, so dw accumulates in shared memory per warp
  const long long warps = static_cast<long long>(gridDim.x) * nw;
  for (long long pix = static_cast<long long>(blockIdx.x) * nw + warp; pix < pixels; pix += warps) {
    const long long n = pix / HW, hw = pix % HW;
    float dl[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) dl[k] = (k < K) ? __ldg(dlogits + (n * K + k) * HW + hw) : 0.f;
    for (int c = lane * 4; c < C; c += 128) {
      const float4 av = ld4(a + pix * C + c);
      float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        if (k < K) {
          const float4 wv = ld4(w + static_cast<size_t>(k) * C + c);
          o.x = fmaf(dl[k], wv.x, o.x); o.y = fmaf(dl[k], wv.y, o.y); o.z = fmaf(dl[k], wv.z, o.z); o.w = fmaf(dl[k], wv.w, o.w);
          float* m = mine + k * C + c;
          m[0] = fmaf(dl[k], av.x, m[0]); m[1] = fmaf(dl[k], av.y, m[1]); m[2] = fmaf(dl[k], av.z, m[2]); m[3] = fmaf(dl[k], av.w, m[3]);
        }
      }
      if (da != nullptr) st4(da + pix * C + c, round4(o));
    }
    if (lane == 0) {
#pragma unroll
      for (int k = 0; k < 8; ++k)
        if (k < K) mine[K * C + k] += dl[k];
    }
  }
  __syncthreads();
  for (int e = threadIdx.x; e < cols; e += blockDim.x) {
    double t = 0.0;
    for (int wv = 0; wv < nw; ++wv) t += static_cast<double>(dyn[static_cast<size_t>(wv) * cols + e]);
    partials[static_cast<size_t>(blockIdx.x) * cols + e] = t;
  }
}

// out[e] += sum over rows of partials[row*stride + col0 + e], e < ncols (fixed order)
__global__ void f32_cols_fold_kernel(const double* __restrict__ partials, int rows, int stride, int col0, int ncols, float* out) {
  pdl_trigger();
  pdl_wait();
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= ncols) return;
  double s = 0.0;
  for (int r = 0; r < rows; ++r) s += partials[static_cast<size_t>(r) * stride + col0 + e];
  out[e] += static_cast<float>(s);
}

// ---- first convolution (Cin = n_channels): raw output, and its weight gradient ---------------------------------
// thread = (pixel, 4 output channels); out = conv (+ optional affine and ReLU, TF32-rounded when `act`)
__global__ void __launch_bounds__(kFT)
f32_conv_in_raw_kernel(const float* __restrict__ x, const float* __restrict__ w, float* __restrict__ out, int N, int Cin,
                       int H, int W, int Cout) {
  pdl_trigger();
  pdl_wait();
  const int c4s = Cout / 4;
  const long long total = static_cast<long long>(N) * H * W * c4s;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c4 = static_cast<int>(i % c4s);
    const long long pix = i / c4s;
    const int wq = static_cast<int>(pix % W), hq = static_cast<int>((pix / W) % H);
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
        for (int k = 0; k < 4; ++k) acc[k] = fmaf(xv, __ldg(w + (static_cast<size_t>(c4 * 4 + k) * Cin + ci) * 9 + t), acc[k]);
      }
    }
    st4(out + pix * Cout + c4 * 4, make_float4(acc[0], acc[1], acc[2], acc[3]));
  }
}

// rows of dw[(ci*9 + t)][co] = sum_pixels x[n, ci, h+dr, w+ds] * dy[n, h, w, co]
__global__ void __launch_bounds__(kFT)
f32_conv_in_wgrad_kernel(const float* __restrict__ x, const float* __restrict__ dy, double* partials, int N, int Cin, int H,
                         int W, int Cout) {
  pdl_trigger();
  pdl_wait();
  __shared__ float smem[kFT * 4];
  const int c4s = Cout / 4, lanes = blockDim.x / c4s, lane = threadIdx.x / c4s, c4 = threadIdx.x % c4s;
  const long long pixels = static_cast<long long>(N) * H * W;
  for (int ci = 0; ci < Cin; ++ci) {
    float acc[9][4] = {};
    if (lane < lanes) {
      for (long long p = static_cast<long long>(blockIdx.x) * lanes + lane; p < pixels; p += static_cast<long long>(gridDim.x) * lanes) {
        const int wq = static_cast<int>(p % W), hq = static_cast<int>((p / W) % H);
        const int n = static_cast<int>(p / (static_cast<long long>(W) * H));
        const float4 g = ld4(dy + p * Cout + c4 * 4);
        const float* xp = x + (static_cast<size_t>(n) * Cin + ci) * H * W;
#pragma unroll
        for (int t = 0; t < 9; ++t) {
          const int hh = hq + t / 3 - 1, ww = wq + t % 3 - 1;
          if (hh < 0 || hh >= H || ww < 0 || ww >= W) continue;
          const float xv = __ldg(xp + static_cast<size_t>(hh) * W + ww);
          acc[t][0] = fmaf(xv, g.x, acc[t][0]); acc[t][1] = fmaf(xv, g.y, acc[t][1]);
          acc[t][2] = fmaf(xv, g.z, acc[t][2]); acc[t][3] = fmaf(xv, g.w, acc[t][3]);
        }
      }
    }
    fold_channels<9>(acc, lane, lanes, c4, c4s, Cout,
                     partials + (static_cast<size_t>(blockIdx.x) * Cin + ci) * 9 * Cout, smem);
  }
}
// grad (Cout, Cin, 3, 3) += sum over rows of partials[row][ci][t][co]
__global__ void f32_conv_in_wgrad_fold_kernel(const double* __restrict__ partials, int rows, int Cin, int Cout, float* grad) {
  pdl_trigger();
  pdl_wait();
  const int total = Cin * 9 * Cout;
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= total) return;
  double s = 0.0;
  for (int r = 0; r < rows; ++r) s += partials[static_cast<size_t>(r) * total + e];
  const int co = e % Cout, t = (e / Cout) % 9, ci = e / (9 * Cout);
  grad[(static_cast<size_t>(co) * Cin + ci) * 9 + t] += static_cast<float>(s);
}

// ---- 3xTF32: operand split and weight packs ---------------------------------------------------------------------
// out (pixels, 2*(C0+C1)) = [hi(x0) | hi(x1) | lo(x0) | lo(x1)], hi = tf32(x), lo = tf32(x - hi)
__global__ void __launch_bounds__(kFT)
f32_split_tf32_kernel(const float* __restrict__ x0, int ld0, int C0, const float* __restrict__ x1, int ld1, int C1,
                      float* __restrict__ out, long long pixels) {
  pdl_trigger();
  pdl_wait();
  const int C = C0 + C1, c4s = C / 4;
  const long long total = pixels * c4s;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i % c4s) * 4;
    const long long p = i / c4s;
    const float4 v = (c < C0) ? ld4(x0 + p * ld0 + c) : ld4(x1 + p * ld1 + (c - C0));
    float4 h, l;
    h.x = tf32_round(v.x); h.y = tf32_round(v.y); h.z = tf32_round(v.z); h.w = tf32_round(v.w);
    l.x = tf32_round(v.x - h.x); l.y = tf32_round(v.y - h.y); l.z = tf32_round(v.z - h.z); l.w = tf32_round(v.w - h.w);
    st4(out + p * 2 * C + c, h);
    st4(out + p * 2 * C + C + c, l);
  }
}

// OIHW fp32 -> 3xTF32 pack (rows, taps, 3*K): per tap [w_hi | w_hi | w_lo] along K.
// forward: rows = Cout, K = Cin; data gradient (dgrad != 0): rows = Cin, K = Cout, taps flipped.
__global__ void f32_pack_weight3_kernel(const float* __restrict__ w, float* __restrict__ out, int Cout, int Cin, int taps,
                                        int dgrad) {
  pdl_trigger();
  pdl_wait();
  const int R = dgrad ? Cin : Cout, Kc = dgrad ? Cout : Cin;
  const long long total = static_cast<long long>(R) * taps * Kc;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int k = static_cast<int>(i % Kc);
    const int t = static_cast<int>((i / Kc) % taps);
    const int r = static_cast<int>(i / (static_cast<long long>(Kc) * taps));
    const float v = dgrad ? __ldg(w + (static_cast<size_t>(k) * Cin + r) * taps + (taps - 1 - t))
                          : __ldg(w + (static_cast<size_t>(r) * Cin + k) * taps + t);
    const float hi = tf32_round(v), lo = tf32_round(v - hi);
    float* o = out + (static_cast<size_t>(r) * taps + t) * 3 * Kc;
    o[k] = hi;
    o[Kc + k] = hi;
    o[2 * Kc + k] = lo;
  }
}

// bilinear (hin,win) -> (hu,wu), centred inside a zero (Ho,Wo) canvas; unrounded (fp32_eval.cu's rounds to TF32)
__global__ void __launch_bounds__(kFT)
f32_upsample_fwd_kernel(const float* __restrict__ in, float* __restrict__ out, int N, int hin, int win, int hu, int wu,
                        int Ho, int Wo, int C, float rh, float rw) {
  pdl_trigger();
  pdl_wait();
  const int c4s = C / 4;
  const int pt = (Ho - hu) / 2, pl = (Wo - wu) / 2;
  const long long total = static_cast<long long>(N) * Ho * Wo * c4s;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i % c4s) * 4;
    const long long pix = i / c4s;
    const int wo = static_cast<int>(pix % Wo), ho = static_cast<int>((pix / Wo) % Ho);
    const int n = static_cast<int>(pix / (static_cast<long long>(Wo) * Ho));
    const int uh = ho - pt, uw = wo - pl;
    float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
    if (uh >= 0 && uh < hu && uw >= 0 && uw < wu) {
      int h0, h1, w0, w1;
      float a0, a1, b0, b1;
      src_index(rh, uh, hin, h0, h1, a0, a1);
      src_index(rw, uw, win, w0, w1, b0, b1);
      const float* base = in + static_cast<size_t>(n) * hin * win * C + c;
      const float4 v00 = ld4(base + (static_cast<size_t>(h0) * win + w0) * C), v01 = ld4(base + (static_cast<size_t>(h0) * win + w1) * C);
      const float4 v10 = ld4(base + (static_cast<size_t>(h1) * win + w0) * C), v11 = ld4(base + (static_cast<size_t>(h1) * win + w1) * C);
      o.x = a0 * (b0 * v00.x + b1 * v01.x) + a1 * (b0 * v10.x + b1 * v11.x);
      o.y = a0 * (b0 * v00.y + b1 * v01.y) + a1 * (b0 * v10.y + b1 * v11.y);
      o.z = a0 * (b0 * v00.z + b1 * v01.z) + a1 * (b0 * v10.z + b1 * v11.z);
      o.w = a0 * (b0 * v00.w + b1 * v01.w) + a1 * (b0 * v10.w + b1 * v11.w);
    }
    st4(out + pix * C + c, o);
  }
}

// ---- operand split for the weight gradient ----------------------------------------------------------------------
__global__ void __launch_bounds__(kFT)
f32_split_bf16_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo, long long n4) {
  pdl_trigger();
  pdl_wait();
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n4; i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float4 v = ld4(x + i * 4);
    const float vv[4] = {v.x, v.y, v.z, v.w};
    float h[4], l[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      h[k] = bf16_round(vv[k]);
      l[k] = vv[k] - h[k];
    }
    uint2 oh, ol;
    oh.x = pack_bf16x2(h[0], h[1]); oh.y = pack_bf16x2(h[2], h[3]);
    ol.x = pack_bf16x2(l[0], l[1]); ol.y = pack_bf16x2(l[2], l[3]);
    *reinterpret_cast<uint2*>(hi + i * 4) = oh;
    *reinterpret_cast<uint2*>(lo + i * 4) = ol;
  }
}

static float ratio_f(int in, int out) { return out > 1 ? static_cast<float>(in - 1) / static_cast<float>(out - 1) : 0.f; }
static int elem_grid(long long items) { return stream_grid(items, kFT, num_sms(), 8); }

}  // namespace ub2

using namespace ub2;

extern "C" {

#define F32_STREAM static_cast<cudaStream_t>(stream)
#define F32_DONE return static_cast<int>(cudaGetLastError())

// Every entry point checks its arguments before it touches the device: a count <= 0, a channel count that is not a
// multiple of 4, a channel stride below its channel count or a NULL pointer the kernel reads or writes returns
// UB2_ERR_SHAPE; a channel stride that is not a multiple of 4, or a pointer that a float4 (uchar4, double) access
// cannot use, UB2_ERR_ALIGN; `rows` other than the matching *_rows query, UB2_ERR_WORKSPACE.
static bool c4(int C) { return C > 0 && C % 4 == 0; }
static bool al16(const void* p) { return aligned_to(p, 16); }
static bool al8(const void* p) { return aligned_to(p, 8); }
static bool al4(const void* p) { return aligned_to(p, 4); }

int ub2_f32_channel_rows(long long pixels, int C) {
  if (!c4(C) || C > 4 * kFT || pixels <= 0) return UB2_ERR_SHAPE;
  return chan_grid(pixels, C);
}

int ub2_f32_channel_stats(const float* x, int ld, long long pixels, int C, double* partials, int rows, void* stream) {
  if (x == nullptr || partials == nullptr || !c4(C) || C > 4 * kFT || ld < C || pixels <= 0) return UB2_ERR_SHAPE;
  if (ld % 4 != 0 || !al16(x) || !al8(partials)) return UB2_ERR_ALIGN;
  if (rows != chan_grid(pixels, C)) return UB2_ERR_WORKSPACE;
  launch(f32_channel_stats_kernel, rows, chan_lanes(C) * (C / 4), 0, F32_STREAM, x, ld, pixels, C, partials);
  F32_DONE;
}

int ub2_f32_scalar_rows(long long n) { return n > 0 ? elem_grid(n) : UB2_ERR_SHAPE; }

int ub2_f32_scalar_stats(const float* x, long long n, double* partials, int rows, void* stream) {
  if (x == nullptr || partials == nullptr || n <= 0) return UB2_ERR_SHAPE;
  if (!al4(x) || !al8(partials)) return UB2_ERR_ALIGN;
  if (rows != elem_grid(n)) return UB2_ERR_WORKSPACE;
  launch(f32_scalar_stats_kernel, rows, kFT, 0, F32_STREAM, x, n, partials);
  F32_DONE;
}

int ub2_f32_affine_act(const float* y, const float* scale, const float* shift, float* out, long long pixels, int C,
                       int relu, void* stream) {
  if (y == nullptr || scale == nullptr || shift == nullptr || out == nullptr || !c4(C) || pixels <= 0) return UB2_ERR_SHAPE;
  if (!al16(y) || !al16(scale) || !al16(shift) || !al16(out)) return UB2_ERR_ALIGN;
  launch(f32_affine_act_kernel, elem_grid(pixels * (C / 4)), kFT, 0, F32_STREAM, y, scale, shift, out, pixels, C, relu);
  F32_DONE;
}

int ub2_f32_maxpool_idx(const float* a, float* p, unsigned char* idx, int N, int H, int W, int C, void* stream) {
  if (a == nullptr || p == nullptr || idx == nullptr || !c4(C) || N <= 0 || H < 2 || W < 2) return UB2_ERR_SHAPE;
  if (!al16(a) || !al16(p) || !al4(idx)) return UB2_ERR_ALIGN;
  launch(f32_maxpool_idx_kernel, elem_grid(static_cast<long long>(N) * (H / 2) * (W / 2) * (C / 4)), kFT, 0, F32_STREAM, a, p, idx, N,
         H, W, C);
  F32_DONE;
}

// The gradient sources of the two BatchNorm-backward passes: dA (channel stride ld_da), dP routed through idx, or both.
static int act_bwd_args(const float* dA, int ld_da, const float* dP, const unsigned char* idx, const float* y, int N, int H,
                        int W, int C) {
  if (y == nullptr || !c4(C) || N <= 0 || H <= 0 || W <= 0) return UB2_ERR_SHAPE;
  if ((dA == nullptr && dP == nullptr) || (dP != nullptr && idx == nullptr) || (dA != nullptr && ld_da < C)) return UB2_ERR_SHAPE;
  if ((dA != nullptr && ld_da % 4 != 0) || !al16(dA) || !al16(dP) || !al4(idx) || !al16(y)) return UB2_ERR_ALIGN;
  return UB2_OK;
}

int ub2_f32_act_bwd_reduce(const float* dA, int ld_da, const float* dP, const unsigned char* idx, const float* y,
                           const float* scale, const float* shift, double* partials, int rows, int N, int H, int W, int C,
                           int relu, void* stream) {
  const int rc = act_bwd_args(dA, ld_da, dP, idx, y, N, H, W, C);
  if (rc != UB2_OK) return rc;
  if (scale == nullptr || shift == nullptr || partials == nullptr || C > 4 * kFT) return UB2_ERR_SHAPE;
  if (!al16(scale) || !al16(shift) || !al8(partials)) return UB2_ERR_ALIGN;
  const long long pixels = static_cast<long long>(N) * H * W;
  if (rows != chan_grid(pixels, C)) return UB2_ERR_WORKSPACE;
  launch(f32_act_bwd_reduce_kernel, rows, chan_lanes(C) * (C / 4), 0, F32_STREAM, dA, ld_da, dP, idx, y, scale, shift, partials, N, H,
         W, C, relu);
  F32_DONE;
}

int ub2_f32_act_bwd_apply(const float* dA, int ld_da, const float* dP, const unsigned char* idx, const float* y,
                          const float* scale, const float* shift, const float* coef, float* dy, int N, int H, int W, int C,
                          int relu, void* stream) {
  const int rc = act_bwd_args(dA, ld_da, dP, idx, y, N, H, W, C);
  if (rc != UB2_OK) return rc;
  if (coef == nullptr || dy == nullptr || (relu && (scale == nullptr || shift == nullptr))) return UB2_ERR_SHAPE;
  if (!al16(scale) || !al16(shift) || !al16(coef) || !al16(dy)) return UB2_ERR_ALIGN;
  launch(f32_act_bwd_apply_kernel, elem_grid(static_cast<long long>(N) * H * W * (C / 4)), kFT, 0, F32_STREAM, dA, ld_da, dP, idx, y,
         scale, shift, coef, dy, N, H, W, C, relu);
  F32_DONE;
}

// (hin,win) resampled to (hu,wu) inside an (Ho,Wo) canvas
static bool resample_geom_ok(int N, int hin, int win, int hu, int wu, int Ho, int Wo, int C) {
  return c4(C) && N > 0 && hin > 0 && win > 0 && hu > 0 && wu > 0 && Ho >= hu && Wo >= wu;
}

int ub2_f32_upsample_bwd(const float* dout, int ld_dout, float* din, int N, int hin, int win, int hu, int wu, int Ho, int Wo,
                         int C, void* stream) {
  if (dout == nullptr || din == nullptr || !resample_geom_ok(N, hin, win, hu, wu, Ho, Wo, C) || ld_dout < C) return UB2_ERR_SHAPE;
  if (ld_dout % 4 != 0 || !al16(dout) || !al16(din)) return UB2_ERR_ALIGN;
  launch(f32_upsample_bwd_kernel, elem_grid(static_cast<long long>(N) * hin * win * (C / 4)), kFT, 0, F32_STREAM, dout, ld_dout, din, N,
         hin, win, hu, wu, Ho, Wo, C, ratio_f(hin, hu), ratio_f(win, wu));
  F32_DONE;
}

int ub2_f32_gate_psi(const float* u, const float* xp, const float* sg, const float* hg, const float* sx, const float* hx,
                     const float* wpsi, float* psi_raw, long long pixels, int Ci, void* stream) {
  if (u == nullptr || xp == nullptr || sg == nullptr || hg == nullptr || sx == nullptr || hx == nullptr || wpsi == nullptr ||
      psi_raw == nullptr || !c4(Ci) || pixels <= 0)
    return UB2_ERR_SHAPE;
  if (!al16(u) || !al16(xp) || !al16(sg) || !al16(hg) || !al16(sx) || !al16(hx) || !al16(wpsi) || !al4(psi_raw)) return UB2_ERR_ALIGN;
  launch(f32_gate_psi_kernel, stream_grid(pixels, kFT / 32, num_sms(), 8), kFT, 0, F32_STREAM, u, xp, sg, hg, sx, hx, wpsi, psi_raw,
         pixels, Ci);
  F32_DONE;
}

int ub2_f32_gate_apply(const float* psi_raw, const float* spsi, const float* hpsi, const float* x, float* out, float* a_out,
                       long long pixels, int Cx, void* stream) {
  if (psi_raw == nullptr || spsi == nullptr || hpsi == nullptr || x == nullptr || out == nullptr || !c4(Cx) || pixels <= 0)
    return UB2_ERR_SHAPE;
  if (!al16(x) || !al16(out) || !al4(a_out)) return UB2_ERR_ALIGN;
  launch(f32_gate_apply_kernel, elem_grid(pixels * (Cx / 4)), kFT, 0, F32_STREAM, psi_raw, spsi, hpsi, x, out, a_out, pixels, Cx);
  F32_DONE;
}

int ub2_f32_gate_rows(long long pixels) { return pixels > 0 ? stream_grid(pixels, kFT / 32, num_sms(), 4) : UB2_ERR_SHAPE; }

int ub2_f32_gate_bwd_a(const float* dout, int ld_do, const float* x, const float* a, const float* psi_raw, float* dx,
                       float* dpsin, double* partials, int rows, long long pixels, int Cx, void* stream) {
  if (dout == nullptr || x == nullptr || a == nullptr || psi_raw == nullptr || dx == nullptr || dpsin == nullptr ||
      partials == nullptr || !c4(Cx) || pixels <= 0 || ld_do < Cx)
    return UB2_ERR_SHAPE;
  if (ld_do % 4 != 0 || !al16(dout) || !al16(x) || !al16(dx) || !al8(partials)) return UB2_ERR_ALIGN;
  if (rows != stream_grid(pixels, kFT / 32, num_sms(), 4)) return UB2_ERR_WORKSPACE;
  launch(f32_gate_bwd_a_kernel, rows, kFT, 0, F32_STREAM, dout, ld_do, x, a, psi_raw, dx, dpsin, partials, pixels, Cx);
  F32_DONE;
}

int ub2_f32_gate_bwd_s(const float* dpsin, const float* psi_raw, const float* coef_psi, const float* u, const float* xp,
                       const float* sg, const float* hg, const float* sx, const float* hx, const float* wpsi, float* ds,
                       double* partials, int rows, long long pixels, int Ci, void* stream) {
  if (dpsin == nullptr || psi_raw == nullptr || coef_psi == nullptr || u == nullptr || xp == nullptr || sg == nullptr ||
      hg == nullptr || sx == nullptr || hx == nullptr || wpsi == nullptr || ds == nullptr || partials == nullptr ||
      !c4(Ci) || Ci > 128 * kGI || pixels <= 0)
    return UB2_ERR_SHAPE;
  if (!al16(u) || !al16(xp) || !al16(sg) || !al16(hg) || !al16(sx) || !al16(hx) || !al16(wpsi) || !al16(ds) || !al8(partials))
    return UB2_ERR_ALIGN;
  if (rows != stream_grid(pixels, kFT / 32, num_sms(), 4)) return UB2_ERR_WORKSPACE;
  const size_t smem = static_cast<size_t>(kFT / 32) * 4 * Ci * sizeof(float);
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(f32_gate_bwd_s_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024);
    if (e != cudaSuccess) return static_cast<int>(e);
  }
  launch(f32_gate_bwd_s_kernel, rows, kFT, smem, F32_STREAM, dpsin, psi_raw, coef_psi, u, xp, sg, hg, sx, hx, wpsi, ds, partials,
         pixels, Ci);
  F32_DONE;
}

int ub2_f32_gate_bwd_xg(const float* ds, const float* xp, const float* u, const float* coef, float* dxp, float* du,
                        long long pixels, int Ci, void* stream) {
  if (ds == nullptr || xp == nullptr || u == nullptr || coef == nullptr || dxp == nullptr || du == nullptr || !c4(Ci) ||
      pixels <= 0)
    return UB2_ERR_SHAPE;
  if (!al16(ds) || !al16(xp) || !al16(u) || !al16(coef) || !al16(dxp) || !al16(du)) return UB2_ERR_ALIGN;
  launch(f32_gate_bwd_xg_kernel, elem_grid(pixels * (Ci / 4)), kFT, 0, F32_STREAM, ds, xp, u, coef, dxp, du, pixels, Ci);
  F32_DONE;
}

int ub2_f32_outc_rows(int N, int H, int W) {
  if (N <= 0 || H <= 0 || W <= 0) return UB2_ERR_SHAPE;
  return stream_grid(static_cast<long long>(N) * H * W, kFT / 32, num_sms(), 2);
}

int ub2_f32_outc_bwd(const float* dlogits, const float* a, const float* w, float* da, double* partials, int rows, float* dw,
                     float* db, int N, int H, int W, int C, int K, void* stream) {
  if (dlogits == nullptr || a == nullptr || w == nullptr || partials == nullptr || !c4(C) || K < 1 || K > 8 || N <= 0 ||
      H <= 0 || W <= 0)
    return UB2_ERR_SHAPE;
  if (!al4(dlogits) || !al16(a) || !al16(w) || !al16(da) || !al8(partials) || !al4(dw) || !al4(db)) return UB2_ERR_ALIGN;
  if (rows != ub2_f32_outc_rows(N, H, W)) return UB2_ERR_WORKSPACE;
  const int cols = K * C + K;
  const size_t smem = static_cast<size_t>(kFT / 32) * cols * sizeof(float);
  if (smem > 48 * 1024) return UB2_ERR_SHAPE;
  launch(f32_outc_bwd_kernel, rows, kFT, smem, F32_STREAM, dlogits, a, w, da, partials, N, H, W, C, K);
  if (dw != nullptr)
    launch(f32_cols_fold_kernel, (K * C + 255) / 256, 256, 0, F32_STREAM, static_cast<const double*>(partials), rows, cols, 0, K * C, dw);
  if (db != nullptr)
    launch(f32_cols_fold_kernel, 1, 256, 0, F32_STREAM, static_cast<const double*>(partials), rows, cols, K * C, K, db);
  F32_DONE;
}

int ub2_f32_conv_in_raw(const float* x, const float* w, float* out, int N, int Cin, int H, int W, int Cout, void* stream) {
  if (x == nullptr || w == nullptr || out == nullptr || !c4(Cout) || Cin <= 0 || N <= 0 || H <= 0 || W <= 0) return UB2_ERR_SHAPE;
  if (!al4(x) || !al4(w) || !al16(out)) return UB2_ERR_ALIGN;
  launch(f32_conv_in_raw_kernel, elem_grid(static_cast<long long>(N) * H * W * (Cout / 4)), kFT, 0, F32_STREAM, x, w, out, N, Cin, H, W,
         Cout);
  F32_DONE;
}

int ub2_f32_conv_in_wgrad(const float* x, const float* dy, double* partials, int rows, float* grad, int N, int Cin, int H,
                          int W, int Cout, void* stream) {
  if (x == nullptr || dy == nullptr || partials == nullptr || grad == nullptr || !c4(Cout) || Cout > 4 * kFT || Cin <= 0 ||
      N <= 0 || H <= 0 || W <= 0)
    return UB2_ERR_SHAPE;
  if (!al4(x) || !al16(dy) || !al8(partials) || !al4(grad)) return UB2_ERR_ALIGN;
  const long long pixels = static_cast<long long>(N) * H * W;
  if (rows != chan_grid(pixels, Cout)) return UB2_ERR_WORKSPACE;
  launch(f32_conv_in_wgrad_kernel, rows, chan_lanes(Cout) * (Cout / 4), 0, F32_STREAM, x, dy, partials, N, Cin, H, W, Cout);
  const int total = Cin * 9 * Cout;
  launch(f32_conv_in_wgrad_fold_kernel, (total + 255) / 256, 256, 0, F32_STREAM, static_cast<const double*>(partials), rows, Cin, Cout,
         grad);
  F32_DONE;
}

int ub2_f32_split_bf16(const float* x, void* hi, void* lo, long long n, void* stream) {
  if (x == nullptr || hi == nullptr || lo == nullptr || n <= 0 || n % 4 != 0) return UB2_ERR_SHAPE;
  if (!al16(x) || !al8(hi) || !al8(lo)) return UB2_ERR_ALIGN;
  launch(f32_split_bf16_kernel, elem_grid(n / 4), kFT, 0, F32_STREAM, x, static_cast<__nv_bfloat16*>(hi), static_cast<__nv_bfloat16*>(lo),
         n / 4);
  F32_DONE;
}

int ub2_f32_split_tf32(const float* x0, int ld0, int C0, const float* x1, int ld1, int C1, float* out, long long pixels,
                       void* stream) {
  if (x0 == nullptr || out == nullptr || !c4(C0) || ld0 < C0 || C1 < 0 || C1 % 4 != 0 || pixels <= 0) return UB2_ERR_SHAPE;
  if (C1 > 0 && (x1 == nullptr || ld1 < C1)) return UB2_ERR_SHAPE;
  if (ld0 % 4 != 0 || (C1 > 0 && ld1 % 4 != 0) || !al16(x0) || !al16(x1) || !al16(out)) return UB2_ERR_ALIGN;
  launch(f32_split_tf32_kernel, elem_grid(pixels * ((C0 + C1) / 4)), kFT, 0, F32_STREAM, x0, ld0, C0, x1, ld1, C1, out, pixels);
  F32_DONE;
}

int ub2_f32_pack_weight3(const float* w, float* out, int Cout, int Cin, int taps, int dgrad, void* stream) {
  if (w == nullptr || out == nullptr || Cout <= 0 || Cin <= 0 || taps <= 0) return UB2_ERR_SHAPE;
  if (!al4(w) || !al4(out)) return UB2_ERR_ALIGN;
  launch(f32_pack_weight3_kernel, elem_grid(static_cast<long long>(Cout) * Cin * taps), kFT, 0, F32_STREAM, w, out, Cout, Cin, taps, dgrad);
  F32_DONE;
}

int ub2_f32_upsample_fwd(const float* in, float* out, int N, int hin, int win, int hu, int wu, int Ho, int Wo, int C,
                         void* stream) {
  if (in == nullptr || out == nullptr || !resample_geom_ok(N, hin, win, hu, wu, Ho, Wo, C)) return UB2_ERR_SHAPE;
  if (!al16(in) || !al16(out)) return UB2_ERR_ALIGN;
  launch(f32_upsample_fwd_kernel, elem_grid(static_cast<long long>(N) * Ho * Wo * (C / 4)), kFT, 0, F32_STREAM, in, out, N, hin, win, hu,
         wu, Ho, Wo, C, ratio_f(hin, hu), ratio_f(win, wu));
  F32_DONE;
}

}  // extern "C"
