// ConvTranspose2d(C, C/2, kernel_size = 2, stride = 2) + F.pad to the skip size (unet/models/layers.py:81,
// :98-102, :217-221).  Because kernel == stride the output pixels of a transposed convolution do not
// overlap: it is a 1x1 convolution to 4*Cout channels — row (i, j, co) of the reshaped weight, done on the
// tensor cores by ub2_conv_fwd with the bias in its epilogue — followed by a pixel shuffle
//   out[n, 2y+i + py, 2x+j + px, co] = t[n, y, x, (i*2+j)*Cout + co]
// with the (possibly odd) padding (py, px) of F.pad and zeros elsewhere.  These kernels are that shuffle,
// its transpose, and the bias gradient (the per-channel sum of the un-padded output gradient), so that no
// ATen permute / pad / contiguous / sum kernel runs on the path.  Bandwidth bound: one 128-bit vector per
// thread and trip, reads and writes coalesced along the channel axis.  The kernels are templated on the element
// type: bf16 (8 channels per vector) for the default path, fp32 (4 channels) for fp32 / TF32 mode, where the
// 1x1 convolution is ub2_conv_fwd_tf32 on the exact fp32 weight of ub2_f32_pack_convt_weight.
#include "launch.cuh"
#include "../../include/unetb200.h"
#include "conv.h"
#include "vec.cuh"

namespace ub2 {

struct ShufGeom {
  int N, h, w, C, cgs, Ho, Wo, py, px;
};

// 16-byte vectors: V channels of T
template <typename T> struct Vec16 { static constexpr int V = 16 / static_cast<int>(sizeof(T)); };
__device__ __forceinline__ void unpack_vec(const uint4& u, float (&f)[8]) {
  const F8 r = unpack8(u);
#pragma unroll
  for (int k = 0; k < 8; ++k) f[k] = r.v[k];
}
__device__ __forceinline__ void unpack_vec(const uint4& u, float (&f)[4]) {
  f[0] = __uint_as_float(u.x); f[1] = __uint_as_float(u.y); f[2] = __uint_as_float(u.z); f[3] = __uint_as_float(u.w);
}

// grid-stride over output vectors (n, Y, X, cg)
template <typename T>
__global__ void __launch_bounds__(256)
shuffle2x2_fwd_kernel(const T* __restrict__ t, int ld_t, T* __restrict__ out, int ld_out, ShufGeom g) {
  constexpr int V = Vec16<T>::V;
  pdl_trigger();
  pdl_wait();
  const long long total = static_cast<long long>(g.N) * g.Ho * g.Wo * g.cgs;
  for (long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int cg = static_cast<int>(idx % g.cgs);
    long long r = idx / g.cgs;
    const int X = static_cast<int>(r % g.Wo);
    r /= g.Wo;
    const int Y = static_cast<int>(r % g.Ho);
    const int n = static_cast<int>(r / g.Ho);
    const int yy = Y - g.py, xx = X - g.px;
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (yy >= 0 && yy < 2 * g.h && xx >= 0 && xx < 2 * g.w) {
      const size_t pix = (static_cast<size_t>(n) * g.h + (yy >> 1)) * g.w + (xx >> 1);
      v = ld_stream16(t + pix * ld_t + (((yy & 1) * 2 + (xx & 1)) * g.C) + cg * V);
    }
    *reinterpret_cast<uint4*>(out + ((static_cast<size_t>(n) * g.Ho + Y) * g.Wo + X) * ld_out + cg * V) = v;
  }
}

// Transpose: dt[n, y, x, (i*2+j)*C + co] = dout[n, 2y+i+py, 2x+j+px, co]; also per-block partial sums of the
// gathered gradient per output channel co (all four sub-positions) for the bias gradient.
// blockDim.x = lanes * cgs: a thread's channel group is fixed, so its partial sums stay in registers (fp32 per
// thread, fp64 per block).
template <typename T>
__global__ void __launch_bounds__(256)
shuffle2x2_bwd_kernel(const T* __restrict__ dout, int ld_dout, T* __restrict__ dt, int ld_dt,
                      double* __restrict__ partials, ShufGeom g) {
  constexpr int V = Vec16<T>::V;
  pdl_trigger();
  pdl_wait();
  __shared__ float smem[256 * V];
  const int lanes = blockDim.x / g.cgs;
  const int lane = threadIdx.x / g.cgs;
  const int cg = threadIdx.x % g.cgs;
  float acc[V];
#pragma unroll
  for (int k = 0; k < V; ++k) acc[k] = 0.f;
  const long long total = static_cast<long long>(g.N) * g.h * g.w * 4;   // (low-res pixel, sub-position)
  if (lane < lanes) {
    for (long long it = static_cast<long long>(blockIdx.x) * lanes + lane; it < total;
         it += static_cast<long long>(gridDim.x) * lanes) {
      const int sub = static_cast<int>(it & 3);
      const long long pix = it >> 2;
      const int x = static_cast<int>(pix % g.w);
      const int y = static_cast<int>((pix / g.w) % g.h);
      const int n = static_cast<int>(pix / (static_cast<long long>(g.w) * g.h));
      const int Y = 2 * y + (sub >> 1) + g.py, X = 2 * x + (sub & 1) + g.px;
      const uint4 v = ld_stream16(dout + ((static_cast<size_t>(n) * g.Ho + Y) * g.Wo + X) * ld_dout + cg * V);
      *reinterpret_cast<uint4*>(dt + static_cast<size_t>(pix) * ld_dt + sub * g.C + cg * V) = v;
      float f[V];
      unpack_vec(v, f);
#pragma unroll
      for (int k = 0; k < V; ++k) acc[k] += f[k];
    }
  }
  if (partials == nullptr) return;
#pragma unroll
  for (int k = 0; k < V; ++k) smem[threadIdx.x * V + k] = (lane < lanes) ? acc[k] : 0.f;
  __syncthreads();
  for (int c = threadIdx.x; c < g.C; c += blockDim.x) {
    const int cgc = c / V, k = c % V;
    double s = 0.0;
    for (int l = 0; l < lanes; ++l) s += static_cast<double>(smem[(l * g.cgs + cgc) * V + k]);
    partials[static_cast<size_t>(blockIdx.x) * g.C + c] = s;
  }
}

// dbias[c] += sum over rows of partials[row][c]   (blockDim = (8, 128), see rows_sum_wide)
__global__ void shuffle_bias_finalize_kernel(const double* __restrict__ partials, int rows, int C, float* dbias) {
  pdl_trigger();
  pdl_wait();
  __shared__ double smem[128 * 9];
  const int c = blockIdx.x * 8 + threadIdx.x;
  double s[1];
  rows_sum_wide<1>(partials, rows, C, c, s, smem);
  if (threadIdx.y == 0 && c < C) dbias[c] += static_cast<float>(s[0]);
}


__device__ __forceinline__ void to_elem(float v, __nv_bfloat16* p) { *p = __float2bfloat16_rn(v); }
__device__ __forceinline__ void to_elem(float v, float* p) { *p = v; }

// (Cin, Cout, 2, 2) fp32 parameter -> the 1x1-convolution packs: forward (4*Cout, Cin) with row (i*2+j)*Cout + co,
// data gradient (Cin, 4*Cout), and the epilogue vectors scale = 1, shift = bias tiled 4x.  T = bf16 rounds the
// weight (the default path); T = float copies it exactly (fp32 mode, whose TF32 packs are made from it).
template <typename T>
__global__ void pack_convt_weight_kernel(const float* __restrict__ w, const float* __restrict__ bias,
                                         T* __restrict__ fwd, T* __restrict__ dg,
                                         float* __restrict__ scale4, float* __restrict__ shift4, int Cin, int Cout) {
  pdl_trigger();
  pdl_wait();
  const long long total = static_cast<long long>(Cin) * Cout * 4;
  for (long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    // idx walks the forward pack (row r = (sub, co), column ci): coalesced writes of the larger pack
    const int ci = static_cast<int>(idx % Cin);
    const int r = static_cast<int>(idx / Cin);
    const int sub = r / Cout, co = r % Cout;
    const float v = __ldg(w + (static_cast<size_t>(ci) * Cout + co) * 4 + sub);
    if (fwd != nullptr) to_elem(v, fwd + idx);
    if (dg != nullptr) to_elem(v, dg + static_cast<size_t>(ci) * 4 * Cout + r);
    if (ci == 0 && scale4 != nullptr) {
      scale4[r] = 1.f;
      shift4[r] = bias != nullptr ? __ldg(bias + co) : 0.f;
    }
  }
}

// grad (Cin, Cout, 2, 2) (+)= sum over splits of partial[s][ci][(i*2+j)*Cout + co]
__global__ void convt_wgrad_reduce_kernel(const float* __restrict__ partial, int splits, int Cin, int Cout,
                                          float* __restrict__ grad, int accumulate) {
  pdl_trigger();
  pdl_wait();
  const long long total = static_cast<long long>(Cin) * Cout * 4;
  for (long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    // idx walks the partial's layout (ci, sub, co): coalesced reads of the larger operand
    const int co = static_cast<int>(idx % Cout);
    const int sub = static_cast<int>((idx / Cout) & 3);
    const int ci = static_cast<int>(idx / (4LL * Cout));
    float s = 0.f;
    for (int k = 0; k < splits; ++k) s += __ldg(partial + static_cast<size_t>(k) * total + idx);   // fixed order
    float* dst = grad + (static_cast<size_t>(ci) * Cout + co) * 4 + sub;
    *dst = accumulate ? *dst + s : s;
  }
}

static int shuf_geom(ShufGeom* g, int N, int h, int w, int C, int Ho, int Wo, int V = 8) {
  if (N <= 0 || h <= 0 || w <= 0 || C <= 0 || C % V != 0 || Ho < 2 * h || Wo < 2 * w) return UB2_ERR_SHAPE;
  g->N = N; g->h = h; g->w = w; g->C = C; g->cgs = C / V; g->Ho = Ho; g->Wo = Wo;
  g->py = (Ho - 2 * h) / 2;    // F.pad(x1, [dx // 2, dx - dx // 2, dy // 2, dy - dy // 2])
  g->px = (Wo - 2 * w) / 2;
  return 0;
}
static int shuf_bwd_grid(const ShufGeom& g) {
  const int lanes = 256 / g.cgs > 0 ? 256 / g.cgs : 1;
  return stream_grid(static_cast<long long>(g.N) * g.h * g.w * 4, lanes, num_sms(), 4);
}
static bool al16(const void* p) { return aligned_to(p, 16); }

}  // namespace ub2

using namespace ub2;

extern "C" {

int ub2_shuffle2x2_fwd(const void* t, int ld_t, void* out, int ld_out, int N, int h, int w, int C, int Ho, int Wo,
                       void* stream) {
  ShufGeom g;
  int rc = shuf_geom(&g, N, h, w, C, Ho, Wo);
  if (rc) return rc;
  if (ld_t % 8 || ld_out % 8) return UB2_ERR_ALIGN;
  const long long total = static_cast<long long>(N) * Ho * Wo * g.cgs;
  launch(shuffle2x2_fwd_kernel<__nv_bfloat16>, stream_grid(total, 256, num_sms(), 8), 256, 0, static_cast<cudaStream_t>(stream),
         static_cast<const __nv_bfloat16*>(t), ld_t, static_cast<__nv_bfloat16*>(out), ld_out, g);
  return static_cast<int>(cudaGetLastError());
}

int ub2_shuffle2x2_rows(int N, int h, int w, int C, int Ho, int Wo) {
  ShufGeom g;
  int rc = shuf_geom(&g, N, h, w, C, Ho, Wo);
  if (rc) return rc;
  if (g.cgs > 256) return UB2_ERR_SHAPE;
  return shuf_bwd_grid(g);
}

int ub2_shuffle2x2_bwd(const void* dout, int ld_dout, void* dt, int ld_dt, double* partials, int rows, float* dbias,
                       int N, int h, int w, int C, int Ho, int Wo, void* stream) {
  ShufGeom g;
  int rc = shuf_geom(&g, N, h, w, C, Ho, Wo);
  if (rc) return rc;
  if (g.cgs > 256) return UB2_ERR_SHAPE;
  if (ld_dout % 8 || ld_dt % 8) return UB2_ERR_ALIGN;
  const int grid = shuf_bwd_grid(g);
  if (partials != nullptr && rows != grid) return UB2_ERR_WORKSPACE;
  const int lanes = 256 / g.cgs;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  launch(shuffle2x2_bwd_kernel<__nv_bfloat16>, grid, lanes * g.cgs, 0, s, static_cast<const __nv_bfloat16*>(dout), ld_dout,
         static_cast<__nv_bfloat16*>(dt), ld_dt, partials, g);
  if (partials != nullptr && dbias != nullptr)
    launch(shuffle_bias_finalize_kernel, (C + 7) / 8, dim3(8, 128), 0, s, static_cast<const double*>(partials), grid, C, dbias);
  return static_cast<int>(cudaGetLastError());
}

int ub2_pack_convt_weight(const float* w, const float* bias, void* fwd, void* dg, float* scale4, float* shift4,
                          int Cin, int Cout, void* stream) {
  if (Cin <= 0 || Cout <= 0) return UB2_ERR_SHAPE;
  const long long total = static_cast<long long>(Cin) * Cout * 4;
  launch(pack_convt_weight_kernel<__nv_bfloat16>, stream_grid(total, 256, num_sms(), 8), 256, 0, static_cast<cudaStream_t>(stream), w, bias,
         static_cast<__nv_bfloat16*>(fwd), static_cast<__nv_bfloat16*>(dg), scale4, shift4, Cin, Cout);
  return static_cast<int>(cudaGetLastError());
}

int ub2_convt_wgrad_reduce(const float* partial, int splits, int Cin, int Cout, float* grad, int accumulate,
                           void* stream) {
  if (Cin <= 0 || Cout <= 0 || splits <= 0) return UB2_ERR_SHAPE;
  const long long total = static_cast<long long>(Cin) * Cout * 4;
  launch(convt_wgrad_reduce_kernel, stream_grid(total, 256, num_sms(), 8), 256, 0, static_cast<cudaStream_t>(stream), partial, splits,
         Cin, Cout, grad, accumulate);
  return static_cast<int>(cudaGetLastError());
}

// ---- fp32 / TF32 mode --------------------------------------------------------------------------------------------
// The same shuffle, transpose, bias gradient and weight pack on fp32 tensors (4 channels per 16-byte vector).  As
// every fp32 entry point, these check their arguments before the device is touched: a count <= 0, C not a multiple
// of 4 or above 1024, Ho < 2h, Wo < 2w, a channel stride below its row (C, or 4*C for t / dt) or a NULL required
// pointer -> UB2_ERR_SHAPE; a channel stride not a multiple of 4 or a 16-byte-vector pointer not 16-byte aligned
// (partials: 8, the pack's scalars: 4) -> UB2_ERR_ALIGN; rows other than ub2_f32_shuffle2x2_rows -> UB2_ERR_WORKSPACE.
static int f32_shuf_geom(ShufGeom* g, int N, int h, int w, int C, int Ho, int Wo) {
  const int rc = shuf_geom(g, N, h, w, C, Ho, Wo, 4);
  if (rc) return rc;
  return g->cgs > 256 ? UB2_ERR_SHAPE : 0;
}

int ub2_f32_shuffle2x2_fwd(const float* t, int ld_t, float* out, int ld_out, int N, int h, int w, int C, int Ho, int Wo,
                           void* stream) {
  ShufGeom g;
  const int rc = f32_shuf_geom(&g, N, h, w, C, Ho, Wo);
  if (rc) return rc;
  if (t == nullptr || out == nullptr || ld_t < 4 * C || ld_out < C) return UB2_ERR_SHAPE;
  if (ld_t % 4 || ld_out % 4 || !al16(t) || !al16(out)) return UB2_ERR_ALIGN;
  const long long total = static_cast<long long>(N) * Ho * Wo * g.cgs;
  launch(shuffle2x2_fwd_kernel<float>, stream_grid(total, 256, num_sms(), 8), 256, 0, static_cast<cudaStream_t>(stream), t, ld_t,
         out, ld_out, g);
  return static_cast<int>(cudaGetLastError());
}

int ub2_f32_shuffle2x2_rows(int N, int h, int w, int C, int Ho, int Wo) {
  ShufGeom g;
  const int rc = f32_shuf_geom(&g, N, h, w, C, Ho, Wo);
  if (rc) return rc;
  return shuf_bwd_grid(g);
}

int ub2_f32_shuffle2x2_bwd(const float* dout, int ld_dout, float* dt, int ld_dt, double* partials, int rows, float* dbias,
                           int N, int h, int w, int C, int Ho, int Wo, void* stream) {
  ShufGeom g;
  const int rc = f32_shuf_geom(&g, N, h, w, C, Ho, Wo);
  if (rc) return rc;
  if (dout == nullptr || dt == nullptr || (partials != nullptr && dbias == nullptr) || ld_dout < C || ld_dt < 4 * C)
    return UB2_ERR_SHAPE;
  if (ld_dout % 4 || ld_dt % 4 || !al16(dout) || !al16(dt) || !aligned_to(partials, 8) ||
      (partials != nullptr && !aligned_to(dbias, 4)))
    return UB2_ERR_ALIGN;
  const int grid = shuf_bwd_grid(g);
  if (partials != nullptr && rows != grid) return UB2_ERR_WORKSPACE;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  launch(shuffle2x2_bwd_kernel<float>, grid, (256 / g.cgs) * g.cgs, 0, s, dout, ld_dout, dt, ld_dt, partials, g);
  if (partials != nullptr)
    launch(shuffle_bias_finalize_kernel, (C + 7) / 8, dim3(8, 128), 0, s, static_cast<const double*>(partials), grid, C, dbias);
  return static_cast<int>(cudaGetLastError());
}

int ub2_f32_pack_convt_weight(const float* w, const float* bias, float* fwd, float* scale4, float* shift4, int Cin, int Cout,
                              void* stream) {
  if (w == nullptr || fwd == nullptr || scale4 == nullptr || shift4 == nullptr || Cin <= 0 || Cout <= 0) return UB2_ERR_SHAPE;
  if (!aligned_to(w, 4) || !aligned_to(bias, 4) || !aligned_to(fwd, 4) || !aligned_to(scale4, 4) || !aligned_to(shift4, 4))
    return UB2_ERR_ALIGN;
  const long long total = static_cast<long long>(Cin) * Cout * 4;
  launch(pack_convt_weight_kernel<float>, stream_grid(total, 256, num_sms(), 8), 256, 0, static_cast<cudaStream_t>(stream), w, bias,
         fwd, static_cast<float*>(nullptr), scale4, shift4, Cin, Cout);
  return static_cast<int>(cudaGetLastError());
}

}  // extern "C"
