// Attention gate (AttentionGate.forward, unet/models/layers.py:171-192) as bandwidth-bound
// passes around the two tcgen05 1x1 projections:
//
//   q  = W_g . g            (low resolution: the 1x1 conv commutes with bilinear resampling)
//   xp = W_x . x            (full resolution, statistics in the conv epilogue)
//   gate_upstats : batch statistics of up(q) for BN_g          (layers.py:153,183,186)
//   gate_psi     : psi_raw = w_psi . relu(BN_g(up q) + BN_x(xp)) + its statistics (:188, :164)
//   gate_apply   : a = sigmoid(BN_psi(psi_raw)); out = x * a   (:165-166, :192)
// and the matching backward passes.  The three train-mode BatchNorms force three
// grid-wide reductions, hence three phases; in eval mode the same kernels run with
// folded running statistics and no reductions.
//
// Thread mapping: `tpp` (power of two <= 32) consecutive threads share a pixel and split its
// 8-channel vectors; per-pixel channel reductions are shuffle reductions inside that group,
// per-channel pixel reductions stay in registers (a thread's channels are fixed) and are
// combined per block in shared memory, then across blocks by a finalize kernel in double.
#include "launch.cuh"
#include "../../include/unetb200.h"
#include "conv.h"
#include "resample.cuh"
#include "vec.cuh"

#include <cstdlib>
#include <mutex>
#include <utility>
#include <vector>

namespace ub2 {

static constexpr int kGateThreads = 256;
static constexpr int kMaxG = 2;  // 8-channel groups per thread (channels <= 512)

struct GateGeom {
  int N, H, W, C, cgs, tpp, slots;
  int pixels;
  int wt, ht;   // strip kernels: column tiles of `slots` pixels x row strips of kGateStrip rows
  LowRes lr;
};
static constexpr int kGateStrip = 16;

static int gate_tpp(int cgs) {
  int t = 1;
  while (t < cgs && t < 32) t *= 2;
  return t;
}
static int make_gate_geom(GateGeom* g, int N, int H, int W, int C, int hin, int win) {
  if (C <= 0 || C % 8 != 0 || N <= 0 || H <= 0 || W <= 0 || hin <= 0 || win <= 0) return UB2_ERR_SHAPE;
  if (static_cast<double>(N) * H * W * (C / 8) >= 2.0e9) return UB2_ERR_SHAPE;  // 32-bit pixel indices
  g->N = N; g->H = H; g->W = W; g->C = C; g->cgs = C / 8;
  g->tpp = gate_tpp(g->cgs);
  if ((g->cgs + g->tpp - 1) / g->tpp > kMaxG) return UB2_ERR_SHAPE;
  g->slots = kGateThreads / g->tpp;
  g->pixels = static_cast<int>(N) * H * W;
  g->wt = (W + g->slots - 1) / g->slots;
  g->ht = (H + kGateStrip - 1) / kGateStrip;
  g->lr = make_lowres(hin, win, H, W);
  return 0;
}
static int gate_strip_grid(const GateGeom& g) { return g.wt * g.ht * g.N; }
static bool al16(const void* p) { return aligned_to(p, 16); }
// A bf16 NHWC operand of C channels read or written with 16-byte vectors: UB2_ERR_SHAPE for a NULL pointer or a
// channel stride below C, UB2_ERR_ALIGN for a stride that is not a multiple of 8 or a pointer off 16 bytes.
static int vec_operand(const void* p, int ld, int C) {
  if (p == nullptr || ld < C) return UB2_ERR_SHAPE;
  return (ld % 8 || !al16(p)) ? UB2_ERR_ALIGN : 0;
}
static int gate_grid(const GateGeom& g, int per_sm) {
  return stream_grid(g.pixels, g.slots, num_sms(), per_sm);
}

__device__ __forceinline__ float group_sum(float v, int tpp) {
  for (int o = tpp >> 1; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Reduce per-thread channel accumulators over the pixel slots of a block and write one
// row of doubles: out_row[ns*C + channel].
template <int G, int NS>
__device__ __forceinline__ void block_reduce_channels(float (&acc)[G][NS][8], const GateGeom& g,
                                                      int slot, int j, double* out_row, float* smem) {
#pragma unroll
  for (int gi = 0; gi < G; ++gi) {
#pragma unroll
    for (int ns = 0; ns < NS; ++ns) {
#pragma unroll
      for (int k = 0; k < 8; ++k) smem[(slot * g.tpp + j) * 8 + k] = acc[gi][ns][k];
      __syncthreads();
      for (int idx = threadIdx.x; idx < g.tpp * 8; idx += blockDim.x) {
        const int jj = idx >> 3, k = idx & 7;
        const int cg = jj + gi * g.tpp;
        if (cg < g.cgs) {
          double s = 0.0;
          for (int sl = 0; sl < g.slots; ++sl) s += static_cast<double>(smem[(sl * g.tpp + jj) * 8 + k]);
          out_row[static_cast<size_t>(ns) * g.C + cg * 8 + k] = s;
        }
      }
      __syncthreads();
    }
  }
}

// Same for per-thread scalars (NS values), written as out_row[ns].
template <int NS>
__device__ __forceinline__ void block_reduce_scalars(float (&acc)[NS], double* out_row, float* smem) {
#pragma unroll
  for (int ns = 0; ns < NS; ++ns) {
    const float w = warp_sum(acc[ns]);
    if ((threadIdx.x & 31) == 0) smem[threadIdx.x >> 5] = w;
    __syncthreads();
    if (threadIdx.x == 0) {
      double s = 0.0;
      for (int i = 0; i < (blockDim.x >> 5); ++i) s += static_cast<double>(smem[i]);
      out_row[ns] = s;
    }
    __syncthreads();
  }
}

// Warp-uniform trip count (the shuffle reductions need every lane): `pv` masks the tail.
#define GATE_PIXEL_LOOP(g)                                                                  \
  const int slot = threadIdx.x / (g).tpp;                                                   \
  const int j = threadIdx.x % (g).tpp;                                                      \
  for (int base = static_cast<int>(blockIdx.x) * (g).slots; base < (g).pixels;  \
       base += static_cast<int>(gridDim.x) * (g).slots)

#define GATE_PIX(g)                     \
  const int pix = base + slot;    \
  const bool pv = pix < (g).pixels;

#define GATE_DECODE(g)                                                        \
  const int wo = static_cast<int>(pix % (g).W);                               \
  const int ho = static_cast<int>((pix / (g).W) % (g).H);                     \
  const int n = static_cast<int>(pix / (static_cast<int>((g).W) * (g).H));

// Strip walk for the passes that need up(q): a block owns `slots` columns x kGateStrip rows of one
// image, a thread one column (x `tpp` lanes over the channels) and walks the rows.  No per-pixel
// integer division, and the two horizontally interpolated low-resolution rows a destination row lies
// between stay in registers (they change every other row for a 2x up-sampling).
//
// Every operand of a row is fetched with cp.async into a per-thread ring in shared memory kD rows ahead:
// the round-1 form of these kernels issued one 16-byte load per thread and row and used it at once —
// 8-12 KB in flight per SM where HBM needs ~35 KB (ncu: long-scoreboard stalls, 0.9-2.7 TB/s, 23-32 %
// occupancy because the prefetch that was tried lived in registers).  A thread only ever reads what it
// fetched itself, so cp.async.wait_group is all the synchronisation the ring needs.
//   qbuf [QR][2][G][threads] uint4   low-resolution rows (columns w0 / w1 of this thread), row h in slot h % QR
//   vbuf [kD][NV][G][threads] uint4  streamed bf16 vectors of an output row (stage ho % kD)
//   sbuf [kD][NS][threads]   float   streamed per-pixel scalars
// Low-resolution rows are requested together with the first output row that needs them, so one
// wait_group per output row covers both.  QR = 4 holds every row in flight for up-sampling factors >= 2
// (H >= 2*hin - 1, the U-Net case), QR = 8 for factors >= 1.
static constexpr int kD = 4;   // output rows in flight per thread
#ifndef UB2_GATE_BWD_S_BLOCKS
#define UB2_GATE_BWD_S_BLOCKS 2   // 3 caps gate_bwd_s at 80 registers (small spill); A/B on the GPU decides
#endif

__device__ __forceinline__ void cp_async16_ca(void* smem, const void* gmem) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(static_cast<uint32_t>(__cvta_generic_to_shared(smem))), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async16_cg(void* smem, const void* gmem) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(static_cast<uint32_t>(__cvta_generic_to_shared(smem))), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async4(void* smem, const void* gmem) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(static_cast<uint32_t>(__cvta_generic_to_shared(smem))), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

template <int G, int QR, int NV, int NS>
struct Strip {
  static constexpr int kQVecs = QR * 2 * G;
  static constexpr int kVVecs = kD * NV * G;
  static constexpr size_t kBytes = static_cast<size_t>(kGateThreads) * (16 * (kQVecs + kVVecs) + 4 * kD * NS);
  // thread -> (column, channel group)
  int slot, j, n, wo, ho0, ho1;
  bool pv;
  // low-resolution roll
  int cur0, cur1, w0, w1, qnext;
  float a0, a1, b0, b1;
  F8 top[G], bot[G];
  uint4* qbuf;
  uint4* vbuf;
  float* sbuf;

  __device__ __forceinline__ void init(const GateGeom& g, uint8_t* smem) {
    slot = threadIdx.x / g.tpp;
    j = threadIdx.x % g.tpp;
    const int bw = static_cast<int>(blockIdx.x) % g.wt;
    const int bh = (static_cast<int>(blockIdx.x) / g.wt) % g.ht;
    n = static_cast<int>(blockIdx.x) / (g.wt * g.ht);
    wo = bw * g.slots + slot;
    pv = wo < g.W;
    ho0 = bh * kGateStrip;
    ho1 = min(ho0 + kGateStrip, g.H);
    cur0 = cur1 = -1;
    src_index(g.lr.rw, pv ? wo : g.W - 1, g.lr.win, w0, w1, b0, b1);
    int h0, h1;
    float l0, l1;
    src_index(g.lr.rh, ho0, g.lr.hin, h0, h1, l0, l1);
    qnext = h0;
    qbuf = reinterpret_cast<uint4*>(smem);
    vbuf = qbuf + kQVecs * kGateThreads;
    sbuf = reinterpret_cast<float*>(vbuf + kVVecs * kGateThreads);
#pragma unroll
    for (int gi = 0; gi < G; ++gi)
#pragma unroll
      for (int k = 0; k < 8; ++k) top[gi].v[k] = bot[gi].v[k] = 0.f;
  }
  __device__ __forceinline__ bool lane_on(const GateGeom& g, int gi) const { return pv && (j + gi * g.tpp) < g.cgs; }

  // Request everything output row `ho` needs (its own commit group; an empty one past the strip).
  // vptr[v]: row-0 pointer of streamed tensor v at this thread's column / first channel group; sptr likewise.
  __device__ __forceinline__ void request(const GateGeom& g, int ho, const __nv_bfloat16* __restrict__ q, int ld_q,
                                          const __nv_bfloat16* const (&vptr)[NV > 0 ? NV : 1], const int (&vld)[NV > 0 ? NV : 1],
                                          const float* const (&sptr)[NS > 0 ? NS : 1]) {
    if (ho < ho1) {
      int h0, h1;
      float l0, l1;
      src_index(g.lr.rh, ho, g.lr.hin, h0, h1, l0, l1);
      const __nv_bfloat16* qimg = q + static_cast<size_t>(n) * g.lr.hin * g.lr.win * ld_q;
      for (; qnext <= h1; ++qnext) {
        uint4* dst = qbuf + static_cast<size_t>((qnext % QR) * 2 * G) * kGateThreads + threadIdx.x;
#pragma unroll
        for (int gi = 0; gi < G; ++gi) {
          if (lane_on(g, gi)) {
            const int cg = j + gi * g.tpp;
            cp_async16_ca(dst + (0 * G + gi) * kGateThreads, qimg + (static_cast<size_t>(qnext) * g.lr.win + w0) * ld_q + cg * 8);
            cp_async16_ca(dst + (1 * G + gi) * kGateThreads, qimg + (static_cast<size_t>(qnext) * g.lr.win + w1) * ld_q + cg * 8);
          }
        }
      }
      const size_t pix = (static_cast<size_t>(n) * g.H + ho) * g.W + (pv ? wo : 0);
      const int st = ho % kD;
#pragma unroll
      for (int v = 0; v < NV; ++v) {
#pragma unroll
        for (int gi = 0; gi < G; ++gi) {
          if (lane_on(g, gi))
            cp_async16_cg(vbuf + static_cast<size_t>((st * NV + v) * G + gi) * kGateThreads + threadIdx.x,
                          vptr[v] + pix * vld[v] + (j + gi * g.tpp) * 8);
        }
      }
#pragma unroll
      for (int k = 0; k < NS; ++k) {
        if (pv) cp_async4(sbuf + static_cast<size_t>(st * NS + k) * kGateThreads + threadIdx.x, sptr[k] + pix);
      }
    }
    cp_async_commit();
  }

  // After the wait for row `ho`: advance the roll to the two low-resolution rows it lies between.
  __device__ __forceinline__ void roll_to(const GateGeom& g, int ho) {
    int h0, h1;
    src_index(g.lr.rh, ho, g.lr.hin, h0, h1, a0, a1);   // block-uniform
    auto hrow = [&](int h, int gi) {
      F8 o;
      if (lane_on(g, gi)) {
        const uint4* src = qbuf + static_cast<size_t>((h % QR) * 2 * G) * kGateThreads + threadIdx.x;
        const F8 a = unpack8(src[(0 * G + gi) * kGateThreads]);
        const F8 b = unpack8(src[(1 * G + gi) * kGateThreads]);
#pragma unroll
        for (int k = 0; k < 8; ++k) o.v[k] = b0 * a.v[k] + b1 * b.v[k];
      } else {
#pragma unroll
        for (int k = 0; k < 8; ++k) o.v[k] = 0.f;
      }
      return o;
    };
    if (h0 != cur0) {
#pragma unroll
      for (int gi = 0; gi < G; ++gi) top[gi] = (h0 == cur1) ? bot[gi] : hrow(h0, gi);
      cur0 = h0;
    }
    if (h1 != cur1) {
#pragma unroll
      for (int gi = 0; gi < G; ++gi) bot[gi] = (h1 == cur0) ? top[gi] : hrow(h1, gi);
      cur1 = h1;
    }
  }
  __device__ __forceinline__ F8 up(int gi) const {
    F8 u;
#pragma unroll
    for (int k = 0; k < 8; ++k) u.v[k] = a0 * top[gi].v[k] + a1 * bot[gi].v[k];
    return u;
  }
  __device__ __forceinline__ F8 vec(int ho, int v, int gi) const {
    return unpack8(vbuf[static_cast<size_t>(((ho % kD) * NV + v) * G + gi) * kGateThreads + threadIdx.x]);
  }
  __device__ __forceinline__ float scalar(int ho, int k) const {
    return sbuf[static_cast<size_t>((ho % kD) * NS + k) * kGateThreads + threadIdx.x];
  }
};

// for (row of the strip) { requests kD-1 rows ahead; waits for this row; rolls }: the body sees
// `ho`, `pix` and the Strip `S` with up(q) / streamed vectors of the row.
#define GATE_STRIP_BEGIN(S, g, q, ld_q, vptr, vld, sptr)                                       \
  extern __shared__ __align__(16) uint8_t strip_smem[];                                        \
  S.init(g, strip_smem);                                                                       \
  _Pragma("unroll") for (int pre = 0; pre < kD - 1; ++pre) S.request(g, S.ho0 + pre, q, ld_q, vptr, vld, sptr); \
  for (int ho = S.ho0; ho < S.ho1; ++ho) {                                                     \
    S.request(g, ho + kD - 1, q, ld_q, vptr, vld, sptr);                                       \
    cp_async_wait<kD - 1>();                                                                   \
    S.roll_to(g, ho);                                                                          \
    const int pix = (S.n * (g).H + ho) * (g).W + (S.pv ? S.wo : 0);
#define GATE_STRIP_END }

// ------------------------------------------------------------------------------ forward
template <int G, int QR>
__global__ void __launch_bounds__(kGateThreads)
gate_upstats_kernel(const __nv_bfloat16* __restrict__ q, int ld_q, double* partials, GateGeom g) {
  pdl_trigger();
  pdl_wait();
  __shared__ float smem[kGateThreads * 8];
  float acc[G][2][8];
#pragma unroll
  for (int a = 0; a < G; ++a)
#pragma unroll
    for (int b = 0; b < 2; ++b)
#pragma unroll
      for (int k = 0; k < 8; ++k) acc[a][b][k] = 0.f;
  Strip<G, QR, 0, 0> S;
  const __nv_bfloat16* const vptr[1] = {nullptr};
  const int vld[1] = {0};
  const float* const sptr[1] = {nullptr};
  GATE_STRIP_BEGIN(S, g, q, ld_q, vptr, vld, sptr)
    (void)pix;
#pragma unroll
    for (int gi = 0; gi < G; ++gi) {
      if (S.lane_on(g, gi)) {
        const F8 u = S.up(gi);
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          acc[gi][0][k] += u.v[k];
          acc[gi][1][k] = fmaf(u.v[k], u.v[k], acc[gi][1][k]);
        }
      }
    }
  GATE_STRIP_END
  block_reduce_channels<G, 2>(acc, g, S.slot, S.j, partials + static_cast<size_t>(blockIdx.x) * 2 * g.C, smem);
}

// Batch statistics of up(q) WITHOUT up-sampling: bilinear interpolation is linear, so the sums over the
// full-resolution pixels are weighted sums over the low-resolution tensor and its 2x2 neighbourhoods,
//   sum u   = sum_h sum_w RW[h] CW[w] q[h,w]
//   sum u^2 = sum_h sum_w D[h] (E[w] q00^2 + 2 F[w] q00 q01) + X[h] (E[w] q00 q10 + F[w] (q00 q11 + q01 q10))
// with q00 = q[h,w], q01 = q[h,w+1], q10 = q[h+1,w], q11 = q[h+1,w+1] and per-row / per-column tables built from
// ATen's own index arithmetic: RW[h] = total weight row h receives, D[h] = sum of its squared weights, X[h] = sum of
// 2 a0 a1 over the output rows that lie between rows h and h+1 (CW, E, F likewise, F without the factor 2).
// One quarter of the pixels, no roll, no row walk: 36 -> ~8 us at the up4 level.  Exact algebra; fp32 rounding only.
__device__ __forceinline__ void lowres_tables(float r, int in, int out, int i, float& wsum, float& wsq, float& cross2) {
  int lo, hi;
  if (r <= 0.f) { lo = 0; hi = out - 1; }
  else {
    lo = static_cast<int>(ceilf((static_cast<float>(i) - 1.f) / r)) - 1;
    hi = static_cast<int>(floorf((static_cast<float>(i) + 1.f) / r)) + 1;
    if (lo < 0) lo = 0;
    if (hi > out - 1) hi = out - 1;
  }
  wsum = wsq = cross2 = 0.f;
  for (int o = lo; o <= hi; ++o) {
    int i0, i1;
    float l0, l1;
    src_index(r, o, in, i0, i1, l0, l1);
    if (i0 == i1) {            // clamped at the last source index: the pixel IS that row / column
      if (i0 == i) { wsum += l0 + l1; wsq += (l0 + l1) * (l0 + l1); }
    } else {
      if (i0 == i) { wsum += l0; wsq += l0 * l0; cross2 += l0 * l1; }
      if (i1 == i) { wsum += l1; wsq += l1 * l1; }
    }
  }
}

template <int G>
__global__ void __launch_bounds__(kGateThreads)
gate_upstats_lowres_kernel(const __nv_bfloat16* __restrict__ q, int ld_q, double* partials, GateGeom g) {
  pdl_trigger();
  pdl_wait();
  __shared__ float smem[kGateThreads * 8];
  extern __shared__ float tab[];
  const int hin = g.lr.hin, win = g.lr.win;
  float* RW = tab; float* D = RW + hin; float* X = D + hin;
  float* CW = X + hin; float* E = CW + win; float* F = E + win;
  for (int h = threadIdx.x; h < hin; h += blockDim.x) {
    float c2;
    lowres_tables(g.lr.rh, hin, g.H, h, RW[h], D[h], c2);
    X[h] = 2.f * c2;
  }
  for (int w = threadIdx.x; w < win; w += blockDim.x) lowres_tables(g.lr.rw, win, g.W, w, CW[w], E[w], F[w]);
  __syncthreads();
  float acc[G][2][8];
#pragma unroll
  for (int a = 0; a < G; ++a)
#pragma unroll
    for (int b = 0; b < 2; ++b)
#pragma unroll
      for (int k = 0; k < 8; ++k) acc[a][b][k] = 0.f;
  const int slot = threadIdx.x / g.tpp, j = threadIdx.x % g.tpp;
  const int lp = g.N * hin * win;
  for (int base = static_cast<int>(blockIdx.x) * g.slots; base < lp; base += static_cast<int>(gridDim.x) * g.slots) {
    const int pix = base + slot;
    if (pix < lp) {
      const int w = pix % win, h = (pix / win) % hin, n = pix / (win * hin);
      const int w1 = min(w + 1, win - 1), h1 = min(h + 1, hin - 1);
      const float rwcw = RW[h] * CW[w], de = D[h] * E[w], df2 = 2.f * D[h] * F[w], xe = X[h] * E[w], xf = X[h] * F[w];
      const __nv_bfloat16* img = q + static_cast<size_t>(n) * hin * win * ld_q;
#pragma unroll
      for (int gi = 0; gi < G; ++gi) {
        const int cg = j + gi * g.tpp;
        if (cg < g.cgs) {
          const F8 q00 = load8(img + (static_cast<size_t>(h) * win + w) * ld_q + cg * 8);
          const F8 q01 = load8(img + (static_cast<size_t>(h) * win + w1) * ld_q + cg * 8);
          const F8 q10 = load8(img + (static_cast<size_t>(h1) * win + w) * ld_q + cg * 8);
          const F8 q11 = load8(img + (static_cast<size_t>(h1) * win + w1) * ld_q + cg * 8);
#pragma unroll
          for (int k = 0; k < 8; ++k) {
            acc[gi][0][k] = fmaf(rwcw, q00.v[k], acc[gi][0][k]);
            const float same = fmaf(de, q00.v[k], df2 * q01.v[k]) * q00.v[k];
            const float next = fmaf(xe, q00.v[k], xf * q01.v[k]) * q10.v[k] + xf * q00.v[k] * q11.v[k];
            acc[gi][1][k] += same + next;
          }
        }
      }
    }
  }
  block_reduce_channels<G, 2>(acc, g, slot, j, partials + static_cast<size_t>(blockIdx.x) * 2 * g.C, smem);
}

// Per-channel coefficient vectors (BN_g scale, BN_x scale, summed shifts, psi weights) live in shared
// memory: 32 registers per thread in the round-1 form, which is what kept these kernels at two or three
// blocks per SM.  A warp reads at most `tpp` distinct 32-byte rows of it at a time (broadcast).
struct GateCoef {
  const float* sg;   // [C] each, contiguous: sg | sx | h | w
  __device__ __forceinline__ F8 get(int which, int cg, int C) const {
    F8 r;
    const float4* p = reinterpret_cast<const float4*>(sg + which * C + cg * 8);
    const float4 a = p[0], b = p[1];
    r.v[0] = a.x; r.v[1] = a.y; r.v[2] = a.z; r.v[3] = a.w;
    r.v[4] = b.x; r.v[5] = b.y; r.v[6] = b.z; r.v[7] = b.w;
    return r;
  }
};
// s_coef: 4*C floats of (dynamic) shared memory behind the strip ring; call before the strip loop
__device__ __forceinline__ GateCoef gate_coef_load(float* s_coef, const float* sg, const float* hg, const float* sx,
                                                   const float* hx, const float* wpsi, int C) {
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    s_coef[c] = __ldg(sg + c);
    s_coef[C + c] = __ldg(sx + c);
    s_coef[2 * C + c] = __ldg(hg + c) + __ldg(hx + c);
    s_coef[3 * C + c] = __ldg(wpsi + c);
  }
  __syncthreads();
  GateCoef k;
  k.sg = s_coef;
  return k;
}

template <int G, int QR>
__global__ void __launch_bounds__(kGateThreads)
gate_psi_kernel(const __nv_bfloat16* __restrict__ q, int ld_q, const __nv_bfloat16* __restrict__ xp,
                int ld_xp, const float* __restrict__ sg, const float* __restrict__ hg,
                const float* __restrict__ sx, const float* __restrict__ hx,
                const float* __restrict__ wpsi, float* __restrict__ psi_raw, double* partials,
                GateGeom g) {
  pdl_trigger();
  pdl_wait();
  __shared__ float smem[kGateThreads / 32];
  float st[2] = {0.f, 0.f};
  typedef Strip<G, QR, 1, 0> S_t;
  S_t S;
  const __nv_bfloat16* const vptr[1] = {xp};
  const int vld[1] = {ld_xp};
  const float* const sptr[1] = {nullptr};
  extern __shared__ __align__(16) uint8_t strip_smem_c[];
  const GateCoef cf = gate_coef_load(reinterpret_cast<float*>(strip_smem_c + S_t::kBytes), sg, hg, sx, hx, wpsi, g.C);
  GATE_STRIP_BEGIN(S, g, q, ld_q, vptr, vld, sptr)
    float dot = 0.f;
#pragma unroll
    for (int gi = 0; gi < G; ++gi) {
      if (S.lane_on(g, gi)) {
        const int cg = S.j + gi * g.tpp;
        const F8 u = S.up(gi);
        const F8 xv = S.vec(ho, 0, gi);
        const F8 vsg = cf.get(0, cg, g.C), vsx = cf.get(1, cg, g.C), vh = cf.get(2, cg, g.C), vw = cf.get(3, cg, g.C);
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const float t = fmaf(u.v[k], vsg.v[k], fmaf(xv.v[k], vsx.v[k], vh.v[k]));
          dot = fmaf(vw.v[k], fmaxf(t, 0.f), dot);
        }
      }
    }
    dot = group_sum(dot, g.tpp);
    if (S.pv && S.j == 0) {
      psi_raw[pix] = dot;
      st[0] += dot;
      st[1] = fmaf(dot, dot, st[1]);
    }
  GATE_STRIP_END
  if (partials != nullptr) block_reduce_scalars<2>(st, partials + static_cast<size_t>(blockIdx.x) * 2, smem);
}

// Inference (no BatchNorm reduction forces phases): psi, sigmoid and the gating of the skip in ONE pass —
// north_star (3).  The skip tensor's channels are streamed through the same ring as two more operands
// (x[:, :Ci] and x[:, Ci:]; the gate's inter-channel count is half the skip's, layers.py:147-148), so the
// thread group that reduced a pixel's psi also scales and stores that pixel.
template <int G, int QR>
__global__ void __launch_bounds__(kGateThreads)
gate_fused_eval_kernel(const __nv_bfloat16* __restrict__ q, int ld_q, const __nv_bfloat16* __restrict__ xp, int ld_xp,
                       const __nv_bfloat16* __restrict__ x, int ld_x, const float* __restrict__ sg,
                       const float* __restrict__ hg, const float* __restrict__ sx, const float* __restrict__ hx,
                       const float* __restrict__ wpsi, const float* __restrict__ spsi, const float* __restrict__ hpsi,
                       __nv_bfloat16* __restrict__ out, int ld_out, GateGeom g) {
  pdl_trigger();
  pdl_wait();
  typedef Strip<G, QR, 3, 0> S_t;
  S_t S;
  const __nv_bfloat16* const vptr[3] = {xp, x, x + g.C};
  const int vld[3] = {ld_xp, ld_x, ld_x};
  const float* const sptr[1] = {nullptr};
  extern __shared__ __align__(16) uint8_t strip_smem_c[];
  const GateCoef cf = gate_coef_load(reinterpret_cast<float*>(strip_smem_c + S_t::kBytes), sg, hg, sx, hx, wpsi, g.C);
  const float ps = __ldg(spsi), ph = __ldg(hpsi);
  GATE_STRIP_BEGIN(S, g, q, ld_q, vptr, vld, sptr)
    float dot = 0.f;
#pragma unroll
    for (int gi = 0; gi < G; ++gi) {
      if (S.lane_on(g, gi)) {
        const int cg = S.j + gi * g.tpp;
        const F8 u = S.up(gi);
        const F8 xv = S.vec(ho, 0, gi);
        const F8 vsg = cf.get(0, cg, g.C), vsx = cf.get(1, cg, g.C), vh = cf.get(2, cg, g.C), vw = cf.get(3, cg, g.C);
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const float t = fmaf(u.v[k], vsg.v[k], fmaf(xv.v[k], vsx.v[k], vh.v[k]));
          dot = fmaf(vw.v[k], fmaxf(t, 0.f), dot);
        }
      }
    }
    dot = group_sum(dot, g.tpp);
    const float a = 1.f / (1.f + __expf(-fmaf(dot, ps, ph)));   // as gate_apply_kernel
#pragma unroll
    for (int gi = 0; gi < G; ++gi) {
      if (S.lane_on(g, gi)) {
        const int cg = S.j + gi * g.tpp;
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          F8 v = S.vec(ho, 1 + half, gi);
#pragma unroll
          for (int k = 0; k < 8; ++k) v.v[k] *= a;
          store8(out + static_cast<size_t>(pix) * ld_out + half * g.C + cg * 8, v);
        }
      }
    }
  GATE_STRIP_END
}

__global__ void __launch_bounds__(256)
gate_apply_kernel(const float* __restrict__ psi_raw, const float* __restrict__ spsi,
                  const float* __restrict__ hpsi, const __nv_bfloat16* __restrict__ x, int ld_x,
                  __nv_bfloat16* __restrict__ out, int ld_out, float* __restrict__ a_out,
                  int pixels, int cgs) {
  pdl_trigger();
  pdl_wait();
  const float s = __ldg(spsi), h = __ldg(hpsi);
  const int total = pixels * cgs;
  const int stride = static_cast<int>(gridDim.x) * blockDim.x;
  // four vectors per trip, loads first: the copy runs at HBM speed only with several 128-bit
  // requests in flight per thread
  for (int i0 = static_cast<int>(blockIdx.x) * blockDim.x + threadIdx.x; i0 < total; i0 += 4 * stride) {
    uint4 raw[4];
    float pr[4];
    int pixv[4], cgv[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int i = i0 + u * stride;
      const bool ok = i < total;
      cgv[u] = ok ? i % cgs : 0;
      pixv[u] = ok ? i / cgs : -1;
      raw[u] = make_uint4(0u, 0u, 0u, 0u);
      pr[u] = 0.f;
      if (ok) {
        raw[u] = ld_stream16(x + static_cast<size_t>(pixv[u]) * ld_x + cgv[u] * 8);
        pr[u] = __ldg(psi_raw + pixv[u]);
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      if (pixv[u] < 0) continue;
      const float z = fmaf(pr[u], s, h);
      const float a = 1.f / (1.f + __expf(-z));
      F8 v = unpack8(raw[u]);
#pragma unroll
      for (int k = 0; k < 8; ++k) v.v[k] *= a;
      store8(out + static_cast<size_t>(pixv[u]) * ld_out + cgv[u] * 8, v);
      if (cgv[u] == 0 && a_out != nullptr) a_out[pixv[u]] = a;
    }
  }
}

// ------------------------------------------------------------------------------ backward
// da = sum_c dOut_c x_c ; d(BN_psi out) = da * a (1-a) ; dx_direct = dOut * a
template <int G>
__global__ void __launch_bounds__(kGateThreads)
gate_bwd_a_kernel(const __nv_bfloat16* __restrict__ dout, int ld_do, const __nv_bfloat16* __restrict__ x,
                  int ld_x, const float* __restrict__ a, const float* __restrict__ psi_raw,
                  __nv_bfloat16* __restrict__ dx, int ld_dx, float* __restrict__ dpsin,
                  double* partials, GateGeom g) {
  pdl_trigger();
  pdl_wait();
  __shared__ float smem[kGateThreads / 32];
  float st[2] = {0.f, 0.f};  // sum dn, sum dn*psi_raw (bn_bwd_finalize convention)
  GATE_PIXEL_LOOP(g) {
    GATE_PIX(g)
    const float av = pv ? __ldg(a + pix) : 0.f;
    float dot = 0.f;
#pragma unroll
    for (int gi = 0; gi < G; ++gi) {
      const int cg = j + gi * g.tpp;
      if (pv && cg < g.cgs) {
        F8 d = load8_stream(dout + static_cast<size_t>(pix) * ld_do + cg * 8);
        const F8 xv = load8_stream(x + static_cast<size_t>(pix) * ld_x + cg * 8);
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          dot = fmaf(d.v[k], xv.v[k], dot);
          d.v[k] *= av;
        }
        store8(dx + static_cast<size_t>(pix) * ld_dx + cg * 8, d);
      }
    }
    dot = group_sum(dot, g.tpp);
    if (pv && j == 0) {
      const float dn = dot * av * (1.f - av);
      dpsin[pix] = dn;
      st[0] += dn;
      st[1] = fmaf(dn, __ldg(psi_raw + pix), st[1]);
    }
  }
  block_reduce_scalars<2>(st, partials + static_cast<size_t>(blockIdx.x) * 2, smem);
}

// ds_c = dpsi_raw * w_psi_c * [t_c > 0]; channel sums (raw, the finalize converts them):
// sum ds, sum ds*xp, sum ds*up(q), sum dpsi_raw*relu(t)
template <int G, int QR>
__global__ void __launch_bounds__(kGateThreads, G == 1 ? UB2_GATE_BWD_S_BLOCKS : 1)
gate_bwd_s_kernel(const float* __restrict__ dpsin, const float* __restrict__ psi_raw,
                  const float* __restrict__ coef_psi, const __nv_bfloat16* __restrict__ q, int ld_q,
                  const __nv_bfloat16* __restrict__ xp, int ld_xp, const float* __restrict__ sg,
                  const float* __restrict__ hg, const float* __restrict__ sx,
                  const float* __restrict__ hx, const float* __restrict__ wpsi,
                  __nv_bfloat16* __restrict__ ds, int ld_ds, double* partials, GateGeom g) {
  pdl_trigger();
  pdl_wait();
  __shared__ float smem[kGateThreads * 8];
  const float cA = __ldg(coef_psi), cB = __ldg(coef_psi + 1), cC = __ldg(coef_psi + 2);
  float acc[G][4][8];
#pragma unroll
  for (int a = 0; a < G; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b)
#pragma unroll
      for (int k = 0; k < 8; ++k) acc[a][b][k] = 0.f;
  typedef Strip<G, QR, 1, 2> S_t;
  S_t S;
  const __nv_bfloat16* const vptr[1] = {xp};
  const int vld[1] = {ld_xp};
  const float* const sptr[2] = {dpsin, psi_raw};
  extern __shared__ __align__(16) uint8_t strip_smem_c[];
  const GateCoef cf = gate_coef_load(reinterpret_cast<float*>(strip_smem_c + S_t::kBytes), sg, hg, sx, hx, wpsi, g.C);
  GATE_STRIP_BEGIN(S, g, q, ld_q, vptr, vld, sptr)
    // BN_psi backward: d psi_raw = A*dn + B*psi_raw + C
    const float dpr = S.pv ? fmaf(cA, S.scalar(ho, 0), fmaf(cB, S.scalar(ho, 1), cC)) : 0.f;
#pragma unroll
    for (int gi = 0; gi < G; ++gi) {
      if (S.lane_on(g, gi)) {
        const int cg = S.j + gi * g.tpp;
        const F8 u = S.up(gi);
        const F8 xv = S.vec(ho, 0, gi);
        const F8 vsg = cf.get(0, cg, g.C), vsx = cf.get(1, cg, g.C), vh = cf.get(2, cg, g.C), vw = cf.get(3, cg, g.C);
        F8 o;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const float t = fmaf(u.v[k], vsg.v[k], fmaf(xv.v[k], vsx.v[k], vh.v[k]));
          const float d = (t > 0.f) ? dpr * vw.v[k] : 0.f;
          o.v[k] = d;
          acc[gi][0][k] += d;
          acc[gi][1][k] = fmaf(d, xv.v[k], acc[gi][1][k]);
          acc[gi][2][k] = fmaf(d, u.v[k], acc[gi][2][k]);
          acc[gi][3][k] = fmaf(dpr, fmaxf(t, 0.f), acc[gi][3][k]);
        }
        store8(ds + static_cast<size_t>(pix) * ld_ds + cg * 8, o);
      }
    }
  GATE_STRIP_END
  block_reduce_channels<G, 4>(acc, g, S.slot, S.j, partials + static_cast<size_t>(blockIdx.x) * 4 * g.C, smem);
}

// Raw sums -> parameter gradients and the backward coefficients of the two BatchNorms:
//   dxp = coef0*ds + coef1*xp + coef2 ;  d(up q) = coef3*ds + coef4*up(q) + coef5
// blockDim = (8, 128): see rows_sum_wide in vec.cuh
__global__ void gate_bwd_finalize_kernel(const double* __restrict__ partials, int rows, int C,
                                         double count, const float* __restrict__ gamma_x,
                                         const float* __restrict__ mean_x,
                                         const float* __restrict__ invstd_x,
                                         const float* __restrict__ gamma_g,
                                         const float* __restrict__ mean_g,
                                         const float* __restrict__ invstd_g, int frozen, float* dgamma_x,
                                         float* dbeta_x, float* dgamma_g, float* dbeta_g, float* dwpsi,
                                         float* coef) {
  pdl_trigger();
  pdl_wait();
  __shared__ double smem[4 * 128 * 9];
  const int c = blockIdx.x * 8 + threadIdx.x;
  double s[4];
  rows_sum_wide<4>(partials, rows, C, c, s, smem);
  if (threadIdx.y != 0 || c >= C) return;
  const double mx = mean_x[c], ix = invstd_x[c], mg = mean_g[c], ig = invstd_g[c];
  const double db = s[0];
  const double dgx = ix * (s[1] - mx * s[0]);
  const double dgg = ig * (s[2] - mg * s[0]);
  if (dbeta_x) dbeta_x[c] += static_cast<float>(db);
  if (dgamma_x) dgamma_x[c] += static_cast<float>(dgx);
  if (dbeta_g) dbeta_g[c] += static_cast<float>(db);
  if (dgamma_g) dgamma_g[c] += static_cast<float>(dgg);
  if (dwpsi) dwpsi[c] += static_cast<float>(s[3]);
  const double Ax = gamma_x[c] * ix, Ag = gamma_g[c] * ig;
  const double Bx = frozen ? 0.0 : -Ax * ix * dgx / count;
  const double Bg = frozen ? 0.0 : -Ag * ig * dgg / count;
  coef[0 * C + c] = static_cast<float>(Ax);
  coef[1 * C + c] = static_cast<float>(Bx);
  coef[2 * C + c] = static_cast<float>(frozen ? 0.0 : -Ax * db / count - Bx * mx);
  coef[3 * C + c] = static_cast<float>(Ag);
  coef[4 * C + c] = static_cast<float>(Bg);
  coef[5 * C + c] = static_cast<float>(frozen ? 0.0 : -Ag * db / count - Bg * mg);
}

// dxp = BN_x backward of ds; dgup = BN_g backward of ds (full resolution, later up-sample^T)
template <int G, int QR>
__global__ void __launch_bounds__(kGateThreads)
gate_bwd_xg_kernel(const __nv_bfloat16* __restrict__ ds, int ld_ds, const __nv_bfloat16* __restrict__ xp,
                   int ld_xp, const __nv_bfloat16* __restrict__ q, int ld_q,
                   const float* __restrict__ coef, __nv_bfloat16* __restrict__ dxp, int ld_dxp,
                   __nv_bfloat16* __restrict__ dgup, int ld_dg, GateGeom g) {
  pdl_trigger();
  pdl_wait();
  typedef Strip<G, QR, 2, 0> S_t;
  S_t S;
  const __nv_bfloat16* const vptr[2] = {ds, xp};
  const int vld[2] = {ld_ds, ld_xp};
  const float* const sptr[1] = {nullptr};
  // the six coefficient rows of gate_bwd_finalize in shared memory (6*C floats behind the ring)
  extern __shared__ __align__(16) uint8_t strip_smem_c[];
  float* s_cf = reinterpret_cast<float*>(strip_smem_c + S_t::kBytes);
  for (int c = threadIdx.x; c < 6 * g.C; c += blockDim.x) s_cf[c] = __ldg(coef + c);
  __syncthreads();
  GateCoef cf;
  cf.sg = s_cf;
  GATE_STRIP_BEGIN(S, g, q, ld_q, vptr, vld, sptr)
#pragma unroll
    for (int gi = 0; gi < G; ++gi) {
      if (S.lane_on(g, gi)) {
        const int cg = S.j + gi * g.tpp;
        const F8 d = S.vec(ho, 0, gi);
        const F8 xv = S.vec(ho, 1, gi);
        const F8 u = S.up(gi);
        F8 ox, og;
        {
          const F8 c0 = cf.get(0, cg, g.C), c1 = cf.get(1, cg, g.C), c2 = cf.get(2, cg, g.C);
#pragma unroll
          for (int k = 0; k < 8; ++k) ox.v[k] = fmaf(c0.v[k], d.v[k], fmaf(c1.v[k], xv.v[k], c2.v[k]));
        }
        {
          const F8 c3 = cf.get(3, cg, g.C), c4 = cf.get(4, cg, g.C), c5 = cf.get(5, cg, g.C);
#pragma unroll
          for (int k = 0; k < 8; ++k) og.v[k] = fmaf(c3.v[k], d.v[k], fmaf(c4.v[k], u.v[k], c5.v[k]));
        }
        store8(dxp + static_cast<size_t>(pix) * ld_dxp + cg * 8, ox);
        store8(dgup + static_cast<size_t>(pix) * ld_dg + cg * 8, og);
      }
    }
  GATE_STRIP_END
}

// ---- launch helpers of the strip kernels
// Ring size of the low-resolution rows: rows h0(ho) .. h1(ho + kD - 1) are alive at once, i.e.
// floor((kD-1) * rh) + 3 of them (rh = (hin-1)/(H-1)); 4 slots cover every up-sampling factor >= 1.5
// (the U-Net's 2x), 8 slots every factor > 0.5.  Down-sampling gates are not an attention-gate geometry.
static int strip_qr(const GateGeom& g) {
  const int alive = static_cast<int>((kD - 1) * static_cast<double>(g.lr.rh) + 1e-4) + 3;
  if (alive <= 4) return 4;
  if (alive <= 8) return 8;
  return 0;
}
// Dynamic shared memory the strip kernels opt in to (their static shared memory stays within the 227 KB of a block).
// A <G, QR> ring plus its coefficient vectors above it cannot launch, so the entry point refuses the shape: at two
// channel groups per thread (Ci > 256) with the 8-row ring, gate_fused_eval (its caller runs gate_psi + gate_apply
// instead) and gate_bwd_xg (Ci > 336).
static constexpr size_t kStripSmemMax = 200 * 1024;
// Opt in to > 48 KB of dynamic shared memory once per (kernel, device).
static int strip_smem_attr(const void* fn, size_t bytes) {
  if (bytes <= 48 * 1024) return 0;
  static std::mutex mu;
  static std::vector<std::pair<const void*, int>> done;
  const int dev = device_index();
  std::lock_guard<std::mutex> lock(mu);
  for (const auto& d : done)
    if (d.first == fn && d.second == dev) return 0;
  cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(kStripSmemMax));
  if (e != cudaSuccess) return static_cast<int>(e);
  done.emplace_back(fn, dev);
  return 0;
}
// Pick the <G, QR> instantiation of a strip kernel template and launch it.
#define GATE_STRIP_DISPATCH(KERNEL, NV, NS, COEF_FLOATS, ...)                                              \
  do {                                                                                                      \
    const int qr_ = strip_qr(g);                                                                            \
    if (qr_ == 0) return UB2_ERR_SHAPE;                                                                     \
    const bool g2_ = g.cgs > g.tpp;                                                                         \
    const size_t coef_ = static_cast<size_t>(COEF_FLOATS) * 4;                                              \
    int rc_ = 0;                                                                                            \
    if (!g2_ && qr_ == 4) {                                                                                 \
      const size_t sm_ = Strip<1, 4, NV, NS>::kBytes + coef_;                                               \
      if (sm_ > kStripSmemMax) return UB2_ERR_SHAPE;                                                        \
      rc_ = strip_smem_attr(reinterpret_cast<const void*>(&KERNEL<1, 4>), sm_);                            \
      if (!rc_) launch(KERNEL<1, 4>, grid, kGateThreads, sm_, s, __VA_ARGS__);                              \
    } else if (!g2_) {                                                                                      \
      const size_t sm_ = Strip<1, 8, NV, NS>::kBytes + coef_;                                               \
      if (sm_ > kStripSmemMax) return UB2_ERR_SHAPE;                                                        \
      rc_ = strip_smem_attr(reinterpret_cast<const void*>(&KERNEL<1, 8>), sm_);                            \
      if (!rc_) launch(KERNEL<1, 8>, grid, kGateThreads, sm_, s, __VA_ARGS__);                              \
    } else if (qr_ == 4) {                                                                                  \
      const size_t sm_ = Strip<2, 4, NV, NS>::kBytes + coef_;                                               \
      if (sm_ > kStripSmemMax) return UB2_ERR_SHAPE;                                                        \
      rc_ = strip_smem_attr(reinterpret_cast<const void*>(&KERNEL<2, 4>), sm_);                            \
      if (!rc_) launch(KERNEL<2, 4>, grid, kGateThreads, sm_, s, __VA_ARGS__);                              \
    } else {                                                                                                \
      const size_t sm_ = Strip<2, 8, NV, NS>::kBytes + coef_;                                               \
      if (sm_ > kStripSmemMax) return UB2_ERR_SHAPE;                                                        \
      rc_ = strip_smem_attr(reinterpret_cast<const void*>(&KERNEL<2, 8>), sm_);                            \
      if (!rc_) launch(KERNEL<2, 8>, grid, kGateThreads, sm_, s, __VA_ARGS__);                              \
    }                                                                                                       \
    if (rc_) return rc_;                                                                                    \
  } while (0)

}  // namespace ub2

using namespace ub2;
typedef const __nv_bfloat16* cbf;
typedef __nv_bfloat16* bf;

extern "C" {

int ub2_gate_rows(int N, int H, int W, int C) {
  GateGeom g;
  int rc = make_gate_geom(&g, N, H, W, C, 1, 1);
  if (rc) return rc;
  return gate_grid(g, 8);
}

int ub2_gate_strip_rows(int N, int H, int W, int C) {
  GateGeom g;
  int rc = make_gate_geom(&g, N, H, W, C, 1, 1);
  if (rc) return rc;
  return gate_strip_grid(g);
}

int ub2_gate_upstats(const void* q, int ld_q, int N, int hin, int win, int H, int W, int Ci,
                     double* partials, int rows, void* stream) {
  GateGeom g;
  int rc = make_gate_geom(&g, N, H, W, Ci, hin, win);
  if (rc) return rc;
  if (partials == nullptr) return UB2_ERR_SHAPE;
  if ((rc = vec_operand(q, ld_q, Ci))) return rc;
  if (!aligned_to(partials, 8)) return UB2_ERR_ALIGN;
  const int grid = gate_strip_grid(g);
  if (grid != rows) return UB2_ERR_WORKSPACE;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  static const int lowres = [] { const char* e = getenv("UB2_UPSTATS_LOWRES"); return e ? atoi(e) : 1; }();
  if (lowres && hin + win <= 4096 && static_cast<double>(N) * hin * win < 2.0e9) {
    // closed form over the low-resolution tensor (gate_upstats_lowres_kernel); same rows, same finalize
    const size_t tab = 3 * static_cast<size_t>(hin + win) * sizeof(float);
    if (g.cgs > g.tpp) launch(gate_upstats_lowres_kernel<2>, grid, kGateThreads, tab, s, static_cast<cbf>(q), ld_q, partials, g);
    else launch(gate_upstats_lowres_kernel<1>, grid, kGateThreads, tab, s, static_cast<cbf>(q), ld_q, partials, g);
    return static_cast<int>(cudaGetLastError());
  }
  GATE_STRIP_DISPATCH(gate_upstats_kernel, 0, 0, 0, static_cast<cbf>(q), ld_q, partials, g);
  return static_cast<int>(cudaGetLastError());
}

int ub2_gate_psi(const void* q, int ld_q, const void* xp, int ld_xp, const float* scale_g,
                 const float* shift_g, const float* scale_x, const float* shift_x, const float* wpsi,
                 float* psi_raw, double* partials, int rows, int N, int hin, int win, int H, int W,
                 int Ci, void* stream) {
  GateGeom g;
  int rc = make_gate_geom(&g, N, H, W, Ci, hin, win);
  if (rc) return rc;
  if (!scale_g || !shift_g || !scale_x || !shift_x || !wpsi || !psi_raw) return UB2_ERR_SHAPE;
  if ((rc = vec_operand(q, ld_q, Ci)) || (rc = vec_operand(xp, ld_xp, Ci))) return rc;
  if (!aligned_to(psi_raw, 4) || !aligned_to(partials, 8)) return UB2_ERR_ALIGN;
  const int grid = gate_strip_grid(g);
  if (partials != nullptr && grid != rows) return UB2_ERR_WORKSPACE;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  GATE_STRIP_DISPATCH(gate_psi_kernel, 1, 0, 4 * Ci, static_cast<cbf>(q), ld_q, static_cast<cbf>(xp), ld_xp, scale_g, shift_g,
                      scale_x, shift_x, wpsi, psi_raw, partials, g);
  return static_cast<int>(cudaGetLastError());
}

int ub2_gate_fused_eval(const void* q, int ld_q, const void* xp, int ld_xp, const void* x, int ld_x, const float* scale_g,
                        const float* shift_g, const float* scale_x, const float* shift_x, const float* wpsi,
                        const float* scale_psi, const float* shift_psi, void* out, int ld_out, int N, int hin, int win,
                        int H, int W, int Ci, int Cx, void* stream) {
  if (Cx != 2 * Ci) return UB2_ERR_SHAPE;   // the fused pass streams the skip as two Ci-channel halves
  GateGeom g;
  int rc = make_gate_geom(&g, N, H, W, Ci, hin, win);
  if (rc) return rc;
  if (!scale_g || !shift_g || !scale_x || !shift_x || !wpsi || !scale_psi || !shift_psi) return UB2_ERR_SHAPE;
  if ((rc = vec_operand(q, ld_q, Ci)) || (rc = vec_operand(xp, ld_xp, Ci)) || (rc = vec_operand(x, ld_x, Cx)) ||
      (rc = vec_operand(out, ld_out, Cx)))
    return rc;
  const int grid = gate_strip_grid(g);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  GATE_STRIP_DISPATCH(gate_fused_eval_kernel, 3, 0, 4 * Ci, static_cast<cbf>(q), ld_q, static_cast<cbf>(xp), ld_xp, static_cast<cbf>(x),
                      ld_x, scale_g, shift_g, scale_x, shift_x, wpsi, scale_psi, shift_psi, static_cast<bf>(out), ld_out, g);
  return static_cast<int>(cudaGetLastError());
}

int ub2_gate_apply(const float* psi_raw, const float* scale_psi, const float* shift_psi, const void* x,
                   int ld_x, void* out, int ld_out, float* a_out, int N, int H, int W, int Cx,
                   void* stream) {
  if (Cx <= 0 || Cx % 8 != 0 || N <= 0 || H <= 0 || W <= 0 || static_cast<double>(N) * H * W * (Cx / 8) >= 2.0e9)
    return UB2_ERR_SHAPE;
  if (!psi_raw || !scale_psi || !shift_psi) return UB2_ERR_SHAPE;
  int rc;
  if ((rc = vec_operand(x, ld_x, Cx)) || (rc = vec_operand(out, ld_out, Cx))) return rc;
  if (!aligned_to(psi_raw, 4) || !aligned_to(a_out, 4)) return UB2_ERR_ALIGN;
  const int pixels = static_cast<int>(N) * H * W;
  launch(gate_apply_kernel, stream_grid(pixels * (Cx / 8), 256, num_sms()), 256, 0, static_cast<cudaStream_t>(stream), psi_raw, scale_psi, shift_psi, static_cast<cbf>(x), ld_x, static_cast<bf>(out), ld_out, a_out, pixels, Cx / 8);
  return static_cast<int>(cudaGetLastError());
}

int ub2_gate_bwd_a(const void* dout, int ld_do, const void* x, int ld_x, const float* a,
                   const float* psi_raw, void* dx, int ld_dx, float* dpsin, double* partials, int rows,
                   int N, int H, int W, int Cx, void* stream) {
  GateGeom g;
  int rc = make_gate_geom(&g, N, H, W, Cx, 1, 1);
  if (rc) return rc;
  if (!a || !psi_raw || !dpsin || !partials) return UB2_ERR_SHAPE;
  if ((rc = vec_operand(dout, ld_do, Cx)) || (rc = vec_operand(x, ld_x, Cx)) || (rc = vec_operand(dx, ld_dx, Cx))) return rc;
  if (!aligned_to(a, 4) || !aligned_to(psi_raw, 4) || !aligned_to(dpsin, 4) || !aligned_to(partials, 8)) return UB2_ERR_ALIGN;
  const int grid = gate_grid(g, 8);
  if (grid != rows) return UB2_ERR_WORKSPACE;
  if (g.cgs > g.tpp)
    launch(gate_bwd_a_kernel<2>, grid, kGateThreads, 0, static_cast<cudaStream_t>(stream), static_cast<cbf>(dout), ld_do, static_cast<cbf>(x), ld_x, a, psi_raw, static_cast<bf>(dx), ld_dx, dpsin, partials, g);
  else
    launch(gate_bwd_a_kernel<1>, grid, kGateThreads, 0, static_cast<cudaStream_t>(stream), static_cast<cbf>(dout), ld_do, static_cast<cbf>(x), ld_x, a, psi_raw, static_cast<bf>(dx), ld_dx, dpsin, partials, g);
  return static_cast<int>(cudaGetLastError());
}

int ub2_gate_bwd_s(const float* dpsin, const float* psi_raw, const float* coef_psi, const void* q,
                   int ld_q, const void* xp, int ld_xp, const float* scale_g, const float* shift_g,
                   const float* scale_x, const float* shift_x, const float* wpsi, void* ds, int ld_ds,
                   double* partials, int rows, int N, int hin, int win, int H, int W, int Ci,
                   void* stream) {
  GateGeom g;
  int rc = make_gate_geom(&g, N, H, W, Ci, hin, win);
  if (rc) return rc;
  if (!dpsin || !psi_raw || !coef_psi || !scale_g || !shift_g || !scale_x || !shift_x || !wpsi || !partials)
    return UB2_ERR_SHAPE;
  if ((rc = vec_operand(q, ld_q, Ci)) || (rc = vec_operand(xp, ld_xp, Ci)) || (rc = vec_operand(ds, ld_ds, Ci))) return rc;
  if (!aligned_to(dpsin, 4) || !aligned_to(psi_raw, 4) || !aligned_to(partials, 8)) return UB2_ERR_ALIGN;
  const int grid = gate_strip_grid(g);
  if (grid != rows) return UB2_ERR_WORKSPACE;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  GATE_STRIP_DISPATCH(gate_bwd_s_kernel, 1, 2, 4 * Ci, dpsin, psi_raw, coef_psi, static_cast<cbf>(q), ld_q, static_cast<cbf>(xp),
                      ld_xp, scale_g, shift_g, scale_x, shift_x, wpsi, static_cast<bf>(ds), ld_ds, partials, g);
  return static_cast<int>(cudaGetLastError());
}

int ub2_gate_bwd_finalize(const double* partials, int rows, int Ci, double count, const float* gamma_x,
                          const float* mean_x, const float* invstd_x, const float* gamma_g,
                          const float* mean_g, const float* invstd_g, int frozen, float* dgamma_x,
                          float* dbeta_x, float* dgamma_g, float* dbeta_g, float* dwpsi, float* coef,
                          void* stream) {
  if (Ci <= 0 || rows <= 0) return UB2_ERR_SHAPE;
  launch(gate_bwd_finalize_kernel, (Ci + 7) / 8, dim3(8, 128), 0, static_cast<cudaStream_t>(stream), partials, rows, Ci, count, gamma_x, mean_x, invstd_x, gamma_g, mean_g, invstd_g, frozen, dgamma_x, dbeta_x, dgamma_g, dbeta_g, dwpsi, coef);
  return static_cast<int>(cudaGetLastError());
}

int ub2_gate_bwd_xg(const void* ds, int ld_ds, const void* xp, int ld_xp, const void* q, int ld_q,
                    const float* coef, void* dxp, int ld_dxp, void* dgup, int ld_dg, int N, int hin,
                    int win, int H, int W, int Ci, void* stream) {
  GateGeom g;
  int rc = make_gate_geom(&g, N, H, W, Ci, hin, win);
  if (rc) return rc;
  if (coef == nullptr) return UB2_ERR_SHAPE;
  if ((rc = vec_operand(ds, ld_ds, Ci)) || (rc = vec_operand(xp, ld_xp, Ci)) || (rc = vec_operand(q, ld_q, Ci)) ||
      (rc = vec_operand(dxp, ld_dxp, Ci)) || (rc = vec_operand(dgup, ld_dg, Ci)))
    return rc;
  const int grid = gate_strip_grid(g);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  GATE_STRIP_DISPATCH(gate_bwd_xg_kernel, 2, 0, 6 * Ci, static_cast<cbf>(ds), ld_ds, static_cast<cbf>(xp), ld_xp, static_cast<cbf>(q),
                      ld_q, coef, static_cast<bf>(dxp), ld_dxp, static_cast<bf>(dgup), ld_dg, g);
  return static_cast<int>(cudaGetLastError());
}

}  // extern "C"
