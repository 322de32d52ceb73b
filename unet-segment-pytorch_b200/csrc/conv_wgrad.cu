// Weight-gradient implicit GEMM on tcgen05 tensor cores.
//
//   dW[tap, c, co] = sum_{n,h,w} in[n, h+r-1, w+s-1, c] * dy[n,h,w,co]
//
// GEMM view: M = taps*(C0+C1) (im2col rows, tile 128), N = Cout (tile BN <= 256),
// K = pixels, walked in chunks of 64 (one TMA box BW x BH x BI).  A source whose channel count is
// not a multiple of the mc-channel A sub-box is padded to whole sub-boxes per tap (M rows that the
// tensor map zero-fills and the epilogue drops), so the partial layout keeps the real rows only.  Both operands
// are read exactly as the activations lie in HBM (NHWC: channels contiguous), i.e.
// MN-major shared-memory tiles — no transposed copies.  Split-K over pixels: each
// work item (m tile, n tile, split) writes an fp32 partial tile; a second kernel
// reduces the splits in a fixed order (deterministic) into the OIHW fp32 gradient.
#include "launch.cuh"
#include "conv.h"
#include "ptx.cuh"

namespace ub2 {

static constexpr int kWMaxStages = 8;
static constexpr int kWThreads = 192;
static constexpr int kKPix = 64;                  // pixels per pipeline stage
static constexpr int kWATileBytes = 128 * kKPix * 2;  // 16 KB

struct WgSmemHeader {
  uint64_t full[kWMaxStages];
  uint64_t empty[kWMaxStages];
  uint64_t tmem_full[2];
  uint64_t tmem_empty[2];
  uint32_t tmem_base;
  uint32_t pad;
};

__global__ void __launch_bounds__(kWThreads, 1)
conv_wgrad_kernel(const __grid_constant__ CUtensorMap tmA0, const __grid_constant__ CUtensorMap tmA1,
                  const __grid_constant__ CUtensorMap tmDY, const ConvWgradParams p) {
  pdl_trigger();
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* tiles = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                              ~static_cast<uintptr_t>(1023));
  WgSmemHeader* hdr = reinterpret_cast<WgSmemHeader*>(tiles + p.stages * p.stage_bytes);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int Ctot = p.C0 + p.C1;
  const int Mtot = p.taps * Ctot;
  const int C0p = (p.C0 + p.mc - 1) & -p.mc;                 // sources padded to whole A sub-boxes
  const int Ctp = C0p + ((p.C1 + p.mc - 1) & -p.mc);
  const int Mp = p.taps * Ctp;                              // padded M rows
  const int total_chunks = p.chunks_w * p.chunks_h * p.chunks_n;
  const int per_split = (total_chunks + p.splits - 1) / p.splits;
  const int total_items = p.m_tiles * p.n_tiles * p.splits;
  const int bn_cols = (p.BN + 31) & ~31;
  const int a_subs = 128 / p.mc;
  const int b_subs = (p.BN + 63) / 64;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA0);
    if (p.C1 > 0) tma_prefetch_desc(&tmA1);
    tma_prefetch_desc(&tmDY);
    for (int i = 0; i < p.stages; ++i) {
      mbar_init(&hdr->full[i], 1);
      mbar_init(&hdr->empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&hdr->tmem_full[i], 1);
      mbar_init(&hdr->tmem_empty[i], 4);
    }
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc(&hdr->tmem_base, p.tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = hdr->tmem_base;
  pdl_wait();   // the prologue above touched no global memory; everything below may (launch.cuh)

  // item -> (split, n tile, m tile); m fastest so CTAs running together share dy tiles in L2.
  // Producer and MMA warps run warp-uniform loops with one elected lane issuing, so operands
  // stay in uniform registers (single-thread loops cost several hundred cycles per stage).
  if (warp == 0) {
    const uint32_t tx_bytes = kWATileBytes + static_cast<uint32_t>(b_subs) * p.b_sub_bytes;
    const int cw_n = p.chunks_w, ch_n = p.chunks_h;
    int stage = 0;
    uint32_t phase = 0;
    for (int it = blockIdx.x; it < total_items; it += gridDim.x) {
      const int mt = it % p.m_tiles;
      const int nt = (it / p.m_tiles) % p.n_tiles;
      const int sp = it / (p.m_tiles * p.n_tiles);
      const int ch_begin = sp * per_split;
      const int ch_end = min(ch_begin + per_split, total_chunks);
      // per sub-box (channel offset, tap shift, source) of this m tile: lane j owns sub-box j
      int sub_c = 0, sub_ds = 0, sub_dr = 0;
      if (lane < a_subs) {
        int m = mt * 128 + lane * p.mc;
        if (m >= Mp) m = Mp - p.mc;  // rows past the end are discarded by the epilogue
        const int tap = m / Ctp;
        sub_c = m % Ctp;
        sub_dr = (p.taps == 9) ? tap / 3 - 1 : 0;
        sub_ds = (p.taps == 9) ? tap % 3 - 1 : 0;
      }
      int cw = ch_begin % cw_n;
      int chh = (ch_begin / cw_n) % ch_n;
      int cn = ch_begin / (cw_n * ch_n);
      for (int ch = ch_begin; ch < ch_end; ++ch) {
        const int w0 = cw * p.BW, h0 = chh * p.BH, i0 = cn * p.BI;
        mbar_wait(&hdr->empty[stage], phase ^ 1);
        uint8_t* sa = tiles + stage * p.stage_bytes;
        if (lane == 0) mbar_expect_tx(&hdr->full[stage], tx_bytes);
        __syncwarp();
        if (lane < a_subs) {
          if (sub_c < C0p)
            tma_load_4d(sa + lane * p.a_sub_bytes, &tmA0, &hdr->full[stage], sub_c, w0 + sub_ds,
                        h0 + sub_dr, i0);
          else
            tma_load_4d(sa + lane * p.a_sub_bytes, &tmA1, &hdr->full[stage], sub_c - C0p, w0 + sub_ds,
                        h0 + sub_dr, i0);
        } else if (lane - a_subs < b_subs) {
          const int j = lane - a_subs;
          tma_load_4d(sa + kWATileBytes + j * p.b_sub_bytes, &tmDY, &hdr->full[stage], nt * p.BN + j * 64,
                      w0, h0, i0);
        }
        if (++cw == cw_n) {
          cw = 0;
          if (++chh == ch_n) {
            chh = 0;
            ++cn;
          }
        }
        if (++stage == p.stages) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else if (warp == 1) {
    const uint32_t idesc = make_idesc_bf16(128, p.BN, 1, 1);  // both operands MN-major
    const uint32_t a_pitch = p.mc * 2;                        // bytes per pixel row in an A sub-box
    const uint32_t a_ltype = (p.mc == 64) ? 2u : (p.mc == 32) ? 4u : 6u;
    // descriptors: hi = SBO (8 pixel rows) | version | swizzle ; lo = addr>>4 | LBO (sub-box stride)
    const uint32_t a_hi = ((8 * a_pitch) >> 4) | (1u << 14) | (a_ltype << 29);
    const uint32_t b_hi = (1024u >> 4) | (1u << 14) | (2u << 29);
    const uint32_t a_lo0 = ((smem_u32(tiles) & 0x3FFFFu) >> 4) | ((static_cast<uint32_t>(p.a_sub_bytes) >> 4) << 16);
    const uint32_t b_lo0 = (((smem_u32(tiles) + kWATileBytes) & 0x3FFFFu) >> 4) |
                           ((static_cast<uint32_t>(p.b_sub_bytes) >> 4) << 16);
    const uint32_t a_kadv = (16 * a_pitch) >> 4;
    const uint32_t stage_inc = static_cast<uint32_t>(p.stage_bytes) >> 4;
    int stage = 0;
    uint32_t phase = 0;
    int n = 0;
    for (int it = blockIdx.x; it < total_items; it += gridDim.x, ++n) {
      const int sp = it / (p.m_tiles * p.n_tiles);
      const int ch_begin = sp * per_split;
      const int ch_end = min(ch_begin + per_split, total_chunks);
      const int as = n & 1;
      mbar_wait(&hdr->tmem_empty[as], ((n >> 1) & 1) ^ 1);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + as * bn_cols;
      for (int ch = ch_begin; ch < ch_end; ++ch) {
        mbar_wait(&hdr->full[stage], phase);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t a_lo = a_lo0 + stage * stage_inc;
          const uint32_t b_lo = b_lo0 + stage * stage_inc;
#pragma unroll
          for (int k = 0; k < kKPix / 16; ++k) {
            const uint64_t da = (static_cast<uint64_t>(a_hi) << 32) | (a_lo + k * a_kadv);
            const uint64_t db = (static_cast<uint64_t>(b_hi) << 32) | (b_lo + k * (2048u >> 4));
            umma_bf16(d_tmem, da, db, idesc, (ch > ch_begin) || (k > 0));
          }
          umma_commit(&hdr->empty[stage]);
          if (ch == ch_end - 1) umma_commit(&hdr->tmem_full[as]);
        }
        __syncwarp();
        if (++stage == p.stages) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else {
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const int nchunks = bn_cols / 32;
    int n = 0;
    for (int it = blockIdx.x; it < total_items; it += gridDim.x, ++n) {
      const int mt = it % p.m_tiles;
      const int nt = (it / p.m_tiles) % p.n_tiles;
      const int sp = it / (p.m_tiles * p.n_tiles);
      const int ch_begin = sp * per_split;
      const int as = n & 1;
      // padded row -> (tap, source channel) -> row of the partial tile; padding rows are not stored
      const int mp = mt * 128 + row;
      const int cp = mp % Ctp;
      const int cs = cp < C0p ? cp : cp - C0p;
      const int m = (mp / Ctp) * Ctot + (cp < C0p ? cp : p.C0 + cs);
      const bool real = mp < Mp && cs < (cp < C0p ? p.C0 : p.C1);
      const bool empty_split = ch_begin >= total_chunks;  // host never creates one; be safe
      mbar_wait(&hdr->tmem_full[as], (n >> 1) & 1);
      tc_fence_after();
      float* dst_row = p.partial + (static_cast<size_t>(sp) * Mtot + m) * p.Cout;
      for (int j = 0; j < nchunks; ++j) {
        uint32_t raw[32];
        tmem_ld32(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + as * bn_cols + j * 32, raw);
        tmem_ld_wait();
        const int cbase = nt * p.BN + j * 32;
        if (real) {
#pragma unroll
          for (int g = 0; g < 8; ++g) {
            const int c = cbase + g * 4;
            if (c < p.Cout && c < (nt + 1) * p.BN) {
              float4 o;
              o.x = empty_split ? 0.f : __uint_as_float(raw[g * 4 + 0]);
              o.y = empty_split ? 0.f : __uint_as_float(raw[g * 4 + 1]);
              o.z = empty_split ? 0.f : __uint_as_float(raw[g * 4 + 2]);
              o.w = empty_split ? 0.f : __uint_as_float(raw[g * 4 + 3]);
              *reinterpret_cast<float4*>(dst_row + c) = o;
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&hdr->tmem_empty[as]);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, p.tmem_cols);
  }
}

static int pow2_floor_w(int x) {
  int r = 1;
  while (r * 2 <= x) r *= 2;
  return r;
}

int conv_wgrad_halo_launch(const ConvWgradArgs& a, cudaStream_t stream);
int conv_wgrad2_launch(const ConvWgradArgs& a, cudaStream_t stream);
extern int g_conv_mode_wgrad;

int conv_wgrad_launch(const ConvWgradArgs& a, cudaStream_t stream) {
  if (g_conv_mode_wgrad != 1) {
    const int rc = conv_wgrad_halo_launch(a, stream);
    if (rc != 1) return rc;
  }
  const int Ctot = a.C0 + a.C1;
  if (a.taps != 1 && a.taps != 9) return UB2_ERR_SHAPE;
  if (a.N <= 0 || a.H <= 0 || a.W <= 0 || a.C0 <= 0 || a.C1 < 0) return UB2_ERR_SHAPE;
  if (a.Cout % 8 != 0) return UB2_ERR_SHAPE;   // any source channel count; Cout in 16-byte rows of dy
  if (g_conv_mode_wgrad != 1) {   // deep layers: two-CTA kernel sharing dy (conv_wgrad2.cu)
    const int rc2 = conv_wgrad2_launch(a, stream);
    if (rc2 != 1) return rc2;
  }
  if (a.ld_in0 % 8 != 0 || (a.C1 > 0 && a.ld_in1 % 8 != 0) || a.ld_dy % 8 != 0) return UB2_ERR_ALIGN;
  // channels per A sub-box: 64, halved while it does not divide both sources, down to 16 (32 bytes: there is no
  // 16-byte swizzle); sources that are not a multiple of it are padded to whole sub-boxes
  int mc = 64;
  while (mc > 16 && (a.C0 % mc != 0 || Ctot % mc != 0)) mc /= 2;
  const int C0p = (a.C0 + mc - 1) / mc * mc;
  const int Mp = a.taps * (C0p + (a.C1 + mc - 1) / mc * mc);

  ConvWgradParams p{};
  p.N = a.N; p.H = a.H; p.W = a.W; p.C0 = a.C0; p.C1 = a.C1; p.Cout = a.Cout; p.taps = a.taps;
  p.mc = mc;
  p.BW = pow2_floor_w(a.W < kKPix ? a.W : kKPix);
  p.BH = pow2_floor_w(a.H < kKPix / p.BW ? a.H : kKPix / p.BW);
  p.BI = kKPix / (p.BW * p.BH);
  p.chunks_w = (a.W + p.BW - 1) / p.BW;
  p.chunks_h = (a.H + p.BH - 1) / p.BH;
  p.chunks_n = (a.N + p.BI - 1) / p.BI;
  const int total_chunks = p.chunks_w * p.chunks_h * p.chunks_n;
  p.m_tiles = (Mp + 127) / 128;
  // N tile rounded up to the MMA's multiple of 16: dy's tensor map zero-fills the channels past Cout
  const int BN = a.Cout <= 256 ? (a.Cout + 15) & ~15 : 256;
  p.BN = BN;
  p.n_tiles = (a.Cout + BN - 1) / BN;
  const int bn_cols = (BN + 31) & ~31;
  int tmem_cols = 32;
  while (tmem_cols < 2 * bn_cols) tmem_cols *= 2;
  p.tmem_cols = tmem_cols;
  p.a_sub_bytes = kKPix * mc * 2;
  p.b_sub_bytes = kKPix * 64 * 2;
  const int b_subs = (BN + 63) / 64;
  p.stage_bytes = kWATileBytes + b_subs * p.b_sub_bytes;
  int stages = (wgrad_smem_budget() - 1024 - static_cast<int>(sizeof(WgSmemHeader))) / p.stage_bytes;
  if (stages > kWMaxStages) stages = kWMaxStages;
  p.stages = stages;

  // split K so that the grid is one full wave of work items, each with >= 4 pixel chunks
  const int tiles = p.m_tiles * p.n_tiles;
  const int sms = num_sms();
  int splits = sms / tiles;
  if (splits > total_chunks / 4) splits = total_chunks / 4;
  if (splits < 1) splits = 1;
  if (a.splits_override > 0) splits = a.splits_override;
  if (splits > total_chunks) splits = total_chunks;
  if (splits > a.max_splits) splits = a.max_splits;
  // no empty trailing split
  const int per = (total_chunks + splits - 1) / splits;
  splits = (total_chunks + per - 1) / per;
  p.splits = splits;
  p.partial = a.partial;

  CUtensorMap tmA0, tmA1, tmDY;
  const uint32_t boxA[4] = {static_cast<uint32_t>(mc), static_cast<uint32_t>(p.BW),
                            static_cast<uint32_t>(p.BH), static_cast<uint32_t>(p.BI)};
  const uint32_t boxB[4] = {64u, static_cast<uint32_t>(p.BW), static_cast<uint32_t>(p.BH),
                            static_cast<uint32_t>(p.BI)};
  int rc = make_tmap_nhwc(&tmA0, a.in0, a.N, a.H, a.W, a.C0, a.ld_in0, boxA, mc * 2);
  if (rc) return rc;
  if (a.C1 > 0) {
    rc = make_tmap_nhwc(&tmA1, a.in1, a.N, a.H, a.W, a.C1, a.ld_in1, boxA, mc * 2);
    if (rc) return rc;
  } else {
    tmA1 = tmA0;
  }
  rc = make_tmap_nhwc(&tmDY, a.dy, a.N, a.H, a.W, a.Cout, a.ld_dy, boxB, 128);
  if (rc) return rc;

  const int total_items = tiles * splits;
  int grid = sms < total_items ? sms : total_items;
  const size_t smem = 1024 + static_cast<size_t>(stages) * p.stage_bytes + sizeof(WgSmemHeader);
  static PerDevice<bool> attr_set_pd;
  bool& attr_set = attr_set_pd.ref();
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(conv_wgrad_kernel,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e != cudaSuccess) return static_cast<int>(e);
    attr_set = true;
  }
  note_variant(11);
  launch_co(conv_wgrad_kernel, grid, kWThreads, smem, stream, tmA0, tmA1, tmDY, p);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return static_cast<int>(e);
  if (a.splits_used) *a.splits_used = splits;
  return 0;
}

}  // namespace ub2
