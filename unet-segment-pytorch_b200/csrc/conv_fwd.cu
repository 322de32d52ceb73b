// NHWC bf16 implicit-GEMM convolution (3x3 pad 1, or 1x1) on tcgen05 tensor cores.
//
//   out[n,h,w,co] = sum_{tap,c} in[n, h+r-1, w+s-1, c] * wgt[co, tap, c]
//
// GEMM view: M = pixels (tiles of 128 = BW x BH x BI box of one TMA load),
// N = Cout (tile BN <= 256), K = taps * (C0 + C1) walked as (tap, channel chunk).
// The channel axis may span two source tensors (skip, upsampled): the
// reference's torch.cat([x2, x1], dim=1) (layers.py:105, :254) is never
// materialised.  The same kernel is the dgrad pass when given the
// tap-flipped / transposed weight pack and the output split over two tensors.
//
// Persistent, warp-specialised: warp 0 = TMA producer, warp 1 = MMA issuer
// (and TMEM owner), warps 2..5 = epilogue.  smem ring of `stages` (A,B) tiles,
// two TMEM accumulator buffers so the epilogue of tile i overlaps the MMAs of
// tile i+1.  Epilogue: optional per-channel affine + ReLU (BN folded for
// inference), optional accumulate into the destination, bf16 store, and
// per-channel sum / sum-of-squares of the rounded outputs (BatchNorm batch
// statistics, layers.py:33) reduced with a register butterfly.
#include "launch.cuh"
#include <cstdlib>
#include "conv.h"
#include "conv_epilogue.cuh"
#include "ptx.cuh"

namespace ub2 {

static constexpr int kMaxStages = 8;
static constexpr int kEpiWarps = 8;                    // 2 per TMEM lane quarter
static constexpr int kThreads = 64 + 32 * kEpiWarps;   // TMA warp + MMA warp + epilogue
static constexpr int kATileBytes = 128 * 64 * 2;       // 16 KB slot

struct FwdSmemHeader {
  uint64_t full[kMaxStages];
  uint64_t empty[kMaxStages];
  uint64_t tmem_full[2];
  uint64_t tmem_empty[2];
  uint32_t tmem_base;
  uint32_t pad;
};

// TAPS: 1 or 9 (unrolled in the producer).  ACC: BatchNorm statistics are kept as per-thread
// running sums over all tiles of the CTA and reduced across lanes once at the end (needs one
// 32-column chunk per epilogue warp: Cout <= 64); otherwise a register butterfly per tile.
template <int TAPS, bool ACC, bool TF32>
__global__ void __launch_bounds__(kThreads, 1)
conv_fwd_kernel(const __grid_constant__ CUtensorMap tmA0, const __grid_constant__ CUtensorMap tmA1,
                const __grid_constant__ CUtensorMap tmB, const ConvFwdParams p) {
  pdl_trigger();
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  // 1024-align the tile ring (128B swizzle atoms repeat every 1024 B).
  uint8_t* tiles = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                              ~static_cast<uintptr_t>(1023));
  const int stage_bytes = p.stage_bytes;
  const int stages = p.stages;
  FwdSmemHeader* hdr = reinterpret_cast<FwdSmemHeader*>(tiles + stages * stage_bytes);
  float* s_stats = reinterpret_cast<float*>(hdr + 1);  // [4 quarters][2][Cout]

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int C0 = p.C0;
  const int Ctot = p.C0 + p.C1;
  const int kc = p.kc;
  // each source is walked in whole kc chunks (C0p, C1p: its channel count rounded up to kc); channels past a
  // source's end are zero-filled by its tensor map, so the weight columns they meet contribute nothing
  const int C0p = (C0 + kc - 1) & -kc;
  const int Ckp = C0p + ((p.C1 + kc - 1) & -kc);
  const int kchunks = Ckp / kc;
  const int tiles_m = p.tiles_w * p.tiles_h * p.tiles_n;
  const int n_tiles = p.n_tiles;
  const int total_tiles = tiles_m * n_tiles;
  const int BN = p.BN;
  const int bn_cols = (BN + 31) & ~31;  // TMEM columns per accumulator buffer

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA0);
    if (p.C1 > 0) tma_prefetch_desc(&tmA1);
    tma_prefetch_desc(&tmB);
    for (int i = 0; i < stages; ++i) {
      mbar_init(&hdr->full[i], 1);
      mbar_init(&hdr->empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&hdr->tmem_full[i], 1);
      mbar_init(&hdr->tmem_empty[i], kEpiWarps);
    }
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc(&hdr->tmem_base, p.tmem_cols);
  if (warp >= 2 && p.stats != nullptr) {
    for (int i = threadIdx.x - 64; i < 4 * 2 * p.Cout; i += 32 * kEpiWarps) s_stats[i] = 0.f;
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = hdr->tmem_base;
  pdl_wait();   // the prologue above touched no global memory; everything below may (launch.cuh)

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer
    // Warp-uniform control flow, one elected lane issues: keeps every operand in uniform
    // registers (a single-thread loop costs ~10x the instructions per k-step).
    const uint32_t esz = TF32 ? 4u : 2u;
    const uint32_t tx_bytes = 128u * kc * esz + static_cast<uint32_t>(BN) * kc * esz;
    const int tw = p.tiles_w, th = p.tiles_h, BW = p.BW, BH = p.BH, BI = p.BI;
    int stage = 0;
    uint32_t phase = 0;
    for (int t = blockIdx.x; t < total_tiles; t += gridDim.x) {
      const int nt = t % n_tiles;
      const int mt = t / n_tiles;
      const int w0 = (mt % tw) * BW;
      const int h0 = ((mt / tw) % th) * BH;
      const int i0 = (mt / (tw * th)) * BI;
      const int n0 = nt * BN;
#pragma unroll
      for (int tap = 0; tap < TAPS; ++tap) {
        const int dr = (TAPS == 9) ? tap / 3 - 1 : 0;
        const int ds = (TAPS == 9) ? tap % 3 - 1 : 0;
        for (int c = 0; c < Ckp; c += kc) {
          mbar_wait(&hdr->empty[stage], phase ^ 1);
          if (elect_one()) {
            uint8_t* sa = tiles + stage * stage_bytes;
            mbar_expect_tx(&hdr->full[stage], tx_bytes);
            if (c < C0p) {
              tma_load_4d(sa, &tmA0, &hdr->full[stage], c, w0 + ds, h0 + dr, i0);
              tma_load_2d(sa + kATileBytes, &tmB, &hdr->full[stage], tap * Ctot + c, n0);
            } else {
              tma_load_4d(sa, &tmA1, &hdr->full[stage], c - C0p, w0 + ds, h0 + dr, i0);
              tma_load_2d(sa + kATileBytes, &tmB, &hdr->full[stage], tap * Ctot + C0 + (c - C0p), n0);
            }
          }
          if (++stage == stages) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer
    const uint32_t idesc = TF32 ? make_idesc_tf32(128, BN) : make_idesc_bf16(128, BN, 0, 0);
    const uint32_t row_bytes = static_cast<uint32_t>(kc) * (TF32 ? 4u : 2u);   // one K chunk of a row
    const uint32_t ltype = (row_bytes == 128) ? 2u : (row_bytes == 64) ? 4u : 6u;
    // descriptor = {hi: SBO (8 rows of one K chunk) | version 1 | swizzle, lo: addr>>4 | LBO 1}
    const uint32_t desc_hi = ((8u * row_bytes) >> 4) | (1u << 14) | (ltype << 29);
    const uint32_t a_lo0 = ((smem_u32(tiles) & 0x3FFFFu) >> 4) | (1u << 16);
    const uint32_t b_lo0 = a_lo0 + (kATileBytes >> 4);
    const uint32_t stage_inc = static_cast<uint32_t>(stage_bytes) >> 4;
    const int kinner = static_cast<int>(row_bytes / 32);   // 32 bytes of K per MMA (16 bf16 or 8 tf32)
    const int ksteps = TAPS * kchunks;
    int stage = 0;
    uint32_t phase = 0;
    int it = 0;
    for (int t = blockIdx.x; t < total_tiles; t += gridDim.x, ++it) {
      const int as = it & 1;
      mbar_wait(&hdr->tmem_empty[as], ((it >> 1) & 1) ^ 1);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + as * bn_cols;
      for (int ks = 0; ks < ksteps; ++ks) {
        mbar_wait(&hdr->full[stage], phase);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t a_lo = a_lo0 + stage * stage_inc;
          const uint32_t b_lo = b_lo0 + stage * stage_inc;
          for (int k = 0; k < kinner; ++k) {
            const uint64_t da = (static_cast<uint64_t>(desc_hi) << 32) | (a_lo + 2 * k);
            const uint64_t db = (static_cast<uint64_t>(desc_hi) << 32) | (b_lo + 2 * k);
            if (TF32) umma_tf32(d_tmem, da, db, idesc, (ks | k) != 0);
            else umma_bf16(d_tmem, da, db, idesc, (ks | k) != 0);
          }
          umma_commit(&hdr->empty[stage]);
          if (ks == ksteps - 1) umma_commit(&hdr->tmem_full[as]);
        }
        __syncwarp();
        if (++stage == stages) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else {
    // ------------------------------------------------------------ epilogue
    const int q = warp & 3;          // TMEM lane quarter this warp may read
    const int grp = (warp - 2) >> 2; // column group: chunks j with (j & 1) == grp
    const int row = q * 32 + lane;
    const int w_l = row % p.BW;
    const int h_l = (row / p.BW) % p.BH;
    const int i_l = row / (p.BW * p.BH);
    const int nchunks = bn_cols / 32;
    const bool want_stats = p.stats != nullptr;
    float* my_stats = s_stats + q * 2 * p.Cout;
    float acc_s[ACC ? 32 : 1], acc_q[ACC ? 32 : 1];
    if (ACC) {
#pragma unroll
      for (int i = 0; i < (ACC ? 32 : 1); ++i) acc_s[i] = acc_q[i] = 0.f;
    }
    int it = 0;
    for (int t = blockIdx.x; t < total_tiles; t += gridDim.x, ++it) {
      const int nt = t % n_tiles;
      const int mt = t / n_tiles;
      const int w = (mt % p.tiles_w) * p.BW + w_l;
      const int h = ((mt / p.tiles_w) % p.tiles_h) * p.BH + h_l;
      const int n = (mt / (p.tiles_w * p.tiles_h)) * p.BI + i_l;
      const int n0 = nt * BN;
      const bool valid = (w < p.W) && (h < p.H) && (n < p.N);
      const size_t pix = (static_cast<size_t>(n) * p.H + h) * p.W + w;
      const int as = it & 1;
      mbar_wait(&hdr->tmem_full[as], (it >> 1) & 1);
      tc_fence_after();
      for (int j = grp; j < nchunks; j += 2) {
        epi_chunk<ACC, TF32>(p, tmem_base + (static_cast<uint32_t>(q * 32) << 16) + as * bn_cols + j * 32,
                       n0 + j * 32, n0 + BN, valid, pix, lane, want_stats, my_stats, acc_s, acc_q);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&hdr->tmem_empty[as]);
    }
    if (want_stats)
      epi_finish<ACC, 32 * kEpiWarps>(p, s_stats, my_stats, lane, grp, nchunks, threadIdx.x - 64, acc_s, acc_q);
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, p.tmem_cols);
  }
}

// ---------------------------------------------------------------------------------------
// host side

static int pow2_floor(int x) {
  int r = 1;
  while (r * 2 <= x) r *= 2;
  return r;
}

int conv_fwd2_launch(const ConvFwdArgs& a, cudaStream_t stream);   // conv_fwd2.cu: cta_group::2 variant

int conv_fwd_launch(const ConvFwdArgs& a, cudaStream_t stream) {
  if (!a.tf32) {
    // wide 3x3 layers: halo block resident in shared memory (conv_halo.cu)
    const int rc = conv_halo_launch(a, stream);
    if (rc != 1) return rc;
  }
  {
    // the remaining bf16 layers with 64-channel chunks: two-CTA kernel sharing the weight tile
    const int rc = conv_fwd2_launch(a, stream);
    if (rc != 1) return rc;
  }
  const int Ctot = a.C0 + a.C1;
  const int esz = a.tf32 ? 4 : 2;
  if (a.taps != 1 && a.taps != 9) return UB2_ERR_SHAPE;
  if (a.N <= 0 || a.H <= 0 || a.W <= 0 || a.C0 <= 0 || a.C1 < 0) return UB2_ERR_SHAPE;
  // output channels in multiples of 8 (one 16-byte store); each source's weight-pack columns start on 16 bytes
  // (a TMA box may not start inside a 16-byte unit): C0 and C1 multiples of 8 bf16 / 4 fp32 channels
  if (a.Cout % 8 != 0) return UB2_ERR_SHAPE;
  if (a.ld_in0 % 8 != 0 || (a.C1 > 0 && a.ld_in1 % 8 != 0) || a.ld0 % 8 != 0) return UB2_ERR_ALIGN;
  if ((a.C0 * esz) % 16 != 0 || (a.C1 * esz) % 16 != 0) return UB2_ERR_ALIGN;
  if (a.tf32 && (a.stats != nullptr || a.accumulate || a.out1 != nullptr)) return UB2_ERR_SHAPE;  // eval only
  // channels per K chunk: 128 bytes, halved while it does not divide both sources, down to 32 bytes (the MMA K);
  // sources that are not a multiple of the chunk are padded to it (zero fill of the activation tensor maps)
  int kc = 128 / esz;
  while (kc > 32 / esz && (a.C0 % kc != 0 || Ctot % kc != 0)) kc /= 2;

  ConvFwdParams p{};
  p.N = a.N; p.H = a.H; p.W = a.W;
  p.C0 = a.C0; p.C1 = a.C1; p.Cout = a.Cout;
  p.taps = a.taps; p.kc = kc;
  p.BW = pow2_floor(a.W < 128 ? a.W : 128);
  p.BH = pow2_floor(a.H < 128 / p.BW ? a.H : 128 / p.BW);
  p.BI = 128 / (p.BW * p.BH);
  p.tiles_w = (a.W + p.BW - 1) / p.BW;
  p.tiles_h = (a.H + p.BH - 1) / p.BH;
  p.tiles_n = (a.N + p.BI - 1) / p.BI;
  // N tile: whole Cout (rounded up to the MMA's multiple of 16; the weight tensor map zero-fills the rows past
  // Cout) when it fits one accumulator buffer; must divide the split point.
  int BN = a.Cout <= 256 ? (a.Cout + 15) & ~15 : 256;
  const int split = (a.out1 != nullptr) ? a.split : (1 << 30);
  if (a.out1 != nullptr) {
    if (a.split % 8 != 0 || a.ld1 % 8 != 0) return UB2_ERR_ALIGN;
  }
  {
    // few pixel tiles (deep layers at small batch): halve the N tile so that the grid covers the SMs
    const int m_tiles = p.tiles_w * p.tiles_h * p.tiles_n;
    while (BN > 64 && BN % 32 == 0 && a.Cout % (BN / 2) == 0 && (split == (1 << 30) || split % (BN / 2) == 0) &&
           m_tiles * ((a.Cout + BN - 1) / BN) * 2 <= num_sms())
      BN /= 2;
  }
  if (a.bn_override > 0) BN = a.bn_override;
  if (BN % 16 != 0 || BN > 256) return UB2_ERR_SHAPE;
  p.BN = BN;
  p.n_tiles = (a.Cout + BN - 1) / BN;
  const int bn_cols = (BN + 31) & ~31;
  int tmem_cols = 32;
  while (tmem_cols < 2 * bn_cols) tmem_cols *= 2;
  p.tmem_cols = tmem_cols;
  const int b_bytes = ((BN * kc * esz) + 1023) & ~1023;
  p.stage_bytes = kATileBytes + b_bytes;
  const int stats_bytes = a.stats ? 4 * 2 * a.Cout * 4 : 0;
  const int budget = 227 * 1024 - 1024 - static_cast<int>(sizeof(FwdSmemHeader)) - stats_bytes;
  int stages = budget / p.stage_bytes;
  if (stages > kMaxStages) stages = kMaxStages;
  if (stages < 2) return UB2_ERR_SHAPE;
  p.stages = stages;
  p.out0 = reinterpret_cast<__nv_bfloat16*>(a.out0); p.ld0 = a.ld0;
  p.out1 = reinterpret_cast<__nv_bfloat16*>(a.out1); p.ld1 = a.ld1; p.split = split;
  p.accumulate = a.accumulate;
  p.scale = a.scale; p.shift = a.shift; p.relu = a.relu;
  p.stats = a.stats;
  p.tf32 = a.tf32;
  {
    static const int wide_env = [] { const char* e = getenv("UB2_WIDE_STORE"); return e ? atoi(e) : 1; }();
    p.wide_store = wide_env && conv_wide_store_ok(a.out0, a.ld0, a.out1, a.ld1, a.split, a.Cout);
  }

  CUtensorMap tmA0, tmA1, tmB;
  const uint32_t boxA[4] = {static_cast<uint32_t>(kc), static_cast<uint32_t>(p.BW),
                            static_cast<uint32_t>(p.BH), static_cast<uint32_t>(p.BI)};
  int rc = make_tmap_nhwc(&tmA0, a.in0, a.N, a.H, a.W, a.C0, a.ld_in0, boxA, kc * esz, esz);
  if (rc) return rc;
  if (a.C1 > 0) {
    rc = make_tmap_nhwc(&tmA1, a.in1, a.N, a.H, a.W, a.C1, a.ld_in1, boxA, kc * esz, esz);
    if (rc) return rc;
  } else {
    tmA1 = tmA0;
  }
  rc = make_tmap_2d(&tmB, a.wgt, static_cast<uint64_t>(a.taps) * Ctot, a.Cout,
                    static_cast<uint64_t>(a.taps) * Ctot, kc, BN, kc * esz, esz);
  if (rc) return rc;

  const int total_tiles = p.tiles_w * p.tiles_h * p.tiles_n * p.n_tiles;
  int grid = num_sms();
  if (a.grid_override > 0) grid = a.grid_override;
  if (grid > total_tiles) grid = total_tiles;
  if (a.stats && grid > a.stats_rows) return UB2_ERR_WORKSPACE;
  const size_t smem = 1024 + static_cast<size_t>(stages) * p.stage_bytes + sizeof(FwdSmemHeader) +
                      stats_bytes;
  static PerDevice<bool> attr_set_pd;
  bool& attr_set = attr_set_pd.ref();
  if (!attr_set) {
    cudaError_t e = cudaSuccess;
    const int lim = 227 * 1024;
    const auto attr = cudaFuncAttributeMaxDynamicSharedMemorySize;
    if (e == cudaSuccess) e = cudaFuncSetAttribute(conv_fwd_kernel<9, true, false>, attr, lim);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(conv_fwd_kernel<9, false, false>, attr, lim);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(conv_fwd_kernel<1, true, false>, attr, lim);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(conv_fwd_kernel<1, false, false>, attr, lim);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(conv_fwd_kernel<9, false, true>, attr, lim);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(conv_fwd_kernel<1, false, true>, attr, lim);
    if (e != cudaSuccess) return static_cast<int>(e);
    attr_set = true;
  }
  // running-sum statistics need one 32-column chunk per epilogue warp and a single N tile
  const bool acc = a.stats != nullptr && bn_cols <= 64 && p.n_tiles == 1;
  note_variant(1);
  if (a.tf32) {
    if (a.taps == 9) launch(conv_fwd_kernel<9, false, true>, grid, kThreads, smem, stream, tmA0, tmA1, tmB, p);
    else launch(conv_fwd_kernel<1, false, true>, grid, kThreads, smem, stream, tmA0, tmA1, tmB, p);
  } else if (a.taps == 9) {
    if (acc) launch(conv_fwd_kernel<9, true, false>, grid, kThreads, smem, stream, tmA0, tmA1, tmB, p);
    else launch(conv_fwd_kernel<9, false, false>, grid, kThreads, smem, stream, tmA0, tmA1, tmB, p);
  } else {
    if (acc) launch(conv_fwd_kernel<1, true, false>, grid, kThreads, smem, stream, tmA0, tmA1, tmB, p);
    else launch(conv_fwd_kernel<1, false, false>, grid, kThreads, smem, stream, tmA0, tmA1, tmB, p);
  }
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return static_cast<int>(e);
  if (a.grid_used) *a.grid_used = grid;
  return 0;
}

}  // namespace ub2
