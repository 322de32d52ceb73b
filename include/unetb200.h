/* libunetb200 — C ABI of the B200 (sm_100a) Attention U-Net hot path.
 *
 * Boundary contract (SURVEY.md §8b):
 *  - plain pointers and sizes only, no torch / C++ types; every entry point returns 0 on
 *    success, a positive cudaError_t, or a negative UB2_ERR_* code (the *_rows / *_blocks
 *    queries return a positive count instead); no exception crosses the boundary;
 *  - the library never allocates, frees or retains device memory: activations, gradients,
 *    statistics and workspaces are owned by the caller (torch's caching allocator);
 *  - every call is asynchronous on the passed cudaStream_t (as void*), never synchronises
 *    the device and is re-entrant (autograd calls the backward entry points from its own
 *    thread); a whole training step can therefore be captured into a CUDA graph;
 *  - activations are NHWC bf16 "(N,H,W,C), channel stride ld" (ld in elements, multiple of 8,
 *    base pointers 16-byte aligned); parameters stay in the reference's fp32 OIHW layout and
 *    are packed to bf16 by ub2_pack_conv_weight; per-channel vectors are fp32;
 *  - reductions are deterministic: kernels write per-block partial rows (doubles), a finalize
 *    kernel sums them in a fixed order.
 *
 * Each entry point cites the reference code (paths relative to the reference repository)
 * whose work it replaces.
 */
#ifndef UNETB200_H
#define UNETB200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define UB2_OK 0
#define UB2_ERR_SHAPE (-1)     /* unsupported shape */
#define UB2_ERR_ALIGN (-2)     /* pointer / stride alignment */
#define UB2_ERR_WORKSPACE (-3) /* workspace rows do not match the *_rows query */
#define UB2_ERR_DRIVER (-4)    /* cuTensorMapEncodeTiled unavailable / failed */
#define UB2_ERR_ARCH (-5)      /* not an sm_100 device */

int ub2_version(void);
int ub2_num_sms(void);
/* Tuning / A-B testing: 0 = automatic kernel choice, 1 = never use the halo-resident 3x3 kernel. */
int ub2_set_conv_mode(int mode);
/* Which kernel the dispatcher launched for the calling thread's last ub2_conv_fwd / ub2_conv_wgrad call:
 * forward and data gradient 1 = one CTA per tap, 2 = CTA pair per tap, 3 = one CTA halo-resident,
 * 4 = CTA pair halo-resident; weight gradient 11..14 in the same order.  Diagnostics / tests only. */
int ub2_last_conv_variant(void);

/* ======================= convolutions on tcgen05 tensor cores =========================== */

/* nn.Conv2d(k=3,p=1,bias=False) of DoubleConv (unet/models/layers.py:32,35) and the 1x1
 * projections of AttentionGate (layers.py:152,158) as an NHWC bf16 implicit GEMM (TMA ->
 * smem -> tcgen05.mma -> TMEM).  The input channel axis may span two tensors (in0: C0
 * channels, in1: C1 channels): torch.cat([x2, x1], dim=1) of Up / AttentionUp (layers.py:105,
 * :254) without the copy.  wgt: (Cout, taps, C0+C1) bf16.  Epilogue options: per-channel
 * scale/shift (eval-mode BatchNorm folded, layers.py:33), ReLU (layers.py:34), accumulate into
 * the destination, split of the output channels over two tensors (channels >= split go to
 * out1), and per-CTA rows of per-channel sum / sum-of-squares (stats: (stats_rows,2,Cout)
 * doubles; *stats_rows_used rows are written) for train-mode BatchNorm.  With the
 * flipped/transposed weight pack it is the data-gradient pass autograd runs for the same conv.
 * Channels: C0, C1 and Cout multiples of 8, not necessarily of 16 (the K chunks past a source's end
 * read zeros through the tensor map, never memory); ld_in0 / ld_in1 / ld0 / ld1 and split multiples
 * of 8.  A C0 or C1 that is not a multiple of 8 returns UB2_ERR_ALIGN: each source's columns of the
 * weight pack must start on 16 bytes.  Only output channels < Cout are written: channels between
 * Cout and ld0 keep their contents.
 */
int ub2_conv_fwd(const void* in0, int ld_in0, int C0, const void* in1, int ld_in1, int C1,
                 const void* wgt, void* out0, int ld0, void* out1, int ld1, int split, int N, int H,
                 int W, int Cout, int taps, const float* scale, const float* shift, int relu,
                 int accumulate, double* stats, int stats_rows, int* stats_rows_used,
                 int bn_override, int grid_override, void* stream);

/* Weight-gradient pass of the same nn.Conv2d (autograd of layers.py:32,35,152,158): split-K
 * partial tiles (splits, taps*(C0+C1), Cout) fp32; *splits_used <= max_splits are written.
 * Channels: C0 >= 1 and C1 >= 0 of any count, Cout a multiple of 8, channel strides multiples of 8. */
int ub2_conv_wgrad(const void* in0, int ld_in0, int C0, const void* in1, int ld_in1, int C1,
                   const void* dy, int ld_dy, float* partial, int max_splits, int* splits_used,
                   int N, int H, int W, int Cout, int taps, int splits_override, void* stream);

/* grad (Cout,Cin,k,k fp32, the .grad of the nn.Conv2d weight) = or += (accumulate) the sum over
 * splits, in a fixed order.  `partial` is scratch: with many splits slot 0 is overwritten. */
int ub2_wgrad_reduce(float* partial, int splits, int Cout, int Cin, int taps, float* grad,
                     int accumulate, void* stream);

/* The same fold for up to UB2_REDUCE_MAX_ITEMS layers in one or two launches (one gradient bucket
 * at a time instead of one or two launches per layer).  `items` is a HOST array read during the
 * call; it is passed to the kernels by value, so the launch can be captured into a CUDA graph. */
#define UB2_REDUCE_MAX_ITEMS 32
typedef struct Ub2ReduceItem {
  float* partial; /* (splits, taps*Cin, Cout) fp32, scratch */
  float* grad;    /* (Cout, Cin, k, k) fp32 */
  int splits, Cout, Cin, taps;
} Ub2ReduceItem;
int ub2_wgrad_reduce_multi(const Ub2ReduceItem* items, int n, int accumulate, void* stream);

/* OIHW fp32 parameter -> bf16 packs: fwd (Cout,taps,Cin) and dgrad (Cin,taps flipped,Cout);
 * either may be NULL; out_scale (optional, per Cout) folds a BatchNorm scale into the pack. */
int ub2_pack_conv_weight(const float* w, void* fwd, void* dgrad, int Cout, int Cin, int taps,
                         const float* out_scale, void* stream);
/* The same for many weights in one launch (once per optimizer step): desc (T,6) int64 =
 * {w, fwd, dgrad, Cout, Cin, taps}; blocks (nblocks,4) int32 = {tensor, Cin tile, Cout tile, edge},
 * one per 16x16 channel tile.  edge = 0 only for a whole tile (16 channels of each) of a weight whose
 * Cout and Cin are multiples of 8; any other tile (partial, or other channel counts) needs edge = 1. */
int ub2_pack_conv_weights_multi(const long long* desc, const int* blocks, int nblocks, void* stream);

/* ======================= BatchNorm / ReLU / MaxPool passes ============================== */
/* The bf16 entry points below (BatchNorm, max-pool, attention gate, network ends, ConvTranspose2d pieces) check their
 * arguments before the device is touched.  UB2_ERR_SHAPE: a count <= 0 (N, H, W, C, Ci, Cx, Cin, Cout, K, h, w, hin,
 * win, splits), a channel count that is not a multiple of 8 or above the kernel's limit (named per entry point), a
 * channel stride below its channel count, or a NULL pointer other than the optional ones named per entry point.
 * UB2_ERR_ALIGN: a channel stride that is not a multiple of 8, a pointer read or written with 16-byte vectors (the
 * NHWC bf16 tensors) that is not 16-byte aligned, pidx not 8-byte aligned, partials not 8-byte aligned, or an fp32
 * pointer not 4-byte aligned.  UB2_ERR_WORKSPACE: rows other than the matching *_rows query. */

/* nn.BatchNorm2d in train mode (layers.py:33,36,153,159,165): per-CTA sums -> batch mean and
 * biased variance; running_mean/var momentum update with the unbiased variance and
 * num_batches_tracked += 1 (all optional); outputs scale = gamma*invstd, shift = beta -
 * mean*scale, mean, invstd. */
int ub2_bn_finalize(const double* partials, int rows, int C, double count, const float* gamma,
                    const float* beta, float* running_mean, float* running_var, long long* nbt,
                    float momentum, float eps, float* scale, float* shift, float* mean, float* invstd,
                    void* stream);
/* nn.BatchNorm2d in eval mode: scale/shift from the running statistics; gamma / beta may be NULL (1 / 0). */
int ub2_bn_eval_coeffs(const float* gamma, const float* beta, const float* running_mean,
                       const float* running_var, float eps, int C, float* scale, float* shift,
                       void* stream);
/* a = relu(scale*y + shift) (nn.ReLU, layers.py:34,37) and, optionally, its 2x2 max-pooled copy
 * (nn.MaxPool2d(2) of Down, layers.py:56) with pidx (N,H/2,W/2,C) uint8 = window position of each
 * maximum (first maximum wins, as ATen); a, pooled, pidx may be NULL; scale/shift NULL = identity.
 * C <= 2048; y, ld_y required; ld_a / ld_p are checked only with a / pooled. */
int ub2_bn_act(const void* y, int ld_y, const float* scale, const float* shift, void* a, int ld_a,
               void* pooled, int ld_p, unsigned char* pidx, int N, int H, int W, int C, int relu,
               void* stream);
/* Backward of BatchNorm+ReLU(+MaxPool routing) — what autograd runs for layers.py:33-34,56:
 *   g = (dA + dP routed to the window position pidx saved by ub2_bn_act) * [scale*y + shift > 0]
 *   reduce  : rows of (sum g, sum g*y);  rows = ub2_bn_bwd_rows(...)
 *   finalize: dgamma/dbeta (+= into the fp32 .grad) and coef (3,C): dy = c0*g + c1*y + c2
 *             (frozen != 0: eval-mode statistics, c1 = c2 = 0)
 *   apply   : dy bf16.  dA or dP may be NULL (not both; dP needs pidx; ld_da / ld_dp are then ignored);
 *             y, scale, shift, partials / coef and dY are required.  C <= 2048. */
int ub2_bn_bwd_rows(int N, int H, int W, int C, int pool);
int ub2_bn_bwd_reduce(const void* dA, int ld_da, const void* dP, int ld_dp, const unsigned char* pidx,
                      const void* y, int ld_y, const float* scale, const float* shift, double* partials,
                      int rows, int N, int H, int W, int C, int relu, void* stream);
int ub2_bn_bwd_finalize(const double* partials, int rows, int C, double count, const float* gamma,
                        const float* mean, const float* invstd, int frozen, float* dgamma, float* dbeta,
                        float* coef, void* stream);
int ub2_bn_bwd_apply(const void* dA, int ld_da, const void* dP, int ld_dp, const unsigned char* pidx,
                     const void* y, int ld_y, const float* scale, const float* shift, const float* coef,
                     void* dY, int ld_dy, int N, int H, int W, int C, int relu, void* stream);

/* ======================= bilinear resampling ============================================ */

/* nn.Upsample(scale_factor=2, bilinear, align_corners=True) + F.pad to the skip size
 * (layers.py:78, :98-102, :212, :247-251): (hin,win) -> (hu,wu) placed centred in (Ho,Wo). */
int ub2_upsample_fwd(const void* src, int ld_src, void* out, int ld_out, int N, int hin, int win, int hu,
                     int wu, int Ho, int Wo, int C, void* stream);
/* Its transpose in gather form (deterministic; ATen's backward uses atomics). */
int ub2_upsample_bwd(const void* dout, int ld_dout, void* din, int ld_din, int accumulate, int N,
                     int hin, int win, int hu, int wu, int Ho, int Wo, int C, void* stream);

/* ConvTranspose2d(C, C/2, 2, stride 2) + F.pad (unet/models/layers.py:81, :98-102, :217-221): the transposed
 * convolution itself is ub2_conv_fwd with the (4*Cout, Cin) reshaped weight (row (i,j,co)) and the bias in its
 * epilogue; these are the pixel shuffle out[n, 2y+i+py, 2x+j+px, co] = t[n, y, x, (i*2+j)*C + co] with the
 * padding of F.pad (zeros), its transpose, and the bias gradient: dbias[co] += sum of the gathered dout.
 * `partials`: (rows, C) doubles with rows = ub2_shuffle2x2_rows(...); pass NULL (and dbias NULL) to skip the bias
 * gradient.  t / dt have channel strides >= 4*C, out / dout >= C; C <= 2048 for the backward. */
int ub2_shuffle2x2_fwd(const void* t, int ld_t, void* out, int ld_out, int N, int h, int w, int C, int Ho, int Wo,
                       void* stream);
int ub2_shuffle2x2_rows(int N, int h, int w, int C, int Ho, int Wo);
int ub2_shuffle2x2_bwd(const void* dout, int ld_dout, void* dt, int ld_dt, double* partials, int rows, float* dbias,
                       int N, int h, int w, int C, int Ho, int Wo, void* stream);
/* The (Cin, Cout, 2, 2) fp32 ConvTranspose2d parameter as 1x1-convolution packs: fwd (4*Cout, Cin) bf16 with row
 * (i*2+j)*Cout + co, dg (Cin, 4*Cout) bf16, and the epilogue vectors scale4 = 1, shift4 = bias tiled four times
 * (each 4*Cout floats; bias may be NULL).  Any output pointer may be NULL, but scale4 and shift4 only together. */
int ub2_pack_convt_weight(const float* w, const float* bias, void* fwd, void* dg, float* scale4, float* shift4,
                          int Cin, int Cout, void* stream);
/* grad (Cin, Cout, 2, 2) fp32 = (or +=) the split-K partials (splits, Cin, 4*Cout) of ub2_conv_wgrad(taps = 1) on
 * the shuffled gradient, summed in a fixed order. */
int ub2_convt_wgrad_reduce(const float* partial, int splits, int Cin, int Cout, float* grad, int accumulate,
                           void* stream);
/* F.interpolate(x, size, mode='bilinear', align_corners=True) of the deep-supervision logits
 * (unet/models/unet.py:206-208) and its transpose in gather form (deterministic): fp32 NCHW,
 * planes = N * channels, (hin,win) -> (Ho,Wo), any scale. */
int ub2_resize_planes_fwd(const float* src, float* out, int planes, int hin, int win, int Ho, int Wo, void* stream);
int ub2_resize_planes_bwd(const float* dout, float* din, int planes, int hin, int win, int Ho, int Wo,
                          void* stream);

/* ======================= attention gate (layers.py:171-192) ============================= */
/* q = W_g.g at low resolution and xp = W_x.x come from ub2_conv_fwd (taps = 1).           */

int ub2_gate_rows(int N, int H, int W, int C);
/* rows for ub2_gate_upstats / ub2_gate_psi / ub2_gate_bwd_s (one per block of their strip grid) */
int ub2_gate_strip_rows(int N, int H, int W, int C);
/* Batch statistics of F.interpolate(q, (H,W), bilinear, align_corners=True) for BN_g
 * (layers.py:183,186) without materialising the up-sampled tensor. */
int ub2_gate_upstats(const void* q, int ld_q, int N, int hin, int win, int H, int W, int Ci,
                     double* partials, int rows, void* stream);
/* The strip passes (upstats, psi, fused_eval, bwd_s, bwd_xg) take Ci <= 512 and (hin - 1) < 2 (H - 1) (a ring of at
 * most 8 low-resolution rows; a stronger down-sampling is UB2_ERR_SHAPE);
 * gate_bwd_a takes Cx <= 512, gate_apply any Cx.  Every pointer is required except partials of ub2_gate_psi (no
 * statistics) and a_out of ub2_gate_apply. */
/* psi_raw = w_psi . relu(BN_g(up q) + BN_x(xp)) (layers.py:188, :164) + rows of (sum, sum sq). */
int ub2_gate_psi(const void* q, int ld_q, const void* xp, int ld_xp, const float* scale_g,
                 const float* shift_g, const float* scale_x, const float* shift_x, const float* wpsi,
                 float* psi_raw, double* partials, int rows, int N, int hin, int win, int H, int W,
                 int Ci, void* stream);
/* a = sigmoid(BN_psi(psi_raw)); out = x * a (layers.py:165-166, :192). */
/* Inference only (BatchNorm frozen, nothing saved): psi, sigmoid and out = x * a in ONE pass over q, xp and x
 * (north_star (3)); needs Cx == 2 * Ci (layers.py:147-148's default inter-channel count) and, for Ci > 256, a
 * 4-row ring, 3 (hin - 1) < 2 (H - 1) (the U-Net's 2x up-sampling): its 8-row ring would not fit a block's shared
 * memory.  Else UB2_ERR_SHAPE, and the caller runs ub2_gate_psi + ub2_gate_apply.  ub2_gate_bwd_xg likewise needs
 * the 4-row ring for Ci > 336. */
int ub2_gate_fused_eval(const void* q, int ld_q, const void* xp, int ld_xp, const void* x, int ld_x, const float* scale_g,
                        const float* shift_g, const float* scale_x, const float* shift_x, const float* wpsi,
                        const float* scale_psi, const float* shift_psi, void* out, int ld_out, int N, int hin, int win,
                        int H, int W, int Ci, int Cx, void* stream);
int ub2_gate_apply(const float* psi_raw, const float* scale_psi, const float* shift_psi, const void* x,
                   int ld_x, void* out, int ld_out, float* a_out, int N, int H, int W, int Cx,
                   void* stream);
/* Backward passes (autograd of layers.py:183-192). */
int ub2_gate_bwd_a(const void* dout, int ld_do, const void* x, int ld_x, const float* a,
                   const float* psi_raw, void* dx, int ld_dx, float* dpsin, double* partials, int rows,
                   int N, int H, int W, int Cx, void* stream);
int ub2_gate_bwd_s(const float* dpsin, const float* psi_raw, const float* coef_psi, const void* q,
                   int ld_q, const void* xp, int ld_xp, const float* scale_g, const float* shift_g,
                   const float* scale_x, const float* shift_x, const float* wpsi, void* ds, int ld_ds,
                   double* partials, int rows, int N, int hin, int win, int H, int W, int Ci,
                   void* stream);
int ub2_gate_bwd_finalize(const double* partials, int rows, int Ci, double count, const float* gamma_x,
                          const float* mean_x, const float* invstd_x, const float* gamma_g,
                          const float* mean_g, const float* invstd_g, int frozen, float* dgamma_x,
                          float* dbeta_x, float* dgamma_g, float* dbeta_g, float* dwpsi, float* coef,
                          void* stream);
int ub2_gate_bwd_xg(const void* ds, int ld_ds, const void* xp, int ld_xp, const void* q, int ld_q,
                    const float* coef, void* dxp, int ld_dxp, void* dgup, int ld_dg, int N, int hin,
                    int win, int H, int W, int Ci, void* stream);

/* ======================= network ends =================================================== */

/* inc.double_conv.0 (layers.py:32 with in_channels = n_channels <= 4): direct fp32 conv of the
 * fp32 NCHW input, NHWC bf16 output + BatchNorm statistic rows (partials may be NULL); and its weight gradient
 * (grad +=).  1 <= Cin <= 4, Cout <= 2048; partials and grad 8- / 4-byte aligned.  Outside the register-window
 * variant (Cin == 1, W % 4 == 0, x 16-byte aligned) the forward keeps the Cin * 9 * Cout weights and 16 floats per
 * thread of its (at most 256-thread) block in 48 KB of shared memory; a larger product is UB2_ERR_SHAPE. */
int ub2_conv_in_rows(int N, int H, int W, int Cout);
int ub2_conv_in_fwd(const float* x, const float* w, void* y, int ld_y, double* partials, int rows, int N,
                    int Cin, int H, int W, int Cout, void* stream);
int ub2_conv_in_wgrad(const float* x, const void* dy, int ld_dy, double* partials, int rows, float* grad,
                      int N, int Cin, int H, int W, int Cout, void* stream);
/* Its data gradient (autograd of layers.py:32 when the network input requires grad): dy NHWC bf16 with
 * channel stride ld_dy (multiple of 8, >= Cout), w the fp32 OIHW parameter, dx fp32 NCHW (N,Cin,H,W), each
 * element written once in a fixed summation order (no atomics).  Same Cin / Cout limits as ub2_conv_in_fwd;
 * for Cin > 1, W % 4 != 0 or pointers not 16-byte aligned also Cin * 9 * Cout <= 12288. */
int ub2_conv_in_dgrad(const void* dy, int ld_dy, const float* w, float* dx, int N, int Cin, int H, int W, int Cout,
                      void* stream);
/* OutConv (layers.py:120-123): 1x1 conv with bias to fp32 NCHW logits, and its backward.  1 <= K <= 8; the backward
 * takes C <= 512.  bias, da, dw and db may be NULL (dw and db accumulate: +=); a and w are 16-byte aligned. */
int ub2_outc_rows(int N, int H, int W, int C);
int ub2_outc_fwd(const void* a, int ld_a, const float* w, const float* bias, float* logits, int N, int H,
                 int W, int C, int K, void* stream);
int ub2_outc_bwd(const float* dlogits, const void* a, int ld_a, const float* w, void* da, int ld_da,
                 double* partials, int rows, float* dw, float* db, int N, int H, int W, int C, int K,
                 void* stream);

/* ======================= loss and metrics =============================================== */

/* Per-(image, class) pixel sums of DiceLoss / BalancedCELoss / DiceBCELoss
 * (unet/utils/loss.py:63-73, :129-148): stats (N,4,C) fp32 = {count, CE sum, intersection,
 * probability sum}; blocks = ub2_seg_stats_blocks(N, HW). */
int ub2_seg_stats_blocks(int N, long long HW);
int ub2_seg_stats(const float* logits, const long long* targets, int N, int C, long long HW,
                  double* partials, int blocks, float* stats, void* stream);
/* dL/dlogits from coef (N,3,C) = {dL/dCE, dL/dI, dL/dP}, times *gscale (optional device scalar:
 * the upstream gradient of the loss). */
int ub2_seg_stats_bwd(const float* logits, const long long* targets, const float* coef, const float* gscale,
                      int N, int C, long long HW, float* dlogits, void* stream);
/* DiceBCELoss.forward (unet/utils/loss.py:184-191, with :70-85 and :134-148) from the statistics:
 * loss (1) fp32 and the gradient table coef (N,3,C) for ub2_seg_stats_bwd, one launch. */
int ub2_dice_bce_head(const float* stats, int N, int C, float ce_weight, float dice_weight, float class_weight,
                      float ce_smooth, float dice_smooth, int ignore_background, float* loss, float* coef,
                      void* stream);
/* SegmentationMetrics.update (unet/utils/metrics.py:55-84): cm ((C+1),(C+1)) int64 +=
 * histogram of (target, prediction); row/col C = ignored / out of range.  mode 0: argmax of
 * fp32 logits (N,C,H,W); 1: int64 class indices; 2: softmax[:,1] > threshold
 * (scripts/predict.py:155-159), optional uint8 0/255 mask_out. */
int ub2_confusion(const void* pred, const long long* target, int mode, int N, int C, long long HW,
                  long long ignore_index, int has_ignore, float threshold, long long* cm,
                  unsigned char* mask_out, void* stream);

/* ======================= fp32 / TF32 evaluation mode ==================================== */

/* BASELINE configs[0] (AttentionUNet fp32 forward) and north_star's "fp32/TF32 mode, logits within
 * 1e-3": the eval-mode forward of every block of unet/models/layers.py with fp32 NHWC activations
 * (element strides), BatchNorm folded with the running statistics, the 3x3 / 1x1 convolutions on
 * the tensor cores as kind::tf32.  Forward only.
 * Every count (N, H, W, C, Ci, Cx, K, hin, win, hu, wu) must be > 0 and channel counts multiples of 4, with
 * Ho >= hu and Wo >= wu, H and W >= 2 for the max-pool and K <= 8 for the head; every pointer is required except the
 * head's bias; float4-accessed tensors (activations, q, xp) need 16-byte-aligned pointers.  Anything else returns
 * UB2_ERR_SHAPE (or UB2_ERR_ALIGN) before the device is touched. */
/* nn.Conv2d (+ folded BN + ReLU) of layers.py:32-37,152,158: in0/in1 fp32 NHWC (virtual concat),
 * wgt = ub2_f32_pack_weight output (Cout,taps,C0+C1) fp32, out fp32 NHWC; out = relu?(scale*acc+shift).
 * exact_out = 0: the result is rounded to TF32 (it feeds the next single-pass convolution: inference);
 * exact_out = 1: the fp32 accumulator is stored as is (the 3xTF32 launches of the training mode).
 * Channels as for ub2_conv_fwd, with C0 and C1 multiples of 4 (16 bytes of fp32): Cout and the channel
 * strides multiples of 8. */
int ub2_conv_fwd_tf32(const float* in0, int ld_in0, int C0, const float* in1, int ld_in1, int C1,
                      const float* wgt, float* out, int ld_out, int N, int H, int W, int Cout, int taps,
                      const float* scale, const float* shift, int relu, int exact_out, void* stream);
int ub2_f32_pack_weight(const float* w, float* out, int Cout, int Cin, int taps, void* stream);
/* first conv + folded BN + ReLU: x fp32 NCHW -> out fp32 NHWC (layers.py:32-34, Cin = n_channels) */
int ub2_f32_conv_in(const float* x, const float* w, const float* scale, const float* shift, float* out, int N,
                    int Cin, int H, int W, int Cout, void* stream);
int ub2_f32_maxpool(const float* src, float* out, int N, int H, int W, int C, void* stream);          /* layers.py:56 */
int ub2_f32_upsample(const float* src, float* out, int N, int hin, int win, int hu, int wu, int Ho, int Wo, int C,
                     void* stream);                                                              /* layers.py:78,98-102 */
/* AttentionGate.forward after the two 1x1 projections q = W_g g (low resolution), xp = W_x x
 * (layers.py:183-192): out = x * sigmoid(BN_psi(w_psi . relu(BN_g(up q) + BN_x(xp)))) */
int ub2_f32_gate(const float* q, const float* xp, const float* x, const float* scale_g, const float* shift_g,
                 const float* scale_x, const float* shift_x, const float* w_psi, const float* scale_psi,
                 const float* shift_psi, float* out, int N, int hin, int win, int H, int W, int Ci, int Cx,
                 void* stream);
int ub2_f32_outc(const float* a, const float* w, const float* bias, float* logits, int N, int H, int W, int C,
                 int K, void* stream);                                                           /* layers.py:120 */

/* ======================= optimizer tail (SURVEY 8f-1) ================================== */

/* torch.nn.utils.clip_grad_norm_(model.parameters(), max_norm) (scripts/train.py:141) fused with
 * torch.optim.AdamW.step() (optimizer built at scripts/train.py:346-350), multi-tensor.
 * Device tables: ptrs (4,T) int64 = {param, grad, exp_avg, exp_avg_sq} fp32 pointers; numel (T)
 * int64; group (T) int32 row of `hyper`; chunks (nchunks,2) int32 = {tensor, first element}, each
 * covering ub2_adamw_chunk_elems() elements; hyper (G,8) fp32 = {lr, beta1, beta2, eps,
 * weight_decay, max_norm (row 0 only; <= 0: no clipping), -, -}; step (1) fp32 device counter.
 * ub2_grad_sumsq writes one fp64 partial per chunk and increments *step; ub2_adamw_step folds
 * them in a fixed order (deterministic), stores the total norm, and updates in place; with
 * write_grads the clipped gradients are written back like clip_grad_norm_ does. */
int ub2_adamw_chunk_elems(void);
int ub2_grad_sumsq(const long long* ptrs, const long long* numel, const int* chunks, int nchunks, int T,
                   double* partial, float* step, void* stream);
int ub2_adamw_step(const long long* ptrs, const long long* numel, const int* group, const int* chunks,
                   int nchunks, int T, const double* partial, const float* hyper, const float* step,
                   float* total_norm, int write_grads, void* stream);
/* ModelEMA.update (unet/utils/general.py:155-184) for all parameters and buffers in one launch:
 * desc (T,4) int64 = {dst, src, numel, kind (0: dst = decay*dst + (1-decay)*src fp32; 1: copy fp32;
 * 2: copy int64)}; chunks (nchunks,2) int32 as for ub2_adamw_step; *decay fp32 in device memory. */
int ub2_ema_update(const long long* desc, const int* chunks, int nchunks, const float* decay, void* stream);

/* ======================= either side of the forward pass (SURVEY 8f-3, 8f-4) ============ */

/* LungTumorDataset.__getitem__ + the albumentations-free transform (unet/data/dataset.py:146-171,
 * unet/data/augmentations.py:117-170) and preprocess_image (scripts/predict.py:100-136) for a
 * batch of already-sized slices: images / labels uint8 (N,H,W) in device memory ->
 * x fp32 (N,1,H,W) = ((px/255) - mean)/std, targets int64 (N,H,W) = label > 127.
 * flags uint8 (N) or NULL: bit 0 horizontal flip (augmentations.py:160-162), bit 1 vertical flip.
 * Bit-exact with numpy's float32 arithmetic (the transform's second uint8 round trip,
 * augmentations.py:148, is the identity on all 256 levels).  labels and targets may both be NULL
 * (inference). */
int ub2_prepare_batch(const unsigned char* images, const unsigned char* labels, const unsigned char* flags,
                      int N, int H, int W, float mean, float std, float* x, long long* targets,
                      void* stream);
/* postprocess_mask + tumor_ratio (scripts/predict.py:138-166, 232-240) for a batch: logits fp32
 * (N,2,H,W) -> mask uint8 (N,H,W) = 255 * (softmax(logits)[1] > threshold), positives int32 (N) =
 * number of mask pixels set (zeroed by the call).  No resize: the caller's slices are model-sized. */
int ub2_predict_mask(const float* logits, int N, int C, long long HW, float threshold, unsigned char* mask,
                     int* positives, void* stream);


/* ======================= fp32 / TF32 training mode ======================================= */
/* Activations and gradients are fp32 NHWC (channel stride `ld` where given, else dense), C % 4 == 0.  Forward and
 * data-gradient convolutions: ONE ub2_conv_fwd_tf32 launch over the 3xTF32 K axis [a_hi | a_lo | a_hi] x [w_hi | w_hi |
 * w_lo] (ub2_f32_split_tf32, ub2_f32_pack_weight3); weight gradient: ub2_conv_wgrad on the (hi, lo) bf16 halves of
 * ub2_f32_split_bf16 (kind::tf32 has no MN-major operand mode).  Reductions write one fp64 row per block
 * (`rows` = the matching *_rows query) that the bf16 path's finalize entry points fold (ub2_bn_finalize,
 * ub2_bn_bwd_finalize, ub2_gate_bwd_finalize).  See csrc/fp32_train.cu for the per-kernel reference lines.
 * Arguments are checked before the device is touched.  UB2_ERR_SHAPE: a count <= 0 (N, H, W, C, Ci, Cx, K, n, pixels,
 * hin, win, hu, wu), a channel count not a multiple of 4, Ho < hu or Wo < wu, a channel stride ld* below its channel
 * count, C > 1024 for the per-channel reductions, Ci > 512 for ub2_f32_gate_bwd_s, K > 8 or 8*(K*C + K) floats over
 * 48 KB for ub2_f32_outc_bwd, or a NULL pointer other than these optional ones:
 *   - dA or dP of the act_bwd passes (not both; dP needs idx; ld_da is ignored without dA), and scale / shift of
 *     ub2_f32_act_bwd_apply when relu == 0;
 *   - x1 of ub2_f32_split_tf32 when C1 == 0 (ld1 is then ignored);
 *   - a_out of ub2_f32_gate_apply; da, dw and db of ub2_f32_outc_bwd (dw and db accumulate: +=).
 * UB2_ERR_ALIGN: a channel stride not a multiple of 4, or a float4-accessed pointer not 16-byte aligned (idx: 4,
 * partials: 8).  UB2_ERR_WORKSPACE: rows other than the matching *_rows query.  ub2_f32_conv_in_wgrad's grad
 * accumulates (+=). */
int ub2_f32_channel_rows(long long pixels, int C);
int ub2_f32_channel_stats(const float* x, int ld, long long pixels, int C, double* partials, int rows, void* stream);
int ub2_f32_scalar_rows(long long n);
int ub2_f32_scalar_stats(const float* x, long long n, double* partials, int rows, void* stream);
int ub2_f32_affine_act(const float* y, const float* scale, const float* shift, float* out, long long pixels, int C, int relu, void* stream);
int ub2_f32_maxpool_idx(const float* a, float* p, unsigned char* idx, int N, int H, int W, int C, void* stream);
int ub2_f32_act_bwd_reduce(const float* dA, int ld_da, const float* dP, const unsigned char* idx, const float* y, const float* scale, const float* shift, double* partials, int rows, int N, int H, int W, int C, int relu, void* stream);
int ub2_f32_act_bwd_apply(const float* dA, int ld_da, const float* dP, const unsigned char* idx, const float* y, const float* scale, const float* shift, const float* coef, float* dy, int N, int H, int W, int C, int relu, void* stream);
int ub2_f32_upsample_bwd(const float* dout, int ld_dout, float* din, int N, int hin, int win, int hu, int wu, int Ho, int Wo, int C, void* stream);
int ub2_f32_gate_psi(const float* u, const float* xp, const float* sg, const float* hg, const float* sx, const float* hx, const float* wpsi, float* psi_raw, long long pixels, int Ci, void* stream);
int ub2_f32_gate_apply(const float* psi_raw, const float* spsi, const float* hpsi, const float* x, float* out, float* a_out, long long pixels, int Cx, void* stream);
int ub2_f32_gate_rows(long long pixels);
int ub2_f32_gate_bwd_a(const float* dout, int ld_do, const float* x, const float* a, const float* psi_raw, float* dx, float* dpsin, double* partials, int rows, long long pixels, int Cx, void* stream);
int ub2_f32_gate_bwd_s(const float* dpsin, const float* psi_raw, const float* coef_psi, const float* u, const float* xp, const float* sg, const float* hg, const float* sx, const float* hx, const float* wpsi, float* ds, double* partials, int rows, long long pixels, int Ci, void* stream);
int ub2_f32_gate_bwd_xg(const float* ds, const float* xp, const float* u, const float* coef, float* dxp, float* du, long long pixels, int Ci, void* stream);
int ub2_f32_outc_rows(int N, int H, int W);
int ub2_f32_outc_bwd(const float* dlogits, const float* a, const float* w, float* da, double* partials, int rows, float* dw, float* db, int N, int H, int W, int C, int K, void* stream);
int ub2_f32_conv_in_raw(const float* x, const float* w, float* out, int N, int Cin, int H, int W, int Cout, void* stream);
int ub2_f32_conv_in_wgrad(const float* x, const float* dy, double* partials, int rows, float* grad, int N, int Cin, int H, int W, int Cout, void* stream);
/* ub2_conv_in_dgrad with fp32 dy (ld_dy multiple of 4, >= Cout): Cout % 4 == 0, any Cin >= 1, with the same
 * shared-memory limit. */
int ub2_f32_conv_in_dgrad(const float* dy, int ld_dy, const float* w, float* dx, int N, int Cin, int H, int W, int Cout, void* stream);
int ub2_f32_split_bf16(const float* x, void* hi, void* lo, long long n, void* stream);
int ub2_f32_split_tf32(const float* x0, int ld0, int C0, const float* x1, int ld1, int C1, float* out, long long pixels, void* stream);
int ub2_f32_pack_weight3(const float* w, float* out, int Cout, int Cin, int taps, int dgrad, void* stream);
int ub2_f32_upsample_fwd(const float* src, float* out, int N, int hin, int win, int hu, int wu, int Ho, int Wo, int C, void* stream);
/* ConvTranspose2d(C, C/2, 2, stride 2) + F.pad in fp32 (layers.py:81, :98-102, :217-221): the ub2_shuffle2x2_* pixel
 * shuffle, its transpose and the bias gradient on fp32 tensors.  t / dt: (N,h,w,4*C) with channel stride ld_t / ld_dt
 * >= 4*C; out / dout: (N,Ho,Wo,C) with stride ld_out / ld_dout >= C (dout may be a channel slice of a wider
 * tensor).  C % 4 == 0 and C <= 1024, Ho >= 2h, Wo >= 2w.  `partials`: (rows, C) doubles with rows =
 * ub2_f32_shuffle2x2_rows(...), folded into dbias (+=); partials == NULL skips the bias gradient and dbias is then
 * ignored.  ub2_f32_pack_convt_weight writes the exact fp32 (4*Cout, Cin) 1x1 weight (row (i*2+j)*Cout + co) that
 * ub2_f32_pack_weight / ub2_f32_pack_weight3 (taps = 1) take as OIHW (4*Cout, Cin, 1, 1), and the epilogue vectors
 * scale4 = 1, shift4 = bias tiled four times (zeros when bias is NULL). */
int ub2_f32_shuffle2x2_fwd(const float* t, int ld_t, float* out, int ld_out, int N, int h, int w, int C, int Ho, int Wo, void* stream);
int ub2_f32_shuffle2x2_rows(int N, int h, int w, int C, int Ho, int Wo);
int ub2_f32_shuffle2x2_bwd(const float* dout, int ld_dout, float* dt, int ld_dt, double* partials, int rows, float* dbias, int N, int h, int w, int C, int Ho, int Wo, void* stream);
int ub2_f32_pack_convt_weight(const float* w, const float* bias, float* fwd, float* scale4, float* shift4, int Cin, int Cout, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* UNETB200_H */
