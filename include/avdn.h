/*
 * avdn.h — C ABI of libavdn.so, the sm_100a device library behind the AVDN
 * (Aerial Vision-and-Dialog Navigation) HAA-Transformer hot path.
 *
 * Conventions (all entry points):
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless
 *     the parameter name ends in `_host`;
 *   - the caller owns every buffer (inputs, outputs, workspace); nothing is
 *     allocated, retained or freed by the library;
 *   - work is enqueued on `stream`; the library never synchronises the device;
 *   - return 0 on success, a negative avdn_status on failure;
 *     avdn_last_error_string() gives the reason (thread-local);
 *   - there is no CPU fallback: on a machine without an sm_100 device every
 *     compute entry point returns AVDN_ERR_NO_DEVICE / AVDN_ERR_LAUNCH.
 *
 * Each declaration cites the reference code (file:line under /root/reference)
 * that it replaces.
 */
#ifndef AVDN_H_
#define AVDN_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CUstream_st* avdn_stream_t; /* == cudaStream_t */

typedef enum avdn_status {
  AVDN_OK = 0,
  AVDN_ERR_BAD_ARG = -1,    /* null pointer, bad shape, bad alignment */
  AVDN_ERR_UNSUPPORTED = -2,/* shape / mode outside what the kernels implement */
  AVDN_ERR_LAUNCH = -3,     /* cudaGetLastError() after a launch */
  AVDN_ERR_NO_DEVICE = -4,  /* no CUDA device / not sm_100 */
  AVDN_ERR_DRIVER = -5      /* driver entry point (tensor-map encode) failed */
} avdn_status;

const char* avdn_last_error_string(void);
/* ABI version; bumped whenever a signature changes. */
int avdn_abi_version(void);
/* 1 if device 0 is compute capability 10.x, 0 otherwise (no exception). */
int avdn_device_supported(void);

#define AVDN_VIEW 224 /* src/env.py:273-274 */

/* ------------------------------------------------------------------------
 * Stage 1 — view renderer (src/env.py:254-332)
 * ---------------------------------------------------------------------- */

/* Map preparation: packs a BGR u8 HWC satellite tile and (optionally) its
 * human-attention map into the renderer's HBM layout: one 8-byte record per
 * pixel of the zero-bordered tile, record(X,Y) = pix(X,Y) | pix(X,Y+1) << 32
 * with pix = B | G<<8 | R<<16 | ATT<<24; X in [0,W+1], Y in [0,H], row pitch
 * W+2 records.  A bilinear 2x2 footprint is then two adjacent records (16
 * contiguous bytes).  The zero border implements BORDER_CONSTANT(0) of
 * cv2.warpPerspective (src/env.py:290,292) without per-tap predicates.
 *   map_bgr  [H,W,3] u8      (self.map_batch[name],           src/env.py:217-221)
 *   att      [H,W,att_ch] u8 or NULL; channel 0 is taken
 *                            (self.attention_map_batch[name], src/env.py:224-231)
 *   tile8    [(H+1)*(W+2)] 8-byte records (out), 8-byte aligned                 */
int avdn_pack_tile(const uint8_t* map_bgr, const uint8_t* att, int att_ch,
                   int H, int W, void* tile8, avdn_stream_t stream);

/* Map preparation (src/env.py:217-231, SURVEY.md §8f N2), bit-exact with OpenCV:
 *  - cv2.resize(im, (new_w, H), INTER_AREA), new_w = int(W * lng_ratio / lat_ratio) <= W: the decimation table
 *    (ofs [new_w+1], sidx / alpha [ofs[new_w]]) is OpenCV's computeResizeAreaTab, built by the caller in float64;
 *    the kernel accumulates src * alpha in float in table order and rounds half to even, as ResizeArea_ does.
 *  - the human-attention raster: zeros + cv2.circle(center, radius, 255, thickness=-1) per spot; spots [n,3] i32 =
 *    (cx, cy, radius) in pixels, hw_scratch [n, rmax+1] i32, att [H,W,ch] u8 fully overwritten.                  */
int avdn_resize_area_width(const uint8_t* src, int H, int W, int new_w, const int32_t* ofs, const int32_t* sidx,
                           const float* alpha, uint8_t* dst, avdn_stream_t stream);
int avdn_raster_attention(const int32_t* spots, int n_spots, int rmax, int32_t* hw_scratch, int H, int W, int ch,
                          uint8_t* att, avdn_stream_t stream);

/* gps_to_img_coords (src/env.py:189-196), batched and bit-exact:
 *   x = rint((lng - bl_lng) / lat_ratio), y = rint((tr_lat - lat) / lat_ratio)
 * in float64 with round-half-even.
 *   corners_gps [P,4,2] f64 (lat,lng);  geo [P,5] f64 = (bl_lat, bl_lng,
 *   tr_lat, tr_lng, lat_ratio) per pose;  corners_px [P,4,2] i32 (x,y) (out)   */
int avdn_gps_to_pixels(const double* corners_gps, const double* geo, int P,
                       int32_t* corners_px, avdn_stream_t stream);

/* cv2.getPerspectiveTransform (src/env.py:287) followed by the matrix
 * inversion cv2.warpPerspective performs internally (src/env.py:290):
 *   corners_px [P,4,2] i32 (FL,FR,BR,BL; x,y)  ->  minv [P,9] f64 row-major.
 * float64, same elimination / rounding order as OpenCV (no FMA contraction);
 * a singular system yields the all-zero matrix, as OpenCV does.                */
int avdn_homography_from_corners(const int32_t* corners_px, int P, double* minv,
                                 avdn_stream_t stream);

/* One packed tile as the renderer sees it. */
typedef struct avdn_tile_desc {
  const void* tile8;     /* avdn_pack_tile output */
  int32_t H, W;          /* un-padded size */
} avdn_tile_desc;

/* cv2.warpPerspective(map, M, (224,224)) and the same warp of the attention
 * map (src/env.py:290-293), fixed-point bilinear, bit-exact, for P poses.
 *   tiles     [n_tiles] avdn_tile_desc (device array)
 *   tile_idx  [P] i32 or NULL (all poses use tiles[0])
 *   minv      [P,9] f64 from avdn_homography_from_corners
 * Outputs, each may be NULL:
 *   views     [P,224,224,3] u8 BGR HWC     = obs['current_view']  (env.py:308)
 *   att       [P,224,224]   u8             = 255 * obs['gt_saliency'] (env.py:293)
 *   norm_nchw [P,3,224,224] f32 RGB, (x-mean)/std (src/xview_et/agent.py:586-592)
 *   norm_nhwc [P,224,224,4] bf16 RGB0, same normalisation rounded to bf16
 *             (channel 3 is zero; this is the trunk's input layout)
 *   norm_lut  [3,256] f32, lut[c][v] = (float(v) - mean[c]) / std[c] for RGB
 *             channel c, computed on the host in float32 exactly as the
 *             reference does; required when norm_nchw or norm_nhwc is given.  */
int avdn_render_views(const avdn_tile_desc* tiles, int n_tiles,
                      const int32_t* tile_idx, const double* minv, int P,
                      uint8_t* views, uint8_t* att, float* norm_nchw,
                      void* norm_nhwc, const float* norm_lut,
                      avdn_stream_t stream);

/* ------------------------------------------------------------------------
 * Tensor-core primitive (tcgen05 / TMEM / TMA): every dense contraction of
 * the path runs through one planned kernel.  It replaces the cuDNN / cuBLAS
 * library calls behind
 *   nn.Conv2d fwd/dgrad/wgrad        src/models/dark_net.py:22-28
 *   nn.Linear / MHA projections      src/models/enc_vl.py:16-22,68
 *   QK^T, PV and their backward      (inside nn.TransformerEncoderLayer)
 *   ET heads / fc2                   src/models/ET_haa.py:98-119,144-167
 * A plan is a caller-owned HOST blob (avdn_gemm_plan_bytes() bytes) holding the
 * encoded TMA descriptors and launch geometry for fixed device pointers; it can
 * be re-run any number of times (and captured in a CUDA graph).  The kernel is
 * persistent (one CTA or CTA pair per SM walks the tile space); outputs leave
 * through TMA stores (reduce-adds for the accumulating modes: `out += ` on a
 * bf16 tensor adds the bf16-rounded tile in bf16).
 * ---------------------------------------------------------------------- */
enum { AVDN_GEMM_PLAIN = 0, AVDN_GEMM_CONV = 1, AVDN_GEMM_WGRAD = 2 };
enum { AVDN_DT_BF16 = 0, AVDN_DT_F32 = 1 };

/* One k-step source of a convolution: which A (CONV) / B (WGRAD) view, the
 * offset added to the box's W and H coordinates, and the operand-B k offset
 * (CONV) or the output column offset (WGRAD) of this filter tap. */
typedef struct avdn_tap { int32_t map, d1, d2, bk; } avdn_tap;

/* A bf16 operand as a rank-4 strided tensor; dim[0] is contiguous.  Strides in
 * elements.  box = TMA box (box[0] = 64, or 32 with bk = 32). */
typedef struct avdn_operand {
  const void* ptr;
  int64_t dim[4];
  int64_t stride[4];
  int32_t box[4];
} avdn_operand;

typedef struct avdn_gemm_core {
  int32_t mode;               /* AVDN_GEMM_* */
  int32_t M, N;               /* logical output extent per batch (PLAIN/WGRAD); N only (CONV) */
  int32_t num_kb;             /* k-steps of 64: ceil(K/64) | taps*cblocks | pixel tiles */
  int32_t split_k;            /* >1 only with accumulate == 2 */
  int32_t batch0, batch1;     /* PLAIN: grid.z = batch0*batch1*split_k -> coords 2,3 */
  int32_t b_batched;          /* PLAIN: 1 if operand B has the batch dims too */
  int32_t cblocks, n_taps;    /* CONV: channel blocks per tap */
  avdn_tap taps[9];
  int32_t tiles_w, tiles_h, tiles_n;   /* spatial tiling of the box over (W,H,N) */
  int32_t box_w, box_h, box_n;
  int32_t valid_w, valid_h, valid_n;   /* CONV: extent of valid output coords */
  int32_t out_H, out_W, out_sh, out_sw, out_oh, out_ow; /* CONV: out pixel (n, h*sh+oh, w*sw+ow) */
  int32_t out_dtype;          /* AVDN_DT_* */
  int32_t accumulate;         /* 0 store, 1 out += (bf16 / fp32 reduce-add), 2 fp32 reduce-add with split-K */
  int32_t relu;
  float alpha;
  uint32_t tx_bytes;          /* filled by avdn_gemm_plan */
  int32_t pad_;
  int64_t ldc, out_bs0, out_bs1;       /* output row pitch / batch strides, elements */
  void* out;
  const float* bias;          /* [N] fp32 or NULL */
  const void* relu_mask;      /* bf16, addressed like `out`: result is zeroed where mask <= 0
                                 (backward of the ReLU whose forward output is `relu_mask`) */
  double* stats;              /* NULL, or [2][N] f64: fused BatchNorm statistics -- per output column the
                                 sum and the sum of squares of the (bf16-rounded) outputs; zeroed by
                                 avdn_gemm_run before the launch (bf16 store epilogue only) */
  /* Fused eval-mode BatchNorm + LeakyReLU (+ shortcut) epilogue (dark_net.py:22-33,224-226 in eval mode,
   * where the BN affine is known before the convolution runs): out = leaky(acc*col_scale + col_shift)
   * (+ residual).  col_scale/col_shift [N] fp32 or both NULL; residual: bf16 tensor addressed like `out`
   * (CONV mode, unit output stride) or NULL.  bf16 TMA-store epilogue only; excludes stats/accumulate.   */
  const float* col_scale;
  const float* col_shift;
  const void* residual;
  float leaky_slope;
  int32_t pad2_;
  /* Fused train-mode BatchNorm BACKWARD statistics (dark_net.py:31 under autograd): this launch is the data
   * gradient `out` = dA of the activation a = leaky(z*scale + shift) of the PRODUCING block, and once a tile of dA
   * is final the epilogue adds, per output column c,
   *     bnb_sums[0][c] += sum g          bnb_sums[1][c] += sum g * (z - mean[c]),   g = dA * leaky'(z*scale+shift)
   * -- the two reductions nn.BatchNorm2d's backward needs -- so no separate pass over (z, dA) runs.
   * bnb_z: bf16 tensor addressed like `out` (the block's stored pre-activation), bnb_scale/shift/mean [N] fp32,
   * bnb_sums [2][N] f64, NOT zeroed by avdn_gemm_run (the parity launches of a stride-2 layer add into one
   * buffer).  With accumulate == 1 the epilogue reads the old dA tile, adds in fp32 and stores (no bf16 TMA
   * reduce-add), so the statistics see the final value.  CONV mode, K-major operands, bf16 TMA-store epilogue;
   * excludes stats / col_scale.  All five NULL = off.                                                     */
  const void* bnb_z;
  const float* bnb_scale;
  const float* bnb_shift;
  const float* bnb_mean;
  double* bnb_sums;
  /* Output classes of a CONV launch (the data gradient of a stride-2 convolution): n_classes > 1 makes every spatial
   * tile n_classes tiles, class k using taps [cls_tap0[k], cls_tap0[k+1]) and writing the output pixels
   * (n, h*out_sh + cls_oh[k], w*out_sw + cls_ow[k]) -- the four output parities of dX = conv_transpose(dZ, w) in ONE
   * launch, the class being the fastest-varying tile index so that the CTAs working side by side read the same dZ
   * tile (once from HBM) and together complete whole output lines.  0 / 1: a single class (out_oh / out_ow above). */
  int32_t n_classes;
  int32_t cls_tap0[5];
  int32_t cls_oh[4], cls_ow[4];
  int32_t pad4_[2];
} avdn_gemm_core;

typedef struct avdn_gemm_desc {
  avdn_gemm_core core;
  int32_t bn;                 /* N tile: 32 (K-major, bf16 out), 64, 128 or 256 */
  int32_t a_mn, b_mn;         /* 0 = K-major operand, 1 = MN-major operand */
  int32_t n_a, n_b;           /* number of A / B views (parity views of stride-2 convs) */
  int32_t grid_m, grid_n, grid_z;  /* tile space: 128-row tiles x bn-column tiles x (batch | taps*split_k) */
  int32_t ctas;               /* 1, or 2 = CTA pairs (tcgen05 cta_group::2): a pair computes 256 x bn and
                                 each CTA loads half of B; needs bn >= 128 */
  int32_t bk;                 /* k-block in elements: 64 (128-byte swizzle) or 32 (64-byte swizzle; K-major
                                 operands, bn = 64: the 32-channel activations of trunk blocks 0 and 2) */
  avdn_operand a[4];
  avdn_operand b[4];
} avdn_gemm_desc;

size_t avdn_gemm_plan_bytes(void);
int avdn_gemm_plan(const avdn_gemm_desc* desc, void* plan_host, size_t plan_bytes);
int avdn_gemm_run(const void* plan_host, avdn_stream_t stream);

/* ------------------------------------------------------------------------
 * Stage 2 — Darknet trunk (src/models/dark_net.py).  Activations are NHWC
 * bf16, channels padded to a multiple of 64, addressed as R rows x C.
 * ---------------------------------------------------------------------- */

/* First convolution 3->32, 3x3, pad 1 (module_list.0.conv_0; K = 27 is too thin
 * for a tcgen05 tile: warp-level mma.sync).  x [N,H,W,4] bf16 (R,G,B,0:
 * avdn_render_views' norm_nhwc), w [32,3,3,3] fp32 (nn.Conv2d layout, rounded to
 * bf16 for the tensor cores), z [N,H,W,32] bf16.  stats: NULL or
 * [2,32] f64 receiving the BatchNorm batch statistics of z (sum, sum of squares;
 * zeroed by the call), to be finished by avdn_bn_finalize.  W % 16 == H % 4 == 0. */
int avdn_conv0_fwd(const void* x_nhwc4, const float* w, void* z, int N, int H, int W, double* stats,
                   avdn_stream_t stream);
/* Eval mode: the same convolution with BatchNorm (running statistics) + LeakyReLU folded into the store:
 * a [N,H,W,32] bf16 = leaky_slope(conv(x) * scale + shift); scale/shift [32] fp32 from avdn_bn_eval_coeffs. */
int avdn_conv0_fwd_eval(const void* x_nhwc4, const float* w, const float* scale, const float* shift, float slope,
                        void* a, int N, int H, int W, avdn_stream_t stream);
/* dw [32,3,3,3] fp32 += sum_pixels dz * x (weight gradient of the same layer). */
int avdn_conv0_wgrad(const void* dz, const void* x_nhwc4, float* dw, int N, int H, int W, avdn_stream_t stream);
/* Train-mode RECOMPUTE path of the same block (nn.Conv2d + nn.BatchNorm2d(train) + nn.LeakyReLU and their autograd
 * backward, dark_net.py:22-33): the block moves the trunk's largest tensors for 0.6 % of its FLOPs, so neither its
 * pre-activation z nor dz is ever stored.
 *   avdn_conv0_fwd_stats  pass 1: stats [2,32] f64 = BatchNorm batch statistics of z (rounded to bf16, i.e. of the z a
 *                         stored tensor would hold; finish with avdn_bn_finalize), zw [32,3,3,3] fp32 =
 *                         sum_px z[px][co] * x[px+tap][ci], xs9 [9,4] f64 = total / border sums of x.  All three are
 *                         zeroed by the call and feed avdn_conv0_bwd.
 *   avdn_conv0_fwd_apply  pass 2: a [N,H,W,32] bf16 = leaky(bf16(conv(x)) * scale + shift).
 *   avdn_conv0_bwd        da [N,H,W,32] bf16 -> dw += scale*Gw + A*Zw + B*Xw (the weight gradient of
 *                         dz = scale*g + A*z + B without forming dz), dgamma += rstd*S2, dbeta += S1;
 *                         sums [2,32] f64 and gw [32,3,3,3] fp32 are scratch.   W % 16 == 0, H % 2 == 0.
 * The three passes (and avdn_conv0_fwd_eval) run on the tcgen05 tensor cores by default (csrc/conv0_tc.cu: one
 * 128-pixel im2col tile per UMMA, every per-channel sum taken as a Gram product of the same tile; any H, W with
 * N*H*W < 2^31).  On that path z is never rounded to bf16 (statistics, activation and the LeakyReLU mask all come
 * from the fp32 accumulator), xs9 carries Xw [3,3,3] f64 (sum of the input patches) instead of the border sums,
 * avdn_conv0_fwd_apply writes mask [N*H*W] u32 (bit 31-c = a[c] > 0; may be NULL when no backward follows) and
 * avdn_conv0_bwd reads it instead of recomputing z (the mma.sync kernels ignore mask), and the library keeps 32 KB
 * of per-device f64 scratch plus the coefficients in constant memory, so calls for one device must be issued on
 * one stream.  avdn_conv0_set_tensor_path(0) (or AVDN_CONV0_TC=0 in the environment)
 * selects the warp-level mma.sync kernels instead; the argument -1 only queries.  Returns the previous setting.
 * fwd_stats and bwd of one step must run under the same setting.                                               */
int avdn_conv0_set_tensor_path(int on);
int avdn_conv0_fwd_stats(const void* x_nhwc4, const float* w, int N, int H, int W, double* stats, float* zw,
                         double* xs9, avdn_stream_t stream);
int avdn_conv0_fwd_apply(const void* x_nhwc4, const float* w, const float* scale, const float* shift, float slope,
                         void* a, void* mask, int N, int H, int W, avdn_stream_t stream);
int avdn_conv0_bwd(const void* x_nhwc4, const float* w, const void* da, const void* mask, const float* scale,
                   const float* shift,
                   const float* mean, const float* rstd, float slope, int N, int H, int W, const float* zw,
                   const double* xs9, double* sums, float* gw, float* dw, float* dgamma, float* dbeta,
                   avdn_stream_t stream);

/* 3x3 stride-1 pad-1 convolution of a THIN layer (nn.Conv2d, dark_net.py:22-28; e.g. module_list.3: 32 -> 64 channels
 * at 112 x 112) with halo-tile reuse of the input (csrc/conv3_halo.cu): x [N,H,W,Cin] bf16, w_f [Cout, 9*Cin] bf16
 * (tap-major, the layout avdn_pack_conv_weights writes), z [N,H,W,Cout] bf16, stats NULL or [2,Cout] f64 (BatchNorm
 * batch statistics of the rounded z, zeroed by the call).  Same result as the avdn_gemm_* CONV launch of that layer.
 * avdn_conv3x3_thin_supported returns 1 for the shapes it covers (Cin 32, Cout 64, H % 16 == 0, W % 8 == 0).      */
int avdn_conv3x3_thin_fwd(const void* x_nhwc, const void* w_f, void* z, int N, int H, int W, int Cin, int Cout,
                          double* stats, avdn_stream_t stream);
int avdn_conv3x3_thin_supported(int H, int W, int Cin, int Cout);
/* Data gradient of the same layer: dx [N,H,W,Cin] bf16 = 3x3 convolution of dz [N,H,W,Cout] bf16 with the mirrored
 * filters, w_d [Cin, 9*Cout] bf16 (avdn_pack_conv_weights' second output).  Overwrites dx.  Same shapes.       */
int avdn_conv3x3_thin_dgrad(const void* dz, const void* w_d, void* dx, int N, int H, int W, int Cin, int Cout,
                            avdn_stream_t stream);
/* Weight gradient of the same layer: dw [Cout,Cin,3,3] fp32 (nn.Conv2d layout) += sum over pixels dz * x.       */
int avdn_conv3x3_thin_wgrad(const void* dz, const void* x_nhwc, float* dw, int N, int H, int W, int Cin, int Cout,
                            avdn_stream_t stream);

/* nn.BatchNorm2d in train mode (dark_net.py:31; eps 1e-5, momentum 0.1): batch
 * statistics of z [R,C] bf16 -> per-channel affine scale = gamma*rstd,
 * shift = beta - mean*scale, plus mean/rstd for the backward pass; updates the
 * running buffers (NULL to skip).  sums [4,C] f64 is scratch (shared with
 * avdn_bn_backward).  Channels >= C_real are padding (scale = shift = 0).
 * C must be 8 * (a divisor of 256).                                           */
int avdn_bn_stats(const void* z, long long R, int C, int C_real, const float* gamma, const float* beta,
                  float* running_mean, float* running_var, float momentum, float eps, double* sums,
                  float* scale, float* shift, float* mean, float* rstd, avdn_stream_t stream);
/* The second half of avdn_bn_stats alone: sums [2,C] f64 (sum, sum of squares over R rows) were
 * produced by the convolution's epilogue (avdn_gemm_core.stats).                              */
int avdn_bn_finalize(const double* sums, long long R, int C, int C_real, const float* gamma, const float* beta,
                     float* running_mean, float* running_var, float momentum, float eps, float* scale,
                     float* shift, float* mean, float* rstd, avdn_stream_t stream);
/* eval mode: the same affine from the running statistics. */
int avdn_bn_eval_coeffs(int C, int C_real, const float* gamma, const float* beta, const float* running_mean,
                        const float* running_var, float eps, float* scale, float* shift, avdn_stream_t stream);
/* a = LeakyReLU_slope(z*scale + shift) (+ residual): BN apply + nn.LeakyReLU()
 * (dark_net.py:33, slope 0.01) + the shortcut add (dark_net.py:224-226).       */
int avdn_bn_apply(const void* z, const float* scale, const float* shift, const void* residual, void* a,
                  long long R, int C, float slope, avdn_stream_t stream);
/* Backward of the above (train mode): dz [R,C] bf16 from da; dgamma/dbeta (+=, the
 * C_real real channels).  The residual branch receives da unchanged (caller).
 * sums [4,C] f64 scratch: two reduction rows, then the per-channel coefficients
 * of the apply pass.                                                           */
int avdn_bn_backward(const void* da, const void* z, const float* scale, const float* shift, const float* mean,
                     const float* rstd, long long R, int C, int C_real, float slope, double* sums, void* dz,
                     float* dgamma, float* dbeta, avdn_stream_t stream);
/* The second half of avdn_bn_backward alone: `sums` [2,C] f64 (sum g, sum g*(z-mean)) were produced by the
 * epilogue of the data-gradient convolution that wrote `da` (avdn_gemm_core.bnb_*); `coef` [4,C] fp32 scratch. */
int avdn_bn_backward_apply(const void* da, const void* z, const float* scale, const float* shift,
                           const float* mean, const float* rstd, long long R, int C, int C_real, float slope,
                           const double* sums, float* coef, void* dz, float* dgamma, float* dbeta,
                           avdn_stream_t stream);

/* Traversal order of the three elementwise BatchNorm passes (a tuning knob, results are the same sums in another
 * order): bit 0 = avdn_bn_apply walks the tensor back to front, bit 1 = the reduction of avdn_bn_backward does,
 * bit 2 = its apply pass does, bit 3 = one-wave grids (implied by the others), bit 4 = eight instead of four
 * 16-byte loads per tensor in flight per thread.  A producer leaves the tail of its
 * output in L2 and a consumer starts at the head.  AVDN_BN_ORDER in the environment sets the initial value
 * (default 25; 0 = the multi-wave front-to-back grids of ABI <= 7); the argument -1 only queries.  Returns the
 * previous setting.                                                                                            */
int avdn_bn_set_order(int mask);

/* nn.Conv2d weight [Cout,Cin,k,k] fp32 -> GEMM operands (bf16, zero padded):
 * wf [Cout_p][k*k][Cin_p] (forward / wgrad layout), wd [Cin_p][k*k][Cout_p] (dgrad). */
int avdn_pack_conv_weight(const float* w, int Cout, int Cin, int k, int Cout_p, int Cin_p, void* wf, void* wd,
                          avdn_stream_t stream);
/* grad [Cout,Cin,k,k] fp32 += dwf [Cout_p][k*k][Cin_p] fp32 (WGRAD output layout). */
int avdn_unpack_conv_wgrad(const float* dwf, int Cout, int Cin, int k, int Cin_p, float* grad,
                           avdn_stream_t stream);
/* The same for a gradient computed on pixel-pair views (32-channel activations keep 128-byte
 * operand rows when two adjacent pixels are read as one row; planners in gemm.py):
 * dwp is [2*Cout_p][k*3][2*Cin_p] (stride 1, k = 3), [2*Cout_p][1][2*Cin_p] (k = 1) or
 * [Cout_p][3*2][2*Cin_p] (stride 2); grad [Cout,Cin,k,k] fp32 += the blocks of each tap.   */
int avdn_unpack_conv_wgrad_pairs(const float* dwp, int Cout, int Cin, int k, int stride, int Cout_p, int Cin_p,
                                 float* grad, avdn_stream_t stream);
/* The three calls above for a whole trunk in ONE launch each.  `items_dev` is a DEVICE array describing the
 * tcgen05 convolution blocks in layer order; avdn_pack_conv_weights packs all of them (w -> wf, wd),
 * avdn_unpack_conv_wgrads adds the WGRAD outputs of entries [first, first+count) into their gradients
 * (grad += dwf, plain or pixel-pair layout).                                                            */
typedef struct avdn_conv_item {
  const float* w;   /* [Cout,Cin,k,k] fp32 master weight (pack) */
  void* wf;         /* bf16 [Cout_p][k*k][Cin_p] (pack) */
  void* wd;         /* bf16 [Cin_p][k*k][Cout_p] (pack) */
  const float* dwf; /* WGRAD output (unpack); NULL: the entry is skipped by avdn_unpack_conv_wgrads */
  float* grad;      /* [Cout,Cin,k,k] fp32 gradient, accumulated (unpack) */
  int32_t Cout, Cin, k, stride, Cout_p, Cin_p;
  int32_t pairs;    /* 1: dwf is in the pixel-pair layout of avdn_unpack_conv_wgrad_pairs */
  int32_t pad_;
} avdn_conv_item;
int avdn_pack_conv_weights(const avdn_conv_item* items_dev, int n_items, avdn_stream_t stream);
int avdn_unpack_conv_wgrads(const avdn_conv_item* items_dev, int first, int count, avdn_stream_t stream);
int avdn_cast_f32_bf16(const float* in, void* out, long long n, avdn_stream_t stream);
/* Trunk output [N,HW,C] bf16 NHWC -> `frames` [N,C,HW] fp32 (the .view at
 * src/xview_et/agent.py:594) and its adjoint for the backward pass.           */
int avdn_nhwc_to_nchw_f32(const void* in, float* out, int N, int HW, int C, avdn_stream_t stream);
int avdn_nchw_f32_to_nhwc(const float* in, void* out, int N, int HW, int C, avdn_stream_t stream);

/* ------------------------------------------------------------------------
 * Stage 3 — episodic cross-modal transformer "ET" (src/models/ET_haa.py,
 * enc_vl.py, encodings.py, model_util.py).  d_model is 768 (hard-coded by the
 * reference: ET_haa.py:98-119).  The dense contractions run through
 * avdn_gemm_*; these are the warp-level kernels around them.  fp32 tensors
 * unless stated.
 * ---------------------------------------------------------------------- */

/* SoftDotAttention(49) over the 512 channels of every frame, T frames per
 * sample, followed by fc2 (ET_haa.py:54-74,138-144):
 *   frames [B*T,512,49], lang_cls [B,49], w_in [49,49], w_out [49,98],
 *   fc2_w [768,49], fc2_b [768]
 *   -> attn [B*T,512], wc [B*T,49], e49 [B*T,49] (saved for backward),
 *      emb [B*T,768] = emb_frames.                                          */
/* fc2_w == NULL: SoftDotAttention only (ViT_LSTM's attention_layer_vision,
 * vln_model.py:219); emb is then not written.                              */
int avdn_frame_attn_fwd(const float* frames, const float* lang_cls, const float* w_in, const float* w_out,
                        const float* fc2_w, const float* fc2_b, int B, int T, float* attn, float* wc, float* e49,
                        float* emb, avdn_stream_t stream);
/* Backward: d_frames [B*T,512,49] is overwritten; the parameter gradients are
 * accumulated (+=).  lang_cls receives no gradient (it is a detached input of
 * the path, src/xview_et/agent.py:527-538 feeds BERT's output).             */
int avdn_frame_attn_bwd(const float* frames, const float* lang_cls, const float* w_in, const float* w_out,
                        const float* fc2_w, int B, int T, const float* attn, const float* wc, const float* e49,
                        const float* d_emb, float* d_frames, float* d_w_in, float* d_w_out, float* d_fc2_w,
                        float* d_fc2_b, avdn_stream_t stream);
/* The same, also accumulating (+=) the gradient of the query into d_lang_cls [B,49] (NULL to skip): in the
 * reference lang_cls = linear_cls comes from the trained BERT head (src/xview_et/agent.py:527-543).
 * fc2_w == NULL (ViT_LSTM's attention_layer_vision, vln_model.py:219, as in avdn_frame_attn_fwd): d_emb is read
 * as d_e49 [B*T,49], the gradient of the attention output, and d_fc2_w / d_fc2_b may be NULL.                */
int avdn_frame_attn_bwd_cls(const float* frames, const float* lang_cls, const float* w_in, const float* w_out,
                        const float* fc2_w, int B, int T, const float* attn, const float* wc, const float* e49,
                        const float* d_emb, float* d_frames, float* d_w_in, float* d_w_out, float* d_fc2_w,
                        float* d_fc2_b, float* d_lang_cls, avdn_stream_t stream);

/* PosEncoding + concat + direction embedding (encodings.py:22-49,
 * enc_vl.py:71-83, ET_haa.py:147):
 *   v[b] = [lang[b] + pe[:L] ; emb_frames[b] + pe[L:L+T] ; (W_d dirs[b] + b_d) + pe[L:L+T]] / with
 *   pe scaled by 1/sqrt(768).  lang [B,L,768], emb_frames [B,T,768], dirs [B,T,2],
 *   wd [768,2], bd [768], pe [>=L+T,768] -> v [B,L+2T,768].
 *   wd == NULL: `dirs` is the already embedded [B,T,768] (EncoderVL.forward's
 *   emb_directions, enc_vl.py:34-40).                                        */
int avdn_embed_fwd(const float* lang, const float* emb_frames, const float* dirs, const float* wd, const float* bd,
                   const float* pe, int B, int L, int T, float* v, avdn_stream_t stream);
/* d_wd [768,2] += , d_bd [768] += from dv [B,L+2T,768] (direction rows). */
int avdn_embed_dir_bwd(const float* dv, const float* dirs, int B, int L, int T, float* d_wd, float* d_bd,
                       avdn_stream_t stream);

/* (residual add +) nn.LayerNorm(768, eps): v = a (+ b); y = LN(v)*gamma + beta.
 * Outputs (each may be NULL except mean/rstd): v_out (the sum, kept for backward),
 * y fp32, y16 bf16 (the next GEMM's operand), mean/rstd [M].                 */
int avdn_ln_fwd(const float* a, const float* b, const float* gamma, const float* beta, long long M, int D, float eps,
                float* v_out, float* y, void* y16, float* mean, float* rstd, avdn_stream_t stream);
/* dy = dy1 (+ dy2) -> dv fp32 and/or dv16 bf16; dgamma/dbeta [768] += .      */
int avdn_ln_bwd(const float* dy1, const float* dy2, const float* v, const float* mean, const float* rstd,
                const float* gamma, long long M, int D, float* dv, void* dv16, float* dgamma, float* dbeta,
                avdn_stream_t stream);

/* Masked softmax of the attention scores.  The block-causal attention mask
 * (model_util.py:213-241) and the key-padding mask (enc_vl.py:44-55) are
 * evaluated as a predicate of (q, k, L, T, lens[b]) — never materialised.
 *   scores [B,H,S,Sp] fp32 (S = L+2T, Sp >= S row pitch) -> P [B,H,S,Sp] bf16,
 *   zero where masked and in the pitch padding.  T = 0: plain key-padding mask, keys k < lens[b] (BERT).  */
int avdn_softmax_fwd(const float* scores, const int* lens, int B, int H, int L, int T, int Sp, void* P,
                     avdn_stream_t stream);
/* dS = alpha * P * (dP - sum_k P*dP), bf16, zero in the padding. */
int avdn_softmax_bwd(const void* P, const float* dP, long long rows, int S, int Sp, float alpha, void* dS,
                     avdn_stream_t stream);
/* Train mode: the nn.Dropout sites of nn.TransformerEncoderLayer (enc_vl.py:16-22, p =
 * dropout_transformer_encoder) and of the heads (ET_haa.py:98-119, p = 0.2).  A mask is never stored:
 * element `idx` of site `site` is kept iff hash24(seed, site, idx) >= p * 2^24, and the forward and the
 * backward kernel evaluate the same hash.  Kept values are scaled by 1/(1-p); p = 0 disables.
 *   avdn_ln_fwd_drop      v = a + dropout(b)            (dropout1 / dropout2; idx = row*768 + col)
 *   avdn_ln_bwd_drop      dv16 = dropout'(dv) (gradient of the branch b); dv fp32 stays the residual gradient
 *   avdn_softmax_fwd_drop P = dropout(softmax) (operand of the PV GEMM), P_full = softmax (for the backward);
 *                         idx = row*Sp + k over [B,H,S,Sp]
 *   avdn_softmax_bwd_drop P = P_full, dP = gradient w.r.t. the dropped probabilities
 *   avdn_dropout_bf16     in-place dropout of a bf16 tensor (FFN hidden activation; its backward is the
 *                         relu_mask epilogue with alpha = 1/(1-p))
 *   avdn_dropout_keep_scale  out[idx] = 0 or 1/(1-p): the mask of a site, for tests
 *   avdn_heads_fwd_drop   sites site (h0, idx = b*256+o), site+1 (h1, b*32+o), site+2 (fc, b*64+o)
 *   avdn_heads_bwd_drop   p of the forward (dropped activations are stored as zeros)                    */
int avdn_ln_fwd_drop(const float* a, const float* b, const float* gamma, const float* beta, long long M, int D,
                     float eps, float* v_out, float* y, void* y16, float* mean, float* rstd, float p,
                     unsigned long long seed, unsigned int site, avdn_stream_t stream);
int avdn_ln_bwd_drop(const float* dy1, const float* dy2, const float* v, const float* mean, const float* rstd,
                     const float* gamma, long long M, int D, float* dv, void* dv16, float* dgamma, float* dbeta,
                     float p, unsigned long long seed, unsigned int site, avdn_stream_t stream);
int avdn_softmax_fwd_drop(const float* scores, const int* lens, int B, int H, int L, int T, int Sp, void* P,
                          void* P_full, float p, unsigned long long seed, unsigned int site, avdn_stream_t stream);
int avdn_softmax_bwd_drop(const void* P, const float* dP, long long rows, int S, int Sp, float alpha, void* dS,
                          float p, unsigned long long seed, unsigned int site, avdn_stream_t stream);
int avdn_dropout_bf16(void* x, long long n, float p, unsigned long long seed, unsigned int site,
                      avdn_stream_t stream);
int avdn_dropout_keep_scale(float* out, long long n, float p, unsigned long long seed, unsigned int site,
                            avdn_stream_t stream);
/* In-place dropout of an fp32 tensor, x16 (bf16 shadow, may be NULL) refreshed; and out = dropout'(a + b)
 * (b may be NULL): the gradient entering a dropout site (BertEmbeddings.dropout, CustomBERTModel.linears[2]). */
int avdn_dropout_f32(float* x, void* x16, long long n, float p, unsigned long long seed, unsigned int site,
                     avdn_stream_t stream);
int avdn_add_dropout_f32(const float* a, const float* b, float* out, long long n, float p, unsigned long long seed,
                         unsigned int site, avdn_stream_t stream);
/* avdn_add_dropout_f32 over a slice that starts at element idx0 of a larger tensor of the same site: element i
 * draws the mask of element idx0 + i (one time step of ViT_LSTM's input dropout, drawn as over the whole rollout). */
int avdn_add_dropout_f32_at(const float* a, const float* b, float* out, long long n, long long idx0, float p,
                            unsigned long long seed, unsigned int site, avdn_stream_t stream);
int avdn_heads_fwd_drop(const float* x, int B, int S, int row_vis, int row_dir, const float* w0, const float* b0,
                        const float* w1, const float* b1, const float* w2, const float* b2, const float* wf,
                        const float* bf, float* h0, float* h1, float* output, float* h_sali, float p,
                        unsigned long long seed, unsigned int site, avdn_stream_t stream);
int avdn_heads_bwd_drop(const float* x, int B, int S, int row_vis, int row_dir, const float* w0, const float* w1,
                        const float* w2, const float* wf, const float* h0, const float* h1, const float* h_sali,
                        const float* d_output, const float* d_h_sali, float* dx, float* dw0, float* db0, float* dw1,
                        float* db1, float* dw2, float* db2, float* dwf, float* dbf, float p, avdn_stream_t stream);

/* Incremental attention of the ET inference path (NavCMTAgent.rollout, src/xview_et/agent.py:580-760 re-runs the
 * whole encoder every step; the rows of earlier steps cannot change because the attention mask is causal over
 * steps, model_util.py:213-241).  The R new rows of a step (frame t, direction t) attend to the first n rows of
 * the layer's cache: qkv_new [B*R,2304] bf16 (q|k|v; q is read), cache [B,Lc,1536] bf16 (k|v per row: language
 * rows, then frame/direction rows of steps 0..t interleaved), ctx [B*R,768] bf16 = softmax(q k^T * scale) v.  */
int avdn_attn_decode(const void* qkv_new, const void* cache, int B, int R, int H, int Lc, int n, float scale,
                     void* ctx, avdn_stream_t stream);

/* ------------------------------------------------------------------------
 * Language encoder (SURVEY.md §8f N1): CustomBERTModel, src/models/vln_model.py:128-159 = HuggingFace BertModel
 * ('bert-base-uncased' architecture) + Linear(768,64)-ReLU-Dropout-Linear(64,49)-ReLU on the pooler output; call
 * sites src/xview_et/agent.py:527-538.  GEMMs: avdn_gemm_*; LayerNorm (eps 1e-12): avdn_ln_*; masked softmax:
 * avdn_softmax_* with T = 0 (key-padding mode: sample b attends keys k < lens[b]); these are the rest.
 * ---------------------------------------------------------------------- */
/* BertEmbeddings: v = (word[ids] + token_type[0]) + position[s]; y = LayerNorm(v) (eps).  ids [B,S] int64 (clamped
 * to the vocabulary).  Outputs as avdn_ln_fwd (v_out / y / y16 may be NULL).                                     */
int avdn_bert_embed_ln(const long long* ids, const float* word, const float* pos, const float* type0,
                       const float* gamma, const float* beta, int B, int S, int vocab, float eps, float* v_out,
                       float* y, void* y16, float* mean, float* rstd, avdn_stream_t stream);
/* d_word[ids] += dv, d_pos[s] += dv, d_type0 += dv  (dv [B*S,768] = gradient w.r.t. v).                          */
int avdn_bert_embed_bwd(const long long* ids, const float* dv, int B, int S, int vocab, float* d_word, float* d_pos,
                        float* d_type0, avdn_stream_t stream);
/* erf-GELU (hidden_act = "gelu") of a bf16 tensor and its backward du = dh * gelu'(u).                          */
int avdn_gelu_fwd(const void* u, void* h, long long n, avdn_stream_t stream);
int avdn_gelu_bwd(const void* u, const void* dh, void* du, long long n, avdn_stream_t stream);
/* Backward of y = act(x w^T + b) for the small fp32 heads (BertPooler, CustomBERTModel.linears): with
 * g = dy * act'(y) (act 0 none / 1 ReLU / 2 tanh):  dx [M,K] (row pitch lddx; += if dx_accumulate; may be NULL),
 * dw [N,K] +=, db [N] += (may be NULL).  x [M,K] row pitch ldx; y, dy [M,N] dense.                                */
int avdn_linear_f32_bwd(const float* x, long long ldx, const float* w, const float* y, const float* dy, int M, int N,
                        int K, int act, float* dx, long long lddx, int dx_accumulate, float* dw, float* db,
                        avdn_stream_t stream);

/* The two masks materialised exactly as the reference builds them (bit-exact
 * parity tests): mask_pad [B,S] u8 (1 = padded key), mask_attn [S,S] f32 (0 / -inf). */
int avdn_build_masks(const int* lens, int B, int L, int T, uint8_t* mask_pad, float* mask_attn,
                     avdn_stream_t stream);
/* out[n] += sum_m in[m][n] (bias gradients); in is bf16 (AVDN_DT_BF16) or fp32. */
int avdn_colsum(const void* in, int in_dtype, long long M, int N, long long ld, float* out, avdn_stream_t stream);

/* Row gather + waypoint MLP + saliency FC (ET_haa.py:157-166):
 *   x [B,S,768]; dir row -> 768->256 ReLU ->32 ReLU ->4 = output [B,4];
 *   vis row -> 768->64 ReLU = h_sali [B,64] (the 8x8 map before the upsample).
 *   h0 [B,256], h1 [B,32] are saved for the backward pass.                    */
int avdn_heads_fwd(const float* x, int B, int S, int row_vis, int row_dir, const float* w0, const float* b0,
                   const float* w1, const float* b1, const float* w2, const float* b2, const float* wf,
                   const float* bf, float* h0, float* h1, float* output, float* h_sali, avdn_stream_t stream);
/* dx [B,S,768] must be zero-filled by the caller; only the two gathered rows are
 * written.  Parameter gradients are accumulated (+=).                          */
int avdn_heads_bwd(const float* x, int B, int S, int row_vis, int row_dir, const float* w0, const float* w1,
                   const float* w2, const float* wf, const float* h0, const float* h1, const float* h_sali,
                   const float* d_output, const float* d_h_sali, float* dx, float* dw0, float* db0, float* dw1,
                   float* db1, float* dw2, float* db2, float* dwf, float* dbf, avdn_stream_t stream);

/* ------------------------------------------------------------------------
 * Agent slice (src/xview_et/agent.py): loss, waypoint post-processing, optimiser
 * ---------------------------------------------------------------------- */

/* Supervision geometry of the training rollout (SURVEY.md §8f N3): compute_iou (src/xview_et/agent.py:46-78) and
 * teacher_action (agent.py:386-507), evaluated by the reference with shapely per sample.  teacher_feedback = 0
 * (self.feedback == 'student'): the target is where the segment view centre -> goal centre leaves the view;
 * 1 ('teacher'): the point of (ground-truth path intersected with the view) closest to the goal, with the student
 * rule as the fallback when the path misses the view (agent.py:451-456).
 *   corners [B,4,2] f64 (lat,lng) current view; gt_path_corners [B,pmax,4,2] f64 with gt_len[b] valid steps;
 *   ended [B] u8  ->  next_pos_ratio [B,2] f32 (target of output[:,0:2]; zero when ended or progress > 0.5),
 *   altitude [B] f32 (teacher_a[i][1]), progress [B] f32 = IoU with the last ground-truth view, where the
 *   reference's "IoU" is intersection area / area of the convex hull of the eight corners.                      */
int avdn_teacher_action(const double* corners, const double* gt_path_corners, int pmax, const int32_t* gt_len,
                        const uint8_t* ended, int B, int teacher_feedback, float* next_pos_ratio, float* altitude,
                        float* progress, avdn_stream_t stream);

/* Per-step loss and its gradient in one kernel (agent.py:663-681,883-885):
 *   loss_i = |p_xy-g_xy|^2 + (ang(p)-ang(g))^2 + (alt-g_alt)^2 + (prog-g_prog)^2
 *            [+ nss_w * NSS(upsample(h_sali_i), att_i/255) if sum(att_i) > 0]
 *   *loss_total += scale * sum_i loss_i   (scale = train_ml / batch_size)
 *   d_output [B,4], d_h_sali [B,64] = scale * d loss_i / d(...)
 * att [B,224,224] u8 is avdn_render_views' attention output (NULL: no NSS term);
 * jitter [B] stands for 1e-5*np.random.rand() of agent.py:666 (NULL: 0).
 * The F.interpolate(8x8 -> 224x224, bilinear, align_corners=False) of
 * ET_haa.py:166-167 and its adjoint are fused in.  float64 accumulation as the
 * reference's promotion through gt_saliency (env.py:293).                      */
int avdn_loss(const float* output, const float* h_sali, const float* gt_xy, const float* gt_alt,
              const float* gt_prog, const uint8_t* att, const float* jitter, int B, float nss_w, int nss_r,
              double scale, double* loss_total, double* loss_i, float* d_output, float* d_h_sali,
              avdn_stream_t stream);
/* pred_saliency [B,1,224,224] = F.interpolate(h_sali.view(B,1,8,8)) (ET_haa.py:166-167). */
int avdn_upsample_saliency(const float* h_sali, int B, float* pred, avdn_stream_t stream);
/* adjoint: d_h_sali [B,64] = upsample^T d_pred [B,1,224,224] (overwrites). */
int avdn_upsample_saliency_bwd(const float* d_pred, int B, float* d_h_sali, avdn_stream_t stream);
/* Human-attention validation scores of N rows (xview_et/agent.py:683-693, evaluated per sample): with
 * sal = avdn_upsample_saliency(h_sali[n]) (the same device code, bit-identical pixels), gt = att[n] / 255 and
 * p = clip(sal, 0, 1), out[n] = (precision = sum p*gt / sum p (0 when sum p == 0), recall = sum p*gt / sum gt
 * (0 when sum gt == 0), nss = NSS(sal, gt) of the row (agent.py:256-270: unbiased std, nss_r in {-1,0,1},
 * sum gt + 0.001), fixation sum = sum gt).  h_sali [N,64] f32, att [N,224,224] u8, out [N,4] f64.
 * float64 sums, one CTA per row, a fixed reduction order: results repeat bit for bit.                       */
int avdn_saliency_metrics(const float* h_sali, const uint8_t* att, int N, int nss_r, double* out,
                          avdn_stream_t stream);
/* agent.py:637-653,738,745-752: normalise xy, clamp altitude / progress, discretise.
 *   output [B,4] f32, edge_len [B] f64 (= |c0-c1|) -> angle_deg [B] i32,
 *   dist [B] f64, altitude_m [B] i32, stop [B] u8, xy_norm [B,2] f32 (or NULL). */
int avdn_postprocess_waypoints(const float* output, const double* edge_len, int B, float stop_threshold,
                               int* angle_deg, double* dist, int* altitude_m, uint8_t* stop, float* xy_norm,
                               avdn_stream_t stream);
/* *out += sum g^2 (float64) — torch.nn.utils.clip_grad_norm_ (agent.py:247). */
int avdn_sumsq(const float* g, long long n, double* out, avdn_stream_t stream);
/* torch.optim.AdamW step over a flat arena (agent.py:153-156,249-251).  When
 * sumsq != NULL the gradient is first scaled by min(1, max_norm/(grad_scale*sqrt(*sumsq)+1e-6));
 * grad_scale multiplies every gradient (1/world_size for data-parallel means). */
int avdn_adamw(float* p, const float* g, float* m, float* v, long long n, float lr, float beta1, float beta2,
               float eps, float wd, int step, const double* sumsq, float max_norm, float grad_scale,
               avdn_stream_t stream);

/* ------------------------------------------------------------------------
 * Config 5 — recurrent policy "ViT_LSTM" (src/models/vln_model.py:163-250) and the
 * simulator update of the greedy rollout (src/xview_lstm/agent.py:592-602,700-730).
 * fp32 CUDA-core kernels: ~3 MFLOP per sample and step next to 15.3 GFLOP of trunk.
 * ---------------------------------------------------------------------- */

/* Which kernels serve avdn_linear_f32 and avdn_lang_attn_fwd: 2 (default) = 32 x 64 tiles with the operands of the
 * next k-step fetched into registers as float4 under the FMAs (used when K, ldx, ldw are multiples of 4 and x, w
 * are 16-byte aligned; the same sums in the same order as version 1, bit-identical) / float4 loads with two to eight
 * rows in flight in the attention (D % 4 == 0, D <= 1024; agrees with version 1 to fp32 summation order); 1 = the
 * first versions.  AVDN_LSTM_KERNELS=1 in the environment selects version 1
 * initially; any other argument than 1 or 2 only queries.  Returns the previous setting.                       */
int avdn_lstm_set_kernels(int version);
/* y[M,N] (+)= act(x[M,K] w[N,K]^T + b[N]); ld* are row pitches in elements;
 * act: 0 none, 1 ReLU, 2 tanh; b may be NULL.  nn.Linear / the two halves of
 * nn.LSTMCell's gate pre-activations (vln_model.py:178-204,224-236).           */
int avdn_linear_f32(const float* x, long long ldx, const float* w, long long ldw, const float* b, float* y,
                    long long ldy, int M, int N, int K, int act, int accumulate, avdn_stream_t stream);
/* nn.LSTMCell pointwise part: gates [B,4H] (order i,f,g,o, both bias vectors already added),
 * c_prev [B,H] or NULL (zero state, vln_model.py:224-226) -> h [B,H] (row pitch ldh), c [B,H]. */
int avdn_lstm_cell(const float* gates, const float* c_prev, float* h_out, long long ldh, float* c_out, int B, int H,
                   avdn_stream_t stream);
/* out[B,N] = W [N,2] . [sin, cos](deg / 180 * 3.14159) + b  (vln_model.py:228-229; float32). */
int avdn_direction_embed(const float* deg, const float* w, const float* b, float* out, int B, int N,
                         avdn_stream_t stream);
/* SoftDotAttention between the two Linear layers (vln_model.py:33-42):
 * attn = softmax_l(ctx[b,l,:] . target[b,:]); weighted[b,:] = sum_l attn_l ctx[b,l,:].
 * ctx [B,L,D], target [B,D] -> attn [B,L] (may be NULL), weighted [B,D] (row pitch ldw). */
int avdn_lang_attn_fwd(const float* ctx, const float* target, int B, int L, int D, float* attn, float* weighted,
                       long long ldw, avdn_stream_t stream);
/* Backward of avdn_lstm_cell (autograd of nn.LSTMCell's pointwise part, vln_model.py:224-236), from the saved
 * pre-activations gates [B,4H] (order i,f,g,o), c_prev [B,H] or NULL (zero state of the first step), and the saved
 * cell state c [B,H]; dh [B,H] has row pitch lddh (h lives inside a wider buffer); dc_next [B,H] or NULL (no
 * gradient from a later step).  dgates [B,4H] is overwritten (it is the gradient of both bias vectors and the
 * operand of the W_ih / W_hh gradients); dc_prev [B,H] is overwritten when c_prev is given, not written otherwise.
 * dc_next and dc_prev may be the same buffer.                                                                  */
int avdn_lstm_cell_bwd(const float* gates, const float* c_prev, const float* c, const float* dh, long long lddh,
                       const float* dc_next, float* dgates, float* dc_prev, int B, int H, avdn_stream_t stream);
/* Gradient of avdn_direction_embed's parameters (vln_model.py:228-229): d_w [N,2] += sum_s d_out[s] [sin, cos](a_s),
 * d_b [N] += sum_s d_out[s], with a_s = deg[s] / 180 * 3.14159 in float32 and the same sin / cos as the forward.
 * deg [B], d_out [B,N].                                                                                        */
int avdn_direction_embed_bwd(const float* deg, const float* d_out, int B, int N, float* d_w, float* d_b,
                             avdn_stream_t stream);
/* Backward of avdn_lang_attn_fwd (SoftDotAttention(768) over the dialog tokens, vln_model.py:33-42): from ctx
 * [B,L,D], target [B,D], the saved attn [B,L] and d_weighted [B,D] (row pitch lddw):
 * d_target [B,D] is overwritten; d_ctx [B,L,D] (the gradient of lang_feature) is accumulated (+=), NULL to skip.
 * Any L (2D + 2L floats of shared memory, at most 48 KB).                                                    */
int avdn_lang_attn_bwd(const float* ctx, const float* target, const float* attn, const float* d_weighted,
                       long long lddw, int B, int L, int D, float* d_target, float* d_ctx, avdn_stream_t stream);
/* One rollout step of the simulator for B samples (xview_lstm/agent.py:607-626,700-730 and
 * move_view_corners, xview_et/agent.py:285-384), float64, one thread per sample:
 *   output [B,4] f32 -> normalise / clamp / discretise (as avdn_postprocess_waypoints);
 *   stop = progress > stop_threshold or last_step: ended[i] = 1 and the pose is kept;
 *   otherwise zoom to the altitude, rotate by -angle about the centre, move forward by
 *   dist; each stage is rejected when a corner leaves (gps_botm_left, gps_top_right).
 * corners [B,4,2] f64 (lat,lng; FL,FR,BR,BL) in/out; bounds [B,4] f64 = (bl_lat, bl_lng,
 * tr_lat, tr_lng); cur_dir [B] f64 in/out (current_directions); ended [B] u8 in/out (sticky).
 * angle_deg / dist / altitude_m may be NULL.                                    */
int avdn_waypoint_step(const float* output, double* corners, const double* bounds, double* cur_dir,
                       uint8_t* ended, int B, float stop_threshold, int last_step, int* angle_deg, double* dist,
                       int* altitude_m, avdn_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* AVDN_H_ */
