/* rgbd_b200 -- C ABI of the B200-native DGGM / E-DSAM depth-guidance hot path.
 *
 * This is the drop-in boundary: a plain-C shared library (librgbd_b200.so) with raw device pointers,
 * sizes and a CUDA stream -- no torch types.  The reference is pure Python (PyTorch nn.Modules in
 * mask2former/utils/custom_model.py, "CM"; numpy/OpenCV in mask2former/utils/data_process.py, "DP"), so the
 * reference-side binding a maintainer adds is a ctypes stub (INTEGRATION.md); the Python mirror in
 * rgb-d-instance-segmentation_b200/ is exactly such a binding.
 *
 * Conventions: every entry point enqueues work on `stream` and returns immediately (no synchronisation, no
 * allocation: the caller supplies outputs and workspaces); return 0 on success, non-zero on error with the
 * text available from rgbd_last_error().  All pointers are DEVICE pointers unless named `*_host`.  Tensors
 * are contiguous unless a stride argument says otherwise; strides are in ELEMENTS.
 */
#ifndef RGBD_B200_H
#define RGBD_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* rgbd_stream_t; /* cudaStream_t */

#define RGBD_ABI_VERSION 4
#define RGBD_HIST_BINS 512 /* CM:701 `bins=512` */

#define RGBD_DTYPE_F32 0
#define RGBD_DTYPE_BF16 1
#define RGBD_DTYPE_U8 2

/* status flags written per image by rgbd_depth_decompose */
#define RGBD_DECOMP_RANGE_NOT_FINITE 1 /* numpy would raise "range ... is not finite" (all-NaN or inf depth) */

int rgbd_abi_version(void);
const char* rgbd_last_error(void);

/* ---- DGGM -------------------------------------------------------------------------------------------------
 * rgbd_dggm_fwd replaces DepthGradientInjectionResidual.forward (CM:1204-1269) for all scales in one launch:
 *   out_i = color_i + ReLU(W_i . (bilinear_down(grad) * nearest_down(mask)) + b_i)
 * and, if `branch1` is non-NULL, the v0.4.0 branch sum `cp1_i + cp2_i` (CM:354-355): out_i = branch1_i + (...).
 * color/out/branch1: n_scales pointers to (B, C[i], Hs[i], Ws[i]) fp32; weight[i]: (C[i], D); bias[i]: (C[i]);
 * grad: (B, D, H, W) with batch stride; mask: (B, 1, H, W) with batch stride.  The pointer ARRAYS are host
 * arrays.  The None-gradient passthrough (CM:1263-1265) is the caller's branch. */
int rgbd_dggm_fwd(int n_scales, const float* const* color_host, const float* const* branch1_host, float* const* out_host,
                  const int* C_host, const int* Hs_host, const int* Ws_host, const float* const* weight_host,
                  const float* const* bias_host, const float* grad, long long grad_batch_stride, const float* mask,
                  long long mask_batch_stride, int B, int D, int H, int W, rgbd_stream_t stream);

/* Parameter gradients of the same module (autograd of CM:1251): dW_i = sum 1[pre>0] dOut (x) gated_i,
 * db_i = sum 1[pre>0] dOut.  Colour features are detached (CM:332-333) and the gradient map is data, so no
 * other gradient exists.  dweight/dbias are overwritten. */
int rgbd_dggm_bwd_params(int n_scales, const float* const* dout_host, const int* C_host, const int* Hs_host,
                         const int* Ws_host, const float* const* weight_host, const float* const* bias_host,
                         float* const* dweight_host, float* const* dbias_host, const float* grad,
                         long long grad_batch_stride, const float* mask, long long mask_batch_stride, int B, int D, int H,
                         int W, rgbd_stream_t stream);

/* rgbd_gradient_features replaces calculate_gradient_features (DP:1247-1305) as called by map_10channel_case2
 * (mask2former/utils/dataloader.py:412-421): Sobel 3x3 (reflect-101), magnitude, invalid-depth zeroing,
 * valid mask, min-max normalisation.  depth: (B,H,W) f32 or u8; norm_out receives n_rep identical channels
 * (channel stride H*W); vmask_out one channel.  Bit-exact with the reference for uint8-valued depth. */
size_t rgbd_gradient_features_workspace_bytes(int B);
int rgbd_gradient_features(const void* depth, int depth_dtype, long long depth_batch_stride, float* norm_out,
                           long long norm_batch_stride, int n_rep, float* vmask_out, long long vmask_batch_stride, int B,
                           int H, int W, float invalid_value, void* workspace, rgbd_stream_t stream);

/* rgbd_pack_pixel_values builds the whole (B,10,H,W) model input of map_10channel_case2 (DL:386-425) on device from the
 * already-resized uint8 colour image (B,H,W,3) and uint8 depth image (B,H,W): channels 0:3 / 3:6 = the Hugging Face
 * processor's rescale + normalize of colour / depth-as-RGB (bit-exact with its numpy arithmetic), 6:9 + 9 = the
 * gradient features above.  workspace: rgbd_gradient_features_workspace_bytes(B). */
int rgbd_pack_pixel_values(const uint8_t* rgb_hwc, const uint8_t* depth, float* pixel_values, long long pv_batch_stride,
                           int B, int H, int W, double rescale_factor, const float* mean3_host, const float* std3_host,
                           float invalid_value, void* workspace, rgbd_stream_t stream);

/* ---- E-DSAM: depth decomposition ------------------------------------------------------------------------------
 * rgbd_depth_decompose replaces, for a whole batch and without host round trips, to_grayscale (CM:466-480) and
 * DSAModule._calculate_depth_histogram / _select_depth_distribution_modes / _define_depth_interval_windows /
 * _generate_depth_region_masks (CM:701-798) plus the adaptive_max_pool2d of every region mask (CM:687).
 * Input: depth3 (B,3,H,W) with batch/channel strides (gray written to gray_out) OR gray_in (B,H,W); ratio (B).
 * Outputs (optional ones may be NULL): hist_out int64 (B,512); edges_out f32 (B,513); n_modes_out (B);
 * peak_bins_out (B,3); centres_out (B,3); windows_out (B,3,2); status_out (B); bias_variant_out (B) = how many
 * conv biases the reference adds for the image (n_modes+1, or num_modes+1 when no mode survives, CM:676-691);
 * codes_out uint8 (B,H,W): bit t = region mask t in the reference's list order (modes by (height, centre) descending, then the remaining
 * region at index n_modes; all zero when no mode survives, CM:676-678); pooled_out_host[l] uint8
 * (B, level_h[l], level_w[l]) = the codes OR-pooled over adaptive_max_pool2d's windows.  codes_out may be NULL when the
 * levels are exactly (H/4,W/4), (H/8,W/8), (H/16,W/16) with H, W multiples of 16 (the Swin pyramid): codes and pooled copies
 * then come from one fused pass and the full-resolution codes need not be stored. */
size_t rgbd_depth_decompose_workspace_bytes(int B);
int rgbd_depth_decompose(const float* depth3, long long depth_batch_stride, long long depth_channel_stride,
                         const float* gray_in, const float* ratio, int B, int H, int W, int num_modes, float* gray_out,
                         long long* hist_out, float* edges_out, int* n_modes_out, int* peak_bins_out, float* centres_out,
                         float* windows_out, int* status_out, int* bias_variant_out, uint8_t* codes_out, int n_levels, const int* level_h_host,
                         const int* level_w_host, uint8_t* const* pooled_out_host, void* workspace, rgbd_stream_t stream);

/* ---- E-DSAM: tensor-core building blocks ------------------------------------------------------------------------
 * rgbd_dsam_pack builds the masked, K-concatenated bf16 operand of a DSAM stage (CM:683-696) from NCHW fp32
 * features and the pooled region codes: out[img][seg][parity][y2][x2][C_pad] (parity_split=1, 3x3 stride 2) or
 * out[img][seg][y][x][C_pad] (parity_split=0, 1x1).  Segments < masked_segs are multiplied by bit(code, seg);
 * the others are plain copies.  The caller zero-initialises `out` once (padding stays zero).  hi_lo=1 writes every
 * segment twice -- bf16(v) and bf16(v - bf16(v)), segment index 2*seg / 2*seg+1 -- for the split-precision ("fp32") mode. */
int rgbd_dsam_pack(const float* feat, const uint8_t* codes, void* out_bf16, int B, int C, int C_pad, int H, int W, int n_seg,
                   int masked_segs, int parity_split, int hi_lo, rgbd_stream_t stream);

/* GroupNorm(groups, C) of an fp32 NCHW tensor (B,C,HW), in place, affine gamma/beta (C) -- the normalisation half of the
 * pixel decoder's input_projections = Conv2d(C_i,256,1) + GroupNorm(32,256) (HF Mask2FormerPixelDecoder, called at
 * CM:383; SURVEY 8f-2); the conv half is rgbd_conv_gemm over the bf16 channels-last copy rgbd_dsam_pack(n_seg=1,
 * masked_segs=0, parity_split=0; codes may then be NULL) makes of the fused feature map. */
int rgbd_group_norm_inplace(float* x, const float* gamma, const float* beta, int B, int C, int HW, int groups, float eps,
                            rgbd_stream_t stream);

/* Row-im2col of the C-channel depth image (C = input_channels of the predictor, 1..4; the reference default is 3) for the
 * multi-scale stem (CM:1458-1460): out[img][H+6][W][64] bf16, channel (j*8+dx)*4+c = depth[img][c][r-3+j][x+dx-3], zero for c >= C. */
int rgbd_ratio_stem_pack(const float* depth3, long long batch_stride, long long channel_stride, void* out_bf16, int B, int C,
                         int H, int W, rgbd_stream_t stream);

/* Implicit-GEMM convolution on tcgen05/TMEM (see csrc/conv_gemm.cu).  A: bf16 channels-last tensor viewed as
 * (a_planes, a_y, a_x, a_c); each of the n_slices K blocks reads kb_elems channels at the tile's base coordinate
 * plus slices[j] = (c0, dx, dy, dplane) (out-of-range reads are zero).  W: bf16 (n_pad, n_slices*kb_elems).
 * Output tile = bx*by (=128) pixels of one image x block_n channels.  y = act(acc*scale[n] + shift[variant][n]);
 * epi_mode 0: bf16 (n_img, out_h, out_w, n_pad) store, optionally multiplied by `gate` (same layout);
 * epi_mode 1: fp32 (n_img, n, out_h, out_w) store, optionally + residual (same layout);
 * epi_mode 2: sums over the cells of a cells_y x cells_x grid into pool (n_img, cells, n_pad) (caller zeroes), as 64-bit
 *             FIXED-POINT integers in units of 1/RGBD_POOL_FIXED_ONE: integer atomics make the sums independent of the
 *             accumulation order, so the ratio (and the integer region codes derived from it) is reproducible run to run;
 * epi_mode 3: masked segment sum (see the codes / m3_* fields). */
#define RGBD_POOL_FIXED_ONE 16777216.0 /* 2^24 */
typedef struct rgbd_conv_gemm_desc {
    const void* a; /* bf16 */
    int a_c, a_x, a_y, a_planes;
    int plane_per_img;
    const void* w; /* bf16 */
    const int* slices; /* device, n_slices x 4 */
    int n_slices, kb_elems;
    int n_img, out_h, out_w, bx, by;
    int n, n_pad, block_n;
    int tile_order; /* 0: x fastest, 1: y fastest */
    int epi_mode, act; /* act: 0 none, 1 relu, 2 sigmoid, 3 statistics (epi_mode 2 only: sums of y and of y*y, no activation) */
    const float* scale;   /* (n_pad) or NULL */
    const float* shift;   /* (n_variants, n_pad) */
    const int* variant;   /* (n_img) or NULL */
    const void* gate;     /* bf16 or NULL */
    void* out;
    const float* residual;
    long long* pool;
    int cells_y, cells_x;
    int conv3x3_reuse; /* 1: 3x3 stride-1 pad-1 conv over a (n_img, a_y, a_x, a_c) tensor with shared-memory reuse of the
                          A tile across the dx taps; W is (n_pad, 9*a_c) ordered (dy, dx, c); slices are ignored;
                          needs kb_elems=64, bx=128, by=1 */
    /* epi_mode 3 (input gradient of a DSAM stage): the N axis is (channel block of 32, segment, 32 channels),
       block_n = 32*m3_n_seg; out/residual are fp32 (n_img, n, in_h, in_w); GEMM pixel (oy, ox) is input pixel
       (oy*m3_stride + m3_py, ox*m3_stride + m3_px); segment s < m3_masked_segs is kept where bit s of codes is set */
    const void* codes;
    int in_h, in_w, m3_py, m3_px, m3_stride, m3_masked_segs, m3_n_seg;
    /* dsam_masked = 1 (forward of a stride-2 DSAM stage, CM:683-696, masking done in shared memory): a is the UNMASKED
       parity-split operand (n_img*4 planes, rgbd_dsam_pack with n_seg=1, masked_segs=0); codes are the pooled region
       codes (n_img, in_h, in_w) at the INPUT resolution; W is (n_pad, 9*(a_c/64)*m3_n_seg*64) ordered
       (tap, channel block, segment, 64 channels), segment m3_n_seg-1 = rgb_projection, m3_masked_segs = m3_n_seg-1;
       needs epi_mode 1, kb_elems 64, plane_per_img 4; slices are ignored. */
    int dsam_masked;
    /* epi_mode 1 only: next_operand != NULL also writes the result as the NEXT stride-2 DSAM stage's operand, i.e. exactly
       what rgbd_dsam_pack(out, next_codes, next_operand, n_img, n, next_c_pad, out_h, out_w, next_n_seg, next_masked_segs,
       parity_split = 1, hi_lo = 0) would produce (bf16, (n_img, next_n_seg, 4, ceil(out_h/2), ceil(out_w/2), next_c_pad));
       next_codes: pooled region codes (n_img, out_h, out_w), needed when next_masked_segs > 0. */
    void* next_operand;
    const void* next_codes;
    int next_c_pad, next_n_seg, next_masked_segs;
    /* epi_mode 2 with act 3: the statistics pass of a train-mode BatchNorm (CM:1380-1421 under .train()): pool receives
       the cell sums of y = acc + shift, pool_sq (same shape, caller zeroes) the cell sums of y*y. */
    long long* pool_sq;
} rgbd_conv_gemm_desc;
int rgbd_conv_gemm(const rgbd_conv_gemm_desc* desc_host, rgbd_stream_t stream);

/* ---- E-DSAM backward (autograd of DSAModule.forward CM:683-696; colour features of stage 0 are detached CM:332) ----
 * rgbd_cast_bf16_pitched: (rows, W) fp32 -> bf16 with row pitch W_pitch (multiple of 8, zero padded).
 * rgbd_dsam_pack_t: like rgbd_dsam_pack but pixel-contiguous: out[img][seg][plane][C_pad][H2][W2_pitch] (zeroed by caller);
 *   with parity_split there are 6 planes: the 4 parity planes and right-shifted-by-one copies of the two px=1 planes
 *   (TMA needs a 16-byte aligned innermost start, so the x-1 tap reads a pre-shifted plane); the last column of a
 *   shifted plane is dropped when it does not fit the pitch (it never meets a non-zero gradient).
 * rgbd_dsam_dbias: db[t][n] = sum over images that use region t (t < variant[b]) of sum_pixels g[b][n]; db overwritten.
 * rgbd_dsam_wgrad: dw[n][seg][tap][C_pad] (fp32, overwritten) = sum_pixels g[b][n][oy][ox] * x_t[b][seg][tap-shifted pixel][c];
 *   g_bf16: (B, N_out, Ho, g_w_pitch); xt_bf16: output of rgbd_dsam_pack_t with plane height x_h and the SAME row pitch.
 * Split precision (DSAModule.grad_precision "fp32"): dst_lo / out_lo, when not NULL, receive the lo parts
 *   bf16(v - float(bf16(v))) in the layout of the hi output (pitch and pad zero, masked pixels +0); rgbd_dsam_wgrad given
 *   both g_lo and xt_lo accumulates G_hi.X_hi + G_lo.X_hi + G_hi.X_lo (~2^-16 relative instead of ~2^-8); NULL lo
 *   pointers select the bf16 operands alone.
 * The input gradient runs through rgbd_conv_gemm with epi_mode 3 (split precision: G packed by rgbd_dsam_pack with
 * hi_lo = 1, weights [W_hi | W_hi | W_lo] per K block). */
int rgbd_cast_bf16_pitched(const float* src, void* dst_bf16, void* dst_lo, long long rows, int W, int W_pitch,
                           rgbd_stream_t stream);
int rgbd_dsam_pack_t(const float* feat, const uint8_t* codes, void* out_bf16, void* out_lo, int B, int C, int C_pad, int H,
                     int W, int W2_pitch, int n_seg, int masked_segs, int parity_split, rgbd_stream_t stream);
int rgbd_dsam_dbias(const float* g, const int* variant, float* db, int B, int N, int HW, int n_bias, rgbd_stream_t stream);
int rgbd_dsam_wgrad(const void* g_bf16, const void* g_lo, int g_w_pitch, const void* xt_bf16, const void* xt_lo, int x_w_pitch,
                    int x_h, float* dw, int B, int N_out, int C_pad, int Ho, int Wo, int n_seg, int parity_split,
                    rgbd_stream_t stream);

/* Fused point-wise middle of EnhancedDepthImageRatioPredictor.forward (CM:1466-1470): feature_fusion (1x1 192->128 +
 * folded BN + ReLU), attention (1x1 128->64 + ReLU, 1x1 64->128 + sigmoid) and the gating multiply, as three chained
 * tcgen05 GEMMs per 128-pixel tile with the intermediates kept in tensor memory.  x1: bf16 (B,H,W,192);
 * w2 (128,192) with the folded BN scale multiplied in, w3 (64,128), w4 (128,64) bf16; sh2 (128): folded BN shift;
 * sh3 (64), sh4 (128): conv biases; out: bf16 (B,H,W,128).  Tile = bx*by (=128) pixels. */
int rgbd_ratio_chain(const void* x1_bf16, const void* w2_bf16, const void* w3_bf16, const void* w4_bf16, const float* sh2,
                     const float* sh3, const float* sh4, void* out_bf16, int B, int H, int W, int bx, int by,
                     rgbd_stream_t stream);

/* Multi-scale stem + point-wise middle of EnhancedDepthImageRatioPredictor.forward (CM:1458-1470) as ONE kernel on CTA
 * pairs: the stem GEMM (K = 256 row-im2col, N = 192) feeds rgbd_ratio_chain's three GEMMs through tensor memory, so the
 * 192-channel stem output never reaches HBM.  r: output of rgbd_ratio_stem_pack, bf16 (B,H+6,W,64); w1 (192,256) bf16 with
 * the folded BN scale multiplied in (K order = 4 slices x (j, dx8, c4), tap dy = 2*slice + j); sh1 (192): folded BN
 * shift; the other arguments as for rgbd_ratio_chain. */
int rgbd_ratio_front(const void* r_bf16, const void* w1_bf16, const void* w2_bf16, const void* w3_bf16, const void* w4_bf16,
                     const float* sh1, const float* sh2, const float* sh3, const float* sh4, void* out_bf16, int B, int H,
                     int W, int bx, int by, int compact_operand, rgbd_stream_t stream);
/* compact_operand = 1: r_bf16 is the output of rgbd_ratio_stem_pack_compact, E (B,2,H+6,Wp,4) bf16 with
 * Wp = rgbd_ratio_stem_compact_width(W): E[b][s][r][xx][c] = depth[b][c][r-3][xx+s-3] (zero outside, c == 3 zero) -- the
 * depth image channels-last in two copies shifted by one pixel; the kernel reads it through sliding-window tensor maps
 * (free im2col along x), so the 128-byte-per-pixel row-im2col tensor is never written.  Then w1 is (192, 224) with K
 * ordered (dy 7, dx 8, c 4); needs bx = 128, by = 1 and an even W. */
int rgbd_ratio_stem_compact_width(int W);
int rgbd_ratio_stem_pack_compact(const float* depth3, long long batch_stride, long long channel_stride, void* out_bf16, int B,
                                 int C, int H, int W, rgbd_stream_t stream);

/* Tail of EnhancedDepthImageRatioPredictor.forward (CM:1473-1485): pooled sums -> conv3x3 256->512 + folded BN +
 * ReLU -> GAP -> MLP -> 0.01 + 0.49*sigmoid.  conv_w (512,256,3,3) fp32; fc_w_host/fc_b_host: 4 layers. */
int rgbd_ratio_tail(const long long* pool_sums, int pool_stride, int cell_pixels, const float* conv_w, const float* conv_scale,
                    const float* conv_shift, const float* const* fc_w_host, const float* const* fc_b_host, float out_min,
                    float out_max, float* gap_ws, float* ratio_out, int B, rgbd_stream_t stream);

/* AdaptiveAvgPool2d(4) (CM:1417) of a bf16 channels-last (B,H,W,256) map for H or W not divisible by 4 (torch's overlapping
 * windows); pool_means (B,16,256) receives the window MEANS in RGBD_POOL_FIXED_ONE fixed point: pass cell_pixels = 1 to the
 * tail.  (Divisible sizes pool inside rgbd_conv_gemm's epilogue and never write the map.) */
int rgbd_adaptive_avg_pool4(const void* x_bf16, long long* pool_means, int B, int H, int W, rgbd_stream_t stream);

/* Tensor-core variant of the tail: rgbd_ratio_tail_prepare turns the pooled sums into the bf16 channels-last 4x4 map
 * a (B,4,4,256) and zeroes gap_fx (B,512); rgbd_conv_gemm (3x3 taps as slices, epi_mode 2 with a 1x1 cell grid, act 1) adds
 * ReLU(BN(conv)) summed over the 16 pixels into gap_fx as fixed point; rgbd_ratio_tail_mlp_fx = GAP/16 -> MLP -> ratio. */
int rgbd_ratio_tail_prepare(const long long* pool_sums, int pool_stride, int cell_pixels, void* a_bf16, long long* gap_fx, int B,
                            rgbd_stream_t stream);
int rgbd_ratio_tail_mlp_fx(const long long* gap_fx, const float* const* fc_w_host, const float* const* fc_b_host, float out_min,
                           float out_max, float* ratio_out, int B, rgbd_stream_t stream);

/* The same tail under .train() (CM:1418-1437 with BatchNorm2d in training mode and active Dropout): conv3x3 256->512 ->
 * BatchNorm over the batch's (B,4,4) samples per channel (biased variance for normalisation; running_mean / running_var,
 * when given, are updated in place: (1-momentum)*old + momentum*(batch mean incl. conv bias | unbiased variance)) -> ReLU
 * -> GAP -> MLP, where drop0 (B,128) / drop1 (B,64) are the Dropout multipliers keep/(1-p) (NULL = no dropout).
 * raw_ws: B*512*16 floats, gap_ws: B*512 floats. */
int rgbd_ratio_tail_train(const long long* pool_sums, int pool_stride, int cell_pixels, const float* conv_w,
                          const float* conv_bias, const float* bn_gamma, const float* bn_beta, float eps, float momentum,
                          float* running_mean, float* running_var, const float* const* fc_w_host,
                          const float* const* fc_b_host, const float* drop0, const float* drop1, float out_min, float out_max,
                          float* raw_ws, float* gap_ws, float* ratio_out, int B, rgbd_stream_t stream);

/* Reference helper API on caller-supplied intermediates (the batched rgbd_depth_decompose never needs them):
 * rgbd_depth_select_modes  = DSAModule._select_depth_distribution_modes (CM:720-752): hist (B,512) int64 + bin_edges
 *   (B,513) fp32 -> up to num_modes peaks (scipy find_peaks with prominence >= threshold * max) ordered by (height, centre)
 *   descending: n_modes_out (B), peak_bins_out (B,3), centres_out (B,3).
 * rgbd_depth_region_codes  = DSAModule._generate_depth_region_masks (CM:774-798): gray (B,pixels) + windows (B,3,2) +
 *   n_windows (B) -> one code byte per pixel, bit t = lo_t <= g <= hi_t, bit n_windows = the remaining region. */
size_t rgbd_depth_helper_workspace_bytes(int B);
/* CustomMask2FormerPixelLevelModule.to_grayscale (CM:392-502), 3-channel float32 tensors: gray = (0.299 r + 0.587 g) + 0.114 b
 * per pixel; rgb3 (B,3,pixels) with element strides batch_stride / channel_stride -> gray_out (B,pixels). */
int rgbd_to_grayscale(const float* rgb3, long long batch_stride, long long channel_stride, float* gray_out, int B,
                      long long pixels, void* workspace, rgbd_stream_t stream);
int rgbd_depth_select_modes(const long long* hist, const float* edges, int B, int num_modes, double prominence_threshold,
                            int* n_modes_out, int* peak_bins_out, float* centres_out, void* workspace, rgbd_stream_t stream);
int rgbd_depth_region_codes(const float* gray, const float* windows, const int* n_windows, int B, long long pixels,
                            uint8_t* codes_out, void* workspace, rgbd_stream_t stream);

/* ---- resize half of the data mapper's front-end (map_10channel_case2, DL:405-414), bit-exact with the libraries the
 * reference calls.  rgbd_resize_pil_bilinear_u8: Pillow Image.resize((w,h), BILINEAR) for (B,H,W,C) uint8 images, C <= 4
 * (HF image processor, PIL backend, resample = 2): antialiased triangle filter, 22-bit fixed-point coefficients, horizontal
 * then vertical pass.  rgbd_resize_cv_linear_u8: cv2.resize(img, (w,h), interpolation=INTER_LINEAR) for (B,H,W) uint8
 * (the depth map the Sobel features are taken from): 11-bit fixed-point weights, OpenCV's border and rounding rules.
 * workspace: rgbd_resize_workspace_bytes(B,H,W,C,h,w) bytes (C = 1 for the OpenCV resize). */
size_t rgbd_resize_workspace_bytes(int B, int H, int W, int C, int h, int w);
int rgbd_resize_pil_bilinear_u8(const uint8_t* src, uint8_t* dst, int B, int H, int W, int C, int h, int w, void* workspace,
                                rgbd_stream_t stream);
int rgbd_resize_cv_linear_u8(const uint8_t* src, uint8_t* dst, int B, int H, int W, int h, int w, void* workspace,
                             rgbd_stream_t stream);

/* Feature-based window-ratio predictor of the version 0.1.3 / 0.3.0 models (`RatioPredictor.forward`, CM:860-898): global
 * average pool of n_levels NCHW fp32 depth-feature maps (B,C_l,HW_l), concatenation, MLP sum(C_l)->64->32->1 with ReLU,
 * ratio = out_min + (out_max - out_min) * sigmoid.  feats_host / C_host / HW_host / fc_*_host are HOST arrays (of device
 * pointers where they hold pointers); pooled_ws: B*sum(C_l) floats; ratio_out: B floats. */
int rgbd_ratio_from_features(int n_levels, const float* const* feats_host, const int* C_host, const int* HW_host, int B,
                             const float* const* fc_w_host, const float* const* fc_b_host, float out_min, float out_max,
                             float* pooled_ws, float* ratio_out, rgbd_stream_t stream);

/* ---- instance post-processing (SURVEY 8f-3): HuggingFace `post_process_instance_segmentation(outputs, threshold,
 * target_sizes, return_binary_maps=True)` as the reference calls it (mask2former/utils/model_essential_part.py:86-91,
 * mask2former/predictor.py:34-36, 701-703) for a batch of images that share one target size.
 * class_logits (B,Q,C1) fp32 (C1 = classes + "no object"), mask_logits (B,Q,h,w) fp32.  Per image the Q best (query,
 * label) candidates are taken in a DEFINED order (class score descending, flattened index ascending on ties; HF's
 * topk(sorted=False) order is unspecified), scored with the mean sigmoid of their 384x384-upsampled mask, kept when the
 * target-size mask is non-empty and score >= threshold, and written compactly in candidate order:
 * out_masks (B,Q,Ht,Wt) bytes 0/1 (first out_count[b] planes valid), out_labels / out_scores / out_query (B,Q),
 * out_count (B), out_segmentation (B,Ht,Wt) int32 or NULL: -1 background, else the id of the last kept segment covering
 * the pixel (HF paints in list order).  Ht = Wt = 384 reproduces target_sizes=None. */
size_t rgbd_postprocess_workspace_bytes(int B, int Q);
int rgbd_postprocess_instances(const float* class_logits, const float* mask_logits, int B, int Q, int C1, int h, int w,
                               int Ht, int Wt, float threshold, void* workspace, uint8_t* out_masks, int* out_labels,
                               float* out_scores, int* out_query, int* out_count, int* out_segmentation,
                               rgbd_stream_t stream);
/* Run-length encoding of int32 label maps, the `return_coco_annotation=True` output of the same HF routine
 * (`convert_segmentation_to_rle`): for every value present, in ascending order, its maximal runs in row-major order with
 * 1-based starts.  seg (B,H,W) int32 with labels in [-1, L); label index k = id + 1.  CSR output, no host synchronisation:
 * offsets (B, L+2): the runs of label k in image b are [offsets[b,k], offsets[b,k+1]) relative to base[b];
 * base (B+1): exclusive scan of the per-image run totals, so the used runs of the batch are runs[0, base[B]);
 * runs (B*H*W, 2): (start, end) of each run, 1-based and inclusive (length = end - start + 1);
 * bad_count (1): pixels whose label lies outside [-1, L); they belong to no run and the caller must check this count.
 * Deterministic: the output depends on the input alone.  L <= 4096, B <= 65535, B*H*W < 2^31.
 * workspace: rgbd_label_map_rle_workspace_bytes(B, H, W, L) bytes (0 for invalid arguments). */
size_t rgbd_label_map_rle_workspace_bytes(int B, int H, int W, int L);
int rgbd_label_map_rle(const int* seg, int B, int H, int W, int L, void* workspace, int* offsets, int* base, int* runs,
                       int* bad_count, rgbd_stream_t stream);
/* pycocotools RLE of every kept segment of a painted map: segment s of image b (s < count[b]) gets exactly the "counts"
 * string of `pycocotools.mask.encode(np.asfortranarray((seg[b] == s).astype(np.uint8)))`, size [H, W]: column-major
 * counts, alternating 0-runs and 1-runs and starting with 0-runs, compressed by `rleToString` (ASCII 48..111).
 * seg (B,H,W) int32 with ids in [-1, L), -1 = background; count (B) int32.  CSR output, no host synchronisation:
 * offsets (B, L+1): segment s's characters are chars[base[b] + offsets[b,s], base[b] + offsets[b,s+1]); segments
 * s >= count[b] are empty; base (B+1): exclusive scan of the per-image character totals;
 * chars (rgbd_instance_rle_capacity(B, H, W, L)) bytes; bad_count (1): pixels whose id lies outside [-1, L) or in
 * [count[b], L), plus 1 per image whose count lies outside [0, L] (that image gets no segments).  The caller must check it.
 * Deterministic: the output depends on the input alone.  L <= 4096, B <= 65535, 7*B*(2*H*W + L) < 2^31.
 * workspace: rgbd_instance_rle_workspace_bytes(B, H, W, L) bytes; both queries return 0 for invalid arguments. */
size_t rgbd_instance_rle_workspace_bytes(int B, int H, int W, int L);
size_t rgbd_instance_rle_capacity(int B, int H, int W, int L);
int rgbd_instance_rle(const int* seg, const int* count, int B, int H, int W, int L, void* workspace, int* offsets, int* base,
                      uint8_t* chars, int* bad_count, rgbd_stream_t stream);
/* Pairwise mask IoU, the core of the evaluator's segm mAP (mask2former/utils/model_essential_part.py:111-170 through
 * torchmetrics): pred (P,pixels) and gt (G,pixels) bytes 0/1 -> iou (P,G) fp32 (0 where the union is empty). */
int rgbd_mask_iou(const uint8_t* pred_masks, const uint8_t* gt_masks, int P, int G, long long pixels, float* iou,
                  rgbd_stream_t stream);

/* ---- neighbours of the path inside the STOCK Hugging Face modules: five opt-in inference kernels
 * (`decoder_ops.install_fast_decoder_ops`) for the pixel decoder / transformer decoder the reference hands the hot path's output
 * to (mask2former/utils/custom_model.py:383 `self.decoder(backbone_features)`, then Mask2FormerModel.forward ->
 * transformer_module) and for the Swin encoder that produces its input (CM:330).  Weights, module tree and state_dict stay
 * Hugging Face's.
 *
 * rgbd_msda_fwd: `multi_scale_deformable_attention(value, spatial_shapes, sampling_locations, attention_weights)` of
 * transformers' modeling_mask2former.py (grid_sample(bilinear, zeros, align_corners=False) per level, stack, weight, sum) in one
 * pass.  value (B,S,H,D) f32|bf16, S = sum of level_hw_host[l] = (h_l, w_l) products (HOST array, n_levels pairs);
 * out (B,Q,H*D) f32|bf16.  reference_points == NULL: `offsets` (B,Q,H,L,P,2) ARE the sampling locations in [0,1] and `attn`
 * (B,Q,H,L*P) the attention weights (softmax = 0) -- the function's own signature.  reference_points (B,Q,L,2) f32 given:
 * `offsets` are the raw sampling offsets (locations = reference + offsets / (w_l, h_l), the quotient rounded to bf16 when the
 * offsets are bf16, as torch does under autocast) and, with softmax = 1, `attn` holds logits softmaxed over L*P here.
 * D must be a multiple of 8. */
int rgbd_msda_fwd(const void* value, int value_dtype, const int* level_hw_host, int n_levels, const void* offsets,
                  int offsets_dtype, const float* reference_points, const void* attn, int attn_dtype, int softmax, void* out,
                  int out_dtype, int B, int S, int Q, int H, int D, int P, rgbd_stream_t stream);
/* rgbd_attention_mask: Mask2FormerMaskPredictor's masked-attention mask: mask_logits (B,Q,h,w) f32|bf16 ->
 * out (B*heads,Q,th*tw) bytes 0/1 = sigmoid(bilinear(mask_logits -> (th,tw), align_corners=False)) < 0.5, repeated per head. */
int rgbd_attention_mask(const void* mask_logits, int dtype, int B, int Q, int h, int w, int th, int tw, int heads, uint8_t* out,
                        rgbd_stream_t stream);
/* rgbd_window_attention: the inner op of transformers' SwinSelfAttention.forward (the stock backbone that produces the path's
 * input pyramid, CM:330): out = softmax(q k^T / sqrt(d) + bias[head] + mask[window % n_mask_windows]) v per (window, head).
 * q / k / v / out (n_windows, N, heads*d) f32|bf16 (the three nn.Linear outputs, untransposed); bias (heads, N, N) f32 =
 * relative_position_bias_table gathered by relative_position_index; mask (n_mask_windows, N, N) f32 (0 / -100 of the shifted
 * blocks) or NULL.  d must be 32, N <= 64.  workspace: rgbd_window_attention_workspace_bytes(N, heads, n_mask_windows) bytes (the
 * additive term bias + mask as one padded table, built by the first of the two launches).  Inference only. */
size_t rgbd_window_attention_workspace_bytes(int N, int heads, int n_mask_windows);
int rgbd_window_attention(const void* q, const void* k, const void* v, int dtype, const float* bias, const float* mask, void* out,
                          long long n_windows, int N, int heads, int head_dim, int n_mask_windows, void* workspace,
                          rgbd_stream_t stream);
/* rgbd_layer_norm: LayerNorm over the last dimension, x (rows, C) f32|bf16 -> out (rows, C) f32|bf16, float32 arithmetic
 * (mean, biased variance, rsqrt(var + eps), * gamma + beta).  C % 4 == 0, C <= 1024.  With out_dtype = bf16 it emits exactly what
 * the nn.Linear consumers of a pre-norm LayerNorm cast its float32 result to under bf16 autocast (SwinLayer.layernorm_before /
 * layernorm_after).  Inference only. */
int rgbd_layer_norm(const void* x, int x_dtype, const float* gamma, const float* beta, void* out, int out_dtype, long long rows,
                    int C, float eps, rgbd_stream_t stream);
/* rgbd_masked_cross_attention: the attention core of nn.MultiheadAttention.forward as transformers'
 * Mask2FormerMaskedAttentionDecoderLayer calls it (batch_first = False, boolean attn_mask): q (L, B, heads*d), k / v (S, B, heads*d)
 * bf16 = the three input projections, mask (B*heads, L, S) bytes (non-zero = may NOT attend), out (L, B, heads*d) bf16 =
 * softmax(q k^T / sqrt(d), masked) v per (image, head); rows whose keys are all masked give zeros.  d must be 32, S even.
 * Inference only. */
int rgbd_masked_cross_attention(const void* q_bf16, const void* k_bf16, const void* v_bf16, const uint8_t* mask, void* out_bf16, int B,
                                int heads, int L, int S, int head_dim, rgbd_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* RGBD_B200_H */
