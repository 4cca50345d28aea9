/*
 * rdvc_corr.h -- C ABI of librdvc_corr.so: the B200 (sm_100a) implementation of
 * the RAFT correlation hot path of RDVC's motion branch.
 *
 * Drop-in boundary.  RDVC (R: = the reference repo) has no correlation code of
 * its own; its encoder calls torchvision's RAFT (R:codec_processing.py:1442,
 * R:test_2frames.py:496), whose CorrBlock (TV: = torchvision 0.26.0
 * models/optical_flow/raft.py) is the path replaced here:
 *
 *   rdvc_corr_build   replaces  CorrBlock.build_pyramid      TV:raft.py:360-392
 *                               (+ _compute_corr_volume      TV:raft.py:424-431)
 *   rdvc_corr_lookup  replaces  CorrBlock.index_pyramid      TV:raft.py:394-422
 *                               (+ grid_sample helper        TV:_utils.py:8-19)
 *   rdvc_corr_pair_host         one frame pair end to end from HOST buffers
 *                               (build + `iters` lookups, copies included);
 *                               the call a non-PyTorch host would bind.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, no C++/torch types.
 *   - All DEVICE buffers are allocated and owned by the caller.  The library
 *     never allocates or frees caller-visible device memory and keeps no
 *     pointer after a call returns (rdvc_corr_pair_host uses a private,
 *     per-thread scratch arena that it owns and that rdvc_corr_release frees).
 *   - Calls are asynchronous on `stream` (a cudaStream_t passed as void*; NULL
 *     = the legacy default stream) except rdvc_corr_pair_host, which
 *     synchronises before returning.  The caller sets the current device.
 *   - Return 0 on success, a negative RDVC_E_* for argument errors, a positive
 *     cudaError_t for CUDA failures.  rdvc_corr_last_error() returns a
 *     thread-local message for the last non-zero return on this thread.
 *   - No CPU fallback exists: on a machine without an sm_100 GPU every compute
 *     entry point fails with a CUDA error.
 *
 * Pyramid layout (one caller-owned buffer, `rdvc_corr_pyramid_bytes` long):
 *   level l lives at byte offset rdvc_corr_level_offset_bytes(..., l) (256-byte
 *   aligned); h_l = h >> l, w_l = w >> l (floor halving, TV:raft.py:390-392).
 *   RDVC_LAYOUT_ROWMAJOR: dense [B*h*w][h_l][w_l] -- the element order of
 *     torchvision's corr_pyramid[l] viewed (B*h*w, 1, h_l, w_l).
 *   RDVC_LAYOUT_TILED (default of the Python mirror): each level image is padded to
 *     whole tiles of tile_w x tile_h pixels (rdvc_corr_tile_shape: 16-byte rows x 4 rows =
 *     one 64-byte DRAM atom; 4 x 4 for fp32, 8 x 4 for bf16) and stored tile by tile,
 *     [B*h*w][ceil(h_l/tile_h)][ceil(w_l/tile_w)][tile_h][tile_w], each image rounded up to a
 *     multiple of 256 bytes (rdvc_corr_level_image_elems); padding holds 0.
 *     The (2r+2)^2 footprint of a lookup then touches ~11 DRAM atoms per level instead of
 *     ~20 (row-major: 10 rows x 40 bytes, each straddling 64-byte atoms): the gather is
 *     DRAM-bound, so bytes fetched are what the layout is chosen for.  The build writes
 *     either layout at the same cost (an image row of the volume is a permutation of the
 *     GEMM's output columns, applied for free when fmap2 is packed).
 */
#ifndef RDVC_CORR_H_
#define RDVC_CORR_H_

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RDVC_CORR_VERSION 103 /* 0.1.3 */

/* element types */
#define RDVC_DT_BF16 0
#define RDVC_DT_F32 1
#define RDVC_DT_F16 2

/* pyramid layouts (see "Pyramid layout" above) */
#define RDVC_LAYOUT_ROWMAJOR 0
#define RDVC_LAYOUT_TILED 1

/* forms of the lookup result (rdvc_corr_lookup_ex) */
#define RDVC_OUT_NCHW 0   /* (B, L*S*S, h, w): what torchvision's index_pyramid returns                      */
#define RDVC_OUT_KMAJOR 1 /* [B*h*w][rdvc_corr_feat_pitch] 16-bit rows: the A operand of rdvc_conv1x1        */

/* activations of rdvc_conv1x1 */
#define RDVC_ACT_NONE 0
#define RDVC_ACT_RELU 1

/* argument errors (negative); CUDA errors are returned as positive cudaError_t */
#define RDVC_OK 0
#define RDVC_E_NULL (-1)        /* a required pointer is NULL                        */
#define RDVC_E_SHAPE (-2)       /* non-positive dimension                            */
#define RDVC_E_TOO_SMALL (-3)   /* h or w < 2 * 2^(num_levels-1)   (TV:raft.py:376)  */
#define RDVC_E_DTYPE (-4)       /* unsupported in_dtype / vol_dtype                  */
#define RDVC_E_UNSUPPORTED (-5) /* D % 64 != 0, D > 256, num_levels > 4, radius > 4, layout */
#define RDVC_E_WORKSPACE (-6)   /* workspace smaller than rdvc_corr_workspace_bytes  */
#define RDVC_E_ALIGN (-7)       /* a device pointer is not 16-byte aligned           */
#define RDVC_E_DRIVER (-8)      /* cuTensorMapEncodeTiled unavailable / failed       */

int rdvc_corr_version(void);
const char* rdvc_corr_last_error(void);
/* "RDVC_SRC_HASH=<sha256 of csrc/ + include/> version=<n> experiments=<0|1>": which sources this binary was built
 * from (the Python loader refuses a library whose hash differs from the tree's) and whether the experiment knobs
 * are compiled in (the product build: 0).                                                                       */
const char* rdvc_corr_build_info(void);

/* ---- sizes ------------------------------------------------------------- */
/* vol_dtype: RDVC_DT_F32 or RDVC_DT_BF16 (storage type of the pyramid). */
size_t rdvc_corr_pyramid_bytes(int B, int h, int w, int num_levels, int vol_dtype, int layout);
size_t rdvc_corr_level_offset_bytes(int B, int h, int w, int level, int vol_dtype, int layout);
/* elements one level image (one query pixel's h_l x w_l map) occupies, padding included:
 * h_l * w_l for ROWMAJOR; whole tiles, rounded up to a multiple of 256 bytes, for TILED */
size_t rdvc_corr_level_image_elems(int h, int w, int level, int vol_dtype, int layout);
/* tile shape (pixels) of RDVC_LAYOUT_TILED for a volume dtype */
int rdvc_corr_tile_shape(int vol_dtype, int* tile_w, int* tile_h);
/* scratch for the K-major bf16 copies of fmap1 and of fmap2 at every pyramid level */
size_t rdvc_corr_workspace_bytes(int B, int D, int h, int w);

/* ---- build: correlation volume + all pyramid levels, written once ------ *
 * fmap1, fmap2 : device, (B, D, h, w) contiguous, in_dtype in {F32, BF16, F16}
 * pyramid      : device, rdvc_corr_pyramid_bytes(...) bytes, 256-byte aligned
 * workspace    : device, rdvc_corr_workspace_bytes(...) bytes, 256-byte aligned
 * Computes  pyr[0][b*N+i][y][x] = sum_c fmap1[b,c,i] * fmap2[b,c,y*w+x] / sqrt(D)
 * with bf16 operands (fp16 operands when in_dtype is F16: nothing of an fp16 input is lost) and fp32
 * accumulation (tcgen05), and pyr[l+1] = 2x2 mean of
 * pyr[l] over (y,x) with the odd trailing row/column dropped.                        */
int rdvc_corr_build(const void* fmap1, const void* fmap2, int B, int D, int h, int w,
                    int in_dtype, void* pyramid, int vol_dtype, int layout, int num_levels,
                    void* workspace, size_t workspace_bytes, void* stream);

/* ---- lookup: (2r+1)^2 bilinear taps x num_levels ----------------------- *
 * coords : device, (B, 2, h, w) fp32, channel 0 = x, channel 1 = y, absolute
 *          pixel units of the 1/8 grid (TV:_utils.py:22-26)
 * out    : device, (B, num_levels*(2r+1)^2, h, w) fp32 contiguous
 * out[b, l*S*S + i*S + j, y, x] = bilinear(pyr[l][b*N + y*w + x],
 *          xs = coords[b,0,y,x]/2^l + (i-r), ys = coords[b,1,y,x]/2^l + (j-r)),
 * zero outside the level, pixel centres at integers (align_corners=True).     */
int rdvc_corr_lookup(const void* pyramid, int vol_dtype, int layout, const float* coords, int B,
                     int h, int w, int num_levels, int radius, float* out, void* stream);

/* The same lookup with a choice of result type and form (TILED pyramids; ROWMAJOR supports F32 / NCHW only):
 *   out_form RDVC_OUT_NCHW,   out_dtype F32 | F16 : (B, L*S*S, h, w); F16 is what the consumer casts the features to
 *                                                   under the reference's default autocast (R:codec_processing.py:1436)
 *   out_form RDVC_OUT_KMAJOR, out_dtype BF16 | F16: the K-major A operand of rdvc_conv1x1, rdvc_corr_feat_bytes long,
 *            16-byte aligned.  Feature k = l*PL + j*S + i of query pixel m holds torchvision channel l*S*S + i*S + j
 *            (PL = S*S rounded up to 8; padding features hold 0) and lives at element
 *            ((k / 8) * rdvc_corr_feat_rows + m) * 8 + k % 8 -- chunk-major [K/8][rows][8]: a warp of 32 consecutive
 *            pixels stores 8 taps of all of them as one contiguous 512-byte run, and a TMA box of it is the
 *            un-swizzled tcgen05 core-matrix layout.  Rows m >= B*h*w (up to the multiple of 8) are not written.  */
int rdvc_corr_lookup_ex(const void* pyramid, int vol_dtype, int layout, const float* coords, int B, int h,
                        int w, int num_levels, int radius, void* out, int out_dtype, int out_form, void* stream);
/* K elements per query pixel: num_levels * PL rounded up to 16 (352 for 4 levels x radius 4); 0 if unsupported */
size_t rdvc_corr_feat_pitch(int num_levels, int radius);
/* rows of every chunk plane: B*h*w rounded up to 8; and the byte size of the whole K-major feature buffer */
size_t rdvc_corr_feat_rows(int B, int h, int w);
size_t rdvc_corr_feat_bytes(int B, int h, int w, int num_levels, int radius);

/* ---- next row f-1: lookup fused with MotionEncoder.convcorr1 ------------- *
 * Replaces index_pyramid (TV:raft.py:394-422) + convcorr1 = Conv2d(L*S*S -> cout, kernel 1) + ReLU (TV:raft.py:185
 * construction, :202 call): the (B, 324, h, w) fp32 lookup tensor (42 MB per iteration at 1080p) is never written;
 * the lookup emits 16-bit K-major feature rows (23 MB, L2-resident) and a tcgen05 GEMM with the bias + ReLU epilogue
 * writes the (B, cout, h, w) tensor convcorr2 reads.  16-bit operands, fp32 accumulation.
 *
 * rdvc_conv1x1_pack_weights (HOST, no GPU needed): conv weight (cout, L*S*S) fp32 in torchvision's channel order ->
 *   [cout][K padded to 64] 16-bit rows in the lookup's column order, zero padded; copy them to the device.
 *   cout: multiple of 32, <= 256.  feat_dtype: BF16 or F16 (must match the lookup's).
 * rdvc_conv1x1: out[b, n, y, x] = act(sum_k feat(k, b*h*w + y*w + x) * Wp[n][k] + bias[n]);  feat: the K-major buffer
 *   described at rdvc_corr_lookup_ex; bias: cout DEVICE floats or NULL; out: (B, cout, h, w) F32 | F16 | BF16.
 * rdvc_corr_lookup_conv1x1: both steps (2 launches); feat_ws: DEVICE scratch of rdvc_corr_feat_bytes(...) bytes.     */
size_t rdvc_conv1x1_packed_weight_bytes(int cout, int num_levels, int radius);
int rdvc_conv1x1_pack_weights(const float* weight, int cout, int num_levels, int radius, int feat_dtype,
                              void* packed_host);
int rdvc_conv1x1(const void* feat, int feat_dtype, const void* packed_w, const float* bias, int B, int h, int w,
                 int num_levels, int radius, int cout, int act, void* out, int out_dtype, void* stream);
int rdvc_corr_lookup_conv1x1(const void* pyramid, int vol_dtype, int layout, const float* coords, int B, int h,
                             int w, int num_levels, int radius, const void* packed_w, const float* bias, int cout,
                             int act, int feat_dtype, void* feat_ws, size_t feat_ws_bytes, void* out, int out_dtype,
                             void* stream);
/* The _ex forms take out_pixel_stride: 0 = the (B, cout, h, w) output above; > 0 = NHWC, pixel m = b*h*w + y*w + x at
 * out + m * out_pixel_stride, channel stride 1, out_dtype F16 | BF16, out 16-byte aligned, out_pixel_stride >= cout and
 * a multiple of 8 (e.g. 256 for a channel slice of a 256-channel channels_last tensor).  Bit-identical values. */
int rdvc_conv1x1_ex(const void* feat, int feat_dtype, const void* packed_w, const float* bias, int B, int h, int w,
                    int num_levels, int radius, int cout, int act, void* out, int out_dtype, long long out_pixel_stride,
                    void* stream);
int rdvc_corr_lookup_conv1x1_ex(const void* pyramid, int vol_dtype, int layout, const float* coords, int B, int h,
                                int w, int num_levels, int radius, const void* packed_w, const float* bias, int cout,
                                int act, int feat_dtype, void* feat_ws, size_t feat_ws_bytes, void* out, int out_dtype,
                                long long out_pixel_stride, void* stream);

/* ---- next row f-2 (last sub-item): the feature encoder's final 1x1 convolution, fused into the operand repack ---- *
 * torchvision's FeatureEncoder ends in conv = Conv2d(128, 256, kernel_size=1) (TV:raft.py:139, called at :150); the
 * stock path writes its (2B, 256, h, w) fp32 result (67 MB at 1080p) and rdvc_corr_build re-reads it to repack.  A
 * 1x1 convolution commutes with the transpose and (being linear, bias included) with the pyramid's mean pooling, so:
 *   rdvc_corr_pack          the repack step of rdvc_corr_build ALONE, on any (B, D, h, w) maps with D % 64 == 0,
 *                           D <= 256: K-major 16-bit rows of x1 and of x2 at every pyramid level (pyramid row order,
 *                           padding rows zero) into a workspace of rdvc_corr_workspace_bytes(B, D, h, w);
 *   rdvc_corr_encoder_tail  every packed 128-channel row -> the 256-channel operand row of the build:
 *                           out[r][n] = round16(sum_k in[r][k] W[n][k] + bias[n]), layout-padding rows stay 0
 *                           (tcgen05 GEMM, fp32 accumulation; ws_out = a workspace for D = 256);
 *   rdvc_corr_build_packed  the GEMM step of rdvc_corr_build ALONE, on a workspace that already holds the rows.
 * Together: pyramid = build(conv(x1), conv(x2)) without the fp32 feature maps ever existing.  packed_w: the weight
 * (256, 128) as 16-bit rows (rdvc_linear_pack_weights, HOST) on the device; bias: 256 DEVICE floats or NULL;
 * op_dtype: BF16, or F16 when the activations are fp16 (the pack keeps fp16 inputs as fp16).                        */
int rdvc_corr_pack(const void* x1, const void* x2, int B, int D, int h, int w, int in_dtype, int vol_dtype,
                   int layout, int num_levels, void* workspace, size_t workspace_bytes, void* stream);
/* rdvc_corr_pack on NHWC maps: pixel (b, y, x) of x1 / x2 at x + ((b * h + y) * w + x) * pixel_stride, channel stride 1
 * (e.g. rdvc_corr_feature_encoder's RDVC_FE_OUT_TRUNK output, read in place; the two maps may be rows of one buffer).
 * in_dtype F16 | BF16; bases 16-byte aligned; pixel_stride >= D, a multiple of 8.  Writes the same bytes as
 * rdvc_corr_pack on the same values.                                                                                */
int rdvc_corr_pack_nhwc(const void* x1, const void* x2, long long pixel_stride, int B, int D, int h, int w, int in_dtype,
                        int vol_dtype, int layout, int num_levels, void* workspace, size_t workspace_bytes, void* stream);
size_t rdvc_linear_packed_weight_bytes(int cout, int cin);
int rdvc_linear_pack_weights(const float* weight, int cout, int cin, int dtype, void* packed_host);
int rdvc_corr_encoder_tail(const void* ws_in, size_t ws_in_bytes, int D_in, const void* packed_w, const float* bias,
                           int D_out, int B, int h, int w, int op_dtype, int vol_dtype, int layout, int num_levels,
                           void* ws_out, size_t ws_out_bytes, void* stream);
int rdvc_corr_build_packed(int B, int D, int h, int w, int op_dtype, void* pyramid, int vol_dtype, int layout,
                           int num_levels, void* workspace, size_t workspace_bytes, void* stream);

/* ---- one frame pair from host memory (blocking) ------------------------ *
 * fmap1_host, fmap2_host : host fp32 (B, D, h, w)
 * coords_host            : host fp32 (iters, B, 2, h, w)
 * out_host               : host fp32 (iters, B, L*S*S, h, w)
 * Copies in, builds, runs `iters` lookups, copies every lookup result out and
 * synchronises.  Pinned host buffers make the copies asynchronous.            */
int rdvc_corr_pair_host(const float* fmap1_host, const float* fmap2_host,
                        const float* coords_host, float* out_host, int B, int D, int h,
                        int w, int num_levels, int radius, int iters, int vol_dtype);

/* ---- next row: flow resize + warp, fused (after RAFT, before the MCN) ---- *
 * Replaces resize_flow (R:codec_processing.py:772-818, called at :1446) and WarpingLayer.forward
 * (R:codec_processing.py:322-367, called at :1456) with one launch.
 * flow     : device, (B, 2, h_in, w_in) fp32 -- RAFT's flow, channel 0 = dx, channel 1 = dy
 * prev     : device, (B, C, H, W) fp32 previous frame, or NULL for a resize only
 * warped   : device, (B, C, H, W) fp32, NULL iff prev is NULL
 * flow_out : device, (B, 2, H, W) fp32 resized + rescaled flow, or NULL to skip materialising it
 * flow_out = bilinear_resize(flow, align_corners=False) * (W/w_in, H/h_in) (the input itself when the
 * sizes match); warped[b,c,i,j] = bilinear(prev[b,c]; i + dy, j + dx) with the sample point clamped
 * to the frame (border padding), pixel centres at integers (align_corners=True).                  */
int rdvc_motion_warp(const float* prev, const float* flow, int B, int C, int H, int W, int h_in,
                     int w_in, float* warped, float* flow_out, void* stream);

/* The same call split in two, for a host that has the next pair ready while the previous result is still
 * crossing PCIe: _submit enqueues everything for one pair on private streams of `slot` (0 or 1) and returns;
 * _wait blocks until that slot's output has landed in out_host.  Two slots overlap one pair's device->host
 * copies (the bottleneck: 508 MB per 1080p pair) with the next pair's host->device copies and kernels.  The
 * host buffers of a slot must stay valid and untouched until its _wait returns.                             */
int rdvc_corr_pair_host_submit(const float* fmap1_host, const float* fmap2_host,
                               const float* coords_host, float* out_host, int B, int D, int h,
                               int w, int num_levels, int radius, int iters, int vol_dtype, int slot);
int rdvc_corr_pair_host_wait(int slot);
/* _submit with a choice of result type: out_dtype F32, or F16 (out_host then holds __half: half the bytes over PCIe;
 * the reference's default consumer runs under autocast and casts the features to fp16 anyway).                   */
int rdvc_corr_pair_host_submit_ex(const float* fmap1_host, const float* fmap2_host,
                                  const float* coords_host, void* out_host, int B, int D, int h,
                                  int w, int num_levels, int radius, int iters, int vol_dtype,
                                  int out_dtype, int slot);

/* ---- next row: frame preparation in front of RAFT / the codec ---------- *
 * Replaces preprocess_frame_raft (R:codec_processing.py:751-761: TF.to_tensor + TF.resize(antialias=True),
 * run on the CPU at :1430-1431) and preprocess_frame_codec (:763-769, to_tensor only: h_out = H, w_out = W).
 * frame_hwc : device, (H, W, C) uint8, C in [1, 4]
 * out       : device, (C, h_out, w_out) fp32 in [0, 1]: bilinear resize with aten's anti-aliasing filter
 *             (_upsample_bilinear2d_aa, align_corners=False) of frame / 255; down-scaling up to 7x.        */
int rdvc_preprocess_frame(const unsigned char* frame_hwc, int H, int W, int C, float* out, int h_out,
                          int w_out, void* stream);

/* ---- next row f-4 (cont.): the motion-compensation network --------------- *
 * Replaces MotionCompensationNetwork.forward (R:codec_processing.py:369-406, called per P-frame at :1458, built
 * from ConvNormAct :117-156 and ResidualBlock :190-217) in inference mode:
 *   refined = warped_ref * sigmoid(conv5x5(resblocks(lrelu(bn(conv5x5(cat(warped_ref, flow, ref_frame)))))))
 * Every convolution is a tcgen05 implicit GEMM over fp16 activations with fp32 accumulation (csrc/mcn_conv_sm100.cuh).
 * The host folds each BatchNorm into its convolution (w' = w * gamma / sqrt(var + eps), bias' = beta - mean * gamma /
 * sqrt(var + eps)) and packs the folded weights once with rdvc_mcn_pack_weights.
 *
 * Activation layout ("plane", rdvc_mcn_plane_bytes): [B][H][ceil(W/2)][2 pixels][32 channels] fp16 -- NHWC with 32
 * channels, rows padded to an even pixel count (the padding pixel holds 0).                                      */
#define RDVC_MCN_ACT_NONE 0
#define RDVC_MCN_ACT_LEAKY 1 /* LeakyReLU(0.2), R:codec_processing.py:110 */
#define RDVC_MCN_REVERSE_ORDER 0x100 /* OR into `act`: walk the tiles last-to-first (same result; lets a layer start on
                                        the part of its input the previous launch wrote last, which is still in L2) */
size_t rdvc_mcn_plane_bytes(int B, int H, int W);
size_t rdvc_mcn_workspace_bytes(int B, int H, int W); /* three planes */
/* HOST function (no GPU needed): conv weight (cout, cin, k, k) fp32, k in {3, 5}, cin <= 32, cout == 32 or <= 8 ->
 * the per-tap fp16 matrices the kernel multiplies by (rdvc_mcn_packed_weight_bytes long; copy them to the device)
 * and the mask of non-zero k-steps.                                                                              */
size_t rdvc_mcn_packed_weight_bytes(int ksize, int cout);
int rdvc_mcn_pack_weights(const float* weight, int cout, int cin, int ksize, void* packed_host,
                          unsigned long long* kmask);
/* cat(warped_ref, flow, ref_frame) (R:codec_processing.py:402), each (B, c_*, H, W) fp32 on the device -> plane. */
int rdvc_mcn_pack_input(const float* warped, const float* flow, const float* ref, int B, int c_warped,
                        int c_flow, int c_ref, int H, int W, void* act, void* stream);
/* One 32 -> 32 layer: act_out = act(conv_k(act_in) + bias [+ residual]).  bias: 32 HOST floats (or NULL = 0), copied
 * at call time.  residual: optional plane added before the activation (ResidualBlock, :212-216).  Not in place.   */
int rdvc_mcn_conv(const void* act_in, const void* packed_weights, unsigned long long kmask,
                  const float* bias, int ksize, int act, const void* residual, void* act_out, int B,
                  int H, int W, void* stream);
/* The output layer fused with the refinement (:403-404): out = warped * sigmoid(conv5x5(act_in) + bias), (B, cout, H, W)
 * fp32, cout <= 8; bias: cout HOST floats.                                                                        */
int rdvc_mcn_conv_out(const void* act_in, const void* packed_weights, unsigned long long kmask,
                      const float* bias, int ksize, int cout, const float* warped, float* out, int B,
                      int H, int W, void* stream);
/* The whole network: 1 + (2 + 2 * num_res_blocks) launches.  packed_weights: HOST array of 2 + 2 * num_res_blocks
 * DEVICE pointers in layer order; kmasks: HOST array, one per layer; biases: HOST, 32 floats per layer.
 * warped / ref: (B, 3, H, W); flow: (B, 2, H, W); out: (B, 3, H, W), all fp32 on the device.                      */
int rdvc_mcn_forward(const float* warped, const float* flow, const float* ref, int B, int H, int W,
                     int num_res_blocks, const void* const* packed_weights,
                     const unsigned long long* kmasks, const float* biases, void* workspace,
                     size_t workspace_bytes, float* out, void* stream);

/* ---- RAFT's recurrent block: the SepConvGRU of every refinement iteration ---------------------------------- *
 * rdvc_corr_convgru replaces ONE ConvGRU.forward (TV:raft.py:223-229) of torchvision's RecurrentBlock (TV:raft.py:238-270;
 * raft_large: hidden size 128, input 256 = [context | motion features], kernels (1, 5) then (5, 1)):
 *   z = sigmoid(convz([h | x])), r = sigmoid(convr([h | x])), q = tanh(convq([r * h | x])), out = (1 - z) h + z q
 * as two tcgen05 implicit GEMMs (csrc/tap_conv_sm100.cuh): 16-bit operands (op_dtype), fp32 accumulation, fp32
 * epilogue; z and r * h pass through the workspace in op_dtype; the blend uses h as given (act_dtype).
 *
 * rdvc_corr_convgru_pack_weights (HOST, no GPU needed): convz / convr / convq weights, each (128, 384, 1, 5) or
 *   (128, 384, 5, 1) contiguous fp32 (both are w[co][ci][tap]) -> rdvc_corr_convgru_packed_weight_bytes() bytes of 16-bit
 *   tap matrices: z|r [k-block 0..5][tap 0..4][256: convz rows, then convr rows][64 channels], then q
 *   [k-block][tap][128][64]; input channel = 64 * k-block + column, tap t multiplies the pixel at offset t - 2 along
 *   the tap axis.  Copy them to the device (16-byte aligned).
 * rdvc_corr_convgru: h, context, motion: DEVICE, NHWC (B, H, W, >= 128), act_dtype F32 | F16 | BF16, channel stride 1 and
 *   the given pixel strides in ELEMENTS (a multiple of 16 bytes; e.g. 256 for a channel slice of a 256-channel
 *   channels_last tensor); base pointers 16-byte aligned.  op_dtype F16 | BF16; 16-bit activations must be op_dtype
 *   (read in place), fp32 activations are rounded into the workspace first.  axis: the tap axis of the pass.
 *   bias_z / bias_r / bias_q: 128 DEVICE floats each.  workspace: DEVICE, rdvc_corr_convgru_workspace_bytes(...), 256-byte
 *   aligned.  out: DEVICE, (B, H, W, 128) contiguous act_dtype, not one of the inputs.  2 launches (3 for F32).      */
#define RDVC_GRU_HORIZONTAL 0 /* 1 x 5 kernel, padding (0, 2): convgru1 */
#define RDVC_GRU_VERTICAL 1   /* 5 x 1 kernel, padding (2, 0): convgru2 */
size_t rdvc_corr_convgru_packed_weight_bytes(void);
int rdvc_corr_convgru_pack_weights(const float* wz, const float* wr, const float* wq, int op_dtype, void* packed_host);
size_t rdvc_corr_convgru_workspace_bytes(int B, int H, int W, int act_dtype);
int rdvc_corr_convgru(const void* h, long long h_pixel_stride, const void* context, long long context_pixel_stride,
                 const void* motion, long long motion_pixel_stride, int act_dtype, int op_dtype, int axis, int B, int H,
                 int W, const void* packed_w, const float* bias_z, const float* bias_r, const float* bias_q,
                 void* workspace, size_t workspace_bytes, void* out, void* stream);

/* ---- RAFT's motion encoder and flow head: the rest of the update block ------------------------------------- *
 * raft_large's MotionEncoder (TV:raft.py:171-211) after convcorr1 and its FlowHead (TV:raft.py:272-285) as convolutions
 * over NHWC 16-bit activations (csrc/tap_conv_sm100.cuh): the 3x3 layers are tcgen05 implicit GEMMs, convflow1 (7x7,
 * 2 -> 128) a CUDA-core direct convolution.  16-bit operands (op_dtype), fp32 accumulation, bias (+ ReLU) in fp32.
 *
 * Layers (RDVC_UC_*), torchvision weight (cout, cin, k, k) contiguous fp32:
 *   CONVCORR2  3x3 256 -> 192 + ReLU     TV:raft.py:186, 203     CONVFLOW1  7x7 2 -> 128 + ReLU   TV:raft.py:188, 205
 *   CONVFLOW2  3x3 128 -> 64 + ReLU      TV:raft.py:189, 205     CONV       3x3 256 -> 126 + ReLU TV:raft.py:192, 208
 *   FH_CONV1   3x3 128 -> 256 + ReLU     TV:raft.py:276, 285     FH_CONV2   3x3 256 -> 2          TV:raft.py:277, 285
 * rdvc_corr_update_conv_pack_weights (HOST, no GPU needed) -> rdvc_corr_update_conv_packed_weight_bytes(layer) bytes of 16-bit
 *   GEMM operand: 3x3 layers [cin / 64][dy * 3 + dx][N][64] (N = cout rounded up to 16: 192, 64, 128, 256, 16; padded
 *   rows zero); CONVFLOW1 [128][128], column (ky * 7 + kx) * 2 + ci (K = 98, padded columns zero).  Copy to the device.
 * rdvc_corr_update_conv: one layer.  in: DEVICE NHWC op_dtype, pixel stride in_pixel_stride elements (>= cin, a multiple of 8;
 *   unused by CONVFLOW1).  flow (CONVFLOW1's input; CONV writes it into output channels 126-127): DEVICE fp32 at
 *   flow[b * s[0] + c * s[1] + y * s[2] + x * s[3]], s = flow_strides (4 HOST long longs, elements).  bias: cout DEVICE
 *   floats.  out: NHWC at out_pixel_stride elements (>= N, a multiple of 16 bytes), op_dtype -- except CONV (F32 or
 *   op_dtype, the activation dtype) and FH_CONV2, which writes (B, 2, H, W) contiguous planes (F32 or op_dtype) and
 *   ignores out_pixel_stride.  Channel slices of a channels_last tensor are read and written in place; nothing outside
 *   [0, N) of each output pixel is written.
 * rdvc_corr_motion_encoder: MotionEncoder.forward (TV:raft.py:200-211) from convcorr1's NHWC output c1 (op_dtype, 256
 *   channels): 4 launches, out = the (B, H, W, 128) motion features [conv | flow] at out_pixel_stride, out_dtype F32 or
 *   op_dtype.  packed_w / bias: 4 DEVICE pointers each, in the order CONVCORR2, CONVFLOW1, CONVFLOW2, CONV.  workspace:
 *   DEVICE, rdvc_corr_motion_encoder_workspace_bytes(...), 256-byte aligned.
 * rdvc_corr_flow_head: FlowHead.forward (TV:raft.py:284-285) on h (NHWC act_dtype, >= 128 channels at h_pixel_stride): out =
 *   (B, 2, H, W) act_dtype.  16-bit act_dtype must be op_dtype; fp32 h is rounded into the workspace first (3 launches,
 *   else 2).  packed_w / bias: FH_CONV1, FH_CONV2.  workspace: rdvc_corr_flow_head_workspace_bytes(...), 256-byte aligned. */
#define RDVC_UC_CONVCORR2 0
#define RDVC_UC_CONVFLOW1 1
#define RDVC_UC_CONVFLOW2 2
#define RDVC_UC_CONV 3
#define RDVC_UC_FH_CONV1 4
#define RDVC_UC_FH_CONV2 5
size_t rdvc_corr_update_conv_packed_weight_bytes(int layer);
int rdvc_corr_update_conv_pack_weights(int layer, const float* weight, int op_dtype, void* packed_host);
int rdvc_corr_update_conv(int layer, const void* in, long long in_pixel_stride, const float* flow, const long long* flow_strides,
                     int B, int H, int W, int op_dtype, const void* packed_w, const float* bias, void* out,
                     long long out_pixel_stride, int out_dtype, void* stream);
size_t rdvc_corr_motion_encoder_workspace_bytes(int B, int H, int W);
int rdvc_corr_motion_encoder(const void* c1, long long c1_pixel_stride, const float* flow, const long long* flow_strides, int B,
                        int H, int W, int op_dtype, const void* const* packed_w, const float* const* bias, void* workspace,
                        size_t workspace_bytes, void* out, long long out_pixel_stride, int out_dtype, void* stream);
size_t rdvc_corr_flow_head_workspace_bytes(int B, int H, int W, int act_dtype);
int rdvc_corr_flow_head(const void* h, long long h_pixel_stride, int act_dtype, int B, int H, int W, int op_dtype,
                   const void* const* packed_w, const float* const* bias, void* workspace, size_t workspace_bytes, void* out,
                   void* stream);

/* ---- RAFT's mask predictor and the convex 8x upsampling ----------------------------------------------------- *
 * raft_large's MaskPredictor (TV:raft.py:311-334: convrelu = 3x3 128 -> 256 + ReLU, conv = 1x1 256 -> 576, x multiplier)
 * followed by torchvision's upsample_flow with a mask (TV:_utils.py:29-48): per output pixel (8y + i, 8x + j) a softmax
 * over the 9 mask channels k * 64 + i * 8 + j (k = ky * 3 + kx), then the convex combination of 8 * flow at
 * (y + ky - 1, x + kx - 1), neighbours outside the image zero (F.unfold, padding 1).  convrelu runs as FH_CONV1's
 * kernel; the 1x1 is a tcgen05 GEMM (csrc/mask_upsample_sm100.cuh) whose epilogue does the softmax, the combination and
 * the pixel shuffle, so the 576-channel mask never reaches memory.  16-bit operands, fp32 accumulation and epilogue.
 *
 * rdvc_corr_mask_conv_pack_weights (HOST, no GPU needed): conv's weight (576, 256) and bias (576), contiguous fp32 ->
 *   rdvc_corr_mask_conv_packed_weight_bytes() bytes of 16-bit GEMM operand, packed [c][k-block][144][64], and bias_host
 *   (576 floats), both in GEMM row order: row n = c * 144 + k * 16 + s holds stock channel k * 64 + 16 c + s (c = 0..3,
 *   k = 0..8, s = 0..15).  Copy both to the device.  convrelu is packed with
 *   rdvc_corr_update_conv_pack_weights(RDVC_UC_FH_CONV1, ...).
 * rdvc_corr_mask_predictor: h: DEVICE NHWC act_dtype (F32 | F16 | BF16; 16-bit must be op_dtype), >= 128 channels at
 *   h_pixel_stride elements (a multiple of 16 bytes), 16-byte aligned.  packed_w / bias: 2 DEVICE pointers each,
 *   convrelu's (FH_CONV1 packing, 256 floats) then conv's (the permuted operand and bias above).  out_form:
 *   RDVC_MASK_OUT_UPSAMPLED: flow DEVICE fp32 (B, 2, H, W) at flow[b * s[0] + c * s[1] + y * s[2] + x * s[3]],
 *     s = flow_strides (4 HOST long longs, elements); out = the upsampled flow (B, 2, 8H, 8W) contiguous fp32.
 *   RDVC_MASK_OUT_MASK: flow ignored; out = multiplier * conv(...) (B, 576, H, W) contiguous act_dtype, stock
 *     channel order (MaskPredictor.forward's contract).
 *   out 16-byte aligned.  workspace: DEVICE, rdvc_corr_mask_predictor_workspace_bytes(...), 256-byte aligned.  2 launches
 *   (3 for F32 h).  Deterministic: no atomics, every output element is written by one thread.                       */
#define RDVC_MASK_OUT_UPSAMPLED 0
#define RDVC_MASK_OUT_MASK 1
size_t rdvc_corr_mask_conv_packed_weight_bytes(void);
int rdvc_corr_mask_conv_pack_weights(const float* weight, const float* bias, int op_dtype, void* packed_host,
                                     float* bias_host);
size_t rdvc_corr_mask_predictor_workspace_bytes(int B, int H, int W, int act_dtype);
int rdvc_corr_mask_predictor(const void* h, long long h_pixel_stride, int act_dtype, int B, int H, int W, int op_dtype,
                             const void* const* packed_w, const float* const* bias, float multiplier, const float* flow,
                             const long long* flow_strides, int out_form, void* workspace, size_t workspace_bytes, void* out,
                             void* stream);

/* ---- RAFT's context encoder (torchvision FeatureEncoder, BatchNorm2d in eval mode, raft_large's configuration) ---- *
 * The 16 convolutions, in parameter-tree order (layer index i of the pack arrays):
 *   0 convnormrelu (7x7 s2, 3 -> 64); 1-4 layer1.{0,1}.convnormrelu{1,2} (3x3, 64 -> 64);
 *   5 layer2.0.convnormrelu1 (3x3 s2, 64 -> 96), 6 layer2.0.downsample (1x1 s2, 64 -> 96), 7 layer2.0.convnormrelu2,
 *   8-9 layer2.1.convnormrelu{1,2} (3x3, 96 -> 96); 10 layer3.0.convnormrelu1 (3x3 s2, 96 -> 128), 11 layer3.0.downsample,
 *   12 layer3.0.convnormrelu2, 13-14 layer3.1.convnormrelu{1,2} (3x3, 128 -> 128); 15 conv (1x1, 128 -> 256, no BN).
 * BatchNorm folds into the convolution in fp64: s = gamma / sqrt(var + eps), w' = w s, b' = beta + (b - mean) s, each
 * rounded once (w' to op_dtype, b' to fp32).  Every activation between layers is NHWC op_dtype; layer2's 96 channels
 * are stored at a 128-channel stride with channels 96-127 zero.  tcgen05 implicit GEMMs
 * (csrc/tap_conv_sm100.cuh), 16-bit operands, fp32 accumulation and epilogues; the residual blocks' epilogue is
 * relu(res + relu(acc + b)) (TV:raft.py:64-71); each stride-2 block's downsample runs in its first convolution.
 *
 * rdvc_corr_context_encoder_pack_weights (HOST, no GPU needed): per layer i, conv_w[i] (cout, cin, k, k) and conv_b[i]
 *   (cout) contiguous fp32; for i < 15 bn_w / bn_b / bn_mean / bn_var [i] (cout) fp32 and eps[i] (entries 15 ignored).
 *   Writes rdvc_corr_context_encoder_packed_weight_bytes() bytes of 16-bit GEMM operand to packed_host and
 *   rdvc_corr_context_encoder_packed_bias_bytes() bytes of fp32 biases to bias_host.  Copy both to the device.
 * rdvc_corr_context_encoder: image DEVICE (B, 3, H, W) in_dtype (F32 | F16 | BF16) at image[b * s[0] + c * s[1] + y * s[2]
 *   + x * s[3]], s = image_strides (4 HOST long longs, elements, >= 0), aligned to its element size; any H, W >= 1.
 *   out: DEVICE NHWC (B, ceil(H / 8), ceil(W / 8), 256) out_dtype (F32 or op_dtype) at out_pixel_stride elements (>= 256,
 *   a multiple of 16 bytes), 16-byte aligned, overlapping neither the image nor the workspace.  out_form:
 *   RDVC_CE_OUT_RAW: conv's output (FeatureEncoder.forward); RDVC_CE_OUT_SPLIT: tanh on channels 0-127 and ReLU on
 *   128-255 (RAFT's hidden state and context).  workspace: DEVICE, rdvc_corr_context_encoder_workspace_bytes(...),
 *   256-byte aligned; after the call it holds every intermediate, each in its own buffer of
 *   align256(B * h * w * c * 2) bytes, in this order: at (H1, W1) = ceil((H, W) / 2), c = 64: the stem operand (per
 *   pixel 4 horizontal taps x 2 row phases x 2 column phases x 3 channels, zero-padded 48 -> 64), then the outputs
 *   of convnormrelu, layer1.0.convnormrelu1, layer1.0, layer1.1.convnormrelu1, layer1; at (H2, W2) = ceil((H1, W1) / 2),
 *   c = 128: layer2.0.convnormrelu1, layer2.0.downsample, layer2.0, layer2.1.convnormrelu1, layer2; at (H3, W3) =
 *   ceil((H2, W2) / 2), c = 128: the same for layer3.  15 launches.  Deterministic: no atomics; tiles never span images, so a sample's result does not
 *   depend on the batch it is in.                                                                                   */
#define RDVC_CE_OUT_RAW 0
#define RDVC_CE_OUT_SPLIT 1
#define RDVC_CE_LAYERS 16
size_t rdvc_corr_context_encoder_packed_weight_bytes(void);
size_t rdvc_corr_context_encoder_packed_bias_bytes(void);
int rdvc_corr_context_encoder_pack_weights(const float* const* conv_w, const float* const* conv_b,
                                           const float* const* bn_w, const float* const* bn_b,
                                           const float* const* bn_mean, const float* const* bn_var, const double* eps,
                                           int op_dtype, void* packed_host, float* bias_host);
size_t rdvc_corr_context_encoder_workspace_bytes(int B, int H, int W, int act_dtype);
int rdvc_corr_context_encoder(const void* image, const long long* image_strides, int in_dtype, int B, int H, int W,
                              int op_dtype, const void* packed_w, const float* biases, int out_form, void* workspace,
                              size_t workspace_bytes, void* out, long long out_pixel_stride, int out_dtype, void* stream);

/* ---- RAFT's feature encoder (torchvision FeatureEncoder, InstanceNorm2d without affine or running statistics,
 * raft_large's configuration) ---- *
 * The context encoder's 16 convolutions and units, each of the first 15 followed by InstanceNorm.  Weights: the
 * context encoder's packing (rdvc_corr_context_encoder_pack_weights) with the identity norm (bn_w = 1, bn_b = 0,
 * bn_mean = 0, bn_var = 1, eps = 0: s = 1 exactly, each weight rounded once).  The normalised layers' conv biases are
 * not used: InstanceNorm subtracts each (sample, channel)'s mean, so IN(y + b) = IN(y) exactly.
 * Per normalised unit (13; a stride-2 unit also carries its block's 1x1 downsample) three launches:
 *   the convolution (tcgen05, fp32 accumulation) stores its raw output y rounded to op_dtype and, per 16 x 8 tile and
 *     channel, (mean, M2) of the stored values over the tile's pixels inside the image;
 *   finalize merges a sample's tiles in a fixed order in fp64 (Chan) -> fp32 mean and rstd = 1 / sqrt(var + eps),
 *     var biased;
 *   apply, in fp32, rounded once to op_dtype: relu(IN(y)) (stem, convnormrelu1), relu(x + relu(IN(y))) (convnormrelu2
 *     of an identity block, x its input) or relu(IN(ds) + relu(IN(y))) (of a stride-2 block, ds its downsample's raw
 *     output).  layer2's channels 96-127 are written as exact zeros.
 * No atomics, and tiles never span images: a sample's result does not depend on the batch it is in.
 *
 * rdvc_corr_feature_encoder_workspace_bytes: 0 for a non-positive size, an unknown act_dtype or a one-element layer3
 *   plane (ceil(H / 8) = ceil(W / 8) = 1, which InstanceNorm cannot normalise).
 * rdvc_corr_feature_encoder: image, image_strides, in_dtype, B, H, W, op_dtype, packed_w, biases: as for
 *   rdvc_corr_context_encoder; eps: RDVC_FE_NORMS HOST doubles (>= 0, finite), indexed like the pack arrays (layer i <
 *   15 of the context encoder's list).  out_form:
 *   RDVC_FE_OUT_FEATURES: FeatureEncoder.forward, NHWC (B, ceil(H / 8), ceil(W / 8), 256) out_dtype (F32 or op_dtype),
 *     out_pixel_stride >= 256;
 *   RDVC_FE_OUT_TRUNK: layer3's output, NHWC (B, ceil(H / 8), ceil(W / 8), 128) op_dtype, out_pixel_stride >= 128 (the
 *     input of the final 1x1, e.g. for TVCorrBlock.build_pyramid_from_encoder).
 *   out: a multiple of 16 bytes per pixel, 16-byte aligned, overlapping neither the image nor the workspace.
 *   workspace: DEVICE, rdvc_corr_feature_encoder_workspace_bytes(...), 256-byte aligned; after the call it holds every
 *   intermediate, each in its own buffer of align256(bytes), in this order:
 *     at (H1, W1), B * H1 * W1 * 64 16-bit values each: the stem operand, then y and the normalised activation a of
 *       convnormrelu, layer1.0.convnormrelu1, layer1.0.convnormrelu2 (a = layer1.0's output), layer1.1.convnormrelu1,
 *       layer1.1.convnormrelu2 (11 buffers);
 *     at (H2, W2), 128-channel pixels: y, downsample y, a of layer2.0.convnormrelu1, then y, a of
 *       layer2.0.convnormrelu2, layer2.1.convnormrelu1, layer2.1.convnormrelu2 (9 buffers);
 *     at (H3, W3): the same for layer3 (with RDVC_FE_OUT_TRUNK the last a goes to out and its buffer is untouched);
 *     per normalised unit u = 0..12 (stem, layer1 x 4, layer2.0 conv1 + downsample, 3 more of layer2, the same for
 *       layer3): float2 (mean, M2) partials [B * ceil(w_u / 16) * ceil(h_u / 8)][NT_u], tiles along x first, NT_u =
 *       64 (layer1), 128, or 256 for a stride-2 unit (channels 128-255: its downsample);
 *     per normalised unit: fp32 [B][2][NT_u], mean then rstd.
 *   1 + 13 x 3 launches, + 1 (the 1x1) for RDVC_FE_OUT_FEATURES.                                                    */
#define RDVC_FE_OUT_FEATURES 0
#define RDVC_FE_OUT_TRUNK 1
#define RDVC_FE_NORMS 15
size_t rdvc_corr_feature_encoder_workspace_bytes(int B, int H, int W, int act_dtype);
int rdvc_corr_feature_encoder(const void* image, const long long* image_strides, int in_dtype, int B, int H, int W,
                              int op_dtype, const void* packed_w, const float* biases, const double* eps, int out_form,
                              void* workspace, size_t workspace_bytes, void* out, long long out_pixel_stride,
                              int out_dtype, void* stream);

/* ---- the whole RAFT call: torchvision raft_large's flow, every network on this library's kernels -------------- *
 * The C counterpart of rc.raft_flow / rc.raft_flow_sequence with all six drop-ins (feature and context encoders,
 * motion encoder, recurrent block, flow head, mask predictor) and TVCorrBlock: images in, flow_preds[-1] out
 * (R:codec_processing.py:1442-1444).  Caller-owned memory, the caller's stream, no allocation, no host
 * synchronisation: a call can be captured into a CUDA graph.  All arguments are checked before the first launch; a
 * refused call enqueues nothing.
 *
 * Weights (HOST, no GPU needed).  rdvc_corr_raft_pack_weights takes raft_large's state_dict(): n (name, contiguous fp32
 * tensor, ndim, shape) entries in any order, the context encoder's BatchNorm buffers included (num_batches_tracked is
 * ignored; BatchNorm and InstanceNorm eps are torchvision's 1e-5).  A missing key, a wrong shape (RDVC_E_SHAPE), an
 * unexpected or duplicate key (RDVC_E_UNSUPPORTED: raft_small's state dict is refused this way) names the key in
 * rdvc_corr_last_error().  op_dtype: RDVC_DT_F16, the operand type of both activation dtypes.  The blob,
 * rdvc_corr_raft_packed_weight_bytes(op_dtype) long: a header { uint32 magic 0x54464152 ("RAFT"), uint32 version 1, int32
 * op_dtype, int32 RDVC_RAFT_SECTIONS, uint64 offset[RDVC_RAFT_SECTIONS], uint64 bytes[RDVC_RAFT_SECTIONS] }, then the
 * sections, each at a 256-byte aligned offset, written ONLY by the existing pack functions (biases used as they are
 * are fp32 copies), in this order:
 *    0, 1  feature encoder: rdvc_corr_context_encoder_pack_weights with the identity norm (weights, biases)
 *    2, 3  context encoder: the same with its BatchNorm folded (weights, biases)
 *    4, 5  feature_encoder.conv: rdvc_linear_pack_weights (256, 128), bias
 *    6, 7  motion_encoder.convcorr1: rdvc_conv1x1_pack_weights (256, 4 levels, radius 4), bias
 *    8-11  motion_encoder convcorr2, convflow1, convflow2, conv: rdvc_corr_update_conv_pack_weights;  12-15 their biases
 *   16, 17 flow_head conv1, conv2 (update-conv packing);  18, 19 their biases
 *   20, 21 recurrent_block convgru1, convgru2: rdvc_corr_convgru_pack_weights;  22-27 biases z, r, q of convgru1, then 2
 *   28, 29 mask_predictor convrelu (FH_CONV1 packing), conv (rdvc_corr_mask_conv_pack_weights);  30, 31 their biases
 *          (31: the permuted bias_host of the mask-conv pack)
 * Copy the blob to the device (cudaMemcpy / cudaMemcpyAsync) at a 256-byte aligned address.
 *
 * rdvc_corr_raft_flow: image1, image2 DEVICE (B, 3, H, W) in_dtype (F32 | F16 | BF16) at image[b * s[0] + c * s[1] + y * s[2]
 *   + x * s[3]], s = image_strides (4 HOST long longs, elements, >= 0, shared by both images).  flow_out: DEVICE
 *   (B, 2, H, W) contiguous fp32, 16-byte aligned.
 * rdvc_corr_raft_flow_sequence: frames (n_frames, 3, H, W) at frame_strides: the n_frames - 1 consecutive pairs (frame i,
 *   frame i + 1); the feature encoder sees each frame once and pair i reads its trunk rows i and i + 1 in place.
 *   flow_out: (n_frames - 1, 2, H, W).  Bit-identical to rdvc_corr_raft_flow on the same pairs.
 * Both: H, W multiples of 8 with H / 8, W / 8 >= 16 (RDVC_E_SHAPE / RDVC_E_TOO_SMALL), iters >= 1 (RDVC_E_SHAPE).
 *   act_dtype F32 (torch's eager fp32) or F16 (fp16 autocast); the operands are fp16 either way, the hidden state,
 *   context and motion features are act_dtype.  vol_dtype F32 | BF16 (the pyramid).  mask_multiplier: the mask
 *   predictor's (0.25 for raft_large).  packed_weights / workspace 256-byte aligned; workspace_bytes >=
 *   rdvc_corr_raft_workspace_bytes(2 B, B, ...) for rdvc_corr_raft_flow, (n_frames, n_frames - 1, ...) for the sequence.
 *   Images, workspace and flow_out must not overlap.
 * rdvc_corr_raft_workspace_bytes(n_images, n_pairs, ...): 0 for invalid arguments (n_pairs < n_images <= 2 n_pairs).
 *   Layout, every buffer at a 256-byte aligned offset, (h, w) = (H, W) / 8, P = n_pairs * h * w pixels:
 *     persistent: the pyramid (rdvc_corr_pyramid_bytes(n_pairs, h, w, 4, vol_dtype, RDVC_LAYOUT_TILED): the bulk,
 *       5.7 GB per 1080p pair with an fp32 volume); the context encoder's split output (P x 256 act_dtype: tanh hidden
 *       state | relu context); coords1 and flow (each (n_pairs, 2, h, w) fp32);
 *     then one scratch region, reused by three phases whose buffers are dead before the next starts:
 *       1. the trunk (n_images x h x w x 128 fp16, NHWC), then the feature encoder's workspace (for n_images) or,
 *          at the same offset, the encoder tail's input and output rows (rdvc_corr_workspace_bytes for D = 128, 256);
 *       2. the context encoder's workspace;
 *       3. the K-major lookup features (rdvc_corr_feat_bytes), convcorr1's output (P x 256 fp16), the motion features,
 *          convgru1's output and the hidden state (P x 128 act_dtype each), and one workspace shared by the motion
 *          encoder, the ConvGRU, the flow head and the mask predictor (the largest of theirs).
 * Order: feature encoder (trunk) -> rdvc_corr_pack_nhwc -> rdvc_corr_encoder_tail -> rdvc_corr_build_packed -> context
 *   encoder (RDVC_CE_OUT_SPLIT) -> coords1 = grid, flow = 0 (one kernel) -> iters x [lookup + convcorr1 (NHWC) ->
 *   motion encoder -> convgru1 -> convgru2 -> flow head, whose conv2 epilogue rounds delta to act_dtype, adds it to
 *   coords1 in fp32 and writes flow = coords1 - grid] -> mask predictor + convex upsampling into flow_out.
 * Launches per call (rdvc_corr_launch_count): 40 x (2 for rdvc_corr_raft_flow, 1 for the sequence) + 3 + 15 + 1
 *   + iters x (12 for F16, 15 for F32) + (2 for F16, 3 for F32).  Deterministic: no atomics anywhere on the path. */
#define RDVC_RAFT_SECTIONS 32
size_t rdvc_corr_raft_packed_weight_bytes(int op_dtype);
int rdvc_corr_raft_pack_weights(const char* const* names, const float* const* tensors, const int* ndims,
                           const long long* const* shapes, int n, int op_dtype, void* packed_host, size_t bytes);
size_t rdvc_corr_raft_workspace_bytes(int n_images, int n_pairs, int H, int W, int act_dtype, int vol_dtype);
int rdvc_corr_raft_flow(const void* image1, const void* image2, const long long* image_strides, int in_dtype, int B, int H,
                   int W, int iters, int act_dtype, int vol_dtype, const void* packed_weights, float mask_multiplier,
                   void* workspace, size_t workspace_bytes, float* flow_out, void* stream);
int rdvc_corr_raft_flow_sequence(const void* frames, const long long* frame_strides, int in_dtype, int n_frames, int H, int W,
                            int iters, int act_dtype, int vol_dtype, const void* packed_weights, float mask_multiplier,
                            void* workspace, size_t workspace_bytes, float* flow_out, void* stream);

/* ---- next row f-4 (last piece): entropy-coder stand-in (HOST functions) ---- *
 * Stands in for the range coder behind EntropyBottleneck.compress / .decompress (R:codec_processing.py:433,447
 * construction, :488-497 compress, :509-536 decompress; compressai's RansEncoder.encode_with_indexes /
 * RansDecoder.decode_with_indexes).  compressai is absent from this image: the BITSTREAM IS NOT the reference's
 * (parity unpinned); interface and modelling contract are: per-index quantised CDF tables of 16-bit precision
 * (cdfs: n_tables rows of max_len entries, row i valid for cdf_lengths[i] entries, first 0, last 65536, strictly
 * increasing; the last slot of a table is the escape for symbols outside [offsets[i], offsets[i] + cdf_lengths[i] - 2),
 * coded with 4-bit bypass digits), rANS with a 32-bit state and 16-bit words.  encode -> decode is bit exact.
 * _encode returns the number of bytes written (0 = error, see rdvc_corr_last_error); out_capacity >=
 * rdvc_ec_max_encoded_bytes(n) always suffices.  _decode returns 0 or a negative RDVC_E_*.                      */
size_t rdvc_ec_max_encoded_bytes(size_t n);
size_t rdvc_ec_encode_with_indexes(const int* symbols, const int* indexes, size_t n, const unsigned int* cdfs,
                                   const int* cdf_lengths, const int* offsets, int n_tables, int max_len,
                                   unsigned char* out, size_t out_capacity);
int rdvc_ec_decode_with_indexes(const unsigned char* in, size_t nbytes, const int* indexes, size_t n,
                                const unsigned int* cdfs, const int* cdf_lengths, const int* offsets, int n_tables,
                                int max_len, int* symbols_out);

/* Frees the per-thread scratch arenas of rdvc_corr_pair_host* (optional). */
void rdvc_corr_release(void);

/* ---- introspection for tests / benches --------------------------------- */
/* Number of kernels this library has launched on the calling thread.         */
unsigned long long rdvc_corr_launch_count(void);
/* Caller-owned cudaEvent_t pair recorded on the build stream immediately before and after
 * the main build kernel of the next rdvc_corr_build calls on this thread (NULL, NULL = off).
 * Lets a bench time the dominant kernel alone, on the stream it runs on.             */
void rdvc_corr_set_profile_events(void* start_event, void* stop_event);
/* How many rdvc_corr_build calls of this process found their plan (TMA descriptors + work split) in the cache. */
unsigned long long rdvc_corr_plan_cache_hits(void);
/* Tuning knobs; unknown keys return RDVC_E_UNSUPPORTED.  [EXP] = accepted only by a library compiled with
 * -DRDVC_EXPERIMENTS (lib/librdvc_corr_exp.so, never the product build): knobs that skip work for timing
 * experiments and the build variants that lost their measurements.
 *   key 0: lookup variant   (0 = auto, 1 = scalar loads, 2 = 128-bit loads,
 *                            [EXP] 3 / 4 = timing only: skip the volume loads / the output stores)
 *   key 1: [EXP] fused-mode build tile shape (0 = auto, 1 = 16x16, 2 = 8x32 fmap2 pixels)
 *   key 2: build m-range slices per fmap2 tile (0 = auto)
 *   key 3: [EXP] bit mask of pyramid levels the build writes (default 15)
 *   key 4: build mode (0 = auto, [EXP] 1 = fused pooling epilogue, 2 = pooled-fmap2 rows)
 *   key 5: linear-mode output path (1 = auto: TMA boxes 16 rows x 256 B where the row pitch allows,
 *          else 32 rows x 128 B, else staged stores; 2 = never the wide boxes; 0 = staged only)
 *   key 6: [EXP] L2 policy of the TMA stores (0 default, 1 evict_last, 2 evict_first)
 *   key 7 / 8: experiment: log2 tile width / height of RDVC_LAYOUT_TILED (0 = default)
 *   key 9: build epilogue warps (0 = auto: 8 for an fp32 volume, 4 for bf16; 4; 8)
 *   key 12: build kernel (0 = auto, 1 = one CTA per tile; [EXP] 2 = CTA pairs / tcgen05 cta_group::2, [EXP] 3 = clusters
 *           of two CTAs that hold neighbouring fmap2 tiles and share ONE fmap1 stream through TMA multicast: both
 *           bit-identical, neither faster at 1080p, see DESIGN.md 3.2)
 *   key 13: experiment: MCN convolutions pull their boxes into L2 this many tiles ahead with TMA prefetches
 *           (default 0 = off: no effect measured at 1-4, slower beyond)
 *   key 14: MCN convolution kernel (0 = auto, 1 = three activation boxes per tile, 2 = one box per tile
 *           with the x halo handled in the epilogue; same results up to fp32 summation order)     */
int rdvc_corr_set_option(int key, int value);

#ifdef __cplusplus
}
#endif
#endif /* RDVC_CORR_H_ */
